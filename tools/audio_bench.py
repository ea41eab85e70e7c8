"""wav2vec2 audio-embedding timing on one GPU at chinese-wav2vec2-base size (7 convs of 512 channels, 12 post-LN layers of
768, 12 heads of 64), seeded synthetic weights and speech-like audio.

    python tools/audio_bench.py [--seconds 10,60,600] [--out audio_bench.json]

Per audio length: the embedding's wall time on the device (CUDA events, after a warm-up call of the same length, mean of
--iters calls), the split into conv stack / positional conv / GEMMs / attention / row kernels (events around every launch
of one extra instrumented call, so the split adds event overhead the total above does not have), algorithmic TFLOP/s per
stage (tools/flops.py) and the CPU oracle's time for the first length on the host cores, where the reference runs it.
Prints one JSON object with the card's name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "stable-video-infinity_b200")):
    sys.path.insert(0, p)
from tools import flops, synth_audio as SA  # noqa: E402

# which nv wrapper each engine launch goes through -> stage
_STAGE = {"audio_conv0_gn_gelu": "conv", "audio_interp_layernorm": "rows", "audio_pos_conv": "pos_conv",
          "layernorm_f32x2": "rows", "attention_small": "attention", "cast_f32_to_bf16": "conv", "gemm": None}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return [s.strip() for s in q.split(",")]
    except Exception as e:  # noqa: BLE001
        return [torch.cuda.get_device_name(0), f"unknown ({e})", "unknown"]


def staged(eng, wav, S):
    """One call with events around every kernel wrapper: milliseconds per stage."""
    from diffsynth import _native as nv
    saved = {n: getattr(nv, n) for n in _STAGE}
    rec = []
    in_conv = [True]

    def wrap(name, fn):
        def f(*a, **k):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            r = fn(*a, **k)
            e.record()
            stage = _STAGE[name] or ("conv" if in_conv[0] else "gemm")
            rec.append((stage, s, e))
            return r
        return f

    try:
        for n, fn in saved.items():
            setattr(nv, n, wrap(n, fn))
        feats = eng.conv_stack(wav)
        in_conv[0] = False
        eng.encode(feats, S)
        torch.cuda.synchronize()
    finally:
        for n, fn in saved.items():
            setattr(nv, n, fn)
    out = {}
    for stage, s, e in rec:
        out[stage] = out.get(stage, 0.0) + s.elapsed_time(e)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", default="10,60,600")
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--out", default="")
    ap.add_argument("--no-cpu", action="store_true")
    a = ap.parse_args()
    from oracle import wav2vec2_oracle as O
    from utils.src.audio_analysis.wav2vec2 import Wav2Vec2FeatureExtractor, Wav2Vec2Model
    cfg = SA.W2V_BASE
    sd = SA.make_state_dict(cfg, seed=1)
    m = Wav2Vec2Model(cfg)
    m.load_state_dict(sd)
    eng = m.eval().engine("cuda:0")
    fe = Wav2Vec2FeatureExtractor()
    name, plimit, maxclk = card()
    res = dict(card=name, power_limit=plimit, max_sm_clock=maxclk, config="chinese-wav2vec2-base shapes, seeded weights",
               cases=[])
    secs = [float(s) for s in a.seconds.split(",")]
    for sec in secs:
        x = SA.make_waveform(sec, seed=2)
        S = int(len(x) / 16000 * 25)
        wav = torch.from_numpy(fe(x).input_values[0]).cuda()
        eng.forward(wav, S)                                   # warm-up at this length
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        for _ in range(a.iters):
            eng.forward(wav, S)
        ev[1].record()
        torch.cuda.synchronize()
        ms = ev[0].elapsed_time(ev[1]) / a.iters
        st = staged(eng, wav, S)
        fl = flops.wav2vec_flops(len(x), cfg)
        case = dict(seconds=sec, seq_len=S, embed_ms=round(ms, 3), tflops_total=round(sum(fl.values()) / ms / 1e9, 2),
                    stage_ms={k: round(v, 3) for k, v in sorted(st.items())},
                    stage_tflops={k: round(fl[k] / st[k] / 1e9, 2) for k in fl if st.get(k)},
                    gflop={k: round(v / 1e9, 2) for k, v in fl.items()})
        res["cases"].append(case)
        print(json.dumps(case), file=sys.stderr)
    if not a.no_cpu:
        x = SA.make_waveform(secs[0], seed=2)
        torch.set_num_threads(os.cpu_count())
        O.get_embedding(x[:16000], sd, cfg)
        t = time.perf_counter()
        O.get_embedding(x, sd, cfg)
        res["cpu_oracle"] = dict(seconds=secs[0], ms=round((time.perf_counter() - t) * 1e3, 1), threads=torch.get_num_threads(),
                                 note="torch fp32 on the host cores (where the reference runs its encoder)")
    s = json.dumps(res)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
