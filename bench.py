"""bench.py — denoised latent frames/sec of the SVI clip-denoising hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload cfg2|cfg3|cfg4|cfg5|cfg1|tiny] [--dump-outputs DIR]

Default workload cfg2 = BASELINE.json configs[1] (the configuration the metric is quoted on): a "step" is ONE
flow-matching denoise step of the clip — two Wan-DiT forwards (classifier-free guidance) + the fused CFG/Euler update —
on synthetic inputs (Wan2.1-T2V-1.3B, 81 frames x 480 x 832 -> latents [1,16,21,60,104], L = 32760 tokens, 512 text
tokens, random-init weights).  value = 21 latent frames / (50 * seconds_per_step).  Timing: CUDA events on the launching
stream, barrier + synchronize on both sides, max over ranks.  The working set of one step (2.8 GB of weights + ~1.5 GB
of activations) is far larger than the 126 MB L2, so no explicit L2 flush is needed ("inputs larger than L2").

Every step — timed (`value`, device-resident inputs) and end-to-end (`e2e`, pinned host buffers copied in and the updated
latents copied out every step) — goes through the pipeline's own step function, SVIVideoPipeline.denoise_step, on one GPU
and on N: ranks split as CFG-parallel x token-axis sequence-parallel (distributed/sequence_parallel.py), which is also the
plan `from_model_manager(use_usp=True)` gives the public pipeline call; total work is fixed -> "scaling": "strong".
N > 1 runs first check the plan against a single-rank step on rank 0's GPU (`sp_parity`).

Other workloads (SURVEY.md §8d; each prints its own JSON line, same keys where they apply):
  cfg3  Wan2.1-I2V-14B (+ merged rank-128 LoRA) 81f x 720 x 1280, L = 75600, 257 CLIP + 512 text tokens (configs[2])
  cfg4  10 chained clips through SVIVideoPipeline.__call__ incl. encoders and VAE -> clips/hour (configs[3])
  cfg5  VAE encode / decode sweep 17..161 frames x 720p -> TF/s and GB/s against both rooflines (configs[4])

--impl reference: the reference's own CPU path for the same step, timed on the host cores.  The reference package
itself cannot be installed offline (missing diffusers / xfuser / xformers / imageio and no GPU attention library for
CPU), so the arm runs the oracle port (oracle/wan_dit_oracle.py, pinned to the reference by tests/golden) on a bounded
sample: one DiT block at the workload's L, extrapolated.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "stable-video-infinity_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

WORKLOADS = {
    # name: (cfg name, latent f, h, w, ctx_len, description)
    "cfg2": ("CFG_T2V_1_3B", 21, 60, 104, 512, "Wan2.1-T2V-1.3B 81fx480x832, 50-step CFG denoise (BASELINE configs[1])"),
    "cfg1": ("CFG_T2V_1_3B", 5, 40, 64, 512, "Wan2.1-T2V-1.3B 17fx320x512 (BASELINE configs[0])"),
    "tiny": ("CFG_TINY_T2V", 3, 16, 16, 64, "tiny 2-layer debug model"),
    "cfg3": ("CFG_I2V_14B", 21, 90, 160, 512, "Wan2.1-I2V-14B + merged rank-128 LoRA, 81fx720x1280, 50-step CFG denoise (BASELINE configs[2])"),
    "cfg3-480p": ("CFG_I2V_14B", 21, 60, 104, 512, "Wan2.1-I2V-14B + merged rank-128 LoRA, 81fx480x832"),
}
CLIP_STEPS = 50
CFG_SCALE = 5.0
METRIC = "denoised latent frames/sec (81fx480p, 50 steps)"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, d.get("bf16_tflops_sustained", d.get("bf16_tflops")), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    return {}, 1400.0, "fallback (B200_PROFILING.md sustained ~1.4 PFLOP/s)"


def host_cpu():
    """Model name + logical cores of the box (the reference arm's speed swings 4x between hosts)."""
    name = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                name = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return {"model": name, "logical_cores": os.cpu_count()}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        time.sleep(0.05)
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = max((int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()), default=None)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        pw = sorted(float(r[6]) for r in self.rows if len(r) > 6 and r[6].replace(".", "", 1).isdigit())
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(sm),
                "power_w": pw[len(pw) // 2] if pw else None}


def build_model(cfg, device, lora_rank=0):
    """Random-init weights of the architecture generated on the device (bf16, like a Wan checkpoint); lora_rank > 0 merges a
    random rank-r LoRA (A [r, d_in], B [d_out, r], alpha = r) into q,k,v,o,ffn.0,ffn.2 through the product's LoRA merge."""
    from diffsynth.models.wan_video_dit import WanModel, precompute_freqs_cis_3d
    from tools import synth
    with torch.device("meta"):
        model = WanModel(**cfg)
    sd = synth.make_dit_state_dict_fast(cfg, seed=0, device=device, dtype=torch.bfloat16)
    model.load_state_dict(sd, assign=True)
    model.freqs = precompute_freqs_cis_3d(128)  # the meta-device construction above produced meta tables
    model.eval()
    if lora_rank:
        from diffsynth.models.lora import GeneralLoRAFromPeft
        g = torch.Generator(device=device).manual_seed(77)
        lora = {}
        for name, p in model.named_parameters():
            if name.endswith(".weight") and p.dim() == 2 and any(t in name for t in (".q.", ".k.", ".v.", ".o.", ".ffn.0.", ".ffn.2.")) \
                    and "audio" not in name and "_img" not in name:
                base = name[:-len(".weight")]
                lora[f"{base}.lora_A.default.weight"] = (torch.randn(lora_rank, p.shape[1], generator=g, device=device) / p.shape[1] ** 0.5).to(torch.bfloat16)
                lora[f"{base}.lora_B.default.weight"] = (torch.randn(p.shape[0], lora_rank, generator=g, device=device) * (0.1 / lora_rank ** 0.5)).to(torch.bfloat16)
        GeneralLoRAFromPeft().load(model, lora, alpha=1.0)      # W += B A on the native GEMM (alpha as gate, W as residual)
        model.lora_merged = len(lora) // 2
    return model


def block_fixture(cfg, L, ctx_len, grid):
    """Seeded inputs of ONE DiT block at the workload's token count (bf16-rounded weights: what a checkpoint holds)."""
    from tools import synth
    one = dict(cfg, num_layers=1)
    sd = {k: v.to(torch.bfloat16).float() for k, v in synth.make_dit_state_dict(one, seed=0).items()}
    g = torch.Generator().manual_seed(0)
    d = cfg["dim"]
    x = torch.randn(1, L, d, generator=g)
    ctx = torch.randn(1, ctx_len, d, generator=g).to(torch.bfloat16).float()
    t_mod = torch.randn(1, 6, d, generator=g) * 0.1
    return one, sd, x, ctx, t_mod


def cpu_block_baseline(cfg, L, ctx_len, grid, max_seconds=45.0):
    """Reference CPU path (oracle port) on the host cores: ONE DiT block forward at the workload's token count
    (1/(layers*100) of a clip), fp32, all cores.  Returns (seconds per block, cores, fixture, oracle output)."""
    from oracle import wan_dit_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    one, sd, x, ctx, t_mod = block_fixture(cfg, L, ctx_len, grid)
    ang = O.rope_angles_3d(128, *grid)
    with torch.no_grad():
        t0 = time.perf_counter()
        out = O.dit_block(sd, 0, x, ctx, t_mod, ang, one)
        dt = time.perf_counter() - t0
        if dt < max_seconds / 3:   # a second run if it is cheap enough (first run includes allocator warm-up)
            t0 = time.perf_counter()
            out = O.dit_block(sd, 0, x, ctx, t_mod, ang, one)
            dt = min(dt, time.perf_counter() - t0)
    return dt, cores, (one, sd, x, ctx, t_mod), out


def native_block_parity(fixture, ref, grid, dev):
    """The same block on the native kernels (WanDiTEngine.run_block) against the oracle output the cpu_baseline leg just
    produced: fraction of elements inside rtol 1e-2 / atol 1e-3, max |err|, mean |err| / std."""
    from diffsynth.models.wan_video_dit import WanModel
    one, sd, x, ctx, t_mod = fixture
    m = WanModel(**one).eval()
    m.load_state_dict(sd)
    m.to(dev)
    eng = m.engine(dev)
    d = one["dim"]
    st = eng.project_context(ctx[0].to(dev, torch.bfloat16))
    mods = (sd["blocks.0.modulation"].reshape(6, d) + t_mod[0]).to(dev).contiguous()
    cos, sin = eng.rope(*grid)
    xg = x[0].to(dev).contiguous()
    eng.run_block(0, xg, mods, st, cos, sin)
    torch.cuda.synchronize()
    out, r = xg.cpu(), ref[0]
    err = (out - r).abs()
    return {"what": f"one DiT block at L={x.shape[1]} (native run_block vs oracle.dit_block, identical bf16-rounded weights)",
            "inside": (err <= 1e-3 + 1e-2 * r.abs()).float().mean().item(), "max": err.max().item(),
            "mean_over_std": err.mean().item() / r.std().item(), "rtol": 1e-2, "atol": 1e-3}


def run_reference_arm(args, wl_name, cfg, f, h, w, ctx_len, desc):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    L = f * (h // 2) * (w // 2)
    times = []
    budget_s = 170.0        # keep the whole arm within a few minutes on any host
    t_start = time.perf_counter()
    warm = args.warmup
    for i in range(args.warmup + args.steps):
        dt, cores, _, _ = cpu_block_baseline(cfg, L, ctx_len, (f, h // 2, w // 2))
        if i == 0 and dt > 8.0:
            warm = min(warm, 1)          # a >8 s sample: one untimed warm-up is all the budget allows
        if i >= warm:
            times.append(dt)
        if len(times) >= args.steps or (times and time.perf_counter() - t_start > budget_s):
            break
    t_blk = sum(times) / len(times)
    step_s = t_blk * cfg["num_layers"] * 2            # one denoise step = 2 forwards x num_layers blocks (+ negligible rest)
    value = f / (CLIP_STEPS * step_s)
    line = {"impl": "reference", "metric": METRIC, "value": value,
            "unit": "latent_frames/s", "n_gpus": args.gpus, "steps": len(times), "warmup": args.warmup,
            "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl_name, "description": desc, "tokens": L},
            "cpu_baseline": {"value": value, "unit": "latent_frames/s", "cores": cores, "kind": "port", "host_cpu": host_cpu(),
                             "sample": f"1 DiT block forward at L={L} per step sample ({t_blk:.2f} s), extrapolated x{cfg['num_layers']} blocks x2 CFG forwards x{CLIP_STEPS} steps"},
            "e2e": {"value": value, "unit": "latent_frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def vae_clip_leg(dev, f, h, w, ms_per_step):
    """Times WanVideoVAE.decode / .encode (public API, random-init weights) at the bench clip shape and folds them into a
    whole-clip figure: one SVI clip = encode(81 frames) + 50 CFG steps + decode(21 latent frames)."""
    from diffsynth.models.wan_video_vae import WanVideoVAE
    from tools import synth_vae
    vae = WanVideoVAE().eval()
    vae.load_state_dict(synth_vae.make_vae_state_dict(seed=0))
    vae.to(dev)
    g = torch.Generator().manual_seed(3)
    z = torch.randn(1, 16, f, h, w, generator=g).to(dev)
    frames = 4 * (f - 1) + 1
    video = (torch.rand(3, frames, 8 * h, 8 * w, generator=g) * 2 - 1).to(dev)
    out = {}
    for name, fn in (("decode", lambda: vae.decode(z, device=dev)), ("encode", lambda: vae.encode([video], device=dev))):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out[name] = a.elapsed_time(b)
    clip_s = (out["encode"] + out["decode"] + CLIP_STEPS * ms_per_step) / 1e3
    return {"vae_decode_ms": out["decode"], "vae_encode_ms": out["encode"], "denoise_s": CLIP_STEPS * ms_per_step / 1e3,
            "clip_s": clip_s, "clips_per_hour": 3600.0 / clip_s, "pixel_frames_per_s": frames / clip_s,
            "note": "81f x 480x832 clip = VAE encode + 50 CFG steps (extrapolated from the timed steps) + VAE decode; "
                    "the umT5 / CLIP encoders add ~57 ms per clip (2 prompts x 25 ms + 7 ms, tools/enc_bench.py) and are not timed here"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=list(WORKLOADS) + ["cfg4", "cfg5"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cfg-parallel", action="store_true", help="N>1: split only the token axis (sp = N); for A/B runs")
    ap.add_argument("--breakdown", action="store_true", help="after the timed run, one extra step with every kernel call "
                    "bracketed by CUDA events; per-call-type sums of rank 0 go to stderr (not part of the JSON line)")
    ap.add_argument("--no-vae", action="store_true", help="skip the clip-boundary VAE leg (decode 21->81 frames, encode 81 frames)")
    ap.add_argument("--no-sp-parity", action="store_true", help="N>1: skip the plan-vs-single-rank check before the timed run")
    ap.add_argument("--clips", type=int, default=10, help="cfg4: clips in the chain")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (float32): "
                    "the updated latents and, on one GPU, the conditional / unconditional velocity fields; inputs are seeded, "
                    "so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "native" or args.workload not in WORKLOADS):
        ap.error("--dump-outputs applies to the native DiT workloads (" + ", ".join(WORKLOADS) + ")")
    if args.workload == "cfg4":
        from tools import clip_loop_bench
        return clip_loop_bench.main_from_bench(args)
    if args.workload == "cfg5":
        from tools import vae_bench
        return vae_bench.sweep_from_bench(args)
    from tools import flops, synth
    cfg_name, f, h, w, ctx_len, desc = WORKLOADS[args.workload]
    cfg = getattr(synth, cfg_name)
    if args.impl == "reference":
        run_reference_arm(args, args.workload, cfg, f, h, w, ctx_len, desc)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the native arm has no CPU fallback")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import torch.distributed as dist
    sp = None
    plan = "single"
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        from diffsynth.distributed.sequence_parallel import init_sp_groups
        sp = init_sp_groups(world, rank, cfg_parallel=not args.no_cfg_parallel)
        plan = sp.describe()
    from diffsynth.pipelines.svi_video import SVIVideoPipeline
    from diffsynth.schedulers.flow_match import FlowMatchScheduler

    i2v = bool(cfg["has_image_input"])
    model = build_model(cfg, dev, lora_rank=128 if args.workload.startswith("cfg3") else 0)
    pipe = SVIVideoPipeline(device=dev, torch_dtype=torch.bfloat16)      # the public object whose step function is timed
    pipe.dit = model
    pipe.use_unified_sequence_parallel = world > 1
    eng = model.engine(dev)
    sched = FlowMatchScheduler(shift=5, sigma_min=0.0, extra_one_step=True)
    sched.set_timesteps(CLIP_STEPS, shift=5.0)
    g = torch.Generator(device="cpu").manual_seed(0)
    lat_host = torch.randn(1, 16, f, h, w, generator=g).pin_memory()
    ctx_pos_host = torch.randn(1, ctx_len, cfg["text_dim"], generator=torch.Generator().manual_seed(1)).pin_memory()
    ctx_neg_host = torch.randn(1, ctx_len, cfg["text_dim"], generator=torch.Generator().manual_seed(2)).pin_memory()
    y_host = clip_host = None
    if i2v:     # SURVEY §8d cfg-3: y = cat[mask(4), randn(16)] with the first-frame mask of svi_video.py:319-326, CLIP feature randn
        inp = synth.make_dit_inputs(cfg, f, h, w, seed=0, ctx_len=ctx_len)
        y_host, clip_host = inp["y"].pin_memory(), inp["clip_feature"].pin_memory()
    lat = lat_host.to(dev).clone()
    y_dev = None if y_host is None else y_host.to(dev)
    clip_dev = None if clip_host is None else clip_host.to(dev)
    ctx_pos, ctx_neg = ctx_pos_host.to(dev), ctx_neg_host.to(dev)
    own0 = sp is None or sp.owns_branch(0)
    own1 = sp is None or sp.owns_branch(1)
    cp = eng.context_state(ctx_pos, clip_dev) if own0 else None
    cn = eng.context_state(ctx_neg, clip_dev) if own1 else pipe.OTHER_RANK
    v_c, v_u = torch.empty_like(lat), torch.empty_like(lat)
    L = f * (h // 2) * (w // 2)

    def sched_at(i):
        k = i % CLIP_STEPS
        return float(sched.timesteps[k]), float(sched.sigmas[k]), (float(sched.sigmas[k + 1]) if k + 1 < CLIP_STEPS else 0.0)

    def step(i, x=lat, cpx=cp, cnx=cn, plan_sp=sp):
        t, sigma, nxt = sched_at(i)
        pipe.denoise_step(eng, x, t, sigma, nxt, cpx, cnx, v_c, v_u, CFG_SCALE, y=y_dev, sp=plan_sp)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- N > 1: the plan against ONE rank doing the whole step (same kernels, no exchange), before anything is timed
    sp_parity = None
    if world > 1 and not args.no_sp_parity:
        xa = lat_host.to(dev).clone()
        step(0, x=xa)
        sync()
        if rank == 0:
            xb = lat_host.to(dev).clone()
            c0 = eng.context_state(ctx_pos, clip_dev)
            c1 = eng.context_state(ctx_neg, clip_dev)
            step(0, x=xb, cpx=c0, cnx=c1, plan_sp=None)
            torch.cuda.synchronize()
            dlt = (xa - xb).abs()
            upd = (xb - lat_host.to(dev)).abs().mean().item()
            sp_parity = {"what": f"latents after one CFG step: plan {plan} vs the same step on rank 0 alone",
                         "max_abs_diff": dlt.max().item(), "mean_abs_diff": dlt.mean().item(), "mean_abs_update": upd,
                         "ok": bool(dlt.max().item() < 2e-2)}
            print("sp_parity " + json.dumps(sp_parity), file=sys.stderr, flush=True)
            del xb, c0, c1
        sync()

    # the models are built: move every live Python object to the permanent generation so that a cyclic-GC pass triggered inside a
    # timed loop has (almost) nothing to traverse.  A full collection over the module trees is a host stall of tens of ms that the
    # e2e leg (one synchronisation per step) cannot hide; whether that is what made one e2e step in three 22 ms longer
    # (profiles/r02_f2_e2e_steps.txt) was not measured — this is hygiene, the per-step wall times stay on stderr
    import gc
    gc.collect()
    gc.freeze()
    for i in range(args.warmup):
        step(i)
    sync()
    eng.attn_events = []      # (start, end) CUDA events around every self-attention launch (roofline leg); forces the eager path
    launches0 = eng.k.launches
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        step(args.warmup + i)
    e1.record()
    sync()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        # taken before anything else runs a step: the steps below reuse lat, v_c and v_u.  The latents are replicated on every
        # rank; v_c / v_u hold the full velocity fields only on one GPU.  Largest workload (cfg3): 3 x 19.4 MB.
        outs = {"latents": lat}
        if world == 1:
            outs.update(velocity_cond=v_c, velocity_uncond=v_u)
        if rank == 0:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, t in outs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), t.float().cpu().numpy())
        sync()
    ms = e0.elapsed_time(e1)
    launches = eng.k.launches - launches0
    attn_ms = [a.elapsed_time(b) for a, b in eng.attn_events]
    eng.attn_events = None
    # CPU time to ENQUEUE one step, measured on an empty launch queue (inside the timed loop the CPU runs ahead until the
    # driver's queue is full and then only measures back-pressure): must stay well below ms_per_step or the job is
    # launch-bound
    host_t0 = time.perf_counter()
    step(args.warmup + args.steps)
    host_ms = (time.perf_counter() - host_t0) * 1e3
    sync()
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    ms_per_step = ms / args.steps
    value = f / (CLIP_STEPS * ms_per_step / 1e3)
    n_ctx = ctx_len
    flops_step = 2 * flops.dit_forward_flops(cfg, L, n_ctx)

    # ---- e2e leg: the same pipeline step with HOST buffers: every step copies the latents and the prompt embeddings a rank
    # needs from pinned host memory (prompt re-projection included) and reads the updated latents back; max over ranks.
    e2e = None
    if not args.no_e2e:
        out_host = torch.empty_like(lat_host).pin_memory()
        lat_h = lat_host.clone().pin_memory()

        hbuf = [lat_h, out_host]      # this step's input / output host buffers; the output is the next step's input

        def e2e_step(i):
            x = hbuf[0].to(dev, non_blocking=True)
            cpx = eng.context_state(ctx_pos_host.to(dev, non_blocking=True), clip_dev) if own0 else None
            cnx = eng.context_state(ctx_neg_host.to(dev, non_blocking=True), clip_dev) if own1 else pipe.OTHER_RANK
            step(i, x=x, cpx=cpx, cnx=cnx)
            hbuf[1].copy_(x, non_blocking=True)
            torch.cuda.current_stream().synchronize()     # the caller consumes the host result every step
            hbuf.reverse()

        # warm-up: every e2e step builds two fresh ContextStates (94 MB of K|V each); the engine keeps the last 8 alive, so the
        # caching allocator only stops calling cudaMalloc (~20 ms per block) once 9 have been built — 5 steps where a rank
        # owns both guidance branches, 10 where the plan gives it one (r02 N=8: 5 warm-up steps left 22 ms of cudaMalloc in
        # every timed e2e step)
        for i in range(max(5 if (own0 and own1) else 10, args.warmup)):
            e2e_step(i)
        sync()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step_wall = []
        for i in range(args.steps):
            t_w = time.perf_counter()
            e2e_step(i)
            step_wall.append(1e3 * (time.perf_counter() - t_w))
        b.record()
        sync()
        e2e_ms = a.elapsed_time(b) / args.steps
        if rank == 0:
            print("e2e step wall times (ms): " + " ".join(f"{t:.1f}" for t in step_wall), file=sys.stderr, flush=True)
        if world > 1:
            tt = torch.tensor([e2e_ms], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            e2e_ms = tt.item()
        # how much of an e2e step is the per-step prompt work (H2D of the embeddings + text MLP + every layer's K|V projection)
        ca, cb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ca.record()
        for _ in range(3):
            eng.context_state(ctx_pos_host.to(dev, non_blocking=True), clip_dev)
        cb.record()
        torch.cuda.synchronize()
        ctx_ms = ca.elapsed_time(cb) / 3
        # one more e2e step with its phases bracketed (stderr): where the e2e - value difference goes
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        t_h0 = time.perf_counter()
        evs[0].record()
        xx = hbuf[0].to(dev, non_blocking=True)
        evs[1].record()
        prof = None
        if os.environ.get("SVI_BENCH_PROFILE") == "1":
            import cProfile
            prof = cProfile.Profile()
            prof.enable()
        cpx = eng.context_state(ctx_pos_host.to(dev, non_blocking=True), clip_dev) if own0 else None
        cnx = eng.context_state(ctx_neg_host.to(dev, non_blocking=True), clip_dev) if own1 else pipe.OTHER_RANK
        if prof is not None:
            import pstats
            prof.disable()
            pstats.Stats(prof, stream=sys.stderr).sort_stats("cumulative").print_stats(18)
        t_h1 = time.perf_counter()
        evs[2].record()
        step(0, x=xx, cpx=cpx, cnx=cnx)
        evs[3].record()
        hbuf[1].copy_(xx, non_blocking=True)
        evs[4].record()
        torch.cuda.synchronize()
        if rank == 0:
            print(f"e2e phases (ms): h2d latents {evs[0].elapsed_time(evs[1]):.2f} | prompt h2d + context_state {evs[1].elapsed_time(evs[2]):.2f} "
                  f"(host {1e3 * (t_h1 - t_h0):.2f}) | step {evs[2].elapsed_time(evs[3]):.2f} | d2h {evs[3].elapsed_time(evs[4]):.2f}",
                  file=sys.stderr, flush=True)
        h2d = lat_host.numel() * 4 + (int(own0) + int(own1)) * ctx_pos_host.numel() * 4
        e2e = {"value": f / (CLIP_STEPS * e2e_ms / 1e3), "unit": "latent_frames/s", "ms_per_step": e2e_ms,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": lat_host.numel() * 4, "context_state_ms_per_prompt": ctx_ms,
               "api": "SVIVideoPipeline.denoise_step (WanDiTEngine.context_state + the plan's forwards + svi_cfg_euler_step), "
                      "pinned host buffers per rank",
               "mode": "CUDA-graph replay of each forward" if eng.use_graphs else "eager"}

    if args.breakdown and rank == 0:
        eng.k.events = []
    if args.breakdown:
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record()
        step(0)
        b1.record()
        sync()
        if rank == 0:
            bd = eng.k.breakdown()
            tot = b0.elapsed_time(b1)
            print(f"breakdown of one step on rank 0, plan {plan} ({tot:.1f} ms wall, {sum(v[0] for v in bd.values()):.1f} ms inside "
                  f"kernel brackets; the rest = exchanges / collectives / gaps)", file=sys.stderr)
            for tag, (ms_, n) in sorted(bd.items(), key=lambda kv: -kv[1][0]):
                print(f"  {ms_:9.2f} ms {100 * ms_ / tot:6.2f}%  n={n:4d}  avg={1e3 * ms_ / n:9.1f} us  {tag}", file=sys.stderr)

    # ---- clip leg (SURVEY.md §8d: "for cfg-4, end-to-end clips/hour with VAE included"): the VAE work one SVI clip adds
    # around the 50 denoising steps — encode of the 81-frame conditioning video and decode of the 21 denoised latent frames.
    clip = None
    if not args.no_vae and world == 1 and args.workload == "cfg2":
        clip = vae_clip_leg(dev, f, h, w, ms_per_step)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks, peak, peak_src = load_peaks()
    Ll = L if sp is None else sp.local_rows(L)
    attn_flops = flops.self_attention_flops(cfg, Ll, L)       # algorithmic FLOPs of one self-attention launch (4 L_q L_k d)
    roof = None
    if attn_ms:
        a_ms = sum(attn_ms) / len(attn_ms)
        ach = attn_flops / (a_ms * 1e-3) / 1e12
        traffic = None   # DRAM bytes per launch from the committed ncu --set full capture (single-GPU shape only)
        tpath = os.path.join(ROOT, "profiles", "attn_traffic.json")
        if sp is None and args.workload == "cfg2" and os.path.exists(tpath):
            traffic = json.load(open(tpath)).get("bytes_per_launch")
        roof = {"kernel": "attn_fwd_kernel (self-attention)", "bound": "tensor", "achieved": ach, "peak": peak,
                "unit": "TFLOP/s", "frac": ach / peak, "traffic": traffic, "peak_source": peak_src,
                "launches_timed": len(attn_ms), "avg_ms": a_ms,
                "share_of_step": sum(attn_ms) / ms}
    line = {"metric": METRIC, "value": value, "unit": "latent_frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": args.workload, "description": desc, "tokens": L, "text_tokens": ctx_len,
                       "cfg_scale": CFG_SCALE, "clip_steps": CLIP_STEPS, "parallelism": plan,
                       "kv_exchange": None if sp is None or sp.sp_size == 1 else
                       ("NVLink peer push (copy engine) consumed by flag-gated attention" if sp._peer is not None else "NCCL all-gather"),
                       "l2_policy": "inputs larger than L2 (weights + activations of a step >> 126 MB)",
                       "numerics": "bf16 operands (two-term bf16 for the embedding / patch / head GEMMs), fp32 accumulate/residual/norm/softmax",
                       "lora_merged_layers": getattr(model, "lora_merged", 0)},
            "timed_mode": "eager launches + CUDA events around every self-attention launch (roofline leg)",
            "api": "SVIVideoPipeline.denoise_step",
            "dit_tflops": flops_step / (ms_per_step * 1e-3) / 1e12,
            "dit_tflops_frac_of_peak": flops_step / (ms_per_step * 1e-3) / 1e12 / (peak * world),
            "gpu_launches": launches, "host_enqueue_ms_per_step": host_ms, "clocks": clocks, "roofline": roof, "e2e": e2e, "clip": clip}
    if sp_parity is not None:
        line["sp_parity"] = sp_parity
    if not args.no_cpu_baseline and world == 1 and cfg["dim"] <= 2048:
        grid = (f, h // 2, w // 2)
        t_blk, cores, fixture, ref = cpu_block_baseline(cfg, L, ctx_len, grid)
        step_s = t_blk * cfg["num_layers"] * 2
        line["cpu_baseline"] = {"value": f / (CLIP_STEPS * step_s), "unit": "latent_frames/s", "cores": cores, "kind": "port",
                                "host_cpu": host_cpu(),
                                "sample": f"1 DiT block forward at L={L} ({t_blk:.2f} s fp32), extrapolated x{cfg['num_layers']} blocks x2 CFG forwards x{CLIP_STEPS} steps"}
        del model, eng, pipe
        torch.cuda.empty_cache()
        line["parity"] = native_block_parity(fixture, ref, grid, dev)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
