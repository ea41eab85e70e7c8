"""Generate tests/golden/wav2vec_tiny.npz by running the REAL reference audio path on CPU.

Runs the reference's own Wav2Vec2Model subclass (utils/src/audio_analysis/wav2vec2.py) and get_embedding
(utils/audio_process.py:18-41) with transformers' Wav2Vec2FeatureExtractor(do_normalize=True) on a tiny seeded config
(tools/synth_audio.py W2V_TINY).  Needs the reference tree and transformers, so it runs only where both exist; its output
is committed and pins oracle/wav2vec2_oracle.py (tests/test_oracle_audio_golden.py).

Import recipe: transformers is imported before librosa / pyloudnorm are stubbed (it probes them with find_spec, so the
stubs carry a __spec__), and the config asks for eager attention (the subclass sets output_attentions, which sdpa
refuses).

usage:  python tests/golden/make_golden_wav2vec.py [--ref /root/reference]
"""
import argparse
import importlib
import importlib.machinery
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from tools import synth_audio as SA  # noqa: E402


def golden_wav2vec(ref_root):
    import transformers
    for name in ("librosa", "pyloudnorm"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.__spec__ = importlib.machinery.ModuleSpec(name, None)
            sys.modules[name] = m
    if ref_root not in sys.path:
        sys.path.insert(0, ref_root)
    w2v = importlib.import_module("utils.src.audio_analysis.wav2vec2")
    ap = importlib.import_module("utils.audio_process")
    cfg = SA.W2V_TINY
    keys = ("hidden_size", "num_hidden_layers", "num_attention_heads", "intermediate_size", "conv_dim", "conv_kernel",
            "conv_stride", "num_conv_pos_embeddings", "num_conv_pos_embedding_groups", "layer_norm_eps",
            "feat_extract_norm", "do_stable_layer_norm", "conv_bias", "hidden_act", "feat_extract_activation")
    hf_cfg = transformers.Wav2Vec2Config(attn_implementation="eager", **{k: cfg[k] for k in keys})
    model = w2v.Wav2Vec2Model(hf_cfg).eval()
    sd = SA.make_state_dict(cfg, seed=0)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and all(k == "masked_spec_embed" for k in missing), (missing, unexpected)
    fe = transformers.Wav2Vec2FeatureExtractor(do_normalize=True)
    speech = SA.make_waveform(2.0077, seed=1)            # non-integer frame count: int() truncation + interpolation
    with torch.no_grad():
        emb = ap.get_embedding(speech, fe, model)
        iv = torch.from_numpy(np.squeeze(fe(speech, sampling_rate=16000).input_values)).float()[None]
        conv = model.feature_extractor(iv)[0].T
        hs = model(iv, seq_len=int(len(speech) / 16000 * 25), output_hidden_states=True).hidden_states

    # the window cut of the reference pipeline (svi_video_talk.py:412-430) at the start and past the end of the audio
    def cut(start, n):
        idx = torch.clamp(torch.arange(start, start + n)[:, None] + (torch.arange(5) - 2)[None], 0, emb.shape[0] - 1)
        return emb[idx][None]

    res = dict(speech=speech, input_values=iv[0].numpy(), conv=conv.numpy(), hidden=torch.stack(hs).numpy(), emb=emb.numpy(),
               cut0=cut(0, 13).numpy(), cut_end=cut(emb.shape[0] - 6, 13).numpy(), cut_end_start=np.array(emb.shape[0] - 6))
    np.savez_compressed(os.path.join(HERE, "wav2vec_tiny.npz"), **res)
    print("wav2vec: emb", tuple(emb.shape), "conv", tuple(conv.shape))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref", default="/root/reference")
    a = ap.parse_args()
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count())
    golden_wav2vec(a.ref)
