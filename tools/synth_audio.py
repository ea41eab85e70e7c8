"""Deterministic synthetic wav2vec2 weights, configs and waveforms (transformers' key names, config.json fields).

Shared by tests/golden/make_golden_wav2vec.py, the tests and tools/audio_bench.py.  W2V_BASE has the shapes of
chinese-wav2vec2-base (the model SVI-Talk loads, reference svi_video_talk.py:26-30); W2V_TINY keeps the kernel / stride
pattern of the conv stack and the group-norm / post-LN variant at a size the CPU runs in milliseconds.
"""
import json
import os

import numpy as np
import torch

_COMMON = dict(conv_kernel=[10, 3, 3, 3, 3, 2, 2], conv_stride=[5, 2, 2, 2, 2, 2, 2], layer_norm_eps=1e-5,
               feat_extract_norm="group", do_stable_layer_norm=False, conv_bias=False, hidden_act="gelu",
               feat_extract_activation="gelu", model_type="wav2vec2", architectures=["Wav2Vec2Model"])
W2V_TINY = dict(_COMMON, hidden_size=64, num_hidden_layers=2, num_attention_heads=4, intermediate_size=128,
                conv_dim=[32] * 7, num_conv_pos_embeddings=16, num_conv_pos_embedding_groups=4)
W2V_BASE = dict(_COMMON, hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072,
                conv_dim=[512] * 7, num_conv_pos_embeddings=128, num_conv_pos_embedding_groups=16)
PREPROCESSOR = dict(do_normalize=True, feature_extractor_type="Wav2Vec2FeatureExtractor", feature_size=1,
                    padding_side="right", padding_value=0.0, return_attention_mask=False, sampling_rate=16000)


def param_shapes(cfg):
    C, D, I = cfg["conv_dim"], cfg["hidden_size"], cfg["intermediate_size"]
    sh = {}
    cin = 1
    for i, (c, k) in enumerate(zip(C, cfg["conv_kernel"])):
        sh[f"feature_extractor.conv_layers.{i}.conv.weight"] = (c, cin, k)
        cin = c
    sh["feature_extractor.conv_layers.0.layer_norm.weight"] = (C[0],)
    sh["feature_extractor.conv_layers.0.layer_norm.bias"] = (C[0],)
    sh["feature_projection.layer_norm.weight"] = (C[-1],)
    sh["feature_projection.layer_norm.bias"] = (C[-1],)
    sh["feature_projection.projection.weight"] = (D, C[-1])
    sh["feature_projection.projection.bias"] = (D,)
    k, g = cfg["num_conv_pos_embeddings"], cfg["num_conv_pos_embedding_groups"]
    sh["encoder.pos_conv_embed.conv.weight_g"] = (1, 1, k)
    sh["encoder.pos_conv_embed.conv.weight_v"] = (D, D // g, k)
    sh["encoder.pos_conv_embed.conv.bias"] = (D,)
    sh["encoder.layer_norm.weight"] = (D,)
    sh["encoder.layer_norm.bias"] = (D,)
    for l in range(cfg["num_hidden_layers"]):
        p = f"encoder.layers.{l}."
        for n in ("q_proj", "k_proj", "v_proj", "out_proj"):
            sh[p + f"attention.{n}.weight"] = (D, D)
            sh[p + f"attention.{n}.bias"] = (D,)
        sh[p + "feed_forward.intermediate_dense.weight"] = (I, D)
        sh[p + "feed_forward.intermediate_dense.bias"] = (I,)
        sh[p + "feed_forward.output_dense.weight"] = (D, I)
        sh[p + "feed_forward.output_dense.bias"] = (D,)
        for n in ("layer_norm", "final_layer_norm"):
            sh[p + n + ".weight"] = (D,)
            sh[p + n + ".bias"] = (D,)
    return sh


def make_state_dict(cfg, seed=0):
    """fp32 weights of roughly unit-variance activations: fan-in scaled matrices, norms around 1, small biases."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for name, shape in param_shapes(cfg).items():
        if name.endswith("weight_g"):
            t = 1.0 + 0.5 * torch.rand(shape, generator=g)
        elif "norm" in name and name.endswith(".weight"):
            t = 1.0 + 0.1 * torch.randn(shape, generator=g)
        elif name.endswith(".bias"):
            t = 0.05 * torch.randn(shape, generator=g)
        else:
            fan_in = int(np.prod(shape[1:]))
            t = torch.randn(shape, generator=g) / fan_in ** 0.5
        sd[name] = t.float()
    return sd


def make_waveform(seconds, sr=16000, seed=0, gain=0.3):
    """Speech-like test signal: a few harmonics with a slow pitch and amplitude drift plus noise, float32 in [-1, 1]."""
    rng = np.random.default_rng(seed)
    n = int(round(seconds * sr))
    t = np.arange(n) / sr
    f0 = 140 + 30 * np.sin(2 * np.pi * 0.7 * t)
    ph = 2 * np.pi * np.cumsum(f0) / sr
    x = sum(np.sin(h * ph) / h for h in range(1, 6)) * (0.6 + 0.4 * np.sin(2 * np.pi * 2.3 * t))
    x = x + 0.05 * rng.standard_normal(n)
    return (gain * x / np.abs(x).max()).astype(np.float32)


def write_model_dir(path, cfg, sd, spelling="weight_g", prefix="", extra=None, fmt="safetensors"):
    """A checkpoint directory as the hub ships it: config.json, preprocessor_config.json and the weights.
    spelling: "weight_g" (weight_g / weight_v) or "parametrizations" (parametrizations.weight.original0 / original1)."""
    os.makedirs(path, exist_ok=True)
    with open(os.path.join(path, "config.json"), "w") as f:
        json.dump(cfg, f)
    with open(os.path.join(path, "preprocessor_config.json"), "w") as f:
        json.dump(PREPROCESSOR, f)
    out = {}
    for k, v in sd.items():
        if spelling == "parametrizations":
            k = k.replace("conv.weight_g", "conv.parametrizations.weight.original0").replace(
                "conv.weight_v", "conv.parametrizations.weight.original1")
        out[prefix + k] = v.contiguous()
    out.update(extra or {})
    if fmt == "safetensors":
        from safetensors.torch import save_file
        save_file(out, os.path.join(path, "model.safetensors"))
    else:
        torch.save(out, os.path.join(path, "pytorch_model.bin"))
    return path
