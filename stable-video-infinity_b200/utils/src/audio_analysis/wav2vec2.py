"""wav2vec2 audio encoder of SVI-Talk on the native kernels (reference utils/src/audio_analysis/wav2vec2.py, a subclass of
transformers' Wav2Vec2Model whose forward interpolates the 50 Hz conv features to `seq_len` video frames).

`Wav2Vec2Model` is a parameter container with transformers' key names (`from_pretrained` reads a hub checkpoint
directory without transformers); its `engine(device)` runs the forward on the GPU:

    waveform --svi_audio_conv0_gn_gelu--> bf16 [T0, 512]             conv 1->512 k10 s5, GroupNorm(512), GELU
             --svi_gemm_bf16 x6 (strided views)--> f32 [T50, 512]     convs k3 s2 (x4), k2 s2 (x2), GELU epilogue
             --svi_audio_interp_layernorm--> bf16 [S, 512]            50 Hz -> 25 Hz, feature-projection LayerNorm
             --svi_gemm_bf16--> f32 [S, 768] --svi_audio_pos_conv-->   projection; + GELU(grouped pos conv)
             --svi_layernorm_f32x2--> 12 x post-LN layers (svi_gemm_bf16, svi_attn_small, svi_layernorm_f32x2)

A convolution with kernel k and stride s over channels-last activations x [T, C] is a GEMM whose A row t is the k*C
contiguous elements from t*s*C, i.e. a view with leading dimension s*C.  For k = 2 = s the rows tile x exactly.  For k = 3,
s = 2 neighbouring rows would overlap (lda < K), which a TMA tensor map cannot describe (its row pitch must cover the row),
so the conv runs as taps {0, 1} (lda = K = 2C) into fp32, then tap 2 (base x + 2C, lda 2C, K = C) accumulated on top
through the residual epilogue, then GELU to bf16.

Only the configuration chinese-wav2vec2-base uses is implemented: feat_extract_norm="group", do_stable_layer_norm=False,
conv_bias=False, hidden_act="gelu".  Anything else raises.
"""
import json
import os
import types

import numpy as np
import torch
import torch.nn as nn

from diffsynth import _native as nv

_PRETRAIN_ONLY = ("quantizer.", "project_q.", "project_hid.", "masked_spec_embed")
_REQUIRED = dict(feat_extract_norm="group", do_stable_layer_norm=False, conv_bias=False, hidden_act="gelu")


def check_config(cfg):
    for k, want in _REQUIRED.items():
        got = cfg.get(k, want)
        if got != want:
            raise ValueError(f"svi_b200 wav2vec2: {k}={got!r} is not supported (only {k}={want!r}, the chinese-wav2vec2-base "
                             f"configuration, is implemented)")
    if cfg.get("feat_extract_activation", "gelu") != "gelu":
        raise ValueError("svi_b200 wav2vec2: only feat_extract_activation='gelu' is supported")
    if len(cfg["conv_dim"]) != len(cfg["conv_kernel"]) or len(cfg["conv_dim"]) != len(cfg["conv_stride"]):
        raise ValueError("svi_b200 wav2vec2: conv_dim / conv_kernel / conv_stride lengths differ")
    for i, (k, s) in enumerate(zip(cfg["conv_kernel"][1:], cfg["conv_stride"][1:])):
        if (k, s) not in ((2, 2), (3, 2)):
            raise ValueError(f"svi_b200 wav2vec2: conv {i + 1} has kernel {k} stride {s}; only (2, 2) and (3, 2) are implemented")


def _lin(i, o):
    return nn.Linear(i, o)


class _ConvLayer(nn.Module):
    def __init__(self, cin, cout, k, norm):
        super().__init__()
        self.conv = nn.Conv1d(cin, cout, k, bias=False)
        if norm:
            self.layer_norm = nn.GroupNorm(cout, cout, affine=True)


class _PosConv(nn.Module):
    def __init__(self, D, k, g):
        super().__init__()
        self.conv = nn.Module()
        self.conv.weight_g = nn.Parameter(torch.ones(1, 1, k))
        self.conv.weight_v = nn.Parameter(torch.zeros(D, D // g, k))
        self.conv.bias = nn.Parameter(torch.zeros(D))


class _Layer(nn.Module):
    def __init__(self, D, I):
        super().__init__()
        self.attention = nn.Module()
        for n in ("q_proj", "k_proj", "v_proj", "out_proj"):
            setattr(self.attention, n, _lin(D, D))
        self.layer_norm = nn.LayerNorm(D)
        self.feed_forward = nn.Module()
        self.feed_forward.intermediate_dense = _lin(D, I)
        self.feed_forward.output_dense = _lin(I, D)
        self.final_layer_norm = nn.LayerNorm(D)


def convert_state_dict(sd):
    """Hub checkpoint -> this container's keys: strip a `wav2vec2.` prefix, drop pre-training-only tensors (quantizer,
    project_q / project_hid, masked_spec_embed) and anything outside the base model (e.g. a CTC `lm_head`), map the
    parametrizations spelling of the positional conv's weight norm to weight_g / weight_v."""
    out = {}
    for k, v in sd.items():
        if k.startswith("wav2vec2."):
            k = k[len("wav2vec2."):]
        elif not k.startswith(("feature_extractor.", "feature_projection.", "encoder.")):
            continue
        if k.startswith(_PRETRAIN_ONLY):
            continue
        k = k.replace("conv.parametrizations.weight.original0", "conv.weight_g").replace(
            "conv.parametrizations.weight.original1", "conv.weight_v")
        out[k] = v
    return out


class Wav2Vec2Model(nn.Module):
    """Parameter container with transformers' names (feature_extractor / feature_projection / encoder)."""

    def __init__(self, config):
        super().__init__()
        check_config(config)
        self.config = types.SimpleNamespace(**config)
        C, K = config["conv_dim"], config["conv_kernel"]
        D, I = config["hidden_size"], config["intermediate_size"]
        self.feature_extractor = nn.Module()
        self.feature_extractor.conv_layers = nn.ModuleList(
            [_ConvLayer(1 if i == 0 else C[i - 1], C[i], K[i], i == 0) for i in range(len(C))])
        self.feature_projection = nn.Module()
        self.feature_projection.layer_norm = nn.LayerNorm(C[-1])
        self.feature_projection.projection = _lin(C[-1], D)
        self.encoder = nn.Module()
        self.encoder.pos_conv_embed = _PosConv(D, config["num_conv_pos_embeddings"], config["num_conv_pos_embedding_groups"])
        self.encoder.layer_norm = nn.LayerNorm(D)
        self.encoder.layers = nn.ModuleList([_Layer(D, I) for _ in range(config["num_hidden_layers"])])
        self._engine = None

    @classmethod
    def from_pretrained(cls, path, local_files_only=True):
        """Read config.json and model.safetensors or pytorch_model.bin (weights_only) from a checkpoint directory."""
        path = os.fspath(path)
        if not os.path.isdir(path):
            raise FileNotFoundError(f"wav2vec2 checkpoint directory not found: {path}")
        with open(os.path.join(path, "config.json")) as f:
            cfg = json.load(f)
        st, pt = os.path.join(path, "model.safetensors"), os.path.join(path, "pytorch_model.bin")
        if os.path.exists(st):
            from safetensors.torch import load_file
            sd = load_file(st)
        elif os.path.exists(pt):
            sd = torch.load(pt, map_location="cpu", weights_only=True)
        else:
            raise FileNotFoundError(f"no model.safetensors or pytorch_model.bin in {path}")
        model = cls(cfg)
        model.load_state_dict({k: v.float() for k, v in convert_state_dict(sd).items()})
        return model.eval()

    def engine(self, device=None):
        p = self.encoder.layers[-1].final_layer_norm.weight
        dev = torch.device(device) if device is not None else p.device
        if dev.type == "cuda" and dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        sig = (str(dev), p.data_ptr(), p._version, self.feature_extractor.conv_layers[0].conv.weight.data_ptr())
        if self._engine is None or self._engine[0] != sig:
            self._engine = (sig, Wav2Vec2Engine(self, dev))
        return self._engine[1]

    @torch.no_grad()
    def forward(self, input_values, seq_len, output_hidden_states=True, device=None):
        """input_values [1, n] (normalised waveform) -> object with .hidden_states (num_hidden_layers + 1 tensors
        [1, seq_len, hidden]) and .last_hidden_state, as the reference's forward (wav2vec2.py:13-64)."""
        eng = self.engine(device if device is not None else
                          (input_values.device if input_values.is_cuda else torch.device("cuda")))
        x0, out = eng.forward(input_values.reshape(-1), seq_len, keep_first=True)
        states = (x0[None],) + tuple(out[:, l][None] for l in range(out.shape[1]))
        return types.SimpleNamespace(hidden_states=states if output_hidden_states else None,
                                     last_hidden_state=states[-1], attentions=None)


def fold_weight_norm(g, v):
    """weight_norm(dim=2): w = g * v / ||v||, the norm over dims 0, 1 for each tap (host, fp32)."""
    g, v = g.detach().float().cpu(), v.detach().float().cpu()
    return g * v / v.norm(dim=(0, 1), keepdim=True)


class Wav2Vec2Engine:
    def __init__(self, model, device):
        nv.require_cuda(device, "the wav2vec2 audio encoder")
        self.device = torch.device(device)
        c = model.config
        self.cfg = c
        self.eps = float(c.layer_norm_eps)
        bf = lambda t: t.detach().to(device=self.device, dtype=torch.bfloat16).contiguous()
        f32 = lambda t: t.detach().to(device=self.device, dtype=torch.float32).contiguous()
        cl = model.feature_extractor.conv_layers
        self.c0_w = f32(cl[0].conv.weight[:, 0, :])
        self.c0_k, self.c0_s = c.conv_kernel[0], c.conv_stride[0]
        self.c0_g, self.c0_b = f32(cl[0].layer_norm.weight), f32(cl[0].layer_norm.bias)
        self.convs = []
        for i in range(1, len(cl)):
            w = cl[i].conv.weight.detach().float()                        # [O, C, k]
            O_, C_, k = w.shape
            wp = w.permute(0, 2, 1).reshape(O_, k * C_)                   # W[o, j*C + c] = w[o, c, j]
            parts = [bf(wp)] if k == 2 else [bf(wp[:, :2 * C_]), bf(wp[:, 2 * C_:])]
            self.convs.append((k, c.conv_stride[i], C_, O_, parts))
        fp = model.feature_projection
        self.fp_g, self.fp_b = f32(fp.layer_norm.weight), f32(fp.layer_norm.bias)
        self.w_proj, self.b_proj = bf(fp.projection.weight), f32(fp.projection.bias)
        pc = model.encoder.pos_conv_embed.conv
        D, G, K = c.hidden_size, c.num_conv_pos_embedding_groups, c.num_conv_pos_embeddings
        cg = D // G
        w = fold_weight_norm(pc.weight_g, pc.weight_v)                   # [D, cg, K]
        self.pos_w = f32(w.reshape(G, cg, cg, K).permute(0, 3, 2, 1))   # [g][j][c][o]
        self.pos_b, self.pos_groups = f32(pc.bias), G
        self.enc_g, self.enc_b = f32(model.encoder.layer_norm.weight), f32(model.encoder.layer_norm.bias)
        self.layers = []
        for ly in model.encoder.layers:
            a = ly.attention
            self.layers.append(dict(
                w_qkv=bf(torch.cat([a.q_proj.weight, a.k_proj.weight, a.v_proj.weight])),
                b_qkv=f32(torch.cat([a.q_proj.bias, a.k_proj.bias, a.v_proj.bias])),
                w_o=bf(a.out_proj.weight), b_o=f32(a.out_proj.bias), n1g=f32(ly.layer_norm.weight), n1b=f32(ly.layer_norm.bias),
                w_f1=bf(ly.feed_forward.intermediate_dense.weight), b_f1=f32(ly.feed_forward.intermediate_dense.bias),
                w_f2=bf(ly.feed_forward.output_dense.weight), b_f2=f32(ly.feed_forward.output_dense.bias),
                n2g=f32(ly.final_layer_norm.weight), n2b=f32(ly.final_layer_norm.bias)))
        self.D, self.H, self.I = D, c.num_attention_heads, c.intermediate_size
        self.launches = 0
        self._ws = None

    def conv_stack(self, wav):
        """normalised waveform f32 [n] (device) -> f32 [T50, C] (Wav2Vec2FeatureEncoder)."""
        dev = self.device
        wav = wav.to(device=dev, dtype=torch.float32).contiguous()
        C = self.c0_w.shape[0]
        T = (wav.numel() - self.c0_k) // self.c0_s + 1
        if T < 1:
            raise ValueError(f"wav2vec2: {wav.numel()} samples are too short for the first convolution")
        x = torch.empty(T, C, device=dev, dtype=torch.bfloat16)
        self._ws = nv.audio_conv0_gn_gelu(wav, self.c0_w, self.c0_g, self.c0_b, 1e-5, self.c0_s, x, self._ws)
        self.launches += 3
        for idx, (k, s, Ci, Co, parts) in enumerate(self.convs):
            To = (T - k) // s + 1
            if To < 1:
                raise ValueError("wav2vec2: the waveform is too short for the convolution stack")
            last = idx == len(self.convs) - 1
            flat = x.view(-1)
            if k == 2:
                y = torch.empty(To, Co, device=dev, dtype=torch.float32 if last else torch.bfloat16)
                nv.gemm(flat.as_strided((To, 2 * Ci), (s * Ci, 1)), parts[0], y, act=nv.ACT_GELU_ERF)
                self.launches += 1
            else:
                acc = torch.empty(To, Co, device=dev, dtype=torch.float32)
                nv.gemm(flat.as_strided((To, 2 * Ci), (s * Ci, 1)), parts[0], acc)
                nv.gemm(flat[2 * Ci:].as_strided((To, Ci), (s * Ci, 1)), parts[1], acc, residual=acc)
                if last:
                    raise ValueError("wav2vec2: the last convolution must have kernel 2 (fp32 GELU epilogue)")
                y = torch.empty(To, Co, device=dev, dtype=torch.bfloat16)
                nv.cast_f32_to_bf16(acc, y, act=nv.ACT_GELU_ERF)
                self.launches += 3
            x, T = y, To
        return x

    def encode(self, feats, seq_len, keep_first=False):
        """conv features f32 [T50, C] -> [seq_len, num_hidden_layers, D] f32 (hidden_states[1:] stacked, written in place
        by each layer's final LayerNorm); keep_first: also return hidden_states[0]."""
        dev, D, S = self.device, self.D, int(seq_len)
        if S < 1:
            raise ValueError("wav2vec2: seq_len must be >= 1")
        C = feats.shape[1]
        f = torch.empty(S, C, device=dev, dtype=torch.bfloat16)
        nv.audio_interp_layernorm(feats, self.fp_g, self.fp_b, self.eps, f)
        h = torch.empty(S, D, device=dev, dtype=torch.float32)
        nv.gemm(f, self.w_proj, h, bias=self.b_proj)
        h2 = torch.empty_like(h)
        nv.audio_pos_conv(h, self.pos_w, self.pos_b, self.pos_groups, h2)
        x0 = h                                                          # h is free again: hidden_states[0]
        xb = torch.empty(S, D, device=dev, dtype=torch.bfloat16)
        nv.layernorm_f32x2(h2, self.enc_g, self.enc_b, self.eps, x0, xb)
        L = len(self.layers)
        out = torch.empty(S, L, D, device=dev, dtype=torch.float32)
        qkv = torch.empty(S, 3 * D, device=dev, dtype=torch.bfloat16)
        att = torch.empty(S, D, device=dev, dtype=torch.bfloat16)
        m = torch.empty(S, self.I, device=dev, dtype=torch.bfloat16)
        t, x1 = h2, torch.empty(S, D, device=dev, dtype=torch.float32)
        hd = D // self.H
        r = x0
        for l, ly in enumerate(self.layers):
            nv.gemm(xb, ly["w_qkv"], qkv, bias=ly["b_qkv"])
            nv.attention_small(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], att, self.H, hd, hd ** -0.5)
            nv.gemm(att, ly["w_o"], t, bias=ly["b_o"], residual=r)
            nv.layernorm_f32x2(t, ly["n1g"], ly["n1b"], self.eps, x1, xb)
            nv.gemm(xb, ly["w_f1"], m, bias=ly["b_f1"], act=nv.ACT_GELU_ERF)
            nv.gemm(m, ly["w_f2"], t, bias=ly["b_f2"], residual=x1)
            r = out[:, l]
            nv.layernorm_f32x2(t, ly["n2g"], ly["n2b"], self.eps, r, xb)
            self.launches += 7
        self.launches += 4
        return (x0, out) if keep_first else out

    def forward(self, wav, seq_len, keep_first=False):
        return self.encode(self.conv_stack(wav), seq_len, keep_first=keep_first)


class Wav2Vec2FeatureExtractor:
    """transformers' Wav2Vec2FeatureExtractor for one unbatched float waveform: input_values = (x - mean) / sqrt(var + 1e-7)
    when do_normalize (numpy, as transformers computes it), else the waveform as float32."""

    def __init__(self, do_normalize=True, sampling_rate=16000, **_):
        self.do_normalize, self.sampling_rate = bool(do_normalize), int(sampling_rate)

    @classmethod
    def from_pretrained(cls, path, local_files_only=True):
        with open(os.path.join(os.fspath(path), "preprocessor_config.json")) as f:
            return cls(**json.load(f))

    def __call__(self, raw_speech, sampling_rate=None, **_):
        if sampling_rate is not None and sampling_rate != self.sampling_rate:
            raise ValueError(f"the feature extractor expects {self.sampling_rate} Hz audio, got {sampling_rate}")
        x = np.asarray(raw_speech, dtype=np.float32)
        if self.do_normalize:
            x = (x - x.mean()) / np.sqrt(x.var() + 1e-7)
        return types.SimpleNamespace(input_values=[x])
