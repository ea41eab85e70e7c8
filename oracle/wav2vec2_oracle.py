"""CPU torch-fp32 restatement of SVI-Talk's audio feature path, the ground truth of the native wav2vec2 encoder.

Restates (does not import):
  - transformers' Wav2Vec2FeatureExtractor with do_normalize: (x - mean) / sqrt(var + 1e-7) over the whole waveform;
  - the reference's Wav2Vec2Model.forward (utils/src/audio_analysis/wav2vec2.py:13-64) on transformers'
    modeling_wav2vec2 for the configuration the shipped chinese-wav2vec2-base uses (feat_extract_norm="group",
    do_stable_layer_norm=False, conv_bias=False, hidden_act="gelu"): Wav2Vec2FeatureEncoder (GroupNorm on the first conv
    only), linear_interpolation (torch_utils.py:16-19), Wav2Vec2FeatureProjection, Wav2Vec2PositionalConvEmbedding
    (weight norm over dims 0, 1 for each tap, SamePad), Wav2Vec2Encoder with post-LN Wav2Vec2EncoderLayer;
  - get_embedding (utils/audio_process.py:18-41): hidden_states[1:] stacked to [S, layers, hidden];
  - the window cut of SVITalkVideoPipeline.get_audio_embedding (svi_video_talk.py:412-430).

`sd` is a state dict with transformers' key names (no `wav2vec2.` prefix), `cfg` a dict with the config.json fields used.
"""
import numpy as np
import torch
import torch.nn.functional as F


def feature_normalize(x):
    """Wav2Vec2FeatureExtractor(do_normalize=True)(x).input_values[0] for one float waveform."""
    x = np.asarray(x, dtype=np.float32)
    return (x - x.mean()) / np.sqrt(x.var() + 1e-7)


def pos_conv_weight(sd):
    """weight_norm(dim=2) of the positional conv: w = g * v / ||v||, the norm over dims 0, 1 for each tap."""
    p = "encoder.pos_conv_embed.conv."
    g, v = sd[p + "weight_g"].float(), sd[p + "weight_v"].float()
    return g * v / v.norm(dim=(0, 1), keepdim=True)


def conv_stack(sd, cfg, x):
    """Wav2Vec2FeatureEncoder: x f32 [n] -> [T50, conv_dim[-1]] (GroupNorm + GELU on conv 0, GELU on the rest)."""
    h = x.float().reshape(1, 1, -1)
    for i, s in enumerate(cfg["conv_stride"]):
        p = f"feature_extractor.conv_layers.{i}."
        h = F.conv1d(h, sd[p + "conv.weight"].float(), stride=s)
        if i == 0:
            h = F.group_norm(h, h.shape[1], sd[p + "layer_norm.weight"].float(), sd[p + "layer_norm.bias"].float(), eps=1e-5)
        h = F.gelu(h)
    return h[0].T


def encoder_layer(sd, cfg, l, x):
    """Post-LN Wav2Vec2EncoderLayer on x [S, D]."""
    p = f"encoder.layers.{l}."
    lin = lambda t, n: F.linear(t, sd[p + n + ".weight"].float(), sd[p + n + ".bias"].float())
    ln = lambda t, n: F.layer_norm(t, t.shape[-1:], sd[p + n + ".weight"].float(), sd[p + n + ".bias"].float(),
                                   cfg["layer_norm_eps"])
    S, D = x.shape
    H = cfg["num_attention_heads"]
    hd = D // H
    q = (lin(x, "attention.q_proj") * hd ** -0.5).reshape(S, H, hd).transpose(0, 1)
    k = lin(x, "attention.k_proj").reshape(S, H, hd).transpose(0, 1)
    v = lin(x, "attention.v_proj").reshape(S, H, hd).transpose(0, 1)
    a = torch.softmax(q @ k.transpose(1, 2), dim=-1) @ v
    x = ln(x + lin(a.transpose(0, 1).reshape(S, D), "attention.out_proj"), "layer_norm")
    x = x + lin(F.gelu(lin(x, "feed_forward.intermediate_dense")), "feed_forward.output_dense")
    return ln(x, "final_layer_norm")


def encode(sd, cfg, feats, seq_len):
    """conv features [T50, C] -> the num_hidden_layers + 1 hidden states [S, D] (Wav2Vec2Model.forward past the
    feature encoder, output_hidden_states=True)."""
    f = F.interpolate(feats.T[None], size=seq_len, mode="linear", align_corners=True)[0].T
    eps = cfg["layer_norm_eps"]
    f = F.layer_norm(f, f.shape[-1:], sd["feature_projection.layer_norm.weight"].float(),
                     sd["feature_projection.layer_norm.bias"].float(), eps)
    h = F.linear(f, sd["feature_projection.projection.weight"].float(), sd["feature_projection.projection.bias"].float())
    k = cfg["num_conv_pos_embeddings"]
    pos = F.conv1d(h.T[None], pos_conv_weight(sd), sd["encoder.pos_conv_embed.conv.bias"].float(), padding=k // 2,
                   groups=cfg["num_conv_pos_embedding_groups"])
    if k % 2 == 0:
        pos = pos[:, :, :-1]
    h = h + F.gelu(pos)[0].T
    h = F.layer_norm(h, h.shape[-1:], sd["encoder.layer_norm.weight"].float(), sd["encoder.layer_norm.bias"].float(), eps)
    states = [h]
    for l in range(cfg["num_hidden_layers"]):
        h = encoder_layer(sd, cfg, l, h)
        states.append(h)
    return states


def seq_len_of(n_samples, sr=16000):
    """int(len / sr * 25): the 25 fps video length get_embedding asks for (audio_process.py:19-20, 31)."""
    return int(n_samples / sr * 25)


@torch.no_grad()
def get_embedding(speech, sd, cfg, sr=16000):
    """audio_process.py:18-41: waveform -> [S, num_hidden_layers, D] f32 (hidden_states[1:] stacked)."""
    x = torch.from_numpy(feature_normalize(speech))
    states = encode(sd, cfg, conv_stack(sd, cfg, x), seq_len_of(len(speech), sr))
    return torch.stack(states[1:], dim=1)


def cut_windows(emb, num_frames, audio_start_idx=0):
    """svi_video_talk.py:412-430: [S, L, D] -> [1, num_frames, 5, L, D], window centre audio_start_idx + i, indices clamped
    to [0, S - 1]."""
    idx = torch.arange(audio_start_idx, audio_start_idx + num_frames)[:, None] + (torch.arange(5) - 2)[None]
    idx = idx.clamp(0, emb.shape[0] - 1)
    return emb[idx][None]

