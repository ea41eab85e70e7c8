"""Algorithmic FLOP / byte counts of the hot path (roofline numerators; multiply-add = 2).  SURVEY.md §8(d) / BASELINE.md §3.
Product-side restatement for bench.py and the measurement tools (the oracle keeps its own copy; tests assert they agree)."""


def dit_block_flops(cfg, L, Lc=512):
    d, ffn = cfg["dim"], cfg["ffn_dim"]
    blk = 8 * L * d * d + 4 * L * L * d + (4 * L * d * d + 4 * Lc * d * d + 4 * L * Lc * d) + 4 * L * d * ffn
    if cfg["has_image_input"]:
        blk += 4 * 257 * d * d + 4 * L * 257 * d
    return blk


def dit_forward_flops(cfg, L, Lc=512):
    d = cfg["dim"]
    pre = 2 * L * (4 * cfg["in_dim"]) * d + 2 * Lc * cfg["text_dim"] * d + 2 * Lc * d * d + 2 * L * d * 64
    return cfg["num_layers"] * dit_block_flops(cfg, L, Lc) + pre


def self_attention_flops(cfg, Lq, Lk):
    return 4.0 * Lq * Lk * cfg["dim"]


def vae_decode_flops(t_lat, h, w):
    """h, w: latent size.  (0.688 + 2.162 (T_lat - 1)) GFLOP per latent position."""
    return (0.688 + 2.162 * (t_lat - 1)) * 1e9 * h * w


def vae_encode_flops(t_lat, H, W):
    """H, W: pixel size.  (6.66 + 5.00 (T_lat - 1)) MFLOP per pixel position."""
    return (6.66 + 5.00 * (t_lat - 1)) * 1e6 * H * W


def vae_min_bytes(t_lat, h, w):
    """Minimal conv in+out traffic (bf16) of the VAE decoder per clip: 8.5 GB per latent frame at 480p (60x104), SURVEY §8d."""
    return 8.5e9 * t_lat * (h * w) / 6240.0


def wav2vec_flops(n_samples, cfg, sr=16000):
    """FLOPs of one wav2vec2 embedding of n_samples (multiply-add = 2), by stage: conv stack, positional conv, GEMMs
    (feature projection + per layer q|k|v, out-projection, feed-forward) and attention (QK^T and PV)."""
    T, cin, conv = n_samples, 1, 0
    for c, k, s in zip(cfg["conv_dim"], cfg["conv_kernel"], cfg["conv_stride"]):
        T = (T - k) // s + 1
        conv += 2 * T * c * cin * k
        cin = c
    S = int(n_samples / sr * 25)
    D, I, L = cfg["hidden_size"], cfg["intermediate_size"], cfg["num_hidden_layers"]
    gemm = 2 * S * cin * D + L * 2 * S * (4 * D * D + 2 * D * I)
    pos = 2 * S * D * (D // cfg["num_conv_pos_embedding_groups"]) * cfg["num_conv_pos_embeddings"]
    attn = L * 4 * S * S * D
    return dict(conv=conv, pos_conv=pos, gemm=gemm, attention=attn)
