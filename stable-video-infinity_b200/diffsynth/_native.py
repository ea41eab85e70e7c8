"""ctypes binding of the C-ABI kernel library ``libsvi_b200.so`` (declared in ``include/svi_b200.h``).

This is the only door between the Python host code and the hand-written sm_100a kernels.  There is no
fallback: if the shared library is missing or a call fails, a ``RuntimeError`` is raised.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# SVI_B200_LIB: another build of the same library (A/B measurements of compiler flags / kernel variants)
_LIB_PATH = os.environ.get("SVI_B200_LIB") or os.path.join(os.path.dirname(_HERE), "lib", "libsvi_b200.so")

ACT_NONE, ACT_GELU_TANH, ACT_SILU, ACT_GELU_ERF, ACT_RELU = 0, 1, 2, 3, 4

_c = ctypes
_vp, _i32, _i64, _f32 = _c.c_void_p, _c.c_int32, _c.c_int64, _c.c_float


class GemmEpilogue(_c.Structure):
    """Mirror of ``svi_gemm_epilogue`` (include/svi_b200.h)."""
    _fields_ = [
        ("out", _vp), ("ldo", _i64), ("out_is_f32", _i32), ("act", _i32),
        ("bias", _vp), ("gate", _vp), ("residual", _vp), ("ldr", _i64),
        ("sumsq", _vp), ("sumsq_groups", _i32), ("sumsq_group_cols", _i32),
        ("ln_stats", _vp), ("ln_u", _vp), ("ln_dim", _i32), ("ln_eps", _f32),
        ("a_next", _vp), ("ld_an", _i64), ("g_next", _vp), ("row_stats", _vp),
        ("sumsq_parts", _i32),
    ]


class ConvDesc(_c.Structure):
    """Mirror of ``svi_conv_desc`` (include/svi_b200.h)."""
    _fields_ = [
        ("x_ring", _vp), ("ring_slots", _i32), ("in_H", _i32), ("in_W", _i32), ("C_in", _i32),
        ("w_packed", _vp), ("w_rows", _i32), ("w_ld", _i64),
        ("kt", _i32), ("kh", _i32), ("kw", _i32), ("pad_h", _i32), ("pad_w", _i32),
        ("H", _i32), ("W", _i32), ("T", _i32),
        ("slot", _i32 * 12),
        ("C_out", _i32), ("tile_w", _i32),
        ("out", _vp), ("out_frame_stride", _i64), ("out_ld", _i32),
        ("n_split", _i32), ("split_offset", _i64),
        ("bias", _vp),
        ("residual", _vp), ("res_frame_stride", _i64), ("res_ld", _i32),
        ("next_ring", _vp), ("next_frame_stride", _i64), ("next_ld", _i32), ("next_slot", _i32 * 4),
        ("next_gamma", _vp), ("next_silu", _i32), ("write_f32", _i32),
        ("variant", _i32),
    ]


# name -> (restype, argtypes); must list every symbol the header declares (checked by tests)
SIGNATURES = {
    "svi_abi_version": (_i32, []),
    "svi_last_error": (_c.c_char_p, []),
    "svi_sm_count": (_i32, []),
    "svi_gemm_bf16": (_i32, [_vp, _i64, _vp, _i64, _i32, _i32, _i32, _c.POINTER(GemmEpilogue), _vp]),
    "svi_attn_fwd": (_i32, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _i32, _i32, _i32, _f32, _i32, _vp, _c.c_size_t, _vp]),
    "svi_attn_workspace_bytes": (_c.c_size_t, [_i32, _i32, _i32]),
    "svi_attn_fwd_qscale": (_i32, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _i32, _i32, _i32, _f32, _i32, _vp, _i32, _i32, _i32, _f32,
                                   _vp, _c.c_size_t, _vp]),
    "svi_attn_plan": (None, [_i32, _i32, _i32, _c.c_size_t, _c.POINTER(_i32), _c.POINTER(_i32)]),
    "svi_attn_fwd_sp": (_i32, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _i32, _i32, _i32, _f32, _vp, _c.c_uint32, _i32, _i32, _vp, _c.c_size_t, _vp]),
    "svi_sp_alloc": (_i32, [_c.c_size_t, _c.POINTER(_vp), _c.c_char_p]),
    "svi_sp_free": (_i32, [_vp]),
    "svi_sp_open": (_i32, [_c.c_char_p, _c.POINTER(_vp)]),
    "svi_sp_close": (_i32, [_vp]),
    "svi_sp_push": (_i32, [_vp, _c.POINTER(_vp), _c.POINTER(_vp), _i32, _c.c_size_t, _vp, _vp]),
    "svi_layernorm_modulate": (_i32, [_vp, _i32, _i32, _f32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "svi_layernorm_modulate_split": (_i32, [_vp, _i32, _i32, _f32, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp]),
    "svi_rmsnorm_rope": (_i32, [_vp, _i64, _i32, _i32, _vp, _i32, _i32, _i32, _f32, _vp, _vp, _vp, _i32, _vp]),
    "svi_qk_norm_rope": (_i32, [_vp, _i64, _i32, _i32, _vp, _i32, _i32, _f32, _vp, _vp, _vp, _vp, _i32, _vp]),
    "svi_patchify_gather_split": (_i32, [_vp, _i32, _vp, _i32, _i32, _i32, _i32, _vp, _i32, _vp]),
    "svi_split_f32_to_bf16x2": (_i32, [_vp, _i64, _i32, _i32, _i32, _vp, _i64, _i32, _vp]),
    "svi_zero": (_i32, [_vp, _c.c_size_t, _vp]),
    "svi_ln_fold_prepare": (_i32, [_vp, _i32, _i32, _vp, _vp, _vp]),
    "svi_ln_fold_combine": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp]),
    "svi_patchify_gather": (_i32, [_vp, _i32, _vp, _i32, _i32, _i32, _i32, _vp, _i32, _vp]),
    "svi_unpatchify": (_i32, [_vp, _i64, _i32, _i32, _i32, _i32, _vp, _vp]),
    "svi_cfg_euler_step": (_i32, [_vp, _vp, _vp, _i64, _f32, _f32, _f32, _vp]),
    "svi_cast_f32_to_bf16": (_i32, [_vp, _vp, _i64, _vp]),
    "svi_cast_bf16_to_f32": (_i32, [_vp, _vp, _i64, _vp]),
    "svi_act_f32_to_bf16": (_i32, [_vp, _vp, _i64, _i32, _vp]),
    "svi_add_rows": (_i32, [_vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "svi_axpby": (_i32, [_vp, _f32, _vp, _f32, _vp, _i64, _vp]),
    "svi_embedding_gather": (_i32, [_vp, _i32, _vp, _i32, _i64, _vp, _vp]),
    "svi_rmsnorm_affine": (_i32, [_vp, _i32, _i32, _f32, _vp, _vp, _vp]),
    "svi_layernorm_f32": (_i32, [_vp, _i32, _i32, _f32, _vp, _vp, _vp, _vp]),
    "svi_mul_bf16": (_i32, [_vp, _vp, _vp, _i64, _vp]),
    "svi_attn_small": (_i32, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _i32, _i32, _i32, _i32, _f32, _vp, _vp, _vp, _vp]),
    "svi_conv3d_causal": (_i32, [_c.POINTER(ConvDesc), _vp]),
    "svi_vae_norm_act": (_i32, [_vp, _i64, _i32, _i64, _vp, _i32, _vp, _i32, _vp]),
    "svi_vae_upsample2x": (_i32, [_vp, _i32, _i32, _i32, _vp, _vp]),
    "svi_vae_space_to_depth": (_i32, [_vp, _i32, _i32, _i32, _vp, _vp]),
    "svi_vae_space_to_depth_act": (_i32, [_vp, _i32, _i32, _i32, _i32, _vp, _vp]),
    "svi_vae_from_planar": (_i32, [_vp, _i32, _i64, _i64, _vp, _vp, _vp, _i32, _i32, _vp]),
    "svi_vae_to_planar": (_i32, [_vp, _i64, _i32, _i64, _vp, _vp, _i32, _vp, _i64, _vp]),
    "svi_softmax_rows": (_i32, [_vp, _i32, _i32, _i64, _f32, _vp, _i64, _vp]),
    "svi_frames_to_uint8": (_i32, [_vp, _i64, _i64, _vp, _vp]),
    "svi_audio_conv0_workspace_bytes": (_c.c_size_t, [_i64, _i32, _i32, _i32]),
    "svi_audio_conv0_gn_gelu": (_i32, [_vp, _i64, _vp, _i32, _i32, _i32, _vp, _vp, _f32, _vp, _vp, _c.c_size_t, _vp]),
    "svi_audio_interp_layernorm": (_i32, [_vp, _i32, _i32, _i32, _vp, _vp, _f32, _vp, _vp]),
    "svi_audio_pos_conv": (_i32, [_vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "svi_layernorm_f32x2": (_i32, [_vp, _i64, _i32, _i32, _f32, _vp, _vp, _vp, _i64, _vp, _vp]),
}

_lib = None


def lib_path():
    return _LIB_PATH


def load():
    """Load the kernel library (once).  Raises RuntimeError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise RuntimeError(
            f"svi_b200: native kernel library not found at {_LIB_PATH}. Build it with "
            f"`python -c 'import __graft_entry__ as g; g.build()'` (or `make`) — there is no CPU fallback.")
    lib = ctypes.CDLL(_LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def require_cuda(device, what):
    """Every engine calls this first: the kernels exist for sm_100a only, so anything but a CUDA device is an error (there is
    no CPU path), and the library must be loadable."""
    if torch.device(device).type != "cuda":
        raise RuntimeError(f"svi_b200: {what} runs only on a CUDA device (sm_100a kernels; no CPU fallback)")
    load()


def _check(rc, name):
    if rc != 0:
        msg = load().svi_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{name} failed (status {rc}): {msg}")


def _stream():
    return _vp(torch.cuda.current_stream().cuda_stream)


def _ptr(t, dtype=None, name="tensor"):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError(f"svi_b200: {name} must be a CUDA tensor (no CPU fallback)")
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError(f"svi_b200: {name} must be {dtype}, got {t.dtype}")
    return _vp(t.data_ptr())


def _rowmajor(t, name):
    if t.dim() != 2 or t.stride(1) != 1:
        raise RuntimeError(f"svi_b200: {name} must be 2-D with unit inner stride, got {tuple(t.shape)} / {t.stride()}")
    return t.stride(0)


def sm_count():
    return load().svi_sm_count()


def gemm(a, w, out, bias=None, act=ACT_NONE, gate=None, residual=None, sumsq=None, sumsq_group_cols=0, ln=None, emit=None):
    """out = epilogue(a[M,K] @ w[N,K]^T); a, w bf16; out f32 or bf16 (may be a column slice view).
    ln = (stats f32 [M,2], u f32 [N], dim, eps): LayerNorm folded into the GEMM (consumer side, svi_gemm_epilogue);
    emit = (a_next bf16 [M,N], g_next f32 [N], row_stats f32 [M,2]): producer side.  Both need M > 128."""
    lda, ldw, ldo = _rowmajor(a, "a"), _rowmajor(w, "w"), _rowmajor(out, "out")
    M, K = a.shape
    N = w.shape[0]
    if w.shape[1] != K or out.shape[0] != M or out.shape[1] != N:
        raise RuntimeError(f"svi_b200.gemm: shape mismatch a{tuple(a.shape)} w{tuple(w.shape)} out{tuple(out.shape)}")
    ep = GemmEpilogue()
    ep.out = _ptr(out, name="out")
    ep.ldo = ldo
    if out.dtype == torch.float32:
        ep.out_is_f32 = 1
    elif out.dtype == torch.bfloat16:
        ep.out_is_f32 = 0
    else:
        raise RuntimeError(f"svi_b200.gemm: out must be f32 or bf16, got {out.dtype}")
    ep.act = act
    ep.bias = _ptr(bias, torch.float32, "bias")
    ep.gate = _ptr(gate, torch.float32, "gate")
    if residual is not None:
        ep.residual = _ptr(residual, torch.float32, "residual")
        ep.ldr = _rowmajor(residual, "residual")
    if sumsq is not None:
        # [M, groups]: atomicAdd per group (the buffer must be zero);  [M, groups, parts] contiguous, parts = group_cols / 128:
        # every 128-column segment stores its partial sum (reproducible, no zeroing) — see svi_gemm_epilogue.sumsq_parts
        ep.sumsq = _ptr(sumsq, torch.float32, "sumsq")
        ep.sumsq_groups = sumsq.shape[1]
        ep.sumsq_group_cols = sumsq_group_cols
        if sumsq.dim() == 3:
            if not sumsq.is_contiguous() or sumsq.shape[2] * 128 != sumsq_group_cols:
                raise RuntimeError("svi_b200.gemm: partial sumsq must be contiguous [M, groups, sumsq_group_cols / 128]")
            ep.sumsq_parts = sumsq.shape[2]
    if ln is not None or emit is not None:
        if M <= 128:
            raise RuntimeError("svi_b200.gemm: the LayerNorm fold runs in the CTA-pair kernel (M > 128)")
    if ln is not None:
        stats, u, dim, eps = ln
        if tuple(stats.shape) != (M, 2) or not stats.is_contiguous() or u.numel() != N:
            raise RuntimeError("svi_b200.gemm: ln stats must be contiguous [M,2] and u [N]")
        ep.ln_stats, ep.ln_u = _ptr(stats, torch.float32, "ln_stats"), _ptr(u, torch.float32, "ln_u")
        ep.ln_dim, ep.ln_eps = int(dim), float(eps)
    if emit is not None:
        a_next, g_next, row_stats = emit
        if a_next.shape[0] != M or a_next.shape[1] != N or tuple(row_stats.shape) != (M, 2) or not row_stats.is_contiguous():
            raise RuntimeError("svi_b200.gemm: emit needs a_next [M,N] and contiguous row_stats [M,2]")
        ep.a_next, ep.ld_an = _ptr(a_next, torch.bfloat16, "a_next"), _rowmajor(a_next, "a_next")
        ep.g_next, ep.row_stats = _ptr(g_next, torch.float32, "g_next"), _ptr(row_stats, torch.float32, "row_stats")
    rc = load().svi_gemm_bf16(_ptr(a, torch.bfloat16, "a"), lda, _ptr(w, torch.bfloat16, "w"), ldw,
                              M, N, K, ctypes.byref(ep), _stream())
    _check(rc, "svi_gemm_bf16")
    return out


def attention(q, k, v, out, num_heads, scale=None, accumulate=False, workspace=None):
    """out[Lq, H*128] (+)= softmax(q k^T * scale) v per head; q,k,v,out bf16 2-D (column-slice views allowed).
    workspace: optional device scratch (attention_workspace_bytes) that lets the launch slice its last wave of units."""
    ldq, ldk, ldv, ldo = (_rowmajor(t, n) for t, n in ((q, "q"), (k, "k"), (v, "v"), (out, "out")))
    if scale is None:
        scale = 128 ** -0.5
    rc = load().svi_attn_fwd(_ptr(q, torch.bfloat16, "q"), ldq, _ptr(k, torch.bfloat16, "k"), ldk,
                             _ptr(v, torch.bfloat16, "v"), ldv, _ptr(out, torch.bfloat16, "out"), ldo,
                             q.shape[0], k.shape[0], num_heads, float(scale), int(bool(accumulate)),
                             *_workspace(workspace), _stream())
    _check(rc, "svi_attn_fwd")
    return out


def attention_qscale(q, k, v, out, num_heads, q_sumsq, q_dim, q_eps, scale=None, accumulate=False, workspace=None):
    """attention() on an UN-normalised q whose full-width RMSNorm factor rsqrt(q_sumsq[r] / q_dim + q_eps) is applied inside
    the softmax (svi_attn_fwd_qscale); q_sumsq f32 [Lq, n] (column 0 is used) or [Lq, n, parts] (the partials of group 0)."""
    ldq, ldk, ldv, ldo = (_rowmajor(t, n) for t, n in ((q, "q"), (k, "k"), (v, "v"), (out, "out")))
    if scale is None:
        scale = 128 ** -0.5
    if q_sumsq.shape[0] != q.shape[0]:
        raise RuntimeError("svi_b200.attention_qscale: q_sumsq must have one row per query row")
    rc = load().svi_attn_fwd_qscale(_ptr(q, torch.bfloat16, "q"), ldq, _ptr(k, torch.bfloat16, "k"), ldk,
                                    _ptr(v, torch.bfloat16, "v"), ldv, _ptr(out, torch.bfloat16, "out"), ldo,
                                    q.shape[0], k.shape[0], num_heads, float(scale), int(bool(accumulate)),
                                    _ptr(q_sumsq, torch.float32, "q_sumsq"), *_sumsq_layout(q_sumsq), int(q_dim),
                                    float(q_eps), *_workspace(workspace), _stream())
    _check(rc, "svi_attn_fwd_qscale")
    return out


def _sumsq_layout(ss):
    """(floats per row, partials per group) of a row-sum-of-squares buffer: [M, groups] or contiguous [M, groups, parts]."""
    if ss.dim() == 3:
        if not ss.is_contiguous():
            raise RuntimeError("svi_b200: a partial sumsq buffer [M, groups, parts] must be contiguous")
        return ss.shape[1] * ss.shape[2], ss.shape[2]
    return _rowmajor(ss, "sumsq"), 0


def _workspace(ws):
    if ws is None:
        return None, 0
    if not ws.is_cuda or not ws.is_contiguous():
        raise RuntimeError("svi_b200: attention workspace must be a contiguous CUDA tensor")
    return _vp(ws.data_ptr()), ws.numel() * ws.element_size()


def attention_plan(units, kv_tiles, sms, workspace_bytes):
    """(n_full, split) the attention launch would use — pure host logic (svi_attn_plan)."""
    a, b = _i32(), _i32()
    load().svi_attn_plan(units, kv_tiles, sms, workspace_bytes, ctypes.byref(a), ctypes.byref(b))
    return a.value, b.value


def attention_workspace_bytes(Lq, Lk, num_heads):
    return int(load().svi_attn_workspace_bytes(Lq, Lk, num_heads))


def attention_sp(q, k, v, out, num_heads, kv_flags, kv_epoch, kv_chunk_rows, kv_self_chunk, scale=None, workspace=None):
    """Self-attention over the rank's full K|V buffer whose remote rows are still being pushed by the peers
    (svi_attn_fwd_sp): kv_flags int32 [n_chunks] device tensor inside the symmetric allocation."""
    ldq, ldk, ldv, ldo = (_rowmajor(t, n) for t, n in ((q, "q"), (k, "k"), (v, "v"), (out, "out")))
    if scale is None:
        scale = 128 ** -0.5
    rc = load().svi_attn_fwd_sp(_ptr(q, torch.bfloat16, "q"), ldq, _ptr(k, torch.bfloat16, "k"), ldk,
                                _ptr(v, torch.bfloat16, "v"), ldv, _ptr(out, torch.bfloat16, "out"), ldo,
                                q.shape[0], k.shape[0], num_heads, float(scale), _ptr(kv_flags, torch.int32, "kv_flags"),
                                int(kv_epoch) & 0xFFFFFFFF, int(kv_chunk_rows), int(kv_self_chunk), *_workspace(workspace),
                                _stream())
    _check(rc, "svi_attn_fwd_sp")
    return out


class _RawCuda:
    """Exposes a raw device allocation to torch through __cuda_array_interface__ (zero copy)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}


def sp_alloc(nbytes, device):
    """Symmetric (peer-mappable) allocation: returns (ptr:int, handle:bytes[64], uint8 tensor view of it)."""
    ptr = _vp()
    handle = ctypes.create_string_buffer(64)
    _check(load().svi_sp_alloc(nbytes, ctypes.byref(ptr), handle), "svi_sp_alloc")
    view = torch.as_tensor(_RawCuda(ptr.value, nbytes), device=device)
    return ptr.value, handle.raw, view


def sp_free(ptr):
    _check(load().svi_sp_free(_vp(ptr)), "svi_sp_free")


def sp_open(handle):
    ptr = _vp()
    _check(load().svi_sp_open(handle, ctypes.byref(ptr)), "svi_sp_open")
    return ptr.value


def sp_close(ptr):
    _check(load().svi_sp_close(_vp(ptr)), "svi_sp_close")


def sp_push(src_ptr, peer_dst, peer_flag, nbytes, epoch_word_ptr, stream):
    """Copy-engine push of this rank's rows + flag word to every peer on `stream` (a torch.cuda.Stream)."""
    n = len(peer_dst)
    arr = _vp * n
    rc = load().svi_sp_push(_vp(src_ptr), arr(*peer_dst), arr(*peer_flag), n, nbytes, _vp(epoch_word_ptr),
                            _vp(stream.cuda_stream))
    _check(rc, "svi_sp_push")


def layernorm_modulate(x, out, eps, gamma=None, beta=None, scale=None, shift=None):
    """out(bf16)[M,D] = LN(x f32 [M,D]) (*gamma + beta) * (1 + scale) + shift."""
    M, D = x.shape
    if not x.is_contiguous() or not out.is_contiguous():
        raise RuntimeError("svi_b200.layernorm_modulate: x and out must be contiguous")
    rc = load().svi_layernorm_modulate(_ptr(x, torch.float32, "x"), M, D, float(eps),
                                       _ptr(gamma, torch.float32, "gamma"), _ptr(beta, torch.float32, "beta"),
                                       _ptr(scale, torch.float32, "scale"), _ptr(shift, torch.float32, "shift"),
                                       _ptr(out, torch.bfloat16, "out"), _stream())
    _check(rc, "svi_layernorm_modulate")
    return out


def layernorm_modulate_split(x, out, eps, gamma=None, beta=None, scale=None, shift=None):
    """out bf16 [M, 2D]: columns [0, D) = bf16(v), [D, 2D) = bf16(v - bf16(v)), v = layernorm_modulate(x)."""
    M, D = x.shape
    if not x.is_contiguous() or not out.is_contiguous() or tuple(out.shape) != (M, 2 * D):
        raise RuntimeError("svi_b200.layernorm_modulate_split: x [M,D] and out [M,2D] must be contiguous")
    rc = load().svi_layernorm_modulate_split(_ptr(x, torch.float32, "x"), M, D, float(eps),
                                             _ptr(gamma, torch.float32, "gamma"), _ptr(beta, torch.float32, "beta"),
                                             _ptr(scale, torch.float32, "scale"), _ptr(shift, torch.float32, "shift"),
                                             _ptr(out, torch.bfloat16, "out"), 2 * D, D, _stream())
    _check(rc, "svi_layernorm_modulate_split")
    return out


def qk_norm_rope(qk, sumsq, eps, wq, wk, rope_cos, rope_sin, row_offset=0):
    """In place on bf16 qk[M, 2D] (q | k side by side, row-strided view allowed): RMSNorm + RoPE of both in one launch;
    sumsq f32 [M, >=2] (columns 0, 1)."""
    ld = _rowmajor(qk, "qk")
    M, D2 = qk.shape
    rc = load().svi_qk_norm_rope(_ptr(qk, torch.bfloat16, "qk"), ld, M, D2 // 2, _ptr(sumsq, torch.float32, "sumsq"),
                                 *_sumsq_layout(sumsq), float(eps), _ptr(wq, torch.float32, "wq"),
                                 _ptr(wk, torch.float32, "wk"), _ptr(rope_cos, torch.float32, "rope_cos"),
                                 _ptr(rope_sin, torch.float32, "rope_sin"), row_offset, _stream())
    _check(rc, "svi_qk_norm_rope")
    return qk


def split_f32_to_bf16x2(src, dst, act=ACT_NONE):
    """dst bf16 [M, 2K] = [bf16(v) | bf16(v - bf16(v))], v = act(src f32 [M, K]) (row-strided views allowed)."""
    M, K = src.shape
    if tuple(dst.shape) != (M, 2 * K):
        raise RuntimeError("svi_b200.split_f32_to_bf16x2: dst must be [M, 2K]")
    rc = load().svi_split_f32_to_bf16x2(_ptr(src, torch.float32, "src"), _rowmajor(src, "src"), M, K, act,
                                        _ptr(dst, torch.bfloat16, "dst"), _rowmajor(dst, "dst"), K, _stream())
    _check(rc, "svi_split_f32_to_bf16x2")
    return dst


def ln_fold_prepare(mods, layers, g_out, rows):
    """mods f32 [>= 6*layers, D] -> g_out f32 [layers, 2, D] (1 + scale), rows bf16 [layers, 2, 4, D] (svi_ln_fold_prepare)."""
    D = mods.shape[1]
    if not (mods.is_contiguous() and g_out.is_contiguous() and rows.is_contiguous()) or g_out.numel() != layers * 2 * D \
            or rows.numel() != layers * 8 * D:
        raise RuntimeError("svi_b200.ln_fold_prepare: contiguous mods [6L,D], g_out [L,2,D], rows [L,2,4,D] required")
    _check(load().svi_ln_fold_prepare(_ptr(mods, torch.float32, "mods"), layers, D, _ptr(g_out, torch.float32, "g_out"),
                                      _ptr(rows, torch.bfloat16, "rows"), _stream()), "svi_ln_fold_prepare")


def ln_fold_combine(o4, bias, u, c):
    """o4 f32 [4, N] -> u = o4[0] + o4[1], c = o4[2] + o4[3] + bias (svi_ln_fold_combine); u, c contiguous f32 [N]."""
    N = o4.shape[1]
    if not o4.is_contiguous() or u.numel() != N or c.numel() != N or not u.is_contiguous() or not c.is_contiguous():
        raise RuntimeError("svi_b200.ln_fold_combine: contiguous o4 [4,N], u [N], c [N] required")
    _check(load().svi_ln_fold_combine(_ptr(o4, torch.float32, "o4"), N, _ptr(bias, torch.float32, "bias"),
                                      _ptr(u, torch.float32, "u"), _ptr(c, torch.float32, "c"), _stream()), "svi_ln_fold_combine")


def zero_(t):
    """t.zero_() as one cudaMemsetAsync node on the current stream (contiguous CUDA tensor)."""
    if not t.is_cuda or not t.is_contiguous():
        raise RuntimeError("svi_b200.zero_: contiguous CUDA tensor required (no CPU fallback)")
    _check(load().svi_zero(_vp(t.data_ptr()), t.numel() * t.element_size(), _stream()), "svi_zero")
    return t


def rmsnorm_rope(t, sumsq, sumsq_col, eps, weight, rope_cos=None, rope_sin=None, row_offset=0):
    """In place on bf16 t[M, D] (row-strided view allowed): full-width RMSNorm + optional RoPE."""
    ldt = _rowmajor(t, "t")
    M, D = t.shape
    ss_ld, ss_parts = _sumsq_layout(sumsq)
    rc = load().svi_rmsnorm_rope(_ptr(t, torch.bfloat16, "t"), ldt, M, D, _ptr(sumsq, torch.float32, "sumsq"),
                                 ss_ld, sumsq_col, ss_parts, float(eps), _ptr(weight, torch.float32, "weight"),
                                 _ptr(rope_cos, torch.float32, "rope_cos"), _ptr(rope_sin, torch.float32, "rope_sin"),
                                 row_offset, _stream())
    _check(rc, "svi_rmsnorm_rope")
    return t


def patchify_gather(x, y, tokens, split=False):
    """x f32 [C0,F,H,W] (+ y f32 [C1,F,H,W]) -> tokens bf16 [L, Kpad]; split: tokens [L, 2 Kpad] = [hi | lo] two-term form."""
    C0, F, H, W = x.shape
    C1 = 0 if y is None else y.shape[0]
    if not x.is_contiguous() or (y is not None and not y.is_contiguous()) or not tokens.is_contiguous():
        raise RuntimeError("svi_b200.patchify_gather: tensors must be contiguous")
    fn = load().svi_patchify_gather_split if split else load().svi_patchify_gather
    rc = fn(_ptr(x, torch.float32, "x"), C0, _ptr(y, torch.float32, "y"), C1, F, H, W,
            _ptr(tokens, torch.bfloat16, "tokens"), tokens.shape[1] // (2 if split else 1), _stream())
    _check(rc, "svi_patchify_gather")
    return tokens


def unpatchify(head_out, out):
    """head_out f32 [L, ld>=4C] -> out f32 [C,F,H,W]."""
    C, F, H, W = out.shape
    rc = load().svi_unpatchify(_ptr(head_out, torch.float32, "head_out"), _rowmajor(head_out, "head_out"),
                               C, F, H, W, _ptr(out, torch.float32, "out"), _stream())
    _check(rc, "svi_unpatchify")
    return out


def cfg_euler_step(latents, v_cond, v_uncond, cfg, sigma, sigma_next):
    rc = load().svi_cfg_euler_step(_ptr(latents, torch.float32, "latents"), _ptr(v_cond, torch.float32, "v_cond"),
                                   _ptr(v_uncond, torch.float32, "v_uncond"), latents.numel(), float(cfg),
                                   float(sigma), float(sigma_next), _stream())
    _check(rc, "svi_cfg_euler_step")
    return latents


def cast_f32_to_bf16(src, dst, act=ACT_NONE):
    if act == ACT_NONE:
        rc = load().svi_cast_f32_to_bf16(_ptr(src, torch.float32, "src"), _ptr(dst, torch.bfloat16, "dst"),
                                         src.numel(), _stream())
    else:
        rc = load().svi_act_f32_to_bf16(_ptr(src, torch.float32, "src"), _ptr(dst, torch.bfloat16, "dst"),
                                        src.numel(), act, _stream())
    _check(rc, "svi_cast_f32_to_bf16")
    return dst


def cast_bf16_to_f32(src, dst):
    rc = load().svi_cast_bf16_to_f32(_ptr(src, torch.bfloat16, "src"), _ptr(dst, torch.float32, "dst"),
                                     src.numel(), _stream())
    _check(rc, "svi_cast_bf16_to_f32")
    return dst


def add_rows(table, t, out):
    rows, D = table.shape
    if not (table.is_contiguous() and t.is_contiguous() and out.is_contiguous()) or rows % t.shape[0]:
        raise RuntimeError("svi_b200.add_rows: contiguous tensors with rows % rows_t == 0 required")
    rc = load().svi_add_rows(_ptr(table, torch.float32, "table"), _ptr(t, torch.float32, "t"), rows, t.shape[0], D,
                             _ptr(out, torch.float32, "out"), _stream())
    _check(rc, "svi_add_rows")
    return out


def axpby(a, alpha, b, beta, out):
    """out = alpha * a + beta * b (f32, same shape, contiguous; out may alias a or b)."""
    if not (a.is_contiguous() and b.is_contiguous() and out.is_contiguous()) or a.shape != b.shape or a.shape != out.shape:
        raise RuntimeError("svi_b200.axpby: a, b, out must be contiguous and of one shape")
    rc = load().svi_axpby(_ptr(a, torch.float32, "a"), float(alpha), _ptr(b, torch.float32, "b"), float(beta),
                          _ptr(out, torch.float32, "out"), a.numel(), _stream())
    _check(rc, "svi_axpby")
    return out


# --------------------------------------------------------------------------------------------- encoders
def embedding_gather(ids, table, out):
    """out f32 [n, dim] = rows ids (int64 [n]) of table bf16 [vocab, dim]."""
    n, (vocab, dim) = ids.numel(), table.shape
    if ids.dtype != torch.int64 or not ids.is_contiguous() or not table.is_contiguous() or not out.is_contiguous():
        raise RuntimeError("svi_b200.embedding_gather: ids must be contiguous int64, table / out contiguous")
    rc = load().svi_embedding_gather(_ptr(ids, name="ids"), n, _ptr(table, torch.bfloat16, "table"), dim, vocab,
                                     _ptr(out, torch.float32, "out"), _stream())
    _check(rc, "svi_embedding_gather")
    return out


def rmsnorm_affine(x, weight, eps, out):
    M, D = x.shape
    if not x.is_contiguous() or not out.is_contiguous():
        raise RuntimeError("svi_b200.rmsnorm_affine: x and out must be contiguous")
    rc = load().svi_rmsnorm_affine(_ptr(x, torch.float32, "x"), M, D, float(eps), _ptr(weight, torch.float32, "weight"),
                                   _ptr(out, torch.bfloat16, "out"), _stream())
    _check(rc, "svi_rmsnorm_affine")
    return out


def layernorm_f32(x, gamma, beta, eps, out):
    M, D = x.shape
    if not x.is_contiguous() or not out.is_contiguous():
        raise RuntimeError("svi_b200.layernorm_f32: x and out must be contiguous")
    rc = load().svi_layernorm_f32(_ptr(x, torch.float32, "x"), M, D, float(eps), _ptr(gamma, torch.float32, "gamma"),
                                  _ptr(beta, torch.float32, "beta"), _ptr(out, torch.float32, "out"), _stream())
    _check(rc, "svi_layernorm_f32")
    return out


def mul_bf16(a, b, out):
    if not (a.is_contiguous() and b.is_contiguous() and out.is_contiguous()) or a.shape != b.shape or a.shape != out.shape:
        raise RuntimeError("svi_b200.mul_bf16: a, b, out must be contiguous and of one shape")
    rc = load().svi_mul_bf16(_ptr(a, torch.bfloat16, "a"), _ptr(b, torch.bfloat16, "b"), _ptr(out, torch.bfloat16, "out"),
                             a.numel(), _stream())
    _check(rc, "svi_mul_bf16")
    return out


def attention_small(q, k, v, out, num_heads, head_dim, scale, bias_table=None, bucket=None, key_mask=None):
    """Short-sequence attention with any head_dim <= 128, optional bucketed relative-position bias and key mask."""
    ldq, ldk, ldv, ldo = (_rowmajor(t, n) for t, n in ((q, "q"), (k, "k"), (v, "v"), (out, "out")))
    if bucket is not None and (bucket.dtype != torch.int32 or tuple(bucket.shape) != (q.shape[0], k.shape[0]) or not bucket.is_contiguous()):
        raise RuntimeError("svi_b200.attention_small: bucket must be contiguous int32 [Lq, Lk]")
    if key_mask is not None and (key_mask.dtype != torch.int32 or key_mask.numel() != k.shape[0]):
        raise RuntimeError("svi_b200.attention_small: key_mask must be int32 [Lk]")
    rc = load().svi_attn_small(_ptr(q, torch.bfloat16, "q"), ldq, _ptr(k, torch.bfloat16, "k"), ldk, _ptr(v, torch.bfloat16, "v"), ldv,
                               _ptr(out, torch.bfloat16, "out"), ldo, q.shape[0], k.shape[0], num_heads, head_dim, float(scale),
                               _ptr(bias_table, torch.float32, "bias_table"), _ptr(bucket, name="bucket"),
                               _ptr(key_mask, name="key_mask"), _stream())
    _check(rc, "svi_attn_small")
    return out


# --------------------------------------------------------------------------------------------- VAE
def conv3d_causal(desc):
    """Launch svi_conv3d_causal with a filled ConvDesc (pointers as ints)."""
    _check(load().svi_conv3d_causal(ctypes.byref(desc), _stream()), "svi_conv3d_causal")


def vae_norm_act(x, n_pix, C, ldx, gamma, silu, out, Cpad):
    rc = load().svi_vae_norm_act(_ptr(x, torch.float32, "x"), n_pix, C, ldx, _ptr(gamma, torch.float32, "gamma"),
                                 int(bool(silu)), _ptr(out, torch.bfloat16, "out"), Cpad, _stream())
    _check(rc, "svi_vae_norm_act")
    return out


def vae_upsample2x(x, H, W, C, out):
    _check(load().svi_vae_upsample2x(_ptr(x, torch.float32, "x"), H, W, C, _ptr(out, torch.bfloat16, "out"), _stream()),
           "svi_vae_upsample2x")
    return out


def vae_space_to_depth(x, H, W, C, out):
    _check(load().svi_vae_space_to_depth(_ptr(x, torch.float32, "x"), H, W, C, _ptr(out, torch.bfloat16, "out"), _stream()),
           "svi_vae_space_to_depth")
    return out


def vae_space_to_depth_act(x, H, W, C, act, out):
    _check(load().svi_vae_space_to_depth_act(_ptr(x, torch.float32, "x"), H, W, C, act, _ptr(out, torch.bfloat16, "out"), _stream()),
           "svi_vae_space_to_depth_act")
    return out


def vae_from_planar(x, C, n_pix, scale, shift, out, ldo, out_is_bf16, ldc=None):
    rc = load().svi_vae_from_planar(_ptr(x, torch.float32, "x"), C, n_pix, n_pix if ldc is None else ldc,
                                    _ptr(scale, torch.float32, "scale"), _ptr(shift, torch.float32, "shift"),
                                    _ptr(out, name="out"), ldo, int(bool(out_is_bf16)), _stream())
    _check(rc, "svi_vae_from_planar")
    return out


def vae_to_planar(x, ldx, C, n_pix, pre_shift, scale, clamp, out, ldc=None):
    rc = load().svi_vae_to_planar(_ptr(x, torch.float32, "x"), ldx, C, n_pix, _ptr(pre_shift, torch.float32, "pre_shift"),
                                  _ptr(scale, torch.float32, "scale"), int(bool(clamp)), _ptr(out, torch.float32, "out"),
                                  n_pix if ldc is None else ldc, _stream())
    _check(rc, "svi_vae_to_planar")
    return out


def frames_to_uint8(video, out):
    """video f32 [3, T, H, W] (contiguous, CUDA) -> out uint8 [T, H, W, 3]: clip((v + 1) * 127.5, 0, 255) truncated."""
    C, T, H, W = video.shape
    if C != 3 or not video.is_contiguous() or not out.is_contiguous() or out.dtype != torch.uint8 or out.numel() != 3 * T * H * W:
        raise RuntimeError("svi_b200.frames_to_uint8: video must be contiguous f32 [3,T,H,W], out contiguous uint8 [T,H,W,3]")
    _check(load().svi_frames_to_uint8(_ptr(video, torch.float32, "video"), T * H * W, T * H * W, _ptr(out, name="out"), _stream()),
           "svi_frames_to_uint8")
    return out


def softmax_rows(s, N, scale, p):
    rc = load().svi_softmax_rows(_ptr(s, torch.float32, "s"), s.shape[0], N, _rowmajor(s, "s"), float(scale),
                                 _ptr(p, torch.bfloat16, "p"), _rowmajor(p, "p"), _stream())
    _check(rc, "svi_softmax_rows")
    return p


# --------------------------------------------------------------------------------------------- wav2vec2 audio encoder
def audio_conv0_gn_gelu(wav, w, gamma, beta, eps, stride, out, workspace=None):
    """out bf16 [T0, C] = GELU(GroupNorm_C(conv1d(wav f32 [n], w f32 [C, k], stride))) (svi_audio_conv0_gn_gelu).
    Returns the workspace (uint8, CUDA); its first 2*C floats hold the channel means and 1/sqrt(var + eps)."""
    C, k = w.shape
    n = wav.numel()
    T0 = (n - k) // stride + 1
    if not (wav.is_contiguous() and w.is_contiguous() and out.is_contiguous()) or tuple(out.shape) != (T0, C):
        raise RuntimeError(f"svi_b200.audio_conv0_gn_gelu: contiguous wav [n], w [C,k] and out [{T0},{C}] required")
    nbytes = int(load().svi_audio_conv0_workspace_bytes(n, C, k, stride))
    if workspace is None or workspace.numel() < nbytes:
        workspace = torch.empty(nbytes, dtype=torch.uint8, device=wav.device)
    rc = load().svi_audio_conv0_gn_gelu(_ptr(wav, torch.float32, "wav"), n, _ptr(w, torch.float32, "w"), C, k, stride,
                                        _ptr(gamma, torch.float32, "gamma"), _ptr(beta, torch.float32, "beta"), float(eps),
                                        _ptr(out, torch.bfloat16, "out"), _ptr(workspace, name="workspace"), workspace.numel(),
                                        _stream())
    _check(rc, "svi_audio_conv0_gn_gelu")
    return workspace


def audio_interp_layernorm(x, gamma, beta, eps, out):
    """out bf16 [S, C] = LayerNorm(linear interpolation (align_corners) of x f32 [T_in, C] to S rows) * gamma + beta."""
    T_in, C = x.shape
    if not x.is_contiguous() or not out.is_contiguous() or out.shape[1] != C:
        raise RuntimeError("svi_b200.audio_interp_layernorm: contiguous x [T_in, C] and out [S, C] required")
    rc = load().svi_audio_interp_layernorm(_ptr(x, torch.float32, "x"), T_in, C, out.shape[0], _ptr(gamma, torch.float32, "gamma"),
                                           _ptr(beta, torch.float32, "beta"), float(eps), _ptr(out, torch.bfloat16, "out"), _stream())
    _check(rc, "svi_audio_interp_layernorm")
    return out


def audio_pos_conv(x, w_packed, bias, groups, out):
    """out f32 [S, D] = x + GELU(grouped conv1d(x, k, padding k/2)[:S] + bias); w_packed f32 [groups, k, cg, cg]."""
    S, D = x.shape
    g, k, cg, cg2 = w_packed.shape
    if g != groups or cg != cg2 or g * cg != D or not (x.is_contiguous() and out.is_contiguous() and w_packed.is_contiguous()) \
            or out.shape != x.shape:
        raise RuntimeError("svi_b200.audio_pos_conv: contiguous x / out [S, D] and w_packed [groups, k, D/groups, D/groups] required")
    rc = load().svi_audio_pos_conv(_ptr(x, torch.float32, "x"), S, D, groups, k, _ptr(w_packed, torch.float32, "w_packed"),
                                   _ptr(bias, torch.float32, "bias"), _ptr(out, torch.float32, "out"), _stream())
    _check(rc, "svi_audio_pos_conv")
    return out


def layernorm_f32x2(x, gamma, beta, eps, out, out_bf16):
    """out f32 [M, D] (row-strided view allowed) and out_bf16 contiguous bf16 [M, D] = LayerNorm(x) * gamma + beta."""
    M, D = x.shape
    if tuple(out.shape) != (M, D) or tuple(out_bf16.shape) != (M, D) or not out_bf16.is_contiguous():
        raise RuntimeError("svi_b200.layernorm_f32x2: out [M, D] and contiguous out_bf16 [M, D] required")
    rc = load().svi_layernorm_f32x2(_ptr(x, torch.float32, "x"), _rowmajor(x, "x"), M, D, float(eps),
                                    _ptr(gamma, torch.float32, "gamma"), _ptr(beta, torch.float32, "beta"),
                                    _ptr(out, torch.float32, "out"), _rowmajor(out, "out"), _ptr(out_bf16, torch.bfloat16, "out_bf16"),
                                    _stream())
    _check(rc, "svi_layernorm_f32x2")
    return out
