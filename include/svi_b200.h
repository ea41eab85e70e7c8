/*
 * svi_b200.h — C ABI of the B200-native (sm_100a) kernel library for the SVI clip-denoising hot path.
 *
 * The reference (vita-epfl/Stable-Video-Infinity) has NO native boundary: its hot path is Python
 * (diffsynth) calling torch library kernels.  This header therefore DEFINES the boundary a maintainer
 * would bind with ctypes (see INTEGRATION.md).  Every entry point cites the reference lines it
 * replaces (paths relative to the reference root).
 *
 * Conventions
 *   - all pointers are borrowed DEVICE pointers (row-major, contiguous unless a leading dimension
 *     `ld*` in ELEMENTS is given); nothing is allocated or retained by the library;
 *   - `stream` is a cudaStream_t passed as void*; kernels are enqueued asynchronously;
 *   - return value: 0 = ok, <0 = error (svi_last_error() gives the message of the calling thread);
 *   - bf16 = __nv_bfloat16 (2 bytes), f32 = float.
 */
#ifndef SVI_B200_H_
#define SVI_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SVI_ACT_NONE 0
#define SVI_ACT_GELU_TANH 1
#define SVI_ACT_SILU 2
#define SVI_ACT_GELU_ERF 3 /* nn.GELU() default (img_emb MLP, wan_video_dit.py:381) */
#define SVI_ACT_RELU 4     /* AudioProjModel (SVI-Talk), wan_video_dit.py:97-106; GEMM epilogue only */

/* ABI version of this header / library pair. */
int svi_abi_version(void);
/* Message of the last failing call made by this thread (never NULL). */
const char* svi_last_error(void);
/* Number of SMs of the current device (148 on B200); <0 on error. */
int svi_sm_count(void);

/*
 * Epilogue of svi_gemm_bf16:  v = acc[m,n] + bias[n];  v = act(v);
 *                             sumsq[m, n / sumsq_group_cols] += v*v   (if sumsq != NULL)
 *                             v = gate[n] * v                          (if gate != NULL)
 *                             v = residual[m,n] + v                    (if residual != NULL)
 *                             out[m,n] = v  (stored as f32 or bf16)
 */
typedef struct svi_gemm_epilogue {
  void* out;             /* [M, ldo] f32 or bf16 */
  int64_t ldo;           /* elements */
  int32_t out_is_f32;    /* 1: out is float, 0: out is bf16 */
  int32_t act;           /* SVI_ACT_* */
  const float* bias;     /* [N] or NULL */
  const float* gate;     /* [N] or NULL */
  const float* residual; /* [M, ldr] f32 or NULL; may alias out when out_is_f32 */
  int64_t ldr;
  float* sumsq;          /* [M, sumsq_groups] f32, accumulated with atomicAdd (sumsq_parts == 0); or NULL */
  int32_t sumsq_groups;  /* number of column groups that are accumulated (columns beyond are skipped) */
  int32_t sumsq_group_cols; /* width of one group in columns; multiple of 32 */
  /* ---- LayerNorm folded into the GEMM (M > 128 only; both sides optional, NULL = off) ------------------------------
   * Consumer: A = bf16(x[m,k] * g[k]) of the UN-normalised rows x and ln_stats[m] = (sum_k x, sum_k x^2) over ln_dim
   * columns; the epilogue reconstructs the product of the normalised, modulated rows:
   *     acc' = rstd_m * (acc - mean_m * ln_u[n]) ,  ln_u = W g   (then + bias: pass c = W t + b as `bias`)
   *   = ( LayerNorm(x; ln_eps) * g + t ) @ W^T + b   — nn.LayerNorm + modulate + Linear, wan_video_dit.py:358,369-373.
   * Producer: from the final value v (after gate / residual) also write a_next[m,n] = bf16(v * g_next[n]) — the folded
   * A operand of the NEXT GEMM — and accumulate row_stats[m] += (sum_n v, sum_n v^2) with atomicAdd. */
  const float* ln_stats; const float* ln_u; int32_t ln_dim; float ln_eps;
  void* a_next; int64_t ld_an; const float* g_next; float* row_stats;
  /* ---- reproducible row sums of squares: sumsq_parts = sumsq_group_cols / 128 (> 0) makes every 128-column segment STORE
   * its partial sum into sumsq[m, segment] (buffer [M, sumsq_groups * sumsq_parts], no zeroing needed) instead of the
   * atomicAdd per group; the consumers (svi_rmsnorm_rope, svi_qk_norm_rope, svi_attn_fwd_qscale) add a group's partials in
   * index order, so a forward is bit-identical from run to run.  Needs sumsq_group_cols % 128 == 0.  0: atomicAdd. */
  int32_t sumsq_parts;
} svi_gemm_epilogue;

/*
 * out = epilogue(A[M,K] @ W[N,K]^T), A and W bf16, fp32 accumulation on tcgen05 tensor cores (TMEM
 * accumulators, TMA-fed 128B-swizzled operand tiles, persistent warp-specialised kernel).
 * Replaces every nn.Linear / F.linear on the path: wan_video_dit.py:227-229,242 (q,k,v,o),
 * :272-303 (cross-attn q,k,v,o,k_img,v_img), :334-335,372-373 (ffn.0/GELU/ffn.2 with gate+residual),
 * :401-404 (head), :429-452 (patch/text/time embeddings as GEMMs), vram_management/layers.py:65-71.
 * Requirements: K % 8 == 0, N % 8 == 0, lda % 8 == 0, ldw % 8 == 0, 16-byte aligned bases.
 */
int svi_gemm_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, int32_t M, int32_t N,
                  int32_t K, const svi_gemm_epilogue* ep, void* stream);

/*
 * Non-causal softmax(Q K^T * scale) V, head_dim 128, bf16 in / bf16 out, fp32 softmax.
 * Q: [Lq, ldq] bf16 with head h at columns [h*128, h*128+128); K, V likewise with ldk / ldv;
 * O: [Lq, ldo].  Any Lq, Lk >= 1 (ragged tails masked).  accumulate != 0: O += result
 * (used for the image branch of cross-attention, wan_video_dit.py:300-301).
 * workspace (optional, 16-byte aligned device memory of workspace_bytes, may be NULL / 0): lets the launch cut the
 * (head, Q-tile-pair) units of its last, partly filled wave of CTAs into K/V slices that are merged by a second
 * kernel (log-sum-exp merge), so all SMs stay busy; svi_attn_workspace_bytes() returns the size that allows every
 * plan.  The library never allocates.  Results are the same function of the inputs either way (fp32 merge).
 * Replaces flash_attention(), wan_video_dit.py:116-147 (the single attention entry point).
 */
int svi_attn_fwd(const void* Q, int64_t ldq, const void* K, int64_t ldk, const void* V, int64_t ldv,
                 void* O, int64_t ldo, int32_t Lq, int32_t Lk, int32_t num_heads, float scale,
                 int32_t accumulate, void* workspace, size_t workspace_bytes, void* stream);
size_t svi_attn_workspace_bytes(int32_t Lq, int32_t Lk, int32_t num_heads);
/*
 * svi_attn_fwd with the full-width RMSNorm of Q folded into the softmax scale: row r of Q is used as
 * Q[r,:] * rsqrt(S_r / q_dim + q_eps), S_r = q_sumsq[r * q_ss_ld] (q_ss_parts <= 1) or the sum of the q_ss_parts partials
 * q_sumsq[r * q_ss_ld + 0 .. q_ss_parts) in index order; i.e. Q holds the UN-normalised projection and q_sumsq the row
 * sums of squares the GEMM epilogue produced (svi_gemm_epilogue.sumsq / sumsq_parts).  The norm's per-channel weight commutes with
 * the dot product and is applied to K by the caller (K' = K * w_q).  Replaces norm_q of CrossAttention.forward,
 * wan_video_dit.py:272, without a pass over Q.
 */
int svi_attn_fwd_qscale(const void* Q, int64_t ldq, const void* K, int64_t ldk, const void* V, int64_t ldv,
                        void* O, int64_t ldo, int32_t Lq, int32_t Lk, int32_t num_heads, float scale,
                        int32_t accumulate, const float* q_sumsq, int32_t q_ss_ld, int32_t q_ss_parts, int32_t q_dim,
                        float q_eps, void* workspace, size_t workspace_bytes, void* stream);
/* The launch plan svi_attn_fwd uses (pure host function, no device needed): `units` = num_heads * ceil(Lq/256) equal
 * CTAs, kv_tiles = ceil(Lk/128), on `sms` SMs with a workspace of workspace_bytes -> units [0, n_full) run whole, the
 * rest are cut into `split` K/V slices each (split == 1: nothing is sliced). */
void svi_attn_plan(int32_t units, int32_t kv_tiles, int32_t sms, size_t workspace_bytes, int32_t* n_full, int32_t* split);

/*
 * ---- sequence-parallel self-attention: K|V exchange over NVLink peer memory -----------------------------------
 * Replaces the xfuser wiring of the reference's multi-GPU path: usp_attn_forward,
 * diffsynth/distributed/xdit_context_parallel.py:108-129 (xFuserLongContextAttention = Ulysses all-to-all / ring
 * attention over NCCL) and the process-group setup in pipelines/svi_video.py:266-275.
 *
 * svi_sp_alloc   cudaMalloc (zero-filled) of a symmetric buffer + its 64-byte CUDA IPC handle; the caller ships the
 *                handle to the peer processes (torch.distributed all_gather_object) which map it with svi_sp_open.
 * svi_sp_push    on `stream`: for every peer i, copy `bytes` from src (this rank's rows of its own buffer) to
 *                peer_dst[i] (the same rows inside peer i's buffer) with the copy engine, then copy the 4-byte word
 *                at `epoch_word` (device memory holding this layer's epoch number) into peer_flag[i] (this rank's
 *                slot in peer i's flag array).  Stream order makes the flag land after the rows.
 * svi_attn_fwd_sp  svi_attn_fwd over the full [Lk, *] K / V buffers of this GPU where rows
 *                [c*kv_chunk_rows, (c+1)*kv_chunk_rows) are produced by rank c: the K/V stream starts on the local
 *                chunk kv_self_chunk and the TMA producer waits for kv_flags[c] == kv_epoch (ld.acquire.sys) before
 *                the first tile that touches chunk c, so the push of the remote rows overlaps the attention math.
 *                kv_flags: device uint32[n_chunks] inside this rank's symmetric allocation.
 * Flags are compared for equality: the caller alternates two buffers/flag arrays by layer parity and numbers the
 * launches 1,2,3,... so a flag cannot advance past the epoch a consumer still waits for (DESIGN.md §6).
 */
int svi_sp_alloc(size_t bytes, void** ptr, unsigned char* handle64);
int svi_sp_free(void* ptr);
int svi_sp_open(const unsigned char* handle64, void** peer_ptr);
int svi_sp_close(void* peer_ptr);
int svi_sp_push(const void* src, void* const* peer_dst, void* const* peer_flag, int32_t n_peers, size_t bytes,
                const void* epoch_word, void* stream);
int svi_attn_fwd_sp(const void* Q, int64_t ldq, const void* K, int64_t ldk, const void* V, int64_t ldv,
                    void* O, int64_t ldo, int32_t Lq, int32_t Lk, int32_t num_heads, float scale,
                    const void* kv_flags, uint32_t kv_epoch, int32_t kv_chunk_rows, int32_t kv_self_chunk,
                    void* workspace, size_t workspace_bytes, void* stream);

/*
 * y[m,:] = LayerNorm(x[m,:]; eps, no affine unless gamma/beta) * (1 + scale[:]) + shift[:]  -> bf16.
 * x f32 [M, D]; gamma/beta/scale/shift f32 [D] or NULL.  D % 8 == 0, D <= 8192.
 * Replaces nn.LayerNorm + modulate(): wan_video_dit.py:150-151,331-333,358,368-372,401-403.
 */
int svi_layernorm_modulate(const float* x, int32_t M, int32_t D, float eps, const float* gamma,
                           const float* beta, const float* scale, const float* shift, void* y_bf16,
                           void* stream);

/*
 * Split-precision variant for the head GEMM's A operand: y[m, 0:D] = bf16(v), y[m, lo_col : lo_col + D] = bf16(v - bf16(v))
 * (row pitch ldy elements).  Feeding the GEMM the two halves in two accumulating passes gives the A operand ~16 mantissa
 * bits; used where a bf16 A operand is the dominant parity error and the GEMM is tiny (DESIGN.md section 2).
 */
int svi_layernorm_modulate_split(const float* x, int32_t M, int32_t D, float eps, const float* gamma,
                                 const float* beta, const float* scale, const float* shift, void* y_bf16,
                                 int64_t ldy, int32_t lo_col, void* stream);

/*
 * In place on bf16 rows t[m, 0:D] (leading dim ldt):  t = t * rsqrt(S_m/D + eps) * w[:],  S_m = sumsq[m*sumsq_ld + sumsq_col]
 * (sumsq_parts <= 1) or the sum, in index order, of the partials sumsq[m*sumsq_ld + sumsq_col*sumsq_parts + 0 .. sumsq_parts)
 * then, if rope_cos != NULL, the interleaved-pair rotation of every head (head_dim 128):
 *   (t[2i], t[2i+1]) <- (t[2i] c_i - t[2i+1] s_i,  t[2i] s_i + t[2i+1] c_i),  c,s = rope[(m + row_offset), i], i<64.
 * Replaces RMSNorm (wan_video_dit.py:186-197, over the FULL width D) + rope_apply (:178-183).
 */
int svi_rmsnorm_rope(void* t_bf16, int64_t ldt, int32_t M, int32_t D, const float* sumsq,
                     int32_t sumsq_ld, int32_t sumsq_col, int32_t sumsq_parts, float eps, const float* w,
                     const float* rope_cos, const float* rope_sin, int32_t row_offset, void* stream);

/* svi_rmsnorm_rope on q and k of the fused QKV buffer in ONE launch: row m holds q at [0, D) and k at [D, 2D);
 * sumsq groups 0 / 1 (as in svi_rmsnorm_rope, sumsq_parts partials each) are their row sums of squares, wq / wk the norm
 * weights (wan_video_dit.py:227-231). */
int svi_qk_norm_rope(void* qk_bf16, int64_t ld, int32_t M, int32_t D, const float* sumsq, int32_t sumsq_ld,
                     int32_t sumsq_parts, float eps, const float* wq, const float* wk, const float* rope_cos, const float* rope_sin,
                     int32_t row_offset, void* stream);

/*
 * Patchify gather (im2col of the k=s=(1,2,2) Conv3d): x f32 [C, F, H, W] -> tokens bf16 [L, Kpad],
 * L = F*(H/2)*(W/2), column index = c*4 + dy*2 + dx (matching Conv3d weight.reshape(d, C*4)),
 * columns [C*4, Kpad) zero.  Replaces patchify's Conv3d input side, wan_video_dit.py:473-477.
 * Up to two sources are concatenated on the channel axis (x: C0 channels, y: C1 channels; y may be NULL),
 * replacing torch.cat([x, y], dim=1), svi_video.py:94.
 */
int svi_patchify_gather(const float* x, int32_t C0, const float* y, int32_t C1, int32_t F, int32_t H,
                        int32_t W, void* tokens_bf16, int32_t Kpad, void* stream);

/* Split-precision variant: tokens bf16 [L, 2*Kpad], columns [0, Kpad) = bf16(v), [Kpad, 2 Kpad) = bf16(v - bf16(v)). */
int svi_patchify_gather_split(const float* x, int32_t C0, const float* y, int32_t C1, int32_t F, int32_t H,
                              int32_t W, void* tokens_bf16, int32_t Kpad, void* stream);

/*
 * Unpatchify scatter: head output f32 [L, ldh] (first 4*C columns = (dy, dx, c)) -> out f32 [C, F, H, W]
 * ('b (f h w) (x y z c) -> b c (f x) (h y) (w z)', wan_video_dit.py:479-484).
 */
int svi_unpatchify(const float* head_out, int64_t ldh, int32_t C, int32_t F, int32_t H, int32_t W,
                   float* out, void* stream);

/*
 * Classifier-free guidance + flow-matching Euler step, fused:
 *   v = v_uncond + cfg * (v_cond - v_uncond);  latents += v * (sigma_next - sigma).
 * v_uncond may be NULL (cfg == 1 path).  svi_video.py:410,420; flow_match.py:53-64.
 */
int svi_cfg_euler_step(float* latents, const float* v_cond, const float* v_uncond, int64_t n,
                       float cfg, float sigma, float sigma_next, void* stream);

/* dst_bf16[i] = bf16(src_f32[i]);  dst_f32[i] = float(src_bf16[i]) */
int svi_cast_f32_to_bf16(const float* src, void* dst_bf16, int64_t n, void* stream);
int svi_cast_bf16_to_f32(const void* src_bf16, float* dst, int64_t n, void* stream);

/* dst[m, k] = bf16(v), dst[m, lo_col + k] = bf16(v - bf16(v)) with v = act(src[m, k]) (act: NONE | SILU | GELU_TANH |
 * GELU_ERF): the two-term bf16 form of an f32 GEMM input (time / text / image embedding MLPs, wan_video_dit.py:429-452). */
int svi_split_f32_to_bf16x2(const float* src, int64_t lds, int32_t M, int32_t K, int32_t act, void* dst_bf16,
                            int64_t ldd, int32_t lo_col, void* stream);
/*
 * Per-timestep vectors of the LayerNorm fold (svi_gemm_epilogue.ln_*):
 * svi_ln_fold_prepare  mods f32 [6*layers, D] (rows shift/scale/gate of self-attention, shift/scale/gate of the FFN per
 *                      block, wan_video_dit.py:356-357) -> g f32 [layers, 2, D] = 1 + scale and rows bf16
 *                      [layers, 2, 4, D] = (g_hi, g_lo, t_hi, t_lo) two-term forms of g and the shift t;
 * svi_ln_fold_combine  o4 f32 [4, N] = rows @ W^T (one svi_gemm_bf16 with M = 4) -> u = o4[0] + o4[1] = W g and
 *                      c = o4[2] + o4[3] + bias = W t + b.
 */
int svi_ln_fold_prepare(const float* mods, int32_t layers, int32_t D, float* g_out, void* rows_bf16, void* stream);
int svi_ln_fold_combine(const float* o4, int32_t N, const float* bias, float* u, float* c, void* stream);
/* cudaMemsetAsync(ptr, 0, bytes) on `stream` (row-sum accumulators of a whole forward in one node). */
int svi_zero(void* ptr, size_t bytes, void* stream);

/* out[i] = act(in[i]) on f32 (SiLU in front of time_projection, wan_video_dit.py:441-442) -> bf16 */
int svi_act_f32_to_bf16(const float* src, void* dst_bf16, int64_t n, int32_t act, void* stream);

/*
 * mod[j, :] = table[j, :] + t[:] (j < rows) — AdaLN modulation rows (wan_video_dit.py:356-357, 402).
 * table f32 [rows, D], t f32 [rows_t, D] with rows % rows_t == 0 (row j uses t[j % rows_t]: one launch covers the
 * modulation tables of all layers); out f32 [rows, D].
 */
int svi_add_rows(const float* table, const float* t, int32_t rows, int32_t rows_t, int32_t D,
                 float* out, void* stream);

/*
 * out[i] = alpha * a[i] + beta * b[i], f32, n % 4 == 0, out may alias a or b.  TeaCache bookkeeping on the token
 * stream: residual = after - before (svi_video.py:67-69) and tokens + residual on a skipped step (:70-72).
 */
int svi_axpby(const float* a, float alpha, const float* b, float beta, float* out, int64_t n, void* stream);


/* ------------------------------------------------------------------------------------------------
 * Wan 3-D causal VAE (reference diffsynth/models/wan_video_vae.py).  Activations are channels-last.
 * ---------------------------------------------------------------------------------------------- */

/*
 * One causal conv launch (CausalConv3d :33-52, Conv2d of Resample :82-174, time_conv, shortcut 1x1x1) as an
 * implicit GEMM on tcgen05.  Input: bf16 frame ring [ring_slots][in_H][in_W][C_in]; `slot[t*3 + a]` names the
 * ring slot read by output frame t at temporal tap a (history frames stay in the ring — no pad/cat copies).
 * Input pixel = output pixel + (k_h - pad_h, k_w - pad_w); out-of-range pixels read as zero.
 * Weights: bf16 [w_rows, w_ld], row = output channel, column = ((a*kh + b)*kw + c)*ceil64(C_in) + channel.
 * Output: f32 channels-last, frame t at out + t*out_frame_stride, pixel pitch out_ld; columns >= n_split
 * (if n_split > 0) go to out + split_offset with column - n_split (upsample3d channel->frame split :153-156).
 * out = conv + bias (+ residual).
 */
typedef struct svi_conv_desc {
  const void* x_ring; int32_t ring_slots, in_H, in_W, C_in;
  const void* w_packed; int32_t w_rows; int64_t w_ld;
  int32_t kt, kh, kw, pad_h, pad_w;
  int32_t H, W, T;            /* output height, width, frames (T <= 4) */
  int32_t slot[12];
  int32_t C_out;
  int32_t tile_w;             /* output tile = (128/tile_w) x tile_w pixels; 8, 16, 32, 64 or 128 */
  float* out; int64_t out_frame_stride; int32_t out_ld;
  int32_t n_split; int64_t split_offset;
  const float* bias;
  const float* residual; int64_t res_frame_stride; int32_t res_ld;
  /* Fused producer of the NEXT conv's input (optional; next_ring == NULL: off).  Requires C_out <= 256 and n_split == 0.
   * For every output pixel: y = act(v / max(||v||_2, 1e-12) * sqrt(C_out) * next_gamma) with v = the conv output
   * (incl. bias / residual), act = SiLU if next_silu, written as bf16 to next_ring + next_slot[t]*next_frame_stride +
   * pixel*next_ld (channels [C_out, next_ld) are left untouched: the caller keeps them zero).  next_gamma == NULL: plain
   * cast.  write_f32 == 0 additionally drops the fp32 output (`out` may then be NULL).  Replaces RMS_norm + nn.SiLU in
   * front of the second CausalConv3d of a ResidualBlock and between blocks (wan_video_vae.py:55-70, 206-210). */
  void* next_ring; int64_t next_frame_stride; int32_t next_ld; int32_t next_slot[4];
  const float* next_gamma; int32_t next_silu; int32_t write_f32;
  /* Kernel choice (same results up to accumulation order).  1: one CTA per 128-pixel patch, one input box per tap.
   * 2: CTA pairs (tcgen05 cta_group::2) on two image rows x 128 pixels; the input row window is loaded once per
   * (k_t, k_h, 64-channel chunk) and the k_w taps read it at shifted row offsets, the weight tile is split between the
   * two CTAs — needs k_w == 3 and pad_w == 1.  0: 2 where it applies and W >= 192, else 1. */
  int32_t variant;
} svi_conv_desc;
int svi_conv3d_causal(const svi_conv_desc* d, void* stream);

/*
 * y[p, 0:C] = bf16( act( x[p, 0:C] / max(||x[p,:]||_2, 1e-12) * sqrt(C) * gamma[0:C] ) ), y[p, C:Cpad] = 0.
 * gamma == NULL: plain cast (no normalisation).  silu != 0: SiLU after the norm.  x f32 [n_pix, ldx].
 * Replaces RMS_norm (:55-70) + nn.SiLU and the fp32->bf16 staging of conv inputs.
 */
int svi_vae_norm_act(const float* x, int64_t n_pix, int32_t C, int64_t ldx, const float* gamma, int32_t silu,
                     void* y_bf16, int32_t Cpad, void* stream);
/* nearest-exact x2 spatial upsample (Upsample :73-79) fused with the bf16 cast: x f32 [H,W,C] -> y bf16 [2H,2W,C] */
int svi_vae_upsample2x(const float* x, int32_t H, int32_t W, int32_t C, void* y_bf16, void* stream);
/* space-to-depth for the stride-2 Conv2d of downsample (:108-113): x f32 [H,W,C] -> y bf16 [H/2,W/2,4C],
 * y[h,w,(dy*2+dx)*C + c] = x[2h+dy, 2w+dx, c] */
int svi_vae_space_to_depth(const float* x, int32_t H, int32_t W, int32_t C, void* y_bf16, void* stream);
/* Same with an activation (SVI_ACT_NONE | SVI_ACT_SILU) applied before the rearrangement: the stride-2 convolutions of
 * the SVI-Dance pose stem consume SiLU(previous conv) (svi_video_dance.py:262-267). */
int svi_vae_space_to_depth_act(const float* x, int32_t H, int32_t W, int32_t C, int32_t act, void* y_bf16, void* stream);
/* planar f32 (channel c at x + c*ldc, n_pix contiguous) -> channels-last (x*scale[c] + shift[c]), f32 [n_pix, ldo]
 * or bf16 (out_is_bf16), columns [C, ldo) zero */
int svi_vae_from_planar(const float* x, int32_t C, int64_t n_pix, int64_t ldc, const float* scale, const float* shift,
                        void* out, int32_t ldo, int32_t out_is_bf16, void* stream);
/* channels-last f32 [n_pix, ldx] -> planar f32 (channel c at out + c*ldc): (x + pre_shift[c]) * scale[c],
 * optional clamp to [-1,1] (WanVideoVAE.single_decode :753-756; latent normalisation :542-549) */
int svi_vae_to_planar(const float* x, int64_t ldx, int32_t C, int64_t n_pix, const float* pre_shift,
                      const float* scale, int32_t clamp, float* out, int64_t ldc, void* stream);
/* planar f32 video [3][n_pix] (channel c at video + c*plane_stride; n_pix = T*H*W) -> uint8 [n_pix][3]:
 * clip((v + 1) * 127.5, 0, 255) truncated — the clip-boundary conversion of tensor2video (svi_video.py:366-370) on the
 * device, so that 1 byte per sample instead of 4 crosses to the host and the frames stay available on the device for the
 * next clip's conditioning (test_svi.py:472). */
int svi_frames_to_uint8(const float* video, int64_t plane_stride, int64_t n_pix, void* out_u8, void* stream);
/* p[r, 0:N] = bf16(softmax(s[r, 0:N] * scale)), p[r, N:ldp] = 0; s f32 [rows, lds] (VAE AttentionBlock :235-273) */
int svi_softmax_rows(const float* s, int32_t rows, int32_t N, int64_t lds, float scale, void* p_bf16, int64_t ldp,
                     void* stream);

/*
 * ---- conditioning encoders (once per clip; SURVEY.md §8f.1) -------------------------------------------------------
 * The projections / MLPs of both encoders are svi_gemm_bf16 calls; these are the remaining ops.
 *
 * svi_embedding_gather  out f32 [n, dim] = table bf16 [vocab, dim] rows ids[i]     (wan_video_text_encoder.py:246)
 * svi_rmsnorm_affine    y bf16 = w * x * rsqrt(mean(x^2) + eps), x f32 [M, D]       (T5LayerNorm :22-35)
 * svi_layernorm_f32     y f32 = LayerNorm(x) * gamma + beta                         (ViT pre_norm,
 *                                                                     wan_video_image_encoder.py:470-471)
 * svi_mul_bf16          out = a * b elementwise (gated-GELU product, T5FeedForward :106)
 * svi_attn_small        softmax(Q K^T * scale + bias) V for short sequences and any head_dim <= 128, fp32 math:
 *                       Q,K,V,O bf16 [L, ld] with head h at columns [h*head_dim, (h+1)*head_dim);
 *                       bias_table f32 [n_buckets, H] + bucket int32 [Lq, Lk] (T5RelativeEmbedding :159-190, the
 *                       bucket of (query, key) is position-only and shared by all layers) or both NULL;
 *                       key_mask int32 [Lk] (0 = masked; T5Attention :73-77) or NULL.
 *                       Replaces T5Attention.forward :55-89 (scale 1, bias, mask) and the CLIP SelfAttention
 *                       (wan_video_image_encoder.py:255-268: head_dim 80, scale 1/sqrt(80)).
 */
int svi_embedding_gather(const int64_t* ids, int32_t n, const void* table_bf16, int32_t dim, int64_t vocab, float* out,
                         void* stream);
int svi_rmsnorm_affine(const float* x, int32_t M, int32_t D, float eps, const float* w, void* y_bf16, void* stream);
int svi_layernorm_f32(const float* x, int32_t M, int32_t D, float eps, const float* gamma, const float* beta, float* y,
                      void* stream);
int svi_mul_bf16(const void* a, const void* b, void* out, int64_t n, void* stream);
int svi_attn_small(const void* Q, int64_t ldq, const void* K, int64_t ldk, const void* V, int64_t ldv, void* O,
                   int64_t ldo, int32_t Lq, int32_t Lk, int32_t num_heads, int32_t head_dim, float scale,
                   const float* bias_table, const int32_t* bucket, const int32_t* key_mask, void* stream);

/*
 * ---- wav2vec2 audio encoder of SVI-Talk (group-norm / post-LN variant, chinese-wav2vec2-base) ------------------------
 * Reference: utils/audio_process.py:18-41 (get_embedding) running utils/src/audio_analysis/wav2vec2.py:13-64 on
 * transformers' modeling_wav2vec2.  Activations are channels-last.  Convolutions 2-7 are svi_gemm_bf16 calls on strided
 * views of the previous activation (K = k*C, lda = s*C; for k = 3 a two-pass split, see DESIGN.md §4); the feature
 * projection, q|k|v, out-projection and feed-forward layers are svi_gemm_bf16, the attention svi_attn_small (head_dim 64).
 *
 * svi_audio_conv0_gn_gelu   out bf16 [T0, C] = GELU_erf(GroupNorm_C(conv1d(wav, w[C, k], stride))), T0 = (n - k)/stride + 1,
 *                           per-channel statistics over the whole time axis (Wav2Vec2GroupNormConvLayer: conv 1->512, k 10,
 *                           s 5, no bias; nn.GroupNorm(512, 512, eps, affine)).  Two passes over the waveform: per-block fp64
 *                           partial sums, merged in block order, then the conv is recomputed and normalised; the fp32 conv
 *                           output is never stored and nothing is accumulated with atomics.  workspace: 16-byte aligned,
 *                           svi_audio_conv0_workspace_bytes(n, C, k, stride) bytes; on completion its first 2*C floats
 *                           hold the channel means and 1/sqrt(var + eps).  C % 32 == 0, C <= 1024, k <= 16.
 * svi_audio_interp_layernorm  y bf16 [S, C] = LayerNorm(F.interpolate(x^T, S, mode='linear', align_corners=True)^T)
 *                           * gamma + beta, x f32 [T_in, C] (torch_utils.py:16-19 + Wav2Vec2FeatureProjection.layer_norm).
 * svi_audio_pos_conv        out f32 [S, D] = x + GELU_erf(conv1d(x, groups, k, padding k/2)[:S] + bias)
 *                           (Wav2Vec2PositionalConvEmbedding incl. Wav2Vec2SamePadLayer, plus the residual add of
 *                           Wav2Vec2Encoder.forward); w_packed f32 [groups][k][cg][cg] with [g][j][c][o] = w[g*cg + o, c, j]
 *                           (weight norm folded on the host), cg = D / groups a multiple of 8 and <= 64, k even.
 *                           out must not alias x.
 * svi_layernorm_f32x2       y f32 [M, ldy] and y_bf16 bf16 [M, D] (contiguous) = LayerNorm(x [M, ldx]) * gamma + beta:
 *                           the post-LN LayerNorms of Wav2Vec2EncoderLayer, whose output is both the next residual (fp32,
 *                           or a slot of the stacked [S, layers, D] result when ldy = layers*D) and the next GEMM's A.
 *                           y may alias x.
 */
size_t svi_audio_conv0_workspace_bytes(int64_t n_samples, int32_t C, int32_t k, int32_t stride);
int svi_audio_conv0_gn_gelu(const float* wav, int64_t n_samples, const float* w, int32_t C, int32_t k, int32_t stride,
                            const float* gamma, const float* beta, float eps, void* out_bf16, void* workspace,
                            size_t workspace_bytes, void* stream);
int svi_audio_interp_layernorm(const float* x, int32_t T_in, int32_t C, int32_t S, const float* gamma, const float* beta,
                               float eps, void* y_bf16, void* stream);
int svi_audio_pos_conv(const float* x, int32_t S, int32_t D, int32_t groups, int32_t k, const float* w_packed,
                       const float* bias, float* out, void* stream);
int svi_layernorm_f32x2(const float* x, int64_t ldx, int32_t M, int32_t D, float eps, const float* gamma,
                        const float* beta, float* y, int64_t ldy, void* y_bf16, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SVI_B200_H_ */
