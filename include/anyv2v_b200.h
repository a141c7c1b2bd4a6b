/*
 * anyv2v_b200 — C ABI of the B200-native AnyV2V hot path (DDIM inversion + PnP edit over the I2VGen-XL UNet).
 *
 * The reference (TIGER-AI-Lab/AnyV2V) is 100 % Python and has no FFI of its own; every kernel it runs is a
 * library call inside PyTorch/diffusers.  This header is therefore the NEW boundary that sits *under* the
 * reference's Python hook surface (i2vgen-xl/pnp_utils.py) — each entry point cites the reference code whose
 * arithmetic it replaces.  Conventions:
 *   - plain pointers and sizes only (no torch types); all device pointers are fp16 unless stated otherwise;
 *   - stream-ordered: every call only enqueues work on `stream` (a CUstream / cudaStream_t handle);
 *   - return 0 on success, negative AV2V_E* otherwise; text via av2v_last_error(); never throws;
 *   - the caller owns every buffer (inputs, outputs, workspaces); the library keeps no persistent device state;
 *   - activations are channels-last: a frame batch [NF, C, H, W] is stored as [NF][H][W][C] (C contiguous),
 *     a token matrix [rows, C] row-major.  Linear weights are [out, in] row-major (torch nn.Linear layout),
 *     3x3 conv weights [Cout][ky][kx][Cin] (torch channels_last memory of [Cout,Cin,3,3]),
 *     temporal conv weights [Cout][kt][Cin].
 */
#ifndef ANYV2V_B200_H_
#define ANYV2V_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* av2v_stream_t; /* cudaStream_t / CUstream */

enum {
  AV2V_OK = 0,
  AV2V_EINVAL = -1,   /* bad shape / null pointer / unsupported dimension */
  AV2V_EALIGN = -2,   /* pointer or stride not aligned as required (16 B) */
  AV2V_ECUDA = -3,    /* CUDA runtime / driver error (text in av2v_last_error) */
  AV2V_ENOSUP = -4    /* valid request that this build does not implement */
};

int av2v_abi_version(void);
const char* av2v_last_error(void); /* thread-local, valid until the next failing call on this thread */
/* device properties the host side sizes its launches with; returns AV2V_ECUDA when no sm_100 device is current */
int av2v_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------------------------------
 * K7  CFG combine + DDIM step (v-prediction, eta = 0) and its inverse.
 * Replaces: pipeline_i2vgen_xl.py:1159-1176 (CFG, reshape, scheduler.step) and :1407-1420 (inversion), with
 * diffusers DDIMScheduler.step / DDIMInverseScheduler.step (vendored twin consisti2v/ddim_inverse_scheduler.py:329-369).
 * Reproduces the reference's rounding sequence: every product / sum is computed in fp32 and rounded to fp16
 * separately (the reference multiplies fp16 CUDA tensors by fp32 0-dim scalars).
 *   v   = v_edit ? v_neg + g*(v_edit - v_neg) : v_neg
 *   x0  = ca*x - cb*v ;  eps = ca*v + cb*x ;  out = cc*x0 + cd*eps
 * DDIM:    ca=sqrt(a_t)   cb=sqrt(1-a_t)   cc=sqrt(a_prev) cd=sqrt(1-a_prev)
 * inverse: ca=sqrt(a_cur) cb=sqrt(1-a_cur) cc=sqrt(a_next) cd=sqrt(1-a_next)
 * The op is elementwise, so the [B,C,F,h,w] <-> [B*F,C,h,w] permutes of the reference are not needed.
 */
typedef struct {
  const void* x;      /* current latents, n fp16 */
  const void* v_neg;  /* model output (uncond chunk when CFG is on), n fp16 */
  const void* v_edit; /* cond chunk, or NULL for no CFG */
  void* out;          /* n fp16; may alias x */
  int64_t n;
  float guidance;
  float ca, cb, cc, cd;
  const float* coef_dev; /* optional device pointer to {ca, cb, cc, cd, guidance}: read by the kernel INSTEAD of the
                            by-value fields, so that one captured CUDA graph can be replayed for every timestep */
} av2v_ddim_args;
int av2v_ddim_step_cfg_f16(const av2v_ddim_args* a, av2v_stream_t stream);
int av2v_ddim_inverse_step_f16(const av2v_ddim_args* a, av2v_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * K6  GroupNorm (+ optional SiLU), channels-last.
 * Replaces: pnp_utils.py:48-49,92,104 (norm1/norm2 + nonlinearity) and every GroupNorm of the UNet
 * (per-frame domain [NF, H*W, C]; per-clip domain of TemporalConvLayer / TransformerTemporalModel = [B, F*H*W, C]).
 * x, y: [n_samples][rows][C] fp16; statistics per (sample, group) over rows x (C/groups) in fp32.
 * workspace: av2v_groupnorm_workspace_floats(n_samples, C) floats — per-(sample, CTA slot, group) partial
 * sums written by the statistics phase (deterministic, no float atomics) and folded in double by the apply phase of the same
 * (persistent) kernel.
 */
int av2v_groupnorm_workspace_floats(int n_samples, int C);
typedef struct {
  const void* x;
  void* y;
  const void* gamma; /* [C] fp16 */
  const void* beta;  /* [C] fp16 */
  float* workspace;  /* >= av2v_groupnorm_workspace_floats(n_samples, C) floats */
  int32_t n_samples, rows, C, groups;
  float eps;
  int32_t silu; /* 1: y = silu(gn(x)) */
  const void* x2;  /* optional second source: the logical input is [x | x2] along the channels (x: [n][rows][C1], x2: [n][rows][C - C1]) —
                      the skip-connection concat of the up-block resnets (pnp_utils.py:48 normalises the concatenated tensor)
                      without a materialised torch.cat; y is the normalised, concatenated [n][rows][C] */
  int32_t C1;      /* channels of x when x2 != NULL (multiple of 8) */
} av2v_groupnorm_args;
int av2v_groupnorm_silu_f16(const av2v_groupnorm_args* a, av2v_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * tcgen05 GEMM core:  out[slot][m, n] = sum_k A[m, k] * Wt[n, k] + bias[n] + rowbias[m / rows_per_rowbias, n]
 *                                        + residual[slot][m, n]
 * A operand modes (all fed by TMA straight from the channels-last activation, no im2col buffer):
 *   AV2V_A_LINEAR : A is [M, K] row-major (lda elements)                      -> nn.Linear / 1x1 conv
 *   AV2V_A_CONV3X3: A is [NF, H, W, Cin]; K = 9*Cin, zero padding 1, any H, W -> Conv2d 3x3 (pnp_utils.py:78,107);
 *                   stride 2 (Downsample2D) samples the taps with TMA element strides; a_channels < Cin reads the
 *                   missing channels as zeros (conv_in: 8 channels in a 64-wide K block, weights zero-padded)
 *   AV2V_A_TCONV3 : A is [B, F*HW, Cin]; K = 3*Cin, zero padding over frames   -> Conv3d (3,1,1) of TemporalConvLayer
 * LINEAR with a2 != NULL: the logical A is [a | a2] along K (columns [0, k_split) from a, [k_split, K) from a2) — the
 * skip-connection concat of the up blocks as a two-source K loop instead of a materialised torch.cat.
 * n_slots > 1 broadcasts one accumulator tile to several output slots, each with its own residual: this is the
 * fused "conv + residual-copy" of PnP feature injection (pnp_utils.py:109-124: h[uncond]=h[cond]=h[src], then
 * input_tensor + h per branch).
 */
enum { AV2V_A_LINEAR = 0, AV2V_A_CONV3X3 = 1, AV2V_A_TCONV3 = 2 };
typedef struct {
  int32_t mode;
  const void* a;  /* activation */
  const void* w;  /* [N, K] fp16 row-major */
  int32_t M, N, K;
  int32_t lda;    /* LINEAR: row stride of A in elements (>= K, multiple of 8) */
  int32_t NF, H, W, Cin;          /* CONV3X3 (M must equal NF*H*W, K == 9*Cin) */
  int32_t B, rows_per_clip, HW;   /* TCONV3  (M == B*rows_per_clip, K == 3*Cin, rows_per_clip = F*HW) */
  const void* bias;               /* [N] or NULL */
  const void* rowbias;            /* [M/rows_per_rowbias, N] or NULL (time-embedding add, pnp_utils.py:89-91) */
  int32_t rows_per_rowbias;
  const void* residual;           /* [n_slots][M, N] (ld = ldo) or NULL */
  void* out;                      /* [n_slots][M, ldo] */
  int32_t ldo;                    /* output row stride in elements (>= N, multiple of 8) */
  int32_t n_slots;                /* >= 1 */
  int64_t slot_stride;            /* elements between slots (residual and out) */
  int32_t geglu;                  /* 1: fused GEGLU epilogue (FeedForward.net[0], SURVEY A.7): w/bias rows are interleaved in
                                     blocks of 32 as [h_0, gate_0, h_1, gate_1, ...]; out has N/2 columns,
                                     out[m, 32k+j] = (acc[m, 64k+j] + b) * gelu_erf(acc[m, 64k+32+j] + b').  LINEAR mode,
                                     N % 64 == 0, no residual / rowbias / slots. */
  int32_t stride;                 /* CONV3X3: 1 (0 = 1) or 2; the output has (H/stride) x (W/stride) pixels, M = NF*(H/stride)*(W/stride) */
  int32_t a_channels;             /* CONV3X3: channels present in the tensor (0 = Cin; else < Cin, multiple of 8): row stride of A */
  const void* a2;                 /* LINEAR: second source of the K loop or NULL */
  int32_t k_split;                /* LINEAR with a2: columns of `a` (multiple of 64, 0 < k_split < K) */
  int32_t lda2;                   /* LINEAR with a2: row stride of a2 in elements */
  int32_t up2_phase;              /* CONV3X3: 0 = plain; 1..4 = output phase (py, px) = ((p-1) >> 1, (p-1) & 1) of Upsample2D (nearest x 2,
                                     then conv 3 x 3) computed WITHOUT the up-sampled tensor: K = 4*Cin, w = the phase's 2 x 2 tap
                                     weights [N][2][2][Cin] (sums of the 3 x 3 taps that land on the same input pixel), A = the low-
                                     resolution input [NF][H][W][Cin], out = the full [NF][2H][2W][ldo] image (only pixels
                                     (2i+py, 2j+px) are written).  Four launches = the layer at 4/9 of its FLOPs. */
} av2v_gemm_args;
int av2v_gemm_f16(const av2v_gemm_args* a, av2v_stream_t stream);

/* Tile plan of a CONV3X3 call, as av2v_gemm_f16 runs it.  One 128-row accumulator tile covers a block of box_h output rows x
 * box_w output columns of one frame, or frames_per_tile (> 1) whole frames when a frame has at most 64 pixels.  Blocks at the
 * right / bottom edge of a frame are partial (TMA clips their loads and stores).  Tiles are ordered (frame, row block,
 * column block): tiles_per_frame = ceil(W_out / box_w) * ceil(H_out / box_h) (1 for whole frames), m_tiles tiles in all.
 * av2v_conv3x3_plan validates the CONV3X3 fields of `a` exactly as av2v_gemm_f16 does (pointers are not looked at) and
 * fills `out`; it makes no CUDA call. */
typedef struct av2v_conv_plan {
  int32_t box_w, box_h, frames_per_tile, tiles_per_frame, m_tiles;
} av2v_conv_plan;
int av2v_conv3x3_plan(const av2v_gemm_args* a, av2v_conv_plan* out);

/* ------------------------------------------------------------------------------------------------------------
 * LayerNorm over the last dimension of a [rows, C] token matrix (norm1/norm2/norm3 of BasicTransformerBlock,
 * consisti2v/.../videoldm_transformer_blocks.py:461-562).  fp32 statistics, one rounding to fp16.
 */
typedef struct {
  const void* x; void* y;
  const void* gamma; const void* beta; /* [C] fp16 */
  int64_t rows; int32_t C;
  float eps;
} av2v_layernorm_args;
int av2v_layernorm_f16(const av2v_layernorm_args* a, av2v_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * K1-K3  PnP self-attention core (head_dim 64): softmax(Q K^T * scale) V on tcgen05, with the PnP Q/K injection
 * folded in.  Replaces pnp_utils.py:189-210 (spatial) and :295-316 (temporal): F.scaled_dot_product_attention
 * plus the slice-assign injection copies.
 *   - q, k, v are token matrices with arbitrary row stride (so a fused [rows, 3C] QKV buffer works), head h
 *     occupies columns [h*64, h*64+64).
 *   - n_v = 1: plain attention for `batch` sequences.  n_v = 3 (injected step): q/k hold ONLY the source branch
 *     (`batch` = source sequences); the probabilities are computed once and applied to the V of the three
 *     branches (v + j*v_branch_stride), writing o + j*o_branch_stride — identical to the reference where
 *     q,k of uncond/cond are overwritten by the source's.
 *   - AV2V_SEQ_ROWS (spatial): sequence b = rows [b*seq, (b+1)*seq).
 *   - AV2V_SEQ_FRAMES (temporal): tokens live frame-major as [clips][F][HW][*]; sequence (clip, pixel) =
 *     rows clip*F*HW + f*HW + pixel, f = 0..F-1 (no [B,C,F,h,w]->[B*hw,F,C] transpose is materialised).
 *     `batch` = clips*HW, seq = F (F must divide 128 or be a multiple of 128).
 */
enum { AV2V_SEQ_ROWS = 0, AV2V_SEQ_FRAMES = 1 };
typedef struct {
  int32_t seq_mode;
  const void* q; const void* k; const void* v; void* o;
  int32_t ldq, ldk, ldv, ldo;  /* row strides in elements, multiples of 8 */
  int32_t batch, seq, heads;   /* head_dim fixed at 64 */
  int32_t HW;                  /* AV2V_SEQ_FRAMES only */
  int32_t n_v;                 /* 1 or 3 */
  int64_t v_branch_stride, o_branch_stride; /* elements */
  float scale;                 /* softmax scale (64^-0.5) */
  int32_t seq_kv;              /* AV2V_SEQ_ROWS: key/value sequence length (cross-attention); 0 = same as seq */
  int32_t kv_batch_div;        /* AV2V_SEQ_ROWS: query sequence b attends to key/value sequence b / kv_batch_div
                                  (context shared by the F frames of a clip: the reference repeat_interleaves it); 0 = 1 */
} av2v_attn_args;
int av2v_attn_pnp_f16(const av2v_attn_args* a, av2v_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Temporal self-attention with the Q/K/V projection fused in — the "fused QKV-project + scaled-dot-product" kernel
 * BASELINE.json's north_star names for the temporal transformers (to_q / to_k / to_v + SDPA of attn1 / attn2;
 * i2vgen-xl/pnp_utils.py:247-334 is the reference's restatement of that processor, ModifiedTmpAttnProcessor).
 * x holds the LayerNorm-ed tokens frame-major as [clips][F][HW][ldx]; wqkv = rows [Wq ; Wk ; Wv], each [heads*64, Cx];
 * o receives softmax(Q K^T * scale) V per (clip, pixel) sequence of F tokens, head h in columns [h*64, h*64+64).
 * F must divide 128, Cx % 64 == 0.  Q, K, V never reach global memory.
 * n_v = 1: plain self-attention.  n_v = 3: the PnP-injected step (pnp_utils.py:295-302) — the `clips` clips are ordered
 * [source | uncond | cond] (clips % 3 == 0); Q and K of every clip are projected from the SOURCE clip of the same index,
 * V from the clip itself: the result the reference gets by overwriting q, k of the uncond / cond chunks.
 */
typedef struct {
  const void* x; const void* wqkv; void* o;
  int32_t ldx, ldo;            /* row strides in elements, multiples of 8 */
  int32_t clips, F, HW, heads, Cx;
  float scale;
  int32_t n_v;                 /* 1 | 3 */
} av2v_tattn_fused_args;
int av2v_tattn_fused_f16(const av2v_tattn_fused_args* a, av2v_stream_t stream);

/* ------------------------------------------------------------------ diagnostics (bring-up; not part of the drop-in path)
 * Role timers of CTA 0 of the last av2v_gemm_f16 launch made with the environment variable AV2V_GEMM_DEBUG=8:
 * out16[0..4] = producer wait-empty, producer total, MMA wait-tmem-empty, MMA wait-full, MMA total (SM cycles).
 * Synchronises the device. */
int av2v_gemm_debug_timers(unsigned long long* out16);
/* TMA descriptor cache (CUtensorMaps keyed by base pointer + shape + strides + box + swizzle, mutex-guarded, bounded): lookups
 * that hit / missed since the library was loaded and the number of cached descriptors.  Any pointer may be NULL. */
int av2v_tmap_cache_stats(long long* hits, long long* misses, int* entries);

#ifdef __cplusplus
}
#endif
#endif /* ANYV2V_B200_H_ */
