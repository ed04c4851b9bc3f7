/* dpb200.h — C-ABI of libdpb200.so: the sm_100a device math behind the reference's Python API boundary.
 *
 * The reference (VainF/Diff-Pruning) has no FFI of its own: its hot path dispatches ATen ops from Python
 * (SURVEY.md §2.3).  Each entry point below replaces the ATen/cuDNN/cuBLAS op(s) the reference reaches from
 * the cited lines.  Conventions (SURVEY.md §8(b2)):
 *   - plain pointers + extents, no torch types; all buffers (inputs, outputs, workspaces) are caller-owned
 *     DEVICE memory; the library never allocates device memory, never synchronises, never throws;
 *   - every call enqueues kernels on `stream` (a cudaStream_t passed as void*), so it is CUDA-graph capturable;
 *   - return value: DP_OK (0) or a negative DP_ERR_*; dp_strerror() names it; dp_last_cuda_error() returns
 *     the cudaError_t captured by the failing launch;
 *   - activations are fp32 NHWC "views": pointer + pixel stride `ld` (elements) >= channels, which lets a
 *     tensor live inside a wider (concatenated) buffer — torch.cat on the skip path never copies
 *     (unet_2d_blocks.py:1822,2035);
 *   - weights stay in the reference layout (OIHW / (out,in)) at the boundary; dp_pack_conv_weight() makes the
 *     K-major operands the kernels consume.
 */
#ifndef DPB200_H
#define DPB200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* dp_stream_t; /* cudaStream_t */

enum {
  DP_OK = 0,
  DP_ERR_SHAPE = -1,       /* inconsistent / unsupported extents */
  DP_ERR_ALIGN = -2,       /* pointer or stride alignment the kernel cannot take */
  DP_ERR_UNSUPPORTED = -3, /* valid request outside what is implemented */
  DP_ERR_CUDA = -4,        /* launch failed: see dp_last_cuda_error() */
  DP_ERR_NULL = -5         /* required pointer is NULL */
};

int dp_version(void);
const char* dp_strerror(int code);
int dp_last_cuda_error(void);
/* number of CUDA kernels this library has launched in this process (monotonic; for gpu_launches accounting) */
int64_t dp_launch_count(void);
/* 1 if the tcgen05/TMA tensor-core path is compiled in and usable on the current device, else 0 */
int dp_tc_available(void);

/* ------------------------------------------------------------------------------------------------
 * Convolution as implicit GEMM.  Replaces aten::convolution / convolution_backward reached from
 *   resnet.py:612,632,635 (ResnetBlock2D conv1/conv2/conv_shortcut), resnet.py:165,218 (Up/Downsample2D),
 *   unet_2d.py:273,304 (conv_in/conv_out), and — as 1x1 convolutions over (N, H*W, C) — every nn.Linear on
 *   the path: embeddings.py:200-212, resnet.py:617, attention_processor.py:440-462 (to_q/k/v/out).
 *   x: [N][H][W][C] (ldx), y: [N][P][Q][K] (ldy), taps R x S, same stride both axes, pad_t/pad_l explicit
 *   (bottom/right padding is implied by P,Q — this is how Downsample2D's F.pad(0,1,0,1), resnet.py:213-215,
 *   is folded in: stride 2, pad_t = pad_l = 0, P = H/2).
 * ------------------------------------------------------------------------------------------------ */
#define DP_CONV_ACCUMULATE 1 /* fprop: y += ; dgrad: dx += (instead of =) */
#define DP_CONV_FORCE_SIMT 2 /* never take the tensor-core path (testing / odd shapes) */
/* fprop / wgrad: x is already split for the tensor-core path (dp_groupnorm_fwd_split), fp16 [N][H][W][2][ldx]: per pixel
 * hi = fp16(s*x) in elements [0, ldx), lo' = fp16((s*x - hi) * 2^11) in [ldx, 2 ldx), s = the power of two of amax_x (see
 * dp_pack_conv_weight_tc).  ldx counts fp16 ELEMENTS, a multiple of 8, >= C; the pad channels [C, ldx) must hold finite values (zeros).
 * Such a launch never falls back to the SIMT path (it cannot read the split form): outside dp_conv_presplit_eligible it fails. */
#define DP_CONV_X_SPLIT 4

typedef struct dp_conv_args {
  int32_t N, H, W, C;
  int32_t P, Q, K;
  int32_t R, S, stride, pad_t, pad_l;
  int32_t flags;
  int32_t splits;      /* wgrad only: split count over the N*P*Q reduction (>= 1) */
  void* x;             /* fprop: in   | dgrad: out (dx) | wgrad: in  */
  int64_t ldx;
  void* y;             /* fprop: out  | dgrad: in (dy)  | wgrad: in (dy) */
  int64_t ldy;
  const float* w;      /* fprop: packed [R*S][C][K] | dgrad: packed [R*S][K][C] (dp_pack_conv_weight) */
  const void* w_tc_hi; /* optional tensor-core operand (dp_pack_conv_weight_tc): fp16 hi part of the scaled weight, GEMM-K contiguous: */
  const void* w_tc_lo; /*   fprop [R*S][K][Cp] | dgrad [R*S][C][Kp] (Cp/Kp = dp_tc_weight_row); w_tc_lo = fp16 scaled residual. NULL => SIMT path */
  const float* bias;   /* fprop epilogue: + bias[K]                                   (nullable) */
  const float* rowadd; /* fprop epilogue: + rowadd[n*ld_rowadd + k] per image n (temb, resnet.py:618-621) (nullable) */
  int64_t ld_rowadd;
  const float* residual; /* fprop epilogue: + residual[pixel*ld_res + k] (resnet.py:637, attention_processor.py:466) (nullable) */
  int64_t ld_res;
  float* workspace;    /* wgrad: [splits][K][R*S*C] fp32 partial sums; fprop / dgrad: optional split-K scratch
                          (dp_conv_splitk_workspace_floats), NULL = never split */
  /* Tensor-core path (3 x fp16 split, conv_tc.cu): "amax slots" = one device uint32 each holding the bit pattern of an upper bound of
   * max|v| over the operand — amax_x for x, amax_y for y / dy (both accumulated by dp_amax), amax_w for the packed weight
   * (written by dp_pack_conv_weight_tc).  A NULL slot sends the launch to the exact-fp32 SIMT kernel. */
  const uint32_t* amax_x; const uint32_t* amax_y; const uint32_t* amax_w;
  uint32_t* amax_out;  /* optional: fprop accumulates max|y| of what it wrote, dgrad max|dx| (dp_amax semantics), on every kernel
                          path — the consumer of that tensor then needs no dp_amax pass */
  float* bias_ws;      /* optional, wgrad: also writes the per-split column sums of dy, [splits][K] — the bias gradient falls out of the
                          pass over dy the weight gradient makes anyway (dp_conv2d_wgrad_reduce adds them to db in fixed order) */
} dp_conv_args;

int dp_conv2d_fprop(const dp_conv_args* a, dp_stream_t stream);
int dp_conv2d_dgrad(const dp_conv_args* a, dp_stream_t stream);
/* Launches with fewer 128-pixel x 128-channel tiles than half the SMs (the 4x4 / 8x8 / 16x16 levels of the UNets, SURVEY.md §8d) split
 * their K loop over the idle SMs when a->workspace holds this many floats (op 0: fprop, 1: dgrad); 0 = the geometry does not split.
 * The splits are summed in fixed order by a second launch: results stay deterministic (ddpm_prune.py:102 accumulates across steps). */
long long dp_conv_splitk_workspace_floats(const dp_conv_args* a, int op);
/* writes split partial sums to a->workspace; dp_conv2d_wgrad_reduce finishes the job */
int dp_conv2d_wgrad(const dp_conv_args* a, dp_stream_t stream);
/* DP_OK when both dp_conv2d_fprop and dp_conv2d_wgrad take DP_CONV_X_SPLIT for this geometry (stride 1, 'same' padding, tensor-core
 * path available; pointers not needed), else DP_ERR_UNSUPPORTED */
int dp_conv_presplit_eligible(const dp_conv_args* a);

/* dW (OIHW, the nn.Parameter .grad) += sum_splits workspace — fixed order, no atomics (deterministic,
 * ddpm_prune.py:102 accumulates across timesteps, SURVEY.md §0.4).  If `w` and score_out/score_in are given,
 * additionally accumulates the signed first-order Taylor terms of THIS pass,
 *   score_out[k] += sum_{c,r,s} W*dW_t ,  score_in[c] += sum_{k,r,s} W*dW_t
 * (the `multivariable=True` score is |sum_t ...|, ddpm_prune.py:60) so scores fall out of backward. */
typedef struct dp_wgrad_reduce_args {
  int32_t K, C, R, S, splits;
  const float* workspace; /* [splits][K][R*S*C] */
  float* dw;              /* [K][C][R][S], accumulated into */
  const float* w;         /* [K][C][R][S] or NULL */
  float* score_out;       /* [K] or NULL */
  float* score_in;        /* [C] or NULL */
  const float* bias_ws;   /* [splits][K] column sums of dy written by dp_conv2d_wgrad (dp_conv_args.bias_ws), or NULL */
  float* db;              /* [K] bias gradient, accumulated into (+= sum over splits, fixed order) */
} dp_wgrad_reduce_args;
int dp_conv2d_wgrad_reduce(const dp_wgrad_reduce_args* a, dp_stream_t stream);

/* OIHW -> w_ck [R*S][C][K] (fprop operand) and w_kc [R*S][K][C] (dgrad operand); either output may be NULL */
int dp_pack_conv_weight(const float* w_oihw, int32_t K, int32_t C, int32_t R, int32_t S, float* w_ck, float* w_kc,
                        dp_stream_t stream);

/* Operands of the tcgen05 path (3 x fp16 split, fp32-grade).  With s = the power of two that brings the tensor's max|w| below 2^14:
 *   hi = fp16(s*w), lo = fp16((s*w - hi) * 2^11), each in both K-major forms:
 *   kc_* [R*S][K][Cp] (fprop B operand, GEMM-K = C)   ck_* [R*S][C][Kp] (dgrad B operand, GEMM-K = K), where
 *   Cp = dp_tc_weight_row(C), Kp = dp_tc_weight_row(K) are the zero-padded row lengths in fp16 ELEMENTS: a multiple of 64 for rows
 *   longer than 64 (every 64-element TMA box row is then one aligned 128-byte line), else a multiple of 8 (16-byte row pitches).
 *   amax_w receives the weight's amax slot (the kernels derive s from it).  A NULL kc pair or ck pair is skipped. */
int dp_tc_weight_row(int channels);
int dp_pack_conv_weight_tc(const float* w_oihw, int32_t K, int32_t C, int32_t R, int32_t S, void* kc_hi, void* kc_lo,
                           void* ck_hi, void* ck_lo, uint32_t* amax_w, dp_stream_t stream);
/* amax slots.  dp_amax: *slot = max(*slot, bits(max |x[r*ld + c]|)) over a [rows][cols] fp32 view (atomicMax on the bit pattern of
 * |v|, which is order-independent: results are run-to-run identical); callers zero their slots once per pass with dp_zero_u32. */
int dp_amax(const float* x, int64_t ld, int64_t rows, int32_t cols, uint32_t* slot, dp_stream_t stream);
int dp_zero_u32(uint32_t* p, int64_t n, dp_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * bf16 tensor tier (conv_bf16.cu): tcgen05.mma kind::f16 on BF16 operands, fp32 accumulation — what torch.autocast(bfloat16) makes of
 * aten::convolution / linear in the finetune step (ddpm_train.py:200-208,255-261 `--mixed_precision bf16`; BASELINE configs[3]).
 * Operands are bf16 NHWC views (pixel stride in ELEMENTS, a multiple of 8) produced by dp_cvt_bf16 or by dp_groupnorm_fwd's y_bf16
 * output; outputs (y, dx, the wgrad workspace) are fp32 exactly as in dp_conv_args, so bias / temb / residual epilogues, the
 * split-K reduce and everything downstream are shared with the fp32-grade tier.
 * ------------------------------------------------------------------------------------------------ */
typedef struct dp_conv_bf16_args {
  int32_t N, H, W, C;
  int32_t P, Q, K;
  int32_t R, S, stride, pad_t, pad_l;
  int32_t flags;            /* DP_CONV_ACCUMULATE */
  int32_t splits;           /* wgrad */
  const void* x_bf16; int64_t ldx;    /* fprop / wgrad input  [N][H][W][ldx]  bf16 */
  const void* dy_bf16; int64_t lddy;  /* dgrad / wgrad input  [N][P][Q][lddy] bf16 */
  float* out; int64_t ld_out;         /* fprop: y [N][P][Q][ld_out] | dgrad: dx [N][H][W][ld_out]   fp32 */
  const void* w_bf16;       /* dp_pack_conv_weight_bf16: fprop kc [R*S][K][Cp] | dgrad ck [R*S][C][Kp], Cp/Kp = dp_bf16_weight_row */
  const float* bias; const float* rowadd; int64_t ld_rowadd; const float* residual; int64_t ld_res;   /* fprop epilogue, as dp_conv_args */
  float* workspace;         /* wgrad: [splits][K][R*S*C] fp32 partial sums (dp_conv2d_wgrad_reduce finishes) */
} dp_conv_bf16_args;
int dp_bf16_available(void);
int dp_bf16_weight_row(int channels);      /* packed weight row length: channels rounded up to 64 (one 128-byte TMA row) */
int dp_bf16_wgrad_ctile(int in_channels);  /* in-channel tile width of dp_conv2d_wgrad_bf16 (grid sizing for the split-K choice) */
int dp_conv2d_fprop_bf16(const dp_conv_bf16_args* a, dp_stream_t stream);
int dp_conv2d_dgrad_bf16(const dp_conv_bf16_args* a, dp_stream_t stream);
int dp_conv2d_wgrad_bf16(const dp_conv_bf16_args* a, dp_stream_t stream);
/* op: 0 fprop, 1 dgrad, 2 wgrad — DP_OK when the bf16 kernels take this geometry (pointers not needed), else DP_ERR_UNSUPPORTED */
int dp_conv_bf16_eligible(const dp_conv_bf16_args* a, int op);
/* fp32 [rows][ld] view with C valid channels -> bf16 (RNE) [rows][ld_dst], ld_dst a multiple of 8, pads zeroed */
int dp_cvt_bf16(const float* src, int64_t ld, int64_t rows, int32_t C, void* dst, int64_t ld_dst, dp_stream_t stream);
/* OIHW fp32 -> bf16 K-major operands kc [R*S][K][Cp] and ck [R*S][C][Kp] (either may be NULL) */
int dp_pack_conv_weight_bf16(const float* w_oihw, int32_t K, int32_t C, int32_t R, int32_t S, void* kc, void* ck, dp_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Batched strided GEMM  C[b] (=|+=) alpha * A[b] x B[b]   (attention core: aten::baddbmm/bmm,
 * attention_processor.py:341-357,452).  A(m,k) = A[b*a_bs + m*a_rs + k*a_cs], one of a_rs/a_cs must be 1;
 * B(k,n) = B[b*b_bs + k*b_rs + n*b_cs], one of b_rs/b_cs must be 1; C row-major with ldc.
 * ------------------------------------------------------------------------------------------------ */
typedef struct dp_gemm_args {
  int32_t M, N, Kd, batch;
  const float* A; int64_t a_rs, a_cs, a_bs;
  const float* B; int64_t b_rs, b_cs, b_bs;
  float* C; int64_t ldc, c_bs;
  float alpha;
  int32_t accumulate;
} dp_gemm_args;
int dp_gemm_batched(const dp_gemm_args* a, dp_stream_t stream);

/* Tensor-core batched GEMM for the attention core (attention_processor.py:341-357,452 and its backward):
 *   C[b][m][n] = alpha * sum_k A[b][m][k] * B[b][n][k]          (both operands K-contiguous, "NT")
 * A: [batch][H*W][Kg] fp32 view (pixel stride ld_a) — the token grid is the image grid so a 128-token tile is a TMA box;
 * B: given pre-split (dp_split_h3) as fp16 b_hi/b_lo [batch][N][Kg8]; C: [batch][H*W][N] view (ldc); amax_a / amax_b: amax slots of
 * A and of the matrix B was split from.  Runs on the persistent tcgen05 kernel; returns DP_ERR_UNSUPPORTED when the shape is not
 * eligible (H*W % 128, alignment) so the caller can fall back to dp_gemm_batched. */
typedef struct dp_gemm_nt_args {
  int32_t batch, H, W, Kg, N;
  const float* A; int64_t ld_a;
  const void* b_hi; const void* b_lo;
  float* C; int64_t ldc;
  float alpha;
  const uint32_t* amax_a; const uint32_t* amax_b;
  uint32_t* amax_out;  /* optional: accumulates max|C| */
} dp_gemm_nt_args;
int dp_gemm_nt_tc(const dp_gemm_nt_args* a, dp_stream_t stream);
/* fp16 hi / lo' split (see dp_pack_conv_weight_tc) of a batched [rows][cols] fp32 matrix (row stride ld, batch stride bs) with the scale of
 * its amax slot (dp_amax over the same matrix must have run), written densely as [batch][rows][cols8] — or transposed,
 * [batch][cols][rows8] — with the row length rounded up to 8 elements (zero pad). */
int dp_split_h3(const float* x, int64_t ld, int64_t bs, int32_t batch, int32_t rows, int32_t cols, int32_t transpose,
                const uint32_t* amax, void* hi, void* lo, dp_stream_t stream);
/* out[b][c][r] = in[b][r][c] for dense [batch][rows][cols] */
int dp_transpose_batched(const float* in, float* out, int32_t batch, int32_t rows, int32_t cols, dp_stream_t stream);

/* row softmax over [rows][cols] fp32 (attention_processor.py:352, upcast_softmax) and its backward
 * dS = P * (dP - sum_j dP*P); in-place allowed (out == in). */
int dp_softmax_fwd(const float* s, float* p, int64_t rows, int32_t cols, dp_stream_t stream);
int dp_softmax_bwd(const float* p, const float* dp, float* ds, int64_t rows, int32_t cols, uint32_t* amax_ds, dp_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * GroupNorm (+ fused SiLU).  Replaces aten::native_group_norm(+backward) and aten::silu(+backward) at
 * resnet.py:592-597,623-630, unet_2d.py:302-303, attention_processor.py:437 (silu = 0 there).
 * x,y: [N][HW][C] views; stats saved as mean/rstd [N][G] for backward.
 * ------------------------------------------------------------------------------------------------ */
typedef struct dp_gn_args {
  int32_t N, HW, C, G;
  float eps;
  int32_t silu;          /* 1: y = silu(gn(x)); the sigmoid runs on the special-function unit (ex2.approx + rcp.approx, ~3e-7 relative) */
  const float* x; int64_t ldx;
  float* y; int64_t ldy; /* fwd: output | bwd: unused */
  const float* gamma; const float* beta;
  float* mean; float* rstd;   /* [N][G]: fwd writes, bwd reads */
  /* backward only */
  const float* dy; int64_t lddy;  /* grad w.r.t. the (post-SiLU) output */
  float* dx; int64_t lddx;        /* grad w.r.t. x */
  const float* dx_add; int64_t ldadd; /* optional: dx = dx_add + (gn grad)  (residual path / accumulation; may alias dx) */
  const float* dx_add2; int64_t ldadd2; /* optional second addend (e.g. the residual branch's dY while dx_add == dx) */
  float* dgamma; float* dbeta;    /* [C], accumulated into (+=) */
  void* workspace;                /* dp_groupnorm_workspace_bytes() */
  /* dropout folded behind the SiLU (resnet.py:631): keep-mask from a counter-based hash of (seed, element index / 4), one 16-bit uniform
   * per element: keep iff u16 >= round(p * 65536), survivors scaled by 65536 / (65536 - round(p * 65536)); the backward regenerates
   * the same mask from the element index ; p = 0 disables */
  float dropout_p; uint64_t dropout_seed;
  const uint64_t* dropout_seed_dev; /* optional DEVICE scalar added to dropout_seed (lets a captured CUDA graph
                                       draw a fresh mask every replay) */
  /* bf16 tier: the forward additionally (or, with y == NULL, only) writes its output rounded to bf16 (RNE) as the next
   * convolution's operand — [N][HW][ldyb] with ldyb a multiple of 8; pad columns are left untouched (never read: TMA bounds) */
  void* y_bf16; int64_t ldyb;
  /* optional amax slots (dp_amax semantics) of the tensors this call writes: forward y, backward dx — the tensor-core convolution
   * that consumes them then needs no separate dp_amax pass */
  uint32_t* amax_y; uint32_t* amax_dx;
  /* optional, backward: caller-owned [N][2][C] floats that outlive the shared workspace.  When set, dp_groupnorm_bwd leaves the
   * per-image channel sums there and does NOT touch dgamma / dbeta; dp_groupnorm_bwd_param adds them later, on any stream ordered
   * after the dp_groupnorm_bwd call (parameter gradients feed nothing inside the pass: they need not sit on the dx chain).
   * Not for the one-pixel LayerNorm shapes (DP_ERR_UNSUPPORTED). */
  float* fin;
} dp_gn_args;
size_t dp_groupnorm_workspace_bytes(int32_t N, int32_t HW, int32_t C, int32_t G);
int dp_groupnorm_fwd(const dp_gn_args* a, dp_stream_t stream);
/* dp_groupnorm_fwd that also (with a->y == NULL: only) writes its output already split for the tensor-core convolutions, in the
 * DP_CONV_X_SPLIT layout [N][HW][2][ldys] fp16 (ldys a multiple of 8, >= C; pad channels untouched).  The scale comes from a bound
 * known before anything is written, B = max|gamma| * sqrt(C/G * HW - 1) + max|beta| (over a group of n values |x - mean| <=
 * sqrt(n - 1) * std), widened for SiLU and dropout; B goes to a->amax_y (required) in place of the measured max|y|.  Single-launch
 * float4 path only (C % 4 == 0, 16-byte aligned views): DP_ERR_UNSUPPORTED otherwise. */
int dp_groupnorm_fwd_split(const dp_gn_args* a, void* y_split, int64_t ldys, dp_stream_t stream);
int dp_groupnorm_bwd(const dp_gn_args* a, dp_stream_t stream);
/* dgamma[c] += sum_n fin[n][1][c], dbeta[c] += sum_n fin[n][0][c] (fixed order) — the tail of native_group_norm_backward for a
 * dp_groupnorm_bwd call that was given `fin` */
int dp_groupnorm_bwd_param(const dp_gn_args* a, dp_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Small fused pointwise / reduction ops of the path
 * ------------------------------------------------------------------------------------------------ */
/* y = silu(x) ; dx (=|+=) dy * silu'(x)      (resnet.py:616 on temb, embeddings.py:205) */
int dp_silu_fwd(const float* x, float* y, int64_t n, dp_stream_t stream);
int dp_silu_bwd(const float* x, const float* dy, float* dx, int64_t n, int32_t accumulate, dp_stream_t stream);

/* GEGLU feed-forward gate of the LDM transformer blocks (ldm_exp/ldm/modules/attention.py:37-44): u = [a | gate] ([rows][2*inner]),
 * out = a * gelu(gate) (exact erf GELU); backward writes du = [dout * gelu(gate) | dout * a * gelu'(gate)]. */
int dp_geglu_fwd(const float* u, int64_t ldu, float* out, int64_t ldo, int64_t rows, int32_t inner, dp_stream_t stream);
int dp_geglu_bwd(const float* u, int64_t ldu, const float* dout, int64_t lddo, float* du, int64_t lddu, int64_t rows, int32_t inner,
                 dp_stream_t stream);

/* out[b][0:half]=sin(t_b*f_i), out[b][half:]=cos(...) (swapped if flip)  — embeddings.py:44-57; freqs [half] */
int dp_timestep_embedding(const int64_t* t, const float* freqs, float* out, int32_t B, int32_t half, int32_t flip,
                          dp_stream_t stream);

/* x_t = sqrt(acp[t_b])*x0 + sqrt(1-acp[t_b])*eps — scheduling_ddpm.py:415-428.  x0/noise NCHW; out NHWC if
 * out_nhwc else NCHW.  acp: alphas_cumprod table [T]. */
int dp_add_noise(const float* x0, const float* noise, const int64_t* t, const float* acp, float* out, int32_t B,
                 int32_t C, int32_t H, int32_t W, int32_t out_nhwc, int64_t ld_out /* NHWC pixel stride, 0 = C */,
                 dp_stream_t stream);

int dp_nchw_to_nhwc(const float* in, float* out, int64_t ld_out, int32_t N, int32_t C, int32_t H, int32_t W,
                    dp_stream_t stream);
int dp_nhwc_to_nchw(const float* in, int64_t ld_in, float* out, int32_t N, int32_t C, int32_t H, int32_t W,
                    int32_t accumulate, dp_stream_t stream);

/* loss = scale_loss * sum((pred-target)^2) ; grad = scale_grad * (pred-target)
 * (F.mse_loss ddpm_prune.py:101: scale_loss = 1/numel, scale_grad = 2/numel;
 *  ddpm_train.py:459: scale_loss = 1/B, scale_grad = 2/B).  Deterministic two-stage reduction.
 *  partial: workspace of dp_mse_partials(n) floats. */
int64_t dp_mse_partials(int64_t n);
int dp_mse_loss_grad(const float* pred, const float* target, float* grad, int64_t n, float scale_loss,
                     float scale_grad, float* partial, float* loss_out, dp_stream_t stream);

/* nearest x2 (resnet.py:155) and its backward (sum of the 2x2 children), NHWC views */
int dp_upsample2x_fwd(const float* x, int64_t ldx, float* y, int64_t ldy, int32_t N, int32_t H, int32_t W, int32_t C,
                      dp_stream_t stream);
int dp_upsample2x_bwd(const float* dy, int64_t lddy, float* dx, int64_t lddx, int32_t N, int32_t H, int32_t W,
                      int32_t C, int32_t accumulate, dp_stream_t stream);

/* out[s][c] (=|+=) sum_{r < seg_rows} x[(s*seg_rows + r)*ld + c]   (bias / temb gradients; fixed order) */
int dp_colsum(const float* x, int64_t ld, int64_t rows, int32_t cols, int64_t seg_rows, float* out, int64_t ld_out,
              int32_t accumulate, dp_stream_t stream);

/* y = a + b over an NHWC view (used where an add cannot be folded into a GEMM epilogue) */
int dp_add_views(const float* a, int64_t lda, const float* b, int64_t ldb, float* y, int64_t ldy, int64_t rows,
                 int32_t cols, dp_stream_t stream);
/* y = a over a [rows][cols] view (device to device, on the stream): gathers the to_q / to_k / to_v weights of an attention block
 * (attention_processor.py:432-441) into the one [3 inner][C] operand their fused projection reads, whenever the weights change */
int dp_copy_rows(const float* a, int64_t lda, float* y, int64_t ldy, int64_t rows, int32_t cols, dp_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Taylor importance reductions — torch_pruning TaylorImportance.__call__
 * (ddpm_exp/torch_pruning/importance.py:385-418).  For a weight viewed as [O][I][RS] and its accumulated grad:
 *   out_*[o] over (i,rs), in_*[i] over (o,rs) of   sum w*dw (signed) | sum |w*dw| | sum (w*dw)^2.
 * Each of the six outputs may be NULL.  GroupNorm gamma: call with I = RS = 1 and use out_abs.
 * ------------------------------------------------------------------------------------------------ */
typedef struct dp_taylor_args {
  int32_t O, I, RS;
  const float* w; const float* dw;
  float* out_signed; float* out_abs; float* out_sq;  /* [O] */
  float* in_signed; float* in_abs; float* in_sq;     /* [I] */
} dp_taylor_args;
int dp_taylor_reduce(const dp_taylor_args* a, dp_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Finetune tail over flat fp32 arenas — ddpm_train.py:462-469:
 *   clip_grad_norm_(1.0) -> torch.optim.Adam.step -> EMAModel.step (training_utils.py:201,216)
 * dp_sumsq: deterministic sum of squares (two-stage) -> out[0].  dp_adam_clip_ema reads the device scalar
 * *sumsq (no host sync), clips, applies Adam (torch's op order) and the EMA lerp in one pass.
 * ------------------------------------------------------------------------------------------------ */
int64_t dp_sumsq_partials(int64_t n);
int dp_sumsq(const float* x, int64_t n, float* partial, float* out, dp_stream_t stream);
typedef struct dp_adam_args {
  int64_t n;
  float* p; const float* g; float* m; float* v; float* ema; /* ema nullable */
  const float* sumsq;   /* device scalar: total grad sum of squares; NULL = no clipping */
  /* hyper-parameters as doubles: the derived constants (1-beta1, 1-beta2, lr/(1-beta1^t), 1-ema_decay ...) are formed
   * in double on the host and rounded once to fp32, exactly like the Python scalars torch feeds its kernels */
  double max_norm, lr, beta1, beta2, eps, ema_decay;
  int32_t step;         /* 1-based; used for the bias corrections when step_scalars == NULL */
  float grad_scale;     /* multiplies g before everything (1/world for DDP mean) */
  const float* step_scalars; /* optional DEVICE [2] = {lr/(1-beta1^t), sqrt(1-beta2^t)} so a captured CUDA graph can be
                                replayed for every step (host-computed kernel arguments would be frozen) */
} dp_adam_args;
int dp_adam_clip_ema(const dp_adam_args* a, dp_stream_t stream);

/* One DDIM update (scheduling_ddim.py:324-390, epsilon prediction), elementwise over n values:
 *   x0 = (x - sqrt_beta_t * eps) / sqrt_alpha_t ; if clip > 0: x0 = clamp(x0, -clip, clip)
 *   out = sqrt_alpha_prev * x0 + dir_coef * eps (+ sigma * noise)        noise may be NULL when sigma == 0 */
int dp_ddim_step(const float* x, const float* eps, const float* noise, float* out, int64_t n, float sqrt_beta_t, float sqrt_alpha_t,
                 float clip, float sqrt_alpha_prev, float dir_coef, float sigma, dp_stream_t stream);

/* y[i] = x[i] * s  (gradient averaging after all-reduce etc.) */
int dp_scale(float* x, int64_t n, float s, dp_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DPB200_H */
