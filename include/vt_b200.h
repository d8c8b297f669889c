/*
 * vt_b200.h — C ABI of the B200 (sm_100a) video-transformer hot-path kernels.
 *
 * Drop-in boundary (SURVEY.md §8b): the reference has no FFI layer of its own — its hot path is the
 * forward/backward of the nn.Modules in transformer.py / video_transformer.py, executed by stock
 * ATen/cuBLAS/cuDNN calls.  This library is what a maintainer binds *underneath* those modules
 * (ctypes stub in INTEGRATION.md); each entry point names the reference call site it replaces
 * (paths relative to the reference repo root).
 *
 * Conventions
 *  - every function: int fn(const <params>*, void* cuda_stream); 0 = ok, non-zero = error
 *    (message via vt_last_error).  No exceptions, no abort, no fallback: unsupported shapes are errors.
 *  - all pointers are device pointers owned by the caller (PyTorch caching allocator); kernels are
 *    enqueued on `cuda_stream` and never allocate, free, synchronise or retain pointers.
 *  - bf16 = raw uint16 storage of __nv_bfloat16; "rows" are contiguous along the last dimension.
 *  - re-entrant: callable from the Python main thread (forward) and the autograd thread (backward).
 */
#ifndef VT_B200_H
#define VT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VT_ABI_VERSION 1

int vt_version(void);
/* copies the calling thread's last error message (NUL terminated) into buf; returns its length */
int vt_last_error(char* buf, size_t buf_bytes);
/* number of SMs of the current device (grid sizing is done inside the library) */
int vt_sm_count(void);
/* leave n SMs free of the persistent GEMM CTAs (each pins an SM's whole shared memory) so that NCCL's all-reduce
 * kernels, issued on a side stream while backward is still running, can be scheduled; 0 restores the default */
int vt_set_reserved_sms(int n);
/* number of kernels this library has launched in this process (mod 2^31); bench.py's gpu_launches */
int vt_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * GEMM on tcgen05 tensor cores:  acc[M,N] = sum_k A[m,k] * B[n,k]   (bf16 x bf16 -> fp32 in TMEM)
 * Operands are fed by TMA into 128B-swizzled shared memory.
 *   a_mn_major = 0 : A stored row-major [M, K] (leading dim lda)      "K-major"
 *   a_mn_major = 1 : A stored row-major [K, M] (leading dim lda)      "MN-major" (no transpose copy)
 *   b_mn_major = 0 : B stored row-major [N, K] (leading dim ldb)      (nn.Linear weight layout)
 *   b_mn_major = 1 : B stored row-major [K, N]
 * Replaces: nn.Linear forward (F.linear -> cuBLASLt addmm) at transformer.py:167 (qkv), :175 (proj),
 *   :267 (temporal_fc), :501-505 (FFN), the Conv2d/Conv3d patch projection :116-126 after im2col,
 *   and autograd's dgrad / wgrad GEMMs of the same layers.
 *
 * Epilogues (thread = accumulator row, fused in the TMEM->register drain):
 *   VT_EPI_BF16  : out_bf16[orow(m), n]  = s(m) * (acc + bias[n])
 *   VT_EPI_F32   : out_f32 [orow(m), n]  = s(m) * (acc + bias[n]) + (aux ? aux_f32[arow(m), n] : 0)
 *                  (residual add / pos+time-embed add / fp32 gradients)
 *   VT_EPI_GELU  : out_bf16[m,n] = z = acc + bias[n];  out2_bf16[m,n] = gelu_erf(z)     (transformer.py:501-503)
 *   VT_EPI_DGELU : out_bf16[m,n] = acc * gelu_erf'(aux_bf16[m,n])                        (autograd of nn.GELU)
 * orow(m) = out_row ? out_row[m] : m  (negative => row skipped);  arow likewise (negative => no addend);  s(m) = row_scale ? row_scale[m] : 1
 * (row_scale carries DropPath's per-row mask/keep factor, transformer.py:34-42, and the 1/T of the cls mean :371-373).
 *
 * Split-K: when `workspace` is given and the tile count under-fills the GPU (weight gradients:
 * K = tokens), K is split; partial tiles go to the fp32 workspace and are summed by a second kernel.
 * Only with VT_EPI_F32, no row maps.
 * ------------------------------------------------------------------------------------------- */
enum { VT_EPI_BF16 = 0, VT_EPI_F32 = 1, VT_EPI_GELU = 2, VT_EPI_DGELU = 3 };

typedef struct {
  const void* a;      /* bf16 */
  const void* b;      /* bf16 */
  int64_t lda, ldb;   /* leading dims in elements (multiples of 8) */
  int32_t M, N, K;
  int32_t a_mn_major, b_mn_major;
  int32_t epilogue;
  const float* bias;       /* [N] or NULL */
  void* out;               /* bf16 or fp32 per epilogue */
  void* out2;              /* VT_EPI_GELU only */
  const void* aux;         /* fp32 (VT_EPI_F32) or bf16 (VT_EPI_DGELU) or NULL */
  int64_t ldo, ldo2, ldaux;
  const int32_t* out_row;  /* [M] or NULL */
  const int32_t* aux_row;  /* [M] or NULL */
  const float* row_scale;  /* [M] or NULL */
  void* workspace;         /* fp32 scratch for split-K or NULL */
  int64_t workspace_bytes;
  int32_t force_splits;    /* 0 = heuristic, >0 = exactly this many K splits (tests) */
  int32_t force_bn;        /* 0 = heuristic, 128 / 192 / 256 (tests) */
  int32_t force_cluster;   /* 0/1 = single CTAs, 2 = clusters of 2 CTAs along M sharing each B tile by TMA multicast,
                              3 = CTA pairs issuing tcgen05.mma.cta_group::2 (256 x BN tiles, half of B per SM) */
  void* debug;             /* diagnostics only: int64 [grid][16] clock64 stamps of the kernel's phases, or NULL */
  /* Affine description of out_row / aux_row for VT_EPI_F32 with aux (the residual scatter of the divided space-time blocks),
   * map_period = 0: none.  GEMM row m -> outer = m / map_period, inner = m % map_period.  Rows with inner < map_skip are
   * "special" (the per-frame cls replicas of the spatial pass): no addend, written to out + map_special_base +
   * outer * map_special_stride (dropped when map_special_base < 0).  Every other row reads its addend from / writes its
   * result to element offset  map_base + (outer % map_tcount) * map_stride_t + (inner - map_skip) * map_stride_p +
   * (outer / map_tcount) * map_stride_b  of aux / out.  With it the epilogue moves whole 32 x 32 boxes by TMA through a
   * tensor map (col, row in sample, sample) of the token stream (reference einops: transformer.py:250, :279-280, :352-356,
   * :375-377) instead of per-thread rows; the out_row / aux_row arrays, when also given, must describe the same mapping
   * (they serve the generic epilogue, which also covers map_tcount > 1: the element-strided boxes that case needs fault
   * on hardware and stay switched off). */
  int32_t map_period, map_skip, map_tcount;
  int32_t force_tail;      /* 0 = heuristic, 1 = never cut the partial last row of tiles into narrow units, 2 = prefer to */
  int64_t map_stride_t, map_stride_p, map_stride_b, map_base;
  int64_t map_special_base, map_special_stride;
  const float* bias2;      /* VT_EPI_F32 with aux only: out = s(m) * (acc + bias[n]) + bias2[n] + aux — the bias of a second
                              linear layer folded into this GEMM (temporal_fc after proj, transformer.py:264-267) */
  int32_t out_zeroed;      /* split-K accumulates into `out` by TMA reduce-add and normally zeroes it first; 1 = the caller
                              already did (a gradient arena / DDP bucket zeroed once per step) */
} vt_gemm_params;

int vt_gemm(const vt_gemm_params* p, void* stream);

/* ---------------------------------------------------------------------------------------------
 * LayerNorm over the last dim (biased variance), fp32 statistics, one warp per row.
 * Replaces nn.LayerNorm at transformer.py:257 / :359 / :439 / :519 and video_transformer.py:251,
 * fused with the einops regroupings around it (transformer.py:250, :352-356): row m of the output
 * is the normalised row in_row[m] of x, so '(b t) p' / '(b p) t' orders and the per-frame cls copy
 * cost no separate pass.
 *   y_bf16[m,:] = (x[in_row ? in_row[m] : m, :] - mean) * rstd * gamma + beta ;  mean/rstd saved.
 * D must be a multiple of 128 and <= 1024.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  const float* x; int64_t ldx;
  const int32_t* in_row;
  const float* gamma; const float* beta;
  void* y;            /* bf16 [rows, D] (or fp32 when y_fp32 != 0) */
  float* mean; float* rstd;   /* [rows] */
  int32_t rows, D;
  float eps;
  int32_t y_fp32;
} vt_ln_fwd_params;
int vt_layernorm_fwd(const vt_ln_fwd_params* p, void* stream);

/* LayerNorm backward.  g = dy*gamma ; dx = rstd*(g - mean(g) - xhat*mean(g*xhat)).
 * Scatter: t = out_row ? out_row[m] : m.
 *   t >= 0 : dx[t,:]        = dx_row + (dres ? dres[t,:] : 0)      (adds the residual-path gradient)
 *   t <  0 : dx_aux[-t-1,:] = dx_row                                (replicated cls rows, summed by caller)
 * dgamma/dbeta: per-CTA partials into `partials` ([blocks, 2, D] fp32, blocks = vt_ln_bwd_blocks()),
 * then reduce with vt_reduce_rows. */
typedef struct {
  const void* dy; int32_t dy_fp32;      /* bf16 [rows, D] (fp32 if dy_fp32) */
  const float* x; int64_t ldx; const int32_t* in_row;
  const float* mean; const float* rstd; const float* gamma;
  const float* dres; float* dx; int64_t lddx;
  float* dx_aux;
  const int32_t* out_row;
  float* partials;
  int32_t rows, D;
} vt_ln_bwd_params;
int vt_ln_bwd_blocks(int32_t rows);
int vt_layernorm_bwd(const vt_ln_bwd_params* p, void* stream);

/* out[j] = (accumulate ? out[j] : 0) + scale * sum_{s<S} in[s*stride + j],  j < n (n % 4 == 0) */
typedef struct { const float* in; float* out; int64_t stride; int32_t S; int64_t n; int32_t accumulate; float scale; } vt_reduce_params;
int vt_reduce_rows(const vt_reduce_params* p, void* stream);

/* Column sums of a bf16 [M,N] matrix (bias gradients): out_f32[n] = sum_m in[m,n].
 * workspace: fp32 [vt_colsum_chunks(M), N].  Deterministic (fixed summation order) in both forms. */
typedef struct { const void* in; int64_t ld; int32_t M, N; float* out; float* workspace;
                 int32_t* counters; /* optional: >= ceil(N/64) zeroed ints -> single-launch form (the last CTA sums the partials and
                                       re-zeroes its counter); NULL -> partials are reduced by a second launch */ } vt_colsum_params;
int vt_colsum_chunks(int32_t M);
int vt_colsum_bf16(const vt_colsum_params* p, void* stream);

/* fp32 -> bf16 casts.  vt_cast: flat.  vt_gather_cast: out[m,:] = bf16(src[in_row[m],:] * row_scale[m])
 * (gradient of the residual scatter + DropPath scale; in_row < 0 => zeros). */
typedef struct { const float* src; void* dst; int64_t n; } vt_cast_params;
int vt_cast_f32_bf16(const vt_cast_params* p, void* stream);
typedef struct { const float* src; int64_t lds; const int32_t* in_row; const float* row_scale; void* dst; int32_t rows, D; } vt_gather_cast_params;
int vt_gather_cast_bf16(const vt_gather_cast_params* p, void* stream);

/* Exact-erf GELU on bf16 (nn.GELU default, transformer.py:483 / :502) as stand-alone bandwidth kernels:
 *   vt_gelu_fwd_bf16: out = gelu(z)            vt_gelu_bwd_bf16: out = dh * gelu'(z)
 * The FFN uses them instead of the fused GEMM epilogues when the epilogue's erf math would out-cost the tile's
 * MMAs (4 erf per 4 columns in 8 epilogue warps); both forms are kept and tested. n = element count (n % 8 == 0). */
typedef struct { const void* z; const void* dh; void* out; int64_t n; } vt_gelu_params;
int vt_gelu_fwd_bf16(const vt_gelu_params* p, void* stream);
int vt_gelu_bwd_bf16(const vt_gelu_params* p, void* stream);

/* cls rows of the divided space-time blocks in one launch:  dst[b, :] = src[b, :] + scale * sum_t extra[b, t, :]
 * (extra NULL: row copy).  src / dst: fp32 rows b * stride apart; extra: fp32 [B, T, D] with batch stride extra_bs.
 * Replaces the cls passthrough of the temporal block and `cls + mean_t(cls replicas)` of the spatial block
 * (transformer.py:282-283, :371-377) and their adjoints. */
typedef struct { const float* src; int64_t src_stride; const float* extra; int64_t extra_bs; int32_t T; float scale;
                 float* dst; int64_t dst_stride; int32_t B, D; } vt_cls_rows_params;
int vt_cls_rows(const vt_cls_rows_params* p, void* stream);

/* The two producers of a layer's dY that also emit its column sums (= the bias gradient autograd's sum over tokens gives
 * nn.Linear, transformer.py:175 / :267 / :505 / :501): vt_gather_cast_bf16 + vt_colsum_bf16, and vt_gelu_bwd_bf16 +
 * vt_colsum_bf16, in one pass each.  colsum fp32 [D] / [N]; workspace fp32 [workspace_rows, D] with workspace_rows >=
 * vt_*_blocks(rows).  Sums are over the bf16-rounded outputs, in a fixed order. */
typedef struct { const float* src; int64_t lds; const int32_t* in_row; const float* row_scale; void* dst; int32_t rows, D;
                 float* colsum; float* workspace; int32_t workspace_rows;
                 int32_t unscaled_sums;   /* 1: colsum is [2, D] — row 1 = sums of the rows before row_scale; workspace [rows, 2 D] */
               } vt_gather_cast_colsum_params;
int vt_gather_cast_colsum_blocks(int32_t rows);
int vt_gather_cast_colsum_bf16(const vt_gather_cast_colsum_params* p, void* stream);
typedef struct { const void* z; const void* dh; void* out; int32_t M, N; float* colsum; float* workspace;
                 int32_t workspace_rows; } vt_gelu_bwd_colsum_params;
int vt_gelu_bwd_colsum_blocks(int32_t M);
int vt_gelu_bwd_colsum_bf16(const vt_gelu_bwd_colsum_params* p, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Multi-head softmax attention core on a packed qkv tensor (no projection):
 *   qkv bf16 [Bp, N, 3, H, hd] (the layout produced by transformer.py:167's reshape), hd = 64
 *   ctx bf16 [Bp, N, H*hd] = softmax(q k^T * scale) v      (transformer.py:170-174)
 *   lse fp32 [Bp, H, N]   (saved for backward);  probs fp32 [Bp,H,N,N] optional (Attention returns it, :177)
 * Three kernels behind one entry point: a tcgen05/TMEM flash kernel for the spatial pass (N = 197: S, dP and the
 * gradient accumulators in TMEM, K/V resident in shared memory, P/dS re-read transposed through MN-major UMMA
 * descriptors), a warp-per-problem kernel for the temporal pass (N = 8, 18 816 problems/layer), and a generic
 * warp-per-query kernel for any other N <= 256 (ViViT N = 9, tests, probs output).
 * ------------------------------------------------------------------------------------------- */
enum { VT_ATTN_AUTO = 0, VT_ATTN_GENERIC = 1, VT_ATTN_TCGEN05 = 2, VT_ATTN_WARP8 = 3 };
typedef struct {
  const void* qkv; void* ctx; float* lse; float* probs;
  int32_t Bp, N, H, hd; float scale;
  int32_t impl;   /* VT_ATTN_AUTO picks: N == 8 -> warp-per-problem kernel; 32 < N <= 256 -> tcgen05 flash kernel; else generic */
} vt_attn_fwd_params;
int vt_attn_fwd(const vt_attn_fwd_params* p, void* stream);
typedef struct {
  const void* qkv; const void* ctx; const void* dctx; const float* lse; void* dqkv;
  int32_t Bp, N, H, hd; float scale;
  int32_t impl;
} vt_attn_bwd_params;
int vt_attn_bwd(const vt_attn_bwd_params* p, void* stream);
/* diagnostics only: int64 [grid][32] clock64 phase stamps of the tcgen05 attention kernels (NULL disables) */
int vt_debug_buffer(void* device_ptr);

/* ---------------------------------------------------------------------------------------------
 * Patch / tubelet embedding operand: non-overlapping Conv2d k16 s16 (transformer.py:116-120,:145-147)
 * or Conv3d k(tube,16,16) (:122-126,:141-143) == im2col + GEMM.
 *   x fp32 [B, T, C, H, W] -> cols bf16 [B*(T/tube)*(H/ph)*(W/pw), C*tube*ph*pw], k = ((c*tube+dt)*ph+i)*pw+j
 * vt_col2im is its adjoint (gradient w.r.t. the clip), fp32 out, from fp32 cols.
 * ------------------------------------------------------------------------------------------- */
typedef struct { const float* x; void* cols; int32_t B, T, C, H, W, tube, ph, pw; } vt_im2col_params;
int vt_im2col_bf16(const vt_im2col_params* p, void* stream);
/* Same operand from the decoder's uint8 clip (SURVEY §8f rank 2; data_transform.py:52-64 ToTensor + :534-539 Normalize fused in):
 *   x u8 [B, T, H, W, C] (channels last) -> cols[row, k] = bf16(x * scale[c] + shift[c]),  scale = 1/(255 std), shift = -mean/std */
typedef struct { const uint8_t* x; const float* scale; const float* shift; void* cols; int32_t B, T, C, H, W, tube, ph, pw; } vt_im2col_u8_params;
int vt_im2col_u8_bf16(const vt_im2col_u8_params* p, void* stream);
typedef struct { const float* cols; float* dx; int32_t B, T, C, H, W, tube, ph, pw; } vt_col2im_params;
int vt_col2im_f32(const vt_col2im_params* p, void* stream);

/* ---------------------------------------------------------------------------------------------
 * MaskFeat HOG target (dataset.py:39-45 -> skimage.feature.hog x3 + 2x2 cell regroup).
 *   frames u8 [F, H, W, 3] (H, W multiples of 16) -> feat fp32 [F, H/16, W/16, 108]
 *   bins (optional) u8 [F, 3, H, W]: orientation bin 0..8 per pixel/channel, 9 = no bin
 *   lut u8 [511*511]: bin of integer gradient (gy+255, gx+255), built on the host with numpy
 * ------------------------------------------------------------------------------------------- */
typedef struct { const uint8_t* frames; const uint8_t* lut; float* feat; uint8_t* bins; int32_t F, H, W; } vt_hog_params;
int vt_hog(const vt_hog_params* p, void* stream);

/* =============================================================================================
 * MaskFeat / MViT path (SURVEY §8 a13-a15).  Block arithmetic = pytorchvideo MultiScaleBlock as configured at
 * video_transformer.py:764-785 (restated in oracle/mvit_oracle.py); head dim is 96 in every block.
 * vt_layernorm_fwd/bwd additionally accept D = 32..256 in steps of 32 (block widths 96 and 192) without row maps.
 * ============================================================================================= */

/* Depthwise Conv3d pooling of one of q/k/v + LayerNorm(hd)  (pytorchvideo _attention_pool, pool_mode="conv"):
 *   element (b, n, h, c) of the input lives at in[b*in_bs + n*in_rs + h*hd + c] (bf16; n = 0 is the cls row, rows
 *   1.. are the (T,Hin,Win) tokens, t-major) — i.e. a q/k/v slice of the fused projection output is read in place.
 *   pooled fp32 [B,H,1+Lo,hd] = cls row copied, other rows conv3d(kernel 3x3x3, stride (st,sh,sw), padding 1, groups=hd)
 *   out    bf16 [B,H,1+Lo,hd] = LayerNorm(pooled; gamma, beta, eps) over hd;  mean/rstd [B*H*(1+Lo)] saved.
 * Lo = To*Ho*Wo with To = (T + 2 - 3)/st + 1 etc.   w: fp32 [hd, 27] (nn.Conv3d weight [hd,1,3,3,3]). */
typedef struct {
  const void* in; int64_t in_bs, in_rs;
  const float* w; const float* gamma; const float* beta;
  float* pooled; void* out; float* mean; float* rstd;
  int32_t B, H, hd, T, Hin, Win, st, sh, sw, To, Ho, Wo;
  float eps;
} vt_pool_fwd_params;
int vt_pool_fwd(const vt_pool_fwd_params* p, void* stream);

/* Backward of vt_pool_fwd.  dout: gradient of `out` (bf16, or fp32 if dout_fp32).  Produces
 *   din (bf16, addressed like `in` with din_bs/din_rs: every (b,n,h,:) is written), dw [hd,27], dgamma, dbeta [hd].
 * scratch: fp32, at least vt_pool_bwd_scratch(rows_out, hd) floats (dpooled + per-CTA partial sums). */
typedef struct {
  const void* dout; int32_t dout_fp32;
  const float* pooled; const float* mean; const float* rstd; const float* gamma;
  const void* in; int64_t in_bs, in_rs; const float* w;
  void* din; int64_t din_bs, din_rs;
  float* dw; float* dgamma; float* dbeta;
  float* scratch; int64_t scratch_floats;
  int32_t B, H, hd, T, Hin, Win, st, sh, sw, To, Ho, Wo;
} vt_pool_bwd_params;
int vt_pool_bwd_scratch(int32_t rows_out, int32_t hd);   /* floats */
int vt_pool_bwd(const vt_pool_bwd_params* p, void* stream);

/* Softmax attention with separate, strided Q / K / V and Nq != Nk (pooling attention):
 *   element (b, h, n, c) of q at q[b*q_bs + h*q_hs + n*q_rs + c] (bf16), same for k, v, o (and dout, dq).
 *   o = softmax(scale * q k^T) v ;  lse fp32 [B,H,Nq] = log sum exp(scale * q k^T).
 * Two implementations: tcgen05 flash kernels (vt_xattention_tc.cu: head dim 96 staged as 128 padded columns = two
 * 128-byte swizzle atoms, S / dP / accumulators in TMEM, K/V streamed by TMA) and CUDA-core kernels for arbitrary
 * strides (two threads per query row, K/V tiles staged in shared memory). */
enum { VT_XATTN_AUTO = 0, VT_XATTN_SIMT = 1, VT_XATTN_TCGEN05 = 2 };
typedef struct {
  const void* q; const void* k; const void* v; void* o; float* lse;
  int64_t q_bs, q_hs, q_rs, k_bs, k_hs, k_rs, v_bs, v_hs, v_rs, o_bs, o_hs, o_rs;
  int32_t B, H, Nq, Nk, hd; float scale;
  int32_t impl;   /* VT_XATTN_AUTO: tcgen05 kernels when every operand is token-major ([B,N,H*hd] slices) or head-major
                     contiguous ([B,H,N,hd]) with 16-byte aligned rows, else the CUDA-core kernels */
} vt_xattn_fwd_params;
int vt_xattn_fwd(const vt_xattn_fwd_params* p, void* stream);
/* dq: bf16 with its own strides.  dk, dv: fp32 [B,H,Nk,hd] contiguous (zeroed by the call, accumulated with atomics).
 * delta: fp32 scratch [B,H,Nq]. */
typedef struct {
  const void* q; const void* k; const void* v; const void* o; const void* dout; const float* lse;
  float* delta; void* dq; float* dk; float* dv;
  int64_t q_bs, q_hs, q_rs, k_bs, k_hs, k_rs, v_bs, v_hs, v_rs, o_bs, o_hs, o_rs, dq_bs, dq_hs, dq_rs;
  int32_t B, H, Nq, Nk, hd; float scale;
  int32_t impl;
} vt_xattn_bwd_params;
int vt_xattn_bwd(const vt_xattn_bwd_params* p, void* stream);

/* Skip-path MaxPool3d on the fp32 token stream (pytorchvideo MultiScaleBlock.pool_skip: kernel s+1, stride s, padding
 * k//2 per axis; cls row copied).  x [B,1+T*H*W,D] -> y [B,1+To*Ho*Wo,D]; idx u8 same shape as y = winning tap
 * ((dt*kh+dh)*kw+dw, first maximum in scan order like torch).  Backward routes dy to the winners. */
typedef struct {
  const float* x; float* y; uint8_t* idx;
  int32_t B, D, T, H, W, kt, kh, kw, st, sh, sw, To, Ho, Wo;
} vt_maxpool_fwd_params;
int vt_maxpool_fwd(const vt_maxpool_fwd_params* p, void* stream);
typedef struct {
  const float* dy; const uint8_t* idx; float* dx;
  int32_t B, D, T, H, W, kt, kh, kw, st, sh, sw, To, Ho, Wo;
} vt_maxpool_bwd_params;
int vt_maxpool_bwd(const vt_maxpool_bwd_params* p, void* stream);

/* Overlapping Conv3d patch embedding operand (create_conv_patch_embed, video_transformer.py:585-618: kernel (3,7,7),
 * stride (2,4,4), padding (1,3,3)):  x fp32 [B,T,C,H,W] (the clip as the reference receives it, before its
 * transpose(1,2) at :912) -> cols bf16 [B*To*Ho*Wo, Kpad], column ((c*kt+dt)*kh+dh)*kw+dw, zero padded to Kpad. */
typedef struct {
  const float* x; void* cols;
  int32_t B, T, C, H, W, kt, kh, kw, st, sh, sw, pt, ph, pw, To, Ho, Wo, Kpad;
} vt_im2col3d_params;
int vt_im2col3d_bf16(const vt_im2col3d_params* p, void* stream);

/* Token preparation (MaskFeat.forward_features :915-919 + SpatioTemporalClsPositionalEncoding):
 *   x[b,0,:]   = cls_token + pos_cls
 *   x[b,1+l,:] = t[b,l,:]*(1-w[b,l]) + mask_token*w[b,l] + pos_s[l % HW,:] + pos_t[l / HW,:]      (w NULL => 0)
 * t fp32 [B*L, C] (conv output incl. bias), x fp32 [B,1+L,C], L = T*HW.
 * Backward: dt bf16 [B*L, C] = dx[b,1+l,:]*(1-w[b,l]) (parameter-table gradients are plain reductions of dx). */
typedef struct {
  const float* t; const float* wmask; const float* mask_token; const float* cls_token;
  const float* pos_s; const float* pos_t; const float* pos_cls; float* x;
  int32_t B, T, HW, C;
} vt_mvit_tokens_fwd_params;
int vt_mvit_tokens_fwd(const vt_mvit_tokens_fwd_params* p, void* stream);
typedef struct { const float* dx; const float* wmask; void* dt; int32_t B, T, HW, C; } vt_mvit_tokens_bwd_params;
int vt_mvit_tokens_bwd(const vt_mvit_tokens_bwd_params* p, void* stream);

/* Masked MSE of MaskFeat.forward (video_transformer.py:882-901):
 *   pred fp32 [B, 1+t*h*w, dt*dc] (decoder output incl. the cls row), target fp32 [B, t*dt, h, w, dc],
 *   mask fp32 [B, t*dt, h, w] (already restricted to the cube centre frames, :889-896)
 *   num[0] = sum_{cells} mask * mean_dc (pred - target)^2        (the caller divides by mask.sum() + 1e-5)
 * Backward: dpred bf16 [B*(1+t*h*w), dt*dc] = coef[0] * mask * (pred - target), cls rows zero; coef is a device
 * scalar (2 * dloss / (dc * (mask.sum() + 1e-5))).  partials: fp32 scratch [vt_mse_blocks(cells) * 4]. */
typedef struct {
  const float* pred; const float* target; const float* mask; float* num; float* partials;
  int32_t B, t, dt, h, w, dc;
  /* fp64 variant (the reference's targets are fp64 numpy arrays, dataset.py:190, which makes its loss fp64,
   * video_transformer.py:899-901): target64 != NULL replaces `target`; differences, squares and all sums are then taken in
   * fp64 and the sum goes to num64[0]; `partials` must hold vt_mse_blocks(cells) * 4 doubles. */
  const double* target64; double* num64;
} vt_mse_fwd_params;
int vt_mse_blocks(int32_t cells);
int vt_mse_fwd(const vt_mse_fwd_params* p, void* stream);
typedef struct {
  const float* pred; const float* target; const float* mask; const float* coef; void* dpred;
  int32_t B, t, dt, h, w, dc;
  const double* target64;   /* fp64 targets (replaces `target`) or NULL */
} vt_mse_bwd_params;
int vt_mse_bwd(const vt_mse_bwd_params* p, void* stream);

/* =============================================================================================
 * Fused per-parameter gradient clipping + optimizer step (SURVEY §8f rank 1; reference model_trainer.py:155-170
 * clip_gradients + optimizer.py:33-38 SGD(momentum 0.9, nesterov) / AdamW(0.9, 0.999)).
 * Multi-tensor form: tensor i has parameter pptr[i], gradient gptr[i], state s1ptr[i] (momentum buffer / exp_avg) and
 * s2ptr[i] (exp_avg_sq), all fp32 device addresses stored as int64 in device arrays; `chunks` is a device table of
 * {int32 tensor, int32 len, int64 offset} (16 bytes each) covering every tensor; lr / wd are per-tensor fp32 arrays.
 *   vt_opt_norm2 : norm2[i] = sum(grad_i^2)                          (the trainer's total norm = sqrt(sum_i norm2[i]))
 *   vt_opt_sgd   : g = grad * min(1, clip / (sqrt(norm2) + 1e-6)) [clip > 0];  d = g + wd*p;  buf = first ? d : mom*buf + d;
 *                  p -= lr * (nesterov ? d + mom*buf : buf)           (torch.optim.SGD, dampening 0)
 *   vt_opt_adamw : p *= 1 - lr*wd;  m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;
 *                  p -= lr/bc1 * m / (sqrt(v)/sqrt(bc2) + eps)         (torch.optim.AdamW; bc_k = 1 - beta_k^step)
 * Gradients are read, never written back (the reference scales p.grad in place; nothing reads it afterwards).
 * ============================================================================================= */
typedef struct {
  const void* chunks; int32_t n_chunks; int32_t n_tensors;
  const int64_t* pptr; const int64_t* gptr; const int64_t* s1ptr; const int64_t* s2ptr;
  float* norm2; const float* lr; const float* wd;
  float clip, momentum, beta1, beta2, eps, bc1, bc2;
  int32_t nesterov, first_step;
} vt_opt_params;
int vt_opt_norm2(const vt_opt_params* p, void* stream);
int vt_opt_sgd(const vt_opt_params* p, void* stream);
int vt_opt_adamw(const vt_opt_params* p, void* stream);

/* =============================================================================================
 * Classification head + loss, long-sequence attention maps, Mixup/CutMix operand (SURVEY §8 a18, f2, f4).
 * ============================================================================================= */

/* Skinny fp32 linear layer  y[M,N] = x[M,K] W[N,K]^T + b  (ClassificationHead.forward, transformer.py:78-80: 8 x 768 -> 400)
 * and its adjoints  dW = dy^T x, db = colsum(dy), dx = dy W  (dw / dx may be NULL to skip).  Warp-per-output GEMV on
 * the fp32 parameters themselves (no bf16 shadow); M <= 4096, K % 4 == 0. */
typedef struct { const float* x; const float* w; const float* b; float* y; int32_t M, N, K; } vt_linear_small_params;
int vt_linear_small_fwd(const vt_linear_small_params* p, void* stream);
typedef struct { const float* dy; const float* x; const float* w; float* dw; float* db; float* dx; int32_t M, N, K; } vt_linear_small_bwd_params;
int vt_linear_small_bwd(const vt_linear_small_bwd_params* p, void* stream);

/* Softmax cross-entropy, mean over rows: nn.CrossEntropyLoss (model_trainer.py:91, :208) with int64 `labels`, or timm's
 * SoftTargetCrossEntropy (:89) with fp32 `soft_targets` [M,N] (exactly one of the two).  One launch writes loss[0],
 * optional per-row losses and dlogits = d loss / d logits. */
typedef struct {
  const float* logits; const int64_t* labels; const float* soft_targets;
  float* loss; float* row_loss; float* dlogits; int32_t M, N;
} vt_softmax_ce_params;
int vt_softmax_ce(const vt_softmax_ce_params* p, void* stream);
/* out[i] = in[i] * scalar[0] (device scalar: chain rule through the loss inside a captured graph) */
typedef struct { const float* in; const float* scalar; float* out; int64_t n; } vt_scale_params;
int vt_scale_by_scalar(const vt_scale_params* p, void* stream);

/* probs[bp,h,i,j] = softmax_j(q_i . k_j * scale) for any N that fits 8 rows of scores in shared memory (N <= ~6000),
 * q/k read in place from the packed projection bf16 [Bp, N, 3, H, 64].  Serves get_last_selfattention
 * (video_transformer.py:258-261, transformer.py:560-561) for the 1569-token joint space-time variants. */
typedef struct { const void* qkv; float* probs; int32_t Bp, N, H, hd; float scale; } vt_attn_probs_params;
int vt_attn_probs(const vt_attn_probs_params* p, void* stream);

/* vt_im2col_u8_bf16 with the batch-level Mixup / CutMix of mixup.py:102-114 folded in: sample b is blended with (mode 1,
 * lam*x + (1-lam)*x.flip(0)) or patched from (mode 2, box rows [yl,yh) x cols [xl,xh)) sample B-1-b after normalisation.
 * plan = device float[6] {mode, lam, yl, yh, xl, xh}. */
typedef struct {
  const uint8_t* x; const float* scale; const float* shift; const float* plan; void* cols;
  int32_t B, T, C, H, W, tube, ph, pw;
} vt_im2col_u8_mix_params;
int vt_im2col_u8_mix_bf16(const vt_im2col_u8_mix_params* p, void* stream);

/* Bicubic resampling of the spatial position table for inputs of another size than img_size
 * (TimeSformer.interpolate_pos_encoding, video_transformer.py:171-191: F.interpolate(mode='bicubic', align_corners=False)
 * with a scale factor).  Row 0 (cls) is copied; patch row 1 + i*src_side + j of the table is grid cell (i, j).
 *   vt_pos_interp_fwd: in fp32 [1 + src_side^2, D] -> out fp32 [1 + out_rows*out_cols, D], output cell (i, j) at row
 *                      1 + i*out_cols + j samples source coordinate ((i + 0.5) * scale_r - 0.5, (j + 0.5) * scale_c - 0.5)
 *                      with the 4 x 4 cubic-convolution taps (A = -0.75) clamped to the grid.
 *   vt_pos_interp_bwd: its adjoint, in = d out [1 + out_rows*out_cols, D] -> out = d table [1 + src_side^2, D]; gather
 *                      form, deterministic.  (out_rows + out_cols) * src_side * 4 bytes must fit in 48 KB.
 * scale_r / scale_c = (float)(1.0 / scale_factor) as ATen computes them for fp32 input.  D % 4 == 0, 16-byte aligned. */
typedef struct {
  const float* in; float* out;
  int32_t D, src_side, out_rows, out_cols;
  float scale_r, scale_c;
} vt_pos_interp_params;
int vt_pos_interp_fwd(const vt_pos_interp_params* p, void* stream);
int vt_pos_interp_bwd(const vt_pos_interp_params* p, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VT_B200_H */
