// Bicubic resampling of the learned spatial position table (TimeSformer.interpolate_pos_encoding, reference
// video_transformer.py:171-191) and its adjoint.  The patch rows of pos_embed [1+S*S, D] are a S x S grid of D-vectors;
// the output grid is out_rows x out_cols, computed exactly like F.interpolate(mode='bicubic', align_corners=False) with a
// given scale factor: src = (dst + 0.5) * scale - 0.5 (scale = 1 / scale_factor, no clamp for cubic), taps floor(src) - 1
// .. + 2 clamped to [0, S-1], cubic convolution weights with A = -0.75.  Row 0 (the cls position) is copied.
// Both kernels derive every weight from the scalar parameters (no host table), so they are legal inside a captured graph.
#include "vt_common.cuh"

namespace vt {

// The four taps of output index `dst` along one axis: clamped source indices and cubic-convolution weights
// (ATen's get_cubic_upsample_coefficients; the order of operations matches upsample_bicubic2d).
__device__ __forceinline__ void pos_cubic_taps(int dst, float scale, int in_size, int idx[4], float w[4]) {
  const float src = scale * ((float)dst + 0.5f) - 0.5f;
  const float fl = floorf(src);
  const float t = src - fl;
  const int i0 = (int)fl;
  constexpr float A = -0.75f;
  const float x1 = t + 1.0f, x2 = 1.0f - t, x3 = x2 + 1.0f;
  w[0] = ((A * x1 - 5.0f * A) * x1 + 8.0f * A) * x1 - 4.0f * A;
  w[1] = ((A + 2.0f) * t - (A + 3.0f)) * t * t + 1.0f;
  w[2] = ((A + 2.0f) * x2 - (A + 3.0f)) * x2 * x2 + 1.0f;
  w[3] = ((A * x3 - 5.0f * A) * x3 + 8.0f * A) * x3 - 4.0f * A;
#pragma unroll
  for (int k = 0; k < 4; ++k) idx[k] = min(max(i0 - 1 + k, 0), in_size - 1);
}

__device__ __forceinline__ float4 f4_fma(float a, float4 x, float4 acc) {
  return make_float4(fmaf(a, x.x, acc.x), fmaf(a, x.y, acc.y), fmaf(a, x.z, acc.z), fmaf(a, x.w, acc.w));
}

// one thread per (output row of the table, 4 channels); row 0 = cls copy
__global__ void __launch_bounds__(256)
pos_interp_fwd_kernel(const float* __restrict__ in, float* __restrict__ out, int D4, int S, int R, int C, float scale_r,
                      float scale_c) {
  const int n = (1 + R * C) * D4;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
    const int row = e / D4, c4 = e - row * D4;
    const float4* src = reinterpret_cast<const float4*>(in);
    if (row == 0) {
      reinterpret_cast<float4*>(out)[c4] = src[c4];
      continue;
    }
    const int i = (row - 1) / C, j = (row - 1) - i * C;
    int ir[4], ic[4];
    float wr[4], wc[4];
    pos_cubic_taps(i, scale_r, S, ir, wr);
    pos_cubic_taps(j, scale_c, S, ic, wc);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int a = 0; a < 4; ++a) {          // along the columns first, then along the rows (upsample_bicubic2d's order)
      float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int b = 0; b < 4; ++b) r = f4_fma(wc[b], __ldg(src + (1 + ir[a] * S + ic[b]) * D4 + c4), r);
      acc = f4_fma(wr[a], r, acc);
    }
    reinterpret_cast<float4*>(out)[(long long)row * D4 + c4] = acc;
  }
}

// Adjoint, gather form (deterministic, no atomics).  Block (cell, channel chunk): cell 0 copies the cls gradient; cell
// 1 + a*S + b sums Wr[i, a] * Wc[j, b] * dout[1 + i*C + j] over the outputs that reach it.  Wr [R, S] / Wc [C, S] are
// the dense 1-D weight matrices (clamped border taps added into the same entry), built in shared memory.
__global__ void __launch_bounds__(128)
pos_interp_bwd_kernel(const float* __restrict__ dout, float* __restrict__ din, int D4, int S, int R, int C, float scale_r,
                      float scale_c) {
  extern __shared__ float sw[];
  float* Wr = sw;                 // [R][S]
  float* Wc = sw + R * S;         // [C][S]
  const int cell = blockIdx.x;
  const int c4 = blockIdx.y * blockDim.x + threadIdx.x;
  const float4* g = reinterpret_cast<const float4*>(dout);
  if (cell == 0) {
    if (c4 < D4) reinterpret_cast<float4*>(din)[c4] = g[c4];
    return;
  }
  for (int k = threadIdx.x; k < (R + C) * S; k += blockDim.x) sw[k] = 0.f;
  __syncthreads();
  for (int k = threadIdx.x; k < R + C; k += blockDim.x) {      // one thread per output row / column: no write races
    int idx[4];
    float w[4];
    const bool is_row = k < R;
    pos_cubic_taps(is_row ? k : k - R, is_row ? scale_r : scale_c, S, idx, w);
    float* dst = is_row ? Wr + k * S : Wc + (k - R) * S;
#pragma unroll
    for (int t = 0; t < 4; ++t) dst[idx[t]] += w[t];
  }
  __syncthreads();
  if (c4 >= D4) return;
  const int a = (cell - 1) / S, b = (cell - 1) - a * S;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int i = 0; i < R; ++i) {
    const float wr = Wr[i * S + a];
    if (wr == 0.f) continue;
    float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int j = 0; j < C; ++j) {
      const float wc = Wc[j * S + b];
      if (wc != 0.f) r = f4_fma(wc, __ldg(g + (long long)(1 + i * C + j) * D4 + c4), r);
    }
    acc = f4_fma(wr, r, acc);
  }
  reinterpret_cast<float4*>(din)[(long long)cell * D4 + c4] = acc;
}

static int pos_interp_check(const vt_pos_interp_params* p, const char* what) {
  VT_REQUIRE(p && p->in && p->out, "%s: null pointer", what);
  VT_REQUIRE(p->D > 0 && p->D % 4 == 0, "%s: D=%d must be a positive multiple of 4", what, p->D);
  VT_REQUIRE(p->src_side > 0 && p->out_rows > 0 && p->out_cols > 0, "%s: bad grid %d -> %d x %d", what, p->src_side,
             p->out_rows, p->out_cols);
  VT_REQUIRE(p->scale_r > 0.f && p->scale_c > 0.f, "%s: scales must be positive", what);
  VT_REQUIRE((long long)(1 + p->out_rows * (long long)p->out_cols) * p->D < (1ll << 31) &&
                 (long long)(1 + p->src_side * (long long)p->src_side) * p->D < (1ll << 31),
             "%s: table too large", what);
  VT_REQUIRE(((reinterpret_cast<uintptr_t>(p->in) | reinterpret_cast<uintptr_t>(p->out)) & 15) == 0,
             "%s: pointers must be 16-byte aligned", what);
  return 0;
}

}  // namespace vt

using namespace vt;

extern "C" int vt_pos_interp_fwd(const vt_pos_interp_params* p, void* stream) {
  if (int rc = pos_interp_check(p, "vt_pos_interp_fwd")) return rc;
  const int D4 = p->D / 4;
  const long long n = (1 + (long long)p->out_rows * p->out_cols) * D4;
  long long blocks = (n + 255) / 256;
  if (blocks > 4096) blocks = 4096;
  pos_interp_fwd_kernel<<<(int)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      p->in, p->out, D4, p->src_side, p->out_rows, p->out_cols, p->scale_r, p->scale_c);
  return check_launch("pos_interp_fwd_kernel");
}

extern "C" int vt_pos_interp_bwd(const vt_pos_interp_params* p, void* stream) {
  if (int rc = pos_interp_check(p, "vt_pos_interp_bwd")) return rc;
  const size_t smem = (size_t)(p->out_rows + p->out_cols) * p->src_side * sizeof(float);
  VT_REQUIRE(smem <= 48 * 1024, "vt_pos_interp_bwd: (%d + %d) x %d weight matrices exceed 48 KB of shared memory",
             p->out_rows, p->out_cols, p->src_side);
  const int D4 = p->D / 4;
  dim3 grid(1 + p->src_side * p->src_side, (D4 + 127) / 128);
  pos_interp_bwd_kernel<<<grid, 128, smem, static_cast<cudaStream_t>(stream)>>>(
      p->in, p->out, D4, p->src_side, p->out_rows, p->out_cols, p->scale_r, p->scale_c);
  return check_launch("pos_interp_bwd_kernel");
}
