// components_kernels.cuh -- curve-band (component) inversion of a synchrosqueezed map, shared by issq_cwt and
// issq_stft (old/ssqueezepy/_ssq_cwt.py:380-402, the `_invert_components` both upstream inverses call).
#pragma once
#include "ssq_common.cuh"

#define SSQ_MAX_COMPONENTS 16

// Component c of column j sums Re Tx[k][j] over the rows lower <= k <= upper, with
//   upper = clip(cc + cw, 0, n_rows), lower = clip(cc - cw, 0, n_rows)   (64-bit: INT32_MAX and negative widths
//   cannot overflow), and an empty band where cc == -1 -- upstream's rule (:388-394).  Row n_rows does not exist, so
// an upper limit of n_rows is the last row.  Every component is summed from the original Tx, so bands may overlap;
// the residual (output row K) sums the rows no band covers.
// Tx: complex64 [channels, n_rows, n]; cc, cw: int32 [channels, n, K]; x: fp32 [channels, K + 1, n].
// One thread per column, rows ascending, one fp32 accumulator per component and one for the residual: the additions
// happen in the same order whatever KB is, so the bits depend on neither the bucket nor the batch.  KB (>= K) sizes
// the register arrays and the unrolled band test; slots K .. KB-1 hold empty bands.  Tx is read once, U rows per
// thread in flight.
template <int KB>
__global__ void __launch_bounds__(128) issq_components_kernel(const float2* __restrict__ Tx, int n_rows, int64_t n,
                                                              int K, const int* __restrict__ cc,
                                                              const int* __restrict__ cw, float scale,
                                                              float* __restrict__ x) {
  constexpr int U = 8;
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t ch = blockIdx.y;
  if (j >= n) return;
  int lo[KB], len[KB];  // band c is the rows lo[c] .. lo[c] + len[c] - 1
  float acc[KB];
#pragma unroll
  for (int c = 0; c < KB; ++c) {
    lo[c] = 0;
    len[c] = 0;
    acc[c] = 0.f;
    if (c < K) {
      const size_t b = ((size_t)ch * n + j) * K + c;
      const int64_t ce = __ldg(cc + b), wi = __ldg(cw + b);
      const int64_t u = min(max(ce + wi, (int64_t)0), (int64_t)n_rows);
      const int64_t l = min(max(ce - wi, (int64_t)0), (int64_t)n_rows);
      if (ce != -1 && u >= l) {
        lo[c] = (int)l;
        len[c] = (int)(u - l) + 1;
      }
    }
  }
  float rest = 0.f;
  const float2* t = Tx + (size_t)ch * n_rows * n + j;
  auto add = [&](int k, float v) {
    bool covered = false;
#pragma unroll
    for (int c = 0; c < KB; ++c) {
      if ((unsigned)(k - lo[c]) < (unsigned)len[c]) {
        acc[c] += v;
        covered = true;
      }
    }
    if (!covered) rest += v;
  };
  int k = 0;
  for (; k + U <= n_rows; k += U) {
    float v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) v[u] = __ldcs(t + (size_t)(k + u) * n).x;
    // most groups of U rows meet no band (a ridge band is a few rows of hundreds): one test per band and group, then
    // the rows go to the residual in the same order as add() would send them
    bool hit = false;
#pragma unroll
    for (int c = 0; c < KB; ++c) hit |= (unsigned)(k + U - 1 - lo[c]) < (unsigned)(len[c] + U - 1);
    if (hit) {
#pragma unroll
      for (int u = 0; u < U; ++u) add(k + u, v[u]);
    } else {
#pragma unroll
      for (int u = 0; u < U; ++u) rest += v[u];
    }
  }
  for (; k < n_rows; ++k) add(k, __ldcs(t + (size_t)k * n).x);
  float* o = x + (size_t)ch * (K + 1) * n + j;
#pragma unroll
  for (int c = 0; c < KB; ++c)
    if (c < K) o[(size_t)c * n] = acc[c] * scale;
  o[(size_t)K * n] = rest * scale;
}

// Launches the kernel with the smallest bucket that holds K (1 <= K <= SSQ_MAX_COMPONENTS, checked by the callers).
static ssq_status issq_components_run(ssq_ctx* ctx, const float2* d_Tx, int64_t channels, int64_t n_rows, int64_t n,
                                      const int* d_cc, const int* d_cw, int K, float scale, float* d_x) {
  const dim3 g((unsigned)((n + 127) / 128), (unsigned)channels);
  if (K <= 2)
    issq_components_kernel<2><<<g, 128, 0, ctx->stream>>>(d_Tx, (int)n_rows, n, K, d_cc, d_cw, scale, d_x);
  else if (K <= 4)
    issq_components_kernel<4><<<g, 128, 0, ctx->stream>>>(d_Tx, (int)n_rows, n, K, d_cc, d_cw, scale, d_x);
  else
    issq_components_kernel<16><<<g, 128, 0, ctx->stream>>>(d_Tx, (int)n_rows, n, K, d_cc, d_cw, scale, d_x);
  SSQ_TRY(ssq_check_launch(ctx, "issq_components_kernel"));
  ctx->last_kernel = "issq_components_kernel";
  return SSQ_OK;
}
