// ssq_common.cuh -- context object, error plumbing and small device helpers
// shared by every kernel file of libssqcuda (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <stdarg.h>
#include <string>
#include <vector>
#include <math.h>
#include "../../include/ssqcuda.h"

#define SSQ_PI 3.14159265358979323846

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
};

// One context = one device + one stream + grow-only workspaces + table cache.
struct ssq_ctx {
  int device = 0;
  int num_sms = 148;
  int max_smem_optin = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool ev_valid = false;
  const char* last_kernel = "";
  uint64_t launches = 0;
  std::string err;
  // workspaces
  DevBuf ws_in, ws_out, ws_aux0, ws_aux1, ws_aux2, ws_fft0, ws_fft1, ws_misc;
  DevBuf rows_tab;     // Bluestein chirp + filter spectrum of the rows path (stft_rows.inl), cached by n_fft
  int rows_n = -1;
  DevBuf ws_ridge[5];  // ridge extraction: energy, E, P, work indices, scale table
  // STFT table cache (window / diff-window / twiddles on device)
  DevBuf tab;
  std::vector<double> tab_window;  // fitted window the tables were built from
  int tab_nfft = -1;
  int tab_kind = -1;
  double tab_sscale = 1.0;
  // CWT twiddle cache
  DevBuf cwt_tw;
  int64_t cwt_tw_n = -1;
  DevBuf cwt_scales;
  std::vector<double> cwt_scales_host;  // content of cwt_scales (cache key)
  // pinned staging of the float64 entry points (two chunks: copy of chunk i+1 overlaps the conversion of chunk i)
  void* pin[2] = {nullptr, nullptr};
  cudaEvent_t pin_ev[2] = {nullptr, nullptr};
  // context options (DESIGN 6c), set only through ssq_ctx_set_option.  The first four select the reference paths
  // the tests check the fast kernels against: the generic shared-memory STFT kernels for n_fft 512 / 1024 / 256,
  // and the ordered, bit-deterministic ssq_cwt tail
  struct Options {
    int no_h32r = 0, no_r1024 = 0, no_r256 = 0, no_cwt_fused = 0;
    // STFT family framed as upstream ssqueezepy frames it (left pad n_fft / 2, the larger side for even n_fft:
    // old/ssqueezepy/utils/common.py:116-120) instead of the crate's (n_fft - 1) / 2 (stft_utils.rs:22); this one
    // does change results -- it is the switch of the upstream-compatible mode (ssqueeze_rs_b200/compat.py)
    int upstream_framing = 0;
  } opt;
};

static thread_local std::string g_tls_err;

static inline ssq_status ssq_fail(ssq_ctx* ctx, ssq_status st, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf; else g_tls_err = buf;
  return st;
}

#define SSQ_CUDA_TRY(ctx, expr)                                                      \
  do {                                                                               \
    cudaError_t _e = (expr);                                                         \
    if (_e != cudaSuccess)                                                           \
      return ssq_fail((ctx), _e == cudaErrorMemoryAllocation ? SSQ_ENOMEM : SSQ_ECUDA, \
                      "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

#define SSQ_TRY(expr)                      \
  do {                                     \
    ssq_status _s = (expr);                \
    if (_s != SSQ_OK) return _s;           \
  } while (0)

static inline ssq_status devbuf_reserve(ssq_ctx* ctx, DevBuf& b, size_t bytes) {
  if (bytes <= b.cap && b.p) return SSQ_OK;
  if (b.p) {
    // the old buffer may still be in use by work queued on the stream
    SSQ_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
  }
  size_t want = bytes < 256 ? 256 : bytes;
  cudaError_t e = cudaMalloc(&b.p, want);
  if (e != cudaSuccess) {
    b.p = nullptr;
    (void)cudaGetLastError();
    return ssq_fail(ctx, SSQ_ENOMEM, "cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
  }
  b.cap = want;
  return SSQ_OK;
}

static inline ssq_status ssq_check_launch(ssq_ctx* ctx, const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess)
    return ssq_fail(ctx, SSQ_ECUDA, "launch of %s failed: %s", what, cudaGetErrorString(e));
  ctx->launches++;
  return SSQ_OK;
}

// ---- device helpers -------------------------------------------------------
// Complex arithmetic on the packed fp32x2 instructions of sm_100 (FADD2 / FMUL2 / FFMA2): one
// instruction per complex add, two per complex multiply.  They occupy the fp32 pipe for two
// cycles, so the flop rate is that of the scalar forms (tools/ubench/fp2.cu: 64 complex adds per
// clock and SM either way) -- what halves is the number of ISSUE SLOTS, the resource these
// kernels run out of.  ptxas folds the operand swaps, sign patterns and scalar broadcasts written
// below into operand modifiers (.LO_HI, .NP, .F32): no MOV is emitted for them.
typedef unsigned long long ssq_u64;
__device__ __forceinline__ ssq_u64 pk2(float2 v) {
  ssq_u64 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(v.x), "f"(v.y));
  return r;
}
__device__ __forceinline__ float2 up2(ssq_u64 v) {
  float2 r;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v));
  return r;
}
// PK = false selects the scalar forms: the packed ones need aligned register pairs, and a kernel
// that already sits at its register cap can lose more to the spills than it gains (the stft mode
// of the n_fft = 512 kernel: 18.5 ms packed with 56 B of spills, 16.8 ms scalar on 384 channels).
template <bool PK = true>
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
  if constexpr (PK) {
    ssq_u64 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(pk2(a)), "l"(pk2(b)));
    return up2(r);
  } else {
    return make_float2(a.x + b.x, a.y + b.y);
  }
}
template <bool PK = true>
__device__ __forceinline__ float2 sub2(float2 a, float2 b) {
  if constexpr (PK) {
    ssq_u64 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(pk2(a)), "l"(pk2(b)));
    return up2(r);
  } else {
    return make_float2(a.x - b.x, a.y - b.y);
  }
}
template <bool PK = true>
__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
  if constexpr (PK) {
    ssq_u64 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(pk2(a)), "l"(pk2(b)));
    return up2(r);
  } else {
    return make_float2(a.x * b.x, a.y * b.y);
  }
}
template <bool PK = true>
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
  if constexpr (PK) {
    ssq_u64 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(pk2(a)), "l"(pk2(b)), "l"(pk2(c)));
    return up2(r);
  } else {
    return make_float2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y));
  }
}
__device__ __forceinline__ float2 bc2(float s) { return make_float2(s, s); }
template <bool PK = true>
__device__ __forceinline__ float2 cmulf(float2 a, float2 b) {  // (a.x b.x - a.y b.y, a.y b.x + a.x b.y)
  return fma2<PK>(make_float2(a.y, a.x), make_float2(-b.y, b.y), mul2<PK>(a, bc2(b.x)));
}
template <bool PK = true>
__device__ __forceinline__ float2 cmulcf(float2 a, float2 b) {  // a * conj(b)
  return fma2<PK>(make_float2(a.y, a.x), make_float2(b.y, -b.y), mul2<PK>(a, bc2(b.x)));
}
template <bool PK = true>
__device__ __forceinline__ float2 caddf(float2 a, float2 b) { return add2<PK>(a, b); }
template <bool PK = true>
__device__ __forceinline__ float2 csubf(float2 a, float2 b) { return sub2<PK>(a, b); }
__device__ __forceinline__ float2 cmi(float2 a) { return make_float2(a.y, -a.x); }  // a * (-i)
__device__ __forceinline__ float2 cpi(float2 a) { return make_float2(-a.y, a.x); }  // a * (+i)

// Internal pad code, never seen at the ABI: reflect padding as upstream ssqueezepy pads, np.pad(mode="reflect"),
// which reflects again and again where a pad is longer than the signal.  run_stft_family selects it for "reflect"
// under the upstream_framing option; the crate's own reflect (SSQ_PAD_REFLECT) leaves those samples at zero.  The two
// differ only for n <= left, where one reflection does not reach every padded sample.
constexpr int SSQ_PAD_REFLECT_UPSTREAM = 2;

// Padded-signal sample fetch in the reference's STFT framing
// (stft_utils.rs:19-65): padded index p, left = (n_fft-1)/2 (n_fft/2 in upstream framing).
// `origin`: global index of x[0] (streaming: x holds the samples [origin, ...) of a longer recording of
// n samples; every index that is read lies inside the carried-over buffer).
// FOLD = false drops the np.pad fold at compile time: the register kernels' edge-sample function keeps the code it
// had before the fold existed (run_stft_family does not send them signals of n <= left in upstream reflect).
template <bool FOLD = true>
__device__ __forceinline__ float stft_sample(const float* __restrict__ x, int64_t n, int64_t p,
                                             int left, int padtype, int64_t origin = 0) {
  int64_t o = p - left;
  if (o >= 0 && o < n) return __ldg(x + (o - origin));
  if (padtype == SSQ_PAD_ZERO) return 0.f;
  if (FOLD && padtype == SSQ_PAD_REFLECT_UPSTREAM && (o < 1 - n || o > 2 * n - 2)) {
    // beyond one reflection (n <= left): np.pad folds the index with period 2 (n - 1), and a 1-sample signal is a
    // constant.  Then n <= n_fft / 2, so o and n fit in 32 bits, and a stream holds the whole recording (origin 0).
    const int period = 2 * ((int)n - 1);
    if (period == 0) return __ldg(x - origin);
    int r = (int)o % period;
    if (r < 0) r += period;
    if (r >= (int)n) r = period - r;
    return __ldg(x + (r - origin));
  }
  if (o < 0) {
    int64_t m = -o;  // stft_utils.rs:34-36
    return m < n ? __ldg(x + (m - origin)) : 0.f;
  }
  int64_t m = 2 * n - 2 - o;  // stft_utils.rs:42-44
  return (m >= 0 && m < n) ? __ldg(x + (m - origin)) : 0.f;
}

// Non-atomic-free float2 accumulate in shared memory: fp32 shared atomics are
// CAS loops on sm_100a (ATOMS.CAST.SPIN), so do one 64-bit CAS for the pair.
__device__ __forceinline__ void smem_add_f2(float2* addr, float re, float im) {
  unsigned long long* p = reinterpret_cast<unsigned long long*>(addr);
  unsigned long long old = *p, assumed;
  do {
    assumed = old;
    float2 v;
    v.x = __uint_as_float((unsigned)(assumed & 0xffffffffull)) + re;
    v.y = __uint_as_float((unsigned)(assumed >> 32)) + im;
    unsigned long long nv = ((unsigned long long)__float_as_uint(v.y) << 32) | __float_as_uint(v.x);
    old = atomicCAS(p, assumed, nv);
  } while (old != assumed);
}
