// istream_kernels.cuh -- the device half of the streaming inverse (ssq_istream_*, DESIGN §3.4c).
//
// istft: every push overlap-adds its own frames into a zeroed buffer A with the batch call's kernels
// (istft_ola_run); istream_finalize_kernel then adds the carry C of undivided partial sums that earlier
// pushes left at the positions the new frames also cover (C + A, always in that order: deterministic),
// divides the samples that became final by the window norm (the batch rule, istft_window_norm), converts
// them to the output format and writes the partial sums of the positions the next frames still reach as
// the next push's carry.
// issq_stft: istream_issq_kernel sums Re Tx over frequency per frame as issq_stft_kernel does.
#pragma once
#include "stft_kernels.cuh"

#define ISTREAM_TILE 128  // output samples per block (x 32 channels); the window-norm table is built once per block

enum { ISTREAM_F32 = 0, ISTREAM_F32_INTERLEAVED = 1, ISTREAM_I16_INTERLEAVED = 2 };

struct IstreamFinParams {
  const float* A;     // [channels, La]: this push's overlap-add, A[q] at padded position base + q
  int64_t La;
  const float* Cin;   // [channels, cstride]: carry of earlier pushes, Cin[q] at base + q for q < clen_in
  float* Cout;        // [channels, cstride]: the next carry, Cout[j] = T(q_carry + j) for j < clen_out
  int64_t cstride, clen_in, clen_out, q_carry;
  int64_t channels;
  int64_t n_emit;     // final samples written by this push
  int64_t q0;         // q of the first of them
  int64_t base;       // padded position of q = 0
  int n_fft, hop;
  int64_t max_hops;
  const float* wpow;  // [n_fft] window^(win_exp + 1)
  float inv_scale;
  void* out;          // n_emit samples x channels in the layout of FMT
  int nb_out;         // blocks along x that write samples; those after them write the carry
};

// T(q): the undivided sum at padded position base + q over every frame pushed so far
__device__ __forceinline__ float istream_total(const IstreamFinParams& P, int64_t c, int64_t q) {
  float t = q < P.La ? P.A[(size_t)c * P.La + q] : 0.f;
  if (q < P.clen_in) t = P.Cin[(size_t)c * P.cstride + q] + t;
  return t;
}

// round to nearest even, saturate (np.clip(np.rint(v), -32768, 32767))
__device__ __forceinline__ int16_t istream_to_i16(float v) {
  return (int16_t)__float2int_rn(fminf(fmaxf(v, -32768.f), 32767.f));
}

// 32 channels x 32 samples per step: x -> sample, y -> channel rows; the interleaved formats transpose through
// `tile` so that their stores run along channels, as deinterleave_kernel does on the way in
template <int FMT>
__device__ __forceinline__ void istream_store(float (*tile)[33], float v, void* out, int64_t channels, int64_t i0,
                                              int64_t c0, int64_t n_emit, int r) {
  const int tx = threadIdx.x;
  if (FMT == ISTREAM_F32) {
    const int64_t c = c0 + r, i = i0 + tx;
    if (c < channels && i < n_emit) reinterpret_cast<float*>(out)[(size_t)c * n_emit + i] = v;
  } else {
    tile[r][tx] = v;
  }
}

template <int FMT>
__device__ __forceinline__ void istream_flush(float (*tile)[33], void* out, int64_t channels, int64_t i0, int64_t c0,
                                              int64_t n_emit) {
  if (FMT == ISTREAM_F32) return;
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int64_t i = i0 + r, c = c0 + threadIdx.x;
    if (i < n_emit && c < channels) {
      const float v = tile[threadIdx.x][r];
      if (FMT == ISTREAM_F32_INTERLEAVED) reinterpret_cast<float*>(out)[(size_t)i * channels + c] = v;
      else reinterpret_cast<int16_t*>(out)[(size_t)i * channels + c] = istream_to_i16(v);
    }
  }
  __syncthreads();
}

template <int FMT>
__global__ void __launch_bounds__(256) istream_finalize_kernel(const IstreamFinParams P) {
  __shared__ float tab[ISTFT_FIN_MAX_HOP];
  __shared__ float tile[32][33];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int64_t c0 = (int64_t)blockIdx.y * 32;
  if ((int)blockIdx.x >= P.nb_out) {  // the next carry: plain copy of T, no division
    const int64_t j0 = (int64_t)(blockIdx.x - P.nb_out) * ISTREAM_TILE;
    for (int r = ty; r < 32; r += blockDim.y) {
      const int64_t c = c0 + r;
      if (c >= P.channels) break;
      for (int i = tx; i < ISTREAM_TILE; i += 32) {
        const int64_t j = j0 + i;
        if (j >= P.clen_out) break;
        P.Cout[(size_t)c * P.cstride + j] = istream_total(P, c, P.q_carry + j);
      }
    }
    return;
  }
  if (P.hop <= ISTFT_FIN_MAX_HOP) {
    istft_wn_table(tab, P.n_fft, P.hop, P.wpow, ty * 32 + tx, 256);
    __syncthreads();
  }
  const int64_t b0 = (int64_t)blockIdx.x * ISTREAM_TILE;
  for (int s = 0; s < ISTREAM_TILE; s += 32) {
    const int64_t i0 = b0 + s, i = i0 + tx;
    if (i0 >= P.n_emit) break;
    const float wn = i < P.n_emit ? istft_window_norm(P.base + P.q0 + i, P.n_fft, P.hop, P.max_hops, tab, P.wpow) : 0.f;
    for (int r = ty; r < 32; r += blockDim.y) {
      const int64_t c = c0 + r;
      float v = 0.f;
      if (c < P.channels && i < P.n_emit) {
        v = istream_total(P, c, P.q0 + i);
        if (wn > ISTFT_WN_TINY) v /= wn;
        v *= P.inv_scale;
      }
      istream_store<FMT>(tile, v, P.out, P.channels, i0, c0, P.n_emit, r);
    }
    istream_flush<FMT>(tile, P.out, P.channels, i0, c0, P.n_emit);
  }
}

// issq_stft of one push: y[c][j] = scale * sum_k Re Tx[c][k][j] with issq_stft_kernel's order of additions
// (bit-equal to the batch call), times inv_scale, in the layout of FMT
template <int FMT>
__global__ void __launch_bounds__(256) istream_issq_kernel(const float2* __restrict__ Tx, int64_t channels,
                                                           int64_t n_freqs, int64_t n_frames, float scale,
                                                           float inv_scale, void* out) {
  __shared__ float tile[32][33];
  const int64_t i0 = (int64_t)blockIdx.x * 32, c0 = (int64_t)blockIdx.y * 32;
  const int64_t j = i0 + threadIdx.x;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int64_t c = c0 + r;
    float v = 0.f;
    if (c < channels && j < n_frames) {
      const float2* t = Tx + (size_t)c * n_freqs * n_frames + j;
      float s0 = 0.f, s1 = 0.f;
      int64_t k = 0;
      for (; k + 1 < n_freqs; k += 2) {
        s0 += t[(size_t)k * n_frames].x;
        s1 += t[(size_t)(k + 1) * n_frames].x;
      }
      if (k < n_freqs) s0 += t[(size_t)k * n_frames].x;
      v = (s0 + s1) * scale;
      v *= inv_scale;
    }
    istream_store<FMT>(tile, v, out, channels, i0, c0, n_frames, r);
  }
  istream_flush<FMT>(tile, out, channels, i0, c0, n_frames);
}
