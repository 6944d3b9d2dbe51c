// stft_kernels.cuh -- fused STFT / synchrosqueezed-STFT kernels (sm_100a).
//
// Replaces the three hot loops of ssq_stft.rs (A: frame FFTs :191-252,
// B: phase_stft :11-39, C: reassignment :276-301) and the frame loop of
// stft.rs:47-85 by ONE kernel: Sx, dSx and w never leave the SM.
//
// Common scheme (generic kernel here, n_fft=2^k fast kernels in stft_fast.cuh):
//   * a tile = F consecutive frames of one channel; persistent CTAs stride
//     over tiles; one warp owns one frame at a time;
//   * z[n] = x[n]*w[n] + i*x[n]*dw[n]*s   (two real FFTs packed in one complex
//     FFT; s is a host-chosen scale that keeps both parts the same magnitude);
//   * split  2*Sx[k] = Z[k]+conj(Z[N-k]),  2i*V[k] = Z[k]-conj(Z[N-k]);
//   * bin = | k - Im(V/Sx) * cphase |  in units of the ssq grid step, which is
//     ssq_stft.rs:32-33 divided by dw (the fs factors cancel), rounded to the
//     nearest grid point with ties to the LOWER index and clamped, exactly the
//     closed form of the reference's linear arg-min (:280-289);
//   * Tx column accumulated in shared memory, then written [n_freqs, n_frames]
//     row-major with >= 128 B contiguous per row.
#pragma once
#include "ssq_common.cuh"

struct StftParams {
  const float* x;       // [channels, x_stride]
  int64_t x_stride;
  int64_t n;            // samples per channel
  int channels;
  int n_fft, hop, n_freqs, log2n, is_pow2;
  int64_t n_frames;
  int left, padtype;
  const float* win;     // [n_fft]
  const float* dwin;    // [n_fft] diff window * s_scale (all zero in stft mode)
  const float2* wpair;  // [n_fft] (win, dwin) interleaved
  const float2* tw;     // [n_fft] exp(-2 pi i j / n_fft)
  float cphase;         // (n_freqs-1)/(pi*s_scale)
  float gate2;          // (2*gamma)^2 : compare with |2 Sx|^2
  float tx_scale;       // dw/2  -> Tx += (2 Sx) * tx_scale
  float leb_val;        // dw/n_freqs
  float dw_f;           // ssq grid step (Hz)
  float dsx_scale;      // fs/(2*s_scale): true dSx = (2V) * dsx_scale
  int mode;             // 0: ssq_stft (accumulate Tx), 1: stft (store Sx)
  int squeezing, modulated;
  float2* out;          // [channels, n_freqs, n_frames]
  float2* aux_Sx;       // optional, same shape
  float2* aux_dSx;      // optional
  float* aux_w;         // optional (Hz, +inf where gated)
  int* aux_kb;          // optional: destination bin of every (source bin, frame), -1 where gated
  int64_t frame0;       // global index of local frame 0 (streaming: the call computes frames
                        // [frame0, frame0 + n_frames) of a recording of n samples, see ssq_stream_*)
  int64_t x_origin;     // global sample index of x[.][0] (0 unless streaming)
  int F;                // frames per tile
  int acc_stride;       // odd >= n_freqs
  int64_t tiles_per_channel, total_tiles;
  // rows mode of the generic kernel (stft_rows.inl): the frame spectra were computed by the batched row passes;
  // Z of local frame f of channel ch is zrows[(ch * n_frames + f) * zld + k] (times zmul[k] when given: Bluestein)
  const float2* zrows;
  const float2* zmul;
  int64_t zld;
  int64_t out_ld;       // row stride of `out` / aux (0: n_frames)
  int64_t fbase;        // istft rows mode: global index of local frame 0 (rows are indexed (ch * n_use + f))
};

// Bin index of the reference's arg-min (ssq_stft.rs:280-289) from the bin-unit
// phase transform value: nearest grid point, ties -> lower, clamp, NaN -> 0.
__device__ __forceinline__ int ssq_bin_from(float binf, int n_freqs) {
  float r = ceilf(binf - 0.5f);
  int k = (r != r) ? 0 : (int)fminf(fmaxf(r, 0.f), (float)(n_freqs - 1));
  return k;
}


// Diagnostic outputs of the ssq kernels (parity tests: a compile-time flag of the register kernels, never
// on the timed path): per (source bin k, frame) Sx, dSx, w (Hz, +inf where gated) and the destination bin.
// (c, d) = 2 Sx, (a, b) = 2 V as the kernel used them; base = (ch * n_freqs) * n_frames + local frame.
__device__ __forceinline__ void ssq_dbg_emit(const StftParams& P, size_t base, int k, float c, float d, float a,
                                             float b, float binf, bool gated, int kb) {
  const size_t o = base + (size_t)k * (P.out_ld ? P.out_ld : P.n_frames);
  if (P.aux_Sx) P.aux_Sx[o] = make_float2(0.5f * c, 0.5f * d);
  if (P.aux_dSx) P.aux_dSx[o] = make_float2(a * P.dsx_scale, b * P.dsx_scale);
  if (P.aux_w) P.aux_w[o] = gated ? __int_as_float(0x7f800000) : binf * P.dw_f;
  if (P.aux_kb) P.aux_kb[o] = gated ? -1 : kb;
}

// Forward DFT of one frame held in shared memory by ONE warp.  A: input
// (destroyed), B: scratch; returns the buffer holding the natural-order result.
// Powers of two: radix-4 (+ one radix-2) Stockham autosort; otherwise a direct
// O(N^2) DFT (correctness path for arbitrary n_fft, as rustfft accepts any).
__device__ __forceinline__ float2* warp_fft_generic(float2* A, float2* B, const float2* twid, int N,
                                                    int log2n, int is_pow2, int lane) {
  if (is_pow2) {
    int s = 0;
    float2* in = A;
    float2* outb = B;
    for (; s + 2 <= log2n; s += 2) {
      const int Ns = 1 << s;
      const int q = N >> 2;
      const int tws = N / (4 * Ns);  // W_{4Ns}^{k t} = tw[k*t*tws]
      for (int j = lane; j < q; j += 32) {
        const int k = j & (Ns - 1);
        float2 a = in[j];
        float2 b = cmulf(in[j + q], twid[k * tws]);
        float2 c = cmulf(in[j + 2 * q], twid[2 * k * tws]);
        float2 d = cmulf(in[j + 3 * q], twid[3 * k * tws]);
        float2 apc = caddf(a, c), amc = csubf(a, c), bpd = caddf(b, d), bmd = csubf(b, d);
        const int o = ((j - k) << 2) + k;
        outb[o] = caddf(apc, bpd);
        outb[o + Ns] = make_float2(amc.x + bmd.y, amc.y - bmd.x);      // a - i b - c + i d
        outb[o + 2 * Ns] = csubf(apc, bpd);
        outb[o + 3 * Ns] = make_float2(amc.x - bmd.y, amc.y + bmd.x);  // a + i b - c - i d
      }
      __syncwarp();
      float2* t = in; in = outb; outb = t;
    }
    if (s < log2n) {
      const int Ns = 1 << s;
      const int h = N >> 1;
      const int tws = N / (2 * Ns);
      for (int j = lane; j < h; j += 32) {
        const int k = j & (Ns - 1);
        float2 a = in[j];
        float2 b = cmulf(in[j + h], twid[k * tws]);
        const int o = ((j - k) << 1) + k;
        outb[o] = caddf(a, b);
        outb[o + Ns] = csubf(a, b);
      }
      __syncwarp();
      float2* t = in; in = outb; outb = t;
    }
    return in;
  }
  for (int k = lane; k < N; k += 32) {
    float sr = 0.f, si = 0.f;
    int idx = 0;
    for (int n = 0; n < N; ++n) {
      float2 t = twid[idx];
      float2 z = A[n];
      sr += z.x * t.x - z.y * t.y;
      si += z.x * t.y + z.y * t.x;
      idx += k;
      if (idx >= N) idx -= N;
    }
    B[k] = make_float2(sr, si);
  }
  __syncwarp();
  return B;
}

// ------------------------------------------------------------------------
// Generic kernel: any n_fft >= 2 (radix-4/2 Stockham for powers of two, direct
// DFT otherwise), warp per frame, everything staged in shared memory.
// Dynamic smem: acc[F*acc_stride] | per-warp work[2*n_fft] | tw[n_fft] | per-warp tags[n_freqs].
// ------------------------------------------------------------------------
__global__ void __launch_bounds__(256) stft_generic_kernel(const StftParams P) {
  extern __shared__ float2 smem[];
  const int N = P.n_fft;
  const int nw = blockDim.x >> 5;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float2* acc = smem;
  float2* work = acc + (size_t)P.F * P.acc_stride + (size_t)warp * 2 * N;
  float2* twid = acc + (size_t)P.F * P.acc_stride + (size_t)nw * 2 * N;
  // per-warp destination-bin tags (n_freqs bytes, rounded up to 8) behind the twiddles
  unsigned char* tag = reinterpret_cast<unsigned char*>(twid + N) + (size_t)warp * ((P.n_freqs + 7) & ~7);
  const bool rows = P.zrows != nullptr;  // spectra come from the row passes: no per-warp work buffers, no twiddles
  if (rows) {
    twid = nullptr;
    tag = reinterpret_cast<unsigned char*>(acc + (size_t)P.F * P.acc_stride) + (size_t)warp * ((P.n_freqs + 7) & ~7);
  } else {
    for (int i = threadIdx.x; i < N; i += blockDim.x) twid[i] = P.tw[i];
  }
  const int64_t old = P.out_ld ? P.out_ld : P.n_frames;

  for (int64_t tile = blockIdx.x; tile < P.total_tiles; tile += gridDim.x) {
    const int ch = (int)(tile / P.tiles_per_channel);
    const int64_t f0 = (tile % P.tiles_per_channel) * P.F;
    const int nf = (int)min((int64_t)P.F, P.n_frames - f0);
    const float* xc = P.x + (size_t)ch * P.x_stride;
    for (int i = threadIdx.x; i < P.F * P.acc_stride; i += blockDim.x) acc[i] = make_float2(0.f, 0.f);
    __syncthreads();

    for (int fl = warp; fl < nf; fl += nw) {
      const int64_t frame = f0 + fl;
      const int64_t start = (P.frame0 + frame) * P.hop;
      const float2* Z;
      if (rows) {
        Z = P.zrows + ((size_t)ch * P.n_frames + frame) * P.zld;
      } else {
        float2* A = work;
        float2* B = work + N;
        for (int n = lane; n < N; n += 32) {
          float xv = stft_sample(xc, P.n, start + n, P.left, P.padtype, P.x_origin);
          A[n] = make_float2(xv * P.win[n], xv * P.dwin[n]);
        }
        __syncwarp();
        Z = warp_fft_generic(A, B, twid, N, P.log2n, P.is_pow2, lane);
      }

      // split + phase transform + reassignment.  Lane owns the S consecutive bins lane*S .. lane*S+S-1
      // (S odd: conflict-free strided reads of Z), so the 32 sources of a step are S bins apart and
      // rarely share a destination; a byte tag per destination bin detects the cases that do (fp32
      // shared atomics are CAS loops on sm_100a), which are then serialised in ascending source order.
      float2* col = acc + (size_t)fl * P.acc_stride;
      const int S = ((P.n_freqs + 31) >> 5) | 1;
      for (int i = 0; i < S; ++i) {
        const int k = lane * S + i;
        const bool valid = k < P.n_freqs;
        int kb = -1;
        float vre = 0.f, vim = 0.f;
        if (valid) {
          float2 zk = Z[k];
          float2 zn = Z[k == 0 ? 0 : N - k];
          if (rows && P.zmul) {
            zk = cmulf(zk, __ldg(P.zmul + k));
            zn = cmulf(zn, __ldg(P.zmul + (k == 0 ? 0 : N - k)));
          }
          float c = zk.x + zn.x, d = zk.y - zn.y;  // 2*Sx
          float a = zk.y + zn.y, b = zn.x - zk.x;  // 2*V
          if (P.modulated) {
            // multiply by exp(+2 pi i k (N/2)/N) = conj(tw[(k*(N/2)) mod N])
            const int m = (int)(((int64_t)k * (N / 2)) % N);
            const float2 t = rows ? __ldg(P.tw + m) : twid[m];
            float2 s2 = make_float2(c * t.x + d * t.y, d * t.x - c * t.y);
            float2 v2 = make_float2(a * t.x + b * t.y, b * t.x - a * t.y);
            c = s2.x; d = s2.y; a = v2.x; b = v2.y;
          }
          const float den = c * c + d * d;
          const bool gated = den < P.gate2;  // |Sx| < gamma (ssq_stft.rs:23)
          const float binf = fabsf((float)k - (b * c - a * d) / den * P.cphase);
          if (P.mode == 0 && (P.aux_Sx || P.aux_dSx || P.aux_w || P.aux_kb))
            ssq_dbg_emit(P, (size_t)ch * P.n_freqs * old + frame, k, c, d, a, b, binf, gated,
                         ssq_bin_from(binf, P.n_freqs));
          if (P.mode == 1) {
            col[k] = make_float2(0.5f * c, 0.5f * d);
          } else if (!gated) {
            kb = ssq_bin_from(binf, P.n_freqs);
            if (P.squeezing == SSQ_SQUEEZE_LEBESGUE) vre = P.leb_val;
            else { vre = c * P.tx_scale; vim = d * P.tx_scale; }
          }
        }
        if (P.mode == 0) {
          const bool on = kb >= 0;
          if (on) tag[kb] = (unsigned char)lane;
          __syncwarp();
          const bool mine = !on || tag[kb] == (unsigned char)lane;
          if (__all_sync(0xffffffffu, mine)) {
            if (on) { float2 t = col[kb]; t.x += vre; t.y += vim; col[kb] = t; }
          } else {
            for (int src = 0; src < 32; ++src) {  // rare: ascending lane = ascending source bin
              if (lane == src && on) { float2 t = col[kb]; t.x += vre; t.y += vim; col[kb] = t; }
              __syncwarp();
            }
          }
          __syncwarp();
        }
      }
      __syncwarp();
    }
    __syncthreads();
    // coalesced store: consecutive threads -> consecutive frames of one row
    float2* outc = P.out + (size_t)ch * P.n_freqs * old + f0;
    const int total = P.n_freqs * P.F;
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
      const int k = i / P.F, f = i - k * P.F;
      if (f < nf) outc[(size_t)k * old + f] = acc[(size_t)f * P.acc_stride + k];
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------
// issq_stft: y[c][j] = scale * sum_k Re Tx[c][k][j]   (coalesced along j)
// (old/ssqueezepy/_ssq_stft.py:190-197)
// ------------------------------------------------------------------------
__global__ void issq_stft_kernel(const float2* __restrict__ Tx, int64_t n_freqs, int64_t n_frames,
                                 float scale, float* __restrict__ y) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t c = blockIdx.y;
  if (j >= n_frames) return;
  const float2* t = Tx + (size_t)c * n_freqs * n_frames + j;
  float s0 = 0.f, s1 = 0.f;
  int64_t k = 0;
  for (; k + 1 < n_freqs; k += 2) {
    s0 += t[(size_t)k * n_frames].x;
    s1 += t[(size_t)(k + 1) * n_frames].x;
  }
  if (k < n_freqs) s0 += t[(size_t)k * n_frames].x;
  y[(size_t)c * n_frames + j] = (s0 + s1) * scale;
}

// ------------------------------------------------------------------------
// istft (old/ssqueezepy/_stft.py:184-256 in the Rust framing).
//   kernel 1: per tile of F frames: stage Sx[k][f0..f0+F) (coalesced rows) in
//     shared memory, one warp per frame does the Hermitian inverse DFT
//     (x = Re(DFT(conj Z))/N), multiplies by w^a and parks the N real samples in
//     the frame's own staging row; then every padded sample of the tile span
//     sums its <= ceil(N/hop) contributing frames (no shared atomics) and one
//     red.global.add per sample merges tile seams (two addends -> exact,
//     order-independent).
//   kernel 2: divide by the window norm sum_j w^(a+1)[p - j*hop] (evaluated
//     on the fly, old/.../stft_utils.py:186-191), unpad at (n_fft-1)/2.
// ------------------------------------------------------------------------
struct IstftParams {
  const float2* Sx;     // [channels, n_freqs, n_frames]
  int channels, n_fft, hop, n_freqs, log2n, is_pow2;
  int64_t n_frames;     // columns of Sx
  int64_t n_use;        // frames that fit in the padded length
  int64_t L;            // padded length n_out + n_fft - 1
  const float* wa;      // [n_fft] window^win_exp / n_fft   (1/n_fft when win_exp == 0)
  const float2* tw;     // [n_fft]
  float* xacc;          // [channels, L], zero-initialised
  int F, acc_stride;
  int64_t tiles_per_channel, total_tiles;
  // rows mode of the generic kernel (stft_rows.inl): the frame spectra were computed by the batched row passes;
  // Z of local frame f of channel ch is zrows[(ch * n_frames + f) * zld + k] (times zmul[k] when given: Bluestein)
  const float2* zrows;
  const float2* zmul;
  int64_t zld;
  int64_t out_ld;       // row stride of `out` / aux (0: n_frames)
  int64_t fbase;        // istft rows mode: global index of local frame 0 (rows are indexed (ch * n_use + f))
};

__global__ void __launch_bounds__(256) istft_ola_kernel(const IstftParams P) {
  extern __shared__ float2 smem[];
  const int N = P.n_fft;
  const int nw = blockDim.x >> 5;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float2* S = smem;  // [F][acc_stride]
  float2* work = S + (size_t)P.F * P.acc_stride + (size_t)warp * 2 * N;
  float2* twid = S + (size_t)P.F * P.acc_stride + (size_t)nw * 2 * N;
  const bool rows = P.zrows != nullptr;
  if (!rows)
    for (int i = threadIdx.x; i < N; i += blockDim.x) twid[i] = P.tw[i];

  for (int64_t tile = blockIdx.x; tile < P.total_tiles; tile += gridDim.x) {
    const int ch = (int)(tile / P.tiles_per_channel);
    const int64_t f0 = (tile % P.tiles_per_channel) * P.F;
    const int nf = (int)min((int64_t)P.F, P.n_use - f0);
    if (rows) {
      for (int fl = warp; fl < nf; fl += nw) {
        const float2* Z = P.zrows + ((size_t)ch * P.n_use + f0 + fl) * P.zld;
        float* rr = reinterpret_cast<float*>(S + (size_t)fl * P.acc_stride);
        for (int n = lane; n < N; n += 32) {
          float2 z = Z[n];
          if (P.zmul) z = cmulf(z, __ldg(P.zmul + n));
          rr[n] = z.x * P.wa[n];
        }
      }
    } else {
    const float2* in = P.Sx + (size_t)ch * P.n_freqs * P.n_frames + f0;
    const int total = P.n_freqs * P.F;
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
      const int k = i / P.F, f = i - k * P.F;
      if (f < nf) S[(size_t)f * P.acc_stride + k] = in[(size_t)k * P.n_frames + f];
    }
    __syncthreads();
    for (int fl = warp; fl < nf; fl += nw) {
      float2* row = S + (size_t)fl * P.acc_stride;
      float2* A = work;
      float2* B = work + N;
      for (int n = lane; n < N; n += 32) {
        float2 v = (n < P.n_freqs) ? row[n] : row[N - n];
        // conj(Zfull[n]): Zfull[n] = Sx[n] (n <= N/2), conj(Sx[N-n]) above
        A[n] = (n < P.n_freqs) ? make_float2(v.x, -v.y) : v;
      }
      __syncwarp();
      float2* Z = warp_fft_generic(A, B, twid, N, P.log2n, P.is_pow2, lane);
      float* rr = reinterpret_cast<float*>(row);
      for (int n = lane; n < N; n += 32) rr[n] = Z[n].x * P.wa[n];
      __syncwarp();
    }
    }
    __syncthreads();
    const int span = (nf - 1) * P.hop + N;
    float* xo = P.xacc + (size_t)ch * P.L + (P.fbase + f0) * P.hop;
    for (int p = threadIdx.x; p < span; p += blockDim.x) {
      int fhi = min(nf - 1, p / P.hop);
      int flo = (p - N + P.hop) / P.hop;  // ceil((p-N+1)/hop) for p-N+1 > 0
      if (p - N + 1 <= 0) flo = 0;
      float s = 0.f;
      for (int f = flo; f <= fhi; ++f)
        s += reinterpret_cast<const float*>(S + (size_t)f * P.acc_stride)[p - f * P.hop];
      atomicAdd(xo + p, s);
    }
    __syncthreads();
  }
}

#define ISTFT_FIN_PER_BLOCK 4096
#define ISTFT_FIN_MAX_HOP 1024
// The window norm wn(p) = sum_j w^(a+1)[p - j hop] only depends on p mod hop once every frame
// that covers p exists (p >= n_fft-1 and p/hop < max_hops): one table of `hop` sums per block
// serves those samples, the two ends of the signal take the explicit loop.  The batch finalize and
// the streaming one (istream_kernels.cuh) both go through these two functions, so that they divide
// every sample by the same float.
// (callers build the table only when hop <= ISTFT_FIN_MAX_HOP, then synchronise)
__device__ __forceinline__ void istft_wn_table(float* tab, int n_fft, int hop, const float* __restrict__ wpow, int tid,
                                               int nthreads) {
  for (int r = tid; r < hop; r += nthreads) {
    float s = 0.f;
    for (int m = r; m < n_fft; m += hop) s += wpow[m];
    tab[r] = s;
  }
}

__device__ __forceinline__ float istft_window_norm(int64_t p, int n_fft, int hop, int64_t max_hops, const float* tab,
                                                   const float* __restrict__ wpow) {
  int64_t jhi = p / hop;
  if (hop <= ISTFT_FIN_MAX_HOP && p >= n_fft - 1 && jhi <= max_hops - 1) return tab[(int)(p - jhi * hop)];
  if (jhi > max_hops - 1) jhi = max_hops - 1;
  const int64_t jlo = (p - n_fft + 1 <= 0) ? 0 : (p - n_fft + hop) / hop;
  float wn = 0.f;
  for (int64_t j = jlo; j <= jhi; ++j) wn += wpow[p - j * hop];
  return wn;
}

#define ISTFT_WN_TINY 1.17549435e-38f  // np.finfo(float32).tiny guard (_stft.py:246-251)

__global__ void __launch_bounds__(256) istft_finalize_kernel(const float* __restrict__ xacc, int64_t L, int64_t n_out,
                                                             int n_fft, int hop, int left, int64_t max_hops,
                                                             const float* __restrict__ wpow, float* __restrict__ out) {
  __shared__ float tab[ISTFT_FIN_MAX_HOP];
  if (hop <= ISTFT_FIN_MAX_HOP) {
    istft_wn_table(tab, n_fft, hop, wpow, threadIdx.x, blockDim.x);
    __syncthreads();
  }
  const int64_t c = blockIdx.y;
  const int64_t n0 = (int64_t)blockIdx.x * ISTFT_FIN_PER_BLOCK;
  for (int i = threadIdx.x; i < ISTFT_FIN_PER_BLOCK; i += blockDim.x) {
    const int64_t n = n0 + i;
    if (n >= n_out) break;
    const int64_t p = n + left;
    const float wn = istft_window_norm(p, n_fft, hop, max_hops, tab, wpow);
    float v = xacc[(size_t)c * L + p];
    if (wn > ISTFT_WN_TINY) v /= wn;
    out[(size_t)c * n_out + n] = v;
  }
}
