// cwt_kernels.cuh -- CWT / ssq_cwt device code (sm_100a).
//
// Replaces cwt.rs:95-326 / ssq_cwt.rs:331-480: one forward FFT of the padded
// signal, per-scale multiply by psi-hat (and by i*xi/dt for the derivative),
// one inverse FFT per (scale, {W, dW}) row, unpad, phase transform and the
// column-local reassignment.
//
// FFT: power-of-two length L = 2^m rows, Stockham autosort in PASSES; a pass
// applies a radix R = 2^r (r <= 7) to T adjacent columns inside shared memory,
// so every global access of a pass is a run of T consecutive complex64
// (256 B for T = 32).  L <= 4096 is a single pass (R = L, T = 1).
// The first pass LOADS through a functor (real padded signal, or
// x-hat * psi-hat generated on the fly: the products never exist in HBM); the
// last pass STORES through a functor (1/L scale, sqrt(scale) for L2 norm,
// unpad, de-normalisation constant), so Wx is written exactly once.
#pragma once
#include "ssq_common.cuh"
#include "fft_regs.cuh"

// ------------------------------------------------------------------------------------
// ssq_cwt reassignment (ssq_cwt.rs:116-222 + phase_cwt :15-47).
// W, D: already scaled by 1/L, psi-hat peak-normalised: true Wx = W * K.
// ------------------------------------------------------------------------------------
struct SsqCwtParams {
  const float2* W;    // [ns, n] (stand-alone kernel only)
  const float2* D;
  float2* Tx;         // stand-alone: [ns, pitch] of one channel; fused: [channels, ns, pitch]; zero-initialised
  int ns;
  int64_t n;          // columns written per row (fused: per (channel, block) row; stand-alone: per thread sweep)
  int64_t pitch;      // row pitch of Tx (n for the batch call; the push's column count for a stream)
  float gate;         // gamma / K (in the units of the W handed to ssq_cwt_item): |W| < gate -> skipped
  float gate2f;       // max(gate^2, 1e-30), at most 3e38: below it (or above 1e30) the exact out-of-line path decides
  int is_log;
  float f0s, inv_step; // lin: w * inv_step - f0s ; log: log2 w * inv_step - f0s   (f0s = f0 * inv_step)
  int flipud, squeezing;
  float K, leb_val;
  int* aux_kb;        // optional diagnostics, same layout as Tx: destination row per (scale, column), -1 = nothing added
  float* aux_w;       // optional: w (Hz), +inf where gated
};

// Rare magnitudes (|W|^2 outside fp32's comfortable range): the scale-free ratio after an exact power-of-two
// rescale, and the gate on the true magnitude.  Out of line: the hot path below must stay short.
__device__ __noinline__ float ssq_cwt_w_slow(float2 Wv, float2 Dv, float gate) {
  const float mag = hypotf(Wv.x, Wv.y);
  if (mag < gate) return __int_as_float(0x7f800000);  // gated (ssq_cwt.rs:29-30)
  float c = Wv.x, d = Wv.y, a = Dv.x, bb = Dv.y;
  if (mag < 1e-15f) {
    const float up = 1.8446744e19f;  // 2^64
    c *= up; d *= up; a *= up; bb *= up;
  } else if (mag > 1e15f) {
    const float dn = 5.4210109e-20f;  // 2^-64
    c *= dn; d *= dn; a *= dn; bb *= dn;
  }
  return fabsf((bb * c - a * d) / ((c * c + d * d) * 6.283185307179586f));
}

// One (scale, column) item: returns the bin on the ssq grid BEFORE the flip, or -1 when nothing is added (gated, w
// not finite, bin outside the grid: ssq_cwt.rs:29-30, :167-169, :177-179).  w_out: the phase transform (+inf when
// gated).  Wv, Dv may carry any common positive factor (the ratio is scale-free); P.gate is expressed in their units.
// The fused last pass is bound by issue slots and this epilogue was half of its instructions (profiles/README.md):
// one range test pair (P.gate2f = max(gate^2, 1e-30) from the host), rcp.approx / lg2.approx (one MUFU each; the
// parity classification carries their error), the grid map as one FMA, round-half-away as a floor conversion.
__device__ __forceinline__ int ssq_cwt_bin(const SsqCwtParams& P, float2 Wv, float2 Dv, float& w_out) {
  const float c = Wv.x, d = Wv.y;
  const float m2 = fmaf(c, c, d * d);
  float w;
  if (m2 >= P.gate2f && m2 < 1e30f) {
    const float num = fmaf(Dv.y, c, -Dv.x * d);  // Im(dW conj W)
    w = fabsf(num) * rcp_approx(m2 * 6.283185307179586f);
  } else {
    w = ssq_cwt_w_slow(Wv, Dv, P.gate);
  }
  w_out = w;
  if (!(w <= 3.4028235e38f)) return -1;  // gated / inf / NaN skipped (:167-169)
  // v = (log2 w - f0) * inv_step  resp. (w - f0) * inv_step, as one FMA with f0s = f0 * inv_step
  float lw;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lw) : "f"(w));  // one MUFU (w is a frequency: never subnormal on the grid)
  const float v = fmaf(P.is_log ? lw : w, P.inv_step, -P.f0s);
  // f64::round, half away from zero (:176, :187): floor(v + 1/2) for v > -1/2 (values in (-1/2, 0) round to -0 ->
  // bin 0), anything at or below -1/2 is a negative bin: dropped; NaN fails the first test
  const int bin = __float2int_rd(v + 0.5f);
  if (!(v > -0.5f) || (unsigned)bin >= (unsigned)P.ns) return -1;  // out of range dropped (:177-179)
  return bin;
}
__device__ __forceinline__ int ssq_cwt_item(const SsqCwtParams& P, float2 Wv, float2 Dv, float& w_out) {
  const int bin = ssq_cwt_bin(P, Wv, Dv, w_out);
  return bin < 0 ? -1 : (P.flipud ? P.ns - 1 - bin : bin);
}

// Stand-alone reassignment (the path taken when the last FFT pass cannot carry the fused epilogue): one thread per
// time column; the thread is the only writer of its Tx column, so the accumulation runs in ascending scale order
// (the reference's order).
__global__ void ssq_cwt_reassign_kernel(const SsqCwtParams P) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= P.n) return;
  const float2* __restrict__ Wc = P.W + b;
  const float2* __restrict__ Dc = P.D + b;
  float2* Tc = P.Tx + b;
  // the W, D values of eight scales are in flight at once, and the thread adds to Tx with a reduction (no value
  // returned: nothing to wait for; same-thread reductions to one address stay in program order)
  constexpr int U = 8;
  for (int i0 = 0; i0 < P.ns; i0 += U) {
    float2 Wb[U], Db[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = min(i0 + u, P.ns - 1);
      Wb[u] = __ldcs(Wc + (size_t)i * P.n);
      Db[u] = __ldcs(Dc + (size_t)i * P.n);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (i0 + u >= P.ns) break;
      float w;
      const int k = ssq_cwt_item(P, Wb[u], Db[u], w);
      if (P.aux_kb) P.aux_kb[(size_t)(i0 + u) * P.n + b] = k;
      if (P.aux_w) P.aux_w[(size_t)(i0 + u) * P.n + b] = w;
      if (k < 0) continue;
      float2* t = Tc + (size_t)k * P.pitch;
      if (P.squeezing == SSQ_SQUEEZE_LEBESGUE) atomicAdd(&t->x, P.leb_val);
      else atomicAdd(t, make_float2(Wb[u].x * P.K, Wb[u].y * P.K));
    }
  }
}

struct FftPass {
  const float2* in;   // [rows, L] (unused by the first pass' functor loads)
  float2* out;        // [rows, L] (unused by the last pass' functor stores)
  int log2L, log2Ns, r, log2T;
  int sign;           // -1 forward, +1 inverse
  const float2* tw_lo;  // W_L^m, m in [0, 2^tw_s)
  const float2* tw_hi;  // W_L^(m << tw_s)
  int tw_s;
  int64_t row0;       // global row index of row 0 of this launch
  // ---- load functor -------------------------------------------------------------
  int load_mode;      // 0 plain, 1 padded real signal, 2 x-hat * psi-hat, 3 windowed STFT frame, 4 plain * mul[idx], 5 istft column, 6 strided rows
  const float* x;     // [channels, x_stride] (mode 1)
  int64_t x_stride, n;
  int padtype;
  const float2* xhat; // [channels, L] (mode 2)
  const float* scales;  // [ns] (mode 2)
  int ns, nd;         // scales per channel, rows per scale (1: W only, 2: W and dW)
  int wavelet;
  float inv_dt;
  int up_shift;       // mode 2: 7 * (number of leading passes skipped as broadcasts), see cwt_host.inl
  // mode 3 (STFT family through the row passes: n_fft > 4096 or not a power of two; stft_rows.inl): row r of the
  // launch is frame fr_first + r % fr_count of channel r / fr_count; element n < fr_nfft is
  // x_pad[frame * hop + n] * (win[n] + i dwin[n]) (* chirp[n] for Bluestein), the rest of the row is zero
  const float2* fr_wpair;  // [n_fft] (win, dwin * s)
  const float2* fr_chirp;  // [n_fft] exp(-i pi n^2 / n_fft) or NULL
  int fr_nfft, fr_hop, fr_left, fr_count;
  int64_t fr_first, fr_origin;
  // mode 5 (istft through the row passes): element n of the row is conj(Zfull[n]) (* chirp[n]), Zfull the Hermitian
  // extension of column fr_first + r % fr_count of in = Sx[channel][n_fft/2+1][fr_ld]
  int64_t fr_ld;
  // mode 4: in[row][idx] * mul[idx] (Bluestein: spectrum of the chirp filter, 1/M folded in)
  const float2* mul;
  // mode 6: rows of fr_nfft points with row stride fr_ld inside rows of L: in[row * fr_ld + idx] (conjugated when
  // conj_in) * fr_chirp[idx] (when given), zero beyond fr_nfft (icwt two-integral branch at any row length)
  int conj_in;
  // ---- CWT stream (cwt_host.inl, CwtBlocks) -----------------------------------------
  // x-hat row r of a stream call is block blk_first + r % blk_nb of channel r / blk_nb; blk_nb == 0 is the batch call
  // (row r is channel r).  Load mode 1 reads the block's extended input e[j] = x~[b C - d + j] (x~: the recording
  // mirrored with the edge sample repeated) from x (rows of x_stride, recording position rec_origin at column 0);
  // store modes 1 and 2 write row (channel, scale) of an output of out_pitch columns from column out_col0 + bl C.
  int blk_nb;
  int64_t blk_C, blk_d, blk_first, rec_n, rec_origin;
  int64_t out_pitch, out_col0;
  // ---- store functor ------------------------------------------------------------
  int store_mode;     // 0 plain, 1 final: scaled, unpadded rows to outW / outD, 2: fused ssq_cwt epilogue
  float2* outW;       // [channels, ns, out_cols]
  float2* outD;       // [channels, ns, out_cols] (may be NULL)
  int64_t out_cols, n1;  // columns [n1, n1 + out_cols) of the padded row: n (unpadded) or L (rpadded, n1 = 0)
  float out_scale;    // K / L   (K = de-normalisation constant of psi-hat)
  int l2_norm;
  // ---- fused ssq_cwt epilogue (store_mode 2, fft128_pass_kernel<TC, true> only) ------------------
  SsqCwtParams E;     // E.Tx: [channels, ns, E.pitch]
};

// Element offset of column 0 of row cs = (x-hat row) * ns + scale in an output of `pitch` columns per row
__device__ __forceinline__ size_t cwt_out_offset(const FftPass& P, unsigned cs, int64_t pitch) {
  if (P.blk_nb == 0) return (size_t)cs * pitch;
  const unsigned rb = cs / (unsigned)P.ns, si = cs - rb * (unsigned)P.ns;
  const unsigned ch = rb / (unsigned)P.blk_nb, bl = rb - ch * (unsigned)P.blk_nb;
  return ((size_t)ch * P.ns + si) * pitch + P.out_col0 + (size_t)bl * P.blk_C;
}

// GMW(gamma=3, beta=60) is evaluated as exp(60 ln w - w^3 - SSQ_GMW_LOGPEAK): peak 1
// instead of the reference's un-normalised 2*exp(...) (~4e17, cwt.rs:536-541), which
// would overflow c*c+d*d in fp32.  The constant is re-applied on store.
#define SSQ_GMW_WC 2.7144176165949063      /* (60/3)^(1/3) */
#define SSQ_GMW_LOGPEAK 39.914641217580179 /* 60 ln wc - wc^3 = 20 ln 20 - 20 */

__device__ __forceinline__ float2 tw_lookup(const FftPass& P, int64_t e) {
  // W_L^e, e in [0, L): two-level table (both tables computed in double on the host)
  const int lo = (int)(e & ((1 << P.tw_s) - 1));
  const int hi = (int)(e >> P.tw_s);
  float2 w = cmulf(__ldg(P.tw_lo + lo), __ldg(P.tw_hi + hi));
  if (P.sign > 0) w.y = -w.y;
  return w;
}

__device__ __forceinline__ float psihat(int wavelet, float w) {
  if (wavelet == SSQ_WAVELET_MORLET) {
    // cwt.rs:496-520: pi^-1/4 * sqrt2 * (exp(-(w-6)^2/2) - exp(-18) exp(-w^2/2)), w >= 0
    if (!(w >= 0.f)) return 0.f;
    if (w > 14.5f) return 0.f;  // exp(-(w-6)^2/2) < 2e-16 of the peak: below fp32 resolution of any sum
    const float norm = 1.0622519320271968f;  // pi^-0.25 * sqrt(2)
    const float kexp = 1.5229979744712629e-08f;  // exp(-18)
    const float d = w - 6.f;
    return norm * (expf(-0.5f * d * d) - kexp * expf(-0.5f * w * w));
  }
  // cwt.rs:522-541 (anything else is GMW): 2*exp(60 ln w - w^3), w > 0; normalised here
  if (!(w > 0.f)) return 0.f;
  // outside (1.0, 4.5) the peak-normalised value is < 1e-17 (60 ln w - w^3 - 39.9 < -40): skip the
  // transcendental evaluation, far below fp32 resolution of any sum it enters
  if (w < 1.0f || w > 4.5f) return 0.f;
  return expf(60.f * logf(w) - w * w * w - (float)SSQ_GMW_LOGPEAK);
}

// Stream call: the reference's pad of the extended block input e (length P.n), then e[j] = x~[b C - d + j] with the
// symmetric fold at the recording ends (x~[q] = x[-1 - q], q < 0; x[2 N - 1 - q], q >= N: np.pad mode "symmetric",
// dask's boundary="reflect"), read in place from the carry-over buffer.  d <= C and d <= N: one fold suffices.
__device__ __forceinline__ float cwt_block_sample(const FftPass& P, int64_t g, int64_t p, int64_t L) {
  int64_t o = p - (L - P.n) / 2;
  if (o < 0 || o >= P.n) {
    if (P.padtype == SSQ_PAD_ZERO) return 0.f;
    o = o < 0 ? -o : 2 * P.n - 2 - o;
    if (o < 0 || o >= P.n) return 0.f;
  }
  const int64_t ch = g / P.blk_nb, b = P.blk_first + (g - ch * P.blk_nb);
  int64_t q = b * P.blk_C - P.blk_d + o;
  if (q < 0) q = -1 - q;
  else if (q >= P.rec_n) q = 2 * P.rec_n - 1 - q;
  return __ldg(P.x + (size_t)ch * P.x_stride + (q - P.rec_origin));
}

__device__ __forceinline__ float cwt_sample(const FftPass& P, int64_t g, int64_t p, int64_t L) {
  if (P.blk_nb) return cwt_block_sample(P, g, p, L);
  // utils/array.rs:52-98: left = (L-n)/2
  const float* x = P.x + (size_t)g * P.x_stride;
  const int64_t left = (L - P.n) / 2;
  const int64_t o = p - left;
  if (o >= 0 && o < P.n) return __ldg(x + o);
  if (P.padtype == SSQ_PAD_ZERO) return 0.f;
  if (o < 0) {
    const int64_t m = -o;
    return m < P.n ? __ldg(x + m) : 0.f;
  }
  const int64_t m = 2 * P.n - 2 - o;
  return (m >= 0 && m < P.n) ? __ldg(x + m) : 0.f;
}

__device__ __forceinline__ float2 pass_load(const FftPass& P, int row, int64_t idx) {
  const int64_t L = (int64_t)1 << P.log2L;
  if (P.load_mode == 0) return P.in[(size_t)row * L + idx];
  const int64_t g = P.row0 + row;
  if (P.load_mode == 1) return make_float2(cwt_sample(P, g, idx, L), 0.f);
  if (P.load_mode == 4) return cmulf(P.in[(size_t)row * L + idx], __ldg(P.mul + idx));
  if (P.load_mode == 6) {
    if (idx >= P.fr_nfft) return make_float2(0.f, 0.f);
    float2 v = P.in[(size_t)row * P.fr_ld + idx];
    if (P.conj_in) v.y = -v.y;
    if (P.fr_chirp) v = cmulf(v, __ldg(P.fr_chirp + idx));
    return v;
  }
  if (P.load_mode == 5) {
    if (idx >= P.fr_nfft) return make_float2(0.f, 0.f);
    const int64_t ch = g / P.fr_count, frame = P.fr_first + (g - ch * P.fr_count);
    const int nfq = P.fr_nfft / 2 + 1;
    const int k = idx < nfq ? (int)idx : P.fr_nfft - (int)idx;
    float2 v = P.in[((size_t)ch * nfq + k) * P.fr_ld + frame];
    if (idx < nfq) v.y = -v.y;
    if (P.fr_chirp) v = cmulf(v, __ldg(P.fr_chirp + idx));
    return v;
  }
  if (P.load_mode == 3) {
    if (idx >= P.fr_nfft) return make_float2(0.f, 0.f);
    const int64_t ch = g / P.fr_count, frame = P.fr_first + (g - ch * P.fr_count);
    const float xv = stft_sample(P.x + (size_t)ch * P.x_stride, P.n, frame * P.fr_hop + idx, P.fr_left, P.padtype, P.fr_origin);
    const float2 w = __ldg(P.fr_wpair + idx);
    float2 v = make_float2(xv * w.x, xv * w.y);
    if (P.fr_chirp) v = cmulf(v, __ldg(P.fr_chirp + idx));
    return v;
  }
  // mode 2: row g -> (channel, scale, which)
  const int which = (int)(g % P.nd);
  const int64_t cs = g / P.nd;
  const int si = (int)(cs % P.ns);
  const int ch = (int)(cs / P.ns);
  // band-limited rows: the skipped leading passes are broadcasts, their output at idx is the
  // spectrum at idx >> up_shift (cwt_host.inl, cwt_skip_level)
  idx >>= P.up_shift;
  // wavelets/base.rs:18-33 with scale 1: xi = 2 pi idx / L (idx <= L/2), 2 pi (idx - L) / L above
  const float xi = 6.283185307179586f * ((idx <= (L >> 1)) ? (float)idx : (float)(idx - L)) / (float)L;
  const float ps = psihat(P.wavelet, __ldg(P.scales + si) * xi);
  if (ps == 0.f) return make_float2(0.f, 0.f);
  const float2 xh = __ldg(P.xhat + (size_t)ch * L + idx);
  float2 v = make_float2(xh.x * ps, xh.y * ps);
  if (which == 1) {  // * i*xi/dt (cwt.rs:205-209, ssq_cwt.rs:374-377)
    const float f = xi * P.inv_dt;
    v = make_float2(-v.y * f, v.x * f);
  }
  return v;
}

__device__ __forceinline__ void pass_store(const FftPass& P, int row, int64_t o, float2 v) {
  const int64_t L = (int64_t)1 << P.log2L;
  if (P.store_mode == 0) {
    P.out[(size_t)row * L + o] = v;
    return;
  }
  const int64_t col = o - P.n1;
  if (col < 0 || col >= P.out_cols) return;
  const int64_t g = P.row0 + row;
  const int which = (int)(g % P.nd);
  const int64_t cs = g / P.nd;  // channel*ns + scale
  float s = P.out_scale;
  if (P.l2_norm) s *= sqrtf(__ldg(P.scales + (int)(cs % P.ns)));  // cwt.rs:253
  float2* dst = which ? P.outD : P.outW;
  dst[cwt_out_offset(P, (unsigned)cs, P.out_pitch) + col] = make_float2(v.x * s, v.y * s);
}

// grid: (L / (R*T), rows).  Dynamic smem: 2 * R * T float2.
__global__ void __launch_bounds__(256) fft_pass_kernel(const FftPass P) {
  extern __shared__ float2 smem[];
  const int R = 1 << P.r, T = 1 << P.log2T;
  const int64_t L = (int64_t)1 << P.log2L;
  const int64_t Ns = (int64_t)1 << P.log2Ns;
  const int64_t Q = L >> P.r;  // L / R: number of butterflies per row
  float2* A = smem;
  float2* B = smem + R * T;
  const int row = blockIdx.y;
  const int64_t j0 = (int64_t)blockIdx.x * T;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int twshift = P.log2L - P.log2Ns - P.r;  // W_{Ns R}^e = W_L^(e << twshift)

  for (int e = tid; e < R * T; e += nt) {
    const int t = e >> P.log2T, c = e & (T - 1);
    const int64_t j = j0 + c;
    float2 v = pass_load(P, row, j + (int64_t)t * Q);
    if (P.log2Ns > 0 && t > 0) {
      const int64_t k = j & (Ns - 1);
      v = cmulf(v, tw_lookup(P, (k * t) << twshift));
    }
    A[e] = v;
  }
  __syncthreads();
  // R-point DFT along t for each of the T columns: radix-2 Stockham sub-stages
  const int half = (R >> 1) * T;
  for (int s = 0; s < P.r; ++s) {
    const int ns = 1 << s;
    const int sub_shift = P.log2L - (s + 1);  // W_{2 ns}^kk = W_L^(kk << sub_shift)
    for (int e = tid; e < half; e += nt) {
      const int b = e >> P.log2T, c = e & (T - 1);
      const int kk = b & (ns - 1);
      const float2 a = A[b * T + c];
      float2 bb = A[(b + (R >> 1)) * T + c];
      if (kk) bb = cmulf(bb, tw_lookup(P, (int64_t)kk << sub_shift));
      const int o = ((b - kk) << 1) + kk;
      B[o * T + c] = caddf(a, bb);
      B[(o + ns) * T + c] = csubf(a, bb);
    }
    __syncthreads();
    float2* t2 = A; A = B; B = t2;
  }
  // store: out[(j-k)*R + k + t*Ns], k = j mod Ns
  if (Ns >= T) {
    for (int e = tid; e < R * T; e += nt) {
      const int t = e >> P.log2T, c = e & (T - 1);
      const int64_t j = j0 + c;
      const int64_t k = j & (Ns - 1);
      pass_store(P, row, ((j - k) << P.r) + k + (int64_t)t * Ns, A[e]);
    }
  } else {
    // Ns < T: the CTA's outputs form one contiguous block [j0*R, (j0+T)*R)
    const int nsr = (int)(Ns << P.r);
    for (int e = tid; e < R * T; e += nt) {
      const int a = e / nsr, rem = e - a * nsr;
      const int t = rem >> P.log2Ns, k = rem & ((int)Ns - 1);
      const int c = a * (int)Ns + k;
      pass_store(P, row, (j0 << P.r) + e, A[t * T + c]);
    }
  }
}

// ------------------------------------------------------------------------------------
// Radix-128 pass, register butterflies (the fast path of every 7-bit pass):
// CTA = 128 (t) x 32 (adjacent columns j); thread (c = tid & 31, g = tid >> 5) loads
// t = g + 8 u (u = 0..15; each load is a 256 B run across the warp), does the 16-point DFT
// over u in registers, multiplies by W_128^{g k1}, exchanges once through shared memory,
// then (c, h) does the two 8-point DFTs over g for k1 in {h, h + 8}:
//   Y[k1 + 16 k2] = sum_g W_8^{g k2} W_128^{g k1} sum_u x[g + 8 u] W_16^{u k1}.
// The inverse transform is conj(forward(conj)): conjugation is folded into load and store.
// Requires log2Ns == 0 (first pass; output block is transposed through shared memory so the
// CTA writes 32 KB contiguously) or Ns >= 32 (outputs of adjacent columns are adjacent).
// grid: (L / (128 TC), rows), 8 TC threads, TC * 129 * 8 B dynamic shared memory.
// ------------------------------------------------------------------------------------
__device__ __forceinline__ void fft4_fwd(float2& a, float2& b, float2& c, float2& d) {
  const float2 apc = caddf(a, c), amc = csubf(a, c), bpd = caddf(b, d), bmd = csubf(b, d);
  a = caddf(apc, bpd);
  b = make_float2(amc.x + bmd.y, amc.y - bmd.x);  // amc - i bmd
  c = csubf(apc, bpd);
  d = make_float2(amc.x - bmd.y, amc.y + bmd.x);  // amc + i bmd
}

// in: v[u], u = 0..15; out: v[a + 4 b] = X[a + 4 b] (natural order)
__device__ __forceinline__ void fft16_fwd(float2 (&v)[16]) {
  const float C1 = 0.92387953251128673848f, S1 = 0.38268343236508978178f, H = 0.70710678118654752440f;
  // step 1: 4-point DFTs over u1 of v[u0 + 4 u1] -> v[u0 + 4 a]
#pragma unroll
  for (int u0 = 0; u0 < 4; ++u0) fft4_fwd(v[u0], v[u0 + 4], v[u0 + 8], v[u0 + 12]);
  // step 2: twiddles W_16^{u0 a} on v[u0 + 4 a]
  v[5] = cmulf(v[5], make_float2(C1, -S1));    // u0=1,a=1: W^1
  v[9] = cmulf(v[9], make_float2(H, -H));      // u0=1,a=2: W^2
  v[13] = cmulf(v[13], make_float2(S1, -C1));  // u0=1,a=3: W^3
  v[6] = cmulf(v[6], make_float2(H, -H));      // u0=2,a=1: W^2
  v[10] = make_float2(v[10].y, -v[10].x);      // u0=2,a=2: W^4 = -i
  v[14] = cmulf(v[14], make_float2(-H, -H));   // u0=2,a=3: W^6
  v[7] = cmulf(v[7], make_float2(S1, -C1));    // u0=3,a=1: W^3
  v[11] = cmulf(v[11], make_float2(-H, -H));   // u0=3,a=2: W^6
  v[15] = cmulf(v[15], make_float2(-C1, S1));  // u0=3,a=3: W^9
  // step 3: 4-point DFTs over u0 for each a: X[a + 4 b] lands in v[4 a + b]
#pragma unroll
  for (int a = 0; a < 4; ++a) fft4_fwd(v[4 * a], v[4 * a + 1], v[4 * a + 2], v[4 * a + 3]);
  // reorder v[4 a + b] -> v[a + 4 b]
  float2 t;
  t = v[1]; v[1] = v[4]; v[4] = t;
  t = v[2]; v[2] = v[8]; v[8] = t;
  t = v[3]; v[3] = v[12]; v[12] = t;
  t = v[6]; v[6] = v[9]; v[9] = t;
  t = v[7]; v[7] = v[13]; v[13] = t;
  t = v[11]; v[11] = v[14]; v[14] = t;
}

__device__ __forceinline__ float2 tw_fwd(const FftPass& P, int64_t e) {  // W_L^e, forward sign
  const int lo = (int)(e & ((1 << P.tw_s) - 1));
  const int hi = (int)(e >> P.tw_s);
  return cmulf(__ldg(P.tw_lo + lo), __ldg(P.tw_hi + hi));
}

// FUSED (the last pass of ssq_cwt, ssq_cwt.rs:365-480 in one pass over the scales): the CTA works on the W row and
// the dW row of ONE scale at once -- adjacent lanes (2 col, 2 col + 1) carry the same column of the two rows, so after
// the second butterfly a lane pair swaps halves (8 shuffles) and each lane holds Wx and dWx of 8 outputs: phase
// transform, bin and the update of Tx happen straight from the registers; Wx / dWx are never written.  The update is
// a vector reduction (red.global.add.v2.f32): several scales may hit one Tx element from different CTAs, so the
// order of additions inside an element is not fixed (rounding-level; the bins are).
template <int TC, bool FUSED = false>  // TC adjacent columns per CTA (16 or 32): TC * 8 B contiguous per global access, 8 * TC threads
__global__ void __launch_bounds__(8 * TC) fft128_pass_kernel(const FftPass P) {
  extern __shared__ float2 buf[];  // [TC * 129]
  __shared__ float2 w128[128];  // W_128^m
  const int cfull = threadIdx.x % TC, g = threadIdx.x / TC;
  const int which_l = FUSED ? (cfull & 1) : 0;      // FUSED: 0 = W row, 1 = dW row
  const int c = FUSED ? (cfull >> 1) : cfull;       // column inside the CTA
  constexpr int CW = FUSED ? TC / 2 : TC;           // columns per CTA
  if (threadIdx.x < 128) w128[threadIdx.x] = tw_fwd(P, (int64_t)threadIdx.x << (P.log2L - 7));
  __shared__ float2* s_tch;  // FUSED: base of the channel's Tx (flip folded in) and of the diagnostics row
  __shared__ size_t s_drow;
  if (FUSED && threadIdx.x == 128) {
    const unsigned cs0 = ((unsigned)P.row0 + 2u * blockIdx.y) >> 1;  // channel * ns + scale (rows: channel, scale, which)
    const unsigned chn0 = cs0 / (unsigned)P.E.ns;
    s_tch = P.E.Tx + cwt_out_offset(P, chn0 * (unsigned)P.E.ns, P.E.pitch) +
            (P.E.flipud ? (size_t)(P.E.ns - 1) * P.E.pitch : (size_t)0);
    s_drow = (size_t)cs0 * P.E.n;
  }
  // in-row indices are 32-bit (L <= 2^27, checked on the host): the passes are issue-bound and 64-bit
  // index arithmetic was a fifth of their instructions
  const int L = 1 << P.log2L;
  const int Q = L >> 7;
  const int Ns = 1 << P.log2Ns;
  const int row = FUSED ? 2 * (int)blockIdx.y + which_l : (int)blockIdx.y;
  const int j0 = blockIdx.x * CW, j = j0 + c;
  const int kk = j & (Ns - 1);
  const int twshift = P.log2L - P.log2Ns - 7;  // W_{128 Ns}^e = W_L^(e << twshift)
  const bool inv = P.sign > 0;

  float2 v[16];
  // Pruned generation (band-limited rows whose leading passes were skipped, up_shift >= 6): input t of EVERY column of
  // the CTA is the same spectrum bin (j0 >> S) + t (Q >> S), so the 128 products x-hat psi-hat are evaluated once per
  // CTA (per row of the pair when FUSED) into shared memory instead of 16 times per thread: expf / logf and the index
  // logic were 35 % of these passes (ncu r2f).
  __shared__ float2 ytab[FUSED ? 256 : 128];
  const bool shared_gen = P.load_mode == 2 && P.up_shift >= 6 && P.up_shift <= P.log2L - 7;
  if (shared_gen) {
    if (threadIdx.x < (FUSED ? 256 : 128)) {
      const int t = threadIdx.x & 127;
      const int wrow = FUSED ? 2 * (int)blockIdx.y + (int)(threadIdx.x >> 7) : (int)blockIdx.y;
      const unsigned gr = (unsigned)P.row0 + (unsigned)wrow;
      const unsigned cs = gr / (unsigned)P.nd;
      const int which = (int)(gr - cs * (unsigned)P.nd);
      const unsigned chn = cs / (unsigned)P.ns;
      const float scale = __ldg(P.scales + (int)(cs - chn * (unsigned)P.ns));
      const int idx = (j0 >> P.up_shift) + t * (Q >> P.up_shift);
      float2 x = make_float2(0.f, 0.f);
      if (idx <= (L >> 1)) {  // negative frequencies: psi-hat = 0 (cwt.rs:496-541)
        const float xi = (6.283185307179586f * (float)idx) * (1.f / (float)L);
        const float ps = psihat(P.wavelet, scale * xi);
        if (ps != 0.f) {
          const float2 h = __ldg(P.xhat + (size_t)chn * L + idx);
          x = make_float2(h.x * ps, h.y * ps);
          if (which == 1) {  // * i*xi/dt (cwt.rs:205-209, ssq_cwt.rs:374-377)
            const float f = xi * P.inv_dt;
            x = make_float2(-x.y * f, x.x * f);
          }
        }
      }
      if (inv) x.y = -x.y;
      ytab[threadIdx.x] = x;
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < 16; ++u) v[u] = ytab[(FUSED ? 128 * which_l : 0) + g + 8 * u];
  } else if (P.load_mode == 2) {
    // x-hat * psi-hat generated on the fly: the row's constants once per thread, and an exact integer
    // early-out -- psihat() returns 0 beyond its cut-off, i.e. for spectrum indices >= blim
    // 32-bit row arithmetic (the host refuses more than 2^31 rows): three 64-bit divisions per thread were
    // 7.6 % of a generation pass
    const unsigned gr = (unsigned)P.row0 + (unsigned)row;
    const unsigned cs = gr / (unsigned)P.nd;
    const int which = (int)(gr - cs * (unsigned)P.nd);
    const unsigned chn = cs / (unsigned)P.ns;
    const float scale = __ldg(P.scales + (int)(cs - chn * (unsigned)P.ns));
    const float2* xh = P.xhat + (size_t)chn * L;
    const float cut = P.wavelet == SSQ_WAVELET_MORLET ? 14.5f : 4.5f;
    const float inv_L = 1.f / (float)L;
    int blim = (L >> 1) + 1;  // negative frequencies: psi-hat = 0 (cwt.rs:496-541)
    if (scale > 0.f) blim = (int)fminf((float)blim, cut * (float)L / (6.283185307179586f * scale) * 1.0001f + 2.f);
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      const int idx = (j + (g + 8 * u) * Q) >> P.up_shift;
      float2 x = make_float2(0.f, 0.f);
      if (idx < blim) {
        const float xi = (6.283185307179586f * (float)idx) * inv_L;  // wavelets/base.rs:18-33, idx <= L/2 (L = 2^k: exact)
        const float ps = psihat(P.wavelet, scale * xi);
        if (ps != 0.f) {
          const float2 h = __ldg(xh + idx);
          x = make_float2(h.x * ps, h.y * ps);
          if (which == 1) {  // * i*xi/dt (cwt.rs:205-209, ssq_cwt.rs:374-377)
            const float f = xi * P.inv_dt;
            x = make_float2(-x.y * f, x.x * f);
          }
        }
      }
      if (inv) x.y = -x.y;
      v[u] = x;
    }
  } else if (P.load_mode == 0) {
    // plain row of a previous pass: one base pointer, 32-bit in-row offsets (the generic functor spent 18
    // instructions per load on 64-bit index arithmetic and mode checks: 29 % of the pass, ncu r1s)
    const float2* inrow = P.in + (size_t)row * L + (j + g * Q);
#pragma unroll
    for (int u = 0; u < 16; ++u) v[u] = inrow[(unsigned)(8 * u) * (unsigned)Q];
    if (inv) {
#pragma unroll
      for (int u = 0; u < 16; ++u) v[u].y = -v[u].y;
    }
  } else {
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      float2 x = pass_load(P, row, j + (g + 8 * u) * Q);
      if (inv) x.y = -x.y;
      v[u] = x;
    }
  }
  if (P.log2Ns > 0) {
    // inter-pass twiddle W^{kk (g + 8u)} = W^{kk g} (W^{8 kk})^u: two table look-ups, then powers by
    // repeated squaring / short products (every power is at most 4 multiplications deep)
    // q[u] = W^{kk g} (W^{8 kk})^u built by doubling (q[u + 2^i] = q[u] p^(2^i)): 3 + 15 complex multiplications
    // instead of 14 + 15, every factor at most 5 products deep
    float2 q[16];
    q[0] = tw_fwd(P, (int64_t)((kk * g) << twshift));
    const float2 p1 = tw_fwd(P, (int64_t)((kk * 8) << twshift));
    const float2 p2 = cmulf(p1, p1), p4 = cmulf(p2, p2), p8 = cmulf(p4, p4);
    q[1] = cmulf(q[0], p1);
    q[2] = cmulf(q[0], p2);
    q[3] = cmulf(q[1], p2);
#pragma unroll
    for (int u = 0; u < 4; ++u) q[4 + u] = cmulf(q[u], p4);
#pragma unroll
    for (int u = 0; u < 8; ++u) q[8 + u] = cmulf(q[u], p8);
#pragma unroll
    for (int u = 0; u < 16; ++u) v[u] = cmulf(v[u], q[u]);
  }
  fft16_fwd(v);  // v[k1] = sum_u x[g + 8u] W_16^{u k1}
  __syncthreads();  // w128 ready
  if (g) {
#pragma unroll
    for (int k1 = 1; k1 < 16; ++k1) v[k1] = cmulf(v[k1], w128[(g * k1) & 127]);
  }
#pragma unroll
  for (int k1 = 0; k1 < 16; ++k1) buf[(k1 * 8 + g) * TC + cfull] = v[k1];
  __syncthreads();
  float2 a[8], b[8];
#pragma unroll
  for (int gg = 0; gg < 8; ++gg) {
    a[gg] = buf[(g * 8 + gg) * TC + cfull];        // k1 = h = g
    b[gg] = buf[((g + 8) * 8 + gg) * TC + cfull];  // k1 = h + 8
  }
  fft8_fwd(a);  // a[k2] = Y[g + 16 k2]
  fft8_fwd(b);  // b[k2] = Y[g + 8 + 16 k2]
  // (the fused epilogue works on the conjugates as they are: |W|^2 and |Im(dW conj W)| do not change, the value added
  // to Tx takes the sign with its factor)
  if (inv && !FUSED) {
#pragma unroll
    for (int k2 = 0; k2 < 8; ++k2) {
      a[k2].y = -a[k2].y;
      b[k2].y = -b[k2].y;
    }
  }
  if constexpr (FUSED) {
    // even lane (W row): keeps a = W[k1 = g], receives the dW row's a; odd lane: keeps b = dW[k1 = g + 8], receives
    // the W row's b.  Each lane then owns 8 outputs o = base + (koff + 16 k2) Ns with both values.
    // CTA-uniform constants (a division and 64-bit products: 10 % of the pass when every thread computed them):
    // thread 0 wrote them before the barrier above
    // (the 1/L of the inverse transform is folded into E.K and E.gate by the host: the phase ratio is scale-free)
    const int base = ((j - kk) << 7) + kk - (int)P.n1;
    const int koff = g + 8 * which_l;
    // row of Tx = flipud ? ns - 1 - bin : bin, as a signed 32-bit element offset from a per-channel base (the host
    // takes this path only while ns * pitch < 2^31): one integer multiply-add per item
    const int rstep = P.E.flipud ? -(int)P.E.pitch : (int)P.E.pitch;
    float2* Tch = s_tch;
    const size_t drow = s_drow;  // diagnostics: [channels, ns, n]
    const bool diag = P.E.aux_kb != nullptr || P.E.aux_w != nullptr;
    const bool leb = P.E.squeezing == SSQ_SQUEEZE_LEBESGUE;
    const float Kx = P.E.K, Ky = inv ? -P.E.K : P.E.K;
    int col = base + koff * Ns;
    const int cstep = 16 * Ns;
#pragma unroll
    for (int k2 = 0; k2 < 8; ++k2, col += cstep) {
      // columns outside the unpadded signal (half of a padded row) are dropped before the exchange: the test is
      // uniform over the warp for the padded lengths of the CWT, a vote keeps it safe in general
      const bool inside = (unsigned)col < (unsigned)P.E.n;
      if (!__any_sync(0xffffffffu, inside)) continue;
      const float2 send = which_l ? a[k2] : b[k2];
      float2 recv;
      recv.x = __shfl_xor_sync(0xffffffffu, send.x, 1);
      recv.y = __shfl_xor_sync(0xffffffffu, send.y, 1);
      if (!inside) continue;
      const float2 Wv = which_l ? recv : a[k2], Dv = which_l ? b[k2] : recv;
      float w;
      const int bin = ssq_cwt_bin(P.E, Wv, Dv, w);
      if (diag) {
        if (P.E.aux_kb) P.E.aux_kb[drow + col] = bin < 0 ? -1 : (P.E.flipud ? P.E.ns - 1 - bin : bin);
        if (P.E.aux_w) P.E.aux_w[drow + col] = w;
      }
      if (bin < 0) continue;
      float2* t = Tch + (bin * rstep + col);
      if (leb) atomicAdd(&t->x, P.E.leb_val);
      else atomicAdd(t, make_float2(Wv.x * Kx, Wv.y * Ky));
    }
    return;
  }
  // store functor with the row's constants hoisted (the per-element version divides 64-bit indices)
  float2* sdst = P.out + (size_t)row * L;
  float sscale = 1.f;
  int soff = 0, scols = L;
  if (P.store_mode == 1) {
    const unsigned gr = (unsigned)P.row0 + (unsigned)row;
    const unsigned cs = gr / (unsigned)P.nd;  // channel * ns + scale
    sdst = ((gr - cs * (unsigned)P.nd) ? P.outD : P.outW) + cwt_out_offset(P, cs, P.out_pitch);
    sscale = P.out_scale;
    if (P.l2_norm) sscale *= sqrtf(__ldg(P.scales + (int)(cs % (unsigned)P.ns)));  // cwt.rs:253
    soff = (int)P.n1;
    scols = (int)P.out_cols;
  }
  auto store = [&](int o, float2 val) {
    const int col = o - soff;
    if (col >= 0 && col < scols) sdst[col] = make_float2(val.x * sscale, val.y * sscale);
  };
  if (P.log2Ns == 0) {
    // out index = j * 128 + k: transpose so that the CTA writes its 4096 outputs contiguously
    __syncthreads();
#pragma unroll
    for (int k2 = 0; k2 < 8; ++k2) {
      buf[c * 129 + g + 16 * k2] = a[k2];
      buf[c * 129 + g + 8 + 16 * k2] = b[k2];
    }
    __syncthreads();
    if (P.store_mode == 0) {
      float2* orow = P.out + (size_t)row * L + (j0 << 7) + threadIdx.x;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int e = threadIdx.x + 8 * TC * i;
        orow[8 * TC * i] = buf[(e >> 7) * 129 + (e & 127)];
      }
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int e = threadIdx.x + 8 * TC * i;
        store((j0 << 7) + e, buf[(e >> 7) * 129 + (e & 127)]);
      }
    }
  } else if (P.store_mode == 0) {
    // intermediate pass: whole rows, no window, no scaling
    float2* orow = P.out + (size_t)row * L + (((j - kk) << 7) + kk + g * Ns);
#pragma unroll
    for (int k2 = 0; k2 < 8; ++k2) {
      orow[(unsigned)(16 * k2) * (unsigned)Ns] = a[k2];
      orow[(unsigned)(16 * k2 + 8) * (unsigned)Ns] = b[k2];
    }
  } else {
    const int base = ((j - kk) << 7) + kk;
#pragma unroll
    for (int k2 = 0; k2 < 8; ++k2) {
      store(base + (g + 16 * k2) * Ns, a[k2]);
      store(base + (g + 8 + 16 * k2) * Ns, b[k2]);
    }
  }
}

// ------------------------------------------------------------------------------------
// icwt, one-integral branch (cwt.rs:590-627): x[c][j] = final_norm * sum_i Re Wx[c][i][j] * norm_i + x_mean,
// scales ascending in i as the reference sums them; coalesced along j.
// ------------------------------------------------------------------------------------
__global__ void icwt_kernel(const float2* __restrict__ Wx, int64_t ns, int64_t n_cols, int64_t x_len,
                            const float* __restrict__ norm, float final_norm, float x_mean, float* __restrict__ x) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t c = blockIdx.y;
  if (j >= x_len) return;
  const float2* w = Wx + (size_t)c * ns * n_cols + j;
  float s = 0.f;
  for (int64_t i = 0; i < ns; ++i) s = fmaf(w[(size_t)i * n_cols].x, __ldg(norm + i), s);
  x[(size_t)c * x_len + j] = fmaf(s, final_norm, x_mean);
}

// ------------------------------------------------------------------------------------
// icwt, two-integral branch (cwt.rs:629-712) in the frequency domain:
//   S[k] = sum_i FFT(Wx[i])[k] * psi-hat(scale_i xi_k) / scale_i   (psi-hat real; peak-normalised here, the constant
//   goes into the final factor), then x = Re(IFFT(S)) * norm + x_mean.
// ------------------------------------------------------------------------------------
// What: [ns] rows of stride ld (spectra of the rows; times zmul[k] when given: Bluestein); N: transform length
__global__ void icwt2_accum_kernel(const float2* __restrict__ What, int64_t ld, const float2* __restrict__ zmul, int ns,
                                   int N, const float* __restrict__ scales, int wavelet, float2* __restrict__ S) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= N) return;
  // wavelets/base.rs:18-33: xi_k = 2 pi k / N up to and including the Nyquist bin, 2 pi (k - N) / N above
  const float xi = 6.283185307179586f * (float)(k <= (N >> 1) ? k : k - N) / (float)N;
  float2 acc = make_float2(0.f, 0.f);
  for (int i = 0; i < ns; ++i) {
    const float sc = __ldg(scales + i);
    const float ps = psihat(wavelet, sc * xi);
    if (ps != 0.f) {
      const float2 w = What[(size_t)i * ld + k];
      const float f = ps / sc;  // 1/scale for both norms (cwt.rs:684-688: 1/scale and 1/sqrt(scale)^2)
      acc.x = fmaf(w.x, f, acc.x);
      acc.y = fmaf(w.y, f, acc.y);
    }
  }
  if (zmul) acc = cmulf(acc, __ldg(zmul + k));
  S[k] = acc;
}

__global__ void icwt2_finalize_kernel(const float2* __restrict__ s, const float2* __restrict__ zmul, int64_t L,
                                      float norm, float x_mean, float* __restrict__ x) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= L) return;
  float2 v = s[j];
  if (zmul) v = cmulf(v, __ldg(zmul + j));
  x[j] = fmaf(v.x, norm, x_mean);
}

