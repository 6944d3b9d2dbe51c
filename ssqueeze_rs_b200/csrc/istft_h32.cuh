// istft_h32.cuh -- inverse STFT for n_fft = 512, any hop (BASELINE.json configs[3]: hop = 32).
//
// old/ssqueezepy/_stft.py:184-256 in the Rust framing (unmodulated, unpad at
// (n_fft-1)/2):
//   * two frames share one complex 512-point FFT: Z = ZA + i ZB with the Hermitian
//     extension built on the fly, x_A = Re, x_B = Im of the inverse transform (the
//     imaginary parts of the DC and Nyquist bins are dropped as irfft does);
//   * with hop == warp size, sample n = lane + 32 j of frame f lands on padded position
//     32 (f + j) + lane, i.e. in the SAME lane for every frame, so a warp adds its frames
//     in a 16-register window;
//   * samples at the two ends of a tile are shared with the neighbouring tiles: every
//     sample is emitted with one red.global.add.f32 into a zeroed buffer
//     (at most two addends per element: exact and order-independent);
//   * istft_finalize_kernel divides by the window norm and unpads.
#pragma once
#include "fft_regs.cuh"

// floor(p / hop) for 0 <= p < 2^23 without the ~20-instruction integer division: float estimate, then corrected
// (the gather of the tile kernels divided twice per sample: 27 % of istft1024's instructions, ncu r1w)
__device__ __forceinline__ int ssq_fast_div(int p, int hop, float inv_hop) {
  int q = (int)((float)p * inv_hop);
  q -= (q * hop > p);
  q += ((q + 1) * hop <= p);
  return q;
}

#define I32_AS 260  // tile column stride (float2): >= 257 and == 4 mod 16 (conflict-free quad writes)

struct Istft32Params {
  const float2* Sx;  // [channels, 257, n_frames]
  int channels;
  int64_t n_frames, n_use, L;
  const float* wa;   // [512] window^win_exp / 512
  const float2* tw;  // [512]
  float* xacc;       // [channels, L] zero-initialised
  int run;           // frames per run (multiple of 4)
  int64_t runs_per_channel, total_runs;
  int hop;           // any hop >= 1
  int n_fft;         // host only: the launchers' guard
};

// A CTA owns 32 consecutive frames (a warp fetching its own quads of frames left every
// 128 B line of Sx "open" for four quads of one warp; with 2368 warps that is ~78 MB of
// partially consumed lines, L2 thrashed and DRAM read 2.2x the input: ncu r1f): the
// [257 x 32] tile is loaded with 256 B row segments, warp w transforms frames 4w..4w+3
// (two packed pairs) and parks the windowed samples in the frame's own tile row; the
// overlap-add is a gather (each padded sample sums the <= 16 rows that cover it: no
// shared-memory atomics), one red.global.add per sample and tile.
// ------------------------------------------------------------------------------------
#define I32T_AS 289  // tile row stride (float2): odd -> conflict-free transposed tile load; 578 floats >= 512
// warps per CTA, tile = 4 NW = 32 frames, 2 CTAs per SM (4 warps x 16 frames, 4 CTAs per SM: 10.2 vs 9.5 ms)
#define I32T_NW 8

template <bool HOP32>  // hop == 32: shifts instead of integer divisions in the gather
__global__ void __launch_bounds__(I32T_NW * 32, 16 / I32T_NW) istft512_tile_kernel(const Istft32Params P) {
  constexpr int N = 512, AS = I32T_AS, NW = I32T_NW, F = 4 * NW;
  static_assert(F == 32, "the tile load maps lane -> frame and warp -> row: 8 warps x 32 frames");
  extern __shared__ float2 smem[];
  float2* tw2tab = smem;      // [8][9]
  float2* S = smem + 72;      // [32][AS]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float2* xch = S + F * AS + warp * N;
  if (threadIdx.x < 64)
    tw2tab[(threadIdx.x >> 3) * 9 + (threadIdx.x & 7)] = P.tw[((threadIdx.x >> 3) * (threadIdx.x & 7) * 8) & (N - 1)];

  H32Lane L;
  L.lane = lane;
  L.j2 = lane + 32;
  L.tw2 = tw2tab + (lane & 7) * 9;
#pragma unroll
  for (int t = 1; t < 8; ++t) {
    L.tw3a[t - 1] = P.tw[(lane * t) & (N - 1)];
    L.tw3b[t - 1] = P.tw[(L.j2 * t) & (N - 1)];
  }
  L.f1 = (lane >> 1) & 3;
  L.rd1a = (lane >> 3) * 8 + ((((lane & 7) >> 1) ^ ((lane >> 4) & 3)) << 1) + (lane & 1);
  L.rd1b = ((lane >> 3) + 4) * 8 + ((((lane & 7) >> 1) ^ (((lane >> 4) + 2) & 3)) << 1) + (lane & 1);
  L.g2 = (lane >> 3) & 1;
  L.wr2 = (lane >> 3) * 64 + (lane & 7);
  L.lane_f = 0.f;
  L.j2_f = 0.f;
  L.l0 = (lane == 0);
  float war[16];  // window^a / N at n = lane + 32 j
#pragma unroll
  for (int j = 0; j < 16; ++j) war[j] = P.wa[lane + 32 * j];
  __syncthreads();

  for (int64_t tile = blockIdx.x; tile < P.total_runs; tile += gridDim.x) {
    const int ch = (int)(tile / P.runs_per_channel);
    const int64_t f0 = (tile % P.runs_per_channel) * F;
    const int nf = (int)min((int64_t)F, P.n_use - f0);
    // ---- tile load: 8 rows per step; lane -> frame, one row per warp (256 B) ----
    {
      const int fr = lane, r0 = warp;
      const float2* g = P.Sx + ((size_t)ch * 257 + r0) * P.n_frames + f0 + fr;
      const size_t gstep = (size_t)8 * P.n_frames;
      float2* s = S + fr * AS + r0;
      const bool ok = fr < nf;
#pragma unroll 8
      for (int it = 0; it < 32; ++it) {  // (all 32 loads in flight at once measured slower: 11.05 vs 10.43 ms)
        s[8 * it] = ok ? __ldg(g) : make_float2(0.f, 0.f);
        g += gstep;
      }
      if (r0 == 0) s[256] = ok ? __ldg(g) : make_float2(0.f, 0.f);
    }
    __syncthreads();
    // ---- transforms: warp w owns frames 4w .. 4w+3 (two packed pairs) --------------------------------
    // hop == 32: sample lane + 32 j of frame f belongs to the 32-sample block f + j, lane `lane`: the warp
    // adds its (up to) four frames in a 16-register window and parks 19 finished blocks in its own first
    // two tile rows (their input has been consumed by then); the gather below then adds <= 5 warp partials
    // per sample instead of <= 16 frames.
    float out[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) out[j] = 0.f;
    float* wsum = reinterpret_cast<float*>(S + 4 * warp * AS) + lane;  // [19][32] floats (two rows hold 1156)
#pragma unroll 1
    for (int pr = 0; pr < 2; ++pr) {
      const int fa = 4 * warp + 2 * pr;
      if (fa >= nf) {
        if (!HOP32 || 4 * warp >= nf) break;
        // hop 32, second pair absent: its two blocks are just the running window
        wsum[(2 * pr) * 32] = out[0];
        wsum[(2 * pr + 1) * 32] = out[1];
#pragma unroll
        for (int j = 0; j < 14; ++j) out[j] = out[j + 2];
        out[14] = out[15] = 0.f;
        continue;
      }
      float2* tA = S + fa * AS;
      float2* tB = tA + AS;  // zero row when the frame does not exist
      float2 va[8], vb[8];
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        if (t < 4) {
          float2 a = tA[lane + 64 * t], b = tB[lane + 64 * t];
          if (t == 0 && L.l0) { a.y = 0.f; b.y = 0.f; }  // DC: imaginary part ignored (irfft)
          va[t] = make_float2(a.x - b.y, -(a.y + b.x));
          a = tA[lane + 32 + 64 * t];
          b = tB[lane + 32 + 64 * t];
          vb[t] = make_float2(a.x - b.y, -(a.y + b.x));
        } else {
          float2 a = tA[512 - 64 * t - lane], b = tB[512 - 64 * t - lane];
          if (t == 4 && L.l0) { a.y = 0.f; b.y = 0.f; }  // Nyquist
          va[t] = make_float2(a.x + b.y, a.y - b.x);
          a = tA[480 - 64 * t - lane];
          b = tB[480 - 64 * t - lane];
          vb[t] = make_float2(a.x + b.y, a.y - b.x);
        }
      }
      __syncwarp();  // both rows fully read before they are overwritten below
      h32_fft512(L, xch, va, vb);  // va[m] = X[lane + 64 m], vb[m] = X[lane + 32 + 64 m]
      if (HOP32) {
#pragma unroll
        for (int m = 0; m < 8; ++m) {
          out[2 * m] = fmaf(va[m].x, war[2 * m], out[2 * m]);
          out[2 * m + 1] = fmaf(vb[m].x, war[2 * m + 1], out[2 * m + 1]);
        }
        wsum[(2 * pr) * 32] = out[0];
#pragma unroll
        for (int j = 0; j < 15; ++j) out[j] = out[j + 1];
        out[15] = 0.f;
#pragma unroll
        for (int m = 0; m < 8; ++m) {  // frame B = -Im (a zero row when it does not exist)
          out[2 * m] = fmaf(-va[m].y, war[2 * m], out[2 * m]);
          out[2 * m + 1] = fmaf(-vb[m].y, war[2 * m + 1], out[2 * m + 1]);
        }
        wsum[(2 * pr + 1) * 32] = out[0];
#pragma unroll
        for (int j = 0; j < 15; ++j) out[j] = out[j + 1];
        out[15] = 0.f;
      } else {
        float* yA = reinterpret_cast<float*>(tA);
        float* yB = reinterpret_cast<float*>(tB);
#pragma unroll
        for (int m = 0; m < 8; ++m) {
          yA[lane + 64 * m] = va[m].x * war[2 * m];
          yA[lane + 32 + 64 * m] = vb[m].x * war[2 * m + 1];
          yB[lane + 64 * m] = -va[m].y * war[2 * m];
          yB[lane + 32 + 64 * m] = -vb[m].y * war[2 * m + 1];
        }
      }
      __syncwarp();
    }
    if (HOP32 && 4 * warp < nf) {  // blocks 4 .. 18 of the warp: the window after its fourth frame
#pragma unroll
      for (int j = 0; j < 15; ++j) wsum[(4 + j) * 32] = out[j];
    }
    __syncthreads();
    // ---- overlap-add gather over the tile span, one red per padded sample ---------------------------
    {
      const int hop = HOP32 ? 32 : P.hop;
      const int span = (nf - 1) * hop + N;
      float* xo = P.xacc + (size_t)ch * P.L + f0 * hop;
      const int64_t room = P.L - f0 * hop;
      const float* Sf = reinterpret_cast<const float*>(S);
      if (HOP32) {
        // sample p = 32 B + l of the tile: sum over warps w of wsum_w[B - 4 w][l] = Sf[p + w (4 * 2 AS - 128)]
        const int wlast = (nf - 1) >> 2;
        for (int p = threadIdx.x; p < span; p += blockDim.x) {
          const int B = p >> 5;
          const int whi = min(wlast, B >> 2);
          const int wlo = B < 19 ? 0 : (B - 15) >> 2;  // ceil((B - 18) / 4)
          float acc = 0.f;
          for (int w = wlo; w <= whi; ++w) acc += Sf[p + w * (8 * AS - 128)];
          if (p < room) atomicAdd(xo + p, acc);
        }
      } else {
        const float inv_hop = 1.f / (float)hop;
        const int step = 2 * AS - hop;
        for (int p = threadIdx.x; p < span; p += blockDim.x) {
          const int fhi = min(nf - 1, ssq_fast_div(p, hop, inv_hop));
          const int flo = p < N ? 0 : ssq_fast_div(p - N + hop, hop, inv_hop);  // ceil((p - N + 1) / hop)
          const float* src = Sf + flo * step + p;
          float acc = 0.f;
          for (int f = flo; f <= fhi; ++f) {
            acc += *src;
            src += step;
          }
          if (p < room && flo <= fhi) atomicAdd(xo + p, acc);
        }
      }
    }
    __syncthreads();
  }
}

static ssq_status istft512_launch(ssq_ctx* ctx, Istft32Params& Q, bool* done) {
  *done = false;
  // the tile span must stay inside the range of ssq_fast_div
  if (Q.n_fft != 512 || ctx->opt.no_h32r || (int64_t)31 * Q.hop + 512 >= ((int64_t)1 << 22)) return SSQ_OK;
  constexpr int NW = I32T_NW, F = 4 * NW;
  Q.run = F;
  Q.runs_per_channel = (Q.n_use + F - 1) / F;
  Q.total_runs = Q.runs_per_channel * Q.channels;
  *done = true;
  const size_t smem = ((size_t)72 + (size_t)F * I32T_AS + (size_t)NW * 512) * sizeof(float2);
  const int grid = (int)std::min<int64_t>(Q.total_runs, (int64_t)ctx->num_sms * (16 / NW));
  void (*k)(const Istft32Params) = Q.hop == 32 ? istft512_tile_kernel<true> : istft512_tile_kernel<false>;
  SSQ_CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<grid, NW * 32, smem, ctx->stream>>>(Q);
  SSQ_TRY(ssq_check_launch(ctx, "istft512_tile_kernel"));
  ctx->last_kernel = "istft512_tile_kernel";
  return SSQ_OK;
}
