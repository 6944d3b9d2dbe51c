// stft_r256.cuh -- fused ssq_stft / stft for n_fft = 256, any hop: the geometry of the reference's README
// and smoke scripts (tests/stft_test.py:137-151, tests/stft_ssq_test.py:137-138: n_fft = 256, hop 64).
//
// The pieces of the n_fft = 1024 kernel (stft_r1024.cuh) with the decomposition 256 = 8 x 32 and FOUR frames
// per warp: lane = (g, c), g = lane >> 3 the frame of the group, c = lane & 7.  A lane holds the 32 samples
// n = c + 8 t of its frame, runs the 32-point DFT over t in registers, the 8 lanes of a group transpose
// through shared memory (lane c keeps kappa = c + 8 j, j = 0..3, for all 8 n1), twiddles W_256^{n1 kappa}
// = (W_256^c)^{n1} W_32^{j n1}, four radix-8 DFTs over n1: lane (g, c) ends with Z_g[c + 8 j + 32 m].
// Z[256 - k] of its bins (m < 4) sits in lane (g, (8 - c) & 7), register (3 - j, 7 - m): one shuffle per
// value (c = 0 pairs with itself).  Items are parked by source bin per frame and re-read with a lane
// stride of 17 bins; the reassignment step is the tag-checked read-modify-write of the other kernels, the
// four frames of a warp going to four different columns of the tile.
#pragma once
#include "stft_r1024.cuh"

#define R256_AS 145  // column stride of the Tx tile (float2); frame f's column starts at f * 145 + 8 (f & 1).
                     // 145 = 1 mod 16 and the 8-slot stagger of odd frames put the two frames of a half-warp
                     // (bins 17 c + i each) on disjoint banks in the reassignment step (stride 131: 55 wavefronts
                     // per frame for an ideal 17, ncu r1v) and keep the read-out (16 frames x one row) conflict-free
#define R256_WS 1088 // per-warp scratch (float2): max(32 * 33 exchange, 544 item values + 272 keys + 272 (16-bit tags))
#define R256_SS 136  // per-frame stride of the parked items / tags (>= 8 * 17)

// Rare path of a reassignment step; the four groups of a warp work on different columns.
__device__ __noinline__ void r256_collision(float2* col, unsigned short* T, int kb, float vre, float vim, bool mine,
                                            int lane) {
  const bool on = kb >= 0;
  {
    // tonal frames: every active lane of a GROUP aims at the same bin -> one reduction, one add per group
    const unsigned act = __ballot_sync(0xffffffffu, on);
    const unsigned gact = act & (0xffu << (lane & 24));
    const int first = gact ? __ffs(gact) - 1 : (lane & 24);
    const int kb0 = __shfl_sync(0xffffffffu, kb, first);
    if (__all_sync(0xffffffffu, !on || kb == kb0)) {
      float sr = on ? vre : 0.f, si = on ? vim : 0.f;
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) {
        sr += __shfl_xor_sync(0xffffffffu, sr, o);
        si += __shfl_xor_sync(0xffffffffu, si, o);
      }
      if (gact && lane == first) smem_rmw_add(col + kb0, sr, si);
      return;
    }
  }
  if (on && !mine) T[kb] = 0xFFFF;
  __syncwarp();
  const bool contended = on && T[kb] == 0xFFFF;
  if (on && !contended) smem_rmw_add(col + kb, vre, vim);
  unsigned m = __ballot_sync(0xffffffffu, contended);
  while (m) {  // ascending lane = ascending source bin within a frame
    const int src = __ffs(m) - 1;
    m &= m - 1;
    if (lane == src) smem_rmw_add(col + kb, vre, vim);
    __syncwarp();
  }
}

#define R256_NW 4  // warps per CTA

// F frames per tile (groups of four per warp).
template <int MODE, int SQZ, int F, bool DBG = false>
__global__ void __launch_bounds__(R256_NW * 32, MODE == 0 ? 4 : 3) ssq_stft256_kernel(const StftParams P) {
  constexpr int N = 256, AS = R256_AS, XS = R1K_XS, SS = R256_SS, NW = R256_NW, GPW = F / (4 * NW);
  constexpr bool PK = true;
  static_assert(F % (4 * NW) == 0, "a warp takes its frames four at a time");
  // stft mode: two groups per FFT (z = x_A w + i x_B w, frame B = frame A + 4)
  constexpr int STEP = (MODE == 1) ? 2 : 1;
  static_assert(GPW % STEP == 0, "stft mode packs pairs of groups");
  extern __shared__ float2 smem[];
  float2* acc = smem;  // [F][AS]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 3, c = lane & 7;
  float2* xch = acc + F * AS + warp * R256_WS;
  // after the second stage the exchange buffer holds the parked items and the tags, per frame g
  float2* sval = xch + g * SS;                                                    // [4][136]
  int* skey = reinterpret_cast<int*>(xch + 4 * SS) + g * SS;                      // [4][136]
  unsigned short* tagA = reinterpret_cast<unsigned short*>(xch + 6 * SS) + g * SS;  // [4][136], 16-bit: two bins per
  unsigned short* tagB = tagA + 4 * SS;                                              // bank word instead of four

  for (int i = threadIdx.x; i < F * AS; i += blockDim.x) acc[i] = make_float2(0.f, 0.f);
  const bool c0 = c == 0;
  const int partner = (lane & 24) | ((8 - c) & 7);
  const float2 wb = P.tw[c];  // W_256^c
  const float txs = (P.modulated && (c & 1)) ? -P.tx_scale : P.tx_scale;  // Sx[k] (-1)^k: k has c's parity
  const int64_t lo = P.left + P.x_origin;
  const int tpc = (int)P.tiles_per_channel, ntiles = (int)P.total_tiles;
  __syncthreads();

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int ch = tile / tpc;
    const int64_t tf0 = (int64_t)(tile - ch * tpc) * F;
    const int nf = (int)min((int64_t)F, P.n_frames - tf0);
    const float* xc = P.x + (size_t)ch * P.x_stride;
#pragma unroll 1
    for (int s = 0; s < GPW; s += STEP) {
      const int fl0 = (warp * GPW + s) * 4;
      if (fl0 >= nf) break;
      const int fl = fl0 + g;
      const bool live = fl < nf;  // frames past the end compute on zeros; their columns are never stored
      float2* col = acc + fl * AS + 8 * (fl & 1);
      float2* colB = (MODE == 1) ? col + 4 * AS : nullptr;  // (a column past nf is written but never stored)
      const size_t dbg_base = DBG ? (size_t)ch * 129 * P.n_frames + tf0 + fl : 0;
      float2 v[32];
      {
        const int64_t p0 = (P.frame0 + tf0 + fl) * (int64_t)P.hop + c;  // padded position of t = 0
        float xs[32];
        if (!live) {
#pragma unroll
          for (int t = 0; t < 32; ++t) xs[t] = 0.f;
        } else if (p0 - c - P.left >= 0 && p0 - c + N - 1 - P.left < P.n) {
          const float* xp = xc + (p0 - lo);
#pragma unroll
          for (int t = 0; t < 32; ++t) xs[t] = __ldg(xp + 8 * t);
        } else {
#pragma unroll
          for (int t = 0; t < 32; ++t) xs[t] = h32r_edge_sample(xc, P.n, p0 + 8 * t, P.left, P.padtype, P.x_origin);
        }
        if (MODE == 1) {
          float xb[32];
          const int64_t p1 = p0 + 4 * (int64_t)P.hop;
          if (fl + 4 >= nf) {
#pragma unroll
            for (int t = 0; t < 32; ++t) xb[t] = 0.f;
          } else if (p1 - c - P.left >= 0 && p1 - c + N - 1 - P.left < P.n) {
            const float* xp = xc + (p1 - lo);
#pragma unroll
            for (int t = 0; t < 32; ++t) xb[t] = __ldg(xp + 8 * t);
          } else {
#pragma unroll
            for (int t = 0; t < 32; ++t) xb[t] = h32r_edge_sample(xc, P.n, p1 + 8 * t, P.left, P.padtype, P.x_origin);
          }
#pragma unroll
          for (int t = 0; t < 32; ++t) v[t] = mul2<PK>(make_float2(xs[t], xb[t]), bc2(__ldg(P.win + c + 8 * t)));
        } else {
#pragma unroll
          for (int t = 0; t < 32; ++t) v[t] = mul2<PK>(bc2(xs[t]), __ldg(P.wpair + c + 8 * t));
        }
      }
      r1k_fft32<PK>(v);  // v[R1K_REG(kappa)] = Y_g[c][kappa]
#pragma unroll
      for (int kp = 0; kp < 32; ++kp) xch[lane * XS + kp] = v[R1K_REG(kp)];
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 4; ++j) {
#pragma unroll
        for (int n1 = 0; n1 < 8; ++n1) v[8 * j + n1] = xch[((lane & 24) + n1) * XS + c + 8 * j];
      }
      __syncwarp();
      {
        // W_256^{n1 (c + 8 j)} = (W_256^c)^{n1} W_32^{j n1}
        float2 pw[8];
        pw[1] = wb;
        pw[2] = cmulf<PK>(wb, wb);
        pw[3] = cmulf<PK>(pw[2], wb);
        pw[4] = cmulf<PK>(pw[2], pw[2]);
        pw[5] = cmulf<PK>(pw[4], wb);
        pw[6] = cmulf<PK>(pw[4], pw[2]);
        pw[7] = cmulf<PK>(pw[4], pw[3]);
#pragma unroll
        for (int n1 = 1; n1 < 8; ++n1) {
          v[n1] = cmulf<PK>(v[n1], pw[n1]);
#pragma unroll
          for (int j = 1; j < 4; ++j) {
            const float2 w = make_float2(r1k_cos32((j * n1) & 31), -r1k_sin32((j * n1) & 31));
            v[8 * j + n1] = cmulf<PK>(v[8 * j + n1], cmulf<PK>(pw[n1], w));
          }
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float2 a[8];
#pragma unroll
        for (int n1 = 0; n1 < 8; ++n1) a[n1] = v[8 * j + n1];
        fft8_fwd<PK>(a);
#pragma unroll
        for (int m = 0; m < 8; ++m) v[8 * j + m] = a[m];  // Z_g[c + 8 j + 32 m]
      }
      // ---- split + phase transform: source bins k = c + 8 j + 32 m, m = 0..3 (and 128 on c = 0) ----
#pragma unroll
      for (int j = 0; j < 4; ++j) {
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          const float2 A = v[8 * j + m];
          const float2 Bs = v[8 * (3 - j) + 7 - m];
          float2 B = make_float2(__shfl_sync(0xffffffffu, Bs.x, partner), __shfl_sync(0xffffffffu, Bs.y, partner));
          if (c0) B = j ? v[8 * (4 - j) + 7 - m] : v[(8 - m) & 7];  // c = 0 pairs with itself
          const int k = c + 8 * j + 32 * m;
          const R1KItem it = (DBG && live) ? r1k_item<MODE, SQZ, 128, true>(P, txs, col, colB, k, (float)k, A, B, dbg_base)
                                           : r1k_item<MODE, SQZ, 128>(P, txs, col, colB, k, (float)k, A, B);
          if (MODE == 0) {
            sval[k] = make_float2(it.vre, it.vim);
            skey[k] = it.kb;
          }
        }
      }
      if (c0) {
        const R1KItem it = (DBG && live) ? r1k_item<MODE, SQZ, 128, true>(P, txs, col, colB, 128, 128.f, v[4], v[4], dbg_base)
                                         : r1k_item<MODE, SQZ, 128>(P, txs, col, colB, 128, 128.f, v[4], v[4]);
        if (MODE == 0) {
          sval[128] = make_float2(it.vre, it.vim);
          skey[128] = it.kb;
        }
      }
      __syncwarp();
      if (MODE == 0) {
        // ---- reassignment: lane (g, c) owns source bins 17 c + i of frame g; one __syncwarp per step ----
        const int kbase = 17 * c;
        R1KItem cur;
        cur.kb = -1;
        cur.vre = cur.vim = 0.f;
        {
          const float2 sv = sval[kbase];  // kbase <= 119
          cur.kb = skey[kbase];
          cur.vre = sv.x;
          cur.vim = sv.y;
        }
        if (cur.kb >= 0) tagA[cur.kb] = (unsigned short)lane;
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 17; ++i) {
          R1KItem nxt;
          nxt.kb = -1;
          nxt.vre = nxt.vim = 0.f;
          if (i < 16 && kbase + i + 1 <= 128) {
            const float2 sv = sval[kbase + i + 1];
            nxt.kb = skey[kbase + i + 1];
            nxt.vre = sv.x;
            nxt.vim = sv.y;
          }
          unsigned short* T = (i & 1) ? tagB : tagA;
          unsigned short* Tn = (i & 1) ? tagA : tagB;
          const bool on = cur.kb >= 0;
          float2* slot = col + (on ? cur.kb : 0);  // read with the tag: the two shared-memory latencies overlap
          float2 t = *slot;
          const bool mine = !on || T[cur.kb] == (unsigned short)lane;
          if (__all_sync(0xffffffffu, mine)) {
            if (on) {
              t.x += cur.vre;
              t.y += cur.vim;
              *slot = t;
            }
          } else {
            r256_collision(col, T, cur.kb, cur.vre, cur.vim, mine, lane);
          }
          if (i < 16 && nxt.kb >= 0) Tn[nxt.kb] = (unsigned short)lane;
          __syncwarp();
          cur = nxt;
        }
      }
      __syncwarp();  // items / tags live in the exchange buffer of the next group
    }
    __syncthreads();
    // ---- coalesced store: thread -> (frame fr, row group v); rows v + RG i ----
    {
      constexpr int RG = NW * 32 / F;
      const int fr = threadIdx.x % F, vv = threadIdx.x / F;
      float2* a = acc + fr * AS + 8 * (fr & 1) + vv;
      float2* gp = P.out + ((size_t)ch * 129 + vv) * P.n_frames + tf0 + fr;
      const size_t gstep = (size_t)RG * P.n_frames;
      const bool ok = fr < nf;
#pragma unroll 4
      for (int i = 0; i < 128 / RG; ++i) {
        const float2 val = a[RG * i];
        if (MODE == 0) a[RG * i] = make_float2(0.f, 0.f);
        if (ok) __stcs(gp, val);
        gp += gstep;
      }
      if (vv == 0) {  // row 128
        const float2 val = a[128];
        if (MODE == 0) a[128] = make_float2(0.f, 0.f);
        if (ok) __stcs(gp, val);
      }
    }
    __syncthreads();
  }
}

template <int F>
static ssq_status stft_r256_launch_f(ssq_ctx* ctx, StftParams& P, bool* done) {
  constexpr int NW = R256_NW;
  StftParams Q = P;
  Q.F = F;
  Q.acc_stride = R256_AS;
  Q.tiles_per_channel = (P.n_frames + F - 1) / F;
  Q.total_tiles = Q.tiles_per_channel * P.channels;
  if (Q.total_tiles > (int64_t)0x7ff00000) return SSQ_OK;
  *done = true;
  const size_t smem = ((size_t)F * R256_AS + (size_t)NW * R256_WS) * sizeof(float2);
  const int grid = (int)std::min<int64_t>(Q.total_tiles, (int64_t)ctx->num_sms * (F == 32 ? 3 : 4));
  const bool leb = P.squeezing == SSQ_SQUEEZE_LEBESGUE;
  void (*k)(const StftParams);
  if constexpr (F == 32) k = ssq_stft256_kernel<1, 0, F>;
  else if (P.aux_Sx || P.aux_dSx || P.aux_w || P.aux_kb)
    k = leb ? ssq_stft256_kernel<0, 1, F, true> : ssq_stft256_kernel<0, 0, F, true>;
  else k = leb ? ssq_stft256_kernel<0, 1, F> : ssq_stft256_kernel<0, 0, F>;
  SSQ_CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<grid, NW * 32, smem, ctx->stream>>>(Q);
  const char* name = P.mode == 1 ? "ssq_stft256_kernel<stft>" : "ssq_stft256_kernel<ssq>";
  SSQ_TRY(ssq_check_launch(ctx, name));
  ctx->last_kernel = name;
  P.F = F;
  return SSQ_OK;
}

static ssq_status stft_r256_launch(ssq_ctx* ctx, StftParams& P, bool* done) {
  *done = false;
  if (P.n_fft != 256 || ctx->opt.no_r256) return SSQ_OK;
  // ssq: 16-frame tiles (one group of four frames per warp); stft: 32-frame tiles, two groups per FFT
  return P.mode == 1 ? stft_r256_launch_f<32>(ctx, P, done) : stft_r256_launch_f<16>(ctx, P, done);
}
