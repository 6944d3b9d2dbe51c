// stft_r1024.cuh -- fused ssq_stft / stft for n_fft = 1024, any hop: the geometry of the reference's own
// multichannel script (tests/stft_ssq_test.py:166-167, 308-309: n_fft = 1024, hop_length = 256).
//
// Same scheme as the n_fft = 512 kernel (stft_h32r.cuh) -- a warp owns a frame, the FFT lives in
// registers, the Tx column is accumulated in a shared-memory tile that leaves as row segments --
// with the decomposition 1024 = 32 x 32: a lane holds the 32 samples n = lane + 32 t, runs a 32-point DFT
// over t in registers (4 x radix-8, constant twiddles, 8 x radix-4), ONE transposition through shared
// memory (8.4 KB per warp, conflict-free both ways with a row stride of 33), the twiddles W_1024^{n1 q}
// as powers of one table entry, and a second 32-point DFT: lane q ends with Z[q + 32 m], m = 0..31.
// Z[1024 - k] of the lane's bins k = q + 32 m (m < 16) sits in lane (32 - q) & 31, register 31 - m: one
// shuffle per value.  The 513 (value, destination bin) items are parked in the exchange buffer by source
// bin and re-read with a lane stride of 17 bins so that the 32 sources of a reassignment step are far
// apart (neighbouring sources often share a destination); the step itself is the tag-checked plain
// read-modify-write of the other kernels.
#pragma once
#include "stft_h32r.cuh"

#define R1K_AS 514  // column stride of the Tx tile (float2), >= 513.  The read-out's half-warp covers 8 frames x 2 row
                    // groups: banks (2 AS fr + 2 v) mod 32 must be distinct -> 2 AS = 4 mod 32 (515 gave 2-way conflicts:
                    // 128 instead of 64 wavefronts per frame, ncu r1t)
#define R1K_XS 33   // exchange row stride (float2)
#define R1K_WS 1300 // per-warp scratch (float2): max(32 * 33 exchange, 520 item values + 260 (520 keys) + 520 (2 x 520 tag words))

__host__ __device__ constexpr float r1k_q(int j) {  // cos(pi j / 16), j = 0..8
  constexpr float q[9] = {1.f,
                          0.98078528040323044f,
                          0.92387953251128676f,
                          0.83146961230254524f,
                          0.70710678118654752f,
                          0.55557023301960222f,
                          0.38268343236508977f,
                          0.19509032201612827f,
                          0.f};
  return q[j];
}
__host__ __device__ constexpr float r1k_cos32(int j) {  // cos(2 pi j / 32), j = 0..31
  return j <= 8 ? r1k_q(j) : j <= 16 ? -r1k_q(16 - j) : j <= 24 ? -r1k_q(j - 16) : r1k_q(32 - j);
}
__host__ __device__ constexpr float r1k_sin32(int j) {
  return j <= 8 ? r1k_q(8 - j) : j <= 16 ? r1k_q(j - 8) : j <= 24 ? -r1k_q(24 - j) : -r1k_q(j - 24);
}

template <bool PK>
__device__ __forceinline__ void r1k_fft4(float2& a, float2& b, float2& c, float2& d) {
  const float2 apc = caddf<PK>(a, c), amc = csubf<PK>(a, c), bpd = caddf<PK>(b, d), bmd = csubf<PK>(b, d);
  a = caddf<PK>(apc, bpd);
  b = caddf<PK>(amc, cmi(bmd));  // amc - i bmd
  c = csubf<PK>(apc, bpd);
  d = caddf<PK>(amc, cpi(bmd));  // amc + i bmd
}

// register holding output m of r1k_fft32
#define R1K_REG(m) (4 * ((m) & 7) + ((m) >> 3))

// 32-point forward DFT in registers.  in: v[t], t = 0..31; out: v[R1K_REG(m)] = sum_t v[t] W_32^{t m}.
template <bool PK>
__device__ __forceinline__ void r1k_fft32(float2 (&v)[32]) {
  // t = t0 + 4 t1: 8-point DFTs over t1 -> v[t0 + 4 k1]
#pragma unroll
  for (int t0 = 0; t0 < 4; ++t0) {
    float2 a[8];
#pragma unroll
    for (int t1 = 0; t1 < 8; ++t1) a[t1] = v[t0 + 4 * t1];
    fft8_fwd<PK>(a);
#pragma unroll
    for (int k1 = 0; k1 < 8; ++k1) v[t0 + 4 * k1] = a[k1];
  }
  // twiddles W_32^{t0 k1}
#pragma unroll
  for (int t0 = 1; t0 < 4; ++t0) {
#pragma unroll
    for (int k1 = 1; k1 < 8; ++k1) {
      const float2 w = make_float2(r1k_cos32((t0 * k1) & 31), -r1k_sin32((t0 * k1) & 31));
      v[t0 + 4 * k1] = cmulf<PK>(v[t0 + 4 * k1], w);
    }
  }
  // 4-point DFTs over t0: X[k1 + 8 k0] -> v[4 k1 + k0]
#pragma unroll
  for (int k1 = 0; k1 < 8; ++k1) r1k_fft4<PK>(v[4 * k1], v[4 * k1 + 1], v[4 * k1 + 2], v[4 * k1 + 3]);
}

struct R1KItem {
  int kb;
  float vre, vim;
};

// A = Z[k], B = Z[1024 - k] -> item of source bin k (kf = (float)k).
template <int MODE, int SQZ, int KMAX = 512, bool DBG = false>
__device__ __forceinline__ R1KItem r1k_item(const StftParams& P, float txs, float2* col, float2* colB, int k,
                                            float kf, float2 A, float2 B, size_t dbg_base = 0) {
  R1KItem it;
  const float c = A.x + B.x, d = A.y - B.y;  // 2 Sx
  if (MODE == 1) {
    col[k] = make_float2(0.5f * c, 0.5f * d);
    if (colB) colB[k] = make_float2(0.5f * (A.y + B.y), 0.5f * (B.x - A.x));  // second frame of the packed pair
    it.kb = -1;
    it.vre = it.vim = 0.f;
    return it;
  }
  const float a = A.y + B.y, b = B.x - A.x;  // 2 V
  const float den = fmaf(c, c, d * d);
  const float num = fmaf(b, c, -a * d);
  const float q = num * rcp_approx(den);
  const float binf = fabsf(fmaf(-q, P.cphase, kf));
  // nearest grid point, ties to the lower index, clamped; NaN converts to 0 -> bin 0 like the reference
  it.kb = min(max(__float2int_ru(binf - 0.5f), 0), KMAX);
  if (DBG) {  // diagnostic stores of the parity tests (with the modulation sign)
    const float ms = (txs < 0.f) != (P.tx_scale < 0.f) ? -1.f : 1.f;
    ssq_dbg_emit(P, dbg_base, k, ms * c, ms * d, ms * a, ms * b, binf, den < P.gate2, it.kb);
  }
  if (den < P.gate2) it.kb = -1;  // |Sx| < gamma (ssq_stft.rs:23): dropped
  if (SQZ == SSQ_SQUEEZE_LEBESGUE) {
    it.vre = P.leb_val;
    it.vim = 0.f;
  } else {
    it.vre = c * txs;
    it.vim = d * txs;
  }
  return it;
}

// Rare path of a reassignment step (two lanes aim at one bin): see h32r_collision.
__device__ __noinline__ void r1k_collision(float2* col, unsigned* T, int kb, float vre, float vim, bool mine,
                                           int lane) {
  const bool on = kb >= 0;
  {
    const unsigned act = __ballot_sync(0xffffffffu, on);
    const int first = __ffs(act) - 1;
    const int kb0 = __shfl_sync(0xffffffffu, kb, first);
    if (__all_sync(0xffffffffu, !on || kb == kb0)) {  // tonal frame: one reduction, one add
      float sr = on ? vre : 0.f, si = on ? vim : 0.f;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        sr += __shfl_xor_sync(0xffffffffu, sr, o);
        si += __shfl_xor_sync(0xffffffffu, si, o);
      }
      if (lane == first) smem_rmw_add(col + kb0, sr, si);
      return;
    }
  }
  if (on && !mine) T[kb] = 0xFF;
  __syncwarp();
  const bool contended = on && T[kb] == 0xFF;
  if (on && !contended) smem_rmw_add(col + kb, vre, vim);
  unsigned m = __ballot_sync(0xffffffffu, contended);
  while (m) {  // ascending lane = ascending source bin (ssq_stft.rs:277-298)
    const int src = __ffs(m) - 1;
    m &= m - 1;
    if (lane == src) smem_rmw_add(col + kb, vre, vim);
    __syncwarp();
  }
}


#define R1K_NW 4  // warps per CTA
#define R1K_F 8   // frames per tile (F / NW per warp)

template <int MODE, int SQZ, bool DBG = false>
__global__ void __launch_bounds__(R1K_NW * 32, 3) ssq_stft1024_kernel(const StftParams P) {
  constexpr int N = 1024, AS = R1K_AS, XS = R1K_XS, NW = R1K_NW, F = R1K_F, FPW = F / NW;
  constexpr bool PK = true;
  static_assert(F % NW == 0 && (F / NW) % 2 == 0, "frames per warp: even (stft mode packs pairs)");
  extern __shared__ float2 smem[];
  float2* acc = smem;  // [F][AS]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float2* xch = acc + F * AS + warp * R1K_WS;
  // after the second DFT the exchange buffer holds the parked items and the tags
  float2* sval = xch;                                            // [513] (520)
  int* skey = reinterpret_cast<int*>(xch + 520);                 // [513] (520 ints = 260 float2)
  unsigned* tagA = reinterpret_cast<unsigned*>(xch + 780);       // [513] (520 words = 260 float2): one word per
  unsigned* tagB = tagA + 520;                                   // bin, so that no two bins share a bank word

  for (int i = threadIdx.x; i < F * AS; i += blockDim.x) acc[i] = make_float2(0.f, 0.f);
  const bool l0 = lane == 0;
  const int partner = (32 - lane) & 31;
  const float2 w1 = P.tw[lane];  // W_1024^{lane}
  const float txs = (P.modulated && (lane & 1)) ? -P.tx_scale : P.tx_scale;  // Sx[k] (-1)^k, k = lane + 32 m
  const int64_t lo = P.left + P.x_origin;
  const int tpc = (int)P.tiles_per_channel, ntiles = (int)P.total_tiles;
  __syncthreads();

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int ch = tile / tpc;
    const int64_t tf0 = (int64_t)(tile - ch * tpc) * F;
    const int nf = (int)min((int64_t)F, P.n_frames - tf0);
    const float* xc = P.x + (size_t)ch * P.x_stride;
    // stft mode: two frames per FFT (z = x_A w + i x_B w; the "V" half of the split is frame B's spectrum)
    constexpr int STEP = (MODE == 1) ? 2 : 1;
#pragma unroll 1
    for (int s = 0; s < FPW; s += STEP) {
      const int fl = warp * FPW + s;
      if (fl >= nf) break;
      float2* col = acc + fl * AS;
      float2* colB = (MODE == 1 && fl + 1 < nf) ? col + AS : nullptr;
      const size_t dbg_base = DBG ? (size_t)ch * 513 * P.n_frames + tf0 + fl : 0;
      float2 v[32];
      {
        const int64_t p0 = (P.frame0 + tf0 + fl) * (int64_t)P.hop + lane;  // padded position of t = 0
        float xs[32];
        if (p0 - lane - P.left >= 0 && p0 - lane + N - 1 - P.left < P.n) {
          const float* xp = xc + (p0 - lo);
#pragma unroll
          for (int t = 0; t < 32; ++t) xs[t] = __ldg(xp + 32 * t);
        } else {
#pragma unroll
          for (int t = 0; t < 32; ++t) xs[t] = h32r_edge_sample(xc, P.n, p0 + 32 * t, P.left, P.padtype, P.x_origin);
        }
        if (MODE == 1) {
          float xb[32];
          const int64_t p1 = p0 + P.hop;
          if (!colB) {
#pragma unroll
            for (int t = 0; t < 32; ++t) xb[t] = 0.f;
          } else if (p1 - lane - P.left >= 0 && p1 - lane + N - 1 - P.left < P.n) {
            const float* xp = xc + (p1 - lo);
#pragma unroll
            for (int t = 0; t < 32; ++t) xb[t] = __ldg(xp + 32 * t);
          } else {
#pragma unroll
            for (int t = 0; t < 32; ++t) xb[t] = h32r_edge_sample(xc, P.n, p1 + 32 * t, P.left, P.padtype, P.x_origin);
          }
#pragma unroll
          for (int t = 0; t < 32; ++t) v[t] = mul2<PK>(make_float2(xs[t], xb[t]), bc2(__ldg(P.win + lane + 32 * t)));
        } else {
#pragma unroll
          for (int t = 0; t < 32; ++t) v[t] = mul2<PK>(bc2(xs[t]), __ldg(P.wpair + lane + 32 * t));
        }
      }
      r1k_fft32<PK>(v);  // v[R1K_REG(kappa)] = Y[lane][kappa]
#pragma unroll
      for (int kp = 0; kp < 32; ++kp) xch[lane * XS + kp] = v[R1K_REG(kp)];
      __syncwarp();
#pragma unroll
      for (int n1 = 0; n1 < 32; ++n1) v[n1] = xch[n1 * XS + lane];
      __syncwarp();
      {
        // W_1024^{n1 lane}, n1 = 4 i + j: (w^4)^i w^j
        const float2 q2 = cmulf<PK>(w1, w1), q3 = cmulf<PK>(q2, w1), w4 = cmulf<PK>(q2, q2);
        v[1] = cmulf<PK>(v[1], w1);
        v[2] = cmulf<PK>(v[2], q2);
        v[3] = cmulf<PK>(v[3], q3);
        float2 b = w4;
#pragma unroll
        for (int i = 1; i < 8; ++i) {
          v[4 * i] = cmulf<PK>(v[4 * i], b);
          v[4 * i + 1] = cmulf<PK>(v[4 * i + 1], cmulf<PK>(b, w1));
          v[4 * i + 2] = cmulf<PK>(v[4 * i + 2], cmulf<PK>(b, q2));
          v[4 * i + 3] = cmulf<PK>(v[4 * i + 3], cmulf<PK>(b, q3));
          if (i < 7) b = cmulf<PK>(b, w4);
        }
      }
      r1k_fft32<PK>(v);  // v[R1K_REG(m)] = Z[lane + 32 m]
      // ---- split + phase transform: source bins k = lane + 32 m, m = 0..15 (and 512 on lane 0) ----
#pragma unroll
      for (int m = 0; m < 16; ++m) {
        const float2 A = v[R1K_REG(m)];
        const float2 Bs = v[R1K_REG(31 - m)];
        float2 B = make_float2(__shfl_sync(0xffffffffu, Bs.x, partner), __shfl_sync(0xffffffffu, Bs.y, partner));
        if (l0) B = v[R1K_REG((32 - m) & 31)];  // lane 0 pairs with itself: Z[1024 - 32 m]
        const int k = lane + 32 * m;
        const R1KItem it = r1k_item<MODE, SQZ, 512, DBG>(P, txs, col, colB, k, (float)k, A, B, dbg_base);
        if (MODE == 0) {
          sval[k] = make_float2(it.vre, it.vim);
          skey[k] = it.kb;
        }
      }
      if (l0) {
        const R1KItem it = r1k_item<MODE, SQZ, 512, DBG>(P, txs, col, colB, 512, 512.f, v[R1K_REG(16)], v[R1K_REG(16)], dbg_base);
        if (MODE == 0) {
          sval[512] = make_float2(it.vre, it.vim);
          skey[512] = it.kb;
        }
      }
      __syncwarp();
      if (MODE == 0) {
        // ---- reassignment: lane owns source bins 17 lane + i; one __syncwarp per step ----
        const int kbase = 17 * lane;
        R1KItem cur;
        cur.kb = -1;
        cur.vre = cur.vim = 0.f;
        if (kbase <= 512) {
          const float2 sv = sval[kbase];
          cur.kb = skey[kbase];
          cur.vre = sv.x;
          cur.vim = sv.y;
        }
        if (cur.kb >= 0) tagA[cur.kb] = (unsigned)lane;
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 17; ++i) {
          R1KItem nxt;
          nxt.kb = -1;
          nxt.vre = nxt.vim = 0.f;
          if (i < 16 && kbase + i + 1 <= 512) {
            const float2 sv = sval[kbase + i + 1];
            nxt.kb = skey[kbase + i + 1];
            nxt.vre = sv.x;
            nxt.vim = sv.y;
          }
          unsigned* T = (i & 1) ? tagB : tagA;
          unsigned* Tn = (i & 1) ? tagA : tagB;
          const bool on = cur.kb >= 0;
          float2* slot = col + (on ? cur.kb : 0);  // read with the tag: the two shared-memory latencies overlap
          float2 t = *slot;
          const bool mine = !on || T[cur.kb] == (unsigned)lane;
          if (__all_sync(0xffffffffu, mine)) {
            if (on) {
              t.x += cur.vre;
              t.y += cur.vim;
              *slot = t;
            }
          } else {
            r1k_collision(col, T, cur.kb, cur.vre, cur.vim, mine, lane);
          }
          if (i < 16 && nxt.kb >= 0) Tn[nxt.kb] = (unsigned)lane;
          __syncwarp();
          cur = nxt;
        }
      }
      __syncwarp();  // items / tags live in the exchange buffer of the next frame
    }
    __syncthreads();
    // ---- coalesced store: thread -> (frame fr, row group v); rows v + RG i ----
    {
      constexpr int RG = NW * 32 / F;
      const int fr = threadIdx.x % F, vv = threadIdx.x / F;
      float2* a = acc + fr * AS + vv;
      float2* g = P.out + ((size_t)ch * 513 + vv) * P.n_frames + tf0 + fr;
      const size_t gstep = (size_t)RG * P.n_frames;
      const bool ok = fr < nf;
#pragma unroll 4
      for (int i = 0; i < 512 / RG; ++i) {
        const float2 val = a[RG * i];
        if (MODE == 0) a[RG * i] = make_float2(0.f, 0.f);
        if (ok) __stcs(g, val);
        g += gstep;
      }
      if (vv == 0) {  // row 512
        const float2 val = a[512];
        if (MODE == 0) a[512] = make_float2(0.f, 0.f);
        if (ok) __stcs(g, val);
      }
    }
    __syncthreads();
  }
}

static ssq_status stft_r1024_launch(ssq_ctx* ctx, StftParams& P, bool* done) {
  *done = false;
  if (P.n_fft != 1024 || ctx->opt.no_r1024) return SSQ_OK;
  constexpr int NW = R1K_NW, F = R1K_F;
  StftParams Q = P;
  Q.F = F;
  Q.acc_stride = R1K_AS;
  Q.tiles_per_channel = (P.n_frames + F - 1) / F;
  Q.total_tiles = Q.tiles_per_channel * P.channels;
  if (Q.total_tiles > (int64_t)0x7ff00000) return SSQ_OK;
  *done = true;
  const size_t smem = ((size_t)F * R1K_AS + (size_t)NW * R1K_WS) * sizeof(float2);
  const int grid = (int)std::min<int64_t>(Q.total_tiles, (int64_t)ctx->num_sms * 3);
  const bool leb = P.squeezing == SSQ_SQUEEZE_LEBESGUE;
  const bool dbg = P.mode == 0 && (P.aux_Sx || P.aux_dSx || P.aux_w || P.aux_kb);
  void (*k)(const StftParams) = P.mode == 1 ? ssq_stft1024_kernel<1, 0>
                                : dbg       ? (leb ? ssq_stft1024_kernel<0, 1, true> : ssq_stft1024_kernel<0, 0, true>)
                                : leb       ? ssq_stft1024_kernel<0, 1>
                                            : ssq_stft1024_kernel<0, 0>;
  SSQ_CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<grid, NW * 32, smem, ctx->stream>>>(Q);
  const char* name = P.mode == 1 ? "ssq_stft1024_kernel<stft>" : "ssq_stft1024_kernel<ssq>";
  SSQ_TRY(ssq_check_launch(ctx, name));
  ctx->last_kernel = name;
  P.F = F;
  return SSQ_OK;
}
