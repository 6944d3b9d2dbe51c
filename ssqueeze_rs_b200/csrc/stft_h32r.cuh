// stft_h32r.cuh -- "rotated" variant of the n_fft = 512 kernel (hop = 32: sliding sample window, in tensor memory in
// the ssq mode; any other hop: per-frame reload): the item staging
// (transposition of the 257 (bin, value) items through shared memory: 48 wavefronts per
// frame on the binding L1TEX data pipe) is removed.
//
// The reassignment needs, in every step, 32 source bins that are far apart (>= 8 bins:
// neighbouring sources often map to the SAME destination bin and would collide).  After a
// plain stage 3 lane l holds Z[l + 64 m] in register m: in step m the warp would hold 32
// CONSECUTIVE bins.  Rotating the last butterfly fixes that for free:
//   va'[r] = Z[l + 64 ((r + rho) & 7)],  rho = l & 7:  fold W_8^{t rho} into the stage-3
//            twiddle, i.e. use W_512^{t (l + 64 rho)};
//   vb'[r] = Z[512 - (l + 64 ((r + rho) & 7))]: the partner butterfly j2 = 64 - l run with the
//            CONJUGATE kernel on twiddles W_512^{t (j2 + 64 (7 - rho))}  (out_b[(7 - rho - r) & 7]).
// Register pair r of lane l is then the conjugate pair (Z[k_a], Z[512 - k_a]),
// k_a = l + 64 ((r + rho) & 7): it yields the ONE source bin k = min(k_a, 512 - k_a); in step r
// lanes with equal rho are 8 bins apart and the others >= 33 apart (a few lane pairs 1-7).
// Swapping the roles of the pair only flips the signs of Im Sx and Re V, so the item is
// computed from (va'[r], vb'[r]) as is and the sign is carried by the signed source bin
// skf[r] = +-k:  |k - q| = |skf - q0|.  Lane 0 (butterflies j = 0 and 32, both self-paired)
// picks its pairs by static register indices.
// Accumulation order inside a bin is no longer ascending in k (rounding-level difference to
// the reference); it is fixed by the schedule, so results stay run-to-run identical.
#pragma once
#include "fft_regs.cuh"

#ifndef H32R_PK
#define H32R_PK(MODE) true  // packed fp32x2 arithmetic in the FFT, both modes (the stft mode spilled with it until the
                            // stage-3 twiddle table left the registers: 15.8 ms packed vs 16.6 ms scalar on 384 channels;
                            // packing its window multiply and split as well spills again: 16.9 ms)
#endif
#define H32R_AS 261  // column stride (float2): bin k at k + (k >> 6) (max 260); odd

__device__ __forceinline__ int h32r_phys(int k) { return k + (k >> 6); }

struct H32RItem {
  int kb;
  float vre, vim;
};

// Pair (A, B) = (Z[k_a], Z[512 - k_a]) -> item of source bin |skf|.  sign(skf) < 0: roles swapped.
// colB != nullptr (stft, hop 32): the FFT carried TWO frames, z = x_A w + i x_B w; the "V" half of the
// split is then the second frame's spectrum and goes to its own column.
// DBG: also emit Sx, dSx, w and the destination bin of this source bin (ssq_dbg_emit) -- the parity tests run the
// SAME kernel with one more store per item.
template <int MODE, int SQZ, bool DBG = false>
__device__ __forceinline__ H32RItem h32r_item(const StftParams& P, float txs, float2* col, float2* colB, float skf,
                                              float2 A, float2 B, size_t dbg_base = 0) {
  H32RItem it;
  const unsigned sgn = __float_as_uint(skf) & 0x80000000u;
  const float2 cd = add2<MODE == 0>(A, make_float2(B.x, -B.y));  // 2 Re Sx, +-2 Im Sx
  const float c = cd.x, d0 = cd.y;
  if (MODE == 1) {
    const int k = (int)fabsf(skf);
    col[h32r_phys(k)] = make_float2(0.5f * c, __uint_as_float(__float_as_uint(0.5f * d0) ^ sgn));
    if (colB) {
      const float2 ba = add2<MODE == 0>(B, make_float2(-A.x, A.y));
      const float b0 = ba.x, a = ba.y;
      colB[h32r_phys(k)] = make_float2(0.5f * a, __uint_as_float(__float_as_uint(0.5f * b0) ^ sgn));
    }
    it.kb = -1;
    it.vre = it.vim = 0.f;
    return it;
  }
  const float2 ba = add2<MODE == 0>(B, make_float2(-A.x, A.y));  // 2 V (Re with the swap sign)
  const float b0 = ba.x, a = ba.y;
  const float den = fmaf(c, c, d0 * d0);
  const float num0 = fmaf(b0, c, -a * d0);
  const float q0 = num0 * rcp_approx(den);
  const float binf = fabsf(fmaf(-q0, P.cphase, skf));
  // nearest grid point, ties to the lower index, clamped; NaN converts to 0 -> bin 0 like the reference
  it.kb = min(max(__float2int_ru(binf - 0.5f), 0), 256);
  if (DBG) {  // undo the role swap (Im Sx and Im V carry its sign) and apply the modulation sign
    const float ms = (txs < 0.f) != (P.tx_scale < 0.f) ? -1.f : 1.f;
    ssq_dbg_emit(P, dbg_base, (int)fabsf(skf), ms * c, ms * __uint_as_float(__float_as_uint(d0) ^ sgn), ms * a,
                 ms * __uint_as_float(__float_as_uint(b0) ^ sgn), binf, den < P.gate2, it.kb);
  }
  if (den < P.gate2) it.kb = -1;  // |Sx| < gamma (ssq_stft.rs:23): dropped
  if (SQZ == SSQ_SQUEEZE_LEBESGUE) {
    it.vre = P.leb_val;
    it.vim = 0.f;
  } else {
    it.vre = c * txs;
    it.vim = d0 * __uint_as_float(__float_as_uint(txs) ^ sgn);  // (sign folded into the factor: 10.68 vs 10.70 ms per 128 channels)
  }
  return it;
}

__device__ __noinline__ void h32r_collision(float2* col, unsigned* T, int kb, float vre, float vim, bool mine,
                                            int lane) {
  const bool on = kb >= 0;
  {  // tonal frames: every active lane aims at the same bin -> one shuffle reduction, one add
    const unsigned act = __ballot_sync(0xffffffffu, on);
    const int first = __ffs(act) - 1;
    const int kb0 = __shfl_sync(0xffffffffu, kb, first);
    if (__all_sync(0xffffffffu, !on || kb == kb0)) {
      float sr = on ? vre : 0.f, si = on ? vim : 0.f;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        sr += __shfl_xor_sync(0xffffffffu, sr, o);
        si += __shfl_xor_sync(0xffffffffu, si, o);
      }
      if (lane == first) smem_rmw_add(col + h32r_phys(kb0), sr, si);
      return;
    }
  }
  if (on && !mine) T[kb] = 0xFF;
  __syncwarp();
  const bool contended = on && T[kb] == 0xFF;
  if (on && !contended) smem_rmw_add(col + h32r_phys(kb), vre, vim);
  unsigned m = __ballot_sync(0xffffffffu, contended);
  if (__popc(m) > 4) {
    // many lanes on few bins (a tone over a noise floor: most of the warp aims at the tone's bin, the rest is
    // scattered): one shuffle reduction per bin instead of one lane at a time -- 10 shuffles whatever the size of the
    // group (a pure-tone input ran 4.4x slower than noise through the serial loop)
    while (m) {
      const int first = __ffs(m) - 1;
      const int kb0 = __shfl_sync(0xffffffffu, kb, first);
      const bool member = contended && kb == kb0;
      float sr = member ? vre : 0.f, si = member ? vim : 0.f;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        sr += __shfl_xor_sync(0xffffffffu, sr, o);
        si += __shfl_xor_sync(0xffffffffu, si, o);
      }
      if (lane == first) smem_rmw_add(col + h32r_phys(kb0), sr, si);
      m &= ~__ballot_sync(0xffffffffu, member);
    }
    __syncwarp();
    return;
  }
  while (m) {  // contended lanes one at a time, ascending lane order (deterministic)
    const int src = __ffs(m) - 1;
    m &= m - 1;
    if (lane == src) smem_rmw_add(col + h32r_phys(kb), vre, vim);
    __syncwarp();
  }
}

template <int MODE, int SQZ, bool DBG = false>
// skf0: signed source bin of step 0; wrapd: increment applied instead of +64 after the step whose
// source lies in [192, 256) (lanes >= 1: k_a jumps to the mirrored half, -448; lane 0: 192 -> 32).
// txs: dw/2, negated on odd lanes when `modulated` (Sx[k] (-1)^k: every source bin of lane l has l's parity)
__device__ __forceinline__ void h32r_frame(const StftParams& P, const H32Lane& L, float skf0, float wrapd, float txs,
                                           float2* xch, float2* col, float2* colB, float2 (&va)[8], float2 (&vb)[8],
                                           size_t dbg_base = 0) {
  const int lane = L.lane;
  const bool l0 = L.l0;
  // tags alias the exchange buffer; one 32-bit word per destination bin: with byte tags four bins share a bank
  // word and the lanes of a step, whose bins differ by multiples of 64, collided two ways (ncu r1r: 30
  // wavefronts per frame for an ideal 15)
  unsigned* tagA = reinterpret_cast<unsigned*>(xch);
  unsigned* tagB = tagA + 264;
  h32_fft512<true, true, H32R_PK(MODE)>(L, xch, va, vb);
  __syncwarp();  // stage-3 reads done before the tags overwrite the buffer

  // pair of step r: lanes >= 1 (va[r], vb[r]); lane 0: r < 4: (va[r], va[(8-r)&7]), r >= 4: (vb[11-r], vb[r-4])
#define H32R_PAIR(r, A, B)                                   \
  float2 A = va[r], B = vb[r];                               \
  if (l0) {                                                  \
    A = (r) < 4 ? va[r] : vb[(11 - (r)) & 7];                \
    B = (r) < 4 ? va[(8 - (r)) & 7] : vb[((r)-4) & 7];       \
  }

  H32RItem cur;
  float skf = skf0;
  {
    H32R_PAIR(0, A, B)
    cur = h32r_item<MODE, SQZ, DBG>(P, txs, col, colB, skf, A, B, dbg_base);
  }
  if (MODE == 0) {
    if (cur.kb >= 0) tagA[cur.kb] = (unsigned)lane;
    __syncwarp();
  }
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    H32RItem nxt;
    nxt.kb = -1;
    nxt.vre = nxt.vim = 0.f;
    if (r < 7) {  // next item's arithmetic overlaps this step's tag / accumulator latency
      skf += (skf >= 192.f) ? wrapd : 64.f;
      H32R_PAIR(r + 1, A, B)
      nxt = h32r_item<MODE, SQZ, DBG>(P, txs, col, colB, skf, A, B, dbg_base);
    }
    if (MODE == 0) {
      unsigned* T = (r & 1) ? tagB : tagA;
      unsigned* Tn = (r & 1) ? tagA : tagB;
      const bool on = cur.kb >= 0;
      // the accumulator is read together with the tag (speculatively: it is only used when no other lane aims at
      // the same bin in this step, and then nobody else writes it), so the two shared-memory latencies overlap
      float2* slot = col + h32r_phys(on ? cur.kb : 0);
      float2 t = *slot;
      const bool mine = !on || T[cur.kb] == (unsigned)lane;
      if (__all_sync(0xffffffffu, mine)) {
        if (on) {
          t.x += cur.vre;
          t.y += cur.vim;
          *slot = t;
        }
      } else {
        h32r_collision(col, T, cur.kb, cur.vre, cur.vim, mine, lane);
      }
      if (r < 7 && nxt.kb >= 0) Tn[nxt.kb] = (unsigned)lane;
      __syncwarp();
    }
    cur = nxt;
  }
#undef H32R_PAIR
  // bin 256 = Z[256] of lane 0 (va[4], self-paired): last, outside the protocol
  if (l0) {
    const H32RItem it = h32r_item<MODE, SQZ, DBG>(P, txs, col, colB, 256.f, va[4], va[4], dbg_base);
    if (MODE == 0 && it.kb >= 0) smem_rmw_add(col + h32r_phys(it.kb), it.vre, it.vim);
  }
  __syncwarp();  // the tag area is the exchange buffer of the next frame
}

// Edge tiles only (reflect / zero padding index map); kept out of line: the main loop has to fit the
// instruction cache (the fully inlined version was 88 KB of SASS, 7 % of the issue slots starved).
__device__ __noinline__ float h32r_edge_sample(const float* x, int64_t n, int64_t p, int left, int padtype,
                                               int64_t origin) {
  return stft_sample<false>(x, n, p, left, padtype, origin);
}

// Warps per CTA, 16 per SM either way.  4 for ssq_stft (16-frame tiles, 128 B row segments, 4 CTAs per SM: half the
// barrier domain of the 8-warp shape, which was 3.6 % slower); 8 for the faster stft mode, which writes at > 2.5 TB/s
// and needs the 256 B segments of 32-frame tiles at full scale (384 channels: 18.1 vs 26.5 ms).
#define H32R_NW(MODE) ((MODE) == 1 ? 8 : 4)

// Tensor memory (TMEM) of the ssq mode: warp w uses lane quarter w (lanes 32w..32w+31), one lane per thread.
// Columns 0..31 hold the lane's window taps, (w, dw*s) at positions lane + 32 j, j = 0..15, in column
// 4t + {0, 1, 2, 3} = (w, dw*s)[lane + 64 t], (w, dw*s)[lane + 32 + 64 t].  At hop 32, columns 32..50 hold the samples of
// the warp's tile: sample lane + 32 b of its first frame in column 32 + b, so frame s of the tile reads its 16 samples
// from columns 32 + s .. 47 + s.  Read by tcgen05.ld (LDTM), which does not go through the L1TEX data pipe that binds
// this kernel (profiles/README.md, round 3): 32 shared wavefronts per frame fewer than the shared tap table, and the
// 16-register sample window is no longer live across the FFT and the reassignment.

__device__ __forceinline__ void h32r_tmem_st32(uint32_t taddr, const float (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,"
      "%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};\n\t"
      "tcgen05.wait::st.sync.aligned;" ::"r"(taddr),
      "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "f"(v[8]), "f"(v[9]),
      "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15]), "f"(v[16]), "f"(v[17]), "f"(v[18]),
      "f"(v[19]), "f"(v[20]), "f"(v[21]), "f"(v[22]), "f"(v[23]), "f"(v[24]), "f"(v[25]), "f"(v[26]), "f"(v[27]),
      "f"(v[28]), "f"(v[29]), "f"(v[30]), "f"(v[31]));
}

__device__ __forceinline__ void h32r_tmem_st16(uint32_t taddr, const float (&v)[17]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "f"(v[8]), "f"(v[9]),
      "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15]));
}

__device__ __forceinline__ void h32r_tmem_st1(uint32_t taddr, float v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr), "f"(v));
}

// the frame's 16 samples and the 32 taps: waits for this thread's earlier sample stores, loads, waits for the loads
__device__ __forceinline__ void h32r_tmem_ld_window(uint32_t taddr_x, uint32_t taddr_w, float (&x)[16], float (&v)[32]) {
  asm volatile(
      "tcgen05.wait::st.sync.aligned;\n\t"
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%48];\n\t"
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32,%33,"
      "%34,%35,%36,%37,%38,%39,%40,%41,%42,%43,%44,%45,%46,%47}, [%49];\n\t"
      "tcgen05.wait::ld.sync.aligned;"
      : "=f"(x[0]), "=f"(x[1]), "=f"(x[2]), "=f"(x[3]), "=f"(x[4]), "=f"(x[5]), "=f"(x[6]), "=f"(x[7]), "=f"(x[8]),
        "=f"(x[9]), "=f"(x[10]), "=f"(x[11]), "=f"(x[12]), "=f"(x[13]), "=f"(x[14]), "=f"(x[15]),
        "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]), "=f"(v[8]),
        "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15]), "=f"(v[16]),
        "=f"(v[17]), "=f"(v[18]), "=f"(v[19]), "=f"(v[20]), "=f"(v[21]), "=f"(v[22]), "=f"(v[23]), "=f"(v[24]),
        "=f"(v[25]), "=f"(v[26]), "=f"(v[27]), "=f"(v[28]), "=f"(v[29]), "=f"(v[30]), "=f"(v[31])
      : "r"(taddr_x), "r"(taddr_w));
}

// load and wait in one statement: the values exist for the compiler only once the wait is done
__device__ __forceinline__ void h32r_tmem_ld32(uint32_t taddr, float (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,"
      "%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];\n\t"
      "tcgen05.wait::ld.sync.aligned;"
      : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]), "=f"(v[8]),
        "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15]), "=f"(v[16]),
        "=f"(v[17]), "=f"(v[18]), "=f"(v[19]), "=f"(v[20]), "=f"(v[21]), "=f"(v[22]), "=f"(v[23]), "=f"(v[24]),
        "=f"(v[25]), "=f"(v[26]), "=f"(v[27]), "=f"(v[28]), "=f"(v[29]), "=f"(v[30]), "=f"(v[31])
      : "r"(taddr));
}

// SLIDE: hop == 32, the sliding window (one new sample per lane and frame; in TMEM in the ssq mode, in registers in the
// stft mode).  Otherwise any hop:
// the 16 samples of every frame are (re)loaded, still a whole frame ahead of their use.
template <int MODE, int SQZ, bool SLIDE, bool DBG = false>
__global__ void __launch_bounds__(H32R_NW(MODE) * 32, 16 / H32R_NW(MODE)) ssq_stft512_h32r_kernel(const StftParams P) {
  constexpr int N = 512, AS = H32R_AS, NW = H32R_NW(MODE), F = 4 * NW;
  // stft at hop 32: two frames per FFT (z = x_A w + i x_B w; frame B's samples are frame A's window
  // shifted by one position), so a warp runs 2 FFTs for its 4 frames
  constexpr bool PAIR = (MODE == 1) && SLIDE;
  // the window taps: a shared table in the stft mode, tensor memory in the ssq mode; at hop 32 the ssq mode's sample
  // window too (RING)
  constexpr bool TM = MODE == 0;
  constexpr bool RING = TM && SLIDE;
  constexpr int TMC = RING ? 64 : 32;  // TMEM columns per CTA
  constexpr int WT = TM ? 0 : N;
  extern __shared__ float2 smem[];
  __shared__ uint32_t tmem_base_s;
  float2* wtab = smem;           // [WT] (w, dw*s)
  float2* tw2tab = smem + WT;    // [8][9]
  float2* acc = smem + WT + 72;  // [32][AS] the tile's Tx columns
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float2* xch = acc + F * AS + warp * N;  // WT + 72 + F * 261 float2 is even (F = 16, 32): the float4 exchange rows stay 16 B aligned

  if (TM && warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     (uint32_t)__cvta_generic_to_shared(&tmem_base_s)),
                 "n"(TMC));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (!TM)
    for (int i = threadIdx.x; i < N; i += blockDim.x) wtab[i] = make_float2(P.win[i], P.dwin[i]);
  if (threadIdx.x < 64)
    tw2tab[(threadIdx.x >> 3) * 9 + (threadIdx.x & 7)] = P.tw[((threadIdx.x >> 3) * (threadIdx.x & 7) * 8) & (N - 1)];
  for (int i = threadIdx.x; i < F * AS; i += blockDim.x) acc[i] = make_float2(0.f, 0.f);

  // ---- per-lane constants ----------------------------------------------------------
  H32Lane L;
  L.lane = lane;
  L.j2 = lane ? 64 - lane : 32;
  L.tw2 = tw2tab + (lane & 7) * 9;
  const int rho = lane & 7;
  const int ea = lane + 64 * rho;  // va: W_512^{t (l + 64 rho)}; vb uses the conjugates (h32_fft512<true>)
#pragma unroll
  for (int t = 1; t < 8; ++t) {
    L.tw3a[t - 1] = P.tw[(ea * t) & (N - 1)];
    L.tw3b[t - 1] = make_float2(0.f, 0.f);  // unused
  }
  L.f1 = (lane >> 1) & 3;
  L.rd1a = (lane >> 3) * 8 + ((((lane & 7) >> 1) ^ ((lane >> 4) & 3)) << 1) + (lane & 1);
  L.rd1b = ((lane >> 3) + 4) * 8 + ((((lane & 7) >> 1) ^ (((lane >> 4) + 2) & 3)) << 1) + (lane & 1);
  L.g2 = (lane >> 3) & 1;
  L.wr2 = (lane >> 3) * 64 + (lane & 7);
  L.lane_f = (float)lane;
  L.j2_f = (float)L.j2;
  L.l0 = (lane == 0);
  const float txs = (P.modulated && (lane & 1)) ? -P.tx_scale : P.tx_scale;
  // signed source bin of step r: skf_0, then +64 per step except once (see h32r_frame)
  float skf0, wrapd;
  if (lane == 0) {
    skf0 = 0.f;
    wrapd = -160.f;
  } else {
    const int ka = lane + 64 * rho;
    skf0 = rho <= 3 ? (float)ka : (float)(ka - 512);
    wrapd = -448.f;
  }
  if (TM) asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  uint32_t taps = 0;  // this warp's lane quarter of the CTA's TMEM columns (column 0)
  if (TM) {
    asm volatile("tcgen05.fence::after_thread_sync;");
    taps = tmem_base_s + ((uint32_t)(warp * 32) << 16);
    float v[32];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      v[4 * t] = P.win[lane + 64 * t];
      v[4 * t + 1] = P.dwin[lane + 64 * t];
      v[4 * t + 2] = P.win[lane + 32 + 64 * t];
      v[4 * t + 3] = P.dwin[lane + 32 + 64 * t];
    }
    h32r_tmem_st32(taps, v);  // waits for the store: the frames below load from it
  }

  // ---- the warp's frames of a tile: [f0, f0 + nfr), nfr in 0..4 ------------------------------
  const float* xc = nullptr;
  int64_t f0 = 0;
  int nfr = 0;
  bool inner = false;
  float xw[17];  // [16] is only used by PAIR
  const int64_t lo = P.left + P.x_origin;  // padded position p of an interior sample lives at x[p - lo]
  // tile indices are 32-bit (checked by the launcher): 64-bit divisions cost ~100 instructions each
  const int tpc = (int)P.tiles_per_channel, ntiles = (int)P.total_tiles;
  auto open_tile = [&](int tile) {  // single call site (see the loop): sets the warp's frames, loads frame f0's window
    const int ch = tile / tpc;
    f0 = (int64_t)(tile - ch * tpc) * F + 4 * warp;
    nfr = (int)max((int64_t)0, min((int64_t)4, P.n_frames - f0));
    f0 += P.frame0;  // from here on f0 is the GLOBAL frame index (sample addressing only)
    xc = P.x + (size_t)ch * P.x_stride;
    const int64_t hop = SLIDE ? 32 : P.hop;
    inner = f0 * hop - P.left >= 0 && (f0 + 3) * hop + N - 1 - P.left + (PAIR ? 32 : 0) < P.n;
    if (nfr > 0) {
      const int64_t p = f0 * hop + lane;
      if (inner) {
#pragma unroll
        for (int j = 0; j < (PAIR ? 17 : 16); ++j) xw[j] = __ldg(xc + (p + 32 * j - lo));
      } else {
#pragma unroll
        for (int j = 0; j < (PAIR ? 17 : 16); ++j) xw[j] = h32r_edge_sample(xc, P.n, p + 32 * j, P.left, P.padtype, P.x_origin);
      }
    }
  };

  // The loop starts one (virtual) tile early so that open_tile is inlined exactly once: the first
  // pass only fetches the window of the CTA's first real tile.
  for (int tile = (int)blockIdx.x - (int)gridDim.x; tile < ntiles; tile += (int)gridDim.x) {
    const bool real = tile >= 0;
    const int tch = real ? tile / tpc : 0;
    const int64_t tf0 = real ? (int64_t)(tile - tch * tpc) * F : 0;
    const int tnf = real ? (int)min((int64_t)F, P.n_frames - tf0) : 0;
    const int next = tile + (int)gridDim.x;
    const int my_n = real ? nfr : 0;
    if (RING && real) h32r_tmem_st16(taps + 32, xw);  // the tile's window, loaded during the previous tile's store
#pragma unroll 1
    for (int s = 0; s < 4; s += (PAIR ? 2 : 1)) {
      const bool active = s < my_n;
      float2 va[8], vb[8];
      float xn = 0.f;  // RING: the sample this lane adds for frame s + 1
      if (active) {
        float tv[TM ? 32 : 1];
        float xs[RING ? 16 : 1];
        if constexpr (RING)
          h32r_tmem_ld_window(taps + 32 + s, taps, xs, tv);
        else if constexpr (TM)
          h32r_tmem_ld32(taps, tv);
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          float2 w0, w1;
          if constexpr (TM) {
            w0 = make_float2(tv[4 * t], tv[4 * t + 1]);
            w1 = make_float2(tv[4 * t + 2], tv[4 * t + 3]);
          } else {
            w0 = wtab[lane + 64 * t];
            w1 = wtab[lane + 32 + 64 * t];
          }
          if (PAIR) {  // real part frame s, imaginary part frame s+1 (same window, samples one position on)
            va[t] = mul2<false>(make_float2(xw[2 * t], xw[2 * t + 1]), bc2(w0.x));
            vb[t] = mul2<false>(make_float2(xw[2 * t + 1], xw[2 * t + 2]), bc2(w1.x));
          } else if constexpr (RING) {
            va[t] = mul2(bc2(xs[2 * t]), w0);
            vb[t] = mul2(bc2(xs[2 * t + 1]), w1);
          } else {
            va[t] = mul2(bc2(xw[2 * t]), w0);
            vb[t] = mul2(bc2(xw[2 * t + 1]), w1);
          }
        }
      }
      if (s == (PAIR ? 2 : 3)) {
        if (!RING && next < ntiles) open_tile(next);
      } else if (s + (PAIR ? 2 : 1) < my_n) {
        if (PAIR) {
#pragma unroll
          for (int j = 0; j < 15; ++j) xw[j] = xw[j + 2];
          const int64_t p = (f0 + s + 2) * 32 + lane + 480;
          if (inner) {
            xw[15] = __ldg(xc + (p - lo));
            xw[16] = __ldg(xc + (p + 32 - lo));
          } else {
            xw[15] = h32r_edge_sample(xc, P.n, p, P.left, P.padtype, P.x_origin);
            xw[16] = h32r_edge_sample(xc, P.n, p + 32, P.left, P.padtype, P.x_origin);
          }
        } else if (RING) {  // a frame ahead of its use; to TMEM after this frame's FFT
          const int64_t p = (f0 + s + 1) * 32 + lane + 480;
          xn = inner ? __ldg(xc + (p - lo)) : h32r_edge_sample(xc, P.n, p, P.left, P.padtype, P.x_origin);
        } else if (SLIDE) {
#pragma unroll
          for (int j = 0; j < 15; ++j) xw[j] = xw[j + 1];
          const int64_t p = (f0 + s + 1) * 32 + lane + 480;
          xw[15] = inner ? __ldg(xc + (p - lo)) : h32r_edge_sample(xc, P.n, p, P.left, P.padtype, P.x_origin);
        } else {
          const int64_t p = (f0 + s + 1) * (int64_t)P.hop + lane;
          if (inner) {
#pragma unroll
            for (int j = 0; j < 16; ++j) xw[j] = __ldg(xc + (p + 32 * j - lo));
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) xw[j] = h32r_edge_sample(xc, P.n, p + 32 * j, P.left, P.padtype, P.x_origin);
          }
        }
      }
      if (active)
        h32r_frame<MODE, SQZ, DBG>(P, L, skf0, wrapd, txs, xch, acc + (4 * warp + s) * AS,
                                   PAIR ? acc + (4 * warp + s + 1) * AS : nullptr, va, vb,
                                   DBG ? (size_t)tch * 257 * P.n_frames + tf0 + 4 * warp + s : 0);
      if (RING && s + 1 < my_n) h32r_tmem_st1(taps + 48 + s, xn);
    }
    // RING: the next tile's window is fetched here, so that the loads are in flight during the tile store below
    if (RING && next < ntiles) open_tile(next);
    if (!real) continue;
    __syncthreads();
    // ---- coalesced store: thread -> (frame fr, row group v in 0..7); rows k = v + 8 i live at
    //      physical k + (k >> 6) = v + 8 i + (i >> 3) = v + 65 io + 8 ii  (i = 8 io + ii)
    {
      const int fr = threadIdx.x % F, v = threadIdx.x / F;
      float2* a = acc + fr * AS + v;
      float2* g = P.out + ((size_t)tch * 257 + v) * P.n_frames + tf0 + fr;
      const size_t gstep = (size_t)8 * P.n_frames;
      const bool ok = fr < tnf;
#pragma unroll 1
      for (int io = 0; io < 4; ++io) {
#pragma unroll
        for (int ii = 0; ii < 8; ++ii) {
          const float2 val = a[8 * ii];
          if (MODE == 0) a[8 * ii] = make_float2(0.f, 0.f);
          if (ok) __stcs(g, val);
          g += gstep;
        }
        a += 65;
      }
      if (v == 0) {  // row 256 at physical 260 (a has advanced by 4 * 65)
        const float2 val = a[0];
        if (MODE == 0) a[0] = make_float2(0.f, 0.f);
        if (ok) __stcs(g, val);
      }
    }
    __syncthreads();
  }
  if (TM) {  // every warp's last TMEM load is done before the allocating warp frees the columns
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
    if (warp == 0)
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base_s), "n"(TMC));
  }
}

static ssq_status stft_h32r_launch(ssq_ctx* ctx, StftParams& P, bool* done) {
  *done = false;
  if (P.n_fft != 512 || ctx->opt.no_h32r) return SSQ_OK;
  const int NW = H32R_NW(P.mode), F = 4 * NW;
  P.F = F;
  P.acc_stride = H32R_AS;
  P.tiles_per_channel = (P.n_frames + F - 1) / F;
  P.total_tiles = P.tiles_per_channel * P.channels;
  if (P.total_tiles > (int64_t)0x7ff00000) return SSQ_OK;  // *done stays false: the older kernels index in 64 bits
  *done = true;
  const size_t wt = P.mode == 1 ? 512 : 0;  // the ssq mode keeps its window taps in tensor memory
  const size_t smem = (wt + 72 + (size_t)F * H32R_AS + (size_t)NW * 512) * sizeof(float2);
  const int grid = (int)std::min<int64_t>(P.total_tiles, (int64_t)ctx->num_sms * (16 / NW));
  const bool leb = P.squeezing == SSQ_SQUEEZE_LEBESGUE;
  void (*k)(const StftParams);
  const bool dbg = P.mode == 0 && (P.aux_Sx || P.aux_dSx || P.aux_w || P.aux_kb);
  if (dbg)  // the same kernel with the diagnostic stores compiled in (parity tests)
    k = P.hop == 32 ? (leb ? ssq_stft512_h32r_kernel<0, 1, true, true> : ssq_stft512_h32r_kernel<0, 0, true, true>)
                    : (leb ? ssq_stft512_h32r_kernel<0, 1, false, true> : ssq_stft512_h32r_kernel<0, 0, false, true>);
  else if (P.hop == 32)
    k = P.mode == 1 ? ssq_stft512_h32r_kernel<1, 0, true>
        : leb       ? ssq_stft512_h32r_kernel<0, 1, true>
                    : ssq_stft512_h32r_kernel<0, 0, true>;
  else
    k = P.mode == 1 ? ssq_stft512_h32r_kernel<1, 0, false>
        : leb       ? ssq_stft512_h32r_kernel<0, 1, false>
                    : ssq_stft512_h32r_kernel<0, 0, false>;
  SSQ_CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<grid, NW * 32, smem, ctx->stream>>>(P);
  const char* name = P.mode == 1 ? "ssq_stft512_h32r_kernel<stft>" : "ssq_stft512_h32r_kernel<ssq>";
  SSQ_TRY(ssq_check_launch(ctx, name));
  ctx->last_kernel = name;
  return SSQ_OK;
}
