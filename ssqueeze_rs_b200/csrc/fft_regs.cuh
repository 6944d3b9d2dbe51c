// fft_regs.cuh -- register-resident FFT building blocks shared by the n_fft = 256 / 512 / 1024 kernels
// (forward and inverse): radix-8 butterflies on packed fp32x2 arithmetic and the 512-point transform of one
// frame per warp (512 = 8 x 8 x 8, 16 complex points per lane, two XOR-swizzled 4 KB exchanges through
// shared memory; every shared-memory access of the transform is bank-conflict free and all per-access
// address arithmetic folds into immediates).
//
//   stage 1  j in {l, l+32}:  in  z[j+64t] (windowed samples), out idx 8j+t              (exchange 1)
//   stage 2  j in {l, l+32}:  in  idx j+64t, times W_64^{(j&7) t}, out idx (j>>3)*64 + (j&7) + 8t  (exchange 2)
//   stage 3  j in {l, 64-l} (lane 0: {0, 32}): in idx j+64t, times W_512^{j t}: X[j+64t] stays in registers;
//            bins k and 512-k needed by the real/imag split sit in the SAME lane.
#pragma once
#include "stft_kernels.cuh"

template <bool PK = true>
__device__ __forceinline__ void fft8_fwd(float2 (&v)[8]) {
  const float S = 0.70710678118654752440f;
  float2 a0 = caddf<PK>(v[0], v[4]), a4 = csubf<PK>(v[0], v[4]);
  float2 a1 = caddf<PK>(v[1], v[5]), a5 = csubf<PK>(v[1], v[5]);
  float2 a2 = caddf<PK>(v[2], v[6]), a6 = csubf<PK>(v[2], v[6]);
  float2 a3 = caddf<PK>(v[3], v[7]), a7 = csubf<PK>(v[3], v[7]);
  // odd branch twiddles W8^1, W8^2, W8^3 (the 1/sqrt2 factors are folded into the last layer)
  float2 p5 = caddf<PK>(a5, cmi(a5));  // a5 * (1 - i)      [* S]
  float2 p6 = cmi(a6);             // a6 * (-i)
  float2 p7 = csubf<PK>(cmi(a7), a7);  // a7 * (-1 - i)     [* S]
  float2 b0 = caddf<PK>(a0, a2), b2 = csubf<PK>(a0, a2);
  float2 b1 = caddf<PK>(a1, a3), b3 = csubf<PK>(a1, a3);
  float2 b4 = caddf<PK>(a4, p6), b6 = csubf<PK>(a4, p6);
  float2 b5 = caddf<PK>(p5, p7), b7 = csubf<PK>(p5, p7);  // both still lack the factor S
  float2 r3 = cmi(b3);                            // -i * b3
  float2 r7 = cmi(b7);                            // -i * b7
  v[0] = caddf<PK>(b0, b1);
  v[4] = csubf<PK>(b0, b1);
  v[2] = caddf<PK>(b2, r3);
  v[6] = csubf<PK>(b2, r3);
  v[1] = fma2<PK>(b5, bc2(S), b4);
  v[5] = fma2<PK>(b5, bc2(-S), b4);
  v[3] = fma2<PK>(r7, bc2(S), b6);
  v[7] = fma2<PK>(r7, bc2(-S), b6);
}

// Same butterfly with the conjugate kernel: v[m] <- sum_t v[t] W_8^{-t m}.
template <bool PK = true>
__device__ __forceinline__ void fft8_inv(float2 (&v)[8]) {
  const float S = 0.70710678118654752440f;
  float2 a0 = caddf<PK>(v[0], v[4]), a4 = csubf<PK>(v[0], v[4]);
  float2 a1 = caddf<PK>(v[1], v[5]), a5 = csubf<PK>(v[1], v[5]);
  float2 a2 = caddf<PK>(v[2], v[6]), a6 = csubf<PK>(v[2], v[6]);
  float2 a3 = caddf<PK>(v[3], v[7]), a7 = csubf<PK>(v[3], v[7]);
  float2 p5 = caddf<PK>(a5, cpi(a5));  // a5 * (1 + i)      [* S]
  float2 p6 = cpi(a6);             // a6 * (+i)
  float2 p7 = csubf<PK>(cpi(a7), a7);  // a7 * (-1 + i)     [* S]
  float2 b0 = caddf<PK>(a0, a2), b2 = csubf<PK>(a0, a2);
  float2 b1 = caddf<PK>(a1, a3), b3 = csubf<PK>(a1, a3);
  float2 b4 = caddf<PK>(a4, p6), b6 = csubf<PK>(a4, p6);
  float2 b5 = caddf<PK>(p5, p7), b7 = csubf<PK>(p5, p7);
  float2 r3 = cpi(b3);  // +i * b3
  float2 r7 = cpi(b7);  // +i * b7
  v[0] = caddf<PK>(b0, b1);
  v[4] = csubf<PK>(b0, b1);
  v[2] = caddf<PK>(b2, r3);
  v[6] = csubf<PK>(b2, r3);
  v[1] = fma2<PK>(b5, bc2(S), b4);
  v[5] = fma2<PK>(b5, bc2(-S), b4);
  v[3] = fma2<PK>(r7, bc2(S), b6);
  v[7] = fma2<PK>(r7, bc2(-S), b6);
}

__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

__device__ __forceinline__ void smem_rmw_add(float2* p, float re, float im) {
  float2 t = *p;
  t.x += re;
  t.y += im;
  *p = t;
}

// Per-lane constants of the 512-point transform.
struct H32Lane {
  int lane, j2, f1, rd1a, rd1b, g2, wr2;
  float lane_f, j2_f;
  bool l0;
  const float2* tw2;
  float2 tw3a[7], tw3b[7];
};

// 512-point forward DFT of one frame: inputs va[t] = z[lane + 64 t], vb[t] = z[lane + 32 + 64 t];
// outputs va[m] = Z[lane + 64 m], vb[m] = Z[L.j2 + 64 m].  Two swizzled exchanges through xch.
// ROT: the last butterfly of vb uses the conjugate kernel (see stft_h32r.cuh).
// TW2POW: stage-2 twiddles by powers of one table entry (saves 12 shared-memory wavefronts, costs 24
// multiplies: a gain where the data pipe binds -- stft/ssq_stft -- and a loss for istft).
template <bool ROT = false, bool TW2POW = ROT, bool PK = true>
__device__ __forceinline__ void h32_fft512(const H32Lane& L, float2* xch, float2 (&va)[8], float2 (&vb)[8]) {
  const int lane = L.lane, j2 = L.j2;
  fft8_fwd<PK>(va);
  fft8_fwd<PK>(vb);
  {
    float4* rowa = reinterpret_cast<float4*>(xch + lane * 8);
    float4* rowb = reinterpret_cast<float4*>(xch + (lane + 32) * 8);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      rowa[q ^ L.f1] = make_float4(va[2 * q].x, va[2 * q].y, va[2 * q + 1].x, va[2 * q + 1].y);
      rowb[q ^ L.f1] = make_float4(vb[2 * q].x, vb[2 * q].y, vb[2 * q + 1].x, vb[2 * q + 1].y);
    }
  }
  __syncwarp();
  // ---- stage 2 ---------------------------------------------------------------------------
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    va[t] = xch[L.rd1a + 64 * t];
    vb[t] = xch[L.rd1b + 64 * t];
  }
  __syncwarp();
  {
    float2 w[8];
    w[1] = L.tw2[1];  // W_64^{r t}, r = lane & 7
    if (TW2POW) {     // the other powers by products at most 3 deep
      w[2] = cmulf<PK>(w[1], w[1]);
      w[3] = cmulf<PK>(w[2], w[1]);
      w[4] = cmulf<PK>(w[2], w[2]);
      w[5] = cmulf<PK>(w[4], w[1]);
      w[6] = cmulf<PK>(w[4], w[2]);
      w[7] = cmulf<PK>(w[4], w[3]);
    } else {
#pragma unroll
      for (int t = 2; t < 8; ++t) w[t] = L.tw2[t];
    }
#pragma unroll
    for (int t = 1; t < 8; ++t) {
      va[t] = cmulf<PK>(va[t], w[t]);
      vb[t] = cmulf<PK>(vb[t], w[t]);
    }
  }
  fft8_fwd<PK>(va);
  fft8_fwd<PK>(vb);
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    xch[L.wr2 + 8 * (t ^ L.g2)] = va[t];
    xch[L.wr2 + 256 + 8 * (t ^ L.g2)] = vb[t];
  }
  __syncwarp();
  // ---- stage 3 ---------------------------------------------------------------------------
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    va[t] = xch[(lane ^ (8 * (t & 1))) + 64 * t];
    vb[t] = xch[(j2 ^ (8 * (t & 1))) + 64 * t];
  }
  __syncwarp();
  if (ROT) {
    // rotated variant (stft_h32r.cuh): the partner butterfly's twiddles are the conjugates of tw3a
    // (W^{t (512 - e_a)}), except for lane 0 whose partner is j = 32: W^{480 t} = conj(W_16^t)
    const float C1 = 0.92387953251128673848f, S1 = 0.38268343236508978178f, H = 0.70710678118654752440f;
    const float2 w16[7] = {{C1, -S1}, {H, -H}, {S1, -C1}, {0.f, -1.f}, {-S1, -C1}, {-H, -H}, {-C1, -S1}};
    // stage-3 twiddles W^{t e_a} as powers of the first (at most 3 products deep): 12 registers of table
    // traded for 6 complex multiplications -- the kernel is bound by latency, not by issue slots
    float2 w3[7];
    w3[0] = L.tw3a[0];
    w3[1] = cmulf<PK>(w3[0], w3[0]);
    w3[2] = cmulf<PK>(w3[1], w3[0]);
    w3[3] = cmulf<PK>(w3[1], w3[1]);
    w3[4] = cmulf<PK>(w3[3], w3[0]);
    w3[5] = cmulf<PK>(w3[3], w3[1]);
    w3[6] = cmulf<PK>(w3[3], w3[2]);
#pragma unroll
    for (int t = 1; t < 8; ++t) {
      const float2 wa = w3[t - 1];
      va[t] = cmulf<PK>(va[t], wa);
      const float2 wb = L.l0 ? w16[t - 1] : wa;
      vb[t] = cmulcf<PK>(vb[t], wb);  // vb * conj(wb)
    }
    fft8_fwd<PK>(va);
    fft8_inv<PK>(vb);
    return;
  }
#pragma unroll
  for (int t = 1; t < 8; ++t) {
    va[t] = cmulf<PK>(va[t], L.tw3a[t - 1]);
    vb[t] = cmulf<PK>(vb[t], L.tw3b[t - 1]);
  }
  fft8_fwd<PK>(va);  // va[m] = Z[lane + 64 m]
  fft8_fwd<PK>(vb);  // vb[m] = Z[j2 + 64 m]
}
