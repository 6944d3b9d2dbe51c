// istft_r1024.cuh -- inverse STFT for n_fft = 1024, any hop (the geometry of the reference's multichannel script,
// tests/stft_ssq_test.py:166-167).  old/ssqueezepy/_stft.py:184-256 in the Rust framing, as istft_h32.cuh:
// a CTA owns a tile of 8 consecutive frames, loads the [513 x 8] tile transposed (frame-major rows), every warp
// turns one packed pair of frames (Z = Z_A + i Z_B with the Hermitian extension, x_A = Re, x_B = Im of the inverse
// transform) with the in-register 32 x 32 decomposition of stft_r1024.cuh (inverse = conj(forward(conj))), parks
// the windowed samples in the frames' own rows, and the overlap-add is a gather over the tile span with one
// red.global.add per padded sample; istft_finalize_kernel divides by the window norm and unpads.
#pragma once
#include "istft_h32.cuh"
#include "stft_r1024.cuh"

#define I1K_AS 514  // tile row stride (float2): 2 AS = 4 mod 32 -> the transposed load (8 frames x 4 rows per warp step) is
                    // bank-conflict free; 1028 floats >= 1024 samples

#define I1K_NW 4    // warps per CTA; F = 2 NW frames per tile

__global__ void __launch_bounds__(I1K_NW * 32, 3) istft1024_tile_kernel(const Istft32Params P) {
  constexpr int N = 1024, AS = I1K_AS, XS = R1K_XS, NW = I1K_NW, F = 2 * NW;
  constexpr bool PK = true;
  static_assert(NW == 4, "the load mapping below assumes 4 warps x 8 frames");
  extern __shared__ float2 smem[];
  float2* S = smem;  // [F][AS]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float2* xch = S + F * AS + warp * (32 * XS);
  const float2 w1 = P.tw[lane];  // W_1024^{lane}
  const int tpc = (int)P.runs_per_channel, ntiles = (int)P.total_runs;

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int ch = tile / tpc;
    const int64_t f0 = (int64_t)(tile - ch * tpc) * F;
    const int nf = (int)min((int64_t)F, P.n_use - f0);
    // ---- tile load: lane -> frame (lane & 7) and row lane >> 3; warp w, step it -> rows 4 w + sub + 16 it ----
    {
      const int fr = lane & 7, r0 = 4 * warp + (lane >> 3);
      const bool ok = fr < nf;
      const float2* g = P.Sx + ((size_t)ch * 513 + r0) * P.n_frames + f0 + fr;
      const size_t gstep = (size_t)16 * P.n_frames;
      float2* s = S + fr * AS + r0;
#pragma unroll 8
      for (int it = 0; it < 32; ++it) {
        s[16 * it] = ok ? __ldg(g) : make_float2(0.f, 0.f);
        g += gstep;
      }
      if (r0 == 0) s[512] = ok ? __ldg(g) : make_float2(0.f, 0.f);
    }
    __syncthreads();
    // ---- transform: warp w owns the packed pair of frames 2w, 2w + 1 ----
    const int fa = 2 * warp;
    if (fa < nf) {
      float2* tA = S + fa * AS;
      float2* tB = tA + AS;  // a zero row when the frame does not exist
      float2 v[32];
#pragma unroll
      for (int t = 0; t < 32; ++t) {
        // conj(Z[n]), n = lane + 32 t; Z[n] = A[n] + i B[n] (n <= 512), conj(A[N - n]) + i conj(B[N - n]) above
        if (t < 16) {
          float2 a = tA[lane + 32 * t], b = tB[lane + 32 * t];
          if (t == 0 && lane == 0) { a.y = 0.f; b.y = 0.f; }  // DC: imaginary part ignored (irfft)
          v[t] = make_float2(a.x - b.y, -(a.y + b.x));
        } else if (t == 16) {
          if (lane == 0) {
            float2 a = tA[512], b = tB[512];  // Nyquist: imaginary part ignored
            v[t] = make_float2(a.x, -b.x);
          } else {
            const float2 a = tA[512 - lane], b = tB[512 - lane];
            v[t] = make_float2(a.x + b.y, a.y - b.x);
          }
        } else {
          const float2 a = tA[1024 - 32 * t - lane], b = tB[1024 - 32 * t - lane];
          v[t] = make_float2(a.x + b.y, a.y - b.x);
        }
      }
      __syncwarp();  // both rows fully read before they are overwritten below
      r1k_fft32<PK>(v);
#pragma unroll
      for (int kp = 0; kp < 32; ++kp) xch[lane * XS + kp] = v[R1K_REG(kp)];
      __syncwarp();
#pragma unroll
      for (int n1 = 0; n1 < 32; ++n1) v[n1] = xch[n1 * XS + lane];
      __syncwarp();
      {
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
      r1k_fft32<PK>(v);  // v[R1K_REG(m)] = conj of the inverse transform at sample lane + 32 m (times N)
      float* yA = reinterpret_cast<float*>(tA);
      float* yB = reinterpret_cast<float*>(tB);
#pragma unroll
      for (int m = 0; m < 32; ++m) {
        const float wa = __ldg(P.wa + lane + 32 * m);  // window^a / N
        const float2 z = v[R1K_REG(m)];
        yA[lane + 32 * m] = z.x * wa;
        yB[lane + 32 * m] = -z.y * wa;
      }
    }
    __syncthreads();
    // ---- overlap-add gather over the tile span, one red per padded sample ----
    {
      const int hop = P.hop;
      const int span = (nf - 1) * hop + N;
      float* xo = P.xacc + (size_t)ch * P.L + f0 * hop;
      const int64_t room = P.L - f0 * hop;
      const float* Sf = reinterpret_cast<const float*>(S);
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
    __syncthreads();
  }
}

static ssq_status istft1024_launch(ssq_ctx* ctx, Istft32Params& Q, bool* done) {
  *done = false;
  if (Q.n_fft != 1024 || ctx->opt.no_r1024) return SSQ_OK;
  constexpr int NW = I1K_NW, F = 2 * NW;
  Q.run = F;
  Q.runs_per_channel = (Q.n_use + F - 1) / F;
  Q.total_runs = Q.runs_per_channel * Q.channels;
  // 32-bit tile indices; the tile span inside the range of ssq_fast_div
  if (Q.total_runs > (int64_t)0x7ff00000 || (int64_t)(F - 1) * Q.hop + 1024 >= ((int64_t)1 << 22)) return SSQ_OK;
  *done = true;
  const size_t smem = ((size_t)F * I1K_AS + (size_t)NW * 32 * R1K_XS) * sizeof(float2);
  const int grid = (int)std::min<int64_t>(Q.total_runs, (int64_t)ctx->num_sms * 3);
  SSQ_CUDA_TRY(ctx, cudaFuncSetAttribute(istft1024_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  istft1024_tile_kernel<<<grid, NW * 32, smem, ctx->stream>>>(Q);
  SSQ_TRY(ssq_check_launch(ctx, "istft1024_tile_kernel"));
  ctx->last_kernel = "istft1024_tile_kernel";
  return SSQ_OK;
}
