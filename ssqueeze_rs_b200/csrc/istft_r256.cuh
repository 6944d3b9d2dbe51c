// istft_r256.cuh -- inverse STFT for n_fft = 256, any hop (the reference's README geometry).  The pieces of
// istft_r1024.cuh with the 8 x 32 decomposition and four lane groups per warp of stft_r256.cuh: lane = (g, c);
// group g turns the packed pair of frames (fl0 + g, fl0 + 4 + g) -- Z = Z_A + i Z_B, Hermitian extension on the
// fly, inverse = conj(forward(conj)) -- so a warp takes 8 frames per step and a 4-warp CTA a tile of 32 frames
// (256 B row segments).
#pragma once
#include "istft_r1024.cuh"
#include "stft_r256.cuh"

#define I256_AS 131  // tile row stride (float2): odd; 262 floats >= 256 samples
#define I256_NW 4    // warps per CTA; F = 8 NW frames per tile

__global__ void __launch_bounds__(I256_NW * 32, 3) istft256_tile_kernel(const Istft32Params P) {
  constexpr int N = 256, AS = I256_AS, XS = R1K_XS, NW = I256_NW, F = 8 * NW;
  constexpr bool PK = true;
  static_assert(NW == 4, "the load mapping below assumes 4 warps x 32 frames");
  extern __shared__ float2 smem[];
  float2* S = smem;  // [F][AS]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 3, c = lane & 7;
  float2* xch = S + F * AS + warp * (32 * XS);
  const float2 wb = P.tw[c];  // W_256^c
  const int tpc = (int)P.runs_per_channel, ntiles = (int)P.total_runs;

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int ch = tile / tpc;
    const int64_t f0 = (int64_t)(tile - ch * tpc) * F;
    const int nf = (int)min((int64_t)F, P.n_use - f0);
    // ---- tile load: lane -> frame, warp w and step it -> row w + 4 it (256 B per row) ----
    {
      const bool ok = lane < nf;
      const float2* gp = P.Sx + ((size_t)ch * 129 + warp) * P.n_frames + f0 + lane;
      const size_t gstep = (size_t)4 * P.n_frames;
      float2* s = S + lane * AS + warp;
#pragma unroll 8
      for (int it = 0; it < 32; ++it) {
        s[4 * it] = ok ? __ldg(gp) : make_float2(0.f, 0.f);
        gp += gstep;
      }
      if (warp == 0) s[128] = ok ? __ldg(gp) : make_float2(0.f, 0.f);
    }
    __syncthreads();
    // ---- transform: warp w, group g: frames 8 w + g (real part) and 8 w + 4 + g (imaginary part) ----
    const int fa = 8 * warp + g;
    if (8 * warp < nf) {  // warp-uniform; rows past nf are zero
      float2* tA = S + fa * AS;
      float2* tB = tA + 4 * AS;
      float2 v[32];
#pragma unroll
      for (int t = 0; t < 32; ++t) {
        // conj(Z[n]), n = c + 8 t; Z[n] = A[n] + i B[n] (n <= 128), conj(A[N - n]) + i conj(B[N - n]) above
        if (t < 16) {
          float2 a = tA[c + 8 * t], b = tB[c + 8 * t];
          if (t == 0 && c == 0) { a.y = 0.f; b.y = 0.f; }  // DC: imaginary part ignored (irfft)
          v[t] = make_float2(a.x - b.y, -(a.y + b.x));
        } else if (t == 16) {
          if (c == 0) {
            const float2 a = tA[128], b = tB[128];  // Nyquist: imaginary part ignored
            v[t] = make_float2(a.x, -b.x);
          } else {
            const float2 a = tA[128 - c], b = tB[128 - c];
            v[t] = make_float2(a.x + b.y, a.y - b.x);
          }
        } else {
          const float2 a = tA[256 - 8 * t - c], b = tB[256 - 8 * t - c];
          v[t] = make_float2(a.x + b.y, a.y - b.x);
        }
      }
      __syncwarp();  // all rows of the warp fully read before they are overwritten below
      r1k_fft32<PK>(v);  // v[R1K_REG(kappa)] = Y[c][kappa]
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
      float* yA = reinterpret_cast<float*>(tA);
      float* yB = reinterpret_cast<float*>(tB);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float2 a[8];
#pragma unroll
        for (int n1 = 0; n1 < 8; ++n1) a[n1] = v[8 * j + n1];
        fft8_fwd<PK>(a);  // a[m] = conj of the inverse transform at sample c + 8 j + 32 m (times N)
#pragma unroll
        for (int m = 0; m < 8; ++m) {
          const int n = c + 8 * j + 32 * m;
          const float wa = __ldg(P.wa + n);  // window^a / N
          yA[n] = a[m].x * wa;
          yB[n] = -a[m].y * wa;
        }
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

static ssq_status istft256_launch(ssq_ctx* ctx, Istft32Params& Q, bool* done) {
  *done = false;
  if (Q.n_fft != 256 || ctx->opt.no_r256) return SSQ_OK;
  constexpr int NW = I256_NW, F = 8 * NW;
  Q.run = F;
  Q.runs_per_channel = (Q.n_use + F - 1) / F;
  Q.total_runs = Q.runs_per_channel * Q.channels;
  // 32-bit tile indices; the tile span inside the range of ssq_fast_div
  if (Q.total_runs > (int64_t)0x7ff00000 || (int64_t)(F - 1) * Q.hop + 256 >= ((int64_t)1 << 22)) return SSQ_OK;
  *done = true;
  const size_t smem = ((size_t)F * I256_AS + (size_t)NW * 32 * R1K_XS) * sizeof(float2);
  const int grid = (int)std::min<int64_t>(Q.total_runs, (int64_t)ctx->num_sms * 3);
  SSQ_CUDA_TRY(ctx, cudaFuncSetAttribute(istft256_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  istft256_tile_kernel<<<grid, NW * 32, smem, ctx->stream>>>(Q);
  SSQ_TRY(ssq_check_launch(ctx, "istft256_tile_kernel"));
  ctx->last_kernel = "istft256_tile_kernel";
  return SSQ_OK;
}
