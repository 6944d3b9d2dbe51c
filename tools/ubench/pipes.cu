// Microbenchmark: do warp shuffles share the L1TEX/shared-memory data pipe with LDS/STS?  And do tensor-memory
// loads / stores (tcgen05.ld / tcgen05.st: LDTM / STTM)?
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o pipes pipes.cu
#include <cstdint>
#include <cstdio>
#include <vector>
#include <algorithm>
#include <cuda_runtime.h>

template <int MODE>
__global__ void __launch_bounds__(256) k(float* out, int iters) {
  __shared__ float2 buf[8][512];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float2* b = buf[warp];
  float2 v[8];
  for (int t = 0; t < 8; ++t) v[t] = make_float2(lane + t, lane - t);
  for (int t = 0; t < 8; ++t) b[lane + 32 * t] = v[t];
  __syncwarp();
  for (int it = 0; it < iters; ++it) {
    if (MODE == 0 || MODE == 2) {  // 8 STS.64 + 8 LDS.64 (conflict-free): 32 wavefronts
#pragma unroll
      for (int t = 0; t < 8; ++t) b[lane + 32 * t] = v[t];
      __syncwarp();
#pragma unroll
      for (int t = 0; t < 8; ++t) v[t] = b[((lane + 1) & 31) + 32 * t];
      __syncwarp();
    }
    if (MODE == 1 || MODE == 2) {  // 16 SHFL.32
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        v[t].x = __shfl_xor_sync(0xffffffffu, v[t].x, 1 + (t & 3));
        v[t].y = __shfl_xor_sync(0xffffffffu, v[t].y, 2 + (t & 3));
      }
    }
    if (MODE == 3) {  // FMA only, for reference
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        v[t].x = fmaf(v[t].x, 1.0001f, v[t].y);
        v[t].y = fmaf(v[t].y, 0.9999f, v[t].x);
      }
    }
    if (MODE == 4) {  // match_any
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        unsigned m = __match_any_sync(0xffffffffu, __float_as_int(v[t].x));
        v[t].x += (float)__popc(m);
      }
    }
  }
  float s = 0;
  for (int t = 0; t < 8; ++t) s += v[t].x + v[t].y;
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}


// ---- tensor memory -------------------------------------------------------------------------------------------
// The shape of the n_fft 512 ssq kernel: 4-warp CTAs, 4 CTAs per SM, each allocating 32 TMEM columns; warp w
// addresses lane quarter w.  One iteration moves 32 columns (x4: 8 instructions, x16: 2, x32: 1) and waits once.
template <int X>
__device__ __forceinline__ void tm_ld(uint32_t (&r)[32], int i, uint32_t taddr);
template <>
__device__ __forceinline__ void tm_ld<4>(uint32_t (&r)[32], int i, uint32_t taddr) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[4 * i]), "=r"(r[4 * i + 1]), "=r"(r[4 * i + 2]), "=r"(r[4 * i + 3])
               : "r"(taddr + 4 * i));
}
template <>
__device__ __forceinline__ void tm_ld<16>(uint32_t (&r)[32], int i, uint32_t taddr) {
  uint32_t* q = r + 16 * i;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
               : "=r"(q[0]), "=r"(q[1]), "=r"(q[2]), "=r"(q[3]), "=r"(q[4]), "=r"(q[5]), "=r"(q[6]), "=r"(q[7]),
                 "=r"(q[8]), "=r"(q[9]), "=r"(q[10]), "=r"(q[11]), "=r"(q[12]), "=r"(q[13]), "=r"(q[14]), "=r"(q[15])
               : "r"(taddr + 16 * i));
}
template <>
__device__ __forceinline__ void tm_ld<32>(uint32_t (&r)[32], int, uint32_t taddr) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,"
               "%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                 "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
                 "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
                 "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
               : "r"(taddr));
}
template <int X>
__device__ __forceinline__ void tm_st(const uint32_t (&r)[32], int i, uint32_t taddr);
template <>
__device__ __forceinline__ void tm_st<4>(const uint32_t (&r)[32], int i, uint32_t taddr) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr + 4 * i), "r"(r[4 * i]),
               "r"(r[4 * i + 1]), "r"(r[4 * i + 2]), "r"(r[4 * i + 3]));
}
template <>
__device__ __forceinline__ void tm_st<16>(const uint32_t (&r)[32], int i, uint32_t taddr) {
  const uint32_t* q = r + 16 * i;
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
               ::"r"(taddr + 16 * i), "r"(q[0]), "r"(q[1]), "r"(q[2]), "r"(q[3]), "r"(q[4]), "r"(q[5]), "r"(q[6]), "r"(q[7]),
               "r"(q[8]), "r"(q[9]), "r"(q[10]), "r"(q[11]), "r"(q[12]), "r"(q[13]), "r"(q[14]), "r"(q[15]));
}
template <>
__device__ __forceinline__ void tm_st<32>(const uint32_t (&r)[32], int, uint32_t taddr) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,"
               "%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
               "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
               "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
               "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31]));
}

// SMEM: 8 STS.64 + 8 LDS.64 per iteration (as mode 0 above); LD / ST: 32 columns of TMEM per iteration in
// instructions of X columns, then tcgen05.wait::ld / wait::st.  Reports clk per warp-iteration per SM by clock64.
template <bool SMEM, bool LD, bool ST, int X>
__global__ void __launch_bounds__(128, 4) ktm(unsigned long long* cycles, float* out, int iters) {
  __shared__ float2 buf[4][512];
  __shared__ uint32_t tmem_base_s;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 32;" ::"r"((uint32_t)__cvta_generic_to_shared(&tmem_base_s)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;");
  const uint32_t taddr = tmem_base_s + ((uint32_t)(warp * 32) << 16);
  float2* b = buf[warp];
  float2 v[8];
  uint32_t r[32], sink = 0;
  for (int t = 0; t < 8; ++t) v[t] = make_float2(lane + t, lane - t);
  for (int t = 0; t < 8; ++t) b[lane + 32 * t] = v[t];
  for (int c = 0; c < 32; ++c) r[c] = lane * 33u + c;
  tm_st<32>(r, 0, taddr);
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  __syncwarp();
  __syncthreads();
  const long long t0 = clock64();
  for (int it = 0; it < iters; ++it) {
    if (LD) {
#pragma unroll
      for (int i = 0; i < 32 / X; ++i) tm_ld<X>(r, i, taddr);
    }
    if (ST) {
#pragma unroll
      for (int i = 0; i < 32 / X; ++i) tm_st<X>(r, i, taddr);
    }
    if (SMEM) {
#pragma unroll
      for (int t = 0; t < 8; ++t) b[lane + 32 * t] = v[t];
      __syncwarp();
#pragma unroll
      for (int t = 0; t < 8; ++t) v[t] = b[((lane + 1) & 31) + 32 * t];
      __syncwarp();
    }
    if (LD) {
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
      for (int c = 0; c < 32; ++c) sink ^= r[c];  // every loaded register is used: no load is dead (~11 LOP3)
    }
    if (ST) asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  __syncthreads();
  const long long t1 = clock64();
  float s = 0;
  for (int t = 0; t < 8; ++t) s += v[t].x + v[t].y;
  for (int c = 0; c < 32; ++c) s += (float)r[c];
  s += (float)sink;
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
  if (threadIdx.x == 0) cycles[blockIdx.x] = (unsigned long long)(t1 - t0);
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 32;" ::"r"(tmem_base_s));
}

template <bool SMEM, bool LD, bool ST, int X>
void run_tm(const char* name, unsigned long long* dc, float* d, int iters, int sms) {
  const int grid = 4 * sms;
  ktm<SMEM, LD, ST, X><<<grid, 128>>>(dc, d, 10);
  ktm<SMEM, LD, ST, X><<<grid, 128>>>(dc, d, iters);
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    printf("%-36s error: %s\n", name, cudaGetErrorString(e));
    return;
  }
  std::vector<unsigned long long> h(grid);
  cudaMemcpy(h.data(), dc, sizeof(unsigned long long) * grid, cudaMemcpyDeviceToHost);
  std::sort(h.begin(), h.end());
  // 4 co-resident CTAs = 16 warps per SM, each running `iters` iterations over the measured interval
  printf("%-36s %6.1f clk per warp-iteration per SM (median CTA, clock64)\n", name, (double)h[grid / 2] / (16.0 * iters));
}

template <int MODE>
void run(const char* name, float* d, int iters) {
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  k<MODE><<<148 * 2, 256>>>(d, 10);
  cudaEventRecord(e0);
  k<MODE><<<148 * 2, 256>>>(d, iters);
  cudaEventRecord(e1);
  cudaEventSynchronize(e1);
  float ms;
  cudaEventElapsedTime(&ms, e0, e1);
  // per SM: 16 warps x iters iterations
  double clk = ms * 1e-3 * 1.965e9 / (16.0 * iters);
  printf("%-28s %8.3f ms  -> %6.1f clk per warp-iteration per SM (at 1965 MHz)\n", name, ms, clk);
}

int main() {
  float* d;
  cudaMalloc(&d, 148 * 2 * 256 * 4);
  const int iters = 20000;
  run<0>("8 STS.64 + 8 LDS.64", d, iters);
  run<1>("16 SHFL", d, iters);
  run<2>("both", d, iters);
  run<3>("16 FFMA (dependent)", d, iters);
  run<4>("8 MATCH.ANY", d, iters);
  int sms = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  unsigned long long* dc;
  cudaMalloc(&dc, sizeof(unsigned long long) * 4 * sms);
  printf("-- 4-warp CTAs, 4 per SM, 32 TMEM columns each; 32 columns per warp-iteration --\n");
  run_tm<true, false, false, 4>("8 STS.64 + 8 LDS.64", dc, d, iters, sms);
  run_tm<false, true, false, 4>("LDTM x4 (8) + wait::ld", dc, d, iters, sms);
  run_tm<false, true, false, 16>("LDTM x16 (2) + wait::ld", dc, d, iters, sms);
  run_tm<false, true, false, 32>("LDTM x32 (1) + wait::ld", dc, d, iters, sms);
  run_tm<false, false, true, 4>("STTM x4 (8) + wait::st", dc, d, iters, sms);
  run_tm<false, false, true, 16>("STTM x16 (2) + wait::st", dc, d, iters, sms);
  run_tm<false, false, true, 32>("STTM x32 (1) + wait::st", dc, d, iters, sms);
  run_tm<true, true, false, 4>("STS/LDS + LDTM x4", dc, d, iters, sms);
  run_tm<true, true, false, 16>("STS/LDS + LDTM x16", dc, d, iters, sms);
  run_tm<true, true, false, 32>("STS/LDS + LDTM x32", dc, d, iters, sms);
  run_tm<true, false, true, 4>("STS/LDS + STTM x4", dc, d, iters, sms);
  run_tm<true, false, true, 16>("STS/LDS + STTM x16", dc, d, iters, sms);
  run_tm<true, false, true, 32>("STS/LDS + STTM x32", dc, d, iters, sms);
  printf("%s\n", cudaGetErrorString(cudaDeviceSynchronize()));
  return 0;
}
