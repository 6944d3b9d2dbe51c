// ssqcuda.cu -- C ABI of libssqcuda (see include/ssqcuda.h) and the host-side
// set-up logic of each transform.  Device code lives in the *.cuh files.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared
#include "ssq_common.cuh"
#include "host_math.h"
#include "stft_kernels.cuh"
#include "fft_regs.cuh"
#include "stft_h32r.cuh"
#include "stft_r1024.cuh"
#include "stft_r256.cuh"
#include "istft_h32.cuh"
#include "istft_r1024.cuh"
#include "istft_r256.cuh"
#include "istream_kernels.cuh"
#include "cwt_kernels.cuh"
#include "components_kernels.cuh"
#include "ridge_kernels.cuh"

#include <algorithm>
#include <ctype.h>
#include <sys/syscall.h>
#include <unistd.h>
#include <thread>
#include <stdlib.h>
#include <new>

static const double kEps64 = 2.2204460492503131e-16;

// ===========================================================================
// library / context
// ===========================================================================
extern "C" const char* ssq_version(void) {
  return "ssqcuda 0.4 (B200 sm_100a; stft, ssq_stft, istft, issq_stft, cwt, cwt_simd, ssq_cwt, icwt, issq_cwt, "
         "ssq_stft streaming, istft / issq_stft streaming, ridge extraction, issq_cwt / issq_stft components)";
}

// lib.rs:16-19
extern "C" const char* ssq_hello_from_bin(void) { return "Hello from ssqueeze!"; }

extern "C" int ssq_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    (void)cudaGetLastError();
    return 0;
  }
  return n;
}

extern "C" ssq_status ssq_ctx_create(int device, ssq_ctx** out) {
  if (!out) return ssq_fail(nullptr, SSQ_EINVAL, "ssq_ctx_create: out is NULL");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    (void)cudaGetLastError();
    return ssq_fail(nullptr, SSQ_ECUDA, "no CUDA device available (%s); libssqcuda has no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  }
  if (device < 0 || device >= n)
    return ssq_fail(nullptr, SSQ_EINVAL, "device %d out of range [0, %d)", device, n);
  ssq_ctx* c = new (std::nothrow) ssq_ctx();
  if (!c) return ssq_fail(nullptr, SSQ_ENOMEM, "out of host memory");
  c->device = device;
  cudaDeviceProp prop;
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
    delete c;
    return ssq_fail(nullptr, SSQ_ECUDA, "cudaSetDevice/GetDeviceProperties: %s", cudaGetErrorString(e));
  }
  if (prop.major < 10) {
    delete c;
    return ssq_fail(nullptr, SSQ_ECUDA, "device %d is sm_%d%d; libssqcuda is built for sm_100a only", device,
                    prop.major, prop.minor);
  }
  c->num_sms = prop.multiProcessorCount;
  c->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
  if ((e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaEventCreate(&c->ev0)) != cudaSuccess || (e = cudaEventCreate(&c->ev1)) != cudaSuccess) {
    delete c;
    return ssq_fail(nullptr, SSQ_ECUDA, "stream/event creation: %s", cudaGetErrorString(e));
  }
  c->stream = c->own_stream;
  *out = c;
  return SSQ_OK;
}

extern "C" ssq_status ssq_ctx_set_option(ssq_ctx* ctx, const char* name, int64_t value) {
  if (!ctx || !name) return ssq_fail(ctx, SSQ_EINVAL, "ssq_ctx_set_option: NULL argument");
  const std::string n(name);
  ssq_ctx::Options& o = ctx->opt;
  if (n == "no_h32r") o.no_h32r = value != 0;
  else if (n == "no_r1024") o.no_r1024 = value != 0;
  else if (n == "no_r256") o.no_r256 = value != 0;
  else if (n == "no_cwt_fused") o.no_cwt_fused = value != 0;
  else if (n == "upstream_framing") o.upstream_framing = value != 0;
  else return ssq_fail(ctx, SSQ_EINVAL, "ssq_ctx_set_option: unknown option '%s'", name);
  return SSQ_OK;
}

extern "C" void ssq_ctx_destroy(ssq_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  DevBuf* bufs[] = {&ctx->ws_in, &ctx->ws_out, &ctx->ws_aux0, &ctx->ws_aux1, &ctx->ws_aux2, &ctx->ws_fft0,
                    &ctx->ws_fft1, &ctx->ws_misc, &ctx->tab, &ctx->cwt_tw, &ctx->cwt_scales};
  for (DevBuf* b : bufs)
    if (b->p) cudaFree(b->p);
  for (DevBuf& b : ctx->ws_ridge)
    if (b.p) cudaFree(b.p);
  if (ctx->rows_tab.p) cudaFree(ctx->rows_tab.p);
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  for (int i = 0; i < 2; ++i) {
    if (ctx->pin[i]) cudaFreeHost(ctx->pin[i]);
    if (ctx->pin_ev[i]) cudaEventDestroy(ctx->pin_ev[i]);
  }
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  delete ctx;
}

extern "C" const char* ssq_last_error(const ssq_ctx* ctx) { return ctx ? ctx->err.c_str() : g_tls_err.c_str(); }

extern "C" ssq_status ssq_ctx_set_stream(ssq_ctx* ctx, void* cuda_stream) {
  if (!ctx) return ssq_fail(nullptr, SSQ_EINVAL, "ctx is NULL");
  ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
  return SSQ_OK;
}

extern "C" ssq_status ssq_ctx_synchronize(ssq_ctx* ctx) {
  if (!ctx) return ssq_fail(nullptr, SSQ_EINVAL, "ctx is NULL");
  SSQ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  SSQ_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return SSQ_OK;
}

extern "C" uint64_t ssq_ctx_launch_count(const ssq_ctx* ctx) { return ctx ? ctx->launches : 0; }

extern "C" float ssq_ctx_last_kernel_ms(ssq_ctx* ctx) {
  if (!ctx || !ctx->ev_valid) return -1.f;
  if (cudaEventSynchronize(ctx->ev1) != cudaSuccess) return -1.f;
  float ms = -1.f;
  if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) != cudaSuccess) return -1.f;
  return ms;
}

extern "C" const char* ssq_ctx_last_kernel_name(const ssq_ctx* ctx) { return ctx ? ctx->last_kernel : ""; }

extern "C" ssq_status ssq_host_alloc(void** p, size_t bytes) {
  if (!p) return ssq_fail(nullptr, SSQ_EINVAL, "p is NULL");
  cudaError_t e = cudaHostAlloc(p, bytes, cudaHostAllocDefault);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    *p = nullptr;
    return ssq_fail(nullptr, SSQ_ENOMEM, "cudaHostAlloc(%zu): %s", bytes, cudaGetErrorString(e));
  }
  return SSQ_OK;
}
extern "C" void ssq_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

// Plain asynchronous copy on a caller-provided stream (the measurement of the box's copy ceiling goes through the
// same runtime instance as the library's own pipeline).
extern "C" ssq_status ssq_memcpy_async(void* dst, const void* src, size_t bytes, int kind, void* cuda_stream) {
  if (kind != 1 && kind != 2) return ssq_fail(nullptr, SSQ_EINVAL, "kind must be 1 (H2D) or 2 (D2H)");
  cudaError_t e = cudaMemcpyAsync(dst, src, bytes, kind == 1 ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost,
                                  (cudaStream_t)cuda_stream);
  if (e != cudaSuccess) return ssq_fail(nullptr, SSQ_ECUDA, "cudaMemcpyAsync: %s", cudaGetErrorString(e));
  return SSQ_OK;
}

// NUMA node the device's PCIe function hangs off (sysfs), -1 when the platform does not say.
extern "C" ssq_status ssq_device_numa_node(int device, int* node) {
  if (!node) return ssq_fail(nullptr, SSQ_EINVAL, "node is NULL");
  *node = -1;
  char bus[32] = {0};
  if (cudaDeviceGetPCIBusId(bus, sizeof(bus), device) != cudaSuccess) {
    (void)cudaGetLastError();
    return ssq_fail(nullptr, SSQ_ECUDA, "cudaDeviceGetPCIBusId(%d) failed", device);
  }
  for (char* q = bus; *q; ++q) *q = (char)tolower((unsigned char)*q);
  char path[128];
  snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", bus);
  if (FILE* f = fopen(path, "r")) {
    int v = -1;
    if (fscanf(f, "%d", &v) == 1) *node = v;
    fclose(f);
  }
  return SSQ_OK;
}

// Pinned host memory placed on the device's NUMA node: the pages are allocated (and pinned) by cudaHostAlloc
// while the calling thread's memory policy is MPOL_BIND to that node, then the policy is restored.  On an 8-GPU box
// the host gather of Tx (44 GB per GPU and step on configs[1]) otherwise lands wherever the rank's thread happens to
// run, and half of the copies cross the socket interconnect.  Falls back to a plain allocation when the node is
// unknown or the policy call is refused.
extern "C" ssq_status ssq_host_alloc_near(void** p, size_t bytes, int device) {
  if (!p) return ssq_fail(nullptr, SSQ_EINVAL, "p is NULL");
  int node = -1;
  (void)ssq_device_numa_node(device, &node);
  bool bound = false;
  if (node >= 0 && node < 1024) {
    unsigned long mask[16] = {0};
    mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
    bound = syscall(SYS_set_mempolicy, 2 /* MPOL_BIND */, mask, (unsigned long)(8 * sizeof(mask))) == 0;
  }
  cudaSetDevice(device);
  const ssq_status st = ssq_host_alloc(p, bytes);
  if (bound) syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0ul);
  return st;
}

// ===========================================================================
// shape queries
// ===========================================================================
extern "C" ssq_status ssq_stft_shape(int64_t n, int n_fft, int hop, int64_t* n_freqs, int64_t* n_frames) {
  if (n < 1 || n_fft < 1 || hop < 1)
    return ssq_fail(nullptr, SSQ_EPANIC, "stft shape: n=%lld n_fft=%d hop=%d (the reference panics: stft.rs:33)",
                    (long long)n, n_fft, hop);
  if (n_freqs) *n_freqs = n_fft / 2 + 1;
  if (n_frames) *n_frames = (n - 1) / hop + 1;
  return SSQ_OK;
}

extern "C" ssq_status ssq_cwt_shape(int64_t n, int64_t* pad_len, int64_t* n1) {
  if (n < 1) return ssq_fail(nullptr, SSQ_EINVAL, "cwt shape: n=%lld", (long long)n);
  const int64_t pl = ssqhost::next_power_of_2(n + n / 2);
  if (pad_len) *pad_len = pl;
  if (n1) *n1 = (pl - n) / 2;
  return SSQ_OK;
}

extern "C" int64_t ssq_cwt_default_scales(int64_t n, int nv, int simd, double* scales) {
  return ssqhost::default_scales(n, nv, simd, scales);
}

// ===========================================================================
// STFT family: host set-up
// ===========================================================================
enum { TAB_SSQ = 0, TAB_STFT = 1, TAB_ISTFT = 2 };

struct StftTables {
  const float* win;
  const float* dwin;
  const float2* tw;
  const float* wa;
  const float* wpow;
  const float2* wpair;  // (win, dwin * s) interleaved; not for TAB_ISTFT (shares the slots of wa / wpow)
  double s_scale;
};

// Uploads (or reuses) the per-window device tables:
// [win N][dwin*s N][tw 2N][wa N][wpow N] floats.
static ssq_status stft_tables(ssq_ctx* ctx, const std::vector<double>& wfit, int kind, int win_exp,
                              StftTables* T) {
  const int N = (int)wfit.size();
  const int key_kind = kind * 16 + (kind == TAB_ISTFT ? (win_exp & 15) : 0);
  const bool hit = ctx->tab.p && ctx->tab_nfft == N && ctx->tab_kind == key_kind &&
                   ctx->tab_window.size() == wfit.size() &&
                   memcmp(ctx->tab_window.data(), wfit.data(), sizeof(double) * N) == 0;
  float* base = nullptr;
  if (!hit) {
    std::vector<float> h((size_t)6 * N, 0.f);
    double s_scale = 1.0;
    for (int i = 0; i < N; ++i) h[i] = (float)wfit[i];
    if (kind == TAB_SSQ) {
      std::vector<double> dw = ssqhost::diff_window(wfit);
      double sw = 0.0, sd = 0.0;
      for (int i = 0; i < N; ++i) {
        sw += wfit[i] * wfit[i];
        sd += dw[i] * dw[i];
      }
      if (sd > 0.0 && sw > 0.0) s_scale = std::sqrt(sw / sd);
      for (int i = 0; i < N; ++i) h[(size_t)N + i] = (float)(dw[i] * s_scale);
    }
    for (int i = 0; i < N; ++i) {
      const double ang = -2.0 * SSQ_PI * (double)i / (double)N;
      h[(size_t)2 * N + 2 * i] = (float)std::cos(ang);
      h[(size_t)2 * N + 2 * i + 1] = (float)std::sin(ang);
    }
    if (kind != TAB_ISTFT) {
      for (int i = 0; i < N; ++i) {
        h[(size_t)4 * N + 2 * i] = h[i];
        h[(size_t)4 * N + 2 * i + 1] = h[(size_t)N + i];
      }
    }
    if (kind == TAB_ISTFT) {
      for (int i = 0; i < N; ++i) {
        const double wa = win_exp == 0 ? 1.0 : std::pow(wfit[i], (double)win_exp);
        h[(size_t)4 * N + i] = (float)(wa / (double)N);
        h[(size_t)5 * N + i] = (float)std::pow(wfit[i], (double)(win_exp + 1));
      }
    }
    SSQ_TRY(devbuf_reserve(ctx, ctx->tab, h.size() * sizeof(float)));
    // the previous tables may still be read by queued kernels
    SSQ_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    SSQ_CUDA_TRY(ctx, cudaMemcpy(ctx->tab.p, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice));
    ctx->tab_window = wfit;
    ctx->tab_nfft = N;
    ctx->tab_kind = key_kind;
    ctx->tab_sscale = s_scale;
  }
  base = (float*)ctx->tab.p;
  T->win = base;
  T->dwin = base + N;
  T->tw = (const float2*)(base + 2 * (size_t)N);
  T->wa = base + 4 * (size_t)N;
  T->wpow = base + 5 * (size_t)N;
  T->wpair = (const float2*)(base + 4 * (size_t)N);
  T->s_scale = ctx->tab_sscale;
  return SSQ_OK;
}

static inline int ilog2_exact(int n) {
  int l = 0;
  while ((1 << l) < n) ++l;
  return ((1 << l) == n) ? l : -1;
}

struct TilePlan {
  int F, acc_stride, nw;
  size_t smem;
  int grid;
};

// tile geometry for the generic (shared-memory) kernels
static ssq_status plan_generic_tiles(ssq_ctx* ctx, int n_fft, int n_freqs, int64_t n_frames, int channels,
                                     TilePlan* tp, int64_t* tiles_per_channel, int64_t* total_tiles) {
  const size_t budget = std::min<size_t>((size_t)ctx->max_smem_optin, 200 * 1024);
  const int acc_stride = n_freqs | 1;
  int F = 32, nw = 8;
  auto need = [&](int F_, int nw_) {
    return ((size_t)F_ * acc_stride + (size_t)nw_ * 2 * n_fft + (size_t)n_fft) * sizeof(float2) +
           (size_t)nw_ * ((n_freqs + 7) & ~7);  // + per-warp tag bytes (stft_generic_kernel)
  };
  // keep the warps first (they are what hides latency), then the frames per tile (row segments of
  // F * 8 B); shrink F down to the warp count before giving up warps
  while (F > nw && need(F, nw) > budget) F >>= 1;
  while (nw > 1 && need(F, nw) > budget) {
    nw >>= 1;
    F = std::max(F >> 1, 1);
  }
  while (F > 1 && need(F, nw) > budget) F >>= 1;
  if (need(F, nw) > budget)
    return ssq_fail(ctx, SSQ_EUNSUPPORTED, "n_fft=%d needs %zu B of shared memory per CTA (> %zu)", n_fft,
                    need(F, nw), budget);
  if ((int64_t)F > n_frames) {
    int f2 = 1;
    while (f2 < n_frames) f2 <<= 1;
    F = std::max(1, std::min(F, f2));
  }
  tp->F = F;
  tp->acc_stride = acc_stride;
  tp->nw = nw;
  tp->smem = need(F, nw);
  *tiles_per_channel = (n_frames + F - 1) / F;
  *total_tiles = *tiles_per_channel * channels;
  const int per_sm = std::max<int>(1, (int)(((size_t)220 * 1024) / (tp->smem + 1024)));
  const int64_t g = std::min<int64_t>(*total_tiles, (int64_t)ctx->num_sms * per_sm);
  tp->grid = (int)std::max<int64_t>(1, g);
  return SSQ_OK;
}

struct StftCall {
  int mode;  // 0 ssq, 1 stft
  const float* d_x;
  int64_t channels, n, x_stride;
  std::vector<double> wfit;
  int n_fft, hop;
  double fs;
  int padtype, squeezing;
  double gamma;
  unsigned flags;
  float2* d_out;
  float2* aux_Sx;
  float2* aux_dSx;
  float* aux_w;
  int* aux_kb = nullptr;
  // streaming (ssq_stream_*): compute frames [frame0, frame0 + n_frames_call) of a recording of n
  // samples, of which d_x holds [x_origin, ...)
  int64_t frame0 = 0;
  int64_t n_frames_call = 0;
  int64_t x_origin = 0;  // global sample index of d_x[.][0]
};

static ssq_status stft_rows_run(ssq_ctx* ctx, StftParams P, bool* done);  // stft_rows.inl
static ssq_status istft_rows_run(ssq_ctx* ctx, IstftParams P, bool* done);

static ssq_status run_stft_family(ssq_ctx* ctx, const StftCall& c) {
  SSQ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const int N = c.n_fft;
  if (N < 2) return ssq_fail(ctx, SSQ_EINVAL, "n_fft=%d: need n_fft >= 2", N);
  if (c.hop < 1) return ssq_fail(ctx, SSQ_EPANIC, "hop=%d: the reference divides by it (ssq_stft.rs:183)", c.hop);
  if (c.n < 1 || c.channels < 1)
    return ssq_fail(ctx, SSQ_EPANIC, "empty input (n=%lld, channels=%lld): usize underflow in the reference",
                    (long long)c.n, (long long)c.channels);
  const int n_freqs = N / 2 + 1;
  const bool streaming = c.n_frames_call > 0;
  const int64_t n_frames = streaming ? c.n_frames_call : (c.n - 1) / c.hop + 1;
  StftTables T;
  SSQ_TRY(stft_tables(ctx, c.wfit, c.mode == 0 ? TAB_SSQ : TAB_STFT, 0, &T));

  StftParams P;
  memset(&P, 0, sizeof(P));
  P.x = c.d_x;
  P.x_stride = c.x_stride;
  P.n = c.n;
  P.channels = (int)c.channels;
  P.n_fft = N;
  P.hop = c.hop;
  P.n_freqs = n_freqs;
  P.log2n = ilog2_exact(N);
  P.is_pow2 = P.log2n >= 0;
  P.n_frames = n_frames;
  P.frame0 = c.frame0;
  P.x_origin = c.x_origin;
  P.left = ctx->opt.upstream_framing ? N / 2 : (N - 1) / 2;  // stft_utils.rs:22 | old/ssqueezepy/utils/common.py:116-120
  P.padtype = c.padtype == SSQ_PAD_ZERO ? SSQ_PAD_ZERO
              : ctx->opt.upstream_framing ? SSQ_PAD_REFLECT_UPSTREAM  // np.pad's reflect (stft_sample)
              : SSQ_PAD_REFLECT;
  P.win = T.win;
  P.dwin = T.dwin;
  P.wpair = T.wpair;
  P.tw = T.tw;
  const double dw_f = 0.5 * c.fs / ((double)n_freqs - 1.0);  // ssq_stft.rs:50,273
  // gamma: NaN = "not given" -> 10 eps (ssq_stft.rs:258-261); an explicit negative value never gates
  // (|Sx| < gamma is always false, ssq_stft.rs:23)
  const double gamma = (c.gamma != c.gamma) ? 10.0 * kEps64 : c.gamma;
  P.cphase = (float)(((double)n_freqs - 1.0) / (SSQ_PI * T.s_scale));
  P.gate2 = gamma < 0.0 ? -1.f : (float)std::min(4.0 * gamma * gamma, 3.0e38);
  P.tx_scale = (float)(0.5 * dw_f);
  P.leb_val = (float)(dw_f / (double)n_freqs);
  P.dw_f = (float)dw_f;
  P.dsx_scale = (float)(0.5 * c.fs / T.s_scale);
  P.mode = c.mode;
  P.squeezing = c.squeezing == SSQ_SQUEEZE_LEBESGUE ? SSQ_SQUEEZE_LEBESGUE : SSQ_SQUEEZE_SUM;
  P.modulated = (c.flags & SSQ_FLAG_MODULATED) ? 1 : 0;
  P.out = c.d_out;
  P.aux_Sx = c.aux_Sx;
  P.aux_dSx = c.aux_dSx;
  P.aux_w = c.aux_w;
  P.aux_kb = c.aux_kb;

  SSQ_CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  bool done = false;
  // diagnostic outputs (aux_*) do not change the kernel selection: the register kernels carry them as a
  // compile-time variant of the same code
  // a signal of n <= left in upstream reflect needs np.pad's repeated reflection, which only the generic kernel and
  // the rows path compile in: the register kernels' edge-sample function keeps the crate's one reflection, so that
  // the code of the benchmarked kernel does not change with it
  const bool fold = P.padtype == SSQ_PAD_REFLECT_UPSTREAM && P.n <= P.left;
  for (auto launch : {stft_h32r_launch, stft_r1024_launch, stft_r256_launch}) {
    if (fold) break;
    SSQ_TRY(launch(ctx, P, &done));
    if (done) break;
  }
  if (!done) SSQ_TRY(stft_rows_run(ctx, P, &done));  // n_fft > 4096, or not a power of two: batched row FFTs
  if (!done) {
    TilePlan tp;
    SSQ_TRY(plan_generic_tiles(ctx, N, n_freqs, n_frames, (int)c.channels, &tp, &P.tiles_per_channel,
                               &P.total_tiles));
    P.F = tp.F;
    P.acc_stride = tp.acc_stride;
    SSQ_CUDA_TRY(ctx, cudaFuncSetAttribute(stft_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)tp.smem));
    stft_generic_kernel<<<tp.grid, tp.nw * 32, tp.smem, ctx->stream>>>(P);
    SSQ_TRY(ssq_check_launch(ctx, "stft_generic_kernel"));
    ctx->last_kernel = "stft_generic_kernel";
  }
  SSQ_CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  ctx->ev_valid = true;
  return SSQ_OK;
}

// ---------------------------------------------------------------------------
// batched device entry points
// ---------------------------------------------------------------------------
extern "C" ssq_status ssq_ssq_stft_batch_diag_f32(ssq_ctx* ctx, const float* d_x, int64_t channels, int64_t n,
                                                  int64_t x_stride, const double* window, int64_t win_n, int n_fft,
                                                  int hop, double fs, int padtype, int squeezing, double gamma,
                                                  unsigned flags, float* d_Tx, float* d_Sx, float* d_dSx, float* d_w,
                                                  int32_t* d_kb) {
  if (!ctx) return ssq_fail(nullptr, SSQ_EINVAL, "ctx is NULL");
  if (!d_x || !d_Tx || !window || win_n < 1) return ssq_fail(ctx, SSQ_EINVAL, "NULL/empty argument");
  if (n_fft <= 0) n_fft = (int)std::min<int64_t>(n, 512);  // ssq_stft.rs:92
  if (win_n > n_fft)
    return ssq_fail(ctx, SSQ_EINVAL, "Window length %lld cannot be greater than n_fft %d", (long long)win_n, n_fft);
  StftCall c;
  c.mode = 0;
  c.d_x = d_x;
  c.channels = channels;
  c.n = n;
  c.x_stride = x_stride > 0 ? x_stride : n;
  c.wfit = ssqhost::fit_window(window, win_n, n_fft);
  c.n_fft = n_fft;
  c.hop = hop;
  c.fs = fs;
  c.padtype = padtype;
  c.squeezing = squeezing;
  c.gamma = gamma;
  c.flags = flags;
  c.d_out = (float2*)d_Tx;
  c.aux_Sx = (float2*)d_Sx;
  c.aux_dSx = (float2*)d_dSx;
  c.aux_w = d_w;
  c.aux_kb = d_kb;
  return run_stft_family(ctx, c);
}

extern "C" ssq_status ssq_ssq_stft_batch_f32(ssq_ctx* ctx, const float* d_x, int64_t channels, int64_t n,
                                             int64_t x_stride, const double* window, int64_t win_n, int n_fft,
                                             int hop, double fs, int padtype, int squeezing, double gamma,
                                             unsigned flags, float* d_Tx) {
  return ssq_ssq_stft_batch_diag_f32(ctx, d_x, channels, n, x_stride, window, win_n, n_fft, hop, fs, padtype, squeezing,
                                     gamma, flags, d_Tx, nullptr, nullptr, nullptr, nullptr);
}

extern "C" ssq_status ssq_stft_batch_f32(ssq_ctx* ctx, const float* d_x, int64_t channels, int64_t n,
                                         int64_t x_stride, const double* window, int64_t win_n, int n_fft,
                                         int hop, int padtype, float* d_Sx) {
  if (!ctx) return ssq_fail(nullptr, SSQ_EINVAL, "ctx is NULL");
  if (!d_x || !d_Sx || !window) return ssq_fail(ctx, SSQ_EINVAL, "NULL argument");
  if (n_fft < 2) return ssq_fail(ctx, SSQ_EINVAL, "n_fft=%d: need n_fft >= 2", n_fft);
  if (win_n < n_fft)
    return ssq_fail(ctx, SSQ_EPANIC,
                    "window length %lld < n_fft %d: the reference panics in rustfft (stft_utils.rs:8, stft.rs:67)",
                    (long long)win_n, n_fft);
  StftCall c;
  c.mode = 1;
  c.d_x = d_x;
  c.channels = channels;
  c.n = n;
  c.x_stride = x_stride > 0 ? x_stride : n;
  c.wfit.assign(window, window + n_fft);  // first n_fft taps (stft_utils.rs:8)
  c.n_fft = n_fft;
  c.hop = hop;
  c.fs = 1.0;
  c.padtype = padtype;
  c.squeezing = SSQ_SQUEEZE_SUM;
  c.gamma = 0.0;
  c.flags = 0;
  c.d_out = (float2*)d_Sx;
  c.aux_Sx = nullptr;
  c.aux_dSx = nullptr;
  c.aux_w = nullptr;
  return run_stft_family(ctx, c);
}

static inline int istft_left(const ssq_ctx* ctx, int n_fft) {
  return ctx->opt.upstream_framing ? n_fft / 2 : (n_fft - 1) / 2;
}

// Overlap-adds the windowed inverse transforms of frames [0, n_use) of Sx (complex64 [channels, n_freqs, n_frames])
// into xacc ([channels, L], zeroed by the caller; frame f lands at f * hop, and (n_use - 1) * hop + n_fft <= L): the
// register tile kernels, then the row passes, then the generic kernel.  The window-norm division is the caller's.
// ev0 / ev1 bracket the dispatch and last_kernel names the kernel that ran.  Shared by the batch call and the stream.
static ssq_status istft_ola_run(ssq_ctx* ctx, const float2* Sx, int64_t channels, int64_t n_freqs, int64_t n_frames,
                                int64_t n_use, int n_fft, int hop, const StftTables& T, float* xacc, int64_t L) {
  Istft32Params Q;
  memset(&Q, 0, sizeof(Q));
  Q.Sx = Sx;
  Q.channels = (int)channels;
  Q.n_frames = n_frames;
  Q.n_use = n_use;
  Q.L = L;
  Q.wa = T.wa;
  Q.tw = T.tw;
  Q.xacc = xacc;
  Q.hop = hop;
  Q.n_fft = n_fft;
  SSQ_CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  bool done = false;
  for (auto launch : {istft512_launch, istft256_launch, istft1024_launch}) {
    SSQ_TRY(launch(ctx, Q, &done));
    if (done) break;
  }
  if (!done) {
    IstftParams P;
    memset(&P, 0, sizeof(P));
    P.Sx = Q.Sx;
    P.channels = Q.channels;
    P.n_fft = n_fft;
    P.hop = hop;
    P.n_freqs = (int)n_freqs;
    P.log2n = ilog2_exact(n_fft);
    P.is_pow2 = P.log2n >= 0;
    P.n_frames = n_frames;
    P.n_use = Q.n_use;
    P.L = L;
    P.wa = T.wa;
    P.tw = T.tw;
    P.xacc = Q.xacc;
    SSQ_TRY(istft_rows_run(ctx, P, &done));  // n_fft > 4096, or not a power of two: batched row FFTs
    if (!done) {
      TilePlan tp;
      SSQ_TRY(plan_generic_tiles(ctx, n_fft, (int)n_freqs, P.n_use, (int)channels, &tp, &P.tiles_per_channel,
                                 &P.total_tiles));
      P.F = tp.F;
      P.acc_stride = tp.acc_stride;
      SSQ_CUDA_TRY(ctx,
                   cudaFuncSetAttribute(istft_ola_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tp.smem));
      istft_ola_kernel<<<tp.grid, tp.nw * 32, tp.smem, ctx->stream>>>(P);
      SSQ_TRY(ssq_check_launch(ctx, "istft_ola_kernel"));
      ctx->last_kernel = "istft_ola_kernel";
    }
  }
  SSQ_CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  ctx->ev_valid = true;
  return SSQ_OK;
}

extern "C" ssq_status ssq_istft_batch_f32(ssq_ctx* ctx, const float* d_Sx, int64_t channels, int64_t n_freqs,
                                          int64_t n_frames, const double* window, int64_t win_n, int n_fft,
                                          int hop, int64_t n_out, int win_exp, float* d_xout) {
  if (!ctx) return ssq_fail(nullptr, SSQ_EINVAL, "ctx is NULL");
  if (!d_Sx || !d_xout || !window || win_n < 1) return ssq_fail(ctx, SSQ_EINVAL, "NULL/empty argument");
  SSQ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (n_fft <= 0) n_fft = (int)(n_freqs - 1) * 2;  // _stft.py:229
  if (n_fft < 2 || n_fft / 2 + 1 != n_freqs)
    return ssq_fail(ctx, SSQ_EINVAL, "Sx has %lld rows but n_fft=%d needs %d", (long long)n_freqs, n_fft,
                    n_fft / 2 + 1);
  if (hop < 1 || n_frames < 1 || channels < 1 || win_exp < 0)
    return ssq_fail(ctx, SSQ_EINVAL, "bad hop/n_frames/channels/win_exp");
  if (n_out <= 0) n_out = (int64_t)hop * n_frames;  // _stft.py:231
  std::vector<double> wfit = ssqhost::fit_window(window, win_n, n_fft);
  StftTables T;
  SSQ_TRY(stft_tables(ctx, wfit, TAB_ISTFT, win_exp, &T));
  const int64_t L = n_out + n_fft - 1;
  const int64_t max_hops = (L - n_fft) / hop + 1;
  SSQ_TRY(devbuf_reserve(ctx, ctx->ws_misc, (size_t)channels * L * sizeof(float)));
  SSQ_CUDA_TRY(ctx, cudaMemsetAsync(ctx->ws_misc.p, 0, (size_t)channels * L * sizeof(float), ctx->stream));
  SSQ_TRY(istft_ola_run(ctx, (const float2*)d_Sx, channels, n_freqs, n_frames, std::min<int64_t>(n_frames, max_hops),
                        n_fft, hop, T, (float*)ctx->ws_misc.p, L));
  dim3 g((unsigned)((n_out + ISTFT_FIN_PER_BLOCK - 1) / ISTFT_FIN_PER_BLOCK), (unsigned)channels);
  istft_finalize_kernel<<<g, 256, 0, ctx->stream>>>((const float*)ctx->ws_misc.p, L, n_out, n_fft, hop,
                                                    istft_left(ctx, n_fft), max_hops, T.wpow, d_xout);
  SSQ_TRY(ssq_check_launch(ctx, "istft_finalize_kernel"));
  return SSQ_OK;
}

extern "C" ssq_status ssq_issq_stft_batch_f32(ssq_ctx* ctx, const float* d_Tx, int64_t channels, int64_t n_freqs,
                                              int64_t n_frames, const double* window, int64_t win_n, int n_fft,
                                              double fs, float* d_y) {
  if (!ctx) return ssq_fail(nullptr, SSQ_EINVAL, "ctx is NULL");
  if (!d_Tx || !d_y || !window || win_n < 1) return ssq_fail(ctx, SSQ_EINVAL, "NULL/empty argument");
  SSQ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (n_fft <= 0) n_fft = (int)(n_freqs - 1) * 2;
  if (n_fft < 2 || n_fft / 2 + 1 != n_freqs)
    return ssq_fail(ctx, SSQ_EINVAL, "Tx has %lld rows but n_fft=%d needs %d", (long long)n_freqs, n_fft,
                    n_fft / 2 + 1);
  if (n_frames < 1 || channels < 1) return ssq_fail(ctx, SSQ_EINVAL, "empty Tx");
  std::vector<double> wfit = ssqhost::fit_window(window, win_n, n_fft);
  const double wc = wfit[(size_t)(n_fft / 2)];
  const float scale = (float)(2.0 / (wc * fs));
  dim3 g((unsigned)((n_frames + 255) / 256), (unsigned)channels);
  SSQ_CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  issq_stft_kernel<<<g, 256, 0, ctx->stream>>>((const float2*)d_Tx, n_freqs, n_frames, scale, d_y);
  SSQ_TRY(ssq_check_launch(ctx, "issq_stft_kernel"));
  ctx->last_kernel = "issq_stft_kernel";
  SSQ_CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  ctx->ev_valid = true;
  return SSQ_OK;
}

// issq_stft with curve bands: the component inversion of issq_components_kernel (components_kernels.cuh) on a hop-1,
// modulated Tx, times the factor of ssq_issq_stft_batch_f32.  The arguments are checked before the context.
extern "C" ssq_status ssq_issq_stft_components_batch_f32(ssq_ctx* ctx, const float* d_Tx, int64_t channels,
                                                         int64_t n_freqs, int64_t n_frames, const double* window,
                                                         int64_t win_n, int n_fft, double fs, const int32_t* d_cc,
                                                         const int32_t* d_cw, int K, float* d_y) {
  if (K < 1 || K > SSQ_MAX_COMPONENTS)
    return ssq_fail(ctx, SSQ_EUNSUPPORTED, "issq_stft: %d components (1..%d supported)", K, SSQ_MAX_COMPONENTS);
  if (!ctx) return ssq_fail(nullptr, SSQ_EINVAL, "ctx is NULL");
  if (!d_Tx || !d_y || !d_cc || !d_cw || !window || win_n < 1) return ssq_fail(ctx, SSQ_EINVAL, "NULL/empty argument");
  if (n_fft <= 0) n_fft = (int)(n_freqs - 1) * 2;
  if (n_fft < 2 || n_fft / 2 + 1 != n_freqs)
    return ssq_fail(ctx, SSQ_EINVAL, "Tx has %lld rows but n_fft=%d needs %d", (long long)n_freqs, n_fft,
                    n_fft / 2 + 1);
  if (n_frames < 1 || channels < 1) return ssq_fail(ctx, SSQ_EINVAL, "empty Tx");
  if (channels > 65535) return ssq_fail(ctx, SSQ_EUNSUPPORTED, "issq_stft: %lld channels in one call", (long long)channels);
  SSQ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  std::vector<double> wfit = ssqhost::fit_window(window, win_n, n_fft);
  const float scale = (float)(2.0 / (wfit[(size_t)(n_fft / 2)] * fs));
  SSQ_CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  SSQ_TRY(issq_components_run(ctx, (const float2*)d_Tx, channels, n_freqs, n_frames, d_cc, d_cw, K, scale, d_y));
  SSQ_CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  ctx->ev_valid = true;
  return SSQ_OK;
}

// ---------------------------------------------------------------------------
// reference-typed entry points (host f64 / c128)
// ---------------------------------------------------------------------------
// ---- float64 <-> float32 at the host boundary of the *_f64 entry points ----------------------------
// The reference returns complex128 / float64 arrays; the device computes in fp32.  For one channel of
// configs[1] the result is 231 MB of complex128: a pageable copy plus a scalar conversion loop cost
// 118 ms per call against 0.1 ms of kernel time.  Chunks of 32 MB go through two pinned buffers (the
// copy of chunk i+1 overlaps the conversion of chunk i) and the conversion runs on a few host threads.
static constexpr size_t kPinFloats = (size_t)8 << 20;  // 32 MB per staging buffer

static ssq_status pin_reserve(ssq_ctx* ctx) {
  for (int i = 0; i < 2; ++i) {
    if (!ctx->pin[i]) SSQ_CUDA_TRY(ctx, cudaHostAlloc(&ctx->pin[i], kPinFloats * sizeof(float), cudaHostAllocDefault));
    if (!ctx->pin_ev[i]) SSQ_CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->pin_ev[i], cudaEventDisableTiming));
  }
  return SSQ_OK;
}

template <class Fn>
static void host_parallel_for(size_t n, Fn fn) {  // fn(begin, end) on up to 8 threads
  unsigned hw = std::thread::hardware_concurrency();
  const size_t nt = std::max<size_t>(1, std::min<size_t>({(size_t)(hw ? hw : 1), (size_t)8, n / ((size_t)1 << 18) + 1}));
  if (nt == 1) {
    fn((size_t)0, n);
    return;
  }
  std::vector<std::thread> th;
  const size_t per = (n + nt - 1) / nt;
  for (size_t t = 1; t < nt; ++t) {
    const size_t b = std::min(n, t * per), e = std::min(n, b + per);
    th.emplace_back([=] { fn(b, e); });
  }
  fn((size_t)0, std::min(n, per));
  for (auto& t : th) t.join();
}

static ssq_status upload_f64_as_f32(ssq_ctx* ctx, const double* x, size_t n, DevBuf& buf) {
  SSQ_TRY(devbuf_reserve(ctx, buf, n * sizeof(float)));
  SSQ_TRY(pin_reserve(ctx));
  size_t off = 0;
  for (int i = 0; off < n; ++i) {
    const size_t m = std::min(kPinFloats, n - off);
    float* h = (float*)ctx->pin[i & 1];
    if (i >= 2) SSQ_CUDA_TRY(ctx, cudaEventSynchronize(ctx->pin_ev[i & 1]));  // the copy that read this buffer
    const double* src = x + off;
    host_parallel_for(m, [=](size_t b, size_t e) {
      for (size_t j = b; j < e; ++j) h[j] = (float)src[j];
    });
    SSQ_CUDA_TRY(ctx, cudaMemcpyAsync((float*)buf.p + off, h, m * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    SSQ_CUDA_TRY(ctx, cudaEventRecord(ctx->pin_ev[i & 1], ctx->stream));
    off += m;
  }
  SSQ_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));  // the staging buffers are reused by the download
  return SSQ_OK;
}

static ssq_status download_f32_as_f64(ssq_ctx* ctx, const void* d, size_t n, double* out) {
  SSQ_TRY(pin_reserve(ctx));
  const float* dsrc = (const float*)d;
  const size_t nchunks = (n + kPinFloats - 1) / kPinFloats;
  auto issue = [&](size_t c) -> cudaError_t {
    const size_t off = c * kPinFloats, m = std::min(kPinFloats, n - off);
    cudaError_t e = cudaMemcpyAsync(ctx->pin[c & 1], dsrc + off, m * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
    if (e != cudaSuccess) return e;
    return cudaEventRecord(ctx->pin_ev[c & 1], ctx->stream);
  };
  if (nchunks) SSQ_CUDA_TRY(ctx, issue(0));
  for (size_t c = 0; c < nchunks; ++c) {
    SSQ_CUDA_TRY(ctx, cudaEventSynchronize(ctx->pin_ev[c & 1]));
    if (c + 1 < nchunks) SSQ_CUDA_TRY(ctx, issue(c + 1));  // into the other buffer, converted in the previous round
    const size_t off = c * kPinFloats, m = std::min(kPinFloats, n - off);
    const float* h = (const float*)ctx->pin[c & 1];
    double* dst = out + off;
    host_parallel_for(m, [=](size_t b, size_t e) {
      for (size_t j = b; j < e; ++j) dst[j] = (double)h[j];
    });
  }
  return SSQ_OK;
}

extern "C" ssq_status ssq_stft_f64(ssq_ctx* ctx, const double* x, int64_t n, int n_fft, int hop,
                                   const double* window, int64_t win_n, int padtype, double* Sx, double* freqs) {
  if (!ctx) return ssq_fail(nullptr, SSQ_EINVAL, "ctx is NULL");
  if (!x || !window || !Sx) return ssq_fail(ctx, SSQ_EINVAL, "NULL argument");
  SSQ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  int64_t n_freqs, n_frames;
  if (ssq_stft_shape(n, n_fft, hop, &n_freqs, &n_frames) != SSQ_OK)
    return ssq_fail(ctx, SSQ_EPANIC, "%s", g_tls_err.c_str());
  SSQ_TRY(upload_f64_as_f32(ctx, x, (size_t)n, ctx->ws_in));
  const size_t cnt = (size_t)n_freqs * n_frames;
  SSQ_TRY(devbuf_reserve(ctx, ctx->ws_out, cnt * sizeof(float2)));
  SSQ_TRY(ssq_stft_batch_f32(ctx, (const float*)ctx->ws_in.p, 1, n, n, window, win_n, n_fft, hop, padtype,
                             (float*)ctx->ws_out.p));
  SSQ_TRY(download_f32_as_f64(ctx, ctx->ws_out.p, cnt * 2, Sx));
  if (freqs) {
    // Array1::linspace(0.0, 0.5, n_freqs) (stft.rs:40)
    const double step = n_freqs > 1 ? 0.5 / (double)(n_freqs - 1) : 0.0;
    for (int64_t i = 0; i < n_freqs; ++i) freqs[i] = step * (double)i;
    if (n_freqs > 1) freqs[n_freqs - 1] = 0.5;
  }
  return SSQ_OK;
}

extern "C" ssq_status ssq_ssq_stft_f64(ssq_ctx* ctx, const double* x, int64_t n, const double* window,
                                       int64_t win_n, int n_fft, int win_len, int hop, double fs, int padtype,
                                       int squeezing, double gamma, unsigned flags, double* Tx, double* ssq_freqs,
                                       double* Sx, double* dSx, double* w, int32_t* kb) {
  if (!ctx) return ssq_fail(nullptr, SSQ_EINVAL, "ctx is NULL");
  if (!x || !window || !Tx || win_n < 1) return ssq_fail(ctx, SSQ_EINVAL, "NULL/empty argument");
  SSQ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (n < 1) return ssq_fail(ctx, SSQ_EPANIC, "empty x: usize underflow at ssq_stft.rs:183");
  if (n_fft <= 0) n_fft = (int)std::min<int64_t>(n, 512);
  if (win_len <= 0) win_len = (int)win_n;
  if (win_len > n_fft)
    return ssq_fail(ctx, SSQ_EINVAL, "Window length %d cannot be greater than n_fft %d", win_len, n_fft);
  if (hop < 1) return ssq_fail(ctx, SSQ_EPANIC, "hop_len=%d: division by zero at ssq_stft.rs:183", hop);
  if (n_fft < 2) return ssq_fail(ctx, SSQ_EINVAL, "n_fft=%d: need n_fft >= 2", n_fft);
  const int64_t n_freqs = n_fft / 2 + 1, n_frames = (n - 1) / hop + 1;
  const size_t cnt = (size_t)n_freqs * n_frames;
  SSQ_TRY(upload_f64_as_f32(ctx, x, (size_t)n, ctx->ws_in));
  SSQ_TRY(devbuf_reserve(ctx, ctx->ws_out, cnt * sizeof(float2)));
  StftCall c;
  c.mode = 0;
  c.d_x = (const float*)ctx->ws_in.p;
  c.channels = 1;
  c.n = n;
  c.x_stride = n;
  c.wfit = ssqhost::fit_window(window, win_n, n_fft);
  c.n_fft = n_fft;
  c.hop = hop;
  c.fs = fs;
  c.padtype = padtype;
  c.squeezing = squeezing;
  c.gamma = gamma;
  c.flags = flags;
  c.d_out = (float2*)ctx->ws_out.p;
  c.aux_Sx = nullptr;
  c.aux_dSx = nullptr;
  c.aux_w = nullptr;
  if (Sx) {
    SSQ_TRY(devbuf_reserve(ctx, ctx->ws_aux0, cnt * sizeof(float2)));
    c.aux_Sx = (float2*)ctx->ws_aux0.p;
  }
  if (dSx) {
    SSQ_TRY(devbuf_reserve(ctx, ctx->ws_aux1, cnt * sizeof(float2)));
    c.aux_dSx = (float2*)ctx->ws_aux1.p;
  }
  if (w) {
    SSQ_TRY(devbuf_reserve(ctx, ctx->ws_aux2, cnt * sizeof(float)));
    c.aux_w = (float*)ctx->ws_aux2.p;
  }
  if (kb) {
    SSQ_TRY(devbuf_reserve(ctx, ctx->ws_misc, cnt * sizeof(int)));
    c.aux_kb = (int*)ctx->ws_misc.p;
  }
  SSQ_TRY(run_stft_family(ctx, c));
  SSQ_TRY(download_f32_as_f64(ctx, ctx->ws_out.p, cnt * 2, Tx));
  if (Sx) SSQ_TRY(download_f32_as_f64(ctx, ctx->ws_aux0.p, cnt * 2, Sx));
  if (dSx) SSQ_TRY(download_f32_as_f64(ctx, ctx->ws_aux1.p, cnt * 2, dSx));
  if (w) SSQ_TRY(download_f32_as_f64(ctx, ctx->ws_aux2.p, cnt, w));
  if (kb) {
    SSQ_CUDA_TRY(ctx, cudaMemcpyAsync(kb, ctx->ws_misc.p, cnt * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SSQ_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  }
  if (ssq_freqs)  // ssq_stft.rs:42-54
    for (int64_t i = 0; i < n_freqs; ++i) ssq_freqs[i] = (double)i * 0.5 * fs / ((double)n_freqs - 1.0);
  return SSQ_OK;
}

extern "C" ssq_status ssq_istft_f64(ssq_ctx* ctx, const double* Sx, int64_t n_freqs, int64_t n_frames,
                                    const double* window, int64_t win_n, int n_fft, int hop, int64_t N,
                                    int win_exp, double* x) {
  if (!ctx) return ssq_fail(nullptr, SSQ_EINVAL, "ctx is NULL");
  if (!Sx || !window || !x) return ssq_fail(ctx, SSQ_EINVAL, "NULL argument");
  SSQ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (n_freqs < 2 || n_frames < 1 || hop < 1) return ssq_fail(ctx, SSQ_EINVAL, "bad Sx shape / hop");
  const int64_t n_out = N > 0 ? N : (int64_t)hop * n_frames;
  const size_t cnt = (size_t)n_freqs * n_frames;
  SSQ_TRY(upload_f64_as_f32(ctx, Sx, cnt * 2, ctx->ws_in));
  SSQ_TRY(devbuf_reserve(ctx, ctx->ws_out, (size_t)n_out * sizeof(float)));
  SSQ_TRY(ssq_istft_batch_f32(ctx, (const float*)ctx->ws_in.p, 1, n_freqs, n_frames, window, win_n, n_fft, hop,
                              n_out, win_exp, (float*)ctx->ws_out.p));
  return download_f32_as_f64(ctx, ctx->ws_out.p, (size_t)n_out, x);
}

extern "C" ssq_status ssq_issq_stft_f64(ssq_ctx* ctx, const double* Tx, int64_t n_freqs, int64_t n_frames,
                                        const double* window, int64_t win_n, int n_fft, int hop, double fs,
                                        double* y) {
  if (!ctx) return ssq_fail(nullptr, SSQ_EINVAL, "ctx is NULL");
  if (!Tx || !window || !y) return ssq_fail(ctx, SSQ_EINVAL, "NULL argument");
  if (hop != 1) return ssq_fail(ctx, SSQ_EINVAL, "inversion with `hop_len != 1` is unsupported.");
  SSQ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (n_freqs < 2 || n_frames < 1) return ssq_fail(ctx, SSQ_EINVAL, "bad Tx shape");
  const size_t cnt = (size_t)n_freqs * n_frames;
  SSQ_TRY(upload_f64_as_f32(ctx, Tx, cnt * 2, ctx->ws_in));
  SSQ_TRY(devbuf_reserve(ctx, ctx->ws_out, (size_t)n_frames * sizeof(float)));
  SSQ_TRY(ssq_issq_stft_batch_f32(ctx, (const float*)ctx->ws_in.p, 1, n_freqs, n_frames, window, win_n, n_fft, fs,
                                  (float*)ctx->ws_out.p));
  return download_f32_as_f64(ctx, ctx->ws_out.p, (size_t)n_frames, y);
}

extern "C" ssq_status ssq_issq_stft_components_f64(ssq_ctx* ctx, const double* Tx, int64_t n_freqs, int64_t n_frames,
                                                   const double* window, int64_t win_n, int n_fft, int hop, double fs,
                                                   const int32_t* cc, const int32_t* cw, int K, double* y) {
  if (K < 1 || K > SSQ_MAX_COMPONENTS)
    return ssq_fail(ctx, SSQ_EUNSUPPORTED, "issq_stft: %d components (1..%d supported)", K, SSQ_MAX_COMPONENTS);
  if (!ctx) return ssq_fail(nullptr, SSQ_EINVAL, "ctx is NULL");
  if (!Tx || !window || !y || !cc || !cw) return ssq_fail(ctx, SSQ_EINVAL, "NULL argument");
  if (hop != 1) return ssq_fail(ctx, SSQ_EINVAL, "inversion with `hop_len != 1` is unsupported.");
  if (n_freqs < 2 || n_frames < 1) return ssq_fail(ctx, SSQ_EINVAL, "bad Tx shape");
  SSQ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t cnt = (size_t)n_freqs * n_frames, nb = (size_t)n_frames * K;
  SSQ_TRY(upload_f64_as_f32(ctx, Tx, cnt * 2, ctx->ws_in));
  SSQ_TRY(devbuf_reserve(ctx, ctx->ws_aux0, 2 * nb * sizeof(int32_t)));
  SSQ_TRY(devbuf_reserve(ctx, ctx->ws_out, (size_t)(K + 1) * n_frames * sizeof(float)));
  int32_t* d_cc = (int32_t*)ctx->ws_aux0.p;
  int32_t* d_cw = d_cc + nb;
  SSQ_CUDA_TRY(ctx, cudaMemcpyAsync(d_cc, cc, nb * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
  SSQ_CUDA_TRY(ctx, cudaMemcpyAsync(d_cw, cw, nb * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
  SSQ_TRY(ssq_issq_stft_components_batch_f32(ctx, (const float*)ctx->ws_in.p, 1, n_freqs, n_frames, window, win_n,
                                             n_fft, fs, d_cc, d_cw, K, (float*)ctx->ws_out.p));
  return download_f32_as_f64(ctx, ctx->ws_out.p, (size_t)(K + 1) * n_frames, y);
}

// ---------------------------------------------------------------------------
// host-buffer batched path: chunked over channels, copies overlapped with
// compute on three streams (H2D | kernel | D2H).
// ---------------------------------------------------------------------------
static ssq_status stft_host_pipeline(ssq_ctx* ctx, int mode, const float* x, int64_t channels, int64_t n,
                                     const double* window, int64_t win_n, int n_fft, int hop, double fs, int padtype,
                                     int squeezing, double gamma, unsigned flags, float* Tx);

extern "C" ssq_status ssq_ssq_stft_host_f32(ssq_ctx* ctx, const float* x, int64_t channels, int64_t n,
                                            const double* window, int64_t win_n, int n_fft, int hop, double fs,
                                            int padtype, int squeezing, double gamma, unsigned flags, float* Tx) {
  return stft_host_pipeline(ctx, 0, x, channels, n, window, win_n, n_fft, hop, fs, padtype, squeezing, gamma, flags, Tx);
}

extern "C" ssq_status ssq_stft_host_f32(ssq_ctx* ctx, const float* x, int64_t channels, int64_t n, const double* window,
                                        int64_t win_n, int n_fft, int hop, int padtype, float* Sx) {
  return stft_host_pipeline(ctx, 1, x, channels, n, window, win_n, n_fft, hop, 1.0, padtype, SSQ_SQUEEZE_SUM, 0.0, 0u, Sx);
}

static ssq_status stft_host_pipeline(ssq_ctx* ctx, int mode, const float* x, int64_t channels, int64_t n,
                                     const double* window, int64_t win_n, int n_fft, int hop, double fs, int padtype,
                                     int squeezing, double gamma, unsigned flags, float* Tx) {
  if (!ctx) return ssq_fail(nullptr, SSQ_EINVAL, "ctx is NULL");
  if (!x || !Tx || !window) return ssq_fail(ctx, SSQ_EINVAL, "NULL argument");
  SSQ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (n_fft <= 0) n_fft = (int)std::min<int64_t>(n, 512);
  int64_t n_freqs, n_frames;
  if (ssq_stft_shape(n, n_fft, hop, &n_freqs, &n_frames) != SSQ_OK)
    return ssq_fail(ctx, SSQ_EPANIC, "%s", g_tls_err.c_str());
  const size_t out_per_ch = (size_t)n_freqs * n_frames * sizeof(float2);
  const size_t in_per_ch = (size_t)n * sizeof(float);
  // chunk so that two output chunks stay below ~8 GiB of device memory
  int64_t chunk = std::max<int64_t>(1, (int64_t)(((size_t)4 << 30) / std::max<size_t>(1, out_per_ch)));
  chunk = std::min(chunk, channels);
  SSQ_TRY(devbuf_reserve(ctx, ctx->ws_in, 2 * chunk * in_per_ch));
  SSQ_TRY(devbuf_reserve(ctx, ctx->ws_out, 2 * chunk * out_per_ch));
  cudaStream_t s_in = nullptr, s_out = nullptr;
  cudaEvent_t e_in[2] = {nullptr, nullptr}, e_k[2] = {nullptr, nullptr}, e_out[2] = {nullptr, nullptr};
  SSQ_CUDA_TRY(ctx, cudaStreamCreateWithFlags(&s_in, cudaStreamNonBlocking));
  SSQ_CUDA_TRY(ctx, cudaStreamCreateWithFlags(&s_out, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) {
    cudaEventCreateWithFlags(&e_in[i], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&e_k[i], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&e_out[i], cudaEventDisableTiming);
  }
  ssq_status st = SSQ_OK;
  int it = 0;
  for (int64_t c0 = 0; c0 < channels && st == SSQ_OK; c0 += chunk, ++it) {
    const int b = it & 1;
    const int64_t cc = std::min(chunk, channels - c0);
    float* din = (float*)ctx->ws_in.p + (size_t)b * chunk * n;
    char* dout = (char*)ctx->ws_out.p + (size_t)b * chunk * out_per_ch;
    // the kernel that last read this input slot / the copy that last drained this output slot
    if (it >= 2) {
      cudaStreamWaitEvent(s_in, e_k[b], 0);
      cudaStreamWaitEvent(ctx->stream, e_out[b], 0);
    }
    cudaMemcpyAsync(din, x + (size_t)c0 * n, (size_t)cc * in_per_ch, cudaMemcpyHostToDevice, s_in);
    cudaEventRecord(e_in[b], s_in);
    cudaStreamWaitEvent(ctx->stream, e_in[b], 0);
    st = mode == 0 ? ssq_ssq_stft_batch_f32(ctx, din, cc, n, n, window, win_n, n_fft, hop, fs, padtype, squeezing, gamma,
                                            flags, (float*)dout)
                   : ssq_stft_batch_f32(ctx, din, cc, n, n, window, win_n, n_fft, hop, padtype, (float*)dout);
    if (st != SSQ_OK) break;
    cudaEventRecord(e_k[b], ctx->stream);
    cudaStreamWaitEvent(s_out, e_k[b], 0);
    cudaMemcpyAsync((char*)Tx + (size_t)c0 * out_per_ch, dout, (size_t)cc * out_per_ch, cudaMemcpyDeviceToHost,
                    s_out);
    cudaEventRecord(e_out[b], s_out);
  }
  cudaStreamSynchronize(s_in);
  cudaStreamSynchronize(ctx->stream);
  cudaStreamSynchronize(s_out);
  cudaError_t e = cudaGetLastError();
  for (int i = 0; i < 2; ++i) {
    cudaEventDestroy(e_in[i]);
    cudaEventDestroy(e_k[i]);
    cudaEventDestroy(e_out[i]);
  }
  cudaStreamDestroy(s_in);
  cudaStreamDestroy(s_out);
  if (st != SSQ_OK) return st;
  if (e != cudaSuccess) return ssq_fail(ctx, SSQ_ECUDA, "host-buffer pipeline: %s", cudaGetErrorString(e));
  return SSQ_OK;
}

// ===========================================================================
// Streaming ssq_stft over a long recording delivered in chunks of interleaved
// [samples, channels] int16 / float32 (SURVEY 8f rank 1: replaces the dask
// map_overlap caller of tests/stft_ssq_test.py:218-283).  Exact at chunk seams:
// a frame is computed once every real sample it covers has arrived, padding
// exists only at the two ends of the recording (the reference's caller re-pads
// every chunk).  Concatenating the per-push outputs along frames equals the
// whole-signal transform bit for bit.
// ===========================================================================
struct ssq_stream {
  ssq_ctx* ctx;
  int64_t channels, n_total, max_chunk, cap;
  std::vector<double> wfit;
  int n_fft, hop, left, padtype, squeezing;
  int mode = 0;        // 0 ssq_stft, 1 stft, 2 cwt, 3 ssq_cwt (ssq_stream_create_cwt, cwt_host.inl)
  unsigned flags = 0;  // SSQ_FLAG_MODULATED (ssq_stft), SSQ_FLAG_L2_NORM (cwt), SSQ_FLAG_NO_FLIPUD (ssq_cwt)
  double fs, gamma;
  // CWT modes: frames are output columns, computed in blocks of `block` columns with `overlap` samples of context on
  // either side (DESIGN §3.6b)
  int64_t block = 0, overlap = 0, pitch_bound = 0;
  int wavelet = 0, freq_dist = 0, maprange = 0;
  std::vector<double> scales;
  double dt = 1.0;
  int64_t n_frames_total;
  int64_t received = 0;   // samples pushed so far
  int64_t origin = 0;     // global index of buf[.][0]
  int64_t f_next = 0;     // next frame to compute
  float* buf[2] = {nullptr, nullptr};  // [channels, cap] ping-pong (tail carried over by a D2D copy)
  int cur = 0;
};

template <typename T>
__global__ void deinterleave_kernel(const T* __restrict__ in, int64_t n_new, int64_t channels, float scale,
                                    float* __restrict__ out, int64_t cap, int64_t pos) {
  // in [n_new, channels] (channels fastest) -> out[ch * cap + pos + i]; 32 x 32 tile transpose
  __shared__ float tile[32][33];
  const int64_t i0 = (int64_t)blockIdx.x * 32, c0 = (int64_t)blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int64_t i = i0 + r, c = c0 + threadIdx.x;
    tile[r][threadIdx.x] = (i < n_new && c < channels) ? (float)in[i * channels + c] * scale : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int64_t c = c0 + r, i = i0 + threadIdx.x;
    if (c < channels && i < n_new) out[c * cap + pos + i] = tile[threadIdx.x][r];
  }
}

static int64_t stream_frames_ready(const ssq_stream* s, int64_t received) {
  if (received >= s->n_total) return s->n_frames_total;
  if (s->mode >= 2) {  // block b is ready once min(N, (b + 1) C + d) samples have arrived
    const int64_t r = received - s->overlap;
    return r < s->block ? 0 : r / s->block * s->block;
  }
  const int64_t a = received - s->n_fft + s->left;  // last frame f with f*hop - left + n_fft - 1 < received
  // frame 0 also reads x[left] through the left reflection: in upstream framing with even n_fft that is one sample
  // past its own last one (left = n_fft - left), so with received == left it is not ready yet
  if (a < 0 || received <= s->left) return 0;
  return std::min<int64_t>(s->n_frames_total, a / s->hop + 1);
}

// The two [channels, cap] carry-over buffers of a new stream; on failure the stream is destroyed.
static ssq_status stream_buffers(ssq_stream* s) {
  ssq_ctx* ctx = s->ctx;
  for (int i = 0; i < 2; ++i) {
    cudaError_t e = cudaMalloc((void**)&s->buf[i], (size_t)s->channels * s->cap * sizeof(float));
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      if (s->buf[0]) cudaFree(s->buf[0]);
      const long long ch = (long long)s->channels, cap = (long long)s->cap;
      delete s;
      return ssq_fail(ctx, SSQ_ENOMEM, "stream buffers (%lld x %lld floats): %s", ch, cap, cudaGetErrorString(e));
    }
  }
  // stft mode pairs frames in one complex FFT: the partner of the last ready frame reads samples not received yet.
  // Its values only reach the real frame through the rounding of the split, unless they are huge or NaN, which
  // never-written device memory (freed by an earlier user in this process) can hold.
  for (int i = 0; i < 2; ++i) {
    cudaError_t e = cudaMemsetAsync(s->buf[i], 0, (size_t)s->channels * s->cap * sizeof(float), ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
      ssq_stream_destroy(s);
      return ssq_fail(ctx, SSQ_ECUDA, "stream buffers: %s", cudaGetErrorString(e));
    }
  }
  return SSQ_OK;
}

extern "C" ssq_status ssq_stream_create(ssq_ctx* ctx, int64_t channels, int64_t n_total, int64_t max_chunk,
                                        const double* window, int64_t win_n, int n_fft, int hop, double fs,
                                        int padtype, int squeezing, double gamma, ssq_stream** out) {
  return ssq_stream_create_ex(ctx, channels, n_total, max_chunk, window, win_n, n_fft, hop, fs, padtype, squeezing, gamma,
                              0, 0u, out);
}

extern "C" ssq_status ssq_stream_create_ex(ssq_ctx* ctx, int64_t channels, int64_t n_total, int64_t max_chunk,
                                           const double* window, int64_t win_n, int n_fft, int hop, double fs,
                                           int padtype, int squeezing, double gamma, int mode, unsigned flags,
                                           ssq_stream** out) {
  if (!ctx) return ssq_fail(nullptr, SSQ_EINVAL, "ctx is NULL");
  if (mode != 0 && mode != 1) return ssq_fail(ctx, SSQ_EINVAL, "stream mode must be 0 (ssq_stft) or 1 (stft)");
  if (!out || !window || win_n < 1) return ssq_fail(ctx, SSQ_EINVAL, "NULL/empty argument");
  *out = nullptr;
  if (channels < 1 || n_total < 1 || max_chunk < 1) return ssq_fail(ctx, SSQ_EINVAL, "bad channels/n_total/max_chunk");
  if (n_fft <= 0) n_fft = (int)std::min<int64_t>(n_total, 512);
  if (n_fft < 2 || hop < 1) return ssq_fail(ctx, SSQ_EINVAL, "bad n_fft/hop");
  if (mode == 0 && win_n > n_fft)
    return ssq_fail(ctx, SSQ_EINVAL, "Window length %lld cannot be greater than n_fft %d", (long long)win_n, n_fft);
  SSQ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  ssq_stream* s = new (std::nothrow) ssq_stream();
  if (!s) return ssq_fail(ctx, SSQ_ENOMEM, "out of host memory");
  s->ctx = ctx;
  s->channels = channels;
  s->n_total = n_total;
  s->max_chunk = max_chunk;
  if (mode == 1) {  // stft takes the first n_fft taps and panics on a shorter window (stft_utils.rs:8, stft.rs:67)
    if (win_n < n_fft) {
      delete s;
      return ssq_fail(ctx, SSQ_EPANIC, "window length %lld < n_fft %d: the reference panics in rustfft (stft_utils.rs:8, stft.rs:67)",
                      (long long)win_n, n_fft);
    }
    s->wfit.assign(window, window + n_fft);
  } else {
    s->wfit = ssqhost::fit_window(window, win_n, n_fft);
  }
  s->mode = mode;
  s->flags = mode == 0 ? (flags & SSQ_FLAG_MODULATED) : 0u;
  s->n_fft = n_fft;
  s->hop = hop;
  s->left = ctx->opt.upstream_framing ? n_fft / 2 : (n_fft - 1) / 2;
  s->padtype = padtype;
  s->squeezing = squeezing;
  s->fs = fs;
  s->gamma = gamma;
  s->n_frames_total = (n_total - 1) / hop + 1;
  s->cap = max_chunk + n_fft + hop + 32;
  SSQ_TRY(stream_buffers(s));
  *out = s;
  return SSQ_OK;
}

extern "C" void ssq_stream_destroy(ssq_stream* s) {
  if (!s) return;
  cudaSetDevice(s->ctx->device);
  cudaStreamSynchronize(s->ctx->stream);
  for (int i = 0; i < 2; ++i)
    if (s->buf[i]) cudaFree(s->buf[i]);
  delete s;
}

extern "C" int64_t ssq_stream_total_frames(const ssq_stream* s) { return s ? s->n_frames_total : 0; }

extern "C" int64_t ssq_stream_frames_after(const ssq_stream* s, int64_t n_new) {
  if (!s || n_new < 0) return 0;
  const int64_t r = std::min<int64_t>(s->n_total, s->received + n_new);
  return stream_frames_ready(s, r) - s->f_next;
}

static ssq_status cwt_stream_run(ssq_stream* s, const float* buf, int64_t c0, int64_t c1, float2* out);  // cwt_host.inl

template <typename T>
static ssq_status stream_push(ssq_stream* s, const T* d_chunk, int64_t n_new, float scale, float* d_Tx,
                              int64_t* frames_written) {
  if (!s) return ssq_fail(nullptr, SSQ_EINVAL, "stream is NULL");
  ssq_ctx* ctx = s->ctx;
  if (frames_written) *frames_written = 0;
  if (n_new < 0 || n_new > s->max_chunk) return ssq_fail(ctx, SSQ_EINVAL, "chunk of %lld samples (max %lld)", (long long)n_new, (long long)s->max_chunk);
  if (s->received + n_new > s->n_total) return ssq_fail(ctx, SSQ_EINVAL, "more samples pushed than n_total");
  if (n_new > 0 && !d_chunk) return ssq_fail(ctx, SSQ_EINVAL, "chunk is NULL");
  SSQ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const int64_t have = s->received - s->origin;
  if (have + n_new > s->cap) return ssq_fail(ctx, SSQ_EINVAL, "internal: stream buffer overflow");
  float* buf = s->buf[s->cur];
  // hop > n_fft: the buffer origin (start of the next frame) can lie beyond the samples received so far;
  // the samples in between belong to no frame and are dropped here instead of being written before buf
  const int64_t skip = std::min<int64_t>(n_new, std::max<int64_t>(0, -have));
  if (n_new - skip > 0) {
    const int64_t m = n_new - skip;
    dim3 g((unsigned)((m + 31) / 32), (unsigned)((s->channels + 31) / 32)), b(32, 8);
    deinterleave_kernel<T><<<g, b, 0, ctx->stream>>>(d_chunk + skip * s->channels, m, s->channels, scale, buf, s->cap,
                                                     have + skip);
    SSQ_TRY(ssq_check_launch(ctx, "deinterleave_kernel"));
  }
  s->received += n_new;
  const int64_t f_end = stream_frames_ready(s, s->received);
  const int64_t count = f_end - s->f_next;
  if (count > 0) {
    if (!d_Tx) return ssq_fail(ctx, SSQ_EINVAL, "d_Tx is NULL but %lld frames are ready", (long long)count);
    if (s->mode >= 2) {
      SSQ_TRY(cwt_stream_run(s, buf, s->f_next, f_end, (float2*)d_Tx));
    } else {
      StftCall c;
      c.mode = s->mode;
      c.d_x = buf;
      c.x_origin = s->origin;
      c.channels = s->channels;
      c.n = s->n_total;
      c.x_stride = s->cap;
      c.wfit = s->wfit;
      c.n_fft = s->n_fft;
      c.hop = s->hop;
      c.fs = s->mode == 1 ? 1.0 : s->fs;
      c.padtype = s->padtype;
      c.squeezing = s->mode == 1 ? SSQ_SQUEEZE_SUM : s->squeezing;
      c.gamma = s->mode == 1 ? 0.0 : s->gamma;
      c.flags = s->flags;
      c.d_out = (float2*)d_Tx;
      c.aux_Sx = nullptr;
      c.aux_dSx = nullptr;
      c.aux_w = nullptr;
      c.frame0 = s->f_next;
      c.n_frames_call = count;
      SSQ_TRY(run_stft_family(ctx, c));
    }
    s->f_next = f_end;
  }
  if (frames_written) *frames_written = std::max<int64_t>(count, 0);
  // carry over the samples the next frame still needs
  if (s->f_next < s->n_frames_total) {
    // the next frame starts at f_next*hop - left; frames that touch the right padding also read the
    // reflected samples x[2n-2-o] >= n - n_fft, which may lie before their own start when hop is large
    // (CWT: the next block reads x~[f_next - d, ...); its reflections at the recording ends lie inside that range)
    const int64_t want = s->mode >= 2 ? std::max<int64_t>(0, s->f_next - s->overlap)
                                      : std::min<int64_t>(std::max<int64_t>(0, s->f_next * s->hop - s->left),
                                                          std::max<int64_t>(0, s->n_total - s->n_fft));
    const int64_t new_origin = std::max<int64_t>(s->origin, want);
    if (new_origin > s->origin) {
      const int64_t keep = s->received - new_origin;
      float* nb = s->buf[s->cur ^ 1];
      if (keep > 0)
        SSQ_CUDA_TRY(ctx, cudaMemcpy2DAsync(nb, (size_t)s->cap * sizeof(float), buf + (new_origin - s->origin),
                                            (size_t)s->cap * sizeof(float), (size_t)keep * sizeof(float),
                                            (size_t)s->channels, cudaMemcpyDeviceToDevice, ctx->stream));
      s->cur ^= 1;
      s->origin = new_origin;
    }
  }
  return SSQ_OK;
}

extern "C" ssq_status ssq_stream_push_i16(ssq_stream* s, const int16_t* d_chunk, int64_t n_new, float scale,
                                          float* d_Tx, int64_t* frames_written) {
  return stream_push<int16_t>(s, d_chunk, n_new, scale, d_Tx, frames_written);
}
extern "C" ssq_status ssq_stream_push_f32(ssq_stream* s, const float* d_chunk, int64_t n_new, float scale,
                                          float* d_Tx, int64_t* frames_written) {
  return stream_push<float>(s, d_chunk, n_new, scale, d_Tx, frames_written);
}

// ---------------------------------------------------------------------------
// Host-side feeder of a stream (SURVEY 8f rank 1, the reader half): the recording lies in HOST memory -- typically a
// memory-mapped (samples, channels) int16 .dat / .bin file as the reference's scripts open them
// (tests/stft_ssq_test.py:218-283, tests/stft_test.py:374-377), i.e. pageable memory.  A ring of `depth` pinned
// staging buffers and device chunk buffers decouples the three stages: the host copy (and page-in) of chunk i+1 into
// its pinned slot runs while chunk i crosses PCIe on a copy stream and chunk i-1 is transformed on the context's
// stream.  ssq_feeder_push returns as soon as the work is queued; the caller's d_Tx is written in stream order.
// ---------------------------------------------------------------------------
struct ssq_feeder {
  ssq_stream* s = nullptr;
  int dtype = 0;  // 0 int16, 1 float32
  int depth = 2;
  size_t elem = 2, slot_bytes = 0;
  std::vector<void*> pinned, dev;
  std::vector<cudaEvent_t> copied, consumed;  // H2D of the slot done / the de-interleave kernel has read the slot
  std::vector<char> used;
  cudaStream_t copy_stream = nullptr;
  int64_t pushes = 0;
};

extern "C" void ssq_feeder_destroy(ssq_feeder* f) {
  if (!f) return;
  if (f->s) cudaSetDevice(f->s->ctx->device);
  if (f->copy_stream) cudaStreamSynchronize(f->copy_stream);
  if (f->s) cudaStreamSynchronize(f->s->ctx->stream);
  for (void* p : f->pinned)
    if (p) cudaFreeHost(p);
  for (void* p : f->dev)
    if (p) cudaFree(p);
  for (cudaEvent_t e : f->copied)
    if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : f->consumed)
    if (e) cudaEventDestroy(e);
  if (f->copy_stream) cudaStreamDestroy(f->copy_stream);
  delete f;
}

extern "C" ssq_status ssq_feeder_create(ssq_stream* s, int dtype, int depth, ssq_feeder** out) {
  if (!s || !out) return ssq_fail(s ? s->ctx : nullptr, SSQ_EINVAL, "ssq_feeder_create: NULL argument");
  *out = nullptr;
  ssq_ctx* ctx = s->ctx;
  if (dtype != 0 && dtype != 1) return ssq_fail(ctx, SSQ_EINVAL, "feeder dtype must be 0 (int16) or 1 (float32)");
  if (depth < 2) depth = 2;
  if (depth > 8) depth = 8;
  SSQ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  ssq_feeder* f = new (std::nothrow) ssq_feeder();
  if (!f) return ssq_fail(ctx, SSQ_ENOMEM, "out of host memory");
  f->s = s;
  f->dtype = dtype;
  f->depth = depth;
  f->elem = dtype == 0 ? sizeof(int16_t) : sizeof(float);
  f->slot_bytes = (size_t)s->max_chunk * (size_t)s->channels * f->elem;
  f->pinned.assign(depth, nullptr);
  f->dev.assign(depth, nullptr);
  f->copied.assign(depth, nullptr);
  f->consumed.assign(depth, nullptr);
  f->used.assign(depth, 0);
  cudaError_t e = cudaStreamCreateWithFlags(&f->copy_stream, cudaStreamNonBlocking);
  for (int i = 0; i < depth && e == cudaSuccess; ++i) {
    if ((e = cudaHostAlloc(&f->pinned[i], f->slot_bytes, cudaHostAllocDefault)) != cudaSuccess) break;
    if ((e = cudaMalloc(&f->dev[i], f->slot_bytes)) != cudaSuccess) break;
    if ((e = cudaEventCreateWithFlags(&f->copied[i], cudaEventDisableTiming)) != cudaSuccess) break;
    if ((e = cudaEventCreateWithFlags(&f->consumed[i], cudaEventDisableTiming)) != cudaSuccess) break;
  }
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    const size_t slot_bytes = f->slot_bytes;
    ssq_feeder_destroy(f);
    return ssq_fail(ctx, e == cudaErrorMemoryAllocation ? SSQ_ENOMEM : SSQ_ECUDA, "feeder buffers (%d x %zu B): %s", depth,
                    slot_bytes, cudaGetErrorString(e));
  }
  *out = f;
  return SSQ_OK;
}

extern "C" ssq_status ssq_feeder_push(ssq_feeder* f, const void* h_chunk, int64_t n_new, float scale, float* d_Tx,
                                      int64_t* frames_written) {
  if (!f) return ssq_fail(nullptr, SSQ_EINVAL, "feeder is NULL");
  ssq_stream* s = f->s;
  ssq_ctx* ctx = s->ctx;
  if (frames_written) *frames_written = 0;
  if (n_new < 0 || n_new > s->max_chunk)
    return ssq_fail(ctx, SSQ_EINVAL, "chunk of %lld samples (max %lld)", (long long)n_new, (long long)s->max_chunk);
  if (n_new > 0 && !h_chunk) return ssq_fail(ctx, SSQ_EINVAL, "chunk is NULL");
  SSQ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const int slot = (int)(f->pushes % f->depth);
  const size_t bytes = (size_t)n_new * (size_t)s->channels * f->elem;
  if (f->used[slot]) {
    // the pinned slot may be overwritten once its H2D copy has completed, the device slot once the kernel that
    // read it has run (ordered on the copy stream, no host wait)
    SSQ_CUDA_TRY(ctx, cudaEventSynchronize(f->copied[slot]));
    SSQ_CUDA_TRY(ctx, cudaStreamWaitEvent(f->copy_stream, f->consumed[slot], 0));
  }
  if (bytes) {
    // pageable (memory-mapped) source: this is where the file is read; large chunks on several host threads (one
    // thread copies ~10 GB/s, the GPU consumes int16 samples faster than that)
    char* dstp = (char*)f->pinned[slot];
    const char* srcp = (const char*)h_chunk;
    if (bytes >= ((size_t)8 << 20)) host_parallel_for(bytes, [=](size_t b, size_t e) { memcpy(dstp + b, srcp + b, e - b); });
    else memcpy(dstp, srcp, bytes);
    SSQ_CUDA_TRY(ctx, cudaMemcpyAsync(f->dev[slot], f->pinned[slot], bytes, cudaMemcpyHostToDevice, f->copy_stream));
  }
  SSQ_CUDA_TRY(ctx, cudaEventRecord(f->copied[slot], f->copy_stream));
  SSQ_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, f->copied[slot], 0));
  ssq_status st = f->dtype == 0
                      ? stream_push<int16_t>(s, (const int16_t*)f->dev[slot], n_new, scale, d_Tx, frames_written)
                      : stream_push<float>(s, (const float*)f->dev[slot], n_new, scale, d_Tx, frames_written);
  // the slot is marked used whatever the transform returned: its H2D copy is in flight either way
  const cudaError_t er = cudaEventRecord(f->consumed[slot], ctx->stream);
  f->used[slot] = 1;
  f->pushes++;
  if (st == SSQ_OK && er != cudaSuccess) return ssq_fail(ctx, SSQ_ECUDA, "cudaEventRecord: %s", cudaGetErrorString(er));
  return st;
}

// ===========================================================================
// Streaming inverse (DESIGN §3.4c): istft / issq_stft over chunks of frames, the inverse of ssq_stream_*.
// istft: padded position p = f * hop + m of frame f belongs to output p - left.  Once r of the used frames (those
// below n_use = min(n_frames_total, max_hops), the batch call's clamp) have arrived, every p < r * hop is final; the
// positions the next frames still reach keep their undivided partial sums in a carry of at most n_fft - hop samples
// per channel.  issq_stft: output j is frame j, final at once.
// ===========================================================================
struct ssq_istream {
  ssq_ctx* ctx;
  int64_t channels, n_frames_total, n_out, max_frames;
  std::vector<double> wfit;
  int n_fft, hop, win_exp, mode, out_format, left;
  int64_t max_hops, n_use;
  float issq_scale;          // mode 1: 2 / (w[n_fft/2] fs), as ssq_issq_stft_batch_f32
  float inv_scale;           // (float)(1.0 / scale) of the creation
  int64_t received = 0;      // frames pushed
  int64_t emitted = 0;       // samples written
  int64_t clen = 0;          // valid samples of carry[cur]
  int64_t cstride = 1;       // max(1, n_fft - hop)
  float* acc = nullptr;      // [channels, (max_frames - 1) * hop + n_fft]: this push's overlap-add
  float* carry[2] = {nullptr, nullptr};
  int cur = 0;
};

// samples final once `frames` frames have been pushed
static int64_t istream_ready(const ssq_istream* s, int64_t frames) {
  if (s->mode == 1) return std::min(frames, s->n_out);
  const int64_t r = std::min(frames, s->n_use);
  if (r >= s->n_use) return s->n_out;
  return std::min<int64_t>(s->n_out, std::max<int64_t>(0, r * s->hop - s->left));
}

extern "C" void ssq_istream_destroy(ssq_istream* s) {
  if (!s) return;
  cudaSetDevice(s->ctx->device);
  cudaStreamSynchronize(s->ctx->stream);
  if (s->acc) cudaFree(s->acc);
  for (int i = 0; i < 2; ++i)
    if (s->carry[i]) cudaFree(s->carry[i]);
  delete s;
}

extern "C" ssq_status ssq_istream_create(ssq_ctx* ctx, int64_t channels, int64_t n_frames_total, int64_t n_out,
                                         int64_t max_frames, const double* window, int64_t win_n, int n_fft, int hop,
                                         int win_exp, int mode, double fs, int out_format, ssq_istream** out) {
  // argument checks first, all on the host: they need neither a context nor a device
  if (!out) return ssq_fail(ctx, SSQ_EINVAL, "ssq_istream_create: out is NULL");
  *out = nullptr;
  if (mode != 0 && mode != 1)
    return ssq_fail(ctx, SSQ_EINVAL, "istream mode %d: must be 0 (istft) or 1 (issq_stft)", mode);
  if (out_format < ISTREAM_F32 || out_format > ISTREAM_I16_INTERLEAVED)
    return ssq_fail(ctx, SSQ_EINVAL,
                    "istream out_format %d: must be 0 (fp32 [channels, samples]), 1 (fp32 [samples, channels]) or "
                    "2 (int16 [samples, channels])",
                    out_format);
  if (!window || win_n < 1) return ssq_fail(ctx, SSQ_EINVAL, "istream: NULL/empty window");
  if (channels < 1 || channels > 65535 || n_frames_total < 1 || max_frames < 1 || n_fft < 2 || hop < 1 ||
      win_exp < 0)
    return ssq_fail(ctx, SSQ_EINVAL,
                    "istream: bad sizes (channels=%lld in [1, 65535], n_frames_total=%lld, max_frames=%lld, n_fft=%d, "
                    "hop=%d, win_exp=%d)",
                    (long long)channels, (long long)n_frames_total, (long long)max_frames, n_fft, hop, win_exp);
  if (mode == 1 && hop != 1)
    return ssq_fail(ctx, SSQ_EINVAL, "istream issq_stft: inversion with `hop_len != 1` is unsupported (hop=%d)", hop);
  if (mode == 1 && n_out > 0 && n_out != n_frames_total)
    return ssq_fail(ctx, SSQ_EINVAL, "istream issq_stft: n_out=%lld, but issq_stft returns one sample per frame (%lld)",
                    (long long)n_out, (long long)n_frames_total);
  if (mode == 1 && !(fs > 0.0)) return ssq_fail(ctx, SSQ_EINVAL, "istream issq_stft: fs must be > 0");
  if (!ctx) return ssq_fail(nullptr, SSQ_EINVAL, "ctx is NULL");
  SSQ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  ssq_istream* s = new (std::nothrow) ssq_istream();
  if (!s) return ssq_fail(ctx, SSQ_ENOMEM, "out of host memory");
  s->ctx = ctx;
  s->channels = channels;
  s->n_frames_total = n_frames_total;
  s->n_out = n_out > 0 ? n_out : (int64_t)hop * n_frames_total;  // _stft.py:231
  s->max_frames = max_frames;
  s->wfit = ssqhost::fit_window(window, win_n, n_fft);
  s->n_fft = n_fft;
  s->hop = hop;
  s->win_exp = win_exp;
  s->mode = mode;
  s->out_format = out_format;
  s->left = istft_left(ctx, n_fft);
  s->max_hops = (s->n_out - 1) / hop + 1;  // (L - n_fft) / hop + 1 with L = n_out + n_fft - 1
  s->n_use = std::min(n_frames_total, s->max_hops);
  s->issq_scale = (float)(2.0 / (s->wfit[(size_t)(n_fft / 2)] * fs));
  s->inv_scale = 1.f;
  s->cstride = std::max(1, n_fft - hop);
  if (mode == 0) {
    const int64_t la = (std::min(max_frames, s->n_use) - 1) * hop + n_fft;
    cudaError_t e = cudaMalloc((void**)&s->acc, (size_t)channels * la * sizeof(float));
    for (int i = 0; i < 2 && e == cudaSuccess; ++i)
      e = cudaMalloc((void**)&s->carry[i], (size_t)channels * s->cstride * sizeof(float));
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      ssq_istream_destroy(s);
      return ssq_fail(ctx, SSQ_ENOMEM, "istream buffers (%lld x %lld floats): %s", (long long)channels, (long long)la,
                      cudaGetErrorString(e));
    }
  }
  *out = s;
  return SSQ_OK;
}

extern "C" int64_t ssq_istream_total_samples(const ssq_istream* s) { return s ? s->n_out : 0; }

extern "C" int64_t ssq_istream_samples_after(const ssq_istream* s, int64_t n_new) {
  if (!s || n_new < 0) return 0;
  return istream_ready(s, std::min(s->n_frames_total, s->received + n_new)) - s->emitted;
}

extern "C" ssq_status ssq_istream_push(ssq_istream* s, const float* d_Sx, int64_t n_new, float scale, void* d_out,
                                       int64_t* samples_written) {
  if (!s) return ssq_fail(nullptr, SSQ_EINVAL, "istream is NULL");
  ssq_ctx* ctx = s->ctx;
  if (samples_written) *samples_written = 0;
  // every check before the first change of state: a refused push leaves the stream as it was
  if (n_new < 0 || n_new > s->max_frames)
    return ssq_fail(ctx, SSQ_EINVAL, "push of %lld frames (max_frames %lld)", (long long)n_new, (long long)s->max_frames);
  if (s->received + n_new > s->n_frames_total)
    return ssq_fail(ctx, SSQ_EINVAL, "push of %lld frames after %lld: more frames than n_frames_total (%lld)",
                    (long long)n_new, (long long)s->received, (long long)s->n_frames_total);
  if (n_new > 0 && !d_Sx) return ssq_fail(ctx, SSQ_EINVAL, "d_Sx is NULL");
  if (!(scale != 0.f) || !std::isfinite(scale)) return ssq_fail(ctx, SSQ_EINVAL, "scale must be finite and non-zero");
  const int64_t n_emit = istream_ready(s, s->received + n_new) - s->emitted;
  if (n_emit > 0 && !d_out)
    return ssq_fail(ctx, SSQ_EINVAL, "d_out is NULL but %lld samples are ready", (long long)n_emit);
  SSQ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const float inv_scale = (float)(1.0 / (double)scale);
  const int64_t n_freqs = s->n_fft / 2 + 1;
  const dim3 blk(32, 8);
  const unsigned gy = (unsigned)((s->channels + 31) / 32);
  if (s->mode == 1) {
    if (n_new > 0) {
      dim3 g((unsigned)((n_new + 31) / 32), gy);
      SSQ_CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
      const float2* Tx = (const float2*)d_Sx;
      if (s->out_format == ISTREAM_F32)
        istream_issq_kernel<ISTREAM_F32><<<g, blk, 0, ctx->stream>>>(Tx, s->channels, n_freqs, n_new, s->issq_scale,
                                                                      inv_scale, d_out);
      else if (s->out_format == ISTREAM_F32_INTERLEAVED)
        istream_issq_kernel<ISTREAM_F32_INTERLEAVED><<<g, blk, 0, ctx->stream>>>(Tx, s->channels, n_freqs, n_new,
                                                                                  s->issq_scale, inv_scale, d_out);
      else
        istream_issq_kernel<ISTREAM_I16_INTERLEAVED><<<g, blk, 0, ctx->stream>>>(Tx, s->channels, n_freqs, n_new,
                                                                                  s->issq_scale, inv_scale, d_out);
      SSQ_TRY(ssq_check_launch(ctx, "istream_issq_kernel"));
      ctx->last_kernel = "istream_issq_kernel";
      SSQ_CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
      ctx->ev_valid = true;
    }
    s->received += n_new;
    s->emitted += n_emit;
    if (samples_written) *samples_written = n_emit;
    return SSQ_OK;
  }
  // frames of this push that the batch call would use; the rest (beyond max_hops) are dropped as it drops them
  const int64_t u = std::max<int64_t>(0, std::min(n_new, s->n_use - s->received));
  if (u > 0) {
    StftTables T;  // re-checked every push: a batch call in between may have replaced the context's tables
    SSQ_TRY(stft_tables(ctx, s->wfit, TAB_ISTFT, s->win_exp, &T));
    const int64_t La = (u - 1) * s->hop + s->n_fft;
    SSQ_CUDA_TRY(ctx, cudaMemsetAsync(s->acc, 0, (size_t)s->channels * La * sizeof(float), ctx->stream));
    SSQ_TRY(istft_ola_run(ctx, (const float2*)d_Sx, s->channels, n_freqs, n_new, u, s->n_fft, s->hop, T, s->acc, La));
    IstreamFinParams P;
    memset(&P, 0, sizeof(P));
    P.A = s->acc;
    P.La = La;
    P.Cin = s->carry[s->cur];
    P.Cout = s->carry[s->cur ^ 1];
    P.cstride = s->cstride;
    P.clen_in = s->clen;
    P.clen_out = s->received + u < s->n_use ? std::max(0, s->n_fft - s->hop) : 0;
    P.q_carry = u * s->hop;
    P.channels = s->channels;
    P.n_emit = n_emit;
    P.base = s->received * s->hop;
    P.q0 = s->emitted + s->left - P.base;  // >= 0: earlier pushes emitted exactly the positions below base
    P.n_fft = s->n_fft;
    P.hop = s->hop;
    P.max_hops = s->max_hops;
    P.wpow = T.wpow;
    P.inv_scale = inv_scale;
    P.out = d_out;
    P.nb_out = (int)((n_emit + ISTREAM_TILE - 1) / ISTREAM_TILE);
    const int64_t nb = P.nb_out + (P.clen_out + ISTREAM_TILE - 1) / ISTREAM_TILE;
    if (nb > 0) {
      dim3 g((unsigned)nb, gy);
      if (s->out_format == ISTREAM_F32)
        istream_finalize_kernel<ISTREAM_F32><<<g, blk, 0, ctx->stream>>>(P);
      else if (s->out_format == ISTREAM_F32_INTERLEAVED)
        istream_finalize_kernel<ISTREAM_F32_INTERLEAVED><<<g, blk, 0, ctx->stream>>>(P);
      else
        istream_finalize_kernel<ISTREAM_I16_INTERLEAVED><<<g, blk, 0, ctx->stream>>>(P);
      SSQ_TRY(ssq_check_launch(ctx, "istream_finalize_kernel"));
    }
    s->cur ^= 1;
    s->clen = P.clen_out;
  }
  s->received += n_new;
  s->emitted += n_emit;
  if (samples_written) *samples_written = n_emit;
  return SSQ_OK;
}

#include "cwt_host.inl"
#include "stft_rows.inl"
#include "ridge_host.inl"
#include "wavelets_host.inl"
