// gprc.cu -- C ABI of libgprc (include/gprc.h): handles, host<->device plumbing and the launch sequences of the
// GP hot path.  No Torch, no cuBLAS/cuSOLVER, no CPU fallback: every numerical step is one of the kernels in
// cov.cuh / gemm.cuh / potrf.cuh / trsv.cuh / gpc.cuh.
#include <chrono>
#include <mutex>
#include <climits>
#include <algorithm>

#include "cov.cuh"
#include "gemm.cuh"
#include "potrf.cuh"
#include "trsv.cuh"
#include "gpc.cuh"
#include "quad.cuh"
#include "ozaki.cuh"
#include "optim.hpp"

namespace gprc {
thread_local std::string g_last_error;

// ---------------------------------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------------------------------
static thread_local gprc_ctx* tl_ctx = nullptr;  // context of the API call in flight (routes dmalloc/dfree to its pool)

// Every entry point that touches a context holds one of these for its duration: it selects the context's device, makes
// the context's caching allocator the current one, and LOCKS the context -- the pool maps, the pending-timer list and
// the pinned scratch are not otherwise synchronised, and bindings such as ctypes release the interpreter lock around
// the call, so two host threads may well arrive with the same (default) context.  Calls on one context are serialised;
// different contexts run concurrently.  The mutex is recursive because entry points nest (fit -> logml helpers).
struct DeviceGuard {
  int prev = -1;
  gprc_ctx* prev_ctx = nullptr;
  std::unique_lock<std::recursive_mutex> lock;
  explicit DeviceGuard(gprc_ctx* c) : lock(c->mutex) {
    cudaGetDevice(&prev);
    if (prev != c->device) cudaSetDevice(c->device);
    prev_ctx = tl_ctx;
    tl_ctx = c;
  }
  ~DeviceGuard() {
    int cur;
    cudaGetDevice(&cur);
    if (cur != prev && prev >= 0) cudaSetDevice(prev);
    tl_ctx = prev_ctx;
  }
};

static void pool_trim(gprc_ctx* c) {
  for (auto& kv : c->pool_free) cudaFree(kv.second);
  c->pool_free.clear();
  c->pool_cached_bytes = 0;
}

static int pool_alloc(gprc_ctx* c, void** p, size_t bytes) {
  const size_t gran = 2u << 20;
  bytes = (bytes + gran - 1) / gran * gran;
  auto it = c->pool_free.lower_bound(bytes);
  if (it != c->pool_free.end() && it->first <= bytes + bytes / 4) {  // reuse a cached block of (nearly) this size
    *p = it->second;
    c->pool_cached_bytes -= it->first;
    c->pool_live[*p] = it->first;
    c->pool_free.erase(it);
    return 0;
  }
  cudaError_t e = cudaMalloc(p, bytes);
  if (e != cudaSuccess) {  // out of memory: give the cache back and retry once
    cudaGetLastError();
    cudaStreamSynchronize(c->stream);
    pool_trim(c);
    e = cudaMalloc(p, bytes);
  }
  if (e != cudaSuccess) return set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
  c->pool_live[*p] = bytes;
  return 0;
}

template <class T>
static int dmalloc(T** p, size_t count) {
  *p = nullptr;
  if (count == 0) count = 1;
  if (tl_ctx) return pool_alloc(tl_ctx, reinterpret_cast<void**>(p), count * sizeof(T));
  GPRC_CUDA(cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T)));
  return 0;
}
// Returned blocks may still be in use by kernels queued on the context's streams; they are only handed out again to
// work queued on the same streams, so stream order keeps that safe.
static void dfree(void* p) {
  if (!p) return;
  if (tl_ctx) {
    auto it = tl_ctx->pool_live.find(p);
    if (it != tl_ctx->pool_live.end()) {
      tl_ctx->pool_free.emplace(it->second, p);
      tl_ctx->pool_cached_bytes += it->second;
      tl_ctx->pool_live.erase(it);
      return;
    }
  }
  cudaFree(p);
}

// kernel spec: host struct -> device struct (sigma_vec uploaded, owned by the caller of make_spec)
struct SpecHolder {
  KSpecDev dev{};
  double* d_sigma = nullptr;
  ~SpecHolder() { dfree(d_sigma); }
};
static int make_spec(gprc_ctx* ctx, const gprc_kernel* k, int d, SpecHolder& h) {
  GPRC_ARG(k != nullptr);
  GPRC_ARG(k->id >= GPRC_CONSTANT && k->id <= GPRC_RATQUAD);
  h.dev.id = k->id;
  h.dev.c = k->c;
  h.dev.sigma = k->sigma;
  h.dev.p = k->p;
  h.dev.l = k->l;
  h.dev.gamma = k->gamma;
  h.dev.alpha = k->alpha;
  h.dev.sigma_vec = nullptr;
  h.dev.sigma_len = 0;
  if (k->id == GPRC_LINEAR && k->sigma_vec && k->sigma_len > 0) {
    GPRC_ARG(k->sigma_len == 1 || k->sigma_len == d);  // stopifnot(length(sigma) == nrow(X)), R/GPRclass.R:298
    GPRC_CHECK(dmalloc(&h.d_sigma, (size_t)k->sigma_len));
    GPRC_CUDA(cudaMemcpyAsync(h.d_sigma, k->sigma_vec, k->sigma_len * sizeof(double), cudaMemcpyHostToDevice,
                              ctx->stream));
    h.dev.sigma_vec = h.d_sigma;
    h.dev.sigma_len = k->sigma_len;
  }
  return 0;
}

__global__ void fill_kernel(double* p, long n, double v) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
// tmp[i + jj n] = (i >= j0 + jj) ? M[i + (j0 + jj) ld] : 0   (download of a lower-triangular factor, explicit zeros)
__global__ void tril_slab_kernel(const double* __restrict__ M, long ld, long n, long j0, long nc,
                                 double* __restrict__ tmp) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  const long jj = blockIdx.y;
  if (i >= n || jj >= nc) return;
  tmp[i + jj * n] = (i >= j0 + jj) ? M[i + (j0 + jj) * ld] : 0.0;
}
// columns [j0, j0 + nc) of a padded square matrix from a host-uploaded slab src (n x ncv, ld = n):
// dst[i + j ld] = src + diag_add on the diagonal inside n x n; identity (or zero) in the padding
__global__ void place_slab_kernel(const double* __restrict__ src, long n, long j0, long ncv, double* __restrict__ dst,
                                  long ld, long n_pad, long nc, double diag_add, int pad_identity) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  const long jj = blockIdx.y;
  if (i >= n_pad || jj >= nc) return;
  const long j = j0 + jj;
  double v;
  if (i < n && jj < ncv) {
    v = src[i + jj * n];
    if (i == j) v += diag_add;
  } else {
    v = (pad_identity && i == j) ? 1.0 : 0.0;
  }
  dst[i + j * ld] = v;
}
__global__ void scale_rows_kernel(double* __restrict__ M, long ld, long rows, long cols, const double* __restrict__ s) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  const long j = blockIdx.y;
  if (i < rows && j < cols) M[i + j * ld] *= s[i];
}
// y[col] = sum_i M[i, col] v[i] for a rows x cols column-major matrix
__global__ void __launch_bounds__(256) gemv_t_rect_kernel(const double* __restrict__ M, long ld, long rows, long cols,
                                                          const double* __restrict__ v, double* __restrict__ y) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long col = (long)blockIdx.x * 8 + warp;
  if (col >= cols) return;
  const double* Mp = M + col * ld;
  double s = 0.0;
  for (long i = lane; i < rows; i += 32) s = fma(Mp[i], v[i], s);
  s = warp_sum(s);
  if (lane == 0) y[col] = s;
}

// dst[t + k * ldt] = (k < n && t < m) ? src[k + t * lds] * (scale ? scale[k] : 1) : 0  over k < n_pad, t < m_pad
__global__ void __launch_bounds__(256) transpose_pad_kernel(const double* __restrict__ src, long lds, long n, long m,
                                                            double* __restrict__ dst, long ldt, long n_pad, long m_pad,
                                                            const double* __restrict__ scale) {
  __shared__ double tile[32][33];
  const long k0 = blockIdx.x * 32L, t0 = blockIdx.y * 32L;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int q = ty; q < 32; q += 8) {
    const long k = k0 + tx, t = t0 + q;
    tile[q][tx] = (k < n && t < m) ? src[k + t * lds] * (scale ? scale[k] : 1.0) : 0.0;
  }
  __syncthreads();
  for (int q = ty; q < 32; q += 8) {
    const long t = t0 + tx, k = k0 + q;
    if (t < m_pad && k < n_pad) dst[t + k * ldt] = tile[tx][q];
  }
}

static inline dim3 grid2(long rows, long cols) { return dim3((unsigned)((rows + 255) / 256), (unsigned)cols); }

}  // namespace gprc

using namespace gprc;

// =================================================================================================================
// handles
// =================================================================================================================
struct PredictWorkspace {
  long mc = 0;          // chunk capacity (multiple of 128)
  double* Ks = nullptr;     // K_star^T: mc x n_pad (test point contiguous, leading dimension mc)
  double* pmean = nullptr;  // (n_pad / 64) x mc
  double* pvar = nullptr;   // (n_pad / 128) x mc
  double* kss = nullptr;    // mc
  int* sched = nullptr;     // persistent substitution kernel: [0..1] work counter, [2] error flag, [4..] per-tile progress
  // INT8 (Ozaki) substitution, ozaki.cuh: digit tiles of V, per-test-point exponent and scale; lazily allocated
  int8_t* ozVs = nullptr;
  int* oz_ecol = nullptr;
  double* oz_scol = nullptr;
  size_t oz_bytes = 0;
  void release() {
    dfree(Ks);
    dfree(pmean);
    dfree(pvar);
    dfree(kss);
    dfree(sched);
    dfree(ozVs);
    dfree(oz_ecol);
    dfree(oz_scol);
    Ks = pmean = pvar = kss = nullptr;
    sched = nullptr;
    ozVs = nullptr;
    oz_ecol = nullptr;
    oz_scol = nullptr;
    oz_bytes = 0;
    mc = 0;
  }
};

struct FactorState {  // a factored SPD matrix and everything derived from it
  long n = 0, n_pad = 0;
  double* L = nullptr;     // n_pad x n_pad, lower
  double* dinv = nullptr;  // nt x 128 x 128 inverted diagonal blocks
  double* diag = nullptr;  // n_pad
  double* W = nullptr;     // lazy: L^-1, n_pad x n_pad lower
  // lazy, INT8 (Ozaki) substitution: digit tiles of the strictly-lower block part of L, row exponents and scales
  int8_t* ozLs = nullptr;
  int* oz_erow = nullptr;
  double* oz_srow = nullptr;
  int oz_digits = 0;
  void release() {
    dfree(L);
    dfree(dinv);
    dfree(diag);
    dfree(W);
    dfree(ozLs);
    dfree(oz_erow);
    dfree(oz_srow);
    L = dinv = diag = W = nullptr;
    ozLs = nullptr;
    oz_erow = nullptr;
    oz_srow = nullptr;
    oz_digits = 0;
  }
};

struct gprc_gpr {
  gprc_ctx* ctx = nullptr;
  int d = 0;
  bool precomputed = false;
  gprc_kernel khost{};
  SpecHolder spec;
  double* X = nullptr;  // d x n
  double* y = nullptr;  // n_pad
  double* alpha = nullptr;
  FactorState F;
  PredictWorkspace ws;
  double noise = 0, logp = 0;
};

struct gprc_gpc {
  gprc_ctx* ctx = nullptr;
  int d = 0;
  bool precomputed = false;
  SpecHolder spec;
  double* X = nullptr;
  double* y = nullptr;      // n_pad
  double* K = nullptr;      // n_pad x n_pad full symmetric (freed after fit unless needed)
  double* f = nullptr;      // n_pad  (f_hat)
  double* sw = nullptr;     // n_pad  sqrt(W) at f_hat
  double* gradl = nullptr;  // n_pad  (y + 1)/2 - P at f_hat
  FactorState F;            // factor of B = I + W^1/2 K W^1/2
  PredictWorkspace ws;
};

// =================================================================================================================
// context
// =================================================================================================================
extern "C" int gprc_version(void) { return 100; }
extern "C" const char* gprc_last_error(void) { return g_last_error.c_str(); }

extern "C" int gprc_ctx_create(gprc_ctx** out, int device) {
  GPRC_ARG(out != nullptr);
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return set_error(-3, __FILE__, __LINE__, "no CUDA device: libgprc has no CPU fallback");
  GPRC_ARG(device >= 0 && device < count);
  GPRC_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  GPRC_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 9) return set_error(-3, __FILE__, __LINE__, "libgprc is built for sm_100a (B200)");
  gprc_ctx* c = new gprc_ctx();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  int prio_lo = 0, prio_hi = 0;
  // any failure below: release what exists so far (gprc_ctx_free copes with null members) and report
#undef GPRC_CUDA_CTX
#define GPRC_CUDA_CTX(call)                                                                 \
  do {                                                                                      \
    cudaError_t e__ = (call);                                                               \
    if (e__ != cudaSuccess) {                                                               \
      gprc_ctx_free(c);                                                                     \
      return gprc::set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e__));              \
    }                                                                                       \
  } while (0)
  GPRC_CUDA_CTX(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
  GPRC_CUDA_CTX(cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, prio_lo));
  GPRC_CUDA_CTX(cudaStreamCreateWithPriority(&c->stream_hi, cudaStreamNonBlocking, prio_hi));
  GPRC_CUDA_CTX(cudaEventCreateWithFlags(&c->ev_start, cudaEventDisableTiming));
  GPRC_CUDA_CTX(cudaEventCreateWithFlags(&c->ev_panel, cudaEventDisableTiming));
  GPRC_CUDA_CTX(cudaEventCreateWithFlags(&c->ev_rest, cudaEventDisableTiming));
  GPRC_CUDA_CTX(cudaMalloc(reinterpret_cast<void**>(&c->d_info), sizeof(long)));
  GPRC_CUDA_CTX(cudaMalloc(reinterpret_cast<void**>(&c->d_scalars), 64 * sizeof(double)));
  GPRC_CUDA_CTX(cudaMalloc(reinterpret_cast<void**>(&c->d_sched), 4096));
  GPRC_CUDA_CTX(cudaMallocHost(reinterpret_cast<void**>(&c->h_scalars), 64 * sizeof(double)));
  GPRC_CUDA_CTX(cudaMallocHost(reinterpret_cast<void**>(&c->h_info), sizeof(long)));
  *out = c;
  return 0;
}

extern "C" void gprc_ctx_free(gprc_ctx* c) {
  if (!c) return;
  {  // the guard (and with it the lock on c->mutex) must be gone before the context is deleted
  DeviceGuard g(c);
  cudaStreamSynchronize(c->stream);
  for (auto& p : c->pending) {
    cudaEventDestroy(p.a);
    cudaEventDestroy(p.b);
  }
  for (auto e : c->event_pool) cudaEventDestroy(e);
  for (auto e : c->marks)
    if (e) cudaEventDestroy(e);
  pool_trim(c);
  for (auto& kv : c->pool_live) cudaFree(kv.first);
  c->pool_live.clear();
  cudaFree(c->d_info);
  cudaFree(c->d_scalars);
  cudaFree(c->d_sched);
  cudaFreeHost(c->h_scalars);
  cudaFreeHost(c->h_info);
  cudaStreamSynchronize(c->stream_hi);
  cudaEventDestroy(c->ev_start);
  cudaEventDestroy(c->ev_panel);
  cudaEventDestroy(c->ev_rest);
  cudaStreamDestroy(c->stream_hi);
  cudaStreamDestroy(c->stream);
  }
  delete c;
}

extern "C" int gprc_ctx_set_option(gprc_ctx* c, int option, int value) {
  GPRC_ARG(c != nullptr);
  if (option == GPRC_OPT_GRAM_DMMA) {
    c->opt_gram_dmma = value;
    return 0;
  }
  if (option == GPRC_OPT_PREDICT_PATH) {
    GPRC_ARG(value >= 0 && value <= 4);
    c->opt_predict_path = value;
    return 0;
  }
  if (option == GPRC_OPT_INT8_TEST_SHRINK) {
    GPRC_ARG(value >= 0 && value <= 60);
    c->opt_int8_test_shrink = value;
    return 0;
  }
  if (option == GPRC_OPT_INT8_TILE) {
    GPRC_ARG(value == 1 || value == 2 || value == 64 || value == 128);
    c->opt_int8_tile = value;
    return 0;
  }
  if (option == GPRC_OPT_CHOL_TILES) {
    GPRC_ARG(value >= 0 && value <= 1000);  // progress[] lives in the 4 KB scheduler scratch: 4 + nt ints
    c->opt_chol_tiles = value;
    return 0;
  }
  if (option == GPRC_OPT_TRSV) {
    GPRC_ARG(value == 0 || value == 1);
    c->opt_trsv = value;
    return 0;
  }
  if (option == GPRC_OPT_INT8_AUTO) {
    c->opt_int8_auto = value ? 1 : 0;
    return 0;
  }
  if (option == GPRC_OPT_OZAKI_DIGITS) {
    GPRC_ARG(value >= 6 && value <= 8);
    c->opt_ozaki_digits = value;
    return 0;
  }
  return set_error(-1, __FILE__, __LINE__, "unknown option");
}

extern "C" int gprc_ctx_set_interrupt(gprc_ctx* c, gprc_interrupt_fn fn, void* user) {
  GPRC_ARG(c != nullptr);
  c->interrupt_fn = fn;
  c->interrupt_user = user;
  return 0;
}

// between chunks of a long call: has the host asked to stop?  (drains the stream first so that nothing is left running)
static int poll_interrupt(gprc_ctx* c) {
  if (!c->interrupt_fn || !c->interrupt_fn(c->interrupt_user)) return 0;
  cudaStreamSynchronize(c->stream);
  return set_error(-8, __FILE__, __LINE__, "interrupted");
}

extern "C" int gprc_ctx_sync(gprc_ctx* c) {
  GPRC_ARG(c != nullptr);
  DeviceGuard g(c);
  GPRC_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

static void resolve_timers(gprc_ctx* c) {
  for (auto& p : c->pending) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) c->timers[p.phase] += ms;
    c->event_pool.push_back(p.a);
    c->event_pool.push_back(p.b);
  }
  c->pending.clear();
}

extern "C" void gprc_ctx_reset_timers(gprc_ctx* c) {
  if (!c) return;
  DeviceGuard g(c);
  cudaStreamSynchronize(c->stream);
  resolve_timers(c);
  for (int i = 0; i < GPRC_T_COUNT; ++i) c->timers[i] = 0.0;
  c->launches = 0;
}

extern "C" int gprc_ctx_get_timers(gprc_ctx* c, double* ms, long* launches) {
  GPRC_ARG(c != nullptr);
  DeviceGuard g(c);
  GPRC_CUDA(cudaStreamSynchronize(c->stream));
  resolve_timers(c);
  if (ms)
    for (int i = 0; i < GPRC_T_COUNT; ++i) ms[i] = c->timers[i];
  if (launches) *launches = c->launches;
  return 0;
}

// give the blocks parked in the context's caching allocator back to the driver (they are otherwise only released when an
// allocation fails, or with the context); returns the number of bytes released through *bytes (nullable)
extern "C" int gprc_ctx_trim(gprc_ctx* c, unsigned long long* bytes) {
  GPRC_ARG(c != nullptr);
  DeviceGuard g(c);
  GPRC_CUDA(cudaStreamSynchronize(c->stream));
  GPRC_CUDA(cudaStreamSynchronize(c->stream_hi));
  if (bytes) *bytes = (unsigned long long)c->pool_cached_bytes;
  pool_trim(c);
  return 0;
}

extern "C" int gprc_ctx_last_predict_path(gprc_ctx* c) { return c ? c->last_predict_path : 0; }
extern "C" long gprc_ctx_last_predict_chunks(gprc_ctx* c) { return c ? c->last_predict_chunks : 0; }

extern "C" int gprc_ctx_mark(gprc_ctx* c, int slot) {
  GPRC_ARG(c != nullptr && slot >= 0 && slot < 8);
  DeviceGuard g(c);
  if (!c->marks[slot]) GPRC_CUDA(cudaEventCreate(&c->marks[slot]));
  GPRC_CUDA(cudaEventRecord(c->marks[slot], c->stream));
  return 0;
}
extern "C" int gprc_ctx_elapsed_ms(gprc_ctx* c, int a, int b, double* ms) {
  GPRC_ARG(c != nullptr && ms != nullptr && a >= 0 && a < 8 && b >= 0 && b < 8 && c->marks[a] && c->marks[b]);
  DeviceGuard g(c);
  GPRC_CUDA(cudaEventSynchronize(c->marks[b]));
  float f = 0.f;
  GPRC_CUDA(cudaEventElapsedTime(&f, c->marks[a], c->marks[b]));
  *ms = f;
  return 0;
}

// ---- device memory helpers --------------------------------------------------------------------------------------
extern "C" int gprc_dev_malloc(gprc_ctx* c, void** dptr, unsigned long long bytes) {
  GPRC_ARG(c != nullptr && dptr != nullptr);
  DeviceGuard g(c);
  GPRC_CUDA(cudaMalloc(dptr, bytes ? bytes : 1));
  return 0;
}
extern "C" int gprc_dev_free(gprc_ctx* c, void* dptr) {
  GPRC_ARG(c != nullptr);
  DeviceGuard g(c);
  GPRC_CUDA(cudaStreamSynchronize(c->stream));
  GPRC_CUDA(cudaFree(dptr));
  return 0;
}
extern "C" int gprc_dev_h2d(gprc_ctx* c, void* dptr, const void* host, unsigned long long bytes) {
  GPRC_ARG(c != nullptr);
  DeviceGuard g(c);
  GPRC_CUDA(cudaMemcpyAsync(dptr, host, bytes, cudaMemcpyHostToDevice, c->stream));
  GPRC_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}
extern "C" int gprc_dev_d2h(gprc_ctx* c, void* host, const void* dptr, unsigned long long bytes) {
  GPRC_ARG(c != nullptr);
  DeviceGuard g(c);
  GPRC_CUDA(cudaMemcpyAsync(host, dptr, bytes, cudaMemcpyDeviceToHost, c->stream));
  GPRC_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}
extern "C" int gprc_host_register(void* host, unsigned long long bytes) {
  GPRC_CUDA(cudaHostRegister(host, bytes, cudaHostRegisterDefault));
  return 0;
}
extern "C" int gprc_host_unregister(void* host) {
  GPRC_CUDA(cudaHostUnregister(host));
  return 0;
}

// =================================================================================================================
// (1) kernel-matrix build
// =================================================================================================================
static int cov_build_dev(gprc_ctx* c, const KSpecDev& k, const double* dA, int d, long nA, const double* dB, long nB,
                         double* out, long ldo, long rows_pad, long cols_pad, bool lower_only, bool symmetric,
                         double diag_add, bool pad_identity, const double* rowscale, const double* weights,
                         double* pmean, long ldpm, const double* colscale = nullptr,
                         const double* colweights = nullptr, int* tile_rows = nullptr) {
  CovParams p;
  p.k = k;
  p.A = dA;
  p.B = dB;
  p.d = d;
  p.nA = nA;
  p.nB = nB;
  p.out = out;
  p.ldo = ldo;
  p.rows_pad = rows_pad;
  p.cols_pad = cols_pad;
  p.lower_only = lower_only;
  p.symmetric = symmetric;
  p.diag_add = diag_add;
  p.pad_identity = pad_identity;
  p.rowscale = rowscale;
  p.weights = weights;
  p.pmean = pmean;
  p.ldpm = ldpm;
  p.colscale = colscale;
  p.colweights = colweights;
  p.col_offset = 0;
  if (tile_rows) *tile_rows = cov_tile_rows(c, p);
  return launch_cov(c, p);
}

extern "C" int gprc_cov_matrix(gprc_ctx* c, const gprc_kernel* k, const double* A, int d, long nA, const double* B,
                               long nB, double* out) {
  GPRC_ARG(c && k && A && B && out && d > 0 && nA >= 0 && nB >= 0);
  if (nA == 0 || nB == 0) return 0;
  DeviceGuard g(c);
  SpecHolder spec;
  GPRC_CHECK(make_spec(c, k, d, spec));
  double *dA = nullptr, *dB = nullptr, *dout = nullptr;
  const long rp = round_up(nA, NB);
  // column chunks bound the device buffer (<= 2 GiB) and the grid's y extent
  long cchunk = std::max<long>(NB, std::min<long>(round_up(nB, NB), ((2L << 30) / 8 / rp) / NB * NB));
  cchunk = std::min<long>(cchunk, 65535L * CT);
  int rc = 0;
  do {
    if ((rc = dmalloc(&dA, (size_t)d * nA))) break;
    if ((rc = dmalloc(&dB, (size_t)d * nB))) break;
    if ((rc = dmalloc(&dout, (size_t)rp * cchunk))) break;
    cudaMemcpyAsync(dA, A, sizeof(double) * d * nA, cudaMemcpyHostToDevice, c->stream);
    cudaMemcpyAsync(dB, B, sizeof(double) * d * nB, cudaMemcpyHostToDevice, c->stream);
    for (long c0 = 0; c0 < nB && rc == 0; c0 += cchunk) {
      const long nc = std::min(cchunk, nB - c0);
      {
        PhaseTimer t(c, GPRC_T_BUILD_K);
        rc = cov_build_dev(c, spec.dev, dA, d, nA, dB + c0 * d, nc, dout, rp, rp, round_up(nc, NB), false, false, 0.0,
                           false, nullptr, nullptr, nullptr, 0);
      }
      if (rc) break;
      cudaError_t e = cudaMemcpy2DAsync(out + c0 * nA, nA * sizeof(double), dout, rp * sizeof(double),
                                        nA * sizeof(double), nc, cudaMemcpyDeviceToHost, c->stream);
      if (e != cudaSuccess) rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
    }
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (rc == 0 && e != cudaSuccess) rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
  } while (0);
  dfree(dA);
  dfree(dB);
  dfree(dout);
  return rc;
}

extern "C" int gprc_cov_pointwise(gprc_ctx* c, const gprc_kernel* k, const double* A, const double* B, int d, long n,
                                  double* out) {
  GPRC_ARG(c && k && A && B && out && d > 0 && n >= 0);
  if (n == 0) return 0;
  DeviceGuard g(c);
  SpecHolder spec;
  GPRC_CHECK(make_spec(c, k, d, spec));
  double *dA = nullptr, *dB = nullptr, *dout = nullptr;
  int rc = 0;
  do {
    if ((rc = dmalloc(&dA, (size_t)d * n))) break;
    if ((rc = dmalloc(&dB, (size_t)d * n))) break;
    if ((rc = dmalloc(&dout, (size_t)n))) break;
    cudaMemcpyAsync(dA, A, sizeof(double) * d * n, cudaMemcpyHostToDevice, c->stream);
    cudaMemcpyAsync(dB, B, sizeof(double) * d * n, cudaMemcpyHostToDevice, c->stream);
    cov_pointwise_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(spec.dev, dA, dB, d, n, dout);
    c->launches++;
    cudaMemcpyAsync(out, dout, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
  } while (0);
  dfree(dA);
  dfree(dB);
  dfree(dout);
  return rc;
}

// =================================================================================================================
// factor + solve shared by GPR, logml and GPC
// =================================================================================================================
static int factor_alloc(FactorState& F, long n) {
  F.n = n;
  F.n_pad = round_up(std::max<long>(n, 1), NB);
  GPRC_CHECK(dmalloc(&F.L, (size_t)F.n_pad * F.n_pad));
  GPRC_CHECK(dmalloc(&F.dinv, (size_t)F.n_pad * NB));
  GPRC_CHECK(dmalloc(&F.diag, (size_t)F.n_pad));
  return 0;
}

// factor F.L in place; returns info through *info (0 ok).  Synchronises the stream.
static int factor_run(gprc_ctx* c, FactorState& F, long* info) {
  *c->h_info = LONG_MAX;
  GPRC_CUDA(cudaMemcpyAsync(c->d_info, c->h_info, sizeof(long), cudaMemcpyHostToDevice, c->stream));
  {
    PhaseTimer t(c, GPRC_T_CHOL);
    GPRC_CHECK(potrf_blocked(c, F.L, F.n_pad, F.n_pad, F.dinv, c->d_info, F.diag));
  }
  GPRC_CUDA(cudaMemcpyAsync(c->h_info, c->d_info, sizeof(long), cudaMemcpyDeviceToHost, c->stream));
  GPRC_CUDA(cudaStreamSynchronize(c->stream));
  const long v = *c->h_info;
  *info = (v == LONG_MAX) ? 0 : v;
  return 0;
}

static int ensure_inverse(gprc_ctx* c, FactorState& F) {
  if (F.W) return 0;
  GPRC_CHECK(dmalloc(&F.W, (size_t)F.n_pad * F.n_pad));
  // scratch for the level products aliases the (unused) strictly upper block triangle of the L buffer;
  // W^T is only needed while inverting
  double* Wt = nullptr;
  GPRC_CHECK(dmalloc(&Wt, (size_t)F.n_pad * F.n_pad));
  int rc;
  {
    PhaseTimer t(c, GPRC_T_TRTRI);
    GPRC_CUDA(cudaMemsetAsync(F.W, 0, sizeof(double) * F.n_pad * F.n_pad, c->stream));  // zeros above the diagonal
    rc = trtri_levels(c, F.L, F.n_pad, F.n_pad, F.dinv, F.W, Wt, F.L);
  }
  dfree(Wt);
  return rc;
}

constexpr long WAVE_COLS = 148L * NB;  // test points of one full wave of 128-wide tiles on 148 SMs

static int workspace_ensure(gprc_ctx* c, PredictWorkspace& ws, long n_pad, long m, double max_bytes = 8.0e9,
                            double extra_bytes_per_col = 0.0, double free_frac = 0.5) {
  size_t free_b = 0, total_b = 0;
  cudaMemGetInfo(&free_b, &total_b);
  // blocks parked in this context's caching pool are available too (pool_alloc gives them back to the driver and retries
  // when cudaMalloc fails); without them the chunk size shrank from step to step as differently sized workspaces piled
  // up in the pool (27 chunks instead of 11 for 10^6 test points at n = 50 000)
  free_b += c->pool_cached_bytes;
  long want = round_up(std::max<long>(m, 1), NB);
  // per test point: Ks column + partial rows
  // (+ the INT8 path's digit planes of V, allocated by its variance pass)
  const double per_col = 8.0 * ((double)n_pad + (double)n_pad / 64 + (double)n_pad / NB + 1) + extra_bytes_per_col;
  const double budget = std::min(max_bytes, free_frac * (double)free_b + (ws.mc ? per_col * ws.mc : 0.0));
  long cap = (long)(budget / per_col) / NB * NB;
  cap = std::max<long>(cap, NB);
  cap = std::min<long>(cap, 1L << 20);
  // everything in one chunk if it fits; otherwise chunks made of whole waves
  if (want > cap && cap >= WAVE_COLS) cap = cap / WAVE_COLS * WAVE_COLS;
  want = std::min(want, cap);
  if (ws.mc >= want) return 0;
  ws.release();
  GPRC_CHECK(dmalloc(&ws.Ks, (size_t)n_pad * want));
  GPRC_CHECK(dmalloc(&ws.pmean, (size_t)(n_pad / CT) * want));
  GPRC_CHECK(dmalloc(&ws.pvar, (size_t)(n_pad / NB) * want));
  GPRC_CHECK(dmalloc(&ws.kss, (size_t)want));
  GPRC_CHECK(dmalloc(&ws.sched, (size_t)(want / NB + 8)));
  ws.mc = want;
  return 0;
}

// variance pass on a chunk whose (row-scaled) K_star is already in ws.Ks:  pvar partials of colSums((W Ks)^2)
static int variance_pass(gprc_ctx* c, FactorState& F, PredictWorkspace& ws, long mcur_pad, double* VoutT, long ldv) {
  const int nt = (int)(F.n_pad / NB), ntc = (int)(mcur_pad / NB);
  TrmmNormPolicy p;
  p.W = F.W;
  p.ldw = F.n_pad;
  p.KsT = ws.Ks;
  p.ldk = ws.mc;
  p.partial = ws.pvar;
  p.ldp = ws.mc;
  p.VoutT = VoutT;
  p.ldv = ldv;
  p.nt = nt;
  p.ntc = ntc;
  const long groups = (nt + TrmmNormPolicy::GROUP - 1) / TrmmNormPolicy::GROUP;
  PhaseTimer t(c, GPRC_T_VAR);
  return launch_gemm(c, p, dim3((unsigned)(groups * TrmmNormPolicy::GROUP * ntc)));
}

// the same partial column norms by blocked forward substitution on K_star^T (no inverse needed)
static int variance_pass_trsm(gprc_ctx* c, FactorState& F, PredictWorkspace& ws, long mcur_pad) {
  const int nt = (int)(F.n_pad / NB), ntc = (int)(mcur_pad / NB);
  PhaseTimer t(c, GPRC_T_VAR);
  for (int i = 0; i < nt; ++i) {
    if (i > 0) {
      TrsmLeftUpdatePolicy up{F.L, F.n_pad, ws.Ks, ws.mc, i};
      GPRC_CHECK(launch_gemm(c, up, dim3((unsigned)ntc)));
    }
    TrsmLeftDiagPolicy dg{F.dinv + (long)i * NB * NB, ws.Ks, ws.mc, i, ws.pvar, ws.mc};
    GPRC_CHECK(launch_gemm(c, dg, dim3((unsigned)ntc)));
  }
  return 0;
}

// ... and as ONE persistent kernel with per-tile progress counters (no launch boundary between block rows)
static int variance_pass_persistent(gprc_ctx* c, FactorState& F, PredictWorkspace& ws, long mcur_pad) {
  static bool configured[64] = {false};
  if (!configured[c->device & 63]) {
    GPRC_CUDA(cudaFuncSetAttribute(trsm_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
    configured[c->device & 63] = true;
  }
  const int nt = (int)(F.n_pad / NB), ntc = (int)(mcur_pad / NB);
  PhaseTimer t(c, GPRC_T_VAR);
  GPRC_CUDA(cudaMemsetAsync(ws.sched, 0, sizeof(int) * (ntc + 8), c->stream));
  TrsmPersistParams p;
  p.L = F.L;
  p.ldl = F.n_pad;
  p.dinv = F.dinv;
  p.T = ws.Ks;
  p.ldt = ws.mc;
  p.partial = ws.pvar;
  p.ldp = ws.mc;
  p.nt = nt;
  p.ntc = ntc;
  p.next = reinterpret_cast<unsigned long long*>(ws.sched);
  p.error = ws.sched + 2;
  p.progress = ws.sched + 4;
  const int grid = std::min(c->sm_count, ntc);
  trsm_persistent_kernel<<<grid, GEMM_THREADS, GEMM_SMEM_BYTES, c->stream>>>(p);
  c->launches++;
  GPRC_CUDA(cudaGetLastError());
  return 0;
}

// ... and with the O(n^2 m) products on the INT8 tensor cores (ozaki.cuh): per block row one tcgen05 update launch,
// the FP64 diagonal solve (same kernel as path 2) and the digit split of the new block row of V.
// ws.sched[3] collects the overflow / watchdog flags; the caller checks it after the chunk.
template <int S>
static int oz_factor_digits(gprc_ctx* c, FactorState& F) {
  const int nt = (int)(F.n_pad / NB);
  if (!F.ozLs || F.oz_digits != S) {
    dfree(F.ozLs);
    F.ozLs = nullptr;
    GPRC_CHECK(dmalloc(&F.ozLs, (size_t)F.n_pad * F.n_pad * S));
    if (!F.oz_erow) GPRC_CHECK(dmalloc(&F.oz_erow, (size_t)F.n_pad));
    if (!F.oz_srow) GPRC_CHECK(dmalloc(&F.oz_srow, (size_t)F.n_pad));
    F.oz_digits = 0;
  } else {
    return 0;
  }
  int* flag = nullptr;
  GPRC_CHECK(dmalloc(&flag, 1));
  GPRC_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), c->stream));
  oz::rowmax_kernel<<<nt, 256, 0, c->stream>>>(F.L, F.n_pad, F.oz_erow, F.oz_srow);
  oz::split_l_kernel<S><<<dim3(4 * nt, nt), 256, 0, c->stream>>>(F.L, F.n_pad, F.oz_erow, F.ozLs, (int)(F.n_pad / oz::BK), flag);
  c->launches += 2;
  GPRC_CUDA(cudaMemcpyAsync(c->h_info, flag, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  GPRC_CUDA(cudaStreamSynchronize(c->stream));
  dfree(flag);
  if (*reinterpret_cast<int*>(c->h_info) != 0)
    return set_error(-7, __FILE__, __LINE__, "INT8 substitution: L has non-finite entries");
  F.oz_digits = S;
  return 0;
}

// launch of the stacked-plane kernel on clusters of two CTAs (ozaki.cuh): pair j = block rows 2 j, 2 j + 1
template <int S>
static int launch_update_stack_pair(gprc_ctx* c, const oz::UpdateParams& up, long mcur_pad) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(2 * (mcur_pad / oz::BN)));
  cfg.blockDim = dim3(oz::THREADS);
  cfg.dynamicSmemBytes = oz::Cfg<S>::SMEM_BYTES;
  cfg.stream = c->stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  GPRC_CUDA(cudaLaunchKernelEx(&cfg, oz::update_stack_kernel<S, 2>, up));
  return 0;
}

template <int S>
static int variance_pass_ozaki_t(gprc_ctx* c, FactorState& F, PredictWorkspace& ws, long mcur, long mcur_pad) {
  static bool configured[64] = {false};
  if (!configured[c->device & 63]) {
    GPRC_CUDA(cudaFuncSetAttribute(oz::update_kernel<S, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, oz::Cfg<S>::SMEM_BYTES));
    GPRC_CUDA(cudaFuncSetAttribute(oz::update128_kernel<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, oz::Cfg2<S>::SMEM_BYTES));
    GPRC_CUDA(cudaFuncSetAttribute(oz::update_stack_kernel<S, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, oz::Cfg<S>::SMEM_BYTES));
    GPRC_CUDA(cudaFuncSetAttribute(oz::update_stack_kernel<S, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, oz::Cfg<S>::SMEM_BYTES));
    configured[c->device & 63] = true;
  }
  // kernel variant (GPRC_OPT_INT8_TILE): 2 = stacked planes on cluster pairs, 1 = stacked planes, 64 = one MMA per digit
  // pair (round 1), 128 = 128 x 128 tiles with the orders in two passes (round 1)
  const int variant = c->opt_int8_tile;
  const bool wide = variant == 128;
  GPRC_CHECK(oz_factor_digits<S>(c, F));
  const size_t need = (size_t)ws.mc * F.n_pad * S;
  if (ws.oz_bytes < need) {
    dfree(ws.ozVs);
    ws.ozVs = nullptr;
    ws.oz_bytes = 0;
    GPRC_CHECK(dmalloc(&ws.ozVs, need));
    ws.oz_bytes = need;
  }
  if (!ws.oz_ecol) GPRC_CHECK(dmalloc(&ws.oz_ecol, (size_t)ws.mc));
  if (!ws.oz_scol) GPRC_CHECK(dmalloc(&ws.oz_scol, (size_t)ws.mc));
  const int nt = (int)(F.n_pad / NB), ntc = (int)(mcur_pad / NB), KB = (int)(F.n_pad / oz::BK);
  int* flag = ws.sched + 3;
  PhaseTimer t(c, GPRC_T_VAR);
  GPRC_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), c->stream));
  oz::colscale_kernel<<<(unsigned)((mcur_pad + 255) / 256), 256, 0, c->stream>>>(ws.kss, mcur, mcur_pad, ws.oz_ecol, ws.oz_scol,
                                                                                            c->opt_int8_test_shrink);
  c->launches++;
  auto split_row = [&](int i) {
    if (wide)
      oz::split_v128_kernel<S><<<dim3((unsigned)(mcur_pad / oz::BN2), 4), 256, 0, c->stream>>>(ws.Ks, ws.mc, i, ws.oz_ecol, ws.ozVs, KB, flag);
    else
      oz::split_v_kernel<S><<<dim3((unsigned)(mcur_pad / oz::BN), 4), 128, 0, c->stream>>>(ws.Ks, ws.mc, i, ws.oz_ecol, ws.ozVs, KB, flag);
    c->launches++;
  };
  auto diag_row = [&](int i) {
    TrsmLeftDiagPolicy dg{F.dinv + (long)i * NB * NB, ws.Ks, ws.mc, i, ws.pvar, ws.mc};
    return launch_gemm(c, dg, dim3((unsigned)ntc));
  };
  if (variant == 2) {
    // block rows in pairs: one INT8 launch brings rows 2 j and 2 j + 1 up to k < 256 j (each V digit tile is fetched once
    // for both); the 128 x 128 block L[2j+1, 2j] that remains inside the pair is applied in FP64 between the two
    // diagonal solves
    for (int j = 0; 2 * j < nt; ++j) {
      const int i0 = 2 * j, i1 = 2 * j + 1;
      const bool has1 = i1 < nt;
      if (j > 0) {
        if (has1) {
          oz::UpdateParams up{F.ozLs, ws.ozVs, F.oz_srow, ws.oz_scol, ws.Ks, ws.mc, j, KB, flag, 0, nullptr};
          GPRC_CHECK(launch_update_stack_pair<S>(c, up, mcur_pad));
        } else {  // odd number of block rows: the last one alone
          oz::UpdateParams up{F.ozLs, ws.ozVs, F.oz_srow, ws.oz_scol, ws.Ks, ws.mc, i0, KB, flag, 0, nullptr};
          oz::update_stack_kernel<S, 1><<<(unsigned)(mcur_pad / oz::BN), oz::THREADS, oz::Cfg<S>::SMEM_BYTES, c->stream>>>(up);
        }
        c->launches++;
      }
      GPRC_CHECK(diag_row(i0));
      if (has1) {
        TrsmLeftUpdatePolicy in_pair{F.L, F.n_pad, ws.Ks, ws.mc, i1, i0};
        GPRC_CHECK(launch_gemm(c, in_pair, dim3((unsigned)ntc)));
        GPRC_CHECK(diag_row(i1));
      }
      if (i1 + 1 < nt) {
        split_row(i0);
        split_row(i1);
      }
    }
    GPRC_CUDA(cudaGetLastError());
    return 0;
  }
  for (int i = 0; i < nt; ++i) {
    if (i > 0) {
      oz::UpdateParams up{F.ozLs, ws.ozVs, F.oz_srow, ws.oz_scol, ws.Ks, ws.mc, i, KB, flag, 0, nullptr};
      if (wide)
        oz::update128_kernel<S><<<(unsigned)(mcur_pad / oz::BN2), oz::THREADS, oz::Cfg2<S>::SMEM_BYTES, c->stream>>>(up);
      else if (variant == 1)
        oz::update_stack_kernel<S, 1><<<(unsigned)(mcur_pad / oz::BN), oz::THREADS, oz::Cfg<S>::SMEM_BYTES, c->stream>>>(up);
      else
        oz::update_kernel<S, false><<<(unsigned)(mcur_pad / oz::BN), oz::THREADS, oz::Cfg<S>::SMEM_BYTES, c->stream>>>(up);
      c->launches++;
    }
    GPRC_CHECK(diag_row(i));
    if (i + 1 < nt) split_row(i);
  }
  GPRC_CUDA(cudaGetLastError());
  return 0;
}

static int oz_factor_digits_any(gprc_ctx* c, FactorState& F) {
  switch (c->opt_ozaki_digits) {
    case 6: return oz_factor_digits<6>(c, F);
    case 8: return oz_factor_digits<8>(c, F);
    default: return oz_factor_digits<7>(c, F);
  }
}

static int variance_pass_ozaki(gprc_ctx* c, FactorState& F, PredictWorkspace& ws, long mcur, long mcur_pad) {
  switch (c->opt_ozaki_digits) {
    case 6: return variance_pass_ozaki_t<6>(c, F, ws, mcur, mcur_pad);
    case 8: return variance_pass_ozaki_t<8>(c, F, ws, mcur, mcur_pad);
    default: return variance_pass_ozaki_t<7>(c, F, ws, mcur, mcur_pad);
  }
}

// mean/var for m test points (device pointers).  weights: alpha (GPR) or (y+1)/2 - P (GPC); rowscale: sqrt(W) or null.
// one chunk of test points on the CURRENT c->stream with workspace w: K_star^T (+ mean partials), variance pass, finalize
static int predict_chunk(gprc_ctx* c, const KSpecDev& k, const double* dX, int d, FactorState& F, PredictWorkspace& w,
                         const double* weights, const double* rowscale, const double* dXs, long c0, long mcur,
                         int path /* 1 inverse, 2 substitution, 3 persistent substitution, 4 INT8 substitution */, double* dmean,
                         double* dvar) {
  GPRC_ARG(mcur > 0 && mcur <= w.mc);  // the chunk must fit the workspace (Ks, pmean, pvar, kss are n_pad x w.mc)
  c->last_predict_chunks++;
  const long mpad = round_up(mcur, NB);
  int mean_tile = CT;  // training points per partial of the mean: 64 (direct build) or 128 (tensor-core build)
  {
    PhaseTimer t(c, GPRC_T_BUILD_KS);
    // K_star^T tile by tile: rows = test points, columns = training points; sqrt(W) scaling and the mean's weighted
    // sums run along the training axis
    GPRC_CHECK(cov_build_dev(c, k, dXs + c0 * d, d, mcur, dX, F.n, w.Ks, w.mc, mpad, F.n_pad, false, false, 0.0, false,
                             nullptr, nullptr, w.pmean, w.mc, rowscale, weights, &mean_tile));
    cov_pointwise_kernel<<<(unsigned)((mcur + 255) / 256), 256, 0, c->stream>>>(k, dXs + c0 * d, dXs + c0 * d, d, mcur,
                                                                               w.kss);
    c->launches++;
  }
  GPRC_CHECK(path == 4   ? variance_pass_ozaki(c, F, w, mcur, mpad)
             : path == 3 ? variance_pass_persistent(c, F, w, mpad)
             : path == 2 ? variance_pass_trsm(c, F, w, mpad)
                         : variance_pass(c, F, w, mpad, nullptr, 0));
  finalize_predict_kernel<<<(unsigned)((mcur + 255) / 256), 256, 0, c->stream>>>(
      w.pmean, w.mc, (int)(F.n_pad / mean_tile), w.pvar, w.mc, (int)(F.n_pad / NB), w.kss, mcur, dmean + c0, dvar + c0);
  c->launches++;
  GPRC_CUDA(cudaGetLastError());
  return 0;
}

static int predict_pointwise_dev(gprc_ctx* c, const KSpecDev& k, const double* dX, int d, FactorState& F,
                                 PredictWorkspace& ws, const double* weights, const double* rowscale,
                                 const double* dXs, long m, double* dmean, double* dvar) {
  // path of the variance pass: 1 = with W = L^-1 (one triangular GEMM per chunk); 2 = blocked substitution, two
  // launches per block row (whole-wave chunks); 3 = the same substitution as one persistent kernel per chunk.
  // auto: large predicts without an inverse at hand take 3, everything else 1.
  int path = c->opt_predict_path;
  bool planned = (path == 0 && !F.W && m >= WAVE_COLS);  // large predict, no inverse at hand: substitution
  if (planned && c->opt_int8_auto && F.n_pad >= 4096) {
    // ... with its products on the INT8 tensor cores once the O(n^2 m) term dominates (2x the FP64 tensor roofline),
    // provided the digit planes fit: S n_pad^2 bytes for L (unless already built) plus one wave of K_star^T and its digits
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    const double S = (double)c->opt_ozaki_digits, np = (double)F.n_pad;
    const double need = (F.ozLs ? 0.0 : S * np * np) + (double)WAVE_COLS * np * (8.0 + S) * 1.1;
    if ((double)free_b + (double)c->pool_cached_bytes > need * 1.05 || ws.ozVs) {
      planned = false;
      path = 4;
    }
  }
  if (path == 0 && !planned) path = 1;
  if (path == 1) GPRC_CHECK(ensure_inverse(c, F));
  c->last_predict_path = planned ? 2 : path;
  c->last_predict_chunks = 0;
  PhaseTimer span(c, GPRC_T_PREDICT);
  if (planned) {
    // Mixed plan.  Whole waves of 148 tiles go through the multi-launch substitution (all CTAs sweep the same block row
    // in lockstep: the L row panel is shared in L2, 35.4 TFLOP/s); the last wave is merged with the remainder into ONE
    // chunk of 148 + r tiles for the persistent kernel, which packs them without idle SMs (33.9 TFLOP/s because its CTAs
    // drift apart along k).  125 000 points = 6.6 waves: 5 waves + a 237-tile persistent chunk instead of 7 sweeps.
    GPRC_CHECK(workspace_ensure(c, ws, F.n_pad, m, 20.0e9));
    const long tiles = (m + NB - 1) / NB, cap_tiles = ws.mc / NB, rem = tiles % 148;
    long last_tiles = (rem == 0) ? 0 : ((tiles >= 148 && cap_tiles >= 148 + rem) ? 148 + rem : rem);
    long c0 = 0;
    for (long left = tiles - last_tiles; left > 0;) {
      const long take = std::min(left, cap_tiles);
      if (c0 > 0) GPRC_CHECK(poll_interrupt(c));
      GPRC_CHECK(predict_chunk(c, k, dX, d, F, ws, weights, rowscale, dXs, c0, std::min(take * NB, m - c0), 2, dmean, dvar));
      c0 += take * NB;
      left -= take;
    }
    if (last_tiles > 0) {
      // the merged tail (148 + r tiles, or r tiles) in pieces of at most cap_tiles: when device memory is short the
      // workspace may hold less than the tail (cap_tiles can be as small as one tile)
      while (c0 < m) {
        if (c0 > 0) GPRC_CHECK(poll_interrupt(c));
        const long mcur = std::min(cap_tiles * NB, m - c0);
        GPRC_CHECK(predict_chunk(c, k, dX, d, F, ws, weights, rowscale, dXs, c0, mcur, 3, dmean, dvar));
        c0 += mcur;
        GPRC_CUDA(cudaMemcpyAsync(c->h_info, ws.sched + 2, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        GPRC_CUDA(cudaStreamSynchronize(c->stream));
        if (*reinterpret_cast<int*>(c->h_info) != 0)
          return set_error(-6, __FILE__, __LINE__, "persistent substitution kernel: a tile dependency never arrived");
      }
    }
    return 0;
  }
  if (path == 3) {
    // everything through the persistent kernel: big balanced chunks
    GPRC_CHECK(workspace_ensure(c, ws, F.n_pad, m, 40.0e9));
    const long tiles = (m + NB - 1) / NB, cap_tiles = ws.mc / NB;
    const long nchunks = (tiles + cap_tiles - 1) / cap_tiles;
    const long per = ((tiles + nchunks - 1) / nchunks) * NB;
    for (long c0 = 0; c0 < m; c0 += per)
      GPRC_CHECK(predict_chunk(c, k, dX, d, F, ws, weights, rowscale, dXs, c0, std::min(per, m - c0), 3, dmean, dvar));
    GPRC_CUDA(cudaMemcpyAsync(c->h_info, ws.sched + 2, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    GPRC_CUDA(cudaStreamSynchronize(c->stream));
    if (*reinterpret_cast<int*>(c->h_info) != 0)
      return set_error(-6, __FILE__, __LINE__, "persistent substitution kernel: a tile dependency never arrived");
    return 0;
  }
  if (path == 4) {
    // INT8 substitution: whole-wave chunks like path 2; the overflow / watchdog flag is read after every chunk and a
    // flagged chunk (a K_star that violates |v| <= sqrt(k**), i.e. not a covariance of this model) is redone in FP64
    // Big chunks: the CTAs of this path are independent (no lockstep sweep to preserve), so many waves per launch
    // amortise the per-block-row launches and leave one short tail instead of one per 148-tile chunk.
    GPRC_CHECK(oz_factor_digits_any(c, F));  // before sizing the workspace: the digit planes of L take n_pad^2 S bytes
    // up to 110 GB and 70 % of what is free for the chunk (K_star^T + its digit planes): 113 664 test points per chunk at
    // n = 50 000 (24 waves of cluster pairs), and the whole 125 000-point shard of an 8-GPU run in ONE chunk
    GPRC_CHECK(workspace_ensure(c, ws, F.n_pad, m, 110.0e9, (double)c->opt_ozaki_digits * (double)F.n_pad, 0.7));
    const bool trace_chunks = getenv("GPRC_TRACE_CHUNKS") != nullptr;  // diagnostics: host wall time per chunk on stderr
    for (long c0 = 0; c0 < m; c0 += ws.mc) {
      const long mcur = std::min(ws.mc, m - c0);
      if (c0 > 0) GPRC_CHECK(poll_interrupt(c));
      const auto w0 = std::chrono::steady_clock::now();
      GPRC_CHECK(predict_chunk(c, k, dX, d, F, ws, weights, rowscale, dXs, c0, mcur, 4, dmean, dvar));
      const auto w1 = std::chrono::steady_clock::now();
      GPRC_CUDA(cudaMemcpyAsync(c->h_info, ws.sched + 3, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
      GPRC_CUDA(cudaStreamSynchronize(c->stream));
      if (trace_chunks)
        fprintf(stderr, "[gprc] INT8 chunk at %ld (%ld points): enqueue %.1f ms, complete %.1f ms\n", c0, mcur,
                std::chrono::duration<double, std::milli>(w1 - w0).count(),
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - w0).count());
      const int flag = *reinterpret_cast<int*>(c->h_info);
      if (flag & ~3) return set_error(-6, __FILE__, __LINE__, "INT8 substitution kernel: a pipeline barrier never completed");
      if (flag) GPRC_CHECK(predict_chunk(c, k, dX, d, F, ws, weights, rowscale, dXs, c0, mcur, 2, dmean, dvar));
    }
    return 0;
  }
  // NB every launch of a substitution-path chunk (path 2) is one grid of <= 148 CTAs that depends on the previous one,
  // so a last chunk of r < 148 tiles leaves 148 - r SMs idle for a whole sweep (125 000 points = 6.6 waves: 6 %).
  // Running several chunk pipelines on concurrent streams was measured and does NOT recover it (2 pipelines 33.45 vs
  // 33.40 TFLOP/s, 4 sub-wave pipelines 32.4, 8: 31.4 -- the block scheduler does not pack the grids); path 3 does.
  GPRC_CHECK(workspace_ensure(c, ws, F.n_pad, m));
  for (long c0 = 0; c0 < m; c0 += ws.mc) {
    if (c0 > 0) GPRC_CHECK(poll_interrupt(c));
    GPRC_CHECK(predict_chunk(c, k, dX, d, F, ws, weights, rowscale, dXs, c0, std::min(ws.mc, m - c0), path, dmean, dvar));
  }
  return 0;
}

// same with K_star (n x m) and kss (m) given on the host (closure kernels)
static int predict_precomputed(gprc_ctx* c, FactorState& F, PredictWorkspace& ws, const double* weights,
                               const double* rowscale, const double* Ks, const double* kss, long m, double* mean,
                               double* var) {
  // default: W = L^-1 once and one triangular GEMM per chunk; a forced GPRC_OPT_PREDICT_PATH of 2 / 4 takes the FP64 /
  // INT8 substitution instead (tests drive the INT8 pass with arbitrary K, K_star through this)
  int path = c->opt_predict_path;
  if (path != 2 && path != 4) path = 1;
  if (path == 1) GPRC_CHECK(ensure_inverse(c, F));
  if (path == 4) {
    GPRC_CHECK(oz_factor_digits_any(c, F));
    GPRC_CHECK(workspace_ensure(c, ws, F.n_pad, m, 8.0e9, (double)c->opt_ozaki_digits * (double)F.n_pad));
  } else {
    GPRC_CHECK(workspace_ensure(c, ws, F.n_pad, m));
  }
  c->last_predict_path = path;
  double *dmean = nullptr, *dvar = nullptr, *stage = nullptr;
  int rc = 0;
  do {
    if ((rc = dmalloc(&dmean, (size_t)ws.mc))) break;
    if ((rc = dmalloc(&dvar, (size_t)ws.mc))) break;
    if ((rc = dmalloc(&stage, (size_t)F.n * std::min<long>(ws.mc, m)))) break;
    for (long c0 = 0; c0 < m && rc == 0; c0 += ws.mc) {
      const long mcur = std::min(ws.mc, m - c0);
      const long mpad = round_up(mcur, NB);
      cudaMemcpyAsync(stage, Ks + c0 * F.n, sizeof(double) * F.n * mcur, cudaMemcpyHostToDevice, c->stream);
      cudaMemcpyAsync(ws.kss, kss + c0, sizeof(double) * mcur, cudaMemcpyHostToDevice, c->stream);
      gemv_t_rect_kernel<<<(unsigned)((mcur + 7) / 8), 256, 0, c->stream>>>(stage, F.n, F.n, mcur, weights, dmean);
      c->launches++;
      int pass = path;
      for (;;) {
        transpose_pad_kernel<<<dim3((unsigned)(F.n_pad / 32), (unsigned)(mpad / 32)), 256, 0, c->stream>>>(
            stage, F.n, F.n, mcur, ws.Ks, ws.mc, F.n_pad, mpad, rowscale);
        c->launches++;
        rc = pass == 4 ? variance_pass_ozaki(c, F, ws, mcur, mpad)
             : pass == 2 ? variance_pass_trsm(c, F, ws, mpad)
                         : variance_pass(c, F, ws, mpad, nullptr, 0);
        if (rc || pass != 4) break;
        cudaMemcpyAsync(c->h_info, ws.sched + 3, sizeof(int), cudaMemcpyDeviceToHost, c->stream);
        cudaError_t e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) {
          rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
          break;
        }
        const int flag = *reinterpret_cast<int*>(c->h_info);
        if (flag & ~3) rc = set_error(-6, __FILE__, __LINE__, "INT8 substitution kernel: a pipeline barrier never completed");
        if (rc || !flag) break;
        pass = 2;  // v left its fixed-point range (K_star is not a covariance of this model): redo the chunk in FP64
      }
      if (rc) break;
      finalize_predict_kernel<<<(unsigned)((mcur + 255) / 256), 256, 0, c->stream>>>(
          nullptr, 0, 0, ws.pvar, ws.mc, (int)(F.n_pad / NB), ws.kss, mcur, nullptr, dvar);
      c->launches++;
      cudaMemcpyAsync(mean + c0, dmean, sizeof(double) * mcur, cudaMemcpyDeviceToHost, c->stream);
      cudaMemcpyAsync(var + c0, dvar, sizeof(double) * mcur, cudaMemcpyDeviceToHost, c->stream);
      cudaError_t e = cudaStreamSynchronize(c->stream);
      if (e != cudaSuccess) rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
    }
  } while (0);
  dfree(dmean);
  dfree(dvar);
  dfree(stage);
  return rc;
}

static int download_lower(gprc_ctx* c, const double* dM, long n, long ld, double* host) {
  double* tmp = nullptr;
  // stream the columns in slabs so that the staging buffer stays small
  const long slab = std::max<long>(1, std::min<long>(n, (256L << 20) / 8 / std::max<long>(n, 1)));
  GPRC_CHECK(dmalloc(&tmp, (size_t)n * slab));
  int rc = 0;
  for (long j0 = 0; j0 < n; j0 += slab) {
    const long nc = std::min(slab, n - j0);
    tril_slab_kernel<<<grid2(n, nc), 256, 0, c->stream>>>(dM, ld, n, j0, nc, tmp);
    c->launches++;
    cudaMemcpyAsync(host + j0 * n, tmp, sizeof(double) * n * nc, cudaMemcpyDeviceToHost, c->stream);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) {
      rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
      break;
    }
  }
  dfree(tmp);
  return rc;
}

// host K (n x n) -> padded device square with diag_add on the diagonal
static int upload_square_padded(gprc_ctx* c, const double* hostK, long n, double* dst, long n_pad, double diag_add,
                                bool pad_identity) {
  double* stage = nullptr;
  const long slab = std::max<long>(1, std::min<long>(n_pad, (256L << 20) / 8 / std::max<long>(n, 1)));
  GPRC_CHECK(dmalloc(&stage, (size_t)n * slab));
  int rc = 0;
  for (long j0 = 0; j0 < n_pad; j0 += slab) {
    const long nc = std::min(slab, n_pad - j0);
    const long ncv = std::max<long>(0, std::min(nc, n - j0));
    if (ncv > 0) cudaMemcpyAsync(stage, hostK + j0 * n, sizeof(double) * n * ncv, cudaMemcpyHostToDevice, c->stream);
    place_slab_kernel<<<grid2(n_pad, nc), 256, 0, c->stream>>>(stage, n, j0, ncv, dst, n_pad, n_pad, nc, diag_add,
                                                               pad_identity ? 1 : 0);
    c->launches++;
    cudaError_t e = cudaStreamSynchronize(c->stream);  // the staging buffer is reused by the next slab
    if (e != cudaSuccess) {
      rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
      break;
    }
  }
  dfree(stage);
  return rc;
}

// =================================================================================================================
// (2)+(3) GPR
// =================================================================================================================
static void gpr_destroy(gprc_gpr* g) {
  if (!g) return;
  dfree(g->X);
  dfree(g->y);
  dfree(g->alpha);
  g->F.release();
  g->ws.release();
  delete g;
}

// K (+ noise I, identity padding) is already in g->F.L; factor, solve, reduce.
static int gpr_finish_fit(gprc_ctx* c, gprc_gpr* g, double* logp, long* info) {
  FactorState& F = g->F;
  GPRC_CHECK(factor_run(c, F, info));
  if (*info != 0) return 0;
  double *work = nullptr, *tmp = nullptr;
  GPRC_CHECK(dmalloc(&work, (size_t)F.n_pad));
  GPRC_CHECK(dmalloc(&tmp, (size_t)F.n_pad));
  int rc = 0;
  {
    PhaseTimer t(c, GPRC_T_SOLVE);
    rc = potrs_vec(c, F.L, F.n_pad, F.n_pad, F.dinv, g->y, work, tmp, g->alpha);
    if (rc == 0) {
      gp_reduce_kernel<<<1, 1024, 0, c->stream>>>(g->y, g->alpha, F.diag, F.n, c->d_scalars);
      c->launches++;
    }
  }
  if (rc == 0) {
    cudaMemcpyAsync(c->h_scalars, c->d_scalars, 4 * sizeof(double), cudaMemcpyDeviceToHost, c->stream);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
  }
  dfree(work);
  dfree(tmp);
  if (rc) return rc;
  // -0.5 * y %*% alpha - sum(log(diag(L))) - n / 2 * log(2 * pi)        R/GPRclass.R:153
  g->logp = -0.5 * c->h_scalars[0] - c->h_scalars[1] - (double)F.n / 2.0 * log(2.0 * M_PI);
  if (logp) *logp = g->logp;
  return 0;
}

static int gpr_fit_common(gprc_ctx* c, const gprc_kernel* k, const double* X, bool x_on_device, int d, long n,
                          const double* y, bool y_on_device, const double* Kpre, double noise, gprc_gpr** out,
                          double* logp, long* info, double* min_leading_logdet) {
  GPRC_ARG(c && out && info && y && n > 0 && noise >= 0.0);
  GPRC_ARG(Kpre != nullptr || (k != nullptr && X != nullptr && d > 0));
  *out = nullptr;
  *info = 0;
  DeviceGuard guard(c);
  gprc_gpr* g = new gprc_gpr();
  g->ctx = c;
  g->d = d;
  g->noise = noise;
  g->precomputed = (Kpre != nullptr);
  int rc = 0;
  do {
    if ((rc = factor_alloc(g->F, n))) break;
    FactorState& F = g->F;
    if ((rc = dmalloc(&g->y, (size_t)F.n_pad))) break;
    if ((rc = dmalloc(&g->alpha, (size_t)F.n_pad))) break;
    cudaMemsetAsync(g->y, 0, sizeof(double) * F.n_pad, c->stream);
    cudaMemcpyAsync(g->y, y, sizeof(double) * n, y_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice,
                    c->stream);
    if (Kpre) {
      // K + new_noise * diag(n) with K supplied by the host (closure kernels, R/GPRclass.R:133,142)
      PhaseTimer t(c, GPRC_T_BUILD_K);
      rc = upload_square_padded(c, Kpre, n, F.L, F.n_pad, noise, true);
    } else {
      if ((rc = make_spec(c, k, d, g->spec))) break;
      g->khost = *k;
      if ((rc = dmalloc(&g->X, (size_t)d * n))) break;
      cudaMemcpyAsync(g->X, X, sizeof(double) * d * n, x_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice,
                      c->stream);
      PhaseTimer t(c, GPRC_T_BUILD_K);
      rc = cov_build_dev(c, g->spec.dev, g->X, d, n, g->X, n, F.L, F.n_pad, F.n_pad, F.n_pad, true, true, noise, true,
                         nullptr, nullptr, nullptr, 0);
    }
    if (rc) break;
    if ((rc = gpr_finish_fit(c, g, logp, info))) break;
    if (min_leading_logdet && *info == 0) *min_leading_logdet = c->h_scalars[3];
  } while (0);
  if (rc != 0 || *info != 0) {
    cudaStreamSynchronize(c->stream);
    gpr_destroy(g);
    return rc;
  }
  *out = g;
  return 0;
}

extern "C" int gprc_gpr_fit(gprc_ctx* c, const gprc_kernel* k, const double* X, int d, long n, const double* y,
                            double noise, gprc_gpr** out, double* logp, long* info) {
  return gpr_fit_common(c, k, X, false, d, n, y, false, nullptr, noise, out, logp, info, nullptr);
}
extern "C" int gprc_gpr_fit_dev(gprc_ctx* c, const gprc_kernel* k, const double* dX, int d, long n, const double* dy,
                                double noise, gprc_gpr** out, double* logp, long* info) {
  return gpr_fit_common(c, k, dX, true, d, n, dy, true, nullptr, noise, out, logp, info, nullptr);
}
extern "C" int gprc_gpr_fit_precomputed(gprc_ctx* c, const double* K, long n, const double* y, double noise,
                                        gprc_gpr** out, double* logp, long* info) {
  GPRC_ARG(K != nullptr);
  return gpr_fit_common(c, nullptr, nullptr, false, 0, n, y, false, K, noise, out, logp, info, nullptr);
}

// Append k training points in place.  The leading n0 x n0 block of the factor (n0 = 128 floor(n / 128)) stays valid;
// rows n0 .. n + k - 1 -- the old partial block row plus the new points, k' <= k + 127 of them -- are recomputed, so that
// every step works on 128-aligned blocks:
//   build  L[n0:, :n0] = K(X_new', X[:, :n0]),  L[n0:, n0:] = K(X_new', X_new') + noise I   (X_new' = points n0 ..)
//   solve  L[n0:, :n0] <- L[n0:, :n0] L11^-T      trsm_flow_kernel
//   Schur  L[n0:, n0:] -= L[n0:, :n0] L[n0:, :n0]^T  SyrkPolicy on the lower tiles
//   factor L[n0:, n0:] in place                  potrf_blocked (inverted diagonal blocks and diag come with it)
// then alpha and logp over the whole new factor as in gpr_finish_fit.  Costs n0^3 / 3 flops less than a refit.
// When n + k outgrows the padding, every buffer is reallocated at round_up(n + k, 128) and L[:n0, :n0] is copied over
// (the old buffers are released only once the new factor is complete).  Otherwise the rows that are overwritten -- the old
// block row n0 / 128, its inverted diagonal block and diagonal entries -- are saved first: on info > 0 they are put back,
// so a failed append leaves the model exactly as it was.  Derived state (W = L^-1, the INT8 digit planes, the predict
// workspace) is dropped on success and rebuilt by the next predict that needs it.
extern "C" int gprc_gpr_append(gprc_gpr* g, const double* Xnew, long k, const double* ynew, double* logp, long* info) {
  GPRC_ARG(g && Xnew && ynew && logp && info && k > 0);
  GPRC_ARG(!g->precomputed);  // closure kernels: the host refits with K built from the closure
  gprc_ctx* c = g->ctx;
  DeviceGuard guard(c);
  *info = 0;
  FactorState& F = g->F;
  const int d = g->d;
  const long n = F.n, n1 = n + k, n0 = n / NB * NB;
  const bool grow = round_up(n1, NB) > F.n_pad;
  const long ld = grow ? round_up(n1, NB) : F.n_pad;  // leading dimension = padded order, as everywhere
  const long rows = ld - n0;                          // rows recomputed, padding included
  double *X = nullptr, *L = F.L, *dinv = F.dinv, *diag = F.diag, *y = g->y, *alpha = g->alpha;
  double *save = nullptr, *work = nullptr, *tmp = nullptr;
  int* sched = nullptr;
  bool restore = false;
  int rc = 0;
  do {
    if ((rc = dmalloc(&X, (size_t)d * n1))) break;
    cudaMemcpyAsync(X, g->X, sizeof(double) * d * n, cudaMemcpyDeviceToDevice, c->stream);
    cudaMemcpyAsync(X + d * n, Xnew, sizeof(double) * d * k, cudaMemcpyHostToDevice, c->stream);
    if (grow) {
      L = dinv = diag = y = alpha = nullptr;
      if ((rc = dmalloc(&L, (size_t)ld * ld))) break;
      if ((rc = dmalloc(&dinv, (size_t)ld * NB))) break;
      if ((rc = dmalloc(&diag, (size_t)ld))) break;
      if ((rc = dmalloc(&y, (size_t)ld))) break;
      if ((rc = dmalloc(&alpha, (size_t)ld))) break;
      if (n0 > 0) {
        cudaMemcpy2DAsync(L, ld * sizeof(double), F.L, F.n_pad * sizeof(double), n0 * sizeof(double), n0,
                          cudaMemcpyDeviceToDevice, c->stream);
        cudaMemcpyAsync(dinv, F.dinv, sizeof(double) * n0 * NB, cudaMemcpyDeviceToDevice, c->stream);
        cudaMemcpyAsync(diag, F.diag, sizeof(double) * n0, cudaMemcpyDeviceToDevice, c->stream);
      }
      cudaMemsetAsync(y, 0, sizeof(double) * ld, c->stream);
      cudaMemcpyAsync(y, g->y, sizeof(double) * n, cudaMemcpyDeviceToDevice, c->stream);
    } else {
      // block row n0 / 128 (all ld columns), then its inverted diagonal block and its diagonal entries
      if ((rc = dmalloc(&save, (size_t)NB * ld + NB * NB + NB))) break;
      cudaMemcpy2DAsync(save, NB * sizeof(double), L + n0, ld * sizeof(double), NB * sizeof(double), ld,
                        cudaMemcpyDeviceToDevice, c->stream);
      cudaMemcpyAsync(save + NB * ld, dinv + n0 * NB, sizeof(double) * NB * NB, cudaMemcpyDeviceToDevice, c->stream);
      cudaMemcpyAsync(save + NB * ld + NB * NB, diag + n0, sizeof(double) * NB, cudaMemcpyDeviceToDevice, c->stream);
      restore = true;
    }
    cudaMemcpyAsync(y + n, ynew, sizeof(double) * k, cudaMemcpyHostToDevice, c->stream);
    {
      PhaseTimer t(c, GPRC_T_BUILD_K);
      if (n0 > 0 && (rc = cov_build_dev(c, g->spec.dev, X + d * n0, d, n1 - n0, X, n0, L + n0, ld, rows, n0, false, false,
                                        0.0, false, nullptr, nullptr, nullptr, 0)))
        break;
      if ((rc = cov_build_dev(c, g->spec.dev, X + d * n0, d, n1 - n0, X + d * n0, n1 - n0, L + n0 + n0 * ld, ld, rows,
                              rows, true, true, g->noise, true, nullptr, nullptr, nullptr, 0)))
        break;
    }
    *c->h_info = LONG_MAX;
    cudaMemcpyAsync(c->d_info, c->h_info, sizeof(long), cudaMemcpyHostToDevice, c->stream);
    {
      PhaseTimer t(c, GPRC_T_CHOL);
      if (n0 > 0) {
        if ((rc = dmalloc(&sched, (size_t)(rows / NB + 4)))) break;
        if ((rc = trsm_flow(c, L, ld, dinv, (int)(n0 / NB), L + n0, ld, rows, sched))) break;
        const long t1 = rows / NB;
        SyrkPolicy sp{L, ld, 1, (int)(n0 / NB), 0, (int)n0};
        if ((rc = launch_gemm(c, sp, dim3((unsigned)(t1 * (t1 + 1) / 2))))) break;
      }
      if ((rc = potrf_blocked(c, L + n0 + n0 * ld, rows, ld, dinv + n0 * NB, c->d_info, diag + n0))) break;
    }
    int* h_error = reinterpret_cast<int*>(c->h_scalars + 8);  // pinned
    *h_error = 0;
    if (sched) cudaMemcpyAsync(h_error, sched + 2, sizeof(int), cudaMemcpyDeviceToHost, c->stream);
    cudaMemcpyAsync(c->h_info, c->d_info, sizeof(long), cudaMemcpyDeviceToHost, c->stream);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) {
      rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
      break;
    }
    if (*h_error) {
      rc = set_error(-6, __FILE__, __LINE__, "triangular solve of the appended rows: a block dependency never arrived");
      break;
    }
    if (*c->h_info != LONG_MAX) {
      *info = n0 + *c->h_info;
      break;
    }
    // alpha and logp over the whole new factor
    if ((rc = dmalloc(&work, (size_t)ld))) break;
    if ((rc = dmalloc(&tmp, (size_t)ld))) break;
    {
      PhaseTimer t(c, GPRC_T_SOLVE);
      if ((rc = potrs_vec(c, L, ld, ld, dinv, y, work, tmp, alpha))) break;
      gp_reduce_kernel<<<1, 1024, 0, c->stream>>>(y, alpha, diag, n1, c->d_scalars);
      c->launches++;
    }
    cudaMemcpyAsync(c->h_scalars, c->d_scalars, 4 * sizeof(double), cudaMemcpyDeviceToHost, c->stream);
    e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) {
      rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
      break;
    }
    restore = false;
  } while (0);
  dfree(sched);
  dfree(work);
  dfree(tmp);
  if (rc != 0 || *info != 0) {
    if (restore) {  // the old block row, its inverted diagonal block and diagonal; y's padding back to zero
      cudaMemcpy2DAsync(L + n0, ld * sizeof(double), save, NB * sizeof(double), NB * sizeof(double), ld,
                        cudaMemcpyDeviceToDevice, c->stream);
      cudaMemcpyAsync(dinv + n0 * NB, save + NB * ld, sizeof(double) * NB * NB, cudaMemcpyDeviceToDevice, c->stream);
      cudaMemcpyAsync(diag + n0, save + NB * ld + NB * NB, sizeof(double) * NB, cudaMemcpyDeviceToDevice, c->stream);
      cudaMemsetAsync(y + n, 0, sizeof(double) * (F.n_pad - n), c->stream);
    }
    if (grow) {
      dfree(L);
      dfree(dinv);
      dfree(diag);
      dfree(y);
      dfree(alpha);
    }
    dfree(X);
    dfree(save);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (rc == 0 && e != cudaSuccess) rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
    return rc;
  }
  dfree(save);
  if (grow) {
    dfree(F.L);
    dfree(F.dinv);
    dfree(F.diag);
    dfree(g->y);
    dfree(g->alpha);
    F.L = L;
    F.dinv = dinv;
    F.diag = diag;
    F.n_pad = ld;
    g->y = y;
    g->alpha = alpha;
  }
  dfree(g->X);
  g->X = X;
  F.n = n1;
  // derived from the old factor: rebuilt on demand by the next predict
  dfree(F.W);
  dfree(F.ozLs);
  dfree(F.oz_erow);
  dfree(F.oz_srow);
  F.W = nullptr;
  F.ozLs = nullptr;
  F.oz_erow = nullptr;
  F.oz_srow = nullptr;
  F.oz_digits = 0;
  g->ws.release();
  // -0.5 * y %*% alpha - sum(log(diag(L))) - n / 2 * log(2 * pi)        R/GPRclass.R:153
  g->logp = -0.5 * c->h_scalars[0] - c->h_scalars[1] - (double)n1 / 2.0 * log(2.0 * M_PI);
  *logp = g->logp;
  return 0;
}

extern "C" int gprc_gpr_predict_dev(gprc_gpr* g, const double* dXs, long m, double* dmean, double* dvar) {
  GPRC_ARG(g && dXs && dmean && dvar && m >= 0);
  GPRC_ARG(!g->precomputed);
  if (m == 0) return 0;
  DeviceGuard guard(g->ctx);
  return predict_pointwise_dev(g->ctx, g->spec.dev, g->X, g->d, g->F, g->ws, g->alpha, nullptr, dXs, m, dmean, dvar);
}

// ---- test grids on the device (SURVEY.md 8f-4): combine_all(lapply(1:D, seq(lo, hi, length.out = per_dim))) ------------
namespace gprc {
// out: d x m (points contiguous), m = per_dim^d; the FIRST dimension varies slowest, the last fastest
// (R/simulation.R:338-349: row k = rep(rep(lst[[k]], each = prod(lengths after k)), times = prod(lengths before k))).
// seq(lo, hi, length.out = n) as numpy.linspace evaluates it: lo + i * ((hi - lo) / (n - 1)), last point = hi exactly.
__global__ void __launch_bounds__(256) grid_points_kernel(const double* __restrict__ limits /* d x 2: lo, hi */, int d,
                                                          int per_dim, long m, double* __restrict__ out) {
  const long j = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  long rest = j;
  for (int k = d - 1; k >= 0; --k) {
    const int i = (int)(rest % per_dim);
    rest /= per_dim;
    const double lo = limits[2 * k], hi = limits[2 * k + 1];
    double v = lo;
    if (per_dim > 1) {
      const double step = (hi - lo) / (double)(per_dim - 1);
      v = (i == per_dim - 1) ? hi : __dadd_rn(__dmul_rn((double)i, step), lo);
    }
    out[j * d + k] = v;
  }
}
}  // namespace gprc

static int grid_size(int d, int per_dim, long* m) {
  GPRC_ARG(d > 0 && per_dim > 0);
  long t = 1;
  for (int k = 0; k < d; ++k) {
    if (t > (1L << 40) / per_dim) return set_error(-1, __FILE__, __LINE__, "grid too large");
    t *= per_dim;
  }
  *m = t;
  return 0;
}

extern "C" int gprc_grid_points(gprc_ctx* c, const double* limits, int d, int per_dim, double* out) {
  GPRC_ARG(c && limits && out);
  long m = 0;
  GPRC_CHECK(grid_size(d, per_dim, &m));
  DeviceGuard guard(c);
  double *dl = nullptr, *dout = nullptr;
  GPRC_CHECK(dmalloc(&dl, (size_t)2 * d));
  int rc = dmalloc(&dout, (size_t)d * m);
  if (!rc) {
    cudaMemcpyAsync(dl, limits, sizeof(double) * 2 * d, cudaMemcpyHostToDevice, c->stream);
    grid_points_kernel<<<(unsigned)((m + 255) / 256), 256, 0, c->stream>>>(dl, d, per_dim, m, dout);
    c->launches++;
    cudaMemcpyAsync(out, dout, sizeof(double) * d * m, cudaMemcpyDeviceToHost, c->stream);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
  }
  dfree(dl);
  dfree(dout);
  return rc;
}

// $predict on the grid simulate_regression() builds (R/simulation.R:101-102) without the grid ever existing on the host
extern "C" int gprc_gpr_predict_grid(gprc_gpr* g, const double* limits, int per_dim, double* mean, double* var) {
  GPRC_ARG(g && limits && mean && var);
  GPRC_ARG(!g->precomputed);
  long m = 0;
  GPRC_CHECK(grid_size(g->d, per_dim, &m));
  gprc_ctx* c = g->ctx;
  DeviceGuard guard(c);
  double *dl = nullptr, *dXs = nullptr, *dmean = nullptr, *dvar = nullptr;
  int rc = 0;
  do {
    if ((rc = dmalloc(&dl, (size_t)2 * g->d))) break;
    if ((rc = dmalloc(&dXs, (size_t)g->d * m))) break;
    if ((rc = dmalloc(&dmean, (size_t)m))) break;
    if ((rc = dmalloc(&dvar, (size_t)m))) break;
    cudaMemcpyAsync(dl, limits, sizeof(double) * 2 * g->d, cudaMemcpyHostToDevice, c->stream);
    grid_points_kernel<<<(unsigned)((m + 255) / 256), 256, 0, c->stream>>>(dl, g->d, per_dim, m, dXs);
    c->launches++;
    if ((rc = predict_pointwise_dev(c, g->spec.dev, g->X, g->d, g->F, g->ws, g->alpha, nullptr, dXs, m, dmean, dvar)))
      break;
    cudaMemcpyAsync(mean, dmean, sizeof(double) * m, cudaMemcpyDeviceToHost, c->stream);
    cudaMemcpyAsync(var, dvar, sizeof(double) * m, cudaMemcpyDeviceToHost, c->stream);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
  } while (0);
  cudaStreamSynchronize(c->stream);
  dfree(dl);
  dfree(dXs);
  dfree(dmean);
  dfree(dvar);
  return rc;
}

extern "C" int gprc_gpr_predict(gprc_gpr* g, const double* Xs, long m, double* mean, double* var) {
  GPRC_ARG(g && Xs && mean && var && m >= 0);
  GPRC_ARG(!g->precomputed);
  if (m == 0) return 0;
  gprc_ctx* c = g->ctx;
  DeviceGuard guard(c);
  double *dXs = nullptr, *dmean = nullptr, *dvar = nullptr;
  int rc = 0;
  do {
    if ((rc = dmalloc(&dXs, (size_t)g->d * m))) break;
    if ((rc = dmalloc(&dmean, (size_t)m))) break;
    if ((rc = dmalloc(&dvar, (size_t)m))) break;
    cudaMemcpyAsync(dXs, Xs, sizeof(double) * g->d * m, cudaMemcpyHostToDevice, c->stream);
    if ((rc = predict_pointwise_dev(c, g->spec.dev, g->X, g->d, g->F, g->ws, g->alpha, nullptr, dXs, m, dmean, dvar)))
      break;
    cudaMemcpyAsync(mean, dmean, sizeof(double) * m, cudaMemcpyDeviceToHost, c->stream);
    cudaMemcpyAsync(var, dvar, sizeof(double) * m, cudaMemcpyDeviceToHost, c->stream);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
  } while (0);
  dfree(dXs);
  dfree(dmean);
  dfree(dvar);
  return rc;
}

extern "C" int gprc_gpr_predict_precomputed(gprc_gpr* g, const double* Ks, const double* kss, long m, double* mean,
                                            double* var) {
  GPRC_ARG(g && Ks && kss && mean && var && m >= 0);
  if (m == 0) return 0;
  DeviceGuard guard(g->ctx);
  return predict_precomputed(g->ctx, g->F, g->ws, g->alpha, nullptr, Ks, kss, m, mean, var);
}

// predict(X_star, pointwise_var = FALSE): Sigma = covariance_matrix(X_star, X_star, k) - t(v) %*% v   R/GPRclass.R:167
extern "C" int gprc_gpr_predict_cov(gprc_gpr* g, const double* Xs, long m, double* mean, double* cov) {
  GPRC_ARG(g && Xs && mean && cov && m > 0);
  GPRC_ARG(!g->precomputed);
  gprc_ctx* c = g->ctx;
  DeviceGuard guard(c);
  FactorState& F = g->F;
  const long mp = round_up(m, NB);
  GPRC_CHECK(ensure_inverse(c, F));
  int mean_tile = CT;
  PredictWorkspace ws;  // private workspace sized for the whole set (V^T must be complete before the product)
  double *dXs = nullptr, *dmean = nullptr, *dVt = nullptr, *dS = nullptr;
  int rc = 0;
  do {
    if ((rc = dmalloc(&ws.Ks, (size_t)F.n_pad * mp))) break;  // K_star^T, mp x n_pad
    if ((rc = dmalloc(&ws.pmean, (size_t)(F.n_pad / CT) * mp))) break;
    if ((rc = dmalloc(&ws.pvar, (size_t)(F.n_pad / NB) * mp))) break;
    if ((rc = dmalloc(&ws.kss, (size_t)mp))) break;
    ws.mc = mp;
    if ((rc = dmalloc(&dXs, (size_t)g->d * m))) break;
    if ((rc = dmalloc(&dmean, (size_t)mp))) break;
    if ((rc = dmalloc(&dVt, (size_t)mp * F.n_pad))) break;
    if ((rc = dmalloc(&dS, (size_t)mp * mp))) break;
    cudaMemcpyAsync(dXs, Xs, sizeof(double) * g->d * m, cudaMemcpyHostToDevice, c->stream);
    {
      PhaseTimer t(c, GPRC_T_BUILD_KS);
      if ((rc = cov_build_dev(c, g->spec.dev, dXs, g->d, m, g->X, F.n, ws.Ks, mp, mp, F.n_pad, false, false, 0.0,
                              false, nullptr, nullptr, ws.pmean, ws.mc, nullptr, g->alpha, &mean_tile)))
        break;
      // Sigma starts as covariance_matrix(X_star, X_star, k); zero padding
      if ((rc = cov_build_dev(c, g->spec.dev, dXs, g->d, m, dXs, m, dS, mp, mp, mp, false, false, 0.0, false, nullptr,
                              nullptr, nullptr, 0)))
        break;
    }
    if ((rc = variance_pass(c, F, ws, mp, dVt, mp))) break;
    finalize_predict_kernel<<<(unsigned)((m + 255) / 256), 256, 0, c->stream>>>(
        ws.pmean, ws.mc, (int)(F.n_pad / mean_tile), nullptr, 0, 0, nullptr, m, dmean, nullptr);
    c->launches++;
    {
      // Sigma -= V^T V  with V^T stored m_pad x n_pad (test point contiguous): C = C - A A^T
      PhaseTimer t(c, GPRC_T_VAR);
      DgemmPolicy<false> p;
      p.A = dVt;
      p.lda = mp;
      p.B = dVt;
      p.ldb = mp;
      p.C = dS;
      p.ldc = mp;
      p.alpha = -1.0;
      p.beta = 1.0;
      p.K = (int)F.n_pad;
      p.tiles_m = (int)(mp / NB);
      if ((rc = launch_gemm(c, p, dim3((unsigned)((mp / NB) * (mp / NB)))))) break;
    }
    cudaMemcpyAsync(mean, dmean, sizeof(double) * m, cudaMemcpyDeviceToHost, c->stream);
    cudaMemcpy2DAsync(cov, m * sizeof(double), dS, mp * sizeof(double), m * sizeof(double), m, cudaMemcpyDeviceToHost,
                      c->stream);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
  } while (0);
  cudaStreamSynchronize(c->stream);
  ws.release();
  dfree(dXs);
  dfree(dmean);
  dfree(dVt);
  dfree(dS);
  return rc;
}

extern "C" int gprc_gpr_get(gprc_gpr* g, int what, double* host) {
  GPRC_ARG(g && host);
  gprc_ctx* c = g->ctx;
  DeviceGuard guard(c);
  switch (what) {
    case GPRC_GET_L: return download_lower(c, g->F.L, g->F.n, g->F.n_pad, host);
    case GPRC_GET_LINV:
      GPRC_CHECK(ensure_inverse(c, g->F));
      return download_lower(c, g->F.W, g->F.n, g->F.n_pad, host);
    case GPRC_GET_ALPHA: return gprc_dev_d2h(c, host, g->alpha, sizeof(double) * g->F.n);
    default: return set_error(-1, __FILE__, __LINE__, "gprc_gpr_get: unknown item");
  }
}
extern "C" long gprc_gpr_n(const gprc_gpr* g) { return g ? g->F.n : 0; }
extern "C" int gprc_gpr_dim(const gprc_gpr* g) { return g ? g->d : 0; }
extern "C" void gprc_gpr_free(gprc_gpr* g) {
  if (!g) return;
  DeviceGuard guard(g->ctx);
  cudaStreamSynchronize(g->ctx->stream);
  gpr_destroy(g);
}

// =================================================================================================================
// fit(): dens / dens_deriv
// =================================================================================================================
extern "C" int gprc_logml(gprc_ctx* c, const gprc_kernel* k, const double* X, int d, long n, const double* y,
                          double noise, double* logp, double* min_leading_logdet, long* info) {
  GPRC_ARG(logp && info);
  gprc_gpr* g = nullptr;
  GPRC_CHECK(gpr_fit_common(c, k, X, false, d, n, y, false, nullptr, noise, &g, logp, info, min_leading_logdet));
  if (g) gprc_gpr_free(g);
  return 0;
}

extern "C" int gprc_logml_batch(gprc_ctx* c, const gprc_kernel* specs, int nspec, const double* X, int d, long n,
                                const double* y, double noise, double* logp, double* min_leading_logdet, long* info) {
  GPRC_ARG(c && specs && nspec >= 0 && X && y && logp && info && n > 0 && d > 0);
  DeviceGuard guard(c);
  // X and y are uploaded once; every evaluation reuses them on the device
  double *dX = nullptr, *dy = nullptr;
  int rc = 0;
  do {
    if ((rc = dmalloc(&dX, (size_t)d * n))) break;
    if ((rc = dmalloc(&dy, (size_t)n))) break;
    cudaMemcpyAsync(dX, X, sizeof(double) * d * n, cudaMemcpyHostToDevice, c->stream);
    cudaMemcpyAsync(dy, y, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream);
    for (int s = 0; s < nspec && rc == 0; ++s) {
      gprc_gpr* g = nullptr;
      double lp = 0.0, ml = 0.0;
      long inf = 0;
      rc = gpr_fit_common(c, &specs[s], dX, true, d, n, dy, true, nullptr, noise, &g, &lp, &inf, &ml);
      logp[s] = (inf == 0) ? lp : NAN;
      if (min_leading_logdet) min_leading_logdet[s] = (inf == 0) ? ml : NAN;
      info[s] = inf;
      if (g) gprc_gpr_free(g);
    }
  } while (0);
  cudaStreamSynchronize(c->stream);
  dfree(dX);
  dfree(dy);
  return rc;
}

// ---- dens_deriv, R/fit.R:126-139 ---------------------------------------------------------------------------------
namespace gprc {
// d k / d v[0], d k / d v[1] for one pair.  textbook != 0: derivative of the kernel w.r.t. the optimiser's parameter
// vector v in the kernel's own positional order (sqrexp (l); gammaexp (l, gamma); rationalquadratic (l, alpha);
// polynomial (sigma, p)).  textbook == 0: the reference's cov_dict[[*]]$deriv called positionally with v, which for
// gammaexp / rationalquadratic reads v[0] as gamma / alpha and v[1] as l (R/fit.R:10,25 vs R/GPRclass.R:397,401; A.6).
__device__ __forceinline__ void kderiv(int id, int textbook, double v0, double v1, double s /* r2 or dot */,
                                       double& d0, double& d1) {
  d0 = d1 = 0.0;
  if (id == GPRC_SQREXP) {  // r^2/l^3 * exp(-r^2/(l^2 * 2))                                      R/fit.R:4-7
    const double l = v0;
    d0 = s / (l * l * l) * exp(-s / (l * l * 2.0));
  } else if (id == GPRC_POLYNOMIAL) {  // c(p (x.y + sigma)^(p-1), (x.y + sigma)^p log(x.y + sigma))  R/fit.R:20-22
    const double b = s + v0, p = v1;
    d0 = p * pow(b, p - 1.0);
    d1 = pow(b, p) * log(b);
  } else if (id == GPRC_GAMMAEXP) {
    const double r = sqrt(s);
    if (textbook) {
      const double l = v0, g = v1, q = pow(r / l, g), e = exp(-q);
      d0 = e * g * q / l;
      d1 = (r > 0.0) ? -e * q * log(r / l) : 0.0;
    } else {  // deriv(x, y, gamma = v[0], l = v[1])                                               R/fit.R:10-13
      const double g = v0, l = v1, q = pow(r / l, g), e = exp(-q);
      d0 = -e * q * log(r / l);  // NaN at r = 0, exactly like R (0 * -Inf)
      d1 = e * g * pow(r, g) / pow(l, g + 1.0);
    }
  } else if (id == GPRC_RATQUAD) {
    if (textbook) {
      const double l = v0, a = v1, base = 1.0 + s / (2.0 * a * l * l);
      d0 = s / (l * l * l) * pow(base, -a - 1.0);
      d1 = pow(base, -a) * (-log(base) + s / (2.0 * a * l * l * base));
    } else {  // deriv(x, y, alpha = v[0], l = v[1])                                                R/fit.R:25-31
      const double a = v0, l = v1, t = 2.0 * l * l * a, base = s / t + 1.0;
      d0 = (pow(base, -a) * (s - (t + s) * log(base))) / (t + s);
      d1 = (s * pow(base, -a - 1.0)) / (l * l * l);
    }
  }
}

// dK0, dK1 (n_pad x n_pad, zero padding) for all pairs of columns of X
__global__ void __launch_bounds__(256) dk_tile_kernel(int id, int textbook, double v0, double v1,
                                                      const double* __restrict__ X, int d, long n, long n_pad,
                                                      double* __restrict__ dK0, double* __restrict__ dK1) {
  const long i = blockIdx.x * 16L + (threadIdx.x & 15), j = blockIdx.y * 16L + (threadIdx.x >> 4);
  if (i >= n_pad || j >= n_pad) return;
  double d0 = 0.0, d1 = 0.0;
  if (i < n && j < n) {
    double s = 0.0;
    const bool dist = (id != GPRC_POLYNOMIAL);
    for (int dd = 0; dd < d; ++dd) {
      const double a = X[i * d + dd], b = X[j * d + dd];
      s = dist ? __dadd_rn(s, __dmul_rn(a - b, a - b)) : __dadd_rn(s, __dmul_rn(a, b));
    }
    kderiv(id, textbook, v0, v1, s, d0, d1);
  }
  dK0[i + j * n_pad] = d0;
  if (dK1) dK1[i + j * n_pad] = d1;
}
// out[k] = sum_{i >= k} W[i, k]^2 = (L^-T L^-1)_kk : warp per column
__global__ void __launch_bounds__(256) colnorm2_lower_kernel(const double* __restrict__ W, long ld, long n,
                                                             double* __restrict__ out) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long col = (long)blockIdx.x * 8 + warp;
  if (col >= n) return;
  const double* Wp = W + col * ld;
  double s = 0.0;
  for (long i = col + lane; i < n; i += 32) s = fma(Wp[i], Wp[i], s);
  s = warp_sum(s);
  if (lane == 0) out[col] = s;
}
// single-CTA reductions: mode 0: out = 0.5 * sum_k (alpha_k^2 - kd_k) rs_k ; mode 1: out = sum_k a_k b_k
__global__ void __launch_bounds__(1024) grad_reduce_kernel(int mode, const double* __restrict__ a,
                                                           const double* __restrict__ b, const double* __restrict__ c,
                                                           long n, double* __restrict__ out) {
  __shared__ double sh[1024];
  const int tid = threadIdx.x;
  const long chunk = (n + 1023) / 1024;
  const long lo = tid * chunk, hi = (lo + chunk < n) ? lo + chunk : n;
  double s = 0.0;
  for (long i = lo; i < hi; ++i) s += (mode == 0) ? (a[i] * a[i] - b[i]) * c[i] : a[i] * b[i];
  sh[tid] = s;
  __syncthreads();
  if (tid == 0) {
    double t = 0.0;
    for (int q = 0; q < 1024; ++q) t += sh[q];
    out[0] = (mode == 0) ? 0.5 * t : t;
  }
}
// partial[b] = sum over the columns j = b, b + gridDim.x, ... of sum_{i >= j} W[i + j ld] Z[i + j ld]
// (tr(W^T Z) for lower-triangular W); the caller adds the partials in a fixed order
__global__ void __launch_bounds__(256) tril_dot_partial_kernel(const double* __restrict__ W, const double* __restrict__ Z,
                                                               long ld, long n, double* __restrict__ partial) {
  __shared__ double sh[256];
  const int tid = threadIdx.x;
  double s = 0.0;
  for (long j = blockIdx.x; j < n; j += gridDim.x)
    for (long i = j + tid; i < n; i += 256) s = fma(W[i + j * ld], Z[i + j * ld], s);
  sh[tid] = s;
  __syncthreads();
  if (tid == 0) {
    double t = 0.0;
    for (int q = 0; q < 256; ++q) t += sh[q];
    partial[blockIdx.x] = t;
  }
}
__global__ void sum_partials_kernel(const double* __restrict__ partial, int n, double* __restrict__ out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double t = 0.0;
    for (int q = 0; q < n; ++q) t += partial[q];
    out[0] = t;
  }
}
}  // namespace gprc

static int logml_grad_impl(gprc_ctx* c, const gprc_kernel* k, const double* X, bool x_on_device, int d, long n,
                           const double* y, bool y_on_device, double noise, int formula, double* grad, int nparam,
                           long* info) {
  GPRC_ARG(c && k && X && y && grad && info && n > 0 && d > 0);
  GPRC_ARG(k->id == GPRC_SQREXP || k->id == GPRC_GAMMAEXP || k->id == GPRC_RATQUAD || k->id == GPRC_POLYNOMIAL);
  const int np_expected = (k->id == GPRC_SQREXP) ? 1 : 2;
  GPRC_ARG(nparam == np_expected);
  const int textbook = (formula == GPRC_GRAD_TEXTBOOK);
  double v0, v1 = 0.0;
  switch (k->id) {
    case GPRC_SQREXP: v0 = k->l; break;
    case GPRC_GAMMAEXP: v0 = k->l; v1 = k->gamma; break;
    case GPRC_RATQUAD: v0 = k->l; v1 = k->alpha; break;
    default: v0 = k->sigma; v1 = k->p; break;
  }
  // as coded the reference inverts the NOISE-FREE K (R/fit.R:136); the textbook formula uses K + noise I
  gprc_gpr* g = nullptr;
  GPRC_CHECK(gpr_fit_common(c, k, X, x_on_device, d, n, y, y_on_device, nullptr, textbook ? noise : 0.0, &g, nullptr,
                            info, nullptr));
  if (*info != 0 || !g) return 0;
  DeviceGuard guard(c);
  FactorState& F = g->F;
  const long np = F.n_pad;
  double *dK0 = nullptr, *dK1 = nullptr, *vec = nullptr, *ones = nullptr, *Z = nullptr;
  int rc = 0;
  do {
    if ((rc = ensure_inverse(c, F))) break;
    if ((rc = dmalloc(&dK0, (size_t)np * np))) break;
    if (nparam > 1 && (rc = dmalloc(&dK1, (size_t)np * np))) break;
    if ((rc = dmalloc(&vec, (size_t)np * 2 + 256)) || (rc = dmalloc(&ones, (size_t)np))) break;
    dk_tile_kernel<<<dim3((unsigned)(np / 16), (unsigned)(np / 16)), 256, 0, c->stream>>>(k->id, textbook, v0, v1, g->X,
                                                                                         d, n, np, dK0, dK1);
    c->launches++;
    double* dKs[2] = {dK0, dK1};
    if (!textbook) {
      fill_kernel<<<(unsigned)((np + 255) / 256), 256, 0, c->stream>>>(ones, np, 1.0);
      colnorm2_lower_kernel<<<(unsigned)((np + 7) / 8), 256, 0, c->stream>>>(F.W, np, n, vec);  // diag(K^-1)
      c->launches += 2;
      for (int p = 0; p < nparam && rc == 0; ++p) {
        rc = gemv_t(c, dKs[p], np, np, ones, vec + np);  // row sums of dK_p (symmetric)
        grad_reduce_kernel<<<1, 1024, 0, c->stream>>>(0, g->alpha, vec, vec + np, n, c->d_scalars + p);
        c->launches++;
      }
    } else {
      if ((rc = dmalloc(&Z, (size_t)np * np))) break;
      for (int p = 0; p < nparam && rc == 0; ++p) {
        // quad = alpha' dK alpha ; trace = tr(Ky^-1 dK) = tr(W^T (W dK))
        if ((rc = gemv_t(c, dKs[p], np, np, g->alpha, vec))) break;
        grad_reduce_kernel<<<1, 1024, 0, c->stream>>>(1, g->alpha, vec, nullptr, n, c->d_scalars + 8 + p);
        // Z = W dK; dK is symmetric, so it is read as its own transpose (both operands stream in 1 KB runs)
        DgemmPolicy<false> pol{F.W, np, dKs[p], np, Z, np, 1.0, 0.0, (int)np, (int)(np / NB)};
        if ((rc = launch_gemm(c, pol, dim3((unsigned)((np / NB) * (np / NB)))))) break;
        tril_dot_partial_kernel<<<256, 256, 0, c->stream>>>(F.W, Z, np, n, vec + np);
        sum_partials_kernel<<<1, 32, 0, c->stream>>>(vec + np, 256, c->d_scalars + 16 + p);
        c->launches += 3;
      }
    }
    if (rc) break;
    cudaMemcpyAsync(c->h_scalars, c->d_scalars, 24 * sizeof(double), cudaMemcpyDeviceToHost, c->stream);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) {
      rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
      break;
    }
    for (int p = 0; p < nparam; ++p)
      grad[p] = textbook ? 0.5 * (c->h_scalars[8 + p] - c->h_scalars[16 + p]) : c->h_scalars[p];
  } while (0);
  cudaStreamSynchronize(c->stream);
  dfree(dK0);
  dfree(dK1);
  dfree(vec);
  dfree(ones);
  dfree(Z);
  gprc_gpr_free(g);
  return rc;
}

extern "C" int gprc_logml_grad(gprc_ctx* c, const gprc_kernel* k, const double* X, int d, long n, const double* y,
                               double noise, int formula, double* grad, int nparam, long* info) {
  return logml_grad_impl(c, k, X, false, d, n, y, false, noise, formula, grad, nparam, info);
}

// =================================================================================================================
// fit(): the optimiser inside the library (optim.hpp), R/fit.R:47-69, 113-162
// =================================================================================================================
extern "C" int gprc_optim_brent(gprc_objective_fn fn, void* user, double lower, double upper, double tol, double* xmin) {
  GPRC_ARG(fn && xmin);
  try {
    *xmin = optim::brent_fmin(
        [&](double x) {
          double v = 0.0;
          if (fn(&x, 1, user, &v) != 0) throw optim::ObjectiveError{};
          return v;
        },
        lower, upper, tol);
  } catch (const optim::ObjectiveError&) {
    return 1;
  }
  return 0;
}

extern "C" int gprc_optim_vmmin(gprc_objective_fn fn, gprc_gradient_fn gr, void* user, double* par, int npar, int maxit,
                                double abstol, double reltol, double* value, int* counts, int* fail) {
  GPRC_ARG(fn && gr && par && npar > 0 && value);
  try {
    optim::VmminResult r = optim::vmmin(
        par, npar,
        [&](const double* p) {
          double v = 0.0;
          if (fn(p, npar, user, &v) != 0) throw optim::ObjectiveError{};
          return v;
        },
        [&](const double* p, double* g) {
          if (gr(p, npar, user, g) != 0) throw optim::ObjectiveError{};
        },
        maxit, abstol, reltol);
    *value = r.value;
    if (counts) {
      counts[0] = r.fncount;
      counts[1] = r.grcount;
    }
    if (fail) *fail = r.fail;
  } catch (const optim::ObjectiveError&) {
    return 1;
  }
  return 0;
}

extern "C" int gprc_optim_until_error(gprc_objective_fn fn, gprc_gradient_fn gr, void* user, const double* start,
                                      int npar, int method, double lower, double upper, double* par, double* value) {
  GPRC_ARG(fn && start && par && value && npar > 0 && (method == 0 || (method == 1 && gr)));
  GPRC_ARG(method == 1 || npar == 1);
  optim::FnN f = [&](const double* p) {
    double v = 0.0;
    if (fn(p, npar, user, &v) != 0) throw optim::ObjectiveError{};
    return v;
  };
  optim::GrN g = [&](const double* p, double* out) {
    if (gr(p, npar, user, out) != 0) throw optim::ObjectiveError{};
  };
  optim::UntilErrorResult r =
      optim::optim_until_error(std::vector<double>(start, start + npar), f, method == 1 ? &g : nullptr, method == 0,
                               lower, upper);
  for (int i = 0; i < npar; ++i) par[i] = r.par[i];
  *value = r.value;
  return 0;
}

namespace {
// the reference passes the optimiser's vector positionally: do.call(func, append(list(x, y), v)), R/fit.R:118
gprc_kernel family_spec(int id, const double* v) {
  gprc_kernel k{};
  k.id = id;
  switch (id) {
    case GPRC_CONSTANT: k.c = v[0]; break;
    case GPRC_LINEAR: k.sigma = v[0]; break;
    case GPRC_POLYNOMIAL: k.sigma = v[0]; k.p = v[1]; break;
    case GPRC_SQREXP: k.l = v[0]; break;
    case GPRC_GAMMAEXP: k.l = v[0]; k.gamma = v[1]; break;
    case GPRC_RATQUAD: k.l = v[0]; k.alpha = v[1]; break;
  }
  return k;
}
}  // namespace

extern "C" int gprc_fit_family(gprc_ctx* c, int kernel_id, const double* X, int d, long n, const double* y,
                               double noise, int minors_rule, double* par, int* npar, double* value,
                               long* evaluations) {
  GPRC_ARG(c && X && y && par && npar && value && n > 0 && d > 0);
  GPRC_ARG(kernel_id >= GPRC_CONSTANT && kernel_id <= GPRC_RATQUAD);
  DeviceGuard guard(c);
  double *dX = nullptr, *dy = nullptr;
  GPRC_CHECK(dmalloc(&dX, (size_t)d * n));
  int rc = dmalloc(&dy, (size_t)n);
  if (rc) {
    dfree(dX);
    return rc;
  }
  cudaMemcpyAsync(dX, X, sizeof(double) * d * n, cudaMemcpyHostToDevice, c->stream);
  cudaMemcpyAsync(dy, y, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream);
  long n_fn = 0, n_gr = 0;
  int hard_error = 0;  // a CUDA / argument error inside an evaluation: abort the search and report it
  const double log_denorm_min = std::log(std::numeric_limits<double>::denorm_min());
  // dens, R/fit.R:117-124
  auto dens = [&](const double* v) -> double {
    gprc_kernel k = family_spec(kernel_id, v);
    gprc_gpr* g = nullptr;
    double lp = 0.0, ml = 0.0;
    long inf = 0;
    ++n_fn;
    const int r = gpr_fit_common(c, &k, dX, true, d, n, dy, true, nullptr, noise, &g, &lp, &inf, &ml);
    if (g) gprc_gpr_free(g);
    if (r != 0) {
      hard_error = r;
      throw optim::ObjectiveError{};
    }
    if (inf != 0 || !std::isfinite(lp)) throw optim::ObjectiveError{};             // chol() failed
    if (minors_rule == 0 && !(ml >= log_denorm_min)) throw optim::ObjectiveError{};  // fit.R:119 with det underflow (A.4)
    return lp;
  };
  const int nparam = (kernel_id == GPRC_GAMMAEXP || kernel_id == GPRC_RATQUAD || kernel_id == GPRC_POLYNOMIAL) ? 2 : 1;
  // dens_deriv as coded, R/fit.R:126-139
  optim::GrN deriv = [&](const double* v, double* gout) {
    gprc_kernel k = family_spec(kernel_id, v);
    long inf = 0;
    ++n_gr;
    const int r = logml_grad_impl(c, &k, dX, true, d, n, dy, true, noise, GPRC_GRAD_AS_CODED, gout, nparam, &inf);
    if (r != 0) {
      hard_error = r;
      throw optim::ObjectiveError{};
    }
    if (inf != 0) throw optim::ObjectiveError{};  // solve(K): computationally singular
  };
  optim::UntilErrorResult best;
  if (kernel_id == GPRC_POLYNOMIAL) {
    // R/fit.R:145-156: Brent over sigma in [0, 5] for every degree 1..10, then which.max
    bool have = false;
    int best_deg = 1;
    for (int deg = 1; deg <= 10 && !hard_error; ++deg) {
      optim::FnN f = [&](const double* sig) {
        const double v[2] = {sig[0], (double)deg};
        return dens(v);
      };
      optim::UntilErrorResult r = optim::optim_until_error({1.0}, f, nullptr, true, 0.0, 5.0);
      if (!have || r.value > best.value) {
        best = r;
        best_deg = deg;
        have = true;
      }
    }
    best.par = {best.par[0], (double)best_deg};
  } else if (nparam == 1) {
    best = optim::optim_until_error({1.0}, dens, nullptr, true, 0.0, 10.0);
  } else {
    best = optim::optim_until_error({1.0, 1.0}, dens, &deriv, false, 0.0, 0.0);
  }
  cudaStreamSynchronize(c->stream);
  dfree(dX);
  dfree(dy);
  if (hard_error) return hard_error;
  *npar = (int)best.par.size();
  for (size_t i = 0; i < best.par.size(); ++i) par[i] = best.par[i];
  *value = best.value;
  if (evaluations) {
    evaluations[0] = n_fn;
    evaluations[1] = n_gr;
  }
  return 0;
}

// =================================================================================================================
// (4) GPC: Laplace-approximation Newton loop, R/GPCclass.R:73-103
// =================================================================================================================
static void gpc_destroy(gprc_gpc* g) {
  if (!g) return;
  dfree(g->X);
  dfree(g->y);
  dfree(g->K);
  dfree(g->f);
  dfree(g->sw);
  dfree(g->gradl);
  g->F.release();
  g->ws.release();
  delete g;
}

static int gpc_fit_common(gprc_ctx* c, const gprc_kernel* k, const double* X, int d, long n, const double* y,
                          const double* Kpre, double eps, int guard, int max_iter, gprc_gpc** out, int* iters,
                          double* trace, int trace_cap, double* sum_diagL, double* sum_log_diagL, int* status) {
  GPRC_ARG(c && out && y && n > 0 && eps > 0.0 && iters && status);
  GPRC_ARG(Kpre != nullptr || (k != nullptr && X != nullptr && d > 0));
  *out = nullptr;
  *iters = 0;
  *status = 0;
  DeviceGuard dg(c);
  gprc_gpc* g = new gprc_gpc();
  g->ctx = c;
  g->d = d;
  g->precomputed = (Kpre != nullptr);
  double *bvec = nullptr, *Kb = nullptr, *cvec = nullptr, *tvec = nullptr, *avec = nullptr, *work = nullptr,
         *tmp = nullptr;
  int rc = 0;
  do {
    if ((rc = factor_alloc(g->F, n))) break;
    FactorState& F = g->F;
    const long np = F.n_pad;
    if ((rc = dmalloc(&g->y, (size_t)np)) || (rc = dmalloc(&g->f, (size_t)np)) || (rc = dmalloc(&g->sw, (size_t)np)) ||
        (rc = dmalloc(&g->gradl, (size_t)np)) || (rc = dmalloc(&g->K, (size_t)np * np)) ||
        (rc = dmalloc(&bvec, (size_t)np)) || (rc = dmalloc(&Kb, (size_t)np)) || (rc = dmalloc(&cvec, (size_t)np)) ||
        (rc = dmalloc(&tvec, (size_t)np)) || (rc = dmalloc(&avec, (size_t)np)) || (rc = dmalloc(&work, (size_t)np)) ||
        (rc = dmalloc(&tmp, (size_t)np)))
      break;
    cudaMemsetAsync(g->y, 0, sizeof(double) * np, c->stream);
    cudaMemcpyAsync(g->y, y, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream);
    cudaMemsetAsync(g->f, 0, sizeof(double) * np, c->stream);  // f <- rep(0, n)              R/GPCclass.R:74
    {
      PhaseTimer t(c, GPRC_T_BUILD_K);
      if (Kpre) {
        if ((rc = upload_square_padded(c, Kpre, n, g->K, np, 0.0, false))) break;
      } else {
        if ((rc = make_spec(c, k, d, g->spec))) break;
        if ((rc = dmalloc(&g->X, (size_t)d * n))) break;
        cudaMemcpyAsync(g->X, X, sizeof(double) * d * n, cudaMemcpyHostToDevice, c->stream);
        // K <- covariance_matrix(X, X, k): full symmetric (K %*% b needs both triangles), zero padding
        if ((rc = cov_build_dev(c, g->spec.dev, g->X, d, n, g->X, n, g->K, np, np, np, false, false, 0.0, false,
                                nullptr, nullptr, nullptr, 0)))
          break;
      }
    }
    const dim3 tgrid((unsigned)(np / 64), (unsigned)(np / 64));
    const unsigned vgrid = (unsigned)((np + 255) / 256);
    double last_objective = 0.0, least_objective = 0.0, objective = 0.0;
    int it = 0;
    PhaseTimer tn(c, GPRC_T_NEWTON);
    while (true) {
      ++it;
      // P, W, B = I + sqrt(W) sqrt(W)' * K (fused), b = W f + (y + 1)/2 - P           R/GPCclass.R:78-81
      gpc_build_B_kernel<<<tgrid, 256, 0, c->stream>>>(g->K, np, g->f, g->y, n, np, F.L, np, g->sw, bvec, nullptr);
      c->launches++;
      long info = 0;
      if ((rc = factor_run(c, F, &info))) break;
      if (info != 0) {
        *status = 2;
        break;
      }
      // intermediate <- solve(t(L), solve(L, sqrt(W) * (K %*% b)))                     R/GPCclass.R:82-83
      if ((rc = gemv_t(c, g->K, np, np, bvec, Kb))) break;
      vec_mul_kernel<<<vgrid, 256, 0, c->stream>>>(g->sw, Kb, np, cvec);
      c->launches++;
      if ((rc = potrs_vec(c, F.L, np, np, F.dinv, cvec, work, tmp, tvec))) break;
      // a <- b - sqrt(W) * intermediate ; f <- K %*% a                                 R/GPCclass.R:84-85
      gpc_a_kernel<<<vgrid, 256, 0, c->stream>>>(bvec, g->sw, tvec, np, avec);
      c->launches++;
      if ((rc = gemv_t(c, g->K, np, np, avec, g->f))) break;
      gpc_objective_kernel<<<1, 1024, 0, c->stream>>>(avec, g->f, g->y, n, c->d_scalars);
      c->launches++;
      cudaMemcpyAsync(c->h_scalars, c->d_scalars, sizeof(double), cudaMemcpyDeviceToHost, c->stream);
      cudaError_t e = cudaStreamSynchronize(c->stream);
      if (e != cudaSuccess) {
        rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
        break;
      }
      objective = c->h_scalars[0];
      // the LAST slot always holds the most recent objective (logq = objective - sum(diag(L)) needs the final one even
      // when the loop runs for more than trace_cap iterations)
      if (trace && trace_cap > 0) trace[std::min(it, trace_cap) - 1] = objective;
      // stopping rule, literally R/GPCclass.R:87-96 (the guard is mis-signed in the reference: SURVEY.md A.2)
      if (it > 1) {
        if (fabs(objective - last_objective) < eps) {
          break;
        } else if (guard && least_objective + 10.0 < objective) {
          *status = 1;
          break;
        }
      } else {
        least_objective = objective;
      }
      last_objective = objective;
      if (max_iter > 0 && it >= max_iter) break;
      if ((rc = poll_interrupt(c))) break;  // a loop that oscillates without converging must stay interruptible
      if (!(objective == objective)) {  // NaN objective can never satisfy the rule: the reference would spin forever
        *status = 2;
        break;
      }
    }
    *iters = it;
    if (rc || *status != 0) break;
    // P, W at f_hat; L <- t(chol(B)); logq pieces                                         R/GPCclass.R:99-103
    gpc_build_B_kernel<<<tgrid, 256, 0, c->stream>>>(g->K, np, g->f, g->y, n, np, F.L, np, g->sw, bvec, g->gradl);
    c->launches++;
    long info = 0;
    if ((rc = factor_run(c, F, &info))) break;
    if (info != 0) {
      *status = 2;
      break;
    }
    gp_reduce_kernel<<<1, 1024, 0, c->stream>>>(nullptr, nullptr, F.diag, n, c->d_scalars);
    c->launches++;
    cudaMemcpyAsync(c->h_scalars, c->d_scalars, 4 * sizeof(double), cudaMemcpyDeviceToHost, c->stream);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) {
      rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
      break;
    }
    if (sum_log_diagL) *sum_log_diagL = c->h_scalars[1];
    if (sum_diagL) *sum_diagL = c->h_scalars[2];
  } while (0);
  cudaStreamSynchronize(c->stream);
  dfree(bvec);
  dfree(Kb);
  dfree(cvec);
  dfree(tvec);
  dfree(avec);
  dfree(work);
  dfree(tmp);
  if (rc != 0 || *status != 0) {
    gpc_destroy(g);
    return rc;
  }
  dfree(g->K);  // predict_class only needs X, f_hat, sqrt(W) and the factor
  g->K = nullptr;
  *out = g;
  return 0;
}

extern "C" int gprc_gpc_fit(gprc_ctx* c, const gprc_kernel* k, const double* X, int d, long n, const double* y,
                            double eps, int guard, int max_iter, gprc_gpc** out, int* iters, double* objective_trace,
                            int trace_cap, double* sum_diagL, double* sum_log_diagL, int* status) {
  return gpc_fit_common(c, k, X, d, n, y, nullptr, eps, guard, max_iter, out, iters, objective_trace, trace_cap,
                        sum_diagL, sum_log_diagL, status);
}
extern "C" int gprc_gpc_fit_precomputed(gprc_ctx* c, const double* K, long n, const double* y, double eps, int guard,
                                        int max_iter, gprc_gpc** out, int* iters, double* objective_trace,
                                        int trace_cap, double* sum_diagL, double* sum_log_diagL, int* status) {
  GPRC_ARG(K != nullptr);
  return gpc_fit_common(c, nullptr, nullptr, 0, n, y, K, eps, guard, max_iter, out, iters, objective_trace, trace_cap,
                        sum_diagL, sum_log_diagL, status);
}

// fs_bar <- t(K_star) %*% ((y + 1)/2 - P); v <- solve(L, sqrt(W) * K_star); Vfs <- k(X*, X*) - colSums(v * v)
// R/GPCclass.R:110-115
extern "C" int gprc_gpc_predict_latent(gprc_gpc* g, const double* Xs, long m, double* fs_bar, double* Vfs) {
  GPRC_ARG(g && Xs && fs_bar && Vfs && m >= 0);
  GPRC_ARG(!g->precomputed);
  if (m == 0) return 0;
  gprc_ctx* c = g->ctx;
  DeviceGuard guard(c);
  double *dXs = nullptr, *dmean = nullptr, *dvar = nullptr;
  int rc = 0;
  do {
    if ((rc = dmalloc(&dXs, (size_t)g->d * m))) break;
    if ((rc = dmalloc(&dmean, (size_t)m))) break;
    if ((rc = dmalloc(&dvar, (size_t)m))) break;
    cudaMemcpyAsync(dXs, Xs, sizeof(double) * g->d * m, cudaMemcpyHostToDevice, c->stream);
    if ((rc = predict_pointwise_dev(c, g->spec.dev, g->X, g->d, g->F, g->ws, g->gradl, g->sw, dXs, m, dmean, dvar)))
      break;
    cudaMemcpyAsync(fs_bar, dmean, sizeof(double) * m, cudaMemcpyDeviceToHost, c->stream);
    cudaMemcpyAsync(Vfs, dvar, sizeof(double) * m, cudaMemcpyDeviceToHost, c->stream);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
  } while (0);
  dfree(dXs);
  dfree(dmean);
  dfree(dvar);
  return rc;
}
extern "C" int gprc_gpc_predict_latent_precomputed(gprc_gpc* g, const double* Ks, const double* kss, long m,
                                                   double* fs_bar, double* Vfs) {
  GPRC_ARG(g && Ks && kss && fs_bar && Vfs && m >= 0);
  if (m == 0) return 0;
  DeviceGuard guard(g->ctx);
  return predict_precomputed(g->ctx, g->F, g->ws, g->gradl, g->sw, Ks, kss, m, fs_bar, Vfs);
}
// one thread per test point: the adaptive QUADPACK recursion runs in the thread's local memory
__global__ void __launch_bounds__(128) logistic_gaussian_kernel(const double* __restrict__ mean,
                                                                const double* __restrict__ sd, long m,
                                                                double* __restrict__ out, int* __restrict__ ier) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= m) return;
  const double mu = mean[i], s = sd[i];
  if (!(s > 0.0) || !isfinite(mu) || !isfinite(s)) {  // dnorm(sd <= 0) is NaN: integrate() stops with "non-finite function value"
    out[i] = NAN;
    if (ier) ier[i] = -1;
    return;
  }
  const gprc_quad::QuadResult r = gprc_quad::logistic_gaussian(mu, s);
  out[i] = r.result;
  if (ier) ier[i] = r.ier;
}

static int quad_dev(gprc_ctx* c, const double* dmean, const double* dsd, long m, double* dout, int* dier) {
  logistic_gaussian_kernel<<<(unsigned)((m + 127) / 128), 128, 0, c->stream>>>(dmean, dsd, m, dout, dier);
  c->launches++;
  GPRC_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int gprc_logistic_gaussian(gprc_ctx* c, const double* mean, const double* sd, long m, double* out, int* ier) {
  GPRC_ARG(c && mean && sd && out && m >= 0);
  if (m == 0) return 0;
  DeviceGuard guard(c);
  double *dm = nullptr, *ds = nullptr, *dout = nullptr;
  int* dier = nullptr;
  int rc = 0;
  do {
    if ((rc = dmalloc(&dm, (size_t)m)) || (rc = dmalloc(&ds, (size_t)m)) || (rc = dmalloc(&dout, (size_t)m)) ||
        (rc = dmalloc(&dier, (size_t)m)))
      break;
    cudaMemcpyAsync(dm, mean, sizeof(double) * m, cudaMemcpyHostToDevice, c->stream);
    cudaMemcpyAsync(ds, sd, sizeof(double) * m, cudaMemcpyHostToDevice, c->stream);
    if ((rc = quad_dev(c, dm, ds, m, dout, dier))) break;
    cudaMemcpyAsync(out, dout, sizeof(double) * m, cudaMemcpyDeviceToHost, c->stream);
    if (ier) cudaMemcpyAsync(ier, dier, sizeof(int) * m, cudaMemcpyDeviceToHost, c->stream);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
  } while (0);
  dfree(dm);
  dfree(ds);
  dfree(dout);
  dfree(dier);
  return rc;
}

extern "C" int gprc_gpc_predict_class(gprc_gpc* g, const double* Xs, long m, double* prob, int* ier) {
  GPRC_ARG(g && Xs && prob && m >= 0);
  GPRC_ARG(!g->precomputed);
  if (m == 0) return 0;
  gprc_ctx* c = g->ctx;
  DeviceGuard guard(c);
  double *dXs = nullptr, *dmean = nullptr, *dvar = nullptr, *dout = nullptr;
  int* dier = nullptr;
  int rc = 0;
  do {
    if ((rc = dmalloc(&dXs, (size_t)g->d * m)) || (rc = dmalloc(&dmean, (size_t)m)) || (rc = dmalloc(&dvar, (size_t)m)) ||
        (rc = dmalloc(&dout, (size_t)m)) || (rc = dmalloc(&dier, (size_t)m)))
      break;
    cudaMemcpyAsync(dXs, Xs, sizeof(double) * g->d * m, cudaMemcpyHostToDevice, c->stream);
    if ((rc = predict_pointwise_dev(c, g->spec.dev, g->X, g->d, g->F, g->ws, g->gradl, g->sw, dXs, m, dmean, dvar)))
      break;
    // dnorm(z, mean = fs_bar[i], sd = Vfs[i]): the latent VARIANCE is passed as sd, as the reference does (A.1)
    if ((rc = quad_dev(c, dmean, dvar, m, dout, dier))) break;
    cudaMemcpyAsync(prob, dout, sizeof(double) * m, cudaMemcpyDeviceToHost, c->stream);
    if (ier) cudaMemcpyAsync(ier, dier, sizeof(int) * m, cudaMemcpyDeviceToHost, c->stream);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
  } while (0);
  dfree(dXs);
  dfree(dmean);
  dfree(dvar);
  dfree(dout);
  dfree(dier);
  return rc;
}

extern "C" int gprc_gpc_get(gprc_gpc* g, int what, double* host) {
  GPRC_ARG(g && host);
  gprc_ctx* c = g->ctx;
  DeviceGuard guard(c);
  switch (what) {
    case GPRC_GET_L: return download_lower(c, g->F.L, g->F.n, g->F.n_pad, host);
    case GPRC_GET_FHAT: return gprc_dev_d2h(c, host, g->f, sizeof(double) * g->F.n);
    case GPRC_GET_SQRTW: return gprc_dev_d2h(c, host, g->sw, sizeof(double) * g->F.n);
    default: return set_error(-1, __FILE__, __LINE__, "gprc_gpc_get: unknown item");
  }
}
extern "C" long gprc_gpc_n(const gprc_gpc* g) { return g ? g->F.n : 0; }
extern "C" int gprc_gpc_dim(const gprc_gpc* g) { return g ? g->d : 0; }
extern "C" void gprc_gpc_free(gprc_gpc* g) {
  if (!g) return;
  DeviceGuard guard(g->ctx);
  cudaStreamSynchronize(g->ctx->stream);
  gpc_destroy(g);
}

// =================================================================================================================
// raw device primitives
// =================================================================================================================
extern "C" int gprc_dev_potrf(gprc_ctx* c, double* dA, long n, long ld, double* dinv, long* info) {
  GPRC_ARG(c && dA && dinv && info && n > 0 && n % NB == 0 && ld % NB == 0 && ld >= n);
  DeviceGuard guard(c);
  *c->h_info = LONG_MAX;
  GPRC_CUDA(cudaMemcpyAsync(c->d_info, c->h_info, sizeof(long), cudaMemcpyHostToDevice, c->stream));
  {
    PhaseTimer t(c, GPRC_T_CHOL);
    GPRC_CHECK(potrf_blocked(c, dA, n, ld, dinv, c->d_info, nullptr));
  }
  GPRC_CUDA(cudaMemcpyAsync(c->h_info, c->d_info, sizeof(long), cudaMemcpyDeviceToHost, c->stream));
  GPRC_CUDA(cudaStreamSynchronize(c->stream));
  *info = (*c->h_info == LONG_MAX) ? 0 : *c->h_info;
  return 0;
}

extern "C" int gprc_dev_dgemm(gprc_ctx* c, int transb, long M, long N, long K, double alpha, const double* dA, long lda,
                              const double* dB, long ldb, double beta, double* dC, long ldc) {
  GPRC_ARG(c && dA && dB && dC && M > 0 && N > 0 && K >= 0);
  GPRC_ARG(M % NB == 0 && N % NB == 0 && K % BK == 0 && lda % 2 == 0 && ldb % 2 == 0);
  DeviceGuard guard(c);
  const dim3 grid((unsigned)((M / NB) * (N / NB)));
  if (transb) {
    DgemmPolicy<false> p{dA, lda, dB, ldb, dC, ldc, alpha, beta, (int)K, (int)(M / NB)};
    return launch_gemm(c, p, grid);
  }
  DgemmPolicy<true> p{dA, lda, dB, ldb, dC, ldc, alpha, beta, (int)K, (int)(M / NB)};
  return launch_gemm(c, p, grid);
}

// Measured INT8 tensor-pipe rate (the roofline denominator of the INT8 variance pass, bench.py): a pure stream of
// 128 x 256 x 32 tcgen05.mma kind::i8 from shared memory on every SM -- no feed, no drain -- repeated for about
// `seconds` (a few milliseconds give the burst figure, seconds the figure under the board's power cap).
extern "C" int gprc_dev_int8_rate(gprc_ctx* c, double seconds, double* tops, double* clk_per_mma) {
  GPRC_ARG(c && tops && seconds > 0.0 && seconds <= 30.0);
  DeviceGuard guard(c);
  constexpr int N = 256, COUNT = 20000;
  const int smem = 65536 + 8 * N * 32 + 1024;
  GPRC_CUDA(cudaFuncSetAttribute(oz::mma_rate_kernel<N, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  long long* d = nullptr;
  GPRC_CUDA(cudaMalloc(&d, 128));
  GPRC_CUDA(cudaMemsetAsync(d, 0, 128, c->stream));
  cudaEvent_t a = PhaseTimer::get_event(c), b = PhaseTimer::get_event(c);
  auto launch = [&]() { oz::mma_rate_kernel<N, false><<<c->sm_count, 128, smem, c->stream>>>(COUNT, 1, 7, d); };
  launch();  // warm-up
  cudaStreamSynchronize(c->stream);
  // one launch is COUNT * 128 clk ~ 1.3 ms: size the repetition count from a first timed launch
  cudaEventRecord(a, c->stream);
  launch();
  cudaEventRecord(b, c->stream);
  cudaStreamSynchronize(c->stream);
  float ms1 = 0.f;
  cudaEventElapsedTime(&ms1, a, b);
  const int reps = std::max(1, (int)(seconds * 1e3 / std::max(ms1, 0.1f)));
  cudaEventRecord(a, c->stream);
  for (int r = 0; r < reps; ++r) launch();
  cudaEventRecord(b, c->stream);
  cudaError_t e = cudaStreamSynchronize(c->stream);
  float ms = 0.f;
  cudaEventElapsedTime(&ms, a, b);
  long long h[2] = {0, 0};
  cudaMemcpy(h, d, 16, cudaMemcpyDeviceToHost);
  cudaFree(d);
  c->event_pool.push_back(a);
  c->event_pool.push_back(b);
  c->launches += reps + 2;
  if (e != cudaSuccess) return set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
  if (h[1] != 0) return set_error(-6, __FILE__, __LINE__, "INT8 rate probe: the MMA stream never completed");
  *tops = 2.0 * 128.0 * N * 32.0 * (double)COUNT * (double)c->sm_count * (double)reps / ((double)ms * 1e-3) * 1e-12;
  if (clk_per_mma) *clk_per_mma = (double)h[0] / (double)COUNT;
  return 0;
}

extern "C" int gprc_dev_trtri(gprc_ctx* c, const double* dL, long n, long ld, const double* dinv, double* dW,
                              double* dscratch) {
  GPRC_ARG(c && dL && dinv && dW && dscratch && n > 0 && n % NB == 0 && ld % NB == 0 && ld >= n);
  DeviceGuard guard(c);
  double* Wt = nullptr;
  GPRC_CHECK(dmalloc(&Wt, (size_t)n * ld));
  int rc;
  {
    PhaseTimer t(c, GPRC_T_TRTRI);
    rc = trtri_levels(c, dL, n, ld, dinv, dW, Wt, dscratch);
  }
  cudaStreamSynchronize(c->stream);
  dfree(Wt);
  return rc;
}

// =================================================================================================================
// posterior sampling helper: multivariate_normal(), R/GPRclass.R:360-370
// =================================================================================================================
namespace gprc {
// Both kernels stride over the columns by gridDim.y: launched on grid_cols() they take any number of columns, where one
// column per grid row would stop at the 65 535 limit of gridDim.y (more draws than that, or a wider covariance).
constexpr long MAX_GRID_Y = 65535;
static inline dim3 grid_cols(long rows, long cols) { return grid2(rows, std::min(cols, MAX_GRID_Y)); }
// zero everything strictly above the diagonal (the uploaded covariance had both triangles)
__global__ void tril_inplace_kernel(double* __restrict__ M, long ld, long n) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  for (long j = i + 1 + blockIdx.y; j < n; j += gridDim.y) M[i + j * ld] = 0.0;
}
__global__ void add_mean_kernel(double* __restrict__ out, long ld, long m, long ns, const double* __restrict__ mean) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= m) return;
  const double mu = mean[i];
  for (long j = blockIdx.y; j < ns; j += gridDim.y) out[i + j * ld] += mu;
}
}  // namespace gprc

extern "C" int gprc_mvn_sample(gprc_ctx* c, const double* mean, const double* cov, long m, const double* Z, long ns,
                               double* out, long* info) {
  GPRC_ARG(c && mean && cov && Z && out && info && m > 0 && ns > 0);
  DeviceGuard guard(c);
  FactorState F;
  double *dZ = nullptr, *dout = nullptr, *dmean = nullptr;
  const long sp = round_up(ns, NB);
  // a failed launch is reported here and the buffers below are still released
  auto launched = []() -> int {
    GPRC_CUDA(cudaGetLastError());
    return 0;
  };
  int rc = 0;
  *info = 0;
  do {
    if ((rc = factor_alloc(F, m))) break;
    const long mp = F.n_pad;
    if ((rc = dmalloc(&dZ, (size_t)mp * sp)) || (rc = dmalloc(&dout, (size_t)mp * sp)) || (rc = dmalloc(&dmean, (size_t)m)))
      break;
    if ((rc = upload_square_padded(c, cov, m, F.L, mp, 0.0, true))) break;
    if ((rc = factor_run(c, F, info))) break;
    if (*info != 0) break;  // the caller falls back to eigen(), as the reference does
    cudaMemsetAsync(dZ, 0, sizeof(double) * mp * sp, c->stream);
    cudaMemcpy2DAsync(dZ, mp * sizeof(double), Z, m * sizeof(double), m * sizeof(double), ns, cudaMemcpyHostToDevice,
                      c->stream);
    cudaMemcpyAsync(dmean, mean, sizeof(double) * m, cudaMemcpyHostToDevice, c->stream);
    tril_inplace_kernel<<<grid_cols(mp, mp), 256, 0, c->stream>>>(F.L, mp, mp);
    c->launches++;
    if ((rc = launched())) break;
    DgemmPolicy<true> pol{F.L, mp, dZ, mp, dout, mp, 1.0, 0.0, (int)mp, (int)(mp / NB)};  // L %*% Z
    if ((rc = launch_gemm(c, pol, dim3((unsigned)((mp / NB) * (sp / NB)))))) break;
    add_mean_kernel<<<grid_cols(m, ns), 256, 0, c->stream>>>(dout, mp, m, ns, dmean);
    c->launches++;
    if ((rc = launched())) break;
    cudaMemcpy2DAsync(out, m * sizeof(double), dout, mp * sizeof(double), m * sizeof(double), ns, cudaMemcpyDeviceToHost,
                      c->stream);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
  } while (0);
  cudaStreamSynchronize(c->stream);
  F.release();
  dfree(dZ);
  dfree(dout);
  dfree(dmean);
  return rc;
}

// =================================================================================================================
// multi-GPU Cholesky + solve (dist.cuh)
// =================================================================================================================
#include "dist.cuh"

extern "C" int gprc_dist_unique_id(char* id128, const char* nccl_path) {
  GPRC_ARG(id128 != nullptr);
  static NcclApi api;
  GPRC_CHECK(nccl_load(api, nccl_path));
  ncclUniqueId id;
  GPRC_NCCL(api, api.GetUniqueId(&id));
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  memcpy(id128, &id, 128);
  return 0;
}

extern "C" int gprc_dist_create(gprc_ctx* c, const char* id128, int rank, int world, const char* nccl_path,
                                gprc_dist** out) {
  GPRC_ARG(c && id128 && out && world >= 1 && rank >= 0 && rank < world);
  *out = nullptr;
  DeviceGuard guard(c);
  gprc_dist* D = new gprc_dist();
  D->ctx = c;
  D->rank = rank;
  D->world = world;
  int rc = nccl_load(D->api, nccl_path);
  if (rc) {
    delete D;
    return rc;
  }
  ncclUniqueId id;
  memcpy(&id, id128, 128);
  ncclResult_t r = D->api.CommInitRank(&D->comm, world, id, rank);
  if (r != ncclSuccess) {
    set_error(-5, __FILE__, __LINE__, D->api.GetErrorString(r));
    delete D;
    return -5;
  }
  int lo = 0, hi = 0;
  cudaDeviceGetStreamPriorityRange(&lo, &hi);
  GPRC_CUDA(cudaStreamCreateWithPriority(&D->s_comm, cudaStreamNonBlocking, hi));
  GPRC_CUDA(cudaEventCreateWithFlags(&D->ev_packed, cudaEventDisableTiming));
  GPRC_CUDA(cudaEventCreateWithFlags(&D->ev_bcast[0], cudaEventDisableTiming));
  GPRC_CUDA(cudaEventCreateWithFlags(&D->ev_bcast[1], cudaEventDisableTiming));
  GPRC_CUDA(cudaEventCreateWithFlags(&D->ev_rest, cudaEventDisableTiming));
  GPRC_CUDA(cudaEventCreateWithFlags(&D->ev_begin, cudaEventDisableTiming));
  *out = D;
  return 0;
}

extern "C" void gprc_dist_free(gprc_dist* D) {
  if (!D) return;
  DeviceGuard guard(D->ctx);
  cudaStreamSynchronize(D->s_comm);
  cudaStreamSynchronize(D->ctx->stream);
  if (D->comm) D->api.CommDestroy(D->comm);
  cudaEventDestroy(D->ev_packed);
  cudaEventDestroy(D->ev_bcast[0]);
  cudaEventDestroy(D->ev_bcast[1]);
  cudaEventDestroy(D->ev_rest);
  cudaEventDestroy(D->ev_begin);
  for (cudaEvent_t e : D->timeline) cudaEventDestroy(e);
  cudaStreamDestroy(D->s_comm);
  delete D;
}

// replicate != nullptr: every rank also assembles the complete factor from the panels it receives anyway (no extra
// communication) and gets an ordinary gprc_gpr handle back, ready for gprc_gpr_predict on its shard of test points.
static int dist_fit_impl(gprc_dist* D, const gprc_kernel* k, const double* X, int d, long n, const double* y,
                         double noise, double* logp, double* alpha, long* info, double* phase_ms,
                         gprc_gpr** replicate) {
  GPRC_ARG(D && k && X && y && logp && info && n > 0 && d > 0 && noise >= 0.0);
  if (replicate) *replicate = nullptr;
  gprc_ctx* c = D->ctx;
  DeviceGuard guard(c);
  NcclApi& api = D->api;
  const int N = D->world, me = D->rank;
  const long n_pad = round_up(n, PANEL);
  const int npan = (int)(n_pad / PANEL), nt = (int)(n_pad / NB);
  const int nown = (npan - me + N - 1) / N;  // panels me, me + N, ...
  const long slab = n_pad * PANEL;
  cudaStream_t s0 = c->stream, s1 = c->stream_hi, sc = D->s_comm;
  static bool configured[64] = {false};
  if (!configured[c->device & 63]) {
    GPRC_CUDA(cudaFuncSetAttribute(potrf_diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PD_SMEM_BYTES));
    configured[c->device & 63] = true;
  }
  gprc_gpr* g = nullptr;
  SpecHolder local_spec;
  if (replicate) {
    g = new gprc_gpr();
    g->ctx = c;
    g->d = d;
    g->noise = noise;
    g->khost = *k;
  }
  SpecHolder& spec = g ? g->spec : local_spec;
  GPRC_CHECK(make_spec(c, k, d, spec));
  const long pbuf_elems = slab + (long)OUTER_BLOCKS * NB * NB;  // panel + its 4 inverted diagonal blocks
  double *dX = nullptr, *Aloc = nullptr, *dinv = nullptr, *diag = nullptr, *Pbuf[2] = {nullptr, nullptr}, *vec = nullptr,
         *dy = nullptr, *partial = nullptr;
  cudaEvent_t e0 = nullptr, e1 = nullptr, e2 = nullptr, e3 = nullptr;
  int rc = 0;
  *info = 0;
  do {
    if ((rc = dmalloc(&dX, (size_t)d * n)) || (rc = dmalloc(&Aloc, (size_t)std::max(nown, 1) * slab)) ||
        (rc = dmalloc(&dinv, (size_t)n_pad * NB)) || (rc = dmalloc(&diag, (size_t)n_pad)) ||
        (rc = dmalloc(&Pbuf[0], (size_t)pbuf_elems)) || (rc = dmalloc(&Pbuf[1], (size_t)pbuf_elems)) ||
        (rc = dmalloc(&vec, (size_t)2 * n_pad)) || (rc = dmalloc(&dy, (size_t)n_pad)) ||
        (rc = dmalloc(&partial, (size_t)((n_pad + BWD_CHUNK - 1) / BWD_CHUNK) * NB)))
      break;
    if (g) {
      g->F.n = n;
      g->F.n_pad = n_pad;
      if ((rc = dmalloc(&g->F.L, (size_t)n_pad * n_pad)) || (rc = dmalloc(&g->alpha, (size_t)n_pad))) break;
    }
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    cudaEventCreate(&e2);
    cudaEventCreate(&e3);
    if (D->timeline_on) {
      const size_t want = (size_t)npan * 6 + 1;
      while (D->timeline.size() < want) {
        cudaEvent_t ev;
        cudaEventCreate(&ev);
        D->timeline.push_back(ev);
      }
      D->timeline_npan = npan;
      D->timeline_ms.assign((size_t)npan * 6, NAN);
    }
    std::vector<char> tl_set(D->timeline_on ? (size_t)npan * 6 : 0, 0);
    auto tl = [&](int p, int slot, cudaStream_t st) {
      if (!D->timeline_on) return;
      cudaEventRecord(D->timeline[(size_t)p * 6 + slot + 1], st);
      tl_set[(size_t)p * 6 + slot] = 1;
    };
    cudaMemcpyAsync(dX, X, sizeof(double) * d * n, cudaMemcpyHostToDevice, s0);
    cudaMemsetAsync(dy, 0, sizeof(double) * n_pad, s0);
    cudaMemcpyAsync(dy, y, sizeof(double) * n, cudaMemcpyHostToDevice, s0);
    cudaMemsetAsync(diag, 0, sizeof(double) * n_pad, s0);
    *c->h_info = LONG_MAX;
    cudaMemcpyAsync(c->d_info, c->h_info, sizeof(long), cudaMemcpyHostToDevice, s0);
    cudaEventRecord(e0, s0);
    // ---- build the owned panels of K + noise I (lower part, identity padding) ----
    for (int q = 0; q < nown && rc == 0; ++q) {
      const long p = me + (long)q * N, c0 = p * PANEL;
      CovParams cp;
      cp.k = spec.dev;
      cp.A = dX;
      cp.B = dX + c0 * d;
      cp.d = d;
      cp.nA = n;
      cp.nB = std::max<long>(0, std::min<long>(PANEL, n - c0));
      cp.out = Aloc + q * slab;
      cp.ldo = n_pad;
      cp.rows_pad = n_pad;
      cp.cols_pad = PANEL;
      cp.lower_only = 1;
      cp.symmetric = 1;
      cp.diag_add = noise;
      cp.pad_identity = 1;
      cp.rowscale = cp.weights = nullptr;
      cp.pmean = nullptr;
      cp.ldpm = 0;
      cp.colscale = cp.colweights = nullptr;
      cp.col_offset = c0;
      rc = launch_cov(c, cp);
    }
    if (rc) break;
    cudaEventRecord(e1, s0);

    // ---- factorisation ----
    // the single-GPU kernels address the matrix as A[row + col * ld] with GLOBAL indices: give them the slab shifted
    // left by the panel's first column
    auto virt = [&](int p) { return Aloc + (long)((p - me) / N) * slab - (long)p * PANEL * n_pad; };
    auto factor_panel = [&](int p) -> int {
      double* Av = virt(p);
      const int J0 = p * OUTER_BLOCKS, Jend = J0 + OUTER_BLOCKS;
      for (int j = J0; j < Jend; ++j) {
        if (j > J0) {
          SyrkPolicy sp{Av, n_pad, 0, j, J0 * NB, j * NB};
          GPRC_CHECK(launch_gemm(c, sp, dim3(nt - j), s1));
        }
        potrf_diag_kernel<<<1, 256, PD_SMEM_BYTES, s1>>>(Av, n_pad, j, dinv + (long)j * NB * NB, c->d_info, diag);
        c->launches++;
        if (j + 1 < nt) {
          TrsmPolicy tp{Av, n_pad, dinv + (long)j * NB * NB, j};
          GPRC_CHECK(launch_gemm(c, tp, dim3(nt - j - 1), s1));
        }
      }
      // pack rows >= 512 p of the 512 columns into the panel buffer (leading dimension = rows kept)
      const long rows = n_pad - (long)p * PANEL;
      GPRC_CUDA(cudaMemcpy2DAsync(Pbuf[p & 1], rows * sizeof(double), Av + (long)p * PANEL * n_pad + (long)p * PANEL,
                                  n_pad * sizeof(double), rows * sizeof(double), PANEL, cudaMemcpyDeviceToDevice, s1));
      GPRC_CUDA(cudaMemcpyAsync(Pbuf[p & 1] + rows * PANEL, dinv + (long)J0 * NB * NB,
                                sizeof(double) * OUTER_BLOCKS * NB * NB, cudaMemcpyDeviceToDevice, s1));
      GPRC_CUDA(cudaEventRecord(D->ev_packed, s1));
      return 0;
    };
    // assemble the complete factor from the broadcast panels (replicated handle only)
    auto unpack = [&](int p) -> int {
      if (!g) return 0;
      const long rows = n_pad - (long)p * PANEL;
      GPRC_CUDA(cudaMemcpy2DAsync(g->F.L + (long)p * PANEL * n_pad + (long)p * PANEL, n_pad * sizeof(double),
                                  Pbuf[p & 1], rows * sizeof(double), rows * sizeof(double), PANEL,
                                  cudaMemcpyDeviceToDevice, s0));
      if (p % N != me)
        GPRC_CUDA(cudaMemcpyAsync(dinv + (long)p * OUTER_BLOCKS * NB * NB, Pbuf[p & 1] + rows * PANEL,
                                  sizeof(double) * OUTER_BLOCKS * NB * NB, cudaMemcpyDeviceToDevice, s0));
      return 0;
    };
    auto update = [&](int p, int first_panel, int count, cudaStream_t st) -> int {
      if (count <= 0) return 0;
      DistUpdatePolicy up;
      up.Aloc = Aloc;
      up.ld = n_pad;
      up.slab_elems = slab;
      up.P = Pbuf[p & 1];
      up.ldp = n_pad - (long)p * PANEL;
      up.prow0_tile = p * OUTER_BLOCKS;
      up.nt = nt;
      up.q0 = (first_panel - me) / N;
      up.first_panel = first_panel;
      up.world = N;
      long tiles = 0;
      for (int tj = 0; tj < OUTER_BLOCKS; ++tj) tiles += nt - (first_panel * OUTER_BLOCKS + tj);
      return launch_gemm(c, up, dim3((unsigned)tiles, (unsigned)count), st);
    };
    auto owner = [&](int p) { return p % N; };
    auto next_owned_after = [&](int p) {  // smallest owned panel index > p
      int q = p + 1;
      q += ((me - q) % N + N) % N;
      return q;
    };

    GPRC_CUDA(cudaEventRecord(D->ev_begin, s0));
    if (D->timeline_on) cudaEventRecord(D->timeline[0], s0);
    GPRC_CUDA(cudaStreamWaitEvent(s1, D->ev_begin, 0));
    GPRC_CUDA(cudaStreamWaitEvent(sc, D->ev_begin, 0));
    if (owner(0) == me) {
      tl(0, 0, s1);
      if ((rc = factor_panel(0))) break;
      tl(0, 1, s1);
      GPRC_CUDA(cudaStreamWaitEvent(sc, D->ev_packed, 0));
    }
    tl(0, 2, sc);
    GPRC_NCCL(api, api.Broadcast(Pbuf[0], Pbuf[0], (size_t)n_pad * PANEL + OUTER_BLOCKS * NB * NB, ncclDouble, owner(0),
                                 D->comm, sc));
    tl(0, 3, sc);
    GPRC_CUDA(cudaEventRecord(D->ev_bcast[0], sc));
    for (int p = 0; p < npan && rc == 0; ++p) {
      const bool own_next = (p + 1 < npan) && owner(p + 1) == me;
      if (own_next) {
        // LA: bring panel p + 1 up to date with panel p, then factor it -- all on the high-priority stream
        GPRC_CUDA(cudaStreamWaitEvent(s1, D->ev_bcast[p & 1], 0));
        if (p > 0) GPRC_CUDA(cudaStreamWaitEvent(s1, D->ev_rest, 0));
        tl(p + 1, 0, s1);
        if ((rc = update(p, p + 1, 1, s1))) break;
        if ((rc = factor_panel(p + 1))) break;
        tl(p + 1, 1, s1);
      }
      if (p + 1 < npan) {
        // broadcast of panel p + 1 into the other buffer: it is free once update p - 1 has finished reading it
        if (p > 0) GPRC_CUDA(cudaStreamWaitEvent(sc, D->ev_rest, 0));
        if (own_next) GPRC_CUDA(cudaStreamWaitEvent(sc, D->ev_packed, 0));
        const long rows = n_pad - (long)(p + 1) * PANEL;
        tl(p + 1, 2, sc);
        GPRC_NCCL(api, api.Broadcast(Pbuf[(p + 1) & 1], Pbuf[(p + 1) & 1],
                                     (size_t)rows * PANEL + OUTER_BLOCKS * NB * NB, ncclDouble, owner(p + 1), D->comm,
                                     sc));
        tl(p + 1, 3, sc);
        GPRC_CUDA(cudaEventRecord(D->ev_bcast[(p + 1) & 1], sc));
      }
      // rest(p): every owned panel right of p (and right of p + 1 if that one was just handled by LA)
      GPRC_CUDA(cudaStreamWaitEvent(s0, D->ev_bcast[p & 1], 0));
      tl(p, 4, s0);
      if ((rc = unpack(p))) break;
      const int first = next_owned_after(own_next ? p + 1 : p);
      const int count = (first < npan) ? (npan - 1 - first) / N + 1 : 0;
      if ((rc = update(p, first, count, s0))) break;
      tl(p, 5, s0);
      GPRC_CUDA(cudaEventRecord(D->ev_rest, s0));
    }
    if (rc) break;
    GPRC_CUDA(cudaStreamWaitEvent(s0, D->ev_packed, 0));
    GPRC_CUDA(cudaStreamWaitEvent(s0, D->ev_bcast[(npan - 1) & 1], 0));
    // the diagonal of L lives where its panel lives; the status word is the minimum over ranks
    GPRC_NCCL(api, api.AllReduce(diag, diag, (size_t)n_pad, ncclDouble, ncclSum, D->comm, s0));
    GPRC_NCCL(api, api.AllReduce(c->d_info, c->d_info, 1, ncclInt64, ncclMin, D->comm, s0));
    cudaEventRecord(e2, s0);

    double* bw = vec;           // working right-hand side
    double* xs = vec + n_pad;   // solution of the current sweep
    if (g) {
      // the factor is complete on every rank: ordinary single-GPU solves
      if ((rc = potrs_vec(c, g->F.L, n_pad, n_pad, dinv, dy, bw, xs, g->alpha))) break;
      cudaMemcpyAsync(xs, g->alpha, sizeof(double) * n_pad, cudaMemcpyDeviceToDevice, s0);
    } else {
    // ---- alpha = L^-T L^-1 y: panels in order, the right-hand side travels by broadcast ----
    cudaMemcpyAsync(bw, dy, sizeof(double) * n_pad, cudaMemcpyDeviceToDevice, s0);
    cudaMemsetAsync(xs, 0, sizeof(double) * n_pad, s0);
    for (int p = 0; p < npan; ++p) {
      if (owner(p) == me) {
        double* Av = virt(p);
        for (int j = p * OUTER_BLOCKS; j < (p + 1) * OUTER_BLOCKS; ++j) {
          const long below = n_pad - (long)(j + 1) * NB;
          const unsigned grid = (unsigned)((below + TRSV_ROWS - 1) / TRSV_ROWS);
          trsv_fwd_step_kernel<<<grid ? grid : 1, 256, 0, s0>>>(Av, n_pad, dinv, j, n_pad, bw, xs);
          c->launches++;
        }
      }
      GPRC_NCCL(api, api.Broadcast(vec, vec, (size_t)2 * n_pad, ncclDouble, owner(p), D->comm, s0));
    }
    cudaMemcpyAsync(bw, xs, sizeof(double) * n_pad, cudaMemcpyDeviceToDevice, s0);  // rhs of L^T x = z
    cudaMemsetAsync(xs, 0, sizeof(double) * n_pad, s0);
    for (int p = npan - 1; p >= 0; --p) {
      if (owner(p) == me) {
        double* Av = virt(p);
        for (int j = (p + 1) * OUTER_BLOCKS - 1; j >= p * OUTER_BLOCKS; --j) {
          const long below = n_pad - (long)(j + 1) * NB;
          const int parts = (int)((below + BWD_CHUNK - 1) / BWD_CHUNK);
          if (parts > 0) {
            trsv_bwd_left_partial_kernel<<<parts, 256, 0, s0>>>(Av, n_pad, j, n_pad, xs, partial);
            c->launches++;
          }
          trsv_bwd_left_diag_kernel<<<1, 256, 0, s0>>>(dinv, j, partial, parts, bw, xs);
          c->launches++;
        }
      }
      GPRC_NCCL(api, api.Broadcast(xs, xs, (size_t)n_pad, ncclDouble, owner(p), D->comm, s0));
    }
    }
    gp_reduce_kernel<<<1, 1024, 0, s0>>>(dy, xs, diag, n, c->d_scalars);
    c->launches++;
    cudaEventRecord(e3, s0);
    cudaMemcpyAsync(c->h_scalars, c->d_scalars, 4 * sizeof(double), cudaMemcpyDeviceToHost, s0);
    cudaMemcpyAsync(c->h_info, c->d_info, sizeof(long), cudaMemcpyDeviceToHost, s0);
    if (alpha) cudaMemcpyAsync(alpha, xs, sizeof(double) * n, cudaMemcpyDeviceToHost, s0);
    cudaError_t e = cudaStreamSynchronize(s0);
    if (e != cudaSuccess) {
      rc = set_error(-2, __FILE__, __LINE__, cudaGetErrorString(e));
      break;
    }
    *info = (*c->h_info == LONG_MAX) ? 0 : *c->h_info;
    *logp = -0.5 * c->h_scalars[0] - c->h_scalars[1] - (double)n / 2.0 * log(2.0 * M_PI);
    if (D->timeline_on) {
      cudaStreamSynchronize(s1);
      cudaStreamSynchronize(sc);
      for (size_t q = 0; q < tl_set.size(); ++q) {
        if (!tl_set[q]) continue;
        float f = 0.f;
        if (cudaEventElapsedTime(&f, D->timeline[0], D->timeline[q + 1]) == cudaSuccess) D->timeline_ms[q] = f;
      }
    }
    if (phase_ms) {
      float f = 0.f;
      cudaEventElapsedTime(&f, e0, e1);
      phase_ms[0] = f;
      cudaEventElapsedTime(&f, e1, e2);
      phase_ms[1] = f;
      cudaEventElapsedTime(&f, e2, e3);
      phase_ms[2] = f;
      cudaEventElapsedTime(&f, e0, e3);
      phase_ms[3] = f;
    }
  } while (0);
  cudaStreamSynchronize(sc);
  cudaStreamSynchronize(s1);
  cudaStreamSynchronize(s0);
  for (cudaEvent_t ev : {e0, e1, e2, e3})
    if (ev) cudaEventDestroy(ev);
  if (g) {
    if (rc == 0 && *info == 0) {
      g->X = dX;
      g->y = dy;
      g->F.dinv = dinv;
      g->F.diag = diag;
      g->logp = *logp;
      dX = dy = dinv = diag = nullptr;
      *replicate = g;
    } else {
      gpr_destroy(g);
    }
  }
  dfree(dX);
  dfree(Aloc);
  dfree(dinv);
  dfree(diag);
  dfree(Pbuf[0]);
  dfree(Pbuf[1]);
  dfree(vec);
  dfree(dy);
  dfree(partial);
  return rc;
}

extern "C" int gprc_dist_set_timeline(gprc_dist* D, int on) {
  GPRC_ARG(D != nullptr);
  D->timeline_on = on != 0;
  return 0;
}
// ms: npan x 6 doubles (row p: look-ahead + factorisation begin / end on the owner, broadcast begin / end, trailing update
// begin / end; milliseconds since the start of the factorisation on this rank's device; NaN = not recorded on this rank)
extern "C" int gprc_dist_get_timeline(gprc_dist* D, double* ms, int cap_panels, int* npan) {
  GPRC_ARG(D && npan);
  *npan = D->timeline_npan;
  if (ms) {
    const int np = std::min(cap_panels, D->timeline_npan);
    for (size_t q = 0; q < (size_t)np * 6 && q < D->timeline_ms.size(); ++q) ms[q] = D->timeline_ms[q];
  }
  return 0;
}

extern "C" int gprc_dist_gpr_fit(gprc_dist* D, const gprc_kernel* k, const double* X, int d, long n, const double* y,
                                 double noise, double* logp, double* alpha, long* info, double* phase_ms) {
  return dist_fit_impl(D, k, X, d, n, y, noise, logp, alpha, info, phase_ms, nullptr);
}

extern "C" int gprc_dist_gpr_fit_replicated(gprc_dist* D, const gprc_kernel* k, const double* X, int d, long n,
                                            const double* y, double noise, gprc_gpr** out, double* logp, long* info,
                                            double* phase_ms) {
  GPRC_ARG(out != nullptr);
  return dist_fit_impl(D, k, X, d, n, y, noise, logp, nullptr, info, phase_ms, out);
}
