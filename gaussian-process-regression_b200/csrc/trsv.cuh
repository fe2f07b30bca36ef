// trsv.cuh -- the O(n^2), HBM-bound passes (north_star subsystem 3a): blocked triangular solves for
// alpha = L^-T (L^-1 y) (R/GPRclass.R:152 -- the reference calls dense solve() twice, i.e. two LU factorisations;
// here two substitutions), the symmetric GEMV of the GPC Newton step (R/GPCclass.R:82,85) and the reductions behind
// logp (R/GPRclass.R:153), logq (R/GPCclass.R:103) and fit()'s leading-minor rule (R/fit.R:119).
#pragma once
#include <cooperative_groups.h>
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "gemm.cuh"
#include "potrf.cuh"  // chol_wait_progress: the watchdog of the persistent kernels

namespace gprc {

constexpr int TRSV_ROWS = 512;  // rows of the rank-128 update per CTA

// One block step of the forward substitution L x = b (used by the multi-GPU solve, where a rank only owns some
// block columns; the single-GPU solve uses the cooperative sweeps below):
//   x_j = Linv_j b_j   (every CTA, redundantly; CTA 0 stores it)
//   b[rows below] -= L[rows, block j] x_j
// b is the working right-hand side (blocks > j are updated in place), x receives the solution.
__global__ void __launch_bounds__(256) trsv_fwd_step_kernel(const double* __restrict__ L, long ld,
                                                            const double* __restrict__ dinv, int j, long n,
                                                            double* __restrict__ b, double* __restrict__ x) {
  __shared__ double bj[NB], xj[NB], part[NB];
  const int tid = threadIdx.x, r = tid & (NB - 1), h = tid >> 7;
  if (tid < NB) bj[tid] = b[(long)j * NB + tid];
  __syncthreads();
  const double* Li = dinv + (long)j * NB * NB;
  double s = 0.0, s2 = 0.0;
#pragma unroll 16
  for (int c = h * 64; c < h * 64 + 64; c += 2) {  // explicit zeros above the diagonal
    s = fma(Li[r + c * NB], bj[c], s);
    s2 = fma(Li[r + (c + 1) * NB], bj[c + 1], s2);
  }
  s += s2;
  if (h == 1) part[r] = s;
  __syncthreads();
  if (h == 0) xj[r] = s + part[r];
  __syncthreads();
  if (blockIdx.x == 0 && tid < NB) x[(long)j * NB + tid] = xj[tid];
  const long row0 = (long)(j + 1) * NB + (long)blockIdx.x * TRSV_ROWS;
#pragma unroll
  for (int q = 0; q < TRSV_ROWS / 256; ++q) {
    const long row = row0 + q * 256 + tid;
    if (row < n) {
      const double* Lp = L + row + (long)j * NB * ld;
      double acc = 0.0, acc2 = 0.0;
#pragma unroll 16
      for (int c = 0; c < NB; c += 2) {
        acc = fma(Lp[(long)c * ld], xj[c], acc);
        acc2 = fma(Lp[(long)(c + 1) * ld], xj[c + 1], acc2);
      }
      b[row] -= acc + acc2;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Whole substitution sweeps in ONE cooperative launch: the block steps above are latency-bound (n/128 dependent
// launches of ~10 us of work each); here the grid stays resident and a grid-wide barrier separates the steps.
// Forward:  every CTA forms x_j = Linv_j b_j itself (128 KB from L2), updates its share of the rows below, sync.
// Backward: every CTA forms x_j = Linv_j^T b_j, updates its share of the columns left of block j, sync.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) trsv_fwd_coop_kernel(const double* __restrict__ L, long ld,
                                                            const double* __restrict__ dinv, int nt, long n,
                                                            double* __restrict__ b, double* __restrict__ x) {
  cooperative_groups::grid_group grid = cooperative_groups::this_grid();
  __shared__ double bj[NB], xj[NB], part[NB], quart[256];
  const int tid = threadIdx.x, r = tid & (NB - 1), h = tid >> 7;
  for (int j = 0; j < nt; ++j) {
    if (tid < NB) bj[tid] = __ldcg(b + (long)j * NB + tid);  // written by other CTAs in the previous step: bypass L1
    __syncthreads();
    const double* Li = dinv + (long)j * NB * NB;
    double s = 0.0, s2 = 0.0;
#pragma unroll 16
    for (int c = h * 64; c < h * 64 + 64; c += 2) {
      s = fma(Li[r + c * NB], bj[c], s);
      s2 = fma(Li[r + (c + 1) * NB], bj[c + 1], s2);
    }
    s += s2;
    if (h == 1) part[r] = s;
    __syncthreads();
    if (h == 0) xj[r] = s + part[r];
    __syncthreads();
    if (blockIdx.x == 0 && tid < NB) x[(long)j * NB + tid] = xj[tid];
    // rows below: 64 rows per CTA pass, 4 threads per row (one quarter of the 128 columns each) for memory-level
    // parallelism; the quarters are combined in shared memory in a fixed order
    const long first = (long)(j + 1) * NB;
    const int rr = tid & 63, cq = tid >> 6;
    for (long row0 = first + (long)blockIdx.x * 64; row0 < n; row0 += (long)gridDim.x * 64) {
      const long row = row0 + rr;
      double acc = 0.0, acc2 = 0.0;
      if (row < n) {
        const double* Lp = L + row + ((long)j * NB + cq * 32) * ld;
        const double* xq = xj + cq * 32;
#pragma unroll 16
        for (int c = 0; c < 32; c += 2) {
          acc = fma(Lp[(long)c * ld], xq[c], acc);
          acc2 = fma(Lp[(long)(c + 1) * ld], xq[c + 1], acc2);
        }
      }
      quart[cq * 64 + rr] = acc + acc2;
      __syncthreads();
      if (tid < 64 && row < n) b[row] = __ldcg(b + row) - ((quart[rr] + quart[64 + rr]) + (quart[128 + rr] + quart[192 + rr]));
      __syncthreads();
    }
    grid.sync();
  }
}

__global__ void __launch_bounds__(256) trsv_bwd_coop_kernel(const double* __restrict__ L, long ld,
                                                            const double* __restrict__ dinv, int nt,
                                                            double* __restrict__ b, double* __restrict__ x) {
  cooperative_groups::grid_group grid = cooperative_groups::this_grid();
  __shared__ double bj[NB], xj[NB];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int gwarp = blockIdx.x * 8 + warp, nwarps = gridDim.x * 8;
  for (int j = nt - 1; j >= 0; --j) {
    if (tid < NB) bj[tid] = __ldcg(b + (long)j * NB + tid);
    __syncthreads();
    const double* Li = dinv + (long)j * NB * NB;
    {
      double s[16];
#pragma unroll
      for (int rr = 0; rr < 16; ++rr) {
        const int r = warp + 8 * rr;
        double acc = 0.0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int c = lane + 32 * q;
          acc = fma(Li[c + r * NB], bj[c], acc);
        }
        s[rr] = acc;
      }
#pragma unroll
      for (int rr = 0; rr < 16; ++rr) {
        const double t = warp_sum(s[rr]);
        if (lane == 0) xj[warp + 8 * rr] = t;
      }
    }
    __syncthreads();
    if (blockIdx.x == 0 && tid < NB) x[(long)j * NB + tid] = xj[tid];
    double xr[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) xr[q] = xj[lane + 32 * q];
    const double* Lrow = L + (long)j * NB;
    const long ncols = (long)j * NB;  // columns left of block j: one warp per column, grid-strided
    for (long k = gwarp; k < ncols; k += nwarps) {
      const double* Lp = Lrow + k * ld;
      double acc = 0.0;
#pragma unroll
      for (int q = 0; q < 4; ++q) acc = fma(Lp[lane + 32 * q], xr[q], acc);
      acc = warp_sum(acc);
      if (lane == 0) b[k] = __ldcg(b + k) - acc;
    }
    grid.sync();
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Round 2: both sweeps as ONE dataflow kernel.  The cooperative sweeps above separate the n / 128 block steps by grid-wide
// barriers, and every step is a dependent chain of a barrier, a 128 x 128 matvec and a rank-128 update: 24 us per step,
// 19 ms at n = 50 000 against a 3 ms HBM floor.  Here a resident grid of G CTAs owns the row blocks cyclically (block i on
// CTA i mod G) and every row block is ONE CTA's job from start to finish:
//   forward   z_i = Linv_i (b_i - sum_{j<i} L[i, j] z_j)        tiles of block ROW i, j ascending
//   backward  x_i = Linv_i^T (z_i - sum_{j>i} L[j, i]^T x_j)     tiles of block COLUMN i, j descending
// A finished block is published with a release store to flag[i]; consumers acquire-poll the flag of the block they need
// next.  Nothing waits on a grid barrier: the CTAs far from the critical path stream their tiles of L at HBM rate while
// the critical path -- the owner of block i turning z_(i-1) into z_i: one 128 x 128 tile (prefetched into L2), the
// inverted diagonal block, one flag -- is a few microseconds per step.  Summation orders are fixed (bitwise reproducible).
// Deadlock freedom: blocks are totally ordered, every CTA handles its blocks in that order, and the grid is launched
// cooperatively (all CTAs resident).  A flag that never arrives raises `error` and traps instead of hanging the GPU.
// ---------------------------------------------------------------------------------------------------------------
// ld_acquire_gpu / st_release_gpu: gemm.cuh (the persistent substitution kernel uses the same pair)
__device__ __forceinline__ void flow_wait(const int* flag, int* error) {
  for (long spin = 0; ld_acquire_gpu(flag) == 0; ++spin) {
    if (spin > (1L << 26)) {  // seconds: a dependency that never arrives
      atomicOr(error, 1);
      __threadfence_system();
      __trap();
    }
  }
}

// z and x (n doubles each) must be filled with the sentinel bit pattern 0xFF..FF (a NaN no arithmetic produces) before
// the launch: a block is published simply by storing its 128 results, and a consumer polls the very elements it needs
// until they differ from the sentinel -- one L2 round trip instead of flag + data, no fences.  Results that are NaN
// themselves are stored as the canonical quiet NaN.
constexpr unsigned long long TRSV_SENTINEL = 0xFFFFFFFFFFFFFFFFull;
constexpr int TRSV_FLOW_SMEM = NB * NB * 8 + 2 * NB * 8;  // inverted diagonal block + two 128-vectors

// polite = true: this consumer is far from the block that is being computed right now (it cannot use the value for a
// while), so it sleeps between polls and leaves the L2 lines of the front to the CTA on the critical path
__device__ __forceinline__ double flow_poll(const double* p, int* error, bool polite = false) {
  unsigned long long v;
  long spin = 0;
  for (;;) {
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    if (v != TRSV_SENTINEL) break;
    if (polite) __nanosleep(400);
    if (++spin > (1L << 26)) {  // seconds: a dependency that never arrives
      atomicOr(error, 1);
      __threadfence_system();
      __trap();
    }
  }
  return __longlong_as_double((long long)v);
}
__device__ __forceinline__ void flow_publish(double* p, double v) {
  unsigned long long u = (unsigned long long)__double_as_longlong(v);
  if (v != v) u = 0x7FF8000000000000ull;  // never the sentinel
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(u) : "memory");
}

// The units of work are half tiles (128 x 64 forward, 64 x 128 backward), double-buffered in registers: while one unit is
// multiplied, the loads of the next are in flight (64 KB per CTA), and the loads of the unit next to the diagonal are
// issued BEFORE its right-hand side is polled, so that the critical path per block step is: poll -> 32 FMAs ->
// combine -> 128 x 128 matvec with the inverted diagonal block from shared memory -> store.
__global__ void __launch_bounds__(256, 1) trsv_flow_kernel(const double* __restrict__ L, long ld,
                                                           const double* __restrict__ dinv, int nt,
                                                           const double* __restrict__ b, double* __restrict__ z,
                                                           double* __restrict__ x, int* __restrict__ error) {
  extern __shared__ __align__(16) unsigned char flow_raw[];
  double* Ls = reinterpret_cast<double*>(flow_raw);  // Linv_i, column-major 128 x 128
  double* part = Ls + NB * NB;                       // [128]
  double* acc_s = part + NB;                         // [128]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = gridDim.x, me = blockIdx.x;

  // ---------------- forward: thread = (row r, 32-column half h of the current 64-column unit) ----------------
  {
    const int r = tid & (NB - 1), h = tid >> 7;
    for (int i = me; i < nt; i += G) {
      __syncthreads();  // the previous block's readers of Ls / acc_s are done
      {
        const double* Li = dinv + (long)i * NB * NB;
        for (int e = tid; e < NB * NB / 2; e += 256)
          reinterpret_cast<double2*>(Ls)[e] = __ldg(reinterpret_cast<const double2*>(Li) + e);
      }
      const double bi = b[(long)i * NB + r];                             // off the critical path
      const double* Lrow = L + (long)i * NB + r + (long)(h * 32) * ld;  // unit u adds 64 u columns
      const double* zq = z + h * 32 + lane;                              // unit u adds 64 u
      double A[32], B[32];
      double a0 = 0.0, a1 = 0.0;
      const int units = 2 * i;
      if (units > 0) {
#pragma unroll
        for (int c = 0; c < 32; ++c) A[c] = Lrow[(long)c * ld];
      }
      for (int u = 0; u < units; u += 2) {
        {  // unit u + 1 -> B (always exists: two units per tile)
          const double* p = Lrow + (long)(u + 1) * 64 * ld;
#pragma unroll
          for (int c = 0; c < 32; ++c) B[c] = p[(long)c * ld];
        }
        {
          const double zl = flow_poll(zq + (long)u * 64, error, u + 4 < units);
#pragma unroll
          for (int c = 0; c < 32; c += 2) {
            a0 = fma(A[c], __shfl_sync(0xffffffffu, zl, c), a0);
            a1 = fma(A[c + 1], __shfl_sync(0xffffffffu, zl, c + 1), a1);
          }
        }
        if (u + 2 < units) {
          const double* p = Lrow + (long)(u + 2) * 64 * ld;
#pragma unroll
          for (int c = 0; c < 32; ++c) A[c] = p[(long)c * ld];
        }
        {
          const double zl = flow_poll(zq + (long)(u + 1) * 64, error, u + 5 < units);
#pragma unroll
          for (int c = 0; c < 32; c += 2) {
            a0 = fma(B[c], __shfl_sync(0xffffffffu, zl, c), a0);
            a1 = fma(B[c + 1], __shfl_sync(0xffffffffu, zl, c + 1), a1);
          }
        }
      }
      // acc = b_i - (the two column halves, fixed order)
      const double mine = a0 + a1;
      if (h == 1) part[r] = mine;
      __syncthreads();  // also: Ls is complete
      if (h == 0) acc_s[r] = bi - (mine + part[r]);
      __syncthreads();
      // z_i = Linv_i acc   (explicit zeros above the diagonal of Linv_i)
      double s0 = 0.0, s1 = 0.0;
#pragma unroll 16
      for (int c = h * 64; c < h * 64 + 64; c += 2) {
        s0 = fma(Ls[r + c * NB], acc_s[c], s0);
        s1 = fma(Ls[r + (c + 1) * NB], acc_s[c + 1], s1);
      }
      const double sv = s0 + s1;
      if (h == 1) part[r] = sv;
      __syncthreads();
      if (h == 0) flow_publish(z + (long)i * NB + r, sv + part[r]);
    }
  }

  // ---------------- backward: warp w owns columns 16 w .. 16 w + 15 of the block, lane l rows l and l + 32 of the
  // current 64-row unit ----------------
  for (int ib = me; ib < nt; ib += G) {
    const int i = nt - 1 - ib;
    __syncthreads();
    {
      const double* Li = dinv + (long)i * NB * NB;
      for (int e = tid; e < NB * NB / 2; e += 256)
        reinterpret_cast<double2*>(Ls)[e] = __ldg(reinterpret_cast<const double2*>(Li) + e);
    }
    // z_i (this block's forward result, complete long ago): lane cc of warp w fetches entry 16 w + cc now
    const double zi = (lane < 16) ? flow_poll(z + (long)i * NB + warp * 16 + lane, error) : 0.0;
    const double* Lcol = L + lane + ((long)i * NB + warp * 16) * ld;  // unit: rows 64 v .. 64 v + 63, v descending
    double A[32], B[32], acc[16];
#pragma unroll
    for (int cc = 0; cc < 16; ++cc) acc[cc] = 0.0;
    const int vhi = 2 * nt - 1, vlo = 2 * (i + 1);  // units vhi, vhi - 1, ..., vlo  (an even number of them)
    if (vhi >= vlo) {
      const double* p = Lcol + (long)vhi * 64;
#pragma unroll
      for (int cc = 0; cc < 16; ++cc) {
        A[2 * cc] = p[(long)cc * ld];
        A[2 * cc + 1] = p[(long)cc * ld + 32];
      }
    }
    for (int v = vhi; v >= vlo; v -= 2) {
      {
        const double* p = Lcol + (long)(v - 1) * 64;
#pragma unroll
        for (int cc = 0; cc < 16; ++cc) {
          B[2 * cc] = p[(long)cc * ld];
          B[2 * cc + 1] = p[(long)cc * ld + 32];
        }
      }
      {
        const bool far = v - 4 > vlo;
        const double x0 = flow_poll(x + (long)v * 64 + lane, error, far), x1 = flow_poll(x + (long)v * 64 + lane + 32, error, far);
#pragma unroll
        for (int cc = 0; cc < 16; ++cc) acc[cc] = fma(A[2 * cc + 1], x1, fma(A[2 * cc], x0, acc[cc]));
      }
      if (v - 2 >= vlo) {
        const double* p = Lcol + (long)(v - 2) * 64;
#pragma unroll
        for (int cc = 0; cc < 16; ++cc) {
          A[2 * cc] = p[(long)cc * ld];
          A[2 * cc + 1] = p[(long)cc * ld + 32];
        }
      }
      {
        const bool far = v - 5 > vlo;
        const double x0 = flow_poll(x + (long)(v - 1) * 64 + lane, error, far),
                     x1 = flow_poll(x + (long)(v - 1) * 64 + lane + 32, error, far);
#pragma unroll
        for (int cc = 0; cc < 16; ++cc) acc[cc] = fma(B[2 * cc + 1], x1, fma(B[2 * cc], x0, acc[cc]));
      }
    }
#pragma unroll
    for (int cc = 0; cc < 16; ++cc) {
      const double t = warp_sum(acc[cc]);
      if (lane == cc) acc_s[warp * 16 + cc] = zi - t;
    }
    __syncthreads();  // acc_s and Ls complete
    // x_i = Linv_i^T acc: entry r is column r of Linv_i dotted with acc
    double tv[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) tv[q] = acc_s[lane + 32 * q];
#pragma unroll
    for (int rr = 0; rr < 16; ++rr) {
      const int rcol = warp * 16 + rr;
      double t = 0.0;
#pragma unroll
      for (int q = 0; q < 4; ++q) t = fma(Ls[lane + 32 * q + rcol * NB], tv[q], t);
      t = warp_sum(t);
      if (lane == 0) flow_publish(x + (long)i * NB + rcol, t);
    }
  }
}

inline int coop_grid(gprc_ctx* ctx, const void* func, long work_items) {
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, func, 256, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
  long g = (long)ctx->sm_count * (per_sm > 2 ? 2 : per_sm);
  if (g > work_items) g = work_items;
  return (int)(g < 1 ? 1 : g);
}

// x = L^-T L^-1 rhs.  work, tmp: n doubles each; rhs is left untouched.
// GPRC_OPT_TRSV = 1: the dataflow kernel (one launch for both sweeps; `work` holds its flags); 0: the round-1 cooperative
// sweeps with grid-wide barriers.
inline int potrs_vec(gprc_ctx* ctx, const double* L, long n, long ld, const double* dinv, const double* rhs,
                     double* work, double* tmp, double* x) {
  int nt = (int)(n / NB);
  const bool use_coop = ctx->opt_trsv == 0;
  if (!use_coop) {
    static bool configured[64] = {false};
    if (!configured[ctx->device & 63]) {
      GPRC_CUDA(cudaFuncSetAttribute(trsv_flow_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TRSV_FLOW_SMEM));
      configured[ctx->device & 63] = true;
    }
    const int grid = std::min(nt, ctx->sm_count);  // one resident CTA per SM (128 KB of shared memory each)
    int* error = reinterpret_cast<int*>(work);
    GPRC_CUDA(cudaMemsetAsync(work, 0, sizeof(int) * 2, ctx->stream));
    GPRC_CUDA(cudaMemsetAsync(tmp, 0xFF, sizeof(double) * n, ctx->stream));  // sentinel: "not yet computed"
    GPRC_CUDA(cudaMemsetAsync(x, 0xFF, sizeof(double) * n, ctx->stream));
    void* args[] = {(void*)&L, (void*)&ld, (void*)&dinv, (void*)&nt, (void*)&rhs, (void*)&tmp, (void*)&x, (void*)&error};
    GPRC_CUDA(cudaLaunchCooperativeKernel((const void*)trsv_flow_kernel, dim3(grid), dim3(256), args, TRSV_FLOW_SMEM,
                                          ctx->stream));
    ctx->launches++;
    return 0;
  }
  GPRC_CUDA(cudaMemcpyAsync(work, rhs, n * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
  {
    const int grid = coop_grid(ctx, (const void*)trsv_fwd_coop_kernel, (n + 63) / 64);
    void* args[] = {(void*)&L, (void*)&ld, (void*)&dinv, (void*)&nt, (void*)&n, (void*)&work, (void*)&tmp};
    GPRC_CUDA(cudaLaunchCooperativeKernel((const void*)trsv_fwd_coop_kernel, dim3(grid), dim3(256), args, 0, ctx->stream));
    ctx->launches++;
  }
  {
    const int grid = coop_grid(ctx, (const void*)trsv_bwd_coop_kernel, (n + 7) / 8);
    void* args[] = {(void*)&L, (void*)&ld, (void*)&dinv, (void*)&nt, (void*)&tmp, (void*)&x};
    GPRC_CUDA(cudaLaunchCooperativeKernel((const void*)trsv_bwd_coop_kernel, dim3(grid), dim3(256), args, 0, ctx->stream));
    ctx->launches++;
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// Triangular solve with a few hundred right-hand sides, as ONE dataflow kernel (the append of training points,
// gprc_gpr_append):  T <- T L^-T  for a panel T of `rows` right-hand sides over the leading 128 nt columns of a factor L.
// T is stored like K_star^T (right-hand side r, column c at T[r + c ldt]); in the append it is the new block row of L
// itself.  Work unit (i, g) = block row i of L, group g of 128 right-hand sides:
//     C = T_i[g] - sum_{j<i} L[i, j] V_j[g]      (DMMA GEMM, K = 128 i; TrsmLeftUpdatePolicy's epilogue)
//     V_i[g] = Linv_i C                          (DMMA GEMM, K = 128, in place)
// The substitution kernels of the predictive variance (TrsmLeft*Policy, trsm_persistent_kernel) run unit (i, g) only once
// unit (i - 1, g) is complete, so one group of right-hand sides keeps ONE SM busy for all nt (nt + 1) / 2 tile products.
// Here the units are handed out i-major by an atomic counter and every unit streams in block j of its GEMM as soon as
// group g's block row j is published (progress[g] >= j + 1, release / acquire, checked by the producer lane per 128-wide
// k-block): the units of one group run on different SMs and overlap, and the critical path per block row is the product
// with the tile next to the diagonal (prefetched into L2 when the unit starts) plus the product with Linv_i.  All groups
// run in the same launch.  Every prerequisite of a unit has a smaller index and units only go to running CTAs, so no
// co-residency is needed; a dependency that never arrives sets `error` (chol_wait_progress) and the host reports it.
// Summation orders are fixed: bitwise reproducible.
// ---------------------------------------------------------------------------------------------------------------
struct TrsmFlowParams {
  const double* L;
  long ldl;
  const double* dinv;
  double* T;
  long ldt;
  int nt, ngroups;
  unsigned long long* next;  // unit counter (zeroed by the host)
  int* error;                // watchdog (zeroed by the host)
  int* progress;             // [ngroups] block rows published per group (zeroed by the host)
};

__global__ void __launch_bounds__(GEMM_THREADS, 1) trsm_flow_kernel(const TrsmFlowParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double* smem = reinterpret_cast<double*>(smem_raw);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + STAGES * STAGE_DOUBLES * 8);
  uint64_t* empty = full + STAGES;
  __shared__ long long s_item;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(smem_u32(full + s), 1);
      mbar_init(smem_u32(empty + s), GEMM_CONSUMERS / 32);
    }
    mbar_fence_init();
  }
  __syncthreads();
  const long long total = (long long)p.nt * p.ngroups;
  long long base = 0;  // k-slices pushed through the ring so far (identical for producer and consumers)
  const WarpCoord wc;
  for (;;) {
    if (threadIdx.x == 0) {
      long long item = (long long)atomicAdd(p.next, 1ULL);
      if (*reinterpret_cast<volatile int*>(p.error)) item = total;
      s_item = item;
    }
    __syncthreads();
    const long long item = s_item;
    if (item >= total) break;
    const int g = (int)(item % p.ngroups), i = (int)(item / p.ngroups);
    double* Ctile = p.T + (long)g * NB + (long)i * NB * p.ldt;  // element (m, n) of the tile at C[n + m * ldt]
    // ---- phase 0: C -= sum_{j<i} L[i, j] V_j, block j as soon as it is published ----
    {
      TileWork w;
      w.A = p.L + (long)i * NB;
      w.lda = p.ldl;
      w.B = p.T + (long)g * NB;  // element (k, n) = V[k, n] = T[n + k * ldt]
      w.ldb = p.ldt;
      w.k_begin = 0;
      w.k_end = i * NB;
      const int KT = i * (NB / BK);
      if (warp == GEMM_CONSUMERS / 32) {
        if (lane == 0) {
          bool ok = true;
          for (int kt = 0; kt < KT; ++kt) {
            if (kt % (NB / BK) == 0) {
              ok = ok && chol_wait_progress(p.progress + g, kt / (NB / BK) + 1, p.error);
              fence_proxy_async();  // V_j was written with ordinary stores and is read by the TMA engine
            }
            const long long gk = base + kt;
            const int s = (int)(gk % STAGES);
            if (gk >= STAGES) mbar_wait(smem_u32(empty + s), (uint32_t)(((gk / STAGES) - 1) & 1));
            if (ok) produce_stage<false>(w, kt * BK, smem + s * STAGE_DOUBLES, smem_u32(full + s));
            else mbar_arrive(smem_u32(full + s));  // watchdog fired: release the consumers (results are garbage, error set)
          }
        }
      } else if (KT > 0) {
        Acc acc;
#pragma unroll
        for (int mb = 0; mb < 8; ++mb)
#pragma unroll
          for (int nb = 0; nb < 4; ++nb) acc[mb][nb][0] = acc[mb][nb][1] = 0.0;
        // the C tile, the tile next to the diagonal and Linv_i: everything the critical path reads after the last poll
        const double* Lnext = p.L + (long)i * NB + (long)(i - 1) * NB * p.ldl;
        const double* Li = p.dinv + (long)i * NB * NB;
#pragma unroll
        for (int qq = 0; qq < 4; ++qq) {
          const int line = threadIdx.x + qq * GEMM_CONSUMERS;
          prefetch_l2(Ctile + (long)(line >> 3) * p.ldt + (line & 7) * 16);
          prefetch_l2(Lnext + (long)(line >> 3) * p.ldl + (line & 7) * 16);
          prefetch_l2(Li + (long)line * 16);
        }
        for (int kt = 0; kt < KT; ++kt) {
          const long long gk = base + kt;
          const int s = (int)(gk % STAGES);
          mbar_wait(smem_u32(full + s), (uint32_t)((gk / STAGES) & 1));
          compute_stage<false>(smem + s * STAGE_DOUBLES, wc, acc);
          __syncwarp();
          if (lane == 0) mbar_arrive(smem_u32(empty + s));
        }
        TrsmLeftUpdatePolicy pol{p.L, p.ldl, p.T, p.ldt, i};
        TrsmLeftUpdatePolicy::Tile tile{Ctile};
        pol.epilogue(tile, acc, smem);
        __threadfence();
        fence_proxy_async();  // phase 1 reads C through the TMA engine
      }
      __syncthreads();
      base += KT;
    }
    // ---- phase 1: V_i = Linv_i C, in place ----
    {
      TileWork w;
      w.A = p.dinv + (long)i * NB * NB;
      w.lda = NB;
      w.B = Ctile;  // element (k, n) = C[k, n]
      w.ldb = p.ldt;
      w.k_begin = 0;
      w.k_end = NB;
      constexpr int KT = NB / BK;
      if (warp == GEMM_CONSUMERS / 32) {
        if (lane == 0) {
          fence_proxy_async();
          for (int kt = 0; kt < KT; ++kt) {
            const long long gk = base + kt;
            const int s = (int)(gk % STAGES);
            if (gk >= STAGES) mbar_wait(smem_u32(empty + s), (uint32_t)(((gk / STAGES) - 1) & 1));
            produce_stage<false>(w, kt * BK, smem + s * STAGE_DOUBLES, smem_u32(full + s));
          }
        }
      } else {
        Acc acc;
#pragma unroll
        for (int mb = 0; mb < 8; ++mb)
#pragma unroll
          for (int nb = 0; nb < 4; ++nb) acc[mb][nb][0] = acc[mb][nb][1] = 0.0;
        for (int kt = 0; kt < KT; ++kt) {
          const long long gk = base + kt;
          const int s = (int)(gk % STAGES);
          mbar_wait(smem_u32(full + s), (uint32_t)((gk / STAGES) & 1));
          compute_stage<false>(smem + s * STAGE_DOUBLES, wc, acc);
          __syncwarp();
          if (lane == 0) mbar_arrive(smem_u32(empty + s));
        }
        // every k-slice of C has landed in shared memory (this warp passed the last full barrier): overwrite C by V_i
#pragma unroll
        for (int mb = 0; mb < 8; ++mb) {
          double* cp = Ctile + (long)wc.row(mb) * p.ldt;
#pragma unroll
          for (int nb = 0; nb < 4; ++nb)
            *reinterpret_cast<double2*>(cp + wc.col(nb, 0)) = make_double2(acc[mb][nb][0], acc[mb][nb][1]);
        }
        __threadfence();
        fence_proxy_async();  // the next units read V_i through the TMA engine
      }
      __syncthreads();
      base += KT;
    }
    if (threadIdx.x == 0) st_release_gpu(p.progress + g, i + 1);
  }
}

// T <- T L^-T for `rows` right-hand sides (T: round_up(rows, 128) x 128 nt, leading dimension ldt; the padding rows are
// solved too and must hold finite values).  sched: ngroups + 4 ints of device scratch.
inline int trsm_flow(gprc_ctx* ctx, const double* L, long ldl, const double* dinv, int nt, double* T, long ldt, long rows,
                     int* sched) {
  static bool configured[64] = {false};
  if (!configured[ctx->device & 63]) {
    GPRC_CUDA(cudaFuncSetAttribute(trsm_flow_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
    configured[ctx->device & 63] = true;
  }
  const int ngroups = (int)((rows + NB - 1) / NB);
  if (nt <= 0 || ngroups <= 0) return 0;
  GPRC_CUDA(cudaMemsetAsync(sched, 0, sizeof(int) * (ngroups + 4), ctx->stream));
  TrsmFlowParams p;
  p.L = L;
  p.ldl = ldl;
  p.dinv = dinv;
  p.T = T;
  p.ldt = ldt;
  p.nt = nt;
  p.ngroups = ngroups;
  p.next = reinterpret_cast<unsigned long long*>(sched);
  p.error = sched + 2;
  p.progress = sched + 4;
  const int grid = (int)std::min<long>((long)nt * ngroups, ctx->sm_count);
  trsm_flow_kernel<<<grid, GEMM_THREADS, GEMM_SMEM_BYTES, ctx->stream>>>(p);
  ctx->launches++;
  GPRC_CUDA(cudaGetLastError());
  return 0;
}

// y = K^T v for a column-major n x n matrix (K symmetric in the callers): warp per column, coalesced.
__global__ void __launch_bounds__(256) gemv_t_kernel(const double* __restrict__ K, long ld, long n,
                                                     const double* __restrict__ v, double* __restrict__ y) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long col = (long)blockIdx.x * 8 + warp;
  if (col >= n) return;
  const double* Kp = K + col * ld;
  double s = 0.0;
  for (long i = lane; i < n; i += 32) s = fma(Kp[i], v[i], s);
  s = warp_sum(s);
  if (lane == 0) y[col] = s;
}
inline int gemv_t(gprc_ctx* ctx, const double* K, long ld, long n, const double* v, double* y) {
  gemv_t_kernel<<<(unsigned)((n + 7) / 8), 256, 0, ctx->stream>>>(K, ld, n, v, y);
  ctx->launches++;
  GPRC_CUDA(cudaGetLastError());
  return 0;
}

// Reductions over the factor and the solution (single CTA, fixed order => reproducible):
//   out[0] = sum_i y_i alpha_i            out[1] = sum_i log L_ii         out[2] = sum_i L_ii
//   out[3] = min_i sum_{k<=i} 2 log L_kk  (log of the smallest leading-minor determinant, R/fit.R:119)
__global__ void __launch_bounds__(1024) gp_reduce_kernel(const double* __restrict__ y, const double* __restrict__ alpha,
                                                         const double* __restrict__ diag, long n,
                                                         double* __restrict__ out) {
  __shared__ double s_dot[1024], s_log[1024], s_sum[1024], s_minpre[1024];
  const int tid = threadIdx.x;
  const long chunk = (n + 1023) / 1024;
  const long lo = tid * chunk, hi = (lo + chunk < n) ? lo + chunk : n;
  double dot = 0.0, slog = 0.0, ssum = 0.0, minpre = INFINITY;
  for (long i = lo; i < hi; ++i) {
    if (y && alpha) dot = fma(y[i], alpha[i], dot);
    if (diag) {
      const double d = diag[i];
      slog += log(d);
      ssum += d;
      minpre = fmin(minpre, 2.0 * slog);
    }
  }
  s_dot[tid] = dot;
  s_log[tid] = slog;
  s_sum[tid] = ssum;
  s_minpre[tid] = minpre;
  __syncthreads();
  if (tid == 0) {
    double tdot = 0.0, tlog = 0.0, tsum = 0.0, tmin = INFINITY;
    for (int t = 0; t < 1024; ++t) {
      tmin = fmin(tmin, 2.0 * tlog + s_minpre[t]);  // prefix of earlier chunks + local min prefix
      tdot += s_dot[t];
      tlog += s_log[t];
      tsum += s_sum[t];
    }
    out[0] = tdot;
    out[1] = tlog;
    out[2] = tsum;
    out[3] = tmin;
  }
}

}  // namespace gprc
