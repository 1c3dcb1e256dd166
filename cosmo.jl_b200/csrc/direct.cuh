// direct.cuh -- direct solve of the reduced KKT system on the device (COSMO_B200_KKT_DIRECT).
//
// The engine's counterpart of QdldlKKTSolver / CholmodKKTSolver (kktsolver.jl:285-349): an exact solve of
//   [P + sigma I, A'; A, -R^-1] [y1; y2] = [x1; x2],   R = diag(rho),
// through the Schur complement of the s-block,  M = P + sigma I + A' R A  (the operator CG runs on,
// kktsolver_indirect.jl:57-67):  y1 = M^-1 (x1 + A'(rho .* x2)),  y2 = rho .* (A y1 - x2)  (engine.cu, kkt_core).
//
// M is held as a dense fp64 Cholesky factor L (M = L L'), whatever the model type: sigma = 1e-6 next to
// rho_i |a_i|^2 terms of order 1e3 is below fp32 resolution.
//
// Storage: lower triangle in 64 x 64 tiles, tile (I, J), I >= J, at tile_off(I, J), row-major inside the tile.
// n is padded to Npad = 64 NT with a unit diagonal and a zero right-hand side, so that no kernel has a ragged edge.
//
// Assembly (one pass per factorisation; every entry is summed in a fixed order, no atomics):
//   sparse rows of A   assemble_sparse_kernel: one warp per row r of M owns the row; it writes sigma, adds the
//                      lower part of P's row r, then walks A' row r (= column r of A) in ascending row order i and
//                      adds rho_i a_ir a_i[c] for c <= r.  Work: sum over sparse rows of nnz_i^2 / 2 scattered adds.
//   dense rows of A    (nnz_i >= 64 and 8 nnz_i >= n, e.g. the 2000 rows of F' and the all-ones row of the portfolio
//                      problem) are gathered, scaled by sqrt(rho_i), into the panel G' (Npad x nd, row-major) and
//                      added as the tile product G'G'^T (tile_update_kernel, the same kernel as the trailing update):
//                      nd n^2 multiply-adds at tile-product rate instead of nnz_i^2 / 2 scattered adds per row.
//
// Factorisation (right-looking tile Cholesky, three launches per tile column K):
//   potrf_kernel         POTRF of tile (K, K) in shared memory, one CTA (a pivot <= 0 sets the failure flag: M is not
//                        positive definite <=> the KKT matrix lacks the inertia (n, m, 0)).
//   trsm_kernel          every panel tile (I, K), I > K:  (I, K) := (I, K) L(K, K)^-T, one CTA per tile.
//   tile_update_kernel   every trailing tile (I, J), K < J <= I:  (I, J) -= L(I, K) L(J, K)^T  (SYRK / GEMM).
//                        fp64 FMAs from shared memory, 4 x 4 outputs per thread.
//
// Solve: trsv_persistent_kernel, one cooperative launch for both sweeps (see there).
#pragma once

#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include "common.cuh"

namespace cosmo {
namespace direct {

constexpr int NB = 64;                 // tile side
constexpr int kThreads = 256;
constexpr int kLd = NB + 1;            // padded row stride of tiles staged in shared memory

__host__ __device__ inline size_t tile_off(long long I, long long J) { return (size_t)((I * (I + 1) / 2 + J) * (NB * NB)); }
__device__ inline size_t elem_off(int r, int c) { return tile_off(r / NB, c / NB) + (size_t)(r % NB) * NB + (c % NB); }

// dense-row rule of the assembly split (see the file comment)
__host__ inline bool dense_row(long long nnz_row, long long n) { return nnz_row >= 64 && 8 * nnz_row >= n; }

// ---- assembly ----------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kThreads) assemble_sparse_kernel(int n, int Npad, double* __restrict__ L, CsrView<T> P,
                                                                    CsrView<T> At, CsrView<T> A, const T* __restrict__ rho,
                                                                    const unsigned char* __restrict__ dense, double sigma) {
  const int lane = threadIdx.x & 31;
  const long long r = ((long long)blockIdx.x * kThreads + threadIdx.x) >> 5;
  if (r >= Npad) return;
  const int ri = (int)r;
  if (ri >= n) {
    if (lane == 0) L[elem_off(ri, ri)] = 1.0;
    return;
  }
  if (lane == 0) L[elem_off(ri, ri)] = sigma;
  __syncwarp();
  for (int k = P.rowptr[ri] + lane; k < P.rowptr[ri + 1]; k += 32) {
    const int c = P.col[k];
    if (c <= ri) L[elem_off(ri, c)] += (double)P.val[k];
  }
  __syncwarp();
  for (int k = At.rowptr[ri]; k < At.rowptr[ri + 1]; ++k) {
    const int i = At.col[k];
    if (dense[i]) continue;
    const double w = (double)rho[i] * (double)At.val[k];
    for (int kk = A.rowptr[i] + lane; kk < A.rowptr[i + 1]; kk += 32) {
      const int c = A.col[kk];
      if (c > ri) break;                // columns ascend inside a row
      L[elem_off(ri, c)] += w * (double)A.val[kk];
    }
    __syncwarp();
  }
}

// G'[c, k] = sqrt(rho_i) A[i, c] for the k-th dense row i (G' zeroed beforehand)
template <typename T>
__global__ void __launch_bounds__(kThreads) gather_dense_kernel(const int* __restrict__ rows, long long ldg, CsrView<T> A,
                                                                 const T* __restrict__ rho, double* __restrict__ Gt) {
  const int k = blockIdx.x;
  const int i = rows[k];
  const double s = sqrt((double)rho[i]);
  for (int kk = A.rowptr[i] + threadIdx.x; kk < A.rowptr[i + 1]; kk += kThreads)
    Gt[(size_t)A.col[kk] * ldg + k] = s * (double)A.val[kk];
}

// ---- tile product: C(I, J) += sign * sum_k X(I, k) X(J, k)^T over the lower tiles I >= J >= base ------------------
// PANEL = false: X = the packed factor, one k (= K, the current tile column), sign = -1 (trailing update).
// PANEL = true:  X = G' (row-major, leading dimension ldg), k over ldg / NB tiles, sign = +1 (dense-row assembly).
template <bool PANEL>
__global__ void __launch_bounds__(kThreads) tile_update_kernel(double* __restrict__ L, int NT, int base, int K,
                                                                const double* __restrict__ Gt, long long ldg, double sign) {
  constexpr int KC = 16;
  __shared__ double As[KC][NB + 1];
  __shared__ double Bs[KC][NB + 1];
  const long long t = blockIdx.x;
  long long Ip = (long long)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
  while (Ip * (Ip + 1) / 2 > t) --Ip;
  while ((Ip + 1) * (Ip + 2) / 2 <= t) ++Ip;
  const int I = base + (int)Ip;
  const int J = base + (int)(t - Ip * (Ip + 1) / 2);
  (void)NT;
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  double acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
  const int nk = PANEL ? (int)(ldg / NB) : 1;
  const int lr = tid >> 2, lc = (tid & 3) * 4;   // loader: row lr, columns lc .. lc + 3 of a 64 x 16 chunk
  for (int k = 0; k < nk; ++k) {
    const double* XA;
    const double* XB;
    long long ld;
    if (PANEL) {
      XA = Gt + (size_t)I * NB * ldg + (size_t)k * NB;
      XB = Gt + (size_t)J * NB * ldg + (size_t)k * NB;
      ld = ldg;
    } else {
      XA = L + tile_off(I, K);
      XB = L + tile_off(J, K);
      ld = NB;
    }
    for (int kc = 0; kc < NB; kc += KC) {
      __syncthreads();
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        As[lc + e][lr] = XA[(size_t)lr * ld + kc + lc + e];
        Bs[lc + e][lr] = XB[(size_t)lr * ld + kc + lc + e];
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < KC; ++kk) {
        double a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = As[kk][ty + 16 * i];
#pragma unroll
        for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx + 16 * j];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
      }
    }
  }
  double* C = L + tile_off(I, J);
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = ty + 16 * i, c = tx + 16 * j;
      C[r * NB + c] = fma(sign, acc[i][j], C[r * NB + c]);
    }
}

// ---- POTRF of tile (K, K) + TRSM of the panel tiles (K + b, K) ---------------------------------------------------
__device__ inline void potrf_smem(double (*D)[kLd], int* fail) {
  const int tid = threadIdx.x;
  for (int j = 0; j < NB; ++j) {
    __syncthreads();
    if (tid == 0) {
      const double d = D[j][j];
      if (!(d > 0.0)) *fail = 1;
      D[j][j] = sqrt(d);
    }
    __syncthreads();
    for (int i = j + 1 + tid; i < NB; i += kThreads) D[i][j] = D[i][j] / D[j][j];
    __syncthreads();
    const int w = NB - 1 - j;
    for (int e = tid; e < w * w; e += kThreads) {
      const int i = j + 1 + e / w, k = j + 1 + e % w;
      if (k <= i) D[i][k] = fma(-D[i][j], D[k][j], D[i][k]);
    }
  }
  __syncthreads();
}

constexpr size_t kPanelSmem = 2 * sizeof(double) * NB * kLd;   // dynamic: D and B, above the 48 KB static limit

// POTRF of tile (K, K) in place, one CTA; also the reciprocal pivots the sweeps multiply by
__global__ void __launch_bounds__(kThreads) potrf_kernel(double* __restrict__ L, double* __restrict__ dinv, int K,
                                                          int* __restrict__ fail_flag) {
  extern __shared__ double psm[];
  double (*D)[kLd] = reinterpret_cast<double (*)[kLd]>(psm);
  __shared__ int fail;
  const int tid = threadIdx.x;
  if (tid == 0) fail = 0;
  double* Dg = L + tile_off(K, K);
  for (int e = tid; e < NB * NB; e += kThreads) D[e / NB][e % NB] = Dg[e];
  potrf_smem(D, &fail);
  for (int e = tid; e < NB * NB; e += kThreads) {
    const int r = e / NB, c = e % NB;
    Dg[e] = c <= r ? D[r][c] : 0.0;
  }
  if (tid < NB) dinv[(size_t)K * NB + tid] = 1.0 / D[tid][tid];
  if (tid == 0 && fail && *fail_flag == 0) *fail_flag = K + 1;   // the first tile column with a pivot <= 0
}

// TRSM of the panel: tile (K + 1 + b, K) := (K + 1 + b, K) L(K, K)^-T, one CTA per tile
__global__ void __launch_bounds__(kThreads) trsm_kernel(double* __restrict__ L, int K) {
  extern __shared__ double psm[];
  double (*D)[kLd] = reinterpret_cast<double (*)[kLd]>(psm);
  double (*B)[kLd] = reinterpret_cast<double (*)[kLd]>(psm + NB * kLd);
  const int tid = threadIdx.x;
  const double* Dg = L + tile_off(K, K);
  double* Bg = L + tile_off(K + 1 + blockIdx.x, K);
  for (int e = tid; e < NB * NB; e += kThreads) {
    D[e / NB][e % NB] = Dg[e];
    B[e / NB][e % NB] = Bg[e];
  }
  // X L(K,K)^T = B, column by column: X[:, j] = B[:, j] / L[j][j], then B[:, l] -= X[:, j] L[l][j] for l > j
  for (int j = 0; j < NB; ++j) {
    __syncthreads();
    if (tid < NB) B[tid][j] = B[tid][j] / D[j][j];
    __syncthreads();
    const int w = NB - 1 - j;
    for (int e = tid; e < NB * w; e += kThreads) {
      const int r = e / w, l = j + 1 + e % w;
      B[r][l] = fma(-B[r][j], D[l][j], B[r][l]);
    }
  }
  __syncthreads();
  for (int e = tid; e < NB * NB; e += kThreads) Bg[e] = B[e / NB][e % NB];
}

// ---- forward + backward sweep in one cooperative launch -------------------------------------------------------------
// CTA g owns the tile rows I = g, g + G, g + 2G, ... and keeps their partial right-hand sides in shared memory.
//   forward  (L y = b):  for J = 0 .. NT-1: the owner of J solves L(J,J) y_J = acc_J (one warp, substitution with the
//                        reciprocal pivots), publishes y_J and sets ready_f[J] = epoch; every other CTA spins on
//                        ready_f[J], reads y_J, and subtracts L(I, J) y_J from each of its rows I > J.
//   backward (L'x = y):  the same for I = NT-1 .. 0 with L(I, I)^T and the transposed products L(I, J)^T x_I.
// The chain of owners is the critical path, so everything that does not depend on the published block is issued before
// the wait: the tile of the next owned row goes to registers, and the next owner stages its diagonal tile.
// A CTA only ever waits for a tile column owned by another CTA of the same cooperative launch (co-resident by the
// launch's guarantee), and the owner of column J publishes it after waiting only for columns < J (forward) or > J
// (backward): the wait graph is acyclic, so the sweep cannot hang.  The flags carry the solve's epoch and are never
// reset.  Every sum runs in a fixed order.
template <typename T>
struct TrsvArgs {
  const double* L;
  const double* dinv;       // Npad reciprocal pivots
  int n, NT, G;
  const T* rhs;             // n
  T* out;                   // n
  double* y;                // Npad: published forward blocks
  double* x;                // Npad: published backward blocks
  unsigned* ready_f;        // NT
  unsigned* ready_b;        // NT
  unsigned epoch;
};

__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(unsigned* p, unsigned v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// diagonal tile J and its reciprocal pivots into shared memory (all threads; the caller synchronises)
__device__ __forceinline__ void stage_diag(const double* L, const double* dinv, int J, double (*Ld)[kLd], double* dv) {
  const double* Dg = L + tile_off(J, J);
  for (int e = threadIdx.x; e < NB * NB; e += kThreads) Ld[e / NB][e % NB] = Dg[e];
  if (threadIdx.x < NB) dv[threadIdx.x] = dinv[(size_t)J * NB + threadIdx.x];
}

__device__ __forceinline__ void spin_until(const unsigned* f, unsigned epoch) {
  while (ld_acquire_gpu(f) != epoch) __nanosleep(20);
}

template <typename T>
__global__ void __launch_bounds__(kThreads, 1) trsv_persistent_kernel(TrsvArgs<T> a) {
  extern __shared__ double smem[];
  double (*Ld)[kLd] = reinterpret_cast<double (*)[kLd]>(smem);   // diagonal tile
  double* dv = smem + NB * kLd;                                   // its reciprocal pivots
  double* vec = dv + NB;                                          // the published block of this step
  double* part = vec + NB;                                        // 4 x NB partial sums
  double* acc = part + 4 * NB;                                    // R x NB partial right-hand sides
  const int tid = threadIdx.x, lane = tid & 31, g = blockIdx.x, G = a.G, NT = a.NT;
  const int nrows = (NT - g + G - 1) / G;                         // tile rows I = g + G r, r < nrows
  for (int e = tid; e < nrows * NB; e += kThreads) {
    const long long idx = (long long)(g + G * (e / NB)) * NB + e % NB;
    acc[e] = idx < a.n ? (double)a.rhs[idx] : 0.0;
  }
  int staged = -1;
  // ---- forward ----
  const int row = tid >> 2, q4 = tid & 3;                         // thread (row, quarter): 16 columns of one tile row
  for (int J = 0; J < NT; ++J) {
    const int r0 = J + 1 > g ? (J + 1 - g + G - 1) / G : 0;       // first owned row > J
    const int I0 = g + G * r0;
    double2 pre[8];
    if (I0 < NT) {
      const double2* Tg = reinterpret_cast<const double2*>(a.L + tile_off(I0, J) + (size_t)row * NB + q4 * 16);
#pragma unroll
      for (int c = 0; c < 8; ++c) pre[c] = __ldg(Tg + c);
    }
    if (J % G == g) {
      if (staged != J) { stage_diag(a.L, a.dinv, J, Ld, dv); staged = J; }
      __syncthreads();
      if (tid < 32) {
        double* ac = acc + (J / G) * NB;
        double v0 = ac[lane], v1 = ac[lane + 32];
        for (int j = 0; j < NB; ++j) {
          const double yj = __shfl_sync(0xffffffffu, j < 32 ? v0 : v1, j & 31) * dv[j];
          if (j < 32) {
            if (lane == j) v0 = yj; else if (lane > j) v0 = fma(-Ld[lane][j], yj, v0);
            v1 = fma(-Ld[lane + 32][j], yj, v1);
          } else {
            if (lane == j - 32) v1 = yj; else if (lane > j - 32) v1 = fma(-Ld[lane + 32][j], yj, v1);
          }
        }
        vec[lane] = v0; vec[lane + 32] = v1;
        ac[lane] = v0; ac[lane + 32] = v1;          // the owner keeps y_J for the backward sweep
        __stcg(a.y + (size_t)J * NB + lane, v0);
        __stcg(a.y + (size_t)J * NB + lane + 32, v1);
        __syncwarp();
        if (lane == 0) { __threadfence(); st_release_gpu(a.ready_f + J, a.epoch); }
      }
      __syncthreads();
    } else {
      if (J + 1 < NT && (J + 1) % G == g) { stage_diag(a.L, a.dinv, J + 1, Ld, dv); staged = J + 1; }
      if (tid == 0) spin_until(a.ready_f + J, a.epoch);
      __syncthreads();
      if (tid < NB) vec[tid] = __ldcg(a.y + (size_t)J * NB + tid);
      __syncthreads();
    }
    // acc_I -= L(I, J) y_J for the owned rows I > J
    for (int r = r0; r < nrows; ++r) {
      const int I = g + G * r;
      double2 v[8];
      if (r == r0) {
#pragma unroll
        for (int c = 0; c < 8; ++c) v[c] = pre[c];
      } else {
        const double2* Tg = reinterpret_cast<const double2*>(a.L + tile_off(I, J) + (size_t)row * NB + q4 * 16);
#pragma unroll
        for (int c = 0; c < 8; ++c) v[c] = __ldg(Tg + c);
      }
      double s = 0.0;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        s = fma(v[c].x, vec[q4 * 16 + 2 * c], s);
        s = fma(v[c].y, vec[q4 * 16 + 2 * c + 1], s);
      }
      s += __shfl_xor_sync(0xffffffffu, s, 1);
      s += __shfl_xor_sync(0xffffffffu, s, 2);
      if (q4 == 0) acc[r * NB + row] -= s;
    }
    __syncthreads();
  }
  // ---- backward ----
  const int col = tid & (NB - 1), q = tid >> 6;                   // thread (column, quarter): 16 rows of one tile column
  for (int I = NT - 1; I >= 0; --I) {
    const int rl = I - 1 >= g ? (I - 1 - g) / G : -1;             // last owned row < I
    const int J0 = rl >= 0 ? g + G * rl : -1;
    double pre[16];
    if (J0 >= 0) {
      const double* Tg = a.L + tile_off(I, J0) + (size_t)(q * 16) * NB + col;
#pragma unroll
      for (int k = 0; k < 16; ++k) pre[k] = __ldg(Tg + (size_t)k * NB);
    }
    if (I % G == g) {
      if (staged != I) { stage_diag(a.L, a.dinv, I, Ld, dv); staged = I; }
      __syncthreads();
      if (tid < 32) {
        double* ac = acc + (I / G) * NB;
        double v0 = ac[lane], v1 = ac[lane + 32];
        for (int j = NB - 1; j >= 0; --j) {
          const double xj = __shfl_sync(0xffffffffu, j < 32 ? v0 : v1, j & 31) * dv[j];
          if (j < 32) {
            if (lane == j) v0 = xj; else if (lane < j) v0 = fma(-Ld[j][lane], xj, v0);
          } else {
            if (lane == j - 32) v1 = xj; else if (lane < j - 32) v1 = fma(-Ld[j][lane + 32], xj, v1);
            v0 = fma(-Ld[j][lane], xj, v0);
          }
        }
        vec[lane] = v0; vec[lane + 32] = v1;
        __stcg(a.x + (size_t)I * NB + lane, v0);
        __stcg(a.x + (size_t)I * NB + lane + 32, v1);
        __syncwarp();
        if (lane == 0) { __threadfence(); st_release_gpu(a.ready_b + I, a.epoch); }
        const long long base = (long long)I * NB;
        if (base + lane < a.n) a.out[base + lane] = (T)v0;
        if (base + lane + 32 < a.n) a.out[base + lane + 32] = (T)v1;
      }
      __syncthreads();
    } else {
      if (I >= 1 && (I - 1) % G == g) { stage_diag(a.L, a.dinv, I - 1, Ld, dv); staged = I - 1; }
      if (tid == 0) spin_until(a.ready_b + I, a.epoch);
      __syncthreads();
      if (tid < NB) vec[tid] = __ldcg(a.x + (size_t)I * NB + tid);
      __syncthreads();
    }
    // acc_J -= L(I, J)^T x_I for the owned rows J < I, the last one (the next owner's) first
    for (int r = rl; r >= 0; --r) {
      const int J = g + G * r;
      double v[16];
      if (r == rl) {
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = pre[k];
      } else {
        const double* Tg = a.L + tile_off(I, J) + (size_t)(q * 16) * NB + col;
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = __ldg(Tg + (size_t)k * NB);
      }
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < 16; ++k) s = fma(v[k], vec[q * 16 + k], s);
      part[q * NB + col] = s;
      __syncthreads();
      if (tid < NB) acc[r * NB + tid] -= (part[tid] + part[NB + tid]) + (part[2 * NB + tid] + part[3 * NB + tid]);
      __syncthreads();
    }
  }
}

inline size_t trsv_smem_bytes(int R) { return sizeof(double) * ((size_t)NB * kLd + 2 * NB + 4 * NB + (size_t)R * NB); }

}  // namespace direct
}  // namespace cosmo
