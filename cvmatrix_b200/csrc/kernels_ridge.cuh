// Cross-validated ridge regression over a fold batch (sm_100a): B = (XTX_f + lambda_l I)^-1 XTY_f for every fold f and
// penalty lambda_l of a pass, by a right-looking blocked Cholesky factorisation in float64, then the weighted PRESS of
// the fold's validation rows for every penalty.  All arithmetic is float64 for both model dtypes.
//
// Every (fold, penalty) pair of a pass owns one (K + M) x K row-major float64 matrix: rows 0 .. K-1 hold the lower
// triangle of XTX + lambda I, rows K .. K+M-1 hold XTY^T.  That is the lower part of the augmented symmetric matrix
// [[XTX + lambda I, XTY], [XTY^T, .]]; factoring its first K columns leaves L in rows 0 .. K-1 and Z^T = (L^-1 XTY)^T in
// rows K .. K+M-1, so the forward substitution falls out of the trailing updates (DESIGN.md, "Cross-validated ridge").
//   k_ridge_load          XTX + lambda I and XTY^T of every pair into the pass scratch; refused folds are marked
//   per panel j (RIDGE_NB columns):
//     k_ridge_potrf_diag  one CTA per pair factors the diagonal block in shared memory; the first pivot that is not
//                         > 0 sets info (1-based column) and retires the pair
//     k_ridge_trsm        L21 = A21 L11^-T for every row below the panel (the Z^T rows included); CTA per (pair, rows)
//     k_ridge_syrk        A22 -= L21 L21^T on the lower tiles of the trailing columns; CTA per (pair, tile), flattened
//   per panel j, last to first (back substitution L^T B = Z, in place in the Z^T rows):
//     k_ridge_bsolve_diag    one CTA per pair, one thread per response column
//     k_ridge_bsolve_update  Z_r -= L_jr^T B_j for the rows r above the panel; CTA per (pair, 64 rows)
//   k_ridge_press / k_ridge_press_accum / k_ridge_finish   PRESS over fixed 32-row chunks (the PLS chunk table), chunks
//                         of a fold added in chunk order; NaN for failed pairs and refused folds
//   k_ridge_coefs         B in the model dtype, when asked
// Retired and refused pairs return before they touch their matrix.  Every reduction has a fixed order that depends on
// the problem only, never on the grid, the window or the pass: identical calls give identical bits.
// All launch geometry and scratch sizes come from ridge_plan (also exported as cvmx_ridge_plan).
#pragma once
#include <algorithm>
#include "common.cuh"
#include "kernels_pls.cuh"
#include "../../include/cvmx.h"

namespace cvmx {

constexpr int RIDGE_NB = 64;             // panel width of the blocked factorisation
constexpr int RIDGE_NBP = RIDGE_NB + 1;  // shared-memory pitch (conflict-free column access)
constexpr int RIDGE_THREADS = 256;
constexpr int RIDGE_TR_ROWS = 128;       // k_ridge_trsm: rows per CTA, one thread per row
constexpr int RIDGE_BS_THREADS = 128;    // k_ridge_bsolve_diag: one thread per response column (M <= 128)
constexpr int RIDGE_PC = 64;             // k_ridge_press: (penalty, response) columns per CTA
constexpr int RIDGE_MAX_M = 128;
constexpr int RIDGE_MAX_L = 1024;
constexpr int64_t RIDGE_PASS_BUDGET = (int64_t)1 << 30;   // pair scratch + staged outputs of one pass
constexpr int64_t RIDGE_PART_BUDGET = (int64_t)256 << 20; // PRESS chunk partials of one launch
constexpr int64_t RIDGE_MAX_SCRATCH = (int64_t)32 << 30;  // a single pair and fold beyond this is refused
constexpr int64_t RIDGE_MAX_SMEM = 227 * 1024;
constexpr int64_t RIDGE_MAX_GRID_X = 2147483647, RIDGE_MAX_GRID_Y = 65535;

// Working state of one pass: pair p = (fold in window) * Lp + (penalty in pass).
struct RidgeState {
  int64_t K, M, Lp;
  double* A;        // [pairs][K + M][K]
  int32_t* state;   // [pairs]  0 active, > 0 failed pivot column (1-based), -1 refused fold
};

__device__ __forceinline__ double* ridge_mat(const RidgeState& s, int64_t pair) { return s.A + pair * (s.K + s.M) * s.K; }

// ---- launch plan (host only, no CUDA call) ---------------------------------------------------------------------
inline int64_t ridge_align(int64_t b) { return (b + 255) / 256 * 256; }
inline int64_t ridge_cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Lower tiles of the trailing update after a panel that ends at column j1: row tiles over [j1, K + M), column tiles
// over [j1, K), column tile <= row tile.  Rows of the first Cc row tiles form a triangle, the rest a rectangle.
struct SyrkTiles {
  int64_t R, Cc, tri, total;
};
inline SyrkTiles ridge_syrk_tiles(int64_t K, int64_t M, int64_t j1) {
  SyrkTiles t;
  t.R = ridge_cdiv(K + M - j1, RIDGE_NB);
  t.Cc = ridge_cdiv(K - j1, RIDGE_NB);
  t.tri = t.Cc * (t.Cc + 1) / 2;
  t.total = t.tri + (t.R - t.Cc) * t.Cc;
  return t;
}

inline size_t ridge_smem_potrf() { return sizeof(double) * RIDGE_NB * RIDGE_NBP; }
inline size_t ridge_smem_trsm() { return sizeof(double) * (RIDGE_NB + RIDGE_TR_ROWS) * RIDGE_NBP; }
inline size_t ridge_smem_syrk() { return sizeof(double) * 2 * RIDGE_NB * RIDGE_NBP; }
inline size_t ridge_smem_bsolve_diag(int64_t M) { return sizeof(double) * (RIDGE_NB + M) * RIDGE_NBP; }
inline size_t ridge_smem_bsolve_update(int64_t M) { return sizeof(double) * (RIDGE_NB + M) * RIDGE_NBP; }
inline size_t ridge_smem_press() {
  return sizeof(double) * ((size_t)PRESS_ROWS * (PRESS_KT + 1) + (size_t)RIDGE_PC * (PRESS_KT + 1) + (size_t)PRESS_ROWS * RIDGE_PC +
                           PRESS_ROWS) +
         sizeof(int64_t) * (PRESS_ROWS + RIDGE_PC);
}

// Fills plan[CVMX_RIDGE_PLAN_LEN] (include/cvmx.h).  Returns CVMX_OK when the shape runs within the device limits, else
// CVMX_ERR_INVALID with plan[CVMX_RIDGE_FEASIBLE] = 0 (the other entries then say what the shape would need).
inline int32_t ridge_plan(int64_t K, int64_t M, int64_t L, int64_t P, int32_t dtype, int32_t mem, int32_t want_B, int64_t* plan) {
  for (int i = 0; i < CVMX_RIDGE_PLAN_LEN; ++i) plan[i] = 0;
  if (K < 1 || K > (int64_t)1 << 20 || M < 1 || M > RIDGE_MAX_M || L < 1 || L > RIDGE_MAX_L || P < 0 || (dtype != CVMX_F32 && dtype != CVMX_F64) ||
      (mem != CVMX_HOST && mem != CVMX_DEVICE))
    return CVMX_ERR_INVALID;
  const int64_t sz = dtype == CVMX_F64 ? 8 : 4, n = K + M;
  const bool host = mem == CVMX_HOST, wB = want_B != 0;
  // bytes per pair: its matrix, state, PRESS accumulator, and (host outputs) its staged press / info / B
  const int64_t pair_bytes = n * K * 8 + 4 + M * 8 + (host ? M * sz + 4 + (wB ? K * M * sz : 0) : 0);
  // bytes per fold: run_folds' XTX / XTY, the weight accumulator, and (host outputs) staged sum_w / status
  const int64_t fold_mats = (K * K + K * M) * sz;
  const int64_t fold_bytes = fold_mats + 8 + (host ? sz + 4 : 0);
  // a window holds as many folds as fit the budget with ALL penalties; when not even one fold does, the window is one
  // fold and its penalties go in passes (so a pass is either all penalties of its folds or one fold: outputs of a pass
  // are always one contiguous range)
  const int64_t budget = RIDGE_PASS_BUDGET - 16 * 256;   // room for the alignment of the scratch arrays
  int64_t W = budget / (fold_bytes + L * pair_bytes);
  W = std::max<int64_t>(1, std::min<int64_t>(W, std::max<int64_t>(P, 1)));
  int64_t Lp = (budget - W * (fold_bytes - fold_mats)) / (W * pair_bytes);
  Lp = std::max<int64_t>(1, std::min<int64_t>(Lp, L));
  const int64_t pairs = W * Lp;
  int64_t o = 0;
  o += ridge_align(pairs * n * K * 8);                     plan[CVMX_RIDGE_END_A] = o;
  o += ridge_align(pairs * 4);                             plan[CVMX_RIDGE_END_STATE] = o;
  o += ridge_align(pairs * M * 8);                         plan[CVMX_RIDGE_END_ACC] = o;
  o += ridge_align(W * 8);                                 plan[CVMX_RIDGE_END_ACC_W] = o;
  o += host ? ridge_align(pairs * M * sz) : 0;             plan[CVMX_RIDGE_END_PRESS] = o;
  o += host ? ridge_align(pairs * 4) : 0;                  plan[CVMX_RIDGE_END_INFO] = o;
  o += host && wB ? ridge_align(pairs * K * M * sz) : 0;   plan[CVMX_RIDGE_END_B] = o;
  o += host ? ridge_align(W * sz) : 0;                     plan[CVMX_RIDGE_END_SUM_W] = o;
  o += host ? ridge_align(W * 4) : 0;                      plan[CVMX_RIDGE_END_STATUS] = o;
  plan[CVMX_RIDGE_SCRATCH_BYTES] = o;
  plan[CVMX_RIDGE_FOLDS_PER_WINDOW] = W;
  plan[CVMX_RIDGE_PENALTIES_PER_PASS] = Lp;
  plan[CVMX_RIDGE_WINDOW_BYTES] = W * fold_mats;
  const int64_t width = Lp * M;
  const int64_t G = std::max<int64_t>(1, std::min<int64_t>(RIDGE_PART_BUDGET / ((width + 1) * 8), RIDGE_MAX_GRID_X));
  plan[CVMX_RIDGE_CHUNKS_PER_LAUNCH] = G;
  plan[CVMX_RIDGE_PART_BYTES] = G * (width + 1) * 8;
  // grids (largest of every launch) and dynamic shared memory
  const int64_t nb0 = std::min<int64_t>(RIDGE_NB, K);
  const int64_t npan = ridge_cdiv(K, RIDGE_NB);
  int64_t* g = plan + CVMX_RIDGE_GRID;
  int64_t* sm = plan + CVMX_RIDGE_SMEM;
  g[2 * CVMX_RK_LOAD] = pairs;              g[2 * CVMX_RK_LOAD + 1] = std::min<int64_t>(256, ridge_cdiv(n * K, 4096));
  g[2 * CVMX_RK_POTRF] = pairs;             g[2 * CVMX_RK_POTRF + 1] = 1;
  g[2 * CVMX_RK_TRSM] = pairs;              g[2 * CVMX_RK_TRSM + 1] = ridge_cdiv(n - nb0, RIDGE_TR_ROWS);
  g[2 * CVMX_RK_SYRK] = K > nb0 ? pairs * ridge_syrk_tiles(K, M, nb0).total : 0;
  g[2 * CVMX_RK_SYRK + 1] = K > nb0 ? 1 : 0;
  g[2 * CVMX_RK_BSOLVE_DIAG] = pairs;       g[2 * CVMX_RK_BSOLVE_DIAG + 1] = 1;
  g[2 * CVMX_RK_BSOLVE_UPDATE] = npan > 1 ? pairs : 0;
  g[2 * CVMX_RK_BSOLVE_UPDATE + 1] = npan > 1 ? npan - 1 : 0;   // rows above the last panel, 64 per CTA
  g[2 * CVMX_RK_PRESS] = G;                 g[2 * CVMX_RK_PRESS + 1] = ridge_cdiv(width, RIDGE_PC);
  g[2 * CVMX_RK_PRESS_ACCUM] = W;           g[2 * CVMX_RK_PRESS_ACCUM + 1] = 1;
  g[2 * CVMX_RK_FINISH] = W;                g[2 * CVMX_RK_FINISH + 1] = 1;
  g[2 * CVMX_RK_COEFS] = wB ? pairs : 0;    g[2 * CVMX_RK_COEFS + 1] = wB ? std::min<int64_t>(RIDGE_MAX_GRID_Y, ridge_cdiv(K * M, RIDGE_THREADS)) : 0;
  sm[CVMX_RK_POTRF] = (int64_t)ridge_smem_potrf();
  sm[CVMX_RK_TRSM] = (int64_t)ridge_smem_trsm();
  sm[CVMX_RK_SYRK] = (int64_t)ridge_smem_syrk();
  sm[CVMX_RK_BSOLVE_DIAG] = (int64_t)ridge_smem_bsolve_diag(M);
  sm[CVMX_RK_BSOLVE_UPDATE] = (int64_t)ridge_smem_bsolve_update(M);
  sm[CVMX_RK_PRESS] = (int64_t)ridge_smem_press();
  bool ok = W * fold_mats + o <= RIDGE_MAX_SCRATCH && (Lp == L || W == 1);
  for (int k = 0; k < CVMX_RK_COUNT; ++k)
    ok = ok && g[2 * k] <= RIDGE_MAX_GRID_X && g[2 * k + 1] <= RIDGE_MAX_GRID_Y && sm[k] <= RIDGE_MAX_SMEM;
  plan[CVMX_RIDGE_FEASIBLE] = ok ? 1 : 0;
  return ok ? CVMX_OK : CVMX_ERR_INVALID;
}

// ---- kernels ------------------------------------------------------------------------------------------------------
// XTX_f + lambda_l I and XTY_f^T (model dtype) -> the pair's float64 matrix; state 0, or -1 for a fold the reference
// refuses (training_XTX_XTY raises: no non-zero training weight while any statistic is used, or nnz <= ddof with a std).
// grid (pairs, any): the y blocks stride over the (K + M) K entries.  alphas: device copy of the pass's penalties.
template <typename T>
__global__ void __launch_bounds__(RIDGE_THREADS) k_ridge_load(const T* __restrict__ xtx, const T* __restrict__ xty,
                                                              const FoldScalars* __restrict__ fs, uint32_t flags,
                                                              const double* __restrict__ alphas, RidgeState s) {
  const int64_t pair = blockIdx.x, f = pair / s.Lp, l = pair - f * s.Lp, K = s.K, M = s.M;
  const int32_t st = fs[f].status;   // bits CVMX_FOLD_NO_NONZERO_W = 1, CVMX_FOLD_NNZ_LE_DDOF = 2
  const bool bad = ((st & 1) && flags != 0u) || ((st & 2) && (flags & 12u) != 0u);
  if (blockIdx.y == 0 && threadIdx.x == 0) s.state[pair] = bad ? -1 : 0;
  if (bad) return;
  const double lam = alphas[l];
  const T* X = xtx + f * K * K;
  const T* Y = xty + f * K * M;
  double* A = ridge_mat(s, pair);
  const int64_t step = (int64_t)gridDim.y * RIDGE_THREADS;
  for (int64_t e = (int64_t)blockIdx.y * RIDGE_THREADS + threadIdx.x; e < K * K; e += step) {
    const int64_t r = e / K, c = e - r * K;
    double v = (double)X[e];
    if (r == c) v += lam;
    A[e] = v;
  }
  for (int64_t e = (int64_t)blockIdx.y * RIDGE_THREADS + threadIdx.x; e < M * K; e += step) {
    const int64_t m = e / K, k = e - m * K;
    A[K * K + e] = (double)Y[k * M + m];
  }
}

// Cholesky of the diagonal block [j, j + nbj) of every active pair, in shared memory, column by column.
__global__ void __launch_bounds__(RIDGE_THREADS) k_ridge_potrf_diag(RidgeState s, int64_t j, int nbj) {
  extern __shared__ double sm[];
  const int64_t pair = blockIdx.x, K = s.K;
  if (s.state[pair] != 0) return;
  double* A = ridge_mat(s, pair);
  const int tid = threadIdx.x;
  for (int e = tid; e < nbj * nbj; e += RIDGE_THREADS) {
    const int r = e / nbj, c = e - r * nbj;
    if (c <= r) sm[r * RIDGE_NBP + c] = A[(j + r) * K + j + c];
  }
  __syncthreads();
  for (int c = 0; c < nbj; ++c) {
    const double d = sm[c * RIDGE_NBP + c];
    if (!(d > 0.0)) {   // every thread read the same pivot: the whole block leaves
      if (tid == 0) s.state[pair] = (int32_t)(j + c + 1);
      return;
    }
    const double dd = sqrt(d);
    __syncthreads();   // the pivot has been read by every thread before it is overwritten
    for (int r = c + tid; r < nbj; r += RIDGE_THREADS) sm[r * RIDGE_NBP + c] = r == c ? dd : sm[r * RIDGE_NBP + c] / dd;
    __syncthreads();
    const int w = nbj - c - 1;
    for (int e = tid; e < w * w; e += RIDGE_THREADS) {
      const int r = c + 1 + e / w, k = c + 1 + e % w;
      if (k <= r) sm[r * RIDGE_NBP + k] = fma(-sm[r * RIDGE_NBP + c], sm[k * RIDGE_NBP + c], sm[r * RIDGE_NBP + k]);
    }
    __syncthreads();
  }
  for (int e = tid; e < nbj * nbj; e += RIDGE_THREADS) {
    const int r = e / nbj, c = e - r * nbj;
    if (c <= r) A[(j + r) * K + j + c] = sm[r * RIDGE_NBP + c];
  }
}

// Rows [r0, r0 + RIDGE_TR_ROWS) below the panel: x L11^T = a, one thread per row.  grid (pairs, row tiles).
__global__ void __launch_bounds__(RIDGE_TR_ROWS) k_ridge_trsm(RidgeState s, int64_t j, int nbj) {
  extern __shared__ double sm[];
  const int64_t pair = blockIdx.x, K = s.K, n = s.K + s.M;
  if (s.state[pair] != 0) return;
  const int64_t r0 = j + nbj + (int64_t)blockIdx.y * RIDGE_TR_ROWS;
  const int nr = (int)(n - r0 < RIDGE_TR_ROWS ? n - r0 : RIDGE_TR_ROWS);
  double* A = ridge_mat(s, pair);
  double* l11 = sm;                           // [RIDGE_NB][RIDGE_NBP]
  double* x = sm + RIDGE_NB * RIDGE_NBP;      // [RIDGE_TR_ROWS][RIDGE_NBP]
  const int tid = threadIdx.x;
  for (int e = tid; e < nbj * nbj; e += RIDGE_TR_ROWS) {
    const int r = e / nbj, c = e - r * nbj;
    l11[r * RIDGE_NBP + c] = c <= r ? A[(j + r) * K + j + c] : 0.0;
  }
  for (int e = tid; e < nr * nbj; e += RIDGE_TR_ROWS) {
    const int i = e / nbj, c = e - i * nbj;
    x[i * RIDGE_NBP + c] = A[(r0 + i) * K + j + c];
  }
  __syncthreads();
  if (tid < nr) {
    double* xi = x + tid * RIDGE_NBP;
    for (int c = 0; c < nbj; ++c) {
      double v = xi[c];
      for (int k = 0; k < c; ++k) v = fma(-xi[k], l11[c * RIDGE_NBP + k], v);
      xi[c] = v / l11[c * RIDGE_NBP + c];   // pivots tested > 0 by k_ridge_potrf_diag
    }
  }
  __syncthreads();
  for (int e = tid; e < nr * nbj; e += RIDGE_TR_ROWS) {
    const int i = e / nbj, c = e - i * nbj;
    A[(r0 + i) * K + j + c] = x[i * RIDGE_NBP + c];
  }
}

// Trailing update A[r][c] -= sum_k L[r][j + k] L[c][j + k] over the lower 64 x 64 tiles of rows [j1, K + M) and columns
// [j1, K), j1 = j + nbj; blockIdx.x = pair * tiles + tile.  Thread (ty, tx) owns rows ty + 16 a, columns tx + 16 b.
__global__ void __launch_bounds__(RIDGE_THREADS) k_ridge_syrk(RidgeState s, int64_t j, int nbj, SyrkTiles t) {
  extern __shared__ double sm[];
  const int64_t bid = blockIdx.x, pair = bid / t.total, tile = bid - pair * t.total;
  if (s.state[pair] != 0) return;
  const int64_t K = s.K, n = s.K + s.M, j1 = j + nbj;
  int64_t rt, ct;
  if (tile < t.tri) {
    rt = (int64_t)((sqrt(8.0 * (double)tile + 1.0) - 1.0) * 0.5);
    while ((rt + 1) * (rt + 2) / 2 <= tile) ++rt;
    while (rt * (rt + 1) / 2 > tile) --rt;
    ct = tile - rt * (rt + 1) / 2;
  } else {
    const int64_t u = tile - t.tri;
    rt = t.Cc + u / t.Cc;
    ct = u - (u / t.Cc) * t.Cc;
  }
  const int64_t ra = j1 + rt * RIDGE_NB, ca = j1 + ct * RIDGE_NB;
  double* A = ridge_mat(s, pair);
  double* As = sm;                         // [64][RIDGE_NBP] rows ra ..
  double* Bs = sm + RIDGE_NB * RIDGE_NBP;  // [64][RIDGE_NBP] rows ca ..
  const int tid = threadIdx.x;
  for (int e = tid; e < RIDGE_NB * RIDGE_NB; e += RIDGE_THREADS) {
    const int i = e / RIDGE_NB, k = e - i * RIDGE_NB;
    As[i * RIDGE_NBP + k] = (k < nbj && ra + i < n) ? A[(ra + i) * K + j + k] : 0.0;
    Bs[i * RIDGE_NBP + k] = (k < nbj && ca + i < K) ? A[(ca + i) * K + j + k] : 0.0;
  }
  __syncthreads();
  const int ty = tid >> 4, tx = tid & 15;
  double acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
#pragma unroll 4
  for (int k = 0; k < RIDGE_NB; ++k) {
    double av[4], bv[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) av[a] = As[(ty + 16 * a) * RIDGE_NBP + k];
#pragma unroll
    for (int b = 0; b < 4; ++b) bv[b] = Bs[(tx + 16 * b) * RIDGE_NBP + k];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) acc[a][b] = fma(av[a], bv[b], acc[a][b]);
  }
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int64_t r = ra + ty + 16 * a;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int64_t c = ca + tx + 16 * b;
      if (r < n && c < K && c <= r) A[r * K + c] -= acc[a][b];
    }
  }
}

// Back substitution, diagonal block: L11^T b = z for every response column (thread m), in place in the Z^T rows.
__global__ void __launch_bounds__(RIDGE_BS_THREADS) k_ridge_bsolve_diag(RidgeState s, int64_t j, int nbj) {
  extern __shared__ double sm[];
  const int64_t pair = blockIdx.x, K = s.K;
  if (s.state[pair] != 0) return;
  const int M = (int)s.M;
  double* A = ridge_mat(s, pair);
  double* l11 = sm;                        // [RIDGE_NB][RIDGE_NBP]
  double* z = sm + RIDGE_NB * RIDGE_NBP;   // [M][RIDGE_NBP]
  const int tid = threadIdx.x;
  for (int e = tid; e < nbj * nbj; e += RIDGE_BS_THREADS) {
    const int r = e / nbj, c = e - r * nbj;
    l11[r * RIDGE_NBP + c] = c <= r ? A[(j + r) * K + j + c] : 0.0;
  }
  for (int e = tid; e < M * nbj; e += RIDGE_BS_THREADS) {
    const int m = e / nbj, c = e - m * nbj;
    z[m * RIDGE_NBP + c] = A[(K + m) * K + j + c];
  }
  __syncthreads();
  if (tid < M) {
    double* zm = z + tid * RIDGE_NBP;
    for (int c = nbj - 1; c >= 0; --c) {
      double v = zm[c];
      for (int k = c + 1; k < nbj; ++k) v = fma(-l11[k * RIDGE_NBP + c], zm[k], v);
      zm[c] = v / l11[c * RIDGE_NBP + c];   // pivots tested > 0 by k_ridge_potrf_diag
    }
  }
  __syncthreads();
  for (int e = tid; e < M * nbj; e += RIDGE_BS_THREADS) {
    const int m = e / nbj, c = e - m * nbj;
    A[(K + m) * K + j + c] = z[m * RIDGE_NBP + c];
  }
}

// Back substitution, update of the rows above the panel: z[m][r] -= sum_k L[j + k][r] b[m][j + k] for r in
// [64 blockIdx.y, + 64) (all < j).  grid (pairs, j / 64).
__global__ void __launch_bounds__(RIDGE_THREADS) k_ridge_bsolve_update(RidgeState s, int64_t j, int nbj) {
  extern __shared__ double sm[];
  const int64_t pair = blockIdx.x, K = s.K;
  if (s.state[pair] != 0) return;
  const int M = (int)s.M;
  const int64_t r0 = (int64_t)blockIdx.y * RIDGE_NB;
  double* A = ridge_mat(s, pair);
  double* Ls = sm;                         // [RIDGE_NB][RIDGE_NBP]: Ls[k][i] = L[j + k][r0 + i]
  double* Bs = sm + RIDGE_NB * RIDGE_NBP;  // [M][RIDGE_NBP]
  const int tid = threadIdx.x;
  for (int e = tid; e < nbj * RIDGE_NB; e += RIDGE_THREADS) {
    const int k = e / RIDGE_NB, i = e - k * RIDGE_NB;
    Ls[k * RIDGE_NBP + i] = A[(j + k) * K + r0 + i];
  }
  for (int e = tid; e < M * nbj; e += RIDGE_THREADS) {
    const int m = e / nbj, c = e - m * nbj;
    Bs[m * RIDGE_NBP + c] = A[(K + m) * K + j + c];
  }
  __syncthreads();
  const int i = tid % RIDGE_NB, g = tid / RIDGE_NB;
  for (int m = g; m < M; m += RIDGE_THREADS / RIDGE_NB) {
    double acc = 0.0;
    for (int k = 0; k < nbj; ++k) acc = fma(Ls[k * RIDGE_NBP + i], Bs[m * RIDGE_NBP + k], acc);
    double* zp = A + (K + m) * K + r0 + i;
    *zp -= acc;
  }
}

// PRESS of one chunk of at most PRESS_ROWS validation rows of one fold for RIDGE_PC (penalty, response) columns
// col = l M + m.  chunks[c] = {first CSR position, rows, fold in window}.  Per row and column: x~ = (x - mu_X) /
// sigma_X (as the flags say), prediction (x~ . b) * sigma_Y + mu_Y; part[c][col] = sum over the chunk's rows (in row
// order) of w (y - prediction)^2, 0 for failed pairs and refused folds.  grid (chunks of the launch, column tiles).
// With pred set, the thread that forms a prediction also stores it (rounded once to T): CSR position q goes to row
// q - pred_pos of pred, element col; failed pairs and refused folds store NaN.
template <typename T>
struct RidgePressParams {
  const T* Z; const T* w; int64_t ld;
  const int64_t* idx;              // CSR indices (normalised to [0, N))
  const int64_t* chunks;           // [nchunks][3], first chunk of this launch
  const T* stats;                  // [Pn][2][ld]: mean row, std row
  uint32_t flags;
  RidgeState s;
  double* part;                    // [nchunks][Lp M]
  double* part_w;                  // [nchunks]
  T* pred;                         // [rows][pred_ld] device predictions from the pass's column 0, or nullptr: none stored
  int64_t pred_ld;                 // row pitch of pred in elements (>= Lp M)
  int64_t pred_pos;                // CSR position of pred's row 0
};

template <typename T>
__global__ void __launch_bounds__(RIDGE_THREADS) k_ridge_press(RidgePressParams<T> p) {
  extern __shared__ double sm[];
  const int64_t c = blockIdx.x;
  const int64_t pos = p.chunks[3 * c], n = p.chunks[3 * c + 1], f = p.chunks[3 * c + 2];
  const int64_t K = p.s.K, M = p.s.M, width = p.s.Lp * M, ld = p.ld;
  const int64_t col0 = (int64_t)blockIdx.y * RIDGE_PC;
  double* xs = sm;                                  // [PRESS_ROWS][PRESS_KT + 1]
  double* bs = xs + PRESS_ROWS * (PRESS_KT + 1);    // [RIDGE_PC][PRESS_KT + 1]
  double* ps = bs + RIDGE_PC * (PRESS_KT + 1);      // [PRESS_ROWS][RIDGE_PC]
  double* wv = ps + PRESS_ROWS * RIDGE_PC;          // [PRESS_ROWS]
  int64_t* rows = reinterpret_cast<int64_t*>(wv + PRESS_ROWS);
  int64_t* cbase = rows + PRESS_ROWS;               // [RIDGE_PC]: offset of the column's Z^T row, -1 when unused
  const int tid = threadIdx.x;
  const T* mean = p.stats + f * 2 * ld;
  const T* sdev = mean + ld;
  const bool cX = p.flags & 1u, cY = p.flags & 2u, sX = p.flags & 4u, sY = p.flags & 8u;
  if (tid < PRESS_ROWS) {
    const int64_t row = tid < n ? p.idx[pos + tid] : -1;
    rows[tid] = row;
    wv[tid] = row < 0 ? 0.0 : (p.w ? (double)p.w[row] : 1.0);
  }
  if (tid < RIDGE_PC) {
    const int64_t col = col0 + tid;
    int64_t base = -1;
    if (col < width) {
      const int64_t l = col / M, m = col - l * M, pair = f * p.s.Lp + l;
      if (p.s.state[pair] == 0) base = pair * (K + M) * K + (K + m) * K;
    }
    cbase[tid] = base;
  }
  __syncthreads();
  if (blockIdx.y == 0 && tid == 0) {
    double sw = 0.0;
    for (int i = 0; i < n; ++i) sw += wv[i];
    p.part_w[c] = sw;
  }
  bool any = false;
  for (int i = 0; i < RIDGE_PC; ++i) any |= cbase[i] >= 0;
  if (!any) {   // refused fold or only failed pairs: nothing below touches the statistics or the matrices
    if (tid < RIDGE_PC && col0 + tid < width) {
      p.part[c * width + col0 + tid] = 0.0;
      if (p.pred) {
        T* pc = p.pred + (pos - p.pred_pos) * p.pred_ld + col0 + tid;
        for (int i = 0; i < n; ++i) pc[i * p.pred_ld] = (T)__longlong_as_double(0x7ff8000000000000LL);
      }
    }
    return;
  }
  const int trow = tid / 8, tc = tid % 8;   // thread owns row trow, columns tc + 8 i
  double acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.0;
  for (int64_t k0 = 0; k0 < K; k0 += PRESS_KT) {
    __syncthreads();
    for (int e = tid; e < PRESS_ROWS * PRESS_KT; e += RIDGE_THREADS) {
      const int i = e / PRESS_KT, kk = e % PRESS_KT;
      const int64_t k = k0 + kk, row = rows[i];
      double x = 0.0;
      if (row >= 0 && k < K) {
        x = (double)p.Z[row * ld + k];
        if (cX) x -= (double)mean[k];
        if (sX) x /= (double)sdev[k];
      }
      xs[i * (PRESS_KT + 1) + kk] = x;
    }
    for (int e = tid; e < RIDGE_PC * PRESS_KT; e += RIDGE_THREADS) {
      const int jj = e / PRESS_KT, kk = e % PRESS_KT;
      const int64_t k = k0 + kk, base = cbase[jj];
      bs[jj * (PRESS_KT + 1) + kk] = (base >= 0 && k < K) ? p.s.A[base + k] : 0.0;
    }
    __syncthreads();
#pragma unroll 4
    for (int kk = 0; kk < PRESS_KT; ++kk) {
      const double xv = xs[trow * (PRESS_KT + 1) + kk];
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] = fma(xv, bs[(tc + 8 * i) * (PRESS_KT + 1) + kk], acc[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) ps[trow * RIDGE_PC + tc + 8 * i] = acc[i];
  __syncthreads();
  if (tid < RIDGE_PC && col0 + tid < width) {
    const int64_t col = col0 + tid, m = col % M;
    T* pc = p.pred ? p.pred + (pos - p.pred_pos) * p.pred_ld + col : nullptr;   // row 0 of the chunk, column col
    double ss = 0.0;
    if (cbase[tid] >= 0) {
      const double mu = cY ? (double)mean[K + m] : 0.0, sd = sY ? (double)sdev[K + m] : 1.0;
      for (int i = 0; i < n; ++i) {
        double pred = ps[i * RIDGE_PC + tid];
        if (sY) pred *= sd;
        if (cY) pred += mu;
        if (pc) pc[i * p.pred_ld] = (T)pred;
        const double res = (double)p.Z[rows[i] * ld + K + m] - pred;
        ss = fma(wv[i] * res, res, ss);
      }
    } else if (pc) {
      for (int i = 0; i < n; ++i) pc[i * p.pred_ld] = (T)__longlong_as_double(0x7ff8000000000000LL);
    }
    p.part[c * width + col] = ss;
  }
}

// acc[f] += the partials of the fold's chunks in [g0, g1), in chunk order (press_chunk_sum); launches over the chunk
// groups of a pass run in group order, so the sum is the same for any group size.  grid: folds [fa, fa + gridDim.x).
__global__ void __launch_bounds__(RIDGE_THREADS) k_ridge_press_accum(const double* __restrict__ part, const double* __restrict__ part_w,
                                                                     const int64_t* __restrict__ chunk_off, int64_t g0, int64_t g1,
                                                                     int64_t fa, int64_t width, double* __restrict__ acc,
                                                                     double* __restrict__ acc_w) {
  const int64_t f = fa + blockIdx.x;
  const int64_t c0 = chunk_off[f] > g0 ? chunk_off[f] : g0, c1 = chunk_off[f + 1] < g1 ? chunk_off[f + 1] : g1;
  if (c1 <= c0) return;
  for (int64_t e = threadIdx.x; e < width; e += RIDGE_THREADS)
    acc[f * width + e] = press_chunk_sum(part, width, c0 - g0, c1 - g0, e, acc[f * width + e]);
  if (threadIdx.x == 0) acc_w[f] = press_chunk_sum(part_w, 1, c0 - g0, c1 - g0, 0, acc_w[f]);
}

// press[f][l][m] (NaN for failed pairs and refused folds), info[f][l], sum_w[f] of the pass.  One block per fold.
template <typename T>
__global__ void __launch_bounds__(RIDGE_THREADS) k_ridge_finish(RidgeState s, const double* __restrict__ acc,
                                                                const double* __restrict__ acc_w, T* __restrict__ press,
                                                                int32_t* __restrict__ info, T* __restrict__ sum_w) {
  const int64_t f = blockIdx.x, Lp = s.Lp, M = s.M;
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  for (int64_t e = threadIdx.x; e < Lp * M; e += RIDGE_THREADS) {
    const int64_t l = e / M;
    press[f * Lp * M + e] = (T)(s.state[f * Lp + l] != 0 ? nan : acc[f * Lp * M + e]);
  }
  for (int64_t l = threadIdx.x; l < Lp; l += RIDGE_THREADS) {
    const int32_t st = s.state[f * Lp + l];
    info[f * Lp + l] = st > 0 ? st : 0;
  }
  if (threadIdx.x == 0) sum_w[f] = (T)acc_w[f];
}

// B[pair][k][m] in the model dtype (NaN for failed pairs and refused folds).  grid (pairs, any).
template <typename T>
__global__ void __launch_bounds__(RIDGE_THREADS) k_ridge_coefs(RidgeState s, T* __restrict__ B) {
  const int64_t pair = blockIdx.x, K = s.K, M = s.M;
  const bool bad = s.state[pair] != 0;
  const double* A = ridge_mat(s, pair);
  T* out = B + pair * K * M;
  for (int64_t e = (int64_t)blockIdx.y * RIDGE_THREADS + threadIdx.x; e < K * M; e += (int64_t)gridDim.y * RIDGE_THREADS) {
    const int64_t k = e / M, m = e - k * M;
    out[e] = bad ? (T)__longlong_as_double(0x7ff8000000000000LL) : (T)A[(K + m) * K + k];
  }
}

}  // namespace cvmx
