// Cross-validated PLS regression over a fold batch (sm_100a): Improved Kernel PLS, Algorithm 2 (Dayal & MacGregor,
// J. Chemometrics 11:73-85, 1997) on every fold's centred / scaled XTX and XTY, then the weighted PRESS of the fold's
// validation rows for every number of components.  All arithmetic is float64 for both model dtypes.
//
// One launch sequence per component covers every fold of a window (DESIGN.md, "Cross-validated PLS"):
//   k_pls_dir     one block per fold: direction w (M > 1: dominant eigenvector of XTY_a^T XTY_a), r-orthogonalisation
//   k_pls_xtx_r   u = XTX r for all folds, one warp per row (the bandwidth-bound step: A * P * K^2 * sizeof(T) bytes)
//   k_pls_update  one block per fold: tTt, p, q_a, rank-1 update of the working XTY
// then k_pls_press (validation rows gathered from the resident Z through the CSR, fixed 32-row chunks) and
// k_pls_press_reduce (chunks of a fold summed in chunk order), and k_pls_coefs when B is wanted.
// Every reduction has a fixed order that depends on the problem only, never on the grid: two calls give the same bits.
#pragma once
#include <vector>
#include "common.cuh"

namespace cvmx {

constexpr int PLS_THREADS = 256;
constexpr int PLS_WARPS = PLS_THREADS / 32;
constexpr int PLS_MAX_M = 128;    // bound of the in-kernel eigen step (S = XTY_a^T XTY_a lives in shared memory)
constexpr int PLS_CH = 32;        // XTY rows staged per step of the S accumulation
constexpr int PLS_SQUARINGS = 16; // eigen step: S^(2^16), then PLS_POWER power iterations with S itself
constexpr int PLS_POWER = 4;
constexpr int PLS_ROWS_PER_BLOCK = PLS_WARPS;   // k_pls_xtx_r: one warp per row of XTX
constexpr int PRESS_ROWS = 32;    // validation rows per PRESS chunk (a chunk never spans two folds)
constexpr int PRESS_AT = 64;      // components per tile of t = x~ R^T
constexpr int PRESS_KT = 32;      // columns per tile
// out-of-fold predictions for HOST outputs: the rows of one PRESS launch are staged in one device buffer of at most this
// many bytes (or one chunk's rows when a chunk alone is larger) and copied out before the buffer is reused
constexpr int64_t CV_PRED_STAGE_BYTES = (int64_t)256 << 20;

enum { PLS_ACTIVE = 0, PLS_STOPPED = 1, PLS_BAD = 2 };

// Working state of one window of folds (device, float64 unless noted).
struct PlsState {
  int64_t K, M, A;
  double* xty;     // [Pn][K][M]  XTY_a
  double* R;       // [Pn][A][K]
  double* Pm;      // [Pn][A][K]
  double* Q;       // [Pn][A][M]
  double* u;       // [Pn][K]     w in k_pls_dir, XTX r afterwards
  double* S;       // [Pn][2][M][M]  eigen step: S itself, and the product of a squaring
  double* y0;      // [Pn]        ||XTY_0||_F
  int32_t* nfit;   // [Pn]
  int32_t* state;  // [Pn]        PLS_*
};

inline size_t pls_state_doubles(int64_t K, int64_t M, int64_t A) {
  return (size_t)(K * M + 2 * A * K + A * M + K + 2 * M * M + 1);
}

// Sum over the block, the same bits in every thread; `red` holds PLS_WARPS doubles.
__device__ __forceinline__ double pls_block_sum(double v, double* red) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
  for (int i = 0; i < PLS_WARPS; ++i) s += red[i];
  return s;
}

__device__ __forceinline__ double warp_sum(double v) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// XTY_0 (model dtype) -> working copy, ||XTY_0||_F, and whether the fold is one the reference refuses
// (training_XTX_XTY raises: no non-zero training weight while any statistic is used, or nnz <= ddof with a std).
template <typename T>
__global__ void __launch_bounds__(PLS_THREADS) k_pls_init(const T* __restrict__ xty_in, const FoldScalars* __restrict__ fs,
                                                          uint32_t flags, PlsState s) {
  __shared__ double red[PLS_WARPS];
  const int64_t f = blockIdx.x, KM = s.K * s.M;
  const T* src = xty_in + f * KM;
  double* dst = s.xty + f * KM;
  double acc = 0.0;
  for (int64_t e = threadIdx.x; e < KM; e += PLS_THREADS) {
    const double v = (double)src[e];
    dst[e] = v;
    acc = fma(v, v, acc);
  }
  const double n2 = pls_block_sum(acc, red);
  if (threadIdx.x == 0) {
    const int32_t st = fs[f].status;   // bits CVMX_FOLD_NO_NONZERO_W = 1, CVMX_FOLD_NNZ_LE_DDOF = 2
    const bool bad = ((st & 1) && flags != 0u) || ((st & 2) && (flags & 12u) != 0u);
    s.y0[f] = sqrt(n2);
    s.nfit[f] = 0;
    s.state[f] = bad ? PLS_BAD : PLS_ACTIVE;
  }
}

// Direction of component a for one fold (block): v, the stop test, w = v / ||v||, r = w - sum_j (p_j^T w) r_j.
// Dynamic shared memory (M > 1): S [M][M] and a chunk of XTY rows [PLS_CH][M].
__global__ void __launch_bounds__(PLS_THREADS) k_pls_dir(PlsState s, int64_t a) {
  extern __shared__ double sm[];
  __shared__ double red[PLS_WARPS];
  __shared__ double q[PLS_MAX_M];
  __shared__ int s_pick;
  const int64_t f = blockIdx.x;
  if (s.state[f] != PLS_ACTIVE) return;
  const int64_t K = s.K;
  const int M = (int)s.M, MM = M * M;   // M <= PLS_MAX_M: 32-bit index arithmetic in the eigen step
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const double* X = s.xty + f * K * M;
  double* v = s.u + f * K;
  double* r = s.R + (f * s.A + a) * K;

  if (M == 1) {
    for (int64_t k = tid; k < K; k += PLS_THREADS) v[k] = X[k];
  } else {
    double* S = sm;
    double* ch = sm + MM;
    double* gS = s.S + f * 2 * MM;   // [0]: S, [1]: squaring product
    for (int e = tid; e < MM; e += PLS_THREADS) S[e] = 0.0;
    for (int64_t k0 = 0; k0 < K; k0 += PLS_CH) {
      const int64_t nr = K - k0 < PLS_CH ? K - k0 : PLS_CH;
      __syncthreads();
      for (int e = tid; e < PLS_CH * M; e += PLS_THREADS) ch[e] = e < nr * M ? X[k0 * M + e] : 0.0;
      __syncthreads();
      for (int e = tid; e < MM; e += PLS_THREADS) {
        const int i = e / M, j = e - i * M;
        if (j < i) continue;
        double acc = S[e];
        for (int rr = 0; rr < PLS_CH; ++rr) acc = fma(ch[rr * M + i], ch[rr * M + j], acc);
        S[e] = acc;
      }
    }
    __syncthreads();
    double acc = 0.0;
    for (int e = tid; e < MM; e += PLS_THREADS) {
      const int i = e / M, j = e - i * M;
      if (j < i) S[e] = S[j * M + i];
    }
    __syncthreads();
    for (int e = tid; e < MM; e += PLS_THREADS) { gS[e] = S[e]; acc = fma(S[e], S[e], acc); }
    const double sn = sqrt(pls_block_sum(acc, red));
    if (!(sn > 0.0)) {   // XTY_a = 0: v = 0, the stop test below holds
      if (tid == 0) s.state[f] = PLS_STOPPED;
      return;
    }
    for (int e = tid; e < MM; e += PLS_THREADS) S[e] /= sn;
    // repeated squaring T <- T T / ||T T||_F: T tends to q q^T at the rate (lambda_2 / lambda_1)^(2^n); T stays exactly
    // symmetric (the products of T[i][k] T[k][j] and T[j][k] T[k][i] are the same numbers in the same order)
    for (int it = 0; it < PLS_SQUARINGS; ++it) {
      __syncthreads();
      acc = 0.0;
      for (int e = tid; e < MM; e += PLS_THREADS) {
        const int i = e / M, j = e - i * M;
        double t = 0.0;
        for (int k = 0; k < M; ++k) t = fma(S[i * M + k], S[k * M + j], t);
        gS[MM + e] = t;
        acc = fma(t, t, acc);
      }
      const double tn = sqrt(pls_block_sum(acc, red));   // syncs: every read of S is done
      for (int e = tid; e < MM; e += PLS_THREADS) S[e] = gS[MM + e] / tn;
    }
    __syncthreads();
    if (tid == 0) {   // start vector: the row of T with the largest diagonal entry (first one on ties)
      int best = 0;
      for (int i = 1; i < M; ++i) if (S[i * M + i] > S[best * M + best]) best = i;
      s_pick = best;
    }
    __syncthreads();
    if (tid < M) q[tid] = S[s_pick * M + tid];
    __syncthreads();
    // power iterations with S itself restore full precision in the dominant direction
    for (int it = 0; it < PLS_POWER; ++it) {
      double y = 0.0;
      if (tid < M)
        for (int k = 0; k < M; ++k) y = fma(gS[tid * M + k], q[k], y);
      const double yn = sqrt(pls_block_sum(tid < M ? y * y : 0.0, red));
      if (tid < M) q[tid] = y / yn;
      __syncthreads();
    }
    // v = XTY_a q, one warp per row
    for (int64_t k = warp; k < K; k += PLS_WARPS) {
      double t = 0.0;
      for (int m = lane; m < M; m += 32) t = fma(X[k * M + m], q[m], t);
      t = warp_sum(t);
      if (lane == 0) v[k] = t;
    }
    __syncthreads();
  }
  double acc = 0.0;
  for (int64_t k = tid; k < K; k += PLS_THREADS) acc = fma(v[k], v[k], acc);
  const double nv = sqrt(pls_block_sum(acc, red));
  if (nv <= 64.0 * 2.220446049250313e-16 * s.y0[f]) {
    if (tid == 0) s.state[f] = PLS_STOPPED;
    return;
  }
  for (int64_t k = tid; k < K; k += PLS_THREADS) { const double w = v[k] / nv; v[k] = w; r[k] = w; }
  for (int64_t j = 0; j < a; ++j) {
    const double* pj = s.Pm + (f * s.A + j) * K;
    const double* rj = s.R + (f * s.A + j) * K;
    double c = 0.0;
    for (int64_t k = tid; k < K; k += PLS_THREADS) c = fma(pj[k], v[k], c);
    c = pls_block_sum(c, red);
    for (int64_t k = tid; k < K; k += PLS_THREADS) r[k] -= c * rj[k];
  }
}

// u = XTX r for every active fold; grid (folds, ceil(K / PLS_ROWS_PER_BLOCK)), one warp per row.
template <typename T>
__global__ void __launch_bounds__(PLS_THREADS) k_pls_xtx_r(const T* __restrict__ xtx, PlsState s, int64_t a) {
  const int64_t f = blockIdx.x, K = s.K;
  if (s.state[f] != PLS_ACTIVE) return;
  const int64_t i = (int64_t)blockIdx.y * PLS_ROWS_PER_BLOCK + (threadIdx.x >> 5);
  if (i >= K) return;
  const int lane = threadIdx.x & 31;
  const T* row = xtx + (f * K + i) * K;
  const double* r = s.R + (f * s.A + a) * K;
  double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0, acc3 = 0.0;
  int64_t k = lane;
  for (; k + 96 < K; k += 128) {
    acc0 = fma((double)row[k], __ldg(r + k), acc0);
    acc1 = fma((double)row[k + 32], __ldg(r + k + 32), acc1);
    acc2 = fma((double)row[k + 64], __ldg(r + k + 64), acc2);
    acc3 = fma((double)row[k + 96], __ldg(r + k + 96), acc3);
  }
  for (; k < K; k += 32) acc0 = fma((double)row[k], __ldg(r + k), acc0);
  const double t = warp_sum((acc0 + acc1) + (acc2 + acc3));
  if (lane == 0) s.u[f * K + i] = t;
}

// tTt = r^T u, p = u / tTt, q_a = XTY_a^T r / tTt, XTY_{a+1} = XTY_a - tTt p q_a^T.  One block per fold.
__global__ void __launch_bounds__(PLS_THREADS) k_pls_update(PlsState s, int64_t a) {
  __shared__ double red[PLS_WARPS];
  __shared__ double part[PLS_THREADS];
  __shared__ double qs[PLS_MAX_M];
  const int64_t f = blockIdx.x;
  if (s.state[f] != PLS_ACTIVE) return;
  const int64_t K = s.K, M = s.M;
  const int tid = threadIdx.x;
  const double* r = s.R + (f * s.A + a) * K;
  const double* u = s.u + f * K;
  double* X = s.xty + f * K * M;
  double acc = 0.0;
  for (int64_t k = tid; k < K; k += PLS_THREADS) acc = fma(r[k], u[k], acc);
  const double tTt = pls_block_sum(acc, red);
  if (!(tTt > 0.0)) {
    if (tid == 0) s.state[f] = PLS_STOPPED;
    return;
  }
  double* p = s.Pm + (f * s.A + a) * K;
  for (int64_t k = tid; k < K; k += PLS_THREADS) p[k] = u[k] / tTt;
  // q_a: thread (m, g) sums the rows k = g (mod G) of column m, the G partial sums are added in g order
  const int G = PLS_THREADS / (int)M;
  const int m = tid % (int)M, g = tid / (int)M;
  if (g < G) {
    double t = 0.0;
    for (int64_t k = g; k < K; k += G) t = fma(X[k * M + m], r[k], t);
    part[g * M + m] = t;
  }
  __syncthreads();
  if (tid < M) {
    double t = 0.0;
    for (int gg = 0; gg < G; ++gg) t += part[gg * M + tid];
    t /= tTt;
    qs[tid] = t;
    s.Q[(f * s.A + a) * M + tid] = t;
  }
  __syncthreads();
  for (int64_t e = tid; e < K * M; e += PLS_THREADS) {
    const int64_t k = e / M, mm = e - k * M;
    X[e] -= (tTt * p[k]) * qs[mm];   // p was written before the two syncs above
  }
  if (tid == 0) s.nfit[f] = (int32_t)(a + 1);
}

// B[f][a] = sum_{j <= min(a, nfit - 1)} r_j q_j^T (K x M, model dtype); NaN for refused folds.
// grid (folds, any): the y blocks stride over the K M entries.
template <typename T>
__global__ void __launch_bounds__(PLS_THREADS) k_pls_coefs(PlsState s, T* __restrict__ B) {
  const int64_t f = blockIdx.x, K = s.K, M = s.M, A = s.A;
  const bool bad = s.state[f] == PLS_BAD;
  const int64_t nf = s.nfit[f];
  for (int64_t e = (int64_t)blockIdx.y * PLS_THREADS + threadIdx.x; e < K * M; e += (int64_t)gridDim.y * PLS_THREADS) {
    const int64_t k = e / M, m = e - k * M;
    double acc = 0.0;
    T* out = B + f * A * K * M + e;
    for (int64_t j = 0; j < A; ++j) {
      if (j < nf) acc = fma(s.R[(f * A + j) * K + k], s.Q[(f * A + j) * M + m], acc);
      out[j * K * M] = bad ? (T)__longlong_as_double(0x7ff8000000000000LL) : (T)acc;
    }
  }
}

// PRESS of one chunk of at most PRESS_ROWS validation rows of one fold.  chunks[c] = {first CSR position, rows, fold}.
// Per row: x~ = (x - mu_X) / sigma_X (as the flags say), t = x~ R^T, y^(a) = sum_{j <= a} t_j q_j^T, prediction
// y^(a) * sigma_Y + mu_Y; part[c][a][m] = sum over the chunk's rows (in row order) of w (y - prediction)^2.
// With pred set, the thread that forms a prediction also stores it (rounded once to T): CSR position q goes to row
// q - pred_pos of pred, element a M + m; a refused fold's rows are NaN.
template <typename T>
struct PressParams {
  const T* Z; const T* w; int64_t ld;
  const int64_t* idx;              // CSR indices (normalised to [0, N))
  const int64_t* chunks;           // [nchunks][3]
  const T* stats;                  // [Pn][2][ld]: mean row, std row
  uint32_t flags;
  PlsState s;
  double* part;                    // [nchunks][A][M]
  double* part_w;                  // [nchunks]
  T* pred;                         // [rows][pred_ld] device predictions, or nullptr: none stored
  int64_t pred_ld;                 // row pitch of pred in elements (>= A M)
  int64_t pred_pos;                // CSR position of pred's row 0
};

inline size_t press_smem_bytes(int64_t M) {
  return sizeof(double) * ((size_t)PRESS_ROWS * (PRESS_KT + 1) + (size_t)PRESS_AT * (PRESS_KT + 1) +
                           (size_t)PRESS_ROWS * PRESS_AT + 2 * (size_t)PRESS_ROWS * M + PRESS_ROWS) +
         sizeof(int64_t) * PRESS_ROWS;
}

template <typename T>
__global__ void __launch_bounds__(PLS_THREADS) k_pls_press(PressParams<T> p) {
  extern __shared__ double sm[];
  const int64_t c = blockIdx.x;
  const int64_t pos = p.chunks[3 * c], n = p.chunks[3 * c + 1], f = p.chunks[3 * c + 2];
  const int64_t K = p.s.K, M = p.s.M, A = p.s.A, ld = p.ld;
  double* xs = sm;                                     // [PRESS_ROWS][PRESS_KT + 1]
  double* rs = xs + PRESS_ROWS * (PRESS_KT + 1);       // [PRESS_AT][PRESS_KT + 1]
  double* ts = rs + PRESS_AT * (PRESS_KT + 1);         // [PRESS_ROWS][PRESS_AT]
  double* ys = ts + PRESS_ROWS * PRESS_AT;             // [PRESS_ROWS][M]
  double* yh = ys + PRESS_ROWS * M;                    // [PRESS_ROWS][M]
  double* wv = yh + PRESS_ROWS * M;                    // [PRESS_ROWS]
  int64_t* rows = reinterpret_cast<int64_t*>(wv + PRESS_ROWS);
  const int tid = threadIdx.x;
  const T* mean = p.stats + f * 2 * ld;
  const T* sdev = mean + ld;
  const bool cX = p.flags & 1u, cY = p.flags & 2u, sX = p.flags & 4u, sY = p.flags & 8u;
  if (tid < PRESS_ROWS) {
    const int64_t row = tid < n ? p.idx[pos + tid] : -1;
    rows[tid] = row;
    wv[tid] = row < 0 ? 0.0 : (p.w ? (double)p.w[row] : 1.0);
  }
  __syncthreads();
  if (tid == 0) {
    double sw = 0.0;
    for (int i = 0; i < n; ++i) sw += wv[i];
    p.part_w[c] = sw;
  }
  const int state = p.s.state[f];
  double* out = p.part + c * A * M;
  if (state == PLS_BAD) {   // the reduce kernel writes NaN press; the statistics of such a fold are not used
    if (p.pred) {
      const int64_t AM = A * M;
      for (int64_t e = tid; e < n * AM; e += PLS_THREADS) {
        const int64_t i = e / AM;
        p.pred[(pos + i - p.pred_pos) * p.pred_ld + (e - i * AM)] = (T)__longlong_as_double(0x7ff8000000000000LL);
      }
    }
    return;
  }
  for (int64_t e = tid; e < PRESS_ROWS * M; e += PLS_THREADS) {
    const int64_t i = e / M, m = e - i * M;
    ys[e] = rows[i] < 0 ? 0.0 : (double)p.Z[rows[i] * ld + K + m];
    yh[e] = 0.0;
  }
  const int64_t nf = p.s.nfit[f];
  const double* R = p.s.R + f * A * K;
  const double* Q = p.s.Q + f * A * M;
  const int trow = tid / 8, tc = tid % 8;   // t tile: thread owns row trow, components tc + 8 i
  for (int64_t a0 = 0; a0 < A; a0 += PRESS_AT) {
    double acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.0;
    if (a0 < nf) {
      for (int64_t k0 = 0; k0 < K; k0 += PRESS_KT) {
        __syncthreads();
        for (int e = tid; e < PRESS_ROWS * PRESS_KT; e += PLS_THREADS) {
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
        for (int e = tid; e < PRESS_AT * PRESS_KT; e += PLS_THREADS) {
          const int j = e / PRESS_KT, kk = e % PRESS_KT;
          const int64_t k = k0 + kk, aa = a0 + j;
          rs[j * (PRESS_KT + 1) + kk] = (aa < nf && k < K) ? R[aa * K + k] : 0.0;
        }
        __syncthreads();
#pragma unroll 4
        for (int kk = 0; kk < PRESS_KT; ++kk) {
          const double xv = xs[trow * (PRESS_KT + 1) + kk];
#pragma unroll
          for (int i = 0; i < 8; ++i) acc[i] = fma(xv, rs[(tc + 8 * i) * (PRESS_KT + 1) + kk], acc[i]);
        }
      }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) ts[trow * PRESS_AT + tc + 8 * i] = acc[i];
    __syncthreads();
    if (tid < M) {
      const int64_t m = tid;
      const double mu = cY ? (double)mean[K + m] : 0.0, sd = sY ? (double)sdev[K + m] : 1.0;
      const int64_t a1 = A - a0 < PRESS_AT ? A - a0 : PRESS_AT;
      T* prow = p.pred ? p.pred + (pos - p.pred_pos) * p.pred_ld + m : nullptr;   // row 0 of the chunk, column m
      for (int64_t j = 0; j < a1; ++j) {
        const int64_t aa = a0 + j;
        const double qm = aa < nf ? Q[aa * M + m] : 0.0;
        double ss = 0.0;
        for (int i = 0; i < n; ++i) {
          double y = yh[i * M + m];
          if (aa < nf) y = fma(ts[i * PRESS_AT + j], qm, y);
          yh[i * M + m] = y;
          double pred = y;
          if (sY) pred *= sd;
          if (cY) pred += mu;
          if (prow) prow[i * p.pred_ld + aa * M] = (T)pred;
          const double res = ys[i * M + m] - pred;
          ss = fma(wv[i] * res, res, ss);
        }
        out[aa * M + m] = ss;
      }
    }
  }
}

// PRESS chunks of folds [c0, c1) of the CSR (host offsets `off`): at most PRESS_ROWS validation rows each, never
// spanning two folds.  tab = [nch][3] {first CSR position, rows, fold - c0}, then chunk_off [c1 - c0 + 1] (first chunk of
// every fold); returns nch.
inline int64_t press_chunk_table(const int64_t* off, int64_t c0, int64_t c1, std::vector<int64_t>& tab) {
  tab.clear();
  std::vector<int64_t> coff((size_t)(c1 - c0) + 1, 0);
  for (int64_t f = c0; f < c1; ++f) {
    for (int64_t p = off[f]; p < off[f + 1]; p += PRESS_ROWS) {
      tab.push_back(p);
      tab.push_back(off[f + 1] - p < PRESS_ROWS ? off[f + 1] - p : PRESS_ROWS);
      tab.push_back(f - c0);
    }
    coff[f - c0 + 1] = (int64_t)tab.size() / 3;
  }
  const int64_t nch = (int64_t)tab.size() / 3;
  tab.insert(tab.end(), coff.begin(), coff.end());
  return nch;
}

// t + part[c0][e] + part[c0 + 1][e] + ... + part[c1 - 1][e] (row pitch `width`), added in chunk order: the PRESS of a
// fold does not depend on how its chunks were spread over CTAs or launches.
__device__ __forceinline__ double press_chunk_sum(const double* __restrict__ part, int64_t width, int64_t c0, int64_t c1, int64_t e,
                                                  double t) {
  for (int64_t c = c0; c < c1; ++c) t += part[c * width + e];
  return t;
}

// press[f][a][m] = sum of the fold's chunk partials in chunk order (NaN for refused folds), sum_w_val[f] likewise.
// chunk_off: [Pn + 1] first chunk of every fold.  One block per fold.
template <typename T>
__global__ void __launch_bounds__(PLS_THREADS) k_pls_press_reduce(const double* __restrict__ part, const double* __restrict__ part_w,
                                                                  const int64_t* __restrict__ chunk_off, PlsState s,
                                                                  T* __restrict__ press, T* __restrict__ sum_w) {
  const int64_t f = blockIdx.x, AM = s.A * s.M;
  const int64_t c0 = chunk_off[f], c1 = chunk_off[f + 1];
  const bool bad = s.state[f] == PLS_BAD;
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  for (int64_t e = threadIdx.x; e < AM; e += PLS_THREADS) press[f * AM + e] = (T)(bad ? nan : press_chunk_sum(part, AM, c0, c1, e, 0.0));
  if (threadIdx.x == 0) sum_w[f] = (T)press_chunk_sum(part_w, 1, c0, c1, 0, 0.0);
}

}  // namespace cvmx
