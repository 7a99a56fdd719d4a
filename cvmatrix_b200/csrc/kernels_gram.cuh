// Weighted Gram kernel on the FP64 tensor cores (DMMA.8x8x4) with the fused fold epilogue.
//
//   G[i][j] = sum_{r in rows} rn(w_r * x_ri) * z_rj        i < K, j < K + M, z = [x | y]
//
// is the contraction behind XTX = WX.T @ X, XTY = WX.T @ Y (cvmatrix/cvmatrix.py:1215-1217) and
// behind the per-fold downdate X_val.T @ mat2_val (cvmatrix/cvmatrix.py:1001).  One CTA owns one
// 128 x 128 output tile of one (fold, row-split) unit; only tiles on or above the diagonal are
// computed and the XTX part is mirrored on store.  The epilogue applies, per element,
//   A = T - G ; A -= sw * (mean_i * mean_j) ; A /= (std_i * std_j)       (cvmatrix.py:1001-1009)
// with each operation individually rounded in the model dtype, exactly as numpy evaluates it.
#pragma once
#include "common.cuh"
#include "kernels_stats.cuh"

namespace cvmx {

constexpr int GB = 128;       // tile edge (output rows and columns per CTA)
constexpr int GBK = 16;       // data rows (reduction index) per pipeline stage
constexpr int GSTAGES = 4;    // ring depth of the row pipeline (6 stages measured: 1 % slower at cfg 2 / cfg 3)
constexpr int GTHREADS = 256; // 8 warps = 2 (rows) x 4 (cols), warp tile 64 x 32
constexpr int GACC = 64;      // accumulator doubles per thread
constexpr int GTILE_ELEMS = GB * GB;

constexpr int GPRODUCERS = 4;                       // producer warps (one warpgroup, one warp per SM sub-partition)
constexpr int GLAUNCH = GTHREADS + 32 * GPRODUCERS;  // k_gram launch size
// Register split (setmaxnreg works per warpgroup): the kernel starts at <= 168 registers / thread (3 warps per
// sub-partition); the producer warpgroup shrinks to 64 and the two compute warpgroups grow to 208.  The grown total
// must stay within what the CTA was launched with (12 warps * 32 * 168 = 64512 registers) or the second
// setmaxnreg.inc never completes: 8 * 32 * 208 + 4 * 32 * 64 = 61440.
constexpr int GREGS_PRODUCER = 64;
constexpr int GREGS_COMPUTE = 208;
static_assert(GTHREADS * GREGS_COMPUTE + 32 * GPRODUCERS * GREGS_PRODUCER <= (GTHREADS + 32 * GPRODUCERS) * 168,
              "setmaxnreg budget exceeds the registers the CTA owns");
// barrier among the GTHREADS compute threads only (the producer warp has left the kernel by then)
__device__ __forceinline__ void compute_barrier() { asm volatile("bar.sync 1, %0;\n" ::"n"(GTHREADS) : "memory"); }

template <typename T> struct GramCfg;
// PITCH: shared-memory row pitch of a staged data-row segment, chosen so that the MMA fragment
// loads (lane -> row l%4, column pair 2*(l/4)) hit distinct banks: f64 LDS.128 needs pitch/2 = 2 (mod 8)
// in 16-byte units -> pitch = 4 (mod 16) doubles; f32 LDS.64 needs pitch/2 = 4 (mod 16) in 8-byte units.
template <> struct GramCfg<double> { static constexpr int PITCH = 132; static constexpr int CPITCH = 130; typedef double2 vec2; };
template <> struct GramCfg<float>  { static constexpr int PITCH = 136; static constexpr int CPITCH = 130; typedef float2 vec2; };

struct GramUnit {          // one (fold, row-split): a contiguous range of the CSR index array
  int64_t row_begin;       // position in `indices` (or absolute row when indices == nullptr)
  int64_t row_end;
  int32_t fold;            // fold number relative to the batch
  int32_t split;           // 0 .. nsplit-1
  int32_t nsplit;          // 1: fused epilogue in k_gram; >1: partials + k_gram_reduce
  int32_t part_base;       // index of split 0 of this fold in the partial workspace
};

template <typename T>
struct EpiParams {
  int mode;                // 0: raw Gram (fit totals)   1: fold downdate + centering + scaling
  uint32_t flags;          // cX | cY<<1 | sX<<2 | sY<<3
  uint32_t want;           // CVMX_WANT_XTX | CVMX_WANT_XTY
  int64_t K, M, ld;
  const T* Ttot;           // K x ld totals [XtWX | XtWY]
  const T* stats;          // [P][2][ld] mean, std of the fold's training set
  const FoldScalars* fs;   // [P]
  T* out_xx; int64_t xx_pitch; int64_t xx_stride;   // fold f, row i, col j -> out_xx[f*stride + i*pitch + j]
  T* out_xy; int64_t xy_pitch; int64_t xy_stride;
};

template <typename T>
struct GramParams {
  const T* Z; const T* w; int64_t ld;
  const int64_t* indices;
  const GramUnit* units;
  const int2* tiles; int ntiles;
  double* partials;        // [n_partial_units][ntiles][GACC][GTHREADS]
  double* raw_out;         // k_gram_reduce: if set, store the summed fragments here ([fold][ntiles][GACC][GTHREADS])
                           // instead of running the epilogue (multi-GPU: all-reduced across ranks, then finished)
  int force_partials;      // k_gram: write partials even for single-unit folds
  EpiParams<T> epi;
  // k_gram_reduce, multi-GPU: the fold's raw Gram lives in npeers buffers of the same layout - this GPU's and its
  // peers', mapped over NVLink (symmetric memory) - and the owner sums them on the fly instead of an all-reduce
  const double* peers[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  int npeers = 0;
  // which kernel produced the accumulators, i.e. which (row, column) a thread's 64 values belong to
  //   0  k_gram<T>   (DMMA m8n8k4 fragments)      1  k_gram_tc   (float32 only: tensor-memory lanes, thread = output row)
  int fmap = 0;
  // Fused fold statistics (k_gram<T, true>; single-unit folds, XTX wanted): in every diagonal-tile CTA the four producer
  // warps - idle between their copies - also consume every stage and continue numpy's sequential column sums of the
  // tile's 128 columns over the staged rows (sum w z, sum (w z) z: the chains of k_moments_pipe without the extra pass
  // over the fold's rows), turn them into the fold's mean / std (finalize_column; mom.stats == epi.stats, the fold
  // scalars come from k_weight_mass before the launch) and signal stat_flags[fold]; every CTA of the fold waits for
  // stat_target arrivals after its main loop.  Column blocks past the last diagonal block (Y columns beyond round_up(K, 128))
  // are chained by the tile (0, bj) from its B operand.  Tiles are ordered chain-tiles-first inside a fold, and the CTAs a
  // CTA waits for have block indices below its own or at most ntiles - 1 above, i.e. they are resident or done.
  int fuse_stats = 0;
  MomentParams<T> mom;
  int* stat_flags = nullptr;
  int stat_target = 0;
};

template <typename T>
__host__ __device__ constexpr size_t gram_smem_bytes() {
  size_t pipe = sizeof(T) * ((size_t)2 * GSTAGES * GBK * GramCfg<T>::PITCH + (size_t)GSTAGES * GBK);
  size_t stage = sizeof(T) * (size_t)GB * GramCfg<T>::CPITCH + 2 * GB * sizeof(double);   // staged tile + reciprocal std rows
  size_t body = (pipe > stage ? pipe : stage);
  return (body + 15) / 16 * 16 + 2 * GSTAGES * sizeof(uint64_t);   // + full / empty mbarriers at the end
}

// Scaling step of the epilogue.  numpy divides every element by (s_i * s_j); here the reciprocals r = 1 / s are formed
// once per tile row / column (float64 for both model dtypes) and an element costs two multiplications,
//   A_ij = rn_T(A_ij * (r_i * r_j)),
// within ~3 ulp of the quotient - matrices owe the reference 1e-12 (1e-5), only the statistics owe it their bits.  The
// IEEE division it replaces is ~25 dependent FP64 instructions per element on the pipe the DMMAs saturate.
template <typename T>
__device__ __forceinline__ T gram_scale(T a, double ri, double rj) { return (T)__dmul_rn((double)a, __dmul_rn(ri, rj)); }

// rrow[r] (r < nrows: tile rows i0 + r, always X columns) and rcol[c] (c < GB: tile columns j0 + c, X or Y) for the
// calling thread group (t = thread index inside the group of nthr threads)
template <typename T>
__device__ __forceinline__ void gram_recip_rows(const EpiParams<T>& e, const T* __restrict__ sdev, int64_t i0, int64_t j0, int t, int nthr,
                                                int nrows, double* rrow, double* rcol) {
  const bool sX = e.flags & 4, sY = e.flags & 8;
  const int64_t K = e.K, C = e.K + e.M;
  for (int x = t; x < nrows + GB; x += nthr) {
    const bool row = x < nrows;
    const int64_t col = row ? i0 + x : j0 + (x - nrows);
    const bool on = col < C && (col < K ? sX : sY) && !(row && col >= K);
    const double r = on ? __ddiv_rn(1.0, (double)sdev[col]) : 1.0;
    if (row) rrow[x] = r; else rcol[x - nrows] = r;
  }
}

// Epilogue of one 128 x 128 tile.
//  pass 1  accumulator fragments -> shared tile sC (raw G, model dtype).  m-tile t covers tile rows
//          wm*64 + 16*(t/2) + 2*g + (t%2); n-tile u covers tile columns wn*32 + 16*(u/2) + 2*h + (u%2) with h the
//          B-fragment column; in the accumulator h = 2*q + e, so a lane owns 4 consecutive columns per (t, u/2).
//  pass 2  in place, one column pair per thread step:  A = T - G ; A -= sw*(m_i*m_j) ; A /= (s_i*s_j)
//          (each op individually rounded; cvmatrix/cvmatrix.py:1001-1009).  Diagonal tiles skip the lower half.
//  pass 3  coalesced stores: the tile itself (a diagonal tile takes its lower half from the upper half, so the
//          result is exactly symmetric) and, for off-diagonal tiles, the mirrored XTX block.
template <typename T, int U = 16>
__device__ __forceinline__ void gram_epilogue(double (&acc)[8][4][2], T* sC, const EpiParams<T>& e, int fold, int bi,
                                              int bj, int fmap = 0) {
  constexpr int CP = GramCfg<T>::CPITCH;
  typedef typename GramCfg<T>::vec2 vec2;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm = warp >> 2, wn = warp & 3, g = lane >> 2, q = lane & 3;
  const int64_t K = e.K, C = e.K + e.M, ld = e.ld;
  const bool diag = bi == bj;

  if (fmap == 1) {
    // accumulators read from tensor memory (k_gram_tc): thread = output row 32 (warp % 4) + lane, linear index
    // ((t * 4 + u) * 2 + e) = column - 64 (warp / 4)
    const int r = 32 * (warp & 3) + lane, cb = 64 * (warp >> 2);
#pragma unroll
    for (int t = 0; t < 8; ++t)
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        vec2 v;
        v.x = (T)acc[t][u][0]; v.y = (T)acc[t][u][1];
        *reinterpret_cast<vec2*>(sC + r * CP + cb + (t * 4 + u) * 2) = v;
      }
  } else {
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const int r = wm * 64 + 16 * (t >> 1) + 2 * g + (t & 1);
#pragma unroll
      for (int up = 0; up < 2; ++up) {
        const int cb = wn * 32 + up * 16 + 4 * q;
        vec2 lo, hi;
        lo.x = (T)acc[t][2 * up][0]; lo.y = (T)acc[t][2 * up + 1][0];
        hi.x = (T)acc[t][2 * up][1]; hi.y = (T)acc[t][2 * up + 1][1];
        *reinterpret_cast<vec2*>(sC + r * CP + cb) = lo;
        *reinterpret_cast<vec2*>(sC + r * CP + cb + 2) = hi;
      }
    }
  }
  // reciprocal standard deviations of the tile's rows and columns, behind the staged tile (gram_smem_bytes reserves them)
  double* rrow = reinterpret_cast<double*>(sC + (size_t)GB * CP);
  double* rcol = rrow + GB;
  if (e.mode == 1 && (e.flags & 12))
    gram_recip_rows<T>(e, e.stats + (size_t)fold * 2 * ld + ld, (int64_t)bi * GB, (int64_t)bj * GB, tid, GTHREADS, GB, rrow, rcol);
  compute_barrier();

  if (e.mode == 1) {
    const bool cX = e.flags & 1, cY = e.flags & 2, sX = e.flags & 4, sY = e.flags & 8;
    const T* __restrict__ mean = e.stats + (size_t)fold * 2 * ld;
    const T* __restrict__ Tt = e.Ttot;
    const T sw = (T)e.fs[fold].sw;
    // thread -> fixed column pair c, rows r0, r0 + 4, ...: the column statistics are loaded once, and the loads of
    // four rows (totals tile from L2, row mean / std) are issued together so their latency overlaps
    const int c = (tid & 63) * 2, r0 = tid >> 6;
    const int64_t j = (int64_t)bj * GB + c;
    if (j < C) {
      const vec2 mj = *reinterpret_cast<const vec2*>(mean + j);
      const T mjj[2] = {mj.x, mj.y};
      const double rjj[2] = {rcol[c], rcol[c + 1]};
      const bool isX[2] = {j < K, j + 1 < K};
      // U rows per batch: the accumulators are dead here, so 16 loads of the totals tile fly together (2 L2 round trips
      // per tile instead of 8; k_gram_tc has no setmaxnreg split and keeps 4)
#pragma unroll 1
      for (int it0 = 0; it0 < GB / 4; it0 += U) {
        vec2 tv[U];
        T mi[U];
        bool ok[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int r = r0 + 4 * (it0 + u);
          const int64_t i = (int64_t)bi * GB + r;
          ok[u] = i < K && !(diag && c + 1 < r);
          if (ok[u]) {
            tv[u] = __ldg(reinterpret_cast<const vec2*>(Tt + i * ld + j));
            mi[u] = __ldg(mean + i);
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (!ok[u]) continue;
          const int r = r0 + 4 * (it0 + u);
          vec2 gv = *reinterpret_cast<const vec2*>(sC + r * CP + c);
          T a[2] = {Rn<T>::sub(tv[u].x, gv.x), Rn<T>::sub(tv[u].y, gv.y)};
          const double ri_u = rrow[r];
#pragma unroll
          for (int x = 0; x < 2; ++x) {
            if (isX[x] ? cX : (cX || cY)) a[x] = Rn<T>::sub(a[x], Rn<T>::mul(sw, Rn<T>::mul(mi[u], mjj[x])));
            if (sX || sY) a[x] = gram_scale<T>(a[x], ri_u, rjj[x]);
          }
          gv.x = a[0]; gv.y = a[1];
          *reinterpret_cast<vec2*>(sC + r * CP + c) = gv;
        }
      }
    }
    compute_barrier();
  }

  const bool wxx = e.want & 1, wxy = e.want & 2;
  T* oxx = e.out_xx + (size_t)fold * e.xx_stride;
  T* oxy = e.out_xy + (size_t)fold * e.xy_stride;
  const bool vec_ok = wxx && (e.xx_pitch % 2 == 0) && (e.xx_stride % 2 == 0) &&
                      (reinterpret_cast<uintptr_t>(e.out_xx) % (2 * sizeof(T)) == 0);
#pragma unroll 1
  for (int idx = tid; idx < GTILE_ELEMS / 2; idx += GTHREADS) {
    const int r = idx >> 6, c = (idx & 63) * 2;
    const int64_t i = (int64_t)bi * GB + r, j = (int64_t)bj * GB + c;
    if (i >= K || j >= C) continue;
    vec2 v;
    if (diag && c + 1 < r) { v.x = sC[c * CP + r]; v.y = sC[(c + 1) * CP + r]; }
    else {
      v = *reinterpret_cast<const vec2*>(sC + r * CP + c);
      if (diag && c < r) v.x = sC[c * CP + r];
    }
    if (j + 1 < K && vec_ok) {
      *reinterpret_cast<vec2*>(oxx + i * e.xx_pitch + j) = v;
    } else {
      const T vv[2] = {v.x, v.y};
#pragma unroll
      for (int x = 0; x < 2; ++x) {
        const int64_t jj = j + x;
        if (jj < K) { if (wxx) oxx[i * e.xx_pitch + jj] = vv[x]; }
        else if (jj < C && wxy) oxy[i * e.xy_pitch + (jj - K)] = vv[x];
      }
    }
  }
  if (!diag && wxx) {  // mirrored XTX block: out[j][i] = out[i][j]; lanes run along i so the stores coalesce
#pragma unroll 1
    for (int idx = tid; idx < GTILE_ELEMS / 2; idx += GTHREADS) {
      const int c = (idx >> 7) * 2, r = idx & 127;
      const int64_t i = (int64_t)bi * GB + r, j = (int64_t)bj * GB + c;
      if (i >= K || j >= K) continue;
      const vec2 v = *reinterpret_cast<const vec2*>(sC + r * CP + c);
      oxx[j * e.xx_pitch + i] = v.x;
      if (j + 1 < K) oxx[(j + 1) * e.xx_pitch + i] = v.y;
    }
  }
}

// ---- fragment bands ------------------------------------------------------------------------------------------------
// A warp tile (64 x 32) is 4 x 2 bands of 16 x 16: band (tp, up) holds the fragments t in {2tp, 2tp + 1} x u in
// {2up, 2up + 1} (fragment rows interleave inside a band, so a band is the smallest unit a warp can skip).  A band mask
// selects bands by bit 2 * tp + up.
constexpr int GBANDS_ALL = 0xFF;
// Diagonal tiles need only the 36 of their 64 bands that lie on or above the diagonal; a band on the diagonal is
// computed in full.  They are spread 9 per SM sub-partition (warp % 4), the DMMA issue limit, against 16 in an
// off-diagonal tile: warp w computes the bands GDIAG_MASK[w] of its own warp tile, except that warp 4 (no band of its
// own) takes rows 0-47 of the tile of warp GDIAG_OWNER4 = 3 and warp 5 rows 0-15 of the tile of warp GDIAG_OWNER5 = 2.
// Without the two moves the sub-partitions would carry 3, 7, 11 and 15 bands.
constexpr int GDIAG_MASK[8] = {0x0B, 0xBF, 0xFC, 0xC0, 0x3F, 0x03, 0x0B, 0xBF};
constexpr int GDIAG_OWNER4 = 3, GDIAG_OWNER5 = 2;
constexpr bool gdiag_bands_ok() {
  int cover[8][8] = {}, smsp[4] = {};
  for (int w = 0; w < 8; ++w) {
    const int tile = w == 4 ? GDIAG_OWNER4 : w == 5 ? GDIAG_OWNER5 : w;
    for (int band = 0; band < 8; ++band)
      if ((GDIAG_MASK[w] >> band) & 1) {
        ++cover[(tile >> 2) * 4 + band / 2][(tile & 3) * 2 + band % 2];
        ++smsp[w % 4];
      }
  }
  for (int r = 0; r < 8; ++r)
    for (int c = 0; c < 8; ++c)
      if (cover[r][c] != (r <= c ? 1 : 0)) return false;
  for (int s = 0; s < 4; ++s)
    if (smsp[s] != 9) return false;
  return GDIAG_MASK[6] == GDIAG_MASK[0] && GDIAG_MASK[7] == GDIAG_MASK[1];   // k_gram runs warps 6, 7 on the code of 0, 1
}
static_assert(gdiag_bands_ok(), "diagonal-tile bands: each band on or above the diagonal exactly once, 9 per sub-partition");

template <int MASK> __device__ __forceinline__ constexpr bool gram_band(int t, int u) { return (MASK >> ((t >> 1) * 2 + (u >> 1))) & 1; }

// One compute warp's row loop: every pipeline stage of the unit, the fragments of the bands in MASK of the warp tile at
// tile rows r0 .. r0 + 63 and columns c0 .. c0 + 31.  A band outside MASK costs no DMMA, no fragment load and no rn(w*x).
template <typename T, int MASK>
__device__ __forceinline__ void gram_rows(double (&acc)[8][4][2], const T* sA, const T* sB, const T* sW, uint64_t* full,
                                          uint64_t* empty, int64_t nrows, int r0, int c0) {
  constexpr int PITCH = GramCfg<T>::PITCH;
  typedef typename GramCfg<T>::vec2 vec2;
  const int lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
#pragma unroll 1
  for (int64_t kt = 0; kt * GBK < nrows; ++kt) {
    const int slot = (int)(kt % GSTAGES);
    mbar_wait(full + slot, (unsigned)(kt / GSTAGES) & 1);
    const T* a_base = sA + (size_t)slot * GBK * PITCH + r0 + 2 * g;
    const T* b_base = sB + (size_t)slot * GBK * PITCH + c0 + 2 * g;
    const T* w_base = sW + slot * GBK;
    const int rows = (int)min((int64_t)GBK, nrows - kt * GBK);
    if (rows == GBK) {
#pragma unroll
      for (int kk = 0; kk < GBK / 4; ++kk) {
        const int k = kk * 4 + q;
        const T wv = w_base[k];
        double a[8], b[4];
#pragma unroll
        for (int tp = 0; tp < 4; ++tp) {
          if (!((MASK >> (2 * tp)) & 3)) continue;
          const vec2 v = *reinterpret_cast<const vec2*>(a_base + k * PITCH + tp * 16);
          a[2 * tp] = (double)Rn<T>::mul(v.x, wv);       // rn(w*x) in the model dtype == WX of the reference
          a[2 * tp + 1] = (double)Rn<T>::mul(v.y, wv);
        }
#pragma unroll
        for (int up = 0; up < 2; ++up) {
          if (!(MASK & (0x55 << up))) continue;
          const vec2 v = *reinterpret_cast<const vec2*>(b_base + k * PITCH + up * 16);
          b[2 * up] = (double)v.x;
          b[2 * up + 1] = (double)v.y;
        }
#pragma unroll
        for (int t = 0; t < 8; ++t)
#pragma unroll
          for (int u = 0; u < 4; ++u)
            if (gram_band<MASK>(t, u)) dmma884(acc[t][u][0], acc[t][u][1], a[t], b[u]);
      }
    } else {
      // tail stage: rows past the end of the unit were never copied - feed exact zeros instead
#pragma unroll 1
      for (int kk = 0; kk * 4 < rows; ++kk) {
        const int k = kk * 4 + q;
        const bool ok = k < rows;
        const T wv = ok ? w_base[k] : T(0);
        double a[8], b[4];
#pragma unroll
        for (int tp = 0; tp < 4; ++tp) {
          if (!((MASK >> (2 * tp)) & 3)) continue;
          vec2 v; v.x = T(0); v.y = T(0);
          if (ok) v = *reinterpret_cast<const vec2*>(a_base + k * PITCH + tp * 16);
          a[2 * tp] = ok ? (double)Rn<T>::mul(v.x, wv) : 0.0;
          a[2 * tp + 1] = ok ? (double)Rn<T>::mul(v.y, wv) : 0.0;
        }
#pragma unroll
        for (int up = 0; up < 2; ++up) {
          if (!(MASK & (0x55 << up))) continue;
          vec2 v; v.x = T(0); v.y = T(0);
          if (ok) v = *reinterpret_cast<const vec2*>(b_base + k * PITCH + up * 16);
          b[2 * up] = (double)v.x;
          b[2 * up + 1] = (double)v.y;
        }
#pragma unroll
        for (int t = 0; t < 8; ++t)
#pragma unroll
          for (int u = 0; u < 4; ++u)
            if (gram_band<MASK>(t, u)) dmma884(acc[t][u][0], acc[t][u][1], a[t], b[u]);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(empty + slot);
  }
}

// Bands MASK of the accumulators to / from a lane-interleaved [GACC][32] shared-memory slot (buf = slot + lane).  The
// sender zeroes what it sent; the receiver computed nothing in those bands and takes the values as they are.
template <int MASK>
__device__ __forceinline__ void gram_bands_out(double (&acc)[8][4][2], double* buf) {
#pragma unroll
  for (int t = 0; t < 8; ++t)
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (gram_band<MASK>(t, u)) {
        buf[((t * 4 + u) * 2 + 0) * 32] = acc[t][u][0];
        buf[((t * 4 + u) * 2 + 1) * 32] = acc[t][u][1];
        acc[t][u][0] = acc[t][u][1] = 0.0;
      }
}
template <int MASK>
__device__ __forceinline__ void gram_bands_in(double (&acc)[8][4][2], const double* buf) {
#pragma unroll
  for (int t = 0; t < 8; ++t)
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (gram_band<MASK>(t, u)) {
        acc[t][u][0] = buf[((t * 4 + u) * 2 + 0) * 32];
        acc[t][u][1] = buf[((t * 4 + u) * 2 + 1) * 32];
      }
}

// Main kernel, warp-specialised.  Data movement is done by the TMA engine: per pipeline stage, the 32 lanes of a
// producer warp (warps 8-11 take the stages round-robin) each issue one 1-KB bulk async copy (cp.async.bulk, SASS UBLKCP) of a gathered row segment
// - 16 rows x {A block, B block} - plus an 8-byte cp.async of the row weight, all completing on the stage's "full"
// mbarrier.  The eight compute warps wait on that barrier, run 4 x 32 DMMA.8x8x4 on the stage (a diagonal tile: only the
// fragment bands of GDIAG_MASK, at most 4 x 36 per sub-partition) and release it through
// the "empty" mbarrier; there is no block-wide barrier in the main loop and no compute warp ever issues a copy
// (with the producer role on a compute warp the ~1300 issue cycles per stage sat on the critical path: ncu showed
// 20 % of all samples in the full-barrier wait).  Row indices are fetched one stage ahead of their use.
template <typename T, bool FUSE = false>   // FUSE: fused fold statistics (GramParams::fuse_stats), a separate instantiation so that
__global__ void __launch_bounds__(GLAUNCH, 1) k_gram(const GramParams<T> p) {   // the plain kernel keeps its registers and schedule
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int PITCH = GramCfg<T>::PITCH;

  T* sA = reinterpret_cast<T*>(smem_raw);
  T* sB = sA + (size_t)GSTAGES * GBK * PITCH;
  T* sW = sB + (size_t)GSTAGES * GBK * PITCH;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + gram_smem_bytes<T>() - 2 * GSTAGES * sizeof(uint64_t));
  uint64_t* empty = full + GSTAGES;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm = warp >> 2, wn = warp & 3;
  const int tile = blockIdx.x % p.ntiles;
  const GramUnit unit = p.units[blockIdx.x / p.ntiles];
  const int2 tl = p.tiles[tile];
  const int bi = tl.x, bj = tl.y;
  const bool diag = bi == bj;
  const int64_t ld = p.ld;
  const int64_t nrows = unit.row_end - unit.row_begin;
  const int64_t nk = (nrows + GBK - 1) / GBK;

  const bool fused_epi = unit.nsplit == 1 && !p.force_partials;
  // fused fold statistics: in a diagonal tile the four producer warps - idle between their copies - also CONSUME every stage:
  // lane = one of the 128 columns of the tile's column block, continuing numpy's sequential column sums over the staged rows
  // (column blocks past the last diagonal block - Y columns when K + M > round_up(K, 128) - belong to the tile (0, bj))
  const bool chain_tile = FUSE && fused_epi && (diag || (bi == 0 && bj >= (int)((p.epi.K + GB - 1) / GB)));
  if (tid == 0) {
    for (int s = 0; s < GSTAGES; ++s) { mbar_init(full + s, 33); mbar_init(empty + s, GTHREADS / 32 + (chain_tile ? GPRODUCERS : 0)); }
    mbar_fence_init();
  }
  __syncthreads();

  // ---- producer state (warp 0): lane -> (row r = lane % 16, operand o = lane / 16) -------------------
  const int pr = lane & 15, po = lane >> 4;
  const int64_t pcol = (int64_t)(po ? bj : bi) * GB;
  const unsigned pbytes = (unsigned)(min((int64_t)GB, ld - pcol) * (int64_t)sizeof(T));   // > 0: tiles start inside ld
  auto fetch_row = [&](int64_t kt) -> int64_t {   // global row of this lane's row in stage kt, -1 if none
    const int64_t pos = unit.row_begin + kt * GBK + pr;
    if (kt >= nk || pos >= unit.row_end) return -1;
    return p.indices ? p.indices[pos] : pos;
  };
  auto issue = [&](int64_t kt, int64_t grow) {    // producer warp only, all lanes
    if (kt >= nk) return;
    const int slot = (int)(kt % GSTAGES);
    const unsigned round = (unsigned)(kt / GSTAGES);
    if (round > 0) mbar_wait(empty + slot, (round & 1) ^ 1);
    const int rows = (int)min((int64_t)GBK, nrows - kt * GBK);
    if (lane == 0) {
      const unsigned a_bytes = (unsigned)(min((int64_t)GB, ld - (int64_t)bi * GB) * (int64_t)sizeof(T));
      const unsigned b_bytes = diag ? 0u : (unsigned)(min((int64_t)GB, ld - (int64_t)bj * GB) * (int64_t)sizeof(T));
      mbar_arrive_expect_tx(full + slot, (unsigned)rows * (a_bytes + b_bytes));
    }
    if (grow >= 0 && !(diag && po)) {
      T* dst = (po ? sB : sA) + ((size_t)slot * GBK + pr) * PITCH;
      bulk_g2s(dst, p.Z + grow * ld + pcol, pbytes, full + slot);
    }
    if (po == 0) {
      if (sizeof(T) == 8) cp_async8(sW + slot * GBK + pr, p.w + (grow >= 0 ? grow : 0), grow >= 0 ? 8 : 0);
      else cp_async4(sW + slot * GBK + pr, p.w + (grow >= 0 ? grow : 0), grow >= 0 ? 4 : 0);
    }
    cp_async_mbar_arrive_noinc(full + slot);
  };

  if (warp >= GTHREADS / 32) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" ::"n"(GREGS_PRODUCER));
    const int pw = warp - GTHREADS / 32;
    if (FUSE && chain_tile) {
      // One loop over ALL stages: every producer warp adds stage j's rows to its 32 column chains, then the warp that owns
      // stage j + GSTAGES - 1 refills the slot stage j - 1 left.  Chains: t = rn(w z), s += t, q += rn(t z), each op rounded, rows in the fold's order (kernels_stats.cuh).
      static_assert(GSTAGES == GPRODUCERS, "one producer warp per ring slot");
      int64_t mine = pw;                                    // next stage this warp issues
      int64_t row = fetch_row(mine);
      if (mine < nk) { const int64_t nr = fetch_row(mine + GPRODUCERS); issue(mine, row); row = nr; mine += GPRODUCERS; }
      T cs = T(0), cq = T(0);
      const int col = pw * 32 + lane;
#pragma unroll 1
      for (int64_t j = 0; j < nk; ++j) {
        const int slot = (int)(j % GSTAGES);
        mbar_wait(full + slot, (unsigned)(j / GSTAGES) & 1);
        const T* zc = (diag ? sA : sB) + (size_t)slot * GBK * PITCH + col;
        const T* wb = sW + slot * GBK;
        const int rows = (int)min((int64_t)GBK, nrows - j * GBK);
#pragma unroll 4
        for (int k = 0; k < rows; ++k) {
          const T z = zc[k * PITCH];
          const T t = Rn<T>::mul(z, wb[k]);
          cs = Rn<T>::add(cs, t);
          cq = Rn<T>::add(cq, Rn<T>::mul(t, z));
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty + slot);
        // refill the slot stage j - 1 left (chain first: its arrival is what the other eleven warps may be waiting for,
        // the copy has three stages of slack)
        if (mine == j + GSTAGES - 1 && mine < nk) { const int64_t nr = fetch_row(mine + GPRODUCERS); issue(mine, row); row = nr; mine += GPRODUCERS; }
      }
      finalize_column<T>(p.mom, unit.fold, (int64_t)bj * GB + col, cs, cq);
      __threadfence();
      __syncwarp();
      if (lane == 0) atomicAdd(p.stat_flags + unit.fold, 1);
      cp_async_wait<0>();
      return;
    }
    int64_t kt = pw;
    int64_t row = fetch_row(kt);
#pragma unroll 1
    for (; kt < nk; kt += GPRODUCERS) {
      const int64_t next_row = fetch_row(kt + GPRODUCERS);
      issue(kt, row);
      row = next_row;
    }
    cp_async_wait<0>();
    return;
  }
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;\n" ::"n"(GREGS_COMPUTE));

  double acc[8][4][2];
#pragma unroll
  for (int t = 0; t < 8; ++t)
#pragma unroll
    for (int u = 0; u < 4; ++u) acc[t][u][0] = acc[t][u][1] = 0.0;

  if (!diag) {
    gram_rows<T, GBANDS_ALL>(acc, sA, sB, sW, full, empty, nrows, wm * 64, wn * 32);
  } else {
    // each warp's fixed band set, chosen once outside the row loop (the branch is warp-uniform)
    const int src = warp == 4 ? GDIAG_OWNER4 : warp == 5 ? GDIAG_OWNER5 : warp;   // whose warp tile this warp computes
    const int r0 = (src >> 2) * 64, c0 = (src & 3) * 32;
    switch (warp) {
      case 0: case 6: gram_rows<T, GDIAG_MASK[0]>(acc, sA, sA, sW, full, empty, nrows, r0, c0); break;
      case 1: case 7: gram_rows<T, GDIAG_MASK[1]>(acc, sA, sA, sW, full, empty, nrows, r0, c0); break;
      case 2: gram_rows<T, GDIAG_MASK[2]>(acc, sA, sA, sW, full, empty, nrows, r0, c0); break;
      case 3: gram_rows<T, GDIAG_MASK[3]>(acc, sA, sA, sW, full, empty, nrows, r0, c0); break;
      case 4: gram_rows<T, GDIAG_MASK[4]>(acc, sA, sA, sW, full, empty, nrows, r0, c0); break;
      default: gram_rows<T, GDIAG_MASK[5]>(acc, sA, sA, sW, full, empty, nrows, r0, c0); break;
    }
  }
  if (FUSE && fused_epi) {
    // The fold's mean / std rows are complete once the producer warps of every diagonal tile have signalled - and in a
    // diagonal tile this is also what says that ITS producer warps have read the last stages: the ring must not be reused
    // (band hand-over, epilogue tile) before that.
    if (tid == 0) {
      int seen;
      do {
        asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(seen) : "l"(p.stat_flags + unit.fold) : "memory");
        if (seen < p.stat_target) __nanosleep(64);
      } while (seen < p.stat_target);
    }
  }
  compute_barrier();   // every stage consumed by every compute warp: the ring can be reused as the epilogue tile

  if (diag) {
    // hand the bands computed for another warp's tile to their standard owners (warp 4 -> 3, warp 5 -> 2), so that every
    // thread holds its own warp tile in the standard fragment layout, with zeros in the bands below the diagonal
    double* hbuf = reinterpret_cast<double*>(smem_raw);          // [2][GACC][32]: slot 0 from warp 4, slot 1 from warp 5
    if (warp == 4) gram_bands_out<GDIAG_MASK[4]>(acc, hbuf + lane);
    if (warp == 5) gram_bands_out<GDIAG_MASK[5]>(acc, hbuf + (size_t)GACC * 32 + lane);
    compute_barrier();
    if (warp == GDIAG_OWNER4) gram_bands_in<GDIAG_MASK[4]>(acc, hbuf + lane);
    if (warp == GDIAG_OWNER5) gram_bands_in<GDIAG_MASK[5]>(acc, hbuf + (size_t)GACC * 32 + lane);
    compute_barrier();
  }

  if (fused_epi) {
    gram_epilogue<T>(acc, reinterpret_cast<T*>(smem_raw), p.epi, unit.fold, bi, bj);
  } else {
    double* dst = p.partials + ((size_t)(unit.part_base + unit.split) * p.ntiles + tile) * (size_t)(GACC * GTHREADS);
#pragma unroll
    for (int t = 0; t < 8; ++t)
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        dst[((t * 4 + u) * 2 + 0) * GTHREADS + tid] = acc[t][u][0];
        dst[((t * 4 + u) * 2 + 1) * GTHREADS + tid] = acc[t][u][1];
      }
  }
}

// Split folds: sum the row-split partials of one (fold, tile) in split order (deterministic) and run
// the same epilogue.  grid = (ntiles, folds-with-splits); fold_units[f] = index of the fold's first unit.
template <typename T>
__global__ void __launch_bounds__(GTHREADS, 1) k_gram_reduce(const GramParams<T> p, const int32_t* __restrict__ fold_units,
                                                             const int32_t* __restrict__ fold_list) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x;
  const int tile = blockIdx.x;
  const int fold = fold_list[blockIdx.y];
  const GramUnit unit = p.units[fold_units[fold]];
  const int2 tl = p.tiles[tile];
  double acc[8][4][2];
  const size_t tile_off = ((size_t)unit.part_base * p.ntiles + tile) * (size_t)(GACC * GTHREADS);
  const double* src = (p.npeers > 0 ? p.peers[0] : p.partials) + tile_off;
  const size_t split_stride = (size_t)p.ntiles * GACC * GTHREADS;
#pragma unroll
  for (int t = 0; t < 8; ++t)
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      acc[t][u][0] = src[((t * 4 + u) * 2 + 0) * GTHREADS + tid];
      acc[t][u][1] = src[((t * 4 + u) * 2 + 1) * GTHREADS + tid];
    }
  if (p.npeers > 0) {
    // peer order is fixed (deterministic); per fragment pair the loads of all peers are issued together, so the
    // NVLink round trips overlap instead of queueing peer after peer
#pragma unroll
    for (int t = 0; t < 8; ++t)
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        double v0[7], v1[7];
#pragma unroll
        for (int q = 1; q < 8; ++q) {
          const bool on = q < p.npeers;
          v0[q - 1] = on ? (p.peers[q] + tile_off)[((t * 4 + u) * 2 + 0) * GTHREADS + tid] : 0.0;
          v1[q - 1] = on ? (p.peers[q] + tile_off)[((t * 4 + u) * 2 + 1) * GTHREADS + tid] : 0.0;
        }
#pragma unroll
        for (int q = 1; q < 8; ++q) { acc[t][u][0] += v0[q - 1]; acc[t][u][1] += v1[q - 1]; }
      }
  } else {
    for (int s = 1; s < unit.nsplit; ++s) {
      const double* ps = src + s * split_stride;
#pragma unroll
      for (int t = 0; t < 8; ++t)
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          acc[t][u][0] += ps[((t * 4 + u) * 2 + 0) * GTHREADS + tid];
          acc[t][u][1] += ps[((t * 4 + u) * 2 + 1) * GTHREADS + tid];
        }
    }
  }
  if (p.raw_out) {
    double* dst = p.raw_out + ((size_t)unit.fold * p.ntiles + tile) * (size_t)(GACC * GTHREADS);
#pragma unroll
    for (int t = 0; t < 8; ++t)
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        dst[((t * 4 + u) * 2 + 0) * GTHREADS + tid] = acc[t][u][0];
        dst[((t * 4 + u) * 2 + 1) * GTHREADS + tid] = acc[t][u][1];
      }
    return;
  }
  gram_epilogue<T>(acc, reinterpret_cast<T*>(smem_raw), p.epi, unit.fold, tl.x, tl.y, p.fmap);
}

// Row-split partials of (fold, tile) summed in split order into raw fragment buffers, element-parallel: the sharded
// (multi-GPU) Gram phase has only folds x tiles reduce CTAs, too few to pull the partials at HBM rate.
//   out[fold][tile][e] = sum_s partials[part_base(fold) + s][tile][e],  e < GACC * GTHREADS
__global__ void __launch_bounds__(256) k_partial_sum(const double* __restrict__ partials, const GramUnit* __restrict__ units,
                                                     const int32_t* __restrict__ fold_units, int ntiles, double* __restrict__ out) {
  const int fold = blockIdx.z, tile = blockIdx.y;
  const GramUnit unit = units[fold_units[fold]];
  const size_t tile_elems = (size_t)GACC * GTHREADS, split_stride = (size_t)ntiles * tile_elems;
  const size_t e = ((size_t)blockIdx.x * 256 + threadIdx.x) * 2;
  const double* src = partials + ((size_t)unit.part_base * ntiles + tile) * tile_elems + e;
  double2 acc = *reinterpret_cast<const double2*>(src);
  int s = 1;
  for (; s + 4 <= unit.nsplit; s += 4) {
    double2 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = *reinterpret_cast<const double2*>(src + (size_t)(s + u) * split_stride);
#pragma unroll
    for (int u = 0; u < 4; ++u) { acc.x += v[u].x; acc.y += v[u].y; }
  }
  for (; s < unit.nsplit; ++s) {
    const double2 v = *reinterpret_cast<const double2*>(src + (size_t)s * split_stride);
    acc.x += v.x; acc.y += v.y;
  }
  *reinterpret_cast<double2*>(out + ((size_t)unit.fold * ntiles + tile) * tile_elems + e) = acc;
}

// Statistics rows of a column-sharded evaluation: every rank holds its own column groups (zeros elsewhere) behind its
// raw Grams in the symmetric buffer; out[i] = sum over peers, read over NVLink (replaces the second all-reduce).
struct PeerList { const double* p[8]; };   // by value in the kernel parameters: no pointer table to upload
template <typename T>
__global__ void k_peer_sum_rows(const PeerList peers, int npeers, int64_t offset, int64_t n, T* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double v[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) v[q] = q < npeers ? peers.p[q][offset + i] : 0.0;   // all peer loads in flight together
  double r = 0.0;
#pragma unroll
  for (int q = 0; q < 8; ++q) r += v[q];
  out[i] = (T)r;
}

// Raw Grams of the folds a rank owns, summed over the peers' buffers (this rank's own included; mapped over NVLink):
//   out[e] = sum_q peers[q][offset + e],  e < n  (n even; peer order fixed -> deterministic)
// Element-parallel, all peer loads of a thread in flight together: the reduction runs at NVLink bandwidth instead of
// the round-trip latency that the per-tile epilogue CTAs (10 per fold) paid 32 times in a row when they summed the peers
// themselves.  The epilogue then reads one local buffer.
__global__ void __launch_bounds__(256) k_peer_sum_frags(const PeerList peers, int npeers, int64_t offset, int64_t n, double* __restrict__ out) {
  const int64_t e = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 2;
  if (e >= n) return;
  double2 v[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) v[q] = q < npeers ? *reinterpret_cast<const double2*>(peers.p[q] + offset + e) : make_double2(0.0, 0.0);
  double2 r = v[0];
#pragma unroll
  for (int q = 1; q < 8; ++q) { r.x += v[q].x; r.y += v[q].y; }
  *reinterpret_cast<double2*>(out + e) = r;
}

// CSR index normalisation: numpy wrap-around for negative indices, error flag for out-of-range ones.
__global__ void k_normalize_indices(int64_t* __restrict__ idx, int64_t n, int64_t N, int32_t* __restrict__ err) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int64_t v = idx[i];
  if (v < 0) v += N;
  if (v < 0 || v >= N) { *err = 1; v = 0; }
  idx[i] = v;
}

// Dense staged rows (rows x cols, contiguous) -> columns [col0, col0 + cols) of the padded device matrix.
template <typename T>
__global__ void k_repack(const T* __restrict__ src, int64_t rows, int64_t cols, T* __restrict__ dst, int64_t ld) {
  const int64_t total = rows * cols;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / cols, c = e - r * cols;
    dst[r * ld + c] = src[e];
  }
}

// Zero the pad columns [c0, ld) of every row (one thread per pad element).
template <typename T>
__global__ void k_zero_pad(T* __restrict__ Z, int64_t rows, int64_t ld, int64_t c0) {
  const int64_t w = ld - c0;
  const int64_t total = rows * w;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / w, c = e - r * w;
    Z[r * ld + c0 + c] = T(0);
  }
}

template <typename T>
__global__ void k_fill(T* __restrict__ p, int64_t n, T v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// ------------------------------------------------------------------------------------------------------
// Small folds (leave-one-out, leave-few-out): the downdate is a rank-n_val update with n_val <= SMALL_MAX_ROWS,
// so the tensor cores have nothing to do and the fold is bound by writing its K x (K+M) result (2.04 MB at
// K = 500).  Pure streaming kernel, no shared memory, no barriers: a thread owns output row i and four
// consecutive columns j..j+3, keeps those four totals in registers and loops over SMALL_FOLDS consecutive
// folds; per fold it reads the fold's row(s) and statistics (L1 / L2 resident), forms
//   G_ij = sum_r rn(w_r x_ar) x_br   with (a, b) = (min(i,j), max(i,j)) for the XTX part
// (first product rounded, then FMAs: bit-identical to numpy for n_val = 1, and exactly symmetric by
// construction), applies the individually rounded epilogue of gram_epilogue and stores 32 contiguous bytes:
// a warp writes 1 KB of one output row per store pair.
// ------------------------------------------------------------------------------------------------------
constexpr int SMALL_MAX_ROWS = 16;
constexpr int SMALL_FOLDS = 32;   // folds streamed per thread
constexpr int STHREADS = 256;     // 2 output rows x 128 column quads per CTA

template <typename T>
struct SmallParams {
  const T* Z; const T* w; int64_t ld;
  const int64_t* offsets; const int64_t* indices; int64_t fold0;   // CSR; folds fold0 .. fold0 + nfolds - 1
  int64_t nfolds;
  int quads;                                                        // column quads per output row: ceil((K+M)/4)
  int rows_per_cta;                                                 // STHREADS / quads_padded
  EpiParams<T> epi;
};

template <typename T>
__global__ void __launch_bounds__(STHREADS, 3) k_small_folds(const SmallParams<T> p) {
  const EpiParams<T>& e = p.epi;
  typedef typename GramCfg<T>::vec2 vec2;
  const int64_t K = e.K, C = e.K + e.M, ld = p.ld;
  const int qpad = STHREADS / p.rows_per_cta;
  const int64_t i = (int64_t)blockIdx.x * p.rows_per_cta + threadIdx.x / qpad;
  const int64_t j = (int64_t)(threadIdx.x % qpad) * 4;
  const int64_t fbeg = (int64_t)blockIdx.y * SMALL_FOLDS;
  const int64_t fend = min(p.nfolds, fbeg + SMALL_FOLDS);
  if (i >= K || j >= C) return;
  const bool cX = e.flags & 1, cY = e.flags & 2, sX = e.flags & 4, sY = e.flags & 8;
  const bool wxx = e.want & 1, wxy = e.want & 2;
  const bool vec_ok = (e.xx_pitch % 2 == 0) && (e.xx_stride % 2 == 0) && (reinterpret_cast<uintptr_t>(e.out_xx) % (2 * sizeof(T)) == 0);
  if (!((wxx && j < K) || (wxy && j + 3 >= K))) return;

  T tt[4];
#pragma unroll
  for (int b = 0; b < 4; ++b) tt[b] = __ldg(e.Ttot + i * ld + j + b);   // j + 3 < ld (ld % 32 == 0)

  for (int64_t f = fbeg; f < fend; ++f) {
    const int64_t beg = p.offsets[p.fold0 + f];
    const int n = (int)(p.offsets[p.fold0 + f + 1] - beg);
    const T* mean = e.stats + (size_t)f * 2 * ld;
    const T* sdev = mean + ld;
    const T mi = __ldg(mean + i), si = __ldg(sdev + i);
    T mj[4], sj[4];
#pragma unroll
    for (int b = 0; b < 4; ++b) { mj[b] = __ldg(mean + j + b); sj[b] = __ldg(sdev + j + b); }
    const T sw = (T)e.fs[f].sw;
    T g[4] = {T(0), T(0), T(0), T(0)};
    for (int r = 0; r < n; ++r) {
      const int64_t row = p.indices[beg + r];
      const T wr = __ldg(p.w + row);
      const T* zr = p.Z + row * ld;
      const T xi = __ldg(zr + i);
      const T wxi = Rn<T>::mul(xi, wr);
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const T zj = __ldg(zr + j + b);
        // XTX below the diagonal takes the mirrored product so that out[i][j] == out[j][i] bit for bit
        const bool swap = (j + b < K) && (j + b < i);
        const T a = swap ? Rn<T>::mul(zj, wr) : wxi;
        const T c = swap ? xi : zj;
        g[b] = (r == 0) ? Rn<T>::mul(a, c) : fma(a, c, g[b]);
      }
    }
    T v[4];
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      T a = Rn<T>::sub(tt[b], g[b]);
      if (j + b < K) {
        if (cX) a = Rn<T>::sub(a, Rn<T>::mul(sw, Rn<T>::mul(mi, mj[b])));
        if (sX) a = Rn<T>::div(a, Rn<T>::mul(si, sj[b]));
      } else {
        if (cX || cY) a = Rn<T>::sub(a, Rn<T>::mul(sw, Rn<T>::mul(mi, mj[b])));
        if (sX && sY) a = Rn<T>::div(a, Rn<T>::mul(si, sj[b]));
        else if (sX) a = Rn<T>::div(a, si);
        else if (sY) a = Rn<T>::div(a, sj[b]);
      }
      v[b] = a;
    }
    T* oxx = e.out_xx + (size_t)f * e.xx_stride + i * e.xx_pitch;
    T* oxy = e.out_xy + (size_t)f * e.xy_stride + i * e.xy_pitch;
    if (j + 3 < K && vec_ok) {
      if (wxx) {
        vec2 lo, hi;
        lo.x = v[0]; lo.y = v[1]; hi.x = v[2]; hi.y = v[3];
        *reinterpret_cast<vec2*>(oxx + j) = lo;
        *reinterpret_cast<vec2*>(oxx + j + 2) = hi;
      }
    } else {
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int64_t jj = j + b;
        if (jj < K) { if (wxx) oxx[jj] = v[b]; }
        else if (jj < C && wxy) oxy[jj - K] = v[b];
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// Leave-one-out specialisation of the streaming kernel: every fold of the launch has exactly one row
// (fold f of the launch uses CSR position pos0 + f) and the preprocessing flags are compile-time constants, so
// the per-element instruction count drops from ~97 (ncu, generic kernel) to ~40.  Same thread layout and the
// same arithmetic (bit-identical results) as k_small_folds.
//   FLAGS = cX | cY << 1 | sX << 2 | sY << 3
// ------------------------------------------------------------------------------------------------------
template <typename T, int FLAGS>
__global__ void __launch_bounds__(STHREADS, 3) k_loo_folds(const SmallParams<T> p, int64_t pos0) {
  const EpiParams<T>& e = p.epi;
  typedef typename GramCfg<T>::vec2 vec2;
  constexpr bool cX = FLAGS & 1, cY = FLAGS & 2, sX = FLAGS & 4, sY = FLAGS & 8;
  const int64_t K = e.K, C = e.K + e.M, ld = p.ld;
  const int qpad = STHREADS / p.rows_per_cta;
  const int64_t i = (int64_t)blockIdx.x * p.rows_per_cta + threadIdx.x / qpad;
  const int64_t j = (int64_t)(threadIdx.x % qpad) * 4;
  const int64_t fbeg = (int64_t)blockIdx.y * SMALL_FOLDS;
  const int nf = (int)(min(p.nfolds, fbeg + SMALL_FOLDS) - fbeg);
  if (i >= K || j >= C) return;
  const bool wxx = e.want & 1, wxy = e.want & 2;
  if (!((wxx && j < K) || (wxy && j + 3 >= K))) return;
  const bool vec_ok = (e.xx_pitch % 2 == 0) && (e.xx_stride % 2 == 0) && (reinterpret_cast<uintptr_t>(e.out_xx) % (2 * sizeof(T)) == 0);
  const bool fast_store = vec_ok && wxx && j + 3 < K;

  T tt[4];
  bool isx[4], swp[4];
#pragma unroll
  for (int b = 0; b < 4; ++b) {
    tt[b] = __ldg(e.Ttot + i * ld + j + b);
    isx[b] = j + b < K;
    swp[b] = isx[b] && (j + b < i);   // XTX below the diagonal: mirrored product -> exactly symmetric output
  }
  const int64_t* __restrict__ rows = p.indices + pos0 + fbeg;
  const T* __restrict__ stat = e.stats + (size_t)fbeg * 2 * ld;
  const FoldScalars* __restrict__ fs = e.fs + fbeg;
  T* oxx = e.out_xx + (size_t)fbeg * e.xx_stride + i * e.xx_pitch + j;
  T* oxy = e.out_xy + (size_t)fbeg * e.xy_stride + i * e.xy_pitch;

#pragma unroll 1
  for (int f = 0; f < nf; ++f) {
    const int64_t row = __ldg(rows + f);
    const T* __restrict__ zr = p.Z + row * ld;
    const T wr = __ldg(p.w + row);
    const T xi = __ldg(zr + i);
    const vec2 z01 = __ldg(reinterpret_cast<const vec2*>(zr + j));
    const vec2 z23 = __ldg(reinterpret_cast<const vec2*>(zr + j + 2));
    const T* __restrict__ mean = stat;
    const T* __restrict__ sdev = stat + ld;
    T mi = T(0), si = T(1), sw = T(0);
    vec2 m01, m23, s01, s23;
    if (cX || cY) {
      mi = __ldg(mean + i);
      m01 = __ldg(reinterpret_cast<const vec2*>(mean + j));
      m23 = __ldg(reinterpret_cast<const vec2*>(mean + j + 2));
      sw = (T)fs[f].sw;
    }
    if (sX || sY) {
      si = __ldg(sdev + i);
      s01 = __ldg(reinterpret_cast<const vec2*>(sdev + j));
      s23 = __ldg(reinterpret_cast<const vec2*>(sdev + j + 2));
    }
    const T zj[4] = {z01.x, z01.y, z23.x, z23.y};
    const T mj[4] = {m01.x, m01.y, m23.x, m23.y};
    const T sj[4] = {s01.x, s01.y, s23.x, s23.y};
    const T wxi = Rn<T>::mul(xi, wr);
    T v[4];
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const T a = swp[b] ? Rn<T>::mul(zj[b], wr) : wxi;
      const T c = swp[b] ? xi : zj[b];
      T r = Rn<T>::sub(tt[b], Rn<T>::mul(a, c));
      if (isx[b]) {
        if (cX) r = Rn<T>::sub(r, Rn<T>::mul(sw, Rn<T>::mul(mi, mj[b])));
        if (sX) r = Rn<T>::div(r, Rn<T>::mul(si, sj[b]));
      } else {
        if (cX || cY) r = Rn<T>::sub(r, Rn<T>::mul(sw, Rn<T>::mul(mi, mj[b])));
        if (sX && sY) r = Rn<T>::div(r, Rn<T>::mul(si, sj[b]));
        else if (sX) r = Rn<T>::div(r, si);
        else if (sY) r = Rn<T>::div(r, sj[b]);
      }
      v[b] = r;
    }
    if (fast_store) {
      vec2 lo, hi;
      lo.x = v[0]; lo.y = v[1]; hi.x = v[2]; hi.y = v[3];
      *reinterpret_cast<vec2*>(oxx) = lo;
      *reinterpret_cast<vec2*>(oxx + 2) = hi;
    } else {
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int64_t jj = j + b;
        if (jj < K) { if (wxx) oxx[b] = v[b]; }
        else if (jj < C && wxy) oxy[jj - K] = v[b];
      }
    }
    stat += 2 * ld;
    oxx += e.xx_stride;
    oxy += e.xy_stride;
  }
}

// ------------------------------------------------------------------------------------------------------
// Leave-one-out, streaming form (default).  The result of fold f is
//   A_ij = (T_ij - w x_i z_j - sw m_i m_j) / (s_i s_j)                       (cvmatrix/cvmatrix.py:1001-1009)
// and the fold is bound by WRITING its K x (K + M) result.  Matrices owe the reference 1e-12, not its bits, so the
// per-element work is cut to two FMAs and two multiplications on operand rows prepared once per fold:
//   v_c = rn(sqrt(w) z_c)         u_c = rn(sqrt(sw) m_c)  (0 where the flags do not centre)         r_c = 1 / s_c  (1 where
//   they do not scale)            A_ij = fma(-v_i, v_j, fma(-urow_i, ucol_j, T_ij)) * (r_i * r_j)
// Every product is symmetric in (i, j) bit for bit (an FMA rounds the exact product once), so XTX comes out exactly
// symmetric without mirroring.  `urow` differs from `ucol` only for X columns when center_Y is set without center_X:
// XTY is then centred (row side needs the X means) but XTX is not.
// k_loo_operands: one thread per (fold, column).  k_loo_tiles: CTA = 32 x 128 output tile (warp = 4 rows, lane = 4
// columns, the 16 totals in registers) streamed over LOO_FOLDS folds; per fold a thread loads 6 + 6 16-byte operand
// vectors (the row side is warp-uniform) and stores 4 x 32 bytes, a warp 4 x 1 KB of contiguous output rows.
// The exact form k_loo_folds (IEEE division, numpy's operation order, bit-identical to the reference for one-row folds)
// stays selectable (cvmx_set_loo_mode).
// ------------------------------------------------------------------------------------------------------
constexpr int LOO_TR = 32, LOO_TC = 128, LOO_FOLDS = 32, LOO_THREADS = 256;

// operand rows are float64 for both model dtypes: a float32 model then rounds ONCE, on the final store (its own
// float32 evaluation of T - G loses ~1e-5 of the centred result to cancellation; SURVEY.md Appendix B)
// STATS: the fold's column sums are the row itself (s = rn(w z), q = rn(s z): numpy's sequential sum of one row), so the
// thread also turns them into the fold's mean / std (finalize_column, into mom.stats == stats) instead of reading the
// output of a separate statistics pass; the fold scalars still come from k_weight_mass.
template <typename T, bool STATS = false>
__global__ void __launch_bounds__(128) k_loo_operands(const T* __restrict__ Z, const T* __restrict__ w, int64_t ld, int64_t K, int64_t M,
                                                      const int64_t* __restrict__ rows, const T* __restrict__ stats,
                                                      const FoldScalars* __restrict__ fs, uint32_t flags, double* __restrict__ opnd,
                                                      const MomentParams<T> mom = MomentParams<T>()) {
  const int64_t c = (int64_t)blockIdx.y * blockDim.x + threadIdx.x;
  const int64_t f = blockIdx.x;
  if (c >= ld) return;
  double* o = opnd + (size_t)f * 4 * ld;
  if (c >= K + M) { o[c] = 0.0; o[ld + c] = 0.0; o[2 * ld + c] = 1.0; o[3 * ld + c] = 0.0; return; }
  const bool cX = flags & 1, cY = flags & 2, sX = flags & 4, sY = flags & 8;
  const bool isX = c < K;
  const int64_t row = rows[f];
  if (STATS) {
    const T z = Z[row * ld + c];
    const T wz = Rn<T>::mul(z, w[row]);
    finalize_column<T>(mom, f, c, Rn<T>::add(T(0), wz), Rn<T>::add(T(0), Rn<T>::mul(wz, z)));
  }
  // (STATS: read back through the pointer just written - `stats` is a restrict-qualified read-only view of the same rows)
  const T* st = STATS ? mom.stats : stats;
  const double mean = (double)st[(size_t)f * 2 * ld + c], sd = (double)st[(size_t)f * 2 * ld + ld + c];
  const double rsw = __dsqrt_rn(fs[f].sw);
  o[c] = __dmul_rn(__dsqrt_rn((double)w[row]), (double)Z[row * ld + c]);
  const double um = __dmul_rn(rsw, mean);
  o[ld + c] = (isX ? cX : (cX || cY)) ? um : 0.0;            // column side
  o[2 * ld + c] = (isX ? sX : sY) ? __ddiv_rn(1.0, sd) : 1.0;
  o[3 * ld + c] = (isX && (cX || cY)) ? um : 0.0;            // row side (X columns only)
}

struct Dbl4 {
  double v[4];
  __device__ __forceinline__ void load(const double* p) {
    const double2 a = __ldg(reinterpret_cast<const double2*>(p)), b = __ldg(reinterpret_cast<const double2*>(p + 2));
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
  }
};

// Column map of a lane inside a 128-column tile.  float64: two column PAIRS 64 columns apart, so that each of the two
// 16-byte stores of a row is contiguous across the warp (512 bytes, whole sectors; four consecutive columns per lane
// would leave every 32-byte sector half-written by each instruction).  float32: four consecutive columns, one 16-byte store.
template <typename T> struct LooMap;
template <> struct LooMap<double> {
  static __device__ __forceinline__ int col(int lane, int b) { return (b < 2 ? 0 : 64) + 2 * lane + (b & 1); }
  static __device__ __forceinline__ void load(const double* base, int lane, double (&v)[4]) {   // base: column 0 of the tile
    const double2 a = __ldg(reinterpret_cast<const double2*>(base + 2 * lane)), b = __ldg(reinterpret_cast<const double2*>(base + 64 + 2 * lane));
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
  }
  static __device__ __forceinline__ void store(double* base, int lane, const double (&o)[4], bool second) {
    *reinterpret_cast<double2*>(base + 2 * lane) = make_double2(o[0], o[1]);
    if (second) *reinterpret_cast<double2*>(base + 64 + 2 * lane) = make_double2(o[2], o[3]);
  }
  static constexpr int FIRST = 2;     // columns b < FIRST belong to the first store
};
template <> struct LooMap<float> {
  static __device__ __forceinline__ int col(int lane, int b) { return 4 * lane + b; }
  static __device__ __forceinline__ void load(const double* base, int lane, double (&v)[4]) {
    const double2 a = __ldg(reinterpret_cast<const double2*>(base + 4 * lane)), b = __ldg(reinterpret_cast<const double2*>(base + 4 * lane + 2));
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
  }
  static __device__ __forceinline__ void store(float* base, int lane, const double (&o)[4], bool) {
    *reinterpret_cast<float4*>(base + 4 * lane) = make_float4((float)o[0], (float)o[1], (float)o[2], (float)o[3]);
  }
  static constexpr int FIRST = 4;
};

template <typename T>
__global__ void __launch_bounds__(LOO_THREADS, 2) k_loo_tiles(const T* __restrict__ Ttot, const double* __restrict__ opnd, int64_t ld, int64_t K,
                                                              int64_t M, int col_tiles, int64_t nfolds, uint32_t want,
                                                              T* __restrict__ out_xx, int64_t xx_pitch, int64_t xx_stride,
                                                              T* __restrict__ out_xy, int64_t xy_pitch, int64_t xy_stride) {
  typedef LooMap<T> Map;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int rt = blockIdx.x / col_tiles, ct = blockIdx.x % col_tiles;
  const int64_t i0 = (int64_t)rt * LOO_TR + 4 * warp, jt = (int64_t)ct * LOO_TC;    // first row of the thread, first column of the tile
  const int64_t C = K + M;
  const int64_t fbeg = (int64_t)blockIdx.y * LOO_FOLDS;
  const int nf = (int)(min(nfolds, fbeg + LOO_FOLDS) - fbeg);
  const bool wxx = want & 1, wxy = want & 2;
  if (i0 >= K || jt >= C) return;
  if (!((wxx && jt < K) || (wxy && jt + LOO_TC > K))) return;
  const int nr = (int)min((int64_t)4, K - i0);                       // live rows of this thread
#define LOO_JC(b) (jt + Map::col(lane, (b)))
  // 16-byte stores: the lane's columns of a store all inside XTX, 16-byte aligned element offsets on every row
  constexpr int VEC = 16 / sizeof(T);
  const bool aligned = wxx && (xx_pitch % VEC == 0) && (xx_stride % VEC == 0) && (reinterpret_cast<uintptr_t>(out_xx) % 16 == 0);
  const bool fast1 = aligned && LOO_JC(Map::FIRST - 1) < K;          // first store (float32: the only one)
  const bool fast2 = aligned && LOO_JC(3) < K;                       // second store (float64)
  const bool fast = fast1 && (Map::FIRST == 4 || fast2 || LOO_JC(2) >= C);   // nothing of this lane needs the scalar path

  double tt[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) tt[a][b] = (double)__ldg(Ttot + min(i0 + a, K - 1) * ld + min(LOO_JC(b), ld - 1));
  const double* __restrict__ op = opnd + (size_t)fbeg * 4 * ld;      // tiles never reach past ld: ld % 32 == 0 and ...
  const bool in_ld = jt + LOO_TC <= ld;                              // ... a partial last tile loads column by column
  T* oxx = out_xx + (size_t)fbeg * xx_stride + i0 * xx_pitch + jt;
  T* oxy = out_xy + (size_t)fbeg * xy_stride + i0 * xy_pitch;

#pragma unroll 1
  for (int f = 0; f < nf; ++f) {
    double vj[4], uj[4], rj[4];
    Dbl4 vi, ui, ri;
    if (in_ld) {
      Map::load(op + jt, lane, vj); Map::load(op + ld + jt, lane, uj); Map::load(op + 2 * ld + jt, lane, rj);
    } else {
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int64_t j = min(LOO_JC(b), ld - 1);
        vj[b] = __ldg(op + j); uj[b] = __ldg(op + ld + j); rj[b] = __ldg(op + 2 * ld + j);
      }
    }
    vi.load(op + i0); ri.load(op + 2 * ld + i0); ui.load(op + 3 * ld + i0);   // warp-uniform (i0 + 3 < ld)
    double o[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b)
        o[a][b] = __dmul_rn(fma(-vi.v[a], vj[b], fma(-ui.v[a], uj[b], tt[a][b])), __dmul_rn(ri.v[a], rj[b]));
    if (fast) {
#pragma unroll
      for (int a = 0; a < 4; ++a)
        if (a < nr) Map::store(oxx + a * xx_pitch, lane, o[a], fast2);
    } else {
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        if (a >= nr) continue;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const int64_t jj = LOO_JC(b);
          if (jj < K) { if (wxx) oxx[a * xx_pitch + (jj - jt)] = (T)o[a][b]; }
          else if (jj < C && wxy) oxy[a * xy_pitch + (jj - K)] = (T)o[a][b];
        }
      }
    }
    op += 4 * ld;
    oxx += xx_stride;
    oxy += xy_stride;
  }
#undef LOO_JC
}

// ------------------------------------------------------------------------------------------------------
// Leave-few-out (2 .. SMALL_MAX_ROWS validation rows per fold), streaming form: one operand row v_r = rn(sqrt(w_r) z_r)
// PER validation row, the downdate accumulated on its own in float64 and the epilogue of gram_epilogue:
//   G_ij = sum_r v_ri v_rj ;  A = rn(T_ij - G_ij) ;  A = rn(A - rn(sw rn(m_i m_j))) ;  A = rn(A (r_i r_j))
// n FMAs + 6 operations per element instead of the exact form's rounded products and IEEE division (k_small_folds,
// ~100 instructions per element).  (Folding the centring into the FMA chain, as the one-row kernel does, was measured
// against the golden fixtures: on data whose mean dwarfs its spread the error is relative to T, 1e-12 of the result.)
// Every product is symmetric in (i, j) and the FMA chain runs over r in the same order for (i, j) and (j, i): XTX is
// exactly symmetric.  Operand rows per fold: [mcol | r | mrow | v_0 .. v_{R-1}] x ld float64 (mcol / mrow: the mean where
// the flags centre that side, else 0), R = the longest fold of the launch.
// ------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(128) k_few_operands(const T* __restrict__ Z, const T* __restrict__ w, int64_t ld, int64_t K, int64_t M,
                                                      const int64_t* __restrict__ offs, const int64_t* __restrict__ indices,
                                                      const T* __restrict__ stats, const FoldScalars* __restrict__ fs, uint32_t flags,
                                                      int R, double* __restrict__ opnd) {
  const int64_t c = (int64_t)blockIdx.y * blockDim.x + threadIdx.x;
  const int64_t f = blockIdx.x;
  if (c >= ld) return;
  double* o = opnd + (size_t)f * (3 + R) * ld;
  const int64_t beg = offs[f];
  const int n = (int)(offs[f + 1] - beg);
  if (c >= K + M) {
    o[c] = 0.0; o[ld + c] = 1.0; o[2 * ld + c] = 0.0;
    for (int r = 0; r < n; ++r) o[(size_t)(3 + r) * ld + c] = 0.0;
    return;
  }
  const bool cX = flags & 1, cY = flags & 2, sX = flags & 4, sY = flags & 8;
  const bool isX = c < K;
  const double mean = (double)stats[(size_t)f * 2 * ld + c], sd = (double)stats[(size_t)f * 2 * ld + ld + c];
  o[c] = (isX ? cX : (cX || cY)) ? mean : 0.0;               // column side
  o[ld + c] = (isX ? sX : sY) ? __ddiv_rn(1.0, sd) : 1.0;
  o[2 * ld + c] = (isX && (cX || cY)) ? mean : 0.0;          // row side (X columns only)
  for (int r = 0; r < n; ++r) {
    const int64_t row = indices[beg + r];
    o[(size_t)(3 + r) * ld + c] = __dmul_rn(__dsqrt_rn((double)w[row]), (double)Z[row * ld + c]);
  }
}

template <typename T>
__global__ void __launch_bounds__(LOO_THREADS, 2) k_few_tiles(const T* __restrict__ Ttot, const double* __restrict__ opnd, int64_t ld, int64_t K,
                                                              int64_t M, int col_tiles, int64_t nfolds, const int64_t* __restrict__ offs,
                                                              const FoldScalars* __restrict__ fs, int R, uint32_t flags, uint32_t want,
                                                              T* __restrict__ out_xx, int64_t xx_pitch,
                                                              int64_t xx_stride, T* __restrict__ out_xy, int64_t xy_pitch,
                                                              int64_t xy_stride) {
  typedef LooMap<T> Map;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int rt = blockIdx.x / col_tiles, ct = blockIdx.x % col_tiles;
  const int64_t i0 = (int64_t)rt * LOO_TR + 4 * warp, jt = (int64_t)ct * LOO_TC;
  const int64_t C = K + M;
  const int64_t fbeg = (int64_t)blockIdx.y * LOO_FOLDS;
  const int nf = (int)(min(nfolds, fbeg + LOO_FOLDS) - fbeg);
  const bool wxx = want & 1, wxy = want & 2;
  if (i0 >= K || jt >= C) return;
  if (!((wxx && jt < K) || (wxy && jt + LOO_TC > K))) return;
  const int nr = (int)min((int64_t)4, K - i0);
#define LOO_JC(b) (jt + Map::col(lane, (b)))
  constexpr int VEC = 16 / sizeof(T);
  const bool aligned = wxx && (xx_pitch % VEC == 0) && (xx_stride % VEC == 0) && (reinterpret_cast<uintptr_t>(out_xx) % 16 == 0);
  const bool fast1 = aligned && LOO_JC(Map::FIRST - 1) < K;
  const bool fast2 = aligned && LOO_JC(3) < K;
  const bool fast = fast1 && (Map::FIRST == 4 || fast2 || LOO_JC(2) >= C);

  T tt[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) tt[a][b] = __ldg(Ttot + min(i0 + a, K - 1) * ld + min(LOO_JC(b), ld - 1));
  // numpy SKIPS the centring of a block the flags do not centre (XTX iff center_X, XTY iff center_X or center_Y): a mean
  // that is NaN there (a fold that holds every row) must not reach the result through 0 * NaN
  bool cen[4];
#pragma unroll
  for (int b = 0; b < 4; ++b) cen[b] = (LOO_JC(b) < K) ? (flags & 1) != 0 : (flags & 3) != 0;
  const size_t fstride = (size_t)(3 + R) * ld;
  const double* __restrict__ op = opnd + (size_t)fbeg * fstride;
  const bool in_ld = jt + LOO_TC <= ld;
  T* oxx = out_xx + (size_t)fbeg * xx_stride + i0 * xx_pitch + jt;
  T* oxy = out_xy + (size_t)fbeg * xy_stride + i0 * xy_pitch;
  auto load_cols = [&](const double* row, double (&v)[4]) {   // the lane's four columns of an operand row
    if (in_ld) { Map::load(row + jt, lane, v); return; }
#pragma unroll
    for (int b = 0; b < 4; ++b) v[b] = __ldg(row + min(LOO_JC(b), ld - 1));
  };

#pragma unroll 1
  for (int f = 0; f < nf; ++f) {
    const int n = (int)(offs[fbeg + f + 1] - offs[fbeg + f]);
    const T sw = (T)fs[fbeg + f].sw;
    double g[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) g[a][b] = 0.0;
#pragma unroll 1
    for (int r = 0; r < n; ++r) {
      const double* vr = op + (size_t)(3 + r) * ld;
      double vj[4];
      Dbl4 vi;
      load_cols(vr, vj); vi.load(vr + i0);                          // the row side is warp-uniform (i0 + 3 < ld)
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) g[a][b] = fma(vi.v[a], vj[b], g[a][b]);
    }
    double mj[4], rj[4];
    Dbl4 mi, ri;
    load_cols(op, mj); load_cols(op + ld, rj);
    ri.load(op + ld + i0); mi.load(op + 2 * ld + i0);
    double o[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        T v = Rn<T>::sub(tt[a][b], (T)g[a][b]);
        if (cen[b]) v = Rn<T>::sub(v, Rn<T>::mul(sw, Rn<T>::mul((T)mi.v[a], (T)mj[b])));
        o[a][b] = __dmul_rn((double)v, __dmul_rn(ri.v[a], rj[b]));
      }
    if (fast) {
#pragma unroll
      for (int a = 0; a < 4; ++a)
        if (a < nr) Map::store(oxx + a * xx_pitch, lane, o[a], fast2);
    } else {
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        if (a >= nr) continue;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const int64_t jj = LOO_JC(b);
          if (jj < K) { if (wxx) oxx[a * xx_pitch + (jj - jt)] = (T)o[a][b]; }
          else if (jj < C && wxy) oxy[a * xy_pitch + (jj - K)] = (T)o[a][b];
        }
      }
    }
    op += fstride;
    oxx += xx_stride;
    oxy += xy_stride;
  }
#undef LOO_JC
}

}  // namespace cvmx
