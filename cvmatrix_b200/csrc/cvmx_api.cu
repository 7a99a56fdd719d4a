// libcvmx: C ABI (include/cvmx.h) over the sm_100a kernels.  Host-side orchestration only; all
// arithmetic of the hot path runs in kernels_stats.cuh / kernels_gram.cuh.  There is no CPU fallback.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "../../include/cvmx.h"
#include "host_stager.h"
#include "kernels_stats.cuh"
#include "kernels_gram.cuh"
#include "kernels_gram_tc.cuh"
#include "kernels_scan.cuh"
#include "kernels_pls.cuh"
#include "kernels_ridge.cuh"
#include <cstdlib>
#include <type_traits>

using namespace cvmx;

namespace {

thread_local std::string g_err;

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <typename U> U* as() const { return reinterpret_cast<U*>(p); }
};

struct Plan {                 // launch plan of one fold range (cached)
  int64_t fold_begin = -1, fold_end = -1; uint32_t want = 0; int64_t csr_version = -1;
  std::vector<GramUnit> units;
  std::vector<int2> tiles;
  std::vector<int32_t> fold_units;   // first unit of each fold
  std::vector<int32_t> split_folds;  // folds with nsplit > 1
  int64_t n_partial_units = 0;
  int64_t max_rows = 0;
};

// Device copies of a launch plan that repeats from step to step (sharded phases): re-uploading four small tables
// costs four DMA operations on the critical path of every step.
struct TableCache {
  std::vector<int64_t> key;
  DevBuf units, tiles, fold_units, split_folds;
  int64_t n_units = 0, n_partial_units = 0;
  int ntiles = 0;
  void release() { units.release(); tiles.release(); fold_units.release(); split_folds.release(); key.clear(); }
};

}  // namespace

struct cvmx_handle {
  int device = 0, dtype = CVMX_F64;
  uint32_t flags = 0;
  int64_t ddof = 1;
  double resolution = 0;
  int sm_count = 148;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  // side stream for the statistics kernels when they can overlap the Gram kernel (large, row-split folds and fit)
  cudaStream_t aux_stream = nullptr, aux2_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_mass = nullptr;
  cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_stage[2] = {nullptr, nullptr};   // fit: staged host->device upload
  DevBuf stage[2];
  // fitted state
  bool fitted = false, weighted = false;
  int64_t N = 0, K = 0, M = 0, ld = 0;
  DevBuf Z, w, Ttot, sum_z, sumsq_z, fit_scal;
  // CSR (device) + host offsets
  int64_t P = 0, csr_version = 0;
  DevBuf d_off, d_idx;
  std::vector<int64_t> h_off;
  // ad-hoc index set (cvmx_training_indices)
  DevBuf a_off, a_idx;
  // scratch
  DevBuf units, tiles, fold_units, split_folds, partials, stats, rawsums, fscal, pwcols, errflag, out_xx, out_xy, out_small;
  Plan plan;
  bool attr_gram = false, attr_mom = false, attr_gram_fused = false;
  // binade scan of the moment chains (kernels_scan.cuh): 0 off, 1 when the chains are the critical path, 2 always
  int scan_mode = 1;
  // leave-one-out batches: 0 streaming form (two FMAs + reciprocal scaling per element, matrices to ~1e-15 of the
  // reference), 1 exact form (numpy's operation order and IEEE division: bit-identical matrices for one-row folds)
  int loo_mode = 0;
  DevBuf loo_ops;
  // cross-validated PLS (cvmx_pls_cv): per-window working state, PRESS chunk table and partials, staged host outputs
  DevBuf pls_ws, pls_tab, pls_part, pls_out;
  // cross-validated ridge (cvmx_ridge_cv): pass scratch (cvmx_ridge_plan's layout), PRESS chunk table and partials, penalties
  DevBuf ridge_ws, ridge_tab, ridge_part, ridge_alpha;
  // out-of-fold predictions of both for host outputs: one PRESS launch's rows, at most CV_PRED_STAGE_BYTES (one chunk's rows)
  DevBuf cv_pred;
  // fused fit + folds (cvmx_fit_folds): raw float64 Gram of every fold of a true partition, [P][ntiles][GACC][GTHREADS],
  // valid while csr_version == fold_gram_version; cvmx_training_batch then only runs statistics + epilogue
  TableCache tc_gram, tc_finish;
  DevBuf fold_gram, fold_raw, chunk_ranges;   // fold_raw: [P][2][ld] raw column sums of every fold, same validity
  int64_t fold_gram_version = -1;
  // row-slab mode (cvmx_fit_end_slab): this handle holds rows [row0, row0 + N) of an N_glob-row data set; the weight
  // vector and the validation sets are ALSO kept in global form for the (pairwise, unsplittable) weight sums
  bool slab = false;
  int64_t N_glob = 0, row0 = 0;
  DevBuf w_glob, g_off, g_idx;
  std::vector<int64_t> g_h_off;
  // decoupled slab chain (cvmx_slab_scan_local / _prepare): which sums the scan planes currently describe
  int slab_scan_mode = 0;        // 0 none, 1 fit totals, 2 fold sums
  int slab_scan_stage = 0;       // 1 local passes done, 2 prepared (passes 2 and 3 done)
  int64_t slab_scan_f0 = 0, slab_scan_f1 = 0, slab_scan_csr = -1;
  bool mass_started = false;     // cvmx_slab_begin: w_glob uploaded and the weight mass launched before the rows arrive
  bool mass_pending = false;     // ... with the weight mass still running on side stream 2 (ev_mass)
  bool fit_pre_done = false;     // fit mode: accumulator -> totals and the weight mass already ran (cvmx_slab_scan_local)
  // streaming / sharded fit (cvmx_fit_begin / cvmx_fit_rows / cvmx_fit_end)
  bool filling = false;
  int64_t fill_units_cap = 0, fill_calls = 0;
  DevBuf ystage;
  DevBuf scan_seg, scan_ok, scan_list, scan_cnt, scan_look, peer_sum;
  // float32 Gram kernel (CVMX_F32_TC): 1 = k_gram_tc (tcgen05 kind::tf32, 3xTF32, ~3e-7 of the raw products) for wide models
  // (K (K + M) >= F32_TC_MIN_WIDTH, the tensor-core-bound regime), k_gram<float> (float64 accumulation on the DMMA pipe) for
  // narrow ones; 0 = always k_gram<float>; 2 = always k_gram_tc.  Decided once per fit (fmap): every raw fragment buffer
  // of a handle - partials, kept fold Grams, the buffers ranks exchange - then has ONE layout, on every rank.
  int f32_tc = 1;
  int fmap = 0;
  bool attr_tc = false;
  // contiguous uploads from PAGEABLE host memory go through a page-locked ring filled by worker threads (host_stager.h);
  // CVMX_HOST_STAGER=0 leaves them to the driver's bounce buffer
  // fold statistics inside the Gram kernel for batches of single-unit folds (GramParams::fuse_stats); CVMX_FUSE_STATS=0: separate pass
  int fuse_stats = 1;
  DevBuf stat_flags;
  HostStager* stager = nullptr;
  int use_stager = 1;
  int scan_spec = 1;    // fold statistics: passes 1 and 3 in one read of the rows from guessed proxies (k_scan_spec); 0: four passes
  int64_t scan_launches = 0;
  int64_t launches = 0;
  // optional per-kernel timing (cvmx_profile_*): event pairs recorded on the handle stream
  bool prof = false;
  std::vector<cudaEvent_t> prof_ev;      // pool
  std::vector<std::pair<int, std::pair<int, int>>> prof_spans;  // (kind, (ev begin, ev end))
  size_t prof_used = 0;
  std::string err;
};

namespace {

int32_t fail(cvmx_t* h, int32_t code, const std::string& msg) {
  if (h) h->err = msg;
  g_err = msg;
  return code;
}

#define CU(h, expr)                                                                                     \
  do {                                                                                                  \
    cudaError_t e__ = (expr);                                                                           \
    if (e__ != cudaSuccess)                                                                             \
      return fail(h, e__ == cudaErrorMemoryAllocation ? CVMX_ERR_NOMEM : CVMX_ERR_CUDA,                  \
                  std::string(#expr) + ": " + cudaGetErrorString(e__));                                 \
  } while (0)

// Every ABI entry works on the handle's device but leaves the CALLER's current device as it found it: the current
// device is per-thread driver state shared with torch, and cvmx_destroy runs from a Python destructor at arbitrary times.
struct DeviceGuard {
  int prev = -1;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) err = cudaSetDevice(dev); else prev = -1;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};
#define ON_DEVICE(h) DeviceGuard guard__((h)->device); CU(h, guard__.err)

enum { PROF_STATS = 0, PROF_GRAM = 1, PROF_REDUCE = 2, PROF_KINDS = 3 };

int prof_mark(cvmx_t* h) {
  if (!h->prof) return -1;
  if (h->prof_used == h->prof_ev.size()) {
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return -1;
    h->prof_ev.push_back(e);
  }
  cudaEventRecord(h->prof_ev[h->prof_used], h->stream);
  return (int)h->prof_used++;
}
void prof_span(cvmx_t* h, int kind, int a, int b) {
  if (h->prof && a >= 0 && b >= 0) h->prof_spans.push_back({kind, {a, b}});
}

// Contiguous host -> device copy on `stream`: page-locked sources go straight to the DMA engine; large pageable ones through
// the stager (`pageable`: the caller looked the source up once per call).
inline cudaError_t h2d_copy(cvmx_t* h, void* dst, const void* src, size_t bytes, cudaStream_t stream, bool pageable) {
  if (pageable && h->use_stager && bytes >= ((size_t)4 << 20)) {
    try {
      if (!h->stager) h->stager = new HostStager();
      return h->stager->copy(dst, src, bytes, stream);
    } catch (...) {   // no worker threads to be had: leave this and later copies to the driver
      h->use_stager = 0;
    }
  }
  return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream);
}

inline size_t esz(const cvmx_t* h) { return h->dtype == CVMX_F64 ? 8 : 4; }
inline int64_t round_up(int64_t a, int64_t b) { return (a + b - 1) / b * b; }

// ---- launch planning -------------------------------------------------------------------------------
// Tiles on or above the diagonal of the K x (K+M) result, restricted to what `want` needs.
void plan_tiles(const cvmx_t* h, uint32_t want, std::vector<int2>& tiles) {
  tiles.clear();
  const int64_t TI = (h->K + GB - 1) / GB, TJ = (h->K + h->M + GB - 1) / GB;
  // Diagonal tiles first (and the tiles (0, bj >= TI) of Y-only column blocks): with fused fold statistics every tile of a
  // fold waits for their column chains before its epilogue - started first, and the diagonal ones issuing 9/16 of the DMMAs
  // of a full tile, they are done before the others need them.
  for (int pass = 0; pass < 2; ++pass)
    for (int64_t bi = 0; bi < TI; ++bi)
      for (int64_t bj = bi; bj < TJ; ++bj) {
        const bool first = bi == bj || (bi == 0 && bj >= TI);   // the tiles that carry column chains (GramParams::fuse_stats)
        if (first != (pass == 0)) continue;
        const bool has_x = bj * GB < h->K;
        const bool has_y = (bj + 1) * GB > h->K && h->M > 0;
        if (((want & CVMX_WANT_XTX) && has_x) || ((want & CVMX_WANT_XTY) && has_y)) tiles.push_back(make_int2((int)bi, (int)bj));
      }
}

// ---- row-split plan of few large folds -------------------------------------------------------------------------------
// The hardware places CTAs greedily (next CTA to the first SM that frees up), so equal-sized units end in a ragged last
// wave: 1150 equal items on 148 SMs leave a quarter of the GPU idle for a whole item.  Unit sizes therefore TAPER - a few
// long units, then halves, quarters, ... - and are launched longest first, which is the classic LPT packing; the sizes
// are chosen by simulating that placement with the measured relative tile costs (a diagonal tile issues 9/16 of the
// DMMAs of a full one and takes 0.79 of its time, measured by tools/tile_cost.py over the same row-split units; ~1.5
// pipeline stages of fixed cost per CTA).  Returns per fold the unit sizes in split order.
double simulate_makespan(std::vector<int64_t> unit_rows, const std::vector<double>& tile_cost, int64_t sms) {
  std::sort(unit_rows.begin(), unit_rows.end(), std::greater<int64_t>());
  std::vector<double> heap((size_t)sms, 0.0);   // min-heap of SM finish times
  auto cmp = std::greater<double>();
  for (int64_t n : unit_rows)
    for (double c : tile_cost) {
      std::pop_heap(heap.begin(), heap.end(), cmp);
      heap.back() += ((double)n + 1.5 * GBK) * c;
      std::push_heap(heap.begin(), heap.end(), cmp);
    }
  return *std::max_element(heap.begin(), heap.end());
}

std::vector<int64_t> taper_sizes(int64_t n, int64_t R, int levels) {
  std::vector<int64_t> tail;
  int64_t r = R;
  for (int l = 0; l < levels; ++l) { r = std::max<int64_t>(256, (r / 2) / GBK * GBK); tail.push_back(r); tail.push_back(r); }
  int64_t tail_sum = 0;
  for (int64_t t : tail) tail_sum += t;
  std::vector<int64_t> sizes;
  const int64_t main_rows = std::max<int64_t>(0, n - tail_sum);
  if (main_rows > 0) {
    const int64_t k = std::max<int64_t>(1, (main_rows + R / 2) / R), per = round_up((main_rows + k - 1) / k, GBK);
    for (int64_t i = 0; i < k; ++i) {
      const int64_t a = std::min(main_rows, i * per), b = std::min(main_rows, (i + 1) * per);
      if (b > a) sizes.push_back(b - a);
    }
  }
  int64_t rem = n;
  for (int64_t v : sizes) rem -= v;
  for (int64_t t : tail) {
    const int64_t v = std::min(rem, t);
    if (v > 0) { sizes.push_back(v); rem -= v; }
  }
  if (rem > 0) { if (sizes.empty()) sizes.push_back(rem); else sizes.back() += rem; }
  return sizes;
}

std::vector<std::vector<int64_t>> plan_tapered(const std::vector<int64_t>& fold_rows, const std::vector<int2>& tiles, int64_t sms,
                                               int64_t r_lo, int64_t r_hi) {
  // the search costs ~10 ms of host time: remember the last few answers (a refit with the same fold sizes re-plans)
  struct Memo { std::vector<int64_t> rows; size_t ntiles; int64_t sms; std::vector<std::vector<int64_t>> sizes; };
  static thread_local std::vector<Memo> memo;
  for (const Memo& m : memo)
    if (m.rows == fold_rows && m.ntiles == tiles.size() && m.sms == sms) return m.sizes;
  std::vector<double> tile_cost;
  for (const int2& t : tiles) tile_cost.push_back(t.x == t.y ? 0.79 : 1.0);
  double best = 1e300;
  std::vector<std::vector<int64_t>> best_sizes;
  for (int64_t R = r_lo; R <= r_hi; R += 8 * GBK)
    for (int levels = 2; levels <= 4; ++levels) {
      std::vector<std::vector<int64_t>> sizes;
      std::vector<int64_t> all;
      for (int64_t n : fold_rows) {
        sizes.push_back(n > 0 ? taper_sizes(n, R, levels) : std::vector<int64_t>{0});
        all.insert(all.end(), sizes.back().begin(), sizes.back().end());
      }
      const double mk = simulate_makespan(all, tile_cost, sms);
      if (mk < best - 1e-9) { best = mk; best_sizes = sizes; }
    }
  if (memo.size() >= 8) memo.erase(memo.begin());
  memo.push_back({fold_rows, tiles.size(), sms, best_sizes});
  return best_sizes;
}

// Launch order = longest unit first (LPT).  A fold's units keep their split numbers and partial slots; fold_units[f] only
// has to point at ANY unit of fold f (k_gram_reduce / k_partial_sum read the fold's part_base and nsplit from it).
void sort_units_longest_first(Plan& pl) {
  std::stable_sort(pl.units.begin(), pl.units.end(),
                   [](const GramUnit& a, const GramUnit& b) { return a.row_end - a.row_begin > b.row_end - b.row_begin; });
  for (size_t i = pl.units.size(); i-- > 0;) pl.fold_units[pl.units[i].fold] = (int32_t)i;
}

// Row-split policy.  Many small folds: one unit per fold, epilogue fused into the Gram kernel.  Few large
// folds: split the rows so that (units x tiles) fills the SMs in whole waves; partials are reduced in
// split order by k_gram_reduce (deterministic).
void plan_units(const cvmx_t* h, const int64_t* off, int64_t f0, int64_t f1, int ntiles, Plan& pl) {
  const int64_t Pn = f1 - f0;
  pl.units.clear(); pl.fold_units.assign(Pn, 0); pl.split_folds.clear();
  pl.n_partial_units = 0; pl.max_rows = 0;
  const int64_t sms = h->sm_count;
  int64_t rows_per_unit = INT64_MAX;
  if (Pn * ntiles < 8 * sms) {
    double best = -1;
    // wide K: the tiles alone fill the GPU, and every split costs ntiles x 128 KB of partial workspace - keep the
    // workspace below ~2 GB by making the units longer
    int64_t total_rows = 0;
    for (int64_t f = f0; f < f1; ++f) total_rows += off[f + 1] - off[f];
    const int64_t max_units = std::max<int64_t>(Pn, (int64_t)(((size_t)2 << 30) / ((size_t)std::max(ntiles, 1) * GACC * GTHREADS * sizeof(double))));
    const int64_t r_min = std::max<int64_t>(2048, round_up((total_rows + max_units - 1) / max_units, GBK));
    for (int64_t R = r_min; R <= r_min + 2048; R += GBK) {
      int64_t items = 0;
      for (int64_t f = f0; f < f1; ++f) items += std::max<int64_t>(1, (off[f + 1] - off[f] + R - 1) / R);
      items *= ntiles;
      const double eff = (double)items / (double)(sms * ((items + sms - 1) / sms));
      if (eff > best + 1e-9) { best = eff; rows_per_unit = R; }
    }
  }
  std::vector<std::vector<int64_t>> tapered;
  if (rows_per_unit != INT64_MAX && ntiles < sms) {     // (wide K: the tiles alone fill the GPU - equal, long units)
    std::vector<int64_t> fold_rows;
    for (int64_t f = f0; f < f1; ++f) fold_rows.push_back(off[f + 1] - off[f]);
    int64_t r_hi = 8192;
    if (const char* e = std::getenv("CVMX_PLAN_RHI")) r_hi = std::max<int64_t>(1024, std::atoll(e));   // experiment knob (DESIGN.md 5.1)
    tapered = plan_tapered(fold_rows, pl.tiles, sms, 1024, r_hi);
  }
  for (int64_t f = f0; f < f1; ++f) {
    const int64_t beg = off[f], n = off[f + 1] - off[f];
    pl.max_rows = std::max(pl.max_rows, n);
    std::vector<int64_t> sizes;
    if (!tapered.empty()) sizes = tapered[f - f0];
    else {
      // equal-sized splits, multiples of GBK rows
      const int64_t ns = (rows_per_unit == INT64_MAX) ? 1 : std::max<int64_t>(1, (n + rows_per_unit - 1) / rows_per_unit);
      const int64_t per = round_up((n + ns - 1) / ns, GBK);
      for (int64_t s = 0; s < ns; ++s) sizes.push_back(std::min(n, (s + 1) * per) - std::min(n, s * per));
    }
    const int64_t ns = (int64_t)sizes.size();
    pl.fold_units[f - f0] = (int32_t)pl.units.size();
    if (ns > 1) pl.split_folds.push_back((int32_t)(f - f0));
    int64_t pos = beg;
    for (int64_t s = 0; s < ns; ++s) {
      GramUnit u;
      u.row_begin = pos; u.row_end = pos + sizes[s];
      pos += sizes[s];
      u.fold = (int32_t)(f - f0); u.split = (int32_t)s; u.nsplit = (int32_t)ns;
      u.part_base = (int32_t)pl.n_partial_units;
      pl.units.push_back(u);
    }
    if (ns > 1) pl.n_partial_units += ns;
  }
  sort_units_longest_first(pl);
}

// The Gram kernel of the model dtype: float64 -> k_gram<double> (DMMA); float32 -> k_gram_tc (tcgen05 / tensor memory) or
// k_gram<float> (mma.sync TF32).  gp.fmap must say which of the two float32 kernels writes the accumulators.
// Narrow float32 models stay on the float64-accumulating kernel: they are not tensor-core-bound, and on cancellation-sensitive
// small cases (centred matrices of a few hundred rows and a handful of columns) float64 accumulation reproduces numpy-float32
// to its own rounding, which the 3xTF32 products (2^-22 per product) do not.
constexpr double F32_TC_MIN_WIDTH = 65536.0;   // K (K + M): K >~ 256
template <typename T> int fmap_of(const cvmx_t* h) { return sizeof(T) == 4 ? h->fmap : 0; }
template <typename T> void choose_fmap(cvmx_t* h, int64_t K, int64_t M) {
  h->fmap = (sizeof(T) == 4 && (h->f32_tc == 2 || (h->f32_tc == 1 && (double)K * (double)(K + M) >= F32_TC_MIN_WIDTH))) ? 1 : 0;
}

template <typename T>
int32_t launch_k_gram(cvmx_t* h, unsigned grid, const GramParams<T>& gp) {
  if constexpr (sizeof(T) == 4) {
    if (gp.fmap == 1) {
      if (!h->attr_tc) {
        CU(h, cudaFuncSetAttribute(k_gram_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gram_tc_smem_bytes()));
        h->attr_tc = true;
      }
      k_gram_tc<<<grid, GLAUNCH, gram_tc_smem_bytes(), h->stream>>>(gp);
      return CVMX_OK;
    }
  }
  if (gp.fuse_stats) {
    if (!h->attr_gram_fused) {
      CU(h, cudaFuncSetAttribute(k_gram<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gram_smem_bytes<T>()));
      h->attr_gram_fused = true;
    }
    k_gram<T, true><<<grid, GLAUNCH, gram_smem_bytes<T>(), h->stream>>>(gp);
    return CVMX_OK;
  }
  k_gram<T><<<grid, GLAUNCH, gram_smem_bytes<T>(), h->stream>>>(gp);
  return CVMX_OK;
}

template <typename T>
int32_t launch_gram(cvmx_t* h, const Plan& pl, const int64_t* d_indices, const EpiParams<T>& epi,
                    cudaEvent_t stats_ready = nullptr, bool fuse_stats = false) {
  const int ntiles = (int)pl.tiles.size();
  if (ntiles == 0 || pl.units.empty()) return CVMX_OK;
  CU(h, h->units.reserve(pl.units.size() * sizeof(GramUnit)));
  CU(h, h->tiles.reserve(pl.tiles.size() * sizeof(int2)));
  CU(h, h->fold_units.reserve(pl.fold_units.size() * sizeof(int32_t)));
  CU(h, cudaMemcpyAsync(h->units.p, pl.units.data(), pl.units.size() * sizeof(GramUnit), cudaMemcpyHostToDevice, h->stream));
  CU(h, cudaMemcpyAsync(h->tiles.p, pl.tiles.data(), pl.tiles.size() * sizeof(int2), cudaMemcpyHostToDevice, h->stream));
  CU(h, cudaMemcpyAsync(h->fold_units.p, pl.fold_units.data(), pl.fold_units.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
  if (pl.n_partial_units) {
    CU(h, h->partials.reserve((size_t)pl.n_partial_units * ntiles * GACC * GTHREADS * sizeof(double)));
    CU(h, h->split_folds.reserve(pl.split_folds.size() * sizeof(int32_t)));
    CU(h, cudaMemcpyAsync(h->split_folds.p, pl.split_folds.data(), pl.split_folds.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
  }
  GramParams<T> gp;
  gp.fmap = fmap_of<T>(h);
  gp.Z = h->Z.as<T>(); gp.w = h->w.as<T>(); gp.ld = h->ld;
  gp.indices = d_indices;
  gp.units = h->units.as<GramUnit>(); gp.tiles = h->tiles.as<int2>(); gp.ntiles = ntiles;
  gp.partials = h->partials.as<double>();
  gp.raw_out = nullptr; gp.force_partials = 0;
  gp.epi = epi;
  if (fuse_stats) {
    const size_t nf = pl.fold_units.size();
    CU(h, h->stat_flags.reserve(nf * sizeof(int)));
    CU(h, cudaMemsetAsync(h->stat_flags.p, 0, nf * sizeof(int), h->stream));
    const int TI = (int)((h->K + GB - 1) / GB);
    int nchain = 0;
    for (const int2& t : pl.tiles) nchain += t.x == t.y || (t.x == 0 && t.y >= TI);
    gp.fuse_stats = 1; gp.stat_flags = h->stat_flags.as<int>(); gp.stat_target = GPRODUCERS * nchain;   // the producer warps of every chain tile
    MomentParams<T>& mp = gp.mom;
    mp.Z = h->Z.as<T>(); mp.w = h->w.as<T>(); mp.ld = h->ld; mp.K = h->K; mp.M = h->M;
    mp.offsets = d_indices; mp.indices = d_indices; mp.fold0 = 0; mp.N = h->N;   // offsets != nullptr: fold mode of finalize_column
    mp.flags = h->flags; mp.resolution = (T)h->resolution;
    mp.sum_z = h->sum_z.as<T>(); mp.sumsq_z = h->sumsq_z.as<T>();
    mp.fs = epi.fs; mp.pw_cols = nullptr; mp.stats = const_cast<T*>(epi.stats); mp.raw = nullptr;
  }
  const size_t smem = gram_smem_bytes<T>();
  if (!h->attr_gram) {
    CU(h, cudaFuncSetAttribute(k_gram<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CU(h, cudaFuncSetAttribute(k_gram_reduce<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    h->attr_gram = true;
  }
  const int64_t grid = (int64_t)pl.units.size() * ntiles;
  if (grid > 0x7fffffffLL) return fail(h, CVMX_ERR_INVALID, "fold batch too large for one launch");
  const bool all_split = pl.split_folds.size() == pl.fold_units.size();
  if (stats_ready && !all_split) CU(h, cudaStreamWaitEvent(h->stream, stats_ready, 0));  // fused epilogues read the statistics
  const int ev0 = prof_mark(h);
  { int32_t rk = launch_k_gram<T>(h, (unsigned)grid, gp); if (rk) return rk; }
  h->launches++;
  const int ev1 = prof_mark(h);
  prof_span(h, PROF_GRAM, ev0, ev1);
  CU(h, cudaGetLastError());
  if (stats_ready && all_split) CU(h, cudaStreamWaitEvent(h->stream, stats_ready, 0));
  if (!pl.split_folds.empty()) {
    for (size_t s0 = 0; s0 < pl.split_folds.size(); s0 += 65535) {
      const unsigned ny = (unsigned)std::min<size_t>(65535, pl.split_folds.size() - s0);
      k_gram_reduce<T><<<dim3(ntiles, ny), GTHREADS, smem, h->stream>>>(gp, h->fold_units.as<int32_t>(),
                                                                          h->split_folds.as<int32_t>() + s0);
      h->launches++;
    }
    prof_span(h, PROF_REDUCE, ev1, prof_mark(h));
    CU(h, cudaGetLastError());
  }
  return CVMX_OK;
}

// Small folds (every fold of the batch has <= SMALL_MAX_ROWS rows): streaming rank-n kernel, no tensor cores.
template <typename T>
int32_t launch_small(cvmx_t* h, const int64_t* d_off, const int64_t* d_idx, const int64_t* off, int64_t f0, int64_t Pn, uint32_t want,
                     const EpiParams<T>& epi, cudaEvent_t stats_ready, bool loo_stats = false) {
  if (stats_ready) CU(h, cudaStreamWaitEvent(h->stream, stats_ready, 0));
  SmallParams<T> sp;
  sp.Z = h->Z.as<T>(); sp.w = h->w.as<T>(); sp.ld = h->ld;
  sp.offsets = d_off; sp.indices = d_idx; sp.fold0 = f0;
  sp.epi = epi;
  sp.quads = (int)((h->K + h->M + 3) / 4);
  int qpad = 1;
  while (qpad < sp.quads) qpad <<= 1;
  if (qpad > STHREADS) return fail(h, CVMX_ERR_INVALID, "small-fold path supports K + M <= 1024 per launch row");
  sp.rows_per_cta = STHREADS / qpad;
  const unsigned gx = (unsigned)((h->K + sp.rows_per_cta - 1) / sp.rows_per_cta);
  const int ev0 = prof_mark(h);
  for (int64_t c0 = 0; c0 < Pn; c0 += (int64_t)65535 * SMALL_FOLDS) {
    const int64_t nf = std::min<int64_t>(Pn - c0, (int64_t)65535 * SMALL_FOLDS);
    SmallParams<T> q = sp;
    q.fold0 = f0 + c0; q.nfolds = nf;
    q.epi.stats = epi.stats + (size_t)c0 * 2 * h->ld;
    q.epi.fs = epi.fs + c0;
    q.epi.out_xx = epi.out_xx ? epi.out_xx + (size_t)c0 * epi.xx_stride : nullptr;
    q.epi.out_xy = epi.out_xy ? epi.out_xy + (size_t)c0 * epi.xy_stride : nullptr;
    const dim3 grid(gx, (unsigned)((nf + SMALL_FOLDS - 1) / SMALL_FOLDS));
    bool loo = true;   // every fold of this launch has exactly one row -> specialised kernel
    for (int64_t f = f0 + c0; f < f0 + c0 + nf && loo; ++f) loo = (off[f + 1] - off[f]) == 1;
    if (loo && h->loo_mode == 0) {
      // streaming form: operand rows of every fold, then 32 x 128 output tiles streamed over the folds
      const int64_t pos0 = off[f0 + c0], ld = h->ld;
      CU(h, h->loo_ops.reserve((size_t)nf * 4 * ld * sizeof(double)));
      if (loo_stats) {   // one-row folds: means / stds inside the operand kernel (no separate statistics pass ran)
        MomentParams<T> mp;
        mp.Z = h->Z.as<T>(); mp.w = h->w.as<T>(); mp.ld = ld; mp.K = h->K; mp.M = h->M;
        mp.offsets = d_off; mp.indices = d_idx; mp.fold0 = 0; mp.N = h->N;   // offsets != nullptr: fold mode of finalize_column
        mp.flags = h->flags; mp.resolution = (T)h->resolution;
        mp.sum_z = h->sum_z.as<T>(); mp.sumsq_z = h->sumsq_z.as<T>();
        mp.fs = q.epi.fs; mp.pw_cols = nullptr; mp.stats = const_cast<T*>(q.epi.stats); mp.raw = nullptr;
        k_loo_operands<T, true><<<dim3((unsigned)nf, (unsigned)((ld + 127) / 128)), 128, 0, h->stream>>>(
            h->Z.as<T>(), h->w.as<T>(), ld, h->K, h->M, d_idx + pos0, q.epi.stats, q.epi.fs, h->flags & 15u, h->loo_ops.as<double>(), mp);
      } else {
        k_loo_operands<T><<<dim3((unsigned)nf, (unsigned)((ld + 127) / 128)), 128, 0, h->stream>>>(
            h->Z.as<T>(), h->w.as<T>(), ld, h->K, h->M, d_idx + pos0, q.epi.stats, q.epi.fs, h->flags & 15u, h->loo_ops.as<double>());
      }
      const int col_tiles = (int)((h->K + h->M + LOO_TC - 1) / LOO_TC), row_tiles = (int)((h->K + LOO_TR - 1) / LOO_TR);
      k_loo_tiles<T><<<dim3((unsigned)(col_tiles * row_tiles), (unsigned)((nf + LOO_FOLDS - 1) / LOO_FOLDS)), LOO_THREADS, 0, h->stream>>>(
          h->Ttot.as<T>(), h->loo_ops.as<double>(), ld, h->K, h->M, col_tiles, nf, want, q.epi.out_xx, q.epi.xx_pitch, q.epi.xx_stride,
          q.epi.out_xy, q.epi.xy_pitch, q.epi.xy_stride);
      h->launches++;
    } else if (loo) {
      const int64_t pos0 = off[f0 + c0];
      switch (h->flags & 15u) {
#define CVMX_LOO_CASE(F) case F: k_loo_folds<T, F><<<grid, STHREADS, 0, h->stream>>>(q, pos0); break;
        CVMX_LOO_CASE(0) CVMX_LOO_CASE(1) CVMX_LOO_CASE(2) CVMX_LOO_CASE(3) CVMX_LOO_CASE(4) CVMX_LOO_CASE(5) CVMX_LOO_CASE(6)
        CVMX_LOO_CASE(7) CVMX_LOO_CASE(8) CVMX_LOO_CASE(9) CVMX_LOO_CASE(10) CVMX_LOO_CASE(11) CVMX_LOO_CASE(12)
        CVMX_LOO_CASE(13) CVMX_LOO_CASE(14) CVMX_LOO_CASE(15)
#undef CVMX_LOO_CASE
      }
    } else if (h->loo_mode == 0) {
      // leave-few-out, streaming form: operand rows of every fold (bounded workspace: sub-batches), then the tile kernel
      const int64_t ld = h->ld;
      int R = 1;
      for (int64_t f = f0 + c0; f < f0 + c0 + nf; ++f) R = (int)std::max<int64_t>(R, off[f + 1] - off[f]);
      const size_t per_fold = (size_t)(3 + R) * ld * sizeof(double);
      const int64_t sub = std::max<int64_t>(LOO_FOLDS, (int64_t)(((size_t)512 << 20) / per_fold) / LOO_FOLDS * LOO_FOLDS);
      const int col_tiles = (int)((h->K + h->M + LOO_TC - 1) / LOO_TC), row_tiles = (int)((h->K + LOO_TR - 1) / LOO_TR);
      for (int64_t s0 = 0; s0 < nf; s0 += sub) {
        const int64_t ns = std::min(sub, nf - s0);
        CU(h, h->loo_ops.reserve((size_t)ns * per_fold));
        const int64_t* offs = d_off + f0 + c0 + s0;
        k_few_operands<T><<<dim3((unsigned)ns, (unsigned)((ld + 127) / 128)), 128, 0, h->stream>>>(
            h->Z.as<T>(), h->w.as<T>(), ld, h->K, h->M, offs, d_idx, q.epi.stats + (size_t)s0 * 2 * ld, q.epi.fs + s0, h->flags & 15u, R,
            h->loo_ops.as<double>());
        k_few_tiles<T><<<dim3((unsigned)(col_tiles * row_tiles), (unsigned)((ns + LOO_FOLDS - 1) / LOO_FOLDS)), LOO_THREADS, 0, h->stream>>>(
            h->Ttot.as<T>(), h->loo_ops.as<double>(), ld, h->K, h->M, col_tiles, ns, offs, q.epi.fs + s0, R, h->flags & 15u, want,
            q.epi.out_xx ? q.epi.out_xx + (size_t)s0 * q.epi.xx_stride : nullptr, q.epi.xx_pitch, q.epi.xx_stride,
            q.epi.out_xy ? q.epi.out_xy + (size_t)s0 * q.epi.xy_stride : nullptr, q.epi.xy_pitch, q.epi.xy_stride);
        h->launches += 2;
      }
      h->launches--;
    } else {
      k_small_folds<T><<<grid, STHREADS, 0, h->stream>>>(q);
    }
    h->launches++;
  }
  prof_span(h, PROF_GRAM, ev0, prof_mark(h));
  CU(h, cudaGetLastError());
  return CVMX_OK;
}

template <typename T>
int32_t launch_moments(cvmx_t* h, MomentParams<T> mp, int64_t nfolds, int64_t max_rows, int col_shard = 0, int n_col_shards = 1,
                       double overlap_ns = 1e30, const int* done_groups = nullptr, int done_groups_total = 0) {
  if (!h->attr_mom) {
    CU(h, cudaFuncSetAttribute(k_moments_pipe<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)moments_pipe_smem<T>(MOM_STAGES_DEEP)));
    h->attr_mom = true;
  }
  const bool pipe = max_rows >= 128;
  // few long chains (they overlap a loaded memory system): deep ring, one CTA per SM; many short chains: 4 stages so
  // that three CTAs share an SM
  {
    const int64_t groups0 = mp.ld / MOM_COLS;
    const int64_t mine0 = groups0 > col_shard ? (groups0 - col_shard + n_col_shards - 1) / n_col_shards : 0;
    mp.stages = (mine0 * nfolds <= 32 && max_rows >= 4096) ? MOM_STAGES_DEEP : MOM_STAGES;
  }
  const size_t smem = moments_pipe_smem<T>(mp.stages);
  // float64 chains go through the binade scan when that is faster AND the chains are not hidden anyway
  // (overlap_ns: device time of the work running beside them).  Cost model (measured, profiles/): a chain CTA
  // needs ~7.6 ns per row and 3 of them share an SM; both variants are bounded by HBM traffic (the scan reads the
  // rows twice, at ~5 TB/s) and the scan has ~0.15 ms of serial passes.  Groups the scan cannot handle fall
  // through to k_moments_pipe below.
  bool scan = false;
  const int64_t max_segs = round_up((max_rows + SCAN_L - 1) / SCAN_L, SCAN_PER_LANE);
  // done_groups: the binade scan already ran for this call (decoupled slab chain) - only the groups it gave up are left
  if (std::is_same<T, double>::value && pipe && !mp.ranges && !done_groups && h->scan_mode != 0 && max_rows < ((int64_t)1 << 25)) {
    const size_t seg_bytes = (size_t)std::min<int64_t>(65535, nfolds) * max_segs * 4 * mp.ld * sizeof(double);
    const int64_t groups0 = mp.ld / MOM_COLS;
    const int64_t mine0 = groups0 > col_shard ? (groups0 - col_shard + n_col_shards - 1) / n_col_shards : 0;
    const double ctas = (double)mine0 * (double)nfolds;
    const double bytes = ctas * (double)max_rows * MOM_COLS * sizeof(double);
    const double waves = std::ceil(ctas / (3.0 * h->sm_count));
    const double pipe_ns = std::max(7.6 * (double)max_rows * waves, bytes / 6000.0);
    const double scan_ns = 2.0 * bytes / 5000.0 + 150e3;
    scan = seg_bytes <= ((size_t)2 << 30) &&
           (h->scan_mode == 2 ? max_rows >= 4 * SCAN_L : (max_rows >= 8192 && scan_ns < pipe_ns && pipe_ns > 0.7 * overlap_ns));
  }
  for (int64_t f0 = 0; f0 < nfolds; f0 += 65535) {
    const unsigned ny = (unsigned)std::min<int64_t>(65535, nfolds - f0);
    MomentParams<T> q = mp;
    if (mp.ranges) q.ranges = mp.ranges + 2 * f0;
    if (mp.offsets || mp.ranges) {
      q.fold0 = mp.fold0 + f0;
      q.fs = mp.fs ? mp.fs + f0 : nullptr;
      q.pw_cols = mp.pw_cols ? mp.pw_cols + f0 * 4 : nullptr;
      q.stats = mp.stats ? mp.stats + (size_t)f0 * 2 * mp.ld : nullptr;
      q.raw = mp.raw ? mp.raw + (size_t)f0 * 2 * mp.ld : nullptr;
    }
    q.grp0 = col_shard; q.grp_stride = n_col_shards;
    if (done_groups) { q.scan_ok = done_groups + f0 * done_groups_total; q.scan_groups = done_groups_total; }
    const int64_t groups = pipe ? mp.ld / MOM_COLS : (mp.ld + 127) / 128;
    const int64_t mine = groups > col_shard ? (groups - col_shard + n_col_shards - 1) / n_col_shards : 0;
    if (mine == 0) continue;
    if constexpr (std::is_same<T, double>::value) {
      if (scan) {
        ScanParams sp;
        sp.p = q; sp.L = SCAN_L; sp.max_segs = max_segs; sp.groups_total = (int)groups;
        CU(h, h->scan_seg.reserve((size_t)ny * max_segs * 4 * mp.ld * sizeof(double)));
        CU(h, h->scan_ok.reserve((size_t)ny * groups * sizeof(int)));
        sp.slow_cap = (int)(max_segs / 4 + 2);
        CU(h, h->scan_list.reserve((size_t)ny * 2 * sp.slow_cap * mp.ld * sizeof(int)));
        CU(h, h->scan_cnt.reserve((size_t)ny * 2 * mp.ld * sizeof(int)));
        sp.seg = h->scan_seg.as<double>(); sp.ok = h->scan_ok.as<int>();
        sp.slow_list = h->scan_list.as<int>(); sp.slow_cnt = h->scan_cnt.as<int>();
        // (measured: capping the streaming grids to a few SMs' worth of CTAs and fatter chain CTAs while a Gram kernel
        // owns the GPU does not change the step time - the passes cost the same SM time either way)
        const int64_t quads = (max_segs + SCAN_WARPS - 1) / SCAN_WARPS;
        const dim3 gseg((unsigned)mine, (unsigned)quads, ny);
        // fold statistics of a fitted model: the totals predict every segment's binade, so passes 1 and 3 share ONE
        // read of the rows (k_scan_spec) and the prefix pass verifies the guess; fit itself has no totals yet
        const bool spec = h->scan_spec && q.offsets && !q.accumulate && h->fitted;
        if (spec) {
          CU(h, h->scan_look.reserve((size_t)ny * 2 * 3 * mp.ld * max_segs * sizeof(double)));
          k_scan_spec<<<gseg, 32 * SCAN_WARPS, 0, h->stream>>>(sp, h->scan_look.as<double>());
          k_scan_prefix<true><<<dim3((unsigned)(mine * SCAN_PREFIX_CTAS), ny), SCAN_PREFIX_THREADS, 0, h->stream>>>(sp, h->scan_look.as<double>());
          h->launches -= 1;
        } else {
          k_scan_segsums<<<gseg, 32 * SCAN_WARPS, 0, h->stream>>>(sp);
          k_scan_prefix<false><<<dim3((unsigned)(mine * SCAN_PREFIX_CTAS), ny), SCAN_PREFIX_THREADS, 0, h->stream>>>(sp, nullptr);
          k_scan_delta<<<gseg, 32 * SCAN_WARPS, 0, h->stream>>>(sp);
        }
        k_scan_chain<2><<<dim3((unsigned)(mine * (SCAN_COLS / 2)), ny), 64 * 2, scan_chain_smem<2>(), h->stream>>>(sp);
        h->launches += 4; h->scan_launches += 1;
        q.scan_ok = sp.ok; q.scan_groups = sp.groups_total;
      }
    }
    if (pipe) k_moments_pipe<T><<<dim3((unsigned)mine, ny), MOM_THREADS, smem, h->stream>>>(q);
    else k_moments_direct<T><<<dim3((unsigned)mine, ny), 128, 0, h->stream>>>(q);
    h->launches++;
  }
  CU(h, cudaGetLastError());
  return CVMX_OK;
}

// Fork the statistics work onto the side stream (ordered after everything already queued on the main stream);
// join_stats() returns the event the consumer of the statistics has to wait for.
int32_t fork_stats(cvmx_t* h, cudaStream_t* saved) {
  CU(h, cudaEventRecord(h->ev_fork, h->stream));
  CU(h, cudaStreamWaitEvent(h->aux_stream, h->ev_fork, 0));
  *saved = h->stream;
  h->stream = h->aux_stream;
  return CVMX_OK;
}
int32_t join_stats(cvmx_t* h, cudaStream_t saved) {
  cudaError_t e = cudaEventRecord(h->ev_join, h->aux_stream);
  h->stream = saved;
  CU(h, e);
  return CVMX_OK;
}

// Statistics of folds [f0, f0 + Pn): weight masses (side stream 2) and moment chains (current stream) run
// concurrently - the chains store raw sums - and k_finalize_stats turns them into means / stds once both are done.
template <typename T>
int32_t launch_fold_stats(cvmx_t* h, const int64_t* d_off, const int64_t* d_idx, int64_t f0, int64_t Pn, int64_t max_rows,
                          int col_shard, int n_col_shards, double overlap_ns, const T* have_raw = nullptr, bool masses_only = false) {
  const size_t sz = sizeof(T);
  const int64_t ld = h->ld;
  CU(h, h->fscal.reserve(Pn * sizeof(FoldScalars)));
  CU(h, h->stats.reserve((size_t)Pn * 2 * ld * sz));
  CU(h, h->rawsums.reserve((size_t)Pn * 2 * ld * sz));
  CU(h, h->pwcols.reserve((size_t)Pn * 4 * sz));
  CU(h, cudaMemsetAsync(h->stats.p, 0, (size_t)Pn * 2 * ld * sz, h->stream));
  CU(h, cudaMemsetAsync(h->fscal.p, 0, Pn * sizeof(FoldScalars), h->stream));
  if (h->flags == 0) return CVMX_OK;
  const int ev0 = prof_mark(h);
  // weight masses on side stream 2 (ordered after the memsets above)
  CU(h, cudaEventRecord(h->ev_mass, h->stream));
  CU(h, cudaStreamWaitEvent(h->aux2_stream, h->ev_mass, 0));
  // row-slab mode: the weight sums run over the GLOBAL weight vector and validation sets (numpy's pairwise tree cannot
  // be cut at slab boundaries); K, M >= 2 there, so the kernel never touches Z
  const T* wm_w = h->slab ? h->w_glob.as<T>() : h->w.as<T>();
  const int64_t* wm_off = h->slab ? h->g_off.as<int64_t>() : d_off;
  const int64_t* wm_idx = h->slab ? h->g_idx.as<int64_t>() : d_idx;
  const int64_t wm_N = h->slab ? h->N_glob : h->N;
  int64_t wm_rows = max_rows;
  if (h->slab) for (int64_t f = f0; f < f0 + Pn; ++f) wm_rows = std::max(wm_rows, h->g_h_off[f + 1] - h->g_h_off[f]);
  for (int64_t c0 = 0; c0 < Pn; c0 += 0x7fffffff) {
    const int64_t nb = std::min<int64_t>(0x7fffffff, Pn - c0);
    if (wm_rows <= 1024)
      k_weight_mass<T, PW_LEVELS_SMALL><<<(unsigned)nb, 1 << PW_LEVELS_SMALL, 0, h->aux2_stream>>>(
          h->Z.as<T>(), wm_w, ld, wm_N, h->K, h->M, h->weighted ? 1 : 0, wm_off, wm_idx, f0 + c0, 0, h->ddof,
          h->fit_scal.as<FitScalars>(), h->fscal.as<FoldScalars>() + c0, h->pwcols.as<T>() + 4 * c0);
    else
      k_weight_mass<T, PW_LEVELS_BIG><<<(unsigned)nb, 1 << PW_LEVELS_BIG, 0, h->aux2_stream>>>(
          h->Z.as<T>(), wm_w, ld, wm_N, h->K, h->M, h->weighted ? 1 : 0, wm_off, wm_idx, f0 + c0, 0, h->ddof,
          h->fit_scal.as<FitScalars>(), h->fscal.as<FoldScalars>() + c0, h->pwcols.as<T>() + 4 * c0);
    h->launches++;
  }
  CU(h, cudaGetLastError());
  CU(h, cudaEventRecord(h->ev_mass, h->aux2_stream));
  if (masses_only) {   // the column sums, means and stds are evaluated inside the Gram kernel (GramParams::fuse_stats)
    CU(h, cudaStreamWaitEvent(h->stream, h->ev_mass, 0));
    prof_span(h, PROF_STATS, ev0, prof_mark(h));
    return CVMX_OK;
  }
  MomentParams<T> mp;
  mp.Z = h->Z.as<T>(); mp.w = h->w.as<T>(); mp.ld = ld; mp.K = h->K; mp.M = h->M;
  mp.offsets = d_off; mp.indices = d_idx; mp.fold0 = f0; mp.N = h->N;
  mp.flags = h->flags; mp.resolution = (T)h->resolution;
  mp.sum_z = h->sum_z.as<T>(); mp.sumsq_z = h->sumsq_z.as<T>();
  mp.fs = h->fscal.as<FoldScalars>(); mp.pw_cols = h->pwcols.as<T>(); mp.stats = h->stats.as<T>();
  mp.raw = have_raw ? const_cast<T*>(have_raw) : h->rawsums.as<T>();
  if (!have_raw) {   // (have_raw: the fold sums were accumulated chunk by chunk during cvmx_fit_folds)
    int32_t rc = launch_moments<T>(h, mp, Pn, max_rows, col_shard, n_col_shards, overlap_ns);
    if (rc) return rc;
  }
  CU(h, cudaStreamWaitEvent(h->stream, h->ev_mass, 0));
  mp.grp0 = 0; mp.grp_stride = 1;
  if (n_col_shards > 1) {
    // only this shard's column groups hold sums; the others must stay zero for the all-reduce
    // (group width of the kernel that produced them)
  }
  for (int64_t c0 = 0; c0 < Pn; c0 += 65535) {
    const unsigned ny = (unsigned)std::min<int64_t>(65535, Pn - c0);
    MomentParams<T> q = mp;
    q.fs = mp.fs + c0; q.pw_cols = mp.pw_cols + c0 * 4; q.stats = mp.stats + (size_t)c0 * 2 * ld; q.raw = mp.raw + (size_t)c0 * 2 * ld;
    q.grp0 = col_shard; q.grp_stride = n_col_shards;
    q.stages = (max_rows >= 128) ? MOM_COLS : 128;   // reused as "columns per group" by k_finalize_stats
    k_finalize_stats<T><<<dim3((unsigned)((ld + 127) / 128), ny), 128, 0, h->stream>>>(q, (int64_t)ny);
    h->launches++;
  }
  CU(h, cudaGetLastError());
  prof_span(h, PROF_STATS, ev0, prof_mark(h));
  return CVMX_OK;
}

template <typename T>
__global__ void k_pack_scalars(const FoldScalars* __restrict__ fs, int64_t n, T* __restrict__ scal, int32_t* __restrict__ status) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (scal) { scal[2 * i] = (T)fs[i].sw; scal[2 * i + 1] = (T)fs[i].nz; }
  if (status) status[i] = fs[i].status;
}

// ---- fit -------------------------------------------------------------------------------------------
int32_t upload_csr(cvmx_t* h, DevBuf& doff, DevBuf& didx, const int64_t* offsets, const int64_t* indices, int64_t P,
                   int64_t nidx, int32_t mem);

// Host CSR of a TRUE partition of the rows (every row in exactly one fold, indices ascending inside a fold): then
// XtWX = sum over folds of the fold Grams, so fit can contract every row once, per fold, and keep the fold Grams.
struct FoldFuse { const int64_t* off; const int64_t* idx; int64_t P; };

template <typename T>
int32_t fit_impl(cvmx_t* h, const void* X, int64_t N, int64_t K, int64_t ldx, const void* Y, int64_t M, int64_t ldy,
                 const void* w, int32_t mem, int64_t g0, int64_t g1, const FoldFuse* ff = nullptr) {
  const size_t sz = sizeof(T);
  const int64_t ld = round_up(K + M, 32);
  h->fitted = false; h->filling = false; h->slab = false;
  choose_fmap<T>(h, K, M);
  h->N = N; h->K = K; h->M = M; h->ld = ld; h->weighted = w != nullptr;
  h->P = 0; h->csr_version++; h->plan = Plan();
  CU(h, h->Z.reserve((size_t)std::max<int64_t>(N, 1) * ld * sz));
  CU(h, h->w.reserve((size_t)std::max<int64_t>(N, 1) * sz));
  CU(h, h->Ttot.reserve((size_t)K * ld * sz));
  CU(h, h->sum_z.reserve(ld * sz));
  CU(h, h->sumsq_z.reserve(ld * sz));
  CU(h, h->fit_scal.reserve(sizeof(FitScalars)));
  const cudaMemcpyKind kind = mem == CVMX_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
  T* Z = h->Z.as<T>();
  // Large host matrix: a pitch-changing 2-D copy makes the DMA engine move 4000-byte rows one by one (~20 GB/s from
  // pinned memory, measured).  Instead stream contiguous chunks into two staging buffers on a copy stream (full PCIe
  // rate), re-pitch each into Z with a kernel, and run the chunk's share of the Gram pass and of the moment chains
  // right behind it, so that fit costs little more than the host->device copy.
  const bool chunked = N > 0 && mem == CVMX_HOST && ldx == K && K > 1 && (size_t)N * K * sz >= ((size_t)64 << 20);
  // a pitch-changing 2-D copy of a narrow matrix (Y: 80-byte rows) is one DMA descriptor per row - ~20 ms for 1M rows -
  // so in the chunked path Y is copied contiguously into a scratch buffer and re-pitched by a kernel
  const bool stage_y = chunked && M > 0 && ldy == M;
  if (N > 0) {
    if (ld > K + M) {
      if (chunked) { k_zero_pad<T><<<h->sm_count * 4, 256, 0, h->stream>>>(Z, N, ld, K + M); h->launches++; }
      else CU(h, cudaMemset2DAsync(Z + (K + M), ld * sz, 0, (ld - K - M) * sz, N, h->stream));
    }
    if (!chunked) CU(h, cudaMemcpy2DAsync(Z, ld * sz, X, ldx * sz, K * sz, N, kind, h->stream));
    if (M > 0 && !stage_y) CU(h, cudaMemcpy2DAsync(Z + K, ld * sz, Y, ldy * sz, M * sz, N, kind, h->stream));
    if (stage_y) {
      CU(h, h->out_xy.reserve((size_t)N * M * sz));   // scratch (reused by host-output fold batches later)
      CU(h, h2d_copy(h, h->out_xy.p, Y, (size_t)N * M * sz, h->stream, HostStager::pageable(Y)));
      k_repack<T><<<h->sm_count * 4, 256, 0, h->stream>>>(h->out_xy.as<T>(), N, M, Z + K, ld);
      h->launches++;
    }
    if (w && mem == CVMX_HOST) CU(h, h2d_copy(h, h->w.p, w, N * sz, h->stream, HostStager::pageable(w)));
    else if (w) CU(h, cudaMemcpyAsync(h->w.p, w, N * sz, kind, h->stream));
    else { k_fill<T><<<(unsigned)((N + 255) / 256), 256, 0, h->stream>>>(h->w.as<T>(), N, T(1)); h->launches++; }
  }
  CU(h, cudaMemsetAsync(h->Ttot.p, 0, (size_t)K * ld * sz, h->stream));
  CU(h, cudaMemsetAsync(h->sum_z.p, 0, ld * sz, h->stream));
  CU(h, cudaMemsetAsync(h->sumsq_z.p, 0, ld * sz, h->stream));
  CU(h, h->pwcols.reserve(4 * sz));

  MomentParams<T> mp;
  mp.Z = Z; mp.w = h->w.as<T>(); mp.ld = ld; mp.K = K; mp.M = M;
  mp.offsets = nullptr; mp.indices = nullptr; mp.fold0 = 0; mp.N = N;
  mp.flags = h->flags; mp.resolution = (T)h->resolution;
  mp.sum_z = h->sum_z.as<T>(); mp.sumsq_z = h->sumsq_z.as<T>();
  mp.fs = nullptr; mp.pw_cols = h->pwcols.as<T>(); mp.stats = nullptr;

  Plan pl;
  plan_tiles(h, (uint32_t)(CVMX_WANT_XTX | (M > 0 ? CVMX_WANT_XTY : 0)), pl.tiles);
  EpiParams<T> epi;
  epi.mode = 0; epi.flags = 0; epi.want = CVMX_WANT_XTX | CVMX_WANT_XTY;
  epi.K = K; epi.M = M; epi.ld = ld;
  epi.Ttot = nullptr; epi.stats = nullptr; epi.fs = nullptr;
  epi.out_xx = h->Ttot.as<T>(); epi.xx_pitch = ld; epi.xx_stride = 0;
  epi.out_xy = h->Ttot.as<T>() + K; epi.xy_pitch = ld; epi.xy_stride = 0;

  // statistics run on the side stream (moment chains: ~15 cycles per row and column, unsplittable by rows)
  cudaStream_t main_stream;
  int32_t rc0 = fork_stats(h, &main_stream);
  if (rc0) return rc0;
  k_weight_mass<T, PW_LEVELS_BIG><<<1, 1 << PW_LEVELS_BIG, 0, h->stream>>>(Z, h->w.as<T>(), ld, N, K, M, h->weighted ? 1 : 0, nullptr, nullptr, 0, 1,
                                                   h->ddof, h->fit_scal.as<FitScalars>(), nullptr, h->pwcols.as<T>());
  h->launches++;
  int32_t rc = CVMX_OK;
  if (!chunked) {
    // the Gram pass that runs beside the chains: ~2 (g1 - g0) K (K + M) flops at ~40 TFLOP/s
    rc = launch_moments<T>(h, mp, 1, N, 0, 1, 2.0 * (double)(g1 - g0) * (double)K * (double)(K + M) / 4e4);
    if (rc) { h->stream = main_stream; return rc; }
    rc = join_stats(h, main_stream);
    if (rc) return rc;
    // totals: Gram over the row slab [g0, g1) with identity indexing, raw epilogue into Ttot
    const int64_t off[2] = {g0, g1};
    plan_units(h, off, 0, 1, (int)pl.tiles.size(), pl);
    if (g1 > g0) {
      rc = launch_gram<T>(h, pl, nullptr, epi);
      if (rc) return rc;
    }
  } else {
    cudaStream_t stats_stream = h->stream;   // side stream (fork_stats made it current)
    h->stream = main_stream;
    const int ntiles = (int)pl.tiles.size();
    const int64_t chunk_rows = std::max<int64_t>(GBK, (int64_t)(((size_t)128 << 20) / ((size_t)K * sz)) / GBK * GBK);
    const int64_t unit_rows = 2816;          // ~176 stages per Gram CTA
    // units of every chunk (clipped to the Gram slab [g0, g1)), numbered globally: one fold with `total` splits
    std::vector<int64_t> chunk_unit0;
    // fused fit + folds: the rows of a chunk are contracted fold by fold (CSR position ranges, gathered through the
    // device CSR); partial slots are numbered fold-major so that one pass sums them per fold
    bool fused = ff != nullptr && g0 == 0 && g1 == N && ff->P > 0;
    std::vector<int64_t> fold_base, fold_n;
    std::vector<int64_t> h_ranges;      // [chunk][fold][2]: CSR positions of the fold's rows inside the chunk
    std::vector<int64_t> chunk_fold_rows;   // [chunk]: longest fold slice
    if (fused) {
      const int64_t P = ff->P;
      struct Piece { int64_t lo, hi; int32_t fold; };
      std::vector<std::vector<Piece>> per_chunk;
      fold_n.assign(P, 0);
      for (int64_t r0 = 0; r0 < N; r0 += chunk_rows) {
        const int64_t r1 = std::min(r0 + chunk_rows, N);
        per_chunk.emplace_back();
        for (int64_t f = 0; f < P; ++f) {
          const int64_t* b = ff->idx + ff->off[f];
          const int64_t* e = ff->idx + ff->off[f + 1];
          const int64_t lo = std::lower_bound(b, e, r0) - ff->idx, hi = std::lower_bound(b, e, r1) - ff->idx;
          const int64_t n = hi - lo;
          h_ranges.push_back(lo); h_ranges.push_back(hi);
          if (f == 0) chunk_fold_rows.push_back(0);
          chunk_fold_rows.back() = std::max(chunk_fold_rows.back(), n);
          if (n <= 0) continue;
          const int64_t ns = (n + unit_rows - 1) / unit_rows, per = round_up((n + ns - 1) / ns, GBK);
          for (int64_t s2 = 0; s2 < ns; ++s2) {
            const int64_t a = lo + std::min(n, s2 * per), z = lo + std::min(n, (s2 + 1) * per);
            if (z > a) { per_chunk.back().push_back({a, z, (int32_t)f}); fold_n[f]++; }
          }
        }
      }
      int64_t tot = 0;
      fold_base.assign(P, 0);
      for (int64_t f = 0; f < P; ++f) { fold_base[f] = tot; tot += fold_n[f]; if (fold_n[f] == 0) fused = false; }
      if ((size_t)(tot + P) * ntiles * GACC * GTHREADS * sizeof(double) > ((size_t)2 << 30)) fused = false;   // many small folds: not worth it
      if (fused) {
        std::vector<int64_t> next(fold_base);
        for (auto& pieces : per_chunk) {
          chunk_unit0.push_back((int64_t)pl.units.size());
          for (auto& pc : pieces) {
            GramUnit u;
            u.row_begin = pc.lo; u.row_end = pc.hi; u.fold = pc.fold; u.split = (int32_t)next[pc.fold]++; u.nsplit = 0; u.part_base = 0;
            pl.units.push_back(u);
          }
        }
      }
    }
    if (fused) {
      int32_t rcu = upload_csr(h, h->d_off, h->d_idx, ff->off, ff->idx, ff->P, ff->off[ff->P], CVMX_HOST);
      if (rcu) { h->stream = main_stream; return rcu; }
    } else {
      for (int64_t r0 = 0; r0 < N; r0 += chunk_rows) {
        chunk_unit0.push_back((int64_t)pl.units.size());
        const int64_t a0 = std::max(r0, g0), a1 = std::min(std::min(r0 + chunk_rows, N), g1);
        for (int64_t u0 = a0; u0 < a1; u0 += unit_rows) {
          GramUnit u;
          u.row_begin = u0; u.row_end = std::min(a1, u0 + unit_rows);
          u.fold = 0; u.split = (int32_t)pl.units.size(); u.nsplit = 0; u.part_base = 0;
          pl.units.push_back(u);
        }
      }
    }
    chunk_unit0.push_back((int64_t)pl.units.size());
    // wide K: one partial per 2816 rows x ntiles tiles would not fit (K = 5000: 107 MB per unit) - then the Gram pass
    // runs after the upload with longer units instead of chunk by chunk
    const bool pipeline_gram = (size_t)pl.units.size() * ntiles * GACC * GTHREADS * sizeof(double) <= ((size_t)2 << 30);
    if (!pipeline_gram) { pl.units.clear(); for (auto& u0 : chunk_unit0) u0 = 0; fused = false; }
    const int32_t total = (int32_t)pl.units.size();
    for (auto& u : pl.units) u.nsplit = total;                // force_partials: always the partial + reduce path
    pl.fold_units.assign(1, 0);
    pl.split_folds.assign(1, 0);
    std::vector<int32_t> h_fold_units(1, 0);
    if (fused) {
      // virtual units: [total + f] = fold f's slots; [total + P] = the P per-fold sums (-> totals)
      const int64_t P = ff->P;
      h_fold_units.assign(P + 1, 0);
      for (int64_t f = 0; f <= P; ++f) {
        GramUnit v;
        v.row_begin = v.row_end = 0; v.split = 0;
        v.fold = f < P ? (int32_t)f : 0; v.part_base = f < P ? (int32_t)fold_base[f] : 0; v.nsplit = f < P ? (int32_t)fold_n[f] : (int32_t)P;
        h_fold_units[f] = (int32_t)pl.units.size();
        pl.units.push_back(v);
      }
      CU(h, h->fold_gram.reserve((size_t)P * ntiles * GACC * GTHREADS * sizeof(double)));
      // the folds' own column sums (numpy order = CSR order inside a fold) are continued chunk by chunk as well
      CU(h, h->fold_raw.reserve((size_t)P * 2 * ld * sz));
      CU(h, h->chunk_ranges.reserve(h_ranges.size() * sizeof(int64_t)));
      CU(h, cudaMemsetAsync(h->fold_raw.p, 0, (size_t)P * 2 * ld * sz, h->stream));
      CU(h, cudaMemcpyAsync(h->chunk_ranges.p, h_ranges.data(), h_ranges.size() * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    }
    GramParams<T> gp;
    gp.fmap = fmap_of<T>(h);
    gp.Z = Z; gp.w = h->w.as<T>(); gp.ld = ld; gp.indices = fused ? h->d_idx.as<int64_t>() : nullptr;
    gp.ntiles = ntiles; gp.raw_out = nullptr; gp.force_partials = 1; gp.epi = epi;
    const size_t smem = gram_smem_bytes<T>();
    if (total > 0) {
      CU(h, h->units.reserve(pl.units.size() * sizeof(GramUnit)));
      CU(h, h->tiles.reserve(pl.tiles.size() * sizeof(int2)));
      CU(h, h->fold_units.reserve(h_fold_units.size() * sizeof(int32_t)));
      CU(h, h->split_folds.reserve(sizeof(int32_t)));
      CU(h, h->partials.reserve((size_t)total * ntiles * GACC * GTHREADS * sizeof(double)));
      CU(h, cudaMemcpyAsync(h->units.p, pl.units.data(), pl.units.size() * sizeof(GramUnit), cudaMemcpyHostToDevice, h->stream));
      CU(h, cudaMemcpyAsync(h->tiles.p, pl.tiles.data(), pl.tiles.size() * sizeof(int2), cudaMemcpyHostToDevice, h->stream));
      CU(h, cudaMemcpyAsync(h->fold_units.p, h_fold_units.data(), h_fold_units.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
      CU(h, cudaMemsetAsync(h->split_folds.p, 0, sizeof(int32_t), h->stream));
      if (!h->attr_gram) {
        CU(h, cudaFuncSetAttribute(k_gram<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CU(h, cudaFuncSetAttribute(k_gram_reduce<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        h->attr_gram = true;
      }
    }
    gp.tiles = h->tiles.as<int2>(); gp.partials = h->partials.as<double>();
    CU(h, h->stage[0].reserve((size_t)chunk_rows * K * sz));
    CU(h, h->stage[1].reserve((size_t)chunk_rows * K * sz));
    CU(h, cudaEventRecord(h->ev_mass, h->stream));                    // Y, w, pad and the unit table are queued
    CU(h, cudaStreamWaitEvent(h->aux2_stream, h->ev_mass, 0));
    const bool x_pageable = HostStager::pageable(X);
    int c = 0;
    for (int64_t r0 = 0; r0 < N; r0 += chunk_rows, ++c) {
      const int64_t nr = std::min(chunk_rows, N - r0);
      const int b = c & 1;
      if (c >= 2) CU(h, cudaStreamWaitEvent(h->aux2_stream, h->ev_stage[b], 0));       // staging buffer free again
      CU(h, h2d_copy(h, h->stage[b].p, (const char*)X + (size_t)r0 * K * sz, (size_t)nr * K * sz, h->aux2_stream, x_pageable));
      CU(h, cudaEventRecord(h->ev_copied[b], h->aux2_stream));
      CU(h, cudaStreamWaitEvent(h->stream, h->ev_copied[b], 0));
      k_repack<T><<<h->sm_count * 8, 256, 0, h->stream>>>(h->stage[b].as<T>(), nr, K, Z + r0 * ld, ld);
      h->launches++;

      CU(h, cudaEventRecord(h->ev_stage[b], h->stream));
      // the chunk's rows of the moment chains, continuing the accumulators of the previous chunk
      CU(h, cudaStreamWaitEvent(stats_stream, h->ev_stage[b], 0));
      MomentParams<T> mc = mp;
      mc.row0 = r0; mc.N = nr; mc.accumulate = c > 0;
      h->stream = stats_stream;
      rc = launch_moments<T>(h, mc, 1, nr);
      if (!rc && fused && h->flags != 0) {
        MomentParams<T> fc = mp;
        fc.ranges = h->chunk_ranges.as<int64_t>() + (size_t)c * ff->P * 2;
        fc.indices = h->d_idx.as<int64_t>();
        fc.raw = h->fold_raw.as<T>(); fc.accumulate = 1;
        fc.pw_cols = nullptr;
        rc = launch_moments<T>(h, fc, ff->P, chunk_fold_rows[c]);
      }
      h->stream = main_stream;
      if (rc) return rc;
      // the chunk's Gram partials
      const int64_t nu = chunk_unit0[c + 1] - chunk_unit0[c];
      if (nu > 0) {
        gp.units = h->units.as<GramUnit>() + chunk_unit0[c];
        const int ev0 = prof_mark(h);
        { int32_t rk = launch_k_gram<T>(h, (unsigned)(nu * ntiles), gp); if (rk) return rk; }
        h->launches++;
        prof_span(h, PROF_GRAM, ev0, prof_mark(h));
      }
    }
    CU(h, cudaGetLastError());
    if (total > 0 && fused) {
      // per-fold sums of the partial slots (kept: cvmx_training_batch finishes the folds from them), then totals =
      // sum over folds
      gp.units = h->units.as<GramUnit>();
      k_partial_sum<<<dim3((unsigned)(GACC * GTHREADS / 512), (unsigned)ntiles, (unsigned)ff->P), 256, 0, h->stream>>>(
          h->partials.as<double>(), h->units.as<GramUnit>(), h->fold_units.as<int32_t>(), ntiles, h->fold_gram.as<double>());
      gp.partials = h->fold_gram.as<double>();
      k_gram_reduce<T><<<dim3(ntiles, 1), GTHREADS, smem, h->stream>>>(gp, h->fold_units.as<int32_t>() + ff->P, h->split_folds.as<int32_t>());
      h->launches += 2;
      CU(h, cudaGetLastError());
    } else if (total > 0) {
      gp.units = h->units.as<GramUnit>();
      k_gram_reduce<T><<<dim3(ntiles, 1), GTHREADS, smem, h->stream>>>(gp, h->fold_units.as<int32_t>(), h->split_folds.as<int32_t>());
      h->launches++;
      CU(h, cudaGetLastError());
    }
    if (fused && total > 0) {
      h->P = ff->P;
      h->h_off.assign(ff->off, ff->off + ff->P + 1);
      h->fold_gram_version = h->csr_version;
    }
    CU(h, cudaEventRecord(h->ev_join, stats_stream));
    if (!pipeline_gram && g1 > g0) {
      Plan pg;
      pg.tiles = pl.tiles;
      const int64_t off[2] = {g0, g1};
      plan_units(h, off, 0, 1, ntiles, pg);
      rc = launch_gram<T>(h, pg, nullptr, epi);
      if (rc) return rc;
    }
  }
  CU(h, cudaStreamWaitEvent(h->stream, h->ev_join, 0));
  FitScalars fsc;
  CU(h, cudaMemcpyAsync(&fsc, h->fit_scal.p, sizeof(fsc), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaStreamSynchronize(h->stream));
  if (fsc.neg_weight) return fail(h, CVMX_ERR_NEG_WEIGHT, "Weights must be non-negative.");
  h->fitted = true;
  return CVMX_OK;
}


// ---- streaming / sharded fit -------------------------------------------------------------------------------
// cvmx_fit in pieces: the caller feeds row blocks (host or device memory, any order, possibly only a slab of the
// rows - the rest may arrive from peer GPUs over NVLink, written straight into cvmx_data_ptr()), each block's
// weighted Gram is folded into a float64 accumulator in fragment layout (partial slot 0), and cvmx_fit_end turns
// the accumulator into the totals and runs the numpy-order statistics over all N rows.
int64_t fill_units_for(const cvmx_t* h, int64_t rows, int ntiles) {
  const int64_t by_ws = std::max<int64_t>(1, (int64_t)(((size_t)2 << 30) / ((size_t)std::max(ntiles, 1) * GACC * GTHREADS * sizeof(double))) - 1);
  int64_t nu = std::max<int64_t>(1, (rows + 2815) / 2816);
  // wide K: the tiles alone fill the GPU; keep the units long
  if ((int64_t)ntiles >= h->sm_count) nu = std::max<int64_t>(1, std::min<int64_t>(nu, (rows + 16383) / 16384 * 2));
  return std::min(nu, by_ws);
}

template <typename T>
int32_t fit_begin_impl(cvmx_t* h, int64_t N, int64_t K, int64_t M, int32_t weighted, int64_t max_block_rows) {
  const size_t sz = sizeof(T);
  const int64_t ld = round_up(K + M, 32);
  h->fitted = false; h->filling = false; h->slab = false;
  choose_fmap<T>(h, K, M);
  h->N = N; h->K = K; h->M = M; h->ld = ld; h->weighted = weighted != 0;
  h->P = 0; h->csr_version++; h->plan = Plan();
  CU(h, h->Z.reserve((size_t)std::max<int64_t>(N, 1) * ld * sz));
  CU(h, h->w.reserve((size_t)std::max<int64_t>(N, 1) * sz));
  CU(h, h->Ttot.reserve((size_t)K * ld * sz));
  CU(h, h->sum_z.reserve(ld * sz));
  CU(h, h->sumsq_z.reserve(ld * sz));
  CU(h, h->fit_scal.reserve(sizeof(FitScalars)));
  CU(h, h->pwcols.reserve(4 * sz));
  std::vector<int2> tiles;
  plan_tiles(h, (uint32_t)(CVMX_WANT_XTX | (M > 0 ? CVMX_WANT_XTY : 0)), tiles);
  const int ntiles = (int)tiles.size();
  h->fill_units_cap = fill_units_for(h, std::max<int64_t>(max_block_rows, 1), ntiles);
  const size_t slot = (size_t)ntiles * GACC * GTHREADS * sizeof(double);
  CU(h, h->partials.reserve((size_t)(h->fill_units_cap + 1) * slot));
  CU(h, h->tiles.reserve(tiles.size() * sizeof(int2)));
  CU(h, h->units.reserve((size_t)(h->fill_units_cap + 1) * sizeof(GramUnit)));
  CU(h, h->fold_units.reserve(sizeof(int32_t)));
  CU(h, h->split_folds.reserve(sizeof(int32_t)));
  CU(h, cudaMemcpyAsync(h->tiles.p, tiles.data(), tiles.size() * sizeof(int2), cudaMemcpyHostToDevice, h->stream));
  CU(h, cudaMemsetAsync(h->partials.p, 0, slot, h->stream));                  // the accumulator
  CU(h, cudaMemsetAsync(h->fold_units.p, 0, sizeof(int32_t), h->stream));
  CU(h, cudaMemsetAsync(h->split_folds.p, 0, sizeof(int32_t), h->stream));
  CU(h, cudaMemsetAsync(h->Ttot.p, 0, (size_t)K * ld * sz, h->stream));
  CU(h, cudaMemsetAsync(h->sum_z.p, 0, ld * sz, h->stream));
  CU(h, cudaMemsetAsync(h->sumsq_z.p, 0, ld * sz, h->stream));
  h->mass_started = h->mass_pending = h->fit_pre_done = false; h->slab_scan_mode = h->slab_scan_stage = 0;
  if (!weighted && N > 0) { k_fill<T><<<(unsigned)((N + 255) / 256), 256, 0, h->stream>>>(h->w.as<T>(), N, T(1)); h->launches++; }
  const size_t smem = gram_smem_bytes<T>();
  if (!h->attr_gram) {
    CU(h, cudaFuncSetAttribute(k_gram<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CU(h, cudaFuncSetAttribute(k_gram_reduce<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    h->attr_gram = true;
  }
  CU(h, cudaStreamSynchronize(h->stream));   // `tiles` is a local
  h->filling = true; h->fill_calls = 0;
  return CVMX_OK;
}

template <typename T>
int32_t fit_rows_impl(cvmx_t* h, int64_t row0, int64_t nr, const void* X, int64_t ldx, const void* Y, int64_t ldy, const void* w,
                      int32_t mem, int32_t gram) {
  const size_t sz = sizeof(T);
  const int64_t K = h->K, M = h->M, ld = h->ld;
  T* Zb = h->Z.as<T>() + (size_t)row0 * ld;
  const int cb = (int)(h->fill_calls & 1);
  h->fill_calls++;
  if (ld > K + M) { k_zero_pad<T><<<h->sm_count * 4, 256, 0, h->stream>>>(Zb, nr, ld, K + M); h->launches++; }
  if (mem == CVMX_HOST) {
    // contiguous copies at full PCIe rate into a staging buffer on the copy stream (they overlap the Gram of the
    // previous block on the main stream), re-pitched into Z by a kernel; strided inputs fall back to 2-D copies
    const bool cx = ldx == K, cy = M > 0 && ldy == M;
    const size_t xb = cx ? (size_t)nr * K * sz : 0, yb = cy ? (size_t)nr * M * sz : 0;
    CU(h, h->stage[cb].reserve(std::max<size_t>(xb + yb, 16)));
    CU(h, cudaStreamWaitEvent(h->aux2_stream, h->ev_stage[cb], 0));      // the kernels that read this buffer two calls ago
    char* st = h->stage[cb].as<char>();
    if (cx) CU(h, h2d_copy(h, st, X, xb, h->aux2_stream, HostStager::pageable(X)));
    else CU(h, cudaMemcpy2DAsync(Zb, ld * sz, X, ldx * sz, K * sz, nr, cudaMemcpyHostToDevice, h->aux2_stream));
    if (cy) CU(h, h2d_copy(h, st + xb, Y, yb, h->aux2_stream, HostStager::pageable(Y)));
    else if (M > 0) CU(h, cudaMemcpy2DAsync(Zb + K, ld * sz, Y, ldy * sz, M * sz, nr, cudaMemcpyHostToDevice, h->aux2_stream));
    if (h->weighted) CU(h, cudaMemcpyAsync(h->w.as<T>() + row0, w, nr * sz, cudaMemcpyHostToDevice, h->aux2_stream));
    CU(h, cudaEventRecord(h->ev_copied[cb], h->aux2_stream));
    CU(h, cudaStreamWaitEvent(h->stream, h->ev_copied[cb], 0));
    if (cx) { k_repack<T><<<h->sm_count * 8, 256, 0, h->stream>>>((const T*)st, nr, K, Zb, ld); h->launches++; }
    if (cy) { k_repack<T><<<h->sm_count * 4, 256, 0, h->stream>>>((const T*)(st + xb), nr, M, Zb + K, ld); h->launches++; }
    CU(h, cudaEventRecord(h->ev_stage[cb], h->stream));
  } else {
    if (ldx == K) { k_repack<T><<<h->sm_count * 8, 256, 0, h->stream>>>((const T*)X, nr, K, Zb, ld); h->launches++; }
    else CU(h, cudaMemcpy2DAsync(Zb, ld * sz, X, ldx * sz, K * sz, nr, cudaMemcpyDeviceToDevice, h->stream));
    if (M > 0 && ldy == M) { k_repack<T><<<h->sm_count * 4, 256, 0, h->stream>>>((const T*)Y, nr, M, Zb + K, ld); h->launches++; }
    else if (M > 0) CU(h, cudaMemcpy2DAsync(Zb + K, ld * sz, Y, ldy * sz, M * sz, nr, cudaMemcpyDeviceToDevice, h->stream));
    if (h->weighted) CU(h, cudaMemcpyAsync(h->w.as<T>() + row0, w, nr * sz, cudaMemcpyDeviceToDevice, h->stream));
  }
  // the caller may reuse its block buffers on return: host blocks are free once the copies above are done (the
  // Gram of this block then overlaps the next block's upload); device blocks are read by kernels on this stream
  if (!gram) {
    if (mem == CVMX_HOST) CU(h, cudaEventSynchronize(h->ev_copied[cb]));
    else CU(h, cudaStreamSynchronize(h->stream));
    return CVMX_OK;
  }

  std::vector<int2> tiles;
  plan_tiles(h, (uint32_t)(CVMX_WANT_XTX | (M > 0 ? CVMX_WANT_XTY : 0)), tiles);
  const int ntiles = (int)tiles.size();
  const int64_t nu = std::min(h->fill_units_cap, fill_units_for(h, nr, ntiles));
  const int64_t per = round_up((nr + nu - 1) / nu, GBK);
  std::vector<GramUnit> units(nu + 1);
  units[0].row_begin = units[0].row_end = 0; units[0].fold = 0; units[0].split = 0; units[0].nsplit = (int32_t)(nu + 1); units[0].part_base = 0;
  for (int64_t u = 0; u < nu; ++u) {
    GramUnit& g = units[u + 1];
    g.row_begin = row0 + std::min(nr, u * per); g.row_end = row0 + std::min(nr, (u + 1) * per);
    g.fold = 0; g.split = (int32_t)(u + 1); g.nsplit = (int32_t)(nu + 1); g.part_base = 0;
  }
  CU(h, cudaMemcpyAsync(h->units.p, units.data(), units.size() * sizeof(GramUnit), cudaMemcpyHostToDevice, h->stream));
  GramParams<T> gp;
  gp.fmap = fmap_of<T>(h);
  gp.Z = h->Z.as<T>(); gp.w = h->w.as<T>(); gp.ld = ld; gp.indices = nullptr;
  gp.units = h->units.as<GramUnit>() + 1; gp.tiles = h->tiles.as<int2>(); gp.ntiles = ntiles;
  gp.partials = h->partials.as<double>(); gp.raw_out = nullptr; gp.force_partials = 1;
  gp.epi = EpiParams<T>();
  const size_t smem = gram_smem_bytes<T>();
  const int ev0 = prof_mark(h);
  { int32_t rk = launch_k_gram<T>(h, (unsigned)(nu * ntiles), gp); if (rk) return rk; }
  const int ev1 = prof_mark(h);
  prof_span(h, PROF_GRAM, ev0, ev1);
  // accumulator (slot 0) += the block's partials, in place
  gp.units = h->units.as<GramUnit>(); gp.raw_out = h->partials.as<double>();
  k_gram_reduce<T><<<dim3(ntiles, 1), GTHREADS, smem, h->stream>>>(gp, h->fold_units.as<int32_t>(), h->split_folds.as<int32_t>());
  prof_span(h, PROF_REDUCE, ev1, prof_mark(h));
  h->launches += 2;
  CU(h, cudaGetLastError());
  if (mem == CVMX_HOST) CU(h, cudaEventSynchronize(h->ev_copied[cb]));
  else CU(h, cudaStreamSynchronize(h->stream));
  return CVMX_OK;
}

// ---- decoupled slab chain (row-slab mode, float64) --------------------------------------------------------------------
// numpy's column sums are sequential over ALL rows, so rank r can only finish its slab's chains once rank r - 1 has.  Only
// pass 4 of the binade scan needs the exact incoming value, though: passes 1 - 3 need the running sum at the slab's first
// row only APPROXIMATELY (to classify segments by binade, inside pass 2's usual error margin), and that is the sum of the
// earlier slabs' pass-1 totals - a row of 4 ld values per slab that the ranks all-gather.  Every rank then runs passes
// 1 - 3 at once and a hop of the rank-to-rank chain costs one short kernel (one exact addition per 256 rows).
//   mode 1: all rows of the slab (fit totals, chains in sum_z / sumsq_z)      mode 2: folds [f0, f1) of the local CSR
int32_t slab_scan_params(cvmx_t* h, int mode, int64_t f0, int64_t f1, ScanParams& sp, int64_t& Pn, int64_t& max_rows, bool& applicable) {
  const int64_t ld = h->ld;
  Pn = mode == 1 ? 1 : f1 - f0;
  max_rows = 0;
  if (mode == 1) max_rows = h->N;
  else for (int64_t f = f0; f < f1; ++f) max_rows = std::max(max_rows, h->h_off[f + 1] - h->h_off[f]);
  const int64_t max_segs = round_up((max_rows + SCAN_L - 1) / SCAN_L, SCAN_PER_LANE);
  const int64_t groups = ld / MOM_COLS;
  const size_t seg_bytes = (size_t)Pn * max_segs * 4 * ld * sizeof(double);
  applicable = h->dtype == CVMX_F64 && h->scan_mode != 0 && Pn <= 65535 && max_rows >= 4 * SCAN_L && max_rows < ((int64_t)1 << 25) &&
               seg_bytes <= ((size_t)2 << 30);
  if (!applicable) return CVMX_OK;
  MomentParams<double> mp;
  mp.Z = h->Z.as<double>(); mp.w = h->w.as<double>(); mp.ld = ld; mp.K = h->K; mp.M = h->M;
  mp.N = h->N; mp.flags = h->flags; mp.resolution = h->resolution;
  mp.sum_z = h->sum_z.as<double>(); mp.sumsq_z = h->sumsq_z.as<double>();
  mp.fs = nullptr; mp.pw_cols = nullptr; mp.stats = nullptr;
  if (mode == 2) { mp.offsets = h->d_off.as<int64_t>(); mp.indices = h->d_idx.as<int64_t>(); mp.fold0 = f0; }
  else { mp.offsets = nullptr; mp.indices = nullptr; mp.fold0 = 0; mp.pw_cols = h->pwcols.as<double>(); }
  mp.grp0 = 0; mp.grp_stride = 1;
  sp.p = mp; sp.L = SCAN_L; sp.max_segs = max_segs; sp.groups_total = (int)groups;
  sp.slow_cap = (int)(max_segs / 4 + 2);
  CU(h, h->scan_seg.reserve(seg_bytes));
  CU(h, h->scan_ok.reserve((size_t)Pn * groups * sizeof(int)));
  CU(h, h->scan_list.reserve((size_t)Pn * 2 * sp.slow_cap * ld * sizeof(int)));
  CU(h, h->scan_cnt.reserve((size_t)Pn * 2 * ld * sizeof(int)));
  sp.seg = h->scan_seg.as<double>(); sp.ok = h->scan_ok.as<int>();
  sp.slow_list = h->scan_list.as<int>(); sp.slow_cnt = h->scan_cnt.as<int>();
  return CVMX_OK;
}

inline dim3 slab_scan_grid(const ScanParams& sp, int64_t Pn) {
  return dim3((unsigned)sp.groups_total, (unsigned)((sp.max_segs + SCAN_WARPS - 1) / SCAN_WARPS), (unsigned)Pn);
}

// passes 1 and 1b: tot_out [Pn][2][2][ld] (device) = this slab's approximate sums and sums of magnitudes
int32_t slab_scan_local(cvmx_t* h, int mode, int64_t f0, int64_t f1, double* tot_out, bool& applicable) {
  ScanParams sp; int64_t Pn, max_rows;
  int32_t rc = slab_scan_params(h, mode, f0, f1, sp, Pn, max_rows, applicable);
  if (rc || !applicable) return rc;
  k_scan_segsums<<<slab_scan_grid(sp, Pn), 32 * SCAN_WARPS, 0, h->stream>>>(sp);
  k_scan_slab_totals<<<dim3((unsigned)((h->ld + 3) / 4), (unsigned)Pn), 128, 0, h->stream>>>(sp, tot_out);
  h->launches += 2; h->scan_launches += 1;
  CU(h, cudaGetLastError());
  h->slab_scan_mode = mode; h->slab_scan_stage = 1; h->slab_scan_f0 = f0; h->slab_scan_f1 = f1; h->slab_scan_csr = h->csr_version;
  return CVMX_OK;
}

// passes 2 and 3 from the approximate start [Pn][2][2][ld] (device): sums of the earlier slabs' tot_out rows
int32_t slab_scan_prepare(cvmx_t* h, int mode, int64_t f0, int64_t f1, const double* start) {
  ScanParams sp; int64_t Pn, max_rows; bool applicable;
  int32_t rc = slab_scan_params(h, mode, f0, f1, sp, Pn, max_rows, applicable);
  if (rc) return rc;
  if (!applicable) return fail(h, CVMX_ERR_INVALID, "cvmx_slab_scan_prepare: cvmx_slab_scan_local reported the scan not applicable");
  sp.start = start;
  k_scan_prefix<false><<<dim3((unsigned)(sp.groups_total * SCAN_PREFIX_CTAS), (unsigned)Pn), SCAN_PREFIX_THREADS, 0, h->stream>>>(sp, nullptr);
  k_scan_delta<<<slab_scan_grid(sp, Pn), 32 * SCAN_WARPS, 0, h->stream>>>(sp);
  h->launches += 2;
  CU(h, cudaGetLastError());
  h->slab_scan_stage = 2;
  return CVMX_OK;
}

template <typename T>
int32_t launch_moments(cvmx_t* h, MomentParams<T> mp, int64_t nfolds, int64_t max_rows, int col_shard, int n_col_shards,
                       double overlap_ns, const int* done_groups, int done_groups_total);

// pass 4 from the exact chains of the previous slab: carry [Pn][2][ld] (fold mode, in / out) or sum_z / sumsq_z (fit mode,
// chain_mp.accumulate says whether they hold a previous slab's values); groups the scan gave up run the chain kernel
// (chain_mp: the MomentParams the undecoupled path would have launched)
int32_t slab_scan_finish(cvmx_t* h, int mode, int64_t f0, int64_t f1, double* carry, const MomentParams<double>& chain_mp) {
  ScanParams sp; int64_t Pn, max_rows; bool applicable;
  int32_t rc = slab_scan_params(h, mode, f0, f1, sp, Pn, max_rows, applicable);
  if (rc) return rc;
  if (!applicable) return fail(h, CVMX_ERR_INVALID, "decoupled slab chain: not prepared");
  sp.p.accumulate = chain_mp.accumulate;
  if (mode == 2) { sp.carry = carry; sp.p.raw = carry; }
  k_scan_chain<2><<<dim3((unsigned)(sp.groups_total * (SCAN_COLS / 2)), (unsigned)Pn), 64 * 2, scan_chain_smem<2>(), h->stream>>>(sp);
  h->launches++;
  CU(h, cudaGetLastError());
  return launch_moments<double>(h, chain_mp, Pn, max_rows, 0, 1, 0.0, sp.ok, sp.groups_total);
}

struct SlabArgs { const void* carry_sum; const void* carry_sumsq; const void* w_glob; int64_t N_glob; int64_t row0; };

// The part of cvmx_fit_end that does not depend on the moment chains: accumulator -> totals, weight mass.
// use_w_glob: the weight mass runs over h->w_glob (row slabs: all N_w weights of the data set).
// mass_aside: the weight mass (ONE CTA walking numpy's pairwise tree over all N_w weights: ~1 ms at N = 1M) runs on side
// stream 2 instead of the main stream; the caller joins h->ev_mass before it reads fit_scal.
template <typename T>
int32_t fit_end_pre(cvmx_t* h, bool use_w_glob, int64_t N_w, bool mass_aside = false) {
  const int64_t K = h->K, M = h->M, ld = h->ld;
  // accumulator -> totals (raw epilogue: mirrored XtWX, XtWY)
  std::vector<int2> tiles;
  plan_tiles(h, (uint32_t)(CVMX_WANT_XTX | (M > 0 ? CVMX_WANT_XTY : 0)), tiles);
  const int ntiles = (int)tiles.size();
  GramUnit v;
  v.row_begin = v.row_end = 0; v.fold = 0; v.split = 0; v.nsplit = 1; v.part_base = 0;
  CU(h, cudaMemcpyAsync(h->units.p, &v, sizeof(GramUnit), cudaMemcpyHostToDevice, h->stream));
  EpiParams<T> epi;
  epi.mode = 0; epi.flags = 0; epi.want = CVMX_WANT_XTX | CVMX_WANT_XTY;
  epi.K = K; epi.M = M; epi.ld = ld;
  epi.Ttot = nullptr; epi.stats = nullptr; epi.fs = nullptr;
  epi.out_xx = h->Ttot.as<T>(); epi.xx_pitch = ld; epi.xx_stride = 0;
  epi.out_xy = h->Ttot.as<T>() + K; epi.xy_pitch = ld; epi.xy_stride = 0;
  GramParams<T> gp;
  gp.fmap = fmap_of<T>(h);
  gp.Z = h->Z.as<T>(); gp.w = h->w.as<T>(); gp.ld = ld; gp.indices = nullptr;
  gp.units = h->units.as<GramUnit>(); gp.tiles = h->tiles.as<int2>(); gp.ntiles = ntiles;
  gp.partials = h->partials.as<double>(); gp.raw_out = nullptr; gp.force_partials = 0; gp.epi = epi;
  k_gram_reduce<T><<<dim3(ntiles, 1), GTHREADS, gram_smem_bytes<T>(), h->stream>>>(gp, h->fold_units.as<int32_t>(), h->split_folds.as<int32_t>());
  h->launches++;
  CU(h, cudaGetLastError());
  // statistics over all rows: weight mass everywhere, moment sums for this column shard (others stay zero)
  if (h->mass_started) { h->mass_started = false; return CVMX_OK; }   // cvmx_slab_begin launched it beside the upload
  cudaStream_t ms = h->stream;
  if (mass_aside) {
    CU(h, cudaEventRecord(h->ev_mass, h->stream));
    CU(h, cudaStreamWaitEvent(h->aux2_stream, h->ev_mass, 0));
    ms = h->aux2_stream;
  }
  k_weight_mass<T, PW_LEVELS_BIG><<<1, 1 << PW_LEVELS_BIG, 0, ms>>>(h->Z.as<T>(), use_w_glob && h->weighted ? h->w_glob.as<T>() : h->w.as<T>(), ld,
                                                                          N_w, K, M, h->weighted ? 1 : 0, nullptr, nullptr, 0, 1,
                                                                          h->ddof, h->fit_scal.as<FitScalars>(), nullptr, h->pwcols.as<T>());
  h->launches++;
  CU(h, cudaGetLastError());
  if (mass_aside) { CU(h, cudaEventRecord(h->ev_mass, h->aux2_stream)); h->mass_pending = true; }
  return CVMX_OK;
}

template <typename T>
int32_t fit_end_impl(cvmx_t* h, int32_t col_shard, int32_t n_col_shards, const SlabArgs* sl = nullptr) {
  const int64_t N = h->N, K = h->K, M = h->M, ld = h->ld;
  if (sl) {
    // row-slab mode: the weight sums need every weight of the data set, the moment chains continue the previous slab's
    if (h->weighted && !h->fit_pre_done && !h->mass_started) {
      CU(h, h->w_glob.reserve((size_t)std::max<int64_t>(sl->N_glob, 1) * sizeof(T)));
      CU(h, cudaMemcpyAsync(h->w_glob.p, sl->w_glob, (size_t)sl->N_glob * sizeof(T), cudaMemcpyDeviceToDevice, h->stream));
    }
    if (sl->carry_sum) {
      CU(h, cudaMemcpyAsync(h->sum_z.p, sl->carry_sum, ld * sizeof(T), cudaMemcpyDeviceToDevice, h->stream));
      CU(h, cudaMemcpyAsync(h->sumsq_z.p, sl->carry_sumsq, ld * sizeof(T), cudaMemcpyDeviceToDevice, h->stream));
    }
    h->slab = true; h->N_glob = sl->N_glob; h->row0 = sl->row0;
  }
  if (!sl && h->mass_started) {   // cvmx_slab_begin followed by a plain cvmx_fit_end: its weight mass ran over the global weights - redo
    CU(h, cudaStreamWaitEvent(h->stream, h->ev_mass, 0));
    h->mass_started = h->mass_pending = false;
  }
  if (!h->fit_pre_done) { int32_t rp = fit_end_pre<T>(h, sl != nullptr, sl ? sl->N_glob : N); if (rp) return rp; }
  h->fit_pre_done = false;
  MomentParams<T> mp;
  mp.Z = h->Z.as<T>(); mp.w = h->w.as<T>(); mp.ld = ld; mp.K = K; mp.M = M;
  mp.offsets = nullptr; mp.indices = nullptr; mp.fold0 = 0; mp.N = N;
  mp.flags = h->flags; mp.resolution = (T)h->resolution;
  mp.sum_z = h->sum_z.as<T>(); mp.sumsq_z = h->sumsq_z.as<T>();
  mp.fs = nullptr; mp.pw_cols = h->pwcols.as<T>(); mp.stats = nullptr;
  mp.accumulate = (sl && sl->carry_sum) ? 1 : 0;
  int32_t rc;
  if (sl && h->slab_scan_mode == 1 && h->slab_scan_stage == 2) {
    // the scan passes that do not need the previous slab's chains already ran (cvmx_slab_scan_local / _prepare)
    if constexpr (std::is_same<T, double>::value) rc = slab_scan_finish(h, 1, 0, 1, nullptr, mp);
    else rc = fail(h, CVMX_ERR_INVALID, "decoupled slab chain: float64 only");
  } else {
    rc = launch_moments<T>(h, mp, 1, N, col_shard, n_col_shards, 0.0);
  }
  h->slab_scan_mode = 0; h->slab_scan_stage = 0;
  if (rc) return rc;
  if (h->mass_pending) { CU(h, cudaStreamWaitEvent(h->stream, h->ev_mass, 0)); h->mass_pending = false; }
  FitScalars fsc;
  CU(h, cudaMemcpyAsync(&fsc, h->fit_scal.p, sizeof(fsc), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaStreamSynchronize(h->stream));
  h->filling = false;
  if (fsc.neg_weight) return fail(h, CVMX_ERR_NEG_WEIGHT, "Weights must be non-negative.");
  h->fitted = true;
  return CVMX_OK;
}

template <typename T>
int32_t sharded_finish(cvmx_t* h, int64_t batch_f0, int64_t f0, int64_t f1, uint32_t want, const double* gram, T* oxx, T* oxy,
                       const double* const* peers = nullptr, int npeers = 0, bool compact = false);

// ---- folds -----------------------------------------------------------------------------------------
// Runs folds [f0, f1) of the CSR (d_off/d_idx on device, off on host) and leaves results in device
// buffers: dxx [P'][K][K], dxy [P'][K][M] (either may be null per `want`), stats scratch, fscal scratch.
template <typename T>
int32_t run_folds(cvmx_t* h, const int64_t* d_off, const int64_t* d_idx, const int64_t* off, int64_t f0, int64_t f1,
                  uint32_t want, T* dxx, T* dxy, bool cacheable) {
  const int64_t Pn = f1 - f0;
  if (Pn <= 0) return CVMX_OK;
  const int64_t ld = h->ld, K = h->K, M = h->M;
  if (cacheable && h->fold_gram_version == h->csr_version && (want & 3u) == (CVMX_WANT_XTX | (M > 0 ? CVMX_WANT_XTY : 0u))) {
    // cvmx_fit_folds kept the raw Gram of every fold: only the statistics and the epilogue are left
    int64_t max_rows = 0;
    for (int64_t f = f0; f < f1; ++f) max_rows = std::max(max_rows, off[f + 1] - off[f]);
    int32_t rc = launch_fold_stats<T>(h, d_off, d_idx, f0, Pn, max_rows, 0, 1, 0.0,
                                      h->flags ? h->fold_raw.as<T>() + (size_t)f0 * 2 * ld : nullptr);
    if (rc) return rc;
    std::vector<int2> tiles;
    plan_tiles(h, want, tiles);
    const double* gram = h->fold_gram.as<double>() + (size_t)f0 * tiles.size() * GACC * GTHREADS;
    return sharded_finish<T>(h, f0, f0, f1, want, gram, dxx, dxy);
  }
  Plan local;
  Plan& pl = cacheable ? h->plan : local;
  const bool hit = cacheable && pl.fold_begin == f0 && pl.fold_end == f1 && pl.want == want && pl.csr_version == h->csr_version;
  if (!hit) {
    plan_tiles(h, want, pl.tiles);
    plan_units(h, off, f0, f1, (int)pl.tiles.size(), pl);
    pl.fold_begin = f0; pl.fold_end = f1; pl.want = want; pl.csr_version = h->csr_version;
  }
  const bool want_mats = (want & (CVMX_WANT_XTX | CVMX_WANT_XTY)) != 0;
  const bool overlap = want_mats && h->flags != 0 && pl.split_folds.size() == (size_t)Pn;
  const bool small = pl.max_rows <= SMALL_MAX_ROWS && K + M <= 4 * STHREADS;
  // single-unit folds (the leave-many-out regime): the Gram kernel's diagonal tiles evaluate the column sums themselves -
  // no second pass over the fold's rows.  Needs every diagonal tile (XTX wanted), no pairwise single-column sums, k_gram.
  // leave-one-out in the streaming form: the operand kernel forms the means / stds of its one-row folds itself
  bool all_one = small && h->loo_mode == 0 && h->fuse_stats && h->flags != 0 && want_mats && K >= 2 && M != 1 && Pn <= (int64_t)65535 * SMALL_FOLDS;
  for (int64_t f = f0; f < f1 && all_one; ++f) all_one = off[f + 1] - off[f] == 1;
  const bool fuse = want_mats && !small && h->fuse_stats && h->flags != 0 && (want & CVMX_WANT_XTX) && pl.split_folds.empty() &&
                    K >= 2 && M != 1 && (K + M <= round_up(K, GB) || (want & CVMX_WANT_XTY)) /* every column block has a chain tile */ &&
                    fmap_of<T>(h) == 0 && d_idx != nullptr;
  cudaStream_t main_stream = h->stream;
  if (overlap) {
    int32_t rc = fork_stats(h, &main_stream);
    if (rc) return rc;
  }
  {
    // device time the chains can hide behind: the Gram kernel when it overlaps them, nothing otherwise
    const double gram_ns = 2.0 * (double)(off[f1] - off[f0]) * (double)K * (double)(K + M) / 4e4;
    int32_t rc = launch_fold_stats<T>(h, d_off, d_idx, f0, Pn, pl.max_rows, 0, 1, overlap ? gram_ns : 0.0, nullptr, fuse || all_one);
    if (rc) { h->stream = main_stream; return rc; }
  }
  if (overlap) {
    int32_t rc = join_stats(h, main_stream);
    if (rc) return rc;
  }
  if (want_mats) {
    EpiParams<T> epi;
    epi.mode = 1; epi.flags = h->flags; epi.want = want;
    epi.K = K; epi.M = M; epi.ld = ld;
    epi.Ttot = h->Ttot.as<T>(); epi.stats = h->stats.as<T>(); epi.fs = h->fscal.as<FoldScalars>();
    epi.out_xx = dxx; epi.xx_pitch = K; epi.xx_stride = K * K;
    epi.out_xy = dxy; epi.xy_pitch = M; epi.xy_stride = K * M;
    // the Gram kernel reads fold rows through absolute CSR positions
    int32_t rc = small ? launch_small<T>(h, d_off, d_idx, off, f0, Pn, want, epi, overlap ? h->ev_join : nullptr, all_one)
                       : launch_gram<T>(h, pl, d_idx, epi, overlap ? h->ev_join : nullptr, fuse);
    if (rc) return rc;
  }
  return CVMX_OK;
}


template <typename T>
int32_t validation_rows_impl(cvmx_t* h, int64_t fold, const void* stats, uint32_t apply, void* out_X, void* out_Y, int32_t mem) {
  const size_t sz = sizeof(T);
  const int64_t K = h->K, M = h->M, ld = h->ld, C = K + M;
  const int64_t beg = h->h_off[fold], n = h->h_off[fold + 1] - beg;
  if (n == 0) return CVMX_OK;
  const T* dstats = nullptr;       // [2][C]: mean row, std row
  if (stats && apply) {
    if (mem == CVMX_HOST) {
      CU(h, h->out_small.reserve(2 * C * sz));
      CU(h, cudaMemcpyAsync(h->out_small.p, stats, 2 * C * sz, cudaMemcpyHostToDevice, h->stream));
      dstats = h->out_small.as<T>();
    } else {
      dstats = (const T*)stats;
    }
  }
  // the kernel indexes mean / std by absolute column of [X | Y]
  const T* mean = dstats, *sdev = dstats ? dstats + C : nullptr;
  const int64_t* idx = h->d_idx.as<int64_t>() + beg;
  T* dX = (T*)out_X; T* dY = (T*)out_Y;
  if (mem == CVMX_HOST) {
    if (out_X) { CU(h, h->out_xx.reserve((size_t)n * K * sz)); dX = h->out_xx.as<T>(); }
    if (out_Y && M) { CU(h, h->out_xy.reserve((size_t)n * M * sz)); dY = h->out_xy.as<T>(); }
  }
  const unsigned grid = (unsigned)(h->sm_count * 8);
  if (out_X) {
    k_validation_rows<T><<<grid, 256, 0, h->stream>>>(h->Z.as<T>(), ld, idx, n, 0, K, (apply & CVMX_CENTER_X) ? mean : nullptr,
                                                      (apply & CVMX_SCALE_X) ? sdev : nullptr, dX);
    h->launches++;
  }
  if (out_Y && M) {
    k_validation_rows<T><<<grid, 256, 0, h->stream>>>(h->Z.as<T>(), ld, idx, n, K, M, (apply & CVMX_CENTER_Y) ? mean : nullptr,
                                                      (apply & CVMX_SCALE_Y) ? sdev : nullptr, dY);
    h->launches++;
  }
  CU(h, cudaGetLastError());
  if (mem == CVMX_HOST) {
    if (out_X) CU(h, cudaMemcpyAsync(out_X, dX, (size_t)n * K * sz, cudaMemcpyDeviceToHost, h->stream));
    if (out_Y && M) CU(h, cudaMemcpyAsync(out_Y, dY, (size_t)n * M * sz, cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
  }
  return CVMX_OK;
}

int32_t upload_tables(cvmx_t* h, TableCache& tc, const std::vector<int64_t>& key, const Plan& pl) {
  CU(h, tc.units.reserve(std::max<size_t>(1, pl.units.size()) * sizeof(GramUnit)));
  CU(h, tc.tiles.reserve(std::max<size_t>(1, pl.tiles.size()) * sizeof(int2)));
  CU(h, tc.fold_units.reserve(std::max<size_t>(1, pl.fold_units.size()) * sizeof(int32_t)));
  CU(h, tc.split_folds.reserve(std::max<size_t>(1, pl.split_folds.size()) * sizeof(int32_t)));
  CU(h, cudaMemcpyAsync(tc.units.p, pl.units.data(), pl.units.size() * sizeof(GramUnit), cudaMemcpyHostToDevice, h->stream));
  CU(h, cudaMemcpyAsync(tc.tiles.p, pl.tiles.data(), pl.tiles.size() * sizeof(int2), cudaMemcpyHostToDevice, h->stream));
  CU(h, cudaMemcpyAsync(tc.fold_units.p, pl.fold_units.data(), pl.fold_units.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
  CU(h, cudaMemcpyAsync(tc.split_folds.p, pl.split_folds.data(), pl.split_folds.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
  tc.key = key;
  tc.n_units = (int64_t)pl.units.size(); tc.n_partial_units = pl.n_partial_units; tc.ntiles = (int)pl.tiles.size();
  return CVMX_OK;
}

// ---- sharded evaluation (multi-GPU: one handle per rank, collectives done by the caller) -------------------------
// phase 1: statistics of folds [f0, f1) restricted to column groups col_shard, col_shard + n, ... ; the other
//          entries of the stats buffer stay zero, so an all-reduce(sum) across ranks assembles the full rows.
template <typename T>
int32_t sharded_stats(cvmx_t* h, int64_t f0, int64_t f1, int col_shard, int n_col_shards) {
  const int64_t Pn = f1 - f0;
  int64_t max_rows = 0;
  for (int64_t f = f0; f < f1; ++f) max_rows = std::max(max_rows, h->h_off[f + 1] - h->h_off[f]);
  // the chains run on the side stream beside the Gram kernel of phase 2; cvmx_sharded_stats_wait joins them
  cudaStream_t main_stream;
  int32_t rc0 = fork_stats(h, &main_stream);
  if (rc0) return rc0;
  // phase 2 (this rank's row shard of the Gram pass) runs beside the chains
  const double gram_ns = 2.0 * (double)(h->h_off[f1] - h->h_off[f0]) * (double)h->K * (double)(h->K + h->M) / 4e4 / n_col_shards;
  int32_t rc = launch_fold_stats<T>(h, h->d_off.as<int64_t>(), h->d_idx.as<int64_t>(), f0, Pn, max_rows, col_shard, n_col_shards, gram_ns);
  int32_t rc2 = join_stats(h, main_stream);
  return rc ? rc : rc2;
}

// phase 2: raw Gram of row shard `shard` of every fold in [f0, f1) -> out [P'][ntiles][GACC][GTHREADS] f64
template <typename T>
int32_t sharded_gram(cvmx_t* h, int64_t f0, int64_t f1, uint32_t want, int shard, int nshards, double* out) {
  const int64_t Pn = f1 - f0;
  TableCache& tc = h->tc_gram;
  const std::vector<int64_t> key = {f0, f1, (int64_t)want, shard, nshards, h->csr_version};
  if (tc.key != key) {
    Plan pl;
    plan_tiles(h, want, pl.tiles);
    const int nt = (int)pl.tiles.size();
    // shard boundaries inside each fold's index range, aligned to the stage size
    std::vector<int64_t> off2(2 * Pn);
    for (int64_t f = 0; f < Pn; ++f) {
      const int64_t beg = h->h_off[f0 + f], n = h->h_off[f0 + f + 1] - beg;
      const int64_t per = round_up((n + nshards - 1) / nshards, GBK);
      off2[2 * f] = beg + std::min(n, shard * per);
      off2[2 * f + 1] = beg + std::min(n, (shard + 1) * per);
    }
    // units: taper each fold's shard so that the greedy CTA placement ends evenly (plan_tapered); wide K: the tiles
    // alone fill the GPU in many waves - one unit per fold shard, no partial workspace to sum
    const int64_t sms = h->sm_count;
    std::vector<std::vector<int64_t>> sizes;
    if (nt >= sms) {
      for (int64_t f = 0; f < Pn; ++f) sizes.push_back({off2[2 * f + 1] - off2[2 * f]});
    } else {
      std::vector<int64_t> fold_rows;
      for (int64_t f = 0; f < Pn; ++f) fold_rows.push_back(off2[2 * f + 1] - off2[2 * f]);
      sizes = plan_tapered(fold_rows, pl.tiles, sms, 1024, 8192);
    }
    pl.fold_units.assign(Pn, 0);
    for (int64_t f = 0; f < Pn; ++f) {
      const int64_t ns = (int64_t)sizes[f].size();
      pl.fold_units[f] = (int32_t)pl.units.size();
      pl.split_folds.push_back((int32_t)f);
      int64_t pos = off2[2 * f];
      for (int64_t s2 = 0; s2 < ns; ++s2) {
        GramUnit u;
        u.row_begin = pos; u.row_end = pos + sizes[f][s2];
        pos += sizes[f][s2];
        u.fold = (int32_t)f; u.split = (int32_t)s2; u.nsplit = (int32_t)ns; u.part_base = (int32_t)pl.n_partial_units;
        pl.units.push_back(u);
      }
      pl.n_partial_units += ns;
    }
    sort_units_longest_first(pl);
    int32_t rcu = upload_tables(h, tc, key, pl);   // the plan repeats from step to step: uploaded once
    if (rcu) return rcu;
  }
  const int ntiles = tc.ntiles;
  const bool direct = tc.n_partial_units == Pn;     // one unit per fold: k_gram writes the fold's raw Gram itself
  if (!direct) CU(h, h->partials.reserve((size_t)tc.n_partial_units * ntiles * GACC * GTHREADS * sizeof(double)));
  GramParams<T> gp;
  gp.fmap = fmap_of<T>(h);
  gp.Z = h->Z.as<T>(); gp.w = h->w.as<T>(); gp.ld = h->ld; gp.indices = h->d_idx.as<int64_t>();
  gp.units = tc.units.as<GramUnit>(); gp.tiles = tc.tiles.as<int2>(); gp.ntiles = ntiles;
  gp.partials = direct ? out : h->partials.as<double>(); gp.raw_out = out; gp.force_partials = 1;
  gp.epi = EpiParams<T>();
  const size_t smem = gram_smem_bytes<T>();
  if (!h->attr_gram) {
    CU(h, cudaFuncSetAttribute(k_gram<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CU(h, cudaFuncSetAttribute(k_gram_reduce<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    h->attr_gram = true;
  }
  const int ev0 = prof_mark(h);
  { int32_t rk = launch_k_gram<T>(h, (unsigned)(tc.n_units * ntiles), gp); if (rk) return rk; }
  h->launches++;
  const int ev1 = prof_mark(h);
  prof_span(h, PROF_GRAM, ev0, ev1);
  if (!direct) {
    for (int64_t t0 = 0; t0 < ntiles; t0 += 65535) {   // grid.y limit
      const unsigned ty = (unsigned)std::min<int64_t>(65535, ntiles - t0);
      k_partial_sum<<<dim3((unsigned)(GACC * GTHREADS / 512), ty, (unsigned)Pn), 256, 0, h->stream>>>(
          h->partials.as<double>() + (size_t)t0 * GACC * GTHREADS, tc.units.as<GramUnit>(), tc.fold_units.as<int32_t>(), ntiles,
          out + (size_t)t0 * GACC * GTHREADS);
    }
    h->launches++;
  }
  prof_span(h, PROF_REDUCE, ev1, prof_mark(h));
  CU(h, cudaGetLastError());
  return CVMX_OK;
}

// phase 3: epilogue of folds [f0, f1) from (all-reduced) raw Grams in the fragment layout of phase 2; `first` is
// the fold of the batch that gram[0] belongs to (a rank may finish only the folds it owns)
template <typename T>
int32_t sharded_finish(cvmx_t* h, int64_t batch_f0, int64_t f0, int64_t f1, uint32_t want, const double* gram, T* oxx, T* oxy,
                       const double* const* peers, int npeers, bool compact) {
  // compact: `gram` holds only folds [f0, f1) (slot f - f0) instead of the whole batch (slot f - batch_f0)
  const int64_t Pn = f1 - f0;
  if (Pn <= 0) return CVMX_OK;
  TableCache& tc = h->tc_finish;
  const std::vector<int64_t> key = {batch_f0, f0, f1, (int64_t)want, h->csr_version, compact ? 1 : 0};
  if (tc.key != key) {
    Plan pl;
    plan_tiles(h, want, pl.tiles);
    pl.fold_units.assign(f1 - batch_f0, 0);
    for (int64_t f = batch_f0; f < f1; ++f) {
      GramUnit u;
      u.row_begin = u.row_end = 0; u.fold = (int32_t)(f - batch_f0); u.split = 0; u.nsplit = 1;
      u.part_base = (int32_t)(compact ? std::max<int64_t>(f - f0, 0) : f - batch_f0);
      pl.fold_units[f - batch_f0] = (int32_t)pl.units.size();
      pl.units.push_back(u);
      if (f >= f0) pl.split_folds.push_back((int32_t)(f - batch_f0));
    }
    int32_t rcu = upload_tables(h, tc, key, pl);
    if (rcu) return rcu;
  }
  const int ntiles = tc.ntiles;
  EpiParams<T> epi;
  epi.mode = 1; epi.flags = h->flags; epi.want = want;
  epi.K = h->K; epi.M = h->M; epi.ld = h->ld;
  epi.Ttot = h->Ttot.as<T>(); epi.stats = h->stats.as<T>(); epi.fs = h->fscal.as<FoldScalars>();
  // outputs are indexed by fold relative to f0
  epi.out_xx = oxx ? oxx - (f0 - batch_f0) * h->K * h->K : nullptr; epi.xx_pitch = h->K; epi.xx_stride = h->K * h->K;
  epi.out_xy = oxy ? oxy - (f0 - batch_f0) * h->K * h->M : nullptr; epi.xy_pitch = h->M; epi.xy_stride = h->K * h->M;
  GramParams<T> gp;
  gp.fmap = fmap_of<T>(h);
  gp.Z = h->Z.as<T>(); gp.w = h->w.as<T>(); gp.ld = h->ld; gp.indices = nullptr;
  gp.units = tc.units.as<GramUnit>(); gp.tiles = tc.tiles.as<int2>(); gp.ntiles = ntiles;
  gp.partials = const_cast<double*>(gram); gp.raw_out = nullptr; gp.force_partials = 0;
  gp.epi = epi;
  for (int q = 0; q < npeers && q < 8; ++q) gp.peers[q] = peers[q];
  gp.npeers = std::min(npeers, 8);
  const size_t smem = gram_smem_bytes<T>();
  const int ev0 = prof_mark(h);
  k_gram_reduce<T><<<dim3(ntiles, (unsigned)Pn), GTHREADS, smem, h->stream>>>(gp, tc.fold_units.as<int32_t>(), tc.split_folds.as<int32_t>());
  h->launches++;
  prof_span(h, PROF_REDUCE, ev0, prof_mark(h));
  CU(h, cudaGetLastError());
  return CVMX_OK;
}

template <typename T>
int32_t export_small(cvmx_t* h, int64_t Pn, void* out_stats, void* out_scal, int32_t* out_status, int32_t mem) {
  const size_t sz = sizeof(T);
  const int64_t C = h->K + h->M;
  const cudaMemcpyKind kind = mem == CVMX_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  if (out_stats)
    CU(h, cudaMemcpy2DAsync(out_stats, C * sz, h->stats.p, h->ld * sz, C * sz, Pn * 2, kind, h->stream));
  if (out_scal || out_status) {
    T* dscal = nullptr; int32_t* dstat = nullptr;
    if (mem == CVMX_HOST) {
      CU(h, h->out_small.reserve(Pn * (2 * sz + sizeof(int32_t))));
      dscal = h->out_small.as<T>();
      dstat = reinterpret_cast<int32_t*>(h->out_small.as<char>() + Pn * 2 * sz);
    } else { dscal = (T*)out_scal; dstat = out_status; }
    k_pack_scalars<T><<<(unsigned)((Pn + 255) / 256), 256, 0, h->stream>>>(h->fscal.as<FoldScalars>(), Pn,
                                                                           out_scal ? dscal : nullptr, out_status ? dstat : nullptr);
    h->launches++;
    CU(h, cudaGetLastError());
    if (mem == CVMX_HOST) {
      if (out_scal) CU(h, cudaMemcpyAsync(out_scal, dscal, Pn * 2 * sz, cudaMemcpyDeviceToHost, h->stream));
      if (out_status) CU(h, cudaMemcpyAsync(out_status, dstat, Pn * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    }
  }
  return CVMX_OK;
}

template <typename T>
int32_t training_impl(cvmx_t* h, const int64_t* d_off, const int64_t* d_idx, const int64_t* off, int64_t f0, int64_t f1,
                      uint32_t want, void* oxx, void* oxy, void* ostats, void* oscal, int32_t* ostatus, int32_t mem,
                      bool cacheable) {
  const size_t sz = sizeof(T);
  const int64_t K = h->K, M = h->M;
  if ((want & CVMX_WANT_XTY) && M == 0) return fail(h, CVMX_ERR_NO_Y, "Response variables `Y` are not provided.");
  if ((want & CVMX_WANT_XTX) && !oxx) return fail(h, CVMX_ERR_INVALID, "out_XTX is NULL");
  if ((want & CVMX_WANT_XTY) && !oxy) return fail(h, CVMX_ERR_INVALID, "out_XTY is NULL");
  if (mem == CVMX_DEVICE) {
    int32_t rc = run_folds<T>(h, d_off, d_idx, off, f0, f1, want, (T*)oxx, (T*)oxy, cacheable);
    if (rc) return rc;
    return export_small<T>(h, f1 - f0, ostats, oscal, ostatus, mem);
  }
  // host outputs: bounded device staging, fold sub-batches
  const size_t per_fold = ((want & CVMX_WANT_XTX) ? (size_t)K * K : 0) * sz + ((want & CVMX_WANT_XTY) ? (size_t)K * M : 0) * sz;
  const int64_t chunk = per_fold ? std::max<int64_t>(1, (int64_t)(((size_t)1 << 30) / per_fold)) : (f1 - f0);
  for (int64_t c0 = f0; c0 < f1; c0 += chunk) {
    const int64_t c1 = std::min(f1, c0 + chunk), Pn = c1 - c0;
    if (want & CVMX_WANT_XTX) CU(h, h->out_xx.reserve((size_t)Pn * K * K * sz));
    if (want & CVMX_WANT_XTY) CU(h, h->out_xy.reserve((size_t)Pn * K * M * sz));
    int32_t rc = run_folds<T>(h, d_off, d_idx, off, c0, c1, want, h->out_xx.as<T>(), h->out_xy.as<T>(),
                              cacheable && chunk >= f1 - f0);
    if (rc) return rc;
    const int64_t d = c0 - f0;
    if (want & CVMX_WANT_XTX)
      CU(h, cudaMemcpyAsync((char*)oxx + (size_t)d * K * K * sz, h->out_xx.p, (size_t)Pn * K * K * sz, cudaMemcpyDeviceToHost, h->stream));
    if (want & CVMX_WANT_XTY)
      CU(h, cudaMemcpyAsync((char*)oxy + (size_t)d * K * M * sz, h->out_xy.p, (size_t)Pn * K * M * sz, cudaMemcpyDeviceToHost, h->stream));
    rc = export_small<T>(h, Pn, ostats ? (char*)ostats + (size_t)d * 2 * (K + M) * sz : nullptr,
                         oscal ? (char*)oscal + (size_t)d * 2 * sz : nullptr, ostatus ? ostatus + d : nullptr, mem);
    if (rc) return rc;
    CU(h, cudaStreamSynchronize(h->stream));
  }
  return CVMX_OK;
}

// Cross-validated PLS over folds [f0, f1) (include/cvmx.h: cvmx_pls_cv).  The range is walked in windows that keep the
// device scratch near 1 GiB, as training_impl stages host outputs: run_folds leaves the window's XTX / XTY, statistics and
// fold scalars in library scratch, the PLS kernels fit every fold, the PRESS kernels score its validation rows.
template <typename T>
int32_t pls_cv_impl(cvmx_t* h, int64_t f0, int64_t f1, int64_t A, void* opress, void* osumw, void* oB, int32_t* onfit,
                    int32_t* ostatus, void* opred, int32_t mem) {
  const size_t sz = sizeof(T);
  const int64_t K = h->K, M = h->M;
  const uint32_t want = CVMX_WANT_XTX | CVMX_WANT_XTY;
  const bool host = mem == CVMX_HOST;
  const size_t ws_fold = pls_state_doubles(K, M, A) * sizeof(double) + 2 * sizeof(int32_t);
  const size_t out_fold = host ? (size_t)A * M * sz + sz + 2 * sizeof(int32_t) + (oB ? (size_t)A * K * M * sz : 0) : 0;
  const size_t per_fold = (size_t)(K * K + K * M) * sz + ws_fold + out_fold;
  const int64_t chunk = std::max<int64_t>(1, (int64_t)(((size_t)1 << 30) / per_fold));
  const cudaMemcpyKind kind = host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  const size_t smem_dir = M > 1 ? (size_t)(M * M + PLS_CH * M) * sizeof(double) : 0;
  const size_t smem_press = press_smem_bytes(M);
  CU(h, cudaFuncSetAttribute(k_pls_dir, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_dir));
  CU(h, cudaFuncSetAttribute(k_pls_press<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_press));
  const int64_t* off = h->h_off.data();
  std::vector<int64_t> tab;
  for (int64_t c0 = f0; c0 < f1; c0 += chunk) {
    const int64_t c1 = std::min(f1, c0 + chunk), Pn = c1 - c0, d = c0 - f0;
    CU(h, h->out_xx.reserve((size_t)Pn * K * K * sz));
    CU(h, h->out_xy.reserve((size_t)Pn * K * M * sz));
    int32_t rc = run_folds<T>(h, h->d_off.as<int64_t>(), h->d_idx.as<int64_t>(), off, c0, c1, want, h->out_xx.as<T>(),
                              h->out_xy.as<T>(), chunk >= f1 - f0);
    if (rc) return rc;
    // working state
    CU(h, h->pls_ws.reserve((size_t)Pn * ws_fold));
    PlsState st;
    st.K = K; st.M = M; st.A = A;
    double* q = h->pls_ws.as<double>();
    st.xty = q; q += Pn * K * M;
    st.R = q; q += Pn * A * K;
    st.Pm = q; q += Pn * A * K;
    st.Q = q; q += Pn * A * M;
    st.u = q; q += Pn * K;
    st.S = q; q += Pn * 2 * M * M;
    st.y0 = q; q += Pn;
    st.nfit = reinterpret_cast<int32_t*>(q);
    st.state = st.nfit + Pn;
    k_pls_init<T><<<(unsigned)Pn, PLS_THREADS, 0, h->stream>>>(h->out_xy.as<T>(), h->fscal.as<FoldScalars>(), h->flags, st);
    h->launches++;
    const dim3 gxr((unsigned)Pn, (unsigned)((K + PLS_ROWS_PER_BLOCK - 1) / PLS_ROWS_PER_BLOCK));
    for (int64_t a = 0; a < A; ++a) {
      k_pls_dir<<<(unsigned)Pn, PLS_THREADS, smem_dir, h->stream>>>(st, a);
      k_pls_xtx_r<T><<<gxr, PLS_THREADS, 0, h->stream>>>(h->out_xx.as<T>(), st, a);
      k_pls_update<<<(unsigned)Pn, PLS_THREADS, 0, h->stream>>>(st, a);
      h->launches += 3;
    }
    CU(h, cudaGetLastError());
    // PRESS: chunks of at most PRESS_ROWS validation rows, never spanning two folds; then chunk_off [Pn + 1]
    const int64_t nch = press_chunk_table(off, c0, c1, tab);
    CU(h, h->pls_tab.reserve(tab.size() * sizeof(int64_t)));
    CU(h, cudaMemcpyAsync(h->pls_tab.p, tab.data(), tab.size() * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    CU(h, h->pls_part.reserve((size_t)std::max<int64_t>(nch, 1) * (A * M + 1) * sizeof(double)));
    double* part = h->pls_part.as<double>();
    double* part_w = part + nch * A * M;
    // predictions: device outputs are written in place (row 0 of the window = CSR position off[c0]); host outputs are
    // staged per launch, so PRESS then runs in launches of at most `per` chunks (partials land in the same slots)
    const int64_t AM = A * M;
    const int64_t per = opred && host ? std::max<int64_t>(1, CV_PRED_STAGE_BYTES / (PRESS_ROWS * AM * (int64_t)sz)) : std::max<int64_t>(nch, 1);
    if (opred && host && nch > 0) CU(h, h->cv_pred.reserve((size_t)std::min(per, nch) * PRESS_ROWS * AM * sz));
    for (int64_t g0 = 0; g0 < nch; g0 += per) {
      const int64_t g1 = std::min(nch, g0 + per);
      const int64_t p0 = tab[3 * g0], p1 = tab[3 * (g1 - 1)] + tab[3 * (g1 - 1) + 1];   // CSR positions of the launch
      PressParams<T> pp;
      pp.Z = h->Z.as<T>(); pp.w = h->weighted ? h->w.as<T>() : nullptr; pp.ld = h->ld;
      pp.idx = h->d_idx.as<int64_t>(); pp.chunks = h->pls_tab.as<int64_t>() + 3 * g0; pp.stats = h->stats.as<T>();
      pp.flags = h->flags; pp.s = st; pp.part = part + g0 * AM; pp.part_w = part_w + g0;
      pp.pred = !opred ? nullptr : host ? h->cv_pred.as<T>() : (T*)opred + (off[c0] - off[f0]) * AM;
      pp.pred_ld = AM;
      pp.pred_pos = host ? p0 : off[c0];
      k_pls_press<T><<<(unsigned)(g1 - g0), PLS_THREADS, smem_press, h->stream>>>(pp);
      h->launches++;
      if (opred && host)
        CU(h, cudaMemcpyAsync((T*)opred + (p0 - off[f0]) * AM, pp.pred, (size_t)(p1 - p0) * AM * sz, cudaMemcpyDeviceToHost, h->stream));
    }
    // outputs: straight into the caller's device buffers, or staged for the copy to the host
    T *dpress = (T*)opress + (size_t)d * A * M, *dsumw = (T*)osumw + d, *dB = oB ? (T*)oB + (size_t)d * A * K * M : nullptr;
    int32_t* dstatus = ostatus + d;
    if (host) {
      CU(h, h->pls_out.reserve((size_t)Pn * out_fold));
      char* o = h->pls_out.as<char>();
      dpress = (T*)o; o += (size_t)Pn * A * M * sz;
      dsumw = (T*)o; o += (size_t)Pn * sz;
      dstatus = (int32_t*)o; o += (size_t)Pn * sizeof(int32_t);
      o += (size_t)Pn * sizeof(int32_t);
      dB = oB ? (T*)o : nullptr;
    }
    k_pls_press_reduce<T><<<(unsigned)Pn, PLS_THREADS, 0, h->stream>>>(part, part_w, h->pls_tab.as<int64_t>() + 3 * nch, st,
                                                                       dpress, dsumw);
    k_pack_scalars<T><<<(unsigned)((Pn + 255) / 256), 256, 0, h->stream>>>(h->fscal.as<FoldScalars>(), Pn, nullptr, dstatus);
    h->launches += 2;
    if (dB) {
      const dim3 gc((unsigned)Pn, (unsigned)std::min<int64_t>(65535, (K * M + PLS_THREADS - 1) / PLS_THREADS));
      k_pls_coefs<T><<<gc, PLS_THREADS, 0, h->stream>>>(st, dB);
      h->launches++;
    }
    CU(h, cudaGetLastError());
    CU(h, cudaMemcpyAsync(onfit + d, st.nfit, (size_t)Pn * sizeof(int32_t), kind, h->stream));
    if (host) {
      CU(h, cudaMemcpyAsync((char*)opress + (size_t)d * A * M * sz, dpress, (size_t)Pn * A * M * sz, kind, h->stream));
      CU(h, cudaMemcpyAsync((T*)osumw + d, dsumw, (size_t)Pn * sz, kind, h->stream));
      CU(h, cudaMemcpyAsync(ostatus + d, dstatus, (size_t)Pn * sizeof(int32_t), kind, h->stream));
      if (oB) CU(h, cudaMemcpyAsync((char*)oB + (size_t)d * A * K * M * sz, dB, (size_t)Pn * A * K * M * sz, kind, h->stream));
    }
    // the next window reuses the scratch and the chunk table's host vector
    CU(h, cudaStreamSynchronize(h->stream));
  }
  return CVMX_OK;
}

// Cross-validated ridge over folds [f0, f1) (include/cvmx.h: cvmx_ridge_cv).  `plan` is ridge_plan's for this call and
// is feasible: every scratch size and launch geometry below comes from it.  Per window run_folds leaves the folds' XTX /
// XTY, statistics and fold scalars in library scratch; per pass of penalties the factorisation, the substitutions and
// PRESS run over every (fold, penalty) pair.  A pass covers all penalties of its window or a one-fold window, so the
// outputs of a pass are one contiguous range of the caller's arrays.
template <typename T>
int32_t ridge_cv_impl(cvmx_t* h, int64_t f0, int64_t f1, const double* alphas, int64_t L, void* opress, void* osumw, void* oB,
                      int32_t* oinfo, int32_t* ostatus, void* opred, int32_t mem, const int64_t* plan) {
  const size_t sz = sizeof(T);
  const int64_t K = h->K, M = h->M;
  const uint32_t want = CVMX_WANT_XTX | CVMX_WANT_XTY;
  const bool host = mem == CVMX_HOST;
  const cudaMemcpyKind kind = host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  const int64_t W = plan[CVMX_RIDGE_FOLDS_PER_WINDOW], Lp = plan[CVMX_RIDGE_PENALTIES_PER_PASS];
  const int64_t G = plan[CVMX_RIDGE_CHUNKS_PER_LAUNCH];
  const int64_t* grid = plan + CVMX_RIDGE_GRID;
  const int64_t* smem = plan + CVMX_RIDGE_SMEM;
  if (f1 <= f0) return CVMX_OK;
  CU(h, cudaFuncSetAttribute(k_ridge_potrf_diag, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem[CVMX_RK_POTRF]));
  CU(h, cudaFuncSetAttribute(k_ridge_trsm, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem[CVMX_RK_TRSM]));
  CU(h, cudaFuncSetAttribute(k_ridge_syrk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem[CVMX_RK_SYRK]));
  CU(h, cudaFuncSetAttribute(k_ridge_bsolve_diag, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem[CVMX_RK_BSOLVE_DIAG]));
  CU(h, cudaFuncSetAttribute(k_ridge_bsolve_update, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem[CVMX_RK_BSOLVE_UPDATE]));
  CU(h, cudaFuncSetAttribute(k_ridge_press<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem[CVMX_RK_PRESS]));
  CU(h, h->ridge_ws.reserve((size_t)plan[CVMX_RIDGE_SCRATCH_BYTES]));
  CU(h, h->ridge_part.reserve((size_t)plan[CVMX_RIDGE_PART_BYTES]));
  CU(h, h->ridge_alpha.reserve((size_t)L * sizeof(double)));
  CU(h, h->out_xx.reserve((size_t)W * K * K * sz));
  CU(h, h->out_xy.reserve((size_t)W * K * M * sz));
  // host predictions: a PRESS launch holds at most as many chunks as fill CV_PRED_STAGE_BYTES at the pass's width (and at
  // most the plan's G), and never more rows than the range has; the bound below covers every pass width <= Lp M
  const int64_t chunk_bytes = PRESS_ROWS * Lp * M * (int64_t)sz, range_bytes = (h->h_off[f1] - h->h_off[f0]) * Lp * M * (int64_t)sz;
  if (opred && host && range_bytes > 0)
    CU(h, h->cv_pred.reserve((size_t)std::min({G * chunk_bytes, std::max(CV_PRED_STAGE_BYTES, chunk_bytes), range_bytes})));
  // the penalties live on the device before any kernel runs; kernels never see a host address
  CU(h, cudaMemcpyAsync(h->ridge_alpha.p, alphas, (size_t)L * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  char* ws = h->ridge_ws.as<char>();
  RidgeState st;
  st.K = K; st.M = M;
  st.A = reinterpret_cast<double*>(ws);
  st.state = reinterpret_cast<int32_t*>(ws + plan[CVMX_RIDGE_END_A]);
  double* acc = reinterpret_cast<double*>(ws + plan[CVMX_RIDGE_END_STATE]);
  double* acc_w = reinterpret_cast<double*>(ws + plan[CVMX_RIDGE_END_ACC]);
  const int64_t* off = h->h_off.data();
  std::vector<int64_t> tab;
  for (int64_t c0 = f0; c0 < f1; c0 += W) {
    const int64_t c1 = std::min(f1, c0 + W), Pn = c1 - c0, d = c0 - f0;
    int32_t rc = run_folds<T>(h, h->d_off.as<int64_t>(), h->d_idx.as<int64_t>(), off, c0, c1, want, h->out_xx.as<T>(),
                              h->out_xy.as<T>(), W >= f1 - f0);
    if (rc) return rc;
    const int64_t nch = press_chunk_table(off, c0, c1, tab);
    if (nch > RIDGE_MAX_GRID_X) return fail(h, CVMX_ERR_INVALID, "cvmx_ridge_cv: too many validation rows in one window");
    CU(h, h->ridge_tab.reserve(std::max<size_t>(tab.size(), 1) * sizeof(int64_t)));
    CU(h, cudaMemcpyAsync(h->ridge_tab.p, tab.data(), tab.size() * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    const int64_t* dtab = h->ridge_tab.as<int64_t>();
    T* dsumw = host ? reinterpret_cast<T*>(ws + plan[CVMX_RIDGE_END_B]) : (T*)osumw + d;
    int32_t* dstatus = host ? reinterpret_cast<int32_t*>(ws + plan[CVMX_RIDGE_END_SUM_W]) : ostatus + d;
    k_pack_scalars<T><<<(unsigned)((Pn + 255) / 256), 256, 0, h->stream>>>(h->fscal.as<FoldScalars>(), Pn, nullptr, dstatus);
    h->launches++;
    for (int64_t l0 = 0; l0 < L; l0 += Lp) {
      const int64_t Lc = std::min(L, l0 + Lp) - l0, pairs = Pn * Lc;
      if (Pn > 1 && Lc != L) return fail(h, CVMX_ERR_INVALID, "cvmx_ridge_cv: inconsistent launch plan");
      st.Lp = Lc;
      const int64_t width = Lc * M;
      // outputs of the pass: folds [c0, c1) x penalties [l0, l0 + Lc), one contiguous range of the caller's arrays
      const size_t o_pm = (size_t)(d * L + l0) * M, o_in = (size_t)(d * L + l0), o_b = (size_t)(d * L + l0) * K * M;
      T* dpress = host ? reinterpret_cast<T*>(ws + plan[CVMX_RIDGE_END_ACC_W]) : (T*)opress + o_pm;
      int32_t* dinfo = host ? reinterpret_cast<int32_t*>(ws + plan[CVMX_RIDGE_END_PRESS]) : oinfo + o_in;
      T* dB = !oB ? nullptr : host ? reinterpret_cast<T*>(ws + plan[CVMX_RIDGE_END_INFO]) : (T*)oB + o_b;
      CU(h, cudaMemsetAsync(acc, 0, (size_t)(plan[CVMX_RIDGE_END_ACC_W] - plan[CVMX_RIDGE_END_STATE]), h->stream));
      const dim3 gl((unsigned)pairs, (unsigned)grid[2 * CVMX_RK_LOAD + 1]);
      k_ridge_load<T><<<gl, RIDGE_THREADS, 0, h->stream>>>(h->out_xx.as<T>(), h->out_xy.as<T>(), h->fscal.as<FoldScalars>(), h->flags,
                                                           h->ridge_alpha.as<double>() + l0, st);
      h->launches++;
      for (int64_t j = 0; j < K; j += RIDGE_NB) {
        const int nbj = (int)std::min<int64_t>(RIDGE_NB, K - j);
        k_ridge_potrf_diag<<<(unsigned)pairs, RIDGE_THREADS, smem[CVMX_RK_POTRF], h->stream>>>(st, j, nbj);
        const dim3 gt((unsigned)pairs, (unsigned)ridge_cdiv(K + M - j - nbj, RIDGE_TR_ROWS));
        k_ridge_trsm<<<gt, RIDGE_TR_ROWS, smem[CVMX_RK_TRSM], h->stream>>>(st, j, nbj);
        h->launches += 2;
        if (j + nbj < K) {
          const SyrkTiles t = ridge_syrk_tiles(K, M, j + nbj);
          k_ridge_syrk<<<(unsigned)(pairs * t.total), RIDGE_THREADS, smem[CVMX_RK_SYRK], h->stream>>>(st, j, nbj, t);
          h->launches++;
        }
      }
      for (int64_t j = (K - 1) / RIDGE_NB * RIDGE_NB; j >= 0; j -= RIDGE_NB) {
        const int nbj = (int)std::min<int64_t>(RIDGE_NB, K - j);
        k_ridge_bsolve_diag<<<(unsigned)pairs, RIDGE_BS_THREADS, smem[CVMX_RK_BSOLVE_DIAG], h->stream>>>(st, j, nbj);
        h->launches++;
        if (j > 0) {
          const dim3 gu((unsigned)pairs, (unsigned)(j / RIDGE_NB));
          k_ridge_bsolve_update<<<gu, RIDGE_THREADS, smem[CVMX_RK_BSOLVE_UPDATE], h->stream>>>(st, j, nbj);
          h->launches++;
        }
      }
      // PRESS over the window's chunks, at most Gl chunks per launch, each launch's sums added in chunk order (the
      // sums do not depend on the group size).  Predictions of the pass: columns [l0 M, l0 M + width) of rows [n][L M]
      const int64_t Gl = opred && host ? std::min(G, std::max<int64_t>(1, CV_PRED_STAGE_BYTES / (PRESS_ROWS * width * (int64_t)sz))) : G;
      for (int64_t g0 = 0; g0 < nch; g0 += Gl) {
        const int64_t g1 = std::min(nch, g0 + Gl);
        const int64_t p0 = tab[3 * g0], p1 = tab[3 * (g1 - 1)] + tab[3 * (g1 - 1) + 1];   // CSR positions of the launch
        RidgePressParams<T> pp;
        pp.Z = h->Z.as<T>(); pp.w = h->weighted ? h->w.as<T>() : nullptr; pp.ld = h->ld;
        pp.idx = h->d_idx.as<int64_t>(); pp.chunks = dtab + 3 * g0; pp.stats = h->stats.as<T>();
        pp.flags = h->flags; pp.s = st;
        pp.part = h->ridge_part.as<double>(); pp.part_w = pp.part + (g1 - g0) * width;
        pp.pred = !opred ? nullptr : host ? h->cv_pred.as<T>() : (T*)opred + (off[c0] - off[f0]) * L * M + l0 * M;
        pp.pred_ld = host ? width : L * M;
        pp.pred_pos = host ? p0 : off[c0];
        const dim3 gp((unsigned)(g1 - g0), (unsigned)ridge_cdiv(width, RIDGE_PC));
        k_ridge_press<T><<<gp, RIDGE_THREADS, smem[CVMX_RK_PRESS], h->stream>>>(pp);
        const int64_t fa = tab[3 * g0 + 2], fb = tab[3 * (g1 - 1) + 2] + 1;
        k_ridge_press_accum<<<(unsigned)(fb - fa), RIDGE_THREADS, 0, h->stream>>>(pp.part, pp.part_w, dtab + 3 * nch, g0, g1, fa,
                                                                                  width, acc, acc_w);
        h->launches += 2;
        if (opred && host) {
          T* dst = (T*)opred + (p0 - off[f0]) * L * M + l0 * M;
          if (width == L * M)
            CU(h, cudaMemcpyAsync(dst, pp.pred, (size_t)(p1 - p0) * width * sz, cudaMemcpyDeviceToHost, h->stream));
          else   // a one-fold pass over some of the penalties: a strided slice of the caller's rows
            CU(h, cudaMemcpy2DAsync(dst, (size_t)L * M * sz, pp.pred, (size_t)width * sz, (size_t)width * sz, (size_t)(p1 - p0),
                                    cudaMemcpyDeviceToHost, h->stream));
        }
      }
      k_ridge_finish<T><<<(unsigned)Pn, RIDGE_THREADS, 0, h->stream>>>(st, acc, acc_w, dpress, dinfo, dsumw);
      h->launches++;
      if (dB) {
        const dim3 gc((unsigned)pairs, (unsigned)grid[2 * CVMX_RK_COEFS + 1]);
        k_ridge_coefs<T><<<gc, RIDGE_THREADS, 0, h->stream>>>(st, dB);
        h->launches++;
      }
      CU(h, cudaGetLastError());
      if (host) {
        CU(h, cudaMemcpyAsync((T*)opress + o_pm, dpress, (size_t)pairs * M * sz, kind, h->stream));
        CU(h, cudaMemcpyAsync(oinfo + o_in, dinfo, (size_t)pairs * sizeof(int32_t), kind, h->stream));
        if (oB) CU(h, cudaMemcpyAsync((T*)oB + o_b, dB, (size_t)pairs * K * M * sz, kind, h->stream));
      }
    }
    if (host) {
      CU(h, cudaMemcpyAsync((T*)osumw + d, dsumw, (size_t)Pn * sz, kind, h->stream));
      CU(h, cudaMemcpyAsync(ostatus + d, dstatus, (size_t)Pn * sizeof(int32_t), kind, h->stream));
    }
    // the next window reuses the scratch and the chunk table's host vector
    CU(h, cudaStreamSynchronize(h->stream));
  }
  return CVMX_OK;
}

// offsets: always a host array here; indices: host or device according to `mem`
int32_t upload_csr(cvmx_t* h, DevBuf& doff, DevBuf& didx, const int64_t* offsets, const int64_t* indices, int64_t P,
                   int64_t nidx, int32_t mem) {
  CU(h, doff.reserve((P + 1) * sizeof(int64_t)));
  CU(h, didx.reserve(std::max<int64_t>(nidx, 1) * sizeof(int64_t)));
  CU(h, h->errflag.reserve(sizeof(int32_t)));
  const cudaMemcpyKind kind = mem == CVMX_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
  CU(h, cudaMemcpyAsync(doff.p, offsets, (P + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
  CU(h, cudaMemsetAsync(h->errflag.p, 0, sizeof(int32_t), h->stream));
  if (nidx > 0) {
    CU(h, cudaMemcpyAsync(didx.p, indices, nidx * sizeof(int64_t), kind, h->stream));
    k_normalize_indices<<<(unsigned)((nidx + 255) / 256), 256, 0, h->stream>>>(didx.as<int64_t>(), nidx, h->N, h->errflag.as<int32_t>());
    h->launches++;
    CU(h, cudaGetLastError());
  }
  int32_t bad = 0;
  CU(h, cudaMemcpyAsync(&bad, h->errflag.p, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaStreamSynchronize(h->stream));
  if (bad) return fail(h, CVMX_ERR_INDEX, "validation index out of bounds for the fitted number of rows");
  return CVMX_OK;
}

template <typename T>
int32_t slab_fold_sums(cvmx_t* h, int64_t f0, int64_t f1, void* carry) {
  const int64_t Pn = f1 - f0, ld = h->ld;
  std::vector<int64_t> ranges(2 * Pn);
  int64_t max_rows = 0;
  for (int64_t f = 0; f < Pn; ++f) {
    ranges[2 * f] = h->h_off[f0 + f]; ranges[2 * f + 1] = h->h_off[f0 + f + 1];
    max_rows = std::max(max_rows, ranges[2 * f + 1] - ranges[2 * f]);
  }
  CU(h, h->chunk_ranges.reserve(ranges.size() * sizeof(int64_t)));
  CU(h, cudaMemcpyAsync(h->chunk_ranges.p, ranges.data(), ranges.size() * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
  CU(h, cudaStreamSynchronize(h->stream));   // `ranges` is a local
  MomentParams<T> fc;
  fc.Z = h->Z.as<T>(); fc.w = h->w.as<T>(); fc.ld = ld; fc.K = h->K; fc.M = h->M;
  fc.offsets = nullptr; fc.indices = h->d_idx.as<int64_t>(); fc.fold0 = 0; fc.N = h->N;
  fc.flags = h->flags; fc.resolution = (T)h->resolution;
  fc.sum_z = h->sum_z.as<T>(); fc.sumsq_z = h->sumsq_z.as<T>();
  fc.fs = nullptr; fc.pw_cols = nullptr; fc.stats = nullptr;
  fc.ranges = h->chunk_ranges.as<int64_t>(); fc.raw = (T*)carry; fc.accumulate = 1;
  const int ev0 = prof_mark(h);
  int32_t rc;
  const bool prepared = h->slab_scan_mode == 2 && h->slab_scan_stage == 2 && h->slab_scan_f0 == f0 && h->slab_scan_f1 == f1 &&
                        h->slab_scan_csr == h->csr_version;
  if (prepared) {
    if constexpr (std::is_same<T, double>::value) rc = slab_scan_finish(h, 2, f0, f1, (double*)carry, fc);
    else rc = fail(h, CVMX_ERR_INVALID, "decoupled slab chain: float64 only");
  } else {
    rc = launch_moments<T>(h, fc, Pn, max_rows);
  }
  h->slab_scan_mode = 0; h->slab_scan_stage = 0;
  prof_span(h, PROF_STATS, ev0, prof_mark(h));
  return rc;
}

}  // namespace

// ---- C ABI -------------------------------------------------------------------------------------------
extern "C" {

int32_t cvmx_version(void) { return CVMX_VERSION; }

const char* cvmx_last_error(const cvmx_t* h) { return h ? h->err.c_str() : g_err.c_str(); }

int32_t cvmx_create(int32_t device, int32_t dtype, uint32_t flags, int64_t ddof, double resolution, cvmx_t** out) {
  if (!out) return fail(nullptr, CVMX_ERR_INVALID, "out is NULL");
  *out = nullptr;
  if (dtype != CVMX_F32 && dtype != CVMX_F64) return fail(nullptr, CVMX_ERR_INVALID, "dtype must be CVMX_F32 or CVMX_F64");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, CVMX_ERR_CUDA, std::string("no CUDA device: libcvmx has no CPU fallback (") + cudaGetErrorString(e) + ")");
  if (device < 0 || device >= ndev) return fail(nullptr, CVMX_ERR_INVALID, "device ordinal out of range");
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return fail(nullptr, CVMX_ERR_CUDA, cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(nullptr, CVMX_ERR_CUDA, std::string("libcvmx is built for sm_100a (B200) only; found ") + prop.name);
  cvmx_t* h = new cvmx_handle();
  h->device = device; h->dtype = dtype; h->flags = flags & 15u; h->ddof = ddof; h->resolution = resolution;
  h->sm_count = prop.multiProcessorCount;
  if (const char* e = std::getenv("CVMX_SCAN")) h->scan_mode = std::max(0, std::min(2, std::atoi(e)));
  if (const char* e = std::getenv("CVMX_LOO_EXACT")) h->loo_mode = std::atoi(e) ? 1 : 0;
  if (const char* e = std::getenv("CVMX_SCAN_SPEC")) h->scan_spec = std::atoi(e) ? 1 : 0;
  if (const char* e = std::getenv("CVMX_FUSE_STATS")) h->fuse_stats = std::atoi(e) ? 1 : 0;
  if (const char* e = std::getenv("CVMX_HOST_STAGER")) h->use_stager = std::atoi(e) ? 1 : 0;
  if (const char* e = std::getenv("CVMX_F32_TC")) h->f32_tc = std::max(0, std::min(2, std::atoi(e)));
  DeviceGuard guard__(device);
  if ((e = guard__.err) != cudaSuccess || (e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking)) != cudaSuccess) {
    delete h;
    return fail(nullptr, CVMX_ERR_CUDA, cudaGetErrorString(e));
  }
  h->stream = h->own_stream;
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);   // the chain kernels must get SMs ahead of queued Gram CTAs
  if ((e = cudaStreamCreateWithPriority(&h->aux_stream, cudaStreamNonBlocking, prio_hi)) != cudaSuccess ||
      (e = cudaStreamCreateWithPriority(&h->aux2_stream, cudaStreamNonBlocking, prio_hi)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&h->ev_mass, cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&h->ev_copied[0], cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&h->ev_copied[1], cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&h->ev_stage[0], cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&h->ev_stage[1], cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming)) != cudaSuccess) {
    delete h;
    return fail(nullptr, CVMX_ERR_CUDA, cudaGetErrorString(e));
  }
  *out = h;
  return CVMX_OK;
}

int32_t cvmx_destroy(cvmx_t* h) {
  if (!h) return CVMX_OK;
  DeviceGuard guard__(h->device);
  cudaStreamSynchronize(h->stream);
  for (DevBuf* b : {&h->stat_flags, &h->peer_sum, &h->w_glob, &h->g_off, &h->g_idx, &h->scan_look, &h->loo_ops, &h->Z, &h->w, &h->Ttot, &h->sum_z, &h->sumsq_z, &h->fit_scal, &h->d_off, &h->d_idx, &h->a_off, &h->a_idx,
                    &h->units, &h->tiles, &h->fold_units, &h->split_folds, &h->partials, &h->stats, &h->rawsums, &h->fscal, &h->pwcols,
                    &h->errflag, &h->out_xx, &h->out_xy, &h->out_small, &h->scan_seg, &h->scan_ok, &h->scan_list, &h->scan_cnt, &h->ystage, &h->fold_gram, &h->fold_raw, &h->chunk_ranges,
                    &h->pls_ws, &h->pls_tab, &h->pls_part, &h->pls_out, &h->ridge_ws, &h->ridge_tab, &h->ridge_part, &h->ridge_alpha, &h->cv_pred})
    b->release();
  h->tc_gram.release(); h->tc_finish.release();
  delete h->stager; h->stager = nullptr;
  for (cudaEvent_t e : h->prof_ev) cudaEventDestroy(e);
  if (h->aux_stream) { cudaStreamSynchronize(h->aux_stream); cudaStreamDestroy(h->aux_stream); }
  if (h->aux2_stream) { cudaStreamSynchronize(h->aux2_stream); cudaStreamDestroy(h->aux2_stream); }
  if (h->ev_mass) cudaEventDestroy(h->ev_mass);
  for (int i = 0; i < 2; ++i) {
    if (h->ev_copied[i]) cudaEventDestroy(h->ev_copied[i]);
    if (h->ev_stage[i]) cudaEventDestroy(h->ev_stage[i]);
    h->stage[i].release();
  }
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
  return CVMX_OK;
}

int32_t cvmx_set_stream(cvmx_t* h, void* s) {
  if (!h) return fail(nullptr, CVMX_ERR_INVALID, "handle is NULL");
  ON_DEVICE(h);
  cudaStreamSynchronize(h->stream);
  h->stream = s ? (cudaStream_t)s : h->own_stream;
  return CVMX_OK;
}

int32_t cvmx_sync(cvmx_t* h) {
  if (!h) return fail(nullptr, CVMX_ERR_INVALID, "handle is NULL");
  ON_DEVICE(h);
  CU(h, cudaStreamSynchronize(h->stream));
  return CVMX_OK;
}

int32_t cvmx_fit(cvmx_t* h, const void* X, int64_t N, int64_t K, int64_t ldx, const void* Y, int64_t M, int64_t ldy,
                 const void* w, int32_t mem, int64_t g0, int64_t g1) {
  if (!h) return fail(nullptr, CVMX_ERR_INVALID, "handle is NULL");
  if (!X || N < 0 || K <= 0 || ldx < K || M < 0 || (M > 0 && (!Y || ldy < M)) || g0 < 0 || g1 > N || g0 > g1)
    return fail(h, CVMX_ERR_INVALID, "cvmx_fit: bad shape arguments");
  ON_DEVICE(h);
  if (!Y) M = 0;
  return h->dtype == CVMX_F64 ? fit_impl<double>(h, X, N, K, ldx, Y, M, ldy, w, mem, g0, g1)
                              : fit_impl<float>(h, X, N, K, ldx, Y, M, ldy, w, mem, g0, g1);
}


int32_t cvmx_fit_begin(cvmx_t* h, int64_t N, int64_t K, int64_t M, int32_t weighted, int64_t max_block_rows) {
  if (!h) return fail(nullptr, CVMX_ERR_INVALID, "handle is NULL");
  if (N < 0 || K <= 0 || M < 0 || max_block_rows <= 0) return fail(h, CVMX_ERR_INVALID, "cvmx_fit_begin: bad shape arguments");
  ON_DEVICE(h);
  return h->dtype == CVMX_F64 ? fit_begin_impl<double>(h, N, K, M, weighted, max_block_rows)
                              : fit_begin_impl<float>(h, N, K, M, weighted, max_block_rows);
}

int32_t cvmx_fit_rows(cvmx_t* h, int64_t row0, int64_t nrows, const void* X, int64_t ldx, const void* Y, int64_t ldy, const void* w,
                      int32_t mem, int32_t gram) {
  if (!h || !h->filling) return fail(h, CVMX_ERR_INVALID, "cvmx_fit_rows: call cvmx_fit_begin first");
  if (row0 < 0 || nrows < 0 || row0 + nrows > h->N || (nrows > 0 && !X) || ldx < h->K || (h->M > 0 && nrows > 0 && (!Y || ldy < h->M)) ||
      (h->weighted && nrows > 0 && !w))
    return fail(h, CVMX_ERR_INVALID, "cvmx_fit_rows: bad block arguments");
  if (nrows == 0) return CVMX_OK;
  ON_DEVICE(h);
  return h->dtype == CVMX_F64 ? fit_rows_impl<double>(h, row0, nrows, X, ldx, Y, ldy, w, mem, gram)
                              : fit_rows_impl<float>(h, row0, nrows, X, ldx, Y, ldy, w, mem, gram);
}

int32_t cvmx_fit_end(cvmx_t* h, int32_t col_shard, int32_t n_col_shards) {
  if (!h || !h->filling) return fail(h, CVMX_ERR_INVALID, "cvmx_fit_end: call cvmx_fit_begin first");
  if (n_col_shards < 1 || col_shard < 0 || col_shard >= n_col_shards) return fail(h, CVMX_ERR_INVALID, "cvmx_fit_end: bad column shard");
  ON_DEVICE(h);
  return h->dtype == CVMX_F64 ? fit_end_impl<double>(h, col_shard, n_col_shards) : fit_end_impl<float>(h, col_shard, n_col_shards);
}

int32_t cvmx_data_ptr(cvmx_t* h, void** Z, void** w, int64_t* ld) {
  if (!h || !(h->filling || h->fitted)) return fail(h, CVMX_ERR_INVALID, "cvmx_data_ptr: no data on the device yet");
  if (Z) *Z = h->Z.p;
  if (w) *w = h->w.p;
  if (ld) *ld = h->ld;
  return CVMX_OK;
}

int32_t cvmx_moments_ptr(cvmx_t* h, void** sum_z, void** sumsq_z, int64_t* count) {
  if (!h || !h->fitted) return fail(h, CVMX_ERR_INVALID, "cvmx_moments_ptr: fit first");
  if (sum_z) *sum_z = h->sum_z.p;
  if (sumsq_z) *sumsq_z = h->sumsq_z.p;
  if (count) *count = h->ld;
  return CVMX_OK;
}

int32_t cvmx_totals_ptr(cvmx_t* h, void** p, int64_t* count, int64_t* ld) {
  if (!h || !h->fitted) return fail(h, CVMX_ERR_INVALID, "cvmx_totals_ptr: fit first");
  if (p) *p = h->Ttot.p;
  if (count) *count = h->K * h->ld;
  if (ld) *ld = h->ld;
  return CVMX_OK;
}

int32_t cvmx_commit_totals(cvmx_t* h) {
  if (!h || !h->fitted) return fail(h, CVMX_ERR_INVALID, "cvmx_commit_totals: fit first");
  return CVMX_OK;  // totals are consumed in place; kept as an explicit step of the sharded-fit protocol
}

int32_t cvmx_get_totals(cvmx_t* h, void* XTX, void* XTY, void* sum_X, void* sum_Y, void* sum_sq_X, void* sum_sq_Y,
                        double* sum_w, int64_t* nnz_w) {
  if (!h || !h->fitted) return fail(h, CVMX_ERR_INVALID, "cvmx_get_totals: fit first");
  ON_DEVICE(h);
  const size_t sz = esz(h);
  const int64_t K = h->K, M = h->M, ld = h->ld;
  const char* T = h->Ttot.as<char>();
  if (XTX) CU(h, cudaMemcpy2DAsync(XTX, K * sz, T, ld * sz, K * sz, K, cudaMemcpyDeviceToHost, h->stream));
  if (XTY && M) CU(h, cudaMemcpy2DAsync(XTY, M * sz, T + K * sz, ld * sz, M * sz, K, cudaMemcpyDeviceToHost, h->stream));
  if (sum_X) CU(h, cudaMemcpyAsync(sum_X, h->sum_z.p, K * sz, cudaMemcpyDeviceToHost, h->stream));
  if (sum_Y && M) CU(h, cudaMemcpyAsync(sum_Y, h->sum_z.as<char>() + K * sz, M * sz, cudaMemcpyDeviceToHost, h->stream));
  if (sum_sq_X) CU(h, cudaMemcpyAsync(sum_sq_X, h->sumsq_z.p, K * sz, cudaMemcpyDeviceToHost, h->stream));
  if (sum_sq_Y && M) CU(h, cudaMemcpyAsync(sum_sq_Y, h->sumsq_z.as<char>() + K * sz, M * sz, cudaMemcpyDeviceToHost, h->stream));
  FitScalars fsc;
  CU(h, cudaMemcpyAsync(&fsc, h->fit_scal.p, sizeof(fsc), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaStreamSynchronize(h->stream));
  if (sum_w) *sum_w = fsc.sum_w;
  if (nnz_w) *nnz_w = fsc.nnz_w;
  return CVMX_OK;
}

int32_t cvmx_set_folds(cvmx_t* h, const int64_t* offsets, const int64_t* indices, int64_t P, int32_t mem) {
  if (!h || !h->fitted) return fail(h, CVMX_ERR_INVALID, "cvmx_set_folds: fit first");
  if (!offsets || P < 0) return fail(h, CVMX_ERR_INVALID, "cvmx_set_folds: bad arguments");
  ON_DEVICE(h);
  h->h_off.resize(P + 1);
  if (mem == CVMX_HOST) std::memcpy(h->h_off.data(), offsets, (P + 1) * sizeof(int64_t));
  else CU(h, cudaMemcpy(h->h_off.data(), offsets, (P + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost));
  if (h->h_off[0] != 0) return fail(h, CVMX_ERR_INVALID, "offsets[0] must be 0");
  for (int64_t f = 0; f < P; ++f)
    if (h->h_off[f + 1] < h->h_off[f]) return fail(h, CVMX_ERR_INVALID, "offsets must be non-decreasing");
  const int64_t nidx = h->h_off[P];
  if (nidx > 0 && !indices) return fail(h, CVMX_ERR_INVALID, "indices is NULL");
  h->P = 0; h->csr_version++;
  int32_t rc = upload_csr(h, h->d_off, h->d_idx, h->h_off.data(), indices, P, nidx, mem);
  if (rc) return rc;
  h->P = P;
  return CVMX_OK;
}


int32_t cvmx_fit_folds(cvmx_t* h, const void* X, int64_t N, int64_t K, int64_t ldx, const void* Y, int64_t M, int64_t ldy,
                       const void* w, int32_t mem, const int64_t* offsets, const int64_t* indices, int64_t P, int32_t is_partition) {
  if (!h) return fail(nullptr, CVMX_ERR_INVALID, "handle is NULL");
  if (!X || N < 0 || K <= 0 || ldx < K || M < 0 || (M > 0 && (!Y || ldy < M)) || !offsets || P < 0 || (P > 0 && offsets[P] > 0 && !indices))
    return fail(h, CVMX_ERR_INVALID, "cvmx_fit_folds: bad arguments");
  ON_DEVICE(h);
  if (!Y) M = 0;
  if (offsets[0] != 0) return fail(h, CVMX_ERR_INVALID, "offsets[0] must be 0");
  for (int64_t f = 0; f < P; ++f)
    if (offsets[f + 1] < offsets[f]) return fail(h, CVMX_ERR_INVALID, "offsets must be non-decreasing");
  // the fusion needs a true partition with ascending indices inside every fold
  bool part = P > 0 && offsets[P] == N;
  if (part && !is_partition) {
    std::vector<unsigned char> seen((size_t)N, 0);
    for (int64_t f = 0; f < P && part; ++f)
      for (int64_t i = offsets[f]; i < offsets[f + 1]; ++i) {
        const int64_t r = indices[i];
        if (r < 0 || r >= N || seen[r] || (i > offsets[f] && indices[i - 1] >= r)) { part = false; break; }
        seen[r] = 1;
      }
  }
  FoldFuse ff{offsets, indices, P};
  int32_t rc = h->dtype == CVMX_F64 ? fit_impl<double>(h, X, N, K, ldx, Y, M, ldy, w, mem, 0, N, part ? &ff : nullptr)
                                    : fit_impl<float>(h, X, N, K, ldx, Y, M, ldy, w, mem, 0, N, part ? &ff : nullptr);
  if (rc) return rc;
  if (h->fold_gram_version == h->csr_version) return CVMX_OK;   // fused: the CSR is already resident
  return cvmx_set_folds(h, offsets, indices, P, CVMX_HOST);
}

int32_t cvmx_folds_are_cached(const cvmx_t* h) { return h && h->fitted && h->fold_gram_version == h->csr_version ? 1 : 0; }

int32_t cvmx_training_batch(cvmx_t* h, int64_t f0, int64_t f1, uint32_t want, void* oxx, void* oxy, void* ostats, void* oscal,
                            int32_t* ostatus, int32_t mem) {
  if (!h || !h->fitted) return fail(h, CVMX_ERR_INVALID, "cvmx_training_batch: fit first");
  if (f0 < 0 || f1 > h->P || f0 > f1) return fail(h, CVMX_ERR_INVALID, "cvmx_training_batch: fold range outside the CSR");
  ON_DEVICE(h);
  return h->dtype == CVMX_F64
             ? training_impl<double>(h, h->d_off.as<int64_t>(), h->d_idx.as<int64_t>(), h->h_off.data(), f0, f1, want, oxx, oxy,
                                     ostats, oscal, ostatus, mem, true)
             : training_impl<float>(h, h->d_off.as<int64_t>(), h->d_idx.as<int64_t>(), h->h_off.data(), f0, f1, want, oxx, oxy,
                                    ostats, oscal, ostatus, mem, true);
}

int32_t cvmx_training_indices(cvmx_t* h, const int64_t* val, int64_t n_val, int32_t idx_mem, uint32_t want, void* oxx, void* oxy,
                              void* ostats, void* oscal, int32_t* ostatus, int32_t out_mem) {
  if (!h || !h->fitted) return fail(h, CVMX_ERR_INVALID, "cvmx_training_indices: fit first");
  if (n_val < 0 || (n_val > 0 && !val)) return fail(h, CVMX_ERR_INVALID, "cvmx_training_indices: bad arguments");
  ON_DEVICE(h);
  const int64_t off[2] = {0, n_val};
  int32_t rc = upload_csr(h, h->a_off, h->a_idx, off, val, 1, n_val, idx_mem);
  if (rc) return rc;
  return h->dtype == CVMX_F64
             ? training_impl<double>(h, h->a_off.as<int64_t>(), h->a_idx.as<int64_t>(), off, 0, 1, want, oxx, oxy, ostats, oscal,
                                     ostatus, out_mem, false)
             : training_impl<float>(h, h->a_off.as<int64_t>(), h->a_idx.as<int64_t>(), off, 0, 1, want, oxx, oxy, ostats, oscal,
                                    ostatus, out_mem, false);
}

int32_t cvmx_sharded_stats(cvmx_t* h, int64_t f0, int64_t f1, int32_t col_shard, int32_t n_col_shards, void** stats_dev,
                           int64_t* stats_count) {
  if (!h || !h->fitted) return fail(h, CVMX_ERR_INVALID, "cvmx_sharded_stats: fit first");
  if (f0 < 0 || f1 > h->P || f0 >= f1 || n_col_shards < 1 || col_shard < 0 || col_shard >= n_col_shards)
    return fail(h, CVMX_ERR_INVALID, "cvmx_sharded_stats: bad fold range or shard");
  ON_DEVICE(h);
  int32_t rc = h->dtype == CVMX_F64 ? sharded_stats<double>(h, f0, f1, col_shard, n_col_shards)
                                    : sharded_stats<float>(h, f0, f1, col_shard, n_col_shards);
  if (stats_dev) *stats_dev = h->stats.p;
  if (stats_count) *stats_count = (f1 - f0) * 2 * h->ld;
  return rc;
}

int32_t cvmx_sharded_stats_wait(cvmx_t* h) {
  if (!h || !h->fitted) return fail(h, CVMX_ERR_INVALID, "cvmx_sharded_stats_wait: fit first");
  ON_DEVICE(h);
  CU(h, cudaStreamWaitEvent(h->stream, h->ev_join, 0));
  return CVMX_OK;
}

int64_t cvmx_sharded_gram_count(cvmx_t* h, int64_t f0, int64_t f1, uint32_t want) {
  if (!h || !h->fitted || f1 <= f0) return 0;
  std::vector<int2> tiles;
  plan_tiles(h, want, tiles);
  return (f1 - f0) * (int64_t)tiles.size() * GACC * GTHREADS;
}

int32_t cvmx_sharded_gram(cvmx_t* h, int64_t f0, int64_t f1, uint32_t want, int32_t row_shard, int32_t n_row_shards, double* gram_dev) {
  if (!h || !h->fitted) return fail(h, CVMX_ERR_INVALID, "cvmx_sharded_gram: fit first");
  if (f0 < 0 || f1 > h->P || f0 >= f1 || n_row_shards < 1 || row_shard < 0 || row_shard >= n_row_shards || !gram_dev)
    return fail(h, CVMX_ERR_INVALID, "cvmx_sharded_gram: bad fold range, shard or buffer");
  if ((want & CVMX_WANT_XTY) && h->M == 0) return fail(h, CVMX_ERR_NO_Y, "Response variables `Y` are not provided.");
  ON_DEVICE(h);
  return h->dtype == CVMX_F64 ? sharded_gram<double>(h, f0, f1, want, row_shard, n_row_shards, gram_dev)
                              : sharded_gram<float>(h, f0, f1, want, row_shard, n_row_shards, gram_dev);
}

int32_t cvmx_sharded_finish(cvmx_t* h, int64_t batch_f0, int64_t f0, int64_t f1, uint32_t want, const double* gram_dev, void* oxx,
                            void* oxy, void* ostats, void* oscal, int32_t* ostatus) {
  if (!h || !h->fitted) return fail(h, CVMX_ERR_INVALID, "cvmx_sharded_finish: fit first");
  if (batch_f0 < 0 || f0 < batch_f0 || f1 > h->P || f0 > f1 || !gram_dev)
    return fail(h, CVMX_ERR_INVALID, "cvmx_sharded_finish: bad fold range or buffer");
  ON_DEVICE(h);
  int32_t rc = h->dtype == CVMX_F64 ? sharded_finish<double>(h, batch_f0, f0, f1, want, gram_dev, (double*)oxx, (double*)oxy)
                                    : sharded_finish<float>(h, batch_f0, f0, f1, want, gram_dev, (float*)oxx, (float*)oxy);
  if (rc || f1 == f0) return rc;
  // statistics / scalars of the owned folds (device pointers)
  const size_t sz = esz(h);
  const int64_t C = h->K + h->M, d = f0 - batch_f0, Pn = f1 - f0;
  if (ostats)
    CU(h, cudaMemcpy2DAsync(ostats, C * sz, h->stats.as<char>() + (size_t)d * 2 * h->ld * sz, h->ld * sz, C * sz, Pn * 2,
                            cudaMemcpyDeviceToDevice, h->stream));
  if (oscal || ostatus) {
    if (h->dtype == CVMX_F64)
      k_pack_scalars<double><<<(unsigned)((Pn + 255) / 256), 256, 0, h->stream>>>(h->fscal.as<FoldScalars>() + d, Pn, (double*)oscal, ostatus);
    else
      k_pack_scalars<float><<<(unsigned)((Pn + 255) / 256), 256, 0, h->stream>>>(h->fscal.as<FoldScalars>() + d, Pn, (float*)oscal, ostatus);
    h->launches++;
    CU(h, cudaGetLastError());
  }
  return CVMX_OK;
}


int32_t cvmx_sharded_finish_peers(cvmx_t* h, int64_t batch_f0, int64_t batch_f1, int64_t f0, int64_t f1, uint32_t want,
                                  const void* const* peer_bufs, int32_t n_peers, int64_t gram_count, void* oxx, void* oxy, void* ostats,
                                  void* oscal, int32_t* ostatus) {
  if (!h || !h->fitted) return fail(h, CVMX_ERR_INVALID, "cvmx_sharded_finish_peers: fit first");
  if (batch_f0 < 0 || f0 < batch_f0 || f1 > batch_f1 || batch_f1 > h->P || f0 > f1 || !peer_bufs || n_peers < 1 || n_peers > 8)
    return fail(h, CVMX_ERR_INVALID, "cvmx_sharded_finish_peers: bad fold range or peer list (at most 8 peers)");
  if (h->dtype != CVMX_F64) return fail(h, CVMX_ERR_INVALID, "cvmx_sharded_finish_peers: float64 handles only");
  ON_DEVICE(h);
  // statistics rows of the whole batch: sum of the peers' column shards, straight into the statistics buffer
  if (gram_count >= 0) {   // (negative: the handle's own statistics are already complete - row-slab mode)
    const int64_t nst = (batch_f1 - batch_f0) * 2 * h->ld;
    PeerList pl8;
    for (int q = 0; q < 8; ++q) pl8.p[q] = q < n_peers ? (const double*)peer_bufs[q] : nullptr;
    k_peer_sum_rows<double><<<(unsigned)((nst + 255) / 256), 256, 0, h->stream>>>(pl8, n_peers, gram_count, nst, h->stats.as<double>());
    h->launches++;
    CU(h, cudaGetLastError());
  }
  if (f1 == f0) return CVMX_OK;
  // the owned folds' raw Grams: sum of the peers' buffers at NVLink bandwidth, then the ordinary local epilogue
  std::vector<int2> tiles;
  plan_tiles(h, want, tiles);
  const int64_t per_fold = (int64_t)tiles.size() * GACC * GTHREADS, nsum = (f1 - f0) * per_fold;
  CU(h, h->peer_sum.reserve((size_t)nsum * sizeof(double)));
  PeerList pg8;
  for (int q = 0; q < 8; ++q) pg8.p[q] = q < n_peers ? (const double*)peer_bufs[q] : nullptr;
  const int ev0 = prof_mark(h);
  k_peer_sum_frags<<<(unsigned)((nsum / 2 + 255) / 256), 256, 0, h->stream>>>(pg8, n_peers, (f0 - batch_f0) * per_fold, nsum, h->peer_sum.as<double>());
  h->launches++;
  prof_span(h, PROF_REDUCE, ev0, prof_mark(h));
  CU(h, cudaGetLastError());
  int32_t rc = sharded_finish<double>(h, batch_f0, f0, f1, want, h->peer_sum.as<double>(), (double*)oxx, (double*)oxy, nullptr, 0, true);
  if (rc) return rc;
  const size_t sz = 8;
  const int64_t C = h->K + h->M, d = f0 - batch_f0, Pn = f1 - f0;
  if (ostats)
    CU(h, cudaMemcpy2DAsync(ostats, C * sz, h->stats.as<char>() + (size_t)d * 2 * h->ld * sz, h->ld * sz, C * sz, Pn * 2,
                            cudaMemcpyDeviceToDevice, h->stream));
  if (oscal || ostatus) {
    k_pack_scalars<double><<<(unsigned)((Pn + 255) / 256), 256, 0, h->stream>>>(h->fscal.as<FoldScalars>() + d, Pn, (double*)oscal, ostatus);
    h->launches++;
    CU(h, cudaGetLastError());
  }
  return CVMX_OK;
}



// ---- row-slab mode: this handle holds rows [row0, row0 + N) of an N_glob-row data set -------------------------------
int32_t cvmx_fit_end_slab(cvmx_t* h, const void* carry_sum, const void* carry_sumsq, const void* w_glob, int64_t N_glob, int64_t row0) {
  if (!h || !h->filling) return fail(h, CVMX_ERR_INVALID, "cvmx_fit_end_slab: call cvmx_fit_begin first");
  if (N_glob < h->N || row0 < 0 || row0 + h->N > N_glob || (h->weighted && !w_glob) || ((carry_sum == nullptr) != (carry_sumsq == nullptr)))
    return fail(h, CVMX_ERR_INVALID, "cvmx_fit_end_slab: bad slab arguments");
  if (h->K < 2 || h->M == 1)
    return fail(h, CVMX_ERR_INVALID, "cvmx_fit_end_slab: row slabs need K >= 2 and M != 1 (single columns are summed pairwise over all rows)");
  ON_DEVICE(h);
  SlabArgs sl{carry_sum, carry_sumsq, w_glob, N_glob, row0};
  return h->dtype == CVMX_F64 ? fit_end_impl<double>(h, 0, 1, &sl) : fit_end_impl<float>(h, 0, 1, &sl);
}

int32_t cvmx_slab_begin(cvmx_t* h, const void* w_glob, int64_t N_glob, int64_t row0) {
  if (!h || !h->filling) return fail(h, CVMX_ERR_INVALID, "cvmx_slab_begin: call cvmx_fit_begin first");
  if (N_glob < h->N || row0 < 0 || row0 + h->N > N_glob || (h->weighted && !w_glob)) return fail(h, CVMX_ERR_INVALID, "cvmx_slab_begin: bad slab arguments");
  if (h->K < 2 || h->M == 1) return fail(h, CVMX_ERR_INVALID, "cvmx_slab_begin: row slabs need K >= 2 and M != 1");
  ON_DEVICE(h);
  const size_t sz = esz(h);
  if (h->weighted) {
    CU(h, h->w_glob.reserve((size_t)std::max<int64_t>(N_glob, 1) * sz));
    CU(h, cudaMemcpyAsync(h->w_glob.p, w_glob, (size_t)N_glob * sz, cudaMemcpyDeviceToDevice, h->stream));
  }
  h->slab = true; h->N_glob = N_glob; h->row0 = row0;
  CU(h, cudaEventRecord(h->ev_mass, h->stream));
  CU(h, cudaStreamWaitEvent(h->aux2_stream, h->ev_mass, 0));
  if (h->dtype == CVMX_F64)
    k_weight_mass<double, PW_LEVELS_BIG><<<1, 1 << PW_LEVELS_BIG, 0, h->aux2_stream>>>(
        h->Z.as<double>(), h->weighted ? h->w_glob.as<double>() : h->w.as<double>(), h->ld, N_glob, h->K, h->M, h->weighted ? 1 : 0, nullptr, nullptr, 0,
        1, h->ddof, h->fit_scal.as<FitScalars>(), nullptr, h->pwcols.as<double>());
  else
    k_weight_mass<float, PW_LEVELS_BIG><<<1, 1 << PW_LEVELS_BIG, 0, h->aux2_stream>>>(
        h->Z.as<float>(), h->weighted ? h->w_glob.as<float>() : h->w.as<float>(), h->ld, N_glob, h->K, h->M, h->weighted ? 1 : 0, nullptr, nullptr, 0,
        1, h->ddof, h->fit_scal.as<FitScalars>(), nullptr, h->pwcols.as<float>());
  h->launches++;
  CU(h, cudaGetLastError());
  CU(h, cudaEventRecord(h->ev_mass, h->aux2_stream));
  h->mass_started = true; h->mass_pending = true;
  return CVMX_OK;
}

int32_t cvmx_slab_scan_local(cvmx_t* h, int64_t f0, int64_t f1, const void* w_glob, int64_t N_glob, int64_t row0, double* tot_out,
                             int32_t* applicable) {
  if (!h || !tot_out || !applicable) return fail(h, CVMX_ERR_INVALID, "cvmx_slab_scan_local: null argument");
  *applicable = 0;
  const bool fit_mode = f0 < 0;
  if (fit_mode) {
    if (!h->filling) return fail(h, CVMX_ERR_INVALID, "cvmx_slab_scan_local: fit totals need cvmx_fit_begin / cvmx_fit_rows first");
    if (N_glob < h->N || row0 < 0 || row0 + h->N > N_glob || (h->weighted && !w_glob)) return fail(h, CVMX_ERR_INVALID, "cvmx_slab_scan_local: bad slab arguments");
    if (h->K < 2 || h->M == 1) return fail(h, CVMX_ERR_INVALID, "cvmx_slab_scan_local: row slabs need K >= 2 and M != 1");
  } else {
    if (!h->fitted || !h->slab) return fail(h, CVMX_ERR_INVALID, "cvmx_slab_scan_local: fit a row slab first (cvmx_fit_end_slab)");
    if (f1 > h->P || f0 >= f1) return fail(h, CVMX_ERR_INVALID, "cvmx_slab_scan_local: bad fold range");
  }
  if (h->dtype != CVMX_F64) return CVMX_OK;   // float32 chains have no scan: the caller keeps the serial hand-over
  ON_DEVICE(h);
  bool app = false;
  if (fit_mode) {
    // everything of cvmx_fit_end_slab that does not depend on the previous slab: global weights, accumulator -> totals, weight mass
    if (h->weighted && !h->mass_started) {
      CU(h, h->w_glob.reserve((size_t)std::max<int64_t>(N_glob, 1) * sizeof(double)));
      CU(h, cudaMemcpyAsync(h->w_glob.p, w_glob, (size_t)N_glob * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    }
    h->slab = true; h->N_glob = N_glob; h->row0 = row0;
    int32_t rp = fit_end_pre<double>(h, true, N_glob, true);
    if (rp) return rp;
    h->fit_pre_done = true;
  }
  int32_t rc = slab_scan_local(h, fit_mode ? 1 : 2, fit_mode ? 0 : f0, fit_mode ? 1 : f1, tot_out, app);
  *applicable = app ? 1 : 0;
  return rc;
}

int32_t cvmx_slab_scan_prepare(cvmx_t* h, int64_t f0, int64_t f1, const double* start) {
  if (!h || !start) return fail(h, CVMX_ERR_INVALID, "cvmx_slab_scan_prepare: null argument");
  const bool fit_mode = f0 < 0;
  const int mode = fit_mode ? 1 : 2;
  if (fit_mode) { f0 = 0; f1 = 1; }
  if (h->slab_scan_mode != mode || h->slab_scan_stage != 1 || h->slab_scan_f0 != f0 || h->slab_scan_f1 != f1 ||
      (mode == 2 && h->slab_scan_csr != h->csr_version))
    return fail(h, CVMX_ERR_INVALID, "cvmx_slab_scan_prepare: call cvmx_slab_scan_local for the same sums first");
  ON_DEVICE(h);
  return slab_scan_prepare(h, mode, f0, f1, start);
}

int32_t cvmx_set_weight_folds(cvmx_t* h, const int64_t* offsets, const int64_t* indices, int64_t P) {
  if (!h || !h->fitted || !h->slab) return fail(h, CVMX_ERR_INVALID, "cvmx_set_weight_folds: fit a row slab first (cvmx_fit_end_slab)");
  if (!offsets || P != h->P || (offsets[P] > 0 && !indices)) return fail(h, CVMX_ERR_INVALID, "cvmx_set_weight_folds: one global index set per fold of cvmx_set_folds");
  ON_DEVICE(h);
  h->g_h_off.assign(offsets, offsets + P + 1);
  const int64_t N_local = h->N;
  h->N = h->N_glob;   // upload_csr normalises against h->N
  int32_t rc = upload_csr(h, h->g_off, h->g_idx, offsets, indices, P, offsets[P], CVMX_HOST);
  h->N = N_local;
  return rc;
}

int32_t cvmx_slab_fold_sums(cvmx_t* h, int64_t f0, int64_t f1, void* carry) {
  if (!h || !h->fitted || !h->slab) return fail(h, CVMX_ERR_INVALID, "cvmx_slab_fold_sums: fit a row slab first (cvmx_fit_end_slab)");
  if (f0 < 0 || f1 > h->P || f0 >= f1 || !carry) return fail(h, CVMX_ERR_INVALID, "cvmx_slab_fold_sums: bad fold range or buffer");
  ON_DEVICE(h);
  return h->dtype == CVMX_F64 ? slab_fold_sums<double>(h, f0, f1, carry) : slab_fold_sums<float>(h, f0, f1, carry);
}

int32_t cvmx_slab_finalize_stats(cvmx_t* h, int64_t f0, int64_t f1, const void* raw) {
  if (!h || !h->fitted || !h->slab) return fail(h, CVMX_ERR_INVALID, "cvmx_slab_finalize_stats: fit a row slab first (cvmx_fit_end_slab)");
  if (f0 < 0 || f1 > h->P || f0 >= f1 || !raw || (int64_t)h->g_h_off.size() != h->P + 1)
    return fail(h, CVMX_ERR_INVALID, "cvmx_slab_finalize_stats: bad fold range / buffer, or cvmx_set_weight_folds not called");
  ON_DEVICE(h);
  int64_t max_rows = 0;
  for (int64_t f = f0; f < f1; ++f) max_rows = std::max(max_rows, h->h_off[f + 1] - h->h_off[f]);
  return h->dtype == CVMX_F64
             ? launch_fold_stats<double>(h, h->d_off.as<int64_t>(), h->d_idx.as<int64_t>(), f0, f1 - f0, max_rows, 0, 1, 0.0, (const double*)raw)
             : launch_fold_stats<float>(h, h->d_off.as<int64_t>(), h->d_idx.as<int64_t>(), f0, f1 - f0, max_rows, 0, 1, 0.0, (const float*)raw);
}

int32_t cvmx_validation_rows(cvmx_t* h, int64_t fold, const void* stats, uint32_t apply, void* out_X, void* out_Y, int32_t mem) {
  if (!h || !h->fitted) return fail(h, CVMX_ERR_INVALID, "cvmx_validation_rows: fit first");
  if (fold < 0 || fold >= h->P) return fail(h, CVMX_ERR_INVALID, "cvmx_validation_rows: fold outside the CSR");
  if (apply && !stats) return fail(h, CVMX_ERR_INVALID, "cvmx_validation_rows: statistics needed for centring / scaling");
  ON_DEVICE(h);
  return h->dtype == CVMX_F64 ? validation_rows_impl<double>(h, fold, stats, apply, out_X, out_Y, mem)
                              : validation_rows_impl<float>(h, fold, stats, apply, out_X, out_Y, mem);
}

int32_t cvmx_pls_cv(cvmx_t* h, int64_t f0, int64_t f1, int64_t n_components, void* out_press, void* out_sum_w_val, void* out_B,
                    int32_t* out_n_fitted, int32_t* out_status, int32_t mem) {
  return cvmx_pls_cv_predict(h, f0, f1, n_components, out_press, out_sum_w_val, out_B, out_n_fitted, out_status, nullptr, mem);
}

int32_t cvmx_pls_cv_predict(cvmx_t* h, int64_t f0, int64_t f1, int64_t n_components, void* out_press, void* out_sum_w_val,
                            void* out_B, int32_t* out_n_fitted, int32_t* out_status, void* out_pred, int32_t mem) {
  if (!h || !h->fitted) return fail(h, CVMX_ERR_INVALID, "cvmx_pls_cv: fit first");
  if (h->slab) return fail(h, CVMX_ERR_INVALID, "cvmx_pls_cv: not available for a row-slab handle");
  if (f0 < 0 || f1 > h->P || f0 > f1) return fail(h, CVMX_ERR_INVALID, "cvmx_pls_cv: fold range outside the CSR");
  if (h->M == 0) return fail(h, CVMX_ERR_NO_Y, "Response variables `Y` are not provided.");
  if (n_components < 1 || n_components > h->K)
    return fail(h, CVMX_ERR_INVALID, "n_components must be between 1 and the number of columns of X (" + std::to_string(h->K) + ")");
  if (h->M > PLS_MAX_M)
    return fail(h, CVMX_ERR_INVALID, "cvmx_pls_cv: at most " + std::to_string(PLS_MAX_M) + " response columns are supported");
  if (f1 > f0 && (!out_press || !out_sum_w_val || !out_n_fitted || !out_status))
    return fail(h, CVMX_ERR_INVALID, "cvmx_pls_cv: an output pointer is NULL");
  ON_DEVICE(h);
  return h->dtype == CVMX_F64
             ? pls_cv_impl<double>(h, f0, f1, n_components, out_press, out_sum_w_val, out_B, out_n_fitted, out_status, out_pred, mem)
             : pls_cv_impl<float>(h, f0, f1, n_components, out_press, out_sum_w_val, out_B, out_n_fitted, out_status, out_pred, mem);
}

int32_t cvmx_ridge_plan(int64_t K, int64_t M, int64_t L, int64_t P, int32_t dtype, int32_t mem, int32_t want_B, int64_t* plan) {
  if (!plan) return fail(nullptr, CVMX_ERR_INVALID, "cvmx_ridge_plan: plan is NULL");
  const int32_t rc = ridge_plan(K, M, L, P, dtype, mem, want_B, plan);
  return rc ? fail(nullptr, rc, "cvmx_ridge_plan: the shape cannot run within the device limits") : CVMX_OK;
}

int32_t cvmx_ridge_cv(cvmx_t* h, int64_t f0, int64_t f1, const double* alphas, int64_t L, void* out_press, void* out_sum_w_val,
                      void* out_B, int32_t* out_info, int32_t* out_status, int32_t mem) {
  return cvmx_ridge_cv_predict(h, f0, f1, alphas, L, out_press, out_sum_w_val, out_B, out_info, out_status, nullptr, mem);
}

int32_t cvmx_ridge_cv_predict(cvmx_t* h, int64_t f0, int64_t f1, const double* alphas, int64_t L, void* out_press,
                              void* out_sum_w_val, void* out_B, int32_t* out_info, int32_t* out_status, void* out_pred,
                              int32_t mem) {
  if (!h || !h->fitted) return fail(h, CVMX_ERR_INVALID, "cvmx_ridge_cv: fit first");
  if (h->slab) return fail(h, CVMX_ERR_INVALID, "cvmx_ridge_cv: not available for a row-slab handle");
  if (f0 < 0 || f1 > h->P || f0 > f1) return fail(h, CVMX_ERR_INVALID, "cvmx_ridge_cv: fold range outside the CSR");
  if (h->M == 0) return fail(h, CVMX_ERR_NO_Y, "Response variables `Y` are not provided.");
  if (h->M > RIDGE_MAX_M)
    return fail(h, CVMX_ERR_INVALID, "cvmx_ridge_cv: at most " + std::to_string(RIDGE_MAX_M) + " response columns are supported");
  if (!alphas || L < 1 || L > RIDGE_MAX_L)
    return fail(h, CVMX_ERR_INVALID, "cvmx_ridge_cv: alphas must hold between 1 and " + std::to_string(RIDGE_MAX_L) + " penalties");
  for (int64_t l = 0; l < L; ++l)
    if (!(alphas[l] >= 0.0 && alphas[l] <= 1.7976931348623157e308))
      return fail(h, CVMX_ERR_INVALID, "cvmx_ridge_cv: every penalty must be finite and >= 0");
  if (mem != CVMX_HOST && mem != CVMX_DEVICE) return fail(h, CVMX_ERR_INVALID, "cvmx_ridge_cv: mem must be CVMX_HOST or CVMX_DEVICE");
  if (f1 > f0 && (!out_press || !out_sum_w_val || !out_info || !out_status))
    return fail(h, CVMX_ERR_INVALID, "cvmx_ridge_cv: an output pointer is NULL");
  int64_t plan[CVMX_RIDGE_PLAN_LEN];
  if (ridge_plan(h->K, h->M, L, f1 - f0, h->dtype, mem, out_B != nullptr, plan) != CVMX_OK || plan[CVMX_RIDGE_FEASIBLE] != 1)
    return fail(h, CVMX_ERR_INVALID, "cvmx_ridge_cv: K = " + std::to_string(h->K) + ", M = " + std::to_string(h->M) +
                                         " cannot run within the device limits");
  ON_DEVICE(h);
  return h->dtype == CVMX_F64
             ? ridge_cv_impl<double>(h, f0, f1, alphas, L, out_press, out_sum_w_val, out_B, out_info, out_status, out_pred, mem, plan)
             : ridge_cv_impl<float>(h, f0, f1, alphas, L, out_press, out_sum_w_val, out_B, out_info, out_status, out_pred, mem, plan);
}

int32_t cvmx_profile_enable(cvmx_t* h, int32_t on) {
  if (!h) return fail(nullptr, CVMX_ERR_INVALID, "handle is NULL");
  ON_DEVICE(h);
  CU(h, cudaStreamSynchronize(h->stream));
  h->prof = on != 0;
  h->prof_spans.clear();
  h->prof_used = 0;
  return CVMX_OK;
}

int32_t cvmx_profile_read(cvmx_t* h, double* ms, int64_t* count) {
  if (!h) return fail(nullptr, CVMX_ERR_INVALID, "handle is NULL");
  ON_DEVICE(h);
  CU(h, cudaStreamSynchronize(h->stream));
  for (int k = 0; k < PROF_KINDS; ++k) { if (ms) ms[k] = 0; if (count) count[k] = 0; }
  for (auto& sp : h->prof_spans) {
    float t = 0;
    CU(h, cudaEventElapsedTime(&t, h->prof_ev[sp.second.first], h->prof_ev[sp.second.second]));
    if (ms) ms[sp.first] += t;
    if (count) count[sp.first] += 1;
  }
  h->prof_spans.clear();
  h->prof_used = 0;
  return CVMX_OK;
}

// Host-side CSR builder for integer fold labels (no device work): labels in [lo, lo + span) -> fold order by first
// appearance, offsets and ascending row indices, in two O(N) counting passes.  scratch: 2 * span int64.
// Serial form: two passes, folds numbered by first appearance.
static int64_t partition_labels_serial(const int64_t* labels, int64_t n, int64_t lo, int64_t span, int64_t* scratch, int64_t* first_rows,
                                       int64_t* offsets, int64_t* indices) {
  int64_t* slot = scratch;          // label -> fold position (-1: unseen)
  int64_t* count = scratch + span;  // per fold position
  for (int64_t l = 0; l < span; ++l) { slot[l] = -1; count[l] = 0; }
  int64_t n_folds = 0;
  for (int64_t i = 0; i < n; ++i) {
    const int64_t l = labels[i] - lo;
    if (l < 0 || l >= span) return -1;
    int64_t s = slot[l];
    if (s < 0) { s = slot[l] = n_folds; first_rows[n_folds++] = i; }
    count[s]++;
  }
  offsets[0] = 0;
  for (int64_t s = 0; s < n_folds; ++s) { offsets[s + 1] = offsets[s] + count[s]; count[s] = offsets[s]; }
  for (int64_t i = 0; i < n; ++i) indices[count[slot[labels[i] - lo]]++] = i;
  return n_folds;
}

// Threaded form for long label arrays with few distinct labels (K-fold / leave-many-out at N = 1M: the serial passes are
// 2-3 ms of a 20-80 ms end-to-end step): every thread histograms a contiguous chunk of the rows and notes the first row of
// each label it sees; the chunks' histograms give every (chunk, fold) its own output range, so the scatter is parallel,
// stable, and needs no atomics.  Same result as the serial form, element for element.
static int64_t partition_labels_threaded(const int64_t* labels, int64_t n, int64_t lo, int64_t span, int64_t* scratch, int64_t* first_rows,
                                         int64_t* offsets, int64_t* indices, int nthreads) {
  // per-thread tables padded to whole cache lines: with five labels all threads' counters would otherwise share one line
  const size_t stride = ((size_t)span + 7) / 8 * 8 + 8;
  std::vector<int64_t> hist((size_t)nthreads * stride, 0), first((size_t)nthreads * stride, -1);
  std::vector<int> bad((size_t)nthreads * 16, 0);
  auto chunk = [&](int t) { return std::make_pair(n * t / nthreads, n * (t + 1) / nthreads); };
  {
    std::vector<std::thread> th;
    for (int t = 0; t < nthreads; ++t)
      th.emplace_back([&, t] {
        int64_t* h = hist.data() + (size_t)t * stride;
        int64_t* f = first.data() + (size_t)t * stride;
        const auto [b, e] = chunk(t);
        for (int64_t i = b; i < e; ++i) {
          const int64_t l = labels[i] - lo;
          if (l < 0 || l >= span) { bad[(size_t)t * 16] = 1; return; }
          if (h[l]++ == 0) f[l] = i;
        }
      });
    for (auto& x : th) x.join();
  }
  for (int t = 0; t < nthreads; ++t) if (bad[(size_t)t * 16]) return -1;
  int64_t* slot = scratch;          // label -> fold position (-1: unseen)
  int64_t* count = scratch + span;  // label -> number of rows
  std::vector<std::pair<int64_t, int64_t>> seen;   // (first row, label)
  for (int64_t l = 0; l < span; ++l) {
    int64_t fr = -1, c = 0;
    for (int t = 0; t < nthreads; ++t) {
      c += hist[(size_t)t * stride + l];
      if (fr < 0) fr = first[(size_t)t * stride + l];   // chunks are in row order: the first chunk that saw the label
    }
    slot[l] = -1; count[l] = c;
    if (c > 0) seen.emplace_back(fr, l);
  }
  std::sort(seen.begin(), seen.end());
  const int64_t n_folds = (int64_t)seen.size();
  offsets[0] = 0;
  for (int64_t s = 0; s < n_folds; ++s) {
    slot[seen[s].second] = s; first_rows[s] = seen[s].first;
    offsets[s + 1] = offsets[s] + count[seen[s].second];
  }
  // hist[t][l] -> first output position of chunk t's rows of label l
  for (int64_t l = 0; l < span; ++l) {
    if (slot[l] < 0) continue;
    int64_t pos = offsets[slot[l]];
    for (int t = 0; t < nthreads; ++t) { const int64_t c = hist[(size_t)t * stride + l]; hist[(size_t)t * stride + l] = pos; pos += c; }
  }
  {
    std::vector<std::thread> th;
    for (int t = 0; t < nthreads; ++t)
      th.emplace_back([&, t] {
        int64_t* pos = hist.data() + (size_t)t * stride;
        const auto [b, e] = chunk(t);
        for (int64_t i = b; i < e; ++i) indices[pos[labels[i] - lo]++] = i;
      });
    for (auto& x : th) x.join();
  }
  return n_folds;
}

int64_t cvmx_partition_labels(const int64_t* labels, int64_t n, int64_t lo, int64_t span, int64_t* scratch,
                              int64_t* first_rows /* span */, int64_t* offsets /* span + 1 */, int64_t* indices /* n */) {
  if (!labels || n < 0 || span <= 0 || !scratch || !first_rows || !offsets || !indices) return -1;
  int nthreads = 1;
  if (n >= 200000 && span <= 4096) {
    nthreads = (int)std::min<unsigned>(8u, std::max(1u, std::thread::hardware_concurrency()));
    if (const char* e = std::getenv("CVMX_PARTITION_THREADS")) nthreads = std::max(1, std::min(64, std::atoi(e)));
  }
  if (nthreads > 1) {
    try {
      return partition_labels_threaded(labels, n, lo, span, scratch, first_rows, offsets, indices, nthreads);
    } catch (...) {   // no threads / no memory for the per-thread histograms: the serial passes need neither
    }
  }
  return partition_labels_serial(labels, n, lo, span, scratch, first_rows, offsets, indices);
}

int64_t cvmx_launch_count(const cvmx_t* h) { return h ? h->launches : 0; }
int64_t cvmx_scan_launch_count(const cvmx_t* h) { return h ? h->scan_launches : 0; }
int32_t cvmx_set_scan_mode(cvmx_t* h, int32_t mode) {
  if (!h || mode < 0 || mode > 2) return fail(h, CVMX_ERR_INVALID, "cvmx_set_scan_mode: mode must be 0, 1 or 2");
  h->scan_mode = mode;
  return CVMX_OK;
}
int32_t cvmx_set_loo_mode(cvmx_t* h, int32_t mode) {
  if (!h || mode < 0 || mode > 1) return fail(h, CVMX_ERR_INVALID, "cvmx_set_loo_mode: mode must be 0 (streaming) or 1 (exact)");
  h->loo_mode = mode;
  return CVMX_OK;
}
int64_t cvmx_ld(const cvmx_t* h) { return h ? h->ld : 0; }

}  // extern "C"
