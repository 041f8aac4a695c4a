// C-ABI entry points of the fused Hamming sweeps (see pg_sweep.cuh and
// include/prograph_b200.h).  Host-side work here: geometry (row blocks x stream splits),
// workspace carving, the split-merge / finalise kernels and the launch bookkeeping.
#include <vector>
#include <mutex>

#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <cub/device/device_radix_sort.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <cstdlib>
#include <cmath>

#include <algorithm>

#include "pg_sweep.cuh"
#include "pg_sweep_sym.cuh"

namespace pg {

// ---- launch timing (CUDA events on the launch stream; read by bench.py) ------------
static std::mutex g_time_mu;
static bool g_time_enabled = false;
static std::vector<std::pair<cudaEvent_t, cudaEvent_t>> g_time_events;

struct SweepTimer {
  cudaEvent_t a = nullptr, b = nullptr;
  cudaStream_t s;
  explicit SweepTimer(cudaStream_t stream) : s(stream) {
    std::lock_guard<std::mutex> g(g_time_mu);
    if (!g_time_enabled) return;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    cudaEventRecord(a, s);
  }
  ~SweepTimer() {
    if (!a) return;
    cudaEventRecord(b, s);
    std::lock_guard<std::mutex> g(g_time_mu);
    g_time_events.emplace_back(a, b);
  }
};

// ---- geometry -------------------------------------------------------------------
struct Geometry {
  int n_rowblocks, n_splits, tiles_per_split, n_tiles, tile_cols;
};

static int tile_cols_for(int words) { return words > 16 ? 32 : 512 / words; }   // long rows: pg_sweep_long.cu

// Splits of the stream shorten the persistent grid's last wave, but every split restarts its
// kNN lists from empty.  Pick the split count that minimises a small cost model (in units of
// "stream rows swept by one CTA"): waves(S) * (cols/S + c_ins * k1 * (1 + ln(cols/(S*k1)))),
// c_ins ~ 18 = a warp-cooperative insertion stalls its 32 rows for about 0.6 stream rows
// (measured: profiles/r1_ncu_notes.md).  k1 = 0 (count / fill / tile) only balances the waves.
static Geometry make_geometry(long long rows, long long stream_rows, int words, int rows_per_cta = kConsumers,
                              int k1 = 17, long long split_limit = 64) {
  Geometry g;
  g.tile_cols = tile_cols_for(words);
  g.n_rowblocks = static_cast<int>(ceil_div(rows, rows_per_cta));
  g.n_tiles = static_cast<int>(ceil_div(stream_rows, g.tile_cols));
  const double resident = static_cast<double>(num_sms()) * 2;
  long long max_splits = g.n_tiles / 8;      // keep >= 8 ring tiles per item
  if (max_splits > 64) max_splits = 64;
  if (max_splits > split_limit) max_splits = split_limit;
  if (max_splits < 1) max_splits = 1;
  long long best_s = 1;
  double best_cost = 1e300;
  for (long long s = 1; s <= max_splits; ++s) {
    const long long tps = ceil_div(g.n_tiles, s);
    const long long real_s = ceil_div(g.n_tiles, tps);
    const double cols = static_cast<double>(tps) * g.tile_cols;
    double waves = static_cast<double>(g.n_rowblocks) * real_s / resident;
    waves = waves < 1.0 ? 1.0 : static_cast<double>(static_cast<long long>(waves + 0.999999));
    double item = cols + 64.0;               // fixed per-item cost: own-row load, list write-back
    if (k1 > 0) {
      const double ratio = cols / k1;
      item += 18.0 * k1 * (1.0 + (ratio > 1.0 ? log(ratio) : 0.0));
    }
    const double cost = waves * item;
    if (cost < best_cost * 0.999) { best_cost = cost; best_s = s; }
  }
  if (const char* ev = std::getenv("PG_SWEEP_SPLITS")) {
    best_s = std::atoll(ev);
    if (best_s < 1) best_s = 1;
    if (best_s > g.n_tiles) best_s = g.n_tiles;
    if (best_s > split_limit) best_s = split_limit;
  }
  g.tiles_per_split = static_cast<int>(ceil_div(g.n_tiles, best_s));
  g.n_splits = static_cast<int>(ceil_div(g.n_tiles, g.tiles_per_split));
  return g;
}

int sweep_long_p5(const SweepParams& prm, const SweepLaunch& l, int words);   // pg_sweep_long.cu
int sweep_wide_p5(const SweepParams& prm, const SweepLaunch& l, int words);   // pg_sweep_wide.cu
int sweep_wide_p8(const SweepParams& prm, const SweepLaunch& l, int words);

static bool long_rows(int planes, int words) { return planes == 5 && words > 16 && words <= 56 && words % 8 == 0; }
// the chunked long-row sweep: P = 5 beyond 1792 residues, P = 8 beyond 256, both up to 32768
static bool wide_rows(int planes, int words) {
  return words % 8 == 0 && words <= kWideMaxWords && ((planes == 5 && words > 56) || (planes == 8 && words > 8));
}

static int dispatch(int planes, int words, const SweepParams& prm, const SweepLaunch& l) {
  if (long_rows(planes, words)) return sweep_long_p5(prm, l, words);
  if (wide_rows(planes, words)) return planes == 5 ? sweep_wide_p5(prm, l, words) : sweep_wide_p8(prm, l, words);
#define PG_CASE(P, W) \
  if (planes == P && words == W) return sweep_p##P##_w##W(prm, l);
  PG_CASE(5, 1) PG_CASE(5, 2) PG_CASE(5, 4) PG_CASE(5, 8) PG_CASE(5, 16)
  PG_CASE(8, 1) PG_CASE(8, 2) PG_CASE(8, 4) PG_CASE(8, 8)
#undef PG_CASE
  set_error("fused sweep supports planes in {5,8} and words in {1,2,4,8}; got planes=%d words=%d", planes, words);
  return PG_ERR_UNSUPPORTED;
}

static int check_common(const void* own, long long own_rows, long long row0, long long rows, const void* str,
                        long long stream_rows, int planes, int words) {
  PG_CHECK_ARG(own && str, "null table pointer");
  PG_CHECK_ARG(rows > 0 && row0 >= 0 && row0 + rows <= own_rows, "own row range [%lld,%lld) outside table of %lld rows",
               row0, row0 + rows, own_rows);
  PG_CHECK_ARG(stream_rows > 0, "empty stream table");
  PG_CHECK_ARG(stream_rows < (1ll << 32), "stream table too large for 32-bit indices");
  PG_CHECK_ARG((reinterpret_cast<uintptr_t>(str) & 15) == 0, "stream table must be 16-byte aligned");
  PG_CHECK_ARG((reinterpret_cast<uintptr_t>(own) & 15) == 0, "own table must be 16-byte aligned");
  if (!(((planes == 5 || planes == 8) && (words == 1 || words == 2 || words == 4 || words == 8)) ||
        (planes == 5 && words == 16) || long_rows(planes, words) || wide_rows(planes, words))) {
    set_error("fused sweep supports planes in {5,8} x words in {1,2,4,8}, planes=5 with words 16,24,..,1024 and "
              "planes=8 with words 16,24,..,1024; got planes=%d words=%d", planes, words);
    return PG_ERR_UNSUPPORTED;
  }
  return PG_OK;
}

static void fill_common(SweepParams& prm, const Geometry& g, const uint32_t* own, long long row0, long long rows,
                        const uint32_t* str, long long stream_rows) {
  memset(&prm, 0, sizeof(prm));
  prm.own = own;
  prm.own_row0 = row0;
  prm.rows = rows;
  prm.row_map = nullptr;
  prm.rows_total = rows;
  prm.str = str;
  prm.str_rows = stream_rows;
  prm.n_rowblocks = g.n_rowblocks;
  prm.n_splits = g.n_splits;
  prm.tiles_per_split = g.tiles_per_split;
  prm.n_tiles = g.n_tiles;
  prm.one = 1u;
}

// A truth table over d = 0..L that is one contiguous run becomes a range test.
static bool lut_as_range(const uint32_t* lut, int lut_words, int* lo, unsigned* span) {
  int first = -1, last = -1, pop = 0;
  for (int d = 0; d < lut_words * 32; ++d) {
    if ((lut[d >> 5] >> (d & 31)) & 1u) {
      if (first < 0) first = d;
      last = d;
      ++pop;
    }
  }
  if (pop == 0) { *lo = 0x7fffffff; *span = 0; return true; }
  if (last - first + 1 != pop) return false;
  *lo = first;
  *span = static_cast<unsigned>(last - first);
  return true;
}

// ---- coalesced write-out of per-row results -------------------------------------------------
// The merge kernels below run one thread per row; a thread that stored its k results straight to
// out[r * k + j] would touch 32 different 128-byte lines per store instruction.  Instead every
// thread parks its row in shared memory (row stride k + 1 keys: conflict-free 8-byte accesses) and
// the block writes its rows * k outputs contiguously.
__device__ __forceinline__ void emit_key(unsigned long long best, long long at, int weight, bool keys_out,
                                         unsigned long long* out_keys, long long* out_idx, void* out_w) {
  if (keys_out) {
    out_keys[at] = best;
  } else if (best == ~0ull) {
    // missing entry: index -1, weight 0 in every weight kind (0.0, not the similarity of d = 0),
    // as the Minkowski GEMM writes it
    out_idx[at] = -1;
    if (weight == PG_W_SIM_F32) reinterpret_cast<float*>(out_w)[at] = 0.0f;
    else write_weight(out_w, at, 0, weight);
  } else {
    out_idx[at] = static_cast<long long>(best & 0xffffffffull);
    write_weight(out_w, at, static_cast<int>(best >> 32), weight);
  }
}

__device__ __forceinline__ void flush_rows(const unsigned long long* sm, long long row_base, long long rows, int kk,
                                           int weight, bool keys_out, unsigned long long* out_keys, long long* out_idx,
                                           void* out_w) {
  __syncthreads();
  const long long here = min(static_cast<long long>(blockDim.x), rows - row_base);
  const int total = static_cast<int>(here) * kk;
  for (int e = threadIdx.x; e < total; e += blockDim.x) {
    const int r = e / kk, j = e - r * kk;
    emit_key(sm[r * (kk + 1) + j], row_base * kk + e, weight, keys_out, out_keys, out_idx, out_w);
  }
}

static int rows_per_merge_block(int kk) { return kk <= 32 ? 128 : 32; }
static size_t merge_smem_bytes(int kk) { return static_cast<size_t>(rows_per_merge_block(kk)) * (kk + 1) * 8; }

// ---- kNN: merge the per-split lists, drop leading entries, widen ---------------------
__global__ void knn_finalize_kernel(const unsigned long long* __restrict__ part, int n_splits, int k1, long long rows,
                                    int k, int drop, int weight, long long* __restrict__ out_idx, void* out_w) {
  extern __shared__ unsigned long long merge_sm[];
  const long long row_base = blockIdx.x * static_cast<long long>(blockDim.x);
  const long long r = row_base + threadIdx.x;
  unsigned long long* mine = merge_sm + threadIdx.x * (k + 1);
  if (r < rows) {
    unsigned long long last = 0;
    bool have_last = false;
    for (int j = 0; j < drop + k; ++j) {
      unsigned long long best = ~0ull;
      if (n_splits == 1) {
        best = j < k1 ? part[static_cast<size_t>(j) * rows + r] : ~0ull;
      } else {
        // keys are unique (index in the low word), so "smallest key above the last one" walks
        // the merged order; each split list is ascending, stop at the first usable entry
        for (int s = 0; s < n_splits; ++s) {
          const unsigned long long* lst = part + static_cast<size_t>(s) * k1 * rows + r;
          for (int i = 0; i < k1; ++i) {
            const unsigned long long v = lst[static_cast<size_t>(i) * rows];
            if (have_last && v <= last) continue;
            if (v < best) best = v;
            break;
          }
        }
      }
      last = best;
      have_last = true;
      if (j >= drop) mine[j - drop] = best;
    }
  }
  flush_rows(merge_sm, row_base, rows, k, weight, false, nullptr, out_idx, out_w);
}

__global__ void sum_splits_kernel(const long long* __restrict__ split_counts, int n_splits, long long rows,
                                  long long* __restrict__ counts, uint8_t* __restrict__ over_flag, int capture_cap) {
  const long long r = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (r >= rows) return;
  long long s = 0;
  bool over = false;
  for (int i = 0; i < n_splits; ++i) {
    const long long c = split_counts[static_cast<size_t>(i) * rows + r];
    over |= c > capture_cap;
    s += c;
  }
  counts[r] = s;
  if (over_flag) over_flag[r] = over ? 1 : 0;   // some split of this row had more hits than the capture holds
}

// Fill from the captures of the count pass: row r's edges are the splits' captured hits in
// split order, i.e. ascending stream index.  One warp per row, lanes along the row's hits (coalesced
// on both sides: dense graphs keep thousands of hits per row).  Rows with an overflowed capture are
// left to the fill sweep over the overflow rows.
__global__ void __launch_bounds__(256) eps_from_capture_kernel(const unsigned long long* __restrict__ capture,
                                                               const long long* __restrict__ split_counts,
                                                               int n_splits, long long rows, int capture_cap,
                                                               const uint8_t* __restrict__ over_flag,
                                                               const long long* __restrict__ indptr, int weight,
                                                               long long* __restrict__ out_idx, void* out_w) {
  const int lane = threadIdx.x & 31;
  const long long warps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
  for (long long r = blockIdx.x * static_cast<long long>(blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += warps) {
    if (over_flag[r]) continue;
    long long at = indptr[r];
    for (int s = 0; s < n_splits; ++s) {
      const int c = static_cast<int>(split_counts[static_cast<size_t>(s) * rows + r]);
      const unsigned long long* src = capture + (static_cast<size_t>(s) * rows + r) * capture_cap;
      for (int j = lane; j < c; j += 32) {
        const unsigned long long e = __ldcs(src + j);
        out_idx[at + j] = static_cast<long long>(e & 0xffffffffull);
        write_weight(out_w, at + j, static_cast<int>(e >> 32), weight);
      }
      at += c;
    }
  }
}

// eps workspace: [split counts: n_splits*rows int64][header 256 B: number of overflow rows, capture slots in use]
//                [overflow flag per row, padded][overflow row list: rows int64][captures: n_splits*rows*cap u64]
// cap = kEpsCapture (128) by default: enough to finish sparse graphs without a second sweep.  A caller that
// knows the graph is dense (degree sample) sizes the workspace with pg_eps_workspace_bytes_capture for the
// largest degree it expects; the count pass keeps as many hits per (split,row) as the workspace holds.
static size_t eps_counts_bytes(const Geometry& g, long long rows) { return static_cast<size_t>(g.n_splits) * rows * 8; }
static size_t eps_capture_bytes(const Geometry& g, long long rows, int cap = kEpsCapture) {
  return static_cast<size_t>(g.n_splits) * rows * static_cast<size_t>(cap) * 8;
}
static size_t eps_flag_bytes(long long rows) { return static_cast<size_t>(round_up(rows, 256)); }
static size_t eps_list_bytes(long long rows) { return static_cast<size_t>(rows) * 8; }
constexpr int kEpsCaptureMax = 1 << 20;
constexpr size_t kEpsCaptureLimit = 8ull << 30;   // do not spend more than 8 GiB on captures

// Geometry and capture slots of an epsilon count / fill pair.  capture = 0: the default geometry with
// kEpsCapture slots per (split,row) when that fits the limit.  capture > 0 (the largest degree a
// caller expects of a dense graph): as many slots, and no more column splits than keep the captures
// within the limit -- every split of a row needs room for ALL of the row's hits, and the wave
// balance that splits buy (C3: 35 splits) is worth less than the second sweep the captures save
// (C3 eps=2, 358.7 M edges: count 15.5 + fill 16.2 ms -> count 16.2 + copy 2.1 ms).
struct EpsPlan {
  Geometry g;
  int cap;          // capture slots per (split,row), 0 = no captures
};
static EpsPlan eps_plan(long long rows, long long stream_rows, int words, int capture) {
  EpsPlan p;
  p.cap = 0;
  if (capture > 0 && rows < (1ll << 31)) {
    const int cap = std::min(std::max(capture, kEpsCapture), kEpsCaptureMax);
    const long long splits = static_cast<long long>(kEpsCaptureLimit / (static_cast<size_t>(rows) * cap * 8));
    if (splits >= 1) {
      p.g = make_geometry(rows, stream_rows, words, kConsumers, 0, splits);
      p.cap = cap;
      return p;
    }
  }
  p.g = make_geometry(rows, stream_rows, words, kConsumers, 0);
  if (eps_capture_bytes(p.g, rows) <= kEpsCaptureLimit && rows < (1ll << 31)) p.cap = kEpsCapture;
  return p;
}
static size_t eps_plan_bytes(const EpsPlan& p, long long rows) {
  size_t bytes = eps_counts_bytes(p.g, rows) + 256;
  if (p.cap > 0) bytes += eps_flag_bytes(rows) + eps_list_bytes(rows) + eps_capture_bytes(p.g, rows, p.cap);
  return bytes;
}


// ---- symmetric kNN sweep (pg_sweep_sym.cuh): host side ---------------------------------
static int dispatch_sym(int planes, int words, const SymParams& prm, const SymLaunch& l, int* resident) {
#define PG_CASE(P, W) \
  if (planes == P && words == W) return sweep_sym_p##P##_w##W(prm, l, resident);
  PG_CASE(5, 1) PG_CASE(5, 2) PG_CASE(5, 4) PG_CASE(5, 8) PG_CASE(5, 16)
  PG_CASE(8, 1) PG_CASE(8, 2) PG_CASE(8, 4) PG_CASE(8, 8)
#undef PG_CASE
  set_error("symmetric sweep supports planes in {5,8} x words in {1,2,4,8} and planes=5, words=16; got planes=%d "
            "words=%d", planes, words);
  return PG_ERR_UNSUPPORTED;
}

static bool sym_shape_ok(int planes, int words) {
  return ((planes == 5 || planes == 8) && (words == 1 || words == 2 || words == 4 || words == 8)) ||
         (planes == 5 && words == 16);
}

// workspace: [filter words: tiles*tile_cols u64][locks: rows u32][stats: 8 u64, error word at +64 B][items]
struct SymLayout {
  int tile_cols, n_tiles, n_blocks, band_tiles, n_bands;
  size_t gnt_bytes, lock_bytes, stats_off, item_off, item_bytes_max, total;
};

// Stream tiles per L2-sized column band: co-resident CTAs work inside one band of the table so that
// its tiles are read from DRAM once and from L2 afterwards (PG_SYM_BAND_MB, default 24 MB of the
// 126 MB L2; the packed row is at least 5 planes wide, which bounds the band count from above).
static int sym_band_tiles(int tile_cols, int row_bytes) {
  double mb = 24.0;
  if (const char* ev = std::getenv("PG_SYM_BAND_MB")) mb = std::atof(ev);
  if (mb <= 0) return 1 << 30;                       // 0: one band (the round-1 schedule)
  long long t = static_cast<long long>(mb * 1048576.0 / (static_cast<double>(tile_cols) * row_bytes));
  if (t < 64) t = 64;
  return static_cast<int>(std::min<long long>(t, 1 << 30));
}

static SymLayout sym_layout(long long rows, int words, int planes = 5) {
  SymLayout s;
  s.tile_cols = tile_cols_for(words);
  s.n_tiles = static_cast<int>(ceil_div(rows, s.tile_cols));
  s.n_blocks = static_cast<int>(ceil_div(rows, kConsumers));
  s.band_tiles = sym_band_tiles(s.tile_cols, planes * words * 4);
  s.n_bands = static_cast<int>(ceil_div(s.n_tiles, s.band_tiles));
  s.gnt_bytes = static_cast<size_t>(round_up(static_cast<int64_t>(s.n_tiles) * s.tile_cols * 8, 256));
  s.lock_bytes = static_cast<size_t>(round_up(rows * 4, 256));
  s.stats_off = s.gnt_bytes + s.lock_bytes;
  s.item_off = s.stats_off + 256;
  // a row block contributes at most len / chunk + 2 items per band it crosses and the planner keeps
  // sum(len) / chunk below 64 items per resident CTA (<= 4 CTAs per SM); sized for 8 planes (most bands)
  const int bands8 = static_cast<int>(ceil_div(s.n_tiles, sym_band_tiles(s.tile_cols, 8 * words * 4)));
  s.item_bytes_max = (static_cast<size_t>(s.n_blocks) * (2 * static_cast<size_t>(bands8) + 2) + 64ull * 4 * 160 + 1024) *
                         sizeof(SymItem) + 8192;       // + the per-CTA offsets
  s.total = s.item_off + s.item_bytes_max;
  return s;
}

static int sym_first_tile(const SymLayout& s, int rb, long long boot_rows) {
  const long long row = static_cast<long long>(rb) * kConsumers < boot_rows ? boot_rows
                                                                            : static_cast<long long>(rb) * kConsumers;
  return static_cast<int>(row / s.tile_cols);
}

// Column band of partition `part` of `parts`: tile range [t0, t1) such that every band holds the
// same number of (own row, stream tile) visits of the triangle.
static void sym_band(const SymLayout& s, long long rows, long long boot_rows, int part, int parts, int* t0, int* t1) {
  std::vector<long long> visits(static_cast<size_t>(s.n_tiles) + 1, 0);
  for (int rb = 0; rb < s.n_blocks; ++rb) {
    const int tb = sym_first_tile(s, rb, boot_rows);
    if (tb >= s.n_tiles) continue;
    const long long in_block = std::min<long long>(kConsumers, rows - static_cast<long long>(rb) * kConsumers);
    visits[tb] += in_block;          // rows that sweep every tile from tb on
  }
  long long total = 0, run = 0;
  for (int t = 0; t < s.n_tiles; ++t) { run += visits[t]; visits[t] = run; total += run; }
  auto bound = [&](int g) {
    if (g <= 0) return 0;
    if (g >= parts) return s.n_tiles;
    const long long want = static_cast<long long>(static_cast<double>(total) * g / parts);
    long long acc = 0;
    for (int t = 0; t < s.n_tiles; ++t) {
      acc += visits[t];
      if (acc >= want) return t + 1;
    }
    return s.n_tiles;
  };
  *t0 = bound(part);
  *t1 = bound(part + 1);
}

// Chunks of (row block, tile range) for the persistent grid.  The column range of the sweep is cut
// into L2-sized bands (SymLayout::band_tiles) and the chunks are handed out band by band: at any
// time the resident CTAs stream tiles of ONE band, which then comes out of L2 instead of DRAM
// (round 1 walked the whole 160 MB table from 296 different positions: 115 GB of DRAM reads per
// build).  Every CTA gets its own item list (SymPlan::first): inside a band the chunks go, longest
// first, to the CTA with the least work so far, so the CTAs reach the end of every band -- and of
// the sweep -- together to within one short chunk.  Chunk boundaries are phase-shifted from row block
// to row block so that CTAs that start together do not walk the same stream rows in lockstep (they
// would fight for the same row locks).
// mode 0: this rank takes row blocks part, part+parts, ... over their whole tile range;
// mode 1: every row block, restricted to this rank's column band (sym_band).
struct SymPlan {
  std::vector<SymItem> items;   // CTA-major: CTA b owns items [first[b], first[b+1])
  std::vector<int> first;       // grid + 1 offsets
  int grid = 0;                 // CTAs that have work
};

static SymPlan sym_plan(const SymLayout& s, long long rows, int part, int parts, int mode, int grid,
                        long long boot_rows, int chunk_floor = 32) {
  const int boot_blocks = static_cast<int>(boot_rows / kConsumers);
  int band0 = 0, band1 = s.n_tiles;
  if (mode == 1) sym_band(s, rows, boot_rows, part, parts, &band0, &band1);
  const int rb_first = mode == 1 ? 0 : part, rb_stride = mode == 1 ? 1 : parts;
  long long total = 0;
  for (int rb = rb_first; rb < s.n_blocks; rb += rb_stride)
    total += std::max(0, band1 - std::max(sym_first_tile(s, rb, boot_rows), band0));
  long long chunk = ceil_div(total, static_cast<long long>(grid) * 24);
  if (const char* ev = std::getenv("PG_SYM_CHUNK")) chunk = std::atoll(ev);
  // L2 bands of equal width over this rank's column range
  const int span = std::max(0, band1 - band0);
  const int n_sub = std::max(1, static_cast<int>(ceil_div(span, s.band_tiles)));
  const int sub_w = std::max(1, static_cast<int>(ceil_div(span, n_sub)));
  if (n_sub > 1 && chunk > sub_w / 2) chunk = sub_w / 2;     // at least two phase-shifted chunks per band crossing
  if (chunk < chunk_floor) chunk = chunk_floor;
  std::vector<std::vector<SymItem>> per_cta(static_cast<size_t>(grid));
  std::vector<long long> load(static_cast<size_t>(grid), 0);
  // min-heap of (load, cta)
  auto heavier = [&](int a, int b) { return load[a] != load[b] ? load[a] > load[b] : a > b; };
  std::vector<int> heap(static_cast<size_t>(grid));
  for (int sb = 0; sb < n_sub; ++sb) {
    const int sb0 = band0 + sb * sub_w, sb1 = std::min(band1, sb0 + sub_w);
    std::vector<SymItem> items;
    unsigned n_seen = 0;
    for (int rb = rb_first; rb < s.n_blocks; rb += rb_stride, ++n_seen) {
      const int tb = std::max(sym_first_tile(s, rb, boot_rows), sb0), te = sb1;
      if (te <= tb) continue;
      const int boot = rb < boot_blocks ? 1 : 0;
      // golden-ratio phase of the first boundary, in (chunk/4, 5*chunk/4]
      const double g = (n_seen + 0.37 * sb) * 0.6180339887498949;
      const double frac = g - static_cast<long long>(g);
      int t = tb;
      const int first = static_cast<int>(chunk / 4 + static_cast<long long>(frac * static_cast<double>(chunk))) + 1;
      while (t < te) {
        int t1 = t + (t == tb ? first : static_cast<int>(chunk));
        if (te - t1 < chunk / 4) t1 = te;     // no crumbs at the end
        if (t1 > te) t1 = te;
        items.push_back(SymItem{rb, t, t1, boot});
        t = t1;
      }
    }
    std::stable_sort(items.begin(), items.end(),
                     [](const SymItem& a, const SymItem& b) { return a.t1 - a.t0 > b.t1 - b.t0; });
    for (int b = 0; b < grid; ++b) heap[b] = b;
    std::make_heap(heap.begin(), heap.end(), heavier);
    for (const SymItem& it : items) {
      std::pop_heap(heap.begin(), heap.end(), heavier);
      const int b = heap.back();
      per_cta[b].push_back(it);
      load[b] += (it.t1 - it.t0) + 4;          // + a fixed per-item cost (own-row load, list merge)
      std::push_heap(heap.begin(), heap.end(), heavier);
    }
  }
  SymPlan plan;
  plan.first.push_back(0);
  for (int b = 0; b < grid; ++b) {
    if (per_cta[b].empty()) continue;
    plan.items.insert(plan.items.end(), per_cta[b].begin(), per_cta[b].end());
    plan.first.push_back(static_cast<int>(plan.items.size()));
  }
  plan.grid = static_cast<int>(plan.first.size()) - 1;
  return plan;
}

// item table in the workspace: [first: grid + 1 ints, padded to 16 B][items]
// smallest kNN chunk (tiles) of the symmetric sweep: see pg_hamming_knn_sym
static int sym_knn_chunk_floor(int words, int parts) { return (parts == 1 ? 256 : 32) * std::max(1, 8 / words); }

static size_t sym_plan_bytes(const SymPlan& p) {
  return static_cast<size_t>(round_up(static_cast<int64_t>(p.first.size()) * 4, 16)) + p.items.size() * sizeof(SymItem);
}
static int sym_upload_plan(const SymPlan& p, const SymLayout& lay, char* wsb, SymParams* prm, cudaStream_t cs) {
  PG_CHECK_ARG(sym_plan_bytes(p) <= lay.item_bytes_max, "item table overflow (%zu items)", p.items.size());
  const size_t first_bytes = static_cast<size_t>(round_up(static_cast<int64_t>(p.first.size()) * 4, 16));
  PG_CUDA(cudaMemcpyAsync(wsb + lay.item_off, p.first.data(), p.first.size() * 4, cudaMemcpyHostToDevice, cs));
  PG_CUDA(cudaMemcpyAsync(wsb + lay.item_off + first_bytes, p.items.data(), p.items.size() * sizeof(SymItem),
                          cudaMemcpyHostToDevice, cs));
  // the vectors die with the caller: pageable copies are staged by the runtime before returning
  prm->cta_first = reinterpret_cast<const int*>(wsb + lay.item_off);
  prm->items = reinterpret_cast<const SymItem*>(wsb + lay.item_off + first_bytes);
  prm->n_items = static_cast<int>(p.items.size());
  return PG_OK;
}

__global__ void sym_init_kernel(unsigned long long* glist, long long n_keys, unsigned long long* glast, long long n_gnt, unsigned* glock,
                                long long rows, unsigned long long* stats, int k1, int seeded) {
  if (blockIdx.x == 0 && threadIdx.x < 9) stats[threadIdx.x] = 0ull;      // 8 counters + the error word
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  if (!seeded)
    for (long long j = i; j < n_keys; j += stride) glist[j] = ~0ull;
  for (long long j = i; j < n_gnt; j += stride) {
    unsigned long long last = ~0ull;
    if (seeded && j < rows) last = glist[j * k1 + (k1 - 1)];
    glast[j] = sym_filter_word(last);
  }
  for (long long j = i; j < rows; j += stride) glock[j] = 0u;
}

// bootstrap: merged split lists [n_splits][k1][rows] -> row-major key lists [rows][k1]
__global__ void knn_part_to_lists_kernel(const unsigned long long* __restrict__ part, int n_splits, int k1,
                                         long long rows, unsigned long long* __restrict__ lists) {
  extern __shared__ unsigned long long merge_sm[];
  const long long row_base = blockIdx.x * static_cast<long long>(blockDim.x);
  const long long r = row_base + threadIdx.x;
  unsigned long long* mine = merge_sm + threadIdx.x * (k1 + 1);
  if (r < rows) {
    unsigned long long last = 0;
    bool ended = false;
    for (int j = 0; j < k1; ++j) {
      unsigned long long best = ~0ull;
      if (!ended) {
        for (int s = 0; s < n_splits; ++s) {
          const unsigned long long* lst = part + static_cast<size_t>(s) * k1 * rows + r;
          for (int i = 0; i < k1; ++i) {
            const unsigned long long v = lst[static_cast<size_t>(i) * rows];
            if (j > 0 && v <= last) continue;
            if (v < best) best = v;
            break;
          }
        }
      }
      last = best;
      ended |= best == ~0ull;
      mine[j] = best;
    }
  }
  flush_rows(merge_sm, row_base, rows, k1, PG_W_I64, true, lists, nullptr, nullptr);
}

// Final lists: merge n_lists sorted key lists per row (one per rank), drop, then either widen to the
// reference's (index int64, weight) arrays or keep the merged keys (KEYS_OUT: the exchange step of the
// multi-GPU build all-gathers 8-byte keys and widens locally).  Every list keeps a cursor and its
// head key in registers; a key present in several lists (the shared bootstrap entries) advances all
// of them, so the merged order has no duplicates.
constexpr int kMaxMergeLists = 16;

__global__ void knn_lists_finalize_kernel(const unsigned long long* __restrict__ lists, int n_lists,
                                          long long list_stride, long long row0, long long rows, int k1, int k,
                                          int drop, int weight, bool keys_out, unsigned long long* __restrict__ out_keys,
                                          long long* __restrict__ out_idx, void* out_w) {
  extern __shared__ unsigned long long merge_sm[];
  const long long row_base = blockIdx.x * static_cast<long long>(blockDim.x);
  const long long r = row_base + threadIdx.x;
  unsigned long long* mine = merge_sm + threadIdx.x * (k + 1);
  if (r < rows) {
    const unsigned long long* base = lists + static_cast<size_t>(row0 + r) * k1;
    unsigned long long head[kMaxMergeLists];
    int pos[kMaxMergeLists];
#pragma unroll
    for (int s = 0; s < kMaxMergeLists; ++s) {
      pos[s] = 0;
      head[s] = s < n_lists ? base[static_cast<size_t>(s) * list_stride] : ~0ull;
    }
    for (int j = 0; j < drop + k; ++j) {
      unsigned long long best = ~0ull;
#pragma unroll
      for (int s = 0; s < kMaxMergeLists; ++s) best = head[s] < best ? head[s] : best;
      if (best != ~0ull) {
#pragma unroll
        for (int s = 0; s < kMaxMergeLists; ++s) {
          if (head[s] == best) {
            ++pos[s];
            head[s] = pos[s] < k1 ? base[static_cast<size_t>(s) * list_stride + pos[s]] : ~0ull;
          }
        }
      }
      if (j >= drop) mine[j - drop] = best;
    }
  }
  flush_rows(merge_sm, row_base, rows, k, weight, keys_out, out_keys, out_idx, out_w);
}

// more lists than cursors fit in registers: "smallest key above the last one", rescanning the lists
__global__ void knn_lists_finalize_scan_kernel(const unsigned long long* __restrict__ lists, int n_lists,
                                               long long list_stride, long long row0, long long rows, int k1, int k,
                                               int drop, int weight, bool keys_out,
                                               unsigned long long* __restrict__ out_keys, long long* __restrict__ out_idx,
                                               void* out_w) {
  extern __shared__ unsigned long long merge_sm[];
  const long long row_base = blockIdx.x * static_cast<long long>(blockDim.x);
  const long long r = row_base + threadIdx.x;
  unsigned long long* mine = merge_sm + threadIdx.x * (k + 1);
  if (r < rows) {
    unsigned long long last = 0;
    bool have_last = false;
    for (int j = 0; j < drop + k; ++j) {
      unsigned long long best = ~0ull;
      for (int s = 0; s < n_lists; ++s) {
        const unsigned long long* lst = lists + static_cast<size_t>(s) * list_stride + static_cast<size_t>(row0 + r) * k1;
        for (int i = 0; i < k1; ++i) {
          const unsigned long long v = lst[i];
          if (have_last && v <= last) continue;
          if (v < best) best = v;
          break;
        }
      }
      last = best;
      have_last = true;
      if (j >= drop) mine[j - drop] = best;
    }
  }
  flush_rows(merge_sm, row_base, rows, k, weight, keys_out, out_keys, out_idx, out_w);
}

// One sorted list per row -> (index, weight): HBM-bound, one thread per OUTPUT element so that the
// 8-byte loads and both stores are coalesced (the per-row version strode 136 B between lanes).
__global__ void knn_keys_widen_kernel(const unsigned long long* __restrict__ keys, long long row0, long long rows,
                                      int k1, int k, int drop, int weight, long long* __restrict__ out_idx,
                                      void* out_w) {
  const long long total = rows * k;
  const int kshift = pow2_shift(k);
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < total;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    long long r;
    int j;
    split_index(e, k, kshift, &r, &j);
    j += drop;
    const unsigned long long key = j < k1 ? __ldcs(keys + (row0 + r) * k1 + j) : ~0ull;
    emit_key(key, e, weight, false, nullptr, out_idx, out_w);
  }
}

// ---- symmetric epsilon graph: edge keys -> CSR -----------------------------------------------
struct EdgeKeyBits { int dbits, idxbits; };
static EdgeKeyBits edge_key_bits(long long rows, int words) {
  EdgeKeyBits b;
  b.dbits = 1;
  while ((1 << b.dbits) <= words * 32) ++b.dbits;          // distances 0 .. 32*words
  b.idxbits = 1;
  while ((1ll << b.idxbits) <= rows) ++b.idxbits;          // rows < 2^idxbits - 1: the all-ones row is the sentinel
  return b;
}

__global__ void edge_decode_kernel(const unsigned long long* __restrict__ keys, long long nnz, long long rows, int dbits,
                                   int idxbits, int weight, long long* __restrict__ indptr,
                                   long long* __restrict__ out_idx, void* out_w) {
  const long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (nnz == 0) {
    for (long long x = e; x <= rows; x += static_cast<long long>(gridDim.x) * blockDim.x) indptr[x] = 0;
    return;
  }
  if (e >= nnz) return;
  const unsigned long long key = keys[e];
  const unsigned long long imask = (1ull << idxbits) - 1ull;
  const long long row = static_cast<long long>(key >> (dbits + idxbits));
  const long long col = static_cast<long long>((key >> dbits) & imask);
  const int d = static_cast<int>(key & ((1ull << dbits) - 1ull));
  out_idx[e] = col;
  write_weight(out_w, e, d, weight);
  // row boundaries: indptr[x] = e for every row x in (row of edge e-1, row of edge e]
  const long long prev = e > 0 ? static_cast<long long>(keys[e - 1] >> (dbits + idxbits)) : -1;
  for (long long x = prev + 1; x <= row; ++x) indptr[x] = e;
  if (e == nnz - 1)
    for (long long x = row + 1; x <= rows; ++x) indptr[x] = nnz;
}

}  // namespace pg

using namespace pg;

extern "C" {

size_t pg_sweep_workspace_bytes(int64_t own_rows, int64_t stream_rows, int words, int k1) {
  if (own_rows <= 0 || stream_rows <= 0 || words <= 0) return 0;
  // the largest split count any sweep of this shape may choose (kNN with k1 entries, the
  // count / fill passes, the two-rows-per-thread kNN variants)
  int n_splits = 1;
  for (int rpc = kConsumers; rpc <= 2 * kConsumers; rpc += kConsumers) {
    const int a = make_geometry(own_rows, stream_rows, words, rpc, 0).n_splits;
    const int b = make_geometry(own_rows, stream_rows, words, rpc, k1 > 0 ? k1 : 1).n_splits;
    n_splits = a > n_splits ? a : n_splits;
    n_splits = b > n_splits ? b : n_splits;
  }
  const size_t per_row = static_cast<size_t>(n_splits) * 8 * static_cast<size_t>(k1 > 1 ? k1 : 1);
  return per_row * static_cast<size_t>(own_rows) + 256;
}

size_t pg_eps_workspace_bytes(int64_t own_rows, int64_t stream_rows, int words) {
  if (own_rows <= 0 || stream_rows <= 0 || words <= 0) return 0;
  return eps_plan_bytes(eps_plan(own_rows, stream_rows, words, 0), own_rows);
}

size_t pg_eps_workspace_bytes_capture(int64_t own_rows, int64_t stream_rows, int words, int capture) {
  if (own_rows <= 0 || stream_rows <= 0 || words <= 0) return 0;
  return eps_plan_bytes(eps_plan(own_rows, stream_rows, words, capture), own_rows);
}

size_t pg_eps_count_workspace_bytes(int64_t own_rows, int64_t stream_rows, int words) {
  if (own_rows <= 0 || stream_rows <= 0 || words <= 0) return 0;
  // counts only: a count pass with this workspace keeps no captures (degree census of a dense graph)
  return eps_counts_bytes(make_geometry(own_rows, stream_rows, words, kConsumers, 0), own_rows) + 256;
}

int pg_hamming_knn(const uint32_t* own, int64_t own_rows, int64_t row0, int64_t rows, const uint32_t* stream_tab,
                   int64_t stream_rows, int planes, int words, int k, int drop, int weight, int64_t* out_idx,
                   void* out_w, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_common(own, own_rows, row0, rows, stream_tab, stream_rows, planes, words);
  if (rc != PG_OK) return rc;
  PG_CHECK_ARG(k >= 1 && drop >= 0, "k must be >= 1 and drop >= 0");
  PG_CHECK_ARG(out_idx && out_w && workspace, "null output/workspace pointer");
  PG_CHECK_ARG(weight == PG_W_I64 || weight == PG_W_SIM_F32 || weight == PG_W_I32, "bad weight kind %d", weight);
  const int k1 = drop + k;
  // experiment knob: PG_KNN_VARIANT=1 runs two own rows per thread (planes 5, words 8 only)
  int tm = 1;
  int variant = 0;
  if (const char* ev = std::getenv("PG_KNN_VARIANT")) variant = std::atoi(ev);
  if (!(planes == 5 && words == 8)) variant = 0;
  if (variant == 1 || variant == 4) tm = 2;
  const Geometry g = make_geometry(rows, stream_rows, words, kConsumers * tm, k1);
  const size_t need = static_cast<size_t>(g.n_splits) * k1 * rows * 8;
  PG_CHECK_ARG(workspace_bytes >= need, "workspace too small: %zu < %zu", workspace_bytes, need);
  const size_t list_bytes = static_cast<size_t>(k1) * kConsumers * tm * 8;
  if (k1 > 32 * kMaxListRounds || list_bytes + 70 * 1024 > 227 * 1024) {
    set_error("k=%d too large for the in-shared-memory lists of the fused sweep", k);
    return PG_ERR_UNSUPPORTED;
  }
  SweepParams prm;
  fill_common(prm, g, own, row0, rows, stream_tab, stream_rows);
  prm.part = static_cast<unsigned long long*>(workspace);
  prm.k1 = k1;
  SweepLaunch l{MODE_KNN, 0, weight, 0, list_bytes, static_cast<cudaStream_t>(stream)};
  l.rows_per_thread = variant == 3 ? 3 : (variant == 4 ? 4 : tm);
  {
    SweepTimer t(l.stream);
    rc = dispatch(planes, words, prm, l);
  }
  if (rc != PG_OK) return rc;
  const int threads = rows_per_merge_block(k);
  knn_finalize_kernel<<<static_cast<unsigned>(ceil_div(rows, threads)), threads, merge_smem_bytes(k), l.stream>>>(
      prm.part, g.n_splits, k1, rows, k, drop, weight, reinterpret_cast<long long*>(out_idx), out_w);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

static int eps_pass(int mode, const uint32_t* own, int64_t own_rows, int64_t row0, int64_t rows,
                    const uint32_t* stream_tab, int64_t stream_rows, int planes, int words, const uint32_t* lut_host,
                    int lut_words, int64_t* counts, const int64_t* indptr, int weight, int64_t* out_idx, void* out_w,
                    void* workspace, size_t workspace_bytes, void* stream, int capture = 0) {
  int rc = check_common(own, own_rows, row0, rows, stream_tab, stream_rows, planes, words);
  if (rc != PG_OK) return rc;
  // the chunked sweep reads its truth table from shared memory: any table over d = 0..32*words
  const int max_lut = wide_rows(planes, words) ? std::max(kMaxLutWords, words + 1) : kMaxLutWords;
  PG_CHECK_ARG(lut_host && lut_words >= 1 && lut_words <= max_lut, "lut_words must be in [1,%d]", max_lut);
  PG_CHECK_ARG(lut_words * 32 > words * 32, "lut must cover distances 0..%d", words * 32);
  PG_CHECK_ARG(workspace, "null workspace");
  PG_CHECK_ARG(capture >= 0, "capture must be >= 0");
  const EpsPlan plan = eps_plan(rows, stream_rows, words, capture);
  const Geometry g = plan.g;
  const size_t need = eps_counts_bytes(g, rows);
  PG_CHECK_ARG(workspace_bytes >= need, "workspace too small: %zu < %zu", workspace_bytes, need);
  const size_t aux = 256 + eps_flag_bytes(rows) + eps_list_bytes(rows);
  // a counts-only workspace (pg_eps_count_workspace_bytes) keeps no captures
  const bool fits = workspace_bytes >= eps_plan_bytes(plan, rows);
  PG_CHECK_ARG(capture == 0 || fits, "workspace too small for capture=%d: size it with pg_eps_workspace_bytes_capture",
               capture);
  const bool capturing = plan.cap > 0 && fits;
  const int capture_cap = capturing ? plan.cap : 0;
  char* wsb = static_cast<char*>(workspace);
  long long* n_over_dev = reinterpret_cast<long long*>(wsb + need);
  uint8_t* over_flag = reinterpret_cast<uint8_t*>(wsb + need + 256);
  long long* over_rows = reinterpret_cast<long long*>(wsb + need + 256 + eps_flag_bytes(rows));
  unsigned long long* capture_buf = reinterpret_cast<unsigned long long*>(wsb + need + aux);
  cudaStream_t cs = static_cast<cudaStream_t>(stream);
  SweepParams prm;
  fill_common(prm, g, own, row0, rows, stream_tab, stream_rows);
  prm.split_counts = static_cast<long long*>(workspace);
  prm.capture_cap = capture_cap;
  if (mode == MODE_COUNT && capturing) prm.capture = capture_buf;
  long long n_over = -1;     // fill: -1 = sweep every row, otherwise the number of overflow rows
  if (mode == MODE_FILL && capturing) {
    PG_CUDA(cudaMemcpyAsync(&n_over, n_over_dev, sizeof(long long), cudaMemcpyDeviceToHost, cs));
    PG_CUDA(cudaStreamSynchronize(cs));
    const long long blocks = std::min<long long>(ceil_div(rows, 8), static_cast<long long>(num_sms()) * 32);
    eps_from_capture_kernel<<<static_cast<unsigned>(blocks), 256, 0, cs>>>(
        capture_buf, prm.split_counts, g.n_splits, rows, capture_cap, over_flag, reinterpret_cast<const long long*>(indptr),
        weight, reinterpret_cast<long long*>(out_idx), out_w);
    PG_LAUNCH_CHECK();
    if (n_over == 0) return PG_OK;
    // second sweep over the overflow rows only, with the count pass's split structure
    prm.row_map = over_rows;
    prm.rows = n_over;
    prm.n_rowblocks = static_cast<int>(ceil_div(n_over, kConsumers));
  }
  for (int i = 0; i < lut_words && i < kMaxLutWords; ++i) prm.lut[i] = lut_host[i];
  const bool ranged = lut_as_range(lut_host, lut_words, &prm.lo, &prm.span);
  SweepLaunch l{mode, ranged ? 0 : 1, weight, 0, 0, static_cast<cudaStream_t>(stream)};
  l.lut_words = lut_words;
  if (mode == MODE_FILL) {
    prm.indptr = reinterpret_cast<const long long*>(indptr);
    prm.out_idx = reinterpret_cast<long long*>(out_idx);
    prm.out_w = out_w;
  }
  void* lut_dev = nullptr;     // a table longer than the parameter block holds: device copy, freed in stream order
  if (!ranged && lut_words > kMaxLutWords) {
    PG_CUDA(temp_alloc(&lut_dev, sizeof(uint32_t) * lut_words, cs));
    const cudaError_t e = cudaMemcpyAsync(lut_dev, lut_host, sizeof(uint32_t) * lut_words, cudaMemcpyHostToDevice, cs);
    if (e != cudaSuccess) {
      cudaFreeAsync(lut_dev, cs);
      set_error("truth table upload failed: %s", cudaGetErrorString(e));
      return PG_ERR_CUDA;
    }
    l.lut_ext = static_cast<const uint32_t*>(lut_dev);
  }
  {
    SweepTimer t(l.stream);
    rc = dispatch(planes, words, prm, l);
  }
  if (lut_dev != nullptr) cudaFreeAsync(lut_dev, cs);
  if (rc != PG_OK) return rc;
  if (mode == MODE_COUNT) {
    const int threads = 256;
    sum_splits_kernel<<<static_cast<unsigned>(ceil_div(rows, threads)), threads, 0, l.stream>>>(
        prm.split_counts, g.n_splits, rows, reinterpret_cast<long long*>(counts), capturing ? over_flag : nullptr,
        capture_cap);
    PG_LAUNCH_CHECK();
    if (capturing) {
      // list of the rows whose capture overflowed (they get a fill sweep of their own)
      thrust::counting_iterator<long long> ids(0);
      size_t tmp_bytes = 0;
      PG_CUDA(cub::DeviceSelect::Flagged(nullptr, tmp_bytes, ids, over_flag, over_rows, n_over_dev,
                                         static_cast<int>(rows), l.stream));
      void* tmp = nullptr;
      PG_CUDA(temp_alloc(&tmp, tmp_bytes, l.stream));
      cudaError_t e = cub::DeviceSelect::Flagged(tmp, tmp_bytes, ids, over_flag, over_rows, n_over_dev,
                                                 static_cast<int>(rows), l.stream);
      count_launch();
      cudaFreeAsync(tmp, l.stream);
      if (e != cudaSuccess) { set_error("cub select failed: %s", cudaGetErrorString(e)); return PG_ERR_CUDA; }
    }
  }
  return PG_OK;
}

int pg_hamming_eps_count(const uint32_t* own, int64_t own_rows, int64_t row0, int64_t rows,
                         const uint32_t* stream_tab, int64_t stream_rows, int planes, int words,
                         const uint32_t* lut_host, int lut_words, int64_t* counts, void* workspace,
                         size_t workspace_bytes, void* stream) {
  PG_CHECK_ARG(counts, "null counts");
  return eps_pass(MODE_COUNT, own, own_rows, row0, rows, stream_tab, stream_rows, planes, words, lut_host, lut_words,
                  counts, nullptr, PG_W_I64, nullptr, nullptr, workspace, workspace_bytes, stream);
}

int pg_hamming_eps_count_capture(const uint32_t* own, int64_t own_rows, int64_t row0, int64_t rows,
                                 const uint32_t* stream_tab, int64_t stream_rows, int planes, int words,
                                 const uint32_t* lut_host, int lut_words, int capture, int64_t* counts, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  PG_CHECK_ARG(counts, "null counts");
  return eps_pass(MODE_COUNT, own, own_rows, row0, rows, stream_tab, stream_rows, planes, words, lut_host, lut_words,
                  counts, nullptr, PG_W_I64, nullptr, nullptr, workspace, workspace_bytes, stream, capture);
}

int pg_hamming_eps_fill_capture(const uint32_t* own, int64_t own_rows, int64_t row0, int64_t rows,
                                const uint32_t* stream_tab, int64_t stream_rows, int planes, int words,
                                const uint32_t* lut_host, int lut_words, int capture, const int64_t* indptr, int weight,
                                int64_t* out_idx, void* out_w, void* workspace, size_t workspace_bytes, void* stream) {
  PG_CHECK_ARG(indptr && out_idx && out_w, "null indptr/output");
  PG_CHECK_ARG(weight == PG_W_I64 || weight == PG_W_SIM_F32, "fill writes int64 distances or float32 similarities");
  return eps_pass(MODE_FILL, own, own_rows, row0, rows, stream_tab, stream_rows, planes, words, lut_host, lut_words,
                  nullptr, indptr, weight, out_idx, out_w, workspace, workspace_bytes, stream, capture);
}

int pg_hamming_eps_fill(const uint32_t* own, int64_t own_rows, int64_t row0, int64_t rows,
                        const uint32_t* stream_tab, int64_t stream_rows, int planes, int words,
                        const uint32_t* lut_host, int lut_words, const int64_t* indptr, int weight, int64_t* out_idx,
                        void* out_w, void* workspace, size_t workspace_bytes, void* stream) {
  PG_CHECK_ARG(indptr && out_idx && out_w, "null indptr/output");
  PG_CHECK_ARG(weight == PG_W_I64 || weight == PG_W_SIM_F32, "fill writes int64 distances or float32 similarities");
  return eps_pass(MODE_FILL, own, own_rows, row0, rows, stream_tab, stream_rows, planes, words, lut_host, lut_words,
                  nullptr, indptr, weight, out_idx, out_w, workspace, workspace_bytes, stream);
}

int pg_hamming_tile(const uint32_t* data, int64_t data_rows, const uint32_t* queries, int64_t query_rows, int64_t q0,
                    int64_t qrows, int planes, int words, int weight, void* out, int64_t ld, void* stream) {
  // own = dataset rows (coalesced stores along n), stream = the query rows
  PG_CHECK_ARG(q0 >= 0 && qrows > 0 && q0 + qrows <= query_rows, "query range outside table");
  PG_CHECK_ARG(q0 % kStreamRowPad == 0, "q0 must be a multiple of %d", kStreamRowPad);
  int rc = check_common(data, data_rows, 0, data_rows, queries, qrows, planes, words);
  if (rc != PG_OK) return rc;
  PG_CHECK_ARG(out && ld >= data_rows, "bad output / leading dimension");
  PG_CHECK_ARG(weight == PG_W_I64 || weight == PG_W_SIM_F32 || weight == PG_W_I32, "bad weight kind %d", weight);
  Geometry g = make_geometry(data_rows, qrows, words, kConsumers, 0);
  g.n_splits = 1;  // every (own, stream) pair is written exactly once; splits only add launches
  g.tiles_per_split = g.n_tiles;
  SweepParams prm;
  fill_common(prm, g, data, 0, data_rows, queries + static_cast<size_t>(q0) * planes * words, qrows);
  prm.out = out;
  prm.ld = ld;
  SweepLaunch l{MODE_TILE, 0, weight, 0, 0, static_cast<cudaStream_t>(stream)};
  SweepTimer t(l.stream);
  return dispatch(planes, words, prm, l);
}

int pg_hamming_flags_tile(const uint32_t* data, int64_t data_rows, const uint32_t* queries, int64_t query_rows, int64_t q0,
                          int64_t qrows, int planes, int words, int d_lo, int d_hi, uint8_t* out, int64_t ld,
                          void* stream) {
  PG_CHECK_ARG(q0 >= 0 && qrows > 0 && q0 + qrows <= query_rows, "query range outside table");
  PG_CHECK_ARG(q0 % kStreamRowPad == 0, "q0 must be a multiple of %d", kStreamRowPad);
  int rc = check_common(data, data_rows, 0, data_rows, queries, qrows, planes, words);
  if (rc != PG_OK) return rc;
  PG_CHECK_ARG(out && ld >= data_rows, "bad output / leading dimension");
  Geometry g = make_geometry(data_rows, qrows, words, kConsumers, 0);
  g.n_splits = 1;
  g.tiles_per_split = g.n_tiles;
  SweepParams prm;
  fill_common(prm, g, data, 0, data_rows, queries + static_cast<size_t>(q0) * planes * words, qrows);
  prm.out = out;
  prm.ld = ld;
  prm.lo = d_lo;
  prm.span = d_hi >= d_lo ? static_cast<unsigned>(d_hi - d_lo) : 0u;
  if (d_hi < d_lo) prm.lo = 0x7fffffff;               // empty range: nothing passes
  SweepLaunch l{MODE_TILE, 0, PG_W_FLAG_U8, 0, 0, static_cast<cudaStream_t>(stream)};
  SweepTimer t(l.stream);
  return dispatch(planes, words, prm, l);
}

size_t pg_knn_sym_workspace_bytes(int64_t rows, int words) {
  if (rows <= 0 || words <= 0) return 0;
  return sym_layout(rows, words).total;
}

int pg_hamming_knn_boot(const uint32_t* table, int64_t table_rows, int64_t row0, int64_t rows, int64_t boot_rows,
                        int planes, int words, int k1, uint64_t* lists, void* workspace, size_t workspace_bytes,
                        void* stream) {
  int rc = check_common(table, table_rows, row0, rows, table, boot_rows, planes, words);
  if (rc != PG_OK) return rc;
  PG_CHECK_ARG(boot_rows <= table_rows, "bootstrap rows exceed the table");
  PG_CHECK_ARG(lists && workspace, "null output/workspace pointer");
  if (!sym_shape_ok(planes, words) || k1 < 1 || k1 > 32) {
    set_error("symmetric sweep: planes/words %d/%d or list length %d not covered", planes, words, k1);
    return PG_ERR_UNSUPPORTED;
  }
  const Geometry g = make_geometry(rows, boot_rows, words, kConsumers, k1);
  const size_t need = static_cast<size_t>(g.n_splits) * k1 * rows * 8;
  PG_CHECK_ARG(workspace_bytes >= need, "workspace too small: %zu < %zu", workspace_bytes, need);
  SweepParams prm;
  fill_common(prm, g, table, row0, rows, table, boot_rows);
  prm.part = static_cast<unsigned long long*>(workspace);
  prm.k1 = k1;
  SweepLaunch l{MODE_KNN, 0, PG_W_I64, 0, static_cast<size_t>(k1) * kConsumers * 8, static_cast<cudaStream_t>(stream)};
  {
    SweepTimer t(l.stream);
    rc = dispatch(planes, words, prm, l);
  }
  if (rc != PG_OK) return rc;
  const int threads = rows_per_merge_block(k1);
  knn_part_to_lists_kernel<<<static_cast<unsigned>(ceil_div(rows, threads)), threads, merge_smem_bytes(k1), l.stream>>>(
      prm.part, g.n_splits, k1, rows, reinterpret_cast<unsigned long long*>(lists));
  PG_LAUNCH_CHECK();
  return PG_OK;
}

int pg_knn_sym_band(int64_t rows, int words, int64_t boot_rows, int part, int parts, int64_t* row_begin,
                    int64_t* row_end) {
  PG_CHECK_ARG(rows > 0 && words > 0 && parts >= 1 && part >= 0 && part < parts && row_begin && row_end,
               "bad band arguments");
  const SymLayout lay = sym_layout(rows, words);
  int t0 = 0, t1 = 0;
  sym_band(lay, rows, boot_rows, part, parts, &t0, &t1);
  *row_begin = std::min<int64_t>(rows, static_cast<int64_t>(t0) * lay.tile_cols);
  *row_end = std::min<int64_t>(rows, static_cast<int64_t>(t1) * lay.tile_cols);
  return PG_OK;
}

int pg_knn_sym_plan(int64_t rows, int planes, int words, int64_t boot_rows, int part, int parts, int mode, int grid,
                    int32_t* items_host, int64_t capacity, int64_t* n_items) {
  PG_CHECK_ARG(rows > 0 && words > 0 && planes > 0 && parts >= 1 && part >= 0 && part < parts && grid >= 1 && n_items &&
                   (mode == 0 || mode == 1) && boot_rows >= 0 && boot_rows % kStreamRowPad == 0,
               "bad plan arguments");
  const SymLayout lay = sym_layout(rows, words, planes);
  const SymPlan plan = sym_plan(lay, rows, part, parts, mode, grid, boot_rows, sym_knn_chunk_floor(words, parts));
  *n_items = static_cast<int64_t>(plan.items.size());
  PG_CHECK_ARG(sym_plan_bytes(plan) <= lay.item_bytes_max, "item table overflow (%zu items)", plan.items.size());
  if (items_host) {
    int cta = 0;
    for (size_t i = 0; i < plan.items.size() && static_cast<int64_t>(i) < capacity; ++i) {
      while (static_cast<int>(i) >= plan.first[cta + 1]) ++cta;
      items_host[5 * i + 0] = plan.items[i].rb;
      items_host[5 * i + 1] = plan.items[i].t0;
      items_host[5 * i + 2] = plan.items[i].t1;
      items_host[5 * i + 3] = plan.items[i].boot;
      items_host[5 * i + 4] = cta;
    }
  }
  return PG_OK;
}

int pg_knn_sym_status(const void* workspace, int64_t rows, int words, void* stream) {
  PG_CHECK_ARG(workspace && rows > 0 && words > 0, "bad status arguments");
  const SymLayout lay = sym_layout(rows, words);
  unsigned err = 0;
  cudaStream_t cs = static_cast<cudaStream_t>(stream);
  PG_CUDA(cudaMemcpyAsync(&err, static_cast<const char*>(workspace) + lay.stats_off + 64, sizeof(err),
                          cudaMemcpyDeviceToHost, cs));
  PG_CUDA(cudaStreamSynchronize(cs));
  if (err != 0) {
    set_error("symmetric sweep: a row lock could not be taken within %u attempts (lists are incomplete)", kLockSpinLimit);
    return PG_ERR_CUDA;
  }
  return PG_OK;
}

int pg_hamming_knn_sym(const uint32_t* table, int64_t rows, int planes, int words, int k1, int part, int parts,
                       int mode, int64_t boot_rows, uint64_t* lists, void* workspace, size_t workspace_bytes,
                       void* stream) {
  const int rb_first = part, rb_stride = parts;
  PG_CHECK_ARG(mode == 0 || mode == 1, "bad partition mode %d", mode);
  PG_CHECK_ARG(table && lists && workspace, "null pointer");
  PG_CHECK_ARG(rows > 0 && rows < (1ll << 31), "row count out of range");
  PG_CHECK_ARG((reinterpret_cast<uintptr_t>(table) & 15) == 0, "table must be 16-byte aligned");
  PG_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "workspace must be 256-byte aligned");
  PG_CHECK_ARG(rb_stride >= 1 && rb_first >= 0 && rb_first < rb_stride, "bad row-block interleave %d/%d", rb_first,
               rb_stride);
  PG_CHECK_ARG(boot_rows >= 0 && boot_rows % kStreamRowPad == 0 && boot_rows <= rows,
               "bootstrap rows must be a multiple of %d within the table", kStreamRowPad);
  if (!sym_shape_ok(planes, words) || k1 < 1 || k1 > 32) {
    set_error("symmetric sweep: planes/words %d/%d or list length %d not covered", planes, words, k1);
    return PG_ERR_UNSUPPORTED;
  }
  const SymLayout lay = sym_layout(rows, words, planes);
  PG_CHECK_ARG(workspace_bytes >= lay.total, "workspace too small: %zu < %zu", workspace_bytes, lay.total);
  cudaStream_t cs = static_cast<cudaStream_t>(stream);
  char* wsb = static_cast<char*>(workspace);
  SymParams prm;
  memset(&prm, 0, sizeof(prm));
  prm.tab = table;
  prm.rows = rows;
  prm.one = 1u;
  prm.k1 = k1;
  prm.boot_rows = boot_rows;
  prm.glist = reinterpret_cast<unsigned long long*>(lists);
  prm.glast = reinterpret_cast<unsigned long long*>(wsb);
  prm.glock = reinterpret_cast<unsigned*>(wsb + lay.gnt_bytes);
  unsigned long long* stats_dev = reinterpret_cast<unsigned long long*>(wsb + lay.stats_off);
  const bool want_stats = std::getenv("PG_SYM_STATS") != nullptr;
  prm.stats = want_stats ? stats_dev : nullptr;
  prm.error = reinterpret_cast<unsigned*>(stats_dev + 8);
  SymLaunch l{0, static_cast<size_t>(k1) * kConsumers * 8, cs, SYM_KNN};
  int resident = 0;
  int rc = dispatch_sym(planes, words, prm, l, &resident);   // grid 0: occupancy query only
  if (rc != PG_OK) return rc;
  // a kNN chunk starts with empty shared-memory lists and ends with a locked merge of 256 lists: on
  // small tables of narrow rows (C3: 160 000 x 20 bytes) that is as long as sweeping 32 tiles, so the
  // chunks are at least 32 * 8/W tiles there (C3 kNN 18.4 -> 16.5 ms, profiles/r4i_chunks.log)
  // On one GPU, tables below ~250 000 rows also build faster with chunks of at least 256 * 8/W tiles
  // (70 000 rows: 12.4 -> 11.8 ms uniform, 13.7 -> 12.5 ms mutational; 131 072 rows: 36.0 -> 34.6 / 40.6 ->
  // 37.3 ms); the bands of a multi-rank build do not (rank 7 of 8 at 1 M rows: 199.8 -> 216 ms with twice
  // the default chunk: fewer merges mean staler row-side filters there) -- profiles/r4p_chunks.log.
  const SymPlan plan = sym_plan(lay, rows, part, parts, mode, resident, boot_rows, sym_knn_chunk_floor(words, parts));
  sym_init_kernel<<<num_sms() * 4, 256, 0, cs>>>(prm.glist, static_cast<long long>(rows) * k1, prm.glast,
                                                 static_cast<long long>(lay.n_tiles) * lay.tile_cols, prm.glock, rows,
                                                 stats_dev, k1, boot_rows > 0 ? 1 : 0);
  PG_LAUNCH_CHECK();
  if (plan.items.empty()) return PG_OK;
  rc = sym_upload_plan(plan, lay, wsb, &prm, cs);
  if (rc != PG_OK) return rc;
  l.grid = plan.grid;
  {
    SweepTimer t(cs);
    rc = dispatch_sym(planes, words, prm, l, nullptr);
  }
  if (rc == PG_OK && want_stats) {
    unsigned long long st[8];
    PG_CUDA(cudaMemcpyAsync(st, stats_dev, sizeof(st), cudaMemcpyDeviceToHost, cs));
    PG_CUDA(cudaStreamSynchronize(cs));
    fprintf(stderr, "[pg sym] rows=%lld boot=%lld items=%d grid=%d | locks %llu, lock spins %llu, list writes %llu | row "
            "inserts %llu\n", static_cast<long long>(rows), static_cast<long long>(boot_rows), prm.n_items, l.grid,
            st[1], st[2], st[3], st[4]);
  }
  return rc;
}

int pg_hamming_eps_sym(const uint32_t* table, int64_t rows, int planes, int words, const uint32_t* lut_host,
                       int lut_words, int part, int parts, int mode, uint64_t* keys, int64_t capacity,
                       uint64_t* counters, void* workspace, size_t workspace_bytes, void* stream) {
  PG_CHECK_ARG(table && keys && counters && workspace && lut_host, "null pointer");
  PG_CHECK_ARG(rows > 0 && rows < (1ll << 27), "row count out of range for packed edge keys");
  PG_CHECK_ARG((reinterpret_cast<uintptr_t>(table) & 15) == 0, "table must be 16-byte aligned");
  PG_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "workspace must be 256-byte aligned");
  PG_CHECK_ARG(parts >= 1 && part >= 0 && part < parts && (mode == 0 || mode == 1), "bad partition %d/%d mode %d", part,
               parts, mode);
  PG_CHECK_ARG(lut_words >= 1 && lut_words <= kMaxLutWords && lut_words * 32 > words * 32, "lut must cover distances 0..%d",
               words * 32);
  PG_CHECK_ARG(capacity >= 0, "negative capacity");
  if (!sym_shape_ok(planes, words)) {
    set_error("symmetric sweep: planes/words %d/%d not covered", planes, words);
    return PG_ERR_UNSUPPORTED;
  }
  SymParams prm;
  memset(&prm, 0, sizeof(prm));
  unsigned span = 0;
  if (!lut_as_range(lut_host, lut_words, &prm.lo, &span)) {
    set_error("symmetric epsilon sweep needs a contiguous distance range");
    return PG_ERR_UNSUPPORTED;
  }
  prm.hi = prm.lo == 0x7fffffff ? -1 : prm.lo + static_cast<int>(span);
  if (prm.lo == 0x7fffffff) prm.lo = 1 << 20;            // empty predicate: nothing passes
  const SymLayout lay = sym_layout(rows, words, planes);
  PG_CHECK_ARG(workspace_bytes >= lay.total, "workspace too small: %zu < %zu", workspace_bytes, lay.total);
  const EdgeKeyBits kb = edge_key_bits(rows, words);
  cudaStream_t cs = static_cast<cudaStream_t>(stream);
  char* wsb = static_cast<char*>(workspace);
  prm.tab = table;
  prm.rows = rows;
  prm.one = 1u;
  prm.k1 = 1;
  prm.sh_col = kb.dbits;
  prm.sh_row = kb.dbits + kb.idxbits;
  prm.keys = reinterpret_cast<unsigned long long*>(keys);
  prm.capacity = capacity;
  prm.counters = reinterpret_cast<unsigned long long*>(counters);
  SymLaunch l{0, 0, cs, SYM_EPS};
  int resident = 0;
  int rc = dispatch_sym(planes, words, prm, l, &resident);
  if (rc != PG_OK) return rc;
  const SymPlan plan = sym_plan(lay, rows, part, parts, mode, resident, 0);
  PG_CUDA(cudaMemsetAsync(counters, 0, 2 * sizeof(uint64_t), cs));
  if (plan.items.empty()) return PG_OK;
  rc = sym_upload_plan(plan, lay, wsb, &prm, cs);
  if (rc != PG_OK) return rc;
  l.grid = plan.grid;
  {
    SweepTimer t(cs);
    rc = dispatch_sym(planes, words, prm, l, nullptr);
  }
  return rc;
}

int pg_edge_keys_to_csr(uint64_t* keys, int64_t n_keys, uint64_t* keys_alt, int64_t rows, int words, int64_t nnz,
                        int weight, int64_t* indptr, int64_t* out_idx, void* out_w, void* stream) {
  PG_CHECK_ARG(indptr && rows > 0 && n_keys >= 0 && nnz >= 0 && nnz <= n_keys, "bad edge list geometry");
  PG_CHECK_ARG(n_keys < (1ll << 31), "too many edge slots for one sort");
  PG_CHECK_ARG(weight == PG_W_I64 || weight == PG_W_SIM_F32, "edges carry int64 distances or float32 similarities");
  cudaStream_t cs = static_cast<cudaStream_t>(stream);
  const EdgeKeyBits kb = edge_key_bits(rows, words);
  const unsigned long long* sorted = reinterpret_cast<const unsigned long long*>(keys);
  if (n_keys > 0) {
    PG_CHECK_ARG(keys && keys_alt && (nnz == 0 || (out_idx && out_w)), "null key / output buffers");
    // (row, column) order = the ascending-index rows of prograph.py:736-753; the distance rides in
    // the low bits and the sentinels (all ones) end up behind the last edge
    cub::DoubleBuffer<unsigned long long> buf(reinterpret_cast<unsigned long long*>(keys),
                                              reinterpret_cast<unsigned long long*>(keys_alt));
    size_t tmp_bytes = 0;
    PG_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, buf, static_cast<int>(n_keys), kb.dbits,
                                           kb.dbits + 2 * kb.idxbits, cs));
    void* tmp = nullptr;
    PG_CUDA(temp_alloc(&tmp, tmp_bytes, cs));
    cudaError_t e = cub::DeviceRadixSort::SortKeys(tmp, tmp_bytes, buf, static_cast<int>(n_keys), kb.dbits,
                                                   kb.dbits + 2 * kb.idxbits, cs);
    count_launch();
    cudaFreeAsync(tmp, cs);
    if (e != cudaSuccess) { set_error("cub radix sort failed: %s", cudaGetErrorString(e)); return PG_ERR_CUDA; }
    sorted = buf.Current();
  }
  const int threads = 256;
  const long long work = nnz > 0 ? nnz : rows + 1;
  edge_decode_kernel<<<static_cast<unsigned>(std::min<long long>(ceil_div(work, threads), 1 << 30)), threads, 0, cs>>>(
      sorted, nnz, rows, kb.dbits, kb.idxbits, weight, reinterpret_cast<long long*>(indptr),
      reinterpret_cast<long long*>(out_idx), out_w);
  PG_LAUNCH_CHECK();
  return PG_OK;
}


static int knn_lists_launch(const uint64_t* lists, int n_lists, int64_t list_stride, int64_t row0, int64_t rows, int k1,
                            int k, int drop, int weight, uint64_t* out_keys, int64_t* out_idx, void* out_w, void* stream) {
  PG_CHECK_ARG(lists && (out_keys || (out_idx && out_w)), "null pointer");
  PG_CHECK_ARG(n_lists >= 1 && rows > 0 && row0 >= 0 && k >= 1 && drop >= 0 && k1 >= 1, "bad list geometry");
  PG_CHECK_ARG(weight == PG_W_I64 || weight == PG_W_SIM_F32 || weight == PG_W_I32, "bad weight kind %d", weight);
  const int threads = rows_per_merge_block(k);
  const size_t msm = merge_smem_bytes(k);
  const unsigned grid = static_cast<unsigned>(ceil_div(rows, threads));
  cudaStream_t cs = static_cast<cudaStream_t>(stream);
  const unsigned long long* src = reinterpret_cast<const unsigned long long*>(lists);
  unsigned long long* ok = reinterpret_cast<unsigned long long*>(out_keys);
  if (n_lists == 1 && out_keys == nullptr) {
    const long long blocks = std::min<long long>(ceil_div(rows * k, 256), static_cast<long long>(num_sms()) * 16);
    knn_keys_widen_kernel<<<static_cast<unsigned>(blocks), 256, 0, cs>>>(src, row0, rows, k1, k, drop, weight,
                                                                        reinterpret_cast<long long*>(out_idx), out_w);
  } else if (n_lists <= kMaxMergeLists) {
    knn_lists_finalize_kernel<<<grid, threads, msm, cs>>>(src, n_lists, list_stride, row0, rows, k1, k, drop, weight,
                                                        out_keys != nullptr, ok, reinterpret_cast<long long*>(out_idx), out_w);
  } else {
    knn_lists_finalize_scan_kernel<<<grid, threads, msm, cs>>>(src, n_lists, list_stride, row0, rows, k1, k, drop, weight,
                                                             out_keys != nullptr, ok, reinterpret_cast<long long*>(out_idx),
                                                             out_w);
  }
  PG_LAUNCH_CHECK();
  return PG_OK;
}

int pg_knn_lists_finalize(const uint64_t* lists, int n_lists, int64_t list_stride, int64_t row0, int64_t rows, int k1,
                          int k, int drop, int weight, int64_t* out_idx, void* out_w, void* stream) {
  PG_CHECK_ARG(out_idx && out_w, "null output pointer");
  return knn_lists_launch(lists, n_lists, list_stride, row0, rows, k1, k, drop, weight, nullptr, out_idx, out_w, stream);
}

int pg_knn_lists_merge(const uint64_t* lists, int n_lists, int64_t list_stride, int64_t row0, int64_t rows, int k1, int k,
                       int drop, uint64_t* out_keys, void* stream) {
  PG_CHECK_ARG(out_keys, "null output pointer");
  return knn_lists_launch(lists, n_lists, list_stride, row0, rows, k1, k, drop, PG_W_I64, out_keys, nullptr, nullptr,
                          stream);
}


int pg_exclusive_scan_i64(const int64_t* in, int64_t n, int64_t* out, void* stream) {
  PG_CHECK_ARG(in && out && n >= 0, "bad scan arguments");
  if (n == 0) {
    PG_CUDA(cudaMemsetAsync(out, 0, sizeof(int64_t), static_cast<cudaStream_t>(stream)));
    return PG_OK;
  }
  // out[0..n-1] exclusive, out[n] = total: run an inclusive scan into out+1 and zero out[0]
  size_t tmp_bytes = 0;
  PG_CUDA(cub::DeviceScan::InclusiveSum(nullptr, tmp_bytes, in, out + 1, static_cast<int>(n),
                                        static_cast<cudaStream_t>(stream)));
  void* tmp = nullptr;
  PG_CUDA(temp_alloc(&tmp, tmp_bytes, static_cast<cudaStream_t>(stream)));
  cudaError_t e = cub::DeviceScan::InclusiveSum(tmp, tmp_bytes, in, out + 1, static_cast<int>(n),
                                                static_cast<cudaStream_t>(stream));
  count_launch();
  cudaFreeAsync(tmp, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) { set_error("cub scan failed: %s", cudaGetErrorString(e)); return PG_ERR_CUDA; }
  PG_CUDA(cudaMemsetAsync(out, 0, sizeof(int64_t), static_cast<cudaStream_t>(stream)));
  return PG_OK;
}

int pg_time_sweeps(int enable) {
  std::lock_guard<std::mutex> g(g_time_mu);
  g_time_enabled = enable != 0;
  return PG_OK;
}

int pg_sweep_time(double* total_ms, int64_t* launches, int reset) {
  std::lock_guard<std::mutex> g(g_time_mu);
  double tot = 0;
  for (auto& ev : g_time_events) {
    cudaEventSynchronize(ev.second);
    float ms = 0;
    cudaEventElapsedTime(&ms, ev.first, ev.second);
    tot += ms;
  }
  if (total_ms) *total_ms = tot;
  if (launches) *launches = static_cast<int64_t>(g_time_events.size());
  if (reset) {
    for (auto& ev : g_time_events) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
    g_time_events.clear();
  }
  return PG_OK;
}

int pg_sweep_times(double* ms, int64_t cap, int64_t* n, int reset) {
  std::lock_guard<std::mutex> g(g_time_mu);
  int64_t i = 0;
  for (auto& ev : g_time_events) {
    cudaEventSynchronize(ev.second);
    float t = 0;
    cudaEventElapsedTime(&t, ev.first, ev.second);
    if (ms && i < cap) ms[i] = t;
    ++i;
  }
  if (n) *n = i;
  if (reset) {
    for (auto& ev : g_time_events) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
    g_time_events.clear();
  }
  return PG_OK;
}

}  // extern "C"
