// Fused all-pairs Hamming sweep for sm_100a.
//
// Replaces  torch.sum(X != Y[:,None,:], axis=2)  (prograph/distance/hamming.py:34) together
// with the consumer that follows it in prograph/prograph.py (sort+slice :757-762,
// where+gather :734-739, or the plain (M,N) result).
//
// Mapping ("own rows in registers, stream rows by broadcast"):
//   * a CTA owns 256 "own" rows, one per consumer thread; the thread keeps its row's
//     P bit planes x W words (P*W registers) for the whole sweep;
//   * the "stream" table is swept through a 4-stage shared-memory ring filled with 1-D
//     bulk async copies (TMA engine, cp.async.bulk + mbarrier).  There is no producer warp:
//     the warp that finishes a stage last re-arms its barrier and issues the copy of the
//     tile four positions ahead, so nobody ever polls for a free slot;
//   * every thread reads the same stream row at the same time, so shared-memory reads are
//     pure broadcasts (two wavefronts per 128-bit load, no bank conflicts);
//   * per pair and 32 residues: 5 LOP3 (xor/or fold of the planes) + 1 POPC + 1 IADD;
//   * the epilogue sees (own row, stream row, distance) in ascending stream order and
//     never writes the distance matrix: kNN keeps a sorted (distance,index) list per
//     own row in shared memory behind a register threshold; the epsilon passes count /
//     emit edges; the tile mode stores distances coalesced along the own index.
// Work items are (row block, stream split) pairs walked by a persistent grid.
#pragma once
#include "pg_common.cuh"

namespace pg {

constexpr int kConsumerWarps = 8;
constexpr int kConsumers = kConsumerWarps * 32;  // threads per CTA; each owns one row
constexpr int kSweepThreads = kConsumers;
constexpr int kStages = 4;
constexpr int kMaxLutWords = 64;                 // truth table in the parameter block: distances up to 2047
                                                 // (the chunked long-row sweep takes longer ones: SweepLaunch::lut_ext)
constexpr int kWideMaxWords = 1024;              // chunked long-row sweep: rows of up to 32768 residues
constexpr int kEpsCapture = 128;                  // default hits per (split, row) kept by the count pass

enum SweepMode { MODE_KNN = 0, MODE_COUNT = 1, MODE_FILL = 2, MODE_TILE = 3 };

template <int W>
struct TileCols {  // stream rows per ring stage: 64 rows of 8 words (2 KB per plane)
  static constexpr int value = 512 / W;
};

struct SweepParams {
  const uint32_t* own;   // packed table holding the own rows
  long long own_row0;    // first own row to process
  long long rows;        // number of own rows to process (length of row_map when it is set)
  const long long* row_map;  // optional: the own rows to process, relative to own_row0 (fill of a row subset)
  long long rows_total;      // row stride of split_counts / capture / part (= rows unless row_map is set)
  const uint32_t* str;   // packed stream table (padded to kStreamRowPad rows)
  long long str_rows;    // valid stream rows
  int n_rowblocks, n_splits, tiles_per_split, n_tiles;
  unsigned one;          // the constant 1, opaque to the compiler: `mad p, one, acc` keeps the
                         // popcount sums on the FMA pipe (IMAD), off the LOP3-saturated ALU pipe
  // kNN
  unsigned long long* part;  // [n_splits][k1][rows] sorted partial lists, key = d<<32 | idx
  int k1;
  // epsilon passes
  int lo;                 // range test (unsigned)(d - lo) <= span when !LUT
  unsigned span;
  long long* split_counts;  // [n_splits][rows]
  unsigned long long* capture;  // count pass: first capture_cap hits of every (split,row), d<<32|idx; or null
  int capture_cap;              // slots per (split,row) of `capture` (kEpsCapture unless the caller sized the workspace for more)
  const long long* indptr;  // [rows+1]                          (fill)
  long long* out_idx;       // edges                              (fill)
  void* out_w;
  // tile
  void* out;
  long long ld;
  uint32_t lut[kMaxLutWords];
};

__device__ __forceinline__ unsigned mad_u32(unsigned a, unsigned b, unsigned c) {
  unsigned r;
  asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}

// Distance of the own row (registers) to one stream row (shared memory, broadcast loads).
template <int P, int W>
__device__ __forceinline__ int ham_rows(const uint32_t (&q)[P * W], const uint32_t* __restrict__ col, unsigned one) {
  uint32_t m[W];
  if constexpr (W % 4 == 0) {
    const uint4* c4 = reinterpret_cast<const uint4*>(col);
#pragma unroll
    for (int p = 0; p < P; ++p) {
#pragma unroll
      for (int h = 0; h < W / 4; ++h) {
        const uint4 v = c4[p * (W / 4) + h];
        const int w = h * 4;
        if (p == 0) {
          m[w + 0] = q[w + 0] ^ v.x;
          m[w + 1] = q[w + 1] ^ v.y;
          m[w + 2] = q[w + 2] ^ v.z;
          m[w + 3] = q[w + 3] ^ v.w;
        } else {
          m[w + 0] |= q[p * W + w + 0] ^ v.x;
          m[w + 1] |= q[p * W + w + 1] ^ v.y;
          m[w + 2] |= q[p * W + w + 2] ^ v.z;
          m[w + 3] |= q[p * W + w + 3] ^ v.w;
        }
      }
    }
  } else if constexpr (W == 2) {
    const uint2* c2 = reinterpret_cast<const uint2*>(col);
#pragma unroll
    for (int p = 0; p < P; ++p) {
      const uint2 v = c2[p];
      if (p == 0) {
        m[0] = q[0] ^ v.x;
        m[1] = q[1] ^ v.y;
      } else {
        m[0] |= q[p * 2 + 0] ^ v.x;
        m[1] |= q[p * 2 + 1] ^ v.y;
      }
    }
  } else {
#pragma unroll
    for (int p = 0; p < P; ++p) {
#pragma unroll
      for (int w = 0; w < W; ++w) {
        const uint32_t v = col[p * W + w];
        if (p == 0) m[w] = q[w] ^ v;
        else m[w] |= q[p * W + w] ^ v;
      }
    }
  }
  unsigned s = __popc(m[0]);
#pragma unroll
  for (int w = 1; w < W; ++w) s = mad_u32(__popc(m[w]), one, s);
  return static_cast<int>(s);
}

// Distances of the own row to FOUR consecutive stream rows (col: the first of them, 16-byte aligned:
// every tile starts aligned and the callers step in groups of four).  Rows of a multiple of four
// words are read with 128-bit loads by ham_rows already.  Narrow rows (W = 1, 2: 20 / 40 bytes at five
// planes) are not 16-byte multiples on their own, so one row at a time means 32- or 64-bit loads --
// five shared-memory instructions per pair, and the shared-memory pipe takes one per clock and SM:
// the W = 1 sweep ran at 27 clocks per pair-warp on 20 clocks of LDS.  Four rows together ARE a
// multiple of 16 bytes: P*W 128-bit loads per four pairs.
template <int P, int W>
__device__ __forceinline__ void ham_rows4(const uint32_t (&q)[P * W], const uint32_t* __restrict__ col, int (&d)[4],
                                          unsigned one) {
  constexpr int COLW = P * W;
  if constexpr (W % 4 == 0) {
#pragma unroll
    for (int r = 0; r < 4; ++r) d[r] = ham_rows<P, W>(q, col + r * COLW, one);
  } else {
    uint32_t v[4 * COLW];
    const uint4* c4 = reinterpret_cast<const uint4*>(col);
#pragma unroll
    for (int i = 0; i < COLW; ++i) {
      const uint4 t = c4[i];
      v[4 * i + 0] = t.x;
      v[4 * i + 1] = t.y;
      v[4 * i + 2] = t.z;
      v[4 * i + 3] = t.w;
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      uint32_t m[W];
#pragma unroll
      for (int w = 0; w < W; ++w) {
        m[w] = q[w] ^ v[r * COLW + w];
#pragma unroll
        for (int p = 1; p < P; ++p) m[w] |= q[p * W + w] ^ v[r * COLW + p * W + w];
      }
      unsigned s = __popc(m[0]);
#pragma unroll
      for (int w = 1; w < W; ++w) s = mad_u32(__popc(m[w]), one, s);
      d[r] = static_cast<int>(s);
    }
  }
}

__device__ __forceinline__ void write_weight(void* out_w, long long at, int d, int weight) {
  if (weight == PG_W_I64) reinterpret_cast<long long*>(out_w)[at] = d;
  else if (weight == PG_W_SIM_F32) reinterpret_cast<float*>(out_w)[at] = sim_f32(d);
  else reinterpret_cast<int*>(out_w)[at] = d;
}

// tile epilogue: the distance (or the range flag lo <= d <= lo + span) of one (stream, own) pair
template <int WEIGHT>
__device__ __forceinline__ void write_tile(void* out, long long at, int d, int lo, unsigned span) {
  if constexpr (WEIGHT == PG_W_FLAG_U8) reinterpret_cast<uint8_t*>(out)[at] = static_cast<unsigned>(d - lo) <= span ? 1 : 0;
  else write_weight(out, at, d, WEIGHT);
}

constexpr int kMaxListRounds = 3;  // sorted lists of up to 96 entries, one entry per lane and round

// Warp-cooperative sorted insertion: the whole warp inserts `key` into the ascending list of
// one own row (list[0..k1), contiguous in shared memory) and returns the distance word of
// the new last entry.  All lanes must call it with the same arguments.  No divergent loop:
// a ballot finds the insertion point, every lane rewrites its own slot.
__device__ __forceinline__ unsigned knn_insert_coop(unsigned long long* list, int k1, unsigned long long key, int lane) {
  unsigned long long cur[kMaxListRounds], prev[kMaxListRounds];
  int pos = 0;
#pragma unroll
  for (int r = 0; r < kMaxListRounds; ++r) {
    const int j = lane + 32 * r;
    const bool in = j < k1;
    cur[r] = in ? list[j] : ~0ull;
    prev[r] = (in && j > 0) ? list[j - 1] : 0ull;
    pos += __popc(__ballot_sync(0xffffffffu, in && cur[r] < key));
  }
  __syncwarp();
#pragma unroll
  for (int r = 0; r < kMaxListRounds; ++r) {
    const int j = lane + 32 * r;
    if (j < k1 && j >= pos) list[j] = (j == pos) ? key : prev[r];
  }
  __syncwarp();
  return static_cast<unsigned>(list[k1 - 1] >> 32);
}

// Position of a CTA in its sequence of (work item, ring tile) pairs.
struct SweepCursor {
  int item, t, t1;
  __device__ __forceinline__ void start(int it, const SweepParams& prm) {
    item = it;
    if (item < prm.n_rowblocks * prm.n_splits) {
      const int split = item / prm.n_rowblocks;
      t = split * prm.tiles_per_split;
      t1 = min(t + prm.tiles_per_split, prm.n_tiles);
    } else {
      t = t1 = 0;
    }
  }
  __device__ __forceinline__ bool valid(const SweepParams& prm) const { return item < prm.n_rowblocks * prm.n_splits; }
  __device__ __forceinline__ void advance(const SweepParams& prm, int stride) {
    if (++t == t1) start(item + stride, prm);
  }
};

// ---- the ring protocol shared by every sweep ------------------------------------------------
// n_stages shared-memory stages, each with a `full` mbarrier that its bulk copies complete on and a
// `done` count of the consumer warps through with it.  There is no producer warp: the warp that
// finishes a stage last re-arms it and issues the copy of the lookahead unit.  A kernel describes its
// lookahead cursor with three callbacks: more() -- is there a unit left; issue(s) -- copy that unit
// into stage s (called by thread 0, or with WARP_ISSUE by all lanes of warp 0 / of the last warp);
// step() -- advance the cursor (every thread, once per unit consumed or primed).

// Barrier set-up, then setup() on every thread (e.g. the truth-table copy), a block barrier, and the
// prologue that fills every stage.
template <bool WARP_ISSUE = false, typename Setup, typename More, typename Issue, typename Step>
__device__ __forceinline__ void ring_start(uint64_t* full, unsigned* done, int n_stages, int tid, Setup&& setup,
                                           More&& more, Issue&& issue, Step&& step) {
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < n_stages; ++s) {
      mbar_init(&full[s], 1);
      done[s] = 0;
    }
    fence_mbar_init();
  }
  setup();
  __syncthreads();
#pragma unroll 1
  for (int s = 0; s < n_stages; ++s) {
    if ((WARP_ISSUE ? (tid >> 5) == 0 : tid == 0) && more()) issue(s);
    step();
  }
}

// This warp is done with `stage`: the last warp through resets the counter and refills the stage
// with the lookahead unit; then the cursor and the (stage, phase) pair move on.
template <bool WARP_ISSUE = false, typename More, typename Issue, typename Step>
__device__ __forceinline__ void ring_release(unsigned* done, int& stage, uint32_t& phase, int n_stages, int lane,
                                             More&& more, Issue&& issue, Step&& step) {
  __syncwarp();
  if constexpr (WARP_ISSUE) {
    unsigned last = 0;
    if (lane == 0) last = atom_add_acq_rel_cta(&done[stage], 1u) == kConsumerWarps - 1;
    last = __shfl_sync(0xffffffffu, last, 0);
    if (last) {
      if (lane == 0) done[stage] = 0;
      if (more()) {
        fence_proxy_async();
        issue(stage);
      }
    }
  } else if (lane == 0) {
    if (atom_add_acq_rel_cta(&done[stage], 1u) == kConsumerWarps - 1) {
      done[stage] = 0;
      if (more()) {
        fence_proxy_async();
        issue(stage);
      }
    }
  }
  step();
  if (++stage == n_stages) { stage = 0; phase ^= 1u; }
}

// ---- the one-sided epilogues ---------------------------------------------------------------
// What a one-sided sweep does with the distances of a thread's own row, in ascending stream order:
// kNN keeps a sorted (distance, index) list in shared memory behind a register threshold, count
// tallies (and captures) the hits of the epsilon predicate, fill writes them as edges, tile stores
// every distance.  LUT_BOUND: distances may lie beyond the truth table of lut_bits entries (the pad
// rows of the long-row sweep) and are tested against its length first.
template <int MODE, bool LUT, int WEIGHT, bool LUT_BOUND = false>
struct SweepEpilogue {
  const SweepParams& prm;
  unsigned long long* lists;   // [kConsumers][k1]
  const uint32_t* lut_s;
  int lut_bits;
  int tid, split;
  long long r;                 // own row relative to own_row0
  bool valid;
  unsigned tau;                // kNN: distance word of the k1-th list entry (the filter threshold)
  long long cnt;               // count / fill cursor
  unsigned long long* cap;

  // Row and state of work item (row block rb, stream split `split`).
  __device__ __forceinline__ void begin(int rb, int split_) {
    split = split_;
    cap = nullptr;
    r = static_cast<long long>(rb) * kConsumers + tid;
    valid = r < prm.rows;
    if (prm.row_map != nullptr && valid) r = prm.row_map[r];
    tau = valid ? 0xffffffffu : 0u;
    cnt = 0;
    if constexpr (MODE == MODE_KNN) {
      unsigned long long* mine = lists + static_cast<size_t>(tid) * prm.k1;
      for (int j = 0; j < prm.k1; ++j) mine[j] = ~0ull;
    }
    if constexpr (MODE == MODE_COUNT) {
      if (valid && prm.capture != nullptr)
        cap = prm.capture + (static_cast<size_t>(split) * prm.rows_total + r) * prm.capture_cap;
    }
    if constexpr (MODE == MODE_FILL) {
      if (valid) {
        cnt = prm.indptr[r];
        for (int s = 0; s < split; ++s) cnt += prm.split_counts[static_cast<size_t>(s) * prm.rows_total + r];
      }
    }
  }
  // the own row in the packed table (row 0 stands in for an invalid one)
  __device__ __forceinline__ size_t own_row() const { return static_cast<size_t>(prm.own_row0 + (valid ? r : 0)); }

  // kNN: the candidates of one stream row are rare, so a ballot first, then the warp inserts them
  // one by one (warp-uniform control flow)
  __device__ __forceinline__ void serve(int dv, long long col) {
    const int lane = tid & 31;
    unsigned cand = __ballot_sync(0xffffffffu, static_cast<unsigned>(dv) < tau);
    while (cand) {
      const int src = __ffs(cand) - 1;
      cand &= cand - 1;
      const unsigned dd = __shfl_sync(0xffffffffu, static_cast<unsigned>(dv), src);
      const unsigned long long key = (static_cast<unsigned long long>(dd) << 32) | static_cast<unsigned>(col);
      unsigned long long* lst = lists + static_cast<size_t>(((tid >> 5) << 5) + src) * prm.k1;
      const unsigned t_new = knn_insert_coop(lst, prm.k1, key, lane);
      if (lane == src) tau = t_new;
    }
  }

  // the distance d to stream row `col`
  __device__ __forceinline__ void offer(int d, long long col) {
    if constexpr (MODE == MODE_KNN) {
      serve(d, col);
    } else if constexpr (MODE == MODE_TILE) {  // out[stream * ld + own]
      if (valid) write_tile<WEIGHT>(prm.out, col * prm.ld + r, d, prm.lo, prm.span);
    } else {
      bool hit;
      if constexpr (LUT && LUT_BOUND) hit = d < lut_bits && ((lut_s[d >> 5] >> (d & 31)) & 1u);
      else if constexpr (LUT) hit = (lut_s[d >> 5] >> (d & 31)) & 1u;
      else hit = static_cast<unsigned>(d - prm.lo) <= prm.span;
      if (hit && valid) {
        if constexpr (MODE == MODE_COUNT) {
          // sparse graphs: keep the first hits so that the fill sweep can be skipped
          if (cap != nullptr && cnt < prm.capture_cap)
            cap[cnt] = (static_cast<unsigned long long>(static_cast<unsigned>(d)) << 32) | static_cast<unsigned>(col);
        } else {
          prm.out_idx[cnt] = col;
          write_weight(prm.out_w, cnt, d, WEIGHT);
        }
        ++cnt;
      }
    }
  }

  // the distances to the four stream rows col .. col+3; kNN: one min + one compare + one vote per
  // group keeps the per-pair overhead on the ALU pipe near zero
  __device__ __forceinline__ void offer4(const int (&d)[4], long long col) {
    if constexpr (MODE == MODE_KNN) {
      const unsigned best = min(min(static_cast<unsigned>(d[0]), static_cast<unsigned>(d[1])),
                                min(static_cast<unsigned>(d[2]), static_cast<unsigned>(d[3])));
      if (__any_sync(0xffffffffu, best < tau)) {
        serve(d[0], col + 0);
        serve(d[1], col + 1);
        serve(d[2], col + 2);
        serve(d[3], col + 3);
      }
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e) offer(d[e], col + e);
    }
  }

  // write back the split's list (kNN) or count
  __device__ __forceinline__ void end() {
    if constexpr (MODE == MODE_KNN) {
      if (valid) {
        const unsigned long long* mine = lists + static_cast<size_t>(tid) * prm.k1;
        unsigned long long* dst = prm.part + static_cast<size_t>(split) * prm.k1 * prm.rows_total + r;
        for (int j = 0; j < prm.k1; ++j) dst[static_cast<size_t>(j) * prm.rows_total] = mine[j];
      }
      __syncwarp();
    } else if constexpr (MODE == MODE_COUNT) {
      if (valid) prm.split_counts[static_cast<size_t>(split) * prm.rows_total + r] = cnt;
    }
  }
};

template <int P, int W, int MODE, bool LUT, int WEIGHT>
__global__ void __launch_bounds__(kSweepThreads, 2) sweep_kernel(const __grid_constant__ SweepParams prm) {
  constexpr int BN = TileCols<W>::value;
  constexpr int COLW = P * W;
  constexpr uint32_t STAGE_BYTES = BN * COLW * 4;
  static_assert(STAGE_BYTES % 16 == 0, "bulk copies move multiples of 16 bytes");

  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint32_t* stage_mem = reinterpret_cast<uint32_t*>(smem_raw);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + kStages * STAGE_BYTES);
  unsigned* done = reinterpret_cast<unsigned*>(full + kStages);   // warps finished with a stage
  uint32_t* lut_s = reinterpret_cast<uint32_t*>(full + 2 * kStages);
  unsigned long long* lists = reinterpret_cast<unsigned long long*>(lut_s + kMaxLutWords);  // [kConsumers][k1]

  const int tid = threadIdx.x;
  const int lane = tid & 31;

  // lookahead cursor: the tile that goes into a stage when its current tile has been consumed
  SweepCursor la;
  la.start(blockIdx.x, prm);
  auto more = [&] { return la.valid(prm); };
  auto issue = [&](int s) {
    mbar_arrive_expect_tx(&full[s], STAGE_BYTES);
    bulk_g2s(stage_mem + s * (BN * COLW), prm.str + static_cast<size_t>(la.t) * BN * COLW, STAGE_BYTES, &full[s]);
  };
  auto step = [&] { if (la.valid(prm)) la.advance(prm, gridDim.x); };
  ring_start(full, done, kStages, tid, [&] { if (LUT && tid < kMaxLutWords) lut_s[tid] = prm.lut[tid]; }, more, issue, step);

  const int n_items = prm.n_rowblocks * prm.n_splits;
  int stage = 0;
  uint32_t phase = 0;
  SweepEpilogue<MODE, LUT, WEIGHT> ep{prm, lists, lut_s, kMaxLutWords * 32, tid};

  for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int split = item / prm.n_rowblocks;
    ep.begin(item - split * prm.n_rowblocks, split);
    uint32_t q[COLW];
    const uint32_t* src = prm.own + ep.own_row() * COLW;
#pragma unroll
    for (int j = 0; j < COLW; ++j) q[j] = ep.valid ? __ldg(src + j) : 0u;
    const unsigned one = prm.one;
    if constexpr (MODE == MODE_KNN) __syncwarp();

    const int t0 = split * prm.tiles_per_split;
    const int t1 = min(t0 + prm.tiles_per_split, prm.n_tiles);
    for (int t = t0; t < t1; ++t) {
      mbar_wait(&full[stage], phase);
      const uint32_t* tile = stage_mem + stage * (BN * COLW);
      const long long col0 = static_cast<long long>(t) * BN;
      const int ncols = static_cast<int>(min(static_cast<long long>(BN), prm.str_rows - col0));
      int c = 0;
      // kNN: four stream rows per vote; narrow rows: four stream rows per group of 128-bit loads (see ham_rows4)
      if constexpr (MODE == MODE_KNN || W % 4 != 0) {
#pragma unroll 1
        for (; c + 4 <= ncols; c += 4) {
          int d[4];
          ham_rows4<P, W>(q, tile + c * COLW, d, one);
          ep.offer4(d, col0 + c);
        }
      }
#pragma unroll 2
      for (; c < ncols; ++c) ep.offer(ham_rows<P, W>(q, tile + c * COLW, one), col0 + c);
      ring_release(done, stage, phase, kStages, lane, more, issue, step);
    }
    ep.end();
  }
}

}  // namespace pg

// ---- host-side launchers ---------------------------------------------------------------
namespace pg {

struct SweepLaunch {
  int mode;    // SweepMode
  int lut;     // 0 range test, 1 LUT
  int weight;  // pgWeight (tile: compile time; fill: runtime)
  size_t list_bytes;  // kNN lists (all own rows of a CTA)
  cudaStream_t stream;
  // chunked long-row sweep: the truth table (count / fill with lut = 1) has lut_words words, in
  // SweepParams::lut when they fit, else in device memory at lut_ext
  int lut_words = kMaxLutWords;
  const uint32_t* lut_ext = nullptr;
};

// The (mode, LUT, weight) instantiation of a launch: f(SweepVariant<...>{}).
template <int M, bool L, int WT>
struct SweepVariant {
  static constexpr int mode = M;
  static constexpr bool lut = L;
  static constexpr int weight = WT;
};

template <typename F>
int with_sweep_variant(const SweepLaunch& l, F&& f) {
  switch (l.mode) {
    case MODE_KNN: return f(SweepVariant<MODE_KNN, false, 0>{});
    case MODE_COUNT: return l.lut ? f(SweepVariant<MODE_COUNT, true, 0>{}) : f(SweepVariant<MODE_COUNT, false, 0>{});
    case MODE_FILL:
      if (l.weight == PG_W_SIM_F32)
        return l.lut ? f(SweepVariant<MODE_FILL, true, PG_W_SIM_F32>{}) : f(SweepVariant<MODE_FILL, false, PG_W_SIM_F32>{});
      return l.lut ? f(SweepVariant<MODE_FILL, true, PG_W_I64>{}) : f(SweepVariant<MODE_FILL, false, PG_W_I64>{});
    case MODE_TILE:
      if (l.weight == PG_W_I64) return f(SweepVariant<MODE_TILE, false, PG_W_I64>{});
      if (l.weight == PG_W_SIM_F32) return f(SweepVariant<MODE_TILE, false, PG_W_SIM_F32>{});
      if (l.weight == PG_W_FLAG_U8) return f(SweepVariant<MODE_TILE, false, PG_W_FLAG_U8>{});
      return f(SweepVariant<MODE_TILE, false, PG_W_I32>{});
  }
  set_error("bad sweep mode %d", l.mode);
  return PG_ERR_INVALID;
}

// Launch `kern` (kSweepThreads threads, `smem` bytes of dynamic shared memory) on a persistent grid:
// one CTA per resident slot, at most n_items.  *resident (if set) receives the resident CTA count;
// n_items = 0 only reports it.
template <typename Kern, typename... Args>
int launch_persistent(Kern kern, size_t smem, long long n_items, cudaStream_t stream, int* resident, Args... args) {
  PG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  int occ = 0;
  PG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kSweepThreads, smem));
  if (occ < 1) { set_error("sweep kernel does not fit on an SM (smem %zu bytes)", smem); return PG_ERR_UNSUPPORTED; }
  const long long slots = static_cast<long long>(num_sms()) * occ;
  if (resident) *resident = static_cast<int>(slots);
  if (n_items <= 0) return PG_OK;
  const long long grid = n_items < slots ? n_items : slots;
  kern<<<static_cast<unsigned>(grid), kSweepThreads, smem, stream>>>(args...);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

template <int P, int W>
inline size_t sweep_smem_bytes(size_t list_bytes) {
  return static_cast<size_t>(kStages) * TileCols<W>::value * P * W * 4 + 2 * kStages * sizeof(uint64_t) +
         kMaxLutWords * 4 + list_bytes;   // ring + barriers/counters + lut + kNN lists
}

template <int P, int W>
int launch_sweep(const SweepParams& prm, const SweepLaunch& l) {
  return with_sweep_variant(l, [&](auto v) {
    using V = decltype(v);
    return launch_persistent(sweep_kernel<P, W, V::mode, V::lut, V::weight>, sweep_smem_bytes<P, W>(l.list_bytes),
                             static_cast<long long>(prm.n_rowblocks) * prm.n_splits, l.stream, nullptr, prm);
  });
}

// defined in pg_sweep_inst.cu, one per (P, W)
#define PG_DECL_SWEEP(P, W) int sweep_p##P##_w##W(const SweepParams& prm, const SweepLaunch& l);
PG_DECL_SWEEP(5, 1) PG_DECL_SWEEP(5, 2) PG_DECL_SWEEP(5, 4) PG_DECL_SWEEP(5, 8) PG_DECL_SWEEP(5, 16)
PG_DECL_SWEEP(8, 1) PG_DECL_SWEEP(8, 2) PG_DECL_SWEEP(8, 4) PG_DECL_SWEEP(8, 8)
#undef PG_DECL_SWEEP

}  // namespace pg
