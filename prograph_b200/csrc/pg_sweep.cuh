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
//     pure broadcasts (two wavefronts per 128-bit load, no bank conflicts) shared by the
//     TM own rows of the thread;
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
constexpr int kConsumers = kConsumerWarps * 32;  // threads per CTA; each owns TM rows
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

// Distances of TM own rows (registers) to one stream row (shared memory, broadcast loads).
template <int P, int W, int TM>
__device__ __forceinline__ void ham_rows(const uint32_t (&q)[TM][P * W], const uint32_t* __restrict__ col,
                                         int (&d)[TM], unsigned one) {
  uint32_t m[TM][W];
  if constexpr (W % 4 == 0) {
    const uint4* c4 = reinterpret_cast<const uint4*>(col);
#pragma unroll
    for (int p = 0; p < P; ++p) {
#pragma unroll
      for (int h = 0; h < W / 4; ++h) {
        const uint4 v = c4[p * (W / 4) + h];
        const int w = h * 4;
#pragma unroll
        for (int i = 0; i < TM; ++i) {
          if (p == 0) {
            m[i][w + 0] = q[i][w + 0] ^ v.x;
            m[i][w + 1] = q[i][w + 1] ^ v.y;
            m[i][w + 2] = q[i][w + 2] ^ v.z;
            m[i][w + 3] = q[i][w + 3] ^ v.w;
          } else {
            m[i][w + 0] |= q[i][p * W + w + 0] ^ v.x;
            m[i][w + 1] |= q[i][p * W + w + 1] ^ v.y;
            m[i][w + 2] |= q[i][p * W + w + 2] ^ v.z;
            m[i][w + 3] |= q[i][p * W + w + 3] ^ v.w;
          }
        }
      }
    }
  } else if constexpr (W == 2) {
    const uint2* c2 = reinterpret_cast<const uint2*>(col);
#pragma unroll
    for (int p = 0; p < P; ++p) {
      const uint2 v = c2[p];
#pragma unroll
      for (int i = 0; i < TM; ++i) {
        if (p == 0) {
          m[i][0] = q[i][0] ^ v.x;
          m[i][1] = q[i][1] ^ v.y;
        } else {
          m[i][0] |= q[i][p * 2 + 0] ^ v.x;
          m[i][1] |= q[i][p * 2 + 1] ^ v.y;
        }
      }
    }
  } else {
#pragma unroll
    for (int p = 0; p < P; ++p) {
#pragma unroll
      for (int w = 0; w < W; ++w) {
        const uint32_t v = col[p * W + w];
#pragma unroll
        for (int i = 0; i < TM; ++i) {
          if (p == 0) m[i][w] = q[i][w] ^ v;
          else m[i][w] |= q[i][p * W + w] ^ v;
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    unsigned s = __popc(m[i][0]);
#pragma unroll
    for (int w = 1; w < W; ++w) s = mad_u32(__popc(m[i][w]), one, s);
    d[i] = static_cast<int>(s);
  }
}

// Distances of TM own rows to FOUR consecutive stream rows (col: the first of them, 16-byte aligned:
// every tile starts aligned and the callers step in groups of four).  Rows of a multiple of four
// words are read with 128-bit loads by ham_rows already.  Narrow rows (W = 1, 2: 20 / 40 bytes at five
// planes) are not 16-byte multiples on their own, so one row at a time means 32- or 64-bit loads --
// five shared-memory instructions per pair, and the shared-memory pipe takes one per clock and SM:
// the W = 1 sweep ran at 27 clocks per pair-warp on 20 clocks of LDS.  Four rows together ARE a
// multiple of 16 bytes: P*W 128-bit loads per four pairs.
template <int P, int W, int TM>
__device__ __forceinline__ void ham_rows4(const uint32_t (&q)[TM][P * W], const uint32_t* __restrict__ col,
                                          int (&d0)[TM], int (&d1)[TM], int (&d2)[TM], int (&d3)[TM], unsigned one) {
  constexpr int COLW = P * W;
  if constexpr (W % 4 == 0) {
    ham_rows<P, W, TM>(q, col + 0 * COLW, d0, one);
    ham_rows<P, W, TM>(q, col + 1 * COLW, d1, one);
    ham_rows<P, W, TM>(q, col + 2 * COLW, d2, one);
    ham_rows<P, W, TM>(q, col + 3 * COLW, d3, one);
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
#pragma unroll
      for (int i = 0; i < TM; ++i) {
        uint32_t m[W];
#pragma unroll
        for (int w = 0; w < W; ++w) {
          m[w] = q[i][w] ^ v[r * COLW + w];
#pragma unroll
          for (int p = 1; p < P; ++p) m[w] |= q[i][p * W + w] ^ v[r * COLW + p * W + w];
        }
        unsigned s = __popc(m[0]);
#pragma unroll
        for (int w = 1; w < W; ++w) s = mad_u32(__popc(m[w]), one, s);
        const int dd = static_cast<int>(s);
        if (r == 0) d0[i] = dd;
        else if (r == 1) d1[i] = dd;
        else if (r == 2) d2[i] = dd;
        else d3[i] = dd;
      }
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

template <int P, int W, int TM, int MODE, bool LUT, int WEIGHT, int MINB = 2>
__global__ void __launch_bounds__(kSweepThreads, MINB) sweep_kernel(const __grid_constant__ SweepParams prm) {
  constexpr int BN = TileCols<W>::value;
  constexpr int COLW = P * W;
  constexpr uint32_t STAGE_BYTES = BN * COLW * 4;
  constexpr int ROWS_CTA = kConsumers * TM;
  static_assert(STAGE_BYTES % 16 == 0, "bulk copies move multiples of 16 bytes");

  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint32_t* stage_mem = reinterpret_cast<uint32_t*>(smem_raw);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + kStages * STAGE_BYTES);
  unsigned* done = reinterpret_cast<unsigned*>(full + kStages);   // warps finished with a stage
  uint32_t* lut_s = reinterpret_cast<uint32_t*>(full + 2 * kStages);
  unsigned long long* lists = reinterpret_cast<unsigned long long*>(lut_s + kMaxLutWords);  // [ROWS_CTA][k1]

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int lane = tid & 31;

  // lookahead cursor: the tile that goes into a stage when its current tile has been consumed
  SweepCursor la;
  la.start(blockIdx.x, prm);
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full[s], 1);
      done[s] = 0;
    }
    fence_mbar_init();
  }
  if (LUT && tid < kMaxLutWords) lut_s[tid] = prm.lut[tid];
  __syncthreads();
#pragma unroll 1
  for (int s = 0; s < kStages; ++s) {   // prologue: fill the ring
    if (tid == 0 && la.valid(prm)) {
      mbar_arrive_expect_tx(&full[s], STAGE_BYTES);
      bulk_g2s(stage_mem + s * (BN * COLW), prm.str + static_cast<size_t>(la.t) * BN * COLW, STAGE_BYTES, &full[s]);
    }
    if (la.valid(prm)) la.advance(prm, gridDim.x);
  }

  const int n_items = prm.n_rowblocks * prm.n_splits;
  int stage = 0;
  uint32_t phase = 0;

  for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int split = item / prm.n_rowblocks;
    const int rb = item - split * prm.n_rowblocks;
    long long r[TM];      // own rows relative to own_row0; lanes hold consecutive rows
    bool valid[TM];
    uint32_t q[TM][COLW];
    unsigned tau[TM];     // kNN: distance word of the k1-th list entry (the filter threshold)
    long long cnt[TM];    // count / fill cursor
    unsigned long long* cap[TM];
#pragma unroll
    for (int i = 0; i < TM; ++i) {
      cap[i] = nullptr;
      r[i] = static_cast<long long>(rb) * ROWS_CTA + i * kConsumers + tid;
      valid[i] = r[i] < prm.rows;
      if (prm.row_map != nullptr && valid[i]) r[i] = prm.row_map[r[i]];
      const uint32_t* src = prm.own + static_cast<size_t>(prm.own_row0 + (valid[i] ? r[i] : 0)) * COLW;
#pragma unroll
      for (int j = 0; j < COLW; ++j) q[i][j] = valid[i] ? __ldg(src + j) : 0u;
      tau[i] = valid[i] ? 0xffffffffu : 0u;
      cnt[i] = 0;
      if constexpr (MODE == MODE_KNN) {
        unsigned long long* mine = lists + static_cast<size_t>(i * kConsumers + tid) * prm.k1;
        for (int j = 0; j < prm.k1; ++j) mine[j] = ~0ull;
      }
      if constexpr (MODE == MODE_COUNT) {
        if (valid[i] && prm.capture != nullptr)
          cap[i] = prm.capture + (static_cast<size_t>(split) * prm.rows_total + r[i]) * prm.capture_cap;
      }
      if constexpr (MODE == MODE_FILL) {
        if (valid[i]) {
          cnt[i] = prm.indptr[r[i]];
          for (int s = 0; s < split; ++s) cnt[i] += prm.split_counts[static_cast<size_t>(s) * prm.rows_total + r[i]];
        }
      }
    }
    const int lo = prm.lo;
    const unsigned span = prm.span;
    const unsigned one = prm.one;
    if constexpr (MODE == MODE_KNN) __syncwarp();

    const int t0 = split * prm.tiles_per_split;
    const int t1 = min(t0 + prm.tiles_per_split, prm.n_tiles);
    for (int t = t0; t < t1; ++t) {
      mbar_wait(&full[stage], phase);
      const uint32_t* tile = stage_mem + stage * (BN * COLW);
      const long long col0 = static_cast<long long>(t) * BN;
      const int ncols = static_cast<int>(min(static_cast<long long>(BN), prm.str_rows - col0));
      // serve the kNN candidates of one stream row: rare, so a ballot first, then the warp
      // inserts them one by one (warp-uniform control flow)
      auto serve = [&](int i, int dv, long long col) {
        unsigned cand = __ballot_sync(0xffffffffu, static_cast<unsigned>(dv) < tau[i]);
        while (cand) {
          const int src = __ffs(cand) - 1;
          cand &= cand - 1;
          const unsigned dd = __shfl_sync(0xffffffffu, static_cast<unsigned>(dv), src);
          const unsigned long long key = (static_cast<unsigned long long>(dd) << 32) | static_cast<unsigned>(col);
          unsigned long long* lst = lists + static_cast<size_t>(i * kConsumers + (warp << 5) + src) * prm.k1;
          const unsigned t_new = knn_insert_coop(lst, prm.k1, key, lane);
          if (lane == src) tau[i] = t_new;
        }
      };
      int c = 0;
      if constexpr (MODE == MODE_KNN) {
        // four stream rows per vote: one min + one compare + one vote per group keeps the
        // per-pair overhead on the ALU pipe near zero
#pragma unroll 1
        for (; c + 4 <= ncols; c += 4) {
          int d0[TM], d1[TM], d2[TM], d3[TM];
          ham_rows4<P, W, TM>(q, tile + c * COLW, d0, d1, d2, d3, one);
#pragma unroll
          for (int i = 0; i < TM; ++i) {
            const unsigned best = min(min(static_cast<unsigned>(d0[i]), static_cast<unsigned>(d1[i])),
                                      min(static_cast<unsigned>(d2[i]), static_cast<unsigned>(d3[i])));
            if (__any_sync(0xffffffffu, best < tau[i])) {
              serve(i, d0[i], col0 + c + 0);
              serve(i, d1[i], col0 + c + 1);
              serve(i, d2[i], col0 + c + 2);
              serve(i, d3[i], col0 + c + 3);
            }
          }
        }
      }
      // what a mode does with the distances of one stream row
      auto consume = [&](int c, const int (&d)[TM]) {
#pragma unroll
        for (int i = 0; i < TM; ++i) {
          if constexpr (MODE == MODE_KNN) {
            serve(i, d[i], col0 + c);
          } else if constexpr (MODE == MODE_COUNT) {
            bool hit;
            if constexpr (LUT) hit = (lut_s[d[i] >> 5] >> (d[i] & 31)) & 1u;
            else hit = static_cast<unsigned>(d[i] - lo) <= span;
            if (hit && valid[i]) {
              // sparse graphs: keep the first hits so that the fill sweep can be skipped
              if (cap[i] != nullptr && cnt[i] < prm.capture_cap)
                cap[i][cnt[i]] = (static_cast<unsigned long long>(static_cast<unsigned>(d[i])) << 32) |
                                 static_cast<unsigned>(col0 + c);
              ++cnt[i];
            }
          } else if constexpr (MODE == MODE_FILL) {
            bool hit;
            if constexpr (LUT) hit = (lut_s[d[i] >> 5] >> (d[i] & 31)) & 1u;
            else hit = static_cast<unsigned>(d[i] - lo) <= span;
            if (hit && valid[i]) {
              prm.out_idx[cnt[i]] = col0 + c;
              write_weight(prm.out_w, cnt[i], d[i], WEIGHT);
              ++cnt[i];
            }
          } else {  // MODE_TILE: out[stream * ld + own]
            if (valid[i]) write_tile<WEIGHT>(prm.out, (col0 + c) * prm.ld + r[i], d[i], lo, span);
          }
        }
      };
      if constexpr (MODE != MODE_KNN && W % 4 != 0) {
        // narrow rows: four stream rows per group of 128-bit loads (see ham_rows4)
#pragma unroll 1
        for (; c + 4 <= ncols; c += 4) {
          int d0[TM], d1[TM], d2[TM], d3[TM];
          ham_rows4<P, W, TM>(q, tile + c * COLW, d0, d1, d2, d3, one);
          consume(c + 0, d0);
          consume(c + 1, d1);
          consume(c + 2, d2);
          consume(c + 3, d3);
        }
      }
#pragma unroll 2
      for (; c < ncols; ++c) {
        int d[TM];
        ham_rows<P, W, TM>(q, tile + c * COLW, d, one);
        consume(c, d);
      }
      // done with this stage: the last warp to get here refills it with the lookahead tile
      __syncwarp();
      if (lane == 0) {
        if (atom_add_acq_rel_cta(&done[stage], 1u) == kConsumerWarps - 1) {
          done[stage] = 0;
          if (la.valid(prm)) {
            fence_proxy_async();
            mbar_arrive_expect_tx(&full[stage], STAGE_BYTES);
            bulk_g2s(stage_mem + stage * (BN * COLW), prm.str + static_cast<size_t>(la.t) * BN * COLW,
                     STAGE_BYTES, &full[stage]);
          }
        }
      }
      if (la.valid(prm)) la.advance(prm, gridDim.x);
      if (++stage == kStages) { stage = 0; phase ^= 1u; }
    }

#pragma unroll
    for (int i = 0; i < TM; ++i) {
      if constexpr (MODE == MODE_KNN) {
        if (valid[i]) {
          const unsigned long long* mine = lists + static_cast<size_t>(i * kConsumers + tid) * prm.k1;
          unsigned long long* dst = prm.part + static_cast<size_t>(split) * prm.k1 * prm.rows_total + r[i];
          for (int j = 0; j < prm.k1; ++j) dst[static_cast<size_t>(j) * prm.rows_total] = mine[j];
        }
      } else if constexpr (MODE == MODE_COUNT) {
        if (valid[i]) prm.split_counts[static_cast<size_t>(split) * prm.rows_total + r[i]] = cnt[i];
      }
    }
    if constexpr (MODE == MODE_KNN) __syncwarp();
  }
}

}  // namespace pg

// ---- host-side launcher, one translation unit per (P, W) ------------------------
namespace pg {

struct SweepLaunch {
  int mode;    // SweepMode
  int lut;     // 0 range test, 1 LUT
  int weight;  // pgWeight (tile: compile time; fill: runtime)
  int grid;    // 0 = let the launcher size a persistent grid
  size_t list_bytes;  // kNN lists (all own rows of a CTA)
  cudaStream_t stream;
  int rows_per_thread = 1;  // 2 selects the two-rows-per-thread kNN instantiation (experiments)
  // chunked long-row sweep: the truth table (count / fill with lut = 1) has lut_words words, in
  // SweepParams::lut when they fit, else in device memory at lut_ext
  int lut_words = kMaxLutWords;
  const uint32_t* lut_ext = nullptr;
};

template <int P, int W>
inline size_t sweep_smem_bytes(size_t list_bytes) {
  return static_cast<size_t>(kStages) * TileCols<W>::value * P * W * 4 + 2 * kStages * sizeof(uint64_t) +
         kMaxLutWords * 4 + list_bytes;   // ring + barriers/counters + lut + kNN lists
}

template <int P, int W, int TM, int MODE, bool LUT, int WEIGHT, int MINB = 2>
int launch_one(const SweepParams& prm, const SweepLaunch& l) {
  auto kern = sweep_kernel<P, W, TM, MODE, LUT, WEIGHT, MINB>;
  const size_t smem = sweep_smem_bytes<P, W>(l.list_bytes);
  PG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  int occ = 0;
  PG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kSweepThreads, smem));
  if (occ < 1) { set_error("sweep kernel does not fit on an SM (smem %zu bytes)", smem); return PG_ERR_UNSUPPORTED; }
  const long long n_items = static_cast<long long>(prm.n_rowblocks) * prm.n_splits;
  long long grid = l.grid > 0 ? l.grid : static_cast<long long>(num_sms()) * occ;
  if (grid > n_items) grid = n_items;
  if (grid < 1) grid = 1;
  kern<<<static_cast<unsigned>(grid), kSweepThreads, smem, l.stream>>>(prm);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

template <int P, int W>
int launch_sweep(const SweepParams& prm, const SweepLaunch& l) {
  switch (l.mode) {
    case MODE_KNN:
      if constexpr (P == 5 && W == 8) {
        if (l.rows_per_thread == 2) return launch_one<P, W, 2, MODE_KNN, false, 0, 2>(prm, l);
        if (l.rows_per_thread == 3) return launch_one<P, W, 1, MODE_KNN, false, 0, 3>(prm, l);   // 3 CTAs / SM
        if (l.rows_per_thread == 4) return launch_one<P, W, 2, MODE_KNN, false, 0, 1>(prm, l);   // 1 CTA / SM
      }
      return launch_one<P, W, 1, MODE_KNN, false, 0>(prm, l);
    case MODE_COUNT:
      return l.lut ? launch_one<P, W, 1, MODE_COUNT, true, 0>(prm, l) : launch_one<P, W, 1, MODE_COUNT, false, 0>(prm, l);
    case MODE_FILL:
      if (l.weight == PG_W_SIM_F32)
        return l.lut ? launch_one<P, W, 1, MODE_FILL, true, PG_W_SIM_F32>(prm, l)
                     : launch_one<P, W, 1, MODE_FILL, false, PG_W_SIM_F32>(prm, l);
      return l.lut ? launch_one<P, W, 1, MODE_FILL, true, PG_W_I64>(prm, l)
                   : launch_one<P, W, 1, MODE_FILL, false, PG_W_I64>(prm, l);
    case MODE_TILE:
      if (l.weight == PG_W_I64) return launch_one<P, W, 1, MODE_TILE, false, PG_W_I64>(prm, l);
      if (l.weight == PG_W_SIM_F32) return launch_one<P, W, 1, MODE_TILE, false, PG_W_SIM_F32>(prm, l);
      if (l.weight == PG_W_FLAG_U8) return launch_one<P, W, 1, MODE_TILE, false, PG_W_FLAG_U8>(prm, l);
      return launch_one<P, W, 1, MODE_TILE, false, PG_W_I32>(prm, l);
  }
  set_error("bad sweep mode %d", l.mode);
  return PG_ERR_INVALID;
}

// defined in pg_sweep_inst.cu, one per (P, W)
#define PG_DECL_SWEEP(P, W) int sweep_p##P##_w##W(const SweepParams& prm, const SweepLaunch& l);
PG_DECL_SWEEP(5, 1) PG_DECL_SWEEP(5, 2) PG_DECL_SWEEP(5, 4) PG_DECL_SWEEP(5, 8) PG_DECL_SWEEP(5, 16)
PG_DECL_SWEEP(8, 1) PG_DECL_SWEEP(8, 2) PG_DECL_SWEEP(8, 4) PG_DECL_SWEEP(8, 8)
#undef PG_DECL_SWEEP

}  // namespace pg
