// Symmetric fused Hamming kNN sweep for sm_100a: every unordered pair {i, j} of one table is
// evaluated once and feeds the neighbour lists of BOTH rows.
//
// Replaces the same reference code as pg_sweep.cuh (hamming.py:34 + sort/slice of
// prograph.py:757-762) for the case build_graph actually runs -- a table against itself --
// where d(i,j) == d(j,i) makes half of the reference's N x N evaluations redundant.
//
// Mapping.  Row block rb (256 rows, one per thread, plane words in registers) sweeps the
// stream tiles from its own diagonal to the end of the table:
//   * stream rows of blocks  < rb : skipped (block pair handled by the lower block);
//   * stream rows of block  == rb : "row side" only -- both (i,j) and (j,i) are seen here;
//   * stream rows of blocks  > rb : row side for i (key (d,j) into the thread's list in shared
//     memory) AND column side for j (key (d,i) into row j's list in global memory).
// Every row has ONE global list of k1 sorted keys d<<32|index behind a per-row spin lock, plus a
// 64-bit filter word glast[j] = (~distance)<<32 | index of its k1-th key that travels to shared
// memory with the stream tile (a second bulk copy on the same mbarrier).  The hot loop tests four stream
// rows at a time against both thresholds with eight IMADs (FMA pipe) and four LOP3s, one vote;
// everything behind the vote is rare and out of line.  A stale filter word is only ever larger
// than the current one, so no candidate is lost; the locked insertion compares full keys, so the
// result is the k1 smallest (distance, index) keys whatever the arrival order.
// Work items are (row block, tile range) chunks from a host-built table (one list per CTA, ordered
// by L2-sized column bands, see sym_plan in pg_sweep.cu); a chunk starts its
// shared-memory lists empty but seeds its filter from the row's global list, and merges its lists
// into the global ones when it ends, so chunks can be short (good load balance) without the
// cold-start insertion storm of the split lists in pg_sweep.cuh.
// Bootstrap: the host first sweeps all rows one-sided against the first boot_rows columns
// (pg_hamming_knn_boot) so that every filter is tight from the first symmetric tile on; the row
// blocks of those rows ("boot" items) then run row side only, behind the bootstrap columns.
// Lock protocol: atom.acquire.gpu CAS by lane 0, __syncwarp, list edited in registers, st.cg of the
// list and the filter word, __syncwarp, st.release.gpu of the lock by lane 0 (bar.warp.sync orders the
// other lanes' stores before the cumulative release).  A lock that cannot be taken within 2^24
// attempts raises the error word the host reads back (PG_ERR_CUDA) instead of trapping the context.
// The filter words are a monotone hint: they are read through the async proxy (bulk copy) while
// other CTAs store to them; ANY value a row's word ever held is a valid (looser) filter, and an
// aligned 8-byte store cannot tear, so the hint needs no ordering.
// Epsilon mode (SYM_EPS) is the same sweep with another consumer (prograph.py:731-753): a pair whose
// distance lies in [lo, hi] appends both directed edges as packed 64-bit keys to a global buffer,
// which the host sorts into the CSR (pg_edge_keys_to_csr) -- no count pass, no second sweep.
#pragma once
#include "pg_sweep.cuh"

namespace pg {

constexpr int kTauInf = 0x3fffffff;   // filter value of a list that is not full yet

struct SymItem { int rb, t0, t1, boot; };   // row block, stream tiles [t0, t1); boot: block of the bootstrap rows

struct SymParams {
  const uint32_t* tab;        // packed table, own == stream
  long long rows;             // valid rows
  const SymItem* items;       // CTA-major: CTA b owns items [cta_first[b], cta_first[b+1])
  const int* cta_first;
  int n_items;
  unsigned one;               // opaque 1 (see SweepParams::one)
  int k1;                     // list length, <= 32
  unsigned long long* glist;  // [rows][k1] ascending keys, ~0 = empty
  unsigned long long* glast;  // [n_tiles * tile_cols] filter word per row: (~tau)<<32 | index of the last key
  unsigned* glock;            // [rows]
  unsigned long long* stats;  // null, or [8] slow-path counters: -, locks, lock spins, list writes, row inserts
  unsigned* error;            // set to 1 when a row lock could not be taken (the host turns it into PG_ERR_CUDA)
  long long boot_rows;        // rows [0, boot_rows) were swept one-sided against every row beforehand
  // epsilon mode (SYM_EPS): edge <=> lo <= d <= hi; edges are appended to `keys` as
  // row << sh_row | column << sh_col | d, both directions of every unordered pair
  int lo, hi;
  int sh_row, sh_col;
  unsigned long long* keys;
  long long capacity;            // slots in `keys`
  unsigned long long* counters;  // [0] slots reserved (multiples of kEdgeChunk), [1] edges written or dropped
};

__device__ __forceinline__ unsigned long long ld_cg_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.global.cg.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_cg_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.global.cg.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned atom_cas_acquire_gpu(unsigned* p, unsigned cmp, unsigned val) {
  unsigned old;
  asm volatile("atom.acquire.gpu.global.cas.b32 %0, [%1], %2, %3;" : "=r"(old) : "l"(p), "r"(cmp), "r"(val) : "memory");
  return old;
}
__device__ __forceinline__ void st_release_gpu_u32(unsigned* p, unsigned v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
constexpr unsigned kLockSpinLimit = 1u << 24;
// filter word of a list whose last key is `last` (~0 = list not full)
__host__ __device__ __forceinline__ unsigned long long sym_filter_word(unsigned long long last) {
  const unsigned tau = (last == ~0ull) ? static_cast<unsigned>(kTauInf) : static_cast<unsigned>(last >> 32);
  return (static_cast<unsigned long long>(~tau) << 32) | (last & 0xffffffffull);
}
__device__ __forceinline__ int mad_s32(int a, unsigned b, int c) {
  int r;
  asm("mad.lo.s32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}

// Warp-cooperative merge of up to 32 candidate keys (one per lane, `is_cand`) into the global
// list of row j.  All lanes call it with the same j.  The list is edited in registers under the
// row's lock; keys that no longer beat the current last key simply do not get in.
static __device__ __noinline__ void sym_serve_col(const SymParams& prm, long long j, unsigned long long key, bool is_cand,
                                           int lane) {
  const int k1 = prm.k1;
  unsigned long long* lst = prm.glist + static_cast<size_t>(j) * k1;
  // the caller's filter (a snapshot at most a few tiles old) already passed: take the lock
  // right away, the merge below re-checks every key against the current list
  unsigned cand = __ballot_sync(0xffffffffu, is_cand);
  if (cand == 0u) return;
  unsigned* lock = prm.glock + j;
  unsigned got = 1u;
  if (lane == 0) {
    unsigned spins = 0;
    while (atom_cas_acquire_gpu(lock, 0u, 1u) != 0u) {
      __nanosleep(100);
      if (++spins > kLockSpinLimit) {     // a protocol bug is reported to the host, the context survives
        got = 0u;
        atomicExch(prm.error, 1u);
        break;
      }
    }
    if (prm.stats != nullptr) {
      atomicAdd(prm.stats + 1, 1ull);
      if (spins) atomicAdd(prm.stats + 2, static_cast<unsigned long long>(spins));
    }
  }
  // bar.warp.sync orders lane 0's acquire before the other lanes' loads of the list
  if (__shfl_sync(0xffffffffu, got, 0) == 0u) return;
  __syncwarp();
  unsigned long long e = lane < k1 ? ld_cg_u64(lst + lane) : ~0ull;
  bool changed = false;
  while (cand) {
    const int src = __ffs(cand) - 1;
    cand &= cand - 1;
    const unsigned long long kk = __shfl_sync(0xffffffffu, key, src);
    const int pos = __popc(__ballot_sync(0xffffffffu, lane < k1 && e < kk));
    const unsigned long long up = __shfl_up_sync(0xffffffffu, e, 1);
    if (pos < k1) {
      if (lane == pos) e = kk;
      else if (lane > pos) e = up;
      changed = true;
    }
  }
  if (changed) {
    if (lane < k1) st_cg_u64(lst + lane, e);
    const unsigned long long last = __shfl_sync(0xffffffffu, e, k1 - 1);
    if (lane == 0) {
      st_cg_u64(prm.glast + j, sym_filter_word(last));
      if (prm.stats != nullptr) atomicAdd(prm.stats + 3, 1ull);
    }
  }
  __syncwarp();                                   // every lane's stores happen before lane 0's release
  if (lane == 0) st_release_gpu_u32(lock, 0u);
}

constexpr int kMaxSymList = 32;   // longest list the symmetric sweep keeps (k + drop)

// Row side: the warp inserts the candidates of one stream row (column `col`) into the
// shared-memory lists of its own rows; returns the lane's updated filter.
static __device__ __noinline__ int sym_serve_row(unsigned long long* warp_lists, int k1, unsigned cand, unsigned dv,
                                          unsigned col, int lane, int tau_seed, int tau,
                                          unsigned long long* stats) {
  if (stats != nullptr && lane == 0) atomicAdd(stats + 4, static_cast<unsigned long long>(__popc(cand)));
  while (cand) {
    const int src = __ffs(cand) - 1;
    cand &= cand - 1;
    const unsigned dd = __shfl_sync(0xffffffffu, dv, src);
    const unsigned long long key = (static_cast<unsigned long long>(dd) << 32) | col;
    const unsigned t_new = knn_insert_coop(warp_lists + static_cast<size_t>(src) * k1, k1, key, lane);
    if (lane == src) tau = min(tau_seed, t_new == 0xffffffffu ? kTauInf : static_cast<int>(t_new));
  }
  return tau;
}

// Position of a CTA in its own item list: the (item, ring tile) that goes into a stage next.
struct SymCursor {
  int idx, end, t, t1;
  __device__ __forceinline__ void start(int i, const SymParams& prm) {
    idx = i;
    if (idx < end) {
      const int4 it = __ldg(reinterpret_cast<const int4*>(prm.items) + idx);
      t = it.y;
      t1 = it.z;
    } else {
      t = t1 = 0;
    }
  }
  __device__ __forceinline__ bool valid() const { return idx < end; }
  __device__ __forceinline__ void advance(const SymParams& prm) {
    if (++t == t1) start(idx + 1, prm);
  }
};

enum SymMode { SYM_KNN = 0, SYM_EPS = 1 };

constexpr int kEdgeChunk = 512;   // edge slots a warp reserves at a time (one global atomic per chunk)

// Epsilon mode: the warp appends the edges of one stream row.  `hit` lanes emit key_fwd (own row ->
// stream row) and, outside the diagonal block, key_rev (stream row -> own row).  Slots come from
// warp-private chunks of the global key buffer; unused slots of a closed chunk hold the sentinel ~0.
// Past the buffer's capacity nothing is written, but the reservations keep counting so that the
// caller learns the size it needs.
static __device__ __noinline__ void sym_emit(const SymParams& prm, bool hit, unsigned long long key_fwd,
                                             unsigned long long key_rev, bool both, int lane, long long& ch_base,
                                             int& ch_used, unsigned long long& n_real) {
  const unsigned m = __ballot_sync(0xffffffffu, hit);
  if (m == 0u) return;
  const int mult = both ? 2 : 1;
  const int n = __popc(m) * mult;
  if (ch_base == -1 || ch_used + n > kEdgeChunk) {
    if (ch_base >= 0)
      for (int sl = ch_used + lane; sl < kEdgeChunk; sl += 32) prm.keys[ch_base + sl] = ~0ull;
    unsigned long long b = 0;
    if (lane == 0) b = atomicAdd(prm.counters, static_cast<unsigned long long>(kEdgeChunk));
    b = __shfl_sync(0xffffffffu, b, 0);
    ch_base = (static_cast<long long>(b) + kEdgeChunk <= prm.capacity) ? static_cast<long long>(b) : -2;
    ch_used = 0;
  }
  if (ch_base >= 0 && hit) {
    const int rank = __popc(m & ((1u << lane) - 1u));
    unsigned long long* at = prm.keys + ch_base + ch_used + rank * mult;
    at[0] = key_fwd;
    if (both) at[1] = key_rev;
  }
  ch_used += n;
  n_real += static_cast<unsigned long long>(n);
}

template <int P, int W, int MODE>
__global__ void __launch_bounds__(kSweepThreads, 2) sweep_sym_kernel(const __grid_constant__ SymParams prm) {
  constexpr int BN = TileCols<W>::value;
  constexpr int COLW = P * W;
  constexpr uint32_t STAGE_BYTES = BN * COLW * 4;
  constexpr uint32_t TAU_BYTES = MODE == SYM_KNN ? BN * 8 : 0;

  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint32_t* stage_mem = reinterpret_cast<uint32_t*>(smem_raw);
  unsigned long long* taus = reinterpret_cast<unsigned long long*>(smem_raw + kStages * STAGE_BYTES);   // [kStages][BN]
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + kStages * (STAGE_BYTES + TAU_BYTES));
  unsigned* done = reinterpret_cast<unsigned*>(full + kStages);
  unsigned long long* lists = reinterpret_cast<unsigned long long*>(full + 2 * kStages);   // [256][k1]

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int lane = tid & 31;
  const int k1 = prm.k1;
  unsigned long long* warp_lists = lists + static_cast<size_t>(warp << 5) * k1;

  const int item_first = __ldg(prm.cta_first + blockIdx.x), item_end = __ldg(prm.cta_first + blockIdx.x + 1);
  SymCursor la;
  la.end = item_end;
  la.start(item_first, prm);
  auto more = [&] { return la.valid(); };
  auto issue = [&](int s) {   // tile la.t (and its filter words) into ring stage s
    mbar_arrive_expect_tx(&full[s], STAGE_BYTES + TAU_BYTES);
    bulk_g2s(stage_mem + s * (BN * COLW), prm.tab + static_cast<size_t>(la.t) * BN * COLW, STAGE_BYTES, &full[s]);
    if constexpr (MODE == SYM_KNN) bulk_g2s(taus + s * BN, prm.glast + static_cast<size_t>(la.t) * BN, TAU_BYTES, &full[s]);
  };
  auto step = [&] { if (la.valid()) la.advance(prm); };
  ring_start(full, done, kStages, tid, [] {}, more, issue, step);

  int stage = 0;
  uint32_t phase = 0;
  const unsigned one = prm.one;
  // epsilon mode: the warp's current chunk of the edge buffer
  long long ch_base = -1;
  int ch_used = 0;
  unsigned long long n_real = 0;

  for (int ii = item_first; ii < item_end; ++ii) {
    const int4 it = __ldg(reinterpret_cast<const int4*>(prm.items) + ii);
    const int rb = it.x, t0 = it.y, t1 = it.z;
    const bool boot = it.w != 0;
    const long long r = static_cast<long long>(rb) * kConsumers + tid;
    const bool valid = r < prm.rows;
    uint32_t q[COLW];
    {
      const uint32_t* src = prm.tab + static_cast<size_t>(valid ? r : 0) * COLW;
#pragma unroll
      for (int j = 0; j < COLW; ++j) q[j] = valid ? __ldg(src + j) : 0u;
    }
    // kNN: the row's global list already bounds what can still matter: ties at its last distance
    // stay admissible (the index decides), hence the +1
    int tau_seed = 0, tau = 0;
    if constexpr (MODE == SYM_KNN) {
      if (valid) {
        const int g = ~static_cast<int>(ld_cg_u64(prm.glast + r) >> 32);
        tau_seed = g >= kTauInf ? kTauInf : g + 1;
      }
      tau = tau_seed;
      unsigned long long* mine = lists + static_cast<size_t>(tid) * k1;
      for (int j = 0; j < k1; ++j) mine[j] = ~0ull;
    }
    // invalid own rows never feed a column list; blocks of the bootstrap rows have no column side
    // (every list already holds its candidates among the bootstrap rows) and start behind them
    const unsigned vmask = (valid && !boot) ? 0xffffffffu : 0u;
    const long long diag_begin = boot ? prm.boot_rows : static_cast<long long>(rb) * kConsumers;
    const long long diag_end = boot ? (1ll << 40) : diag_begin + kConsumers;
    // epsilon mode: edge  <=>  lo <= d <= hi; an invalid own row gets an unreachable lower bound
    const int nlo = valid ? -prm.lo : -(1 << 28);
    const int hi = prm.hi;
    const unsigned mone = 0u - one;
    __syncwarp();

    for (int t = t0; t < t1; ++t) {
      mbar_wait(&full[stage], phase);
      const uint32_t* tile = stage_mem + stage * (BN * COLW);
      const unsigned long long* tnt = taus + stage * BN;
      const long long col0 = static_cast<long long>(t) * BN;
      const int ncols = static_cast<int>(min(static_cast<long long>(BN), prm.rows - col0));
      int c = static_cast<int>(min(static_cast<long long>(ncols), max(0ll, diag_begin - col0)));
      const int c_mid = static_cast<int>(min(static_cast<long long>(ncols), max(static_cast<long long>(c), diag_end - col0)));

      // one stream row behind the vote (rare): kNN serves both lists, epsilon appends the edges
      auto rare = [&](int dv, int cc_, bool col_on) {
        const unsigned col = static_cast<unsigned>(col0 + cc_);
        if constexpr (MODE == SYM_KNN) {
          const unsigned rc = __ballot_sync(0xffffffffu, dv < tau);
          if (rc) tau = sym_serve_row(warp_lists, k1, rc, static_cast<unsigned>(dv), col, lane, tau_seed, tau, prm.stats);
          if (col_on) {
            // exact test against the snapshot of row col's last key: ties are decided by the index
            const unsigned long long fw = tnt[cc_];
            const unsigned long long lastk = (static_cast<unsigned long long>(~static_cast<unsigned>(fw >> 32)) << 32) |
                                             (fw & 0xffffffffull);
            const unsigned long long mine = (static_cast<unsigned long long>(static_cast<unsigned>(dv)) << 32) |
                                            static_cast<unsigned>(r);
            const bool cc = vmask != 0u && mine < lastk;
            if (__any_sync(0xffffffffu, cc)) sym_serve_col(prm, col, mine, cc, lane);
          }
        } else {
          const bool hit = (dv + nlo) >= 0 && dv <= hi;
          const unsigned long long own = static_cast<unsigned long long>(r), oth = col;
          const unsigned long long dd = static_cast<unsigned long long>(static_cast<unsigned>(dv));
          sym_emit(prm, hit, (own << prm.sh_row) | (oth << prm.sh_col) | dd, (oth << prm.sh_row) | (own << prm.sh_col) | dd,
                   col_on, lane, ch_base, ch_used, n_real);
        }
      };

      // filter test + rare path of the four stream rows cg .. cg+3 with distances e0 .. e3
      auto vote = [&](int cg, int e0, int e1, int e2, int e3) {
        int any;
        if constexpr (MODE == SYM_KNN) {
          // filter words of the four stream rows: .y / .w = ~tau_j, .x / .z = index of the last key
          const int4 na = *reinterpret_cast<const int4*>(tnt + cg);
          const int4 nb = *reinterpret_cast<const int4*>(tnt + cg + 2);
          const unsigned cm = cg >= c_mid ? vmask : 0u;
          // sign bit set <=> candidate: d - tau < 0 (row side), d + ~tau_j < 0 i.e. d <= tau_j (column side)
          const int s0 = mad_s32(e0, one, -tau), s1 = mad_s32(e1, one, -tau);
          const int s2 = mad_s32(e2, one, -tau), s3 = mad_s32(e3, one, -tau);
          const int u0 = mad_s32(e0, one, na.y), u1 = mad_s32(e1, one, na.w);
          const int u2 = mad_s32(e2, one, nb.y), u3 = mad_s32(e3, one, nb.w);
          any = (s0 | s1 | s2) | s3 | static_cast<int>(static_cast<unsigned>((u0 | u1 | u2) | u3) & cm);
        } else {
          // sign bit set <=> no edge: d - lo < 0 or hi - d < 0; all four miss <=> the AND keeps the sign
          const int a0 = mad_s32(e0, one, nlo), a1 = mad_s32(e1, one, nlo);
          const int a2 = mad_s32(e2, one, nlo), a3 = mad_s32(e3, one, nlo);
          const int b0 = mad_s32(e0, mone, hi), b1 = mad_s32(e1, mone, hi);
          const int b2 = mad_s32(e2, mone, hi), b3 = mad_s32(e3, mone, hi);
          any = ~((a0 | b0) & (a1 | b1) & (a2 | b2) & (a3 | b3));
        }
        if (__any_sync(0xffffffffu, any < 0)) {
          const bool col_on = cg >= c_mid;
          rare(e0, cg + 0, col_on);
          rare(e1, cg + 1, col_on);
          rare(e2, cg + 2, col_on);
          rare(e3, cg + 3, col_on);
        }
      };

#pragma unroll 1
      for (; c + 4 <= ncols; c += 4) {
        int d[4];
        ham_rows4<P, W>(q, tile + c * COLW, d, one);
        vote(c, d[0], d[1], d[2], d[3]);
      }
#pragma unroll 1
      for (; c < ncols; ++c) {   // ragged end of the table (last tile only)
        rare(ham_rows<P, W>(q, tile + c * COLW, one), c, c >= c_mid);
      }

      ring_release(done, stage, phase, kStages, lane, more, issue, step);
    }

    if constexpr (MODE == SYM_KNN) {
      // merge the chunk's lists into the rows' global lists
      __syncwarp();
      const long long wrow0 = static_cast<long long>(rb) * kConsumers + (warp << 5);
#pragma unroll 1
      for (int src = 0; src < 32; ++src) {   // ascending keys, one row at a time
        if (wrow0 + src >= prm.rows) break;
        const unsigned long long lk = lane < k1 ? warp_lists[static_cast<size_t>(src) * k1 + lane] : ~0ull;
        sym_serve_col(prm, wrow0 + src, lk, lk != ~0ull, lane);
      }
      __syncwarp();
    }
  }
  if constexpr (MODE == SYM_EPS) {
    if (ch_base >= 0)
      for (int sl = ch_used + lane; sl < kEdgeChunk; sl += 32) prm.keys[ch_base + sl] = ~0ull;
    if (lane == 0 && n_real) atomicAdd(prm.counters + 1, n_real);
  }
}

struct SymLaunch {
  int grid;
  size_t list_bytes;
  cudaStream_t stream;
  int mode = SYM_KNN;
};

// grid == 0: only report the resident grid (CTAs) through *resident; otherwise grid is the CTA count
// of a plan made for at most that many CTAs, so launch_persistent launches all of them
template <int P, int W, int MODE>
int launch_sweep_sym_mode(const SymParams& prm, const SymLaunch& l, int* resident) {
  const size_t smem = static_cast<size_t>(kStages) * (TileCols<W>::value * P * W * 4 +
                                                      (MODE == SYM_KNN ? TileCols<W>::value * 8 : 0)) +
                      2 * kStages * sizeof(uint64_t) + l.list_bytes;
  return launch_persistent(sweep_sym_kernel<P, W, MODE>, smem, l.grid, l.stream, resident, prm);
}

template <int P, int W>
int launch_sweep_sym(const SymParams& prm, const SymLaunch& l, int* resident) {
  if (l.mode == SYM_EPS) return launch_sweep_sym_mode<P, W, SYM_EPS>(prm, l, resident);
  return launch_sweep_sym_mode<P, W, SYM_KNN>(prm, l, resident);
}

#define PG_DECL_SWEEP_SYM(P, W) int sweep_sym_p##P##_w##W(const SymParams& prm, const SymLaunch& l, int* resident);
PG_DECL_SWEEP_SYM(5, 1) PG_DECL_SWEEP_SYM(5, 2) PG_DECL_SWEEP_SYM(5, 4) PG_DECL_SWEEP_SYM(5, 8) PG_DECL_SWEEP_SYM(5, 16)
PG_DECL_SWEEP_SYM(8, 1) PG_DECL_SWEEP_SYM(8, 2) PG_DECL_SWEEP_SYM(8, 4) PG_DECL_SWEEP_SYM(8, 8)
#undef PG_DECL_SWEEP_SYM

}  // namespace pg
