// Minkowski p=2 on integer tokens as an int8 tensor-core contraction (tcgen05, sm_100a).
//
// For integer-valued rows the reference's  pow(sum(pow(X - Y, 2)), 1/2)  (minkowski.py:36)
// depends only on the exact integer  S = |x|^2 + |y|^2 - 2 x.y :
//   * int64 tokens  : d = sqrtf(float(S))                         (float32 result)
//   * fp16 staging  : d = fp16(sqrtf(fp16(S)))  (prograph.py:726; every term of the chain is an
//                     exactly representable integer, the fp32 sum is exact, see DESIGN.md)
// and x.y is a plain GEMM with K = L: the one metric on this path that really is a dense
// contraction.  It runs here as  tcgen05.mma.cta_group::1.kind::i8  (uint8 x uint8 -> int32,
// exact) with the accumulator in TMEM:
//   * operands are stored in HBM already in the K-major, no-swizzle core-matrix layout the
//     MMA reads from shared memory (8 rows x 16 bytes per core matrix), so tiles are moved
//     with 1-D bulk async copies (cp.async.bulk + mbarrier), no tensor map needed;
//   * one CTA = 256 query rows = TWO resident A tiles against the whole dataset streamed in
//     128-row B tiles through a ring; every B tile is multiplied with both A tiles (M=128, N=128,
//     K=32 per instruction), which halves the bytes streamed out of L2 per pair: with one A tile
//     the MMA issuer waited for B tiles 37 % of the time (every SM pulled 20 B/clk, 5.8 TB/s in
//     aggregate, profiles/r1_ncu_notes.md);
//   * four 128-column TMEM accumulators (all of TMEM): two per A tile, so the MMAs of tile t+1 run
//     while the epilogues of tile t drain;
//   * warp roles: 8 epilogue warps in two groups, group g owns A tile g (thread = TMEM lane =
//     query row, one sorted list per row), 1 producer lane, one MMA-issuing lane PER A TILE (a single
//     thread issuing all sixteen MMAs of a B tile was the bottleneck: with descriptors rebuilt per
//     instruction it needed ~130 clocks per MMA, the tensor pipe 64); the dataset norms ride along
//     with the B tiles into a small shared-memory ring;
//   * epilogues: materialised tile (minkowski.py:36-40) or fused kNN: a candidate test in
//     S-space against a per-row integer threshold (min + one vote per 32 columns), rare
//     warp-cooperative insertion into a sorted (value, index) list in shared memory; the
//     N x N matrix never reaches HBM;
//   * rows wider than GMAX_RESIDENT_K (CHUNKED): the A tiles no longer fit, so every ring stage
//     carries one GKC-wide K-chunk of A tile 0, A tile 1 and the B tile, and the issuers accumulate
//     the chunks of a B tile into the same TMEM accumulator; the epilogues are unchanged.
#include <cstdlib>

#include "pg_sweep.cuh"   // knn_insert_coop, kMaxListRounds

namespace pg {

constexpr int GM = 128;         // query rows per A tile (MMA M)
constexpr int GA = 2;           // A tiles per CTA: every B tile is multiplied with both
constexpr int GROWS = GM * GA;  // query rows per CTA
constexpr int GN = 128;         // dataset rows per B tile (MMA N)
constexpr int GSTAGES = 4;      // deepest B ring (fewer stages when the lists need the room)
constexpr int GTHREADS = 352;   // 8 epilogue warps (two groups) + producer warp + one MMA warp per A tile
constexpr int GPROD_WARP = 8;
constexpr int GMMA_WARP = 9;    // warps 9 and 10: the MMA issuers of A tile 0 and 1 (warp 9 owns the TMEM allocation)
constexpr int GPROD_LANES = 8;  // lanes of the producer warp that each copy a slice of a B tile
constexpr int GACC = 4;         // TMEM accumulators (4 x 128 columns = all 512): two per A tile
constexpr int GNORM_SLOTS = 8;  // ring of per-tile dataset norms (512 B each)
constexpr int PAD_NORM = 0x3fffffff;
constexpr int GMAX_RESIDENT_K = 256;   // widest row whose two A tiles stay resident next to the B ring
constexpr int GKC = 128;        // K-chunk of the chunked mode: a stage is 3 x 16 KB, so three stages fit next to
                                // the tile-store staging and two next to 42-entry lists (256 would leave one / ten)
// Widest row (K) of the GEMM.  With tokens <= 255, S <= 255^2 * 8192 = 532 684 800 < PAD_NORM / 2 =
// 536 870 911, the bound gemm_eps_common enforces on the S range, and a pad column's S = nq + PAD_NORM
// stays below 2^31, so every sum of the epilogues is exact in int32.  With the fp16 chain's tokens
// <= 31, S <= 961 * 8192 < 2^24: torch's fp32 accumulation of the fp16 squares is exact and the
// reference's value is still fp16(sqrt(fp16(S))).
constexpr int GMAX_K = 8192;

enum GemmValue { GV_F16 = 0, GV_F32 = 1 };     // which rounding chain turns S into the distance
enum GemmMode { GM_TILE = 0, GM_KNN = 1, GM_COUNT = 2, GM_FILL = 3 };

// ---- tcgen05 / TMEM PTX -----------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_holder, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_holder)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum), "r"(0u)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// issue only: the registers are valid after tmem_ld_wait()
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}

// K-major, no swizzle: core matrix = 8 rows x 16 B contiguous (128 B); LBO = distance between the
// two core matrices an MMA reads along K, SBO = distance between 8-row groups (cute/arch/
// mma_sm100_desc.hpp, canonical layout ((8,n),2):((1,SBO),LBO) in 16-byte units).
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3fff);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3fff) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3fff) << 32;
  d |= 1ull << 46;   // descriptor version for sm_100
  return d;          // layout_type (bits 61-63) = 0: SWIZZLE_NONE
}

// ---- S -> value -> ordered key -------------------------------------------------------------
template <int VK>
__device__ __forceinline__ uint32_t value_bits(int S, bool similarity) {
  const float s = static_cast<float>(S);
  if (VK == GV_F16) {
    const float sh = __half2float(__float2half_rn(s));
    __half d = __float2half_rn(sqrtf(sh));
    if (similarity) d = __float2half_rn(__fdiv_rn(1.0f, __half2float(__float2half_rn(1.0f + __half2float(d)))));
    return static_cast<uint32_t>(__half_as_ushort(d));
  } else {
    float d = sqrtf(s);
    if (similarity) d = __fdiv_rn(1.0f, 1.0f + d);
    return __float_as_uint(d);
  }
}
// values are non-negative: their bit patterns order like the values; similarities sort descending
__device__ __forceinline__ uint32_t order_key(uint32_t bits, bool similarity) { return similarity ? ~bits : bits; }

struct GemmParams {
  const uint8_t* A; const int* normA; long long M;       // queries (own rows)
  const uint8_t* B; const int* normB; long long N;       // dataset (stream rows)
  int K;                                                 // padded width, multiple of 32
  int stages;                                            // depth of the B ring (3 or 4)
  int debug;                                             // experiments (PG_GEMM_DEBUG): 1 = epilogues only hand the accumulator back
  int issuers;                                           // MMA-issuing warps: 1 (both A tiles) or 2 (one per A tile)
  int similarity;
  // tile
  void* out; long long ld;
  // kNN
  int k1, k, drop;
  long long* out_idx; void* out_val;
  // epsilon graph: keep iff s_lo <= S <= s_lo + s_span (the reference's edge test is monotone in S)
  int s_lo; unsigned s_span;
  long long* group_counts;      // [2][M] hits of every row in the first / second half of the dataset
  const long long* indptr;      // [M+1] (fill)
};

// Warp-cooperative sorted insertion of (key, S) into one row's list (see knn_insert_coop in
// pg_sweep.cuh); the exact integer sum S travels with its key so that the candidate threshold
// is simply the S of the last entry.  Precondition: key < list[k1-1].
__device__ __forceinline__ int knn_insert_coop_s(unsigned long long* list, int* slist, int k1,
                                                 unsigned long long key, int S, int lane) {
  unsigned long long cur[kMaxListRounds], prev[kMaxListRounds];
  int sprev[kMaxListRounds];
  int pos = 0;
#pragma unroll
  for (int r = 0; r < kMaxListRounds; ++r) {
    const int j = lane + 32 * r;
    const bool in = j < k1;
    cur[r] = in ? list[j] : ~0ull;
    prev[r] = (in && j > 0) ? list[j - 1] : 0ull;
    sprev[r] = (in && j > 0) ? slist[j - 1] : 0;
    pos += __popc(__ballot_sync(0xffffffffu, in && cur[r] < key));
  }
  __syncwarp();
#pragma unroll
  for (int r = 0; r < kMaxListRounds; ++r) {
    const int j = lane + 32 * r;
    if (j < k1 && j >= pos) {
      list[j] = (j == pos) ? key : prev[r];
      slist[j] = (j == pos) ? S : sprev[r];
    }
  }
  __syncwarp();
  return slist[k1 - 1];
}

// Rare path of the fused kNN, kept out of line so that the 32 call sites of a chunk stay small
// (inlined, the insertion blew the instruction cache: ~5700 clk per insert).
// `cand`: lanes whose row may have a candidate in this column (S below the S of the row's last
// list entry -- a superset of the true candidates because the key is monotone in S); the exact
// test is the lexicographic comparison of the full key with the last entry.
// Returns the lane's updated threshold (tprime = S_last - nq).
template <int VK>
__device__ __noinline__ int gemm_knn_serve(unsigned cand, int S, unsigned col, unsigned long long* warp_lists,
                                           int* warp_slists, int k1, bool sim, int lane, int nq, int tprime) {
  while (cand) {
    const int src = __ffs(cand) - 1;
    cand &= cand - 1;
    const int s_src = __shfl_sync(0xffffffffu, S, src);
    const uint32_t key32 = order_key(value_bits<VK>(s_src, sim), sim);
    const unsigned long long key = (static_cast<unsigned long long>(key32) << 32) | col;
    unsigned long long* lst = warp_lists + static_cast<size_t>(src) * k1;
    if (key < lst[k1 - 1]) {
      const int s_last = knn_insert_coop_s(lst, warp_slists + static_cast<size_t>(src) * k1, k1, key, s_src, lane);
      if (lane == src) tprime = s_last - nq;
    }
  }
  return tprime;
}

// Single-lane waits of the producer / MMA issuer: poll with a short sleep (try_wait with a
// suspend-time hint was measured to wake only at the time limit).
__device__ __forceinline__ void mbar_wait_poll(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(32);
    if (++spins > (1u << 26)) __trap();
  }
}
template <int VK, int MODE, int ISSUERS, bool CHUNKED>
__global__ void __launch_bounds__(GTHREADS, 1) mink_gemm_kernel(const __grid_constant__ GemmParams prm) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const int K = prm.K;
  const uint32_t tile_bytes = GM * K;                     // A and B tiles have the same shape
  uint8_t* sA = smem;                                     // [GA] tiles
  uint8_t* sB = smem + GA * tile_bytes;
  const int n_stages = prm.stages;
  // CHUNKED: the ring is [stages][A tile 0, A tile 1, B tile][GM rows x GKC] and nothing is resident
  constexpr uint32_t chunk_bytes = GM * GKC;
  int* sNorm = reinterpret_cast<int*>(smem + (CHUNKED ? 3 * chunk_bytes * n_stages : tile_bytes * (GA + n_stages)));   // [GNORM_SLOTS][GN]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sNorm + GNORM_SLOTS * GN);
  uint64_t* full = bars;                  // [GSTAGES] B tile (+ its norms) landed
  uint64_t* empty = bars + GSTAGES;       // [GSTAGES] MMAs reading the stage have completed
  uint64_t* acc_full = bars + 2 * GSTAGES;    // [GACC] accumulator ready for the epilogue
  uint64_t* acc_empty = acc_full + GACC;      // [GACC] epilogue has drained the accumulator
  uint64_t* a_full = acc_empty + GACC;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(a_full + 1);
  unsigned long long* lists = reinterpret_cast<unsigned long long*>(tmem_holder + 2);   // [GROWS][k1]
  int* slists = reinterpret_cast<int*>(lists + GROWS * prm.k1);                         // [GROWS][k1] exact sums
  // tile mode (no lists): per-warp 32 x 36-word transpose buffers, 16-byte aligned
  uint32_t* tile_stage = reinterpret_cast<uint32_t*>((reinterpret_cast<uintptr_t>(tmem_holder + 2) + 15) & ~uintptr_t(15));
  const bool tile_fast = MODE == GM_TILE && (reinterpret_cast<uintptr_t>(prm.out) & 15) == 0 &&
                         ((static_cast<size_t>(prm.ld) * (VK == GV_F16 ? 2 : 4)) & 15) == 0;

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int lane = tid & 31;
  const long long row0 = static_cast<long long>(blockIdx.x) * GROWS;
  // blockIdx.y splits the dataset (tile mode with few query rows): this CTA sweeps tiles
  // [t_begin, t_begin + n_tiles); `t` below counts tiles within that range
  const int all_tiles = static_cast<int>((prm.N + GN - 1) / GN);
  const int tiles_per_split = (all_tiles + static_cast<int>(gridDim.y) - 1) / static_cast<int>(gridDim.y);
  const int t_begin = static_cast<int>(blockIdx.y) * tiles_per_split;
  const int n_tiles = max(0, min(tiles_per_split, all_tiles - t_begin));
  const bool sim = prm.similarity != 0;

  if (tid == 0) {
    for (int s = 0; s < n_stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], ISSUERS); }   // one commit per issuer
    for (int a = 0; a < GACC; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], 4); }
    mbar_init(a_full, 1);
    fence_mbar_init();
  }
  if (warp == GMMA_WARP) tmem_alloc(tmem_holder, GACC * GN);  // all 512 columns: four int32 accumulators
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == GPROD_WARP) {
    // ---------------- producer ----------------
    // GPROD_LANES lanes each issue a slice of the tile so that several bulk requests are in flight
    // (measured neutral against one 32 KB request; the kernel is not copy-bound, see
    // profiles/r1_ncu_notes.md).
    if constexpr (CHUNKED) {
      // In the global table the K-chunk [c0, c0 + kc) of an 8-row group is kc * 8 contiguous bytes at
      // (row / 8) * 8K + c0 * 8, and in the ring it sits at SBO = GKC * 8 intervals (a narrower last
      // chunk leaves the end of each interval unused): lane g < 16 copies row group g of all three tiles.
      const int nchunks = (K + GKC - 1) / GKC;
      int stage = 0;
      uint32_t phase = 0;
      for (int t = 0; t < n_tiles; ++t) {
        for (int c = 0; c < nchunks; ++c) {
          const int c0 = c * GKC;
          const uint32_t piece = static_cast<uint32_t>(min(GKC, K - c0)) * 8u;
          if (lane == 0) {
            mbar_wait_poll(&empty[stage], phase ^ 1u);
            mbar_arrive_expect_tx(&full[stage], 3 * (GM / 8) * piece + (c == 0 ? GN * 4 : 0));
            // norms ride with the first chunk; slot reuse (tile t + 8) waits for a stage whose MMAs
            // (tile >= t + 6: at least two chunks per tile, at most four stages) follow the epilogues of tile t + 4
            if (c == 0)
              bulk_g2s(sNorm + (t % GNORM_SLOTS) * GN, prm.normB + static_cast<size_t>(t_begin + t) * GN, GN * 4,
                       &full[stage]);
          }
          __syncwarp();
          if (lane < GM / 8) {
            uint8_t* dst = smem + static_cast<size_t>(stage) * 3 * chunk_bytes + lane * (GKC * 8);
            const size_t off = static_cast<size_t>(lane) * 8 * K + static_cast<size_t>(c0) * 8;
            bulk_g2s(dst, prm.A + static_cast<size_t>(row0) * K + off, piece, &full[stage]);
            bulk_g2s(dst + chunk_bytes, prm.A + static_cast<size_t>(row0 + GM) * K + off, piece, &full[stage]);
            bulk_g2s(dst + 2 * chunk_bytes, prm.B + static_cast<size_t>(t_begin + t) * GN * K + off, piece, &full[stage]);
          }
          if (++stage == n_stages) { stage = 0; phase ^= 1u; }
        }
      }
    } else {
    if (lane == 0) {        // both A tiles: 256 consecutive rows of the core-matrix table (padded to GROWS)
      mbar_arrive_expect_tx(a_full, GA * tile_bytes);
      bulk_g2s(sA, prm.A + static_cast<size_t>(row0) * K, tile_bytes, a_full);
      bulk_g2s(sA + tile_bytes, prm.A + static_cast<size_t>(row0 + GM) * K, tile_bytes, a_full);
    }
    const uint32_t slice = tile_bytes / GPROD_LANES;
    int stage = 0;
    uint32_t phase = 0;
    for (int t = 0; t < n_tiles; ++t) {
      if (lane == 0) {
        mbar_wait_poll(&empty[stage], phase ^ 1u);
        mbar_arrive_expect_tx(&full[stage], tile_bytes + GN * 4);
        // the norms of tile t live in slot t % GNORM_SLOTS until both epilogues of tile t are done;
        // slot reuse (tile t + 8) is ordered behind the MMAs of tile t + 8 - stages >= t + 4, which
        // themselves wait for the epilogues of tile t + 2
        bulk_g2s(sNorm + (t % GNORM_SLOTS) * GN, prm.normB + static_cast<size_t>(t_begin + t) * GN,
                 GN * 4, &full[stage]);
      }
      __syncwarp();
      if (lane < GPROD_LANES) {
        bulk_g2s(sB + static_cast<size_t>(stage) * tile_bytes + lane * slice,
                 prm.B + static_cast<size_t>(t_begin + t) * GN * K + lane * slice, slice,
                 &full[stage]);
      }
      if (++stage == n_stages) { stage = 0; phase ^= 1u; }
    }
    }
  } else if (warp >= GMMA_WARP) {
    // ---------------- MMA issuers ----------------
    // issuers == 2: warp GMMA_WARP + a multiplies A tile a with every B tile (short lists / queries: the
    // MMA side alone reaches 71 % of the tensor peak instead of 58 %); issuers == 1: warp GMMA_WARP
    // issues for both A tiles (long lists: measured 346 ms against 401 ms for the 1 M x 1 M k=16 graph).
    const int a_first = warp - GMMA_WARP;
    if (lane == 0 && a_first < ISSUERS) {
      // instruction descriptor: D=S32, A=B=UINT8, K-major both, N=128, M=128
      const uint32_t idesc = (2u << 4) | (static_cast<uint32_t>(GN >> 3) << 17) | (static_cast<uint32_t>(GM >> 4) << 24);
      if constexpr (CHUNKED) {
        // The chunks of a B tile accumulate into one accumulator (the flag is 0 only for the first
        // k-step of the first chunk); every chunk frees its stage, the last one hands the accumulator
        // to the epilogue.  One descriptor per ring, advanced by 16 units per k-step, chunk_bytes per
        // operand and 3 * chunk_bytes per stage.
        constexpr uint32_t chunk_units = chunk_bytes >> 4;
        const uint64_t desc0 = umma_desc(smem_u32(smem), 128, GKC * 8);
        const int nchunks = (K + GKC - 1) / GKC;
        int stage = 0;
        uint32_t phase = 0;
        for (int t = 0; t < n_tiles; ++t) {
          for (int c = 0; c < nchunks; ++c) {
            const int ksteps = min(GKC, K - c * GKC) / 32;
            mbar_wait_poll(&full[stage], phase);
            const uint64_t sdesc = desc0 + static_cast<uint64_t>(stage) * 3 * chunk_units;
            const uint64_t bdesc = sdesc + 2 * chunk_units;
#pragma unroll
            for (int i = 0; i < (ISSUERS == 1 ? GA : 1); ++i) {
              const int a = ISSUERS == 1 ? i : a_first;
              const int acc = a + GA * (t & 1);
              if (c == 0) {
                mbar_wait_poll(&acc_empty[acc], ((t >> 1) & 1) ^ 1u);
                tc_fence_after();
              }
              const uint64_t adesc = sdesc + static_cast<uint64_t>(a) * chunk_units;
              const uint32_t d_addr = tmem_base + acc * GN;
#pragma unroll
              for (int j = 0; j < GKC / 32; ++j)
                if (j < ksteps) umma_i8(d_addr, adesc + 16u * j, bdesc + 16u * j, idesc, (c | j) != 0 ? 1u : 0u);
              if (c == nchunks - 1) umma_commit(&acc_full[acc]);
            }
            umma_commit(&empty[stage]);
            if (++stage == n_stages) { stage = 0; phase ^= 1u; }
          }
        }
      } else {
      const uint32_t sbo = static_cast<uint32_t>(K / 16) * 128u;
      mbar_wait_poll(a_full, 0);
      // Descriptors are built ONCE: a k-step advances the start address by 256 bytes (16 descriptor
      // units), a ring stage by tile_bytes.  Rebuilding them for every instruction (two 64-bit shift /
      // or chains) cost the issuing thread more clocks per MMA than the tensor pipe needs to execute one.
      const uint64_t adesc0 = umma_desc(smem_u32(sA), 128, sbo);
      const uint64_t bdesc0 = umma_desc(smem_u32(sB), 128, sbo);
      const uint32_t stage_units = tile_bytes >> 4;
      const int ksteps = K / 32;
      int stage = 0;
      uint32_t phase = 0;
      if constexpr (ISSUERS == 1) {
        const uint64_t adesc1 = adesc0 + stage_units;
        for (int t = 0; t < n_tiles; ++t) {
          mbar_wait_poll(&full[stage], phase);
          const uint64_t bdesc = bdesc0 + static_cast<uint64_t>(stage) * stage_units;
#pragma unroll
          for (int a = 0; a < GA; ++a) {
            const int acc = a + GA * (t & 1);               // A tile a alternates between accumulators a and a + 2
            mbar_wait_poll(&acc_empty[acc], ((t >> 1) & 1) ^ 1u);
            tc_fence_after();
            const uint64_t adesc = a == 0 ? adesc0 : adesc1;
            const uint32_t d_addr = tmem_base + acc * GN;
            umma_i8(d_addr, adesc, bdesc, idesc, 0u);
#pragma unroll 4
            for (int j = 1; j < ksteps; ++j) umma_i8(d_addr, adesc + 16u * j, bdesc + 16u * j, idesc, 1u);
            umma_commit(&acc_full[acc]);    // this A tile's accumulator is complete
          }
          umma_commit(&empty[stage]);       // the stage may be refilled once all MMAs reading it are done
          if (++stage == n_stages) { stage = 0; phase ^= 1u; }
        }
      } else {
        const uint64_t adesc = adesc0 + static_cast<uint64_t>(a_first) * stage_units;
        for (int t = 0; t < n_tiles; ++t) {
          const int acc = a_first + GA * (t & 1);
          mbar_wait_poll(&full[stage], phase);
          mbar_wait_poll(&acc_empty[acc], ((t >> 1) & 1) ^ 1u);
          tc_fence_after();
          const uint64_t bdesc = bdesc0 + static_cast<uint64_t>(stage) * stage_units;
          const uint32_t d_addr = tmem_base + acc * GN;
          umma_i8(d_addr, adesc, bdesc, idesc, 0u);
#pragma unroll 4
          for (int j = 1; j < ksteps; ++j) umma_i8(d_addr, adesc + 16u * j, bdesc + 16u * j, idesc, 1u);
          umma_commit(&acc_full[acc]);      // this A tile's accumulator is complete
          umma_commit(&empty[stage]);       // the stage may be refilled once BOTH issuers' MMAs have read it
          if (++stage == n_stages) { stage = 0; phase ^= 1u; }
        }
      }
      }
    }
  } else {
    // ---------------- epilogue: warp group g owns A tile g; thread = TMEM lane = query row ---------
    const int group = warp >> 2;                 // A tile of this group
    const int r_loc = tid & (GM - 1);            // query row within the A tile = TMEM lane
    const int qwarp = warp & 3;                  // TMEM lane quarter this warp may read
    const long long row = row0 + group * GM + r_loc;
    const bool valid = row < prm.M;
    const int nq = valid ? prm.normA[row] : 0;
    unsigned long long* my_list = lists + (static_cast<size_t>(group) * GM + r_loc) * prm.k1;
    int tprime = valid ? 0x7fffffff : static_cast<int>(0x80000000);   // candidate iff (nx - 2 dot) < tprime
    if (MODE == GM_KNN) {
      int* my_slist = slists + (static_cast<size_t>(group) * GM + r_loc) * prm.k1;
      for (int j = 0; j < prm.k1; ++j) { my_list[j] = ~0ull; my_slist[j] = 0x7fffffff; }
      __syncwarp();
    }
    long long ecur = 0;    // epsilon modes: hits counted / next edge slot of this (row, group)
    if (MODE == GM_FILL && valid) ecur = prm.indptr[row];
    const int eoff = nq - prm.s_lo;    // in range iff (unsigned)(v + eoff) <= s_span
    const uint32_t lane_base = static_cast<uint32_t>(qwarp * 32) << 16;
    for (int t = 0; t < n_tiles; ++t) {
      const int acc = group + GA * (t & 1);    // group g drains accumulators g and g + 2 in turn
      mbar_wait(&acc_full[acc], (t >> 1) & 1);
      tc_fence_after();
      if (prm.debug & 1) {                    // timing experiment: how fast is the MMA side on its own?
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[acc]);
        continue;
      }
      const long long col_tile = static_cast<long long>(t_begin + t) * GN;
      const int* nrm = sNorm + (t % GNORM_SLOTS) * GN;
      uint32_t dotbuf[2][32];
      tmem_ld32_issue(tmem_base + lane_base + acc * GN, dotbuf[0]);
#pragma unroll
      for (int c = 0; c < GN / 32; ++c) {
        uint32_t (&dot)[32] = dotbuf[c & 1];
        tmem_ld_wait();
        if (c + 1 < GN / 32) tmem_ld32_issue(tmem_base + lane_base + acc * GN + (c + 1) * 32, dotbuf[(c + 1) & 1]);
        const long long col0 = col_tile + c * 32;
        int v[32];   // nx - 2 dot  (S = nq + v)
        const int4* np = reinterpret_cast<const int4*>(nrm + c * 32);
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const int4 nx = np[g];
          v[4 * g + 0] = nx.x - 2 * static_cast<int>(dot[4 * g + 0]);
          v[4 * g + 1] = nx.y - 2 * static_cast<int>(dot[4 * g + 1]);
          v[4 * g + 2] = nx.z - 2 * static_cast<int>(dot[4 * g + 2]);
          v[4 * g + 3] = nx.w - 2 * static_cast<int>(dot[4 * g + 3]);
        }
        if (MODE == GM_TILE) {
          // Thread = query row holds 32 consecutive columns.  Storing them directly makes every
          // store instruction touch 32 rows (32 half-used sectors); instead the warp transposes the
          // 32 x 32 block through shared memory and writes whole 128-byte (fp16: 64-byte) row
          // segments, four (eight) rows per instruction.
          constexpr int WPR = VK == GV_F16 ? 16 : 32;          // 32-bit words per row segment
          constexpr int STRIDE = WPR + 4;                      // conflict-free for 16-byte accesses
          uint32_t* stg = tile_stage + static_cast<size_t>(warp) * 32 * 36;
          const bool fast = tile_fast && col0 + 32 <= prm.N;   // warp-uniform
          if (fast) {
            uint32_t* mine = stg + lane * STRIDE;
#pragma unroll
            for (int g = 0; g < WPR / 4; ++g) {
              uint32_t w[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                if (VK == GV_F16)
                  w[e] = value_bits<VK>(nq + v[8 * g + 2 * e], sim) | (value_bits<VK>(nq + v[8 * g + 2 * e + 1], sim) << 16);
                else
                  w[e] = value_bits<VK>(nq + v[4 * g + e], sim);
              }
              *reinterpret_cast<uint4*>(mine + 4 * g) = make_uint4(w[0], w[1], w[2], w[3]);
            }
            __syncwarp();
            constexpr int LPR = WPR / 4;                       // lanes per row segment
            constexpr int RPI = 32 / LPR;                      // rows per store instruction
            const long long wrow0 = row0 + group * GM + qwarp * 32;
#pragma unroll
            for (int it = 0; it < 32 / RPI; ++it) {
              const int rr = it * RPI + lane / LPR;
              const uint4 val = *reinterpret_cast<const uint4*>(stg + rr * STRIDE + 4 * (lane % LPR));
              if (wrow0 + rr < prm.M) {
                unsigned char* o = static_cast<unsigned char*>(prm.out) +
                                   (static_cast<size_t>(wrow0 + rr) * prm.ld + col0) * (VK == GV_F16 ? 2 : 4);
                reinterpret_cast<uint4*>(o)[lane % LPR] = val;
              }
            }
            __syncwarp();
          } else if (valid) {
            const size_t at = static_cast<size_t>(row) * prm.ld + col0;
            if (VK == GV_F16) {
              unsigned short* o = static_cast<unsigned short*>(prm.out) + at;
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (col0 + j < prm.N) o[j] = static_cast<unsigned short>(value_bits<VK>(nq + v[j], sim));
            } else {
              uint32_t* o = static_cast<uint32_t*>(prm.out) + at;
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (col0 + j < prm.N) o[j] = value_bits<VK>(nq + v[j], sim);
            }
          }
        } else if (MODE == GM_COUNT) {
          int c32 = 0;
#pragma unroll
          for (int j = 0; j < 32; ++j) c32 += (static_cast<unsigned>(v[j] + eoff) <= prm.s_span) ? 1 : 0;
          ecur += valid ? c32 : 0;
        } else if (MODE == GM_FILL) {
          if (valid) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              if (static_cast<unsigned>(v[j] + eoff) <= prm.s_span) {
                prm.out_idx[ecur] = col0 + j;
                const uint32_t bits = value_bits<VK>(nq + v[j], sim);
                if (VK == GV_F16) static_cast<unsigned short*>(prm.out_val)[ecur] = static_cast<unsigned short>(bits);
                else static_cast<uint32_t*>(prm.out_val)[ecur] = bits;
                ++ecur;
              }
            }
          }
        } else {
          // pad columns of the last B tile (index >= N) are never candidates: their S is huge but
          // finite, so with fewer than k1 dataset rows they would fill the empty list slots
          if (col0 + 32 > prm.N) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (col0 + j >= prm.N) v[j] = 0x7fffffff;
          }
          // tree minimum of the 32 values (a linear chain would serialise 31 dependent mins)
          int m8[8];
#pragma unroll
          for (int g = 0; g < 8; ++g) m8[g] = min(min(v[4 * g], v[4 * g + 1]), min(v[4 * g + 2], v[4 * g + 3]));
          const int best = min(min(min(m8[0], m8[1]), min(m8[2], m8[3])), min(min(m8[4], m8[5]), min(m8[6], m8[7])));
          if (__any_sync(0xffffffffu, best < tprime)) {
            unsigned long long* warp_lists = lists + (static_cast<size_t>(group) * GM + qwarp * 32) * prm.k1;
            int* warp_slists = slists + (static_cast<size_t>(group) * GM + qwarp * 32) * prm.k1;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const unsigned cand = __ballot_sync(0xffffffffu, v[j] < tprime);
              if (cand)
                tprime = gemm_knn_serve<VK>(cand, nq + v[j], static_cast<unsigned>(col0 + j), warp_lists, warp_slists,
                                            prm.k1, sim, lane, nq, tprime);
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[acc]);
    }
    if (MODE == GM_COUNT && valid) prm.group_counts[row] = ecur;      // second half of the scratch stays 0
    if (MODE == GM_KNN) {
      // every row has one list (ascending, keys unique): drop, widen, write out
      __syncwarp();
      if (valid) {
        for (int j = prm.drop; j < prm.drop + prm.k; ++j) {
          const unsigned long long key = j < prm.k1 ? my_list[j] : ~0ull;
          const size_t at = static_cast<size_t>(row) * prm.k + (j - prm.drop);
          if (key == ~0ull) {
            prm.out_idx[at] = -1;
            if (VK == GV_F16) static_cast<unsigned short*>(prm.out_val)[at] = 0;
            else static_cast<uint32_t*>(prm.out_val)[at] = 0;
          } else {
            uint32_t bits = static_cast<uint32_t>(key >> 32);
            if (sim) bits = ~bits;
            prm.out_idx[at] = static_cast<long long>(key & 0xffffffffull);
            if (VK == GV_F16) static_cast<unsigned short*>(prm.out_val)[at] = static_cast<unsigned short>(bits);
            else static_cast<uint32_t*>(prm.out_val)[at] = bits;
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == GMMA_WARP) tmem_dealloc(tmem_base, GACC * GN);
}

// ---- operand packing: tokens -> K-major core-matrix layout + squared norms -----------------
template <typename T>
__global__ void gemm_pack_kernel(const T* __restrict__ tokens, long long N, int L, long long ld, uint8_t* __restrict__ table,
                                 int* __restrict__ norms, long long rows_padded, int K, int max_token,
                                 int* __restrict__ flag) {
  // one thread per (row, 16-byte chunk)
  const int chunks = K / 16;
  const long long total = rows_padded * chunks;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long row = i / chunks;
    const int ch = static_cast<int>(i - row * chunks);
    uint32_t w[4] = {0, 0, 0, 0};
    int sq = 0;
    if (row < N) {
      for (int b = 0; b < 16; ++b) {
        const int l = ch * 16 + b;
        if (l < L) {
          const double val = static_cast<double>(tokens[static_cast<size_t>(row) * ld + l]);
          const int tok = static_cast<int>(val);
          if (val != static_cast<double>(tok) || tok < 0 || tok > max_token) { atomicExch(flag, 1); continue; }
          w[b >> 2] |= static_cast<uint32_t>(tok) << (8 * (b & 3));
          sq += tok * tok;
        }
      }
      if (sq) atomicAdd(norms + row, sq);
    } else if (ch == 0) {
      norms[row] = PAD_NORM;     // pad rows can never be candidates
    }
    uint4* dst = reinterpret_cast<uint4*>(table + ((row >> 3) * chunks + ch) * 128 + (row & 7) * 16);
    *dst = make_uint4(w[0], w[1], w[2], w[3]);
  }
}
template <>
__global__ void gemm_pack_kernel<__half>(const __half* __restrict__ tokens, long long N, int L, long long ld,
                                         uint8_t* __restrict__ table, int* __restrict__ norms, long long rows_padded,
                                         int K, int max_token, int* __restrict__ flag) {
  const int chunks = K / 16;
  const long long total = rows_padded * chunks;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long row = i / chunks;
    const int ch = static_cast<int>(i - row * chunks);
    uint32_t w[4] = {0, 0, 0, 0};
    int sq = 0;
    if (row < N) {
      for (int b = 0; b < 16; ++b) {
        const int l = ch * 16 + b;
        if (l < L) {
          const float val = __half2float(tokens[static_cast<size_t>(row) * ld + l]);
          const int tok = static_cast<int>(val);
          if (val != static_cast<float>(tok) || tok < 0 || tok > max_token) { atomicExch(flag, 1); continue; }
          w[b >> 2] |= static_cast<uint32_t>(tok) << (8 * (b & 3));
          sq += tok * tok;
        }
      }
      if (sq) atomicAdd(norms + row, sq);
    } else if (ch == 0) {
      norms[row] = PAD_NORM;
    }
    uint4* dst = reinterpret_cast<uint4*>(table + ((row >> 3) * chunks + ch) * 128 + (row & 7) * 16);
    *dst = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

static size_t gemm_smem_bytes(int K, int k1, int stages, bool tile_mode = false, bool chunked = false) {
  return (chunked ? static_cast<size_t>(3) * GM * GKC * stages : static_cast<size_t>(GM) * K * (GA + stages)) + GNORM_SLOTS * GN * 4 + (2 * GSTAGES + 2 * GACC + 1) * sizeof(uint64_t) +
         16 + static_cast<size_t>(GROWS) * k1 * 12 + (tile_mode ? 16 + 8 * 32 * 36 * 4 : 0);
}

template <int VK, int MODE, int ISSUERS, bool CHUNKED>
static int launch_gemm_issuers(GemmParams prm, cudaStream_t s);

// One MMA-issuing warp (both A tiles, 320 threads) or two (one per A tile, 352 threads).  Two issuers
// lift the MMA side from 58 % to 71 % of the tensor peak and win where the epilogue is light (k = 1
// queries: 1 M x 1 M in 207 ms instead of 227 ms); with long lists the extra warp costs more than it
// gives (k = 16: 346 ms with one issuer, 397-401 ms with two).  PG_GEMM_ISSUERS overrides.
template <int VK, int MODE>
static int launch_gemm(GemmParams prm, cudaStream_t s) {
  int issuers = (MODE == GM_KNN && prm.k1 <= 4) ? 2 : 1;
  if (const char* ev = std::getenv("PG_GEMM_ISSUERS")) issuers = std::atoi(ev) == 2 ? 2 : 1;
  if (prm.K > GMAX_RESIDENT_K)
    return issuers == 2 ? launch_gemm_issuers<VK, MODE, 2, true>(prm, s) : launch_gemm_issuers<VK, MODE, 1, true>(prm, s);
  return issuers == 2 ? launch_gemm_issuers<VK, MODE, 2, false>(prm, s) : launch_gemm_issuers<VK, MODE, 1, false>(prm, s);
}

template <int VK, int MODE, int ISSUERS, bool CHUNKED>
static int launch_gemm_issuers(GemmParams prm, cudaStream_t s) {
  auto kern = mink_gemm_kernel<VK, MODE, ISSUERS, CHUNKED>;
  if (const char* ev = std::getenv("PG_GEMM_DEBUG")) prm.debug = std::atoi(ev);
  prm.issuers = ISSUERS;
  // wide rows / long lists: give up ring stages (down to 2) before giving up the fused path
  size_t smem = 0;
  for (prm.stages = GSTAGES; prm.stages >= 2; --prm.stages) {
    smem = gemm_smem_bytes(prm.K, MODE == GM_KNN ? prm.k1 : 0, prm.stages, MODE == GM_TILE, CHUNKED);
    if (smem <= 227 * 1024) break;
  }
  if (smem > 227 * 1024) { set_error("minkowski GEMM: k or row width too large for shared memory (%zu bytes)", smem); return PG_ERR_UNSUPPORTED; }
  PG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const unsigned gx = static_cast<unsigned>(ceil_div(prm.M, GROWS));
  unsigned gy = 1;
  if (MODE == GM_TILE) {   // few query rows: split the dataset so that every SM gets a CTA or two
    const long long tiles = ceil_div(prm.N, GN);
    long long want = ceil_div(2 * static_cast<long long>(num_sms()), gx);
    if (want > tiles / 8) want = tiles / 8;
    if (want > 65535) want = 65535;
    gy = static_cast<unsigned>(want < 1 ? 1 : want);
  }
  kern<<<dim3(gx, gy), ISSUERS == 2 ? GTHREADS : GTHREADS - 32, smem, s>>>(prm);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

// ---- int8 tensor-pipe peak probe -------------------------------------------------------------
// Back-to-back  tcgen05.mma.cta_group::1.kind::i8  M=128, N=256, K=32  on operands that stay in shared
// memory (pseudo-random bytes), accumulating into the two halves of TMEM in turn; one batch of MMAs
// is always in flight behind the one being issued.  Nothing is loaded, expanded or read back, so the
// rate is an upper bound for ANY formulation of the path on the int8 tensor pipe -- in particular for
// the one-hot Hamming GEMM (2 * 21 * L int8 operations per pair, SURVEY.md 8d), which would in
// addition have to expand its operands and run an epilogue.
constexpr int PROBE_K = 256;
constexpr int PROBE_BATCH = 16;      // tiles (8 MMAs each) per commit

__global__ void __launch_bounds__(128, 1) i8_mma_peak_kernel(int batches) {
  extern __shared__ __align__(1024) unsigned char smem[];
  uint8_t* sA = smem;                               // 128 x 256
  uint8_t* sB = smem + GM * PROBE_K;                // 256 x 256
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 3 * GM * PROBE_K);
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + 2);
  for (int i = threadIdx.x; i < 3 * GM * PROBE_K / 4; i += blockDim.x)
    reinterpret_cast<uint32_t*>(smem)[i] = (i * 2654435761u + blockIdx.x * 40503u) & 0x1f1f1f1fu;   // tokens 0..31
  if (threadIdx.x == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    fence_mbar_init();
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy stores -> tensor-core reads
  if (threadIdx.x < 32) tmem_alloc(tmem_holder, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;
  if (threadIdx.x == 0) {
    // D=S32, A=B=UINT8, K-major both, N=256, M=128
    const uint32_t idesc = (2u << 4) | (static_cast<uint32_t>(256 >> 3) << 17) | (static_cast<uint32_t>(GM >> 4) << 24);
    const uint32_t sbo = static_cast<uint32_t>(PROBE_K / 16) * 128u;
    const uint32_t a_addr = smem_u32(sA), b_addr = smem_u32(sB);
    for (int b = 0; b < batches; ++b) {
      if (b >= 2) mbar_wait_poll(&bars[b & 1], ((b >> 1) - 1) & 1);     // batch b - 2 has completed
      for (int t = 0; t < PROBE_BATCH; ++t) {
        const uint32_t acc = tmem_base + ((t & 1) ? 256u : 0u);
        for (int j = 0; j < PROBE_K / 32; ++j)
          umma_i8(acc, umma_desc(a_addr + j * 256, 128, sbo), umma_desc(b_addr + j * 256, 128, sbo), idesc, j > 0 ? 1u : 0u);
      }
      umma_commit(&bars[b & 1]);
    }
    for (int b = batches > 2 ? batches - 2 : 0; b < batches; ++b) mbar_wait_poll(&bars[b & 1], (b >> 1) & 1);
  }
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x < 32) tmem_dealloc(tmem_base, 512);
}

}  // namespace pg

using namespace pg;

extern "C" {

int pg_measure_i8_mma_peak(int batches, double* int8_ops_per_s, double* ms_out) {
  PG_CHECK_ARG(batches >= 1 && batches <= (1 << 20), "bad probe arguments");
  const size_t smem = 3 * static_cast<size_t>(GM) * PROBE_K + 64;
  PG_CUDA(cudaFuncSetAttribute(i8_mma_peak_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  cudaEvent_t a, b;
  PG_CUDA(cudaEventCreate(&a));
  PG_CUDA(cudaEventCreate(&b));
  float best = 1e30f;
  for (int rep = 0; rep < 4; ++rep) {
    PG_CUDA(cudaEventRecord(a, 0));
    i8_mma_peak_kernel<<<num_sms(), 128, smem>>>(batches);
    PG_CUDA(cudaEventRecord(b, 0));
    PG_CUDA(cudaEventSynchronize(b));
    float ms = 0;
    PG_CUDA(cudaEventElapsedTime(&ms, a, b));
    if (rep > 0 && ms < best) best = ms;
  }
  PG_CUDA(cudaGetLastError());
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  // per CTA: batches * PROBE_BATCH tiles of 128 x 256 x 256 multiply-adds
  const double ops = 2.0 * GM * 256.0 * PROBE_K * PROBE_BATCH * static_cast<double>(batches) * num_sms();
  if (int8_ops_per_s) *int8_ops_per_s = ops / (best * 1e-3);
  if (ms_out) *ms_out = best;
  return PG_OK;
}

int pg_gemm_width(int L) { return L <= 0 ? 0 : (L + 31) / 32 * 32; }
int64_t pg_gemm_rows(int64_t N) { return N <= 0 ? 0 : round_up(N, GROWS); }   // a CTA loads GROWS query rows

int pg_gemm_pack(const void* tokens, int dtype, int64_t N, int L, int64_t ld, uint8_t* table, int32_t* norms, int K,
                 int max_token, int* flag, void* stream) {
  PG_CHECK_ARG(tokens && table && norms && flag, "null pointer");
  PG_CHECK_ARG(N > 0 && L > 0 && ld >= L, "bad shape");
  PG_CHECK_ARG(K % 32 == 0 && K >= L, "K must be a multiple of 32 and >= L");
  PG_CHECK_ARG(max_token >= 1 && max_token <= 255, "max_token must be in [1,255]");
  const long long rows_padded = pg_gemm_rows(N);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PG_CUDA(cudaMemsetAsync(norms, 0, sizeof(int32_t) * rows_padded, s));
  const long long total = rows_padded * (K / 16);
  long long blocks = ceil_div(total, 256);
  const long long cap = static_cast<long long>(num_sms()) * 32;
  if (blocks > cap) blocks = cap;
#define PG_GP(T)                                                                                               \
  gemm_pack_kernel<T><<<static_cast<unsigned>(blocks), 256, 0, s>>>(static_cast<const T*>(tokens), N, L, ld, table, \
                                                                     norms, rows_padded, K, max_token, flag)
  switch (dtype) {
    case PG_U8: PG_GP(uint8_t); break;
    case PG_I16: PG_GP(int16_t); break;
    case PG_I32: PG_GP(int32_t); break;
    case PG_I64: PG_GP(long long); break;
    case PG_F16: PG_GP(__half); break;
    case PG_F32: PG_GP(float); break;
    case PG_F64: PG_GP(double); break;
    default: set_error("unsupported token dtype %d", dtype); return PG_ERR_INVALID;
  }
#undef PG_GP
  PG_LAUNCH_CHECK();
  return PG_OK;
}

static int gemm_common(GemmParams& prm, const uint8_t* A, const int32_t* normA, int64_t M, const uint8_t* B,
                       const int32_t* normB, int64_t N, int K, int value_kind, int similarity) {
  PG_CHECK_ARG(A && normA && B && normB, "null operand");
  PG_CHECK_ARG(M > 0 && N > 0 && N < (1ll << 32), "bad operand sizes");
  PG_CHECK_ARG(value_kind == GV_F16 || value_kind == GV_F32, "bad value kind %d", value_kind);
  if (K % 32 != 0 || K < 32 || K > GMAX_K) {
    set_error("minkowski GEMM supports rows of up to %d tokens (K=%d)", GMAX_K, K);
    return PG_ERR_UNSUPPORTED;
  }
  memset(&prm, 0, sizeof(prm));
  prm.A = A; prm.normA = normA; prm.M = M;
  prm.B = B; prm.normB = normB; prm.N = N;
  prm.K = K;
  prm.similarity = similarity;
  return PG_OK;
}

int pg_minkowski2_gemm_tile(const uint8_t* A, const int32_t* normA, int64_t M, const uint8_t* B, const int32_t* normB,
                            int64_t N, int K, int value_kind, int similarity, void* out, int64_t ld, void* stream) {
  GemmParams prm;
  int rc = gemm_common(prm, A, normA, M, B, normB, N, K, value_kind, similarity);
  if (rc != PG_OK) return rc;
  PG_CHECK_ARG(out && ld >= N, "bad output");
  prm.out = out;
  prm.ld = ld;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return value_kind == GV_F16 ? launch_gemm<GV_F16, GM_TILE>(prm, s) : launch_gemm<GV_F32, GM_TILE>(prm, s);
}

int pg_minkowski2_gemm_knn(const uint8_t* A, const int32_t* normA, int64_t M, const uint8_t* B, const int32_t* normB,
                           int64_t N, int K, int value_kind, int similarity, int k, int drop, int64_t* out_idx,
                           void* out_val, void* stream) {
  GemmParams prm;
  int rc = gemm_common(prm, A, normA, M, B, normB, N, K, value_kind, similarity);
  if (rc != PG_OK) return rc;
  PG_CHECK_ARG(out_idx && out_val && k >= 1 && drop >= 0, "bad kNN arguments");
  if (k + drop > 32 * kMaxListRounds) { set_error("k=%d too large for the fused lists", k); return PG_ERR_UNSUPPORTED; }
  prm.k = k;
  prm.drop = drop;
  prm.k1 = k + drop;
  prm.out_idx = reinterpret_cast<long long*>(out_idx);
  prm.out_val = out_val;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return value_kind == GV_F16 ? launch_gemm<GV_F16, GM_KNN>(prm, s) : launch_gemm<GV_F32, GM_KNN>(prm, s);
}

static int gemm_eps_common(GemmParams& prm, int s_lo, int s_hi, int64_t* group_counts) {
  PG_CHECK_ARG(group_counts, "null group counts");
  PG_CHECK_ARG(s_lo >= 0 && s_hi >= s_lo && s_hi < PAD_NORM / 2, "bad S range [%d, %d]", s_lo, s_hi);
  prm.s_lo = s_lo;
  prm.s_span = static_cast<unsigned>(s_hi - s_lo);
  prm.group_counts = reinterpret_cast<long long*>(group_counts);
  return PG_OK;
}

__global__ void gemm_sum_groups_kernel(const long long* __restrict__ gc, long long M, long long* __restrict__ counts) {
  const long long r = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (r < M) counts[r] = gc[r] + gc[M + r];
}

int pg_minkowski2_gemm_eps_count(const uint8_t* A, const int32_t* normA, int64_t M, const uint8_t* B,
                                 const int32_t* normB, int64_t N, int K, int s_lo, int s_hi, int64_t* group_counts,
                                 int64_t* counts, void* stream) {
  GemmParams prm;
  int rc = gemm_common(prm, A, normA, M, B, normB, N, K, GV_F32, 0);
  if (rc != PG_OK) return rc;
  rc = gemm_eps_common(prm, s_lo, s_hi, group_counts);
  if (rc != PG_OK) return rc;
  PG_CHECK_ARG(counts, "null counts");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PG_CUDA(cudaMemsetAsync(group_counts, 0, sizeof(int64_t) * 2 * M, s));
  rc = launch_gemm<GV_F32, GM_COUNT>(prm, s);
  if (rc != PG_OK) return rc;
  gemm_sum_groups_kernel<<<static_cast<unsigned>(ceil_div(M, 256)), 256, 0, s>>>(prm.group_counts, M,
                                                                                 reinterpret_cast<long long*>(counts));
  PG_LAUNCH_CHECK();
  return PG_OK;
}

int pg_minkowski2_gemm_eps_fill(const uint8_t* A, const int32_t* normA, int64_t M, const uint8_t* B,
                                const int32_t* normB, int64_t N, int K, int value_kind, int similarity, int s_lo,
                                int s_hi, const int64_t* group_counts, const int64_t* indptr, int64_t* out_idx,
                                void* out_val, void* stream) {
  GemmParams prm;
  int rc = gemm_common(prm, A, normA, M, B, normB, N, K, value_kind, similarity);
  if (rc != PG_OK) return rc;
  rc = gemm_eps_common(prm, s_lo, s_hi, const_cast<int64_t*>(group_counts));
  if (rc != PG_OK) return rc;
  PG_CHECK_ARG(indptr && out_idx && out_val, "null indptr / output");
  prm.indptr = reinterpret_cast<const long long*>(indptr);
  prm.out_idx = reinterpret_cast<long long*>(out_idx);
  prm.out_val = out_val;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return value_kind == GV_F16 ? launch_gemm<GV_F16, GM_FILL>(prm, s) : launch_gemm<GV_F32, GM_FILL>(prm, s);
}

}  // extern "C"
