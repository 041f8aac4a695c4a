// Fused Hamming sweep for long rows (more than 512 residues: W = 24..56 words per plane).
//
// The own row no longer fits in registers, so the sweep is chunked along the sequence: a ring
// tile holds 32 complete stream rows; for every 8-word chunk the thread loads its own row's
// chunk (P*8 registers, from L1/L2) and adds the chunk's mismatch count to 32 per-stream-row
// accumulators; after the last chunk the accumulators are the full distances and go through the
// same epilogues as pg::sweep_kernel (kNN lists behind a threshold, epsilon count / capture /
// fill, tile).  Same ring (bulk copies + mbarriers, the last warp to finish a stage refills
// it), same work items, same parameter block.
#include "pg_sweep.cuh"

namespace pg {

constexpr int LCH = 8;    // words per chunk
constexpr int LBN = 32;   // stream rows per ring tile
constexpr int LSTAGES = 3;

template <int P>
__device__ __forceinline__ int ham_chunk(const uint32_t (&q)[P * LCH], const uint32_t* __restrict__ col, int pstride,
                                         unsigned one) {
  uint32_t m[LCH];
#pragma unroll
  for (int p = 0; p < P; ++p) {
    const uint4* c4 = reinterpret_cast<const uint4*>(col + p * pstride);
#pragma unroll
    for (int h = 0; h < LCH / 4; ++h) {
      const uint4 v = c4[h];
      const int w = h * 4;
      if (p == 0) {
        m[w + 0] = q[w + 0] ^ v.x;
        m[w + 1] = q[w + 1] ^ v.y;
        m[w + 2] = q[w + 2] ^ v.z;
        m[w + 3] = q[w + 3] ^ v.w;
      } else {
        m[w + 0] |= q[p * LCH + w + 0] ^ v.x;
        m[w + 1] |= q[p * LCH + w + 1] ^ v.y;
        m[w + 2] |= q[p * LCH + w + 2] ^ v.z;
        m[w + 3] |= q[p * LCH + w + 3] ^ v.w;
      }
    }
  }
  unsigned s = __popc(m[0]);
#pragma unroll
  for (int w = 1; w < LCH; ++w) s = mad_u32(__popc(m[w]), one, s);
  return static_cast<int>(s);
}

template <int P, int MODE, bool LUT, int WEIGHT>
__global__ void __launch_bounds__(kSweepThreads, 2) sweep_long_kernel(const __grid_constant__ SweepParams prm,
                                                                      const int Wt) {
  const int COLW = P * Wt;                         // words per packed row
  const uint32_t STAGE_BYTES = LBN * COLW * 4;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint32_t* stage_mem = reinterpret_cast<uint32_t*>(smem_raw);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + static_cast<size_t>(LSTAGES) * STAGE_BYTES);
  unsigned* done = reinterpret_cast<unsigned*>(full + kStages);
  uint32_t* lut_s = reinterpret_cast<uint32_t*>(full + 2 * kStages);
  unsigned long long* lists = reinterpret_cast<unsigned long long*>(lut_s + kMaxLutWords);   // [256][k1]

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int lane = tid & 31;

  // the work-item cursor counts ring tiles of LBN rows here
  SweepCursor la;
  la.start(blockIdx.x, prm);
  if (tid == 0) {
    for (int s = 0; s < LSTAGES; ++s) {
      mbar_init(&full[s], 1);
      done[s] = 0;
    }
    fence_mbar_init();
  }
  if (LUT && tid < kMaxLutWords) lut_s[tid] = prm.lut[tid];
  __syncthreads();
#pragma unroll 1
  for (int s = 0; s < LSTAGES; ++s) {
    if (tid == 0 && la.valid(prm)) {
      mbar_arrive_expect_tx(&full[s], STAGE_BYTES);
      bulk_g2s(stage_mem + static_cast<size_t>(s) * LBN * COLW, prm.str + static_cast<size_t>(la.t) * LBN * COLW,
               STAGE_BYTES, &full[s]);
    }
    if (la.valid(prm)) la.advance(prm, gridDim.x);
  }

  const int n_items = prm.n_rowblocks * prm.n_splits;
  const int n_chunks = Wt / LCH;
  const unsigned one = prm.one;
  const int lo = prm.lo;
  const unsigned span = prm.span;
  int stage = 0;
  uint32_t phase = 0;

  for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int split = item / prm.n_rowblocks;
    const int rb = item - split * prm.n_rowblocks;
    long long r = static_cast<long long>(rb) * kConsumers + tid;
    const bool valid = r < prm.rows;
    if (prm.row_map != nullptr && valid) r = prm.row_map[r];
    const uint32_t* ownp = prm.own + static_cast<size_t>(prm.own_row0 + (valid ? r : 0)) * COLW;
    unsigned tau = valid ? 0xffffffffu : 0u;
    long long cnt = 0;
    unsigned long long* cap = nullptr;
    unsigned long long* my_list = lists + static_cast<size_t>(tid) * prm.k1;
    if constexpr (MODE == MODE_KNN) {
      for (int j = 0; j < prm.k1; ++j) my_list[j] = ~0ull;
      __syncwarp();
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

    const int t0 = split * prm.tiles_per_split;
    const int t1 = min(t0 + prm.tiles_per_split, prm.n_tiles);
    for (int t = t0; t < t1; ++t) {
      mbar_wait(&full[stage], phase);
      const uint32_t* tile = stage_mem + static_cast<size_t>(stage) * LBN * COLW;
      const long long col0 = static_cast<long long>(t) * LBN;
      const int ncols = static_cast<int>(min(static_cast<long long>(LBN), prm.str_rows - col0));
      int acc[LBN];
#pragma unroll
      for (int j = 0; j < LBN; ++j) acc[j] = 0;
#pragma unroll 1
      for (int ch = 0; ch < n_chunks; ++ch) {
        uint32_t q[P * LCH];
#pragma unroll
        for (int p = 0; p < P; ++p) {
          const uint4* src = reinterpret_cast<const uint4*>(ownp + p * Wt + ch * LCH);
          const uint4 a = __ldg(src), b = __ldg(src + 1);
          q[p * LCH + 0] = a.x; q[p * LCH + 1] = a.y; q[p * LCH + 2] = a.z; q[p * LCH + 3] = a.w;
          q[p * LCH + 4] = b.x; q[p * LCH + 5] = b.y; q[p * LCH + 6] = b.z; q[p * LCH + 7] = b.w;
        }
#pragma unroll
        for (int j = 0; j < LBN; ++j) acc[j] += ham_chunk<P>(q, tile + j * COLW + ch * LCH, Wt, one);
      }
      if (ncols < LBN) {      // table end: the zero pad rows must never look like neighbours
        // kNN: all ones, which fails the candidate test even against the empty threshold of a list
        // that is not full yet (stream rows < k1); the range and LUT tests reject 0x3fffffff
        const int pad = MODE == MODE_KNN ? -1 : 0x3fffffff;
#pragma unroll
        for (int j = 0; j < LBN; ++j)
          if (j >= ncols) acc[j] = pad;
      }

      if constexpr (MODE == MODE_KNN) {
#pragma unroll
        for (int g = 0; g < LBN / 4; ++g) {
          const unsigned best = min(min(static_cast<unsigned>(acc[4 * g]), static_cast<unsigned>(acc[4 * g + 1])),
                                    min(static_cast<unsigned>(acc[4 * g + 2]), static_cast<unsigned>(acc[4 * g + 3])));
          if (__any_sync(0xffffffffu, best < tau)) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int dv = acc[4 * g + e];
              unsigned cand = __ballot_sync(0xffffffffu, static_cast<unsigned>(dv) < tau);
              while (cand) {
                const int src = __ffs(cand) - 1;
                cand &= cand - 1;
                const unsigned dd = __shfl_sync(0xffffffffu, static_cast<unsigned>(dv), src);
                const unsigned long long key =
                    (static_cast<unsigned long long>(dd) << 32) | static_cast<unsigned>(col0 + 4 * g + e);
                const unsigned t_new =
                    knn_insert_coop(lists + static_cast<size_t>((warp << 5) + src) * prm.k1, prm.k1, key, lane);
                if (lane == src) tau = t_new;
              }
            }
          }
        }
      } else {
#pragma unroll
        for (int j = 0; j < LBN; ++j) {
          const int d = acc[j];
          if constexpr (MODE == MODE_TILE) {
            if (valid && j < ncols) write_tile<WEIGHT>(prm.out, (col0 + j) * prm.ld + r, d, prm.lo, prm.span);
          } else {
            bool hit;
            if constexpr (LUT) hit = d < kMaxLutWords * 32 && ((lut_s[d >> 5] >> (d & 31)) & 1u);
            else hit = static_cast<unsigned>(d - lo) <= span;
            if (hit && valid) {
              if constexpr (MODE == MODE_COUNT) {
                if (cap != nullptr && cnt < prm.capture_cap)
                  cap[cnt] = (static_cast<unsigned long long>(static_cast<unsigned>(d)) << 32) |
                             static_cast<unsigned>(col0 + j);
              } else {
                prm.out_idx[cnt] = col0 + j;
                write_weight(prm.out_w, cnt, d, WEIGHT);
              }
              ++cnt;
            }
          }
        }
      }

      __syncwarp();
      if (lane == 0) {
        if (atom_add_acq_rel_cta(&done[stage], 1u) == kConsumerWarps - 1) {
          done[stage] = 0;
          if (la.valid(prm)) {
            fence_proxy_async();
            mbar_arrive_expect_tx(&full[stage], STAGE_BYTES);
            bulk_g2s(stage_mem + static_cast<size_t>(stage) * LBN * COLW,
                     prm.str + static_cast<size_t>(la.t) * LBN * COLW, STAGE_BYTES, &full[stage]);
          }
        }
      }
      if (la.valid(prm)) la.advance(prm, gridDim.x);
      if (++stage == LSTAGES) { stage = 0; phase ^= 1u; }
    }

    if constexpr (MODE == MODE_KNN) {
      if (valid) {
        unsigned long long* dst = prm.part + static_cast<size_t>(split) * prm.k1 * prm.rows_total + r;
        for (int j = 0; j < prm.k1; ++j) dst[static_cast<size_t>(j) * prm.rows_total] = my_list[j];
      }
      __syncwarp();
    } else if constexpr (MODE == MODE_COUNT) {
      if (valid) prm.split_counts[static_cast<size_t>(split) * prm.rows_total + r] = cnt;
    }
  }
}

template <int P, int MODE, bool LUT, int WEIGHT>
static int launch_long_one(const SweepParams& prm, const SweepLaunch& l, int Wt) {
  auto kern = sweep_long_kernel<P, MODE, LUT, WEIGHT>;
  const size_t smem = static_cast<size_t>(LSTAGES) * LBN * P * Wt * 4 + 2 * kStages * sizeof(uint64_t) +
                      kMaxLutWords * 4 + l.list_bytes;
  if (smem > 227 * 1024) { set_error("long-row sweep does not fit in shared memory (%zu bytes)", smem); return PG_ERR_UNSUPPORTED; }
  PG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  int occ = 0;
  PG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kSweepThreads, smem));
  if (occ < 1) { set_error("long-row sweep does not fit on an SM"); return PG_ERR_UNSUPPORTED; }
  const long long n_items = static_cast<long long>(prm.n_rowblocks) * prm.n_splits;
  long long grid = static_cast<long long>(num_sms()) * occ;
  if (grid > n_items) grid = n_items;
  if (grid < 1) grid = 1;
  kern<<<static_cast<unsigned>(grid), kSweepThreads, smem, l.stream>>>(prm, Wt);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

// planes = 5 only (protein alphabets); words = 24..56, a multiple of 8
int sweep_long_p5(const SweepParams& prm, const SweepLaunch& l, int words) {
  constexpr int P = 5;
  switch (l.mode) {
    case MODE_KNN: return launch_long_one<P, MODE_KNN, false, 0>(prm, l, words);
    case MODE_COUNT:
      return l.lut ? launch_long_one<P, MODE_COUNT, true, 0>(prm, l, words)
                   : launch_long_one<P, MODE_COUNT, false, 0>(prm, l, words);
    case MODE_FILL:
      if (l.weight == PG_W_SIM_F32)
        return l.lut ? launch_long_one<P, MODE_FILL, true, PG_W_SIM_F32>(prm, l, words)
                     : launch_long_one<P, MODE_FILL, false, PG_W_SIM_F32>(prm, l, words);
      return l.lut ? launch_long_one<P, MODE_FILL, true, PG_W_I64>(prm, l, words)
                   : launch_long_one<P, MODE_FILL, false, PG_W_I64>(prm, l, words);
    case MODE_TILE:
      if (l.weight == PG_W_I64) return launch_long_one<P, MODE_TILE, false, PG_W_I64>(prm, l, words);
      if (l.weight == PG_W_SIM_F32) return launch_long_one<P, MODE_TILE, false, PG_W_SIM_F32>(prm, l, words);
      if (l.weight == PG_W_FLAG_U8) return launch_long_one<P, MODE_TILE, false, PG_W_FLAG_U8>(prm, l, words);
      return launch_long_one<P, MODE_TILE, false, PG_W_I32>(prm, l, words);
  }
  set_error("bad sweep mode %d", l.mode);
  return PG_ERR_INVALID;
}

}  // namespace pg
