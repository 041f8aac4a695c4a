// Fused Hamming sweep for long rows: P = 5 with W = 24..56 words per plane (513..1792 residues), and in
// the chunked mode P = 5 with W = 64..1024 and P = 8 with W = 16..1024 (up to 32768 residues).
//
// The own row no longer fits in registers, so the sweep is chunked along the sequence: for every
// 8-word chunk the thread loads its own row's chunk (P*8 registers, from L1/L2) and adds the chunk's
// mismatch count to 32 per-stream-row accumulators; after the last chunk the accumulators are the
// full distances and go through the same epilogues as pg::sweep_kernel (kNN lists behind a
// threshold, epsilon count / capture / fill, tile).  Same ring (bulk copies + mbarriers, the last
// warp to finish a stage refills it), same work items, same parameter block.
//
// Ring unit.  Without CHUNKED a stage holds 32 complete stream rows (P*W words each: 35 KB at W = 56).
// With CHUNKED a stage holds one word chunk of 32 stream rows -- P planes x CW = 32 words (1024
// residues) of each, 20 KB at P = 5 and 32 KB at P = 8 -- and the ring walks (stream tile, chunk)
// pairs; the accumulators stay in registers across the chunks of a tile and the epilogue runs after
// the last one.  The global layout [rows][P][W] is unchanged: a stage is 32*P bulk copies of
// cw*4 bytes (cw = CW, or W mod CW for the last chunk of a row: 8..24 words), issued by the 32 lanes
// of the refilling warp, one stream row per lane.  The stage count is chosen per launch (3, or 2
// when the kNN lists would otherwise cost a CTA per SM or not fit), truth tables of more than
// kMaxLutWords words come from device memory (WideArgs::lut_ext).
#pragma once
#include "pg_sweep.cuh"

namespace pg {

constexpr int LCH = 8;    // words per chunk
constexpr int LBN = 32;   // stream rows per ring tile
constexpr int LSTAGES = 3;
constexpr int kWideChunk = 32;        // CHUNKED: words per plane and stream row in one ring stage

// CHUNKED: what the parameter block does not hold (an argument of its own, so that the parameter
// layout of the whole-row instantiations stays as it is)
struct WideArgs {
  const uint32_t* lut_ext;   // truth table of more than kMaxLutWords words in device memory, or null
  int lut_words;             // words of the truth table (prm.lut or lut_ext)
  int stages;                // ring stages
};

template <int P, int CH = LCH>
__device__ __forceinline__ int ham_chunk(const uint32_t (&q)[P * CH], const uint32_t* __restrict__ col, int pstride,
                                         unsigned one) {
  uint32_t m[CH];
#pragma unroll
  for (int p = 0; p < P; ++p) {
    const uint4* c4 = reinterpret_cast<const uint4*>(col + p * pstride);
#pragma unroll
    for (int h = 0; h < CH / 4; ++h) {
      const uint4 v = c4[h];
      const int w = h * 4;
      if (p == 0) {
        m[w + 0] = q[w + 0] ^ v.x;
        m[w + 1] = q[w + 1] ^ v.y;
        m[w + 2] = q[w + 2] ^ v.z;
        m[w + 3] = q[w + 3] ^ v.w;
      } else {
        m[w + 0] |= q[p * CH + w + 0] ^ v.x;
        m[w + 1] |= q[p * CH + w + 1] ^ v.y;
        m[w + 2] |= q[p * CH + w + 2] ^ v.z;
        m[w + 3] |= q[p * CH + w + 3] ^ v.w;
      }
    }
  }
  unsigned s = __popc(m[0]);
#pragma unroll
  for (int w = 1; w < CH; ++w) s = mad_u32(__popc(m[w]), one, s);
  return static_cast<int>(s);
}

// CHUNKED: issue the copy of ring unit (tile t, chunk c) into stage memory `dst`; all 32 lanes of
// a warp call it, lane j copies the P plane segments of stream row j of the tile.
template <int P>
__device__ __forceinline__ void issue_wide_unit(uint32_t* dst, uint64_t* bar, const uint32_t* str, int Wt, int t,
                                                int c, int lane) {
  const int cw = min(kWideChunk, Wt - c * kWideChunk);
  if (lane == 0) mbar_arrive_expect_tx(bar, static_cast<uint32_t>(LBN * P * cw * 4));
  __syncwarp();
  const uint32_t* src = str + (static_cast<size_t>(t) * LBN + lane) * P * Wt + c * kWideChunk;
  uint32_t* d = dst + lane * P * cw;
#pragma unroll
  for (int p = 0; p < P; ++p) bulk_g2s(d + p * cw, src + static_cast<size_t>(p) * Wt, static_cast<uint32_t>(cw * 4), bar);
}

template <int P, int MODE, bool LUT, int WEIGHT, bool CHUNKED = false>
__global__ void __launch_bounds__(kSweepThreads, 2) sweep_long_kernel(const __grid_constant__ SweepParams prm,
                                                                      const int Wt, const WideArgs wide) {
  const int COLW = P * Wt;                         // words per packed row
  const uint32_t STAGE_BYTES = LBN * COLW * 4;
  // CHUNKED: own-row words per register load (8 at P = 5; 4 at P = 8 keep q[] at 32 registers)
  constexpr int SUB = P == 8 ? 4 : LCH;
  constexpr uint32_t WIDE_STAGE_WORDS = LBN * P * kWideChunk;
  const int n_stages = CHUNKED ? wide.stages : LSTAGES;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint32_t* stage_mem = reinterpret_cast<uint32_t*>(smem_raw);
  uint64_t* full = reinterpret_cast<uint64_t*>(
      smem_raw + (CHUNKED ? static_cast<size_t>(n_stages) * WIDE_STAGE_WORDS * 4 : static_cast<size_t>(LSTAGES) * STAGE_BYTES));
  unsigned* done = reinterpret_cast<unsigned*>(full + kStages);
  uint32_t* lut_s = reinterpret_cast<uint32_t*>(full + 2 * kStages);
  // CHUNKED: the truth table takes round_up(lut_words, 4) words in count / fill mode only
  const int lut_room = !CHUNKED ? kMaxLutWords : (LUT ? (wide.lut_words + 3) & ~3 : 0);
  unsigned long long* lists = reinterpret_cast<unsigned long long*>(lut_s + lut_room);   // [256][k1]

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int lane = tid & 31;

  // the work-item cursor counts ring tiles of LBN rows here; CHUNKED: (tile, chunk) units, la_c the chunk
  SweepCursor la;
  la.start(blockIdx.x, prm);
  const int n_wide = CHUNKED ? (Wt + kWideChunk - 1) / kWideChunk : 1;
  int la_c = 0;
  if (tid == 0) {
    for (int s = 0; s < n_stages; ++s) {
      mbar_init(&full[s], 1);
      done[s] = 0;
    }
    fence_mbar_init();
  }
  if constexpr (CHUNKED) {
    if (LUT) {
      const uint32_t* src = wide.lut_ext != nullptr ? wide.lut_ext : prm.lut;
      for (int i = tid; i < wide.lut_words; i += kSweepThreads) lut_s[i] = src[i];
    }
  } else {
    if (LUT && tid < kMaxLutWords) lut_s[tid] = prm.lut[tid];
  }
  __syncthreads();
#pragma unroll 1
  for (int s = 0; s < n_stages; ++s) {
    if constexpr (CHUNKED) {
      if (warp == 0 && la.valid(prm))
        issue_wide_unit<P>(stage_mem + static_cast<size_t>(s) * WIDE_STAGE_WORDS, &full[s], prm.str, Wt, la.t, la_c, lane);
      if (la.valid(prm) && ++la_c == n_wide) { la_c = 0; la.advance(prm, gridDim.x); }
    } else {
      if (tid == 0 && la.valid(prm)) {
        mbar_arrive_expect_tx(&full[s], STAGE_BYTES);
        bulk_g2s(stage_mem + static_cast<size_t>(s) * LBN * COLW, prm.str + static_cast<size_t>(la.t) * LBN * COLW,
                 STAGE_BYTES, &full[s]);
      }
      if (la.valid(prm)) la.advance(prm, gridDim.x);
    }
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
      if constexpr (!CHUNKED) mbar_wait(&full[stage], phase);
      const uint32_t* tile = stage_mem + static_cast<size_t>(stage) * LBN * COLW;
      const long long col0 = static_cast<long long>(t) * LBN;
      const int ncols = static_cast<int>(min(static_cast<long long>(LBN), prm.str_rows - col0));
      int acc[LBN];
#pragma unroll
      for (int j = 0; j < LBN; ++j) acc[j] = 0;
      if constexpr (CHUNKED) {
#pragma unroll 1
        for (int c = 0; c < n_wide; ++c) {
          mbar_wait(&full[stage], phase);
          const int cw = min(kWideChunk, Wt - c * kWideChunk);
          const uint32_t* unit = stage_mem + static_cast<size_t>(stage) * WIDE_STAGE_WORDS;
#pragma unroll 1
          for (int h = 0; h < cw; h += SUB) {
            uint32_t q[P * SUB];
#pragma unroll
            for (int p = 0; p < P; ++p) {
              const uint4* src = reinterpret_cast<const uint4*>(ownp + p * Wt + c * kWideChunk + h);
#pragma unroll
              for (int v = 0; v < SUB / 4; ++v) {
                const uint4 a = __ldg(src + v);
                q[p * SUB + 4 * v + 0] = a.x; q[p * SUB + 4 * v + 1] = a.y;
                q[p * SUB + 4 * v + 2] = a.z; q[p * SUB + 4 * v + 3] = a.w;
              }
            }
#pragma unroll
            for (int j = 0; j < LBN; ++j) acc[j] += ham_chunk<P, SUB>(q, unit + j * P * cw + h, cw, one);
          }
          // done with this unit: the last warp to get here refills the stage with the lookahead unit
          __syncwarp();
          unsigned last = 0;
          if (lane == 0) last = atom_add_acq_rel_cta(&done[stage], 1u) == kConsumerWarps - 1;
          last = __shfl_sync(0xffffffffu, last, 0);
          if (last) {
            if (lane == 0) done[stage] = 0;
            if (la.valid(prm)) {
              fence_proxy_async();
              issue_wide_unit<P>(stage_mem + static_cast<size_t>(stage) * WIDE_STAGE_WORDS, &full[stage], prm.str, Wt,
                                 la.t, la_c, lane);
            }
          }
          if (la.valid(prm) && ++la_c == n_wide) { la_c = 0; la.advance(prm, gridDim.x); }
          if (++stage == n_stages) { stage = 0; phase ^= 1u; }
        }
      } else {
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
            if constexpr (LUT && CHUNKED) hit = d < wide.lut_words * 32 && ((lut_s[d >> 5] >> (d & 31)) & 1u);
            else if constexpr (LUT) hit = d < kMaxLutWords * 32 && ((lut_s[d >> 5] >> (d & 31)) & 1u);
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

      if constexpr (!CHUNKED) {
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

// Shared memory of a CHUNKED launch with `stages` ring stages.
template <int P, int MODE, bool LUT>
static size_t wide_smem_bytes(const SweepLaunch& l, int stages) {
  const size_t lut = LUT ? static_cast<size_t>((l.lut_words + 3) & ~3) * 4 : 0;
  return static_cast<size_t>(stages) * LBN * P * kWideChunk * 4 + 2 * kStages * sizeof(uint64_t) + lut +
         (MODE == MODE_KNN ? l.list_bytes : 0);
}

template <int P, int MODE, bool LUT, int WEIGHT, bool CHUNKED>
static int launch_long_one(const SweepParams& prm, const SweepLaunch& l, int Wt) {
  auto kern = sweep_long_kernel<P, MODE, LUT, WEIGHT, CHUNKED>;
  WideArgs wide{l.lut_ext, l.lut_words, 0};
  size_t smem = 0;
  int occ = 0;
  if constexpr (CHUNKED) {
    // 3 stages unless 2 give more CTAs per SM (long kNN lists) or 3 do not fit at all
    for (int st = LSTAGES; st >= 2; --st) {
      const size_t b = wide_smem_bytes<P, MODE, LUT>(l, st);
      if (b > 227 * 1024) continue;
      int o = 0;
      PG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(b)));
      PG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, kern, kSweepThreads, b));
      if (o > occ) { occ = o; smem = b; wide.stages = st; }
    }
    if (wide.stages == 0) { set_error("chunked long-row sweep does not fit in shared memory"); return PG_ERR_UNSUPPORTED; }
    PG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  } else {
    smem = static_cast<size_t>(LSTAGES) * LBN * P * Wt * 4 + 2 * kStages * sizeof(uint64_t) + kMaxLutWords * 4 +
           l.list_bytes;
    if (smem > 227 * 1024) { set_error("long-row sweep does not fit in shared memory (%zu bytes)", smem); return PG_ERR_UNSUPPORTED; }
    PG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    PG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kSweepThreads, smem));
  }
  if (occ < 1) { set_error("long-row sweep does not fit on an SM"); return PG_ERR_UNSUPPORTED; }
  const long long n_items = static_cast<long long>(prm.n_rowblocks) * prm.n_splits;
  long long grid = static_cast<long long>(num_sms()) * occ;
  if (grid > n_items) grid = n_items;
  if (grid < 1) grid = 1;
  kern<<<static_cast<unsigned>(grid), kSweepThreads, smem, l.stream>>>(prm, Wt, wide);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

// Every mode and weight of the long-row sweep at P planes; CHUNKED selects the chunked ring.
template <int P, bool CHUNKED>
static int launch_long(const SweepParams& prm, const SweepLaunch& l, int words) {
  switch (l.mode) {
    case MODE_KNN: return launch_long_one<P, MODE_KNN, false, 0, CHUNKED>(prm, l, words);
    case MODE_COUNT:
      return l.lut ? launch_long_one<P, MODE_COUNT, true, 0, CHUNKED>(prm, l, words)
                   : launch_long_one<P, MODE_COUNT, false, 0, CHUNKED>(prm, l, words);
    case MODE_FILL:
      if (l.weight == PG_W_SIM_F32)
        return l.lut ? launch_long_one<P, MODE_FILL, true, PG_W_SIM_F32, CHUNKED>(prm, l, words)
                     : launch_long_one<P, MODE_FILL, false, PG_W_SIM_F32, CHUNKED>(prm, l, words);
      return l.lut ? launch_long_one<P, MODE_FILL, true, PG_W_I64, CHUNKED>(prm, l, words)
                   : launch_long_one<P, MODE_FILL, false, PG_W_I64, CHUNKED>(prm, l, words);
    case MODE_TILE:
      if (l.weight == PG_W_I64) return launch_long_one<P, MODE_TILE, false, PG_W_I64, CHUNKED>(prm, l, words);
      if (l.weight == PG_W_SIM_F32) return launch_long_one<P, MODE_TILE, false, PG_W_SIM_F32, CHUNKED>(prm, l, words);
      if (l.weight == PG_W_FLAG_U8) return launch_long_one<P, MODE_TILE, false, PG_W_FLAG_U8, CHUNKED>(prm, l, words);
      return launch_long_one<P, MODE_TILE, false, PG_W_I32, CHUNKED>(prm, l, words);
  }
  set_error("bad sweep mode %d", l.mode);
  return PG_ERR_INVALID;
}

}  // namespace pg
