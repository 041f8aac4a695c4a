// Growing a built graph by new rows (graph.extend_neighbours): the two HBM-bound kernels that
// join an old row's stored neighbours with what a one-sided sweep found among the new columns.
//   pg_knn_extend_merge  sorted kNN lists of an old row + the row's candidates among the new rows
//   pg_csr_append        epsilon CSR rows of the old columns followed by those of the new columns
#include <algorithm>
#include <type_traits>

#include "pg_common.cuh"

namespace pg {

// ---- kNN: merge two sorted lists per row -------------------------------------------------------
// Order (weight asc, index asc) for distances, (weight desc, index asc) for float32 similarities:
// sim_f32 is strictly decreasing in d, so both are the (distance, index) order of the build.
template <bool SIM>
__device__ __forceinline__ bool goes_first(typename std::conditional<SIM, float, long long>::type wa, long long ia,
                                           typename std::conditional<SIM, float, long long>::type wb, long long ib) {
  if (wa != wb) return SIM ? wa > wb : wa < wb;
  return ia <= ib;
}

// One thread per row merges; with PARK, it writes its row to shared memory (row stride k + 1:
// conflict-free) and the block stores its rows * k outputs contiguously, as knn_lists_finalize
// does.  Rows too wide for that (k beyond a few hundred) are stored by their thread directly.
template <bool SIM, bool PARK>
__global__ void knn_extend_merge_kernel(const long long* __restrict__ prev_idx, const void* __restrict__ prev_w, int ka,
                                        const long long* __restrict__ cand_idx, const void* __restrict__ cand_w, int kb,
                                        long long rows, long long col_base, int k, long long* __restrict__ out_idx,
                                        void* __restrict__ out_w) {
  using W = typename std::conditional<SIM, float, long long>::type;
  extern __shared__ unsigned long long ext_sm[];
  long long* sm_idx = reinterpret_cast<long long*>(ext_sm);
  W* sm_w = reinterpret_cast<W*>(sm_idx + static_cast<size_t>(blockDim.x) * (k + 1));
  const long long row_base = blockIdx.x * static_cast<long long>(blockDim.x);
  const long long r = row_base + threadIdx.x;
  if (r < rows) {
    const long long* pi = prev_idx + r * ka;
    const W* pw = reinterpret_cast<const W*>(prev_w) + r * ka;
    const long long* ci = cand_idx + r * kb;
    const W* cw = reinterpret_cast<const W*>(cand_w) + r * kb;
    int a = 0, b = 0;
    long long ia = ka > 0 ? pi[0] : -1, ib = kb > 0 ? ci[0] : -1;
    W wa = ka > 0 ? pw[0] : W(0), wb = kb > 0 ? cw[0] : W(0);
    if (ib >= 0) ib += col_base;
    for (int j = 0; j < k; ++j) {
      long long idx = -1;
      W w = W(0);                                   // missing entry: index -1, weight 0 (0.0f)
      const bool has_a = ia >= 0, has_b = ib >= 0;
      if (has_a && (!has_b || goes_first<SIM>(wa, ia, wb, ib))) {
        idx = ia;
        w = wa;
        ++a;
        ia = a < ka ? pi[a] : -1;
        if (a < ka) wa = pw[a];
      } else if (has_b) {
        idx = ib;
        w = wb;
        ++b;
        ib = b < kb ? ci[b] : -1;
        if (ib >= 0) { ib += col_base; wb = cw[b]; }
      }
      if (PARK) {
        sm_idx[threadIdx.x * (k + 1) + j] = idx;
        sm_w[threadIdx.x * (k + 1) + j] = w;
      } else {
        out_idx[r * k + j] = idx;
        reinterpret_cast<W*>(out_w)[r * k + j] = w;
      }
    }
  }
  if (PARK) {
    __syncthreads();
    const long long here = min(static_cast<long long>(blockDim.x), rows - row_base);
    const int total = static_cast<int>(here) * k;
    for (int e = threadIdx.x; e < total; e += blockDim.x) {
      const int rr = e / k, j = e - rr * k;
      out_idx[row_base * k + e] = sm_idx[rr * (k + 1) + j];
      reinterpret_cast<W*>(out_w)[row_base * k + e] = sm_w[rr * (k + 1) + j];
    }
  }
}

constexpr size_t kExtendParkLimit = 200u << 10;   // parked rows of one block, below the 227 KB per block

template <bool SIM>
static int extend_merge_launch(const long long* pi, const void* pw, int ka, const long long* ci, const void* cw, int kb,
                               long long rows, long long col_base, int k, long long* oi, void* ow, cudaStream_t cs) {
  const int threads = k <= 32 ? 128 : 32;
  const size_t smem = static_cast<size_t>(threads) * (k + 1) * (8 + (SIM ? 4 : 8));
  const unsigned grid = static_cast<unsigned>(ceil_div(rows, threads));
  if (smem <= kExtendParkLimit) {
    if (smem > (48u << 10))
      PG_CUDA(cudaFuncSetAttribute(knn_extend_merge_kernel<SIM, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   static_cast<int>(smem)));
    knn_extend_merge_kernel<SIM, true><<<grid, threads, smem, cs>>>(pi, pw, ka, ci, cw, kb, rows, col_base, k, oi, ow);
  } else {
    knn_extend_merge_kernel<SIM, false><<<grid, threads, 0, cs>>>(pi, pw, ka, ci, cw, kb, rows, col_base, k, oi, ow);
  }
  PG_LAUNCH_CHECK();
  return PG_OK;
}

// ---- epsilon: append CSR rows ----------------------------------------------------------------
// One warp per output row: out row r = old row r, then added row r with col_base added to its
// indices.  The entries of row r of a part start at idx[indptr[r] - indptr[0]], so row slices of
// a larger CSR are taken as they are.  out_indptr[r + 1] is the sum of both parts' row ends: the
// scan over the output rows is already in the two input indptr arrays.
template <typename W>
__global__ void __launch_bounds__(256) csr_append_kernel(const long long* __restrict__ old_indptr,
                                                         const long long* __restrict__ old_idx, const W* __restrict__ old_w,
                                                         const long long* __restrict__ add_indptr,
                                                         const long long* __restrict__ add_idx, const W* __restrict__ add_w,
                                                         long long rows, long long col_base,
                                                         long long* __restrict__ out_indptr, long long* __restrict__ out_idx,
                                                         W* __restrict__ out_w) {
  const int lane = threadIdx.x & 31;
  const long long warps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
  const long long o0 = old_indptr[0], a0 = add_indptr[0];
  for (long long r = blockIdx.x * static_cast<long long>(blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += warps) {
    const long long os = old_indptr[r] - o0, oe = old_indptr[r + 1] - o0;
    const long long as = add_indptr[r] - a0, ae = add_indptr[r + 1] - a0;
    const long long dst = os + as;
    if (lane == 0) {
      out_indptr[r + 1] = oe + ae;
      if (r == 0) out_indptr[0] = 0;
    }
    const long long no = oe - os, na = ae - as;
    for (long long e = lane; e < no; e += 32) {
      out_idx[dst + e] = old_idx[os + e];
      out_w[dst + e] = old_w[os + e];
    }
    for (long long e = lane; e < na; e += 32) {
      out_idx[dst + no + e] = add_idx[as + e] + col_base;
      out_w[dst + no + e] = add_w[as + e];
    }
  }
}

}  // namespace pg

using namespace pg;

extern "C" {

int pg_knn_extend_merge(const int64_t* prev_idx, const void* prev_w, int ka, const int64_t* cand_idx,
                        const void* cand_w, int kb, int64_t rows, int64_t col_base, int k, int weight,
                        int64_t* out_idx, void* out_w, void* stream) {
  PG_CHECK_ARG(out_idx && out_w, "null output pointer");
  PG_CHECK_ARG(ka >= 0 && kb >= 0 && k >= 1 && rows >= 0 && col_base >= 0, "bad merge geometry ka=%d kb=%d k=%d", ka,
               kb, k);
  PG_CHECK_ARG((ka == 0 || (prev_idx && prev_w)) && (kb == 0 || (cand_idx && cand_w)), "null input pointer");
  PG_CHECK_ARG(weight == PG_W_I64 || weight == PG_W_SIM_F32, "bad weight kind %d", weight);
  if (rows == 0) return PG_OK;
  cudaStream_t cs = static_cast<cudaStream_t>(stream);
  const long long* pi = reinterpret_cast<const long long*>(prev_idx);
  const long long* ci = reinterpret_cast<const long long*>(cand_idx);
  long long* oi = reinterpret_cast<long long*>(out_idx);
  return weight == PG_W_SIM_F32 ? extend_merge_launch<true>(pi, prev_w, ka, ci, cand_w, kb, rows, col_base, k, oi, out_w, cs)
                                : extend_merge_launch<false>(pi, prev_w, ka, ci, cand_w, kb, rows, col_base, k, oi, out_w, cs);
}

int pg_csr_append(const int64_t* old_indptr, const int64_t* old_idx, const void* old_w, const int64_t* add_indptr,
                  const int64_t* add_idx, const void* add_w, int64_t rows, int64_t col_base, int weight,
                  int64_t* out_indptr, int64_t* out_idx, void* out_w, void* stream) {
  PG_CHECK_ARG(out_indptr && (rows == 0 || (old_indptr && add_indptr)), "null pointer");
  PG_CHECK_ARG(rows >= 0 && col_base >= 0, "bad append geometry rows=%lld col_base=%lld", (long long)rows,
               (long long)col_base);
  PG_CHECK_ARG(weight == PG_W_I64 || weight == PG_W_SIM_F32, "bad weight kind %d", weight);
  cudaStream_t cs = static_cast<cudaStream_t>(stream);
  if (rows == 0) {
    PG_CUDA(cudaMemsetAsync(out_indptr, 0, sizeof(int64_t), cs));
    return PG_OK;
  }
  const long long blocks = std::min<long long>(ceil_div(rows, 8), static_cast<long long>(num_sms()) * 32);
  const long long* op = reinterpret_cast<const long long*>(old_indptr);
  const long long* ap = reinterpret_cast<const long long*>(add_indptr);
  const long long* oi = reinterpret_cast<const long long*>(old_idx);
  const long long* ai = reinterpret_cast<const long long*>(add_idx);
  long long* xp = reinterpret_cast<long long*>(out_indptr);
  long long* xi = reinterpret_cast<long long*>(out_idx);
  if (weight == PG_W_SIM_F32)
    csr_append_kernel<float><<<static_cast<unsigned>(blocks), 256, 0, cs>>>(
        op, oi, static_cast<const float*>(old_w), ap, ai, static_cast<const float*>(add_w), rows, col_base, xp, xi,
        static_cast<float*>(out_w));
  else
    csr_append_kernel<long long><<<static_cast<unsigned>(blocks), 256, 0, cs>>>(
        op, oi, static_cast<const long long*>(old_w), ap, ai, static_cast<const long long*>(add_w), rows, col_base, xp,
        xi, static_cast<long long*>(out_w));
  PG_LAUNCH_CHECK();
  return PG_OK;
}

}  // extern "C"
