// Mutation masks and index selections on the packed table (HBM-bound, one pass each).
//   prograph.py:488-492  boolean_mutant_array        -> pg_mutant_bits / pg_mutant_bool
//   prograph.py:494-505  calc_mutated_positions      -> pg_mutant_any
//   prograph.py:254-343  indexing (distances, positions, Bool) and
//   prograph.py:349-368  get_mutated_positions       -> pg_select_rows + pg_flag_indices
//   prograph.py:147-154, :305  distance census        -> pg_distance_hist
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <vector>

#include "pg_common.cuh"

namespace pg {

constexpr int kMaxMaskWords = 128;  // selection masks passed as kernel parameters: rows up to 4096 residues

struct WordVec { uint32_t w[kMaxMaskWords]; };
struct LutVec { uint32_t w[kMaxMaskWords + 1]; };     // truth table over d = 0 .. 32*words: one word more

__global__ void mutant_bits_kernel(const uint32_t* __restrict__ table, long long N, int planes, int words,
                                   const uint32_t* __restrict__ ref, uint32_t* __restrict__ mut) {
  const long long total = N * words;
  const int wshift = pow2_shift(words);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    long long n;
    int w;
    split_index(i, words, wshift, &n, &w);
    const uint32_t* row = table + static_cast<size_t>(n) * planes * words + w;
    uint32_t m = 0;
    for (int p = 0; p < planes; ++p) m |= __ldcs(row + p * words) ^ __ldg(ref + p * words + w);
    mut[i] = m;
  }
}

// One thread per (row, half word): 16 mask bits become 16 bytes -- one 128-bit store, and consecutive
// threads write consecutive 16-byte pieces of the output (whole sectors per store instruction; the
// first version wrote 32 bytes per thread as two half-sector stores and reached 3.5 TB/s).  A nibble
// expands to four 0/1 bytes with one multiply ((n * 0x00204081) & 0x01010101).  The two threads of a
// word read the same plane words (one L1 line).  HBM-bound: reads planes * words * 4 bytes, writes L
// bytes per row.
template <int ILP>
__global__ void __launch_bounds__(256) mutant_bool_kernel(const uint32_t* __restrict__ table, long long N, int planes,
                                                          int words, int L, const uint32_t* __restrict__ ref,
                                                          uint8_t* __restrict__ out) {
  const int halves = 2 * words;
  const long long total = N * halves;
  const bool vec16 = (L % 16 == 0) && (reinterpret_cast<uintptr_t>(out) % 16 == 0);
  const int hshift = pow2_shift(halves);
  const long long step = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i0 = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i0 < total; i0 += step * ILP) {
    // ILP independent (row, half word) items per thread: all their plane words are requested before
    // the first mask is formed (20 bytes of loads per item do not cover the HBM latency on their own)
    uint32_t m[ILP];
    long long n[ILP];
    int h[ILP];
#pragma unroll
    for (int u = 0; u < ILP; ++u) {
      const long long i = i0 + u * step;
      m[u] = 0;
      n[u] = -1;
      h[u] = 0;
      if (i < total) {
        split_index(i, halves, hshift, &n[u], &h[u]);
        const int w = h[u] >> 1;
        const uint32_t* row = table + static_cast<size_t>(n[u]) * planes * words + w;
        for (int p = 0; p < planes; ++p) m[u] |= __ldg(row + p * words) ^ __ldg(ref + p * words + w);
      }
    }
#pragma unroll
    for (int u = 0; u < ILP; ++u) {
      if (n[u] < 0) continue;
      const int have = min(16, L - h[u] * 16);
      if (have <= 0) continue;
      const uint32_t mm = (h[u] & 1) ? (m[u] >> 16) : (m[u] & 0xffffu);
      uint32_t b[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) b[k] = (((mm >> (4 * k)) & 0xfu) * 0x00204081u) & 0x01010101u;
      uint8_t* dst = out + static_cast<size_t>(n[u]) * L + h[u] * 16;
      if (have == 16 && vec16) {
        __stcs(reinterpret_cast<uint4*>(dst), make_uint4(b[0], b[1], b[2], b[3]));
      } else {
        for (int l = 0; l < have; ++l) dst[l] = static_cast<uint8_t>((b[l >> 2] >> (8 * (l & 3))) & 1u);
      }
    }
  }
}

__global__ void mutant_any_kernel(const uint32_t* __restrict__ mut, long long N, int words, uint32_t* __restrict__ any_bits) {
  // grid-stride OR per word column; a warp OR-reduces, one atomicOr per warp and word
  for (int w = 0; w < words; ++w) {
    uint32_t acc = 0;
    for (long long n = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; n < N;
         n += static_cast<long long>(gridDim.x) * blockDim.x)
      acc |= mut[static_cast<size_t>(n) * words + w];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc |= __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0 && acc) atomicOr(any_bits + w, acc);
  }
}

// The masks of the selection: rows of up to kMaxMaskWords words take them as kernel parameters
// (constant-bank reads, nothing to copy); longer rows read them from a small device buffer.
struct ParamMasks {
  LutVec lut;
  WordVec inside, outside;
  __device__ uint32_t in(int w) const { return inside.w[w]; }
  __device__ uint32_t out(int w) const { return outside.w[w]; }
  __device__ uint32_t lut_word(int i) const { return lut.w[i]; }
};
struct BufferMasks {
  const uint32_t* buf;   // [inside: words][outside: words][lut: words + 1]
  int words;
  __device__ uint32_t in(int w) const { return __ldg(buf + w); }
  __device__ uint32_t out(int w) const { return __ldg(buf + words + w); }
  __device__ uint32_t lut_word(int i) const { return __ldg(buf + 2 * words + i); }
};

template <typename Masks>
__global__ void select_rows_kernel(const uint32_t* __restrict__ mut, long long N, int words, const Masks masks,
                                   int use_lut, int pos_mode, uint8_t* __restrict__ flag) {
  for (long long n = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; n < N;
       n += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint32_t* m = mut + static_cast<size_t>(n) * words;
    int d = 0;
    bool any_in = false, all_in = true, none_out = true;
    for (int w = 0; w < words; ++w) {
      const uint32_t v = m[w], in = masks.in(w);
      d += __popc(v);
      any_in |= (v & in) != 0;
      all_in &= (v & in) == in;
      none_out &= (v & masks.out(w)) == 0;
    }
    bool ok = true;
    if (use_lut) ok = (masks.lut_word(d >> 5) >> (d & 31)) & 1u;
    if (pos_mode == 1) ok = ok && any_in && none_out;
    else if (pos_mode == 2) ok = ok && all_in && none_out;
    else if (pos_mode == 3) ok = ok && !any_in;
    flag[n] = ok ? 1 : 0;
  }
}

// SHARED: per-block bins in shared memory, flushed with one global atomic per non-empty bin; rows too
// long for the bins to fit in shared memory count straight into `hist`.
template <bool SHARED>
__global__ void distance_hist_kernel(const uint32_t* __restrict__ mut, long long N, int words, long long* __restrict__ hist,
                                     int bins) {
  extern __shared__ unsigned sh[];
  if (SHARED) {
    for (int i = threadIdx.x; i < bins; i += blockDim.x) sh[i] = 0;
    __syncthreads();
  }
  for (long long n = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; n < N;
       n += static_cast<long long>(gridDim.x) * blockDim.x) {
    int d = 0;
    for (int w = 0; w < words; ++w) d += __popc(mut[static_cast<size_t>(n) * words + w]);
    if (SHARED) atomicAdd(&sh[d], 1u);
    else atomicAdd(reinterpret_cast<unsigned long long*>(hist + d), 1ull);
  }
  if (SHARED) {
    __syncthreads();
    for (int i = threadIdx.x; i < bins; i += blockDim.x)
      if (sh[i]) atomicAdd(reinterpret_cast<unsigned long long*>(hist + i), static_cast<unsigned long long>(sh[i]));
  }
}

// Informative columns.  A thread walks the table with a stride that is a multiple of the row length,
// so it always meets the same (plane, word) position: one register accumulator of x ^ row 0, OR-ed
// per block in shared memory, then one global atomic per position and block (skipped when the bits
// are already there).  HBM-bound: reads the table once.
template <typename V>
__device__ __forceinline__ void or_into(uint32_t* dst, const V& v);
template <>
__device__ __forceinline__ void or_into<uint32_t>(uint32_t* dst, const uint32_t& v) {
  if (v) atomicOr(dst, v);
}
template <>
__device__ __forceinline__ void or_into<uint4>(uint32_t* dst, const uint4& v) {
  if (v.x) atomicOr(dst + 0, v.x);
  if (v.y) atomicOr(dst + 1, v.y);
  if (v.z) atomicOr(dst + 2, v.z);
  if (v.w) atomicOr(dst + 3, v.w);
}
__device__ __forceinline__ uint32_t xor_or(uint32_t acc, uint32_t a, uint32_t b) { return acc | (a ^ b); }
__device__ __forceinline__ uint4 xor_or(uint4 acc, uint4 a, uint4 b) {
  return make_uint4(acc.x | (a.x ^ b.x), acc.y | (a.y ^ b.y), acc.z | (a.z ^ b.z), acc.w | (a.w ^ b.w));
}

template <typename V>
__global__ void __launch_bounds__(256) varying_columns_kernel(const V* __restrict__ table, long long total, int row_elems,
                                                              long long stride, uint32_t* __restrict__ varying) {
  extern __shared__ uint32_t sh_var[];                       // [row_elems * words per V]
  constexpr int VW = sizeof(V) / 4;
  for (int i = threadIdx.x; i < row_elems * VW; i += blockDim.x) sh_var[i] = 0;
  __syncthreads();
  const long long g = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (g < stride) {
    const int pos = static_cast<int>(g % row_elems);
    const V ref = __ldg(table + pos);
    V acc = {};
    for (long long e = g; e < total; e += stride) acc = xor_or(acc, __ldcs(table + e), ref);
    or_into<V>(sh_var + pos * VW, acc);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < row_elems * VW; i += blockDim.x) {
    const uint32_t v = sh_var[i];
    if (v && (__ldcg(varying + i) & v) != v) atomicOr(varying + i, v);
  }
}

// One thread per (row, output word): bit b of every plane comes from source column cols[32*w2 + b].
template <int P>
__global__ void __launch_bounds__(256) compact_columns_kernel(const uint32_t* __restrict__ table, long long N,
                                                              long long rows_padded, int words,
                                                              const int* __restrict__ cols, uint32_t* __restrict__ out,
                                                              int out_words) {
  extern __shared__ int sh_cols[];                           // [out_words * 32]
  for (int i = threadIdx.x; i < out_words * 32; i += blockDim.x) sh_cols[i] = __ldg(cols + i);
  __syncthreads();
  const long long total = rows_padded * out_words;
  const int wshift = pow2_shift(out_words);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    long long n;
    int w2;
    split_index(i, out_words, wshift, &n, &w2);
    uint32_t acc[P];
#pragma unroll
    for (int p = 0; p < P; ++p) acc[p] = 0;
    if (n < N) {
      const uint32_t* row = table + static_cast<size_t>(n) * P * words;
      for (int b = 0; b < 32; ++b) {
        const int c = sh_cols[w2 * 32 + b];
        if (c < 0) continue;
        const int sw = c >> 5, sb = c & 31;
#pragma unroll
        for (int p = 0; p < P; ++p) acc[p] |= ((__ldg(row + p * words + sw) >> sb) & 1u) << b;
      }
    }
    uint32_t* dst = out + static_cast<size_t>(n) * P * out_words + w2;
#pragma unroll
    for (int p = 0; p < P; ++p) dst[p * out_words] = acc[p];
  }
}

struct AcceptVec { uint8_t a[1024]; };

__global__ void flags_or_rows_kernel(const uint8_t* __restrict__ flags, int rows, long long N, long long ld, AcceptVec acc,
                                     uint8_t* __restrict__ covered) {
  for (long long n = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; n < N;
       n += static_cast<long long>(gridDim.x) * blockDim.x) {
    uint8_t c = covered[n];
    for (int r = 0; r < rows; ++r)
      if (acc.a[r]) c |= flags[static_cast<size_t>(r) * ld + n];
    covered[n] = c;
  }
}

static unsigned grid_for(long long work, int threads) {
  long long b = ceil_div(work, threads);
  const long long cap = static_cast<long long>(num_sms()) * 16;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return static_cast<unsigned>(b);
}

}  // namespace pg

using namespace pg;

extern "C" {

int pg_mutant_bits(const uint32_t* table, int64_t N, int planes, int words, const uint32_t* ref, uint32_t* mut,
                   void* stream) {
  PG_CHECK_ARG(table && ref && mut && N > 0 && planes > 0 && words > 0, "bad arguments");
  mutant_bits_kernel<<<grid_for(N * words, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(table, N, planes, words,
                                                                                             ref, mut);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

int pg_mutant_bool(const uint32_t* table, int64_t N, int planes, int words, int L, const uint32_t* ref, uint8_t* out,
                   void* stream) {
  PG_CHECK_ARG(table && ref && out && N > 0 && planes > 0 && words > 0 && L > 0 && L <= words * 32, "bad arguments");
  // two items per thread: 107.7 us at 1 M x 256 (3.86 TB/s); one: 112.1 us, four: 140.4 us (profiles/r4c_mb.log)
  const unsigned grid = grid_for(ceil_div(N * words * 2, 2ll), 256);
  mutant_bool_kernel<2><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(table, N, planes, words, L, ref, out);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

int pg_flags_or_rows(const uint8_t* flags, int64_t rows, int64_t N, int64_t ld, const uint8_t* accept_host,
                     uint8_t* covered, void* stream) {
  PG_CHECK_ARG(flags && accept_host && covered && N > 0 && ld >= N, "bad arguments");
  PG_CHECK_ARG(rows >= 1 && rows <= 1024, "at most 1024 flag rows per call");
  AcceptVec acc;
  memset(&acc, 0, sizeof(acc));
  memcpy(acc.a, accept_host, static_cast<size_t>(rows));
  flags_or_rows_kernel<<<grid_for(N, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(flags, static_cast<int>(rows), N, ld,
                                                                                        acc, covered);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

int pg_mutant_any(const uint32_t* mut, int64_t N, int words, uint32_t* any_bits, void* stream) {
  PG_CHECK_ARG(mut && any_bits && N > 0 && words > 0, "bad arguments");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PG_CUDA(cudaMemsetAsync(any_bits, 0, sizeof(uint32_t) * words, s));
  mutant_any_kernel<<<grid_for(N, 256), 256, 0, s>>>(mut, N, words, any_bits);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

int pg_varying_columns(const uint32_t* table, int64_t N, int planes, int words, uint32_t* varying, void* stream) {
  PG_CHECK_ARG(table && varying && N > 0 && planes > 0 && words > 0, "bad arguments");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int row_words = planes * words;
  PG_CUDA(cudaMemsetAsync(varying, 0, sizeof(uint32_t) * row_words, s));
  const bool vec = row_words % 4 == 0 && reinterpret_cast<uintptr_t>(table) % 16 == 0;
  const int row_elems = vec ? row_words / 4 : row_words;
  const long long total = static_cast<long long>(N) * row_elems;
  long long threads = static_cast<long long>(num_sms()) * 8 * 256;
  if (threads > total) threads = total;
  const long long stride = max(1ll, threads / row_elems) * row_elems;      // a multiple of the row length
  const unsigned grid = static_cast<unsigned>(ceil_div(stride, 256));
  const size_t smem = sizeof(uint32_t) * row_words;
  if (smem > 48 * 1024) {       // one word per (plane, word) position: more than the default dynamic shared memory
    PG_CUDA(cudaFuncSetAttribute(vec ? reinterpret_cast<const void*>(varying_columns_kernel<uint4>)
                                     : reinterpret_cast<const void*>(varying_columns_kernel<uint32_t>),
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  }
  if (vec)
    varying_columns_kernel<uint4><<<grid, 256, smem, s>>>(reinterpret_cast<const uint4*>(table), total, row_elems, stride,
                                                         varying);
  else
    varying_columns_kernel<uint32_t><<<grid, 256, smem, s>>>(table, total, row_elems, stride, varying);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

int pg_compact_columns(const uint32_t* table, int64_t N, int planes, int words, const int32_t* cols, uint32_t* out,
                       int out_words, void* stream) {
  PG_CHECK_ARG(table && cols && out && N > 0 && words > 0, "bad arguments");
  PG_CHECK_ARG(out_words > 0 && (out_words & (out_words - 1)) == 0 || out_words % 8 == 0, "out_words must come from pg_packed_words");
  PG_CHECK_ARG(out_words <= 1024, "out_words too large");
  const long long rows_padded = pg_packed_rows(N);
  const size_t smem = sizeof(int) * out_words * 32;
  const unsigned grid = grid_for(rows_padded * out_words, 256);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (smem > 48 * 1024 && (planes == 5 || planes == 8)) {    // more than 384 output words: up to 128 KB
    PG_CUDA(cudaFuncSetAttribute(planes == 5 ? reinterpret_cast<const void*>(compact_columns_kernel<5>)
                                             : reinterpret_cast<const void*>(compact_columns_kernel<8>),
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  }
  if (planes == 5)
    compact_columns_kernel<5><<<grid, 256, smem, s>>>(table, N, rows_padded, words, cols, out, out_words);
  else if (planes == 8)
    compact_columns_kernel<8><<<grid, 256, smem, s>>>(table, N, rows_padded, words, cols, out, out_words);
  else {
    set_error("pg_compact_columns supports 5 or 8 planes, got %d", planes);
    return PG_ERR_UNSUPPORTED;
  }
  PG_LAUNCH_CHECK();
  return PG_OK;
}

int pg_select_rows(const uint32_t* mut, int64_t N, int words, const uint32_t* dist_lut_host, int lut_words,
                   const uint32_t* inside_host, const uint32_t* outside_host, int pos_mode, uint8_t* flag,
                   void* stream) {
  PG_CHECK_ARG(mut && flag && N > 0 && words > 0, "bad arguments");
  PG_CHECK_ARG(pos_mode >= 0 && pos_mode <= 3, "bad pos_mode %d", pos_mode);
  PG_CHECK_ARG(pos_mode == 0 || inside_host, "positions mask missing");
  PG_CHECK_ARG(!dist_lut_host || (lut_words >= 1 && lut_words <= words + 1 && lut_words * 32 > words * 32),
               "distance lut must cover 0..%d", words * 32);
  PG_CHECK_ARG(!(pos_mode == 1 || pos_mode == 2) || outside_host, "unchanged-positions mask missing");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int use_lut = dist_lut_host ? 1 : 0;
  if (words <= kMaxMaskWords) {
    ParamMasks m;
    memset(&m, 0, sizeof(m));
    if (outside_host) memcpy(m.outside.w, outside_host, sizeof(uint32_t) * words);
    if (dist_lut_host) memcpy(m.lut.w, dist_lut_host, sizeof(uint32_t) * lut_words);
    if (inside_host) memcpy(m.inside.w, inside_host, sizeof(uint32_t) * words);
    select_rows_kernel<ParamMasks><<<grid_for(N, 256), 256, 0, s>>>(mut, N, words, m, use_lut, pos_mode, flag);
    PG_LAUNCH_CHECK();
    return PG_OK;
  }
  // rows longer than 32 * kMaxMaskWords residues: the masks go through a device buffer
  std::vector<uint32_t> host(static_cast<size_t>(3 * words + 1), 0u);
  if (inside_host) memcpy(host.data(), inside_host, sizeof(uint32_t) * words);
  if (outside_host) memcpy(host.data() + words, outside_host, sizeof(uint32_t) * words);
  if (dist_lut_host) memcpy(host.data() + 2 * words, dist_lut_host, sizeof(uint32_t) * lut_words);
  void* buf = nullptr;
  PG_CUDA(temp_alloc(&buf, sizeof(uint32_t) * host.size(), s));
  cudaError_t e = cudaMemcpyAsync(buf, host.data(), sizeof(uint32_t) * host.size(), cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) {
    BufferMasks m{static_cast<const uint32_t*>(buf), words};
    select_rows_kernel<BufferMasks><<<grid_for(N, 256), 256, 0, s>>>(mut, N, words, m, use_lut, pos_mode, flag);
    count_launch();
    e = cudaGetLastError();
  }
  cudaFreeAsync(buf, s);
  if (e != cudaSuccess) { set_error("select rows failed: %s", cudaGetErrorString(e)); return PG_ERR_CUDA; }
  return PG_OK;
}

int pg_flag_indices(const uint8_t* flag, int64_t N, int64_t* out_idx, int64_t* count_out, void* stream) {
  PG_CHECK_ARG(flag && out_idx && count_out && N > 0 && N < (1ll << 31), "bad arguments");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  thrust::counting_iterator<long long> ids(0);
  size_t tmp_bytes = 0;
  PG_CUDA(cub::DeviceSelect::Flagged(nullptr, tmp_bytes, ids, flag, reinterpret_cast<long long*>(out_idx),
                                     reinterpret_cast<long long*>(count_out), static_cast<int>(N), s));
  void* tmp = nullptr;
  PG_CUDA(temp_alloc(&tmp, tmp_bytes, s));
  cudaError_t e = cub::DeviceSelect::Flagged(tmp, tmp_bytes, ids, flag, reinterpret_cast<long long*>(out_idx),
                                             reinterpret_cast<long long*>(count_out), static_cast<int>(N), s);
  count_launch();
  cudaFreeAsync(tmp, s);
  if (e != cudaSuccess) { set_error("cub select failed: %s", cudaGetErrorString(e)); return PG_ERR_CUDA; }
  return PG_OK;
}

int pg_distance_hist(const uint32_t* mut, int64_t N, int words, int64_t* hist, void* stream) {
  PG_CHECK_ARG(mut && hist && N > 0 && words > 0, "bad arguments");
  const int bins = words * 32 + 1;
  const size_t smem = static_cast<size_t>(bins) * sizeof(unsigned);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (smem > 227 * 1024) {      // rows of more than 58 111 residues
    distance_hist_kernel<false><<<grid_for(N, 256), 256, 0, s>>>(mut, N, words, reinterpret_cast<long long*>(hist), bins);
    PG_LAUNCH_CHECK();
    return PG_OK;
  }
  // bins of rows longer than 12 288 residues exceed the default 48 KB of dynamic shared memory
  if (smem > 48 * 1024)
    PG_CUDA(cudaFuncSetAttribute(distance_hist_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(smem)));
  distance_hist_kernel<true><<<grid_for(N, 256), 256, smem, s>>>(mut, N, words, reinterpret_cast<long long*>(hist), bins);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

}  // extern "C"
