// Element-wise metric tiles and the consumers of a materialised (rows x N) distance tile.
//
//   pg_minkowski_tile        minkowski.py:36-40 with the reference's rounding chain
//   pg_hamming_values_tile   hamming.py:34 on arbitrary numeric values
//   pg_tile_topk             prograph.py:757-762 (stable sort + slice) as select-then-sort
//   pg_tile_threshold_*      prograph.py:734-739 / :544 (where + gather) as ballot +
//                            block prefix-sum compaction
#include <math_constants.h>
#include <cub/device/device_radix_sort.cuh>

#include <type_traits>

#include "pg_common.cuh"

namespace pg {

// =============================================================================
// Element-wise tiles
// =============================================================================
enum ValKind { VK_F16 = 0, VK_F32 = 1, VK_F64 = 2, VK_I64 = 3 };
enum PowKind { PK_ONE = 0, PK_TWO = 1, PK_THREE = 2, PK_SQRT = 3, PK_GENERAL = 4 };

__device__ __forceinline__ float rh(float x) { return __half2float(__float2half_rn(x)); }  // round through fp16

template <int PK>
__device__ __forceinline__ float pow_f32(float x, float e) {
  if (PK == PK_ONE) return x;
  if (PK == PK_TWO) return x * x;
  if (PK == PK_THREE) return (x * x) * x;
  if (PK == PK_SQRT) return sqrtf(x);
  return powf(x, e);
}
// fp16 tensor ** scalar: every multiply of the optimised exponents rounds to fp16
template <int PK>
__device__ __forceinline__ float pow_f16(float x, float e) {
  if (PK == PK_ONE) return x;
  if (PK == PK_TWO) return rh(x * x);
  if (PK == PK_THREE) return rh(rh(x * x) * x);
  if (PK == PK_SQRT) return rh(sqrtf(x));
  return rh(powf(x, e));
}
template <int PK>
__device__ __forceinline__ double pow_f64(double x, double e) {
  if (PK == PK_ONE) return x;
  if (PK == PK_TWO) return x * x;
  if (PK == PK_THREE) return (x * x) * x;
  if (PK == PK_SQRT) return sqrt(x);
  return pow(x, e);
}
__device__ __forceinline__ long long ipow(long long b, int e) {  // wraps like torch's integer pow
  long long r = 1;
  while (e > 0) {
    if (e & 1) r *= b;
    b *= b;
    e >>= 1;
  }
  return r;
}

static int pow_kind(double e) {
  if (e == 1.0) return PK_ONE;
  if (e == 2.0) return PK_TWO;
  if (e == 3.0) return PK_THREE;
  if (e == 0.5) return PK_SQRT;
  return PK_GENERAL;
}

template <typename T> struct Compute { using type = float; };
template <> struct Compute<double> { using type = double; };
template <> struct Compute<long long> { using type = long long; };

template <typename T> __device__ __forceinline__ typename Compute<T>::type load_val(const T* p) { return *p; }
template <> __device__ __forceinline__ float load_val<__half>(const __half* p) { return __half2float(*p); }

constexpr int ET_N = 128;  // dataset rows per CTA
constexpr int ET_M = 64;   // query rows per CTA
constexpr int ET_D = 16;   // components per staging chunk
constexpr int ET_NPT = 4;  // dataset rows per thread (consecutive: one 128-bit shared-memory load for 4-byte types)
constexpr int ET_MPT = 8;  // queries per thread (the same for all lanes of a warp: broadcast loads)

struct ElemParams {
  const void* X; long long N;
  const void* Y; long long q0, qrows;
  int D;
  void* out; long long ld;
  float p_f, root_f;     // exponents as the tensor dtype sees them (fp16-rounded for VK_F16)
  double p_d, root_d;
  int p_int;             // integer exponent for VK_I64
  int similarity;
  int weight;            // hamming-values output kind
  const int* only_if;    // optional device flag: run only when *only_if != 0 (the p = 1 rank-1 path declined)
};

// One term of the sum for a (dataset value x, query value y) pair, in the accumulator's type.
template <typename CT, int VK, int METRIC, int PKIN>
__device__ __forceinline__ CT elem_term(CT x, CT y, const ElemParams& prm) {
  if constexpr (METRIC == 1) {
    return (x != y) ? CT(1) : CT(0);
  } else if constexpr (VK == VK_F16) {
    return pow_f16<PKIN>(rh(x - y), prm.p_f);
  } else if constexpr (VK == VK_F32) {
    return pow_f32<PKIN>(x - y, prm.p_f);
  } else if constexpr (VK == VK_F64) {
    return pow_f64<PKIN>(x - y, prm.p_d);
  } else {
    const long long d = x - y;
    if constexpr (PKIN == PK_ONE) return d;
    else if constexpr (PKIN == PK_TWO) return d * d;
    else if constexpr (PKIN == PK_THREE) return (d * d) * d;
    else return ipow(d, prm.p_int);
  }
}

// METRIC 0: minkowski, 1: hamming on values.  A 256-thread CTA computes a 128 (dataset rows) x 64
// (queries) block; a thread owns 4 consecutive dataset rows x 8 queries = 32 running sums in
// registers.  The operands are staged through shared memory component-major (Xs[c][row]): per
// component a thread reads its 4 dataset values with one vector load and the 8 query values with
// broadcast loads -- 3 loads for 32 terms (the first version read 9 scalars for 8 terms).  Every pair
// still adds its terms in ascending component order, so the rounding chain of minkowski.py:36-40 is
// untouched.
template <typename T, int VK, int METRIC, int PKIN, int PKROOT>
__global__ void __launch_bounds__(256) elem_tile_kernel(const ElemParams prm) {
  using CT = typename Compute<T>::type;
  // the accumulator type: fp32 for f16 / f32 sums, double for f64, int64 for integer inputs / counts
  using AT = typename std::conditional<METRIC == 1, long long, CT>::type;
  // fp16 rows with one of the multiply-only exponents run their per-element chain in native half2
  // arithmetic: fp16 subtract / multiply round exactly like "compute in fp32, round to fp16" (the
  // reference's chain; double rounding through a format of >= 2p+2 bits is innocuous), two pairs per
  // instruction, no conversion round trips.  The running sum stays fp32, as torch.sum keeps it.
  constexpr bool HALF2 = VK == VK_F16 && METRIC == 0 && (PKIN == PK_ONE || PKIN == PK_TWO || PKIN == PK_THREE);
  using ST = typename std::conditional<HALF2, __half, CT>::type;      // staging type in shared memory
  __shared__ __align__(16) ST Xs[ET_D][ET_N];
  __shared__ __align__(16) ST Ys[ET_D][ET_M];
  const T* X = static_cast<const T*>(prm.X);
  const T* Y = static_cast<const T*>(prm.Y);
  const int tid = threadIdx.x;
  const int tx = tid & 31;   // lanes: dataset rows 4*tx .. 4*tx+3
  const int ty = tid >> 5;   // warps: queries 8*ty .. 8*ty+7
  const long long n0 = static_cast<long long>(blockIdx.x) * ET_N;
  const long long m0 = static_cast<long long>(blockIdx.y) * ET_M;
  if (prm.only_if != nullptr && *prm.only_if == 0) return;

  AT acc[ET_MPT][ET_NPT];
#pragma unroll
  for (int i = 0; i < ET_MPT; ++i)
#pragma unroll
    for (int j = 0; j < ET_NPT; ++j) acc[i][j] = AT(0);

  for (int d0 = 0; d0 < prm.D; d0 += ET_D) {
    // stage: thread (row = tid % 128, half = tid / 128) reads 8 consecutive components of one dataset
    // row; thread (q = tid % 64, quarter = tid / 64) reads 4 consecutive components of one query row
    {
      const int r = tid & (ET_N - 1), c0 = (tid >> 7) * 8;
      const long long n = n0 + r;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int c = c0 + k;
        ST v = ST(0);
        if (n < prm.N && d0 + c < prm.D) {
          if constexpr (HALF2) v = X[static_cast<size_t>(n) * prm.D + d0 + c];
          else v = load_val<T>(X + static_cast<size_t>(n) * prm.D + d0 + c);
        }
        Xs[c][r] = v;
      }
      const int q = tid & (ET_M - 1), qc0 = (tid >> 6) * 4;
      const long long m = m0 + q;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int c = qc0 + k;
        ST v = ST(0);
        if (m < prm.qrows && d0 + c < prm.D) {
          if constexpr (HALF2) v = Y[static_cast<size_t>(prm.q0 + m) * prm.D + d0 + c];
          else v = load_val<T>(Y + static_cast<size_t>(prm.q0 + m) * prm.D + d0 + c);
        }
        Ys[c][q] = v;
      }
    }
    __syncthreads();
    const int dn = min(ET_D, prm.D - d0);
    for (int c = 0; c < dn; ++c) {
      if constexpr (HALF2) {
        const __half2 x01 = *reinterpret_cast<const __half2*>(&Xs[c][tx * ET_NPT]);
        const __half2 x23 = *reinterpret_cast<const __half2*>(&Xs[c][tx * ET_NPT + 2]);
#pragma unroll
        for (int i = 0; i < ET_MPT; ++i) {
          const __half2 yy = __half2half2(Ys[c][ty * ET_MPT + i]);
          __half2 a = __hsub2(x01, yy), b = __hsub2(x23, yy);
          if (PKIN == PK_TWO) { a = __hmul2(a, a); b = __hmul2(b, b); }
          if (PKIN == PK_THREE) { a = __hmul2(__hmul2(a, a), a); b = __hmul2(__hmul2(b, b), b); }
          const float2 fa = __half22float2(a), fb = __half22float2(b);
          acc[i][0] += fa.x; acc[i][1] += fa.y; acc[i][2] += fb.x; acc[i][3] += fb.y;
        }
      } else {
        CT x[ET_NPT], y[ET_MPT];
#pragma unroll
        for (int j = 0; j < ET_NPT; ++j) x[j] = Xs[c][tx * ET_NPT + j];
#pragma unroll
        for (int i = 0; i < ET_MPT; ++i) y[i] = Ys[c][ty * ET_MPT + i];
#pragma unroll
        for (int i = 0; i < ET_MPT; ++i)
#pragma unroll
          for (int j = 0; j < ET_NPT; ++j)
            acc[i][j] += static_cast<AT>(elem_term<CT, VK, METRIC, PKIN>(x[j], y[i], prm));
      }
    }
    __syncthreads();
  }

#pragma unroll
  for (int i = 0; i < ET_MPT; ++i) {
    const long long m = m0 + ty * ET_MPT + i;
    if (m >= prm.qrows) continue;
#pragma unroll
    for (int j = 0; j < ET_NPT; ++j) {
      const long long n = n0 + tx * ET_NPT + j;
      if (n >= prm.N) continue;
      const size_t at = static_cast<size_t>(m) * prm.ld + n;
      if constexpr (METRIC == 1) {
        if (prm.weight == PG_W_I64) static_cast<long long*>(prm.out)[at] = acc[i][j];
        else if (prm.weight == PG_W_SIM_F32) static_cast<float*>(prm.out)[at] = sim_f32(static_cast<int>(acc[i][j]));
        else static_cast<int*>(prm.out)[at] = static_cast<int>(acc[i][j]);
      } else if constexpr (VK == VK_F16) {
        float d = pow_f16<PKROOT>(rh(acc[i][j]), prm.root_f);
        if (prm.similarity) d = rh(__fdiv_rn(1.0f, rh(1.0f + d)));
        static_cast<__half*>(prm.out)[at] = __float2half_rn(d);
      } else if constexpr (VK == VK_F32 || VK == VK_I64) {
        const float sum = static_cast<float>(acc[i][j]);
        float d = pow_f32<PKROOT>(sum, prm.root_f);
        if (prm.similarity) d = __fdiv_rn(1.0f, 1.0f + d);
        static_cast<float*>(prm.out)[at] = d;
      } else {
        double d = pow_f64<PKROOT>(acc[i][j], prm.root_d);
        if (prm.similarity) d = 1.0 / (1.0 + d);
        static_cast<double*>(prm.out)[at] = d;
      }
    }
  }
}

// bytes of one output entry of elem_tile_kernel
template <typename T, int VK, int METRIC>
static size_t elem_out_bytes(const ElemParams& prm) {
  if (METRIC == 1) return prm.weight == PG_W_I64 ? 8 : 4;
  if (VK == VK_F16) return 2;
  if (VK == VK_F64) return 8;
  return 4;                                       // float32 out for f32 and int64 inputs
}

template <typename T, int VK, int METRIC>
static int launch_elem(const ElemParams& prm, int pk_in, int pk_root, cudaStream_t s) {
  // query blocks go on gridDim.y (at most 65535): larger tiles are launched in chunks of query rows
  constexpr long long kChunk = 65535ll * ET_M;
  const size_t row_bytes = static_cast<size_t>(prm.ld) * elem_out_bytes<T, VK, METRIC>(prm);
  for (long long c0 = 0; c0 < prm.qrows; c0 += kChunk) {
    ElemParams part = prm;
    part.q0 = prm.q0 + c0;
    part.qrows = std::min(kChunk, prm.qrows - c0);
    part.out = static_cast<char*>(prm.out) + static_cast<size_t>(c0) * row_bytes;
    dim3 grid(static_cast<unsigned>(ceil_div(part.N, ET_N)), static_cast<unsigned>(ceil_div(part.qrows, ET_M)));
#define PG_EL(PI, PR) elem_tile_kernel<T, VK, METRIC, PI, PR><<<grid, 256, 0, s>>>(part)
    if (METRIC == 1) {
      PG_EL(PK_ONE, PK_ONE);
    } else {
      // the common pairs get their own instantiation; everything else takes the powf path
      if (pk_in == PK_TWO && pk_root == PK_SQRT) PG_EL(PK_TWO, PK_SQRT);
      else if (pk_in == PK_ONE && pk_root == PK_ONE) PG_EL(PK_ONE, PK_ONE);
      else if (pk_in == PK_THREE) PG_EL(PK_THREE, PK_GENERAL);
      else if (pk_in == PK_SQRT && pk_root == PK_TWO) PG_EL(PK_SQRT, PK_TWO);
      else PG_EL(PK_GENERAL, PK_GENERAL);
    }
#undef PG_EL
    PG_LAUNCH_CHECK();
  }
  return PG_OK;
}

// =============================================================================
// Minkowski p = 1: a rank-1 difference
// =============================================================================
// The reference takes no absolute value (minkowski.py:36): for p = 1 the "distance" is
//   pow(sum(x - y), 1) = sum(x) - sum(y).
// In int64 arithmetic that identity always holds (wrap-around included); in fp16 / float32 it holds
// bit for bit when every value is an integer of magnitude <= 255 and D * 510 < 2^24 (each difference,
// and the fp32 running sum, are then exact).  So: one pass of row sums (+ a validity flag for the
// float types) and an outer difference written at HBM speed instead of an O(N * M * D) kernel; when the
// flag says the rows are not small integers, the element-wise kernel runs instead (both are
// launched, each looks at the flag: no host round trip).
template <typename T>
__global__ void row_sums_kernel(const T* __restrict__ X, long long row0, long long rows, int D, long long* __restrict__ sums,
                                int* __restrict__ flag) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
  const long long nwarps = (gridDim.x * static_cast<long long>(blockDim.x)) >> 5;
  for (long long r = warp0; r < rows; r += nwarps) {
    const T* src = X + static_cast<size_t>(row0 + r) * D;
    long long acc = 0;
    bool bad = false;
    for (int c = lane; c < D; c += 32) {
      if constexpr (sizeof(T) == 8) {          // int64
        acc += static_cast<long long>(src[c]);
      } else {
        const float v = static_cast<float>(load_val<T>(src + c));
        bad |= !(v == truncf(v) && fabsf(v) <= 255.0f);
        acc += static_cast<long long>(v);
      }
    }
    acc = warp_sum(acc);
    if (__any_sync(0xffffffffu, bad) && lane == 0) atomicExch(flag, 1);
    if (lane == 0) sums[r] = acc;
  }
}

template <int VK>
__global__ void __launch_bounds__(256) mink1_tile_kernel(const long long* __restrict__ sx, long long N,
                                                         const long long* __restrict__ sy, long long qrows, int similarity,
                                                         void* out, long long ld, const int* __restrict__ flag) {
  if (*flag != 0) return;
  const long long n = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (n >= N) return;
  const long long x = sx[n];
  const long long m_end = min(qrows, (static_cast<long long>(blockIdx.y) + 1) * 8);
  for (long long m = static_cast<long long>(blockIdx.y) * 8; m < m_end; ++m) {
    const long long S = x - __ldg(sy + m);
    const size_t at = static_cast<size_t>(m) * ld + n;
    if (VK == VK_F16) {
      float d = rh(static_cast<float>(S));
      if (similarity) d = rh(__fdiv_rn(1.0f, rh(1.0f + d)));
      static_cast<__half*>(out)[at] = __float2half_rn(d);
    } else {
      float d = static_cast<float>(S);
      if (similarity) d = __fdiv_rn(1.0f, 1.0f + d);
      static_cast<float*>(out)[at] = d;
    }
  }
}

// Row sums + the rank-1 tile; returns the scratch block (to be freed on the stream by the caller,
// after the element-wise kernel that may follow) and the device flag that kernel has to look at.
template <typename T, int VK>
static int launch_mink1(const T* X, long long N, const T* Y, long long q0, long long qrows, int D, int similarity, void* out,
                        long long ld, void** scratch, int** flag_dev, cudaStream_t s) {
  void* tmp = nullptr;
  PG_CUDA(temp_alloc(&tmp, static_cast<size_t>(N + qrows) * 8 + 16, s));
  *scratch = tmp;
  long long* sx = static_cast<long long*>(tmp);
  long long* sy = sx + N;
  int* flag = reinterpret_cast<int*>(sy + qrows);
  *flag_dev = flag;
  PG_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), s));
  const int threads = 256;
  const long long cap = static_cast<long long>(num_sms()) * 16;
  row_sums_kernel<T><<<static_cast<unsigned>(std::min<long long>(cap, ceil_div(N * 32, threads))), threads, 0, s>>>(
      X, 0, N, D, sx, flag);
  PG_LAUNCH_CHECK();
  row_sums_kernel<T><<<static_cast<unsigned>(std::min<long long>(cap, ceil_div(qrows * 32, threads))), threads, 0, s>>>(
      Y, q0, qrows, D, sy, flag);
  PG_LAUNCH_CHECK();
  dim3 grid(static_cast<unsigned>(ceil_div(N, threads)), static_cast<unsigned>(ceil_div(qrows, 8)));
  mink1_tile_kernel<VK><<<grid, threads, 0, s>>>(sx, N, sy, qrows, similarity, out, ld, flag);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

// =============================================================================
// Ordered keys (torch.sort order: ascending, NaN last, -0 == +0)
// =============================================================================
__device__ __forceinline__ uint32_t key_f32(float v) {
  if (v != v) return 0xffffffffu;
  if (v == 0.0f) v = 0.0f;
  const uint32_t b = __float_as_uint(v);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ unsigned long long key_f64(double v) {
  if (v != v) return ~0ull;
  if (v == 0.0) v = 0.0;
  const unsigned long long b = static_cast<unsigned long long>(__double_as_longlong(v));
  return (b >> 63) ? ~b : (b | (1ull << 63));
}
template <typename T> struct KeyOf;
template <> struct KeyOf<__half> { using K = uint32_t; __device__ static K get(__half v) { return key_f32(__half2float(v)); } };
template <> struct KeyOf<float> { using K = uint32_t; __device__ static K get(float v) { return key_f32(v); } };
template <> struct KeyOf<int> { using K = uint32_t; __device__ static K get(int v) { return static_cast<uint32_t>(v) ^ 0x80000000u; } };
template <> struct KeyOf<double> { using K = unsigned long long; __device__ static K get(double v) { return key_f64(v); } };
template <> struct KeyOf<long long> {
  using K = unsigned long long;
  __device__ static K get(long long v) { return static_cast<unsigned long long>(v) ^ (1ull << 63); }
};

// =============================================================================
// Stable top-k of each row: radix-select the k1-th key, gather, bitonic sort (key, idx)
// =============================================================================
constexpr int TK_THREADS = 256;

template <typename T>
__global__ void __launch_bounds__(TK_THREADS) tile_topk_kernel(const T* __restrict__ tile, long long N, long long ld,
                                                                int k, int drop, int descending,
                                                                long long* __restrict__ out_idx, T* __restrict__ out_val,
                                                                int cap /* pow2 >= k1 */) {
  using K = typename KeyOf<T>::K;
  constexpr int KBITS = sizeof(K) * 8;
  extern __shared__ __align__(16) unsigned char tk_smem[];
  K* skey = reinterpret_cast<K*>(tk_smem);                                  // [cap]
  uint32_t* sidx = reinterpret_cast<uint32_t*>(tk_smem + sizeof(K) * cap);   // [cap]
  __shared__ unsigned hist[256];
  __shared__ K s_prefix;
  __shared__ long long s_want;
  __shared__ int s_less, s_eq_taken;
  __shared__ int s_warp_cnt[TK_THREADS / 32];

  const long long row = blockIdx.x;
  const T* src = tile + static_cast<size_t>(row) * ld;
  const int tid = threadIdx.x;
  long long k1 = static_cast<long long>(drop) + k;
  if (k1 > N) k1 = N;
  const K flip = descending ? ~K(0) : K(0);

  // ---- radix select: the key of rank k1 (1-based) -------------------------------------
  if (tid == 0) { s_prefix = 0; s_want = k1; }
  __syncthreads();
  for (int shift = KBITS - 8; shift >= 0; shift -= 8) {
    hist[tid] = 0;
    __syncthreads();
    const K prefix = s_prefix;
    for (long long i = tid; i < N; i += TK_THREADS) {
      const K key = KeyOf<T>::get(src[i]) ^ flip;
      const bool match = (shift == KBITS - 8) || ((key >> (shift + 8)) == (prefix >> (shift + 8)));
      if (match) atomicAdd(&hist[static_cast<unsigned>(key >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (tid == 0) {
      long long want = s_want;
      int dgt = 0;
      for (; dgt < 256; ++dgt) {
        if (want <= hist[dgt]) break;
        want -= hist[dgt];
      }
      s_want = want;
      s_prefix = prefix | (static_cast<K>(dgt) << shift);
    }
    __syncthreads();
  }
  const K kth = s_prefix;
  const int need_eq = static_cast<int>(s_want);      // entries equal to kth to take, lowest indices first
  const int n_less = static_cast<int>(k1) - need_eq;  // entries strictly below kth

  // ---- gather ------------------------------------------------------------------------------
  for (int i = tid; i < cap; i += TK_THREADS) { skey[i] = ~K(0); sidx[i] = 0xffffffffu; }
  if (tid == 0) { s_less = 0; s_eq_taken = 0; }
  __syncthreads();
  const int lane = tid & 31, warp = tid >> 5;
  for (long long base = 0; base < N; base += TK_THREADS) {
    const long long i = base + tid;
    bool eq = false;
    if (i < N) {
      const K key = KeyOf<T>::get(src[i]) ^ flip;
      if (key < kth) {
        const int at = atomicAdd(&s_less, 1);
        skey[at] = key;
        sidx[at] = static_cast<uint32_t>(i);
      }
      eq = key == kth;
    }
    // ordered placement of the ties: ballot + block prefix sum
    const int taken = s_eq_taken;
    const unsigned bal = __ballot_sync(0xffffffffu, eq);
    if (lane == 0) s_warp_cnt[warp] = __popc(bal);
    __syncthreads();
    int before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < TK_THREADS / 32; ++w) {
      const int c = s_warp_cnt[w];
      if (w < warp) before += c;
      total += c;
    }
    if (eq) {
      const int pos = taken + before + __popc(bal & ((1u << lane) - 1u));
      if (pos < need_eq) {
        skey[n_less + pos] = kth;
        sidx[n_less + pos] = static_cast<uint32_t>(i);
      }
    }
    __syncthreads();
    if (tid == 0) s_eq_taken = taken + total;
    __syncthreads();
  }

  // ---- bitonic sort of (key, idx) ---------------------------------------------------------
  for (int size = 2; size <= cap; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = tid; i < cap / 2; i += TK_THREADS) {
        const int lo = (i / stride) * stride * 2 + (i % stride);
        const int hi = lo + stride;
        const bool up = ((lo & size) == 0);
        const K ka = skey[lo], kb = skey[hi];
        const uint32_t ia = sidx[lo], ib = sidx[hi];
        const bool a_gt_b = (ka > kb) || (ka == kb && ia > ib);
        if (a_gt_b == up) {
          skey[lo] = kb; skey[hi] = ka;
          sidx[lo] = ib; sidx[hi] = ia;
        }
      }
      __syncthreads();
    }
  }
  for (int j = tid; j < k; j += TK_THREADS) {
    const int src_pos = drop + j;
    const size_t at = static_cast<size_t>(row) * k + j;
    if (src_pos < k1) {
      const uint32_t ix = sidx[src_pos];
      out_idx[at] = ix;
      out_val[at] = src[ix];
    } else {
      out_idx[at] = -1;
      out_val[at] = T(0);
    }
  }
}

// =============================================================================
// Top-k of each row when k + drop exceeds the shared-memory sort: the reference sorts whole rows
// (prograph.py:757-762, any k).  Two stable device-wide radix sorts: (1) all entries of the tile by
// their order-preserving key, the value being the entry's position row*N + i -- equal keys keep
// ascending positions; (2) by row.  What comes out is every row in (key, index) order.
// =============================================================================
template <typename T>
__global__ void sort_keys_kernel(const T* __restrict__ tile, long long rows, long long N, long long ld, int descending,
                                 typename KeyOf<T>::K* __restrict__ keys, uint32_t* __restrict__ pos) {
  using K = typename KeyOf<T>::K;
  const K flip = descending ? ~K(0) : K(0);
  const long long total = rows * N;
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < total;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = e / N, i = e - r * N;
    keys[e] = KeyOf<T>::get(tile[static_cast<size_t>(r) * ld + i]) ^ flip;
    pos[e] = static_cast<uint32_t>(e);
  }
}

__global__ void sort_rows_of_kernel(const uint32_t* __restrict__ pos, long long total, unsigned N, uint32_t* __restrict__ row_of) {
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < total;
       e += static_cast<long long>(gridDim.x) * blockDim.x)
    row_of[e] = pos[e] / N;
}

template <typename T>
__global__ void sort_take_kernel(const T* __restrict__ tile, const uint32_t* __restrict__ pos, long long rows, long long N,
                                 long long ld, int k, int drop, long long* __restrict__ out_idx, T* __restrict__ out_val) {
  const long long total = rows * k;
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < total;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = e / k;
    const int j = static_cast<int>(e - r * k);
    if (drop + j < N) {
      const long long i = static_cast<long long>(pos[r * N + drop + j]) - r * N;
      out_idx[e] = i;
      out_val[e] = tile[static_cast<size_t>(r) * ld + i];
    } else {
      out_idx[e] = -1;
      out_val[e] = T(0);
    }
  }
}

template <typename T>
static int tile_topk_by_sort(const T* tile, long long rows, long long N, long long ld, int k, int drop, int descending,
                             long long* out_idx, T* out_val, cudaStream_t s) {
  using K = typename KeyOf<T>::K;
  const long long total = rows * N;
  if (total >= (1ll << 31)) { set_error("tile too large for one key sort: split the rows"); return PG_ERR_UNSUPPORTED; }
  const int n = static_cast<int>(total);
  K* keys = nullptr;
  uint32_t* pos = nullptr;
  uint32_t* rowk = nullptr;
  const size_t kbytes = round_up(sizeof(K) * static_cast<size_t>(n), size_t(256));
  const size_t pbytes = round_up(sizeof(uint32_t) * static_cast<size_t>(n), size_t(256));
  unsigned char* slab = nullptr;
  PG_CUDA(temp_alloc(reinterpret_cast<void**>(&slab), 2 * kbytes + 4 * pbytes, s));
  keys = reinterpret_cast<K*>(slab);
  pos = reinterpret_cast<uint32_t*>(slab + 2 * kbytes);
  rowk = reinterpret_cast<uint32_t*>(slab + 2 * kbytes + 2 * pbytes);
  cub::DoubleBuffer<K> kb(keys, reinterpret_cast<K*>(slab + kbytes));
  cub::DoubleBuffer<uint32_t> pb(pos, reinterpret_cast<uint32_t*>(slab + 2 * kbytes + pbytes));
  cub::DoubleBuffer<uint32_t> rb(rowk, reinterpret_cast<uint32_t*>(slab + 2 * kbytes + 3 * pbytes));
  const unsigned grid = static_cast<unsigned>(std::min<long long>(ceil_div(total, 256), static_cast<long long>(num_sms()) * 16));
  sort_keys_kernel<T><<<grid, 256, 0, s>>>(tile, rows, N, ld, descending, kb.Current(), pb.Current());
  count_launch();
  int row_bits = 1;
  while ((1ll << row_bits) < rows) ++row_bits;
  size_t t1 = 0, t2 = 0;
  cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, t1, kb, pb, n, 0, static_cast<int>(sizeof(K) * 8), s);
  if (e == cudaSuccess) e = cub::DeviceRadixSort::SortPairs(nullptr, t2, rb, pb, n, 0, row_bits, s);
  void* tmp = nullptr;
  if (e == cudaSuccess) e = temp_alloc(&tmp, std::max(t1, t2), s);
  size_t tb = std::max(t1, t2);
  if (e == cudaSuccess) e = cub::DeviceRadixSort::SortPairs(tmp, tb, kb, pb, n, 0, static_cast<int>(sizeof(K) * 8), s);
  if (e == cudaSuccess) {
    sort_rows_of_kernel<<<grid, 256, 0, s>>>(pb.Current(), total, static_cast<unsigned>(N), rb.Current());
    e = cub::DeviceRadixSort::SortPairs(tmp, tb, rb, pb, n, 0, row_bits, s);
    count_launch();
  }
  if (e == cudaSuccess) {
    const long long out_total = rows * k;
    sort_take_kernel<T><<<static_cast<unsigned>(std::min<long long>(ceil_div(out_total, 256), 1 << 20)), 256, 0, s>>>(
        tile, pb.Current(), rows, N, ld, k, drop, out_idx, out_val);
    count_launch();
    e = cudaGetLastError();
  }
  if (tmp) cudaFreeAsync(tmp, s);
  cudaFreeAsync(slab, s);
  if (e != cudaSuccess) { set_error("tile top-k by sort failed: %s", cudaGetErrorString(e)); return PG_ERR_CUDA; }
  return PG_OK;
}

// =============================================================================
// Threshold -> CSR compaction
// =============================================================================
struct ThreshParams {
  int cmp, swap, guard;
  float eps_f;
  double eps_d;
  int eps_is_int;     // integer tiles: compare exactly (python int eps) instead of in float32
};

__device__ __forceinline__ bool cmp_apply(int cmp, double a, double b) {
  switch (cmp) {
    case PG_LT: return a < b;
    case PG_LE: return a <= b;
    case PG_EQ: return a == b;
    case PG_NE: return a != b;
    case PG_GE: return a >= b;
    default: return a > b;
  }
}
// v is converted exactly to double for every supported dtype except |int64| > 2^53 (not a
// distance).  eps was rounded to the tile dtype on the host (fp16 / fp32) as torch does.  An
// integer tile against a python float compares in float32 (torch's promotion): both operands are
// rounded to float32, whose values double holds exactly.
template <typename T> __device__ __forceinline__ double as_double(T v) { return static_cast<double>(v); }
template <> __device__ __forceinline__ double as_double<__half>(__half v) { return static_cast<double>(__half2float(v)); }

template <typename T>
__device__ __forceinline__ bool keep_value(T v, const ThreshParams& tp) {
  if (sizeof(T) == 1) return v != T(0);  // mask input
  const double x = as_double<T>(v);
  const double xc = (std::is_integral<T>::value && !tp.eps_is_int) ? static_cast<double>(static_cast<float>(v)) : x;
  const bool c = tp.swap ? cmp_apply(tp.cmp, tp.eps_d, xc) : cmp_apply(tp.cmp, xc, tp.eps_d);
  if (tp.guard == 1) return c && (x > 0.0);
  if (tp.guard == 2) return c && (x < 1.0);
  return c;
}

template <typename T>
__global__ void __launch_bounds__(256) tile_thresh_count_kernel(const T* __restrict__ tile, long long N, long long ld,
                                                                 ThreshParams tp, long long* __restrict__ counts) {
  const long long row = blockIdx.x;
  const T* src = tile + static_cast<size_t>(row) * ld;
  int c = 0;
  for (long long i = threadIdx.x; i < N; i += 256) c += keep_value<T>(src[i], tp) ? 1 : 0;
  __shared__ int wsum[8];
  c = warp_sum(c);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    long long t = 0;
    for (int w = 0; w < 8; ++w) t += wsum[w];
    counts[row] = t;
  }
}

template <typename T>
__global__ void __launch_bounds__(256) tile_thresh_fill_kernel(const T* __restrict__ tile, long long N, long long ld,
                                                                ThreshParams tp, const long long* __restrict__ indptr,
                                                                long long* __restrict__ out_idx, T* __restrict__ out_val) {
  const long long row = blockIdx.x;
  const T* src = tile + static_cast<size_t>(row) * ld;
  __shared__ int wcnt[8];
  __shared__ long long s_base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_base = indptr[row];
  __syncthreads();
  for (long long base = 0; base < N; base += 256) {
    const long long i = base + threadIdx.x;
    T v = T(0);
    bool keep = false;
    if (i < N) { v = src[i]; keep = keep_value<T>(v, tp); }
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) wcnt[warp] = __popc(bal);
    __syncthreads();
    int before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      const int c = wcnt[w];
      if (w < warp) before += c;
      total += c;
    }
    const long long start = s_base;
    if (keep) {
      const long long at = start + before + __popc(bal & ((1u << lane) - 1u));
      out_idx[at] = i;
      if (out_val) out_val[at] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) s_base = start + total;
    __syncthreads();
  }
}

static int fill_thresh(ThreshParams& tp, int dtype, int cmp, double eps, int swap, int guard) {
  PG_CHECK_ARG(cmp >= PG_LT && cmp <= PG_GT, "bad comparison opcode %d", cmp);
  const int kind = guard & ~PG_EPS_FLOAT;
  PG_CHECK_ARG(kind >= 0 && kind <= 2, "bad guard %d", guard);
  tp.cmp = cmp;
  tp.swap = swap;
  tp.guard = kind;
  // a python scalar is compared the way torch compares it: rounded to a float tile's dtype; exactly
  // against an integer tile when it is an int; in float32 against an integer tile when it is a float
  tp.eps_is_int = (guard & PG_EPS_FLOAT) ? 0 : 1;
  const bool to_f32 = dtype == PG_F32 || ((dtype == PG_I32 || dtype == PG_I64) && !tp.eps_is_int);
  if (dtype == PG_F16) tp.eps_d = static_cast<double>(__half2float(__float2half_rn(static_cast<float>(eps))));
  else if (to_f32) tp.eps_d = static_cast<double>(static_cast<float>(eps));
  else tp.eps_d = eps;
  tp.eps_f = static_cast<float>(tp.eps_d);
  return PG_OK;
}

}  // namespace pg

using namespace pg;

extern "C" {

int pg_minkowski_tile(const void* X, int64_t N, const void* Y, int64_t M, int64_t q0, int64_t qrows, int D, int dtype,
                      double p, int similarity, void* out, int64_t ld, void* stream) {
  PG_CHECK_ARG(X && Y && out, "null pointer");
  PG_CHECK_ARG(N > 0 && M > 0 && D > 0, "empty operand");
  PG_CHECK_ARG(q0 >= 0 && qrows > 0 && q0 + qrows <= M, "query range outside Y");
  PG_CHECK_ARG(ld >= N, "leading dimension too small");
  PG_CHECK_ARG(p != 0.0, "p must be non-zero");
  ElemParams prm;
  memset(&prm, 0, sizeof(prm));
  prm.X = X; prm.N = N; prm.Y = Y; prm.q0 = q0; prm.qrows = qrows; prm.D = D;
  prm.out = out; prm.ld = ld; prm.similarity = similarity;
  const double root = 1.0 / p;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (p == 1.0 && D <= 32768 && qrows <= 8ll * 65535 && (dtype == PG_F16 || dtype == PG_F32 || dtype == PG_I64)) {
    // no abs in the reference: p = 1 is sum(x) - sum(y), a rank-1 tile; the element-wise kernel is
    // launched behind it and only runs if the float rows turn out not to be small integers
    void* scratch = nullptr;
    int* flag = nullptr;
    int rc;
    if (dtype == PG_I64) {
      rc = launch_mink1<long long, VK_I64>(static_cast<const long long*>(X), N, static_cast<const long long*>(Y), q0, qrows, D,
                                           similarity, out, ld, &scratch, &flag, s);
    } else if (dtype == PG_F32) {
      rc = launch_mink1<float, VK_F32>(static_cast<const float*>(X), N, static_cast<const float*>(Y), q0, qrows, D, similarity,
                                       out, ld, &scratch, &flag, s);
      if (rc == PG_OK) {
        prm.p_f = prm.root_f = 1.0f;
        prm.only_if = flag;
        rc = launch_elem<float, VK_F32, 0>(prm, PK_ONE, PK_ONE, s);
      }
    } else {
      rc = launch_mink1<__half, VK_F16>(static_cast<const __half*>(X), N, static_cast<const __half*>(Y), q0, qrows, D,
                                        similarity, out, ld, &scratch, &flag, s);
      if (rc == PG_OK) {
        prm.p_f = prm.root_f = 1.0f;
        prm.only_if = flag;
        rc = launch_elem<__half, VK_F16, 0>(prm, PK_ONE, PK_ONE, s);
      }
    }
    if (scratch != nullptr) cudaFreeAsync(scratch, s);
    return rc;
  }
  if (dtype == PG_F16) {
    // exp_scalar.to<Half>(): both exponents are rounded to fp16 before use
    prm.p_f = __half2float(__float2half_rn(static_cast<float>(p)));
    prm.root_f = __half2float(__float2half_rn(static_cast<float>(root)));
    return launch_elem<__half, VK_F16, 0>(prm, pow_kind(prm.p_f), pow_kind(prm.root_f), s);
  }
  if (dtype == PG_F32) {
    prm.p_f = static_cast<float>(p);
    prm.root_f = static_cast<float>(root);
    return launch_elem<float, VK_F32, 0>(prm, pow_kind(prm.p_f), pow_kind(prm.root_f), s);
  }
  if (dtype == PG_F64) {
    prm.p_d = p;
    prm.root_d = root;
    return launch_elem<double, VK_F64, 0>(prm, pow_kind(p), pow_kind(root), s);
  }
  if (dtype == PG_I64) {
    PG_CHECK_ARG(p == static_cast<double>(static_cast<int>(p)) && p > 0,
                 "integer inputs need a positive integer p (promote to float32 for other exponents)");
    prm.p_int = static_cast<int>(p);
    prm.root_f = static_cast<float>(root);
    // the integer power is exact; only the root kind matters for the instantiation choice
    const int pkr = pow_kind(prm.root_f);
    if (pkr == PK_SQRT) return launch_elem<long long, VK_I64, 0>(prm, PK_TWO, PK_SQRT, s);
    if (pkr == PK_ONE) return launch_elem<long long, VK_I64, 0>(prm, PK_ONE, PK_ONE, s);
    if (prm.p_int == 3) return launch_elem<long long, VK_I64, 0>(prm, PK_THREE, PK_GENERAL, s);
    return launch_elem<long long, VK_I64, 0>(prm, PK_GENERAL, PK_GENERAL, s);
  }
  set_error("minkowski tile: unsupported dtype %d", dtype);
  return PG_ERR_INVALID;
}

int pg_hamming_values_tile(const void* X, int64_t N, const void* Y, int64_t M, int64_t q0, int64_t qrows, int D,
                           int dtype, int weight, void* out, int64_t ld, void* stream) {
  PG_CHECK_ARG(X && Y && out, "null pointer");
  PG_CHECK_ARG(N > 0 && M > 0 && D > 0, "empty operand");
  PG_CHECK_ARG(q0 >= 0 && qrows > 0 && q0 + qrows <= M, "query range outside Y");
  PG_CHECK_ARG(ld >= N, "leading dimension too small");
  ElemParams prm;
  memset(&prm, 0, sizeof(prm));
  prm.X = X; prm.N = N; prm.Y = Y; prm.q0 = q0; prm.qrows = qrows; prm.D = D;
  prm.out = out; prm.ld = ld; prm.weight = weight;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  switch (dtype) {
    case PG_F16: return launch_elem<__half, VK_F16, 1>(prm, 0, 0, s);
    case PG_F32: return launch_elem<float, VK_F32, 1>(prm, 0, 0, s);
    case PG_F64: return launch_elem<double, VK_F64, 1>(prm, 0, 0, s);
    case PG_I64: return launch_elem<long long, VK_I64, 1>(prm, 0, 0, s);
  }
  set_error("hamming values tile: unsupported dtype %d", dtype);
  return PG_ERR_INVALID;
}

int pg_tile_topk(const void* tile, int dtype, int64_t rows, int64_t N, int64_t ld, int k, int drop, int descending,
                 int64_t* out_idx, void* out_val, void* stream) {
  PG_CHECK_ARG(tile && out_idx && out_val, "null pointer");
  PG_CHECK_ARG(rows > 0 && N > 0 && ld >= N, "bad tile shape");
  PG_CHECK_ARG(N < (1ll << 32), "row too long for 32-bit indices");
  PG_CHECK_ARG(k >= 1 && drop >= 0, "k must be >= 1 and drop >= 0");
  long long k1 = static_cast<long long>(k) + drop;
  if (k1 > N) k1 = N;
  int cap = 2;
  while (cap < k1) cap <<= 1;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (cap > 4096) {      // longer than the shared-memory sort holds: sort the whole rows, like the reference
    long long* oi = reinterpret_cast<long long*>(out_idx);
    switch (dtype) {
      case PG_F16: return tile_topk_by_sort(static_cast<const __half*>(tile), rows, N, ld, k, drop, descending, oi, static_cast<__half*>(out_val), s);
      case PG_F32: return tile_topk_by_sort(static_cast<const float*>(tile), rows, N, ld, k, drop, descending, oi, static_cast<float*>(out_val), s);
      case PG_F64: return tile_topk_by_sort(static_cast<const double*>(tile), rows, N, ld, k, drop, descending, oi, static_cast<double*>(out_val), s);
      case PG_I32: return tile_topk_by_sort(static_cast<const int*>(tile), rows, N, ld, k, drop, descending, oi, static_cast<int*>(out_val), s);
      case PG_I64: return tile_topk_by_sort(static_cast<const long long*>(tile), rows, N, ld, k, drop, descending, oi, static_cast<long long*>(out_val), s);
      default: set_error("tile top-k: unsupported dtype %d", dtype); return PG_ERR_INVALID;
    }
  }
#define PG_TK(T)                                                                                              \
  do {                                                                                                        \
    const size_t smem = (sizeof(KeyOf<T>::K) + 4) * static_cast<size_t>(cap);                                 \
    PG_CUDA(cudaFuncSetAttribute(tile_topk_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024)); \
    tile_topk_kernel<T><<<static_cast<unsigned>(rows), TK_THREADS, smem, s>>>(                                \
        static_cast<const T*>(tile), N, ld, k, drop, descending, reinterpret_cast<long long*>(out_idx),        \
        static_cast<T*>(out_val), cap);                                                                       \
  } while (0)
  switch (dtype) {
    case PG_F16: PG_TK(__half); break;
    case PG_F32: PG_TK(float); break;
    case PG_F64: PG_TK(double); break;
    case PG_I32: PG_TK(int); break;
    case PG_I64: PG_TK(long long); break;
    default: set_error("tile top-k: unsupported dtype %d", dtype); return PG_ERR_INVALID;
  }
#undef PG_TK
  PG_LAUNCH_CHECK();
  return PG_OK;
}

int pg_tile_threshold_count(const void* tile, int dtype, int64_t rows, int64_t N, int64_t ld, int cmp, double eps,
                            int swap, int guard, int64_t* counts, void* stream) {
  PG_CHECK_ARG(tile && counts, "null pointer");
  PG_CHECK_ARG(rows > 0 && N > 0 && ld >= N, "bad tile shape");
  ThreshParams tp;
  int rc = fill_thresh(tp, dtype, cmp, eps, swap, guard);
  if (rc != PG_OK) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
#define PG_TC(T) \
  tile_thresh_count_kernel<T><<<static_cast<unsigned>(rows), 256, 0, s>>>(static_cast<const T*>(tile), N, ld, tp, \
                                                                          reinterpret_cast<long long*>(counts))
  switch (dtype) {
    case PG_U8: PG_TC(uint8_t); break;
    case PG_F16: PG_TC(__half); break;
    case PG_F32: PG_TC(float); break;
    case PG_F64: PG_TC(double); break;
    case PG_I32: PG_TC(int); break;
    case PG_I64: PG_TC(long long); break;
    default: set_error("tile threshold: unsupported dtype %d", dtype); return PG_ERR_INVALID;
  }
#undef PG_TC
  PG_LAUNCH_CHECK();
  return PG_OK;
}

int pg_tile_threshold_fill(const void* tile, int dtype, int64_t rows, int64_t N, int64_t ld, int cmp, double eps,
                           int swap, int guard, const int64_t* indptr, int64_t* out_idx, void* out_val, void* stream) {
  PG_CHECK_ARG(tile && indptr && out_idx, "null pointer");
  PG_CHECK_ARG(rows > 0 && N > 0 && ld >= N, "bad tile shape");
  ThreshParams tp;
  int rc = fill_thresh(tp, dtype, cmp, eps, swap, guard);
  if (rc != PG_OK) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
#define PG_TF(T)                                                                                          \
  tile_thresh_fill_kernel<T><<<static_cast<unsigned>(rows), 256, 0, s>>>(                                 \
      static_cast<const T*>(tile), N, ld, tp, reinterpret_cast<const long long*>(indptr),                 \
      reinterpret_cast<long long*>(out_idx), static_cast<T*>(out_val))
  switch (dtype) {
    case PG_U8: PG_TF(uint8_t); break;
    case PG_F16: PG_TF(__half); break;
    case PG_F32: PG_TF(float); break;
    case PG_F64: PG_TF(double); break;
    case PG_I32: PG_TF(int); break;
    case PG_I64: PG_TF(long long); break;
    default: set_error("tile threshold: unsupported dtype %d", dtype); return PG_ERR_INVALID;
  }
#undef PG_TF
  PG_LAUNCH_CHECK();
  return PG_OK;
}

}  // extern "C"
