/* prograph_b200.h -- C ABI of the B200-native graph-construction path.
 *
 * The reference (acmater/prograph) is pure Python and has no FFI; its plug-in seam
 * is the distance-function protocol  fn(X[N,D], Y[M,D], similarity=False) -> (M,N)
 * (prograph/distance/hamming.py:8-39, minkowski.py:8-41) consumed by
 * Prograph.build_graph / calc_neighbours / neighbourhood / indexing
 * (prograph/prograph.py:254-343, 526-588, 656-765).  The entry points below are what a
 * ctypes binding on the reference side calls instead of the torch broadcasting
 * expressions; each one names the reference lines it replaces.  INTEGRATION.md shows
 * the binding.
 *
 * Conventions
 *   - every function returns PG_OK (0) or a negative pgStatus; pg_last_error() gives
 *     the message of the last failure on the calling thread;
 *   - all pointers are DEVICE pointers unless the name ends in _host; the caller owns
 *     every buffer, the library allocates nothing that outlives a call except where a
 *     workspace pointer + size is passed in explicitly;
 *   - every launch goes to the cudaStream_t passed as `stream` (a void*; NULL = legacy
 *     default stream); calls are asynchronous unless stated otherwise;
 *   - row indices are 64-bit, distances of the Hamming family are 32-bit inside the
 *     library and widened to the reference's dtypes (int64 / float32) on output.
 */
#ifndef PROGRAPH_B200_H
#define PROGRAPH_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  PG_OK = 0,
  PG_ERR_INVALID = -1,      /* bad argument (maps to ValueError)                    */
  PG_ERR_UNSUPPORTED = -2,  /* configuration outside the fused kernels (host falls
                               back to the tile kernels, never to the CPU)          */
  PG_ERR_CUDA = -3,         /* CUDA runtime error (RuntimeError)                    */
  PG_ERR_RANGE = -4         /* a token does not fit the requested bit planes        */
} pgStatus;

typedef enum {
  PG_U8 = 0, PG_I16 = 1, PG_I32 = 2, PG_I64 = 3, PG_F16 = 4, PG_F32 = 5, PG_F64 = 6
} pgDtype;

/* comparison opcodes, python's operator.{lt,le,eq,ne,ge,gt} (prograph.py:665,734-736) */
typedef enum { PG_LT = 0, PG_LE = 1, PG_EQ = 2, PG_NE = 3, PG_GE = 4, PG_GT = 5 } pgCmp;

/* how a Hamming distance d is written out */
typedef enum {
  PG_W_I64 = 0,   /* d as int64                      (hamming.py:34)                */
  PG_W_SIM_F32 = 1,/* 1/(1+d) as float32             (hamming.py:37-38)             */
  PG_W_I32 = 2,   /* d as int32 (library-internal tiles)                            */
  PG_W_FLAG_U8 = 3/* lo <= d <= hi as one byte 0/1 (pg_hamming_flags_tile only)      */
} pgWeight;

int         pg_version(void);
const char* pg_last_error(void);
/* sm count, compute capability and resident-CTA figure used for grid sizing */
int pg_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---------------------------------------------------------------------------
 * Packed token table.  Replaces the fp16 staging copy of prograph.py:726 for integer
 * tokens: residue l of row n is spread over `planes` bit planes; word w of plane p
 * holds bit p of residues 32w..32w+31.  Layout [rows_padded][planes][words] uint32,
 * rows_padded = pg_packed_rows(N), words = pg_packed_words(L); pad rows/residues are 0
 * (the reference pads with token 0, distance/utils.py:32-38).
 * ------------------------------------------------------------------------- */
int     pg_packed_words(int L);             /* 1,2,4,8 or a multiple of 8            */
int64_t pg_packed_rows(int64_t N);          /* N rounded up to the stream tile       */
size_t  pg_packed_bytes(int64_t N, int L, int planes);
/* tokens: [N][L] of `dtype` with row stride ld (elements).  Lw = words of the output
 * (>= pg_packed_words(L); lets two operands of different width share one width).
 * *flag (device int, caller-zeroed) is set to 1 if a token is negative, non-integral
 * or >= 2^planes.  */
int pg_pack_tokens(const void* tokens, int dtype, int64_t N, int L, int64_t ld,
                   uint32_t* packed, int planes, int words, int* flag, void* stream);

/* fused tokeniser + pack (prograph.py:454-474 then :726): chars is the (N, L) matrix of residue
 * letters (numpy 'S1' view, zero bytes pad shorter strings), lut256_host maps a byte to its token
 * (letter i of the alphabet -> i+1, everything else -> 0) */
int pg_pack_chars(const uint8_t* chars, int64_t N, int L, int64_t ld, const uint8_t* lut256_host,
                  uint32_t* packed, int planes, int words, void* stream);

/* ---------------------------------------------------------------------------
 * Fused Hamming sweeps: "own" rows live in registers, the "stream" table is swept
 * through shared memory; the (own x stream) distance matrix never reaches HBM.
 * Replaces hamming.py:34 + the consumer that follows it in prograph.py.
 * Covered packed shapes (planes x words per plane, as pg_packed_words gives them): planes 5 or 8
 * with words 1, 2, 4 and every multiple of 8 up to 1024 (rows of up to 32768 residues); other
 * shapes return PG_ERR_UNSUPPORTED before any device work.  The symmetric sweeps below cover
 * words <= 8, and 16 at 5 planes.
 * ------------------------------------------------------------------------- */

/* size in bytes of the workspace the fused sweeps need (split partials) */
size_t pg_sweep_workspace_bytes(int64_t own_rows, int64_t stream_rows, int words, int k1);

/* workspace of the two epsilon passes: per-split row counts plus, when it fits, room for the
 * first 128 hits of every (split,row): sparse graphs (e.g. the default eps=1 graph of
 * Prograph.__init__, prograph.py:140-141) are then finished by a compaction kernel instead of
 * a second sweep */
size_t pg_eps_workspace_bytes(int64_t own_rows, int64_t stream_rows, int words);
/* the same with room for `capture` hits per (split,row): a caller that knows the graph is dense
 * -- a degree sample -- lets the count pass keep every hit (pg_hamming_eps_count_capture), and
 * pg_hamming_eps_fill_capture becomes one coalesced copy instead of a second sweep.  The column
 * range is then cut into no more splits than keep the captures within 8 GiB; if one split is
 * already too much, the default geometry and captures are used.  Count, fill and this function
 * must be given the same `capture`. */
size_t pg_eps_workspace_bytes_capture(int64_t own_rows, int64_t stream_rows, int words, int capture);

/* kNN (prograph.py:755-765: sort each row, keep sorted positions drop..drop+k-1).
 * For every own row r in [row0,row0+rows): the first (drop+k) stream rows in
 * (distance, index) order; positions [drop, drop+k) are written:
 *   out_idx[r*k + j]  int64,  out_w[r*k + j] per `weight`.
 * If stream_rows < drop+k the tail is filled with idx = -1 and weight 0 (int64 0, or 0.0f for
 * similarities; the same for every kNN output of this library).  The lists of 256 own rows live in
 * shared memory: k + drop <= 78 at every covered width except 5 planes with 1025..1792 residues
 * (words 40..56, whose ring holds whole rows: fewer there), else PG_ERR_UNSUPPORTED.  */
int pg_hamming_knn(const uint32_t* own, int64_t own_rows, int64_t row0, int64_t rows,
                   const uint32_t* stream_tab, int64_t stream_rows,
                   int planes, int words, int k, int drop, int weight,
                   int64_t* out_idx, void* out_w,
                   void* workspace, size_t workspace_bytes, void* stream);

/* (qrows, N) membership flags of query rows [q0,q0+qrows) against all data rows:
 * out[(q-q0)*ld + n] = 1 if d_lo <= d(q, n) <= d_hi else 0 (uint8).  One fused sweep answers a whole
 * batch of neighbourhood queries (prograph.py:571-588 `hamming(...) <= eps`, and the batched frontier
 * of neighbourhood_clustering, prograph.py:590-615) without materialising distances.  q0 % 512 == 0.  */
int pg_hamming_flags_tile(const uint32_t* data, int64_t data_rows, const uint32_t* queries,
                          int64_t query_rows, int64_t q0, int64_t qrows, int planes, int words,
                          int d_lo, int d_hi, uint8_t* out, int64_t ld, void* stream);
/* covered[n] |= OR over the rows r with accept_host[r] != 0 of flags[r*ld + n]  (uint8 0/1 arrays) */
int pg_flags_or_rows(const uint8_t* flags, int64_t rows, int64_t N, int64_t ld,
                     const uint8_t* accept_host, uint8_t* covered, void* stream);

/* Symmetric kNN of a table against itself (the case build_graph runs, prograph.py:755-765):
 * d(i,j) == d(j,i), so every unordered pair is evaluated once and offered to the lists of both
 * rows -- half of the reference's N x N evaluations.  The triangle is cut into `parts` pieces
 * (part = rank, parts = world size; 0, 1 for one GPU): mode 0 gives this rank the row blocks
 * (256 rows) part, part + parts, ...; mode 1 gives it every row block restricted to a band of
 * stream rows (pg_knn_sym_band; bands hold equal numbers of pair evaluations), so that a row's
 * column-side candidates all meet on one rank.  The call leaves in lists[r*k1 .. r*k1+k1) the k1
 * smallest keys  distance<<32 | index  this rank saw for row r, ascending, ~0 = empty.  With several
 * ranks the per-rank lists are exchanged (all-to-all: every rank receives all ranks' lists of its own
 * rows), merged by pg_knn_lists_merge, all-gathered as 8-byte keys and widened by
 * pg_knn_lists_finalize.  k1 <= 32; wider lists take pg_hamming_knn.
 * Row locks: a lock that cannot be taken within 2^24 attempts sets an error word in the workspace
 * instead of trapping; pg_knn_sym_status (synchronises the stream) turns it into PG_ERR_CUDA.
 *
 * Bootstrap (boot_rows > 0, a multiple of 512): the caller first runs pg_hamming_knn_boot, which
 * sweeps rows [row0,row0+rows) one-sided against table rows [0,boot_rows) and writes their
 * lists; `lists` of ALL rows (all-gathered when the bootstrap was sharded) then enter
 * pg_hamming_knn_sym as the starting lists.  Every row's filter is tight from the first tile on,
 * which keeps the locked list updates rare.  */
size_t pg_knn_sym_workspace_bytes(int64_t rows, int words);
int pg_hamming_knn_boot(const uint32_t* table, int64_t table_rows, int64_t row0, int64_t rows,
                        int64_t boot_rows, int planes, int words, int k1, uint64_t* lists,
                        void* workspace /* pg_sweep_workspace_bytes(rows, boot_rows, words, k1) */,
                        size_t workspace_bytes, void* stream);
int pg_hamming_knn_sym(const uint32_t* table, int64_t rows, int planes, int words, int k1,
                       int part, int parts, int mode, int64_t boot_rows, uint64_t* lists,
                       void* workspace, size_t workspace_bytes, void* stream);
/* after pg_hamming_knn_sym on the same workspace / stream: PG_OK, or PG_ERR_CUDA if the sweep gave
 * up on a row lock (its lists are then incomplete).  Synchronises `stream`.  */
int pg_knn_sym_status(const void* workspace, int64_t rows, int words, void* stream);
/* host only: the stream rows [row_begin, row_end) of band `part` of `parts` (mode 1) */
int pg_knn_sym_band(int64_t rows, int words, int64_t boot_rows, int part, int parts,
                    int64_t* row_begin, int64_t* row_end);
/* host only: the work items (row block, first tile, end tile, boot flag: 4 x int32 each) the
 * symmetric sweeps deal to a persistent grid of `grid` CTAs, in dealing order: CTA b takes items
 * b, b + grid, ...  Items are ordered by L2-sized column bands (PG_SYM_BAND_MB, default 24 MB) so
 * that co-resident CTAs stream the same part of the table.  *n_items = number of items;
 * items_host may be NULL (count only) or hold `capacity` items.  */
int pg_knn_sym_plan(int64_t rows, int planes, int words, int64_t boot_rows, int part, int parts,
                    int mode, int grid, int32_t* items_host, int64_t capacity, int64_t* n_items);
/* Symmetric epsilon graph of a table against itself (prograph.py:731-753): one sweep over the
 * triangle of unordered pairs appends BOTH directed edges of every pair whose distance passes the
 * truth table `lut_host` (which must be one contiguous range of distances, else
 * PG_ERR_UNSUPPORTED) to `keys` as  row << (idxbits+dbits) | column << dbits | distance.  Slots are
 * handed out in chunks of 512; unused slots hold the sentinel ~0.  counters[0] (device) = slots
 * reserved, counters[1] = edges; if counters[0] > capacity the buffer was too small (nothing is
 * written past it) and the call is repeated with counters[0] slots.  part / parts / mode as in
 * pg_hamming_knn_sym; workspace: pg_knn_sym_workspace_bytes.  */
int pg_hamming_eps_sym(const uint32_t* table, int64_t rows, int planes, int words,
                       const uint32_t* lut_host, int lut_words, int part, int parts, int mode,
                       uint64_t* keys, int64_t capacity, uint64_t* counters,
                       void* workspace, size_t workspace_bytes, void* stream);
/* sort n_keys edge keys (sentinels included; keys_alt: scratch of the same size) by (row, column)
 * and write the CSR arrays of the first nnz: indptr[rows+1], out_idx int64, out_w per `weight`
 * (int64 distance or float32 similarity).  Replaces prod_neighbours + merge/fill, prograph.py:626-654,
 * 743-753.  */
int pg_edge_keys_to_csr(uint64_t* keys, int64_t n_keys, uint64_t* keys_alt, int64_t rows, int words,
                        int64_t nnz, int weight, int64_t* indptr, int64_t* out_idx, void* out_w,
                        void* stream);

/* merge n_lists key lists per row (list s of row r at lists[s*list_stride + r*k1]), drop the first
 * `drop` merged positions and write the next k as out_idx[(r-row0)*k + j] / out_w per `weight`
 * for rows [row0, row0+rows); missing entries get idx = -1 (as pg_hamming_knn).  */
int pg_knn_lists_finalize(const uint64_t* lists, int n_lists, int64_t list_stride,
                          int64_t row0, int64_t rows, int k1, int k, int drop, int weight,
                          int64_t* out_idx, void* out_w, void* stream);
/* the same merge, keeping the 8-byte keys: out_keys[(r-row0)*k + j], ~0 = missing (what the ranks
 * of a multi-GPU build all-gather before widening with pg_knn_lists_finalize(n_lists=1, drop=0)) */
int pg_knn_lists_merge(const uint64_t* lists, int n_lists, int64_t list_stride,
                       int64_t row0, int64_t rows, int k1, int k, int drop,
                       uint64_t* out_keys, void* stream);

/* workspace of a count pass that only counts (no capture of the first hits): the degree census of
 * a graph too dense to materialise */
size_t pg_eps_count_workspace_bytes(int64_t own_rows, int64_t stream_rows, int words);
/* epsilon graph, pass 1 (prograph.py:731-736): per own row, the number of stream rows
 * whose distance d has bit d set in `lut` (a host array of (L+32)/32 words: the
 * truth table of  comp(d, eps) & (d > 0)  -- or any other predicate of d -- evaluated
 * by the caller for d = 0..L).  lut_words <= 64 (distances up to 2047), and up to words + 1 for the
 * rows of more than 1792 residues at 5 planes and more than 256 at 8 (copied to the device for
 * the sweep).  counts[r] int64, r relative to row0.  */
int pg_hamming_eps_count(const uint32_t* own, int64_t own_rows, int64_t row0, int64_t rows,
                         const uint32_t* stream_tab, int64_t stream_rows,
                         int planes, int words, const uint32_t* lut_host, int lut_words,
                         int64_t* counts, void* workspace, size_t workspace_bytes, void* stream);

/* epsilon graph, pass 2 (prograph.py:736-739 + prod_neighbours :626-654): writes, for
 * row r, its neighbours in ascending index order at indptr[r]..indptr[r+1]:
 *   out_idx int64, out_w per `weight`.  indptr is the exclusive scan of `counts`
 * (pg_exclusive_scan_i64).  The workspace must be the one pass 1 filled.  */
int pg_hamming_eps_fill(const uint32_t* own, int64_t own_rows, int64_t row0, int64_t rows,
                        const uint32_t* stream_tab, int64_t stream_rows,
                        int planes, int words, const uint32_t* lut_host, int lut_words,
                        const int64_t* indptr, int weight, int64_t* out_idx, void* out_w,
                        void* workspace, size_t workspace_bytes, void* stream);
/* both passes for a workspace sized by pg_eps_workspace_bytes_capture(..., capture) */
int pg_hamming_eps_count_capture(const uint32_t* own, int64_t own_rows, int64_t row0, int64_t rows,
                                 const uint32_t* stream_tab, int64_t stream_rows,
                                 int planes, int words, const uint32_t* lut_host, int lut_words,
                                 int capture, int64_t* counts,
                                 void* workspace, size_t workspace_bytes, void* stream);
int pg_hamming_eps_fill_capture(const uint32_t* own, int64_t own_rows, int64_t row0, int64_t rows,
                                const uint32_t* stream_tab, int64_t stream_rows,
                                int planes, int words, const uint32_t* lut_host, int lut_words,
                                int capture, const int64_t* indptr, int weight, int64_t* out_idx, void* out_w,
                                void* workspace, size_t workspace_bytes, void* stream);

/* materialised distance tile (hamming.py:34-38): out[m*ld + n] for query rows
 * m in [q0,q0+qrows) of `queries` against all `data_rows` rows of `data`;
 * `weight` picks int64 / float32-similarity / int32.  */
int pg_hamming_tile(const uint32_t* data, int64_t data_rows,
                    const uint32_t* queries, int64_t query_rows, int64_t q0, int64_t qrows,
                    int planes, int words, int weight, void* out, int64_t ld, void* stream);

/* out[i] = sum_{j<i} in[j], out[n] = total (n+1 outputs); int64; used for indptr */
int pg_exclusive_scan_i64(const int64_t* in, int64_t n, int64_t* out, void* stream);

/* ---------------------------------------------------------------------------
 * Growing a built graph by new rows (extend_neighbours): the old rows' stored neighbours joined
 * with what a one-sided sweep found for them among the new rows, whose indices start at col_base.
 * ------------------------------------------------------------------------- */
/* kNN: for each of `rows` rows, merge the sorted list prev_idx/prev_w[r*ka ..) with the sorted
 * candidates cand_idx/cand_w[r*kb ..) (cand indices + col_base) and write the first k entries to
 * out_idx/out_w[r*k ..).  weight PG_W_I64: (distance asc, index asc); PG_W_SIM_F32: (similarity
 * desc, index asc).  idx = -1 ends an input list; missing outputs get idx = -1 and weight 0 (0.0f).
 * Any ka, kb >= 0 and k >= 1.  */
int pg_knn_extend_merge(const int64_t* prev_idx, const void* prev_w, int ka,
                        const int64_t* cand_idx, const void* cand_w, int kb,
                        int64_t rows, int64_t col_base, int k, int weight,
                        int64_t* out_idx, void* out_w, void* stream);
/* epsilon: out row r = old row r followed by added row r with col_base added to its indices.
 * The entries of row r of a part are idx[indptr[r] - indptr[0] ..) (row slices of a larger CSR are
 * taken as they are); out_indptr[0] = 0, (rows+1) entries.  Weights int64 (PG_W_I64) or float32
 * (PG_W_SIM_F32); out_idx / out_w hold the sum of both parts' entries.  */
int pg_csr_append(const int64_t* old_indptr, const int64_t* old_idx, const void* old_w,
                  const int64_t* add_indptr, const int64_t* add_idx, const void* add_w,
                  int64_t rows, int64_t col_base, int weight,
                  int64_t* out_indptr, int64_t* out_idx, void* out_w, void* stream);

/* ---------------------------------------------------------------------------
 * Element-wise metric tiles (float / generic values).
 * ------------------------------------------------------------------------- */
/* minkowski.py:36-40.  X [N][D], Y [M][D] of `dtype` in {PG_F16, PG_F32, PG_F64, PG_I64};
 * out (rows q0..q0+qrows of Y) x N, dtype F16 for F16 input, F32 for F32/I64, F64 for
 * F64; every rounding step of the reference chain is reproduced (DESIGN.md).  */
int pg_minkowski_tile(const void* X, int64_t N, const void* Y, int64_t M, int64_t q0, int64_t qrows,
                      int D, int dtype, double p, int similarity, void* out, int64_t ld, void* stream);
/* hamming.py:34 on arbitrary numeric values (x != y counted per component, IEEE: NaN
 * differs from everything): out int64 (or float32 similarity). */
int pg_hamming_values_tile(const void* X, int64_t N, const void* Y, int64_t M, int64_t q0, int64_t qrows,
                           int D, int dtype, int weight, void* out, int64_t ld, void* stream);

/* ---------------------------------------------------------------------------
 * Minkowski p=2 on integer tokens as a tensor-core contraction (tcgen05 kind::i8, TMEM
 * accumulators): S = |x|^2 + |y|^2 - 2 x.y is exact in int32 and the reference's rounding
 * chain (minkowski.py:36-40) is a function of S alone.
 *   value_kind 0: fp16 chain  d = fp16(sqrt(fp16(S)))   (the dtype build_graph stages, prograph.py:726)
 *   value_kind 1: int64 tokens d = sqrtf(float(S))       (float32 result)
 * Operand tables: uint8 rows in K-major 8x16-byte core-matrix order
 *   byte(r, k) = ((r/8)*(K/16) + k/16)*128 + (r%8)*16 + k%16,  K = pg_gemm_width(L),
 * padded to pg_gemm_rows(N) rows, plus int32 squared norms per row (pad rows: 0x3fffffff).
 * K <= 8192 (PG_ERR_UNSUPPORTED above): up to K = 256 the two A tiles of a CTA stay resident in
 * shared memory, wider rows stream 128-wide K-chunks of both A tiles and the B tile through the ring
 * (same layout, same results).  With tokens <= 255, S <= 255^2 * 8192 stays below 2^29.
 * Measured on one B200 at a 1000 W power limit, kNN k=1 over 262 144 rows: 685 / 283 / 69 Gpairs/s at
 * K = 512 / 1184 / 5376, L2-bound (profiles/gemm_wide_time.log).
 * ------------------------------------------------------------------------- */
int     pg_gemm_width(int L);
int64_t pg_gemm_rows(int64_t N);
int pg_gemm_pack(const void* tokens, int dtype, int64_t N, int L, int64_t ld,
                 uint8_t* table, int32_t* norms, int K, int max_token, int* flag, void* stream);
/* *flag is set when a value is not an integer in [0, max_token] (<= 255; the fp16 chain needs <= 45 so that
 * every squared difference is exact in fp16) */
/* out[m*ld + n] (fp16 for value_kind 0, float32 for 1): queries A (M rows) x dataset B (N rows) */
int pg_minkowski2_gemm_tile(const uint8_t* A, const int32_t* normA, int64_t M,
                            const uint8_t* B, const int32_t* normB, int64_t N, int K,
                            int value_kind, int similarity, void* out, int64_t ld, void* stream);
/* fused kNN (prograph.py:755-765 with distance=minkowski): sorted positions [drop, drop+k) of every
 * query row in (value, index) order -- descending value for similarity; out_val fp16 / float32.
 * If N < drop+k the tail is filled with idx = -1 and value 0 (as pg_hamming_knn).  The lists of 256
 * query rows share shared memory with the operand ring: k + drop <= 68 at K = 32, 63 at K = 64, 31 at
 * K = 256, 42 at every K in (256, 8192] (K-chunked ring), else PG_ERR_UNSUPPORTED. */
int pg_minkowski2_gemm_knn(const uint8_t* A, const int32_t* normA, int64_t M,
                           const uint8_t* B, const int32_t* normB, int64_t N, int K,
                           int value_kind, int similarity, int k, int drop,
                           int64_t* out_idx, void* out_val, void* stream);

/* fused epsilon graph (prograph.py:731-753 with distance=minkowski): the edge test
 * comp(d, eps) & (d > 0) is monotone in S, so the caller passes it as the integer range
 * [s_lo, s_hi].  Pass 1: group_counts [2][M] (hits in the first / second half of the dataset,
 * a workspace the fill pass reads back) and counts [M]; pass 2 writes ascending column indices
 * and values (fp16 / float32) at indptr[r].. */
int pg_minkowski2_gemm_eps_count(const uint8_t* A, const int32_t* normA, int64_t M,
                                 const uint8_t* B, const int32_t* normB, int64_t N, int K,
                                 int s_lo, int s_hi, int64_t* group_counts, int64_t* counts, void* stream);
int pg_minkowski2_gemm_eps_fill(const uint8_t* A, const int32_t* normA, int64_t M,
                                const uint8_t* B, const int32_t* normB, int64_t N, int K,
                                int value_kind, int similarity, int s_lo, int s_hi,
                                const int64_t* group_counts, const int64_t* indptr,
                                int64_t* out_idx, void* out_val, void* stream);

/* ---------------------------------------------------------------------------
 * Consumers of a materialised (rows x N) tile: used for Minkowski, for user supplied
 * distance callables (README.md:48) and for single-row queries.
 * ------------------------------------------------------------------------- */
/* stable top-k of each tile row (prograph.py:757-762): positions [drop, drop+k) of the
 * row sorted by (value, index) ascending, or descending with NaN first when
 * `descending` (torch.sort semantics).  out_idx int64 [rows][k], out_val tile dtype.
 * k + drop <= 4096: radix select + sort in shared memory, one CTA per row; above that the
 * whole tile is sorted (two stable device-wide radix sorts: by value, then by row), as the
 * reference sorts whole rows for any k (rows * N < 2^31 per call). */
int pg_tile_topk(const void* tile, int dtype, int64_t rows, int64_t N, int64_t ld,
                 int k, int drop, int descending, int64_t* out_idx, void* out_val, void* stream);

/* threshold test of prograph.py:734-736 / :544 on a tile:
 *   keep = cmp(v, eps)            swap = 0
 *   keep = cmp(eps, v)            swap = 1   (similarity: operands swapped, :734)
 *   and, per `guard & 3`: 0 none, 1  v > 0  (:736),  2  v < 1  (:734).
 * eps is compared the way torch compares a tensor with a python scalar: for fp16 / float32 /
 * float64 tiles it is rounded to the tile dtype; for int32 / int64 tiles it is compared exactly
 * (a python int, |v| <= 2^53), unless `guard` carries PG_EPS_FLOAT (a python float): then both
 * operands are rounded to float32 and compared there, as torch promotes int < float to float32.
 * Pass 1 writes counts[r]; pass 2 writes ascending column indices and the values at
 * indptr[r].. ; `tile` may also be a uint8 mask (dtype PG_U8, cmp ignored). */
#define PG_EPS_FLOAT 4
int pg_tile_threshold_count(const void* tile, int dtype, int64_t rows, int64_t N, int64_t ld,
                            int cmp, double eps, int swap, int guard, int64_t* counts, void* stream);
int pg_tile_threshold_fill(const void* tile, int dtype, int64_t rows, int64_t N, int64_t ld,
                           int cmp, double eps, int swap, int guard, const int64_t* indptr,
                           int64_t* out_idx, void* out_val, void* stream);

/* ---------------------------------------------------------------------------
 * Mutation masks and index selections (prograph.py:254-343, 349-368, 488-505).
 * All work on the packed table; `ref` is one packed row (planes*words words).
 * ------------------------------------------------------------------------- */
/* mut[n][w] = OR_p (table[n][p][w] ^ ref[p][w]): bit l set <=> residue l differs from
 * the reference row (boolean_mutant_array, :488-492, as a bit mask). */
int pg_mutant_bits(const uint32_t* table, int64_t N, int planes, int words,
                   const uint32_t* ref, uint32_t* mut, void* stream);
/* the same as the reference's (N, L) bool array (one byte per residue) */
int pg_mutant_bool(const uint32_t* table, int64_t N, int planes, int words, int L,
                   const uint32_t* ref, uint8_t* out, void* stream);
/* any_bits[w] = OR_n mut[n][w]  (calc_mutated_positions, :494-505) */
int pg_mutant_any(const uint32_t* mut, int64_t N, int words, uint32_t* any_bits, void* stream);
/* Informative columns of a table swept against itself (build_graph, prograph.py:726-765):
 * a residue position at which every row carries the same token adds 0 to every pairwise
 * Hamming distance (hamming.py:34), so the sweeps may run on the other positions only.
 * varying[p*words + w] = OR_n (table[n][p][w] ^ table[0][p][w])  (device, planes*words words;
 * OR over p = bit l set <=> position l is not constant). */
int pg_varying_columns(const uint32_t* table, int64_t N, int planes, int words,
                       uint32_t* varying, void* stream);
/* out[n][p][w2] bit b = table[n][p][.] bit cols[32*w2 + b] (cols: device int32[out_words*32],
 * -1 = padding -> 0); out has pg_packed_rows(N) rows, pad rows are zeroed. */
int pg_compact_columns(const uint32_t* table, int64_t N, int planes, int words,
                       const int32_t* cols, uint32_t* out, int out_words, void* stream);
/* row selection: flag[n] = dist_ok & pos_ok with
 *   dist_ok = dist_lut == NULL or bit popc(mut[n]) of dist_lut set       (:300-308)
 *   pos_ok  = pos_mode 0: true
 *             1 ("or") : (mut & inside) != 0 and (mut & outside) == 0    (:316-325)
 *             2 ("and"): (mut & inside) == inside and (mut & outside) == 0
 *             3        : (mut & inside) == 0    (get_mutated_positions, :362-365;
 *                        `inside` then holds the positions that must stay constant)
 * `outside` = the positions that must be unchanged (the reference walks the positions of
 * the reference sequence's own length that are not selected, :316,:322-324).
 * dist_lut_host / inside_host / outside_host are HOST arrays of `words` (lut: lut_words)
 * uint32. flag: uint8 [N]. */
int pg_select_rows(const uint32_t* mut, int64_t N, int words,
                   const uint32_t* dist_lut_host, int lut_words,
                   const uint32_t* inside_host, const uint32_t* outside_host, int pos_mode,
                   uint8_t* flag, void* stream);
/* ascending indices of the set flags (np.where, :308,:325): *count_out (device int64)
 * receives the number written; out_idx must hold N entries. */
int pg_flag_indices(const uint8_t* flag, int64_t N, int64_t* out_idx, int64_t* count_out, void* stream);
/* hist[d] += 1 for d = popc(mut[n]) (the distance-from-reference histogram used for
 * np.unique(d_data), :305, and __str__, :147-154); hist: int64 [words*32+1], zeroed by
 * the caller. */
int pg_distance_hist(const uint32_t* mut, int64_t N, int words, int64_t* hist, void* stream);

/* ---------------------------------------------------------------------------
 * Measurement helpers.
 * ------------------------------------------------------------------------- */
/* integer-pipe peak for the roofline: runs a register-only kernel with the same
 * 5 LOP3 : 1 POPC : 1 IADD mix as the Hamming inner loop (mix 0), LOP3 only (1) or
 * POPC only (2) and returns lane-ops per second (synchronous). */
int pg_measure_int_peak(int mix, int iters, double* lane_ops_per_s, double* ms);
/* int8 tensor-pipe peak: back-to-back tcgen05.mma kind::i8 (M=128, N=256, K=32) on operands resident
 * in shared memory, 148 CTAs; returns int8 operations (2 per multiply-add) per second
 * (synchronous).  The upper bound of a one-hot int8 GEMM formulation of Hamming (2*21*L operations
 * per pair) that DESIGN.md compares the popcount sweep with.  */
int pg_measure_i8_mma_peak(int batches, double* int8_ops_per_s, double* ms);
/* number of kernel launches issued by this library since the last reset */
int64_t pg_launch_count(int reset);
/* average device time (CUDA events on the launch stream) of the fused sweep kernel since
 * the last reset: total ms and launches. Enable with pg_time_sweeps(1). */
int pg_time_sweeps(int enable);
int pg_sweep_time(double* total_ms, int64_t* launches, int reset);
/* the same, one entry per timed launch in launch order (ms[0..min(cap,*n))) */
int pg_sweep_times(double* ms, int64_t cap, int64_t* n, int reset);

#ifdef __cplusplus
}
#endif
#endif /* PROGRAPH_B200_H */
