"""Device engine: torch owns memory and streams, every distance / selection / compaction kernel
is a C-ABI call into libprograph_b200.so (hand-written sm_100a kernels).  No CPU fallback anywhere.
"""
import ctypes as C
import numbers

import numpy as np
import torch

from . import _lib as L

_PG_DTYPE = {
    torch.uint8: L.U8, torch.int16: L.I16, torch.int32: L.I32, torch.int64: L.I64,
    torch.float16: L.F16, torch.float32: L.F32, torch.float64: L.F64, torch.bool: L.U8,
}


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _host_u32(a):
    a = np.ascontiguousarray(a, dtype=np.uint32)
    return a, a.ctypes.data_as(C.c_void_p)


SWEEP_MAX_WORDS = 1024     # 32768 residues per row: the longest rows the one-sided sweeps take


def sweep_covers(planes, words):
    """Whether the one-sided fused sweeps (pg_hamming_knn, _eps_*, _tile, _flags_tile) take a packed
    table of `planes` bit planes and `words` 32-residue words per plane: every width pg_packed_words
    gives up to 32768 residues, at 5 planes (alphabets of up to 31 tokens) and at 8 (up to 255)."""
    return planes in (5, 8) and 1 <= words <= SWEEP_MAX_WORDS and (words in (1, 2, 4) or words % 8 == 0)


class PackedTable:
    """Bit-plane token table on the device: int32 tensor [rows_padded, planes, words]."""
    __slots__ = ("data", "rows", "L", "planes", "words", "informative")

    def __init__(self, data, rows, L_, planes, words):
        self.data, self.rows, self.L, self.planes, self.words = data, rows, L_, planes, words
        self.informative = None     # graph.informative_table: the table the self-sweeps of this one run on

    def row(self, i):
        """One packed row (planes*words words) as a device tensor."""
        return self.data[i].reshape(-1)


class GemmTable:
    """uint8 token rows in the K-major core-matrix order the tcgen05 kernel reads, plus the
    int32 squared norm of every row (pg_gemm_pack)."""
    __slots__ = ("data", "norms", "rows", "L", "K", "max_token")

    def __init__(self, data, norms, rows, L_, K, max_token):
        self.data, self.norms, self.rows, self.L, self.K, self.max_token = data, norms, rows, L_, K, max_token


class CudaEngine:
    """One engine per process/GPU.  ``device`` defaults to ``cuda:LOCAL_RANK`` as set by the
    launcher, i.e. the current torch device."""

    sharded_pack = True   # packed row shards can be all-gathered into one table (graph.pack_table)

    def __init__(self, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("prograph_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = L.load()
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        torch.cuda.set_device(self.device)

    # ---- plumbing -----------------------------------------------------------------
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def empty(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.device)

    def to_device(self, a, dtype=None):
        """numpy / torch (any device) -> contiguous tensor on this engine's device."""
        if isinstance(a, np.ndarray):
            a = torch.from_numpy(np.ascontiguousarray(a))
        elif not isinstance(a, torch.Tensor):
            a = torch.as_tensor(np.asarray(a))
        if a.dtype == torch.bool:
            a = a.to(torch.uint8)
        a = a.to(self.device, non_blocking=True)
        if dtype is not None and a.dtype != dtype:
            a = a.to(dtype)
        return a.contiguous()

    def synchronize(self):
        torch.cuda.synchronize(self.device)

    def launch_count(self, reset=False):
        return int(self.lib.pg_launch_count(1 if reset else 0))

    # ---- packed tables --------------------------------------------------------------
    def packed_words(self, L_):
        return int(self.lib.pg_packed_words(int(L_)))

    def pack(self, tokens, planes=None, words=None):
        """tokens: (N, L) integer-valued array/tensor.  Returns a PackedTable, raising
        OverflowError when a value is negative, fractional or >= 2**planes."""
        t = self.to_device(tokens)
        if t.dim() != 2 or t.shape[0] == 0 or t.shape[1] == 0:
            raise ValueError("pack expects a non-empty (N, L) array")
        if t.dtype not in _PG_DTYPE or t.dtype == torch.bool:
            t = t.to(torch.int64)
        N, L_ = int(t.shape[0]), int(t.shape[1])
        words = self.packed_words(L_) if words is None else int(words)
        tries = (5, 8) if planes is None else (int(planes),)
        flag = self.empty((1,), torch.int32)
        for pl in tries:
            rows_pad = int(self.lib.pg_packed_rows(N))
            out = self.empty((rows_pad, pl, words), torch.int32)
            flag.zero_()
            L.check(self.lib.pg_pack_tokens(_ptr(t), _PG_DTYPE[t.dtype], N, L_, int(t.stride(0)), _ptr(out), pl, words,
                                            _ptr(flag), self._stream()))
            if int(flag.item()) == 0:
                return PackedTable(out, N, L_, pl, words)
        raise OverflowError("values are not integer tokens in [0, 256): the bit-plane path does not apply")

    def pack_chars(self, chars, lut256, planes=5):
        """Residue letters straight to bit planes: `chars` is the (N, L) uint8 matrix of sequence
        bytes (zero padded), `lut256` the byte -> token table (tokenize + pack in one pass)."""
        c = self.to_device(chars)
        if c.dtype != torch.uint8 or c.dim() != 2 or c.shape[0] == 0 or c.shape[1] == 0:
            raise ValueError("pack_chars expects a non-empty (N, L) uint8 matrix")
        lut = np.ascontiguousarray(lut256, dtype=np.uint8)
        assert lut.shape == (256,)
        N, L_ = int(c.shape[0]), int(c.shape[1])
        words = self.packed_words(L_)
        out = self.empty((int(self.lib.pg_packed_rows(N)), planes, words), torch.int32)
        L.check(self.lib.pg_pack_chars(_ptr(c), N, L_, int(c.stride(0)), lut.ctypes.data_as(C.c_void_p), _ptr(out),
                                       int(planes), words, self._stream()))
        return PackedTable(out, N, L_, planes, words)

    def varying_columns(self, table):
        """Residue positions at which the rows of `table` do not all carry the same token
        (pg_varying_columns), ascending, as an int32 array."""
        var = self.empty((table.planes * table.words,), torch.int32)
        L.check(self.lib.pg_varying_columns(_ptr(table.data), table.rows, table.planes, table.words, _ptr(var),
                                            self._stream()))
        bits = var.cpu().numpy().view(np.uint32).reshape(table.planes, table.words)
        mask = np.bitwise_or.reduce(bits, axis=0)
        return np.nonzero(np.unpackbits(mask.view(np.uint8), bitorder="little"))[0].astype(np.int32)

    def compact_columns(self, table, cols):
        """The packed table restricted to the residue positions `cols` (pg_compact_columns): the same
        pairwise Hamming distances when every dropped position is constant over the rows."""
        cols = np.asarray(cols, dtype=np.int32)
        words = self.packed_words(max(1, len(cols)))
        src = np.full(words * 32, -1, dtype=np.int32)
        src[: len(cols)] = cols
        out = self.empty((int(self.lib.pg_packed_rows(table.rows)), table.planes, words), torch.int32)
        L.check(self.lib.pg_compact_columns(_ptr(table.data), table.rows, table.planes, table.words,
                                            _ptr(self.to_device(src)), _ptr(out), words, self._stream()))
        return PackedTable(out, table.rows, max(1, len(cols)), table.planes, words)

    # ---- fused Hamming sweeps -----------------------------------------------------------
    def _workspace(self, rows, stream_rows, words, k1):
        nbytes = int(self.lib.pg_sweep_workspace_bytes(int(rows), int(stream_rows), int(words), int(k1)))
        return self.empty((nbytes,), torch.uint8), nbytes

    @staticmethod
    def _check_pair(own, stream):
        if own.planes != stream.planes or own.words != stream.words:
            raise ValueError("packed operands must share planes and words")

    def hamming_knn(self, own, row0, rows, stream, k, drop=1, similarity=False):
        """prograph.py:755-765 for own rows [row0,row0+rows) against `stream`: sorted
        positions [drop, drop+k) of every row in (distance, index) order."""
        self._check_pair(own, stream)
        weight = L.W_SIM_F32 if similarity else L.W_I64
        idx = self.empty((rows, k), torch.int64)
        w = self.empty((rows, k), torch.float32 if similarity else torch.int64)
        ws, nbytes = self._workspace(rows, stream.rows, own.words, k + drop)
        L.check(self.lib.pg_hamming_knn(_ptr(own.data), own.rows, int(row0), int(rows), _ptr(stream.data), stream.rows,
                                        own.planes, own.words, int(k), int(drop), weight, _ptr(idx), _ptr(w), _ptr(ws),
                                        nbytes, self._stream()))
        return idx, w

    SYM_MAX_LIST = 32      # list length (k + drop) the symmetric sweep keeps per row

    def _sym_check(self, table, k1=1):
        if k1 > self.SYM_MAX_LIST or table.words > 16 or (table.words > 8 and table.planes != 5):
            raise L.Unsupported("shape not covered by the symmetric sweep")

    def hamming_knn_boot(self, table, row0, rows, boot_rows, k1):
        """Bootstrap lists (pg_hamming_knn_boot): rows [row0,row0+rows) one-sided against table rows
        [0, boot_rows); (rows, k1) int64 keys distance<<32 | index, -1 = empty."""
        self._sym_check(table, k1)
        lists = self.empty((rows, k1), torch.int64)
        ws, nbytes = self._workspace(rows, boot_rows, table.words, k1)
        L.check(self.lib.pg_hamming_knn_boot(_ptr(table.data), table.rows, int(row0), int(rows), int(boot_rows),
                                             table.planes, table.words, int(k1), _ptr(lists), _ptr(ws), nbytes,
                                             self._stream()))
        return lists

    def hamming_knn_sym(self, table, k1, rank=0, world=1, lists=None, boot_rows=0, mode=0):
        """Symmetric sweep of `table` against itself (pg_hamming_knn_sym): this rank's piece of the
        triangle (mode 0: row blocks rank, rank+world, ...; mode 1: a band of stream rows);
        returns the (rows, k1) int64 tensor of sorted keys
        distance<<32 | index (-1 = empty) this rank found for EVERY row of the table.  `lists`:
        the bootstrap lists of all rows when boot_rows > 0 (updated in place)."""
        self._sym_check(table, k1)
        if boot_rows:
            assert lists is not None and tuple(lists.shape) == (table.rows, k1) and lists.is_contiguous()
        else:
            lists = self.empty((table.rows, k1), torch.int64)
        nbytes = int(self.lib.pg_knn_sym_workspace_bytes(table.rows, table.words))
        ws = self.empty((nbytes,), torch.uint8)
        L.check(self.lib.pg_hamming_knn_sym(_ptr(table.data), table.rows, table.planes, table.words, int(k1),
                                            int(rank), int(world), int(mode), int(boot_rows), _ptr(lists), _ptr(ws),
                                            nbytes, self._stream()))
        self._sym_pending = (ws, table.rows, table.words)
        return lists

    def sym_check(self):
        """Status of the last symmetric kNN sweep (pg_knn_sym_status): raises if the kernel gave up
        on a row lock.  Synchronises the stream, so callers queue the rest of the build first."""
        pending, self._sym_pending = getattr(self, "_sym_pending", None), None
        if pending is not None:
            ws, rows, words = pending
            L.check(self.lib.pg_knn_sym_status(_ptr(ws), int(rows), int(words), self._stream()))

    def sym_plan(self, rows, planes, words, boot_rows=0, rank=0, world=1, mode=0, grid=296):
        """Work items (row block, first tile, end tile, boot, CTA) of the symmetric sweeps
        (host-only planner, pg_knn_sym_plan): (n, 5) int32."""
        return sym_plan(rows, planes, words, boot_rows, rank, world, mode, grid)

    def sym_band(self, rows, words, boot_rows, rank, world):
        """Stream rows [begin, end) of this rank's band (mode 1 of hamming_knn_sym)."""
        a, b = C.c_int64(0), C.c_int64(0)
        L.check(self.lib.pg_knn_sym_band(int(rows), int(words), int(boot_rows), int(rank), int(world), C.byref(a),
                                         C.byref(b)))
        return a.value, b.value

    def knn_lists_finalize(self, lists, row0, rows, k, drop=1, similarity=False):
        """lists: (n_lists, N, k1) or (N, k1) key lists -> (idx, w) of rows [row0,row0+rows)."""
        if lists.dim() == 2:
            lists = lists.unsqueeze(0)
        lists = lists.contiguous()
        n_lists, n, k1 = lists.shape
        weight = L.W_SIM_F32 if similarity else L.W_I64
        idx = self.empty((rows, k), torch.int64)
        w = self.empty((rows, k), torch.float32 if similarity else torch.int64)
        L.check(self.lib.pg_knn_lists_finalize(_ptr(lists), n_lists, n * k1, int(row0), int(rows), k1, int(k),
                                               int(drop), weight, _ptr(idx), _ptr(w), self._stream()))
        return idx, w

    def knn_lists_merge(self, lists, k, drop=1):
        """(n_lists, rows, k1) sorted key lists -> (rows, k) merged keys after dropping the first `drop`
        (pg_knn_lists_merge); -1 = missing."""
        lists = lists.contiguous()
        n_lists, rows, k1 = lists.shape
        out = self.empty((rows, k), torch.int64)
        L.check(self.lib.pg_knn_lists_merge(_ptr(lists), n_lists, rows * k1, 0, rows, k1, int(k), int(drop), _ptr(out),
                                            self._stream()))
        return out

    def knn_extend_merge(self, prev_idx, prev_w, cand_idx, cand_w, col_base, k, similarity=False):
        """(rows, k) kNN lists of rows whose sorted lists `prev_*` (rows, kA) meet sorted candidates
        `cand_*` (rows, kB) from a table whose row 0 is row `col_base` of the graph
        (pg_knn_extend_merge): the first k of the merge in (distance, index) order."""
        rows, ka = prev_idx.shape
        kb = cand_idx.shape[1]
        wdt = torch.float32 if similarity else torch.int64
        prev_idx, prev_w = prev_idx.contiguous(), prev_w.to(wdt).contiguous()
        cand_idx, cand_w = cand_idx.contiguous(), cand_w.to(wdt).contiguous()
        idx = self.empty((rows, k), torch.int64)
        w = self.empty((rows, k), wdt)
        L.check(self.lib.pg_knn_extend_merge(_ptr(prev_idx), _ptr(prev_w), ka, _ptr(cand_idx), _ptr(cand_w), kb, rows,
                                             int(col_base), int(k), L.W_SIM_F32 if similarity else L.W_I64, _ptr(idx),
                                             _ptr(w), self._stream()))
        return idx, w

    def csr_append(self, old, add, col_base, similarity=False):
        """CSR whose row r is row r of `old` followed by row r of `add` with `col_base` added to its
        indices (pg_csr_append).  Both are (indptr, idx, w) of the same rows; an indptr may start
        above 0 (a row slice of a larger CSR whose idx / w are cut to those rows)."""
        wdt = torch.float32 if similarity else torch.int64
        (oip, oi, ow), (aip, ai, aw) = ([t.contiguous() for t in part[:2]] + [part[2].to(wdt).contiguous()]
                                        for part in (old, add))
        rows = oip.numel() - 1
        nnz = oi.numel() + ai.numel()
        self.check_edge_budget(nnz)
        indptr = self.empty((rows + 1,), torch.int64)
        idx = self.empty((nnz,), torch.int64)
        w = self.empty((nnz,), wdt)
        L.check(self.lib.pg_csr_append(_ptr(oip), _ptr(oi), _ptr(ow), _ptr(aip), _ptr(ai), _ptr(aw),
                                       rows, int(col_base), L.W_SIM_F32 if similarity else L.W_I64, _ptr(indptr),
                                       _ptr(idx), _ptr(w), self._stream()))
        return indptr, idx, w

    def hamming_eps(self, own, row0, rows, stream, lut, similarity=False, capture=None):
        """prograph.py:731-753 for own rows [row0,row0+rows): CSR (indptr, idx, w) of the
        stream rows whose distance d has bit d set in `lut` (uint32 words, host).  `capture`:
        the largest degree the caller expects (a degree sample of a dense graph): the count pass
        then keeps every hit and the fill pass is one copy instead of a second sweep."""
        self._check_pair(own, stream)
        lut, lut_p = _host_u32(lut)
        counts = self.empty((rows,), torch.int64)
        cap = int(min(capture, 1 << 20)) if capture else 0
        nbytes = int(self.lib.pg_eps_workspace_bytes_capture(int(rows), int(stream.rows), int(own.words), cap))
        ws = self.empty((nbytes,), torch.uint8)
        L.check(self.lib.pg_hamming_eps_count_capture(_ptr(own.data), own.rows, int(row0), int(rows), _ptr(stream.data),
                                                      stream.rows, own.planes, own.words, lut_p, len(lut), cap,
                                                      _ptr(counts), _ptr(ws), nbytes, self._stream()))
        indptr = self.exclusive_scan(counts)
        nnz = int(indptr[-1].item())
        self.check_edge_budget(nnz)
        weight = L.W_SIM_F32 if similarity else L.W_I64
        idx = self.empty((nnz,), torch.int64)
        w = self.empty((nnz,), torch.float32 if similarity else torch.int64)
        if nnz:
            L.check(self.lib.pg_hamming_eps_fill_capture(_ptr(own.data), own.rows, int(row0), int(rows),
                                                         _ptr(stream.data), stream.rows, own.planes, own.words, lut_p,
                                                         len(lut), cap, _ptr(indptr), weight, _ptr(idx), _ptr(w), _ptr(ws),
                                                         nbytes, self._stream()))
        return indptr, idx, w

    def hamming_eps_degrees(self, own, row0, rows, stream, lut):
        """Number of edges of own rows [row0,row0+rows) (pg_hamming_eps_count without captures): the
        degree census of a graph, whether or not its CSR could be materialised.  (rows,) int64."""
        self._check_pair(own, stream)
        lut, lut_p = _host_u32(lut)
        counts = self.empty((rows,), torch.int64)
        nbytes = int(self.lib.pg_eps_count_workspace_bytes(int(rows), int(stream.rows), int(own.words)))
        ws = self.empty((nbytes,), torch.uint8)
        L.check(self.lib.pg_hamming_eps_count(_ptr(own.data), own.rows, int(row0), int(rows), _ptr(stream.data),
                                              stream.rows, own.planes, own.words, lut_p, len(lut), _ptr(counts),
                                              _ptr(ws), nbytes, self._stream()))
        return counts

    def hamming_eps_mean_degree(self, own, row0, rows, stream, lut):
        """(mean, largest) number of edges per row over a row sample: sizes the edge buffer of the
        symmetric sweep, tells dense graphs apart and sizes their captures."""
        deg = self.hamming_eps_degrees(own, row0, rows, stream, lut)
        total, top = torch.stack([deg.sum(), deg.max()]).tolist()
        return float(total) / rows, int(top)

    def hamming_eps_sym(self, table, lut, rank=0, world=1, mode=0, capacity=None):
        """Symmetric epsilon sweep (pg_hamming_eps_sym): this rank's piece of the triangle of
        unordered pairs; returns (keys, edges): the reserved slots of the edge-key buffer (both
        directions of every passing pair, sentinels -1 in unused slots) and the number of edges
        among them.  Raises Unsupported when `lut` is not one contiguous range of distances."""
        self._sym_check(table)
        if table.rows >= (1 << 27):
            raise L.Unsupported("shape not covered by the symmetric sweep")
        lut, lut_p = _host_u32(lut)
        nbytes = int(self.lib.pg_knn_sym_workspace_bytes(table.rows, table.words))
        ws = self.empty((nbytes,), torch.uint8)
        cap = int(capacity) if capacity is not None else 96 * table.rows // max(1, world) + (4 << 20)
        counters = self.empty((2,), torch.int64)
        for attempt in range(2):
            self.check_edge_budget(cap)
            keys = self.empty((cap,), torch.int64)
            L.check(self.lib.pg_hamming_eps_sym(_ptr(table.data), table.rows, table.planes, table.words, lut_p, len(lut),
                                                int(rank), int(world), int(mode), _ptr(keys), cap, _ptr(counters), _ptr(ws),
                                                nbytes, self._stream()))
            reserved, edges = (int(v) for v in counters.tolist())
            if reserved <= cap:
                return keys[:reserved], edges
            del keys
            cap = reserved                 # the sweep counted what it needs: run it once more
        raise RuntimeError("symmetric epsilon sweep: edge buffer overflow after resizing")

    def edge_keys_to_csr(self, keys, rows, words, nnz, similarity=False):
        """Edge keys (any order, sentinels -1) -> CSR (indptr, idx, w) with rows ascending and, within
        a row, ascending neighbour index (pg_edge_keys_to_csr)."""
        keys = keys.contiguous()
        if keys.numel() >= (1 << 31):
            raise L.Unsupported("edge list too long for one key sort")
        alt = self.empty((keys.numel(),), torch.int64)
        indptr = self.empty((rows + 1,), torch.int64)
        idx = self.empty((nnz,), torch.int64)
        w = self.empty((nnz,), torch.float32 if similarity else torch.int64)
        L.check(self.lib.pg_edge_keys_to_csr(_ptr(keys), keys.numel(), _ptr(alt), int(rows), int(words), int(nnz),
                                             L.W_SIM_F32 if similarity else L.W_I64, _ptr(indptr), _ptr(idx), _ptr(w),
                                             self._stream()))
        return indptr, idx, w

    def hamming_tile(self, data, queries, q0=0, qrows=None, weight=L.W_I64):
        """hamming.py:34-38: (qrows, N) distances of query rows [q0,q0+qrows) vs all data rows."""
        self._check_pair(data, queries)
        qrows = queries.rows - q0 if qrows is None else qrows
        dt = {L.W_I64: torch.int64, L.W_SIM_F32: torch.float32, L.W_I32: torch.int32}[weight]
        out = self.empty((qrows, data.rows), dt)
        L.check(self.lib.pg_hamming_tile(_ptr(data.data), data.rows, _ptr(queries.data), queries.rows, int(q0),
                                         int(qrows), data.planes, data.words, weight, _ptr(out), data.rows,
                                         self._stream()))
        return out

    def hamming_flags(self, data, queries, qrows, d_lo, d_hi):
        """(qrows, N) uint8 flags d_lo <= d(query, row) <= d_hi of the first `qrows` rows of the packed
        `queries` table against every row of `data` (pg_hamming_flags_tile): a batch of neighbourhood
        queries (prograph.py:571-588) in one fused sweep."""
        self._check_pair(data, queries)
        out = self.empty((qrows, data.rows), torch.uint8)
        L.check(self.lib.pg_hamming_flags_tile(_ptr(data.data), data.rows, _ptr(queries.data), queries.rows, 0, int(qrows),
                                               data.planes, data.words, int(d_lo), int(d_hi), _ptr(out), data.rows,
                                               self._stream()))
        return out

    def gather_packed(self, table, rows):
        """The packed rows `rows` (host index array) of `table` as a small PackedTable of its own."""
        idx = torch.as_tensor(np.asarray(rows, dtype=np.int64), device=self.device)
        pad = int(self.lib.pg_packed_rows(len(rows)))
        data = torch.zeros((pad, table.planes, table.words), dtype=torch.int32, device=self.device)
        data[: len(rows)] = table.data[idx]
        return PackedTable(data, len(rows), table.L, table.planes, table.words)

    def flags_or_rows(self, flags, accept, covered):
        """covered |= OR of the rows of `flags` selected by the host mask `accept` (pg_flags_or_rows)."""
        acc = np.ascontiguousarray(accept, dtype=np.uint8)
        rows, n = flags.shape
        for r0 in range(0, rows, 1024):
            part = acc[r0:r0 + 1024]
            L.check(self.lib.pg_flags_or_rows(_ptr(flags[r0:]), len(part), n, int(flags.stride(0)),
                                              part.ctypes.data_as(C.c_void_p), _ptr(covered), self._stream()))
        return covered

    def check_edge_budget(self, nnz):
        """An epsilon graph can be dense (the reference would run out of host memory the same way):
        refuse before allocating instead of taking the GPU down.  cudaMemGetInfo costs anything from
        0.1 to several milliseconds (measured: tools/host_gaps.py), which is a third of a small graph's
        build, so the driver is only asked when the request is a sizeable part of what was free at the
        last look (refreshed at least every few seconds)."""
        import time
        need = nnz * 16
        now = time.monotonic()
        hint = getattr(self, "_free_hint", None)
        if hint is not None and now - hint[1] < 5.0 and need < 0.2 * hint[0]:
            return
        free, _ = torch.cuda.mem_get_info(self.device)
        avail = free + torch.cuda.memory_reserved(self.device) - torch.cuda.memory_allocated(self.device)
        self._free_hint = (avail, now)
        if need > 0.9 * avail:
            raise MemoryError(f"the requested graph has {nnz} edges ({need / 2**30:.1f} GiB as int64 index/weight "
                              f"pairs) and does not fit in device memory; lower eps or build a kNN graph")

    def exclusive_scan(self, counts):
        out = self.empty((counts.numel() + 1,), torch.int64)
        L.check(self.lib.pg_exclusive_scan_i64(_ptr(counts), counts.numel(), _ptr(out), self._stream()))
        return out

    # ---- element-wise tiles ----------------------------------------------------------------
    def minkowski_tile(self, X, Y, q0, qrows, p=2, similarity=False):
        """minkowski.py:36-40 on device tensors X (N,D), Y (M,D) of one dtype in
        {float16, float32, float64, int64}."""
        assert X.dtype == Y.dtype and X.shape[1] == Y.shape[1]
        out_dt = {torch.float16: torch.float16, torch.float32: torch.float32, torch.int64: torch.float32,
                  torch.float64: torch.float64}[X.dtype]
        out = self.empty((qrows, X.shape[0]), out_dt)
        L.check(self.lib.pg_minkowski_tile(_ptr(X), X.shape[0], _ptr(Y), Y.shape[0], int(q0), int(qrows), X.shape[1],
                                           _PG_DTYPE[X.dtype], float(p), 1 if similarity else 0, _ptr(out), X.shape[0],
                                           self._stream()))
        return out

    def hamming_values_tile(self, X, Y, q0, qrows, similarity=False):
        """hamming.py:34-38 on arbitrary numeric values (not packable as tokens)."""
        assert X.dtype == Y.dtype and X.shape[1] == Y.shape[1]
        weight = L.W_SIM_F32 if similarity else L.W_I64
        out = self.empty((qrows, X.shape[0]), torch.float32 if similarity else torch.int64)
        L.check(self.lib.pg_hamming_values_tile(_ptr(X), X.shape[0], _ptr(Y), Y.shape[0], int(q0), int(qrows),
                                                X.shape[1], _PG_DTYPE[X.dtype], weight, _ptr(out), X.shape[0],
                                                self._stream()))
        return out

    # ---- Minkowski p=2 on integer tokens: tcgen05 int8 contraction ---------------------------
    # rows of up to 256 tokens keep their A tiles resident; wider rows stream K-chunks (pg_gemm.cu)
    GEMM_MAX_WIDTH = 8192

    def gemm_pack(self, tokens, max_token=255, K=None):
        """(N, L) integer-valued tokens -> GemmTable; OverflowError if a value is not an integer
        in [0, max_token]; Unsupported for rows wider than the kernel handles."""
        t = self.to_device(tokens)
        if t.dim() != 2 or t.shape[0] == 0 or t.shape[1] == 0:
            raise ValueError("gemm_pack expects a non-empty (N, L) array")
        if t.dtype not in _PG_DTYPE or t.dtype == torch.bool:
            t = t.to(torch.int64)
        N, L_ = int(t.shape[0]), int(t.shape[1])
        K = int(self.lib.pg_gemm_width(L_)) if K is None else int(K)
        if K > self.GEMM_MAX_WIDTH:
            raise L.Unsupported(f"rows wider than {self.GEMM_MAX_WIDTH} tokens take the element-wise kernel")
        rows_pad = int(self.lib.pg_gemm_rows(N))
        data = self.empty((rows_pad * K,), torch.uint8)
        norms = self.empty((rows_pad,), torch.int32)
        flag = torch.zeros((1,), dtype=torch.int32, device=self.device)
        L.check(self.lib.pg_gemm_pack(_ptr(t), _PG_DTYPE[t.dtype], N, L_, int(t.stride(0)), _ptr(data), _ptr(norms), K,
                                      int(max_token), _ptr(flag), self._stream()))
        if int(flag.item()):
            raise OverflowError(f"values are not integer tokens in [0, {max_token}]")
        return GemmTable(data, norms, N, L_, K, max_token)

    def minkowski2_gemm_tile(self, data, queries, value_kind, similarity=False):
        """(M, N) Minkowski p=2 matrix of integer-token tables (minkowski.py:36-40);
        value_kind 0 -> fp16 chain, 1 -> float32 root of the exact integer sum."""
        assert data.K == queries.K
        out = self.empty((queries.rows, data.rows), torch.float16 if value_kind == 0 else torch.float32)
        L.check(self.lib.pg_minkowski2_gemm_tile(_ptr(queries.data), _ptr(queries.norms), queries.rows, _ptr(data.data),
                                                 _ptr(data.norms), data.rows, data.K, int(value_kind),
                                                 1 if similarity else 0, _ptr(out), data.rows, self._stream()))
        return out

    def minkowski2_gemm_knn(self, data, queries, k, drop, value_kind, similarity=False):
        """Fused Minkowski p=2 kNN of every query row against `data` (prograph.py:755-765)."""
        assert data.K == queries.K
        idx = self.empty((queries.rows, k), torch.int64)
        val = self.empty((queries.rows, k), torch.float16 if value_kind == 0 else torch.float32)
        L.check(self.lib.pg_minkowski2_gemm_knn(_ptr(queries.data), _ptr(queries.norms), queries.rows, _ptr(data.data),
                                                _ptr(data.norms), data.rows, data.K, int(value_kind),
                                                1 if similarity else 0, int(k), int(drop), _ptr(idx), _ptr(val),
                                                self._stream()))
        return idx, val

    def minkowski2_gemm_eps(self, data, queries, s_lo, s_hi, value_kind, similarity=False):
        """Fused Minkowski p=2 epsilon graph: CSR (indptr, idx, val) of the dataset rows whose exact
        integer sum S lies in [s_lo, s_hi] (the caller derives the range from comp / eps)."""
        assert data.K == queries.K
        M = queries.rows
        gc = self.empty((2 * M,), torch.int64)
        counts = self.empty((M,), torch.int64)
        L.check(self.lib.pg_minkowski2_gemm_eps_count(_ptr(queries.data), _ptr(queries.norms), M, _ptr(data.data),
                                                      _ptr(data.norms), data.rows, data.K, int(s_lo), int(s_hi), _ptr(gc),
                                                      _ptr(counts), self._stream()))
        indptr = self.exclusive_scan(counts)
        nnz = int(indptr[-1].item())
        self.check_edge_budget(nnz)
        idx = self.empty((nnz,), torch.int64)
        val = self.empty((nnz,), torch.float16 if value_kind == 0 else torch.float32)
        if nnz:
            L.check(self.lib.pg_minkowski2_gemm_eps_fill(_ptr(queries.data), _ptr(queries.norms), M, _ptr(data.data),
                                                         _ptr(data.norms), data.rows, data.K, int(value_kind),
                                                         1 if similarity else 0, int(s_lo), int(s_hi), _ptr(gc),
                                                         _ptr(indptr), _ptr(idx), _ptr(val), self._stream()))
        return indptr, idx, val

    # ---- tile consumers ----------------------------------------------------------------------
    def tile_topk(self, tile, k, drop=1, descending=False):
        rows, N = tile.shape
        idx = self.empty((rows, k), torch.int64)
        val = self.empty((rows, k), tile.dtype)
        L.check(self.lib.pg_tile_topk(_ptr(tile), _PG_DTYPE[tile.dtype], rows, N, int(tile.stride(0)), int(k), int(drop),
                                      1 if descending else 0, _ptr(idx), _ptr(val), self._stream()))
        return idx, val

    @staticmethod
    def _thresh_guard(eps, guard):
        """`guard` with L.EPS_FLOAT set when eps is a python float: torch compares an integer tile
        with an int exactly and with a float in float32 (pg_tile_threshold_count)."""
        return int(guard) | (0 if isinstance(eps, numbers.Integral) else L.EPS_FLOAT)

    def tile_threshold_counts(self, tile, cmp, eps, swap=False, guard=0):
        """Per-row number of tile entries passing the threshold test (pg_tile_threshold_count)."""
        rows, N = tile.shape
        counts = self.empty((rows,), torch.int64)
        L.check(self.lib.pg_tile_threshold_count(_ptr(tile), _PG_DTYPE[tile.dtype], rows, N, int(tile.stride(0)), int(cmp),
                                                 float(eps), 1 if swap else 0, self._thresh_guard(eps, guard), _ptr(counts),
                                                 self._stream()))
        return counts

    def tile_threshold(self, tile, cmp, eps, swap=False, guard=0, values=True):
        """CSR of the tile entries passing the threshold test (see pg_tile_threshold_count)."""
        rows, N = tile.shape
        dt = _PG_DTYPE[tile.dtype]
        guard = self._thresh_guard(eps, guard)
        counts = self.empty((rows,), torch.int64)
        L.check(self.lib.pg_tile_threshold_count(_ptr(tile), dt, rows, N, int(tile.stride(0)), int(cmp), float(eps),
                                                 1 if swap else 0, guard, _ptr(counts), self._stream()))
        indptr = self.exclusive_scan(counts)
        nnz = int(indptr[-1].item())
        self.check_edge_budget(nnz)
        idx = self.empty((nnz,), torch.int64)
        val = self.empty((nnz,), tile.dtype) if values else None
        if nnz:
            L.check(self.lib.pg_tile_threshold_fill(_ptr(tile), dt, rows, N, int(tile.stride(0)), int(cmp), float(eps),
                                                    1 if swap else 0, guard, _ptr(indptr), _ptr(idx), _ptr(val),
                                                    self._stream()))
        return indptr, idx, val

    # ---- masks ------------------------------------------------------------------------------
    def mutant_bits(self, table, ref):
        """ref: packed row tensor (planes*words int32) on the device."""
        mut = self.empty((table.rows, table.words), torch.int32)
        L.check(self.lib.pg_mutant_bits(_ptr(table.data), table.rows, table.planes, table.words, _ptr(ref), _ptr(mut),
                                        self._stream()))
        return mut

    def mutant_bool(self, table, ref):
        out = self.empty((table.rows, table.L), torch.uint8)
        L.check(self.lib.pg_mutant_bool(_ptr(table.data), table.rows, table.planes, table.words, table.L, _ptr(ref),
                                        _ptr(out), self._stream()))
        return out

    def mutant_any(self, mut):
        out = self.empty((mut.shape[1],), torch.int32)
        L.check(self.lib.pg_mutant_any(_ptr(mut), mut.shape[0], mut.shape[1], _ptr(out), self._stream()))
        return out.cpu().numpy().view(np.uint32)

    def select_rows(self, mut, dist_lut=None, inside=None, outside=None, pos_mode=0):
        flag = self.empty((mut.shape[0],), torch.uint8)
        lut_p, lut_n, keep = C.c_void_p(0), 0, []
        if dist_lut is not None:
            a, lut_p = _host_u32(dist_lut)
            lut_n = len(a)
            keep.append(a)
        in_p = C.c_void_p(0)
        if inside is not None:
            b, in_p = _host_u32(inside)
            keep.append(b)
        out_p = C.c_void_p(0)
        if outside is not None:
            c, out_p = _host_u32(outside)
            keep.append(c)
        L.check(self.lib.pg_select_rows(_ptr(mut), mut.shape[0], mut.shape[1], lut_p, lut_n, in_p, out_p,
                                        int(pos_mode), _ptr(flag), self._stream()))
        return flag

    def flag_indices(self, flag):
        n = flag.numel()
        out = self.empty((n,), torch.int64)
        cnt = self.empty((1,), torch.int64)
        L.check(self.lib.pg_flag_indices(_ptr(flag), n, _ptr(out), _ptr(cnt), self._stream()))
        return out[: int(cnt.item())]

    def distance_hist(self, mut):
        hist = torch.zeros((mut.shape[1] * 32 + 1,), dtype=torch.int64, device=self.device)
        L.check(self.lib.pg_distance_hist(_ptr(mut), mut.shape[0], mut.shape[1], _ptr(hist), self._stream()))
        return hist.cpu().numpy()

    # ---- measurement -------------------------------------------------------------------------
    def int_peak(self, mix=0, iters=4096):
        ops, ms = C.c_double(0), C.c_double(0)
        L.check(self.lib.pg_measure_int_peak(int(mix), int(iters), C.byref(ops), C.byref(ms)))
        return ops.value, ms.value

    def i8_mma_peak(self, batches=256):
        """int8 operations per second of back-to-back tcgen05 MMAs on resident operands (pg_measure_i8_mma_peak)."""
        ops, ms = C.c_double(0), C.c_double(0)
        L.check(self.lib.pg_measure_i8_mma_peak(int(batches), C.byref(ops), C.byref(ms)))
        return ops.value, ms.value

    def time_sweeps(self, enable=True):
        self.lib.pg_time_sweeps(1 if enable else 0)

    def sweep_time(self, reset=True):
        ms, n = C.c_double(0), C.c_int64(0)
        self.lib.pg_sweep_time(C.byref(ms), C.byref(n), 1 if reset else 0)
        return ms.value, n.value

    def sweep_times(self, reset=True, cap=4096):
        """Per-launch times (ms) of the timed sweeps, in launch order."""
        buf = (C.c_double * cap)()
        n = C.c_int64(0)
        self.lib.pg_sweep_times(buf, cap, C.byref(n), 1 if reset else 0)
        return [buf[i] for i in range(min(cap, n.value))]


def sym_plan(rows, planes, words, boot_rows=0, rank=0, world=1, mode=0, grid=296):
    """Host-only planner of the symmetric sweeps (no GPU needed): (n_items, 5) int32 array of
    (row block, first tile, end tile, boot flag, CTA) -- every CTA walks its items in this order."""
    lib = L.load()
    n = C.c_int64(0)
    L.check(lib.pg_knn_sym_plan(int(rows), int(planes), int(words), int(boot_rows), int(rank), int(world), int(mode),
                                int(grid), None, 0, C.byref(n)))
    items = np.zeros((n.value, 5), dtype=np.int32)
    L.check(lib.pg_knn_sym_plan(int(rows), int(planes), int(words), int(boot_rows), int(rank), int(world), int(mode),
                                int(grid), items.ctypes.data_as(C.c_void_p), n.value, C.byref(n)))
    return items


_ENGINE = None


def get_engine():
    """The process-wide CUDA engine (created on first use)."""
    global _ENGINE
    if _ENGINE is None:
        _ENGINE = CudaEngine()
    return _ENGINE


def set_engine(engine):
    """Install another engine object (tests inject a checker-backed one to exercise the
    host logic on machines without a GPU).  Returns the previous engine."""
    global _ENGINE
    prev, _ENGINE = _ENGINE, engine
    return prev
