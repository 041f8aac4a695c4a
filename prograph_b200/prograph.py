"""``Prograph``: host-side mirror of the reference class for the graph-construction path.

Same constructor, ``__call__`` / ``__getitem__`` access, pandas-frame storage and method
names as prograph/prograph.py:24-946; everything that touches pairwise distances, neighbour
lists or mutation masks runs on the GPU through libprograph_b200.so:

    build_graph                       prograph.py:656-765   fused sweeps / tile kernels
    calc_neighbours, neighbourhood,   prograph.py:526-588   packed one-row queries
    nearest_neighbour, __str__        prograph.py:546-569, 147
    indexing, positions, distances,   prograph.py:242-343   mask kernels + compaction
    get_mutated_positions,            prograph.py:349-368
    boolean_mutant_array,             prograph.py:488-492
    calc_mutated_positions            prograph.py:494-505
    degree, get_neighbour_coords,     prograph.py:797-897   CSR-native (no per-row loops)
    adjacency, laplacian

The ML adapters (sklearn / pytorch loaders, fit), networkx export, dirichlet / local_variance of
the reference are outside this path and are not re-implemented: when the reference package is
importable next to this one, those methods are the reference's own, bound to this object
(``__getattr__``), so ``pg("sklearn")``, ``pg.fit(...)`` etc. keep working on the GPU-built graph;
without it they raise with a message that says so.
"""
import operator

import numpy as np
import pandas as pd
import torch
from scipy import sparse

from . import graph as _graph
from .distance import hamming, minkowski  # noqa: F401  (re-exported for drop-in imports)
from .distance.hamming import hamming_matrix
from .engine import get_engine, sweep_covers
from .protein import Protein

_MISSING = "This sequence is not in the dataset."


def _reference_class():
    """The reference's own ``Prograph`` class when acmater/prograph is installed beside this package
    (everything outside the graph-construction path stays its code), else None."""
    try:
        import prograph as _ref
        return getattr(_ref, "Prograph", None)
    except Exception:           # not installed, or one of its optional imports is missing
        return None


class Prograph:
    """A protein dataset stored as a pandas frame plus its neighbour graph.

    Parameters (prograph.py:96-101)
    ----------
    file : str
        ``.csv`` with a sequence column and label columns, or a pickled frame (``.pkl``).
    seed_seq : str, optional
        Seed (wild-type) sequence; defaults to the first row.
    seqs_col : str, default "Sequence"
    columns : list of str, default ["Fitness"]
    index_col : int or str, default 0
    amino_acids : str, default 'ACDEFGHIKLMNPQRSTVWY'
        Alphabet; letter i maps to token i+1, 0 pads shorter sequences.
    """

    def __init__(self, file, seed_seq=None, seqs_col="Sequence", columns=["Fitness"], index_col=0,
                 amino_acids="ACDEFGHIKLMNPQRSTVWY"):
        try:
            ext = file.split(".")[-1]
            if ext == "csv":
                self.graph = self.csvDataLoader(file, seqs_col=seqs_col, columns=columns, index_col=index_col)
            elif ext == "pkl":
                self.graph = pd.read_pickle(file)
            else:
                raise ValueError(ext)
        except Exception:
            raise FileNotFoundError("File could not be opened")          # prograph.py:109-110

        self.file = file
        self.seed_seq = seed_seq
        self.seqs_col = seqs_col
        self.columns = columns
        self.index_col = index_col
        self.amino_acids = amino_acids

        self.seed = Protein(seed_seq) if seed_seq else Protein(**self.graph.loc[0])
        self.seq_len = len(self.seed)
        self.len = len(self)

        self.tokens = {aa.encode("utf-8"): i + 1 for i, aa in enumerate(self.amino_acids)}
        self.tokenized = self.tokenize(self.graph[seqs_col])
        self.seq_idxs = {seq: idx for idx, seq in enumerate(self.graph[seqs_col])}
        self._token_dict = None
        self._packed = None          # device bit planes of self.tokenized
        self._tables = {}            # id(first tuple) -> (first tuple, CSR table) of recent builds

        self.mutated_positions = self.calc_mutated_positions()
        self.sequence_mutation_locations = self.boolean_mutant_array(self.seed.Sequence)

        if "Tokenized" not in self.graph:
            self.graph["Tokenized"] = [row for row in self.tokenized]
        if "Neighbours" not in self.graph:
            self.graph["Neighbours"] = self.build_graph(eps=1)             # prograph.py:140-141

        if file.split(".")[-1] == "pkl":
            from .io import attach_sidecar
            attach_sidecar(self, file)

        self.learners = {}
        print(self)

    # ------------------------------------------------------------------ basics
    @property
    def token_dict(self):
        """{tuple(tokens): row index}; built on first use (prograph.py:131)."""
        if self._token_dict is None:
            self._token_dict = {tuple(seq): idx for idx, seq in enumerate(self.tokenized)}
        return self._token_dict

    def __str__(self):
        hist = self._distance_hist(self.query(self.seed.Sequence))
        present = np.nonzero(hist)[0]
        return f"""
            Prograph
            Number of Sequences : {len(self)}
            Max Distance        : {int(present.max())}
            Longest Sequence    : {np.max([len(x) for x in self("Sequence")])}
            Number of Distances : {len(present)}
            Seed Sequence       : {self.coloured_seed_string()}
                Modified positions are shown in green"""

    def __repr__(self):
        return (f"Prograph(file={self.file}, seed_seq='{self.seed.Sequence}', seqs_col='{self.seqs_col}', "
                f"columns={self.columns}, index_col={self.index_col}, amino_acids='{self.amino_acids}')")

    def __len__(self):
        return len(self.graph)

    def __getitem__(self, idx):
        return self.graph.iloc[self.query(idx)]

    def __call__(self, label=None, **kwargs):
        return self.label_iter(label, **kwargs)

    def label_iter(self, label, **kwargs):
        """A copy of one frame column (or of the whole frame for ``None``); "pytorch" / "sklearn" hand
        over to the reference's data adapters (prograph.py:185-202)."""
        if label == "pytorch":
            return self.pytorch_dataloaders(**kwargs)
        if label == "sklearn":
            return self.sklearn_data(**kwargs)
        if label is None:
            return self.graph.copy()
        return self.graph[label].copy()

    def __getattr__(self, name):
        """Methods outside the graph-construction path (sklearn_data, pytorch_dataloaders, fit,
        graph_to_networkx, dirichlet, local_variance, ...) are the reference's own, bound to this
        object, when the reference package is importable."""
        if name.startswith("__") or name in ("graph", "tokenized"):
            raise AttributeError(name)
        ref = _reference_class()
        if ref is not None and hasattr(ref, name):
            attr = getattr(ref, name)
            return attr.__get__(self, type(self)) if hasattr(attr, "__get__") else attr
        raise AttributeError(f"{type(self).__name__!s} has no attribute {name!r}: it is outside the graph-construction "
                             "path of prograph_b200 and the reference package (acmater/prograph) is not importable")

    def query(self, sequence):
        """Row index (or indices) for an int, str, token tuple, list or array (prograph.py:204-240)."""
        if isinstance(sequence, (int, np.integer)):
            assert sequence <= self.len, "Index exceeds bounds of dataset"
            return sequence
        if isinstance(sequence, (np.ndarray, list)):
            first = sequence[0]
            if isinstance(first, (int, np.integer, np.bool_)):
                return sequence
            if isinstance(first, str):
                return [self.seq_idxs.get(seq, _MISSING) for seq in sequence]
            print("Wrong data format in numpy array or list iterable.")
            return None
        if isinstance(sequence, str):
            return self.seq_idxs.get(sequence, _MISSING)
        if isinstance(sequence, tuple):
            assert len(sequence) == self.seq_len, "Tuple not valid length for dataset."
            hits = np.where(np.all(np.asarray(sequence) == self.tokenized, axis=1))[0]
            assert len(hits) > 0, "Not a valid tuple representation of a protein in this dataset."
            return int(hits[0])
        raise ValueError("Input format not understood.")

    @staticmethod
    def csvDataLoader(csvfile, seqs_col, columns="all", index_col=None):
        """Load the sequence column, the requested label columns and, if present, a stored
        ``Neighbours`` column (prograph.py:401-435)."""
        data = pd.read_csv(csvfile, index_col=index_col)
        if columns == "all":
            columns = [c for c in data.keys() if c != seqs_col]
        columns = [seqs_col] + list(columns)
        if "Neighbours" in data:
            columns += ["Neighbours"]
        return data[columns]

    # ------------------------------------------------------------------ tokens
    def custom_tokenize(self, seq, tokenizer=None):
        if tokenizer is None:
            return np.array([self.tokens[aa.encode("utf-8")] for aa in seq])
        return "This feature is not ready yet"

    def _letter_table(self):
        """Byte -> token table of the tokeniser kernels: one byte per letter, tokens below 256."""
        assert len(self.amino_acids) < 256, "alphabets of 256 or more letters do not fit one-byte tokens"
        table = np.zeros(256, dtype=np.uint8)
        for ch, tok in self.tokens.items():
            assert len(ch) == 1, f"letter {ch!r} is not a single byte: the device tokeniser works on bytes"
            table[ch[0]] = tok
        return table

    @staticmethod
    def _letter_codes(sequences):
        """(N, L) uint8 matrix of the sequences' bytes, zero padded to the longest one."""
        chars = np.array(sequences, dtype="bytes").reshape(-1, 1).view("S1")
        return chars.view(np.uint8).reshape(chars.shape) if chars.size else np.zeros(chars.shape, np.uint8)

    def tokenize(self, sequences):
        """Letters -> 1..len(alphabet) through a 256-entry byte table; shorter sequences are
        right-padded with 0 (prograph.py:454-474 semantics, one pass instead of 20)."""
        return self._letter_table().astype(np.int64)[self._letter_codes(sequences)]

    def embedding(self, embedded, name):
        self.graph[f"{name}_embedded"] = embedded

    def _device_tokens(self):
        """Bit planes of the dataset on the device, packed straight from the sequence letters
        (tokenise + pack fused, pg_pack_chars) -- one byte per residue crosses PCIe."""
        if self._packed is None or self._packed.rows != len(self.tokenized):
            planes = 5 if len(self.amino_acids) < 32 else 8
            self._packed = get_engine().pack_chars(self._letter_codes(self.graph[self.seqs_col]),
                                                   self._letter_table(), planes=planes)
        return self._packed

    def _mutant_bits(self, row):
        """Device bit mask (N, words) of the residues differing from dataset row `row`."""
        table = self._device_tokens()
        return get_engine().mutant_bits(table, table.row(int(row)))

    def _distance_hist(self, row):
        return get_engine().distance_hist(self._mutant_bits(row))[: self.tokenized.shape[1] + 1]

    # ------------------------------------------------------------------ masks
    def boolean_mutant_array(self, seq=None):
        """(N, L) bool: residue differs from the given dataset sequence (prograph.py:488-492)."""
        table = self._device_tokens()
        out = get_engine().mutant_bool(table, table.row(int(self.query(seq))))
        return out.cpu().numpy().view(np.bool_)

    def calc_mutated_positions(self):
        """Positions at which any sequence differs from the seed (prograph.py:494-505)."""
        eng = get_engine()
        table = self._device_tokens()
        seed_tok = self.tokenize(self.seed.Sequence)
        if seed_tok.shape[1] != self.tokenized.shape[1]:
            raise ValueError("seed sequence length differs from the tokenised width")
        seed = eng.pack(seed_tok.astype(np.int64), planes=table.planes, words=table.words)
        any_bits = eng.mutant_any(eng.mutant_bits(table, seed.row(0)))
        L_ = len(self.seed)
        pos = [l for l in range(L_) if (any_bits[l >> 5] >> np.uint32(l & 31)) & np.uint32(1)]
        return np.array(pos, dtype=np.int64)

    def coloured_seed_string(self):
        green, reset = "\033[32m", "\033[0m"
        marked = set(int(i) for i in self.mutated_positions)
        return "".join(f"{green}{c}{reset}" if i in marked else c for i, c in enumerate(self.seed.Sequence))

    def positions(self, positions):
        return self.indexing(positions=positions)

    def distances(self, distances):
        return self.indexing(distances=distances)

    @staticmethod
    def _position_words(positions, n_words):
        words = np.zeros(n_words, dtype=np.uint32)
        for pos in positions:
            pos = int(pos)
            if pos < 0 or pos >= n_words * 32:
                raise IndexError(f"position {pos} is out of bounds")
            words[pos >> 5] |= np.uint32(1) << np.uint32(pos & 31)
        return words

    def indexing(self, reference_seq=None, distances=None, positions=None, percentage=None, Bool="or",
                 complement=False):
        """Row indices selected by Hamming distance from a reference sequence and / or by the
        set of mutated positions (prograph.py:254-343).

        distances : int or list of int -- keep rows at exactly these distances; each must occur.
        positions : list of int -- keep rows mutated *only* inside these positions: at least
            one of them for ``Bool="or"``, all of them for ``"and"``.
        percentage : float in [0, 1] -- random sub-sample of the selection (global numpy RNG).
        complement : also return the unselected indices.
        """
        assert Bool == "or" or Bool == "and", "Not a valid boolean value."
        if reference_seq is None:
            reference_seq = self.seed.Sequence
        eng = get_engine()
        n = len(self)
        flag = None
        if distances is not None or positions is not None:
            ref_row = self.query(reference_seq)
            mut = self._mutant_bits(ref_row)
            n_words = mut.shape[1]
            lut = None
            if distances is not None:
                if type(distances) == int:
                    distances = [distances]
                assert type(distances) == list, "Distances must be provided as integer or list"
                hist = eng.distance_hist(mut)
                lut = np.zeros(n_words + 1, dtype=np.uint32)
                for d in distances:
                    assert 0 <= d < len(hist) and hist[d] > 0, f"{d} is not a valid distance"
                    lut[d >> 5] |= np.uint32(1) << np.uint32(d & 31)
            inside = outside = None
            mode = 0
            if positions is not None:
                # only positions inside the reference sequence's own length are checked for
                # "unchanged" (prograph.py:316 ranges over len(reference sequence))
                ref_len = len(self[reference_seq]["Sequence"])
                inside = self._position_words(positions, n_words)
                chosen = set(int(p) for p in positions)
                outside = self._position_words([x for x in range(ref_len) if x not in chosen], n_words)
                mode = 1 if Bool == "or" else 2
            flag = eng.select_rows(mut, dist_lut=lut, inside=inside, outside=outside, pos_mode=mode)
            idxs = eng.flag_indices(flag).cpu().numpy()
        else:
            idxs = np.array(range(n))

        if percentage is not None:
            assert 0 <= percentage <= 1, "Percentage must be between 0 and 1"
            pick = np.zeros(len(idxs), dtype=bool)
            pick[np.random.choice(np.arange(len(idxs)), size=int(len(idxs) * percentage), replace=False)] = 1
            return idxs[pick]

        assert len(idxs) != 0, "No possible valid indices have been provided."
        if complement:
            if flag is None:
                return idxs, np.array([], dtype=idxs.dtype)
            rest = eng.flag_indices((flag ^ 1).contiguous()).cpu().numpy()
            return idxs, rest
        return idxs

    def get_mutated_positions(self, positions):
        """(N,) bool: rows whose mutations avoid every dataset-mutated position *other* than
        the given ones (prograph.py:349-368)."""
        for pos in positions:
            assert pos in self.mutated_positions, "{} is not a position that was mutated in this dataset".format(pos)
        constants = np.setdiff1d(self.mutated_positions, positions)
        mut = self._mutant_bits(self.query(self.seed.Sequence))
        inside = self._position_words(constants, mut.shape[1])
        flag = get_engine().select_rows(mut, inside=inside, pos_mode=3)
        return flag.cpu().numpy().view(np.bool_)

    # ------------------------------------------------------------------ queries
    def _hamming_flag(self, row, comp, eps):
        """Device flag (N,) of comp(d(row, .), eps) for the Hamming distance."""
        mut = self._mutant_bits(row)
        lut = _graph.distance_lut(mut.shape[1] * 32, comp, eps, similarity=False, guard=False)
        return get_engine().select_rows(mut, dist_lut=lut)

    def calc_neighbours(self, seq, eps=1, distance=hamming, comp=operator.eq, weights=False):
        """Column indices j with ``comp(distance(seq, j), eps)`` (prograph.py:526-544; no d>0
        filter here, so the sequence itself appears for ``eps=0``)."""
        row = self.query(seq)
        if distance is hamming:
            return get_engine().flag_indices(self._hamming_flag(row, comp, eps)).cpu().numpy()
        d = distance(self.tokenized, self.tokenized[row].reshape(1, -1))
        return np.where(np.asarray(torch.as_tensor(comp(d, eps)).cpu()))[1]

    def nearest_neighbour(self, seq, distance=hamming, batch_size=8):
        """Closest dataset row to every query sequence and the overall minimum distance (the
        intended behaviour of prograph.py:546-569, whose shipped body stops on a NameError)."""
        queries = self.tokenize(seq)
        if distance is hamming:
            eng = get_engine()
            table = self._device_tokens()
            width = max(queries.shape[1], self.tokenized.shape[1])
            if eng.packed_words(width) == table.words and queries.max(initial=0) < (1 << table.planes) and \
                    sweep_covers(table.planes, table.words):
                q = eng.pack(queries, planes=table.planes, words=table.words)
                idx, d = eng.hamming_knn(q, 0, q.rows, table, 1, drop=0)
                idx, d = idx.cpu().numpy()[:, 0], d.cpu().numpy()[:, 0]
                return self[idx], d.min()
        d = torch.as_tensor(distance(self.tokenized, queries)).cpu().numpy()
        return self[np.argmin(d, axis=1)], np.min(d)

    def neighbourhood(self, seq, eps, distance=hamming):
        """Frame rows within Hamming distance ``eps`` of a sequence (prograph.py:571-588; the
        reference ignores ``distance`` here and so does this)."""
        flag = self._hamming_flag(self.query(seq), operator.le, eps)
        return self[flag.cpu().numpy().view(np.bool_)]

    def neighbourhood_clustering(self, eps, distance=hamming, batch=128):
        """Greedy cover: walk the sequences in order, every uncovered one seeds the cluster of its
        eps-neighbourhood (prograph.py:590-615; clusters may overlap, as in the reference).

        The reference asks for one neighbourhood per seed.  Here the next `batch` uncovered rows form
        a frontier whose neighbourhood flags come out of ONE fused sweep (pg_hamming_flags_tile); the
        greedy order inside the frontier is then resolved on its batch x batch corner -- a frontier row
        that an earlier seed of the same batch covers is no seed -- and the member lists of the seeds are
        compacted in one pass.  Sequences of more than 32768 residues are not covered by the fused sweep
        and raise Unsupported."""
        eng = get_engine()
        table = self._device_tokens()
        n = len(self)
        hi = int(np.floor(eps)) if eps >= 0 else -1                 # integer distances: d <= eps
        covered_dev = torch.zeros(n, dtype=torch.uint8, device=eng.device)
        covered = np.zeros(n, dtype=bool)
        clusters = {}
        start = 0
        while start < n:
            rest = np.nonzero(~covered[start:])[0]
            if len(rest) == 0:
                break
            front = rest[:batch] + start
            flags = eng.hamming_flags(table, eng.gather_packed(table, front), len(front), 0, hi)
            corner = flags[:, torch.as_tensor(front, device=eng.device)].cpu().numpy().astype(bool)   # [seed, frontier row]
            accept = np.zeros(len(front), dtype=np.uint8)
            taken = np.zeros(len(front), dtype=bool)                 # frontier rows covered inside this batch
            for b in range(len(front)):
                if not taken[b]:
                    accept[b] = 1
                    taken |= corner[b]
            seeds = np.nonzero(accept)[0]
            flat = eng.flag_indices(flags[torch.as_tensor(seeds, device=eng.device)].reshape(-1)).cpu().numpy()
            which, members = np.divmod(flat, n)
            bounds = np.searchsorted(which, np.arange(len(seeds) + 1))
            for s_i, b in enumerate(seeds):
                clusters[int(front[b])] = self.graph.iloc[members[bounds[s_i]:bounds[s_i + 1]]]
            eng.flags_or_rows(flags, accept, covered_dev)
            covered = covered_dev.cpu().numpy().astype(bool)
            start = int(front[-1]) + 1
        return clusters

    @staticmethod
    def get_every_n(a, n=2):
        """Chunks of n rows, the last one possibly shorter (prograph.py:617-624)."""
        for i in range(-(-a.shape[0] // n)):
            yield a[n * i:n * (i + 1)]

    # ------------------------------------------------------------------ graph build
    def build_graph(self, idxs=None, batch_size=8, eps=None, k=None, weighted=False, similarity=False,
                    representation="Tokenized", distance=hamming, comp=operator.le):
        """Neighbour lists of every node: epsilon graph (``eps``) or kNN graph (``k``).

        Same arguments, validation and return value as prograph.py:656-765: a list with one
        ``(indices int64, weights)`` tuple per node; indices are relative to ``idxs`` when a
        sub-graph is requested; ``weighted`` is accepted and unused like in the reference;
        kNN ties are ordered by (distance, index) and sorted position 0 is dropped.
        """
        _graph.validate(eps, k)
        if representation == "Tokenized" and len(self.tokenized) == len(self.graph):
            rep = self.tokenized
        else:
            rep = self(representation)
        packed = None
        if representation == "Tokenized" and idxs is None and distance is hamming and rep is self.tokenized:
            packed = self._device_tokens()       # already on the device, packed from the letters
        table = _graph.build_neighbours(rep, eps=eps, k=k, similarity=similarity, distance=distance, comp=comp,
                                        batch_size=batch_size, idxs=idxs, packed=packed)
        lists = table.as_list()
        self._remember(table if isinstance(table, _graph.NeighbourTable) else table.to_csr(), lists)
        return lists

    # ------------------------------------------------------------------ CSR-native exports
    def _remember(self, table, lists):
        """Keep the CSR arrays of recent builds so that the exports below need no per-row
        loop; a frame column is matched to its table by the identity of its first tuple."""
        if lists:
            self._tables[id(lists[0])] = (lists[0], table)
            while len(self._tables) > 8:
                self._tables.pop(next(iter(self._tables)))

    def _table_for(self, graph):
        """CSR arrays of a graph column (cached table of the build that produced it, else a
        flattening of the lists the column holds)."""
        col = self.graph[graph]
        if len(col):
            hit = self._tables.get(id(col.iloc[0]))
            if hit is not None and hit[0] is col.iloc[0] and hit[1].n_rows == len(col):
                return hit[1]
        lists = list(col)
        indptr = np.zeros(len(lists) + 1, dtype=np.int64)
        if lists:
            np.cumsum([len(x[0]) for x in lists], out=indptr[1:])
        idx = np.concatenate([np.asarray(x[0], dtype=np.int64) for x in lists]) if lists else np.zeros(0, np.int64)
        ws = [np.asarray(x[1]) for x in lists if len(x[1])]
        w = np.concatenate(ws) if ws else np.zeros(0, np.int64)
        return _graph.NeighbourTable(indptr, idx, w)

    def degree(self, graph="Neighbours", boolean_weights=False):
        """Out-degree of every node: neighbour count, or the float32 sum of edge weights
        (prograph.py:797-821)."""
        t = self._table_for(graph)
        if boolean_weights:
            return t.degrees().astype(np.float32)
        return _graph.row_sums_f32(t.indptr, t.w)

    def get_neighbour_coords(self, graph="Neighbours", boolean_weights=False):
        """COO coordinates (I, J, weights) of the adjacency (prograph.py:823-853)."""
        t = self._table_for(graph)
        I = np.repeat(np.arange(t.n_rows), t.degrees())
        if boolean_weights:
            return I, t.idx, np.ones(I.shape)
        return I, t.idx, t.w.astype(np.float32)

    def adjacency(self, graph="Neighbours", boolean_weights=False):
        I, J, V = self.get_neighbour_coords(graph=graph, boolean_weights=boolean_weights)
        return sparse.coo_matrix((V, (I, J)), shape=(len(self), len(self)))

    def laplacian(self, graph="Neighbours", boolean_weights=False, mode="outdegree"):
        """Graph Laplacian D - A as a sparse matrix (prograph.py:872-897)."""
        Lm = (-1) * self.adjacency(graph, boolean_weights)
        if mode == "outdegree":
            D = self.degree(graph, boolean_weights)
        elif mode == "indegree":
            D = (-1) * np.array(Lm.sum(0)).reshape(-1,)
        else:
            raise ValueError("Not a valid degree mode.")
        Lm = Lm.tolil() if not hasattr(Lm, "setdiag") else Lm
        Lm.setdiag(D)
        return Lm
