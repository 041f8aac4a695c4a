"""Host-side rules of the chunked long-row Hamming sweep (no GPU needed): the width predicate every
dispatch site shares, and the argument check of the C entries beyond 32768 residues.  Only shapes
the library rejects are passed to it: a supported shape would reach CUDA."""
import ctypes as C

import pytest

from prograph_b200 import _lib
from prograph_b200.engine import SWEEP_MAX_WORDS, sweep_covers


def test_sweep_covers_edges():
    assert SWEEP_MAX_WORDS == 1024
    for planes in (5, 8):
        for words in (1, 2, 4, 8, 16, 24, 56, 64, 72, 1016, 1024):
            assert sweep_covers(planes, words), (planes, words)
        for words in (0, 3, 5, 12, 20, 60, 1025, 1032, 2048):
            assert not sweep_covers(planes, words), (planes, words)
    for planes in (1, 4, 6, 7, 9):
        assert not sweep_covers(planes, 8)


def test_sweep_covers_every_packed_width_up_to_32768_residues():
    lib = _lib.load()
    for L in (1, 32, 33, 128, 129, 256, 257, 1792, 1793, 2048, 2049, 4096, 32767, 32768):
        w = lib.pg_packed_words(L)
        assert sweep_covers(5, w) and sweep_covers(8, w), (L, w)
    for L in (32769, 40000, 65536):
        w = lib.pg_packed_words(L)
        assert not sweep_covers(5, w) and not sweep_covers(8, w), (L, w)


@pytest.mark.parametrize("planes", [5, 8])
def test_sweep_entries_reject_rows_beyond_32768_residues(planes):
    """W = 1032 (32769..33024 residues) is PG_ERR_UNSUPPORTED at both plane counts, from the argument
    check that runs before any device call (the pointers are never dereferenced)."""
    lib = _lib.load()
    words = 1032
    fake = C.c_void_p(1 << 20)            # non-null and 16-byte aligned
    null = C.c_void_p(0)
    lut = (C.c_uint32 * (words + 1))()
    lut[0] = 2
    calls = {
        "pg_hamming_knn": lambda: lib.pg_hamming_knn(fake, 512, 0, 1, fake, 1, planes, words, 1, 0, _lib.W_I64, fake,
                                                     fake, fake, 1 << 20, null),
        "pg_hamming_eps_count": lambda: lib.pg_hamming_eps_count(fake, 512, 0, 1, fake, 1, planes, words, lut, words + 1,
                                                                 fake, fake, 1 << 20, null),
        "pg_hamming_eps_fill": lambda: lib.pg_hamming_eps_fill(fake, 512, 0, 1, fake, 1, planes, words, lut, words + 1,
                                                               fake, _lib.W_I64, fake, fake, fake, 1 << 20, null),
        "pg_hamming_eps_count_capture": lambda: lib.pg_hamming_eps_count_capture(
            fake, 512, 0, 1, fake, 1, planes, words, lut, words + 1, 0, fake, fake, 1 << 20, null),
        "pg_hamming_eps_fill_capture": lambda: lib.pg_hamming_eps_fill_capture(
            fake, 512, 0, 1, fake, 1, planes, words, lut, words + 1, 0, fake, _lib.W_I64, fake, fake, fake, 1 << 20, null),
        "pg_hamming_tile": lambda: lib.pg_hamming_tile(fake, 1, fake, 1, 0, 1, planes, words, _lib.W_I64, fake, 1, null),
        "pg_hamming_flags_tile": lambda: lib.pg_hamming_flags_tile(fake, 1, fake, 1, 0, 1, planes, words, 0, 1, fake, 1,
                                                                   null),
    }
    for name, call in calls.items():
        assert call() == _lib.ERR_UNSUPPORTED, name
        assert f"planes={planes} words={words}" in _lib.last_error(), (name, _lib.last_error())
