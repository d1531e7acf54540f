"""Host side of the condensed block loads: the column cap, the chunking of a block and the
C signatures of the block entries (no GPU needed: the argument checks return before any
launch)."""
import ctypes as C
import os
import re

import pytest

from conftest import ROOT
from spectralelementmethod_b200 import _lib
from spectralelementmethod_b200.condensed import block_chunks

BLOCK_ENTRIES = ["semk_sc_block_max_cols", "semk_sc_element_block_f64",
                 "semk_sc_load_stored_block_f64", "semk_sc_backsolve_stored_block_f64"]


def test_block_max_cols():
    lib = _lib.load()
    assert [lib.semk_sc_block_max_cols(n1) for n1 in range(13)] == \
        [-1, -1, -1] + [32] * 9 + [-1]


@pytest.mark.parametrize("k, cap, per_col, free, want", [
    (1, 32, 10, 1000, [(0, 1)]),
    (32, 32, 10, 1000, [(0, 32)]),
    (33, 32, 10, 1000, [(0, 32), (32, 33)]),
    (7, 32, 100, 250, [(0, 2), (2, 4), (4, 6), (6, 7)]),
    (5, 32, 100, 10, [(0, 1), (1, 2), (2, 3), (3, 4), (4, 5)]),   # at least one column
    (5, 1, 1, 1000, [(0, 1), (1, 2), (2, 3), (3, 4), (4, 5)]),
])
def test_block_chunks(k, cap, per_col, free, want):
    assert block_chunks(k, cap, per_col, free) == want


def test_block_chunks_rejects_empty_blocks():
    with pytest.raises(ValueError):
        block_chunks(0, 32, 1, 1)
    with pytest.raises(ValueError):
        block_chunks(3, -1, 1, 1)


def test_header_and_bindings_agree():
    text = open(os.path.join(ROOT, "include", "semk.h")).read()
    ctype = {"int": C.c_int, "int64_t": C.c_int64, "double": C.c_double, "uint32_t": C.c_uint32}
    for name in BLOCK_ENTRIES:
        m = re.search(r"\bint\s+%s\(([^)]*)\);" % name, text)
        assert m, name
        params = [" ".join(p.split()) for p in m.group(1).split(",")]
        want = [C.c_void_p if "*" in p else ctype[p.replace("const ", "").split()[0]]
                for p in params]
        res, args = _lib.SIGNATURES[name]
        assert res is C.c_int and list(args) == want, name


def test_block_entries_check_their_arguments():
    lib = _lib.load()
    scale = (C.c_double * 33)(*([1.0] * 33))

    def element(n1=9, mode=2, k=3, F=None, mask=0, c_out=None, ldc=0, U=None, ldu=0):
        return lib.semk_sc_element_block_f64(n1, 4, 8, 1, 1, 8, 8, 8, 8, None, mode, k, F, 100,
                                             mask, scale, 8, 1 << 20, c_out, ldc, U, ldu, 8, None)

    assert element(k=33) == _lib.ERR_UNSUPPORTED
    assert element(n1=2) == _lib.ERR_UNSUPPORTED
    assert element(n1=12) == _lib.ERR_UNSUPPORTED
    assert element(k=0) == _lib.ERR_INVALID
    assert element(mode=1) == _lib.ERR_INVALID
    assert element(mask=1) == _lib.ERR_INVALID          # a nodal column without F
    assert element(mask=8) == _lib.ERR_INVALID          # bit beyond k
    assert element(mode=4) == _lib.ERR_INVALID          # BACKSOLVE without U
    assert element(mode=4, U=8, ldu=10, c_out=8, ldc=4 * 49 - 1) == _lib.ERR_INVALID  # short c
    assert element(mode=2, c_out=8, ldc=4 * 49 - 1) == _lib.ERR_INVALID
    assert lib.semk_sc_load_stored_block_f64(9, 4, 8, 8, 8, 8, 8, 33, None, 0, 0, scale, 8,
                                             1 << 20, 8, 1 << 20, None) == _lib.ERR_UNSUPPORTED
    assert lib.semk_sc_load_stored_block_f64(9, 4, 8, 8, 8, 8, 8, 2, None, 0, 0, scale, 8,
                                             1, 8, 1 << 20, None) == _lib.ERR_INVALID
    assert lib.semk_sc_backsolve_stored_block_f64(9, 4, 8, None, 0, 8, 8, 33, 8, 10,
                                                  None) == _lib.ERR_UNSUPPORTED
    assert lib.semk_sc_backsolve_stored_block_f64(9, 4, 8, None, 0, 8, 8, 0, 8, 10,
                                                  None) == _lib.ERR_INVALID
    assert lib.semk_sc_backsolve_stored_block_f64(1, 4, 8, None, 0, 8, 8, 1, 8, 10,
                                                  None) == _lib.ERR_UNSUPPORTED
