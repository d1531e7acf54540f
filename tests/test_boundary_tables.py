"""Host tables of flux / Robin boundaries (device.boundary_face_tables, device.csr_by_key) and
the C ABI of the Robin term (semk_bdiag, semk_poisson_apply_bdiag_f64, semk_pcg_solve_bdiag_f64,
semk_face_sum_f64).  Pure NumPy / gcc: no GPU."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from spectralelementmethod_b200 import _lib, device, grid_importers, meshgen
from spectralelementmethod_b200.mapping import _subface_slice


def _meshes(tmp_path):
    yield "S 5x3 p4", meshgen.structured_quad_mesh(5, 3, 4, "S"), ("ebc", "nbc")
    yield "C 4x4 p3", meshgen.structured_quad_mesh(4, 4, 3, "C"), ("ebc", "nbc")
    yield "C 1x1 p2", meshgen.structured_quad_mesh(1, 1, 2, "C"), ("ebc", "nbc")
    yield "annulus", meshgen.annulus_sector_mesh(3, 5, 4), ("sphere", "shell", "symaxis")
    path = str(tmp_path / "shuffled.msh")
    meshgen.write_gmsh22_binary(path, 4, 3, 3, "C", shuffle_seed=7)
    yield "gmsh", grid_importers.load_msh(path, 2), ("ebc", "nbc")


def test_face_nodes_match_boundary_node_ind(tmp_path):
    for label, mesh, names in _meshes(tmp_path):
        maps = mesh.node_map_array()
        n1 = maps.shape[1]
        for name in names:
            cells, faces, nodes, local = device.boundary_face_tables(mesh, name)
            assert nodes.shape == (cells.size, n1) and nodes.dtype == np.uint32, label
            assert cells.size > 0 and np.all(np.diff(cells) >= 0), label
            # face by face: the node ids of boundary_node_ind, in the same order
            assert np.array_equal(nodes.ravel(), mesh.boundary_node_ind(name)), (label, name)
            lin = np.arange(n1 * n1).reshape(n1, n1)
            for c, f, loc, ids in zip(cells, faces, local, nodes):
                assert np.array_equal(loc, _subface_slice(int(f), lin, 2))
                assert np.array_equal(ids, maps[c].ravel()[loc])
            # the (cell, face) pairs of the mesh's own registry, cells ascending
            bnd = mesh._boundary_id_lookup[name]
            want = sorted(mesh._boundary_faces[bnd], key=lambda cf: cf[0])
            assert [(int(c), int(f)) for c, f in zip(cells, faces)] == want


def test_unknown_boundary_name_raises_key_error():
    mesh = meshgen.structured_quad_mesh(2, 2, 2)
    with pytest.raises(KeyError):
        device.boundary_face_tables(mesh, "no such boundary")


def test_csr_lists_every_entry_once_ascending(tmp_path):
    for label, mesh, names in _meshes(tmp_path):
        for name in names:
            cells, faces, nodes, local = device.boundary_face_tables(mesh, name)
            n1 = nodes.shape[1]
            NN = n1 * n1
            for keys in (nodes, cells[:, None] * NN + local):
                uniq, ptr, pos = device.csr_by_key(keys)
                flat = keys.ravel()
                assert np.all(np.diff(uniq.astype(np.int64)) > 0)
                assert np.array_equal(uniq, np.unique(flat))
                assert ptr[0] == 0 and ptr[-1] == flat.size and np.all(np.diff(ptr) >= 1)
                # every (face, k) exactly once
                assert np.array_equal(np.sort(pos), np.arange(flat.size))
                for j in range(uniq.size):
                    run = pos[ptr[j]:ptr[j + 1]].astype(np.int64)
                    assert np.all(np.diff(run) > 0), label
                    assert np.all(flat[run] == uniq[j])
            # corner cells of the structured meshes carry two faces of one boundary: their
            # shared local node appears twice among the element-local slots
            if label.startswith("C 4x4"):
                uniq, ptr, pos = device.csr_by_key(cells[:, None] * NN + local)
                assert np.diff(ptr).max() == 2


def test_bdiag_struct_layout_matches_header(tmp_path):
    fields = [f[0] for f in _lib.semk_bdiag._fields_]
    src = ['#include <stdio.h>', '#include <stddef.h>', '#include "semk.h"', 'int main(void) {',
           '  printf("%zu\\n", sizeof(struct semk_bdiag));']
    src += ['  printf("%%zu\\n", offsetof(struct semk_bdiag, %s));' % f for f in fields]
    src += ['  return 0; }']
    c = tmp_path / "bdiag_layout.c"
    c.write_text("\n".join(src))
    exe = tmp_path / "bdiag_layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(c), "-o", str(exe)])
    out = subprocess.check_output([str(exe)]).decode().split()
    assert int(out[0]) == ctypes.sizeof(_lib.semk_bdiag) == 32
    for f, off in zip(fields, out[1:]):
        assert getattr(_lib.semk_bdiag, f).offset == int(off), f


def test_boundary_symbols_are_exported_and_bound():
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in ("semk_poisson_apply_bdiag_f64", "semk_pcg_solve_bdiag_f64", "semk_face_sum_f64"):
        assert hasattr(lib, name)
        assert name in _lib.SIGNATURES
    assert _lib.load().semk_version() == 100
