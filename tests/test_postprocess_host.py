"""Host side of the nodal-field post-processing (DOFManager.node_coordinates / gradient /
error_norms / boundary_flux): the exported C entry, the last-element-wins table and the
node -> entries CSR of the whole L2G map, against NumPy on the golden Gmsh meshes (the
shuffled ones included).  No GPU."""
import glob
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT
from spectralelementmethod_b200 import _lib, device, discrete, grid_importers as gi, meshgen
from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS

GOLDEN = sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "msh_*.npz")))


def test_field_entry_is_exported_and_declared():
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], check=True,
                         capture_output=True, text=True).stdout
    assert " T semk_field_grad_f64" in out
    with open(os.path.join(ROOT, "include", "semk.h")) as f:
        assert "int semk_field_grad_f64(" in f.read()
    res, args = _lib.SIGNATURES["semk_field_grad_f64"]
    assert res is _lib._I and len(args) == 22


def _managers(tmp_path, path):
    z = np.load(path)
    p = int(z["meta"][2])
    msh = tmp_path / "m.msh"
    msh.write_bytes(z["msh_bytes"].tobytes())
    b1 = LagrangeGaussLobatto(p)
    for cls, rcm in ((discrete.DOFManager, False), (discrete.DOFManager, True),
                     (discrete.DOFManagerSC, True)):
        yield cls(gi.load_msh(str(msh), 2), 1, TensorProductQS(b1, b1), rcm_order=rcm)


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[4:-4] for p in GOLDEN])
def test_winner_and_node_csr_match_numpy(tmp_path, path):
    for mngr in _managers(tmp_path, path):
        l2g = mngr.node_map_array().reshape(mngr.mesh.n_cells, -1)
        n = mngr.mesh.n_nodes
        # the reference's element loop: a later element overwrites a shared node
        owner = np.full(n, -1, dtype=np.int64)
        for e in range(l2g.shape[0]):
            owner[l2g[e]] = e * l2g.shape[1] + np.arange(l2g.shape[1])
        want = np.zeros(l2g.size, dtype=np.uint8)
        want[owner[owner >= 0]] = 1
        win = device.winner_table(l2g, n)
        assert np.array_equal(win, want)
        assert int(win.sum()) == n                  # every node has exactly one winner
        # node -> entries CSR: the stable order of csr_by_key, on the CPU through torch
        ptr, pos = device.node_entries_csr(device.as_i32_bits(l2g, "cpu"), n)
        uniq, wptr, wpos = device.csr_by_key(l2g)
        assert np.array_equal(uniq, np.arange(n))
        assert np.array_equal(ptr.numpy().view(np.uint32), wptr)
        assert np.array_equal(pos.numpy().view(np.uint32), wpos)
        # and it reproduces the sums over the elements sharing a node
        vals = np.random.default_rng(0).standard_normal(l2g.size)
        p_, q_ = ptr.numpy().astype(np.int64), pos.numpy().astype(np.int64)
        sums = np.array([vals[q_[p_[j]:p_[j + 1]]].sum() for j in range(n)])
        want_sums = np.zeros(n)
        np.add.at(want_sums, l2g.ravel(), vals)
        assert np.allclose(sums, want_sums, rtol=1e-13, atol=1e-13)


def test_node_csr_of_a_structured_mesh_counts_the_sharing_elements():
    p, nx, ny = 3, 4, 3
    mesh = meshgen.structured_quad_mesh(nx, ny, p, "C")
    b1 = LagrangeGaussLobatto(p)
    mngr = discrete.DOFManager(mesh, 1, TensorProductQS(b1, b1), rcm_order=False)
    l2g = mngr.node_map_array().reshape(mesh.n_cells, -1)
    ptr, _pos = device.node_entries_csr(torch.from_numpy(l2g.astype(np.int64)).to(torch.int32),
                                        mesh.n_nodes)
    counts = np.diff(ptr.numpy())
    # interior vertices: 4 cells, edge nodes: 2, everything else: 1
    assert sorted(np.unique(counts).tolist()) == [1, 2, 4]
    assert int((counts == 4).sum()) == (nx - 1) * (ny - 1)
    assert counts.sum() == l2g.size
