"""Multi-rank host logic on CPU: world_size-2 `gloo` runs of the strip
partition, the interface exchange, the owner-weighted dot products and the
distributed PCG driver.  The rank-local operator is played by the CPU oracle
(test infrastructure) so that no GPU is needed; on the GPU box the same
classes drive the CUDA operator (bench.py --gpus N, tests/test_gpu_parity.py).
"""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ORACLE_DIR, ROOT, rel_l2

KIND, NXL, NY, P = "C", 3, 4, 3


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


class CpuKernels(object):
    """Torch-on-CPU stand-in for operators.PCGKernels (same scalar protocol as
    csrc/semk_vec.cu)."""

    def __init__(self, dirichlet):
        self.fixed = torch.as_tensor(dirichlet)

    def init(self, b, Ax, dinv, r, p, sc, n_dot):
        bb = torch.where(self.fixed, torch.zeros_like(b), b)
        r.copy_(torch.where(self.fixed, torch.zeros_like(b), bb - Ax))
        p.copy_(dinv * r)
        sc[0] = torch.dot(r[:n_dot], p[:n_dot])
        sc[1] = 0.0
        sc[2] = sc[0]
        sc[3] = torch.dot(r[:n_dot], r[:n_dot])
        sc[4] = torch.dot(bb[:n_dot], bb[:n_dot])
        sc[5:] = 0.0

    def update_xr(self, p, Ap, dinv, x, r, sc, n_dot):
        ok = bool(sc[1] > 0)
        alpha = float(sc[0] / sc[1]) if ok else 0.0
        x += alpha * p
        r -= alpha * Ap
        sc[2] = torch.dot(r[:n_dot] * dinv[:n_dot], r[:n_dot])
        sc[3] = torch.dot(r[:n_dot], r[:n_dot])
        sc[5] += 1
        if not ok:
            sc[7] = 1.0

    def update_p(self, r, dinv, p, sc):
        beta = float(sc[2] / sc[0]) if float(sc[0]) != 0.0 else 0.0
        p.mul_(beta).add_(dinv * r)
        sc[0] = sc[2]


def _worker(rank, world, port, out):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, ORACLE_DIR)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import sem_oracle as so
        from spectralelementmethod_b200 import discrete
        from spectralelementmethod_b200.basis_functions import (LagrangeGaussLobatto,
                                                                TensorProductQS)
        from spectralelementmethod_b200.distributed import (DistributedOperator, StripPartition,
                                                            distributed_pcg)
        bounds = (-1.0, -1.0 + 2.0 * world, -1.0, 1.0)
        part = StripPartition(rank, world, NXL, NY, P, bounds=bounds)
        mesh = part.build_local_mesh(KIND)
        b1 = LagrangeGaussLobatto(P)
        mngr = discrete.DOFManager(mesh, 1, TensorProductQS(b1, b1), rcm_order=False)
        on = mngr.boundary_node_mask("ebc")
        l2g = mngr.node_map_array()
        basis = so.Basis(P)
        geo = so.geometry(basis, mesh.nodes, l2g)
        L = so.local_stiffness(basis, geo["invJ"], geo["JxW"])
        n = part.n_local
        A = so.assemble_csr(L, l2g, n)
        M = (~on).astype(float)

        def local_apply(u, outv, dot):
            un = u.numpy()
            y = M * (A @ (M * un)) + (1 - M) * un
            if outv is None:
                outv = torch.empty_like(u)
            outv.copy_(torch.from_numpy(y))
            if dot is not None:
                dot[0] = float((M * un) @ (A @ (M * un)) + ((1 - M) * un) @ un)
            return outv

        dop = DistributedOperator(part, local_apply, dirichlet=on)
        gid = part.global_ids()
        rng = np.random.default_rng(5)
        ug = rng.standard_normal(part.n_global)
        u = torch.from_numpy(ug[gid].copy())
        y = dop.apply(u)
        # the two halves separately (the staged host apply computes the local part elsewhere)
        y2 = dop.finish(local_apply(u, None, None), u)
        dotv = dop.owned_dot(u, u)

        # RHS / diagonal / lifted system, assembled across ranks
        bl = torch.from_numpy(so.assemble_vector(geo["JxW"], l2g, n))
        dop.exchange_add(bl)
        dl = torch.from_numpy(A.diagonal().copy())
        dop.exchange_add(dl)
        dl[torch.from_numpy(on)] = 1.0
        x_phys_nodes = np.zeros((2, n))
        x_phys_nodes[:, l2g.ravel()] = np.moveaxis(geo["x_phys"], 1, 0).reshape(2, -1)
        g = np.where(on, 0.2 * ((x_phys_nodes[0] + 1) + (x_phys_nodes[1] + 1)), 0.0)
        gt = torch.from_numpy(g)
        t = torch.from_numpy(M * (A @ g))
        dop.exchange_add(t)
        bh = bl - t
        bh[torch.from_numpy(on)] = gt[torch.from_numpy(on)]
        x0 = torch.where(torch.from_numpy(on), bh, torch.zeros_like(bh))
        it, rel, ok = distributed_pcg(dop, bh, x0, 1.0 / dl, CpuKernels(on), rtol=1e-13,
                                      maxiter=3000, check_every=7)
        res = dict(gid=gid, y=y.numpy(), y2=y2.numpy(), dot=float(dotv), x=x0.numpy(), it=it, ok=ok, rel=rel,
                   n_owned=part.n_owned, on=on, b=bl.numpy(), d=dl.numpy())
        torch.save(res, os.path.join(out, "rank%d.pt" % rank))
    finally:
        dist.destroy_process_group()


@pytest.fixture(scope="module")
def two_rank_results(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("dist"))
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    return [torch.load(os.path.join(out, "rank%d.pt" % r), weights_only=False) for r in range(world)]


def _global_reference():
    import sem_oracle as so
    world = 2
    nxg = NXL * world
    NX, NYn = nxg * P + 1, NY * P + 1
    X, Y = np.meshgrid(np.linspace(-1.0, -1.0 + 2.0 * world, NX), np.linspace(-1, 1, NYn),
                       indexing="ij")
    s = 0.08 * np.sin(np.pi * X) * np.sin(np.pi * Y)
    nodes = np.vstack([(X + s).ravel(), (Y + s).ravel()])
    l2g = so.mesh_l2g(nxg, NY, P)
    basis = so.Basis(P)
    geo = so.geometry(basis, nodes, l2g)
    L = so.local_stiffness(basis, geo["invJ"], geo["JxW"])
    n = nodes.shape[1]
    A = so.assemble_csr(L, l2g, n)
    on, vals = so.dirichlet_data(nodes, l2g, geo["x_phys"], so.mesh_boundary_faces(nxg, NY))
    b = so.assemble_vector(geo["JxW"], l2g, n)
    return dict(A=A, on=on, vals=vals, b=b, n=n, sol=so.solve_direct(A, b, on, vals))


def test_partition_description():
    from spectralelementmethod_b200.distributed import StripPartition
    parts = [StripPartition(r, 3, 4, 5, 2) for r in range(3)]
    NYn = 5 * 2 + 1
    assert [p.n_local for p in parts] == [9 * NYn] * 3
    assert parts[0].left is None and parts[0].right == 1 and parts[2].right is None
    assert [p.n_owned for p in parts] == [8 * NYn, 8 * NYn, 9 * NYn]
    assert sum(p.n_owned for p in parts) == parts[0].n_global == 25 * NYn
    # shared columns carry the same global ids and bit-identical coordinates
    assert np.array_equal(parts[0].global_ids()[parts[0].right_slice],
                          parts[1].global_ids()[parts[1].left_slice])
    for kind in ("S", "C"):
        c0, c1 = parts[0].local_coordinates(kind), parts[1].local_coordinates(kind)
        assert np.array_equal(c0[:, parts[0].right_slice], c1[:, parts[1].left_slice])
    with pytest.raises(ValueError):
        StripPartition(3, 3, 4, 5, 2)
    m0, m2 = parts[0].build_local_mesh(), parts[2].build_local_mesh()
    assert len(m0._boundary_cells[0]) == 5 + 4 - 1 and len(m2._boundary_cells[0]) == 4
    assert len(m0._boundary_cells[1]) == 4 and len(m2._boundary_cells[1]) == 5 + 4 - 1


def test_two_rank_apply_matches_global_operator(two_rank_results):
    ref = _global_reference()
    rng = np.random.default_rng(5)
    ug = rng.standard_normal(ref["n"])
    M = (~ref["on"]).astype(float)
    want = M * (ref["A"] @ (M * ug)) + (1 - M) * ug
    for r in two_rank_results:
        assert rel_l2(r["y"], want[r["gid"]]) < 1e-12
        assert np.array_equal(r["y2"], r["y"])          # finish(local_apply(u), u) == apply(u)
        assert np.array_equal(r["on"], ref["on"][r["gid"]])
        assert rel_l2(r["b"], ref["b"][r["gid"]]) < 1e-13
        assert rel_l2(r["d"], (M * ref["A"].diagonal() + (1 - M))[r["gid"]]) < 1e-13
    # owner-weighted dot counts every node once
    assert abs(two_rank_results[0]["dot"] - ug @ ug) < 1e-11 * (ug @ ug)
    assert two_rank_results[0]["dot"] == two_rank_results[1]["dot"]


def test_two_rank_pcg_matches_global_direct_solve(two_rank_results):
    ref = _global_reference()
    its = {r["it"] for r in two_rank_results}
    assert len(its) == 1 and all(r["ok"] for r in two_rank_results)
    for r in two_rank_results:
        assert rel_l2(r["x"], ref["sol"][r["gid"]]) < 1e-11
        assert r["rel"] <= 1e-13


# --------------------------------------------------------------------------
# statically condensed operator on two ranks (CondensedStripView)
# --------------------------------------------------------------------------
def _worker_condensed(rank, world, port, out):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, ORACLE_DIR)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import sem_oracle as so
        from spectralelementmethod_b200 import discrete, meshgen
        from spectralelementmethod_b200.basis_functions import (LagrangeGaussLobatto,
                                                                TensorProductQS)
        from spectralelementmethod_b200.distributed import (CondensedStripView,
                                                            DistributedOperator, StripPartition,
                                                            distributed_pcg)
        bounds = (-1.0, -1.0 + 2.0 * world, -1.0, 1.0)
        part = StripPartition(rank, world, NXL, NY, P, bounds=bounds)
        mesh = part.build_local_mesh(KIND)
        b1 = LagrangeGaussLobatto(P)
        mngr = discrete.DOFManagerSC(mesh, 1, TensorProductQS(b1, b1), rcm_order=False)
        on_full = mngr.boundary_node_mask("ebc")
        l2g = mngr.node_map_array()
        lex = meshgen.structured_node_maps(NXL, NY, P).reshape(-1)
        lex_ids = np.empty(mesh.n_nodes, dtype=np.int64)
        lex_ids[l2g.reshape(-1)] = lex
        gid = part.global_ids()[lex_ids]
        basis = so.Basis(P)
        geo = so.geometry(basis, mesh.nodes, l2g)
        c = so.condensed_system(P, geo["invJ"], geo["JxW"], l2g)
        n_ext = c["n_ext"]
        view = CondensedStripView(part, n_ext)
        # interface columns keep their place and order in the exterior-first numbering
        assert np.array_equal(lex_ids[view.left_slice], np.arange(part.NY))
        assert np.array_equal(lex_ids[view.right_slice],
                              np.arange(part.n_local - part.NY, part.n_local))
        on = on_full[:n_ext]
        assert not on_full[n_ext:].any()
        S = c["Sg"]
        M = (~on).astype(float)

        def local_apply(u, outv, dot):
            un = u.numpy()
            y = M * (S @ (M * un)) + (1 - M) * un
            if outv is None:
                outv = torch.empty_like(u)
            outv.copy_(torch.from_numpy(y))
            if dot is not None:
                dot[0] = float((M * un) @ (S @ (M * un)) + ((1 - M) * un) @ un)
            return outv

        dop = DistributedOperator(view, local_apply, dirichlet=on)
        bl = torch.from_numpy(c["grhs"].copy())
        dop.exchange_add(bl)
        dl = torch.from_numpy(S.diagonal().copy())
        dop.exchange_add(dl)
        dl[torch.from_numpy(on)] = 1.0
        x, y = mesh.nodes
        # Dirichlet data from the (bit-identical across ranks) node coordinates
        g = np.where(on_full, 0.3 * x - 0.2 * y + 0.1, 0.0)
        ge = g[:n_ext]
        t = torch.from_numpy(M * (S @ ge))
        dop.exchange_add(t)
        bh = bl - t
        ont = torch.from_numpy(on)
        bh[ont] = torch.from_numpy(ge)[ont]
        x0 = torch.where(ont, bh, torch.zeros_like(bh))
        it, rel, ok = distributed_pcg(dop, bh, x0, 1.0 / dl, CpuKernels(on), rtol=1e-13,
                                      maxiter=3000, check_every=7)
        # rank-local interior back-substitution (sem/discrete.py:513-524)
        sol = np.zeros(mesh.n_nodes)
        sol[:n_ext] = x0.numpy()
        inner = np.linalg.solve(c["Aii"], (c["f_int"] - np.einsum("eij,ej->ei", c["Aie"],
                                                                  sol[c["ids"]]))[..., None])
        sol[c["int_ids"]] = inner[..., 0]
        torch.save(dict(gid=gid, sol=sol, it=it, ok=ok, rel=rel, n_owned=view.n_owned,
                        n_ext=n_ext, coords=np.asarray(mesh.nodes)),
                   os.path.join(out, "rank%d.pt" % rank))
    finally:
        dist.destroy_process_group()


@pytest.fixture(scope="module")
def two_rank_condensed(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("dist_sc"))
    world = 2
    mp.spawn(_worker_condensed, args=(world, _free_port(), out), nprocs=world, join=True)
    return [torch.load(os.path.join(out, "rank%d.pt" % r), weights_only=False) for r in range(world)]


def test_two_rank_condensed_pcg_matches_global_direct_solve(two_rank_condensed):
    import sem_oracle as so
    ref = _global_reference()
    # same problem with the Dirichlet data of the condensed workers
    world = 2
    nxg = NXL * world
    NX, NYn = nxg * P + 1, NY * P + 1
    X, Y = np.meshgrid(np.linspace(-1.0, -1.0 + 2.0 * world, NX), np.linspace(-1, 1, NYn),
                       indexing="ij")
    s = 0.08 * np.sin(np.pi * X) * np.sin(np.pi * Y)
    xg, yg = (X + s).ravel(), (Y + s).ravel()
    vals = np.where(ref["on"], 0.3 * xg - 0.2 * yg + 0.1, 0.0)
    want = so.solve_direct(ref["A"], ref["b"], ref["on"], vals)
    its = {r["it"] for r in two_rank_condensed}
    assert len(its) == 1 and all(r["ok"] for r in two_rank_condensed)
    total_owned = 0
    for r in two_rank_condensed:
        assert np.array_equal(r["coords"][0], xg[r["gid"]])      # the id maps line up
        assert rel_l2(r["sol"], want[r["gid"]]) < 1e-11
        total_owned += r["n_owned"]
    # owned exterior nodes of all ranks = distinct exterior nodes of the global mesh
    n_int = (NXL * world) * NY * (P - 1) ** 2
    assert total_owned == ref["n"] - n_int


def test_condensed_strip_view_description():
    from spectralelementmethod_b200.distributed import CondensedStripView, StripPartition
    parts = [StripPartition(r, 3, 4, 5, 2) for r in range(3)]
    NYn = 5 * 2 + 1
    # exterior nodes of a 4 x 5 strip of order 2: all nodes but one interior node per element
    n_ext = parts[0].n_local - 4 * 5
    views = [CondensedStripView(p, n_ext) for p in parts]
    assert [v.n_local for v in views] == [n_ext] * 3
    assert [v.n_owned for v in views] == [n_ext - NYn, n_ext - NYn, n_ext]
    assert views[1].left == 0 and views[1].right == 2 and views[2].right is None
    assert views[0].left_slice == slice(0, NYn)
    assert views[0].right_slice == slice(n_ext - NYn, n_ext)
    assert views[1].NY == NYn and views[1].base is parts[1]


def test_unknown_exchange_is_rejected_before_any_set_up():
    """Both strip wrappers check ``exchange`` before they build a mesh, a DOF manager or a
    device operator: no GPU and no process group is needed to get the error."""
    from spectralelementmethod_b200.distributed import (DistributedCondensedPoisson,
                                                        DistributedPoisson, StripPartition)
    part = StripPartition(0, 2, 2, 2, 2)
    for cls in (DistributedPoisson, DistributedCondensedPoisson):
        with pytest.raises(ValueError, match="exchange"):
            cls(part, 2, exchange="bogus")


# --------------------------------------------------------------------------
# two-level preconditioner on two ranks: algorithm-level emulation (oracle operators,
# the product's host tables and partition views) of the scheme the device path will use
# --------------------------------------------------------------------------
def _worker_two_level(rank, world, port, out):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, ORACLE_DIR)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import sem_oracle as so
        from spectralelementmethod_b200 import discrete, meshgen
        from spectralelementmethod_b200.basis_functions import (LagrangeGaussLobatto,
                                                                TensorProductQS)
        from spectralelementmethod_b200.condensed import coarse_tables, condensed_tables
        from spectralelementmethod_b200.distributed import (CondensedStripView,
                                                            DistributedOperator, StripPartition,
                                                            distributed_pcg)
        nxl, ny, p = 4, 6, 4
        bounds = (-1.0, -1.0 + 2.0 * world, -1.0, 1.0)
        part = StripPartition(rank, world, nxl, ny, p, bounds=bounds)
        mesh = part.build_local_mesh("C")
        b1 = LagrangeGaussLobatto(p)
        mngr = discrete.DOFManagerSC(mesh, 1, TensorProductQS(b1, b1), rcm_order=False)
        on_full = mngr.boundary_node_mask("ebc")
        l2g = mngr.node_map_array()
        N, NE = p + 1, 4 * p
        lex = meshgen.structured_node_maps(nxl, ny, p).reshape(-1)
        lex_ids = np.empty(mesh.n_nodes, dtype=np.int64)
        lex_ids[l2g.reshape(-1)] = lex
        gid = part.global_ids()[lex_ids]
        geo = so.geometry(so.Basis(p), mesh.nodes, l2g)
        c = so.condensed_system(p, geo["invJ"], geo["JxW"], l2g)
        n_ext, ids, S_e = c["n_ext"], c["ids"], c["S"]
        D = on_full[:n_ext]
        ext_loc = np.asarray(mesh.get_geometries()[0].exterior_node_ind)
        l2g_ext, nptr, npos = condensed_tables(l2g.reshape(-1, N * N), ext_loc, n_ext)
        ct = coarse_tables(l2g_ext, nptr, npos, D, np.asarray(b1.nodes))
        n_v, Dc = ct["n_v"], ct["dirichlet_c"]
        vc = ct["vert_c"].astype(np.int64)
        view_f = CondensedStripView(part, n_ext)
        view_c = CondensedStripView(part, n_v, column=ny + 1)
        # the coarse interface columns are the leading / trailing compact vertex ids
        vids = np.unique(ids[:, :4])
        assert np.array_equal(lex_ids[vids[view_c.left_slice]], np.arange(0, part.NY, p))
        assert np.array_equal(lex_ids[vids[view_c.right_slice]],
                              part.n_local - part.NY + np.arange(0, part.NY, p))
        Mf, Mc = (~D).astype(float), (~Dc).astype(float)
        S = c["Sg"]
        Phi = ct["phi"][None] * (~D)[ids][:, :, None] * (~Dc)[vc][:, None, :]
        Ace = np.einsum("eka,ekj,ejc->eac", Phi, S_e, Phi)
        vptr, vpos = ct["vptr"].astype(np.int64), ct["vpos"].astype(np.int64)

        def fine_apply(u, outv, dot):
            un = u.numpy()
            y = Mf * (S @ (Mf * un)) + (1 - Mf) * un
            outv = torch.empty_like(u) if outv is None else outv
            outv.copy_(torch.from_numpy(y))
            if dot is not None:
                dot[0] = float(un @ y)
            return outv

        def coarse_apply(u, outv, dot):
            un = u.numpy()
            yl = np.einsum("eac,ec->ea", Ace, un[vc]).ravel()
            y = np.where(Dc, un, np.add.reduceat(yl[vpos], vptr[:-1]))
            outv = torch.empty_like(u) if outv is None else outv
            outv.copy_(torch.from_numpy(y))
            if dot is not None:
                dot[0] = float(un @ y)
            return outv

        dop = DistributedOperator(view_f, fine_apply, dirichlet=D)
        dop_c = DistributedOperator(view_c, coarse_apply, dirichlet=Dc)
        tD, tDc = torch.from_numpy(D), torch.from_numpy(Dc)
        dl = torch.from_numpy(S.diagonal().copy())
        dop.exchange_add(dl)
        dl[tD] = 1.0
        dcl = torch.from_numpy(np.add.reduceat(np.einsum("eaa->ea", Ace).ravel()[vpos], vptr[:-1]))
        dop_c.exchange_add(dcl)
        dcl[tDc] = 1.0
        pv, pw = ct["pv"].astype(np.int64), ct["pw"]
        rptr, ridx, rw = ct["rptr"].astype(np.int64), ct["ridx"].astype(np.int64), ct["rw"]
        class Ops(object):
            """NumPy stand-ins of the rank-local device pieces."""
            dinv_c = 1.0 / dcl

            @staticmethod
            def residual(bv, Ax):
                bm = torch.where(tD, torch.zeros_like(bv), bv)
                return torch.where(tD, torch.zeros_like(bv), bv - Ax), bm

            @staticmethod
            def jacobi(r):
                return r / dl

            @staticmethod
            def restrict(r, n_owned):
                rn = r.numpy().copy()
                rn[n_owned:] = 0.0                       # owned fine nodes only
                rc = np.zeros(n_v)
                nz = rptr[1:] > rptr[:-1]
                rc[nz] = np.add.reduceat(rw * rn[ridx], rptr[:-1][nz])
                return torch.from_numpy(rc)

            @staticmethod
            def prolong_add(xc, z):
                xn = xc.numpy()
                z += torch.from_numpy(pw[:, 0] * xn[pv[:, 0]] + pw[:, 1] * xn[pv[:, 1]])

            @staticmethod
            def new_coarse():
                return torch.zeros(n_v, dtype=torch.float64)

        # third level: GLOBAL vertex aggregates (both owners of a shared vertex column agree),
        # A3 = P2^T Ac P2 summed over the ranks, replicated dense inverse
        from spectralelementmethod_b200.condensed import aggregate_csr
        from spectralelementmethod_b200.distributed import (distributed_multilevel_pcg,
                                                            strip_vertex_aggregates)
        agg, n_agg, ktile = strip_vertex_aggregates(part, lex_ids[vids], Dc, max_tiles=6)
        valid = agg != 0xFFFFFFFF
        assert n_agg <= 6 and (agg[valid] < n_agg).all() and not valid[Dc].any()
        a_e = np.where(valid, agg.astype(np.int64), -1)[vc]                       # [E, 4]
        A3 = np.zeros((n_agg, n_agg))
        rows, cols = np.repeat(a_e, 4, axis=1).ravel(), np.tile(a_e, (1, 4)).ravel()
        okk = (rows >= 0) & (cols >= 0)
        np.add.at(A3, (rows[okk], cols[okk]), Ace.reshape(-1)[okk])
        A3t = torch.from_numpy(A3)
        dist.all_reduce(A3t)
        A3 = A3t.numpy()
        A3[np.diag(A3) == 0.0, np.diag(A3) == 0.0] = 1.0
        aptr_o, aidx_o = aggregate_csr(agg, n_agg, view_c.n_owned)

        class Top(object):
            A3inv = torch.from_numpy(np.linalg.inv(0.5 * (A3 + A3.T)))

            @staticmethod
            def agg_restrict(q, n_owned):
                assert n_owned == view_c.n_owned
                out = np.zeros(n_agg)
                np.add.at(out, agg[aidx_o].astype(np.int64), q.numpy()[aidx_o])
                return torch.from_numpy(out)

            @staticmethod
            def agg_prolong_add(y3, z):
                zn = z.numpy()
                zn[valid] += y3.numpy()[agg[valid].astype(np.int64)]

        # lifted right-hand side (as in the condensed worker above)
        bl = torch.from_numpy(c["grhs"].copy())
        dop.exchange_add(bl)
        x_, y_ = mesh.nodes
        g = np.where(on_full, 0.3 * x_ - 0.2 * y_ + 0.1, 0.0)[:n_ext]
        t = torch.from_numpy(Mf * (S @ g))
        dop.exchange_add(t)
        bh = bl - t
        bh[tD] = torch.from_numpy(g)[tD]
        results = {}
        for name, top, flexible in (("two", None, False), ("three", Top, True)):
            x = torch.where(tD, bh, torch.zeros_like(bh))
            it, rel, ok, inner_total = distributed_multilevel_pcg(
                dop, dop_c, Ops, bh, x, rtol=1e-13, maxiter=200, inner_rtol=1e-2,
                inner_maxiter=500, flexible=flexible, top=top)
            assert ok and rel <= 1e-13
            sol = np.zeros(mesh.n_nodes)
            sol[:n_ext] = x.numpy()
            inner = np.linalg.solve(c["Aii"], (c["f_int"] - np.einsum("eij,ej->ei", c["Aie"],
                                                                      sol[ids]))[..., None])
            sol[c["int_ids"]] = inner[..., 0]
            results[name] = dict(sol=sol, it=it, inner=int(inner_total))
        torch.save(dict(gid=gid, results=results, n_agg=n_agg, ktile=ktile),
                   os.path.join(out, "rank%d.pt" % rank))
    finally:
        dist.destroy_process_group()


def test_two_rank_multilevel_pcg_emulation(tmp_path):
    import sem_oracle as so
    world, nxl, ny, p = 2, 4, 6, 4
    out = str(tmp_path)
    mp.spawn(_worker_two_level, args=(world, _free_port(), out), nprocs=world, join=True)
    res = [torch.load(os.path.join(out, "rank%d.pt" % r), weights_only=False) for r in range(world)]
    nxg = nxl * world
    NX, NYn = nxg * p + 1, ny * p + 1
    X, Y = np.meshgrid(np.linspace(-1.0, -1.0 + 2.0 * world, NX), np.linspace(-1, 1, NYn),
                       indexing="ij")
    s = 0.08 * np.sin(np.pi * X) * np.sin(np.pi * Y)
    nodes = np.vstack([(X + s).ravel(), (Y + s).ravel()])
    l2g = so.mesh_l2g(nxg, ny, p)
    basis = so.Basis(p)
    geo = so.geometry(basis, nodes, l2g)
    L = so.local_stiffness(basis, geo["invJ"], geo["JxW"])
    A = so.assemble_csr(L, l2g, nodes.shape[1])
    on, _ = so.dirichlet_data(nodes, l2g, geo["x_phys"], so.mesh_boundary_faces(nxg, ny))
    vals = np.where(on, 0.3 * nodes[0] - 0.2 * nodes[1] + 0.1, 0.0)
    want = so.solve_direct(A, so.assemble_vector(geo["JxW"], l2g, nodes.shape[1]), on, vals)
    for name in ("two", "three"):
        r0, r1 = res[0]["results"][name], res[1]["results"][name]
        assert r0["it"] == r1["it"] and r0["it"] < 40                # mesh-independent count
        assert r0["inner"] == r1["inner"] > 0
        for r, rk in ((r0, res[0]), (r1, res[1])):
            assert rel_l2(r["sol"], want[rk["gid"]]) < 1e-10
    # the aggregation level cuts the inner iterations, the outer count stays
    two, three = res[0]["results"]["two"], res[0]["results"]["three"]
    assert three["inner"] < two["inner"] and abs(three["it"] - two["it"]) <= 3
