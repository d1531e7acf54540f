"""The native multilevel driver (semk_sc_mlpcg_solve_f64, csrc/semk_ml.cu) on one GPU:
three-level preconditioner (Jacobi + vertex coarse space + aggregation with a dense
inverse) against the golden solutions of the live reference and the NumPy emulation of
the same algorithm (tests/test_two_level_host.py); true residuals; re-entrancy of the
native drivers; the peer-memory exchange kernel driven on one GPU (self-exchange)."""
import ctypes as C
import threading

import numpy as np
import pytest
import torch

import sem_oracle as so
from conftest import build_package_case, golden_case_names, load_case, rel_l2
from spectralelementmethod_b200 import _lib, discrete, meshgen
from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS
from spectralelementmethod_b200.condensed import element_tiles, top_level_inverse
from test_two_level_host import emulate

pytestmark = pytest.mark.gpu

SC_CASES = [n for n in golden_case_names() if "_sc" in n]


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def host(t):
    return t.detach().cpu().numpy()


@pytest.mark.parametrize("name", SC_CASES)
def test_three_level_solve_vs_reference_golden(name):
    """Solutions of the reference's own DOFManagerSC.solve (tests/golden) <= 1e-12."""
    g = load_case(name)
    mesh, mngr = build_package_case(g["kind"], g["nx"], g["ny"], g["p"], g["sc"], g["rcm"])
    sc = mngr.condensed_poisson_operator(dirichlet=g["on_ebc"])
    u, info = sc.solve(1.0, g["ebc_vals"], rtol=1e-13, preconditioner="three-level")
    assert info.converged, info
    assert rel_l2(host(u), g["solution"]) < 1e-12
    assert info.true_rel_residual is not None and info.true_rel_residual < 1e-11
    assert info.inner_iterations > 0 and info.inner_solves == info.iterations


@pytest.mark.parametrize("flexible", [True, False])
def test_three_level_matches_the_numpy_emulation(flexible):
    """Same host tables, same algorithm: outer / inner iteration counts and the solution
    against the NumPy emulation; the aggregated operator against the host assembly."""
    p, n = 4, 24
    mesh, mngr = build_package_case("C", n, n, p, True, False)
    on = mngr.boundary_node_mask("ebc")
    l2g = mngr.node_map_array()
    basis = so.Basis(p)
    geo = so.geometry(basis, mesh.nodes, l2g)
    c = so.condensed_system(p, geo["invJ"], geo["JxW"], l2g)
    x_, y_ = mesh.nodes
    vals = np.where(on, 0.2 * ((x_ + 1) + (y_ + 1)), 0.0)

    class M(object):
        _structured_shape = (n, n)
    tile = element_tiles(M(), n * n, max_tiles=36)
    extra = {}
    xj, itj, x2, it2, ct, Ace, _ = emulate(p, c, on, vals, basis.nodes, tile=tile, extra=extra)
    sc = mngr.condensed_poisson_operator(dirichlet=on, geometric_factors=(geo["invJ"], geo["JxW"]))
    b = sc.lift(sc.rhs(1.0), vals)
    x3, info = sc.solve_pcg(b, rtol=1e-12, preconditioner="three-level", max_tiles=36,
                            flexible=flexible)
    top, tt, n_agg = sc._build_top(36)
    assert n_agg == extra["at"]["n_agg"]
    assert np.array_equal(host(tt["agg"]).view(np.uint32), extra["at"]["agg"])
    assert rel_l2(host(tt["A3inv"]), extra["A3inv"]) < 1e-9
    assert info.converged and abs(info.iterations - extra["it3"]) <= 2
    assert abs(info.inner_iterations - extra["inner3"]) <= max(8, extra["inner3"] // 10)
    assert rel_l2(host(x3), extra["x3"]) < 1e-10
    # the reported true residual is the recomputed one
    assert abs(info.true_rel_residual - sc.true_residual(b, x3)) <= 1e-3 * info.true_rel_residual \
        + 1e-16
    assert info.true_rel_residual < 1e-11
    # two levels through the same driver: same solution, more inner iterations
    x2d, info2 = sc.solve_pcg(b, rtol=1e-12, preconditioner="two-level", flexible=flexible)
    assert info2.converged and abs(info2.iterations - it2) <= 3
    assert rel_l2(host(x2d), host(x3)) < 1e-10
    assert info.inner_iterations * 2 < info2.inner_iterations
    # bit-reproducible run to run
    x3b, infob = sc.solve_pcg(b, rtol=1e-12, preconditioner="three-level", max_tiles=36,
                              flexible=flexible)
    assert torch.equal(x3, x3b) and infob.iterations == info.iterations


def test_three_level_at_size_and_on_an_unstructured_mesh():
    mesh, mngr = build_package_case("C", 96, 96, 8, True, False)
    on = mngr.boundary_node_mask("ebc")
    x, y = mesh.nodes
    vals = np.where(on, 0.2 * ((x + 1) + (y + 1)), 0.0)
    sc = mngr.condensed_poisson_operator(dirichlet=on)
    u3, info3 = sc.solve(1.0, vals, rtol=1e-12, preconditioner="three-level", max_tiles=144)
    u2, info2 = sc.solve(1.0, vals, rtol=1e-12, preconditioner="two-level")
    assert info3.converged and info2.converged
    assert info3.iterations < 60 and abs(info3.iterations - info2.iterations) <= 4
    assert info3.inner_iterations <= 40 * info3.iterations          # mesh-independent inner count
    assert info3.inner_iterations * 2 < info2.inner_iterations
    assert rel_l2(host(u3), host(u2)) < 1e-9
    full = mngr.poisson_operator(dirichlet=on)
    b = full.lift(full.rhs(1.0), vals)
    assert float((b - full.apply(u3)).norm() / b.norm()) < 1e-10
    # irregular vertex valence: aggregates along a Morton curve
    pm = meshgen.pinwheel_mesh(7, 4, rings=6)
    b1 = LagrangeGaussLobatto(4)
    pmngr = discrete.DOFManagerSC(pm, 1, TensorProductQS(b1, b1), rcm_order=True)
    pon = pmngr.boundary_node_mask("ebc")
    px, py = pm.nodes
    pvals = np.where(pon, 0.3 * px - 0.2 * py + 0.1, 0.0)
    psc = pmngr.condensed_poisson_operator(dirichlet=pon)
    a3, i3 = psc.solve(1.0, pvals, rtol=1e-13, preconditioner="three-level", max_tiles=8)
    aj, ij = psc.solve(1.0, pvals, rtol=1e-13)
    assert i3.converged and rel_l2(host(a3), host(aj)) < 1e-10


@pytest.mark.parametrize("mesh_kind", ["structured", "pinwheel"])
def test_coarse_operator_ell_rows_equal_the_element_form(mesh_kind):
    """The assembled ELL rows of the vertex coarse operator (what the driver multiplies
    with) against the element-matrix form, Dirichlet identity rows and fused dot included."""
    if mesh_kind == "structured":
        mesh, mngr = build_package_case("C", 12, 10, 5, True, True)
    else:
        mesh = meshgen.pinwheel_mesh(7, 4, rings=3)
        b1 = LagrangeGaussLobatto(4)
        mngr = discrete.DOFManagerSC(mesh, 1, TensorProductQS(b1, b1), rcm_order=True)
    sc = mngr.condensed_poisson_operator(dirichlet=mngr.boundary_node_mask("ebc"))
    cs, t, n_v = sc._build_coarse()
    assert cs.ell_width >= 9
    xc = torch.from_numpy(np.random.default_rng(4).standard_normal(n_v)).cuda()
    d1 = torch.zeros(1, dtype=torch.float64, device="cuda")
    d2 = torch.zeros(1, dtype=torch.float64, device="cuda")
    y1 = sc.coarse_apply(xc, dot_out=d1)
    y2 = sc.coarse_apply(xc, dot_out=d2, ell=True)
    assert rel_l2(host(y2), host(y1)) < 1e-13
    assert abs(float(d1) - float(d2)) < 1e-12 * abs(float(d1))
    fixed = t["dirichlet_c"].bool()
    assert torch.equal(y2[fixed], xc[fixed])


def test_top_level_operator_matches_the_host_assembly():
    mesh, mngr = build_package_case("C", 12, 10, 5, True, True)
    on = mngr.boundary_node_mask("ebc")
    sc = mngr.condensed_poisson_operator(dirichlet=on)
    cs, t, n_v = sc._build_coarse()
    top, tt, n_agg = sc._build_top(max_tiles=9)
    want = top_level_inverse(host(t["Ace"]), host(t["vert_c"]).view(np.uint32),
                             host(tt["agg"]).view(np.uint32), n_agg)
    assert rel_l2(host(tt["A3inv"]), want) < 1e-10


def test_concurrent_solves_on_two_streams_and_threads():
    """The native drivers are re-entrant per (host thread, stream, workspace): two
    different problems solved at the same time give the results of the serial runs."""
    cases = []
    for kind, n, p in (("C", 40, 6), ("S", 48, 5)):
        mesh, mngr = build_package_case(kind, n, n, p, True, False)
        on = mngr.boundary_node_mask("ebc")
        sc = mngr.condensed_poisson_operator(dirichlet=on)
        b = sc.lift(sc.rhs(1.0), None)
        cases.append((sc, b))
    serial = []
    for sc, b in cases:
        xj, ij = sc.solve_pcg(b, rtol=1e-12, check_every=7)
        x3, i3 = sc.solve_pcg(b, rtol=1e-12, preconditioner="three-level", max_tiles=16)
        serial.append((xj, ij.iterations, x3, i3.iterations))
    torch.cuda.synchronize()
    out = [None, None]
    errs = []

    def work(k):
        try:
            sc, b = cases[k]
            stream = torch.cuda.Stream()
            stream.wait_stream(torch.cuda.default_stream())
            with torch.cuda.stream(stream):
                for _ in range(3):
                    xj, ij = sc.solve_pcg(b, rtol=1e-12, check_every=7)
                    x3, i3 = sc.solve_pcg(b, rtol=1e-12, preconditioner="three-level",
                                          max_tiles=16)
                stream.synchronize()
            out[k] = (xj, ij.iterations, x3, i3.iterations)
        except Exception as exc:        # noqa: BLE001 -- reported by the main thread
            errs.append(exc)
    threads = [threading.Thread(target=work, args=(k,)) for k in range(2)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errs, errs
    for k in range(2):
        assert out[k][1] == serial[k][1] and out[k][3] == serial[k][3]
        assert torch.equal(out[k][0], serial[k][0]) and torch.equal(out[k][2], serial[k][2])


def test_maxiter_is_respected_by_the_graph_path():
    mesh, mngr = build_package_case("C", 24, 24, 6, True, False)
    sc = mngr.condensed_poisson_operator(dirichlet=mngr.boundary_node_mask("ebc"))
    b = sc.lift(sc.rhs(1.0), None)
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.default_stream())
    with torch.cuda.stream(stream):      # a non-default stream takes the CUDA-graph path
        x, info = sc.solve_pcg(b, rtol=1e-14, maxiter=23, check_every=10)
        stream.synchronize()
    assert info.iterations == 23 and not info.converged


@pytest.mark.parametrize("with_dirichlet", [False, True])
def test_halo_exchange_kernel_self_exchange(with_dirichlet):
    """csrc/semk_peer.cu on ONE GPU: a periodic strip whose left and right neighbour are
    the rank itself (both CTAs of the single launch exchange through the rank's own
    region) -- push, epoch flags, wait, add, Dirichlet identity rows and the dot fix-up."""
    lib = _lib.load()
    n_col, n_local = 1237, 20000
    region = C.c_void_p()
    handle = (C.c_ubyte * 64)()
    _lib.check(lib.semk_peer_alloc(int(lib.semk_halo_region_bytes(n_col)), C.byref(region), handle))
    try:
        rng = np.random.default_rng(3)
        status = torch.zeros(1, dtype=torch.int32, device="cuda")
        stream = torch.cuda.current_stream().cuda_stream
        for epoch in (1, 2, 3):                        # both parities of the double buffer
            y0 = rng.standard_normal(n_local)
            u0 = rng.standard_normal(n_local)
            mask = np.zeros(n_local, dtype=np.uint8)
            if with_dirichlet:
                mask[rng.integers(0, n_col, 40)] = 1
                mask[n_local - n_col + rng.integers(0, n_col, 40)] = 1
            y = torch.from_numpy(y0.copy()).cuda()
            u = torch.from_numpy(u0).cuda()
            m = torch.from_numpy(mask).cuda()
            dot = torch.tensor([5.0], dtype=torch.float64, device="cuda")
            _lib.check(lib.semk_halo_exchange_f64(
                n_col, n_local, y.data_ptr(), u.data_ptr() if with_dirichlet else None,
                m.data_ptr() if with_dirichlet else None, region, region, region, epoch,
                dot.data_ptr(), status.data_ptr(), stream))
            want = y0.copy()
            want[:n_col] = y0[:n_col] + y0[n_local - n_col:]
            want[n_local - n_col:] = y0[n_local - n_col:] + y0[:n_col]
            dup = 0.0
            if with_dirichlet:
                fixed = mask.astype(bool)
                edge = np.zeros(n_local, dtype=bool)
                edge[:n_col] = edge[n_local - n_col:] = True
                want[fixed & edge] = u0[fixed & edge]
                right = fixed.copy()
                right[:n_local - n_col] = False
                dup = float(u0[right] @ u0[right])       # the column this rank does not own
            assert int(status.item()) == 0
            assert np.array_equal(host(y), want)         # one add per node: exact
            assert abs(float(dot.item()) - (5.0 - dup)) <= 1e-12 * max(1.0, dup)
    finally:
        torch.cuda.synchronize()
        _lib.check(lib.semk_peer_free(region))


@pytest.mark.parametrize("nx,ny,p", [(12, 24, 8), (13, 9, 4), (6, 16, 5)])
def test_overlapped_apply_and_exchange_on_one_gpu(nx, ny, p):
    """PoissonOperator.apply_halo on ONE GPU: boundary tile columns first, the light exchange
    kernel on the side stream with the rank as its own left and right neighbour (a periodic
    strip), interior patches meanwhile.  Must equal the serial sequence apply -> exchange
    bit for bit, and the range-split apply must equal the one-launch apply."""
    lib = _lib.load()
    mesh, mngr = build_package_case("C", nx, ny, p, False, False)
    on = mngr.boundary_node_mask("ebc")
    op = mngr.poisson_operator(dirichlet=on, boundary_columns_first=True)
    ref = mngr.poisson_operator(dirichlet=on)
    split = op.boundary_split()
    assert split is not None and 0 < split[0] < op.n_patch
    rng = np.random.default_rng(11)
    u = dev(rng.standard_normal(op.n_nodes))
    y_one = op.apply(u)
    # another element order only reorders the 3- and 4-term sums at tile corners
    assert rel_l2(host(y_one), host(ref.apply(u))) < 1e-14
    y_two = op.new_vector(0.0)
    op.apply_range(u, y_two, 0, split[0], 0, split[1], 0, split[2])
    op.apply_range(u, y_two, split[0], op.n_patch, split[1], op._op.n_shared_chunk, split[2],
                   op._op.n_shared)
    assert torch.equal(y_two, y_one)
    n_col = ny * p + 1
    region = C.c_void_p()
    handle = (C.c_ubyte * 64)()
    _lib.check(lib.semk_peer_alloc(int(lib.semk_halo_region_bytes(n_col)), C.byref(region), handle))
    try:
        status = torch.zeros(1, dtype=torch.int32, device="cuda")
        halo = _lib.semk_halo()
        halo.n_col, halo.mine, halo.left, halo.right = n_col, region, region, region
        halo.epoch, halo.status = 0, status.data_ptr()
        m = torch.from_numpy(on.astype(np.uint8)).cuda()
        stream = torch.cuda.current_stream().cuda_stream
        for rep in range(3):
            y = op.apply_halo(u, op.new_vector(), split, halo, m)
            torch.cuda.synchronize()
            assert int(status.item()) == 0 and halo.epoch == 2 * rep + 1
            want = y_one.clone()
            halo.epoch += 1
            _lib.check(lib.semk_halo_exchange_f64(
                n_col, op.n_nodes, want.data_ptr(), u.data_ptr(), m.data_ptr(), region, region,
                region, halo.epoch, None, status.data_ptr(), stream))
            torch.cuda.synchronize()
            assert torch.equal(y, want)
    finally:
        torch.cuda.synchronize()
        _lib.check(lib.semk_peer_free(region))


def test_comm_allreduce_single_rank_is_a_noop():
    lib = _lib.load()
    comm = _lib.semk_comm()
    comm.rank, comm.world, comm.capacity = 0, 1, 64
    region = C.c_void_p()
    handle = (C.c_ubyte * 64)()
    _lib.check(lib.semk_peer_alloc(int(lib.semk_comm_region_bytes(1, 64)), C.byref(region), handle))
    try:
        status = torch.zeros(1, dtype=torch.int32, device="cuda")
        comm.regions[0] = region.value
        comm.status = status.data_ptr()
        buf = torch.arange(10, dtype=torch.float64, device="cuda")
        _lib.check(lib.semk_comm_allreduce_f64(C.byref(comm), buf.data_ptr(), 10,
                                               torch.cuda.current_stream().cuda_stream))
        assert torch.equal(buf, torch.arange(10, dtype=torch.float64, device="cuda"))
        with pytest.raises(ValueError):
            _lib.check(lib.semk_comm_allreduce_f64(C.byref(comm), buf.data_ptr(), 65, None))
    finally:
        torch.cuda.synchronize()
        _lib.check(lib.semk_peer_free(region))


def test_refinement_on_the_true_residual():
    """solve_pcg_refined: the recursive residual of CG runs ahead of the true one; refinement
    cycles bring ||b - S x|| / ||b|| down to the tolerance (or to the attainable accuracy)."""
    mesh, mngr = build_package_case("C", 96, 96, 8, True, False)
    sc = mngr.condensed_poisson_operator(dirichlet=mngr.boundary_node_mask("ebc"))
    b = sc.lift(sc.rhs(1.0), None)
    x0, i0 = sc.solve_pcg(b, rtol=1e-12, preconditioner="three-level")
    x1, i1, cycles = sc.solve_pcg_refined(b, rtol=1e-12)
    assert abs(cycles[0][0] - i0.true_rel_residual) <= 0.5 * i0.true_rel_residual + 1e-15
    assert cycles[-1][0] <= max(1e-12, 0.5 * cycles[0][0]) or len(cycles) == 1
    assert sc.true_residual(b, x1) <= sc.true_residual(b, x0) * 1.0000001
    assert rel_l2(host(x1), host(x0)) < 1e-8
