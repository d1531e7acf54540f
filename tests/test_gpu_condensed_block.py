"""Blocks of loads on the condensed operator (rhs_many, backsolve_many, solve_many,
solve_load_many; csrc/semk_sc.cu sc_element_block_kernel and the stored-operator block
streams): every column is bitwise the single-load call on that column, whatever the chunk
width and the order of the columns, and the eigensolver's preconditioner returns the bits of
the column-by-column loop."""
import numpy as np
import pytest
import torch

from conftest import build_package_case, load_case, rel_l2
from spectralelementmethod_b200 import condensed, discrete, meshgen
from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS

pytestmark = pytest.mark.gpu

_OPS = {}


def operator(p, store, kind="C"):
    """Condensed operator on a 3 x 2 element mesh with Dirichlet nodes on "ebc"."""
    key = (p, store, kind)
    if key not in _OPS:
        mesh, mngr = build_package_case(kind, 3, 2, p, True, True)
        kw = dict(store_interior=store != "none", store_interior_inverse=store == "inverse")
        _OPS[key] = (mngr, mngr.condensed_poisson_operator(
            dirichlet=mngr.boundary_node_mask("ebc"), **kw))
    return _OPS[key]


def mixed_loads(n, k, seed=0):
    """Scalar, nodal CUDA and nodal host loads, interleaved."""
    rng = np.random.default_rng(seed)
    out = []
    for j in range(k):
        if j % 3 == 0:
            out.append(0.5 + j)
        elif j % 3 == 1:
            out.append(torch.from_numpy(rng.standard_normal(n)).cuda())
        else:
            out.append(rng.standard_normal(n))
    return out


def forget_single_cache(sc):
    """Point the single-load cache at a load no test uses, so that a single backsolve
    recomputes the interiors (backsolve_many always does)."""
    sc.rhs(-7.25)


@pytest.mark.parametrize("k", [1, 2, 7, 32, 33])
@pytest.mark.parametrize("p", list(range(2, 11)))
def test_rhs_and_backsolve_many_equal_single_calls(p, k):
    mngr, sc = operator(p, "none" if k % 2 else "stored")
    F = mixed_loads(sc.n_nodes, k, seed=p)
    X = torch.from_numpy(np.random.default_rng(k).standard_normal((k, sc.n_ext))).cuda()
    forget_single_cache(sc)
    singles_u = [sc.backsolve(X[j], F[j]) for j in range(k)]
    U = sc.backsolve_many(X, F)
    G = sc.rhs_many(F)
    singles_g = [sc.rhs(F[j]) for j in range(k)]
    assert G.shape == (k, sc.n_ext) and U.shape == (k, sc.n_nodes)
    for j in range(k):
        assert torch.equal(G[j], singles_g[j]), j
        assert torch.equal(U[j], singles_u[j]), j


@pytest.mark.parametrize("store", ["none", "stored", "inverse"])
@pytest.mark.parametrize("p", [3, 8, 10])
def test_block_tensor_loads_every_storage_mode(p, store):
    mngr, sc = operator(p, store, kind="S")
    k = 9
    F = torch.from_numpy(np.random.default_rng(p).standard_normal((k, sc.n_nodes))).cuda()
    G = sc.rhs_many(F)
    for j in range(k):
        assert torch.equal(G[j], sc.rhs(F[j])), j
    # the whole solve: with W kept the load pass keeps c and the back-solve streams W
    vals = np.where(mngr.boundary_node_mask("ebc"), 0.25, 0.0)
    U, infos = sc.solve_many(F, vals, rtol=1e-10)
    for j in range(k):
        u, info = sc.solve(F[j], vals, rtol=1e-10)
        assert torch.equal(U[j], u), j
        assert infos[j].iterations == info.iterations


def test_chunk_width_and_column_order_do_not_change_bits(monkeypatch):
    mngr, sc = operator(6, "stored")
    F = mixed_loads(sc.n_nodes, 12, seed=3)
    G32 = sc.rhs_many(F)
    U32, _ = sc.solve_many(F, rtol=1e-10)
    monkeypatch.setattr(condensed.CondensedPoissonOperator, "_block_cap", lambda self: 1)
    G1 = sc.rhs_many(F)
    U1, _ = sc.solve_many(F, rtol=1e-10)
    assert torch.equal(G1, G32) and torch.equal(U1, U32)
    monkeypatch.setattr(condensed.CondensedPoissonOperator, "_block_cap", lambda self: 5)
    perm = [7, 2, 11, 0, 5, 9, 1, 3, 10, 4, 8, 6]
    Gp = sc.rhs_many([F[j] for j in perm])
    Up, _ = sc.solve_many([F[j] for j in perm], rtol=1e-10)
    for q, j in enumerate(perm):
        assert torch.equal(Gp[q], G32[j]) and torch.equal(Up[q], U32[j])


def test_interleaving_with_single_calls_keeps_the_single_cache():
    mngr, sc = operator(5, "stored")
    f = torch.from_numpy(np.random.default_rng(1).standard_normal(sc.n_nodes)).cuda()
    x = torch.from_numpy(np.random.default_rng(2).standard_normal(sc.n_ext)).cuda()
    g = sc.rhs(f)
    u_cached = sc.backsolve(x, f)           # the stored path with the cached interior load
    F = mixed_loads(sc.n_nodes, 4)
    sc.rhs_many(F)
    sc.solve_many(F, rtol=1e-8)
    assert torch.equal(sc.backsolve(x, f), u_cached)
    assert torch.equal(sc.rhs(f), g)


@pytest.mark.parametrize("mesh_kind", ["pinwheel", "weighted_robin_reaction"])
def test_solve_many_equals_solve_on_unstructured_and_weighted_operators(mesh_kind):
    if mesh_kind == "pinwheel":
        mesh = meshgen.pinwheel_mesh(7, 4, rings=3)
        b1 = LagrangeGaussLobatto(4)
        mngr = discrete.DOFManagerSC(mesh, 1, TensorProductQS(b1, b1), rcm_order=True)
        sc = mngr.condensed_poisson_operator(dirichlet=mngr.boundary_node_mask("ebc"))
        flux = None
    else:
        mesh, mngr = build_package_case("C", 4, 3, 5, True, True)
        E, NN = mngr.mesh.node_map_array().reshape(-1, 36).shape
        react = np.random.default_rng(5).uniform(0.1, 1.0, (E, NN))
        sc = mngr.condensed_poisson_operator(
            weight=lambda x, y: 1.0 + 0.5 * x * x, reaction=react, robin={"nbc": 2.0},
            store_interior=True)
        flux = [{"nbc": 1.0}, None, {"nbc": lambda x, y: x + y}]
    F = mixed_loads(sc.n_nodes, 3, seed=7)
    vals = np.where(mngr.boundary_node_mask("ebc"), 0.5, 0.0)
    U, infos = sc.solve_many(F, dirichlet_values=vals, flux=flux, rtol=1e-11,
                             preconditioner="three-level")
    for j in range(3):
        u, info = sc.solve(F[j], vals, flux=None if flux is None else flux[j], rtol=1e-11,
                           preconditioner="three-level")
        assert torch.equal(U[j], u), j
        assert infos[j].iterations == info.iterations and infos[j].converged


@pytest.mark.parametrize("name", ["C448_sc_rcm", "S888_sc_rcm"])
def test_solve_many_on_golden_cases(name):
    g = load_case(name)
    mesh, mngr = build_package_case(g["kind"], g["nx"], g["ny"], g["p"], g["sc"], g["rcm"])
    sc = mngr.condensed_poisson_operator(dirichlet=g["on_ebc"])
    U, infos = sc.solve_many([1.0, 2.0], dirichlet_values=[g["ebc_vals"], 2.0 * g["ebc_vals"]],
                             rtol=1e-13)
    assert all(i.converged for i in infos)
    assert rel_l2(U[0].cpu().numpy(), g["solution"]) < 1e-12
    assert rel_l2(U[1].cpu().numpy(), 2.0 * g["solution"]) < 1e-12
    u0, _ = sc.solve(1.0, g["ebc_vals"], rtol=1e-13)
    assert torch.equal(U[0], u0)


@pytest.mark.parametrize("store", ["none", "stored"])
def test_solve_load_many_equals_solve_load(store):
    mngr, sc = operator(8, store)
    k = 5
    rng = np.random.default_rng(11)
    R = torch.from_numpy(rng.standard_normal((k, sc.n_nodes))).cuda()
    R[:, :sc.n_ext][:, sc.dirichlet_dev.bool()] = 0.0
    F = torch.from_numpy(rng.standard_normal((k, sc.n_nodes))).cuda()
    out = torch.empty((k, sc.n_nodes), dtype=torch.float64, device="cuda")
    U, infos = sc.solve_load_many(list(R), F, rtol=1e-2, out=out)
    assert U is out
    for j in range(k):
        u, info = sc.solve_load(R[j], F[j], rtol=1e-2)
        assert torch.equal(U[j], u) and infos[j].iterations == info.iterations


@pytest.mark.parametrize("dirichlet", ["ebc", None])
def test_eigenpairs_equal_the_column_by_column_preconditioner(monkeypatch, dirichlet):
    mesh, mngr = build_package_case("C", 8, 8, 4, True, True)
    lam, X, info = mngr.poisson_eigenpairs(4, dirichlet=dirichlet)

    def column_by_column(self, R, F, rtol=1e-8, preconditioner="three-level", out=None):
        infos = []
        for j in range(len(R)):
            u, i = self.solve_load(R[j], F[j], rtol=rtol, preconditioner=preconditioner)
            out[j].copy_(u)
            infos.append(i)
        return out, infos

    monkeypatch.setattr(condensed.CondensedPoissonOperator, "solve_load_many", column_by_column)
    lam_ref, X_ref, info_ref = mngr.poisson_eigenpairs(4, dirichlet=dirichlet)
    assert np.array_equal(lam, lam_ref) and torch.equal(X, X_ref)
    assert info["iterations"] == info_ref["iterations"]
    assert info["preconditioner_applications"] == info_ref["preconditioner_applications"]
    assert info["inner_iterations"] == info_ref["inner_iterations"]


def test_block_errors():
    mngr, sc = operator(4, "none")
    n = sc.n_nodes
    with pytest.raises(ValueError):
        sc.rhs_many([])
    with pytest.raises(ValueError):
        sc.rhs_many(torch.zeros((0, n), dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        sc.rhs_many(torch.zeros((2, n), dtype=torch.float32, device="cuda"))
    with pytest.raises(ValueError):
        sc.rhs_many(torch.zeros((2, n + 1), dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        sc.rhs_many(torch.zeros((2, n), dtype=torch.float64))
    with pytest.raises(ValueError):
        sc.backsolve_many(torch.zeros((3, sc.n_ext), dtype=torch.float64, device="cuda"),
                          [1.0, 2.0])
    with pytest.raises(ValueError):
        sc.solve_many([1.0, 2.0], dirichlet_values=[None])
    with pytest.raises(ValueError):
        sc.solve_load_many(torch.zeros((2, n), dtype=torch.float64, device="cuda"), [1.0])
    with pytest.raises(ValueError):
        sc.solve_load_many([torch.zeros(n, dtype=torch.float64, device="cuda")], [1.0],
                           out=torch.zeros((1, n + 1), dtype=torch.float64, device="cuda"))
    g = load_case("S324_sc")
    mesh, m2 = build_package_case(g["kind"], g["nx"], g["ny"], g["p"], g["sc"], g["rcm"])
    NN = (g["p"] + 1) ** 2
    E = m2.mesh.node_map_array().reshape(-1, NN).shape[0]
    eye = np.tile(np.eye(NN) * 4.0, (E, 1, 1))
    cs = condensed.CondensedLocalSystems(m2, eye, np.ones((E, NN)))
    for call in (lambda: cs.rhs_many([1.0]), lambda: cs.solve_many([1.0]),
                 lambda: cs.backsolve_many([cs.new_vector(0.0)], [1.0]),
                 lambda: cs.solve_load_many([cs.new_vector(0.0)], [1.0])):
        with pytest.raises(NotImplementedError):
            call()


@pytest.mark.parametrize("p", [2, 8])
def test_single_load_entry_combined_modes_equal_single_bit_calls(p):
    """semk_sc_element_react_f64 runs the factorisation bits and the load bits (one-column
    block passes) in turn: a combined mode, c_out in either load mode and a permuted
    slot_of_elem give the outputs of the single-bit calls."""
    from spectralelementmethod_b200 import _lib, device
    mngr, sc = operator(p, "stored")
    f64 = dict(dtype=torch.float64, device=sc.dev)
    E, NE, NI = sc.n_elem, sc.n_ext_loc, sc.n_int_loc
    rng = np.random.default_rng(p)
    f = torch.from_numpy(rng.standard_normal(sc.n_nodes)).cuda()
    x = torch.from_numpy(rng.standard_normal(sc.n_nodes)).cuda()
    slot = torch.from_numpy(rng.permutation(E).astype(np.int64)).cuda()
    G_slot = torch.empty_like(sc.G)
    G_slot[slot] = sc.G

    def call(mode, outs, G=sc.G, slot_of_elem=None):
        shapes = dict(S=(E, sc.s_stride), sdiag=(E, NE), W=(E, NE, NI), g=(E, NE), c=(E, NI))
        res = {k: (x.clone() if k == "u" else torch.full(shapes[k], -1.0, **f64)) for k in outs}
        P = lambda k: device.ptr(res.get(k))      # noqa: E731
        bad = torch.zeros(1, dtype=torch.int32, device=sc.dev)
        _lib.check(sc._lib.semk_sc_element_react_f64(
            sc.n1, E, device.ptr(slot_of_elem), device.ptr(G), sc.g_stride, 1,
            device.ptr(sc.tab.dev()[0]), device.ptr(sc._t["ext_loc"]), device.ptr(sc.l2g_dev),
            device.ptr(sc.JxW), device.ptr(f), 0.75, mode, P("S"), sc.s_stride, P("sdiag"),
            P("g"), P("u"), P("W"), P("c"), None, None, device.ptr(bad), device.stream_ptr()))
        assert int(bad.item()) == 0
        return res

    SCHUR, STORE, RHS, BACK = _lib.SC_SCHUR, _lib.SC_STORE, _lib.SC_RHS, _lib.SC_BACKSOLVE
    schur = call(SCHUR, "S sdiag".split())
    store = call(STORE, ["W"])
    rhs = call(RHS, ["g", "c"])
    back = call(BACK, ["u"])
    both = call(SCHUR | STORE | RHS, "S sdiag W g c".split())
    for k, ref in (("S", schur), ("sdiag", schur), ("W", store), ("g", rhs), ("c", rhs)):
        assert torch.equal(both[k], ref[k]), k
    loads = call(RHS | BACK, ["g", "u"])
    assert torch.equal(loads["g"], rhs["g"]) and torch.equal(loads["u"], back["u"])
    back_c = call(BACK, ["u", "c"], G=G_slot, slot_of_elem=slot)
    assert torch.equal(back_c["u"], back["u"]) and torch.equal(back_c["c"], rhs["c"])
