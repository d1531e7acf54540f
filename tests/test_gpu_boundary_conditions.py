"""Flux and Robin boundary conditions on the device: boundary loads and Robin diagonals against
the reference user's host recipe (``boundary_elements`` + ``bfe.dSxW``), the Robin apply / PCG
of the plain operator (semk_poisson_apply_bdiag_f64, semk_pcg_solve_bdiag_f64), the condensed
operator's Robin term through the element reaction diagonal, and manufactured solutions."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import build_package_case
from spectralelementmethod_b200 import _lib, device, discrete, meshgen
from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS

pytestmark = pytest.mark.gpu


def host_recipe(mngr, name, g):
    """b[bfe.node_ind] += g * bfe.dSxW over the boundary elements (g: scalar, nodal values or a
    NumPy callable of the face-node coordinates)."""
    b = np.zeros(mngr.ndof)
    for _fe, bfe in mngr.boundary_elements(name, x_phys=True, Jacobian=True):
        ind = np.asarray(bfe.node_ind).ravel()
        if callable(g):
            gv = g(*bfe.x_phys)
        elif np.ndim(g):
            gv = g[ind]
        else:
            gv = g
        b[ind] += gv * bfe.dSxW
    return b


def rel(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def g_np(x, y):
    return 1.0 + 0.3 * x * x - 0.7 * np.sin(y)


def g_torch(x, y):
    return 1.0 + 0.3 * x * x - 0.7 * torch.sin(y)


@pytest.mark.parametrize("kind,p", [("S", 2), ("S", 5), ("C", 5), ("C", 8), ("S", 8)])
def test_boundary_load_matches_reference_recipe(kind, p):
    _mesh, mngr = build_package_case(kind, 4, 3, p, False, False)
    op = mngr.poisson_operator()
    rng = np.random.default_rng(p)
    nodal = rng.standard_normal(mngr.ndof)
    for name in ("ebc", "nbc"):
        for g_dev, g_host in ((2.5, 2.5), (nodal, nodal), (torch.from_numpy(nodal).cuda(), nodal),
                              (g_torch, g_np)):
            b = op.boundary_load(name, g_dev).cpu().numpy()
            assert rel(b, host_recipe(mngr, name, g_host)) < 1e-12, (name, g_dev)
    if kind == "S":
        # the length of the right + top sides of [-1, 1]^2
        assert abs(float(op.boundary_load("nbc", 1.0).sum()) - 4.0) < 1e-14
    # the condensed operator: the exterior vector of the same load
    _m2, mngr_sc = build_package_case(kind, 4, 3, p, True, True)
    sc = mngr_sc.condensed_poisson_operator()
    want = host_recipe(mngr_sc, "nbc", g_np)
    assert not want[sc.n_ext:].any()
    got = sc.boundary_load("nbc", g_torch).cpu().numpy()
    assert got.size == sc.n_ext and rel(got, want[:sc.n_ext]) < 1e-12
    with pytest.raises(KeyError):
        op.boundary_load("no such boundary", 1.0)


def test_boundary_load_on_the_annulus():
    p = 8
    mesh = meshgen.annulus_sector_mesh(3, 16, p)         # pi / 16 of arc per element
    b1 = LagrangeGaussLobatto(p)
    mngr = discrete.DOFManager(mesh, 1, TensorProductQS(b1, b1), rcm_order=False)
    op = mngr.poisson_operator()
    for name in ("sphere", "shell", "symaxis"):
        for g_dev, g_host in ((1.0, 1.0), (g_torch, g_np)):
            assert rel(op.boundary_load(name, g_dev).cpu().numpy(),
                       host_recipe(mngr, name, g_host)) < 1e-12, name
    assert abs(float(op.boundary_load("sphere", 1.0).sum()) - np.pi) < 1e-9


def _robin_pair(dirichlet=None):
    _mesh, mngr = build_package_case("C", 4, 3, 4, False, False)
    alpha_t = lambda x, y: 1.5 + x * x                   # noqa: E731
    alpha_n = lambda x, y: 1.5 + x * x                   # noqa: E731
    plain = mngr.poisson_operator(dirichlet=dirichlet)
    robin = mngr.poisson_operator(dirichlet=dirichlet, robin={"nbc": alpha_t, "ebc": 0.75})
    diag = host_recipe(mngr, "nbc", alpha_n) + host_recipe(mngr, "ebc", 0.75)
    return mngr, plain, robin, diag


def test_robin_matrix_is_plain_plus_boundary_diagonal():
    mngr, plain, robin, diag = _robin_pair()
    D = (robin.to_scipy_csr() - plain.to_scipy_csr()).toarray()
    assert np.abs(D - np.diag(diag)).max() <= 1e-13 * np.abs(diag).max()
    # masked, Dirichlet on "ebc": the Robin diagonal stays off the masked rows and columns
    mask = mngr.boundary_node_mask("ebc")
    mngr, plain, robin, diag = _robin_pair(mask)
    D = (robin.to_scipy_csr(masked=True) - plain.to_scipy_csr(masked=True)).toarray()
    assert np.abs(D - np.diag(np.where(mask, 0.0, diag))).max() <= 1e-13 * np.abs(diag).max()
    D = (robin.to_scipy_csr() - plain.to_scipy_csr()).toarray()
    assert np.abs(D - np.diag(diag)).max() <= 1e-13 * np.abs(diag).max()
    # the diagonal (Jacobi) sees the term
    for masked in (True, False):
        dr = robin.diagonal(masked).cpu().numpy()
        dp = plain.diagonal(masked).cpu().numpy()
        add = np.where(mask, 0.0, diag) if masked else diag
        assert np.abs(dr - dp - add).max() <= 1e-13 * np.abs(dp).max()
    # the fused dot and bitwise reproducibility
    u = torch.from_numpy(np.random.default_rng(1).standard_normal(robin.n_nodes)).cuda()
    outs = []
    for _ in range(2):
        d = torch.zeros(1, dtype=torch.float64, device="cuda")
        y = robin.apply(u, dot_out=d)
        want = float(torch.dot(u, y))
        assert abs(float(d) - want) <= 1e-13 * abs(want)
        outs.append((y, d))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


def test_condensed_robin_is_the_schur_complement_of_the_plain_robin_matrix():
    _mesh, mngr = build_package_case("C", 3, 3, 4, True, True)
    robin = {"nbc": lambda x, y: 1.0 + 0.5 * y * y, "ebc": 2.0}
    A = mngr.poisson_operator(robin=robin).to_scipy_csr().toarray()
    sc = mngr.condensed_poisson_operator(robin=robin)
    ne = sc.n_ext
    S = A[:ne, :ne] - A[:ne, ne:] @ np.linalg.solve(A[ne:, ne:], A[ne:, :ne])
    e = sc.new_vector(0.0)
    cols = []
    for j in range(ne):
        e[j] = 1.0
        cols.append(sc.apply(e, flags=0).cpu().numpy())
        e[j] = 0.0
    Sd = np.stack(cols, axis=1)
    assert np.abs(Sd - S).max() <= 1e-11 * np.abs(S).max()
    with pytest.raises(ValueError):
        mngr.condensed_poisson_operator(robin={"nbc": -1.0})
    with pytest.raises(KeyError):
        mngr.condensed_poisson_operator(robin={"no such boundary": 1.0})


# -- manufactured solutions: u symmetric in x and y, so that the two faces at a corner of
# one named boundary agree on the flux there --------------------------------------------------
def u_exact(x, y, m=np):
    return m.cos(0.9 * x + 0.3) + m.cos(0.9 * y + 0.3) + 0.5 * m.sin(0.7 * (x + y))


def f_exact(x, y):
    return 0.81 * (np.cos(0.9 * x + 0.3) + np.cos(0.9 * y + 0.3)) + 0.49 * np.sin(0.7 * (x + y))


def _du(s, t):
    return -0.9 * torch.sin(0.9 * s + 0.3) + 0.35 * torch.cos(0.7 * (s + t))


def flux_nbc(x, y):        # right (x = 1): u_x; top (y = 1): u_y
    return torch.where(x >= y, _du(x, y), _du(y, x))


def flux_ebc(x, y):        # left (x = -1): -u_x; bottom (y = -1): -u_y
    return torch.where(x <= y, -_du(x, y), -_du(y, x))


def _gll_coordinates(mngr):
    mesh = mngr.mesh
    l2g = mesh.node_map_array().reshape(mesh.n_cells, -1).astype(np.int64)
    xp = device.element_geometry(mngr._basis, mesh.nodes, l2g, jacobian=False)["x_phys"]
    X = np.zeros((2, mesh.n_nodes))
    X[:, l2g.ravel()] = xp.reshape(mesh.n_cells, 2, -1).transpose(1, 0, 2).reshape(2, -1)
    return X


CASES = {
    "flux": dict(robin=None, dirichlet="ebc",
                 flux=lambda a: {"nbc": flux_nbc}),
    "robin": dict(robin={"nbc": 2.0}, dirichlet="ebc",
                  flux=lambda a: {"nbc": lambda x, y: flux_nbc(x, y) + 2.0 * u_exact(x, y, torch)}),
    "pure-robin": dict(robin={"nbc": 2.0, "ebc": 2.0}, dirichlet=None,
                       flux=lambda a: {"nbc": lambda x, y: flux_nbc(x, y) + 2.0 * u_exact(x, y, torch),
                                       "ebc": lambda x, y: flux_ebc(x, y) + 2.0 * u_exact(x, y, torch)}),
}


def _solve_all(case, p, rtol=1e-12):
    c = CASES[case]
    _mesh, mngr = build_package_case("C", 8, 8, p, True, True)
    X = _gll_coordinates(mngr)
    ue = u_exact(X[0], X[1])
    f = torch.from_numpy(f_exact(X[0], X[1])).cuda()
    mask = mngr.boundary_node_mask(c["dirichlet"]) if c["dirichlet"] else None
    dv = torch.from_numpy(ue).cuda() if mask is not None else None
    flux = c["flux"](None)
    out = {}
    plain = mngr.poisson_operator(dirichlet=mask, robin=c["robin"])
    u, info = plain.solve(f, dv, flux=flux, rtol=rtol)
    assert info.converged, (case, p, info)
    out["plain"] = (u.cpu().numpy(), info)
    sc = mngr.condensed_poisson_operator(dirichlet=mask, robin=c["robin"])
    for prec in ("jacobi", "two-level", "three-level"):
        u, info = sc.solve(f, dv, flux=flux, rtol=rtol, preconditioner=prec)
        assert info.converged, (case, p, prec, info)
        out[prec] = (u.cpu().numpy(), info)
    return ue, out


@pytest.mark.parametrize("case", sorted(CASES))
def test_manufactured_solutions(case):
    rtol = 1e-12
    ue8, o8 = _solve_all(case, 8, rtol)
    ue4, o4 = _solve_all(case, 4, rtol)
    for name, (u, info) in o8.items():
        err8 = np.abs(u - ue8).max()
        err4 = np.abs(o4[name][0] - ue4).max()
        assert err8 < 1e-8, (case, name, err8)
        assert err8 * 100 < err4, (case, name, err8, err4)
        assert np.abs(u - o8["plain"][0]).max() < 1e-9, (case, name)
        if name in ("two-level", "three-level"):
            assert info.true_rel_residual <= 10 * rtol, (case, name, info.true_rel_residual)


def test_zero_robin_changes_nothing_and_unsupported_paths_refuse():
    _mesh, mngr = build_package_case("C", 4, 8, 8, False, False)
    mask = mngr.boundary_node_mask("ebc")
    plain = mngr.poisson_operator(dirichlet=mask)
    zero = mngr.poisson_operator(dirichlet=mask, robin={"nbc": 0.0})
    u = torch.from_numpy(np.random.default_rng(5).standard_normal(plain.n_nodes)).cuda()
    for flags in (None, 0):
        dp = torch.zeros(1, dtype=torch.float64, device="cuda")
        dz = torch.zeros(1, dtype=torch.float64, device="cuda")
        assert torch.equal(plain.apply(u, flags=flags, dot_out=dp),
                           zero.apply(u, flags=flags, dot_out=dz))
        assert torch.equal(dp, dz)
    b = plain.lift(plain.rhs(1.0) + plain.boundary_load("nbc", 0.3), np.zeros(plain.n_nodes))
    xp, ip = plain.solve_pcg(b, rtol=1e-12)
    xz, iz = zero.solve_pcg(b, rtol=1e-12)
    assert torch.equal(xp, xz) and ip.iterations == iz.iterations
    robin = mngr.poisson_operator(dirichlet=mask, robin={"nbc": 1.0})
    y = robin.new_vector()
    with pytest.raises(NotImplementedError):
        robin.apply_atomic(u)
    with pytest.raises(NotImplementedError):
        robin.apply_range(u, y, 0, 1, 0, 0, 0, 0)
    with pytest.raises(NotImplementedError):
        robin.apply_host(u.cpu().numpy(), np.empty(robin.n_nodes))
    with pytest.raises(NotImplementedError):
        robin.apply_host(u.cpu().numpy(), np.empty(robin.n_nodes), stages=1)
    with pytest.raises(NotImplementedError):
        robin.apply_host_many([u.cpu().numpy()], [np.empty(robin.n_nodes)])
    with pytest.raises(NotImplementedError):
        robin.boundary_split()
    with pytest.raises(ValueError):
        mngr.poisson_operator(robin={"nbc": -0.5})
    with pytest.raises(ValueError):
        mngr.poisson_operator(robin={"nbc": lambda x, y: x})
    with pytest.raises(KeyError):
        mngr.poisson_operator(robin={"no such boundary": 1.0})
    # the C entry with an empty term launches the plain apply
    bd = _lib.semk_bdiag()
    y0 = plain.new_vector()
    _lib.check(plain._lib.semk_poisson_apply_bdiag_f64(
        C.byref(plain._op), C.byref(bd), device.ptr(u), device.ptr(y0), 0, None,
        device.stream_ptr()))
    assert torch.equal(y0, plain.apply(u, flags=0))
