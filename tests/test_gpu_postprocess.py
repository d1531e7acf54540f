"""Nodal fields after a solve on the device (DOFManager.node_coordinates / gradient /
error_norms / boundary_flux, csrc/semk_geom.cu's field kernel): against the host mirror's
recipes (fe.gradient, fe.integrate, bfe.gradient . bfe.unit_normal), exactness on polynomials,
the energy identity against the Poisson apply, reproducibility, convergence of a manufactured
solution, and the error paths."""
import os

import numpy as np
import pytest
import torch

from conftest import ROOT, build_package_case
from spectralelementmethod_b200 import device, discrete, grid_importers as gi, meshgen
from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS

pytestmark = pytest.mark.gpu


def _basis(p):
    b1 = LagrangeGaussLobatto(p)
    return TensorProductQS(b1, b1)


def make_case(case, tmp_path=None):
    """(kind, p) -> DOF manager: structured straight / curved meshes, a shuffled Gmsh mesh,
    the annulus, and a condensed (DOFManagerSC) numbering."""
    kind, p = case
    if kind in ("S", "C"):
        return build_package_case(kind, 4, 3, p, False, False)[1]
    if kind == "SC":
        return build_package_case("C", 3, 3, p, True, True)[1]
    if kind == "annulus":
        return discrete.DOFManager(meshgen.annulus_sector_mesh(3, 8, p), 1, _basis(p),
                                   rcm_order=False)
    z = np.load(os.path.join(ROOT, "tests", "golden", "msh_%s.npz" % kind))
    path = tmp_path / "m.msh"
    path.write_bytes(z["msh_bytes"].tobytes())
    return discrete.DOFManager(gi.load_msh(str(path), 2), 1, _basis(int(z["meta"][2])),
                               rcm_order=True)


CASES = ([("S", p) for p in (2, 5, 8, 10, 12)] + [("C", p) for p in (2, 5, 8, 10, 16)]
         + [("q5_3x3_shuffled", 5), ("q8_2x2_shuffled", 8), ("annulus", 5), ("annulus", 10),
            ("SC", 8)])
IDS = ["%s-p%d" % c for c in CASES]


def f_t(x, y):
    return torch.sin(0.8 * x + 0.2) * torch.cos(0.5 * y) + 0.1 * x * y


def gradf_t(x, y):
    return (0.8 * torch.cos(0.8 * x + 0.2) * torch.cos(0.5 * y) + 0.1 * y,
            -0.5 * torch.sin(0.8 * x + 0.2) * torch.sin(0.5 * y) + 0.1 * x)


def w_np(x, y):
    return 1.0 + 0.25 * x * x + 0.1 * np.cos(y)


def w_t(x, y):
    return 1.0 + 0.25 * x * x + 0.1 * torch.cos(y)


def rel(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(b), 1e-300))


def example_coordinates(mngr):
    """The NumPy construction examples/poisson.py used before node_coordinates."""
    mesh = mngr.mesh
    l2g = mesh.node_map_array().reshape(mesh.n_cells, -1).astype(np.int64)
    xp = device.element_geometry(mngr._basis, mesh.nodes, l2g, jacobian=False)["x_phys"]
    X = np.zeros((2, mesh.n_nodes))
    X[:, l2g.ravel()] = xp.reshape(mesh.n_cells, 2, -1).transpose(1, 0, 2).reshape(2, -1)
    return X


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_against_the_host_mirror(case, tmp_path):
    mngr = make_case(case, tmp_path)
    n = mngr.mesh.n_nodes
    X = mngr.node_coordinates()
    assert np.array_equal(X.cpu().numpy(), example_coordinates(mngr))
    un = np.random.default_rng(case[1]).standard_normal(n)
    u = torch.from_numpy(un).cuda()
    g_dev, _ = mngr._element_gradients(u)
    g_dev = g_dev.cpu().numpy()
    ue = f_t(X[0], X[1])
    ge = torch.stack(gradf_t(X[0], X[1]))
    uen, gen = ue.cpu().numpy(), ge.cpu().numpy()
    num, den = np.zeros((2, n)), np.zeros(n)
    l2 = h1 = l2r = h1r = 0.0
    for e, fe in enumerate(mngr.finite_elements(x_phys=True, Jacobian=True)):
        ind = np.asarray(fe.node_ind)
        G = fe.gradient(un[ind])
        assert rel(g_dev[:, e].reshape(G.shape), G) < 1e-12, e
        np.add.at(num[0], ind, fe.detJxW * G[0])
        np.add.at(num[1], ind, fe.detJxW * G[1])
        np.add.at(den, ind, fe.detJxW)
        l2 += fe.integrate((un[ind] - uen[ind]) ** 2)
        h1 += fe.integrate((G[0] - gen[0][ind]) ** 2 + (G[1] - gen[1][ind]) ** 2)
        l2r += fe.integrate(uen[ind] ** 2)
        h1r += fe.integrate(gen[0][ind] ** 2 + gen[1][ind] ** 2)
    assert rel(mngr.gradient(u).cpu().numpy(), num / den) < 1e-12
    for ex, gx in ((f_t, gradf_t), (ue, ge)):        # callables and nodal values alike
        nrm = mngr.error_norms(u, ex, gx)
        for key, want in (("l2", l2), ("h1_semi", h1), ("l2_ref", l2r), ("h1_semi_ref", h1r)):
            assert abs(nrm[key] ** 2 - want) <= 1e-12 * abs(want), (key, nrm[key] ** 2, want)
        assert nrm["max_nodal"] == np.abs(un - uen).max()
    # the flux through every named boundary, scalar and callable weights
    for name in mngr.mesh._boundary_names:
        for w_dev, w_host in ((1.0, lambda x, y: 1.0), (w_t, w_np)):
            want, scale = 0.0, 0.0
            for fe, bfe in mngr.boundary_elements(name, x_phys=True, Jacobian=True):
                gn = (bfe.gradient(un[np.asarray(fe.node_ind)]) * bfe.unit_normal).sum(axis=0)
                terms = w_host(*bfe.x_phys) * gn * bfe.dSxW
                want += float(np.sum(terms))
                scale += float(np.abs(terms).sum())
            got = mngr.boundary_flux(u, name, w_dev)
            assert abs(got - want) <= 1e-12 * scale, (name, got, want)
    # the face normals against the host mirror's n_dSxW
    name = mngr.mesh._boundary_names[0]
    bf = device.BoundaryFaces(device.basis_tables(mngr._basis), mngr.mesh, name, X.device)
    want = np.stack([bfe.n_dSxW for _fe, bfe in mngr.boundary_elements(name, x_phys=True,
                                                                       Jacobian=True)])
    assert rel(bf.n_dSxW.cpu().numpy(), want) < 1e-14


@pytest.mark.parametrize("p", [2, 5, 8, 10])
def test_polynomials_have_exact_gradients_on_affine_meshes(p):
    mngr = build_package_case("S", 4, 3, p, False, False)[1]
    X = mngr.node_coordinates()
    x, y = X[0], X[1]
    rng = np.random.default_rng(p)
    u = torch.zeros_like(x)
    gx, gy = torch.zeros_like(x), torch.zeros_like(x)
    for i in range(p + 1):
        for j in range(p + 1 - i):
            c = float(rng.uniform(-1, 1)) / (i + j + 1)
            u += c * x ** i * y ** j
            if i:
                gx += c * i * x ** (i - 1) * y ** j
            if j:
                gy += c * j * x ** i * y ** (j - 1)
    g = mngr.gradient(u)
    scale = float(torch.stack([gx, gy]).abs().max())
    assert float((g - torch.stack([gx, gy])).abs().max()) <= 1e-12 * scale
    nrm = mngr.error_norms(u, u, (gx, gy))
    assert nrm["l2"] == 0.0 and nrm["max_nodal"] == 0.0
    assert nrm["h1_semi"] <= 1e-12 * nrm["h1_semi_ref"]


@pytest.mark.parametrize("case", [("S", 5), ("C", 8), ("q5_3x3_shuffled", 5), ("annulus", 8),
                                  ("SC", 8)], ids=lambda c: "%s-p%d" % c)
def test_energy_identity_against_the_apply(case, tmp_path):
    mngr = make_case(case, tmp_path)
    u = torch.from_numpy(np.random.default_rng(3).standard_normal(mngr.mesh.n_nodes)).cuda()
    op = mngr.poisson_operator()
    energy = float(torch.dot(u, op.apply_unmasked(u)))
    nrm = mngr.error_norms(u)
    assert abs(nrm["h1_semi"] ** 2 - energy) <= 1e-12 * energy
    assert nrm["l2_ref"] == 0.0 and nrm["h1_semi_ref"] == 0.0
    assert nrm["max_nodal"] == float(u.abs().max())
    # without a reference gradient the H1 entries are absent
    part = mngr.error_norms(u, exact=torch.zeros_like(u))
    assert part["h1_semi"] is None and part["h1_semi_ref"] is None and part["l2"] == nrm["l2"]


@pytest.mark.parametrize("p", [2, 4, 8])
def test_flux_of_a_quadratic_is_the_integral_of_its_laplacian(p):
    mngr = build_package_case("S", 4, 3, p, False, False)[1]
    X = mngr.node_coordinates()
    u = X[0] ** 2 + X[1] ** 2
    fe, fn = mngr.boundary_flux(u, "ebc"), mngr.boundary_flux(u, "nbc")
    assert abs(fe + fn - 16.0) <= 1e-12 * 16.0
    assert abs(fn - 8.0) <= 1e-12 * 8.0         # 2 x on x = 1 and 2 y on y = 1, each side 2 long
    assert abs(mngr.boundary_flux(u, "nbc", 0.5) - 4.0) <= 1e-12 * 4.0


def test_results_are_bitwise_reproducible_and_independent_of_the_operator():
    mngr = build_package_case("C", 6, 5, 8, True, True)[1]
    u = torch.from_numpy(np.random.default_rng(9).standard_normal(mngr.mesh.n_nodes)).cuda()
    a = (mngr.node_coordinates(), mngr.gradient(u), mngr.error_norms(u, f_t, gradf_t),
         mngr.boundary_flux(u, "nbc", w_t))
    b = (mngr.node_coordinates(), mngr.gradient(u), mngr.error_norms(u, f_t, gradf_t),
         mngr.boundary_flux(u, "nbc", w_t))
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert a[2] == b[2] and a[3] == b[3]
    # the plain and the condensed solution of one problem, through the same methods
    X = mngr.node_coordinates()
    on_ebc = mngr.boundary_node_mask("ebc")
    dv = f_t(X[0], X[1])
    plain, _ = mngr.poisson_operator(dirichlet=on_ebc).solve(1.0, dv, rtol=1e-13)
    cond, _ = mngr.condensed_poisson_operator(dirichlet=on_ebc).solve(1.0, dv, rtol=1e-13)
    np_, nc = mngr.error_norms(plain, f_t, gradf_t), mngr.error_norms(cond, f_t, gradf_t)
    for key in np_:
        assert abs(np_[key] - nc[key]) <= 1e-9 * max(abs(np_[key]), 1.0), key
    assert abs(mngr.boundary_flux(plain, "nbc") - mngr.boundary_flux(cond, "nbc")) < 1e-9
    assert float((mngr.gradient(plain) - mngr.gradient(cond)).abs().max()) < 1e-8


# -- the manufactured problem of examples/poisson.py --bc neumann -----------------------------
def u_exact(x, y):
    return torch.cos(0.9 * x + 0.3) + torch.cos(0.9 * y + 0.3) + 0.5 * torch.sin(0.7 * (x + y))


def _du(s, t):
    return -0.9 * torch.sin(0.9 * s + 0.3) + 0.35 * torch.cos(0.7 * (s + t))


def grad_exact(x, y):
    return _du(x, y), _du(y, x)


def f_exact(x, y):
    return (0.81 * (torch.cos(0.9 * x + 0.3) + torch.cos(0.9 * y + 0.3))
            + 0.49 * torch.sin(0.7 * (x + y)))


def flux_nbc(x, y):
    return torch.where(x >= y, _du(x, y), _du(y, x))


def test_manufactured_neumann_problem_converges_in_the_order():
    rows = []
    for p in range(4, 11):
        mngr = build_package_case("C", 6, 6, p, False, False)[1]
        X = mngr.node_coordinates()
        op = mngr.poisson_operator(dirichlet=mngr.boundary_node_mask("ebc"))
        u, info = op.solve(f_exact(X[0], X[1]), u_exact(X[0], X[1]), flux={"nbc": flux_nbc},
                           rtol=1e-13)
        assert info.converged, (p, info)
        nrm = mngr.error_norms(u, u_exact, grad_exact)
        g_int = float(op.boundary_load("nbc", flux_nbc).sum())
        rows.append((p, nrm["l2"], nrm["h1_semi"], abs(mngr.boundary_flux(u, "nbc") - g_int)))
    for r in rows:
        print("p=%2d  L2 %.3e  H1 %.3e  |flux - int g| %.3e" % r)
    floor = (1e-11, 1e-9, 1e-9)                     # roundoff level of each column
    for col in range(3):
        errs = [r[col + 1] for r in rows]
        for a, b in zip(errs, errs[1:]):
            assert b < a or b < floor[col], (col, errs)
        assert errs[-1] < 1e-3 * errs[0] and errs[-1] < floor[col] * 100, (col, errs)


def test_error_paths():
    mngr = build_package_case("S", 3, 3, 4, False, False)[1]
    n = mngr.mesh.n_nodes
    good = torch.zeros(n, dtype=torch.float64, device="cuda")
    for bad in (torch.zeros(n + 1, dtype=torch.float64, device="cuda"),
                torch.zeros(n, dtype=torch.float32, device="cuda"), np.zeros(n)):
        for call in (mngr.gradient, mngr.error_norms, lambda v: mngr.boundary_flux(v, "nbc")):
            with pytest.raises(ValueError):
                call(bad)
    with pytest.raises(ValueError):
        mngr.error_norms(good, exact=torch.zeros(n - 1, dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        mngr.error_norms(good, good, grad_exact=good)
    with pytest.raises(ValueError):
        mngr.boundary_flux(good, "nbc", weight=torch.zeros(3, dtype=torch.float64, device="cuda"))
    with pytest.raises(KeyError):
        mngr.boundary_flux(good, "no such boundary")
    # a mirrored mesh: every element inverted
    inv = build_package_case("S", 3, 3, 4, False, False)[1]
    inv.mesh.nodes[0] *= -1.0
    for call in (inv.node_coordinates, lambda: inv.gradient(good),
                 lambda: inv.error_norms(good), lambda: inv.boundary_flux(good, "nbc")):
        with pytest.raises(AssertionError):
            call()
