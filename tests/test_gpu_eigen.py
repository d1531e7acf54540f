"""Lowest eigenpairs of the Poisson operator on the device (eigen.py, csrc/semk_block.cu): the
block Gram and combine kernels against NumPy, eigenvalues against the exact spectrum of the
square and against dense scipy on the assembled discrete problem, and the solver's invariants."""
import numpy as np
import pytest
import torch
from scipy import linalg as sla

from spectralelementmethod_b200 import _lib, device, discrete, meshgen
from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS
from spectralelementmethod_b200.eigen import BlockKernels

pytestmark = pytest.mark.gpu


def manager(nx, ny, p, kind="S", sc=True):
    b1 = LagrangeGaussLobatto(p)
    mesh = meshgen.structured_quad_mesh(nx, ny, p, kind)
    cls = discrete.DOFManagerSC if sc else discrete.DOFManager
    return cls(mesh, 1, TensorProductQS(b1, b1), rcm_order=False)


GRAM_KERNELS = ["default", "dfma", "dmma"]


@pytest.fixture(scope="module")
def kernels():
    return {g: BlockKernels(torch.device("cuda", 0), max_mk=96 * 96, gram_kernel=g)
            for g in GRAM_KERNELS}


@pytest.fixture(scope="module")
def blk(kernels):
    return kernels["default"]


def padded_block(rng, m, n, pad=5):
    """[m, n] view with row stride n + pad of a random CUDA block."""
    full = torch.from_numpy(rng.standard_normal((m, n + pad))).cuda()
    return full[:, :n]


# -- block kernels ----------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 1000, 1000003])
@pytest.mark.parametrize("m", [1, 7, 48, 96])
@pytest.mark.parametrize("k", [1, 7, 48, 96])
@pytest.mark.parametrize("gram_kernel", GRAM_KERNELS)
def test_block_gram_against_numpy(kernels, gram_kernel, n, m, k):
    blk = kernels[gram_kernel]
    rng = np.random.default_rng(n + 100 * m + k)
    X, Y = padded_block(rng, m, n), padded_block(rng, k, n)
    assert X.stride(0) > n and Y.stride(0) > n
    w = torch.from_numpy(rng.uniform(0.5, 2.0, n)).cuda()
    Xh, Yh, wh = X.cpu().numpy(), Y.cpu().numpy(), w.cpu().numpy()
    for wd, wn in ((None, np.ones(n)), (w, wh)):
        G = blk.gram(X, Y, wd)
        ref = (Xh * wn) @ Yh.T
        scale = (np.abs(Xh) * wn) @ np.abs(Yh).T
        assert G.shape == (m, k)
        assert np.all(np.abs(G - ref) <= 1e-14 * scale + 1e-300), np.abs(G - ref).max()
        assert np.array_equal(G, blk.gram(X, Y, wd))            # bitwise reproducible


@pytest.mark.parametrize("n", [1, 1000, 1000003])
@pytest.mark.parametrize("m", [1, 7, 48, 96])
@pytest.mark.parametrize("k", [1, 7, 48, 96])
def test_block_combine_against_numpy(blk, n, m, k):
    rng = np.random.default_rng(7 * n + 10 * m + k)
    X = padded_block(rng, m, n)
    C = rng.standard_normal((m, k))
    Y0 = padded_block(rng, k, n, pad=3)
    Xh, Y0h = X.cpu().numpy(), Y0.cpu().numpy()
    for beta in (0.0, 1.0):
        Y = Y0.clone() if beta else torch.full_like(Y0, float("nan"))   # beta = 0 ignores Y
        Y = torch.cat([Y, torch.zeros_like(Y[:, :3])], 1)[:, :n]
        blk.combine(X, C, Y, beta)
        ref = beta * Y0h + C.T @ Xh
        scale = abs(beta) * np.abs(Y0h) + np.abs(C).T @ np.abs(Xh)
        got = Y.cpu().numpy()
        assert np.all(np.abs(got - ref) <= 1e-14 * scale + 1e-300), np.abs(got - ref).max()
        Y2 = Y0.clone() if beta else torch.empty_like(Y0)
        Y2 = torch.cat([Y2, torch.zeros_like(Y2[:, :3])], 1)[:, :n]
        blk.combine(X, C, Y2, beta)
        assert torch.equal(Y, Y2)


def test_block_kernels_reject_out_of_range():
    lib = _lib.load()
    assert lib.semk_block_gram_partials_len(97, 1) == -1
    X = torch.zeros((97, 16), dtype=torch.float64, device="cuda")
    G = torch.zeros(97 * 97, dtype=torch.float64, device="cuda")
    part = torch.zeros(int(lib.semk_block_gram_partials_len(96, 96)), dtype=torch.float64,
                       device="cuda")
    st = device.stream_ptr()
    with pytest.raises(ValueError):
        _lib.check(lib.semk_block_gram_f64(16, 97, device.ptr(X), 16, 1, device.ptr(X), 16, None,
                                           device.ptr(G), device.ptr(part), st))
    with pytest.raises(ValueError):
        _lib.check(lib.semk_block_gram_f64(16, 1, device.ptr(X), 15, 1, device.ptr(X), 16, None,
                                           device.ptr(G), device.ptr(part), st))
    with pytest.raises(ValueError):
        _lib.check(lib.semk_block_combine_f64(16, 97, device.ptr(X), 16, 1, device.ptr(G), 0.0,
                                              device.ptr(X), 16, st))
    with pytest.raises(ValueError):
        _lib.check(lib.semk_block_combine_f64(16, 1, device.ptr(X), 16, 97, device.ptr(G), 0.0,
                                              device.ptr(X), 16, st))


# -- exact eigenvalues of the square ----------------------------------------------------------
def exact(kind, count):
    r = np.arange(0, 12)
    if kind == "dirichlet":
        v = [np.pi ** 2 / 4 * (a * a + b * b) for a in r[1:] for b in r[1:]]
    elif kind == "example":
        v = [np.pi ** 2 / 16 * ((2 * a + 1) ** 2 + (2 * b + 1) ** 2) for a in r for b in r]
    else:
        v = [np.pi ** 2 / 4 * (a * a + b * b) for a in r for b in r]
    return np.sort(v)[:count]


BOUNDARIES = {"dirichlet": ["ebc", "nbc"], "example": "ebc", "neumann": None}


@pytest.mark.parametrize("mesh_kind", ["S", "C"])
@pytest.mark.parametrize("bc", ["dirichlet", "example", "neumann"])
def test_exact_eigenvalues_of_the_square(mesh_kind, bc):
    dm = manager(8, 8, 8, mesh_kind)
    lam, X, info = dm.poisson_eigenpairs(10, dirichlet=BOUNDARIES[bc], tol=1e-8)
    assert info["status"] == "converged" and info["converged"].all(), info
    assert info["preconditioner"] == "three-level"
    ref = exact(bc, 10)
    if bc == "neumann":
        assert abs(lam[0]) <= 1e-10
        x0 = X[0].cpu().numpy()
        assert np.abs(np.abs(x0) - 0.5).max() <= 1e-6      # M-normalised constant on [-1, 1]^2
        assert np.all(np.abs(lam[1:] - ref[1:]) <= 1e-10 * ref[1:])
    else:
        assert np.all(np.abs(lam - ref) <= 1e-10 * ref), (lam, ref)


# -- against dense scipy on the assembled discrete problem -------------------------------------
def dense_reference(dm, mask, robin, weight):
    op = dm.poisson_operator(dirichlet=mask, robin=robin, weight=weight)
    K = op.to_scipy_csr(masked=False).toarray()
    M = op.mass_diagonal().cpu().numpy()
    free = np.ones(dm.mesh.n_nodes, bool) if mask is None else ~mask
    lam, V = sla.eigh(K[np.ix_(free, free)], np.diag(M[free]))
    return lam, V, free, M


def check_against_dense(dm, k, dirichlet, robin, weight):
    lam, X, info = dm.poisson_eigenpairs(k, dirichlet=dirichlet, robin=robin, weight=weight,
                                         maxiter=3000)
    assert info["status"] == "converged", info
    mask = None if dirichlet is None else dm.boundary_node_mask(dirichlet)
    ref, V, free, M = dense_reference(dm, mask, robin, weight)
    # 1e-10 relative to each eigenvalue; a zero one (pure Neumann) to 1e-10 absolute
    bound = np.where(np.abs(ref[:k]) < 1e-8, 1e-10, 1e-10 * np.abs(ref[:k]))
    assert np.all(np.abs(lam - ref[:k]) <= bound), (lam, ref[:k])
    Xf = X.cpu().numpy()[:, free].T * np.sqrt(M[free])[:, None]
    Vf = V * np.sqrt(M[free])[:, None]
    # clusters of equal eigenvalues that lie wholly within the first k
    i = 0
    while i < k:
        j = i + 1
        while j < len(ref) and ref[j] - ref[j - 1] <= 1e-8 * max(abs(ref[j]), 1.0):
            j += 1
        if j <= k:
            ang = sla.subspace_angles(Xf[:, i:j], Vf[:, i:j])
            assert ang.max() <= 1e-6, (i, j, ang)
        i = j


def weight_fn(x, y):
    return 1.0 + 0.5 * x * x + 0.25 * torch.sin(y)


@pytest.mark.parametrize("sc", [True, False])
def test_against_dense_scipy_structured(sc):
    dm = manager(4, 4, 8, "C", sc=sc)                     # 1089 nodes
    check_against_dense(dm, 8, "ebc", {"nbc": 2.0}, None)
    dm = manager(5, 4, 6, "S", sc=sc)                     # 775 nodes
    check_against_dense(dm, 8, "ebc", None, weight_fn)


def test_against_dense_scipy_pinwheel():
    b1 = LagrangeGaussLobatto(4)
    mesh = meshgen.pinwheel_mesh(7, 4, rings=3)           # 589 nodes, unstructured
    dm = discrete.DOFManagerSC(mesh, 1, TensorProductQS(b1, b1), rcm_order=True)
    check_against_dense(dm, 8, None, {"ebc": 2.0}, weight_fn)
    check_against_dense(dm, 8, "ebc", None, None)


# -- invariants ---------------------------------------------------------------------------------
def test_orthonormality_dirichlet_zeros_and_reproducibility():
    dm = manager(8, 8, 6, "C")
    lam, X, info = dm.poisson_eigenpairs(12, dirichlet="ebc", robin={"nbc": 1.5})
    mask = dm.boundary_node_mask("ebc")
    M = dm.poisson_operator().mass_diagonal().cpu().numpy()
    Xh = X.cpu().numpy()
    assert X.shape == (12, dm.mesh.n_nodes) and X.is_cuda
    assert np.abs((Xh * M) @ Xh.T - np.eye(12)).max() <= 1e-12
    assert np.all(Xh[:, mask] == 0.0)
    assert np.all(np.diff(lam) >= 0)
    lam2, X2, _ = dm.poisson_eigenpairs(12, dirichlet="ebc", robin={"nbc": 1.5})
    assert np.array_equal(lam, lam2) and torch.equal(X, X2)
    assert len(info["residuals"]) == 12 and info["converged"].all()
    assert info["preconditioner_applications"] > 0 and info["iterations"] > 0


@pytest.mark.parametrize("dirichlet", ["ebc", None])
def test_jacobi_and_multilevel_agree(dirichlet):
    """None: pure Neumann, K singular -- the preconditioners are built for K + M (Jacobi
    1/diag(K + M), the condensed operator with reaction JxW)."""
    lam_j, _, info_j = manager(6, 6, 4, sc=False).poisson_eigenpairs(6, dirichlet=dirichlet,
                                                                     maxiter=3000)
    lam_m, _, info_m = manager(6, 6, 4, sc=True).poisson_eigenpairs(6, dirichlet=dirichlet)
    assert info_j["preconditioner"] == "jacobi" and info_m["preconditioner"] == "three-level"
    assert info_j["status"] == "converged" and info_m["status"] == "converged"
    bound = np.where(lam_m < 1e-8, 1e-10, 1e-10 * lam_m)
    assert np.all(np.abs(lam_j - lam_m) <= bound), (lam_j, lam_m)
    if dirichlet is None:
        assert abs(lam_m[0]) <= 1e-10 and abs(lam_j[0]) <= 1e-10


def test_zero_robin_coefficient_is_the_neumann_problem():
    """alpha = 0 on every boundary leaves K singular: the solver must still precondition K + M."""
    dm = manager(6, 6, 4)
    lam_r, _, info_r = dm.poisson_eigenpairs(6, robin={"ebc": 0.0, "nbc": 0.0})
    lam_n, _, _ = dm.poisson_eigenpairs(6)
    assert info_r["status"] == "converged"
    assert abs(lam_r[0]) <= 1e-10
    assert np.all(np.abs(lam_r[1:] - lam_n[1:]) <= 1e-10 * lam_n[1:])


def test_multilevel_iterations_do_not_grow_with_the_mesh():
    its = {}
    for ne in (32, 128):
        _, _, info = manager(ne, ne, 4).poisson_eigenpairs(4, dirichlet="ebc")
        assert info["status"] == "converged"
        its[ne] = info["iterations"]
    assert its[128] <= 1.5 * its[32], its
