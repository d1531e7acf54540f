"""The separable element operator (semk_op.separable): on axis-aligned elements K1 writes the
cross factor G01 as an exact zero, and the apply kernels run y = D^T (G00 . D u) +
(G11 . u D^T) D with three barriers per patch.  Every product and sum it forms is one the
three-factor kernel forms when G01 is +-0, so on the same G the two kernels must give the
SAME BITS: clearing the field on an operator runs the three-factor kernel on its G.  The
three-factor kernels are in turn checked against the oracle (tests/test_gpu_parity.py);
a few cases repeat that comparison here."""
import contextlib
import math

import numpy as np
import pytest
import torch

import sem_oracle as so
from conftest import build_package_case, rel_l2
from spectralelementmethod_b200 import _lib, discrete, meshgen
from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS

pytestmark = pytest.mark.gpu


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def g01_slab(op):
    nnp = op.n1 * op.n1 * op.elems_per_patch
    return op.G[:, nnp:2 * nnp]


@contextlib.contextmanager
def three_factor(op):
    """The same operator (same G, same tables) through the three-factor kernel."""
    assert op.separable and op._op.separable == 1
    op._op.separable = 0
    try:
        yield op
    finally:
        op._op.separable = 1


def manager(nodes, nx, ny, p):
    mesh = meshgen.structured_quad_mesh(nx, ny, p, nodes=nodes)
    b1 = LagrangeGaussLobatto(p)
    return discrete.DOFManager(mesh, 1, TensorProductQS(b1, b1), rcm_order=False)


def lattice(nx, ny, p, transform=None, stretch=False):
    xy = meshgen.lattice_coordinates("S", nx, ny, p)
    if stretch:      # graded lattice: x = X^3-ish, y = sinh-like; still a tensor lattice
        X = np.linspace(0.0, 1.0, nx * p + 1) ** 1.7
        Y = np.sinh(2.0 * np.linspace(-1.0, 1.0, ny * p + 1))
        xy[0] = np.repeat(X, ny * p + 1)
        xy[1] = np.tile(Y, nx * p + 1)
    if transform is not None:
        xy = transform(xy)
    return np.ascontiguousarray(xy)


def rot(deg):
    c, s = math.cos(math.radians(deg)), math.sin(math.radians(deg))
    return lambda xy: np.stack([c * xy[0] - s * xy[1], s * xy[0] + c * xy[1]])


def test_g01_is_exactly_zero_on_axis_aligned_lattices():
    nx, ny, p = 6, 16, 6                 # whole 2 x 8 tiles: no empty slots
    rng = np.random.default_rng(1)
    u = dev(rng.standard_normal((nx * p + 1) * (ny * p + 1)))
    cases = {
        "S": lattice(nx, ny, p),
        "stretched": lattice(nx, ny, p, stretch=True),
        "rot+90": lattice(nx, ny, p, lambda xy: np.stack([-xy[1], xy[0]])),  # det J > 0
    }
    for name, nodes in cases.items():
        mngr = manager(nodes, nx, ny, p)
        op = mngr.poisson_operator()
        assert op.separable, name
        assert not bool(g01_slab(op).any()), name
        assert op.kernel_name.endswith(",SEP>"), op.kernel_name
        assert op.algorithmic_bytes_per_apply == 16 * op.n_nodes + 20 * op.n_elem * (p + 1) ** 2
        # G00 and G11 are positive on every element node (det J > 0 after the rotation too)
        nnp = op.n1 * op.n1 * op.elems_per_patch
        assert bool((op.G[:, :nnp] > 0).all()) and bool((op.G[:, 2 * nnp:3 * nnp] > 0).all())
        # the element-local geometry agrees with the weak-form symmetry: A is symmetric
        v = dev(rng.standard_normal(op.n_nodes))
        a = float(torch.dot(v, op.apply_unmasked(u)))
        b = float(torch.dot(u, op.apply_unmasked(v)))
        assert abs(a - b) <= 1e-12 * max(abs(a), abs(b)), name
    # curved and 30-degree-rotated elements keep their cross factor and three factors
    for name, nodes in (("C", meshgen.lattice_coordinates("C", nx, ny, p)),
                        ("rot30", lattice(nx, ny, p, rot(30.0)))):
        op = manager(nodes, nx, ny, p).poisson_operator()
        assert not op.separable and op._op.separable == 0, name
        assert bool(g01_slab(op).any()), name
        assert op.algorithmic_bytes_per_apply == 16 * op.n_nodes + 28 * op.n_elem * (p + 1) ** 2


def test_pair_mapping_keeps_three_factors():
    mesh, mngr = build_package_case("S", 2, 8, 16, False, False)
    op = mngr.poisson_operator(mode="pair")
    assert op.kernel_variant == 1 and not op.separable
    assert not bool(g01_slab(op).any())


def _modes(p, pe):
    n1 = p + 1
    out = ["column"]
    if pe in (8, 16) or (pe == 32 and n1 <= 7):
        out.append("box")
    return out


def _pes(p):
    return [4, 8, 16] + ([32] if p + 1 <= 7 else [])


CASES = [(p, pe, mode) for p in range(2, 16) for pe in _pes(p) for mode in _modes(p, pe)]


@pytest.mark.parametrize("p,pe,mode", CASES)
def test_separable_kernel_is_bit_identical_to_three_factor_kernel(p, pe, mode):
    nx, ny = 5, 19                       # ragged tiles: empty slots in the last patches
    mesh, mngr = build_package_case("S", nx, ny, p, False, False)
    n = mngr.ndof
    rng = np.random.default_rng(100 + p)
    u = dev(rng.standard_normal(n))
    on = np.zeros(n, dtype=bool)
    ids = np.arange(n).reshape(nx * p + 1, ny * p + 1)
    on[ids[0, :]] = True
    on[ids[:, 0]] = True
    on[ids[nx * p - 1, ny * p - 1]] = True
    for dirichlet in (None, on):
        try:
            op = mngr.poisson_operator(mode=mode, elems_per_patch=pe, dirichlet=dirichlet)
        except NotImplementedError:
            pytest.skip("patch of %d elements does not fit shared memory at p = %d" % (pe, p))
        assert op.separable and op.kernel_variant == (2 if mode == "box" else 0)
        assert not bool(g01_slab(op).any())
        d0 = torch.zeros(1, dtype=torch.float64, device="cuda")
        d1 = torch.zeros(1, dtype=torch.float64, device="cuda")
        for flags in (None, 0, _lib.MASK_IN, _lib.MASK_OUT, _lib.MASK_IN | _lib.MASK_OUT):
            y_sep = op.apply(u, flags=flags, dot_out=d0)
            with three_factor(op):
                y_3 = op.apply(u, flags=flags, dot_out=d1)
            assert torch.equal(y_sep, y_3), (dirichlet is not None, flags)
            assert torch.equal(d0, d1), (dirichlet is not None, flags)


@pytest.mark.parametrize("as_callable", [False, True])
def test_weighted_and_robin_operators(as_callable):
    nx, ny, p = 4, 16, 8
    mesh, mngr = build_package_case("S", nx, ny, p, False, False)
    n = mngr.ndof
    rng = np.random.default_rng(7)
    u = dev(rng.standard_normal(n))
    if as_callable:
        weight = lambda x, y: 2.0 + x * y          # noqa: E731
    else:
        weight = rng.uniform(1.0, 3.0, size=(nx * ny, p + 1, p + 1))
    op = mngr.poisson_operator(weight=weight, robin={"nbc": 0.5})
    assert op.separable and not bool(g01_slab(op).any())
    d0 = torch.zeros(1, dtype=torch.float64, device="cuda")
    d1 = torch.zeros(1, dtype=torch.float64, device="cuda")
    y_sep = op.apply(u, dot_out=d0)
    with three_factor(op):
        y_3 = op.apply(u, dot_out=d1)
    assert torch.equal(y_sep, y_3) and torch.equal(d0, d1)


def test_staged_host_apply_and_native_pcg():
    nx, ny, p = 8, 24, 8
    mesh, mngr = build_package_case("S", nx, ny, p, False, False)
    n = mngr.ndof
    on = np.zeros(n, dtype=bool)
    on[: ny * p + 1] = True
    op = mngr.poisson_operator(dirichlet=on)
    assert op.separable
    rng = np.random.default_rng(9)
    uh = torch.from_numpy(rng.standard_normal(n)).pin_memory()
    y_dev = op.apply(uh.cuda())
    for stages in (1, 3, 8):
        yh = torch.full((n,), float("nan"), dtype=torch.float64).pin_memory()
        op.apply_host(uh, yh, stages=stages)
        assert torch.equal(yh, y_dev.cpu())
        with three_factor(op):
            y3 = torch.full((n,), float("nan"), dtype=torch.float64).pin_memory()
            op.apply_host(uh, y3, stages=stages)
        assert torch.equal(yh, y3)
    b = op.lift(op.rhs(1.0), None)
    x0, i0 = op.solve_pcg(b, rtol=1e-10, maxiter=20000)
    with three_factor(op):
        x1, i1 = op.solve_pcg(b, rtol=1e-10, maxiter=20000)
    assert i0.converged and i0.iterations == i1.iterations and torch.equal(x0, x1)


@pytest.mark.parametrize("nx,ny,p,pe,mode", [(2, 8, 10, 8, "box"), (4, 16, 6, 16, "column"),
                                            (3, 9, 4, 8, "box")])
def test_separable_kernel_vs_oracle_and_atomic(nx, ny, p, pe, mode):
    mesh, mngr = build_package_case("S", nx, ny, p, False, False)
    r = so.run_case("S", nx, ny, p, False, False, solve=False)
    rng = np.random.default_rng(12)
    u = rng.standard_normal(mngr.ndof)
    ref = so.apply_dense_batched(r["L"], r["l2g"], u)
    op = mngr.poisson_operator(mode=mode, elems_per_patch=pe)     # device geometry (T2)
    assert op.separable
    y = op.apply_unmasked(dev(u))
    assert rel_l2(y.cpu().numpy(), ref) < 1e-11
    ya = op.apply_atomic(dev(u), flags=0)
    assert rel_l2(ya.cpu().numpy(), y.cpu().numpy()) < 1e-12


def test_resident_ctas_and_smem_report_the_separable_footprint():
    mesh, mngr = build_package_case("S", 4, 16, 8, False, False)
    op = mngr.poisson_operator()
    c = mngr.poisson_operator(mode="column")
    assert op.separable and c.separable and op.kernel_variant == 2
    lib = _lib.load()
    args = (op.n1, op.elems_per_patch, op.g_patch_stride, int(op.plan_scalars[_lib.PS_PN_STRIDE]),
            int(op.plan_scalars[_lib.PS_EL_STRIDE]), int(op.plan_scalars[_lib.PS_INV_STRIDE]))
    full = lib.semk_patch_smem_bytes(*args)
    sep = lib.semk_patch_smem_bytes_sep(1, *args)
    assert full - sep == 8 * op.n1 * op.n1 * op.elems_per_patch
    assert op.smem_bytes == sep and c.smem_bytes == sep
    assert lib.semk_patch_smem_bytes_sep(0, *args) == full
    assert op.resident_ctas == lib.semk_resident_ctas_sep(2, 1, *args) > 0
    assert lib.semk_resident_ctas_sep(0, 0, *args) == lib.semk_resident_ctas(*args)
    # at p = 8 the separable kernel keeps three CTAs per SM
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert op.resident_ctas == 3 * sms
