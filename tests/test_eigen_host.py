"""Argument checks of the eigensolver and the block kernels' size query (no GPU needed)."""
import numpy as np
import pytest

from spectralelementmethod_b200 import _lib, discrete, meshgen
from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS
from spectralelementmethod_b200.eigen import _dirichlet_mask


def small_manager():
    b1 = LagrangeGaussLobatto(2)
    return discrete.DOFManagerSC(meshgen.structured_quad_mesh(2, 2, 2), 1,
                                 TensorProductQS(b1, b1), rcm_order=False)


def test_block_count_limits_and_free_nodes():
    dm = small_manager()
    for k in (0, 33):
        with pytest.raises(ValueError):
            dm.poisson_eigenpairs(k)
    with pytest.raises(ValueError):                       # 3 x 3 free nodes remain
        dm.poisson_eigenpairs(9, dirichlet=["ebc", "nbc"])


def test_dirichlet_argument_forms():
    dm = small_manager()
    ebc = dm.boundary_node_mask("ebc")
    assert _dirichlet_mask(dm, None) is None
    assert np.array_equal(_dirichlet_mask(dm, "ebc"), ebc)
    assert np.array_equal(_dirichlet_mask(dm, ebc), ebc)
    both = _dirichlet_mask(dm, ["ebc", "nbc"])
    assert np.array_equal(both, ebc | dm.boundary_node_mask("nbc"))
    with pytest.raises(ValueError):
        _dirichlet_mask(dm, np.zeros(3, dtype=bool))


def test_gram_partials_length():
    lib = _lib.load()
    per = lib.semk_block_gram_partials_len(1, 1) - 2
    assert per > 0
    assert lib.semk_block_gram_partials_len(48, 48) == per * 48 * 48 + 2
    for m, k in ((97, 1), (1, 97), (0, 5)):
        assert lib.semk_block_gram_partials_len(m, k) == -1
