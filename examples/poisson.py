#!/usr/bin/env python
"""Poisson's equation on a plate -- the reference's example on the B200 engine.

Mirrors the flow of the reference's examples/poisson.py (mesh -> essential /
natural boundary conditions -> operators -> solve) through the drop-in API of
this package; the per-element einsum loop (examples/poisson.py:145-200) and
the sparse direct solve (:203-259, sem/discrete.py:502-528) are replaced by
the matrix-free device operator and the device-resident Jacobi-PCG.

    -lap(u) = 1 on [-1, 1]^2,  u = 0.2 ((x + 1) + (y + 1)) on "ebc" (left + bottom),
    du/dn = 0 on "nbc" (right + top)              (examples/poisson.py:125-143, :200)

    python examples/poisson.py [--n 64] [--order 8] [--msh file.msh] [--kind S|C]
                               [--solver matrix-free|condensed|condensed-two-level]
                               [--bc reference|neumann|robin]

``--solver condensed`` follows the reference example literally: static
condensation of the element interiors (DOFManagerSC, sem/discrete.py:404-528),
solve on the element-exterior DOFs, interior back-substitution -- on the device;
``condensed-two-level`` adds the vertex coarse space to the Jacobi preconditioner.

``--bc neumann`` / ``--bc robin`` solve a manufactured problem instead: u smooth and known,
f = -lap(u) as nodal values, u on "ebc", and on "nbc" the flux condition du/dn = g
(``neumann``) or the Robin condition du/dn + 2 u = g (``robin``) with g taken from u; the
max nodal error against u is printed.

With ``--msh`` the mesh is read from a Gmsh 2.2 binary file with physical
names "ebc", "nbc" (lines) and a surface (the reference's examples/meshes/
square.geo); otherwise a structured n x n mesh is built (and, with
``--write-msh``, written out and read back through the importer).
"""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from spectralelementmethod_b200 import discrete, grid_importers, meshgen  # noqa: E402
from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS  # noqa: E402


def u_exact(x, y, m=np):
    """Manufactured solution of ``--bc neumann|robin`` (symmetric in x and y, so the two faces
    at the corner (1, 1) of "nbc" agree on the flux there)."""
    return m.cos(0.9 * x + 0.3) + m.cos(0.9 * y + 0.3) + 0.5 * m.sin(0.7 * (x + y))


def f_exact(x, y):
    return 0.81 * (np.cos(0.9 * x + 0.3) + np.cos(0.9 * y + 0.3)) + 0.49 * np.sin(0.7 * (x + y))


def flux_nbc(x, y):
    """du/dn on "nbc" (right side: du/dx; top side: du/dy) on CUDA tensors."""
    import torch

    def du(s, t):
        return -0.9 * torch.sin(0.9 * s + 0.3) + 0.35 * torch.cos(0.7 * (s + t))
    return torch.where(x >= y, du(x, y), du(y, x))


def gll_coordinates(mngr):
    """Physical coordinates of every GLL node (the solution's nodes), [2, n_nodes]."""
    from spectralelementmethod_b200 import device
    mesh = mngr.mesh
    l2g = mesh.node_map_array().reshape(mesh.n_cells, -1).astype(np.int64)
    xp = device.element_geometry(mngr._basis, mesh.nodes, l2g, jacobian=False)["x_phys"]
    X = np.zeros((2, mesh.n_nodes))
    X[:, l2g.ravel()] = xp.reshape(mesh.n_cells, 2, -1).transpose(1, 0, 2).reshape(2, -1)
    return X


def run(n=16, order=8, msh=None, kind="S", write_msh=None, rtol=1e-12, quiet=False,
        solver="matrix-free", bc="reference"):
    import torch
    t0 = time.perf_counter()
    if msh is None and write_msh is not None:
        msh = meshgen.write_gmsh22_binary(write_msh, n, n, order, kind)
    if msh is not None:
        mesh = grid_importers.load_msh(msh, 2)
    else:
        mesh = meshgen.structured_quad_mesh(n, n, order, kind)
    b1 = LagrangeGaussLobatto(order)
    mngr = discrete.DOFManagerSC(mesh, 1, TensorProductQS(b1, b1), rcm_order=False)

    # essential boundary values, boundary element by boundary element, like the reference
    soln = np.zeros(mngr.ndof)
    on_ebc = np.zeros(mngr.ndof, dtype=bool)
    f, extra, robin = 1.0, {}, None
    if bc == "reference":
        for _fe, bfe in mngr.boundary_elements("ebc", x_phys=True):
            loc = bfe.node_ind
            x, y = bfe.x_phys
            soln[loc] = 0.2 * ((x + 1) + (y + 1))
            on_ebc[loc] = True
    elif bc in ("neumann", "robin"):
        X = gll_coordinates(mngr)
        on_ebc = mngr.boundary_node_mask("ebc")
        soln = u_exact(X[0], X[1])
        f = torch.from_numpy(f_exact(X[0], X[1])).cuda()
        if bc == "neumann":
            extra["flux"] = {"nbc": flux_nbc}
        else:
            robin = {"nbc": 2.0}
            extra["flux"] = {"nbc": lambda x, y: flux_nbc(x, y) + 2.0 * u_exact(x, y, torch)}
    else:
        raise ValueError("bc must be 'reference', 'neumann' or 'robin'")
    t_setup = time.perf_counter() - t0

    t0 = time.perf_counter()
    if solver in ("condensed", "condensed-two-level"):
        op = mngr.condensed_poisson_operator(dirichlet=on_ebc, robin=robin)
        if solver == "condensed-two-level":
            extra["preconditioner"] = "two-level"
    elif solver == "matrix-free":
        op = mngr.poisson_operator(dirichlet=on_ebc, robin=robin)
    else:
        raise ValueError("solver must be 'matrix-free', 'condensed' or 'condensed-two-level'")
    u, info = op.solve(f=f, dirichlet_values=torch.from_numpy(soln).to(op.dev), rtol=rtol,
                       **extra)
    torch.cuda.synchronize()
    t_solve = time.perf_counter() - t0
    u = u.cpu().numpy()
    if not quiet:
        print("mesh: %d cells of order %d, %d DOF (%d on the essential boundary)"
              % (mesh.n_cells, order, mngr.ndof, int(on_ebc.sum())))
        print("host set-up %.2f s; %s operator + PCG %.2f s: %d iterations, relative residual %.2e"
              % (t_setup, solver, t_solve, info.iterations, info.rel_residual))
        print("u: min %.6f  max %.6f  mean %.6f" % (u.min(), u.max(), u.mean()))
        if bc != "reference":
            print("%s boundary on \"nbc\": max nodal error %.3e" % (bc, np.abs(u - soln).max()))
    return mngr, on_ebc, soln, u, info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=64, help="cells per side of the structured mesh")
    ap.add_argument("--order", type=int, default=8)
    ap.add_argument("--kind", default="S", choices=["S", "C"], help="straight or curved cells")
    ap.add_argument("--msh", default=None, help="Gmsh 2.2 binary mesh to read instead")
    ap.add_argument("--write-msh", default=None,
                    help="write the structured mesh to this .msh file and read it back")
    ap.add_argument("--solver", default="matrix-free", choices=["matrix-free", "condensed", "condensed-two-level"])
    ap.add_argument("--bc", default="reference", choices=["reference", "neumann", "robin"],
                    help="reference: the reference example (du/dn = 0 on \"nbc\"); neumann / "
                         "robin: a manufactured problem with flux / Robin data on \"nbc\"")
    args = ap.parse_args()
    run(args.n, args.order, args.msh, args.kind, args.write_msh, solver=args.solver, bc=args.bc)


if __name__ == "__main__":
    main()
