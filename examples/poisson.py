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
                               [--bc reference|neumann|robin] [--convergence] [--eigen K]

``--solver condensed`` follows the reference example literally: static
condensation of the element interiors (DOFManagerSC, sem/discrete.py:404-528),
solve on the element-exterior DOFs, interior back-substitution -- on the device;
``condensed-two-level`` adds the vertex coarse space to the Jacobi preconditioner.

``--bc neumann`` / ``--bc robin`` solve a manufactured problem instead: u smooth and known,
f = -lap(u) as nodal values, u on "ebc", and on "nbc" the flux condition du/dn = g
(``neumann``) or the Robin condition du/dn + 2 u = g (``robin``) with g taken from u; the
max nodal, L2 and H1 errors against u are printed (``DOFManager.error_norms``), and the flux
of the solution through "nbc" (``DOFManager.boundary_flux``) beside the integral of the
exact flux.  ``--convergence`` solves that problem on the same mesh for p = 2 ... 10 and
prints one row per order: the errors fall exponentially in p.

``--eigen K`` computes the K smallest eigenvalues of -lap(u) = lambda u with the example's
boundary layout instead -- u = 0 on "ebc", du/dn = 0 on "nbc" (``DOFManager.poisson_eigenpairs``)
-- and prints them beside the exact ones, pi^2/16 ((2m+1)^2 + (2n+1)^2), m, n >= 0.

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


def _du(s, t):
    import torch
    return -0.9 * torch.sin(0.9 * s + 0.3) + 0.35 * torch.cos(0.7 * (s + t))


def grad_exact(x, y):
    """Gradient of ``u_exact`` on CUDA tensors."""
    return _du(x, y), _du(y, x)


def flux_nbc(x, y):
    """du/dn on "nbc" (right side: du/dx; top side: du/dy) on CUDA tensors."""
    import torch
    return torch.where(x >= y, _du(x, y), _du(y, x))


def run(n=16, order=8, msh=None, kind="S", write_msh=None, rtol=1e-12, quiet=False,
        solver="matrix-free", bc="reference", report=None):
    """Solve; returns (mngr, on_ebc, essential values, u, info).  With ``bc`` neumann / robin,
    ``report`` (a dict, if given) receives the error norms and the "nbc" fluxes."""
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
        X = mngr.node_coordinates().cpu().numpy()
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
    post = {} if report is None else report
    if bc != "reference":
        post.update(mngr.error_norms(u, lambda x, y: u_exact(x, y, torch), grad_exact),
                    flux=mngr.boundary_flux(u, "nbc"),
                    flux_exact=float(op.boundary_load("nbc", flux_nbc).sum()))
    u = u.cpu().numpy()
    if not quiet:
        print("mesh: %d cells of order %d, %d DOF (%d on the essential boundary)"
              % (mesh.n_cells, order, mngr.ndof, int(on_ebc.sum())))
        print("host set-up %.2f s; %s operator + PCG %.2f s: %d iterations, relative residual %.2e"
              % (t_setup, solver, t_solve, info.iterations, info.rel_residual))
        print("u: min %.6f  max %.6f  mean %.6f" % (u.min(), u.max(), u.mean()))
        if bc != "reference":
            print("%s boundary on \"nbc\": max nodal error %.3e" % (bc, np.abs(u - soln).max()))
            print("errors: L2 %.3e  H1 semi-norm %.3e" % (post["l2"], post["h1_semi"]))
            print("flux through \"nbc\": %.15f (integral of the exact flux %.15f)"
                  % (post["flux"], post["flux_exact"]))
    return mngr, on_ebc, soln, u, info


def convergence(n=8, kind="S", solver="matrix-free", bc="neumann", orders=range(2, 11)):
    """The manufactured problem of ``--bc neumann|robin`` on one structured n x n mesh for
    every order: one row of errors per order."""
    print("%3s %9s %6s %11s %11s %11s %11s" % ("p", "DOF", "iters", "max nodal", "L2", "H1 semi",
                                               "flux error"))
    for p in orders:
        rep = {}
        mngr, _on_ebc, _soln, _u, info = run(n, p, None, kind, rtol=1e-13, quiet=True,
                                             solver=solver, bc=bc, report=rep)
        print("%3d %9d %6d %11.3e %11.3e %11.3e %11.3e"
              % (p, mngr.ndof, info.iterations, rep["max_nodal"], rep["l2"], rep["h1_semi"],
                 abs(rep["flux"] - rep["flux_exact"])))


def eigen(k, n=16, order=8, kind="S", msh=None):
    """The k smallest eigenvalues with u = 0 on "ebc" and natural "nbc", beside the exact ones of
    the square [-1, 1]^2."""
    if msh is not None:
        mesh = grid_importers.load_msh(msh, 2)
    else:
        mesh = meshgen.structured_quad_mesh(n, n, order, kind)
    b1 = LagrangeGaussLobatto(order)
    mngr = discrete.DOFManagerSC(mesh, 1, TensorProductQS(b1, b1), rcm_order=False)
    t0 = time.perf_counter()
    lam, _x, info = mngr.poisson_eigenpairs(k, dirichlet="ebc")
    t = time.perf_counter() - t0
    r = np.arange(k + 1)
    ex = np.sort((np.pi ** 2 / 16) * ((2 * r[:, None] + 1) ** 2 + (2 * r[None, :] + 1) ** 2),
                 axis=None)[:k]
    print("mesh: %d cells of order %d, %d DOF; %d LOBPCG iterations (%s preconditioner), %.2f s"
          % (mesh.n_cells, order, mngr.ndof, info["iterations"], info["preconditioner"], t))
    print("%3s %22s %22s %10s" % ("i", "lambda", "exact", "rel. err"))
    for i in range(k):
        print("%3d %22.15f %22.15f %10.2e" % (i, lam[i], ex[i], abs(lam[i] - ex[i]) / ex[i]))
    return lam, ex


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
    ap.add_argument("--convergence", action="store_true",
                    help="solve the manufactured problem (--bc neumann unless robin is given) "
                         "for p = 2 ... 10 on the structured --n x --n mesh and print the "
                         "errors per order")
    ap.add_argument("--eigen", type=int, default=0, metavar="K",
                    help="print the K smallest eigenvalues (u = 0 on \"ebc\", natural \"nbc\") "
                         "beside the exact ones instead of solving")
    args = ap.parse_args()
    if args.eigen:
        eigen(args.eigen, args.n, args.order, args.kind, args.msh)
        return
    if args.convergence:
        convergence(args.n, args.kind, args.solver, "robin" if args.bc == "robin" else "neumann")
        return
    run(args.n, args.order, args.msh, args.kind, args.write_msh, solver=args.solver, bc=args.bc)


if __name__ == "__main__":
    main()
