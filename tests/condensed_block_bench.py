#!/usr/bin/env python
"""Cost of the condensed block loads on a B200 (not part of the test suite).

At config 2 (1024 x 1024 elements, p = 8, Dirichlet on "ebc"):

1. The split of one ``solve_load`` at rtol 1e-2, the preconditioner application of
   ``poisson_eigenpairs``: load pass (element kernel, RHS mode, interior load kept), PCG
   (three-level driver) and back-solve (stream over W), each closed by a device synchronise.
2. The block passes at k = 1, 2, 4, 8, 16, 32 against k single passes, alternated in one run,
   as time per column: the element pass in RHS mode (with c, as in the solve) and in BACKSOLVE
   mode, the stored back-solve over W and, on an operator that also keeps A_ii^-1, the stored
   load.  The stored kernels also report their bytes per column.  Every block column is checked
   to be bitwise the single pass.
3. ``poisson_eigenpairs(16, dirichlet="ebc")``: wall time and per-phase split, beside the
   figures recorded before the block preconditioner (profiles/eigen_bench_config2.json).

The card's name and power limit are read in the same run.  One JSON line is printed (and
written to ``--out`` if given).

    python tests/condensed_block_bench.py [--nx 1024] [--order 8] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from eigen_bench import card, eigen_run, manager  # noqa: E402

KS = (1, 2, 4, 8, 16, 32)


def sync_time(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def split_of_solve_load(sc, r, f, reps=3):
    """Load pass / PCG / back-solve of solve_load, the same calls in the same order."""
    import torch
    from spectralelementmethod_b200 import _lib, device
    rows = []
    for _ in range(reps + 1):
        t_load, g = sync_time(lambda: sc.rhs(f))
        b = torch.empty_like(g)

        def finish():
            _lib.check(sc._lib.semk_sc_rhs_finish_f64(
                sc.n_ext, device.ptr(g), device.ptr(r), device.ptr(sc.dirichlet_dev),
                device.ptr(b), device.stream_ptr()))
        t_fin, _ = sync_time(finish)
        t_pcg, (x, info) = sync_time(lambda: sc.solve_pcg(b, rtol=1e-2,
                                                          preconditioner="three-level"))
        t_back, _ = sync_time(lambda: sc.backsolve(x, f))
        rows.append({"load_s": t_load, "finish_s": t_fin, "pcg_s": t_pcg, "backsolve_s": t_back,
                     "outer_iterations": info.iterations,
                     "inner_iterations": info.inner_iterations})
    rows = rows[1:]                       # the first round warms up every shape
    return {key: float(np.median([r[key] for r in rows])) for key in rows[0]}


def block_passes(sc, F, stored_load=False):
    """Per-column time of the block passes against single passes, alternated per k."""
    import torch
    from spectralelementmethod_b200 import _lib, device
    f64 = dict(dtype=torch.float64, device=sc.dev)
    E, NE, NI = sc.n_elem, sc.n_ext_loc, sc.n_int_loc
    kmax = F.shape[0]
    g_blk = torch.empty((kmax, E, NE), **f64)
    c_blk = torch.empty((kmax, E, NI), **f64)
    g_one = torch.empty((E, NE), **f64)
    c_one = torch.empty((E, NI), **f64)
    U = torch.zeros((kmax, sc.n_nodes), **f64)
    U[:, :sc.n_ext].copy_(F[:, :sc.n_ext])
    Uo = U[0].clone()
    cols = [(1.0, F[j], True) for j in range(kmax)]
    out = []

    def load_of(k):
        return sc._chunk_load(cols, list(range(k)), F)

    if stored_load:
        def blk_rhs(k):
            _, ldf, mask, scales = load_of(k)
            _lib.check(sc._lib.semk_sc_load_stored_block_f64(
                sc.n1, E, device.ptr(sc._W), device.ptr(sc._Ainv), device.ptr(sc.l2g_dev),
                device.ptr(sc._t["ext_loc"]), device.ptr(sc.JxW), k, device.ptr(F), ldf, mask,
                scales, device.ptr(g_blk), E * NE, device.ptr(c_blk), E * NI,
                device.stream_ptr()))

        def one_rhs(j):
            _lib.check(sc._lib.semk_sc_load_stored_f64(
                sc.n1, E, device.ptr(sc._W), device.ptr(sc._Ainv), device.ptr(sc.l2g_dev),
                device.ptr(sc._t["ext_loc"]), device.ptr(sc.JxW), device.ptr(F[j]), 1.0,
                device.ptr(g_one), device.ptr(c_one), device.stream_ptr()))
        # bytes: A_ii^-1, W, JxW and l2g once; per column the gathered load and g, c written
        NN = sc.n1 * sc.n1
        kinds = {"load_stored": (blk_rhs, one_rhs, 8 * E * (NI * NI + NE * NI) + 12 * E * NN,
                                 8 * E * (NN + NE + NI))}
    else:
        def blk_rhs(k):
            sc._element_block(_lib.SC_RHS, load_of(k), g_loc=g_blk, c=c_blk)

        def one_element(mode, f, g_loc=None, u=None, c=None):
            """The single-load C entry: one load pass of the element kernel."""
            _lib.check(sc._lib.semk_sc_element_react_f64(
                sc.n1, E, None, device.ptr(sc.G), sc.g_stride, 1, device.ptr(sc.tab.dev()[0]),
                device.ptr(sc._t["ext_loc"]), device.ptr(sc.l2g_dev), device.ptr(sc.JxW),
                device.ptr(f), 1.0, mode, None, sc.s_stride, None, device.ptr(g_loc),
                device.ptr(u), None, device.ptr(c), device.ptr(sc._react), None,
                device.ptr(sc._bad), device.stream_ptr()))

        def one_rhs(j):
            one_element(_lib.SC_RHS, F[j], g_loc=g_one, c=c_one)

        def blk_back(k):
            sc._element_block(_lib.SC_BACKSOLVE, load_of(k), U=U)

        def one_back(j):
            one_element(_lib.SC_BACKSOLVE, F[j], u=Uo)

        def blk_stored(k):
            _lib.check(sc._lib.semk_sc_backsolve_stored_block_f64(
                sc.n1, E, device.ptr(sc._W), device.ptr(c_blk), E * NI, device.ptr(sc.l2g_dev),
                device.ptr(sc._t["ext_loc"]), k, device.ptr(U), U.stride(0),
                device.stream_ptr()))

        def one_stored(j):
            _lib.check(sc._lib.semk_sc_backsolve_stored_f64(
                sc.n1, E, device.ptr(sc._W), device.ptr(c_one), device.ptr(sc.l2g_dev),
                device.ptr(sc._t["ext_loc"]), device.ptr(Uo), device.stream_ptr()))
        kinds = {"element_rhs": (blk_rhs, one_rhs, None, None),
                 "element_backsolve": (blk_back, one_back, None, None),
                 # bytes: W once; per column c and u_e read, u_i written
                 "backsolve_stored": (blk_stored, one_stored, 8 * E * NE * NI,
                                      8 * E * (2 * NI + NE))}
    for name, (blk, one, shared_bytes, col_bytes) in kinds.items():
        blk(1)
        one(0)
        for k in KS:
            if k > kmax:
                break
            t_one, _ = sync_time(lambda: [one(j) for j in range(k)])
            t_blk, _ = sync_time(lambda: blk(k))
            row = {"pass": name, "k": k, "single_ms_per_col": 1e3 * t_one / k,
                   "block_ms_per_col": 1e3 * t_blk / k, "speedup": t_one / t_blk}
            if shared_bytes is not None:
                nbytes = shared_bytes + k * col_bytes
                row["block_bytes_per_col_MB"] = nbytes / k / 1e6
                row["block_GB_per_s"] = nbytes / t_blk / 1e9
            out.append(row)
    # bitwise: the last block pass of each kind against a single pass on column kmax - 1
    j = kmax - 1
    blk_rhs(kmax)
    one_rhs(j)
    out.append({"pass": "rhs" if not stored_load else "load_stored",
                "bitwise_last_column": bool(torch.equal(g_blk[j], g_one)
                                            and torch.equal(c_blk[j], c_one))})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=1024)
    ap.add_argument("--order", type=int, default=8)
    ap.add_argument("--k", type=int, default=16)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    torch.cuda.set_device(0)
    res = {"card": card(), "nx": a.nx, "p": a.order}
    dm = manager(a.nx, a.order)
    mask = dm.boundary_node_mask("ebc")
    op = dm.poisson_operator(dirichlet=mask)
    mass = op.mass_diagonal()
    del op
    sc = dm.condensed_poisson_operator(dirichlet=mask)
    res["W_stored"] = sc._W is not None
    n = sc.n_nodes
    inv_mass_int = torch.zeros(n, dtype=torch.float64, device=sc.dev)
    inv_mass_int[sc.n_ext:] = 1.0 / mass[sc.n_ext:]
    del mass
    gen = torch.Generator(device=sc.dev).manual_seed(0)
    r = torch.randn(n, dtype=torch.float64, device=sc.dev, generator=gen)
    r[:sc.n_ext][sc.dirichlet_dev.bool()] = 0.0
    res["solve_load_split"] = split_of_solve_load(sc, r, r * inv_mass_int)
    F = torch.randn((max(KS), n), dtype=torch.float64, device=sc.dev, generator=gen)
    res["block_passes"] = block_passes(sc, F)
    del sc
    torch.cuda.empty_cache()
    sci = dm.condensed_poisson_operator(dirichlet=mask, store_interior=True,
                                        store_interior_inverse=True)
    res["block_passes"] += block_passes(sci, F, stored_load=True)
    del sci, F, r, inv_mass_int, dm
    torch.cuda.empty_cache()
    res["eigen"] = eigen_run(a.nx, a.order, a.k)
    with open(os.path.join(ROOT, "profiles", "eigen_bench_config2.json")) as fh:
        before = json.loads(fh.readline())
    ref = [e for e in before["eigen"] if e.get("gram_kernel") == "dmma"][0]
    res["eigen_before"] = {key: ref[key] for key in ("wall_s", "iterations",
                                                     "preconditioner_applications",
                                                     "inner_iterations", "time_split_s")}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
