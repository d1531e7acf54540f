#!/usr/bin/env python
"""Cost of the Robin boundary term on a B200 (not part of the test suite).

1. Matrix-free apply at config 2 (1024 x 1024 elements, p = 8, Dirichlet on "ebc") with and
   without ``robin={"nbc": 1.0}``: the two operators alternate over several rounds of
   ``--steps`` applies each; the medians are reported.
2. Condensed three-level solve (1.0 load, ``--rtol``) in three cases: Dirichlet on "ebc" only
   (today's case, the reference point), Dirichlet on "ebc" + Robin on "nbc" (alpha = 1, g = 1),
   and pure Robin on "ebc" and "nbc" (no Dirichlet node): time to solution (set-up excluded),
   outer and inner iteration counts, true residual.

The card's name and power limit are read in the same run and printed with the numbers.

    python tests/robin_bench.py [--nx 1024] [--sc-nx 1024] [--steps 200] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    import torch
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=30)
        info["nvidia_smi"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi"] = "unavailable: %s" % e
    return info


def time_applies(ops, u, steps, rounds):
    import torch
    out = torch.empty_like(u)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = {k: [] for k in ops}
    for op in ops.values():
        for _ in range(10):
            op.apply(u, out=out)
    torch.cuda.synchronize()
    for _ in range(rounds):
        for k, op in ops.items():
            ev0.record()
            for _ in range(steps):
                op.apply(u, out=out)
            ev1.record()
            torch.cuda.synchronize()
            times[k].append(ev0.elapsed_time(ev1) / steps)
    return {k: {"ms_per_apply_median": float(np.median(v)), "ms_per_apply_all": v}
            for k, v in times.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=1024)
    ap.add_argument("--sc-nx", type=int, default=1024)
    ap.add_argument("--order", type=int, default=8)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--rtol", type=float, default=1e-12)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    from spectralelementmethod_b200 import discrete, meshgen
    from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS

    torch.cuda.set_device(0)
    res = {"card": card(), "order": args.order}
    b1 = LagrangeGaussLobatto(args.order)

    # 1. apply, config 2
    mesh = meshgen.structured_quad_mesh(args.nx, args.nx, args.order, "S")
    mngr = discrete.DOFManager(mesh, 1, TensorProductQS(b1, b1), rcm_order=False)
    on = mngr.boundary_node_mask("ebc")
    ops = {"plain": mngr.poisson_operator(dirichlet=on),
           "robin_nbc": mngr.poisson_operator(dirichlet=on, robin={"nbc": 1.0})}
    x, y = mesh.nodes
    u = torch.from_numpy(np.sin(3 * x) * np.cos(2 * y)).cuda()
    app = time_applies(ops, u, args.steps, args.rounds)
    app["boundary_nodes"] = int(ops["robin_nbc"]._bdiag.n)
    app["n_nodes"] = int(ops["plain"].n_nodes)
    app["elements"] = "%dx%d" % (args.nx, args.nx)
    app["extra_percent"] = 100.0 * (app["robin_nbc"]["ms_per_apply_median"]
                                    / app["plain"]["ms_per_apply_median"] - 1.0)
    res["apply"] = app
    print(json.dumps({"apply": app, "card": res["card"]}), flush=True)
    del ops, u, mngr, mesh
    torch.cuda.empty_cache()

    # 2. condensed three-level time to solution
    mesh = meshgen.structured_quad_mesh(args.sc_nx, args.sc_nx, args.order, "S")
    mngr = discrete.DOFManagerSC(mesh, 1, TensorProductQS(b1, b1), rcm_order=False)
    on = mngr.boundary_node_mask("ebc")
    cases = [("dirichlet_ebc", on, None, None),
             ("dirichlet_ebc_robin_nbc", on, {"nbc": 1.0}, {"nbc": 1.0}),
             ("pure_robin", None, {"ebc": 1.0, "nbc": 1.0}, {"ebc": 1.0, "nbc": 1.0})]
    res["condensed_three_level"] = {"elements": "%dx%d" % (args.sc_nx, args.sc_nx),
                                    "rtol": args.rtol}
    for name, mask, robin, flux in cases:
        t0 = time.perf_counter()
        sc = mngr.condensed_poisson_operator(dirichlet=mask, robin=robin)
        sc._build_top()                       # coarse levels: set-up, not solve
        torch.cuda.synchronize()
        t_setup = time.perf_counter() - t0
        vals = torch.zeros(sc.n_nodes, dtype=torch.float64, device="cuda")
        sc.solve(1.0, vals, flux=flux, rtol=args.rtol, preconditioner="three-level")  # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _u, info = sc.solve(1.0, vals, flux=flux, rtol=args.rtol, preconditioner="three-level")
        torch.cuda.synchronize()
        t = time.perf_counter() - t0
        r = {"seconds_to_solution": t, "setup_seconds": t_setup,
             "outer_iterations": info.iterations, "inner_iterations": info.inner_iterations,
             "inner_solves": info.inner_solves, "true_rel_residual": info.true_rel_residual,
             "converged": info.converged}
        res["condensed_three_level"][name] = r
        print(json.dumps({name: r}), flush=True)
        del sc, _u
        torch.cuda.empty_cache()
    print(json.dumps(res), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
