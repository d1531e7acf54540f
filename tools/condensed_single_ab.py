#!/usr/bin/env python
"""Time of the condensed single-load passes through their C entries (the same signatures in
every build), for an A/B of two builds run alternately in separate processes.

At config 2 (1024 x 1024 elements, p = 8, Dirichlet on "ebc", W and A_ii^-1 kept): element
pass in RHS mode with c, element pass in BACKSOLVE mode (``semk_sc_element_react_f64``),
back-solve over W (``semk_sc_backsolve_stored_f64``) and load over A_ii^-1 and W
(``semk_sc_load_stored_f64``); CUDA events around ``--reps`` calls after two warm-up calls,
per-call median of ``--rounds`` windows.  The inputs (12.5 + 19 GB of W and A_ii^-1) exceed the
126 MB L2.  Prints one JSON line with the card's name and power limit.

    python tools/condensed_single_ab.py --root TREE [--tag NAME] [--nx 1024] [--order 8]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument("--tag", default="")
    ap.add_argument("--nx", type=int, default=1024)
    ap.add_argument("--order", type=int, default=8)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    sys.path.insert(0, args.root)
    import torch
    from spectralelementmethod_b200 import _lib, device, discrete, meshgen
    from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS
    torch.cuda.set_device(0)
    b1 = LagrangeGaussLobatto(args.order)
    dm = discrete.DOFManagerSC(meshgen.structured_quad_mesh(args.nx, args.nx, args.order, "S"), 1,
                               TensorProductQS(b1, b1), rcm_order=False)
    sc = dm.condensed_poisson_operator(dirichlet=dm.boundary_node_mask("ebc"),
                                       store_interior=True, store_interior_inverse=True)
    f64 = dict(dtype=torch.float64, device=sc.dev)
    E, NE, NI = sc.n_elem, sc.n_ext_loc, sc.n_int_loc
    f = torch.from_numpy(np.random.default_rng(0).standard_normal(sc.n_nodes)).cuda()
    u = torch.from_numpy(np.random.default_rng(1).standard_normal(sc.n_nodes)).cuda()
    g_loc, c = torch.empty((E, NE), **f64), torch.empty((E, NI), **f64)
    lib, P, st = sc._lib, device.ptr, device.stream_ptr()

    def element(mode, g=None, uu=None, cc=None):
        _lib.check(lib.semk_sc_element_react_f64(
            sc.n1, E, None, P(sc.G), sc.g_stride, 1, P(sc.tab.dev()[0]), P(sc._t["ext_loc"]),
            P(sc.l2g_dev), P(sc.JxW), P(f), 1.0, mode, None, sc.s_stride, None, P(g), P(uu),
            None, P(cc), None, None, P(sc._bad), st))

    passes = {
        "element_rhs_c": lambda: element(_lib.SC_RHS, g=g_loc, cc=c),
        "element_backsolve": lambda: element(_lib.SC_BACKSOLVE, uu=u),
        "backsolve_stored": lambda: _lib.check(lib.semk_sc_backsolve_stored_f64(
            sc.n1, E, P(sc._W), P(c), P(sc.l2g_dev), P(sc._t["ext_loc"]), P(u), st)),
        "load_stored": lambda: _lib.check(lib.semk_sc_load_stored_f64(
            sc.n1, E, P(sc._W), P(sc._Ainv), P(sc.l2g_dev), P(sc._t["ext_loc"]), P(sc.JxW),
            P(f), 1.0, P(g_loc), P(c), st)),
    }
    out = {}
    for name, fn in passes.items():
        fn()
        fn()
        windows = []
        for _ in range(args.rounds):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            for _ in range(args.reps):
                fn()
            b.record()
            torch.cuda.synchronize()
            windows.append(a.elapsed_time(b) / args.reps)
        out[name] = {"ms_median": float(np.median(windows)), "ms_windows": windows}
    assert int(sc._bad.item()) == 0
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        smi = "unavailable: %s" % e
    print(json.dumps({"tag": args.tag, "device": torch.cuda.get_device_name(0), "nvidia_smi": smi,
                      "nx": args.nx, "order": args.order, "reps": args.reps, "passes": out}))


if __name__ == "__main__":
    main()
