#!/usr/bin/env python
"""Cost of the nodal-field post-processing on a B200 (not part of the test suite).

At config 2 (1024 x 1024 elements, p = 8, straight cells, lexicographic numbering) the four
DOFManager methods -- ``node_coordinates``, ``gradient``, ``error_norms`` (nodal reference
values and gradient) and ``boundary_flux(u, "nbc")`` -- and, for scale, one unmasked
matrix-free apply are timed with CUDA events: ``--rounds`` rounds in which each of them runs
``--steps`` times in turn; the per-call medians over the rounds are reported.  The working set
(about 1 GB of mesh nodes alone) is far larger than the 126 MB L2, so every call streams from
HBM.  Each method ends in a device synchronise of its own (the Jacobian check), which the
times include.

The algorithmic bytes of each call (every array the call needs, touched once) and the
bandwidth they imply are printed beside the times, with the card's name and power limit
read in the same run.

    python tests/postprocess_bench.py [--nx 1024] [--order 8] [--steps 10] [--rounds 5]
                                      [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

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


def algorithmic_bytes(n_nodes, n_elem, NN, n_bnd_cells):
    """Bytes each call must move at least: mesh nodes (2 doubles per node), the L2G map
    (uint32 per entry), nodal vectors, element-local outputs, CSR tables."""
    n, ent = n_nodes, n_elem * NN
    geo = 16 * n + 4 * ent                          # mesh nodes + L2G
    return {
        "node_coordinates": geo + ent + 16 * n,     # + winner bytes, coordinates written
        # kernel: + u, grad_loc and jxw_loc written; three CSR sums: ptr, pos, values, out;
        # the division: 3 nodal rows read, 2 written
        "gradient": geo + 8 * n + 24 * ent + 3 * (4 * n + 4 * ent + 8 * ent + 8 * n)
        + 40 * n,
        "error_norms": geo + 8 * n + 8 * n + 16 * n,  # + u, u_ref, g_ref
        "boundary_flux": n_bnd_cells * NN * (16 + 4 + 8 + 16),
        "apply": None,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=1024)
    ap.add_argument("--order", type=int, default=8)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    from spectralelementmethod_b200 import discrete, meshgen
    from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS

    torch.cuda.set_device(0)
    b1 = LagrangeGaussLobatto(args.order)
    mesh = meshgen.structured_quad_mesh(args.nx, args.nx, args.order, "S")
    mngr = discrete.DOFManager(mesh, 1, TensorProductQS(b1, b1), rcm_order=False)
    op = mngr.poisson_operator()
    X = mngr.node_coordinates()
    u = torch.sin(3 * X[0]) * torch.cos(2 * X[1])
    u_ref = u + 1e-3 * torch.cos(X[0])
    g_ref = torch.stack([3 * torch.cos(3 * X[0]) * torch.cos(2 * X[1]),
                         -2 * torch.sin(3 * X[0]) * torch.sin(2 * X[1])])
    y = torch.empty_like(u)
    calls = {
        "node_coordinates": lambda: mngr.node_coordinates(),
        "gradient": lambda: mngr.gradient(u),
        "error_norms": lambda: mngr.error_norms(u, u_ref, g_ref),
        "boundary_flux": lambda: mngr.boundary_flux(u, "nbc"),
        "apply": lambda: op.apply_unmasked(u, out=y),
    }
    for f in calls.values():                        # warm-up: tables, modules, allocator
        f()
        f()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = {k: [] for k in calls}
    for _ in range(args.rounds):
        for k, f in calls.items():
            ev0.record()
            for _ in range(args.steps):
                f()
            ev1.record()
            torch.cuda.synchronize()
            times[k].append(ev0.elapsed_time(ev1) / args.steps)
    NN = (args.order + 1) ** 2
    n_bnd = len(set(c for c, _f in mesh._boundary_faces[mesh._boundary_id_lookup["nbc"]]))
    nbytes = algorithmic_bytes(mesh.n_nodes, mesh.n_cells, NN, n_bnd)
    res = {"card": card(), "elements": "%dx%d" % (args.nx, args.nx), "order": args.order,
           "n_nodes": int(mesh.n_nodes), "steps": args.steps, "rounds": args.rounds, "calls": {}}
    for k, v in times.items():
        ms = float(np.median(v))
        r = {"ms_median": ms, "ms_all": v}
        if nbytes[k] is not None:
            r["algorithmic_bytes"] = int(nbytes[k])
            r["GB_per_s"] = nbytes[k] / (ms * 1e-3) / 1e9
        r["vs_apply"] = ms / float(np.median(times["apply"]))
        res["calls"][k] = r
        print(json.dumps({k: r}), flush=True)
    print(json.dumps(res), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
