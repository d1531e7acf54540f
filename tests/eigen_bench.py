#!/usr/bin/env python
"""Cost of the block eigensolver on a B200 (not part of the test suite).

1. The block kernels at config-2 length (n = 8193^2 nodes; every block is far larger than the
   126 MB L2, so each call streams from HBM), timed with CUDA events over ``--reps`` calls:
   - the Gram kernel at m = k = 48 with a weight (the Rayleigh-Ritz Gram matrices of block
     size 16), its DFMA and DMMA inner products (semk_block_gram_dfma_f64 / _dmma_f64)
     alternated in one run;
   - the same 48 x 48 Gram matrix (no weight) from 48 calls of semk_multi_dot_f64, alternated
     with one call of the Gram kernel;
   - the combine kernel at m = 48, k = 32 (the X and P update), beta = 0 and beta = 1.
   Bytes and flops come from the shapes (semk.h); the bound is the larger of bytes over
   7.7 TB/s and flops over the FP64 rate measured earlier in this project
   (profiles/r02_dmma_rate.txt: 37 TFLOP/s DMMA, 35.6 TFLOP/s DFMA).
2. The tolerance of the condensed three-level solve that preconditions LOBPCG: iterations and
   time of the 16 smallest pairs at ``--sweep-nx`` elements per side for several values.
3. The 16 smallest pairs at config 2 (1024 x 1024 elements, p = 8, Dirichlet on "ebc",
   tol = 1e-8), once with each Gram kernel: wall time (set-up of both operators included, and
   separately), iterations and the per-phase split of the solver.

The card's name and power limit are read in the same run.  One JSON line is printed (and
written to ``--out`` if given).

    python tests/eigen_bench.py [--nx 1024] [--order 8] [--k 16] [--reps 5] [--sweep-nx 256]
                                [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HBM = 7.7e12
FP64 = {"dfma": 35.6e12, "dmma": 37.0e12}


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


def timed(fn, reps):
    import torch
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


def rate(name, t, nbytes, flops, peak):
    bound = max(nbytes / HBM, flops / peak)
    return {"kernel": name, "time_ms": 1e3 * t, "GB_per_s": nbytes / t / 1e9,
            "TFLOP_per_s": flops / t / 1e12, "bound_ms": 1e3 * bound,
            "bound_by": "HBM bandwidth" if nbytes / HBM >= flops / peak else "FP64 rate",
            "share_of_bound": bound / t}


def block_kernels(n, reps):
    import torch
    from spectralelementmethod_b200 import _lib, device
    from spectralelementmethod_b200.eigen import BlockKernels
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    m, k = 48, 48
    g = torch.Generator(device=dev).manual_seed(0)
    X = torch.rand((m, n), dtype=torch.float64, device=dev, generator=g)
    Y = torch.rand((k, n), dtype=torch.float64, device=dev, generator=g)
    w = torch.rand(n, dtype=torch.float64, device=dev, generator=g)
    kern = {v: BlockKernels(dev, max_mk=m * k, gram_kernel=v) for v in ("dfma", "dmma")}
    blk = BlockKernels(dev, max_mk=m * k)
    G = torch.empty(m * k, dtype=torch.float64, device=dev)
    out = []
    gram_bytes, gram_flops = 8 * n * (m + k + 1), 2 * n * m * k
    ts = {"dfma": [], "dmma": []}
    res = {}
    for _ in range(3):                   # alternate the two inner products
        for v in ("dfma", "dmma"):
            ts[v].append(timed(lambda: kern[v].gram(X, Y, w, out=G), reps))
            res[v] = G.clone()
    for v in ("dfma", "dmma"):
        out.append(rate("gram_%s m=k=48 w" % v, min(ts[v]), gram_bytes, gram_flops, FP64[v]))
    out.append({"dfma_vs_dmma_max_rel_diff":
                float(((res["dfma"] - res["dmma"]).abs().max() / res["dfma"].abs().max()).item())})
    # the same Gram matrix by m calls of semk_multi_dot_f64 (out[j] = Y_j . X_i, j < k)
    md = torch.empty((m, k + 1), dtype=torch.float64, device=dev)
    part = torch.zeros(int(lib.semk_multi_dot_partials_len(k)), dtype=torch.float64, device=dev)

    def multi():
        for i in range(m):
            _lib.check(lib.semk_multi_dot_f64(n, k, device.ptr(Y), n, device.ptr(X[i]),
                                              device.ptr(md[i]), device.ptr(part),
                                              device.stream_ptr()))
    tg, tm = [], []
    for _ in range(3):
        tg.append(timed(lambda: blk.gram(X, Y, None, out=G), reps))
        tm.append(timed(multi, max(1, reps // 2)))
    agree = float(((md[:, :k].reshape(-1) - G).abs().max() / G.abs().max()).item())
    out.append(rate("gram m=k=48 (no w)", min(tg), 8 * n * (m + k), gram_flops, FP64["dfma"]))
    out.append(dict(rate("48 x multi_dot k=48", min(tm), 8 * n * m * (k + 1), gram_flops,
                         FP64["dfma"]), max_rel_diff_to_gram=agree,
                    speedup_of_gram=min(tm) / min(tg)))
    Yc = Y[:32]
    C = torch.rand((m, 32), dtype=torch.float64, device=dev, generator=g)
    for beta in (0.0, 1.0):
        t = min(timed(lambda: blk.combine(X, C, Yc, beta), reps) for _ in range(2))
        out.append(rate("combine m=48 k=32 beta=%g" % beta, t,
                        8 * n * (m + 32 * (2 if beta else 1)), 2 * n * m * 32, FP64["dfma"]))
    del X, Y, w, Yc
    torch.cuda.empty_cache()
    return out


def manager(nx, p):
    from spectralelementmethod_b200 import discrete, meshgen
    from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS
    b1 = LagrangeGaussLobatto(p)
    return discrete.DOFManagerSC(meshgen.structured_quad_mesh(nx, nx, p, "S"), 1,
                                 TensorProductQS(b1, b1), rcm_order=False)


def eigen_run(nx, p, k, gram_kernel="default"):
    import torch
    from spectralelementmethod_b200 import eigen
    eigen.GRAM_KERNEL = gram_kernel
    dm = manager(nx, p)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    lam, X, info = dm.poisson_eigenpairs(k, dirichlet="ebc", tol=1e-8)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    exact = np.sort([np.pi ** 2 / 16 * ((2 * a + 1) ** 2 + (2 * b + 1) ** 2)
                     for a in range(12) for b in range(12)])[:k]
    r = {"nx": nx, "p": p, "k": k, "n_nodes": int(dm.mesh.n_nodes), "wall_s": wall,
         "iterations": info["iterations"], "status": info["status"],
         "preconditioner_applications": info["preconditioner_applications"],
         "inner_iterations": info["inner_iterations"], "restarts": info["restarts"],
         "time_split_s": info["time"], "block_GB": info["block_bytes"] / 1e9,
         "max_residual": float(np.max(info["residuals"])),
         "max_rel_err_vs_exact": float(np.max(np.abs(lam - exact) / exact))}
    r["setup_s"] = wall - sum(info["time"].values())
    r["gram_kernel"] = gram_kernel
    eigen.GRAM_KERNEL = "default"
    del X
    torch.cuda.empty_cache()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=1024)
    ap.add_argument("--order", type=int, default=8)
    ap.add_argument("--k", type=int, default=16)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sweep-nx", type=int, default=256)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from spectralelementmethod_b200 import eigen
    torch.cuda.set_device(0)
    res = {"card": card()}
    n = (a.nx * a.order + 1) ** 2
    res["block_kernels"] = block_kernels(n, a.reps)
    sweep = []
    default = eigen.CONDENSED_RTOL
    for rtol in (1e-1, 1e-2, 1e-3):
        eigen.CONDENSED_RTOL = rtol
        sweep.append(dict(eigen_run(a.sweep_nx, a.order, a.k), condensed_rtol=rtol))
    eigen.CONDENSED_RTOL = default
    res["condensed_rtol_sweep"] = sweep
    res["eigen"] = [dict(eigen_run(a.nx, a.order, a.k, g), condensed_rtol=default)
                    for g in ("dfma", "dmma")]
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
