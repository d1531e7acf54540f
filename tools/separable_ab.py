"""In-process A/B of the separable apply (semk_op.separable = 1) against the three-factor
kernel on the same operator and the same G (field cleared), at config 2 (1024 x 1024
S elements, p = 8, the box kernel).  Rounds alternate the two kernels; each round times
`--applies` back-to-back applies with CUDA events.  Every output of the two kernels is
compared bit for bit.

    python tools/separable_ab.py --out profiles/separable_ab_config2.json
    python tools/separable_ab.py --geom-dump DIR/geom.npz      # K1 outputs on an S mesh
    python tools/separable_ab.py --geom-compare A.npz B.npz    # bitwise comparison
    python tools/separable_ab.py --dump-compare A.npy B.npy    # two bench --dump-outputs

The bench's apply output y = A u of the smooth field u = sin 3x cos 2y cancels by about h^2
(||y||_inf is ~1e-5 of the terms it sums), so the difference of two builds is measured
against the term scale ||diag(A)||_inf ||u||_inf of the config-2 operator as well.

The geometry dump lets two builds be compared: K1 drops the roundoff of J01 / J10 on
axis-aligned elements, and x_phys, det J, the diagonal of invJ, G00, G11 and JxW must come
out bitwise unchanged."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def manager(nx, ny, p):
    from spectralelementmethod_b200 import discrete, meshgen
    from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS
    mesh = meshgen.structured_quad_mesh(nx, ny, p, "S")
    b1 = LagrangeGaussLobatto(p)
    return discrete.DOFManager(mesh, 1, TensorProductQS(b1, b1), rcm_order=False)


def geom_dump(path, nx=128, ny=128, p=8):
    import torch
    from spectralelementmethod_b200 import device
    mngr = manager(nx, ny, p)
    mesh = mngr.mesh
    N = p + 1
    g = device.element_geometry(mngr._basis, mesh.nodes, mesh.node_map_array())
    op = mngr.poisson_operator()
    nnp = N * N * op.elems_per_patch
    G = op.G
    np.savez(path, x_phys=g["x_phys"], detJ=g["detJ"],
             invJ_diag=np.stack([g["invJ"][:, 0, 0], g["invJ"][:, 1, 1]]),
             invJ_off=np.stack([g["invJ"][:, 0, 1], g["invJ"][:, 1, 0]]),
             G00=G[:, :nnp].cpu().numpy(), G01=G[:, nnp:2 * nnp].cpu().numpy(),
             G11=G[:, 2 * nnp:3 * nnp].cpu().numpy(), JxW=op.JxW.cpu().numpy())
    torch.cuda.synchronize()


def geom_compare(a, b):
    A, B = np.load(a), np.load(b)
    out = {}
    for k in A.files:
        x, y = A[k], B[k]
        same = bool(np.array_equal(x.view(np.uint64), y.view(np.uint64)))
        out[k] = {"bitwise_equal": same, "max_abs_diff": float(np.abs(x - y).max()),
                  "max_abs": float(np.abs(x).max()), "nonzero_a": int(np.count_nonzero(x)),
                  "nonzero_b": int(np.count_nonzero(y))}
    return out


def dump_compare(a, b, nx=1024, p=8):
    import torch
    ya, yb = np.load(a), np.load(b)
    op = manager(nx, nx, p).poisson_operator()
    dmax = float(op.diagonal(masked=False).abs().max())
    nodes = op.dof_mngr.mesh.nodes
    umax = float(np.abs(np.sin(3 * nodes[0]) * np.cos(2 * nodes[1])).max())
    diff = float(np.abs(ya - yb).max())
    ymax = float(np.abs(ya).max())
    torch.cuda.synchronize()
    return {"entries": int(ya.size), "bitwise_equal": bool(np.array_equal(ya, yb)),
            "max_abs_diff": diff, "y_inf": ymax, "diag_inf": dmax, "u_inf": umax,
            "diff_over_y_inf": diff / ymax, "diff_over_term_scale": diff / (dmax * umax)}


def ab(args):
    import torch
    t0 = time.time()
    mngr = manager(args.nx, args.nx, args.p)
    op = mngr.poisson_operator()
    setup = time.time() - t0
    assert op.separable, "config 2 is a tensor lattice: the operator must be separable"
    n = op.n_nodes
    g = torch.Generator(device="cuda").manual_seed(0)
    u = torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
    ys = {1: torch.empty_like(u), 0: torch.empty_like(u)}
    dots = {1: torch.zeros(1, dtype=torch.float64, device="cuda"),
            0: torch.zeros(1, dtype=torch.float64, device="cuda")}
    times = {1: [], 0: []}
    for sep in (1, 0):                       # warm-up of both instantiations
        op._op.separable = sep
        for _ in range(10):
            op.apply(u, out=ys[sep], dot_out=dots[sep])
    torch.cuda.synchronize()
    same = bool(torch.equal(ys[1], ys[0]) and torch.equal(dots[1], dots[0]))
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(args.rounds):
        for sep in ((1, 0) if r % 2 == 0 else (0, 1)):
            op._op.separable = sep
            ev0.record()
            for _ in range(args.applies):
                op.apply(u, out=ys[sep])
            ev1.record()
            ev1.synchronize()
            times[sep].append(ev0.elapsed_time(ev1) / args.applies)
    op._op.separable = 1
    same = same and bool(torch.equal(ys[1], ys[0]))
    med = {k: float(np.median(v)) for k, v in times.items()}
    res = {
        "gpu": gpu_info(),
        "case": "%dx%d S elements, p=%d, %d DOF, %s" % (args.nx, args.nx, args.p, n, op.kernel_name),
        "applies_per_round": args.applies, "rounds_per_kernel": args.rounds,
        "ms_per_apply_separable": times[1], "ms_per_apply_three_factor": times[0],
        "median_ms_separable": med[1], "median_ms_three_factor": med[0],
        "speedup": med[0] / med[1],
        "gdof_per_s_separable": n / med[1] / 1e6, "gdof_per_s_three_factor": n / med[0] / 1e6,
        "algorithmic_bytes_separable": op.algorithmic_bytes_per_apply,
        "algorithmic_bytes_three_factor": 16 * n + 28 * op.n_elem * op.n1 * op.n1,
        "resident_ctas": op.resident_ctas, "smem_bytes_per_cta": op.smem_bytes,
        "outputs_bit_identical": same, "setup_seconds": setup,
    }
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=1024)
    ap.add_argument("--p", type=int, default=8)
    ap.add_argument("--applies", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default="")
    ap.add_argument("--geom-dump", default="")
    ap.add_argument("--geom-compare", nargs=2, default=None)
    ap.add_argument("--dump-compare", nargs=2, default=None)
    args = ap.parse_args()
    if args.geom_dump:
        geom_dump(args.geom_dump)
        return
    if args.geom_compare:
        res = geom_compare(*args.geom_compare)
    elif args.dump_compare:
        res = dump_compare(*args.dump_compare)
    else:
        res = ab(args)
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
