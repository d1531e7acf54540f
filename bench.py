#!/usr/bin/env python
"""Benchmark of the hot path: FP64 matrix-free Poisson operator apply (p = 8).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # engine arm
    python bench.py --impl reference [--gpus N] [--steps K] ...    # CPU reference arm
    python bench.py ... --dump-outputs DIR     # engine arm, plus the last step's output in DIR

A "step" is one operator apply y = Ahat u over the whole mesh:
  N = 1 : BASELINE.json configs[1], 1024 x 1024 elements, p = 8 (67 125 249 DOF);
  N > 1 : BASELINE.json configs[4], 884 x 884 elements per GPU (50 027 329 DOF
          per GPU), strip-partitioned, interface exchange included (weak scaling).
The working set (>= 2.6 GB per GPU) is far larger than the 126 MB L2, so no
cache flush is needed between timed iterations.

One JSON line is printed by rank 0 (see the task contract): value = GDOF/s of
the device-resident apply, e2e = the same apply through the C ABI on pinned
HOST buffers (H2D + apply + D2H per step), roofline = algorithmic bytes /
measured time of the apply kernels vs the measured HBM copy peak,
cpu_baseline = the reference's dense local apply (oracle port) on host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Poisson operator-apply GDOF/s (FP64, p=8)"
ORDER = 8
DUMP_ENTRIES = 4000000          # float64 entries written by --dump-outputs (32 MB) over all ranks


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--nx", type=int, default=0, help="elements per side per GPU (0 = config default)")
    ap.add_argument("--e2e-steps", type=int, default=8)
    ap.add_argument("--e2e-stages", type=int, default=16,
                    help="pipeline stages of the host-buffer apply (1 = copy, apply, copy back)")
    ap.add_argument("--pcg-iters", type=int, default=300,
                    help="PCG iterations timed for the time-to-solution estimate (0 = skip)")
    ap.add_argument("--pcg-full", action="store_true", help="run PCG to rtol 1e-12")
    ap.add_argument("--condensed-full", action="store_true",
                    help="run only the condensed PCG to rtol 1e-12 (time to solution)")
    ap.add_argument("--condensed-multi", action="store_true",
                    help="under torchrun: also time the distributed condensed PCG (capped); "
                         "opt-in, the default multi-GPU line is the apply + uncondensed PCG only")
    ap.add_argument("--two-level", action="store_true",
                    help="also time the two-level preconditioner (seconds at 67 M DOF)")
    ap.add_argument("--no-parity", action="store_true",
                    help="under torchrun: skip the multi-GPU self-check before timing")
    ap.add_argument("--no-tts", action="store_true",
                    help="under torchrun: skip the distributed multilevel time to solution")
    ap.add_argument("--stokes-inner-rtol", type=float, default=1e-8,
                    help="tolerance of the Poisson solves inside the Stokes preconditioner")
    ap.add_argument("--no-condensed", action="store_true",
                    help="skip the statically condensed operator (reported beside the headline)")
    ap.add_argument("--cpu-sample", type=int, default=64,
                    help="elements per side of the CPU-baseline sample mesh (0 = skip)")
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "nccl"],
                    help="multi-GPU interface exchange: fused NVLink peer-memory kernel or NCCL p2p")
    ap.add_argument("--kind", default="S", choices=["S", "C"])
    ap.add_argument("--order", type=int, default=8,
                    help="polynomial order (exploration only: the metric is quoted at p = 8)")
    ap.add_argument("--pe", type=int, default=0, help="elements per patch (0 = automatic)")
    ap.add_argument("--tile", default="", help="patch tile shape bx,by (elements), e.g. 2,8")
    ap.add_argument("--sweep", default="",
                    help="order sweep on the curved mesh (BASELINE configs[2]): comma list of "
                         "orders, e.g. 4,6,8,10,12,16; prints one JSON object and writes "
                         "gpurun_out/r02_sweep.json")
    ap.add_argument("--sweep-tag", default="", help="suffix of the sweep's output file")
    ap.add_argument("--ho-mode", default="", help="apply-kernel variant passed to poisson_operator")
    ap.add_argument("--ablate", type=int, default=0,
                    help="internal profiling knob: extra apply flag bits (results are wrong)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the apply output of the last step to "
                         "DIR/apply_output.npy (float64; a fixed seeded sample of its entries "
                         "when the whole vector exceeds %d entries)" % DUMP_ENTRIES)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "engine" or args.sweep):
        ap.error("--dump-outputs applies to the engine arm's apply only")
    global ORDER, METRIC
    if args.order != ORDER:
        ORDER = args.order
        METRIC = "Poisson operator-apply GDOF/s (FP64, p=%d)" % ORDER
    return args


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def committed_traffic(name, sources):
    """Measured DRAM bytes of one apply from the newest committed ncu capture
    (profiles/rNN_<name>).  ncu cannot run inside a timed bench, so the number is read from
    the capture -- but only while the kernel sources it was taken from are unchanged: the
    file records their SHA-256 and a mismatch yields (None, "stale ...") instead of a
    silently outdated figure."""
    import glob
    import hashlib
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r[0-9][0-9]_" + name)))
    if not files:
        return None, None
    with open(files[-1]) as f:
        tj = json.load(f)
    want = tj.get("source_sha256")
    if want is not None:
        h = hashlib.sha256()
        for src in sources:
            with open(os.path.join(ROOT, "spectralelementmethod_b200", "csrc", src), "rb") as f:
                h.update(f.read())
        if h.hexdigest() != want:
            return None, "stale: %s changed since the capture %s" % (
                "+".join(sources), os.path.basename(files[-1]))
    return tj["dram_bytes_per_apply"], tj["source"]


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self._proc = None
        self._thr = None

    def _reader(self):
        for line in self._proc.stdout:
            cells = [c.strip() for c in line.split(",")]
            if len(cells) >= 9:
                self.rows.append(cells)

    def __enter__(self):
        try:
            self._proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self._thr = threading.Thread(target=self._reader, daemon=True)
            self._thr.start()
            time.sleep(0.15)        # first sample lands before the timed region starts
        except Exception:
            self._proc = None
        return self

    def __exit__(self, *a):
        if self._proc is not None:
            self._proc.terminate()
            try:
                self._proc.wait(timeout=3)
            except Exception:
                self._proc.kill()
            self._thr.join(timeout=3)

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for name, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------
# CPU baseline (the oracle port of the reference's apply), bounded sample
# --------------------------------------------------------------------------
def _cpu_problem(n_side, kind):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import sem_oracle as so
    basis = so.Basis(ORDER)
    nodes, l2g = so.build_case(kind, n_side, n_side, ORDER, False, False)
    geo = so.geometry(basis, nodes, l2g)
    L = so.local_stiffness(basis, geo["invJ"], geo["JxW"])
    u = np.sin(3 * nodes[0]) * np.cos(2 * nodes[1])
    if so.c_lib() is not None:
        so.c_set_threads(os.cpu_count())     # torchrun exports OMP_NUM_THREADS=1 to its workers
        fn = lambda: so.apply_dense_c(L, l2g, u)                 # noqa: E731
        how = ("dense local apply, C/OpenMP restatement (oracle/sem_oracle_c.c), %d threads"
               % so.c_threads())
        cores = so.c_threads()
    else:
        fn = lambda: so.apply_dense_local(L, l2g, u)             # noqa: E731
        how = "dense local einsum loop, single Python thread (oracle/sem_oracle.py)"
        cores = 1
    return fn, nodes.shape[1], how, cores


def cpu_baseline(n_side, kind, target_seconds=10.0):
    """The reference's operator apply on host cores: dense 4-index local
    stiffness (examples/poisson.py:181-193) applied element by element and
    scatter-added (examples/squirmer-axisymmetric.py:284-295) -- the oracle
    port, with every host thread it can use -- on an n_side x n_side, p = 8
    sample of the workload (the dense Lse needs 52 KB per element, so the full
    1024 x 1024 mesh cannot even be stored: 55 GB)."""
    fn, ndof, how, cores = _cpu_problem(n_side, kind)
    fn()
    reps, t0 = 0, time.perf_counter()
    while True:
        fn()
        reps += 1
        el = time.perf_counter() - t0
        if el >= target_seconds or reps >= 100000:
            break
    return {"value": ndof * reps / el / 1e9, "unit": "GDOF/s", "cores": cores, "kind": "port",
            "sample": "%dx%d elements p=%d (%d DOF), %d applies in %.1f s; %s"
                      % (n_side, n_side, ORDER, ndof, reps, el, how)}


def live_reference_baseline(n_side, kind, apply_seconds=3.0):
    """The UNMODIFIED reference (oracle/_ref, an offline `pip install --target` of
    /root/reference made by oracle/install_ref.sh; five compatibility shims, no source
    edits) timed on this host: its own apply -- a Python loop of dense local einsums,
    examples/squirmer-axisymmetric.py:268-295 -- and its whole DOFManagerSC solver pipeline
    (sem/discrete.py:283-528), on a bounded n_side x n_side sample.  None when the
    reference tree did not travel."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import live_reference as lr
        if not lr.available():
            return None
        reps, el, ndof = lr.time_apply(kind, n_side, n_side, ORDER, apply_seconds)
        pipe = lr.time_pipeline(kind, n_side, n_side, ORDER)
    except Exception as exc:             # a reported baseline, never fatal
        return {"error": repr(exc)}
    return {"kind": "reference", "cores": 1,
            "apply_gdof_per_s": ndof * reps / el / 1e9,
            "apply_sample": "%dx%d elements p=%d (%d DOF), %d applies in %.1f s; the reference's "
                            "own Python loop of dense local einsums (single thread)"
                            % (n_side, n_side, ORDER, ndof, reps, el),
            "solve": dict(pipe, sample="%dx%d elements p=%d: DOFManagerSC numbering, "
                                       "FiniteElement + local stiffness per element, Schur "
                                       "assembly, spsolve, back-solve (live reference)"
                                       % (n_side, n_side, ORDER))}


def cpu_solve_baseline(n_side, kind):
    """The reference's whole solver pipeline on the host, once, on the same bounded
    sample: dense local stiffness per element, hierarchical reorder, local Schur
    complements, COO assembly, spsolve and interior back-substitution
    (DOFManagerSC, sem/discrete.py:404-528; oracle port, vectorised NumPy/SciPy --
    the reference itself loops over elements in Python)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import sem_oracle as so
    t0 = time.perf_counter()
    basis = so.Basis(ORDER)
    nodes, l2g = so.build_case(kind, n_side, n_side, ORDER, True, False)
    geo = so.geometry(basis, nodes, l2g)
    L = so.local_stiffness(basis, geo["invJ"], geo["JxW"])
    t1 = time.perf_counter()
    on, vals = so.dirichlet_data(nodes, l2g, geo["x_phys"], so.mesh_boundary_faces(n_side, n_side))
    ext = so.hier_order(ORDER + 1)[:4 * ORDER]
    n_ext = int(np.unique(l2g.reshape(l2g.shape[0], -1)[:, ext]).size)
    so.solve_schur(L, geo["JxW"], l2g, n_ext, on, vals)
    t2 = time.perf_counter()
    return {"seconds": t2 - t0, "operator_seconds": t1 - t0, "solve_seconds": t2 - t1,
            "dof": int(nodes.shape[1]), "kind": "port",
            "sample": "%dx%d elements p=%d: local operators + Schur + spsolve + back-solve "
                      "(DOFManagerSC path), NumPy/SciPy" % (n_side, n_side, ORDER)}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle
    port; the Python reference cannot travel to the GPU box), rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_side = args.cpu_sample or 64
    fn, ndof, how, cores = _cpu_problem(n_side, args.kind)
    for _ in range(max(args.warmup, 1)):
        fn()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fn()
    el = time.perf_counter() - t0
    value = ndof * args.steps / el / 1e9
    sample = ("%dx%d elements p=%d (%d DOF) per step: bounded sample of the 1024x1024 workload; %s"
              % (n_side, n_side, ORDER, ndof, how))
    live = live_reference_baseline(min(n_side, 24), args.kind) if 2 <= ORDER <= 10 else None
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "GDOF/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": el / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        # the engine arm's workload; every step is a bounded sample of it (cpu_baseline.sample)
        "config": {"workload": ("structured 1024x1024-element quad mesh Poisson, p=%d, FP64, "
                                "rcm_order=False (BASELINE configs[1])" % ORDER) if args.gpus <= 1 else
                               ("weak scaling: 884x884 elements p=8 per GPU, strip-partitioned over %d "
                                "GPUs (BASELINE configs[4])" % args.gpus),
                   "order": ORDER, "sample_elements_per_side": n_side},
        "cpu_baseline": {"value": value, "unit": "GDOF/s", "cores": cores, "kind": "port",
                         "sample": sample, "host_cores": os.cpu_count(),
                         "live_reference": live,
                         "note": "value = the C/OpenMP port on every host core (faster than the "
                                 "reference's own Python loop, reported beside it as "
                                 "live_reference): the conservative denominator"},
        "e2e": {"value": value, "unit": "GDOF/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------
# engine arm
# --------------------------------------------------------------------------
def run_condensed(args, nx, dev, peak):
    """The reference's own solver formulation on the device (DOFManagerSC: local Schur
    complements, condensed system over the element-exterior DOFs, interior
    back-substitution; sem/discrete.py:404-528) on the same mesh: condensed apply and
    Jacobi-PCG per iteration, reported beside the matrix-free headline."""
    import torch
    from spectralelementmethod_b200 import discrete, meshgen
    from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS
    t0 = time.perf_counter()
    mesh = meshgen.structured_quad_mesh(nx, nx, ORDER, args.kind)
    b1 = LagrangeGaussLobatto(ORDER)
    mngr = discrete.DOFManagerSC(mesh, 1, TensorProductQS(b1, b1), rcm_order=False)
    on = mngr.boundary_node_mask("ebc")
    t_host = time.perf_counter() - t0
    t0 = time.perf_counter()
    sc = mngr.condensed_poisson_operator(dirichlet=on)
    torch.cuda.synchronize()
    t_setup = time.perf_counter() - t0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    sdiag = torch.empty((sc.n_elem, sc.n_ext_loc), dtype=torch.float64, device=dev)
    sc._element_pass(1, S=sc.S, sdiag_loc=sdiag)          # the Schur pass alone, timed
    ev1.record()
    torch.cuda.synchronize()
    t_schur = ev0.elapsed_time(ev1) / 1e3
    del sdiag
    u = torch.randn(sc.n_ext, dtype=torch.float64, device=dev,
                    generator=torch.Generator(device=dev).manual_seed(0))
    out = torch.empty_like(u)
    for _ in range(5):
        sc.apply(u, out=out)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(args.steps):
        sc.apply(u, out=out)
    ev1.record()
    torch.cuda.synchronize()
    t_apply = ev0.elapsed_time(ev1) / 1e3 / args.steps
    alg = sc.algorithmic_bytes_per_apply
    res = {"formulation": "static condensation (DOFManagerSC), packed local Schur complements",
           "dof_exterior": sc.n_ext, "dof_total": sc.n_nodes, "elements": sc.n_elem,
           "host_numbering_seconds": t_host, "setup_seconds": t_setup,
           "schur_pass_seconds": t_schur,
           "ms_per_apply": t_apply * 1e3, "algorithmic_bytes_per_apply": alg,
           "achieved_GBps": alg / t_apply / 1e9, "frac_of_hbm_peak": alg / t_apply / 1e9 / peak,
           "gdof_total_per_s": sc.n_nodes / t_apply / 1e9,
           "kernel": "sc_matvec_kernel<%d> + sc_node_kernel (one condensed apply)" % (ORDER + 1)}
    # measured DRAM bytes of one condensed apply, from the committed ncu capture of this very
    # configuration; null for any other workload
    res["traffic"] = None
    if sc.n_elem == 1024 * 1024 and ORDER == 8:
        res["traffic"], res["traffic_source"] = committed_traffic("traffic_condensed.json",
                                                                  ["semk_sc.cu"])
    if args.pcg_iters > 0 or args.pcg_full:
        b = sc.lift(sc.rhs(1.0), None)

        def run(iters):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            xs, info = sc.solve_pcg(b, rtol=1e-12, maxiter=iters, check_every=50)
            torch.cuda.synchronize()
            return time.perf_counter() - t0, info, xs
        run(50)
        el0, i0, _ = run(100)
        full = args.pcg_full or args.condensed_full
        el, info, xs = run(200000 if full else 100 + args.pcg_iters)
        ms_it = (el - el0) / max(info.iterations - i0.iterations, 1) * 1e3
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sc.backsolve(xs, 1.0)
        torch.cuda.synchronize()
        res["pcg"] = {"iterations": info.iterations, "seconds": el, "converged": info.converged,
                      "rel_residual": info.rel_residual, "ms_per_iteration": ms_it,
                      "backsolve_seconds": time.perf_counter() - t0,
                      "note": "homogeneous Dirichlet on ebc, f=1, rtol 1e-12"
                              + ("" if full else "; capped")}
    # time to solution with the multilevel preconditioner (Jacobi + vertex coarse space +
    # aggregation level, native driver semk_sc_mlpcg_solve_f64): always runs to rtol 1e-12;
    # never fatal for the line
    for pre in ("three-level",) + (("two-level",) if args.two_level else ()):
        key = pre.replace("-", "_") + "_pcg"
        try:
            b2 = sc.lift(sc.rhs(1.0), None)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            sc._build_coarse()
            torch.cuda.synchronize()
            t_coarse = time.perf_counter() - t0
            t0 = time.perf_counter()
            if pre == "three-level":
                sc._build_top()
            torch.cuda.synchronize()
            t_top = time.perf_counter() - t0
            sc.solve_pcg(b2, rtol=1e-12, maxiter=2, preconditioner=pre)      # warm-up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            x2, info2 = sc.solve_pcg(b2, rtol=1e-12, preconditioner=pre)
            torch.cuda.synchronize()
            t_solve = time.perf_counter() - t0
            refined = None
            if pre == "three-level":
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                x3, info3, cycles = sc.solve_pcg_refined(b2, rtol=1e-12)
                torch.cuda.synchronize()
                refined = {"seconds": time.perf_counter() - t0,
                           "true_rel_residual_per_cycle": [c[0] for c in cycles],
                           "outer_iterations_per_cycle": [c[1] for c in cycles],
                           "note": "the same solve followed by refinement cycles on the true "
                                   "residual until it meets rtol or stops halving"}
                del x3
            t0 = time.perf_counter()
            sc.backsolve(x2, 1.0)
            torch.cuda.synchronize()
            res[key] = {
                "preconditioner": "Jacobi + vertex coarse space"
                                  + (" + vertex aggregation with a dense inverse (inner PCG, rtol "
                                     "1e-2)" if pre == "three-level" else " (inner Jacobi-PCG, rtol 1e-2)")
                                  + ", flexible CG outside",
                "outer_iterations": info2.iterations, "inner_iterations": info2.inner_iterations,
                "seconds": t_solve, "coarse_build_seconds": t_coarse, "top_build_seconds": t_top,
                "backsolve_seconds": time.perf_counter() - t0, "converged": info2.converged,
                "rel_residual": info2.rel_residual,
                "true_rel_residual": info2.true_rel_residual,
                "refined": refined,
                "note": "homogeneous Dirichlet on ebc, f=1, rtol 1e-12 (time to solution); "
                        "rel_residual is the recursive one, true_rel_residual = ||b - S x|| / ||b|| "
                        "recomputed from the returned iterate"}
        except Exception as exc:
            res[key] = {"error": repr(exc)}
    return res


SWEEP_NX = {2: 2048, 3: 1536, 4: 1024, 5: 1024, 6: 1024, 7: 1024, 8: 1024, 9: 896, 10: 768,
            11: 704, 12: 640, 13: 576, 14: 576, 15: 512, 16: 512}


def run_stokes(args, peak):
    """BASELINE configs[3]: the axisymmetric Stokes system of examples/squirmer-axisymmetric.py
    (2 DOF per node, Jacobian [[0, Lve], [E2e, -Me]] at Re = 0 and with the advection blocks
    at Re = 1) on a graded annulus-sector mesh scaled to ~1e7 DOF: matrix-free apply
    throughput and its HBM roofline.  (The non-symmetric solve is GMRES with a nodal
    block-Jacobi preconditioner: parity-tested on small meshes, not mesh-independent.)"""
    import numpy as np
    import torch
    from spectralelementmethod_b200 import discrete, meshgen
    from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS
    nr, nt, p = 224, 352, 8
    t0 = time.perf_counter()
    mesh = meshgen.annulus_sector_mesh(nr, nt, p, 100.0)
    b1 = LagrangeGaussLobatto(p)
    dm = discrete.DOFManager(mesh, 2, TensorProductQS(b1, b1), rcm_order=False)
    out = {"workload": "annulus sector r in [1, 100], %dx%d elements p=%d, stream function + "
                       "vorticity (BASELINE configs[3])" % (nr, nt, p)}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for n_rey in (0.0, 1.0):
        op = dm.axisymmetric_stokes_operator(n_rey=n_rey)
        torch.cuda.synchronize()
        setup = time.perf_counter() - t0
        x = torch.from_numpy(np.sin(np.arange(op.n_dof) * 1e-3)).cuda()
        if op.advection:
            op.linearize(x)
        y = op.new_vector()
        for _ in range(5):
            op.apply_unmasked(x, out=y)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(args.steps):
            op.apply_unmasked(x, out=y)
        ev1.record()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / args.steps
        alg = op.algorithmic_bytes_per_apply
        out["re_%g" % n_rey] = {
            "dof": op.n_dof, "n_factors": op.n_fac, "elems_per_patch": op.elems_per_patch,
            "smem_bytes_per_cta": op.smem_bytes, "setup_seconds": setup, "ms_per_apply": ms,
            "gdof_per_s": op.n_dof / ms / 1e6, "algorithmic_bytes": alg,
            "achieved_GBps": alg / ms / 1e6, "frac_of_hbm_peak": alg / ms / 1e6 / peak,
            "kernel": "stokes_patch_kernel<9,%d,%s> + stokes_shared_nodes_kernel"
                      % (op.elems_per_patch, "ADV" if op.advection else "STOKES")}
        del op, x, y
        t0 = time.perf_counter()
    # CPU baseline of this row (reported beside, not the target): the reference's own dense
    # local apply of the Stokes blocks -- np.einsum('pqrs,rs', Lve, vort), np.einsum('pqrs,rs',
    # E2e, sfn) and the diagonal mass term, examples/squirmer-axisymmetric.py:284-295 -- over
    # precomputed dense operators (oracle restatement, vectorised over elements, one thread)
    if args.cpu_sample > 0:
        try:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import sem_oracle as so
            snr, snt = 12, 16
            nodes = so.annulus_nodes(snr, snt, p, 100.0)
            l2g = so.mesh_l2g(snr, snt, p)
            basis = so.Basis(p)
            geo = so.geometry(basis, nodes, l2g)
            ops = so.stokes_local_operators(basis, geo["x_phys"], geo["invJ"], geo["JxW"])
            Lv = np.where(np.isfinite(ops["Lve"]), ops["Lve"], 0.0)
            E2, Me = ops["E2e"], ops["Me"]
            rng = np.random.default_rng(0)
            sf, vo = rng.standard_normal((2, nodes.shape[1]))
            n_dof_s = 2 * nodes.shape[1]
            reps, t0c = 0, time.perf_counter()
            while time.perf_counter() - t0c < 5.0:
                r0 = np.einsum("epqrs,ers->epq", Lv, vo[l2g])
                r1 = np.einsum("epqrs,ers->epq", E2, sf[l2g]) - Me * vo[l2g]
                y = np.zeros(n_dof_s)
                np.add.at(y[0::2], l2g.ravel(), r0.ravel())
                np.add.at(y[1::2], l2g.ravel(), r1.ravel())
                reps += 1
            el = time.perf_counter() - t0c
            out["cpu_baseline"] = {
                "value": n_dof_s * reps / el / 1e9, "unit": "GDOF/s", "cores": 1, "kind": "port",
                "sample": "%dx%d elements p=%d (%d DOF), %d applies in %.1f s; dense local "
                          "einsum apply of Lve / E2e / Me (oracle restatement of "
                          "examples/squirmer-axisymmetric.py:284-295), NumPy, one thread"
                          % (snr, snt, p, n_dof_s, reps, el)}
        except Exception as exc:       # a reported baseline, never fatal
            out["cpu_baseline"] = {"error": repr(exc)}

    # time to solution of the Stokes problem (Re = 0, squirmer boundary data) at the same
    # size: flexible GMRES, block-triangular preconditioner from the weighted condensed
    # Poisson operator (multilevel PCG inside), accepted on the TRUE residual
    from spectralelementmethod_b200 import stokes
    t0 = time.perf_counter()
    mesh = meshgen.annulus_sector_mesh(nr, nt, p, 100.0)
    dm = discrete.DOFManagerSC(mesh, 2, TensorProductQS(b1, b1), rcm_order=False)
    op = dm.axisymmetric_stokes_operator(n_rey=0.0)
    bc = stokes.squirmer_boundary_data(
        dm, 1.0, stokes.squirmer_vslip_profile(1.0),
        x_phys=op.x_phys.cpu().numpy().reshape(op.n_elem, 2, p + 1, p + 1))
    op.set_essential(bc.essential)
    rhs = op.from_host(bc.cint) - op.residual(op.from_host(bc.state0))
    prec = op._poisson_prec = stokes.PoissonBlockPreconditioner(op, rtol=args.stokes_inner_rtol)
    prec.poisson_solve(torch.zeros(op.n_nodes, dtype=torch.float64, device=op.dev))  # builds the levels
    torch.cuda.synchronize()
    setup = time.perf_counter() - t0
    prec.solves = prec.inner_outer_iterations = 0
    t0 = time.perf_counter()
    d, info = op.solve_gmres(rhs, rtol=1e-8, restart=300, maxiter=900, precondition="poisson")
    torch.cuda.synchronize()
    out["time_to_solution"] = {
        "seconds": time.perf_counter() - t0, "setup_seconds": setup, "dof": op.n_dof,
        "rtol": 1e-8, "gmres_iterations": info.iterations, "cycles": info.restarts,
        "converged": info.converged, "true_rel_residual": info.true_rel_residual,
        "poisson_solves": prec.solves, "poisson_pcg_outer_iterations": prec.inner_outer_iterations,
        "inner_rtol": args.stokes_inner_rtol,
        "method": "flexible GMRES on the matrix-free Jacobian [[0, Lve], [E2e, -Me]], right "
                  "preconditioner: om_G = -b_G/M_G, om_I = K^-1(a - L om_G), psi = K^-1(b + M om_I) "
                  "with K = Lve on the interior nodes (rho-weighted stiffness + JxW/rho), statically condensed, solved by the "
                  "three-level PCG driver; convergence accepted on the true residual"}
    return out


def sweep_bytes_per_dof(p):
    """SURVEY 8(d): B(p) = 16 + 28 ((p+1)/p)^2 algorithmic bytes per global DOF per apply."""
    return 16.0 + 28.0 * ((p + 1.0) / p) ** 2


def run_sweep(args):
    """BASELINE configs[2]: the apply at orders p = 4..16 on the curved (mapped) mesh, one
    GPU; per order the mesh size keeps ~50-70 M DOF.  One JSON object with a row per order."""
    import numpy as np
    import torch
    from spectralelementmethod_b200 import discrete, meshgen
    from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    peak, peak_kind = measured_peaks()
    rows = []
    for p in [int(v) for v in args.sweep.split(",") if v]:
        nx = args.nx or SWEEP_NX[p]
        mesh = meshgen.structured_quad_mesh(nx, nx, p, "C")
        b1 = LagrangeGaussLobatto(p)
        mngr = discrete.DOFManager(mesh, 1, TensorProductQS(b1, b1), rcm_order=False)
        on_ebc = mngr.boundary_node_mask("ebc")
        kw = {}
        if args.ho_mode:
            kw["mode"] = args.ho_mode
        op = mngr.poisson_operator(dirichlet=on_ebc, elems_per_patch=args.pe or None, **kw)
        x, y = mesh.nodes
        u = torch.from_numpy(np.sin(3 * x) * np.cos(2 * y)).to(dev)
        out = torch.empty_like(u)
        for _ in range(max(args.warmup, 3)):
            op.apply(u, out=out)
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(args.steps):
            op.apply(u, out=out)
        ev1.record()
        torch.cuda.synchronize()
        t = ev0.elapsed_time(ev1) / 1e3 / args.steps
        alg = op.algorithmic_bytes_per_apply
        rows.append({"order": p, "elements": "%dx%d" % (nx, nx), "dof": int(op.n_nodes),
                     "kernel": getattr(op, "kernel_name", None),
                     "elems_per_patch": op.elems_per_patch,
                     "resident_ctas": getattr(op, "resident_ctas", None),
                     "smem_bytes_per_cta": getattr(op, "smem_bytes", None),
                     "ms_per_apply": t * 1e3, "gdof_per_s": op.n_nodes / t / 1e9,
                     "algorithmic_bytes": alg, "achieved_GBps": alg / t / 1e9,
                     "frac_of_hbm_peak": alg / t / 1e9 / peak,
                     "checksum": float(out.double().sum())})
        print("sweep p=%d: %.3f ms, %.1f GDOF/s, %.1f %% of peak" %
              (p, t * 1e3, op.n_nodes / t / 1e9, 100 * alg / t / 1e9 / peak), file=sys.stderr,
              flush=True)
        del op, mngr, mesh, u, out
        torch.cuda.empty_cache()
    res = {"sweep": "Poisson apply, curved mesh (kind C), FP64, one B200", "steps": args.steps,
           "peak_GBps": peak, "peak_source": peak_kind, "rows": rows}
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    with open(os.path.join(ROOT, "gpurun_out", "r02_sweep%s.json" % args.sweep_tag), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res), flush=True)


def dump_output(out_dir, name, y, n_keep):
    """Writes the device vector y to out_dir/name.npy as float64: whole when it has at most
    n_keep entries, else the entries at sorted indices drawn with a fixed seed from its length
    alone, so that two builds run with the same arguments can be compared entry for entry."""
    import numpy as np
    import torch
    if y.numel() > n_keep:
        idx = np.unique(np.random.default_rng(0).integers(0, y.numel(), size=n_keep))
        y = y[torch.from_numpy(idx).to(y.device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), y.to(torch.float64).cpu().numpy())


def run_engine(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from spectralelementmethod_b200 import discrete, meshgen
    from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    multi = world > 1
    if multi:
        dist.init_process_group("nccl", device_id=dev)

    parity = None
    if multi and not args.no_parity:
        # driver-visible parity of the partitioned path: a small global problem per rank,
        # distributed apply / dot / PCG / condensed / multilevel against the single-GPU
        # operator, peer == NCCL bitwise; raises (and fails the run) on any mismatch
        from spectralelementmethod_b200 import distributed_check
        t0 = time.perf_counter()
        parity = distributed_check.run(rank, world, dev)
        torch.cuda.synchronize()
        dist.barrier()
        parity["seconds"] = time.perf_counter() - t0

    t_setup = time.perf_counter()
    if not multi:
        nx = args.nx or 1024
        mesh = meshgen.structured_quad_mesh(nx, nx, ORDER, args.kind)
        b1 = LagrangeGaussLobatto(ORDER)
        mngr = discrete.DOFManager(mesh, 1, TensorProductQS(b1, b1), rcm_order=False)
        on_ebc = mngr.boundary_node_mask("ebc")
        tile = tuple(int(v) for v in args.tile.split(",")) if args.tile else None
        op = mngr.poisson_operator(dirichlet=on_ebc, elems_per_patch=args.pe or None, tile=tile)
        if args.ablate:
            abl = op._masked_flags | args.ablate
            apply_fn = lambda u, out: op.apply(u, out=out, flags=abl)   # noqa: E731
        else:
            apply_fn = lambda u, out: op.apply(u, out=out)          # noqa: E731
        n_local = n_global = op.n_nodes
        n_global_units = n_global
        workload = ("structured %dx%d-element quad mesh Poisson, p=%d, FP64, rcm_order=False "
                    "(BASELINE configs[1])" % (nx, nx, ORDER))
        dp = None
    else:
        from spectralelementmethod_b200.distributed import DistributedPoisson, StripPartition
        nx = args.nx or 884
        part = StripPartition(rank, world, nx, nx, ORDER, bounds=(-1.0, -1.0 + 2.0 * world, -1.0, 1.0))
        dp = DistributedPoisson(part, ORDER, args.kind, elems_per_patch=args.pe or None,
                                exchange=args.exchange)
        op = dp.op
        apply_fn = lambda u, out: dp.apply(u, out=out)          # noqa: E731
        n_local = op.n_nodes
        n_global_units = part.n_global
        workload = ("weak scaling: %dx%d elements p=8 per GPU, strip-partitioned over %d GPUs, "
                    "%s interface exchange (BASELINE configs[4])"
                    % (nx, nx, world, "NVLink peer-memory" if dp.exchange == "peer" else "NCCL p2p"))
    torch.cuda.synchronize()
    t_setup = time.perf_counter() - t_setup

    x, y = op.dof_mngr.mesh.nodes
    u = torch.from_numpy(np.sin(3 * x) * np.cos(2 * y)).to(dev)
    out = torch.empty_like(u)

    def barrier():
        if multi:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident apply: W warm-ups, K timed steps ----------------------
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:      # samples clocks from the warm-up onwards
        for _ in range(max(args.warmup, 3)):
            apply_fn(u, out)
        barrier()
        ev0.record()
        for _ in range(args.steps):
            apply_fn(u, out)
        ev1.record()
        barrier()
        elapsed = ev0.elapsed_time(ev1) / 1e3
    if args.dump_outputs:
        # the caller of the timed apply receives `out`; under torchrun each rank its own part
        dump_output(args.dump_outputs, "apply_output" + ("_rank%d" % rank if multi else ""), out,
                    DUMP_ENTRIES // world)
    if multi:
        t = torch.tensor([elapsed], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed = float(t)
    ms_per_step = elapsed / args.steps * 1e3
    value = n_global_units / (elapsed / args.steps) / 1e9

    # ---- roofline of the apply kernels (local operator only, rank 0's GPU) -------
    for _ in range(3):
        op.apply(u, out=out)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(args.steps):
        op.apply(u, out=out)
    ev1.record()
    torch.cuda.synchronize()
    t_kernel = ev0.elapsed_time(ev1) / 1e3 / args.steps
    peak, peak_kind = measured_peaks()
    alg_bytes = op.algorithmic_bytes_per_apply
    achieved = alg_bytes / t_kernel / 1e9
    # measured DRAM bytes of one apply: from the committed ncu capture of this very
    # configuration (profiles/r01_traffic.json); null for any other workload
    traffic, traffic_src = None, None
    if (not multi and op.n_elem == 1024 * 1024 and op.elems_per_patch == 16 and not args.tile
            and args.kind == "S"):
        traffic, traffic_src = committed_traffic(
            "traffic.json", ["semk_apply.cu", "semk_patch.cuh", "semk_box.cu", "semk_elem.cuh"])
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peak_kind,
                "kernel": "%s + shared_nodes_kernel (one apply)" % op.kernel_name,
                "algorithmic_bytes_per_launch": alg_bytes,
                "ms_per_launch": t_kernel * 1e3}

    # ---- e2e: host buffers through the C ABI (H2D + apply + D2H per step) ---------
    u_host = torch.empty(n_local, dtype=torch.float64).pin_memory()
    y_host = torch.empty(n_local, dtype=torch.float64).pin_memory()
    u_host.copy_(u)
    scratch = (op.new_vector(), op.new_vector())

    def e2e_step():
        if dp is None:
            op.apply_host(u_host, y_host, scratch, stages=args.e2e_stages)
        else:
            # per rank the staged pipeline of the local apply, then the interface exchange on
            # the device and a second download of the two exchanged columns
            dp.apply_host(u_host, y_host, scratch, stages=args.e2e_stages)
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        e2e_step()
    barrier()
    e2e_el = time.perf_counter() - t0
    if multi:
        t = torch.tensor([e2e_el], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_el = float(t)
    e2e_value = n_global_units / (e2e_el / args.e2e_steps) / 1e9
    e2e_single = None
    if dp is None and args.e2e_steps > 1:
        # one GPU: the same steps as ONE batched call (semk_poisson_apply_host_batch_f64): every
        # step still uploads its own input and downloads its own result inside the timed
        # region, but the upload of step k+1 overlaps the download of step k (two scratch
        # sets), so the full-duplex link is busy both ways for the whole batch.  The
        # call-per-step number above is kept beside it as `single_call_value`.
        u_host2 = torch.empty(n_local, dtype=torch.float64).pin_memory()
        y_host2 = torch.empty(n_local, dtype=torch.float64).pin_memory()
        u_host2.copy_(u_host)
        ups = [u_host if k % 2 == 0 else u_host2 for k in range(args.e2e_steps)]
        downs = [y_host if k % 2 == 0 else y_host2 for k in range(args.e2e_steps)]
        scratch4 = scratch + (op.new_vector(), op.new_vector())
        op.apply_host_many(ups[:2], downs[:2], scratch4, stages=args.e2e_stages)
        y_host2.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        op.apply_host_many(ups, downs, scratch4, stages=args.e2e_stages)
        e2e_batch_el = time.perf_counter() - t0
        if not torch.equal(y_host2, y_host):
            raise AssertionError("batched host apply: results of consecutive steps differ")
        e2e_single = e2e_value
        e2e_value = n_global_units / (e2e_batch_el / args.e2e_steps) / 1e9
        del u_host2, y_host2, scratch4
    if dp is None:
        e2e_ok = bool(torch.equal(y_host.to(dev), out))
    else:
        # the host-buffer step must reproduce the device-resident distributed apply bit for
        # bit on every rank (same kernels, same two-term interface sums)
        # reference: the device-resident distributed apply through the same local operator
        # (bitwise), and the overlapped production apply (its corner sums associate in the
        # boundary-columns-first patch order: equal to rounding)
        y_dev = dp.dop.finish(dp.host_operator().apply(u), u)
        dp.apply(u, out=out)
        same = torch.equal(y_host.to(dev), y_dev)
        close = float((y_dev - out).abs().max()) <= 1e-12 * float(out.abs().max())
        ok = torch.tensor([1.0 if (same and close) else 0.0], device=dev)
        del y_dev
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        e2e_ok = bool(float(ok) >= 1.0)
        if not e2e_ok:
            raise AssertionError("multi-GPU e2e result differs from the device-resident apply")
    if dp is not None and dp.halo is not None:
        dp.halo.check()         # a neighbour that never delivered a column would have raised a flag

    # ---- PCG time-to-solution (reported beside the headline) -----------------------
    pcg = None
    if args.pcg_iters > 0 or args.pcg_full:
        maxiter = 200000 if args.pcg_full else args.pcg_iters
        if dp is None:
            b = op.lift(op.rhs(1.0), None)

            def run(iters):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                xs, info = op.solve_pcg(b, rtol=1e-12, maxiter=iters, check_every=50)
                torch.cuda.synchronize()
                return time.perf_counter() - t0, info.iterations, info.rel_residual, info.converged
        else:
            b = dp.lift(dp.rhs(1.0), None)

            def run(iters):
                barrier()
                t0 = time.perf_counter()
                xs, it, rel, ok = dp.solve_pcg(b, rtol=1e-12, maxiter=iters, check_every=50)
                barrier()
                return time.perf_counter() - t0, it, rel, ok
        # ms/iteration from the slope between two capped solves: the fixed cost of a solve
        # (Jacobi diagonal on first use, work vectors, CUDA-graph capture) cancels
        run(50)
        base_iters = 100
        el0, it0, _, _ = run(base_iters)
        el, it, rel, ok = run(maxiter if args.pcg_full else base_iters + maxiter)
        pcg = {"iterations": it, "seconds": el, "converged": ok, "rel_residual": rel,
               "ms_per_iteration": (el - el0) / max(it - it0, 1) * 1e3,
               "fixed_seconds_per_solve": max(el0 - it0 * (el - el0) / max(it - it0, 1), 0.0)}
        pcg["note"] = ("homogeneous Dirichlet on ebc, f=1, rtol 1e-12"
                       + ("" if args.pcg_full else "; capped at %d iterations" % pcg["iterations"]))

    condensed = None
    if not multi and not args.no_condensed and 2 <= ORDER <= 10:
        try:
            condensed = run_condensed(args, nx, dev, peak)
        except Exception as exc:       # reported, never fatal for the headline line
            condensed = {"error": repr(exc)}
    if multi and (args.condensed_full or args.condensed_multi) and 2 <= ORDER <= 10:
        # distributed PCG on the condensed system (every rank must take the same path: the
        # constructor and the solves are collective, so no try/except here)
        from spectralelementmethod_b200.distributed import DistributedCondensedPoisson
        dc = DistributedCondensedPoisson(part, ORDER, args.kind, exchange=args.exchange)
        bc = dc.lift(dc.rhs(1.0), None)

        def run_c(iters):
            barrier()
            t0 = time.perf_counter()
            xs, it, rel, ok = dc.solve_pcg(bc, rtol=1e-12, maxiter=iters, check_every=50)
            barrier()
            return time.perf_counter() - t0, it, rel, ok
        run_c(50)
        el0, it0, _, _ = run_c(100)
        full_c = args.pcg_full or args.condensed_full
        el, it, rel, ok = run_c(200000 if full_c else 100 + args.pcg_iters)
        condensed = {"formulation": "static condensation, strip-partitioned, distributed PCG on "
                                    "the exterior DOFs (%s exchange)" % dc.exchange,
                     "dof_exterior_per_gpu": dc.sc.n_ext,
                     "pcg": {"iterations": it, "seconds": el, "converged": ok, "rel_residual": rel,
                             "ms_per_iteration": (el - el0) / max(it - it0, 1) * 1e3,
                             "note": "homogeneous Dirichlet on ebc, f=1, rtol 1e-12"
                                     + ("" if full_c else "; capped")}}
        if dc.halo is not None:
            dc.halo.check()

    stokes_blk = None
    if not multi and not args.no_condensed:
        try:
            stokes_blk = run_stokes(args, peak)
        except Exception as exc:       # reported, never fatal for the headline line
            stokes_blk = {"error": repr(exc)}

    # the metric's second half, PCG time to solution (rtol 1e-12), by the fastest device path:
    # static condensation + multilevel-preconditioned flexible CG + interior back-solve
    tts = None
    method = ("static condensation + three-level PCG (Jacobi + vertex coarse space + vertex "
              "aggregation with a dense inverse; native driver semk_sc_mlpcg_solve_f64) + interior "
              "back-solve; operator set-up reported separately")
    if not multi:
        tl = (condensed or {}).get("three_level_pcg") or {}
        if tl.get("converged"):
            setup_s = (condensed.get("host_numbering_seconds", 0.0) + condensed.get("setup_seconds", 0.0)
                       + tl.get("coarse_build_seconds", 0.0) + tl.get("top_build_seconds", 0.0))
            tts = {"seconds": tl["seconds"] + tl["backsolve_seconds"], "rtol": 1e-12,
                   "dof": int(n_global_units), "outer_iterations": tl["outer_iterations"],
                   "inner_iterations": tl["inner_iterations"],
                   "rel_residual": tl["rel_residual"],
                   "true_rel_residual": tl["true_rel_residual"], "method": method,
                   "setup_seconds": setup_s,
                   "including_setup_seconds": setup_s + tl["seconds"] + tl["backsolve_seconds"]}
    elif not args.no_tts and 2 <= ORDER <= 10:
        # every rank takes the same path: constructor and solves are collective
        from spectralelementmethod_b200.distributed import DistributedCondensedPoisson
        del u, out
        torch.cuda.empty_cache()
        barrier()
        t0 = time.perf_counter()
        dcm = DistributedCondensedPoisson(part, ORDER, args.kind, exchange=args.exchange)
        bcm = dcm.lift(dcm.rhs(1.0), None)
        barrier()
        t_op = time.perf_counter() - t0
        t0 = time.perf_counter()
        ml = dcm._multilevel(3)
        barrier()
        t_ml = time.perf_counter() - t0
        dcm.solve_pcg(bcm, rtol=1e-12, maxiter=2, preconditioner="three-level")     # warm-up
        barrier()
        t0 = time.perf_counter()
        xs, it, rel, ok = dcm.solve_pcg(bcm, rtol=1e-12, preconditioner="three-level")
        torch.cuda.synchronize()
        t_solve = time.perf_counter() - t0
        us = dcm.sc.backsolve(xs, 1.0)
        barrier()
        t_total = time.perf_counter() - t0
        tt = torch.tensor([t_total, t_solve], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        inf = dcm.last_info
        chk = torch.tensor([float(us.sum())], dtype=torch.float64, device=dev)
        tts = {"seconds": float(tt[0]), "solve_seconds": float(tt[1]), "rtol": 1e-12,
               "dof": int(n_global_units), "converged": bool(ok), "outer_iterations": int(it),
               "inner_iterations": int(inf.inner_iterations), "rel_residual": float(rel),
               "true_rel_residual": float(inf.true_rel_residual),
               "aggregates": int(ml.get("aggregate_tile", 0)) and
               "%d x %d element tiles" % (ml["aggregate_tile"], ml["aggregate_tile"]),
               "method": method + "; strip partition, halo exchanges and all-reduces are "
                                  "peer-memory kernels issued by the driver",
               "setup_seconds": t_op + t_ml, "operator_setup_seconds": t_op,
               "multilevel_setup_seconds": t_ml,
               "including_setup_seconds": t_op + t_ml + float(tt[0]),
               "rank0_solution_checksum": float(chk)}
        if not ok:
            raise AssertionError("distributed multilevel PCG did not converge: %r" % (tts,))
        dcm.close()

    cpu = None
    if rank == 0 and not multi and args.cpu_sample > 0:
        cpu = cpu_baseline(args.cpu_sample, args.kind)
        if 2 <= ORDER <= 10:
            try:
                cpu["solve"] = cpu_solve_baseline(args.cpu_sample, args.kind)
            except Exception as exc:     # a reported baseline, never fatal
                cpu["solve"] = {"error": repr(exc)}
            cpu["live_reference"] = live_reference_baseline(min(args.cpu_sample, 24), args.kind)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "GDOF/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": workload, "order": ORDER, "dof_total": int(n_global_units),
                       "dof_per_gpu": int(n_local), "elements_per_gpu": int(op.n_elem),
                       "elems_per_patch": op.elems_per_patch, "kind": args.kind,
                       "resident_ctas": getattr(op, "resident_ctas", None),
                       "grid_cap": getattr(op, "max_ctas", 0) or None,
                       "smem_bytes_per_cta": getattr(op, "smem_bytes", None),
                       "l2_policy": "inputs (>= 2.6 GB per GPU) exceed the 126 MB L2; no flush",
                       "setup_seconds": t_setup},
            "roofline": roofline,
            "e2e": {"value": e2e_value, "unit": "GDOF/s", "h2d_bytes_per_step": 8 * n_local * world,
                    "d2h_bytes_per_step": 8 * n_local * world, "steps": args.e2e_steps,
                    "pipeline_stages": args.e2e_stages,
                    "call": ("apply_host_many: %d steps in one semk_poisson_apply_host_batch_f64 call, "
                             "upload of step k+1 overlapping the download of step k"
                             % args.e2e_steps) if e2e_single is not None else
                            ("one synchronous host-buffer call per step" if dp is None else
                             "DistributedPoisson.apply_host per rank and step: staged local apply, "
                             "device-side interface exchange, exchanged columns downloaded again"),
                    "single_call_value": e2e_single,
                    "matches_device_result": e2e_ok},
            # own kernels per apply: patch kernel + interface kernel (+ the fused exchange kernel)
            "gpu_launches": (3 if (dp is not None and dp.halo is not None) else 2) * args.steps,
            "clocks": clocks.summary(),
            "pcg": pcg,
            "condensed": condensed,
            "stokes": stokes_blk,
            "time_to_solution": tts,
            "parity": parity,
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    if multi:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.sweep:
        run_sweep(args)
    else:
        run_engine(args)


if __name__ == "__main__":
    main()
