#!/usr/bin/env python
"""Outputs of the condensed single-load paths, for a bitwise comparison of two builds.

For p = 2..10 on a 3 x 2 element mesh (Dirichlet on "ebc"), with the storage modes none / W /
W + A_ii^-1 and scalar, CUDA and host loads: ``rhs``, ``backsolve`` with a cache hit and with
a cache miss, ``solve``, ``solve_load``, ``solve_many``; the same on one operator with a weight,
a reaction term and Robin data; and calls of ``semk_sc_element_react_f64`` that combine the
factorisation and load bits (one with a permuted ``slot_of_elem``).  Everything is written to
one ``.npz``; ``--compare A B`` checks two such files for exact equality of every bit.

    python tools/condensed_single_dump.py --root TREE --out FILE.npz
    python tools/condensed_single_dump.py --compare A.npz B.npz [--json OUT]
"""
import argparse
import json
import os
import sys

import numpy as np


def operator(p, store, extra=False):
    from spectralelementmethod_b200 import discrete, meshgen
    from spectralelementmethod_b200.basis_functions import LagrangeGaussLobatto, TensorProductQS
    b1 = LagrangeGaussLobatto(p)
    mngr = discrete.DOFManagerSC(meshgen.structured_quad_mesh(3, 2, p, "C"), 1,
                                 TensorProductQS(b1, b1), rcm_order=True)
    kw = dict(store_interior=store != "none", store_interior_inverse=store == "inverse")
    if extra:
        NN = (p + 1) ** 2
        react = np.random.default_rng(5).uniform(0.1, 1.0, (6, NN))
        kw.update(weight=lambda x, y: 1.0 + 0.5 * x * x, reaction=react, robin={"nbc": 2.0})
    return mngr, mngr.condensed_poisson_operator(dirichlet=mngr.boundary_node_mask("ebc"), **kw)


def loads(sc, seed):
    import torch
    rng = np.random.default_rng(seed)
    return {"scalar": 1.5, "cuda": torch.from_numpy(rng.standard_normal(sc.n_nodes)).cuda(),
            "host": rng.standard_normal(sc.n_nodes)}


def dump_operator(out, tag, mngr, sc, seed):
    import torch
    rng = np.random.default_rng(100 + seed)
    host = lambda t: t.detach().cpu().numpy().copy()   # noqa: E731
    x = torch.from_numpy(rng.standard_normal(sc.n_ext)).cuda()
    vals = np.where(mngr.boundary_node_mask("ebc"), 0.25, 0.0)
    F = loads(sc, seed)
    for name, f in F.items():
        out[f"{tag}/{name}/rhs"] = host(sc.rhs(f))
        out[f"{tag}/{name}/backsolve_hit"] = host(sc.backsolve(x, f))
        sc.rhs(-7.25)                                   # the cache now holds another load
        out[f"{tag}/{name}/backsolve_miss"] = host(sc.backsolve(x, f))
        u, info = sc.solve(f, vals, rtol=1e-10)
        out[f"{tag}/{name}/solve"] = host(u)
        out[f"{tag}/{name}/solve_its"] = np.array(info.iterations)
    r = torch.from_numpy(rng.standard_normal(sc.n_nodes)).cuda()
    if sc.has_dirichlet:
        r[torch.from_numpy(np.flatnonzero(mngr.boundary_node_mask("ebc"))).cuda()] = 0.0
    u, info = sc.solve_load(r, F["cuda"], rtol=1e-8)
    out[f"{tag}/solve_load"] = host(u)
    U, infos = sc.solve_many(list(F.values()), vals, rtol=1e-10)
    out[f"{tag}/solve_many"] = host(U)


def dump_abi(out, tag, sc, seed):
    """semk_sc_element_react_f64 with combined factorisation / load bits."""
    import torch
    from spectralelementmethod_b200 import _lib, device
    f64 = dict(dtype=torch.float64, device=sc.dev)
    E, NE, NI = sc.n_elem, sc.n_ext_loc, sc.n_int_loc
    rng = np.random.default_rng(200 + seed)
    f = torch.from_numpy(rng.standard_normal(sc.n_nodes)).cuda()
    x = torch.from_numpy(rng.standard_normal(sc.n_nodes)).cuda()
    perm = rng.permutation(E)
    slot = torch.from_numpy(perm.astype(np.int64)).cuda()
    Gp = torch.empty_like(sc.G)
    Gp[slot] = sc.G

    def call(mode, G=sc.G, slot_of_elem=None, S=False, W=False, g=False, u=False, c=False):
        res = {"S": torch.zeros((E, sc.s_stride), **f64) if S else None,
               "sdiag": torch.zeros((E, NE), **f64) if S else None,
               "W": torch.zeros((E, NE, NI), **f64) if W else None,
               "g": torch.zeros((E, NE), **f64) if g else None,
               "u": x.clone() if u else None,
               "c": torch.zeros((E, NI), **f64) if c else None}
        bad = torch.zeros(1, dtype=torch.int32, device=sc.dev)
        _lib.check(sc._lib.semk_sc_element_react_f64(
            sc.n1, E, device.ptr(slot_of_elem), device.ptr(G), sc.g_stride, 1,
            device.ptr(sc.tab.dev()[0]), device.ptr(sc._t["ext_loc"]), device.ptr(sc.l2g_dev),
            device.ptr(sc.JxW), device.ptr(f), 0.75, int(mode), device.ptr(res["S"]),
            sc.s_stride, device.ptr(res["sdiag"]), device.ptr(res["g"]), device.ptr(res["u"]),
            device.ptr(res["W"]), device.ptr(res["c"]), device.ptr(sc._react), None,
            device.ptr(bad), device.stream_ptr()))
        assert int(bad.item()) == 0
        return {k: v.cpu().numpy().copy() for k, v in res.items() if v is not None}

    SCHUR, STORE, RHS, BACK = _lib.SC_SCHUR, _lib.SC_STORE, _lib.SC_RHS, _lib.SC_BACKSOLVE
    runs = {"schur_store_rhs_c": call(SCHUR | STORE | RHS, S=True, W=True, g=True, c=True),
            "rhs_backsolve": call(RHS | BACK, g=True, u=True),
            "backsolve_c_slot": call(BACK, G=Gp, slot_of_elem=slot, u=True, c=True),
            "rhs_c": call(RHS, g=True, c=True)}
    for run, res in runs.items():
        for k, v in res.items():
            out[f"{tag}/abi/{run}/{k}"] = v


def dump(root, path):
    sys.path.insert(0, root)
    import torch
    torch.cuda.set_device(0)
    out = {}
    for p in range(2, 11):
        for store in ("none", "stored", "inverse"):
            mngr, sc = operator(p, store)
            dump_operator(out, f"p{p}/{store}", mngr, sc, p)
            if store == "stored":
                dump_abi(out, f"p{p}", sc, p)
    mngr, sc = operator(5, "stored", extra=True)
    dump_operator(out, "p5/weighted_reaction_robin", mngr, sc, 55)
    dump_abi(out, "p5/weighted_reaction_robin", sc, 55)
    np.savez(path, **out)
    print("wrote %d arrays to %s" % (len(out), path))


def compare(a, b, json_out=None):
    A, B = np.load(a), np.load(b)
    keys = sorted(set(A.files) | set(B.files))
    missing = [k for k in keys if k not in A.files or k not in B.files]
    differ = []
    for k in keys:
        if k in missing:
            continue
        x, y = A[k], B[k]
        if x.shape != y.shape or x.dtype != y.dtype or x.tobytes() != y.tobytes():
            differ.append(k)
    res = {"files": [os.path.basename(a), os.path.basename(b)], "arrays": len(keys),
           "bitwise_equal": len(keys) - len(missing) - len(differ), "missing": missing,
           "differ": differ}
    print(json.dumps(res))
    if json_out:
        with open(json_out, "w") as fh:
            json.dump(res, fh, indent=1)
    return not missing and not differ


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument("--out")
    ap.add_argument("--compare", nargs=2)
    ap.add_argument("--json")
    args = ap.parse_args()
    if args.compare:
        sys.exit(0 if compare(*args.compare, json_out=args.json) else 1)
    dump(args.root, args.out)
