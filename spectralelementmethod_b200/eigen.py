"""Lowest eigenpairs of the Poisson operator on the device: K x = lambda M x.

``K`` is the stiffness of -div(w grad u) with the operator's boundary conditions (Dirichlet
nodes removed, Robin diagonal included) and ``M`` the diagonal GLL mass.  The solver is LOBPCG
(Knyazev 2001) on the free nodes, driven from the host:

    lam, X, info = dof_mngr.poisson_eigenpairs(16, dirichlet="ebc")

Every pass over whole vectors runs on the device: the masked matrix-free apply (one per new
column), the preconditioner, and the two block kernels of csrc/semk_block.cu -- the Gram
kernel ``S^T diag(w) T`` that forms all inner products of two blocks in one read, and the
combine kernel ``Y = beta Y + X C`` that updates a block by a small matrix.  Only the
Rayleigh-Ritz problems (at most 96 x 96) are solved on the host (``scipy.linalg.eigh``).

Blocks are rows of [3k, n] tensors: X (k rows) first, then the search directions P and the
preconditioned residuals W of the active columns, so that the basis S = [X P W] of the
Rayleigh-Ritz step is one strided block.  Two such buffers for S and two for K S alternate:
the update S C is written to the other buffer (the combine kernel needs disjoint input and
output), which also holds the residuals and the raw W of the next step.
"""
import time

import numpy as np
import torch

from . import _lib, device

__all__ = ["poisson_eigenpairs", "BlockKernels", "CONDENSED_RTOL", "GRAM_KERNEL", "MAX_PAIRS"]

MAX_PAIRS = 32                 # 3 k <= 96: the block kernels' limit
# Relative tolerance of the condensed three-level solve that preconditions each residual.
# LOBPCG needs only a spectrally equivalent preconditioner: on 256 x 256 elements at p = 8
# (k = 16 pairs, tol 1e-8) 1e-1, 1e-2 and 1e-3 took 38, 32 and 32 iterations, 836, 1350 and 1953
# inner iterations and 7.0, 6.0 and 6.3 s on a B200 (DESIGN.md section 7,
# profiles/eigen_bench_config2.json): 1e-2 is the fastest.
CONDENSED_RTOL = 1e-2
# Which Gram kernel the solver calls: "default" (semk_block_gram_f64), "dfma" or "dmma".
GRAM_KERNEL = "default"
_BLOCKS_PER_PAIR = 12          # S and K S, two [3k, n] buffers each
_SCRATCH_VECTORS = 12          # what one condensed solve allocates, at most, in nodal vectors


class BlockKernels(object):
    """The C-ABI block kernels (semk_block_gram_f64, semk_block_combine_f64) on [m, n] row
    blocks: CUDA float64 tensors whose rows are contiguous (``stride(1) == 1``) at a row stride
    ``stride(0) >= n``."""

    _GRAM = {"default": "semk_block_gram_f64", "dfma": "semk_block_gram_dfma_f64",
             "dmma": "semk_block_gram_dmma_f64"}

    def __init__(self, dev, max_mk=96 * 96, gram_kernel="default"):
        """gram_kernel : "default" (semk_block_gram_f64), "dfma" or "dmma" -- the inner product
        of the Gram kernel; see include/semk.h."""
        self._lib = _lib.load()
        self.dev = dev
        if gram_kernel not in self._GRAM:
            raise ValueError("gram_kernel must be 'default', 'dfma' or 'dmma'")
        self._gram_fn = getattr(self._lib, self._GRAM[gram_kernel])
        # semk_block_gram_partials_len is 2 + (CTAs) * m * k; a buffer sized for the largest
        # product serves every call
        per = int(self._lib.semk_block_gram_partials_len(1, 1)) - 2
        self.partials = torch.zeros(2 + per * int(max_mk), dtype=torch.float64, device=dev)
        self._G = torch.empty(max_mk, dtype=torch.float64, device=dev)

    @staticmethod
    def _block(X, what):
        if not (isinstance(X, torch.Tensor) and X.is_cuda and X.dtype == torch.float64
                and X.dim() == 2 and X.stride(1) == 1 and X.stride(0) >= X.shape[1]):
            raise ValueError("%s must be a float64 CUDA [m, n] block with contiguous rows" % what)
        return X

    def gram(self, X, Y, w=None, out=None):
        """G = X diag(w) Y^T as a float64 NumPy [m, k] array (``out``: a CUDA tensor of at least
        m*k entries to keep it on the device instead; returned as [m, k] view)."""
        self._block(X, "X")
        self._block(Y, "Y")
        m, n = X.shape
        k = Y.shape[0]
        if Y.shape[1] != n or (w is not None and w.numel() != n):
            raise ValueError("X, Y and w must have the same length")
        if m * k > self._G.numel():
            raise ValueError("m * k = %d exceeds this BlockKernels' size" % (m * k))
        G = self._G if out is None else out
        _lib.check(self._gram_fn(
            n, m, device.ptr(X), X.stride(0), k, device.ptr(Y), Y.stride(0), device.ptr(w),
            device.ptr(G), device.ptr(self.partials), device.stream_ptr()))
        if out is not None:
            return out[:m * k].view(m, k)
        return G[:m * k].view(m, k).cpu().numpy()

    def combine(self, X, C, Y, beta=0.0):
        """Y = beta Y + C^T X, i.e. Y[j] = beta Y[j] + sum_i C[i, j] X[i] (C: [m, k], host or
        device); Y must not overlap X."""
        self._block(X, "X")
        self._block(Y, "Y")
        m, n = X.shape
        Cd = torch.as_tensor(np.ascontiguousarray(C, dtype=np.float64)).to(self.dev) \
            if not isinstance(C, torch.Tensor) else C.to(self.dev, torch.float64).contiguous()
        if Cd.shape != (m, Y.shape[0]) or Y.shape[1] != n:
            raise ValueError("C must be [m, k] for X [m, n] and Y [k, n]")
        _lib.check(self._lib.semk_block_combine_f64(
            n, m, device.ptr(X), X.stride(0), Y.shape[0], device.ptr(Cd), float(beta),
            device.ptr(Y), Y.stride(0), device.stream_ptr()))
        return Y


def _dirichlet_mask(dm, dirichlet):
    """None, a bool[n_nodes] mask, or one boundary name / a list of names -> mask or None."""
    if dirichlet is None:
        return None
    if isinstance(dirichlet, str):
        dirichlet = [dirichlet]
    arr = np.asarray(dirichlet)
    if arr.dtype == np.bool_:
        if arr.shape != (dm.mesh.n_nodes,):
            raise ValueError("dirichlet must be bool[n_nodes], a boundary name or a list of names")
        return arr
    mask = np.zeros(dm.mesh.n_nodes, dtype=bool)
    for name in dirichlet:
        mask |= dm.boundary_node_mask(name)
    return mask


def _start_block(dm, k, out):
    """Deterministic start vectors: smooth random fields sum_q c cos(a x + b y + phi) of the
    node coordinates, parameters from a CPU generator with seed 0."""
    xy = dm.node_coordinates()
    x, y = xy[0], xy[1]
    ext = float(max((x.max() - x.min()).item(), (y.max() - y.min()).item(), 1e-300))
    rng = np.random.default_rng(0)
    for j in range(k):
        a, b = rng.uniform(-1.0, 1.0, (2, 8)) * (3.0 * np.pi / ext)
        ph = rng.uniform(0.0, 2.0 * np.pi, 8)
        c = rng.standard_normal(8)
        row = out[j]
        row.zero_()
        for q in range(8):
            row.add_(torch.cos(float(a[q]) * x + float(b[q]) * y + float(ph[q])), alpha=float(c[q]))
    return out


class _Timer(object):
    """Wall time per phase, each closed by a device synchronise."""

    def __init__(self):
        self.t = {"apply": 0.0, "preconditioner": 0.0, "block": 0.0, "rayleigh_ritz": 0.0}
        self._phase, self._t0 = None, 0.0

    def __call__(self, phase):
        torch.cuda.synchronize()
        now = time.perf_counter()
        if self._phase is not None:
            self.t[self._phase] += now - self._t0
        self._phase, self._t0 = phase, now

    def stop(self):
        self(None)


def poisson_eigenpairs(dm, k, dirichlet=None, robin=None, weight=None, tol=1e-8, maxiter=500):
    """The ``k`` smallest eigenpairs of ``K x = lambda M x`` (see DOFManager.poisson_eigenpairs).
    Returns (lam float64[k] ascending, X CUDA [k, n_nodes] M-orthonormal and zero on the
    Dirichlet nodes, info dict)."""
    from scipy import linalg as sla
    from .discrete import DOFManagerSC
    k = int(k)
    if k < 1 or k > MAX_PAIRS:
        raise ValueError("k must be in [1, %d] (the block kernels take at most 3k = 96 vectors)"
                         % MAX_PAIRS)
    mask = _dirichlet_mask(dm, dirichlet)
    n = int(dm.mesh.n_nodes)
    n_free = n - (int(mask.sum()) if mask is not None else 0)
    if k >= n_free:
        raise ValueError("k = %d must be smaller than the number of free nodes (%d)" % (k, n_free))
    op = dm.poisson_operator(dirichlet=mask, robin=robin, weight=weight)
    dev = op.dev
    # a Robin boundary makes K definite only where its alpha is nonzero
    has_robin = op._bdiag is not None and op._bdiag.n > 0 and bool((op._bd_val != 0.0).any())
    singular = not op.has_dirichlet and not has_robin
    f64 = dict(dtype=torch.float64, device=dev)
    free = (torch.ones(n, **f64) if mask is None
            else torch.from_numpy((~mask).astype(np.float64)).to(dev))
    mass = op.mass_diagonal()
    M = mass * free
    Minv = free / mass

    # -- preconditioner T ~ K^-1 (K + M in the singular case) ----------------------------
    n1 = op.n1
    sc = None
    if isinstance(dm, DOFManagerSC) and 3 <= n1 <= 11:
        sc = dm.condensed_poisson_operator(dirichlet=mask, weight=weight, robin=robin,
                                           reaction=op.JxW if singular else None)
        inv_mass_int = torch.zeros(n, **f64)
        inv_mass_int[sc.n_ext:] = 1.0 / mass[sc.n_ext:]
        kind = "three-level"
    else:
        d = op.diagonal(masked=True)
        if singular:
            d = d + mass
        dinv = free / d
        kind = "jacobi"
    stats = {"applications": 0, "inner_iterations": 0}

    def precondition(R, J, W, F):
        """W[q] = T R[J[q]]; F: len(J) free rows for the loads of the condensed solves."""
        stats["applications"] += len(J)
        if sc is None:
            for q, j in enumerate(J):
                torch.mul(R[int(j)], dinv, out=W[q])
            return
        rows = [R[int(j)] for j in J]
        for q, r in enumerate(rows):
            torch.mul(r, inv_mass_int, out=F[q])
        _, pinfos = sc.solve_load_many(rows, F, rtol=CONDENSED_RTOL, preconditioner="three-level",
                                       out=W)
        stats["inner_iterations"] += sum(pinfo.iterations for pinfo in pinfos)

    # -- block storage -------------------------------------------------------------------
    # the block buffers plus the preconditioner's temporaries; the returned X (k vectors) is
    # copied out after three of the four buffers are freed
    n_vec = _BLOCKS_PER_PAIR * k + (_SCRATCH_VECTORS if sc is not None else 0)
    need = 8 * n * n_vec
    if sc is not None:       # the element-local loads of one chunk of the block solve
        need += 8 * sc.n_elem * (sc.n_ext_loc + sc.n_int_loc) * min(k, sc._block_cap())
    avail = torch.cuda.mem_get_info(dev)[0]
    if need > avail:
        raise MemoryError("poisson_eigenpairs: %d nodal vectors for k = %d need %.1f GB of device "
                          "memory, %.1f GB are free (operators included)"
                          % (n_vec, k, need / 1e9, avail / 1e9))
    cur, Kcur, nxt, Knxt = [torch.empty((3 * k, n), **f64) for _ in range(4)]
    blk = BlockKernels(dev, max_mk=9 * k * k, gram_kernel=GRAM_KERNEL)
    clock = _Timer()

    def apply_rows(src, dst):
        for q in range(src.shape[0]):
            op.apply(src[q], out=dst[q])

    def cholqr2(src, dst):
        """dst = src R^-1 with R^T R = src^T M src, twice (CholQR2, Yamamoto et al. 2015) --
        composed into one transform of ``src``."""
        G = blk.gram(src, src, M)
        Rinv = sla.solve_triangular(np.linalg.cholesky(0.5 * (G + G.T)).T, np.eye(len(G)))
        blk.combine(src, Rinv, dst)
        G2 = blk.gram(dst, dst, M)
        R2inv = sla.solve_triangular(np.linalg.cholesky(0.5 * (G2 + G2.T)).T, np.eye(len(G2)))
        blk.combine(src, Rinv @ R2inv, dst)

    # -- start: M-orthonormal X, K X, Rayleigh-Ritz on X alone -----------------------------
    clock("block")
    _start_block(dm, k, nxt[:k])
    nxt[:k].mul_(free)
    cholqr2(nxt[:k], cur[:k])
    clock("apply")
    apply_rows(cur[:k], Kcur[:k])
    clock("block")
    A = blk.gram(cur[:k], Kcur[:k])
    B = blk.gram(cur[:k], cur[:k], M)
    clock("rayleigh_ritz")
    lam, V = sla.eigh(0.5 * (A + A.T), 0.5 * (B + B.T))
    clock("block")
    blk.combine(cur[:k], V, nxt[:k])
    blk.combine(Kcur[:k], V, Knxt[:k])
    cur, Kcur, nxt, Knxt = nxt, Knxt, cur, Kcur

    active = np.ones(k, dtype=bool)
    p_cols = None            # columns whose search direction P sits in cur[k:k + len(p_cols)]
    history, restarts = [], 0
    status = "maxiter"
    it = 0
    rel = np.full(k, np.inf)
    while True:
        # residuals R = K X - M X Lambda of all pairs and their M^-1 norms
        clock("block")
        X, KX = cur[:k], Kcur[:k]
        R = nxt[k:2 * k]
        lam_col = torch.from_numpy(np.ascontiguousarray(lam)).to(dev)[:, None]
        torch.mul(X, M, out=R)
        R.mul_(lam_col)
        torch.sub(KX, R, out=R)
        rn = np.sqrt(np.maximum(np.diag(blk.gram(R, R, Minv)), 0.0))
        rel = rn / max(float(np.abs(lam).max()), 1e-300)
        history.append(float(rel.max()))
        active &= rel > tol                   # soft locking: converged pairs stay in X
        if not active.any():
            if np.all(rel <= tol):
                status = "converged"
                break
            # a locked pair drifted past tol while the others converged: iterate on it again,
            # from [X W] (it has no search direction)
            active = rel > tol
            p_cols = None
        if it >= maxiter:
            break
        it += 1
        J = np.flatnonzero(active)
        ka = len(J)
        # P of the columns that are still active, compacted to the front of its slot
        kp = 0
        if p_cols is not None:
            keep = np.searchsorted(p_cols, J)
            for q, s in enumerate(keep):
                if q != s:
                    cur[k + q].copy_(cur[k + s])
                    Kcur[k + q].copy_(Kcur[k + s])
            kp = ka
        # W = T R on the active columns, M-orthogonal to X, M-orthonormal (CholQR2), K W
        clock("preconditioner")
        Wraw = nxt[:ka]
        precondition(R, J, Wraw, nxt[2 * k:2 * k + ka])
        clock("block")
        Wraw.mul_(free)
        C1 = blk.gram(X, Wraw, M)
        blk.combine(X, -C1, Wraw, beta=1.0)
        W = cur[k + kp:k + kp + ka]
        try:
            cholqr2(Wraw, W)
        except np.linalg.LinAlgError:
            status = "breakdown"
            break
        clock("apply")
        apply_rows(W, Kcur[k + kp:k + kp + ka])
        # Rayleigh-Ritz on S = [X P W]; drop P (restart) when the basis is ill-conditioned
        while True:
            clock("block")
            m = k + kp + ka
            A = blk.gram(cur[:m], Kcur[:m])
            B = blk.gram(cur[:m], cur[:m], M)
            clock("rayleigh_ritz")
            A, B = 0.5 * (A + A.T), 0.5 * (B + B.T)
            d = 1.0 / np.sqrt(np.diag(B))
            As, Bs = A * d[:, None] * d[None, :], B * d[:, None] * d[None, :]
            ok = True
            try:
                eb = np.linalg.eigvalsh(Bs)
                ok = eb[0] > 1e-12 * eb[-1]
                if ok:
                    vals, V = sla.eigh(As, Bs)
            except np.linalg.LinAlgError:
                ok = False
            if ok or kp == 0:
                break
            # restart from [X W]: W moves down into the slot of P
            restarts += 1
            clock("block")
            for q in range(ka):
                cur[k + q].copy_(cur[k + kp + q])
                Kcur[k + q].copy_(Kcur[k + kp + q])
            kp = 0
        if not ok:
            status = "breakdown"
            break
        lam = vals[:k]
        C = V[:, :k] * d[:, None]
        # X <- S C_x and P <- [P W] C_pw (active columns), one combine per block
        Call = np.zeros((m, k + ka))
        Call[:, :k] = C
        Call[k:, k:] = C[k:, J]
        clock("block")
        blk.combine(cur[:m], Call, nxt[:k + ka])
        blk.combine(Kcur[:m], Call, Knxt[:k + ka])
        cur, Kcur, nxt, Knxt = nxt, Knxt, cur, Kcur
        p_cols = J

    # final CholQR2 so that X^T M X = I to rounding
    clock("block")
    cholqr2(cur[:k], nxt[:k])
    del cur, Kcur, Knxt
    X = nxt[:k].clone()
    del nxt
    clock.stop()
    info = {
        "iterations": it,
        "status": status,
        "residuals": rel,
        "converged": rel <= tol,
        "preconditioner": kind,
        "preconditioner_applications": stats["applications"],
        "inner_iterations": stats["inner_iterations"],
        "restarts": restarts,
        "history": history,
        "block_bytes": need,
        "time": dict(clock.t),
    }
    return np.asarray(lam, dtype=np.float64).copy(), X, info
