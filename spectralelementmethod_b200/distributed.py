"""Element-partitioned multi-GPU execution (one process per GPU, NCCL).

The reference is single-process (SURVEY.md 8e); the only coupling between
elements is the scatter-add over shared nodes (sem/discrete.py:499) and, in a
Krylov solver, the inner products.  A structured mesh is cut into vertical
strips of whole element columns, one per rank:

    rank r owns element columns [r*nx_local, (r+1)*nx_local)

Each rank builds an ordinary local mesh of its strip with the natural local
numbering (node id = i_local*NY + j).  The node column shared with the left
neighbour is ids [0, NY), the one shared with the right neighbour is ids
[n - NY, n) -- both contiguous, so the interface exchange needs no pack
kernels.  The right neighbour owns a shared column: rank r's owned nodes are
the prefix [0, n_owned), n_owned = n - NY (n on the last rank), which is what
the PCG kernels' ``n_dot`` argument expects.

Per operator apply: one local apply (partial sums on the interface columns)
and ONE exchange kernel that pushes the boundary columns into the neighbours'
memory over NVLink (CUDA IPC peer pointers), waits for theirs, adds them and
re-imposes the Dirichlet identity rows (``PeerHalo``, csrc/semk_peer.cu).  An
NCCL send/recv path (``exchange="nccl"``) is kept for comparison and for
process groups without peer access; the CPU tests use it over gloo.
p.Ap is taken on the *partial* sums before the exchange: summed over ranks it
equals the global p.Ap exactly, so it rides on the same all-reduce.
"""
import numpy as np
import torch
import torch.distributed as dist

__all__ = ["StripPartition", "CondensedStripView", "DistributedOperator", "PeerHalo",
           "PeerComm", "distributed_pcg", "distributed_multilevel_pcg",
           "strip_vertex_aggregates", "DistributedPoisson",
           "DistributedCondensedPoisson"]


class _StripColumns(object):
    """Contiguous id ranges of the two interface columns and the owned prefix of a strip, from
    ``NY`` (entries of one column), ``n_local`` and ``right`` (the right neighbour owns the
    column it shares)."""

    @property
    def left_slice(self):
        return slice(0, self.NY)

    @property
    def right_slice(self):
        return slice(self.n_local - self.NY, self.n_local)

    @property
    def n_owned(self):
        return self.n_local - (self.NY if self.right is not None else 0)


class StripPartition(_StripColumns):
    """Description of one rank's strip of a global (nx_local*world) x ny mesh."""

    def __init__(self, rank, world, nx_local, ny, p, bounds=(-1.0, 1.0, -1.0, 1.0)):
        if not (0 <= rank < world):
            raise ValueError("rank out of range")
        self.rank, self.world = int(rank), int(world)
        self.nx_local, self.ny, self.p = int(nx_local), int(ny), int(p)
        self.nx_global = self.nx_local * self.world
        self.NY = self.ny * self.p + 1
        self.NX_local = self.nx_local * self.p + 1
        self.n_local = self.NX_local * self.NY
        self.left = rank - 1 if rank > 0 else None
        self.right = rank + 1 if rank < world - 1 else None
        x0, x1, y0, y1 = bounds
        w = (x1 - x0) / self.world
        self.bounds_global = bounds
        self.bounds_local = (x0 + rank * w, x0 + (rank + 1) * w, y0, y1)
        self.n_global = (self.nx_global * self.p + 1) * self.NY

    def global_ids(self):
        """Global lattice id of every local node (global id = i*NY + j)."""
        i0 = self.rank * self.nx_local * self.p
        return (np.arange(self.n_local, dtype=np.int64) + i0 * self.NY)

    def local_coordinates(self, kind="S"):
        """Coordinates of the local lattice, cut from the global lattice so
        that shared columns are bit-identical on both ranks."""
        x0, x1, y0, y1 = self.bounds_global
        gx = np.linspace(x0, x1, self.nx_global * self.p + 1)
        i0 = self.rank * self.nx_local * self.p
        X, Y = np.meshgrid(gx[i0:i0 + self.NX_local], np.linspace(y0, y1, self.NY), indexing="ij")
        if kind == "C":
            s = 0.08 * np.sin(np.pi * X) * np.sin(np.pi * Y)
            X, Y = X + s, Y + s
        elif kind != "S":
            raise ValueError("kind must be 'S' or 'C'")
        return np.vstack([X.ravel(), Y.ravel()])

    def build_local_mesh(self, kind="S"):
        """Local Mesh with the global problem's boundaries: 'ebc' = global
        left edge (rank 0 only) + bottom, 'nbc' = global right edge (last rank
        only) + top."""
        from . import meshgen
        from .discrete import Mesh
        from .geometry import Quadrilateral
        nx, ny, p = self.nx_local, self.ny, self.p
        mesh = Mesh(2)
        mesh.set_nodes(self.local_coordinates(kind))
        g = mesh.add_geometry(Quadrilateral(p + 1, p + 1))
        r = mesh.new_region("interior")
        ebc, nbc = mesh.new_boundary("ebc"), mesh.new_boundary("nbc")
        mesh.add_cells(meshgen.structured_node_maps(nx, ny, p), g, r)
        cell = np.arange(nx * ny).reshape(nx, ny)
        if self.left is None:
            mesh.add_boundary_cells(cell[0, :], ebc, 1, 0)
        mesh.add_boundary_cells(cell[:, 0], ebc, 1, 2)
        if self.right is None:
            mesh.add_boundary_cells(cell[-1, :], nbc, 1, 1)
        mesh.add_boundary_cells(cell[:, -1], nbc, 1, 3)
        mesh._structured_shape = (nx, ny)
        return mesh


class CondensedStripView(_StripColumns):
    """A strip partition seen through the exterior-first numbering of
    ``DOFManagerSC`` (sem/discrete.py:314-359) on the rank-local mesh: condensed
    vectors have ``n_ext`` entries, and because the renumbering keeps the
    exterior nodes in ascending old id, the column shared with the left
    neighbour is still ids ``[0, NY)`` and the one shared with the right
    neighbour ids ``[n_ext - NY, n_ext)``, in the same order along the column
    (every node of an interface column is an element-exterior node).  Exposes
    the attributes ``DistributedOperator`` / ``PeerHalo`` / ``distributed_pcg``
    read from a ``StripPartition``."""

    def __init__(self, part, n_ext, column=None):
        self.base = part
        self.rank, self.world = part.rank, part.world
        self.left, self.right = part.left, part.right
        # entries of one interface column: all its nodes for exterior vectors; ``column`` =
        # ny + 1 describes vertex (coarse) vectors, whose compact ids are ordered the same way
        self.NY = part.NY if column is None else int(column)
        self.n_local = int(n_ext)


def _all_ok(ok, group, device):
    """Collective AND of a per-rank success flag."""
    t = torch.tensor([1.0 if ok else 0.0], device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MIN, group=group)
    return float(t) >= 1.0


class _PeerRegions(object):
    """One exported region per rank + the mappings of a set of peers (CUDA IPC).  Set-up and
    tear-down are COLLECTIVE and symmetric: either every rank ends up with all its mappings
    or every rank raises, and nobody frees a region that a peer may still have mapped
    (close the mappings, barrier, then free)."""

    def __init__(self, nbytes, peers, group, device):
        import ctypes as C
        from . import _lib
        self._lib = lib = _lib.load()
        self._check = _lib.check
        self.group, self.device = group, device
        self.mine = C.c_void_p()
        self.mapped = {}                     # peer rank -> c_void_p
        handle = (C.c_ubyte * 64)()
        err = None
        try:
            _lib.check(lib.semk_peer_alloc(int(nbytes), C.byref(self.mine), handle))
        except Exception as e:              # noqa: BLE001 -- re-raised collectively below
            err = e
        handles = [None] * dist.get_world_size(group)
        dist.all_gather_object(handles, bytes(handle) if err is None else None, group=group)
        for peer in peers:
            if err is not None:
                break
            try:
                if handles[peer] is None:
                    raise RuntimeError("rank %d could not export its region" % peer)
                buf = (C.c_ubyte * 64).from_buffer_copy(handles[peer])
                ptr = C.c_void_p()
                _lib.check(lib.semk_peer_open(buf, C.byref(ptr)))
                self.mapped[peer] = ptr
            except Exception as e:          # noqa: BLE001
                err = e
        if not _all_ok(err is None, group, device):
            self.close()
            raise RuntimeError("peer-memory regions unavailable on at least one rank: %r" % (err,))

    def close(self):
        """Collective: all ranks unmap their peers before anyone frees."""
        if self.device is not None and torch.cuda.is_available():
            torch.cuda.synchronize(self.device)
        for ptr in self.mapped.values():
            if ptr:
                self._lib.semk_peer_close(ptr)
        self.mapped = {}
        dist.barrier(group=self.group)
        if self.mine:
            self._lib.semk_peer_free(self.mine)
            self.mine.value = None


class PeerHalo(object):
    """Interface exchange over NVLink peer memory: every rank exports one
    exchange region (flags + receive buffers) through CUDA IPC and maps its
    neighbours' regions; ``exchange`` launches the single fused kernel
    semk_halo_exchange_f64 (push, publish epoch, wait, add, Dirichlet fix-up).
    All ranks must call ``exchange`` the same number of times (SPMD).  ``c`` is the
    semk_halo struct the native multilevel driver uses to issue exchanges itself; the
    epoch counter lives there, so Python- and C-issued exchanges share one sequence."""

    def __init__(self, part, group=None, device=None):
        from . import _lib
        self._lib = lib = _lib.load()
        self._check = _lib.check
        self.part = part
        self.group = group
        self.device = device
        nbytes = int(lib.semk_halo_region_bytes(part.NY))
        peers = [q for q in (part.left, part.right) if q is not None]
        self._regions = _PeerRegions(nbytes, peers, group, device)
        self.status = torch.zeros(1, dtype=torch.int32, device=device)
        self.c = _lib.semk_halo()
        self.c.n_col = part.NY
        self.c.mine = self._regions.mine.value
        self.c.left = self._regions.mapped[part.left].value if part.left is not None else None
        self.c.right = self._regions.mapped[part.right].value if part.right is not None else None
        self.c.epoch = 0
        self.c.status = self.status.data_ptr()

    @property
    def epoch(self):
        return int(self.c.epoch)

    def exchange(self, y, u=None, dirichlet=None, dot_inout=None):
        """Sum the interface columns of y across neighbours in place; with
        ``dirichlet`` (uint8 device mask) also y = u on the Dirichlet nodes of
        those columns, and the doubly counted u^2 leaves ``dot_inout``."""
        self.c.epoch += 1
        stream = torch.cuda.current_stream(self.device).cuda_stream
        self._check(self._lib.semk_halo_exchange_f64(
            self.part.NY, y.numel(), y.data_ptr(),
            u.data_ptr() if u is not None else None,
            dirichlet.data_ptr() if dirichlet is not None else None,
            self.c.mine, self.c.left, self.c.right, self.c.epoch,
            dot_inout.data_ptr() if dot_inout is not None else None,
            self.status.data_ptr(), stream))
        return y

    def check(self):
        """Raise if a neighbour failed to deliver a column (synchronises)."""
        if int(self.status.item()) != 0:
            raise RuntimeError("peer halo exchange timed out waiting for a neighbour")

    def close(self):
        self._regions.close()


class PeerComm(object):
    """Small-vector all-reduce over NVLink peer memory (semk_comm_allreduce_f64,
    csrc/semk_ml.cu): every rank maps every other rank's region; one single-CTA kernel per
    all-reduce pushes, publishes an epoch, waits and sums in rank order, so the result is
    bit-identical on all ranks and the launch can sit inside a native solver loop."""

    def __init__(self, rank, world, capacity, group=None, device=None):
        from . import _lib
        self._lib = lib = _lib.load()
        self._check = _lib.check
        if world > _lib.COMM_MAX_WORLD:
            raise NotImplementedError("PeerComm supports up to %d ranks" % _lib.COMM_MAX_WORLD)
        self.rank, self.world, self.capacity = int(rank), int(world), int(capacity)
        self.group, self.device = group, device
        nbytes = int(lib.semk_comm_region_bytes(self.world, self.capacity))
        peers = [q for q in range(self.world) if q != self.rank]
        self._regions = _PeerRegions(nbytes, peers, group, device)
        self.status = torch.zeros(1, dtype=torch.int32, device=device)
        self.c = _lib.semk_comm()
        self.c.rank, self.c.world, self.c.capacity = self.rank, self.world, self.capacity
        for q in range(self.world):
            self.c.regions[q] = (self._regions.mine.value if q == self.rank
                                 else self._regions.mapped[q].value)
        self.c.status = self.status.data_ptr()

    def allreduce(self, buf, n=None):
        """buf[:n] <- sum over ranks, in place (float64 CUDA tensor, n <= capacity)."""
        import ctypes as C
        n = buf.numel() if n is None else int(n)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        self._check(self._lib.semk_comm_allreduce_f64(C.byref(self.c), buf.data_ptr(), n, stream))
        return buf

    def check(self):
        if int(self.status.item()) != 0:
            raise RuntimeError("peer all-reduce timed out waiting for a rank")

    def close(self):
        self._regions.close()


class DistributedOperator(object):
    """Global operator = local operators + interface exchange.

    local_apply(u, out, dot_out) -> out : the rank-local operator *without*
        Dirichlet identity rows on interface nodes resolved (partial sums on
        the interface columns).  In production this is
        ``PoissonOperator.apply``; the CPU tests inject an oracle-based one.
    dirichlet : bool tensor [n_local] or None -- identity rows are re-imposed
        on the interface columns after the exchange (each side wrote u there,
        the sum would double it).
    """

    def __init__(self, part, local_apply, dirichlet=None, group=None, device=None, halo=None,
                 dot=None, overlap=None):
        self.part = part
        self.local_apply = local_apply
        # overlap(u, out, dirichlet_u8) -> out: local apply + peer exchange in one native call
        # with the exchange hidden behind the interior patches (PoissonOperator.apply_halo);
        # used whenever no fused dot is requested
        self.overlap = overlap
        self._dot = dot               # dot(a, b, out): the C-ABI reduction (PCGKernels.dot)
        self.group = group
        self.device = device
        self.halo = halo              # PeerHalo: fused NVLink exchange (else NCCL / gloo p2p)
        self._dir_u8 = None
        if halo is not None and dirichlet is not None:
            self._dir_u8 = torch.as_tensor(np.asarray(dirichlet).astype(np.uint8)).to(device)
        NY = part.NY
        kw = dict(dtype=torch.float64, device=device)
        self._recv_left = torch.empty(NY, **kw) if part.left is not None else None
        self._recv_right = torch.empty(NY, **kw) if part.right is not None else None
        self._fix_ids = None          # Dirichlet nodes on interface columns
        self._fix_nonowned = None     # ... those this rank does not own (its right column)
        if dirichlet is not None:
            d = torch.as_tensor(dirichlet).to("cpu").bool()
            ids = []
            if part.left is not None:
                ids.append(torch.nonzero(d[part.left_slice]).ravel())
            if part.right is not None:
                right = torch.nonzero(d[part.right_slice]).ravel() + (part.n_local - NY)
                ids.append(right)
                if right.numel():
                    self._fix_nonowned = right.to(device)
            if ids:
                ids = torch.cat(ids)
                if ids.numel():
                    self._fix_ids = ids.to(device)

    def exchange_add(self, y):
        """Sum the interface columns of y across neighbouring ranks, in place."""
        part = self.part
        if self.halo is not None:
            return self.halo.exchange(y)
        ops = []
        if part.left is not None:
            ops.append(dist.P2POp(dist.isend, y[part.left_slice], part.left, self.group))
            ops.append(dist.P2POp(dist.irecv, self._recv_left, part.left, self.group))
        if part.right is not None:
            ops.append(dist.P2POp(dist.isend, y[part.right_slice], part.right, self.group))
            ops.append(dist.P2POp(dist.irecv, self._recv_right, part.right, self.group))
        if not ops:
            return y
        for req in dist.batch_isend_irecv(ops):
            req.wait()
        if part.left is not None:
            y[part.left_slice] += self._recv_left
        if part.right is not None:
            y[part.right_slice] += self._recv_right
        return y

    def apply(self, u, out=None, dot_out=None):
        """y = A_global u on this rank's nodes.  ``dot_out`` (1-element
        tensor) receives this rank's share of u.y; all-reduce it for the
        global value."""
        if self.overlap is not None and dot_out is None and self.halo is not None:
            return self.overlap(u, out, self._dir_u8)
        return self.finish(self.local_apply(u, out, dot_out), u, dot_out)

    def finish(self, y, u, dot_out=None):
        """Second half of ``apply`` for a local result ``y`` (also one computed elsewhere, such
        as the staged host apply's): sum the interface columns across neighbours and re-impose
        the Dirichlet identity rows on them, in place.  ``dot_out``: this rank's share of u.y
        from the local apply, corrected here for the shared column."""
        if self.halo is not None:
            return self.halo.exchange(y, u, self._dir_u8, dot_out)
        self.exchange_add(y)
        if self._fix_ids is not None:
            y[self._fix_ids] = u[self._fix_ids]
        if dot_out is not None and self._fix_nonowned is not None:
            # identity rows on a shared column were counted by both ranks
            dup = u[self._fix_nonowned]
            dot_out -= (dup * dup).sum()
        return y

    def owned_dot(self, a, b):
        """a . b over the owned prefix, summed over the ranks (1-element tensor)."""
        n = self.part.n_owned
        if self._dot is not None:
            s = torch.empty(1, dtype=torch.float64, device=a.device)
            self._dot(a[:n], b[:n], s)
        else:                         # CPU stand-in of the tests
            s = torch.dot(a[:n], b[:n]).reshape(1)
        dist.all_reduce(s, group=self.group)
        return s


def distributed_pcg(dop, b, x, dinv, kernels, rtol=1e-12, maxiter=200000, check_every=25):
    """Jacobi-PCG over all ranks with device-resident scalars.

    kernels: object with init(b, Ax, dinv, r, p, sc, n_dot), update_xr(p, Ap,
    dinv, x, r, sc, n_dot), update_p(r, dinv, p, sc) -- the C-ABI vector
    kernels (operators.PCGKernels) or a CPU stand-in in the tests.  Two
    all-reduces per iteration (p.Ap; [r.z, r.r]); the host polls the scalars
    every ``check_every`` iterations.  Returns (iterations, rel_residual,
    converged)."""
    part = dop.part
    n_dot = part.n_owned
    r, p, Ap = torch.empty_like(b), torch.empty_like(b), torch.empty_like(b)
    sc = torch.zeros(8, dtype=torch.float64, device=b.device)
    dop.apply(x, out=Ap)
    kernels.init(b, Ap, dinv, r, p, sc, n_dot)
    dist.all_reduce(sc[0:5], group=dop.group)
    sc[2] = sc[0]
    h = sc.cpu()
    bb = float(h[4])
    tol2 = rtol * rtol
    if bb == 0.0 or float(h[3]) <= tol2 * bb:
        return 0, (float(h[3]) / bb) ** 0.5 if bb > 0 else 0.0, True
    it = 0
    while it < maxiter:
        fused = hasattr(kernels, "update_px")   # x += alpha p rides with the p update
        for _ in range(min(check_every, maxiter - it)):
            dop.apply(p, out=Ap, dot_out=sc[1:2])
            dist.all_reduce(sc[1:2], group=dop.group)
            if fused:
                kernels.update_r(p, Ap, dinv, r, sc, n_dot)
            else:
                kernels.update_xr(p, Ap, dinv, x, r, sc, n_dot)
            dist.all_reduce(sc[2:4], group=dop.group)
            if fused:
                kernels.update_px(r, dinv, p, x, sc)
            else:
                kernels.update_p(r, dinv, p, sc)
            it += 1
        h = sc.cpu()
        if getattr(dop, "halo", None) is not None:
            dop.halo.check()
        if float(h[7]) != 0.0:
            from ._lib import SolverFailure
            raise SolverFailure("distributed PCG breakdown (p.Ap <= 0 or non-finite)")
        if float(h[3]) <= tol2 * bb:
            return it, (float(h[3]) / bb) ** 0.5, True
    return it, (float(h[3]) / bb) ** 0.5, False


def distributed_multilevel_pcg(dop, dop_c, ops, b, x, rtol=1e-12, maxiter=1000, inner_rtol=1e-2,
                               inner_maxiter=20000, flexible=True, top=None):
    """Host twin of the native multilevel driver (semk_sc_mlpcg_solve_f64, csrc/semk_ml.cu)
    on a strip partition: the same algorithm, step by step, with the rank-local pieces
    injected -- NumPy stand-ins in the world_size-2 gloo tests, which is how the N > 1
    logic (owned prefixes, interface sums, replicated top level) is covered on CPU.

        M^-1 r = D^-1 r + P xc,  xc ~= Ac^-1 P^T r   (inner PCG on the vertex coarse operator,
        preconditioned by Dc^-1, or by Dc^-1 + P2 A3inv P2^T when ``top`` is given)

    dop / dop_c : DistributedOperator of the fine (exterior) and the coarse (vertex) level.
    ops : residual(b, Ax) -> (r, b_masked) ; jacobi(r) -> z ; restrict(r, n_owned) -> rc ;
          prolong_add(xc, z) ; new_coarse() ; dinv_c.
    top : None, or an object with agg_restrict(q, n_owned) -> r3 (this rank's owned vertices,
          global aggregate ids), A3inv (replicated dense inverse) and agg_prolong_add(y3, z).
    The restriction runs over OWNED fine nodes only and the coarse interface column is then
    summed across neighbours; r3 is summed over all ranks.  ``flexible``: Polak-Ribiere beta
    (the inner solve makes the preconditioner vary from step to step).
    Returns (outer iterations, relative residual, converged, total inner iterations)."""
    group = dop.group

    def inner_precond(q):
        z = ops.dinv_c * q
        if top is not None:
            r3 = top.agg_restrict(q, dop_c.part.n_owned)
            dist.all_reduce(r3, group=group)
            top.agg_prolong_add(top.A3inv @ r3, z)
        return z

    def inner_solve(rc):
        xc = ops.new_coarse()
        r = rc.clone()
        bb = float(dop_c.owned_dot(r, r))
        if bb == 0.0:
            return xc, 0
        z = inner_precond(r)
        p = z.clone()
        rz = float(dop_c.owned_dot(r, z))
        Ap = torch.empty_like(p)
        dot = torch.zeros(1, dtype=torch.float64, device=rc.device)
        it = 0
        while it < inner_maxiter:
            dop_c.apply(p, out=Ap, dot_out=dot)
            dist.all_reduce(dot, group=group)
            pAp = float(dot)
            if not pAp > 0.0:
                from ._lib import SolverFailure
                raise SolverFailure("inner PCG breakdown (p.Ap <= 0 or non-finite)")
            alpha = rz / pAp
            xc += alpha * p
            r -= alpha * Ap
            it += 1
            if float(dop_c.owned_dot(r, r)) <= inner_rtol * inner_rtol * bb:
                break
            z = inner_precond(r)
            rz_new = float(dop_c.owned_dot(r, z))
            p.mul_(rz_new / rz).add_(z)
            rz = rz_new
        return xc, it

    def precondition(res):
        z = ops.jacobi(res)
        rc = ops.restrict(res, dop.part.n_owned)
        dop_c.exchange_add(rc)
        xc, itc = inner_solve(rc)
        ops.prolong_add(xc, z)
        return z, itc

    r, bm = ops.residual(b, dop.apply(x))
    bb = float(dop.owned_dot(bm, bm))
    rr = float(dop.owned_dot(r, r))
    tol2 = rtol * rtol
    if bb == 0.0 or rr <= tol2 * bb:
        return 0, (rr / bb) ** 0.5 if bb > 0 else 0.0, True, 0
    z, inner_total = precondition(r)
    p = z.clone()
    rz = float(dop.owned_dot(r, z))
    dot = torch.zeros(1, dtype=torch.float64, device=b.device)
    Ap = torch.empty_like(b)
    it = 0
    while it < maxiter:
        dop.apply(p, out=Ap, dot_out=dot)
        dist.all_reduce(dot, group=group)
        pAp = float(dot)
        if not pAp > 0.0:
            from ._lib import SolverFailure
            raise SolverFailure("multilevel PCG breakdown (p.Ap <= 0 or non-finite)")
        alpha = rz / pAp
        x += alpha * p
        r -= alpha * Ap
        it += 1
        rr = float(dop.owned_dot(r, r))
        if rr <= tol2 * bb:
            return it, (rr / bb) ** 0.5, True, inner_total
        z, itc = precondition(r)
        inner_total += itc
        rz_new = float(dop.owned_dot(r, z))
        beta = -alpha * float(dop.owned_dot(z, Ap)) / rz if flexible else rz_new / rz
        p.mul_(beta).add_(z)
        rz = rz_new
    return it, (rr / bb) ** 0.5, False, inner_total


def strip_vertex_aggregates(part, vertex_lex_ids, dirichlet_c, max_tiles=4096):
    """GLOBAL aggregate id of every local vertex of a strip partition (third level of the
    multilevel preconditioner): k x k element tiles of the global mesh; a vertex joins the
    tile of the element to its lower left, vertices on the essential boundary join nothing
    (0xffffffff).  Both owners of a shared vertex column compute the same ids because
    they are derived from GLOBAL lattice positions.  ``vertex_lex_ids``: rank-local
    lexicographic node id (i * NY + j) of every vertex, in compact vertex order.
    Returns (agg uint32[n_v], n_agg, k)."""
    p, NY = part.p, part.NY
    nxg, ny = part.nx_global, part.ny
    k = 1
    while -(-nxg // k) * -(-ny // k) > max_tiles:
        k += 1
    k = max(k, min(4, max(nxg, ny)))
    tx, ty = -(-nxg // k), -(-ny // k)
    i_node, j_node = np.divmod(np.asarray(vertex_lex_ids, dtype=np.int64), NY)
    I = part.rank * part.nx_local + i_node // p
    J = j_node // p
    tile = (np.maximum(I - 1, 0) // k) * ty + np.maximum(J - 1, 0) // k
    agg = tile.astype(np.uint32)
    agg[np.asarray(dirichlet_c, dtype=bool)] = 0xFFFFFFFF
    return agg, int(tx * ty), int(k)


class _StripPoissonBase(object):
    """What the strip-partitioned plain and condensed Poisson paths share: the interface
    exchange, the global apply, diagonal, load and lifting, and Jacobi-PCG over all ranks, all
    written against the rank-local operator (``op`` or ``sc``).  ``_OP_SLOT`` names the argument
    of semk_pcg_dist_solve_f64 ("op" or "sc_op") that takes that operator's struct."""

    _OP_SLOT = None

    def __init__(self, part, group, exchange):
        if exchange not in ("auto", "peer", "nccl"):
            raise ValueError("exchange must be 'auto', 'peer' or 'nccl'")
        self.part = part
        self.group = group
        self._comm = None
        self._dinv = None

    def _open_halo(self, strip, exchange, device):
        """``halo``: the peer-memory exchange of ``strip`` (a StripPartition or a
        CondensedStripView), or None for NCCL p2p; ``exchange``: which of the two it is."""
        self.halo = None
        if exchange in ("auto", "peer"):
            # PeerHalo sets itself up collectively: either every rank maps its neighbours
            # or every rank raises; "auto" then falls back to NCCL p2p on all ranks
            try:
                self.halo = PeerHalo(strip, self.group, device)
            except RuntimeError:
                if exchange == "peer":
                    raise
        self.exchange = "peer" if self.halo is not None else "nccl"

    def _connect(self, local, strip, overlap=None):
        """``dop``: the global operator over the rank-local operator ``local`` on ``strip``."""
        from .operators import PCGKernels
        self._local = local
        self.kernels = PCGKernels(local, n=local._n_vec)
        self.dop = DistributedOperator(
            strip, lambda u, out, dot: local.apply(u, out=out, dot_out=dot),
            dirichlet=self.on_ebc[:local._n_vec] if local.has_dirichlet else None,
            group=self.group, device=local.dev, halo=self.halo, dot=self.kernels.dot,
            overlap=overlap)
        self._mask = local.dirichlet_dev.bool() if local.has_dirichlet else None

    def apply(self, u, out=None, dot_out=None):
        return self.dop.apply(u, out=out, dot_out=dot_out)

    def diagonal(self):
        d = self._local.diagonal(masked=False)
        self.dop.exchange_add(d)
        if self._mask is not None:
            d[self._mask] = 1.0
        return d

    def rhs(self, f=1.0):
        return self.dop.exchange_add(self._local.rhs(f))

    def lift(self, b, g=None):
        """b_f - A_fe g on free rows, g on Dirichlet rows (global operator).  ``g``: a CUDA
        tensor of the local operator's vector length, or a whole nodal vector, of which the
        condensed operator reads the leading n_ext entries."""
        if self._mask is None:
            return b.clone()
        gv = torch.zeros_like(b)
        if g is not None:
            if g.numel() == self._local.n_nodes:
                g = g[:self._local._n_vec]
            gv[self._mask] = g[self._mask]
        from ._lib import MASK_OUT
        t = self._local.apply(gv, flags=MASK_OUT)
        self.dop.exchange_add(t)
        out = b - t
        out[self._mask] = gv[self._mask]
        return out

    def _start(self, b, x0):
        """PCG start iterate; the global inverse diagonal on first use (collective)."""
        x = self._local._start_iterate(b, x0)
        if self._dinv is None:
            self._dinv = 1.0 / self.diagonal()
        return x

    def solve_pcg(self, b, x0=None, rtol=1e-12, maxiter=200000, check_every=25, native=True):
        """Jacobi-PCG over all ranks.  With the peer-memory exchange the native driver
        semk_pcg_dist_solve_f64 runs the whole loop (``native=False``: the host-driven loop
        with NCCL all-reduces, which is also what the NCCL / gloo paths use).  Returns (x,
        iterations, rel_residual, converged)."""
        x = self._start(b, x0)
        if self.halo is not None and native:
            it, rel, ok = self._native_jacobi_pcg(b, x, rtol, maxiter, check_every)
        else:
            it, rel, ok = distributed_pcg(self.dop, b, x, self._dinv, self.kernels, rtol=rtol,
                                          maxiter=maxiter, check_every=check_every)
        return x, it, rel, ok

    def _native_jacobi_pcg(self, b, x, rtol, maxiter, check_every):
        """semk_pcg_dist_solve_f64 on a partition whose exchanges run over peer memory: the
        whole loop (applies, interface exchanges, both all-reduces of an iteration) is issued by
        the native driver.  The PeerComm of its all-reduces is opened on first use and kept."""
        import ctypes as C
        from . import _lib, device
        lib = _lib.load()
        if self._comm is None:
            self._comm = PeerComm(self.part.rank, self.part.world, 64, self.group, b.device)
        n = b.numel()
        work = torch.empty(3 * (n + 32), dtype=torch.float64, device=b.device)
        sc = torch.zeros(32, dtype=torch.float64, device=b.device)
        info = _lib.semk_pcg_info()
        ops = {"op": None, "sc_op": None}
        ops[self._OP_SLOT] = C.byref(self._local._op)
        torch.cuda.synchronize(b.device)        # ranks enter together (the peer kernels give up
        dist.barrier(group=self.group)          # after ~2 s of waiting)
        rc = lib.semk_pcg_dist_solve_f64(
            ops["op"], ops["sc_op"], C.byref(self.halo.c), C.byref(self._comm.c),
            int(self.dop.part.n_owned), device.ptr(b), device.ptr(x), device.ptr(self._dinv),
            device.ptr(work), device.ptr(sc), device.ptr(self._local.vec_partials), float(rtol),
            int(maxiter), int(check_every), C.byref(info), device.stream_ptr())
        _lib.check(rc)
        self.halo.check()
        self._comm.check()
        return info.iterations, info.rel_residual, info.status == 0

    def close(self):
        """Collective tear-down of the peer-memory regions."""
        if self._comm is not None:
            self._comm.close()
            self._comm = None
        if self.halo is not None:
            self.halo.close()
            self.halo = None


class DistributedPoisson(_StripPoissonBase):
    """The whole multi-GPU Poisson path for the strip-partitioned structured
    configurations (BASELINE.json configs[4]): local mesh + DOF manager +
    device operator on each rank, interface exchange, global Jacobi-PCG."""

    _OP_SLOT = "op"

    def __init__(self, part, order, kind="S", group=None, elems_per_patch=None, exchange="auto",
                 overlap=True):
        _StripPoissonBase.__init__(self, part, group, exchange)
        from . import discrete
        from .basis_functions import LagrangeGaussLobatto, TensorProductQS
        self.mesh = part.build_local_mesh(kind)
        b1 = LagrangeGaussLobatto(order)
        self.mngr = discrete.DOFManager(self.mesh, 1, TensorProductQS(b1, b1), rcm_order=False)
        self.on_ebc = self.mngr.boundary_node_mask("ebc")
        self.op = op = self.mngr.poisson_operator(dirichlet=self.on_ebc,
                                                  elems_per_patch=elems_per_patch,
                                                  boundary_columns_first=overlap)
        self._open_halo(part, exchange, op.dev)
        split = op.boundary_split() if (overlap and self.halo is not None) else None
        self.overlapped = split is not None
        fn = None
        if split is not None:
            halo = self.halo

            def fn(u, out, dir_u8):
                return op.apply_halo(u, out, split, halo.c, dir_u8)
        self._connect(op, part, overlap=fn)

    def host_operator(self):
        """The local operator of the staged host apply: the same elements in the plain tile
        order (the boundary-columns-first order of ``self.op`` would make the very first stage
        need both ends of u, i.e. all of it, before anything can be computed).  Built on first
        use."""
        if getattr(self, "_op_host", None) is None:
            self._op_host = (self.mngr.poisson_operator(dirichlet=self.on_ebc,
                                                        elems_per_patch=self.op.elems_per_patch)
                             if self.op._boundary_first else self.op)
        return self._op_host

    def apply_host(self, u_host, y_host, scratch=None, stages=16):
        """y = A_global u on HOST buffers (pinned float64[n_local] in this rank's node order):
        the rank-local apply runs as the staged pipeline of ``PoissonOperator.apply_host``
        (upload of stage i+1, compute of stage i and download of stage i-1 overlap), then the
        interface columns are exchanged on the device and those two columns are downloaded
        again.  Collective: every rank calls it.  ``scratch``: (d_u, d_y) device vectors."""
        op = self.host_operator()
        if scratch is None:
            scratch = (op.new_vector(), op.new_vector())
        op.apply_host(u_host, y_host, scratch, stages=stages)
        d_u, d_y = scratch[0], scratch[1]
        self.dop.finish(d_y, d_u)
        part, NY, n = self.part, self.part.NY, self.part.n_local
        yh = y_host if isinstance(y_host, torch.Tensor) else torch.from_numpy(y_host)
        if part.left is not None:
            yh[:NY].copy_(d_y[:NY], non_blocking=True)
        if part.right is not None:
            yh[n - NY:].copy_(d_y[n - NY:], non_blocking=True)
        torch.cuda.current_stream(op.dev).synchronize()
        return y_host


class DistributedCondensedPoisson(_StripPoissonBase):
    """The statically condensed Poisson path (condensed.CondensedPoissonOperator,
    the reference's DOFManagerSC formulation, sem/discrete.py:404-528) on a strip
    partition: each rank condenses its own elements (the Schur complements are
    element-local, so nothing changes there), the condensed apply exchanges the
    interface columns of the exterior vector exactly like the uncondensed one
    (``CondensedStripView``), PCG runs on the exterior DOFs of all ranks and the
    interior back-substitution is rank-local."""

    _OP_SLOT = "sc_op"

    def __init__(self, part, order, kind="S", group=None, exchange="auto"):
        _StripPoissonBase.__init__(self, part, group, exchange)
        from . import discrete, meshgen
        from .basis_functions import LagrangeGaussLobatto, TensorProductQS
        self.mesh = part.build_local_mesh(kind)
        b1 = LagrangeGaussLobatto(order)
        self.mngr = discrete.DOFManagerSC(self.mesh, 1, TensorProductQS(b1, b1), rcm_order=False)
        self.on_ebc = self.mngr.boundary_node_mask("ebc")
        self.sc = sc = self.mngr.condensed_poisson_operator(dirichlet=self.on_ebc)
        self.view = CondensedStripView(part, sc.n_ext)
        # new local id -> lexicographic local id (StripPartition.global_ids() is indexed by those)
        lex = meshgen.structured_node_maps(part.nx_local, part.ny, part.p).reshape(-1)
        self.lexicographic_ids = np.empty(self.mesh.n_nodes, dtype=np.int64)
        self.lexicographic_ids[self.mngr.node_map_array().reshape(-1)] = lex
        self._open_halo(self.view, exchange, sc.dev)
        self._connect(sc, self.view)

    def global_ids(self):
        """Global (lexicographic, whole-mesh) node id of every local node in
        this rank's exterior-first numbering."""
        return self.part.global_ids()[self.lexicographic_ids]

    def solve_pcg(self, b, x0=None, rtol=1e-12, maxiter=200000, check_every=25,
                  preconditioner="jacobi", inner_rtol=1e-2, inner_maxiter=20000, flexible=True,
                  inner_chunk=4, max_tiles=4096, native=True):
        """Distributed PCG on the exterior DOFs.  "jacobi": semk_pcg_dist_solve_f64 with the
        peer-memory exchange (``native=False`` or NCCL exchange: the host-driven loop
        distributed_pcg with NCCL all-reduces).  "two-level" / "three-level": the native
        multilevel driver (semk_sc_mlpcg_solve_f64) -- every exchange and all-reduce is a
        peer-memory kernel issued by the driver itself, so it needs exchange="peer".
        Returns (x, iterations, rel_residual, converged); ``last_info`` keeps the PCGInfo
        (true residual, inner iterations) of a multilevel solve."""
        if preconditioner not in ("jacobi", "two-level", "three-level"):
            raise ValueError("preconditioner must be 'jacobi', 'two-level' or 'three-level'")
        if preconditioner == "jacobi":
            return _StripPoissonBase.solve_pcg(self, b, x0, rtol, maxiter, check_every, native)
        x = self._start(b, x0)
        ml = self._multilevel(3 if preconditioner == "three-level" else 2, max_tiles)
        # ranks enter together: the peer kernels give up after ~2 s of waiting
        torch.cuda.synchronize(self.sc.dev)
        dist.barrier(group=self.group)
        xs, info = self.sc.solve_pcg(
            b, x0=x, rtol=rtol, maxiter=maxiter, preconditioner=preconditioner,
            inner_rtol=inner_rtol, inner_maxiter=inner_maxiter, flexible=flexible,
            inner_chunk=inner_chunk, max_tiles=max_tiles,
            dist=(ml["dist"], self._dinv, ml["dinv_c"]))
        self.halo.check()
        ml["halo_c"].check()
        ml["comm"].check()
        self.last_info = info
        self.last_inner_iterations = info.inner_iterations
        return xs, info.iterations, info.rel_residual, info.converged

    def _multilevel(self, levels, max_tiles=4096):
        """Coarse levels of the multilevel preconditioner on the strip partition (lazy):
        the rank-local vertex coarse operator of condensed.CondensedPoissonOperator with its
        own interface exchange (the coarse interface columns are the leading / trailing
        ny + 1 compact vertex ids), the global inverse diagonal of the coarse operator, the
        peer-memory communicator and -- for three levels -- global vertex aggregates with a
        replicated dense inverse of the aggregated operator."""
        tl = getattr(self, "_ml", None)
        if tl is not None and tl["levels"] >= levels:
            return tl
        if self.halo is None:
            raise NotImplementedError("the native multilevel driver needs the peer-memory "
                                      "exchange (exchange='peer' / 'auto' with peer access)")
        import ctypes as C
        from . import _lib
        sc = self.sc
        cs, t, n_v = sc._build_coarse()
        if tl is None:
            view_c = CondensedStripView(self.part, n_v, column=self.part.ny + 1)
            halo_c = PeerHalo(view_c, self.group, sc.dev)
            dc = t["diag_c_local"].clone()
            halo_c.exchange(dc)
            if sc.has_dirichlet:
                dc[t["dirichlet_c"].bool()] = 1.0
            tl = dict(levels=2, view_c=view_c, halo_c=halo_c, dinv_c=1.0 / dc, comm=None)
        n_agg = 0
        if levels == 3:
            vids = np.unique(sc.l2g_ext_host[:, :4])
            agg, n_agg, k = strip_vertex_aggregates(self.part, self.lexicographic_ids[vids],
                                                    t["dirichlet_c_host"], max_tiles)
            sc._top = None
            sc._build_top(agg=agg, n_agg=n_agg, n_owned_c=tl["view_c"].n_owned,
                          reduce=lambda A: dist.all_reduce(A, group=self.group), source_rank=0)
            tl["aggregate_tile"] = k
        if tl["comm"] is None or tl["comm"].capacity < n_agg + 8:
            if tl["comm"] is not None:
                tl["comm"].close()
            tl["comm"] = PeerComm(self.part.rank, self.part.world, max(n_agg + 8, 64), self.group,
                                  sc.dev)
        d = _lib.semk_ml_dist()
        d.comm = C.pointer(tl["comm"].c)
        d.halo_f = C.pointer(self.halo.c)
        d.halo_c = C.pointer(tl["halo_c"].c)
        d.n_owned_f = self.view.n_owned
        d.n_owned_c = tl["view_c"].n_owned
        tl["dist"] = d
        tl["levels"] = levels
        self._ml = tl
        return tl

    def close(self):
        """Collective tear-down of the peer-memory regions."""
        tl = getattr(self, "_ml", None)
        if tl is not None:
            tl["halo_c"].close()
            if tl["comm"] is not None:
                tl["comm"].close()
            self._ml = None
        _StripPoissonBase.close(self)

    def solve(self, f=1.0, dirichlet_values=None, **pcg_kwargs):
        """Condensed load, lifting, distributed PCG on the exterior DOFs, rank-local
        interior back-substitution.  Returns (u_local[n_nodes], iterations,
        rel_residual, converged)."""
        b = self.lift(self.rhs(f), dirichlet_values)
        x, it, rel, ok = self.solve_pcg(b, **pcg_kwargs)
        return self.sc.backsolve(x, f), it, rel, ok
