"""The device-resident Poisson operator (additive API; SURVEY.md 8b).

The reference has no operator object: examples/poisson.py:145-259 builds a
dense 4-index local stiffness per element, assembles a COO Schur system and
calls SuperLU.  ``PoissonOperator`` is the matrix-free replacement of that
whole path on one GPU:

    op = dof_mngr.poisson_operator(dirichlet=on_ebc)
    y  = op.apply(u)                      # y = Ahat u, Ahat = M A M + (I - M)
    d  = op.diagonal()                    # diag(Ahat)
    b  = op.rhs(f=1.0)                    # assembled load vector  Q^T (JxW f)
    x, info = op.solve_pcg(op.lift(b, g)) # Jacobi-PCG, Dirichlet data g lifted

Boundary conditions.  With the operator's weight ``w`` (1 unless ``weight=`` was given) both
operators here and in condensed.py solve

    -div(w grad u) = f                      in the domain
    u = u_D                                 on Dirichlet nodes
    w du/dn = g                             on boundaries given only flux data
    w du/dn + alpha u = g                   on Robin boundaries (alpha >= 0)

and homogeneous Neumann everywhere else.  The weak form adds
``sum_faces sum_k g(x_k) dSxW_k v(x_k)`` to the load (``boundary_load``; ``solve(flux={name:
g})``) and ``alpha(x_k) dSxW_k`` to the diagonal at face node k (``robin={name: alpha}`` of the
constructor).  ``dSxW`` is the face's GLL weight times ``|dx/dxi_t|``, the host mirror's
``SubFiniteElement.dSxW`` (same face numbering 0:W 1:E 2:S 3:N, same orientation); the face
quadrature is collocated at the GLL nodes like the volume mass, so the Robin term is
diagonal.  Dirichlet wins on a node that is also on a flux or Robin face: ``lift`` discards
the load there and the Robin diagonal enters no masked row or column.

Vectors are ``torch.float64`` CUDA tensors of length ``n_nodes`` in the
reference's global node order (whatever numbering the DOF manager produced:
lexicographic, exterior-first, RCM).  Every number is computed by the CUDA
kernels behind the C ABI (include/semk.h); nothing here falls back to NumPy.
"""
import ctypes as C

import os

import numpy as np
import torch

from . import _lib, device
from ._lib import DIRICHLET_IDENTITY, MASK_IN, MASK_OUT

__all__ = ["PoissonOperator", "PCGInfo", "default_element_order", "choose_elems_per_patch"]

# tiles are elongated along the second element axis, along which node ids are
# contiguous in the lexicographic numbering: long coalesced runs, few strided
# interface nodes (measured: 2x8 is 7 % faster than 4x4 at p = 8)
_TILES = {32: (4, 8), 16: (2, 8), 8: (1, 8), 4: (1, 4)}
_SMEM_TARGET = 113 * 1024    # <= this keeps >= 2 persistent CTAs per SM
_SMEM_LIMIT = 227 * 1024


def g_patch_stride_of(n1, pe):
    n = 3 * n1 * n1 * pe
    return n + (n & 1)              # even => 16-byte multiples for the TMA bulk copy


def eloc_patch_stride_of(n1, pe):
    return (n1 * n1 * pe + 7) & ~7   # index table, 16-byte multiples


def pn_patch_stride_of(max_patch_nodes):
    return (int(max_patch_nodes) + 3) & ~3   # node list, 16-byte multiples


def patch_smem_bytes(n1, pe, max_patch_nodes, pn_stride=None, inv_stride=None):
    """Dynamic shared memory of one CTA of the apply kernel (asks the library,
    which owns the layout: csrc/semk_apply.cu patch_smem_layout)."""
    if pn_stride is None:
        pn_stride = pn_patch_stride_of(max_patch_nodes)
    if inv_stride is None:
        inv_stride = 4 * pn_stride          # inverse table, 4 contributions per node
    return int(_lib.load().semk_patch_smem_bytes(n1, pe, g_patch_stride_of(n1, pe),
                                                 int(pn_stride),
                                                 eloc_patch_stride_of(n1, pe),
                                                 int(inv_stride)))


def choose_elems_per_patch(n1):
    """Largest patch (16, 8 or 4 elements) whose shared-memory footprint still
    lets three CTAs share an SM; else the largest that fits at all."""
    p = n1 - 1

    def est(pe):
        bx, by = _TILES[pe]
        return patch_smem_bytes(n1, pe, (bx * p + 1) * (by * p + 1))
    if n1 <= 5:
        # low orders: 4 x 8 tiles -- small elements amortise the per-patch barriers and tables
        # better and have fewer interface nodes (measured on the curved mesh: p = 4 74.2 %
        # of the HBM peak against 68.2 % with 16-element patches, p = 2 58 % against 41 %;
        # at p = 6 the 16-element patch is ahead again, profiles/r02_sweep_pe32.json)
        return 32
    for pe in (16, 8, 4):
        if est(pe) <= _SMEM_TARGET:
            return pe
    for pe in (16, 8, 4):
        if est(pe) <= _SMEM_LIMIT:
            return pe
    raise NotImplementedError("no patch size fits shared memory for n1=%d" % n1)


def _morton_order(cx, cy):
    def spread(v):
        v = v.astype(np.uint64)
        v = (v | (v << 16)) & np.uint64(0x0000FFFF0000FFFF)
        v = (v | (v << 8)) & np.uint64(0x00FF00FF00FF00FF)
        v = (v | (v << 4)) & np.uint64(0x0F0F0F0F0F0F0F0F)
        v = (v | (v << 2)) & np.uint64(0x3333333333333333)
        v = (v | (v << 1)) & np.uint64(0x5555555555555555)
        return v

    def quant(c):
        lo, hi = c.min(), c.max()
        scale = 65535.0 / (hi - lo) if hi > lo else 0.0
        return np.floor((c - lo) * scale).astype(np.uint32)
    key = spread(quant(cx)) | (spread(quant(cy)) << np.uint64(1))
    return np.argsort(key, kind="stable").astype(np.int64)


def default_element_order(mesh, elems_per_patch, tile=None, boundary_columns_first=False):
    """Engine slot order (slot -> element) that makes consecutive runs of
    ``elems_per_patch`` elements compact patches: tiles of a structured grid
    when the mesh builder recorded one, else a Morton curve through the cell
    centroids.  ``boundary_columns_first`` (structured meshes): the first and the last tile
    column come first in the patch sequence -- the columns a strip partition shares with its
    neighbours are then final after the first 2 * (tiles per column) patches, and their
    exchange overlaps the rest of the apply (semk_poisson_apply_halo_f64)."""
    shape = getattr(mesh, "_structured_shape", None)
    if shape is not None and shape[0] * shape[1] == mesh.n_cells:
        nx, ny = shape
        bx, by = tile if tile is not None else _TILES[elems_per_patch]
        if bx * by != elems_per_patch:
            raise ValueError("tile shape does not match elems_per_patch")
        ex, ey = np.divmod(np.arange(nx * ny, dtype=np.int64), ny)
        # tiles enumerated along the contiguous node direction: the resident CTAs work
        # on a compact window of the mesh at any time (best DRAM / L2 locality)
        ntx, nty = (nx + bx - 1) // bx, (ny + by - 1) // by
        col = ex // bx
        if boundary_columns_first and ntx > 2:
            rank = np.empty(ntx, dtype=np.int64)
            rank[0], rank[ntx - 1] = 0, 1
            rank[1:ntx - 1] = np.arange(2, ntx)
            col = rank[col]
        tile_id = col * nty + ey // by
        key = tile_id * (bx * by) + (ex % bx) * by + ey % by
        if nx % bx == 0 and ny % by == 0:
            return np.argsort(key, kind="stable").astype(np.int64)
        # the mesh is not a whole number of tiles: one patch per tile all the same, the
        # missing elements of the ragged tiles become empty slots (-1)
        order = np.full(ntx * nty * bx * by, -1, dtype=np.int64)
        order[key] = np.arange(nx * ny, dtype=np.int64)
        return order
    if not hasattr(mesh, "_centroids"):
        mesh._compute_cell_centroids()
    return _morton_order(mesh._centroids[:, 0], mesh._centroids[:, 1])


class PCGInfo(object):
    """iterations / status / recursive relative residual of a solve; the multilevel driver
    also reports the TRUE residual ||b - A x|| / ||b|| of the returned iterate and the
    inner (coarse-level) iteration count."""
    __slots__ = ("iterations", "status", "rel_residual", "bnorm", "converged",
                 "true_rel_residual", "inner_iterations", "inner_solves")

    def __init__(self, iterations, status, rel_residual, bnorm, true_rel_residual=None,
                 inner_iterations=None, inner_solves=None):
        self.iterations = int(iterations)
        self.status = int(status)
        self.rel_residual = float(rel_residual)
        self.bnorm = float(bnorm)
        self.converged = self.status == 0
        self.true_rel_residual = None if true_rel_residual is None else float(true_rel_residual)
        self.inner_iterations = None if inner_iterations is None else int(inner_iterations)
        self.inner_solves = None if inner_solves is None else int(inner_solves)

    def __repr__(self):
        return ("PCGInfo(iterations=%d, status=%d, rel_residual=%.3e, bnorm=%.6e)"
                % (self.iterations, self.status, self.rel_residual, self.bnorm))


class _PoissonBase(object):
    """Vector plumbing, Dirichlet lifting and the Jacobi-PCG start of the plain and the
    condensed Poisson operators (condensed.CondensedPoissonOperator).  Their vectors are
    contiguous float64 CUDA tensors of length ``_n_vec`` (n_nodes, or the n_ext exterior DOFs
    that lead the exterior-first numbering); a subclass provides ``apply`` and ``diagonal``,
    ``has_dirichlet`` and the uint8 mask ``dirichlet_dev`` over its vector."""

    def _vec(self, v, name="vector", n=None):
        n = self._n_vec if n is None else n
        if not (isinstance(v, torch.Tensor) and v.is_cuda and v.dtype == torch.float64
                and v.is_contiguous() and v.numel() == n):
            raise ValueError("%s must be a contiguous float64 CUDA tensor of length %d" % (name, n))
        return v

    def new_vector(self, fill=None):
        if fill is None:
            return torch.empty(self._n_vec, dtype=torch.float64, device=self.dev)
        return torch.full((self._n_vec,), float(fill), dtype=torch.float64, device=self.dev)

    def from_host(self, a):
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(self.dev)

    def apply_unmasked(self, u, out=None):
        """y = A u: the operator without Dirichlet rows."""
        return self.apply(u, out=out, flags=0)

    def lift(self, b, dirichlet_values=None):
        """RHS of the SPD system Ahat x = bhat: free rows b_f - A_fe g_e,
        Dirichlet rows g_e (sem/discrete.py:505-509).  ``dirichlet_values``: CUDA tensor or
        host array of the operator's vector length, or a whole nodal vector (n_nodes), of
        which the condensed operator reads the leading n_ext entries."""
        self._vec(b, "b")
        if not self.has_dirichlet:
            return b.clone()
        mask = self.dirichlet_dev.bool()
        g = torch.zeros_like(b)
        if dirichlet_values is not None:
            gv = dirichlet_values if isinstance(dirichlet_values, torch.Tensor) \
                else self.from_host(dirichlet_values)
            if gv.numel() == self.n_nodes:
                gv = gv[:self._n_vec]
            g[mask] = gv[mask]
        out = b - self.apply(g, flags=MASK_OUT)      # A (I-M) g on the free rows
        out[mask] = g[mask]
        return out

    def jacobi_inverse(self):
        if self._dinv is None:
            self._dinv = 1.0 / self.diagonal(masked=True)
        return self._dinv

    def _start_iterate(self, b, x0):
        """PCG start: a copy of ``x0``, else zeros with b on the Dirichlet rows."""
        if x0 is not None:
            return self._vec(x0, "x0").clone()
        x = torch.zeros_like(b)
        if self.has_dirichlet:
            mask = self.dirichlet_dev.bool()
            x[mask] = b[mask]
        return x

    # -- flux and Robin boundaries -----------------------------------------------------
    def boundary_faces(self, name):
        """Device face tables of the named boundary (device.BoundaryFaces), built on first
        use and kept.  An unknown name raises the ``KeyError`` of ``boundary_elements``."""
        cache = self.__dict__.setdefault("_bfaces", {})
        if name not in cache:
            cache[name] = device.BoundaryFaces(self.tab, self.dof_mngr.mesh, name, self.dev)
        return cache[name]

    def _face_values(self, bf, g, what):
        """``g`` on the face nodes of ``bf`` as a [F, n1] CUDA tensor: a scalar, nodal values
        (CUDA tensor or host array of n_nodes entries), or a callable ``g(x, y)`` on CUDA tensors
        of the face-node coordinates (the convention of a callable ``weight``)."""
        shape = (bf.n_faces, self.n1)
        if callable(g):
            v = g(bf.x[:, 0, :], bf.x[:, 1, :])
            return torch.as_tensor(v, dtype=torch.float64, device=self.dev).expand(shape)
        if isinstance(g, torch.Tensor) or np.ndim(g) != 0:
            gv = g if isinstance(g, torch.Tensor) else self.from_host(g)
            return self._vec(gv, what, self.n_nodes)[bf.node_ids_dev]
        return torch.full(shape, float(g), dtype=torch.float64, device=self.dev)

    def boundary_load(self, name, g):
        """Load of the flux condition ``w du/dn = g`` on the named boundary: the vector of the
        operator's length with ``sum_faces sum_k g(x_k) dSxW_k`` on every face node (the
        reference recipe ``b[bfe.node_ind] += g * bfe.dSxW`` over
        ``boundary_elements(name)``), summed over the faces in a fixed order.  ``g``: a scalar,
        nodal values (n_nodes) or a callable ``g(x, y)`` on CUDA tensors."""
        bf = self.boundary_faces(name)
        out = self.new_vector(0.0)
        if bf.n == 0:
            return out
        if int(bf.nodes[-1]) >= self._n_vec:
            raise AssertionError("boundary nodes must be element-exterior nodes")
        out[bf.nodes_dev] = bf.face_sum(self._face_values(bf, g, "g") * bf.dSxW)
        return out

    def _robin_terms(self, robin):
        """[(BoundaryFaces, alpha dSxW [F, n1])] of ``robin = {name: alpha}``; alpha in the
        forms of ``boundary_load``, >= 0 on every face node."""
        terms = []
        for name, alpha in dict(robin).items():
            if not callable(alpha) and np.ndim(alpha) == 0 and not float(alpha) >= 0.0:
                raise ValueError("the Robin coefficient of %r must be >= 0" % (name,))
            bf = self.boundary_faces(name)
            if bf.n_faces == 0:
                continue
            a = self._face_values(bf, alpha, "alpha")
            if not bool((a >= 0.0).all()):
                raise ValueError("the Robin coefficient of %r must be >= 0" % (name,))
            terms.append((bf, (a * bf.dSxW).contiguous()))
        return terms

    def _load(self, f, flux):
        """rhs(f) plus the boundary load of every ``flux = {name: g}`` entry, in dict order."""
        b = self.rhs(f)
        for name, g in (flux or {}).items():
            b += self.boundary_load(name, g)
        return b


class PoissonOperator(_PoissonBase):
    def __init__(self, dof_mngr, dirichlet=None, geometric_factors=None, elems_per_patch=None,
                 elem_order=None, keep_l2g=True, tile=None, weight=None, mode="auto",
                 boundary_columns_first=False, robin=None):
        """robin : {boundary name: alpha}, optional -- Robin condition w du/dn + alpha u = g
            on those boundaries: ``alpha dSxW`` joins the diagonal of every face node
            (semk_bdiag).  alpha >= 0: a scalar, nodal values (n_nodes) or a callable
            alpha(x, y) on CUDA tensors.  The load g goes to ``solve(flux=...)`` /
            ``boundary_load``."""
        _lib.require_device()
        self._lib = _lib.load()
        mesh = dof_mngr.mesh
        self.dof_mngr = dof_mngr
        self.tab = device.basis_tables(dof_mngr._basis)
        n1 = self.n1 = self.tab.n1
        NN = n1 * n1
        l2g = mesh.node_map_array().reshape(-1, NN)
        self.n_elem = int(l2g.shape[0])          # elements; engine slots: self.n_order
        self.n_nodes = self._n_vec = int(mesh.n_nodes)
        self.dev = torch.device("cuda", torch.cuda.current_device())

        if dirichlet is not None:
            dirichlet = np.asarray(dirichlet)
            if dirichlet.dtype != np.bool_ or dirichlet.shape != (self.n_nodes,):
                raise ValueError("dirichlet must be bool[n_nodes] (True = essential-BC node)")
        self.dirichlet_host = dirichlet
        self.has_dirichlet = dirichlet is not None and bool(dirichlet.any())

        pe = self.elems_per_patch = int(elems_per_patch or choose_elems_per_patch(n1))
        user_order = elem_order is not None
        if elem_order is None:
            elem_order = default_element_order(mesh, pe, tile, boundary_columns_first)
        self._tile = tuple(tile) if tile is not None else _TILES[pe]
        self._boundary_first = bool(boundary_columns_first and not user_order and getattr(
            mesh, "_structured_shape", None) is not None)
        sc, ar = _lib.hostplan(n1, l2g, self.n_nodes, elem_order, pe, dirichlet, arrays=(
            _lib.PA_PNBLK, _lib.PA_PATCH_HDR, _lib.PA_SHARED_REC, _lib.PA_SHARED_EXT,
            _lib.PA_SHARED_CHUNK, _lib.PA_ELBLK, _lib.PA_INVBLK, _lib.PA_ELEM_OF_SLOT,
            _lib.PA_PATCH_MAXNODE, _lib.PA_CHUNK_MAXPATCH, _lib.PA_REC_MAXPATCH))
        # engine slots = elements + empty padding slots (-1 entries of the order)
        self.n_order = int(ar[_lib.PA_ELEM_OF_SLOT].size)
        # thread mapping of the apply kernel: "column" (one thread per element column) or
        # "pair" (a column lane + a row lane per element column; high orders, n1 >= 9)
        if mode == "auto":
            mode = os.environ.get("SEMK_APPLY_MODE", "auto")      # A/B runs
        # "box": the column mapping with an arithmetic gather (csrc/semk_box.cu) -- tiled
        # structured meshes whose numbering is a regular lattice; verified patch by patch
        # on the device below (_mark_box_patches), anything else falls back to "column"
        box_ok = (not user_order and self._tile == _TILES[pe] and 3 <= n1 <= 17
                  and (pe in (8, 16) or (pe == 32 and n1 <= 7))
                  and getattr(mesh, "_structured_shape", None) is not None)
        if mode == "auto":
            # measured: the pair mapping only wins at p = 16 (profiles/r02_sweep_pair.json);
            # the box gather is 1.5 - 2.5 % ahead of the table-driven one wherever it applies
            # (profiles/r02_box_ab.txt)
            mode = "pair" if n1 == 17 else ("box" if box_ok else "column")
        if mode not in ("column", "pair", "box"):
            raise ValueError("mode must be 'auto', 'column', 'pair' or 'box'")
        if mode == "box" and not box_ok:
            mode = "column"          # not a tiled structured mesh: the table-driven kernel
        self.kernel_variant = {"column": 0, "pair": 1, "box": 2}[mode]
        self.kernel_name = {0: "patch_kernel<%d,%d,APPLY>", 1: "ho_patch_kernel<%d,%d>",
                            2: "patch_kernel<%d,%d,APPLY,BOX>"}[self.kernel_variant] % (n1, pe)
        actual = int(self._lib.semk_resident_ctas_variant(
            self.kernel_variant, n1, pe, g_patch_stride_of(n1, pe), int(sc[_lib.PS_PN_STRIDE]),
            int(sc[_lib.PS_EL_STRIDE]), int(sc[_lib.PS_INV_STRIDE])))
        if actual <= 0:
            raise NotImplementedError(
                "patch of %d elements does not fit in shared memory (%s); pass a smaller "
                "elems_per_patch or a more local elem_order" % (pe, _lib.last_error()))
        self.plan_scalars = sc
        self.resident_ctas = actual
        smem = patch_smem_bytes(n1, pe, sc[_lib.PS_MAX_PATCH_NODES], sc[_lib.PS_PN_STRIDE],
                                sc[_lib.PS_INV_STRIDE])
        self.smem_bytes = smem

        t = {}
        for k in (_lib.PA_PNBLK, _lib.PA_PATCH_HDR, _lib.PA_SHARED_REC, _lib.PA_SHARED_EXT,
                  _lib.PA_SHARED_CHUNK):
            t[k] = device.as_i32_bits(ar[k], self.dev)
        t[_lib.PA_ELBLK] = torch.from_numpy(ar[_lib.PA_ELBLK].view(np.int16)).to(self.dev)
        t[_lib.PA_INVBLK] = torch.from_numpy(ar[_lib.PA_INVBLK].view(np.int16)).to(self.dev)
        t[_lib.PA_ELEM_OF_SLOT] = torch.from_numpy(ar[_lib.PA_ELEM_OF_SLOT]).to(self.dev)
        self._tables = t
        # what the staged host apply needs to cut the patch sequence into stages
        hdr = ar[_lib.PA_PATCH_HDR].reshape(-1, 8)
        self._stage_info = (hdr[:, 4].astype(np.int64), ar[_lib.PA_PATCH_MAXNODE].astype(np.int64),
                            ar[_lib.PA_CHUNK_MAXPATCH][:sc[_lib.PS_N_SHARED_CHUNK]].astype(np.int64),
                            ar[_lib.PA_REC_MAXPATCH][:sc[_lib.PS_N_SHARED_REC]].astype(np.int64))
        self._stage_cache = {}
        self.elem_of_slot_host = ar[_lib.PA_ELEM_OF_SLOT]
        self.n_slot_elems = sc[_lib.PS_N_SLOT_ELEMS]
        self.n_patch = sc[_lib.PS_N_PATCH]
        self.n_shared = sc[_lib.PS_N_SHARED]
        self.n_slots = sc[_lib.PS_N_SLOTS]

        f64 = dict(dtype=torch.float64, device=self.dev)
        self.g_patch_stride = g_patch_stride_of(n1, pe)
        self.G = torch.zeros((self.n_patch, self.g_patch_stride), **f64)
        self.JxW = torch.empty((self.n_elem, NN), **f64)
        self.l2g_dev = device.as_i32_bits(l2g, self.dev)
        device.stiffness_factors(self.tab, mesh, self.l2g_dev, self.n_order, self.G,
                                 self.g_patch_stride, pe, self.JxW,
                                 elem_of_slot=t[_lib.PA_ELEM_OF_SLOT],
                                 geometric_factors=geometric_factors, weight=weight)
        self.weighted = weight is not None
        self.box_ld = 0
        if self.kernel_variant == 2:
            self.box_ld = self._mark_box_patches(l2g, t)
            if self.box_ld == 0:             # the numbering is not a regular lattice
                self.kernel_variant = 0
                self.kernel_name = "patch_kernel<%d,%d,APPLY>" % (n1, pe)
                self.resident_ctas = int(self._lib.semk_resident_ctas_variant(
                    0, n1, pe, g_patch_stride_of(n1, pe), int(sc[_lib.PS_PN_STRIDE]),
                    int(sc[_lib.PS_EL_STRIDE]), int(sc[_lib.PS_INV_STRIDE])))
        # separable element operator (semk_op.separable): every element is axis-aligned, so
        # K1 wrote the G01 slab as exact zeros (weights included) -- one device reduction.
        # The pair mapping (kernel_variant 1) has no separable form and keeps three factors.
        nnp = NN * pe
        self.separable = (self.kernel_variant != 1 and self.n_patch > 0
                          and not bool(self.G[:, nnp:2 * nnp].any()))
        if self.separable:
            self.kernel_name = self.kernel_name[:-1] + ",SEP>"
            self.resident_ctas = int(self._lib.semk_resident_ctas_sep(
                self.kernel_variant, 1, n1, pe, g_patch_stride_of(n1, pe),
                int(sc[_lib.PS_PN_STRIDE]), int(sc[_lib.PS_EL_STRIDE]),
                int(sc[_lib.PS_INV_STRIDE])))
            if self.resident_ctas <= 0:
                raise NotImplementedError("separable patch kernel: %s" % _lib.last_error())
            self.smem_bytes = int(self._lib.semk_patch_smem_bytes_sep(
                1, n1, pe, g_patch_stride_of(n1, pe), int(sc[_lib.PS_PN_STRIDE]),
                eloc_patch_stride_of(n1, pe), int(sc[_lib.PS_INV_STRIDE])))
        # CTA b of the persistent kernel runs patches b, b + grid, ...; a grid that is a
        # multiple of the patches per tile column would pin every CTA to one tile row (a
        # measured 10 % slowdown): step off the resonance by one CTA
        actual = self.resident_ctas
        self.max_ctas = 0
        shape = getattr(mesh, "_structured_shape", None)
        if shape is not None and not user_order:
            by = (tile if tile is not None else _TILES[pe])[1]
            per_column = -(-shape[1] // by)
            if per_column > 1 and actual > 1 and (actual % per_column == 0 or per_column % actual == 0):
                self.max_ctas = actual - 1
        if not keep_l2g:
            self.l2g_dev = None

        self.slot_buf = torch.zeros(max(self.n_slots, 1), **f64)
        self.partials = torch.zeros(
            int(self._lib.semk_partials_len(self.n_patch, self.n_shared)), **f64)
        self.vec_partials = torch.zeros(int(self._lib.semk_vec_partials_len(self.n_nodes)), **f64)
        self.dirichlet_dev = (torch.from_numpy(dirichlet.astype(np.uint8)).to(self.dev)
                              if dirichlet is not None else None)

        op = _lib.semk_op()
        op.n1, op.elems_per_patch = n1, pe
        op.n_elem, op.n_nodes, op.n_patch = self.n_order, self.n_nodes, self.n_patch
        op.max_patch_nodes = sc[_lib.PS_MAX_PATCH_NODES]
        op.max_ctas = self.max_ctas
        op.g_patch_stride = self.g_patch_stride
        op.G = self.G.data_ptr()
        op.patch_hdr = t[_lib.PA_PATCH_HDR].data_ptr()
        op.pnode = t[_lib.PA_PNBLK].data_ptr()
        op.pn_patch_stride = sc[_lib.PS_PN_STRIDE]
        op.eloc = t[_lib.PA_ELBLK].data_ptr()
        op.eloc_patch_stride = sc[_lib.PS_EL_STRIDE]
        op.inv = t[_lib.PA_INVBLK].data_ptr()
        op.inv_patch_stride = sc[_lib.PS_INV_STRIDE]
        op.inv_width = sc[_lib.PS_INV_WIDTH]
        op.n_slots = self.n_slots
        op.slot_buf = self.slot_buf.data_ptr()
        op.n_shared = sc[_lib.PS_N_SHARED_REC]
        op.shared_rec = t[_lib.PA_SHARED_REC].data_ptr()
        op.shared_ext = t[_lib.PA_SHARED_EXT].data_ptr()
        op.n_shared_chunk = sc[_lib.PS_N_SHARED_CHUNK]
        op.shared_chunk = t[_lib.PA_SHARED_CHUNK].data_ptr()
        op.partials = self.partials.data_ptr()
        op.D_host = self.tab.D_host.ctypes.data
        op.dirichlet = self.dirichlet_dev.data_ptr() if self.has_dirichlet else None
        op.kernel_variant = self.kernel_variant
        op.box_ld = self.box_ld
        op.separable = int(self.separable)
        self._op = op
        self._masked_flags = (MASK_IN | MASK_OUT | DIRICHLET_IDENTITY) if self.has_dirichlet else 0
        self._dinv = None
        self._bdiag = None
        if robin:
            self._init_robin(robin)

    # -- helpers ---------------------------------------------------------------------
    def _init_robin(self, robin):
        """semk_bdiag of the Robin boundaries: the distinct nodes of all of them, ascending,
        and their assembled sum of alpha dSxW (per boundary a fixed-order face sum, then the
        boundaries in dict order)."""
        dense = self.new_vector(0.0)
        node_sets = [np.zeros(0, dtype=np.uint32)]
        for bf, a_dsxw in self._robin_terms(robin):
            dense[bf.nodes_dev] += bf.face_sum(a_dsxw)
            node_sets.append(bf.nodes)
        nodes = np.unique(np.concatenate(node_sets))
        self._bd_node = device.as_i32_bits(nodes, self.dev)
        self._bd_val = dense[torch.from_numpy(nodes.astype(np.int64)).to(self.dev)].contiguous()
        self._bd_partials = torch.zeros(int(self._lib.semk_vec_partials_len(nodes.size)),
                                        dtype=torch.float64, device=self.dev)
        bd = _lib.semk_bdiag()
        bd.n = int(nodes.size)
        bd.node = self._bd_node.data_ptr()
        bd.val = self._bd_val.data_ptr()
        bd.partials = self._bd_partials.data_ptr()
        self._bdiag = bd

    def _no_robin(self, what):
        if self._bdiag is not None:
            raise NotImplementedError("%s does not include the Robin boundary term; use apply / "
                                      "solve_pcg of this operator" % what)

    def _mark_box_patches(self, l2g, t):
        """kernel_variant 2 (csrc/semk_box.cu): find the patches that are regular tile boxes
        -- node (m, t) of slot le = lx*by + ly has the id base + (lx*p + m)*ld + ly*p + t --
        and carry no Dirichlet node, and write the mask of their non-empty slots into word 3
        of their device header (0 = table-driven path).  Runs on the device.  Returns the row
        stride ``ld`` of the lattice, 0 if no patch qualifies."""
        n1, pe, p = self.n1, self.elems_per_patch, self.n1 - 1
        bx, by = self._tile
        if l2g.shape[0] == 0 or p < 1:
            return 0
        ld = int(l2g[0, n1]) - int(l2g[0, 0])
        if ld < by * p + 1 or self.n_nodes >= 2 ** 31:
            return 0
        L = self.l2g_dev.view(self.n_elem, n1 * n1)
        base = L[:, 0].clone()
        k = torch.arange(n1, device=self.dev, dtype=torch.int32)
        pattern = (k[:, None] * ld + k[None, :]).reshape(-1)
        ok_elem = ((L - base[:, None]) == pattern[None, :]).all(dim=1)
        if self.dirichlet_host is not None and self.has_dirichlet:
            dmask = torch.from_numpy(self.dirichlet_host).to(self.dev)
            ok_elem &= ~dmask[L.long()].any(dim=1)
            del dmask
        slots = t[_lib.PA_ELEM_OF_SLOT]
        n_patch = int(self.n_patch)
        if slots.numel() < n_patch * pe:
            slots = torch.cat([slots, slots.new_full((n_patch * pe - slots.numel(),), -1)])
        slots = slots.view(n_patch, pe)
        present = slots >= 0
        idx = slots.clamp(min=0)
        le = torch.arange(pe, device=self.dev, dtype=torch.int64)
        off = ((le // by) * p * ld + (le % by) * p).to(torch.int32)
        hdr = t[_lib.PA_PATCH_HDR].view(n_patch, 8)
        base_p = hdr[:, 4]
        good = ok_elem[idx] & (base[idx] == base_p[:, None] + off[None, :])
        ok_patch = (good | ~present).all(dim=1) & present[:, 0]
        mask = (present.to(torch.int64) << le[None, :]).sum(dim=1)
        mask = torch.where(mask >= 2 ** 31, mask - 2 ** 32, mask)      # uint32 bits in an int32
        hdr[:, 3] = torch.where(ok_patch, mask, torch.zeros_like(mask)).to(torch.int32)
        self.n_box_patches = int(ok_patch.sum().item())
        return ld if self.n_box_patches > 0 else 0

    @property
    def algorithmic_bytes_per_apply(self):
        """SURVEY.md 8(d): read u, write y, 3 geometric factors (2 for a separable operator,
        whose apply does not read G01) + one uint32 L2G entry per element-local node."""
        per_node = 20 if self.separable else 28
        return 16 * self.n_nodes + per_node * self.n_elem * self.n1 * self.n1

    # -- operator --------------------------------------------------------------------
    def apply(self, u, out=None, flags=None, dot_out=None):
        """y = Ahat u with Ahat = M A M + (I - M) (A if no Dirichlet mask).
        ``flags`` overrides the masking (bit-or of MASK_IN, MASK_OUT,
        DIRICHLET_IDENTITY; 0 = the pure Neumann operator A).  ``dot_out``:
        optional 1-element device tensor receiving u.y.  A Robin operator adds its boundary
        diagonal on the rows and columns the flags leave unmasked."""
        self._vec(u, "u")
        y = self.new_vector() if out is None else self._vec(out, "out")
        if flags is None:
            flags = self._masked_flags
        if self._bdiag is not None:
            _lib.check(self._lib.semk_poisson_apply_bdiag_f64(
                C.byref(self._op), C.byref(self._bdiag), device.ptr(u), device.ptr(y), int(flags),
                device.ptr(dot_out), device.stream_ptr()))
            return y
        _lib.check(self._lib.semk_poisson_apply_f64(
            C.byref(self._op), device.ptr(u), device.ptr(y), int(flags), device.ptr(dot_out),
            device.stream_ptr()))
        return y

    def apply_atomic(self, u, out=None, flags=None):
        """Same operator through the independent atomic-scatter kernel."""
        self._no_robin("apply_atomic")
        if self.l2g_dev is None:
            raise RuntimeError("operator was built with keep_l2g=False")
        self._vec(u, "u")
        y = self.new_vector() if out is None else self._vec(out, "out")
        if flags is None:
            flags = self._masked_flags
        _lib.check(self._lib.semk_poisson_apply_atomic_f64(
            self.n1, self.n_order, self.n_nodes, device.ptr(self.l2g_dev),
            device.ptr(self._tables[_lib.PA_ELEM_OF_SLOT]), device.ptr(self.G),
            self.g_patch_stride, self.elems_per_patch,
            device.ptr(self.tab.D_host), device.ptr(self.dirichlet_dev), device.ptr(u),
            device.ptr(y), int(flags), device.stream_ptr()))
        return y

    def stage_table(self, n_stages):
        """Cut the patch sequence into ``n_stages`` equal runs and tabulate, per
        stage, what it needs and what it completes (``semk_stage``):
        interface chunks / records whose highest patch is done, the prefix of
        u its patches read, the prefix of y that is final afterwards."""
        n_stages = max(1, min(int(n_stages), 64, self.n_patch))
        if n_stages in self._stage_cache:
            return self._stage_cache[n_stages]
        pmin, pmax, cmax, rmax = self._stage_info
        ends = (np.arange(1, n_stages + 1, dtype=np.int64) * self.n_patch) // n_stages
        need = np.maximum.accumulate(pmax) + 1                   # u read by patches [0, p]
        # smallest node id still touched by a patch >= p (n_nodes past the end)
        open_from = np.append(np.minimum.accumulate(pmin[::-1])[::-1], self.n_nodes)
        arr = (_lib.semk_stage * n_stages)()
        for i, pe in enumerate(ends.tolist()):
            last = i == n_stages - 1
            arr[i].patch_end = pe
            arr[i].chunk_end = int(np.searchsorted(cmax, pe, side="left"))
            arr[i].rec_end = int(np.searchsorted(rmax, pe, side="left"))
            arr[i].u_need = self.n_nodes if last else int(need[pe - 1])
            arr[i].y_final = self.n_nodes if last else int(open_from[pe])
        self._stage_cache[n_stages] = (arr, n_stages)
        return self._stage_cache[n_stages]

    def boundary_split(self):
        """(patch_end, chunk_end, rec_end) of the two boundary tile columns of a structured
        mesh whose plan was built with ``boundary_columns_first``: the patches that touch the
        first / last node column and the prefixes of the interface tables they complete.
        None when the plan has no such prefix."""
        self._no_robin("boundary_split (the halo-overlapped apply)")
        if not getattr(self, "_boundary_first", False):
            return None
        shape = getattr(self.dof_mngr.mesh, "_structured_shape", None)
        bx, by = self._tile
        ntx, nty = -(-shape[0] // bx), -(-shape[1] // by)
        if ntx <= 2:
            return None
        pe = 2 * nty
        _pmin, _pmax, cmax, rmax = self._stage_info
        return (int(pe), int(np.searchsorted(cmax, pe, side="left")),
                int(np.searchsorted(rmax, pe, side="left")))

    def apply_range(self, u, y, pb, pe, cb, ce, rb, re, flags=None):
        """Patches [pb, pe) and interface entries [cb, ce) / [rb, re) of the apply."""
        self._no_robin("apply_range")
        if flags is None:
            flags = self._masked_flags
        _lib.check(self._lib.semk_poisson_apply_range_f64(
            C.byref(self._op), device.ptr(u), device.ptr(y), int(flags), int(pb), int(pe), int(cb),
            int(ce), int(rb), int(re), device.stream_ptr()))
        return y

    def apply_halo(self, u, out, split, halo, dirichlet_u8):
        """The apply of one rank of a strip partition with its interface exchange overlapped
        (semk_poisson_apply_halo_f64): the patches of ``split`` (``boundary_split``) first,
        then the exchange of ``halo`` (a semk_halo struct; uint8 Dirichlet mask
        ``dirichlet_u8``) on a side stream while the interior patches run."""
        self._no_robin("apply_halo")
        y = self.new_vector() if out is None else out
        _lib.check(self._lib.semk_poisson_apply_halo_f64(
            C.byref(self._op), device.ptr(u), device.ptr(y), int(self._masked_flags), split[0],
            split[1], split[2], C.byref(halo), device.ptr(dirichlet_u8), device.stream_ptr()))
        return y

    def apply_host(self, u_host, y_host, scratch=None, stages=16):
        """End-to-end call on HOST buffers (numpy float64 or pinned torch CPU
        tensors): H2D copy, apply, D2H copy, synchronised on return.  With
        ``stages`` > 1 the three phases are pipelined over that many runs of
        patches (upload of the next run and download of the previous one
        overlap the compute; semk_poisson_apply_host_staged_f64)."""
        self._no_robin("apply_host")
        if scratch is None:
            scratch = (self.new_vector(), self.new_vector())
        if stages and stages > 1:
            arr, n = self.stage_table(stages)
            _lib.check(self._lib.semk_poisson_apply_host_staged_f64(
                C.byref(self._op), arr, n, device.ptr(u_host), device.ptr(y_host),
                device.ptr(scratch[0]), device.ptr(scratch[1]), int(self._masked_flags),
                device.stream_ptr()))
            return y_host
        _lib.check(self._lib.semk_poisson_apply_host_f64(
            C.byref(self._op), device.ptr(u_host), device.ptr(y_host), device.ptr(scratch[0]),
            device.ptr(scratch[1]), int(self._masked_flags), device.stream_ptr()))
        return y_host

    def apply_host_many(self, u_hosts, y_hosts, scratch=None, stages=16):
        """A batch of independent applies on HOST buffers (lists of pinned torch CPU tensors
        or numpy arrays, float64[n_nodes] each): like ``apply_host`` per pair, but with two
        device scratch sets, so that the upload of apply k+1 overlaps the download of apply
        k (semk_poisson_apply_host_batch_f64).  ``scratch``: four device vectors
        (d_u0, d_y0, d_u1, d_y1) or None.  Synchronised on return."""
        self._no_robin("apply_host_many")
        if len(u_hosts) != len(y_hosts):
            raise ValueError("u_hosts and y_hosts must have the same length")
        n = len(u_hosts)
        if scratch is None:
            scratch = tuple(self.new_vector() for _ in range(4))
        if len(scratch) != 4:
            raise ValueError("scratch must hold four device vectors")
        for a in list(u_hosts) + list(y_hosts):
            if int(a.numel() if isinstance(a, torch.Tensor) else a.size) != self.n_nodes:
                raise ValueError("host buffers must hold n_nodes float64 values")
        arr, n_st = self.stage_table(stages)
        ups = (C.c_void_p * max(n, 1))(*[device.ptr(a) for a in u_hosts])
        downs = (C.c_void_p * max(n, 1))(*[device.ptr(a) for a in y_hosts])
        _lib.check(self._lib.semk_poisson_apply_host_batch_f64(
            C.byref(self._op), arr, n_st, n, ups, downs, device.ptr(scratch[0]),
            device.ptr(scratch[1]), device.ptr(scratch[2]), device.ptr(scratch[3]),
            int(self._masked_flags), device.stream_ptr()))
        return y_hosts

    def assemble(self, loc, out=None, mask=False, fill_dirichlet=0.0):
        """Assemble an element-local field ``loc[n_slot_elems, NN]`` (engine
        slot order) into a global vector (the reference's ``grhs[inds] +=``)."""
        y = self.new_vector() if out is None else self._vec(out, "out")
        _lib.check(self._lib.semk_assemble_f64(
            C.byref(self._op), device.ptr(loc), device.ptr(y), MASK_OUT if mask else 0,
            float(fill_dirichlet), device.stream_ptr()))
        return y

    def diagonal(self, masked=True):
        """diag(Ahat) (masked: 1 on Dirichlet rows) or diag(A), Robin diagonal included."""
        loc = torch.empty((self.n_slot_elems, self.n1 * self.n1), dtype=torch.float64,
                          device=self.dev)
        _lib.check(self._lib.semk_poisson_local_diag_f64(
            C.byref(self._op), device.ptr(self.tab.dev()[0]), device.ptr(loc), device.stream_ptr()))
        mask = masked and self.has_dirichlet
        d = self.assemble(loc, mask=mask, fill_dirichlet=1.0)
        if self._bdiag is not None and self._bdiag.n > 0:
            nodes = self._bd_node.long() & 0xFFFFFFFF
            val = self._bd_val
            if mask:
                val = torch.where(self.dirichlet_dev[nodes].bool(), torch.zeros_like(val), val)
            d[nodes] += val
        return d

    def rhs(self, f=1.0):
        """Load vector b = Q^T (JxW . f); ``f`` a scalar or nodal values
        (examples/poisson.py:200 uses f = 1).  The volume load only: flux and Robin data enter
        through ``boundary_load`` (``solve(flux=...)``)."""
        fv = None
        scale = 1.0
        if isinstance(f, torch.Tensor):
            fv = self._vec(f, "f")
        elif np.ndim(f) == 0:
            scale = float(f)
        else:
            fv = self.from_host(f)
        if fv is not None and self.l2g_dev is None:
            raise RuntimeError("operator was built with keep_l2g=False")
        loc = torch.empty((self.n_slot_elems, self.n1 * self.n1), dtype=torch.float64,
                          device=self.dev)
        _lib.check(self._lib.semk_weighted_local_f64(
            self.n1, self.n_order, self.n_slot_elems, device.ptr(self.JxW),
            device.ptr(self.l2g_dev), device.ptr(self._tables[_lib.PA_ELEM_OF_SLOT]),
            device.ptr(fv), device.ptr(loc), device.stream_ptr()))
        b = self.assemble(loc)
        if scale != 1.0:
            b *= scale
        return b

    def mass_diagonal(self):
        """Diagonal (lumped = exact for GLL collocation) mass matrix."""
        return self.rhs(1.0)

    # -- solver ----------------------------------------------------------------------
    def solve_pcg(self, b, x0=None, rtol=1e-12, maxiter=200000, check_every=25):
        """Jacobi-preconditioned CG on Ahat x = b (b already lifted).  Returns
        (x, PCGInfo).  The loop runs on the device (native driver,
        csrc/semk_vec.cu); the host polls 64 bytes every ``check_every``
        iterations."""
        self._vec(b, "b")
        x = self._start_iterate(b, x0)
        dinv = self.jacobi_inverse()
        work = torch.empty(3 * (self.n_nodes + 32), dtype=torch.float64, device=self.dev)
        sc = torch.zeros(8, dtype=torch.float64, device=self.dev)
        info = _lib.semk_pcg_info()
        if self._bdiag is not None:
            rc = self._lib.semk_pcg_solve_bdiag_f64(
                C.byref(self._op), C.byref(self._bdiag), device.ptr(b), device.ptr(x),
                device.ptr(dinv), device.ptr(work), device.ptr(sc), device.ptr(self.vec_partials),
                float(rtol), int(maxiter), int(check_every), C.byref(info), device.stream_ptr())
        else:
            rc = self._lib.semk_pcg_solve_f64(
                C.byref(self._op), device.ptr(b), device.ptr(x), device.ptr(dinv),
                device.ptr(work), device.ptr(sc), device.ptr(self.vec_partials), float(rtol),
                int(maxiter), int(check_every), C.byref(info), device.stream_ptr())
        _lib.check(rc)
        return x, PCGInfo(info.iterations, info.status, info.rel_residual, info.bnorm)

    def solve(self, f=1.0, dirichlet_values=None, flux=None, **pcg_kwargs):
        """Poisson solve in one call: assemble the load, add the boundary loads of ``flux =
        {name: g}`` (``boundary_load``), lift the Dirichlet data, run PCG.  Returns (u,
        PCGInfo)."""
        b = self.lift(self._load(f, flux), dirichlet_values)
        return self.solve_pcg(b, **pcg_kwargs)

    # -- small-mesh test helper ----------------------------------------------------------
    def to_scipy_csr(self, masked=False, tol=0.0):
        """Assembled matrix by applying the operator to unit vectors (tests,
        small meshes only)."""
        from scipy import sparse
        n = self.n_nodes
        if n > 20000:
            raise ValueError("to_scipy_csr is meant for small meshes")
        cols = []
        e = self.new_vector(0.0)
        y = self.new_vector()
        flags = None if masked else 0
        for j in range(n):
            e[j] = 1.0
            self.apply(e, out=y, flags=flags)
            e[j] = 0.0
            c = y.cpu().numpy()
            c[np.abs(c) <= tol] = 0.0
            cols.append(sparse.csc_matrix(c.reshape(-1, 1)))
        return sparse.hstack(cols).tocsr()


class PCGKernels(object):
    """The C-ABI vector kernels of Jacobi-PCG bound to one operator's scratch
    (used by distributed.distributed_pcg, where the loop is driven from Python
    so that NCCL all-reduces can sit between the kernels)."""

    def __init__(self, op, n=None):
        self.op = op
        self._lib = op._lib
        # vector length: the operator's nodal vectors, or the condensed (exterior) vectors of
        # a CondensedPoissonOperator (same scratch / mask attributes)
        self.n = op.n_nodes if n is None else int(n)

    def init(self, b, Ax, dinv, r, p, sc, n_dot):
        _lib.check(self._lib.semk_pcg_init_f64(
            self.n, int(n_dot), device.ptr(b), device.ptr(Ax), device.ptr(dinv),
            device.ptr(self.op.dirichlet_dev if self.op.has_dirichlet else None),
            device.ptr(r), device.ptr(p), device.ptr(sc), device.ptr(self.op.vec_partials),
            device.stream_ptr()))

    def update_xr(self, p, Ap, dinv, x, r, sc, n_dot):
        _lib.check(self._lib.semk_pcg_update_xr_f64(
            self.n, int(n_dot), device.ptr(p), device.ptr(Ap), device.ptr(dinv), device.ptr(x),
            device.ptr(r), device.ptr(sc), device.ptr(self.op.vec_partials), device.stream_ptr()))

    def update_r(self, p, Ap, dinv, r, sc, n_dot):
        """update_xr without the x update (paired with update_px)."""
        _lib.check(self._lib.semk_pcg_update_xr_f64(
            self.n, int(n_dot), device.ptr(p), device.ptr(Ap), device.ptr(dinv), None,
            device.ptr(r), device.ptr(sc), device.ptr(self.op.vec_partials), device.stream_ptr()))

    def update_px(self, r, dinv, p, x, sc):
        """p = dinv r + beta p and x += alpha p_old in one pass."""
        _lib.check(self._lib.semk_pcg_update_px_f64(
            self.n, device.ptr(r), device.ptr(dinv), device.ptr(p), device.ptr(x), device.ptr(sc),
            device.ptr(self.op.vec_partials), device.stream_ptr()))

    def update_p(self, r, dinv, p, sc):
        _lib.check(self._lib.semk_pcg_update_p_f64(
            self.n, device.ptr(r), device.ptr(dinv), device.ptr(p), device.ptr(sc),
            device.ptr(self.op.vec_partials), device.stream_ptr()))

    def dot(self, a, b, out):
        _lib.check(self._lib.semk_dot_f64(
            int(a.numel()), device.ptr(a), device.ptr(b), device.ptr(out),
            device.ptr(self.op.vec_partials), device.stream_ptr()))
        return out
