"""Static condensation on the device (SURVEY.md 8(f) row 1).

The reference's solver formulation is ``DOFManagerSC`` (sem/discrete.py:283-528):
per element the interior DOFs are eliminated, ``S_e = A_ee - A_ei A_ii^-1 A_ie``
(compute_local_sc_system, :438-476), the condensed system over the element-
exterior DOFs is assembled as COO triplets (:478-500) and solved with SuperLU
(:502-511), and the interiors follow by per-element back-substitution (:513-524).

``CondensedPoissonOperator`` is that path on one GPU, matrix-based per element
and assembly-free globally:

    sc = dof_mngr.condensed_poisson_operator(dirichlet=on_ebc)   # DOFManagerSC
    y  = sc.apply(u_ext)                  # y = Shat u, Shat = M S M + (I - M)
    g  = sc.rhs(f=1.0)                    # condensed load  Q_e^T (f_e - A_ei A_ii^-1 f_i)
    u, info = sc.solve(1.0, ebc_values)   # PCG on the exterior DOFs + interior back-solve

Condensed vectors are ``torch.float64`` CUDA tensors of length ``n_ext`` =
``dof_mngr.ndof_exterior`` (the leading ids of the exterior-first numbering);
``solve`` returns the full nodal vector.  The local Schur complements are
built by the element kernel of csrc/semk_sc.cu from the same geometric factors
the matrix-free operator uses and stored packed (2p(4p+1) doubles per
element); nothing here falls back to NumPy.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib, device
from ._lib import DIRICHLET_IDENTITY, MASK_IN, MASK_OUT
from .operators import PCGInfo, _PoissonBase

__all__ = ["CondensedPoissonOperator", "CondensedLocalSystems", "condensed_tables", "coarse_tables",
           "condensed_tables_device", "coarse_tables_device",
           "element_tiles", "aggregate_tables", "aggregate_csr", "top_level_inverse"]


def condensed_tables(l2g, ext_loc, n_ext):
    """Host tables of the condensed operator (pure NumPy, T0 tier):
    ``l2g_ext[E, 4p]`` = global ids of each element's exterior nodes in the
    hierarchical local order (fe.global_dof_ind_hier[:ndof_exterior],
    sem/discrete.py:491-492) and the node -> entries table of the assembly:
    ``node_pos[node_ptr[g]:node_ptr[g+1]]`` are the positions ``e * 4p + k`` of
    the entries of node g, ascending (a stable sort) -- the fixed summation
    order that replaces ``grhs[inds_ext] += ...`` (sem/discrete.py:499)."""
    l2g_ext = np.ascontiguousarray(l2g[:, ext_loc], dtype=np.uint32)
    if int(l2g_ext.max()) >= n_ext:
        raise AssertionError("exterior nodes are not numbered first")
    if l2g_ext.size >= 2 ** 32:
        raise NotImplementedError("more than 2^32 element-exterior entries")
    flat = l2g_ext.ravel()
    node_pos = np.argsort(flat, kind="stable").astype(np.uint32)
    counts = np.bincount(flat, minlength=n_ext)
    if (counts == 0).any():
        raise AssertionError("an exterior id is not used by any element")
    node_ptr = np.zeros(n_ext + 1, dtype=np.uint32)
    np.cumsum(counts, out=node_ptr[1:])
    return l2g_ext, node_ptr, node_pos


def _u32(t):
    """int32-bit-pattern tensor of uint32 values -> int64 values."""
    return t.to(torch.int64) & 0xFFFFFFFF


def condensed_tables_device(l2g_dev, ext_loc, n_ext):
    """``condensed_tables`` on the device: the same integer tables (stable sort, so the
    node -> entries order is bit-identical to the host builder's) without the host pass
    over 32 M entries at config 2.  ``l2g_dev``: int32-bit-pattern CUDA tensor [E, NN].
    Returns int32-bit-pattern CUDA tensors (l2g_ext, node_ptr, node_pos)."""
    dev = l2g_dev.device
    ext = torch.as_tensor(np.asarray(ext_loc, dtype=np.int64), device=dev)
    l2g_ext = l2g_dev[:, ext].contiguous()
    flat = _u32(l2g_ext.reshape(-1))
    if int(flat.max()) >= n_ext:
        raise AssertionError("exterior nodes are not numbered first")
    if flat.numel() >= 2 ** 31:
        raise NotImplementedError("more than 2^31 element-exterior entries")
    node_pos = torch.sort(flat, stable=True).indices.to(torch.int32)
    counts = torch.bincount(flat, minlength=n_ext)
    if bool((counts == 0).any()):
        raise AssertionError("an exterior id is not used by any element")
    node_ptr = torch.zeros(n_ext + 1, dtype=torch.int64, device=dev)
    torch.cumsum(counts, 0, out=node_ptr[1:])
    return l2g_ext, node_ptr.to(torch.int32), node_pos


def coarse_tables_device(l2g_ext, node_ptr, node_pos, dirichlet, gll_nodes):
    """``coarse_tables`` on the device (same tables, same orders; see there).  Inputs are the
    int32-bit-pattern CUDA tensors of ``condensed_tables_device`` and a bool CUDA tensor (or
    None).  Returns a dict of CUDA tensors (uint32 tables as int32 bit patterns) + n_v."""
    dev = l2g_ext.device
    E, NE = l2g_ext.shape
    p = NE // 4
    N = p + 1
    n_ext = int(node_ptr.numel() - 1)
    t = (1.0 + np.asarray(gll_nodes, dtype=np.float64)) / 2.0
    if t.size != N:
        raise ValueError("gll_nodes must have p + 1 entries")
    va = np.zeros(NE, dtype=np.int64)
    vb = np.zeros(NE, dtype=np.int64)
    wa = np.zeros(NE)
    wb = np.zeros(NE)
    va[:4] = vb[:4] = np.arange(4)
    wa[:4] = 1.0
    inner = np.arange(1, N - 1)
    for edge, (a, b) in enumerate(((0, 1), (2, 3), (0, 2), (1, 3))):
        k = 4 + edge * (N - 2) + np.arange(N - 2)
        va[k], vb[k] = a, b
        wa[k], wb[k] = 1.0 - t[inner], t[inner]
    phi = np.zeros((NE, 4))
    phi[np.arange(NE), va] += wa
    phi[np.arange(NE), vb] += wb
    i64 = dict(dtype=torch.int64, device=dev)
    va_d, vb_d = torch.as_tensor(va, device=dev), torch.as_tensor(vb, device=dev)
    wa_d, wb_d = torch.as_tensor(wa, device=dev), torch.as_tensor(wb, device=dev)
    vert = _u32(l2g_ext[:, :4])
    vids = torch.unique(vert)                                  # sorted
    n_v = int(vids.numel())
    vmap = torch.full((n_ext,), -1, **i64)
    vmap[vids] = torch.arange(n_v, **i64)
    vert_c = vmap[vert]
    if dirichlet is None:
        dirichlet = torch.zeros(n_ext, dtype=torch.bool, device=dev)
    dirichlet = dirichlet[:n_ext]
    dirichlet_c = dirichlet[vids]
    first = _u32(node_pos)[_u32(node_ptr[:-1])]
    e = torch.div(first, NE, rounding_mode="floor")
    k = first - e * NE
    pv = torch.stack([vert_c[e, va_d[k]], vert_c[e, vb_d[k]]], dim=1)
    pw = torch.stack([wa_d[k], wb_d[k]], dim=1)
    pw[dirichlet] = 0.0
    pw[dirichlet_c[pv]] = 0.0
    flat_v, flat_w = pv.reshape(-1), pw.reshape(-1)
    flat_g = torch.arange(n_ext, **i64).repeat_interleave(2)
    keep = flat_w != 0.0
    kv = flat_v[keep]
    order = torch.sort(kv, stable=True).indices
    ridx = flat_g[keep][order]
    rw = flat_w[keep][order].contiguous()
    rptr = torch.zeros(n_v + 1, **i64)
    torch.cumsum(torch.bincount(kv, minlength=n_v), 0, out=rptr[1:])
    vflat = vert_c.reshape(-1)
    vpos = torch.sort(vflat, stable=True).indices
    vptr = torch.zeros(n_v + 1, **i64)
    torch.cumsum(torch.bincount(vflat, minlength=n_v), 0, out=vptr[1:])
    i32 = lambda a: a.to(torch.int32).contiguous()             # noqa: E731 (bit patterns < 2^31)
    return dict(phi=phi, vert_c=i32(vert_c), n_v=n_v, dirichlet_c=dirichlet_c,
                pv=i32(pv), pw=pw.contiguous(), rptr=i32(rptr), ridx=i32(ridx), rw=rw,
                vptr=i32(vptr), vpos=i32(vpos))


def _load_key(f):
    """Identity of a load ``f`` for the cached interior solution A_ii^-1 f_i (None: not
    cacheable)."""
    if isinstance(f, torch.Tensor):
        return ("tensor", f.data_ptr(), f._version, tuple(f.shape))
    if f is None or np.ndim(f) == 0:
        return ("scalar", None if f is None else float(f))
    return None


class CondensedPoissonOperator(_PoissonBase):
    def __init__(self, dof_mngr, dirichlet=None, geometric_factors=None, weight=None,
                 store_interior="auto", reaction=None, store_interior_inverse=False, robin=None):
        """store_interior : keep W_e = A_ii^-1 A_ie of every element (12.5 KB per element at
        p = 8) so that the interior back-substitution is one streaming pass instead of a
        refactorisation per element; "auto" = when it takes less than a third of the free
        device memory.

        robin : {boundary name: alpha}, optional -- Robin condition w du/dn + alpha u = g (see
        operators.py): ``alpha dSxW`` is added to ``reaction`` on the element-local face nodes
        before the local Schur complements are formed, so the term reaches S_e, the vertex
        coarse space and the aggregation level unchanged.  alpha >= 0: a scalar, nodal values
        (n_nodes) or a callable alpha(x, y) on CUDA tensors."""
        self._store_interior = store_interior
        # store_interior_inverse: also keep A_ii^-1 of every element (19 KB at p = 8): the
        # condensed load of ANY right-hand side then is a streaming pass
        # (semk_sc_load_stored_block_f64) instead of a refactorisation per element -- for
        # solvers that call rhs() many times
        self._store_inverse = bool(store_interior_inverse)
        self._init_common(dof_mngr, dirichlet)
        self._init_geometry(geometric_factors, weight)
        # reaction : float[E, N, N] element-local nodal values c >= 0 (array or CUDA tensor):
        # the operator becomes stiffness + diag(c), e.g. the JxW/rho term of the vector
        # Laplacian of examples/squirmer-axisymmetric.py:210-211
        self._react = None
        if reaction is not None:
            self._react = device._f64(reaction, self.dev).reshape(self.n_elem, -1).contiguous()
            if self._react.shape[1] != self.n1 * self.n1:
                raise ValueError("reaction must have one value per element-local node")
        if robin:
            self._add_robin(robin)
        self._schur_pass()

    def _add_robin(self, robin):
        """reaction += alpha dSxW on the element-local face nodes, [E, NN] in reference element
        order.  A corner cell has one local node on two faces: the face values are summed per
        element-local slot in a fixed order (BoundaryFaces.face_sum onto "local")."""
        terms = self._robin_terms(robin)
        react = (torch.zeros((self.n_elem, self.n1 * self.n1), dtype=torch.float64, device=self.dev)
                 if self._react is None else self._react.clone())
        flat = react.view(-1)
        for bf, a_dsxw in terms:
            if bf.n and int(bf.nodes[-1]) >= self.n_ext:
                raise AssertionError("boundary nodes must be element-exterior nodes")
            flat[bf.keys_dev] += bf.face_sum(a_dsxw, onto="local")
        self._react = react

    def _init_common(self, dof_mngr, dirichlet):
        """Masks, local orders, the exterior L2G / node -> entries tables, S and the
        scratch of the condensed operator (everything but the local systems)."""
        _lib.require_device()
        self._lib = _lib.load()
        mesh = dof_mngr.mesh
        if not getattr(mesh, "condensed", False):
            raise ValueError("static condensation needs the exterior-first numbering of "
                             "DOFManagerSC (sem/discrete.py:314-359)")
        if dof_mngr.ndof_per_node != 1:
            raise NotImplementedError("condensed_poisson_operator supports one DOF per node")
        self.dof_mngr = dof_mngr
        self.n_nodes = int(mesh.n_nodes)
        self.n_ext = self._n_vec = int(mesh.n_nodes_cell_exterior)
        full_mask = None
        if dirichlet is not None:
            dirichlet = np.asarray(dirichlet)
            if dirichlet.dtype != np.bool_ or dirichlet.shape not in ((self.n_nodes,),
                                                                      (self.n_ext,)):
                raise ValueError("dirichlet must be bool[n_nodes] or bool[ndof_exterior] "
                                 "(True = essential-BC node)")
            full_mask = np.zeros(self.n_nodes, dtype=bool)
            full_mask[:dirichlet.size] = dirichlet
            if full_mask[self.n_ext:].any():
                raise ValueError("essential-BC nodes must be element-exterior nodes")
        self.tab = device.basis_tables(dof_mngr._basis)
        n1 = self.n1 = self.tab.n1
        if n1 < 3 or n1 > 11:
            raise NotImplementedError("static condensation supports orders 2..10")
        NN = n1 * n1
        self.dev = torch.device("cuda", torch.cuda.current_device())

        geo = mesh.get_geometries()[0]
        ext_loc = np.ascontiguousarray(geo.exterior_node_ind, dtype=np.int32)
        m = np.arange(1, n1 - 1)
        lex_interior = (m[:, None] * n1 + m[None, :]).ravel()
        if not np.array_equal(np.asarray(geo.interior_node_ind, dtype=np.int64), lex_interior):
            raise AssertionError("interior local order is not lexicographic")
        self.n_ext_loc = int(ext_loc.size)
        self.n_int_loc = NN - self.n_ext_loc
        self.s_stride = self.n_ext_loc * (self.n_ext_loc + 1) // 2
        self.ext_loc_host = ext_loc

        l2g = mesh.node_map_array().reshape(-1, NN)
        self.n_elem = int(l2g.shape[0])
        # the integer tables are built on the device (stable sorts: bit-identical to the host
        # builder `condensed_tables`, tests/test_gpu_condensed.py)
        self.l2g_dev = device.as_i32_bits(l2g, self.dev)
        l2g_ext, node_ptr, node_pos = condensed_tables_device(self.l2g_dev, ext_loc, self.n_ext)
        self._l2g_ext_host = None
        self._t = dict(
            ext_loc=torch.from_numpy(ext_loc).to(self.dev),
            l2g_ext=l2g_ext, node_ptr=node_ptr, node_pos=node_pos,
        )
        self._finish_common(full_mask)

    @property
    def l2g_ext_host(self):
        """Exterior L2G table on the host, uint32[E, 4p] (downloaded on first use)."""
        if self._l2g_ext_host is None:
            self._l2g_ext_host = self._t["l2g_ext"].cpu().numpy().view(np.uint32)
        return self._l2g_ext_host

    def _init_geometry(self, geometric_factors, weight):
        """Geometric factors, one plain [3][NN] block per element in reference element
        order (the engine layout of semk_op.G with one-element patches)."""
        NN = self.n1 * self.n1
        f64 = dict(dtype=torch.float64, device=self.dev)
        self.g_stride = (3 * NN + 1) & ~1
        self.G = torch.zeros((self.n_elem, self.g_stride), **f64)
        self.JxW = torch.empty((self.n_elem, NN), **f64)
        device.stiffness_factors(self.tab, self.dof_mngr.mesh, self.l2g_dev, self.n_elem, self.G,
                                 self.g_stride, 1, self.JxW, geometric_factors=geometric_factors,
                                 weight=weight)

    def _finish_common(self, full_mask):
        f64 = dict(dtype=torch.float64, device=self.dev)
        n1 = self.n1
        self.has_dirichlet = full_mask is not None and bool(full_mask.any())
        self.dirichlet_host = None if full_mask is None else full_mask[:self.n_ext].copy()
        self.dirichlet_dev = (torch.from_numpy(self.dirichlet_host.astype(np.uint8)).to(self.dev)
                              if full_mask is not None else None)
        self.S = torch.empty((self.n_elem, self.s_stride), **f64)
        self.y_loc = torch.empty((self.n_elem, self.n_ext_loc), **f64)
        self.partials = torch.zeros(int(self._lib.semk_vec_partials_len(self.n_ext)), **f64)
        self.vec_partials = torch.zeros(int(self._lib.semk_vec_partials_len(self.n_ext)), **f64)
        self._bad = torch.zeros(1, dtype=torch.int32, device=self.dev)

        op = _lib.semk_sc_op()
        op.n1, op.n_ext_loc = n1, self.n_ext_loc
        op.n_elem, op.n_ext, op.s_stride = self.n_elem, self.n_ext, self.s_stride
        op.S = self.S.data_ptr()
        op.l2g_ext = self._t["l2g_ext"].data_ptr()
        op.y_loc = self.y_loc.data_ptr()
        op.node_ptr = self._t["node_ptr"].data_ptr()
        op.node_pos = self._t["node_pos"].data_ptr()
        op.dirichlet = self.dirichlet_dev.data_ptr() if self.has_dirichlet else None
        op.partials = self.partials.data_ptr()
        self._op = op
        self._masked_flags = (MASK_IN | MASK_OUT | DIRICHLET_IDENTITY) if self.has_dirichlet else 0

    def _schur_pass(self):
        """Local Schur complements (packed, kept), the assembled diagonal and -- memory
        permitting -- the interior solution operators W_e."""
        sdiag = torch.empty((self.n_elem, self.n_ext_loc), dtype=torch.float64, device=self.dev)
        self._W = self._c = self._c_key = None
        mode = _lib.SC_SCHUR
        want = getattr(self, "_store_interior", False)
        nbytes = 8 * self.n_elem * self.n_ext_loc * self.n_int_loc
        if want == "auto":
            want = 3 * nbytes < torch.cuda.mem_get_info(self.dev)[0]
        self._Ainv = None
        if want and not isinstance(self, CondensedLocalSystems):
            self._W = torch.empty((self.n_elem, self.n_ext_loc, self.n_int_loc),
                                  dtype=torch.float64, device=self.dev)
            mode |= _lib.SC_STORE
            if getattr(self, "_store_inverse", False):
                self._Ainv = torch.empty((self.n_elem, self.n_int_loc, self.n_int_loc),
                                         dtype=torch.float64, device=self.dev)
                mode |= _lib.SC_STORE_INV
        self._element_pass(mode, S=self.S, sdiag_loc=sdiag, W=self._W, Ainv=self._Ainv)
        self._diag_unmasked = self.assemble(sdiag)
        del sdiag
        self._dinv = None

    # -- element kernel ----------------------------------------------------------------
    def _element_pass(self, mode, S=None, sdiag_loc=None, W=None, Ainv=None):
        """One factorisation pass of sc_element_kernel (csrc/semk_sc.cu): modes SCHUR, STORE,
        STORE_INV.  The loads run in _element_block."""
        self._bad.zero_()
        _lib.check(self._lib.semk_sc_element_react_f64(
            self.n1, self.n_elem, None, device.ptr(self.G), self.g_stride, 1,
            device.ptr(self.tab.dev()[0]), device.ptr(self._t["ext_loc"]), None, None, None, 1.0,
            int(mode), device.ptr(S), self.s_stride, device.ptr(sdiag_loc), None, None,
            device.ptr(W), None, device.ptr(self._react), device.ptr(Ainv), device.ptr(self._bad),
            device.stream_ptr()))
        if int(self._bad.item()) != 0:
            raise AssertionError("an element-interior stiffness block is not positive definite")

    # -- helpers -----------------------------------------------------------------------
    @property
    def algorithmic_bytes_per_apply(self):
        """Packed S_e + one uint32 L2G entry per element-exterior node, read u,
        write y."""
        return (8 * self.s_stride + 4 * self.n_ext_loc) * self.n_elem + 16 * self.n_ext

    def local_schur(self):
        """The local Schur complements as dense host arrays ``[E, 4p, 4p]``
        (tests; compare with compute_local_sc_system, sem/discrete.py:438-476)."""
        ne = self.n_ext_loc
        packed = self.S.cpu().numpy()
        out = np.zeros((self.n_elem, ne, ne))
        r, c = np.tril_indices(ne)
        out[:, r, c] = packed
        out[:, c, r] = packed
        return out

    # -- operator ----------------------------------------------------------------------
    def apply(self, u, out=None, flags=None, dot_out=None):
        """y = Shat u over the exterior DOFs (S u with ``flags=0``)."""
        self._vec(u, "u")
        y = self.new_vector() if out is None else self._vec(out, "out")
        if flags is None:
            flags = self._masked_flags
        _lib.check(self._lib.semk_sc_apply_f64(
            C.byref(self._op), device.ptr(u), device.ptr(y), int(flags), device.ptr(dot_out),
            device.stream_ptr()))
        return y

    def assemble(self, loc, out=None, mask=False, fill_dirichlet=0.0):
        """Sum an element-local exterior field ``loc[E, 4p]`` into a condensed
        vector (``grhs[inds_ext] += ...``, sem/discrete.py:499)."""
        y = self.new_vector() if out is None else self._vec(out, "out")
        _lib.check(self._lib.semk_sc_assemble_f64(
            C.byref(self._op), device.ptr(loc), device.ptr(y), MASK_OUT if mask else 0,
            float(fill_dirichlet), device.stream_ptr()))
        return y

    def diagonal(self, masked=True):
        d = self._diag_unmasked.clone()
        if masked and self.has_dirichlet:
            d[self.dirichlet_dev.bool()] = 1.0
        return d

    def rhs(self, f=1.0):
        """Condensed load vector: assembled ``f_e - A_ei A_ii^-1 f_i`` with the
        element load ``JxW . f`` (examples/poisson.py:200; scalar or nodal f).  With W kept,
        the interior solution of a CUDA or scalar load rides along: back-substitution of the
        same load later is a stream over W (backsolve)."""
        cols, _ = self._block_loads([f])
        (_, g_loc, c, _), = self._block_rhs(cols, None, keep_c=True)
        if c is not None:
            self._c, self._c_key = c[0], _load_key(f)
        return self.assemble(g_loc[0])

    def _build_coarse(self):
        """Vertex coarse space of the two-level preconditioner (lazy): host tables
        (coarse_tables), the element coarse matrices Ace = Phi_e^T S_e Phi_e and the
        inverse diagonal of the coarse operator, all on the device."""
        if getattr(self, "_coarse", None) is not None:
            return self._coarse
        sub = [b for _, b in self.dof_mngr._basis.iter_subbases()][0]
        ct = coarse_tables_device(self._t["l2g_ext"], self._t["node_ptr"], self._t["node_pos"],
                                  self.dirichlet_dev.bool() if self.dirichlet_dev is not None
                                  else None, np.asarray(sub.nodes))
        f64 = dict(dtype=torch.float64, device=self.dev)
        n_v = ct["n_v"]
        t = dict(
            phi=device._f64(ct["phi"], self.dev),
            vert_c=ct["vert_c"], vptr=ct["vptr"], vpos=ct["vpos"], pv=ct["pv"], pw=ct["pw"],
            rptr=ct["rptr"], ridx=ct["ridx"], rw=ct["rw"],
            dirichlet_c=ct["dirichlet_c"].to(torch.uint8),
            Ace=torch.empty((self.n_elem, 16), **f64),
            y_loc_c=torch.empty((self.n_elem, 4), **f64),
            partials=torch.zeros(int(self._lib.semk_vec_partials_len(n_v)), **f64),
        )
        _lib.check(self._lib.semk_sc_coarse_elem_f64(
            C.byref(self._op), device.ptr(t["phi"]), device.ptr(t["Ace"]), device.stream_ptr()))
        cs = _lib.semk_sc_coarse()
        cs.n_v = n_v
        cs.Ace = t["Ace"].data_ptr()
        cs.vert_c = t["vert_c"].data_ptr()
        cs.y_loc_c = t["y_loc_c"].data_ptr()
        cs.vptr = t["vptr"].data_ptr()
        cs.vpos = t["vpos"].data_ptr()
        cs.dirichlet_c = t["dirichlet_c"].data_ptr() if self.has_dirichlet else None
        cs.partials = t["partials"].data_ptr()
        cs.pv = t["pv"].data_ptr()
        cs.pw = t["pw"].data_ptr()
        cs.rptr = t["rptr"].data_ptr()
        cs.ridx = t["ridx"].data_ptr()
        cs.rw = t["rw"].data_ptr()
        # diagonal of the coarse operator: assemble Ace[e][a][a]; 1 on Dirichlet vertices
        dloc = t["Ace"][:, [0, 5, 10, 15]].contiguous()
        dc = torch.empty(n_v, **f64)
        _lib.check(self._lib.semk_sc_coarse_assemble_f64(
            self.n_elem, C.byref(cs), device.ptr(dloc), device.ptr(dc), device.stream_ptr()))
        t["diag_c_local"] = dc.clone()      # this rank's elements only (distributed: + exchange)
        if self.has_dirichlet:
            dc[t["dirichlet_c"].bool()] = 1.0
        if not bool((dc > 0).all()):
            raise AssertionError("coarse operator has a non-positive diagonal entry")
        t["dinv_c"] = 1.0 / dc
        t["dirichlet_c_host"] = ct["dirichlet_c"].cpu().numpy()
        self._vertex_valence_max = int((_u32(ct["vptr"][1:]) - _u32(ct["vptr"][:-1])).max())
        # the same operator as ELL rows for the multilevel driver: one SpMV per inner
        # iteration instead of element product + vertex sum (a vertex of valence d couples
        # to at most 2 d other vertices)
        width = 2 * self._vertex_valence_max + 1
        if width <= 32:
            t["ell_cols"] = torch.empty((width, n_v), dtype=torch.int32, device=self.dev)
            t["ell_vals"] = torch.empty((width, n_v), **f64)
            over = torch.zeros(1, dtype=torch.int32, device=self.dev)
            _lib.check(self._lib.semk_sc_coarse_ell_build_f64(
                C.byref(cs), width, device.ptr(t["ell_cols"]), device.ptr(t["ell_vals"]),
                device.ptr(over), device.stream_ptr()))
            if int(over.item()) != 0:
                raise AssertionError("ELL row overflow in the coarse operator")
            cs.ell_width = width
            cs.ell_cols = t["ell_cols"].data_ptr()
            cs.ell_vals = t["ell_vals"].data_ptr()
        self._coarse = (cs, t, n_v)
        return self._coarse

    def _build_top(self, max_tiles=4096, agg=None, n_agg=None, n_owned_c=None, reduce=None,
                   source_rank=None):
        """Third level (lazy): vertex aggregates and the dense inverse of the aggregated
        coarse operator A3 = P2^T Ac P2, assembled and inverted on the device.

        One GPU: aggregates = element tiles (element_tiles / aggregate_tables).  A strip
        partition passes ``agg`` (GLOBAL aggregate id of every local vertex), the global
        ``n_agg``, the owned vertex prefix ``n_owned_c`` and ``reduce`` (sums this rank's A3
        over all ranks in place) -- the inverse is then replicated on every rank."""
        if getattr(self, "_top", None) is not None:
            return self._top
        cs, t, n_v = self._build_coarse()
        if agg is None:
            tile = element_tiles(self.dof_mngr.mesh, self.n_elem, max_tiles)
            vptr = t["vptr"].cpu().numpy().view(np.uint32)
            vpos = t["vpos"].cpu().numpy().view(np.uint32)
            at = aggregate_tables(t["vert_c"].cpu().numpy().view(np.uint32), vptr, vpos,
                                  t["dirichlet_c_host"], tile)
            agg, n_agg = at["agg"], at["n_agg"]
        agg = np.ascontiguousarray(agg, dtype=np.uint32)
        n_agg = int(n_agg)
        n_owned_c = n_v if n_owned_c is None else int(n_owned_c)
        aptr_all, aidx_all = aggregate_csr(agg, n_agg, n_v)
        aptr, aidx = aggregate_csr(agg, n_agg, n_owned_c)
        tt = dict(agg=device.as_i32_bits(agg, self.dev),
                  aptr=device.as_i32_bits(aptr, self.dev),
                  aidx=device.as_i32_bits(aidx, self.dev),
                  aptr_all=device.as_i32_bits(aptr_all, self.dev),
                  aidx_all=device.as_i32_bits(aidx_all, self.dev))
        A3 = torch.empty((n_agg, n_agg), dtype=torch.float64, device=self.dev)
        _lib.check(self._lib.semk_sc_top_assemble_f64(
            C.byref(cs), n_agg, device.ptr(tt["agg"]), device.ptr(tt["aptr_all"]),
            device.ptr(tt["aidx_all"]), device.ptr(A3), device.stream_ptr()))
        if reduce is not None:
            reduce(A3)
        A3 = 0.5 * (A3 + A3.t())
        d = torch.diagonal(A3)
        d[d == 0.0] = 1.0                     # aggregates without a free vertex
        # set-up only: dense SPD inverse by the vendor library (it enters the preconditioner,
        # not the solution); the solve itself runs on this repo's kernels
        inv = torch.linalg.inv(A3)
        if not bool(torch.isfinite(inv).all()):
            raise AssertionError("the aggregated coarse operator is singular")
        tt["A3inv"] = (0.5 * (inv + inv.t())).contiguous()
        if source_rank is not None:           # bit-identical copies on every rank
            import torch.distributed as dist
            dist.broadcast(tt["A3inv"], src=source_rank)
        # what the driver streams every inner iteration: an FP32 copy (symmetric rounding keeps
        # it symmetric; it only enters the preconditioner)
        tt["A3inv_f32"] = tt["A3inv"].to(torch.float32).contiguous()
        del A3, inv
        top = _lib.semk_sc_top()
        top.n_agg = n_agg
        top.agg = tt["agg"].data_ptr()
        top.aptr = tt["aptr"].data_ptr()
        top.aidx = tt["aidx"].data_ptr()
        top.A3inv = tt["A3inv"].data_ptr()
        top.A3inv_f32 = tt["A3inv_f32"].data_ptr()
        self._top = (top, tt, n_agg)
        return self._top

    def coarse_apply(self, xc, out=None, dot_out=None, ell=False):
        """y = Ac x on the vertex coarse space (tests / diagnostics); ``ell``: through the
        assembled ELL rows the multilevel driver uses instead of the element matrices."""
        cs, t, n_v = self._build_coarse()
        y = torch.empty(n_v, dtype=torch.float64, device=self.dev) if out is None else out
        if ell:
            _lib.check(self._lib.semk_sc_coarse_ell_apply_f64(
                C.byref(cs), device.ptr(xc), device.ptr(y), device.ptr(dot_out),
                device.stream_ptr()))
            return y
        flags = (MASK_IN | MASK_OUT | DIRICHLET_IDENTITY) if self.has_dirichlet else 0
        _lib.check(self._lib.semk_sc_coarse_apply_f64(
            self.n_elem, C.byref(cs), device.ptr(xc), device.ptr(y), flags, device.ptr(dot_out),
            device.stream_ptr()))
        return y

    def solve_pcg_refined(self, b, rtol=1e-12, max_cycles=3, **kw):
        """Multilevel PCG followed by iterative refinement on the TRUE residual: CG stops on
        its recursive residual, which at large condition numbers runs ahead of
        ``||b - Shat x|| / ||b||`` (2e-9 against 7e-13 at config 2); every cycle recomputes
        the true residual and solves for the correction until it meets ``rtol`` or stops
        halving (the attainable accuracy in FP64).  Returns (x, PCGInfo of the first solve
        with ``true_rel_residual`` of the final iterate, list of (true residual, outer
        iterations) per cycle)."""
        kw.setdefault("preconditioner", "three-level")
        x, info = self.solve_pcg(b, rtol=rtol, **kw)
        lib = self._lib
        mask = device.ptr(self.dirichlet_dev) if self.has_dirichlet else None
        r, bm, Ax = torch.empty_like(b), torch.empty_like(b), torch.empty_like(b)
        hist = []
        last = float("inf")
        for _ in range(max_cycles):
            self.apply(x, out=Ax)
            _lib.check(lib.semk_vec_resid_f64(self.n_ext, device.ptr(b), device.ptr(Ax), mask,
                                              device.ptr(r), device.ptr(bm), device.stream_ptr()))
            true = float(torch.linalg.vector_norm(r) / torch.linalg.vector_norm(bm))
            hist.append((true, info.iterations if not hist else it2))
            if true <= rtol or true > 0.5 * last:
                break
            last = true
            d, i2 = self.solve_pcg(r, rtol=min(0.1, max(rtol / true, 1e-14)), **kw)
            it2 = i2.iterations
            _lib.check(lib.semk_vec_scale_add_f64(self.n_ext, 1.0, device.ptr(d), device.ptr(x),
                                                  device.ptr(x), device.stream_ptr()))
        info.true_rel_residual = hist[-1][0]
        return x, info, hist

    def solve_pcg(self, b, x0=None, rtol=1e-12, maxiter=200000, check_every=25,
                  preconditioner="jacobi", inner_rtol=1e-2, inner_maxiter=20000, flexible=True,
                  inner_chunk=4, max_tiles=4096, dist=None):
        """PCG on Shat x = b (b already lifted); returns (x, PCGInfo).

        preconditioner : "jacobi" (diagonal of Shat); "two-level" (Jacobi + a vertex coarse
            space, M^-1 = D^-1 + P Ac^-1 P^T with linear interpolation along element edges
            and an inner Jacobi-PCG on Ac to ``inner_rtol``): the outer iteration count no
            longer grows with the mesh size; "three-level": the inner solve is itself
            preconditioned by Jacobi + an aggregation level with a dense inverse, so the
            inner count stops growing as well.  The multilevel variants run the native driver
            semk_sc_mlpcg_solve_f64 (flexible CG outside: the inner solve is inexact) and
            report the true residual of the returned iterate.
        dist : (semk_ml_dist, dinv, dinv_c) of a strip partition (distributed.py), else None."""
        self._vec(b, "b")
        if preconditioner not in ("jacobi", "two-level", "three-level"):
            raise ValueError("preconditioner must be 'jacobi', 'two-level' or 'three-level'")
        x = self._start_iterate(b, x0)
        if preconditioner != "jacobi":
            cs, t, n_v = self._build_coarse()
            levels = 3 if preconditioner == "three-level" else 2
            top, n_agg = None, 0
            if levels == 3:
                top, tt, n_agg = self._build_top(max_tiles)
            dptr, dinv, dinv_c = None, self.jacobi_inverse(), t["dinv_c"]
            if dist is not None:
                dptr, dinv, dinv_c = C.byref(dist[0]), dist[1], dist[2]
            work = torch.empty(4 * (self.n_ext + 32), dtype=torch.float64, device=self.dev)
            work_c = torch.empty(6 * (n_v + 32) + 2 * (n_agg + 64), dtype=torch.float64,
                                 device=self.dev)
            sc = torch.zeros(64, dtype=torch.float64, device=self.dev)
            opts = _lib.semk_ml_opts(float(rtol), float(inner_rtol), int(maxiter),
                                     int(inner_maxiter), levels, 1 if flexible else 0,
                                     int(inner_chunk), 0)
            info = _lib.semk_ml_info()
            rc = self._lib.semk_sc_mlpcg_solve_f64(
                C.byref(self._op), C.byref(cs), C.byref(top) if top is not None else None, dptr,
                device.ptr(b), device.ptr(x), device.ptr(dinv), device.ptr(dinv_c),
                device.ptr(work), device.ptr(work_c), device.ptr(sc),
                device.ptr(self.vec_partials), C.byref(opts), C.byref(info), device.stream_ptr())
            _lib.check(rc)
            self.last_inner_iterations = int(info.inner_iterations)
            return x, PCGInfo(info.iterations, info.status, info.rel_residual, info.bnorm,
                              info.true_rel_residual, info.inner_iterations, info.inner_solves)
        dinv = self.jacobi_inverse()
        info = _lib.semk_pcg_info()
        work = torch.empty(3 * (self.n_ext + 32), dtype=torch.float64, device=self.dev)
        sc = torch.zeros(8, dtype=torch.float64, device=self.dev)
        rc = self._lib.semk_sc_pcg_solve_f64(
            C.byref(self._op), device.ptr(b), device.ptr(x), device.ptr(dinv), device.ptr(work),
            device.ptr(sc), device.ptr(self.vec_partials), float(rtol), int(maxiter),
            int(check_every), C.byref(info), device.stream_ptr())
        _lib.check(rc)
        return x, PCGInfo(info.iterations, info.status, info.rel_residual, info.bnorm)

    def true_residual(self, b, x):
        """||b - Shat x|| / ||b|| over the free rows (diagnostics; one apply)."""
        r = b - self.apply(x)
        bm = b
        if self.has_dirichlet:
            m = self.dirichlet_dev.bool()
            r = torch.where(m, torch.zeros_like(r), r)
            bm = torch.where(m, torch.zeros_like(b), b)
        return float(r.norm() / bm.norm())

    def backsolve(self, x_ext, f=1.0, out=None):
        """Full nodal vector from the exterior solution: interiors
        ``u_i = A_ii^-1 (f_i - A_ie u_e)`` element by element
        (_solve_interior_dofs, sem/discrete.py:513-524)."""
        self._vec(x_ext, "x_ext")
        u = (torch.empty(self.n_nodes, dtype=torch.float64, device=self.dev) if out is None
             else self._vec(out, "out", self.n_nodes))
        if self._W is not None and self._c is not None and self._c_key == _load_key(f):
            self._block_backsolve(x_ext[None], [0], None, self._c, u[None])
        else:
            cols, _ = self._block_loads([f])
            self._block_backsolve(x_ext[None], [0], self._chunk_load(cols, [0], None), None,
                                  u[None])
        return u

    def solve(self, f=1.0, dirichlet_values=None, flux=None, **pcg_kwargs):
        """The whole DOFManagerSC.solve path (sem/discrete.py:526-528): condensed
        load (plus the boundary loads of ``flux = {name: g}``, which have no interior
        entries), Dirichlet lifting, PCG on the exterior DOFs, interior
        back-substitution.  Returns (u[n_nodes], PCGInfo)."""
        b = self.lift(self._load(f, flux), dirichlet_values)
        x, info = self.solve_pcg(b, **pcg_kwargs)
        return self.backsolve(x, f), info

    def solve_load(self, r, f, rtol=1e-8, preconditioner="three-level"):
        """u = A^-1 r for an assembled nodal load vector ``r`` (length n_nodes, zero on the
        Dirichlet nodes).  ``f = r * inv_mass_int``: r divided by the mass on the element-
        interior nodes and zero on the exterior ones, the nodal values whose element load JxW f
        is r on every interior node.  Condensed load of f plus the exterior entries of r
        (semk_sc_rhs_finish_f64), PCG on the exterior DOFs to ``rtol``, interior
        back-substitution.  Returns (u[n_nodes], PCGInfo)."""
        g = self.rhs(f)
        b = torch.empty_like(g)
        _lib.check(self._lib.semk_sc_rhs_finish_f64(
            self.n_ext, device.ptr(g), device.ptr(r), device.ptr(self.dirichlet_dev)
            if self.has_dirichlet else None, device.ptr(b), device.stream_ptr()))
        x, info = self.solve_pcg(b, rtol=rtol, preconditioner=preconditioner)
        return self.backsolve(x, f), info

    # -- blocks of loads ---------------------------------------------------------------
    # Column j of every *_many result is bitwise the single-load call on load j: the block
    # kernels (semk_sc_element_block_f64 and the stored-operator streams) factorise each
    # element once per chunk of columns and repeat the single kernels' operations per column,
    # and every column takes the path the single call would take.
    def _block_cap(self):
        return int(self._lib.semk_sc_block_max_cols(self.n1))

    def _block_chunks(self, k):
        """Column ranges of a block of k loads (block_chunks with this operator's cap, the
        temporaries g_loc and c of one column and the free device memory); one column without
        asking the device (the single-load calls)."""
        if k == 1:
            return [(0, 1)]
        per_col = 8 * self.n_elem * (self.n_ext_loc + self.n_int_loc)
        return block_chunks(k, self._block_cap(), per_col, torch.cuda.mem_get_info(self.dev)[0])

    def _block_loads(self, F):
        """(columns [(f_scale, nodal CUDA vector or None, cacheable)], F if it is a block)."""
        if isinstance(F, torch.Tensor):
            if not (F.is_cuda and F.dtype == torch.float64 and F.dim() == 2
                    and F.shape[1] == self.n_nodes and F.stride(1) == 1 and F.shape[0] >= 1):
                raise ValueError("F must be a float64 CUDA [k, n_nodes] block (k >= 1) with "
                                 "contiguous rows, or a sequence of loads")
            return [(1.0, F[j], True) for j in range(F.shape[0])], F
        cols = []
        for f in F:
            if isinstance(f, torch.Tensor):
                cols.append((1.0, self._vec(f, "f", self.n_nodes), True))
            elif np.ndim(f) == 0:
                cols.append((float(f), None, True))
            else:     # a host array: not cacheable, as in rhs / backsolve
                cols.append((1.0, self._vec(self.from_host(f), "f", self.n_nodes), False))
        if not cols:
            raise ValueError("a block of loads needs at least one column")
        return cols, None

    def _block_groups(self, cols):
        """Column index lists, each taking one path.  With W kept, the columns whose interior
        solution the single path caches (CUDA and scalar loads) are split from the others
        (host arrays), so that each column's load and back-solve use the single path's
        kernels."""
        k = len(cols)
        if getattr(self, "_W", None) is None:
            return [(False, list(range(k)))]
        hit = [j for j in range(k) if cols[j][2]]
        miss = [j for j in range(k) if not cols[j][2]]
        return [(cached, g) for cached, g in ((True, hit), (False, miss)) if g]

    def _chunk_load(self, cols, idx, block):
        """(F, ldf, nodal mask, f_scale ctypes array) of the columns ``idx``."""
        sub = [cols[j] for j in idx]
        mask = 0
        for q, (_, t, _) in enumerate(sub):
            if t is not None:
                mask |= 1 << q
        scales = (C.c_double * len(sub))(*[s for s, _, _ in sub])
        if not mask:
            return None, 0, 0, scales
        if len(sub) == 1:
            return sub[0][1], self.n_nodes, mask, scales
        if block is not None and idx == list(range(idx[0], idx[0] + len(idx))):
            return block[idx[0]:idx[0] + len(idx)], block.stride(0), mask, scales
        Fs = torch.empty((len(sub), self.n_nodes), dtype=torch.float64, device=self.dev)
        for q, (_, t, _) in enumerate(sub):
            if t is not None:
                Fs[q].copy_(t)
        return Fs, self.n_nodes, mask, scales

    def _element_block(self, mode, load, g_loc=None, c=None, U=None):
        """One launch of sc_element_block_kernel (csrc/semk_sc.cu)."""
        F, ldf, mask, scales = load
        self._bad.zero_()
        _lib.check(self._lib.semk_sc_element_block_f64(
            self.n1, self.n_elem, device.ptr(self.G), self.g_stride, 1,
            device.ptr(self.tab.dev()[0]), device.ptr(self._t["ext_loc"]),
            device.ptr(self.l2g_dev), device.ptr(self.JxW), device.ptr(self._react), int(mode),
            len(scales), device.ptr(F), int(ldf), mask, scales, device.ptr(g_loc),
            self.n_elem * self.n_ext_loc, device.ptr(c), self.n_elem * self.n_int_loc,
            device.ptr(U), 0 if U is None else U.stride(0), device.ptr(self._bad),
            device.stream_ptr()))
        if int(self._bad.item()) != 0:
            raise AssertionError("an element-interior stiffness block is not positive definite")

    def _block_rhs(self, cols, block, keep_c):
        """Element-local condensed loads, chunk by chunk: yields (column ids, g_loc [kc, E, 4p],
        c [kc, E, (p-1)^2] = A_ii^-1 f_i or None, load descriptor).  ``keep_c``: compute c where
        the single path would cache it (W kept, cacheable load)."""
        f64 = dict(dtype=torch.float64, device=self.dev)
        stored_load = self._Ainv is not None      # kept with W only
        for cacheable, group in self._block_groups(cols):
            for j0, j1 in self._block_chunks(len(group)):
                idx = group[j0:j1]
                kc = len(idx)
                load = self._chunk_load(cols, idx, block)
                F, ldf, mask, scales = load
                g_loc = torch.empty((kc, self.n_elem, self.n_ext_loc), **f64)
                c = None
                if cacheable and (keep_c or stored_load):
                    c = torch.empty((kc, self.n_elem, self.n_int_loc), **f64)
                if cacheable and stored_load:
                    _lib.check(self._lib.semk_sc_load_stored_block_f64(
                        self.n1, self.n_elem, device.ptr(self._W), device.ptr(self._Ainv),
                        device.ptr(self.l2g_dev), device.ptr(self._t["ext_loc"]),
                        device.ptr(self.JxW), kc, device.ptr(F), int(ldf), mask, scales,
                        device.ptr(g_loc), self.n_elem * self.n_ext_loc, device.ptr(c),
                        self.n_elem * self.n_int_loc, device.stream_ptr()))
                else:
                    self._element_block(_lib.SC_RHS, load, g_loc=g_loc, c=c)
                yield idx, g_loc, (c if keep_c else None), load

    def _block_backsolve(self, X, idx, load, c, U):
        """Rows ``idx`` of the nodal block U from the exterior solutions X [kc, n_ext]: the
        stream over W with the loads' c, else the element pass on the loads."""
        contiguous = idx == list(range(idx[0], idx[0] + len(idx)))
        Ub = U[idx[0]:idx[0] + len(idx)] if contiguous else torch.empty(
            (len(idx), self.n_nodes), dtype=torch.float64, device=self.dev)
        Ub[:, :self.n_ext].copy_(X)
        if c is not None:
            _lib.check(self._lib.semk_sc_backsolve_stored_block_f64(
                self.n1, self.n_elem, device.ptr(self._W), device.ptr(c),
                self.n_elem * self.n_int_loc, device.ptr(self.l2g_dev),
                device.ptr(self._t["ext_loc"]), len(idx), device.ptr(Ub), Ub.stride(0),
                device.stream_ptr()))
        else:
            self._element_block(_lib.SC_BACKSOLVE, load, U=Ub)
        if not contiguous:
            for q, j in enumerate(idx):
                U[j].copy_(Ub[q])

    def _block_out(self, out, k, n, what="out"):
        if out is None:
            return torch.empty((k, n), dtype=torch.float64, device=self.dev)
        if not (isinstance(out, torch.Tensor) and out.is_cuda and out.dtype == torch.float64
                and tuple(out.shape) == (k, n) and out.stride(1) == 1):
            raise ValueError("%s must be a float64 CUDA [%d, %d] block with contiguous rows"
                             % (what, k, n))
        return out

    def _block_vectors(self, X, k, n, what):
        """Rows of a [k, n] CUDA block or a sequence of k vectors of length n."""
        rows = list(X) if not isinstance(X, torch.Tensor) or X.dim() == 2 else None
        if rows is None or len(rows) != k:
            raise ValueError("%s must be a [%d, %d] block or %d vectors" % (what, k, n, k))
        return [self._vec(r, what, n) for r in rows]

    def rhs_many(self, F):
        """Condensed loads of a block of loads, ``[k, n_ext]``: row j is ``rhs(F[j])``.
        ``F``: a float64 CUDA ``[k, n_nodes]`` block or a sequence of loads in any form
        ``rhs`` accepts."""
        cols, block = self._block_loads(F)
        out = torch.empty((len(cols), self.n_ext), dtype=torch.float64, device=self.dev)
        for idx, g_loc, _, _ in self._block_rhs(cols, block, keep_c=False):
            for q, j in enumerate(idx):
                self.assemble(g_loc[q], out=out[j])
        return out

    def backsolve_many(self, X_ext, F, out=None):
        """Full nodal vectors ``[k, n_nodes]`` from exterior solutions ``X_ext`` ([k, n_ext] or
        k vectors) and their loads ``F``: row j is ``backsolve(X_ext[j], F[j])`` when that call
        does not find the load in the single-load cache (the interiors are recomputed)."""
        cols, block = self._block_loads(F)
        k = len(cols)
        X = self._block_vectors(X_ext, k, self.n_ext, "X_ext")
        U = self._block_out(out, k, self.n_nodes)
        for j0, j1 in self._block_chunks(k):
            idx = list(range(j0, j1))
            Xc = torch.stack(X[j0:j1])
            self._block_backsolve(Xc, idx, self._chunk_load(cols, idx, block), None, U)
        return U

    def _solve_block(self, cols, block, out, condensed_rhs, pcg):
        """Shared loop of solve_many / solve_load_many: per chunk the block load pass, per
        column ``condensed_rhs(j, g)`` and ``pcg(j, b)``, then the block back-solve."""
        k = len(cols)
        U = self._block_out(out, k, self.n_nodes)
        infos = [None] * k
        for idx, g_loc, c, load in self._block_rhs(cols, block, keep_c=True):
            X = torch.empty((len(idx), self.n_ext), dtype=torch.float64, device=self.dev)
            for q, j in enumerate(idx):
                x, infos[j] = pcg(j, condensed_rhs(j, self.assemble(g_loc[q])))
                X[q].copy_(x)
            del g_loc
            self._block_backsolve(X, idx, load, c, U)
        return U, infos

    def solve_many(self, F, dirichlet_values=None, flux=None, **pcg_kwargs):
        """``solve`` for a block of loads: returns (U [k, n_nodes], [PCGInfo] * k), row j
        bitwise ``solve(F[j], ...)``.  ``F`` as in ``rhs_many``; ``dirichlet_values`` and
        ``flux`` are one value for every column or a list of k.  PCG runs column by column."""
        cols, block = self._block_loads(F)
        k = len(cols)

        def per_column(v, what):
            if isinstance(v, (list, tuple)):
                if len(v) != k:
                    raise ValueError("%s: a list must have one entry per load (%d)" % (what, k))
                return list(v)
            return [v] * k

        dv = per_column(dirichlet_values, "dirichlet_values")
        fl = per_column(flux, "flux")

        def condensed_rhs(j, b):
            for name, g in (fl[j] or {}).items():
                b += self.boundary_load(name, g)
            return self.lift(b, dv[j])

        return self._solve_block(cols, block, None, condensed_rhs,
                                 lambda j, b: self.solve_pcg(b, **pcg_kwargs))

    def solve_load_many(self, R, F, rtol=1e-8, preconditioner="three-level", out=None):
        """``solve_load`` for a block: R and F are [k, n_nodes] blocks or sequences of k nodal
        CUDA vectors; returns (U [k, n_nodes] or ``out``, [PCGInfo] * k), row j bitwise
        ``solve_load(R[j], F[j], rtol, preconditioner)``."""
        cols, block = self._block_loads(F)
        R = self._block_vectors(R, len(cols), self.n_nodes, "R")
        mask = device.ptr(self.dirichlet_dev) if self.has_dirichlet else None

        def condensed_rhs(j, g):
            b = torch.empty_like(g)
            _lib.check(self._lib.semk_sc_rhs_finish_f64(
                self.n_ext, device.ptr(g), device.ptr(R[j]), mask, device.ptr(b),
                device.stream_ptr()))
            return b

        return self._solve_block(cols, block, out, condensed_rhs,
                                 lambda j, b: self.solve_pcg(b, rtol=rtol,
                                                             preconditioner=preconditioner))


def block_chunks(k, cap, bytes_per_col, free_bytes):
    """Column ranges ``[(j0, j1)]`` of a block of ``k`` loads: at most ``cap`` columns each,
    fewer when ``free_bytes`` would not hold ``bytes_per_col`` per column, at least one."""
    k, cap = int(k), int(cap)
    if k < 1 or cap < 1:
        raise ValueError("a block needs k >= 1 columns and a cap >= 1")
    width = max(1, min(cap, int(free_bytes) // max(int(bytes_per_col), 1)))
    return [(j0, min(j0 + width, k)) for j0 in range(0, k, width)]


class CondensedLocalSystems(CondensedPoissonOperator):
    """Static condensation of the CALLER'S OWN dense local systems: the literal
    inputs of ``DOFManagerSC.assemble_global_sc_system`` / ``solve``
    (sem/discrete.py:478-528) -- per element a symmetric local matrix and
    right-hand side in hierarchical local order (``reorder_local_system_hier``,
    :428-436) -- condensed, solved (PCG on the exterior DOFs) and back-substituted
    on the device.  Interior blocks must be positive definite (Cholesky).

        cs = CondensedLocalSystems(dof_mngr, lmats_h[E, NN, NN], lrhs_h[E, NN], dirichlet=on_ebc)
        u, info = cs.solve(dirichlet_values)
    """

    def __init__(self, dof_mngr, lmats_h, lrhs_h, dirichlet=None, symmetry_rtol=1e-10):
        self._init_common(dof_mngr, dirichlet)
        NN = self.n1 * self.n1
        lmats_h = np.asarray(lmats_h, dtype=np.float64)
        lrhs_h = np.asarray(lrhs_h, dtype=np.float64)
        if lmats_h.shape != (self.n_elem, NN, NN) or lrhs_h.shape != (self.n_elem, NN):
            raise ValueError("local systems must be [n_cells, NN, NN] matrices and [n_cells, NN] "
                             "right-hand sides in hierarchical local order")
        scale = np.abs(lmats_h).max()
        if np.abs(lmats_h - np.swapaxes(lmats_h, 1, 2)).max() > symmetry_rtol * max(scale, 1e-300):
            raise NotImplementedError("the device static condensation needs symmetric local "
                                      "matrices (Cholesky of the interior blocks)")
        geo = dof_mngr.mesh.get_geometries()[0]
        hier = np.asarray(geo.hierarchical_node_order, dtype=np.int64)
        l2g = dof_mngr.mesh.node_map_array().reshape(-1, NN)
        self._A = device._f64(lmats_h, self.dev)
        self._f = device._f64(lrhs_h, self.dev)
        self._l2g_hier = device.as_i32_bits(np.ascontiguousarray(l2g[:, hier]), self.dev)
        self._schur_pass()

    def _element_pass(self, mode, S=None, sdiag_loc=None, g_loc=None, u=None, W=None, Ainv=None):
        """One launch of the element kernel on the local systems (W and Ainv are never kept)."""
        self._bad.zero_()
        _lib.check(self._lib.semk_sc_element_dense_f64(
            self.n1, self.n_elem, device.ptr(self._A), device.ptr(self._f),
            device.ptr(self._l2g_hier), int(mode), device.ptr(S), self.s_stride,
            device.ptr(sdiag_loc), device.ptr(g_loc), device.ptr(u), device.ptr(self._bad),
            device.stream_ptr()))
        if int(self._bad.item()) != 0:
            raise AssertionError("an element-interior block is not positive definite")

    def rhs(self, f=None):
        """Condensed load of the caller's local right-hand sides."""
        g_loc = torch.empty((self.n_elem, self.n_ext_loc), dtype=torch.float64, device=self.dev)
        self._element_pass(_lib.SC_RHS, g_loc=g_loc)
        return self.assemble(g_loc)

    def backsolve(self, x_ext, f=None, out=None):
        self._vec(x_ext, "x_ext")
        u = (torch.empty(self.n_nodes, dtype=torch.float64, device=self.dev) if out is None
             else self._vec(out, "out", self.n_nodes))
        u[:self.n_ext].copy_(x_ext)
        self._element_pass(_lib.SC_BACKSOLVE, u=u)
        return u

    def solve(self, dirichlet_values=None, **pcg_kwargs):
        b = self.lift(self.rhs(), dirichlet_values)
        x, info = self.solve_pcg(b, **pcg_kwargs)
        return self.backsolve(x), info

    def _no_blocks(self, *args, **kwargs):
        raise NotImplementedError("CondensedLocalSystems holds one load (the caller's local "
                                  "right-hand sides); blocks of loads are not supported")

    rhs_many = backsolve_many = solve_many = solve_load_many = _no_blocks


def coarse_tables(l2g_ext, node_ptr, node_pos, dirichlet, gll_nodes):
    """Host tables of the vertex coarse space of the two-level preconditioner
    (additive API, no reference equivalent: the reference solves the condensed
    system directly, sem/discrete.py:511).

    Coarse DOFs = the distinct element vertices (compact index 0..n_v-1).  The
    prolongation P interpolates LINEARLY ALONG ELEMENT EDGES: an exterior node
    at GLL position t on an edge gets (1 - t) and t from the edge's two end
    vertices, a vertex node gets its own coarse value -- at most two weights
    per row (``pv``, ``pw``), taken from the first element that contains the
    node.  Rows of Dirichlet nodes and weights on Dirichlet vertices are zero,
    so the coarse space vanishes on the essential boundary.

    Returns a dict: ``phi[4p, 4]`` (the local interpolation matrix in the
    hierarchical exterior order), ``vert_c[E, 4]`` compact vertex ids of every
    element, ``n_v``, ``dirichlet_c[n_v]``, ``pv[n_ext, 2]`` / ``pw[n_ext, 2]``
    (prolongation), ``rptr / ridx / rw`` (CSR of the transpose: restriction),
    ``vptr / vpos`` (vertex -> element-local entries ``e * 4 + a``, ascending:
    assembly order of the coarse operator)."""
    l2g_ext = np.asarray(l2g_ext)
    E, NE = l2g_ext.shape
    p = NE // 4
    N = p + 1
    n_ext = int(node_ptr.size - 1)
    t = (1.0 + np.asarray(gll_nodes, dtype=np.float64)) / 2.0
    if t.size != N:
        raise ValueError("gll_nodes must have p + 1 entries")
    va = np.zeros(NE, dtype=np.int64)
    vb = np.zeros(NE, dtype=np.int64)
    wa = np.zeros(NE)
    wb = np.zeros(NE)
    va[:4] = vb[:4] = np.arange(4)
    wa[:4] = 1.0
    inner = np.arange(1, N - 1)
    # hierarchical exterior order (sem/geometry.py:151-212): vertices (0,0), (0,N-1), (N-1,0),
    # (N-1,N-1); then the open edges m = 0, m = N-1 (running along n), n = 0, n = N-1 (along m)
    for edge, (a, b) in enumerate(((0, 1), (2, 3), (0, 2), (1, 3))):
        k = 4 + edge * (N - 2) + np.arange(N - 2)
        va[k], vb[k] = a, b
        wa[k], wb[k] = 1.0 - t[inner], t[inner]
    phi = np.zeros((NE, 4))
    phi[np.arange(NE), va] += wa
    phi[np.arange(NE), vb] += wb
    vert = l2g_ext[:, :4].astype(np.int64)
    vids = np.unique(vert)
    n_v = int(vids.size)
    vmap = np.full(n_ext, -1, dtype=np.int64)
    vmap[vids] = np.arange(n_v)
    vert_c = vmap[vert]
    dirichlet = (np.zeros(n_ext, dtype=bool) if dirichlet is None
                 else np.asarray(dirichlet, dtype=bool)[:n_ext])
    dirichlet_c = dirichlet[vids]
    first = node_pos[node_ptr[:-1].astype(np.int64)].astype(np.int64)
    e, k = np.divmod(first, NE)
    pv = np.stack([vert_c[e, va[k]], vert_c[e, vb[k]]], axis=1)
    pw = np.stack([wa[k], wb[k]], axis=1)
    pw[dirichlet] = 0.0
    pw[dirichlet_c[pv]] = 0.0
    flat_v, flat_w = pv.ravel(), pw.ravel()
    flat_g = np.repeat(np.arange(n_ext, dtype=np.int64), 2)
    keep = flat_w != 0.0
    order = np.argsort(flat_v[keep], kind="stable")
    ridx = flat_g[keep][order].astype(np.uint32)
    rw = np.ascontiguousarray(flat_w[keep][order])
    rptr = np.zeros(n_v + 1, dtype=np.uint32)
    np.cumsum(np.bincount(flat_v[keep], minlength=n_v), out=rptr[1:])
    vflat = vert_c.ravel()
    vpos = np.argsort(vflat, kind="stable").astype(np.uint32)
    vptr = np.zeros(n_v + 1, dtype=np.uint32)
    np.cumsum(np.bincount(vflat, minlength=n_v), out=vptr[1:])
    return dict(phi=phi, vert_c=vert_c.astype(np.uint32), n_v=n_v, dirichlet_c=dirichlet_c,
                pv=pv.astype(np.uint32), pw=np.ascontiguousarray(pw), rptr=rptr, ridx=ridx, rw=rw,
                vptr=vptr, vpos=vpos)


def element_tiles(mesh, n_elem, max_tiles=4096):
    """Tile id of every element for the aggregation level of the three-level
    preconditioner: k x k blocks of a structured mesh, runs of k^2 elements along a
    Morton curve through the centroids otherwise; k is the smallest that gives at
    most ``max_tiles`` tiles (the top level is inverted densely)."""
    shape = getattr(mesh, "_structured_shape", None)
    if shape is not None and shape[0] * shape[1] == n_elem:
        nx, ny = shape
        k = 1
        while -(-nx // k) * -(-ny // k) > max_tiles:
            k += 1
        k = max(k, min(4, max(nx, ny)))
        ex, ey = np.divmod(np.arange(n_elem, dtype=np.int64), ny)
        return (ex // k) * (-(-ny // k)) + ey // k
    from .operators import _morton_order
    if not hasattr(mesh, "_centroids"):
        mesh._compute_cell_centroids()
    order = _morton_order(mesh._centroids[:, 0], mesh._centroids[:, 1])
    per = max(16, -(-n_elem // max_tiles))
    tile = np.empty(n_elem, dtype=np.int64)
    tile[order] = np.arange(n_elem, dtype=np.int64) // per
    return tile


def aggregate_tables(vert_c, vptr, vpos, dirichlet_c, tile):
    """Piecewise-constant aggregation of the coarse (vertex) DOFs: a vertex joins the
    tile of the first element that contains it; vertices on the essential boundary
    join nothing.  Returns ``agg[n_v]`` (uint32, 0xffffffff = none), ``n_agg`` and the
    CSR ``aptr / aidx`` of the vertices of every aggregate."""
    n_v = int(vptr.size - 1)
    first_elem = vpos[vptr[:-1].astype(np.int64)].astype(np.int64) // 4
    free = ~np.asarray(dirichlet_c, dtype=bool)
    raw = np.asarray(tile, dtype=np.int64)[first_elem]
    uniq, inv = np.unique(raw[free], return_inverse=True)
    n_agg = int(uniq.size)
    agg = np.full(n_v, 0xFFFFFFFF, dtype=np.uint32)
    agg[free] = inv.astype(np.uint32)
    free_ids = np.flatnonzero(free)
    order = np.argsort(inv, kind="stable")
    aidx = free_ids[order].astype(np.uint32)
    aptr = np.zeros(n_agg + 1, dtype=np.uint32)
    np.cumsum(np.bincount(inv, minlength=n_agg), out=aptr[1:])
    return dict(agg=agg, n_agg=n_agg, aptr=aptr, aidx=aidx)


def aggregate_csr(agg, n_agg, n_limit):
    """CSR (aptr, aidx) of the vertices ``v < n_limit`` of every aggregate, ascending."""
    agg = np.asarray(agg, dtype=np.uint32)[:int(n_limit)]
    ids = np.flatnonzero(agg != 0xFFFFFFFF)
    a = agg[ids].astype(np.int64)
    order = np.argsort(a, kind="stable")
    aidx = ids[order].astype(np.uint32)
    aptr = np.zeros(int(n_agg) + 1, dtype=np.uint32)
    np.cumsum(np.bincount(a, minlength=int(n_agg)), out=aptr[1:])
    return aptr, aidx


def top_level_inverse(Ace, vert_c, agg, n_agg):
    """Dense inverse of the third-level operator P2^T Ac P2 from the element coarse
    matrices on the HOST (the NumPy emulation in tests/test_two_level_host.py; the product
    assembles and inverts it on the device, CondensedPoissonOperator._build_top)."""
    from scipy import sparse
    a = agg.astype(np.int64)[np.asarray(vert_c, dtype=np.int64)]          # [E, 4]
    a[a == 0xFFFFFFFF] = -1
    rows = np.repeat(a, 4, axis=1).ravel()
    cols = np.tile(a, (1, 4)).ravel()
    vals = np.asarray(Ace, dtype=np.float64).reshape(-1)
    ok = (rows >= 0) & (cols >= 0)
    A3 = sparse.coo_matrix((vals[ok], (rows[ok], cols[ok])), shape=(n_agg, n_agg)).toarray()
    A3 = 0.5 * (A3 + A3.T)
    inv = np.linalg.inv(A3)
    if not np.isfinite(inv).all():
        raise AssertionError("the aggregated coarse operator is singular")
    return np.ascontiguousarray(0.5 * (inv + inv.T))
