"""Thin torch <-> libsemk glue: device tensors in, C-ABI kernel launches out.

PyTorch is only the carrier of device memory and streams here; every number is
produced by the hand-written sm_100a kernels in csrc/.  All functions raise if
no CUDA device is present -- there is no CPU fallback.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib

__all__ = ["stream_ptr", "as_i32_bits", "basis_tables", "element_geometry", "ptr",
           "boundary_face_tables", "csr_by_key", "BoundaryFaces", "winner_table",
           "node_entries_csr", "field_grad"]


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device (or host) address of a tensor / numpy array, or NULL for None."""
    if t is None:
        return None
    if isinstance(t, np.ndarray):
        return C.c_void_p(t.ctypes.data)
    return C.c_void_p(t.data_ptr())


def as_i32_bits(a, device="cuda"):
    """uint32 numpy array -> int32 torch tensor with the same bits (torch has
    no arithmetic on uint32; the kernels reinterpret)."""
    a = np.ascontiguousarray(a, dtype=np.uint32)
    return torch.from_numpy(a.view(np.int32)).to(device)


def _f64(a, device="cuda"):
    if isinstance(a, torch.Tensor):
        return a.to(device=device, dtype=torch.float64).contiguous()
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(device)


class BasisTables(object):
    """Device copies of the 1-D tables the kernels need for one tensor basis."""

    def __init__(self, basis):
        subs = [b for _, b in basis.iter_subbases()]
        if basis.ndim != 2 or len(subs) != 2:
            raise NotImplementedError("Only supporting 2D elements right now")
        b0, b1 = subs
        if b0.n_coeffs != b1.n_coeffs or not (np.array_equal(b0.D1, b1.D1)
                                              and np.array_equal(b0.nodes, b1.nodes)):
            raise NotImplementedError("the engine needs the same 1-D basis in both directions")
        self.n1 = int(b0.n_coeffs)
        if self.n1 < 2 or self.n1 > _lib.MAX_N1:
            raise NotImplementedError("Basis only available up to order %d." % (_lib.MAX_N1 - 1))
        self.D_host = np.ascontiguousarray(b0.D1, dtype=np.float64)
        self.Einv_host = np.ascontiguousarray(b0.interp_eq_inv, dtype=np.float64)
        self.w_host = np.ascontiguousarray(b0.quad_rule.weights, dtype=np.float64)
        self._dev = None

    def dev(self):
        if self._dev is None:
            self._dev = (_f64(self.D_host), _f64(self.Einv_host), _f64(self.w_host))
        return self._dev


def basis_tables(basis):
    tab = getattr(basis, "_semk_tables", None)
    if tab is None:
        tab = BasisTables(basis)
        basis._semk_tables = tab
    return tab


def geom_factors(tab, nodes_dev, l2g_dev, n_elem, elem_of_slot=None, G=None, g_patch_stride=0,
                 elems_per_patch=1, JxW=None, x_phys=None, J=None, invJ=None, detJ=None,
                 check=True):
    """Launch K1 (csrc/semk_geom.cu).  Raises AssertionError on a non-positive
    Jacobian, like the reference's ``assert np.all(det_jacobian > 0)``
    (sem/mapping.py:117)."""
    lib = _lib.load()
    D, Einv, w = tab.dev()
    bad = torch.zeros(1, dtype=torch.int32, device=nodes_dev.device)
    _lib.check(lib.semk_geom_factors_f64(
        tab.n1, int(n_elem), ptr(nodes_dev[0]), ptr(nodes_dev[1]), ptr(l2g_dev), ptr(Einv),
        ptr(D), ptr(w), ptr(elem_of_slot), ptr(G), int(g_patch_stride), int(elems_per_patch),
        ptr(JxW), ptr(x_phys), ptr(J), ptr(invJ), ptr(detJ), ptr(bad), stream_ptr()))
    if check and int(bad.item()) != 0:
        raise AssertionError("non-positive Jacobian determinant in the mesh")


def field_grad(tab, nodes_dev, l2g_dev, n_elem, n_nodes, elems=None, u=None, winner=None,
               xy=None, grad_loc=None, weighted=False, jxw_loc=None, u_ref=None, g_ref=None,
               sums=None, partials=None):
    """Launch the nodal-field kernel (csrc/semk_geom.cu, semk_field_grad_f64): K1's geometry
    again, then the gradient of ``u`` and whichever outputs are given.  Raises AssertionError
    on a non-positive Jacobian, like ``geom_factors``."""
    lib = _lib.load()
    D, Einv, w = tab.dev()
    bad = torch.zeros(1, dtype=torch.int32, device=nodes_dev.device)
    _lib.check(lib.semk_field_grad_f64(
        tab.n1, int(n_elem), ptr(nodes_dev[0]), ptr(nodes_dev[1]), ptr(l2g_dev), ptr(Einv),
        ptr(D), ptr(w), ptr(elems), int(n_nodes), ptr(u), ptr(winner), ptr(xy), ptr(grad_loc),
        int(bool(weighted)), ptr(jxw_loc), ptr(u_ref), ptr(g_ref), ptr(sums), ptr(partials),
        ptr(bad), stream_ptr()))
    if int(bad.item()) != 0:
        raise AssertionError("non-positive Jacobian determinant in the mesh")


def winner_table(l2g, n_nodes):
    """``uint8`` per entry of the L2G map (any shape, flat order): 1 where the entry is the
    last one naming its node -- the element whose value the reference's element loop keeps
    (fancy assignment keeps the last value for repeated indices).  Pure NumPy."""
    flat = np.asarray(l2g).ravel()
    last = np.empty(int(n_nodes), dtype=np.int64)
    last[flat] = np.arange(flat.size, dtype=np.int64)
    return (last[flat] == np.arange(flat.size, dtype=np.int64)).astype(np.uint8)


def node_entries_csr(l2g_t, n_nodes):
    """Node -> entries CSR of the whole L2G map: ``pos[ptr[j]:ptr[j+1]]`` the flat entries
    ``e * NN + k`` naming node j, ascending (a stable sort: the order of ``csr_by_key``, and
    the fixed order in which ``semk_face_sum_f64`` sums element-local values onto nodes).
    ``l2g_t``: int32-bit-pattern tensor [E, NN] on any device; returns int32-bit-pattern
    tensors (ptr [n_nodes + 1], pos [E * NN]) on that device."""
    flat = l2g_t.reshape(-1).to(torch.int64) & 0xFFFFFFFF
    if flat.numel() >= 2 ** 31:
        raise NotImplementedError("more than 2^31 L2G entries")
    pos = torch.sort(flat, stable=True).indices.to(torch.int32)
    ptr_ = torch.zeros(int(n_nodes) + 1, dtype=torch.int64, device=flat.device)
    torch.cumsum(torch.bincount(flat, minlength=int(n_nodes)), 0, out=ptr_[1:])
    return ptr_.to(torch.int32), pos


def stiffness_factors(tab, mesh, l2g_dev, n_slots, G, g_stride, elems_per_patch, JxW,
                      elem_of_slot=None, geometric_factors=None, weight=None):
    """Geometric factors of the stiffness into ``G`` (engine layout: ``n_slots`` slots,
    ``elems_per_patch`` per row of stride ``g_stride``; ``elem_of_slot`` maps slot -> element,
    None = the identity) and the quadrature weights into ``JxW[E, NN]``: from the mesh nodes
    by K1, or from the caller's ``geometric_factors = (invJ[E,2,2,N,N], JxW[E,N,N])``.
    ``weight`` makes it the stiffness of -div(w grad u): nodal values [E, N, N], or a callable
    w(x, y) of the physical coordinates (needs the device geometry)."""
    if callable(weight) and geometric_factors is not None:
        raise ValueError("a callable weight needs the device geometry (geometric_factors=None)")
    lib = _lib.load()
    n1 = tab.n1
    n_elem, NN = JxW.shape
    dev = G.device
    x_phys = None
    if geometric_factors is None:
        nodes_dev = torch.from_numpy(np.ascontiguousarray(mesh.nodes, dtype=np.float64)).to(dev)
        if nodes_dev.shape[0] != 2:
            raise NotImplementedError("Only supporting 2D elements right now")
        if callable(weight):
            x_phys = torch.empty((n_elem, 2, NN), dtype=torch.float64, device=dev)
        geom_factors(tab, nodes_dev, l2g_dev, n_slots, elem_of_slot=elem_of_slot, G=G,
                     g_patch_stride=g_stride, elems_per_patch=elems_per_patch, JxW=JxW,
                     x_phys=x_phys)
        del nodes_dev
    else:
        invJ, jxw = geometric_factors
        invJ = _f64(np.asarray(invJ).reshape(n_elem, 4, NN), dev)
        JxW.copy_(_f64(np.asarray(jxw).reshape(n_elem, NN), dev))
        _lib.check(lib.semk_gfactors_from_invj_f64(
            n1, n_slots, ptr(invJ), ptr(JxW), ptr(elem_of_slot), ptr(G), g_stride,
            elems_per_patch, stream_ptr()))
        torch.cuda.current_stream().synchronize()
        del invJ
    if weight is None:
        return
    # scale the geometric factors node by node (the rho_JxW einsums of
    # examples/squirmer-axisymmetric.py:194-213 with w = x_phys[0])
    if callable(weight):
        w = weight(x_phys[:, 0, :], x_phys[:, 1, :])
        w = torch.as_tensor(w, dtype=torch.float64, device=dev).expand(n_elem, NN)
    else:
        w = _f64(np.asarray(weight, dtype=np.float64).reshape(n_elem, NN), dev)
    w = w.contiguous()
    _lib.check(lib.semk_scale_gfactors_f64(
        n1, n_slots, ptr(w), ptr(elem_of_slot), ptr(G), g_stride, elems_per_patch,
        stream_ptr()))
    torch.cuda.current_stream().synchronize()


def boundary_face_tables(mesh, name):
    """Faces of the named boundary, in the order ``DOFManager.boundary_elements(name)`` visits
    them (cells ascending, the faces of a cell in registration order).  Pure NumPy.

    Returns ``cells[F]``, ``faces[F]`` (0:W 1:E 2:S 3:N), and per face ``nodes[F, n1]`` (uint32
    node ids) and ``local[F, n1]`` (element-local lexicographic indices) of its GLL nodes in the
    reference orientation of ``mapping._subface_slice`` (faces 0 and 3 reversed).  An unknown
    name raises the ``KeyError`` of ``boundary_elements``."""
    from .mapping import _subface_slice
    bnd_id = mesh._boundary_id_lookup[name]
    maps = mesh.node_map_array()
    if maps.ndim != 3 or maps.shape[1] != maps.shape[2]:
        raise NotImplementedError("boundary tables need 2-D cells with the same order in both "
                                  "directions")
    n1 = int(maps.shape[1])
    pairs = sorted(mesh._boundary_faces[bnd_id], key=lambda cf: cf[0])      # stable
    cells = np.array([c for c, _ in pairs], dtype=np.int64)
    faces = np.array([f for _, f in pairs], dtype=np.int64)
    lin = np.arange(n1 * n1, dtype=np.int64).reshape(n1, n1)
    local = np.empty((cells.size, n1), dtype=np.int64)
    for f in range(4):
        local[faces == f] = _subface_slice(f, lin, 2)
    nodes = maps.reshape(-1, n1 * n1)[cells[:, None], local]
    return cells, faces, np.ascontiguousarray(nodes, dtype=np.uint32), local


def csr_by_key(keys):
    """Group the entries of ``keys`` (any shape; entry i is ``keys.ravel()[i]``) by value:
    ``uniq`` ascending, and ``pos[ptr[j]:ptr[j+1]]`` the flat positions of the entries equal to
    ``uniq[j]``, ascending.  Pure NumPy.  That is the fixed summation order in which
    ``semk_face_sum_f64`` adds face-node entries onto nodes."""
    flat = np.asarray(keys).ravel()
    if flat.size >= 2 ** 32:
        raise NotImplementedError("more than 2^32 face-node entries")
    pos = np.argsort(flat, kind="stable").astype(np.uint32)
    uniq, counts = np.unique(flat, return_counts=True)
    ptr = np.zeros(uniq.size + 1, dtype=np.uint32)
    np.cumsum(counts, out=ptr[1:])
    return uniq, ptr, pos


class BoundaryFaces(object):
    """Face tables of one named boundary on the device (``boundary_face_tables``), with:

    * ``x [F, 2, n1]``: physical coordinates of the face nodes, and ``dSxW [F, n1]``: the face's
      GLL weight times ``|dx/dxi_t|`` -- the host mirror's ``SubFiniteElement.x_phys`` /
      ``dSxW``; ``n_dSxW [F, 2, n1]``: the outward normal times ``dSxW``
      (``SubFiniteElement.n_dSxW``, the normal of ``SubMapping._compute_normal_vec``).  K1
      runs on the boundary cells only (as ``DOFManager.boundary_elements`` does) and the face
      slice and the tangent length follow ``SubMapping._tangents``.
    * ``nodes``: the distinct boundary nodes, ascending, and ``keys``: the distinct
      element-local slots ``cell * NN + local`` of the face nodes; ``face_sum`` adds
      face-node values ``[F, n1]`` onto either in a fixed order (``csr_by_key``)."""

    def __init__(self, tab, mesh, name, dev):
        n1, NN = tab.n1, tab.n1 * tab.n1
        self.name = name
        self.cells, self.faces, self.node_ids, self.local = boundary_face_tables(mesh, name)
        if self.node_ids.shape[1] != n1:
            raise ValueError("the mesh and the basis have different orders")
        F = self.n_faces = int(self.cells.size)
        self.dev = dev
        self.nodes, ptr, pos = csr_by_key(self.node_ids)
        self.n = int(self.nodes.size)
        self._csr = {"nodes": (self.n, as_i32_bits(ptr, dev), as_i32_bits(pos, dev))}
        keys, kptr, kpos = csr_by_key(self.cells[:, None] * NN + self.local)
        self.keys = keys
        self._csr["local"] = (int(keys.size), as_i32_bits(kptr, dev), as_i32_bits(kpos, dev))
        self.nodes_dev = torch.from_numpy(self.nodes.astype(np.int64)).to(dev)
        self.keys_dev = torch.from_numpy(keys.astype(np.int64)).to(dev)
        self.node_ids_dev = torch.from_numpy(self.node_ids.astype(np.int64)).to(dev)
        f64 = dict(dtype=torch.float64, device=dev)
        self.x = torch.empty((F, 2, n1), **f64)
        self.dSxW = torch.empty((F, n1), **f64)
        self.n_dSxW = torch.empty((F, 2, n1), **f64)
        if F == 0:
            return
        l2g = as_i32_bits(mesh.node_map_array().reshape(-1, NN)[self.cells], dev)
        nodes_dev = torch.from_numpy(np.ascontiguousarray(mesh.nodes, dtype=np.float64)).to(dev)
        x_phys = torch.empty((F, 2, NN), **f64)
        J = torch.empty((F, 2, 2, NN), **f64)
        geom_factors(tab, nodes_dev, l2g, F, x_phys=x_phys, J=J)
        loc = torch.from_numpy(self.local).to(dev)[:, None, :].expand(F, 2, n1)
        self.x.copy_(torch.gather(x_phys, 2, loc))
        # the face runs along parametric direction 1 - face // 2: that column of J is the
        # (unnormalised) tangent
        along = torch.from_numpy(1 - self.faces // 2).to(dev)
        tan = torch.gather(J[torch.arange(F, device=dev), :, along, :], 2, loc)
        dS = torch.sqrt(tan[:, 0] * tan[:, 0] + tan[:, 1] * tan[:, 1])
        w = _f64(tab.w_host, dev)[None, :]
        self.dSxW.copy_(dS * w)
        # counter-clockwise tangent (faces 0 and 3 run against the parametric direction),
        # turned clockwise: (t_y, -t_x) points out of the cell
        sgn = torch.from_numpy(np.where((self.faces == 0) | (self.faces == 3), -1.0, 1.0)).to(dev)
        self.n_dSxW[:, 0].copy_(sgn[:, None] * tan[:, 1] * w)
        self.n_dSxW[:, 1].copy_(-sgn[:, None] * tan[:, 0] * w)

    def face_sum(self, vals, onto="nodes"):
        """Sum face-node values ``vals [F, n1]`` onto the distinct boundary nodes (``onto =
        "nodes"``, order of ``nodes``) or element-local slots (``"local"``, order of ``keys``);
        a fixed-order sum on the device (semk_face_sum_f64): bitwise reproducible."""
        n, row_ptr, pos = self._csr[onto]
        out = torch.empty(n, dtype=torch.float64, device=self.dev)
        if n == 0:
            return out
        vals = vals.to(dtype=torch.float64).contiguous()
        if vals.numel() != self.n_faces * self.node_ids.shape[1]:
            raise ValueError("face values must be [n_faces, n1]")
        _lib.check(_lib.load().semk_face_sum_f64(n, ptr(row_ptr), ptr(pos), ptr(vals), ptr(out),
                                                 stream_ptr()))
        return out


def element_geometry(basis, nodes, l2g, jacobian=True):
    """Geometry of a batch of elements, returned as host arrays in the
    reference's layouts: x_phys [E,2,N,N]; J, invJ [E,2,2,N,N]; detJ [E,N,N]."""
    _lib.require_device()
    tab = basis_tables(basis)
    N = tab.n1
    l2g = np.ascontiguousarray(l2g, dtype=np.uint32).reshape(-1, N * N)
    E = l2g.shape[0]
    nodes_dev = _f64(nodes)
    if nodes_dev.shape[0] != 2:
        raise NotImplementedError("Only supporting 2D elements right now")
    l2g_dev = as_i32_bits(l2g)
    kw = dict(dtype=torch.float64, device="cuda")
    out = {"x_phys": torch.empty((E, 2, N, N), **kw)}
    if jacobian:
        out["J"] = torch.empty((E, 2, 2, N, N), **kw)
        out["invJ"] = torch.empty((E, 2, 2, N, N), **kw)
        out["detJ"] = torch.empty((E, N, N), **kw)
    geom_factors(tab, nodes_dev, l2g_dev, E, x_phys=out["x_phys"], J=out.get("J"),
                 invJ=out.get("invJ"), detJ=out.get("detJ"), check=jacobian)
    return {k: v.cpu().numpy() for k, v in out.items()}
