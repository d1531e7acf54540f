"""Meshes, cells, DOF numbering and finite-element views -- host mirror of the
reference's ``sem.discrete``.

Same classes and call signatures as sem/discrete.py (``Mesh``, ``Cell``,
``SubCell``, ``DOFManager``, ``DOFManagerSC``, ``FiniteElement``,
``SubFiniteElement``, ``Static_COO_Matrix``, ``OutsideDomain``), redesigned
around whole-mesh arrays instead of per-cell Python objects:

* a ``Mesh`` keeps the node maps of all cells of one geometry in a single
  ``uint32[E, N, N]`` block; ``Cell.node_ind_lexicographic`` is a view into it,
  so the in-place renumbering semantics of ``Mesh._permute_nodes``
  (sem/discrete.py:1115-1127) are preserved while every numbering pass
  (static condensation order, RCM graph, centroids, boundary masks) is one
  vectorised NumPy expression instead of a loop over cells;
* per-element geometry (``fe.x_phys``, ``fe.invJ``, ``fe.detJxW`` ...) is
  evaluated by the CUDA geometry kernel in batches (``device.element_geometry``)
  -- there is no NumPy fallback for it;
* additive API (no reference equivalent): ``Mesh.add_cells`` /
  ``add_boundary_cells`` bulk builders, ``DOFManager.node_map_array``,
  ``boundary_node_ind`` / ``boundary_node_mask`` and
  ``DOFManager.poisson_operator`` which returns the matrix-free device
  operator (operators.PoissonOperator).

The integer tables produced here (L2G maps, hierarchical DOF ids, Dirichlet
masks) are tier T0 of the parity contract: bit-exact against the reference.
"""
import bisect
from collections import namedtuple

import numpy as np
from scipy import linalg, sparse
from scipy.sparse import csgraph

from . import mapping as _mapping
from .mapping import _subface_slice

__all__ = ["OutsideDomain", "Static_COO_Matrix", "DOFManager", "DOFManagerSC",
           "FiniteElement", "SubFiniteElement", "CellBase", "Cell", "SubCell", "Mesh"]

_GEOM_BATCH = 4096   # elements per device geometry batch in finite_elements()


class OutsideDomain(Exception):
    """A physical point lies outside the domain of the mesh."""


class Static_COO_Matrix(object):
    """COO triplets pre-sized for in-place filling; exported to scipy with
    ``tocoo`` (reference: sem/discrete.py:26-41)."""

    def __init__(self, data, row_col, shape):
        self.data = data
        self.row_col = row_col
        self.row = row_col[0]
        self.col = row_col[1]
        self.shape = shape

    def tocoo(self):
        return sparse.coo_matrix((self.data, self.row_col))


# ==========================================================================
# DOF managers
# ==========================================================================
class DOFManager(object):
    """Degrees of freedom on a mesh (reference: sem/discrete.py:44-280)."""

    _compute_flag_keys = {"x_phys", "Jacobian"}
    default_compute_flags = dict.fromkeys(_compute_flag_keys, False)

    def __init__(self, mesh, dofs_per_node=1, basis=None, mapping_basis=None,
                 rcm_order=True):
        self._mesh = mesh
        self._dpn = dofs_per_node
        self._mesh._compute_cell_centroids()
        self._basis = basis
        self._map_basis = basis if mapping_basis is None else mapping_basis
        # NOTE (inherited): the manager renumbers the mesh *in place*; two
        # managers on one mesh conflict (sem/discrete.py:119-122).
        if rcm_order:
            self._reorder_nodes_rcm()

    # -- sizes -------------------------------------------------------------------
    @property
    def ndof_per_node(self):
        return self._dpn

    @property
    def ndof(self):
        return self._dpn * self._mesh.n_nodes

    @property
    def mesh(self):
        return self._mesh

    # -- flags -------------------------------------------------------------------
    def _resolve_cmpflag_dependencies(self, compute_flags):
        unknown = set(compute_flags) - self._compute_flag_keys
        if unknown:
            raise ValueError("Unrecognized flags {}.".format(unknown))
        for flag, default in self.default_compute_flags.items():
            compute_flags.setdefault(flag, default)
        if compute_flags["Jacobian"]:
            compute_flags["x_phys"] = True

    # -- node ordering -------------------------------------------------------------
    def _graph_node_sets(self):
        """Rows of node ids whose pairwise products form the connectivity
        graph: every node of every cell (sem/discrete.py:142-167)."""
        return [blk.node_maps.reshape(blk.n_cells, -1) for blk in self._mesh._blocks_flushed()]

    def _graph_size(self):
        return self._mesh.n_nodes

    def _get_connectivity_graph(self):
        """Node connectivity graph in CSR form.  Entries are all (i, j) pairs
        of nodes sharing a cell; ``tocsr`` canonicalises (duplicates summed,
        indices sorted), so the result is identical to the reference's
        cell-by-cell construction."""
        rows, cols = [], []
        for ids in self._graph_node_sets():
            n = ids.shape[1]
            rows.append(np.repeat(ids, n, axis=1).ravel())
            cols.append(np.tile(ids, (1, n)).ravel())
        rows = np.concatenate(rows).astype(np.uint32, copy=False)
        cols = np.concatenate(cols).astype(np.uint32, copy=False)
        size = self._graph_size()
        graph = sparse.coo_matrix((np.ones(rows.size, dtype=bool), (rows, cols)), (size, size))
        return graph.tocsr()

    def _reorder_nodes_rcm(self):
        """Reverse Cuthill-McKee renumbering of all nodes
        (sem/discrete.py:169-178)."""
        perm = csgraph.reverse_cuthill_mckee(self._get_connectivity_graph(), True)
        self._mesh._permute_nodes(perm)

    # -- element views -------------------------------------------------------------
    def _precomputed_geometry(self, first, count, flags):
        """Device geometry of cells [first, first+count) as host arrays, or
        None when no geometric quantity was requested."""
        if not flags.get("x_phys"):
            return None
        from . import device
        maps = self._mesh.node_map_array()[first:first + count]
        return device.element_geometry(self._map_basis, self._mesh.nodes, maps,
                                       jacobian=bool(flags.get("Jacobian")))

    def get_finite_element(self, i, **compute_flags):
        self._resolve_cmpflag_dependencies(compute_flags)
        cell = self._mesh.get_cell(i)
        return FiniteElement(self, cell, compute_flags)

    def finite_elements(self, **compute_flags):
        """Iterate over all finite elements, with the requested geometry
        (``x_phys=True`` and/or ``Jacobian=True``) attached.  Geometry is
        evaluated on the GPU in batches (sem/discrete.py:189-209 built one
        Mapping per cell on the host)."""
        self._resolve_cmpflag_dependencies(compute_flags)
        mesh = self._mesh
        homogeneous = mesh._is_homogeneous()
        geo, base = None, 0
        for i in range(mesh.n_cells):
            pre = None
            if compute_flags["x_phys"] and homogeneous:
                if geo is None or i >= base + _GEOM_BATCH:
                    base = i
                    geo = self._precomputed_geometry(base, _GEOM_BATCH, compute_flags)
                pre = {k: v[i - base] for k, v in geo.items()}
            yield FiniteElement(self, mesh.get_cell(i), compute_flags, _precomputed=pre)

    def boundary_elements(self, name, **compute_flags):
        """Pairs (parent element, boundary sub-element) on the named boundary
        (sem/discrete.py:211-219)."""
        self._resolve_cmpflag_dependencies(compute_flags)
        mesh = self._mesh
        cells = sorted(mesh._boundary_cells[mesh._boundary_id_lookup[name]])
        geo = None
        if compute_flags["x_phys"] and cells and mesh._is_homogeneous():
            from . import device
            maps = mesh.node_map_array()[np.asarray(cells)]
            geo = device.element_geometry(self._map_basis, mesh.nodes, maps,
                                          jacobian=bool(compute_flags["Jacobian"]))
        for j, c in enumerate(cells):
            pre = None if geo is None else {k: v[j] for k, v in geo.items()}
            parent = FiniteElement(self, mesh.get_cell(c), compute_flags, _precomputed=pre)
            for bnd_fe in parent.boundary_elements(name):
                yield parent, bnd_fe

    # -- field evaluation ------------------------------------------------------------
    def interpolate(self, coeffs, x_phys):
        fe, x_param = self.find_elem_containing_point(x_phys)
        return fe.interpolate(coeffs[..., fe.node_ind], x_param)

    def values_at_nodes(self, coeffs):
        """GLL coefficients -> values at the (equispaced) mesh nodes
        (sem/discrete.py:235-258), all cells at once.  A CUDA tensor (e.g. a
        solution of ``poisson_operator(...).solve``) is resampled on the device
        (csrc/semk_field.cu) and a CUDA tensor is returned."""
        if not isinstance(coeffs, np.ndarray) and hasattr(coeffs, "is_cuda"):
            return self._values_at_nodes_device(coeffs)
        out = np.empty_like(coeffs)
        for blk in self._mesh._blocks_flushed():
            maps = blk.node_maps
            out[..., maps] = self._basis.interpolate_on_grid_eq(coeffs[..., maps])
        return out

    def _values_at_nodes_device(self, coeffs):
        import torch
        from . import _lib, device
        if not (coeffs.is_cuda and coeffs.dtype == torch.float64
                and coeffs.shape[-1] == self._mesh.n_nodes):
            raise ValueError("coeffs must be a float64 CUDA tensor [..., n_nodes]")
        lib = _lib.load()
        tab = device.basis_tables(self._basis)
        t = self._device_field_tables(coeffs.device)
        src = coeffs.contiguous().reshape(-1, coeffs.shape[-1])
        out = torch.empty_like(src)
        for i in range(src.shape[0]):
            _lib.check(lib.semk_values_at_nodes_f64(
                tab.n1, t["n_elem"], device.ptr(t["l2g"]), device.ptr(t["winner"]),
                device.ptr(t["emat"]), device.ptr(src[i]), device.ptr(out[i]),
                device.stream_ptr()))
        return out.reshape(coeffs.shape)

    def _device_field_tables(self, dev):
        """Device tables of the nodal-field kernels, built once and kept: the L2G map, the
        winner bytes of the last-element-wins rule (``device.winner_table``) and the 1-D
        equispaced interpolation matrix."""
        cache = getattr(self, "_field_tables", None)
        if cache is None or cache["dev"] != dev:
            import torch
            from . import device
            NN = device.basis_tables(self._basis).n1 ** 2
            l2g = self.node_map_array().reshape(-1, NN)
            sub = [b for _, b in self._basis.iter_subbases()][0]
            winner = device.winner_table(l2g, self._mesh.n_nodes)
            cache = dict(dev=dev, l2g=device.as_i32_bits(l2g, dev),
                         winner=torch.from_numpy(winner).to(dev),
                         emat=device._f64(np.ascontiguousarray(sub.interp_eq_mat), dev),
                         n_elem=int(l2g.shape[0]))
            self._field_tables = cache
        return cache

    # -- nodal fields after a solve: coordinates, gradients, norms, fluxes (device) -----------
    def _post_tables(self, dev):
        """``_device_field_tables`` plus what the post-processing methods need (on first use):
        the mesh nodes, the node -> entries CSR of the whole L2G map
        (``device.node_entries_csr``) and reduction scratch."""
        import torch
        from . import _lib, device
        t = self._device_field_tables(dev)
        if "csr" not in t:
            tab, ftab = device.basis_tables(self._map_basis), device.basis_tables(self._basis)
            if not (tab.n1 == ftab.n1 and np.array_equal(tab.D_host, ftab.D_host)
                    and np.array_equal(tab.w_host, ftab.w_host)):
                raise NotImplementedError("nodal fields need the isoparametric case")
            nodes = device._f64(self._mesh.nodes, dev)
            if nodes.shape[0] != 2:
                raise NotImplementedError("Only supporting 2D elements right now")
            t.update(tab=tab, nodes=nodes,
                     csr=device.node_entries_csr(t["l2g"], self._mesh.n_nodes),
                     partials=torch.zeros(int(_lib.load().semk_vec_partials_len(0)),
                                          dtype=torch.float64, device=dev))
        return t

    def _nodal_input(self, u, what="u"):
        import torch
        if not (isinstance(u, torch.Tensor) and u.is_cuda and u.dtype == torch.float64
                and tuple(u.shape) == (self._mesh.n_nodes,)):
            raise ValueError("%s must be a float64 CUDA tensor [n_nodes]" % what)
        return u.contiguous()

    def _element_gradients(self, u, elems=None, weighted=False):
        """Physical gradient of the nodal vector ``u`` on the elements ``elems`` (int64 CUDA
        tensor, None = all): ``(grad [2, n, NN], JxW [n, NN])`` with ``grad[:, i]`` the
        host mirror's ``fe.gradient(u[fe.node_ind])`` of element ``elems[i]`` (times JxW
        when ``weighted``).  One pass of csrc/semk_geom.cu's field kernel."""
        import torch
        from . import device
        u = self._nodal_input(u)
        t = self._post_tables(u.device)
        n = t["n_elem"] if elems is None else int(elems.numel())
        NN = t["tab"].n1 ** 2
        g = torch.empty((2, n, NN), dtype=torch.float64, device=u.device)
        jxw = torch.empty((n, NN), dtype=torch.float64, device=u.device)
        device.field_grad(t["tab"], t["nodes"], t["l2g"], n, self._mesh.n_nodes, elems=elems,
                          u=u, grad_loc=g, weighted=weighted, jxw_loc=jxw)
        return g, jxw

    def node_coordinates(self):
        """Physical coordinates of every GLL node -- the points the operators' nodal vectors
        live on -- as a CUDA tensor ``[2, n_nodes]``: ``fe.x_phys`` of the last element
        containing the node (the loop ``X[:, fe.node_ind] = fe.x_phys`` over
        ``finite_elements``), by the geometry kernel's arithmetic (csrc/semk_geom.cu)."""
        import torch
        from . import _lib, device
        _lib.require_device()
        dev = torch.device("cuda", torch.cuda.current_device())
        t = self._post_tables(dev)
        n = self._mesh.n_nodes
        xy = torch.zeros((2, n), dtype=torch.float64, device=dev)
        device.field_grad(t["tab"], t["nodes"], t["l2g"], t["n_elem"], n, winner=t["winner"],
                          xy=xy)
        return xy

    def gradient(self, u):
        """Gradient of the nodal vector ``u`` (a float64 CUDA tensor ``[n_nodes]``, as both
        Poisson operators return) at the nodes, a CUDA tensor ``[2, n_nodes]``: the
        JxW-weighted average of the element gradients (``fe.gradient``) of the elements
        sharing a node, ``sum_e JxW grad u_e / sum_e JxW`` -- the lumped L2 projection onto
        the continuous space.  The sums run over a fixed order (bitwise reproducible)."""
        import torch
        from . import _lib, device
        g, jxw = self._element_gradients(u, weighted=True)
        t = self._post_tables(g.device)
        ptr_, pos = t["csr"]
        n = self._mesh.n_nodes
        out = torch.empty((3, n), dtype=torch.float64, device=g.device)
        for i, v in enumerate((g[0], g[1], jxw)):
            _lib.check(_lib.load().semk_face_sum_f64(n, device.ptr(ptr_), device.ptr(pos),
                                                     device.ptr(v), device.ptr(out[i]),
                                                     device.stream_ptr()))
        return out[:2] / out[2]

    def _reference_values(self, f, rows, X, what):
        """``exact`` / ``grad_exact`` of ``error_norms`` as a [rows, n_nodes] CUDA tensor:
        nodal values (a gradient also as a pair of components) or a callable of the node
        coordinates (``X[0]``, computed on first need); scalars are broadcast."""
        import torch
        n = self._mesh.n_nodes
        dev = torch.device("cuda", torch.cuda.current_device())
        if callable(f):
            if X[0] is None:
                X[0] = self.node_coordinates()
            f = f(X[0][0], X[0][1])
        parts = list(f) if rows == 2 and isinstance(f, (tuple, list)) else [f]
        parts = [torch.as_tensor(c, dtype=torch.float64, device=dev) for c in parts]
        parts = [c.expand(n) if c.ndim == 0 else c for c in parts]
        want = "[n_nodes]" if rows == 1 else "[2, n_nodes]"
        if len(parts) > 1:
            if len(parts) != 2 or any(tuple(c.shape) != (n,) for c in parts):
                raise ValueError("%s must have shape %s" % (what, want))
            parts = [torch.stack(parts)]
        v = parts[0]
        if tuple(v.shape) != ((n,) if rows == 1 else (2, n)):
            raise ValueError("%s must have shape %s" % (what, want))
        return v.contiguous()

    def error_norms(self, u, exact=None, grad_exact=None):
        """Norms of the error of the nodal vector ``u`` (float64 CUDA ``[n_nodes]``) against
        ``exact`` (nodal values or a callable ``f(x, y)`` on CUDA tensors of the node
        coordinates, the convention of ``robin=`` / ``flux=``) and its gradient
        ``grad_exact`` (``[2, n_nodes]``, a pair of nodal components, or a callable returning
        the pair).  A dict:

        * ``l2``: ``sqrt(sum_e fe.integrate((u - exact)^2))``, ``h1_semi``: the same of
          ``|grad u - grad_exact|^2``, ``max_nodal``: ``max |u - exact|`` over the nodes;
        * ``l2_ref`` / ``h1_semi_ref``: the norms of ``exact`` / ``grad_exact`` themselves.

        ``exact=None``: the norms of ``u`` itself (the reference and its gradient are zero).
        ``grad_exact=None`` with an ``exact``: the H1 entries are None.  The integrals use
        GLL collocation quadrature at the element nodes -- the reference's
        ``FiniteElement.integrate`` -- not over-integration.  One pass of the field kernel with
        a fixed-order reduction (csrc/semk_geom.cu): bitwise reproducible."""
        import math
        import torch
        from . import device
        u = self._nodal_input(u)
        t = self._post_tables(u.device)
        X = [None]
        u_ref = None if exact is None else self._reference_values(exact, 1, X, "exact")
        g_ref = None if grad_exact is None else self._reference_values(grad_exact, 2, X,
                                                                        "grad_exact")
        sums = torch.empty(5, dtype=torch.float64, device=u.device)
        device.field_grad(t["tab"], t["nodes"], t["l2g"], t["n_elem"], self._mesh.n_nodes, u=u,
                          u_ref=u_ref, g_ref=g_ref, sums=sums, partials=t["partials"])
        s = sums.tolist()
        h1 = exact is None or grad_exact is not None
        return dict(l2=math.sqrt(s[0]), h1_semi=math.sqrt(s[1]) if h1 else None,
                    max_nodal=s[2], l2_ref=math.sqrt(s[3]),
                    h1_semi_ref=math.sqrt(s[4]) if h1 else None)

    def boundary_flux(self, u, name, weight=1.0):
        """Flux of the nodal vector ``u`` (float64 CUDA ``[n_nodes]``) through the named
        boundary, ``sum_faces sum_k w_k (grad u . n dS w)_k`` -- the host recipe
        ``sum bfe.integrate(w * (bfe.gradient(u[fe.node_ind]) . bfe.unit_normal))`` over
        ``boundary_elements(name)``, with the outward normal of
        ``SubMapping._compute_normal_vec`` -- as a float.  ``weight`` (the ``w`` of a
        ``-div(w grad u)`` operator; operators do not keep theirs): a scalar, nodal values or
        a callable ``w(x, y)`` on CUDA tensors of the face-node coordinates.  The field
        kernel runs on the boundary cells only; the sum is semk_dot_f64's fixed order.
        An unknown name raises the ``KeyError`` of ``boundary_elements``."""
        import torch
        from . import _lib, device
        u = self._nodal_input(u)
        dev = u.device
        cache = self.__dict__.setdefault("_bfaces_dev", {})
        if (name, dev) not in cache:
            cache[(name, dev)] = device.BoundaryFaces(device.basis_tables(self._basis),
                                                      self._mesh, name, dev)
        bf = cache[(name, dev)]
        if bf.n_faces == 0:
            return 0.0
        t = self._post_tables(dev)
        cells, inv = np.unique(bf.cells, return_inverse=True)
        g, _ = self._element_gradients(u, elems=torch.from_numpy(cells).to(dev))
        NN = t["tab"].n1 ** 2
        idx = torch.from_numpy(inv[:, None] * NN + bf.local).to(dev)
        gn = g[0].reshape(-1)[idx] * bf.n_dSxW[:, 0] + g[1].reshape(-1)[idx] * bf.n_dSxW[:, 1]
        if callable(weight):
            w = torch.as_tensor(weight(bf.x[:, 0, :], bf.x[:, 1, :]), dtype=torch.float64,
                                device=dev).expand(gn.shape)
        elif isinstance(weight, torch.Tensor) or np.ndim(weight) != 0:
            w = self._nodal_input(torch.as_tensor(weight, dtype=torch.float64, device=dev),
                                  "weight")[bf.node_ids_dev]
        else:
            w = torch.full(gn.shape, float(weight), dtype=torch.float64, device=dev)
        w, gn = w.contiguous(), gn.contiguous()
        out = torch.empty(1, dtype=torch.float64, device=dev)
        _lib.check(_lib.load().semk_dot_f64(int(gn.numel()), device.ptr(w), device.ptr(gn),
                                            device.ptr(out), device.ptr(t["partials"]),
                                            device.stream_ptr()))
        return float(out)

    # -- batched point location / evaluation on the device (additive API) -------------------
    def _locate_tables(self):
        """Device tables of the batched point location (lazy): GLL-point coordinates of
        every element (geometry kernel), cell centroids, and a uniform bin grid listing each
        element in every bin its bounding box (inflated by 10 %) touches."""
        cache = getattr(self, "_locate_cache", None)
        if cache is not None:
            return cache
        import torch
        from . import _lib, device
        _lib.require_device()
        mesh = self._mesh
        tab = device.basis_tables(self._map_basis)
        N = tab.n1
        NN = N * N
        l2g = mesh.node_map_array().reshape(-1, NN)
        E = int(l2g.shape[0])
        dev = torch.device("cuda", torch.cuda.current_device())
        nodes_dev = device._f64(mesh.nodes, dev)
        l2g_dev = device.as_i32_bits(l2g, dev)
        x_phys = torch.empty((E, 2, NN), dtype=torch.float64, device=dev)
        device.geom_factors(tab, nodes_dev, l2g_dev, E, x_phys=x_phys, check=False)
        if not hasattr(mesh, "_centroids"):
            mesh._compute_cell_centroids()
        lo = x_phys.amin(dim=2).cpu().numpy()
        hi = x_phys.amax(dim=2).cpu().numpy()
        pad = 0.1 * (hi - lo) + 1e-12 * np.abs(hi).max()
        lo, hi = lo - pad, hi + pad
        g0, g1 = lo.min(axis=0), hi.max(axis=0)
        n_side = int(min(4096, max(1, np.ceil(np.sqrt(E)))))
        h = (g1 - g0) / n_side
        h[h <= 0] = 1.0
        i0 = np.clip(np.floor((lo - g0) / h).astype(np.int64), 0, n_side - 1)
        i1 = np.clip(np.floor((hi - g0) / h).astype(np.int64), 0, n_side - 1)
        span = i1 - i0 + 1
        bins, elems = [], []
        ids = np.arange(E, dtype=np.int64)
        for di in range(int(span[:, 0].max())):
            for dj in range(int(span[:, 1].max())):
                ok = (di < span[:, 0]) & (dj < span[:, 1])
                bins.append((i0[ok, 0] + di) * n_side + i0[ok, 1] + dj)
                elems.append(ids[ok])
        bins, elems = np.concatenate(bins), np.concatenate(elems)
        order = np.argsort(bins, kind="stable")
        bin_ptr = np.zeros(n_side * n_side + 1, dtype=np.uint32)
        np.cumsum(np.bincount(bins, minlength=n_side * n_side), out=bin_ptr[1:])
        sub = [b for _, b in self._basis.iter_subbases()][0]
        msub = [b for _, b in self._map_basis.iter_subbases()][0]
        cache = dict(
            dev=dev, n1=N, n_elem=E, x_phys=x_phys, l2g=l2g_dev,
            centroids=device._f64(mesh._centroids, dev),
            nodes=device._f64(np.asarray(msub.nodes), dev),
            bw=device._f64(np.asarray(msub.bary_wts), dev),
            D=device._f64(np.asarray(msub.D1), dev),
            f_nodes=device._f64(np.asarray(sub.nodes), dev),
            f_bw=device._f64(np.asarray(sub.bary_wts), dev), f_n1=int(sub.n_coeffs),
            bin_ptr=device.as_i32_bits(bin_ptr, dev),
            bin_elems=device.as_i32_bits(elems[order].astype(np.uint32), dev),
            grid=(float(g0[0]), float(g0[1]), float(h[0]), float(h[1]), n_side))
        self._locate_cache = cache
        return cache

    def locate_points(self, points, strict=True):
        """Batched ``find_elem_containing_point`` on the device (sem/discrete.py:263-280 with
        Mapping.inv, sem/mapping.py:146-178): ``points[2, M]`` (array or CUDA tensor) ->
        ``(cells int64[M], x_param float64[2, M])`` as CUDA tensors; the cell found is the one
        with the nearest centroid among the cells containing the point, like the reference's
        search order.  ``strict``: raise ``OutsideDomain`` if a point is in no cell (else
        those entries are -1 / NaN)."""
        import torch
        from . import _lib, device
        t = self._locate_tables()
        pts = device._f64(points, t["dev"]).reshape(2, -1).contiguous()
        M = int(pts.shape[1])
        cells = torch.empty(M, dtype=torch.int64, device=t["dev"])
        xi = torch.empty((2, M), dtype=torch.float64, device=t["dev"])
        x0, y0, hx, hy, n_side = t["grid"]
        _lib.check(_lib.load().semk_locate_points_f64(
            t["n1"], t["n_elem"], device.ptr(t["x_phys"]), device.ptr(t["centroids"]),
            device.ptr(t["nodes"]), device.ptr(t["bw"]), device.ptr(t["D"]), x0, y0, hx, hy,
            n_side, n_side, device.ptr(t["bin_ptr"]), device.ptr(t["bin_elems"]), M,
            device.ptr(pts), 8, 1e-8, device.ptr(cells), device.ptr(xi), device.stream_ptr()))
        if strict and M and bool((cells < 0).any()):
            bad = int(torch.nonzero(cells < 0)[0])
            raise OutsideDomain("Point {} appears outside the domain of the mesh.".format(
                pts[:, bad].cpu().numpy()))
        return cells, xi

    def interpolate_points(self, coeffs, points, strict=True):
        """Batched ``interpolate`` (sem/discrete.py:221-233): values of the field with GLL
        coefficients ``coeffs[..., n_nodes]`` (CUDA tensor or array) at ``points[2, M]``;
        returns a CUDA tensor ``[..., M]``."""
        import torch
        from . import _lib, device
        t = self._locate_tables()
        if t["f_n1"] != t["n1"]:
            raise NotImplementedError("only the isoparametric case is usable "
                                      "(sem/discrete.py:594-597)")
        cells, xi = self.locate_points(points, strict=strict)
        c = device._f64(coeffs, t["dev"])
        if c.shape[-1] != self._mesh.n_nodes:
            raise ValueError("coeffs must have n_nodes entries along the last axis")
        src = c.reshape(-1, c.shape[-1]).contiguous()
        M = int(cells.numel())
        out = torch.empty((src.shape[0], M), dtype=torch.float64, device=t["dev"])
        for i in range(src.shape[0]):
            _lib.check(_lib.load().semk_interpolate_points_f64(
                t["f_n1"], M, device.ptr(cells), device.ptr(xi), device.ptr(t["l2g"]),
                device.ptr(t["f_nodes"]), device.ptr(t["f_bw"]), device.ptr(src[i]),
                device.ptr(out[i]), device.stream_ptr()))
        return out.reshape(tuple(c.shape[:-1]) + (M,))

    def get_global_matrix_equation(self):
        raise NotImplementedError()

    def find_elem_containing_point(self, point):
        point = np.asarray(point, float)
        dist = np.sqrt(np.sum((point - self._mesh._centroids) ** 2, axis=1))
        flags = dict(x_phys=True, Jacobian=True)
        for i in np.argsort(dist):
            fe = FiniteElement(self, self._mesh.get_cell(int(i)), flags)
            try:
                return fe, fe.mapping.inv(point)
            except _mapping.OutsideDomain:
                continue
        raise OutsideDomain("Point {} appears outside the domain of the mesh.".format(point))

    # -- additive API ----------------------------------------------------------------
    def node_map_array(self):
        """The whole L2G map, ``uint32[E, N, N]`` (a view; homogeneous meshes)."""
        return self._mesh.node_map_array()

    def boundary_node_ind(self, name):
        """All node ids on the named boundary, face by face in the order of
        ``boundary_elements(name)`` (duplicates at corners kept)."""
        return self._mesh.boundary_node_ind(name)

    def boundary_node_mask(self, name):
        """``bool[n_nodes]``, True on the named boundary -- the reference's
        ``on_ebc`` polarity (True = essential-BC node, sem/discrete.py:505)."""
        mask = np.zeros(self._mesh.n_nodes, dtype=bool)
        mask[self.boundary_node_ind(name)] = True
        return mask

    def poisson_operator(self, dirichlet=None, geometric_factors=None, **kwargs):
        """Matrix-free Poisson stiffness operator on the GPU for this
        discretisation (additive API; see operators.PoissonOperator).

        dirichlet : bool[n_nodes], optional -- True on essential-BC nodes.
        geometric_factors : (invJ[E,2,2,N,N], detJxW[E,N,N]), optional --
            use externally supplied factors (e.g. the reference's own
            ``fe.invJ`` / ``fe.detJxW``) instead of the device geometry kernel
            (parity tier T1).
        weight (keyword) : float[E, N, N] element-local nodal values or a
            callable ``w(x, y)`` on device tensors -- the operator becomes the
            stiffness of -div(w grad u) (the rho-weighted twin of the recipe,
            examples/squirmer-axisymmetric.py:194-213).
        robin (keyword) : {boundary name: alpha} -- Robin condition
            w du/dn + alpha u = g on those boundaries (alpha >= 0; scalar, nodal values or a
            callable alpha(x, y)).  Flux data g of flux or Robin boundaries goes to
            ``op.solve(flux={name: g})`` or ``op.boundary_load(name, g)``; see
            operators.py for the weak form.
        """
        if self._dpn != 1:
            raise NotImplementedError("poisson_operator supports one DOF per node")
        from .operators import PoissonOperator
        return PoissonOperator(self, dirichlet=dirichlet,
                               geometric_factors=geometric_factors, **kwargs)

    def poisson_eigenpairs(self, k, dirichlet=None, robin=None, weight=None, tol=1e-8,
                           maxiter=500):
        """The ``k`` smallest eigenpairs of ``K x = lambda M x`` on the GPU: ``K`` the stiffness
        of -div(w grad u) with these boundary conditions, ``M`` the diagonal GLL mass
        (block eigensolver LOBPCG, see eigen.py).

        k : 1 <= k <= 32 and smaller than the number of free nodes.
        dirichlet : bool[n_nodes], a boundary name or a list of names, optional -- u = 0 there.
        robin : {boundary name: alpha}, optional -- w du/dn + alpha u = 0 there (alpha >= 0);
            every other boundary is natural (w du/dn = 0).
        weight : as for ``poisson_operator``.
        tol : pair i has converged when ||K x_i - lambda_i M x_i||_{M^-1} / max_j |lambda_j|
            <= tol (x_i M-normalised); the eigenvalue error is about its square.

        The preconditioner follows from the DOF manager: the condensed three-level solve for a
        ``DOFManagerSC`` (orders 2..10), applied to all active residuals of an iteration at once
        (``CondensedPoissonOperator.solve_load_many``: one element factorisation per chunk of up
        to 32 columns, every column bitwise the single solve), Jacobi otherwise; for K + M when
        K is singular (no Dirichlet node, no Robin boundary).  Returns ``(lam, X, info)``: ``lam`` float64[k]
        ascending, ``X`` a CUDA tensor [k, n_nodes], M-orthonormal and zero on the Dirichlet
        nodes, ``info`` a dict (iterations, per-pair residuals, converged flags, preconditioner
        applications, time per phase)."""
        from .eigen import poisson_eigenpairs
        return poisson_eigenpairs(self, k, dirichlet=dirichlet, robin=robin, weight=weight,
                                  tol=tol, maxiter=maxiter)

    def axisymmetric_stokes_operator(self, n_rey=0.0, essential=None, **kwargs):
        """Matrix-free Jacobian / residual of the axisymmetric stream function - vorticity
        system of examples/squirmer-axisymmetric.py:163-297 on the GPU (two DOFs per node;
        additive API, see stokes.AxisymmetricStokesOperator).

        essential : bool[2*n_nodes] (or bool[ndof_exterior]), optional -- True on
            essential-BC DOFs (the complement of the example's ``dof_mask``).
        """
        from .stokes import AxisymmetricStokesOperator
        return AxisymmetricStokesOperator(self, n_rey=n_rey, essential=essential, **kwargs)


class DOFManagerSC(DOFManager):
    """DOF manager that numbers cell-exterior nodes first so that cell
    interiors can be condensed out (reference: sem/discrete.py:283-528)."""

    def __init__(self, mesh, dofs_per_node=1, basis=None, mapping_basis=None,
                 rcm_order=True):
        DOFManager.__init__(self, mesh, dofs_per_node, basis, mapping_basis, rcm_order=False)
        self._do_static_condensation()
        if rcm_order:
            self._reorder_nodes_rcm()

    @property
    def ndof_exterior(self):
        return self._mesh.n_nodes_cell_exterior * self._dpn

    @property
    def ndof_interior(self):
        return self._mesh.n_nodes_cell_interior * self._dpn

    def _do_static_condensation(self):
        """Renumber: distinct exterior nodes in ascending old id, then the
        interior nodes in ascending old id (sem/discrete.py:314-359)."""
        mesh = self._mesh
        if self._fast_static_condensation():
            return
        ext, itr = [], []
        for blk in mesh._blocks_flushed():
            flat = blk.node_maps.reshape(blk.n_cells, -1)
            geo = mesh._geometries[blk.geometry_id]
            ext.append(flat[:, geo.exterior_node_ind].ravel())
            itr.append(flat[:, geo.interior_node_ind].ravel())
        # np.unique / np.sort of the reference, by marking (linear time; the results are the
        # same sorted id lists): exterior ids may repeat, interior ids are private to a cell
        ext_flat, int_flat = np.concatenate(ext), np.concatenate(itr)
        mark = np.zeros(mesh.n_nodes, dtype=bool)
        mark[ext_flat] = True
        ext_ids = np.flatnonzero(mark)
        mark[:] = False
        mark[int_flat] = True
        int_ids = np.flatnonzero(mark)
        if int_ids.size != int_flat.size:          # repeated interior ids: keep the duplicates
            int_ids = np.sort(int_flat.astype(int))
        order = np.concatenate((ext_ids, int_ids))
        if order.size != mesh.n_nodes:
            raise AssertionError("exterior/interior split does not cover the mesh nodes")
        mesh._permute_nodes(order)
        mesh.n_nodes_cell_exterior = ext_ids.size
        mesh.n_nodes_cell_interior = int_ids.size
        mesh.condensed = True

    def _fast_static_condensation(self):
        """The same renumbering by the multi-threaded host helper (csrc/semk_hostnum.cpp) for
        the common case -- one block of cells, contiguous arrays, every node exterior in all
        its cells or interior to exactly one.  Returns False (nothing touched) when the case
        is not covered or the library is not built; the NumPy expressions below then run."""
        mesh = self._mesh
        blocks = mesh._blocks_flushed()
        if len(blocks) != 1 or mesh.n_nodes < (1 << 16):
            return False
        blk = blocks[0]
        maps, nodes = blk.node_maps, mesh.nodes
        if not (isinstance(maps, np.ndarray) and maps.dtype == np.uint32 and maps.flags.c_contiguous
                and maps.flags.writeable and isinstance(nodes, np.ndarray)
                and nodes.dtype == np.float64 and nodes.ndim == 2 and nodes.flags.writeable
                and nodes.strides[1] == 8 and nodes.strides[0] % 8 == 0
                and nodes.shape[1] >= mesh.n_nodes):
            return False
        try:
            from . import _lib
            lib = _lib.load()
        except (ImportError, OSError):
            return False
        import ctypes as C
        geo = mesh._geometries[blk.geometry_id]
        ext_idx = np.ascontiguousarray(geo.exterior_node_ind, dtype=np.int32).ravel()
        int_idx = np.ascontiguousarray(geo.interior_node_ind, dtype=np.int32).ravel()
        nn = int(np.prod(maps.shape[1:]))
        order = np.empty(mesh.n_nodes, dtype=np.uint32)
        n_ext, n_int = C.c_int64(0), C.c_int64(0)
        rc = lib.semk_host_sc_numbering(
            int(mesh.n_nodes), int(blk.n_cells), nn, maps.ctypes.data, ext_idx.ctypes.data,
            int(ext_idx.size), int_idx.ctypes.data, int(int_idx.size), nodes.ctypes.data,
            int(nodes.shape[0]), int(nodes.strides[0] // 8), C.byref(n_ext), C.byref(n_int),
            order.ctypes.data, _lib.host_threads())
        if rc != 0:
            return False        # (the helper leaves everything untouched unless it succeeds)
        mesh.n_nodes_cell_exterior = int(n_ext.value)
        mesh.n_nodes_cell_interior = int(n_int.value)
        mesh.condensed = True
        return True

    def _graph_node_sets(self):
        out = []
        for blk in self._mesh._blocks_flushed():
            geo = self._mesh._geometries[blk.geometry_id]
            out.append(blk.node_maps.reshape(blk.n_cells, -1)[:, geo.exterior_node_ind])
        return out

    def _graph_size(self):
        return self._mesh.n_nodes_cell_exterior

    def _reorder_nodes_rcm(self):
        """RCM over the exterior nodes only; interior ids stay put
        (sem/discrete.py:389-402)."""
        mesh = self._mesh
        n, n_ext = mesh.n_nodes, mesh.n_nodes_cell_exterior
        perm = np.empty(n, np.uint32)
        perm[:n_ext] = csgraph.reverse_cuthill_mckee(self._get_connectivity_graph(), True)
        perm[n_ext:] = np.arange(n_ext, n)
        mesh._permute_nodes(perm)

    def condensed_poisson_operator(self, dirichlet=None, **kwargs):
        """The statically condensed Poisson operator on the GPU: local Schur
        complements, condensed apply / PCG over the element-exterior DOFs and
        interior back-substitution (the device twin of assemble_global_sc_system
        + solve; additive API, see condensed.CondensedPoissonOperator).

        dirichlet : bool[n_nodes] or bool[ndof_exterior], optional -- True on
            essential-BC nodes (the ``on_ebc`` polarity of ``solve``).
        robin (keyword) : {boundary name: alpha} -- Robin condition
            w du/dn + alpha u = g, as for ``poisson_operator``; the term enters the local
            Schur complements through the element reaction diagonal.
        """
        from .condensed import CondensedPoissonOperator
        return CondensedPoissonOperator(self, dirichlet=dirichlet, **kwargs)

    def solve_device(self, local_systems, dof_vec, on_ebc, rtol=1e-12, maxiter=200000,
                     preconditioner="jacobi"):
        """``solve`` on the GPU (sem/discrete.py:526-528 with the Schur assembly of
        :478-500 folded in): takes the same hierarchically ordered
        ``local_systems`` = iterable of ``(lmat_h, lrhs_h)`` as
        ``assemble_global_sc_system`` / ``solve``, the same ``on_ebc`` polarity
        (True = essential-BC DOF, values read from ``dof_vec``) and writes the
        solution into ``dof_vec`` in place.  The local matrices must be symmetric
        with positive definite interior blocks; the condensed system is solved by
        PCG instead of SuperLU (``preconditioner``: "jacobi" or "two-level", see
        CondensedPoissonOperator.solve_pcg).  Returns the PCG info."""
        if self._dpn != 1:
            raise NotImplementedError("solve_device supports one DOF per node")
        from .condensed import CondensedLocalSystems
        local_systems = list(local_systems)
        lm = np.stack([np.asarray(ls[0], dtype=np.float64) for ls in local_systems])
        lr = np.stack([np.asarray(ls[1], dtype=np.float64) for ls in local_systems])
        on_ebc = np.asarray(on_ebc)
        if on_ebc.dtype != np.bool_ or on_ebc.shape != (self.ndof_exterior,):
            raise ValueError("on_ebc must be bool[ndof_exterior]")
        cs = CondensedLocalSystems(self, lm, lr, dirichlet=on_ebc)
        vals = np.zeros(self.ndof)
        vals[:self.ndof_exterior][on_ebc] = np.asarray(dof_vec)[:self.ndof_exterior][on_ebc]
        u, info = cs.solve(vals, rtol=rtol, maxiter=maxiter, preconditioner=preconditioner)
        if not info.converged:
            from ._lib import SolverFailure
            raise SolverFailure("condensed PCG did not converge: %r" % (info,))
        dof_vec[...] = u.cpu().numpy()
        return info

    # -- Schur-complement assembly (host; kept for literal drop-in use) ------------
    def init_global_linear_system(self):
        """Empty COO Schur system over the exterior DOFs and a zero RHS
        (sem/discrete.py:404-426)."""
        n_entries = 0
        for blk in self._mesh._blocks_flushed():
            geo = self._mesh._geometries[blk.geometry_id]
            n_entries += blk.n_cells * (geo.n_exterior_nodes * self._dpn) ** 2
        row_col = np.zeros((2, n_entries), dtype=np.uint32)
        entries = np.zeros(n_entries, dtype=np.float64)
        nd = self.ndof_exterior
        return Static_COO_Matrix(entries, row_col, (nd, nd)), np.zeros(nd, dtype=np.float64)

    @staticmethod
    def reorder_local_system_hier(fe, local_system):
        """Lexicographic -> hierarchical (exterior first) local ordering
        (sem/discrete.py:428-436)."""
        lmat, lrhs = local_system
        h = fe.loc_dof_ind_hier
        return lmat[np.ix_(h, h)], lrhs[h]

    @staticmethod
    def compute_local_sc_system(fe, local_system):
        """Local Schur complement S = A_ee - A_ei A_ii^{-1} A_ie and its RHS
        from a hierarchically ordered local system (sem/discrete.py:438-476)."""
        lmat, lrhs = local_system
        ne = fe.ndof_exterior
        Aee, Aei, Aie, Aii = lmat[:ne, :ne], lmat[:ne, ne:], lmat[ne:, :ne], lmat[ne:, ne:]
        # X = A_ei A_ii^{-1}, obtained from the transposed solve like the reference
        X = linalg.solve(Aii.T, Aei.T, check_finite=False).T
        sc_mat = Aee - X.dot(Aie)
        sc_rhs = lrhs[:ne] - X.dot(lrhs[ne:])
        if not (np.isfinite(sc_mat[ne:, ne:]).all() and np.isfinite(sc_rhs[ne:]).all()):
            raise AssertionError("non-finite Schur complement")
        return sc_mat, sc_rhs

    def assemble_global_sc_system(self, global_sc_system, local_systems):
        """Fill the COO triplets and scatter-add the RHS
        (sem/discrete.py:478-500)."""
        gmat, grhs = global_sc_system
        at = 0
        for fe, loc_sys in zip(self.finite_elements(), local_systems):
            sc_mat, sc_rhs = self.compute_local_sc_system(fe, loc_sys)
            ne = fe.ndof_exterior
            ids = fe.global_dof_ind_hier[:ne]
            gmat.row[at:at + ne * ne] = np.repeat(ids, ne)
            gmat.col[at:at + ne * ne] = np.tile(ids, ne)
            gmat.data[at:at + ne * ne] = sc_mat.ravel()
            grhs[ids] += sc_rhs
            at += ne * ne

    def _solve_boundary_dofs(self, global_sc_system, dof_vec, on_ebc):
        """Direct solve of the condensed system with the essential-BC rows and
        columns eliminated; ``on_ebc`` True = Dirichlet
        (sem/discrete.py:502-511)."""
        sc_mat, sc_rhs = global_sc_system
        free = ~on_ebc
        ext = dof_vec[:self.ndof_exterior]
        A = sc_mat.tocoo().tocsr()[free]
        rhs = sc_rhs[free] - A[:, on_ebc].dot(ext[on_ebc])
        ext[free] = sparse.linalg.spsolve(A[:, free], rhs)

    def _solve_interior_dofs(self, local_systems, dof_vec):
        """Element-interior back-substitution (sem/discrete.py:513-524)."""
        for fe, (lmat, lrhs) in zip(self.finite_elements(), local_systems):
            ne = fe.ndof_exterior
            ids = fe.global_dof_ind_hier
            dof_vec[ids[ne:]] = linalg.solve(
                lmat[ne:, ne:], lrhs[ne:] - lmat[ne:, :ne].dot(dof_vec[ids[:ne]]))

    def solve(self, global_sc_system, local_systems, dof_vec, on_ebc):
        import scipy.sparse.linalg  # noqa: F401  (makes sparse.linalg resolvable)
        self._solve_boundary_dofs(global_sc_system, dof_vec, on_ebc)
        self._solve_interior_dofs(local_systems, dof_vec)


# ==========================================================================
# finite-element views
# ==========================================================================
class FiniteElement(object):
    """One cell + its local DOFs + (optionally) its geometry
    (reference: sem/discrete.py:531-705)."""

    def __init__(self, dof_mngr, cell, compute_flags, _precomputed=None):
        self._cell = cell
        self._dpn = dof_mngr._dpn
        self._basis = dof_mngr._basis
        self._quad_rule = self._basis._quad_rule
        self._mapping = _mapping.Mapping(dof_mngr._map_basis, cell, compute_flags,
                                         _precomputed=_precomputed)
        self._cmpflags = compute_flags
        self._l_dof_ind_hier, self._g_dof_ind_hier = self._compute_hier_dofs()

    def _compute_hier_dofs(self):
        """dof = dpn*node + component, in the hierarchical node order
        (sem/discrete.py:561-576)."""
        dpn = self._dpn
        comp = np.arange(dpn, dtype=np.uint32)
        loc = self._cell.geometry.hierarchical_node_order.astype(np.uint32)
        glo = self._cell.node_ind_hierarchical.astype(np.uint32)
        l_dofs = (dpn * loc[:, None] + comp).ravel().astype(np.uint32)
        g_dofs = (dpn * glo[:, None] + comp).ravel().astype(np.uint32)
        return l_dofs, g_dofs

    # -- geometry ------------------------------------------------------------------
    @property
    def ndim(self):
        return self._basis.ndim

    @property
    def x_phys(self):
        return self._mapping.x_phys

    @property
    def J(self):
        return self._mapping.J

    @property
    def invJ(self):
        return self._mapping.invJ

    @property
    def detJxW(self):
        return self._quad_rule.xweight(self.mapping.detJ)

    # -- sizes -----------------------------------------------------------------------
    @property
    def ndof(self):
        return self.n_nodes * self._dpn

    @property
    def ndof_exterior(self):
        return self.n_exterior_nodes * self._dpn

    @property
    def ndof_interior(self):
        return self.n_interior_nodes * self._dpn

    @property
    def n_nodes(self):
        return self._cell.n_nodes

    @property
    def n_exterior_nodes(self):
        return self._cell.n_exterior_nodes

    @property
    def n_interior_nodes(self):
        return self._cell.n_interior_nodes

    # -- index tables ------------------------------------------------------------------
    @property
    def loc_dof_ind_hier(self):
        return self._l_dof_ind_hier

    @property
    def global_dof_ind_hier(self):
        return self._g_dof_ind_hier

    @property
    def exterior_dof_ind(self):
        return self._g_dof_ind_hier[:self.ndof_exterior]

    @property
    def interior_dof_ind(self):
        return self._g_dof_ind_hier[self.ndof_exterior:]

    @property
    def node_ind(self):
        """Global node ids of the cell, lexicographic ``uint32[N, N]`` -- one
        row block of the L2G map."""
        return self._cell.node_ind_lexicographic

    # -- helpers -----------------------------------------------------------------------
    @property
    def basis(self):
        return self._basis

    @property
    def mapping(self):
        return self._mapping

    @property
    def quadrature(self):
        return self._quad_rule

    def local(self, arr):
        return arr[self.node_ind]

    def interpolate(self, coeffs, x_param):
        if not ((x_param >= -1).all() and (x_param <= 1).all()):
            raise AssertionError("parametric point outside [-1, 1]")
        return self._basis.interpolate(coeffs, x_param)

    def deriv(self, coeffs, dim):
        """d/dx_dim in physical space (sem/discrete.py:674-678)."""
        return np.einsum("i...,i...", self.invJ[:, dim], self._basis.gradient(coeffs))

    def gradient(self, coeffs):
        """Physical gradient: invJ^T applied to the parametric gradient
        (sem/discrete.py:680-684)."""
        return np.einsum("ij...,i...->j...", self.invJ, self._basis.gradient(coeffs))

    def integrate(self, coeffs):
        return (coeffs * self.detJxW).sum()

    def values_at_nodes(self, coeffs):
        return self._basis.interpolate_on_grid_eq(coeffs)

    def sub_fe(self, face):
        return SubFiniteElement(self, face)

    def boundary_elements(self, name):
        bnd_id = self._cell._mesh._boundary_id_lookup[name]
        for _ndim, face in self._cell._boundary_data.get(bnd_id, []):
            yield SubFiniteElement(self, face)


class SubFiniteElement(FiniteElement):
    """Finite element on a face of a parent element
    (reference: sem/discrete.py:708-774)."""

    def __init__(self, parent_fe, face):
        self._parent_fe = parent_fe
        self._cell = parent_fe._cell.sub_cell(face)
        self._dpn = parent_fe._dpn
        self._cmpflags = parent_fe._cmpflags
        self._basis = parent_fe.basis.get_subbasis(face // 2)
        self._mapping = parent_fe.mapping.get_submapping(face)
        self._quad_rule = self._basis._quad_rule
        self._l_dof_ind_hier, self._g_dof_ind_hier = self._compute_hier_dofs()

    @property
    def parent_fe(self):
        return self._parent_fe

    @property
    def n_dS(self):
        return self._mapping.n_dS

    @property
    def dS(self):
        return self._mapping.dS

    @property
    def dSxW(self):
        return self._quad_rule.xweight(self.dS)

    @property
    def unit_normal(self):
        return self._mapping.unit_normal

    @property
    def n_dSxW(self):
        return self._quad_rule.xweight(self.n_dS)

    def slice_from_parent(self, arr):
        return _subface_slice(self._mapping._face, arr, self._parent_fe.ndim)

    def parent_dofs(self):
        """Local DOF ids, in the parent's numbering, of this face's nodes
        (sem/discrete.py:757-766)."""
        par = self._parent_fe
        lin = np.arange(par.n_nodes).reshape(par.basis.coeff_shape)
        nodes = _subface_slice(self._mapping._face, lin, par.ndim)
        comp = np.arange(self._dpn)
        return (nodes[:, None] * self._dpn + comp).ravel().astype(np.uint32)

    def integrate(self, coeffs):
        return (coeffs * self.dSxW).sum(axis=-1)

    def gradient(self, coeffs):
        grad = self._parent_fe.gradient(coeffs)
        return _subface_slice(self._mapping._face, grad, self._parent_fe.ndim)


# ==========================================================================
# cells
# ==========================================================================
class CellBase(object):
    """Nodes of one cell as views into the mesh arrays
    (reference: sem/discrete.py:777-854)."""

    def __init__(self, mesh, geometry, node_map):
        self._mesh = mesh
        self._geometry = geometry
        self._node_map = node_map

    @property
    def geometry(self):
        return self._geometry

    @property
    def ndim(self):
        return self._geometry.ndim

    @property
    def n_nodes(self):
        return self._geometry.n_nodes

    @property
    def n_exterior_nodes(self):
        return self._geometry.n_exterior_nodes

    @property
    def n_interior_nodes(self):
        return self._geometry.n_interior_nodes

    def _pick(self, local_ids):
        return self._node_map.flat[local_ids]

    @property
    def node_ind_lexicographic(self):
        return self._node_map

    @property
    def node_ind_hierarchical(self):
        return self._pick(self._geometry._hier_node_order)

    @property
    def vertex_node_ind(self):
        return self._pick(self._geometry.vertex_node_ind)

    @property
    def exterior_node_ind(self):
        return self._pick(self._geometry.exterior_node_ind)

    @property
    def interior_node_ind(self):
        return self._pick(self._geometry.interior_node_ind)

    @property
    def nodes_lexicographic(self):
        return self._mesh.nodes[:, self.node_ind_lexicographic]

    @property
    def nodes_hierarchical(self):
        return self._mesh.nodes[:, self.node_ind_hierarchical]

    @property
    def vertex_nodes(self):
        return self._mesh.nodes[:, self.vertex_node_ind]

    @property
    def exterior_nodes(self):
        return self._mesh.nodes[:, self.exterior_node_ind]

    @property
    def interior_nodes(self):
        return self._mesh.nodes[:, self.interior_node_ind]

    def sub_cell(self, face):
        return SubCell(self, face)


class Cell(CellBase):
    def __init__(self, mesh, geometry, node_map, region_id, adj_map, boundary_data):
        CellBase.__init__(self, mesh, geometry, node_map)
        self._region_id = region_id
        self._adj_map = adj_map
        self._boundary_data = boundary_data

    @property
    def region_id(self):
        return self._region_id

    @property
    def region_name(self):
        return self._mesh._region_names[self._region_id]

    def neighbor(self, face):
        other = self._adj_map[face]
        if other is not None:
            return self._mesh.get_cell(other)

    def boundary_cells(self, name):
        bnd_id = self._mesh._boundary_id_lookup[name]
        for _ndim, face in self._boundary_data.get(bnd_id, []):
            yield self.sub_cell(face)


class SubCell(CellBase):
    """The cell formed by one face of a parent cell
    (reference: sem/discrete.py:885-917)."""

    def __init__(self, parent_cell, face):
        pc = parent_cell
        CellBase.__init__(self, pc._mesh, pc.geometry.sub_geometry(face // 2),
                          _subface_slice(face, pc._node_map, pc.ndim))
        self._parent_cell = pc


# ==========================================================================
# mesh
# ==========================================================================
class _CellBlock(object):
    """A run of consecutive cells sharing one geometry."""
    __slots__ = ("geometry_id", "region_ids", "node_maps")

    def __init__(self, geometry_id, region_ids, node_maps):
        self.geometry_id = geometry_id
        self.region_ids = region_ids
        self.node_maps = node_maps

    @property
    def n_cells(self):
        return self.node_maps.shape[0]


class Mesh(object):
    """A finite-element mesh (reference: sem/discrete.py:920-1127)."""

    CellData = namedtuple("CellData", ["geometry_id", "region_id", "node_map"])
    BoundaryData = namedtuple("BoundaryData", ["ndim", "index"])

    def __init__(self, ndim):
        self._ndim = ndim
        self._geometries = []
        self._blocks = []          # consolidated cell blocks
        self._block_start = []     # first cell number of each block
        self._pending = []         # (geometry_id, region_id, node_map) not yet consolidated
        self._n_cells = 0
        self._adj_map = {}         # cell -> list (created lazily)
        self._adj_array = None     # int64[E, faces], -1 = none (set in bulk by the importer)
        self._region_names = []
        self._region_id_lookup = {}
        self._boundary_names = []
        self._boundary_id_lookup = {}
        self._boundary_map = {}    # cell -> {bnd_id: [BoundaryData]}
        self._boundary_cells = []  # bnd_id -> set(cell)
        self._boundary_faces = []  # bnd_id -> [(cell, face)] in insertion order
        self._finalized = False
        self.condensed = False

    # -- sizes -----------------------------------------------------------------------
    @property
    def ndim(self):
        return self._ndim

    @property
    def n_nodes(self):
        return self.nodes.shape[1]

    @property
    def n_cells(self):
        return self._n_cells

    @property
    def n_boundary_cells(self):
        return len(self._boundary_map)

    # -- construction ------------------------------------------------------------------
    def add_geometry(self, geometry):
        if geometry.ndim > self.ndim:
            raise ValueError("Cell geometry has more dimensions than the mesh.")
        self._geometries.append(geometry)
        return len(self._geometries) - 1

    def new_region(self, name):
        self._region_names.append(name)
        self._region_id_lookup[name] = len(self._region_names) - 1
        return len(self._region_names) - 1

    def new_boundary(self, name):
        self._boundary_names.append(name)
        bnd_id = len(self._boundary_names) - 1
        self._boundary_id_lookup[name] = bnd_id
        self._boundary_cells.append(set())
        self._boundary_faces.append([])
        return bnd_id

    def set_nodes(self, nodes):
        """Node coordinates, ``ndim``-by-N.  Kept by reference like the
        reference does (np.asarray), so later renumbering also permutes the
        caller's array (sem/discrete.py:1018-1029)."""
        self.nodes = np.asarray(nodes)
        if self.nodes.shape[0] != self.ndim:
            raise ValueError("Points have the wrong number of dimensions.")

    def add_cell(self, node_ind, geometry_id, region_id):
        """Append one cell given its lexicographic node ids
        (sem/discrete.py:1031-1048)."""
        geo = self._geometries[geometry_id]
        node_ind = np.array(node_ind, dtype=np.uint32).reshape(geo.shape)
        self._pending.append((geometry_id, region_id, node_ind))
        self._n_cells += 1

    def add_cells(self, node_ind, geometry_id, region_id=0):
        """Bulk ``add_cell``: ``node_ind[E, *geometry.shape]`` (additive API).
        The array is adopted without copying when it is C-contiguous uint32."""
        self._flush()
        geo = self._geometries[geometry_id]
        maps = np.ascontiguousarray(node_ind, dtype=np.uint32)
        maps = maps.reshape((-1,) + tuple(geo.shape))
        regions = np.broadcast_to(np.asarray(region_id, dtype=np.int32), (maps.shape[0],)).copy()
        self._append_block(_CellBlock(geometry_id, regions, maps))
        self._n_cells += maps.shape[0]

    def add_boundary_cell(self, cell_number, bnd_id, ndim, index):
        """Mark face ``index`` of a cell as lying on boundary ``bnd_id``
        (sem/discrete.py:1050-1068)."""
        per_cell = self._boundary_map.setdefault(cell_number, {})
        per_cell.setdefault(bnd_id, []).append(Mesh.BoundaryData(ndim, index))
        self._boundary_cells[bnd_id].add(cell_number)
        self._boundary_faces[bnd_id].append((cell_number, index))

    def add_boundary_cells(self, cell_numbers, bnd_id, ndim, index):
        """Bulk ``add_boundary_cell`` for one face index (additive API)."""
        for c in np.asarray(cell_numbers).ravel().tolist():
            self.add_boundary_cell(int(c), bnd_id, ndim, index)

    # -- block bookkeeping ---------------------------------------------------------------
    def _append_block(self, blk):
        start = self._block_start[-1] + self._blocks[-1].n_cells if self._blocks else 0
        self._blocks.append(blk)
        self._block_start.append(start)

    def _flush(self):
        """Consolidate cells added one by one into blocks."""
        pend, self._pending = self._pending, []
        i = 0
        while i < len(pend):
            gid = pend[i][0]
            j = i
            while j < len(pend) and pend[j][0] == gid:
                j += 1
            maps = np.stack([p[2] for p in pend[i:j]])
            regions = np.array([p[1] for p in pend[i:j]], dtype=np.int32)
            self._append_block(_CellBlock(gid, regions, maps))
            i = j

    def _merge_blocks(self):
        """Fuse runs of consecutive blocks that share a geometry into one block, so that
        homogeneity is decided by geometry id and not by how the cells arrived (one
        ``add_cells`` call per ``$Elements`` header of a Gmsh file -- Gmsh's own writer emits
        one header per element --, ``add_cell`` after a ``get_cell``, ...).  The reference
        accepts any blocking (sem/discrete.py:1031-1048 keeps one array per cell).  Cell
        views handed out before more cells were added keep pointing at the old arrays."""
        blocks = self._blocks
        if len(blocks) < 2:
            return
        merged, i = [], 0
        while i < len(blocks):
            j = i + 1
            while j < len(blocks) and blocks[j].geometry_id == blocks[i].geometry_id:
                j += 1
            if j - i == 1:
                merged.append(blocks[i])
            else:
                merged.append(_CellBlock(
                    blocks[i].geometry_id,
                    np.concatenate([b.region_ids for b in blocks[i:j]]),
                    np.ascontiguousarray(np.concatenate([b.node_maps for b in blocks[i:j]]))))
            i = j
        if len(merged) != len(blocks):
            self._blocks = merged
            self._block_start = []
            start = 0
            for blk in merged:
                self._block_start.append(start)
                start += blk.n_cells

    def _blocks_flushed(self):
        self._flush()
        self._merge_blocks()
        return self._blocks

    def _is_homogeneous(self):
        return len(self._blocks_flushed()) == 1

    def node_map_array(self):
        """L2G map of the whole mesh as one ``uint32[E, *shape]`` array (view)."""
        blocks = self._blocks_flushed()
        if len(blocks) != 1:
            raise NotImplementedError("mixed cell geometries have no single node-map array")
        return blocks[0].node_maps

    # -- access ------------------------------------------------------------------------
    def get_geometries(self):
        return self._geometries

    def get_cell(self, i):
        self._blocks_flushed()
        if i < 0 or i >= self._n_cells:
            raise IndexError("cell number out of range")
        b = bisect.bisect_right(self._block_start, i) - 1
        blk = self._blocks[b]
        k = i - self._block_start[b]
        geo = self._geometries[blk.geometry_id]
        adj = self._adj_map.get(i)
        if adj is None:
            if self._adj_array is not None:
                adj = [None if v < 0 else int(v) for v in self._adj_array[i]]
            else:
                adj = [None] * geo.n_sub_geometries()
            self._adj_map[i] = adj
        return Cell(self, geo, blk.node_maps[k], int(blk.region_ids[k]), adj,
                    self._boundary_map.get(i, {}))

    @property
    def cells(self):
        for i in range(self.n_cells):
            yield self.get_cell(i)

    def cells_on_boundary(self, name):
        for c in sorted(self._boundary_cells[self._boundary_id_lookup[name]]):
            yield self.get_cell(c)

    def cells_are_neighbors(self, cell1, cell2):
        """Face number of ``cell1`` shared with ``cell2`` or -1
        (sem/discrete.py:1095-1106)."""
        common = np.isin(cell1.vertex_node_ind, cell2.vertex_node_ind)
        for side, verts in enumerate(cell1.geometry.corner_verts):
            if np.all(common == verts):
                return side
        return -1

    def boundary_node_ind(self, name):
        """Node ids of all faces on the named boundary, in the order
        ``DOFManager.boundary_elements(name)`` visits them (cells ascending,
        faces in insertion order)."""
        bnd_id = self._boundary_id_lookup[name]
        maps = self.node_map_array()
        if maps.ndim != 3:
            raise NotImplementedError("boundary_node_ind needs 2-D cells")
        pairs = sorted(self._boundary_faces[bnd_id], key=lambda cf: cf[0])  # stable
        if not pairs:
            return np.zeros(0, dtype=np.uint32)
        cells = np.array([c for c, _ in pairs])
        faces = np.array([f for _, f in pairs])
        out = np.empty((len(pairs), max(maps.shape[1:])), dtype=np.uint32)
        width = np.empty(len(pairs), dtype=int)
        for f in np.unique(faces):
            sel = np.nonzero(faces == f)[0]
            sl = _subface_slice(int(f), maps[cells[sel]], 2)
            out[sel, :sl.shape[1]] = sl
            width[sel] = sl.shape[1]
        if (width == out.shape[1]).all():
            return out.ravel()
        return np.concatenate([out[i, :width[i]] for i in range(len(pairs))])

    # -- derived data / renumbering --------------------------------------------------------
    def _compute_cell_centroids(self):
        """Mean of the vertex coordinates of each cell (2-D, like the
        reference, sem/discrete.py:1108-1113)."""
        cent = np.zeros((self.n_cells, 2))
        for blk, start in zip(self._blocks_flushed(), self._block_start):
            geo = self._geometries[blk.geometry_id]
            vid = blk.node_maps.reshape(blk.n_cells, -1)[:, geo.vertex_node_ind]
            cent[start:start + blk.n_cells] = self.nodes[:, vid].mean(axis=2).T
        self._centroids = cent

    def _permute_nodes(self, perm):
        """New node k is old node perm[k]: permutes the coordinate columns in
        place and rewrites every node map through the inverse permutation
        (sem/discrete.py:1115-1127)."""
        self.nodes[:, :perm.size] = self.nodes[:, perm]
        # inverse permutation in the node maps' own dtype (uint32): half the gather traffic
        inv = np.zeros(perm.size, dtype=np.uint32 if perm.size < 2 ** 32 else perm.dtype)
        inv[perm] = np.arange(perm.size, dtype=inv.dtype)
        for blk in self._blocks_flushed():
            blk.node_maps[...] = inv[blk.node_maps]
