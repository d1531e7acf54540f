"""Axisymmetric Stokes / Navier-Stokes in stream function - vorticity form on the GPU
(SURVEY.md 8(f) row 3, BASELINE config 4; additive API).

The reference has this system only as an example script: examples/squirmer-axisymmetric.py
builds dense 4-index local operators ``E2e, Lve`` and Kronecker-sparse ``Ae, Me`` per
element in Python (`pre_assembly`, :163-257), dense local Jacobians / residuals
(`compute_local_system`, :259-297), a Schur-complement COO system and SuperLU inside a
Newton loop (`solve`, :389-457).  ``AxisymmetricStokesOperator`` is the matrix-free
replacement: two DOFs per node (DOF id = 2*node + comp, comp 0 = stream function, 1 =
vorticity; sem/discrete.py:561-576), vectors are ``torch.float64`` CUDA tensors of length
``2*n_nodes`` in the reference's global DOF order.

    dm  = DOFManagerSC(mesh, 2, basis)                       # or DOFManager
    op  = dm.axisymmetric_stokes_operator(n_rey=0.0)
    bc  = squirmer_boundary_data(dm, speed=1.0, slip_vel=...)  # the example's BC recipe
    op.set_essential(bc.essential)
    y   = op.apply(u)                 # y = J u, J = [[Ae.w, Ae.psi + Lve], [E2e, -Me]]
    res = op.residual(state)          # nonlinear residual (assembled res_l)
    state, info = op.newton_solve(bc.state0, bc.cint)   # Newton + restarted GMRES

Every number is computed by the CUDA kernels behind the C ABI (csrc/semk_stokes.cu); the
host side holds the Hessenberg least-squares problem of GMRES (a few dozen doubles).
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _lib, device
from .operators import PoissonOperator, _TILES

__all__ = ["AxisymmetricStokesOperator", "GMRESInfo", "PoissonBlockPreconditioner",
           "squirmer_boundary_data", "squirmer_force", "squirmer_speed",
           "sfn_potential", "sfn_free_stream", "squirmer_vslip_profile", "zero_slip_vel"]

N_FAC_STOKES, N_FAC_ADV = 7, 12
_SMEM_TARGET = 75 * 1024      # three persistent CTAs per SM
_SMEM_LIMIT = 227 * 1024


def f_patch_stride_of(n1, pe, n_fac):
    n = n_fac * n1 * n1 * pe
    return n + (n & 1)


def choose_stokes_elems_per_patch(n1, n_fac):
    """Largest patch (8 or 4 elements) whose shared-memory footprint lets three CTAs share
    an SM; else the largest that fits."""
    lib = _lib.load()
    p = n1 - 1

    def est(pe):
        bx, by = _TILES[pe]
        mpn = ((bx * p + 1) * (by * p + 1) + 3) & ~3
        el = (n1 * n1 * pe + 7) & ~7
        return int(lib.semk_stokes_smem_bytes(n1, pe, f_patch_stride_of(n1, pe, n_fac), mpn, el,
                                              4 * mpn))
    for pe in (8, 4):
        if est(pe) <= _SMEM_TARGET:
            return pe
    for pe in (8, 4):
        if est(pe) <= _SMEM_LIMIT:
            return pe
    raise NotImplementedError("no patch size fits shared memory for n1=%d" % n1)


class GMRESInfo(object):
    __slots__ = ("iterations", "restarts", "converged", "rel_residual", "bnorm",
                 "true_rel_residual")

    def __init__(self, iterations, restarts, converged, rel_residual, bnorm,
                 true_rel_residual=None):
        self.iterations, self.restarts = int(iterations), int(restarts)
        self.converged = bool(converged)
        self.rel_residual, self.bnorm = float(rel_residual), float(bnorm)
        self.true_rel_residual = true_rel_residual

    def __repr__(self):
        return ("GMRESInfo(iterations=%d, restarts=%d, converged=%s, rel_residual=%.3e)"
                % (self.iterations, self.restarts, self.converged, self.rel_residual))


class AxisymmetricStokesOperator(object):
    def __init__(self, dof_mngr, n_rey=0.0, essential=None, elems_per_patch=None,
                 geometric_factors=None, advection=None):
        """n_rey: Reynolds number (examples/squirmer-axisymmetric.py:163); with 0 the system
        is the linear Stokes problem.  advection: force the 12-factor block (default:
        n_rey != 0).  geometric_factors: optional (invJ[E,2,2,N,N], detJxW[E,N,N],
        x_phys[E,2,N,N]) from outside (the reference's own fe.invJ / fe.detJxW / fe.x_phys:
        parity tier T1) instead of the device geometry kernel."""
        _lib.require_device()
        if dof_mngr.ndof_per_node != 2:
            raise ValueError("the stream function - vorticity system needs dofs_per_node = 2")
        self._lib = _lib.load()
        self.dof_mngr = dof_mngr
        self.n_rey = float(n_rey)
        self.advection = bool(self.n_rey != 0.0 if advection is None else advection)
        self.n_fac = N_FAC_ADV if self.advection else N_FAC_STOKES
        tab = device.basis_tables(dof_mngr._basis)
        n1 = tab.n1
        pe = int(elems_per_patch or choose_stokes_elems_per_patch(n1, self.n_fac))
        if pe not in (4, 8):
            raise ValueError("elems_per_patch must be 4 or 8 for the two-field kernel")
        # plan tables, JxW, element order: the scalar operator's (same mesh, same patches)
        po = self._po = PoissonOperator(dof_mngr, elems_per_patch=pe, keep_l2g=True)
        self.tab, self.n1, self.elems_per_patch = tab, n1, pe
        self.n_elem, self.n_nodes, self.n_order = po.n_elem, po.n_nodes, po.n_order
        self.n_dof = 2 * self.n_nodes
        self.dev = po.dev
        NN = n1 * n1
        f64 = dict(dtype=torch.float64, device=self.dev)
        mesh = dof_mngr.mesh
        if geometric_factors is None:
            nodes_dev = device._f64(mesh.nodes, self.dev)
            self.invJ = torch.empty((self.n_elem, 4, NN), **f64)
            self.x_phys = torch.empty((self.n_elem, 2, NN), **f64)
            self.JxW = po.JxW
            J = torch.empty((self.n_elem, 4, NN), **f64)
            detJ = torch.empty((self.n_elem, NN), **f64)
            device.geom_factors(tab, nodes_dev, po.l2g_dev, self.n_elem, x_phys=self.x_phys, J=J,
                                invJ=self.invJ, detJ=detJ)
            del J, detJ, nodes_dev
        else:
            invJ, jxw, xph = geometric_factors
            self.invJ = device._f64(np.asarray(invJ).reshape(self.n_elem, 4, NN), self.dev)
            self.JxW = device._f64(np.asarray(jxw).reshape(self.n_elem, NN), self.dev)
            self.x_phys = device._f64(np.asarray(xph).reshape(self.n_elem, 2, NN), self.dev)
        self.f_patch_stride = f_patch_stride_of(n1, pe, self.n_fac)
        self.F = torch.zeros((po.n_patch, self.f_patch_stride), **f64)
        self._eos = po._tables[_lib.PA_ELEM_OF_SLOT]
        _lib.check(self._lib.semk_stokes_factors_f64(
            n1, self.n_order, device.ptr(self.invJ), device.ptr(self.JxW), device.ptr(self.x_phys),
            device.ptr(self._eos), device.ptr(self.F), self.f_patch_stride, pe,
            device.stream_ptr()))
        self.slot_buf = torch.zeros(2 * max(po.n_slots, 1), **f64)
        sop = _lib.semk_stokes_op()
        C.memmove(C.byref(sop.plan), C.byref(po._op), C.sizeof(_lib.semk_op))
        sop.plan.G = self.F.data_ptr()
        sop.plan.g_patch_stride = self.f_patch_stride
        sop.plan.slot_buf = self.slot_buf.data_ptr()
        sop.plan.dirichlet = None
        sop.plan.max_ctas = 0
        sop.n_fac = self.n_fac
        sop.n_ess = 0
        sop.ess_dof = None
        self._sop = sop
        self.smem_bytes = int(self._lib.semk_stokes_smem_bytes(
            n1, pe, self.f_patch_stride, po.plan_scalars[_lib.PS_PN_STRIDE],
            po.plan_scalars[_lib.PS_EL_STRIDE], po.plan_scalars[_lib.PS_INV_STRIDE]))
        self.essential_host = None
        self._ess_dev = None
        self._binv = None
        self._linearized = not self.advection
        if essential is not None:
            self.set_essential(essential)

    # -- helpers ---------------------------------------------------------------------
    def _vec(self, v, name="vector"):
        if not (isinstance(v, torch.Tensor) and v.is_cuda and v.dtype == torch.float64
                and v.is_contiguous() and v.numel() == self.n_dof):
            raise ValueError("%s must be a contiguous float64 CUDA tensor of length 2*n_nodes"
                             % name)
        return v

    def new_vector(self, fill=None):
        if fill is None:
            return torch.empty(self.n_dof, dtype=torch.float64, device=self.dev)
        return torch.full((self.n_dof,), float(fill), dtype=torch.float64, device=self.dev)

    def from_host(self, a):
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(self.dev)

    @property
    def algorithmic_bytes_per_apply(self):
        """read (psi, omega), write both rows, n_fac factors + one uint32 L2G entry per
        element-local node (the two-field analogue of SURVEY.md 8(d))."""
        return 32 * self.n_nodes + (8 * self.n_fac + 4) * self.n_elem * self.n1 * self.n1

    def set_essential(self, essential):
        """essential: bool[2*n_nodes] (or bool[ndof_exterior], padded with False), True =
        essential-BC DOF -- the complement of the example's ``dof_mask``
        (examples/squirmer-axisymmetric.py:102,366)."""
        essential = np.asarray(essential)
        if essential.dtype != np.bool_ or essential.ndim != 1 or essential.size > self.n_dof:
            raise ValueError("essential must be bool[<= 2*n_nodes]")
        full = np.zeros(self.n_dof, dtype=bool)
        full[:essential.size] = essential
        self.essential_host = full
        ids = np.flatnonzero(full).astype(np.int64)
        self._ess_dev = torch.from_numpy(ids).to(self.dev)
        self._sop.n_ess = int(ids.size)
        self._sop.ess_dof = self._ess_dev.data_ptr() if ids.size else None
        self._binv = None

    def _fix(self, y, src=None):
        if self._sop.n_ess:
            _lib.check(self._lib.semk_scatter_fix_f64(
                self._sop.n_ess, device.ptr(self._ess_dev), device.ptr(src), device.ptr(y),
                device.stream_ptr()))
        return y

    # -- operator --------------------------------------------------------------------
    def _apply_raw(self, u, y, zero_rows, adv_scale=1.0):
        if self.advection and not self._linearized:
            raise RuntimeError("call linearize(state) before applying the Jacobian (n_rey != 0)")
        _lib.check(self._lib.semk_stokes_apply_f64(
            C.byref(self._sop), device.ptr(u), device.ptr(y), int(bool(zero_rows)),
            float(adv_scale), device.stream_ptr()))
        return y

    def apply_unmasked(self, u, out=None):
        """y = J u: the assembled local Jacobians, no boundary conditions."""
        self._vec(u, "u")
        y = self.new_vector() if out is None else self._vec(out, "out")
        return self._apply_raw(u, y, False)

    def apply(self, u, out=None):
        """y = Jhat u, Jhat = M J M + (I - M): rows and columns of the essential DOFs
        replaced by the identity (the elimination of
        examples/squirmer-axisymmetric.py:362-370 in operator form)."""
        self._vec(u, "u")
        y = self.new_vector() if out is None else self._vec(out, "out")
        if not self._sop.n_ess:
            return self._apply_raw(u, y, False)
        um = self._fix(u.clone())
        self._apply_raw(um, y, True)
        return self._fix(y, u)

    def linearize(self, state):
        """Advection coefficients of the Jacobian about ``state`` (the example recomputes
        ``Ae.dot_dense(vort)`` / ``Ae.dot_dense(sfn)`` per Newton step, :276-283)."""
        if not self.advection:
            return
        self._vec(state, "state")
        po = self._po
        _lib.check(self._lib.semk_stokes_linearize_f64(
            self.n1, self.n_order, device.ptr(self.tab.dev()[0]), device.ptr(self.invJ),
            device.ptr(self.JxW), device.ptr(self.x_phys), device.ptr(po.l2g_dev),
            device.ptr(self._eos), device.ptr(state), self.n_rey, device.ptr(self.F),
            self.f_patch_stride, self.elems_per_patch, device.stream_ptr()))
        self._linearized = True
        self._binv = None

    def residual(self, state, out=None):
        """Assembled nonlinear residual ``res`` of the example (:284-295): the advection
        term is bilinear, so it is the Jacobian about ``state`` applied to ``state`` with
        the advection part halved.  Leaves the operator linearised about ``state``."""
        self._vec(state, "state")
        y = self.new_vector() if out is None else self._vec(out, "out")
        self.linearize(state)
        return self._apply_raw(state, y, False, adv_scale=0.5 if self.advection else 1.0)

    # -- nodal 2x2 block-Jacobi preconditioner ---------------------------------------------
    def block_jacobi(self):
        """Inverse of the node's 2x2 diagonal block [[Ae.w, Lve], [E2e, -Me]] (assembled
        diagonals; identity on essential DOFs), as ``float64[n_nodes, 4]`` row-major."""
        if self._binv is not None:
            return self._binv
        po = self._po
        NN = self.n1 * self.n1
        f64 = dict(dtype=torch.float64, device=self.dev)
        loc = [torch.empty((po.n_slot_elems, NN), **f64) for _ in range(4)]
        _lib.check(self._lib.semk_stokes_local_diag_f64(
            C.byref(self._sop), device.ptr(self.tab.dev()[0]), po.n_slot_elems,
            device.ptr(loc[0]), device.ptr(loc[1]), device.ptr(loc[2]), device.ptr(loc[3]),
            device.stream_ptr()))
        dL, dE, dM, dA = (po.assemble(l) for l in loc)
        self._diagonals = (dL, dE, dM, dA)
        ess = torch.zeros(self.n_dof, dtype=torch.bool, device=self.dev)
        if self._sop.n_ess:
            ess[self._ess_dev] = True
        e0, e1 = ess[0::2], ess[1::2]
        one, zero = torch.ones_like(dL), torch.zeros_like(dL)
        # B = [[a, b], [c, d]]; essential row / column -> identity
        a = torch.where(e0, one, dA)
        b = torch.where(e0 | e1, zero, dL)
        c = torch.where(e0 | e1, zero, dE)
        d = torch.where(e1, one, -dM)
        det = a * d - b * c
        bad = det == 0
        det = torch.where(bad, one, det)
        binv = torch.stack([d / det, -b / det, -c / det, a / det], dim=1)
        binv[bad] = torch.tensor([1.0, 0.0, 0.0, 1.0], **f64)
        self._binv = binv.contiguous()
        return self._binv

    def block_jacobi_diagonals(self):
        """Assembled nodal diagonals (Lve, E2e, Me, advection) behind ``block_jacobi``."""
        self.block_jacobi()
        if getattr(self, "_diagonals", None) is None:
            self._binv = None
            self.block_jacobi()
        return self._diagonals

    # -- restarted GMRES (right preconditioned, CGS2 orthogonalisation) -------------------
    def solve_gmres(self, b, x0=None, rtol=1e-10, restart=60, maxiter=2000, precondition=True,
                    scale_rows=None):
        """Solve Jhat x = b for the unknown DOFs (essential entries of x stay at x0's, b's
        essential entries are ignored).  precondition: True = nodal 2x2 block-Jacobi, False =
        none, "poisson" = PoissonBlockPreconditioner (Re = 0, DOFManagerSC), or a callable
        ``(src, dst)``.  Replaces the sparse direct solve of the Schur
        system (examples/squirmer-axisymmetric.py:360-370).  Returns (x, GMRESInfo)."""
        self._vec(b, "b")
        lib, n = self._lib, self.n_dof
        st = device.stream_ptr
        m = int(max(1, min(restart, maxiter)))
        f64 = dict(dtype=torch.float64, device=self.dev)
        V = torch.empty((m + 1, n), **f64)
        w, z = self.new_vector(), self.new_vector()
        # a preconditioner that contains iterative solves is not one fixed linear operator:
        # FLEXIBLE GMRES keeps z_j = P^-1 v_j, so that x = sum_j y_j z_j satisfies the Arnoldi
        # relation A z_j = V h_j exactly and the recurrence residual is the true one
        flexible = callable(precondition) or precondition == "poisson"
        Z = torch.empty((m, n), **f64) if flexible else None
        x = torch.zeros(n, **f64) if x0 is None else self._vec(x0, "x0").clone()
        bb = self._fix(b.clone())
        hdev = torch.empty(m + 2, **f64)
        partials = torch.empty(int(lib.semk_multi_dot_partials_len(m + 2)), **f64)
        custom = precondition if callable(precondition) else None
        if precondition == "poisson":
            custom = self._poisson_prec = (getattr(self, "_poisson_prec", None)
                                           or PoissonBlockPreconditioner(self))
        binv = self.block_jacobi() if (precondition and custom is None) else None
        # Row equilibration (default with the Poisson preconditioner): the rows of the system
        # differ by eight orders of magnitude on the graded annulus (rho^2 JxW against rho),
        # so a tolerance on ||b - A x||_2 says little about the small rows.  Solve
        # (D A) x = D b, D = 1 / diag(Lve) on the wte rows and 1 / diag(E2e) on the wdef rows;
        # the preconditioner of D A is P^-1 D^-1 (a similarity transform of A P^-1).  All
        # residuals reported are those of the scaled system.
        if scale_rows is None:
            scale_rows = precondition == "poisson"
        D = Dinv = None
        if scale_rows:
            dL, dE = self.block_jacobi_diagonals()[:2]
            D = torch.ones(n, **f64)
            D[0::2] = torch.where(dL != 0, 1.0 / dL, torch.ones_like(dL))
            D[1::2] = torch.where(dE != 0, 1.0 / dE, torch.ones_like(dE))
            self._fix(D, torch.ones(n, **f64))
            Dinv = 1.0 / D
            tmp = self.new_vector()

        def scale(d, vec, out):
            _lib.check(lib.semk_vec_scale_f64(n, device.ptr(d), device.ptr(vec), device.ptr(out),
                                              st()))
            return out
        if D is not None:
            scale(D, bb, bb)

        def dots(k, vec):
            _lib.check(lib.semk_multi_dot_f64(n, k, device.ptr(V), n, device.ptr(vec),
                                              device.ptr(hdev), device.ptr(partials), st()))
            return hdev[:k].cpu().numpy()

        def norm(vec):
            _lib.check(lib.semk_multi_dot_f64(n, 1, device.ptr(vec), n, device.ptr(vec),
                                              device.ptr(hdev), device.ptr(partials), st()))
            return math.sqrt(max(float(hdev[0].item()), 0.0))

        def precond(src, dst):
            if Dinv is not None:
                src = scale(Dinv, src, tmp)
            if custom is not None:
                custom(src, dst)
            elif binv is None:
                dst.copy_(src)
            else:
                _lib.check(lib.semk_block2_apply_f64(self.n_nodes, device.ptr(binv),
                                                     device.ptr(src), device.ptr(dst), st()))
            return dst

        bnorm = norm(bb)
        if bnorm == 0.0:
            return x, GMRESInfo(0, 0, True, 0.0, 0.0)
        total, restarts, rel = 0, 0, 1.0
        converged = False
        last_true = float("inf")
        while total < maxiter:
            # TRUE residual r = b - Jhat x on the unknowns at the start of every cycle (x's
            # essential entries do not enter: masked).  A cycle that ended on the recurrence
            # residual is only accepted when the true residual agrees (iterative refinement:
            # the next cycle solves for the correction); if a cycle no longer halves the true
            # residual the attainable accuracy of the system has been reached
            xm = self._fix(x.clone())
            self._apply_raw(xm, w, True)
            if D is not None:
                scale(D, w, w)
            _lib.check(lib.semk_vec_scale_add_f64(n, -1.0, device.ptr(w), device.ptr(bb),
                                                  device.ptr(V[0]), st()))
            beta = norm(V[0])
            rel = beta / bnorm
            if rel <= rtol:
                converged = True
                break
            if rel > 0.5 * last_true:
                break
            last_true = rel
            _lib.check(lib.semk_vec_scale_add_f64(n, 1.0 / beta, device.ptr(V[0]), None,
                                                  device.ptr(V[0]), st()))
            H = np.zeros((m + 1, m))
            cs, sn = np.zeros(m), np.zeros(m)
            g = np.zeros(m + 1)
            g[0] = beta
            k_used = 0
            for j in range(m):
                zj = Z[j] if flexible else z
                precond(V[j], zj)
                self._apply_raw(zj, V[j + 1], True)
                if D is not None:
                    scale(D, V[j + 1], V[j + 1])
                h = dots(j + 1, V[j + 1]).copy()
                _lib.check(lib.semk_multi_axpy_f64(n, j + 1, device.ptr(V), n, device.ptr(hdev),
                                                   -1.0, device.ptr(V[j + 1]), st()))
                # second Gram-Schmidt pass; the last entry is ||w||^2 (w is row j+1 of V)
                h2 = dots(j + 2, V[j + 1])
                _lib.check(lib.semk_multi_axpy_f64(n, j + 1, device.ptr(V), n, device.ptr(hdev),
                                                   -1.0, device.ptr(V[j + 1]), st()))
                h += h2[:j + 1]
                hn2 = h2[j + 1] - float(np.dot(h2[:j + 1], h2[:j + 1]))
                hn = math.sqrt(hn2) if hn2 > 0.0 else 0.0
                H[:j + 1, j] = h
                H[j + 1, j] = hn
                for i in range(j):                       # previous rotations
                    t = cs[i] * H[i, j] + sn[i] * H[i + 1, j]
                    H[i + 1, j] = -sn[i] * H[i, j] + cs[i] * H[i + 1, j]
                    H[i, j] = t
                den = math.hypot(H[j, j], H[j + 1, j])
                cs[j], sn[j] = (1.0, 0.0) if den == 0.0 else (H[j, j] / den, H[j + 1, j] / den)
                H[j, j] = den
                H[j + 1, j] = 0.0
                g[j + 1] = -sn[j] * g[j]
                g[j] = cs[j] * g[j]
                total += 1
                k_used = j + 1
                rel = abs(g[j + 1]) / bnorm
                if hn == 0.0 or rel <= rtol or total >= maxiter:
                    break
                _lib.check(lib.semk_vec_scale_add_f64(n, 1.0 / hn, device.ptr(V[j + 1]), None,
                                                      device.ptr(V[j + 1]), st()))
            yk = np.linalg.solve(np.triu(H[:k_used, :k_used]), g[:k_used])
            hdev[:k_used] = torch.from_numpy(yk).to(self.dev)
            if flexible:
                _lib.check(lib.semk_multi_axpy_f64(n, k_used, device.ptr(Z), n, device.ptr(hdev),
                                                   1.0, device.ptr(x), st()))
            else:
                w.zero_()
                _lib.check(lib.semk_multi_axpy_f64(n, k_used, device.ptr(V), n, device.ptr(hdev),
                                                   1.0, device.ptr(w), st()))
                precond(w, z)
                _lib.check(lib.semk_vec_scale_add_f64(n, 1.0, device.ptr(z), device.ptr(x),
                                                      device.ptr(x), st()))
            restarts += 1
        # true residual of the returned iterate
        xm = self._fix(x.clone())
        self._apply_raw(xm, w, True)
        if D is not None:
            scale(D, w, w)
        _lib.check(lib.semk_vec_scale_add_f64(n, -1.0, device.ptr(w), device.ptr(bb),
                                              device.ptr(w), st()))
        true_rel = norm(w) / bnorm
        return x, GMRESInfo(total, restarts, converged, rel, bnorm, true_rel)

    # -- Newton driver -----------------------------------------------------------------
    def newton_solve(self, state0, cint=None, it_max=10, tol=1e-6, max_n_diverge=3,
                     gmres_rtol=1e-10, restart=60, gmres_maxiter=4000, verbose=False,
                     precondition=True):
        """Newton-Raphson of examples/squirmer-axisymmetric.py:389-457 with the Schur /
        SuperLU step replaced by GMRES on the matrix-free Jacobian.  state0 holds the
        initial guess with the essential values in place; cint: natural-BC contour
        integrals (length <= 2*n_nodes, zero-padded).  Convergence test and divergence
        counter as in the example (norm of the vorticity increment).  Returns
        (state, list of (||d_vort||, GMRESInfo))."""
        from ._lib import SolverFailure
        state = self._vec(state0, "state0").clone()
        c = torch.zeros(self.n_dof, dtype=torch.float64, device=self.dev)
        if cint is not None:
            cv = cint if isinstance(cint, torch.Tensor) else self.from_host(cint)
            c[:cv.numel()] = cv
        history = []
        n_diverge, last = 0, float("inf")
        for itn in range(it_max):
            res = self.residual(state)
            rhs = c - res
            d, info = self.solve_gmres(rhs, rtol=gmres_rtol, restart=restart,
                                       maxiter=gmres_maxiter, precondition=precondition)
            self._fix(d)
            state += d
            du = float(torch.linalg.vector_norm(d[1::2]).item())
            history.append((du, info))
            if verbose:
                print("[Iteration %d]: ||du|| = %g  (%r)" % (itn, du, info))
            if du > last:
                n_diverge += 1
                if n_diverge >= max_n_diverge:
                    raise SolverFailure("Solution diverged %d times (||du|| = %g)"
                                        % (n_diverge, du))
            if abs(du) <= tol:
                return state, history
            last = du
        raise SolverFailure("Calculation failed to reach specified tolerance after %d Newton "
                            "iterations (||du|| = %g)" % (it_max, history[-1][0]))

    # -- small-mesh test helper ----------------------------------------------------------
    def to_scipy_csr(self, masked=False):
        from scipy import sparse
        n = self.n_dof
        if n > 20000:
            raise ValueError("to_scipy_csr is meant for small meshes")
        cols = []
        e = self.new_vector(0.0)
        y = self.new_vector()
        for j in range(n):
            e[j] = 1.0
            (self.apply if masked else self.apply_unmasked)(e, out=y)
            e[j] = 0.0
            cols.append(sparse.csc_matrix(y.cpu().numpy().reshape(-1, 1)))
        return sparse.hstack(cols).tocsr()


class PoissonBlockPreconditioner(object):
    """Block-triangular preconditioner of the Stokes (Re = 0) system from ONE weighted Poisson
    operator, for right-preconditioned GMRES (mesh-independent iteration counts in the CPU
    study oracle/precond_study_stokes.py: 72-121 iterations from 345 to 24 257 DOF).

    With I = nodes where the stream function is unknown, G = nodes where it is essential but
    the vorticity is not (the sphere), rows wte (L om = a) paired with om_I and rows wdef
    (E psi - M om = b) paired with psi_I / om_G:
        om_G = -b_G / M_G
        om_I = Khat^-1 (a - L_IG om_G)
        psi  = Khat^-1 (b_I + M_I om_I)
    Khat = Lve on I (rho-weighted stiffness + the JxW/rho reaction term) with Dirichlet rows on
    every psi-essential node: the statically condensed operator of section 7 row 1
    (``condensed_poisson_operator(weight=rho, reaction=JxW/rho)``) solved by the native
    multilevel PCG driver to ``rtol``; the inner solves are iterative, so the outer method is
    FLEXIBLE GMRES and convergence is accepted on the true residual.
    Needs a ``DOFManagerSC`` (exterior-first numbering) built with ``rcm_order=False``.
    The glue between the solves is three small C-ABI kernels (semk_stokes_prec_*_f64)."""

    def __init__(self, op, rtol=1e-8, preconditioner="three-level", reaction_term=True):
        from . import discrete
        # (with advection, n_rey != 0, the same Stokes blocks precondition the linearised
        # Navier-Stokes Jacobian: the advection terms are first order; flexible GMRES absorbs
        # the difference at moderate Reynolds numbers)
        dm = op.dof_mngr
        mesh = dm.mesh
        if not getattr(mesh, "condensed", False):
            raise ValueError("needs the exterior-first numbering of DOFManagerSC")
        if op.essential_host is None:
            raise ValueError("set the essential DOFs first (set_essential)")
        ess_s, ess_w = op.essential_host[0::2], op.essential_host[1::2]
        if (ess_w & ~ess_s).any():
            raise NotImplementedError("vorticity essential where the stream function is free")
        self.op, self.rtol, self.kind = op, float(rtol), preconditioner
        before = mesh.node_map_array().copy()
        sdm = discrete.DOFManagerSC(mesh, 1, dm._basis, rcm_order=False)
        if not np.array_equal(before, mesh.node_map_array()):
            raise AssertionError("the scalar manager renumbered the mesh: build the Stokes "
                                 "manager as DOFManagerSC(mesh, 2, basis, rcm_order=False)")
        # Khat = Lve restricted to I: rho-weighted stiffness + the JxW/rho reaction term (the
        # CPU study needs a third fewer outer iterations with it than with the bare stiffness)
        reaction = None
        if reaction_term:
            rho = op.x_phys[:, 0, :]
            reaction = torch.where(rho > 0, op.JxW / rho.clamp_min(1e-300), torch.zeros_like(rho))
        self.sc = sdm.condensed_poisson_operator(dirichlet=ess_s, weight=lambda x, y: x,
                                                 reaction=reaction, store_interior=True,
                                                 store_interior_inverse=True)
        dev = op.dev
        self.free_s = torch.from_numpy(~ess_s).to(dev)                 # I
        self.gamma = torch.from_numpy(ess_s & ~ess_w).to(dev)          # G
        self.n_ext = self.sc.n_ext
        # lumped element-interior weights: f_nodal = r / JxW reproduces the interior load r
        # (interior nodes are private to their element), 0 on exterior nodes
        mass = op._po.assemble(self._local_jxw(op))
        inv = torch.zeros_like(mass)
        inv[self.n_ext:] = 1.0 / mass[self.n_ext:]
        self.inv_mass_int = inv
        dM = op.block_jacobi_diagonals()[2]
        self.M = dM
        self.neg_inv_M_gamma = torch.where(self.gamma, -1.0 / dM, torch.zeros_like(dM))
        self.free_u8 = self.free_s.to(torch.uint8).contiguous()
        f64 = dict(dtype=torch.float64, device=dev)
        self._t, self._y = torch.empty(op.n_dof, **f64), torch.empty(op.n_dof, **f64)
        self._r, self._f = torch.empty(op.n_nodes, **f64), torch.empty(op.n_nodes, **f64)
        self.solves = 0
        self.inner_outer_iterations = 0

    @staticmethod
    def _local_jxw(op):
        """JxW in engine slot order (zeros in the empty padding slots)."""
        po = op._po
        NN = op.n1 * op.n1
        loc = torch.zeros((po.n_slot_elems, NN), dtype=torch.float64, device=op.dev)
        eos = po._tables[_lib.PA_ELEM_OF_SLOT]
        ok = eos >= 0
        loc[:eos.numel()][ok] = po.JxW[eos[ok]]
        return loc

    def poisson_solve(self, r, f=None):
        """u = Khat^-1 r for a nodal residual r (zero on the Dirichlet nodes); f = r *
        inv_mass_int if the caller has it already."""
        if f is None:
            f = r * self.inv_mass_int
        u, info = self.sc.solve_load(r, f, rtol=self.rtol, preconditioner=self.kind)
        self.solves += 1
        self.inner_outer_iterations += info.iterations
        return u

    def __call__(self, src, dst):
        op, lib, n = self.op, self.op._lib, self.op.n_nodes
        st = device.stream_ptr
        t, r, f = self._t, self._r, self._f
        _lib.check(lib.semk_stokes_prec_gamma_f64(n, device.ptr(src), device.ptr(
            self.neg_inv_M_gamma), device.ptr(t), st()))                    # om_G
        y = op.apply_unmasked(t, out=self._y)                               # row 0 = L om_G
        _lib.check(lib.semk_stokes_prec_rhs_f64(
            n, 0, device.ptr(src), device.ptr(y), None, None, device.ptr(self.free_u8),
            device.ptr(self.inv_mass_int), device.ptr(r), device.ptr(f), st()))
        om_i = self.poisson_solve(r, f)
        _lib.check(lib.semk_stokes_prec_rhs_f64(
            n, 1, device.ptr(src), None, device.ptr(self.M), device.ptr(om_i),
            device.ptr(self.free_u8), device.ptr(self.inv_mass_int), device.ptr(r), device.ptr(f),
            st()))
        psi = self.poisson_solve(r, f)
        _lib.check(lib.semk_stokes_prec_out_f64(n, device.ptr(self.free_u8), device.ptr(psi),
                                                device.ptr(om_i), device.ptr(t), device.ptr(dst),
                                                st()))
        return dst


# --------------------------------------------------------------------------------------
# The example's problem data (examples/squirmer-axisymmetric.py:17-46,109-161)
# --------------------------------------------------------------------------------------
def squirmer_vslip_profile(beta):
    def vslip(sin_th, cos_th):
        return 3. / 2 * sin_th * (1. + beta * cos_th)
    return vslip


def zero_slip_vel(sin_th, cos_th):
    return np.zeros_like(sin_th)


def sfn_potential(rho, z):
    """Stream function of irrotational flow past the unit sphere (:27-37)."""
    r = np.sqrt(rho ** 2 + z ** 2)
    sin_th = rho / r
    return -(r ** 2 - 1 / r) / 2. * sin_th ** 2


def sfn_free_stream(rho, z):
    r = np.sqrt(rho ** 2 + z ** 2)
    sin_th = rho / r
    return 0.5 * (r * sin_th) ** 2


class SquirmerBoundaryData(object):
    """state0: initial guess with essential values; essential: bool[2 n_nodes]; cint:
    natural-BC contour integrals [2 n_nodes]."""
    __slots__ = ("state0", "essential", "cint")

    def __init__(self, state0, essential, cint):
        self.state0, self.essential, self.cint = state0, essential, cint


def squirmer_boundary_data(dof_mngr, speed=1.0, slip_vel=zero_slip_vel, x_phys=None):
    """Initial guess and boundary conditions of the example, through the drop-in API:
    `set_initial_guess` (:109-117: potential flow) and `_apply_bcs_to_fe` (:119-161):
      "sphere":  sfn = 0 essential; natural BC on the vorticity-definition row
                 cint -= xweight(rho * rho (n_rho v_z - n_z v_rho)), n = -n_dS (from the body
                 into the fluid);
      "symaxis": sfn = vort = 0 essential;
      "shell":   sfn = -speed * free stream, vort = 0 essential.
    x_phys: optional host [E, 2, N, N] GLL-point coordinates (saves one geometry pass)."""
    mesh = dof_mngr.mesh
    n = mesh.n_nodes
    sfn, vort = np.zeros(n), np.zeros(n)
    ess_s, ess_w = np.zeros(n, dtype=bool), np.zeros(n, dtype=bool)
    cint_w = np.zeros(n)
    l2g = mesh.node_map_array()
    N = l2g.shape[-1]
    if x_phys is None:
        x_phys = device.element_geometry(dof_mngr._map_basis, mesh.nodes,
                                         l2g.reshape(-1, N * N), jacobian=False)["x_phys"]
    with np.errstate(invalid="ignore", divide="ignore"):
        sfn[l2g.reshape(-1)] = sfn_potential(x_phys[:, 0].reshape(-1), x_phys[:, 1].reshape(-1))
    for name in ("sphere", "symaxis", "shell"):
        for _parent, bnd in dof_mngr.boundary_elements(name, x_phys=True, Jacobian=True):
            loc = bnd.node_ind
            if name == "sphere":
                sfn[loc] = 0
                ess_s[loc] = True
                rho, z = bnd.x_phys
                # the example's `bnd_fe.normal()`: non-normalised, from the body into the fluid
                n_rho, n_z = -bnd.n_dS
                r = np.sqrt(rho ** 2 + z ** 2)
                sin_th, cos_th = rho / r, z / r
                v = slip_vel(sin_th, cos_th)
                v_rho, v_z = v * cos_th, -v * sin_th
                n_grad_sfn = rho * (n_rho * v_z - n_z * v_rho)
                cint_w[loc] += -bnd.quadrature.xweight(rho * n_grad_sfn)
            elif name == "symaxis":
                sfn[loc] = 0
                vort[loc] = 0
                ess_s[loc] = True
                ess_w[loc] = True
            else:
                rho, z = bnd.x_phys
                sfn[loc] = -sfn_free_stream(rho, z) * speed
                vort[loc] = 0
                ess_s[loc] = True
                ess_w[loc] = True
    state0 = np.empty(2 * n)
    state0[0::2], state0[1::2] = sfn, vort
    essential = np.empty(2 * n, dtype=bool)
    essential[0::2], essential[1::2] = ess_s, ess_w
    cint = np.zeros(2 * n)
    cint[1::2] = cint_w
    return SquirmerBoundaryData(state0, essential, cint)


def squirmer_force(dof_mngr, soln_vec, slip_vel, n_rey):
    """Total hydrodynamic force on the unit sphere in the swimming direction
    (`calc_force`, examples/squirmer-axisymmetric.py:458-513, through the current API: the
    example's version still uses the package's older element interface).  On r = 1, with
    the polar angle from the +z axis,
        stress = pi Re v_s^2 sin cos + pi (d omega / d r + omega) sin^2 - 2 pi omega sin^2,
    integrated along the arc.  soln_vec: host array [2 n_nodes] (interleaved)."""
    vort = np.asarray(soln_vec, dtype=np.float64)[1::2]
    total = 0.0
    for parent, bnd in dof_mngr.boundary_elements("sphere", x_phys=True, Jacobian=True):
        rho, z = bnd.x_phys                           # r = 1: (sin, cos) of the polar angle
        sin_th, cos_th = rho, z
        vslip = slip_vel(sin_th, cos_th)
        w_loc = vort[parent.node_ind]
        grad = bnd.gradient(w_loc)                    # d omega / d(rho, z) on the face
        dw_dr = grad[0] * rho + grad[1] * z
        w_s = vort[bnd.node_ind]
        sin2 = sin_th ** 2
        bernoulli = np.pi * n_rey * vslip ** 2 * sin_th * cos_th
        w_asym = np.pi * (dw_dr + w_s) * sin2
        viscous = -2 * np.pi * w_s * sin2
        total += float(((bernoulli + w_asym + viscous) * bnd.dSxW).sum())
    return total


def squirmer_speed(dof_mngr, n_rey, beta, speed_guess=(0.99, 1.01), it_max=10, tol=1e-5,
                   newton_tol=1e-6, precondition="poisson", verbose=False, **newton_kw):
    """Swimming speed of a squirmer: secant iteration on the speed at which the force on the
    body vanishes (`calc_speed`, examples/squirmer-axisymmetric.py:630-744), every force
    evaluation a full Newton solve of the flow on the device.  Returns (speed, state,
    list of (speed, force))."""
    from ._lib import SolverFailure
    slip = squirmer_vslip_profile(beta)
    op = None
    x_phys = None
    history = []

    def force_at(speed, guess):
        nonlocal op, x_phys
        if op is None:
            op = dof_mngr.axisymmetric_stokes_operator(n_rey=n_rey)
            N = op.n1
            x_phys = op.x_phys.cpu().numpy().reshape(op.n_elem, 2, N, N)
        bc = squirmer_boundary_data(dof_mngr, speed, slip, x_phys=x_phys)
        op.set_essential(bc.essential)
        op._poisson_prec = None
        s0 = bc.state0 if guess is None else np.where(bc.essential, bc.state0, guess)
        state, _ = op.newton_solve(op.from_host(s0), bc.cint, tol=newton_tol,
                                   precondition=precondition, **newton_kw)
        sol = state.cpu().numpy()
        f = squirmer_force(dof_mngr, sol, slip, n_rey)
        history.append((float(speed), f))
        if verbose:
            print("speed = %.10g  =>  force = %.6e" % (speed, f))
        return f, sol

    speed0, speed1 = (float(v) for v in speed_guess)
    if speed0 == speed1:
        raise ValueError("Two distinct guesses for the speed must be supplied.")
    force0, sol = force_at(speed0, None)
    force1, sol = force_at(speed1, sol)
    for _ in range(it_max):
        speed2 = (speed1 * force0 - speed0 * force1) / (force0 - force1)
        force2, sol = force_at(speed2, sol)
        if abs(speed2 - speed1) < tol:
            return speed2, sol, history
        speed0, speed1, force0, force1 = speed1, speed2, force1, force2
    raise SolverFailure("Swimming speed could not be found within the desired tolerance in "
                        "the max number of iterations (%d)." % it_max)
