// semk_geom.cu -- K1: per-element geometric factors (set-up, runs once per mesh).
//
// Reference being replaced, per element (all Python/NumPy/LAPACK there):
//   x_phys  = compute_coeffs_grid_eq(mesh.nodes[:, L2G])     sem/mapping.py:98-103,
//             two lu_solve sweeps with the equispaced->GLL matrix E
//                                                   sem/basis_functions.py:599-624
//   J[i,a]  = d x_i / d xi_a = gradient(x_phys).swapaxes(0,1)   sem/mapping.py:113
//   detJ, invJ = det_inv_2x2(J)  (adjugate * (1/det))        sem/linalg.py:105-115
//   JxW     = (detJ * w_m) * w_n                          sem/quadratures.py:268-275
//   G_ab    = JxW * sum_i invJ[a,i] invJ[b,i]  (implicit in examples/poisson.py:166-193)
//
// Differences by design (SURVEY.md section 0 fact 5 / hard part 7): E^{-1} is
// applied as an explicit, correctly rounded matrix instead of an LU solve, and
// an element-local origin is subtracted before the contractions so that the
// cancellation in J = D x does not grow with 1/h.  One CTA per element slot,
// one thread per node; this kernel is not on the per-iteration path.
#include "semk_common.cuh"

namespace {

// K1's arithmetic for node k = (m, n) of element `row` (its L2G row), shared by geom_kernel
// and field_grad_kernel so that the two cannot drift apart: gather the equispaced nodes,
// subtract the element-local origin (node 0), E^{-1} on axis 0 then axis 1 (GLL
// coefficients of x - origin, left in sA), J = D x, the closed-form 2x2 inverse and
// JxW = detJ w_m w_n.  Sets *bad_flag on detJ <= 0.  Every thread of the CTA calls it (it
// synchronises); the results are meaningful where `on`.  On return sB is free and sA is
// still read by no one.
struct NodeGeom {
  double ox, oy, xg, yg;        // origin; x_phys - origin at the node
  double j00, j01, j10, j11;    // J[i][a] = d x_i / d xi_a
  double det, i00, i01, i10, i11, jw;
};

template <int N>
__device__ __forceinline__ NodeGeom node_geometry(const uint32_t *__restrict__ row,
                                                  const double *__restrict__ nodes_x,
                                                  const double *__restrict__ nodes_y,
                                                  const double *sE, const double *sD,
                                                  const double *sw, double (*sA)[N * N],
                                                  double (*sB)[N * N], int k, bool on, int m,
                                                  int n, int32_t *__restrict__ bad_flag) {
  NodeGeom r;
  const uint32_t g0 = row[0];
  r.ox = nodes_x[g0];
  r.oy = nodes_y[g0];
  __syncthreads();  // tables loaded / previous iteration done with sA, sB
  if (on) {
    const uint32_t g = row[k];
    sA[0][k] = __dsub_rn(nodes_x[g], r.ox);
    sA[1][k] = __dsub_rn(nodes_y[g], r.oy);
  }
  __syncthreads();
  // equispaced values -> GLL coefficients: axis 0, then axis 1
  double t0 = 0.0, t1 = 0.0;
  if (on) {
#pragma unroll
    for (int q = 0; q < N; ++q) {
      const double c = sE[m * N + q];
      t0 = fma(c, sA[0][q * N + n], t0);
      t1 = fma(c, sA[1][q * N + n], t1);
    }
    sB[0][k] = t0;
    sB[1][k] = t1;
  }
  // Axis-aligned element: x depends on m only and y on n only (or, rotated by 90 degrees,
  // x on n and y on m).  Then J01 = J10 = 0 (J00 = J11 = 0) in exact arithmetic -- E^{-1}
  // reproduces constants and D annihilates them -- and the roundoff J = D x would leave
  // there is dropped, so that G01 comes out as an exact zero (the separable apply).  The
  // dropped products lie far below an ulp of det, invJ's other entries, G00 and G11.
  const bool x_m = !on || (sA[0][k] == sA[0][m * N] && sA[1][k] == sA[1][n]);
  const bool x_n = !on || (sA[0][k] == sA[0][n] && sA[1][k] == sA[1][m * N]);
  const bool axis_mn = __syncthreads_and(x_m) != 0;
  const bool axis_nm = !axis_mn && __syncthreads_and(x_n) != 0;  // (uniform branch)
  r.xg = 0.0;
  r.yg = 0.0;
  if (on) {
#pragma unroll
    for (int s = 0; s < N; ++s) {
      const double c = sE[n * N + s];
      r.xg = fma(c, sB[0][m * N + s], r.xg);
      r.yg = fma(c, sB[1][m * N + s], r.yg);
    }
    sA[0][k] = r.xg;  // all reads of sA happened before the previous barrier
    sA[1][k] = r.yg;
  }
  __syncthreads();
  if (on) {
    double j00 = 0.0, j01 = 0.0, j10 = 0.0, j11 = 0.0;
#pragma unroll
    for (int q = 0; q < N; ++q) {
      const double d0 = sD[m * N + q];  // d/dxi0 acts on the first index
      const double d1 = sD[n * N + q];  // d/dxi1 acts on the second index
      j00 = fma(d0, sA[0][q * N + n], j00);
      j10 = fma(d0, sA[1][q * N + n], j10);
      j01 = fma(d1, sA[0][m * N + q], j01);
      j11 = fma(d1, sA[1][m * N + q], j11);
    }
    if (axis_mn) j01 = j10 = 0.0;
    if (axis_nm) j00 = j11 = 0.0;
    const double det = __dsub_rn(__dmul_rn(j00, j11), __dmul_rn(j01, j10));
    if (!(det > 0.0)) atomicExch(bad_flag, 1);
    const double rdet = __drcp_rn(det);
    r.j00 = j00;
    r.j01 = j01;
    r.j10 = j10;
    r.j11 = j11;
    r.det = det;
    r.i00 = __dmul_rn(j11, rdet);
    r.i01 = __dmul_rn(-j01, rdet);
    r.i10 = __dmul_rn(-j10, rdet);
    r.i11 = __dmul_rn(j00, rdet);
    r.jw = __dmul_rn(__dmul_rn(det, sw[m]), sw[n]);
  }
  return r;
}

template <int N>
__global__ void __launch_bounds__(((N * N + 31) / 32) * 32)
    geom_kernel(int64_t n_elem, const double *__restrict__ nodes_x,
                const double *__restrict__ nodes_y, const uint32_t *__restrict__ l2g,
                const double *__restrict__ Einv, const double *__restrict__ D,
                const double *__restrict__ w, const int64_t *__restrict__ elem_of_slot,
                double *__restrict__ G, int64_t g_patch_stride, int pe,
                double *__restrict__ JxW,
                double *__restrict__ x_phys, double *__restrict__ Jout,
                double *__restrict__ invJout, double *__restrict__ detJout,
                int32_t *__restrict__ bad_flag) {
  constexpr int NN = N * N;
  __shared__ double sE[NN], sD[NN], sw[N];
  __shared__ double sA[2][NN], sB[2][NN];
  const int k = threadIdx.x;
  const bool on = k < NN;
  const int m = on ? k / N : 0, n = on ? k % N : 0;
  if (on) {
    sE[k] = Einv[k];
    sD[k] = D[k];
  }
  if (k < N) sw[k] = w[k];

  for (int64_t slot = blockIdx.x; slot < n_elem; slot += gridDim.x) {
    const int64_t e = elem_of_slot ? elem_of_slot[slot] : slot;
    if (e < 0) continue;  // empty slot of the engine order (uniform over the CTA): G stays 0
    const NodeGeom q =
        node_geometry<N>(l2g + e * NN, nodes_x, nodes_y, sE, sD, sw, sA, sB, k, on, m, n, bad_flag);
    if (on) {
      const double i00 = q.i00, i01 = q.i01, i10 = q.i10, i11 = q.i11, jw = q.jw;
      if (G) {
        // patch-interleaved layout: ((c*N + m)*PE + le)*N + n inside the patch block
        const int64_t patch = slot / pe;
        const int lp = (int)(slot - patch * pe);
        const int64_t grow = (int64_t)N * pe;
        double *gs = G + patch * g_patch_stride + (int64_t)m * grow + lp * N + n;
        gs[0] = jw * (i00 * i00 + i01 * i01);
        gs[N * grow] = jw * (i00 * i10 + i01 * i11);
        gs[2 * N * grow] = jw * (i10 * i10 + i11 * i11);
      }
      if (JxW) JxW[e * NN + k] = jw;
      if (detJout) detJout[e * NN + k] = q.det;
      if (x_phys) {
        x_phys[(e * 2 + 0) * NN + k] = q.xg + q.ox;
        x_phys[(e * 2 + 1) * NN + k] = q.yg + q.oy;
      }
      if (Jout) {
        double *jp = Jout + e * 4 * NN;
        jp[k] = q.j00;
        jp[NN + k] = q.j01;
        jp[2 * NN + k] = q.j10;
        jp[3 * NN + k] = q.j11;
      }
      if (invJout) {
        double *ip = invJout + e * 4 * NN;
        ip[k] = i00;
        ip[NN + k] = i01;
        ip[2 * NN + k] = i10;
        ip[3 * NN + k] = i11;
      }
    }
  }
}

// Nodal fields after a solve (one CTA per element, one thread per node, like K1): the
// geometry again by node_geometry (nothing per element is stored between calls), then
// ur = D u, us = u D^T through shared memory and grad u = invJ^T (ur, us)
// (FiniteElement.gradient).  Outputs, each optional:
//   xy       [2][n_nodes]: x_phys at the entries whose winner byte is set;
//   grad_loc [2][n_elem][NN] (list order): grad u, times JxW when `weighted`;
//   jxw_loc  [n_elem][NN] (list order): JxW;
//   sums     [5]: JxW-sums of (u - u_ref)^2, |grad u - g_ref|^2, max |u - u_ref|,
//            JxW-sums of u_ref^2, |g_ref|^2 (u_ref / g_ref NULL = 0), reduced in a fixed
//            order over the CTAs (semk_finish_reduction); the max goes through the spare
//            slot after the arrival counter of `partials` and is exact in any order.
template <int N>
__global__ void __launch_bounds__(((N * N + 31) / 32) * 32)
    field_grad_kernel(int64_t n_elem, const double *__restrict__ nodes_x,
                      const double *__restrict__ nodes_y, const uint32_t *__restrict__ l2g,
                      const double *__restrict__ Einv, const double *__restrict__ D,
                      const double *__restrict__ w, const int64_t *__restrict__ elems,
                      const double *__restrict__ u, int64_t n_nodes,
                      const uint8_t *__restrict__ winner, double *__restrict__ xy,
                      double *__restrict__ grad_loc, int weighted, double *__restrict__ jxw_loc,
                      const double *__restrict__ u_ref, const double *__restrict__ g_ref,
                      double *__restrict__ sums, double *__restrict__ partials,
                      int32_t *__restrict__ bad_flag) {
  constexpr int NN = N * N;
  __shared__ double sE[NN], sD[NN], sw[N];
  __shared__ double sA[2][NN], sB[2][NN], sU[NN];
  const int k = threadIdx.x;
  const bool on = k < NN;
  const int m = on ? k / N : 0, n = on ? k % N : 0;
  if (on) {
    sE[k] = Einv[k];
    sD[k] = D[k];
  }
  if (k < N) sw[k] = w[k];
  double acc[4] = {0.0, 0.0, 0.0, 0.0};  // (u-u_ref)^2, |grad-g_ref|^2, u_ref^2, |g_ref|^2
  double umax = 0.0;

  for (int64_t slot = blockIdx.x; slot < n_elem; slot += gridDim.x) {
    const int64_t e = elems ? elems[slot] : slot;
    const uint32_t *row = l2g + e * NN;
    const uint32_t g = on ? row[k] : 0u;
    const double uk = (u && on) ? u[g] : 0.0;
    const NodeGeom q =
        node_geometry<N>(row, nodes_x, nodes_y, sE, sD, sw, sA, sB, k, on, m, n, bad_flag);
    if (on && xy && winner[e * NN + k]) {
      xy[g] = q.xg + q.ox;
      xy[n_nodes + g] = q.yg + q.oy;
    }
    if (!u) continue;  // coordinates only (uniform over the grid)
    if (on) sU[k] = uk;  // the previous element's reads of sU precede node_geometry's barriers
    __syncthreads();
    if (on) {
      double ur = 0.0, us = 0.0;
#pragma unroll
      for (int r = 0; r < N; ++r) {
        ur = fma(sD[m * N + r], sU[r * N + n], ur);
        us = fma(sD[n * N + r], sU[m * N + r], us);
      }
      const double gx = q.i00 * ur + q.i10 * us;
      const double gy = q.i01 * ur + q.i11 * us;
      if (grad_loc) {
        const double s = weighted ? q.jw : 1.0;
        grad_loc[slot * NN + k] = s * gx;
        grad_loc[(n_elem + slot) * NN + k] = s * gy;
      }
      if (jxw_loc) jxw_loc[slot * NN + k] = q.jw;
      if (sums) {
        const double ue = u_ref ? u_ref[g] : 0.0;
        const double gex = g_ref ? g_ref[g] : 0.0, gey = g_ref ? g_ref[n_nodes + g] : 0.0;
        const double du = uk - ue, dgx = gx - gex, dgy = gy - gey;
        acc[0] = fma(q.jw, du * du, acc[0]);
        acc[1] = fma(q.jw, dgx * dgx + dgy * dgy, acc[1]);
        acc[2] = fma(q.jw, ue * ue, acc[2]);
        acc[3] = fma(q.jw, gex * gex + gey * gey, acc[3]);
        umax = fmax(umax, fabs(du));
      }
    }
  }
  if (!sums) return;
  // block max, then one atomicMax on the bit pattern (order-preserving for doubles >= 0)
  __shared__ double smax[32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) umax = fmax(umax, __shfl_down_sync(0xffffffffu, umax, o));
  if ((threadIdx.x & 31u) == 0) smax[threadIdx.x >> 5] = umax;
  __syncthreads();
  unsigned long long *max_slot =
      reinterpret_cast<unsigned long long *>(semk_red_counter(partials) + 1);
  if (threadIdx.x == 0) {
    double bm = 0.0;
    for (unsigned i = 0; i < (blockDim.x + 31u) >> 5; ++i) bm = fmax(bm, smax[i]);
    atomicMax(max_slot, (unsigned long long)__double_as_longlong(bm));
  }
  double tot[4];
  if (semk_finish_reduction<4>(acc, partials, tot) && threadIdx.x == 0) {
    sums[0] = tot[0];
    sums[1] = tot[1];
    sums[2] = __longlong_as_double((long long)__ldcg(max_slot));
    sums[3] = tot[2];
    sums[4] = tot[3];
    *max_slot = 0ull;
  }
}

// G from the reference's own invJ / detJxW arrays (parity tier T1).
__global__ void gfactors_from_invj_kernel(int n1, int64_t n_elem,
                                          const double *__restrict__ invJ,
                                          const double *__restrict__ JxW,
                                          const int64_t *__restrict__ elem_of_slot,
                                          double *__restrict__ G, int64_t g_patch_stride,
                                          int pe) {
  const int NN = n1 * n1;
  const int64_t total = n_elem * NN;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t slot = i / NN;
    const int k = (int)(i - slot * NN);
    const int64_t e = elem_of_slot ? elem_of_slot[slot] : slot;
    if (e < 0) continue;
    const double *ip = invJ + e * 4 * NN;
    const double i00 = ip[k], i01 = ip[NN + k], i10 = ip[2 * NN + k], i11 = ip[3 * NN + k];
    const double jw = JxW[e * NN + k];
    const int m = k / n1, n = k - m * n1;
    const int64_t patch = slot / pe;
    const int lp = (int)(slot - patch * pe);
    const int64_t row = (int64_t)n1 * pe;
    double *gs = G + patch * g_patch_stride + (int64_t)m * row + lp * n1 + n;
    gs[0] = jw * (i00 * i00 + i01 * i01);
    gs[n1 * row] = jw * (i00 * i10 + i01 * i11);
    gs[2 * n1 * row] = jw * (i10 * i10 + i11 * i11);
  }
}

// G <- weight * G, node by node (weight in the reference's element-local layout).
__global__ void scale_gfactors_kernel(int n1, int64_t n_elem, const double *__restrict__ weight,
                                      const int64_t *__restrict__ elem_of_slot,
                                      double *__restrict__ G, int64_t g_patch_stride, int pe) {
  const int NN = n1 * n1;
  const int64_t total = n_elem * NN;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t slot = i / NN;
    const int k = (int)(i - slot * NN);
    const int64_t e = elem_of_slot ? elem_of_slot[slot] : slot;
    if (e < 0) continue;
    const double w = weight[e * NN + k];
    const int m = k / n1, n = k - m * n1;
    const int64_t patch = slot / pe;
    const int lp = (int)(slot - patch * pe);
    const int64_t row = (int64_t)n1 * pe;
    double *gs = G + patch * g_patch_stride + (int64_t)m * row + lp * n1 + n;
    gs[0] *= w;
    gs[n1 * row] *= w;
    gs[2 * n1 * row] *= w;
  }
}

}  // namespace

extern "C" int semk_geom_factors_f64(int n1, int64_t n_elem, const double *nodes_x,
                                     const double *nodes_y, const uint32_t *l2g,
                                     const double *Einv, const double *D, const double *w,
                                     const int64_t *elem_of_slot, double *G,
                                     int64_t g_patch_stride, int elems_per_patch, double *JxW,
                                     double *x_phys, double *J, double *invJ, double *detJ,
                                     int32_t *bad_flag, void *stream) {
  SEMK_REQUIRE(n_elem >= 0, "semk_geom_factors_f64: negative n_elem");
  SEMK_REQUIRE(nodes_x && nodes_y && l2g && Einv && D && w && bad_flag,
               "semk_geom_factors_f64: null input pointer");
  SEMK_REQUIRE(!G || (elems_per_patch >= 1 &&
                      g_patch_stride >= (int64_t)3 * n1 * n1 * elems_per_patch),
               "semk_geom_factors_f64: g_patch_stride too small");
  if (n_elem == 0) return SEMK_OK;
  const unsigned grid = (unsigned)(n_elem < (1 << 20) ? n_elem : (1 << 20));
#define SEMK_CALL(NV)                                                                      \
  geom_kernel<NV><<<grid, ((NV * NV + 31) / 32) * 32, 0, semk_stream(stream)>>>(           \
      n_elem, nodes_x, nodes_y, l2g, Einv, D, w, elem_of_slot, G, g_patch_stride,           \
      elems_per_patch > 0 ? elems_per_patch : 1, JxW, x_phys, J, invJ, detJ, bad_flag)
  SEMK_DISPATCH_N1(n1, SEMK_CALL)
#undef SEMK_CALL
  SEMK_LAUNCH_CHECK("geom_kernel");
  return SEMK_OK;
}

extern "C" int semk_gfactors_from_invj_f64(int n1, int64_t n_elem, const double *invJ,
                                           const double *JxW, const int64_t *elem_of_slot,
                                           double *G, int64_t g_patch_stride,
                                           int elems_per_patch, void *stream) {
  SEMK_REQUIRE(n1 >= 2 && n1 <= SEMK_MAX_N1, "semk_gfactors_from_invj_f64: bad n1");
  SEMK_REQUIRE(invJ && JxW && G, "semk_gfactors_from_invj_f64: null pointer");
  SEMK_REQUIRE(elems_per_patch >= 1 && g_patch_stride >= (int64_t)3 * n1 * n1 * elems_per_patch,
               "semk_gfactors_from_invj_f64: g_patch_stride too small");
  if (n_elem <= 0) return SEMK_OK;
  const int NN = n1 * n1;
  const int64_t total = n_elem * NN;
  const int block = 256;
  const int64_t want = (total + block - 1) / block;
  const unsigned grid = (unsigned)(want < 148 * 32 ? want : 148 * 32);
  gfactors_from_invj_kernel<<<grid, block, 0, semk_stream(stream)>>>(
      n1, n_elem, invJ, JxW, elem_of_slot, G, g_patch_stride, elems_per_patch);
  SEMK_LAUNCH_CHECK("gfactors_from_invj_kernel");
  return SEMK_OK;
}

extern "C" int semk_scale_gfactors_f64(int n1, int64_t n_elem, const double *weight,
                                       const int64_t *elem_of_slot, double *G,
                                       int64_t g_patch_stride, int elems_per_patch,
                                       void *stream) {
  SEMK_REQUIRE(n1 >= 2 && n1 <= SEMK_MAX_N1, "semk_scale_gfactors_f64: bad n1");
  SEMK_REQUIRE(weight && G, "semk_scale_gfactors_f64: null pointer");
  SEMK_REQUIRE(elems_per_patch >= 1 && g_patch_stride >= (int64_t)3 * n1 * n1 * elems_per_patch,
               "semk_scale_gfactors_f64: g_patch_stride too small");
  if (n_elem <= 0) return SEMK_OK;
  const int64_t total = n_elem * n1 * n1;
  const int block = 256;
  const int64_t want = (total + block - 1) / block;
  const unsigned grid = (unsigned)(want < 148 * 32 ? want : 148 * 32);
  scale_gfactors_kernel<<<grid, block, 0, semk_stream(stream)>>>(n1, n_elem, weight, elem_of_slot, G,
                                                                g_patch_stride, elems_per_patch);
  SEMK_LAUNCH_CHECK("scale_gfactors_kernel");
  return SEMK_OK;
}

extern "C" int semk_field_grad_f64(int n1, int64_t n_elem, const double *nodes_x,
                                   const double *nodes_y, const uint32_t *l2g, const double *Einv,
                                   const double *D, const double *w, const int64_t *elems,
                                   int64_t n_nodes, const double *u, const uint8_t *winner,
                                   double *xy, double *grad_loc, int weighted, double *jxw_loc,
                                   const double *u_ref, const double *g_ref, double *sums,
                                   double *partials, int32_t *bad_flag, void *stream) {
  SEMK_REQUIRE(n_elem >= 0 && n_nodes > 0, "semk_field_grad_f64: bad sizes");
  SEMK_REQUIRE(nodes_x && nodes_y && l2g && Einv && D && w && bad_flag,
               "semk_field_grad_f64: null input pointer");
  SEMK_REQUIRE(!xy || winner, "semk_field_grad_f64: xy needs winner");
  SEMK_REQUIRE(u || !(grad_loc || jxw_loc || sums), "semk_field_grad_f64: outputs need u");
  SEMK_REQUIRE(!sums || partials, "semk_field_grad_f64: sums need partials");
  SEMK_REQUIRE(!xy || (xy != u && xy != u_ref && xy != g_ref),
               "semk_field_grad_f64: xy aliases an input");
  if (n_elem == 0) return SEMK_OK;
  // the fixed-order reduction bounds the grid (kSemkRedMaxBlocks CTAs of partials)
  const int64_t cap = sums ? kSemkRedMaxBlocks : (1 << 20);
  const unsigned grid = (unsigned)(n_elem < cap ? n_elem : cap);
#define SEMK_CALL(NV)                                                                      \
  field_grad_kernel<NV><<<grid, ((NV * NV + 31) / 32) * 32, 0, semk_stream(stream)>>>(     \
      n_elem, nodes_x, nodes_y, l2g, Einv, D, w, elems, u, n_nodes, winner, xy, grad_loc,   \
      weighted, jxw_loc, u_ref, g_ref, sums, partials, bad_flag)
  SEMK_DISPATCH_N1(n1, SEMK_CALL)
#undef SEMK_CALL
  SEMK_LAUNCH_CHECK("field_grad_kernel");
  return SEMK_OK;
}
