// semk_vec.cu -- K4: fused vector kernels of Jacobi-PCG and the native driver.
//
// The reference solves the assembled (Schur-complement) system with SuperLU
// (`sparse.linalg.spsolve`, sem/discrete.py:511) plus per-element interior
// back-substitution (:513-524).  The engine replaces the solve on this path
// by a device-resident Jacobi-preconditioned CG on
//     Ahat = M A M + (I - M),   M = diag(free-DOF mask)
// (the Dirichlet elimination of sem/discrete.py:505-510 written as an SPD
// operator on the full vector).  All scalars stay on the device:
//     sc[0]=rz  sc[1]=pAp  sc[2]=rz_new  sc[3]=rr  sc[4]=bb
//     sc[5]=iterations done  sc[6]=converged flag  sc[7]=breakdown flag
// Kernels are HBM-bound streams; each vector is touched once per kernel and
// the dot products are fused into the pass that produces their operands.
// Reductions are deterministic: per-CTA partials + the last CTA to finish
// sums them in a fixed order (no floating-point atomics).
#include "semk_common.cuh"

namespace {

constexpr int kVecThreads = 256;
constexpr int kVecMaxBlocks = kSemkRedMaxBlocks;

inline int vec_blocks(int64_t n) {
  const int64_t want = (n + kVecThreads * 4 - 1) / (kVecThreads * 4);
  return (int)(want < 1 ? 1 : (want < kVecMaxBlocks ? want : kVecMaxBlocks));
}

// partials layout and the last-arrival reduction: semk_common.cuh
__device__ __forceinline__ unsigned long long *counter_of(double *partials) {
  return semk_red_counter(partials);
}
template <int NV>
__device__ __forceinline__ bool finish_reduction(double (&v)[NV], double *partials,
                                                 double (&tot)[NV]) {
  return semk_finish_reduction<NV>(v, partials, tot);
}

__global__ void __launch_bounds__(kVecThreads)
    pcg_init_kernel(int64_t n, int64_t n_dot, const double *__restrict__ b,
                    const double *__restrict__ Ax, const double *__restrict__ dinv,
                    const uint8_t *__restrict__ dirichlet, double *__restrict__ r,
                    double *__restrict__ p, double *__restrict__ sc,
                    double *__restrict__ partials) {
  double acc[3] = {0.0, 0.0, 0.0};
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const bool fixed = dirichlet && dirichlet[i];
    const double bi = fixed ? 0.0 : b[i];
    const double ri = fixed ? 0.0 : bi - Ax[i];
    const double zi = dinv[i] * ri;
    r[i] = ri;
    p[i] = zi;
    if (i < n_dot) {
      acc[0] = fma(ri, zi, acc[0]);
      acc[1] = fma(ri, ri, acc[1]);
      acc[2] = fma(bi, bi, acc[2]);
    }
  }
  double tot[3];
  if (finish_reduction<3>(acc, partials, tot) && threadIdx.x == 0) {
    sc[0] = tot[0];
    sc[1] = 0.0;
    sc[2] = tot[0];
    sc[3] = tot[1];
    sc[4] = tot[2];
    sc[5] = 0.0;
    sc[6] = 0.0;
    sc[7] = 0.0;
  }
}

// VEC: all vector pointers are 16-byte aligned -> 128-bit loads/stores, two pairs
// per thread and iteration in flight (these kernels are pure HBM streams).
// XP ("x rides with p"): the native driver defers x += alpha p from the first kernel to
// the second one, which reads p anyway -- one vector pass less per iteration (6 + 4
// instead of 7 + 4).  The two public entry points keep x in the first kernel.
template <bool VEC, bool XP>
__global__ void __launch_bounds__(kVecThreads)
    pcg_update_xr_kernel(int64_t n, int64_t n_dot, const double *__restrict__ p,
                         const double *__restrict__ Ap, const double *__restrict__ dinv,
                         double *__restrict__ x, double *__restrict__ r, double *__restrict__ sc,
                         double *__restrict__ partials, double tol2) {
  const volatile double *vsc = sc;
  if (vsc[6] != 0.0 || vsc[7] != 0.0) return;  // converged / broken down: freeze
  const double rz = vsc[0], pAp = vsc[1];
  const bool ok = (pAp > 0.0) && (rz == rz);
  const double alpha = ok ? rz / pAp : 0.0;
  double acc[2] = {0.0, 0.0};
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  auto one = [&](int64_t i) {
    if (!XP) x[i] = fma(alpha, p[i], x[i]);
    const double ri = fma(-alpha, Ap[i], r[i]);
    r[i] = ri;
    if (i < n_dot) {
      acc[0] = fma(ri * dinv[i], ri, acc[0]);
      acc[1] = fma(ri, ri, acc[1]);
    }
  };
  if (VEC) {
    const int64_t npair = n >> 1;
    const double2 *p2 = reinterpret_cast<const double2 *>(p);
    const double2 *Ap2 = reinterpret_cast<const double2 *>(Ap);
    const double2 *d2 = reinterpret_cast<const double2 *>(dinv);
    double2 *x2 = reinterpret_cast<double2 *>(x);
    double2 *r2 = reinterpret_cast<double2 *>(r);
    const double2 zero2 = make_double2(0.0, 0.0);
    for (int64_t j0 = tid; j0 < npair; j0 += 2 * nthreads) {
      const int64_t jj[2] = {j0, j0 + nthreads};
      const bool on[2] = {true, jj[1] < npair};
      double2 pv[2], av[2], xv[2], rv[2], dv[2];
#pragma unroll
      for (int q = 0; q < 2; ++q) {  // all loads of both pairs first
        av[q] = on[q] ? Ap2[jj[q]] : zero2;
        rv[q] = on[q] ? r2[jj[q]] : zero2;
        dv[q] = on[q] ? d2[jj[q]] : zero2;
        if (!XP) {
          pv[q] = on[q] ? p2[jj[q]] : zero2;
          xv[q] = on[q] ? x2[jj[q]] : zero2;
        }
      }
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        if (!on[q]) continue;
        double2 ro;
        ro.x = fma(-alpha, av[q].x, rv[q].x);
        ro.y = fma(-alpha, av[q].y, rv[q].y);
        r2[jj[q]] = ro;
        if (!XP) {
          double2 xo;
          xo.x = fma(alpha, pv[q].x, xv[q].x);
          xo.y = fma(alpha, pv[q].y, xv[q].y);
          x2[jj[q]] = xo;
        }
        if (2 * jj[q] < n_dot) {
          acc[0] = fma(ro.x * dv[q].x, ro.x, acc[0]);
          acc[1] = fma(ro.x, ro.x, acc[1]);
        }
        if (2 * jj[q] + 1 < n_dot) {
          acc[0] = fma(ro.y * dv[q].y, ro.y, acc[0]);
          acc[1] = fma(ro.y, ro.y, acc[1]);
        }
      }
    }
    if ((n & 1) && tid == 0) one(n - 1);
  } else {
    for (int64_t i = tid; i < n; i += nthreads) one(i);
  }
  double tot[2];
  if (finish_reduction<2>(acc, partials, tot) && threadIdx.x == 0) {
    sc[2] = tot[0];
    sc[3] = tot[1];
    sc[5] += 1.0;
    if (!ok) sc[7] = 1.0;
    if (tot[1] <= tol2 * sc[4]) sc[6] = 1.0;
  }
}

// p = z + beta p (z = dinv r).  XP: also x += alpha p_old; on the iteration that
// converged (sc[6] == 1, set by the first kernel) only that last x update is done and
// the state moves on to 2 = frozen.
template <bool VEC, bool XP>
__global__ void __launch_bounds__(kVecThreads)
    pcg_update_p_kernel(int64_t n, const double *__restrict__ r, const double *__restrict__ dinv,
                        double *__restrict__ p, double *__restrict__ x, double *__restrict__ sc,
                        double *__restrict__ partials) {
  const volatile double *vsc = sc;
  const double conv = vsc[6];
  if (vsc[7] != 0.0 || conv == 2.0 || (!XP && conv != 0.0)) return;
  const double rz_new = vsc[2], rz = vsc[0], pAp = vsc[1];
  const double beta = (rz != 0.0) ? rz_new / rz : 0.0;
  const double alpha = XP ? rz / pAp : 0.0;  // the first kernel vetted pAp > 0
  const bool move_p = conv == 0.0;
  __shared__ bool is_last;
  __syncthreads();  // every thread of this CTA has read the scalars
  if (threadIdx.x == 0) {
    // every CTA has read the scalars before it arrives; the last arrival rotates them
    __threadfence();
    const unsigned long long t = atomicAdd(counter_of(partials), 1ull);
    is_last = (t == (unsigned long long)gridDim.x - 1ull);
  }
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  auto one = [&](int64_t i) {
    const double pi = p[i];
    if (XP) x[i] = fma(alpha, pi, x[i]);
    if (move_p) p[i] = fma(beta, pi, dinv[i] * r[i]);
  };
  if (VEC) {
    const int64_t npair = n >> 1;
    const double2 *r2 = reinterpret_cast<const double2 *>(r);
    const double2 *d2 = reinterpret_cast<const double2 *>(dinv);
    double2 *p2 = reinterpret_cast<double2 *>(p);
    double2 *x2 = reinterpret_cast<double2 *>(x);
    const double2 zero2 = make_double2(0.0, 0.0);
    for (int64_t j0 = tid; j0 < npair; j0 += 2 * nthreads) {
      const int64_t jj[2] = {j0, j0 + nthreads};
      const bool on[2] = {true, jj[1] < npair};
      double2 rv[2], dv[2], pv[2], xv[2];
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        pv[q] = on[q] ? p2[jj[q]] : zero2;
        rv[q] = (on[q] && move_p) ? r2[jj[q]] : zero2;
        dv[q] = (on[q] && move_p) ? d2[jj[q]] : zero2;
        if (XP) xv[q] = on[q] ? x2[jj[q]] : zero2;
      }
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        if (!on[q]) continue;
        if (XP) {
          double2 xo;
          xo.x = fma(alpha, pv[q].x, xv[q].x);
          xo.y = fma(alpha, pv[q].y, xv[q].y);
          x2[jj[q]] = xo;
        }
        if (move_p) {
          double2 o;
          o.x = fma(beta, pv[q].x, dv[q].x * rv[q].x);
          o.y = fma(beta, pv[q].y, dv[q].y * rv[q].y);
          p2[jj[q]] = o;
        }
      }
    }
    if ((n & 1) && tid == 0) one(n - 1);
  } else {
    for (int64_t i = tid; i < n; i += nthreads) one(i);
  }
  __syncthreads();
  if (is_last && threadIdx.x == 0) {
    if (move_p)
      sc[0] = rz_new;
    else
      sc[6] = 2.0;  // the converged iterate is complete: frozen from now on
    *counter_of(partials) = 0ull;
  }
}

__global__ void __launch_bounds__(kVecThreads)
    dot_kernel(int64_t n, const double *__restrict__ a, const double *__restrict__ b,
               double *__restrict__ out, double *__restrict__ partials) {
  double acc[1] = {0.0};
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    acc[0] = fma(a[i], b[i], acc[0]);
  double tot[1];
  if (finish_reduction<1>(acc, partials, tot) && threadIdx.x == 0) out[0] = tot[0];
}

}  // namespace

extern "C" int64_t semk_vec_partials_len(int64_t n) {
  (void)n;
  return 4 * kVecMaxBlocks + 2;
}

extern "C" int semk_pcg_init_f64(int64_t n, int64_t n_dot, const double *b, const double *Ax,
                                 const double *dinv, const uint8_t *dirichlet, double *r,
                                 double *p, double *sc, double *partials, void *stream) {
  SEMK_REQUIRE(n > 0 && n_dot >= 0 && n_dot <= n, "semk_pcg_init_f64: bad sizes");
  SEMK_REQUIRE(b && Ax && dinv && r && p && sc && partials, "semk_pcg_init_f64: null pointer");
  pcg_init_kernel<<<vec_blocks(n), kVecThreads, 0, semk_stream(stream)>>>(
      n, n_dot, b, Ax, dinv, dirichlet, r, p, sc, partials);
  SEMK_LAUNCH_CHECK("pcg_init_kernel");
  return SEMK_OK;
}

static inline bool aligned16(const void *a, const void *b, const void *c, const void *d,
                             const void *e) {
  return ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) |
           reinterpret_cast<uintptr_t>(c) | reinterpret_cast<uintptr_t>(d) |
           reinterpret_cast<uintptr_t>(e)) &
          15u) == 0;
}

static int update_xr(int64_t n, int64_t n_dot, const double *p, const double *Ap,
                     const double *dinv, double *x, double *r, double *sc, double *partials,
                     double tol2, bool x_rides_with_p, cudaStream_t st) {
  const bool vec = aligned16(p, Ap, dinv, x, r);
  const dim3 g(vec_blocks(n)), b(kVecThreads);
#define SEMK_GO(V, X) \
  pcg_update_xr_kernel<V, X><<<g, b, 0, st>>>(n, n_dot, p, Ap, dinv, x, r, sc, partials, tol2)
  if (vec && x_rides_with_p) SEMK_GO(true, true);
  else if (vec) SEMK_GO(true, false);
  else if (x_rides_with_p) SEMK_GO(false, true);
  else SEMK_GO(false, false);
#undef SEMK_GO
  SEMK_LAUNCH_CHECK("pcg_update_xr_kernel");
  return SEMK_OK;
}

static int update_p(int64_t n, const double *r, const double *dinv, double *p, double *x,
                    double *sc, double *partials, cudaStream_t st) {
  const bool vec = aligned16(r, dinv, p, x ? x : p, p);
  const dim3 g(vec_blocks(n)), b(kVecThreads);
#define SEMK_GO(V, X) pcg_update_p_kernel<V, X><<<g, b, 0, st>>>(n, r, dinv, p, x, sc, partials)
  if (vec && x) SEMK_GO(true, true);
  else if (vec) SEMK_GO(true, false);
  else if (x) SEMK_GO(false, true);
  else SEMK_GO(false, false);
#undef SEMK_GO
  SEMK_LAUNCH_CHECK("pcg_update_p_kernel");
  return SEMK_OK;
}

extern "C" int semk_pcg_update_xr_f64(int64_t n, int64_t n_dot, const double *p, const double *Ap,
                                      const double *dinv, double *x, double *r, double *sc,
                                      double *partials, void *stream) {
  SEMK_REQUIRE(n > 0 && n_dot >= 0 && n_dot <= n, "semk_pcg_update_xr_f64: bad sizes");
  SEMK_REQUIRE(p && Ap && dinv && r && sc && partials, "semk_pcg_update_xr_f64: null pointer");
  // tol2 < 0: the device-side convergence freeze is disabled (caller decides).
  // x == NULL: the caller updates x together with p (semk_pcg_update_px_f64).
  return update_xr(n, n_dot, p, Ap, dinv, x ? x : r, r, sc, partials, -1.0, x == nullptr,
                   semk_stream(stream));
}

extern "C" int semk_pcg_update_p_f64(int64_t n, const double *r, const double *dinv, double *p,
                                      double *sc, double *partials, void *stream) {
  SEMK_REQUIRE(n > 0, "semk_pcg_update_p_f64: bad size");
  SEMK_REQUIRE(r && dinv && p && sc && partials, "semk_pcg_update_p_f64: null pointer");
  return update_p(n, r, dinv, p, nullptr, sc, partials, semk_stream(stream));
}

extern "C" int semk_pcg_update_px_f64(int64_t n, const double *r, const double *dinv, double *p,
                                      double *x, double *sc, double *partials, void *stream) {
  SEMK_REQUIRE(n > 0, "semk_pcg_update_px_f64: bad size");
  SEMK_REQUIRE(r && dinv && p && x && sc && partials, "semk_pcg_update_px_f64: null pointer");
  return update_p(n, r, dinv, p, x, sc, partials, semk_stream(stream));
}

extern "C" int semk_dot_f64(int64_t n, const double *a, const double *b, double *out,
                            double *partials, void *stream) {
  SEMK_REQUIRE(n > 0 && a && b && out && partials, "semk_dot_f64: bad argument");
  dot_kernel<<<vec_blocks(n), kVecThreads, 0, semk_stream(stream)>>>(n, a, b, out, partials);
  SEMK_LAUNCH_CHECK("dot_kernel");
  return SEMK_OK;
}

// The native PCG loop, generic over the operator: `apply(in, out, dot)` queues
// out = Ahat in on `st` and, when dot != nullptr, leaves in.out in *dot (device).
template <class ApplyFn>
static int pcg_solve_impl(ApplyFn apply, int64_t n, const uint8_t *dirichlet, const double *b,
                          double *x, const double *dinv, double *work, double *sc,
                          double *vec_partials, double rtol, int maxiter, int check_every,
                          semk_pcg_info *info, cudaStream_t st) {
  const int64_t n_pad = (n + 31) & ~(int64_t)31;  // keeps the sub-vectors 16-byte aligned
  double *r = work, *p = work + n_pad, *Ap = work + 2 * n_pad;
  const double tol2 = rtol * rtol;
  // pinned landing zone for the 64-byte scalar block: one per host thread (a solve blocks
  // its thread while it polls, so solves on different threads / streams never share it)
  thread_local double *h_sc = nullptr;
  if (!h_sc) SEMK_CUDA_CHECK(cudaMallocHost(&h_sc, 8 * sizeof(double)));

  int rc = apply(x, Ap, nullptr);
  if (rc != SEMK_OK) return rc;
  rc = semk_pcg_init_f64(n, n, b, Ap, dinv, dirichlet, r, p, sc, vec_partials, st);
  if (rc != SEMK_OK) return rc;

  auto poll = [&]() -> int {
    SEMK_CUDA_CHECK(cudaMemcpyAsync(h_sc, sc, 8 * sizeof(double), cudaMemcpyDeviceToHost, st));
    SEMK_CUDA_CHECK(cudaStreamSynchronize(st));
    return SEMK_OK;
  };
  rc = poll();
  if (rc != SEMK_OK) return rc;
  info->bnorm = sqrt(h_sc[4]);
  info->iterations = 0;
  info->status = 0;
  if (h_sc[4] == 0.0 || h_sc[3] <= tol2 * h_sc[4]) {
    info->rel_residual = h_sc[4] > 0.0 ? sqrt(h_sc[3] / h_sc[4]) : 0.0;
    return SEMK_OK;
  }

  auto one_iteration = [&]() -> int {
    int e = apply(p, Ap, sc + 1);
    if (e != SEMK_OK) return e;
    // x += alpha p rides with the p update (one vector pass less per iteration)
    e = update_xr(n, n, p, Ap, dinv, x, r, sc, vec_partials, tol2, true, st);
    if (e != SEMK_OK) return e;
    return update_p(n, r, dinv, p, x, sc, vec_partials, st);
  };

  // Capture `check_every` iterations once and replay: removes per-launch host
  // cost from the loop.  Falls back to eager launches if capture is refused.
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  bool use_graph = false;
  if (check_every > 1 && st != nullptr) {
    if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
      int e = SEMK_OK;
      for (int k = 0; k < check_every && e == SEMK_OK; ++k) e = one_iteration();
      cudaError_t ce = cudaStreamEndCapture(st, &graph);
      if (e == SEMK_OK && ce == cudaSuccess && graph &&
          cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess)
        use_graph = true;
      else
        (void)cudaGetLastError();
    } else {
      (void)cudaGetLastError();
    }
  }

  int status = 1;  // maxiter unless proven otherwise
  int launched = 0;
  rc = SEMK_OK;
  while (launched < maxiter) {
    // the graph holds exactly check_every iterations: a shorter tail is launched eagerly so
    // that maxiter is never exceeded
    if (use_graph && maxiter - launched >= check_every) {
      if (cudaGraphLaunch(exec, st) != cudaSuccess) {
        semk_set_error("PCG driver: cudaGraphLaunch failed");
        rc = SEMK_ERR_CUDA;
        break;
      }
      launched += check_every;
    } else {
      for (int k = 0; k < check_every && launched < maxiter && rc == SEMK_OK; ++k, ++launched)
        rc = one_iteration();
      if (rc != SEMK_OK) break;
    }
    rc = poll();
    if (rc != SEMK_OK) break;
    if (h_sc[7] != 0.0) {
      status = SEMK_ERR_BREAKDOWN;
      break;
    }
    if (h_sc[6] != 0.0) {
      status = 0;
      break;
    }
  }
  if (exec) cudaGraphExecDestroy(exec);
  if (graph) cudaGraphDestroy(graph);
  if (rc != SEMK_OK) return rc;
  info->iterations = (int32_t)h_sc[5];
  info->status = status;
  info->rel_residual = sqrt(h_sc[3] / h_sc[4]);
  if (status == SEMK_ERR_BREAKDOWN) {
    semk_set_error("PCG driver: breakdown (p.Ap <= 0 or non-finite)");
    return SEMK_ERR_BREAKDOWN;
  }
  return SEMK_OK;
}

extern "C" int semk_pcg_solve_f64(const semk_op *op, const double *b, double *x,
                                  const double *dinv, double *work, double *sc,
                                  double *vec_partials, double rtol, int maxiter, int check_every,
                                  semk_pcg_info *info, void *stream) {
  SEMK_REQUIRE(op && b && x && dinv && work && sc && vec_partials && info,
               "semk_pcg_solve_f64: null pointer");
  SEMK_REQUIRE(maxiter >= 0 && check_every >= 1 && rtol >= 0.0, "semk_pcg_solve_f64: bad control");
  cudaStream_t st = semk_stream(stream);
  const int flags = SEMK_MASK_IN | SEMK_MASK_OUT | SEMK_DIRICHLET_IDENTITY;
  auto apply = [&](const double *in, double *out, double *dot) -> int {
    return semk_poisson_apply_f64(op, in, out, flags, dot, st);
  };
  return pcg_solve_impl(apply, op->n_nodes, op->dirichlet, b, x, dinv, work, sc, vec_partials,
                        rtol, maxiter, check_every, info, st);
}

// The same loop with the Robin boundary diagonal in every apply (and in pAp).
extern "C" int semk_pcg_solve_bdiag_f64(const semk_op *op, const semk_bdiag *bdiag,
                                        const double *b, double *x, const double *dinv,
                                        double *work, double *sc, double *vec_partials,
                                        double rtol, int maxiter, int check_every,
                                        semk_pcg_info *info, void *stream) {
  SEMK_REQUIRE(op && b && x && dinv && work && sc && vec_partials && info,
               "semk_pcg_solve_bdiag_f64: null pointer");
  SEMK_REQUIRE(maxiter >= 0 && check_every >= 1 && rtol >= 0.0,
               "semk_pcg_solve_bdiag_f64: bad control");
  cudaStream_t st = semk_stream(stream);
  const int flags = SEMK_MASK_IN | SEMK_MASK_OUT | SEMK_DIRICHLET_IDENTITY;
  auto apply = [&](const double *in, double *out, double *dot) -> int {
    return semk_poisson_apply_bdiag_f64(op, bdiag, in, out, flags, dot, st);
  };
  return pcg_solve_impl(apply, op->n_nodes, op->dirichlet, b, x, dinv, work, sc, vec_partials,
                        rtol, maxiter, check_every, info, st);
}

// The same loop on the statically condensed operator Shat = M S M + (I - M) over the
// element-exterior DOFs (sem/discrete.py:502-511 solves that system with SuperLU).
extern "C" int semk_sc_pcg_solve_f64(const semk_sc_op *op, const double *b, double *x,
                                     const double *dinv, double *work, double *sc,
                                     double *vec_partials, double rtol, int maxiter,
                                     int check_every, semk_pcg_info *info, void *stream) {
  SEMK_REQUIRE(op && b && x && dinv && work && sc && vec_partials && info,
               "semk_sc_pcg_solve_f64: null pointer");
  SEMK_REQUIRE(maxiter >= 0 && check_every >= 1 && rtol >= 0.0,
               "semk_sc_pcg_solve_f64: bad control");
  cudaStream_t st = semk_stream(stream);
  const int flags = SEMK_MASK_IN | SEMK_MASK_OUT | SEMK_DIRICHLET_IDENTITY;
  auto apply = [&](const double *in, double *out, double *dot) -> int {
    return semk_sc_apply_f64(op, in, out, flags, dot, st);
  };
  return pcg_solve_impl(apply, op->n_ext, op->dirichlet, b, x, dinv, work, sc, vec_partials,
                        rtol, maxiter, check_every, info, st);
}

// ---------------------------------------------------------------------------------------
// Small vector kernels of the multilevel preconditioner as separate entry points (the
// native driver is semk_sc_mlpcg_solve_f64, csrc/semk_ml.cu; these serve tests and
// host-driven experiments).
// ---------------------------------------------------------------------------------------
namespace {

__global__ void __launch_bounds__(kVecThreads)
    resid_kernel(int64_t n, const double *__restrict__ b, const double *__restrict__ Ax,
                 const uint8_t *__restrict__ dirichlet, double *__restrict__ r,
                 double *__restrict__ bm) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const bool fixed = dirichlet && dirichlet[i];
    const double bi = fixed ? 0.0 : b[i];
    bm[i] = bi;
    r[i] = fixed ? 0.0 : bi - Ax[i];
  }
}

__global__ void __launch_bounds__(kVecThreads)
    scale_kernel(int64_t n, const double *__restrict__ d, const double *__restrict__ r,
                 double *__restrict__ z) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    z[i] = d[i] * r[i];
}

// rc = P^T r: one thread per coarse row, fixed summation order
__global__ void __launch_bounds__(kVecThreads)
    restrict_kernel(int64_t n_v, const uint32_t *__restrict__ rptr,
                    const uint32_t *__restrict__ ridx, const double *__restrict__ rw,
                    const double *__restrict__ r, int64_t n_owned, double *__restrict__ rc) {
  // n_owned: only fine nodes [0, n_owned) contribute (multi-GPU: every global node is
  // restricted by its owner; one GPU: n_owned = n)
  for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < n_v;
       v += (int64_t)gridDim.x * blockDim.x) {
    double s = 0.0;
    for (uint32_t q = rptr[v]; q < rptr[v + 1]; ++q) {
      const uint32_t g = ridx[q];
      if ((int64_t)g < n_owned) s = fma(rw[q], r[g], s);
    }
    rc[v] = s;
  }
}

// z += P xc
__global__ void __launch_bounds__(kVecThreads)
    prolong_add_kernel(int64_t n, const uint32_t *__restrict__ pv, const double *__restrict__ pw,
                       const double *__restrict__ xc, double *__restrict__ z) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const double wa = pw[2 * i], wb = pw[2 * i + 1];
    double acc = z[i];
    if (wa != 0.0) acc = fma(wa, xc[pv[2 * i]], acc);
    if (wb != 0.0) acc = fma(wb, xc[pv[2 * i + 1]], acc);
    z[i] = acc;
  }
}

__global__ void __launch_bounds__(kVecThreads)
    axpy2_kernel(int64_t n, double alpha, const double *__restrict__ p,
                 const double *__restrict__ Ap, double *__restrict__ x, double *__restrict__ r) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    x[i] = fma(alpha, p[i], x[i]);
    r[i] = fma(-alpha, Ap[i], r[i]);
  }
}

__global__ void __launch_bounds__(kVecThreads)
    xpay_kernel(int64_t n, double beta, const double *__restrict__ z, double *__restrict__ p) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    p[i] = fma(beta, p[i], z[i]);
}

}  // namespace

// ---- the pieces of the two-level preconditioner as separate entry points (the multi-GPU
// outer loop, distributed.distributed_two_level_pcg, is driven from Python so that the
// exchanges and all-reduces can sit between them) -------------------------------------------
extern "C" int semk_vec_resid_f64(int64_t n, const double *b, const double *Ax,
                                  const uint8_t *dirichlet, double *r, double *b_masked,
                                  void *stream) {
  SEMK_REQUIRE(n > 0 && b && Ax && r && b_masked, "semk_vec_resid_f64: bad argument");
  resid_kernel<<<vec_blocks(n), kVecThreads, 0, semk_stream(stream)>>>(n, b, Ax, dirichlet, r,
                                                                      b_masked);
  SEMK_LAUNCH_CHECK("resid_kernel");
  return SEMK_OK;
}

extern "C" int semk_vec_scale_f64(int64_t n, const double *d, const double *r, double *z,
                                  void *stream) {
  SEMK_REQUIRE(n > 0 && d && r && z, "semk_vec_scale_f64: bad argument");
  scale_kernel<<<vec_blocks(n), kVecThreads, 0, semk_stream(stream)>>>(n, d, r, z);
  SEMK_LAUNCH_CHECK("scale_kernel");
  return SEMK_OK;
}

extern "C" int semk_vec_axpy2_f64(int64_t n, double alpha, const double *p, const double *Ap,
                                  double *x, double *r, void *stream) {
  SEMK_REQUIRE(n > 0 && p && Ap && x && r, "semk_vec_axpy2_f64: bad argument");
  axpy2_kernel<<<vec_blocks(n), kVecThreads, 0, semk_stream(stream)>>>(n, alpha, p, Ap, x, r);
  SEMK_LAUNCH_CHECK("axpy2_kernel");
  return SEMK_OK;
}

extern "C" int semk_vec_xpay_f64(int64_t n, double beta, const double *z, double *p,
                                 void *stream) {
  SEMK_REQUIRE(n > 0 && z && p, "semk_vec_xpay_f64: bad argument");
  xpay_kernel<<<vec_blocks(n), kVecThreads, 0, semk_stream(stream)>>>(n, beta, z, p);
  SEMK_LAUNCH_CHECK("xpay_kernel");
  return SEMK_OK;
}

extern "C" int semk_sc_restrict_f64(const semk_sc_coarse *cs, const double *r, int64_t n_owned,
                                    double *rc, void *stream) {
  SEMK_REQUIRE(cs && cs->n_v > 0 && cs->rptr && cs->ridx && cs->rw && r && rc && n_owned >= 0,
               "semk_sc_restrict_f64: bad argument");
  restrict_kernel<<<vec_blocks(cs->n_v), kVecThreads, 0, semk_stream(stream)>>>(
      cs->n_v, cs->rptr, cs->ridx, cs->rw, r, n_owned, rc);
  SEMK_LAUNCH_CHECK("restrict_kernel");
  return SEMK_OK;
}

extern "C" int semk_sc_prolong_add_f64(int64_t n_ext, const semk_sc_coarse *cs, const double *xc,
                                       double *z, void *stream) {
  SEMK_REQUIRE(n_ext > 0 && cs && cs->pv && cs->pw && xc && z,
               "semk_sc_prolong_add_f64: bad argument");
  prolong_add_kernel<<<vec_blocks(n_ext), kVecThreads, 0, semk_stream(stream)>>>(
      n_ext, cs->pv, cs->pw, xc, z);
  SEMK_LAUNCH_CHECK("prolong_add_kernel");
  return SEMK_OK;
}

