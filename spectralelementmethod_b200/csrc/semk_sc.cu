// semk_sc.cu -- static condensation on the device (SURVEY.md 8(f) row 1).
//
// The reference's solver formulation (DOFManagerSC, sem/discrete.py:283-528):
// eliminate the (p-1)^2 interior DOFs of every element,
//     S_e = A_ee - A_ei A_ii^{-1} A_ie,   g_e = f_e - A_ei A_ii^{-1} f_i
// (compute_local_sc_system, :438-476), assemble and solve the condensed system
// over the element-exterior DOFs (:478-511) and recover the interiors element
// by element (:513-524).  Here:
//
//   sc_element_kernel<N>  one CTA per element.  Rebuilds the 4-index local
//       stiffness of examples/poisson.py:166-193 entry by entry from the
//       geometric factors (closed form below), Cholesky-factorises the interior
//       block in shared memory (A_ii = L L^T), Z = L^{-1} A_ie, and writes
//       S_e = A_ee - Z^T Z (packed lower triangle).  Set-up work.
//   sc_element_block_kernel<N>  the same factorisation for up to 32 loads
//       (f_i columns of Z): g_e = f_e - Z^T (L^{-1} f_i) or the back-substitution
//       u_i = L^{-T} (L^{-1} f_i - Z u_e); once-per-solve work, recomputed instead
//       of stored (19 KB per element at p = 8 against 4 KB for S_e).
//   sc_matvec_kernel<N>   the condensed apply, HBM-bound: persistent CTAs stream the
//       packed S_e blocks through a double-buffered TMA pipeline (evict-first),
//       gather the 4p exterior values through the L2G map one group ahead and
//       form y_loc = S_e u_e, one thread per row, fixed summation order.
//   sc_node_kernel        every exterior node sums its entries of y_loc in the
//       fixed order of the node -> entries table (the reference's
//       `grhs[inds_ext] += ...`, :499, without atomics), applies the Dirichlet
//       elimination (:505-510) and takes the fused u.y.
//
// Local stiffness entry (p,q),(r,s) of  y = D^T (G00 ur + G01 us) + (G01 ur + G11 us) D,
// ur = D u, us = u D^T (SURVEY.md appendix C):
//   A = [q==s] sum_m D[m][p] G00[m][q] D[m][r]  +  D[r][p] G01[r][q] D[q][s]
//     + D[p][r] G01[p][s] D[s][q]               +  [p==r] sum_n G11[p][n] D[n][s] D[n][q]
#include <math.h>

#include "semk_common.cuh"

namespace {

constexpr int kScThreads = 128;
constexpr int kScTX = 16, kScTY = 8;  // trailing-update thread tile of the factorisation

template <int N>
struct ScCfg {
  static constexpr int NN = N * N;
  static constexpr int NE = 4 * (N - 1);         // exterior nodes of an element
  static constexpr int NI = (N - 2) * (N - 2);   // interior nodes
  static constexpr int NS = NE * (NE + 1) / 2;   // packed S_e (always even)
  static constexpr int LDI = NI | 1;             // odd row strides: conflict-free columns
  static constexpr int LDZ = NE + 1;             // NE columns of A_ie + the load column
  static constexpr int kDoubles =
      3 * NN + NN + NN + NI * LDI + NI * LDZ + NE * NE + NI + NE + NE + NI + NI * LDI;
  static constexpr size_t kSmem = sizeof(double) * kDoubles + sizeof(int) * (NE + 4);
  static constexpr int EPB = kScThreads / NE;    // elements per CTA step of the matvec
};

struct ScElemArgs {
  int64_t n_elem;
  const int64_t *slot_of_elem;
  const double *G;
  int64_t g_patch_stride;
  int pe;
  const double *D;
  const int32_t *ext_loc;
  int mode;
  double *S_out;
  int64_t s_stride;
  double *sdiag_loc;
  double *W_out;               // [n_elem][NE][NI] A_ii^{-1} A_ie, transposed (mode STORE), or nullptr
  const double *react;         // [n_elem][NN] nodal reaction term added to the local diagonal, or nullptr
  double *Ainv_out;            // [n_elem][NI][NI] A_ii^{-1} (mode STORE_INV), or nullptr
  int32_t *bad_flag;
  // dense mode (semk_sc_element_dense_f64): the caller's own local systems, hierarchical
  // local order (exterior DOFs first), instead of the Poisson recipe on G; the only mode
  // whose loads (RHS, BACKSOLVE) this kernel takes -- the recipe's loads run in
  // sc_element_block_kernel
  double *g_loc;
  double *u;
  const double *A_dense;       // [n_elem][NN][NN] or nullptr
  const double *f_dense;       // [n_elem][NN]
  const uint32_t *l2g_hier;    // [n_elem][NN] global ids in hierarchical local order
};

// ---- element work shared by sc_element_kernel and sc_element_block_kernel -----------------
// Local stiffness entry (p,q),(r,s) from the staged factors (closed form in the file header).
template <int N>
__device__ __forceinline__ double sc_entry(const double *sG, const double *sD, const double *sR,
                                           int p, int q, int r, int s) {
  constexpr int NN = N * N;
  double v = sD[r * N + p] * sG[NN + r * N + q] * sD[q * N + s] +
             sD[p * N + r] * sG[NN + p * N + s] * sD[s * N + q];
  if (q == s) {
#pragma unroll
    for (int m = 0; m < N; ++m) v = fma(sD[m * N + p] * sD[m * N + r], sG[m * N + q], v);
  }
  if (p == r) {
#pragma unroll
    for (int n = 0; n < N; ++n)
      v = fma(sD[n * N + s] * sD[n * N + q], sG[2 * NN + p * N + n], v);
    if (q == s) v += sR[p * N + q];
  }
  return v;
}

// Stage element e's geometric factors, D, reaction term and exterior index table.
template <int N>
__device__ __forceinline__ void sc_stage_element(int64_t e, const int64_t *slot_of_elem,
                                                 const double *G, int64_t g_patch_stride, int pe,
                                                 const double *D, const double *react,
                                                 const int32_t *ext_loc, double *sG, double *sD,
                                                 double *sR, int *sExt, int tid) {
  constexpr int NN = N * N, NE = ScCfg<N>::NE;
  const int NP = N * pe;
  const int64_t slot = slot_of_elem ? slot_of_elem[e] : e;
  const int64_t patch = slot / pe;
  const int lp = (int)(slot - patch * pe);
  const double *g = G + patch * g_patch_stride + lp * N;
  for (int i = tid; i < 3 * NN; i += kScThreads) {
    const int c = i / NN, k = i - c * NN;
    const int m = k / N, n = k - m * N;
    sG[i] = g[(c * N + m) * NP + n];
  }
  for (int i = tid; i < NN; i += kScThreads) sD[i] = D[i];
  for (int i = tid; i < NN; i += kScThreads) sR[i] = react ? react[e * NN + i] : 0.0;
  for (int i = tid; i < NE; i += kScThreads) sExt[i] = ext_loc[i];
}

// Interior block (lower triangle) into sA and A_ie into the first NE columns of sZ.
template <int N>
__device__ __forceinline__ void sc_build_interior(const double *sG, const double *sD,
                                                  const double *sR, const int *sExt, double *sA,
                                                  double *sZ, int ldz, int tid) {
  constexpr int NE = ScCfg<N>::NE, NI = ScCfg<N>::NI, LDI = ScCfg<N>::LDI, M = N - 2;
  for (int idx = tid; idx < NI * NI; idx += kScThreads) {
    const int i = idx / NI, j = idx - i * NI;
    if (j <= i)
      sA[i * LDI + j] = sc_entry<N>(sG, sD, sR, 1 + i / M, 1 + i % M, 1 + j / M, 1 + j % M);
  }
  for (int idx = tid; idx < NI * NE; idx += kScThreads) {
    const int i = idx / NE, k = idx - i * NE;
    const int x = sExt[k];
    sZ[i * ldz + k] = sc_entry<N>(sG, sD, sR, 1 + i / M, 1 + i % M, x / N, x % N);
  }
}

// A_ii = L L^T, right-looking, in place (lower triangle); sInv[i] = 1 / L[i][i].
template <int N>
__device__ __forceinline__ void sc_cholesky(double *sA, double *sInv, int *sBad, int tid) {
  constexpr int NI = ScCfg<N>::NI, LDI = ScCfg<N>::LDI;
  const int tx = tid % kScTX, ty = tid / kScTX;
  for (int k = 0; k < NI; ++k) {
    const double d = sA[k * LDI + k];  // nobody writes (k,k) during step k
    const double inv = 1.0 / sqrt(d);
    if (tid == 0) {
      sInv[k] = inv;
      if (!(d > 0.0)) *sBad = 1;
    }
    for (int i = k + 1 + tid; i < NI; i += kScThreads) sA[i * LDI + k] *= inv;
    __syncthreads();
    for (int i = k + 1 + ty; i < NI; i += kScTY) {
      const double lik = sA[i * LDI + k];
      for (int j = k + 1 + tx; j <= i; j += kScTX)
        sA[i * LDI + j] = fma(-lik, sA[j * LDI + k], sA[i * LDI + j]);
    }
    __syncthreads();
  }
}

// Columns [0, ncols) of sZ <- L^{-1} sZ: one thread per column, forward substitution.
template <int N>
__device__ __forceinline__ void sc_forward(const double *sA, const double *sInv, double *sZ,
                                           int ldz, int ncols, int tid) {
  constexpr int NI = ScCfg<N>::NI, LDI = ScCfg<N>::LDI;
  if (tid < ncols) {
    for (int i = 0; i < NI; ++i) {
      double acc = sZ[i * ldz + tid];
      for (int j = 0; j < i; ++j) acc = fma(-sA[i * LDI + j], sZ[j * ldz + tid], acc);
      sZ[i * ldz + tid] = acc * sInv[i];
    }
  }
}

// Column col of sZ <- L^{-T} sZ (backward substitution in place), by the calling thread.
template <int N>
__device__ __forceinline__ void sc_backward_col(const double *sA, const double *sInv, double *sZ,
                                                int ldz, int col) {
  constexpr int NI = ScCfg<N>::NI, LDI = ScCfg<N>::LDI;
  for (int i = NI - 1; i >= 0; --i) {
    double acc = sZ[i * ldz + col];
    for (int j = i + 1; j < NI; ++j) acc = fma(-sA[j * LDI + i], sZ[j * ldz + col], acc);
    sZ[i * ldz + col] = acc * sInv[i];
  }
}

template <int N>
__global__ void __launch_bounds__(kScThreads) sc_element_kernel(ScElemArgs a) {
  using C = ScCfg<N>;
  constexpr int NN = C::NN, NE = C::NE, NI = C::NI, NS = C::NS, LDI = C::LDI, LDZ = C::LDZ;
  extern __shared__ __align__(128) double sc_smem[];
  double *sG = sc_smem;            // [3][N][N] geometric factors G00, G01, G11
  double *sD = sG + 3 * NN;        // [N][N]
  double *sR = sD + NN;            // [N][N] reaction (nodal diagonal) term, zeros without one
  double *sA = sR + NN;            // [NI][LDI] interior block -> Cholesky factor (lower)
  double *sZ = sA + NI * LDI;      // [NI][LDZ] A_ie | f_i  ->  L^{-1} of both
  double *sE = sZ + NI * LDZ;      // [NE][NE] A_ee (lower part used)
  double *sInv = sE + NE * NE;     // [NI] 1 / L[i][i]
  double *sFe = sInv + NI;         // [NE] exterior part of the load
  double *sUe = sFe + NE;          // [NE] exterior values (back-substitution)
  double *sT = sUe + NE;           // [NI] back-substitution vector
  double *sX = sT + NI;            // [NI][LDI] L^{-1} (mode STORE_INV only)
  int *sExt = reinterpret_cast<int *>(sX + NI * LDI);  // [NE] lexicographic index of exterior k
  int *sBad = sExt + NE;
  const int tid = threadIdx.x;
  const bool need_f = (a.mode & (SEMK_SC_RHS | SEMK_SC_BACKSOLVE)) != 0;  // dense mode only

  auto entry = [&](int p, int q, int r, int s) -> double {
    return sc_entry<N>(sG, sD, sR, p, q, r, s);
  };

  for (int64_t e = blockIdx.x; e < a.n_elem; e += gridDim.x) {
    __syncthreads();  // the previous element is completely done with shared memory
    if (!a.A_dense) {
      sc_stage_element<N>(e, a.slot_of_elem, a.G, a.g_patch_stride, a.pe, a.D, a.react,
                          a.ext_loc, sG, sD, sR, sExt, tid);
    }
    if (tid == 0) *sBad = 0;
    __syncthreads();
    // ---- local stiffness blocks --------------------------------------------------
    if (a.A_dense) {
      // the caller's local matrix, hierarchical order: rows / columns [0, NE) exterior,
      // [NE, NN) interior (reorder_local_system_hier, sem/discrete.py:428-436)
      const double *A = a.A_dense + e * (int64_t)NN * NN;
      for (int idx = tid; idx < NI * NI; idx += kScThreads) {
        const int i = idx / NI, j = idx - i * NI;
        if (j <= i) sA[i * LDI + j] = A[(int64_t)(NE + i) * NN + NE + j];
      }
      for (int idx = tid; idx < NI * NE; idx += kScThreads) {
        const int i = idx / NE, k = idx - i * NE;
        sZ[i * LDZ + k] = A[(int64_t)(NE + i) * NN + k];
      }
      for (int idx = tid; idx < NE * NE; idx += kScThreads) {
        const int k = idx / NE, l = idx - k * NE;
        if (l <= k) sE[idx] = A[(int64_t)k * NN + l];
      }
      if (need_f) {
        const double *fh = a.f_dense + e * (int64_t)NN;
        const uint32_t *row = a.l2g_hier + e * (int64_t)NN;
        for (int i = tid; i < NI; i += kScThreads) sZ[i * LDZ + NE] = fh[NE + i];
        for (int k = tid; k < NE; k += kScThreads) {
          sFe[k] = fh[k];
          if (a.mode & SEMK_SC_BACKSOLVE) sUe[k] = a.u[row[k]];
        }
      }
    } else {
    sc_build_interior<N>(sG, sD, sR, sExt, sA, sZ, LDZ, tid);
    for (int idx = tid; idx < NE * NE; idx += kScThreads) {
      const int k = idx / NE, l = idx - k * NE;
      if (l <= k) {
        const int x = sExt[k], z = sExt[l];
        sE[idx] = entry(x / N, x % N, z / N, z % N);
      }
    }
    }
    __syncthreads();
    sc_cholesky<N>(sA, sInv, sBad, tid);
    // ---- Z = L^{-1} [A_ie | f_i] ------------------------------------------------------
    sc_forward<N>(sA, sInv, sZ, LDZ, NE + (need_f ? 1 : 0), tid);
    __syncthreads();
    if (tid == 0 && *sBad) *a.bad_flag = 1;
    // ---- S_e = A_ee - Z^T Z (packed lower triangle, row major) ----------------------
    if (a.mode & SEMK_SC_SCHUR) {
      double *So = a.S_out + e * a.s_stride;
      for (int q = tid; q < NS; q += kScThreads) {
        int k = (int)((sqrt(8.0 * q + 1.0) - 1.0) * 0.5);
        while ((k + 1) * (k + 2) / 2 <= q) ++k;
        while (k * (k + 1) / 2 > q) --k;
        const int l = q - k * (k + 1) / 2;
        double acc = sE[k * NE + l];
        for (int i = 0; i < NI; ++i) acc = fma(-sZ[i * LDZ + k], sZ[i * LDZ + l], acc);
        So[q] = acc;
        if (k == l && a.sdiag_loc) a.sdiag_loc[e * NE + k] = acc;
      }
    }
    // ---- g_e = f_e - Z^T (L^{-1} f_i) ------------------------------------------------
    if (a.mode & SEMK_SC_RHS) {
      for (int k = tid; k < NE; k += kScThreads) {
        double acc = sFe[k];
        for (int i = 0; i < NI; ++i) acc = fma(-sZ[i * LDZ + k], sZ[i * LDZ + NE], acc);
        a.g_loc[e * NE + k] = acc;
      }
    }
    // ---- u_i = L^{-T} (L^{-1} f_i - Z u_e) -------------------------------------------
    if (a.mode & SEMK_SC_BACKSOLVE) {
      for (int i = tid; i < NI; i += kScThreads) {
        double acc = sZ[i * LDZ + NE];
        for (int k = 0; k < NE; ++k) acc = fma(-sZ[i * LDZ + k], sUe[k], acc);
        sT[i] = acc;
      }
      __syncthreads();
      if (tid < 32) {
        for (int i = NI - 1; i >= 0; --i) {
          const double xi = sT[i] * sInv[i];
          __syncwarp();
          if (tid == 0) sT[i] = xi;
          for (int j = tid; j < i; j += 32) sT[j] = fma(-sA[i * LDI + j], xi, sT[j]);
          __syncwarp();
        }
      }
      __syncthreads();
      const uint32_t *row = a.l2g_hier + e * (int64_t)NN;
      for (int i = tid; i < NI; i += kScThreads) a.u[row[NE + i]] = sT[i];
    }
    // ---- keep A_ii^{-1} = L^{-T} L^{-1} (symmetric, dense): with W it turns the condensed
    // load of ANY later right-hand side into a streaming pass (sc_load_stored_block_kernel) --
    if ((a.mode & SEMK_SC_STORE_INV) && a.Ainv_out) {
      __syncthreads();
      if (tid < NI) {   // column tid of L^{-1}: forward substitution of the unit vector
        for (int i = 0; i < tid; ++i) sX[i * LDI + tid] = 0.0;
        sX[tid * LDI + tid] = sInv[tid];
        for (int i = tid + 1; i < NI; ++i) {
          double acc = 0.0;
          for (int j = tid; j < i; ++j) acc = fma(-sA[i * LDI + j], sX[j * LDI + tid], acc);
          sX[i * LDI + tid] = acc * sInv[i];
        }
      }
      __syncthreads();
      double *Ao = a.Ainv_out + e * (int64_t)NI * NI;
      for (int idx = tid; idx < NI * NI; idx += kScThreads) {
        const int i = idx / NI, j = idx - i * NI;
        const int k0 = i > j ? i : j;
        double acc = 0.0;
        for (int k = k0; k < NI; ++k) acc = fma(sX[k * LDI + i], sX[k * LDI + j], acc);
        Ao[idx] = acc;
      }
    }
    // ---- keep the interior solution operator W = A_ii^{-1} A_ie = L^{-T} Z, one thread per
    // column, backward substitution in place; the back-substitution u_i = c - W u_e then is
    // one streaming pass (sc_backsolve_stored_block_kernel) instead of a refactorisation per
    // element --------------------------------------------------------------------------------
    if ((a.mode & SEMK_SC_STORE) && a.W_out) {
      __syncthreads();  // every reader of Z is done
      if (tid < NE) sc_backward_col<N>(sA, sInv, sZ, LDZ, tid);
      __syncthreads();
      double *Wo = a.W_out + e * (int64_t)NE * NI;
      for (int idx = tid; idx < NE * NI; idx += kScThreads) {
        const int k = idx / NI, i = idx - k * NI;
        Wo[idx] = sZ[i * LDZ + k];
      }
    }
  }
}

// ---- loads: up to kScBlockMaxCols load columns per pass --------------------------------------
// Column j's load is f_scale[j] * JxW * (nodal_mask bit j ? F[j][l2g] : 1), and every column
// goes through the same operations in the same order whatever k and the other columns, so each
// column is bitwise the result of a one-column pass (the single-load entries).
constexpr int kScBlockMaxCols = 32;

struct ScBlockLoad {
  int k;                            // load columns, 1..kScBlockMaxCols
  const double *F;                  // [k][ldf] nodal loads (rows of scalar columns unread)
  int64_t ldf;
  uint32_t nodal_mask;              // bit j: column j is nodal
  double f_scale[kScBlockMaxCols];
};

__device__ __forceinline__ double sc_block_load(const ScBlockLoad &L, int j, const double *jw,
                                                const uint32_t *row, int x) {
  const double f = ((L.nodal_mask >> j) & 1u) ? L.F[j * L.ldf + row[x]] : 1.0;
  return L.f_scale[j] * jw[x] * f;
}

struct ScBlockArgs {
  int64_t n_elem;
  const int64_t *slot_of_elem;
  const double *G;
  int64_t g_patch_stride;
  int pe;
  const double *D;
  const int32_t *ext_loc;
  const uint32_t *l2g;
  const double *JxW;
  const double *react;
  int mode;                         // SEMK_SC_RHS or SEMK_SC_BACKSOLVE
  ScBlockLoad L;
  double *g_loc;                    // RHS: [k][ldg], row j = [n_elem][NE]
  int64_t ldg;
  double *c_out;                    // optional: [k][ldc], row j = [n_elem][NI] = A_ii^{-1} f_i
  int64_t ldc;
  double *U;                        // BACKSOLVE: [k][ldu] nodal vectors
  int64_t ldu;
  int32_t *bad_flag;
};

// shared memory of sc_element_block_kernel: Z takes (NE + k) | 1 columns; sV holds f_e (RHS) or
// u_e (BACKSOLVE) of every column, sT the k back-substitution vectors (BACKSOLVE only)
template <int N>
size_t sc_block_smem(int k, int mode) {
  using C = ScCfg<N>;
  const size_t ldz = (size_t)((C::NE + k) | 1);
  const size_t nd = 3 * C::NN + 2 * C::NN + C::NI * C::LDI + C::NI * ldz + C::NI +
                    (size_t)k * C::NE + (mode == SEMK_SC_BACKSOLVE ? (size_t)k * C::NI : 0);
  return sizeof(double) * nd + sizeof(int) * (C::NE + 4);
}

template <int N>
__global__ void __launch_bounds__(kScThreads, 1) sc_element_block_kernel(ScBlockArgs a) {
  using C = ScCfg<N>;
  constexpr int NN = C::NN, NE = C::NE, NI = C::NI, LDI = C::LDI, M = N - 2;
  const int k = a.L.k, ldz = (NE + k) | 1;
  const bool back = a.mode == SEMK_SC_BACKSOLVE;
  extern __shared__ __align__(128) double sc_smem[];
  double *sG = sc_smem;            // [3][N][N]
  double *sD = sG + 3 * NN;        // [N][N]
  double *sR = sD + NN;            // [N][N]
  double *sA = sR + NN;            // [NI][LDI] -> Cholesky factor
  double *sZ = sA + NI * LDI;      // [NI][ldz] A_ie | f_i of every column -> L^{-1} of all
  double *sInv = sZ + NI * ldz;    // [NI]
  double *sV = sInv + NI;          // [k][NE] f_e (RHS) or u_e (BACKSOLVE)
  double *sT = sV + k * NE;        // [k][NI] (BACKSOLVE)
  int *sExt = reinterpret_cast<int *>(sT + (back ? k * NI : 0));
  int *sBad = sExt + NE;
  const int tid = threadIdx.x;
  for (int64_t e = blockIdx.x; e < a.n_elem; e += gridDim.x) {
    __syncthreads();
    sc_stage_element<N>(e, a.slot_of_elem, a.G, a.g_patch_stride, a.pe, a.D, a.react, a.ext_loc, sG, sD,
                        sR, sExt, tid);
    if (tid == 0) *sBad = 0;
    __syncthreads();
    sc_build_interior<N>(sG, sD, sR, sExt, sA, sZ, ldz, tid);
    const double *jw = a.JxW + e * NN;
    const uint32_t *row = a.l2g + e * NN;
    for (int idx = tid; idx < k * NI; idx += kScThreads) {
      const int j = idx / NI, i = idx - j * NI;
      sZ[i * ldz + NE + j] = sc_block_load(a.L, j, jw, row, (1 + i / M) * N + 1 + i % M);
    }
    for (int idx = tid; idx < k * NE; idx += kScThreads) {
      const int j = idx / NE, q = idx - j * NE;
      sV[idx] = back ? a.U[j * a.ldu + row[sExt[q]]] : sc_block_load(a.L, j, jw, row, sExt[q]);
    }
    __syncthreads();
    sc_cholesky<N>(sA, sInv, sBad, tid);
    sc_forward<N>(sA, sInv, sZ, ldz, NE + k, tid);
    __syncthreads();
    if (tid == 0 && *sBad) *a.bad_flag = 1;
    if (!back) {
      // g_e = f_e - Z^T (L^{-1} f_i)
      for (int idx = tid; idx < k * NE; idx += kScThreads) {
        const int j = idx / NE, q = idx - j * NE;
        double acc = sV[idx];
        for (int i = 0; i < NI; ++i) acc = fma(-sZ[i * ldz + q], sZ[i * ldz + NE + j], acc);
        a.g_loc[j * a.ldg + e * NE + q] = acc;
      }
    } else {
      // u_i = L^{-T} (L^{-1} f_i - Z u_e): the product one thread per entry, the backward
      // sweep one warp per column
      for (int idx = tid; idx < k * NI; idx += kScThreads) {
        const int j = idx / NI, i = idx - j * NI;
        const double *ue = sV + j * NE;
        double acc = sZ[i * ldz + NE + j];
        for (int q = 0; q < NE; ++q) acc = fma(-sZ[i * ldz + q], ue[q], acc);
        sT[idx] = acc;
      }
      __syncthreads();
      const int warp = tid >> 5, lane = tid & 31;
      for (int j = warp; j < k; j += kScThreads / 32) {
        double *t = sT + j * NI;
        for (int i = NI - 1; i >= 0; --i) {
          const double xi = t[i] * sInv[i];
          __syncwarp();
          if (lane == 0) t[i] = xi;
          for (int jj = lane; jj < i; jj += 32) t[jj] = fma(-sA[i * LDI + jj], xi, t[jj]);
          __syncwarp();
        }
      }
      __syncthreads();
      for (int idx = tid; idx < k * NI; idx += kScThreads) {
        const int j = idx / NI, i = idx - j * NI;
        a.U[j * a.ldu + row[(1 + i / M) * N + 1 + i % M]] = sT[idx];
      }
    }
    if (a.c_out) {  // c = L^{-T} (L^{-1} f_i), one thread per column
      __syncthreads();
      if (tid < k) sc_backward_col<N>(sA, sInv, sZ, ldz, NE + tid);
      __syncthreads();
      for (int idx = tid; idx < k * NI; idx += kScThreads) {
        const int j = idx / NI, i = idx - j * NI;
        a.c_out[j * a.ldc + e * NI + i] = sZ[i * ldz + NE + j];
      }
    }
  }
}

// An unroll count of 0 is ignored: the wider tiles' element loops stay the compiler's choice.
constexpr int kScCompilerUnroll = 0;
#pragma nv_diag_suppress 20168

// Back-substitution from the stored interior operator: u_i = c - W u_e for every element and
// each of k <= KB columns, one thread per interior row; W is stored transposed ([NE][NI]), so
// the NI threads of an element read consecutive doubles, and it is read once for all columns
// (a pure stream: 12.5 KB per element at p = 8).  KB (1, 2, 4, ... 32) is the register tile:
// the launch takes the smallest that holds k, so that a few columns do not pay for 32
// predicated accumulators.  The one-column tile is a latency-bound stream: it keeps eight
// CTAs per SM (32 registers) and eight loads of W in flight per thread.
template <int N, int KB>
__global__ void __launch_bounds__(256, KB == 1 ? 8 : 1)
    sc_backsolve_stored_block_kernel(int64_t n_elem, const double *__restrict__ W,
                                     const double *__restrict__ c, int64_t ldc,
                                     const uint32_t *__restrict__ l2g,
                                     const int32_t *__restrict__ ext_loc, int k,
                                     double *__restrict__ U, int64_t ldu) {
  using C = ScCfg<N>;
  constexpr int NN = C::NN, NE = C::NE, NI = C::NI, M = N - 2;
  constexpr int GT = ((NI + 31) / 32) * 32;
  constexpr int GPB = 256 / GT;
  extern __shared__ __align__(128) double sc_smem[];   // [GPB][k][NE] exterior values
  const int tid = threadIdx.x;
  const int grp = tid / GT, i = tid - grp * GT;
  double *sUe = sc_smem + (grp < GPB ? grp : 0) * k * NE;
  const int64_t n_steps = (n_elem + GPB - 1) / GPB;
  for (int64_t step = blockIdx.x; step < n_steps; step += gridDim.x) {
    const int64_t e = step * GPB + grp;
    const bool on = grp < GPB && e < n_elem;
    __syncthreads();
    if (on) {
      const uint32_t *row = l2g + e * NN;
      for (int idx = i; idx < k * NE; idx += GT) {
        const int j = idx / NE, q = idx - j * NE;
        sUe[idx] = U[j * ldu + row[ext_loc[q]]];
      }
    }
    __syncthreads();
    if (on && i < NI) {
      double acc[KB];
#pragma unroll
      for (int j = 0; j < KB; ++j)
        acc[j] = (j < k && c) ? c[j * ldc + e * (int64_t)NI + i] : 0.0;
      const double *Wt = W + e * (int64_t)NE * NI + i;
#pragma unroll(KB == 1 ? 8 : kScCompilerUnroll)
      for (int q = 0; q < NE; ++q) {
        const double w = __ldcs(Wt + (int64_t)q * NI);
#pragma unroll
        for (int j = 0; j < KB; ++j)
          if (j < k) acc[j] = fma(-w, sUe[j * NE + q], acc[j]);
      }
      const int64_t g = l2g[e * NN + (1 + i / M) * N + 1 + i % M];
#pragma unroll
      for (int j = 0; j < KB; ++j)
        if (j < k) U[j * ldu + g] = acc[j];
    }
  }
}

// Condensed load from the stored interior operators: for every element and each of k <= KB
// columns  c = A_ii^{-1} f_i,  g = f_e - W^T f_i  (A_ei A_ii^{-1} = W^T by symmetry).  A pure
// stream over A_ii^{-1} (19 KB) and W (12.5 KB per element at p = 8), read once for all columns,
// instead of a refactorisation per element.  The one-column tile keeps seven loads of
// A_ii^{-1} in flight per thread.
template <int N, int KB>
__global__ void __launch_bounds__(256)
    sc_load_stored_block_kernel(int64_t n_elem, const double *__restrict__ W,
                                const double *__restrict__ Ainv, const uint32_t *__restrict__ l2g,
                                const int32_t *__restrict__ ext_loc,
                                const double *__restrict__ JxW, ScBlockLoad L,
                                double *__restrict__ g_loc, int64_t ldg,
                                double *__restrict__ c_out, int64_t ldc) {
  using C = ScCfg<N>;
  constexpr int NN = C::NN, NE = C::NE, NI = C::NI, M = N - 2;
  constexpr int GT = ((NI + 31) / 32) * 32;
  constexpr int GPB = 256 / GT;
  extern __shared__ __align__(128) double sc_smem[];   // [GPB][k][NN] element loads
  const int k = L.k;
  const int tid = threadIdx.x;
  const int grp = tid / GT, i = tid - grp * GT;
  double *sF = sc_smem + (grp < GPB ? grp : 0) * k * NN;
  const int64_t n_steps = (n_elem + GPB - 1) / GPB;
  for (int64_t step = blockIdx.x; step < n_steps; step += gridDim.x) {
    const int64_t e = step * GPB + grp;
    const bool on = grp < GPB && e < n_elem;
    __syncthreads();
    if (on) {
      const uint32_t *row = l2g + e * NN;
      const double *jw = JxW + e * NN;
      for (int idx = i; idx < k * NN; idx += GT) {
        const int j = idx / NN, x = idx - j * NN;
        sF[idx] = sc_block_load(L, j, jw, row, x);
      }
    }
    __syncthreads();
    double acc[KB];
    if (on && i < NI) {
      const double *Ac = Ainv + e * (int64_t)NI * NI + i;
#pragma unroll
      for (int j = 0; j < KB; ++j) acc[j] = 0.0;
#pragma unroll(KB == 1 ? 7 : kScCompilerUnroll)
      for (int jj = 0; jj < NI; ++jj) {
        const double v = __ldcs(Ac + (int64_t)jj * NI);
        const int x = (1 + jj / M) * N + 1 + jj % M;
#pragma unroll
        for (int j = 0; j < KB; ++j)
          if (j < k) acc[j] = fma(v, sF[j * NN + x], acc[j]);
      }
#pragma unroll
      for (int j = 0; j < KB; ++j)
        if (j < k) c_out[j * ldc + e * (int64_t)NI + i] = acc[j];
    }
    if (on && i < NE) {
      const double *Wr = W + e * (int64_t)NE * NI + (int64_t)i * NI;
      const int xe = ext_loc[i];
#pragma unroll
      for (int j = 0; j < KB; ++j) acc[j] = j < k ? sF[j * NN + xe] : 0.0;
      for (int jj = 0; jj < NI; ++jj) {
        const double w = Wr[jj];
        const int x = (1 + jj / M) * N + 1 + jj % M;
#pragma unroll
        for (int j = 0; j < KB; ++j)
          if (j < k) acc[j] = fma(-w, sF[j * NN + x], acc[j]);
      }
#pragma unroll
      for (int j = 0; j < KB; ++j)
        if (j < k) g_loc[j * ldg + e * (int64_t)NE + i] = acc[j];
    }
  }
}

// ---- condensed apply, element part: y_loc = S_e u[l2g_ext] ------------------------------
// Persistent and double-buffered: while group i (EPB elements) is being multiplied,
// the TMA engine (cp.async.bulk, evict-first: S is streamed exactly once per apply)
// fills the other stage with the S blocks of the CTA's next group and every thread has
// its next u value in flight (index load, then value load); one barrier per group.
// One thread per row of S_e; entry (r, c), r >= c, of the packed block sits at
// r (r + 1) / 2 + c, so a half-warp reading one column hits 16 distinct banks
// (triangular numbers are a permutation mod 16).
template <int N>
__global__ void __launch_bounds__(kScThreads)
    sc_matvec_kernel(int64_t n_elem, const double *__restrict__ S,
                         const uint32_t *__restrict__ l2g_ext, const double *__restrict__ u,
                         const uint8_t *__restrict__ mask_in, double *__restrict__ y_loc) {
  using C = ScCfg<N>;
  constexpr int NE = C::NE, NS = C::NS, EPB = C::EPB;
  constexpr int STG = EPB * NS, UST = EPB * NE;
  extern __shared__ __align__(128) double sc_smem[];
  double *sS = sc_smem;                                            // [2][EPB][NS]
  double *sU = sS + 2 * STG;                                       // [2][EPB][NE]
  uint64_t *mbar = reinterpret_cast<uint64_t *>(sU + 2 * UST);     // [2]
  const int tid = threadIdx.x;
  const int le = tid / NE, k = tid - le * NE;
  const bool lane_on = le < EPB;
  const int64_t n_groups = (n_elem + EPB - 1) / EPB;
  const uint64_t policy = semk_policy_evict_first();
  if (tid == 0) {
    semk_mbar_init(&mbar[0], 1);
    semk_mbar_init(&mbar[1], 1);
    semk_fence_mbar_init();
  }
  __syncthreads();
  auto count_of = [&](int64_t grp) -> int {
    const int64_t left = n_elem - grp * EPB;
    return (int)(left < (int64_t)EPB ? left : (int64_t)EPB);
  };
  auto issue = [&](int64_t grp, int s) {  // thread 0
    const uint32_t bytes = (uint32_t)(count_of(grp) * NS * sizeof(double));
    semk_mbar_expect_tx(&mbar[s], bytes);
    semk_bulk_g2s_hint(sS + s * STG, S + grp * EPB * NS, bytes, &mbar[s], policy);
  };
  auto gather = [&](int64_t grp) -> double {
    double v = 0.0;
    if (lane_on && le < count_of(grp)) {
      const uint32_t g = l2g_ext[(grp * EPB + le) * NE + k];
      v = u[g];
      if (mask_in && mask_in[g]) v = 0.0;
    }
    return v;
  };
  int64_t grp = blockIdx.x;
  if (grp >= n_groups) return;
  if (tid == 0) issue(grp, 0);
  double unext = gather(grp);
  if (lane_on) sU[tid] = unext;
  __syncthreads();
  for (int it = 0;; ++it) {
    const int s = it & 1;
    const int64_t nxt = grp + gridDim.x;
    const bool more = nxt < n_groups;
    if (more) {
      if (tid == 0) issue(nxt, s ^ 1);  // stage s^1 was last read before the barrier below
      unext = gather(nxt);
    }
    semk_mbar_wait(&mbar[s], (uint32_t)((it >> 1) & 1));
    if (lane_on && le < count_of(grp)) {
      const double *sm = sS + s * STG + le * NS;
      const double *uu = sU + s * UST + le * NE;
      const int kk = k * (k + 1) / 2;
      double acc = 0.0;
#pragma unroll
      for (int j = 0; j < NE; ++j) {
        const int idx = (j <= k) ? kk + j : j * (j + 1) / 2 + k;
        acc = fma(sm[idx], uu[j], acc);
      }
      y_loc[(grp * EPB + le) * NE + k] = acc;
    }
    if (!more) break;
    if (lane_on) sU[(s ^ 1) * UST + tid] = unext;
    __syncthreads();
    grp = nxt;
  }
}

template <int N>
constexpr size_t sc_matvec_smem() {
  return sizeof(double) * (2 * (size_t)ScCfg<N>::EPB * (ScCfg<N>::NS + ScCfg<N>::NE)) + 16;
}

// ---- vertex coarse space of the two-level preconditioner ----------------------------------
// Ace = Phi_e^T S_e Phi_e, Phi_e = diag(free nodes) phi diag(free vertices).
template <int N>
__global__ void __launch_bounds__(kScThreads)
    sc_coarse_elem_kernel(int64_t n_elem, const double *__restrict__ S,
                          const uint32_t *__restrict__ l2g_ext,
                          const uint8_t *__restrict__ dirichlet, const double *__restrict__ phi,
                          double *__restrict__ Ace) {
  using C = ScCfg<N>;
  constexpr int NE = C::NE, NS = C::NS, EPB = C::EPB;
  extern __shared__ __align__(128) double sc_smem[];
  double *sS = sc_smem;                 // [EPB][NS]
  double *sP0 = sS + EPB * NS;          // [NE][4] phi
  double *sPhi = sP0 + NE * 4;          // [EPB][NE][4] masked Phi_e
  double *sT = sPhi + EPB * NE * 4;     // [EPB][NE][4] S_e Phi_e
  const int tid = threadIdx.x;
  const int le = tid / NE, k = tid - le * NE;
  for (int i = tid; i < NE * 4; i += kScThreads) sP0[i] = phi[i];
  const int64_t n_groups = (n_elem + EPB - 1) / EPB;
  for (int64_t grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
    __syncthreads();
    const int64_t e0 = grp * EPB;
    const int ne = (int)((n_elem - e0) < (int64_t)EPB ? (n_elem - e0) : (int64_t)EPB);
    const double2 *src = reinterpret_cast<const double2 *>(S + e0 * NS);
    double2 *dst = reinterpret_cast<double2 *>(sS);
    for (int q = tid; q < ne * (NS / 2); q += kScThreads) dst[q] = src[q];
    const bool on = le < ne;
    if (on) {
      const uint32_t *ids = l2g_ext + (e0 + le) * NE;
      const double fn = (dirichlet && dirichlet[ids[k]]) ? 0.0 : 1.0;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const double fv = (dirichlet && dirichlet[ids[c]]) ? 0.0 : 1.0;  // vertices: k = 0..3
        sPhi[(le * NE + k) * 4 + c] = sP0[k * 4 + c] * fn * fv;
      }
    }
    __syncthreads();
    if (on) {
      const double *s = sS + le * NS;
      const double *ph = sPhi + le * NE * 4;
      const int kk = k * (k + 1) / 2;
      double t[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
      for (int j = 0; j < NE; ++j) {
        const double sv = s[(j <= k) ? kk + j : j * (j + 1) / 2 + k];
#pragma unroll
        for (int c = 0; c < 4; ++c) t[c] = fma(sv, ph[j * 4 + c], t[c]);
      }
#pragma unroll
      for (int c = 0; c < 4; ++c) sT[(le * NE + k) * 4 + c] = t[c];
    }
    __syncthreads();
    for (int q = tid; q < ne * 16; q += kScThreads) {
      const int l2 = q >> 4, a = (q >> 2) & 3, c = q & 3;
      const double *ph = sPhi + l2 * NE * 4;
      const double *tt = sT + l2 * NE * 4;
      double acc = 0.0;
      for (int j = 0; j < NE; ++j) acc = fma(ph[j * 4 + a], tt[j * 4 + c], acc);
      Ace[(e0 + l2) * 16 + a * 4 + c] = acc;
    }
  }
}

template <int N>
constexpr size_t sc_coarse_elem_smem() {
  return sizeof(double) * ((size_t)ScCfg<N>::EPB * ScCfg<N>::NS + (size_t)ScCfg<N>::NE * 4 +
                           2 * (size_t)ScCfg<N>::EPB * ScCfg<N>::NE * 4);
}

// element part of the coarse apply: y_loc_c[e][a] = sum_c Ace[e][a][c] x[vert_c[e][c]]
__global__ void __launch_bounds__(256)
    sc_coarse_matvec_kernel(int64_t n_elem, const double *__restrict__ Ace,
                            const uint32_t *__restrict__ vert_c, const double *__restrict__ x,
                            double *__restrict__ y_loc_c) {
  const int64_t total = n_elem * 4;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e = i >> 2;
    const double *A = Ace + e * 16 + (i & 3) * 4;
    const uint32_t *v = vert_c + e * 4;
    double acc = A[0] * x[v[0]];
    acc = fma(A[1], x[v[1]], acc);
    acc = fma(A[2], x[v[2]], acc);
    acc = fma(A[3], x[v[3]], acc);
    y_loc_c[i] = acc;
  }
}

// ---- condensed apply / assembly, node part ------------------------------------------------
constexpr int kNodeThreads = 256;

__global__ void __launch_bounds__(kNodeThreads)
    sc_node_kernel(int64_t n_ext, const uint32_t *__restrict__ node_ptr,
                   const uint32_t *__restrict__ node_pos, const double *__restrict__ loc,
                   const uint8_t *__restrict__ dirichlet, const double *__restrict__ u,
                   double *__restrict__ y, int flags, double fill, double *__restrict__ partials,
                   double *__restrict__ dot_out) {
  double acc[1] = {0.0};
  const bool mask_out = dirichlet && (flags & SEMK_MASK_OUT);
  const bool identity = (flags & SEMK_DIRICHLET_IDENTITY) && u;
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < n_ext;
       g += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t q0 = node_ptr[g], q1 = node_ptr[g + 1];
    double s = 0.0;
    for (uint32_t q = q0; q < q1; ++q) s += loc[node_pos[q]];
    if (mask_out && dirichlet[g]) s = identity ? u[g] : fill;
    y[g] = s;
    if (dot_out) acc[0] = fma(u[g], s, acc[0]);
  }
  if (dot_out) {
    double tot[1];
    if (semk_finish_reduction<1>(acc, partials, tot) && threadIdx.x == 0) dot_out[0] = tot[0];
  }
}

inline unsigned node_blocks(int64_t n) {
  const int64_t want = (n + kNodeThreads - 1) / kNodeThreads;
  return (unsigned)(want < 1 ? 1 : (want < kSemkRedMaxBlocks ? want : kSemkRedMaxBlocks));
}

int check_sc_op(const semk_sc_op *op, const char *who) {
  if (!op) {
    semk_set_error(std::string(who) + ": null operator");
    return SEMK_ERR_INVALID;
  }
  if (op->n1 < 3 || op->n1 > 11) {
    semk_set_error(std::string(who) + ": static condensation supports orders 2..10");
    return SEMK_ERR_UNSUPPORTED;
  }
  const int ne = 4 * (op->n1 - 1);
  if (op->n_ext_loc != ne || op->s_stride != (int64_t)ne * (ne + 1) / 2 || op->n_elem <= 0 ||
      op->n_ext <= 0 || !op->S || !op->l2g_ext || !op->y_loc || !op->node_ptr ||
      !op->node_pos) {
    semk_set_error(std::string(who) + ": inconsistent semk_sc_op");
    return SEMK_ERR_INVALID;
  }
  if ((reinterpret_cast<uintptr_t>(op->S) & 15u) != 0) {
    semk_set_error(std::string(who) + ": S must be 16-byte aligned");
    return SEMK_ERR_INVALID;
  }
  return SEMK_OK;
}

// launch of a stored block kernel with the smallest register tile KB >= k
template <int N, int KB>
int launch_load_stored_block(int64_t n_elem, const double *W, const double *Ainv,
                             const uint32_t *l2g, const int32_t *ext_loc, const double *JxW,
                             const ScBlockLoad &L, double *g_loc, int64_t ldg, double *c_out,
                             int64_t ldc, cudaStream_t st) {
  constexpr int GT = ((ScCfg<N>::NI + 31) / 32) * 32, GPB = 256 / GT;
  const size_t smem = sizeof(double) * (size_t)GPB * L.k * ScCfg<N>::NN;
  SEMK_CUDA_CHECK(cudaFuncSetAttribute(sc_load_stored_block_kernel<N, KB>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)(sizeof(double) * GPB * KB * ScCfg<N>::NN)));
  const int64_t steps = (n_elem + GPB - 1) / GPB;
  const unsigned grid = (unsigned)(steps < 148 * 16 ? steps : 148 * 16);
  sc_load_stored_block_kernel<N, KB><<<grid, 256, smem, st>>>(n_elem, W, Ainv, l2g, ext_loc, JxW,
                                                              L, g_loc, ldg, c_out, ldc);
  return SEMK_OK;
}

template <int N, int KB>
int launch_backsolve_stored_block(int64_t n_elem, const double *W, const double *c, int64_t ldc,
                                  const uint32_t *l2g, const int32_t *ext_loc, int k, double *U,
                                  int64_t ldu, cudaStream_t st) {
  constexpr int GT = ((ScCfg<N>::NI + 31) / 32) * 32, GPB = 256 / GT;
  const size_t smem = sizeof(double) * (size_t)GPB * k * ScCfg<N>::NE;
  const int64_t steps = (n_elem + GPB - 1) / GPB;
  const unsigned grid = (unsigned)(steps < 148 * 16 ? steps : 148 * 16);
  sc_backsolve_stored_block_kernel<N, KB><<<grid, 256, smem, st>>>(n_elem, W, c, ldc, l2g,
                                                                   ext_loc, k, U, ldu);
  return SEMK_OK;
}

template <int N>
int launch_load_stored_block_tiled(int64_t n_elem, const double *W, const double *Ainv,
                                   const uint32_t *l2g, const int32_t *ext_loc, const double *JxW,
                                   const ScBlockLoad &L, double *g_loc, int64_t ldg,
                                   double *c_out, int64_t ldc, cudaStream_t st) {
#define SEMK_TILE(KB) \
  return launch_load_stored_block<N, KB>(n_elem, W, Ainv, l2g, ext_loc, JxW, L, g_loc, ldg, \
                                         c_out, ldc, st)
  if (L.k <= 1) SEMK_TILE(1);
  if (L.k <= 2) SEMK_TILE(2);
  if (L.k <= 4) SEMK_TILE(4);
  if (L.k <= 8) SEMK_TILE(8);
  if (L.k <= 16) SEMK_TILE(16);
  SEMK_TILE(32);
#undef SEMK_TILE
}

template <int N>
int launch_backsolve_stored_block_tiled(int64_t n_elem, const double *W, const double *c,
                                        int64_t ldc, const uint32_t *l2g, const int32_t *ext_loc,
                                        int k, double *U, int64_t ldu, cudaStream_t st) {
#define SEMK_TILE(KB) \
  return launch_backsolve_stored_block<N, KB>(n_elem, W, c, ldc, l2g, ext_loc, k, U, ldu, st)
  if (k <= 1) SEMK_TILE(1);
  if (k <= 2) SEMK_TILE(2);
  if (k <= 4) SEMK_TILE(4);
  if (k <= 8) SEMK_TILE(8);
  if (k <= 16) SEMK_TILE(16);
  SEMK_TILE(32);
#undef SEMK_TILE
}

}  // namespace

#define SEMK_DISPATCH_SC(n1, CALL)                                                   \
  switch (n1) {                                                                      \
    case 3: CALL(3); break;                                                          \
    case 4: CALL(4); break;                                                          \
    case 5: CALL(5); break;                                                          \
    case 6: CALL(6); break;                                                          \
    case 7: CALL(7); break;                                                          \
    case 8: CALL(8); break;                                                          \
    case 9: CALL(9); break;                                                          \
    case 10: CALL(10); break;                                                        \
    case 11: CALL(11); break;                                                        \
    default:                                                                         \
      semk_set_error("static condensation supports orders 2..10 (n1 in [3, 11])");   \
      return SEMK_ERR_UNSUPPORTED;                                                   \
  }

static int launch_sc_element(int n1, const ScElemArgs &a, void *stream);
static int launch_sc_element_block(int n1, const ScBlockArgs &a, void *stream);

// one load column f_scale * JxW * (f_nodal ? f_nodal[l2g] : 1): the k = 1 case of ScBlockLoad
static ScBlockLoad sc_single_load(const double *f_nodal, double f_scale) {
  ScBlockLoad L{};
  L.k = 1;
  L.F = f_nodal;
  L.nodal_mask = f_nodal ? 1u : 0u;
  L.f_scale[0] = f_scale;
  return L;
}

extern "C" int semk_sc_element_f64(int n1, int64_t n_elem, const int64_t *slot_of_elem,
                                   const double *G, int64_t g_patch_stride, int elems_per_patch,
                                   const double *D, const int32_t *ext_loc, const uint32_t *l2g,
                                   const double *JxW, const double *f_nodal, double f_scale,
                                   int mode, double *S_out, int64_t s_stride, double *sdiag_loc,
                                   double *g_loc, double *u, double *W_out, double *c_out,
                                   int32_t *bad_flag, void *stream) {
  return semk_sc_element_react_f64(n1, n_elem, slot_of_elem, G, g_patch_stride, elems_per_patch,
                                   D, ext_loc, l2g, JxW, f_nodal, f_scale, mode, S_out, s_stride,
                                   sdiag_loc, g_loc, u, W_out, c_out, nullptr, nullptr, bad_flag,
                                   stream);
}

// The factorisation outputs (SCHUR, STORE, STORE_INV) are one pass of sc_element_kernel, the
// loads (RHS, then BACKSOLVE) one-column passes of sc_element_block_kernel, in that order.
extern "C" int semk_sc_element_react_f64(int n1, int64_t n_elem, const int64_t *slot_of_elem,
                                         const double *G, int64_t g_patch_stride,
                                         int elems_per_patch, const double *D,
                                         const int32_t *ext_loc, const uint32_t *l2g,
                                         const double *JxW, const double *f_nodal,
                                         double f_scale, int mode, double *S_out,
                                         int64_t s_stride, double *sdiag_loc, double *g_loc,
                                         double *u, double *W_out, double *c_out,
                                         const double *react, double *Ainv_out,
                                         int32_t *bad_flag, void *stream) {
  SEMK_REQUIRE(n_elem > 0 && G && D && ext_loc && bad_flag &&
                   elems_per_patch > 0 && g_patch_stride > 0,
               "semk_sc_element_f64: bad argument");
  SEMK_REQUIRE(mode != 0 && (mode & ~31) == 0, "semk_sc_element_f64: bad mode");
  SEMK_REQUIRE(!(mode & SEMK_SC_STORE_INV) || Ainv_out,
               "semk_sc_element_f64: STORE_INV needs Ainv_out");
  SEMK_REQUIRE(!(mode & SEMK_SC_STORE) || W_out, "semk_sc_element_f64: STORE needs W_out");
  SEMK_REQUIRE(!c_out || (mode & (SEMK_SC_RHS | SEMK_SC_BACKSOLVE)),
               "semk_sc_element_f64: c_out needs a load (RHS or BACKSOLVE mode)");
  if (n1 < 3 || n1 > 11) {
    semk_set_error("semk_sc_element_f64: static condensation supports orders 2..10");
    return SEMK_ERR_UNSUPPORTED;
  }
  const int ne = 4 * (n1 - 1), ni = (n1 - 2) * (n1 - 2);
  if (mode & SEMK_SC_SCHUR)
    SEMK_REQUIRE(S_out && s_stride == (int64_t)ne * (ne + 1) / 2,
                 "semk_sc_element_f64: SCHUR needs S_out and the packed stride");
  if (mode & SEMK_SC_RHS)
    SEMK_REQUIRE(g_loc && JxW && l2g, "semk_sc_element_f64: RHS needs g_loc, JxW, l2g");
  if (mode & SEMK_SC_BACKSOLVE)
    SEMK_REQUIRE(u && JxW && l2g, "semk_sc_element_f64: BACKSOLVE needs u, JxW, l2g");
  if (mode & (SEMK_SC_SCHUR | SEMK_SC_STORE | SEMK_SC_STORE_INV)) {
    ScElemArgs a{};
    a.n_elem = n_elem;
    a.slot_of_elem = slot_of_elem;
    a.G = G;
    a.g_patch_stride = g_patch_stride;
    a.pe = elems_per_patch;
    a.D = D;
    a.ext_loc = ext_loc;
    a.mode = mode & (SEMK_SC_SCHUR | SEMK_SC_STORE | SEMK_SC_STORE_INV);
    a.S_out = S_out;
    a.s_stride = s_stride;
    a.sdiag_loc = sdiag_loc;
    a.W_out = W_out;
    a.react = react;
    a.Ainv_out = Ainv_out;
    a.bad_flag = bad_flag;
    const int rc = launch_sc_element(n1, a, stream);
    if (rc != SEMK_OK) return rc;
  }
  ScBlockArgs b{};
  b.n_elem = n_elem;
  b.slot_of_elem = slot_of_elem;
  b.G = G;
  b.g_patch_stride = g_patch_stride;
  b.pe = elems_per_patch;
  b.D = D;
  b.ext_loc = ext_loc;
  b.l2g = l2g;
  b.JxW = JxW;
  b.react = react;
  b.L = sc_single_load(f_nodal, f_scale);
  b.g_loc = g_loc;
  b.ldg = n_elem * ne;
  b.c_out = c_out;
  b.ldc = n_elem * ni;
  b.U = u;                          // one column: the row stride ldu is never used
  b.bad_flag = bad_flag;
  for (const int load_mode : {SEMK_SC_RHS, SEMK_SC_BACKSOLVE}) {
    if (!(mode & load_mode)) continue;
    b.mode = load_mode;
    const int rc = launch_sc_element_block(n1, b, stream);
    if (rc != SEMK_OK) return rc;
    b.c_out = nullptr;              // written by the first load pass
  }
  return SEMK_OK;
}

extern "C" int semk_sc_element_dense_f64(int n1, int64_t n_elem, const double *A_hier,
                                         const double *f_hier, const uint32_t *l2g_hier, int mode,
                                         double *S_out, int64_t s_stride, double *sdiag_loc,
                                         double *g_loc, double *u, int32_t *bad_flag,
                                         void *stream) {
  SEMK_REQUIRE(n_elem > 0 && A_hier && bad_flag, "semk_sc_element_dense_f64: bad argument");
  SEMK_REQUIRE(mode != 0 && (mode & ~7) == 0, "semk_sc_element_dense_f64: bad mode");
  if (n1 < 3 || n1 > 11) {
    semk_set_error("semk_sc_element_dense_f64: static condensation supports orders 2..10");
    return SEMK_ERR_UNSUPPORTED;
  }
  const int ne = 4 * (n1 - 1);
  if (mode & SEMK_SC_SCHUR)
    SEMK_REQUIRE(S_out && s_stride == (int64_t)ne * (ne + 1) / 2,
                 "semk_sc_element_dense_f64: SCHUR needs S_out and the packed stride");
  if (mode & SEMK_SC_RHS)
    SEMK_REQUIRE(g_loc && f_hier, "semk_sc_element_dense_f64: RHS needs g_loc and f_hier");
  if (mode & SEMK_SC_BACKSOLVE)
    SEMK_REQUIRE(u && f_hier && l2g_hier,
                 "semk_sc_element_dense_f64: BACKSOLVE needs u, f_hier, l2g_hier");
  ScElemArgs a{};
  a.n_elem = n_elem;
  a.pe = 1;
  a.mode = mode;
  a.S_out = S_out;
  a.s_stride = s_stride;
  a.sdiag_loc = sdiag_loc;
  a.bad_flag = bad_flag;
  a.g_loc = g_loc;
  a.u = u;
  a.A_dense = A_hier;
  a.f_dense = f_hier;
  a.l2g_hier = l2g_hier;
  return launch_sc_element(n1, a, stream);
}

static int launch_sc_element(int n1, const ScElemArgs &a, void *stream) {
  const int64_t n_elem = a.n_elem;
  cudaStream_t st = semk_stream(stream);
  const unsigned grid = (unsigned)(n_elem < 148 * 16 ? n_elem : 148 * 16);
#define SEMK_CALL(NV)                                                                      \
  do {                                                                                     \
    SEMK_CUDA_CHECK(cudaFuncSetAttribute(sc_element_kernel<NV>,                       \
                                         cudaFuncAttributeMaxDynamicSharedMemorySize,      \
                                         (int)ScCfg<NV>::kSmem));                          \
    sc_element_kernel<NV><<<grid, kScThreads, ScCfg<NV>::kSmem, st>>>(a);             \
  } while (0)
  SEMK_DISPATCH_SC(n1, SEMK_CALL)
#undef SEMK_CALL
  SEMK_LAUNCH_CHECK("sc_element_kernel");
  return SEMK_OK;
}

static int launch_sc_element_block(int n1, const ScBlockArgs &a, void *stream) {
  const int64_t n_elem = a.n_elem;
  cudaStream_t st = semk_stream(stream);
  const unsigned grid = (unsigned)(n_elem < 148 * 16 ? n_elem : 148 * 16);
#define SEMK_CALL(NV)                                                                      \
  do {                                                                                     \
    const size_t smem = sc_block_smem<NV>(a.L.k, a.mode);                                  \
    SEMK_CUDA_CHECK(cudaFuncSetAttribute(sc_element_block_kernel<NV>,                      \
                                         cudaFuncAttributeMaxDynamicSharedMemorySize,      \
                                         (int)sc_block_smem<NV>(kScBlockMaxCols,           \
                                                                SEMK_SC_BACKSOLVE)));      \
    sc_element_block_kernel<NV><<<grid, kScThreads, smem, st>>>(a);                        \
  } while (0)
  SEMK_DISPATCH_SC(n1, SEMK_CALL)
#undef SEMK_CALL
  SEMK_LAUNCH_CHECK("sc_element_block_kernel");
  return SEMK_OK;
}

extern "C" int semk_sc_backsolve_stored_f64(int n1, int64_t n_elem, const double *W,
                                           const double *c, const uint32_t *l2g,
                                           const int32_t *ext_loc, double *u, void *stream) {
  SEMK_REQUIRE(n_elem > 0 && W && l2g && ext_loc && u, "semk_sc_backsolve_stored_f64: bad argument");
  const int64_t ldc = n_elem * (n1 - 2) * (n1 - 2);
  cudaStream_t st = semk_stream(stream);
  int rc = SEMK_OK;
#define SEMK_CALL(NV) \
  rc = launch_backsolve_stored_block_tiled<NV>(n_elem, W, c, ldc, l2g, ext_loc, 1, u, 0, st)
  SEMK_DISPATCH_SC(n1, SEMK_CALL)
#undef SEMK_CALL
  if (rc != SEMK_OK) return rc;
  SEMK_LAUNCH_CHECK("sc_backsolve_stored_block_kernel");
  return SEMK_OK;
}

extern "C" int semk_sc_load_stored_f64(int n1, int64_t n_elem, const double *W, const double *Ainv,
                                       const uint32_t *l2g, const int32_t *ext_loc,
                                       const double *JxW, const double *f_nodal, double f_scale,
                                       double *g_loc, double *c_out, void *stream) {
  SEMK_REQUIRE(n_elem > 0 && W && Ainv && l2g && ext_loc && JxW && g_loc && c_out,
               "semk_sc_load_stored_f64: bad argument");
  const ScBlockLoad L = sc_single_load(f_nodal, f_scale);
  const int64_t ldg = n_elem * 4 * (n1 - 1), ldc = n_elem * (n1 - 2) * (n1 - 2);
  cudaStream_t st = semk_stream(stream);
  int rc = SEMK_OK;
#define SEMK_CALL(NV)                                                                          \
  rc = launch_load_stored_block_tiled<NV>(n_elem, W, Ainv, l2g, ext_loc, JxW, L, g_loc, ldg, \
                                          c_out, ldc, st)
  SEMK_DISPATCH_SC(n1, SEMK_CALL)
#undef SEMK_CALL
  if (rc != SEMK_OK) return rc;
  SEMK_LAUNCH_CHECK("sc_load_stored_block_kernel");
  return SEMK_OK;
}

extern "C" int semk_sc_block_max_cols(int n1) {
  return (n1 >= 3 && n1 <= 11) ? kScBlockMaxCols : -1;
}

// common checks of the block entries; fills the load descriptor
static int sc_block_load_args(const char *who, int n1, int k, const double *F, int64_t ldf,
                              uint32_t nodal_mask, const double *f_scale, ScBlockLoad *L) {
  if (n1 < 3 || n1 > 11) {
    semk_set_error(std::string(who) + ": static condensation supports orders 2..10");
    return SEMK_ERR_UNSUPPORTED;
  }
  if (k > kScBlockMaxCols) {
    semk_set_error(std::string(who) + ": more load columns than semk_sc_block_max_cols");
    return SEMK_ERR_UNSUPPORTED;
  }
  SEMK_REQUIRE(k >= 1, (std::string(who) + ": k must be >= 1").c_str());
  SEMK_REQUIRE(f_scale, (std::string(who) + ": f_scale must not be NULL").c_str());
  const uint32_t cols = k == 32 ? 0xFFFFFFFFu : ((1u << k) - 1u);
  SEMK_REQUIRE((nodal_mask & ~cols) == 0 && (!nodal_mask || (F && ldf > 0)),
               (std::string(who) + ": nodal columns need F and ldf > 0").c_str());
  L->k = k;
  L->F = F;
  L->ldf = ldf;
  L->nodal_mask = nodal_mask;
  for (int j = 0; j < kScBlockMaxCols; ++j) L->f_scale[j] = j < k ? f_scale[j] : 0.0;
  return SEMK_OK;
}

extern "C" int semk_sc_element_block_f64(int n1, int64_t n_elem, const double *G,
                                         int64_t g_patch_stride, int elems_per_patch,
                                         const double *D, const int32_t *ext_loc,
                                         const uint32_t *l2g, const double *JxW,
                                         const double *react, int mode, int k, const double *F,
                                         int64_t ldf, uint32_t nodal_mask, const double *f_scale,
                                         double *g_loc, int64_t ldg, double *c_out, int64_t ldc,
                                         double *U, int64_t ldu, int32_t *bad_flag,
                                         void *stream) {
  ScBlockArgs a{};
  int rc = sc_block_load_args("semk_sc_element_block_f64", n1, k, F, ldf, nodal_mask, f_scale,
                              &a.L);
  if (rc != SEMK_OK) return rc;
  SEMK_REQUIRE(n_elem > 0 && G && D && ext_loc && l2g && JxW && bad_flag && elems_per_patch > 0 &&
                   g_patch_stride > 0,
               "semk_sc_element_block_f64: bad argument");
  SEMK_REQUIRE(mode == SEMK_SC_RHS || mode == SEMK_SC_BACKSOLVE,
               "semk_sc_element_block_f64: mode must be SEMK_SC_RHS or SEMK_SC_BACKSOLVE");
  const int ne = 4 * (n1 - 1), ni = (n1 - 2) * (n1 - 2);
  if (mode == SEMK_SC_RHS)
    SEMK_REQUIRE(g_loc && ldg >= n_elem * ne,
                 "semk_sc_element_block_f64: RHS needs g_loc [k][ldg >= n_elem * 4p]");
  else
    SEMK_REQUIRE(U && ldu > 0, "semk_sc_element_block_f64: BACKSOLVE needs U [k][ldu > 0]");
  SEMK_REQUIRE(!c_out || ldc >= n_elem * ni,
               "semk_sc_element_block_f64: c_out needs ldc >= n_elem * (p-1)^2");
  a.n_elem = n_elem;
  a.G = G;
  a.g_patch_stride = g_patch_stride;
  a.pe = elems_per_patch;
  a.D = D;
  a.ext_loc = ext_loc;
  a.l2g = l2g;
  a.JxW = JxW;
  a.react = react;
  a.mode = mode;
  a.g_loc = g_loc;
  a.ldg = ldg;
  a.c_out = c_out;
  a.ldc = ldc;
  a.U = U;
  a.ldu = ldu;
  a.bad_flag = bad_flag;
  return launch_sc_element_block(n1, a, stream);
}

extern "C" int semk_sc_load_stored_block_f64(int n1, int64_t n_elem, const double *W,
                                             const double *Ainv, const uint32_t *l2g,
                                             const int32_t *ext_loc, const double *JxW, int k,
                                             const double *F, int64_t ldf, uint32_t nodal_mask,
                                             const double *f_scale, double *g_loc, int64_t ldg,
                                             double *c_out, int64_t ldc, void *stream) {
  ScBlockLoad L;
  int rc = sc_block_load_args("semk_sc_load_stored_block_f64", n1, k, F, ldf, nodal_mask,
                              f_scale, &L);
  if (rc != SEMK_OK) return rc;
  const int ne = 4 * (n1 - 1), ni = (n1 - 2) * (n1 - 2);
  SEMK_REQUIRE(n_elem > 0 && W && Ainv && l2g && ext_loc && JxW && g_loc && c_out &&
                   ldg >= n_elem * ne && ldc >= n_elem * ni,
               "semk_sc_load_stored_block_f64: bad argument");
  cudaStream_t st = semk_stream(stream);
#define SEMK_CALL(NV)                                                                      \
  rc = launch_load_stored_block_tiled<NV>(n_elem, W, Ainv, l2g, ext_loc, JxW, L, g_loc, ldg, \
                                          c_out, ldc, st)
  SEMK_DISPATCH_SC(n1, SEMK_CALL)
#undef SEMK_CALL
  if (rc != SEMK_OK) return rc;
  SEMK_LAUNCH_CHECK("sc_load_stored_block_kernel");
  return SEMK_OK;
}

extern "C" int semk_sc_backsolve_stored_block_f64(int n1, int64_t n_elem, const double *W,
                                                  const double *c, int64_t ldc,
                                                  const uint32_t *l2g, const int32_t *ext_loc,
                                                  int k, double *U, int64_t ldu, void *stream) {
  const char *who = "semk_sc_backsolve_stored_block_f64";
  if (n1 < 3 || n1 > 11) {
    semk_set_error(std::string(who) + ": static condensation supports orders 2..10");
    return SEMK_ERR_UNSUPPORTED;
  }
  if (k > kScBlockMaxCols) {
    semk_set_error(std::string(who) + ": more columns than semk_sc_block_max_cols");
    return SEMK_ERR_UNSUPPORTED;
  }
  const int ni = (n1 - 2) * (n1 - 2);
  SEMK_REQUIRE(k >= 1 && n_elem > 0 && W && l2g && ext_loc && U && ldu > 0 &&
                   (!c || ldc >= n_elem * ni),
               "semk_sc_backsolve_stored_block_f64: bad argument");
  cudaStream_t st = semk_stream(stream);
#define SEMK_CALL(NV) \
  rc = launch_backsolve_stored_block_tiled<NV>(n_elem, W, c, ldc, l2g, ext_loc, k, U, ldu, st)
  int rc = SEMK_OK;
  SEMK_DISPATCH_SC(n1, SEMK_CALL)
#undef SEMK_CALL
  if (rc != SEMK_OK) return rc;
  SEMK_LAUNCH_CHECK("sc_backsolve_stored_block_kernel");
  return SEMK_OK;
}

extern "C" int semk_sc_apply_f64(const semk_sc_op *op, const double *u, double *y, int flags,
                                 double *dot_out, void *stream) {
  int rc = check_sc_op(op, "semk_sc_apply_f64");
  if (rc != SEMK_OK) return rc;
  SEMK_REQUIRE(u && y && u != y, "semk_sc_apply_f64: null / aliased vectors");
  SEMK_REQUIRE(!dot_out || op->partials, "semk_sc_apply_f64: dot_out needs op->partials");
  cudaStream_t st = semk_stream(stream);
  const uint8_t *mask_in = (op->dirichlet && (flags & SEMK_MASK_IN)) ? op->dirichlet : nullptr;
  int n_sm = 148;
  {
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess)
      (void)cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
  }
#define SEMK_CALL(NV)                                                                      \
  do {                                                                                     \
    const int64_t groups = (op->n_elem + ScCfg<NV>::EPB - 1) / ScCfg<NV>::EPB;             \
    {                                                                                      \
      int per_sm = 0;                                                                      \
      SEMK_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(                       \
          &per_sm, sc_matvec_kernel<NV>, kScThreads, sc_matvec_smem<NV>()));       \
      if (per_sm < 1) per_sm = 1;                                                          \
      const int64_t cap = (int64_t)n_sm * per_sm;                                          \
      const unsigned grid = (unsigned)(groups < cap ? groups : cap);                       \
      sc_matvec_kernel<NV><<<grid, kScThreads, sc_matvec_smem<NV>(), st>>>(         \
          op->n_elem, op->S, op->l2g_ext, u, mask_in, op->y_loc);                          \
    }                                                                                      \
  } while (0)
  SEMK_DISPATCH_SC(op->n1, SEMK_CALL)
#undef SEMK_CALL
  SEMK_LAUNCH_CHECK("sc_matvec_kernel");
  sc_node_kernel<<<node_blocks(op->n_ext), kNodeThreads, 0, st>>>(
      op->n_ext, op->node_ptr, op->node_pos, op->y_loc, op->dirichlet, u, y, flags, 0.0,
      op->partials, dot_out);
  SEMK_LAUNCH_CHECK("sc_node_kernel");
  return SEMK_OK;
}

extern "C" int semk_sc_assemble_f64(const semk_sc_op *op, const double *loc, double *out,
                                    int flags, double fill_dirichlet, void *stream) {
  int rc = check_sc_op(op, "semk_sc_assemble_f64");
  if (rc != SEMK_OK) return rc;
  SEMK_REQUIRE(loc && out, "semk_sc_assemble_f64: null pointer");
  sc_node_kernel<<<node_blocks(op->n_ext), kNodeThreads, 0, semk_stream(stream)>>>(
      op->n_ext, op->node_ptr, op->node_pos, loc, op->dirichlet, nullptr, out,
      flags & SEMK_MASK_OUT, fill_dirichlet, nullptr, nullptr);
  SEMK_LAUNCH_CHECK("sc_node_kernel");
  return SEMK_OK;
}

extern "C" int semk_face_sum_f64(int64_t n, const uint32_t *ptr, const uint32_t *pos,
                                 const double *vals, double *out, void *stream) {
  SEMK_REQUIRE(n > 0 && ptr && pos && vals && out, "semk_face_sum_f64: bad argument");
  sc_node_kernel<<<node_blocks(n), kNodeThreads, 0, semk_stream(stream)>>>(
      n, ptr, pos, vals, nullptr, nullptr, out, 0, 0.0, nullptr, nullptr);
  SEMK_LAUNCH_CHECK("sc_node_kernel");
  return SEMK_OK;
}

extern "C" int semk_sc_coarse_elem_f64(const semk_sc_op *op, const double *phi, double *Ace_out,
                                       void *stream) {
  int rc = check_sc_op(op, "semk_sc_coarse_elem_f64");
  if (rc != SEMK_OK) return rc;
  SEMK_REQUIRE(phi && Ace_out, "semk_sc_coarse_elem_f64: null pointer");
  cudaStream_t st = semk_stream(stream);
#define SEMK_CALL(NV)                                                                      \
  do {                                                                                     \
    const int64_t groups = (op->n_elem + ScCfg<NV>::EPB - 1) / ScCfg<NV>::EPB;             \
    const unsigned grid = (unsigned)(groups < 148 * 8 ? groups : 148 * 8);                 \
    sc_coarse_elem_kernel<NV><<<grid, kScThreads, sc_coarse_elem_smem<NV>(), st>>>(        \
        op->n_elem, op->S, op->l2g_ext, op->dirichlet, phi, Ace_out);                      \
  } while (0)
  SEMK_DISPATCH_SC(op->n1, SEMK_CALL)
#undef SEMK_CALL
  SEMK_LAUNCH_CHECK("sc_coarse_elem_kernel");
  return SEMK_OK;
}

static int check_coarse(int64_t n_elem, const semk_sc_coarse *cs, const char *who) {
  if (!cs || n_elem <= 0 || cs->n_v <= 0 || !cs->Ace || !cs->vert_c || !cs->y_loc_c || !cs->vptr ||
      !cs->vpos) {
    semk_set_error(std::string(who) + ": inconsistent semk_sc_coarse");
    return SEMK_ERR_INVALID;
  }
  return SEMK_OK;
}

extern "C" int semk_sc_coarse_apply_f64(int64_t n_elem, const semk_sc_coarse *cs, const double *x,
                                        double *y, int flags, double *dot_out, void *stream) {
  int rc = check_coarse(n_elem, cs, "semk_sc_coarse_apply_f64");
  if (rc != SEMK_OK) return rc;
  SEMK_REQUIRE(x && y && x != y, "semk_sc_coarse_apply_f64: null / aliased vectors");
  SEMK_REQUIRE(!dot_out || cs->partials, "semk_sc_coarse_apply_f64: dot_out needs partials");
  cudaStream_t st = semk_stream(stream);
  const int64_t want = (n_elem * 4 + 255) / 256;
  const unsigned grid = (unsigned)(want < 148 * 8 ? want : 148 * 8);
  sc_coarse_matvec_kernel<<<grid, 256, 0, st>>>(n_elem, cs->Ace, cs->vert_c, x, cs->y_loc_c);
  SEMK_LAUNCH_CHECK("sc_coarse_matvec_kernel");
  sc_node_kernel<<<node_blocks(cs->n_v), kNodeThreads, 0, st>>>(
      cs->n_v, cs->vptr, cs->vpos, cs->y_loc_c, cs->dirichlet_c, x, y, flags, 0.0, cs->partials,
      dot_out);
  SEMK_LAUNCH_CHECK("sc_node_kernel");
  return SEMK_OK;
}

extern "C" int semk_sc_coarse_assemble_f64(int64_t n_elem, const semk_sc_coarse *cs,
                                           const double *loc, double *out, void *stream) {
  int rc = check_coarse(n_elem, cs, "semk_sc_coarse_assemble_f64");
  if (rc != SEMK_OK) return rc;
  SEMK_REQUIRE(loc && out, "semk_sc_coarse_assemble_f64: null pointer");
  sc_node_kernel<<<node_blocks(cs->n_v), kNodeThreads, 0, semk_stream(stream)>>>(
      cs->n_v, cs->vptr, cs->vpos, loc, nullptr, nullptr, out, 0, 0.0, nullptr, nullptr);
  SEMK_LAUNCH_CHECK("sc_node_kernel");
  return SEMK_OK;
}
