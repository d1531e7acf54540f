// semk_elem.cuh -- element-level building blocks shared by the patch kernels
// (semk_apply.cu: Poisson; semk_stokes.cu: axisymmetric Stokes): the differentiation
// matrix as a kernel parameter, its even-odd factorisation and the conflict-free
// transpose-scratch stride.
#pragma once
#include "semk_common.cuh"

#include <cmath>
#include <cstring>

namespace {

// Differentiation matrix, passed BY VALUE as a kernel parameter: the entries
// live in the parameter constant bank and every use below has a compile-time
// index, so the DFMAs read them through uniform registers (LDCU.128) -- no
// shared memory, no per-thread registers.
//
// `v` is the plain row-major matrix (used by the atomic cross-check kernel).
// `eo[0]` / `eo[1]` hold the even-odd factorisation of D and of D^T used by
// the production kernel: a GLL differentiation matrix is centro-antisymmetric
// (D[N-1-i][N-1-k] = -D[i][k]), so with e_k = v_k + v_{N-1-k},
// o_k = v_k - v_{N-1-k} (k < h = N/2) and the centre value v_c (odd N)
//     S_i = sum_k M[i][k] o_k,   A_i = sum_k P[i][k] e_k + C[i] v_c,
//     out_i = S_i + A_i,  out_{N-1-i} = S_i - A_i,
//     out_c = sum_k R[k] o_k + Dcc v_c
// with M = (D[i][k] - D[i][N-1-k])/2, P = (D[i][k] + D[i][N-1-k])/2,
// C[i] = D[i][c], R[k] = D[c][k]: 2h^2 + 2h FMAs + 4h adds instead of N^2
// FMAs (56 instead of 81 FP64 instructions at N = 9).
constexpr int kMaxH = SEMK_MAX_N1 / 2;
struct EvenOdd {
  double P[kMaxH * kMaxH], M[kMaxH * kMaxH], C[kMaxH], R[kMaxH], Dcc;
};
struct DMat {
  double v[SEMK_MAX_N1 * SEMK_MAX_N1];
};
struct DMatEO {
  EvenOdd eo[2];  // [0]: D, [1]: D^T
};

DMat make_dmat(int n1, const double *D_host) {
  DMat d;
  std::memset(&d, 0, sizeof(d));
  std::memcpy(d.v, D_host, sizeof(double) * n1 * n1);
  return d;
}

// Returns false if D is not centro-antisymmetric to 1e-12 (relative).
bool make_dmat_eo(int n1, const double *D, DMatEO *out) {
  std::memset(out, 0, sizeof(*out));
  const int N = n1, h = N / 2, c = (N & 1) ? h : -1;
  double dmax = 0.0, viol = 0.0;
  for (int i = 0; i < N; ++i)
    for (int k = 0; k < N; ++k) {
      const double a = D[i * N + k], b = D[(N - 1 - i) * N + (N - 1 - k)];
      dmax = std::fmax(dmax, std::fabs(a));
      viol = std::fmax(viol, std::fabs(a + b));
    }
  if (!(viol <= 1e-12 * dmax)) return false;
  for (int tr = 0; tr < 2; ++tr) {
    EvenOdd &E = out->eo[tr];
    auto d = [&](int i, int k) { return tr ? D[k * N + i] : D[i * N + k]; };
    for (int i = 0; i < h; ++i) {
      for (int k = 0; k < h; ++k) {
        E.M[i * h + k] = 0.5 * (d(i, k) - d(i, N - 1 - k));
        E.P[i * h + k] = 0.5 * (d(i, k) + d(i, N - 1 - k));
      }
      if (c >= 0) {
        E.C[i] = d(i, c);
        E.R[i] = d(c, i);
      }
    }
    if (c >= 0) E.Dcc = d(c, c);
  }
  return true;
}

// out[i] = sum_k D[i][k] v[k]      (derivative along the in-thread axis)
template <int N>
__device__ __forceinline__ void apply_D(const DMat &dm, const double (&v)[N], double (&out)[N]) {
#pragma unroll
  for (int i = 0; i < N; ++i) {
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < N; ++k) acc = fma(dm.v[i * N + k], v[k], acc);
    out[i] = acc;
  }
}
// out[i] = sum_k D[k][i] v[k]      (transpose: the weak-form "test" side)
template <int N>
__device__ __forceinline__ void apply_Dt(const DMat &dm, const double (&v)[N], double (&out)[N]) {
#pragma unroll
  for (int i = 0; i < N; ++i) {
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < N; ++k) acc = fma(dm.v[k * N + i], v[k], acc);
    out[i] = acc;
  }
}
// Even-odd application of D (TR = 0) or D^T (TR = 1).
template <int N, int TR>
__device__ __forceinline__ void apply_eo(const DMatEO &dm, const double (&v)[N],
                                         double (&out)[N]) {
  constexpr int h = N / 2;
  constexpr bool odd = (N & 1) != 0;
  const EvenOdd &E = dm.eo[TR];
  double e[h > 0 ? h : 1], o[h > 0 ? h : 1];
#pragma unroll
  for (int k = 0; k < h; ++k) {
    e[k] = v[k] + v[N - 1 - k];
    o[k] = v[k] - v[N - 1 - k];
  }
#pragma unroll
  for (int i = 0; i < h; ++i) {
    double S = 0.0, A = odd ? E.C[i] * v[h] : 0.0;
#pragma unroll
    for (int k = 0; k < h; ++k) {
      S = fma(E.M[i * h + k], o[k], S);
      A = fma(E.P[i * h + k], e[k], A);
    }
    out[i] = S + A;
    out[N - 1 - i] = S - A;
  }
  if (odd) {
    double acc = E.Dcc * v[h];
#pragma unroll
    for (int k = 0; k < h; ++k) acc = fma(E.R[k], o[k], acc);
    out[h] = acc;
  }
}

// Uniform front end: the production kernel passes DMatEO, the cross-check DMat.
template <int N>
__device__ __forceinline__ void mat_D(const DMat &dm, const double (&v)[N], double (&o)[N]) {
  apply_D<N>(dm, v, o);
}
template <int N>
__device__ __forceinline__ void mat_Dt(const DMat &dm, const double (&v)[N], double (&o)[N]) {
  apply_Dt<N>(dm, v, o);
}
template <int N>
__device__ __forceinline__ void mat_D(const DMatEO &dm, const double (&v)[N], double (&o)[N]) {
  apply_eo<N, 0>(dm, v, o);
}
template <int N>
__device__ __forceinline__ void mat_Dt(const DMatEO &dm, const double (&v)[N], double (&o)[N]) {
  apply_eo<N, 1>(dm, v, o);
}

// Row stride of the CTA-wide transpose scratch: N*PE columns (one per thread)
// padded so that RS == 1 (mod 16).  With 8-byte words and 16 bank pairs both
// access patterns of a half-warp are then conflict-free:
//   column pattern  A[m*RS + tidp]          -> bank = const + tidp
//   row pattern     A[t*RS + le*N + s]      -> bank = const + t + le*N = const + tidp
__host__ __device__ constexpr int scratch_row_stride(int N, int PE) {
  return ((N * PE - 1 + 15) & ~15) + 1;  // == semk_scratch_row_stride (include/semk.h)
}

enum { MODE_APPLY = 0, MODE_ASSEMBLE = 1 };


// Shared-memory carve-up of the persistent patch kernel (offsets multiples of
// 16 B): one G buffer, two stages of {node block, index block}, one copy of
// the working arrays.  `sep`: the separable kernel stages only the G00 and G11 slabs
// (2 NN PE doubles) instead of the whole patch block.
struct PatchSmem {
  size_t hdr, gs, stage0, stage_bytes, pn_off, el_off;  // per stage: node block | index block
  size_t inv, ua, bs, red, total;
};
__host__ __device__ inline PatchSmem patch_smem_layout(int N, int PE, int mode,
                                                       int64_t g_patch_stride,
                                                       int64_t pn_patch_stride,
                                                       int64_t eloc_patch_stride,
                                                       int64_t inv_patch_stride,
                                                       bool sep = false) {
  PatchSmem L;
  const size_t scratch = (size_t)N * scratch_row_stride(N, PE);
  size_t o = 32;  // four mbarriers: tables[2], G, inverse table
  L.hdr = o;      // two 32-byte patch headers (ring)
  o += 64;
  L.gs = o;
  const size_t g_doubles = sep ? 2 * (size_t)N * N * PE : (size_t)g_patch_stride;
  o += (mode == MODE_APPLY) ? sizeof(double) * g_doubles : 0;
  L.stage0 = o;
  L.pn_off = 0;
  size_t st = 4 * (size_t)pn_patch_stride;
  L.el_off = st;
  st += 2 * (size_t)eloc_patch_stride;
  st = (st + 15) & ~(size_t)15;
  L.stage_bytes = st;
  o += 2 * st;
  L.inv = o;  // inverse table of the patch being written out (single buffer)
  o += 2 * (size_t)inv_patch_stride;
  o = (o + 15) & ~(size_t)15;
  L.ua = o;  // scratch A
  o += (mode == MODE_APPLY) ? 8 * scratch : 0;
  o = (o + 15) & ~(size_t)15;
  L.bs = o;  // scratch B: the element results the write-out gathers from; its head doubles
             // as the block-reduction scratch at the very end
  o += 8 * scratch > 256 ? 8 * scratch : 256;
  L.red = L.bs;
  L.total = o;
  return L;
}


}  // namespace

// semk_ho.cu: the column / row thread-pair variant of the apply kernel (high orders)
int semk_ho_launch(const semk_op &op, const double *u, double *y, int flags, double *partials,
                   cudaStream_t st, int *grid_out, int64_t pb, int64_t pe);
int64_t semk_ho_resident(int n1, int elems_per_patch, size_t smem);
// semk_box.cu: the BOX instantiations of the patch kernel (regular structured numberings);
// dm_eo points at the caller's DMatEO; op.separable picks the separable instantiation
int semk_box_launch(const semk_op &op, const void *dm_eo, const double *u, double *y, int flags,
                    double *partials, cudaStream_t st, int *grid_out, int64_t pb, int64_t pe);
int64_t semk_box_resident(int n1, int elems_per_patch, bool sep, size_t smem);
