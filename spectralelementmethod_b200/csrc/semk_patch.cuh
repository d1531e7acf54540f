// semk_patch.cuh -- the persistent, software-pipelined patch kernel (K2 / K3) and its
// launcher, shared by semk_apply.cu (table-driven gather, any numbering) and semk_box.cu
// (the BOX instantiations: arithmetic gather for regularly numbered structured meshes).
// See semk_apply.cu for the reference lines the kernel replaces.
#pragma once
#include "semk_common.cuh"

#include <cmath>
#include <cstring>

#include "semk_elem.cuh"

namespace {

// The element-local operator for one column-owning thread.
//   tidp = le*N + t identifies (element-in-CTA, column);  ucol[m] = u[m][t] on
//   entry, ycol[m] = y[m][t] on exit.
//   A, B: CTA-wide scratch, N rows of RS doubles.
//   g: this thread's column base inside the patch's G block; the factor
//      (c, m) of this column sits at g[(c*N + m) * g_row].
//   g_ready: mbarrier guarding a TMA-staged G (nullptr when g is global).
// Contains four __syncthreads(); every thread of the CTA must call it.
struct NoHook {
  __device__ __forceinline__ void operator()() const {}
};

template <int N, int RS, class DM, class Hook = NoHook, class Hook0 = NoHook>
__device__ __forceinline__ void local_poisson(const DM &dm, int le, int t, bool active,
                                              const double (&ucol)[N], double (&ycol)[N],
                                              double *__restrict__ A, double *__restrict__ B,
                                              const double *__restrict__ g, int g_row,
                                              uint64_t *g_ready, uint32_t g_parity = 0,
                                              Hook g_consumed = Hook(),
                                              Hook0 after_first_barrier = Hook0()) {
  const int tidp = le * N + t;
  double ur[N], tmp[N], us[N];
  if (active) {
#pragma unroll
    for (int m = 0; m < N; ++m) A[m * RS + tidp] = ucol[m];
  }
  __syncthreads();
  after_first_barrier();  // every thread has left the previous patch's write-out
  if (active) {
    mat_D<N>(dm, ucol, ur);  // ur[m][t] = sum_r D[m][r] u[r][t]
#pragma unroll
    for (int s = 0; s < N; ++s) tmp[s] = A[t * RS + le * N + s];  // row t of u
    mat_D<N>(dm, tmp, us);                                        // us[t][n] = sum_s D[n][s] u[t][s]
#pragma unroll
    for (int n = 0; n < N; ++n) B[t * RS + le * N + n] = us[n];
  }
  __syncthreads();
  // G staged by TMA: every thread observes the mbarrier phase itself (acquire)
  if (g_ready) semk_mbar_wait(g_ready, g_parity);
  double w1[N];
  if (active) {
#pragma unroll
    for (int m = 0; m < N; ++m) {
      const double usc = B[m * RS + tidp];  // us[m][t]
      const double g00 = g[m * g_row], g01 = g[(N + m) * g_row], g11 = g[(2 * N + m) * g_row];
      tmp[m] = g00 * ur[m] + g01 * usc;  // w0[m][t]
      w1[m] = g01 * ur[m] + g11 * usc;   // w1[m][t]
    }
    mat_Dt<N>(dm, tmp, ycol);  // y0[p][t] = sum_m D[m][p] w0[m][t]
#pragma unroll
    for (int m = 0; m < N; ++m) A[m * RS + tidp] = w1[m];
  }
  __syncthreads();
  g_consumed();  // every thread has read its G entries: the G buffer may be refilled
  if (active) {
#pragma unroll
    for (int n = 0; n < N; ++n) tmp[n] = A[t * RS + le * N + n];  // row t of w1
    mat_Dt<N>(dm, tmp, us);                                       // y1[t][q] = sum_n w1[t][n] D[n][q]
#pragma unroll
    for (int q = 0; q < N; ++q) B[t * RS + le * N + q] = us[q];
  }
  __syncthreads();
  if (active) {
#pragma unroll
    for (int m = 0; m < N; ++m) ycol[m] += B[m * RS + tidp];
  }
}

// The separable element operator of an axis-aligned element (G01 == 0):
//   y = D^T (G00 . D u)  +  (G11 . u D^T) D  =  y0 + y1.
// The column-owning thread tidp = le*N + t forms y0 of its column in registers; thread
// `tid` also owns row t' = tid / PE of slot le' = tid % PE and forms y1 of that row in
// registers.  Only u crosses from the column to the row layout (scratch A) and only y1
// crosses back (scratch B): two shared-memory round trips instead of four, two barriers
// instead of four.  Every product and sum is the one local_poisson forms when its G01
// entries are +-0, so the two routines give the same bits on the same G: there w0 =
// fl(G00 ur + G01 us) = fl(G00 ur), here the product is rounded on its own (__dmul_rn, so
// that the compiler cannot fuse it into the even-odd sums of mat_Dt as an FMA).
//   g0: this thread's column base in the G00 slab, factor m at g0[m * g_row];
//   g1: the G11 slab; row thread tid reads node (t', n) of slot le' at g1[tid * N + n]
//       (with N odd, consecutive threads hit distinct banks).
//   row_active: slot le' of row thread tid holds an element (false for tid >= N * PE).
// On return ycol = y0 + y1 = fl(y0 + y1) as in local_poisson; scratch B still holds y1 at
// node positions m*RS + tidp, which the caller may overwrite in place (own entries).
// Contains two __syncthreads(); every thread of the CTA must call it.
template <int N, int PE, int RS, class DM, class Hook = NoHook, class Hook0 = NoHook>
__device__ __forceinline__ void local_poisson_sep(const DM &dm, int le, int t, int tid,
                                                  bool active, bool row_active,
                                                  const double (&ucol)[N], double (&ycol)[N],
                                                  double *__restrict__ A, double *__restrict__ B,
                                                  const double *__restrict__ g0, int g_row,
                                                  const double *__restrict__ g1,
                                                  uint64_t *g_ready, uint32_t g_parity = 0,
                                                  Hook g_consumed = Hook(),
                                                  Hook0 after_first_barrier = Hook0()) {
  const int tidp = le * N + t;
  if (active) {
#pragma unroll
    for (int m = 0; m < N; ++m) A[m * RS + tidp] = ucol[m];
  }
  __syncthreads();
  after_first_barrier();  // every thread has left the previous patch's write-out
  if (g_ready) semk_mbar_wait(g_ready, g_parity);
  if (row_active) {
    const int ler = tid % PE, tr = tid / PE;
    double ur[N], w[N];
#pragma unroll
    for (int s = 0; s < N; ++s) ur[s] = A[tr * RS + ler * N + s];  // row t' of u
    mat_D<N>(dm, ur, w);  // us[t'][n] = sum_s D[n][s] u[t'][s]
#pragma unroll
    for (int n = 0; n < N; ++n) w[n] = __dmul_rn(g1[tid * N + n], w[n]);  // w1[t'][n]
    mat_Dt<N>(dm, w, ur);  // y1[t'][q] = sum_n w1[t'][n] D[n][q]
#pragma unroll
    for (int q = 0; q < N; ++q) B[tr * RS + ler * N + q] = ur[q];
  }
  if (active) {
    double w[N];
    mat_D<N>(dm, ucol, w);  // ur[m][t] = sum_r D[m][r] u[r][t]
#pragma unroll
    for (int m = 0; m < N; ++m) w[m] = __dmul_rn(g0[m * g_row], w[m]);  // w0[m][t]
    mat_Dt<N>(dm, w, ycol);  // y0[p][t] = sum_m D[m][p] w0[m][t]
  }
  __syncthreads();
  g_consumed();  // every thread has read its G entries: the G buffer may be refilled
  if (active) {
#pragma unroll
    for (int m = 0; m < N; ++m) ycol[m] += B[m * RS + tidp];
  }
}

template <int N, int PE>
struct PatchCfg {
  static constexpr int kThreads = ((N * PE + 31) / 32) * 32;
  static constexpr int kRS = scratch_row_stride(N, PE);
};

// Resident CTAs per SM the kernel is compiled for (register budget): what the
// shared-memory footprint of the standard tiles (2x8, 1x8, 1x4 elements) allows.
// `g_slabs`: G slabs staged per patch (3, or 2 for the separable kernel).
__host__ __device__ constexpr int patch_min_blocks(int N, int PE, int g_slabs = 3) {
  const int bx = PE == 32 ? 4 : (PE == 16 ? 2 : 1), by = PE == 4 ? 4 : 8, p = N - 1;
  const long long mpn = (long long)(bx * p + 1) * (by * p + 1);
  const long long mpn4 = (mpn + 3) & ~3LL;
  const long long nn = (long long)N * N;
  const long long g = 8 * ((g_slabs * nn * PE + 1) & ~1LL);
  const long long tab = 2 * ((4 * mpn4 + 2 * ((nn * PE + 7) & ~7LL) + 15) & ~15LL) + 64;
  const long long scr = 8LL * N * scratch_row_stride(N, PE);
  const long long ua = scr;
  const long long total = 32 + g + tab + 8 * mpn4 + ua + (scr > 256 ? scr : 256) + 1024;
  const long long by_smem = 233472 / total;
  const int threads = ((N * PE + 31) / 32) * 32;
  const long long by_regs = 65536 / ((long long)threads * 96);  // assume <= 96 registers/thread
  long long r = by_smem < by_regs ? by_smem : by_regs;
  return r < 1 ? 1 : (r > 8 ? 8 : (int)r);
}

constexpr int kGatherBatch = 8;

// Persistent, software-pipelined patch kernel.
//
// Each CTA loops over patches blockIdx.x, blockIdx.x + gridDim.x, ...  While it
// works on patch i, the TMA engine is already filling the other pipeline stage
// with patch i+1's geometric factors, node block and index block (issued one
// whole patch-time ahead: DRAM latency is off the critical path), and the
// nodal values of patch i+1 are gathered into registers right after the
// element operator of patch i, so that the loads are in flight during the
// assembly and the write-out.  CTAs never exit between patches,
// so no SM slot idles on CTA launch / retire (~2.4 k cycles each on this chip).
//
// MODE_APPLY:    y = A u (masked per flags), optional dot partials.
// MODE_ASSEMBLE: y = assembly of the element-local field `loc` (slot order).
//
// BOX (apply only): regularly numbered structured meshes (semk_op.box_ld > 0).  A patch
// whose header word 3 is non-zero is a full tile box: node (m, t) of its slot
// le = lx * by + ly has the global id  base + (lx * p + m) * box_ld + ly * p + t, it holds no
// Dirichlet node, and word 3 is the mask of its non-empty slots.  Such a patch needs no
// index tables for its gather: the 2 N shared-memory look-ups per thread (index block,
// node block) are replaced by address arithmetic -- same loads, same order, bit-identical
// results, 1.5 - 2.5 % faster at p = 6 .. 12 (profiles/r02_box_ab.txt).  Patches with
// word 3 == 0 (Dirichlet nodes, anything irregular) take the table-driven gather inside
// the same kernel; the write-out always uses the tables.
// Measured and dropped (same file): copying the column with 8-byte cp.async straight into
// the scratch (LDGSTS; no gain, 0.675 vs 0.671 ms at p = 8) and an arithmetic write-out of
// the tile-interior nodes (the index arithmetic costs more issue slots than the two table
// look-ups per node it saves: 0.775 ms); not copying the (then unused) index block of a box
// patch into shared memory (0.694 vs 0.659 ms -- kept copying it).
//
// SEP (apply only; semk_op.separable): the G01 slab of every patch is zero.  The TMA stages
// only the G00 and G11 slabs and the element operator is local_poisson_sep: three barriers
// per patch instead of five, seven shared-memory passes of N doubles per thread instead of
// twelve, two thirds of the G bytes.  Same results, bit for bit, as the three-factor kernel
// on the same G (DESIGN.md section 3).
template <int N, int PE, int MODE, bool BOX = false, bool SEP = false>
__global__ void __launch_bounds__(PatchCfg<N, PE>::kThreads, patch_min_blocks(N, PE, SEP ? 2 : 3))
    patch_kernel(semk_op op, DMatEO dm, const double *__restrict__ u,
                 const double *__restrict__ loc, double *__restrict__ y, int flags,
                 double fill_dirichlet, double *__restrict__ dot_partials, int64_t patch_begin,
                 int64_t patch_end) {
  constexpr int NN = N * N;
  constexpr int NP = N * PE;
  constexpr int kThreads = PatchCfg<N, PE>::kThreads;
  constexpr int RS = PatchCfg<N, PE>::kRS;
  static_assert(!SEP || MODE == MODE_APPLY, "the separable operator is an apply");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const PatchSmem L = patch_smem_layout(N, PE, MODE, op.g_patch_stride, op.pn_patch_stride,
                                        op.eloc_patch_stride, op.inv_patch_stride, SEP);
  uint64_t *mbar = reinterpret_cast<uint64_t *>(smem_raw);  // [0..1]: tables, [2]: G, [3]: inv
  double *Gs = reinterpret_cast<double *>(smem_raw + L.gs);
  const uint16_t *inv_s = reinterpret_cast<const uint16_t *>(smem_raw + L.inv);
  double *As = reinterpret_cast<double *>(smem_raw + L.ua);
  double *Bs = reinterpret_cast<double *>(smem_raw + L.bs);
  double *red = reinterpret_cast<double *>(smem_raw + L.red);

  const int tid = threadIdx.x;
  const int le = tid / N, t = tid - le * N;
  const uint32_t pn_bytes = 4u * (uint32_t)op.pn_patch_stride;
  const uint32_t el_bytes = 2u * (uint32_t)op.eloc_patch_stride;
  const uint32_t g_bytes = (uint32_t)(op.g_patch_stride * sizeof(double));
  const uint32_t inv_bytes = 2u * (uint32_t)op.inv_patch_stride;
  const int inv_w4 = (int)(op.inv_width >> 2);  // 8-byte groups of inverse entries per node

  auto stage_ptr = [&](int s) { return smem_raw + L.stage0 + (size_t)s * L.stage_bytes; };
  // Patch headers travel two patches ahead through a 2-entry ring: the header of patch
  // i+1 names the (deduplicated) table blocks the copy for patch i+1 must fetch, so it
  // has to be in shared memory when that copy is issued, during patch i.
  uint32_t *hdr_ring = reinterpret_cast<uint32_t *>(smem_raw + L.hdr);
  // one thread: tables of `patch` (blocks pi, ei) into stage s, plus -- if it exists --
  // the header of the patch after it (`patch_after`) into ring entry `slot_after`
  auto issue_tables = [&](uint32_t pi, uint32_t ei, int s, int64_t patch_after, int slot_after) {
    unsigned char *base = stage_ptr(s);
    const bool more = patch_after >= 0;
    semk_mbar_expect_tx(&mbar[s], pn_bytes + el_bytes + (more ? 32u : 0u));
    semk_bulk_g2s(base + L.pn_off, op.pnode + (int64_t)pi * op.pn_patch_stride, pn_bytes, &mbar[s]);
    semk_bulk_g2s(base + L.el_off, op.eloc + (int64_t)ei * op.eloc_patch_stride, el_bytes, &mbar[s]);
    if (more) semk_bulk_g2s(hdr_ring + 8 * slot_after, op.patch_hdr + 8 * patch_after, 32u, &mbar[s]);
  };
  // The inverse table is single-buffered: patch i's table is fetched right after the
  // first barrier of patch i (when every thread has left patch i-1's write-out, its last
  // reader) and is first needed five barriers later (three with SEP), in patch i's own
  // write-out.
  auto issue_inv = [&](uint32_t block) {  // one thread
    semk_mbar_expect_tx(&mbar[3], inv_bytes);
    semk_bulk_g2s(smem_raw + L.inv, op.inv + (int64_t)block * op.inv_patch_stride, inv_bytes,
                  &mbar[3]);
  };
  auto issue_g = [&](int64_t patch) {  // one thread
    const double *src = op.G + patch * op.g_patch_stride;
    if (SEP) {  // slabs 0 (G00) and 2 (G11); the zero G01 slab stays in global memory
      constexpr uint32_t slab = (uint32_t)(NN * PE * sizeof(double));
      semk_mbar_expect_tx(&mbar[2], 2 * slab);
      semk_bulk_g2s(Gs, src, slab, &mbar[2]);
      semk_bulk_g2s(Gs + NN * PE, src + 2 * NN * PE, slab, &mbar[2]);
    } else {
      semk_mbar_expect_tx(&mbar[2], g_bytes);
      semk_bulk_g2s(Gs, src, g_bytes, &mbar[2]);
    }
  };

  // this CTA's patch sequence: round-robin over the grid, so that at any time the
  // resident CTAs work on a compact window of the mesh (DRAM page / L2 locality)
  const int64_t step = (int64_t)gridDim.x;
  const int64_t p_first = patch_begin + (int64_t)blockIdx.x;
  const int64_t p_end = patch_end;  // (a sub-range of the patches: staged host apply)
  if (tid == 0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) semk_mbar_init(&mbar[i], 1);
    semk_fence_mbar_init();
    if (p_first < p_end) {
      // the first header is read directly (block indices needed right now) and also
      // copied into ring entry 0; the second patch's header goes to entry 1
      const uint32_t pi = op.patch_hdr[8 * p_first + 5], ei = op.patch_hdr[8 * p_first + 6];
      const int64_t p2 = p_first + step;
      unsigned char *base = stage_ptr(0);
      semk_mbar_expect_tx(&mbar[0], pn_bytes + el_bytes + 32u + (p2 < p_end ? 32u : 0u));
      semk_bulk_g2s(base + L.pn_off, op.pnode + (int64_t)pi * op.pn_patch_stride, pn_bytes, &mbar[0]);
      semk_bulk_g2s(base + L.el_off, op.eloc + (int64_t)ei * op.eloc_patch_stride, el_bytes, &mbar[0]);
      semk_bulk_g2s(hdr_ring, op.patch_hdr + 8 * p_first, 32u, &mbar[0]);
      if (p2 < p_end) semk_bulk_g2s(hdr_ring + 8, op.patch_hdr + 8 * p2, 32u, &mbar[0]);
      if (MODE == MODE_APPLY) issue_g(p_first);
    }
  }
  __syncthreads();  // mbarrier initialisation visible to every waiter

  // This thread's column of nodal values for the patch about to be processed,
  // gathered straight from global memory through the staged tables (entries of
  // nodes shared by several elements of the patch hit L1) and carried in
  // registers across the loop: the gather for patch i+1 is issued right after
  // the element operator of patch i, so its latency hides behind the assembly
  // and write-out of patch i.
  double ucol[N];
  uint32_t ucol_dir = 0;  // bit m set: entry m of the staged column is a Dirichlet node
  auto gather_column = [&](int s_tab, int64_t patch_of) {
    const unsigned char *sbn = stage_ptr(s_tab);
    const uint32_t *pnb = reinterpret_cast<const uint32_t *>(sbn + L.pn_off);
    const uint32_t id0 = hdr_ring[8 * s_tab + 4];  // ring entry = iteration parity = stage
    const uint16_t *elb = reinterpret_cast<const uint16_t *>(sbn + L.el_off);
    const bool act = (le < PE) && (patch_of * PE + le < op.n_elem);
    if (BOX && hdr_ring[8 * s_tab + 3] != 0u) {
      // regular box: addresses by arithmetic, values to registers (no table look-ups)
      ucol_dir = 0;
      if (le < PE && ((hdr_ring[8 * s_tab + 3] >> le) & 1u)) {
        const int lx = le / (PE == 4 ? 4 : 8), ly = le - lx * (PE == 4 ? 4 : 8);
        const double *src = u + id0 + (int64_t)(lx * (N - 1)) * op.box_ld + (ly * (N - 1) + t);
#pragma unroll
        for (int m = 0; m < N; ++m) ucol[m] = src[(int64_t)m * op.box_ld];
      } else {
#pragma unroll
        for (int m = 0; m < N; ++m) ucol[m] = 0.0;
      }
      return;
    }
    if (act) {
      uint32_t pn[N];
#pragma unroll
      for (int m = 0; m < N; ++m) pn[m] = pnb[elb[m * NP + tid]];
      // loads only: nothing below may depend on the values until the next patch
      // starts, or the warp would stall here instead of overlapping the latency
      ucol_dir = 0;
#pragma unroll
      for (int m = 0; m < N; ++m) {
        ucol[m] = u[id0 + (pn[m] & SEMK_NODE_ID_MASK)];
        ucol_dir |= (pn[m] >> 31) << m;
      }
    }
  };
  if (MODE == MODE_APPLY && p_first < p_end) {
    semk_mbar_wait(&mbar[0], 0);
    gather_column(0, p_first);
  }
  __syncthreads();

  double dot = 0.0;
  const bool want_dot = (MODE == MODE_APPLY) && (dot_partials != nullptr);
  int it = 0;
  for (int64_t patch = p_first; patch < p_end; patch += step, ++it) {
    const int s = it & 1;
    const uint32_t par = (uint32_t)((it >> 1) & 1);
    const int64_t next = patch + step;
    const bool has_next = next < p_end;
    unsigned char *sb = stage_ptr(s);
    const uint32_t *pn_s = reinterpret_cast<const uint32_t *>(sb + L.pn_off);
    semk_mbar_wait(&mbar[s], par);
    const uint32_t *hdr = hdr_ring + 8 * s;  // read before this patch's first barrier
    const int npn = (int)hdr[0];
    const int npriv = (int)hdr[1];
    const int slot_base = (int)hdr[2];
    const uint32_t id0 = hdr[4];
    const uint32_t inv_block = hdr[7];
    const int64_t slot0 = patch * PE;
    const bool active = (le < PE) && (slot0 + le < op.n_elem);


    double ycol[N];
    if (MODE == MODE_APPLY) {
      if ((flags & SEMK_MASK_IN) && ucol_dir) {
#pragma unroll
        for (int m = 0; m < N; ++m)
          if ((ucol_dir >> m) & 1u) ucol[m] = 0.0;
      }
      // The single G buffer is refilled for the next patch as soon as every thread
      // has consumed this patch's factors (hook runs right after that barrier):
      // the copy then has the rest of this patch and the start of the next to land.
      auto refill_g = [&]() {
        if (tid == 0 && has_next) issue_g(next);
      };
      // Table stage s^1 (patch i-1's tables) is free once every thread has passed the
      // first barrier of this patch's operator: no end-of-patch barrier is needed.
      auto refill_tables = [&]() {
        if (tid == 0) issue_inv(inv_block);
        if (tid == 0 && has_next) {
          const uint32_t *hn = hdr_ring + 8 * (s ^ 1);  // header of the next patch
          const int64_t after = next + step;
          issue_tables(hn[5], hn[6], s ^ 1, after < p_end ? after : -1, s);
        }
      };
      if (SEP) {
        const bool row_active = tid < NP && slot0 + tid % PE < op.n_elem;
        local_poisson_sep<N, PE, RS>(dm, le, t, tid, active, row_active, ucol, ycol, As, Bs,
                                     Gs + tid, NP, Gs + NN * PE, &mbar[2], (uint32_t)(it & 1),
                                     refill_g, refill_tables);
      } else {
        local_poisson<N, RS>(dm, le, t, active, ucol, ycol, As, Bs, Gs + tid, NP, &mbar[2],
                             (uint32_t)(it & 1), refill_g, refill_tables);
      }
      // u . y taken element by element: sum_e (Q_e u) . y_e = u . (sum_e Q_e^T y_e), so the
      // write-out never looks at u again.  Dirichlet rows are left out here (under MASK_IN
      // their entries of u are zero anyway) and come back as identity rows below.
      if (want_dot && active) {
#pragma unroll
        for (int m = 0; m < N; ++m) {
          const bool drop = (flags & SEMK_MASK_OUT) && ((ucol_dir >> m) & 1u);
          dot = fma(drop ? 0.0 : ucol[m], ycol[m], dot);
        }
      }
      // next patch: its tables landed long ago; start its gather now
      if (has_next) {
        semk_mbar_wait(&mbar[s ^ 1], (uint32_t)(((it + 1) >> 1) & 1));
        gather_column(s ^ 1, next);
      }
    } else {
      __syncthreads();  // previous patch's write-out done: its table stage may be refilled
      if (tid == 0) issue_inv(inv_block);
      if (tid == 0 && has_next) {
        const uint32_t *hn = hdr_ring + 8 * (s ^ 1);
        const int64_t after = next + step;
        issue_tables(hn[5], hn[6], s ^ 1, after < p_end ? after : -1, s);
      }
      if (active) {
        const double *lr = loc + (slot0 + le) * NN;
#pragma unroll
        for (int m = 0; m < N; ++m) ycol[m] = lr[m * N + t];
      }
    }

    // ---- assemble by GATHERING (no atomics, no colour phases): every thread leaves its
    // column of element results in scratch B (its own entries, the ones it just read; the
    // separable operator's y1 is overwritten in place),
    // then each patch node sums its <= inv_width contributions in a fixed order (ascending
    // element slot) straight from B and is stored: private nodes -> y, shared nodes ->
    // interface slots ------------------------------------------------------------------
    if (active) {
#pragma unroll
      for (int m = 0; m < N; ++m) Bs[m * RS + le * N + t] = ycol[m];
    }
    semk_mbar_wait(&mbar[3], (uint32_t)(it & 1));  // this patch's inverse table has landed
    __syncthreads();
    for (int k0 = tid; k0 < npn; k0 += kGatherBatch * kThreads) {
      uint32_t pnv[kGatherBatch];
      uint2 ev[kGatherBatch];
#pragma unroll
      for (int j = 0; j < kGatherBatch; ++j) {
        const int k = k0 + j * kThreads;
        const bool in = k < npn;
        pnv[j] = in ? pn_s[k] : 0xffffffffu;
        ev[j] = in ? reinterpret_cast<const uint2 *>(inv_s)[(size_t)k * inv_w4]
                   : make_uint2(0xffffffffu, 0xffffffffu);
      }
      double vv[kGatherBatch];
#pragma unroll
      for (int j = 0; j < kGatherBatch; ++j) {
        // (every listed node has at least one contribution)
        const uint32_t e0 = ev[j].x & 0xffffu, e1 = ev[j].x >> 16;
        const uint32_t e2 = ev[j].y & 0xffffu, e3 = ev[j].y >> 16;
        double v = (e0 != 0xffffu) ? Bs[e0] : 0.0;
        if (e1 != 0xffffu) v += Bs[e1];
        if (e2 != 0xffffu) v += Bs[e2];
        if (e3 != 0xffffu) v += Bs[e3];
        vv[j] = v;
      }
      if (inv_w4 > 1) {  // irregular meshes: more than four elements of the patch at a node
#pragma unroll
        for (int j = 0; j < kGatherBatch; ++j) {
          const int k = k0 + j * kThreads;
          if (k >= npn) continue;
          for (int w = 1; w < inv_w4; ++w) {
            const uint2 e = reinterpret_cast<const uint2 *>(inv_s)[(size_t)k * inv_w4 + w];
            const uint32_t q[4] = {e.x & 0xffffu, e.x >> 16, e.y & 0xffffu, e.y >> 16};
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (q[i] != 0xffffu) vv[j] += Bs[q[i]];
          }
        }
      }
#pragma unroll
      for (int j = 0; j < kGatherBatch; ++j) {
        const int k = k0 + j * kThreads;
        if (k >= npn) continue;
        const uint32_t pn = pnv[j];
        double v = vv[j];
        if (k < npriv) {
          const uint32_t g = id0 + (pn & SEMK_NODE_ID_MASK);
          if ((pn & SEMK_NODE_DIRICHLET) && (flags & SEMK_MASK_OUT)) {
            if (MODE == MODE_APPLY) {
              v = 0.0;
              if (flags & SEMK_DIRICHLET_IDENTITY) {
                v = u[g];
                dot = fma(v, v, dot);  // the identity rows' share of u . y
              }
            } else {
              v = fill_dirichlet;
            }
          }
          y[g] = v;
        } else {
          op.slot_buf[slot_base + (k - npriv)] = v;
        }
      }
    }
    // no barrier here: the next patch's first operator barrier orders this write-out
    // (reads of stage s, of the inverse table and of B) before anything that overwrites them
  }
  if (want_dot) __syncthreads();  // the reduction scratch aliases B: let the write-out finish
  if (want_dot) {
    const double sres = semk_block_sum(dot, red);
    if (tid == 0) dot_partials[blockIdx.x] = sres;
  }
}

template <int PE, int MODE, bool BOX = false, bool SEP = false>
struct PatchLaunch {
  // CTAs per SM of this instantiation for the given dynamic shared memory
  template <int N>
  static int occupancy(size_t smem, int *per_sm, int *sms) {
    static size_t configured = 0;  // per instantiation; one device per process
    static int cached_per_sm = 0, cached_sms = 0;
    auto kern = patch_kernel<N, PE, MODE, BOX, SEP>;
    if (smem > configured || cached_per_sm == 0) {
      SEMK_CUDA_CHECK(
          cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      SEMK_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(
          &cached_per_sm, kern, PatchCfg<N, PE>::kThreads, smem));
      int dev = 0;
      SEMK_CUDA_CHECK(cudaGetDevice(&dev));
      SEMK_CUDA_CHECK(cudaDeviceGetAttribute(&cached_sms, cudaDevAttrMultiProcessorCount, dev));
      configured = smem;
    }
    *per_sm = cached_per_sm;
    *sms = cached_sms;
    return SEMK_OK;
  }

  template <int N>
  static int run(const semk_op &op, const DMatEO &dm, const double *u, const double *loc,
                 double *y, int flags, double fill, double *partials, cudaStream_t st,
                 int *grid_out, int64_t pb, int64_t pe) {
    const size_t smem = patch_smem_layout(N, PE, MODE, op.g_patch_stride, op.pn_patch_stride,
                                          op.eloc_patch_stride, op.inv_patch_stride, SEP)
                            .total;
    if (smem > 227 * 1024) {
      semk_set_error("patch kernel: shared memory request exceeds 227 KB");
      return SEMK_ERR_UNSUPPORTED;
    }
    int per_sm = 0, sms = 0;
    int rc = occupancy<N>(smem, &per_sm, &sms);
    if (rc != SEMK_OK) return rc;
    if (per_sm < 1) {
      semk_set_error("patch kernel: does not fit on an SM");
      return SEMK_ERR_UNSUPPORTED;
    }
    // persistent grid: every CTA stays resident and loops over its patches, round-robin
    const int64_t resident = (int64_t)per_sm * sms;
    const int64_t np = pe - pb;
    // (op.max_ctas: the caller may cap the grid, e.g. to keep it from being a multiple of
    // the number of patches per tile column -- see semk.h)
    const int64_t want = (op.max_ctas > 0 && op.max_ctas < resident) ? op.max_ctas : resident;
    const unsigned grid = (unsigned)(np < want ? np : want);
    if (grid_out) *grid_out = (int)grid;
    if (grid == 0) return SEMK_OK;
    patch_kernel<N, PE, MODE, BOX, SEP><<<grid, PatchCfg<N, PE>::kThreads, smem, st>>>(
        op, dm, u, loc, y, flags, fill, partials, pb, pe);
    SEMK_LAUNCH_CHECK("patch_kernel");
    return SEMK_OK;
  }
};

}  // namespace
