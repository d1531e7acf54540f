// semk_apply.cu -- K2/K3/K5: matrix-free Poisson apply, assembly, diagonal.
//
// Reference being replaced (per element, in a Python loop):
//   Lse[p,q,r,s] from four O(N^5) einsums            examples/poisson.py:181-193
//   u_loc = u[L2G];  y_loc = einsum('pqrs,rs', L, u_loc)
//                                    examples/squirmer-axisymmetric.py:268-295
//   scatter-add through the L2G map                  sem/discrete.py:491-499
//   Dirichlet row/column elimination                 sem/discrete.py:505-510
//
// Here the dense Lse is never formed.  With the symmetric geometric factors
// G (semk_geom.cu) the local operator is (SURVEY.md appendix C)
//   ur = D u,  us = u D^T,  w0 = G00.ur + G01.us,  w1 = G01.ur + G11.us,
//   y  = D^T w0 + w1 D.
//
// Kernel layout (patch kernel, the production path):
//   * one CTA per patch of PE element slots, N threads per element; thread t
//     of an element owns column t (nodes [m][t], m = 0..N-1) in registers.
//   * contractions along the in-thread axis are N*N DFMAs whose D operand is
//     a compile-time-indexed __constant__ entry (folded into the DFMA as a
//     constant-bank operand: no shared-memory traffic, no registers);
//     the other axis is reached by transposing through shared memory.
//   * the patch's geometric factors (59% of all HBM traffic) arrive by one
//     TMA bulk copy (cp.async.bulk -> SASS UBLKCP) signalled on an mbarrier,
//     issued before the nodal gather so the two overlap.
//   * nodal values are gathered once per patch into shared memory through the
//     patch node table (coalesced for locality-preserving numberings), with
//     the Dirichlet mask carried in the table's flag bits.
//   * assembly inside the patch is a fixed-order gather (no atomics); private nodes are
//     stored straight to y, shared nodes go to interface slots that the tiny
//     `shared_nodes_kernel` sums in a fixed order => bit-reproducible.
#include "semk_patch.cuh"

namespace {

// Interface reduction: sum the partial sums of every shared node in a fixed
// order (ascending patch) and write the node's final value.
//   CTAs [0, chunk_blocks): one warp per affine chunk of <= 32 two-patch nodes --
//     node ids and both slot runs are arithmetic progressions, so a whole patch
//     edge is reduced with coalesced accesses and 32 bytes of table per chunk;
//   remaining CTAs: per-node records (nodes touched by 3+ patches), slot list inline.
// sub-range of the interface tables (both sorted by the highest patch involved, so the
// entries that are complete after patches [0, P) form a prefix): staged host apply
struct InterfaceRange {
  int64_t chunk_begin, chunk_end, rec_begin, rec_end;
};

constexpr int kChunkWarps = 8;   // warps per CTA of 256 threads
#ifndef SEMK_CHUNK_UNROLL
#define SEMK_CHUNK_UNROLL 4
#endif
constexpr int kChunkUnroll = SEMK_CHUNK_UNROLL;  // chunks per warp

// Writes the final value of a shared node; returns its identity-row share of u . y
// (the rest of u . y is taken element by element in the patch kernel).
template <int MODE>
__device__ __forceinline__ double finish_shared_node(const semk_op &op, uint32_t g, bool dir,
                                                     double v, const double *__restrict__ u,
                                                     double *__restrict__ y, int flags,
                                                     double fill_dirichlet, bool want_dot) {
  double d = 0.0;
  if (dir && (flags & SEMK_MASK_OUT)) {
    if (MODE == MODE_APPLY) {
      v = 0.0;
      if (flags & SEMK_DIRICHLET_IDENTITY) {
        v = u[g];
        d = v * v;
      }
    } else {
      v = fill_dirichlet;
    }
  }
  y[g] = v;
  return want_dot ? d : 0.0;
}

template <int MODE>
__global__ void __launch_bounds__(256)
    shared_nodes_kernel(semk_op op, const double *__restrict__ u, double *__restrict__ y,
                        int flags, double fill_dirichlet, double *__restrict__ dot_partials,
                        int64_t partial_offset, int chunk_blocks, InterfaceRange rng) {
  __shared__ double red[32];
  double dot = 0.0;
  const bool want_dot = (MODE == MODE_APPLY) && (dot_partials != nullptr);
  if ((int)blockIdx.x < chunk_blocks) {
    const int lane = threadIdx.x & 31;
    // each warp reduces kChunkUnroll chunks: all table loads first, then all slot
    // loads, then the stores (three dependent memory levels, kept wide)
    const int64_t cbase =
        rng.chunk_begin + ((int64_t)blockIdx.x * kChunkWarps + (threadIdx.x >> 5)) * kChunkUnroll;
    uint4 c0[kChunkUnroll], c1[kChunkUnroll];
    double va[kChunkUnroll], vb[kChunkUnroll];
#pragma unroll
    for (int k = 0; k < kChunkUnroll; ++k) {
      const int64_t c = cbase + k;
      const bool on = c < rng.chunk_end;
      // c0 = {node0, dn, a0, da}, c1 = {b0, db, len, Dirichlet mask}
      c0[k] = on ? reinterpret_cast<const uint4 *>(op.shared_chunk)[2 * c] : make_uint4(0, 0, 0, 0);
      c1[k] = on ? reinterpret_cast<const uint4 *>(op.shared_chunk)[2 * c + 1]
                 : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int k = 0; k < kChunkUnroll; ++k) {
      const bool on = lane < (int)c1[k].z;
      va[k] = on ? op.slot_buf[c0[k].z + (uint32_t)lane * c0[k].w] : 0.0;
      vb[k] = on ? op.slot_buf[c1[k].x + (uint32_t)lane * c1[k].y] : 0.0;
    }
#pragma unroll
    for (int k = 0; k < kChunkUnroll; ++k) {
      if (lane < (int)c1[k].z) {
        const uint32_t g = c0[k].x + (uint32_t)lane * c0[k].y;
        dot += finish_shared_node<MODE>(op, g, ((c1[k].w >> lane) & 1u) != 0, va[k] + vb[k], u, y,
                                        flags, fill_dirichlet, want_dot);
      }
    }
  } else {
    // per-node records (nodes touched by 3+ patches): one node per thread, the whole
    // slot list inline in a 32-byte record, so two dependent memory levels
    const int64_t nb = (int64_t)gridDim.x - chunk_blocks;
    const int64_t stride = nb * blockDim.x;
    for (int64_t i = rng.rec_begin + ((int64_t)blockIdx.x - chunk_blocks) * blockDim.x + threadIdx.x;
         i < rng.rec_end; i += stride) {
      const uint4 r0 = reinterpret_cast<const uint4 *>(op.shared_rec)[2 * i];
      const uint4 r1 = reinterpret_cast<const uint4 *>(op.shared_rec)[2 * i + 1];
      const uint32_t cnt = r0.y;
      const uint32_t sl[6] = {r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
      double val[6];
#pragma unroll
      for (int j = 0; j < 6; ++j)
        val[j] = ((uint32_t)j < cnt && !(cnt > 6 && j == 5)) ? op.slot_buf[sl[j]] : 0.0;
      double v = val[0];  // ascending patch order: deterministic
#pragma unroll
      for (int j = 1; j < 6; ++j)
        if ((uint32_t)j < cnt && !(cnt > 6 && j == 5)) v += val[j];
      if (cnt > 6) {
        const uint32_t *ext = op.shared_ext + r1.w;
        for (uint32_t j = 5; j < cnt; ++j) v += op.slot_buf[ext[j - 5]];
      }
      dot += finish_shared_node<MODE>(op, r0.x & SEMK_NODE_ID_MASK,
                                      (r0.x & SEMK_NODE_DIRICHLET) != 0, v, u, y, flags,
                                      fill_dirichlet, want_dot);
    }
  }
  if (want_dot) {
    const double s = semk_block_sum(dot, red);
    if (threadIdx.x == 0) dot_partials[partial_offset + blockIdx.x] = s;
  }
}

// Final, fixed-order sum of the per-CTA partials (single CTA).
__global__ void __launch_bounds__(1024)
    reduce_partials_kernel(const double *__restrict__ partials, int64_t n,
                           double *__restrict__ out) {
  __shared__ double red[32];
  double s = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) s += partials[i];
  s = semk_block_sum(s, red);
  if (threadIdx.x == 0) out[0] = s;
}

constexpr int kSharedBlocks = 148 * 64;  // upper bound on the per-node part of the interface kernel

inline void interface_blocks(const InterfaceRange &r, int *chunk_blocks, int *rec_blocks) {
  const int64_t per_block = (int64_t)kChunkWarps * kChunkUnroll;
  *chunk_blocks = (int)((r.chunk_end - r.chunk_begin + per_block - 1) / per_block);
  const int64_t want = (r.rec_end - r.rec_begin + 255) / 256;
  *rec_blocks = (int)(want < kSharedBlocks ? want : kSharedBlocks);
}

template <int MODE>
int launch_interface(const semk_op &op, const double *u, double *y, int flags, double fill,
                     double *partials, int64_t partial_offset, cudaStream_t st, int *blocks_out,
                     const InterfaceRange *range = nullptr) {
  const InterfaceRange all{0, op.n_shared_chunk, 0, op.n_shared};
  const InterfaceRange r = range ? *range : all;
  int chunk_blocks = 0, rec_blocks = 0;
  interface_blocks(r, &chunk_blocks, &rec_blocks);
  if (blocks_out) *blocks_out = chunk_blocks + rec_blocks;
  if (chunk_blocks + rec_blocks == 0) return SEMK_OK;
  shared_nodes_kernel<MODE><<<chunk_blocks + rec_blocks, 256, 0, st>>>(
      op, u, y, flags, fill, partials, partial_offset, chunk_blocks, r);
  SEMK_LAUNCH_CHECK("shared_nodes_kernel");
  return SEMK_OK;
}

// ---- simple atomic-scatter kernel (independent cross-check) -------------------
// Groups PEA consecutive element slots per CTA; reads the L2G map and the
// patch-interleaved G straight from global memory.
template <int N, int PEA>
__global__ void __launch_bounds__(PatchCfg<N, PEA>::kThreads)
    atomic_kernel(DMat dm, int64_t n_elem, const uint32_t *__restrict__ l2g,
                  const int64_t *__restrict__ elem_of_slot, const double *__restrict__ G,
                  int64_t g_patch_stride, int pe_plan, const uint8_t *__restrict__ dirichlet,
                  const double *__restrict__ u, double *__restrict__ y, int flags) {
  constexpr int NN = N * N;
  constexpr int RS = PatchCfg<N, PEA>::kRS;
  __shared__ double As[N * RS], Bs[N * RS];
  const int tid = threadIdx.x;
  const int le = tid / N, t = tid - le * N;
  const int64_t slot = (int64_t)blockIdx.x * PEA + le;
  bool active = (le < PEA) && (slot < n_elem);
  int64_t e = -1;
  if (active) e = elem_of_slot ? elem_of_slot[slot] : slot;
  active = active && e >= 0;  // (a negative entry is an empty slot of the engine order)
  double ucol[N], ycol[N];
  uint32_t gid[N];
  const double *g = G;
  if (active) {
    const uint32_t *row = l2g + e * NN;
#pragma unroll
    for (int m = 0; m < N; ++m) {
      gid[m] = row[m * N + t];
      double v = u[gid[m]];
      if (dirichlet && (flags & SEMK_MASK_IN) && dirichlet[gid[m]]) v = 0.0;
      ucol[m] = v;
    }
    const int64_t patch = slot / pe_plan;
    const int lp = (int)(slot - patch * pe_plan);
    g = G + patch * g_patch_stride + lp * N + t;
  }
  local_poisson<N, RS>(dm, le < PEA ? le : 0, t, active, ucol, ycol, As, Bs, g, N * pe_plan,
                       nullptr);
  if (active) {
#pragma unroll
    for (int m = 0; m < N; ++m) atomicAdd(y + gid[m], ycol[m]);
  }
}

__global__ void dirichlet_fix_kernel(int64_t n, const uint8_t *__restrict__ dirichlet,
                                     const double *__restrict__ u, double *__restrict__ y,
                                     int flags) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    if (dirichlet[i]) y[i] = (flags & SEMK_DIRICHLET_IDENTITY) ? u[i] : 0.0;
}

// ---- K5: element-local diagonal ------------------------------------------------
// diag[p][q] = sum_m G00[m][q] D[m][p]^2 + 2 G01[p][q] D[p][p] D[q][q]
//            + sum_n G11[p][n] D[n][q]^2
__global__ void local_diag_kernel(int n1, int pe, int64_t n_slot_elems,
                                  const double *__restrict__ G, int64_t g_patch_stride,
                                  const double *__restrict__ D, double *__restrict__ loc) {
  const int NN = n1 * n1;
  const int NP = n1 * pe;
  const int64_t total = n_slot_elems * NN;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t slot = i / NN;
    const int k = (int)(i - slot * NN);
    const int p = k / n1, q = k - p * n1;
    const int64_t patch = slot / pe;
    const int lp = (int)(slot - patch * pe);
    const double *g = G + patch * g_patch_stride + lp * n1;  // + (c*n1 + m)*NP + n
    double acc = 2.0 * g[(n1 + p) * NP + q] * D[p * n1 + p] * D[q * n1 + q];
    for (int m = 0; m < n1; ++m) {
      const double d0 = D[m * n1 + p], d1 = D[m * n1 + q];
      acc = fma(g[m * NP + q], d0 * d0, acc);
      acc = fma(g[(2 * n1 + p) * NP + m], d1 * d1, acc);
    }
    loc[i] = acc;
  }
}

__global__ void weighted_local_kernel(int NN, int64_t n_elem, const double *__restrict__ JxW,
                                      const uint32_t *__restrict__ l2g,
                                      const int64_t *__restrict__ elem_of_slot,
                                      const double *__restrict__ f, double *__restrict__ loc) {
  const int64_t total = n_elem * NN;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t slot = i / NN;
    const int k = (int)(i - slot * NN);
    const int64_t e = elem_of_slot ? elem_of_slot[slot] : slot;
    double v = 0.0;  // empty slot
    if (e >= 0) {
      v = JxW[e * NN + k];
      if (f) v *= f[l2g[e * NN + k]];
    }
    loc[i] = v;
  }
}


// elements per patch supported by the compiled kernels
inline bool pe_supported(int pe) { return pe == 4 || pe == 8 || pe == 16 || pe == 32; }

// 32-element patches (4 x 8 tiles) exist for the low orders only (n1 <= kBigPatchMaxN1):
// small elements amortise the per-patch barriers and tables better over a larger patch and
// have a smaller share of interface nodes.
constexpr int kBigPatchMaxN1 = 7;
template <int NV, int MODE, bool SEP = false, bool OK = (NV <= kBigPatchMaxN1)>
struct BigPatch {
  static int run(const semk_op &op, const DMatEO &dm, const double *u, const double *loc,
                 double *y, int flags, double fill, double *partials, cudaStream_t st,
                 int *grid_out, int64_t pb, int64_t pe) {
    return PatchLaunch<32, MODE, false, SEP>::template run<NV>(op, dm, u, loc, y, flags, fill,
                                                               partials, st, grid_out, pb, pe);
  }
  static int occupancy(size_t smem, int *per_sm, int *sms) {
    return PatchLaunch<32, MODE, false, SEP>::template occupancy<NV>(smem, per_sm, sms);
  }
};
template <int NV, int MODE, bool SEP>
struct BigPatch<NV, MODE, SEP, false> {
  static int run(const semk_op &, const DMatEO &, const double *, const double *, double *, int,
                 double, double *, cudaStream_t, int *, int64_t, int64_t) {
    semk_set_error("32-element patches are compiled for n1 <= 7 only");
    return SEMK_ERR_UNSUPPORTED;
  }
  static int occupancy(size_t, int *, int *) {
    semk_set_error("32-element patches are compiled for n1 <= 7 only");
    return SEMK_ERR_UNSUPPORTED;
  }
};

template <int MODE, bool SEP>
int launch_patch_table(const semk_op &op, const DMatEO &dm, const double *u, const double *loc,
                       double *y, int flags, double fill, double *partials, cudaStream_t st,
                       int *grid_out, int64_t pb, int64_t pe) {
#define SEMK_CALL(NV)                                                                     \
  do {                                                                                    \
    int rc;                                                                               \
    if (op.elems_per_patch == 32)                                                         \
      rc = BigPatch<NV, MODE, SEP>::run(op, dm, u, loc, y, flags, fill, partials, st, grid_out, \
                                        pb, pe);                                          \
    else if (op.elems_per_patch == 16)                                                    \
      rc = PatchLaunch<16, MODE, false, SEP>::template run<NV>(op, dm, u, loc, y, flags, fill, \
                                                               partials, st, grid_out, pb, pe); \
    else if (op.elems_per_patch == 8)                                                     \
      rc = PatchLaunch<8, MODE, false, SEP>::template run<NV>(op, dm, u, loc, y, flags, fill, \
                                                              partials, st, grid_out, pb, pe); \
    else                                                                                  \
      rc = PatchLaunch<4, MODE, false, SEP>::template run<NV>(op, dm, u, loc, y, flags, fill, \
                                                              partials, st, grid_out, pb, pe); \
    if (rc != SEMK_OK) return rc;                                                         \
  } while (0)
  SEMK_DISPATCH_N1(op.n1, SEMK_CALL)
#undef SEMK_CALL
  return SEMK_OK;
}

template <int MODE>
int launch_patch(const semk_op &op, const DMatEO &dm, const double *u, const double *loc,
                 double *y, int flags, double fill, double *partials, cudaStream_t st,
                 int *grid_out, int64_t pb = 0, int64_t pe = -1) {
  if (pe < 0) pe = op.n_patch;
  if (MODE == MODE_APPLY && op.kernel_variant == 1)
    return semk_ho_launch(op, u, y, flags, partials, st, grid_out, pb, pe);
  if (MODE == MODE_APPLY && op.kernel_variant == 2)
    return semk_box_launch(op, &dm, u, y, flags, partials, st, grid_out, pb, pe);
  if constexpr (MODE == MODE_APPLY) {
    if (op.separable)
      return launch_patch_table<MODE, true>(op, dm, u, loc, y, flags, fill, partials, st,
                                            grid_out, pb, pe);
  }
  return launch_patch_table<MODE, false>(op, dm, u, loc, y, flags, fill, partials, st, grid_out,
                                         pb, pe);
}

int check_op(const semk_op *op, const char *who) {
  if (!op) {
    semk_set_error(std::string(who) + ": null operator");
    return SEMK_ERR_INVALID;
  }
  if (op->n1 < 2 || op->n1 > SEMK_MAX_N1) {
    semk_set_error(std::string(who) + ": n1 outside [2, 17]");
    return SEMK_ERR_UNSUPPORTED;
  }
  if (!pe_supported(op->elems_per_patch)) {
    semk_set_error(std::string(who) + ": elems_per_patch must be 4, 8, 16 or 32");
    return SEMK_ERR_UNSUPPORTED;
  }
  const int64_t nnp = (int64_t)op->n1 * op->n1 * op->elems_per_patch;
  if (!op->pnode || !op->eloc || !op->patch_hdr || !op->inv || (op->pn_patch_stride & 3) != 0 ||
      op->inv_width < 4 || (op->inv_width & 3) != 0 ||
      op->inv_patch_stride != op->pn_patch_stride * op->inv_width ||
      op->pn_patch_stride < op->max_patch_nodes ||
      (reinterpret_cast<uintptr_t>(op->patch_hdr) & 15u) != 0 ||
      (op->eloc_patch_stride & 7) != 0 ||
      op->eloc_patch_stride < nnp ||
      (op->n_slots > 0 && !op->slot_buf) ||
      (op->n_shared > 0 && (!op->shared_rec || !op->shared_ext)) ||
      (op->n_shared_chunk > 0 && !op->shared_chunk)) {
    semk_set_error(std::string(who) + ": operator tables incomplete");
    return SEMK_ERR_INVALID;
  }
  if ((op->g_patch_stride & 1) != 0 || op->g_patch_stride < 3 * nnp) {
    semk_set_error(std::string(who) +
                   ": g_patch_stride must be even (16-byte TMA granularity) and >= 3*NN*PE");
    return SEMK_ERR_INVALID;
  }
  return SEMK_OK;
}

}  // namespace

extern "C" int64_t semk_partials_len(int64_t n_patch, int64_t n_shared) {
  // persistent grid (<= n_patch) + chunk CTAs (<= n_shared / 2 / 8 + 1) + record CTAs
  return n_patch + n_shared / (2 * kChunkWarps) + kSharedBlocks + 16;
}

namespace {

template <bool SEP>
int64_t resident_ctas_table(int n1, int elems_per_patch, size_t smem) {
  int per_sm = 0, sms = 0;
  auto run = [&]() -> int {
#define SEMK_CALL(NV)                                                                           \
  do {                                                                                          \
    int rc;                                                                                     \
    if (elems_per_patch == 32)                                                                  \
      rc = BigPatch<NV, MODE_APPLY, SEP>::occupancy(smem, &per_sm, &sms);                       \
    else if (elems_per_patch == 16)                                                             \
      rc = PatchLaunch<16, MODE_APPLY, false, SEP>::template occupancy<NV>(smem, &per_sm, &sms); \
    else if (elems_per_patch == 8)                                                              \
      rc = PatchLaunch<8, MODE_APPLY, false, SEP>::template occupancy<NV>(smem, &per_sm, &sms);  \
    else                                                                                        \
      rc = PatchLaunch<4, MODE_APPLY, false, SEP>::template occupancy<NV>(smem, &per_sm, &sms);  \
    if (rc != SEMK_OK) return rc;                                                               \
  } while (0)
    SEMK_DISPATCH_N1(n1, SEMK_CALL)
#undef SEMK_CALL
    return SEMK_OK;
  };
  if (run() != SEMK_OK) return -1;
  return (int64_t)per_sm * sms;
}

}  // namespace

extern "C" int64_t semk_patch_smem_bytes_sep(int separable, int n1, int elems_per_patch,
                                             int64_t g_patch_stride, int64_t pn_patch_stride,
                                             int64_t eloc_patch_stride,
                                             int64_t inv_patch_stride) {
  return (int64_t)patch_smem_layout(n1, elems_per_patch, MODE_APPLY, g_patch_stride,
                                    pn_patch_stride, eloc_patch_stride, inv_patch_stride,
                                    separable != 0)
      .total;
}

extern "C" int64_t semk_patch_smem_bytes(int n1, int elems_per_patch, int64_t g_patch_stride,
                                         int64_t pn_patch_stride, int64_t eloc_patch_stride,
                                         int64_t inv_patch_stride) {
  return semk_patch_smem_bytes_sep(0, n1, elems_per_patch, g_patch_stride, pn_patch_stride,
                                   eloc_patch_stride, inv_patch_stride);
}

// kernel_variant 1 has no separable instantiation: it reports its own (three-factor) footprint
extern "C" int64_t semk_resident_ctas_sep(int kernel_variant, int separable, int n1,
                                          int elems_per_patch, int64_t g_patch_stride,
                                          int64_t pn_patch_stride, int64_t eloc_patch_stride,
                                          int64_t inv_patch_stride) {
  if ((kernel_variant != 0 && kernel_variant != 1 && kernel_variant != 2) ||
      !pe_supported(elems_per_patch) || (kernel_variant == 1 && elems_per_patch == 32))
    return -1;
  const bool sep = separable != 0 && kernel_variant != 1;
  const int64_t smem = semk_patch_smem_bytes_sep(sep, n1, elems_per_patch, g_patch_stride,
                                                 pn_patch_stride, eloc_patch_stride,
                                                 inv_patch_stride);
  if (smem > 227 * 1024) return -1;
  if (kernel_variant == 1) return semk_ho_resident(n1, elems_per_patch, (size_t)smem);
  if (kernel_variant == 2) return semk_box_resident(n1, elems_per_patch, sep, (size_t)smem);
  return sep ? resident_ctas_table<true>(n1, elems_per_patch, (size_t)smem)
             : resident_ctas_table<false>(n1, elems_per_patch, (size_t)smem);
}

extern "C" int64_t semk_resident_ctas(int n1, int elems_per_patch, int64_t g_patch_stride,
                                      int64_t pn_patch_stride, int64_t eloc_patch_stride,
                                      int64_t inv_patch_stride) {
  return semk_resident_ctas_sep(0, 0, n1, elems_per_patch, g_patch_stride, pn_patch_stride,
                                eloc_patch_stride, inv_patch_stride);
}

extern "C" int64_t semk_resident_ctas_variant(int kernel_variant, int n1, int elems_per_patch,
                                              int64_t g_patch_stride, int64_t pn_patch_stride,
                                              int64_t eloc_patch_stride,
                                              int64_t inv_patch_stride) {
  return semk_resident_ctas_sep(kernel_variant, 0, n1, elems_per_patch, g_patch_stride,
                                pn_patch_stride, eloc_patch_stride, inv_patch_stride);
}


extern "C" int semk_poisson_apply_f64(const semk_op *op, const double *u, double *y, int flags,
                                      double *dot_out, void *stream) {
  int rc = check_op(op, "semk_poisson_apply_f64");
  if (rc != SEMK_OK) return rc;
  SEMK_REQUIRE(u && y && u != y, "semk_poisson_apply_f64: u and y must be distinct buffers");
  SEMK_REQUIRE(op->G && op->D_host, "semk_poisson_apply_f64: missing G or D");
  SEMK_REQUIRE(!dot_out || op->partials, "semk_poisson_apply_f64: dot_out needs op->partials");
  cudaStream_t st = semk_stream(stream);
  DMatEO dm;
  if (!make_dmat_eo(op->n1, op->D_host, &dm)) {
    semk_set_error(
        "semk_poisson_apply_f64: differentiation matrix is not centro-antisymmetric "
        "(the engine needs a basis whose nodes are symmetric about 0)");
    return SEMK_ERR_UNSUPPORTED;
  }
  double *partials = dot_out ? op->partials : nullptr;
  int grid = 0;
  rc = launch_patch<MODE_APPLY>(*op, dm, u, nullptr, y, flags, 0.0, partials, st, &grid);
  if (rc != SEMK_OK) return rc;
  int shared_blocks = 0;
  rc = launch_interface<MODE_APPLY>(*op, u, y, flags, 0.0, partials, grid, st, &shared_blocks);
  if (rc != SEMK_OK) return rc;
  if (dot_out) {
    reduce_partials_kernel<<<1, 1024, 0, st>>>(partials, grid + shared_blocks, dot_out);
    SEMK_LAUNCH_CHECK("reduce_partials_kernel");
  }
  return SEMK_OK;
}

namespace {

constexpr int kBdiagThreads = 256;

// Robin diagonal on the distinct boundary nodes, after the apply has made y final:
// y[g] += val u[g], and (dot_out) u[g] * val u[g] summed in a fixed order and added to the
// apply's own u.y.  One thread per boundary node; a few ten thousand nodes at most per
// operator, so this is a short gather, not a stream.
__global__ void __launch_bounds__(kBdiagThreads)
    bdiag_kernel(int64_t n, const uint32_t *__restrict__ node, const double *__restrict__ val,
                 const uint8_t *__restrict__ masked, const double *__restrict__ u,
                 double *__restrict__ y, double *__restrict__ partials,
                 double *__restrict__ dot_out) {
  double acc[1] = {0.0};
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t g = node[i];
    if (masked && masked[g]) continue;
    const double ug = u[g];
    const double t = val[i] * ug;
    y[g] += t;
    acc[0] = fma(ug, t, acc[0]);
  }
  if (dot_out) {
    double tot[1];
    if (semk_finish_reduction<1>(acc, partials, tot) && threadIdx.x == 0) dot_out[0] += tot[0];
  }
}

}  // namespace

extern "C" int semk_poisson_apply_bdiag_f64(const semk_op *op, const semk_bdiag *bdiag,
                                            const double *u, double *y, int flags,
                                            double *dot_out, void *stream) {
  if (!bdiag || bdiag->n == 0) return semk_poisson_apply_f64(op, u, y, flags, dot_out, stream);
  SEMK_REQUIRE(op && bdiag->n > 0 && bdiag->n <= op->n_nodes && bdiag->node && bdiag->val,
               "semk_poisson_apply_bdiag_f64: inconsistent semk_bdiag");
  SEMK_REQUIRE(!dot_out || bdiag->partials,
               "semk_poisson_apply_bdiag_f64: dot_out needs bdiag->partials");
  int rc = semk_poisson_apply_f64(op, u, y, flags, dot_out, stream);
  if (rc != SEMK_OK) return rc;
  const uint8_t *masked =
      (op->dirichlet && (flags & (SEMK_MASK_IN | SEMK_MASK_OUT))) ? op->dirichlet : nullptr;
  const int64_t want = (bdiag->n + kBdiagThreads - 1) / kBdiagThreads;
  const unsigned grid = (unsigned)(want < kSemkRedMaxBlocks ? want : kSemkRedMaxBlocks);
  bdiag_kernel<<<grid, kBdiagThreads, 0, semk_stream(stream)>>>(
      bdiag->n, bdiag->node, bdiag->val, masked, u, y, bdiag->partials, dot_out);
  SEMK_LAUNCH_CHECK("bdiag_kernel");
  return SEMK_OK;
}

// A sub-range of the apply: patches [patch_begin, patch_end) and the interface entries
// [chunk_begin, chunk_end) / [rec_begin, rec_end) (both tables are sorted by the highest
// patch involved, so "everything patches [0, P) complete" is a prefix of each).
extern "C" int semk_poisson_apply_range_f64(const semk_op *op, const double *u, double *y,
                                            int flags, int64_t patch_begin, int64_t patch_end,
                                            int64_t chunk_begin, int64_t chunk_end,
                                            int64_t rec_begin, int64_t rec_end, void *stream) {
  int rc = check_op(op, "semk_poisson_apply_range_f64");
  if (rc != SEMK_OK) return rc;
  SEMK_REQUIRE(u && y && u != y && op->G && op->D_host,
               "semk_poisson_apply_range_f64: bad arguments");
  SEMK_REQUIRE(0 <= patch_begin && patch_begin <= patch_end && patch_end <= op->n_patch &&
                   0 <= chunk_begin && chunk_begin <= chunk_end &&
                   chunk_end <= op->n_shared_chunk && 0 <= rec_begin && rec_begin <= rec_end &&
                   rec_end <= op->n_shared,
               "semk_poisson_apply_range_f64: range outside the operator");
  cudaStream_t st = semk_stream(stream);
  DMatEO dm;
  if (!make_dmat_eo(op->n1, op->D_host, &dm)) {
    semk_set_error("semk_poisson_apply_range_f64: D is not centro-antisymmetric");
    return SEMK_ERR_UNSUPPORTED;
  }
  if (patch_end > patch_begin) {
    rc = launch_patch<MODE_APPLY>(*op, dm, u, nullptr, y, flags, 0.0, nullptr, st, nullptr,
                                  patch_begin, patch_end);
    if (rc != SEMK_OK) return rc;
  }
  const InterfaceRange r{chunk_begin, chunk_end, rec_begin, rec_end};
  return launch_interface<MODE_APPLY>(*op, u, y, flags, 0.0, nullptr, 0, st, nullptr, &r);
}

extern "C" int semk_assemble_f64(const semk_op *op, const double *loc, double *out, int flags,
                                 double fill_dirichlet, void *stream) {
  int rc = check_op(op, "semk_assemble_f64");
  if (rc != SEMK_OK) return rc;
  SEMK_REQUIRE(loc && out, "semk_assemble_f64: null pointer");
  cudaStream_t st = semk_stream(stream);
  DMatEO dm;
  std::memset(&dm, 0, sizeof(dm));
  rc = launch_patch<MODE_ASSEMBLE>(*op, dm, nullptr, loc, out, flags, fill_dirichlet, nullptr, st,
                                   nullptr);
  if (rc != SEMK_OK) return rc;
  return launch_interface<MODE_ASSEMBLE>(*op, nullptr, out, flags, fill_dirichlet, nullptr, 0, st,
                                         nullptr);
}

extern "C" int semk_poisson_local_diag_f64(const semk_op *op, const double *D_dev, double *loc,
                                           void *stream) {
  int rc = check_op(op, "semk_poisson_local_diag_f64");
  if (rc != SEMK_OK) return rc;
  SEMK_REQUIRE(loc && op->G && D_dev, "semk_poisson_local_diag_f64: null pointer");
  cudaStream_t st = semk_stream(stream);
  const int64_t n_slot_elems = op->n_patch * op->elems_per_patch;
  const int64_t total = n_slot_elems * op->n1 * op->n1;
  const int64_t want = (total + 255) / 256;
  const unsigned grid = (unsigned)(want < 148 * 16 ? want : 148 * 16);
  local_diag_kernel<<<grid, 256, 0, st>>>(op->n1, op->elems_per_patch, n_slot_elems, op->G,
                                          op->g_patch_stride, D_dev, loc);
  SEMK_LAUNCH_CHECK("local_diag_kernel");
  return SEMK_OK;
}

extern "C" int semk_weighted_local_f64(int n1, int64_t n_elem, int64_t n_slot_elems,
                                       const double *JxW, const uint32_t *l2g,
                                       const int64_t *elem_of_slot, const double *f, double *loc,
                                       void *stream) {
  SEMK_REQUIRE(n1 >= 2 && n1 <= SEMK_MAX_N1, "semk_weighted_local_f64: bad n1");
  SEMK_REQUIRE(JxW && loc && (!f || l2g), "semk_weighted_local_f64: null pointer");
  SEMK_REQUIRE(n_slot_elems >= n_elem, "semk_weighted_local_f64: n_slot_elems < n_elem");
  cudaStream_t st = semk_stream(stream);
  const int NN = n1 * n1;
  if (n_slot_elems > n_elem)
    SEMK_CUDA_CHECK(cudaMemsetAsync(loc + n_elem * NN, 0,
                                    sizeof(double) * (n_slot_elems - n_elem) * NN, st));
  if (n_elem <= 0) return SEMK_OK;
  const int64_t total = n_elem * NN;
  const int64_t want = (total + 255) / 256;
  const unsigned grid = (unsigned)(want < 148 * 16 ? want : 148 * 16);
  weighted_local_kernel<<<grid, 256, 0, st>>>(NN, n_elem, JxW, l2g, elem_of_slot, f, loc);
  SEMK_LAUNCH_CHECK("weighted_local_kernel");
  return SEMK_OK;
}

extern "C" int semk_poisson_apply_atomic_f64(int n1, int64_t n_elem, int64_t n_nodes,
                                             const uint32_t *l2g, const int64_t *elem_of_slot,
                                             const double *G, int64_t g_patch_stride,
                                             int elems_per_patch, const double *D_host,
                                             const uint8_t *dirichlet, const double *u, double *y,
                                             int flags, void *stream) {
  SEMK_REQUIRE(l2g && G && D_host && u && y && u != y,
               "semk_poisson_apply_atomic_f64: null or aliased pointer");
  SEMK_REQUIRE(n_elem > 0 && n_nodes > 0 && elems_per_patch > 0,
               "semk_poisson_apply_atomic_f64: empty problem");
  SEMK_REQUIRE(n1 >= 2 && n1 <= SEMK_MAX_N1, "semk_poisson_apply_atomic_f64: bad n1");
  cudaStream_t st = semk_stream(stream);
  const DMat dm = make_dmat(n1, D_host);
  SEMK_CUDA_CHECK(cudaMemsetAsync(y, 0, sizeof(double) * n_nodes, st));
  constexpr int PEA = 8;
  const unsigned grid = (unsigned)((n_elem + PEA - 1) / PEA);
#define SEMK_CALL(NV)                                                                       \
  atomic_kernel<NV, PEA><<<grid, PatchCfg<NV, PEA>::kThreads, 0, st>>>(                     \
      dm, n_elem, l2g, elem_of_slot, G, g_patch_stride, elems_per_patch, dirichlet, u, y, flags)
  SEMK_DISPATCH_N1(n1, SEMK_CALL)
#undef SEMK_CALL
  SEMK_LAUNCH_CHECK("atomic_kernel");
  if (dirichlet && (flags & SEMK_MASK_OUT)) {
    const int64_t want = (n_nodes + 255) / 256;
    const unsigned g2 = (unsigned)(want < 148 * 16 ? want : 148 * 16);
    dirichlet_fix_kernel<<<g2, 256, 0, st>>>(n_nodes, dirichlet, u, y, flags);
    SEMK_LAUNCH_CHECK("dirichlet_fix_kernel");
  }
  return SEMK_OK;
}

// Copy streams / events of the staged host apply, one set per device, created on
// first use (never destroyed: they live as long as the process).
namespace {
constexpr int kMaxStages = 64;
struct HostPipe {
  cudaStream_t h2d = nullptr, d2h = nullptr;
  cudaEvent_t start = nullptr, up[kMaxStages] = {}, done[kMaxStages] = {}, finish = nullptr;
  cudaEvent_t computed[2] = {}, downloaded[2] = {};  // per scratch set (batched applies)
  bool ready = false;
};
HostPipe *host_pipe() {
  static HostPipe pipes[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  HostPipe &p = pipes[dev];
  if (!p.ready) {
    if (cudaStreamCreateWithFlags(&p.h2d, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaStreamCreateWithFlags(&p.d2h, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    auto mk = [](cudaEvent_t *e) {
      return cudaEventCreateWithFlags(e, cudaEventDisableTiming) == cudaSuccess;
    };
    if (!mk(&p.start) || !mk(&p.finish)) return nullptr;
    for (int i = 0; i < kMaxStages; ++i)
      if (!mk(&p.up[i]) || !mk(&p.done[i])) return nullptr;
    for (int i = 0; i < 2; ++i)
      if (!mk(&p.computed[i]) || !mk(&p.downloaded[i])) return nullptr;
    p.ready = true;
  }
  return &p;
}

// n_applies independent applies y_k = A u_k on host buffers, each cut into the same stages.
// Three streams: uploads, compute (`st`), downloads.  Within an apply, stage i computes while
// stage i+1 uploads and stage i-1 downloads; across applies (n_sets = 2 scratch sets) the
// upload of apply k+1 also overlaps the download of apply k, so both directions of the link
// stay busy from the first byte to the last.  Events are re-recorded from apply to apply: a
// cudaStreamWaitEvent binds to the record that precedes it in host order.
int host_staged_impl(const semk_op *op, const semk_stage *stages, int n_stages, int n_applies,
                     const double *const *u_hosts, double *const *y_hosts, double *const *d_u,
                     double *const *d_y, int n_sets, int flags, cudaStream_t st, const char *who) {
  {
    int64_t pp = 0, pc = 0, pr = 0, pu = 0, py = 0;
    for (int i = 0; i < n_stages; ++i) {
      const semk_stage &s = stages[i];
      if (!(s.patch_end >= pp && s.chunk_end >= pc && s.rec_end >= pr && s.u_need >= pu &&
            s.y_final >= py && s.u_need <= op->n_nodes && s.y_final <= op->n_nodes)) {
        semk_set_error(std::string(who) + ": stage table not monotone");
        return SEMK_ERR_INVALID;
      }
      pp = s.patch_end, pc = s.chunk_end, pr = s.rec_end, pu = s.u_need, py = s.y_final;
    }
    if (!(pp == op->n_patch && pc == op->n_shared_chunk && pr == op->n_shared &&
          pu == op->n_nodes && py == op->n_nodes)) {
      semk_set_error(std::string(who) + ": last stage must complete the operator");
      return SEMK_ERR_INVALID;
    }
  }
  DMatEO dm;
  if (!make_dmat_eo(op->n1, op->D_host, &dm)) {
    semk_set_error(std::string(who) + ": D is not centro-antisymmetric");
    return SEMK_ERR_UNSUPPORTED;
  }
  HostPipe *P = host_pipe();
  if (!P) {
    semk_set_error(std::string(who) + ": could not create copy streams");
    return SEMK_ERR_CUDA;
  }
  // the copy streams start after whatever the caller queued on `stream`
  SEMK_CUDA_CHECK(cudaEventRecord(P->start, st));
  SEMK_CUDA_CHECK(cudaStreamWaitEvent(P->h2d, P->start, 0));
  SEMK_CUDA_CHECK(cudaStreamWaitEvent(P->d2h, P->start, 0));
  for (int k = 0; k < n_applies; ++k) {
    const int b = k % n_sets;
    const double *u_host = u_hosts[k];
    double *y_host = y_hosts[k], *du = d_u[b], *dy = d_y[b];
    if (k >= n_sets) {
      // scratch set b is reused: its previous apply must have been computed (u) and
      // downloaded (y) before this one overwrites it
      SEMK_CUDA_CHECK(cudaStreamWaitEvent(P->h2d, P->computed[b], 0));
      SEMK_CUDA_CHECK(cudaStreamWaitEvent(st, P->downloaded[b], 0));
    }
    int64_t pb = 0, cb = 0, rb = 0, ub = 0, yb = 0;
    for (int i = 0; i < n_stages; ++i) {
      const semk_stage &s = stages[i];
      // upload the part of u this stage's patches read ...
      if (s.u_need > ub)
        SEMK_CUDA_CHECK(cudaMemcpyAsync(du + ub, u_host + ub, sizeof(double) * (size_t)(s.u_need - ub),
                                        cudaMemcpyHostToDevice, P->h2d));
      SEMK_CUDA_CHECK(cudaEventRecord(P->up[i], P->h2d));
      SEMK_CUDA_CHECK(cudaStreamWaitEvent(st, P->up[i], 0));
      // ... run its patches and the interface entries they complete ...
      int rc = launch_patch<MODE_APPLY>(*op, dm, du, nullptr, dy, flags, 0.0, nullptr, st, nullptr,
                                        pb, s.patch_end);
      if (rc != SEMK_OK) return rc;
      const InterfaceRange r{cb, s.chunk_end, rb, s.rec_end};
      rc = launch_interface<MODE_APPLY>(*op, du, dy, flags, 0.0, nullptr, 0, st, nullptr, &r);
      if (rc != SEMK_OK) return rc;
      SEMK_CUDA_CHECK(cudaEventRecord(P->done[i], st));
      // ... and download the part of y that is final now
      SEMK_CUDA_CHECK(cudaStreamWaitEvent(P->d2h, P->done[i], 0));
      if (s.y_final > yb)
        SEMK_CUDA_CHECK(cudaMemcpyAsync(y_host + yb, dy + yb, sizeof(double) * (size_t)(s.y_final - yb),
                                        cudaMemcpyDeviceToHost, P->d2h));
      pb = s.patch_end, cb = s.chunk_end, rb = s.rec_end, ub = s.u_need, yb = s.y_final;
    }
    SEMK_CUDA_CHECK(cudaEventRecord(P->computed[b], st));
    SEMK_CUDA_CHECK(cudaEventRecord(P->downloaded[b], P->d2h));
  }
  SEMK_CUDA_CHECK(cudaEventRecord(P->finish, P->d2h));
  SEMK_CUDA_CHECK(cudaStreamWaitEvent(st, P->finish, 0));
  SEMK_CUDA_CHECK(cudaStreamSynchronize(st));
  return SEMK_OK;
}
}  // namespace

extern "C" int semk_poisson_apply_host_staged_f64(const semk_op *op, const semk_stage *stages,
                                                  int n_stages, const double *u_host,
                                                  double *y_host, double *d_u, double *d_y,
                                                  int flags, void *stream) {
  int rc = check_op(op, "semk_poisson_apply_host_staged_f64");
  if (rc != SEMK_OK) return rc;
  SEMK_REQUIRE(stages && n_stages >= 1 && n_stages <= kMaxStages,
               "semk_poisson_apply_host_staged_f64: 1..64 stages");
  SEMK_REQUIRE(u_host && y_host && d_u && d_y && d_u != d_y,
               "semk_poisson_apply_host_staged_f64: null / aliased buffers");
  SEMK_REQUIRE(op->G && op->D_host, "semk_poisson_apply_host_staged_f64: missing G or D");
  return host_staged_impl(op, stages, n_stages, 1, &u_host, &y_host, &d_u, &d_y, 1, flags,
                          semk_stream(stream), "semk_poisson_apply_host_staged_f64");
}

extern "C" int semk_poisson_apply_host_batch_f64(const semk_op *op, const semk_stage *stages,
                                                 int n_stages, int n_applies,
                                                 const double *const *u_hosts,
                                                 double *const *y_hosts, double *d_u0,
                                                 double *d_y0, double *d_u1, double *d_y1,
                                                 int flags, void *stream) {
  int rc = check_op(op, "semk_poisson_apply_host_batch_f64");
  if (rc != SEMK_OK) return rc;
  SEMK_REQUIRE(stages && n_stages >= 1 && n_stages <= kMaxStages,
               "semk_poisson_apply_host_batch_f64: 1..64 stages");
  SEMK_REQUIRE(n_applies >= 0 && (n_applies == 0 || (u_hosts && y_hosts)),
               "semk_poisson_apply_host_batch_f64: null buffer lists");
  SEMK_REQUIRE(d_u0 && d_y0 && d_u1 && d_y1 && d_u0 != d_y0 && d_u1 != d_y1 && d_u0 != d_u1 &&
                   d_y0 != d_y1 && d_u0 != d_y1 && d_u1 != d_y0,
               "semk_poisson_apply_host_batch_f64: four distinct device scratch vectors needed");
  for (int k = 0; k < n_applies; ++k)
    SEMK_REQUIRE(u_hosts[k] && y_hosts[k] && u_hosts[k] != y_hosts[k],
                 "semk_poisson_apply_host_batch_f64: null / aliased host buffers");
  SEMK_REQUIRE(op->G && op->D_host, "semk_poisson_apply_host_batch_f64: missing G or D");
  if (n_applies == 0) return SEMK_OK;
  double *du[2] = {d_u0, d_u1}, *dy[2] = {d_y0, d_y1};
  return host_staged_impl(op, stages, n_stages, n_applies, u_hosts, y_hosts, du, dy, 2, flags,
                          semk_stream(stream), "semk_poisson_apply_host_batch_f64");
}

extern "C" int semk_poisson_apply_host_f64(const semk_op *op, const double *u_host,
                                           double *y_host, double *d_u, double *d_y, int flags,
                                           void *stream) {
  SEMK_REQUIRE(op && u_host && y_host && d_u && d_y, "semk_poisson_apply_host_f64: null pointer");
  cudaStream_t st = semk_stream(stream);
  const size_t bytes = sizeof(double) * (size_t)op->n_nodes;
  SEMK_CUDA_CHECK(cudaMemcpyAsync(d_u, u_host, bytes, cudaMemcpyHostToDevice, st));
  int rc = semk_poisson_apply_f64(op, d_u, d_y, flags, nullptr, st);
  if (rc != SEMK_OK) return rc;
  SEMK_CUDA_CHECK(cudaMemcpyAsync(y_host, d_y, bytes, cudaMemcpyDeviceToHost, st));
  SEMK_CUDA_CHECK(cudaStreamSynchronize(st));
  return SEMK_OK;
}
