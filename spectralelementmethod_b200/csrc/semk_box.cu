// semk_box.cu -- the BOX instantiations of the patch kernel (semk_op.kernel_variant == 2):
// operator apply on regularly numbered structured meshes with an arithmetic gather (node ids
// of a tile box computed instead of looked up).  Same operator, same tables for everything
// irregular and for the write-out, results bit-identical to the table-driven kernel
// (semk_apply.cu); see semk_patch.cuh.
//
// Reference being replaced: the dense local apply + scatter of
// examples/squirmer-axisymmetric.py:268-295 / sem/discrete.py:491-510, as in semk_apply.cu.
#include "semk_patch.cuh"

namespace {

#ifndef SEMK_BOX_MIN_N1
#define SEMK_BOX_MIN_N1 3
#endif
#ifndef SEMK_BOX_MAX_N1
#define SEMK_BOX_MAX_N1 17
#endif

// 32-element patches (4 x 8 tiles) exist for the low orders only, as in semk_apply.cu
constexpr int kBoxBigPatchMaxN1 = 7;
template <int NV, int PE>
constexpr bool box_ok() {
  return NV >= SEMK_BOX_MIN_N1 && NV <= SEMK_BOX_MAX_N1 && (PE != 32 || NV <= kBoxBigPatchMaxN1);
}

template <int NV, int PE, bool SEP, bool OK = box_ok<NV, PE>()>
struct BoxN {
  static int run(const semk_op &op, const DMatEO &dm, const double *u, double *y, int flags,
                 double *partials, cudaStream_t st, int *grid_out, int64_t pb, int64_t pe) {
    return PatchLaunch<PE, MODE_APPLY, true, SEP>::template run<NV>(
        op, dm, u, nullptr, y, flags, 0.0, partials, st, grid_out, pb, pe);
  }
  static int occupancy(size_t smem, int *per_sm, int *sms) {
    return PatchLaunch<PE, MODE_APPLY, true, SEP>::template occupancy<NV>(smem, per_sm, sms);
  }
};
template <int NV, int PE, bool SEP>
struct BoxN<NV, PE, SEP, false> {
  static int run(const semk_op &, const DMatEO &, const double *, double *, int, double *,
                 cudaStream_t, int *, int64_t, int64_t) {
    semk_set_error("box kernel: compiled for 3 <= n1 <= 17 (32-element patches: n1 <= 7) only");
    return SEMK_ERR_UNSUPPORTED;
  }
  static int occupancy(size_t, int *, int *) {
    semk_set_error("box kernel: compiled for 3 <= n1 <= 17 (32-element patches: n1 <= 7) only");
    return SEMK_ERR_UNSUPPORTED;
  }
};

template <bool SEP>
int box_launch(const semk_op &op, const DMatEO &dm, const double *u, double *y, int flags,
               double *partials, cudaStream_t st, int *grid_out, int64_t pb, int64_t pe) {
#define SEMK_CALL(NV)                                                                          \
  do {                                                                                         \
    int rc;                                                                                    \
    if (op.elems_per_patch == 32) {                                                            \
      rc = BoxN<NV, 32, SEP>::run(op, dm, u, y, flags, partials, st, grid_out, pb, pe);        \
    } else if (op.elems_per_patch == 16) {                                                     \
      rc = BoxN<NV, 16, SEP>::run(op, dm, u, y, flags, partials, st, grid_out, pb, pe);        \
    } else if (op.elems_per_patch == 8) {                                                      \
      rc = BoxN<NV, 8, SEP>::run(op, dm, u, y, flags, partials, st, grid_out, pb, pe);         \
    } else {                                                                                   \
      semk_set_error("box kernel: elems_per_patch must be 8, 16 or 32");                       \
      rc = SEMK_ERR_UNSUPPORTED;                                                               \
    }                                                                                          \
    if (rc != SEMK_OK) return rc;                                                              \
  } while (0)
  SEMK_DISPATCH_N1(op.n1, SEMK_CALL)
#undef SEMK_CALL
  return SEMK_OK;
}

template <bool SEP>
int64_t box_resident(int n1, int elems_per_patch, size_t smem) {
  int per_sm = 0, sms = 0;
  auto run = [&]() -> int {
#define SEMK_CALL(NV)                                                         \
  do {                                                                        \
    int rc;                                                                   \
    if (elems_per_patch == 32) {                                              \
      rc = BoxN<NV, 32, SEP>::occupancy(smem, &per_sm, &sms);                 \
    } else if (elems_per_patch == 16) {                                       \
      rc = BoxN<NV, 16, SEP>::occupancy(smem, &per_sm, &sms);                 \
    } else if (elems_per_patch == 8) {                                        \
      rc = BoxN<NV, 8, SEP>::occupancy(smem, &per_sm, &sms);                  \
    } else                                                                    \
      rc = SEMK_ERR_UNSUPPORTED;                                              \
    if (rc != SEMK_OK) return rc;                                             \
  } while (0)
    SEMK_DISPATCH_N1(n1, SEMK_CALL)
#undef SEMK_CALL
    return SEMK_OK;
  };
  if (run() != SEMK_OK) return -1;
  return (int64_t)per_sm * sms;
}

}  // namespace

int semk_box_launch(const semk_op &op, const void *dm_eo, const double *u, double *y, int flags,
                    double *partials, cudaStream_t st, int *grid_out, int64_t pb, int64_t pe) {
  const DMatEO &dm = *static_cast<const DMatEO *>(dm_eo);  // (DMatEO is TU-local: passed opaquely)
  if (op.box_ld <= 0) {
    semk_set_error("box kernel: semk_op.box_ld not set (the numbering is not a regular lattice)");
    return SEMK_ERR_INVALID;
  }
  return op.separable ? box_launch<true>(op, dm, u, y, flags, partials, st, grid_out, pb, pe)
                      : box_launch<false>(op, dm, u, y, flags, partials, st, grid_out, pb, pe);
}

int64_t semk_box_resident(int n1, int elems_per_patch, bool sep, size_t smem) {
  return sep ? box_resident<true>(n1, elems_per_patch, smem)
             : box_resident<false>(n1, elems_per_patch, smem);
}
