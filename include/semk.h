/*
 * semk.h -- C ABI of libsemk, the sm_100a spectral-element operator engine.
 *
 * This is the drop-in boundary for the one hot path of
 * nchisholm/SpectralElementMethod that this repository accelerates:
 *
 *     per-element geometric factors -> matrix-free Poisson stiffness apply ->
 *     global assembly over the local-to-global (L2G) node map with Dirichlet
 *     masking -> Jacobi-preconditioned conjugate gradients.
 *
 * The reference has no FFI of its own (it is pure Python); each entry point
 * below names the reference code it replaces (path:line under the reference
 * tree).  The Python binding a maintainer would add is in INTEGRATION.md and
 * is what spectralelementmethod_b200/_lib.py implements with ctypes.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no C++ or torch types.
 *   - every function returns an int status: 0 = ok, <0 = error
 *     (semk_last_error() gives the message for the calling thread).
 *   - "device" pointers are caller-owned device memory (torch tensors'
 *     data_ptr()), contiguous, 16-byte aligned.  The library allocates no
 *     device memory except inside the *_host convenience entry points.
 *   - stream is a cudaStream_t passed as void* (0 = legacy default stream).
 *   - element fields are C-ordered [m][n] = (xi0 index, xi1 index), n1 = p+1
 *     points per direction, NN = n1*n1; node ids are uint32 like the
 *     reference's node maps (sem/discrete.py:1044).
 */
#ifndef SEMK_H
#define SEMK_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SEMK_VERSION 100          /* 0.1.0 */
#define SEMK_MAX_N1 17            /* orders 1..16 */

/* status codes */
#define SEMK_OK 0
#define SEMK_ERR_INVALID (-1)     /* bad argument (ValueError in the Python mirror) */
#define SEMK_ERR_CUDA (-2)        /* CUDA runtime error */
#define SEMK_ERR_JACOBIAN (-3)    /* non-positive Jacobian (AssertionError, sem/mapping.py:117) */
#define SEMK_ERR_BREAKDOWN (-4)   /* PCG breakdown: pAp <= 0 or non-finite (SolverFailure) */
#define SEMK_ERR_UNSUPPORTED (-5) /* order / size outside the compiled range (NotImplementedError) */

/* node-table flag bits (upper bits of the uint32 entries of plan tables) */
#define SEMK_NODE_ID_MASK 0x3fffffffu
#define SEMK_NODE_SHARED 0x40000000u
#define SEMK_NODE_DIRICHLET 0x80000000u

/* apply flags */
#define SEMK_MASK_IN 1            /* treat Dirichlet entries of the input as zero      */
#define SEMK_MASK_OUT 2           /* zero the Dirichlet rows of the result              */
#define SEMK_DIRICHLET_IDENTITY 4 /* with MASK_OUT: y_D = u_D instead of 0 (SPD system) */

int semk_version(void);
const char *semk_last_error(void);
/* 1 if a CUDA device is usable from this process, else 0 (never an error). */
int semk_device_available(void);

/* ------------------------------------------------------------------------
 * Host-side plan: groups elements into patches (one CTA each), builds the
 * patch node tables, the per-element patch-local index table, the in-patch
 * tables and the deterministic interface reduction lists.  Pure host
 * code, no CUDA call -- usable (and tested) without a GPU.
 *
 * Replaces the bookkeeping of the reference's assembly loop
 * (sem/discrete.py:478-500: per-element meshgrid of global DOF ids, COO
 * triplets, `grhs[inds_ext] += ...`) with static tables.
 * ------------------------------------------------------------------------ */
typedef struct semk_hostplan semk_hostplan;

enum semk_plan_array {
  SEMK_PA_PATCH_NODE_PTR = 0, /* int32  [n_patch+1]   offsets into PNODE (multiples of 4)    */
  SEMK_PA_PNODE = 1,          /* uint32 [n_pnode]     global id | flags, per patch in the order
                                 [private | shared], each class ascending; padded with
                                 0xffffffff to a multiple of 4                              */
  SEMK_PA_PATCH_NPRIV = 2,    /* int32  [n_patch]     private nodes: the leading entries of the list,
                                 which the patch itself writes to the result                */
  SEMK_PA_PATCH_SLOT_BASE = 3,/* int32  [n_patch]     first interface slot of the patch      */
  SEMK_PA_ELOC = 4,           /* uint16 [n_patch][eloc_patch_stride]: per patch a table
                                 [m][le][t] (NN*PE entries) of patch-local node indices:
                                 node (m,t) of the le-th element of the patch            */
  SEMK_PA_ELEM_OF_SLOT = 5,   /* int64  [n_order]     element id stored at engine slot s, -1 = empty */
  SEMK_PA_SHARED_NODE = 6,    /* uint32 [n_shared]    global id | flags, ascending id        */
  SEMK_PA_SHARED_PTR = 7,     /* int32  [n_shared+1]  offsets into SHARED_SLOT               */
  SEMK_PA_SHARED_SLOT = 8,    /* int32  [n_slots]     interface slots of each shared node,
                                 ascending patch (slot = PATCH_SLOT_BASE[p] + k)             */
  SEMK_PA_PATCH_NNODES = 9,  /* int32  [n_patch]     number of distinct nodes of the patch  */
  SEMK_PA_PNBLK = 10,         /* uint32 [n_pn_unique][pn_stride] device node blocks: a patch's node
                                 list as in PNODE but RELATIVE to the patch's smallest node
                                 id (flags kept in the top bits), 0xffffffff padded.
                                 Identical blocks are stored once; PATCH_HDR word 5 says
                                 which block a patch uses                                   */
  SEMK_PA_ELBLK = 11,         /* uint16 [n_el_unique][el_stride] device index blocks: the ELOC
                                 table [m][le][t];
                                 deduplicated like PNBLK (PATCH_HDR word 6)                 */
  SEMK_PA_SHARED_REC = 12,    /* uint32 [n_shared_rec][8] {node id | flags, count, slot 0..5} for the
                                 shared nodes touched by 3+ patches (corners), sorted by the
                                 highest patch touching the node; counts above 6:
                                 slots 0..4 inline, word 7 = offset of the rest in SHARED_EXT   */
  SEMK_PA_SHARED_EXT = 13,    /* uint32 [...]         overflow slot lists of SHARED_REC            */
  SEMK_PA_SHARED_CHUNK = 14,  /* uint32 [n_shared_chunk][8] affine chunks of 1..32 two-patch nodes:
                                 {node0, dn, a0, da, b0, db, len, Dirichlet mask};
                                 node_k = node0 + k dn, slots a0 + k da (lower patch), b0 + k db */
  SEMK_PA_PATCH_HDR = 15,     /* uint32 [n_patch][8]  {n nodes, n private, first interface slot, 0,
                                 base node id, PNBLK block, ELBLK block, INVBLK block}; word 3
                                 is left 0 by the plan builder: a caller that selects
                                 semk_op.kernel_variant 2 writes the non-empty-slot mask of every
                                 patch it has verified to be a regular tile box there (see
                                 semk_op.box_ld)                                              */
  SEMK_PA_PATCH_MAXNODE = 16, /* uint32 [n_patch]     largest node id of the patch (the smallest is
                                 PATCH_HDR word 4)                                            */
  SEMK_PA_CHUNK_MAXPATCH = 17,/* int32  [n_shared_chunk] higher of the two patches of a chunk; the
                                 chunk table is sorted by it                                  */
  SEMK_PA_REC_MAXPATCH = 18,  /* int32  [n_shared_rec]   highest patch touching a record's node; the
                                 record table is sorted by it (then by node id)               */
  SEMK_PA_INVBLK = 19,        /* uint16 [n_inv_unique][inv_stride] inverse tables: for patch node k the
                                 entries [k*inv_width, (k+1)*inv_width) are the positions of
                                 its element-local contributions in the CTA's transposition
                                 scratch (m*RS + le*n1 + t, RS = semk_scratch_row_stride),
                                 ascending element slot, 0xffff padded; deduplicated
                                 (PATCH_HDR word 7)                                           */
  SEMK_PA_COUNT = 20
};

/* Row stride (doubles) of the patch kernel's transposition scratch: rows of
 * n1*PE thread-indexed entries padded so that the stride is 1 (mod 16). */
int semk_scratch_row_stride(int n1, int elems_per_patch);

enum semk_plan_scalar {
  SEMK_PS_N_PATCH = 0,
  SEMK_PS_N_PNODE = 1,
  SEMK_PS_N_SLOTS = 2,
  SEMK_PS_N_SHARED = 3,
  SEMK_PS_MAX_PATCH_NODES = 4,
  SEMK_PS_N_SLOT_ELEMS = 5,   /* n_patch * elems_per_patch (last patch padded) */
  SEMK_PS_ELOC_STRIDE = 6,    /* uint16 entries per patch block of ELOC: NN*PE rounded up to 8 */
  SEMK_PS_PN_STRIDE = 7,      /* uint32 entries per patch block of PNBLK (multiple of 4)       */
  SEMK_PS_EL_STRIDE = 8,      /* uint16 entries per patch block of ELBLK (multiple of 8)       */
  SEMK_PS_N_SHARED_CHUNK = 9,/* number of affine interface chunks                             */
  SEMK_PS_N_SHARED_REC = 10,  /* number of per-node interface records                          */
  SEMK_PS_N_PN_UNIQUE = 11,   /* distinct node blocks in PNBLK                                 */
  SEMK_PS_N_EL_UNIQUE = 12,   /* distinct index blocks in ELBLK                                */
  SEMK_PS_N_INV_UNIQUE = 13,  /* distinct inverse blocks in INVBLK                              */
  SEMK_PS_INV_WIDTH = 14,     /* contributions stored per node (multiple of 4; 4 = structured)   */
  SEMK_PS_INV_STRIDE = 15,    /* uint16 entries per inverse block = PN_STRIDE * INV_WIDTH        */
  SEMK_PS_COUNT = 16
};

/* l2g: host uint32 [n_elem][NN] (the reference's cell.node_ind_lexicographic,
 *      sem/discrete.py:810-812, stacked).  elem_order: host int64 [n_order]
 *      engine order, slot -> element (NULL = identity, n_order ignored);
 *      consecutive runs of elems_per_patch slots form one patch.  Every
 *      element appears exactly once; entries equal to -1 are EMPTY slots
 *      (padding that keeps patches compact tiles when the mesh is not a whole
 *      number of tiles); no patch may consist of empty slots only.
 *      dirichlet: host uint8 [n_nodes] (1 = essential-BC node, the reference's
 *      on_ebc polarity, sem/discrete.py:505) or NULL. */
int semk_hostplan_create(int n1, int64_t n_elem, int64_t n_nodes, const uint32_t *l2g,
                         const int64_t *elem_order, int64_t n_order, int elems_per_patch,
                         const uint8_t *dirichlet, semk_hostplan **out);
/* The same with an explicit thread count for the per-patch passes (0 = what OpenMP would use;
 * under torchrun OMP_NUM_THREADS is 1, so set-up code passes its own share of the box).  The
 * tables are byte-identical for every thread count. */
int semk_hostplan_create_mt(int n1, int64_t n_elem, int64_t n_nodes, const uint32_t *l2g,
                            const int64_t *elem_order, int64_t n_order, int elems_per_patch,
                            const uint8_t *dirichlet, int n_threads, semk_hostplan **out);
int64_t semk_hostplan_scalar(const semk_hostplan *plan, int which);
const void *semk_hostplan_array(const semk_hostplan *plan, int which, int64_t *n_bytes);
void semk_hostplan_destroy(semk_hostplan *plan);

/* ------------------------------------------------------------------------
 * Device tables of one operator (all device pointers; filled by the caller
 * from a host plan).
 * ------------------------------------------------------------------------ */
typedef struct semk_op {
  int32_t n1;               /* points per direction */
  int32_t elems_per_patch;
  int64_t n_elem;           /* engine slots: elements + empty padding slots (n_order of the plan) */
  int64_t n_nodes;
  int64_t n_patch;
  int64_t max_patch_nodes;
  int64_t max_ctas;         /* 0, or a cap on the persistent grid of the apply kernel.  CTA b runs
                               patches b, b + grid, ...: when the grid is a multiple of the
                               number of patches per tile column of a structured mesh every
                               CTA stays on one tile row for ever and the apply runs ~10 %
                               slower (measured: 111 tiles per column, grid 444); capping the
                               grid at resident - 1 removes the resonance                   */
  int64_t g_patch_stride;   /* doubles per patch block of G (even, >= 3*NN*PE)          */
  const double *G;          /* [n_patch][g_patch_stride]; inside a patch block the factor
                               c (0: G00, 1: G01, 2: G11) at node (m, t) of the le-th
                               element sits at ((c*n1 + m)*PE + le)*n1 + t, i.e. rows of
                               n1*PE doubles indexed by thread (le, t): coalesced, and
                               bank-conflict free once staged in shared memory           */
  const uint32_t *patch_hdr;/* [n_patch][8] per-patch headers (SEMK_PA_PATCH_HDR)           */
  const uint32_t *pnode;    /* [n_pn_unique][pn_patch_stride] node blocks (SEMK_PA_PNBLK)  */
  int64_t pn_patch_stride;  /* uint32 entries per node block (multiple of 4)             */
  const uint16_t *eloc;     /* [n_el_unique][eloc_patch_stride] index blocks (SEMK_PA_ELBLK) */
  int64_t eloc_patch_stride;/* uint16 entries per index block (multiple of 8)            */
  const uint16_t *inv;      /* [n_inv_unique][inv_patch_stride] inverse blocks (SEMK_PA_INVBLK) */
  int64_t inv_patch_stride; /* uint16 entries per inverse block (SEMK_PS_INV_STRIDE)      */
  int64_t inv_width;        /* SEMK_PS_INV_WIDTH                                           */
  int64_t n_slots;
  double *slot_buf;         /* [n_slots] interface partial sums, contiguous per patch (scratch) */
  int64_t n_shared;           /* number of per-node interface records                        */
  const uint32_t *shared_rec; /* [n_shared][8] packed interface records (SEMK_PA_SHARED_REC) */
  const uint32_t *shared_ext; /* overflow slot lists (SEMK_PA_SHARED_EXT)                    */
  int64_t n_shared_chunk;     /* number of affine interface chunks                           */
  const uint32_t *shared_chunk; /* [n_shared_chunk][8] (SEMK_PA_SHARED_CHUNK)                */
  double *partials;         /* [semk_partials_len()] dot-product scratch    */
  const double *D_host;     /* HOST pointer, [NN] differentiation matrix    */
  const uint8_t *dirichlet; /* [n_nodes] 1 = essential-BC node, or NULL (PCG: not an unknown) */
  int64_t kernel_variant;   /* thread mapping of the apply kernel: 0 = one thread per element
                               column (patch_kernel, csrc/semk_apply.cu); 1 = a column lane +
                               a row lane per element column (ho_patch_kernel, csrc/semk_ho.cu;
                               n1 >= 9): twice the warps at half the registers, for the high
                               orders where the column mapping is latency-bound; 2 = the column
                               mapping with an arithmetic gather / write-out for regularly
                               numbered structured meshes (csrc/semk_box.cu; needs box_ld) */
  int64_t box_ld;           /* kernel_variant 2: node-id stride between consecutive node rows of the
                               lattice.  A patch whose PATCH_HDR word 3 is non-zero is a tile box:
                               node (m, t) of its slot le = lx*by + ly has the id
                               base + (lx*p + m)*box_ld + ly*p + t (base = PATCH_HDR word 4) and
                               carries no Dirichlet node; word 3 = mask of its non-empty slots.
                               Patches with word 3 == 0 use the tables.  0 = not a lattice */
  int64_t separable;        /* 1: the G01 slab of every patch block is zero (axis-aligned elements),
                               and kernel_variants 0 and 2 run the separable element operator
                               y = D^T (G00 . D u) + (G11 . u D^T) D, which stages and reads only
                               the G00 and G11 slabs.  G keeps its three-slab layout (the zero
                               G01 slab is simply not read).  kernel_variant 1 ignores the
                               field.  0 = the three-factor operator                          */
} semk_op;

/* number of doubles the `partials` scratch of an operator must hold
 * (n_shared = total number of shared nodes, SEMK_PS_N_SHARED) */
int64_t semk_partials_len(int64_t n_patch, int64_t n_shared);
/* CTAs of the apply kernel that are co-resident on the current device for this
 * configuration = the grid of the persistent kernel; <0 on error */
int64_t semk_resident_ctas(int n1, int elems_per_patch, int64_t g_patch_stride,
                           int64_t pn_patch_stride, int64_t eloc_patch_stride,
                           int64_t inv_patch_stride);
/* the same for a given semk_op.kernel_variant */
int64_t semk_resident_ctas_variant(int kernel_variant, int n1, int elems_per_patch,
                                   int64_t g_patch_stride, int64_t pn_patch_stride,
                                   int64_t eloc_patch_stride, int64_t inv_patch_stride);
/* dynamic shared memory (bytes) one CTA of the apply kernel needs */
int64_t semk_patch_smem_bytes(int n1, int elems_per_patch, int64_t g_patch_stride,
                              int64_t pn_patch_stride, int64_t eloc_patch_stride,
                              int64_t inv_patch_stride);
/* the two queries above for an operator with the given semk_op.separable (1: the separable
 * kernel, which stages two of the three G slabs); separable = 0 is the plain query */
int64_t semk_resident_ctas_sep(int kernel_variant, int separable, int n1, int elems_per_patch,
                               int64_t g_patch_stride, int64_t pn_patch_stride,
                               int64_t eloc_patch_stride, int64_t inv_patch_stride);
int64_t semk_patch_smem_bytes_sep(int separable, int n1, int elems_per_patch,
                                  int64_t g_patch_stride, int64_t pn_patch_stride,
                                  int64_t eloc_patch_stride, int64_t inv_patch_stride);

/* ------------------------------------------------------------------------
 * K1: geometric factors.  Replaces, per element, Mapping._compute_x_phys /
 * _compute_jacobian (sem/mapping.py:98-119: compute_coeffs_grid_eq LU solves,
 * sem/basis_functions.py:599-624; tensor gradient, :626-650), det_inv_2x2
 * (sem/linalg.py:105-115), FiniteElement.detJxW (sem/discrete.py:594-597 with
 * TensorQuadratureRule.xweight, sem/quadratures.py:268-275) and the
 * G = JxW * invJ invJ^T contraction implicit in examples/poisson.py:166-193.
 *
 * nodes_x/nodes_y: device [n_nodes] (rows of the reference's mesh.nodes);
 * l2g: device uint32 [n_elem][NN]; Einv, D: device [NN]; w: device [n1].
 * elem_of_slot: device int64 [n_elem] or NULL (identity).  Outputs are
 * optional (NULL = skip): G in the engine's patch-interleaved layout (see
 * semk_op.G) for patches of elems_per_patch slots and block stride
 * g_patch_stride (the caller zero-fills the padding of a ragged last patch);
 * JxW [n_elem][NN], x_phys [n_elem][2][NN], J / invJ [n_elem][2][2][NN],
 * detJ [n_elem][NN] in the reference's element order and layouts.
 * bad_flag: device int32, set to 1 if any detJ <= 0 (caller zeroes it).
 * ------------------------------------------------------------------------ */
int semk_geom_factors_f64(int n1, int64_t n_elem, const double *nodes_x, const double *nodes_y,
                          const uint32_t *l2g, const double *Einv, const double *D,
                          const double *w, const int64_t *elem_of_slot, double *G,
                          int64_t g_patch_stride, int elems_per_patch, double *JxW,
                          double *x_phys, double *J, double *invJ, double *detJ,
                          int32_t *bad_flag, void *stream);

/* Nodal fields after a solve: K1's geometry recomputed (the same device arithmetic, so
 * nothing per element is kept between calls), then the physical gradient of a nodal
 * vector u, grad u = invJ^T (D u, u D^T) -- FiniteElement.gradient (sem/discrete.py:680-684).
 * One pass over the elements `elems` (device int64 [n_elem], NULL = all, in order), one CTA
 * per element.  Replaces, with n_nodes-long device vectors and every output optional
 * (NULL = skip):
 *   xy [2][n_nodes]: GLL-node coordinates, x_phys written at the entries whose winner byte
 *     is set (winner as in semk_values_at_nodes_f64: the last element containing a node);
 *     the loop `X[:, node_ind] = fe.x_phys` over finite_elements(x_phys=True).
 *   grad_loc [2][n_elem][NN] (component-major, element in list order): grad u per element
 *     (fe.gradient(u[fe.node_ind])), times JxW when `weighted` (for the JxW-weighted nodal
 *     average: sum each component and jxw_loc onto nodes with semk_face_sum_f64);
 *     jxw_loc [n_elem][NN]: JxW (fe.detJxW).
 *   sums [5] (device): sum over elements of fe.integrate((u - u_ref)^2),
 *     fe.integrate(|grad u - g_ref|^2), max |u - u_ref| over the nodes,
 *     fe.integrate(u_ref^2), fe.integrate(|g_ref|^2); u_ref [n_nodes] and g_ref
 *     [2][n_nodes] nodal, NULL = 0.  GLL collocation quadrature, as the reference's.
 *     Fixed-order reduction: bitwise reproducible.  partials: semk_vec_partials_len()
 *     doubles, zeroed once; no other call may use them concurrently.
 * u may be NULL when only xy is asked for.  bad_flag as in semk_geom_factors_f64. */
int semk_field_grad_f64(int n1, int64_t n_elem, const double *nodes_x, const double *nodes_y,
                        const uint32_t *l2g, const double *Einv, const double *D, const double *w,
                        const int64_t *elems, int64_t n_nodes, const double *u,
                        const uint8_t *winner, double *xy, double *grad_loc, int weighted,
                        double *jxw_loc, const double *u_ref, const double *g_ref, double *sums,
                        double *partials, int32_t *bad_flag, void *stream);

/* G (engine slot layout) from externally supplied factors in the reference's
 * layouts: invJ [n_elem][2][2][NN] (fe.invJ) and JxW [n_elem][NN]
 * (fe.detJxW).  Parity tier T1 (SURVEY.md 8c). */
int semk_gfactors_from_invj_f64(int n1, int64_t n_elem, const double *invJ, const double *JxW,
                                const int64_t *elem_of_slot, double *G, int64_t g_patch_stride,
                                int elems_per_patch, void *stream);

/* Weighted stiffness: G <- weight * G node by node, weight in the reference's
 * element-local layout [n_elem][NN].  Turns the operator into the stiffness
 * of -div(weight grad u): the rho-weighted twin of the Poisson recipe, the
 * four `rho_JxW` einsums of examples/squirmer-axisymmetric.py:194-213
 * (weight = x_phys[0] there). */
int semk_scale_gfactors_f64(int n1, int64_t n_elem, const double *weight,
                            const int64_t *elem_of_slot, double *G, int64_t g_patch_stride,
                            int elems_per_patch, void *stream);

/* ------------------------------------------------------------------------
 * K2: y = A u, the assembled Poisson stiffness operator, matrix-free.
 * Replaces the dense local apply np.einsum('pqrs,rs', L, u[L2G])
 * (examples/squirmer-axisymmetric.py:268-270,284-295) with L from
 * examples/poisson.py:166-193, the scatter-add of sem/discrete.py:491-499
 * and the Dirichlet row/column elimination of sem/discrete.py:505-510.
 * u, y: device [n_nodes], distinct buffers.  dot_out: device double or NULL;
 * receives sum_k u_k y_k over the (masked) input and the result.
 * Deterministic: no floating-point atomics.
 * ------------------------------------------------------------------------ */
int semk_poisson_apply_f64(const semk_op *op, const double *u, double *y, int flags,
                           double *dot_out, void *stream);

/* Same operator, simple one-element-per-thread-group kernel with
 * red.global.add.f64 scatter on a zeroed y (not deterministic in the last
 * bit).  Kept as the independent cross-check of the patch kernel.
 * l2g: device uint32 [n_elem][NN]; dirichlet: device uint8 [n_nodes] or NULL. */
int semk_poisson_apply_atomic_f64(int n1, int64_t n_elem, int64_t n_nodes, const uint32_t *l2g,
                                  const int64_t *elem_of_slot, const double *G,
                                  int64_t g_patch_stride, int elems_per_patch,
                                  const double *D_host, const uint8_t *dirichlet,
                                  const double *u, double *y, int flags, void *stream);

/* Host-buffer convenience call (the e2e path of bench.py): copies u from
 * host, applies, copies y back; all on `stream`, synchronises before return.
 * d_u, d_y: device scratch [n_nodes]. */
int semk_poisson_apply_host_f64(const semk_op *op, const double *u_host, double *y_host,
                                double *d_u, double *d_y, int flags, void *stream);

/* The same with the three phases PIPELINED over `n_stages` (<= 64) stages of
 * the patch sequence: while stage i computes, stage i+1's part of u is being
 * uploaded and stage i-1's part of y downloaded (two internal copy streams;
 * PCIe is full duplex).  Stage i runs patches [stages[i-1].patch_end,
 * stages[i].patch_end) and the interface chunks / records up to chunk_end /
 * rec_end (the tables are sorted by the highest patch involved, so these are
 * prefixes); it needs u[0, u_need) on the device and makes y[0, y_final)
 * final.  All five columns are non-decreasing and the last stage ends at
 * (n_patch, n_shared_chunk, n_shared, n_nodes, n_nodes).  With a numbering
 * that does not follow the patch order the stage table degenerates (u_need =
 * n_nodes early, y_final = 0 until the end) and the call behaves like
 * semk_poisson_apply_host_f64.  Blocks until y_host is complete. */
typedef struct semk_stage {
  int64_t patch_end, chunk_end, rec_end, u_need, y_final;
} semk_stage;
int semk_poisson_apply_host_staged_f64(const semk_op *op, const semk_stage *stages, int n_stages,
                                       const double *u_host, double *y_host, double *d_u,
                                       double *d_y, int flags, void *stream);

/* A batch of n_applies independent applies y_k = A u_k on host buffers (u_hosts[k],
 * y_hosts[k]: pinned host memory, [n_nodes] each), every one cut into the same stages as
 * above, with TWO device scratch sets (d_u0, d_y0), (d_u1, d_y1) used alternately: besides
 * the overlap inside one apply, the upload of apply k+1 overlaps the download of apply k,
 * so the full-duplex link is busy in both directions for the whole call (one apply alone
 * leaves the first upload and the last download uncovered).  The many-right-hand-sides form
 * of the reference's per-solve loop `for f in rhs: A @ f` over the assembled operator
 * (sem/discrete.py:491-510 + examples/squirmer-axisymmetric.py:284-295).  Blocks until every
 * y_hosts[k] is complete.  Results are bit-identical to semk_poisson_apply_f64. */
int semk_poisson_apply_host_batch_f64(const semk_op *op, const semk_stage *stages, int n_stages,
                                      int n_applies, const double *const *u_hosts,
                                      double *const *y_hosts, double *d_u0, double *d_y0,
                                      double *d_u1, double *d_y1, int flags, void *stream);

/* ------------------------------------------------------------------------
 * K3: generic assembly  out[g] = sum over element-local entries mapped to g
 * of loc[slot][k]  (the reference's `grhs[inds] += local` pattern,
 * sem/discrete.py:499, for any element-local field).  loc: device
 * [n_slot_elems][NN] in engine slot order.  flags: SEMK_MASK_OUT zeroes
 * Dirichlet rows (fill_dirichlet is written there instead).
 * ------------------------------------------------------------------------ */
int semk_assemble_f64(const semk_op *op, const double *loc, double *out, int flags,
                      double fill_dirichlet, void *stream);

/* K5: element-local diagonal of the stiffness matrix, diag[p,q] = L[p,q,p,q]
 * (SURVEY.md appendix C closed form), written to loc [n_slot_elems][NN] in
 * engine slot order; assemble with semk_assemble_f64.  D_dev: device [NN]. */
int semk_poisson_local_diag_f64(const semk_op *op, const double *D_dev, double *loc,
                                void *stream);

/* RHS/mass: loc[slot][k] = JxW[elem][k] * f[l2g[elem][k]]  (f NULL = 1, the
 * reference's rhs = JxW, examples/poisson.py:200).  JxW in reference element
 * order, l2g device uint32 [n_elem][NN], elem_of_slot device or NULL. */
int semk_weighted_local_f64(int n1, int64_t n_elem, int64_t n_slot_elems, const double *JxW,
                            const uint32_t *l2g, const int64_t *elem_of_slot, const double *f,
                            double *loc, void *stream);

/* ------------------------------------------------------------------------
 * K4: fused vector kernels of Jacobi-PCG (replaces sparse.linalg.spsolve,
 * sem/discrete.py:511, on the path).  Scalars live on the device:
 *   sc[0]=rz  sc[1]=pAp  sc[2]=rz_new  sc[3]=rr  sc[4]=bb
 *   sc[5]=iterations done  sc[6]=converged flag  sc[7]=breakdown flag.
 * Once sc[6] or sc[7] is set the update kernels return without touching
 * x, r, p (the iterate is frozen at the converged iteration).
 * n = vector length, n_dot = leading entries that enter dot products
 * (multi-GPU: owned nodes first, duplicates last).
 * partials: device scratch of semk_vec_partials_len(n) doubles, zeroed once
 * by the caller before first use (holds an arrival counter).
 * ------------------------------------------------------------------------ */
int64_t semk_vec_partials_len(int64_t n);
/* r = b - Ax (Ax given);  z = dinv*r;  p = z;  sc[0] = r.z, sc[3] = r.r, sc[4] = b.b.
 * dirichlet (device uint8 [n] or NULL): rows that are not unknowns -- r is forced
 * to 0 there and they do not enter ||b|| (the reduced system of sem/discrete.py:505-510). */
int semk_pcg_init_f64(int64_t n, int64_t n_dot, const double *b, const double *Ax,
                      const double *dinv, const uint8_t *dirichlet, double *r, double *p,
                      double *sc, double *partials, void *stream);
/* alpha = sc[0]/sc[1];  x += alpha p;  r -= alpha Ap;  sc[2] = r.(dinv r), sc[3] = r.r,
 * sc[5] += 1; sc[7] = 1 on breakdown (pAp <= 0 or NaN; x, r are then left unchanged).
 * x == NULL: x is left alone here and updated by semk_pcg_update_px_f64, which reads p
 * anyway (one vector pass less per iteration). */
int semk_pcg_update_xr_f64(int64_t n, int64_t n_dot, const double *p, const double *Ap,
                           const double *dinv, double *x, double *r, double *sc,
                           double *partials, void *stream);
/* beta = sc[2]/sc[0];  p = dinv*r + beta p;  then sc[0] = sc[2] */
int semk_pcg_update_p_f64(int64_t n, const double *r, const double *dinv, double *p, double *sc,
                          double *partials, void *stream);
/* the same, plus x += alpha p_old with alpha = sc[0]/sc[1] (pairs with x == NULL above) */
int semk_pcg_update_px_f64(int64_t n, const double *r, const double *dinv, double *p, double *x,
                           double *sc, double *partials, void *stream);
/* out[0] = sum_{k<n} a_k b_k (deterministic two-stage reduction) */
int semk_dot_f64(int64_t n, const double *a, const double *b, double *out, double *partials,
                 void *stream);

typedef struct semk_pcg_info {
  int32_t iterations;
  int32_t status;          /* 0 converged, 1 maxiter reached, SEMK_ERR_BREAKDOWN */
  double rel_residual;     /* recursive ||r|| / ||b|| at exit */
  double bnorm;
} semk_pcg_info;

/* Native single-GPU PCG driver on Ahat = M A M + (I - M): solves
 * Ahat x = b from the initial guess in x.  work: device [3*(n+32)] or
 * more (r, p, Ap, 256-byte aligned); sc: device [8]; vec_partials as above.  Convergence
 * ||r|| <= rtol*||b|| is polled every check_every iterations (one 64-byte
 * D2H copy); no other host synchronisation.  Re-entrant per (host thread, stream,
 * workspace): concurrent solves need their own work / sc / vec_partials AND their own
 * operator scratch (op->partials, slot buffers); an operator is bound to one stream at
 * a time.  At most maxiter iterations are run. */
int semk_pcg_solve_f64(const semk_op *op, const double *b, double *x, const double *dinv,
                       double *work, double *sc, double *vec_partials, double rtol,
                       int maxiter, int check_every, semk_pcg_info *info, void *stream);

/* ------------------------------------------------------------------------
 * Robin boundary term of the plain operator.  The weak form of
 *     w du/dn + alpha u = g   on a boundary
 * adds sum_faces sum_k alpha(x_k) dSxW_k u_k v_k to the bilinear form; with the face
 * quadrature collocated at the GLL nodes that is a DIAGONAL term on the boundary nodes
 * (the reference user adds alpha * bfe.dSxW to the diagonal of the local matrix).  It is
 * kept apart from semk_op so that operators without it keep their launch arguments.
 * ------------------------------------------------------------------------ */
typedef struct semk_bdiag {
  int64_t n;                /* distinct boundary nodes */
  const uint32_t *node;     /* [n] their ids, ascending */
  const double *val;        /* [n] assembled sum of alpha dSxW over the faces through the node */
  double *partials;         /* [semk_vec_partials_len()] dot-product scratch, zeroed once */
} semk_bdiag;

/* semk_poisson_apply_f64, then y[node[k]] += val[k] u[node[k]] on every node that the flags
 * do not mask (a Dirichlet node under SEMK_MASK_IN or SEMK_MASK_OUT gets nothing; flags == 0:
 * every node, the unmasked operator).  dot_out includes the term (deterministic, fixed-order
 * reduction).  bdiag == NULL or bdiag->n == 0: exactly the launches of
 * semk_poisson_apply_f64. */
int semk_poisson_apply_bdiag_f64(const semk_op *op, const semk_bdiag *bdiag, const double *u,
                                 double *y, int flags, double *dot_out, void *stream);
/* semk_pcg_solve_f64 on M (A + diag) M + (I - M) (graph-captured like it). */
int semk_pcg_solve_bdiag_f64(const semk_op *op, const semk_bdiag *bdiag, const double *b,
                             double *x, const double *dinv, double *work, double *sc,
                             double *vec_partials, double rtol, int maxiter, int check_every,
                             semk_pcg_info *info, void *stream);

/* ------------------------------------------------------------------------
 * Static condensation on the device (SURVEY.md 8(f) row 1): the reference's
 * actual solver formulation, DOFManagerSC (sem/discrete.py:283-528).  Element
 * interiors are eliminated element by element,
 *     S_e = A_ee - A_ei A_ii^{-1} A_ie,   g_e = f_e - A_ei A_ii^{-1} f_i
 * (compute_local_sc_system, sem/discrete.py:438-476), the condensed system over
 * the element-exterior DOFs is solved (here: Jacobi-PCG instead of
 * spsolve, :502-511) and the interiors follow by back-substitution
 * (_solve_interior_dofs, :513-524).
 *
 * Requires the exterior-first numbering of DOFManagerSC (:314-359): global
 * ids [0, n_ext) are the element-exterior nodes.  The local exterior order is
 * the reference's hierarchical one (4 vertices, then the open edges xi0=-1,
 * xi0=+1, xi1=-1, xi1=+1; sem/geometry.py:151-212), n_ext_loc = 4p entries;
 * the local interior order is lexicographic, (p-1)^2 entries.  Orders 2..10
 * (n1 = 3..11: the reference's own table range).
 *
 * The local stiffness is never stored: it is rebuilt from the geometric
 * factors G (engine layout, see semk_op.G) inside the element kernel, the
 * interior block is Cholesky-factorised in shared memory (A_ii = L L^T),
 * Z = L^{-1} A_ie, and S_e = A_ee - Z^T Z is kept PACKED (lower triangle, row
 * major, s_stride = n_ext_loc (n_ext_loc + 1) / 2 doubles per element).
 * ------------------------------------------------------------------------ */
typedef struct semk_sc_op {
  int32_t n1;
  int32_t n_ext_loc;          /* 4 (n1 - 1) */
  int64_t n_elem;             /* elements, reference element order */
  int64_t n_ext;              /* element-exterior global nodes = the leading ids */
  int64_t s_stride;           /* doubles per element block of S */
  const double *S;            /* [n_elem][s_stride] packed local Schur complements */
  const uint32_t *l2g_ext;    /* [n_elem][n_ext_loc] global ids of the exterior nodes of each
                                 element, hierarchical local order (fe.global_dof_ind_hier
                                 [:ndof_exterior], sem/discrete.py:491-492) */
  double *y_loc;              /* [n_elem][n_ext_loc] scratch: element-local results */
  const uint32_t *node_ptr;   /* [n_ext + 1] CSR offsets into node_pos */
  const uint32_t *node_pos;   /* [n_elem * n_ext_loc] for every exterior node the positions
                                 (elem * n_ext_loc + k) of its element-local entries,
                                 ascending: the fixed summation order of the assembly */
  const uint8_t *dirichlet;   /* [n_ext] 1 = essential-BC node (on_ebc of
                                 DOFManagerSC.solve, sem/discrete.py:502-505), or NULL */
  double *partials;           /* [semk_vec_partials_len()] dot-product scratch, zeroed once */
} semk_sc_op;

/* what the element kernel produces (bit-or) */
#define SEMK_SC_SCHUR 1       /* S (packed) and, if sdiag_loc != NULL, its diagonal          */
#define SEMK_SC_RHS 2         /* g_loc = f_e - A_ei A_ii^{-1} f_i                            */
#define SEMK_SC_BACKSOLVE 4   /* u_i = A_ii^{-1} (f_i - A_ie u_e) written into u             */
#define SEMK_SC_STORE_INV 16  /* also keep A_ii^{-1} (Ainv_out, semk_sc_element_react_f64): with W it
                                 makes the condensed load of any later right-hand side a stream */
#define SEMK_SC_STORE 8       /* also keep W = A_ii^{-1} A_ie (W_out), so that later back-
                                 substitutions are one streaming pass                       */

/* The element passes (one CTA per element): the factorisation outputs (SCHUR, STORE,
 * STORE_INV) in one pass, then each load output (RHS, then BACKSOLVE) as the k = 1 case of
 * semk_sc_element_block_f64 below.
 * slot_of_elem: device int64 [n_elem], engine slot holding element e's factors in G
 *   (inverse of SEMK_PA_ELEM_OF_SLOT), or NULL = identity; G / g_patch_stride /
 *   elems_per_patch as in semk_op (elems_per_patch = 1: plain [n_elem][3][NN] blocks).
 * D: device [NN].  ext_loc: device int32 [n_ext_loc] lexicographic local index of the
 *   k-th exterior node.  l2g: device uint32 [n_elem][NN].
 * Load f (modes RHS, BACKSOLVE): f_loc[k] = f_scale * JxW[e][k] * (f_nodal ?
 *   f_nodal[l2g[e][k]] : 1)  -- the reference's rhs = JxW (examples/poisson.py:200).
 * SCHUR: S_out [n_elem][s_stride]; sdiag_loc [n_elem][n_ext_loc] or NULL.
 * RHS: g_loc [n_elem][n_ext_loc].  BACKSOLVE: u device [n_nodes], exterior entries
 *   read, interior entries written.
 * STORE: W_out device [n_elem][n_ext_loc][n_int] = (A_ii^{-1} A_ie)^T (12.5 KB per element at
 *   p = 8; 180 GB of HBM make it affordable).  c_out (optional, RHS or BACKSOLVE mode): device
 *   [n_elem][n_int] = A_ii^{-1} f_i.  With both, _solve_interior_dofs (sem/discrete.py:513-524)
 *   becomes semk_sc_backsolve_stored_f64.
 * bad_flag: device int32, set to 1 when an interior block is not positive definite. */
int semk_sc_element_f64(int n1, int64_t n_elem, const int64_t *slot_of_elem, const double *G,
                        int64_t g_patch_stride, int elems_per_patch, const double *D,
                        const int32_t *ext_loc, const uint32_t *l2g, const double *JxW,
                        const double *f_nodal, double f_scale, int mode, double *S_out,
                        int64_t s_stride, double *sdiag_loc, double *g_loc, double *u,
                        double *W_out, double *c_out, int32_t *bad_flag, void *stream);
/* The same with a nodal reaction term: the local matrix is the stiffness of the recipe plus
 * diag(react[e][k]) (react: device [n_elem][NN], reference element order, or NULL).  Used for
 * the vector-Laplacian block Lve = rho-weighted stiffness + JxW/rho of
 * examples/squirmer-axisymmetric.py:210-211 inside the Stokes preconditioner. */
int semk_sc_element_react_f64(int n1, int64_t n_elem, const int64_t *slot_of_elem, const double *G,
                              int64_t g_patch_stride, int elems_per_patch, const double *D,
                              const int32_t *ext_loc, const uint32_t *l2g, const double *JxW,
                              const double *f_nodal, double f_scale, int mode, double *S_out,
                              int64_t s_stride, double *sdiag_loc, double *g_loc, double *u,
                              double *W_out, double *c_out, const double *react,
                              double *Ainv_out, int32_t *bad_flag, void *stream);
/* Condensed load from the stored interior operators (W: SEMK_SC_STORE, Ainv: SEMK_SC_STORE_INV):
 * c = A_ii^{-1} f_i and g_loc = f_e - W^T f_i with f = f_scale * JxW * f_nodal[l2g] -- the RHS
 * mode of the element kernel (compute_local_sc_system, sem/discrete.py:438-476) without
 * refactorising the interior block; the k = 1 case of semk_sc_load_stored_block_f64. */
int semk_sc_load_stored_f64(int n1, int64_t n_elem, const double *W, const double *Ainv,
                            const uint32_t *l2g, const int32_t *ext_loc, const double *JxW,
                            const double *f_nodal, double f_scale, double *g_loc, double *c_out,
                            void *stream);
/* u_i = c - W u_e for every element (c NULL: zero load): exterior entries of u read,
 * interior entries written; W, c from semk_sc_element_f64.  The k = 1 case of
 * semk_sc_backsolve_stored_block_f64. */
int semk_sc_backsolve_stored_f64(int n1, int64_t n_elem, const double *W, const double *c,
                                 const uint32_t *l2g, const int32_t *ext_loc, double *u,
                                 void *stream);

/* Block loads: the three entries above for k load columns at once (host-only query of the
 * largest k: semk_sc_block_max_cols, 32 for n1 in 3..11 and -1 otherwise; a larger k returns
 * SEMK_ERR_UNSUPPORTED).  Every block is a [k][ld] device array, row j at offset j * ld.
 * Column j's load is f_scale[j] * JxW * (bit j of nodal_mask ? F[j][l2g] : 1); f_scale is a
 * host array of k entries, F [k][ldf] is read only in the nodal columns.  Column j of every
 * output is bitwise the output of the single-load entry on load j: the same operations in
 * the same order, whatever k and the other columns.
 *
 * semk_sc_element_block_f64: one CTA per element factorises A_ii once for all k columns.
 *   mode SEMK_SC_RHS: g_loc [k][ldg >= n_elem * 4p] = f_e - A_ei A_ii^{-1} f_i (the condensed
 *   load of compute_local_sc_system, sem/discrete.py:438-476).  Mode SEMK_SC_BACKSOLVE:
 *   U [k][ldu] nodal vectors, exterior entries read, interior entries written with
 *   u_i = A_ii^{-1} (f_i - A_ie u_e) (_solve_interior_dofs, sem/discrete.py:513-524).  In
 *   either mode, if c_out is not NULL: c_out [k][ldc >= n_elem * (p-1)^2] = A_ii^{-1} f_i.
 *   G ... react as semk_sc_element_react_f64.
 * semk_sc_load_stored_block_f64: semk_sc_load_stored_f64 per column, A_ii^{-1} and W read once.
 * semk_sc_backsolve_stored_block_f64: semk_sc_backsolve_stored_f64 per column, W read once;
 *   c [k][ldc] or NULL (zero load). */
int semk_sc_block_max_cols(int n1);
int semk_sc_element_block_f64(int n1, int64_t n_elem, const double *G, int64_t g_patch_stride,
                              int elems_per_patch, const double *D, const int32_t *ext_loc,
                              const uint32_t *l2g, const double *JxW, const double *react,
                              int mode, int k, const double *F, int64_t ldf, uint32_t nodal_mask,
                              const double *f_scale, double *g_loc, int64_t ldg, double *c_out,
                              int64_t ldc, double *U, int64_t ldu, int32_t *bad_flag,
                              void *stream);
int semk_sc_load_stored_block_f64(int n1, int64_t n_elem, const double *W, const double *Ainv,
                                  const uint32_t *l2g, const int32_t *ext_loc, const double *JxW,
                                  int k, const double *F, int64_t ldf, uint32_t nodal_mask,
                                  const double *f_scale, double *g_loc, int64_t ldg, double *c_out,
                                  int64_t ldc, void *stream);
int semk_sc_backsolve_stored_block_f64(int n1, int64_t n_elem, const double *W, const double *c,
                                       int64_t ldc, const uint32_t *l2g, const int32_t *ext_loc,
                                       int k, double *U, int64_t ldu, void *stream);

/* The same element kernel on the CALLER'S OWN local systems instead of the Poisson
 * recipe -- the literal inputs of DOFManagerSC.assemble_global_sc_system / solve
 * (sem/discrete.py:478-528): A_hier device [n_elem][NN][NN] and f_hier device
 * [n_elem][NN], the dense local matrices / right-hand sides in HIERARCHICAL local
 * order (reorder_local_system_hier, :428-436: the 4p exterior DOFs first); l2g_hier:
 * device uint32 [n_elem][NN] = fe.global_dof_ind_hier (:491-492).  The local matrices
 * must be symmetric with positive definite interior blocks (Cholesky; bad_flag
 * otherwise); only their lower triangles are read.  Outputs as semk_sc_element_f64. */
int semk_sc_element_dense_f64(int n1, int64_t n_elem, const double *A_hier, const double *f_hier,
                              const uint32_t *l2g_hier, int mode, double *S_out, int64_t s_stride,
                              double *sdiag_loc, double *g_loc, double *u, int32_t *bad_flag,
                              void *stream);

/* y = S u over the exterior DOFs: per element y_loc = S_e u[l2g_ext] (dense symmetric
 * 4p x 4p product from the packed block), then every exterior node sums its entries of
 * y_loc in the fixed order of node_pos.  flags as semk_poisson_apply_f64 (Dirichlet
 * elimination of sem/discrete.py:505-510); dot_out: device double or NULL, receives
 * u . y.  Deterministic: no floating-point atomics.  u, y: device [n_ext], distinct. */
int semk_sc_apply_f64(const semk_sc_op *op, const double *u, double *y, int flags,
                      double *dot_out, void *stream);

/* out[g] = sum of loc[node_pos[..]] for every exterior node (`grhs[inds_ext] += ...`,
 * sem/discrete.py:499); loc: device [n_elem][n_ext_loc].  SEMK_MASK_OUT writes
 * fill_dirichlet on Dirichlet rows. */
int semk_sc_assemble_f64(const semk_sc_op *op, const double *loc, double *out, int flags,
                         double fill_dirichlet, void *stream);

/* out[i] = sum of vals[pos[q]], q in [ptr[i], ptr[i+1]), summed in that order: the
 * deterministic gather-sum of face-node entries (face, k) onto distinct nodes (boundary
 * loads and Robin terms).  ptr: device uint32 [n + 1]; pos: device uint32 [ptr[n]]. */
int semk_face_sum_f64(int64_t n, const uint32_t *ptr, const uint32_t *pos, const double *vals,
                      double *out, void *stream);

/* Jacobi-PCG on Shat = M S M + (I - M); arguments as semk_pcg_solve_f64 with vectors
 * of length n_ext. */
int semk_sc_pcg_solve_f64(const semk_sc_op *op, const double *b, double *x, const double *dinv,
                          double *work, double *sc, double *vec_partials, double rtol,
                          int maxiter, int check_every, semk_pcg_info *info, void *stream);

/* ------------------------------------------------------------------------
 * Two-level preconditioner for the condensed system (additive; the reference
 * solves it directly, sem/discrete.py:511): Jacobi + a vertex coarse space,
 *     M^{-1} = diag(Shat)^{-1} + P Ac^{-1} P^T,    Ac = P^T Shat P,
 * P = linear interpolation along element edges from the element vertices
 * (condensed.coarse_tables).  Ac is kept as 4 x 4 element matrices
 * Ace = Phi_e^T S_e Phi_e and applied like the fine operator (element product,
 * then the fixed-order node sum); Ac^{-1} is an inner Jacobi-PCG to a loose
 * tolerance.  Makes the outer iteration count independent of the mesh size.
 * ------------------------------------------------------------------------ */
typedef struct semk_sc_coarse {
  int64_t n_v;                /* coarse DOFs = distinct element vertices */
  const double *Ace;          /* [n_elem][16] element coarse matrices, row major */
  const uint32_t *vert_c;     /* [n_elem][4] compact vertex ids of every element */
  double *y_loc_c;            /* [n_elem][4] scratch */
  const uint32_t *vptr;       /* [n_v + 1] CSR offsets into vpos */
  const uint32_t *vpos;       /* [n_elem * 4] entries (e * 4 + a) of every vertex, ascending */
  const uint8_t *dirichlet_c; /* [n_v] 1 = vertex on the essential boundary, or NULL */
  double *partials;           /* [semk_vec_partials_len()] dot scratch, zeroed once */
  const uint32_t *pv;         /* [n_ext][2] prolongation: the (at most) two vertices of a node */
  const double *pw;           /* [n_ext][2] ... and their weights (0 = unused) */
  const uint32_t *rptr;       /* [n_v + 1] restriction = transpose of the above, CSR */
  const uint32_t *ridx;       /* [nnz] exterior node of every entry */
  const double *rw;           /* [nnz] weight of every entry */
  /* optional: the same operator assembled into ELL rows (semk_sc_coarse_ell_build_f64),
   * column major -- entry k of row v at [k * n_v + v]; identity rows on Dirichlet
   * vertices.  The multilevel driver prefers it (one SpMV kernel per inner iteration). */
  int64_t ell_width;          /* 0 = not built */
  const uint32_t *ell_cols;   /* [ell_width][n_v] */
  const double *ell_vals;     /* [ell_width][n_v] */
} semk_sc_coarse;

/* Ace = Phi_e^T S_e Phi_e for every element; phi: device [n_ext_loc][4], the local
 * interpolation matrix; rows of Dirichlet nodes and columns of Dirichlet vertices
 * (op->dirichlet) are zeroed.  Ace_out: device [n_elem][16]. */
int semk_sc_coarse_elem_f64(const semk_sc_op *op, const double *phi, double *Ace_out,
                            void *stream);
/* y = Ac x (identity rows on Dirichlet vertices with the usual flags); dot_out as in
 * semk_sc_apply_f64.  x, y: device [n_v], distinct. */
int semk_sc_coarse_apply_f64(int64_t n_elem, const semk_sc_coarse *cs, const double *x, double *y,
                             int flags, double *dot_out, void *stream);
/* Assemble Ac into ELL rows of `width` entries (<= 32; a vertex of valence d needs 2 d + 1):
 * cols / vals: device [width][n_v], written; *overflow (device int) is set to 1 if a row
 * does not fit.  Fixed summation order (ascending element), no atomics. */
int semk_sc_coarse_ell_build_f64(const semk_sc_coarse *cs, int width, uint32_t *cols, double *vals,
                                 int32_t *overflow, void *stream);
/* y = Ac x from the ELL rows (cs->ell_*), dot_out = x . y (or NULL).  x, y distinct. */
int semk_sc_coarse_ell_apply_f64(const semk_sc_coarse *cs, const double *x, double *y,
                                 double *dot_out, void *stream);
/* out[v] = sum of loc[vpos[..]]; loc: device [n_elem][4] (diagonal of Ac, ...). */
int semk_sc_coarse_assemble_f64(int64_t n_elem, const semk_sc_coarse *cs, const double *loc,
                                double *out, void *stream);
/* Third level under the vertex coarse space: the inner coarse solve is preconditioned by
 * Jacobi + a piecewise-constant aggregation of the vertices (element tiles) with a DENSE
 * inverse at the top, so that the inner iteration count is mesh-independent as well
 * (oracle/precond_study_three_level.py).  agg: device uint32 [n_v], aggregate of every
 * vertex (0xffffffff = none: essential boundary); aptr / aidx: CSR of the vertices of
 * every aggregate that this rank OWNS (one GPU: all of them); A3inv: device
 * [n_agg][n_agg], inverse of P2^T Ac P2, row major.  On several GPUs the aggregate ids
 * are global and A3inv is replicated. */
typedef struct semk_sc_top {
  int64_t n_agg;
  const uint32_t *agg;
  const uint32_t *aptr;
  const uint32_t *aidx;
  const double *A3inv;        /* FP64 copy (may be NULL when A3inv_f32 is given) */
  const float *A3inv_f32;     /* FP32 copy, preferred by the driver: half the bytes per inner
                                 iteration; the inverse only enters the preconditioner */
} semk_sc_top;

/* A3 = P2^T Ac P2 (this rank's elements only) from the element coarse matrices cs->Ace:
 * aptr_all / aidx_all: CSR of ALL local vertices of every aggregate (owned or not).
 * A3: device [n_agg][n_agg], overwritten.  One thread per row, fixed order, no atomics. */
int semk_sc_top_assemble_f64(const semk_sc_coarse *cs, int64_t n_agg, const uint32_t *agg,
                             const uint32_t *aptr_all, const uint32_t *aidx_all, double *A3,
                             void *stream);

/* ------------------------------------------------------------------------
 * Small-vector all-reduce over NVLink peer memory (no reference equivalent:
 * the reference is single-process; SURVEY.md 8(e) names the inner products of
 * the Krylov solver as the second exchange of the partitioned path).  Every
 * rank owns one REGION, exported through CUDA IPC (semk_peer_alloc /
 * semk_peer_open) and mapped by every other rank:
 *   bytes [0, 8)     : uint64 call counter (epoch), advanced by the kernel itself, so
 *                      launches can be captured in a CUDA graph;
 *   bytes [64, 128)  : uint64 flag[8] -- flag[s] = last epoch published by rank s;
 *   bytes [256, ...) : double recv[2][world][capacity] (double-buffered by epoch parity).
 * One single-CTA kernel per all-reduce: push my vector into every rank's recv slot,
 * publish the epoch (system-scope release), wait for every rank's flag (acquire), sum
 * the world slots IN RANK ORDER -- the result is bit-identical on all ranks.
 * ------------------------------------------------------------------------ */
#define SEMK_COMM_MAX_WORLD 8
typedef struct semk_comm {
  int32_t rank, world;
  int64_t capacity;                      /* doubles per all-reduce */
  void *regions[SEMK_COMM_MAX_WORLD];    /* regions[r]: rank r's region (regions[rank] = own) */
  int32_t *status;                       /* device int, set to 1 when a rank did not show up
                                            within ~2 s (the kernel gives up instead of hanging) */
} semk_comm;
int64_t semk_comm_region_bytes(int32_t world, int64_t capacity);
/* buf[0, n) <- sum over ranks, in place; n <= capacity; every rank must make the same
 * sequence of calls.  world == 1: no-op. */
int semk_comm_allreduce_f64(const semk_comm *comm, double *buf, int64_t n, void *stream);

/* One side-pair of interface columns of a strip partition (semk_halo_exchange_f64) as a
 * struct, so that a native driver can issue exchanges itself: `epoch` is the last epoch
 * used and is advanced by whoever issues an exchange (host side, SPMD). */
typedef struct semk_halo {
  int64_t n_col;
  void *mine, *left, *right;            /* regions: own, left / right neighbour (or NULL) */
  uint64_t epoch;
  int32_t *status;                      /* device int */
} semk_halo;

/* Jacobi-PCG on a strip partition with everything issued natively: exactly one of op
 * (matrix-free operator, vectors of n_nodes) / sc_op (condensed operator, vectors of n_ext)
 * is given; after every apply the interface columns are exchanged through `halo`, and the
 * two reductions of an iteration (p.Ap; [r.r, r.z]) are peer-memory all-reduces through
 * `comm` (NULL or world 1: one GPU, no exchange).  n_owned: owned prefix for the dot
 * products.  work: device [3 * (n + 32)]; sc: device [32]; other arguments as
 * semk_pcg_solve_f64.  dinv: inverse diagonal of the GLOBAL operator. */
int semk_pcg_dist_solve_f64(const semk_op *op, const semk_sc_op *sc_op, semk_halo *halo,
                            const semk_comm *comm, int64_t n_owned, const double *b, double *x,
                            const double *dinv, double *work, double *sc, double *vec_partials,
                            double rtol, int maxiter, int check_every, semk_pcg_info *info,
                            void *stream);

/* How the multilevel solver below is spread over the ranks of a strip partition
 * (NULL or comm == NULL: one GPU).  Owned DOFs are a prefix on both levels (the right
 * neighbour owns a shared column): dot products and restrictions run over the owned
 * prefix and are summed with semk_comm_allreduce_f64; operator applies are followed by
 * the interface exchange of their level. */
typedef struct semk_ml_dist {
  const semk_comm *comm;
  semk_halo *halo_f;                    /* exterior (fine) vectors */
  semk_halo *halo_c;                    /* vertex (coarse) vectors */
  int64_t n_owned_f, n_owned_c;
} semk_ml_dist;

typedef struct semk_ml_opts {
  double rtol;                          /* outer: recursive ||r|| <= rtol ||b|| */
  double inner_rtol;                    /* inner coarse solves */
  int32_t maxiter, inner_maxiter;
  int32_t levels;                       /* 2: Jacobi inside the coarse solve; 3: + aggregation */
  int32_t flexible;                     /* 1: flexible CG (Polak-Ribiere beta), the inner solve
                                           makes the preconditioner vary from step to step */
  int32_t inner_chunk;                  /* inner iterations queued between two polls (>= 1) */
  int32_t reserved;
} semk_ml_opts;

typedef struct semk_ml_info {
  int32_t iterations;                   /* outer */
  int32_t status;                       /* 0 converged, 1 maxiter, SEMK_ERR_BREAKDOWN */
  double rel_residual;                  /* recursive ||r|| / ||b|| at exit */
  double true_rel_residual;             /* ||b - Shat x|| / ||b|| recomputed at exit */
  double bnorm;
  int64_t inner_iterations;             /* summed over the inner solves */
  int32_t inner_solves;
  int32_t reserved;
} semk_ml_info;

/* Multilevel-preconditioned (flexible) CG on Shat x = b, one entry point for one GPU
 * and for a strip partition:
 *     M^{-1} r = dinv r + P xc,   xc ~= Ac^{-1} P^T r  by an inner PCG on the vertex
 *     coarse operator, itself preconditioned by dinv_c (levels = 2) or by
 *     dinv_c + P2 A3inv P2^T (levels = 3, `top` required).
 * The inner iteration keeps its scalars on the device (alpha, beta, convergence and
 * breakdown flags are produced by single-CTA kernels that also carry the all-reduce),
 * is queued `inner_chunk` iterations at a time and polled through one 128-byte copy.
 * work: device [4 * (n_ext + 32)]; work_c: device [6 * (n_v + 32) + 2 * (n_agg + 64)];
 * sc: device [64]; vec_partials as in semk_pcg_solve_f64.  dinv / dinv_c: inverse
 * diagonals of the GLOBAL operators (interface entries already summed). */
int semk_sc_mlpcg_solve_f64(const semk_sc_op *op, const semk_sc_coarse *cs, const semk_sc_top *top,
                            const semk_ml_dist *dist, const double *b, double *x,
                            const double *dinv, const double *dinv_c, double *work,
                            double *work_c, double *sc, double *vec_partials,
                            const semk_ml_opts *opts, semk_ml_info *info, void *stream);

/* The pieces of the two-level preconditioner as separate entry points, for the
 * multi-GPU outer loop (driven from the host so that the interface exchanges and
 * all-reduces can sit between them):
 *   resid   : r = b - Ax and b_masked = b, both zero on Dirichlet rows (dirichlet NULL = none)
 *   scale   : z = d * r
 *   axpy2   : x += alpha p ; r -= alpha Ap
 *   xpay    : p = z + beta p
 *   restrict: rc = P^T r over the fine nodes [0, n_owned) only (owner-weighted)
 *   prolong : z += P xc */
int semk_vec_resid_f64(int64_t n, const double *b, const double *Ax, const uint8_t *dirichlet,
                       double *r, double *b_masked, void *stream);
int semk_vec_scale_f64(int64_t n, const double *d, const double *r, double *z, void *stream);
int semk_vec_axpy2_f64(int64_t n, double alpha, const double *p, const double *Ap, double *x,
                       double *r, void *stream);
int semk_vec_xpay_f64(int64_t n, double beta, const double *z, double *p, void *stream);
int semk_sc_restrict_f64(const semk_sc_coarse *cs, const double *r, int64_t n_owned, double *rc,
                         void *stream);
int semk_sc_prolong_add_f64(int64_t n_ext, const semk_sc_coarse *cs, const double *xc, double *z,
                            void *stream);

/* ------------------------------------------------------------------------
 * Field evaluation (SURVEY.md 8(f) row 4): DOFManager.values_at_nodes
 * (sem/discrete.py:235-258) -- GLL coefficients -> values at the equispaced
 * mesh nodes, element by element through TensorProduct.interpolate_on_grid_eq
 * (sem/basis_functions.py:539-569).  l2g: device uint32 [n_elem][NN];
 * Emat: device [NN], the 1-D matrix `_interp_eq_mat` (basis functions at the
 * equispaced points); winner: device uint8 [n_elem][NN], 1 where the element
 * is the LAST one of the reference's loop containing that node (its value is
 * the one the reference keeps); coeffs, values: device [n_nodes], distinct.
 * ------------------------------------------------------------------------ */
int semk_values_at_nodes_f64(int n1, int64_t n_elem, const uint32_t *l2g, const uint8_t *winner,
                             const double *Emat, const double *coeffs, double *values,
                             void *stream);

/* Batched point location and field evaluation (rest of SURVEY.md 8(f) row 4):
 * DOFManager.find_elem_containing_point (sem/discrete.py:263-280: cells tried in ascending
 * centroid distance), Mapping.inv (sem/mapping.py:146-178: Newton from xi = 0, it_max = 8,
 * |dx| <= tol = 1e-8, inside iff -1 <= xi <= 1; sem/rootfind.py:22-53) and
 * DOFManager.interpolate (sem/discrete.py:221-233), one thread per point.
 *   x_phys    : device [n_elem][2][NN] GLL-point coordinates (semk_geom_factors_f64)
 *   centroids : device [n_elem][2] mean of the four vertices (sem/discrete.py:1108-1113)
 *   gll_nodes, bary_wts : device [n1]; D: device [NN]
 *   bins      : uniform grid bins_x x bins_y of cell size (bin_hx, bin_hy) anchored at
 *               (bin_x0, bin_y0); bin (i, j) lists elements bin_elems[bin_ptr[i*bins_y+j] ..
 *               bin_ptr[i*bins_y+j+1]) -- every element must be listed in all bins its
 *               (slightly inflated) bounding box touches
 *   points    : device [2][n_points]
 *   elem_out  : device int64 [n_points], -1 = not inside any candidate (OutsideDomain)
 *   xi_out    : device [2][n_points] parametric coordinates (NaN when not found)
 * A Newton run that does not converge within it_max steps counts as "not this element"
 * (the reference raises SolverFailure there). */
int semk_locate_points_f64(int n1, int64_t n_elem, const double *x_phys, const double *centroids,
                           const double *gll_nodes, const double *bary_wts, const double *D,
                           double bin_x0, double bin_y0, double bin_hx, double bin_hy, int bins_x,
                           int bins_y, const uint32_t *bin_ptr, const uint32_t *bin_elems,
                           int64_t n_points, const double *points, int it_max, double tol,
                           int64_t *elem_out, double *xi_out, void *stream);
/* values[q] = sum_mn coeffs[l2g[elem[q]][m][n]] l_m(xi0) l_n(xi1) (NaN where elem < 0) */
int semk_interpolate_points_f64(int n1, int64_t n_points, const int64_t *elem, const double *xi,
                                const uint32_t *l2g, const double *gll_nodes,
                                const double *bary_wts, const double *coeffs, double *values,
                                void *stream);

/* ------------------------------------------------------------------------
 * Multi-GPU: interface exchange of a strip partition over NVLink peer memory
 * (SURVEY.md 8(e); the reference itself is single-process -- its serial
 * analogue is the scatter-add `grhs[inds] += ...`, sem/discrete.py:499).
 *
 * Every rank owns one exchange REGION in device memory, exported to its two
 * neighbours through CUDA IPC:
 *   bytes [0, 256)  : four uint64 flag words -- [0..1] published by the LEFT
 *                     neighbour for epoch parity 0 / 1, [2..3] by the RIGHT one;
 *   then            : double recv[4][n_col] -- [0..1] columns received from the
 *                     left neighbour (parity 0 / 1), [2..3] from the right one.
 * ------------------------------------------------------------------------ */
#define SEMK_PEER_HANDLE_BYTES 64
int64_t semk_halo_region_bytes(int64_t n_col);
/* cudaMalloc + zero a region and export it; handle_out: host [64] */
int semk_peer_alloc(int64_t bytes, void **dev_ptr, unsigned char *handle_out);
/* map a neighbour's region (handle from its semk_peer_alloc) into this process */
int semk_peer_open(const unsigned char *handle, void **dev_ptr);
int semk_peer_close(void *dev_ptr);
int semk_peer_free(void *dev_ptr);
/* One kernel: push my boundary columns y[0, n_col) / y[n_local - n_col, n_local)
 * (partial sums of the local apply) into the neighbours' regions, publish
 * `epoch` (strictly increasing from 1, the same sequence on every rank), wait
 * for the neighbours' columns of the same epoch, add them into y, re-impose
 * the identity rows y = u on Dirichlet nodes of the shared columns
 * (dirichlet: device uint8 [n_local] or NULL) and subtract the doubly counted
 * u^2 of the column this rank does not own (the right one) from *dot_inout
 * (device scalar holding this rank's fused u.y, or NULL).  left_region /
 * right_region: peer pointers from semk_peer_open, NULL = no neighbour.
 * status: device int, set to 1 if a neighbour did not show up within ~2 s
 * (the kernel then gives up instead of hanging the GPU). */
int semk_halo_exchange_f64(int64_t n_col, int64_t n_local, double *y, const double *u,
                           const uint8_t *dirichlet, void *my_region, void *left_region,
                           void *right_region, uint64_t epoch, double *dot_inout, int *status,
                           void *stream);

/* ------------------------------------------------------------------------
 * Axisymmetric Stokes / linearised Navier-Stokes in stream function - vorticity
 * form (SURVEY.md 8(f) row 3, BASELINE config 4).  Two DOFs per node, DOF id =
 * 2*node + comp (comp 0: stream function, 1: vorticity; sem/discrete.py:561-576),
 * so nodal vectors are device [n_nodes][2] = 16-byte (psi, omega) pairs.
 *
 * Replaces, matrix-free, the dense local operators of the reference's example:
 *   pre_assembly          examples/squirmer-axisymmetric.py:163-257  (E2e, Lve, Ae, Me)
 *   compute_local_system  examples/squirmer-axisymmetric.py:259-297  (Jacobian blocks
 *                         jac[0::2,0::2] = Ae.vort, jac[0::2,1::2] = Ae.sfn + Lve,
 *                         jac[1::2,0::2] = E2e, jac[1::2,1::2] = -Me, and the residual)
 *   the scatter-add       examples/squirmer-axisymmetric.py:336-358 / sem/discrete.py:499
 *
 * The operator reuses the plan tables of a semk_op built for the same mesh
 * (semk_hostplan_build); its G / g_patch_stride name the FACTOR block
 * [n_patch][n_fac][n1][PE][n1] (same thread-major layout as G) holding
 *   0..2  rho*JxW*(invJ invJ^T)   (:194-207)      3, 4  2*JxW*invJ[0][0], 2*JxW*invJ[1][0] (:221-222)
 *   5     JxW/rho, 0 where rho = 0 (:211)         6     rho^2*JxW (:252)
 *   7..11 advection coefficients of the linearisation about a state (:227-249; n_fac = 12)
 * and its slot_buf holds 2*n_slots doubles.
 * ------------------------------------------------------------------------ */
typedef struct semk_stokes_op {
  semk_op plan;
  int32_t n_fac;          /* 7: Stokes (Re = 0); 12: with the advection coefficients */
  int32_t reserved;
  int64_t n_ess;          /* essential (Dirichlet) DOFs */
  const int64_t *ess_dof; /* device [n_ess] DOF ids 2*node + comp */
} semk_stokes_op;

int64_t semk_stokes_smem_bytes(int n1, int elems_per_patch, int64_t f_patch_stride,
                               int64_t pn_patch_stride, int64_t eloc_patch_stride,
                               int64_t inv_patch_stride);
/* factors 0..6 from the geometry in the reference's layouts: invJ [n_elem][2][2][NN]
 * (fe.invJ), JxW [n_elem][NN] (fe.detJxW), x_phys [n_elem][2][NN] (fe.x_phys; [0] = rho) */
int semk_stokes_factors_f64(int n1, int64_t n_slot_elems, const double *invJ, const double *JxW,
                            const double *x_phys, const int64_t *elem_of_slot, double *F,
                            int64_t f_patch_stride, int elems_per_patch, void *stream);
/* factors 7..11: linearise the advection operator Ae about `state` (device [n_nodes][2]);
 * D: device [NN]; l2g: device uint32 [n_elem][NN] */
int semk_stokes_linearize_f64(int n1, int64_t n_slot_elems, const double *D, const double *invJ,
                              const double *JxW, const double *x_phys, const uint32_t *l2g,
                              const int64_t *elem_of_slot, const double *state, double n_rey,
                              double *F, int64_t f_patch_stride, int elems_per_patch,
                              void *stream);
/* y = J u (assembled local Jacobians, no boundary conditions); with
 * zero_essential_rows != 0 the rows listed in ess_dof are zeroed afterwards (the
 * caller keeps the essential entries of u at zero: J restricted to the unknowns,
 * examples/squirmer-axisymmetric.py:362-370).  adv_scale multiplies the advection
 * terms: 1 = Jacobian, 0.5 with u = state = the nonlinear residual (the term is
 * bilinear).  u, y: distinct, 16-byte aligned.  Deterministic (no atomics). */
int semk_stokes_apply_f64(const semk_stokes_op *op, const double *u, double *y,
                          int zero_essential_rows, double adv_scale, void *stream);
/* element-local diagonals (engine slot order, [n_slot_elems][NN]) of Lve, E2e, Me and of
 * the advection block d row0 / d psi (locA may be NULL): inputs of the nodal 2x2
 * block-Jacobi preconditioner after semk_assemble_f64 */
int semk_stokes_local_diag_f64(const semk_stokes_op *op, const double *D_dev,
                               int64_t n_slot_elems, double *locL, double *locE, double *locM,
                               double *locA, void *stream);
/* y[idx[i]] = src ? src[idx[i]] : 0 */
int semk_scatter_fix_f64(int64_t n, const int64_t *idx, const double *src, double *y,
                         void *stream);

/* Glue of the Poisson block preconditioner of the Stokes system (stokes.py,
 * PoissonBlockPreconditioner): vectors src / t / y / dst are (psi, omega) pairs [n_nodes][2],
 * the others nodal [n_nodes].
 *   gamma : t = (0, nimg * src_omega)                      (om_G = -b_G / M_G)
 *   rhs   : which 0: r = src_psi - y_psi;  which 1: r = src_omega + coef * om;
 *           r = 0 outside free_mask;  f = r * inv_mass_int  (nodal load for semk_sc_element_*)
 *   out   : dst = (free ? psi : 0, free ? om_i : t_omega)
 *   semk_sc_rhs_finish_f64: b = dirichlet ? 0 : g + r over the element-exterior DOFs */
int semk_stokes_prec_gamma_f64(int64_t n_nodes, const double *src, const double *nimg, double *t,
                               void *stream);
int semk_stokes_prec_rhs_f64(int64_t n_nodes, int which, const double *src, const double *y,
                             const double *coef, const double *om, const uint8_t *free_mask,
                             const double *inv_mass_int, double *r, double *f, void *stream);
int semk_stokes_prec_out_f64(int64_t n_nodes, const uint8_t *free_mask, const double *psi,
                             const double *om_i, const double *t, double *dst, void *stream);
int semk_sc_rhs_finish_f64(int64_t n, const double *g, const double *r, const uint8_t *dirichlet,
                           double *b, void *stream);

/* Building blocks of the restarted GMRES that replaces the reference's sparse direct
 * solve of the non-symmetric system (examples/squirmer-axisymmetric.py:360-370):
 * out[j] = V_j . w for j < k with V_j = V + j*ldv (one pass, fixed-order reduction);
 * w += sign * sum_j h[j] V_j (h on the device); out = alpha a (+ b);
 * z_n = B_n r_n with nodal 2x2 blocks binv [n_nodes][4]. */
int64_t semk_multi_dot_partials_len(int k);
int semk_multi_dot_f64(int64_t n, int k, const double *V, int64_t ldv, const double *w,
                       double *out, double *partials, void *stream);
int semk_multi_axpy_f64(int64_t n, int k, const double *V, int64_t ldv, const double *h,
                        double sign, double *w, void *stream);
int semk_vec_scale_add_f64(int64_t n, double alpha, const double *a, const double *b,
                           double *out, void *stream);
int semk_block2_apply_f64(int64_t n_nodes, const double *binv, const double *r, double *z,
                          void *stream);

/* Block-vector kernels of the block eigensolver (eigen.py).  A block of m vectors of length n
 * is stored as rows X + i*ldx, i < m, ldx >= n; 1 <= m, k <= 96.
 *   semk_block_gram_f64    : G[i*k + j] = sum_t X[i*ldx + t] * w[t] * Y[j*ldy + t]   (w == NULL:
 *                            w = 1).  X, Y and w are read once; fixed per-CTA ranges, the last
 *                            CTA adds the partial matrices in CTA order: bitwise reproducible for
 *                            a given (n, m, k).  partials: semk_block_gram_partials_len(m, k)
 *                            doubles (-1 for m or k out of range), zero-filled once before the
 *                            first call; every call leaves it ready for the next one, of any
 *                            m' k' <= m k.
 *   semk_block_combine_f64 : Y[j] = beta * Y[j] + sum_i C[i*k + j] X[i], j < k (C [m][k] on the
 *                            device; Y must not overlap X; beta == 0 does not read Y). */
int64_t semk_block_gram_partials_len(int m, int k);
int semk_block_gram_f64(int64_t n, int m, const double *X, int64_t ldx, int k, const double *Y,
                        int64_t ldy, const double *w, double *G, double *partials, void *stream);
/* The same Gram matrix with the inner product fixed: DFMA (FP64 FMA) or DMMA (FP64 mma.sync
 * m8n8k4).  semk_block_gram_f64 is the one of the two that measured faster (DESIGN.md section 7);
 * each is bitwise reproducible on its own. */
int semk_block_gram_dfma_f64(int64_t n, int m, const double *X, int64_t ldx, int k,
                             const double *Y, int64_t ldy, const double *w, double *G,
                             double *partials, void *stream);
int semk_block_gram_dmma_f64(int64_t n, int m, const double *X, int64_t ldx, int k,
                             const double *Y, int64_t ldy, const double *w, double *G,
                             double *partials, void *stream);
int semk_block_combine_f64(int64_t n, int m, const double *X, int64_t ldx, int k, const double *C,
                           double beta, double *Y, int64_t ldy, void *stream);

/* A sub-range of semk_poisson_apply_f64: patches [patch_begin, patch_end) and the interface
 * entries [chunk_begin, chunk_end) / [rec_begin, rec_end).  Both interface tables are sorted
 * by the highest patch involved, so what patches [0, P) complete is a prefix of each
 * (SEMK_PA_CHUNK_MAXPATCH / SEMK_PA_REC_MAXPATCH).  No fused dot. */
int semk_poisson_apply_range_f64(const semk_op *op, const double *u, double *y, int flags,
                                 int64_t patch_begin, int64_t patch_end, int64_t chunk_begin,
                                 int64_t chunk_end, int64_t rec_begin, int64_t rec_end,
                                 void *stream);
/* y = A u on a strip partition with the interface exchange overlapped with the local apply
 * (SURVEY.md 8(e): "overlap with interior-element compute by processing interface elements
 * first"): the plan's patch sequence must start with the boundary tile columns, patches
 * [0, bnd_patch_end) with interface prefixes bnd_chunk_end / bnd_rec_end; they run first,
 * the exchange (semk_halo_exchange_f64, a 128-thread variant) runs on a high-priority side
 * stream while `stream` works through the remaining patches, then the streams join.
 * Advances halo->epoch.  dirichlet: device uint8 [n_nodes] or NULL. */
int semk_poisson_apply_halo_f64(const semk_op *op, const double *u, double *y, int flags,
                                int64_t bnd_patch_end, int64_t bnd_chunk_end, int64_t bnd_rec_end,
                                semk_halo *halo, const uint8_t *dirichlet, void *stream);

/* ------------------------------------------------------------------------
 * Host-side (no GPU) multi-threaded integer tables.
 * semk_host_sc_numbering: DOFManagerSC._do_static_condensation (sem/discrete.py:314-359) +
 * Mesh._permute_nodes (sem/discrete.py:1115-1127) for a homogeneous mesh, in place, bit-exact
 * with the reference's np.unique / np.sort numbering; SEMK_ERR_UNSUPPORTED = a mesh the fast
 * path does not cover (the caller falls back to the whole-array NumPy expressions).
 * semk_host_structured_maps: the node maps of the hand-built structured mesh of
 * tests/test_discrete.py:22-38 (node id = i*NY + j).  n_threads: 0 = all processors.
 * ------------------------------------------------------------------------ */
int semk_host_structured_maps(int64_t nx, int64_t ny, int32_t p, int64_t node_offset,
                              uint32_t *out, int32_t n_threads);
int semk_host_sc_numbering(int64_t n_nodes, int64_t n_cells, int32_t nn, uint32_t *maps,
                           const int32_t *ext_idx, int32_t n_ext_idx, const int32_t *int_idx,
                           int32_t n_int_idx, double *nodes, int32_t ndim, int64_t node_stride,
                           int64_t *n_ext_out, int64_t *n_int_out, uint32_t *order_out,
                           int32_t n_threads);

#ifdef __cplusplus
}
#endif
#endif /* SEMK_H */
