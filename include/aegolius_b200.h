/*
 * aegolius_b200.h — C ABI of libaegolius_b200.so (B200 / sm_100a evaluator for SPOMSO's SDF hot path).
 *
 * The reference (SPOMSO 1.4.0, pure Python) has no FFI: its boundary for this path is the Python method
 *   GenericGeometry.create(co) -> ndarray[(N,), f64]        Code/spomso/spomso/cores/geom.py:29-43
 *   GenericGeometry.propagate(co, *params)                  Code/spomso/spomso/cores/geom.py:45-60
 *   sdf_point_cloud_3d / sdf_point_cloud_2d(co, points)     Code/spomso/spomso/cores/sdf_3D.py:283-286, sdf_2D.py:221-224
 *   from_sdf(sdf, co_resolution)                            Code/spomso/spomso/cores/vector_functions.py:130-139
 * Each entry point below names the reference interface it replaces. The host side (Python, ctypes) flattens
 * the SPOMSO object tree into an `ab_program` (linear op list) and calls these functions; see INTEGRATION.md.
 *
 * Conventions: every function returns AB_OK (0) or a negative ab_status; the message for the last error of the
 * calling thread is returned by ab_last_error(). No exceptions cross the boundary. The caller owns every buffer.
 * `stream` is a cudaStream_t passed as void* (NULL = default stream). Device entry points are asynchronous on
 * `stream`; *_host entry points block until the result is in the host buffer.
 */
#ifndef AEGOLIUS_B200_H
#define AEGOLIUS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AB_VERSION 102 /* 0.1.2 */

typedef enum ab_status {
  AB_OK = 0,
  AB_EINVAL = -1,          /* bad argument / malformed program */
  AB_EUNSUPPORTED_OP = -2, /* opcode unknown to this build */
  AB_ECUDA = -3,           /* CUDA runtime error (message has the cudaError string) */
  AB_ETOOLARGE = -4,       /* program exceeds AB_MAX_OPS / AB_MAX_ARGS / slot limits */
  AB_ENODEVICE = -5        /* no CUDA device: there is NO CPU fallback */
} ab_status;

typedef enum ab_dtype { AB_F32 = 0, AB_F64 = 1 } ab_dtype;

/* What to compute besides the field value (forward-mode dual numbers inside the interpreter). */
typedef enum ab_grad_mode {
  AB_GRAD_NONE = 0,
  AB_GRAD_SPATIAL = 1, /* d field / d(x,y,z): analytic counterpart of from_sdf (vector_functions.py:130-139) */
  AB_GRAD_PARAM = 2    /* d field / d theta for one scalar parameter: replaces jacfwd(geometry, argnums=k),
                          Code/examples/autodiff/gradient_map_3D.py:84. ab_program.dargs holds d args / d theta; every
                          argument is read as a dual number and the tangent is propagated op by op (P_FIELD reads its
                          tangent from ab_program.dblobs). Limits: at most
                          AB_MAX_ARGS/2 arguments; table arguments (instance / vertex / sector tables, per-quadrant
                          radii, norm order) must have zero tangent (AB_EUNSUPPORTED_OP otherwise). */
} ab_grad_mode;

/* Limits of one program (it travels to the kernel as a __grid_constant__ parameter, i.e. constant bank 0). */
#define AB_MAX_OPS 640
#define AB_MAX_ARGS 2816
#define AB_MAX_PSLOTS 16
#define AB_MAX_VSLOTS 16
#define AB_MAX_BLOBS 4

/* One interpreter instruction (8 bytes). `a`/`b` are small immediates (slot numbers, axis, flags),
 * `arg` is the offset of this op's first argument in ab_program.args. */
typedef struct ab_op {
  uint16_t opcode;
  uint8_t a;
  uint8_t b;
  uint32_t arg;
} ab_op;

/* Opcodes. State per grid point: coordinate p=(x,y,z), accumulator acc, P-slots (saved coordinates),
 * V-slots (saved values). Reference semantics cited per group; exact formulas in DESIGN.md §3. */
typedef enum ab_opcode {
  AB_OP_END = 0,
  /* --- stack --- (children of a combine node all start from the parent's coordinates: combine.py:129-135) */
  AB_OP_SAVE_P = 1,  /* P[a] = p */
  AB_OP_LOAD_P = 2,  /* p = P[a] */
  AB_OP_PUSH_V = 3,  /* V[a] = acc */
  /* --- coordinate ops --- */
  AB_OP_AFFINE = 8,      /* 12 args M(3x3 row-major), b: p = M p + b. Folded apply_ec_transforms (transformations.py:232-242),
                            shear_* (modifications.py:579-774), rotate_sdf (:1308), mirror/linear_instancing frames (:978-985) */
  AB_OP_TRANSLATE = 9,   /* 3 args b: p = p + b (move_sdf :1268; pure moves) */
  AB_OP_SCALE_P = 10,    /* 1 arg k: p = p * k (rounding_cs :120-144, scale_sdf :1289) */
  AB_OP_ELONGATE = 11,   /* 6 args lo(3),hi(3): p -= min(max(p,lo),hi)  (elongation :75-98) */
  AB_OP_TWIST = 12,      /* 1 arg pitch (twist :502-527) */
  AB_OP_BEND = 13,       /* 8 args (bend :529-577) */
  AB_OP_ABSX_SUB = 14,   /* 1 arg h: x = |x| - h (mirror core :991-993) */
  AB_OP_SYMMETRY = 15,   /* a = axis: p[a] = |p[a]| (symmetry :932-955) */
  AB_OP_ROTSYM = 16,     /* 2 args angle, radius (rotational_symmetry :1020-1031, after its pre-rotation as AFFINE) */
  AB_OP_REVOLVE = 17,    /* 1 arg radius (revolution :411-436) */
  AB_OP_AXIS_REVOLVE = 18, /* 3 args radius, cos, sin (axis_revolution :438-472) */
  AB_OP_REP_INF = 19,    /* 6 args d(3), d/2(3) (infinite_repetition :803-825) */
  AB_OP_REP_FIN = 20,    /* 12 args c,d,s,s/2 (finite_repetition :827-873) */
  AB_OP_LIN_INST = 21,   /* a = (n>2); 6 args (linear_instancing :1035-1088, after its frame as AFFINE) */
  AB_OP_CURVE_INST = 22, /* a = mode (0 positions only, 1 positions + 3x3 frames); args: n, then n records
                            (curve_instancing :1090-1132, aligned :1134-1196, fully aligned :1198-1266) */
  AB_OP_ZERO_Z = 23,     /* z = 0 */
  /* fused forms emitted by the flattener's peephole pass (one dispatch instead of two or three):
     optional PUSH_V (b = V slot + 1, 0 = none), then p = f(P[a]) */
  AB_OP_NEXT_AFFINE = 24,    /* [V[b-1] = acc;] p = M P[a] + t   (PUSH_V + LOAD_P + AFFINE) */
  AB_OP_NEXT_TRANSLATE = 25, /* [V[b-1] = acc;] p = P[a] + t     (PUSH_V + LOAD_P + TRANSLATE) */
  AB_OP_NEXT_LOAD = 26,      /* [V[b-1] = acc;] p = P[a]         (PUSH_V + LOAD_P) */
  /* --- value ops --- */
  AB_OP_ROUND = 32,      /* acc -= r (rounding :100) */
  AB_OP_ABS = 33,        /* boundary :146 */
  AB_OP_NEG = 34,        /* invert :277 */
  AB_OP_SIGN = 35,       /* sign :301 */
  AB_OP_ONION = 36,      /* |acc| - t (onion :371) */
  AB_OP_CONCENTRIC = 37, /* |acc - h| (concentric :390) */
  AB_OP_SCALE_V = 38,    /* acc *= k (node scale, transformations.py:242) */
  AB_OP_EXTRUDE_BEGIN = 39, /* a = V slot; 1 arg h/2: V[a] = |z| - h/2 ; z = 0 (extrusion :474-500) */
  AB_OP_EXTRUDE_END = 40,   /* a = V slot */
  AB_OP_POLY_SIGN = 41,     /* acc *= interior sign of a planar polygon / polyline at the coordinates saved in P[a]; table: n, then
                               b = 0: n (x, y) vertices of a simple closed polygon, crossing-number rule (SegmentedLine.polygon(),
                               geom_2d.py:530-555, 601-626, triangulation_functions.py:390-430); b = 1: n segment records
                               (px, py, lx, ux, nx, ny), the x-interval / side-of-segment product of ParametricCurve.shape()
                               (geom_2d.py:415-457) restated term by term */
  /* post-processing value maps (post_processing.py:380-560; wrappers modifications.py:1361-1587) */
  AB_OP_PP_SIGMOID = 48, AB_OP_PP_POS_SIGMOID = 49, AB_OP_PP_CAPPED_EXP = 50, AB_OP_PP_HARD_BIN = 51,
  AB_OP_PP_LINEAR = 52, AB_OP_PP_RELU = 53, AB_OP_PP_SMOOTH_RELU = 54, AB_OP_PP_SLOWSTART = 55,
  AB_OP_PP_GAUSS_BOUNDARY = 56, AB_OP_PP_GAUSS_FALLOFF = 57,
  /* --- combine ops: acc = f(V[a], acc)  (combine.py:51-78); if b != 0 the result is also stored to V[b-1]
     (fused PUSH_V of a left-deep combine chain) --- */
  AB_OP_C_UNION = 64, AB_OP_C_INTERSECT = 65, AB_OP_C_SUBTRACT = 66, AB_OP_C_SUM = 67, AB_OP_C_DIFF = 68,
  AB_OP_C_SMIN2 = 69,     /* smoothmin_poly2, 1 arg w (combine.py:12-18) */
  AB_OP_C_SMIN3 = 70,     /* smoothmin_poly3 (combine.py:20-26) */
  AB_OP_C_SMAX3 = 71,     /* -smin3(-a,-b) */
  AB_OP_C_SSUB3 = 72,     /* -smin3(-a, b) */
  AB_OP_C_BOLTZ_INT = 73, /* smoothmax_boltz(a, b) (combine.py:29-34) */
  AB_OP_C_BOLTZ_SUB = 74, /* smoothmax_boltz(a,-b) */
  /* --- 3D primitives: acc = sdf(p) (sdf_3D.py) --- */
  AB_OP_P_SPHERE = 96, AB_OP_P_CYLINDER = 97, AB_OP_P_BOX = 98, AB_OP_P_TORUS = 99, AB_OP_P_CHAINLINK = 100,
  AB_OP_P_BRAID = 101, AB_OP_P_ARC3D = 102, AB_OP_P_PLANE = 103, AB_OP_P_UPLANE = 104, AB_OP_P_SEGMENT = 105,
  AB_OP_P_CONE = 106, AB_OP_P_OINF_CONE = 107, AB_OP_P_INF_CONE = 108, AB_OP_P_SOLID_ANGLE = 109,
  AB_OP_P_TRIANGLE3D = 110, AB_OP_P_QUAD3D = 111, AB_OP_P_SEGLINE = 112, AB_OP_P_AXIS = 113,
  AB_OP_P_POINT_CLOUD = 114, /* a = dim (2|3), b = blob index: nearest-point distance (sdf_3D.py:283-286) */
  AB_OP_P_FIELD = 115,       /* b = blob index of a DEVICE field (blob.dim = 1, one value of the evaluation dtype per point
                                of the call, indexed like `out`): value = field[point]. Carries the output of a grid
                                stencil (conv_averaging / conv_edge_detection / signed as a modification,
                                modifications.py:220-275, 1586-1637) back into the op list. Under AB_GRAD_PARAM the
                                tangent is ab_program.dblobs[b][point] (the stencil applied to the tangent of its input);
                                no spatial derivative passes through it */
  /* --- 2D primitives (sdf_2D.py), evaluated on (x,y) --- */
  AB_OP_P_CIRCLE = 128, AB_OP_P_NEU_CIRCLE = 129, AB_OP_P_BOX2D = 130, AB_OP_P_SEGMENT2D = 131,
  AB_OP_P_RBOX2D = 132, AB_OP_P_TRIANGLE2D = 133, AB_OP_P_ARC = 134, AB_OP_P_SECTOR = 135,
  AB_OP_P_INF_SECTOR = 136, AB_OP_P_NGON = 137, AB_OP_P_SEGLINE2D = 138,
  AB_OP_P_POLYGON2D = 139, /* simple polygon: min edge distance, sign by crossing number (sdf_2D.py:201-218) */
  AB_OP__COUNT = 160
} ab_opcode;

/* A point cloud referenced by an op. `data` is (3, count) row-major float64 on the host (SPOMSO's own layout,
 * geom_3d.py:759-777; 2D clouds carry a zero z row) when on_device == 0, or a device pointer to `count`
 * (x, y, z, 0) records of the evaluation dtype (float4 / double4) prepared by ab_cloud_upload when on_device == 1. */
typedef struct ab_blob {
  const void* data;
  uint64_t count;
  int32_t dim;
  int32_t on_device;
} ab_blob;

typedef struct ab_program {
  const ab_op* ops;
  uint32_t n_ops;
  const double* args;  /* fp64 pool; narrowed to fp32 by the library for AB_F32 */
  uint32_t n_args;
  const double* dargs; /* d args / d theta (AB_GRAD_PARAM only), same length as args, else NULL */
  const ab_blob* blobs;
  uint32_t n_blobs;
  uint32_t n_pslots;   /* P-slots used (<= AB_MAX_PSLOTS) */
  uint32_t n_vslots;   /* V-slots used (<= AB_MAX_VSLOTS) */
  const ab_blob* dblobs; /* NULL, or n_blobs entries: entry b is the DEVICE tangent row d field_b / d theta of a P_FIELD blob
                            (dim = 1, indexed and advanced exactly like blob b). AB_GRAD_PARAM needs one for every P_FIELD
                            blob the program reads; other entries and other modes ignore it */
} ab_program;

/* Regular grid exactly as generate_grid builds it (helper_functions.py:23-93): per axis
 * np.linspace(-size/2, size/2, res); flat index k = (ix*res[1] + iy)*res[2] + iz (z fastest).
 * 2D grids: res[2] = 1, size[2] = 0. The slab [slab_begin, slab_end) is a range of ix planes; outputs are
 * indexed from the slab's first point. */
typedef struct ab_grid {
  double size[3];
  uint32_t res[3];
  uint32_t slab_begin;
  uint32_t slab_end;
} ab_grid;

int ab_version(void);
const char* ab_last_error(void);
/* Number of CUDA devices visible (0 => every compute call returns AB_ENODEVICE). */
int ab_device_count(void);

/* Replaces GenericGeometry.create(co) for co produced by generate_grid (geom.py:29-43): coordinates are
 * regenerated in-kernel. out: device pointer, (slab points,) of dtype. out_grad: device pointer (3, grad_stride)
 * of dtype for AB_GRAD_SPATIAL, (1, grad_stride) for AB_GRAD_PARAM, NULL for AB_GRAD_NONE. */
int ab_eval_grid(const ab_program* prog, const ab_grid* grid, int dtype, int grad_mode, void* out, void* out_grad,
                 uint64_t grad_stride, int device, void* stream);

/* Replaces GenericGeometry.create(co) for arbitrary co (geom.py:29-43). co: DEVICE pointer (3, co_stride) of
 * co_dtype (SPOMSO hands in float64). */
int ab_eval_points(const ab_program* prog, const void* co, int co_dtype, uint64_t co_stride, uint64_t n, int dtype,
                   int grad_mode, void* out, void* out_grad, uint64_t grad_stride, int device, void* stream);

/* Fused least-squares objective for shape optimisation, the device counterpart of jax.value_and_grad(worker) in
 * Code/examples/autodiff/position_optimization.py:101-179: one AB_GRAD_PARAM evaluation (prog->dargs holds d args / d theta)
 * whose per-point results are not stored but reduced in the kernel:
 *   accum_dev[0] = sum_k (F_k - target_k)^2,   accum_dev[1] = sum_k 2 (F_k - target_k) dF_k/dtheta     (doubles, DEVICE)
 * target_dev: DEVICE array of `dtype`, one value per grid point of the slab. accum_dev is zeroed by the call. */
int ab_eval_grid_loss(const ab_program* prog, const ab_grid* grid, int dtype, const void* target_dev, double* accum_dev,
                      int device, void* stream);

/* Program-specialised kernels (optional). aegolius_b200/build.py can compile the interpreter with only the ops of one
 * program (csrc/ab_interp_spec.cu -> its own shared object exporting ab_spec_launch); registering that launcher here makes
 * every later evaluation whose ops are all in `op_mask` (AB_OP__COUNT bytes, 1 = compiled in) with the same dtype and
 * grad_mode use it instead of the general tiers (AB_GRAD_PARAM kernels also serve ab_eval_grid_loss). Same results,
 * smaller kernel. */
int ab_spec_register(int dtype, int grad_mode, const uint8_t* op_mask, uint32_t mask_len, void* launch_fn,
                     uint64_t kparams_size);
int ab_spec_clear(void);
/* Kernel tier an op needs: 0 lite, 1 mid, 2 full (the library runs a program on the smallest tier covering its ops). */
int ab_op_tier(int opcode);
uint64_t ab_spec_hits(void);

/* Program-compiled kernels (aegolius_b200/codegen.py): ONE straight-line kernel per program structure, generated from
 * the flattened op list (the evaluation order of geom.py:29-60 / modifications.py:88-98 / combine.py:115-163 unrolled
 * on the host), built by nvcc into its own shared object and registered here. `signature[i]` = opcode | a << 16 |
 * b << 24 of op i, for the n_sig ops before the terminator; `flavor` bit 0 = the binary serves 2D grids (else 3D grids and
 * point lists), bit 1 = it stores with multimem.st (ab_eval_grid_multicast), bit 2 = compact 16 x 16 tiles (whole planes of
 * 3D grids only; preferred there); `launch_fn` has the ab_spec_launch contract. Arguments still travel with every launch, so one binary
 * serves every parameter value. ab_eval_* prefer a registered program over the interpreter tiers; results are
 * bit-identical. ab_prog_enable(0) makes them ignore the registry (returns the previous setting). */
/* Multi-GPU field assembly without a gather pass (SURVEY §8e "optional all-gather of the assembled field"): `out_mc` /
 * `out_grad_mc` are MULTICAST addresses of a symmetric allocation that every rank of the node has mapped (NVLS over
 * NVSwitch), offset to this rank's slab. The rank evaluates its slab exactly like ab_eval_grid, but the kernel stores
 * with multimem.st, so each value lands in every GPU's copy of the field. Needs a program-compiled kernel built with the
 * multicast store path (flavor bit 1); AB_EUNSUPPORTED_OP otherwise. The caller synchronises the ranks afterwards. */
int ab_eval_grid_multicast(const ab_program* prog, const ab_grid* grid, int dtype, int grad_mode, void* out_mc,
                           void* out_grad_mc, uint64_t grad_stride, int device, void* stream);

int ab_prog_register(const uint32_t* signature, uint32_t n_sig, int dtype, int grad_mode, int flavor, void* launch_fn,
                     uint64_t kparams_size);
int ab_prog_clear(void);
uint64_t ab_prog_hits(void);
int ab_prog_enable(int on);
uint64_t ab_prog_signature_hash(const uint32_t* signature, uint32_t n_sig, int dtype, int grad_mode);
/* Host-only: offset of every op's arguments in the pool the kernels see (one entry per op before the terminator; fixed-size
 * ops first, tables last, each on a 4-scalar boundary) and the pool length. What a program-compiled kernel hard-codes. */
int ab_prog_arg_layout(const ab_program* prog, uint32_t* offsets_out, uint32_t* n_args_out);

/* Host-buffer variants (what the Python drop-in calls when the user wants a NumPy array back): allocate/reuse
 * device scratch, run, copy the result to `out_host` (pinned or pageable), synchronise. */
int ab_eval_grid_host(const ab_program* prog, const ab_grid* grid, int dtype, int grad_mode, void* out_host,
                      void* out_grad_host, uint64_t grad_stride, int device);
int ab_eval_points_host(const ab_program* prog, const double* co_host, uint64_t co_stride, uint64_t n, int dtype,
                        int grad_mode, void* out_host, void* out_grad_host, uint64_t grad_stride, int device);

/* Replaces sdf_point_cloud_3d / sdf_point_cloud_2d (sdf_3D.py:283-286, sdf_2D.py:221-224) on a grid: unsigned
 * distance to the nearest cloud point, exact (q-p)^2 form. cloud: DEVICE (x, y, z, 0) records from ab_cloud_upload.
 * Two exact paths that return identical bits: tiled brute force (small n*m) and an implicit octree / quadtree built
 * per call on `stream` (n*m >= 2^30; the reference asks a cKDTree). The environment variable AB_NN_ALGO=brute|tree
 * forces one of them (used by the parity tests). */
int ab_nn_grid(const void* cloud_dev, uint64_t m, int dim, const ab_grid* grid, int dtype, void* out, int device,
               void* stream);
int ab_nn_points(const void* cloud_dev, uint64_t m, int dim, const void* co, int co_dtype, uint64_t co_stride,
                 uint64_t n, int dtype, void* out, int device, void* stream);

/* Converts a host (dim, m) float64 cloud (row stride in elements) into device (x, y, z, 0) records of `dtype`;
 * *out_dev is cudaMalloc'ed (free with ab_device_free). */
int ab_cloud_upload(const double* points_host, uint64_t m, int dim, uint64_t row_stride, int dtype, int device,
                    void** out_dev);

/* ---- whole-field kernels that follow the SDF evaluation in SPOMSO pipelines (device pointers, asynchronous) ---- */

/* Replaces conv_averaging (post_processing.py:552-599): `iterations` passes of a box filter of ksize[3] samples over a
 * C-ordered field of res[3] samples (2D fields: res[2] = ksize[2] = 1); scipy.ndimage.convolve placement, mode
 * 'reflect'. field and out must not overlap. iterations == 0 copies. */
int ab_box_filter(const void* field_dev, const uint32_t res[3], const uint32_t ksize[3], uint32_t iterations, int dtype,
                  void* out_dev, int device, void* stream);
/* Replaces conv_edge_detection (post_processing.py:602-623): 9u - (3x3 sum over the first two axes), 'reflect'. */
int ab_edge_filter(const void* field_dev, const uint32_t res[3], int dtype, void* out_dev, int device, void* stream);
/* `signed` (modifications.py:220-275): turns an unsigned distance field on a 3D grid into a signed one. boundary = field <
 * threshold (the caller passes the smallest grid step, modifications.py:239-240); crossing parities along axes 0 and 1
 * (forward / flipped cumulative sums, :242-258), conv_averaging((2,2,1), 1) (:260), the outer layer takes its inner
 * neighbour (:262-263), field * (1 - 2 (interior > 1/2)) (:265-268). A field that already has a negative sample is
 * copied through (:234-235). Every axis needs >= 3 samples. Asynchronous on `stream`; out_dev != field_dev. */
int ab_signed_field(const void* field_dev, const uint32_t res[3], double threshold, int dtype, void* out_dev, int device,
                    void* stream);
/* The same, a slab at a time. ab_signed_mask packs the boundary mask (field < threshold) of a C-ordered block of res[3]
 * samples (planes of the field): bit (i2 % 32) of uint32 word [i0][i1][i2 / 32], rows padded to whole words, so the
 * masks of consecutive slabs concatenate into the mask of the field. It ORs 1 into flags_dev[0] when a sample is negative
 * and into flags_dev[1] when one is NaN (the caller zeroes the two ints). */
int ab_signed_mask(const void* field_dev, const uint32_t res[3], double threshold, int dtype, uint32_t* mask_dev,
                   int* flags_dev, int device, void* stream);
/* Planes [x0, x1) of the signed field of a field of res[3] samples, from the mask and flags of the WHOLE field and the
 * field's own values: field_dev holds planes [field_plane0, ...) (field_plane0 <= x0), out_dev receives planes [x0, x1).
 * The planes concatenate bit-identically to ab_signed_field. Every axis needs >= 3 samples. */
int ab_signed_field_slab(const uint32_t* mask_dev, const int* flags_dev, const void* field_dev, uint32_t field_plane0,
                         const uint32_t res[3], uint32_t x0, uint32_t x1, int dtype, void* out_dev, int device,
                         void* stream);
/* ab_signed_field_slab on a field and its parameter tangent at once (tangent_dev laid out like field_dev, out_tangent_dev
 * like out_dev): one interior and smoothing, then out = +-field and out_tangent = +-tangent with the same sign per sample.
 * The mask and flags come from the field's values only (the boundary mask is piecewise constant in the parameter); when the
 * field had a negative sample and no NaN both pass through unchanged. out_dev bit-identical to ab_signed_field_slab. */
int ab_signed_field_slab_tangent(const uint32_t* mask_dev, const int* flags_dev, const void* field_dev,
                                 const void* tangent_dev, uint32_t field_plane0, const uint32_t res[3], uint32_t x0,
                                 uint32_t x1, int dtype, void* out_dev, void* out_tangent_dev, int device, void* stream);

/* Vector-field modifiers (vector_modification_functions.py:14-172; methods modifications.py:1712-1971). */
#define AB_MAX_VEC_OPS 32
typedef enum ab_vec_opcode {
  AB_VOP_ADD = 1,       /* add_vectors        :23-28   operand 0: scalar | vec3 | (N,) | (3,N) */
  AB_VOP_SUB = 2,       /* subtract_vectors   :31-36 */
  AB_VOP_RESCALE = 3,   /* rescale_vectors    :39-41   operand 0: scalar | (N,) | (3,N) */
  AB_VOP_ROT_Z = 4,     /* rotate_vectors_z_axis :104-113 and rotate_vectors_phi :44-52; operand 0: angle scalar | (N,) */
  AB_VOP_ROT_THETA = 5, /* rotate_vectors_theta :55-69 */
  AB_VOP_ROT_X = 6,     /* :72-81 */
  AB_VOP_ROT_Y = 7,     /* :84-93 (the reference's sign convention) */
  AB_VOP_ROT_AXIS = 8,  /* rotate_vectors_axis :116-131; operand 0: axis vec3 | (3,N); operand 1: angle scalar | (N,) */
  AB_VOP_REVOLVE_X = 9, /* revolve_field_x :134-146; operand 0: coordinates (3,N) */
  AB_VOP_REVOLVE_Y = 10,
  AB_VOP_REVOLVE_Z = 11,
  AB_VOP_NORMALIZE = 12 /* batch_normalize :14-20 */
} ab_vec_opcode;
typedef enum ab_vec_kind { AB_VK_NONE = 0, AB_VK_SCALAR = 1, AB_VK_VEC3 = 2, AB_VK_ARRAY = 3, AB_VK_VEC_ARRAY = 4 } ab_vec_kind;
typedef struct ab_vec_op {
  uint32_t opcode;
  uint32_t kind0, kind1;
  double c[3];        /* AB_VK_VEC3 operand */
  double s0, s1;      /* AB_VK_SCALAR operands */
  const void* a0;     /* DEVICE arrays of `dtype`: (N,) for AB_VK_ARRAY, (3, stride) for AB_VK_VEC_ARRAY */
  const void* a1;
  uint64_t stride0, stride1;
} ab_vec_op;
/* Applies ops[0..n_ops) in order to the (3, vec_stride) field in place, one pass over memory. */
int ab_vec_apply(void* vec_dev, uint64_t vec_stride, uint64_t n, const ab_vec_op* ops, uint32_t n_ops, int dtype,
                 int device, void* stream);
typedef enum ab_vec_component_id { AB_VC_X = 0, AB_VC_Y = 1, AB_VC_Z = 2, AB_VC_PHI = 3, AB_VC_THETA = 4, AB_VC_LENGTH = 5 } ab_vec_component_id;
/* VectorField.x/y/z/phi/theta/length (geom.py:262-362): phi = atan2(y, x), theta = acos(z), length = |v|. */
int ab_vec_component(const void* vec_dev, uint64_t vec_stride, uint64_t n, int what, int dtype, void* out_dev,
                     int device, void* stream);

/* Replaces from_sdf (vector_functions.py:130-139): np.gradient of the reshaped field (unit spacing, 2nd-order
 * central inside, 1st-order one-sided on the faces) and, if normalize != 0, batch_normalize
 * (vector_modification_functions.py:14-20). field: DEVICE (points of the whole grid) of dtype; out: DEVICE
 * (dims, out_stride). The slab selects which ix planes are written (halo planes are read from `field`, which
 * must hold planes [max(slab_begin-1,0), min(slab_end+1,res0)) starting at `field_plane0`). */
int ab_fd_gradient(const void* field, uint32_t field_plane0, const ab_grid* grid, int dims, int dtype, int normalize,
                   void* out, uint64_t out_stride, int device, void* stream);

/* Device / pinned-host memory helpers for callers without their own CUDA allocator (ctypes users). */
int ab_device_alloc(uint64_t bytes, int device, void** out_dev);
int ab_device_free(void* dev, int device);
int ab_host_alloc_pinned(uint64_t bytes, void** out_host);
/* flags: bit 0 = cudaHostAllocPortable, bit 1 = cudaHostAllocWriteCombined. */
int ab_host_alloc_pinned_flags(uint64_t bytes, unsigned flags, void** out_host);
int ab_host_free_pinned(void* host);
int ab_memcpy_d2h(void* dst_host, const void* src_dev, uint64_t bytes, int device, void* stream);
int ab_memcpy_h2d(void* dst_dev, const void* src_host, uint64_t bytes, int device, void* stream);
int ab_stream_sync(int device, void* stream);

/* Number of kernels this library has launched in the calling process (bench.py's gpu_launches). */
uint64_t ab_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* AEGOLIUS_B200_H */
