// ab_capi.cu — the C ABI of libaegolius_b200.so (see include/aegolius_b200.h for the contract and the reference
// interfaces each entry point replaces). Plain pointers and sizes in, status codes out; no torch types.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <type_traits>
#include <unordered_map>
#include <vector>

#include "ab_kernels_aux.cuh"
#include "ab_nn_tree.cuh"
#include "ab_fields.cuh"

using namespace ab;

// ---- error handling ---------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
#define CUDA_TRY(expr)                                                                        \
  do {                                                                                        \
    cudaError_t e_ = (expr);                                                                  \
    if (e_ != cudaSuccess) return fail(AB_ECUDA, "%s: %s", #expr, cudaGetErrorString(e_));    \
  } while (0)

extern "C" int ab_version(void) { return AB_VERSION; }
extern "C" const char* ab_last_error(void) { return g_err; }
extern "C" uint64_t ab_launch_count(void) { return g_launches.load(); }
extern "C" int ab_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

static int use_device(int device) {
  int n = ab_device_count();
  if (n == 0) return fail(AB_ENODEVICE, "no CUDA device visible: aegolius_b200 has no CPU fallback");
  if (device < 0 || device >= n) return fail(AB_EINVAL, "device %d out of range (have %d)", device, n);
  CUDA_TRY(cudaSetDevice(device));
  return AB_OK;
}

struct DevInfo {
  int sms = 0;
  size_t smem_optin = 0;
  bool ok = false;
};
static DevInfo g_dev[64];
static std::mutex g_dev_mu;
static int dev_info(int device, DevInfo& out) {
  std::lock_guard<std::mutex> lk(g_dev_mu);
  if (!g_dev[device].ok) {
    cudaDeviceProp p;
    CUDA_TRY(cudaGetDeviceProperties(&p, device));
    g_dev[device].sms = p.multiProcessorCount;
    g_dev[device].smem_optin = p.sharedMemPerBlockOptin;
    // stream-ordered scratch (the octree of ab_nn_tree.cuh) stays in the pool between calls instead of going back to the
    // driver at every synchronisation
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
      uint64_t keep = ~0ull;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    g_dev[device].ok = true;
  }
  out = g_dev[device];
  return AB_OK;
}

// ---- program validation ---------------------------------------------------------------------------------------------------
static int op_arg_count(const ab_op& op, const double* args, uint32_t n_args, int* out) {
  int n = -1;
  switch (op.opcode) {
    case AB_OP_END: case AB_OP_SAVE_P: case AB_OP_LOAD_P: case AB_OP_PUSH_V: case AB_OP_SYMMETRY: case AB_OP_ZERO_Z:
    case AB_OP_ABS: case AB_OP_NEG: case AB_OP_SIGN: case AB_OP_EXTRUDE_END: case AB_OP_C_UNION: case AB_OP_C_INTERSECT:
    case AB_OP_NEXT_LOAD:
    case AB_OP_C_SUBTRACT: case AB_OP_C_SUM: case AB_OP_C_DIFF: case AB_OP_P_POINT_CLOUD: case AB_OP_P_FIELD:
      n = 0; break;
    case AB_OP_SCALE_P: case AB_OP_TWIST: case AB_OP_ABSX_SUB: case AB_OP_REVOLVE: case AB_OP_ROUND: case AB_OP_ONION:
    case AB_OP_CONCENTRIC: case AB_OP_SCALE_V: case AB_OP_EXTRUDE_BEGIN: case AB_OP_PP_HARD_BIN: case AB_OP_PP_RELU:
    case AB_OP_C_SMIN2: case AB_OP_C_SMIN3: case AB_OP_C_SMAX3: case AB_OP_C_SSUB3: case AB_OP_C_BOLTZ_INT:
    case AB_OP_C_BOLTZ_SUB: case AB_OP_P_SPHERE: case AB_OP_P_AXIS: case AB_OP_P_CIRCLE:
      n = 1; break;
    case AB_OP_PP_SIGMOID: case AB_OP_PP_POS_SIGMOID: case AB_OP_PP_CAPPED_EXP: case AB_OP_PP_LINEAR:
    case AB_OP_PP_SMOOTH_RELU: case AB_OP_PP_GAUSS_BOUNDARY: case AB_OP_PP_GAUSS_FALLOFF: case AB_OP_P_CYLINDER:
    case AB_OP_P_TORUS: case AB_OP_P_OINF_CONE: case AB_OP_P_INF_CONE: case AB_OP_P_NEU_CIRCLE: case AB_OP_P_BOX2D:
      n = 2; break;
    case AB_OP_TRANSLATE: case AB_OP_NEXT_TRANSLATE: case AB_OP_AXIS_REVOLVE: case AB_OP_PP_SLOWSTART: case AB_OP_P_BOX: case AB_OP_P_CHAINLINK:
      n = 3; break;
    case AB_OP_P_BRAID: case AB_OP_P_PLANE: case AB_OP_P_UPLANE: case AB_OP_P_CONE: case AB_OP_P_ARC:
      n = 4; break;
    case AB_OP_P_ARC3D: case AB_OP_P_SEGMENT2D: case AB_OP_P_INF_SECTOR: n = 5; break;
    case AB_OP_ELONGATE: case AB_OP_REP_INF: case AB_OP_LIN_INST: case AB_OP_P_SOLID_ANGLE: case AB_OP_P_RBOX2D:
    case AB_OP_P_SECTOR:
      n = 6; break;
    case AB_OP_P_SEGMENT: case AB_OP_P_NGON: n = 7; break;
    case AB_OP_BEND: n = 8; break;
    case AB_OP_AFFINE: case AB_OP_NEXT_AFFINE: case AB_OP_REP_FIN: n = 12; break;
    case AB_OP_P_TRIANGLE2D: n = 16; break;
    case AB_OP_P_TRIANGLE3D: n = 34; break;
    case AB_OP_P_QUAD3D: n = 44; break;
    case AB_OP_ROTSYM: {
      if ((uint64_t)op.arg + 4 > n_args) return fail(AB_EINVAL, "ROTSYM header out of range");
      double c = args[op.arg + 2];
      if (!(c >= 1) || c > 1024 || c != (double)(int)c) return fail(AB_EINVAL, "bad ROTSYM sector count %g", c);
      n = 4 + 2 * (int)c;
    } break;
    case AB_OP_CURVE_INST: case AB_OP_P_SEGLINE: case AB_OP_P_SEGLINE2D: case AB_OP_P_POLYGON2D: case AB_OP_POLY_SIGN: {
      if (op.arg >= n_args) return fail(AB_EINVAL, "op argument offset out of range");
      double c = args[op.arg];
      if (!(c >= 0) || c > 1e6) return fail(AB_EINVAL, "bad element count %g", c);
      int per = op.opcode == AB_OP_CURVE_INST ? (op.a ? 12 : 3) : (op.opcode == AB_OP_P_SEGLINE ? 3 : 2);
      if (op.opcode == AB_OP_POLY_SIGN) per = op.b ? 6 : 2;
      n = (op.opcode == AB_OP_CURVE_INST ? 4 : 1) + (int)c * per;
    } break;
    default: return fail(AB_EUNSUPPORTED_OP, "opcode %u is not supported by this build", (unsigned)op.opcode);
  }
  *out = n;
  return AB_OK;
}

static int validate(const ab_program* prog) {
  if (!prog || !prog->ops || (prog->n_args && !prog->args)) return fail(AB_EINVAL, "null program");
  if (prog->n_ops == 0) return fail(AB_EINVAL, "empty program");
  if (prog->n_ops > AB_MAX_OPS || prog->n_args > AB_MAX_ARGS)
    return fail(AB_ETOOLARGE, "program too large: %u ops / %u args (limits %d / %d)", prog->n_ops, prog->n_args,
                AB_MAX_OPS, AB_MAX_ARGS);
  if (prog->n_pslots > AB_MAX_PSLOTS || prog->n_vslots > AB_MAX_VSLOTS)
    return fail(AB_ETOOLARGE, "too many stack slots (%u P, %u V)", prog->n_pslots, prog->n_vslots);
  if (prog->n_blobs > AB_MAX_BLOBS) return fail(AB_ETOOLARGE, "too many blobs");
  bool have_value = false;
  for (uint32_t i = 0; i < prog->n_ops; i++) {
    const ab_op& op = prog->ops[i];
    int n = 0;
    int rc = op_arg_count(op, prog->args, prog->n_args, &n);
    if (rc) return rc;
    if (n > 0 && (uint64_t)op.arg + n > prog->n_args) return fail(AB_EINVAL, "op %u reads past the argument pool", i);
    switch (op.opcode) {
      case AB_OP_SAVE_P: case AB_OP_LOAD_P:
        if (op.a >= prog->n_pslots) return fail(AB_EINVAL, "op %u: P slot %u >= n_pslots %u", i, op.a, prog->n_pslots);
        break;
      case AB_OP_POLY_SIGN:
        if (op.a >= prog->n_pslots) return fail(AB_EINVAL, "op %u: P slot %u >= n_pslots %u", i, op.a, prog->n_pslots);
        if (op.b > 1) return fail(AB_EINVAL, "op %u: POLY_SIGN rule %u", i, op.b);
        break;
      case AB_OP_NEXT_AFFINE: case AB_OP_NEXT_TRANSLATE: case AB_OP_NEXT_LOAD:
        if (op.a >= prog->n_pslots) return fail(AB_EINVAL, "op %u: P slot %u >= n_pslots %u", i, op.a, prog->n_pslots);
        if (op.b > prog->n_vslots) return fail(AB_EINVAL, "op %u: fused V slot %u > n_vslots %u", i, op.b, prog->n_vslots);
        break;
      case AB_OP_PUSH_V: case AB_OP_EXTRUDE_BEGIN: case AB_OP_EXTRUDE_END:
        if (op.a >= prog->n_vslots) return fail(AB_EINVAL, "op %u: V slot %u >= n_vslots %u", i, op.a, prog->n_vslots);
        break;
      case AB_OP_P_POINT_CLOUD:
        if (op.b >= prog->n_blobs || !prog->blobs) return fail(AB_EINVAL, "op %u: blob %u missing", i, op.b);
        if (op.a != 2 && op.a != 3) return fail(AB_EINVAL, "op %u: point cloud dim must be 2 or 3", i);
        if (prog->blobs[op.b].count == 0 || prog->blobs[op.b].count > 0xffffffffull)
          return fail(AB_EINVAL, "op %u: point cloud size out of range", i);
        break;
      case AB_OP_P_FIELD:
        if (op.b >= prog->n_blobs || !prog->blobs) return fail(AB_EINVAL, "op %u: blob %u missing", i, op.b);
        if (prog->blobs[op.b].dim != 1 || !prog->blobs[op.b].on_device || !prog->blobs[op.b].data)
          return fail(AB_EINVAL, "op %u: P_FIELD needs a device blob with dim = 1", i);
        break;
      case AB_OP_SYMMETRY: case AB_OP_P_AXIS:
        if (op.a > 2) return fail(AB_EINVAL, "op %u: axis %u", i, op.a);
        break;
      default:
        if (op.opcode >= AB_OP_C_UNION && op.opcode <= AB_OP_C_BOLTZ_SUB &&
            (op.a >= prog->n_vslots || op.b > prog->n_vslots))
          return fail(AB_EINVAL, "op %u: V slot out of range (a %u, b %u, n_vslots %u)", i, op.a, op.b, prog->n_vslots);
    }
    if (op.opcode >= AB_OP_P_SPHERE) have_value = true;
    if (op.opcode == AB_OP_END) break;
  }
  if (!have_value) return fail(AB_EINVAL, "program has no primitive");
  return AB_OK;
}

// ---- grid description -> kernel form ---------------------------------------------------------------------------------------
static int make_gridk(const ab_grid* grid, GridK& g, uint64_t* n_points) {
  if (!grid) return fail(AB_EINVAL, "null grid");
  for (int c = 0; c < 3; c++)
    if (grid->res[c] == 0) return fail(AB_EINVAL, "grid resolution of 0");
  if (grid->slab_begin >= grid->slab_end || grid->slab_end > grid->res[0])
    return fail(AB_EINVAL, "bad slab [%u, %u) for res0 %u", grid->slab_begin, grid->slab_end, grid->res[0]);
  // 2D grids (res[2] == 1) are remapped to index axes (1, nx, ny) so that the fast index axis is y and a thread's run
  // of consecutive points stays inside one row; parameter sets 1 and 2 then describe x and y, z is +0
  const bool is2d = grid->res[2] == 1 && grid->res[1] > 1 && grid->size[2] == 0.0;
  const uint32_t n1 = is2d ? grid->res[0] : grid->res[1];
  const uint32_t n2 = is2d ? grid->res[1] : grid->res[2];
  const uint64_t plane = (uint64_t)n1 * n2;  // 2D: the whole grid is one "plane" of index axis 0
  if (plane > 0x7fffffffull) return fail(AB_ETOOLARGE, "one grid plane has more than 2^31 points");
  g.n1 = n1;
  g.n2 = n2;
  g.plane = (uint32_t)plane;
  g.is2d = is2d ? 1u : 0u;
  g.i0_begin = is2d ? 0u : grid->slab_begin;
  g.i1_begin = is2d ? grid->slab_begin : 0u;
  g.m1 = (uint32_t)(0x100000000ull / n1 > 0xffffffffull ? 0xffffffffull : 0x100000000ull / n1);
  g.m2 = (uint32_t)(0x100000000ull / n2 > 0xffffffffull ? 0xffffffffull : 0x100000000ull / n2);
  for (int c = 0; c < 3; c++) {
    // parameter set c describes index axis c: (x, y, z) in 3D, (unused, x, y) in 2D
    int src = is2d ? c - 1 : c;
    uint32_t n = src >= 0 ? grid->res[src] : 1;
    double sz = src >= 0 ? grid->size[src] : 0.0;
    double start = -sz / 2, stop = sz / 2;
    double step = n > 1 ? (stop - start) / (double)(n - 1) : 0.0;  // np.linspace: delta / div
    g.last[c] = n - 1;
    g.start[c] = start;
    g.stop[c] = n > 1 ? stop : start + 0.0;
    if (n == 1) g.stop[c] = (sz == 0.0) ? 0.0 : start;  // linspace(a, b, 1) == [a]; 2D grids: z = +0
    g.step[c] = step;
    g.hi[c] = (float)step;
    g.lo[c] = (float)(step - (double)g.hi[c]);
    g.centre[c] = (float)((double)(n - 1) * 0.5);
  }
  *n_points = (uint64_t)(grid->slab_end - grid->slab_begin) * (is2d ? (uint64_t)n2 : plane);
  return AB_OK;
}

// ---- blobs (point clouds) ---------------------------------------------------------------------------------------------------
template <typename T>
static int upload_cloud(const double* pts, uint64_t m, int dim, uint64_t row_stride, cudaStream_t st, void** out_dev,
                        bool async) {
  typedef typename Vec4<T>::type V4;
  std::vector<V4> rec(m);
  for (uint64_t i = 0; i < m; i++) {
    rec[i].x = (T)pts[i];
    rec[i].y = (T)pts[row_stride + i];
    rec[i].z = dim == 3 ? (T)pts[2 * row_stride + i] : (T)0;
    rec[i].w = (T)0;
  }
  void* d = nullptr;
  if (async) {
    CUDA_TRY(cudaMallocAsync(&d, m * sizeof(V4), st));
    CUDA_TRY(cudaMemcpyAsync(d, rec.data(), m * sizeof(V4), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));  // rec is a stack-lifetime staging buffer
  } else {
    CUDA_TRY(cudaMalloc(&d, m * sizeof(V4)));
    CUDA_TRY(cudaMemcpy(d, rec.data(), m * sizeof(V4), cudaMemcpyHostToDevice));
    // a copy from pageable memory returns once the data is STAGED; the DMA into `d` may still be in flight, and the
    // consumers run on non-blocking streams that do not order themselves after the legacy stream: wait for it here
    CUDA_TRY(cudaStreamSynchronize(cudaStreamLegacy));
  }
  *out_dev = d;
  return AB_OK;
}

extern "C" int ab_cloud_upload(const double* points_host, uint64_t m, int dim, uint64_t row_stride, int dtype,
                               int device, void** out_dev) {
  if (!points_host || !out_dev || m == 0 || (dim != 2 && dim != 3)) return fail(AB_EINVAL, "bad cloud arguments");
  int rc = use_device(device);
  if (rc) return rc;
  return dtype == AB_F64 ? upload_cloud<double>(points_host, m, dim, row_stride, 0, out_dev, false)
                         : upload_cloud<float>(points_host, m, dim, row_stride, 0, out_dev, false);
}

// clouds of at least this many points get an octree when they are a leaf of a program
static const uint64_t kTreeLeafMin = 2048;
template <typename T>
static int build_tree(const typename Vec4<T>::type* cloud, uint32_t m, int dim, const DevInfo& di, cudaStream_t st,
                      void** buf_out, const TreeRef<T>** ref_out);

// ---- interpreter launch ----------------------------------------------------------------------------------------------------

// arguments that the kernels read as plain tables (no tangent): see raw_args() uses in ab_ops.cuh
static bool structural_arg(int opcode, int k) {
  switch (opcode) {
    case AB_OP_ROTSYM: return k != 1;  // everything but the radius
    case AB_OP_CURVE_INST: case AB_OP_P_SEGLINE: case AB_OP_P_SEGLINE2D: case AB_OP_P_POLYGON2D: case AB_OP_POLY_SIGN: case AB_OP_P_TRIANGLE3D:
    case AB_OP_P_QUAD3D: case AB_OP_P_TRIANGLE2D: case AB_OP_P_RBOX2D:
      return true;
    case AB_OP_P_NEU_CIRCLE: return k == 1;  // the norm order
    default: return false;
  }
}

template <typename T>
struct EvalTarget {
  int grid_mode;
  GridK g;
  const void* co;
  uint64_t co_stride;
  int co_is_f64;
  uint64_t n;
  T* out;
  T* grad;
  uint64_t grad_stride;
  const T* target;     // loss mode (ab_eval_grid_loss): no per-point outputs
  double* loss_accum;
  int multicast;       // out / grad are multicast addresses: only a program-compiled kernel built for multimem.st may run
};

template <typename S, typename T>
static int dispatch_nt(const KParams<T>& kp, int device, cudaStream_t st) {
  DevInfo di;
  int rc = dev_info(device, di);
  if (rc) return rc;
  LaunchCfg cfg{di.sms, di.smem_optin};
  int status = AB_OK;
  cudaError_t e;
  constexpr bool kHasOwnLite = !std::is_same<S, Pack<float, 4>>::value && !std::is_same<S, Dual<Pack<float, 2>, 3>>::value;
  if (kp.tier == 0 && kHasOwnLite) {
    // (fp32 lite programs never get here: run_program sends them to the wider lite kernels)
    if constexpr (kHasOwnLite) e = launch_interp<S, T, 0>(kp, cfg, st, &status);
    else e = cudaErrorInvalidValue;
  } else if (kp.tier <= 1) {
    if constexpr (sizeof(T) == 4) e = launch_interp<S, T, 1>(kp, cfg, st, &status);
    else e = launch_interp<S, T, 2>(kp, cfg, st, &status);  // fp64 has no mid-tier build
  } else e = launch_interp<S, T, 2>(kp, cfg, st, &status);
  if (e != cudaSuccess) return fail(AB_ECUDA, "interpreter launch: %s", cudaGetErrorString(e));
  if (status != AB_OK) return fail(status, "interpreter stacks (%u P, %u V slots) do not fit in shared memory", kp.n_pslots, kp.n_vslots);
  g_launches++;
  return AB_OK;
}

// ---- program-specialised kernels (ab_interp_spec.cu, built on request) ------------------------------------------------------
typedef int (*ab_spec_fn)(const void*, int, unsigned long long, void*, int*);
struct SpecEntry {
  int dtype, grad_mode;
  uint8_t mask[AB_OP__COUNT];  // ops compiled into the kernel
  ab_spec_fn fn;
};
static std::vector<SpecEntry> g_specs;
static std::mutex g_spec_mu;
static std::atomic<uint64_t> g_spec_hits{0};
static std::atomic<uint64_t> g_prog_hits{0};

extern "C" int ab_spec_register(int dtype, int grad_mode, const uint8_t* op_mask, uint32_t mask_len, void* launch_fn,
                                uint64_t kparams_size) {
  if (!op_mask || !launch_fn || mask_len != AB_OP__COUNT) return fail(AB_EINVAL, "bad specialisation descriptor");
  if (dtype != AB_F32 && dtype != AB_F64) return fail(AB_EINVAL, "bad dtype %d", dtype);
  if (grad_mode != AB_GRAD_NONE && grad_mode != AB_GRAD_SPATIAL && grad_mode != AB_GRAD_PARAM) return fail(AB_EINVAL, "bad grad_mode %d", grad_mode);
  const uint64_t want = dtype == AB_F32 ? sizeof(KParams<float>) : sizeof(KParams<double>);
  if (kparams_size != want) return fail(AB_EINVAL, "specialised kernel built against another library version (KParams %llu != %llu bytes)", (unsigned long long)kparams_size, (unsigned long long)want);
  SpecEntry e{};
  e.dtype = dtype;
  e.grad_mode = grad_mode;
  memcpy(e.mask, op_mask, AB_OP__COUNT);
  e.fn = (ab_spec_fn)launch_fn;
  std::lock_guard<std::mutex> lk(g_spec_mu);
  g_specs.insert(g_specs.begin(), e);  // newest first
  return AB_OK;
}
extern "C" int ab_op_tier(int opcode) { return (opcode < 0 || opcode >= AB_OP__COUNT) ? -1 : op_tier(opcode); }
extern "C" int ab_spec_clear(void) {
  std::lock_guard<std::mutex> lk(g_spec_mu);
  g_specs.clear();
  return AB_OK;
}
extern "C" uint64_t ab_spec_hits(void) { return g_spec_hits.load(); }

static ab_spec_fn find_spec(const ab_program* prog, int dtype, int grad_mode) {
  std::lock_guard<std::mutex> lk(g_spec_mu);
  for (const SpecEntry& e : g_specs) {
    if (e.dtype != dtype || e.grad_mode != grad_mode) continue;
    bool ok = true;
    for (uint32_t i = 0; i < prog->n_ops && ok; i++) ok = prog->ops[i].opcode < AB_OP__COUNT && e.mask[prog->ops[i].opcode];
    if (ok) return e.fn;
  }
  return nullptr;
}

template <typename T>
static int dispatch_spec(ab_spec_fn fn, const KParams<T>& kp, int device, cudaStream_t st, std::atomic<uint64_t>& hits) {
  DevInfo di;
  int rc = dev_info(device, di);
  if (rc) return rc;
  int status = AB_OK;
  const cudaError_t e = (cudaError_t)fn(&kp, di.sms, (unsigned long long)di.smem_optin, st, &status);
  if (e != cudaSuccess) return fail(AB_ECUDA, "specialised interpreter launch: %s", cudaGetErrorString(e));
  if (status != AB_OK) return fail(status, "interpreter stacks (%u P, %u V slots) do not fit in shared memory", kp.n_pslots, kp.n_vslots);
  g_launches++;
  hits++;
  return AB_OK;
}


// ---- program-compiled kernels (aegolius_b200/codegen.py) ------------------------------------------------------------------------
// One straight-line kernel per program STRUCTURE: the sequence of (opcode, a, b) before the terminator. Arguments still
// travel in KParams at every launch, so a parameter sweep or an optimisation loop reuses one binary. The generated shared
// object exports a launcher with the signature of ab_spec_fn; it is registered here under the structure's signature and
// run_program prefers it over the interpreter tiers. Same op bodies, same arithmetic: results are bit-identical.
struct ProgEntry {
  int dtype, grad_mode;  // grad_mode | flavor << 8; flavor bit 0: the binary serves 2D grids (else 3D grids and point lists),
                         // bit 1: it stores through multimem.st (outputs are multicast addresses, ab_eval_grid_multicast),
                         // bit 2: compact 16 x 16 tiles (whole planes of 3D grids only; preferred there when registered)
  std::vector<uint32_t> sig;
  ab_spec_fn fn;
};
static std::unordered_map<uint64_t, std::vector<ProgEntry>> g_progs;
static std::mutex g_prog_mu;
static std::atomic<int> g_prog_enabled{1};

static uint64_t sig_hash(const uint32_t* sig, uint32_t n, int dtype, int grad_mode) {
  uint64_t h = 1469598103934665603ull;  // FNV-1a over the signature words, dtype and gradient mode
  auto mix = [&](uint32_t w) {
    for (int k = 0; k < 4; k++) {
      h ^= (w >> (8 * k)) & 0xffu;
      h *= 1099511628211ull;
    }
  };
  for (uint32_t i = 0; i < n; i++) mix(sig[i]);
  mix((uint32_t)dtype);
  mix((uint32_t)grad_mode);
  return h;
}

extern "C" uint64_t ab_prog_signature_hash(const uint32_t* signature, uint32_t n_sig, int dtype, int grad_mode) {
  return (signature && n_sig <= AB_MAX_OPS) ? sig_hash(signature, n_sig, dtype, grad_mode) : 0;
}

extern "C" int ab_prog_register(const uint32_t* signature, uint32_t n_sig, int dtype, int grad_mode, int flavor,
                                void* launch_fn, uint64_t kparams_size) {
  if (!signature || n_sig == 0 || n_sig > AB_MAX_OPS || !launch_fn) return fail(AB_EINVAL, "bad compiled-program descriptor");
  if (dtype != AB_F32 && dtype != AB_F64) return fail(AB_EINVAL, "bad dtype %d", dtype);
  if (grad_mode != AB_GRAD_NONE && grad_mode != AB_GRAD_SPATIAL && grad_mode != AB_GRAD_PARAM) return fail(AB_EINVAL, "bad grad_mode %d", grad_mode);
  if (flavor < 0 || flavor > 7 || ((flavor & 4) && (flavor & 1))) return fail(AB_EINVAL, "bad flavor %d", flavor);
  grad_mode |= flavor << 8;
  const uint64_t want = dtype == AB_F32 ? sizeof(KParams<float>) : sizeof(KParams<double>);
  if (kparams_size != want) return fail(AB_EINVAL, "compiled program built against another library version (KParams %llu != %llu bytes)", (unsigned long long)kparams_size, (unsigned long long)want);
  ProgEntry e;
  e.dtype = dtype;
  e.grad_mode = grad_mode;
  e.sig.assign(signature, signature + n_sig);
  e.fn = (ab_spec_fn)launch_fn;
  std::lock_guard<std::mutex> lk(g_prog_mu);
  auto& bucket = g_progs[sig_hash(signature, n_sig, dtype, grad_mode)];
  for (ProgEntry& o : bucket)
    if (o.dtype == dtype && o.grad_mode == grad_mode && o.sig == e.sig) {
      o.fn = e.fn;  // re-registration replaces the launcher
      return AB_OK;
    }
  bucket.push_back(std::move(e));
  return AB_OK;
}
extern "C" int ab_prog_clear(void) {
  std::lock_guard<std::mutex> lk(g_prog_mu);
  g_progs.clear();
  return AB_OK;
}
extern "C" uint64_t ab_prog_hits(void) { return g_prog_hits.load(); }
// 0: run_program ignores the registered compiled kernels (tests compare them against the interpreter); returns the old value
extern "C" int ab_prog_enable(int on) { return g_prog_enabled.exchange(on ? 1 : 0); }

static ab_spec_fn find_prog(const ab_program* prog, uint32_t n_ops, int dtype, int grad_mode, int flavor) {
  if (!g_prog_enabled.load()) return nullptr;
  grad_mode |= flavor << 8;
  uint32_t sig[AB_MAX_OPS];
  for (uint32_t i = 0; i < n_ops; i++)
    sig[i] = (uint32_t)prog->ops[i].opcode | ((uint32_t)prog->ops[i].a << 16) | ((uint32_t)prog->ops[i].b << 24);
  const uint64_t h = sig_hash(sig, n_ops, dtype, grad_mode);
  std::lock_guard<std::mutex> lk(g_prog_mu);
  auto it = g_progs.find(h);
  if (it == g_progs.end()) return nullptr;
  for (const ProgEntry& e : it->second)
    if (e.dtype == dtype && e.grad_mode == grad_mode && e.sig.size() == n_ops && !memcmp(e.sig.data(), sig, n_ops * 4)) return e.fn;
  return nullptr;
}

template <typename S, typename T, int TIER, bool PARAM = false>
static int dispatch_fixed(const KParams<T>& kp, int device, cudaStream_t st) {
  DevInfo di;
  int rc = dev_info(device, di);
  if (rc) return rc;
  LaunchCfg cfg{di.sms, di.smem_optin};
  int status = AB_OK;
  cudaError_t e = launch_interp<S, T, TIER, PARAM>(kp, cfg, st, &status);
  if (e != cudaSuccess) return fail(AB_ECUDA, "interpreter launch: %s", cudaGetErrorString(e));
  if (status != AB_OK) return fail(status, "interpreter stacks (%u P, %u V slots) do not fit in shared memory", kp.n_pslots, kp.n_vslots);
  g_launches++;
  return AB_OK;
}


// Offsets of every op's arguments in the kernel's repacked pool: each op on a 16-byte boundary (vector loads from shared
// memory); first the ops with a fixed argument count, in program order, then the tables (instance records, sector tables,
// polylines ...). The offsets of the fixed ones then depend on the op sequence alone, which is what lets a
// program-compiled kernel (codegen.py) address them as compile-time constants of the constant bank.
static int arg_layout(const ab_program* prog, uint32_t n_ops, uint32_t* offsets, int* counts, uint32_t* total) {
  uint32_t cursor = 0;
  for (int pass = 0; pass < 2; pass++) {
    for (uint32_t i = 0; i < n_ops; i++) {
      if ((int)is_table_op(prog->ops[i].opcode) != pass) continue;
      int cnt = 0;
      int rc = op_arg_count(prog->ops[i], prog->args, prog->n_args, &cnt);
      if (rc) return rc;
      if (cursor + (uint32_t)cnt + 4 > AB_MAX_ARGS)
        return fail(AB_ETOOLARGE, "program arguments exceed %d after alignment", AB_MAX_ARGS);
      offsets[i] = cursor;
      if (counts) counts[i] = cnt;
      cursor = (cursor + (uint32_t)cnt + 3u) & ~3u;
    }
  }
  *total = cursor;
  return AB_OK;
}

// host-only view of the layout above (tests compare it with codegen.fixed_arg_offsets)
extern "C" int ab_prog_arg_layout(const ab_program* prog, uint32_t* offsets_out, uint32_t* n_args_out) {
  int rc = validate(prog);
  if (rc) return rc;
  if (!offsets_out || !n_args_out) return fail(AB_EINVAL, "null pointer");
  uint32_t n_ops = prog->n_ops;
  while (n_ops > 0 && prog->ops[n_ops - 1].opcode == AB_OP_END) n_ops--;
  return arg_layout(prog, n_ops, offsets_out, nullptr, n_args_out);
}

template <typename T>
static int run_program(const ab_program* prog, const EvalTarget<T>& tg, int grad_mode, int device, cudaStream_t st) {
  int rc = validate(prog);
  if (rc) return rc;
  if (tg.n == 0) return AB_OK;
  const bool loss_mode = tg.loss_accum != nullptr;
  if (!loss_mode && !tg.out) return fail(AB_EINVAL, "null output pointer");
  if (grad_mode != AB_GRAD_NONE && grad_mode != AB_GRAD_SPATIAL && grad_mode != AB_GRAD_PARAM)
    return fail(AB_EINVAL, "bad grad_mode %d", grad_mode);
  if (!loss_mode && grad_mode != AB_GRAD_NONE && (!tg.grad || tg.grad_stride < tg.n))
    return fail(AB_EINVAL, "gradient output missing or grad_stride < n");
  if (grad_mode == AB_GRAD_PARAM && !prog->dargs) return fail(AB_EINVAL, "AB_GRAD_PARAM needs ab_program.dargs");

  static thread_local KParams<T> kp;  // ~28 KB: keep it off the stack
  kp.n = tg.n;
  kp.out = tg.out;
  kp.grad = tg.grad;
  kp.grad_stride = tg.grad_stride;
  kp.co = tg.co;
  kp.co_stride = tg.co_stride;
  kp.co_is_f64 = tg.co_is_f64;
  kp.grid_mode = tg.grid_mode;
  kp.g = tg.g;
  kp.n_ops = prog->n_ops;
  while (kp.n_ops > 0 && prog->ops[kp.n_ops - 1].opcode == AB_OP_END) kp.n_ops--;  // no dispatch spent on the terminator
  kp.n_pslots = prog->n_pslots ? prog->n_pslots : 1;
  kp.n_vslots = prog->n_vslots ? prog->n_vslots : 1;
  kp.tier = 0;
  for (uint32_t i = 0; i < kp.n_ops; i++) {
    const int t = op_tier(prog->ops[i].opcode);
    if (t > kp.tier) kp.tier = t;
  }
  // repack the arguments into the kernel's pool (layout: arg_layout above)
  uint32_t cursor = 0;
  {
    static thread_local uint32_t offs[AB_MAX_OPS];
    static thread_local int cnts[AB_MAX_OPS];
    rc = arg_layout(prog, kp.n_ops, offs, cnts, &cursor);
    if (rc) return rc;
    if (grad_mode == AB_GRAD_PARAM && cursor + 4 > kParamHalf)
      return fail(AB_ETOOLARGE, "program arguments exceed %u in parameter-tangent mode", kParamHalf);
    for (uint32_t i = 0; i < kp.n_ops; i++) {
      const uint32_t dense = (uint32_t)dense_opcode(prog->ops[i].opcode);  // validated above
      const uint32_t off = offs[i];
      const int cnt = cnts[i];
      kp.ops[i] = make_uint2(dense, off | ((uint32_t)prog->ops[i].a << 16) | ((uint32_t)prog->ops[i].b << 24));
      for (int k = 0; k < cnt; k++) kp.args[off + k] = (T)prog->args[prog->ops[i].arg + k];
      if (grad_mode == AB_GRAD_PARAM) {
        // tangents of the arguments go to the upper half of the pool; table-driven ops are structural (their tables are
        // read without tangents), so a parameter that reaches one of them cannot be differentiated here
        for (int k = 0; k < cnt; k++) {
          const double dk = prog->dargs[prog->ops[i].arg + k];
          kp.args[kParamHalf + off + k] = (T)dk;
          if (dk != 0.0 && structural_arg(prog->ops[i].opcode, k))
            return fail(AB_EUNSUPPORTED_OP, "op %u (opcode %u): the differentiated parameter reaches a table argument (index %d); "
                        "parameter tangents through instance / vertex / sector tables are not supported", i,
                        (unsigned)prog->ops[i].opcode, k);
        }
      }
    }
  }
  kp.n_args = grad_mode == AB_GRAD_PARAM ? kParamHalf + cursor : cursor;
  kp.dargs_off = grad_mode == AB_GRAD_PARAM ? kParamHalf : 0;

  std::vector<void*> temp_blobs;
  const char* field_base[AB_MAX_BLOBS] = {nullptr, nullptr, nullptr, nullptr};
  const char* dfield_base[AB_MAX_BLOBS] = {nullptr, nullptr, nullptr, nullptr};
  static_assert(AB_MAX_BLOBS == 4, "field_base initialiser");
  for (uint32_t b = 0; b < AB_MAX_BLOBS; b++) {
    kp.blob[b] = nullptr;
    kp.blob_count[b] = 0;
    kp.blob_tree[b] = nullptr;
    kp.dblob[b] = nullptr;
  }
  bool blob_used[AB_MAX_BLOBS] = {false, false, false, false};
  for (uint32_t i = 0; i < prog->n_ops; i++)
    if (prog->ops[i].opcode == AB_OP_P_POINT_CLOUD || prog->ops[i].opcode == AB_OP_P_FIELD) blob_used[prog->ops[i].b] = true;
  for (uint32_t b = 0; b < prog->n_blobs; b++) {
    const ab_blob& bl = prog->blobs[b];
    if (!blob_used[b]) continue;  // e.g. the not-yet-computed field of a later stencil stage in a prefix program
    if (bl.dim == 1) {  // a per-point field (P_FIELD): used in place, advanced with the output pointer per launch
      if (!bl.data || !bl.on_device || bl.count < tg.n) return fail(AB_EINVAL, "field blob %u must be a device array of >= %llu values", b, (unsigned long long)tg.n);
      if (grad_mode == AB_GRAD_SPATIAL) return fail(AB_EUNSUPPORTED_OP, "no derivative passes through a grid stencil (P_FIELD, blob %u)", b);
      field_base[b] = (const char*)bl.data;
      kp.blob[b] = bl.data;
      kp.blob_count[b] = 0;
      if (grad_mode == AB_GRAD_PARAM) {  // the stencil's tangent row, bound and advanced like the field
        const ab_blob* db = prog->dblobs ? &prog->dblobs[b] : nullptr;
        if (!db || !db->data || !db->on_device || db->dim != 1 || db->count < tg.n)
          return fail(AB_EINVAL, "AB_GRAD_PARAM: field blob %u needs a device tangent row (ab_program.dblobs) of >= %llu values", b,
                      (unsigned long long)tg.n);
        dfield_base[b] = (const char*)db->data;
        kp.dblob[b] = db->data;
      }
      continue;
    }
    if (!bl.data || bl.count == 0 || bl.count > 0xffffffffull) return fail(AB_EINVAL, "blob %u empty or too large", b);
    if (bl.on_device) {
      kp.blob[b] = bl.data;
    } else {
      void* d = nullptr;
      rc = upload_cloud<T>((const double*)bl.data, bl.count, 3, bl.count, st, &d, true);
      if (rc) return rc;
      temp_blobs.push_back(d);
      kp.blob[b] = d;
    }
    kp.blob_count[b] = (uint32_t)bl.count;
    // large clouds: the leaf walks an octree instead of scanning the blob (dimension = that of the leaf using the blob)
    if (bl.count >= kTreeLeafMin) {
      int bdim = 3;
      for (uint32_t i = 0; i < prog->n_ops; i++)
        if (prog->ops[i].opcode == AB_OP_P_POINT_CLOUD && prog->ops[i].b == b) bdim = prog->ops[i].a == 2 ? 2 : 3;
      DevInfo di;
      rc = dev_info(device, di);
      if (rc) return rc;
      void* tbuf = nullptr;
      const TreeRef<T>* ref = nullptr;
      rc = build_tree<T>((const typename Vec4<T>::type*)kp.blob[b], (uint32_t)bl.count, bdim, di, st, &tbuf, &ref);
      if (tbuf) temp_blobs.push_back(tbuf);
      if (rc) {
        for (void* d : temp_blobs) cudaFreeAsync(d, st);
        return rc;
      }
      kp.blob_tree[b] = ref;
    }
  }

  // a registered program-specialised kernel that covers every op of this program takes precedence over the tiers
  const int base_flavor = ((tg.grid_mode && tg.g.is2d) ? 1 : 0) | (tg.multicast ? 2 : 0);
  ab_spec_fn compiled = nullptr;
  if (tg.grid_mode && !tg.g.is2d && !loss_mode)  // whole planes of a 3D grid: the compact-tile build, if there is one
    compiled = find_prog(prog, kp.n_ops, sizeof(T) == 4 ? AB_F32 : AB_F64, grad_mode, base_flavor | 4);
  if (!compiled) compiled = find_prog(prog, kp.n_ops, sizeof(T) == 4 ? AB_F32 : AB_F64, grad_mode, base_flavor);
  if (tg.multicast && !compiled)
    return fail(AB_EUNSUPPORTED_OP, "no multicast-store kernel is registered for this program structure (build it with "
                "aegolius_b200.codegen.ensure(..., multicast=True)); the interpreter tiers store to one GPU only");
  const ab_spec_fn spec = compiled ? nullptr : find_spec(prog, sizeof(T) == 4 ? AB_F32 : AB_F64, grad_mode);
  constexpr int WV = sizeof(T) == 4 ? 4 : 2;  // one 128-bit store per thread
  constexpr int WG = sizeof(T) == 4 ? 2 : 1;  // dual numbers carry 4x the state: halve the points per thread
  // the kernel indexes points with 32 bits: split big jobs into launches of < 2^31 points (whole planes in grid mode)
  const uint64_t kMax = 0x7fffffffull - 4096;
  uint64_t done = 0;
  rc = AB_OK;
  while (done < tg.n && rc == AB_OK) {
    uint64_t chunk = tg.n - done;
    if (chunk > kMax) {
      chunk = kMax;
      if (tg.grid_mode) {
        const uint64_t unit = tg.g.is2d ? tg.g.n2 : tg.g.plane;  // whole ix planes (rows of y in 2D)
        uint64_t planes = kMax / unit;
        if (planes == 0) return fail(AB_ETOOLARGE, "one grid plane has more than 2^31 points");
        chunk = planes * unit;
      } else {
        chunk &= ~3ull;
      }
    }
    kp.n = chunk;
    kp.out = tg.out ? tg.out + done : nullptr;
    kp.grad = tg.grad ? tg.grad + done : nullptr;
    kp.target = tg.target ? tg.target + done : nullptr;
    kp.loss_accum = tg.loss_accum;
    for (uint32_t b = 0; b < AB_MAX_BLOBS; b++)
      if (field_base[b]) {
        kp.blob[b] = field_base[b] + done * sizeof(T);
        if (dfield_base[b]) kp.dblob[b] = dfield_base[b] + done * sizeof(T);
      }
    if (tg.grid_mode) {
      if (tg.g.is2d) kp.g.i1_begin = tg.g.i1_begin + (uint32_t)(done / tg.g.n2);
      else kp.g.i0_begin = tg.g.i0_begin + (uint32_t)(done / tg.g.plane);
    } else {
      kp.co = (const char*)tg.co + done * (tg.co_is_f64 ? 8 : 4);
    }
    if (compiled) rc = dispatch_spec<T>(compiled, kp, device, st, g_prog_hits);
    else if (spec) rc = dispatch_spec<T>(spec, kp, device, st, g_spec_hits);
    else if (grad_mode == AB_GRAD_NONE) {
      if constexpr (sizeof(T) == 4) {
        // lite programs are cheap per op, so 8 points per thread (two 128-bit stores) halve the per-point dispatch and
        // index overhead at still < 100 registers
        if (kp.tier == 0) rc = dispatch_fixed<Pack<T, 8>, T, 0>(kp, device, st);
        else rc = dispatch_nt<Pack<T, WV>, T>(kp, device, st);
      } else rc = dispatch_nt<Pack<T, WV>, T>(kp, device, st);
    }
    else if (grad_mode == AB_GRAD_SPATIAL) {
      if constexpr (sizeof(T) == 4) {
        if (kp.tier == 0) rc = dispatch_fixed<Dual<Pack<T, 4>, 3>, T, 0>(kp, device, st);  // lite: 4 points per thread
        else rc = dispatch_nt<Dual<Pack<T, WG>, 3>, T>(kp, device, st);
      } else rc = dispatch_nt<Dual<Pack<T, WG>, 3>, T>(kp, device, st);
    }
    else rc = dispatch_fixed<Dual<Pack<T, WG>, 1>, T, 2, true>(kp, device, st);
    done += chunk;
  }
  for (void* d : temp_blobs) cudaFreeAsync(d, st);
  return rc;
}

template <typename T>
static int eval_grid_t(const ab_program* prog, const ab_grid* grid, int grad_mode, void* out, void* out_grad,
                       uint64_t grad_stride, int device, cudaStream_t st, int multicast = 0) {
  EvalTarget<T> tg{};
  tg.multicast = multicast;
  int rc = make_gridk(grid, tg.g, &tg.n);
  if (rc) return rc;
  tg.grid_mode = 1;
  tg.out = (T*)out;
  tg.grad = (T*)out_grad;
  tg.grad_stride = grad_stride;
  return run_program<T>(prog, tg, grad_mode, device, st);
}

template <typename T>
static int eval_grid_loss_t(const ab_program* prog, const ab_grid* grid, const void* target, double* accum, int device,
                            cudaStream_t st) {
  EvalTarget<T> tg{};
  int rc = make_gridk(grid, tg.g, &tg.n);
  if (rc) return rc;
  tg.grid_mode = 1;
  tg.target = (const T*)target;
  tg.loss_accum = accum;
  CUDA_TRY(cudaMemsetAsync(accum, 0, 2 * sizeof(double), st));
  return run_program<T>(prog, tg, AB_GRAD_PARAM, device, st);
}

extern "C" int ab_eval_grid_loss(const ab_program* prog, const ab_grid* grid, int dtype, const void* target_dev,
                                 double* accum_dev, int device, void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  if (!target_dev || !accum_dev) return fail(AB_EINVAL, "null pointer");
  if (dtype == AB_F32) return eval_grid_loss_t<float>(prog, grid, target_dev, accum_dev, device, (cudaStream_t)stream);
  if (dtype == AB_F64) return eval_grid_loss_t<double>(prog, grid, target_dev, accum_dev, device, (cudaStream_t)stream);
  return fail(AB_EINVAL, "bad dtype %d", dtype);
}

extern "C" int ab_eval_grid(const ab_program* prog, const ab_grid* grid, int dtype, int grad_mode, void* out,
                            void* out_grad, uint64_t grad_stride, int device, void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  if (dtype == AB_F32) return eval_grid_t<float>(prog, grid, grad_mode, out, out_grad, grad_stride, device, (cudaStream_t)stream);
  if (dtype == AB_F64) return eval_grid_t<double>(prog, grid, grad_mode, out, out_grad, grad_stride, device, (cudaStream_t)stream);
  return fail(AB_EINVAL, "bad dtype %d", dtype);
}

extern "C" int ab_eval_grid_multicast(const ab_program* prog, const ab_grid* grid, int dtype, int grad_mode, void* out_mc,
                                      void* out_grad_mc, uint64_t grad_stride, int device, void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  if (grad_mode == AB_GRAD_PARAM) return fail(AB_EINVAL, "ab_eval_grid_multicast: AB_GRAD_NONE or AB_GRAD_SPATIAL");
  if (dtype == AB_F32) return eval_grid_t<float>(prog, grid, grad_mode, out_mc, out_grad_mc, grad_stride, device, (cudaStream_t)stream, 1);
  if (dtype == AB_F64) return eval_grid_t<double>(prog, grid, grad_mode, out_mc, out_grad_mc, grad_stride, device, (cudaStream_t)stream, 1);
  return fail(AB_EINVAL, "bad dtype %d", dtype);
}

template <typename T>
static int eval_points_t(const ab_program* prog, const void* co, int co_dtype, uint64_t co_stride, uint64_t n,
                         int grad_mode, void* out, void* out_grad, uint64_t grad_stride, int device, cudaStream_t st) {
  if (n && !co) return fail(AB_EINVAL, "null coordinates");
  if (co_stride < n) return fail(AB_EINVAL, "co_stride < n");
  EvalTarget<T> tg{};
  tg.grid_mode = 0;
  tg.co = co;
  tg.co_stride = co_stride;
  tg.co_is_f64 = co_dtype == AB_F64;
  tg.n = n;
  tg.out = (T*)out;
  tg.grad = (T*)out_grad;
  tg.grad_stride = grad_stride;
  return run_program<T>(prog, tg, grad_mode, device, st);
}

extern "C" int ab_eval_points(const ab_program* prog, const void* co, int co_dtype, uint64_t co_stride, uint64_t n,
                              int dtype, int grad_mode, void* out, void* out_grad, uint64_t grad_stride, int device,
                              void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  if (co_dtype != AB_F32 && co_dtype != AB_F64) return fail(AB_EINVAL, "bad co_dtype %d", co_dtype);
  if (dtype == AB_F32)
    return eval_points_t<float>(prog, co, co_dtype, co_stride, n, grad_mode, out, out_grad, grad_stride, device, (cudaStream_t)stream);
  if (dtype == AB_F64)
    return eval_points_t<double>(prog, co, co_dtype, co_stride, n, grad_mode, out, out_grad, grad_stride, device, (cudaStream_t)stream);
  return fail(AB_EINVAL, "bad dtype %d", dtype);
}

// ---- host-buffer variants: per-device scratch, result copied back --------------------------------------------------------------
struct Scratch {
  void* p = nullptr;
  size_t cap = 0;
};
static Scratch g_scratch[64][3];
static std::mutex g_scratch_mu;
static int scratch(int device, int which, size_t bytes, void** out) {
  Scratch& s = g_scratch[device][which];
  if (s.cap < bytes) {
    if (s.p) cudaFree(s.p);
    s.p = nullptr;
    s.cap = 0;
    CUDA_TRY(cudaMalloc(&s.p, bytes));
    s.cap = bytes;
  }
  *out = s.p;
  return AB_OK;
}

static int grad_rows(int grad_mode) { return grad_mode == AB_GRAD_SPATIAL ? 3 : (grad_mode == AB_GRAD_PARAM ? 1 : 0); }

// Pipelined host variant: the slab is cut into chunks of whole planes; chunk i+1 is evaluated on the compute stream
// while chunk i travels device->host on the copy stream (double-buffered scratch, events in both directions), so the
// PCIe copy, which dominates end to end, is the only thing left on the critical path.
struct Pipe {
  cudaStream_t comp = nullptr, copy = nullptr;
  cudaEvent_t done[2] = {nullptr, nullptr}, freed[2] = {nullptr, nullptr};
  bool ok = false;
};
static Pipe g_pipe[64];
static int pipe_for(int device, Pipe** out) {
  Pipe& p = g_pipe[device];
  if (!p.ok) {
    CUDA_TRY(cudaStreamCreateWithFlags(&p.comp, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&p.copy, cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) {
      CUDA_TRY(cudaEventCreateWithFlags(&p.done[i], cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&p.freed[i], cudaEventDisableTiming));
    }
    p.ok = true;
  }
  *out = &p;
  return AB_OK;
}

extern "C" int ab_eval_grid_host(const ab_program* prog, const ab_grid* grid, int dtype, int grad_mode, void* out_host,
                                 void* out_grad_host, uint64_t grad_stride, int device) {
  int rc = use_device(device);
  if (rc) return rc;
  if (dtype != AB_F32 && dtype != AB_F64) return fail(AB_EINVAL, "bad dtype %d", dtype);
  GridK g;
  uint64_t n = 0;
  rc = make_gridk(grid, g, &n);
  if (rc) return rc;
  if (!out_host) return fail(AB_EINVAL, "null output pointer");
  std::lock_guard<std::mutex> lk(g_scratch_mu);
  const size_t es = dtype == AB_F32 ? 4 : 8;
  const int rows = grad_rows(grad_mode);
  if (rows && (!out_grad_host || grad_stride < n)) return fail(AB_EINVAL, "gradient output missing or grad_stride < n");
  Pipe* pp = nullptr;
  rc = pipe_for(device, &pp);
  if (rc) return rc;
  // chunk = whole planes, about 256 MB of output each (at least one plane, at most the slab)
  const uint64_t plane = g.is2d ? g.n2 : g.plane;  // one ix plane (a row of y in 2D)
  const uint64_t bytes_per_plane = plane * es * (1 + rows);
  uint64_t planes_per_chunk = (256ull << 20) / (bytes_per_plane ? bytes_per_plane : 1);
  if (planes_per_chunk < 1) planes_per_chunk = 1;
  const uint64_t total_planes = grid->slab_end - grid->slab_begin;
  if (planes_per_chunk > total_planes) planes_per_chunk = total_planes;
  const uint64_t chunk_pts = planes_per_chunk * plane;
  const uint64_t dstride = (chunk_pts + 7) & ~7ull;  // rows 32-byte aligned against each other (whole-sector stores)
  void* d_out[2] = {nullptr, nullptr};
  void* d_grad[2] = {nullptr, nullptr};
  void* base = nullptr;
  const size_t per_buf = (size_t)dstride * es * (1 + rows);
  rc = scratch(device, 0, per_buf * 2, &base);
  if (rc) return rc;
  for (int b = 0; b < 2; b++) {
    d_out[b] = (char*)base + b * per_buf;
    d_grad[b] = rows ? (char*)d_out[b] + (size_t)dstride * es : nullptr;
  }
  // host blobs (point clouds) go to the device ONCE, before the chunk loop: per chunk they would be re-staged and re-uploaded
  // with a blocking copy, which serialises the compute / copy pipeline
  ab_program dprog = *prog;
  std::vector<ab_blob> dblobs(prog->blobs ? prog->blobs : nullptr, prog->blobs ? prog->blobs + prog->n_blobs : nullptr);
  std::vector<void*> uploaded;
  auto release = [&]() {
    for (void* d : uploaded) cudaFree(d);
  };
  for (uint32_t b = 0; b < prog->n_blobs && prog->blobs; b++) {
    ab_blob& bl = dblobs[b];
    if (bl.on_device || bl.dim == 1 || !bl.data || bl.count == 0 || bl.count > 0xffffffffull) continue;
    void* d = nullptr;
    rc = dtype == AB_F64 ? upload_cloud<double>((const double*)bl.data, bl.count, 3, bl.count, 0, &d, false)
                         : upload_cloud<float>((const double*)bl.data, bl.count, 3, bl.count, 0, &d, false);
    if (rc) {
      release();
      return rc;
    }
    uploaded.push_back(d);
    bl.data = d;
    bl.on_device = 1;
  }
  if (!dblobs.empty()) dprog.blobs = dblobs.data();
  uint64_t done_planes = 0;
  int c = 0;
  rc = AB_OK;
  cudaError_t ce = cudaSuccess;
  while (done_planes < total_planes && rc == AB_OK && ce == cudaSuccess) {
    const uint64_t np = (total_planes - done_planes < planes_per_chunk) ? total_planes - done_planes : planes_per_chunk;
    const uint64_t pts = np * plane, off = done_planes * plane;
    const int b = c & 1;
    ab_grid sub = *grid;
    sub.slab_begin = grid->slab_begin + (uint32_t)done_planes;
    sub.slab_end = sub.slab_begin + (uint32_t)np;
    if (c >= 2) ce = cudaStreamWaitEvent(pp->comp, pp->freed[b], 0);
    if (ce != cudaSuccess) break;
    rc = ab_eval_grid(&dprog, &sub, dtype, grad_mode, d_out[b], d_grad[b], dstride, device, pp->comp);
    if (rc) break;
    if ((ce = cudaEventRecord(pp->done[b], pp->comp)) != cudaSuccess) break;
    if ((ce = cudaStreamWaitEvent(pp->copy, pp->done[b], 0)) != cudaSuccess) break;
    if ((ce = cudaMemcpyAsync((char*)out_host + off * es, d_out[b], pts * es, cudaMemcpyDeviceToHost, pp->copy)) != cudaSuccess) break;
    if (rows)  // all gradient rows of the chunk in one strided copy
      if ((ce = cudaMemcpy2DAsync((char*)out_grad_host + off * es, (size_t)grad_stride * es, d_grad[b], (size_t)dstride * es,
                                  pts * es, rows, cudaMemcpyDeviceToHost, pp->copy)) != cudaSuccess) break;
    if ((ce = cudaEventRecord(pp->freed[b], pp->copy)) != cudaSuccess) break;
    done_planes += np;
    c++;
  }
  // also on the error paths: no copy may still be writing into the caller's buffers when this function returns
  const cudaError_t se = cudaStreamSynchronize(pp->copy);
  cudaStreamSynchronize(pp->comp);
  release();
  if (rc) return rc;
  if (ce != cudaSuccess) return fail(AB_ECUDA, "host pipeline: %s", cudaGetErrorString(ce));
  if (se != cudaSuccess) return fail(AB_ECUDA, "host pipeline: %s", cudaGetErrorString(se));
  return AB_OK;
}

extern "C" int ab_eval_points_host(const ab_program* prog, const double* co_host, uint64_t co_stride, uint64_t n,
                                   int dtype, int grad_mode, void* out_host, void* out_grad_host, uint64_t grad_stride,
                                   int device) {
  int rc = use_device(device);
  if (rc) return rc;
  if (dtype != AB_F32 && dtype != AB_F64) return fail(AB_EINVAL, "bad dtype %d", dtype);
  if (n == 0) return validate(prog);
  if (!co_host || !out_host) return fail(AB_EINVAL, "null pointer");
  if (co_stride < n) return fail(AB_EINVAL, "co_stride < n");
  std::lock_guard<std::mutex> lk(g_scratch_mu);
  const size_t es = dtype == AB_F32 ? 4 : 8;
  const int rows = grad_rows(grad_mode);
  if (rows && (!out_grad_host || grad_stride < n)) return fail(AB_EINVAL, "gradient output missing or grad_stride < n");
  const uint64_t dstride = (n + 7) & ~7ull;
  void *d_out = nullptr, *d_grad = nullptr, *d_co = nullptr;
  rc = scratch(device, 0, n * es, &d_out);
  if (rc) return rc;
  rc = scratch(device, 2, 3 * n * 8, &d_co);
  if (rc) return rc;
  if (rows) {
    rc = scratch(device, 1, dstride * rows * es, &d_grad);
    if (rc) return rc;
  }
  for (int r = 0; r < 3; r++)
    CUDA_TRY(cudaMemcpyAsync((double*)d_co + (size_t)r * n, co_host + (size_t)r * co_stride, n * 8, cudaMemcpyHostToDevice, 0));
  rc = ab_eval_points(prog, d_co, AB_F64, n, n, dtype, grad_mode, d_out, d_grad, dstride, device, nullptr);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(out_host, d_out, n * es, cudaMemcpyDeviceToHost, 0));
  for (int r = 0; r < rows; r++)
    CUDA_TRY(cudaMemcpyAsync((char*)out_grad_host + (size_t)r * grad_stride * es, (char*)d_grad + (size_t)r * dstride * es,
                             n * es, cudaMemcpyDeviceToHost, 0));
  CUDA_TRY(cudaStreamSynchronize(0));
  return AB_OK;
}

// ---- point cloud -> distance field -------------------------------------------------------------------------------------------
template <typename T, int Q, int TILE>
static int launch_nn(const NNParams<T>& kp, int device, cudaStream_t st) {
  DevInfo di;
  int rc = dev_info(device, di);
  if (rc) return rc;
  constexpr int NT = 256;
  void (*kern)(NNParams<T>);
  if constexpr (sizeof(T) == 4) kern = ab_nn_kernel_f32x2<Q, NT, TILE>;
  else kern = ab_nn_kernel<T, Q, NT, TILE>;
  int occ = 0;
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NT, 0));
  if (occ < 1) occ = 1;
  const uint64_t tile_pts = (uint64_t)NT * Q;
  uint64_t n_tiles = (kp.n + tile_pts - 1) / tile_pts;
  uint64_t resident = (uint64_t)di.sms * occ;
  unsigned grid = (unsigned)(n_tiles < resident ? n_tiles : resident);
  kern<<<grid, NT, 0, st>>>(kp);
  CUDA_TRY(cudaGetLastError());
  g_launches++;
  return AB_OK;
}

// Builds the implicit octree / quadtree of ab_nn_tree.cuh over a device cloud on the stream (8 launches). *buf_out owns
// every piece (release with cudaFreeAsync on the same stream), *ref_out is the device descriptor inside it.
template <typename T>
static int build_tree(const typename Vec4<T>::type* cloud, uint32_t m, int dim, const DevInfo& di, cudaStream_t st,
                      void** buf_out, const TreeRef<T>** ref_out) {
  typedef typename Vec4<T>::type V4;
  const double lg = std::log2((double)m);
  int levels = dim == 3 ? (int)std::ceil(lg / 3.0) : (int)std::ceil(lg / 2.0) - 1;  // tuned on B200, flat optimum
  const int max_levels = dim == 3 ? 8 : 12;
  levels = levels < 1 ? 1 : (levels > max_levels ? max_levels : levels);
  const uint64_t cells = 1ull << (dim * levels);
  const uint64_t n_chunks = (cells + 1 + kScanChunk - 1) / kScanChunk;
  const uint64_t start_len = n_chunks * kScanChunk;
  const uint64_t n_inner = ((1ull << (dim * levels)) - 1) / ((1ull << dim) - 1);
  auto al = [](uint64_t b) { return (b + 255) & ~255ull; };
  const uint64_t off_start = 0, off_totals = off_start + al(start_len * 4), off_key = off_totals + al(n_chunks * 4),
                 off_rank = off_key + al((uint64_t)m * 4), off_bbox = off_rank + al((uint64_t)m * 4),
                 off_ref = off_bbox + al(6 * 8), off_pts = off_ref + al(sizeof(TreeRef<T>)),
                 off_occ = off_pts + al((uint64_t)m * sizeof(V4)), total = off_occ + al(n_inner);
  char* buf = nullptr;
  CUDA_TRY(cudaMallocAsync((void**)&buf, total, st));
  *buf_out = buf;
  uint32_t* start = (uint32_t*)(buf + off_start);
  uint32_t* totals = (uint32_t*)(buf + off_totals);
  uint32_t* key = (uint32_t*)(buf + off_key);
  uint32_t* rank = (uint32_t*)(buf + off_rank);
  unsigned long long* bbox = (unsigned long long*)(buf + off_bbox);
  TreeRef<T>* ref = (TreeRef<T>*)(buf + off_ref);
  V4* pts = (V4*)(buf + off_pts);
  uint8_t* occ = (uint8_t*)(buf + off_occ);
  *ref_out = ref;
  CUDA_TRY(cudaMemsetAsync(start, 0, start_len * 4, st));
  CUDA_TRY(cudaMemsetAsync(bbox, 0xff, 3 * 8, st));
  CUDA_TRY(cudaMemsetAsync(bbox + 3, 0, 3 * 8, st));
  const unsigned gm = (unsigned)std::min<uint64_t>(((uint64_t)m + 255) / 256, (uint64_t)di.sms * 16);
  ab_tree_bbox_kernel<T><<<std::min<unsigned>(gm, (unsigned)di.sms * 4), 256, 0, st>>>(cloud, m, bbox);
  ab_tree_geom_kernel<T><<<1, 1, 0, st>>>(bbox, levels, 32u, pts, start, occ, ref);
  if (dim == 3) ab_tree_count_kernel<T, 3><<<gm, 256, 0, st>>>(cloud, m, ref, levels, start, key, rank);
  else ab_tree_count_kernel<T, 2><<<gm, 256, 0, st>>>(cloud, m, ref, levels, start, key, rank);
  ab_scan_totals_kernel<<<(unsigned)n_chunks, kScanNT, 0, st>>>(start, totals);
  ab_scan_offsets_kernel<<<1, kScanNT, 0, st>>>(totals, (uint32_t)n_chunks);
  ab_scan_apply_kernel<<<(unsigned)n_chunks, kScanNT, 0, st>>>(start, totals);
  ab_tree_scatter_kernel<T><<<gm, 256, 0, st>>>(cloud, m, start, key, rank, pts);
  const unsigned go = (unsigned)std::min<uint64_t>((n_inner + 255) / 256, (uint64_t)di.sms * 16);
  if (dim == 3) ab_tree_occupancy_kernel<3><<<go, 256, 0, st>>>(start, levels, occ);
  else ab_tree_occupancy_kernel<2><<<go, 256, 0, st>>>(start, levels, occ);
  CUDA_TRY(cudaGetLastError());
  g_launches += 8;
  return AB_OK;
}

// exact nearest neighbour through the octree: build, then one packet walk per warp (grids) / one walk per thread (lists)
template <typename T>
static int launch_nn_tree(const NNParams<T>& kp, int device, cudaStream_t st) {
  DevInfo di;
  int rc = dev_info(device, di);
  if (rc) return rc;
  const int dim = kp.dim;
  void* buf = nullptr;
  const TreeRef<T>* ref = nullptr;
  int status = build_tree<T>(kp.cloud, kp.m, dim, di, st, &buf, &ref);
  auto run = [&]() -> int {
    TreeParams<T> tp{};
    tp.q = kp;
    tp.tree = ref;
    constexpr int NT = 128;
    uint64_t warps;
    if (kp.grid_mode) {  // one warp per 2x4x4 (1x4x8) block of samples, see the kernel
      const uint64_t n0 = kp.n / kp.g.plane;
      warps = n0 == 1 ? (uint64_t)((kp.g.n1 + 3) / 4) * ((kp.g.n2 + 7) / 8)
                      : ((n0 + 1) / 2) * ((kp.g.n1 + 3) / 4) * ((kp.g.n2 + 3) / 4);
    } else {
      warps = (kp.n + 31) / 32;
    }
    const uint64_t ctas = (warps + NT / 32 - 1) / (NT / 32);
    if (ctas > 0x7fffffffull) return fail(AB_ETOOLARGE, "too many queries for one launch (%llu)", (unsigned long long)kp.n);
    const unsigned gq = (unsigned)ctas;
    if (kp.grid_mode) {
      if (dim == 3) ab_nn_tree_packet_kernel<T, 3, NT><<<gq, NT, 0, st>>>(tp);
      else ab_nn_tree_packet_kernel<T, 2, NT><<<gq, NT, 0, st>>>(tp);
    } else {
      if (dim == 3) ab_nn_tree_kernel<T, 3, NT><<<gq, NT, 0, st>>>(tp);
      else ab_nn_tree_kernel<T, 2, NT><<<gq, NT, 0, st>>>(tp);
    }
    CUDA_TRY(cudaGetLastError());
    g_launches += 1;
    return AB_OK;
  };
  if (status == AB_OK) status = run();
  if (buf) cudaFreeAsync(buf, st);
  return status;
}

template <typename T>
static int nn_t(const void* cloud, uint64_t m, int dim, int grid_mode, const GridK& g, const void* co, int co_dtype,
                uint64_t co_stride, uint64_t n, void* out, int device, cudaStream_t st) {
  if (!cloud || m == 0 || m > 0xffffffffull) return fail(AB_EINVAL, "bad cloud (m = %llu)", (unsigned long long)m);
  if (dim != 2 && dim != 3) return fail(AB_EINVAL, "dim must be 2 or 3");
  if (n == 0) return AB_OK;
  if (!out) return fail(AB_EINVAL, "null output pointer");
  NNParams<T> kp{};
  kp.n = n;
  kp.out = (T*)out;
  kp.cloud = (const typename Vec4<T>::type*)cloud;
  kp.m = (uint32_t)m;
  kp.dim = dim;
  kp.grid_mode = grid_mode;
  kp.g = g;
  kp.co = co;
  kp.co_stride = co_stride;
  kp.co_is_f64 = co_dtype == AB_F64;
  {
    // AB_NN_ALGO=brute|tree forces one of the two exact paths (they return identical bits); default: by problem size
    const char* algo = getenv("AB_NN_ALGO");
    const bool force_tree = algo && !strcmp(algo, "tree"), force_brute = algo && !strcmp(algo, "brute");
    if (force_tree || (!force_brute && m >= 256 && (double)n * (double)m >= 1073741824.0)) return launch_nn_tree<T>(kp, device, st);
  }
  if constexpr (sizeof(T) == 4) {
    // few queries: split the cloud across lanes / warps / CTAs (warp-shuffle min + atomic min), else one query per lane
    DevInfo di;
    int rc = dev_info(device, di);
    if (rc) return rc;
    if (n < (uint64_t)di.sms * 2 * 2048 && m >= 4096) {
      constexpr int QW = 16, NT = 128;
      const uint64_t groups = (n + QW - 1) / QW;
      // aim for ~8 waves of warps over the machine, slices of at least 1024 points
      uint64_t want_slices = ((uint64_t)di.sms * 64 * 8 + groups - 1) / groups;
      uint64_t max_slices = (m + 1023) / 1024;
      if (want_slices > max_slices) want_slices = max_slices;
      if (want_slices < 1) want_slices = 1;
      uint32_t slice = (uint32_t)((m + want_slices - 1) / want_slices);
      slice = (slice + 31) & ~31u;
      const uint32_t n_slices = (uint32_t)((m + slice - 1) / slice);
      const uint32_t gy = (n_slices + (NT / 32) - 1) / (NT / 32);
      if (groups <= 0x7fffffffull && gy <= 65535) {
        CUDA_TRY(cudaMemsetAsync(out, 0x7f, n * sizeof(float), st));
        ab_nn_split_kernel_f32<QW, NT><<<dim3((unsigned)groups, gy), NT, 0, st>>>(kp, slice);
        CUDA_TRY(cudaGetLastError());
        ab_nn_finalize_kernel<<<(unsigned)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096), 256, 0, st>>>((float*)out, n);
        CUDA_TRY(cudaGetLastError());
        g_launches += 2;
        return AB_OK;
      }
    }
    return launch_nn<T, 16, 512>(kp, device, st);
  }
  else return launch_nn<T, 4, 512>(kp, device, st);
}

extern "C" int ab_nn_grid(const void* cloud_dev, uint64_t m, int dim, const ab_grid* grid, int dtype, void* out,
                          int device, void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  GridK g;
  uint64_t n = 0;
  rc = make_gridk(grid, g, &n);
  if (rc) return rc;
  if (dtype == AB_F32) return nn_t<float>(cloud_dev, m, dim, 1, g, nullptr, 0, 0, n, out, device, (cudaStream_t)stream);
  if (dtype == AB_F64) return nn_t<double>(cloud_dev, m, dim, 1, g, nullptr, 0, 0, n, out, device, (cudaStream_t)stream);
  return fail(AB_EINVAL, "bad dtype %d", dtype);
}

extern "C" int ab_nn_points(const void* cloud_dev, uint64_t m, int dim, const void* co, int co_dtype,
                            uint64_t co_stride, uint64_t n, int dtype, void* out, int device, void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  if (n && !co) return fail(AB_EINVAL, "null coordinates");
  if (co_stride < n) return fail(AB_EINVAL, "co_stride < n");
  GridK g{};
  if (dtype == AB_F32) return nn_t<float>(cloud_dev, m, dim, 0, g, co, co_dtype, co_stride, n, out, device, (cudaStream_t)stream);
  if (dtype == AB_F64) return nn_t<double>(cloud_dev, m, dim, 0, g, co, co_dtype, co_stride, n, out, device, (cudaStream_t)stream);
  return fail(AB_EINVAL, "bad dtype %d", dtype);
}

// ---- from_sdf ------------------------------------------------------------------------------------------------------------------
template <typename T>
static int fd_t(const void* field, uint32_t plane0, const ab_grid* grid, int dims, int normalize, void* out,
                uint64_t out_stride, int device, cudaStream_t st) {
  FDParams<T> kp{};
  kp.field = (const T*)field;
  const bool three = dims == 3;
  // view: 3D (n0, n1, n2) = res; 2D (1, nx, ny). The slab runs over the first axis of the reference layout.
  kp.n0 = three ? grid->res[0] : 1;
  kp.n1 = three ? grid->res[1] : grid->res[0];
  kp.n2 = three ? grid->res[2] : grid->res[1];
  kp.o0 = three ? plane0 : 0;
  kp.o1 = three ? 0 : plane0;
  kp.b0 = three ? grid->slab_begin : 0;
  kp.e0 = three ? grid->slab_end : 1;
  kp.b1 = three ? 0 : grid->slab_begin;
  kp.e1 = three ? grid->res[1] : grid->slab_end;
  kp.has0 = three ? 1 : 0;
  kp.normalize = normalize;
  kp.chunk = 16;  // planes per CTA; measured at 513^3 (profiles/r02_stencils.md): 16: 0.479 ms, 32: 0.491, 64: 0.514, whole axis: 0.590
  kp.out = (T*)out;
  kp.out_stride = out_stride;
  const uint64_t n = (uint64_t)(kp.e0 - kp.b0) * (kp.e1 - kp.b1) * kp.n2;
  if (out_stride < n) return fail(AB_EINVAL, "out_stride < slab points");
  const uint32_t rows = kp.e1 - kp.b1, chunks = (kp.e0 - kp.b0 + kp.chunk - 1) / kp.chunk;
  if (rows > 65535 || chunks > 65535) return fail(AB_ETOOLARGE, "from_sdf: more than 65535 rows per plane");
  // odd row lengths (129, 513, 1025 ...): spread the warps of a row evenly over its CTAs
  const uint32_t warps = (kp.n2 + 31) / 32, ctas = (warps + 7) / 8;
  const int nt = (int)((warps + ctas - 1) / ctas) * 32;
  const dim3 fgrid(ctas, rows, chunks);
  if (three && normalize) ab_fd_kernel<T, true, true><<<fgrid, nt, 0, st>>>(kp);
  else if (three) ab_fd_kernel<T, true, false><<<fgrid, nt, 0, st>>>(kp);
  else if (normalize) ab_fd_kernel<T, false, true><<<fgrid, nt, 0, st>>>(kp);
  else ab_fd_kernel<T, false, false><<<fgrid, nt, 0, st>>>(kp);
  CUDA_TRY(cudaGetLastError());
  g_launches++;
  return AB_OK;
}

extern "C" int ab_fd_gradient(const void* field, uint32_t field_plane0, const ab_grid* grid, int dims, int dtype,
                              int normalize, void* out, uint64_t out_stride, int device, void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  if (!field || !out || !grid) return fail(AB_EINVAL, "null pointer");
  if (dims != 2 && dims != 3) return fail(AB_EINVAL, "dims must be 2 or 3");
  if (grid->slab_begin >= grid->slab_end || grid->slab_end > grid->res[0]) return fail(AB_EINVAL, "bad slab");
  if (field_plane0 > grid->slab_begin) return fail(AB_EINVAL, "field does not cover the slab");
  if (grid->slab_begin > 0 && field_plane0 > grid->slab_begin - 1) return fail(AB_EINVAL, "field lacks the lower halo plane");
  if (dtype == AB_F32) return fd_t<float>(field, field_plane0, grid, dims, normalize, out, out_stride, device, (cudaStream_t)stream);
  if (dtype == AB_F64) return fd_t<double>(field, field_plane0, grid, dims, normalize, out, out_stride, device, (cudaStream_t)stream);
  return fail(AB_EINVAL, "bad dtype %d", dtype);
}

// ---- whole-field kernels: box filter, edge filter, vector-field modifiers ------------------------------------------------------
static unsigned stream_grid(const DevInfo& di, uint64_t n, int nt) {
  const uint64_t want = (n + nt - 1) / nt, cap = (uint64_t)di.sms * 32;
  return (unsigned)std::max<uint64_t>(1, std::min(want, cap));
}

// launch geometry of the stencil kernels: see Field3 in ab_fields.cuh (2D fields are viewed as (1, nx, ny))
static int field_launch(const uint32_t res[3], bool allow_2d_view, Field3& f, dim3& grid, int& nt, int* is2d) {
  const bool two_d = allow_2d_view && res[2] == 1;
  f.n0 = two_d ? 1 : res[0];
  f.n1 = two_d ? res[0] : res[1];
  f.n2 = two_d ? res[1] : res[2];
  if (is2d) *is2d = two_d ? 1 : 0;
  if (f.n1 > 65535 || f.n0 > 65535) return fail(AB_ETOOLARGE, "field axis longer than 65535 samples");
  // SPOMSO grids are odd (129, 513, 1025 ...): spread the warps of a row evenly over its CTAs instead of leaving a nearly
  // empty last one (513 -> 3 x 192 threads, 1025 -> 5 x 224)
  const uint32_t warps = (f.n2 + 31) / 32, ctas = (warps + 7) / 8;
  nt = (int)((warps + ctas - 1) / ctas) * 32;
  grid = dim3(ctas, f.n1, f.n0);
  return AB_OK;
}

template <typename T>
static int box_filter_t(const void* field, const uint32_t res[3], const uint32_t ksize[3], uint32_t iterations, void* out,
                        int device, cudaStream_t st) {
  DevInfo di;
  int rc = dev_info(device, di);
  if (rc) return rc;
  const uint64_t n = (uint64_t)res[0] * res[1] * res[2];
  const T norm = (T)((double)ksize[0] * ksize[1] * ksize[2]);
  Field3 f;
  dim3 grid;
  int nt, is2d;
  rc = field_launch(res, ksize[2] == 1, f, grid, nt, &is2d);
  if (rc) return rc;
  int axes[3], n_axes = 0;
  for (int a = 0; a < 3; a++)
    if (ksize[a] > 1) axes[n_axes++] = a;
  if (iterations == 0) {
    CUDA_TRY(cudaMemcpyAsync(out, field, n * sizeof(T), cudaMemcpyDeviceToDevice, st));
    return AB_OK;
  }
  if (n_axes == 0) {  // a 1x1x1 kernel: u / 1
    ab_scale_copy_kernel<T><<<stream_grid(di, n, 256), 256, 0, st>>>((const T*)field, (T*)out, n, norm);
    CUDA_TRY(cudaGetLastError());
    g_launches++;
    return AB_OK;
  }
  const uint32_t passes = iterations * (uint32_t)n_axes;
  T* tmp = nullptr;
  if (passes > 1) CUDA_TRY(cudaMallocAsync((void**)&tmp, n * sizeof(T), st));
  const T* src = (const T*)field;
  uint32_t p = 0;
  for (uint32_t it = 0; it < iterations; it++) {
    for (int ai = 0; ai < n_axes; ai++, p++) {
      const int a = axes[ai];
      T* dst = ((passes - 1 - p) & 1u) ? tmp : (T*)out;  // the last pass lands in `out`
      const int k = (int)ksize[a];
      const int t0 = -((k & 1) ? k / 2 : k / 2 - 1);  // scipy.ndimage.convolve placement, see oracle/fields_np.py
      const int va = is2d ? a + 1 : a;  // axis in the (n0, n1, n2) view
      const int divide = ai == n_axes - 1 ? 1 : 0;
      bool done = false;
      if (va < 2 && k <= 9) {  // slow axes, small windows: march along the axis with the window in registers
        const uint32_t chunk = 32, n_axis = va == 0 ? f.n0 : f.n1;
        const uint32_t chunks = (n_axis + chunk - 1) / chunk;
        const dim3 mgrid = va == 0 ? dim3(grid.x, f.n1, chunks) : dim3(grid.x, chunks, f.n0);
        switch (k) {
#define AB_BOX_K(KK) case KK: ab_box_march_kernel<T, KK><<<mgrid, nt, 0, st>>>(src, dst, f, va, t0, norm, divide, chunk); done = true; break;
          AB_BOX_K(2) AB_BOX_K(3) AB_BOX_K(4) AB_BOX_K(5) AB_BOX_K(6) AB_BOX_K(7) AB_BOX_K(8) AB_BOX_K(9)
#undef AB_BOX_K
          default: break;
        }
      }
      if (!done) {
        const uint32_t rows = 16;  // y rows one thread marches over
        const dim3 bgrid(grid.x, (f.n1 + rows - 1) / rows, grid.z);
        ab_box_axis_kernel<T><<<bgrid, nt, 0, st>>>(src, dst, f, va, k, t0, norm, divide, rows);
      }
      src = dst;
    }
  }
  cudaError_t e = cudaGetLastError();
  if (tmp) cudaFreeAsync(tmp, st);
  if (e != cudaSuccess) return fail(AB_ECUDA, "box filter launch: %s", cudaGetErrorString(e));
  g_launches += passes;
  return AB_OK;
}

static int check_field_args(const void* field, const uint32_t* res, const void* out) {
  if (!field || !out || !res) return fail(AB_EINVAL, "null pointer");
  if (res[0] == 0 || res[1] == 0 || res[2] == 0) return fail(AB_EINVAL, "empty field");
  if ((uint64_t)res[0] * res[1] * res[2] > 0x7fffffffull * 4) return fail(AB_ETOOLARGE, "field too large");
  return AB_OK;
}

extern "C" int ab_box_filter(const void* field_dev, const uint32_t res[3], const uint32_t ksize[3], uint32_t iterations,
                             int dtype, void* out_dev, int device, void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  rc = check_field_args(field_dev, res, out_dev);
  if (rc) return rc;
  if (!ksize || ksize[0] == 0 || ksize[1] == 0 || ksize[2] == 0) return fail(AB_EINVAL, "kernel sizes must be >= 1");
  if (field_dev == out_dev) return fail(AB_EINVAL, "box filter cannot run in place");
  if (dtype == AB_F32) return box_filter_t<float>(field_dev, res, ksize, iterations, out_dev, device, (cudaStream_t)stream);
  if (dtype == AB_F64) return box_filter_t<double>(field_dev, res, ksize, iterations, out_dev, device, (cudaStream_t)stream);
  return fail(AB_EINVAL, "bad dtype %d", dtype);
}

extern "C" int ab_edge_filter(const void* field_dev, const uint32_t res[3], int dtype, void* out_dev, int device, void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  rc = check_field_args(field_dev, res, out_dev);
  if (rc) return rc;
  if (field_dev == out_dev) return fail(AB_EINVAL, "edge filter cannot run in place");
  Field3 f;
  dim3 grid;
  int nt, is2d;
  rc = field_launch(res, true, f, grid, nt, &is2d);
  if (rc) return rc;
  const uint32_t chunk = 32;
  // 3D: (z chunks, y, x chunks); 2D view: (z chunks, y chunks, 1)
  const dim3 egrid = is2d ? dim3(grid.x, (f.n1 + chunk - 1) / chunk, 1) : dim3(grid.x, f.n1, (f.n0 + chunk - 1) / chunk);
  if (dtype == AB_F32) ab_edge_kernel<float, 4><<<egrid, nt, 0, (cudaStream_t)stream>>>((const float*)field_dev, (float*)out_dev, f, is2d, chunk);
  else if (dtype == AB_F64) ab_edge_kernel<double, 4><<<egrid, nt, 0, (cudaStream_t)stream>>>((const double*)field_dev, (double*)out_dev, f, is2d, chunk);
  else return fail(AB_EINVAL, "bad dtype %d", dtype);
  CUDA_TRY(cudaGetLastError());
  g_launches++;
  return AB_OK;
}

// ---- signed: unsigned -> signed distance field (modifications.py:220-275) ---------------------------------------------------------
static uint32_t mask_words(uint32_t n2) { return (n2 + 31u) / 32u; }

template <typename T>
static int signed_mask_t(const void* field, const uint32_t res[3], double threshold, uint32_t* mask, int* flags, cudaStream_t st) {
  const uint32_t words = mask_words(res[2]), wpb = std::min<uint32_t>(words, 8u);  // mask words (warps) per CTA
  const dim3 g((words + wpb - 1) / wpb, res[1], res[0]);
  ab_signed_mask_kernel<T><<<g, wpb * 32, 0, st>>>((const T*)field, Field3{res[0], res[1], res[2]}, words, (T)threshold, mask, flags);
  CUDA_TRY(cudaGetLastError());
  g_launches++;
  return AB_OK;
}

// planes [x0, x1) of the signed field from the whole mask: the (2,2,1) smoothing reads interior planes i and i + 1, the face
// clamp reads planes 1 and n0 - 2 instead of 0 and n0 - 1, so the interior is needed on [c(x0), c(x1 - 1) + 2) with
// c = clamp to [1, n0 - 2]. The box filter runs on that block as if it were a whole field: at a cut its last plane is
// reflected wrongly and never read; at the face n0 - 1 it reflects like the whole field (same taps, same order).
template <typename T>
static int signed_slab_t(const uint32_t* mask, const int* flags, const void* field, const void* tangent, uint32_t field_plane0,
                         const uint32_t res[3], uint32_t x0, uint32_t x1, void* out, void* out_tangent, int device,
                         cudaStream_t st) {
  const uint32_t n0 = res[0], n1 = res[1], n2 = res[2], words = mask_words(n2);
  auto clampi = [&](uint32_t i) { return i < 1 ? 1u : (i > n0 - 2 ? n0 - 2 : i); };
  const uint32_t s0 = clampi(x0), s1 = clampi(x1 - 1) + 2, m = s1 - s0;  // interior / smoothed planes [s0, s1)
  const uint64_t nw = (uint64_t)m * n1 * words, ni = (uint64_t)m * n1 * n2, plane = (uint64_t)n1 * n2;
  auto al = [](uint64_t b) { return (b + 255) & ~255ull; };
  const uint64_t off_int = 4 * al(nw * 4), off_smooth = off_int + al(ni * sizeof(T)), total = off_smooth + al(ni * sizeof(T));
  char* buf = nullptr;
  CUDA_TRY(cudaMallocAsync((void**)&buf, total, st));
  uint32_t* par = (uint32_t*)buf;
  uint32_t *pin0 = par, *pout0 = (uint32_t*)(buf + al(nw * 4)), *pin1 = (uint32_t*)(buf + 2 * al(nw * 4)),
           *pout1 = (uint32_t*)(buf + 3 * al(nw * 4));
  T *interior = (T*)(buf + off_int), *smooth = (T*)(buf + off_smooth);
  int rc = AB_OK;
  do {
    const uint64_t cols = std::max<uint64_t>((uint64_t)n1 * words, (uint64_t)m * words);
    ab_signed_scan_kernel<<<dim3((unsigned)((cols + 255) / 256), 2), 256, 0, st>>>(mask, n0, n1, words, s0, s1, pin0, pout0, pin1, pout1);
    const Field3 fm{m, n1, n2};
    ab_signed_interior_kernel<T><<<dim3((n2 + 255) / 256, n1, m), 256, 0, st>>>(pin0, pout0, pin1, pout1, fm, words, interior);
    const uint32_t ks[3] = {2, 2, 1}, rm[3] = {m, n1, n2};
    rc = box_filter_t<T>(interior, rm, ks, 1, smooth, device, st);  // conv_averaging(interior, (2, 2, 1), 1)
    if (rc) break;
    const dim3 ga((n2 + 255) / 256, n1, x1 - x0);
    const uint64_t skip = (uint64_t)(x0 - field_plane0) * plane;
    if (tangent)  // the same sign per sample on the tangent row (tangent pointers null: value only)
      ab_signed_apply_kernel<T, true><<<ga, 256, 0, st>>>((const T*)field + skip, (const T*)tangent + skip, smooth,
                                                          Field3{n0, n1, n2}, x0, s0, flags, (T*)out, (T*)out_tangent);
    else
      ab_signed_apply_kernel<T, false><<<ga, 256, 0, st>>>((const T*)field + skip, nullptr, smooth, Field3{n0, n1, n2}, x0, s0,
                                                           flags, (T*)out, nullptr);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { rc = fail(AB_ECUDA, "signed launch: %s", cudaGetErrorString(e)); break; }
    g_launches += 3;
  } while (0);
  cudaFreeAsync(buf, st);
  return rc;
}

static int check_signed_res(const uint32_t res[3]) {
  if (res[0] < 3 || res[1] < 3 || res[2] < 3) return fail(AB_EINVAL, "signed needs at least 3 samples per axis (the reference pads an empty interior otherwise)");
  if (res[0] > 65535 || res[1] > 65535) return fail(AB_ETOOLARGE, "field axis longer than 65535 samples");
  return AB_OK;
}

extern "C" int ab_signed_mask(const void* field_dev, const uint32_t res[3], double threshold, int dtype, uint32_t* mask_dev,
                              int* flags_dev, int device, void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  rc = check_field_args(field_dev, res, mask_dev);
  if (rc) return rc;
  if (!flags_dev) return fail(AB_EINVAL, "null pointer");
  if (res[0] > 65535 || res[1] > 65535) return fail(AB_ETOOLARGE, "field axis longer than 65535 samples");
  if (dtype == AB_F32) return signed_mask_t<float>(field_dev, res, threshold, mask_dev, flags_dev, (cudaStream_t)stream);
  if (dtype == AB_F64) return signed_mask_t<double>(field_dev, res, threshold, mask_dev, flags_dev, (cudaStream_t)stream);
  return fail(AB_EINVAL, "bad dtype %d", dtype);
}

extern "C" int ab_signed_field_slab(const uint32_t* mask_dev, const int* flags_dev, const void* field_dev, uint32_t field_plane0,
                                    const uint32_t res[3], uint32_t x0, uint32_t x1, int dtype, void* out_dev, int device,
                                    void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  rc = check_field_args(field_dev, res, out_dev);
  if (rc) return rc;
  if (!mask_dev || !flags_dev) return fail(AB_EINVAL, "null pointer");
  rc = check_signed_res(res);
  if (rc) return rc;
  if (x0 >= x1 || x1 > res[0]) return fail(AB_EINVAL, "bad slab [%u, %u) of %u planes", x0, x1, res[0]);
  if (field_plane0 > x0) return fail(AB_EINVAL, "field does not cover the slab");
  if (field_dev == out_dev) return fail(AB_EINVAL, "signed cannot run in place");
  if (dtype == AB_F32) return signed_slab_t<float>(mask_dev, flags_dev, field_dev, nullptr, field_plane0, res, x0, x1, out_dev, nullptr, device, (cudaStream_t)stream);
  if (dtype == AB_F64) return signed_slab_t<double>(mask_dev, flags_dev, field_dev, nullptr, field_plane0, res, x0, x1, out_dev, nullptr, device, (cudaStream_t)stream);
  return fail(AB_EINVAL, "bad dtype %d", dtype);
}

extern "C" int ab_signed_field_slab_tangent(const uint32_t* mask_dev, const int* flags_dev, const void* field_dev,
                                            const void* tangent_dev, uint32_t field_plane0, const uint32_t res[3], uint32_t x0,
                                            uint32_t x1, int dtype, void* out_dev, void* out_tangent_dev, int device,
                                            void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  rc = check_field_args(field_dev, res, out_dev);
  if (rc) return rc;
  if (!mask_dev || !flags_dev || !tangent_dev || !out_tangent_dev) return fail(AB_EINVAL, "null pointer");
  rc = check_signed_res(res);
  if (rc) return rc;
  if (x0 >= x1 || x1 > res[0]) return fail(AB_EINVAL, "bad slab [%u, %u) of %u planes", x0, x1, res[0]);
  if (field_plane0 > x0) return fail(AB_EINVAL, "field does not cover the slab");
  if (field_dev == out_dev || tangent_dev == out_tangent_dev || field_dev == out_tangent_dev || tangent_dev == out_dev ||
      out_dev == out_tangent_dev)
    return fail(AB_EINVAL, "signed cannot run in place (inputs, outputs: four distinct buffers)");
  if (dtype == AB_F32) return signed_slab_t<float>(mask_dev, flags_dev, field_dev, tangent_dev, field_plane0, res, x0, x1, out_dev, out_tangent_dev, device, (cudaStream_t)stream);
  if (dtype == AB_F64) return signed_slab_t<double>(mask_dev, flags_dev, field_dev, tangent_dev, field_plane0, res, x0, x1, out_dev, out_tangent_dev, device, (cudaStream_t)stream);
  return fail(AB_EINVAL, "bad dtype %d", dtype);
}

extern "C" int ab_signed_field(const void* field_dev, const uint32_t res[3], double threshold, int dtype, void* out_dev, int device,
                               void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  rc = check_field_args(field_dev, res, out_dev);
  if (rc) return rc;
  rc = check_signed_res(res);
  if (rc) return rc;
  if (field_dev == out_dev) return fail(AB_EINVAL, "signed cannot run in place");
  if (dtype != AB_F32 && dtype != AB_F64) return fail(AB_EINVAL, "bad dtype %d", dtype);
  cudaStream_t st = (cudaStream_t)stream;
  const uint64_t nw = (uint64_t)res[0] * res[1] * mask_words(res[2]);
  char* buf = nullptr;
  CUDA_TRY(cudaMallocAsync((void**)&buf, 256 + nw * 4, st));
  int* flags = (int*)buf;
  uint32_t* mask = (uint32_t*)(buf + 256);
  do {
    if (cudaMemsetAsync(flags, 0, 2 * sizeof(int), st) != cudaSuccess) { rc = fail(AB_ECUDA, "memset"); break; }
    rc = dtype == AB_F32 ? signed_mask_t<float>(field_dev, res, threshold, mask, flags, st)
                         : signed_mask_t<double>(field_dev, res, threshold, mask, flags, st);
    if (rc) break;
    rc = dtype == AB_F32 ? signed_slab_t<float>(mask, flags, field_dev, nullptr, 0, res, 0, res[0], out_dev, nullptr, device, st)
                         : signed_slab_t<double>(mask, flags, field_dev, nullptr, 0, res, 0, res[0], out_dev, nullptr, device, st);
  } while (0);
  cudaFreeAsync(buf, st);
  return rc;
}

static int check_vec_op(const ab_vec_op& op, uint32_t i, uint64_t n) {
  auto scalar_ok = [&](uint32_t kind, const void* a) { return kind == AB_VK_SCALAR || (kind == AB_VK_ARRAY && a); };
  switch (op.opcode) {
    case AB_VOP_ADD: case AB_VOP_SUB:
      if (scalar_ok(op.kind0, op.a0) || op.kind0 == AB_VK_VEC3 || (op.kind0 == AB_VK_VEC_ARRAY && op.a0 && op.stride0 >= n)) return AB_OK;
      break;
    case AB_VOP_RESCALE:
      if (scalar_ok(op.kind0, op.a0) || (op.kind0 == AB_VK_VEC_ARRAY && op.a0 && op.stride0 >= n)) return AB_OK;
      break;
    case AB_VOP_ROT_Z: case AB_VOP_ROT_THETA: case AB_VOP_ROT_X: case AB_VOP_ROT_Y:
      if (scalar_ok(op.kind0, op.a0)) return AB_OK;
      break;
    case AB_VOP_ROT_AXIS:
      if ((op.kind0 == AB_VK_VEC3 || (op.kind0 == AB_VK_VEC_ARRAY && op.a0 && op.stride0 >= n)) && scalar_ok(op.kind1, op.a1)) return AB_OK;
      break;
    case AB_VOP_REVOLVE_X: case AB_VOP_REVOLVE_Y: case AB_VOP_REVOLVE_Z:
      if (op.kind0 == AB_VK_VEC_ARRAY && op.a0 && op.stride0 >= n) return AB_OK;
      break;
    case AB_VOP_NORMALIZE: return AB_OK;
    default: return fail(AB_EUNSUPPORTED_OP, "vector op %u: unknown opcode %u", i, op.opcode);
  }
  return fail(AB_EINVAL, "vector op %u (opcode %u): operand kinds (%u, %u) not accepted or array missing / too short", i,
              op.opcode, op.kind0, op.kind1);
}

template <typename T>
static int vec_apply_t(void* vec, uint64_t stride, uint64_t n, const ab_vec_op* ops, uint32_t n_ops, int device, cudaStream_t st) {
  DevInfo di;
  int rc = dev_info(device, di);
  if (rc) return rc;
  VecParams<T> vp{};
  vp.vec = (T*)vec;
  vp.stride = stride;
  vp.n = n;
  vp.n_ops = n_ops;
  for (uint32_t i = 0; i < n_ops; i++) {
    VecOpK& k = vp.ops[i];
    k.opcode = ops[i].opcode;
    k.kind0 = ops[i].kind0;
    k.kind1 = ops[i].kind1;
    for (int j = 0; j < 3; j++) k.c[j] = ops[i].c[j];
    k.s0 = ops[i].s0;
    k.s1 = ops[i].s1;
    k.a0 = ops[i].a0;
    k.a1 = ops[i].a1;
    k.stride0 = ops[i].stride0;
    k.stride1 = ops[i].stride1;
  }
  ab_vec_kernel<T><<<stream_grid(di, n, 256), 256, 0, st>>>(vp);
  CUDA_TRY(cudaGetLastError());
  g_launches++;
  return AB_OK;
}

extern "C" int ab_vec_apply(void* vec_dev, uint64_t vec_stride, uint64_t n, const ab_vec_op* ops, uint32_t n_ops, int dtype,
                            int device, void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  if (n == 0 || n_ops == 0) return AB_OK;
  if (!vec_dev || !ops) return fail(AB_EINVAL, "null pointer");
  if (vec_stride < n) return fail(AB_EINVAL, "vec_stride < n");
  if (n_ops > AB_MAX_VEC_OPS) return fail(AB_ETOOLARGE, "too many vector ops (%u > %d)", n_ops, AB_MAX_VEC_OPS);
  for (uint32_t i = 0; i < n_ops; i++) {
    rc = check_vec_op(ops[i], i, n);
    if (rc) return rc;
  }
  if (dtype == AB_F32) return vec_apply_t<float>(vec_dev, vec_stride, n, ops, n_ops, device, (cudaStream_t)stream);
  if (dtype == AB_F64) return vec_apply_t<double>(vec_dev, vec_stride, n, ops, n_ops, device, (cudaStream_t)stream);
  return fail(AB_EINVAL, "bad dtype %d", dtype);
}

extern "C" int ab_vec_component(const void* vec_dev, uint64_t vec_stride, uint64_t n, int what, int dtype, void* out_dev,
                                int device, void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  if (n == 0) return AB_OK;
  if (!vec_dev || !out_dev) return fail(AB_EINVAL, "null pointer");
  if (vec_stride < n) return fail(AB_EINVAL, "vec_stride < n");
  if (what < AB_VC_X || what > AB_VC_LENGTH) return fail(AB_EINVAL, "bad component id %d", what);
  DevInfo di;
  rc = dev_info(device, di);
  if (rc) return rc;
  const unsigned grid = stream_grid(di, n, 256);
  if (dtype == AB_F32) ab_vec_component_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>((const float*)vec_dev, vec_stride, n, what, (float*)out_dev);
  else if (dtype == AB_F64) ab_vec_component_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>((const double*)vec_dev, vec_stride, n, what, (double*)out_dev);
  else return fail(AB_EINVAL, "bad dtype %d", dtype);
  CUDA_TRY(cudaGetLastError());
  g_launches++;
  return AB_OK;
}

// ---- memory helpers ---------------------------------------------------------------------------------------------------------------
extern "C" int ab_device_alloc(uint64_t bytes, int device, void** out_dev) {
  int rc = use_device(device);
  if (rc) return rc;
  if (!out_dev) return fail(AB_EINVAL, "null pointer");
  CUDA_TRY(cudaMalloc(out_dev, bytes ? bytes : 1));
  return AB_OK;
}
extern "C" int ab_device_free(void* dev, int device) {
  int rc = use_device(device);
  if (rc) return rc;
  CUDA_TRY(cudaFree(dev));
  return AB_OK;
}
extern "C" int ab_host_alloc_pinned(uint64_t bytes, void** out_host) {
  if (!out_host) return fail(AB_EINVAL, "null pointer");
  if (ab_device_count() == 0) return fail(AB_ENODEVICE, "no CUDA device visible");
  CUDA_TRY(cudaHostAlloc(out_host, bytes ? bytes : 1, cudaHostAllocDefault));
  return AB_OK;
}
// flags: bit 0 cudaHostAllocPortable, bit 1 cudaHostAllocWriteCombined (device -> host result buffers are written by the
// GPU and read once by the CPU: write-combined pages skip the cache snoop on every PCIe write)
extern "C" int ab_host_alloc_pinned_flags(uint64_t bytes, unsigned flags, void** out_host) {
  if (!out_host) return fail(AB_EINVAL, "null pointer");
  if (ab_device_count() == 0) return fail(AB_ENODEVICE, "no CUDA device visible");
  unsigned f = cudaHostAllocDefault;
  if (flags & 1u) f |= cudaHostAllocPortable;
  if (flags & 2u) f |= cudaHostAllocWriteCombined;
  CUDA_TRY(cudaHostAlloc(out_host, bytes ? bytes : 1, f));
  return AB_OK;
}
extern "C" int ab_host_free_pinned(void* host) {
  CUDA_TRY(cudaFreeHost(host));
  return AB_OK;
}
extern "C" int ab_memcpy_d2h(void* dst_host, const void* src_dev, uint64_t bytes, int device, void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  return AB_OK;
}
extern "C" int ab_memcpy_h2d(void* dst_dev, const void* src_host, uint64_t bytes, int device, void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
  return AB_OK;
}
extern "C" int ab_stream_sync(int device, void* stream) {
  int rc = use_device(device);
  if (rc) return rc;
  CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  return AB_OK;
}
