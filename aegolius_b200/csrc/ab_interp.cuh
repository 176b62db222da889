// ab_interp.cuh — the SDF interpreter kernel (sm_100a).
//
// One launch evaluates one flattened geometry tree on a slab of grid points (or on an explicit point list). The whole
// program (op list + argument pool) is a __grid_constant__ kernel parameter: it lives in constant bank 0, costs no
// separate H2D copy and cannot race between concurrent launches. Control flow is identical for every point, so opcode
// dispatch is warp-uniform; per thread W consecutive points along the fastest grid axis live in registers (Pack<T,W>),
// the saved-coordinate / saved-value stacks live in shared memory as conflict-free 16-byte columns, and the field is
// written with one 128-bit streaming store per thread (coalesced: a warp writes 512 contiguous bytes).
//
// Grid layout (generate_grid, helper_functions.py:23-93): flat k = (ix*ny + iy)*nz + iz, z fastest; the slab is a range
// of ix planes, i.e. one contiguous range of k. Coordinates are regenerated from (ix,iy,iz): 0 bytes read per point.
#pragma once
#include <type_traits>
#ifndef AB_TIER_FULL
#define AB_TIER_FULL 2
#endif
#ifndef AB_DISPATCH_BRX
#define AB_DISPATCH_BRX 0 /* 1 = indexed-branch dispatch, 0 = uniform compare tree (faster on B200, see the dispatch comment) */
#endif
#include "../../include/aegolius_b200.h"
#include "ab_ops.cuh"

namespace ab {

struct GridK {
  // index axes (ix, iy, iz), iz fastest. 2D grids are (nx, ny, 1) with size_z = 0, so z == 0.
  uint32_t n1, n2;          // ny, nz
  uint32_t plane;           // ny * nz
  uint32_t i0_begin;        // first ix plane of the slab (3D)
  uint32_t i1_begin;        // 2D grids are remapped to index axes (1, nx, ny): the slab offset then applies to axis 1
  uint32_t is2d;            // 1: x = axis-1 sample, y = axis-2 sample, z = +0 (parameter sets 1 and 2 hold x and y)
  uint32_t last[3];         // res-1 per axis (for the exact linspace end point)
  double start[3], step[3], stop[3];  // linspace parameters per axis (fp64 path: bit-identical to numpy)
  float hi[3], lo[3], centre[3];      // fp32 path: x = (i - centre) * (hi + lo), one rounding
  uint32_t m1, m2;                    // floor(2^32 / n1), floor(2^32 / n2): mulhi quotient estimates (one fix-up step)
};

// quotient / remainder of a small numerator by a runtime constant: q_est = umulhi(t, floor(2^32/n)) is floor(t/n) or one
// less, so a single correction step makes it exact (also for n == 1).
AB_DEV void divmod_small(uint32_t t, uint32_t n, uint32_t magic, uint32_t& q, uint32_t& r) {
  q = __umulhi(t, magic);
  r = t - q * n;
  if (r >= n) {
    q++;
    r -= n;
  }
}

// dense opcode numbering used inside the kernel (the host remaps ab_opcode -> DenseOp so that the dispatch switch
// compiles to one indexed branch instead of a compare tree)
#define AB_OPLIST(X)                                                                                                   \
  X(END) X(SAVE_P) X(LOAD_P) X(PUSH_V) X(NEXT_AFFINE) X(NEXT_TRANSLATE) X(NEXT_LOAD) X(AFFINE) X(TRANSLATE) X(SCALE_P) X(ELONGATE) X(TWIST) X(BEND) X(ABSX_SUB)        \
  X(SYMMETRY) X(ROTSYM) X(REVOLVE) X(AXIS_REVOLVE) X(REP_INF) X(REP_FIN) X(LIN_INST) X(CURVE_INST) X(ZERO_Z) X(ROUND)  \
  X(ABS) X(NEG) X(SIGN) X(ONION) X(CONCENTRIC) X(SCALE_V) X(EXTRUDE_BEGIN) X(EXTRUDE_END) X(POLY_SIGN) X(PP_SIGMOID)                \
  X(PP_POS_SIGMOID) X(PP_CAPPED_EXP) X(PP_HARD_BIN) X(PP_LINEAR) X(PP_RELU) X(PP_SMOOTH_RELU) X(PP_SLOWSTART)          \
  X(PP_GAUSS_BOUNDARY) X(PP_GAUSS_FALLOFF) X(C_UNION) X(C_INTERSECT) X(C_SUBTRACT) X(C_SUM) X(C_DIFF) X(C_SMIN2)       \
  X(C_SMIN3) X(C_SMAX3) X(C_SSUB3) X(C_BOLTZ_INT) X(C_BOLTZ_SUB) X(P_SPHERE) X(P_CYLINDER) X(P_BOX) X(P_TORUS)         \
  X(P_CHAINLINK) X(P_BRAID) X(P_ARC3D) X(P_PLANE) X(P_UPLANE) X(P_SEGMENT) X(P_CONE) X(P_OINF_CONE) X(P_INF_CONE)      \
  X(P_SOLID_ANGLE) X(P_TRIANGLE3D) X(P_QUAD3D) X(P_SEGLINE) X(P_AXIS) X(P_POINT_CLOUD) X(P_FIELD) X(P_CIRCLE) X(P_NEU_CIRCLE)     \
  X(P_BOX2D) X(P_SEGMENT2D) X(P_RBOX2D) X(P_TRIANGLE2D) X(P_ARC) X(P_SECTOR) X(P_INF_SECTOR) X(P_NGON) X(P_SEGLINE2D) \
  X(P_POLYGON2D)
enum DenseOp : uint16_t {
#define AB_X(name) D_##name,
  AB_OPLIST(AB_X)
#undef AB_X
      D__COUNT
};
inline int dense_opcode(int ab_opcode) {
  switch (ab_opcode) {
#define AB_X(name) \
  case AB_OP_##name: return D_##name;
    AB_OPLIST(AB_X)
#undef AB_X
    default: return -1;
  }
}

template <typename T>
struct Vec4;
template <>
struct Vec4<float> {
  typedef float4 type;
};
template <>
struct Vec4<double> {
  typedef double4 type;
};

}  // namespace ab
#include "ab_spec_default.h"
#include "ab_tree.cuh"
namespace ab {

template <typename T>
struct KParams {
  uint64_t n;        // points in this launch (< 2^31: the host splits larger slabs on plane boundaries)
  T* out;            // (n,)
  T* grad;           // (K, grad_stride) or nullptr
  uint64_t grad_stride;
  const void* co;    // points mode: (3, co_stride) of float/double
  uint64_t co_stride;
  int32_t co_is_f64;
  int32_t grid_mode;
  GridK g;
  uint32_t tile_stride[3];  // (d0, d1, d2): decomposition of gridDim.x * tile points, filled in by the launcher
  uint32_t n_ops, n_args, n_pslots, n_vslots;
  uint32_t off_args, off_pstack, off_vstack;  // byte offsets inside dynamic shared memory (filled in by the launcher)
  int32_t tier;  // 0 = every op is in the lite set (host-side choice of kernel variant)
  uint32_t dargs_off;  // AB_GRAD_PARAM: args[dargs_off + i] = d args[i] / d theta (second half of the pool), else 0
  const void* blob[AB_MAX_BLOBS];  // (x, y, z, 0) records of T
  uint32_t blob_count[AB_MAX_BLOBS];
  const void* blob_tree[AB_MAX_BLOBS];  // device TreeRef<T> of the blob (large clouds) or nullptr: scan the blob
  const void* dblob[AB_MAX_BLOBS];  // AB_GRAD_PARAM: tangent row of a P_FIELD blob (indexed like blob[b]), else nullptr
  // AB_GRAD_PARAM loss mode (ab_eval_grid_loss): instead of storing F and dF/dtheta the kernel accumulates
  // loss_accum[0] += sum (F - target)^2, loss_accum[1] += sum 2 (F - target) dF/dtheta   (target indexed like out)
  const T* target;
  double* loss_accum;
  uint2 ops[AB_MAX_OPS];  // kernel-side encoding: x = dense opcode (a full word), y = argument offset | a << 16 | b << 24
  T args[AB_MAX_ARGS];
};

// ---- coordinate generation ------------------------------------------------------------------------------------------
AB_DEV float grid_coord(const GridK& g, int c, uint32_t i, float) {
  float k = (float)i - g.centre[c];
  return fmaf(k, g.hi[c], k * g.lo[c]);
}
AB_DEV double grid_coord(const GridK& g, int c, uint32_t i, double) {
  // np.linspace: arange(n) * step + start, last sample forced to stop (no FMA contraction: bit-identical)
  return (i == g.last[c]) ? g.stop[c] : __dadd_rn(__dmul_rn((double)i, g.step[c]), g.start[c]);
}

// W consecutive samples of one axis starting at index i: k_j = (i - centre) + j is exact in fp32, then the same one-rounding
// product as grid_coord, issued as packed f32x2 (3 packed instructions per 2 samples instead of 4 scalar per sample)
template <int W>
AB_DEV void grid_coord_run(const GridK& g, int c, int32_t i, Pack<float, W>& out) {
  const float k0 = (float)i - g.centre[c];
  Pack<float, W> k;
#pragma unroll
  for (int j = 0; j < W; j++) k.v[j] = (float)j;
  k = k + k0;
  out = fma_(k, g.hi[c], k * g.lo[c]);
}
template <int W>
AB_DEV void grid_coord_run(const GridK& g, int c, int32_t i, Pack<double, W>& out) {
#pragma unroll
  for (int j = 0; j < W; j++) out.v[j] = (i + j >= 0) ? grid_coord(g, c, (uint32_t)(i + j), 0.0) : 0.0;
}

// ---- walking the slab tile by tile ------------------------------------------------------------------------------------------
// A CTA owns tiles blockIdx.x, blockIdx.x + gridDim.x, ...; every thread carries the index-axis coordinates (i0, i1, i2) of
// its own first point in the current tile: two real divisions per thread at kernel start (tile_walk_begin), then three
// carried additions per tile (the launcher decomposed the stride gridDim.x * tile points into tile_stride[]). No division
// or multiply-high in the loop. Shared by the interpreter and by the program-compiled kernels (codegen.py).
struct TileWalk {
  uint32_t i0, i1, i2;  // local to the launch (the slab offsets i0_begin / i1_begin are added when coordinates are made)
};
template <typename T>
AB_DEV void tile_walk_begin(const KParams<T>& kp, uint32_t tile_pts, uint32_t w_pts, TileWalk& w) {
  w.i0 = w.i1 = w.i2 = 0;
  if (kp.grid_mode) {
    const uint32_t start = blockIdx.x * tile_pts + threadIdx.x * w_pts;
    w.i0 = start / kp.g.plane;
    const uint32_t rem = start - w.i0 * kp.g.plane;
    w.i1 = rem / kp.g.n2;
    w.i2 = rem - w.i1 * kp.g.n2;
  }
}
// coordinates of this thread's W consecutive points (first local index idx) and the step to the CTA's next tile.
// IS2D: -1 = read kp.g.is2d (interpreter), 0 / 1 = known at compile time (program-compiled kernels: saves 3 W selects)
template <int IS2D = -1, typename T, int W>
AB_DEV void tile_coords(const KParams<T>& kp, TileWalk& w, uint32_t idx, uint32_t n32, Pack<T, W>& cx, Pack<T, W>& cy,
                        Pack<T, W>& cz) {
  typedef Pack<T, W> P;
  if (kp.grid_mode) {
    uint32_t i2 = w.i2, i1 = w.i1 + kp.g.i1_begin, i0 = w.i0 + kp.g.i0_begin;
    P ua, ub, uc;  // samples along index axes (slow, middle, fast)
    if (i2 + W <= kp.g.n2) {  // the W points share one row: the common case
      ua = P(grid_coord(kp.g, 0, i0, T()));
      ub = P(grid_coord(kp.g, 1, i1, T()));
      grid_coord_run(kp.g, 2, (int32_t)i2, uc);
    } else if (kp.g.n2 >= (uint32_t)W) {  // exactly one row boundary inside the run: points j >= s sit on the next row
      const int s = (int)(kp.g.n2 - i2);
      uint32_t j1 = i1 + 1, j0 = i0;
      if (j1 == kp.g.n1 + kp.g.i1_begin) {
        j1 = kp.g.i1_begin;
        ++j0;
      }
      const T a0 = grid_coord(kp.g, 0, i0, T()), a1 = grid_coord(kp.g, 1, i1, T());
      const T n0 = grid_coord(kp.g, 0, j0, T()), n1 = grid_coord(kp.g, 1, j1, T());
      P ra, rb;
      grid_coord_run(kp.g, 2, (int32_t)i2, ra);
      grid_coord_run(kp.g, 2, -s, rb);
#pragma unroll
      for (int j = 0; j < W; j++) {
        const bool first = j < s;
        ua.v[j] = first ? a0 : n0;
        ub.v[j] = first ? a1 : n1;
        uc.v[j] = first ? ra.v[j] : rb.v[j];
      }
    } else {  // rows shorter than the run (tiny grids): walk point by point
#pragma unroll
      for (int j = 0; j < W; j++) {
        ua.v[j] = grid_coord(kp.g, 0, i0, T());
        ub.v[j] = grid_coord(kp.g, 1, i1, T());
        uc.v[j] = grid_coord(kp.g, 2, i2, T());
        if (++i2 == kp.g.n2) {
          i2 = 0;
          if (++i1 == kp.g.n1 + kp.g.i1_begin) {
            i1 = kp.g.i1_begin;
            ++i0;
          }
        }
      }
    }
    if (IS2D < 0 ? kp.g.is2d != 0 : IS2D != 0) {  // index axes (1, nx, ny): x = axis-1 sample, y = axis-2 sample, z = +0
      cx = ub;
      cy = uc;
      cz = P(T(0));
    } else {
      cx = ua;
      cy = ub;
      cz = uc;
    }
    // advance this thread's first point by gridDim.x tiles
    w.i2 += kp.tile_stride[2];
    if (w.i2 >= kp.g.n2) {
      w.i2 -= kp.g.n2;
      w.i1++;
    }
    w.i1 += kp.tile_stride[1];
    if (w.i1 >= kp.g.n1) {
      w.i1 -= kp.g.n1;
      w.i0++;
    }
    w.i0 += kp.tile_stride[0];
  } else {
#pragma unroll
    for (int j = 0; j < W; j++) {
      const uint64_t k = idx + j < n32 ? idx + j : n32 - 1;
      if (kp.co_is_f64) {
        const double* c = (const double*)kp.co;
        cx.v[j] = (T)__ldcs(c + k);
        cy.v[j] = (T)__ldcs(c + kp.co_stride + k);
        cz.v[j] = (T)__ldcs(c + 2 * kp.co_stride + k);
      } else {
        const float* c = (const float*)kp.co;
        cx.v[j] = (T)__ldcs(c + k);
        cy.v[j] = (T)__ldcs(c + kp.co_stride + k);
        cz.v[j] = (T)__ldcs(c + 2 * kp.co_stride + k);
      }
    }
  }
}

// The common case of tile_coords for a whole warp at once: every thread's W points share one row, so the two slow
// coordinates are per-thread broadcasts and only the fast one varies along the run. Program-compiled kernels of short
// programs emit their body twice (codegen.py, `rowsplit`): in the copy behind this function the compiler sees that all W
// lanes of x and y hold one value and evaluates everything that depends on them alone once per thread instead of W times
// (common-subexpression elimination does it: the general path merges two coordinate branches and hides that).
template <typename T, int W>
AB_DEV bool tile_run_in_one_row(const KParams<T>& kp, const TileWalk& w) { return kp.grid_mode && w.i2 + W <= kp.g.n2; }
template <int IS2D, typename T, int W>
AB_DEV void tile_coords_uniform(const KParams<T>& kp, TileWalk& w, Pack<T, W>& cx, Pack<T, W>& cy, Pack<T, W>& cz) {
  typedef Pack<T, W> P;
  const T a0 = grid_coord(kp.g, 0, w.i0 + kp.g.i0_begin, T()), a1 = grid_coord(kp.g, 1, w.i1 + kp.g.i1_begin, T());
  P uc;
  grid_coord_run(kp.g, 2, (int32_t)w.i2, uc);
  if (IS2D) {
    cx = P(a1);
    cy = uc;
    cz = P(T(0));
  } else {
    cx = P(a0);
    cy = P(a1);
    cz = uc;
  }
  w.i2 += kp.tile_stride[2];
  if (w.i2 >= kp.g.n2) {
    w.i2 -= kp.g.n2;
    w.i1++;
  }
  w.i1 += kp.tile_stride[1];
  if (w.i1 >= kp.g.n1) {
    w.i1 -= kp.g.n1;
    w.i0++;
  }
  w.i0 += kp.tile_stride[0];
}

// ---- stack in shared memory: element [slot][tid] is one 16-byte Pack column --------------------------------------------
template <typename P>
AB_DEV void st_pack(P* base, int slot, int nt, const P& v) { base[slot * nt + threadIdx.x] = v; }
template <typename P>
AB_DEV P ld_pack(const P* base, int slot, int nt) { return base[slot * nt + threadIdx.x]; }

// 32-byte packs are stored as two 16-byte columns so that consecutive threads stay on consecutive banks
AB_DEV void st_pack(Pack<float, 8>* base, int slot, int nt, const Pack<float, 8>& v) {
  float4* b = reinterpret_cast<float4*>(base);
  b[(slot * 2 + 0) * nt + threadIdx.x] = make_float4(v.v[0], v.v[1], v.v[2], v.v[3]);
  b[(slot * 2 + 1) * nt + threadIdx.x] = make_float4(v.v[4], v.v[5], v.v[6], v.v[7]);
}
AB_DEV Pack<float, 8> ld_pack(const Pack<float, 8>* base, int slot, int nt) {
  const float4* b = reinterpret_cast<const float4*>(base);
  const float4 lo = b[(slot * 2 + 0) * nt + threadIdx.x], hi = b[(slot * 2 + 1) * nt + threadIdx.x];
  Pack<float, 8> r;
  r.v[0] = lo.x; r.v[1] = lo.y; r.v[2] = lo.z; r.v[3] = lo.w;
  r.v[4] = hi.x; r.v[5] = hi.y; r.v[6] = hi.z; r.v[7] = hi.w;
  return r;
}

template <typename T, int W>
struct StackIO {
  typedef Pack<T, W> P;
  static constexpr int cols = 1;
  static AB_DEV void st(P* base, int slot, int nt, const P& v) { st_pack(base, slot, nt, v); }
  static AB_DEV P ld(const P* base, int slot, int nt) { return ld_pack(base, slot, nt); }
};
template <typename S>
struct StackOf;
template <typename T, int W>
struct StackOf<Pack<T, W>> {
  typedef Pack<T, W> P;
  static constexpr int cols = 1;
  static AB_DEV void st(P* base, int slot, int nt, const P& v) { st_pack(base, slot, nt, v); }
  static AB_DEV P ld(const P* base, int slot, int nt) { return ld_pack(base, slot, nt); }
};
template <typename Pk, int K>
struct StackOf<Dual<Pk, K>> {
  typedef Pk P;
  static constexpr int cols = 1 + K;
  static AB_DEV void st(P* base, int slot, int nt, const Dual<Pk, K>& v) {
    st_pack(base, slot * cols, nt, v.v);
#pragma unroll
    for (int k = 0; k < K; k++) st_pack(base, slot * cols + 1 + k, nt, v.d[k]);
  }
  static AB_DEV Dual<Pk, K> ld(const P* base, int slot, int nt) {
    Dual<Pk, K> r;
    r.v = ld_pack(base, slot * cols, nt);
#pragma unroll
    for (int k = 0; k < K; k++) r.d[k] = ld_pack(base, slot * cols + 1 + k, nt);
    return r;
  }
};

// ---- 128-bit stores ---------------------------------------------------------------------------------------------------------
// AB_STORE_POLICY: 0 = streaming (st.global.cs: the field is written once and not read back by this kernel), 1 = default
// write-back, 2 = st.global.cg, 3 = write-through (measured on B200 in profiles/r02_jit_sweep.md), 4 = multimem.st: `out`
// is the MULTICAST address of a symmetric allocation (NVLS), so one store lands in the same place of every GPU's buffer
// and the field is assembled on all ranks by the evaluation itself (distributed.evaluate_multicast), no gather pass.
#ifndef AB_STORE_POLICY
#define AB_STORE_POLICY 0
#endif
#if AB_STORE_POLICY == 4
AB_DEV void ab_st(float4* p, const float4& v) {
  asm volatile("multimem.st.weak.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
AB_DEV void ab_st(float2* p, const float2& v) {
  asm volatile("multimem.st.weak.global.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory");
}
AB_DEV void ab_st(float* p, const float& v) { asm volatile("multimem.st.weak.global.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory"); }
AB_DEV void ab_st(double* p, const double& v) { asm volatile("multimem.st.weak.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory"); }
AB_DEV void ab_st(double2* p, const double2& v) {  // (no .v2.f64 form: the 16 bytes travel as four 32-bit lanes)
  const float a = __int_as_float(__double2loint(v.x)), b = __int_as_float(__double2hiint(v.x));
  const float c = __int_as_float(__double2loint(v.y)), d = __int_as_float(__double2hiint(v.y));
  asm volatile("multimem.st.weak.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
#else
template <typename V>
AB_DEV void ab_st(V* p, const V& v) {
#if AB_STORE_POLICY == 0
  __stcs(p, v);
#elif AB_STORE_POLICY == 1
  *p = v;
#elif AB_STORE_POLICY == 2
  __stcg(p, v);
#else
  __stwt(p, v);
#endif
}
#endif
AB_DEV void store_pack(float* dst, const Pack<float, 4>& v, uint64_t idx, uint64_t n, bool aligned) {
  if (aligned && idx + 4 <= n) {
    ab_st(reinterpret_cast<float4*>(dst + idx), make_float4(v.v[0], v.v[1], v.v[2], v.v[3]));
  } else {
#pragma unroll
    for (int i = 0; i < 4; i++)
      if (idx + i < n) ab_st(dst + idx + i, v.v[i]);
  }
}
AB_DEV void store_pack(float* dst, const Pack<float, 8>& v, uint64_t idx, uint64_t n, bool aligned) {
  if (aligned && idx + 8 <= n) {
    ab_st(reinterpret_cast<float4*>(dst + idx), make_float4(v.v[0], v.v[1], v.v[2], v.v[3]));
    ab_st(reinterpret_cast<float4*>(dst + idx) + 1, make_float4(v.v[4], v.v[5], v.v[6], v.v[7]));
  } else {
#pragma unroll
    for (int i = 0; i < 8; i++)
      if (idx + i < n) ab_st(dst + idx + i, v.v[i]);
  }
}
AB_DEV void store_pack(float* dst, const Pack<float, 2>& v, uint64_t idx, uint64_t n, bool aligned) {
  if (aligned && idx + 2 <= n) {
    ab_st(reinterpret_cast<float2*>(dst + idx), make_float2(v.v[0], v.v[1]));
  } else {
#pragma unroll
    for (int i = 0; i < 2; i++)
      if (idx + i < n) ab_st(dst + idx + i, v.v[i]);
  }
}
AB_DEV void store_pack(double* dst, const Pack<double, 2>& v, uint64_t idx, uint64_t n, bool aligned) {
  if (aligned && idx + 2 <= n) {
    ab_st(reinterpret_cast<double2*>(dst + idx), make_double2(v.v[0], v.v[1]));
  } else {
#pragma unroll
    for (int i = 0; i < 2; i++)
      if (idx + i < n) ab_st(dst + idx + i, v.v[i]);
  }
}
template <typename T>
AB_DEV void store_pack(T* dst, const Pack<T, 1>& v, uint64_t idx, uint64_t n, bool) {
  if (idx < n) ab_st(dst + idx, v.v[0]);
}

// Pack<float, 8> through a per-warp transposition in shared memory: a thread owns 8 consecutive points (32 bytes), so its
// two direct 128-bit stores would each cover only half of every 32-byte sector the warp touches. Staged through 1 KB of
// shared memory per warp (two conflict-free STS.128 + two LDS.128, __syncwarp), every STG.128 of the warp writes 512
// contiguous bytes. `stage` = this warp's 64 float4; idx0 = first local point of the WARP (lane 0's idx).
AB_DEV void store_pack_w8_transposed(float* dst, const Pack<float, 8>& v, uint32_t idx0, uint64_t n, bool aligned, float4* stage) {
  const int lane = threadIdx.x & 31;
  auto swz = [](int i) { return i ^ ((i >> 3) & 1); };
  stage[swz(2 * lane)] = make_float4(v.v[0], v.v[1], v.v[2], v.v[3]);
  stage[swz(2 * lane + 1)] = make_float4(v.v[4], v.v[5], v.v[6], v.v[7]);
  __syncwarp();
  const float4 a = stage[swz(lane)], b = stage[swz(32 + lane)];
  __syncwarp();
  const uint64_t ia = (uint64_t)idx0 + 4 * lane, ib = ia + 128;
  if (aligned && ib + 4 <= n) {
    ab_st(reinterpret_cast<float4*>(dst + ia), a);
    ab_st(reinterpret_cast<float4*>(dst + ib), b);
  } else {
    const float va[4] = {a.x, a.y, a.z, a.w}, vb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
    for (int i = 0; i < 4; i++) {
      if (ia + i < n) ab_st(dst + ia + i, va[i]);
      if (ib + i < n) ab_st(dst + ib + i, vb[i]);
    }
  }
}

// ---- seeding ------------------------------------------------------------------------------------------------------------
template <typename T, int W>
AB_DEV void seed(Pt<Pack<T, W>>& p, const Pack<T, W>& x, const Pack<T, W>& y, const Pack<T, W>& z) {
  p.x = x;
  p.y = y;
  p.z = z;
}
template <typename T, int W, int K>
AB_DEV void seed(Pt<Dual<Pack<T, W>, K>>& p, const Pack<T, W>& x, const Pack<T, W>& y, const Pack<T, W>& z) {
  typedef Dual<Pack<T, W>, K> D;
  p.x = D(x);
  p.y = D(y);
  p.z = D(z);
  if (K == 3) {  // spatial tangents: d/dx, d/dy, d/dz
    p.x.d[0] = Pack<T, W>(T(1));
    p.y.d[1 % K] = Pack<T, W>(T(1));
    p.z.d[2 % K] = Pack<T, W>(T(1));
  }
}
template <typename T, int W>
AB_DEV void emit(const KParams<T>& kp, const Pack<T, W>& acc, uint32_t idx, bool aligned) {
  store_pack(kp.out, acc, idx, kp.n, aligned);
}
template <typename T, int W, int K>
AB_DEV void emit(const KParams<T>& kp, const Dual<Pack<T, W>, K>& acc, uint32_t idx, bool aligned) {
  store_pack(kp.out, acc.v, idx, kp.n, aligned);
  const bool ga = aligned && (kp.grad_stride % W == 0);
#pragma unroll
  for (int k = 0; k < K; k++) store_pack(kp.grad + (uint64_t)k * kp.grad_stride, acc.d[k], idx, kp.n, ga);
}

// ---- compact tiles (program-compiled kernels with warp-cooperative ops, 3D grids) ---------------------------------------------
// The flat walk above gives a warp 32 W CONSECUTIVE points: a 0.37-long needle on the 1025^3 headline grid. Warp-
// cooperative ops (nearest curve instance: candidates = instances within d_min + 2 R of the warp's reference point, R = warp
// radius) want a small R. Here a CTA of 128 threads owns a tile of TR rows (i1) x 16 columns (i2) of one i0 plane, W = 2 or
// 4 points per thread along i2; a warp covers 4 (8) rows x 16 columns (R is ~4x smaller) and a thread's points never
// straddle a row. SPOMSO rows have an odd length, so a fixed column grid would start every row segment at a different offset inside
// its 32-byte sector (measured: 37 % more DRAM traffic than the algorithmic bytes, read-modify-write of half-written
// sectors). The column blocks are therefore anchored per ROW at the row's first 32-byte boundary in the OUTPUT buffer:
// every 64-byte segment a warp stores is two whole sectors and every thread's pair is 8-byte aligned; the price is one
// extra, partly masked column block per row.
constexpr uint32_t kTileCols = 16;
// rows of a tile for W points per thread: a warp covers 32 W / 16 rows x 16 columns (W = 2: 4 x 16, W = 4: 8 x 16, about the
// same warp radius), a CTA of 4 warps stacks them: 16 rows (W = 2) or 32 rows (W = 4)
__host__ __device__ constexpr uint32_t compact_tile_rows(int W) { return 8u * (uint32_t)W; }
struct CompactWalk {
  uint32_t b0, b1, b2;  // tile coordinates: i0 plane (local to the launch), row block, column block
};
__host__ __device__ inline uint32_t compact_col_blocks(uint32_t n2) { return (n2 + kTileCols - 1) / kTileCols + 1; }
template <typename T>
AB_DEV void compact_walk_begin(const KParams<T>& kp, uint32_t nb1, uint32_t nb2, CompactWalk& w) {
  const uint32_t t = blockIdx.x;
  w.b0 = t / (nb1 * nb2);
  const uint32_t rem = t - w.b0 * (nb1 * nb2);
  w.b1 = rem / nb2;
  w.b2 = rem - w.b1 * nb2;
}
// coordinates of this thread's W points of the current tile, their flat index in the launch's output and validity (bit j of
// `valid` = point j is inside the grid); then the step to the CTA's next tile (tile_stride[] = gridDim.x decomposed over
// (plane blocks, row blocks, column blocks))
template <typename T, int W>
AB_DEV void compact_coords(const KParams<T>& kp, CompactWalk& w, uint32_t nb1, uint32_t nb2, Pack<T, W>& cx, Pack<T, W>& cy,
                           Pack<T, W>& cz, uint32_t& idx, uint32_t& valid) {
  constexpr uint32_t per_row = kTileCols / W;   // threads along a row segment
  constexpr uint32_t warp_rows = 32 / per_row;  // rows of one warp
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t i1 = w.b1 * compact_tile_rows(W) + warp * warp_rows + lane / per_row;
  const uint32_t row0 = (w.b0 * kp.g.n1 + i1) * kp.g.n2;  // flat index of the row's first sample
  // samples of this row before its first 32-byte boundary in the output buffer (0 .. 32 / sizeof(T) - 1)
  constexpr uint32_t per_sector = 32 / sizeof(T);
  const uint32_t lead = (per_sector - (uint32_t)((reinterpret_cast<uintptr_t>(kp.out) / sizeof(T) + row0) % per_sector)) % per_sector;
  // block b2 holds columns [lead + 16 (b2 - 1), lead + 16 b2): block 0 is the (short) lead-in up to the boundary
  const int32_t i2 = (int32_t)(lead + w.b2 * kTileCols + (lane % per_row) * W) - (int32_t)kTileCols;
  const bool row_ok = i1 < kp.g.n1;
  valid = 0;
#pragma unroll
  for (int j = 0; j < W; j++) valid |= (row_ok && i2 + j >= 0 && i2 + j < (int32_t)kp.g.n2) ? (1u << j) : 0u;
  const uint32_t c1 = row_ok ? i1 : kp.g.n1 - 1;
  // masked lanes: a nearby position (their coordinates only have to be finite)
  const int32_t c2 = i2 < -(W - 1) ? -(W - 1) : (i2 >= (int32_t)kp.g.n2 ? (int32_t)kp.g.n2 - 1 : i2);
  cx = Pack<T, W>(grid_coord(kp.g, 0, w.b0 + kp.g.i0_begin, T()));
  cy = Pack<T, W>(grid_coord(kp.g, 1, c1, T()));
  grid_coord_run(kp.g, 2, c2, cz);
  idx = row0 + (uint32_t)i2;  // (wraps for masked lanes, which never store)
  w.b2 += kp.tile_stride[2];
  if (w.b2 >= nb2) {
    w.b2 -= nb2;
    w.b1++;
  }
  w.b1 += kp.tile_stride[1];
  if (w.b1 >= nb1) {
    w.b1 -= nb1;
    w.b0++;
  }
  w.b0 += kp.tile_stride[0];
}
template <typename T, int W>
AB_DEV void store_masked(T* dst, const Pack<T, W>& v, uint32_t idx, uint32_t valid) {
  T* p = dst + idx;
  if (valid == (1u << W) - 1 && (reinterpret_cast<uintptr_t>(p) & (W * sizeof(T) - 1)) == 0) {
    store_pack(dst, v, idx, (uint64_t)idx + W, true);
  } else {
#pragma unroll
    for (int j = 0; j < W; j++)
      if (valid & (1u << j)) ab_st(p + j, v.v[j]);
  }
}
template <typename T, int W>
AB_DEV void emit_compact(const KParams<T>& kp, const Pack<T, W>& acc, uint32_t idx, uint32_t valid) {
  store_masked(kp.out, acc, idx, valid);
}
template <typename T, int W, int K>
AB_DEV void emit_compact(const KParams<T>& kp, const Dual<Pack<T, W>, K>& acc, uint32_t idx, uint32_t valid) {
  store_masked(kp.out, acc.v, idx, valid);
#pragma unroll
  for (int k = 0; k < K; k++) store_masked(kp.grad + (uint64_t)k * kp.grad_stride, acc.d[k], idx, valid);
}

// P_FIELD: the value of a precomputed per-point field (the output of a grid stencil), indexed like `out`
template <typename T, int W>
AB_DEV void load_field(const void* field, uint32_t idx, uint64_t n, Pack<T, W>& out) {
  const T* f = reinterpret_cast<const T*>(field);
#pragma unroll
  for (int j = 0; j < W; j++) out.v[j] = f[idx + j < n ? idx + j : n - 1];
}
template <typename T, int W, int K>
AB_DEV void load_field(const void* field, uint32_t idx, uint64_t n, Dual<Pack<T, W>, K>& out) {
  Pack<T, W> v;
  load_field(field, idx, n, v);
  out = Dual<Pack<T, W>, K>(v);  // zero tangents (rejected on the host for the gradient modes anyway)
}
// with the tangent row of the field (AB_GRAD_PARAM: the stencil applied to d field / d theta), same index clamp; the value
// kernels ignore it, the spatial ones never get here (the host rejects P_FIELD there)
template <typename T, int W>
AB_DEV void load_field(const void* field, const void*, uint32_t idx, uint64_t n, Pack<T, W>& out) {
  load_field(field, idx, n, out);
}
template <typename T, int W>
AB_DEV void load_field(const void* field, const void* dfield, uint32_t idx, uint64_t n, Dual<Pack<T, W>, 1>& out) {
  load_field(field, idx, n, out.v);
  load_field(dfield, idx, n, out.d[0]);
}
template <typename T, int W, int K>
AB_DEV void load_field(const void* field, const void*, uint32_t idx, uint64_t n, Dual<Pack<T, W>, K>& out) {
  load_field(field, idx, n, out);
}

// loss mode of the parameter-tangent kernel: r = F - target, sums of r^2 and 2 r dF/dtheta in double
template <typename T, int W, int K>
AB_DEV void accumulate_loss(const KParams<T>& kp, const Dual<Pack<T, W>, K>& acc, uint32_t idx, double& loss, double& dloss) {
#pragma unroll
  for (int j = 0; j < W; j++) {
    if (idx + j < kp.n) {
      const double r = (double)(acc.v.v[j] - kp.target[idx + j]);
      loss += r * r;
      dloss += 2.0 * r * (double)acc.d[0].v[j];
    }
  }
}
template <typename T, int W>
AB_DEV void accumulate_loss(const KParams<T>&, const Pack<T, W>&, uint32_t, double&, double&) {}

// nearest cloud point inside the interpreter (sdf_3D.py:283-286), for a cloud that sits anywhere in a tree: queries arrive
// already warped by the ops above the leaf. Large clouds come with an octree (built by the host per call, ab_tree.cuh) and
// every lane walks it; small ones are scanned with uniform (broadcast) loads. Same (q-p)^2 expression either way, so the
// two agree to the bit (up to which of two exactly equidistant points wins). The walk is inlined on purpose: as a
// __noinline__ function (divergent loops inside a callee) it returned wrong winners / faulted when called from this kernel
// with nvcc 12.9, while the identical code inlined, or called from a small kernel, is correct.
template <typename T>
AB_DEV uint32_t cloud_nearest_tree(const TreeRef<T>& t, T x, T y, T z, int dim) {
  T best;
  uint32_t bi;
  // every lane of the warp is here with a neighbouring sample (the op stream is warp-uniform): walk the tree once for all
  if (dim == 3) tree_nearest_packet<T, 3, 0, true>(t, x, y, z, best, bi);
  else tree_nearest_packet<T, 2, 0, true>(t, x, y, T(0), best, bi);
  return bi;
}

template <typename S, typename T>
AB_DEV S prim_point_cloud(const Pt<S>& p, const void* __restrict__ cloud_v, uint32_t m, int dim, const void* tree_v) {
  typedef typename Vec4<T>::type V4;
  const V4* __restrict__ cloud = reinterpret_cast<const V4*>(cloud_v);
  constexpr int W = S::width;
  auto vx = value_of(p.x), vy = value_of(p.y), vz = value_of(p.z);
  T best[W];
  uint32_t bi[W];
  if (tree_v) {
    const TreeRef<T> tree = *reinterpret_cast<const TreeRef<T>*>(tree_v);
    cloud = tree.pts;  // winners are positions in the cell-ordered copy
#pragma unroll 1
    for (int i = 0; i < W; i++) bi[i] = cloud_nearest_tree<T>(tree, vx.v[i], vy.v[i], vz.v[i], dim);
  } else {
#pragma unroll
    for (int i = 0; i < W; i++) {
      best[i] = T(3.0e38);
      bi[i] = 0;
    }
    for (uint32_t j = 0; j < m; j++) {
      const V4 c = cloud[j];
#pragma unroll
      for (int i = 0; i < W; i++) {
        T dx = vx.v[i] - (T)c.x, dy = vy.v[i] - (T)c.y, dz = (dim == 3) ? vz.v[i] - (T)c.z : T(0);
        T d2 = s_fma(dx, dx, s_fma(dy, dy, dz * dz));
        if (d2 < best[i]) {
          best[i] = d2;
          bi[i] = j;
        }
      }
    }
  }
  // rebuild the distance to the winner with tangents (d|q-c|/dq = (q-c)/|q-c|)
  Pack<T, W> cx, cy, cz;
#pragma unroll
  for (int i = 0; i < W; i++) {
    const V4 c = cloud[bi[i]];
    cx.v[i] = (T)c.x;
    cy.v[i] = (T)c.y;
    cz.v[i] = (dim == 3) ? (T)c.z : T(0);
  }
  S dx = add_lane(p.x, -cx), dy = add_lane(p.y, -cy);
  if (dim == 3) return norm3_(dx, dy, add_lane(p.z, -cz));
  return norm2_(dx, dy);
}

__host__ __device__ inline size_t prog_ops_bytes(uint32_t n_ops) { return ((size_t)n_ops * sizeof(uint2) + 15) & ~(size_t)15; }
template <typename T>
__host__ __device__ inline size_t prog_args_bytes(uint32_t n_args) { return ((size_t)n_args * sizeof(T) + 15) & ~(size_t)15; }

// fused PUSH_V after a combine op (b = V slot + 1, 0 = none)
#define AB_CPUSH                                  \
  do {                                            \
    if (sb) SK::st(vstack, sb - 1, NT, acc);      \
  } while (0)

// ---- the interpreter -------------------------------------------------------------------------------------------------------
// TIER 0 ("lite") contains only the ops without transcendental functions or tables (stack, affine family, elongate,
// mirror core, symmetry, revolve, infinite repetition, the value ops, the polynomial combines and the sqrt-only
// primitives): 40 registers instead of ~120, so 3x the resident warps, and a 23 KB body instead of 170 KB. The host
// picks the smallest tier that covers the program (op_tier below). TIER 1 adds every op with one transcendental or a
// small table (twist, bend, rotational symmetry, instancing, Boltzmann combines, post-processing maps, cones, arcs,
// n-gons ...) at 72 registers; TIER 2 adds the widest primitives (triangles, quads, sectors, solid angles, polylines, polygons, point clouds).
// minimum resident CTAs per SM asked of the register allocator, per tier (128-thread CTAs): lite 6, mid 5, full 4
template <typename S>
struct IsDual { static constexpr bool value = false; };
template <typename P, int K>
struct IsDual<Dual<P, K>> { static constexpr bool value = true; };
// resident CTAs per SM the kernels are compiled for (register cap 65536 / (128 n)); measured on B200: the mid duals are
// best at 7 (72 registers, no spills; 8 costs C3+gradient 15 %), the lite kernels at 8 (64 registers)
#ifndef AB_MID_CTAS
#define AB_MID_CTAS 7
#endif
#ifndef AB_LITE_CTAS
#define AB_LITE_CTAS 8
#endif
#ifndef AB_FULL_CTAS
#define AB_FULL_CTAS 4
#endif
template <typename S, int TIER>
__host__ __device__ constexpr int min_ctas() {  // the wide lite dual kernel (4 points x 4 components) needs ~3x the registers
#ifdef AB_SPEC_MIN_CTAS
  return AB_SPEC_MIN_CTAS;  // specialised build: the caller knows which op set it compiled
#endif
  if (sizeof(typename S::scalar) == 8) return TIER <= 1 ? 6 : 4;  // fp64 values take two registers: keep the 80-register cap
  return (IsDual<S>::value && S::width >= 4) ? 3 : (TIER == 0 ? AB_LITE_CTAS : (TIER == 1 ? AB_MID_CTAS : AB_FULL_CTAS));
}

#ifndef AB_BIG_CTA
#define AB_BIG_CTA 0
#endif
// AB_BIG_CTA (experiment): one CTA of AB_BIG_CTA threads per SM for the mid/full tiers; the warps that share an SM
// sub-partition (wid % 4) are kept in lockstep with a named barrier per op, so they fetch every op body once instead of
// thrashing the per-sub-partition instruction cache from unrelated program positions.
template <typename S, int TIER>
__host__ __device__ constexpr bool big_cta() { return AB_BIG_CTA > 0 && TIER >= 1 && !(IsDual<S>::value && S::width >= 4); }
template <typename S, int TIER>
__host__ __device__ constexpr int max_threads() { return big_cta<S, TIER>() ? AB_BIG_CTA : 128; }

template <typename S, typename T, int TIER, bool PARAM = false>
__global__ void __launch_bounds__((max_threads<S, TIER>()), (big_cta<S, TIER>() ? 1 : min_ctas<S, TIER>())) ab_interp_kernel(const __grid_constant__ KParams<T> kp) {
  static_assert(TIER == AB_TIER_FULL, "one tier per translation unit");
  constexpr int W = S::width;
  const int NT = blockDim.x;
  typedef Pack<T, W> P;
  typedef StackOf<S> SK;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // shared memory: [ops][args][P stack][V stack]. The program is staged once per (persistent) CTA; afterwards every op
  // fetch is one broadcast LDS.64 and its arguments come in with 128-bit broadcast loads.
  uint2* s_ops = reinterpret_cast<uint2*>(smem_raw);
  T* s_args = reinterpret_cast<T*>(smem_raw + kp.off_args);
  P* pstack = reinterpret_cast<P*>(smem_raw + kp.off_pstack);  // [n_pslots*3*cols][NT]
  P* vstack = reinterpret_cast<P*>(smem_raw + kp.off_vstack);  // [n_vslots*cols][NT]
  for (uint32_t i = threadIdx.x; i < kp.n_ops; i += NT) s_ops[i] = kp.ops[i];
  for (uint32_t i = threadIdx.x; i < kp.n_args; i += NT) s_args[i] = kp.args[i];
  __syncthreads();

  const uint32_t tile_pts = (uint32_t)NT * W;
  const uint32_t n32 = (uint32_t)kp.n;
  const uint32_t n_tiles = (n32 + tile_pts - 1) / tile_pts;
  TileWalk walk;
  tile_walk_begin(kp, tile_pts, (uint32_t)W, walk);

  double loss_sum = 0.0, dloss_sum = 0.0;  // loss mode only (PARAM kernels)
  for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const uint32_t idx = tile * tile_pts + threadIdx.x * W;  // first local point of this thread
    P cx, cy, cz;
    tile_coords(kp, walk, idx, n32, cx, cy, cz);

    Pt<S> p;
    seed(p, cx, cy, cz);
    S acc = constant_like(p.x, T(0));

    for (uint32_t pc = 0; pc < kp.n_ops; pc++) {
      // one 64-bit broadcast load per op. Dispatch: with an unmasked 32-bit switch variable nvcc emits one indexed
      // branch (LDC of the table entry + BRX); with a value it can narrow to 8/16 bits it emits a ~7-level tree of
      // uniform compares and branches. Measured on B200 (profiles/r01_sweeps.md) the tree is FASTER here (C1: 254 vs
      // 228 Gpts/s): the indexed branch waits on a dependent constant load and resolves late, the uniform tree does not.
      if constexpr (big_cta<S, TIER>()) {
        const int part = (threadIdx.x >> 5) & 3;
        asm volatile("bar.sync %0, %1;" ::"r"(1 + part), "r"(NT / 4));
      }
      const uint2 w = s_ops[pc];
      const uint32_t code = AB_DISPATCH_BRX ? w.x : (w.x & 0xffu);
      const int sa = (int)((w.y >> 16) & 0xffu), sb = (int)(w.y >> 24);
      const T* a_val = reinterpret_cast<const T*>(__builtin_assume_aligned(s_args + (w.y & 0xffffu), 16));
      // PARAM: every argument is read as a dual number carrying d arg / d theta (ab_ops.cuh, ArgD)
      typename std::conditional<PARAM, ArgD<S>, const T*>::type a;
      if constexpr (PARAM) a = ArgD<S>{a_val, a_val + kp.dargs_off};
      else a = a_val;
      switch (code) {
        case D_END: break;
        case D_SAVE_P:
          SK::st(pstack, sa * 3 + 0, NT, p.x);
          SK::st(pstack, sa * 3 + 1, NT, p.y);
          SK::st(pstack, sa * 3 + 2, NT, p.z);
          break;
        case D_LOAD_P:
          p.x = SK::ld(pstack, sa * 3 + 0, NT);
          p.y = SK::ld(pstack, sa * 3 + 1, NT);
          p.z = SK::ld(pstack, sa * 3 + 2, NT);
          break;
#if AB_SPEC_PUSH_V
        case D_PUSH_V: SK::st(vstack, sa, NT, acc); break;
#endif
        // fused [PUSH_V] + LOAD_P + transform (program.py::_fuse): one dispatch per child of a combine chain
        case D_NEXT_AFFINE:
        case D_NEXT_TRANSLATE:
        case D_NEXT_LOAD:
          if (sb) SK::st(vstack, sb - 1, NT, acc);
          p.x = SK::ld(pstack, sa * 3 + 0, NT);
          p.y = SK::ld(pstack, sa * 3 + 1, NT);
          p.z = SK::ld(pstack, sa * 3 + 2, NT);
          if (code == D_NEXT_AFFINE) op_affine(p, a);
          else if (code == D_NEXT_TRANSLATE) op_translate(p, a);
          break;
        // coordinate ops
#if AB_SPEC_AFFINE
        case D_AFFINE: op_affine(p, a); break;
#endif
#if AB_SPEC_TRANSLATE
        case D_TRANSLATE: op_translate(p, a); break;
#endif
#if AB_SPEC_SCALE_P
        case D_SCALE_P: op_scale_p(p, a); break;
#endif
#if AB_SPEC_ELONGATE
        case D_ELONGATE: op_elongate(p, a); break;
#endif
#if AB_TIER_FULL
#if AB_SPEC_TWIST
        case D_TWIST: op_twist(p, a); break;
#endif
#endif
#if AB_TIER_FULL
#if AB_SPEC_BEND
        case D_BEND: op_bend(p, a); break;
#endif
#endif
#if AB_SPEC_ABSX_SUB
        case D_ABSX_SUB: op_absx_sub(p, a); break;
#endif
        case D_SYMMETRY:
          if (sa == 0) p.x = abs_(p.x);
          else if (sa == 1) p.y = abs_(p.y);
          else p.z = abs_(p.z);
          break;
#if AB_TIER_FULL
#if AB_SPEC_ROTSYM
        case D_ROTSYM: op_rotsym(p, a); break;
#endif
#endif
#if AB_SPEC_REVOLVE
        case D_REVOLVE: op_revolve(p, a); break;
#endif
#if AB_TIER_FULL
#if AB_SPEC_AXIS_REVOLVE
        case D_AXIS_REVOLVE: op_axis_revolve(p, a); break;
#endif
#endif
#if AB_SPEC_REP_INF
        case D_REP_INF: op_rep_inf(p, a); break;
#endif
#if AB_TIER_FULL
#if AB_SPEC_REP_FIN
        case D_REP_FIN: op_rep_fin(p, a); break;
#endif
#endif
#if AB_TIER_FULL
#if AB_SPEC_LIN_INST
        case D_LIN_INST: op_lin_inst(p, a, sa); break;
#endif
#endif
#if AB_TIER_FULL
#if AB_SPEC_CURVE_INST
        case D_CURVE_INST: op_curve_inst(p, a, sa); break;
#endif
#endif
#if AB_SPEC_ZERO_Z
        case D_ZERO_Z: p.z = constant_like(p.z, T(0)); break;
#endif
        // value ops
#if AB_SPEC_ROUND
        case D_ROUND: acc = acc - a[0]; break;
#endif
#if AB_SPEC_ABS
        case D_ABS: acc = abs_(acc); break;
#endif
#if AB_SPEC_NEG
        case D_NEG: acc = -acc; break;
#endif
#if AB_SPEC_SIGN
        case D_SIGN: acc = sign_(acc); break;
#endif
#if AB_SPEC_ONION
        case D_ONION: acc = abs_(acc) - a[0]; break;
#endif
#if AB_SPEC_CONCENTRIC
        case D_CONCENTRIC: acc = abs_(acc - a[0]); break;
#endif
#if AB_SPEC_SCALE_V
        case D_SCALE_V: acc = acc * a[0]; break;
#endif
        case D_EXTRUDE_BEGIN:
          SK::st(vstack, sa, NT, abs_(p.z) - a[0]);
          p.z = constant_like(p.z, T(0));
          break;
#if AB_SPEC_EXTRUDE_END
        case D_EXTRUDE_END: acc = op_extrude_end<S, T>(acc, SK::ld(vstack, sa, NT)); break;
#endif
#if AB_TIER_FULL >= 2
        case D_POLY_SIGN:
          acc = op_poly_sign(acc, SK::ld(pstack, sa * 3 + 0, NT), SK::ld(pstack, sa * 3 + 1, NT), a, sb);
          break;
#endif
        // post-processing (post_processing.py:380-560)
#if AB_TIER_FULL
#if AB_SPEC_PP_SIGMOID
        case D_PP_SIGMOID: acc = pp_sigmoid(acc, a); break;
#endif
#endif
#if AB_TIER_FULL
        case D_PP_POS_SIGMOID: acc = pp_pos_sigmoid(acc, a); break;
#endif
#if AB_TIER_FULL
#if AB_SPEC_PP_CAPPED_EXP
        case D_PP_CAPPED_EXP: acc = pp_capped_exp(acc, a); break;
#endif
#endif
#if AB_TIER_FULL
        case D_PP_HARD_BIN: acc = pp_hard_bin(acc, a); break;
#endif
#if AB_TIER_FULL
#if AB_SPEC_PP_LINEAR
        case D_PP_LINEAR: acc = pp_linear(acc, a); break;
#endif
#endif
#if AB_TIER_FULL
#if AB_SPEC_PP_RELU
        case D_PP_RELU: acc = pp_relu(acc, a); break;
#endif
#endif
#if AB_TIER_FULL
        case D_PP_SMOOTH_RELU: acc = pp_smooth_relu(acc, a); break;
#endif
#if AB_TIER_FULL
        case D_PP_SLOWSTART: acc = pp_slowstart(acc, a); break;
#endif
#if AB_TIER_FULL
        case D_PP_GAUSS_BOUNDARY: acc = pp_gauss_boundary(acc, a); break;
#endif
#if AB_TIER_FULL
        case D_PP_GAUSS_FALLOFF: acc = pp_gauss_falloff(acc, a); break;
#endif
        // combine: acc = f(V[a], acc)
#if AB_SPEC_C_UNION
        case D_C_UNION: acc = min_(SK::ld(vstack, sa, NT), acc); AB_CPUSH; break;
#endif
#if AB_SPEC_C_INTERSECT
        case D_C_INTERSECT: acc = max_(SK::ld(vstack, sa, NT), acc); AB_CPUSH; break;
#endif
#if AB_SPEC_C_SUBTRACT
        case D_C_SUBTRACT: acc = max_(SK::ld(vstack, sa, NT), -acc); AB_CPUSH; break;
#endif
#if AB_SPEC_C_SUM
        case D_C_SUM: acc = SK::ld(vstack, sa, NT) + acc; AB_CPUSH; break;
#endif
#if AB_SPEC_C_DIFF
        case D_C_DIFF: acc = SK::ld(vstack, sa, NT) - acc; AB_CPUSH; break;
#endif
#if AB_SPEC_C_SMIN2
        case D_C_SMIN2: acc = smin_poly2(SK::ld(vstack, sa, NT), acc, a[0]); AB_CPUSH; break;
#endif
#if AB_SPEC_C_SMIN3
        case D_C_SMIN3: acc = smin_poly3(SK::ld(vstack, sa, NT), acc, a[0]); AB_CPUSH; break;
#endif
#if AB_SPEC_C_SMAX3
        case D_C_SMAX3: acc = -smin_poly3(-SK::ld(vstack, sa, NT), -acc, a[0]); AB_CPUSH; break;
#endif
#if AB_SPEC_C_SSUB3
        case D_C_SSUB3: acc = -smin_poly3(-SK::ld(vstack, sa, NT), acc, a[0]); AB_CPUSH; break;
#endif
#if AB_TIER_FULL
#if AB_SPEC_C_BOLTZ_INT
        case D_C_BOLTZ_INT: acc = smax_boltz(SK::ld(vstack, sa, NT), acc, a[0]); AB_CPUSH; break;
#endif
#endif
#if AB_TIER_FULL
#if AB_SPEC_C_BOLTZ_SUB
        case D_C_BOLTZ_SUB: acc = smax_boltz(SK::ld(vstack, sa, NT), -acc, a[0]); AB_CPUSH; break;
#endif
#endif
        // 3D primitives
#if AB_SPEC_P_SPHERE
        case D_P_SPHERE: acc = prim_sphere(p, a); break;
#endif
#if AB_SPEC_P_FIELD
        case D_P_FIELD: load_field(kp.blob[sb], kp.dblob[sb], idx, kp.n, acc); break;
#endif
#if AB_SPEC_P_CYLINDER
        case D_P_CYLINDER: acc = prim_cylinder(p, a); break;
#endif
#if AB_SPEC_P_BOX
        case D_P_BOX: acc = prim_box(p, a); break;
#endif
#if AB_SPEC_P_TORUS
        case D_P_TORUS: acc = prim_torus(p, a); break;
#endif
#if AB_SPEC_P_CHAINLINK
        case D_P_CHAINLINK: acc = prim_chainlink(p, a); break;
#endif
#if AB_TIER_FULL
#if AB_SPEC_P_BRAID
        case D_P_BRAID: acc = prim_braid(p, a); break;
#endif
#endif
#if AB_TIER_FULL
#if AB_SPEC_P_ARC3D
        case D_P_ARC3D: acc = prim_arc3d(p, a); break;
#endif
#endif
#if AB_SPEC_P_PLANE
        case D_P_PLANE: acc = prim_plane(p, a); break;
#endif
#if AB_SPEC_P_UPLANE
        case D_P_UPLANE: acc = prim_uplane(p, a); break;
#endif
#if AB_SPEC_P_SEGMENT
        case D_P_SEGMENT: acc = prim_segment(p, a); break;
#endif
#if AB_TIER_FULL
#if AB_SPEC_P_CONE
        case D_P_CONE: acc = prim_cone(p, a); break;
#endif
#endif
#if AB_TIER_FULL
#if AB_SPEC_P_OINF_CONE
        case D_P_OINF_CONE: acc = prim_inf_cone(p, a, true); break;
#endif
#endif
#if AB_TIER_FULL
#if AB_SPEC_P_INF_CONE
        case D_P_INF_CONE: acc = prim_inf_cone(p, a, false); break;
#endif
#endif
#if AB_TIER_FULL >= 2
#if AB_SPEC_P_SOLID_ANGLE
        case D_P_SOLID_ANGLE: acc = prim_solid_angle(p, a); break;
#endif
#endif
#if AB_TIER_FULL >= 2
#if AB_SPEC_P_TRIANGLE3D
        case D_P_TRIANGLE3D: acc = prim_triangle3d(p, a); break;
#endif
#endif
#if AB_TIER_FULL >= 2
#if AB_SPEC_P_QUAD3D
        case D_P_QUAD3D: acc = prim_quad3d(p, a); break;
#endif
#endif
#if AB_TIER_FULL >= 2
#if AB_SPEC_P_SEGLINE
        case D_P_SEGLINE: acc = prim_segline(p, a, 3); break;
#endif
#endif
        case D_P_AXIS:
          if (sa == 0) acc = p.x - a[0];
          else if (sa == 1) acc = p.y - a[0];
          else acc = p.z - a[0];
          break;
#if AB_TIER_FULL >= 2
#if AB_SPEC_P_POINT_CLOUD
        case D_P_POINT_CLOUD: acc = prim_point_cloud<S, T>(p, kp.blob[sb], kp.blob_count[sb], sa, kp.blob_tree[sb]); break;
#endif
#endif
        // 2D primitives
#if AB_SPEC_P_CIRCLE
        case D_P_CIRCLE: acc = prim_circle(p, a); break;
#endif
#if AB_TIER_FULL
#if AB_SPEC_P_NEU_CIRCLE
        case D_P_NEU_CIRCLE: acc = prim_neu_circle(p, a); break;
#endif
#endif
#if AB_SPEC_P_BOX2D
        case D_P_BOX2D: acc = prim_box2d(p, a); break;
#endif
#if AB_SPEC_P_SEGMENT2D
        case D_P_SEGMENT2D: acc = prim_segment2d(p, a); break;
#endif
#if AB_TIER_FULL
#if AB_SPEC_P_RBOX2D
        case D_P_RBOX2D: acc = prim_rbox2d(p, a); break;
#endif
#endif
#if AB_TIER_FULL >= 2
#if AB_SPEC_P_TRIANGLE2D
        case D_P_TRIANGLE2D: acc = prim_triangle2d(p, a); break;
#endif
#endif
#if AB_TIER_FULL
#if AB_SPEC_P_ARC
        case D_P_ARC: acc = prim_arc(p, a); break;
#endif
#endif
#if AB_TIER_FULL >= 2
#if AB_SPEC_P_SECTOR
        case D_P_SECTOR: acc = prim_sector(p, a); break;
#endif
#endif
#if AB_TIER_FULL
#if AB_SPEC_P_INF_SECTOR
        case D_P_INF_SECTOR: acc = prim_inf_sector(p, a); break;
#endif
#endif
#if AB_TIER_FULL
#if AB_SPEC_P_NGON
        case D_P_NGON: acc = prim_ngon(p, a); break;
#endif
#endif
#if AB_TIER_FULL >= 2
#if AB_SPEC_P_SEGLINE2D
        case D_P_SEGLINE2D: acc = prim_segline(p, a, 2); break;
#endif
#endif
#if AB_TIER_FULL >= 2
#if AB_SPEC_P_POLYGON2D
        case D_P_POLYGON2D: acc = prim_polygon2d(p, a); break;
#endif
#endif
        default: break;  // unknown opcodes are rejected on the host (AB_EUNSUPPORTED_OP)
      }
    }
    if constexpr (PARAM) {
      if (kp.loss_accum) {  // fused least-squares reduction: nothing is written per point
        accumulate_loss(kp, acc, idx, loss_sum, dloss_sum);
        continue;
      }
    }
    const bool aligned = ((reinterpret_cast<uintptr_t>(kp.out) & 15) == 0);
    emit(kp, acc, idx, aligned);
  }
  if constexpr (PARAM) {
    if (kp.loss_accum) {
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        loss_sum += __shfl_xor_sync(0xffffffffu, loss_sum, off);
        dloss_sum += __shfl_xor_sync(0xffffffffu, dloss_sum, off);
      }
      if ((threadIdx.x & 31) == 0) {
        atomicAdd(kp.loss_accum, loss_sum);
        atomicAdd(kp.loss_accum + 1, dloss_sum);
      }
    }
  }
}

// ---- launcher (one explicit instantiation per translation unit: ab_interp_*.cu) ---------------------------------------------
struct LaunchCfg {
  int sms;
  size_t smem_optin;
};
// returns cudaSuccess or the CUDA error; *status is AB_OK / AB_ETOOLARGE
template <typename S, typename T, int TIER, bool PARAM = false>
cudaError_t launch_interp(const KParams<T>& kp, const LaunchCfg& cfg, cudaStream_t st, int* status);

// ops whose argument count depends on the program (tables): the launcher packs them after the fixed-size arguments
inline bool is_table_op(int ab_opcode) {
  switch (ab_opcode) {
    case AB_OP_ROTSYM: case AB_OP_CURVE_INST: case AB_OP_P_SEGLINE: case AB_OP_P_SEGLINE2D: case AB_OP_P_POLYGON2D:
    case AB_OP_POLY_SIGN: return true;
    default: return false;
  }
}
// AB_GRAD_PARAM: args[kParamHalf + i] = d args[i] / d theta (second half of the pool)
constexpr uint32_t kParamHalf = (AB_MAX_ARGS / 2) & ~3u;

inline int op_tier(int ab_opcode);
inline bool is_lite_op(int ab_opcode) {
  switch (ab_opcode) {
    case AB_OP_END: case AB_OP_SAVE_P: case AB_OP_LOAD_P: case AB_OP_PUSH_V: case AB_OP_AFFINE: case AB_OP_TRANSLATE:
    case AB_OP_NEXT_AFFINE: case AB_OP_NEXT_TRANSLATE: case AB_OP_NEXT_LOAD:
    case AB_OP_SCALE_P: case AB_OP_ELONGATE: case AB_OP_ABSX_SUB: case AB_OP_SYMMETRY: case AB_OP_REVOLVE:
    case AB_OP_REP_INF: case AB_OP_ZERO_Z: case AB_OP_ROUND: case AB_OP_ABS: case AB_OP_NEG: case AB_OP_SIGN:
    case AB_OP_ONION: case AB_OP_CONCENTRIC: case AB_OP_SCALE_V: case AB_OP_EXTRUDE_BEGIN: case AB_OP_EXTRUDE_END:
    case AB_OP_C_UNION: case AB_OP_C_INTERSECT: case AB_OP_C_SUBTRACT: case AB_OP_C_SUM: case AB_OP_C_DIFF:
    case AB_OP_C_SMIN2: case AB_OP_C_SMIN3: case AB_OP_C_SMAX3: case AB_OP_C_SSUB3: case AB_OP_P_SPHERE:
    case AB_OP_P_CYLINDER: case AB_OP_P_BOX: case AB_OP_P_TORUS: case AB_OP_P_CHAINLINK: case AB_OP_P_PLANE:
    case AB_OP_P_UPLANE: case AB_OP_P_SEGMENT: case AB_OP_P_AXIS: case AB_OP_P_CIRCLE: case AB_OP_P_BOX2D:
    case AB_OP_P_SEGMENT2D: case AB_OP_P_FIELD:
      return true;
    default: return false;
  }
}

inline int op_tier(int ab_opcode) {
  if (is_lite_op(ab_opcode)) return 0;
  switch (ab_opcode) {
    case AB_OP_P_SOLID_ANGLE: case AB_OP_P_SECTOR: case AB_OP_P_TRIANGLE3D: case AB_OP_P_QUAD3D: case AB_OP_P_SEGLINE:
    case AB_OP_P_SEGLINE2D: case AB_OP_P_POINT_CLOUD: case AB_OP_P_TRIANGLE2D: case AB_OP_P_POLYGON2D: case AB_OP_POLY_SIGN:
      return 2;
    default: return 1;
  }
}

#ifdef AB_INTERP_INSTANTIATE
template <typename S, typename T, int TIER, bool PARAM>
cudaError_t launch_interp(const KParams<T>& kp, const LaunchCfg& cfg, cudaStream_t st, int* status) {
  typedef StackOf<S> SK;
  *status = AB_OK;
  const size_t per_thread = (size_t)sizeof(typename SK::P) * SK::cols * ((size_t)kp.n_pslots * 3 + kp.n_vslots);
  const size_t prog_bytes = prog_ops_bytes(kp.n_ops) + prog_args_bytes<T>(kp.n_args);
  // prefer 128 threads; shrink the CTA when the stacks would not leave room for >= 2 CTAs per SM
  int nt = 128;
  if (big_cta<S, TIER>()) nt = AB_BIG_CTA;
  else if (prog_bytes + per_thread * 128 > 96 * 1024) nt = 64;
  if (prog_bytes + per_thread * nt > cfg.smem_optin) nt = 32;
  const size_t smem = prog_bytes + per_thread * nt;
  if (smem > cfg.smem_optin) {
    *status = AB_ETOOLARGE;
    return cudaSuccess;
  }
  auto kern = ab_interp_kernel<S, T, TIER, PARAM>;
  cudaError_t e;
  if (smem > 48 * 1024) {
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  int occ = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, nt, smem);
  if (e != cudaSuccess) return e;
  if (occ < 1) {
    *status = AB_ETOOLARGE;
    return cudaSuccess;
  }
  const uint64_t tile_pts = (uint64_t)nt * S::width;
  const uint64_t n_tiles = (kp.n + tile_pts - 1) / tile_pts;
  const uint64_t resident = (uint64_t)cfg.sms * occ;  // persistent CTAs: a whole number of resident waves
  const unsigned grid = (unsigned)(n_tiles < resident ? n_tiles : resident);
  KParams<T>& k = const_cast<KParams<T>&>(kp);
  k.off_args = (uint32_t)prog_ops_bytes(kp.n_ops);
  k.off_pstack = (uint32_t)prog_bytes;
  k.off_vstack = (uint32_t)(prog_bytes + (size_t)sizeof(typename SK::P) * SK::cols * kp.n_pslots * 3 * nt);
  if (kp.grid_mode) {
    const uint64_t d = (uint64_t)grid * tile_pts;
    k.tile_stride[0] = (uint32_t)(d / kp.g.plane);
    const uint64_t rem = d % kp.g.plane;
    k.tile_stride[1] = (uint32_t)(rem / kp.g.n2);
    k.tile_stride[2] = (uint32_t)(rem % kp.g.n2);
  }
  kern<<<grid, nt, smem, st>>>(kp);
  return cudaGetLastError();
}
#endif

}  // namespace ab
