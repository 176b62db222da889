// ab_fields.cuh — kernels on whole fields that sit AFTER the interpreter in SPOMSO pipelines (SURVEY §8f N3, N4):
//   * ab_box_axis_kernel / ab_edge_kernel : conv_averaging / conv_edge_detection (post_processing.py:552-623), i.e.
//     scipy.ndimage.convolve with mode='reflect' restated tap by tap (oracle/fields_np.py documents the tap placement);
//   * ab_vec_kernel : the elementwise vector-field modifiers of vector_modification_functions.py:14-172 as a short op
//     list applied in one pass over the (3, N) field, so a from_sdf -> rotate_z -> rotate_axis pipeline
//     (sdf_vector_field.py:152-165) stays on the device and touches HBM once;
//   * ab_vec_component_kernel : x / y / z / phi / theta / length (geom.py:262-362).
// All are HBM-bound streaming kernels: one element per thread, coalesced along the fastest axis.
#pragma once
#include "ab_math.cuh"

namespace ab {

// scipy.ndimage 'reflect' (d c b a | a b c d | d c b a), valid for any offset
AB_DEV int reflect_index(int i, int n) {
  if ((unsigned)i < (unsigned)n) return i;  // the common case
  const int period = 2 * n;
  i %= period;
  if (i < 0) i += period;
  return i >= n ? period - 1 - i : i;
}

// The stencil kernels see the field as a C-ordered (n0, n1, n2) array (2D fields arrive as (1, nx, ny)) and take their
// coordinates from the launch grid: x = blockIdx.z, y = blockIdx.y, z = blockIdx.x * blockDim.x + threadIdx.x — no integer
// division, loads coalesced along z.
struct Field3 {
  uint32_t n0, n1, n2;
};

// one axis of the separable box filter: the sum of k taps starting at offset t0 along `axis`; the last pass of an iteration
// also divides by the kernel volume (the reference's filter is ones / norm). A thread owns one (x, z) and marches over
// `rows` consecutive y, so the address arithmetic is a pointer increment per output and the taps are k loads that hit
// L1 / L2 (x- and y-taps are whole rows apart, z-taps are neighbours in the same row).
template <typename T>
__global__ void __launch_bounds__(256) ab_box_axis_kernel(const T* __restrict__ in, T* __restrict__ out, Field3 f, int axis, int k,
                                                          int t0, T norm, int divide, uint32_t rows) {
  const uint32_t z = blockIdx.x * blockDim.x + threadIdx.x, x = blockIdx.z;
  if (z >= f.n2) return;
  const uint32_t y0 = blockIdx.y * rows, y1 = y0 + rows < f.n1 ? y0 + rows : f.n1;
  const uint64_t plane = (uint64_t)f.n1 * f.n2;
  const T* src = in + x * plane + (uint64_t)y0 * f.n2 + z;
  T* dst = out + x * plane + (uint64_t)y0 * f.n2 + z;
  if (axis == 2) {
    const bool inner = (int)z + t0 >= 0 && (int)z + t0 + k <= (int)f.n2;  // no reflection for this thread
    for (uint32_t y = y0; y < y1; y++, src += f.n2, dst += f.n2) {
      T s = T(0);
      if (inner) {
        for (int t = 0; t < k; t++) s = s + src[t0 + t];
      } else {
        const T* row = src - z;
        for (int t = 0; t < k; t++) s = s + row[reflect_index((int)z + t0 + t, (int)f.n2)];
      }
      *dst = divide ? s / norm : s;
    }
  } else if (axis == 1) {
    for (uint32_t y = y0; y < y1; y++, src += f.n2, dst += f.n2) {
      T s = T(0);
      if ((int)y + t0 >= 0 && (int)y + t0 + k <= (int)f.n1) {
        const T* p = src + (int64_t)t0 * f.n2;
        for (int t = 0; t < k; t++, p += f.n2) s = s + *p;
      } else {
        const T* col = in + x * plane + z;
        for (int t = 0; t < k; t++) s = s + col[(uint64_t)reflect_index((int)y + t0 + t, (int)f.n1) * f.n2];
      }
      *dst = divide ? s / norm : s;
    }
  } else {
    const bool inner = (int)x + t0 >= 0 && (int)x + t0 + k <= (int)f.n0;
    for (uint32_t y = y0; y < y1; y++, src += f.n2, dst += f.n2) {
      T s = T(0);
      if (inner) {
        const T* p = src + (int64_t)t0 * (int64_t)plane;
        for (int t = 0; t < k; t++, p += plane) s = s + *p;
      } else {
        const T* col = in + (uint64_t)y * f.n2 + z;
        for (int t = 0; t < k; t++) s = s + col[(uint64_t)reflect_index((int)x + t0 + t, (int)f.n0) * plane];
      }
      *dst = divide ? s / norm : s;
    }
  }
}

// The same pass for the two slow axes with the window in registers: a thread marches ALONG the filter axis over `chunk`
// outputs, keeps the last K samples and adds them in tap order (the same order as the generic kernel and the oracle, so
// the bits agree), i.e. one load per output instead of K.
template <typename T, int K>
__global__ void __launch_bounds__(256) ab_box_march_kernel(const T* __restrict__ in, T* __restrict__ out, Field3 f, int axis, int t0,
                                                           T norm, int divide, uint32_t chunk) {
  const uint32_t z = blockIdx.x * blockDim.x + threadIdx.x;
  if (z >= f.n2) return;
  const uint64_t plane = (uint64_t)f.n1 * f.n2;
  // axis 0: fixed y = blockIdx.y, march x over chunk blockIdx.z; axis 1: fixed x = blockIdx.z, march y over chunk blockIdx.y
  const uint32_t n_axis = axis == 0 ? f.n0 : f.n1;
  const uint64_t stride = axis == 0 ? plane : (uint64_t)f.n2;
  const uint32_t a0 = (axis == 0 ? blockIdx.z : blockIdx.y) * chunk;
  const uint32_t a1 = a0 + chunk < n_axis ? a0 + chunk : n_axis;
  const uint64_t base = axis == 0 ? (uint64_t)blockIdx.y * f.n2 + z : (uint64_t)blockIdx.z * plane + z;
  const T* col = in + base;
  T* dst = out + base + (uint64_t)a0 * stride;
  T w[K];
#pragma unroll
  for (int t = 0; t < K - 1; t++) w[t + 1] = col[(uint64_t)reflect_index((int)a0 + t0 + t, (int)n_axis) * stride];
  constexpr int U = 4;  // outputs per step: their loads are issued together (the march is latency-bound otherwise)
  for (uint32_t a = a0; a < a1; a += U) {
    T nw[U];
#pragma unroll
    for (int u = 0; u < U; u++)
      nw[u] = a + u < a1 ? col[(uint64_t)reflect_index((int)(a + u) + t0 + K - 1, (int)n_axis) * stride] : T(0);
#pragma unroll
    for (int u = 0; u < U; u++) {
      if (a + u >= a1) break;
#pragma unroll
      for (int t = 0; t < K - 1; t++) w[t] = w[t + 1];
      w[K - 1] = nw[u];
      T s = T(0);
#pragma unroll
      for (int t = 0; t < K; t++) s = s + w[t];
      *dst = divide ? s / norm : s;
      dst += stride;
    }
  }
}

template <typename T>
__global__ void ab_scale_copy_kernel(const T* __restrict__ in, T* __restrict__ out, uint64_t n, T norm) {
  for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (uint64_t)gridDim.x * blockDim.x) out[e] = in[e] / norm;
}

// 9 u - sum of the 3x3 neighbourhood over the two axes (0, 1) of a 3D field or (1, 2) of the (1, nx, ny) view of a 2D one.
// A thread marches along the first stencil axis over `chunk` outputs. The 3x3 sum is kept as three ROW sums (one per march
// position: left + centre + right along the cross axis) plus the three centre samples: a step loads the three samples of
// the look-ahead row, forms its row sum (2 adds), and writes 9 c - (r0 + r1 + r2): 5 arithmetic instructions per output
// instead of 10, no window shuffling. (The sum is associated row-wise, the reference's convolution tap by tap: the results
// differ in the last bits only, tests/test_gpu_fields.py bounds it at 1e-12.)
template <typename T, int U>
__global__ void __launch_bounds__(256) ab_edge_kernel(const T* __restrict__ in, T* __restrict__ out, Field3 f, int is2d, uint32_t chunk) {
  const uint32_t z = blockIdx.x * blockDim.x + threadIdx.x;
  if (z >= f.n2) return;
  const uint64_t plane = (uint64_t)f.n1 * f.n2;
  // march axis A / cross axis B: 3D (x, y) with y = blockIdx.y fixed; 2D view (y, z) with z fixed
  const uint32_t nA = is2d ? f.n1 : f.n0, nB = is2d ? f.n2 : f.n1;
  const uint64_t sA = is2d ? (uint64_t)f.n2 : plane, sB = is2d ? 1 : (uint64_t)f.n2;
  const uint32_t bpos = is2d ? z : blockIdx.y;
  const uint32_t a0 = (is2d ? blockIdx.y : blockIdx.z) * chunk;
  const uint32_t a1 = a0 + chunk < nA ? a0 + chunk : nA;
  // offsets of the two outer cross-axis taps relative to the column of this thread ('reflect' at the faces)
  const int64_t om = ((int64_t)reflect_index((int)bpos - 1, (int)nB) - (int64_t)bpos) * (int64_t)sB;
  const int64_t op = ((int64_t)reflect_index((int)bpos + 1, (int)nB) - (int64_t)bpos) * (int64_t)sB;
  const T* col = in + (is2d ? (uint64_t)z : (uint64_t)blockIdx.y * f.n2 + z);
  T* dst = out + (is2d ? (uint64_t)z : (uint64_t)blockIdx.y * f.n2 + z) + (uint64_t)a0 * sA;
  auto row = [&](const T* p, T& sum, T& centre) {
    centre = p[0];
    sum = (p[om] + centre) + p[op];
  };
  T r0, r1, r2, c0, c1, c2;  // rows a-1, a, a+1 of the output being written
  row(col + (uint64_t)reflect_index((int)a0 - 1, (int)nA) * sA, r1, c1);
  row(col + (uint64_t)a0 * sA, r2, c2);
  // U outputs per step, their 3 U loads issued together: the march is latency-bound (ncu: 82 % long-scoreboard stalls at U = 4)
  uint32_t a = a0;
  const T* pn = col + (uint64_t)(a0 + 1) * sA;
  // whole steps whose look-ahead rows a+1 .. a+U lie inside the field: plain pointer increments, no reflection, no tail tests
  for (; a + U <= a1 && a + U < nA; a += U) {
    T nm[U], nc[U], np_[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      nm[u] = pn[om];
      nc[u] = pn[0];
      np_[u] = pn[op];
      pn += sA;
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      r0 = r1; c0 = c1; r1 = r2; c1 = c2;
      c2 = nc[u];
      r2 = (nm[u] + c2) + np_[u];
      *dst = T(9) * c1 - ((r0 + r1) + r2);
      dst += sA;
    }
  }
  for (; a < a1; a++) {  // the last outputs of the chunk / of the axis: reflected look-ahead row
    r0 = r1; c0 = c1; r1 = r2; c1 = c2;
    row(col + (uint64_t)reflect_index((int)a + 1, (int)nA) * sA, r2, c2);
    *dst = T(9) * c1 - ((r0 + r1) + r2);
    dst += sA;
  }
  (void)c0;
}

// ---- signed: unsigned distance field -> signed distance field (modifications.py:220-275) -----------------------------------------
// boundary = field < threshold (the smallest grid step). Along axis 0 and along axis 1 the reference counts the entries
// into a boundary run on the way forward (chu) and the exits (chuu); a sample is "interior" along an axis when the inclusive
// prefix count of entries at i is odd OR the prefix count of exits at n-1-i is odd (the reference flips the cumulative sum,
// not the sequence); the two axes are AND-ed, smoothed by the (2,2,1) box filter, the outermost samples take their inner
// neighbour's value, and the field is negated where the result exceeds 1/2. If the field has a negative sample it is
// returned untouched.
//
// Along axis 0 a plane's interior depends on the whole column (the mirrored plane n0-1-i too), so the kernels work from a
// packed boundary mask of the whole field: bit (i2 & 31) of word [i0][i1][i2 / 32] (rows padded to whole words), 1 bit per
// sample. A slab of the field is signed from the whole mask plus its own planes of the field; the mask can be packed slab
// by slab (by different ranks) and concatenated.

// the mask of a C-ordered (n0, n1, n2) block of the field: one warp per mask word (__ballot_sync of 32 consecutive z);
// flags[0] |= a sample is negative, flags[1] |= a sample is NaN
template <typename T>
__global__ void __launch_bounds__(256) ab_signed_mask_kernel(const T* __restrict__ field, Field3 f, uint32_t words, T threshold,
                                                             uint32_t* __restrict__ mask, int* __restrict__ flags) {
  const uint32_t lane = threadIdx.x & 31u, w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (w >= words) return;  // whole warps
  const uint64_t row = (uint64_t)blockIdx.z * f.n1 + blockIdx.y;
  const uint32_t i2 = w * 32u + lane;
  bool b = false, neg = false, nan = false;
  if (i2 < f.n2) {
    const T v = field[row * f.n2 + i2];
    b = v < threshold;
    neg = v < T(0);
    nan = v != v;
  }
  const unsigned word = __ballot_sync(0xffffffffu, b);
  const bool any_neg = __any_sync(0xffffffffu, neg), any_nan = __any_sync(0xffffffffu, nan);
  if (lane == 0) {
    mask[row * words + w] = word;
    if (any_neg) atomicOr(flags, 1);
    if (any_nan) atomicOr(flags + 1, 1);
  }
}

// Bit-sliced crossing parities: a thread owns one mask word (32 columns) and marches it along the scanned axis, keeping
// the entry and exit parities as words:  in ^= b & ~prev (entries counted from i = 1),  out ^= b & ~next (up to n-2).
// It stores in(i) to pin[i] and out(i) to pout[n-1-i] for the positions i the caller asked for (plain stores, each slot
// written once), so in | out at a position is the interior test along that axis.
// blockIdx.y = 0: along axis 0, thread = (i1, word), stores planes [x0, x1) (slab-local);
// blockIdx.y = 1: along axis 1 inside the planes [x0, x1), thread = (i0 - x0, word), stores every i1.
__global__ void __launch_bounds__(256) ab_signed_scan_kernel(const uint32_t* __restrict__ mask, uint32_t n0, uint32_t n1,
                                                             uint32_t words, uint32_t x0, uint32_t x1, uint32_t* __restrict__ pin0,
                                                             uint32_t* __restrict__ pout0, uint32_t* __restrict__ pin1,
                                                             uint32_t* __restrict__ pout1) {
  const int axis = blockIdx.y;
  const uint64_t plane_w = (uint64_t)n1 * words;
  const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint64_t src, step, dst, dstep;
  uint32_t n, lo, hi;
  uint32_t *pin, *pout;
  if (axis == 0) {
    if (c >= plane_w) return;
    src = c; step = plane_w; n = n0; lo = x0; hi = x1; dst = c; dstep = plane_w; pin = pin0; pout = pout0;
  } else {
    if (c >= (uint64_t)(x1 - x0) * words) return;
    const uint64_t p = c / words, w = c - p * words;
    src = (x0 + p) * plane_w + w; step = words; n = n1; lo = 0; hi = n1; dst = p * plane_w + w; dstep = words;
    pin = pin1; pout = pout1;
  }
  uint32_t in = 0, out = 0, prev = ~0u;
  constexpr int U = 8;  // loads issued together: the march is latency-bound
  for (uint32_t i0 = 0; i0 < n; i0 += U) {
    uint32_t b[U + 1];
#pragma unroll
    for (int u = 0; u <= U; u++) b[u] = i0 + u < n ? mask[src + (uint64_t)(i0 + u) * step] : ~0u;  // ~0: no exit at n-1
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint32_t i = i0 + u;
      if (i >= n) break;
      in ^= b[u] & ~prev;
      out ^= b[u] & ~b[u + 1];
      prev = b[u];
      if (i >= lo && i < hi) pin[dst + (uint64_t)(i - lo) * dstep] = in;
      const uint32_t j = n - 1 - i;
      if (j >= lo && j < hi) pout[dst + (uint64_t)(j - lo) * dstep] = out;
    }
  }
}

// interior = (in0 | out0) & (in1 | out1) as a 0 / 1 field of T over the planes of the parity words
template <typename T>
__global__ void __launch_bounds__(256) ab_signed_interior_kernel(const uint32_t* __restrict__ pin0, const uint32_t* __restrict__ pout0,
                                                                 const uint32_t* __restrict__ pin1, const uint32_t* __restrict__ pout1,
                                                                 Field3 f, uint32_t words, T* __restrict__ interior) {
  const uint32_t i2 = blockIdx.x * blockDim.x + threadIdx.x, i1 = blockIdx.y, i0 = blockIdx.z;
  if (i2 >= f.n2) return;
  const uint64_t kw = ((uint64_t)i0 * f.n1 + i1) * words + (i2 >> 5);
  const uint32_t word = (pin0[kw] | pout0[kw]) & (pin1[kw] | pout1[kw]);
  interior[((uint64_t)i0 * f.n1 + i1) * f.n2 + i2] = (word >> (i2 & 31u)) & 1u ? T(1) : T(0);
}

// out = field * (1 - 2 (smooth[clamped index] > 1/2)) for the planes [x0, x0 + gridDim.z) of a field of f (global sizes);
// `field` and `out` start at plane x0, `smooth` at plane s0. Untouched when the field had a negative sample (and no NaN:
// np.amin of a field with a NaN is NaN, which is not < 0). TANGENT: the same sign applied to `tangent` -> `out_tangent`
// (laid out like field / out): the sign pattern is piecewise constant in the parameter, so it is the derivative
template <typename T, bool TANGENT>
__global__ void __launch_bounds__(256) ab_signed_apply_kernel(const T* __restrict__ field, const T* __restrict__ tangent,
                                                              const T* __restrict__ smooth, Field3 f, uint32_t x0, uint32_t s0,
                                                              const int* __restrict__ flags, T* __restrict__ out,
                                                              T* __restrict__ out_tangent) {
  const uint32_t i2 = blockIdx.x * blockDim.x + threadIdx.x, i1 = blockIdx.y, i0 = x0 + blockIdx.z;
  if (i2 >= f.n2) return;
  const uint64_t plane = (uint64_t)f.n1 * f.n2;
  const uint64_t k = (uint64_t)blockIdx.z * plane + (uint64_t)i1 * f.n2 + i2;
  const T v = field[k];
  if (flags[0] && !flags[1]) {
    out[k] = v;
    if constexpr (TANGENT) out_tangent[k] = tangent[k];
    return;
  }
  auto inner = [](uint32_t i, uint32_t n) { return i < 1 ? 1u : (i > n - 2 ? n - 2 : i); };  // [1:-1] then edge padding
  const T s = smooth[(uint64_t)(inner(i0, f.n0) - s0) * plane + (uint64_t)inner(i1, f.n1) * f.n2 + inner(i2, f.n2)];
  out[k] = s > T(0.5) ? -v : v;
  if constexpr (TANGENT) out_tangent[k] = s > T(0.5) ? -tangent[k] : tangent[k];
}

// ---- vector-field modifiers ----------------------------------------------------------------------------------------------
struct VecOpK {
  uint32_t opcode;
  uint32_t kind0, kind1;  // AB_VK_*
  double c[3];            // constant 3-vector operand
  double s0, s1;          // constant scalar operands
  const void* a0;         // per-point operand 0: (N,) or (3, stride0) of T
  const void* a1;         // per-point operand 1 (rotate_axis: the angle)
  uint64_t stride0, stride1;
};

template <typename T>
struct VecParams {
  T* vec;  // (3, stride), updated in place
  uint64_t stride, n;
  uint32_t n_ops;
  VecOpK ops[AB_MAX_VEC_OPS];
};

AB_DEV void sincos_(float a, float& s, float& c) { sincosf(a, &s, &c); }
AB_DEV void sincos_(double a, double& s, double& c) { sincos(a, &s, &c); }
AB_DEV float atan2_(float y, float x) { return atan2f(y, x); }
AB_DEV double atan2_(double y, double x) { return atan2(y, x); }

template <typename T>
AB_DEV T scalar_operand(uint32_t kind, double s, const void* a, uint64_t e) {
  return kind == AB_VK_ARRAY ? reinterpret_cast<const T*>(a)[e] : (T)s;
}

template <typename T>
AB_DEV void rot2(T& a, T& b, T sa, T ca) {  // (a, b) <- (a ca - b sa, a sa + b ca)
  const T na = a * ca - b * sa, nb = a * sa + b * ca;
  a = na;
  b = nb;
}

template <typename T>
__global__ void __launch_bounds__(256) ab_vec_kernel(const __grid_constant__ VecParams<T> vp) {
  for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < vp.n; e += (uint64_t)gridDim.x * blockDim.x) {
    T v0 = vp.vec[e], v1 = vp.vec[vp.stride + e], v2 = vp.vec[2 * vp.stride + e];
    for (uint32_t k = 0; k < vp.n_ops; k++) {
      const VecOpK& op = vp.ops[k];
      switch (op.opcode) {
        case AB_VOP_ADD: case AB_VOP_SUB: case AB_VOP_RESCALE: {
          T o0, o1, o2;
          if (op.kind0 == AB_VK_VEC3) {
            o0 = (T)op.c[0]; o1 = (T)op.c[1]; o2 = (T)op.c[2];
          } else if (op.kind0 == AB_VK_VEC_ARRAY) {
            const T* a = reinterpret_cast<const T*>(op.a0);
            o0 = a[e]; o1 = a[op.stride0 + e]; o2 = a[2 * op.stride0 + e];
          } else {
            o0 = o1 = o2 = scalar_operand<T>(op.kind0, op.s0, op.a0, e);
          }
          if (op.opcode == AB_VOP_ADD) { v0 = v0 + o0; v1 = v1 + o1; v2 = v2 + o2; }
          else if (op.opcode == AB_VOP_SUB) { v0 = v0 - o0; v1 = v1 - o1; v2 = v2 - o2; }
          else { v0 = v0 * o0; v1 = v1 * o1; v2 = v2 * o2; }
          break;
        }
        case AB_VOP_ROT_Z: case AB_VOP_ROT_X: case AB_VOP_ROT_Y: {
          T sa, ca;
          sincos_(scalar_operand<T>(op.kind0, op.s0, op.a0, e), sa, ca);
          if (op.opcode == AB_VOP_ROT_Z) rot2(v0, v1, sa, ca);
          else if (op.opcode == AB_VOP_ROT_X) rot2(v1, v2, sa, ca);
          else rot2(v0, v2, sa, ca);  // the reference's convention (vector_modification_functions.py:84-93)
          break;
        }
        case AB_VOP_ROT_THETA: {  // :55-69
          T sa, ca;
          sincos_(scalar_operand<T>(op.kind0, op.s0, op.a0, e), sa, ca);
          T r0 = v0, r1 = v1;
          const T m = s_sqrt(r0 * r0 + r1 * r1);
          if (m != T(0)) { r0 = r0 / m; r1 = r1 / m; }
          const T t0 = r0 * v2, t1 = r1 * v2, t2 = -r0 * v0 - r1 * v1;
          v0 = v0 * ca + t0 * sa;
          v1 = v1 * ca + t1 * sa;
          v2 = v2 * ca + t2 * sa;
          break;
        }
        case AB_VOP_ROT_AXIS: {  // Rodrigues with the axis as given (:116-131)
          T a0, a1, a2;
          if (op.kind0 == AB_VK_VEC3) {
            a0 = (T)op.c[0]; a1 = (T)op.c[1]; a2 = (T)op.c[2];
          } else {
            const T* a = reinterpret_cast<const T*>(op.a0);
            a0 = a[e]; a1 = a[op.stride0 + e]; a2 = a[2 * op.stride0 + e];
          }
          T sa, ca;
          sincos_(scalar_operand<T>(op.kind1, op.s1, op.a1, e), sa, ca);
          const T c0 = a1 * v2 - a2 * v1, c1 = a2 * v0 - a0 * v2, c2 = a0 * v1 - a1 * v0;
          const T dot = a0 * v0 + a1 * v1 + a2 * v2, w = (T(1) - ca) * dot;
          v0 = v0 * ca + sa * c0 + w * a0;
          v1 = v1 * ca + sa * c1 + w * a1;
          v2 = v2 * ca + sa * c2 + w * a2;
          break;
        }
        case AB_VOP_REVOLVE_X: case AB_VOP_REVOLVE_Y: case AB_VOP_REVOLVE_Z: {  // :134-172
          const T* r = reinterpret_cast<const T*>(op.a0);
          const T r0 = r[e], r1 = r[op.stride0 + e], r2 = r[2 * op.stride0 + e];
          T sa, ca;
          if (op.opcode == AB_VOP_REVOLVE_X) {
            sincos_(atan2_(r2, r1), sa, ca);
            rot2(v1, v2, sa, ca);
          } else if (op.opcode == AB_VOP_REVOLVE_Y) {
            sincos_(atan2_(r2, r0), sa, ca);
            rot2(v0, v2, sa, ca);
          } else {
            sincos_(atan2_(r1, r0), sa, ca);
            rot2(v0, v1, sa, ca);
          }
          break;
        }
        case AB_VOP_NORMALIZE: {  // batch_normalize (:14-20): zero vectors stay zero
          const T m = s_sqrt(v0 * v0 + v1 * v1 + v2 * v2);
          if (m != T(0)) { v0 = v0 / m; v1 = v1 / m; v2 = v2 / m; }
          break;
        }
        default: break;
      }
    }
    vp.vec[e] = v0;
    vp.vec[vp.stride + e] = v1;
    vp.vec[2 * vp.stride + e] = v2;
  }
}

template <typename T>
__global__ void ab_vec_component_kernel(const T* __restrict__ vec, uint64_t stride, uint64_t n, int what, T* __restrict__ out) {
  constexpr int U = 4;  // elements per thread and step, loads issued together
  const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t e0 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e0 < n; e0 += step * U) {
    T v0[U], v1[U], v2[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint64_t e = e0 + u * step;
      const bool live = e < n;
      v0[u] = live && what != AB_VC_Y && what != AB_VC_Z ? vec[e] : T(0);
      v1[u] = live && what != AB_VC_X && what != AB_VC_Z ? vec[stride + e] : T(0);
      v2[u] = live && what != AB_VC_X && what != AB_VC_Y && what != AB_VC_PHI ? vec[2 * stride + e] : T(0);
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint64_t e = e0 + u * step;
      if (e >= n) break;
      T r;
      switch (what) {
        case AB_VC_X: r = v0[u]; break;
        case AB_VC_Y: r = v1[u]; break;
        case AB_VC_Z: r = v2[u]; break;
        case AB_VC_PHI: r = atan2_(v1[u], v0[u]); break;
        case AB_VC_THETA: r = sizeof(T) == 4 ? (T)acosf((float)v2[u]) : (T)acos((double)v2[u]); break;
        default: r = s_sqrt(v0[u] * v0[u] + v1[u] * v1[u] + v2[u] * v2[u]); break;
      }
      out[e] = r;
    }
  }
}

}  // namespace ab
