// Device-side helpers shared by the kernels.  All parity-critical float arithmetic uses the
// explicit round-to-nearest intrinsics (__fmul_rn / __fadd_rn ...) so it can never be contracted
// into FMA, whatever the compile flags (SURVEY.md §7.3: the reference's PCL/FLANN binaries do
// not use FMA and its float32 covariance is rounding- and order-sensitive at the 1e-3 level).
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "ppp_internal.cuh"

typedef unsigned long long u64;

#define PPP_KEY_INF 0xFFFFFFFFFFFFFFFFull

__device__ __forceinline__ bool finite3(float x, float y, float z) {
  return isfinite(x) && isfinite(y) && isfinite(z);
}

// [upstream] flann::L2_Simple<float>: ((dx*dx) + dy*dy) + dz*dz, sequential float32, no FMA.
__device__ __forceinline__ float d2_flann(float ax, float ay, float az, float bx, float by, float bz) {
  float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
  float r = __fmul_rn(dx, dx);
  r = __fadd_rn(r, __fmul_rn(dy, dy));
  r = __fadd_rn(r, __fmul_rn(dz, dz));
  return r;
}

// The same value with the x and y lanes in ONE packed instruction each (sm_100 FADD2 / FMUL2: IEEE round-to-nearest
// per lane, subnormals kept, so the bits are those of d2_flann): 6 instructions per candidate instead of 8 in
// loops that are bound by instruction issue.  qxy = pack2(qx, qy); c.x / c.y arrive as an aligned register pair
// from the 128-bit load.
__device__ __forceinline__ u64 pack2(float lo, float hi) {
  u64 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ float d2_flann_x2(u64 qxy, float qz, const float4& c) {
  u64 cxy, d, m;
  float mx, my;
  asm("mov.b64 %0, {%1, %2};" : "=l"(cxy) : "f"(c.x), "f"(c.y));
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(qxy), "l"(cxy));
  asm("mul.rn.f32x2 %0, %1, %1;" : "=l"(m) : "l"(d));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(mx), "=f"(my) : "l"(m));
  const float dz = __fsub_rn(qz, c.z);
  return __fadd_rn(__fadd_rn(mx, my), __fmul_rn(dz, dz));
}

// (d2, idx) total order as one unsigned 64-bit compare: d2 >= +0 so its bit pattern is monotone.
__device__ __forceinline__ u64 make_key(float d2, int idx) {
  return ((u64)__float_as_uint(d2) << 32) | (u64)(uint32_t)idx;
}
__device__ __forceinline__ float key_d2(u64 k) { return __uint_as_float((uint32_t)(k >> 32)); }
__device__ __forceinline__ int key_idx(u64 k) { return (int)(uint32_t)(k & 0xFFFFFFFFull); }

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// Cell coordinate along one axis, clamped to [-PPP_CELL_LIM, PPP_CELL_LIM]. Monotone non-decreasing in `a`
// (float sub, mul by a positive constant, floor and the clamp are monotone), which is what the ring-termination
// bound relies on.  Why the clamp keeps every search exact: grid cells lie in [0, nu - 1] and nu, nv <= 2^27
// (nu * nv <= 2^28, both >= 2), so clamping moves a far query's cell TOWARDS every grid cell and the cell distance
// to any point only shrinks.  ring_bound2 is a lower bound on the distance derived from that cell distance, so it
// stays a lower bound; the rounding of the unclamped coordinate (<= 3 * 2^-24 of it) is covered by its slack term,
// which grows with |cu| + |cv| >= 2^29 for a clamped query.  The clamp keeps every sum a search forms in int32:
// |cu|, |cv| <= 2^29, rings R <= PPP_RING_MAX = 2^30 (a ring loop stops once its block covers the grid, R <=
// 2^29 + 2^27), so cu +- R, cv +- R and their differences stay below 2^31 in magnitude.
constexpr int PPP_CELL_LIM = 1 << 29;
constexpr int PPP_RING_MAX = 1 << 30;   // a block of this half-width around any clamped cell covers the whole grid
__device__ __forceinline__ int cell_coord_raw(float a, float amin, float inv_h) {
  return clampi(__float2int_rd(__fmul_rn(__fsub_rn(a, amin), inv_h)), -PPP_CELL_LIM, PPP_CELL_LIM);
}

__device__ __forceinline__ float axis_of(float x, float y, float z, int a) { return a == 0 ? x : (a == 1 ? y : z); }

// The (clamped, possibly outside the grid) cell of a query.
__device__ __forceinline__ void query_cell(const GridView& g, float qx, float qy, float qz, int& cu, int& cv) {
  cu = cell_coord_raw(axis_of(qx, qy, qz, g.au), g.min_u, g.inv_h);
  cv = cell_coord_raw(axis_of(qx, qy, qz, g.av), g.min_v, g.inv_h);
}

// Squared lower bound on the distance from a query in cell (cu,cv) to any point whose cell lies
// outside the (2R+1)x(2R+1) block around it: (R*h - slack)^2, rounded down, shrunk by 1e-6 so a
// float32 d2 (relative error <= 3*2^-24) of an unseen point can never tie or beat an accepted one.
__device__ __forceinline__ float ring_bound2(const GridView& g, int R, int cu, int cv) {
  // slack grows with the magnitude of the cell coordinates involved (queries may lie far outside the grid)
  // (the magnitude sum is formed in float: |cu| + |cv| + R can pass 2^31 for a clamped far query)
  const float mag = __fadd_ru(__fadd_ru(__int2float_ru(abs(cu)), __int2float_ru(abs(cv))), __fadd_ru(__int2float_ru(R), 2.0f));
  float extra = __fmul_ru(g.h, __fmul_ru(mag, 4.76837158203125e-07f));
  float rb = __fsub_rd(__fsub_rd(__fmul_rd((float)R, g.h), g.slack), extra);
  if (rb <= 0.0f) return 0.0f;
  return __fmul_rd(__fmul_rd(rb, rb), 0.999999f);
}

// ---------------------------------------------------------------------------------------------
// PCL 1.10 normal estimation restated for the device (SURVEY.md Appendix A.5-A.7) [upstream].
// Transcendentals are evaluated in double and rounded to float: that is the correctly rounded
// float result except in ~2^-29 of cases, which is what glibc's float routines return to <1 ulp.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void compute_roots2(float b, float c, float roots[3]) {
  roots[0] = 0.0f;
  float bb = __fmul_rn(b, b);
  float d = (float)((double)bb - 4.0 * (double)c);  // Scalar d = Scalar (b * b - 4.0 * c)
  if (d < 0.0f) d = 0.0f;
  float sd = __fsqrt_rn(d);
  roots[2] = __fmul_rn(0.5f, __fadd_rn(b, sd));
  roots[1] = __fmul_rn(0.5f, __fsub_rn(b, sd));
}

__device__ __forceinline__ void swapf(float& a, float& b) { float t = a; a = b; b = t; }

__device__ __forceinline__ void compute_roots(float m00, float m01, float m02, float m11, float m12, float m22,
                                              float roots[3]) {
  // c0 = m00*m11*m22 + 2*m01*m02*m12 - m00*m12*m12 - m11*m02*m02 - m22*m01*m01 (left to right)
  float c0 = __fmul_rn(__fmul_rn(m00, m11), m22);
  c0 = __fadd_rn(c0, __fmul_rn(__fmul_rn(__fmul_rn(2.0f, m01), m02), m12));
  c0 = __fsub_rn(c0, __fmul_rn(__fmul_rn(m00, m12), m12));
  c0 = __fsub_rn(c0, __fmul_rn(__fmul_rn(m11, m02), m02));
  c0 = __fsub_rn(c0, __fmul_rn(__fmul_rn(m22, m01), m01));
  float c1 = __fsub_rn(__fmul_rn(m00, m11), __fmul_rn(m01, m01));
  c1 = __fadd_rn(c1, __fmul_rn(m00, m22));
  c1 = __fsub_rn(c1, __fmul_rn(m02, m02));
  c1 = __fadd_rn(c1, __fmul_rn(m11, m22));
  c1 = __fsub_rn(c1, __fmul_rn(m12, m12));
  float c2 = __fadd_rn(__fadd_rn(m00, m11), m22);
  if (fabsf(c0) < 1.1920928955078125e-07f) {
    compute_roots2(c2, c1, roots);
  } else {
    const float s_inv3 = (float)(1.0 / 3.0);
    const float s_sqrt3 = 1.7320508075688772f;  // sqrtf(3.0f)
    float c2_over_3 = __fmul_rn(c2, s_inv3);
    float a_over_3 = __fmul_rn(__fsub_rn(c1, __fmul_rn(c2, c2_over_3)), s_inv3);
    if (a_over_3 > 0.0f) a_over_3 = 0.0f;
    float t = __fsub_rn(__fmul_rn(__fmul_rn(2.0f, c2_over_3), c2_over_3), c1);
    float half_b = __fmul_rn(0.5f, __fadd_rn(c0, __fmul_rn(c2_over_3, t)));
    float q = __fadd_rn(__fmul_rn(half_b, half_b), __fmul_rn(__fmul_rn(a_over_3, a_over_3), a_over_3));
    if (q > 0.0f) q = 0.0f;
    float rho = __fsqrt_rn(-a_over_3);
    float theta = __fmul_rn((float)atan2((double)__fsqrt_rn(-q), (double)half_b), s_inv3);
    double sd, cd;
    sincos((double)theta, &sd, &cd);
    float cos_theta = (float)cd;
    float sin_theta = (float)sd;
    roots[0] = __fadd_rn(c2_over_3, __fmul_rn(__fmul_rn(2.0f, rho), cos_theta));
    roots[1] = __fsub_rn(c2_over_3, __fmul_rn(rho, __fadd_rn(cos_theta, __fmul_rn(s_sqrt3, sin_theta))));
    roots[2] = __fsub_rn(c2_over_3, __fmul_rn(rho, __fsub_rn(cos_theta, __fmul_rn(s_sqrt3, sin_theta))));
    if (roots[0] >= roots[1]) swapf(roots[0], roots[1]);
    if (roots[1] >= roots[2]) {
      swapf(roots[1], roots[2]);
      if (roots[0] >= roots[1]) swapf(roots[0], roots[1]);
    }
    if (roots[0] <= 0.0f) compute_roots2(c2, c1, roots);
  }
}

__device__ __forceinline__ void cross3(float a0, float a1, float a2, float b0, float b1, float b2, float o[3]) {
  o[0] = __fsub_rn(__fmul_rn(a1, b2), __fmul_rn(a2, b1));
  o[1] = __fsub_rn(__fmul_rn(a2, b0), __fmul_rn(a0, b2));
  o[2] = __fsub_rn(__fmul_rn(a0, b1), __fmul_rn(a1, b0));
}
__device__ __forceinline__ float sqnorm3(const float v[3]) {
  // Eigen 3-vector redux: x*x + (y*y + z*z)
  return __fadd_rn(__fmul_rn(v[0], v[0]), __fadd_rn(__fmul_rn(v[1], v[1]), __fmul_rn(v[2], v[2])));
}

// acc: the nine PCL accumulators (xx xy xz yy yz zz x y z) summed over m neighbours in list order.
// Writes nx, ny, nz, curvature (already flipped towards the viewpoint).
__device__ __forceinline__ void normal_from_accumulators(float acc[9], int m, float qx, float qy, float qz,
                                                         float vpx, float vpy, float vpz, float out[4]) {
  float cnt = (float)m;
  if ((m & (m - 1)) == 0) {
    // m = 16, 8, 32 ...: dividing by a power of two is the multiplication by its (exact) reciprocal, bit for bit
    const float inv = __fdiv_rn(1.0f, cnt);
#pragma unroll
    for (int i = 0; i < 9; i++) acc[i] = __fmul_rn(acc[i], inv);
  } else {
#pragma unroll
    for (int i = 0; i < 9; i++) acc[i] = __fdiv_rn(acc[i], cnt);
  }
  float cov[6];
  cov[0] = __fsub_rn(acc[0], __fmul_rn(acc[6], acc[6]));
  cov[1] = __fsub_rn(acc[1], __fmul_rn(acc[6], acc[7]));
  cov[2] = __fsub_rn(acc[2], __fmul_rn(acc[6], acc[8]));
  cov[3] = __fsub_rn(acc[3], __fmul_rn(acc[7], acc[7]));
  cov[4] = __fsub_rn(acc[4], __fmul_rn(acc[7], acc[8]));
  cov[5] = __fsub_rn(acc[5], __fmul_rn(acc[8], acc[8]));
  float scale = 0.0f;
#pragma unroll
  for (int i = 0; i < 6; i++) scale = fmaxf(scale, fabsf(cov[i]));
  // fmaxf drops NaN operands; std::max(scale, |c|) in Eigen's maxCoeff keeps the running value on
  // a NaN compare as well, and a NaN covariance yields a NaN normal either way.
  if (scale <= 1.17549435e-38f) scale = 1.0f;
  float s[6];
#pragma unroll
  for (int i = 0; i < 6; i++) s[i] = __fdiv_rn(cov[i], scale);
  float roots[3];
  compute_roots(s[0], s[1], s[2], s[3], s[4], s[5], roots);
  float eigenvalue = __fmul_rn(roots[0], scale);
  float d0 = __fsub_rn(s[0], roots[0]), d1 = __fsub_rn(s[3], roots[0]), d2 = __fsub_rn(s[5], roots[0]);
  float v1[3], v2[3], v3[3];
  cross3(d0, s[1], s[2], s[1], d1, s[4], v1);
  cross3(d0, s[1], s[2], s[2], s[4], d2, v2);
  cross3(s[1], d1, s[4], s[2], s[4], d2, v3);
  float l1 = sqnorm3(v1), l2 = sqnorm3(v2), l3 = sqnorm3(v3);
  float vx, vy, vz, l;
  if (l1 >= l2 && l1 >= l3) { vx = v1[0]; vy = v1[1]; vz = v1[2]; l = l1; }
  else if (l2 >= l1 && l2 >= l3) { vx = v2[0]; vy = v2[1]; vz = v2[2]; l = l2; }
  else { vx = v3[0]; vy = v3[1]; vz = v3[2]; l = l3; }
  float sl = __fsqrt_rn(l);
  float nx = __fdiv_rn(vx, sl), ny = __fdiv_rn(vy, sl), nz = __fdiv_rn(vz, sl);
  float eig_sum = __fadd_rn(__fadd_rn(cov[0], cov[3]), cov[5]);
  float curv = (eig_sum != 0.0f) ? fabsf(__fdiv_rn(eigenvalue, eig_sum)) : 0.0f;
  // flipNormalTowardsViewpoint
  float wx = __fsub_rn(vpx, qx), wy = __fsub_rn(vpy, qy), wz = __fsub_rn(vpz, qz);
  float c = __fadd_rn(__fadd_rn(__fmul_rn(wx, nx), __fmul_rn(wy, ny)), __fmul_rn(wz, nz));
  if (c < 0.0f) { nx = __fmul_rn(nx, -1.0f); ny = __fmul_rn(ny, -1.0f); nz = __fmul_rn(nz, -1.0f); }
  out[0] = nx; out[1] = ny; out[2] = nz; out[3] = curv;
}

__device__ __forceinline__ void accumulate_point(float acc[9], float x, float y, float z) {
  acc[0] = __fadd_rn(acc[0], __fmul_rn(x, x));
  acc[1] = __fadd_rn(acc[1], __fmul_rn(x, y));
  acc[2] = __fadd_rn(acc[2], __fmul_rn(x, z));
  acc[3] = __fadd_rn(acc[3], __fmul_rn(y, y));
  acc[4] = __fadd_rn(acc[4], __fmul_rn(y, z));
  acc[5] = __fadd_rn(acc[5], __fmul_rn(z, z));
  acc[6] = __fadd_rn(acc[6], x);
  acc[7] = __fadd_rn(acc[7], y);
  acc[8] = __fadd_rn(acc[8], z);
}

// 32 bytes with one instruction (p must be 32-byte aligned).
__device__ __forceinline__ void st_global_256(void* p, float a, float b, float c, float d, float e, float f, float g, float h) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d), "f"(e), "f"(f), "f"(g),
               "f"(h)
               : "memory");
}

// Store one normal record. stride_f == 4: {nx,ny,nz,curv}; stride_f >= 8: pcl::Normal layout
// {nx,ny,nz,0, curv,0,0,0}; other strides: nx,ny,nz at 0..2, curvature at 3.  map (optional): record
// number of each row, negative = the row is not stored (halo rows of a slab whose records go to
// another GPU's buffer over NVLink).
__device__ __forceinline__ void store_normal(float* base, const int32_t* __restrict__ map, int64_t row, int stride_f,
                                             const float o[4], const NormalRoute* __restrict__ route = nullptr) {
  if (map) {
    row = __ldg(map + row);
    if (row < 0) return;
  }
  if (route) {   // multi-GPU: the record goes to the rank that holds this original index (NVLink store)
    int r = 0;
    while (r + 1 < route->world && row >= route->start[r + 1]) r++;
    base = route->base[r];
    row -= route->start[r];
  }
  float* p = base + row * (int64_t)stride_f;
  if (stride_f == 8) {
    if (((uintptr_t)base & 31) == 0) {   // one 256-bit store per pcl::Normal record (sm_100: STG.256)
      st_global_256(p, o[0], o[1], o[2], 0.0f, o[3], 0.0f, 0.0f, 0.0f);
    } else {
      reinterpret_cast<float4*>(p)[0] = make_float4(o[0], o[1], o[2], 0.0f);
      reinterpret_cast<float4*>(p)[1] = make_float4(o[3], 0.0f, 0.0f, 0.0f);
    }
  } else if (stride_f == 4) {
    reinterpret_cast<float4*>(p)[0] = make_float4(o[0], o[1], o[2], o[3]);
  } else if (stride_f > 8) {
    p[0] = o[0]; p[1] = o[1]; p[2] = o[2]; p[3] = 0.0f; p[4] = o[3];
  } else {
    p[0] = o[0]; p[1] = o[1]; p[2] = o[2]; p[3] = o[3];
  }
}

// The PCL normal of one query from its neighbour records, added in list order: pcl::NormalEstimation's contract.
// Under PPP_COV_SHIFTED the first record is the origin every record is taken relative to.
struct CovAcc {
  float acc[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float kx = 0.f, ky = 0.f, kz = 0.f;
  int m = 0;
  bool shifted;
  __device__ __forceinline__ explicit CovAcc(unsigned flags) : shifted((flags & PPP_COV_SHIFTED) != 0) {}
  __device__ __forceinline__ void add(float4 rec) {
    float x = rec.x, y = rec.y, z = rec.z;
    if (m == 0) { kx = x; ky = y; kz = z; }
    if (shifted) { x = __fsub_rn(x, kx); y = __fsub_rn(y, ky); z = __fsub_rn(z, kz); }
    accumulate_point(acc, x, y, z);
    m++;
  }
  // NaN for a non-finite query or fewer than 3 neighbours; the record of `row` is stored if `store` (the lanes of a
  // warp that all computed it leave the store to one of them).  P: the search parameters.
  template <class Params>
  __device__ __forceinline__ void finish(const Params& P, bool fin, int64_t row, float qx, float qy, float qz,
                                         bool store = true) {
    float o[4];
    if (!fin || m < 3) o[0] = o[1] = o[2] = o[3] = CUDART_NAN_F;
    else normal_from_accumulators(acc, m, qx, qy, qz, P.vpx, P.vpy, P.vpz, o);
    if (store) store_normal(P.normals, P.nmap, row, P.nsf, o, P.route);
  }
};

// MLS result record (ppp_dev_mls_smooth) of a point without an output row: flag 0, every other field NaN.
__device__ __forceinline__ void mls_no_row(float o[8]) {
#pragma unroll
  for (int k = 0; k < 8; k++) o[k] = CUDART_NAN_F;
  o[3] = 0.0f;
}

// Store one 32-byte MLS result record {x, y, z, flag, nx, ny, nz, curvature}: at base + 8 * row, or, with a map,
// at the record of global index map[row] (negative: not stored) in its home rank's buffer when a route is given.
__device__ __forceinline__ void store_mls_record(float* base, const int32_t* __restrict__ map, int64_t row, const float o[8],
                                                 const NormalRoute* __restrict__ route) {
  if (map) {
    row = __ldg(map + row);
    if (row < 0) return;
  }
  if (route) {
    int r = 0;
    while (r + 1 < route->world && row >= route->start[r + 1]) r++;
    base = route->base[r];
    row -= route->start[r];
  }
  float4* p = reinterpret_cast<float4*>(base + row * 8);
  p[0] = make_float4(o[0], o[1], o[2], o[3]);
  p[1] = make_float4(o[4], o[5], o[6], o[7]);
}

// Visit every indexed point whose cell lies in the square annulus R_prev < max(|du|,|dv|) <= R
// around (cu, cv)  (R_prev = -1: the whole (2R+1)^2 block).  [ulo, uhi] optionally restricts the
// visited cell columns (callers that only want points of an x-interval).
template <typename F>
__device__ __forceinline__ void visit_annulus_pos(const GridView& g, int cu, int cv, int R_prev, int R, F&& f,
                                                  int ulo = -2147483647, int uhi = 2147483647) {
  int v0 = max(cv - R, 0), v1 = min(cv + R, g.nv - 1);
  ulo = max(ulo, 0);
  uhi = min(uhi, g.nu - 1);
  for (int v = v0; v <= v1; v++) {
    int adv = abs(v - cv);
    const int32_t* row = g.cell_start + (int64_t)v * g.nu;
    if (adv > R_prev) {
      int a = max(cu - R, ulo), b = min(cu + R, uhi);
      if (a <= b) {
        int s = __ldg(row + a), e = __ldg(row + b + 1);
        for (int i = s; i < e; i++) f(__ldg(g.sorted + i), i);
      }
    } else {
      int a = max(cu - R, ulo), b = min(cu - R_prev - 1, uhi);
      if (a <= b) {
        int s = __ldg(row + a), e = __ldg(row + b + 1);
        for (int i = s; i < e; i++) f(__ldg(g.sorted + i), i);
      }
      a = max(cu + R_prev + 1, ulo); b = min(cu + R, uhi);
      if (a <= b) {
        int s = __ldg(row + a), e = __ldg(row + b + 1);
        for (int i = s; i < e; i++) f(__ldg(g.sorted + i), i);
      }
    }
  }
}

// The same, for callers that do not need the sorted position of the visited record.
template <typename F>
__device__ __forceinline__ void visit_annulus(const GridView& g, int cu, int cv, int R_prev, int R, F&& f,
                                              int ulo = -2147483647, int uhi = 2147483647) {
  visit_annulus_pos(g, cu, cv, R_prev, R, [&](float4 c, int) { f(c); }, ulo, uhi);
}

__device__ __forceinline__ bool block_covers_grid(const GridView& g, int cu, int cv, int R) {
  return cu - R <= 0 && cu + R >= g.nu - 1 && cv - R <= 0 && cv + R >= g.nv - 1;
}

