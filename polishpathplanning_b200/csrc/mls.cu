// Moving-least-squares smoothing: pcl::MovingLeastSquares as the reference's smooth() runs it
// (src/Path_Generation.cpp:340-360: polynomial order 3, search radius 15, no upsampling, SIMPLE
// projection, weight exp(-d2 / r^2)).  [upstream, recalled: PCL 1.10.0 MLSResult::computeMLSSurface,
// projectQueryPoint, projectPointSimpleToPolynomialSurface, getPolynomialPartialDerivative.]
//
// Every quantity is a sum over the radius ball, so no neighbour list is built: one thread per query
// (queries in sorted cell order, warp-uniform row loops as in k_radius_normals32) streams the candidate
// block of the column grid twice.
//   visit 1: count and the sums of d = p - q and d d^T in double (shifted by the query), which give the
//            centroid and the unnormalised covariance in one pass;
//   eigen33 (double), Darboux frame;
//   visit 2: the weighted moments sum w u^a v^b (a + b <= 2 order: every entry of P W P^T) and the
//            right-hand side sum w f u^a v^b (a + b <= order);
//   Cholesky (Eigen's unblocked LLT, including its behaviour on a non-positive pivot) in registers and
//   the SIMPLE projection.
// The contract is a tolerance against the FMA-free CPU oracle (DESIGN.md §2), so the accumulations use
// explicit FMAs although the library is built with --fmad=false.
//
// Device records and several GPUs (ppp_dev_mls_smooth): each query stores one 32-byte record
// {x, y, z, flag, nx, ny, nz, curvature} instead of the compacted rows, by original index on a plain cloud and, on
// a slab attached by ppp_exch_attach, through the cloud's route into the home rank's buffer (as store_normal does
// for the normal estimators).  Only owned rows (nmap >= 0) are queries there; halo copies are candidates only.
// ppp_dev_mls_compact turns a range of records into rows in source order at a caller-given row base.
#include <cmath>

#include "ppp_device.cuh"

namespace {

struct MlsParams {
  GridView g;
  int64_t nq;           // sorted positions [0, nq) are the queries
  int R;                // candidate block half-width in cells
  float r2;             // membership: d2 < (float)(r*r)
  double inv_sq_radius; // weight exp(-d2 * inv_sq_radius), 1 / (r*r) in double
  const unsigned char* choice;   // multi-projection index: only queries whose point chose my_proj (nullptr: all)
  int my_proj;
  float4* xyz_out;      // by original index: smoothed x, y, z
  float4* nrm_out;      // by original index: nx, ny, nz, curvature (nullptr: not wanted)
  int32_t* emit;        // by original index: 1 = the point has an output row (zero-filled by the caller)
};

// Record mode (k_mls<ORDER, true>; MlsParams' xyz_out / nrm_out / emit unused): every query stores its 32-byte record.
// A parameter of its own, so that the single-GPU instance is compiled from MlsParams alone.
struct MlsRecords {
  float* rec;                    // records by original index, or unused with a route
  const int32_t* nmap;           // slab row -> global index, negative for halo copies (nullptr: every row is a query)
  const NormalRoute* route;      // with nmap: the record goes to the home rank of the global index
};

// Candidates of the (2R+1)^2 cell block around (cu, cv) that lie strictly within the radius, row by row;
// every lane of the warp runs the same number of iterations per row (the longest row of the warp).
template <typename F>
__device__ __forceinline__ void mls_visit(const MlsParams& P, bool act, int cu, int cv, float qx, float qy, float qz,
                                          F&& f) {
  const GridView& g = P.g;
  const u64 qxy = pack2(qx, qy);
#pragma unroll 1
  for (int dv = -P.R; dv <= P.R; dv++) {
    int s = 0, e = 0;
    const int v = cv + dv;
    if (act && v >= 0 && v < g.nv) {
      const int a = max(cu - P.R, 0), b = min(cu + P.R, g.nu - 1);
      if (a <= b) {
        const int64_t rowp = (int64_t)v * g.nu;
        PPP_DEV_ASSERT(rowp + b + 1 <= (int64_t)g.nu * g.nv);
        s = __ldg(g.cell_start + rowp + a);
        e = __ldg(g.cell_start + rowp + b + 1);
      }
    }
    const int n_it = __reduce_max_sync(0xffffffffu, e - s);
#pragma unroll 1
    for (int it = 0; it < n_it; it++) {
      const int i = s + it;
      if (i < e) {
        PPP_DEV_ASSERT(i >= 0 && i < g.n_sorted);
        const float4 c = __ldg(g.sorted + i);
        if (d2_flann_x2(qxy, qz, c) < P.r2) f(c);
      }
    }
  }
}

// ---- pcl::eigen33 in double: smallest eigenvalue and its eigenvector ---------------------------------
__device__ __forceinline__ void compute_roots2_d(double b, double c, double roots[3]) {
  roots[0] = 0.0;
  double d = b * b - 4.0 * c;
  if (d < 0.0) d = 0.0;
  const double sd = sqrt(d);
  roots[2] = 0.5 * (b + sd);
  roots[1] = 0.5 * (b - sd);
}

__device__ __forceinline__ void compute_roots_d(const double m[6], double roots[3]) {
  const double m00 = m[0], m01 = m[1], m02 = m[2], m11 = m[3], m12 = m[4], m22 = m[5];
  const double c0 = m00 * m11 * m22 + 2.0 * m01 * m02 * m12 - m00 * m12 * m12 - m11 * m02 * m02 - m22 * m01 * m01;
  const double c1 = m00 * m11 - m01 * m01 + m00 * m22 - m02 * m02 + m11 * m22 - m12 * m12;
  const double c2 = m00 + m11 + m22;
  if (fabs(c0) < 2.220446049250313e-16) {
    compute_roots2_d(c2, c1, roots);
    return;
  }
  const double s_inv3 = 1.0 / 3.0;
  const double s_sqrt3 = 1.7320508075688772;
  const double c2_over_3 = c2 * s_inv3;
  double a_over_3 = (c1 - c2 * c2_over_3) * s_inv3;
  if (a_over_3 > 0.0) a_over_3 = 0.0;
  const double half_b = 0.5 * (c0 + c2_over_3 * (2.0 * c2_over_3 * c2_over_3 - c1));
  double q = half_b * half_b + a_over_3 * a_over_3 * a_over_3;
  if (q > 0.0) q = 0.0;
  const double rho = sqrt(-a_over_3);
  const double theta = atan2(sqrt(-q), half_b) * s_inv3;
  double sin_theta, cos_theta;
  sincos(theta, &sin_theta, &cos_theta);
  roots[0] = c2_over_3 + 2.0 * rho * cos_theta;
  roots[1] = c2_over_3 - rho * (cos_theta + s_sqrt3 * sin_theta);
  roots[2] = c2_over_3 - rho * (cos_theta - s_sqrt3 * sin_theta);
  double t;
  if (roots[0] >= roots[1]) { t = roots[0]; roots[0] = roots[1]; roots[1] = t; }
  if (roots[1] >= roots[2]) {
    t = roots[1]; roots[1] = roots[2]; roots[2] = t;
    if (roots[0] >= roots[1]) { t = roots[0]; roots[0] = roots[1]; roots[1] = t; }
  }
  if (roots[0] <= 0.0) compute_roots2_d(c2, c1, roots);
}

// cov: 00 01 02 11 12 22.  n: unit eigenvector of the smallest eigenvalue; returns that eigenvalue.
__device__ __forceinline__ double eigen33_d(const double cov[6], double n[3]) {
  double scale = 0.0;
#pragma unroll
  for (int i = 0; i < 6; i++) scale = fmax(scale, fabs(cov[i]));
  if (scale <= 2.2250738585072014e-308) scale = 1.0;
  double s[6];
#pragma unroll
  for (int i = 0; i < 6; i++) s[i] = cov[i] / scale;
  double roots[3];
  compute_roots_d(s, roots);
  const double d0 = s[0] - roots[0], d1 = s[3] - roots[0], d2 = s[5] - roots[0];
  // rows r0 = (d0, s1, s2), r1 = (s1, d1, s4), r2 = (s2, s4, d2); the longest of r0xr1, r0xr2, r1xr2
  const double v1[3] = {s[1] * s[4] - s[2] * d1, s[2] * s[1] - d0 * s[4], d0 * d1 - s[1] * s[1]};
  const double v2[3] = {s[1] * d2 - s[2] * s[4], s[2] * s[2] - d0 * d2, d0 * s[4] - s[1] * s[2]};
  const double v3[3] = {d1 * d2 - s[4] * s[4], s[4] * s[2] - s[1] * d2, s[1] * s[4] - d1 * s[2]};
  const double l1 = v1[0] * v1[0] + (v1[1] * v1[1] + v1[2] * v1[2]);
  const double l2 = v2[0] * v2[0] + (v2[1] * v2[1] + v2[2] * v2[2]);
  const double l3 = v3[0] * v3[0] + (v3[1] * v3[1] + v3[2] * v3[2]);
  double v[3], l;
  if (l1 >= l2 && l1 >= l3) { v[0] = v1[0]; v[1] = v1[1]; v[2] = v1[2]; l = l1; }
  else if (l2 >= l1 && l2 >= l3) { v[0] = v2[0]; v[1] = v2[1]; v[2] = v2[2]; l = l2; }
  else { v[0] = v3[0]; v[1] = v3[1]; v[2] = v3[2]; l = l3; }
  const double sl = sqrt(l);
  n[0] = v[0] / sl; n[1] = v[1] / sl; n[2] = v[2] / sl;
  return roots[0] * scale;
}

__device__ __forceinline__ double dot3(const double a[3], const double b[3]) {
  return a[0] * b[0] + (a[1] * b[1] + a[2] * b[2]);
}

// Moment index of u^a v^b, a + b <= D, a outer / b inner (PCL's monomial order for D = order).
template <int D>
__host__ __device__ constexpr int mono(int a, int b) { return a * (D + 1) - a * (a - 1) / 2 + b; }

template <int ORDER, bool RECORDS>
__global__ void __launch_bounds__(128) k_mls(MlsParams P, MlsRecords Q) {
  pdl_prologue();
  constexpr int NC = (ORDER + 1) * (ORDER + 2) / 2;   // coefficients (10 at order 3)
  constexpr int D2 = ORDER > 1 ? 2 * ORDER : 0;
  constexpr int NM = (D2 + 1) * (D2 + 2) / 2;         // moments sum w u^a v^b, a + b <= 2 order (28 at order 3)
  const GridView& g = P.g;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool valid = t < P.nq;
  float qx = 0.f, qy = 0.f, qz = 0.f;
  int64_t row = 0;
  if (valid) {
    PPP_DEV_ASSERT(t < g.n_sorted);
    const float4 p = __ldg(g.sorted + t);
    qx = p.x; qy = p.y; qz = p.z;
    row = __float_as_int(p.w);
    valid = P.choice == nullptr || __ldg(P.choice + row) == P.my_proj;
    if (RECORDS && Q.nmap) valid = valid && __ldg(Q.nmap + row) >= 0;   // halo copies are candidates, never queries
  }
  if ((P.choice || (RECORDS && Q.nmap)) && !__any_sync(0xffffffffu, valid)) return;
  int cu = 0, cv = 0;
  if (valid) {
    cu = cell_coord_raw(axis_of(qx, qy, qz, g.au), g.min_u, g.inv_h);
    cv = cell_coord_raw(axis_of(qx, qy, qz, g.av), g.min_v, g.inv_h);
  }
  const double qd[3] = {(double)qx, (double)qy, (double)qz};

  // ---- visit 1: neighbour count, centroid, covariance --------------------------------------------
  int m = 0;
  double s1[3] = {0.0, 0.0, 0.0}, s2[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  mls_visit(P, valid, cu, cv, qx, qy, qz, [&](const float4& c) {
    const double dx = (double)c.x - qd[0], dy = (double)c.y - qd[1], dz = (double)c.z - qd[2];
    m++;
    s1[0] += dx; s1[1] += dy; s1[2] += dz;
    s2[0] = __fma_rn(dx, dx, s2[0]); s2[1] = __fma_rn(dx, dy, s2[1]); s2[2] = __fma_rn(dx, dz, s2[2]);
    s2[3] = __fma_rn(dy, dy, s2[3]); s2[4] = __fma_rn(dy, dz, s2[4]); s2[5] = __fma_rn(dz, dz, s2[5]);
  });
  const bool emit = valid && m >= 3;   // fewer than 3 neighbours: no output row
  const double inv_m = emit ? 1.0 / (double)m : 0.0;
  const double mu[3] = {s1[0] * inv_m, s1[1] * inv_m, s1[2] * inv_m};   // centroid - q
  double cov[6];
  cov[0] = s2[0] - s1[0] * mu[0]; cov[1] = s2[1] - s1[0] * mu[1]; cov[2] = s2[2] - s1[0] * mu[2];
  cov[3] = s2[3] - s1[1] * mu[1]; cov[4] = s2[4] - s1[1] * mu[2]; cov[5] = s2[5] - s1[2] * mu[2];
  double n[3] = {0.0, 0.0, 1.0};
  double lambda0 = 0.0;
  if (emit) lambda0 = eigen33_d(cov, n);
  const double trace = cov[0] + cov[3] + cov[5];
  const double curvature = trace != 0.0 ? fabs(lambda0 / trace) : 0.0;
  // distance of q from the plane through the centroid: (q - c).n = -(mu.n); mean = q - distance n
  const double dist = -dot3(mu, n);
  const double mean[3] = {qd[0] - dist * n[0], qd[1] - dist * n[1], qd[2] - dist * n[2]};
  // Eigen unitOrthogonal, u = n x v
  double va[3];
  if (!(fabs(n[0]) <= fabs(n[2]) * 1e-12) || !(fabs(n[1]) <= fabs(n[2]) * 1e-12)) {
    const double inv = 1.0 / sqrt(n[0] * n[0] + n[1] * n[1]);
    va[0] = -n[1] * inv; va[1] = n[0] * inv; va[2] = 0.0;
  } else {
    const double inv = 1.0 / sqrt(n[1] * n[1] + n[2] * n[2]);
    va[0] = 0.0; va[1] = -n[2] * inv; va[2] = n[1] * inv;
  }
  const double ua[3] = {n[1] * va[2] - n[2] * va[1], n[2] * va[0] - n[0] * va[2], n[0] * va[1] - n[1] * va[0]};
  const double qm[3] = {qd[0] - mean[0], qd[1] - mean[1], qd[2] - mean[2]};
  const double uq = dot3(qm, ua), vq = dot3(qm, va);

  double outp[3] = {mean[0] + uq * ua[0] + vq * va[0], mean[1] + uq * ua[1] + vq * va[1], mean[2] + uq * ua[2] + vq * va[2]};
  double outn[3] = {n[0], n[1], n[2]};

  if constexpr (ORDER > 1) {
    // ---- visit 2: weighted moments and right-hand side ---------------------------------------------
    const bool fit = emit && m >= NC;
    double M[NM], F[NC];
#pragma unroll
    for (int i = 0; i < NM; i++) M[i] = 0.0;
#pragma unroll
    for (int i = 0; i < NC; i++) F[i] = 0.0;
    mls_visit(P, fit, cu, cv, qx, qy, qz, [&](const float4& c) {
      const double d[3] = {(double)c.x - mean[0], (double)c.y - mean[1], (double)c.z - mean[2]};
      const double w = exp(-dot3(d, d) * P.inv_sq_radius);
      const double u = dot3(d, ua), v = dot3(d, va), f = dot3(d, n);
      double vp[D2 + 1];
      vp[0] = 1.0;
#pragma unroll
      for (int b = 1; b <= D2; b++) vp[b] = vp[b - 1] * v;
      double wu = w;
#pragma unroll
      for (int a = 0; a <= D2; a++) {
#pragma unroll
        for (int b = 0; a + b <= D2; b++) M[mono<D2>(a, b)] = __fma_rn(wu, vp[b], M[mono<D2>(a, b)]);
        if (a <= ORDER) {
          const double wfu = wu * f;
#pragma unroll
          for (int b = 0; a + b <= ORDER; b++) F[mono<ORDER>(a, b)] = __fma_rn(wfu, vp[b], F[mono<ORDER>(a, b)]);
        }
        wu *= u;
      }
    });
    if (fit) {
      // A = P W P^T from the moments; Eigen's unblocked LLT (left-looking; on a pivot <= 0 it stops and the
      // solve runs on the partly factored matrix, as PCL's llt().solveInPlace does)
      double L[NC * (NC + 1) / 2];   // lower triangle, row-major
#pragma unroll
      for (int i = 0; i < NC; i++) {
#pragma unroll
        for (int j = 0; j <= i; j++) {
          int ia = 0, ib = 0, ja = 0, jb = 0;
#pragma unroll
          for (int a = 0, k = 0; a <= ORDER; a++)
#pragma unroll
            for (int b = 0; a + b <= ORDER; b++, k++) {
              if (k == i) { ia = a; ib = b; }
              if (k == j) { ja = a; jb = b; }
            }
          L[i * (i + 1) / 2 + j] = M[mono<D2>(ia + ja, ib + jb)];
        }
      }
      bool ok = true;
#pragma unroll
      for (int k = 0; k < NC; k++) {
        if (ok) {
          double x = L[k * (k + 1) / 2 + k];
#pragma unroll
          for (int j = 0; j < k; j++) x -= L[k * (k + 1) / 2 + j] * L[k * (k + 1) / 2 + j];
          if (x <= 0.0) {
            ok = false;
          } else {
            x = sqrt(x);
            L[k * (k + 1) / 2 + k] = x;
#pragma unroll
            for (int i = k + 1; i < NC; i++) {
              double a = L[i * (i + 1) / 2 + k];
#pragma unroll
              for (int j = 0; j < k; j++) a -= L[i * (i + 1) / 2 + j] * L[k * (k + 1) / 2 + j];
              L[i * (i + 1) / 2 + k] = a / x;
            }
          }
        }
      }
      double c[NC];
#pragma unroll
      for (int i = 0; i < NC; i++) {   // L y = F
        double a = F[i];
#pragma unroll
        for (int j = 0; j < i; j++) a -= L[i * (i + 1) / 2 + j] * c[j];
        c[i] = a / L[i * (i + 1) / 2 + i];
      }
#pragma unroll
      for (int i = NC - 1; i >= 0; i--) {   // L^T c = y
        double a = c[i];
#pragma unroll
        for (int j = i + 1; j < NC; j++) a -= L[j * (j + 1) / 2 + i] * c[j];
        c[i] = a / L[i * (i + 1) / 2 + i];
      }
      if (isfinite(c[0])) {
        // getPolynomialPartialDerivative at (uq, vq): z, z_u, z_v
        double z = 0.0, zu = 0.0, zv = 0.0;
        double u_pow = 1.0, u_prev = 0.0;
#pragma unroll
        for (int a = 0; a <= ORDER; a++) {
          double v_pow = 1.0, v_prev = 0.0;
#pragma unroll
          for (int b = 0; a + b <= ORDER; b++) {
            const double cj = c[mono<ORDER>(a, b)];
            z += u_pow * v_pow * cj;
            if (a >= 1) zu += cj * a * u_prev * v_pow;
            if (b >= 1) zv += cj * b * u_pow * v_prev;
            v_prev = v_pow;
            v_pow *= vq;
          }
          u_prev = u_pow;
          u_pow *= uq;
        }
#pragma unroll
        for (int i = 0; i < 3; i++) {
          outp[i] += z * n[i];
          outn[i] = n[i] - (zu * ua[i] + zv * va[i]);
        }
        const double nn = outn[0] * outn[0] + (outn[1] * outn[1] + outn[2] * outn[2]);
        if (nn > 0.0) {
          const double sn = sqrt(nn);
          outn[0] /= sn; outn[1] /= sn; outn[2] /= sn;
        }
      }
    }
  }
  if constexpr (RECORDS) {   // every query's record is written, so nothing of an earlier call survives in the buffer
    if (!valid) return;
    PPP_DEV_ASSERT(row >= 0);
    float o[8];
    if (emit) {
      o[0] = (float)outp[0]; o[1] = (float)outp[1]; o[2] = (float)outp[2]; o[3] = 1.0f;
      o[4] = (float)outn[0]; o[5] = (float)outn[1]; o[6] = (float)outn[2]; o[7] = (float)curvature;
    } else {
      mls_no_row(o);
    }
    store_mls_record(Q.rec, Q.nmap, row, o, Q.route);
    return;
  }
  if (!emit) return;
  PPP_DEV_ASSERT(row >= 0);
  P.xyz_out[row] = make_float4((float)outp[0], (float)outp[1], (float)outp[2], 0.0f);
  if (P.nrm_out) P.nrm_out[row] = make_float4((float)outn[0], (float)outn[1], (float)outn[2], (float)curvature);
  P.emit[row] = 1;
}

// Compaction: row row_base + pos[i] of the output gets point i's results (pos = exclusive scan of emit).  Inputs
// xyz (x, y, z) and nrm (nx, ny, nz, curvature) are read as float4 at a stride of in_sf floats; output points are
// records of out_sf floats whose other fields come from the source records src_rec (nullptr: x, y, z only).
__global__ void __launch_bounds__(256) k_mls_scatter(const int32_t* __restrict__ emit, const int32_t* __restrict__ pos,
                                                     int64_t n, const float* __restrict__ xyz, const float* __restrict__ nrm, int in_sf,
                                                     const float* __restrict__ src_rec, int out_sf, float* __restrict__ xyz_c,
                                                     float4* __restrict__ nrm_c, int32_t* __restrict__ src_c, int64_t row_base,
                                                     int32_t idx_base) {
  pdl_prologue();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !__ldg(emit + i)) return;
  const int32_t at = __ldg(pos + i);
  PPP_DEV_ASSERT(at >= 0 && at < __ldg(pos + n) && (int64_t)at <= i);
  const int64_t o = row_base + at;
  const float4 p = __ldg(reinterpret_cast<const float4*>(xyz + i * in_sf));
  float* d = xyz_c + o * out_sf;
  if (src_rec)
    for (int k = 3; k < out_sf; k++) d[k] = __ldg(src_rec + i * out_sf + k);
  d[0] = p.x; d[1] = p.y; d[2] = p.z;
  if (nrm_c) nrm_c[o] = __ldg(reinterpret_cast<const float4*>(nrm + i * in_sf));
  src_c[o] = idx_base + (int32_t)i;
}

// Output flags of n records: emit[i] = 1 where record i has a row.
__global__ void __launch_bounds__(256) k_mls_flags(const float* __restrict__ rec, int64_t n, int32_t* __restrict__ emit) {
  pdl_prologue();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) emit[i] = __ldg(rec + i * 8 + 3) == 1.0f ? 1 : 0;
}

// Records of the points that are not indexed (a non-finite coordinate): no row.
__global__ void __launch_bounds__(256) k_mls_default_rows(const float4* __restrict__ xyz4, int64_t n, float* rec,
                                                          const int32_t* __restrict__ nmap, const NormalRoute* __restrict__ route) {
  pdl_prologue();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = __ldg(xyz4 + i);
  if (p.w == p.w) return;
  float o[8];
  mls_no_row(o);
  store_mls_record(rec, nmap, i, o, route);
}

template <int ORDER, bool RECORDS>
int launch_mls_order(ppp_ctx* ctx, const MlsParams& P, const MlsRecords& Q) {
  static const char* names[4] = {"mls_plane", "mls_plane", "mls_order2", "mls_order3"};
  auto kern = k_mls<ORDER, RECORDS>;
  const unsigned blocks = (unsigned)((P.nq + 127) / 128);
  PPP_LAUNCH(ctx, names[ORDER], kern, blocks, 128, 0, P, Q);
  PPP_CHECK_LAUNCH();
  return PPP_OK;
}

// out: the output fields of MlsParams (xyz_out ... route); the rest is filled in here.
template <bool RECORDS>
int launch_mls(ppp_ctx* ctx, const GridStore& gs, double radius, int order, const unsigned char* choice, int my_proj,
               const MlsParams& out, const MlsRecords& Q) {
  if (gs.v.n_sorted <= 0) return PPP_OK;
  MlsParams P = out;
  P.g = gs.v;
  P.nq = gs.v.n_sorted;
  P.r2 = (float)(radius * radius);   // [upstream] pcl::KdTreeFLANN::radiusSearch
  P.R = radius_rings(gs.v, std::sqrt((double)P.r2));
  P.inv_sq_radius = 1.0 / (radius * radius);
  P.choice = choice; P.my_proj = my_proj;
  switch (order) {
    case 0: case 1: return launch_mls_order<1, RECORDS>(ctx, P, Q);
    case 2: return launch_mls_order<2, RECORDS>(ctx, P, Q);
    default: return launch_mls_order<3, RECORDS>(ctx, P, Q);
  }
}

// k_mls over every indexed point of the cloud (through the multi-projection index where the cloud needs it).
template <bool RECORDS>
int mls_over_cloud(ppp_cloud* c, double radius, int order, const MlsParams& out, const MlsRecords& Q) {
  const double h = cloud_cell_for_radius(c, radius);
  GridStore* g;
  PPP_TRY(cloud_get_grid(c, h, &g));
  PPP_TRY(cloud_decide_projection(c, *g));
  if (c->mp_state == 1) {
    // not a height field: every point is answered through the projection that spreads its block out best
    MPSet* mp;
    PPP_TRY(cloud_get_mp(c, h, 2, &mp));   // cloud_cell_for_radius sizes the cells so that two rings cover the radius
    for (int p = 0; p < 3; p++) PPP_TRY(launch_mls<RECORDS>(c->ctx, *mp->g[p], radius, order, mp->choice, p, out, Q));
    return PPP_OK;
  }
  return launch_mls<RECORDS>(c->ctx, *g, radius, order, nullptr, 0, out, Q);
}

}  // namespace

int mls_smooth_launch(ppp_cloud* c, double radius, int order, float* xyz_c, float4* nrm_c, int32_t* src_c, int64_t* n_rows) {
  ppp_ctx* ctx = c->ctx;
  *n_rows = 0;
  if (order < 0 || order > 3) {
    ppp_set_error("ppp_mls_smooth: polynomial order %d is not supported (0..3)", order);
    return PPP_ERR_UNSUPPORTED;
  }
  if (c->n == 0) return PPP_OK;
  float4 *xyz = nullptr, *nrm = nullptr;
  int32_t *emit = nullptr, *pos = nullptr;
  PPP_TRY(dev_alloc(ctx, &xyz, (size_t)c->n));
  if (nrm_c) PPP_TRY(dev_alloc(ctx, &nrm, (size_t)c->n));
  PPP_TRY(dev_alloc(ctx, &emit, (size_t)c->n));
  PPP_TRY(dev_alloc(ctx, &pos, (size_t)c->n + 1));
  PPP_CUDA(cudaMemsetAsync(emit, 0, (size_t)c->n * sizeof(int32_t), ctx->stream));
  MlsParams out{};
  out.xyz_out = xyz; out.nrm_out = nrm; out.emit = emit;
  PPP_TRY(mls_over_cloud<false>(c, radius, order, out, MlsRecords{}));
  PPP_TRY(scan_exclusive_i32(ctx, emit, pos, c->n));
  {
    const unsigned blocks = (unsigned)((c->n + 255) / 256);
    PPP_LAUNCH(ctx, "mls_scatter", k_mls_scatter, blocks, 256, 0, (const int32_t*)emit, (const int32_t*)pos, c->n,
               (const float*)xyz, (const float*)nrm, 4, (const float*)nullptr, 3, xyz_c, nrm_c, src_c, (int64_t)0,
               (int32_t)0);
    PPP_CHECK_LAUNCH();
  }
  int32_t total = 0;
  PPP_CUDA(cudaMemcpyAsync(&total, pos + c->n, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  PPP_CUDA(cudaStreamSynchronize(ctx->stream));
  dev_free(ctx, xyz); dev_free(ctx, nrm); dev_free(ctx, emit); dev_free(ctx, pos);
  *n_rows = total;
  return PPP_OK;
}

int mls_smooth_records(ppp_cloud* c, double radius, int order, float* rec) {
  ppp_ctx* ctx = c->ctx;
  if (c->n == 0) return PPP_OK;
  MlsRecords out{};
  out.rec = rec; out.nmap = c->nmap; out.route = c->nmap ? c->route : nullptr;
  PPP_TRY(mls_over_cloud<true>(c, radius, order, MlsParams{}, out));
  if (c->n_finite < c->n) {   // non-finite points are not indexed: their records are written here
    const unsigned blocks = (unsigned)((c->n + 255) / 256);
    PPP_LAUNCH(ctx, "mls_default_rows", k_mls_default_rows, blocks, 256, 0, (const float4*)c->xyz4, c->n, rec, out.nmap, out.route);
    PPP_CHECK_LAUNCH();
  }
  return PPP_OK;
}

int mls_compact_launch(ppp_ctx* ctx, const float* rec, int64_t n, const float* src_rec, int out_sf, int32_t idx_base,
                       int64_t row_base, float* points_out, float4* normals_out, int32_t* src_out, int64_t cap_rows,
                       int64_t* n_rows) {
  *n_rows = 0;
  if (n == 0) return PPP_OK;
  int32_t *emit = nullptr, *pos = nullptr;
  PPP_TRY(dev_alloc(ctx, &emit, (size_t)n));
  PPP_TRY(dev_alloc(ctx, &pos, (size_t)n + 1));
  const unsigned blocks = (unsigned)((n + 255) / 256);
  PPP_LAUNCH(ctx, "mls_flags", k_mls_flags, blocks, 256, 0, rec, n, emit);
  PPP_CHECK_LAUNCH();
  PPP_TRY(scan_exclusive_i32(ctx, emit, pos, n));
  int32_t total = 0;
  PPP_TRY(fetch_small(ctx, pos + n, sizeof(int32_t), &total));
  *n_rows = total;
  if (points_out) {
    if (row_base + total > cap_rows) {
      ppp_set_error("ppp_dev_mls_compact: the output holds %lld rows, rows up to %lld are needed", (long long)cap_rows,
                    (long long)(row_base + total));
      dev_free(ctx, emit); dev_free(ctx, pos);
      return PPP_ERR_CAPACITY;
    }
    PPP_LAUNCH(ctx, "mls_scatter", k_mls_scatter, blocks, 256, 0, (const int32_t*)emit, (const int32_t*)pos, n, rec, rec + 4, 8,
               src_rec, out_sf, points_out, normals_out, src_out, row_base, idx_base);
    PPP_CHECK_LAUNCH();
  }
  dev_free(ctx, emit); dev_free(ctx, pos);
  return PPP_OK;
}

// The exchange halo that keeps every MLS neighbour of an owned point in that point's slab (ppp_mls_halo).
//
// A candidate c is a neighbour of the query q when d2 = fl(fl(fl(dx^2) + fl(dy^2)) + fl(dz^2)) < r2, with
// dx = fl(q.x - c.x) and r2 = (float)(r * r) (d2_flann_x2, MlsParams::r2).
//  1. Rounding is monotone and the added terms are >= 0, so d2 >= fl(dx^2).  Let t be the smallest float with
//     fl(t * t) >= r2.  |dx| >= t would give fl(dx^2) >= fl(t * t) >= r2: a neighbour has |dx| < t.
//  2. t is a float and float subtraction is monotone, so |fl(q.x - c.x)| < t needs |q.x - c.x| < t exactly.
//  3. The exchange (exchange.cu, ex_dest_mask) owns a point by its histogram bin and copies c into slab o when
//     (double)c.x < fl(cut[o+1] + halo) or (double)c.x >= fl(cut[o] - halo).  The bin, fl((x - gmin) * inv), and
//     the cut, fl(gmin + span * bin / 1024), are each a few double roundings of quantities no larger than
//     M + span <= 3 M (M = largest finite |x|), so an owned q lies within 12 * 2^-53 * M of its slab's limits,
//     and fl(cut +- halo) moves the limit by at most 2^-53 * (M + halo).
// So halo = t + 2^-44 * (M + t + 1) (2^-44 = 512 * 2^-53, the 1 covers the span floor of 1e-9 and M = 0) puts
// every neighbour of every owned point into its slab.
double mls_halo(double radius, double x_abs_max) {
  if (!(radius > 0) || !std::isfinite((float)(radius * radius)) || !(x_abs_max >= 0) || !std::isfinite(x_abs_max))
    return std::nan("");
  const float r2 = (float)(radius * radius);
  auto sq = [](float v) { return (float)((double)v * (double)v); };   // the product is exact in double: fl32(v * v)
  float t = (float)std::sqrt((double)r2);
  while (t > 0.0f && sq(std::nextafter(t, 0.0f)) >= r2) t = std::nextafter(t, 0.0f);
  while (sq(t) < r2) t = std::nextafter(t, INFINITY);
  return (double)t + 0x1p-44 * (x_abs_max + (double)t + 1.0);
}
