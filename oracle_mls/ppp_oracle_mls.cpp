// ppp_oracle_mls.cpp — CPU ORACLE for the MLS pre-filter. TEST INFRASTRUCTURE ONLY.
//
// smooth() of the reference (src/Path_Generation.cpp:340-360): pcl::MovingLeastSquares<PointXYZRGB,
// PointXYZRGB> with setPolynomialOrder(3), setSearchRadius(15) and PCL 1.10 defaults otherwise -- no
// upsampling, SIMPLE projection, weight exp(-d2 / r^2).  Restated literally, point by point, on the
// kd-tree radius search of oracle/ppp_oracle.cpp (compiled into this library unchanged):
// [upstream, recalled] MovingLeastSquares::computeMLSPointNormal, MLSResult::computeMLSSurface,
// compute3DCentroid, computeCovarianceMatrix, eigen33 (double), Eigen unitOrthogonal, the Eigen
// unblocked LLT, projectQueryPoint / projectPointSimpleToPolynomialSurface / projectPointToMLSPlane and
// getPolynomialPartialDerivative.  Sums run in the neighbour list's (d2, idx) order; no FMA (Makefile).
// tests/golden/mls_f64_numpy.py is the independent second restatement this file is checked against.
#include "../oracle/ppp_oracle.cpp"

namespace {

// pcl::computeRoots2 / computeRoots / eigen33 for Matrix3d (same statements as the float versions above).
inline void compute_roots2_d(double b, double c, double roots[3]) {
  roots[0] = 0.0;
  double d = b * b - 4.0 * c;
  if (d < 0.0) d = 0.0;
  double sd = std::sqrt(d);
  roots[2] = 0.5 * (b + sd);
  roots[1] = 0.5 * (b - sd);
}

inline void compute_roots_d(const double m[6], double roots[3]) {
  const double m00 = m[0], m01 = m[1], m02 = m[2], m11 = m[3], m12 = m[4], m22 = m[5];
  double c0 = m00 * m11 * m22 + 2.0 * m01 * m02 * m12 - m00 * m12 * m12 - m11 * m02 * m02 - m22 * m01 * m01;
  double c1 = m00 * m11 - m01 * m01 + m00 * m22 - m02 * m02 + m11 * m22 - m12 * m12;
  double c2 = m00 + m11 + m22;
  if (std::fabs(c0) < std::numeric_limits<double>::epsilon()) {
    compute_roots2_d(c2, c1, roots);
    return;
  }
  const double s_inv3 = 1.0 / 3.0;
  const double s_sqrt3 = std::sqrt(3.0);
  double c2_over_3 = c2 * s_inv3;
  double a_over_3 = (c1 - c2 * c2_over_3) * s_inv3;
  if (a_over_3 > 0.0) a_over_3 = 0.0;
  double half_b = 0.5 * (c0 + c2_over_3 * (2.0 * c2_over_3 * c2_over_3 - c1));
  double q = half_b * half_b + a_over_3 * a_over_3 * a_over_3;
  if (q > 0.0) q = 0.0;
  double rho = std::sqrt(-a_over_3);
  double theta = std::atan2(std::sqrt(-q), half_b) * s_inv3;
  double cos_theta = std::cos(theta);
  double sin_theta = std::sin(theta);
  roots[0] = c2_over_3 + 2.0 * rho * cos_theta;
  roots[1] = c2_over_3 - rho * (cos_theta + s_sqrt3 * sin_theta);
  roots[2] = c2_over_3 - rho * (cos_theta - s_sqrt3 * sin_theta);
  if (roots[0] >= roots[1]) std::swap(roots[0], roots[1]);
  if (roots[1] >= roots[2]) {
    std::swap(roots[1], roots[2]);
    if (roots[0] >= roots[1]) std::swap(roots[0], roots[1]);
  }
  if (roots[0] <= 0.0) compute_roots2_d(c2, c1, roots);
}

inline void cross3_d(const double a[3], const double b[3], double o[3]) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}
inline double dot3_d(const double a[3], const double b[3]) { return a[0] * b[0] + (a[1] * b[1] + a[2] * b[2]); }

// cov: 00 01 02 11 12 22.  Returns the smallest eigenvalue, n = its unit eigenvector.
inline double eigen33_d(const double cov[6], double n[3]) {
  double scale = 0.0;
  for (int i = 0; i < 6; i++) scale = std::max(scale, std::fabs(cov[i]));
  if (scale <= std::numeric_limits<double>::min()) scale = 1.0;
  double s[6];
  for (int i = 0; i < 6; i++) s[i] = cov[i] / scale;
  double roots[3];
  compute_roots_d(s, roots);
  double d0 = s[0] - roots[0], d1 = s[3] - roots[0], d2 = s[5] - roots[0];
  double r0[3] = {d0, s[1], s[2]}, r1[3] = {s[1], d1, s[4]}, r2[3] = {s[2], s[4], d2};
  double v1[3], v2[3], v3[3];
  cross3_d(r0, r1, v1); cross3_d(r0, r2, v2); cross3_d(r1, r2, v3);
  double l1 = dot3_d(v1, v1), l2 = dot3_d(v2, v2), l3 = dot3_d(v3, v3);
  const double* v; double l;
  if (l1 >= l2 && l1 >= l3) { v = v1; l = l1; }
  else if (l2 >= l1 && l2 >= l3) { v = v2; l = l2; }
  else { v = v3; l = l3; }
  double sl = std::sqrt(l);
  n[0] = v[0] / sl; n[1] = v[1] / sl; n[2] = v[2] / sl;
  return roots[0] * scale;
}

struct MlsRow {
  float xyz[3];
  float nrm[4];
  int fit;   // 1: polynomial projection, 0: plane projection
};

// One query (computeMLSPointNormal with upsampling NONE).  nb: the radius neighbours in (d2, idx) order.
void mls_point(const Pts& P, const Key* nb, int m, const float* qf, double radius, int order, MlsRow& out,
               std::vector<double>& buf) {
  // compute3DCentroid
  double c[3] = {0, 0, 0};
  for (int j = 0; j < m; j++) {
    const float* p = P.at(nb[j].idx);
    c[0] += p[0]; c[1] += p[1]; c[2] += p[2];
  }
  for (int i = 0; i < 3; i++) c[i] /= (double)m;
  // computeCovarianceMatrix (unnormalised)
  double cov[6] = {0, 0, 0, 0, 0, 0};   // 00 01 02 11 12 22
  for (int j = 0; j < m; j++) {
    const float* p = P.at(nb[j].idx);
    double x = p[0] - c[0], y = p[1] - c[1], z = p[2] - c[2];
    cov[3] += y * y; cov[4] += y * z; cov[5] += z * z;
    cov[0] += x * x; cov[1] += y * x; cov[2] += z * x;
  }
  double n[3];
  const double eigen_value = eigen33_d(cov, n);
  const double d_plane = -1.0 * (n[0] * c[0] + n[1] * c[1] + n[2] * c[2] + 0.0 * 1.0);
  const double q[3] = {(double)qf[0], (double)qf[1], (double)qf[2]};
  const double distance = dot3_d(q, n) + d_plane;
  const double mean[3] = {q[0] - distance * n[0], q[1] - distance * n[1], q[2] - distance * n[2]};
  double curvature = cov[0] + cov[3] + cov[5];
  if (curvature != 0) curvature = std::fabs(eigen_value / curvature);
  // Darboux frame: v = n.unitOrthogonal(), u = n x v
  double va[3], ua[3];
  if (!(std::fabs(n[0]) <= std::fabs(n[2]) * 1e-12) || !(std::fabs(n[1]) <= std::fabs(n[2]) * 1e-12)) {
    double invnm = 1.0 / std::sqrt(n[0] * n[0] + n[1] * n[1]);
    va[0] = -n[1] * invnm; va[1] = n[0] * invnm; va[2] = 0.0;
  } else {
    double invnm = 1.0 / std::sqrt(n[1] * n[1] + n[2] * n[2]);
    va[0] = 0.0; va[1] = -n[2] * invnm; va[2] = n[1] * invnm;
  }
  cross3_d(n, va, ua);
  // polynomial fit
  const int nc = (order + 1) * (order + 2) / 2;
  bool have_c = false;
  double cvec[10];
  if (order > 1 && m >= nc) {
    const double sq_r = radius * radius;
    buf.assign((size_t)m * (nc + 2), 0.0);
    double* w = buf.data();            // m
    double* f = w + m;                 // m
    double* Pm = f + m;                // nc x m
    for (int ni = 0; ni < m; ni++) {
      const float* p = P.at(nb[ni].idx);
      double de[3] = {p[0] - mean[0], p[1] - mean[1], p[2] - mean[2]};
      w[ni] = std::exp(-dot3_d(de, de) / sq_r);
      const double u = dot3_d(de, ua), v = dot3_d(de, va);
      f[ni] = dot3_d(de, n);
      int j = 0;
      double u_pow = 1;
      for (int ui = 0; ui <= order; ++ui) {
        double v_pow = 1;
        for (int vi = 0; vi <= order - ui; ++vi) {
          Pm[(size_t)(j++) * m + ni] = u_pow * v_pow;
          v_pow *= v;
        }
        u_pow *= u;
      }
    }
    // P_weight = P diag(w); A = P_weight P^T (lower triangle: all the LLT reads); c = P_weight f
    double A[10][10];
    for (int i = 0; i < nc; i++) {
      for (int k = 0; k <= i; k++) {
        double s = 0;
        for (int ni = 0; ni < m; ni++) s += (Pm[(size_t)i * m + ni] * w[ni]) * Pm[(size_t)k * m + ni];
        A[i][k] = s;
      }
      double s = 0;
      for (int ni = 0; ni < m; ni++) s += (Pm[(size_t)i * m + ni] * w[ni]) * f[ni];
      cvec[i] = s;
    }
    // Eigen llt_inplace<.., Lower>::unblocked: on a pivot <= 0 it returns, and solveInPlace still runs on
    // the partly factored matrix
    for (int k = 0; k < nc; k++) {
      double x = A[k][k];
      double sn = 0;
      for (int j = 0; j < k; j++) sn += A[k][j] * A[k][j];
      if (k > 0) x -= sn;
      if (x <= 0.0) break;
      A[k][k] = x = std::sqrt(x);
      for (int i = k + 1; i < nc; i++) {
        double s = 0;
        for (int j = 0; j < k; j++) s += A[i][j] * A[k][j];
        if (k > 0) A[i][k] -= s;
        A[i][k] /= x;
      }
    }
    for (int i = 0; i < nc; i++) {
      double s = cvec[i];
      for (int j = 0; j < i; j++) s -= A[i][j] * cvec[j];
      cvec[i] = s / A[i][i];
    }
    for (int i = nc - 1; i >= 0; i--) {
      double s = cvec[i];
      for (int j = i + 1; j < nc; j++) s -= A[j][i] * cvec[j];
      cvec[i] = s / A[i][i];
    }
    have_c = true;
  }
  // projectQueryPoint(SIMPLE, nr_coeff)
  const double dq[3] = {q[0] - mean[0], q[1] - mean[1], q[2] - mean[2]};
  const double u = dot3_d(dq, ua), v = dot3_d(dq, va);
  double pt[3], nr[3] = {n[0], n[1], n[2]};
  double w = 0;
  out.fit = 0;
  if (have_c && std::isfinite(cvec[0])) {
    // getPolynomialPartialDerivative(u, v): z, z_u, z_v
    double z = 0, z_u = 0, z_v = 0;
    int j = 0;
    double u_pow = 1, u_pow_prev = 0;
    for (int ui = 0; ui <= order; ++ui) {
      double v_pow = 1, v_pow_prev = 0;
      for (int vi = 0; vi <= order - ui; ++vi) {
        z += u_pow * v_pow * cvec[j];
        if (ui >= 1) z_u += cvec[j] * ui * u_pow_prev * v_pow;
        if (vi >= 1) z_v += cvec[j] * vi * u_pow * v_pow_prev;
        v_pow_prev = v_pow;
        v_pow *= v;
        ++j;
      }
      u_pow_prev = u_pow;
      u_pow *= u;
    }
    w = z;
    for (int i = 0; i < 3; i++) nr[i] -= (z_u * ua[i] + z_v * va[i]);
    double sq = dot3_d(nr, nr);
    if (sq > 0) { double s = std::sqrt(sq); nr[0] /= s; nr[1] /= s; nr[2] /= s; }
    out.fit = 1;
  }
  for (int i = 0; i < 3; i++) pt[i] = mean[i] + u * ua[i] + v * va[i] + w * n[i];
  for (int i = 0; i < 3; i++) { out.xyz[i] = (float)pt[i]; out.nrm[i] = (float)nr[i]; }
  out.nrm[3] = (float)curvature;
}

}  // namespace

extern "C" {

// MovingLeastSquares::process with the reference's settings.  Rows (ascending source index) for every finite
// point with >= 3 neighbours: pts_out 3 floats, normals_out (nullable) 4 floats {nx, ny, nz, curvature},
// src_out the source index, fit_out (nullable) 1 = polynomial projection / 0 = plane.  Returns the row count,
// -1 for an order outside 0..3.
int64_t ppo_mls_smooth(void* h, double radius, int order, float* pts_out, float* normals_out, int32_t* src_out,
                       int8_t* fit_out, int threads) {
  if (order < 0 || order > 3) return -1;
  Cloud* C = (Cloud*)h;
  const Pts& P = C->P;
  const float r2 = (float)(radius * radius);
  threads = clamp_threads(threads);
  std::vector<MlsRow> rows((size_t)P.n);
  std::vector<char> emit((size_t)P.n, 0);
#pragma omp parallel num_threads(threads)
  {
    std::vector<Key> nb;
    std::vector<double> buf;
#pragma omp for schedule(dynamic, 256)
    for (int64_t i = 0; i < P.n; i++) {
      const float* q = P.at(i);
      if (!finite3(q)) continue;
      C->tree.radius(q, r2, nb);
      if (nb.size() < 3) continue;
      mls_point(P, nb.data(), (int)nb.size(), q, radius, order, rows[(size_t)i], buf);
      emit[(size_t)i] = 1;
    }
  }
  int64_t o = 0;
  for (int64_t i = 0; i < P.n; i++) {
    if (!emit[(size_t)i]) continue;
    const MlsRow& r = rows[(size_t)i];
    for (int k = 0; k < 3; k++) pts_out[3 * o + k] = r.xyz[k];
    if (normals_out)
      for (int k = 0; k < 4; k++) normals_out[4 * o + k] = r.nrm[k];
    src_out[o] = (int32_t)i;
    if (fit_out) fit_out[o] = (int8_t)r.fit;
    o++;
  }
  return o;
}

}  // extern "C"
