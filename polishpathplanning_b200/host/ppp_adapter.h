// ppp_adapter.h — C++ mirrors of the reference's hot-path classes over the C ABI (include/ppp_gpu.h).
//
//   class path_generater   include/Path_Generate.h:35-76 + src/Path_Generation.cpp  (gen-2, ./main)
//   class SectPath         include/contour_alg.h:50-91   + src/contour_alg.cpp      (config.txt flow)
//
// Same member names, argument meaning and call order as the reference; only the bodies of the
// hot-path members are replaced by calls into libppp_gpu.so.  Everything else of the reference
// (dynamic adjustment, way-point export, PCLVisualizer, the GSL Spline) stays the reference's own
// host code: Spline(n, y, x, z) is constructed from the three double arrays returned here
// (include/Spline.h:10-20).  Without GSL in this image `Spline` is the node triple itself.
#pragma once
#include <algorithm>
#include <chrono>
#include <cmath>
#include <limits>
#include <cstdio>
#include <fstream>
#include <map>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/ppp_gpu.h"
#include "pcd_io_min.h"
#include "pcl_min.h"

typedef pcl::PointCloud<pcl::PointXYZRGB> PointCloudType;
typedef pcl::PointXYZRGB PointType;
typedef std::map<double, std::vector<double>> MAP;

#ifndef PPP_HAVE_GSL
// Stand-in for include/Spline.h when GSL is absent: the ordered nodes a Spline is built from.
// point(y) evaluates gsl_interp_steffen restated (Steffen 1990 monotone cubic; [upstream, recalled]).
class Spline {
public:
  Spline() {}
  Spline(int number, const double* point_y, const double* point_x, const double* point_z)
      : y(point_y, point_y + number), x(point_x, point_x + number), z(point_z, point_z + number) {
    ok_ = number >= 3;
    for (int i = 1; i < number && ok_; i++) ok_ = y[i] > y[i - 1];
    if (ok_) { coeffs(x, cx_); coeffs(z, cz_); }
  }
  bool valid() const { return ok_; }  // GSL aborts on < 3 nodes or non-increasing y; here: check before use
  Eigen::Vector3d point(double yy) const { return Eigen::Vector3d(eval(cx_, yy), yy, eval(cz_, yy)); }
  double miny() const { return y.empty() ? 0.0 : y.front(); }
  double bigy() const { return y.empty() ? 0.0 : y.back(); }
  std::vector<double> y, x, z;

private:
  struct C { std::vector<double> a, b, c, d; };
  static double cps(double v) { return std::copysign(1.0, v); }
  void coeffs(const std::vector<double>& ya, C& o) const {
    size_t n = y.size();
    std::vector<double> yp(n);
    yp[0] = (ya[1] - ya[0]) / (y[1] - y[0]);
    for (size_t i = 1; i + 1 < n; i++) {
      double hi = y[i + 1] - y[i], him1 = y[i] - y[i - 1];
      double si = (ya[i + 1] - ya[i]) / hi, sim1 = (ya[i] - ya[i - 1]) / him1;
      double pi = (sim1 * hi + si * him1) / (him1 + hi);
      yp[i] = (cps(sim1) + cps(si)) * std::min(std::fabs(sim1), std::min(std::fabs(si), 0.5 * std::fabs(pi)));
    }
    yp[n - 1] = (ya[n - 1] - ya[n - 2]) / (y[n - 1] - y[n - 2]);
    o.a.resize(n - 1); o.b.resize(n - 1); o.c.resize(n - 1); o.d.resize(n - 1);
    for (size_t i = 0; i + 1 < n; i++) {
      double hi = y[i + 1] - y[i], si = (ya[i + 1] - ya[i]) / hi;
      o.a[i] = (yp[i] + yp[i + 1] - 2 * si) / hi / hi;
      o.b[i] = (3 * si - 2 * yp[i] - yp[i + 1]) / hi;
      o.c[i] = yp[i];
      o.d[i] = ya[i];
    }
  }
  double eval(const C& o, double yy) const {
    if (!ok_ || !(yy >= y.front() && yy <= y.back())) return std::numeric_limits<double>::quiet_NaN();
    size_t i = std::upper_bound(y.begin(), y.end(), yy) - y.begin();
    i = i ? i - 1 : 0;
    if (i > y.size() - 2) i = y.size() - 2;
    double dx = yy - y[i];
    return o.d[i] + dx * (o.c[i] + dx * (o.b[i] + dx * o.a[i]));
  }
  bool ok_ = false;
  C cx_, cz_;
};
#endif

namespace ppp_host {

inline void check(int st, const char* what) {
  if (st != PPP_OK) throw std::runtime_error(std::string(what) + ": " + ppp_last_error());
}

// Device copy + index of one host cloud; rebuilt lazily after invalidate() (the reference mutates
// xyz in voxel_down / trans2center / smooth / remove_outlier / transformPointCloud).
class DeviceCloud {
public:
  explicit DeviceCloud(int device = 0) { check(ppp_create(device, &ctx_), "ppp_create"); }
  ~DeviceCloud() { ppp_cloud_free(cloud_); ppp_destroy(ctx_); }
  DeviceCloud(const DeviceCloud&) = delete;
  DeviceCloud& operator=(const DeviceCloud&) = delete;
  void invalidate() { ppp_cloud_free(cloud_); cloud_ = nullptr; }
  ppp_cloud* get(const PointCloudType& c) {
    if (!cloud_) check(ppp_cloud_upload(ctx_, c.points.data(), c.points.size(), sizeof(PointType), &cloud_), "ppp_cloud_upload");
    return cloud_;
  }
private:
  ppp_ctx* ctx_ = nullptr;
  ppp_cloud* cloud_ = nullptr;
};

struct Contours {
  std::vector<int64_t> offsets;  // S + 1
  std::vector<double> y, x, z;
  Spline path(int s) const {
    int64_t a = offsets[s], n = offsets[s + 1] - a;
    return Spline((int)n, y.data() + a, x.data() + a, z.data() + a);
  }
};

inline Contours slice_contours(ppp_cloud* c, const std::vector<float>& planes, int mode) {
  Contours r;
  int S = (int)planes.size();
  r.offsets.assign(S + 1, 0);
  check(ppp_slice_contours(c, planes.data(), S, 2.0f, 1, mode, r.offsets.data(), nullptr, nullptr, nullptr, 0), "ppp_slice_contours(size)");
  int64_t n = r.offsets[S];
  r.y.resize(n); r.x.resize(n); r.z.resize(n);
  check(ppp_slice_contours(c, planes.data(), S, 2.0f, 1, mode, r.offsets.data(), r.y.data(), r.x.data(), r.z.data(), n), "ppp_slice_contours");
  return r;
}

// rangedX_index(position): ONE band pass in the common case.  The index buffer is sized from the previous call
// on this thread (bands of neighbouring planes have similar populations); only when it turns out too small does
// the library report the required size and a second pass fill it.  (The reference's sweep loops call this once
// per plane, src/Path_Generation.cpp:716-723.)
inline std::vector<int> ranged_x_index(ppp_cloud* c, int position) {
  static thread_local int64_t cap_hint = 16384;
  const float px = (float)position;
  int64_t off[2] = {0, 0};
  std::vector<int> idx((size_t)cap_hint);
  int st = ppp_slice_bands(c, &px, 1, 2.0f, 1, off, idx.data(), (int64_t)idx.size());
  if (st == PPP_ERR_CAPACITY) {
    idx.resize((size_t)off[1]);
    st = ppp_slice_bands(c, &px, 1, 2.0f, 1, off, idx.data(), (int64_t)idx.size());
  }
  check(st, "ppp_slice_bands");
  idx.resize((size_t)off[1]);
  cap_hint = std::max<int64_t>(16384, off[1] + off[1] / 4);
  return idx;
}

// insert_point with the caller's index list (strictly ascending, as rangedX_index returns it)
inline MAP insert_point(ppp_cloud* c, const std::vector<int>& indices, float plane_x, int mode) {
  int64_t n = 0;
  std::vector<double> y(indices.size() + 1), x(indices.size() + 1), z(indices.size() + 1);
  check(ppp_insert_point(c, indices.data(), (int64_t)indices.size(), plane_x, mode, y.data(), x.data(), z.data(),
                         (int64_t)y.size(), &n), "ppp_insert_point");
  MAP m;
  for (int64_t i = 0; i < n; i++) m[y[i]] = {x[i], z[i]};
  return m;
}

// smooth() (src/Path_Generation.cpp:340-360): MovingLeastSquares, order 3, radius 15, on the device.  The cloud
// is replaced by the smoothed records (x, y, z from the fit, every other field from the source point; points with
// fewer than 3 neighbours are dropped) and written to smooth_<file name>.pcd in the working directory.
inline void mls_smooth(ppp_cloud* dc, PointCloudType& cloud, const std::string& cloud_name) {
  const size_t n = cloud.points.size();
  std::vector<PointType> xyz(n);
  std::vector<int32_t> src(n);
  int64_t m = 0;
  check(ppp_mls_smooth(dc, 15.0, 3, xyz.data(), sizeof(PointType), nullptr, src.data(), &m), "ppp_mls_smooth");
  std::vector<PointType, decltype(cloud.points.get_allocator())> out((size_t)m);
  for (int64_t i = 0; i < m; i++) {
    out[(size_t)i] = cloud.points[(size_t)src[(size_t)i]];
    out[(size_t)i].x = xyz[(size_t)i].x; out[(size_t)i].y = xyz[(size_t)i].y; out[(size_t)i].z = xyz[(size_t)i].z;
  }
  cloud.points.swap(out);
  cloud.width = (uint32_t)m; cloud.height = 1;
  const size_t slash = cloud_name.find_last_of('/');
  const std::string out_name = "smooth_" + (slash == std::string::npos ? cloud_name : cloud_name.substr(slash + 1));
  if (savePCDFile(out_name, cloud) != 0) fprintf(stderr, "smooth: could not write %s\n", out_name.c_str());
}

// voxel_down() (src/Path_Generation.cpp:53-59): pcl::VoxelGrid with leaf sizes (lx, ly, lz) on the device.  The cloud
// is replaced by one point per occupied voxel: x, y, z from the device, r, g, b, a averaged over the voxel's members
// as PCL's CentroidPoint does (float sums in member order, divided by the count, truncated).  Where PCL warns that the
// leaf is too small and keeps the input, so does this.  Returns false then.
inline bool voxel_down(ppp_cloud* dc, PointCloudType& cloud, float lx, float ly, float lz) {
  const size_t n = cloud.points.size();
  const float leaf[3] = {lx, ly, lz};
  std::vector<PointType, decltype(cloud.points.get_allocator())> out(n);
  std::vector<int64_t> off(n + 1);
  std::vector<int32_t> members(n);
  int64_t m = 0;
  const int st = ppp_voxel_grid(dc, leaf, out.data(), sizeof(PointType), off.data(), members.data(), &m);
  if (st == PPP_ERR_UNSUPPORTED) {
    fprintf(stderr, "[pcl::VoxelGrid::applyFilter] %s\n", ppp_last_error());
    return false;
  }
  check(st, "ppp_voxel_grid");
  out.resize((size_t)m);
  for (int64_t r = 0; r < m; r++) {
    float sum[4] = {0.f, 0.f, 0.f, 0.f};   // bytes b, g, r, a of the rgba word
    for (int64_t j = off[(size_t)r]; j < off[(size_t)r + 1]; j++) {
      const uint32_t w = cloud.points[(size_t)members[(size_t)j]].rgba;
      for (int c = 0; c < 4; c++) sum[c] += (float)((w >> (8 * c)) & 0xFFu);
    }
    const float cnt = (float)(off[(size_t)r + 1] - off[(size_t)r]);
    uint32_t w = 0;
    for (int c = 0; c < 4; c++) w |= ((uint32_t)(sum[c] / cnt) & 0xFFu) << (8 * c);
    out[(size_t)r].rgba = w;
  }
  cloud.points.swap(out);
  cloud.width = (uint32_t)m; cloud.height = 1;
  return true;
}

inline MAP to_map(const Contours& c, int s) {
  MAP m;
  for (int64_t i = c.offsets[s]; i < c.offsets[s + 1]; i++) m[c.y[i]] = {c.x[i], c.z[i]};
  return m;
}

}  // namespace ppp_host

// -------------------------------------------------------------------------------------------------
class path_generater {
public:
  path_generater() {}
  path_generater(std::string cloud_name, double Radius) : toolRadius(Radius), file_name(cloud_name) {
    cloud = std::make_shared<PointCloudType>();
    cloud_with_normals = std::make_shared<pcl::PointCloud<pcl::Normal>>();
    if (ppp_host::loadPCDFile(cloud_name, *cloud) == -1) {
      fprintf(stderr, "Cloudn't read file!\n");  // the reference prints PCL_ERROR and carries on
    } else {
      Path_set = {};
      for (size_t i = 0; i < cloud->points.size(); i++) {  // src/Path_Generation.cpp:23-31
        cloud->points[i].r = (uint8_t)255;
        cloud->points[i].g = (uint8_t)255;
        cloud->points[i].b = (uint8_t)255;
        cloud->points[i].x *= 1000;
        cloud->points[i].y *= 1000;
        cloud->points[i].z *= 1000;
      }
    }
  }

  void Set_kdtree() { dev_.get(*cloud); }  // kdtree.setInputCloud(cloud)

  void smooth() {  // src/Path_Generation.cpp:340-360
    ppp_host::mls_smooth(dev_.get(*cloud), *cloud, file_name);
    dev_.invalidate();
  }

  // src/Path_Generation.cpp:53-59: VoxelGrid::setLeafSize(lx, ly, lz); filter(*cloud).  The reference's leaf size is
  // not part of this repository, so it is an argument here.
  void voxel_down(float lx, float ly, float lz) {
    if (ppp_host::voxel_down(dev_.get(*cloud), *cloud, lx, ly, lz)) dev_.invalidate();
  }

  void estimate_normal() {  // NormalEstimation, setRadiusSearch(2.5), viewpoint (0,0,0)
    const float vp[3] = {0, 0, 0};
    cloud_with_normals->points.resize(cloud->points.size());
    cloud_with_normals->width = (uint32_t)cloud->points.size();
    ppp_host::check(ppp_normals_radius(dev_.get(*cloud), 2.5, vp, PPP_COV_PCL110, cloud_with_normals->points.data(), sizeof(pcl::Normal)),
                    "ppp_normals_radius");
  }

  std::vector<int> rangedX_index(int position) {  // PassThrough "x", [-2 + position, 2 + position]
    return ppp_host::ranged_x_index(dev_.get(*cloud), position);
  }

  MAP insert_point(std::vector<int> indices, Eigen::Vector3f PlanePoint) {
    return ppp_host::insert_point(dev_.get(*cloud), indices, PlanePoint[0], PPP_PAIR_GEN2);
  }

  void slicing_method() {  // src/Path_Generation.cpp:282-321: all planes of the sweep in ONE device pass
    auto t0 = std::chrono::steady_clock::now();
    float mn[3], mx[3];
    ppp_host::check(ppp_cloud_bbox(dev_.get(*cloud), mn, mx), "ppp_cloud_bbox");  // getMinMax3D
    int step_size = (int)(toolRadius * 2);
    std::vector<float> planes;
    float x = mn[0];
    x += step_size / 2;
    while (x < mx[0] && step_size > 0) { planes.push_back(x); x += step_size; }
    last_ = ppp_host::slice_contours(dev_.get(*cloud), planes, PPP_PAIR_GEN2);
    long us = (long)std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
    printf("use time: %ld\nnumber of paths: %d\n", us, (int)planes.size());
    append_csv(us);
  }

  // Plane sweep + path_track of src/Path_Generation.cpp:689-755.  The per-slice dynamic adjustment
  // (compute_boundary / dynamic_adjust_path / drawpath) is sequential host logic outside the hot
  // path and stays with the reference; the ordered nodes it consumes are in Path_set.
  void Contact_Path_Generation() {
    printf("Start Path Planning!\n");
    auto t0 = std::chrono::steady_clock::now();
    float mn[3], mx[3];
    ppp_host::check(ppp_cloud_bbox(dev_.get(*cloud), mn, mx), "ppp_cloud_bbox");
    int step_size = (int)(toolRadius * 2);
    std::vector<float> planes;
    float locateX = mn[0] + toolRadius;
    while (locateX < mx[0] && step_size > 0) { planes.push_back(locateX); locateX += step_size; }
    last_ = ppp_host::slice_contours(dev_.get(*cloud), planes, PPP_PAIR_GEN2);
    Path_set.clear();
    for (size_t s = 0; s < planes.size(); s++) Path_set.push_back(last_.path((int)s));
    long us = (long)std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
    printf("Toal Using Time: %ld\nNumber of paths: %d\n", us, (int)planes.size());
    append_csv(us);
  }

  void invalidate_device_copy() { dev_.invalidate(); }
  const std::vector<Spline>& paths() const { return Path_set; }
  const ppp_host::Contours& last_contours() const { return last_; }
  pcl::PointCloud<pcl::PointXYZRGB>::Ptr cloud;
  pcl::PointCloud<pcl::Normal>::Ptr cloud_with_normals;

private:
  void append_csv(long us) {
    std::ofstream f("output.csv", std::ios::app);
    if (f.is_open()) f << us << std::endl;
  }
  ppp_host::DeviceCloud dev_;
  ppp_host::Contours last_;
  double toolRadius = 15;
  std::vector<Spline> Path_set;
  std::string file_name;
};

// -------------------------------------------------------------------------------------------------
class SectPath {
public:
  SectPath() {}
  SectPath(std::string configName, std::string CloudFileName) : cloud_name(CloudFileName) {
    read_config(configName);
    cloud = std::make_shared<PointCloudType>();
    normal_cloud = std::make_shared<pcl::PointCloud<pcl::Normal>>();
    if (ppp_host::loadPCDFile(cloud_name, *cloud) == -1) {
      fprintf(stderr, "Cloudn't read file!\n");
    } else {
      for (size_t i = 0; i < cloud->points.size(); ++i) {  // src/contour_alg.cpp:14-24
        cloud->points[i].r = cloud->points[i].g = cloud->points[i].b = (uint8_t)255;
        if (ifChangeRange) { cloud->points[i].x *= 1000; cloud->points[i].y *= 1000; cloud->points[i].z *= 1000; }
      }
    }
    // src/contour_alg.cpp:27-29.  trans2center (PCA alignment) is outside the accelerated path (DESIGN.md, out of
    // scope): say so instead of silently skipping it.
    if (ifSmooth) smooth();
    if (ifAlign) fprintf(stderr, "SectPath: Alignment=true is not available in this build (trans2center is out of scope)\n");
    if (ifRemove && cloud->points.size() > 50) remove_outlier();
  }
  virtual ~SectPath() {}

  void smooth() {  // the MLS pre-filter shared with path_generater::smooth()
    ppp_host::mls_smooth(dev_.get(*cloud), *cloud, cloud_name);
    dev_.invalidate();
  }

  void estimate_normal() {
    const float vp[3] = {0, 0, 0};
    normal_cloud->points.resize(cloud->points.size());
    ppp_host::check(ppp_normals_radius(dev_.get(*cloud), 2.5, vp, PPP_COV_PCL110, normal_cloud->points.data(), sizeof(pcl::Normal)),
                    "ppp_normals_radius");
  }

  // src/contour_alg.cpp:101-108: StatisticalOutlierRemoval, setMeanK(50), setStddevMulThresh(1.0),
  // filter(*cloud).  The kNN pass runs on the device; the statistics are the reference's scalar loop.
  void remove_outlier() {
    const int mean_k = 50;
    const double std_mul = 1.0;
    std::vector<float> distances(cloud->points.size());
    int64_t valid_distances = 0;
    ppp_host::check(ppp_sor_mean_distances(dev_.get(*cloud), mean_k, 0, distances.data(), &valid_distances),
                    "ppp_sor_mean_distances");
    double sum = 0, sq_sum = 0;
    for (const float& distance : distances) {
      sum += distance;
      sq_sum += distance * distance;
    }
    double mean = sum / static_cast<double>(valid_distances);
    double variance = (sq_sum - sum * sum / static_cast<double>(valid_distances)) / (static_cast<double>(valid_distances) - 1);
    double distance_threshold = mean + std_mul * std::sqrt(variance);
    size_t o = 0;
    for (size_t i = 0; i < distances.size(); i++)
      if (!(distances[i] > distance_threshold)) cloud->points[o++] = cloud->points[i];
    cloud->points.resize(o);
    cloud->width = (uint32_t)o; cloud->height = 1;
    dev_.invalidate();
  }

  virtual void GenPath() {  // src/contour_alg.cpp:287-339: centre-out sweep, all planes in one pass
    printf("Start Path Planning!\n");
    auto t0 = std::chrono::high_resolution_clock::now();
    float mn[3], mx[3];
    ppp_host::check(ppp_cloud_bbox(dev_.get(*cloud), mn, mx), "ppp_cloud_bbox");
    int step_size = (int)(toolRadius * 2);
    std::vector<float> front, back;
    float loc = (mn[0] + mx[0]) / 2 - step_size;
    while (loc > mn[0] && step_size > 0) { front.insert(front.begin(), loc); loc -= step_size; }
    loc = (mn[0] + mx[0]) / 2;
    while (loc < mx[0] && step_size > 0) { back.push_back(loc); loc += step_size; }
    std::vector<float> planes(front);
    planes.insert(planes.end(), back.begin(), back.end());
    last_ = ppp_host::slice_contours(dev_.get(*cloud), planes, PPP_PAIR_SECT);
    Path_set.clear();
    for (size_t s = 0; s < planes.size(); s++) Path_set.push_back(last_.path((int)s));
    double ms = std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::high_resolution_clock::now() - t0).count() * 0.001;
    printf("Toal Using Time: %lf (ms)\nNumber of paths: %d\nNumber of Point Cloud: %ld\n", ms, (int)planes.size(), (long)cloud->size());
  }

  const std::vector<Spline>& paths() const { return Path_set; }
  const ppp_host::Contours& last_contours() const { return last_; }
  PointCloudType::Ptr cloud;
  pcl::PointCloud<pcl::Normal>::Ptr normal_cloud;

protected:
  // key = value, '#' comments, all whitespace stripped (src/contour_alg.cpp:32-67)
  virtual void read_config(std::string filename) {
    std::ifstream f(filename);
    std::string line;
    while (std::getline(f, line)) {
      std::string s;
      for (char ch : line) if (ch != ' ' && ch != '\t' && ch != '\r') s += ch;
      if (s.empty() || s[0] == '#') continue;
      size_t p = s.find('=');
      if (p == std::string::npos) continue;
      std::string key = s.substr(0, p), val = s.substr(p + 1);
      if (key == "Tool_Radius") toolRadius = atof(val.c_str());
      else if (key == "PathResolution") PathResolution = atof(val.c_str());
      else if (key == "RPYresolution") RPYres = atof(val.c_str());
      else if (key == "Endeffectorlength") EElen = (float)atof(val.c_str());
      else if (key == "pathFile") pathFile = val;
      else if (key == "Smooth") ifSmooth = (val == "true");
      else if (key == "Alignment") ifAlign = (val == "true");
      else if (key == "ChangeRange") ifChangeRange = (val == "true");
      else if (key == "RemoveOutlier") ifRemove = (val == "true");
    }
  }

  std::vector<int> rangedX_index(int position) {
    return ppp_host::ranged_x_index(dev_.get(*cloud), position);
  }
  MAP insert_point(std::vector<int> indices, Eigen::Vector3f PlanePoint) {
    return ppp_host::insert_point(dev_.get(*cloud), indices, PlanePoint[0], PPP_PAIR_SECT);
  }
  Spline OnePath(Eigen::Vector3f plane_point) {
    return ppp_host::slice_contours(dev_.get(*cloud), {plane_point[0]}, PPP_PAIR_SECT).path(0);
  }

  ppp_host::DeviceCloud dev_;
  ppp_host::Contours last_;
  double toolRadius = 12, PathResolution = 0, RPYres = 0;
  float EElen = 0;
  bool ifAlign = false, ifSmooth = false, ifChangeRange = true, ifRemove = false;
  std::vector<Spline> Path_set;
  std::string cloud_name, pathFile;
};
