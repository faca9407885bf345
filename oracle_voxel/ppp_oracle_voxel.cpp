// ppp_oracle_voxel.cpp — CPU ORACLE for the VoxelGrid pre-filter. TEST INFRASTRUCTURE ONLY.
//
// voxel_down() of the reference (src/Path_Generation.cpp:53-59): pcl::VoxelGrid<PointXYZRGB>::applyFilter with
// PCL 1.10 defaults (min_points_per_voxel 0, downsample_all_data true), restated statement by statement:
// [upstream, recalled] getMinMax3D over the finite points, the int64 overflow check, min_b / max_b / div_b /
// divb_mul, the per-point voxel index in float32 and int, std::sort of cloud_point_index_idx by idx only, the
// run-length pass, and CentroidPoint (AccumulatorXYZ: float sums divided by the count; AccumulatorRGBA: per-channel
// float sums, each divided by the count and truncated).  No FMA contraction (Makefile).
//
// order 0 sorts with libstdc++'s std::sort and PCL's comparator, on the same vector PCL builds (finite points in
// ascending index): the order PCL sums each voxel in.  order 1 uses std::stable_sort: ascending source index
// inside each voxel, the order of the device.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <vector>

namespace {

struct cloud_point_index_idx {   // pcl::cloud_point_index_idx
  unsigned int idx;
  unsigned int cloud_point_index;
  bool operator<(const cloud_point_index_idx& p) const { return idx < p.idx; }
};

inline bool finite3(const float* p) { return std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2]); }

}  // namespace

extern "C" {

// pts: n records of sf floats (x, y, z first; with sf >= 5, float 4 holds the rgba bits).  Output, room for n rows:
// out (rows x sf floats: centroid x, y, z, pad 1.0f, averaged rgba where sf >= 5, zeros elsewhere), row_off (rows + 1),
// members (one per finite point: source indices grouped by row, in the summation order).  Returns the row count,
// -1 for an invalid leaf, -2 where PCL warns and keeps the input (index overflow), -3 where floorf(bbox * inv) leaves
// the int range.
int64_t ppo_voxel_grid(const float* pts, int64_t n, int64_t sf, const float leaf[3], float* out, int64_t* row_off,
                       int32_t* members, int order) {
  float inv[3];
  for (int d = 0; d < 3; d++) {
    if (!(leaf[d] > 0) || !std::isfinite(leaf[d])) return -1;
    inv[d] = 1.0f / leaf[d];   // setLeafSize: inverse_leaf_size_ = Array4f::Ones() / leaf_size_
    if (!std::isfinite(inv[d])) return -1;
  }
  // getMinMax3D (non-dense cloud: finite points only)
  float mn[3] = {std::numeric_limits<float>::max(), std::numeric_limits<float>::max(), std::numeric_limits<float>::max()};
  float mx[3] = {-std::numeric_limits<float>::max(), -std::numeric_limits<float>::max(), -std::numeric_limits<float>::max()};
  int64_t n_finite = 0;
  for (int64_t i = 0; i < n; i++) {
    const float* p = pts + i * sf;
    if (!finite3(p)) continue;
    n_finite++;
    for (int d = 0; d < 3; d++) { mn[d] = std::min(mn[d], p[d]); mx[d] = std::max(mx[d], p[d]); }
  }
  row_off[0] = 0;
  if (n_finite == 0) return 0;
  int64_t dxyz[3];
  for (int d = 0; d < 3; d++) {
    const float e = (mx[d] - mn[d]) * inv[d];
    if (!(e < 9.2e18f)) return -2;   // the int64 cast below is defined up to here; PCL's product is then far too big
    dxyz[d] = static_cast<int64_t>(e) + 1;
  }
  // dx * dy * dz > INT32_MAX (each factor fits 2^63, so check the partial product first)
  if (dxyz[0] > INT32_MAX || dxyz[1] > INT32_MAX || dxyz[2] > INT32_MAX || dxyz[0] * dxyz[1] > INT32_MAX ||
      dxyz[0] * dxyz[1] * dxyz[2] > INT32_MAX)
    return -2;
  int min_b[3], max_b[3], div_b[3];
  for (int d = 0; d < 3; d++) {
    const float lo = std::floor(mn[d] * inv[d]), hi = std::floor(mx[d] * inv[d]);
    if (!(lo >= -2147483648.0f && hi < 2147483648.0f)) return -3;
    min_b[d] = static_cast<int>(lo);
    max_b[d] = static_cast<int>(hi);
    div_b[d] = (int)((unsigned)max_b[d] - (unsigned)min_b[d] + 1u);   // int arithmetic, wrapping as on the CPU
  }
  const unsigned divb_mul[3] = {1u, (unsigned)div_b[0], (unsigned)div_b[0] * (unsigned)div_b[1]};
  std::vector<cloud_point_index_idx> index_vector;
  index_vector.reserve((size_t)n_finite);
  for (int64_t i = 0; i < n; i++) {
    const float* p = pts + i * sf;
    if (!finite3(p)) continue;
    unsigned ijk[3];
    for (int d = 0; d < 3; d++)
      ijk[d] = (unsigned)static_cast<int>(std::floor(p[d] * inv[d]) - static_cast<float>(min_b[d]));
    const unsigned idx = ijk[0] * divb_mul[0] + ijk[1] * divb_mul[1] + ijk[2] * divb_mul[2];
    index_vector.push_back({idx, (unsigned)i});
  }
  if (order == 0) std::sort(index_vector.begin(), index_vector.end(), std::less<cloud_point_index_idx>());
  else std::stable_sort(index_vector.begin(), index_vector.end(), std::less<cloud_point_index_idx>());
  int64_t rows = 0;
  size_t index = 0;
  while (index < index_vector.size()) {
    size_t i = index + 1;
    while (i < index_vector.size() && index_vector[i].idx == index_vector[index].idx) ++i;
    // CentroidPoint::add / get for PointXYZRGB
    float xyz[3] = {0.f, 0.f, 0.f};
    float rgba[4] = {0.f, 0.f, 0.f, 0.f};   // b, g, r, a (bytes 0..3 of the rgba word)
    for (size_t li = index; li < i; ++li) {
      const float* p = pts + (int64_t)index_vector[li].cloud_point_index * sf;
      for (int d = 0; d < 3; d++) xyz[d] += p[d];
      if (sf >= 5) {
        uint32_t w;
        std::memcpy(&w, p + 4, 4);
        for (int c = 0; c < 4; c++) rgba[c] += (float)((w >> (8 * c)) & 0xFFu);
      }
      members[li] = (int32_t)index_vector[li].cloud_point_index;
    }
    const size_t cnt = i - index;
    float* o = out + rows * sf;
    for (int64_t k = 0; k < sf; k++) o[k] = 0.f;
    for (int d = 0; d < 3; d++) o[d] = xyz[d] / static_cast<float>(cnt);
    if (sf >= 4) o[3] = 1.0f;
    if (sf >= 5) {
      uint32_t w = 0;
      for (int c = 0; c < 4; c++) w |= (static_cast<uint32_t>(rgba[c] / static_cast<float>(cnt)) & 0xFFu) << (8 * c);
      std::memcpy(o + 4, &w, 4);
    }
    rows++;
    row_off[rows] = (int64_t)i;
    index = i;
  }
  return rows;
}

}  // extern "C"
