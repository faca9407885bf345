// Minimal PCD reader (ascii / binary, float x y z [rgb|rgba]) and writer (binary, FIELDS x y z rgb) standing in
// for pcl::io::loadPCDFile / savePCDFile<pcl::PointXYZRGB> (src/Path_Generation.cpp:8,340-360) when PCL is absent.
#pragma once
#include <cstdio>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>
#include <vector>

#include "pcl_min.h"

namespace ppp_host {
// returns 0 on success, -1 on failure (like pcl::io::loadPCDFile)
inline int loadPCDFile(const std::string& path, pcl::PointCloud<pcl::PointXYZRGB>& cloud) {
  std::ifstream f(path, std::ios::binary);
  if (!f) return -1;
  std::vector<std::string> fields;
  std::vector<int> sizes, counts;
  std::vector<char> types;
  long npts = -1;
  std::string data_kind, line;
  while (std::getline(f, line)) {
    if (line.empty() || line[0] == '#') continue;
    std::istringstream ss(line);
    std::string key;
    ss >> key;
    if (key == "FIELDS") { std::string s; while (ss >> s) fields.push_back(s); }
    else if (key == "SIZE") { int v; while (ss >> v) sizes.push_back(v); }
    else if (key == "TYPE") { char c; while (ss >> c) types.push_back(c); }
    else if (key == "COUNT") { int v; while (ss >> v) counts.push_back(v); }
    else if (key == "POINTS") ss >> npts;
    else if (key == "DATA") { ss >> data_kind; break; }
  }
  if (npts < 0 || fields.empty() || sizes.size() != fields.size()) return -1;
  if (counts.empty()) counts.assign(fields.size(), 1);
  int off_x = -1, off_y = -1, off_z = -1, off_rgb = -1, rec = 0, col_x = -1, col_y = -1, col_z = -1, col_rgb = -1, col = 0;
  for (size_t i = 0; i < fields.size(); i++) {
    if (fields[i] == "x") { off_x = rec; col_x = col; }
    else if (fields[i] == "y") { off_y = rec; col_y = col; }
    else if (fields[i] == "z") { off_z = rec; col_z = col; }
    else if (fields[i] == "rgb" || fields[i] == "rgba") { off_rgb = rec; col_rgb = col; }
    rec += sizes[i] * counts[i];
    col += counts[i];
  }
  if (off_x < 0 || off_y < 0 || off_z < 0) return -1;
  cloud.points.assign((size_t)npts, pcl::PointXYZRGB());
  cloud.width = (uint32_t)npts; cloud.height = 1; cloud.is_dense = true;
  if (data_kind == "binary") {
    std::vector<char> buf((size_t)rec);
    for (long i = 0; i < npts; i++) {
      if (!f.read(buf.data(), rec)) return -1;
      pcl::PointXYZRGB& p = cloud.points[(size_t)i];
      memcpy(&p.x, &buf[off_x], 4); memcpy(&p.y, &buf[off_y], 4); memcpy(&p.z, &buf[off_z], 4);
      if (off_rgb >= 0) memcpy(&p.rgba, &buf[off_rgb], 4);
    }
  } else if (data_kind == "ascii") {
    for (long i = 0; i < npts; i++) {
      if (!std::getline(f, line)) return -1;
      std::istringstream ss(line);
      std::vector<double> v;
      double d;
      while (ss >> d) v.push_back(d);
      if ((int)v.size() < col) return -1;
      pcl::PointXYZRGB& p = cloud.points[(size_t)i];
      p.x = (float)v[col_x]; p.y = (float)v[col_y]; p.z = (float)v[col_z];
      if (col_rgb >= 0) p.rgb = (float)v[col_rgb];
    }
  } else {
    return -1;
  }
  return 0;
}

// binary PCD v0.7, FIELDS x y z rgb (the layout polishpathplanning_b200.synth.write_pcd writes); 0 / -1
inline int savePCDFile(const std::string& path, const pcl::PointCloud<pcl::PointXYZRGB>& cloud) {
  std::ofstream f(path, std::ios::binary);
  if (!f) return -1;
  const size_t n = cloud.points.size();
  f << "# .PCD v0.7 - Point Cloud Data file format\nVERSION 0.7\nFIELDS x y z rgb\nSIZE 4 4 4 4\nTYPE F F F F\n"
       "COUNT 1 1 1 1\nWIDTH " << n << "\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS " << n << "\nDATA binary\n";
  for (const pcl::PointXYZRGB& p : cloud.points) {
    float rec[4] = {p.x, p.y, p.z, 0.0f};
    memcpy(&rec[3], &p.rgba, 4);
    f.write(reinterpret_cast<const char*>(rec), sizeof(rec));
  }
  return f ? 0 : -1;
}
}  // namespace ppp_host
