// VoxelGrid downsampling: pcl::VoxelGrid<PointXYZRGB>::applyFilter as the reference's voxel_down() runs it
// (src/Path_Generation.cpp:53-59; min_points_per_voxel 0, downsample_all_data true).  [upstream, recalled:
// PCL 1.10.0 VoxelGrid::applyFilter, CentroidPoint / AccumulatorXYZ.]
//
//   key pass:   per finite point, ijk = (int)(floorf(p * inv) - (float)min_b) and the voxel key
//               idx = ijk . (1, div_b.x, div_b.x * div_b.y) in wrapping uint32 arithmetic (PCL computes it in int
//               and stores it as unsigned int); non-finite points are marked and dropped by the first sort pass;
//   sort:       stable LSD radix sort of (key, point index) over the bits the largest possible key needs, 8 bits a
//               pass; the digit offsets of every (digit, warp segment) come from scan_exclusive_i32; the scatter is
//               stable because each warp walks its segment in order, 32 items at a time, ranking equal digits with
//               __match_any_sync.  The input is in ascending point order, so every voxel's members end up in
//               ascending source index;
//   segments:   boundary flags -> scan -> voxel ordinals -> row offsets;
//   centroid:   per voxel, a sequential float32 sum of x, y, z (and of the rgba bytes of the source records, when
//               given) in member order, then a division by (float)count (the library is built with --fmad=false, and
//               the adds and the divisions are explicitly rounded), written as a whole record of the caller's stride.
// PCL sums in the order its unstable std::sort leaves each voxel, which only differs in the last bits of the
// centroids: the tolerance contract is in include/ppp_gpu.h (ppp_voxel_grid) and DESIGN.md §2.
#include <algorithm>
#include <cmath>

#include "ppp_device.cuh"

namespace {

constexpr int VX_WARPS = 8;               // warps per block of the sort kernels
constexpr int VX_SEG = 32 * 32;           // items per warp segment (the unit of the digit histogram)
constexpr int VX_DIGIT_BITS = 8;
constexpr int VX_DIGITS = 1 << VX_DIGIT_BITS;

struct VoxelKeyParams {
  float inv[3];      // 1.0f / leaf
  float minb_f[3];   // (float)min_b
  uint32_t mul1, mul2;   // div_b.x, div_b.x * div_b.y (wrapping)
};

__global__ void __launch_bounds__(256) k_voxel_keys(const float4* __restrict__ xyz4, int64_t n, VoxelKeyParams p,
                                                    uint32_t* __restrict__ keys, int32_t* __restrict__ vals) {
  pdl_prologue();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 q = xyz4[i];
  if (!(q.w == 0.0f)) {   // w is NaN for a non-finite point
    keys[i] = 0u;
    vals[i] = -1;
    return;
  }
  const int i0 = (int)__fsub_rn(floorf(__fmul_rn(q.x, p.inv[0])), p.minb_f[0]);
  const int i1 = (int)__fsub_rn(floorf(__fmul_rn(q.y, p.inv[1])), p.minb_f[1]);
  const int i2 = (int)__fsub_rn(floorf(__fmul_rn(q.z, p.inv[2])), p.minb_f[2]);
  keys[i] = (uint32_t)i0 + (uint32_t)i1 * p.mul1 + (uint32_t)i2 * p.mul2;
  vals[i] = (int32_t)i;
}

// counts[d * n_seg + s] = items of warp segment s whose digit is d (items with a negative value are not counted).
__global__ void __launch_bounds__(VX_WARPS * 32) k_voxel_hist(const uint32_t* __restrict__ keys, const int32_t* __restrict__ vals,
                                                             int64_t n, int shift, int digits, int n_seg,
                                                             int32_t* __restrict__ counts) {
  pdl_prologue();
  __shared__ int32_t h[VX_WARPS][VX_DIGITS];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int seg = blockIdx.x * VX_WARPS + w;
  if (seg >= n_seg) return;
  for (int d = lane; d < digits; d += 32) h[w][d] = 0;
  __syncwarp();
  const int64_t a = (int64_t)seg * VX_SEG, b = n < a + VX_SEG ? n : a + VX_SEG;
  const uint32_t mask = (uint32_t)digits - 1u;
  for (int64_t i = a + lane; i < b; i += 32)
    if (vals[i] >= 0) atomicAdd(&h[w][(keys[i] >> shift) & mask], 1);
  __syncwarp();
  for (int d = lane; d < digits; d += 32) counts[(int64_t)d * n_seg + seg] = h[w][d];
}

// Stable scatter: item j of warp segment s with digit d goes to offsets[d * n_seg + s] + (earlier items of the
// segment with digit d).  Items with a negative value are dropped.
__global__ void __launch_bounds__(VX_WARPS * 32) k_voxel_scatter(const uint32_t* __restrict__ keys, const int32_t* __restrict__ vals,
                                                                int64_t n, int shift, int digits, int n_seg,
                                                                const int32_t* __restrict__ offsets, int64_t m,
                                                                uint32_t* __restrict__ keys_out, int32_t* __restrict__ vals_out) {
  pdl_prologue();
  __shared__ int32_t base[VX_WARPS][VX_DIGITS];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int seg = blockIdx.x * VX_WARPS + w;
  if (seg >= n_seg) return;
  for (int d = lane; d < digits; d += 32) base[w][d] = offsets[(int64_t)d * n_seg + seg];
  __syncwarp();
  const int64_t a = (int64_t)seg * VX_SEG, b = n < a + VX_SEG ? n : a + VX_SEG;
  const uint32_t mask = (uint32_t)digits - 1u;
  const unsigned lt = (1u << lane) - 1u;
  for (int64_t i0 = a; i0 < b; i0 += 32) {
    const int64_t i = i0 + lane;
    uint32_t k = 0u;
    int32_t v = -1;
    if (i < b) { k = keys[i]; v = vals[i]; }
    const uint32_t d = v >= 0 ? (k >> shift) & mask : (uint32_t)VX_DIGITS;   // dropped items form their own group
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const int rank = __popc(peers & lt);
    int32_t pos = 0;
    if (v >= 0) pos = base[w][d] + rank;
    __syncwarp();
    if (v >= 0 && rank == 0) base[w][d] += __popc(peers);
    __syncwarp();
    if (v >= 0) {
      PPP_DEV_ASSERT(pos >= 0 && pos < m);
      keys_out[pos] = k;
      vals_out[pos] = v;
    }
  }
}

__global__ void __launch_bounds__(256) k_voxel_flags(const uint32_t* __restrict__ keys, int64_t m, int32_t* __restrict__ flags) {
  pdl_prologue();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) flags[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1 : 0;
}

// row_off[ord[i]] = i at every first member of a voxel; row_off[rows] = m.
__global__ void __launch_bounds__(256) k_voxel_offsets(const int32_t* __restrict__ flags, const int32_t* __restrict__ ord,
                                                       int64_t m, int64_t* __restrict__ row_off) {
  pdl_prologue();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m && flags[i]) {
    PPP_DEV_ASSERT(ord[i] >= 0 && ord[i] < m);
    row_off[ord[i]] = i;
  }
  if (i == 0) row_off[ord[m]] = m;
}

// One thread per voxel: a CentroidPoint record of sf words (row r at out + r * sf).  x, y, z: AccumulatorXYZ, a float32
// sum in member order divided by (float)count; word 3 (sf >= 4): the pad float 1.0f of a default-constructed point;
// word 4 (sf >= 5), with source records src of sf words: AccumulatorRGBA over their word 4, per byte channel a float32
// sum in member order divided by the count and truncated; every other word 0.  vec: sf % 4 == 0 and out 16-byte
// aligned, so that whole records go out as 16-byte stores.  Records and members index the n points of the cloud.
// RGBA: src is not NULL (the colour sums live in registers only where they are needed).
template <bool RGBA>
__global__ void __launch_bounds__(256) k_voxel_centroid(const int64_t* __restrict__ row_off, const int32_t* __restrict__ rows_dev,
                                                        const int32_t* __restrict__ members, const float4* __restrict__ xyz4,
                                                        int64_t n, const uint32_t* __restrict__ src, int sf, bool vec,
                                                        float* __restrict__ out) {
  pdl_prologue();
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= *rows_dev) return;
  const int64_t a = row_off[r], b = row_off[r + 1];
  float sx = 0.f, sy = 0.f, sz = 0.f;
  float c0 = 0.f, c1 = 0.f, c2 = 0.f, c3 = 0.f;   // bytes 0..3 of the rgba word
  for (int64_t j = a; j < b; j++) {
    const int32_t i = members[j];
    PPP_DEV_ASSERT(i >= 0 && i < n);
    const float4 p = xyz4[i];
    sx = __fadd_rn(sx, p.x);
    sy = __fadd_rn(sy, p.y);
    sz = __fadd_rn(sz, p.z);
    if (RGBA) {
      const uint32_t w = src[(int64_t)i * sf + 4];
      c0 = __fadd_rn(c0, (float)(w & 0xffu));
      c1 = __fadd_rn(c1, (float)((w >> 8) & 0xffu));
      c2 = __fadd_rn(c2, (float)((w >> 16) & 0xffu));
      c3 = __fadd_rn(c3, (float)(w >> 24));
    }
  }
  const float cnt = (float)(b - a);
  const float x = __fdiv_rn(sx, cnt), y = __fdiv_rn(sy, cnt), z = __fdiv_rn(sz, cnt);
  uint32_t rgba = 0u;
  if (RGBA)   // past 2^24 a channel sum has rounded and its quotient can reach 256: only the low byte is kept
    rgba = (__float2uint_rz(__fdiv_rn(c0, cnt)) & 0xffu) | (__float2uint_rz(__fdiv_rn(c1, cnt)) & 0xffu) << 8 |
           (__float2uint_rz(__fdiv_rn(c2, cnt)) & 0xffu) << 16 | (__float2uint_rz(__fdiv_rn(c3, cnt)) & 0xffu) << 24;
  PPP_DEV_ASSERT(r < n);
  float* o = out + r * sf;
  if (vec) {
    float4* o4 = reinterpret_cast<float4*>(o);
    o4[0] = make_float4(x, y, z, 1.0f);
    for (int q = 1; q < sf / 4; q++) o4[q] = make_float4(q == 1 ? __uint_as_float(rgba) : 0.f, 0.f, 0.f, 0.f);
  } else {
    o[0] = x; o[1] = y; o[2] = z;
    if (sf > 3) o[3] = 1.0f;
    if (sf > 4) o[4] = __uint_as_float(rgba);
    for (int k = 5; k < sf; k++) o[k] = 0.f;
  }
}

inline unsigned blocks_for(int64_t n, int t) { return (unsigned)((n + t - 1) / t); }

}  // namespace

int voxel_grid_launch(ppp_cloud* c, const float leaf[3], const float* src, int sf, float* rows_dev, int64_t* row_off_dev,
                      int32_t* members_dev, int64_t* n_rows) {
  ppp_ctx* ctx = c->ctx;
  *n_rows = 0;
  const int64_t m = c->n_finite;
  if (m == 0) return PPP_OK;   // PCL leaves this case undefined (getMinMax3D of nothing): no rows
  // Host constants, in float32 exactly as applyFilter computes them.
  float inv[3];
  int64_t ext[3];
  int minb[3];
  int64_t divb[3];
  for (int d = 0; d < 3; d++) {
    inv[d] = 1.0f / leaf[d];
    const float e = (c->bmax[d] - c->bmin[d]) * inv[d];
    if (!(e < 2147483648.0f)) {   // includes a non-finite product: dx alone would exceed INT32_MAX
      ppp_set_error("ppp_voxel_grid: Leaf size is too small for the input dataset. Integer indices would overflow.");
      return PPP_ERR_UNSUPPORTED;
    }
    ext[d] = (int64_t)e + 1;
  }
  if (ext[0] * ext[1] > 2147483647ll || ext[0] * ext[1] * ext[2] > 2147483647ll) {
    ppp_set_error("ppp_voxel_grid: Leaf size is too small for the input dataset. Integer indices would overflow.");
    return PPP_ERR_UNSUPPORTED;
  }
  for (int d = 0; d < 3; d++) {
    const float lo = floorf(c->bmin[d] * inv[d]), hi = floorf(c->bmax[d] * inv[d]);
    // PCL casts these to int; beyond the int range that cast is undefined and so are its voxels
    if (!(lo >= -2147483648.0f && hi < 2147483648.0f)) {
      ppp_set_error("ppp_voxel_grid: coordinate / leaf size exceeds the int range of the voxel coordinates on axis %d", d);
      return PPP_ERR_UNSUPPORTED;
    }
    minb[d] = (int)lo;
    divb[d] = (int64_t)(int)hi - minb[d] + 1;
  }
  VoxelKeyParams kp;
  for (int d = 0; d < 3; d++) { kp.inv[d] = inv[d]; kp.minb_f[d] = (float)minb[d]; }
  kp.mul1 = (uint32_t)divb[0];
  kp.mul2 = (uint32_t)divb[0] * (uint32_t)divb[1];
  // Bits of the largest key: div_b can exceed (dx, dy, dz) by one voxel per axis, and past 2^32 keys wrap as PCL's do.
  const double kmax = (double)divb[0] * (double)divb[1] * (double)divb[2] - 1.0;
  int bits = 32;
  if (kmax < 4294967296.0) { bits = 0; while (bits < 32 && (uint64_t)kmax >> bits) bits++; }
  const int passes = std::max(1, (bits + VX_DIGIT_BITS - 1) / VX_DIGIT_BITS);   // pass 0 also drops non-finite points

  const int64_t n = c->n;
  uint32_t *keys[2] = {nullptr, nullptr};
  int32_t *vals_tmp = nullptr, *vals_mid = nullptr;
  int32_t *counts = nullptr, *offsets = nullptr, *flags = nullptr, *ord = nullptr;
  const int n_seg_max = (int)((n + VX_SEG - 1) / VX_SEG);
  PPP_TRY(dev_alloc(ctx, &keys[0], (size_t)n));
  PPP_TRY(dev_alloc(ctx, &keys[1], (size_t)n));
  PPP_TRY(dev_alloc(ctx, &vals_tmp, (size_t)n));
  if ((passes & 1) == 0) PPP_TRY(dev_alloc(ctx, &vals_mid, (size_t)m));
  PPP_TRY(dev_alloc(ctx, &counts, (size_t)VX_DIGITS * n_seg_max));
  PPP_TRY(dev_alloc(ctx, &offsets, (size_t)VX_DIGITS * n_seg_max + 1));
  PPP_TRY(dev_alloc(ctx, &flags, (size_t)m));
  PPP_TRY(dev_alloc(ctx, &ord, (size_t)m + 1));
  // stage s (0: key pass over the n points, p + 1: sort pass p over the m finite ones) writes keys[s & 1] and its values:
  // the key pass into vals_tmp (n entries), the last stage into members_dev (m entries, so the key pass never goes
  // there), the stages between alternately into vals_tmp and members_dev backwards from the last; where that would make
  // the first sort pass write its own input vals_tmp (an even number of passes), it writes vals_mid
  auto vals_of = [&](int s) {
    return s == 0 ? vals_tmp : ((passes - s) & 1) == 0 ? members_dev : s == 1 ? vals_mid : vals_tmp;
  };
  PPP_LAUNCH(ctx, "voxel_keys", k_voxel_keys, blocks_for(n, 256), 256, 0, (const float4*)c->xyz4, n, kp, keys[0], vals_of(0));
  PPP_CHECK_LAUNCH();
  for (int p = 0; p < passes; p++) {
    const int64_t len = p == 0 ? n : m;
    const int n_seg = (int)((len + VX_SEG - 1) / VX_SEG);
    const int shift = p * VX_DIGIT_BITS;
    const int digits = 1 << std::min(VX_DIGIT_BITS, std::max(1, bits - shift));
    const uint32_t* kin = keys[p & 1];
    const int32_t* vin = vals_of(p);
    PPP_LAUNCH(ctx, "voxel_hist", k_voxel_hist, blocks_for(n_seg, VX_WARPS), VX_WARPS * 32, 0, kin, vin, len, shift, digits, n_seg,
               counts);
    PPP_CHECK_LAUNCH();
    PPP_TRY(scan_exclusive_i32(ctx, counts, offsets, (int64_t)digits * n_seg));
    PPP_LAUNCH(ctx, "voxel_scatter", k_voxel_scatter, blocks_for(n_seg, VX_WARPS), VX_WARPS * 32, 0, kin, vin, len, shift, digits,
               n_seg, (const int32_t*)offsets, m, keys[(p + 1) & 1], vals_of(p + 1));
    PPP_CHECK_LAUNCH();
  }
  const uint32_t* ksorted = keys[passes & 1];
  PPP_LAUNCH(ctx, "voxel_flags", k_voxel_flags, blocks_for(m, 256), 256, 0, ksorted, m, flags);
  PPP_CHECK_LAUNCH();
  PPP_TRY(scan_exclusive_i32(ctx, flags, ord, m));
  PPP_LAUNCH(ctx, "voxel_offsets", k_voxel_offsets, blocks_for(m, 256), 256, 0, (const int32_t*)flags, (const int32_t*)ord, m,
             row_off_dev);
  PPP_CHECK_LAUNCH();
  const bool vec = sf % 4 == 0 && (uintptr_t)rows_dev % 16 == 0;
  auto* centroid = src ? k_voxel_centroid<true> : k_voxel_centroid<false>;
  PPP_LAUNCH(ctx, "voxel_centroid", centroid, blocks_for(m, 256), 256, 0, (const int64_t*)row_off_dev,
             (const int32_t*)(ord + m), (const int32_t*)members_dev, (const float4*)c->xyz4, n, (const uint32_t*)src, sf, vec,
             rows_dev);
  PPP_CHECK_LAUNCH();
  int32_t rows = 0;
  PPP_CUDA(cudaMemcpyAsync(&rows, ord + m, 4, cudaMemcpyDeviceToHost, ctx->stream));
  PPP_CUDA(cudaStreamSynchronize(ctx->stream));
  dev_free(ctx, keys[0]); dev_free(ctx, keys[1]); dev_free(ctx, vals_tmp); dev_free(ctx, vals_mid);
  dev_free(ctx, counts); dev_free(ctx, offsets); dev_free(ctx, flags); dev_free(ctx, ord);
  *n_rows = rows;
  return PPP_OK;
}
