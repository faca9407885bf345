// Cloud ingest (pack + bounding box = getMinMax3D) and the column-grid spatial index that
// replaces pcl::KdTreeFLANN::setInputCloud (src/Path_Generation.cpp:335-338,695;
// src/contour_alg.cpp:292) and NormalEstimation's private search::KdTree (:326-327).
//
// Index = counting sort of the finite points by cell id (v*nu + u) over a dense cell table:
// histogram (atomics) -> exclusive scan -> scatter.  Rows of cells are contiguous in the sorted
// array, so a query's candidates are (2R+1) contiguous ranges that consecutive (sorted) queries
// share: coalesced float4 loads, L1/L2 reuse, no tree walk.
#include <stdlib.h>

#include <algorithm>
#include <cmath>

#include "ppp_device.cuh"

namespace {

__device__ __forceinline__ uint32_t f2ord(float f) {
  uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
inline float ord2f(uint32_t u) {
  uint32_t b = (u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u;
  float f;
  memcpy(&f, &b, 4);
  return f;
}

// Subsample of the density estimate: every 2^shift-th point, 8192 .. 16383 of them (all points of a smaller cloud).
__host__ __device__ inline int ds_sub_shift(long long n) {
  int sh = 0;
  while ((n >> sh) >= 16384) sh++;
  return sh;
}

struct BBoxAcc {
  uint32_t mn[3];
  uint32_t mx[3];
  unsigned long long n_finite;
};

// first use of a context's ingest scratch (later ingests find it reset by k_density_sample's last block);
// acc is the first member of IngestScratch, the ticket follows it
__global__ void k_bbox_init(BBoxAcc* acc) {
  pdl_prologue();
  for (int d = 0; d < 3; d++) { acc->mn[d] = 0xFFFFFFFFu; acc->mx[d] = 0u; }
  acc->n_finite = 0ull;
  *(unsigned*)(acc + 1) = 0u;
}

// Pack stride-`sf` records to float4 (original order) and reduce the bounding box of the finite
// points.  One pass over the raw cloud: 12 useful bytes of each record in, 16 out.
__global__ void __launch_bounds__(256) k_pack_bbox(const float* __restrict__ raw, int64_t n, int sf, int vec_ok,
                                                   float4* __restrict__ xyz4, BBoxAcc* __restrict__ acc,
                                                   float4* __restrict__ sub, int sub_shift,
                                                   const long long* __restrict__ n_dev) {
  pdl_prologue();
  if (n_dev) {   // the point count is only known on the device (a slab the exchange has just received)
    n = *n_dev;
    sub_shift = ds_sub_shift(n);
  }
  const int64_t sub_mask = ((int64_t)1 << sub_shift) - 1;   // every 2^sub_shift-th point also goes to the compact subsample
  float mn[3] = {CUDART_INF_F, CUDART_INF_F, CUDART_INF_F};
  float mx[3] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
  unsigned cnt = 0;
  constexpr int PPT = 4;  // points per thread per sweep: PPT independent loads in flight
  for (int64_t base = (int64_t)blockIdx.x * blockDim.x * PPT; base < n; base += (int64_t)gridDim.x * blockDim.x * PPT) {
    float x[PPT], y[PPT], z[PPT];
#pragma unroll
    for (int j = 0; j < PPT; j++) {
      int64_t i = base + (int64_t)j * blockDim.x + threadIdx.x;
      x[j] = y[j] = z[j] = 0.f;
      if (i < n) {
        if (vec_ok) {
          float4 p = __ldg(reinterpret_cast<const float4*>(raw + i * sf));
          x[j] = p.x; y[j] = p.y; z[j] = p.z;
        } else {
          const float* p = raw + i * sf;
          x[j] = __ldg(p); y[j] = __ldg(p + 1); z[j] = __ldg(p + 2);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < PPT; j++) {
      int64_t i = base + (int64_t)j * blockDim.x + threadIdx.x;
      if (i >= n) continue;
      bool fin = finite3(x[j], y[j], z[j]);
      const float4 rec = make_float4(x[j], y[j], z[j], fin ? 0.0f : CUDART_NAN_F);
      xyz4[i] = rec;
      PPP_DEV_ASSERT(!sub || (i >> sub_shift) < 16384);
      if (sub && (i & sub_mask) == 0) sub[i >> sub_shift] = rec;
      if (fin) {
        cnt++;
        mn[0] = fminf(mn[0], x[j]); mx[0] = fmaxf(mx[0], x[j]);
        mn[1] = fminf(mn[1], y[j]); mx[1] = fmaxf(mx[1], y[j]);
        mn[2] = fminf(mn[2], z[j]); mx[2] = fmaxf(mx[2], z[j]);
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int d = 0; d < 3; d++) {
      mn[d] = fminf(mn[d], __shfl_xor_sync(0xffffffffu, mn[d], o));
      mx[d] = fmaxf(mx[d], __shfl_xor_sync(0xffffffffu, mx[d], o));
    }
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  // block-level combine, then ONE set of global atomics per block (per-warp atomics on the same
  // seven addresses serialise in L2 and dominated this kernel)
  __shared__ float s_mn[8][3], s_mx[8][3];
  __shared__ unsigned s_cnt[8];
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int d = 0; d < 3; d++) { s_mn[w][d] = mn[d]; s_mx[w][d] = mx[d]; }
    s_cnt[w] = cnt;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned tot = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); i++) {
      tot += s_cnt[i];
#pragma unroll
      for (int d = 0; d < 3; d++) { mn[d] = fminf(mn[d], s_mn[i][d]); mx[d] = fmaxf(mx[d], s_mx[i][d]); }
    }
    if (tot) {
#pragma unroll
      for (int d = 0; d < 3; d++) {
        atomicMin(&acc->mn[d], f2ord(mn[d]));
        atomicMax(&acc->mx[d], f2ord(mx[d]));
      }
      atomicAdd(&acc->n_finite, (unsigned long long)tot);
    }
  }
}

__device__ __forceinline__ int cell_of(const GridView& g, float x, float y, float z) {
  int cu = clampi(cell_coord_raw(axis_of(x, y, z, g.au), g.min_u, g.inv_h), 0, g.nu - 1);
  int cv = clampi(cell_coord_raw(axis_of(x, y, z, g.av), g.min_v, g.inv_h), 0, g.nv - 1);
  return cv * g.nu + cu;
}

__global__ void __launch_bounds__(256) k_cell_count(GridView g, const float4* __restrict__ xyz4, int64_t n,
                                                    int32_t* __restrict__ counts) {
  pdl_prologue();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 p = __ldg(xyz4 + i);
  if (p.w != p.w) return;  // non-finite point: not indexed
  const int cell = cell_of(g, p.x, p.y, p.z);
  PPP_DEV_ASSERT(cell >= 0 && cell < g.nu * g.nv);
  atomicAdd(counts + cell, 1);
}

// counts[] still holds the histogram; each point claims slot start[c] + (--counts[c]).
__global__ void __launch_bounds__(256) k_cell_scatter(GridView g, const float4* __restrict__ xyz4, int64_t n,
                                                      int32_t* __restrict__ counts, const int32_t* __restrict__ start,
                                                      float4* __restrict__ sorted) {
  pdl_prologue();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 p = __ldg(xyz4 + i);
  if (p.w != p.w) return;
  int c = cell_of(g, p.x, p.y, p.z);
  int slot = __ldg(start + c) + atomicSub(counts + c, 1) - 1;
  PPP_DEV_ASSERT(c >= 0 && c < g.nu * g.nv && slot >= 0 && slot < g.n_sorted);
  sorted[slot] = make_float4(p.x, p.y, p.z, __int_as_float((int)i));
}

// original index per sorted position as a plain array (ppp_dev_sorted_order; built on request only: the record's w
// carries the same number, and a second scattered store per point cost the index build 10 %)
__global__ void __launch_bounds__(256) k_extract_order(const float4* __restrict__ sorted, int64_t n, int32_t* __restrict__ order) {
  pdl_prologue();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) order[i] = __float_as_int(__ldg(&sorted[i].w));
}

// Surface density around a sample of the points: block b takes point b * stride_s of the cloud and looks at
// every 2^shift-th point (the compact subsample k_pack_bbox wrote on its way through the cloud).  Each thread keeps the two smallest squared distances it meets -- in space, and in
// projection onto the two axes of largest extent (the primary column grid); the 8th smallest of the block's 512
// values of either kind is (almost always exactly) the 8th nearest point of the subsample.  The 3-D value gives
// the surface density whatever the shape; the ratio of the two says how the surface projects: ~1 for a height
// field, 2-3 where sheets cover each other, tens along a vertical wall or the silhouette of a closed shape.
// out: [0, S) squared 3-D distance, [S, 2S) squared projected distance.
constexpr int DS_KTH = 8;
constexpr int DS_THREADS = 512;
__device__ __forceinline__ float ds_ord2f(uint32_t u) {
  uint32_t b = (u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u;
  return __uint_as_float(b);
}

// kth smallest of the 2 * DS_THREADS values in s (one warp; the values are consumed)
__device__ __forceinline__ float ds_kth_smallest(const float* s) {
  float v[2 * DS_THREADS / 32];
#pragma unroll
  for (int i = 0; i < 2 * DS_THREADS / 32; i++) v[i] = s[i * 32 + (threadIdx.x & 31)];
  float kth = CUDART_INF_F;
  for (int r = 0; r < DS_KTH; r++) {
    float mine = CUDART_INF_F;
    int at = 0;
#pragma unroll
    for (int i = 0; i < 2 * DS_THREADS / 32; i++) if (v[i] < mine) { mine = v[i]; at = i; }
    float w = mine;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) w = fminf(w, __shfl_xor_sync(0xffffffffu, w, o));
    kth = w;
    const unsigned holders = __ballot_sync(0xffffffffu, mine == w && w < CUDART_INF_F);
    if (holders && (int)(threadIdx.x & 31) == __ffs(holders) - 1) {   // remove it from ONE lane's values
#pragma unroll
      for (int i = 0; i < 2 * DS_THREADS / 32; i++) if (i == at) v[i] = CUDART_INF_F;
    }
  }
  return kth;
}

// The LAST block to finish (ticket) copies the samples and the bounding box into mapped host memory, puts the
// scratch back to its initial state for the next cloud and raises the host's flag: no separate init kernel, no
// device-to-device copy, no fetch kernel on the critical path of an ingest.
struct IngestScratch {
  BBoxAcc acc;
  unsigned ticket;
  unsigned pad[3];
  float samples[2 * 128];
};

__global__ void __launch_bounds__(DS_THREADS) k_density_sample(const float4* __restrict__ xyz4, int64_t n, int64_t stride_s,
                                                               const float4* __restrict__ sub, int m, IngestScratch* __restrict__ scr, int S,
                                                               unsigned* __restrict__ host_out, unsigned* __restrict__ host_flag,
                                                               unsigned seq, const long long* __restrict__ n_dev,
                                                               const unsigned* __restrict__ extra_src, int extra_words) {
  pdl_prologue();
  __shared__ float s_d[2 * DS_THREADS], s_p[2 * DS_THREADS];
  __shared__ bool s_last;
  if (n_dev) {   // point count known on the device only: the same choices cloud_ingest makes on the host
    n = *n_dev;
    const long long ds_s = n < (long long)gridDim.x ? n : (long long)gridDim.x;
    stride_s = ds_s > 0 ? (n / ds_s > 1 ? n / ds_s : 1) : 1;
    const int sh = ds_sub_shift(n);
    m = (int)((n + ((long long)1 << sh) - 1) >> sh);
  }
  const BBoxAcc* acc = &scr->acc;
  float* out = scr->samples;
  // the axis the primary grid does not span: smallest extent, ties drop z, then y (as cloud_ingest decides)
  int drop = 2;
  {
    double ext[3];
    for (int d = 0; d < 3; d++) ext[d] = (double)ds_ord2f(acc->mx[d]) - (double)ds_ord2f(acc->mn[d]);
    if (ext[1] < ext[drop]) drop = 1;
    if (ext[0] < ext[drop]) drop = 0;
  }
  const bool has_q = (int64_t)blockIdx.x * stride_s < n;
  const float4 q = has_q ? __ldg(xyz4 + (int64_t)blockIdx.x * stride_s) : make_float4(0.f, 0.f, 0.f, CUDART_NAN_F);
  const bool qfin = q.w == q.w;
  float d0 = CUDART_INF_F, d1 = CUDART_INF_F, p0 = CUDART_INF_F, p1 = CUDART_INF_F;
  if (qfin) {
    constexpr int PPT = 8;   // independent loads in flight per thread (the subsample is compact: coalesced lines from L2)
    for (int j0 = (int)threadIdx.x; j0 < m; j0 += DS_THREADS * PPT) {
      float4 p[PPT];
#pragma unroll
      for (int u = 0; u < PPT; u++) {
        const int j = j0 + u * DS_THREADS;
        p[u] = j < m ? __ldg(sub + j) : make_float4(CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F);
      }
#pragma unroll
      for (int u = 0; u < PPT; u++) {
        const float dx = q.x - p[u].x, dy = q.y - p[u].y, dz = q.z - p[u].z;
        const float d2 = dx * dx + dy * dy + dz * dz;
        if (!(d2 > 0.0f) || !(d2 < CUDART_INF_F)) continue;     // the sample itself, exact duplicates, non-finite points
        const float p2 = drop == 0 ? dy * dy + dz * dz : (drop == 1 ? dx * dx + dz * dz : dx * dx + dy * dy);
        if (d2 < d0) { d1 = d0; d0 = d2; } else if (d2 < d1) d1 = d2;
        if (p2 < p0) { p1 = p0; p0 = p2; } else if (p2 < p1) p1 = p2;
      }
    }
  }
  s_d[threadIdx.x] = d0; s_d[DS_THREADS + threadIdx.x] = d1;
  s_p[threadIdx.x] = p0; s_p[DS_THREADS + threadIdx.x] = p1;
  __syncthreads();
  if (threadIdx.x < 32) {
    const float r2 = ds_kth_smallest(s_d);
    if (threadIdx.x == 0) { out[blockIdx.x] = r2; __threadfence(); }
  } else if (threadIdx.x < 64) {
    const float r2 = ds_kth_smallest(s_p);
    if ((threadIdx.x & 31) == 0) { out[S + blockIdx.x] = r2; __threadfence(); }
  }
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(&scr->ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  // payload: 2 * S samples, then the bounding-box accumulator (8 words)
  const volatile unsigned* vs = (const volatile unsigned*)scr->samples;
  for (int i = threadIdx.x; i < 2 * S; i += blockDim.x) host_out[i] = ((int)(i % S) < (int)gridDim.x) ? vs[i] : 0x7FC00000u;
  const volatile unsigned* va = (const volatile unsigned*)&scr->acc;
  if (threadIdx.x < (int)(sizeof(BBoxAcc) / 4)) host_out[2 * S + threadIdx.x] = va[threadIdx.x];
  // ... the point count, and whatever else the caller wants with the same hand-shake (the exchange's summary)
  if (threadIdx.x == 0) { host_out[2 * S + 8] = (unsigned)((unsigned long long)n & 0xFFFFFFFFull); host_out[2 * S + 9] = (unsigned)((unsigned long long)n >> 32); }
  for (int i = threadIdx.x; i < extra_words; i += blockDim.x) host_out[2 * S + 10 + i] = ((const volatile unsigned*)extra_src)[i];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int d = 0; d < 3; d++) { scr->acc.mn[d] = 0xFFFFFFFFu; scr->acc.mx[d] = 0u; }
    scr->acc.n_finite = 0ull;
    scr->ticket = 0u;
    *(volatile unsigned*)host_flag = seq;
  }
}

struct G3 { GridView g[3]; };

// Points in the (2R+1)^2 cell block around p in grid g.
__device__ __forceinline__ int block_population(const GridView& g, float x, float y, float z, int R) {
  const int cu = cell_coord_raw(axis_of(x, y, z, g.au), g.min_u, g.inv_h);
  const int cv = cell_coord_raw(axis_of(x, y, z, g.av), g.min_v, g.inv_h);
  const int a = max(cu - R, 0), b = min(cu + R, g.nu - 1);
  if (a > b) return 0;
  int cnt = 0;
  for (int v = max(cv - R, 0); v <= min(cv + R, g.nv - 1); v++) {
    const int32_t* row = g.cell_start + (int64_t)v * g.nu;
    cnt += __ldg(row + b + 1) - __ldg(row + a);
  }
  return cnt;
}

// choice[i]: the projection whose candidate block around point i holds the fewest points.  Every block is a
// superset of the 3-D ball of radius R*h around the point (projecting only shortens distances), so the smallest
// block is simply the one with the fewest points that are NOT neighbours.  hist[p]: how many points chose p.
__global__ void __launch_bounds__(256) k_mp_choose(G3 G, const float4* __restrict__ xyz4, int64_t n, int R,
                                                   unsigned char* __restrict__ choice, unsigned long long* __restrict__ hist) {
  pdl_prologue();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int pick = -1;
  if (i < n) {
    const float4 p = __ldg(xyz4 + i);
    pick = 0;
    if (p.w == p.w) {
      int best_cnt = 2147483647;
#pragma unroll
      for (int k = 2; k >= 0; k--) {     // ties: prefer x,y then x,z then y,z
        const int cnt = block_population(G.g[k], p.x, p.y, p.z, R);
        if (cnt < best_cnt) { pick = k; best_cnt = cnt; }
      }
    }
    choice[i] = (unsigned char)pick;
  }
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const unsigned bal = __ballot_sync(0xffffffffu, pick == k);
    if ((threadIdx.x & 31) == 0 && bal) atomicAdd(hist + k, (unsigned long long)__popc(bal));
  }
}

}  // namespace

int cloud_ingest(ppp_cloud* c, const void* pts_dev, size_t stride_bytes) {
  return cloud_ingest_ex(c, pts_dev, stride_bytes, c->n, nullptr, nullptr, 0, nullptr);
}

// n_dev != nullptr: the point count lies in device memory (*n_dev <= n_cap, written by earlier work of the stream) and
// reaches the host together with the ingest results -- c->n is set from it; `extra_bytes` of device memory at
// extra_src travel with the same hand-shake into extra_out (multiples of 4).
int cloud_ingest_ex(ppp_cloud* c, const void* pts_dev, size_t stride_bytes, int64_t n_cap, const long long* n_dev,
                    const void* extra_src, size_t extra_bytes, void* extra_out) {
  ppp_ctx* ctx = c->ctx;
  int sf = (int)(stride_bytes / 4);
  int vec_ok = (stride_bytes % 16 == 0) && (((uintptr_t)pts_dev) % 16 == 0);
  if (!n_dev) n_cap = c->n;
  PPP_TRY(dev_alloc_keep(ctx, &c->xyz4, (size_t)n_cap));
  constexpr int DS_SAMPLES = 128;
  static_assert(offsetof(IngestScratch, ticket) == sizeof(BBoxAcc), "k_bbox_init zeroes the ticket behind the accumulator");
  BBoxAcc h;
  std::vector<float> ds_h((size_t)2 * DS_SAMPLES, NAN);
  for (int d = 0; d < 3; d++) { h.mn[d] = 0xFFFFFFFFu; h.mx[d] = 0u; }
  h.n_finite = 0ull;
  if (n_cap > 0) {
    const int sub_shift = ds_sub_shift(n_cap);
    const int sub_m = (int)((n_cap + ((int64_t)1 << sub_shift) - 1) >> sub_shift);
    const int ds_blocks = (int)std::min<int64_t>(DS_SAMPLES, n_cap);
    const int64_t stride_s0 = std::max<int64_t>(1, n_cap / ds_blocks);
    constexpr size_t SUB_BYTES = (size_t)16384 * sizeof(float4);
    if (!ctx->ingest_dev) {
      PPP_CUDA(cudaMalloc(&ctx->ingest_dev, SUB_BYTES + sizeof(IngestScratch)));   // [subsample][scratch]
      ctx->ingest_clean = false;
    }
    float4* sub = (float4*)ctx->ingest_dev;
    IngestScratch* scr = (IngestScratch*)((char*)ctx->ingest_dev + SUB_BYTES);
    if (!ctx->ingest_clean) {
      PPP_LAUNCH(ctx, "bbox_init", k_bbox_init, 1, 1, 0, &scr->acc);
      PPP_CHECK_LAUNCH();
    }
    ctx->ingest_clean = false;   // until this ingest's last block has reset it
    int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n_cap + 1023) / 1024, (int64_t)ctx->sm_count * 16));
    PPP_LAUNCH(ctx, "pack_bbox", k_pack_bbox, blocks, 256, 0, (const float*)pts_dev, n_cap, sf, vec_ok, c->xyz4, &scr->acc, sub, sub_shift, n_dev);
    PPP_CHECK_LAUNCH();
    // surface density + projection quality from a sample; its last block delivers samples + bounding box to the host
    const unsigned seq = ++ctx->fetch_seq ? ctx->fetch_seq : ++ctx->fetch_seq;
    const int extra_words = (int)(extra_bytes / 4);
    PPP_LAUNCH(ctx, "density_sample", k_density_sample, ds_blocks, DS_THREADS, 0, (const float4*)c->xyz4, n_cap, stride_s0, (const float4*)sub, sub_m,
               scr, DS_SAMPLES, (unsigned*)ctx->fetch_host, (unsigned*)fetch_flag(ctx), seq, n_dev, (const unsigned*)extra_src, extra_words);
    PPP_CHECK_LAUNCH();
    PPP_TRY(fetch_wait(ctx, seq));
    ctx->ingest_clean = true;
    const char* pay = (const char*)ctx->fetch_host;
    memcpy(ds_h.data(), pay, ds_h.size() * sizeof(float));
    memcpy(&h, pay + ds_h.size() * sizeof(float), sizeof(h));
    if (n_dev) {
      long long n_real = 0;
      memcpy(&n_real, pay + ds_h.size() * sizeof(float) + sizeof(h), sizeof(n_real));
      c->n = std::min<int64_t>(std::max<long long>(n_real, 0), n_cap);
    }
    if (extra_out && extra_bytes) memcpy(extra_out, pay + ds_h.size() * sizeof(float) + sizeof(h) + 8, extra_bytes);
  } else if (n_dev) {
    c->n = 0;
    if (extra_out && extra_bytes) PPP_TRY(fetch_small(ctx, extra_src, extra_bytes, extra_out));
  }
  // the choices the kernels made from the point count
  const int sub_shift = ds_sub_shift(c->n);
  const int64_t stride_m = (int64_t)1 << sub_shift;
  const int ds_s = (int)std::min<int64_t>(DS_SAMPLES, c->n);
  c->n_finite = (int64_t)h.n_finite;
  for (int d = 0; d < 3; d++) {
    // [upstream] getMinMax3D starts from +/-FLT_MAX; an all-non-finite cloud keeps those.
    c->bmin[d] = c->n_finite ? ord2f(h.mn[d]) : 3.402823466e+38f;
    c->bmax[d] = c->n_finite ? ord2f(h.mx[d]) : -3.402823466e+38f;
  }
  // (u, v) = the two axes with the largest extent; ties keep x, y.
  double ext[3];
  for (int d = 0; d < 3; d++) ext[d] = c->n_finite ? (double)c->bmax[d] - (double)c->bmin[d] : 0.0;
  int drop = 2;  // the axis with the smallest extent is not gridded (ties: drop z, then y)
  if (ext[1] < ext[drop]) drop = 1;
  if (ext[0] < ext[drop]) drop = 0;
  c->drop = drop;
  c->au = drop == 0 ? 1 : 0;
  c->av = drop == 2 ? 1 : 2;
  double area = std::max(ext[c->au], 1e-9) * std::max(ext[c->av], 1e-9);
  c->density = c->n_finite > 0 ? (double)c->n_finite / area : 0.0;     // fallback: points per bounding-rectangle area
  // sampled estimate: the area out to the k-th neighbour of a Poisson process is Gamma(k) distributed (median
  // 7.67 for k = 8); the samples saw every stride_m-th point only
  std::vector<float> r2;
  int piled = 0;
  for (int i = 0; i < ds_s; i++)
    if (std::isfinite(ds_h[i]) && ds_h[i] > 0) {
      r2.push_back(ds_h[i]);
      piled += ds_h[DS_SAMPLES + i] * 4.0f < ds_h[i] ? 1 : 0;   // the same count within 1/4 of the area: 4x denser in projection
    }
  // Not a height field over the primary axis pair if a noticeable share of the surface piles up in projection
  // (vertical walls, silhouettes of closed shapes): use one column grid per axis pair (MPSet).
  c->mp_state = (r2.size() >= 32 && c->n_finite >= 4096 && piled * 25 > (int)r2.size()) ? 1 : 0;
  if (const char* e = getenv("PPP_PROJECTIONS")) {            // tuning / test aid: 1 = never, 3 = always
    if (e[0] == '1') c->mp_state = 0;
    if (e[0] == '3') c->mp_state = 1;
  }
  if (getenv("PPP_DEBUG"))
    fprintf(stderr, "[ppp] ingest: %d of %zu samples pile up in projection -> %s\n", piled, r2.size(),
            c->mp_state ? "three projections" : "one column grid");
  if (r2.size() >= 16 && c->n_finite >= 64) {
    std::nth_element(r2.begin(), r2.begin() + r2.size() / 2, r2.end());
    const double r2_med = (double)r2[r2.size() / 2];
    const double seen = (double)((c->n + stride_m - 1) / stride_m) * ((double)c->n_finite / (double)c->n);
    const double rho_sub = 7.67 / (3.14159265358979 * r2_med);
    c->density = rho_sub * (double)c->n_finite / std::max(seen, 1.0);
  }
  return PPP_OK;
}

// Cell size for a k-search: 2 rings of cells should cover the expected k-th neighbour distance
// with ~35% head room (queries that need more simply expand further rings).
double cloud_cell_for_k(const ppp_cloud* c, int k) {
  if (c->cell_hint > 0) return c->cell_hint;
  double rho = c->density > 0 ? c->density : 1.0;
  double rk = std::sqrt((double)std::max(k, 1) / (3.14159265358979 * rho));
  double f = 1.35;
  if (const char* e = getenv("PPP_CELL_FACTOR")) { double v = atof(e); if (v > 0.5 && v < 4.0) f = v; }  // tuning aid
  return f * rk / (double)PPP_KNN_RINGS;
}
// Cell size for a radius search: R = 2 rings cover r exactly (plus rounding slack).
double cloud_cell_for_radius(const ppp_cloud* c, double r) {
  (void)c;
  return r * 0.5 * (1.0 + 1e-3);
}

int cloud_get_grid(ppp_cloud* c, double h, GridStore** out) { return cloud_get_grid_drop(c, h, c->drop, out); }

int cloud_get_grid_drop(ppp_cloud* c, double h, int drop, GridStore** out) {
  ppp_ctx* ctx = c->ctx;
  const int au = drop == 0 ? 1 : 0, av = drop == 2 ? 1 : 2;
  // cap the dense cell table (nu*nv <= 2^28) by growing h if needed
  double eu = c->n_finite ? (double)c->bmax[au] - (double)c->bmin[au] : 0.0;
  double ev = c->n_finite ? (double)c->bmax[av] - (double)c->bmin[av] : 0.0;
  if (!(h > 0)) h = 1.0;
  while ((std::floor(eu / h) + 2) * (std::floor(ev / h) + 2) > 268435456.0) h *= 1.5;
  for (auto& g : c->grids)
    if (g.drop == drop && std::fabs(g.h - h) <= 1e-9 * h) { *out = &g; return PPP_OK; }
  if (c->grids.size() >= c->grids.capacity()) {
    ppp_set_error("too many different cell sizes on one cloud (%zu grids)", c->grids.size());
    return PPP_ERR_UNSUPPORTED;   // pointers into c->grids are handed out: the vector must not reallocate
  }
  GridStore gs;
  gs.h = h;
  gs.drop = drop;
  GridView& v = gs.v;
  v.au = au; v.av = av;
  v.h = (float)h;
  v.inv_h = 1.0f / v.h;
  v.min_u = c->n_finite ? c->bmin[au] : 0.0f;
  v.min_v = c->n_finite ? c->bmin[av] : 0.0f;
  v.nu = (int)std::floor(eu * (double)v.inv_h) + 2;
  v.nv = (int)std::floor(ev * (double)v.inv_h) + 2;
  // rounding slack: cell coordinates are exact to a few ulps of (a-min)*inv_h
  v.slack = (float)(h * (double)(v.nu + v.nv) * 9.5367431640625e-07 + 1e-30);
  v.n_sorted = (int)c->n_finite;
  int64_t ncells = (int64_t)v.nu * v.nv;
  PPP_TRY(dev_alloc_keep(ctx, &gs.sorted, (size_t)std::max<int64_t>(c->n_finite, 1) + PPP_SORTED_PAD));
  PPP_TRY(dev_alloc_keep(ctx, &gs.cell_start, (size_t)ncells + 1));
  int32_t* counts = nullptr;
  PPP_TRY(dev_alloc(ctx, &counts, (size_t)ncells));
  PPP_CUDA(cudaMemsetAsync(counts, 0, (size_t)ncells * sizeof(int32_t), ctx->stream));
  v.sorted = gs.sorted;
  v.cell_start = gs.cell_start;
  if (c->n > 0) {
    unsigned blocks = (unsigned)((c->n + 255) / 256);
    PPP_LAUNCH(ctx, "cell_count", k_cell_count, blocks, 256, 0, v, (const float4*)c->xyz4, c->n, counts);
    PPP_CHECK_LAUNCH();
  }
  PPP_TRY(scan_exclusive_i32(ctx, counts, gs.cell_start, ncells));
  if (c->n > 0) {
    unsigned blocks = (unsigned)((c->n + 255) / 256);
    PPP_LAUNCH(ctx, "cell_scatter", k_cell_scatter, blocks, 256, 0, v, (const float4*)c->xyz4, c->n, counts,
               (const int32_t*)gs.cell_start, gs.sorted);
    PPP_CHECK_LAUNCH();
  }
  dev_free(ctx, counts);
  PPP_CUDA(cudaEventCreateWithFlags(&gs.ready, cudaEventDisableTiming));
  PPP_CUDA(cudaEventRecord(gs.ready, ctx->stream));
  c->grids.push_back(gs);
  *out = &c->grids.back();
  return PPP_OK;
}

// Whether the primary column grid is enough was decided at ingest from the sample (c->mp_state).
int cloud_decide_projection(ppp_cloud* c, const GridStore& g) {
  (void)g;
  if (c->mp_state < 0) c->mp_state = 0;
  return PPP_OK;
}

int cloud_get_mp(ppp_cloud* c, double h, int R0, MPSet** out) {
  ppp_ctx* ctx = c->ctx;
  for (auto& m : c->mps)
    if (m.R0 == R0 && std::fabs(m.h - h) <= 1e-9 * h) { *out = &m; return PPP_OK; }
  if (c->mps.size() >= c->mps.capacity()) { ppp_set_error("too many multi-projection index sets on one cloud"); return PPP_ERR_UNSUPPORTED; }
  MPSet m;
  m.h = h; m.R0 = R0;
  for (int p = 0; p < 3; p++) PPP_TRY(cloud_get_grid_drop(c, h, p, &m.g[p]));
  PPP_TRY(dev_alloc_keep(ctx, &m.choice, (size_t)std::max<int64_t>(c->n, 1)));
  unsigned long long* hist = nullptr;
  PPP_TRY(dev_alloc(ctx, &hist, 3));
  PPP_CUDA(cudaMemsetAsync(hist, 0, 3 * sizeof(unsigned long long), ctx->stream));
  if (c->n > 0) {
    G3 G;
    for (int p = 0; p < 3; p++) G.g[p] = m.g[p]->v;
    PPP_LAUNCH(ctx, "mp_choose", k_mp_choose, (unsigned)((c->n + 255) / 256), 256, 0, G, (const float4*)c->xyz4, c->n, R0,
               m.choice, hist);
    PPP_CHECK_LAUNCH();
  }
  if (getenv("PPP_DEBUG")) {
    unsigned long long hh[3] = {0, 0, 0};
    PPP_TRY(fetch_small(ctx, hist, sizeof(hh), hh));
    fprintf(stderr, "[ppp] projections chosen (h = %g, R0 = %d): yz %llu, xz %llu, xy %llu\n", h, R0, hh[0], hh[1], hh[2]);
  }
  dev_free(ctx, hist);
  PPP_CUDA(cudaEventCreateWithFlags(&m.ready, cudaEventDisableTiming));
  PPP_CUDA(cudaEventRecord(m.ready, ctx->stream));
  c->mps.push_back(m);
  *out = &c->mps.back();
  return PPP_OK;
}

int grid_sorted_order(ppp_cloud* c, GridStore& gs) {
  if (gs.order) return PPP_OK;
  ppp_ctx* ctx = c->ctx;
  const int64_t n = gs.v.n_sorted;
  PPP_TRY(dev_alloc_keep(ctx, &gs.order, (size_t)std::max<int64_t>(n, 1)));
  if (n > 0) {
    PPP_LAUNCH(ctx, "extract_order", k_extract_order, (unsigned)((n + 255) / 256), 256, 0, (const float4*)gs.sorted, n, gs.order);
    PPP_CHECK_LAUNCH();
  }
  return PPP_OK;
}

// ---------------------------------------------------------------------------------------------
__global__ void k_fetch_small(const unsigned* __restrict__ src, unsigned* __restrict__ dst, int words,
                              unsigned* __restrict__ flag, unsigned seq) {
  pdl_prologue();
  for (int i = threadIdx.x; i < words; i += blockDim.x) dst[i] = src[i];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) *(volatile unsigned*)flag = seq;
}

int fetch_wait(ppp_ctx* ctx, unsigned seq) {
  volatile unsigned* flag = fetch_flag(ctx);
  for (unsigned long spin = 1;; spin++) {
    if (*flag == seq) return PPP_OK;
    if ((spin & 0x1FFFul) == 0) {
      cudaError_t e = cudaStreamQuery(ctx->stream);
      if (e == cudaSuccess) {
        if (*flag == seq) return PPP_OK;
        ppp_set_error("fetch: the stream drained without the kernel signalling (sequence %u)", seq);
        return PPP_ERR_CUDA;
      }
      if (e != cudaErrorNotReady) {
        ppp_set_error("fetch: %s", cudaGetErrorString(e));
        return PPP_ERR_CUDA;
      }
    }
  }
}

int fetch_small(ppp_ctx* ctx, const void* dev_src, size_t bytes, void* host_dst) {
  if (bytes == 0) { PPP_CUDA(cudaStreamSynchronize(ctx->stream)); return PPP_OK; }
  if (bytes > FETCH_BYTES || (bytes & 3) || ((uintptr_t)dev_src & 3) || !ctx->fetch_host) {
    PPP_CUDA(cudaMemcpyAsync(host_dst, dev_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    PPP_CUDA(cudaStreamSynchronize(ctx->stream));
    return PPP_OK;
  }
  const unsigned seq = ++ctx->fetch_seq ? ctx->fetch_seq : ++ctx->fetch_seq;   // never 0 (the flag's initial value)
  PPP_LAUNCH(ctx, "fetch_small", k_fetch_small, 1, 256, 0, (const unsigned*)dev_src, (unsigned*)ctx->fetch_host, (int)(bytes / 4),
             (unsigned*)fetch_flag(ctx), seq);
  PPP_CHECK_LAUNCH();
  PPP_TRY(fetch_wait(ctx, seq));
  memcpy(host_dst, ctx->fetch_host, bytes);
  return PPP_OK;
}
