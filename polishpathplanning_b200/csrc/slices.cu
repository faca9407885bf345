// Plane-slice band extraction for ALL planes in one pass over the cloud, and the per-slice
// contour: left/right classification, pairing (gen-2 variant A / SectPath variant B),
// interpolation onto the plane and the std::map ascending-y ordering.
// Replaces rangedX_index (src/Path_Generation.cpp:94-104; src/contour_alg.cpp:153-163),
// insert_point (src/Path_Generation.cpp:107-206; src/contour_alg.cpp:165-237) and the map ->
// array flattening in path_track / OnePath (src/Path_Generation.cpp:659-676; src/contour_alg.cpp:240-257).
#include <algorithm>
#include <functional>
#include <cmath>
#include <vector>

#include <cooperative_groups.h>

#include "ppp_device.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int CT_THREADS = 256;

// ---------------------------------------------------------------------------------------------
// bands
// ---------------------------------------------------------------------------------------------
struct BandSet {
  const float* lo;      // sorted ascending (NaN planes last, never matched)
  const float* hi;      // same order
  const int32_t* slice; // original slice number of sorted entry
  int S;
  // A sweep with constant pitch (the usual case): lo[t] ~ lo0 + t * pitch and hi[t] ~ hi0 + t * pitch to within a
  // quarter pitch (checked on the host).  The slices that can contain x then follow from two multiplications
  // instead of two binary searches of log2(S) dependent loads each; the exact limits are re-tested either way.
  int regular;
  float lo0, hi0, inv_pitch;
};

// slices containing x form the contiguous sorted range [first hi >= x, first lo > x)
__device__ __forceinline__ void band_range(const BandSet& b, float x, int& first, int& last) {
  int l = 0, r = b.S;
  while (l < r) { int m = (l + r) >> 1; if (__ldg(b.lo + m) <= x) l = m + 1; else r = m; }
  last = l;  // exclusive
  l = 0; r = b.S;
  while (l < r) { int m = (l + r) >> 1; if (__ldg(b.hi + m) < x) l = m + 1; else r = m; }
  first = l;
}

// PassThrough: finite point, !(x < lo || x > hi).
// Each block owns a contiguous chunk of the cloud and histograms its members per slice in shared
// memory (global atomics on S counters serialise at ~50 ns per update; shared-memory atomics do
// not), then touches each global counter once.  The fill pass reserves one contiguous range per
// (block, slice) the same way and places members with shared-memory ranks.  Order inside a band
// is arbitrary here; k_band_sort restores PassThrough's ascending-index order where a caller
// needs it (ppp_slice_bands output, the order-dependent gen-2 pairing).
constexpr int BAND_SMEM_BINS = 12288;  // 48 KB of int32

template <typename F>
__device__ __forceinline__ void for_memberships(const BandSet& b, float x, F&& f) {
  int first, last;
  if (b.regular) {
    // t with hi[t] >= x: t >= (x - hi0) / pitch;  t with lo[t] <= x: t <= (x - lo0) / pitch;  one slice of margin
    // on either side covers the quarter-pitch tolerance and the rounding (non-finite x: empty range)
    const float a = (x - b.hi0) * b.inv_pitch, c = (x - b.lo0) * b.inv_pitch;
    if (!(a == a) || !(c == c)) return;
    first = max((int)fminf(fmaxf(ceilf(a) - 1.0f, 0.0f), 2.0e9f), 0);
    last = min((int)fminf(fmaxf(floorf(c) + 2.0f, 0.0f), 2.0e9f), b.S);
  } else {
    band_range(b, x, first, last);
  }
  for (int t = first; t < last; t++) {
    // lo/hi are sorted together only when all bands have one width; re-test to stay exact otherwise
    if (x < __ldg(b.lo + t) || x > __ldg(b.hi + t)) continue;
    f(t);
  }
}

__global__ void __launch_bounds__(256) k_band_count(BandSet b, const float4* __restrict__ xyz4, int64_t n, int64_t chunk,
                                                    int use_smem, int w_is_flag, int32_t* __restrict__ counts,
                                                    int S_all, int64_t* __restrict__ offsets_out) {
  pdl_prologue();
  extern __shared__ int32_t s_cnt[];
  __shared__ long long s_scan[256];
  __shared__ bool s_last;
  if (use_smem) {
    for (int t = threadIdx.x; t < b.S; t += blockDim.x) s_cnt[t] = 0;
    __syncthreads();
  }
  int64_t beg = (int64_t)blockIdx.x * chunk, end = min(beg + chunk, n);
  for (int64_t i = beg + threadIdx.x; i < end; i += blockDim.x) {
    float4 p = __ldg(xyz4 + i);
    if (w_is_flag && p.w != p.w) continue;   // packed cloud: w = NaN marks a non-finite point
    for_memberships(b, p.x, [&](int t) {
      if (use_smem) atomicAdd(s_cnt + t, 1);
      else atomicAdd(counts + __ldg(b.slice + t), 1);
    });
  }
  if (use_smem) {
    __syncthreads();
    for (int t = threadIdx.x; t < b.S; t += blockDim.x) {
      int c = s_cnt[t];
      if (c) atomicAdd(counts + __ldg(b.slice + t), c);
    }
  }
  if (!offsets_out) return;
  // The LAST block to finish turns the S_all counts into the band offsets (exclusive scan, int64, total at [S_all])
  // and zeroes the counts -- they are the fill pass's cursors -- and the ticket (counts[S_all]): no scan launch and no
  // memset between the two passes of the band builder (each costs the chain ~10-20 us when the GPU is busy).
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd((unsigned*)(counts + S_all), 1u) == gridDim.x - 1;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const int per = (S_all + (int)blockDim.x - 1) / (int)blockDim.x;
  const int t0 = min((int)threadIdx.x * per, S_all), t1 = min(t0 + per, S_all);
  long long sum = 0;
  for (int t = t0; t < t1; t++) sum += ((const volatile int32_t*)counts)[t];
  s_scan[threadIdx.x] = sum;
  __syncthreads();
  for (int o = 1; o < (int)blockDim.x; o <<= 1) {     // inclusive scan of the per-thread sums (Hillis-Steele)
    const long long v = (int)threadIdx.x >= o ? s_scan[threadIdx.x - o] : 0;
    __syncthreads();
    s_scan[threadIdx.x] += v;
    __syncthreads();
  }
  long long run = s_scan[threadIdx.x] - sum;
  for (int t = t0; t < t1; t++) {
    offsets_out[t] = run;
    run += ((const volatile int32_t*)counts)[t];
    counts[t] = 0;
  }
  if (threadIdx.x == blockDim.x - 1) { offsets_out[S_all] = s_scan[blockDim.x - 1]; counts[S_all] = 0; }
}

__global__ void __launch_bounds__(256) k_band_fill(BandSet b, const float4* __restrict__ xyz4, int64_t n, int64_t chunk,
                                                   int use_smem, int w_is_flag, int32_t* __restrict__ cursor,
                                                   const int64_t* __restrict__ offsets, int32_t* __restrict__ idx_out) {
  pdl_prologue();
  extern __shared__ int32_t s_mem[];
  int32_t* s_cnt = s_mem;
  int32_t* s_base = s_mem + b.S;
  int64_t beg = (int64_t)blockIdx.x * chunk, end = min(beg + chunk, n);
  if (use_smem) {
    for (int t = threadIdx.x; t < b.S; t += blockDim.x) s_cnt[t] = 0;
    __syncthreads();
    for (int64_t i = beg + threadIdx.x; i < end; i += blockDim.x) {
      float4 p = __ldg(xyz4 + i);
      if (w_is_flag && p.w != p.w) continue;   // packed cloud: w = NaN marks a non-finite point
      for_memberships(b, p.x, [&](int t) { atomicAdd(s_cnt + t, 1); });
    }
    __syncthreads();
    for (int t = threadIdx.x; t < b.S; t += blockDim.x) {
      int c = s_cnt[t];
      s_base[t] = c ? atomicAdd(cursor + __ldg(b.slice + t), c) : 0;
      s_cnt[t] = 0;
    }
    __syncthreads();
  }
  for (int64_t i = beg + threadIdx.x; i < end; i += blockDim.x) {
    float4 p = __ldg(xyz4 + i);
    if (w_is_flag && p.w != p.w) continue;   // packed cloud: w = NaN marks a non-finite point
    for_memberships(b, p.x, [&](int t) {
      int s = __ldg(b.slice + t);
      int pos = use_smem ? s_base[t] + atomicAdd(s_cnt + t, 1) : atomicAdd(cursor + s, 1);
      PPP_DEV_ASSERT(pos >= 0 && offsets[s] + pos < offsets[s + 1]);
      idx_out[offsets[s] + pos] = (int32_t)i;
    });
  }
}

// Bitonic sorting network on a (possibly non power-of-two) array with virtual +inf padding: every
// compare-exchange puts the minimum at the lower index, partners beyond n are skipped.
// One thread per COMPARATOR (no idle half), and a warp owns 64 consecutive elements through every step whose
// span fits in them -- whole stages up to k = 64 and the j <= 32 tail of every later stage --, so those steps are
// separated by __syncwarp only: 21 block-wide barriers for 2048 elements instead of 66.
template <typename T>
__device__ __forceinline__ void cta_sort_ce(T* a, int i, int l, int n) {
  PPP_DEV_ASSERT(i >= 0 && i < l);
  if (l < n) { T x = a[i], y = a[l]; if (y < x) { a[i] = y; a[l] = x; } }
}
// Steps j0, j0 / 2, .., 1 of a merge over a[0 .. 2 * half) (n valid elements in front); ends with a block barrier.
template <typename T>
__device__ void cta_jsteps(T* a, int n, int half, int j0) {
  const int nt = blockDim.x;
  for (int j = j0; j > 32; j >>= 1) {
    for (int c = threadIdx.x; c < half; c += nt) { const int i = 2 * c - (c & (j - 1)); cta_sort_ce(a, i, i + j, n); }
    __syncthreads();
  }
  for (int c0 = threadIdx.x; c0 - (int)(threadIdx.x & 31) < half; c0 += nt) {   // warp-uniform trip count
    const int c = c0;
    for (int j = min(j0, 32); j > 0; j >>= 1) {
      if (c < half) { const int i = 2 * c - (c & (j - 1)); cta_sort_ce(a, i, i + j, n); }
      __syncwarp();
    }
  }
  __syncthreads();
}

template <typename T>
__device__ void cta_sort(T* a, int n) {
  if (n <= 1) return;   // uniform over the block
  int np2 = 2;
  while (np2 < n) np2 <<= 1;
  const int half = np2 >> 1;                       // comparators per step
  const int nt = blockDim.x;                       // a multiple of 32
  // stages k = 2 .. 64: warp-local throughout
  for (int c0 = threadIdx.x; c0 - (int)(threadIdx.x & 31) < half; c0 += nt) {   // warp-uniform trip count
    const int c = c0;
    for (int k = 2; k <= min(np2, 64); k <<= 1) {
      const int hk = k >> 1;
      if (c < half) { const int b = c / hk, o = c - b * hk; cta_sort_ce(a, b * k + o, b * k + (k - 1 - o), n); }
      __syncwarp();
      for (int j = k >> 2; j > 0; j >>= 1) {
        if (c < half) { const int i = 2 * c - (c & (j - 1)); cta_sort_ce(a, i, i + j, n); }
        __syncwarp();
      }
    }
  }
  __syncthreads();
  for (int k = 128; k <= np2; k <<= 1) {
    const int hk = k >> 1;
    for (int c = threadIdx.x; c < half; c += nt) { const int b = c / hk, o = c - b * hk; cta_sort_ce(a, b * k + o, b * k + (k - 1 - o), n); }
    __syncthreads();
    cta_jsteps(a, n, half, k >> 2);
  }
}

__global__ void __launch_bounds__(1024) k_band_sort(const int64_t* __restrict__ offsets, int32_t* __restrict__ idx, int smem_cap) {
  pdl_prologue();
  extern __shared__ int32_t s_idx[];
  int s = blockIdx.x;
  int64_t o = offsets[s];
  int n = (int)(offsets[s + 1] - o);
  if (n <= 1) return;
  if (n <= smem_cap) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) s_idx[i] = idx[o + i];
    __syncthreads();
    cta_sort(s_idx, n);
    for (int i = threadIdx.x; i < n; i += blockDim.x) idx[o + i] = s_idx[i];
  } else {
    cta_sort(idx + o, n);
  }
}

// ---------------------------------------------------------------------------------------------
// contours
// ---------------------------------------------------------------------------------------------
struct ContourParams {
  GridView g;
  GridView g3[3];                // multi-projection index: g3[choice[point]] is searched for that point
  const unsigned char* choice;   // nullptr: the single grid g
  const float4* xyz4;
  const float* planes;   // S, original order
  const float* lo;       // S, original order
  const float* hi;
  const int64_t* band_off;
  const int32_t* band_idx;
  int mode;              // PPP_PAIR_GEN2 / PPP_PAIR_SECT
  // scratch, all indexed by band offset
  int32_t *El, *Er;      // left / right members (ascending index)
  u64* keys;
  float *ys, *zs;
  int32_t *posR, *posL, *lp, *rp;
  unsigned char *fl, *fr;
  double *ty, *tz;       // un-compacted nodes per slice
  int32_t* n_nodes;      // S
  const uint32_t* member; // optional membership bitmap (explicit index lists)
};

// The grid in which the neighbourhood of point `idx` is searched.
template <typename PARAMS>
__device__ __forceinline__ const GridView& grid_for(const PARAMS& P, int idx) {
  return P.choice ? P.g3[__ldg(P.choice + idx)] : P.g;
}

__device__ __forceinline__ uint32_t f2ord_dev(float f) {
  uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// CTA-wide exclusive prefix count of a per-thread flag over the current tile; `running` is
// advanced by the tile total (kept identical in every thread).
__device__ __forceinline__ int cta_flag_rank(bool flag, int* s_warp, int& running) {
  unsigned m = __ballot_sync(0xffffffffu, flag);
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) s_warp[w] = __popc(m);
  __syncthreads();
  int base = 0, tot = 0;
  const int nw = (blockDim.x + 31) >> 5;
  for (int i = 0; i < nw; i++) {
    int c = s_warp[i];
    if (i < w) base += c;
    tot += c;
  }
  int r = running + base + __popc(m & ((1u << lane) - 1u));
  running += tot;
  __syncthreads();
  return r;
}

// Nearest member of one side of the slice (x in [lo,hi]; left: x > plane, right: x < plane).
// metric 0: flann d2, ties -> lowest index.   (variant B; contract (d2, idx))
// metric 1: Eigen norm sqrtf(dx^2 + (dy^2 + dz^2)), ties -> highest index (std::map<float,int>
//           overwrite in src/Path_Generation.cpp:143-150: equal keys keep the last j).
// Searches the grid ring by ring; gives up after RMAX rings and scans the side's member list.
// Returns {original index, sorted position} of the winner ({-1, -1}: the side is empty).  `list`: the band's
// members as original indices (by_pos == 0) or as sorted positions (by_pos != 0); the position of a winner
// found by scanning an index list is unknown (-1) -- rec_of() then reads the packed cloud instead.
template <bool MEMBER>
__device__ int2 nn_side(const GridView& g, const float4* __restrict__ xyz4, float qx, float qy, float qz, float lo,
                        float hi, float plane, bool want_left, int metric, const int32_t* list, int nlist,
                        const uint32_t* __restrict__ member, int by_pos) {
  if (nlist <= 0) return make_int2(-1, -1);
  // Ring by ring while that is cheaper than walking the band's member list (~2.5 points per cell against
  // nlist entries); a band along the silhouette of a closed shape has tens of thousands of members whose
  // nearest member on the other side can be centimetres away.
  const int RMAX = max(6, min(64, (int)(0.5f * sqrtf(0.4f * (float)nlist))));
  u64 best = PPP_KEY_INF;
  int best_pos = -1;
  // membership of the slice: the x-interval of the band, or (explicit index lists) a bitmap
  auto consider = [&](float cx, float cy, float cz, int idx, int pos) {
    if (MEMBER) { if (!((__ldg(member + (idx >> 5)) >> (idx & 31)) & 1u)) return; }
    else if (cx < lo || cx > hi) return;
    if (want_left ? !(cx > plane) : !(cx < plane)) return;
    u64 key;
    if (metric == 0) {
      key = make_key(d2_flann(qx, qy, qz, cx, cy, cz), idx);
    } else {
      float dx = __fsub_rn(qx, cx), dy = __fsub_rn(qy, cy), dz = __fsub_rn(qz, cz);
      float nn = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fadd_rn(__fmul_rn(dy, dy), __fmul_rn(dz, dz))));
      key = ((u64)__float_as_uint(nn) << 32) | (u64)(~(uint32_t)idx);
    }
    if (key < best) { best = key; best_pos = pos; }
  };
  int cu = cell_coord_raw(axis_of(qx, qy, qz, g.au), g.min_u, g.inv_h);
  int cv = cell_coord_raw(axis_of(qx, qy, qz, g.av), g.min_v, g.inv_h);
  // when x is the fast grid axis only the cell columns that overlap the wanted x-interval can
  // hold members (cell coordinates are monotone in x)
  int ulo = -2147483647, uhi = 2147483647;
  if (g.au == 0 && !MEMBER) {
    ulo = cell_coord_raw(want_left ? plane : lo, g.min_u, g.inv_h);
    uhi = cell_coord_raw(want_left ? hi : plane, g.min_u, g.inv_h);
  }
  int R = 1, R_prev = -1;
  bool done = false;
  while (true) {
    visit_annulus_pos(g, cu, cv, R_prev, R, [&](float4 c, int pos) { consider(c.x, c.y, c.z, __float_as_int(c.w), pos); }, ulo, uhi);
    if (best != PPP_KEY_INF) {
      float b2 = ring_bound2(g, R, cu, cv);
      float v = __uint_as_float((uint32_t)(best >> 32));
      if (metric == 0 ? (v < b2) : (v < __fsqrt_rd(b2))) { done = true; break; }
    }
    if (block_covers_grid(g, cu, cv, R)) { done = true; break; }
    if (R >= RMAX) break;
    R_prev = R;
    R++;
  }
  if (!done) {
    best = PPP_KEY_INF;
    best_pos = -1;
    for (int t = 0; t < nlist; t++) {
      const int e = list[t];
      if (by_pos) {
        float4 c = __ldg(g.sorted + e);
        consider(c.x, c.y, c.z, __float_as_int(c.w), e);
      } else {
        float4 c = __ldg(xyz4 + e);
        if (c.w == c.w) consider(c.x, c.y, c.z, e, -1);   // w = NaN: not finite (explicit lists), on neither side
      }
    }
  }
  if (best == PPP_KEY_INF) return make_int2(-1, -1);
  uint32_t low = (uint32_t)(best & 0xFFFFFFFFull);
  return make_int2(metric == 0 ? (int)low : (int)(~low), best_pos);
}

// Record {x, y, z, bits(original index)} of a point given as {original index, sorted position or -1}.
__device__ __forceinline__ float4 rec_of(const GridView& g, const float4* __restrict__ xyz4, int2 h) {
  if (h.y >= 0) return __ldg(g.sorted + h.y);
  float4 c = __ldg(xyz4 + h.x);
  c.w = __int_as_float(h.x);
  return c;
}

// kdtree.nearestKSearch(p, 1) for a CLOUD POINT p: the lowest index among the points at float
// distance 0 from it (itself unless the cloud has duplicates).  Such points always share p's
// cell: d2 == 0 in float needs every coordinate difference below ~3.7e-23, which distinct floats
// only manage below 1e-15 in magnitude, far from any cell boundary other than the grid origin
// (and nothing lies below the origin: it is the cloud minimum).  So the own cell is enough.
__device__ int2 nn_full(const GridView& g, float qx, float qy, float qz, int2 self) {
  int cu = clampi(cell_coord_raw(axis_of(qx, qy, qz, g.au), g.min_u, g.inv_h), 0, g.nu - 1);
  int cv = clampi(cell_coord_raw(axis_of(qx, qy, qz, g.av), g.min_v, g.inv_h), 0, g.nv - 1);
  const int32_t* cs = g.cell_start + (int64_t)cv * g.nu + cu;
  int2 best = self;
  for (int i = __ldg(cs), e = __ldg(cs + 1); i < e; i++) {
    float4 c = __ldg(g.sorted + i);
    int idx = __float_as_int(c.w);
    if (idx < best.x && d2_flann(qx, qy, qz, c.x, c.y, c.z) == 0.0f) best = make_int2(idx, i);
  }
  return best;
}

__device__ __forceinline__ int lower_pos(const int32_t* a, int n, int v) {
  int l = 0, r = n;
  while (l < r) { int m = (l + r) >> 1; if (a[m] < v) l = m + 1; else r = m; }
  return l;
}

// gen-2 pairing (variant A).  CTA per slice.  The index lists, nearest-neighbour positions, flags
// and sort keys of a slice live in shared memory when they fit (9 bytes per band member), so the
// order-dependent greedy flag pass — one thread replaying src/Path_Generation.cpp:137-179 — runs
// at shared-memory latency; larger bands use the global scratch arrays with the same code.
template <bool MEMBER>
__global__ void __launch_bounds__(1024) k_contour(ContourParams P, int smem_cap) {
  pdl_prologue();
  extern __shared__ __align__(16) unsigned char s_dyn[];
  __shared__ int s_warp[32];
  __shared__ int s_npairs, s_nl, s_nr;
  const int s = blockIdx.x;
  const int64_t o = P.band_off[s];
  const int B = (int)(P.band_off[s + 1] - o);
  const float plane = P.planes[s], lo = P.lo[s], hi = P.hi[s];
  const int32_t* band = P.band_idx + o;
  const int Bp = (B + 1) & ~1;
  const bool in_smem = B <= smem_cap;
  int32_t* ids = in_smem ? reinterpret_cast<int32_t*>(s_dyn) : P.El + o;          // El then Er
  int32_t* pos = in_smem ? reinterpret_cast<int32_t*>(s_dyn) + Bp : P.posR + o;   // posR then posL
  unsigned char* flg = in_smem ? s_dyn + 8 * (size_t)Bp : P.fl + o;               // fl then fr
  u64* keys = in_smem ? reinterpret_cast<u64*>(s_dyn + 4 * (size_t)Bp) : P.keys + o;  // aliases pos after the greedy pass
  // ---- classify: El (x > plane), Er (x < plane), order preserved; x == plane dropped ----
  if (threadIdx.x == 0) { s_nl = 0; s_nr = 0; }
  __syncthreads();
  {
    int cl = 0, cr = 0;
    for (int i = threadIdx.x; i < B; i += (int)blockDim.x) {
      const float4 p = __ldg(P.xyz4 + band[i]);
      // (point - PlanePoint).dot((1,0,0)); a non-finite point (w = NaN; explicit lists only) is on neither side
      float d = p.w == p.w ? __fsub_rn(p.x, plane) : 0.0f;
      cl += d > 0.0f;
      cr += d < 0.0f;
    }
    if (cl) atomicAdd(&s_nl, cl);
    if (cr) atomicAdd(&s_nr, cr);
  }
  __syncthreads();
  const int nL = s_nl, nR = s_nr;
  int32_t* El = ids;
  int32_t* Er = ids + nL;
  int32_t* posR = pos;
  int32_t* posL = pos + nL;
  unsigned char* fl = flg;
  unsigned char* fr = flg + nL;
  {
    int rl_run = 0, rr_run = 0;
    for (int base = 0; base < B; base += (int)blockDim.x) {
      int i = base + threadIdx.x;
      int idx = -1;
      bool isL = false, isR = false;
      if (i < B) {
        idx = band[i];
        const float4 p = __ldg(P.xyz4 + idx);
        float d = p.w == p.w ? __fsub_rn(p.x, plane) : 0.0f;
        isL = d > 0.0f;
        isR = d < 0.0f;
      }
      int rl = cta_flag_rank(isL, s_warp, rl_run);
      int rr = cta_flag_rank(isR, s_warp, rr_run);
      if (isL) El[rl] = idx;
      if (isR) Er[rr] = idx;
    }
  }
  __syncthreads();
  int npairs = 0;
  float* ys = P.ys + o;
  float* zs = P.zs + o;
  if (nL > 0 && nR > 0) {
    // nearest right of every left, nearest left of every right (flag-independent) ...
    for (int i = threadIdx.x; i < nL; i += (int)blockDim.x) {
      float4 pl = __ldg(P.xyz4 + El[i]);
      int r = nn_side<MEMBER>(grid_for(P, El[i]), P.xyz4, pl.x, pl.y, pl.z, lo, hi, plane, false, 1, Er, nR, P.member, 0).x;
      posR[i] = lower_pos(Er, nR, r);
      fl[i] = 0;
    }
    for (int j = threadIdx.x; j < nR; j += (int)blockDim.x) {
      float4 pr = __ldg(P.xyz4 + Er[j]);
      int l = nn_side<MEMBER>(grid_for(P, Er[j]), P.xyz4, pr.x, pr.y, pr.z, lo, hi, plane, true, 1, El, nL, P.member, 0).x;
      posL[j] = lower_pos(El, nL, l);
      fr[j] = 0;
    }
    __syncthreads();
    // ... then the order-dependent greedy flag pass, replayed by one thread
    if (threadIdx.x == 0) {
      int nl = 0, nr = 0;
      for (int i = 0; i < nL; i++) {
        if (fl[i]) continue;
        int j = posR[i];
        if (fr[j]) continue;
        P.rp[o + nr++] = Er[j];
        fr[j] = 1;
        int i2 = posL[j];
        if (!fl[i2]) { P.lp[o + nl++] = El[i2]; fl[i2] = 1; }
      }
      s_npairs = nl;  // interpolation runs over left_pair.size() (src/Path_Generation.cpp:189)
    }
    __syncthreads();
    npairs = s_npairs;
    // ---- interpolate onto the plane (float32, no FMA) ----
    for (int i = threadIdx.x; i < npairs; i += (int)blockDim.x) {
      float4 r = __ldg(P.xyz4 + P.rp[o + i]);
      float4 l = __ldg(P.xyz4 + P.lp[o + i]);
      float t = __fdiv_rn(__fsub_rn(plane, r.x), __fsub_rn(l.x, r.x));
      float y = __fadd_rn(r.y, __fmul_rn(t, __fsub_rn(l.y, r.y)));
      float z = __fadd_rn(r.z, __fmul_rn(t, __fsub_rn(l.z, r.z)));
      ys[i] = y;
      zs[i] = z;
      // std::map<double,...> key order; -0.0 and +0.0 are one key
      keys[i] = ((u64)f2ord_dev(__fadd_rn(y, 0.0f)) << 32) | (u64)(uint32_t)i;
    }
    __syncthreads();
    cta_sort(keys, npairs);
  }
  // ---- unique keys: key of the first insertion, value of the last ----
  int nodes = 0;
  double* ty = P.ty + o;
  double* tz = P.tz + o;
  for (int base = 0; base < npairs; base += (int)blockDim.x) {
    int i = base + threadIdx.x;
    bool first = false, last = false;
    u64 k = 0;
    if (i < npairs) {
      k = keys[i];
      first = (i == 0) || ((keys[i - 1] >> 32) != (k >> 32));
      last = (i == npairs - 1) || ((keys[i + 1] >> 32) != (k >> 32));
    }
    // r = number of run starts strictly before i; run index of i = r (if it starts a run) else r - 1
    int r = cta_flag_rank(first, s_warp, nodes);
    if (i < npairs) {
      uint32_t pi = (uint32_t)(k & 0xFFFFFFFFull);
      int run = first ? r : r - 1;
      if (first) ty[run] = (double)ys[pi];
      if (last) tz[run] = (double)zs[pi];
    }
  }
  if (threadIdx.x == 0) P.n_nodes[s] = nodes;
}

// ---- SectPath pairing (variant B), fully parallel over band members ---------------------------
// One thread per band member m (any order inside a band).  A member with x > plane is a
// "left" query i of src/contour_alg.cpp:185-211: pr = NN_Er(pl); right_pair = NN_full(pr);
// pl' = NN_El(pr); left_pair = NN_full(pl'); node = interpolation of the pair onto the plane.
// The map insertion order of the reference is the ascending-index order of El, so the original
// index of the left query decides between equal-y nodes (k_slice_order).
struct PairParams {
  GridView g;
  GridView g3[3];                // multi-projection index: g3[choice[point]] is searched for that point
  const unsigned char* choice;   // nullptr: the single grid g
  const float4* xyz4;
  const float* planes;
  const float* lo;
  const float* hi;
  const int64_t* band_off;
  const int32_t* band_idx;
  int S;
  int64_t M;
  u64* keys;
  float* ys;
  float* zs;
  const uint32_t* member;   // optional membership bitmap (explicit index lists)
  int by_pos;               // band_idx holds SORTED POSITIONS (bands built from the cell-major order: members
                            // that are neighbours in the list are neighbours in space) instead of original indices
};

// Member m of the band lists as {original index, sorted position or -1} and its record.
__device__ __forceinline__ int2 member_handle(const PairParams& P, int64_t m, float4* rec) {
  const int e = __ldg(P.band_idx + m);
  if (P.by_pos) {
    *rec = __ldg(P.g.sorted + e);
    return make_int2(__float_as_int(rec->w), e);
  }
  *rec = __ldg(P.xyz4 + e);
  return make_int2(e, -1);
}

// Each warp takes PAIR_CHUNK consecutive members, keeps the left ones (about half) in a small
// shared-memory list and then works on that list with all lanes busy: a thread-per-member
// mapping leaves the lanes of right members idle during the long nearest-neighbour searches.
constexpr int PAIR_CHUNK = 56;   // ~28 left members per chunk: usually one full round of 32 lanes
constexpr int PAIR_WARPS = 4;

template <bool MEMBER>
__global__ void __launch_bounds__(PAIR_WARPS * 32) k_pair_nodes(PairParams P) {
  pdl_prologue();
  __shared__ int64_t s_m[PAIR_WARPS][64];
  __shared__ int s_s[PAIR_WARPS][64];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t base = ((int64_t)blockIdx.x * PAIR_WARPS + w) * PAIR_CHUNK;
  const int64_t M = __ldg(P.band_off + P.S);   // the launch may be sized from a host-side bound
  if (base >= M) return;
  int cnt = 0;
  for (int half = 0; half < 2; half++) {
    const int off = half * 32 + lane;
    const int64_t m = base + off;
    bool isL = false;
    int s = 0;
    if (off < PAIR_CHUNK && m < M) {
      // slice of member m: last s with band_off[s] <= m
      int l = 0, r = P.S;
      while (l < r) { int mid = (l + r) >> 1; if (__ldg(P.band_off + mid + 1) <= m) l = mid + 1; else r = mid; }
      s = l;
      float4 rec;
      member_handle(P, m, &rec);
      // index lists hold packed records, whose w = NaN marks a non-finite point (explicit lists only): neither side
      isL = (P.by_pos || rec.w == rec.w) && __fsub_rn(rec.x, __ldg(P.planes + s)) > 0.0f;
      if (!isL) { P.keys[m] = PPP_KEY_INF; P.ys[m] = 0.f; P.zs[m] = 0.f; }
    }
    const unsigned bal = __ballot_sync(0xffffffffu, isL);
    if (isL) {
      const int pos = cnt + __popc(bal & ((1u << lane) - 1u));
      s_m[w][pos] = m;
      s_s[w][pos] = s;
    }
    cnt += __popc(bal);
  }
  __syncwarp();
  for (int i = lane; i < cnt; i += 32) {
    const int64_t m = s_m[w][i];
    const int s = s_s[w][i];
    const float plane = __ldg(P.planes + s), lo = __ldg(P.lo + s), hi = __ldg(P.hi + s);
    const int64_t bo = __ldg(P.band_off + s);
    const int32_t* band = P.band_idx + bo;
    const int B = (int)(__ldg(P.band_off + s + 1) - bo);
    float4 pl;
    const int2 hq = member_handle(P, m, &pl);
    const GridView& gq = grid_for(P, hq.x);     // the left point's neighbourhood grid
    u64 key = PPP_KEY_INF;
    float y = 0.f, z = 0.f;
    const int2 ri = nn_side<MEMBER>(gq, P.xyz4, pl.x, pl.y, pl.z, lo, hi, plane, false, 0, band, B, P.member, P.by_pos);
    if (ri.x >= 0) {
      const float4 pr = rec_of(gq, P.xyz4, ri);
      const int2 rc = nn_full(gq, pr.x, pr.y, pr.z, ri);
      const GridView& gr = grid_for(P, ri.x);   // ... and the right point's
      const int2 li = nn_side<MEMBER>(gr, P.xyz4, pr.x, pr.y, pr.z, lo, hi, plane, true, 0, band, B, P.member, P.by_pos);
      const float4 pl2 = rec_of(gr, P.xyz4, li);
      const int2 lc = nn_full(gr, pl2.x, pl2.y, pl2.z, li);
      const float4 a = rec_of(gq, P.xyz4, rc);  // index_right
      const float4 b = rec_of(gr, P.xyz4, lc);  // index_left
      float t = __fdiv_rn(__fsub_rn(plane, a.x), __fsub_rn(b.x, a.x));
      y = __fadd_rn(a.y, __fmul_rn(t, __fsub_rn(b.y, a.y)));
      z = __fadd_rn(a.z, __fmul_rn(t, __fsub_rn(b.z, a.z)));
      // low word = slot inside the band (the payload address); equal-y ties are resolved by
      // original index in k_slice_order
      key = ((u64)f2ord_dev(__fadd_rn(y, 0.0f)) << 32) | (u64)(uint32_t)(m - bo);
    }
    P.keys[m] = key;
    P.ys[m] = y;
    P.zs[m] = z;
  }
}

// CTA per slice: sort the slice's node keys (INF = not a node) by (y, slot), then keep one node
// per distinct y with std::map semantics: the key of the FIRST insertion (lowest left index; only
// matters for -0.0 / +0.0) and the value of the LAST insertion (highest left index).
constexpr int SO_THREADS = 1024;

__device__ void slice_order_single(const int64_t* __restrict__ band_off, const int32_t* __restrict__ band_idx,
                                   const float4* __restrict__ sorted_if_pos, const u64* __restrict__ keys_g,
                                   const float* __restrict__ ys, const float* __restrict__ zs, u64* __restrict__ scratch,
                                   u64* s_keys64, int smem_cap, int skip_big, double* __restrict__ ty, double* __restrict__ tz,
                                   int32_t* __restrict__ n_nodes, int s, int* s_warp, int* s_valid_p) {
  const int64_t o = band_off[s];
  const int B = (int)(band_off[s + 1] - o);
  if (skip_big && B > smem_cap) return;   // left to the cluster kernel that follows (uniform over the block)
  u64* k = (B <= smem_cap) ? s_keys64 : (scratch + o);
  __syncthreads();
  if (threadIdx.x == 0) *s_valid_p = 0;
  __syncthreads();
  // keep only the node keys (left members that found a pair); their order does not matter yet
  for (int i = threadIdx.x; i < B; i += blockDim.x) {
    u64 key = keys_g[o + i];
    if (key != PPP_KEY_INF) {
      const int at = atomicAdd(s_valid_p, 1);
      PPP_DEV_ASSERT(at >= 0 && at < B && (k != s_keys64 || at < smem_cap));
      k[at] = key;
    }
  }
  __syncthreads();
  const int nv = *s_valid_p;
  cta_sort(k, nv);
  int nodes = 0;
  for (int base = 0; base < nv; base += blockDim.x) {
    int i = base + threadIdx.x;
    bool first = false;
    u64 key = 0;
    if (i < nv) {
      key = k[i];
      first = (i == 0) || ((k[i - 1] >> 32) != (key >> 32));
    }
    int r = cta_flag_rank(first, s_warp, nodes);
    if (first) {
      int slot = (int)(uint32_t)(key & 0xFFFFFFFFull);
      // original index of a member: the list entry itself, or (position lists) the w of its sorted record
      auto id_of = [&](int sl) {
        const int e = __ldg(band_idx + o + sl);
        return sorted_if_pos ? __float_as_int(__ldg(&sorted_if_pos[e].w)) : e;
      };
      int lo_idx = -1, hi_idx = -1, lo_slot = slot, hi_slot = slot;
      for (int j = i + 1; j < nv && (k[j] >> 32) == (key >> 32); j++) {
        if (lo_idx < 0) lo_idx = hi_idx = id_of(slot);   // ids are only needed when a y value repeats
        int sl = (int)(uint32_t)(k[j] & 0xFFFFFFFFull);
        int id = id_of(sl);
        if (id < lo_idx) { lo_idx = id; lo_slot = sl; }
        if (id > hi_idx) { hi_idx = id; hi_slot = sl; }
      }
      PPP_DEV_ASSERT(r >= 0 && r < B && lo_slot >= 0 && lo_slot < B && hi_slot >= 0 && hi_slot < B);
      ty[o + r] = (double)ys[o + lo_slot];
      tz[o + r] = (double)zs[o + hi_slot];
    }
  }
  if (threadIdx.x == 0) n_nodes[s] = nodes;
}

__global__ void __launch_bounds__(SO_THREADS) k_slice_order(const int64_t* __restrict__ band_off, const int32_t* __restrict__ band_idx,
                                                           const float4* __restrict__ sorted_if_pos,
                                                           const u64* __restrict__ keys_g, const float* __restrict__ ys,
                                                           const float* __restrict__ zs, u64* __restrict__ scratch,
                                                           int smem_cap, int skip_big, double* __restrict__ ty, double* __restrict__ tz,
                                                           int32_t* __restrict__ n_nodes) {
  pdl_prologue();
  extern __shared__ u64 s_keys64[];
  __shared__ int s_warp[32];
  __shared__ int s_valid;
  slice_order_single(band_off, band_idx, sorted_if_pos, keys_g, ys, zs, scratch, s_keys64, smem_cap, skip_big, ty, tz, n_nodes,
                     (int)blockIdx.x, s_warp, &s_valid);
}

// ---- the same, one thread-block CLUSTER per slice ------------------------------------------------------------
// For slices whose node keys do not fit one CTA's shared memory (the silhouette bands of a closed workpiece hold tens
// of thousands of members) and for sweeps with fewer slices than SMs (a rank's share of the planes at 8 GPUs): the C
// CTAs of a cluster each filter 1/C of the band, the keys go -- by distributed-shared-memory stores -- into ONE
// array spread over the C shared memories (chunk = np2 / C keys per CTA), and the bitonic network runs on it: every
// stage up to k = chunk and the j < chunk tail of the later stages stay inside a CTA (cta_sort / cta_jsteps), the
// few remaining steps exchange across CTAs through DSMEM with a cluster barrier each (C = 4: 3 + 2 + 1 of them).
// The map-order pass reads its left neighbour and the tail of equal-y runs across the CTA boundary the same way.
// A slice too large even for C x SOC_CHUNK_MAX keys is sorted by CTA 0 in global scratch like before.
constexpr int SOC_CHUNK_MAX = 16384;   // keys per CTA: 128 KB

template <int C>
__global__ void __cluster_dims__(C, 1, 1) __launch_bounds__(SO_THREADS, 1)
k_slice_order_cl(const int64_t* __restrict__ band_off, const int32_t* __restrict__ band_idx, const float4* __restrict__ sorted_if_pos,
                 const u64* __restrict__ keys_g, const float* __restrict__ ys, const float* __restrict__ zs, u64* __restrict__ scratch,
                 int chunk_cap, int S, int min_B, int max_B, double* __restrict__ ty, double* __restrict__ tz,
                 int32_t* __restrict__ n_nodes) {
  pdl_prologue();
  extern __shared__ u64 s_arr[];     // this CTA's chunk of the slice's distributed key array
  __shared__ int s_warp[32];
  __shared__ int s_cnt, s_fill, s_first;
  cg::cluster_group cl = cg::this_cluster();
  const int r = (int)cl.block_rank();
  const int nt = blockDim.x;
  // the clusters of the grid share the slices whose band size lies in (min_B, max_B]; every test below that decides
  // the control flow depends on the slice alone, so the CTAs of a cluster stay together
  for (int s = blockIdx.x / C; s < S; s += gridDim.x / C) {
  const int64_t o = band_off[s];
  const int B = (int)(band_off[s + 1] - o);
  if (B <= min_B || B > max_B) continue;
  const int seg = (B + C - 1) / C;
  const int b0 = min(r * seg, B), b1 = min(b0 + seg, B);   // my part of the band
  if (threadIdx.x == 0) { s_cnt = 0; s_fill = 0; s_first = 0; }
  __syncthreads();
  int mine = 0;
  for (int i = b0 + threadIdx.x; i < b1; i += nt) mine += keys_g[o + i] != PPP_KEY_INF ? 1 : 0;
  mine = __reduce_add_sync(0xffffffffu, mine);
  if ((threadIdx.x & 31) == 0 && mine) atomicAdd(&s_cnt, mine);
  cl.sync();
  int nv = 0, before = 0;
#pragma unroll
  for (int q = 0; q < C; q++) {
    const int cq = *cl.map_shared_rank(&s_cnt, q);
    if (q < r) before += cq;
    nv += cq;
  }
  int np2 = 2;
  while (np2 < nv) np2 <<= 1;
  const int chunk = max(np2 / C, 64);    // keys per CTA, a power of two
  if (chunk > chunk_cap) {               // uniform over the cluster: CTA 0 takes the slice alone, in global scratch
    cl.sync();                           // ... once nobody reads this CTA's counters any more
    if (r == 0) slice_order_single(band_off, band_idx, sorted_if_pos, keys_g, ys, zs, scratch, s_arr, 0, 0, ty, tz, n_nodes, s, s_warp, &s_cnt);
    continue;                            // (the others wait for it at the next slice's first cluster barrier)
  }
  const int csh = 31 - __clz(chunk);
  auto elem = [&](int g) -> u64* {
    PPP_DEV_ASSERT(g >= 0 && (g >> csh) < C && chunk <= chunk_cap);
    return cl.map_shared_rank(s_arr, g >> csh) + (g & (chunk - 1));
  };
  // the node keys (left members that found a pair) -> their place in the distributed array; order inside is arbitrary
  for (int i = b0 + threadIdx.x; i < b1; i += nt) {
    const u64 key = keys_g[o + i];
    if (key != PPP_KEY_INF) *elem(before + atomicAdd(&s_fill, 1)) = key;
  }
  cl.sync();
  const int base = r * chunk;
  const int n_loc = max(0, min(nv - base, chunk));
  cta_sort(s_arr, n_loc);
  cl.sync();
  const int half = np2 >> 1;
  const int c_lo = r * (chunk >> 1), c_hi = min((r + 1) * (chunk >> 1), half);   // this CTA's comparators of a cross step
  for (int k = 2 * chunk; k <= np2; k <<= 1) {
    const int hk = k >> 1;
    for (int c = c_lo + threadIdx.x; c < c_hi; c += nt) {
      const int b = c / hk, oo = c - b * hk, i = b * k + oo, l = b * k + (k - 1 - oo);
      if (l < nv) { u64* pi = elem(i); u64* pl = elem(l); const u64 x = *pi, y = *pl; if (y < x) { *pi = y; *pl = x; } }
    }
    cl.sync();
    for (int j = k >> 2; j >= chunk; j >>= 1) {
      for (int c = c_lo + threadIdx.x; c < c_hi; c += nt) {
        const int i = 2 * c - (c & (j - 1)), l = i + j;
        if (l < nv) { u64* pi = elem(i); u64* pl = elem(l); const u64 x = *pi, y = *pl; if (y < x) { *pi = y; *pl = x; } }
      }
      cl.sync();
    }
    cta_jsteps(s_arr, n_loc, chunk >> 1, chunk >> 1);
    cl.sync();
  }
  // std::map order: one node per distinct y, key of the first insertion, value of the last (see k_slice_order)
  int firsts = 0;
  for (int il = threadIdx.x; il < n_loc; il += nt) {
    const int g = base + il;
    firsts += (g == 0 || ((*elem(g - 1)) >> 32) != (s_arr[il] >> 32)) ? 1 : 0;
  }
  firsts = __reduce_add_sync(0xffffffffu, firsts);
  if ((threadIdx.x & 31) == 0 && firsts) atomicAdd(&s_first, firsts);
  cl.sync();
  int nodes = 0, total = 0;
#pragma unroll
  for (int q = 0; q < C; q++) {
    const int fq = *cl.map_shared_rank(&s_first, q);
    if (q < r) nodes += fq;
    total += fq;
  }
  for (int bt = 0; bt < n_loc; bt += nt) {
    const int il = bt + threadIdx.x;
    const int g = base + il;
    bool first = false;
    u64 key = 0;
    if (il < n_loc) {
      key = s_arr[il];
      first = g == 0 || ((*elem(g - 1)) >> 32) != (key >> 32);
    }
    const int rnk = cta_flag_rank(first, s_warp, nodes);
    if (first) {
      const int slot = (int)(uint32_t)(key & 0xFFFFFFFFull);
      auto id_of = [&](int sl) {
        const int e = __ldg(band_idx + o + sl);
        return sorted_if_pos ? __float_as_int(__ldg(&sorted_if_pos[e].w)) : e;
      };
      int lo_idx = -1, hi_idx = -1, lo_slot = slot, hi_slot = slot;
      for (int j = g + 1; j < nv; j++) {
        const u64 kj = *elem(j);
        if ((kj >> 32) != (key >> 32)) break;
        if (lo_idx < 0) lo_idx = hi_idx = id_of(slot);   // ids are only needed when a y value repeats
        const int sl = (int)(uint32_t)(kj & 0xFFFFFFFFull);
        const int id = id_of(sl);
        if (id < lo_idx) { lo_idx = id; lo_slot = sl; }
        if (id > hi_idx) { hi_idx = id; hi_slot = sl; }
      }
      PPP_DEV_ASSERT(rnk >= 0 && rnk < B && lo_slot >= 0 && lo_slot < B && hi_slot >= 0 && hi_slot < B);
      ty[o + rnk] = (double)ys[o + lo_slot];
      tz[o + rnk] = (double)zs[o + hi_slot];
    }
  }
  if (r == 0 && threadIdx.x == 0) n_nodes[s] = total;
  cl.sync();   // no CTA leaves (or starts the next slice) while a neighbour may still read its shared memory
  }
}

__global__ void k_set_member_bits(const int32_t* __restrict__ idx, int64_t m, uint32_t* __restrict__ bits) {
  pdl_prologue();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) atomicOr(bits + (idx[i] >> 5), 1u << (idx[i] & 31));
}

__global__ void __launch_bounds__(256) k_compact_nodes(const int64_t* __restrict__ band_off, const int64_t* __restrict__ node_off,
                                                      const float* __restrict__ planes, const double* __restrict__ ty,
                                                      const double* __restrict__ tz, double* __restrict__ y,
                                                      double* __restrict__ x, double* __restrict__ z) {
  pdl_prologue();
  int s = blockIdx.x;
  int64_t so = band_off[s], d = node_off[s];
  int n = (int)(node_off[s + 1] - d);
  double px = (double)planes[s];
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    y[d + i] = ty[so + i];
    x[d + i] = px;
    z[d + i] = tz[so + i];
  }
}

// Sync-free variant: the host does not know the node total when it launches this, so the kernel
// itself picks the destination (caller's buffers if the total fits, else the cloud's) and leaves
// {node total, band members, largest band, used caller's buffers} for one fetch at the very end.
struct NodeDest {
  double *ey, *ex, *ez; int64_t ecap;   // caller-owned (may be page-locked host memory), optional
  double *oy, *ox, *oz;                 // cloud-owned, large enough for any total
  int64_t* ext_off; int64_t ext_off_cap;
};

// n_nodes != nullptr: the node offsets are not known yet -- every block sums the node counts of the slices before its
// own (and all of them) itself and stores its entry of node_off: for the few hundred to few thousand slices of a
// sweep that is cheaper than one more launch in a chain whose every launch waits for a free SM slot.
__global__ void __launch_bounds__(256) k_compact_nodes_auto(const int64_t* __restrict__ band_off, int64_t* __restrict__ node_off,
                                                           const int32_t* __restrict__ n_nodes,
                                                           int S, const float* __restrict__ planes, const double* __restrict__ ty,
                                                           const double* __restrict__ tz, NodeDest D, int64_t* __restrict__ summary,
                                                           unsigned* __restrict__ host_out, unsigned* __restrict__ host_flag, unsigned seq) {
  pdl_prologue();
  __shared__ bool s_last;
  __shared__ long long s_sum[2][8];
  const int s = blockIdx.x;
  int64_t total, d;
  int n;
  if (n_nodes) {
    long long before = 0, all = 0;
    for (int t = threadIdx.x; t < S; t += blockDim.x) {
      const long long v = n_nodes[t];
      all += v;
      if (t < s) before += v;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      before += __shfl_xor_sync(0xffffffffu, before, o);
      all += __shfl_xor_sync(0xffffffffu, all, o);
    }
    if ((threadIdx.x & 31) == 0) { s_sum[0][threadIdx.x >> 5] = before; s_sum[1][threadIdx.x >> 5] = all; }
    __syncthreads();
    before = 0; all = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) { before += s_sum[0][w]; all += s_sum[1][w]; }
    d = before; total = all; n = n_nodes[s];
    if (threadIdx.x == 0) {
      node_off[s] = d;
      if (s == S - 1) node_off[S] = total;
    }
  } else {
    total = node_off[S];
    d = node_off[s];
    n = (int)(node_off[s + 1] - d);
  }
  const bool ext = D.ey && total <= D.ecap;
  double* y = ext ? D.ey : D.oy; double* x = ext ? D.ex : D.ox; double* z = ext ? D.ez : D.oz;
  const int64_t so = band_off[s];
  const double px = (double)planes[s];
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    y[d + i] = ty[so + i];
    x[d + i] = px;
    z[d + i] = tz[so + i];
  }
  if (D.ext_off && D.ext_off_cap >= (int64_t)S + 1) {
    if (threadIdx.x == 0) D.ext_off[s] = d;
    if (threadIdx.x == 1 && s == S - 1) D.ext_off[S] = total;
  }
  if (threadIdx.x == 0) {
    atomicMax((unsigned long long*)(summary + 2), (unsigned long long)(band_off[s + 1] - so));
    if (s == 0) { summary[0] = total; summary[1] = band_off[S]; summary[3] = ext ? 1 : 0; }
  }
  if (!host_out) return;
  // The last block to finish hands the summary to the host itself (mapped memory + flag, as cloud_ingest does): no
  // fetch kernel at the end of the chain.  Node stores may go to page-locked host memory: system-scope fence in every block.
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd((unsigned long long*)(summary + 4), 1ull) == (unsigned long long)gridDim.x - 1ull;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  if (threadIdx.x < 8) host_out[threadIdx.x] = ((const volatile unsigned*)summary)[threadIdx.x];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) *(volatile unsigned*)host_flag = seq;
}

}  // namespace

static void band_limits_host(float plane_x, float half_width, int truncate_center, float* lo, float* hi) {
  if (truncate_center) {
    int position = (int)plane_x;  // rangedX_index(int position) receives the float plane x
    int hw = (int)half_width;
    *lo = (float)(-hw + position);
    *hi = (float)(hw + position);
  } else {
    *lo = plane_x - half_width;
    *hi = plane_x + half_width;
  }
}

// Host staging + counting pass shared by the two band builders: limits per plane, planes sorted by
// lower limit, upload, k_band_count, exclusive scan.  Leaves counts zeroed for the fill pass.
struct BandPrep {
  float* fdev = nullptr;      // [planes S][lo S][hi S][lo_sorted S][hi_sorted S]
  int32_t* pdev = nullptr;    // sorted position -> plane
  int32_t* counts = nullptr;  // S
  int64_t* offsets = nullptr; // S + 1
  BandSet b{};
  int Sv = 0, use_smem = 0;
  unsigned blocks = 1;
  int64_t chunk = 0;
  int max_depth = 0;          // most bands any single x can belong to
  float max_width = 0.f;      // widest band (hi - lo)
  const float4* src = nullptr;  // records the bands are drawn from: the packed cloud (entries = original indices) ...
  int64_t n_src = 0;            // ... or the cell-major sorted array of a grid (entries = sorted positions)
  int w_is_flag = 1;
};

static int bands_prepare(ppp_cloud* c, const float* plane_x_host, int S, float half_width, int truncate_center, BandPrep* bp,
                         const GridStore* by_pos_of = nullptr) {
  ppp_ctx* ctx = c->ctx;
  bp->src = by_pos_of ? by_pos_of->v.sorted : c->xyz4;
  bp->n_src = by_pos_of ? (int64_t)by_pos_of->v.n_sorted : c->n;
  bp->w_is_flag = by_pos_of ? 0 : 1;
  std::vector<float> lo(S), hi(S);
  std::vector<int32_t> perm(S);
  for (int s = 0; s < S; s++) {
    if (std::isfinite(plane_x_host[s]) && std::fabs(plane_x_host[s]) < 2.0e9f) band_limits_host(plane_x_host[s], half_width, truncate_center, &lo[s], &hi[s]);
    else lo[s] = hi[s] = NAN;
    perm[s] = s;
  }
  std::stable_sort(perm.begin(), perm.end(), [&](int a, int b) {
    bool na = std::isnan(lo[a]), nb = std::isnan(lo[b]);
    if (na != nb) return nb;
    if (na) return false;
    return lo[a] < lo[b];
  });
  // host staging: [planes S][lo S][hi S][lo_sorted S][hi_sorted S] + perm
  std::vector<float> stage(5 * (size_t)S);
  int Sv = 0;  // sorted entries with valid limits
  for (int s = 0; s < S; s++) {
    stage[s] = plane_x_host[s];
    stage[S + s] = lo[s];
    stage[2 * S + s] = hi[s];
  }
  for (int t = 0; t < S; t++) {
    int s = perm[t];
    if (!std::isnan(lo[s])) { Sv = t + 1; bp->max_width = std::max(bp->max_width, hi[s] - lo[s]); }
    stage[3 * S + t] = lo[s];
    stage[4 * S + t] = hi[s];
  }
  {  // overlap depth of the closed intervals [lo, hi], taken in ascending lo
    std::vector<float> ends;  // min-heap of the upper limits still open
    int depth = 0;
    for (int t = 0; t < Sv; t++) {
      const float l = stage[3 * S + t], h = stage[4 * S + t];
      while (!ends.empty() && ends.front() < l) { std::pop_heap(ends.begin(), ends.end(), std::greater<float>()); ends.pop_back(); }
      ends.push_back(h); std::push_heap(ends.begin(), ends.end(), std::greater<float>());
      depth = std::max(depth, (int)ends.size());
    }
    bp->max_depth = depth;
  }
  PPP_TRY(dev_alloc(ctx, &bp->fdev, 5 * (size_t)std::max(S, 1)));
  PPP_TRY(dev_alloc(ctx, &bp->pdev, (size_t)std::max(S, 1)));
  PPP_TRY(dev_alloc(ctx, &bp->counts, (size_t)S + 1));     // [S]: the count kernel's ticket
  PPP_TRY(dev_alloc(ctx, &bp->offsets, (size_t)S + 1));
  PPP_CUDA(cudaMemsetAsync(bp->counts, 0, ((size_t)S + 1) * sizeof(int32_t), ctx->stream));
  if (S > 0) {
    // pageable sources: the runtime stages them before returning, so the vectors may go out of scope
    PPP_CUDA(cudaMemcpyAsync(bp->fdev, stage.data(), stage.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    PPP_CUDA(cudaMemcpyAsync(bp->pdev, perm.data(), (size_t)S * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
  }
  bp->b = BandSet{bp->fdev + 3 * (size_t)S, bp->fdev + 4 * (size_t)S, bp->pdev, Sv, 0, 0.f, 0.f, 0.f};
  if (Sv >= 8 && !getenv("PPP_BANDS_SEARCH")) {   // constant pitch?  (PPP_BANDS_SEARCH: always the binary searches)
    const float* slo = stage.data() + 3 * (size_t)S;
    const float* shi = stage.data() + 4 * (size_t)S;
    const double pitch = ((double)slo[Sv - 1] - (double)slo[0]) / (double)(Sv - 1);
    bool ok = pitch > 0 && std::isfinite(pitch);
    for (int t = 0; ok && t < Sv; t++) {
      ok = std::fabs((double)slo[t] - ((double)slo[0] + t * pitch)) <= 0.25 * pitch &&
           std::fabs((double)shi[t] - ((double)shi[0] + t * pitch)) <= 0.25 * pitch;
    }
    if (ok) { bp->b.regular = 1; bp->b.lo0 = slo[0]; bp->b.hi0 = shi[0]; bp->b.inv_pitch = (float)(1.0 / pitch); }
  }
  bp->Sv = Sv;
  bp->use_smem = Sv <= BAND_SMEM_BINS / 2;  // fill needs two arrays
  bp->blocks = (unsigned)std::max<int64_t>(1, std::min<int64_t>((bp->n_src + 1023) / 1024, (int64_t)ctx->sm_count * 8));
  bp->chunk = (bp->n_src + bp->blocks - 1) / bp->blocks;
  if (bp->n_src > 0 && Sv > 0) {
    // the kernel's last block also scans the counts into the offsets and zeroes them for the fill pass
    PPP_LAUNCH(ctx, "band_count", k_band_count, bp->blocks, 256, bp->use_smem ? (size_t)Sv * 4 : 0, bp->b, bp->src,
               bp->n_src, bp->chunk, bp->use_smem, bp->w_is_flag, bp->counts, S, (int64_t*)bp->offsets);
    PPP_CHECK_LAUNCH();
    return PPP_OK;
  }
  PPP_TRY(scan_exclusive_i32_to_i64(ctx, bp->counts, bp->offsets, S));   // no points or no valid plane: all zero
  return PPP_OK;
}

static int bands_fill(ppp_cloud* c, const BandPrep& bp, int32_t* idx) {
  ppp_ctx* ctx = c->ctx;
  if (bp.n_src <= 0 || bp.Sv <= 0) return PPP_OK;
  if (bp.use_smem) PPP_CUDA(cudaFuncSetAttribute(k_band_fill, cudaFuncAttributeMaxDynamicSharedMemorySize, BAND_SMEM_BINS * 4));
  PPP_LAUNCH(ctx, "band_fill", k_band_fill, bp.blocks, 256, bp.use_smem ? (size_t)bp.Sv * 8 : 0, bp.b, bp.src, bp.n_src,
             bp.chunk, bp.use_smem, bp.w_is_flag, bp.counts, (const int64_t*)bp.offsets, idx);
  PPP_CHECK_LAUNCH();
  return PPP_OK;
}

// Device arrays produced: offsets (S+1, int64), idx (total), planes/lo/hi (3*S floats, original
// order).  sort_bands != 0: every band in ascending point index (PassThrough order).
int bands_launch(ppp_cloud* c, const float* plane_x_host, int S, float half_width, int truncate_center, int sort_bands,
                 int64_t** offsets_dev_out, int32_t** idx_dev_out, int64_t* total_out, float** planes_dev_out,
                 std::vector<int64_t>* offsets_host_out) {
  ppp_ctx* ctx = c->ctx;
  *offsets_dev_out = nullptr; *idx_dev_out = nullptr; *planes_dev_out = nullptr; *total_out = 0;
  BandPrep bp;
  PPP_TRY(bands_prepare(c, plane_x_host, S, half_width, truncate_center, &bp));
  int64_t* offsets = bp.offsets;
  std::vector<int64_t> off_h((size_t)S + 1, 0);
  PPP_TRY(fetch_small(ctx, offsets, ((size_t)S + 1) * sizeof(int64_t), off_h.data()));
  int64_t total = off_h[S];
  int32_t* idx = nullptr;
  PPP_TRY(dev_alloc(ctx, &idx, (size_t)std::max<int64_t>(total, 1)));
  if (total > 0) {
    PPP_TRY(bands_fill(c, bp, idx));
    if (sort_bands) {
      int64_t maxB = 0;
      for (int s = 0; s < S; s++) maxB = std::max(maxB, off_h[s + 1] - off_h[s]);
      int smem_cap = (int)std::min<int64_t>(std::max<int64_t>(maxB, 1), 49152);  // <= 192 KB of int32
      if (smem_cap * 4 > 40 * 1024)
        PPP_CUDA(cudaFuncSetAttribute(k_band_sort, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_cap * 4));
      PPP_LAUNCH(ctx, "band_sort", k_band_sort, (unsigned)S, 1024, (size_t)smem_cap * 4, (const int64_t*)offsets, idx,
                 smem_cap);
      PPP_CHECK_LAUNCH();
    }
  }
  dev_free(ctx, bp.counts);
  dev_free(ctx, bp.pdev);
  *offsets_dev_out = offsets;
  *idx_dev_out = idx;
  *planes_dev_out = bp.fdev;  // [planes][lo][hi] in original order (+ sorted copies behind)
  *total_out = total;
  if (offsets_host_out) *offsets_host_out = std::move(off_h);
  return PPP_OK;
}

// Orders the nodes of every slice, in two launches that split the slices by band size:
//   1. one CTA per slice (k_slice_order) -- or, when a sweep has at most half as many slices as the GPU has SMs, a
//      cluster of 2 / 4 / 8 CTAs per slice -- for the bands up to cap1 members, sized from `band_est`;
//   2. a few persistent clusters of 8 CTAs (k_slice_order_cl<8>, 128 KB of keys per CTA) for the bands beyond cap1:
//      the silhouette bands of a closed workpiece, a flat face parallel to the planes.  Only launched when such bands
//      are to be expected (`expect_big`, or an estimate beyond cap1); otherwise the first launch sorts a band that
//      does exceed cap1 after all in `scratch` (slow, but an empty second launch costs every sweep ~5 us).
// `scratch` (M keys) also takes what even a cluster cannot hold (> 131072 node keys in one slice).
static int launch_slice_order(ppp_ctx* ctx, int S, int64_t band_est, bool expect_big, const int64_t* band_off, const int32_t* band_idx,
                              const float4* sorted_if_pos, const u64* keys, const float* ys, const float* zs, u64* scratch,
                              double* ty, double* tz, int32_t* n_nodes) {
  if (S <= 0) return PPP_OK;
  band_est = std::max<int64_t>(band_est, 1);
  int C = 1;
  // clusters pay while all of them fit the GPU at once (measured, slices x members -> best C: 25 x 4k -> 4, 71 x 11k -> 2,
  // 100 x 5.6k -> 1, 141 x 5.6k -> 1): the largest C with S * C CTAs on the SMs in one wave
  if (band_est >= 4096 && band_est <= 4 * (int64_t)SOC_CHUNK_MAX)
    while (C < 8 && S * C * 2 <= ctx->sm_count) C *= 2;
  if (const char* e = getenv("PPP_SLICE_CLUSTER")) {   // tuning / test aid: first launch with clusters of 1 / 2 / 4 / 8
    const int v = atoi(e);
    if (v == 1 || v == 2 || v == 4 || v == 8) C = v;
  }
  int64_t np2 = 1;
  while (np2 < band_est) np2 <<= 1;
  const int smem_cap = (int)std::min<int64_t>(std::max<int64_t>(band_est, 1024), 24576);  // C == 1: <= 192 KB of u64
  const int chunk_cap = (int)std::min<int64_t>(std::max<int64_t>(np2 / C, 1024), SOC_CHUNK_MAX);
  const int64_t cap1 = C == 1 ? (int64_t)smem_cap : (int64_t)chunk_cap * C;
  const bool big = expect_big || band_est > cap1;   // a second launch takes the bands beyond cap1
  if (C == 1) {
    if ((size_t)smem_cap * 8 > 40 * 1024)
      PPP_CUDA(cudaFuncSetAttribute(k_slice_order, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_cap * 8));
    // short bands: 256 threads sort them with a quarter of the barrier traffic, and more slices share an SM
    const int so_threads = smem_cap <= 4608 ? 256 : SO_THREADS;
    PPP_LAUNCH(ctx, "slice_order", k_slice_order, (unsigned)S, so_threads, (size_t)smem_cap * 8, band_off, band_idx, sorted_if_pos,
               keys, ys, zs, scratch, smem_cap, big ? 1 : 0, ty, tz, n_nodes);
    PPP_CHECK_LAUNCH();
  } else {
    const int max_B = big ? (int)cap1 : 2147483647;
    const size_t smem = (size_t)chunk_cap * 8;
    const unsigned grid = (unsigned)S * (unsigned)C;
    if (C == 2) {
      auto kern = k_slice_order_cl<2>;
      if (smem > 40 * 1024) PPP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      PPP_LAUNCH(ctx, "slice_order", kern, grid, SO_THREADS, smem, band_off, band_idx, sorted_if_pos, keys, ys, zs, scratch, chunk_cap, S, -1, max_B, ty, tz, n_nodes);
    } else if (C == 4) {
      auto kern = k_slice_order_cl<4>;
      if (smem > 40 * 1024) PPP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      PPP_LAUNCH(ctx, "slice_order", kern, grid, SO_THREADS, smem, band_off, band_idx, sorted_if_pos, keys, ys, zs, scratch, chunk_cap, S, -1, max_B, ty, tz, n_nodes);
    } else {
      auto kern = k_slice_order_cl<8>;
      if (smem > 40 * 1024) PPP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      PPP_LAUNCH(ctx, "slice_order", kern, grid, SO_THREADS, smem, band_off, band_idx, sorted_if_pos, keys, ys, zs, scratch, chunk_cap, S, -1, max_B, ty, tz, n_nodes);
    }
    PPP_CHECK_LAUNCH();
  }
  if (!big) return PPP_OK;
  // the bands beyond cap1
  auto kern = k_slice_order_cl<8>;
  const size_t smem = (size_t)SOC_CHUNK_MAX * 8;
  PPP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const unsigned clusters = (unsigned)std::min(S, 16);
  PPP_LAUNCH(ctx, "slice_order_big", kern, clusters * 8u, SO_THREADS, smem, band_off, band_idx, sorted_if_pos, keys, ys, zs, scratch,
             SOC_CHUNK_MAX, S, (int)cap1, 2147483647, ty, tz, n_nodes);
  PPP_CHECK_LAUNCH();
  return PPP_OK;
}

static int finish_nodes(ppp_cloud* c, int S, const int64_t* band_off_dev, const float* planes_dev, const int32_t* n_nodes,
                        const double* ty, const double* tz, int64_t* total_nodes_out) {
  ppp_ctx* ctx = c->ctx;
  if (c->c_S_cap < S + 1) {
    dev_free(ctx, c->c_node_off);
    PPP_TRY(dev_alloc_keep(ctx, &c->c_node_off, (size_t)S + 1));
    c->c_S_cap = S + 1;
  }
  PPP_TRY(scan_exclusive_i32_to_i64(ctx, n_nodes, c->c_node_off, S));
  int64_t total = 0;
  PPP_TRY(fetch_small(ctx, c->c_node_off + S, sizeof(int64_t), &total));
  // caller-provided device buffers (ppp_dev_set_contour_buffers) take the nodes when they are large
  // enough; otherwise the cloud-owned buffers are (re)allocated
  const bool ext = c->ext_y && c->ext_cap >= total;
  if (!ext && (c->c_cap < total || !c->c_y)) {
    dev_free(ctx, c->c_y); dev_free(ctx, c->c_x); dev_free(ctx, c->c_z);
    size_t cap = (size_t)std::max<int64_t>(total, 1);
    PPP_TRY(dev_alloc_keep(ctx, &c->c_y, cap)); PPP_TRY(dev_alloc_keep(ctx, &c->c_x, cap)); PPP_TRY(dev_alloc_keep(ctx, &c->c_z, cap));
    c->c_cap = (int64_t)cap;
  }
  if (c->ext_off && c->ext_off_cap >= (int64_t)S + 1)   // per-slice node offsets for a remote consumer
    PPP_CUDA(cudaMemcpyAsync(c->ext_off, c->c_node_off, ((size_t)S + 1) * sizeof(int64_t), cudaMemcpyDefault, ctx->stream));
  c->out_y = ext ? c->ext_y : c->c_y;
  c->out_x = ext ? c->ext_x : c->c_x;
  c->out_z = ext ? c->ext_z : c->c_z;
  if (total > 0) {
    PPP_LAUNCH(ctx, "compact_nodes", k_compact_nodes, (unsigned)S, 256, 0, band_off_dev, (const int64_t*)c->c_node_off,
               planes_dev, ty, tz, c->out_y, c->out_x, c->out_z);
    PPP_CHECK_LAUNCH();
  }
  *total_nodes_out = total;
  return PPP_OK;
}

// band_off_host: S+1 offsets (for sizing shared memory).  Variant A needs index-sorted bands.
template <typename PARAMS>
static void set_grids(PARAMS& P, const GridStore& gs, const MPSet* mp) {
  P.g = gs.v;
  P.choice = mp ? mp->choice : nullptr;
  for (int p = 0; p < 3; p++) P.g3[p] = mp ? mp->g[p]->v : gs.v;
}

int contours_launch(ppp_cloud* c, const GridStore& gs, const float* planes_dev, int S, const int64_t* band_off_dev,
                    const int32_t* band_idx_dev, int64_t band_total, const std::vector<int64_t>& band_off_host, int mode,
                    int64_t* total_nodes_out, const uint32_t* member_bits, const MPSet* mp) {
  ppp_ctx* ctx = c->ctx;
  *total_nodes_out = 0;
  size_t M = (size_t)std::max<int64_t>(band_total, 1);
  double *ty = nullptr, *tz = nullptr;
  int32_t* n_nodes = nullptr;
  PPP_TRY(dev_alloc(ctx, &ty, M)); PPP_TRY(dev_alloc(ctx, &tz, M));
  PPP_TRY(dev_alloc(ctx, &n_nodes, (size_t)std::max(S, 1)));
  int st = PPP_OK;
  if (mode == PPP_PAIR_SECT) {
    PairParams P{};
    set_grids(P, gs, mp); P.xyz4 = c->xyz4;
    P.planes = planes_dev; P.lo = planes_dev + S; P.hi = planes_dev + 2 * (size_t)S;
    P.band_off = band_off_dev; P.band_idx = band_idx_dev; P.S = S; P.M = band_total;
    P.member = member_bits; P.by_pos = 0;
    PPP_TRY(dev_alloc(ctx, &P.keys, M)); PPP_TRY(dev_alloc(ctx, &P.ys, M)); PPP_TRY(dev_alloc(ctx, &P.zs, M));
    if (band_total > 0) {
      const int64_t per_block = (int64_t)PAIR_WARPS * PAIR_CHUNK;
      auto kern = member_bits ? k_pair_nodes<true> : k_pair_nodes<false>;
      PPP_LAUNCH(ctx, "pair_nodes", kern, (unsigned)((band_total + per_block - 1) / per_block), PAIR_WARPS * 32, 0, P);
      PPP_CHECK_LAUNCH();
    }
    int64_t maxB = 0;
    for (int s = 0; s < S; s++) maxB = std::max(maxB, band_off_host[s + 1] - band_off_host[s]);
    u64* scratch = nullptr;
    if (maxB > 24576) PPP_TRY(dev_alloc(ctx, &scratch, M));   // slices beyond every shared-memory path
    PPP_TRY(launch_slice_order(ctx, S, maxB, false, band_off_dev, band_idx_dev, (const float4*)nullptr, (const u64*)P.keys, (const float*)P.ys,
                               (const float*)P.zs, scratch, ty, tz, n_nodes));
    st = finish_nodes(c, S, band_off_dev, planes_dev, n_nodes, ty, tz, total_nodes_out);
    dev_free(ctx, P.keys); dev_free(ctx, P.ys); dev_free(ctx, P.zs); dev_free(ctx, scratch);
  } else {
    ContourParams P{};
    set_grids(P, gs, mp); P.xyz4 = c->xyz4;
    P.planes = planes_dev; P.lo = planes_dev + S; P.hi = planes_dev + 2 * (size_t)S;
    P.band_off = band_off_dev; P.band_idx = band_idx_dev; P.mode = mode;
    P.ty = ty; P.tz = tz; P.n_nodes = n_nodes;
    P.member = member_bits;
    PPP_TRY(dev_alloc(ctx, &P.El, M)); PPP_TRY(dev_alloc(ctx, &P.Er, M));
    PPP_TRY(dev_alloc(ctx, &P.keys, M));
    PPP_TRY(dev_alloc(ctx, &P.ys, M)); PPP_TRY(dev_alloc(ctx, &P.zs, M));
    PPP_TRY(dev_alloc(ctx, &P.lp, M)); PPP_TRY(dev_alloc(ctx, &P.rp, M));
    PPP_TRY(dev_alloc(ctx, &P.posR, M)); PPP_TRY(dev_alloc(ctx, &P.posL, M));
    PPP_TRY(dev_alloc(ctx, &P.fl, M)); PPP_TRY(dev_alloc(ctx, &P.fr, M));
    if (S > 0) {
      int64_t maxB = 0;
      for (int s = 0; s < S; s++) maxB = std::max(maxB, band_off_host[s + 1] - band_off_host[s]);
      int smem_cap = (int)std::min<int64_t>(std::max<int64_t>(maxB, 2), 22000);  // 9 bytes per member, <= 198 KB
      size_t smem = 9 * (size_t)((smem_cap + 1) & ~1) + 16;
      auto kern = member_bits ? k_contour<true> : k_contour<false>;
      if (smem > 40 * 1024) PPP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      PPP_LAUNCH(ctx, "contour_gen2", kern, (unsigned)S, 1024, smem, P, smem_cap);
      PPP_CHECK_LAUNCH();
    }
    st = finish_nodes(c, S, band_off_dev, planes_dev, n_nodes, ty, tz, total_nodes_out);
    dev_free(ctx, P.El); dev_free(ctx, P.Er); dev_free(ctx, P.keys); dev_free(ctx, P.ys); dev_free(ctx, P.zs);
    dev_free(ctx, P.lp); dev_free(ctx, P.rp); dev_free(ctx, P.posR); dev_free(ctx, P.posL); dev_free(ctx, P.fl);
    dev_free(ctx, P.fr);
  }
  dev_free(ctx, ty); dev_free(ctx, tz); dev_free(ctx, n_nodes);
  return st;
}

// insert_point(indices, PlanePoint) with an EXPLICIT index list (ascending, as rangedX_index
// returns it): one slice whose members are exactly `indices`; membership tests use a bitmap
// instead of the band's x-interval.
int contours_from_indices_launch(ppp_cloud* c, const GridStore& gs, const int32_t* idx_host, int64_t m, float plane_x,
                                 int mode, int64_t* total_nodes_out, const MPSet* mp) {
  ppp_ctx* ctx = c->ctx;
  *total_nodes_out = 0;
  float stage[3] = {plane_x, -INFINITY, INFINITY};
  int64_t off_h[2] = {0, m};
  float* planes = nullptr; int64_t* boff = nullptr; int32_t* bidx = nullptr; uint32_t* bits = nullptr;
  size_t words = (size_t)(c->n + 31) / 32 + 1;
  PPP_TRY(dev_alloc(ctx, &planes, 3)); PPP_TRY(dev_alloc(ctx, &boff, 2));
  PPP_TRY(dev_alloc(ctx, &bidx, (size_t)std::max<int64_t>(m, 1))); PPP_TRY(dev_alloc(ctx, &bits, words));
  PPP_CUDA(cudaMemcpyAsync(planes, stage, sizeof(stage), cudaMemcpyHostToDevice, ctx->stream));
  PPP_CUDA(cudaMemcpyAsync(boff, off_h, sizeof(off_h), cudaMemcpyHostToDevice, ctx->stream));
  if (m) PPP_CUDA(cudaMemcpyAsync(bidx, idx_host, (size_t)m * 4, cudaMemcpyHostToDevice, ctx->stream));
  PPP_CUDA(cudaMemsetAsync(bits, 0, words * 4, ctx->stream));
  PPP_CUDA(cudaStreamSynchronize(ctx->stream));  // the small host arrays above live on this stack frame
  if (m) {
    PPP_LAUNCH(ctx, "set_member_bits", k_set_member_bits, (unsigned)((m + 255) / 256), 256, 0, (const int32_t*)bidx, m, bits);
    PPP_CHECK_LAUNCH();
  }
  std::vector<int64_t> offv = {0, m};
  int st = contours_launch(c, gs, planes, 1, boff, bidx, m, offv, mode, total_nodes_out, bits, mp);
  dev_free(ctx, planes); dev_free(ctx, boff); dev_free(ctx, bidx); dev_free(ctx, bits);
  return st;
}

// ---------------------------------------------------------------------------------------------
// SectPath pairing without a mid-chain host synchronisation.  bands_launch / contours_launch fetch two
// sizes on the way (band members, node total) to size their allocations; each fetch is a device->host
// round trip, and in the host-pointer path those round trips queue behind the 32 MB copy of the
// normals (measured: the chain took 690 us under the copy against 320 us alone).  Here every buffer is
// sized from a HOST-side bound instead -- a point belongs to at most `max_depth` bands, a band yields
// at most one node per member -- the kernels read the real sizes from device memory, and one fetch
// at the end returns {node total, band members, largest band, destination used}.
// Returns PPP_ERR_UNSUPPORTED (nothing launched) when the bound is too large to allocate blindly.
// ---------------------------------------------------------------------------------------------
int slice_contours_sect_async(ppp_cloud* c, const GridStore& gs, const float* plane_x_host, int S, float half_width,
                              int truncate_center, int64_t* total_nodes_out, int64_t* total_members_out, const MPSet* mp) {
  ppp_ctx* ctx = c->ctx;
  if (S <= 0 || c->n <= 0) return PPP_ERR_UNSUPPORTED;
  // Bands are drawn from the grid's cell-major array and hold SORTED POSITIONS: consecutive members of a band
  // are neighbours in space, so the pairing searches of a warp walk the same cells (L1 / L2 reuse instead of a
  // DRAM gather per member), and every record they need is one contiguous-ish load from the sorted array.
  BandPrep bp;
  // (With the multi-projection index a position means something different in every grid: lists of original
  // indices are used there.)
  PPP_TRY(bands_prepare(c, plane_x_host, S, half_width, truncate_center, &bp, mp ? nullptr : &gs));
  const int64_t Mb = (int64_t)std::max(bp.max_depth, 1) * c->n;   // >= band members
  int st = PPP_OK;
  int32_t* idx = nullptr; double *ty = nullptr, *tz = nullptr; int32_t* n_nodes = nullptr;
  u64 *keys = nullptr, *scratch = nullptr; float *ys = nullptr, *zs = nullptr; int64_t* summary = nullptr;
  auto cleanup = [&]() {
    dev_free(ctx, bp.counts); dev_free(ctx, bp.pdev); dev_free(ctx, bp.offsets); dev_free(ctx, bp.fdev);
    dev_free(ctx, idx); dev_free(ctx, ty); dev_free(ctx, tz); dev_free(ctx, n_nodes);
    dev_free(ctx, keys); dev_free(ctx, scratch); dev_free(ctx, ys); dev_free(ctx, zs); dev_free(ctx, summary);
  };
  if ((double)Mb * 72.0 > 6.0e9) {   // ~72 B of temporaries per possible member
    cleanup();
    return PPP_ERR_UNSUPPORTED;
  }
  const size_t M = (size_t)Mb;
  auto body = [&]() -> int {
    PPP_TRY(dev_alloc(ctx, &idx, M));
    PPP_TRY(bands_fill(c, bp, idx));
    PPP_TRY(dev_alloc(ctx, &ty, M)); PPP_TRY(dev_alloc(ctx, &tz, M));
    PPP_TRY(dev_alloc(ctx, &n_nodes, (size_t)S));
    PPP_TRY(dev_alloc(ctx, &keys, M)); PPP_TRY(dev_alloc(ctx, &ys, M)); PPP_TRY(dev_alloc(ctx, &zs, M));
    PPP_TRY(dev_alloc(ctx, &scratch, M));
    PPP_TRY(dev_alloc(ctx, &summary, 5));   // {nodes, members, largest band, used caller's buffers, ticket}
    PPP_CUDA(cudaMemsetAsync(summary, 0, 5 * sizeof(int64_t), ctx->stream));
    const float* planes_dev = bp.fdev;
    PairParams P{};
    set_grids(P, gs, mp); P.xyz4 = c->xyz4;
    P.planes = planes_dev; P.lo = planes_dev + S; P.hi = planes_dev + 2 * (size_t)S;
    P.band_off = bp.offsets; P.band_idx = idx; P.S = S; P.M = Mb;
    P.member = nullptr; P.keys = keys; P.ys = ys; P.zs = zs; P.by_pos = mp ? 0 : 1;
    const int64_t per_block = (int64_t)PAIR_WARPS * PAIR_CHUNK;
    PPP_LAUNCH(ctx, "pair_nodes", k_pair_nodes<false>, (unsigned)((Mb + per_block - 1) / per_block), PAIR_WARPS * 32, 0, P);
    PPP_CHECK_LAUNCH();
    // shared-memory capacity of the per-slice sort: the largest band of the previous call on this
    // cloud, else an estimate from the mean population of a band; larger bands sort in `scratch`
    // size of the largest band: that of the previous call on this cloud, else what a uniform spread of the points along
    // x would put into the widest band (+50 %); whatever turns out larger goes to the cluster launch
    const double ext_x = std::max((double)c->bmax[0] - (double)c->bmin[0], 1e-6);
    const int64_t uniform = (int64_t)std::min((double)Mb, 1.5 * (double)c->n_finite * std::min(1.0, (double)bp.max_width / ext_x)) + 512;
    int64_t guess = c->max_band_hint > 0 ? c->max_band_hint + c->max_band_hint / 4 : uniform;
    // closed / steep workpieces (multi-projection index) have silhouette bands many times the mean
    PPP_TRY(launch_slice_order(ctx, S, guess, mp != nullptr, (const int64_t*)bp.offsets, (const int32_t*)idx, mp ? (const float4*)nullptr : gs.v.sorted,
                               (const u64*)keys, (const float*)ys, (const float*)zs, scratch, ty, tz, n_nodes));
    if (c->c_S_cap < S + 1) {
      dev_free(ctx, c->c_node_off);
      PPP_TRY(dev_alloc_keep(ctx, &c->c_node_off, (size_t)S + 1));
      c->c_S_cap = S + 1;
    }
    const bool inline_scan = S <= 4096;   // the compaction kernel sums the node counts itself
    if (!inline_scan) PPP_TRY(scan_exclusive_i32_to_i64(ctx, n_nodes, c->c_node_off, S));
    if (c->c_cap < Mb || !c->c_y) {   // cloud-owned result buffers that hold any possible total
      dev_free(ctx, c->c_y); dev_free(ctx, c->c_x); dev_free(ctx, c->c_z);
      c->c_y = c->c_x = c->c_z = nullptr; c->c_cap = 0;
      PPP_TRY(dev_alloc_keep(ctx, &c->c_y, M)); PPP_TRY(dev_alloc_keep(ctx, &c->c_x, M)); PPP_TRY(dev_alloc_keep(ctx, &c->c_z, M));
      c->c_cap = Mb;
    }
    NodeDest D{c->ext_y, c->ext_x, c->ext_z, c->ext_y ? c->ext_cap : 0, c->c_y, c->c_x, c->c_z, c->ext_off, c->ext_off_cap};
    const unsigned seq = ++ctx->fetch_seq ? ctx->fetch_seq : ++ctx->fetch_seq;
    PPP_LAUNCH(ctx, "compact_nodes", k_compact_nodes_auto, (unsigned)S, 256, 0, (const int64_t*)bp.offsets,
               c->c_node_off, inline_scan ? (const int32_t*)n_nodes : (const int32_t*)nullptr, S, planes_dev, (const double*)ty, (const double*)tz, D, summary,
               (unsigned*)ctx->fetch_host, (unsigned*)fetch_flag(ctx), seq);
    PPP_CHECK_LAUNCH();
    int64_t h[4] = {0, 0, 0, 0};
    PPP_TRY(fetch_wait(ctx, seq));                       // the one synchronisation of the chain
    memcpy(h, ctx->fetch_host, sizeof(h));
    const bool ext = h[3] != 0;
    c->out_y = ext ? c->ext_y : c->c_y;
    c->out_x = ext ? c->ext_x : c->c_x;
    c->out_z = ext ? c->ext_z : c->c_z;
    c->max_band_hint = h[2];
    *total_nodes_out = h[0];
    *total_members_out = h[1];
    return PPP_OK;
  };
  st = body();
  cleanup();
  return st;
}
