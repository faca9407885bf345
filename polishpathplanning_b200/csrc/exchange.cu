// Multi-GPU exchange stage of the hot path (SURVEY.md §8e): a cloud that starts out split by ORIGINAL
// INDEX over the ranks (rank r holds records [start[r], start[r+1]) of the file) is redistributed into
// x-slabs of equal point count plus a halo, entirely by hand-written kernels that store into the
// destination GPU's memory over NVLink / NVSwitch -- no NCCL collective, no host staging:
//
//   phase 0  k_ex_minmax    x-range + finite count of the local chunk  -> every peer's slot
//   phase 1  k_ex_hist      1024-bin x histogram over the GLOBAL range -> every peer's slot
//   phase 2  k_ex_count     equal-count cuts from the summed histograms (identical on every rank, derived by
//                           every block), destinations of every record (owner slab + halo copies), per-tile
//                           counts; send counts -> every peer
//   phase 3  k_ex_scatter   records -> the destination's receive buffer at
//                           (sum of the counts of lower ranks) + (counts of the rank's earlier tiles) + (rank inside the tile),
//                           i.e. in ascending GLOBAL INDEX order, so every (d2, index) tie-break and the
//                           El / Er insertion order are those of the single-GPU run
//   phase 4  results        normals go straight from the search kernels to their HOME rank (the rank
//                           that holds that original index range; store_normal + NormalRoute), contour
//                           nodes to rank 0's region; a flag per rank closes the step.
//
// Every phase that feeds a peer ends with the LAST block of the producing kernel (atomic ticket)
// publishing a per-(phase, source) flag with system-scope release stores into every peer's arena;
// the consumer's stream first runs k_ex_wait, one warp polling its own arena's flags (acquire loads,
// bounded by a time-out so a dead peer gives an error instead of a hang).  Flags carry the step number,
// so nothing is reset between steps; the only slots written before a step's first wait (the min/max
// slots) are double-buffered by step parity, everything else is written after a wait that proves every
// rank has finished the previous step.
//
// The reference is single-process; what this stage shards is its whole-cloud estimate_normal
// (src/Path_Generation.cpp:323-333) and the plane sweep (src/Path_Generation.cpp:689-755).
#include <stddef.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "ppp_device.cuh"

namespace {

constexpr int EX_BINS = 1024;         // x histogram bins: slab populations are equal to within total / 1024
constexpr int EX_PHASES = 6;          // 0..3 exchange, 4 normals delivered, 5 contours delivered
constexpr int EX_TILE = 2048;         // records per block of the count / scatter kernels
constexpr int EX_THREADS = 256;
constexpr unsigned long long EX_TIMEOUT_NS = 10ull * 1000 * 1000 * 1000;

struct ExLayout {
  size_t flags, mm, hist, cnt, halo, recv, home, nodes, node_off_bytes, node_arr_bytes, node_region, total;
};

inline size_t a256(size_t v) { return (v + 255) / 256 * 256; }

ExLayout ex_layout(int world, int64_t cap_recv, int64_t cap_home, int home_stride_f, int S_cap, int64_t node_cap) {
  ExLayout L{};
  size_t at = 0;
  L.flags = at; at += a256((size_t)EX_PHASES * 32 * sizeof(uint32_t));       // one 128-byte line per phase
  L.mm = at;    at += a256((size_t)2 * PPP_MAX_RANKS * sizeof(float4));       // [parity][src] = {min, max, finite lo, finite hi}
  L.hist = at;  at += a256((size_t)PPP_MAX_RANKS * EX_BINS * sizeof(int32_t)); // [src][bin]
  L.cnt = at;   at += a256((size_t)2 * PPP_MAX_RANKS * PPP_MAX_RANKS * sizeof(int32_t));  // [0]: records, [1]: owned; [src][dst]
  L.halo = at;  at += a256((size_t)PPP_MAX_RANKS * sizeof(double));          // [src]: the halo src cut its copies with
  L.recv = at;  at += a256((size_t)std::max<int64_t>(cap_recv, 1) * sizeof(float4));
  L.home = at;  at += a256((size_t)std::max<int64_t>(cap_home, 1) * home_stride_f * sizeof(float));
  L.node_off_bytes = a256(((size_t)S_cap + 1) * sizeof(int64_t));
  L.node_arr_bytes = a256((size_t)std::max<int64_t>(node_cap, 1) * sizeof(double));
  L.node_region = L.node_off_bytes + 3 * L.node_arr_bytes;
  L.nodes = at; at += (size_t)world * L.node_region;
  L.total = at;
  (void)world;
  return L;
}

// Device view of all arenas (passed by value).
struct ExView {
  int rank, world;
  unsigned char* arena[PPP_MAX_RANKS];
  unsigned long long off_flags, off_mm, off_hist, off_cnt, off_halo, off_recv;
  long long cap_recv;
};

// Local scratch (device memory of the owning rank only).
struct ExScratch {
  uint32_t mn, mx;                  // ordered-uint min / max of the finite x of the chunk
  unsigned long long n_fin;
  unsigned int ticket[4];           // last-block detection, one per producing kernel
  int32_t hist[EX_BINS];
  int32_t cutbin[PPP_MAX_RANKS + 1];
  double cutx[PPP_MAX_RANKS + 1];
  double gmin, gmax, inv;           // global finite x-range, bins per unit
  double halo_min;                  // narrowest halo any rank cut its copies with this step
  int32_t sendcnt[PPP_MAX_RANKS], sendown[PPP_MAX_RANKS];
  // summary fetched by the host after the exchange
  long long n_local, n_owned;
  int32_t err;                      // 1: wait timed out, 2: receive buffer overflow
  int32_t pad;
};

__device__ __forceinline__ uint32_t ex_f2ord(float f) {
  uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float ex_ord2f(uint32_t u) {
  uint32_t b = (u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u;
  return __uint_as_float(b);
}

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ uint32_t* ex_flag(const ExView& V, int dst, int phase, int src) {
  return reinterpret_cast<uint32_t*>(V.arena[dst] + V.off_flags) + phase * 32 + src;
}

// Called by every thread of a block after the block's last store of the phase.  Returns true in the
// block that finished last (all other blocks' stores are then visible to it).
__device__ __forceinline__ bool ex_last_block(unsigned int* ticket) {
  __shared__ bool s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int t = atomicAdd(ticket, 1u);
    s_last = (t == gridDim.x - 1);
    if (s_last) *ticket = 0;     // ready for the next step
  }
  __syncthreads();
  if (s_last) __threadfence();
  return s_last;
}

// Last block only, after its peer stores: make them visible system-wide, then raise this rank's flag
// of `phase` in every arena (including the own one, which keeps k_ex_wait uniform).
__device__ __forceinline__ void ex_publish(const ExView& V, int phase, uint32_t step) {
  __threadfence_system();
  __syncthreads();
  if ((int)threadIdx.x < V.world) st_release_sys(ex_flag(V, threadIdx.x, phase, V.rank), step);
}

__device__ __forceinline__ void ex_load_xyz(const float* __restrict__ raw, int64_t i, int sf, int vec_ok, float& x, float& y, float& z) {
  if (vec_ok) {
    float4 p = __ldg(reinterpret_cast<const float4*>(raw + i * sf));
    x = p.x; y = p.y; z = p.z;
  } else {
    const float* p = raw + i * sf;
    x = __ldg(p); y = __ldg(p + 1); z = __ldg(p + 2);
  }
}

// ---- waits ------------------------------------------------------------------------------------
__global__ void k_ex_wait(ExView V, int phase, uint32_t step, int only_src, ExScratch* sc) {
  pdl_prologue();
  const int src = threadIdx.x;
  if (src >= V.world || (only_src >= 0 && src != only_src)) return;
  const uint32_t* f = ex_flag(V, V.rank, phase, src);
  const unsigned long long t0 = globaltimer_ns();
  while ((int32_t)(ld_acquire_sys(f) - step) < 0) {
    if (globaltimer_ns() - t0 > EX_TIMEOUT_NS) { atomicMax(&sc->err, 1); break; }
    __nanosleep(200);
  }
}

// Raise this rank's flag of `phase` everywhere: closes a phase whose stores were issued by earlier
// kernels of the stream (the search kernels' normal records, the contour compaction).
__global__ void k_ex_signal(ExView V, int phase, uint32_t step) {
  pdl_prologue();
  __threadfence_system();
  if ((int)threadIdx.x < V.world) st_release_sys(ex_flag(V, threadIdx.x, phase, V.rank), step);
}

__global__ void k_ex_reset(ExScratch* sc) {
  pdl_prologue();
  sc->mn = 0xFFFFFFFFu; sc->mx = 0u; sc->n_fin = 0ull;
  for (int i = 0; i < 4; i++) sc->ticket[i] = 0;
  for (int i = threadIdx.x; i < EX_BINS; i += blockDim.x) sc->hist[i] = 0;
  sc->err = 0;
}

// ---- phase 0: x-range of the chunk --------------------------------------------------------------
__global__ void __launch_bounds__(EX_THREADS) k_ex_minmax(ExView V, const float* __restrict__ raw, int64_t n, int sf, int vec_ok,
                                                          uint32_t step, ExScratch* sc) {
  pdl_prologue();
  float mn = CUDART_INF_F, mx = -CUDART_INF_F;
  unsigned cnt = 0;
  constexpr int PPT = 4;   // independent loads in flight per thread
  for (int64_t b0 = (int64_t)blockIdx.x * blockDim.x * PPT; b0 < n; b0 += (int64_t)gridDim.x * blockDim.x * PPT) {
    float x[PPT], y[PPT], z[PPT];
#pragma unroll
    for (int j = 0; j < PPT; j++) {
      const int64_t i = b0 + (int64_t)j * blockDim.x + threadIdx.x;
      x[j] = y[j] = z[j] = CUDART_NAN_F;
      if (i < n) ex_load_xyz(raw, i, sf, vec_ok, x[j], y[j], z[j]);
    }
#pragma unroll
    for (int j = 0; j < PPT; j++)
      if (finite3(x[j], y[j], z[j])) { mn = fminf(mn, x[j]); mx = fmaxf(mx, x[j]); cnt++; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  // block-level combine, then ONE set of atomics per block (per-warp atomics on three addresses serialise in L2)
  __shared__ float s_mn[EX_THREADS / 32], s_mx[EX_THREADS / 32];
  __shared__ unsigned s_c[EX_THREADS / 32];
  if ((threadIdx.x & 31) == 0) { s_mn[threadIdx.x >> 5] = mn; s_mx[threadIdx.x >> 5] = mx; s_c[threadIdx.x >> 5] = cnt; }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned tot = 0;
    for (int i = 0; i < EX_THREADS / 32; i++) { mn = fminf(mn, s_mn[i]); mx = fmaxf(mx, s_mx[i]); tot += s_c[i]; }
    if (tot) {
      atomicMin(&sc->mn, ex_f2ord(mn));
      atomicMax(&sc->mx, ex_f2ord(mx));
      atomicAdd(&sc->n_fin, (unsigned long long)tot);
    }
  }
  if (!ex_last_block(&sc->ticket[0])) return;
  // last block: this rank's {min, max, finite count} into every arena, then the flag
  const uint32_t omn = *(volatile uint32_t*)&sc->mn, omx = *(volatile uint32_t*)&sc->mx;
  const unsigned long long nf = *(volatile unsigned long long*)&sc->n_fin;
  if ((int)threadIdx.x < V.world) {
    float4* slot = reinterpret_cast<float4*>(V.arena[threadIdx.x] + V.off_mm) + (step & 1u) * PPP_MAX_RANKS + V.rank;
    *slot = make_float4(nf ? ex_ord2f(omn) : CUDART_INF_F, nf ? ex_ord2f(omx) : -CUDART_INF_F,
                        __uint_as_float((uint32_t)(nf & 0xFFFFFFFFull)), __uint_as_float((uint32_t)(nf >> 32)));
  }
  __syncthreads();
  if (threadIdx.x == 0) { sc->mn = 0xFFFFFFFFu; sc->mx = 0u; sc->n_fin = 0ull; }
  ex_publish(V, 0, step);
}

// Global finite x-range from the min/max slots of the own arena (identical on every rank).
__device__ __forceinline__ void ex_global_range(const ExView& V, uint32_t step, double& gmin, double& gmax) {
  const float4* slots = reinterpret_cast<const float4*>(V.arena[V.rank] + V.off_mm) + (step & 1u) * PPP_MAX_RANKS;
  float mn = CUDART_INF_F, mx = -CUDART_INF_F;
  for (int r = 0; r < V.world; r++) {
    const volatile float* s = reinterpret_cast<const volatile float*>(slots + r);
    mn = fminf(mn, s[0]); mx = fmaxf(mx, s[1]);
  }
  if (!(mn <= mx)) { mn = 0.f; mx = 0.f; }   // no finite point anywhere
  gmin = (double)mn; gmax = (double)mx;
}

__device__ __forceinline__ int ex_bin(float x, double gmin, double inv) {
  int b = (int)floor(((double)x - gmin) * inv);
  return b < 0 ? 0 : (b > EX_BINS - 1 ? EX_BINS - 1 : b);
}

// ---- phase 1: histogram of x over the global range -----------------------------------------------
__global__ void __launch_bounds__(1024) k_ex_hist(ExView V, const float* __restrict__ raw, int64_t n, int sf, int vec_ok,
                                                        uint32_t step, ExScratch* sc) {
  pdl_prologue();
  __shared__ int32_t s_hist[EX_BINS];
  for (int i = threadIdx.x; i < EX_BINS; i += blockDim.x) s_hist[i] = 0;
  double gmin, gmax;
  ex_global_range(V, step, gmin, gmax);
  const double span = fmax(gmax - gmin, 1e-9);
  const double inv = (double)EX_BINS / span;
  __syncthreads();
  constexpr int PPT = 4;
  for (int64_t b0 = (int64_t)blockIdx.x * blockDim.x * PPT; b0 < n; b0 += (int64_t)gridDim.x * blockDim.x * PPT) {
    float x[PPT], y[PPT], z[PPT];
#pragma unroll
    for (int j = 0; j < PPT; j++) {
      const int64_t i = b0 + (int64_t)j * blockDim.x + threadIdx.x;
      x[j] = y[j] = z[j] = CUDART_NAN_F;
      if (i < n) ex_load_xyz(raw, i, sf, vec_ok, x[j], y[j], z[j]);
    }
#pragma unroll
    for (int j = 0; j < PPT; j++)
      if (finite3(x[j], y[j], z[j])) atomicAdd(&s_hist[ex_bin(x[j], gmin, inv)], 1);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < EX_BINS; i += blockDim.x) {
    int c = s_hist[i];
    if (c) atomicAdd(&sc->hist[i], c);
  }
  if (!ex_last_block(&sc->ticket[1])) return;
  if (threadIdx.x == 0) { sc->gmin = gmin; sc->gmax = gmax; sc->inv = inv; }
  for (int d = 0; d < V.world; d++) {
    int32_t* dst = reinterpret_cast<int32_t*>(V.arena[d] + V.off_hist) + (size_t)V.rank * EX_BINS;
    for (int i = threadIdx.x; i < EX_BINS; i += blockDim.x) dst[i] = *(volatile int32_t*)&sc->hist[i];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < EX_BINS; i += blockDim.x) sc->hist[i] = 0;
  ex_publish(V, 1, step);
}

// ---- phase 2: equal-count cuts + destination counts -------------------------------------------------
// The slab limits every rank derives, identically, from the summed histograms.
struct ExCuts {
  int32_t cutbin[PPP_MAX_RANKS + 1];
  double cutx[PPP_MAX_RANKS + 1];
  double gmin, gmax, inv;
};

// cut r = upper edge of the first bin at which the cumulative count reaches total * r / world (integer
// arithmetic, so every rank -- and every block -- computes the same bins from the same histograms).
// Block-wide; EX_BINS / blockDim.x bins per thread.  C lives in shared memory.
__device__ void ex_compute_cuts(const ExView& V, uint32_t step, ExCuts* C, long long* s_cum /* EX_BINS */, long long* s_part /* blockDim.x */) {
  const int32_t* H = reinterpret_cast<const int32_t*>(V.arena[V.rank] + V.off_hist);
  const int per = EX_BINS / (int)blockDim.x;
  long long sum = 0;
  for (int j = 0; j < per; j++) {
    long long t = 0;
    for (int r = 0; r < V.world; r++) t += *(volatile const int32_t*)(H + (size_t)r * EX_BINS + threadIdx.x * per + j);
    s_cum[threadIdx.x * per + j] = t;
    sum += t;
  }
  s_part[threadIdx.x] = sum;
  __syncthreads();
  for (int o = 1; o < (int)blockDim.x; o <<= 1) {     // inclusive scan of the per-thread sums (Hillis-Steele)
    long long t = (int)threadIdx.x >= o ? s_part[threadIdx.x - o] : 0;
    __syncthreads();
    s_part[threadIdx.x] += t;
    __syncthreads();
  }
  long long run = s_part[threadIdx.x] - sum;
  for (int j = 0; j < per; j++) { run += s_cum[threadIdx.x * per + j]; s_cum[threadIdx.x * per + j] = run; }
  if (threadIdx.x == 0) {
    double gmin, gmax;
    ex_global_range(V, step, gmin, gmax);
    C->gmin = gmin; C->gmax = gmax;
    C->inv = (double)EX_BINS / fmax(gmax - gmin, 1e-9);
  }
  __syncthreads();
  const long long total = s_cum[EX_BINS - 1];
  if ((int)threadIdx.x <= V.world) {
    const int r = threadIdx.x;
    int cb;
    if (r == 0) cb = 0;
    else if (r == V.world) cb = EX_BINS;
    else {
      // smallest k with cum[k] * world >= total * r  -> cut bin k + 1
      int lo = 0, hi = EX_BINS - 1;
      while (lo < hi) { int m = (lo + hi) >> 1; if (s_cum[m] * V.world >= total * r) hi = m; else lo = m + 1; }
      cb = lo + 1;
    }
    C->cutbin[r] = cb;
    const double span = fmax(C->gmax - C->gmin, 1e-9);
    C->cutx[r] = r == 0 ? -CUDART_INF : (r == V.world ? CUDART_INF : C->gmin + span * (double)cb / (double)EX_BINS);
  }
  __syncthreads();
}

// Destination mask of one record: bit d set = rank d receives it; *owner = the slab that owns it.
// Owner by BIN (consistent with the cuts by construction); halo copies by comparing x with the cut
// positions.  Non-finite points belong to rank 0 (they keep their place in the index numbering and
// get a NaN normal there, as in PCL) and are never anybody's halo.
template <typename CUTS>
__device__ __forceinline__ unsigned ex_dest_mask(const CUTS* sc, int world, float x, float y, float z, double halo, int* owner) {
  if (!finite3(x, y, z)) { *owner = 0; return 1u; }
  const int b = ex_bin(x, sc->gmin, sc->inv);
  int o = 0;
  while (o + 1 < world && b >= sc->cutbin[o + 1]) o++;
  *owner = o;
  unsigned m = 1u << o;
  const double xd = (double)x;
  for (int d = o - 1; d >= 0 && xd < sc->cutx[d + 1] + halo; d--) m |= 1u << d;
  for (int d = o + 1; d < world && xd >= sc->cutx[d] - halo; d++) m |= 1u << d;
  return m;
}

// Every block derives the cuts itself (a thousand bins: cheaper than one more launch between two waits), counts
// the destinations of its tile, and the last block publishes this rank's send counts to every peer.
__global__ void __launch_bounds__(EX_THREADS) k_ex_count(ExView V, const float* __restrict__ raw, int64_t n, int sf, int vec_ok,
                                                         double halo, uint32_t step, ExScratch* sc, int32_t* __restrict__ tilecnt,
                                                         int ntiles) {
  pdl_prologue();
  __shared__ long long s_cum[EX_BINS];
  __shared__ long long s_part[EX_THREADS];
  __shared__ ExCuts C;
  __shared__ int s_cnt[PPP_MAX_RANKS], s_own[PPP_MAX_RANKS];
  if (threadIdx.x < PPP_MAX_RANKS) { s_cnt[threadIdx.x] = 0; s_own[threadIdx.x] = 0; }
  ex_compute_cuts(V, step, &C, s_cum, s_part);
  const int world = V.world;
  if (blockIdx.x == 0) {      // for the scatter kernel and the host's summary
    if ((int)threadIdx.x <= world) { sc->cutbin[threadIdx.x] = C.cutbin[threadIdx.x]; sc->cutx[threadIdx.x] = C.cutx[threadIdx.x]; }
    if (threadIdx.x == 0) { sc->gmin = C.gmin; sc->gmax = C.gmax; sc->inv = C.inv; }
  }
  const int64_t base = (int64_t)blockIdx.x * EX_TILE;
  for (int it = 0; it < EX_TILE / EX_THREADS; it++) {
    const int64_t i = base + (int64_t)it * EX_THREADS + threadIdx.x;
    if (i < n) {
      float x, y, z;
      ex_load_xyz(raw, i, sf, vec_ok, x, y, z);
      int owner;
      unsigned m = ex_dest_mask(&C, world, x, y, z, halo, &owner);
      atomicAdd(&s_own[owner], 1);
      while (m) { int d = __ffs(m) - 1; m &= m - 1; atomicAdd(&s_cnt[d], 1); }
    }
  }
  __syncthreads();
  if ((int)threadIdx.x < world) {
    tilecnt[(size_t)threadIdx.x * ntiles + blockIdx.x] = s_cnt[threadIdx.x];
    if (s_cnt[threadIdx.x]) atomicAdd(&sc->sendcnt[threadIdx.x], s_cnt[threadIdx.x]);
    if (s_own[threadIdx.x]) atomicAdd(&sc->sendown[threadIdx.x], s_own[threadIdx.x]);
  }
  if (!ex_last_block(&sc->ticket[2])) return;
  // last block: this rank's row of the count tables (records, owned) into every arena
  if ((int)threadIdx.x < world * world) {
    const int peer = threadIdx.x / world, dst = threadIdx.x % world;
    int32_t* tab = reinterpret_cast<int32_t*>(V.arena[peer] + V.off_cnt);
    tab[V.rank * PPP_MAX_RANKS + dst] = *(volatile int32_t*)&sc->sendcnt[dst];
    tab[PPP_MAX_RANKS * PPP_MAX_RANKS + V.rank * PPP_MAX_RANKS + dst] = *(volatile int32_t*)&sc->sendown[dst];
  }
  if ((int)threadIdx.x < world) reinterpret_cast<double*>(V.arena[threadIdx.x] + V.off_halo)[V.rank] = halo;
  __syncthreads();
  if (threadIdx.x < PPP_MAX_RANKS) { sc->sendown[threadIdx.x] = 0; sc->sendcnt[threadIdx.x] = 0; }
  ex_publish(V, 2, step);
}

// ---- phase 3: the records, straight into the destination's receive buffer ---------------------------
// Record = {x, y, z, bits(global index)}; a halo copy carries ~global index (negative).
// Positions are stable: records of a tile are taken in (iteration, thread) order = ascending index.  All
// records of the tile are loaded up front (EX_ITERS independent loads per thread), the per-(iteration, warp,
// destination) counts meet in shared memory once, a handful of threads turn them into offsets, and each
// record's position is  base + offset(iteration, warp) + rank inside the warp (ballot).
constexpr int EX_ITERS = EX_TILE / EX_THREADS;
constexpr int EX_WARPS = EX_THREADS / 32;

__global__ void __launch_bounds__(EX_THREADS) k_ex_scatter(ExView V, const float* __restrict__ raw, int64_t n, int sf, int vec_ok,
                                                           int64_t global_start, double halo, uint32_t step, ExScratch* sc,
                                                           const int32_t* __restrict__ tilecnt, int ntiles) {
  pdl_prologue();
  __shared__ int s_off[EX_ITERS * EX_WARPS][PPP_MAX_RANKS];
  __shared__ long long s_base[PPP_MAX_RANKS];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int world = V.world;
  // where this tile's records start in every destination: the counts of the lower ranks (count table) plus the
  // counts of this rank's earlier tiles (summed here: at most a few thousand values, no scan kernel in between)
  if ((int)threadIdx.x < world) {
    const int d = threadIdx.x;
    const int32_t* tab = reinterpret_cast<const int32_t*>(V.arena[V.rank] + V.off_cnt);
    long long b = 0;
    for (int s = 0; s < V.rank; s++) b += *(volatile const int32_t*)(tab + s * PPP_MAX_RANKS + d);
    s_base[d] = b;
  }
  __syncthreads();
  for (int d = 0; d < world; d++) {
    int part = 0;
    for (int t = threadIdx.x; t < (int)blockIdx.x; t += EX_THREADS) part += __ldg(tilecnt + (size_t)d * ntiles + t);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0 && part) atomicAdd((unsigned long long*)&s_base[d], (unsigned long long)part);
  }
  const int64_t base = (int64_t)blockIdx.x * EX_TILE;
  float x[EX_ITERS], y[EX_ITERS], z[EX_ITERS];
  unsigned mask[EX_ITERS];   // bits 0..15 destinations, bits 16..19 owner
#pragma unroll
  for (int it = 0; it < EX_ITERS; it++) {
    const int64_t i = base + (int64_t)it * EX_THREADS + threadIdx.x;
    x[it] = y[it] = z[it] = 0.f;
    if (i < n) ex_load_xyz(raw, i, sf, vec_ok, x[it], y[it], z[it]);
  }
#pragma unroll
  for (int it = 0; it < EX_ITERS; it++) {
    const int64_t i = base + (int64_t)it * EX_THREADS + threadIdx.x;
    int owner = 0;
    unsigned m = 0;
    if (i < n) m = ex_dest_mask(sc, world, x[it], y[it], z[it], halo, &owner);
    mask[it] = m | ((unsigned)owner << 16);
    for (int d = 0; d < world; d++) {
      const unsigned bal = __ballot_sync(0xffffffffu, (m >> d) & 1u);
      if (lane == 0) s_off[it * EX_WARPS + w][d] = __popc(bal);
    }
  }
  __syncthreads();
  if ((int)threadIdx.x < world) {   // exclusive scan over the (iteration, warp) pairs of one destination
    int run = 0;
    for (int j = 0; j < EX_ITERS * EX_WARPS; j++) { int c = s_off[j][threadIdx.x]; s_off[j][threadIdx.x] = run; run += c; }
  }
  __syncthreads();
#pragma unroll
  for (int it = 0; it < EX_ITERS; it++) {
    const unsigned m = mask[it] & 0xFFFFu;
    const int owner = (int)(mask[it] >> 16);
    const int g = (int)(global_start + base + (int64_t)it * EX_THREADS + threadIdx.x);
    for (int d = 0; d < world; d++) {
      const unsigned bal = __ballot_sync(0xffffffffu, (m >> d) & 1u);
      if ((m >> d) & 1u) {
        const long long at = s_base[d] + s_off[it * EX_WARPS + w][d] + __popc(bal & ((1u << lane) - 1u));
        if (at < V.cap_recv)
          reinterpret_cast<float4*>(V.arena[d] + V.off_recv)[at] = make_float4(x[it], y[it], z[it], __int_as_float(d == owner ? g : ~g));
        else
          atomicMax(&sc->err, 2);
      }
    }
  }
  if (!ex_last_block(&sc->ticket[3])) return;
  ex_publish(V, 3, step);
}

// After the records have landed: local row -> global index (-1 for halo copies), and the summary.
__global__ void __launch_bounds__(256) k_ex_rowmap(ExView V, ExScratch* sc, int32_t* __restrict__ rowmap) {
  pdl_prologue();
  __shared__ long long s_n[2];
  if (threadIdx.x == 0) {
    const int32_t* tab = reinterpret_cast<const int32_t*>(V.arena[V.rank] + V.off_cnt);
    long long n_local = 0, n_owned = 0;
    for (int s = 0; s < V.world; s++) {
      n_local += *(volatile const int32_t*)(tab + s * PPP_MAX_RANKS + V.rank);
      n_owned += *(volatile const int32_t*)(tab + PPP_MAX_RANKS * PPP_MAX_RANKS + s * PPP_MAX_RANKS + V.rank);
    }
    if (n_local > V.cap_recv) {   // senders dropped what does not fit; the receiver reports it
      n_local = V.cap_recv;
      if (blockIdx.x == 0) atomicMax(&sc->err, 2);
    }
    if (blockIdx.x == 0) {
      sc->n_local = n_local; sc->n_owned = n_owned;
      const double* hs = reinterpret_cast<const double*>(V.arena[V.rank] + V.off_halo);
      double hm = *(volatile const double*)hs;
      for (int s = 1; s < V.world; s++) hm = fmin(hm, *(volatile const double*)(hs + s));
      sc->halo_min = hm;
    }
    s_n[0] = n_local;
  }
  __syncthreads();
  const long long n_local = s_n[0];
  const float4* recv = reinterpret_cast<const float4*>(V.arena[V.rank] + V.off_recv);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_local; i += (int64_t)gridDim.x * blockDim.x) {
    const int g = __float_as_int(recv[i].w);
    rowmap[i] = g >= 0 ? g : -1;
  }
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct ppp_exch {
  ppp_ctx* ctx = nullptr;
  int rank = 0, world = 1;
  int64_t n_total = 0;
  int64_t starts[PPP_MAX_RANKS + 1] = {};
  int64_t cap_recv = 0, cap_home = 0, node_cap = 0;
  int S_cap = 0;
  int home_sf = 8;
  ExLayout L{};
  unsigned char* arena = nullptr;
  unsigned char* peer[PPP_MAX_RANKS] = {};
  bool ipc_opened[PPP_MAX_RANKS] = {};
  bool connected = false;
  ExView V{};
  ExScratch* sc = nullptr;
  NormalRoute* route = nullptr;
  int32_t* rowmap = nullptr;
  int32_t* tilecnt = nullptr;
  int64_t tilecnt_cap = 0;
  uint32_t step = 0;
  // the chunk of the step in flight
  const float* raw = nullptr;
  int64_t n = 0;
  int sf = 0, vec_ok = 0, ntiles = 0;
  double halo = 0;     // the narrowest halo any rank's phases were given this step (checked by ppp_dev_mls_smooth)
  double xmag = 0;     // largest finite |x| of the step's cloud (ppp_dev_mls_smooth checks the halo against it)
  int64_t n_local = 0;
};

#define EX_LOCK(ex) ApiScope _api_scope((ex)->ctx)
#define EX_REQUIRE(cond, msg)                       \
  do {                                              \
    if (!(cond)) {                                  \
      ppp_set_error("%s: %s", __func__, msg);       \
      return PPP_ERR_INVALID;                       \
    }                                               \
  } while (0)

static void ex_refresh_view(ppp_exch* ex) {
  ExView& V = ex->V;
  V.rank = ex->rank; V.world = ex->world;
  for (int r = 0; r < PPP_MAX_RANKS; r++) V.arena[r] = r < ex->world ? ex->peer[r] : nullptr;
  V.off_flags = ex->L.flags; V.off_mm = ex->L.mm; V.off_hist = ex->L.hist; V.off_cnt = ex->L.cnt; V.off_halo = ex->L.halo; V.off_recv = ex->L.recv;
  V.cap_recv = ex->cap_recv;
}

static int ex_upload_route(ppp_exch* ex) {
  NormalRoute h{};
  h.world = ex->world;
  for (int r = 0; r <= ex->world; r++) h.start[r] = ex->starts[r];
  for (int r = 0; r < ex->world; r++) h.base[r] = reinterpret_cast<float*>(ex->peer[r] + ex->L.home);
  PPP_CUDA(cudaMemcpyAsync(ex->route, &h, sizeof(h), cudaMemcpyHostToDevice, ex->ctx->stream));
  PPP_CUDA(cudaStreamSynchronize(ex->ctx->stream));   // `h` lives on this stack frame
  return PPP_OK;
}

extern "C" {

int ppp_exch_create(ppp_ctx* ctx, int rank, int world, const int64_t* starts, int64_t cap_recv, int S_cap, int64_t node_cap,
                    size_t normal_stride_bytes, ppp_exch** out) {
  if (!ctx || !out || !starts) { ppp_set_error("ppp_exch_create: NULL argument"); return PPP_ERR_INVALID; }
  *out = nullptr;
  if (world < 1 || world > PPP_MAX_RANKS || rank < 0 || rank >= world) { ppp_set_error("ppp_exch_create: bad rank/world (at most %d ranks)", PPP_MAX_RANKS); return PPP_ERR_INVALID; }
  if (normal_stride_bytes != 16 && normal_stride_bytes != 32) { ppp_set_error("ppp_exch_create: normal stride must be 16 or 32 bytes"); return PPP_ERR_INVALID; }
  for (int r = 0; r < world; r++)
    if (starts[r] > starts[r + 1] || starts[0] != 0) { ppp_set_error("ppp_exch_create: starts must ascend from 0"); return PPP_ERR_INVALID; }
  if (starts[world] >= 2147483647ll) { ppp_set_error("ppp_exch_create: at most 2^31-2 points in total (int32 indices, as PCL)"); return PPP_ERR_INVALID; }
  if (cap_recv < 1 || S_cap < 0 || node_cap < 0) { ppp_set_error("ppp_exch_create: bad capacities"); return PPP_ERR_INVALID; }
  ApiScope scope(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  ppp_exch* ex = new ppp_exch();
  ex->ctx = ctx; ex->rank = rank; ex->world = world;
  for (int r = 0; r <= world; r++) ex->starts[r] = starts[r];
  ex->n_total = starts[world];
  ex->cap_recv = cap_recv; ex->S_cap = S_cap; ex->node_cap = node_cap;
  ex->home_sf = (int)(normal_stride_bytes / 4);
  // one layout for all ranks: the home capacity is the largest index range
  int64_t cap_home = 1;
  for (int r = 0; r < world; r++) cap_home = std::max(cap_home, starts[r + 1] - starts[r]);
  ex->cap_home = cap_home;
  ex->L = ex_layout(world, cap_recv, cap_home, ex->home_sf, S_cap, node_cap);
  cudaError_t e = cudaMalloc((void**)&ex->arena, ex->L.total);
  if (e == cudaSuccess) e = cudaMemset(ex->arena, 0, ex->L.total);
  if (e == cudaSuccess) e = cudaMalloc((void**)&ex->sc, sizeof(ExScratch));
  if (e == cudaSuccess) e = cudaMemset(ex->sc, 0, sizeof(ExScratch));
  if (e == cudaSuccess) e = cudaMalloc((void**)&ex->route, sizeof(NormalRoute));
  if (e == cudaSuccess) e = cudaMalloc((void**)&ex->rowmap, (size_t)cap_recv * sizeof(int32_t));
  if (e != cudaSuccess) {
    ppp_set_error("ppp_exch_create: allocation of %zu bytes failed: %s", ex->L.total, cudaGetErrorString(e));
    cudaGetLastError();
    cudaFree(ex->arena); cudaFree(ex->sc); cudaFree(ex->route); cudaFree(ex->rowmap);
    delete ex;
    return PPP_ERR_NOMEM;
  }
  k_ex_reset<<<1, 256, 0, ctx->stream>>>(ex->sc);
  ctx->launches++;
  PPP_CUDA(cudaStreamSynchronize(ctx->stream));
  ex->peer[rank] = ex->arena;
  *out = ex;
  return PPP_OK;
}

int ppp_exch_ipc_handle(ppp_exch* ex, unsigned char handle[PPP_PEER_HANDLE_BYTES]) {
  if (!ex || !handle) { ppp_set_error("ppp_exch_ipc_handle: NULL argument"); return PPP_ERR_INVALID; }
  EX_LOCK(ex);
  PPP_CUDA(cudaSetDevice(ex->ctx->device));
  cudaIpcMemHandle_t h;
  PPP_CUDA(cudaIpcGetMemHandle(&h, ex->arena));
  memcpy(handle, &h, sizeof(h));
  return PPP_OK;
}

// handles: world x 64 bytes, entry r = rank r's ppp_exch_ipc_handle (the own entry is ignored).
int ppp_exch_connect_ipc(ppp_exch* ex, const unsigned char* handles) {
  if (!ex || !handles) { ppp_set_error("ppp_exch_connect_ipc: NULL argument"); return PPP_ERR_INVALID; }
  EX_LOCK(ex);
  PPP_CUDA(cudaSetDevice(ex->ctx->device));
  for (int r = 0; r < ex->world; r++) {
    if (r == ex->rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + (size_t)r * PPP_PEER_HANDLE_BYTES, sizeof(h));
    void* p = nullptr;
    PPP_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    ex->peer[r] = (unsigned char*)p;
    ex->ipc_opened[r] = true;
  }
  ex_refresh_view(ex);
  PPP_TRY(ex_upload_route(ex));
  ex->connected = true;
  return PPP_OK;
}

// Ranks that live in THIS process (one process driving several contexts; the single-GPU loop-back the
// tests use): all[r] = rank r's exchange.  Arenas on other devices need peer access enabled by the caller.
int ppp_exch_connect_local(ppp_exch* ex, ppp_exch* const* all) {
  if (!ex || !all) { ppp_set_error("ppp_exch_connect_local: NULL argument"); return PPP_ERR_INVALID; }
  EX_LOCK(ex);
  PPP_CUDA(cudaSetDevice(ex->ctx->device));
  for (int r = 0; r < ex->world; r++) {
    EX_REQUIRE(all[r] && all[r]->world == ex->world && all[r]->rank == r && all[r]->L.total == ex->L.total, "mismatching exchange objects");
    ex->peer[r] = all[r]->arena;
    if (all[r]->ctx->device != ex->ctx->device) {
      cudaError_t e = cudaDeviceEnablePeerAccess(all[r]->ctx->device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { ppp_set_error("peer access %d -> %d: %s", ex->ctx->device, all[r]->ctx->device, cudaGetErrorString(e)); cudaGetLastError(); return PPP_ERR_CUDA; }
      cudaGetLastError();
    }
  }
  ex_refresh_view(ex);
  PPP_TRY(ex_upload_route(ex));
  ex->connected = true;
  return PPP_OK;
}

// Unmap the peers' arenas (after the last step; synchronises).  Ranks in different processes call this,
// meet at a barrier of their own, and only then destroy: an arena must not be freed while a peer still
// has it mapped.
int ppp_exch_disconnect(ppp_exch* ex) {
  if (!ex) return PPP_OK;
  EX_LOCK(ex);
  cudaSetDevice(ex->ctx->device);
  cudaDeviceSynchronize();
  for (int r = 0; r < ex->world; r++) {
    if (ex->ipc_opened[r]) { cudaIpcCloseMemHandle(ex->peer[r]); ex->ipc_opened[r] = false; }
    if (r != ex->rank) ex->peer[r] = nullptr;
  }
  cudaGetLastError();
  ex->connected = false;
  return PPP_OK;
}

int ppp_exch_destroy(ppp_exch* ex) {
  if (!ex) return PPP_OK;
  ppp_exch_disconnect(ex);
  {
    EX_LOCK(ex);
    cudaSetDevice(ex->ctx->device);
    cudaFree(ex->arena); cudaFree(ex->sc); cudaFree(ex->route); cudaFree(ex->rowmap); cudaFree(ex->tilecnt);
    cudaGetLastError();
  }
  delete ex;
  return PPP_OK;
}

// Enqueue one phase of the exchange of this rank's chunk (device records of stride_bytes, the file's
// records [starts[rank], starts[rank] + n)).  Phases 0..3 in order; a process that drives one rank calls
// them back to back, a process that drives several ranks issues phase p for every rank before p + 1.
int ppp_exch_phase(ppp_exch* ex, int phase, const void* chunk_dev, int64_t n, size_t stride_bytes, double halo) {
  if (!ex) { ppp_set_error("ppp_exch_phase: NULL argument"); return PPP_ERR_INVALID; }
  EX_REQUIRE(ex->connected, "not connected (ppp_exch_connect_ipc / _local)");
  EX_REQUIRE(phase >= 0 && phase <= 3, "phase must be 0..3");
  EX_REQUIRE(n >= 0 && (n == 0 || chunk_dev), "bad chunk");
  EX_REQUIRE(stride_bytes >= 12 && stride_bytes % 4 == 0, "stride_bytes must be >= 12 and a multiple of 4");
  EX_REQUIRE(n == ex->starts[ex->rank + 1] - ex->starts[ex->rank], "chunk size differs from this rank's index range");
  EX_REQUIRE(halo >= 0, "halo must be >= 0");
  ppp_ctx* ctx = ex->ctx;
  EX_LOCK(ex);
  PPP_CUDA(cudaSetDevice(ctx->device));
  const float* raw = (const float*)chunk_dev;
  const int sf = (int)(stride_bytes / 4);
  const int vec_ok = (stride_bytes % 16 == 0) && (((uintptr_t)chunk_dev) % 16 == 0);
  const int sweep_blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n + 1023) / 1024, (int64_t)ctx->sm_count * 4));
  const int ntiles = (int)std::max<int64_t>(1, (n + EX_TILE - 1) / EX_TILE);
  if (phase == 0) {
    ex->step++;
    ex->raw = raw; ex->n = n; ex->sf = sf; ex->vec_ok = vec_ok; ex->halo = halo; ex->ntiles = ntiles;
    PPP_LAUNCH(ctx, "ex_minmax", k_ex_minmax, sweep_blocks, EX_THREADS, 0, ex->V, raw, n, sf, vec_ok, ex->step, ex->sc);
    PPP_CHECK_LAUNCH();
    return PPP_OK;
  }
  EX_REQUIRE(raw == ex->raw && n == ex->n, "phases of one step must be given the same chunk");
  ex->halo = std::min(ex->halo, halo);
  if (phase == 1) {
    PPP_LAUNCH(ctx, "ex_wait", k_ex_wait, 1, 32, 0, ex->V, 0, ex->step, -1, ex->sc);
    // two 1024-thread blocks per SM: every block ends with one atomic per non-empty bin
    const int hist_blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n + 4095) / 4096, (int64_t)ctx->sm_count * 2));
    PPP_LAUNCH(ctx, "ex_hist", k_ex_hist, hist_blocks, 1024, 0, ex->V, raw, n, sf, vec_ok, ex->step, ex->sc);
    PPP_CHECK_LAUNCH();
  } else if (phase == 2) {
    if (ex->tilecnt_cap < (int64_t)ntiles * ex->world) {
      PPP_CUDA(cudaStreamSynchronize(ctx->stream));
      cudaFree(ex->tilecnt);
      ex->tilecnt = nullptr; ex->tilecnt_cap = 0;
      PPP_CUDA(cudaMalloc((void**)&ex->tilecnt, (size_t)ntiles * ex->world * sizeof(int32_t)));
      ex->tilecnt_cap = (int64_t)ntiles * ex->world;
    }
    PPP_LAUNCH(ctx, "ex_wait", k_ex_wait, 1, 32, 0, ex->V, 1, ex->step, -1, ex->sc);
    PPP_LAUNCH(ctx, "ex_count", k_ex_count, ntiles, EX_THREADS, 0, ex->V, raw, n, sf, vec_ok, halo, ex->step, ex->sc, ex->tilecnt, ntiles);
    PPP_CHECK_LAUNCH();
  } else {
    PPP_LAUNCH(ctx, "ex_wait", k_ex_wait, 1, 32, 0, ex->V, 2, ex->step, -1, ex->sc);
    PPP_LAUNCH(ctx, "ex_scatter", k_ex_scatter, ntiles, EX_THREADS, 0, ex->V, raw, n, sf, vec_ok, ex->starts[ex->rank], halo,
               ex->step, ex->sc, (const int32_t*)ex->tilecnt, ntiles);
    PPP_CHECK_LAUNCH();
  }
  return PPP_OK;
}

// Wait until every rank's records have landed, build the row map, fetch the summary (synchronises).
// cuts: world + 1 slab limits (cuts[0] = -inf, cuts[world] = +inf): rank r owns cuts[r] <= x < cuts[r+1];
// x_range: global finite x-range.  The received slab is the device array ppp_exch_slab().
int ppp_exch_finish(ppp_exch* ex, int64_t* n_local, int64_t* n_owned, double* cuts, double x_range[2]) {
  if (!ex) { ppp_set_error("ppp_exch_finish: NULL argument"); return PPP_ERR_INVALID; }
  ppp_ctx* ctx = ex->ctx;
  EX_LOCK(ex);
  PPP_CUDA(cudaSetDevice(ctx->device));
  PPP_LAUNCH(ctx, "ex_wait", k_ex_wait, 1, 32, 0, ex->V, 3, ex->step, -1, ex->sc);
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((ex->cap_recv + 255) / 256, (int64_t)ctx->sm_count * 8));
  PPP_LAUNCH(ctx, "ex_rowmap", k_ex_rowmap, blocks, 256, 0, ex->V, ex->sc, ex->rowmap);
  PPP_CHECK_LAUNCH();
  // summary: one fetch of the scratch block from the cut positions to the error word
  struct Summary {
    double cutx[PPP_MAX_RANKS + 1];
    double gmin, gmax, inv, halo_min;
    int32_t sendcnt[PPP_MAX_RANKS], sendown[PPP_MAX_RANKS];
    long long n_local, n_owned;
    int32_t err, pad;
  } sum;
  static_assert(offsetof(ExScratch, pad) + sizeof(int32_t) - offsetof(ExScratch, cutx) == sizeof(Summary), "summary mirrors the scratch tail");
  PPP_TRY(fetch_small(ctx, (const char*)ex->sc + offsetof(ExScratch, cutx), sizeof(sum), &sum));
  struct { long long n_local, n_owned; int32_t err; } tail = {sum.n_local, sum.n_owned, sum.err};
  struct { const double* cutx; double gmin, gmax; } mid = {sum.cutx, sum.gmin, sum.gmax};
  if (tail.err) {
    ppp_set_error(tail.err == 1 ? "ppp_exch_finish: timed out waiting for a peer rank"
                                : "ppp_exch_finish: receive buffer too small (cap_recv %lld)", (long long)ex->cap_recv);
    PPP_CUDA(cudaMemsetAsync((char*)ex->sc + offsetof(ExScratch, err), 0, sizeof(int32_t), ctx->stream));
    return tail.err == 1 ? PPP_ERR_CUDA : PPP_ERR_CAPACITY;
  }
  ex->n_local = tail.n_local;
  ex->xmag = std::max(std::fabs(mid.gmin), std::fabs(mid.gmax));
  ex->halo = std::min(ex->halo, sum.halo_min);
  if (n_local) *n_local = tail.n_local;
  if (n_owned) *n_owned = tail.n_owned;
  if (cuts) for (int r = 0; r <= ex->world; r++) cuts[r] = mid.cutx[r];
  if (x_range) { x_range[0] = mid.gmin; x_range[1] = mid.gmax; }
  return PPP_OK;
}

const void* ppp_exch_slab(ppp_exch* ex) { return ex ? (const void*)(ex->arena + ex->L.recv) : nullptr; }
const int32_t* ppp_exch_row_map(ppp_exch* ex) { return ex ? ex->rowmap : nullptr; }
void* ppp_exch_home_normals(ppp_exch* ex) { return ex ? (void*)(ex->arena + ex->L.home) : nullptr; }

// The received slab as a cloud (pack + bounding box as ppp_dev_cloud_attach), wired so that the normal
// estimators store every OWNED row's record into its home rank's buffer (halo rows are skipped) and,
// when to_rank0 != 0, ppp_dev_slice_contours writes its nodes and per-slice offsets into this rank's
// region of rank 0's arena.
int ppp_exch_attach(ppp_exch* ex, int to_rank0, ppp_cloud** out) {
  if (!ex || !out) { ppp_set_error("ppp_exch_attach: NULL argument"); return PPP_ERR_INVALID; }
  EX_LOCK(ex);
  PPP_TRY(ppp_dev_cloud_attach(ex->ctx, ex->arena + ex->L.recv, (size_t)ex->n_local, 16, out));
  (*out)->nmap = ex->rowmap;
  (*out)->route = ex->route;
  (*out)->ex_halo = ex->halo; (*out)->ex_xmag = ex->xmag; (*out)->ex_home_bytes = ex->home_sf * 4;
  if (to_rank0) {
    unsigned char* reg = ex->peer[0] + ex->L.nodes + (size_t)ex->rank * ex->L.node_region;
    PPP_TRY(ppp_dev_set_contour_offsets_buffer(*out, (int64_t*)reg, (int64_t)ex->S_cap + 1));
    if (ex->node_cap > 0)
      PPP_TRY(ppp_dev_set_contour_buffers(*out, (double*)(reg + ex->L.node_off_bytes), (double*)(reg + ex->L.node_off_bytes + ex->L.node_arr_bytes),
                                          (double*)(reg + ex->L.node_off_bytes + 2 * ex->L.node_arr_bytes), ex->node_cap));
  }
  return PPP_OK;
}

// ppp_exch_finish + ppp_exch_attach with ONE host synchronisation: the slab is ingested (pack, bounding box, density
// sample) straight behind the exchange kernels, the kernels take its size from device memory, and the exchange summary
// travels to the host with the ingest results.
int ppp_exch_finish_attach(ppp_exch* ex, int to_rank0, int64_t* n_local, int64_t* n_owned, double* cuts, double x_range[2],
                           ppp_cloud** out) {
  if (!ex || !out) { ppp_set_error("ppp_exch_finish_attach: NULL argument"); return PPP_ERR_INVALID; }
  ppp_ctx* ctx = ex->ctx;
  EX_LOCK(ex);
  PPP_CUDA(cudaSetDevice(ctx->device));
  PPP_LAUNCH(ctx, "ex_wait", k_ex_wait, 1, 32, 0, ex->V, 3, ex->step, -1, ex->sc);
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((ex->cap_recv + 255) / 256, (int64_t)ctx->sm_count * 8));
  PPP_LAUNCH(ctx, "ex_rowmap", k_ex_rowmap, blocks, 256, 0, ex->V, ex->sc, ex->rowmap);
  PPP_CHECK_LAUNCH();
  struct Summary {
    double cutx[PPP_MAX_RANKS + 1];
    double gmin, gmax, inv, halo_min;
    int32_t sendcnt[PPP_MAX_RANKS], sendown[PPP_MAX_RANKS];
    long long n_local, n_owned;
    int32_t err, pad;
  } sum;
  static_assert(offsetof(ExScratch, pad) + sizeof(int32_t) - offsetof(ExScratch, cutx) == sizeof(Summary), "summary mirrors the scratch tail");
  ppp_cloud* c = new ppp_cloud();
  c->ctx = ctx;
  c->n = 0;
  c->grids.reserve(48);
  c->mps.reserve(16);
  int st = cloud_ingest_ex(c, ex->arena + ex->L.recv, 16, ex->cap_recv, &ex->sc->n_local, (const char*)ex->sc + offsetof(ExScratch, cutx),
                           sizeof(sum), &sum);
  if (st == PPP_OK && sum.err) {
    ppp_set_error(sum.err == 1 ? "ppp_exch_finish_attach: timed out waiting for a peer rank"
                               : "ppp_exch_finish_attach: receive buffer too small (cap_recv %lld)", (long long)ex->cap_recv);
    cudaMemsetAsync((char*)ex->sc + offsetof(ExScratch, err), 0, sizeof(int32_t), ctx->stream);
    st = sum.err == 1 ? PPP_ERR_CUDA : PPP_ERR_CAPACITY;
  }
  if (st != PPP_OK) { ppp_cloud_free(c); return st; }
  ex->n_local = sum.n_local;
  ex->xmag = std::max(std::fabs(sum.gmin), std::fabs(sum.gmax));
  ex->halo = std::min(ex->halo, sum.halo_min);
  if (n_local) *n_local = sum.n_local;
  if (n_owned) *n_owned = sum.n_owned;
  if (cuts) for (int r = 0; r <= ex->world; r++) cuts[r] = sum.cutx[r];
  if (x_range) { x_range[0] = sum.gmin; x_range[1] = sum.gmax; }
  c->nmap = ex->rowmap;
  c->route = ex->route;
  c->ex_halo = ex->halo; c->ex_xmag = ex->xmag; c->ex_home_bytes = ex->home_sf * 4;
  if (to_rank0) {
    unsigned char* reg = ex->peer[0] + ex->L.nodes + (size_t)ex->rank * ex->L.node_region;
    st = ppp_dev_set_contour_offsets_buffer(c, (int64_t*)reg, (int64_t)ex->S_cap + 1);
    if (st == PPP_OK && ex->node_cap > 0)
      st = ppp_dev_set_contour_buffers(c, (double*)(reg + ex->L.node_off_bytes), (double*)(reg + ex->L.node_off_bytes + ex->L.node_arr_bytes),
                                       (double*)(reg + ex->L.node_off_bytes + 2 * ex->L.node_arr_bytes), ex->node_cap);
    if (st != PPP_OK) { ppp_cloud_free(c); return st; }
  }
  *out = c;
  return PPP_OK;
}

// Rank 0's view of rank r's contour region (device pointers into the own arena).
int ppp_exch_nodes_region(ppp_exch* ex, int r, const int64_t** offsets, const double** y, const double** x, const double** z) {
  if (!ex || r < 0 || r >= ex->world) { ppp_set_error("ppp_exch_nodes_region: bad argument"); return PPP_ERR_INVALID; }
  unsigned char* reg = ex->arena + ex->L.nodes + (size_t)r * ex->L.node_region;
  if (offsets) *offsets = (const int64_t*)reg;
  if (y) *y = (const double*)(reg + ex->L.node_off_bytes);
  if (x) *x = (const double*)(reg + ex->L.node_off_bytes + ex->L.node_arr_bytes);
  if (z) *z = (const double*)(reg + ex->L.node_off_bytes + 2 * ex->L.node_arr_bytes);
  return PPP_OK;
}

// Results phases.  what = PPP_EXCH_NORMALS (0): the normal records this rank's search kernels have stored
// into their home ranks; PPP_EXCH_CONTOURS (1): the contour nodes written to rank 0's region.
// signal: everything this rank has enqueued so far is in place -> flag in every arena.  wait: later work
// of the stream (and a host synchronise) sees every rank's results of that kind for this step: the home
// buffer holds the normals of the own index range / rank 0's regions hold all contours.  Signalling the
// normals before the slicing is enqueued lets the copy of the home buffer to the host run under it.
int ppp_exch_results_signal(ppp_exch* ex, int what) {
  if (!ex || what < 0 || what > 1) { ppp_set_error("ppp_exch_results_signal: bad argument"); return PPP_ERR_INVALID; }
  EX_LOCK(ex);
  PPP_CUDA(cudaSetDevice(ex->ctx->device));
  PPP_LAUNCH(ex->ctx, "ex_signal", k_ex_signal, 1, 32, 0, ex->V, 4 + what, ex->step);
  PPP_CHECK_LAUNCH();
  return PPP_OK;
}

int ppp_exch_results_wait(ppp_exch* ex, int what) {
  if (!ex || what < 0 || what > 1) { ppp_set_error("ppp_exch_results_wait: bad argument"); return PPP_ERR_INVALID; }
  EX_LOCK(ex);
  PPP_CUDA(cudaSetDevice(ex->ctx->device));
  PPP_LAUNCH(ex->ctx, "ex_wait", k_ex_wait, 1, 32, 0, ex->V, 4 + what, ex->step, -1, ex->sc);
  PPP_CHECK_LAUNCH();
  return PPP_OK;
}

// 0 if no wait of this exchange has timed out since the last call (synchronises the stream).
int ppp_exch_check(ppp_exch* ex) {
  if (!ex) { ppp_set_error("ppp_exch_check: NULL argument"); return PPP_ERR_INVALID; }
  EX_LOCK(ex);
  PPP_CUDA(cudaSetDevice(ex->ctx->device));
  int32_t err = 0;
  PPP_TRY(fetch_small(ex->ctx, (const char*)ex->sc + offsetof(ExScratch, err), sizeof(err), &err));
  if (err) {
    PPP_CUDA(cudaMemsetAsync((char*)ex->sc + offsetof(ExScratch, err), 0, sizeof(int32_t), ex->ctx->stream));
    ppp_set_error("ppp_exch_check: %s", err == 1 ? "timed out waiting for a peer rank" : "receive buffer overflow");
    return err == 1 ? PPP_ERR_CUDA : PPP_ERR_CAPACITY;
  }
  return PPP_OK;
}

// Page-lock an existing host range (e.g. a shared-memory mapping every rank's process has opened) so
// that host<->device copies run at full PCIe rate and kernels can store into it.  *dev_ptr (optional):
// the address kernels / ppp_dev_set_contour_buffers must use for the start of the range.
int ppp_host_register(void* p, size_t bytes, void** dev_ptr) {
  if (!p || !bytes) { ppp_set_error("ppp_host_register: NULL argument"); return PPP_ERR_INVALID; }
  cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped);
  if (e != cudaSuccess) { ppp_set_error("cudaHostRegister(%zu bytes): %s", bytes, cudaGetErrorString(e)); cudaGetLastError(); return PPP_ERR_CUDA; }
  if (dev_ptr) {
    e = cudaHostGetDevicePointer(dev_ptr, p, 0);
    if (e != cudaSuccess) { ppp_set_error("cudaHostGetDevicePointer: %s", cudaGetErrorString(e)); cudaGetLastError(); cudaHostUnregister(p); return PPP_ERR_CUDA; }
  }
  return PPP_OK;
}
int ppp_host_unregister(void* p) {
  if (!p) return PPP_OK;
  cudaError_t e = cudaHostUnregister(p);
  if (e != cudaSuccess) { ppp_set_error("cudaHostUnregister: %s", cudaGetErrorString(e)); cudaGetLastError(); return PPP_ERR_CUDA; }
  return PPP_OK;
}

// Stream-ordered copies between (page-locked) host memory and device buffers; no synchronisation.
int ppp_dev_upload(ppp_ctx* ctx, void* dev_dst, const void* host_src, size_t bytes) {
  if (!ctx || (bytes && (!dev_dst || !host_src))) { ppp_set_error("ppp_dev_upload: NULL argument"); return PPP_ERR_INVALID; }
  ApiScope scope(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  if (bytes) PPP_CUDA(cudaMemcpyAsync(dev_dst, host_src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  return PPP_OK;
}
int ppp_dev_download_async(ppp_ctx* ctx, void* host_dst, const void* dev_src, size_t bytes) {
  if (!ctx || (bytes && (!host_dst || !dev_src))) { ppp_set_error("ppp_dev_download_async: NULL argument"); return PPP_ERR_INVALID; }
  ApiScope scope(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  if (bytes) PPP_CUDA(cudaMemcpyAsync(host_dst, dev_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  return PPP_OK;
}

}  // extern "C"
