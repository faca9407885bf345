// Exact k-nearest-neighbour / radius search on the column grid, with the PCL normal estimation
// fused behind it.  Replaces pcl::KdTreeFLANN::nearestKSearch / radiusSearch and
// pcl::NormalEstimation::compute (src/Path_Generation.cpp:323-333, src/contour_alg.cpp:142-151).
//
// One thread per query, queries taken in sorted (cell-major) order so a warp's 32 queries share
// the same few cell rows: candidate loads are float4, contiguous per row and hit L1/L2.  The
// per-query result list lives in shared memory (column layout: entry j of thread t at
// [j*blockDim + t], bank = t, conflict-free) as 64-bit keys (d2 bits << 32 | index), so the
// reference's (d2, index) order is a single unsigned compare and the list is already in the
// order the PCL covariance must be accumulated in.
#include <stdlib.h>

#include <algorithm>
#include <cmath>

#include "ppp_device.cuh"
#include "sortnet.cuh"

namespace {

struct SearchParams {
  GridView g;
  const float4* xyz4;   // original order (neighbour gather for the covariance)
  const float* q;       // external queries (nullptr: the cloud's own points in sorted order)
  int q_sf;
  int64_t nq;
  int64_t first;        // self mode: first sorted position
  int cap;              // list capacity (k in k-mode)
  int kk;               // k-mode: min(k, indexed points)
  int mode;             // 0 = k nearest, 1 = radius (d2 < r2, fixed block radius R0)
  int R0;
  float r2;
  int32_t* idx_out;     // k-mode: row*cap ; radius mode: offsets[row]
  float* d2_out;
  const int64_t* offsets;
  float* normals;
  const int32_t* nmap;  // optional row map for the normal records (row -> record, < 0: not stored)
  const NormalRoute* route;  // optional: records go to their home rank's buffer (multi-GPU)
  int nsf;
  float vpx, vpy, vpz;
  unsigned flags;
  // fast path -> generic path hand-over: queries the fixed-radius fast kernel could not finish
  int32_t* redo_list;   // query numbers t (fast kernel appends; generic kernel consumes)
  int32_t* redo_count;
  int use_redo;         // generic kernel: take the query number from redo_list[thread]
  // multi-projection index: this launch answers only the self-queries whose point chose projection my_proj
  const unsigned char* choice;   // per original index, nullptr: every query
  int my_proj;
};

// Query t: row t of the query array P.q (ext), or the t-th of the cloud's own points in cell order, whose row is its
// original index.
__device__ __forceinline__ void load_query(const SearchParams& P, bool ext, int64_t t, float& qx, float& qy, float& qz,
                                           int64_t& row) {
  if (ext) {
    const float* qp = P.q + t * P.q_sf;
    qx = __ldg(qp); qy = __ldg(qp + 1); qz = __ldg(qp + 2);
    row = t;
  } else {
    float4 p = __ldg(P.g.sorted + P.first + t);
    qx = p.x; qy = p.y; qz = p.z;
    row = __float_as_int(p.w);
  }
}

// Self-query `row` belongs to this launch?  (Warps none of whose lanes do leave at once.)
__device__ __forceinline__ bool query_is_mine(const SearchParams& P, bool valid, int64_t row) {
  return valid && (P.choice == nullptr || __ldg(P.choice + row) == P.my_proj);
}

__device__ __forceinline__ void list_insert(u64* L, int BD, int& cnt, int cap, u64 key) {
  int j = cnt < cap ? cnt++ : cap - 1;
  while (j > 0) {
    u64 prev = L[(j - 1) * BD];
    if (prev < key) break;
    L[j * BD] = prev;
    j--;
  }
  L[j * BD] = key;
}

__global__ void __launch_bounds__(128) k_search(SearchParams P) {
  pdl_prologue();
  extern __shared__ u64 s_keys[];
  const int BD = blockDim.x;
  int64_t t = (int64_t)blockIdx.x * BD + threadIdx.x;
  if (P.use_redo) {
    if (t >= *P.redo_count) return;
    t = P.redo_list[t];
  } else if (t >= P.nq) {
    return;
  }
  const GridView& g = P.g;
  float qx, qy, qz;
  int64_t row;
  load_query(P, P.q != nullptr, t, qx, qy, qz, row);
  if (!P.use_redo && P.choice && __ldg(P.choice + row) != P.my_proj) return;
  u64* L = s_keys + threadIdx.x;
  int cnt = 0;
  const bool fin = finite3(qx, qy, qz);
  if (fin && g.n_sorted > 0) {
    int cu = cell_coord_raw(axis_of(qx, qy, qz, g.au), g.min_u, g.inv_h);
    int cv = cell_coord_raw(axis_of(qx, qy, qz, g.av), g.min_v, g.inv_h);
    if (P.mode == 1) {
      u64 tau = make_key(P.r2, 0);
      visit_annulus(g, cu, cv, -1, P.R0, [&](float4 c) {
        u64 key = make_key(d2_flann(qx, qy, qz, c.x, c.y, c.z), __float_as_int(c.w));
        if (key < tau) {
          list_insert(L, BD, cnt, P.cap, key);
          if (cnt == P.cap) tau = min(tau, L[(P.cap - 1) * BD] + 1);  // full: keep the cap smallest
        }
      });
    } else {
      u64 tau = PPP_KEY_INF;
      // queries outside the gridded rectangle: skip the rings that cannot contain any cell
      int du = max(max(-cu, cu - (g.nu - 1)), 0), dv = max(max(-cv, cv - (g.nv - 1)), 0);
      int R = max(P.R0, max(du, dv));
      int R_prev = -1;
      while (true) {
        visit_annulus(g, cu, cv, R_prev, R, [&](float4 c) {
          u64 key = make_key(d2_flann(qx, qy, qz, c.x, c.y, c.z), __float_as_int(c.w));
          if (key < tau) {
            list_insert(L, BD, cnt, P.cap, key);
            if (cnt == P.cap) tau = L[(P.cap - 1) * BD];
          }
        });
        if (cnt >= P.kk && (P.kk == 0 || key_d2(L[(P.kk - 1) * BD]) < ring_bound2(g, R, cu, cv))) break;
        if (block_covers_grid(g, cu, cv, R)) break;
        R_prev = R;
        R++;
      }
    }
  }
  // ---- outputs ----
  if (P.idx_out) {
    if (P.mode == 0) {
      int32_t* io = P.idx_out + row * (int64_t)P.cap;
      float* dout = P.d2_out ? P.d2_out + row * (int64_t)P.cap : nullptr;
      for (int j = 0; j < P.cap; j++) {
        u64 key = j < cnt ? L[j * BD] : 0;
        io[j] = j < cnt ? key_idx(key) : -1;
        if (dout) dout[j] = j < cnt ? key_d2(key) : CUDART_INF_F;
      }
    } else {
      int64_t o = P.offsets[row];
      for (int j = 0; j < cnt; j++) {
        u64 key = L[j * BD];
        P.idx_out[o + j] = key_idx(key);
        if (P.d2_out) P.d2_out[o + j] = key_d2(key);
      }
    }
  }
  if (P.normals) {
    float o[4];
    if (!fin || cnt < 3) {
      o[0] = o[1] = o[2] = o[3] = CUDART_NAN_F;
    } else {
      float acc[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      float kx = 0.f, ky = 0.f, kz = 0.f;
      const bool shifted = (P.flags & PPP_COV_SHIFTED) != 0;
      if (shifted) {
        float4 f = __ldg(P.xyz4 + key_idx(L[0]));
        kx = f.x; ky = f.y; kz = f.z;
      }
      for (int j = 0; j < cnt; j++) {
        float4 a = __ldg(P.xyz4 + key_idx(L[j * BD]));
        float x = a.x, y = a.y, z = a.z;
        if (shifted) { x = __fsub_rn(x, kx); y = __fsub_rn(y, ky); z = __fsub_rn(z, kz); }
        accumulate_point(acc, x, y, z);
      }
      normal_from_accumulators(acc, cnt, qx, qy, qz, P.vpx, P.vpy, P.vpz, o);
    }
    store_normal(P.normals, P.nmap, row, P.nsf, o, P.route);
  }
}


// ---------------------------------------------------------------------------------------------
// k <= 64: 32-bit FIXED-POINT keys.  The queries are the cloud's own points in cell order or, with EXT, a query
// array (its row t is the query's position); only the load of the query differs.
//     key = floor(d2 * scale) << SH | ordinal         scale = (2^(32 - SH) - margin) / (ring bound)^2  per query
// Candidates arrive uniformly in d2 (area), so 22 bits of fixed point over [0, bound^2] resolve the k-th
// neighbourhood nearly as finely as the float itself does (2.2e-6 mm^2 at cfg2 against an ulp of 4.8e-7), where a
// truncated float spends its bits on the nearest neighbours.  The ordinal (SH = 3 + RB bits) names the candidate by
// (row of the block, slot in the row); its sorted position is rebuilt from the row start at the very end, and the
// exact d2 -- needed only if the caller asked for distances -- is recomputed from the gathered record with the same
// arithmetic.  So the per-thread store is 4 bytes per slot and the sorted words ARE the result.  floor(d2 * scale) is
// one FFMA.RZ against 2^23 (exact floor of the real product: monotone in d2).
// Slots 0..K-1 hold the K best so far in order (free values behind the keys), slots K..K+NEW-1 take the newcomers; a
// flush sorts the newcomers, folds them into the kept K with one row of minima (the half-cleaner of a bitonic merge)
// and a K-input bitonic merge, every exchange one unsigned min + one unsigned max, and writes the K words back.
// Before the first flush the newcomers start at slot FIRST: FIRST = K leaves slots 0..K-1 to the free values, which
// are in order from the start; FIRST = 0 uses all K + NEW slots for them, and the first flush sorts slots 0..K-1 too.
// Two candidates whose keys agree in the fixed-point bits (including the best one just dropped) leave their order to
// the exact hand-over kernel k_knn_warp.
//   K = 16: 16 newcomers, FIRST = 0, ordinals of 3 + 7 bits (rows of up to 128 candidates), 22 bits of d2.
//   K = 32: 16 newcomers (63 + 80 exchanges per flush), ordinals of 3 + 6 bits, 23 bits of d2.
//   K = 64: 32 newcomers (191 + 192 exchanges), ordinals of 3 + 7 bits, 22 bits of d2 -- the list lives in 96
//   registers during a flush.
// ---------------------------------------------------------------------------------------------
constexpr int F_MAXR = 3;
static_assert(PPP_KNN_RINGS <= F_MAXR, "the ordinal names the block row in 3 bits: 2 R0 + 1 <= 7");

// Free value of slot j with SH ordinal bits: above every key (fixed-point values stay below 2^(32 - SH) - 608), and
// distinct in the fixed-point bits from every other free slot, so free slots never look like an undecided pair.
template <int SH>
__device__ constexpr unsigned free_word(int j) {
  return (((1u << (32 - SH)) - 128u + (unsigned)j) << SH) | ((1u << SH) - 1u);
}

template <int K, int NEW, int RB, int BD, int MB, int FIRST, bool EXT>
__global__ void __launch_bounds__(BD, MB) k_knnf(SearchParams P) {
  static_assert(FIRST == 0 || FIRST == K, "newcomers start at slot 0 or behind the kept K");
  pdl_prologue();
  extern __shared__ __align__(128) unsigned s_fkeys[];
  constexpr int SLOTS = K + NEW;
  constexpr int PPP_ASSERT_SLOTS = SLOTS;
  constexpr int SH = 3 + RB;                        // ordinal bits: row of the block, slot in the row
  constexpr unsigned OMASK = (1u << SH) - 1u;
  constexpr unsigned FIXTOP = 1u << (32 - SH);      // fixed-point values stay below FIXTOP - 608
  constexpr int ROWCAP = 1 << RB;
  static_assert(ROWCAP + 4 <= PPP_SORTED_PAD, "unclamped candidate loads run up to ROWCAP + 3 records past a row");
  static_assert(SLOTS <= 128, "free values are FIXTOP - 128 + slot");
  constexpr unsigned FREE0 = free_word<SH>(0);
  const GridView& g = P.g;
  const int64_t t = (int64_t)blockIdx.x * BD + threadIdx.x;
  bool valid = t < P.nq;
  float qx = 0.f, qy = 0.f, qz = 0.f;
  int64_t row = 0;
  if (valid) load_query(P, EXT, t, qx, qy, qz, row);
  valid = query_is_mine(P, valid, row);
  if (P.choice && !__any_sync(0xffffffffu, valid)) return;   // none of this warp's points chose this projection
  const bool fin = valid && finite3(qx, qy, qz);
  const bool act = fin && g.n_sorted > 0;
  unsigned* keys = s_fkeys + threadIdx.x;                     // slot j of this thread at keys[j * BD]
  int* rows = (int*)(s_fkeys + SLOTS * BD) + threadIdx.x;     // first sorted position of block row j at rows[j * BD]
  const unsigned keys_sa = (unsigned)__cvta_generic_to_shared(keys);
  constexpr unsigned SLOT_B = BD * 4;
  const int R = P.R0;
  const int kk = P.kk;       // neighbours wanted (<= K)
  int cu = 0, cv = 0;
  float tau = -1.0f, scale = 0.0f;   // inactive lanes accept nothing
  if (act) {
    cu = cell_coord_raw(axis_of(qx, qy, qz, g.au), g.min_u, g.inv_h);
    cv = cell_coord_raw(axis_of(qx, qy, qz, g.av), g.min_v, g.inv_h);
    tau = ring_bound2(g, R, cu, cv);
    scale = tau > 0.0f ? fminf(__fdiv_rd((float)(FIXTOP - 608u), tau), 3.0e38f) : 0.0f;   // d2 <= tau  =>  d2 * scale < FIXTOP - 608
  }
#pragma unroll
  for (int i = 0; i < SLOTS; i++) keys[i * BD] = free_word<SH>(i);   // ascending: slots 0..K-1 are "in order" from the start
  const u64 qxy = pack2(qx, qy);
  bool ambiguous = false, overflow = false;
  bool in_order = FIRST == K;   // slots 0..K-1 are sorted (warp-uniform: flushes are)
  unsigned wsa = keys_sa + (unsigned)FIRST * SLOT_B;   // cursor of the newcomers

  auto flush = [&]() {
    unsigned b[NEW];
#pragma unroll
    for (int i = 0; i < NEW; i++) b[i] = keys[(K + i) * BD];
    SortNetU32<NEW>::sort(b);
    unsigned a[K];
#pragma unroll
    for (int i = 0; i < K; i++) a[i] = keys[i * BD];
    if constexpr (FIRST == 0) {
      if (!in_order) SortNetU32<K>::sort(a);
      in_order = true;
    }
    // kept (ascending) ++ newcomers (descending) is bitonic: the half-cleaner leaves the K smallest in a[]; the
    // smallest of what it discards is the (K+1)-th of the union
    unsigned next = 0xFFFFFFFFu;
#pragma unroll
    for (int i = K - NEW; i < K; i++) {
      const unsigned o = b[K - 1 - i];
      next = min(next, max(a[i], o));
      a[i] = min(a[i], o);
    }
    SortNetU32<K>::bitonic_merge(a);
    // equal fixed-point bits: the order of the two is left to the exact kernel (free values differ from each other and
    // from every key there)
    ambiguous |= (a[K - 1] ^ next) <= OMASK;
#pragma unroll
    for (int i = 0; i + 1 < K; i++) ambiguous |= (a[i] ^ a[i + 1]) <= OMASK;
#pragma unroll
    for (int i = 0; i < K; i++) keys[i * BD] = a[i];
#pragma unroll
    for (int i = 0; i < NEW; i++) keys[(K + i) * BD] = free_word<SH>(K + i);
    // newcomers go to slots K.. from now on, also when fewer than K slots hold keys: slots 0..K-1 stay in order
    wsa = keys_sa + (unsigned)K * SLOT_B;
    // every d2 whose key could still sort at or before the kk-th: floor(d2 * scale) <= F  =>  d2 < (F + 1) / scale
    if (kk > 0) {
      const unsigned kth = keys[(kk - 1) * BD];
      if (kth < FREE0) tau = fminf(tau, __fdiv_ru((float)((kth >> SH) + 1u), scale));
    }
  };

  constexpr int U = 4;
  const unsigned trig_sa = keys_sa + (unsigned)(K + NEW - U) * SLOT_B;   // room for one more iteration?
#pragma unroll 1
  for (int j = 0; j <= 2 * R + 1; j++) {
    const int dv = (j & 1) ? -((j + 1) >> 1) : (j >> 1);  // rows nearest first
    int s = 0, cnt = 0;
    const int v = cv + dv;
    const bool drain = j == 2 * R + 1;
    if (!drain && act && v >= 0 && v < g.nv) {
      int a0 = max(cu - R, 0), b0 = min(cu + R, g.nu - 1);
      if (a0 <= b0) {
        const int32_t* rowp = g.cell_start + (int64_t)v * g.nu;
        s = __ldg(rowp + a0);
        cnt = __ldg(rowp + b0 + 1) - s;
      }
    }
    if (!drain) rows[j * BD] = s;
    if (cnt > ROWCAP) { overflow = true; cnt = ROWCAP; }   // the ordinal cannot name more: exact path
    // the drain pseudo-row runs one empty iteration whose flush is unconditional
    const int n_it = (__reduce_max_sync(0xffffffffu, cnt) + U - 1) / U + (drain ? 1 : 0);
    const unsigned trig = drain ? 0u : trig_sa;
    int i0 = s;
    int rem = cnt;
    unsigned ord = (unsigned)j << RB;
#pragma unroll 1
    for (int it = 0; it < n_it; it++, i0 += U, ord += U, rem -= U) {
      float4 c4[U];
      PPP_DEV_ASSERT(i0 >= 0 && i0 + U - 1 < g.n_sorted + PPP_SORTED_PAD);
#pragma unroll
      for (int u = 0; u < U; u++) c4[u] = __ldg(g.sorted + (i0 + u));   // never clamped: see PPP_SORTED_PAD
#pragma unroll
      for (int u = 0; u < U; u++) {
        const float d2 = d2_flann_x2(qxy, qz, c4[u]);
        if (u < rem && d2 <= tau) {
          // floor(d2 * scale) sits in the low mantissa bits of the sum; the multiplication shifts the exponent out
          const unsigned key = __float_as_uint(__fmaf_rz(d2, scale, 8388608.0f)) * (1u << SH) + ord + (unsigned)u;
          PPP_DEV_ASSERT(wsa >= keys_sa && wsa < keys_sa + (unsigned)(PPP_ASSERT_SLOTS) * SLOT_B);
          asm volatile("st.shared.b32 [%0], %1;" ::"r"(wsa), "r"(key) : "memory");
          wsa += SLOT_B;
        }
      }
      if (__any_sync(0xffffffffu, wsa > trig)) flush();
    }
  }
  if (!valid) return;
  bool complete = !act || kk == 0;
  if (!complete) complete = keys[(kk - 1) * BD] < FREE0;
  if (!complete || ambiguous || overflow) {
    P.redo_list[atomicAdd(P.redo_count, 1)] = (int32_t)t;
    return;
  }
  const int k = P.cap;
  int m = 0;   // neighbours found: keys come first in slots 0..K-1
  if (act) {
    if (keys[(K - 1) * BD] < FREE0) {
      m = K;
    } else {
#pragma unroll
      for (int step = K / 2; step >= 1; step >>= 1)
        if (keys[(m + step - 1) * BD] < FREE0) m += step;
    }
    m = min(m, k);
  }
  int32_t* io = P.idx_out ? P.idx_out + row * (int64_t)k : nullptr;
  float* dout = (P.idx_out && P.d2_out) ? P.d2_out + row * (int64_t)k : nullptr;
  const bool al32 = (k & 7) == 0 && (((uintptr_t)P.idx_out | (uintptr_t)P.d2_out) & 31) == 0;
  const bool want_n = P.normals && fin && m >= 3;
  const bool shifted = (P.flags & PPP_COV_SHIFTED) != 0;
  float acc[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float kx = 0.f, ky = 0.f, kz = 0.f;
  // eight neighbours at a time; ONE gather of the neighbour's sorted record serves the id list, the covariance
  // and (if asked for) the exact distance.  K = 16 unrolls its two blocks of eight (the rolled loop spills twice as
  // much there); K = 32 / 64 keep one copy of the loop body.
  constexpr bool UNROLL = K <= 16;
#pragma unroll (UNROLL ? K / 8 : 1)
  for (int jb = 0; jb < (UNROLL ? K : k); jb += 8) {
    if (UNROLL && jb >= k) break;
    float4 nb[8];
#pragma unroll
    for (int u = 0; u < 8; u++) {
      nb[u] = make_float4(0.f, 0.f, 0.f, __int_as_float(-1));
      if (jb + u < m) {   // a free value names no row
        const unsigned key = keys[(jb + u) * BD];
        const int rj = (int)((key >> RB) & 7u), pos = rows[rj * BD] + (int)(key & (unsigned)(ROWCAP - 1));
        PPP_DEV_ASSERT(rj <= 2 * R && pos >= 0 && pos < g.n_sorted);
        nb[u] = __ldg(g.sorted + pos);
      }
    }
    if (io) {
      float dd[8];
      if (dout) {
#pragma unroll
        for (int u = 0; u < 8; u++) dd[u] = jb + u < m ? d2_flann(qx, qy, qz, nb[u].x, nb[u].y, nb[u].z) : CUDART_INF_F;
      }
      if (al32) {
        // rows of a multiple of 8 neighbours are 32-byte aligned: one 256-bit store per eight ids instead of eight
        st_global_256(io + jb, nb[0].w, nb[1].w, nb[2].w, nb[3].w, nb[4].w, nb[5].w, nb[6].w, nb[7].w);
        if (dout) {
          reinterpret_cast<float4*>(dout + jb)[0] = make_float4(dd[0], dd[1], dd[2], dd[3]);
          reinterpret_cast<float4*>(dout + jb)[1] = make_float4(dd[4], dd[5], dd[6], dd[7]);
        }
      } else {
#pragma unroll
        for (int u = 0; u < 8; u++) {
          if (jb + u < k) {
            io[jb + u] = __float_as_int(nb[u].w);
            if (dout) dout[jb + u] = dd[u];
          }
        }
      }
    }
    if (want_n) {
      if (jb == 0 && shifted) { kx = nb[0].x; ky = nb[0].y; kz = nb[0].z; }
#pragma unroll
      for (int u = 0; u < 8; u++) {
        if (jb + u < m) {
          float x = nb[u].x, y = nb[u].y, z = nb[u].z;
          if (shifted) { x = __fsub_rn(x, kx); y = __fsub_rn(y, ky); z = __fsub_rn(z, kz); }
          accumulate_point(acc, x, y, z);
        }
      }
    }
  }
  if (P.normals) {
    float o[4];
    if (want_n) normal_from_accumulators(acc, m, qx, qy, qz, P.vpx, P.vpy, P.vpz, o);
    else o[0] = o[1] = o[2] = o[3] = CUDART_NAN_F;
    store_normal(P.normals, P.nmap, row, P.nsf, o, P.route);
  }
}

// ---------------------------------------------------------------------------------------------
// Fixed-radius normals (NormalEstimation::setRadiusSearch, the reference's default r = 2.5) with
// 32-bit COMPOSITE sort keys.  Every candidate with d2 < r2 is parked, unmoved, in a shared-memory
// store per thread (full 64-bit keys).  At the end ONE 32-input Batcher network sorts the composite keys
//     c = (bits(d2) & ~31) | slot
// (a compare-exchange is one unsigned min + one unsigned max: 2 instructions instead of 6 for 64-bit
// keys), and the covariance is accumulated by walking the slots in that order.  Dropping 5 mantissa
// bits can only misorder two candidates whose d2 agree in the upper 27 bits; a query with such a pair,
// or with more than C_SLOTS neighbours, goes to the hand-over kernels (exact for any count), so every
// accumulation runs in the exact (d2, index) order.
// ---------------------------------------------------------------------------------------------
constexpr int C_SLOTS = 32;   // keys ordered per network pass
constexpr int C_STORE = 36;   // storage slots: U spare ones, so a query overflows only beyond 32 neighbours

__global__ void __launch_bounds__(128, 6) k_radius_normals32(SearchParams P) {
  pdl_prologue();
  extern __shared__ u64 s_keys[];
  constexpr int BD = 128;
  constexpr int U = 4;
  const int64_t t = (int64_t)blockIdx.x * BD + threadIdx.x;
  const GridView& g = P.g;
  bool valid = t < P.nq;
  float qx = 0.f, qy = 0.f, qz = 0.f;
  int64_t row = 0;
  if (valid) {
    float4 p = __ldg(g.sorted + P.first + t);
    qx = p.x; qy = p.y; qz = p.z;
    row = __float_as_int(p.w);
  }
  valid = query_is_mine(P, valid, row);
  if (P.choice && !__any_sync(0xffffffffu, valid)) return;
  const bool act = valid && g.n_sorted > 0;  // self queries are finite by construction
  u64* store = s_keys + threadIdx.x;
  const int R = P.R0;
  int cu = 0, cv = 0;
  u64 tau = 0;
  if (act) {
    cu = cell_coord_raw(axis_of(qx, qy, qz, g.au), g.min_u, g.inv_h);
    cv = cell_coord_raw(axis_of(qx, qy, qz, g.av), g.min_v, g.inv_h);
    tau = make_key(P.r2, 0);
  }
  int ns = 0;
  bool overflow = false;
#pragma unroll 1
  for (int dv = -R; dv <= R; dv++) {
    int s = 0, e = 0;
    int v = cv + dv;
    if (act && v >= 0 && v < g.nv) {
      int a = max(cu - R, 0), b = min(cu + R, g.nu - 1);
      if (a <= b) {
        const int32_t* rowp = g.cell_start + (int64_t)v * g.nu;
        s = __ldg(rowp + a);
        e = __ldg(rowp + b + 1);
      }
    }
    const int n_it = (__reduce_max_sync(0xffffffffu, e - s) + U - 1) / U;
#pragma unroll 1
    for (int it = 0; it < n_it; it++) {
      float4 c4[U];
      bool in[U];
#pragma unroll
      for (int u = 0; u < U; u++) {
        int i = s + it * U + u;
        in[u] = i < e;
        c4[u] = __ldg(g.sorted + (in[u] ? i : 0));
      }
      u64* wptr = store + ns * BD;
#pragma unroll
      for (int u = 0; u < U; u++) {
        float d2 = d2_flann_x2(pack2(qx, qy), qz, c4[u]);
        u64 key = make_key(d2, __float_as_int(c4[u].w));
        if (in[u] && key < tau) {
          *wptr = key;
          wptr += BD;
        }
      }
      ns = (int)(wptr - store) / BD;
      if (ns > C_STORE - U) { overflow = true; tau = 0; }  // no room for another U candidates: hand over
    }
  }
  if (!valid) return;
  unsigned c[C_SLOTS];
#pragma unroll
  for (int i = 0; i < C_SLOTS; i++) {
    unsigned hi = (unsigned)(store[i * BD] >> 32);
    c[i] = i < ns ? ((hi & 0xFFFFFFE0u) | (unsigned)i) : 0xFFFFFFFFu;
  }
  SortNetU32<C_SLOTS>::sort(c);
  bool ambiguous = false;
#pragma unroll
  for (int i = 0; i + 1 < C_SLOTS; i++) ambiguous |= (i + 1 < ns) && ((c[i] ^ c[i + 1]) < 32u);
  if (overflow || ns > C_SLOTS || ambiguous) {
    int slot = atomicAdd(P.redo_count, 1);
    P.redo_list[slot] = (int32_t)t;
    return;
  }
  float o[4];
  const int m = ns;
  if (!act || m < 3) {
    o[0] = o[1] = o[2] = o[3] = CUDART_NAN_F;
  } else {
    float acc[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const bool shifted = (P.flags & PPP_COV_SHIFTED) != 0;
    float kx = 0.f, ky = 0.f, kz = 0.f;
    if (shifted) {
      float4 f = __ldg(P.xyz4 + key_idx(store[(c[0] & 31u) * BD]));
      kx = f.x; ky = f.y; kz = f.z;
    }
#pragma unroll
    for (int jb = 0; jb < C_SLOTS; jb += 4) {
      if (jb < m) {
        float4 a[4];
#pragma unroll
        for (int u = 0; u < 4; u++)
          if (jb + u < m) a[u] = __ldg(P.xyz4 + key_idx(store[(c[jb + u] & 31u) * BD]));
#pragma unroll
        for (int u = 0; u < 4; u++) {
          if (jb + u < m) {
            float x = a[u].x, y = a[u].y, z = a[u].z;
            if (shifted) { x = __fsub_rn(x, kx); y = __fsub_rn(y, ky); z = __fsub_rn(z, kz); }
            accumulate_point(acc, x, y, z);
          }
        }
      }
    }
    normal_from_accumulators(acc, m, qx, qy, qz, P.vpx, P.vpy, P.vpz, o);
  }
  store_normal(P.normals, P.nmap, row, P.nsf, o, P.route);
}

// ---------------------------------------------------------------------------------------------
// Ring-expanding k-nearest search, one WARP per query: the hand-over path of k_knnf (sparse
// regions, cloud borders, near-ties, dense rows; typically well under 1% of the queries).  The 32 lanes stride over the
// candidates of each ring (coalesced), each lane keeps its own sorted list of at most k keys in
// shared memory, and after every ring the k smallest of the 32 lists are extracted with warp-wide
// 64-bit min reductions to test the exactness bound.  A thread-per-query kernel is latency-bound
// here: few queries, each a long chain of dependent loads.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ u64 warp_min_u64(u64 v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    u64 t = __shfl_xor_sync(0xffffffffu, v, o);
    v = t < v ? t : v;
  }
  return v;
}

constexpr int WARPQ_WARPS = 4;

constexpr int WQ_SEG_MAX = 128;   // cell ranges of one ring handled in the flattened way (rings up to 31)

__global__ void __launch_bounds__(WARPQ_WARPS * 32) k_knn_warp(SearchParams P) {
  pdl_prologue();
  extern __shared__ u64 s_keys[];
  __shared__ int s_seg[WARPQ_WARPS][WQ_SEG_MAX];
  __shared__ int s_pre[WARPQ_WARPS][WQ_SEG_MAX + 1];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const GridView& g = P.g;
  const int k = P.cap, kk = P.kk;
  u64* L = s_keys + (size_t)w * 32 * k + lane;  // entry j of this lane at L[j * 32]
  const int n_redo = *P.redo_count;
  // persistent warps: the number of hand-over queries is only known on the device
  for (int64_t slot = (int64_t)blockIdx.x * WARPQ_WARPS + w; slot < n_redo; slot += (int64_t)gridDim.x * WARPQ_WARPS) {
  const int64_t t = P.redo_list[slot];
  float qx, qy, qz;
  int64_t row;
  load_query(P, P.q != nullptr, t, qx, qy, qz, row);
  const int cu = cell_coord_raw(axis_of(qx, qy, qz, g.au), g.min_u, g.inv_h);
  const int cv = cell_coord_raw(axis_of(qx, qy, qz, g.av), g.min_v, g.inv_h);
  int cnt = 0;
  u64 tau = PPP_KEY_INF;  // warp-uniform acceptance threshold (k-th best after the last ring)
  u64 mine = PPP_KEY_INF;  // lane j ends up holding the j-th nearest key ...
  u64 mine2 = PPP_KEY_INF; // ... and the (32+j)-th (k <= 64)
  int du = max(max(-cu, cu - (g.nu - 1)), 0), dv0 = max(max(-cv, cv - (g.nv - 1)), 0);
  int R = max(P.R0, max(du, dv0));
  int R_prev = -1;
  while (true) {
    // annulus R_prev < max(|du|,|dv|) <= R.  Its cell ranges (one per row, two for the rows that only add the
    // two outer column strips) are looked up by all lanes at once, then the lanes stride over the CONCATENATION
    // of the ranges with four candidates in flight each: a query costs a couple of dependent memory latencies
    // per ring instead of two per row (this kernel is latency-bound: a few hundred queries, one warp each).
    const int v0 = max(cv - R, 0), v1 = min(cv + R, g.nv - 1);
    const int nseg = 2 * (v1 - v0 + 1);
    if (nseg > 0 && nseg <= WQ_SEG_MAX) {
      int* seg_s = s_seg[w];
      int* seg_p = s_pre[w];
      for (int sg0 = 0; sg0 < nseg; sg0 += 32) {
        const int sg = sg0 + lane;
        int s0 = 0, len = 0;
        if (sg < nseg) {
          const int v = v0 + (sg >> 1), part = sg & 1;
          const bool full = abs(v - cv) > R_prev;
          int a, b;
          if (full) { a = max(cu - R, 0); b = part == 0 ? min(cu + R, g.nu - 1) : -1; }
          else if (part == 0) { a = max(cu - R, 0); b = min(cu - R_prev - 1, g.nu - 1); }
          else { a = max(cu + R_prev + 1, 0); b = min(cu + R, g.nu - 1); }
          if (a <= b) {
            const int32_t* rowp = g.cell_start + (int64_t)v * g.nu;
            s0 = __ldg(rowp + a);
            len = __ldg(rowp + b + 1) - s0;
          }
        }
        // exclusive prefix of the lengths (warp scan, carried over the chunks of 32 segments)
        int inc = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int tt = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += tt; }
        const int carry = sg0 == 0 ? 0 : seg_p[sg0];
        if (sg < nseg) { seg_s[sg] = s0; seg_p[sg + 1] = carry + inc; }
        if (sg0 == 0 && lane == 0) seg_p[0] = 0;
        __syncwarp();
      }
      const int T = seg_p[nseg];
      for (int base = 0; base < T; base += 128) {
        float4 c4[4];
        bool in[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int i = base + u * 32 + lane;
          in[u] = i < T;
          int lo = 0, hi = nseg - 1;           // last segment whose prefix is <= i
          while (lo < hi) { int mid = (lo + hi + 1) >> 1; if (seg_p[mid] <= i) lo = mid; else hi = mid - 1; }
          c4[u] = __ldg(g.sorted + (in[u] ? seg_s[lo] + (i - seg_p[lo]) : 0));
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
          if (!in[u]) continue;
          u64 key = make_key(d2_flann(qx, qy, qz, c4[u].x, c4[u].y, c4[u].z), __float_as_int(c4[u].w));
          // a full lane list only takes keys below its own last entry (list_insert overwrites it)
          if (key < tau && (cnt < k || key < L[(k - 1) * 32])) list_insert(L, 32, cnt, k, key);
        }
      }
    } else {
    for (int v = v0; v <= v1; v++) {
      const int32_t* rowp = g.cell_start + (int64_t)v * g.nu;
      const bool full = abs(v - cv) > R_prev;
      for (int part = 0; part < (full ? 1 : 2); part++) {
        int a, b;
        if (full) { a = max(cu - R, 0); b = min(cu + R, g.nu - 1); }
        else if (part == 0) { a = max(cu - R, 0); b = min(cu - R_prev - 1, g.nu - 1); }
        else { a = max(cu + R_prev + 1, 0); b = min(cu + R, g.nu - 1); }
        if (a > b) continue;
        const int s = __ldg(rowp + a), e = __ldg(rowp + b + 1);
        for (int i = s + lane; i < e; i += 32) {
          float4 c = __ldg(g.sorted + i);
          u64 key = make_key(d2_flann(qx, qy, qz, c.x, c.y, c.z), __float_as_int(c.w));
          // a full lane list only takes keys below its own last entry (list_insert overwrites it)
          if (key < tau && (cnt < k || key < L[(k - 1) * 32])) list_insert(L, 32, cnt, k, key);
        }
      }
    }
    }
    __syncwarp();
    // k smallest of the 32 sorted lists
    int head = 0;
    u64 kth = PPP_KEY_INF;
    mine = PPP_KEY_INF;
    mine2 = PPP_KEY_INF;
    for (int j = 0; j < kk; j++) {
      u64 h = head < cnt ? L[head * 32] : PPP_KEY_INF;
      u64 m = warp_min_u64(h);
      if (m == PPP_KEY_INF) break;
      if (h == m) head++;  // keys are unique (distinct point indices)
      if (lane == (j & 31)) { if (j < 32) mine = m; else mine2 = m; }
      kth = (j == kk - 1) ? m : kth;
    }
    if (kth != PPP_KEY_INF && key_d2(kth) < ring_bound2(g, R, cu, cv)) break;
    if (block_covers_grid(g, cu, cv, R)) break;
    if (kth != PPP_KEY_INF) tau = kth;  // nothing at or beyond the current k-th can enter any more
    R_prev = R;
    R++;
  }
  const int have = __popc(__ballot_sync(0xffffffffu, mine != PPP_KEY_INF)) +
                   __popc(__ballot_sync(0xffffffffu, mine2 != PPP_KEY_INF));
  if (P.idx_out && lane < k) {
    P.idx_out[row * (int64_t)k + lane] = mine != PPP_KEY_INF ? key_idx(mine) : -1;
    if (P.d2_out) P.d2_out[row * (int64_t)k + lane] = mine != PPP_KEY_INF ? key_d2(mine) : CUDART_INF_F;
  }
  if (P.idx_out && 32 + lane < k) {
    P.idx_out[row * (int64_t)k + 32 + lane] = mine2 != PPP_KEY_INF ? key_idx(mine2) : -1;
    if (P.d2_out) P.d2_out[row * (int64_t)k + 32 + lane] = mine2 != PPP_KEY_INF ? key_d2(mine2) : CUDART_INF_F;
  }
  if (P.normals) {
    float o[4];
    if (have < 3) {
      o[0] = o[1] = o[2] = o[3] = CUDART_NAN_F;
    } else {
      // sequential accumulation in list order, computed redundantly by every lane
      float acc[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      const bool shifted = (P.flags & PPP_COV_SHIFTED) != 0;
      float kx = 0.f, ky = 0.f, kz = 0.f;
      // every lane fetches ITS neighbour's record (one memory latency for all of them); the accumulation then walks
      // the list through shuffles -- sixteen dependent loads in a row were a third of this latency-bound kernel
      float4 rec = make_float4(0.f, 0.f, 0.f, 0.f), rec2 = rec;
      if (mine != PPP_KEY_INF) rec = __ldg(P.xyz4 + key_idx(mine));
      if (mine2 != PPP_KEY_INF) rec2 = __ldg(P.xyz4 + key_idx(mine2));
      for (int j = 0; j < have; j++) {
        const bool lo32 = j < 32;
        float4 a;
        a.x = __shfl_sync(0xffffffffu, lo32 ? rec.x : rec2.x, j & 31);
        a.y = __shfl_sync(0xffffffffu, lo32 ? rec.y : rec2.y, j & 31);
        a.z = __shfl_sync(0xffffffffu, lo32 ? rec.z : rec2.z, j & 31);
        if (shifted && j == 0) { kx = a.x; ky = a.y; kz = a.z; }
        float x = a.x, y = a.y, z = a.z;
        if (shifted) { x = __fsub_rn(x, kx); y = __fsub_rn(y, ky); z = __fsub_rn(z, kz); }
        accumulate_point(acc, x, y, z);
      }
      normal_from_accumulators(acc, have, qx, qy, qz, P.vpx, P.vpy, P.vpz, o);
    }
    if (lane == 0) store_normal(P.normals, P.nmap, row, P.nsf, o, P.route);
  }
  __syncwarp();
  }  // slot loop
}

// ---------------------------------------------------------------------------------------------
// Fixed-radius normals, one WARP per query: hand-over path of k_radius_normals32 (queries with
// more than 32 neighbours or a near-tie).  Lanes stride over the candidates of the (2R0+1)^2
// block, each keeping its in-radius keys sorted in a small shared-memory list; the lists are then
// merged by repeated warp-wide 64-bit min, and every lane accumulates the covariance in that
// (d2, index) order.  Queries whose neighbours overflow a lane list (hundreds of neighbours) are
// passed on to the generic kernel through redo2.
// ---------------------------------------------------------------------------------------------
constexpr int RW_CAPL = 16;  // keys per lane: up to 512 neighbours per query if evenly spread

__global__ void __launch_bounds__(WARPQ_WARPS * 32) k_radius_warp(SearchParams P, int32_t* __restrict__ redo2_count,
                                                                  int32_t* __restrict__ redo2_list) {
  pdl_prologue();
  __shared__ u64 s_l[WARPQ_WARPS * 32 * RW_CAPL];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const GridView& g = P.g;
  u64* L = s_l + (size_t)w * 32 * RW_CAPL + lane;
  const int n_redo = *P.redo_count;
  const u64 tau = make_key(P.r2, 0);
  for (int64_t slot = (int64_t)blockIdx.x * WARPQ_WARPS + w; slot < n_redo; slot += (int64_t)gridDim.x * WARPQ_WARPS) {
    const int64_t t = P.redo_list[slot];
    float4 p = __ldg(g.sorted + P.first + t);
    const float qx = p.x, qy = p.y, qz = p.z;
    const int64_t row = __float_as_int(p.w);
    const int cu = cell_coord_raw(axis_of(qx, qy, qz, g.au), g.min_u, g.inv_h);
    const int cv = cell_coord_raw(axis_of(qx, qy, qz, g.av), g.min_v, g.inv_h);
    const int R = P.R0;
    int cnt = 0;
    bool over = false;
    const int v0 = max(cv - R, 0), v1 = min(cv + R, g.nv - 1);
    for (int v = v0; v <= v1; v++) {
      const int32_t* rowp = g.cell_start + (int64_t)v * g.nu;
      int a = max(cu - R, 0), b = min(cu + R, g.nu - 1);
      if (a > b) continue;
      const int s = __ldg(rowp + a), e = __ldg(rowp + b + 1);
      for (int i = s + lane; i < e; i += 32) {
        float4 c = __ldg(g.sorted + i);
        u64 key = make_key(d2_flann(qx, qy, qz, c.x, c.y, c.z), __float_as_int(c.w));
        if (key < tau) {
          if (cnt == RW_CAPL) over = true;
          else list_insert(L, 32, cnt, RW_CAPL, key);
        }
      }
    }
    __syncwarp();
    if (__any_sync(0xffffffffu, over)) {
      if (lane == 0) redo2_list[atomicAdd(redo2_count, 1)] = (int32_t)t;
      continue;
    }
    float acc[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const bool shifted = (P.flags & PPP_COV_SHIFTED) != 0;
    float kx = 0.f, ky = 0.f, kz = 0.f;
    int head = 0, m = 0;
    while (true) {
      u64 h = head < cnt ? L[head * 32] : PPP_KEY_INF;
      u64 mn = warp_min_u64(h);
      if (mn == PPP_KEY_INF) break;
      if (h == mn) head++;
      float4 a = __ldg(P.xyz4 + key_idx(mn));
      if (shifted && m == 0) { kx = a.x; ky = a.y; kz = a.z; }
      float x = a.x, y = a.y, z = a.z;
      if (shifted) { x = __fsub_rn(x, kx); y = __fsub_rn(y, ky); z = __fsub_rn(z, kz); }
      accumulate_point(acc, x, y, z);
      m++;
    }
    float o[4];
    if (m < 3) o[0] = o[1] = o[2] = o[3] = CUDART_NAN_F;
    else normal_from_accumulators(acc, m, qx, qy, qz, P.vpx, P.vpy, P.vpz, o);
    if (lane == 0) store_normal(P.normals, P.nmap, row, P.nsf, o, P.route);
    __syncwarp();
  }
}

__global__ void __launch_bounds__(128) k_radius_count(SearchParams P, int32_t* __restrict__ counts, int32_t* __restrict__ max_count) {
  pdl_prologue();
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int cnt = 0;
  bool have = t < P.nq;
  if (P.use_redo) {
    have = t < *P.redo_count;
    if (have) t = P.redo_list[t];
  }
  if (have) {
    const GridView& g = P.g;
    float qx, qy, qz;
    int64_t row;
    load_query(P, P.q != nullptr, t, qx, qy, qz, row);
    const bool mine = P.use_redo || P.choice == nullptr || P.q != nullptr || __ldg(P.choice + row) == P.my_proj;
    if (mine && finite3(qx, qy, qz) && g.n_sorted > 0) {
      int cu = cell_coord_raw(axis_of(qx, qy, qz, g.au), g.min_u, g.inv_h);
      int cv = cell_coord_raw(axis_of(qx, qy, qz, g.av), g.min_v, g.inv_h);
      const float r2 = P.r2;
      visit_annulus(g, cu, cv, -1, P.R0, [&](float4 c) {
        cnt += d2_flann(qx, qy, qz, c.x, c.y, c.z) < r2 ? 1 : 0;
      });
    }
    if (counts && mine) counts[row] = cnt;
  }
  int m = cnt;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(max_count, m);
}


// ---------------------------------------------------------------------------------------------
// "next" row 1 of SURVEY.md §8f: principal curvatures at arbitrary query points, the device side
// of compute_transform (src/Path_Generation.cpp:362-400, k = 10;
// src/Path_Alg/path_dynamic_alg.cpp:77-110, k = 50): kNN of the query (done by the search
// kernels into idx), then pcl::PrincipalCurvaturesEstimation::computePointPrincipalCurvatures
// [upstream, recalled] with neighbour [0] as the centre.  One thread per query.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_principal_curvatures(const int32_t* __restrict__ idx, int64_t nq, int k,
                                                              const float* __restrict__ normals, int nsf,
                                                              float* __restrict__ out, int32_t* __restrict__ nn0) {
  pdl_prologue();
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nq) return;
  const int32_t* nb = idx + t * (int64_t)k;
  float* o = out + 5 * t;
  int m = 0;
  while (m < k && nb[m] >= 0) m++;
  if (m == 0) {
    for (int i = 0; i < 5; i++) o[i] = CUDART_NAN_F;
    if (nn0) nn0[t] = -1;
    return;
  }
  if (nn0) nn0[t] = nb[0];
  const float* n0 = normals + (int64_t)nb[0] * nsf;
  const float a0 = __ldg(n0), a1 = __ldg(n0 + 1), a2 = __ldg(n0 + 2);
  float M[9];
  const float nn[3] = {a0, a1, a2};
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) M[3 * i + j] = __fsub_rn(i == j ? 1.0f : 0.0f, __fmul_rn(nn[i], nn[j]));
  auto project = [&](int j, float p[3]) {
    const float* nj = normals + (int64_t)nb[j] * nsf;
    const float b0 = __ldg(nj), b1 = __ldg(nj + 1), b2 = __ldg(nj + 2);
#pragma unroll
    for (int i = 0; i < 3; i++)
      p[i] = __fadd_rn(__fmul_rn(M[3 * i], b0), __fadd_rn(__fmul_rn(M[3 * i + 1], b1), __fmul_rn(M[3 * i + 2], b2)));
  };
  float cen[3] = {0.f, 0.f, 0.f};
  for (int j = 0; j < m; j++) {
    float p[3];
    project(j, p);
    cen[0] = __fadd_rn(cen[0], p[0]); cen[1] = __fadd_rn(cen[1], p[1]); cen[2] = __fadd_rn(cen[2], p[2]);
  }
  const float fm = (float)m;
  cen[0] = __fdiv_rn(cen[0], fm); cen[1] = __fdiv_rn(cen[1], fm); cen[2] = __fdiv_rn(cen[2], fm);
  float c00 = 0.f, c01 = 0.f, c02 = 0.f, c11 = 0.f, c12 = 0.f, c22 = 0.f;
  for (int j = 0; j < m; j++) {
    float p[3];
    project(j, p);
    float d0 = __fsub_rn(p[0], cen[0]), d1 = __fsub_rn(p[1], cen[1]), d2 = __fsub_rn(p[2], cen[2]);
    c00 = __fadd_rn(c00, __fmul_rn(d0, d0)); c01 = __fadd_rn(c01, __fmul_rn(d0, d1)); c02 = __fadd_rn(c02, __fmul_rn(d0, d2));
    c11 = __fadd_rn(c11, __fmul_rn(d1, d1)); c12 = __fadd_rn(c12, __fmul_rn(d1, d2)); c22 = __fadd_rn(c22, __fmul_rn(d2, d2));
  }
  // eigen33 (values): scale, roots of the scaled matrix, rescale
  float scale = fmaxf(fmaxf(fmaxf(fabsf(c00), fabsf(c01)), fmaxf(fabsf(c02), fabsf(c11))), fmaxf(fabsf(c12), fabsf(c22)));
  if (scale <= 1.17549435e-38f) scale = 1.0f;
  float ev[3];
  compute_roots(__fdiv_rn(c00, scale), __fdiv_rn(c01, scale), __fdiv_rn(c02, scale), __fdiv_rn(c11, scale),
                __fdiv_rn(c12, scale), __fdiv_rn(c22, scale), ev);
  ev[0] = __fmul_rn(ev[0], scale); ev[1] = __fmul_rn(ev[1], scale); ev[2] = __fmul_rn(ev[2], scale);
  // computeCorrespondingEigenVector for the largest eigenvalue
  const float e = __fdiv_rn(ev[2], scale);
  const float s00 = __fsub_rn(__fdiv_rn(c00, scale), e), s11 = __fsub_rn(__fdiv_rn(c11, scale), e),
              s22 = __fsub_rn(__fdiv_rn(c22, scale), e);
  const float s01 = __fdiv_rn(c01, scale), s02 = __fdiv_rn(c02, scale), s12 = __fdiv_rn(c12, scale);
  float v1[3], v2[3], v3[3];
  cross3(s00, s01, s02, s01, s11, s12, v1);
  cross3(s00, s01, s02, s02, s12, s22, v2);
  cross3(s01, s11, s12, s02, s12, s22, v3);
  float l1 = sqnorm3(v1), l2 = sqnorm3(v2), l3 = sqnorm3(v3);
  float vx, vy, vz, l;
  if (l1 >= l2 && l1 >= l3) { vx = v1[0]; vy = v1[1]; vz = v1[2]; l = l1; }
  else if (l2 >= l1 && l2 >= l3) { vx = v2[0]; vy = v2[1]; vz = v2[2]; l = l2; }
  else { vx = v3[0]; vy = v3[1]; vz = v3[2]; l = l3; }
  const float sl = __fsqrt_rn(l);
  const float inv = __fdiv_rn(1.0f, fm);
  o[0] = __fdiv_rn(vx, sl); o[1] = __fdiv_rn(vy, sl); o[2] = __fdiv_rn(vz, sl);
  o[3] = __fmul_rn(ev[2], inv);
  o[4] = __fmul_rn(ev[1], inv);
}

// compute_coverage (src/Path_Generation.cpp:483-496): every point within `radius` of a query gets
// its coverage flag set.  No ordering is needed, so candidates are marked as they are scanned.
__global__ void __launch_bounds__(128) k_coverage_mark(SearchParams P, unsigned char* __restrict__ flags,
                                                       const float* __restrict__ r2_per_query) {
  pdl_prologue();
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= P.nq) return;
  const GridView& g = P.g;
  const float* qp = P.q + t * P.q_sf;
  const float qx = __ldg(qp), qy = __ldg(qp + 1), qz = __ldg(qp + 2);
  if (!finite3(qx, qy, qz) || g.n_sorted == 0) return;
  int cu = cell_coord_raw(axis_of(qx, qy, qz, g.au), g.min_u, g.inv_h);
  int cv = cell_coord_raw(axis_of(qx, qy, qz, g.av), g.min_v, g.inv_h);
  const float r2 = r2_per_query ? __ldg(r2_per_query + t) : P.r2;   // the block radius R0 covers the largest of them
  if (!(r2 > 0.0f)) return;                                        // NaN / zero radius: nothing is strictly inside
  visit_annulus(g, cu, cv, -1, P.R0, [&](float4 c) {
    if (d2_flann(qx, qy, qz, c.x, c.y, c.z) < r2) flags[__float_as_int(c.w)] = 1;
  });
}

// counts for non-finite self points that are not in the sorted array: zero-fill first
// StatisticalOutlierRemoval first pass (src/contour_alg.cpp:101-108): mean of the distances to the
// mean_k nearest neighbours, from the sorted d2 rows of a (mean_k + 1)-NN search.  The additions run
// in list order in double, exactly as the reference's scalar loop; entry 0 (the query itself) is skipped.
__global__ void __launch_bounds__(256) k_sor_mean(const float4* __restrict__ xyz4, const float* __restrict__ d2, int64_t n,
                                                  int k, int sqrt_float, float* __restrict__ dist,
                                                  unsigned long long* __restrict__ n_valid) {
  pdl_prologue();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool ok = false;
  if (i < n) {
    float4 p = __ldg(xyz4 + i);
    ok = isfinite(p.x) && isfinite(p.y) && isfinite(p.z);
    float out = 0.0f;
    if (ok) {
      const float* row = d2 + i * k;
      double sum = 0.0;
      for (int j = 1; j < k; j++) {
        float v = __ldg(row + j);
        sum = __dadd_rn(sum, sqrt_float ? (double)__fsqrt_rn(v) : __dsqrt_rn((double)v));
      }
      out = (float)__ddiv_rn(sum, (double)(k - 1));
    }
    dist[i] = out;
  }
  unsigned cnt = __syncthreads_count(ok);
  if (threadIdx.x == 0 && cnt) atomicAdd(n_valid, (unsigned long long)cnt);
}

__global__ void k_fill_i32(int32_t* p, int64_t n, int32_t v) {
  pdl_prologue();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// Self-mode outputs are written by original index of the *indexed* points only; rows of
// non-finite points get their defaults here (idx -1 / d2 inf / NaN normals).
__global__ void k_default_rows(const float4* __restrict__ xyz4, int64_t n, int cap, int32_t* idx_out, float* d2_out,
                               float* normals, int nsf, const int32_t* __restrict__ nmap,
                               const NormalRoute* __restrict__ route) {
  pdl_prologue();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 p = __ldg(xyz4 + i);
  if (p.w == p.w) return;
  if (idx_out)
    for (int j = 0; j < cap; j++) {
      idx_out[i * (int64_t)cap + j] = -1;
      if (d2_out) d2_out[i * (int64_t)cap + j] = CUDART_INF_F;
    }
  if (normals) {
    float o[4] = {CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F};
    store_normal(normals, nmap, i, nsf, o, route);
  }
}

int pick_block(ppp_ctx* ctx, int cap, int* block, size_t* smem) {
  // largest block in {128, 64, 32} whose list storage fits in opt-in shared memory
  size_t lim = ctx->smem_optin ? ctx->smem_optin : 48 * 1024;
  for (int b = 128; b >= 32; b >>= 1) {
    size_t need = (size_t)cap * 8 * b;
    if (need <= lim) { *block = b; *smem = need; return PPP_OK; }
  }
  ppp_set_error("neighbour list capacity %d exceeds the shared-memory path (max %zu entries per query)", cap,
                lim / (8 * 32));
  return PPP_ERR_UNSUPPORTED;
}

}  // namespace

int radius_rings(const GridView& g, double r) {
  // need R*h - slack >= r
  // r comes from sqrt((float)(r*r)); a float32 d2 below r2 can belong to a point up to ~1e-7 beyond it.
  // A radius whose float32 square is infinite (r = inf here) admits every finite point: capped at PPP_RING_MAX,
  // the block around any (clamped) query cell covers the whole grid, and the d2 < r2 test decides.
  r *= 1.0 + 1e-6;
  const double Rd = std::ceil((r + (double)g.slack) / (double)g.h - 1e-12);
  if (!(Rd < (double)PPP_RING_MAX)) return PPP_RING_MAX;
  int R = (int)Rd;
  while (R < PPP_RING_MAX && (double)R * (double)g.h - (double)g.slack < r) R++;
  return std::max(R, 0);
}

static int launch_search(ppp_cloud* c, SearchParams& P) {
  ppp_ctx* ctx = c->ctx;
  int block; size_t smem;
  PPP_TRY(pick_block(ctx, std::max(P.cap, 1), &block, &smem));
  if (P.use_redo) {  // few, scattered queries: small blocks spread them over all SMs
    block = 32;
    smem = (size_t)std::max(P.cap, 1) * 8 * block;
  }
  if (smem > 40 * 1024)
    PPP_CUDA(cudaFuncSetAttribute(k_search, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (P.nq > 0) {
    unsigned blocks = (unsigned)((P.nq + block - 1) / block);
    PPP_LAUNCH(ctx, P.use_redo ? "knn_redo" : P.mode == 0 ? (P.normals ? "knn_normals" : "knn") : (P.normals ? "radius_normals" : "radius_fill"),
               k_search, blocks, block, smem, P);
    PPP_CHECK_LAUNCH();
  }
  return PPP_OK;
}

static int prepare_fast(ppp_cloud* c, SearchParams& P, int32_t** redo_out) {
  ppp_ctx* ctx = c->ctx;
  int32_t* redo = nullptr;
  PPP_TRY(dev_alloc(ctx, &redo, (size_t)P.nq + 1));
  PPP_CUDA(cudaMemsetAsync(redo, 0, sizeof(int32_t), ctx->stream));
  P.redo_count = redo;
  P.redo_list = redo + 1;
  P.use_redo = 0;
  *redo_out = redo;
  return PPP_OK;
}

// fast fixed-block kernel, then the ring-expanding warp kernel on whatever it handed over
static int launch_knn_fast(ppp_cloud* c, SearchParams& P) {
  ppp_ctx* ctx = c->ctx;
  int32_t* redo = nullptr;
  PPP_TRY(prepare_fast(c, P, &redo));
  // measured with the cloud's own points (1M points, ms): k = 16 0.196 / 0.198 / 0.201 with 128 / 64 / 96 threads;
  // k = 32 128 threads x 6 blocks (80 registers) 0.351, x 5 (93) 0.359, 64 threads x 12 / 10 / 8 0.354 / 0.365 / 0.359;
  // k = 64 0.789 with 128 threads x 4 blocks, 0.829 with 64 x 8.
  // (Tried and rejected on measurements: a second pass of the k <= 16 kernel with a 7 x 7 block over the ~0.2 % of
  // queries the 5 x 5 block cannot finish, before the one-warp-per-query kernel: each extra launch costs the life
  // time of one block, 30-50 us, whatever the number of queries -- 0.308 ms against 0.266 ms for the stage.  RB = 9
  // -- rows of up to 512 candidates -- for workpieces with walls: box with walls search 0.41 -> 0.72 ms for a
  // hand-over kernel that only went 0.73 -> 0.53 ms: the warp-uniform row loops of the thread-per-query kernel pay
  // for the longest row of 32 queries.)
  constexpr int block = 128;
  const unsigned blocks = (unsigned)((P.nq + block - 1) / block);
  const bool ext = P.q != nullptr;   // a query array instead of the cloud's own points in cell order
  // per thread: `slots` key words, then the first sorted position of each of the 2 R0 + 1 block rows
  auto launch = [&](auto kern, int slots) -> int {
    const size_t smem = (size_t)(slots + 2 * P.R0 + 1) * 4 * block;
    if (smem > 40 * 1024) PPP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    PPP_LAUNCH(ctx, P.normals ? "knn_normals" : "knn", kern, blocks, block, smem, P);
    PPP_CHECK_LAUNCH();
    return PPP_OK;
  };
  if (P.cap <= 16) PPP_TRY(launch(ext ? k_knnf<16, 16, 7, 128, 8, 0, true> : k_knnf<16, 16, 7, 128, 8, 0, false>, 16 + 16));
  else if (P.cap <= 32) PPP_TRY(launch(ext ? k_knnf<32, 16, 6, 128, 6, 32, true> : k_knnf<32, 16, 6, 128, 6, 32, false>, 32 + 16));
  else PPP_TRY(launch(ext ? k_knnf<64, 32, 7, 128, 4, 64, true> : k_knnf<64, 32, 7, 128, 4, 64, false>, 64 + 32));
  {
    // hand-over queries: one warp each, persistent warps (their number is only known on the device)
    P.use_redo = 1;
    size_t smem = (size_t)WARPQ_WARPS * 32 * P.cap * 8;
    // (opt in from 40 KB of dynamic shared memory on: the kernels carry static arrays too -- k = 48 asks for exactly
    // 48 KB here and was refused by the launch without it)
    if (smem > 40 * 1024) PPP_CUDA(cudaFuncSetAttribute(k_knn_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    unsigned blocks = (unsigned)std::min<int64_t>((P.nq + WARPQ_WARPS - 1) / WARPQ_WARPS, (int64_t)ctx->sm_count * 8);
    PPP_LAUNCH(ctx, "knn_redo", k_knn_warp, blocks, WARPQ_WARPS * 32, smem, P);
    PPP_CHECK_LAUNCH();
  }
  if (getenv("PPP_DEBUG")) {
    int32_t n_redo = 0;
    fetch_small(ctx, redo, 4, &n_redo);
    fprintf(stderr, "[ppp] knn fast path: %lld queries, %d handed to the ring-expanding kernel (h=%g, R0=%d)\n",
            (long long)P.nq, n_redo, (double)P.g.h, P.R0);
  }
  dev_free(ctx, redo);
  return PPP_OK;
}

int knn_launch(ppp_cloud* c, const GridStore& gs, const float* q_dev, int64_t nq, int q_stride_f, int64_t first, int k,
               int32_t* idx_dev, float* d2_dev, bool with_normals, const float vp[3], unsigned flags,
               float* normals_dev, int normal_stride_f, const unsigned char* choice, int my_proj) {
  ppp_ctx* ctx = c->ctx;
  SearchParams P{};
  P.g = gs.v; P.xyz4 = c->xyz4; P.q = q_dev; P.q_sf = q_stride_f; P.nq = nq; P.first = first;
  P.cap = k; P.kk = (int)std::min<int64_t>(k, c->n_finite); P.mode = 0; P.R0 = PPP_KNN_RINGS; P.r2 = 0;
  P.idx_out = idx_dev; P.d2_out = d2_dev; P.offsets = nullptr;
  P.normals = with_normals ? normals_dev : nullptr; P.nsf = normal_stride_f; P.nmap = c->nmap; P.route = c->route;
  P.vpx = vp ? vp[0] : 0; P.vpy = vp ? vp[1] : 0; P.vpz = vp ? vp[2] : 0; P.flags = flags;
  P.choice = q_dev ? nullptr : choice; P.my_proj = my_proj;
  if (!q_dev && c->n_finite < c->n && first == 0) {
    unsigned blocks = (unsigned)((c->n + 255) / 256);
    PPP_LAUNCH(ctx, "default_rows", k_default_rows, blocks, 256, 0, (const float4*)c->xyz4, c->n, k, idx_dev, d2_dev,
               P.normals, normal_stride_f, c->nmap, c->route);
    PPP_CHECK_LAUNCH();
  }
  if (k <= 64 && nq > 0) return launch_knn_fast(c, P);
  return launch_search(c, P);
}

int radius_count_launch(ppp_cloud* c, const GridStore& gs, const float* q_dev, int64_t nq, int q_stride_f,
                        int64_t first, float r2, int32_t* counts_dev) {
  ppp_ctx* ctx = c->ctx;
  SearchParams P{};
  P.g = gs.v; P.xyz4 = c->xyz4; P.q = q_dev; P.q_sf = q_stride_f; P.nq = nq; P.first = first;
  P.mode = 1; P.r2 = r2; P.R0 = radius_rings(gs.v, std::sqrt((double)r2));
  int32_t* mx = nullptr;
  PPP_TRY(dev_alloc(ctx, &mx, 1));
  PPP_CUDA(cudaMemsetAsync(mx, 0, 4, ctx->stream));
  if (!q_dev && c->n_finite < c->n && counts_dev) {
    unsigned blocks = (unsigned)((c->n + 255) / 256);
    PPP_LAUNCH(ctx, "fill_i32", k_fill_i32, blocks, 256, 0, counts_dev, c->n, 0);
    PPP_CHECK_LAUNCH();
  }
  if (nq > 0) {
    unsigned blocks = (unsigned)((nq + 127) / 128);
    PPP_LAUNCH(ctx, "radius_count", k_radius_count, blocks, 128, 0, P, counts_dev, mx);
    PPP_CHECK_LAUNCH();
  }
  int hmx = 0;
  PPP_TRY(fetch_small(ctx, mx, 4, &hmx));
  dev_free(ctx, mx);
  return hmx;  // >= 0: maximum neighbour count (used to size the fill pass)
}

int radius_fill_launch(ppp_cloud* c, const GridStore& gs, const float* q_dev, int64_t nq, int q_stride_f,
                       int64_t first, float r2, const int64_t* offsets_dev, int32_t* idx_dev, float* d2_dev) {
  // the caller has run radius_count_launch and passes the maximum count through d2-independent path:
  // recompute it here (cheap) so this entry stays self-contained.
  int mx = radius_count_launch(c, gs, q_dev, nq, q_stride_f, first, r2, nullptr);
  if (mx < 0) return mx;
  SearchParams P{};
  P.g = gs.v; P.xyz4 = c->xyz4; P.q = q_dev; P.q_sf = q_stride_f; P.nq = nq; P.first = first;
  P.cap = std::max(mx, 1); P.mode = 1; P.r2 = r2; P.R0 = radius_rings(gs.v, std::sqrt((double)r2));
  P.idx_out = idx_dev; P.d2_out = d2_dev; P.offsets = offsets_dev;
  return launch_search(c, P);
}

int normals_radius_launch(ppp_cloud* c, const GridStore& gs, int64_t first, int64_t count, float r2,
                          const float vp[3], unsigned flags, float* normals_dev, int normal_stride_f,
                          const unsigned char* choice, int my_proj) {
  ppp_ctx* ctx = c->ctx;
  SearchParams P{};
  P.g = gs.v; P.xyz4 = c->xyz4; P.q = nullptr; P.nq = count; P.first = first;
  P.mode = 1; P.r2 = r2; P.R0 = radius_rings(gs.v, std::sqrt((double)r2));
  P.normals = normals_dev; P.nsf = normal_stride_f; P.nmap = c->nmap; P.route = c->route;
  P.vpx = vp ? vp[0] : 0; P.vpy = vp ? vp[1] : 0; P.vpz = vp ? vp[2] : 0; P.flags = flags;
  P.choice = choice; P.my_proj = my_proj;
  if (c->n_finite < c->n && first == 0) {
    unsigned blocks = (unsigned)((c->n + 255) / 256);
    PPP_LAUNCH(ctx, "default_rows", k_default_rows, blocks, 256, 0, (const float4*)c->xyz4, c->n, 0, (int32_t*)nullptr,
               (float*)nullptr, normals_dev, normal_stride_f, c->nmap, c->route);
    PPP_CHECK_LAUNCH();
  }
  if (count <= 0) return PPP_OK;
  // expected neighbours per query from the surface density; the fixed-capacity fast kernel pays
  // off while most queries stay within its 32-entry lists
  const double expect = c->density * 3.14159265358979 * (double)r2;
  const bool fast = expect <= 24.0;
  int32_t* redo = nullptr;
  int n_redo = 0;
  if (fast) {
    PPP_TRY(prepare_fast(c, P, &redo));
    P.cap = 32;
    {
      size_t smem = (size_t)C_STORE * 8 * 128;
      PPP_CUDA(cudaFuncSetAttribute(k_radius_normals32, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      unsigned blocks = (unsigned)((P.nq + 127) / 128);
      PPP_LAUNCH(ctx, "radius_normals", k_radius_normals32, blocks, 128, smem, P);
      PPP_CHECK_LAUNCH();
    }
    // hand-over queries: one warp each (persistent warps); what even that cannot hold goes on to the
    // generic kernel through a second list
    int32_t* redo2 = nullptr;
    PPP_TRY(dev_alloc(ctx, &redo2, (size_t)P.nq + 1));
    PPP_CUDA(cudaMemsetAsync(redo2, 0, sizeof(int32_t), ctx->stream));
    {
      unsigned blocks = (unsigned)std::min<int64_t>((P.nq + WARPQ_WARPS - 1) / WARPQ_WARPS, (int64_t)ctx->sm_count * 8);
      PPP_LAUNCH(ctx, "radius_redo", k_radius_warp, blocks, WARPQ_WARPS * 32, 0, P, redo2, redo2 + 1);
      PPP_CHECK_LAUNCH();
    }
    PPP_TRY(fetch_small(ctx, redo2, 4, &n_redo));
    dev_free(ctx, redo);
    redo = redo2;
    if (n_redo == 0) { dev_free(ctx, redo); return PPP_OK; }
    P.redo_count = redo2;
    P.redo_list = redo2 + 1;
    P.use_redo = 1;
  }
  // generic path: all queries, or only the ones the fast kernel handed over
  const int64_t nq = fast ? n_redo : count;
  SearchParams C = P;
  C.nq = nq;
  int32_t* mx = nullptr;
  PPP_TRY(dev_alloc(ctx, &mx, 1));
  PPP_CUDA(cudaMemsetAsync(mx, 0, 4, ctx->stream));
  {
    unsigned blocks = (unsigned)((nq + 127) / 128);
    PPP_LAUNCH(ctx, "radius_count", k_radius_count, blocks, 128, 0, C, (int32_t*)nullptr, mx);
    PPP_CHECK_LAUNCH();
  }
  int hmx = 0;
  PPP_TRY(fetch_small(ctx, mx, 4, &hmx));
  dev_free(ctx, mx);
  C.cap = std::max(hmx, 1);
  int st = launch_search(c, C);
  dev_free(ctx, redo);
  return st;
}

int coverage_mark_launch(ppp_cloud* c, const GridStore& gs, const float* q_dev, int64_t nq, int q_stride_f, float r2,
                         unsigned char* flags_dev, const float* r2_per_query_dev) {
  ppp_ctx* ctx = c->ctx;
  if (nq <= 0) return PPP_OK;
  SearchParams P{};
  P.g = gs.v; P.xyz4 = c->xyz4; P.q = q_dev; P.q_sf = q_stride_f; P.nq = nq;
  P.mode = 1; P.r2 = r2; P.R0 = radius_rings(gs.v, std::sqrt((double)r2));
  unsigned blocks = (unsigned)((nq + 127) / 128);
  PPP_LAUNCH(ctx, "coverage_mark", k_coverage_mark, blocks, 128, 0, P, flags_dev, r2_per_query_dev);
  PPP_CHECK_LAUNCH();
  return PPP_OK;
}

static int sor_mean_inner(ppp_cloud* c, const GridStore& gs, int k, int sqrt_float, int32_t* idx, float* d2,
                          float* dist_dev, unsigned long long* n_valid_dev) {
  ppp_ctx* ctx = c->ctx;
  PPP_TRY(knn_launch(c, gs, nullptr, c->n_finite, 0, 0, k, idx, d2, false, nullptr, 0, nullptr, 0));
  PPP_CUDA(cudaMemsetAsync(n_valid_dev, 0, 8, ctx->stream));
  unsigned blocks = (unsigned)((c->n + 255) / 256);
  PPP_LAUNCH(ctx, "sor_mean", k_sor_mean, blocks, 256, 0, (const float4*)c->xyz4, (const float*)d2, c->n, k, sqrt_float,
             dist_dev, n_valid_dev);
  PPP_CHECK_LAUNCH();
  return PPP_OK;
}

int sor_mean_distances_launch(ppp_cloud* c, const GridStore& gs, int mean_k, int sqrt_float, float* dist_dev,
                              unsigned long long* n_valid_dev) {
  ppp_ctx* ctx = c->ctx;
  const int k = mean_k + 1;
  int32_t* idx = nullptr; float* d2 = nullptr;
  PPP_TRY(dev_alloc(ctx, &idx, (size_t)c->n * k));
  int st = dev_alloc(ctx, &d2, (size_t)c->n * k);
  if (st == PPP_OK) st = sor_mean_inner(c, gs, k, sqrt_float, idx, d2, dist_dev, n_valid_dev);
  dev_free(ctx, idx); dev_free(ctx, d2);
  return st;
}

int principal_curvatures_launch(ppp_cloud* c, const int32_t* idx_dev, int64_t nq, int k, const float* normals_dev,
                                int normal_stride_f, float* out_dev, int32_t* nn0_dev) {
  ppp_ctx* ctx = c->ctx;
  if (nq <= 0) return PPP_OK;
  unsigned blocks = (unsigned)((nq + 127) / 128);
  PPP_LAUNCH(ctx, "principal_curvatures", k_principal_curvatures, blocks, 128, 0, idx_dev, nq, k, normals_dev,
             normal_stride_f, out_dev, nn0_dev);
  PPP_CHECK_LAUNCH();
  return PPP_OK;
}
