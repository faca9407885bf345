// Internal declarations shared by the translation units of libppp_gpu.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/ppp_gpu.h"

// ---------------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------------
void ppp_set_error(const char* fmt, ...);

#define PPP_CUDA(call)                                                                         \
  do {                                                                                         \
    cudaError_t _e = (call);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      ppp_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e));      \
      return PPP_ERR_CUDA;                                                                     \
    }                                                                                          \
  } while (0)

#define PPP_TRY(call)              \
  do {                             \
    int _s = (call);               \
    if (_s != PPP_OK) return _s;   \
  } while (0)

// ---------------------------------------------------------------------------------------------
// context / cloud
// ---------------------------------------------------------------------------------------------
struct KernelStat {
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;
  double ms = 0;
  int64_t launches = 0;
};

struct ppp_ctx {
  int device = 0;
  int sm_count = 148;
  size_t smem_optin = 0;
  cudaStream_t stream = nullptr;       // CURRENT working stream (launches, stream-ordered allocations)
  cudaStream_t main_stream = nullptr;  // what ppp_stream() returns; timers and ppp_sync refer to it
  cudaStream_t aux_stream = nullptr;   // high priority: the slicing chain runs here, concurrently with the kNN kernel
  cudaStream_t copy_stream = nullptr;  // device->host result copies that overlap later kernels
  void* fetch_host = nullptr;          // mapped pinned scratch for fetch_small (FETCH_BYTES payload + one flag line)
  unsigned fetch_seq = 0;              // sequence number the next fetch kernel stores behind its payload
  void* ingest_dev = nullptr;          // persistent device scratch of cloud_ingest (bounding box, ticket, samples)
  bool ingest_clean = false;           // ... holds its initial values (the last ingest's kernel reset it)
  unsigned long long* scan_state[2] = {nullptr, nullptr};   // chained-scan tile words, one array per working stream
  int64_t scan_state_cap[2] = {0, 0};
  // Temporaries of the API call in progress (ApiScope): whatever an early error return leaves behind
  // is released when the outermost call ends.  Guarded by `mu` like everything else here.
  std::vector<void*> temps;
  int api_depth = 0;
  std::recursive_mutex mu;
  int64_t launches = 0;
  bool profile = false;
  bool trace = false;                  // ppp_kernel_trace: per-launch start/end on the real streams (overlap kept)
  cudaEvent_t trace_base = nullptr;
  struct TraceRec { const char* name; int aux; cudaEvent_t a, b; };
  std::vector<TraceRec> trace_recs;
  std::map<std::string, KernelStat> kstats;
  cudaEvent_t t_begin[16] = {}, t_end[16] = {};
  double t_ms[16] = {};
  int64_t t_regions[16] = {};
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> t_pending[16];
};

// Device-side view of the column grid (passed by value to kernels).
// Cells tile the two largest-extent axes (u, v) of the cloud; a cell row (fixed v) is contiguous
// in `sorted`, so the candidates of a query are (2R+1) contiguous ranges.
struct GridView {
  const float4* sorted;       // n_sorted records: x, y, z, __int_as_float(original index)
  const int32_t* cell_start;  // nu*nv + 1
  int nu, nv;                 // cells along u (fastest) and v
  int au, av;                 // which of x(0) y(1) z(2) are u and v
  float min_u, min_v;
  float inv_h, h;
  float slack;                // rounding slack (same unit as h) subtracted from ring bounds
  int n_sorted;
};

// Where the normal records of a slab go in the multi-GPU path (exchange.cu): row i of the slab is global
// point g = nmap[i] (negative: halo copy, not stored); its record belongs to the rank whose original
// index range [start[r], start[r+1]) holds g and is stored at base[r] + (g - start[r]) * stride
// -- base[r] is that rank's "home" buffer, local memory or a peer mapping over NVLink.
constexpr int PPP_MAX_RANKS = 16;
struct NormalRoute {
  int world;
  long long start[PPP_MAX_RANKS + 1];
  float* base[PPP_MAX_RANKS];
};

// Records allocated (not initialised) behind the n_sorted indexed ones: the fixed-point k-nearest kernel reads its
// candidate rows four records at a time without clamping the position (whatever lies there is rejected by
// the range test), at most PPP_SORTED_PAD - 1 records beyond the end of a row.
constexpr int PPP_SORTED_PAD = 160;

// Rings of cells in the fixed candidate block of the fast k-nearest kernels (2: a 5 x 5 block).
constexpr int PPP_KNN_RINGS = 2;

struct GridStore {
  GridView v{};
  int drop = 2;              // the axis this grid does NOT span (2: cells over x, y)
  float4* sorted = nullptr;
  int32_t* cell_start = nullptr;
  int32_t* order = nullptr;  // original index per sorted position (built on request: grid_sorted_order)
  double h = 0;
  cudaEvent_t ready = nullptr;  // recorded after the build: consumers on other streams wait on it
};

// Runs a section of host code with ctx->stream switched to the auxiliary stream (after it has
// waited on `after`), then makes the main stream wait for everything the section enqueued.
// Calls into the library are serialised by the context mutex, so the swap is race-free.
struct AuxScope {
  ppp_ctx* ctx;
  cudaStream_t saved;
  bool active;
  // While per-kernel profiling is on everything stays on the main stream, so that each kernel's
  // CUDA-event duration is that of the kernel running alone (overlapped kernels share the SMs).
  AuxScope(ppp_ctx* c, cudaEvent_t after) : ctx(c), saved(c->stream), active(!c->profile) {
    if (!active) return;
    if (after) cudaStreamWaitEvent(ctx->aux_stream, after, 0);
    ctx->stream = ctx->aux_stream;
  }
  ~AuxScope() {
    if (!active) return;
    cudaEvent_t ev;
    if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) == cudaSuccess) {
      cudaEventRecord(ev, ctx->aux_stream);
      cudaStreamWaitEvent(ctx->main_stream, ev, 0);
      cudaEventDestroy(ev);
    }
    ctx->stream = saved;
  }
};

// Multi-projection index (workpieces that are not height fields: closed shapes, vertical walls).  A column
// grid over two axes piles a surface that runs along the third axis into a few cells; with one grid per axis
// pair every point has at least one projection in which its neighbourhood is spread out (any surface normal
// has a component >= 0.577 along some axis, so the foreshortening is <= 1.73).  choice[i] = the projection
// whose candidate block around point i holds the fewest points (while holding enough).  Results do not
// depend on the choice -- every grid gives the exact answer -- only the amount of scanning does.
struct MPSet {
  double h = 0;
  int R0 = 0;
  GridStore* g[3] = {nullptr, nullptr, nullptr};   // g[p]: the grid that drops axis p
  unsigned char* choice = nullptr;                 // per ORIGINAL index: 0..2
  cudaEvent_t ready = nullptr;                     // recorded once all three grids and the choice are built
};

struct ppp_cloud {
  ppp_ctx* ctx = nullptr;
  int64_t n = 0;
  int64_t n_finite = 0;
  float4* xyz4 = nullptr;  // original order, w = 0 (finite) / NaN (non-finite point)
  float bmin[3] = {0, 0, 0}, bmax[3] = {0, 0, 0};
  double density = 0;  // finite points per unit area of the SURFACE around a typical point (sampled, see cloud_ingest)
  int au = 0, av = 1;
  int drop = 2;        // primary projection: the axis of smallest extent is not gridded
  int mp_state = -1;   // -1 not decided yet, 0 the primary column grid is enough, 1 multi-projection index
  std::vector<MPSet> mps;
  float cell_hint = 0;
  std::vector<GridStore> grids;
  GridStore* index_grid = nullptr;   // the primary grid of the last ppp_dev_index (ppp_dev_sorted_order)
  // results of the last ppp_dev_slice_contours (owned by the cloud)
  int64_t* c_node_off = nullptr;
  double *c_y = nullptr, *c_x = nullptr, *c_z = nullptr;
  int64_t c_cap = 0;
  int c_S_cap = 0;
  double *ext_y = nullptr, *ext_x = nullptr, *ext_z = nullptr;  // optional caller-owned node buffers
  int64_t ext_cap = 0;
  const int32_t* nmap = nullptr;   // ppp_dev_set_normal_row_map
  const NormalRoute* route = nullptr;  // device pointer (exchange.cu); with nmap: normals go to their home rank
  int64_t max_band_hint = 0;       // largest band of the last sync-free slicing call (sizes its shared memory)
  int64_t* ext_off = nullptr;      // ppp_dev_set_contour_offsets_buffer
  int64_t ext_off_cap = 0;
  double *out_y = nullptr, *out_x = nullptr, *out_z = nullptr;  // where the last call wrote the nodes
  // an exchange slab (ppp_exch_attach): the halo it was cut with, the largest finite |x| of the whole cloud and the
  // record stride of the home buffers, which ppp_dev_mls_smooth checks before it delivers records there
  double ex_halo = 0, ex_xmag = 0;
  int ex_home_bytes = 0;
};

// ---------------------------------------------------------------------------------------------
// launch wrapper: counts launches, optional per-kernel CUDA-event timing
// ---------------------------------------------------------------------------------------------
struct LaunchScope {
  ppp_ctx* ctx;
  const char* name;
  cudaEvent_t a = nullptr, b = nullptr;
  LaunchScope(ppp_ctx* c, const char* n) : ctx(c), name(n) {
    ctx->launches++;
    if (ctx->profile || ctx->trace) {
      cudaEventCreate(&a);
      cudaEventCreate(&b);
      cudaEventRecord(a, ctx->stream);
    }
  }
  ~LaunchScope() {
    if (a) {
      cudaEventRecord(b, ctx->stream);
      if (ctx->trace) ctx->trace_recs.push_back({name, ctx->stream == ctx->aux_stream ? 1 : 0, a, b});
      else ctx->kstats[name].pending.emplace_back(a, b);
    }
  }
};

// Programmatic dependent launch (sm_90+): every kernel of the library starts with pdl_prologue() -- it releases
// the launch of the NEXT kernel of the stream at once and then waits until the PREVIOUS one has completed and its
// stores are visible --, and is launched with the programmatic-stream-serialization attribute: the blocks of a
// kernel are set up on the SMs the predecessor's last blocks leave idle and start the moment it ends, instead of
// ~2.5 us later.  Results cannot change: no kernel touches memory before the wait.  PPP_PDL=0 launches the
// classic way (the prologue is a no-op then).
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_prologue() {
#ifdef PPP_PDL_EARLY
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
  asm volatile("griddepcontrol.wait;" ::: "memory");
}
#endif
bool ppp_pdl_enabled();

// Bounds-checked build (python -m polishpathplanning_b200.build --check -> libppp_gpu_check.so, loaded through
// PPP_GPU_LIB): the index arithmetic of the kernels that read or write without clamping is asserted on the device and a
// violation traps.  compute-sanitizer is not available on the measurement pool; tests/test_gpu_bounds.py runs a small
// pass over every such kernel with this build instead.  In the normal build the macro expands to nothing.
#ifdef PPP_CHECK_BOUNDS
#define PPP_DEV_ASSERT(cond)                                                                                     \
  do {                                                                                                           \
    if (!(cond)) {                                                                                               \
      printf("PPP_DEV_ASSERT failed: %s (%s:%d) block %d thread %d\n", #cond, __FILE__, __LINE__, (int)blockIdx.x, \
             (int)threadIdx.x);                                                                                  \
      __trap();                                                                                                  \
    }                                                                                                            \
  } while (0)
#else
#define PPP_DEV_ASSERT(cond) do { } while (0)
#endif

// `kernel` must be a plain identifier (bind template instantiations to a local `auto kern = ...`).
#define PPP_LAUNCH(ctx, name, kernel, grid, block, smem, ...)                             \
  do {                                                                                    \
    LaunchScope _ls((ctx), (name));                                                       \
    if (ppp_pdl_enabled()) {                                                              \
      cudaLaunchConfig_t _cfg = {};                                                       \
      _cfg.gridDim = dim3(grid); _cfg.blockDim = dim3(block);                             \
      _cfg.dynamicSmemBytes = (smem); _cfg.stream = (ctx)->stream;                        \
      cudaLaunchAttribute _at[1];                                                         \
      _at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                     \
      _at[0].val.programmaticStreamSerializationAllowed = 1;                              \
      _cfg.attrs = _at; _cfg.numAttrs = 1;                                                \
      cudaLaunchKernelEx(&_cfg, kernel, __VA_ARGS__);                                     \
    } else {                                                                              \
      kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);                     \
    }                                                                                     \
  } while (0)

#define PPP_CHECK_LAUNCH() PPP_CUDA(cudaGetLastError())

// Lets `kern` launch with `bytes` of dynamic shared memory.  Past 48 KB a kernel has to opt in, and the limit applies
// to its static arrays plus the dynamic memory: the opt-in starts at 40 KB of dynamic memory because the kernels
// carry up to 8 KB of static arrays (k = 48 asked the kNN hand-over kernel for exactly 48 KB and the launch was
// refused without it).
template <class K>
int smem_optin(K kern, size_t bytes) {
  if (bytes > 40 * 1024) PPP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return PPP_OK;
}


// A few bytes of device memory to the host in stream order, then synchronise: a tiny kernel stores
// them into mapped pinned memory.  Unlike a cudaMemcpyAsync this does not queue behind a large
// device->host copy another stream has in flight on the copy engine (the mid-chain size fetches of
// the slicing path otherwise stall until the normals' 32 MB copy has drained).
constexpr size_t FETCH_BYTES = 64 * 1024;
int fetch_small(ppp_ctx* ctx, const void* dev_src, size_t bytes, void* host_dst);
// The flag word behind the payload area and the host side of the hand-shake: a kernel on ctx->stream stores its
// payload into ctx->fetch_host, fences (system scope) and stores `seq` into the flag; the host spins on the flag --
// a few hundred nanoseconds after the store lands, where waking up from cudaStreamSynchronize costs several
// microseconds -- and looks at the stream's status now and then so that a failed kernel cannot hang it.
inline volatile unsigned* fetch_flag(ppp_ctx* ctx) { return (volatile unsigned*)((char*)ctx->fetch_host + FETCH_BYTES); }
int fetch_wait(ppp_ctx* ctx, unsigned seq);

// Stream-ordered device memory.  dev_alloc: a temporary of the current API call (tracked until
// dev_free, see ApiScope); dev_alloc_keep: memory that outlives the call (cloud, grids, result buffers).
template <typename T>
int dev_alloc_keep(ppp_ctx* ctx, T** p, size_t count) {
  *p = nullptr;
  if (count == 0) count = 1;
  cudaError_t e = cudaMallocAsync((void**)p, count * sizeof(T), ctx->stream);
  if (e != cudaSuccess) {
    ppp_set_error("cudaMallocAsync(%zu bytes): %s", count * sizeof(T), cudaGetErrorString(e));
    cudaGetLastError();
    return e == cudaErrorMemoryAllocation ? PPP_ERR_NOMEM : PPP_ERR_CUDA;
  }
  return PPP_OK;
}
template <typename T>
int dev_alloc(ppp_ctx* ctx, T** p, size_t count) {
  int st = dev_alloc_keep(ctx, p, count);
  if (st == PPP_OK && ctx->api_depth > 0) ctx->temps.push_back((void*)*p);
  return st;
}
template <typename T>
void dev_free(ppp_ctx* ctx, T* p) {
  if (!p) return;
  for (size_t i = ctx->temps.size(); i-- > 0;)
    if (ctx->temps[i] == (void*)p) { ctx->temps.erase(ctx->temps.begin() + (long)i); break; }
  cudaFreeAsync((void*)p, ctx->stream);
}

// One per extern "C" entry point (the LOCK macro): holds the context mutex for the call and, when the
// outermost call returns, frees the temporaries an error path did not get to.
struct ApiScope {
  ppp_ctx* ctx;
  std::lock_guard<std::recursive_mutex> lk;
  explicit ApiScope(ppp_ctx* c) : ctx(c), lk(c->mu) { ctx->api_depth++; }
  ~ApiScope() {
    if (--ctx->api_depth == 0 && !ctx->temps.empty()) {
      cudaDeviceSynchronize();   // error path: kernels on either stream may still use them
      cudaGetLastError();
      for (void* p : ctx->temps) cudaFreeAsync(p, ctx->main_stream);
      ctx->temps.clear();
    }
  }
};

// scan.cu
int scan_exclusive_i32(ppp_ctx* ctx, const int32_t* in, int32_t* out, int64_t n);       // out[n] = total too (n+1 outputs)
int scan_exclusive_i32_to_i64(ppp_ctx* ctx, const int32_t* in, int64_t* out, int64_t n);  // n+1 outputs

// grid.cu
int cloud_ingest(ppp_cloud* c, const void* pts_dev, size_t stride_bytes);
int cloud_ingest_ex(ppp_cloud* c, const void* pts_dev, size_t stride_bytes, int64_t n_cap, const long long* n_dev,
                    const void* extra_src, size_t extra_bytes, void* extra_out);
int cloud_get_grid(ppp_cloud* c, double h, GridStore** out);               // primary projection
int grid_sorted_order(ppp_cloud* c, GridStore& gs);                        // builds gs.order on first request
int cloud_get_grid_drop(ppp_cloud* c, double h, int drop, GridStore** out);
// Decides (once per cloud, one synchronisation) whether the primary column grid `g` piles points up; afterwards
// c->mp_state is 0 or 1.
int cloud_decide_projection(ppp_cloud* c, const GridStore& g);
// The three grids of cell size h and the per-point choice for candidate blocks of (2*R0+1)^2 cells.
int cloud_get_mp(ppp_cloud* c, double h, int R0, MPSet** out);
double cloud_cell_for_k(const ppp_cloud* c, int k);
double cloud_cell_for_radius(const ppp_cloud* c, double r);

// knn.cu
// choice / my_proj (multi-projection index): only the self-queries whose point chose projection my_proj are
// answered by this call (through the grid `g`, which must be that projection's); the caller loops over the three.
int knn_launch(ppp_cloud* c, const GridStore& g, const float* q_dev, int64_t nq, int q_stride_f, int64_t first,
               int k, int32_t* idx_dev, float* d2_dev, bool with_normals, const float vp[3], unsigned flags,
               float* normals_dev, int normal_stride_f, const unsigned char* choice = nullptr, int my_proj = 0);
int radius_count_launch(ppp_cloud* c, const GridStore& g, const float* q_dev, int64_t nq, int q_stride_f,
                        int64_t first, float r2, int32_t* counts_dev);
int radius_fill_launch(ppp_cloud* c, const GridStore& g, const float* q_dev, int64_t nq, int q_stride_f,
                       int64_t first, float r2, const int64_t* offsets_dev, int32_t* idx_dev, float* d2_dev);
int normals_radius_launch(ppp_cloud* c, const GridStore& g, int64_t first, int64_t count, float r2,
                          const float vp[3], unsigned flags, float* normals_dev, int normal_stride_f,
                          const unsigned char* choice = nullptr, int my_proj = 0);

int principal_curvatures_launch(ppp_cloud* c, const int32_t* idx_dev, int64_t nq, int k, const float* normals_dev,
                                int normal_stride_f, float* out_dev, int32_t* nn0_dev);
int sor_mean_distances_launch(ppp_cloud* c, const GridStore& gs, int mean_k, int sqrt_float, float* dist_dev,
                              unsigned long long* n_valid_dev);
// Cells of the ring block around a query that cover radius r on grid g (two at cloud_cell_for_radius's cell size).
int radius_rings(const GridView& g, double r);
int coverage_mark_launch(ppp_cloud* c, const GridStore& gs, const float* q_dev, int64_t nq, int q_stride_f, float r2,
                         unsigned char* flags_dev, const float* r2_per_query_dev = nullptr);

// mls.cu
// ppp_mls_smooth's device part: compacted rows (xyz_c: 3 floats per row; nrm_c nullable: nx ny nz curvature;
// src_c: source index) for every finite point with >= 3 neighbours, in ascending source order.  Synchronises.
int mls_smooth_launch(ppp_cloud* c, double radius, int order, float* xyz_c, float4* nrm_c, int32_t* src_c, int64_t* n_rows);
// ppp_dev_mls_smooth's device part: one 32-byte record per point (by original index into rec, or to the home ranks
// through c->route on an exchange slab, where only owned rows are queries).  Does not synchronise.
int mls_smooth_records(ppp_cloud* c, double radius, int order, float* rec);
// ppp_dev_mls_compact's device part: *n_rows = rows of the n records; with points_out, rows [row_base, row_base +
// *n_rows) are written (PPP_ERR_CAPACITY past cap_rows).  Synchronises once.
int mls_compact_launch(ppp_ctx* ctx, const float* rec, int64_t n, const float* src_rec, int out_sf, int32_t idx_base,
                       int64_t row_base, float* points_out, float4* normals_out, int32_t* src_out, int64_t cap_rows,
                       int64_t* n_rows);
// The exchange halo an MLS call of this radius needs (ppp_mls_halo).
double mls_halo(double radius, double x_abs_max);

// voxel.cu
// ppp_voxel_grid's and ppp_dev_voxel_grid's device part (leaf already validated): one record of sf words per voxel in
// ascending key order into rows_dev (room for n records; x, y, z, 1.0f, the averaged rgba word 4 of the source
// records src when it is not NULL, zeros elsewhere), row_off_dev (rows + 1) and members_dev (the n_finite source
// indices grouped by row, ascending within a row).  PPP_ERR_UNSUPPORTED where PCL refuses the leaf, before anything is
// written.  Synchronises.
int voxel_grid_launch(ppp_cloud* c, const float leaf[3], const float* src, int sf, float* rows_dev, int64_t* row_off_dev,
                      int32_t* members_dev, int64_t* n_rows);

// slices.cu
int bands_launch(ppp_cloud* c, const float* plane_x_host, int S, float half_width, int truncate_center, int sort_bands,
                 int64_t** offsets_dev_out, int32_t** idx_dev_out, int64_t* total_out, float** planes_dev_out,
                 std::vector<int64_t>* offsets_host_out);
int contours_launch(ppp_cloud* c, const GridStore& g, const float* planes_dev, int S, const int64_t* band_off_dev,
                    const int32_t* band_idx_dev, int64_t band_total, const std::vector<int64_t>& band_off_host, int mode,
                    int64_t* total_nodes_out, const uint32_t* member_bits = nullptr, const MPSet* mp = nullptr);
int slice_contours_sect_async(ppp_cloud* c, const GridStore& gs, const float* plane_x_host, int S, float half_width,
                              int truncate_center, int64_t* total_nodes_out, int64_t* total_members_out, const MPSet* mp = nullptr);
int contours_from_indices_launch(ppp_cloud* c, const GridStore& gs, const int32_t* idx_host, int64_t m, float plane_x,
                                 int mode, int64_t* total_nodes_out, const MPSet* mp = nullptr);
