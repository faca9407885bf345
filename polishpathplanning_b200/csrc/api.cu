// extern "C" surface of libppp_gpu.so (include/ppp_gpu.h): context, cloud handles, host-pointer
// wrappers around the device pipeline.  No CPU fallback anywhere: without a usable CUDA device
// ppp_create fails and nothing else can be called.
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

#include "ppp_internal.cuh"
#include <cstring>
#include <cuda.h>

static thread_local char g_err[1024] = "";

void ppp_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

#define LOCK(ctx) ApiScope _api_scope(ctx)

#define REQUIRE(cond, msg)            \
  do {                                \
    if (!(cond)) {                    \
      ppp_set_error("%s: %s", __func__, msg); \
      return PPP_ERR_INVALID;         \
    }                                 \
  } while (0)

extern "C" {

int ppp_abi_version(void) { return PPP_ABI_VERSION; }
const char* ppp_last_error(void) { return g_err; }

int ppp_create(int device, ppp_ctx** out) {
  if (!out) { ppp_set_error("ppp_create: out is NULL"); return PPP_ERR_INVALID; }
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    ppp_set_error("ppp_create: no CUDA device (%s); libppp_gpu has no CPU fallback",
                  e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    cudaGetLastError();
    return PPP_ERR_CUDA;
  }
  if (device < 0 || device >= ndev) { ppp_set_error("ppp_create: device %d out of range [0,%d)", device, ndev); return PPP_ERR_INVALID; }
  PPP_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  PPP_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) {
    ppp_set_error("ppp_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
    return PPP_ERR_UNSUPPORTED;
  }
  ppp_ctx* ctx = new ppp_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  ctx->smem_optin = prop.sharedMemPerBlockOptin;
  int prio_lo = 0, prio_hi = 0;
  PPP_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
  PPP_CUDA(cudaStreamCreateWithPriority(&ctx->main_stream, cudaStreamNonBlocking, prio_lo));
  PPP_CUDA(cudaStreamCreateWithPriority(&ctx->aux_stream, cudaStreamNonBlocking, prio_hi));
  PPP_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  PPP_CUDA(cudaHostAlloc(&ctx->fetch_host, FETCH_BYTES + 128, cudaHostAllocMapped));
  *fetch_flag(ctx) = 0u;
  ctx->stream = ctx->main_stream;
  cudaMemPool_t pool;
  PPP_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
  uint64_t thr = UINT64_MAX;  // keep freed blocks cached: temporaries are re-used every call
  PPP_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
  *out = ctx;
  return PPP_OK;
}

void ppp_destroy(ppp_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->main_stream);
  cudaStreamSynchronize(ctx->aux_stream);
  for (auto& kv : ctx->kstats)
    for (auto& p : kv.second.pending) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); }
  for (int t = 0; t < 16; t++)
    for (auto& p : ctx->t_pending[t]) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); }
  cudaStreamDestroy(ctx->main_stream);
  if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->fetch_host) cudaFreeHost(ctx->fetch_host);
  for (int i = 0; i < 2; i++) if (ctx->scan_state[i]) cudaFree(ctx->scan_state[i]);
  if (ctx->ingest_dev) cudaFree(ctx->ingest_dev);
  delete ctx;
}

void* ppp_stream(ppp_ctx* ctx) { return ctx ? (void*)ctx->main_stream : nullptr; }

int ppp_sync(ppp_ctx* ctx) {
  REQUIRE(ctx, "ctx is NULL");
  PPP_CUDA(cudaStreamSynchronize(ctx->main_stream));
  return PPP_OK;
}

void* ppp_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return p;
}
void ppp_host_free(void* p) { if (p) cudaFreeHost(p); }

int64_t ppp_launch_count(ppp_ctx* ctx) { return ctx ? ctx->launches : 0; }

int ppp_timer_begin(ppp_ctx* ctx, int tag) {
  REQUIRE(ctx && tag >= 0 && tag < 16, "bad ctx/tag");
  LOCK(ctx);
  cudaEvent_t a, b;
  PPP_CUDA(cudaEventCreate(&a));
  PPP_CUDA(cudaEventCreate(&b));
  PPP_CUDA(cudaEventRecord(a, ctx->main_stream));
  ctx->t_pending[tag].emplace_back(a, b);
  return PPP_OK;
}
int ppp_timer_end(ppp_ctx* ctx, int tag) {
  REQUIRE(ctx && tag >= 0 && tag < 16, "bad ctx/tag");
  LOCK(ctx);
  REQUIRE(!ctx->t_pending[tag].empty(), "timer_end without timer_begin");
  PPP_CUDA(cudaEventRecord(ctx->t_pending[tag].back().second, ctx->main_stream));
  return PPP_OK;
}
int ppp_timer_read(ppp_ctx* ctx, int tag, double* total_ms, int64_t* regions, int reset) {
  REQUIRE(ctx && tag >= 0 && tag < 16, "bad ctx/tag");
  LOCK(ctx);
  PPP_CUDA(cudaStreamSynchronize(ctx->main_stream));
  for (auto& p : ctx->t_pending[tag]) {
    float ms = 0;
    PPP_CUDA(cudaEventElapsedTime(&ms, p.first, p.second));
    ctx->t_ms[tag] += ms;
    ctx->t_regions[tag]++;
    cudaEventDestroy(p.first);
    cudaEventDestroy(p.second);
  }
  ctx->t_pending[tag].clear();
  if (total_ms) *total_ms = ctx->t_ms[tag];
  if (regions) *regions = ctx->t_regions[tag];
  if (reset) { ctx->t_ms[tag] = 0; ctx->t_regions[tag] = 0; }
  return PPP_OK;
}

int ppp_kernel_profile(ppp_ctx* ctx, int enable) {
  REQUIRE(ctx, "ctx is NULL");
  LOCK(ctx);
  ctx->profile = enable != 0;
  return PPP_OK;
}
int ppp_kernel_profile_read(ppp_ctx* ctx, char* buf, size_t cap, int reset) {
  REQUIRE(ctx && buf && cap > 0, "bad arguments");
  LOCK(ctx);
  PPP_CUDA(cudaStreamSynchronize(ctx->main_stream));
  PPP_CUDA(cudaStreamSynchronize(ctx->aux_stream));
  std::string s;
  for (auto& kv : ctx->kstats) {
    KernelStat& st = kv.second;
    for (auto& p : st.pending) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, p.first, p.second) == cudaSuccess) { st.ms += ms; st.launches++; }
      cudaEventDestroy(p.first);
      cudaEventDestroy(p.second);
    }
    st.pending.clear();
    char line[256];
    snprintf(line, sizeof(line), "%s=%.6f:%lld;", kv.first.c_str(), st.ms, (long long)st.launches);
    s += line;
  }
  if (reset) ctx->kstats.clear();
  snprintf(buf, cap, "%s", s.c_str());
  return PPP_OK;
}

int ppp_kernel_trace(ppp_ctx* ctx, int enable) {
  REQUIRE(ctx, "ctx is NULL");
  LOCK(ctx);
  ctx->trace = enable != 0;
  if (ctx->trace) {
    if (!ctx->trace_base) PPP_CUDA(cudaEventCreate(&ctx->trace_base));
    PPP_CUDA(cudaEventRecord(ctx->trace_base, ctx->main_stream));
  }
  return PPP_OK;
}
int ppp_kernel_trace_read(ppp_ctx* ctx, char* buf, size_t cap) {
  REQUIRE(ctx && buf && cap > 0, "bad arguments");
  LOCK(ctx);
  PPP_CUDA(cudaStreamSynchronize(ctx->main_stream));
  PPP_CUDA(cudaStreamSynchronize(ctx->aux_stream));
  std::string s;
  for (auto& r : ctx->trace_recs) {
    float t0 = 0, t1 = 0;
    if (ctx->trace_base && cudaEventElapsedTime(&t0, ctx->trace_base, r.a) == cudaSuccess &&
        cudaEventElapsedTime(&t1, ctx->trace_base, r.b) == cudaSuccess) {
      char line[256];
      snprintf(line, sizeof(line), "%s=%d:%.6f:%.6f;", r.name, r.aux, t0, t1);
      s += line;
    }
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  cudaGetLastError();
  ctx->trace_recs.clear();
  snprintf(buf, cap, "%s", s.c_str());
  return PPP_OK;
}

// ---------------------------------------------------------------------------------------------
// cloud
// ---------------------------------------------------------------------------------------------
static int cloud_new(ppp_ctx* ctx, size_t n, ppp_cloud** out) {
  ppp_cloud* c = new ppp_cloud();
  c->ctx = ctx;
  c->n = (int64_t)n;
  c->grids.reserve(48);   // pointers into these vectors are handed out: they never reallocate
  c->mps.reserve(16);
  *out = c;
  return PPP_OK;
}

int ppp_dev_cloud_attach(ppp_ctx* ctx, const void* pts_dev, size_t n, size_t stride_bytes, ppp_cloud** out) {
  REQUIRE(ctx && out, "ctx/out is NULL");
  REQUIRE(stride_bytes >= 12 && stride_bytes % 4 == 0, "stride_bytes must be >= 12 and a multiple of 4");
  REQUIRE(n == 0 || pts_dev, "pts is NULL");
  REQUIRE(n < 2147483647ull, "at most 2^31-2 points (int32 indices, as PCL)");
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  ppp_cloud* c = nullptr;
  PPP_TRY(cloud_new(ctx, n, &c));
  int st = cloud_ingest(c, pts_dev, stride_bytes);
  if (st != PPP_OK) { ppp_cloud_free(c); return st; }
  *out = c;
  return PPP_OK;
}

int ppp_cloud_upload(ppp_ctx* ctx, const void* pts_host, size_t n, size_t stride_bytes, ppp_cloud** out) {
  REQUIRE(ctx && out, "ctx/out is NULL");
  REQUIRE(stride_bytes >= 12 && stride_bytes % 4 == 0, "stride_bytes must be >= 12 and a multiple of 4");
  REQUIRE(n == 0 || pts_host, "pts is NULL");
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  void* raw = nullptr;
  PPP_TRY(dev_alloc(ctx, (char**)&raw, std::max<size_t>(n * stride_bytes, 16)));
  if (n) PPP_CUDA(cudaMemcpyAsync(raw, pts_host, n * stride_bytes, cudaMemcpyHostToDevice, ctx->stream));
  int st = ppp_dev_cloud_attach(ctx, raw, n, stride_bytes, out);
  dev_free(ctx, (char*)raw);
  return st;
}

int ppp_cloud_free(ppp_cloud* c) {
  if (!c) return PPP_OK;
  ppp_ctx* ctx = c->ctx;
  LOCK(ctx);
  cudaSetDevice(ctx->device);
  dev_free(ctx, c->xyz4);
  for (auto& g : c->grids) {
    dev_free(ctx, g.sorted); dev_free(ctx, g.cell_start); dev_free(ctx, g.order);
    if (g.ready) cudaEventDestroy(g.ready);
  }
  for (auto& m : c->mps) {
    dev_free(ctx, m.choice);
    if (m.ready) cudaEventDestroy(m.ready);
  }
  dev_free(ctx, c->c_node_off); dev_free(ctx, c->c_y); dev_free(ctx, c->c_x); dev_free(ctx, c->c_z);
  delete c;
  return PPP_OK;
}

int64_t ppp_cloud_size(const ppp_cloud* c) { return c ? c->n : -1; }

int ppp_cloud_bbox(const ppp_cloud* c, float mn[3], float mx[3]) {
  REQUIRE(c && mn && mx, "NULL argument");
  for (int d = 0; d < 3; d++) { mn[d] = c->bmin[d]; mx[d] = c->bmax[d]; }
  return PPP_OK;
}

int ppp_cloud_set_cell_hint(ppp_cloud* c, float cell) {
  REQUIRE(c, "cloud is NULL");
  REQUIRE(cell >= 0 && std::isfinite(cell), "cell size must be >= 0");
  c->cell_hint = cell;
  return PPP_OK;
}

int ppp_dev_set_contour_buffers(ppp_cloud* c, double* y_dev, double* x_dev, double* z_dev, int64_t cap) {
  REQUIRE(c, "cloud is NULL");
  REQUIRE((y_dev && x_dev && z_dev && cap > 0) || (!y_dev && !x_dev && !z_dev), "give all three buffers or none");
  c->ext_y = y_dev; c->ext_x = x_dev; c->ext_z = z_dev; c->ext_cap = y_dev ? cap : 0;
  return PPP_OK;
}

int ppp_dev_set_contour_offsets_buffer(ppp_cloud* c, int64_t* offsets_dev, int64_t cap_entries) {
  REQUIRE(c, "cloud is NULL");
  REQUIRE((offsets_dev && cap_entries > 0) || (!offsets_dev && cap_entries == 0), "give a buffer and its capacity, or neither");
  c->ext_off = offsets_dev; c->ext_off_cap = cap_entries;
  return PPP_OK;
}

// Stream-ordered 32-bit flags (stream memory operations, no kernel): signal = write `value` once all
// earlier work of the context's stream has finished; wait = hold later work of the stream until
// *flag >= value.  The flag may live in a peer buffer, which makes the pair a cross-GPU completion
// signal for data delivered with plain NVLink stores.
typedef CUresult (*stream_write32_fn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
typedef CUresult (*stream_wait32_fn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
static int driver_entry(const char* name, void** fn) {
  cudaDriverEntryPointQueryResult qr;
  cudaError_t e = cudaGetDriverEntryPoint(name, fn, cudaEnableDefault, &qr);
  if (e != cudaSuccess || qr != cudaDriverEntryPointSuccess || !*fn) {
    ppp_set_error("driver entry point %s unavailable", name);
    return PPP_ERR_UNSUPPORTED;
  }
  return PPP_OK;
}

int ppp_dev_signal(ppp_ctx* ctx, uint32_t* flag_dev, uint32_t value) {
  REQUIRE(ctx && flag_dev, "NULL argument");
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  static stream_write32_fn fn = nullptr;
  if (!fn) PPP_TRY(driver_entry("cuStreamWriteValue32", (void**)&fn));
  CUresult r = fn((CUstream)ctx->stream, (CUdeviceptr)(uintptr_t)flag_dev, value, CU_STREAM_WRITE_VALUE_DEFAULT);
  if (r != CUDA_SUCCESS) { ppp_set_error("cuStreamWriteValue32 failed (%d)", (int)r); return PPP_ERR_CUDA; }
  return PPP_OK;
}

int ppp_dev_wait(ppp_ctx* ctx, const uint32_t* flag_dev, uint32_t value) {
  REQUIRE(ctx && flag_dev, "NULL argument");
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  static stream_wait32_fn fn = nullptr;
  if (!fn) PPP_TRY(driver_entry("cuStreamWaitValue32", (void**)&fn));
  CUresult r = fn((CUstream)ctx->stream, (CUdeviceptr)(uintptr_t)flag_dev, value, CU_STREAM_WAIT_VALUE_GEQ);
  if (r != CUDA_SUCCESS) { ppp_set_error("cuStreamWaitValue32 failed (%d)", (int)r); return PPP_ERR_CUDA; }
  return PPP_OK;
}

int ppp_dev_set_normal_row_map(ppp_cloud* c, const int32_t* row_map_dev) {
  REQUIRE(c, "cloud is NULL");
  c->nmap = row_map_dev;
  return PPP_OK;
}

// Buffers other processes' GPUs can write: plain cudaMalloc memory exported as a CUDA IPC handle.
int ppp_peer_buffer_alloc(ppp_ctx* ctx, size_t bytes, void** dev_ptr, unsigned char handle[PPP_PEER_HANDLE_BYTES]) {
  REQUIRE(ctx && dev_ptr && handle && bytes > 0, "bad argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == PPP_PEER_HANDLE_BYTES, "handle size");
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  void* p = nullptr;
  PPP_CUDA(cudaMalloc(&p, bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaMemset(p, 0, bytes);
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    ppp_set_error("peer buffer (memset / cudaIpcGetMemHandle): %s", cudaGetErrorString(e));
    return PPP_ERR_CUDA;
  }
  memcpy(handle, &h, sizeof(h));
  *dev_ptr = p;
  return PPP_OK;
}

int ppp_peer_buffer_open(ppp_ctx* ctx, const unsigned char handle[PPP_PEER_HANDLE_BYTES], void** dev_ptr) {
  REQUIRE(ctx && dev_ptr && handle, "bad argument");
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  PPP_CUDA(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return PPP_OK;
}

int ppp_peer_buffer_close(ppp_ctx* ctx, void* dev_ptr) {
  REQUIRE(ctx, "context is NULL");
  if (!dev_ptr) return PPP_OK;
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  PPP_CUDA(cudaIpcCloseMemHandle(dev_ptr));
  return PPP_OK;
}

int ppp_peer_buffer_free(ppp_ctx* ctx, void* dev_ptr) {
  REQUIRE(ctx, "context is NULL");
  if (!dev_ptr) return PPP_OK;
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  PPP_CUDA(cudaFree(dev_ptr));
  return PPP_OK;
}

int ppp_dev_download(ppp_ctx* ctx, void* host_dst, const void* dev_src, size_t bytes) {
  REQUIRE(ctx && (bytes == 0 || (host_dst && dev_src)), "bad argument");
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  if (bytes) PPP_CUDA(cudaMemcpyAsync(host_dst, dev_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  PPP_CUDA(cudaStreamSynchronize(ctx->stream));
  return PPP_OK;
}

const int32_t* ppp_dev_sorted_order(ppp_cloud* c) {
  if (!c || c->grids.empty()) return nullptr;
  ApiScope scope(c->ctx);
  if (cudaSetDevice(c->ctx->device) != cudaSuccess) return nullptr;
  if (grid_sorted_order(c, c->grids.back()) != PPP_OK) return nullptr;
  return c->grids.back().order;
}

int ppp_dev_index(ppp_cloud* c, int k_hint, double radius_hint) {
  REQUIRE(c, "cloud is NULL");
  LOCK(c->ctx);
  PPP_CUDA(cudaSetDevice(c->ctx->device));
  GridStore* g;
  double h = radius_hint > 0 ? cloud_cell_for_radius(c, radius_hint) : cloud_cell_for_k(c, k_hint > 0 ? k_hint : 16);
  return cloud_get_grid(c, h, &g);
}

// ---------------------------------------------------------------------------------------------
// device-level pipeline entries
// ---------------------------------------------------------------------------------------------
int ppp_dev_normals_knn(ppp_cloud* c, int k, const float vp[3], unsigned flags, int64_t first, int64_t count,
                        float* normals_dev, size_t normal_stride_bytes, int32_t* knn_idx_dev, float* knn_d2_dev) {
  REQUIRE(c, "cloud is NULL");
  REQUIRE(k >= 1, "k must be >= 1");
  REQUIRE(normal_stride_bytes >= 16 && normal_stride_bytes % 4 == 0, "normal stride must be >= 16 and a multiple of 4");
  REQUIRE(normals_dev || knn_idx_dev, "nothing to compute");
  LOCK(c->ctx);
  PPP_CUDA(cudaSetDevice(c->ctx->device));
  if (count < 0) count = c->n_finite - first;
  REQUIRE(first >= 0 && first + count <= c->n_finite, "query range outside the indexed points");
  GridStore* g;
  const double h = cloud_cell_for_k(c, k);
  PPP_TRY(cloud_get_grid(c, h, &g));
  PPP_TRY(cloud_decide_projection(c, *g));
  if (c->mp_state == 1 && first == 0 && count == c->n_finite && k <= 64) {
    // not a height field: one grid per axis pair, every point searched in the projection that spreads its
    // neighbourhood out best (three launches, each warp leaves at once unless some of its points are its own)
    MPSet* mp;
    PPP_TRY(cloud_get_mp(c, h, PPP_KNN_RINGS, &mp));
    for (int p = 0; p < 3; p++)
      PPP_TRY(knn_launch(c, *mp->g[p], nullptr, count, 0, 0, k, knn_idx_dev, knn_d2_dev, normals_dev != nullptr, vp, flags,
                         normals_dev, (int)(normal_stride_bytes / 4), mp->choice, p));
    return PPP_OK;
  }
  return knn_launch(c, *g, nullptr, count, 0, first, k, knn_idx_dev, knn_d2_dev, normals_dev != nullptr, vp, flags,
                    normals_dev, (int)(normal_stride_bytes / 4));
}

int ppp_dev_normals_radius(ppp_cloud* c, double radius, const float vp[3], unsigned flags, int64_t first, int64_t count,
                           float* normals_dev, size_t normal_stride_bytes) {
  REQUIRE(c && normals_dev, "NULL argument");
  REQUIRE(radius > 0 && std::isfinite(radius), "radius must be > 0");
  REQUIRE(normal_stride_bytes >= 16 && normal_stride_bytes % 4 == 0, "normal stride must be >= 16 and a multiple of 4");
  LOCK(c->ctx);
  PPP_CUDA(cudaSetDevice(c->ctx->device));
  if (count < 0) count = c->n_finite - first;
  REQUIRE(first >= 0 && first + count <= c->n_finite, "query range outside the indexed points");
  GridStore* g;
  const double h = cloud_cell_for_radius(c, radius);
  PPP_TRY(cloud_get_grid(c, h, &g));
  float r2 = (float)(radius * radius);  // [upstream] pcl::KdTreeFLANN::radiusSearch
  PPP_TRY(cloud_decide_projection(c, *g));
  if (c->mp_state == 1 && first == 0 && count == c->n_finite) {
    MPSet* mp;
    PPP_TRY(cloud_get_mp(c, h, 2, &mp));     // cloud_cell_for_radius sizes the cells so that two rings cover the radius
    for (int p = 0; p < 3; p++)
      PPP_TRY(normals_radius_launch(c, *mp->g[p], 0, count, r2, vp, flags, normals_dev, (int)(normal_stride_bytes / 4), mp->choice, p));
    return PPP_OK;
  }
  return normals_radius_launch(c, *g, first, count, r2, vp, flags, normals_dev, (int)(normal_stride_bytes / 4));
}

static int pick_any_grid(ppp_cloud* c, GridStore** g) {
  for (size_t i = c->grids.size(); i-- > 0;)
    if (c->grids[i].drop == c->drop) { *g = &c->grids[i]; return PPP_OK; }
  return cloud_get_grid(c, cloud_cell_for_k(c, 16), g);
}

int ppp_dev_slice_contours(ppp_cloud* c, const float* plane_x_host, int S, float half_width, int truncate_center,
                           int pairing_mode, const int64_t** node_offsets_dev, const double** y_dev,
                           const double** x_dev, const double** z_dev, int64_t* total_nodes, int64_t* total_members) {
  REQUIRE(c, "cloud is NULL");
  REQUIRE(S >= 0 && (S == 0 || plane_x_host), "bad planes");
  REQUIRE(pairing_mode == PPP_PAIR_GEN2 || pairing_mode == PPP_PAIR_SECT, "unknown pairing mode");
  REQUIRE(half_width >= 0 && std::isfinite(half_width), "half_width must be >= 0");
  ppp_ctx* ctx = c->ctx;
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  GridStore* g;
  PPP_TRY(pick_any_grid(c, &g));
  PPP_TRY(cloud_decide_projection(c, *g));
  MPSet* mp = nullptr;
  if (c->mp_state == 1) PPP_TRY(cloud_get_mp(c, g->h, PPP_KNN_RINGS, &mp));
  int st;
  int64_t M = 0, total = 0;
  {
    // The slicing chain depends on the packed cloud and the grid only, not on the neighbour
    // search: it runs on the high-priority auxiliary stream, concurrently with a kNN / normals
    // kernel still executing on the main stream; the main stream waits for it on scope exit.
    AuxScope aux(ctx, mp ? mp->ready : g->ready);   // (the projections are built after the primary grid)
    // SectPath pairing: the chain without mid-way host round trips, unless its allocation bound is too large
    st = pairing_mode == PPP_PAIR_SECT && !getenv("PPP_SLICE_SYNC")
             ? slice_contours_sect_async(c, *g, plane_x_host, S, half_width, truncate_center, &total, &M, mp)
             : PPP_ERR_UNSUPPORTED;
    if (st == PPP_ERR_UNSUPPORTED) {
      int64_t* boff = nullptr; int32_t* bidx = nullptr; float* planes = nullptr;
      std::vector<int64_t> off_h;
      st = bands_launch(c, plane_x_host, S, half_width, truncate_center, pairing_mode == PPP_PAIR_GEN2, &boff, &bidx, &M,
                        &planes, &off_h);
      if (st == PPP_OK) st = contours_launch(c, *g, planes, S, boff, bidx, M, off_h, pairing_mode, &total, nullptr, mp);
      dev_free(ctx, boff); dev_free(ctx, bidx); dev_free(ctx, planes);
    }
  }
  if (st != PPP_OK) return st;
  if (node_offsets_dev) *node_offsets_dev = c->c_node_off;
  if (y_dev) *y_dev = c->out_y;
  if (x_dev) *x_dev = c->out_x;
  if (z_dev) *z_dev = c->out_z;
  if (total_nodes) *total_nodes = total;
  if (total_members) *total_members = M;
  return PPP_OK;
}

// ---------------------------------------------------------------------------------------------
// host-pointer API
// ---------------------------------------------------------------------------------------------
int ppp_knn(ppp_cloud* c, const float* q, size_t nq, size_t q_stride_bytes, int k, int32_t* idx_out, float* d2_out) {
  REQUIRE(c && (idx_out || (q ? nq == 0 : c->n == 0)), "NULL argument");
  REQUIRE(k >= 1, "k must be >= 1");
  REQUIRE(!q || (q_stride_bytes >= 12 && q_stride_bytes % 4 == 0), "query stride must be >= 12 and a multiple of 4");
  ppp_ctx* ctx = c->ctx;
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  GridStore* g;
  PPP_TRY(cloud_get_grid(c, cloud_cell_for_k(c, k), &g));
  int64_t rows = q ? (int64_t)nq : c->n;
  int32_t* idx_d = nullptr; float* d2_d = nullptr; float* q_d = nullptr;
  PPP_TRY(dev_alloc(ctx, &idx_d, (size_t)rows * k));
  if (d2_out) PPP_TRY(dev_alloc(ctx, &d2_d, (size_t)rows * k));
  int st;
  if (q) {
    PPP_TRY(dev_alloc(ctx, (char**)&q_d, nq * q_stride_bytes + 16));
    if (nq) PPP_CUDA(cudaMemcpyAsync(q_d, q, nq * q_stride_bytes, cudaMemcpyHostToDevice, ctx->stream));
    st = knn_launch(c, *g, q_d, (int64_t)nq, (int)(q_stride_bytes / 4), 0, k, idx_d, d2_d, false, nullptr, 0, nullptr, 0);
  } else {
    st = knn_launch(c, *g, nullptr, c->n_finite, 0, 0, k, idx_d, d2_d, false, nullptr, 0, nullptr, 0);
  }
  if (st == PPP_OK && rows) {
    PPP_CUDA(cudaMemcpyAsync(idx_out, idx_d, (size_t)rows * k * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (d2_out) PPP_CUDA(cudaMemcpyAsync(d2_out, d2_d, (size_t)rows * k * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  dev_free(ctx, idx_d); dev_free(ctx, d2_d); dev_free(ctx, (char*)q_d);
  if (st != PPP_OK) return st;
  PPP_CUDA(e);
  return PPP_OK;
}

int ppp_radius(ppp_cloud* c, const float* q, size_t nq, size_t q_stride_bytes, double radius, int32_t* counts,
               const int64_t* offsets, int32_t* idx_out, float* d2_out) {
  REQUIRE(c && counts, "NULL argument");
  REQUIRE(radius > 0 && std::isfinite(radius), "radius must be > 0");
  REQUIRE(!q || (q_stride_bytes >= 12 && q_stride_bytes % 4 == 0), "query stride must be >= 12 and a multiple of 4");
  REQUIRE(!idx_out || offsets, "offsets required with idx_out");
  ppp_ctx* ctx = c->ctx;
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  GridStore* g;
  PPP_TRY(cloud_get_grid(c, cloud_cell_for_radius(c, radius), &g));
  float r2 = (float)(radius * radius);
  int64_t rows = q ? (int64_t)nq : c->n;
  int64_t nquery = q ? (int64_t)nq : c->n_finite;
  float* q_d = nullptr;
  if (q) {
    PPP_TRY(dev_alloc(ctx, (char**)&q_d, nq * q_stride_bytes + 16));
    if (nq) PPP_CUDA(cudaMemcpyAsync(q_d, q, nq * q_stride_bytes, cudaMemcpyHostToDevice, ctx->stream));
  }
  int qsf = (int)(q_stride_bytes / 4);
  int32_t* cnt_d = nullptr;
  PPP_TRY(dev_alloc(ctx, &cnt_d, (size_t)rows));
  int st = PPP_OK;
  if (!idx_out) {
    int mx = radius_count_launch(c, *g, q_d, nquery, qsf, 0, r2, cnt_d);
    if (mx < 0) st = mx;
    if (st == PPP_OK && rows) PPP_CUDA(cudaMemcpyAsync(counts, cnt_d, (size_t)rows * 4, cudaMemcpyDeviceToHost, ctx->stream));
  } else {
    int64_t total = offsets[rows];
    int64_t* off_d = nullptr; int32_t* idx_d = nullptr; float* d2_d = nullptr;
    PPP_TRY(dev_alloc(ctx, &off_d, (size_t)rows + 1));
    PPP_TRY(dev_alloc(ctx, &idx_d, (size_t)std::max<int64_t>(total, 1)));
    if (d2_out) PPP_TRY(dev_alloc(ctx, &d2_d, (size_t)std::max<int64_t>(total, 1)));
    PPP_CUDA(cudaMemcpyAsync(off_d, offsets, ((size_t)rows + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    st = radius_fill_launch(c, *g, q_d, nquery, qsf, 0, r2, off_d, idx_d, d2_d);
    if (st == PPP_OK && total) {
      PPP_CUDA(cudaMemcpyAsync(idx_out, idx_d, (size_t)total * 4, cudaMemcpyDeviceToHost, ctx->stream));
      if (d2_out) PPP_CUDA(cudaMemcpyAsync(d2_out, d2_d, (size_t)total * 4, cudaMemcpyDeviceToHost, ctx->stream));
    }
    cudaStreamSynchronize(ctx->stream);
    dev_free(ctx, off_d); dev_free(ctx, idx_d); dev_free(ctx, d2_d);
  }
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  dev_free(ctx, cnt_d); dev_free(ctx, (char*)q_d);
  if (st != PPP_OK) return st;
  PPP_CUDA(e);
  return PPP_OK;
}

static int normals_host(ppp_cloud* c, int k, double radius, const float vp[3], unsigned flags, void* normals_out,
                        size_t stride, int32_t* knn_idx_out) {
  ppp_ctx* ctx = c->ctx;
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  float* n_d = nullptr; int32_t* idx_d = nullptr;
  size_t nbytes = (size_t)c->n * stride;
  PPP_TRY(dev_alloc(ctx, (char**)&n_d, std::max<size_t>(nbytes, 16)));
  if (stride > 32) PPP_CUDA(cudaMemsetAsync(n_d, 0, nbytes, ctx->stream));
  if (knn_idx_out) PPP_TRY(dev_alloc(ctx, &idx_d, (size_t)c->n * k));
  int st = k > 0 ? ppp_dev_normals_knn(c, k, vp, flags, 0, -1, n_d, stride, idx_d, nullptr)
                 : ppp_dev_normals_radius(c, radius, vp, flags, 0, -1, n_d, stride);
  if (st == PPP_OK && c->n) {
    PPP_CUDA(cudaMemcpyAsync(normals_out, n_d, nbytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (knn_idx_out) PPP_CUDA(cudaMemcpyAsync(knn_idx_out, idx_d, (size_t)c->n * k * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  dev_free(ctx, (char*)n_d); dev_free(ctx, idx_d);
  if (st != PPP_OK) return st;
  PPP_CUDA(e);
  return PPP_OK;
}

int ppp_normals_knn(ppp_cloud* c, int k, const float vp[3], unsigned flags, void* normals_out, size_t stride,
                    int32_t* knn_idx_out) {
  REQUIRE(c && (normals_out || c->n == 0), "NULL argument");
  REQUIRE(k >= 1, "k must be >= 1");
  REQUIRE(stride >= 16 && stride % 4 == 0, "normal stride must be >= 16 and a multiple of 4");
  if (c->n == 0) return PPP_OK;
  return normals_host(c, k, 0.0, vp, flags, normals_out, stride, knn_idx_out);
}

int ppp_normals_radius(ppp_cloud* c, double radius, const float vp[3], unsigned flags, void* normals_out, size_t stride) {
  REQUIRE(c && (normals_out || c->n == 0), "NULL argument");
  REQUIRE(radius > 0 && std::isfinite(radius), "radius must be > 0");
  REQUIRE(stride >= 16 && stride % 4 == 0, "normal stride must be >= 16 and a multiple of 4");
  if (c->n == 0) return PPP_OK;  // the reference carries on with an empty cloud after a failed load
  return normals_host(c, 0, radius, vp, flags, normals_out, stride, nullptr);
}

int ppp_slice_bands(ppp_cloud* c, const float* plane_x, int S, float half_width, int truncate_center, int64_t* offsets,
                    int32_t* idx_out, int64_t idx_cap) {
  REQUIRE(c && offsets, "NULL argument");
  REQUIRE(S >= 0 && (S == 0 || plane_x), "bad planes");
  REQUIRE(half_width >= 0 && std::isfinite(half_width), "half_width must be >= 0");
  ppp_ctx* ctx = c->ctx;
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  int64_t* boff = nullptr; int32_t* bidx = nullptr; float* planes = nullptr; int64_t M = 0;
  PPP_TRY(bands_launch(c, plane_x, S, half_width, truncate_center, 1, &boff, &bidx, &M, &planes, nullptr));
  int st = PPP_OK;
  PPP_CUDA(cudaMemcpyAsync(offsets, boff, ((size_t)S + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (idx_out) {
    if (idx_cap < M) { ppp_set_error("ppp_slice_bands: idx_cap %lld < required %lld", (long long)idx_cap, (long long)M); st = PPP_ERR_CAPACITY; }
    else if (M) PPP_CUDA(cudaMemcpyAsync(idx_out, bidx, (size_t)M * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  dev_free(ctx, boff); dev_free(ctx, bidx); dev_free(ctx, planes);
  PPP_CUDA(e);
  return st;
}

// Is p ordinary page-locked host memory (cudaHostAlloc / cudaHostRegister)?  Under UVA such memory is
// addressable from kernels with the same pointer value.
static bool host_ptr_is_pinned(const void* p) {
  if (!p) return false;
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return at.type == cudaMemoryTypeHost && at.devicePointer == p;
}

int ppp_slice_contours(ppp_cloud* c, const float* plane_x, int S, float half_width, int truncate_center, int pairing_mode,
                       int64_t* node_offsets, double* y, double* x, double* z, int64_t node_cap) {
  REQUIRE(c && node_offsets, "NULL argument");
  REQUIRE(!y || (x && z), "y, x, z must be given together");
  ppp_ctx* ctx = c->ctx;
  LOCK(ctx);
  const int64_t* off_d; const double *y_d, *x_d, *z_d; int64_t total = 0, M = 0;
  // Page-locked result arrays are filled by the compaction kernel itself (coalesced stores over PCIe
  // while the chain runs): three separate ~1 MB device->host copies measured ~80 us EACH here.
  const bool direct = y && node_cap > 0 && host_ptr_is_pinned(y) && host_ptr_is_pinned(x) && host_ptr_is_pinned(z);
  double *sy = c->ext_y, *sx = c->ext_x, *sz = c->ext_z;
  const int64_t scap = c->ext_cap;
  if (direct) { c->ext_y = y; c->ext_x = x; c->ext_z = z; c->ext_cap = node_cap; }
  int st = ppp_dev_slice_contours(c, plane_x, S, half_width, truncate_center, pairing_mode, &off_d, &y_d, &x_d, &z_d, &total, &M);
  if (direct) { c->ext_y = sy; c->ext_x = sx; c->ext_z = sz; c->ext_cap = scap; }
  if (st != PPP_OK) return st;
  PPP_TRY(fetch_small(ctx, off_d, ((size_t)S + 1) * 8, node_offsets));   // synchronises the stream
  if (y) {
    if (node_cap < total) {
      ppp_set_error("ppp_slice_contours: node_cap %lld < required %lld", (long long)node_cap, (long long)total);
      return PPP_ERR_CAPACITY;
    }
    if (total && y_d != y) {
      PPP_CUDA(cudaMemcpyAsync(y, y_d, (size_t)total * 8, cudaMemcpyDeviceToHost, ctx->stream));
      PPP_CUDA(cudaMemcpyAsync(x, x_d, (size_t)total * 8, cudaMemcpyDeviceToHost, ctx->stream));
      PPP_CUDA(cudaMemcpyAsync(z, z_d, (size_t)total * 8, cudaMemcpyDeviceToHost, ctx->stream));
      PPP_CUDA(cudaStreamSynchronize(ctx->stream));
    }
  }
  return PPP_OK;
}

// estimate_normal() + the whole plane sweep in one call (the gen-3 GenPath does exactly this
// sequence: src/Path_Alg/path_dynamic_alg.cpp:343 then the sweep).  Same results as
// ppp_normals_knn / ppp_normals_radius followed by ppp_slice_contours; the device->host copy of
// the normals runs on a second stream while the band / pairing / ordering kernels execute.
int ppp_normals_and_contours(ppp_cloud* c, int k, double radius, const float vp[3], unsigned flags, void* normals_out,
                             size_t stride, const float* plane_x, int S, float half_width, int truncate_center,
                             int pairing_mode, int64_t* node_offsets, double* y, double* x, double* z, int64_t node_cap) {
  REQUIRE(c && node_offsets && (normals_out || c->n == 0), "NULL argument");
  REQUIRE((k >= 1) != (radius > 0), "give either k >= 1 or radius > 0");
  REQUIRE(stride >= 16 && stride % 4 == 0, "normal stride must be >= 16 and a multiple of 4");
  REQUIRE(!y || (x && z), "y, x, z must be given together");
  ppp_ctx* ctx = c->ctx;
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  float* n_d = nullptr;
  size_t nbytes = (size_t)c->n * stride;
  cudaEvent_t ev = nullptr;
  int st = PPP_OK;
  if (c->n > 0) {
    PPP_TRY(dev_alloc(ctx, (char**)&n_d, std::max<size_t>(nbytes, 16)));
    if (stride > 32) PPP_CUDA(cudaMemsetAsync(n_d, 0, nbytes, ctx->stream));
    st = k >= 1 ? ppp_dev_normals_knn(c, k, vp, flags, 0, -1, n_d, stride, nullptr, nullptr)
                : ppp_dev_normals_radius(c, radius, vp, flags, 0, -1, n_d, stride);
    if (st == PPP_OK) {
      PPP_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
      PPP_CUDA(cudaEventRecord(ev, ctx->stream));
      PPP_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ev, 0));
      PPP_CUDA(cudaMemcpyAsync(normals_out, n_d, nbytes, cudaMemcpyDeviceToHost, ctx->copy_stream));
      // Host-pointer path: the long pole after the search is the normals' device->host copy, so the
      // search must finish as early as possible.  Hold the slicing chain (auxiliary stream) until the
      // search is done; it then runs in the shadow of the copy instead of competing for the SMs.
      PPP_CUDA(cudaStreamWaitEvent(ctx->aux_stream, ev, 0));
    }
  }
  if (st == PPP_OK) st = ppp_slice_contours(c, plane_x, S, half_width, truncate_center, pairing_mode, node_offsets, y, x, z, node_cap);
  cudaError_t e = cudaStreamSynchronize(ctx->copy_stream);
  if (ev) cudaEventDestroy(ev);
  dev_free(ctx, (char*)n_d);
  if (st != PPP_OK) return st;
  PPP_CUDA(e);
  return PPP_OK;
}

// compute_coverage (src/Path_Generation.cpp:483-496) for a batch of nodes: flags (N bytes, host,
// in/out) gets 1 for every point within `radius` (d2 < (float)(r*r)) of any query.
int ppp_coverage_mark(ppp_cloud* c, const float* q, size_t nq, size_t q_stride_bytes, double radius, unsigned char* flags) {
  REQUIRE(c && (flags || c->n == 0), "NULL argument");
  REQUIRE(nq == 0 || q, "queries are NULL");
  REQUIRE(radius > 0 && std::isfinite(radius), "radius must be > 0");
  REQUIRE(q_stride_bytes >= 12 && q_stride_bytes % 4 == 0, "query stride must be >= 12 and a multiple of 4");
  ppp_ctx* ctx = c->ctx;
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  if (c->n == 0 || nq == 0) return PPP_OK;
  GridStore* g;
  PPP_TRY(cloud_get_grid(c, cloud_cell_for_radius(c, radius), &g));
  unsigned char* f_d = nullptr; float* q_d = nullptr;
  PPP_TRY(dev_alloc(ctx, &f_d, (size_t)c->n));
  PPP_TRY(dev_alloc(ctx, (char**)&q_d, nq * q_stride_bytes + 16));
  PPP_CUDA(cudaMemcpyAsync(f_d, flags, (size_t)c->n, cudaMemcpyHostToDevice, ctx->stream));
  PPP_CUDA(cudaMemcpyAsync(q_d, q, nq * q_stride_bytes, cudaMemcpyHostToDevice, ctx->stream));
  int st = coverage_mark_launch(c, *g, q_d, (int64_t)nq, (int)(q_stride_bytes / 4), (float)(radius * radius), f_d);
  if (st == PPP_OK) PPP_CUDA(cudaMemcpyAsync(flags, f_d, (size_t)c->n, cudaMemcpyDeviceToHost, ctx->stream));
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  dev_free(ctx, f_d); dev_free(ctx, (char*)q_d);
  if (st != PPP_OK) return st;
  PPP_CUDA(e);
  return PPP_OK;
}

// compute_coverage for a batch of nodes that each bring their OWN radius: what Area2Cloud does for every path
// node (src/Path_Generation.cpp:466-470: compute_coverage(point, comput_lan), the half-width of the node's
// contact ellipse; the value is negative there and PCL squares it, so only |radius| matters).
// A NaN radius marks nothing.
int ppp_coverage_mark_radii(ppp_cloud* c, const float* q, size_t nq, size_t q_stride_bytes, const double* radii,
                            unsigned char* flags) {
  REQUIRE(c && (flags || c->n == 0), "NULL argument");
  REQUIRE(nq == 0 || (q && radii), "queries / radii are NULL");
  REQUIRE(q_stride_bytes >= 12 && q_stride_bytes % 4 == 0, "query stride must be >= 12 and a multiple of 4");
  ppp_ctx* ctx = c->ctx;
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  if (c->n == 0 || nq == 0) return PPP_OK;
  std::vector<float> r2(nq);
  double rmax = 0, rfin = 0;   // largest |radius| (NaN radii mark nothing), largest finite one
  for (size_t i = 0; i < nq; i++) {
    r2[i] = (float)(radii[i] * radii[i]);   // [upstream] pcl::KdTreeFLANN::radiusSearch squares the radius in double
    const double a = std::fabs(radii[i]);
    if (a > rmax) rmax = a;
    if (std::isfinite(a) && a > rfin) rfin = a;
  }
  if (!(rmax > 0)) return PPP_OK;
  // The block radius below covers the largest radius, infinite ones included (an infinite float32 r2 marks every
  // finite point); any cell size serves those, so the grid is sized by the finite radii.
  GridStore* g;
  PPP_TRY(cloud_get_grid(c, rfin > 0 ? cloud_cell_for_radius(c, rfin) : cloud_cell_for_k(c, 16), &g));
  unsigned char* f_d = nullptr; float* q_d = nullptr; float* r_d = nullptr;
  PPP_TRY(dev_alloc(ctx, &f_d, (size_t)c->n));
  PPP_TRY(dev_alloc(ctx, (char**)&q_d, nq * q_stride_bytes + 16));
  PPP_TRY(dev_alloc(ctx, &r_d, nq));
  PPP_CUDA(cudaMemcpyAsync(f_d, flags, (size_t)c->n, cudaMemcpyHostToDevice, ctx->stream));
  PPP_CUDA(cudaMemcpyAsync(q_d, q, nq * q_stride_bytes, cudaMemcpyHostToDevice, ctx->stream));
  PPP_CUDA(cudaMemcpyAsync(r_d, r2.data(), nq * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  int st = coverage_mark_launch(c, *g, q_d, (int64_t)nq, (int)(q_stride_bytes / 4), (float)(rmax * rmax), f_d, r_d);
  if (st == PPP_OK) PPP_CUDA(cudaMemcpyAsync(flags, f_d, (size_t)c->n, cudaMemcpyDeviceToHost, ctx->stream));
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  dev_free(ctx, f_d); dev_free(ctx, (char*)q_d); dev_free(ctx, r_d);
  if (st != PPP_OK) return st;
  PPP_CUDA(e);
  return PPP_OK;
}

// compute_transform's device part for a batch of query points (src/Path_Generation.cpp:362-400):
// kNN(k) of each query, then computePointPrincipalCurvatures around neighbour [0] on the given
// normals (n records of normal_stride_bytes, nx ny nz first).  out: nq x 5 floats
// (pcx, pcy, pcz, pc1, pc2); nn0 (nullable): index of the nearest point (whose normal the caller
// crosses with the curvature direction).
int ppp_principal_curvatures(ppp_cloud* c, const void* normals, size_t normal_stride_bytes, const float* q, size_t nq,
                             size_t q_stride_bytes, int k, float* out, int32_t* nn0) {
  REQUIRE(c && normals && (nq == 0 || (q && out)), "NULL argument");
  REQUIRE(k >= 1, "k must be >= 1");
  REQUIRE(normal_stride_bytes >= 12 && normal_stride_bytes % 4 == 0, "normal stride must be >= 12 and a multiple of 4");
  REQUIRE(q_stride_bytes >= 12 && q_stride_bytes % 4 == 0, "query stride must be >= 12 and a multiple of 4");
  ppp_ctx* ctx = c->ctx;
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  if (nq == 0) return PPP_OK;
  GridStore* g;
  PPP_TRY(cloud_get_grid(c, cloud_cell_for_k(c, k), &g));
  float *q_d = nullptr, *n_d = nullptr, *o_d = nullptr;
  int32_t *idx_d = nullptr, *nn0_d = nullptr;
  PPP_TRY(dev_alloc(ctx, (char**)&q_d, nq * q_stride_bytes + 16));
  PPP_TRY(dev_alloc(ctx, (char**)&n_d, (size_t)c->n * normal_stride_bytes + 16));
  PPP_TRY(dev_alloc(ctx, &o_d, nq * 5));
  PPP_TRY(dev_alloc(ctx, &idx_d, nq * (size_t)k));
  PPP_TRY(dev_alloc(ctx, &nn0_d, nq));
  PPP_CUDA(cudaMemcpyAsync(q_d, q, nq * q_stride_bytes, cudaMemcpyHostToDevice, ctx->stream));
  PPP_CUDA(cudaMemcpyAsync(n_d, normals, (size_t)c->n * normal_stride_bytes, cudaMemcpyHostToDevice, ctx->stream));
  int st = knn_launch(c, *g, q_d, (int64_t)nq, (int)(q_stride_bytes / 4), 0, k, idx_d, nullptr, false, nullptr, 0, nullptr, 0);
  if (st == PPP_OK)
    st = principal_curvatures_launch(c, idx_d, (int64_t)nq, k, n_d, (int)(normal_stride_bytes / 4), o_d, nn0_d);
  if (st == PPP_OK) {
    PPP_CUDA(cudaMemcpyAsync(out, o_d, nq * 5 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (nn0) PPP_CUDA(cudaMemcpyAsync(nn0, nn0_d, nq * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  }
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  dev_free(ctx, (char*)q_d); dev_free(ctx, (char*)n_d); dev_free(ctx, o_d); dev_free(ctx, idx_d); dev_free(ctx, nn0_d);
  if (st != PPP_OK) return st;
  PPP_CUDA(e);
  return PPP_OK;
}

// insert_point(std::vector<int> indices, Eigen::Vector3f PlanePoint) with the caller's own index
// list (src/Path_Generation.cpp:107-206, src/contour_alg.cpp:165-237).  indices must be strictly
// ascending and in range, as rangedX_index returns them.  y/x/z hold node_cap nodes; *n_nodes is the
// node count (PPP_ERR_CAPACITY if it exceeds node_cap; y == NULL: count only).
int ppp_insert_point(ppp_cloud* c, const int32_t* indices, int64_t m, float plane_x, int pairing_mode, double* y,
                     double* x, double* z, int64_t node_cap, int64_t* n_nodes) {
  REQUIRE(c && n_nodes && (m == 0 || indices), "NULL argument");
  REQUIRE(m >= 0, "negative index count");
  REQUIRE(pairing_mode == PPP_PAIR_GEN2 || pairing_mode == PPP_PAIR_SECT, "unknown pairing mode");
  REQUIRE(!y || (x && z), "y, x, z must be given together");
  for (int64_t i = 0; i < m; i++) {
    REQUIRE(indices[i] >= 0 && indices[i] < c->n, "index out of range");
    REQUIRE(i == 0 || indices[i] > indices[i - 1], "indices must be strictly ascending");
  }
  ppp_ctx* ctx = c->ctx;
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  GridStore* g;
  PPP_TRY(pick_any_grid(c, &g));
  PPP_TRY(cloud_decide_projection(c, *g));
  MPSet* mp = nullptr;
  if (c->mp_state == 1) PPP_TRY(cloud_get_mp(c, g->h, PPP_KNN_RINGS, &mp));
  int64_t total = 0;
  PPP_TRY(contours_from_indices_launch(c, *g, indices, m, plane_x, pairing_mode, &total, mp));
  *n_nodes = total;
  int st = PPP_OK;
  if (y) {
    if (node_cap < total) {
      ppp_set_error("ppp_insert_point: node_cap %lld < required %lld", (long long)node_cap, (long long)total);
      st = PPP_ERR_CAPACITY;
    } else if (total) {
      PPP_CUDA(cudaMemcpyAsync(y, c->out_y, (size_t)total * 8, cudaMemcpyDeviceToHost, ctx->stream));
      PPP_CUDA(cudaMemcpyAsync(x, c->out_x, (size_t)total * 8, cudaMemcpyDeviceToHost, ctx->stream));
      PPP_CUDA(cudaMemcpyAsync(z, c->out_z, (size_t)total * 8, cudaMemcpyDeviceToHost, ctx->stream));
    }
  }
  PPP_CUDA(cudaStreamSynchronize(ctx->stream));
  return st;
}

// First pass of pcl::StatisticalOutlierRemoval as SectPath::remove_outlier runs it
// (src/contour_alg.cpp:101-108, mean_k = 50): dist_out[i] = (float)(sum_j sqrt(d2_j) / mean_k) over the
// mean_k nearest neighbours of point i (itself excluded), 0 for non-finite points; *n_valid = number of
// finite points.  The reference's sequential mean / stddev / threshold pass over dist_out stays with
// the caller (host adapters: remove_outlier).
int ppp_sor_mean_distances(ppp_cloud* c, int mean_k, unsigned flags, float* dist_out, int64_t* n_valid) {
  REQUIRE(c && n_valid && (dist_out || c->n == 0), "NULL argument");
  REQUIRE(mean_k >= 1, "mean_k must be >= 1");
  REQUIRE((flags & ~(unsigned)PPP_SOR_SQRT_FLOAT) == 0, "unknown flags");
  ppp_ctx* ctx = c->ctx;
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  if (c->n_finite <= mean_k) {
    ppp_set_error("ppp_sor_mean_distances: %lld finite points, need more than mean_k = %d", (long long)c->n_finite, mean_k);
    return PPP_ERR_UNSUPPORTED;
  }
  GridStore* g;
  PPP_TRY(cloud_get_grid(c, cloud_cell_for_k(c, mean_k + 1), &g));
  float* dist_d = nullptr; unsigned long long* nv_d = nullptr;
  PPP_TRY(dev_alloc(ctx, &dist_d, (size_t)c->n));
  PPP_TRY(dev_alloc(ctx, &nv_d, 1));
  int st = sor_mean_distances_launch(c, *g, mean_k, (flags & PPP_SOR_SQRT_FLOAT) ? 1 : 0, dist_d, nv_d);
  unsigned long long nv = 0;
  if (st == PPP_OK) {
    PPP_CUDA(cudaMemcpyAsync(dist_out, dist_d, (size_t)c->n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PPP_CUDA(cudaMemcpyAsync(&nv, nv_d, 8, cudaMemcpyDeviceToHost, ctx->stream));
  }
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  dev_free(ctx, dist_d); dev_free(ctx, nv_d);
  if (st != PPP_OK) return st;
  PPP_CUDA(e);
  *n_valid = (int64_t)nv;
  return PPP_OK;
}

// smooth(): pcl::MovingLeastSquares with polynomial order `order` and search radius `radius`
// (src/Path_Generation.cpp:340-360), no upsampling, SIMPLE projection.  Rows are written for the finite points
// with at least 3 neighbours, in ascending source order; points_out / normals_out / src_index_out hold n rows.
int ppp_mls_smooth(ppp_cloud* c, double radius, int order, void* points_out, size_t out_stride_bytes, float* normals_out,
                   int32_t* src_index_out, int64_t* n_out) {
  REQUIRE(c && n_out && ((points_out && src_index_out) || c->n == 0), "NULL argument");
  REQUIRE(radius > 0 && std::isfinite((float)(radius * radius)), "radius must be > 0 with a finite float32 square");
  REQUIRE(order >= 0 && order <= 3, "order must be 0..3");
  REQUIRE(out_stride_bytes >= 12 && out_stride_bytes % 4 == 0, "output stride must be >= 12 and a multiple of 4");
  ppp_ctx* ctx = c->ctx;
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  *n_out = 0;
  if (c->n == 0) return PPP_OK;
  float* xyz_d = nullptr; float4* nrm_d = nullptr; int32_t* src_d = nullptr;
  PPP_TRY(dev_alloc(ctx, &xyz_d, (size_t)c->n * 3));
  if (normals_out) PPP_TRY(dev_alloc(ctx, &nrm_d, (size_t)c->n));
  PPP_TRY(dev_alloc(ctx, &src_d, (size_t)c->n));
  int64_t m = 0;
  int st = mls_smooth_launch(c, radius, order, xyz_d, nrm_d, src_d, &m);
  if (st == PPP_OK && m > 0) {
    PPP_CUDA(cudaMemcpy2DAsync(points_out, out_stride_bytes, xyz_d, 12, 12, (size_t)m, cudaMemcpyDeviceToHost, ctx->stream));
    if (normals_out) PPP_CUDA(cudaMemcpyAsync(normals_out, nrm_d, (size_t)m * 16, cudaMemcpyDeviceToHost, ctx->stream));
    PPP_CUDA(cudaMemcpyAsync(src_index_out, src_d, (size_t)m * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  dev_free(ctx, xyz_d); dev_free(ctx, nrm_d); dev_free(ctx, src_d);
  if (st != PPP_OK) return st;
  PPP_CUDA(e);
  *n_out = m;
  return PPP_OK;
}

double ppp_mls_halo(double radius, double x_abs_max) { return mls_halo(radius, x_abs_max); }

// voxel_down(): pcl::VoxelGrid with leaf sizes leaf[0..2] (src/Path_Generation.cpp:53-59); contract in the header.
int ppp_voxel_grid(ppp_cloud* c, const float leaf[3], void* points_out, size_t out_stride_bytes, int64_t* row_offsets,
                   int32_t* members, int64_t* n_out) {
  REQUIRE(c && leaf && n_out && (points_out || c->n == 0), "NULL argument");
  for (int d = 0; d < 3; d++)
    REQUIRE(leaf[d] > 0 && std::isfinite(leaf[d]) && std::isfinite(1.0f / leaf[d]),
            "leaf sizes must be > 0 and finite, with a finite float inverse");
  REQUIRE(out_stride_bytes >= 12 && out_stride_bytes % 4 == 0, "output stride must be >= 12 and a multiple of 4");
  ppp_ctx* ctx = c->ctx;
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  *n_out = 0;
  if (c->n_finite == 0) {
    if (row_offsets) row_offsets[0] = 0;
    return PPP_OK;
  }
  float4* rows_d = nullptr; int64_t* off_d = nullptr; int32_t* mem_d = nullptr;
  PPP_TRY(dev_alloc(ctx, &rows_d, (size_t)c->n));
  PPP_TRY(dev_alloc(ctx, &off_d, (size_t)c->n + 1));
  PPP_TRY(dev_alloc(ctx, &mem_d, (size_t)c->n));
  int64_t m = 0;
  int st = voxel_grid_launch(c, leaf, rows_d, off_d, mem_d, &m);
  std::vector<float4> rows;
  if (st == PPP_OK) {
    rows.resize((size_t)m);
    PPP_CUDA(cudaMemcpyAsync(rows.data(), rows_d, (size_t)m * 16, cudaMemcpyDeviceToHost, ctx->stream));
    if (row_offsets) PPP_CUDA(cudaMemcpyAsync(row_offsets, off_d, (size_t)(m + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (members) PPP_CUDA(cudaMemcpyAsync(members, mem_d, (size_t)c->n_finite * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  dev_free(ctx, rows_d); dev_free(ctx, off_d); dev_free(ctx, mem_d);
  if (st != PPP_OK) return st;
  PPP_CUDA(e);
  const size_t put = out_stride_bytes >= 16 ? 16 : 12;   // x, y, z and the pad float where the record has one
  for (int64_t r = 0; r < m; r++) memcpy((char*)points_out + (size_t)r * out_stride_bytes, &rows[(size_t)r], put);
  *n_out = m;
  return PPP_OK;
}

// ppp_mls_smooth's per-point part with the results left in device memory: one 32-byte record per point, by original
// index, or on an exchange slab to the home ranks (only owned rows are queries there).  Does not synchronise.
int ppp_dev_mls_smooth(ppp_cloud* c, double radius, int order, void* rows_dev, size_t row_stride_bytes) {
  REQUIRE(c, "cloud is NULL");
  REQUIRE(radius > 0 && std::isfinite((float)(radius * radius)), "radius must be > 0 with a finite float32 square");
  REQUIRE(order >= 0 && order <= 3, "order must be 0..3");
  REQUIRE(row_stride_bytes == 32, "records are 32 bytes: {x, y, z, flag, nx, ny, nz, curvature}");
  if (c->route) {
    REQUIRE(c->nmap, "an exchange slab needs its row map (ppp_dev_set_normal_row_map(NULL) cleared it)");
    REQUIRE(c->ex_home_bytes == 32, "the exchange keeps 16-byte home records; MLS records need an exchange created with 32");
    const double need = mls_halo(radius, c->ex_xmag);
    if (!(c->ex_halo >= need)) {
      ppp_set_error("ppp_dev_mls_smooth: the exchange halo %.17g is narrower than the %.17g radius %.17g needs (ppp_mls_halo)",
                    c->ex_halo, need, radius);
      return PPP_ERR_INVALID;
    }
  } else {
    REQUIRE(rows_dev || c->n == 0, "rows_dev is NULL");
    REQUIRE((uintptr_t)rows_dev % 16 == 0, "rows_dev must be 16-byte aligned");
  }
  LOCK(c->ctx);
  PPP_CUDA(cudaSetDevice(c->ctx->device));
  return mls_smooth_records(c, radius, order, (float*)rows_dev);
}

// Records [0, n) -> rows in source order (see the header).  Synchronises once.
int ppp_dev_mls_compact(ppp_ctx* ctx, const void* rows_dev, int64_t n, const void* src_dev, size_t src_stride_bytes,
                        int64_t src_index_base, int64_t row_base, void* points_out, size_t out_stride_bytes, float* normals_out,
                        int32_t* src_index_out, int64_t cap_rows, int64_t* n_rows) {
  REQUIRE(ctx && n_rows, "NULL argument");
  *n_rows = 0;
  REQUIRE(n >= 0 && (rows_dev || n == 0) && (uintptr_t)rows_dev % 16 == 0, "rows_dev: n 16-byte aligned records");
  REQUIRE(src_index_base >= 0 && src_index_base + n <= 2147483647ll, "source indices must fit int32");
  const bool fill = points_out || src_index_out || normals_out;
  if (fill) {
    REQUIRE(points_out && src_index_out, "points_out and src_index_out are both needed to fill");
    REQUIRE(out_stride_bytes >= 12 && out_stride_bytes % 4 == 0, "output stride must be >= 12 and a multiple of 4");
    REQUIRE(!src_dev || src_stride_bytes == out_stride_bytes, "source records must have the output stride");
    REQUIRE((uintptr_t)normals_out % 16 == 0, "normals_out must be 16-byte aligned");
    REQUIRE(row_base >= 0 && cap_rows >= 0, "bad row base / capacity");
  }
  LOCK(ctx);
  PPP_CUDA(cudaSetDevice(ctx->device));
  PPP_TRY(mls_compact_launch(ctx, (const float*)rows_dev, n, fill ? (const float*)src_dev : nullptr, (int)(out_stride_bytes / 4),
                            (int32_t)src_index_base, row_base, fill ? (float*)points_out : nullptr, (float4*)normals_out,
                            src_index_out, cap_rows, n_rows));
  if (fill) PPP_CUDA(cudaStreamSynchronize(ctx->stream));   // the rows are in place (host memory included) on return
  return PPP_OK;
}

}  // extern "C"
