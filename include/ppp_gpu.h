/* ppp_gpu.h — C ABI of libppp_gpu.so, the B200 (sm_100a) drop-in for the data-parallel geometric
 * core of tsai0507/PolishPathPlanning.
 *
 * The reference has no plugin / FFI boundary: its hot path is a set of C++ member functions that
 * call PCL/FLANN on class-owned clouds (SURVEY.md §8b).  Each entry point below replaces the
 * body of the reference function(s) cited next to it (paths relative to /root/reference); the
 * adapter classes in polishpathplanning_b200/host/ keep the reference's own signatures and call
 * these.  INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *  - plain C, no exceptions cross the boundary; every function returns PPP_OK (0) or a negative
 *    ppp_status; ppp_last_error() gives a message (thread-local).
 *  - "host API": all pointers are HOST memory, calls are synchronous.  "device API" (ppp_dev_*):
 *    data pointers are DEVICE memory on the context's GPU, work is enqueued on ppp_stream()
 *    and the call returns without waiting unless stated.
 *  - points: records of `stride_bytes` (>= 12, multiple of 4) whose first three floats are x,y,z
 *    (pcl::PointXYZRGB: stride 32, include/Path_Generate.h:32-33).  Non-finite points are kept in
 *    the index numbering but never returned as neighbours / band members, as PCL does.
 *  - neighbour order and all ties: ascending (squared distance, point index)  (SURVEY.md App. A.3/A.4).
 *  - one context per GPU per process; query calls on one cloud are serialised internally, so the
 *    reference's two sweep threads (src/Path_Alg/path_dynamic_alg.cpp:308-334) may share a handle.
 *  - there is NO CPU fallback: without a CUDA device ppp_create fails with PPP_ERR_CUDA.
 */
#ifndef PPP_GPU_H
#define PPP_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PPP_ABI_VERSION 2

typedef enum ppp_status {
  PPP_OK = 0,
  PPP_ERR_INVALID = -1,   /* bad argument */
  PPP_ERR_CUDA = -2,      /* CUDA runtime error / no device */
  PPP_ERR_NOMEM = -3,     /* allocation failed */
  PPP_ERR_CAPACITY = -4,  /* caller-provided output too small; required size reported */
  PPP_ERR_UNSUPPORTED = -5
} ppp_status;

typedef struct ppp_ctx ppp_ctx;
typedef struct ppp_cloud ppp_cloud;

/* flags for the normal estimators */
#define PPP_COV_PCL110 0u   /* PCL 1.10.0 single-pass E[xx]-E[x]E[x] covariance (default) */
#define PPP_COV_SHIFTED 1u  /* later PCL: first neighbour subtracted before accumulation */

/* pairing modes of ppp_slice_contours */
#define PPP_PAIR_GEN2 0 /* variant A: path_generater::insert_point, src/Path_Generation.cpp:107-206 */
#define PPP_PAIR_SECT 1 /* variant B: SectPath::insert_point,      src/contour_alg.cpp:165-237   */

/* ------------------------------------------------------------------------------------------ */
/* context                                                                                      */
int ppp_abi_version(void);
int ppp_create(int device, ppp_ctx** out);
void ppp_destroy(ppp_ctx* ctx);
const char* ppp_last_error(void);
void* ppp_stream(ppp_ctx* ctx); /* cudaStream_t all work of this context is enqueued on */
int ppp_sync(ppp_ctx* ctx);
/* pinned host staging buffers (optional; any host memory is accepted by the host API) */
void* ppp_host_alloc(size_t bytes);
void ppp_host_free(void* p);
/* Number of kernels this library has launched on the context since creation (bench gpu_launches). */
int64_t ppp_launch_count(ppp_ctx* ctx);
/* CUDA-event timing on the context's stream: tag 0..15; begin/end bracket a region, read returns
 * the accumulated milliseconds and number of regions since the last reset (synchronises). */
int ppp_timer_begin(ppp_ctx* ctx, int tag);
int ppp_timer_end(ppp_ctx* ctx, int tag);
int ppp_timer_read(ppp_ctx* ctx, int tag, double* total_ms, int64_t* regions, int reset);
/* Per-kernel device time of the library's own kernels (CUDA events around each launch while
 * enabled). names: ';'-separated "name=ms_total:launches" written into buf. */
int ppp_kernel_profile(ppp_ctx* ctx, int enable);
int ppp_kernel_profile_read(ppp_ctx* ctx, char* buf, size_t cap, int reset);
/* Launch trace: while enabled every launch is bracketed by CUDA events on the stream it really runs on
 * (the overlap of the two working streams is kept, unlike the profile above).  read: ';'-separated
 * "name=stream:start_ms:end_ms" relative to the moment the trace was enabled; clears the trace. */
int ppp_kernel_trace(ppp_ctx* ctx, int enable);
int ppp_kernel_trace_read(ppp_ctx* ctx, char* buf, size_t cap);

/* ------------------------------------------------------------------------------------------ */
/* cloud = device-resident copy + spatial index.
 * Replaces: pcl::KdTreeFLANN::setInputCloud (Set_kdtree, src/Path_Generation.cpp:335-338,695;
 * src/contour_alg.cpp:292), the private search::KdTree inside NormalEstimation
 * (src/Path_Generation.cpp:326-327) and pcl::getMinMax3D (src/Path_Generation.cpp:293,709). */
int ppp_cloud_upload(ppp_ctx* ctx, const void* pts_host, size_t n, size_t stride_bytes, ppp_cloud** out);
int ppp_dev_cloud_attach(ppp_ctx* ctx, const void* pts_dev, size_t n, size_t stride_bytes, ppp_cloud** out);
int ppp_cloud_free(ppp_cloud* cloud);
int64_t ppp_cloud_size(const ppp_cloud* cloud);
int ppp_cloud_bbox(const ppp_cloud* cloud, float min_xyz[3], float max_xyz[3]); /* getMinMax3D */
/* Optional tuning: cell size (same unit as the points) used by the next index build for
 * k-searches; 0 = automatic from the cloud's surface density. */
int ppp_cloud_set_cell_hint(ppp_cloud* cloud, float cell_size);

/* ------------------------------------------------------------------------------------------ */
/* neighbour searches.  q == NULL: the cloud's own points are the queries (nq ignored).
 * Replaces pcl::KdTreeFLANN::nearestKSearch / radiusSearch call sites (SURVEY.md §2.2).
 * Order: d2 = ((dx*dx + dy*dy) + dz*dz) in float32, lists sorted by (d2, idx); a query's row holds the
 * min(k, finite points) smallest.  Ties, d2 = inf included, go to the lower index: a query so far away that
 * its float32 d2 to every point overflows gets the k lowest finite indices, each with d2 = inf.  Any finite
 * query is answered exactly, up to +-FLT_MAX; a query with a NaN or infinite coordinate gets -1 / inf.  */
int ppp_knn(ppp_cloud* cloud, const float* q, size_t nq, size_t q_stride_bytes, int k,
            int32_t* idx_out /* nq*k, -1 padded */, float* d2_out /* nullable */);
/* two-call sizing: idx_out == NULL writes counts only; otherwise offsets (nq+1) must be the
 * exclusive scan of counts and lists are written sorted by (d2, idx). Membership d2 < (float)(r*r).
 * LIMIT: a list is ordered in shared memory, so the fill call (and ppp_normals_radius on clouds whose
 * queries have more than 32 neighbours) returns PPP_ERR_UNSUPPORTED when ANY query has more than
 * ~900 neighbours (sharedMemPerBlockOptin / 256 entries; at the reference's radius 2.5 that is a scan
 * denser than ~45 points/mm^2).  Counts-only calls have no limit.
 * A radius whose float32 square overflows (|r| above ~1.84e19) admits every point at a finite d2, as
 * PCL's float comparison does.                                                                     */
int ppp_radius(ppp_cloud* cloud, const float* q, size_t nq, size_t q_stride_bytes, double radius,
               int32_t* counts, const int64_t* offsets, int32_t* idx_out, float* d2_out);

/* ------------------------------------------------------------------------------------------ */
/* estimate_normal(): pcl::NormalEstimation::compute (src/Path_Generation.cpp:323-333,
 * src/contour_alg.cpp:142-151, src/slicing_method.cpp:204-214).  normals_out: n records of
 * normal_stride_bytes; stride 32 = pcl::Normal {nx,ny,nz,0, curvature,0,0,0}; stride 16 = {nx,ny,nz,curvature}.
 * < 3 neighbours or a non-finite point => all four values NaN.  knn_idx_out (n*k) nullable.    */
int ppp_normals_knn(ppp_cloud* cloud, int k, const float viewpoint[3], unsigned flags, void* normals_out,
                    size_t normal_stride_bytes, int32_t* knn_idx_out);
int ppp_normals_radius(ppp_cloud* cloud, double radius, const float viewpoint[3], unsigned flags,
                       void* normals_out, size_t normal_stride_bytes);

/* ------------------------------------------------------------------------------------------ */
/* rangedX_index() for ALL planes in one pass: pcl::PassThrough on "x"
 * (src/Path_Generation.cpp:94-104, src/contour_alg.cpp:153-163).  truncate_center != 0 reproduces
 * the reference's int-truncated band centre: limits (float)(-hw + (int)x), (float)(hw + (int)x).
 * offsets: S+1.  idx_out == NULL: sizing call (offsets only).  idx_cap = capacity of idx_out.  */
int ppp_slice_bands(ppp_cloud* cloud, const float* plane_x, int S, float half_width, int truncate_center,
                    int64_t* offsets, int32_t* idx_out, int64_t idx_cap);

/* rangedX_index + insert_point + the map->array flattening of path_track / OnePath
 * (src/Path_Generation.cpp:107-206,659-676; src/contour_alg.cpp:165-264) for all planes.
 * Output per slice: nodes in ascending y (std::map order, last insertion wins on equal y), as the
 * three double arrays the reference hands to Spline(n, y, x, z) (include/Spline.h:10-20).
 * node_offsets: S+1.  y/x/z capacity node_cap (total); on PPP_ERR_CAPACITY node_offsets[S] holds the
 * required total.  y == NULL: sizing call.                                                     */
int ppp_slice_contours(ppp_cloud* cloud, const float* plane_x, int S, float half_width, int truncate_center,
                       int pairing_mode, int64_t* node_offsets, double* y, double* x, double* z,
                       int64_t node_cap);

/* insert_point(indices, PlanePoint) with the CALLER's index list instead of the band of the plane
 * (same reference lines as above; every reference call site passes rangedX_index(PlanePoint[0]),
 * for which ppp_slice_contours is the one-call equivalent).  indices: strictly ascending.
 * *n_nodes = node count; y == NULL: count only; PPP_ERR_CAPACITY if node_cap is too small.
 * The list may name points that are not finite (a band never does: PassThrough drops them).  Such
 * a point is on neither side of the plane and never a nearest neighbour.  For a NaN or infinite y
 * or z that is the reference's own result: its (p - PlanePoint).dot((1,0,0)) is NaN.  For x = +-inf
 * with finite y and z the reference would put the point on a side and hand it to FLANN as a query,
 * whose answer is not defined; it is dropped here as well.                                      */
int ppp_insert_point(ppp_cloud* cloud, const int32_t* indices, int64_t m, float plane_x, int pairing_mode,
                     double* y, double* x, double* z, int64_t node_cap, int64_t* n_nodes);

/* "next" row of SURVEY.md §8f: the device part of compute_transform (src/Path_Generation.cpp:362-400,
 * k = 10; src/Path_Alg/path_dynamic_alg.cpp:77-110, k = 50) for a batch of query points:
 * kdtree.nearestKSearch(point, k) + PrincipalCurvaturesEstimation::computePointPrincipalCurvatures
 * around neighbour [0].  normals: n host records (nx ny nz first).  out: nq x 5 floats
 * (pcx, pcy, pcz, pc1, pc2); nn0 (nullable): nearest point index per query.                    */
int ppp_principal_curvatures(ppp_cloud* cloud, const void* normals, size_t normal_stride_bytes, const float* q,
                             size_t nq, size_t q_stride_bytes, int k, float* out, int32_t* nn0);

/* "next" row of SURVEY.md §8f-3: first pass of pcl::StatisticalOutlierRemoval as run by
 * SectPath::remove_outlier (src/contour_alg.cpp:101-108; twins src/Path_Alg/path_slicing_alg.cpp:101-108):
 * kNN(mean_k + 1) of every point, dist_out[i] = (float)(sum of the mean_k neighbour distances / mean_k),
 * 0 for non-finite points; *n_valid = finite points.  The sequential mean/stddev/threshold pass over
 * dist_out is the caller's (host adapters' remove_outlier()).  flags: PPP_SOR_SQRT_FLOAT evaluates
 * sqrt(d2) in float (the overload a translation unit with <math.h> picks) instead of double.
 * PPP_ERR_UNSUPPORTED if the cloud has no more than mean_k finite points (the reference reads past
 * the neighbour list there).                                                                      */
#define PPP_SOR_SQRT_FLOAT 1u
int ppp_sor_mean_distances(ppp_cloud* cloud, int mean_k, unsigned flags, float* dist_out, int64_t* n_valid);

/* "next" row of SURVEY.md §8f: compute_coverage (src/Path_Generation.cpp:483-496) for a batch of
 * path nodes.  flags: N bytes (host, in/out); flags[i] = 1 for every point i within `radius` of a
 * query (kdtree.radiusSearch membership).  get_coverage() is the mean of the flags.
 * Flags of points no query reaches are left as they were; a non-finite query marks nothing; a radius
 * whose float32 square overflows marks every point at a finite d2.                               */
int ppp_coverage_mark(ppp_cloud* cloud, const float* q, size_t nq, size_t q_stride_bytes, double radius,
                      unsigned char* flags);

/* The same for nodes that each bring their own radius, as Area2Cloud calls it per path node
 * (src/Path_Generation.cpp:466-470); only |radius| matters (PCL squares it), a NaN radius marks nothing,
 * a zero or subnormal one (float32 square 0) too, and an infinite one, or one whose float32 square
 * overflows, marks every point at a finite d2 from its query. */
int ppp_coverage_mark_radii(ppp_cloud* cloud, const float* q, size_t nq, size_t q_stride_bytes, const double* radii,
                            unsigned char* flags);

/* smooth(): the MLS pre-filter (src/Path_Generation.cpp:340-360; SectPath with Smooth = true,
 * src/contour_alg.cpp:27): pcl::MovingLeastSquares, polynomial order `order` (0..3; 0 and 1 project onto the
 * local plane), search radius `radius`, no upsampling, SIMPLE projection, weight exp(-d^2 / radius^2), normals
 * computed.  One output row per finite point with at least 3 neighbours (d2 < (float)(radius*radius), the point
 * itself included), in ascending source order; other points have none.  The caller provides room for n rows:
 * points_out: records of out_stride_bytes (>= 12, multiple of 4) of which only x, y, z are written;
 * normals_out (nullable): {nx, ny, nz, curvature} per row; src_index_out: source index of each row;
 * *n_out: rows written.
 * Tolerance contract (the fit is double-precision arithmetic summed in a different order than PCL's):
 * the rows and the branch taken per row (polynomial fit or plane) are exact; x, y, z are within 2 float ulps
 * of the CPU restatement and almost always identical; normals and curvature within 1e-5.
 * PPP_ERR_INVALID for a radius whose float32 square overflows (the candidate block would be unbounded). */
int ppp_mls_smooth(ppp_cloud* cloud, double radius, int order, void* points_out, size_t out_stride_bytes,
                   float* normals_out, int32_t* src_index_out, int64_t* n_out);

/* smooth() with the results left in device memory, on one GPU or on the x-slabs of a multi-GPU exchange
 * (src/Path_Generation.cpp:340-360, as ppp_mls_smooth; same radius, order and contract).  Every point gets one
 * record of row_stride_bytes = 32: {x, y, z, flag, nx, ny, nz, curvature}, flag 1.0f where the point has an output
 * row; other records (fewer than 3 neighbours, a non-finite point) have flag 0 and NaN elsewhere.  Every record is
 * written by every call.
 *  - plain cloud: record i of rows_dev (16-byte aligned) is point i's.
 *  - slab from ppp_exch_attach / ppp_exch_finish_attach: rows_dev is ignored; only owned rows are queries (halo copies
 *    are candidates only) and each record is stored into its HOME rank's buffer (ppp_exch_home_normals, record =
 *    global index - starts[home]), over NVLink where the home is another GPU.  ppp_exch_results_signal / _wait with
 *    PPP_EXCH_NORMALS cover these records.  PPP_ERR_INVALID if the exchange was created with 16-byte normal records,
 *    or if the halo any rank's phases were given is narrower than ppp_mls_halo(radius, largest finite |x| of the
 *    cloud) (the ranks publish their halos with the exchange, so every rank refuses together). PPP_ERR_INVALID too if
 *    the slab's row map was cleared.
 * Does not synchronise.  PPP_ERR_INVALID for the radii and orders ppp_mls_smooth refuses. */
int ppp_dev_mls_smooth(ppp_cloud* cloud, double radius, int order, void* rows_dev, size_t row_stride_bytes);
/* Records [0, n) of rows_dev (device memory, e.g. a home buffer) -> rows in ascending record order: *n_rows = rows
 * with flag 1.  Counting call: points_out, normals_out and src_index_out all NULL.  Filling call: rows
 * [row_base, row_base + *n_rows) of points_out (out_stride_bytes; x, y, z from the records, every other field from
 * src_dev, the source records of stride src_stride_bytes = out_stride_bytes, when it is not NULL), normals_out
 * (nullable, 16 bytes a row: nx, ny, nz, curvature) and src_index_out (src_index_base + record number).  The outputs
 * may be device memory or mapped host memory (ppp_host_register, ppp_host_alloc).  PPP_ERR_CAPACITY when
 * row_base + *n_rows > cap_rows (*n_rows is still reported).  Synchronises: after a filling call the rows are in
 * place.  Ranks of an exchange compact their
 * home ranges with row_base = the rows of the lower ranks: together the ranks write ppp_mls_smooth's rows.       */
int ppp_dev_mls_compact(ppp_ctx* ctx, const void* rows_dev, int64_t n, const void* src_dev, size_t src_stride_bytes,
                        int64_t src_index_base, int64_t row_base, void* points_out, size_t out_stride_bytes,
                        float* normals_out, int32_t* src_index_out, int64_t cap_rows, int64_t* n_rows);
/* The exchange halo an MLS call of this radius needs on a cloud whose finite x lie within [-x_abs_max, x_abs_max]:
 * the smallest float t with fl32(t * t) >= (float)(radius * radius), plus 2^-44 * (x_abs_max + t + 1) for the double
 * rounding of the exchange's cut positions (derivation in csrc/mls.cu).  NaN for a radius ppp_mls_smooth refuses. */
double ppp_mls_halo(double radius, double x_abs_max);

/* voxel_down(): pcl::VoxelGrid<PointXYZRGB> (src/Path_Generation.cpp:53-59) with leaf sizes leaf[0..2] and PCL's
 * defaults otherwise (min_points_per_voxel 0, downsample_all_data).  Voxel coordinates are computed as PCL 1.10 does,
 * in float32 from the bounding box of the finite points (ppp_cloud_bbox); non-finite points belong to no voxel.  One
 * row per occupied voxel, in ascending voxel key order: the centroid of its members.  The caller provides room for n
 * rows:
 *   points_out: records of out_stride_bytes (>= 12, multiple of 4) of which only x, y, z (the float32 sum of the
 *               members in ascending source order, divided by (float)count) and, when the stride is >= 16, the pad
 *               float 1.0f at byte 12 are written;
 *   row_offsets (nullable, rows + 1 entries) and members (nullable, one entry per finite point): the members of row r
 *               are members[row_offsets[r] .. row_offsets[r + 1]), ascending source indices (for averaging other
 *               fields, e.g. rgba, on the host);
 *   *n_out: rows written.
 * A cloud without a finite point has 0 rows (PCL leaves that case undefined).
 * PPP_ERR_INVALID for a leaf size that is <= 0 or not finite, or whose float inverse is not finite.
 * PPP_ERR_UNSUPPORTED, with PCL's message "Leaf size is too small for the input dataset. Integer indices would
 * overflow.", where PCL warns and returns the input unchanged: dx * dy * dz > INT32_MAX, dx = (int64)((max.x -
 * min.x) * inv.x) + 1 in float32 (an extent whose product with the inverse leaf is not finite included).  Also
 * PPP_ERR_UNSUPPORTED where floorf(bbox * inv) leaves the int range (PCL's voxel coordinates are undefined there).
 * Contract: the rows, row offsets and members are those of PCL.  PCL sums each voxel in the order its unstable
 * std::sort leaves the members, so a centroid coordinate of a voxel with n members of magnitude <= M can differ from
 * PCL's by at most (2n + 1) * 2^-24 * M; in practice most rows are bit-identical (DESIGN.md §2).          */
int ppp_voxel_grid(ppp_cloud* cloud, const float leaf[3], void* points_out, size_t out_stride_bytes,
                   int64_t* row_offsets, int32_t* members, int64_t* n_out);
/* voxel_down() with the rows left in device memory, as whole records the next cloud can be attached from
 * (ppp_dev_cloud_attach(ctx, rows_dev, *n_rows, stride_bytes, ...)).  Same leaf validation, refusals (PCL's message
 * included), rows, row offsets, members and x, y, z as ppp_voxel_grid.  All buffers are device memory:
 *   rows_dev:        room for ppp_cloud_size(cloud) records of stride_bytes (>= 12, multiple of 4); every word of a
 *                    row's record is written: x, y, z; the pad float 1.0f at byte 12 (stride >= 16); at byte 16
 *                    (stride >= 20) PCL's AccumulatorRGBA over the rgba words at byte 16 of the members' source
 *                    records (per byte channel a float32 sum in ascending source order, divided by the count and
 *                    truncated); 0 elsewhere.  16-byte stores where the stride is a multiple of 16 and rows_dev is
 *                    16-byte aligned;
 *   src_dev:         the cloud's n source records in its index order, of the same stride (the buffer given to
 *                    ppp_dev_cloud_attach); required when stride_bytes >= 20, ignored below;
 *   row_offsets_dev: nullable, room for rows + 1 entries (at most the finite points + 1);
 *   members_dev:     nullable, one entry per finite point (as ppp_voxel_grid's);
 *   *n_rows:         rows written.
 * A cloud without a finite point has 0 rows and row_offsets_dev[0] = 0.  On an error rows_dev is untouched and
 * *n_rows is 0.  Synchronises once: on return the rows are in place. */
int ppp_dev_voxel_grid(ppp_cloud* cloud, const float leaf[3], const void* src_dev, size_t stride_bytes, void* rows_dev,
                       int64_t* row_offsets_dev, int32_t* members_dev, int64_t* n_rows);

/* estimate_normal() followed by the plane sweep, as one call: what SectPath-derived GenPath does
 * (src/Path_Alg/path_dynamic_alg.cpp:343-366: estimate_normal(); kdtree.setInputCloud; sweep).
 * Exactly the results of ppp_normals_knn (k >= 1, radius = 0) or ppp_normals_radius (k = 0,
 * radius > 0) followed by ppp_slice_contours, but the device->host copy of the normals overlaps
 * the slicing kernels.                                                                          */
int ppp_normals_and_contours(ppp_cloud* cloud, int k, double radius, const float viewpoint[3], unsigned flags,
                             void* normals_out, size_t normal_stride_bytes, const float* plane_x, int S,
                             float half_width, int truncate_center, int pairing_mode, int64_t* node_offsets,
                             double* y, double* x, double* z, int64_t node_cap);

/* ------------------------------------------------------------------------------------------ */
/* device API (results stay in HBM; used by bench.py's device-resident leg and the multi-GPU
 * sharding in polishpathplanning_b200/parallel.py).  Query sub-ranges are given in SORTED
 * (cell-major) order so that a rank's share is spatially compact: [first, first+count).
 *  - ranges: 0 <= first <= (finite points), count < 0 = up to the end, first + count <= (finite points); anything
 *    else is PPP_ERR_INVALID, with nothing written or launched.  The ranges of ppp_dev_normals_knn(k) refer to the
 *    order ppp_dev_sorted_order returns after ppp_dev_index(cloud, k, 0), those of ppp_dev_normals_radius(r) to the
 *    order after ppp_dev_index(cloud, 0, r).  A sub-range is always searched on that (primary) grid; the full range
 *    of a cloud that is not a height field runs on one grid per axis pair.  The results are the same either way:
 *    the union of the sub-range calls over [0, finite points) is the full-range call, bit for bit.
 *  - rows written: those of the range's points (by original index).  The rows of the non-finite points get their
 *    defaults (ids -1, d2 inf, NaN normal) only from the call whose range starts at 0.  Through a row map
 *    (ppp_dev_set_normal_row_map) a normal record goes to record map[row] instead, or nowhere for a negative entry;
 *    ids and d2 are not mapped.
 *  - normal records: stride 16 {nx, ny, nz, curvature}; stride 32 pcl::Normal {nx, ny, nz, 0, curvature, 0, 0, 0};
 *    strides 20..28 floats 0..3 = {nx, ny, nz, curvature}; strides above 32 floats 0..4 = {nx, ny, nz, 0, curvature}.
 *    Every other float of a record is left as it was (the host API zero-fills records wider than 32 bytes).
 *  - alignment: normals_dev 16 bytes when the stride is a multiple of 16 (16-byte vector stores; 32-byte ones from a
 *    32-byte aligned buffer at stride 32), 4 otherwise; knn_idx_dev, knn_d2_dev and pts_dev of ppp_dev_cloud_attach
 *    4 bytes.  Misaligned buffers are PPP_ERR_INVALID.                                                           */
int ppp_dev_index(ppp_cloud* cloud, int k_hint, double radius_hint); /* (re)build the grid now */
int ppp_dev_normals_knn(ppp_cloud* cloud, int k, const float viewpoint[3], unsigned flags, int64_t first,
                        int64_t count, float* normals_dev, size_t normal_stride_bytes,
                        int32_t* knn_idx_dev /* n*k rows by ORIGINAL index, nullable */,
                        float* knn_d2_dev /* nullable */);
int ppp_dev_normals_radius(ppp_cloud* cloud, double radius, const float viewpoint[3], unsigned flags,
                           int64_t first, int64_t count, float* normals_dev, size_t normal_stride_bytes);
/* contours for the planes [0,S) given on the HOST (small); results in device buffers owned by
 * the cloud until the next call; pointers returned through the out arguments. Synchronises once
 * to learn the node total.  */
int ppp_dev_slice_contours(ppp_cloud* cloud, const float* plane_x_host, int S, float half_width,
                           int truncate_center, int pairing_mode, const int64_t** node_offsets_dev,
                           const double** y_dev, const double** x_dev, const double** z_dev,
                           int64_t* total_nodes, int64_t* total_band_members);
/* Optional: caller-owned device buffers (cap doubles each) that ppp_dev_slice_contours fills
 * instead of the cloud-owned ones whenever the node total fits (e.g. an NCCL gather buffer). */
int ppp_dev_set_contour_buffers(ppp_cloud* cloud, double* y_dev, double* x_dev, double* z_dev, int64_t cap);
/* Optional: device buffer (cap_entries int64) that also receives the S+1 per-slice node offsets
 * of every ppp_dev_slice_contours call (entry S = node total), e.g. inside a peer buffer.       */
int ppp_dev_set_contour_offsets_buffer(ppp_cloud* cloud, int64_t* offsets_dev, int64_t cap_entries);
/* Stream-ordered 32-bit flags (stream memory operations, no kernel launch).  signal: *flag = value
 * once all earlier work of the context's stream has finished; wait: later work of the stream is
 * held until *flag >= value.  With the flag in a peer buffer the pair is the completion signal for
 * results delivered to another GPU by plain NVLink stores.                                        */
int ppp_dev_signal(ppp_ctx* ctx, uint32_t* flag_dev, uint32_t value);
int ppp_dev_wait(ppp_ctx* ctx, const uint32_t* flag_dev, uint32_t value);
/* Optional: where the normal record of local row i goes: record row_map_dev[i] of the normals buffer
 * (negative: not stored).  With a buffer obtained from ppp_peer_buffer_open the search kernel
 * stores each finished normal straight into another GPU's memory over NVLink, so a slab's owned
 * rows land in rank 0's global array while the kernel runs and no gather collective follows
 * (SURVEY.md §8e "Gather").  NULL restores the identity.  The map must stay valid while in use.  */
int ppp_dev_set_normal_row_map(ppp_cloud* cloud, const int32_t* row_map_dev);
/* Device buffers that the GPUs of OTHER processes on this node can write (CUDA IPC over
 * NVLink/NVSwitch).  alloc: owner side, returns the pointer and a 64-byte handle to ship to the peers
 * (any transport, e.g. a torch.distributed broadcast); the memory is zero-filled.  open/close: peer
 * side; free: owner side.                                                                         */
#define PPP_PEER_HANDLE_BYTES 64
int ppp_peer_buffer_alloc(ppp_ctx* ctx, size_t bytes, void** dev_ptr, unsigned char handle[PPP_PEER_HANDLE_BYTES]);
int ppp_peer_buffer_open(ppp_ctx* ctx, const unsigned char handle[PPP_PEER_HANDLE_BYTES], void** dev_ptr);
int ppp_peer_buffer_close(ppp_ctx* ctx, void* dev_ptr);
int ppp_peer_buffer_free(ppp_ctx* ctx, void* dev_ptr);
/* stream-ordered device -> host copy of a raw device range, then synchronise */
int ppp_dev_download(ppp_ctx* ctx, void* host_dst, const void* dev_src, size_t bytes);
/* original index of the point at sorted position p (device array of one int32 per finite point) of the grid the
 * last ppp_dev_index built or found; NULL before any ppp_dev_index.  Valid while the cloud lives.              */
const int32_t* ppp_dev_sorted_order(ppp_cloud* cloud);

/* ------------------------------------------------------------------------------------------ */
/* multi-GPU exchange (SURVEY.md §8e; csrc/exchange.cu).  The reference is one process on one CPU; what
 * is sharded here is its whole-cloud estimate_normal (src/Path_Generation.cpp:323-333) and its plane
 * sweep (src/Path_Generation.cpp:689-755).  One ppp_exch per rank (= per GPU).  A cloud that starts
 * split by ORIGINAL INDEX (rank r holds records [starts[r], starts[r+1]) of the file) is redistributed
 * into x-slabs of equal point count plus a halo by kernels that store straight into the destination
 * GPU's memory over NVLink (no NCCL, no host staging); the received slab keeps ascending global index
 * order, so all tie-breaks are those of the single-GPU run.  Results travel the same way: every normal
 * record goes from the search kernel to its HOME rank (the rank holding that original index range),
 * contour nodes go to rank 0's region.                                                            */
typedef struct ppp_exch ppp_exch;
#define PPP_EXCH_MAX_RANKS 16
/* starts: world + 1 ascending offsets from 0 (starts[world] = total points).  cap_recv: capacity of the
 * receive buffer in points (own slab + halo copies).  S_cap / node_cap: capacity of one rank's contour
 * region (planes / nodes).  normal_stride_bytes: 16 {nx,ny,nz,curvature} or 32 (pcl::Normal).      */
int ppp_exch_create(ppp_ctx* ctx, int rank, int world, const int64_t* starts, int64_t cap_recv, int S_cap, int64_t node_cap,
                    size_t normal_stride_bytes, ppp_exch** out);
/* Tear-down between processes: every rank disconnects (unmaps the peers' arenas), the ranks meet at a
 * barrier of their own, then every rank destroys (an arena is not freed while a peer has it mapped).  */
int ppp_exch_disconnect(ppp_exch* ex);
int ppp_exch_destroy(ppp_exch* ex);
/* ranks in other processes: ship every rank's 64-byte handle to all (any transport), then connect.   */
int ppp_exch_ipc_handle(ppp_exch* ex, unsigned char handle[PPP_PEER_HANDLE_BYTES]);
int ppp_exch_connect_ipc(ppp_exch* ex, const unsigned char* handles /* world x 64 bytes */);
/* ranks in this process (one process driving several contexts / GPUs): all[r] = rank r's exchange.   */
int ppp_exch_connect_local(ppp_exch* ex, ppp_exch* const* all);
/* Enqueue phase 0..3 of the exchange of this rank's chunk (device records; n = starts[rank+1] -
 * starts[rank]).  One rank per process: call 0,1,2,3 back to back.  Several ranks per process: issue
 * phase p for every rank before phase p + 1.  halo: width of the copies on either side of a slab.   */
int ppp_exch_phase(ppp_exch* ex, int phase, const void* chunk_dev, int64_t n, size_t stride_bytes, double halo);
/* Wait for every rank's records, then (synchronises) report the slab: n_local points of which n_owned
 * are owned, cuts[world + 1] (rank r owns cuts[r] <= x < cuts[r+1]; -inf / +inf at the ends), global
 * finite x-range.  PPP_ERR_CAPACITY: cap_recv too small; PPP_ERR_CUDA: a peer did not answer in time. */
int ppp_exch_finish(ppp_exch* ex, int64_t* n_local, int64_t* n_owned, double* cuts, double x_range[2]);
const void* ppp_exch_slab(ppp_exch* ex);          /* device: n_local records {x, y, z, bits(global index or ~index)} */
const int32_t* ppp_exch_row_map(ppp_exch* ex);    /* device: local row -> global index, -1 for halo copies */
void* ppp_exch_home_normals(ppp_exch* ex);        /* device: normal records of the own index range */
/* The slab as a cloud whose normal estimators deliver each owned row's record to its home rank; with
 * to_rank0 != 0 ppp_dev_slice_contours also writes its nodes + per-slice offsets to rank 0's region.   */
int ppp_exch_attach(ppp_exch* ex, int to_rank0, ppp_cloud** out);
/* ppp_exch_finish followed by ppp_exch_attach, with one host synchronisation instead of two (the slab is ingested
 * straight behind the exchange kernels; its size reaches the host together with the bounding box). */
int ppp_exch_finish_attach(ppp_exch* ex, int to_rank0, int64_t* n_local, int64_t* n_owned, double* cuts, double x_range[2],
                           ppp_cloud** out);
int ppp_exch_nodes_region(ppp_exch* ex, int r, const int64_t** offsets_dev, const double** y_dev, const double** x_dev,
                          const double** z_dev);   /* rank 0: device pointers of rank r's contour region */
/* what: PPP_EXCH_NORMALS / PPP_EXCH_CONTOURS.  signal: the results of that kind this rank has enqueued so
 * far have been delivered; wait: later work of the stream sees every rank's results of that kind (home
 * normals complete / rank 0's regions complete).                                                       */
#define PPP_EXCH_NORMALS 0
#define PPP_EXCH_CONTOURS 1
int ppp_exch_results_signal(ppp_exch* ex, int what);
int ppp_exch_results_wait(ppp_exch* ex, int what);
int ppp_exch_check(ppp_exch* ex);                 /* PPP_OK unless a wait has timed out (synchronises) */
/* page-lock an existing host range (e.g. a shared-memory mapping opened by every rank's process);
 * *dev_ptr (nullable) = the address of its first byte as kernels see it.                             */
int ppp_host_register(void* p, size_t bytes, void** dev_ptr);
int ppp_host_unregister(void* p);
/* stream-ordered copies between page-locked host memory and device buffers (no synchronisation)      */
int ppp_dev_upload(ppp_ctx* ctx, void* dev_dst, const void* host_src, size_t bytes);
int ppp_dev_download_async(ppp_ctx* ctx, void* host_dst, const void* dev_src, size_t bytes);

#ifdef __cplusplus
}
#endif
#endif /* PPP_GPU_H */
