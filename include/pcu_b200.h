/*
 * pcu_b200.h -- C ABI of the B200-native nearest-neighbour path (libpcu_b200.so).
 *
 * This is the drop-in boundary for the ONE hot path of fwilliams/point-cloud-utils that this
 * repository replaces: exact L2 k-nearest-neighbour search between two 3-D point clouds and the
 * Chamfer / Hausdorff scalars built on it.  Each entry point names the reference interface it
 * stands in for (paths relative to /root/reference):
 *
 *   pcu_b200_knn_*                   shortest_distances_nanoflann<>      src/point_cloud_distance.cpp:21-99
 *                                    as called by k_nearest_neighbors    src/point_cloud_distance.cpp:123-164
 *   pcu_b200_nn_stats_*              the k = 1 sweep + dists.maxCoeff    src/point_cloud_distance.cpp:219-225
 *                                    (one_sided_hausdorff_distance       src/point_cloud_distance.cpp:186-234)
 *                                    and norm(...).mean() of chamfer     point_cloud_utils/__init__.py:112-113
 *   pcu_b200_chamfer_*               chamfer_distance, p_norm = 2        point_cloud_utils/__init__.py:84-120
 *   pcu_b200_batched_chamfer_*       a Python loop of chamfer_distance over pairs (the docstring's
 *                                    "[m, n, d] minibatch", __init__.py:89-90, which the 2-D-only
 *                                    binding never implemented)
 *
 * Conventions
 *   - Plain C: raw pointers, sizes, an opaque workspace handle and a CUDA stream passed as void*.
 *     No C++ / torch / numpy types cross this boundary and no exception does either.
 *   - Every function returns a pcu_b200_status; the message of the last failure on the calling
 *     thread is available from pcu_b200_last_error().
 *   - Point clouds are dense row-major (n, 3) arrays of float (…_f32) or double (…_f64).
 *   - The caller owns every input and output buffer.  The library never allocates user-visible
 *     memory; scratch lives in the workspace (grown on demand, reused across calls).  One
 *     workspace serves one stream at a time.
 *   - "device" entry points take DEVICE pointers, enqueue work on `stream` and return without
 *     synchronising; results are valid once the stream reaches that point.  "host" entry points
 *     take HOST pointers (pinned or pageable), copy them to device staging owned by the workspace
 *     on the workspace's own streams -- the copy of the second cloud overlaps the first kernels --
 *     and return after the results have landed in the caller's buffers.  Page-locked inputs are
 *     DMA'd as they are; pageable inputs of 4 MB and more go through a 32 MB page-locked ring of
 *     the workspace, filled by eight copy threads in 512 KB chunks and drained in transfers of up
 *     to 4 MB (pcu_b200_options::host_staging; the threads start with the first such copy).
 *   - Scratch grows with stream-ordered allocation (cudaMallocAsync): no entry point synchronises
 *     the device.  A workspace serves one stream at a time; a call on another stream than the
 *     previous one is ordered after it on the device.
 *   - Results follow the reference bit for bit: squared distance is ((qx-px)^2+(qy-py)^2)+(qz-pz)^2,
 *     every operation rounded in the input precision, no FMA (nanoflann.hpp:496-507); indices are
 *     int64 (ptrdiff_t in the reference); rows are ascending by distance; queries whose answer
 *     depends on how equal distances are ordered are re-answered on the GPU by a replica of the
 *     reference's kd-tree traversal (visit order decides, nanoflann.hpp:194-227) built with the
 *     caller's max_points_per_leaf; fewer than k neighbours (k > m) pads with -1 / -1.0
 *     (src/point_cloud_distance.cpp:90-93).
 */
#ifndef PCU_B200_H
#define PCU_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCU_B200_ABI_VERSION 3

typedef enum pcu_b200_status {
    PCU_B200_OK = 0,
    PCU_B200_INVALID_ARGUMENT = 1, /* maps to ValueError in the Python layer (pybind11::value_error in the reference) */
    PCU_B200_CUDA_ERROR = 2,       /* maps to RuntimeError */
    PCU_B200_OUT_OF_MEMORY = 3,    /* maps to MemoryError */
    PCU_B200_NO_DEVICE = 4,        /* no usable sm_100 device: the product has no CPU fallback */
    PCU_B200_INTERNAL = 5
} pcu_b200_status;

typedef struct pcu_b200_workspace pcu_b200_workspace;

/* Per-direction result of the fused k = 1 sweep (no per-point distance buffer is written). */
typedef struct pcu_b200_nn_stats {
    double sum_dist;      /* sum over queries of sqrt(d2_min), accumulated in fp64                */
    double sum_sq_dist;   /* sum over queries of d2_min, accumulated in fp64                      */
    double max_sq_dist;   /* largest d2_min (exact: the input-precision value widened to double)  */
    int64_t argmax_query; /* first (lowest-index) query attaining it (Eigen maxCoeff, :221-223)   */
    int64_t argmax_data;  /* its nearest neighbour in the dataset (:225)                          */
    int64_t n_queries;    /* n                                                                    */
    int64_t n_tied;       /* -1: the fused sweeps track distances only (ties only matter to witness_tied) */
    int64_t n_far;        /* queries that needed the ring-expansion slow path (diagnostic)        */
    int64_t witness_tied; /* 1: argmax_query had several equally near neighbours, so argmax_data  */
                          /* is the lowest such index, not necessarily the reference's pick; the  */
                          /* host entry points resolve this themselves, device callers use        */
                          /* pcu_b200_resolve_witness_* (value, sums and argmax_query are final)   */
    double pair_value;    /* bidirectional calls (pcu_b200_chamfer_*): the pair's Chamfer value in fp64,  */
                          /* sum_dist[x->y] / n + sum_dist[y->x] / m, written to BOTH records by the sweep */
                          /* that finishes second (what a multi-GPU caller sums across ranks);            */
                          /* one-directional calls: sum_dist / n_queries                                  */
} pcu_b200_nn_stats;

/* Tunables; zero-initialise and override what you need.  0 always means "library default". */
typedef struct pcu_b200_options {
    int max_points_per_leaf; /* reference kwarg; only influences how exact-distance ties are ordered (default 10) */
    float cell_occupancy;    /* target dataset points per grid cell (0 = default: 1.5 for k = 1; 3 / 4 / 7 / 12  */
                             /* at k = 4 / 8 / 16 / 32, interpolated in between -- measured, DESIGN.md section 4) */
    int disable_tie_replay;  /* diagnostic only.  1: keep the (distance, lowest index) order for tied queries;        */
                             /* 2: replay on full reference trees only (no pruned build); 3: pruned build with    */
                             /* zero slack (every walk hits a stub, which exercises the full-rebuild path)        */
    int binning;             /* 0: automatic; 1: always the multi-launch grid build; 2: the one-CTA-per-cloud     */
                             /* build whenever a cloud's cell counters fit in shared memory (diagnostic only)    */
    int host_staging;        /* host entry points, inputs of >= 4 MB: 0 pageable memory goes through the          */
                             /* workspace's pinned ring filled by copy threads, pinned memory is DMA'd as it is;  */
                             /* 1 always the ring; 2 never (plain cudaMemcpyAsync: the driver stages)             */
} pcu_b200_options;

/* ---- library / error plumbing ------------------------------------------------------------ */
int pcu_b200_abi_version(void);
const char* pcu_b200_last_error(void);
/* Number of CUDA devices this build can run on (compute capability 10.x); 0 if none. */
int pcu_b200_device_count(void);
/* The device a call that names none runs on.  The reference's interface (src/point_cloud_distance.cpp:123-131,
 * :186-193) has no device argument, so the replacement has to pick one: the environment variable
 * PCU_B200_DEVICE if set; else the CUDA runtime's current device of the calling thread when that is not 0
 * (torch.cuda.set_device / `with torch.cuda.device(i)`); else LOCAL_RANK when a launcher (torchrun) set it
 * and that many devices are visible; else 0. */
int pcu_b200_current_device(void);
/* Kernels launched by this library on the calling process since load (bench.py's gpu_launches). */
int64_t pcu_b200_launch_count(void);

/* Page-locked host memory (cudaHostAlloc / cudaFreeHost), for callers that want their big result buffers to
 * be copy targets the DMA engines can write directly: the numpy-facing binding backs k-NN results of 1 MiB and
 * more with such blocks (recycled through a small pool), because a device-to-host copy into freshly allocated
 * pageable memory runs at ~3 GB/s -- the page faults, not PCIe -- against ~50 GB/s into pinned memory.
 * The block is placed on the NUMA node of the calling thread's current GPU (the PCI device's numa_node in sysfs):
 * on two-socket hosts a page-locked buffer on the other node is copied at half the rate or less. */
int pcu_b200_host_alloc(void** out_ptr, int64_t bytes);
int pcu_b200_host_free(void* ptr);

/* ---- workspace ---------------------------------------------------------------------------- */
int pcu_b200_workspace_create(int device, pcu_b200_workspace** out_ws);
int pcu_b200_workspace_destroy(pcu_b200_workspace* ws);
/* The device the workspace was created on (-1 for NULL).  Every entry point runs there and leaves the
 * calling thread's current device as it found it. */
int pcu_b200_workspace_device(const pcu_b200_workspace* ws);
/* Bytes of device scratch currently held. */
int64_t pcu_b200_workspace_bytes(const pcu_b200_workspace* ws);
int pcu_b200_workspace_set_options(pcu_b200_workspace* ws, const pcu_b200_options* opts);
/* Diagnostic: how much finer than the default the two clouds' grids of the NEXT call with the last call's
 * shapes will be (1 = default cells per point).  The library learns this from the fill statistics each
 * call leaves behind: surfaces and other thin point sets get finer grids from the second call on.  It
 * changes speed only, never results. */
int pcu_b200_workspace_grid_refinement(const pcu_b200_workspace* ws, float out_mult[2]);
/* Per-stage device timing (diagnostic; bench.py's roofline pass).  When enabled, every device entry
 * point records CUDA events on the launching stream between its stages; after that stream has been
 * synchronised, last_profile() returns the milliseconds of the LAST call's 8 stages (descriptors,
 * bbox+grid, histogram, scan, scatter, search, search_far, finalize) and their count (0 if none); after a
 * host entry point and with capacity >= 10, two more: the host-to-device copies in front of the first stage
 * and the device-to-host copies behind the last ("h2d", "d2h"). */
int pcu_b200_workspace_set_profiling(pcu_b200_workspace* ws, int enabled);
int pcu_b200_workspace_last_profile(pcu_b200_workspace* ws, float* out_ms, int capacity);
const char* pcu_b200_profile_stage_name(int stage);

/* ---- k nearest neighbours, DEVICE pointers -------------------------------------------------
 * out_dist : (n, k) row-major, input precision; sqrt(d2) unless squared != 0
 * out_idx  : (n, k) row-major int64 indices into dataset
 * out_n_tied (may be NULL): device int64 that receives the number of queries that went through
 *            the tie replay.
 * The call never synchronises: the kd-tree replay is one cooperative launch gated, on the device, on
 * the number of flagged queries (it returns at once when that number is zero).
 * Replaces shortest_distances_nanoflann (src/point_cloud_distance.cpp:21-99).                    */
int pcu_b200_knn_f32(pcu_b200_workspace* ws, const float* query, int64_t n, const float* dataset, int64_t m, int k,
                     int squared, float* out_dist, int64_t* out_idx, int64_t* out_n_tied, void* stream);
int pcu_b200_knn_f64(pcu_b200_workspace* ws, const double* query, int64_t n, const double* dataset, int64_t m, int k,
                     int squared, double* out_dist, int64_t* out_idx, int64_t* out_n_tied, void* stream);

/* ---- fused k = 1 sweep + reductions, DEVICE pointers ---------------------------------------
 * out_stats : device pointer to ONE pcu_b200_nn_stats (query -> dataset direction).
 * Replaces the k = 1 sweep, dists.maxCoeff and corrs(i, 0) of one_sided_hausdorff_distance
 * (src/point_cloud_distance.cpp:219-225).                                                        */
int pcu_b200_nn_stats_f32(pcu_b200_workspace* ws, const float* query, int64_t n, const float* dataset, int64_t m,
                          pcu_b200_nn_stats* out_stats, void* stream);
int pcu_b200_nn_stats_f64(pcu_b200_workspace* ws, const double* query, int64_t n, const double* dataset, int64_t m,
                          pcu_b200_nn_stats* out_stats, void* stream);

/* Re-answers stats->argmax_query with the reference's tie order (kd-tree replay built with
 * max_points_per_leaf) and stores the result in stats->argmax_data; clears witness_tied.
 * `stats` is a DEVICE pointer to one record produced by the calls above for (query, dataset).
 * Synchronises the stream once (the workspace scratch is re-carved for the replay).              */
int pcu_b200_resolve_witness_f32(pcu_b200_workspace* ws, const float* query, int64_t n, const float* dataset,
                                 int64_t m, pcu_b200_nn_stats* stats, void* stream);
int pcu_b200_resolve_witness_f64(pcu_b200_workspace* ws, const double* query, int64_t n, const double* dataset,
                                 int64_t m, pcu_b200_nn_stats* stats, void* stream);

/* ---- fused bidirectional Chamfer (+ Hausdorff), DEVICE pointers ----------------------------
 * out_stats : device pointer to TWO pcu_b200_nn_stats: [0] = x -> y, [1] = y -> x.
 * out_value : device pointer to one scalar of the input precision:
 *             chamfer = stats[0].sum_dist / n + stats[1].sum_dist / m   (no 1/2, not squared;
 *             point_cloud_utils/__init__.py:112-115).  May be NULL.
 * Both clouds are binned once and swept in one launch; no distance buffer is materialised.       */
int pcu_b200_chamfer_f32(pcu_b200_workspace* ws, const float* x, int64_t n, const float* y, int64_t m,
                         pcu_b200_nn_stats* out_stats, float* out_value, void* stream);
int pcu_b200_chamfer_f64(pcu_b200_workspace* ws, const double* x, int64_t n, const double* y, int64_t m,
                         pcu_b200_nn_stats* out_stats, double* out_value, void* stream);

/* ---- prepared clouds: bin a fixed cloud ONCE, use it as one side of many calls ---------------
 * The reference rebuilds its kd-tree on every call -- three times per direction (src/point_cloud_distance.cpp:41-42,
 * nanoflann.hpp:1357, 2288) -- even when one cloud never changes (a loss against a fixed target evaluated every
 * iteration).  pcu_b200_cloud_prepare_* copies the points into a private device block and bins them there; the
 * *_prepared_* calls take the handle as the SECOND cloud (y / target / dataset), bin only the first cloud and run
 * the same fused sweeps: results are those of the unprepared calls bit for bit.  Host variants copy only the first
 * cloud over PCIe.  A handle may serve calls on several workspaces / streams of its device at once (it is
 * read-only after preparation, apart from an occupancy pyramid every user would write identically).
 * pcu_b200_cloud_destroy synchronises the device. */
typedef struct pcu_b200_cloud pcu_b200_cloud;
int pcu_b200_cloud_prepare_f32(pcu_b200_workspace* ws, const float* points, int64_t n, pcu_b200_cloud** out_cloud, void* stream);
int pcu_b200_cloud_prepare_f64(pcu_b200_workspace* ws, const double* points, int64_t n, pcu_b200_cloud** out_cloud, void* stream);
int pcu_b200_cloud_prepare_host_f32(pcu_b200_workspace* ws, const float* points, int64_t n, pcu_b200_cloud** out_cloud);
int pcu_b200_cloud_prepare_host_f64(pcu_b200_workspace* ws, const double* points, int64_t n, pcu_b200_cloud** out_cloud);
/* The same for k-NN calls: the cell size is chosen for searches with this k, and the reference's kd-tree replica (leaf
 * size max_points_per_leaf, 0 = 10) is built once into the handle, so that pcu_b200_knn_prepared_* neither bins the
 * dataset nor builds the tree -- it only replays its tied rows on it (the reference builds its tree in every call,
 * src/point_cloud_distance.cpp:41-42).  A call whose options name another leaf size builds its own tree as usual.
 * The handle's tree counters and pyramid are shared state: one k-NN call at a time per handle. */
int pcu_b200_cloud_prepare_knn_f32(pcu_b200_workspace* ws, const float* points, int64_t n, int k, int max_points_per_leaf,
                                   pcu_b200_cloud** out_cloud, void* stream);
int pcu_b200_cloud_prepare_knn_f64(pcu_b200_workspace* ws, const double* points, int64_t n, int k, int max_points_per_leaf,
                                   pcu_b200_cloud** out_cloud, void* stream);
int pcu_b200_cloud_prepare_knn_host_f32(pcu_b200_workspace* ws, const float* points, int64_t n, int k, int max_points_per_leaf,
                                        pcu_b200_cloud** out_cloud);
int pcu_b200_cloud_prepare_knn_host_f64(pcu_b200_workspace* ws, const double* points, int64_t n, int k, int max_points_per_leaf,
                                        pcu_b200_cloud** out_cloud);
/* k nearest neighbours of `query` in a prepared cloud: outputs as pcu_b200_knn_* (same results, bit for bit). */
int pcu_b200_knn_prepared_f32(pcu_b200_workspace* ws, const float* query, int64_t n, pcu_b200_cloud* dataset, int k, int squared,
                              float* out_dist, int64_t* out_idx, int64_t* out_n_tied, void* stream);
int pcu_b200_knn_prepared_f64(pcu_b200_workspace* ws, const double* query, int64_t n, pcu_b200_cloud* dataset, int k, int squared,
                              double* out_dist, int64_t* out_idx, int64_t* out_n_tied, void* stream);
int pcu_b200_knn_prepared_host_f32(pcu_b200_workspace* ws, const float* query, int64_t n, pcu_b200_cloud* dataset, int k, int squared,
                                   float* out_dist, int64_t* out_idx, int64_t* out_n_tied);
int pcu_b200_knn_prepared_host_f64(pcu_b200_workspace* ws, const double* query, int64_t n, pcu_b200_cloud* dataset, int k, int squared,
                                   double* out_dist, int64_t* out_idx, int64_t* out_n_tied);
int pcu_b200_cloud_destroy(pcu_b200_cloud* cloud);
int64_t pcu_b200_cloud_size(const pcu_b200_cloud* cloud);
/* DEVICE pointer to the handle's private (n, 3) copy of the points (what pcu_b200_resolve_witness_* wants as the
 * prepared side's array). */
const void* pcu_b200_cloud_points(const pcu_b200_cloud* cloud);
/* out_stats: TWO records ([0] = x -> y, [1] = y -> x) as for pcu_b200_chamfer_*; out_value may be NULL */
int pcu_b200_chamfer_prepared_f32(pcu_b200_workspace* ws, const float* x, int64_t n, const pcu_b200_cloud* y,
                                  pcu_b200_nn_stats* out_stats, float* out_value, void* stream);
int pcu_b200_chamfer_prepared_f64(pcu_b200_workspace* ws, const double* x, int64_t n, const pcu_b200_cloud* y,
                                  pcu_b200_nn_stats* out_stats, double* out_value, void* stream);
/* out_stats: ONE record (query -> dataset) as for pcu_b200_nn_stats_* */
int pcu_b200_nn_stats_prepared_f32(pcu_b200_workspace* ws, const float* query, int64_t n, const pcu_b200_cloud* dataset,
                                   pcu_b200_nn_stats* out_stats, void* stream);
int pcu_b200_nn_stats_prepared_f64(pcu_b200_workspace* ws, const double* query, int64_t n, const pcu_b200_cloud* dataset,
                                   pcu_b200_nn_stats* out_stats, void* stream);
int pcu_b200_chamfer_prepared_host_f32(pcu_b200_workspace* ws, const float* x, int64_t n, const pcu_b200_cloud* y,
                                       pcu_b200_nn_stats* out_stats, float* out_value);
int pcu_b200_chamfer_prepared_host_f64(pcu_b200_workspace* ws, const double* x, int64_t n, const pcu_b200_cloud* y,
                                       pcu_b200_nn_stats* out_stats, double* out_value);
int pcu_b200_nn_stats_prepared_host_f32(pcu_b200_workspace* ws, const float* query, int64_t n, const pcu_b200_cloud* dataset,
                                        pcu_b200_nn_stats* out_stats);
int pcu_b200_nn_stats_prepared_host_f64(pcu_b200_workspace* ws, const double* query, int64_t n, const pcu_b200_cloud* dataset,
                                        pcu_b200_nn_stats* out_stats);

/* ---- batched Chamfer over independent pairs, DEVICE pointers -------------------------------
 * x : (B, n, 3), y : (B, m, 3) dense; out_per_pair : (B) scalars of the input precision;
 * out_sum (may be NULL): device double = sum of the B per-pair values (the quantity a multi-GPU
 * caller all-reduces).                                                                            */
int pcu_b200_batched_chamfer_f32(pcu_b200_workspace* ws, const float* x, const float* y, int64_t batch, int64_t n,
                                 int64_t m, float* out_per_pair, double* out_sum, void* stream);

/* ---- point-cloud normals from k nearest neighbours (SURVEY.md 8f, N1) ----------------------
 * Replaces estimate_point_cloud_normals_knn_internal (src/point_cloud_normals.cpp:375-411, estimator :115-173):
 * for every point its k nearest points of the same cloud (itself included), the unit normal of the plane
 * fitted to them, and -- when view_dirs (n, 3) is not NULL -- orientation towards the view direction and
 * dropping of points whose normal makes an angle above drop_angle_threshold (radians) with it.
 * out_idx (capacity n) / out_normals (capacity n x 3): the kept points in ascending row order; out_count: how
 * many.  The neighbour sets are the reference's bit for bit (same exact k-NN, same tie order); the plane fit is
 * the smallest eigenvector of the fp64 scatter matrix, equal to the reference's JacobiSVD vector up to rounding
 * and, without view directions, up to sign.  DEVICE pointers; out_count is a device int64. */
int pcu_b200_normals_knn_f32(pcu_b200_workspace* ws, const float* points, int64_t n, const float* view_dirs, int k,
                             double drop_angle_threshold, int64_t* out_idx, float* out_normals, int64_t* out_count, void* stream);
int pcu_b200_normals_knn_f64(pcu_b200_workspace* ws, const double* points, int64_t n, const double* view_dirs, int k,
                             double drop_angle_threshold, int64_t* out_idx, double* out_normals, int64_t* out_count, void* stream);

/* ---- duplicate removal (SURVEY.md 8f, N2) ---------------------------------------------------
 * Replaces deduplicate_point_cloud / deduplicate_mesh_vertices (src/remove_duplicates.cpp:108-176, helpers :11-79;
 * libigl's round + unique_rows underneath).  epsilon > 0: rows are compared after round(p / epsilon) (division in the
 * cloud's precision, halves away from zero); otherwise as they are.  Unique rows come in ascending lexicographic
 * order of the compared values.
 *   out_points (capacity n x 3): points[out_svi];  out_svi (capacity n): for every unique row the FIRST input row of its
 *   cluster (libigl returns an unspecified member: its row sort is not stable);  out_svj (n): unique row of every input
 *   row;  faces (may be NULL): (n_faces, face_cols) int32 or int64 vertex indices -> out_faces (capacity n_faces x
 *   face_cols) holds the re-indexed faces whose corners stay distinct, in their original order.
 *   out_counts: 3 device int64 = { unique points, surviving faces, faces with a corner outside [0, n) (dropped) }.
 * DEVICE pointers. */
int pcu_b200_deduplicate_f32(pcu_b200_workspace* ws, const float* points, int64_t n, double epsilon, const void* faces, int64_t n_faces,
                             int face_cols, int faces_are_i64, float* out_points, int32_t* out_svi, int32_t* out_svj, void* out_faces,
                             int64_t* out_counts, void* stream);
int pcu_b200_deduplicate_f64(pcu_b200_workspace* ws, const double* points, int64_t n, double epsilon, const void* faces, int64_t n_faces,
                             int face_cols, int faces_are_i64, double* out_points, int32_t* out_svi, int32_t* out_svj, void* out_faces,
                             int64_t* out_counts, void* stream);

/* ---- point-cloud normals from all points in a ball (SURVEY.md 8f, N1) -----------------------
 * Replaces estimate_point_cloud_normals_ball_internal (src/point_cloud_normals.cpp:303-370, estimator :48-113).
 * The neighbourhood of a point is what the reference's call nanoflann radiusSearch(query, ball_radius) returns:
 * every point (itself included) whose SQUARED distance, rounded like the reference's metric, is below
 * (scalar)radius -- nanoflann's radius is in squared units and the reference passes ball_radius as it is -- while
 * the weight function sees the true distance: 1 ("constant") or (1 - d/r)^4 (4 d/r + 1) ("rbf").  Points with
 * fewer than min_pts_per_ball neighbours are dropped; with max_pts_per_ball > 0 a uniformly random subset of that
 * size is fitted (the reference shuffles with rand(); here selection sampling from a hash of seed, row, position:
 * same distribution, reproducible for a given seed, not the same subset).  Outputs as for the k-NN variant. */
typedef struct pcu_b200_ball_options {
    double radius;                 /* > 0 */
    double drop_angle_threshold;   /* radians; only used with view directions */
    int32_t min_pts_per_ball;      /* >= 3 */
    int32_t max_pts_per_ball;      /* <= 0: no limit, else >= 3 */
    int32_t weight_function;       /* 0 "constant", 1 "rbf" */
    uint32_t seed;                 /* subset selection when max_pts_per_ball > 0 */
} pcu_b200_ball_options;
int pcu_b200_normals_ball_f32(pcu_b200_workspace* ws, const float* points, int64_t n, const float* view_dirs,
                              const pcu_b200_ball_options* options, int64_t* out_idx, float* out_normals, int64_t* out_count, void* stream);
int pcu_b200_normals_ball_f64(pcu_b200_workspace* ws, const double* points, int64_t n, const double* view_dirs,
                              const pcu_b200_ball_options* options, int64_t* out_idx, double* out_normals, int64_t* out_count, void* stream);

/* ---- voxel-grid down-sampling (SURVEY.md 8f, N2) --------------------------------------------
 * Replaces downsample_point_cloud_voxel_grid_internal (src/sample_point_cloud.cpp:336-367, :163-244): every point
 * goes to voxel int(floor((p - min_bound) / voxel_size)) per axis, computed in the cloud's precision exactly like the
 * reference; every voxel with at least min_points_per_voxel points yields one output row, the mean of its points and
 * of its rows of `attrib` ((n, attrib_cols) float or double, attrib_cols may be 0).  Exact: voxel assignment, the set
 * of output voxels, their point counts (out_counts, may be NULL).  Different by construction and documented: the
 * reference's row order is the iteration order of a std::unordered_map -- here rows follow the first point of each
 * voxel in the input; the reference sums in the cloud's precision point by point -- here in fp64, so means agree to
 * the rounding of its float sums.  Capacity of the outputs: n rows; out_rows: device int64.  DEVICE pointers. */
int pcu_b200_voxel_downsample_f32(pcu_b200_workspace* ws, const float* points, int64_t n, const void* attrib, int attrib_cols,
                                  int attrib_is_f64, const double voxel_size[3], const double min_bound[3], const double max_bound[3],
                                  int min_points_per_voxel, float* out_points, void* out_attrib, int32_t* out_counts, int64_t* out_rows,
                                  void* stream);
int pcu_b200_voxel_downsample_f64(pcu_b200_workspace* ws, const double* points, int64_t n, const void* attrib, int attrib_cols,
                                  int attrib_is_f64, const double voxel_size[3], const double min_bound[3], const double max_bound[3],
                                  int min_points_per_voxel, double* out_points, void* out_attrib, int32_t* out_counts, int64_t* out_rows,
                                  void* stream);

/* ---- Poisson-disk down-sampling ------------------------------------------------------------------
 * Replaces downsample_point_cloud_poisson_disk (src/sample_point_cloud.cpp:240-333; exported at
 * point_cloud_utils/__init__.py:4-5).  The reference's sampler (libigl's blue-noise loop, seeded through rand()) is not
 * in its tree; the result here is defined instead as the greedy maximal independent set in ascending key order:
 *   key(i) = (h(i) << 32) | i,  h(i) = mix32(seed ^ mix32(i * 0x9e3779b9 + 0x85ebca6b))  (mix32: normals.cuh);
 *   rows i and j conflict iff d2(i, j) < r2, with the reference-rounded d2 of this library and r2 = (T)r * (T)r in the
 *   cloud's precision T; a row is a sample iff it conflicts with no sample of smaller key.
 * Unique (independent of scheduling), separated and maximal.  out_idx: int32 rows of the samples, ASCENDING (the
 * reference returns its placement order); capacity n.  out_count: device int64.
 * target_num_samples > 0: `radius` is ignored and the reference's radius search (:278-326: arange(n) when the target is
 * >= n, halving from |bbox| / 50, doubling, at most 20 bisection steps with sample_num_tolerance) runs operation for
 * operation in T; the call then synchronises `stream` once per radius trial (and once for the bounding box).  Without
 * it nothing synchronises.  Argument errors (:265-270): target_num_samples <= 0 with radius <= 0, sample_num_tolerance
 * outside (0, 1].  ABI version 3 is unchanged: the entries are an addition, detected by symbol.  DEVICE pointers. */
int pcu_b200_poisson_disk_downsample_f32(pcu_b200_workspace* ws, const float* points, int64_t n, double radius, int target_num_samples,
                                         uint32_t seed, float sample_num_tolerance, int32_t* out_idx, int64_t* out_count, void* stream);
int pcu_b200_poisson_disk_downsample_f64(pcu_b200_workspace* ws, const double* points, int64_t n, double radius, int target_num_samples,
                                         uint32_t seed, float sample_num_tolerance, int32_t* out_idx, int64_t* out_count, void* stream);
/* The last Poisson-disk call on this workspace (synchronises the device): out[0] radius trials, out[1] rounds of the
 * parallel MIS summed over its trials. */
int pcu_b200_debug_poisson_stats(pcu_b200_workspace* ws, int64_t out[2]);

/* ---- dense pairwise distances and Sinkhorn (SURVEY.md 8f, N4) -------------------------------
 * Replace the numpy code of point_cloud_utils/_sinkhorn.py: pairwise_distances (:4-34), sinkhorn (:37-126) and the
 * cost (P * M).sum() of earth_movers_distance (:129-156).  DEVICE pointers, row-major dense arrays:
 *   pairwise: a (nb, n, d), b (nb, m, d) -> out (nb, n, m), out[k, i, j] = || a[k, i] - b[k, j] ||_p;
 *             norm_kind 0: p = 2 (np.linalg.norm default), 1: p = 1, 2: inf, 3: -inf, 4: p = 0 (count of non-zeros),
 *             5: general p (the double argument)
 *   sinkhorn: weights a (nb, n), b (nb, m), costs M (nb, n, m), eps, max_iters, stop_thresh -> plan out_P (nb, n, m);
 *             out_cost (nb) fp64 = sum_ij P * M per batch or NULL; out_iters: device int32 or NULL.  The log-domain
 *             iteration of the reference, its convergence test evaluated on the device (no host synchronisation).
 * Floating point: element-wise expressions in the arrays' precision and the reference's order, the two reductions in
 * fp64 -- agreement with numpy to rounding (tests/test_sinkhorn.py states the tolerances). */
int pcu_b200_pairwise_distances_f32(pcu_b200_workspace* ws, const float* a, const float* b, int64_t nb, int64_t n, int64_t m, int d,
                                    int norm_kind, double p, float* out, void* stream);
int pcu_b200_pairwise_distances_f64(pcu_b200_workspace* ws, const double* a, const double* b, int64_t nb, int64_t n, int64_t m, int d,
                                    int norm_kind, double p, double* out, void* stream);
int pcu_b200_sinkhorn_f32(pcu_b200_workspace* ws, const float* a, const float* b, const float* M, int64_t nb, int64_t n, int64_t m,
                          double eps, int max_iters, double stop_thresh, float* out_P, double* out_cost, int32_t* out_iters, void* stream);
int pcu_b200_sinkhorn_f64(pcu_b200_workspace* ws, const double* a, const double* b, const double* M, int64_t nb, int64_t n, int64_t m,
                          double eps, int max_iters, double stop_thresh, double* out_P, double* out_cost, int32_t* out_iters, void* stream);

/* ---- 64-bit 3-D Morton codes (SURVEY.md 8f, N3) --------------------------------------------
 * Replace MortonCode64 (src/common/morton_code.cpp:43-163) and the bindings morton_encode / morton_decode /
 * morton_add / morton_subtract / morton_knn (src/morton.cpp:185-239, :253-310, :26-103, :106-183, :324-414).
 * Integer work: bit-identical.  pts: (n, 3) int32 (or int64, truncated to int32 as the reference does);
 * coordinates in [-2^20, 2^20).  morton_knn: `codes` ascending; out_idx (m, k) = the k consecutive positions
 * around the lower bound of each query code (k <= n: the binding clamps like morton.cpp:351); sort_dist != 0
 * orders each row by squared distance to the query point -- an order the reference leaves undefined (its
 * comparator reads uninitialised variables, :381-398); the set of positions is the reference's.  DEVICE pointers. */
int pcu_b200_morton_encode_i32(pcu_b200_workspace* ws, const int32_t* pts, int64_t n, uint64_t* out_codes, void* stream);
int pcu_b200_morton_encode_i64(pcu_b200_workspace* ws, const int64_t* pts, int64_t n, uint64_t* out_codes, void* stream);
int pcu_b200_morton_decode(pcu_b200_workspace* ws, const uint64_t* codes, int64_t n, int32_t* out_pts, void* stream);
int pcu_b200_morton_add(pcu_b200_workspace* ws, const uint64_t* a, const uint64_t* b, int64_t n, uint64_t* out, void* stream);
int pcu_b200_morton_subtract(pcu_b200_workspace* ws, const uint64_t* a, const uint64_t* b, int64_t n, uint64_t* out, void* stream);
int pcu_b200_morton_knn(pcu_b200_workspace* ws, const uint64_t* codes, int64_t n, const uint64_t* qcodes, int64_t m, int k,
                        int sort_dist, int64_t* out_idx, void* stream);

/* ---- HOST-pointer conveniences (H2D + kernels + D2H, synchronous) --------------------------
 * The calls the numpy-facing binding makes; these are what `e2e` in bench.py times.              */
int pcu_b200_knn_host_f32(pcu_b200_workspace* ws, const float* query, int64_t n, const float* dataset, int64_t m,
                          int k, int squared, float* out_dist, int64_t* out_idx, int64_t* out_n_tied);
int pcu_b200_knn_host_f64(pcu_b200_workspace* ws, const double* query, int64_t n, const double* dataset, int64_t m,
                          int k, int squared, double* out_dist, int64_t* out_idx, int64_t* out_n_tied);
int pcu_b200_nn_stats_host_f32(pcu_b200_workspace* ws, const float* query, int64_t n, const float* dataset,
                               int64_t m, pcu_b200_nn_stats* out_stats);
int pcu_b200_nn_stats_host_f64(pcu_b200_workspace* ws, const double* query, int64_t n, const double* dataset,
                               int64_t m, pcu_b200_nn_stats* out_stats);
int pcu_b200_chamfer_host_f32(pcu_b200_workspace* ws, const float* x, int64_t n, const float* y, int64_t m,
                              pcu_b200_nn_stats* out_stats, float* out_value);
int pcu_b200_chamfer_host_f64(pcu_b200_workspace* ws, const double* x, int64_t n, const double* y, int64_t m,
                              pcu_b200_nn_stats* out_stats, double* out_value);
int pcu_b200_batched_chamfer_host_f32(pcu_b200_workspace* ws, const float* x, const float* y, int64_t batch,
                                      int64_t n, int64_t m, float* out_per_pair, double* out_sum);
int pcu_b200_morton_encode_host_i32(pcu_b200_workspace* ws, const int32_t* pts, int64_t n, uint64_t* out_codes);
int pcu_b200_morton_encode_host_i64(pcu_b200_workspace* ws, const int64_t* pts, int64_t n, uint64_t* out_codes);
int pcu_b200_morton_decode_host(pcu_b200_workspace* ws, const uint64_t* codes, int64_t n, int32_t* out_pts);
int pcu_b200_morton_add_host(pcu_b200_workspace* ws, const uint64_t* a, const uint64_t* b, int64_t n, uint64_t* out);
int pcu_b200_morton_subtract_host(pcu_b200_workspace* ws, const uint64_t* a, const uint64_t* b, int64_t n, uint64_t* out);
int pcu_b200_morton_knn_host(pcu_b200_workspace* ws, const uint64_t* codes, int64_t n, const uint64_t* qcodes, int64_t m, int k,
                             int sort_dist, int64_t* out_idx);
int pcu_b200_normals_knn_host_f32(pcu_b200_workspace* ws, const float* points, int64_t n, const float* view_dirs, int k,
                                  double drop_angle_threshold, int64_t* out_idx, float* out_normals, int64_t* out_count);
int pcu_b200_normals_knn_host_f64(pcu_b200_workspace* ws, const double* points, int64_t n, const double* view_dirs, int k,
                                  double drop_angle_threshold, int64_t* out_idx, double* out_normals, int64_t* out_count);
/* voxel-grid down-sampling / duplicate removal on HOST arrays (outputs sized for the worst case as in the device
 * forms; out_rows / out_counts are HOST integers here) */
int pcu_b200_voxel_downsample_host_f32(pcu_b200_workspace* ws, const float* points, int64_t n, const void* attrib, int attrib_cols,
                                       int attrib_is_f64, const double voxel_size[3], const double min_bound[3], const double max_bound[3],
                                       int min_points_per_voxel, float* out_points, void* out_attrib, int32_t* out_counts, int64_t* out_rows);
int pcu_b200_voxel_downsample_host_f64(pcu_b200_workspace* ws, const double* points, int64_t n, const void* attrib, int attrib_cols,
                                       int attrib_is_f64, const double voxel_size[3], const double min_bound[3], const double max_bound[3],
                                       int min_points_per_voxel, double* out_points, void* out_attrib, int32_t* out_counts, int64_t* out_rows);
/* Poisson-disk down-sampling on HOST arrays: out_idx (capacity n) and out_count are HOST memory */
int pcu_b200_poisson_disk_downsample_host_f32(pcu_b200_workspace* ws, const float* points, int64_t n, double radius, int target_num_samples,
                                              uint32_t seed, float sample_num_tolerance, int32_t* out_idx, int64_t* out_count);
int pcu_b200_poisson_disk_downsample_host_f64(pcu_b200_workspace* ws, const double* points, int64_t n, double radius, int target_num_samples,
                                              uint32_t seed, float sample_num_tolerance, int32_t* out_idx, int64_t* out_count);
int pcu_b200_deduplicate_host_f32(pcu_b200_workspace* ws, const float* points, int64_t n, double epsilon, const void* faces, int64_t n_faces,
                                  int face_cols, int faces_are_i64, float* out_points, int32_t* out_svi, int32_t* out_svj, void* out_faces,
                                  int64_t* out_counts);
int pcu_b200_deduplicate_host_f64(pcu_b200_workspace* ws, const double* points, int64_t n, double epsilon, const void* faces, int64_t n_faces,
                                  int face_cols, int faces_are_i64, double* out_points, int32_t* out_svi, int32_t* out_svj, void* out_faces,
                                  int64_t* out_counts);
int pcu_b200_normals_ball_host_f32(pcu_b200_workspace* ws, const float* points, int64_t n, const float* view_dirs,
                                   const pcu_b200_ball_options* options, int64_t* out_idx, float* out_normals, int64_t* out_count);
int pcu_b200_normals_ball_host_f64(pcu_b200_workspace* ws, const double* points, int64_t n, const double* view_dirs,
                                   const pcu_b200_ball_options* options, int64_t* out_idx, double* out_normals, int64_t* out_count);

/* Timeline of the last kd-tree build on the workspace's device (globaltimer, ns; synchronises the device):
 * [0] start, [1] set-up done, [2 + l] grid-wide level l done (l < 28), [30] grid-wide phase done, [31] last CTA done,
 * [32] grid-wide levels, [33] subtrees built by single CTAs. */
int pcu_b200_debug_kd_times(pcu_b200_workspace* ws, uint64_t* out40);

/* ---- diagnostics ----------------------------------------------------------------------------
 * Builds the kd-tree replica used by the tie replay for HOST points and copies it out, so tests can
 * compare it node for node with the reference's tree.  order: (m) slot -> point index (nanoflann's
 * vAcc); per node (capacity node_cap, at most 2 m - 1 are used): split dimension (-1 = leaf),
 * divlow, divhigh, slot range [first, last), children.  Returns the node count through out_nodes.  */
int pcu_b200_debug_kd_tree_f32(pcu_b200_workspace* ws, const float* points, int64_t m, int max_points_per_leaf,
                               int32_t* order, int64_t node_cap, int32_t* feat, float* div_lo, float* div_hi,
                               int32_t* first, int32_t* last, int32_t* kid0, int32_t* kid1, int64_t* out_nodes);
int pcu_b200_debug_kd_tree_f64(pcu_b200_workspace* ws, const double* points, int64_t m, int max_points_per_leaf,
                               int32_t* order, int64_t node_cap, int32_t* feat, double* div_lo, double* div_hi,
                               int32_t* first, int32_t* last, int32_t* kid0, int32_t* kid1, int64_t* out_nodes);

#ifdef __cplusplus
}
#endif
#endif /* PCU_B200_H */
