// pcu_b200.cu -- workspace, launch sequencing and the C ABI declared in include/pcu_b200.h.
//
// Host side of the B200 nearest-neighbour path.  It owns no algorithmic decisions that depend on
// the data: grid shapes, far-query lists and tie lists are produced and consumed on the device, so
// a device-pointer call enqueues a fixed sequence of launches and returns without synchronising.
#include <cuda_runtime.h>
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <new>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/pcu_b200.h"
#include "host_util.h"
#include "staging.h"
#include "common.cuh"
#include "grid.cuh"
#include "search.cuh"
#include "nn1.cuh"
#include "topk.cuh"
#include "pyramid.cuh"
#include "kdreplay.cuh"
#include "normals.cuh"
#include "morton.cuh"
#include "sinkhorn.cuh"
#include "voxel.cuh"
#include "dedup.cuh"
#include "poisson.cuh"

using namespace pcu;

namespace {

thread_local std::string g_error;
std::atomic<long long> g_launches{0};

int fail(int status, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_error = buf;
    return status;
}

#define PCU_CUDA(expr)                                                                                   \
    do {                                                                                                 \
        cudaError_t e__ = (expr);                                                                        \
        if (e__ != cudaSuccess)                                                                          \
            return fail(e__ == cudaErrorMemoryAllocation ? PCU_B200_OUT_OF_MEMORY : PCU_B200_CUDA_ERROR, \
                        "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__);    \
    } while (0)

#define PCU_TRY(expr)                      \
    do {                                   \
        int s__ = (expr);                  \
        if (s__ != PCU_B200_OK) return s__; \
    } while (0)

#define PCU_LAUNCH(kernel, grid, block, stream, ...)                   \
    do {                                                               \
        kernel<<<grid, block, 0, stream>>>(__VA_ARGS__);               \
        g_launches.fetch_add(1, std::memory_order_relaxed);            \
        PCU_CUDA(cudaGetLastError());                                  \
    } while (0)

// Launch with programmatic stream serialisation: the kernel (which starts with grid_dependency_wait())
// may have its CTAs scheduled while its predecessor in the stream is still draining.
#define PCU_LAUNCH_PDL(kernel, grid, block, stream, ...)                                       \
    do {                                                                                       \
        cudaLaunchConfig_t cfg__ = {};                                                         \
        cfg__.gridDim = dim3(grid);                                                            \
        cfg__.blockDim = dim3(block);                                                          \
        cfg__.stream = stream;                                                                 \
        cudaLaunchAttribute attr__[1];                                                         \
        attr__[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                     \
        attr__[0].val.programmaticStreamSerializationAllowed = 1;                              \
        cfg__.attrs = attr__;                                                                  \
        cfg__.numAttrs = 1;                                                                    \
        PCU_CUDA(cudaLaunchKernelEx(&cfg__, kernel, __VA_ARGS__));                             \
        g_launches.fetch_add(1, std::memory_order_relaxed);                                    \
    } while (0)

#define PCU_LAUNCH_PDL_SMEM(kernel, grid, block, smem, stream, ...)                            \
    do {                                                                                       \
        cudaLaunchConfig_t cfg__ = {};                                                         \
        cfg__.gridDim = dim3(grid);                                                            \
        cfg__.blockDim = dim3(block);                                                          \
        cfg__.dynamicSmemBytes = (smem);                                                       \
        cfg__.stream = stream;                                                                 \
        cudaLaunchAttribute attr__[1];                                                         \
        attr__[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                     \
        attr__[0].val.programmaticStreamSerializationAllowed = 1;                              \
        cfg__.attrs = attr__;                                                                  \
        cfg__.numAttrs = 1;                                                                    \
        PCU_CUDA(cudaLaunchKernelEx(&cfg__, kernel, __VA_ARGS__));                             \
        g_launches.fetch_add(1, std::memory_order_relaxed);                                    \
    } while (0)

// Descriptor-taking kernels exist in two flavours: descriptors by value in parameter space (single
// pair: `plan.by_value`) or in a device array (batches).  K<T, CloudsX<T>[, SweepsX<T>][, extra...]>.
#define PCU_LAUNCH_C(K, grid, block)                                                                      \
    do {                                                                                                  \
        if (plan.by_value) PCU_LAUNCH_PDL((K<T, CloudsVal<T>>), grid, block, stream, plan.cv);            \
        else PCU_LAUNCH_PDL((K<T, CloudsPtr<T>>), grid, block, stream, plan.cp);                          \
    } while (0)
#define PCU_LAUNCH_CS(K, grid, block, ...)                                                                \
    do {                                                                                                  \
        if (plan.by_value)                                                                                \
            PCU_LAUNCH_PDL((K<T, CloudsVal<T>, SweepsVal<T>, ##__VA_ARGS__>), grid, block, stream, plan.cv, plan.sv); \
        else                                                                                              \
            PCU_LAUNCH_PDL((K<T, CloudsPtr<T>, SweepsPtr<T>, ##__VA_ARGS__>), grid, block, stream, plan.cp, plan.sp); \
    } while (0)

// Per-field byte strides between consecutive pairs of a batch (side 0 = first cloud of each pair,
// side 1 = second cloud; direction 0 = first -> second, direction 1 = second -> first).
struct CloudStrides { size_t raw, sorted, rank, cell_start, grid, wall_lo, wall_hi, bbox_partial, scan_state, scan_ticket, occupied, pyramid, shape; };
struct SweepStrides { size_t out_dist, out_idx, partial, far_list, vfar_list, counters, tie_list; };

template <typename U>
__device__ __forceinline__ U* advance(U* p, size_t bytes) {
    return p ? reinterpret_cast<U*>(reinterpret_cast<unsigned char*>(const_cast<typename std::remove_const<U>::type*>(p)) + bytes) : p;
}

// Writes the cloud / sweep descriptors of every pair of a batch.  They are generated on the device
// from two prototypes, so a call never stages descriptors through host memory that a later call
// could overwrite while this one is still queued.
template <typename T>
struct DescriptorArgs {
    Cloud<T> cloud[2];
    Sweep<T> sweep[2];
    CloudStrides cs[2];
    SweepStrides ss[2];
    long long batch;
    int nsweeps;
    pcu_b200_nn_stats* stats;
    T* value_out;   // per-pair Chamfer values (bidirectional calls), or null
};

template <typename T>
__global__ void descriptors_kernel(const __grid_constant__ DescriptorArgs<T> a, Cloud<T>* clouds, Sweep<T>* sweeps) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= a.batch) return;
    for (int s = 0; s < 2; ++s) {
        Cloud<T> c = a.cloud[s];
        const CloudStrides& st = a.cs[s];
        c.raw = advance(c.raw, p * st.raw);
        c.sorted = advance(c.sorted, p * st.sorted);
        c.rank = advance(c.rank, p * st.rank);
        c.cell_start = advance(c.cell_start, p * st.cell_start);
        c.grid = advance(c.grid, p * st.grid);
        c.wall_lo = advance(c.wall_lo, p * st.wall_lo);
        c.wall_hi = advance(c.wall_hi, p * st.wall_hi);
        c.bbox_partial = advance(c.bbox_partial, p * st.bbox_partial);
        c.scan_state = advance(c.scan_state, p * st.scan_state);
        c.scan_ticket = advance(c.scan_ticket, p * st.scan_ticket);
        c.occupied = advance(c.occupied, p * st.occupied);
        if (p != 0) c.hint_out = nullptr;   // the first pair of a batch speaks for all of them
        c.pyramid = advance(c.pyramid, p * st.pyramid);
        c.shape = advance(c.shape, p * st.shape);
        clouds[2 * p + s] = c;
    }
    for (int d = 0; d < a.nsweeps; ++d) {
        Sweep<T> w = a.sweep[d];
        const SweepStrides& st = a.ss[d];
        w.qcloud = (int)(2 * p + d);
        w.dcloud = (int)(2 * p + 1 - d);
        w.out_dist = advance(w.out_dist, p * st.out_dist);
        w.out_idx = advance(w.out_idx, p * st.out_idx);
        w.partial = advance(w.partial, p * st.partial);
        w.far_list = advance(w.far_list, p * st.far_list);
        w.vfar_list = advance(w.vfar_list, p * st.vfar_list);
        w.counters = advance(w.counters, p * st.counters);
        w.tie_list = advance(w.tie_list, p * st.tie_list);
        w.stats = a.stats ? a.stats + p * a.nsweeps + d : nullptr;
        w.pair_stats = a.stats ? a.stats + p * a.nsweeps : nullptr;
        w.pair_ticket = advance(a.sweep[0].counters, p * a.ss[0].counters) + 4;
        w.value_out = (a.nsweeps == 2 && a.value_out) ? a.value_out + p : nullptr;
        sweeps[p * a.nsweeps + d] = w;
    }
}

}  // namespace

struct pcu_b200_workspace {
    int device = 0;
    cudaStream_t own_stream = nullptr;
    unsigned char* arena = nullptr;      // scratch of the device-pointer entry points
    size_t arena_bytes = 0;
    unsigned char* io = nullptr;         // device copies of host inputs / outputs (host entry points)
    size_t io_bytes = 0;
    unsigned char* aux = nullptr;        // intermediate results that outlive a nested call's re-carving of the arena (normals)
    size_t aux_bytes = 0;
    pcu_b200_options opts{};
    int sm_count = 148;
    // optional per-stage timing (bench.py's roofline pass): events recorded on the launching stream
    unsigned small_attr = 0;             // bin_small_kernel instantiations whose shared-memory limit has been raised
    // grid-sizing feedback: the kernels leave {cell_cap, non-empty cells, n, valid, unsettled queries, queries, valid, -}
    // per cloud in this
    // host-mapped buffer; the next call with the same shapes reads it (no synchronisation: a hint only)
    volatile unsigned* hint_host = nullptr;
    unsigned* hint_dev = nullptr;
    long long hint_key[5] = {0, 0, 0, 0, 0};   // n, m, k, sizeof(T), batch of the call the hints belong to
    float cell_mult[2] = {1.f, 1.f};           // current refinement of the two clouds' grids (cells per point x this)
    float cell_mult_ceiling[2] = {32.f, 32.f}; // lowered when a refinement left too many queries unsettled
    cudaStream_t copy_stream = nullptr;  // host entry points: the H2D copies run here, the kernels on own_stream
    cudaEvent_t arrived[2] = {};         // recorded on copy_stream behind each cloud's copy
    unsigned char* host_slot = nullptr;  // 4 KB of pinned host memory: small results land here, then in the caller's buffers
    const unsigned* replay_overflows = nullptr;   // device counter of the last KNN call's tie replay (null: none ran)
    cudaStream_t last_stream = nullptr;  // stream of the previous call (see adopt_stream)
    bool has_last_stream = false;
    cudaEvent_t handover = nullptr;
    bool profiling = false;
    cudaEvent_t marks[11] = {};   // 0 .. 8: stage boundaries of a device call; 9 / 10: before the H2D / after the D2H of a host call
    int marks_used = 0;
    bool host_marks = false;      // marks 9 and 10 belong to the last call
    HostStager* stager = nullptr; // pinned ring + copy threads for pageable inputs of the host entry points (created on first use)
    long long poisson_trials = 0;                  // radius trials of the last Poisson-disk call
    unsigned long long* poisson_rounds = nullptr;  // device: MIS rounds of the last Poisson-disk call, summed over its trials
};

// A cloud binned once (pcu_b200_cloud_prepare_*): its cell-sorted points, cell table, grid header, wall tables and
// pyramid buffers live in one private device block, described by the same Cloud<T> record the kernels take.
struct pcu_b200_cloud {
    int device = 0;
    int is_f64 = 0;
    long long n = 0;
    unsigned char* block = nullptr;
    size_t bytes = 0;
    Cloud<float> desc32{};
    Cloud<double> desc64{};
    const void* raw = nullptr;   // the handle's own copy of the caller's (n, 3) array (inside block)
    int knn_k = 1;               // the k the cell size was chosen for
    int leaf = 0;                // > 0: the block also holds the reference-tree replica built with this leaf size
    KdReplayBuffers<float> kd32{};
    KdReplayBuffers<double> kd64{};
};
template <typename T> KdReplayBuffers<T>& cloud_tree(pcu_b200_cloud* c);
template <> KdReplayBuffers<float>& cloud_tree<float>(pcu_b200_cloud* c) { return c->kd32; }
template <> KdReplayBuffers<double>& cloud_tree<double>(pcu_b200_cloud* c) { return c->kd64; }

#define PCU_STAGE_NAMES "descriptors", "bbox+grid", "histogram", "scan", "scatter", "search", "search_far", "finalize", "h2d", "d2h"

namespace {

// Makes ws->device current for the duration of an entry point and puts the caller's device back on every
// exit path (a torch program with cuda:0 current that passes cuda:1 tensors keeps cuda:0 current).
struct DeviceGuard {
    int previous = -1;
    bool switched = false;
    cudaError_t status = cudaSuccess;
    explicit DeviceGuard(int device) {
        status = cudaGetDevice(&previous);
        if (status == cudaSuccess && previous != device) {
            status = cudaSetDevice(device);
            switched = status == cudaSuccess;
        }
    }
    ~DeviceGuard() { if (switched) cudaSetDevice(previous); }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};
#define PCU_ON_DEVICE(ws)                                                                              \
    DeviceGuard device_guard__((ws)->device);                                                          \
    if (device_guard__.status != cudaSuccess)                                                          \
        return fail(PCU_B200_CUDA_ERROR, "cudaSetDevice(%d) failed: %s", (ws)->device, cudaGetErrorString(device_guard__.status))

// A workspace serves one stream at a time.  When a call arrives on another stream than the previous one,
// the new stream is made to wait (on the device) for everything the previous call enqueued: the scratch is shared.
int adopt_stream(pcu_b200_workspace* ws, cudaStream_t stream) {
    if (ws->has_last_stream && ws->last_stream != stream) {
        if (!ws->handover) PCU_CUDA(cudaEventCreateWithFlags(&ws->handover, cudaEventDisableTiming));
        PCU_CUDA(cudaEventRecord(ws->handover, ws->last_stream));
        PCU_CUDA(cudaStreamWaitEvent(stream, ws->handover, 0));
    }
    ws->last_stream = stream;
    ws->has_last_stream = true;
    return PCU_B200_OK;
}

// Scratch grows with stream-ordered allocation: the old block is released and the new one obtained in the
// order of `stream`, so earlier calls still queued there keep their memory until they are done and neither
// the host nor the rest of the device is synchronised.
int grow_block(unsigned char*& block, size_t& have, size_t bytes, cudaStream_t stream, const char* what) {
    if (bytes <= have) return PCU_B200_OK;
    if (block) {
        PCU_CUDA(cudaFreeAsync(block, stream));
        block = nullptr;
        have = 0;
    }
    const size_t want = align_up(bytes + bytes / 8, 1 << 20);
    void* p = nullptr;
    cudaError_t e = cudaMallocAsync(&p, want, stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(PCU_B200_OUT_OF_MEMORY, "cudaMallocAsync of %zu bytes of %s failed: %s", want, what, cudaGetErrorString(e));
    }
    block = (unsigned char*)p;
    have = want;
    return PCU_B200_OK;
}

int ensure_arena(pcu_b200_workspace* ws, size_t bytes, cudaStream_t stream) {
    PCU_TRY(adopt_stream(ws, stream));
    return grow_block(ws->arena, ws->arena_bytes, bytes, stream, "scratch");
}

int ensure_io(pcu_b200_workspace* ws, size_t bytes, cudaStream_t stream) {
    return grow_block(ws->io, ws->io_bytes, bytes, stream, "staging");
}

void mark(pcu_b200_workspace* ws, int index, cudaStream_t stream) {
    if (!ws->profiling) return;
    cudaEventRecord(ws->marks[index], stream);
    if (index <= 8) ws->marks_used = index + 1;
    if (index == 0) ws->host_marks = false;
    if (index == 10) ws->host_marks = true;
}

int cell_cap_for(long long n, double occupancy) {
    double c = (double)n / occupancy;
    if (c < 1.0) c = 1.0;
    if (c > (double)(1 << 27)) c = (double)(1 << 27);
    return (int)c;
}

float occupancy_for(const pcu_b200_workspace* ws, int k) {
    if (ws->opts.cell_occupancy > 0.f) return ws->opts.cell_occupancy;
    // k = 1: 1.5 points per cell (measured on C3, profiles/r2d_occ.log: the sweep visits fewer candidates -- 139 -> 124 us --
    // while the scan over more cells and the far pass grow by less; 1.25 and 1.75 are within 1 % of it, 1.0 loses 8 %)
    if (k <= 1) return 1.5f;
    // k > 1 (thread-per-query lists): measured on 2 x 10^6 queries against 10^6 uniform points (profiles/r2r_knn_occ.log) --
    // fewer points per cell mean fewer candidates in the 27 cells but more queries left to the slow warp pass; the best
    // trade-off was 3 at k = 4 (0.239 vs 0.277 ms per 10^6 queries at 2), 4 at k = 8, 7 at k = 16, 12 at k = 32
    // (2.78 vs 3.02 ms at 16).  Piecewise linear through those points.
    static const float ks[] = {2.f, 4.f, 8.f, 16.f, 32.f}, occ[] = {2.f, 3.f, 4.f, 7.f, 12.f};
    const float kf = (float)k;
    if (kf <= ks[0]) return occ[0];
    for (int i = 1; i < 5; ++i)
        if (kf <= ks[i]) return occ[i - 1] + (occ[i] - occ[i - 1]) * (kf - ks[i - 1]) / (ks[i] - ks[i - 1]);
    return 0.375f * kf;     // k > 32: the generic pyramid path, same slope as the last segment
}

// What one call works on: `batch` independent pairs (first cloud: n points, second: m points).
template <typename T>
struct PlanSpec {
    long long batch = 1;
    const T* a = nullptr;   // (batch, n, 3)
    const T* b = nullptr;   // (batch, m, 3)
    long long n = 0, m = 0;
    int nsweeps = 1;        // 1: first -> second;  2: both directions
    int k = 1;
    int squared = 0;
    bool want_stats = false;
    bool want_out = false;
    float occupancy = 2.f;
    float cell_mult[2] = {1.f, 1.f};   // grid refinement from the previous call's fill statistics
    unsigned* hint_dev = nullptr;      // 2 x 4 words of host-mapped memory, or null
    int binning = 0;                // pcu_b200_options::binning
    bool prepared_second = false;   // the second cloud is a pcu_b200_cloud: its descriptor replaces the carved one, it is not binned
    T* out_dist = nullptr;          // want_out (batch == 1)
    long long* out_idx = nullptr;
    pcu_b200_nn_stats* stats = nullptr;   // caller's device buffer, or null -> carved from the arena
    T* value_out = nullptr;               // per-pair Chamfer values (nsweeps == 2), or null
    long long replay_points = 0;
};

// Scratch layout of one call.  Every per-cloud / per-sweep buffer is an array over the batch with
// a uniform stride, so descriptors can be generated on the device.
template <typename T>
struct Plan {
    DescriptorArgs<T> args{};
    Cloud<T>* d_clouds = nullptr;
    Sweep<T>* d_sweeps = nullptr;
    bool by_value = false;        // single pair: descriptors travel in kernel-parameter space
    CloudsVal<T> cv{};
    SweepsVal<T> sv{};
    CloudsPtr<T> cp{};
    SweepsPtr<T> sp{};
    pcu_b200_nn_stats* d_stats = nullptr;
    unsigned char* zero_begin = nullptr;   // zeroed per call: [cell counters | scan states, tickets, sweep counters]
    size_t zero_bytes = 0;
    size_t zero_cells_bytes = 0;           // leading part that only the multi-launch grid build needs zeroed
    bool one_cta_binning = false;          // bin_small_kernel instead of the five grid-wide passes
    long long max_n = 0;
    int max_cap = 0;
    int max_bbox_blocks = 1;
    int far_blocks = 1;
    int nclouds = 0, nsweeps_total = 0;
    size_t total = 0;
    KdReplayBuffers<T> replay{};

    template <typename U>
    static U* take_strided(Carver& cv, size_t count_per_item, long long batch, size_t& stride_bytes) {
        stride_bytes = align_up(count_per_item * sizeof(U));
        return reinterpret_cast<U*>(cv.take<unsigned char>(stride_bytes * (size_t)batch));
    }

    // Carves (or, with base == nullptr, just measures) the layout.
    void layout(unsigned char* base, const PlanSpec<T>& sp) {
        Carver cv(base);
        const long long B = sp.batch;
        nclouds = (int)(2 * B);
        nsweeps_total = (int)(B * sp.nsweeps);
        d_clouds = cv.take<Cloud<T>>((size_t)nclouds);
        d_sweeps = cv.take<Sweep<T>>((size_t)nsweeps_total);
        d_stats = sp.stats ? sp.stats : (sp.want_stats ? cv.take<pcu_b200_nn_stats>((size_t)nsweeps_total) : nullptr);
        args = DescriptorArgs<T>{};
        args.batch = B;
        args.nsweeps = sp.nsweeps;
        args.stats = sp.want_stats ? d_stats : nullptr;
        args.value_out = sp.value_out;
        const long long sizes[2] = {sp.n, sp.m};
        const T* raws[2] = {sp.a, sp.b};
        max_n = std::max(sp.n, sp.m);
        max_cap = 0;
        max_bbox_blocks = 1;
        // far pass: a fixed number of CTAs per sweep (warp-stride loop over the far list)
        far_blocks = (int)std::max<long long>(4, 296 / std::max<long long>(1, B * sp.nsweeps));
        // zeroed region first: cell counters and sweep counters
        const size_t zero_from = cv.off;
        for (int s = 0; s < 2; ++s) {
            Cloud<T>& cl = args.cloud[s];
            cl.raw = raws[s];
            cl.n = sizes[s];
            cl.cell_cap = cell_cap_for(sizes[s], sp.occupancy / sp.cell_mult[s]);
            cl.hint_out = sp.hint_dev ? sp.hint_dev + 8 * s : nullptr;
            cl.stride = std::min(kMaxGridDim, cl.cell_cap) + 1;
            cl.bbox_blocks = (int)std::min<long long>(kMaxBBoxBlocks, std::max<long long>(1, (3 * sizes[s] + 2 * kThreads * kBBoxPerThread - 1) / (2 * kThreads * kBBoxPerThread)));
            max_bbox_blocks = std::max(max_bbox_blocks, cl.bbox_blocks);
            args.cs[s].raw = (size_t)3 * sizes[s] * sizeof(T);
            cl.cell_start = take_strided<unsigned>(cv, (size_t)cl.cell_cap + 1, B, args.cs[s].cell_start);
            max_cap = std::max(max_cap, cl.cell_cap);
        }
        zero_cells_bytes = cv.off - zero_from;
        for (int s = 0; s < 2; ++s) {
            Cloud<T>& cl = args.cloud[s];
            cl.scan_state = take_strided<unsigned long long>(cv, ((size_t)cl.cell_cap + 1 + kScanTile - 1) / kScanTile + 1, B,
                                                             args.cs[s].scan_state);
            cl.scan_ticket = take_strided<unsigned>(cv, 2, B, args.cs[s].scan_ticket);   // [0] scan tiles, [1] bbox CTAs
            cl.occupied = take_strided<unsigned>(cv, 1, B, args.cs[s].occupied);
        }
        // One CTA per cloud when the counters fit in shared memory and the clouds are small: five dependent
        // launches then cost more than one CTA's serial passes (measured on B200, pair of n points: 64 vs 71 us
        // at n = 1024, 62 vs 69 us at 4096, break-even near 12k; at 65536 one SM needs ~130 us for what the
        // grid-wide passes do in ~50 us, and a batch of 1024 such pairs is 5 % slower, so larger clouds keep
        // the grid-wide passes whatever the batch size).
        const bool fits = max_cap + 1 <= kSmallMaxCells && max_n <= kSmallMaxPoints;
        one_cta_binning = !sp.prepared_second && fits && (sp.binning == 2 || (sp.binning == 0 && max_n <= 8192));
        for (int d = 0; d < sp.nsweeps; ++d)
            args.sweep[d].counters = take_strided<unsigned>(cv, 8, B, args.ss[d].counters);
        zero_begin = base ? base + zero_from : nullptr;
        zero_bytes = cv.off - zero_from;
        for (int s = 0; s < 2; ++s) {
            Cloud<T>& cl = args.cloud[s];
            CloudStrides& st = args.cs[s];
            cl.sorted = take_strided<Pt<T>>(cv, (size_t)cl.n, B, st.sorted);
            cl.rank = take_strided<unsigned>(cv, (size_t)cl.n, B, st.rank);
            cl.grid = take_strided<GridHeader<T>>(cv, 1, B, st.grid);
            cl.wall_lo = take_strided<T>(cv, (size_t)3 * cl.stride, B, st.wall_lo);
            cl.wall_hi = take_strided<T>(cv, (size_t)3 * cl.stride, B, st.wall_hi);
            cl.bbox_partial = take_strided<T>(cv, (size_t)cl.bbox_blocks * 6, B, st.bbox_partial);
            cl.pyramid = take_strided<unsigned>(cv, (size_t)cl.cell_cap + 64, B, st.pyramid);
            cl.shape = take_strided<PyramidShape>(cv, 1, B, st.shape);
        }
        for (int d = 0; d < sp.nsweeps; ++d) {
            Sweep<T>& sw = args.sweep[d];
            SweepStrides& st = args.ss[d];
            sw.k = sp.k;
            sw.squared = sp.squared;
            const long long nq = sizes[d];
            sw.main_blocks = (int)((nq + kThreads - 1) / kThreads);
            sw.far_blocks = far_blocks;
            sw.far_list = take_strided<unsigned>(cv, (size_t)nq, B, st.far_list);
            sw.vfar_list = take_strided<unsigned>(cv, (size_t)nq, B, st.vfar_list);
            if (sp.want_out) {
                sw.tie_list = take_strided<long long>(cv, (size_t)nq, B, st.tie_list);
                sw.out_dist = sp.out_dist;   // batch == 1 on this path
                sw.out_idx = sp.out_idx;
            }
            if (sp.want_stats)
                sw.partial = take_strided<SweepPartial<T>>(cv, (size_t)sw.main_blocks + 2 * far_blocks, B, st.partial);
        }
        if (sp.replay_points > 0) replay.carve(cv, sp.replay_points);
        total = cv.off;
        // descriptor sources
        this->cp.p = d_clouds;
        this->sp.p = d_sweeps;
        by_value = B == 1;
        if (by_value) {
            for (int s = 0; s < 2; ++s) this->cv.v[s] = args.cloud[s];
            for (int d = 0; d < sp.nsweeps; ++d) {
                Sweep<T> w = args.sweep[d];
                w.qcloud = d; w.dcloud = 1 - d;
                w.stats = args.stats ? args.stats + d : nullptr;
                w.pair_stats = args.stats;
                w.pair_ticket = args.sweep[0].counters + 4;
                w.value_out = (sp.nsweeps == 2) ? args.value_out : nullptr;
                this->sv.v[d] = w;
            }
        }
    }
};

template <typename T>
int upload_descriptors(Plan<T>& plan, cudaStream_t stream) {
    if (plan.by_value) return PCU_B200_OK;   // nothing to upload: descriptors ride along with every launch
    const unsigned blocks = (unsigned)((plan.args.batch + 127) / 128);
    PCU_LAUNCH(descriptors_kernel<T>, blocks, 128, stream, plan.args, plan.d_clouds, plan.d_sweeps);
    return PCU_B200_OK;
}

// Grid-sizing feedback.  A grid sized for `occupancy` points per cell of the bounding BOX fills only a
// few of its cells when the cloud is a surface (or any thin set), and those hold many points each, so
// every query wades through long candidate runs.  The binning kernels report how many cells were
// non-empty; when the same shapes come again on this workspace (a loss evaluated every iteration, a
// benchmark loop) and the non-empty cells held well over the target, the grid gets more cells --
// assuming the non-empty count grows like h^-2 (a surface), so r times fewer points per non-empty cell
// cost r^1.5 times more cells -- up to 32 times the default; a refined grid that turns out too fine for
// the data it now sees (few points per non-empty cell, or many queries left unsettled by their 27
// cells) shrinks again.  Box-filling clouds never trigger it
// (uniform data sits at 0.9 of the threshold), results never depend on it.
template <typename T>
void apply_grid_feedback(pcu_b200_workspace* ws, PlanSpec<T>& spec) {
    const long long key[5] = {spec.n, spec.m, spec.k, (long long)sizeof(T), spec.batch};
    if (!ws->hint_host) return;
    bool same = true;
    for (int i = 0; i < 5; ++i) same = same && key[i] == ws->hint_key[i];
    if (!same) {
        for (int i = 0; i < 5; ++i) ws->hint_key[i] = key[i];
        ws->cell_mult[0] = ws->cell_mult[1] = 1.f;
        ws->cell_mult_ceiling[0] = ws->cell_mult_ceiling[1] = 32.f;
        for (int i = 0; i < 16; ++i) ws->hint_host[i] = 0u;
    } else {
        const long long sizes[2] = {spec.n, spec.m};
        for (int s = 0; s < 2; ++s) {
            volatile unsigned* h = ws->hint_host + 8 * s;
            const unsigned cap = h[0], nonempty = h[1], pts = h[2], valid = h[3];
            if (!valid || nonempty == 0u || pts != (unsigned)sizes[s]) continue;
            if (cap != (unsigned)cell_cap_for(sizes[s], spec.occupancy / ws->cell_mult[s])) continue;   // measured under another grid
            const double per_cell = (double)pts / (double)nonempty;
            const double r = per_cell / (1.3 * (double)spec.occupancy);
            // share of the queries searched against this cloud that the 3 x 3 x 3 cells could not settle:
            // many of them means the cells are too fine for where the queries are (or the clouds are far
            // apart), and finer cells only deepen the slow passes
            const double far_share = (h[6] && h[5]) ? (double)h[4] / (double)h[5] : 0.0;
            double m = (double)ws->cell_mult[s];
            if (far_share > 0.05) {
                if (m > 1.0) ws->cell_mult_ceiling[s] = (float)std::max(1.0, 0.6 * m);   // do not come back up here
                m *= 0.35;
            } else if (r > 1.6) m *= r * std::sqrt(r);                             // dead band 0.8 .. 1.6
            else if (r < 0.8) m *= (r / 0.8) * std::sqrt(r / 0.8);
            m = std::min((double)ws->cell_mult_ceiling[s], m);
            ws->cell_mult[s] = m < 1.5 ? 1.f : (float)m;
            h[3] = 0u; h[6] = 0u;   // consumed
        }
    }
    spec.cell_mult[0] = ws->cell_mult[0];
    spec.cell_mult[1] = ws->cell_mult[1];
    spec.hint_dev = ws->hint_dev;
}

template <typename T>
int prepare_plan(pcu_b200_workspace* ws, Plan<T>& plan, PlanSpec<T>& spec, cudaStream_t stream) {
    apply_grid_feedback(ws, spec);
    plan.layout(nullptr, spec);
    PCU_TRY(ensure_arena(ws, plan.total, stream));
    plan.layout(ws->arena, spec);
    return PCU_B200_OK;
}

// bbox -> grid -> histogram -> scan -> scatter for every cloud of the plan
// `ready` (host entry points, single pairs): two events, recorded on the copy stream when the first / the second
// cloud has arrived on the device.  The first cloud is then binned -- all five passes -- while the second is
// still crossing PCIe, and only the second cloud's passes follow its copy.
// `between` (host entry points; may be null): host work to do once the first cloud's passes have been enqueued and
// before the second cloud's `ready` event is waited for -- the staged copy of the second cloud, which keeps the host
// busy, so that the GPU bins the first cloud meanwhile.  It records ready[1] itself.
template <typename T>
int enqueue_binning(pcu_b200_workspace* ws, const Plan<T>& plan, cudaStream_t stream, const cudaEvent_t* ready = nullptr,
                    bool first_only = false, const std::function<int()>* between = nullptr) {
    const int nclouds = plan.nclouds;
    if ((ready != nullptr || first_only) && plan.by_value && !plan.one_cta_binning) {
        PCU_CUDA(cudaMemsetAsync(plan.zero_begin, 0, plan.zero_bytes, stream));
        const unsigned scan_blocks = (unsigned)(((long long)plan.max_cap + 1 + kScanTile - 1) / kScanTile);
        const unsigned bin_blocks = (unsigned)((plan.max_n + kThreads - 1) / kThreads);
        for (int s = 0; s < (first_only ? 1 : 2); ++s) {   // first_only: the second cloud is a prepared one
            if (s == 1 && between != nullptr) PCU_TRY((*between)());
            if (ready != nullptr) PCU_CUDA(cudaStreamWaitEvent(stream, ready[s], 0));
            CloudsVal<T> one;
            one.v[0] = plan.cv.v[s];
            one.v[1] = plan.cv.v[s];
            PCU_LAUNCH_PDL((bbox_partial_kernel<T, CloudsVal<T>, true>), dim3(plan.max_bbox_blocks, 1), kThreads, stream, one);
            mark(ws, 2, stream);
            PCU_LAUNCH_PDL((cell_count_kernel<T, CloudsVal<T>>), dim3(bin_blocks, 1), kThreads, stream, one);
            mark(ws, 3, stream);
            PCU_LAUNCH_PDL((scan_lookback_kernel<T, CloudsVal<T>>), dim3(scan_blocks, 1), kScanThreads, stream, one);
            mark(ws, 4, stream);
            PCU_LAUNCH_PDL((scatter_kernel<T, CloudsVal<T>>), dim3(bin_blocks, 1), kThreads, stream, one);
            mark(ws, 5, stream);
        }
        if (first_only && between != nullptr) PCU_TRY((*between)());
        return PCU_B200_OK;
    }
    if (between != nullptr) PCU_TRY((*between)());   // the other build paths take both clouds at once
    if (ready != nullptr) {
        PCU_CUDA(cudaStreamWaitEvent(stream, ready[0], 0));
        if (!first_only) PCU_CUDA(cudaStreamWaitEvent(stream, ready[1], 0));
    }
    if (plan.one_cta_binning) {
        PCU_CUDA(cudaMemsetAsync(plan.zero_begin + plan.zero_cells_bytes, 0, plan.zero_bytes - plan.zero_cells_bytes, stream));
        const size_t smem = ((size_t)plan.max_cap + 1) * sizeof(unsigned);
        const unsigned bit = 1u << ((sizeof(T) == 8 ? 2 : 0) + (plan.by_value ? 1 : 0));
        if (!(ws->small_attr & bit)) {
            const size_t most = (size_t)kSmallMaxCells * sizeof(unsigned);
            if (plan.by_value)
                PCU_CUDA(cudaFuncSetAttribute(bin_small_kernel<T, CloudsVal<T>>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)most));
            else
                PCU_CUDA(cudaFuncSetAttribute(bin_small_kernel<T, CloudsPtr<T>>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)most));
            ws->small_attr |= bit;
        }
        if (plan.by_value) PCU_LAUNCH_PDL_SMEM((bin_small_kernel<T, CloudsVal<T>>), dim3(nclouds), kSmallThreads, smem, stream, plan.cv);
        else PCU_LAUNCH_PDL_SMEM((bin_small_kernel<T, CloudsPtr<T>>), dim3(nclouds), kSmallThreads, smem, stream, plan.cp);
        for (int stage = 2; stage <= 5; ++stage) mark(ws, stage, stream);   // the whole build shows up as "bbox+grid"
        return PCU_B200_OK;
    }
    PCU_CUDA(cudaMemsetAsync(plan.zero_begin, 0, plan.zero_bytes, stream));
    const unsigned scan_blocks = (unsigned)(((long long)plan.max_cap + 1 + kScanTile - 1) / kScanTile);
    if (plan.by_value) {
        PCU_LAUNCH_PDL((bbox_partial_kernel<T, CloudsVal<T>, true>), dim3(plan.max_bbox_blocks, nclouds), kThreads, stream, plan.cv);
    } else {
        PCU_LAUNCH_PDL((bbox_partial_kernel<T, CloudsPtr<T>, false>), dim3(plan.max_bbox_blocks, nclouds), kThreads, stream, plan.cp);
        PCU_LAUNCH_PDL((grid_setup_kernel<T, CloudsPtr<T>>), dim3(1, nclouds), kThreads, stream, plan.cp);
    }
    mark(ws, 2, stream);
    const unsigned bin_blocks = (unsigned)((plan.max_n + kThreads - 1) / kThreads);
    PCU_LAUNCH_C(cell_count_kernel, dim3(bin_blocks, nclouds), kThreads);
    mark(ws, 3, stream);
    PCU_LAUNCH_C(scan_lookback_kernel, dim3(scan_blocks, nclouds), kScanThreads);
    mark(ws, 4, stream);
    PCU_LAUNCH_C(scatter_kernel, dim3(bin_blocks, nclouds), kThreads);
    mark(ws, 5, stream);
    return PCU_B200_OK;
}

template <typename T>
int check_cloud_args(const void* a, long long n, const void* b, long long m) {
    if (!a || !b) return fail(PCU_B200_INVALID_ARGUMENT, "null point-cloud pointer");
    if (n <= 0 || m <= 0)
        return fail(PCU_B200_INVALID_ARGUMENT,
                    "Invalid input set with zero elements: both clouds must have shape (n, 3) with n > 0 "
                    "(got %lld and %lld rows)", n, m);
    // rows, cell prefixes and list entries are 32-bit throughout the pipeline, whatever the coordinate type
    const long long lim = 0x7fffffffLL;
    if (n >= lim || m >= lim)
        return fail(PCU_B200_INVALID_ARGUMENT, "point cloud too large (%lld, %lld rows; at most 2^31 - 2 are supported)", n, m);
    return PCU_B200_OK;
}

template <typename T> const Cloud<T>& cloud_desc(const pcu_b200_cloud* c);
template <> const Cloud<float>& cloud_desc<float>(const pcu_b200_cloud* c) { return c->desc32; }
template <> const Cloud<double>& cloud_desc<double>(const pcu_b200_cloud* c) { return c->desc64; }

// ---- k nearest neighbours ---------------------------------------------------------------------
template <typename T>
int knn_device(pcu_b200_workspace* ws, const T* query, long long n, const T* dataset, long long m, int k, int squared,
               T* out_dist, long long* out_idx, long long* out_n_tied, cudaStream_t stream, pcu_b200_cloud* prepared = nullptr) {
    if (!ws) return fail(PCU_B200_INVALID_ARGUMENT, "null workspace");
    if (k <= 0) return fail(PCU_B200_INVALID_ARGUMENT, "Invalid value for k (%d) must be greater than 0.", k);
    if (prepared != nullptr) {
        if (prepared->is_f64 != (sizeof(T) == 8 ? 1 : 0)) return fail(PCU_B200_INVALID_ARGUMENT, "the prepared cloud has another precision than the points");
        if (prepared->device != ws->device) return fail(PCU_B200_INVALID_ARGUMENT, "the prepared cloud lives on device %d, the workspace on %d", prepared->device, ws->device);
        dataset = (const T*)prepared->raw;
        m = prepared->n;
    }
    PCU_TRY(check_cloud_args<T>(query, n, dataset, m));
    if (!out_dist || !out_idx) return fail(PCU_B200_INVALID_ARGUMENT, "null output pointer");
    if ((double)n * (double)k >= 9e18) return fail(PCU_B200_INVALID_ARGUMENT, "n * k overflows");
    PCU_ON_DEVICE(ws);

    PlanSpec<T> spec;
    spec.a = query; spec.n = n; spec.b = dataset; spec.m = m;
    spec.nsweeps = 1; spec.k = k; spec.squared = squared; spec.want_out = true;
    spec.occupancy = occupancy_for(ws, k);
    spec.binning = ws->opts.binning;
    spec.out_dist = out_dist; spec.out_idx = out_idx;
    const int leaf = ws->opts.max_points_per_leaf > 0 ? ws->opts.max_points_per_leaf : 10;
    // a prepared cloud that owns the reference tree (same leaf size) spares the call the build
    const bool own_tree = prepared != nullptr && prepared->leaf == leaf && ws->opts.disable_tie_replay == 0;
    spec.replay_points = (ws->opts.disable_tie_replay == 1 || own_tree) ? 0 : m;
    spec.prepared_second = prepared != nullptr;
    Plan<T> plan;
    PCU_TRY(prepare_plan(ws, plan, spec, stream));
    if (prepared != nullptr) plan.cv.v[1] = cloud_desc<T>(prepared);   // a single pair: descriptors travel by value
    mark(ws, 0, stream);
    PCU_TRY(upload_descriptors(plan, stream));
    mark(ws, 1, stream);
    PCU_TRY(enqueue_binning(ws, plan, stream, nullptr, prepared != nullptr));
    const unsigned qblocks = (unsigned)((n + kThreads - 1) / kThreads);
    if (k == 1) {
        PCU_LAUNCH_CS(nn1_kernel, dim3(qblocks, 1), kThreads, true, false);
        mark(ws, 6, stream);
        PCU_LAUNCH_CS(nn1_far_kernel, dim3(plan.far_blocks, 1), kThreads, true, false);
        PCU_LAUNCH_CS(nn1_vfar_kernel, dim3(plan.far_blocks, 1), kThreads, true, false);
        mark(ws, 7, stream);
    } else if (k <= 32) {
        // thread-per-query lists in registers (capacity = next power of two), warp pass for the rest
        if (k <= 4)       PCU_LAUNCH_CS(knn_thread_kernel, dim3(qblocks, 1), kThreads, 4);
        else if (k <= 8)  PCU_LAUNCH_CS(knn_thread_kernel, dim3(qblocks, 1), kThreads, 8);
        else if (k <= 16) PCU_LAUNCH_CS(knn_thread_kernel, dim3(qblocks, 1), kThreads, 16);
        else              PCU_LAUNCH_CS(knn_thread_kernel, dim3(qblocks, 1), kThreads, 32);
        mark(ws, 6, stream);
        PCU_LAUNCH_CS(knn_warp_kernel, dim3(plan.far_blocks, 1), kThreads);
        PCU_LAUNCH_CS(knn_descend_kernel, dim3(plan.far_blocks, 1), kThreads, false);
        mark(ws, 7, stream);
    } else {
        // large k: generic path, every query descends the occupancy pyramid
        PCU_LAUNCH_CS(pyramid_build_kernel, dim3(1, 1), kThreads);
        PCU_LAUNCH_CS(knn_descend_kernel, dim3(std::min<unsigned>(qblocks, 2368u), 1), kThreads, true);
        mark(ws, 6, stream);
        mark(ws, 7, stream);
    }
    if (own_tree) {
        KdReplayBuffers<T>& tree = cloud_tree<T>(prepared);
        const int rs = enqueue_tie_replay_prebuilt<T>(tree, query, dataset, k, squared, plan.args.sweep[0].tie_list,
                                                      plan.args.sweep[0].counters + 1, n, out_dist, out_idx, stream, g_launches);
        if (rs != PCU_B200_OK) return fail(rs, "tie replay failed: %s", cudaGetErrorString(cudaGetLastError()));
        ws->replay_overflows = tree.overflows;
    } else if (ws->opts.disable_tie_replay != 1) {
        const int rs = enqueue_tie_replay<T>(plan.replay, query, dataset, m, k, squared, leaf, plan.args.sweep[0].tie_list,
                                             plan.args.sweep[0].counters + 1, n, out_dist, out_idx, ws->opts.disable_tie_replay, stream, g_launches);
        if (rs != PCU_B200_OK) return fail(rs, "tie replay failed: %s", cudaGetErrorString(cudaGetLastError()));
        ws->replay_overflows = plan.replay.overflows;
    } else {
        ws->replay_overflows = nullptr;
    }
    if (out_n_tied) {
        PCU_LAUNCH(widen_counter_kernel, 1, 1, stream, plan.args.sweep[0].counters + 1, out_n_tied);
    }
    mark(ws, 8, stream);
    return PCU_B200_OK;
}

// ---- fused k = 1 statistics -------------------------------------------------------------------
// nsweeps == 1: query -> dataset.  nsweeps == 2: x -> y and y -> x over the same two binned clouds.

template <typename T>
int stats_device(pcu_b200_workspace* ws, const T* a, long long n, const T* b, long long m, bool both,
                 pcu_b200_nn_stats* out_stats, T* out_value, cudaStream_t stream, const cudaEvent_t* ready = nullptr,
                 const pcu_b200_cloud* prepared = nullptr, const std::function<int()>* between = nullptr) {
    if (!ws) return fail(PCU_B200_INVALID_ARGUMENT, "null workspace");
    if (prepared != nullptr) {
        if (prepared->is_f64 != (sizeof(T) == 8 ? 1 : 0)) return fail(PCU_B200_INVALID_ARGUMENT, "the prepared cloud has another precision than the points");
        if (prepared->device != ws->device) return fail(PCU_B200_INVALID_ARGUMENT, "the prepared cloud lives on device %d, the workspace on %d", prepared->device, ws->device);
        b = (const T*)prepared->raw;
        m = prepared->n;
    }
    PCU_TRY(check_cloud_args<T>(a, n, b, m));
    if (!out_stats) return fail(PCU_B200_INVALID_ARGUMENT, "null output pointer");
    PCU_ON_DEVICE(ws);
    const int ns = both ? 2 : 1;
    PlanSpec<T> spec;
    spec.a = a; spec.n = n; spec.b = b; spec.m = m;
    spec.nsweeps = ns; spec.k = 1; spec.want_stats = true;
    spec.occupancy = occupancy_for(ws, 1);
    spec.binning = ws->opts.binning;
    spec.stats = out_stats;
    spec.value_out = both ? out_value : nullptr;
    spec.prepared_second = prepared != nullptr;
    Plan<T> plan;
    PCU_TRY(prepare_plan(ws, plan, spec, stream));
    if (prepared != nullptr) plan.cv.v[1] = cloud_desc<T>(prepared);   // a single pair: descriptors travel by value
    mark(ws, 0, stream);
    PCU_TRY(upload_descriptors(plan, stream));
    mark(ws, 1, stream);
    PCU_TRY(enqueue_binning(ws, plan, stream, ready, prepared != nullptr, between));
    const unsigned qblocks = (unsigned)((std::max(n, m) + kThreads - 1) / kThreads);
    PCU_LAUNCH_CS(nn1_kernel, dim3(qblocks, ns), kThreads, false, true);
    mark(ws, 6, stream);
    PCU_LAUNCH_CS(nn1_far_kernel, dim3(plan.far_blocks, ns), kThreads, false, true);
    PCU_LAUNCH_CS(nn1_vfar_kernel, dim3(plan.far_blocks, ns), kThreads, false, true);
    mark(ws, 7, stream);
    mark(ws, 8, stream);
    return PCU_B200_OK;
}

// ---- Hausdorff witness under ties ---------------------------------------------------------------
template <typename T>
int resolve_witness_device(pcu_b200_workspace* ws, const T* query, long long n, const T* dataset, long long m,
                           pcu_b200_nn_stats* stats, cudaStream_t stream) {
    if (!ws) return fail(PCU_B200_INVALID_ARGUMENT, "null workspace");
    PCU_TRY(check_cloud_args<T>(query, n, dataset, m));
    if (!stats) return fail(PCU_B200_INVALID_ARGUMENT, "null stats pointer");
    PCU_ON_DEVICE(ws);
    // the arena is re-carved in stream order: the sweep that produced `stats` has been enqueued before us
    KdReplayBuffers<T> rb;
    Carver measure(nullptr);
    rb.carve(measure, m);
    PCU_TRY(ensure_arena(ws, measure.off, stream));
    Carver cv(ws->arena);
    rb.carve(cv, m);
    const int leaf = ws->opts.max_points_per_leaf > 0 ? ws->opts.max_points_per_leaf : 10;
    const int rs = enqueue_witness_replay<T>(rb, query, n, dataset, m, leaf, stats, stream, g_launches);
    if (rs != PCU_B200_OK) return fail(rs, "witness replay failed: %s", cudaGetErrorString(cudaGetLastError()));
    return PCU_B200_OK;
}

// ---- normals from k nearest neighbours (SURVEY.md 8f N1) -------------------------------------------
// Self-query top-k (the point itself is its own first neighbour, as in the reference), plane fit, optional
// orientation / filtering by view directions, order-preserving compaction of the kept points.
template <typename T>
int normals_knn_device(pcu_b200_workspace* ws, const T* points, long long n, const T* view_dirs, int k,
                       double drop_angle_threshold, long long* out_idx, T* out_normals, long long* out_count,
                       cudaStream_t stream) {
    if (!ws) return fail(PCU_B200_INVALID_ARGUMENT, "null workspace");
    if (k <= 0) return fail(PCU_B200_INVALID_ARGUMENT, "Invalid number of neighbors (%d) must be greater than 0.", k);
    if (!points || n <= 0)
        return fail(PCU_B200_INVALID_ARGUMENT, "Invalid point set with zero elements: points must have shape (n, 3) (got %lld rows)", n);
    if (!out_idx || !out_normals || !out_count) return fail(PCU_B200_INVALID_ARGUMENT, "null output pointer");
    PCU_ON_DEVICE(ws);
    const long long nblocks = (n + kThreads - 1) / kThreads;
    Carver measure(nullptr);
    auto carve = [&](Carver& cv, long long*& nn_idx, T*& nn_dist, T*& dense, unsigned char*& keep, unsigned*& counts) {
        nn_idx = cv.take<long long>((size_t)n * k);
        nn_dist = cv.take<T>((size_t)n * k);
        dense = cv.take<T>((size_t)3 * n);
        keep = cv.take<unsigned char>((size_t)n);
        counts = cv.take<unsigned>((size_t)nblocks);
    };
    long long* nn_idx; T *nn_dist, *dense; unsigned char* keep; unsigned* counts;
    carve(measure, nn_idx, nn_dist, dense, keep, counts);
    PCU_TRY(adopt_stream(ws, stream));
    PCU_TRY(grow_block(ws->aux, ws->aux_bytes, measure.off, stream, "neighbour scratch"));
    Carver cv(ws->aux);
    carve(cv, nn_idx, nn_dist, dense, keep, counts);
    PCU_TRY(knn_device<T>(ws, points, n, points, n, k, 1, nn_dist, nn_idx, nullptr, stream));
    PCU_LAUNCH((normals_knn_kernel<T>), (unsigned)nblocks, kThreads, stream, points, n, nn_idx, k, view_dirs, drop_angle_threshold, dense, keep);
    PCU_LAUNCH(keep_count_kernel, (unsigned)nblocks, kThreads, stream, keep, n, counts);
    PCU_LAUNCH(keep_offsets_kernel, 1, 1024, stream, counts, nblocks, out_count);
    PCU_LAUNCH((keep_scatter_kernel<T>), (unsigned)nblocks, kThreads, stream, keep, n, counts, dense, out_idx, out_normals);
    return PCU_B200_OK;
}

// ---- normals from all points in a ball (SURVEY.md 8f N1, the radius variant) ---------------------------
// The cloud is binned once (cells no finer than half the reach of the search, at most 8 per point), one thread per
// point walks the cells its ball touches; the compaction is the k-NN variant's.
template <typename T>
int normals_ball_device(pcu_b200_workspace* ws, const T* points, long long n, const T* view_dirs, const pcu_b200_ball_options* o,
                        long long* out_idx, T* out_normals, long long* out_count, cudaStream_t stream) {
    if (!ws) return fail(PCU_B200_INVALID_ARGUMENT, "null workspace");
    if (!o) return fail(PCU_B200_INVALID_ARGUMENT, "null options");
    // the checks of the binding, src/point_cloud_normals.cpp:316-327
    if (!(o->radius > 0.0)) return fail(PCU_B200_INVALID_ARGUMENT, "Invalid radius (%f) must be greater than 0.", o->radius);
    if (o->min_pts_per_ball < 3) return fail(PCU_B200_INVALID_ARGUMENT, "Invalid min_pts_per_ball (%d) must be greater than 3.", o->min_pts_per_ball);
    if (o->max_pts_per_ball > 0 && o->max_pts_per_ball < 3)
        return fail(PCU_B200_INVALID_ARGUMENT, "Invalid max_pts_per_ball (%d) must either be negative (no max) or a number greater than 3.", o->max_pts_per_ball);
    if (o->weight_function != 0 && o->weight_function != 1)
        return fail(PCU_B200_INVALID_ARGUMENT, "Invalid weight_function, must be one of 'constant' or 'rbf'.");
    if (!points || n <= 0)
        return fail(PCU_B200_INVALID_ARGUMENT, "Invalid point set with zero elements: points must have shape (n, 3) (got %lld rows)", n);
    PCU_TRY(check_cloud_args<T>(points, n, points, 1));
    if (!out_idx || !out_normals || !out_count) return fail(PCU_B200_INVALID_ARGUMENT, "null output pointer");
    PCU_ON_DEVICE(ws);
    PlanSpec<T> spec;
    spec.a = points; spec.n = n; spec.b = points; spec.m = 1;
    spec.nsweeps = 1; spec.k = 1;
    spec.occupancy = 0.125f;          // the cell budget; the cell size itself is held up by min_cell below
    spec.binning = 1;
    spec.prepared_second = true;      // the one-point second cloud is a dummy: only the first is binned
    Plan<T> plan;
    plan.layout(nullptr, spec);
    PCU_TRY(adopt_stream(ws, stream));
    PCU_TRY(ensure_arena(ws, plan.total, stream));
    plan.layout(ws->arena, spec);
    const double reach = std::sqrt((double)(T)o->radius);     // the search radius is a squared distance (normals.cuh)
    plan.cv.v[0].min_cell = (float)std::min(1e30, 0.5 * reach);
    plan.cv.v[0].hint_out = nullptr;
    const long long nblocks = (n + kThreads - 1) / kThreads;
    Carver measure(nullptr);
    auto carve = [&](Carver& cv, T*& dense, unsigned char*& keep, unsigned*& counts) {
        dense = cv.take<T>((size_t)3 * n);
        keep = cv.take<unsigned char>((size_t)n);
        counts = cv.take<unsigned>((size_t)nblocks);
    };
    T* dense; unsigned char* keep; unsigned* counts;
    carve(measure, dense, keep, counts);
    PCU_TRY(grow_block(ws->aux, ws->aux_bytes, measure.off, stream, "normal scratch"));
    Carver cv(ws->aux);
    carve(cv, dense, keep, counts);
    mark(ws, 0, stream);
    mark(ws, 1, stream);
    PCU_TRY(enqueue_binning(ws, plan, stream, nullptr, true));
    BallParams bp;
    bp.radius = o->radius; bp.drop_angle_threshold = o->drop_angle_threshold;
    bp.min_pts = o->min_pts_per_ball; bp.max_pts = o->max_pts_per_ball;
    bp.weight_kind = o->weight_function; bp.seed = o->seed;
    PCU_LAUNCH((cell_order_kernel<T>), (unsigned)std::min<long long>(((long long)plan.cv.v[0].cell_cap + kThreads - 1) / kThreads, 148 * 64), kThreads, stream, plan.cv.v[0]);
    PCU_LAUNCH((normals_ball_kernel<T>), (unsigned)nblocks, kThreads, stream, plan.cv.v[0], view_dirs, bp, dense, keep);
    mark(ws, 6, stream);
    PCU_LAUNCH(keep_count_kernel, (unsigned)nblocks, kThreads, stream, keep, n, counts);
    PCU_LAUNCH(keep_offsets_kernel, 1, 1024, stream, counts, nblocks, out_count);
    PCU_LAUNCH((keep_scatter_kernel<T>), (unsigned)nblocks, kThreads, stream, keep, n, counts, dense, out_idx, out_normals);
    mark(ws, 7, stream);
    mark(ws, 8, stream);
    return PCU_B200_OK;
}

// ---- duplicate removal (SURVEY.md 8f N2, src/remove_duplicates.cpp) ----------------------------------------
// Stable LSD radix sort of `n` records between two buffers; returns the buffer holding the sorted records.
template <typename Rec>
int radix_sort_records(Rec* a, Rec* b, long long n, int words, unsigned* hist, unsigned long long* totals, unsigned* base, int* constant,
                       cudaStream_t stream, Rec** sorted) {
    const unsigned ntiles = (unsigned)((n + kSortTile - 1) / kSortTile);
    const int bits = (int)sizeof(a->key[0]) * 8;
    Rec *in = a, *out = b;
    for (int w = words - 1; w >= 0; --w)          // least significant word first
        for (int shift = 0; shift < bits; shift += 8) {
            PCU_LAUNCH((sort_hist_kernel<Rec>), ntiles, kSortThreads, stream, (const Rec*)in, n, w, shift, hist, ntiles);
            PCU_LAUNCH(sort_scan_rows, kSortBins, kSortThreads, stream, hist, ntiles, totals);
            PCU_LAUNCH(sort_scan_bins, 1, kSortBins, stream, (const unsigned long long*)totals, n, base, constant);
            PCU_LAUNCH((sort_scatter_kernel<Rec>), ntiles, kSortThreads, stream, (const Rec*)in, out, n, w, shift, (const unsigned*)hist, ntiles,
                       (const unsigned*)base, (const int*)constant);
            std::swap(in, out);
        }
    *sorted = in;
    return PCU_B200_OK;
}

// faces == nullptr: points only.  out_pts (n, 3), out_svi (n) and out_faces (nf, cols) are sized for the worst case;
// out_counts[0] = unique points, [1] = surviving faces, [2] = faces with a corner out of range (an error for the caller).
template <typename T, typename I>
int dedup_device(pcu_b200_workspace* ws, const T* pts, long long n, double epsilon, const I* faces, long long nf, int cols,
                 T* out_pts, int* out_svi, int* out_svj, I* out_faces, long long* out_counts, cudaStream_t stream) {
    using Rec = typename DedupRec<T>::type;
    if (!ws) return fail(PCU_B200_INVALID_ARGUMENT, "null workspace");
    if (!pts || n <= 0) return fail(PCU_B200_INVALID_ARGUMENT, "points must be a non-empty (n, 3) array");
    if (n >= 0x7fffffffLL) return fail(PCU_B200_INVALID_ARGUMENT, "point cloud too large (%lld rows)", n);
    if (!out_pts || !out_svi || !out_svj || !out_counts) return fail(PCU_B200_INVALID_ARGUMENT, "null output pointer");
    if (faces != nullptr && (nf < 0 || cols <= 0 || cols > 16 || (nf > 0 && !out_faces)))
        return fail(PCU_B200_INVALID_ARGUMENT, "faces must be an (m, c) array with 1 <= c <= 16");
    if (nf >= 0x7fffffffLL) return fail(PCU_B200_INVALID_ARGUMENT, "too many faces (%lld)", nf);
    PCU_ON_DEVICE(ws);
    const long long nblocks = (n + kThreads - 1) / kThreads;
    const long long fblocks = faces ? (nf + kThreads - 1) / kThreads : 0;
    const unsigned ntiles = (unsigned)((n + kSortTile - 1) / kSortTile);
    Carver measure(nullptr);
    struct Scratch { Rec *a, *b; unsigned* hist; unsigned long long* totals; unsigned* base; int* constant; unsigned char* head;
                     unsigned* counts; unsigned char* fkeep; unsigned* fcounts; unsigned* bad; } sc;
    auto carve = [&](Carver& cv) {
        sc.a = cv.take<Rec>((size_t)n);
        sc.b = cv.take<Rec>((size_t)n);
        sc.hist = cv.take<unsigned>((size_t)kSortBins * ntiles);
        sc.totals = cv.take<unsigned long long>(kSortBins);
        sc.base = cv.take<unsigned>(kSortBins);
        sc.constant = cv.take<int>(1);
        sc.head = cv.take<unsigned char>((size_t)n);
        sc.counts = cv.take<unsigned>((size_t)nblocks);
        sc.fkeep = cv.take<unsigned char>((size_t)std::max<long long>(1, nf));
        sc.fcounts = cv.take<unsigned>((size_t)std::max<long long>(1, fblocks));
        sc.bad = cv.take<unsigned>(1);
    };
    carve(measure);
    PCU_TRY(ensure_arena(ws, measure.off, stream));
    Carver cv(ws->arena);
    carve(cv);
    PCU_CUDA(cudaMemsetAsync(out_counts, 0, 3 * sizeof(long long), stream));
    PCU_LAUNCH((dedup_keys_kernel<T>), (unsigned)nblocks, kThreads, stream, pts, n, (T)epsilon, sc.a);
    Rec* sorted = nullptr;
    PCU_TRY(radix_sort_records<Rec>(sc.a, sc.b, n, 3, sc.hist, sc.totals, sc.base, sc.constant, stream, &sorted));
    PCU_LAUNCH((dedup_heads_kernel<Rec>), (unsigned)nblocks, kThreads, stream, (const Rec*)sorted, n, sc.head);
    PCU_LAUNCH(keep_count_kernel, (unsigned)nblocks, kThreads, stream, (const unsigned char*)sc.head, n, sc.counts);
    PCU_LAUNCH(keep_offsets_kernel, 1, 1024, stream, sc.counts, nblocks, out_counts);
    PCU_LAUNCH((dedup_emit_kernel<T, Rec>), (unsigned)nblocks, kThreads, stream, (const Rec*)sorted, n, (const unsigned char*)sc.head,
               (const unsigned*)sc.counts, pts, out_pts, out_svi, out_svj);
    if (faces != nullptr && nf > 0) {
        PCU_CUDA(cudaMemsetAsync(sc.bad, 0, sizeof(unsigned), stream));
        PCU_LAUNCH((dedup_faces_flag_kernel<I>), (unsigned)fblocks, kThreads, stream, faces, nf, cols, n, (const int*)out_svj, sc.fkeep, sc.bad);
        PCU_LAUNCH(keep_count_kernel, (unsigned)fblocks, kThreads, stream, (const unsigned char*)sc.fkeep, nf, sc.fcounts);
        PCU_LAUNCH(keep_offsets_kernel, 1, 1024, stream, sc.fcounts, fblocks, out_counts + 1);
        PCU_LAUNCH((dedup_faces_emit_kernel<I>), (unsigned)fblocks, kThreads, stream, faces, nf, cols, (const int*)out_svj,
                   (const unsigned char*)sc.fkeep, (const unsigned*)sc.fcounts, out_faces);
        PCU_LAUNCH(widen_counter_kernel, 1, 1, stream, sc.bad, out_counts + 2);
    }
    return PCU_B200_OK;
}

template <typename T>
int dedup_dispatch(pcu_b200_workspace* ws, const T* pts, long long n, double epsilon, const void* faces, long long nf, int cols,
                   int faces_are_i64, T* out_pts, int* out_svi, int* out_svj, void* out_faces, long long* out_counts, cudaStream_t stream) {
    if (faces_are_i64)
        return dedup_device<T, long long>(ws, pts, n, epsilon, (const long long*)faces, nf, cols, out_pts, out_svi, out_svj,
                                          (long long*)out_faces, out_counts, stream);
    return dedup_device<T, int>(ws, pts, n, epsilon, (const int*)faces, nf, cols, out_pts, out_svi, out_svj, (int*)out_faces, out_counts, stream);
}

// ---- Morton codes (SURVEY.md 8f N3) -------------------------------------------------------------------
inline unsigned blocks_for(long long n) { return (unsigned)((n + kThreads - 1) / kThreads); }

template <typename I>
int morton_encode_device(pcu_b200_workspace* ws, const I* pts, long long n, unsigned long long* out_codes, cudaStream_t stream) {
    if (!ws) return fail(PCU_B200_INVALID_ARGUMENT, "null workspace");
    if (!pts || n <= 0) return fail(PCU_B200_INVALID_ARGUMENT, "pts must be an array of shape [n, 3] but got an empty array");
    if (!out_codes) return fail(PCU_B200_INVALID_ARGUMENT, "null output pointer");
    PCU_ON_DEVICE(ws);
    PCU_LAUNCH((morton_encode_kernel<I>), blocks_for(n), kThreads, stream, pts, n, out_codes);
    return PCU_B200_OK;
}

int morton_decode_device(pcu_b200_workspace* ws, const unsigned long long* codes, long long n, int* out_pts, cudaStream_t stream) {
    if (!ws) return fail(PCU_B200_INVALID_ARGUMENT, "null workspace");
    if (!codes || n <= 0) return fail(PCU_B200_INVALID_ARGUMENT, "codes must be an array of shape [n] but got an empty array");
    if (!out_pts) return fail(PCU_B200_INVALID_ARGUMENT, "null output pointer");
    PCU_ON_DEVICE(ws);
    PCU_LAUNCH(morton_decode_kernel, blocks_for(n), kThreads, stream, codes, n, out_pts);
    return PCU_B200_OK;
}

int morton_addsub_device(pcu_b200_workspace* ws, const unsigned long long* a, const unsigned long long* b, long long n, int op,
                         unsigned long long* out, cudaStream_t stream) {
    if (!ws) return fail(PCU_B200_INVALID_ARGUMENT, "null workspace");
    if (!a || !b || n <= 0) return fail(PCU_B200_INVALID_ARGUMENT, "codes_1 and codes_2 must be arrays of shape [n,] but got an empty array");
    if (!out) return fail(PCU_B200_INVALID_ARGUMENT, "null output pointer");
    PCU_ON_DEVICE(ws);
    PCU_LAUNCH(morton_addsub_kernel, blocks_for(n), kThreads, stream, a, b, n, op, out);
    return PCU_B200_OK;
}

int morton_knn_device(pcu_b200_workspace* ws, const unsigned long long* codes, long long n, const unsigned long long* qcodes,
                      long long m, int k, int sort_dist, long long* out_idx, cudaStream_t stream) {
    if (!ws) return fail(PCU_B200_INVALID_ARGUMENT, "null workspace");
    if (k <= 0) return fail(PCU_B200_INVALID_ARGUMENT, "k must be greater than 0");
    if (!codes || n <= 0 || !qcodes || m <= 0) return fail(PCU_B200_INVALID_ARGUMENT, "codes must be an array of shape [n] but got an empty array");
    if ((long long)k > n) return fail(PCU_B200_INVALID_ARGUMENT, "k (%d) exceeds the number of codes (%lld): clamp it first (morton.cpp:351)", k, n);
    if (!out_idx) return fail(PCU_B200_INVALID_ARGUMENT, "null output pointer");
    PCU_ON_DEVICE(ws);
    PCU_LAUNCH(morton_knn_kernel, blocks_for(m), kThreads, stream, codes, n, qcodes, m, k, sort_dist, out_idx);
    return PCU_B200_OK;
}

// ---- prepared clouds ---------------------------------------------------------------------------------------
// Bins `points` once into a private block: the layout of an ordinary plan whose second cloud is a one-point
// dummy, with only the first cloud binned; the handle keeps that cloud's descriptor.
template <typename T>
int cloud_prepare_device(pcu_b200_workspace* ws, const T* points, long long n, pcu_b200_cloud** out, cudaStream_t stream,
                         int knn_k = 1, int leaf = 0) {
    if (!ws || !out) return fail(PCU_B200_INVALID_ARGUMENT, "null argument");
    *out = nullptr;
    if (knn_k <= 0) return fail(PCU_B200_INVALID_ARGUMENT, "Invalid value for k (%d) must be greater than 0.", knn_k);
    if (leaf < 0) return fail(PCU_B200_INVALID_ARGUMENT, "max_points_per_leaf must be >= 0");
    PCU_TRY(check_cloud_args<T>(points, n, points, 1));
    PCU_ON_DEVICE(ws);
    PlanSpec<T> spec;
    spec.a = points; spec.n = n; spec.b = points; spec.m = 1;
    spec.nsweeps = 1; spec.k = 1;
    spec.occupancy = occupancy_for(ws, knn_k);   // the cell size the searches with this k want
    spec.binning = 1;                 // the grid-wide passes: the handle's buffers are global memory either way
    spec.prepared_second = true;      // (also keeps the dummy out of the one-CTA build)
    Plan<T> plan;
    plan.layout(nullptr, spec);
    const size_t raw_bytes = align_up(sizeof(T) * 3 * (size_t)n);
    size_t tree_bytes = 0;
    if (leaf > 0) {
        Carver measure(nullptr);
        KdReplayBuffers<T> probe;
        probe.carve(measure, n);
        tree_bytes = measure.off;
    }
    pcu_b200_cloud* c = new (std::nothrow) pcu_b200_cloud();
    if (!c) return fail(PCU_B200_OUT_OF_MEMORY, "out of host memory");
    c->device = ws->device; c->is_f64 = sizeof(T) == 8 ? 1 : 0; c->n = n; c->bytes = plan.total + raw_bytes + tree_bytes;
    c->knn_k = knn_k;
    cudaError_t e = cudaMalloc((void**)&c->block, c->bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        delete c;
        return fail(PCU_B200_OUT_OF_MEMORY, "cudaMalloc of %zu bytes for a prepared cloud failed: %s", plan.total + raw_bytes, cudaGetErrorString(e));
    }
    T* raw_copy = reinterpret_cast<T*>(c->block + plan.total);
    auto bail = [&](int status) { cudaFree(c->block); delete c; return status; };
    if (cudaMemcpyAsync(raw_copy, points, sizeof(T) * 3 * n, cudaMemcpyDeviceToDevice, stream) != cudaSuccess)
        return bail(fail(PCU_B200_CUDA_ERROR, "copy of the points failed: %s", cudaGetErrorString(cudaGetLastError())));
    spec.a = raw_copy; spec.b = raw_copy;
    plan.layout(c->block, spec);
    const int st = enqueue_binning(ws, plan, stream, nullptr, true);
    if (st != PCU_B200_OK) return bail(st);
    if (leaf > 0) {   // the full reference tree, once: k-NN calls against the handle only replay their tied rows on it
        Carver cv(c->block + plan.total + raw_bytes);
        KdReplayBuffers<T>& tree = cloud_tree<T>(c);
        tree.carve(cv, n);
        const int ts = build_kd_replica<T>(tree, raw_copy, n, leaf, nullptr, KdPrune<T>{}, stream, g_launches);
        if (ts != PCU_B200_OK) return bail(fail(ts, "building the reference tree failed: %s", cudaGetErrorString(cudaGetLastError())));
        c->leaf = leaf;
    }
    Cloud<T> d = plan.cv.v[0];
    d.hint_out = nullptr;             // a prepared cloud takes no part in the grid-sizing feedback
    if (sizeof(T) == 8) std::memcpy(&c->desc64, &d, sizeof d); else std::memcpy(&c->desc32, &d, sizeof d);
    c->raw = raw_copy;
    *out = c;
    return PCU_B200_OK;
}

// ---- voxel-grid down-sampling (SURVEY.md 8f N2) -----------------------------------------------------------
template <typename T, typename A>
int voxel_downsample_device(pcu_b200_workspace* ws, const T* pts, long long n, const A* attr, int attr_cols, const double size[3],
                            const double min_bound[3], const double max_bound[3], int min_points, T* out_pts, A* out_attr,
                            int* out_counts, long long* out_rows, cudaStream_t stream) {
    if (!ws) return fail(PCU_B200_INVALID_ARGUMENT, "null workspace");
    if (!pts || n <= 0) return fail(PCU_B200_INVALID_ARGUMENT, "points must be a non-empty (n, 3) array");
    if (n >= 0x7fffffffLL) return fail(PCU_B200_INVALID_ARGUMENT, "point cloud too large (%lld rows)", n);
    if (!out_pts || !out_rows || attr_cols < 0 || (attr_cols > 0 && (!attr || !out_attr)))
        return fail(PCU_B200_INVALID_ARGUMENT, "null pointer");
    VoxelGrid<T> g;
    for (int a = 0; a < 3; ++a) {   // src/sample_point_cloud.cpp:175-182, in the cloud's precision like the reference's casts (:346-354)
        g.size[a] = (T)size[a];
        g.min_bound[a] = (T)min_bound[a];
        if (g.size[a] <= (T)0) return fail(PCU_B200_INVALID_ARGUMENT, "Voxel size is negative");
        if (g.size[a] * (T)2147483647 < (T)max_bound[a] - g.min_bound[a]) return fail(PCU_B200_INVALID_ARGUMENT, "Voxel size is too small");
    }
    PCU_ON_DEVICE(ws);
    const long long nblocks = (n + kThreads - 1) / kThreads;
    unsigned slots = 64;
    while ((long long)slots < 2 * n) slots <<= 1;     // load factor <= 1/2
    Carver measure(nullptr);
    auto carve = [&](Carver& cv, int*& table, VoxelAcc*& acc, int*& slot_of, double*& attr_sum, unsigned char*& keep, unsigned*& counts) {
        table = cv.take<int>(slots);
        acc = cv.take<VoxelAcc>(slots);
        slot_of = cv.take<int>((size_t)n);
        attr_sum = cv.take<double>((size_t)slots * (attr_cols > 0 ? attr_cols : 0) + 1);
        keep = cv.take<unsigned char>((size_t)n);
        counts = cv.take<unsigned>((size_t)nblocks);
    };
    int *table, *slot_of; VoxelAcc* acc; double* attr_sum; unsigned char* keep; unsigned* counts;
    carve(measure, table, acc, slot_of, attr_sum, keep, counts);
    PCU_TRY(ensure_arena(ws, measure.off, stream));
    Carver cv(ws->arena);
    carve(cv, table, acc, slot_of, attr_sum, keep, counts);
    PCU_LAUNCH(voxel_init_kernel, (slots + kThreads - 1) / kThreads, kThreads, stream, table, acc, slots);
    if (attr_cols > 0) PCU_CUDA(cudaMemsetAsync(attr_sum, 0, sizeof(double) * (size_t)slots * attr_cols, stream));
    PCU_LAUNCH((voxel_insert_kernel<T, A>), (unsigned)nblocks, kThreads, stream, pts, n, g, table, slots, acc, slot_of, attr, attr_cols, attr_sum);
    PCU_LAUNCH(voxel_flag_kernel, (unsigned)nblocks, kThreads, stream, slot_of, acc, n, min_points, keep);
    PCU_LAUNCH(keep_count_kernel, (unsigned)nblocks, kThreads, stream, keep, n, counts);
    PCU_LAUNCH(keep_offsets_kernel, 1, 1024, stream, counts, nblocks, out_rows);
    PCU_LAUNCH((voxel_emit_kernel<T, A>), (unsigned)nblocks, kThreads, stream, keep, n, counts, slot_of, acc, attr_sum, attr_cols, out_pts, out_attr, out_counts);
    return PCU_B200_OK;
}

template <typename T>
int voxel_downsample_dispatch(pcu_b200_workspace* ws, const T* pts, long long n, const void* attr, int attr_cols, int attr_is_f64,
                              const double size[3], const double min_bound[3], const double max_bound[3], int min_points, T* out_pts,
                              void* out_attr, int* out_counts, long long* out_rows, cudaStream_t stream) {
    if (attr_is_f64)
        return voxel_downsample_device<T, double>(ws, pts, n, (const double*)attr, attr_cols, size, min_bound, max_bound, min_points,
                                                  out_pts, (double*)out_attr, out_counts, out_rows, stream);
    return voxel_downsample_device<T, float>(ws, pts, n, (const float*)attr, attr_cols, size, min_bound, max_bound, min_points, out_pts,
                                             (float*)out_attr, out_counts, out_rows, stream);
}

// ---- Poisson-disk down-sampling (downsample_point_cloud_poisson_disk, src/sample_point_cloud.cpp:240-333) -------
template <typename T> T unordered_host(typename std::conditional<sizeof(T) == 4, uint32_t, unsigned long long>::type u) {
    using B = decltype(u);
    const B sign = (B)1 << (8 * sizeof(B) - 1);
    const B bits = (u & sign) ? (u & ~sign) : ~u;
    T v;
    std::memcpy(&v, &bits, sizeof v);
    return v;
}

// One call: the key sort and the gather into key order once, then one radius trial per value of r the target search
// asks for (a single trial without target_num_samples).  A trial enqueues binning -> cell order -> the cooperative MIS
// launch -> flags -> compaction into out_idx / out_count; the target search reads each trial's count back (one stream
// synchronisation per trial, plus one for the bounding box), the radius form does not synchronise at all.
int poisson_check_args(const pcu_b200_workspace* ws, const void* pts, long long n, double radius, int target, float tol,
                       const void* out_idx, const void* out_count) {
    if (!ws) return fail(PCU_B200_INVALID_ARGUMENT, "null workspace");
    // the checks of the binding (:265-270), then the shape rules of this library
    if (target <= 0 && radius <= 0.0) return fail(PCU_B200_INVALID_ARGUMENT, "Cannot have both num_samples <= 0 and radius <= 0");
    if (tol > 1.0 || tol <= 0.0) return fail(PCU_B200_INVALID_ARGUMENT, "sample_num_tolerance must be in (0, 1]");
    if (!pts || n <= 0) return fail(PCU_B200_INVALID_ARGUMENT, "points must be a non-empty (n, 3) array");
    if (n >= 0x7fffffffLL) return fail(PCU_B200_INVALID_ARGUMENT, "point cloud too large (%lld rows; at most 2^31 - 2 are supported)", n);
    if (!out_idx || !out_count) return fail(PCU_B200_INVALID_ARGUMENT, "null output pointer");
    return PCU_B200_OK;
}

template <typename T>
int poisson_device(pcu_b200_workspace* ws, const T* pts, long long n, double radius, int target, unsigned seed, float tol,
                   int* out_idx, long long* out_count, cudaStream_t stream) {
    using bits_t = typename Real<T>::bits_t;
    PCU_TRY(poisson_check_args(ws, pts, n, radius, target, tol, out_idx, out_count));
    PCU_ON_DEVICE(ws);
    PCU_TRY(adopt_stream(ws, stream));
    ws->poisson_trials = 0;
    if (!ws->poisson_rounds) PCU_CUDA(cudaMalloc((void**)&ws->poisson_rounds, sizeof(unsigned long long)));
    PCU_CUDA(cudaMemsetAsync(ws->poisson_rounds, 0, sizeof(unsigned long long), stream));
    const long long nblocks = (n + kThreads - 1) / kThreads;
    if (target > 0 && (long long)target >= n) {            // :279-283
        PCU_LAUNCH(poisson_all_rows_kernel, (unsigned)nblocks, kThreads, stream, n, out_idx, out_count);
        return PCU_B200_OK;
    }
    const unsigned ntiles = (unsigned)((n + kSortTile - 1) / kSortTile);
    struct Scratch { PoissonRec *a, *b; unsigned* hist; unsigned long long* totals; unsigned* base; int* constant; T* ranked; int* row_of;
                     unsigned char* state; unsigned char* keep; unsigned* counts; unsigned* counters; bits_t* box; } sc;
    auto carve = [&](Carver& cv) {
        sc.a = cv.take<PoissonRec>((size_t)n);
        sc.b = cv.take<PoissonRec>((size_t)n);
        sc.hist = cv.take<unsigned>((size_t)kSortBins * ntiles);
        sc.totals = cv.take<unsigned long long>(kSortBins);
        sc.base = cv.take<unsigned>(kSortBins);
        sc.constant = cv.take<int>(1);
        sc.ranked = cv.take<T>((size_t)3 * n);
        sc.row_of = cv.take<int>((size_t)n);
        sc.state = cv.take<unsigned char>((size_t)n);
        sc.keep = cv.take<unsigned char>((size_t)n);
        sc.counts = cv.take<unsigned>((size_t)nblocks);
        sc.counters = cv.take<unsigned>(5);           // 3 round counts + the grid barrier (poisson_mis_kernel)
        sc.box = cv.take<bits_t>(6);
    };
    Carver measure(nullptr);
    carve(measure);
    PCU_TRY(grow_block(ws->aux, ws->aux_bytes, measure.off, stream, "Poisson-disk scratch"));
    Carver cv(ws->aux);
    carve(cv);
    // the binned copy: the ranked points with a one-point dummy second cloud that is never binned (as normals_ball_device)
    PlanSpec<T> spec;
    spec.a = sc.ranked; spec.n = n; spec.b = sc.ranked; spec.m = 1;
    spec.nsweeps = 1; spec.k = 1;
    spec.occupancy = 0.125f;          // the cell budget; the cell size itself is held up by min_cell
    spec.binning = 1;
    spec.prepared_second = true;
    Plan<T> plan;
    plan.layout(nullptr, spec);
    PCU_TRY(ensure_arena(ws, plan.total, stream));
    plan.layout(ws->arena, spec);
    plan.cv.v[0].hint_out = nullptr;

    PCU_LAUNCH(poisson_keys_kernel, (unsigned)nblocks, kThreads, stream, n, seed, sc.a);
    PoissonRec* sorted = nullptr;
    PCU_TRY(radix_sort_records<PoissonRec>(sc.a, sc.b, n, 1, sc.hist, sc.totals, sc.base, sc.constant, stream, &sorted));
    PCU_LAUNCH((poisson_gather_kernel<T>), (unsigned)nblocks, kThreads, stream, (const PoissonRec*)sorted, n, pts, sc.ranked, sc.row_of);

    int mis_blocks = 0;
    {
        int sms = 0, fit = 0;
        PCU_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ws->device));
        PCU_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit, poisson_mis_kernel<T>, kThreads, 0));
        mis_blocks = (int)std::max<long long>(1, std::min<long long>(nblocks, (long long)std::max(1, fit) * sms));
    }
    auto trial = [&](T r) -> int {
        ++ws->poisson_trials;
        const T r2 = r * r;                                 // rr = r * r on a Scalar r (:72)
        if (!(r2 > (T)0)) {                                 // nothing conflicts (also a NaN radius)
            PCU_LAUNCH(poisson_all_rows_kernel, (unsigned)nblocks, kThreads, stream, n, out_idx, out_count);
            return PCU_B200_OK;
        }
        plan.cv.v[0].min_cell = (float)std::min(1e30, 0.5 * std::sqrt((double)r2));
        PCU_TRY(enqueue_binning(ws, plan, stream, nullptr, true));
        PCU_LAUNCH((cell_order_kernel<T>), (unsigned)std::min<long long>(((long long)plan.cv.v[0].cell_cap + kThreads - 1) / kThreads, 148 * 64),
                   kThreads, stream, plan.cv.v[0]);
        PCU_CUDA(cudaMemsetAsync(sc.state, 0, (size_t)n, stream));
        PCU_CUDA(cudaMemsetAsync(sc.counters, 0, 5 * sizeof(unsigned), stream));
        Cloud<T> cl = plan.cv.v[0];
        T rr = r2;
        unsigned long long* rounds = ws->poisson_rounds;
        void* args[] = {(void*)&cl, (void*)&rr, (void*)&sc.state, (void*)&sc.counters, (void*)&rounds};
        PCU_CUDA(cudaLaunchCooperativeKernel((void*)poisson_mis_kernel<T>, dim3(mis_blocks), dim3(kThreads), args, 0, stream));
        g_launches.fetch_add(1, std::memory_order_relaxed);
        PCU_LAUNCH(poisson_flag_kernel, (unsigned)nblocks, kThreads, stream, (const unsigned char*)sc.state, (const int*)sc.row_of, n, sc.keep);
        PCU_LAUNCH(keep_count_kernel, (unsigned)nblocks, kThreads, stream, (const unsigned char*)sc.keep, n, sc.counts);
        PCU_LAUNCH(keep_offsets_kernel, 1, 1024, stream, sc.counts, nblocks, out_count);
        PCU_LAUNCH(poisson_scatter_kernel, (unsigned)nblocks, kThreads, stream, (const unsigned char*)sc.keep, n, (const unsigned*)sc.counts, out_idx);
        return PCU_B200_OK;
    };
    if (target <= 0) return trial((T)radius);

    // target_num_samples > 0: the search of :285-326, operation for operation in the cloud's precision; every trial's
    // sample count is read back before the next radius is chosen
    long long* host_count = reinterpret_cast<long long*>(ws->host_slot);
    auto run = [&](T r, long long& count) -> int {
        PCU_TRY(trial(r));
        PCU_CUDA(cudaMemcpyAsync(host_count, out_count, sizeof(long long), cudaMemcpyDeviceToHost, stream));
        PCU_CUDA(cudaStreamSynchronize(stream));
        count = *host_count;
        return PCU_B200_OK;
    };
    const unsigned long long num_min = (unsigned long long)(int)((T)target * (T)(1.0f - tol));
    const unsigned long long num_max = (unsigned long long)(int)((T)target * (T)(1.0f + tol));
    PCU_CUDA(cudaMemsetAsync(sc.box, 0xff, 3 * sizeof(bits_t), stream));
    PCU_CUDA(cudaMemsetAsync(sc.box + 3, 0, 3 * sizeof(bits_t), stream));
    PCU_LAUNCH((poisson_bbox_kernel<T>), (unsigned)std::min<long long>(nblocks, 4 * 148), kThreads, stream, pts, n, sc.box);
    bits_t* host_box = reinterpret_cast<bits_t*>(ws->host_slot + 64);
    PCU_CUDA(cudaMemcpyAsync(host_box, sc.box, 6 * sizeof(bits_t), cudaMemcpyDeviceToHost, stream));
    PCU_CUDA(cudaStreamSynchronize(stream));
    T ext[3];
    for (int a = 0; a < 3; ++a) ext[a] = unordered_host<T>(host_box[3 + a]) - unordered_host<T>(host_box[a]);
    const T sq01 = ext[0] * ext[0] + ext[1] * ext[1];
    const T bbsize = std::sqrt(sq01 + ext[2] * ext[2]);    // (bmax - bmin).norm()
    T rmin = (T)((double)bbsize / 50.0), rmax = (T)((double)bbsize / 50.0);
    long long count = 0;
    do {
        rmin = (T)((double)rmin / 2.0);
        PCU_TRY(run(rmin, count));
    } while ((unsigned long long)count < (unsigned long long)target);
    // (the reference never ends this loop when bbsize is 0 or not finite -- the radius cannot grow: stop there)
    do {
        rmax = (T)((double)rmax * 2.0);
        PCU_TRY(run(rmax, count));
    } while ((unsigned long long)count > (unsigned long long)target && (T)((double)rmax * 2.0) > rmax);
    int iter = 0;
    while (iter < 20 && ((unsigned long long)count < num_min || (unsigned long long)count > num_max)) {
        iter += 1;
        const T cur = (T)((double)(T)(rmin + rmax) / 2.0);
        PCU_TRY(run(cur, count));
        if (count > (long long)target) rmin = cur;
        if (count < (long long)target) rmax = cur;
    }
    return PCU_B200_OK;
}

// ---- dense pairwise distances, Sinkhorn (SURVEY.md 8f N4) ------------------------------------------------
template <typename T>
int pairwise_device(pcu_b200_workspace* ws, const T* a, const T* b, long long nb, long long n, long long m, int d, int norm_kind,
                    double p, T* out, cudaStream_t stream) {
    if (!ws) return fail(PCU_B200_INVALID_ARGUMENT, "null workspace");
    if (!a || !b || !out) return fail(PCU_B200_INVALID_ARGUMENT, "null pointer");
    if (nb <= 0 || n <= 0 || m <= 0 || d <= 0) return fail(PCU_B200_INVALID_ARGUMENT, "Invalid shape: a and b must be [m, n, d] or [n, d] with positive sizes");
    if (norm_kind < kNorm2 || norm_kind > kNormP) return fail(PCU_B200_INVALID_ARGUMENT, "unknown norm");
    if (nb > 65535 || n > 65535) return fail(PCU_B200_INVALID_ARGUMENT, "pairwise_distances: at most 65535 batches and rows per launch");
    PCU_ON_DEVICE(ws);
    PCU_LAUNCH((pairwise_kernel<T>), dim3(blocks_for(m), (unsigned)n, (unsigned)nb), kThreads, stream, a, b, n, m, d, norm_kind, p, out);
    return PCU_B200_OK;
}

// a: (nb, n) weights, b: (nb, m) weights, M: (nb, n, m) costs -> P: (nb, n, m); out_cost (nb) fp64 = sum P * M, or null;
// out_iters: device int32, iterations run (or null).  No host synchronisation: the iteration's three kernels are
// enqueued max_iters times and return at once after the convergence test has passed on the device.
template <typename T>
int sinkhorn_device(pcu_b200_workspace* ws, const T* a, const T* b, const T* M, long long nb, long long n, long long m, double eps,
                    int max_iters, double stop_thresh, T* out_P, double* out_cost, int* out_iters, cudaStream_t stream) {
    if (!ws) return fail(PCU_B200_INVALID_ARGUMENT, "null workspace");
    if (!a || !b || !M || !out_P) return fail(PCU_B200_INVALID_ARGUMENT, "null pointer");
    if (nb <= 0 || n <= 0 || m <= 0) return fail(PCU_B200_INVALID_ARGUMENT, "Got unexpected shape for M, should be [nb, m, n] with positive sizes");
    if (nb > 65535 || n > 65535) return fail(PCU_B200_INVALID_ARGUMENT, "sinkhorn: at most 65535 batches and rows per launch");
    if (max_iters < 0) return fail(PCU_B200_INVALID_ARGUMENT, "max_iters must be >= 0");
    PCU_ON_DEVICE(ws);
    Carver measure(nullptr);
    auto carve = [&](Carver& cv, T*& u, T*& v, double*& eu, double*& ev, int*& flags) {
        u = cv.take<T>((size_t)nb * n);
        v = cv.take<T>((size_t)nb * m);
        eu = cv.take<double>((size_t)nb);
        ev = cv.take<double>((size_t)nb);
        flags = cv.take<int>(2);   // [0] done, [1] iterations
    };
    T *u, *v; double *eu, *ev; int* flags;
    carve(measure, u, v, eu, ev, flags);
    PCU_TRY(ensure_arena(ws, measure.off, stream));
    Carver cv(ws->arena);
    carve(cv, u, v, eu, ev, flags);
    PCU_CUDA(cudaMemsetAsync(ws->arena, 0, measure.off, stream));   // u = v = 0 (:101-102), accumulators, flags
    if (out_cost) PCU_CUDA(cudaMemsetAsync(out_cost, 0, sizeof(double) * nb, stream));
    const T e = (T)eps;
    for (int it = 0; it < max_iters; ++it) {
        PCU_LAUNCH((sinkhorn_half_kernel<T, false>), dim3((unsigned)n, (unsigned)nb), kThreads, stream, M, a, v, u, n, m, e, eu, flags);
        PCU_LAUNCH((sinkhorn_half_kernel<T, true>), dim3((unsigned)((m + 31) / 32), (unsigned)nb), kThreads, stream, M, b, u, v, m, n, e, ev, flags);
        PCU_LAUNCH(sinkhorn_check_kernel, 1, kThreads, stream, eu, ev, nb, stop_thresh, flags, flags + 1);
    }
    PCU_LAUNCH((sinkhorn_plan_kernel<T>), dim3(blocks_for(m), (unsigned)n, (unsigned)nb), kThreads, stream, M, u, v, n, m, e, out_P, out_cost);
    if (out_iters) PCU_CUDA(cudaMemcpyAsync(out_iters, flags + 1, sizeof(int), cudaMemcpyDeviceToDevice, stream));
    return PCU_B200_OK;
}

// ---- batched Chamfer ---------------------------------------------------------------------------
template <typename T>
int batched_chamfer_device(pcu_b200_workspace* ws, const T* x, const T* y, long long batch, long long n, long long m,
                           T* out_per_pair, double* out_sum, cudaStream_t stream) {
    if (!ws) return fail(PCU_B200_INVALID_ARGUMENT, "null workspace");
    if (batch <= 0) return fail(PCU_B200_INVALID_ARGUMENT, "batch must be positive (got %lld)", batch);
    PCU_TRY(check_cloud_args<T>(x, n, y, m));
    if (!out_per_pair && !out_sum) return fail(PCU_B200_INVALID_ARGUMENT, "null output pointer");
    PCU_ON_DEVICE(ws);
    // gridDim.y carries the cloud / sweep index: at most 65535, i.e. 32767 pairs per slice
    const long long slice = 16384;
    for (long long first = 0; first < batch; first += slice) {
        const long long B = std::min(slice, batch - first);
        PlanSpec<T> spec;
        spec.batch = B;
        spec.a = x + first * 3 * n; spec.n = n; spec.b = y + first * 3 * m; spec.m = m;
        spec.nsweeps = 2; spec.k = 1; spec.want_stats = true;
        spec.occupancy = occupancy_for(ws, 1);
        spec.binning = ws->opts.binning;
        Plan<T> plan;
        PCU_TRY(prepare_plan(ws, plan, spec, stream));
        mark(ws, 0, stream);
        PCU_TRY(upload_descriptors(plan, stream));
        mark(ws, 1, stream);
        PCU_TRY(enqueue_binning(ws, plan, stream));
        const unsigned qblocks = (unsigned)((std::max(n, m) + kThreads - 1) / kThreads);
        PCU_LAUNCH_CS(nn1_kernel, dim3(qblocks, plan.nsweeps_total), kThreads, false, true);
        mark(ws, 6, stream);
        PCU_LAUNCH_CS(nn1_far_kernel, dim3(plan.far_blocks, plan.nsweeps_total), kThreads, false, true);
        PCU_LAUNCH_CS(nn1_vfar_kernel, dim3(plan.far_blocks, plan.nsweeps_total), kThreads, false, true);
        mark(ws, 7, stream);
        PCU_LAUNCH(chamfer_value_kernel<T>, 1, kThreads, stream, plan.d_stats, B,
                   out_per_pair ? out_per_pair + first : (T*)nullptr, out_sum, first > 0 ? 1 : 0);
        mark(ws, 8, stream);
    }
    return PCU_B200_OK;
}

}  // namespace

// =================================================================================================
extern "C" {

int pcu_b200_abi_version(void) { return PCU_B200_ABI_VERSION; }
const char* pcu_b200_last_error(void) { return g_error.c_str(); }
int64_t pcu_b200_launch_count(void) { return g_launches.load(); }

int pcu_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int usable = 0;
    for (int d = 0; d < n; ++d) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d) == cudaSuccess && major == 10) ++usable;
    }
    return usable;
}

// Which device a call that names none should run on (the reference's interface has no device argument):
// PCU_B200_DEVICE if set; else the CUDA runtime's current device when the caller has chosen one other than 0
// (torch.cuda.set_device / torch.cuda.device(...) in this thread); else LOCAL_RANK when a launcher such as
// torchrun set it and that many devices are visible; else device 0.
int pcu_b200_current_device(void) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) { cudaGetLastError(); return 0; }
    auto from_env = [&](const char* name) {
        const char* v = std::getenv(name);
        if (!v || !*v) return -1;
        char* end = nullptr;
        const long d = std::strtol(v, &end, 10);
        return (end && *end == '\0' && d >= 0 && d < count) ? (int)d : -1;
    };
    int d = from_env("PCU_B200_DEVICE");
    if (d >= 0) return d;
    int cur = 0;
    if (cudaGetDevice(&cur) != cudaSuccess) { cudaGetLastError(); cur = 0; }
    if (cur > 0) return cur;
    d = from_env("LOCAL_RANK");
    return d >= 0 ? d : 0;
}

int pcu_b200_workspace_device(const pcu_b200_workspace* ws) { return ws ? ws->device : -1; }

int pcu_b200_host_alloc(void** out_ptr, int64_t bytes) {
    if (!out_ptr || bytes <= 0) return fail(PCU_B200_INVALID_ARGUMENT, "bad argument");
    *out_ptr = nullptr;
    int device = 0;
    if (cudaGetDevice(&device) != cudaSuccess) { cudaGetLastError(); device = 0; }
    cudaError_t e;
    {
        NearDevice near(device);   // pages on the NUMA node of the calling thread's current GPU (staging.h)
        e = cudaHostAlloc(out_ptr, (size_t)bytes, cudaHostAllocPortable);
        // touch the pages while bound: placement is decided at first touch if the driver left any of it lazy
        if (e == cudaSuccess) for (size_t off = 0; off < (size_t)bytes; off += 4096) static_cast<volatile char*>(*out_ptr)[off] = 0;
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        *out_ptr = nullptr;
        return fail(PCU_B200_OUT_OF_MEMORY, "cudaHostAlloc of %lld bytes failed: %s", (long long)bytes, cudaGetErrorString(e));
    }
    return PCU_B200_OK;
}

int pcu_b200_host_free(void* ptr) {
    if (!ptr) return PCU_B200_OK;
    cudaError_t e = cudaFreeHost(ptr);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(PCU_B200_CUDA_ERROR, "cudaFreeHost failed: %s", cudaGetErrorString(e)); }
    return PCU_B200_OK;
}

int pcu_b200_workspace_create(int device, pcu_b200_workspace** out_ws) {
    if (!out_ws) return fail(PCU_B200_INVALID_ARGUMENT, "null out_ws");
    *out_ws = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(PCU_B200_NO_DEVICE, "no CUDA device visible: this library has no CPU fallback");
    }
    if (device < 0 || device >= n) return fail(PCU_B200_INVALID_ARGUMENT, "device %d out of range (0..%d)", device, n - 1);
    int major = 0, sms = 0;
    PCU_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    PCU_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    if (major != 10)
        return fail(PCU_B200_NO_DEVICE, "device %d has compute capability %d.x; this build only carries sm_100a code",
                    device, major);
    pcu_b200_workspace* ws = new (std::nothrow) pcu_b200_workspace();
    if (!ws) return fail(PCU_B200_OUT_OF_MEMORY, "out of host memory");
    ws->device = device;
    ws->sm_count = sms;
    DeviceGuard guard(device);
    if (guard.status != cudaSuccess) { delete ws; return fail(PCU_B200_CUDA_ERROR, "cudaSetDevice(%d): %s", device, cudaGetErrorString(guard.status)); }
    cudaError_t e = cudaStreamCreateWithFlags(&ws->own_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ws->copy_stream, cudaStreamNonBlocking);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&ws->arrived[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaHostAlloc((void**)&ws->host_slot, 4096, cudaHostAllocDefault);
    if (e != cudaSuccess) {
        cudaGetLastError();
        pcu_b200_workspace_destroy(ws);
        return fail(PCU_B200_CUDA_ERROR, "workspace streams / events / pinned slot: %s", cudaGetErrorString(e));
    }
    void* hint = nullptr;
    if (cudaHostAlloc(&hint, 16 * sizeof(unsigned), cudaHostAllocMapped) == cudaSuccess) {
        std::memset(hint, 0, 16 * sizeof(unsigned));
        void* dev_view = nullptr;
        if (cudaHostGetDevicePointer(&dev_view, hint, 0) == cudaSuccess) {
            ws->hint_host = (volatile unsigned*)hint;
            ws->hint_dev = (unsigned*)dev_view;
        } else {
            cudaGetLastError();
            cudaFreeHost(hint);
        }
    } else {
        cudaGetLastError();   // no feedback then; everything else works
    }
    *out_ws = ws;
    return PCU_B200_OK;
}

int pcu_b200_workspace_destroy(pcu_b200_workspace* ws) {
    if (!ws) return PCU_B200_OK;
    DeviceGuard guard(ws->device);
    cudaDeviceSynchronize();
    if (ws->arena) cudaFree(ws->arena);
    if (ws->io) cudaFree(ws->io);
    if (ws->aux) cudaFree(ws->aux);
    if (ws->poisson_rounds) cudaFree(ws->poisson_rounds);
    if (ws->handover) cudaEventDestroy(ws->handover);
    if (ws->hint_host) cudaFreeHost((void*)ws->hint_host);
    if (ws->own_stream) cudaStreamDestroy(ws->own_stream);
    if (ws->copy_stream) cudaStreamDestroy(ws->copy_stream);
    for (auto& e : ws->arrived) if (e) cudaEventDestroy(e);
    if (ws->host_slot) cudaFreeHost(ws->host_slot);
    for (auto& e : ws->marks) if (e) cudaEventDestroy(e);
    delete ws->stager;            // (the device is idle: nothing is in flight out of the ring)
    delete ws;
    return PCU_B200_OK;
}

int64_t pcu_b200_workspace_bytes(const pcu_b200_workspace* ws) {
    return ws ? (int64_t)(ws->arena_bytes + ws->io_bytes + ws->aux_bytes) : 0;
}

int pcu_b200_workspace_set_profiling(pcu_b200_workspace* ws, int enabled) {
    if (!ws) return fail(PCU_B200_INVALID_ARGUMENT, "null workspace");
    PCU_ON_DEVICE(ws);
    if (enabled && !ws->marks[0])
        for (auto& e : ws->marks) PCU_CUDA(cudaEventCreate(&e));
    ws->profiling = enabled != 0;
    ws->marks_used = 0;
    return PCU_B200_OK;
}

int pcu_b200_workspace_last_profile(pcu_b200_workspace* ws, float* out_ms, int capacity) {
    if (!ws || !out_ms) return -1;
    if (!ws->profiling || ws->marks_used < 9) return 0;
    cudaEvent_t last = ws->host_marks ? ws->marks[10] : ws->marks[8];
    if (cudaEventSynchronize(last) != cudaSuccess) { cudaGetLastError(); return -1; }
    int n = 0;
    for (; n < 8 && n < capacity; ++n) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ws->marks[n], ws->marks[n + 1]) != cudaSuccess) { cudaGetLastError(); return -1; }
        out_ms[n] = ms;
    }
    if (ws->host_marks && capacity >= 10) {   // host entry points: the copies either side of the device call
        float h2d = 0.f, d2h = 0.f;
        if (cudaEventElapsedTime(&h2d, ws->marks[9], ws->marks[0]) != cudaSuccess ||
            cudaEventElapsedTime(&d2h, ws->marks[8], ws->marks[10]) != cudaSuccess) { cudaGetLastError(); return -1; }
        out_ms[8] = h2d; out_ms[9] = d2h;
        n = 10;
    }
    return n;
}

const char* pcu_b200_profile_stage_name(int stage) {
    static const char* names[] = {PCU_STAGE_NAMES};
    return stage >= 0 && stage < 10 ? names[stage] : "";
}

int pcu_b200_workspace_grid_refinement(const pcu_b200_workspace* ws, float out_mult[2]) {
    if (!ws || !out_mult) return fail(PCU_B200_INVALID_ARGUMENT, "null argument");
    out_mult[0] = ws->cell_mult[0];
    out_mult[1] = ws->cell_mult[1];
    return PCU_B200_OK;
}

int pcu_b200_workspace_set_options(pcu_b200_workspace* ws, const pcu_b200_options* opts) {
    if (!ws || !opts) return fail(PCU_B200_INVALID_ARGUMENT, "null argument");
    if (opts->max_points_per_leaf < 0) return fail(PCU_B200_INVALID_ARGUMENT, "max_points_per_leaf must be >= 0");
    if (opts->cell_occupancy < 0.f) return fail(PCU_B200_INVALID_ARGUMENT, "cell_occupancy must be >= 0");
    if (opts->disable_tie_replay < 0 || opts->disable_tie_replay > 3)
        return fail(PCU_B200_INVALID_ARGUMENT, "disable_tie_replay must be 0 .. 3");
    if (opts->binning < 0 || opts->binning > 2) return fail(PCU_B200_INVALID_ARGUMENT, "binning must be 0, 1 or 2");
    if (opts->host_staging < 0 || opts->host_staging > 2) return fail(PCU_B200_INVALID_ARGUMENT, "host_staging must be 0, 1 or 2");
    ws->opts = *opts;
    return PCU_B200_OK;
}

int pcu_b200_knn_f32(pcu_b200_workspace* ws, const float* query, int64_t n, const float* dataset, int64_t m, int k,
                     int squared, float* out_dist, int64_t* out_idx, int64_t* out_n_tied, void* stream) {
    return knn_device<float>(ws, query, n, dataset, m, k, squared, out_dist, (long long*)out_idx,
                             (long long*)out_n_tied, (cudaStream_t)stream);
}
int pcu_b200_knn_f64(pcu_b200_workspace* ws, const double* query, int64_t n, const double* dataset, int64_t m, int k,
                     int squared, double* out_dist, int64_t* out_idx, int64_t* out_n_tied, void* stream) {
    return knn_device<double>(ws, query, n, dataset, m, k, squared, out_dist, (long long*)out_idx,
                              (long long*)out_n_tied, (cudaStream_t)stream);
}
int pcu_b200_nn_stats_f32(pcu_b200_workspace* ws, const float* query, int64_t n, const float* dataset, int64_t m,
                          pcu_b200_nn_stats* out_stats, void* stream) {
    return stats_device<float>(ws, query, n, dataset, m, false, out_stats, nullptr, (cudaStream_t)stream);
}
int pcu_b200_nn_stats_f64(pcu_b200_workspace* ws, const double* query, int64_t n, const double* dataset, int64_t m,
                          pcu_b200_nn_stats* out_stats, void* stream) {
    return stats_device<double>(ws, query, n, dataset, m, false, out_stats, nullptr, (cudaStream_t)stream);
}
int pcu_b200_resolve_witness_f32(pcu_b200_workspace* ws, const float* query, int64_t n, const float* dataset,
                                 int64_t m, pcu_b200_nn_stats* stats, void* stream) {
    return resolve_witness_device<float>(ws, query, n, dataset, m, stats, (cudaStream_t)stream);
}
int pcu_b200_resolve_witness_f64(pcu_b200_workspace* ws, const double* query, int64_t n, const double* dataset,
                                 int64_t m, pcu_b200_nn_stats* stats, void* stream) {
    return resolve_witness_device<double>(ws, query, n, dataset, m, stats, (cudaStream_t)stream);
}
int pcu_b200_chamfer_f32(pcu_b200_workspace* ws, const float* x, int64_t n, const float* y, int64_t m,
                         pcu_b200_nn_stats* out_stats, float* out_value, void* stream) {
    return stats_device<float>(ws, x, n, y, m, true, out_stats, out_value, (cudaStream_t)stream);
}
int pcu_b200_chamfer_f64(pcu_b200_workspace* ws, const double* x, int64_t n, const double* y, int64_t m,
                         pcu_b200_nn_stats* out_stats, double* out_value, void* stream) {
    return stats_device<double>(ws, x, n, y, m, true, out_stats, out_value, (cudaStream_t)stream);
}

int pcu_b200_cloud_prepare_f32(pcu_b200_workspace* ws, const float* points, int64_t n, pcu_b200_cloud** out_cloud, void* stream) {
    return cloud_prepare_device<float>(ws, points, n, out_cloud, (cudaStream_t)stream);
}
int pcu_b200_cloud_prepare_f64(pcu_b200_workspace* ws, const double* points, int64_t n, pcu_b200_cloud** out_cloud, void* stream) {
    return cloud_prepare_device<double>(ws, points, n, out_cloud, (cudaStream_t)stream);
}
int pcu_b200_cloud_prepare_knn_f32(pcu_b200_workspace* ws, const float* points, int64_t n, int k, int max_points_per_leaf,
                                   pcu_b200_cloud** out_cloud, void* stream) {
    return cloud_prepare_device<float>(ws, points, n, out_cloud, (cudaStream_t)stream, k, max_points_per_leaf > 0 ? max_points_per_leaf : 10);
}
int pcu_b200_cloud_prepare_knn_f64(pcu_b200_workspace* ws, const double* points, int64_t n, int k, int max_points_per_leaf,
                                   pcu_b200_cloud** out_cloud, void* stream) {
    return cloud_prepare_device<double>(ws, points, n, out_cloud, (cudaStream_t)stream, k, max_points_per_leaf > 0 ? max_points_per_leaf : 10);
}
int pcu_b200_knn_prepared_f32(pcu_b200_workspace* ws, const float* query, int64_t n, pcu_b200_cloud* dataset, int k, int squared,
                              float* out_dist, int64_t* out_idx, int64_t* out_n_tied, void* stream) {
    if (!dataset) return fail(PCU_B200_INVALID_ARGUMENT, "null prepared cloud");
    return knn_device<float>(ws, query, n, nullptr, 0, k, squared, out_dist, (long long*)out_idx, (long long*)out_n_tied,
                             (cudaStream_t)stream, dataset);
}
int pcu_b200_knn_prepared_f64(pcu_b200_workspace* ws, const double* query, int64_t n, pcu_b200_cloud* dataset, int k, int squared,
                              double* out_dist, int64_t* out_idx, int64_t* out_n_tied, void* stream) {
    if (!dataset) return fail(PCU_B200_INVALID_ARGUMENT, "null prepared cloud");
    return knn_device<double>(ws, query, n, nullptr, 0, k, squared, out_dist, (long long*)out_idx, (long long*)out_n_tied,
                              (cudaStream_t)stream, dataset);
}
int pcu_b200_cloud_destroy(pcu_b200_cloud* cloud) {
    if (!cloud) return PCU_B200_OK;
    DeviceGuard guard(cloud->device);
    cudaDeviceSynchronize();          // calls that use the cloud may still be queued
    if (cloud->block) cudaFree(cloud->block);
    delete cloud;
    return PCU_B200_OK;
}
int64_t pcu_b200_cloud_size(const pcu_b200_cloud* cloud) { return cloud ? cloud->n : 0; }
const void* pcu_b200_cloud_points(const pcu_b200_cloud* cloud) { return cloud ? cloud->raw : nullptr; }
int pcu_b200_chamfer_prepared_f32(pcu_b200_workspace* ws, const float* x, int64_t n, const pcu_b200_cloud* y,
                                  pcu_b200_nn_stats* out_stats, float* out_value, void* stream) {
    if (!y) return fail(PCU_B200_INVALID_ARGUMENT, "null prepared cloud");
    return stats_device<float>(ws, x, n, nullptr, 0, true, out_stats, out_value, (cudaStream_t)stream, nullptr, y);
}
int pcu_b200_chamfer_prepared_f64(pcu_b200_workspace* ws, const double* x, int64_t n, const pcu_b200_cloud* y,
                                  pcu_b200_nn_stats* out_stats, double* out_value, void* stream) {
    if (!y) return fail(PCU_B200_INVALID_ARGUMENT, "null prepared cloud");
    return stats_device<double>(ws, x, n, nullptr, 0, true, out_stats, out_value, (cudaStream_t)stream, nullptr, y);
}
int pcu_b200_nn_stats_prepared_f32(pcu_b200_workspace* ws, const float* query, int64_t n, const pcu_b200_cloud* dataset,
                                   pcu_b200_nn_stats* out_stats, void* stream) {
    if (!dataset) return fail(PCU_B200_INVALID_ARGUMENT, "null prepared cloud");
    return stats_device<float>(ws, query, n, nullptr, 0, false, out_stats, nullptr, (cudaStream_t)stream, nullptr, dataset);
}
int pcu_b200_nn_stats_prepared_f64(pcu_b200_workspace* ws, const double* query, int64_t n, const pcu_b200_cloud* dataset,
                                   pcu_b200_nn_stats* out_stats, void* stream) {
    if (!dataset) return fail(PCU_B200_INVALID_ARGUMENT, "null prepared cloud");
    return stats_device<double>(ws, query, n, nullptr, 0, false, out_stats, nullptr, (cudaStream_t)stream, nullptr, dataset);
}

int pcu_b200_voxel_downsample_f32(pcu_b200_workspace* ws, const float* points, int64_t n, const void* attrib, int attrib_cols,
                                  int attrib_is_f64, const double voxel_size[3], const double min_bound[3], const double max_bound[3],
                                  int min_points_per_voxel, float* out_points, void* out_attrib, int32_t* out_counts, int64_t* out_rows,
                                  void* stream) {
    return voxel_downsample_dispatch<float>(ws, points, n, attrib, attrib_cols, attrib_is_f64, voxel_size, min_bound, max_bound,
                                            min_points_per_voxel, out_points, out_attrib, out_counts, (long long*)out_rows, (cudaStream_t)stream);
}
int pcu_b200_voxel_downsample_f64(pcu_b200_workspace* ws, const double* points, int64_t n, const void* attrib, int attrib_cols,
                                  int attrib_is_f64, const double voxel_size[3], const double min_bound[3], const double max_bound[3],
                                  int min_points_per_voxel, double* out_points, void* out_attrib, int32_t* out_counts, int64_t* out_rows,
                                  void* stream) {
    return voxel_downsample_dispatch<double>(ws, points, n, attrib, attrib_cols, attrib_is_f64, voxel_size, min_bound, max_bound,
                                             min_points_per_voxel, out_points, out_attrib, out_counts, (long long*)out_rows, (cudaStream_t)stream);
}

int pcu_b200_poisson_disk_downsample_f32(pcu_b200_workspace* ws, const float* points, int64_t n, double radius, int target_num_samples,
                                         uint32_t seed, float sample_num_tolerance, int32_t* out_idx, int64_t* out_count, void* stream) {
    return poisson_device<float>(ws, points, n, radius, target_num_samples, seed, sample_num_tolerance, out_idx, (long long*)out_count,
                                 (cudaStream_t)stream);
}
int pcu_b200_poisson_disk_downsample_f64(pcu_b200_workspace* ws, const double* points, int64_t n, double radius, int target_num_samples,
                                         uint32_t seed, float sample_num_tolerance, int32_t* out_idx, int64_t* out_count, void* stream) {
    return poisson_device<double>(ws, points, n, radius, target_num_samples, seed, sample_num_tolerance, out_idx, (long long*)out_count,
                                  (cudaStream_t)stream);
}
int pcu_b200_debug_poisson_stats(pcu_b200_workspace* ws, int64_t out[2]) {
    if (!ws || !out) return fail(PCU_B200_INVALID_ARGUMENT, "null argument");
    PCU_ON_DEVICE(ws);
    unsigned long long rounds = 0;
    if (ws->poisson_rounds) {
        PCU_CUDA(cudaDeviceSynchronize());
        PCU_CUDA(cudaMemcpy(&rounds, ws->poisson_rounds, sizeof rounds, cudaMemcpyDeviceToHost));
    }
    out[0] = ws->poisson_trials;
    out[1] = (int64_t)rounds;
    return PCU_B200_OK;
}

int pcu_b200_pairwise_distances_f32(pcu_b200_workspace* ws, const float* a, const float* b, int64_t nb, int64_t n, int64_t m, int d,
                                    int norm_kind, double p, float* out, void* stream) {
    return pairwise_device<float>(ws, a, b, nb, n, m, d, norm_kind, p, out, (cudaStream_t)stream);
}
int pcu_b200_pairwise_distances_f64(pcu_b200_workspace* ws, const double* a, const double* b, int64_t nb, int64_t n, int64_t m, int d,
                                    int norm_kind, double p, double* out, void* stream) {
    return pairwise_device<double>(ws, a, b, nb, n, m, d, norm_kind, p, out, (cudaStream_t)stream);
}
int pcu_b200_sinkhorn_f32(pcu_b200_workspace* ws, const float* a, const float* b, const float* M, int64_t nb, int64_t n, int64_t m,
                          double eps, int max_iters, double stop_thresh, float* out_P, double* out_cost, int32_t* out_iters, void* stream) {
    return sinkhorn_device<float>(ws, a, b, M, nb, n, m, eps, max_iters, stop_thresh, out_P, out_cost, out_iters, (cudaStream_t)stream);
}
int pcu_b200_sinkhorn_f64(pcu_b200_workspace* ws, const double* a, const double* b, const double* M, int64_t nb, int64_t n, int64_t m,
                          double eps, int max_iters, double stop_thresh, double* out_P, double* out_cost, int32_t* out_iters, void* stream) {
    return sinkhorn_device<double>(ws, a, b, M, nb, n, m, eps, max_iters, stop_thresh, out_P, out_cost, out_iters, (cudaStream_t)stream);
}

int pcu_b200_morton_encode_i32(pcu_b200_workspace* ws, const int32_t* pts, int64_t n, uint64_t* out_codes, void* stream) {
    return morton_encode_device<int32_t>(ws, pts, n, (unsigned long long*)out_codes, (cudaStream_t)stream);
}
int pcu_b200_morton_encode_i64(pcu_b200_workspace* ws, const int64_t* pts, int64_t n, uint64_t* out_codes, void* stream) {
    return morton_encode_device<long long>(ws, (const long long*)pts, n, (unsigned long long*)out_codes, (cudaStream_t)stream);
}
int pcu_b200_morton_decode(pcu_b200_workspace* ws, const uint64_t* codes, int64_t n, int32_t* out_pts, void* stream) {
    return morton_decode_device(ws, (const unsigned long long*)codes, n, out_pts, (cudaStream_t)stream);
}
int pcu_b200_morton_add(pcu_b200_workspace* ws, const uint64_t* a, const uint64_t* b, int64_t n, uint64_t* out, void* stream) {
    return morton_addsub_device(ws, (const unsigned long long*)a, (const unsigned long long*)b, n, 0, (unsigned long long*)out, (cudaStream_t)stream);
}
int pcu_b200_morton_subtract(pcu_b200_workspace* ws, const uint64_t* a, const uint64_t* b, int64_t n, uint64_t* out, void* stream) {
    return morton_addsub_device(ws, (const unsigned long long*)a, (const unsigned long long*)b, n, 1, (unsigned long long*)out, (cudaStream_t)stream);
}
int pcu_b200_morton_knn(pcu_b200_workspace* ws, const uint64_t* codes, int64_t n, const uint64_t* qcodes, int64_t m, int k,
                        int sort_dist, int64_t* out_idx, void* stream) {
    return morton_knn_device(ws, (const unsigned long long*)codes, n, (const unsigned long long*)qcodes, m, k, sort_dist,
                             (long long*)out_idx, (cudaStream_t)stream);
}

int pcu_b200_normals_knn_f32(pcu_b200_workspace* ws, const float* points, int64_t n, const float* view_dirs, int k,
                             double drop_angle_threshold, int64_t* out_idx, float* out_normals, int64_t* out_count, void* stream) {
    return normals_knn_device<float>(ws, points, n, view_dirs, k, drop_angle_threshold, (long long*)out_idx, out_normals,
                                     (long long*)out_count, (cudaStream_t)stream);
}
int pcu_b200_normals_knn_f64(pcu_b200_workspace* ws, const double* points, int64_t n, const double* view_dirs, int k,
                             double drop_angle_threshold, int64_t* out_idx, double* out_normals, int64_t* out_count, void* stream) {
    return normals_knn_device<double>(ws, points, n, view_dirs, k, drop_angle_threshold, (long long*)out_idx, out_normals,
                                      (long long*)out_count, (cudaStream_t)stream);
}

int pcu_b200_normals_ball_f32(pcu_b200_workspace* ws, const float* points, int64_t n, const float* view_dirs,
                              const pcu_b200_ball_options* options, int64_t* out_idx, float* out_normals, int64_t* out_count, void* stream) {
    return normals_ball_device<float>(ws, points, n, view_dirs, options, (long long*)out_idx, out_normals, (long long*)out_count, (cudaStream_t)stream);
}
int pcu_b200_normals_ball_f64(pcu_b200_workspace* ws, const double* points, int64_t n, const double* view_dirs,
                              const pcu_b200_ball_options* options, int64_t* out_idx, double* out_normals, int64_t* out_count, void* stream) {
    return normals_ball_device<double>(ws, points, n, view_dirs, options, (long long*)out_idx, out_normals, (long long*)out_count, (cudaStream_t)stream);
}

int pcu_b200_deduplicate_f32(pcu_b200_workspace* ws, const float* points, int64_t n, double epsilon, const void* faces, int64_t n_faces,
                             int face_cols, int faces_are_i64, float* out_points, int32_t* out_svi, int32_t* out_svj, void* out_faces,
                             int64_t* out_counts, void* stream) {
    return dedup_dispatch<float>(ws, points, n, epsilon, faces, n_faces, face_cols, faces_are_i64, out_points, out_svi, out_svj, out_faces,
                                 (long long*)out_counts, (cudaStream_t)stream);
}
int pcu_b200_deduplicate_f64(pcu_b200_workspace* ws, const double* points, int64_t n, double epsilon, const void* faces, int64_t n_faces,
                             int face_cols, int faces_are_i64, double* out_points, int32_t* out_svi, int32_t* out_svj, void* out_faces,
                             int64_t* out_counts, void* stream) {
    return dedup_dispatch<double>(ws, points, n, epsilon, faces, n_faces, face_cols, faces_are_i64, out_points, out_svi, out_svj, out_faces,
                                  (long long*)out_counts, (cudaStream_t)stream);
}

int pcu_b200_debug_kd_times(pcu_b200_workspace* ws, uint64_t* out40) {
    if (!ws || !out40) return fail(PCU_B200_INVALID_ARGUMENT, "null argument");
    PCU_ON_DEVICE(ws);
    PCU_CUDA(cudaDeviceSynchronize());
    PCU_CUDA(cudaMemcpyFromSymbol(out40, g_kd_times, sizeof(unsigned long long) * 40));
    return PCU_B200_OK;
}

int pcu_b200_batched_chamfer_f32(pcu_b200_workspace* ws, const float* x, const float* y, int64_t batch, int64_t n,
                                 int64_t m, float* out_per_pair, double* out_sum, void* stream) {
    return batched_chamfer_device<float>(ws, x, y, batch, n, m, out_per_pair, out_sum, (cudaStream_t)stream);
}

}  // extern "C"

#include "host_entry.inl"
