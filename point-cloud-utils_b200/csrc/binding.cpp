// binding.cpp -- pybind11 module `_pcu_internal`: the Python-facing mirror of the two bindings the
// reference generates with numpyeigen for this path,
//     k_nearest_neighbors           /root/reference/src/point_cloud_distance.cpp:123-164
//     one_sided_hausdorff_distance  /root/reference/src/point_cloud_distance.cpp:186-234
// with the same argument names, defaults, dtype rules (float32 / float64, both clouds alike),
// shape rules ((n, 3), n > 0), error type (ValueError), int64 indices and squeezed outputs
// (tests/test_examples.py:363-368).  All computation goes through the C ABI of libpcu_b200.so
// (include/pcu_b200.h); there is no CPU implementation behind these functions.
//
// Besides the numpy entry points the module exposes raw-pointer variants (`*_device`) that the
// Python package uses for CUDA torch tensors: the caller passes data_ptr()s and a stream handle,
// nothing is copied and nothing synchronises.
#include <pybind11/pybind11.h>
#include <pybind11/numpy.h>
#include <pybind11/stl.h>

#include <algorithm>
#include <array>
#include <cstdint>
#include <map>
#include <memory>
#include <mutex>
#include <sstream>
#include <stdexcept>
#include <string>
#include <tuple>

#include "../../include/pcu_b200.h"

namespace py = pybind11;

namespace {

[[noreturn]] void raise_status(int status) {
    const std::string msg = pcu_b200_last_error();
    switch (status) {
        case PCU_B200_INVALID_ARGUMENT: throw py::value_error(msg);
        case PCU_B200_OUT_OF_MEMORY: throw std::bad_alloc();
        default: throw std::runtime_error("pcu_b200: " + msg);
    }
}
inline void check(int status) { if (status != PCU_B200_OK) raise_status(status); }

// One workspace per (device, stream): a workspace serves one stream at a time.  Calls that share a
// workspace (several Python threads on the same stream) are serialised by that workspace's own mutex:
// enqueueing is what must not interleave, the work itself is ordered by the stream.  Calls on different
// devices or streams never wait for each other.
// The numpy (host-pointer) entry points run on the workspace's private stream; they get workspaces of
// their own under the key kHostKey, so they never share scratch with a device-pointer call that may still
// be queued on one of the caller's streams (stream handle 0 is torch's default stream, not "host").
constexpr uintptr_t kHostKey = ~(uintptr_t)0;
struct Slot {
    pcu_b200_workspace* ws = nullptr;
    std::mutex busy;
};
struct Pool {
    std::mutex mu;
    std::map<std::pair<int, uintptr_t>, std::unique_ptr<Slot>> items;
    Slot& get(int device, uintptr_t stream) {
        std::lock_guard<std::mutex> lock(mu);
        auto key = std::make_pair(device, stream);
        auto it = items.find(key);
        if (it != items.end()) return *it->second;
        std::unique_ptr<Slot> slot(new Slot());
        check(pcu_b200_workspace_create(device, &slot->ws));
        Slot& ref = *slot;
        items[key] = std::move(slot);
        return ref;
    }
    void clear() {
        std::lock_guard<std::mutex> lock(mu);
        for (auto& kv : items) pcu_b200_workspace_destroy(kv.second->ws);
        items.clear();
    }
};
Pool& pool() { static Pool p; return p; }
// Released GIL + exclusive use of one workspace for the duration of one call.
struct CallScope {
    py::gil_scoped_release nogil;
    std::lock_guard<std::mutex> lock;
    explicit CallScope(Slot& slot) : nogil(), lock(slot.busy) {}
};

// Result arrays of 1 MiB and more are backed by page-locked host memory: the device-to-host copy of a large
// k-NN result into a fresh pageable numpy array is bound by page faults (~3 GB/s measured, 0.6 s for the
// 1.9 GB of BASELINE configs[3]), into pinned memory by PCIe.  Page-locking is slow itself, so blocks are
// recycled: when the numpy array that owns one is garbage-collected the block returns to this pool (at most
// kKeepBytes stay cached; anything beyond is unpinned and released).  Allocation failure or a pool over its
// budget of outstanding blocks falls back to an ordinary numpy array.
class PinnedPool {
public:
    static constexpr size_t kMinBytes = size_t(1) << 20;
    static constexpr size_t kKeepBytes = size_t(6) << 30;
    static constexpr size_t kMaxOutstanding = size_t(24) << 30;
    void* take(size_t bytes, size_t& capacity) {
        capacity = (bytes + (size_t(2) << 20) - 1) & ~((size_t(2) << 20) - 1);
        {
            std::lock_guard<std::mutex> lock(mu_);
            auto it = free_.lower_bound(capacity);
            if (it != free_.end() && it->first <= capacity + capacity / 4) {
                void* p = it->second;
                capacity = it->first;
                cached_ -= it->first;
                free_.erase(it);
                outstanding_ += capacity;
                return p;
            }
            if (outstanding_ + capacity > kMaxOutstanding) return nullptr;
            outstanding_ += capacity;
        }
        void* p = nullptr;
        if (pcu_b200_host_alloc(&p, (int64_t)capacity) != PCU_B200_OK) {
            std::lock_guard<std::mutex> lock(mu_);
            outstanding_ -= capacity;
            return nullptr;
        }
        return p;
    }
    void give(void* p, size_t capacity) {
        bool release = false;
        {
            std::lock_guard<std::mutex> lock(mu_);
            outstanding_ -= capacity;
            if (closed_ || cached_ + capacity > kKeepBytes) release = true;
            else { free_.emplace(capacity, p); cached_ += capacity; }
        }
        if (release) pcu_b200_host_free(p);
    }
    void clear(bool close) {
        std::multimap<size_t, void*> drop;
        {
            std::lock_guard<std::mutex> lock(mu_);
            drop.swap(free_);
            cached_ = 0;
            if (close) closed_ = true;
        }
        for (auto& kv : drop) pcu_b200_host_free(kv.second);
    }
private:
    std::mutex mu_;
    std::multimap<size_t, void*> free_;
    size_t cached_ = 0, outstanding_ = 0;
    bool closed_ = false;
};
PinnedPool& pinned_pool() { static PinnedPool* p = new PinnedPool(); return *p; }   // outlives late array destructors

struct PinnedBlock { void* ptr; size_t capacity; };

// A C-contiguous (rows, cols) array of T: page-locked and pool-backed when it is large, ordinary otherwise.
template <typename T>
py::array_t<T> result_array(py::ssize_t rows, py::ssize_t cols) {
    const size_t bytes = (size_t)rows * (size_t)cols * sizeof(T);
    if (bytes >= PinnedPool::kMinBytes) {
        size_t capacity = 0;
        void* p = pinned_pool().take(bytes, capacity);
        if (p != nullptr) {
            auto* block = new PinnedBlock{p, capacity};
            py::capsule owner(block, [](void* b) {
                auto* blk = static_cast<PinnedBlock*>(b);
                pinned_pool().give(blk->ptr, blk->capacity);
                delete blk;
            });
            return py::array_t<T>({rows, cols}, {(py::ssize_t)(cols * sizeof(T)), (py::ssize_t)sizeof(T)}, static_cast<T*>(p), owner);
        }
    }
    return py::array_t<T>({rows, cols});
}

// pcu.pinned_empty: an (n, 3) array of T in page-locked memory next to the current GPU, for callers who fill their
// clouds in place (what torch's pin_memory() gives, with the placement taken care of: pcu_b200_host_alloc)
template <typename T>
py::array pinned_cloud(py::ssize_t rows, py::ssize_t cols) {
    if (rows <= 0 || cols <= 0) throw py::value_error("shape must be positive");
    const size_t bytes = (size_t)rows * (size_t)cols * sizeof(T);
    void* p = nullptr;
    check(pcu_b200_host_alloc(&p, (int64_t)bytes));
    py::capsule owner(p, [](void* q) { pcu_b200_host_free(q); });
    return py::array_t<T>({rows, cols}, {(py::ssize_t)(cols * sizeof(T)), (py::ssize_t)sizeof(T)}, static_cast<T*>(p), owner);
}

struct Options { int leaf = 10; float occupancy = 0.f; int disable_replay = 0; int binning = 0; int host_staging = 0; };
Options& defaults() { static Options o; return o; }

// Validates the per-call options (with the GIL held); they are applied to the workspace inside the
// call's exclusive section so that concurrent callers cannot mix them up.
pcu_b200_options make_options(int max_points_per_leaf) {
    if (max_points_per_leaf <= 0) throw py::value_error("max_points_per_leaf must be greater than 0.");
    pcu_b200_options o{};
    o.max_points_per_leaf = max_points_per_leaf;
    o.cell_occupancy = defaults().occupancy;
    o.disable_tie_replay = defaults().disable_replay;
    o.binning = defaults().binning;
    o.host_staging = defaults().host_staging;
    return o;
}

enum class Dt { f32, f64 };

Dt common_dtype(const py::array& a, const py::array& b, const char* na, const char* nb) {
    // numpyeigen: dense_float / dense_double only, second argument npe_matches(first)
    // (point_cloud_distance.cpp:124-125, :187-188)
    const bool a32 = a.dtype().is(py::dtype::of<float>()), a64 = a.dtype().is(py::dtype::of<double>());
    if (!a32 && !a64) {
        std::ostringstream ss;
        ss << "Invalid scalar type (" << std::string(py::str(a.dtype())) << ") for argument '" << na
           << "'. Expected one of ['float32', 'float64'].";
        throw py::value_error(ss.str());
    }
    if (!b.dtype().is(a.dtype())) {
        std::ostringstream ss;
        ss << "Invalid scalar type (" << std::string(py::str(b.dtype())) << ") for argument '" << nb
           << "'. Expected it to match argument '" << na << "' which is of type " << std::string(py::str(a.dtype())) << ".";
        throw py::value_error(ss.str());
    }
    return a32 ? Dt::f32 : Dt::f64;
}

void check_shapes(const py::array& a, const py::array& b, const char* na, const char* nb) {
    auto shape_str = [](const py::array& x) {
        std::ostringstream ss;
        ss << "(";
        for (py::ssize_t i = 0; i < x.ndim(); ++i) ss << (i ? ", " : "") << x.shape(i);
        ss << ")";
        return ss.str();
    };
    if (a.ndim() != 2 || b.ndim() != 2) {
        std::ostringstream ss;
        ss << "Only 3D inputs are supported: " << na << " and " << nb << " must have shape (n, 3) and (m, 3). Got "
           << na << ".shape = " << shape_str(a) << ", " << nb << ".shape = " << shape_str(b) << ".";
        throw py::value_error(ss.str());
    }
    if (a.shape(0) == 0 || b.shape(0) == 0) {
        std::ostringstream ss;
        ss << "Invalid input set with zero elements: " << na << " and " << nb
           << " must have shape (n, 3) and (m, 3). Got " << na << ".shape = " << shape_str(a) << ", " << nb
           << ".shape = " << shape_str(b) << ".";
        throw py::value_error(ss.str());
    }
    if (a.shape(1) != 3 || b.shape(1) != 3) {
        std::ostringstream ss;
        ss << "Only 3D inputs are supported: " << na << " and " << nb << " must have shape (n, 3) and (m, 3). Got "
           << na << ".shape = " << shape_str(a) << ", " << nb << ".shape = " << shape_str(b) << ".";
        throw py::value_error(ss.str());
    }
}

template <typename T>
py::array_t<T, py::array::c_style> dense(const py::array& a) {
    return py::array_t<T, py::array::c_style | py::array::forcecast>::ensure(a);
}

// device < 0: the caller named none (the reference's interface has no such argument) -> the library's rule
// (PCU_B200_DEVICE, the CUDA runtime's current device, LOCAL_RANK, 0; see pcu_b200_current_device)
int current_device_or_default(int device) { return device < 0 ? pcu_b200_current_device() : device; }

template <typename T>
py::tuple knn_numpy(const py::array& q_in, const py::array& d_in, int k, bool squared, int leaf, int device) {
    auto q = dense<T>(q_in);
    auto d = dense<T>(d_in);
    const int64_t n = q.shape(0), m = d.shape(0);
    py::array_t<T> dists = result_array<T>((py::ssize_t)n, (py::ssize_t)k);
    py::array_t<int64_t> corrs = result_array<int64_t>((py::ssize_t)n, (py::ssize_t)k);
    Slot& slot = pool().get(device, kHostKey);
    pcu_b200_workspace* ws = slot.ws;
    const pcu_b200_options opts = make_options(leaf);
    int status;
    int64_t tied = 0;
    {
        CallScope scope(slot);
        pcu_b200_workspace_set_options(ws, &opts);
        if (sizeof(T) == 4)
            status = pcu_b200_knn_host_f32(ws, (const float*)q.data(), n, (const float*)d.data(), m, k, squared,
                                           (float*)dists.mutable_data(), corrs.mutable_data(), &tied);
        else
            status = pcu_b200_knn_host_f64(ws, (const double*)q.data(), n, (const double*)d.data(), m, k, squared,
                                           (double*)dists.mutable_data(), corrs.mutable_data(), &tied);
    }
    check(status);
    // npe::move hands the matrix to numpy and squeezes every size-1 dimension
    // (pinned for (n, 1) -> (n,) by tests/test_examples.py:363-368)
    return py::make_tuple(dists.attr("squeeze")(), corrs.attr("squeeze")());
}

py::tuple k_nearest_neighbors(const py::array& query_points, const py::array& dataset_points, int k,
                              bool squared_distances, int max_points_per_leaf, int num_threads, int device) {
    (void)num_threads;  // CPU thread count of the reference; results never depended on it
    if (k <= 0) throw py::value_error("Invalid value for k (" + std::to_string(k) + ") must be greater than 0.");
    const Dt dt = common_dtype(query_points, dataset_points, "query_points", "dataset_points");
    check_shapes(query_points, dataset_points, "query_points", "dataset_points");
    const int dev = current_device_or_default(device);
    return dt == Dt::f32 ? knn_numpy<float>(query_points, dataset_points, k, squared_distances, max_points_per_leaf, dev)
                         : knn_numpy<double>(query_points, dataset_points, k, squared_distances, max_points_per_leaf, dev);
}

py::dict stats_to_dict(const pcu_b200_nn_stats& s) {
    py::dict d;
    d["sum_dist"] = s.sum_dist;
    d["sum_sq_dist"] = s.sum_sq_dist;
    d["max_sq_dist"] = s.max_sq_dist;
    d["argmax_query"] = s.argmax_query;
    d["argmax_data"] = s.argmax_data;
    d["n_queries"] = s.n_queries;
    d["n_tied"] = s.n_tied;
    d["n_far"] = s.n_far;
    d["witness_tied"] = s.witness_tied;
    d["pair_value"] = s.pair_value;
    return d;
}

template <typename T>
pcu_b200_nn_stats one_sided_numpy(const py::array& s_in, const py::array& t_in, int leaf, int device) {
    auto s = dense<T>(s_in);
    auto t = dense<T>(t_in);
    Slot& slot = pool().get(device, kHostKey);
    pcu_b200_workspace* ws = slot.ws;
    const pcu_b200_options opts = make_options(leaf);
    pcu_b200_nn_stats st{};
    int status;
    {
        CallScope scope(slot);
        pcu_b200_workspace_set_options(ws, &opts);
        if (sizeof(T) == 4)
            status = pcu_b200_nn_stats_host_f32(ws, (const float*)s.data(), s.shape(0), (const float*)t.data(), t.shape(0), &st);
        else
            status = pcu_b200_nn_stats_host_f64(ws, (const double*)s.data(), s.shape(0), (const double*)t.data(), t.shape(0), &st);
    }
    check(status);
    return st;
}

template <typename T>
T metric_value(double max_sq, bool squared) {
    const T d2 = (T)max_sq;  // exact: max_sq is the input-precision value widened
    return squared ? d2 : (T)std::sqrt(d2);  // correctly rounded sqrt in the input precision (:84-88)
}

py::object one_sided_hausdorff_distance(const py::array& source, const py::array& target, bool return_index,
                                        bool squared_distances, int max_points_per_leaf, int device) {
    const Dt dt = common_dtype(source, target, "source", "target");
    check_shapes(source, target, "source", "target");
    const int dev = current_device_or_default(device);
    const pcu_b200_nn_stats st = dt == Dt::f32 ? one_sided_numpy<float>(source, target, max_points_per_leaf, dev)
                                               : one_sided_numpy<double>(source, target, max_points_per_leaf, dev);
    const double value = dt == Dt::f32 ? (double)metric_value<float>(st.max_sq_dist, squared_distances)
                                       : metric_value<double>(st.max_sq_dist, squared_distances);
    if (return_index) return py::make_tuple(value, st.argmax_query, st.argmax_data);
    return py::float_(value);
}

// Fused bidirectional sweep on numpy inputs: (chamfer value in input precision, stats x->y, stats y->x)
py::tuple chamfer_stats(const py::array& x_in, const py::array& y_in, int max_points_per_leaf, int device) {
    const Dt dt = common_dtype(x_in, y_in, "x", "y");
    check_shapes(x_in, y_in, "x", "y");
    const int dev = current_device_or_default(device);
    Slot& slot = pool().get(dev, kHostKey);
    pcu_b200_workspace* ws = slot.ws;
    const pcu_b200_options opts = make_options(max_points_per_leaf);
    pcu_b200_nn_stats st[2] = {};
    int status;
    py::object value;
    if (dt == Dt::f32) {
        auto x = dense<float>(x_in);
        auto y = dense<float>(y_in);
        float v = 0.f;
        { CallScope scope(slot); pcu_b200_workspace_set_options(ws, &opts);
          status = pcu_b200_chamfer_host_f32(ws, x.data(), x.shape(0), y.data(), y.shape(0), st, &v); }
        check(status);
        value = py::module_::import("numpy").attr("float32")(v);
    } else {
        auto x = dense<double>(x_in);
        auto y = dense<double>(y_in);
        double v = 0.0;
        { CallScope scope(slot); pcu_b200_workspace_set_options(ws, &opts);
          status = pcu_b200_chamfer_host_f64(ws, x.data(), x.shape(0), y.data(), y.shape(0), st, &v); }
        check(status);
        value = py::module_::import("numpy").attr("float64")(v);
    }
    return py::make_tuple(value, stats_to_dict(st[0]), stats_to_dict(st[1]));
}

// validate_input of the reference (src/point_cloud_normals.cpp:25-42) plus the npe dtype rule
Dt validate_normals_input(const py::array& points, const py::array& view_dirs) {
    const Dt dt = common_dtype(points, view_dirs, "points", "view_dirs");
    auto shape_of = [](const py::array& a) {
        std::ostringstream ss;
        ss << "(";
        for (py::ssize_t i = 0; i < a.ndim(); ++i) ss << (i ? ", " : "") << a.shape(i);
        ss << ")";
        return ss.str();
    };
    if (points.ndim() != 2 || points.shape(0) == 0 || points.shape(1) != 3)      // validate_input, :25-33
        throw py::value_error("Invalid point set with zero elements: points must have shape (n, 3), but got points.shape = " +
                              shape_of(points) + ".");
    if (view_dirs.ndim() != 2 || (view_dirs.shape(0) != 0 && (view_dirs.shape(0) != points.shape(0) || view_dirs.shape(1) != 3)))
        throw py::value_error("Invalid view directions does not match the number of points. If view directions are passed in, "
                              "they must have the same shape as points. Got points.shape = " + shape_of(points) +
                              ", and view_dirs.shape = " + shape_of(view_dirs) + ".");   // :34-42
    return dt;
}

// estimate_point_cloud_normals_knn_internal (src/point_cloud_normals.cpp:375-411): (indices of the kept points,
// their unit normals).  view_dirs is a (0, 3) array when no view directions are given, as in the reference's wrapper.
template <typename T>
py::tuple normals_knn_numpy(const py::array& p_in, const py::array& v_in, int k, int leaf, double drop_angle, int device) {
    auto pts = dense<T>(p_in);
    auto dirs = dense<T>(v_in);
    const int64_t n = pts.shape(0);
    const bool has_dirs = dirs.shape(0) != 0;
    py::array_t<int64_t> idx({(py::ssize_t)n});
    py::array_t<T> normals({(py::ssize_t)n, (py::ssize_t)3});
    int64_t kept = 0;
    Slot& slot = pool().get(device, kHostKey);
    pcu_b200_workspace* ws = slot.ws;
    const pcu_b200_options opts = make_options(leaf);
    int status;
    {
        CallScope scope(slot);
        pcu_b200_workspace_set_options(ws, &opts);
        if (sizeof(T) == 4)
            status = pcu_b200_normals_knn_host_f32(ws, (const float*)pts.data(), n, has_dirs ? (const float*)dirs.data() : nullptr, k,
                                                   drop_angle, idx.mutable_data(), (float*)normals.mutable_data(), &kept);
        else
            status = pcu_b200_normals_knn_host_f64(ws, (const double*)pts.data(), n, has_dirs ? (const double*)dirs.data() : nullptr, k,
                                                   drop_angle, idx.mutable_data(), (double*)normals.mutable_data(), &kept);
    }
    check(status);
    idx.resize({(py::ssize_t)kept});
    normals.resize({(py::ssize_t)kept, (py::ssize_t)3});
    return py::make_tuple(idx, normals);
}

py::tuple estimate_point_cloud_normals_knn_internal(const py::array& points, const py::array& view_dirs, int num_neighbors,
                                                    int max_points_per_leaf, double drop_angle_threshold, int num_threads,
                                                    int random_seed, int device) {
    (void)num_threads; (void)random_seed;   // CPU threading / rand() seeding of the reference: no effect on the k-NN variant
    if (num_neighbors <= 0)
        throw py::value_error("Invalid number of neighbors (" + std::to_string(num_neighbors) + ") must be greater than 0.");
    const Dt dt = validate_normals_input(points, view_dirs);
    const int dev = current_device_or_default(device);
    return dt == Dt::f32 ? normals_knn_numpy<float>(points, view_dirs, num_neighbors, max_points_per_leaf, drop_angle_threshold, dev)
                         : normals_knn_numpy<double>(points, view_dirs, num_neighbors, max_points_per_leaf, drop_angle_threshold, dev);
}

void normals_knn_device(bool is_f64, uintptr_t points, int64_t n, uintptr_t view_dirs, int k, double drop_angle,
                        uintptr_t out_idx, uintptr_t out_normals, uintptr_t out_count, int max_points_per_leaf, int device,
                        uintptr_t stream) {
    if (k <= 0) throw py::value_error("Invalid number of neighbors (" + std::to_string(k) + ") must be greater than 0.");
    Slot& slot = pool().get(device, stream);
    pcu_b200_workspace* ws = slot.ws;
    const pcu_b200_options opts = make_options(max_points_per_leaf);
    int status;
    {
        CallScope scope(slot);
        pcu_b200_workspace_set_options(ws, &opts);
        status = is_f64 ? pcu_b200_normals_knn_f64(ws, (const double*)points, n, (const double*)view_dirs, k, drop_angle,
                                                   (int64_t*)out_idx, (double*)out_normals, (int64_t*)out_count, (void*)stream)
                        : pcu_b200_normals_knn_f32(ws, (const float*)points, n, (const float*)view_dirs, k, drop_angle,
                                                   (int64_t*)out_idx, (float*)out_normals, (int64_t*)out_count, (void*)stream);
    }
    check(status);
}

// estimate_point_cloud_normals_ball_internal (src/point_cloud_normals.cpp:303-370), argument order of the reference
pcu_b200_ball_options ball_options(double radius, int min_pts, int max_pts, double drop_angle, const std::string& weight_function, int seed) {
    if (radius <= 0.0) throw py::value_error("Invalid radius (" + std::to_string(radius) + ") must be greater than 0.");
    if (min_pts < 3) throw py::value_error("Invalid min_pts_per_ball (" + std::to_string(min_pts) + ") must be greater than 3.");
    if (max_pts > 0 && max_pts < 3)
        throw py::value_error("Invalid max_pts_per_ball (" + std::to_string(max_pts) +
                              ") must either be negative (no max) or a number greater than 3.");
    pcu_b200_ball_options o;
    o.radius = radius; o.drop_angle_threshold = drop_angle; o.min_pts_per_ball = min_pts; o.max_pts_per_ball = max_pts;
    if (weight_function == "constant") o.weight_function = 0;
    else if (weight_function == "rbf") o.weight_function = 1;
    else throw py::value_error("Invalid weight_function, must be one of 'constant' or 'rbf'.");
    o.seed = (uint32_t)seed;
    return o;
}

template <typename T>
py::tuple normals_ball_numpy(const py::array& p_in, const py::array& v_in, const pcu_b200_ball_options& o, int device) {
    auto pts = dense<T>(p_in);
    auto dirs = dense<T>(v_in);
    const int64_t n = pts.shape(0);
    const bool has_dirs = dirs.shape(0) != 0;
    py::array_t<int64_t> idx({(py::ssize_t)n});
    py::array_t<T> normals({(py::ssize_t)n, (py::ssize_t)3});
    int64_t kept = 0;
    Slot& slot = pool().get(device, kHostKey);
    pcu_b200_workspace* ws = slot.ws;
    int status;
    {
        CallScope scope(slot);
        if (sizeof(T) == 4)
            status = pcu_b200_normals_ball_host_f32(ws, (const float*)pts.data(), n, has_dirs ? (const float*)dirs.data() : nullptr, &o,
                                                    idx.mutable_data(), (float*)normals.mutable_data(), &kept);
        else
            status = pcu_b200_normals_ball_host_f64(ws, (const double*)pts.data(), n, has_dirs ? (const double*)dirs.data() : nullptr, &o,
                                                    idx.mutable_data(), (double*)normals.mutable_data(), &kept);
    }
    check(status);
    idx.resize({(py::ssize_t)kept});
    normals.resize({(py::ssize_t)kept, (py::ssize_t)3});
    return py::make_tuple(idx, normals);
}

py::tuple estimate_point_cloud_normals_ball_internal(const py::array& points, const py::array& view_dirs, double radius,
                                                     int min_pts_per_ball, int max_pts_per_ball, double drop_angle_threshold,
                                                     int max_points_per_leaf, int num_threads, const std::string& weight_function,
                                                     int random_seed, int device) {
    (void)max_points_per_leaf; (void)num_threads;   // kd-tree leaf size / CPU threads of the reference: no effect on the result
    const pcu_b200_ball_options o = ball_options(radius, min_pts_per_ball, max_pts_per_ball, drop_angle_threshold, weight_function, random_seed);
    const Dt dt = validate_normals_input(points, view_dirs);
    const int dev = current_device_or_default(device);
    return dt == Dt::f32 ? normals_ball_numpy<float>(points, view_dirs, o, dev) : normals_ball_numpy<double>(points, view_dirs, o, dev);
}

void normals_ball_device(bool is_f64, uintptr_t points, int64_t n, uintptr_t view_dirs, double radius, int min_pts, int max_pts,
                         double drop_angle, const std::string& weight_function, int seed, uintptr_t out_idx, uintptr_t out_normals,
                         uintptr_t out_count, int device, uintptr_t stream) {
    const pcu_b200_ball_options o = ball_options(radius, min_pts, max_pts, drop_angle, weight_function, seed);
    Slot& slot = pool().get(device, stream);
    pcu_b200_workspace* ws = slot.ws;
    int status;
    {
        CallScope scope(slot);
        status = is_f64 ? pcu_b200_normals_ball_f64(ws, (const double*)points, n, (const double*)view_dirs, &o, (int64_t*)out_idx,
                                                    (double*)out_normals, (int64_t*)out_count, (void*)stream)
                        : pcu_b200_normals_ball_f32(ws, (const float*)points, n, (const float*)view_dirs, &o, (int64_t*)out_idx,
                                                    (float*)out_normals, (int64_t*)out_count, (void*)stream);
    }
    check(status);
}

// ---- Morton codes (src/morton.cpp) ----------------------------------------------------------------
// dtype rules of the bindings: pts int32 / int64; codes uint32 / uint64 (uint32 codes are widened, as the
// reference's MortonCode64(uint64_t) constructor does implicitly); results are uint64 / int32 / int64 like the reference's.
py::array_t<uint64_t, py::array::c_style> as_codes(const py::array& a, const char* name) {
    if (!a.dtype().is(py::dtype::of<uint64_t>()) && !a.dtype().is(py::dtype::of<uint32_t>()))
        throw py::value_error(std::string("Invalid scalar type (") + std::string(py::str(a.dtype())) + ") for argument '" + name +
                              "'. Expected one of ['uint32', 'uint64'].");
    if (a.ndim() == 0 || a.size() == 0) throw py::value_error(std::string(name) + " must be an array of shape [n] but got an empty array");
    if (!(a.ndim() == 1 || (a.ndim() == 2 && a.shape(1) == 1)))
        throw py::value_error(std::string(name) + " must be an array of shape [n] but got an invalid number of columns");
    return py::array_t<uint64_t, py::array::c_style | py::array::forcecast>::ensure(a);
}

py::array morton_encode(const py::array& pts, int num_threads, int device) {
    (void)num_threads;
    const bool i32 = pts.dtype().is(py::dtype::of<int32_t>()), i64 = pts.dtype().is(py::dtype::of<int64_t>());
    if (!i32 && !i64)
        throw py::value_error("Invalid scalar type (" + std::string(py::str(pts.dtype())) + ") for argument 'pts'. Expected one of ['int32', 'int64'].");
    if (pts.ndim() != 2 || pts.shape(0) <= 0) throw py::value_error("pts must be an array of shape [n, 3] but got an empty array");
    if (pts.shape(1) != 3) throw py::value_error("pts must be an array of shape [n, 3] but got an invalid number of columns");
    const int64_t n = pts.shape(0);
    py::array_t<uint64_t> codes({(py::ssize_t)n});
    Slot& slot = pool().get(current_device_or_default(device), kHostKey);
    int status;
    if (i32) {
        auto p = py::array_t<int32_t, py::array::c_style | py::array::forcecast>::ensure(pts);
        CallScope scope(slot);
        status = pcu_b200_morton_encode_host_i32(slot.ws, p.data(), n, codes.mutable_data());
    } else {
        auto p = py::array_t<int64_t, py::array::c_style | py::array::forcecast>::ensure(pts);
        CallScope scope(slot);
        status = pcu_b200_morton_encode_host_i64(slot.ws, p.data(), n, codes.mutable_data());
    }
    check(status);
    return codes;
}

py::array morton_decode(const py::array& codes_in, int num_threads, int device) {
    (void)num_threads;
    auto codes = as_codes(codes_in, "codes");
    const int64_t n = codes.size();
    py::array_t<int32_t> pts({(py::ssize_t)n, (py::ssize_t)3});
    Slot& slot = pool().get(current_device_or_default(device), kHostKey);
    int status;
    { CallScope scope(slot); status = pcu_b200_morton_decode_host(slot.ws, codes.data(), n, pts.mutable_data()); }
    check(status);
    return pts;
}

py::array morton_addsub(const py::array& a_in, const py::array& b_in, int num_threads, int device, bool subtract) {
    (void)num_threads;
    auto a = as_codes(a_in, "codes_1");
    auto b = as_codes(b_in, "codes_2");
    if (a.size() != b.size()) throw py::value_error("codes_1 and codes_2 must have the same number of entries.");
    const int64_t n = a.size();
    py::array_t<uint64_t> out({(py::ssize_t)n});
    Slot& slot = pool().get(current_device_or_default(device), kHostKey);
    int status;
    {
        CallScope scope(slot);
        status = subtract ? pcu_b200_morton_subtract_host(slot.ws, a.data(), b.data(), n, out.mutable_data())
                          : pcu_b200_morton_add_host(slot.ws, a.data(), b.data(), n, out.mutable_data());
    }
    check(status);
    return out;
}

py::array morton_knn(const py::array& codes_in, const py::array& qcodes_in, int k, bool sort_dist, int device) {
    if (k <= 0) throw py::value_error("k must be greater than 0");
    auto codes = as_codes(codes_in, "codes");
    auto qcodes = as_codes(qcodes_in, "qcodes");
    if (!qcodes_in.dtype().is(codes_in.dtype()))
        throw py::value_error("Invalid scalar type for argument 'qcodes'. Expected it to match argument 'codes'.");
    const int64_t n = codes.size(), m = qcodes.size();
    k = (int)std::min<int64_t>(k, n);                       // morton.cpp:351
    py::array_t<int64_t> idx({(py::ssize_t)m, (py::ssize_t)k});
    Slot& slot = pool().get(current_device_or_default(device), kHostKey);
    int status;
    { CallScope scope(slot); status = pcu_b200_morton_knn_host(slot.ws, codes.data(), n, qcodes.data(), m, k, sort_dist ? 1 : 0, idx.mutable_data()); }
    check(status);
    return idx;
}

// ---- prepared clouds (handles travel as integers; point-cloud-utils_b200/__init__.py wraps them in PreparedCloud) ----
uintptr_t cloud_prepare_numpy(const py::array& pts_in, int device, int knn_k, int leaf) {
    const bool f32 = pts_in.dtype().is(py::dtype::of<float>()), f64 = pts_in.dtype().is(py::dtype::of<double>());
    if (!f32 && !f64)
        throw py::value_error("Invalid scalar type (" + std::string(py::str(pts_in.dtype())) + ") for argument 'points'. Expected one of ['float32', 'float64'].");
    if (pts_in.ndim() != 2 || pts_in.shape(1) != 3 || pts_in.shape(0) == 0)
        throw py::value_error("Only 3D inputs are supported: points must have shape (n, 3) with n > 0.");
    const int dev = current_device_or_default(device);
    Slot& slot = pool().get(dev, kHostKey);
    pcu_b200_cloud* cloud = nullptr;
    int status;
    if (f32) {
        auto p = dense<float>(pts_in);
        CallScope scope(slot);
        status = knn_k > 0 ? pcu_b200_cloud_prepare_knn_host_f32(slot.ws, p.data(), p.shape(0), knn_k, leaf, &cloud)
                           : pcu_b200_cloud_prepare_host_f32(slot.ws, p.data(), p.shape(0), &cloud);
    } else {
        auto p = dense<double>(pts_in);
        CallScope scope(slot);
        status = knn_k > 0 ? pcu_b200_cloud_prepare_knn_host_f64(slot.ws, p.data(), p.shape(0), knn_k, leaf, &cloud)
                           : pcu_b200_cloud_prepare_host_f64(slot.ws, p.data(), p.shape(0), &cloud);
    }
    check(status);
    return (uintptr_t)cloud;
}
uintptr_t cloud_prepare_device(bool is_f64, uintptr_t pts, int64_t n, int device, uintptr_t stream, int knn_k, int leaf) {
    Slot& slot = pool().get(device, stream);
    pcu_b200_cloud* cloud = nullptr;
    int status;
    {
        CallScope scope(slot);
        if (knn_k > 0)
            status = is_f64 ? pcu_b200_cloud_prepare_knn_f64(slot.ws, (const double*)pts, n, knn_k, leaf, &cloud, (void*)stream)
                            : pcu_b200_cloud_prepare_knn_f32(slot.ws, (const float*)pts, n, knn_k, leaf, &cloud, (void*)stream);
        else
            status = is_f64 ? pcu_b200_cloud_prepare_f64(slot.ws, (const double*)pts, n, &cloud, (void*)stream)
                            : pcu_b200_cloud_prepare_f32(slot.ws, (const float*)pts, n, &cloud, (void*)stream);
    }
    check(status);
    return (uintptr_t)cloud;
}
void cloud_destroy(uintptr_t cloud) {
    py::gil_scoped_release nogil;
    pcu_b200_cloud_destroy((pcu_b200_cloud*)cloud);
}
// k nearest neighbours of numpy points in a prepared cloud: (dists, corrs) like k_nearest_neighbors
template <typename T>
py::tuple knn_prepared_numpy_t(const py::array& q_in, pcu_b200_cloud* cloud, int k, bool squared, int leaf, int device) {
    auto q = dense<T>(q_in);
    const int64_t n = q.shape(0);
    py::array_t<T> dists = result_array<T>((py::ssize_t)n, (py::ssize_t)k);
    py::array_t<int64_t> corrs = result_array<int64_t>((py::ssize_t)n, (py::ssize_t)k);
    Slot& slot = pool().get(device, kHostKey);
    const pcu_b200_options opts = make_options(leaf);
    int status;
    int64_t tied = 0;
    {
        CallScope scope(slot);
        pcu_b200_workspace_set_options(slot.ws, &opts);
        if (sizeof(T) == 4)
            status = pcu_b200_knn_prepared_host_f32(slot.ws, (const float*)q.data(), n, cloud, k, squared, (float*)dists.mutable_data(),
                                                    corrs.mutable_data(), &tied);
        else
            status = pcu_b200_knn_prepared_host_f64(slot.ws, (const double*)q.data(), n, cloud, k, squared, (double*)dists.mutable_data(),
                                                    corrs.mutable_data(), &tied);
    }
    check(status);
    return py::make_tuple(dists.attr("squeeze")(), corrs.attr("squeeze")());
}
py::tuple knn_prepared_numpy(const py::array& q_in, uintptr_t cloud, bool cloud_is_f64, int k, bool squared, int max_points_per_leaf, int device) {
    if (k <= 0) throw py::value_error("Invalid value for k (" + std::to_string(k) + ") must be greater than 0.");
    const bool f32 = q_in.dtype().is(py::dtype::of<float>()), f64 = q_in.dtype().is(py::dtype::of<double>());
    if ((!f32 && !f64) || f64 != cloud_is_f64)
        throw py::value_error("Invalid scalar type (" + std::string(py::str(q_in.dtype())) + "): expected the prepared cloud's " +
                              (cloud_is_f64 ? "float64" : "float32") + ".");
    if (q_in.ndim() != 2 || q_in.shape(1) != 3)
        throw py::value_error("Only 3D inputs are supported: points must have shape (n, 3).");
    if (q_in.shape(0) == 0) throw py::value_error("Invalid input set with zero elements: points must have shape (n, 3) with n > 0.");
    const int dev = current_device_or_default(device);
    return f32 ? knn_prepared_numpy_t<float>(q_in, (pcu_b200_cloud*)cloud, k, squared, max_points_per_leaf, dev)
               : knn_prepared_numpy_t<double>(q_in, (pcu_b200_cloud*)cloud, k, squared, max_points_per_leaf, dev);
}
void knn_prepared_device(bool is_f64, uintptr_t query, int64_t n, uintptr_t cloud, int k, bool squared, uintptr_t out_dist,
                         uintptr_t out_idx, uintptr_t out_n_tied, int max_points_per_leaf, int device, uintptr_t stream) {
    if (k <= 0) throw py::value_error("Invalid value for k (" + std::to_string(k) + ") must be greater than 0.");
    Slot& slot = pool().get(device, stream);
    const pcu_b200_options opts = make_options(max_points_per_leaf);
    int status;
    {
        CallScope scope(slot);
        pcu_b200_workspace_set_options(slot.ws, &opts);
        status = is_f64 ? pcu_b200_knn_prepared_f64(slot.ws, (const double*)query, n, (pcu_b200_cloud*)cloud, k, squared, (double*)out_dist,
                                                    (int64_t*)out_idx, (int64_t*)out_n_tied, (void*)stream)
                        : pcu_b200_knn_prepared_f32(slot.ws, (const float*)query, n, (pcu_b200_cloud*)cloud, k, squared, (float*)out_dist,
                                                    (int64_t*)out_idx, (int64_t*)out_n_tied, (void*)stream);
    }
    check(status);
}

// fused sweep(s) of numpy points against a prepared cloud: (value or None, stats[, stats])
py::tuple stats_prepared_numpy(const py::array& x_in, uintptr_t cloud, bool cloud_is_f64, bool both, int max_points_per_leaf, int device) {
    const bool f32 = x_in.dtype().is(py::dtype::of<float>()), f64 = x_in.dtype().is(py::dtype::of<double>());
    if ((!f32 && !f64) || f64 != cloud_is_f64)
        throw py::value_error("Invalid scalar type (" + std::string(py::str(x_in.dtype())) + "): expected the prepared cloud's " +
                              (cloud_is_f64 ? "float64" : "float32") + ".");
    if (x_in.ndim() != 2 || x_in.shape(1) != 3)
        throw py::value_error("Only 3D inputs are supported: points must have shape (n, 3).");
    if (x_in.shape(0) == 0) throw py::value_error("Invalid input set with zero elements: points must have shape (n, 3) with n > 0.");
    const int dev = current_device_or_default(device);
    Slot& slot = pool().get(dev, kHostKey);
    const pcu_b200_options opts = make_options(max_points_per_leaf);
    pcu_b200_nn_stats st[2] = {};
    int status;
    py::object value = py::none();
    auto* y = (const pcu_b200_cloud*)cloud;
    if (f32) {
        auto x = dense<float>(x_in);
        float v = 0.f;
        { CallScope scope(slot); pcu_b200_workspace_set_options(slot.ws, &opts);
          status = both ? pcu_b200_chamfer_prepared_host_f32(slot.ws, x.data(), x.shape(0), y, st, &v)
                        : pcu_b200_nn_stats_prepared_host_f32(slot.ws, x.data(), x.shape(0), y, st); }
        check(status);
        if (both) value = py::module_::import("numpy").attr("float32")(v);
    } else {
        auto x = dense<double>(x_in);
        double v = 0.0;
        { CallScope scope(slot); pcu_b200_workspace_set_options(slot.ws, &opts);
          status = both ? pcu_b200_chamfer_prepared_host_f64(slot.ws, x.data(), x.shape(0), y, st, &v)
                        : pcu_b200_nn_stats_prepared_host_f64(slot.ws, x.data(), x.shape(0), y, st); }
        check(status);
        if (both) value = py::module_::import("numpy").attr("float64")(v);
    }
    if (both) return py::make_tuple(value, stats_to_dict(st[0]), stats_to_dict(st[1]));
    return py::make_tuple(value, stats_to_dict(st[0]));
}
void stats_prepared_device(bool is_f64, bool both, uintptr_t a, int64_t n, uintptr_t cloud, uintptr_t out_stats, uintptr_t out_value,
                           int max_points_per_leaf, int device, uintptr_t stream) {
    Slot& slot = pool().get(device, stream);
    const pcu_b200_options opts = make_options(max_points_per_leaf);
    int status;
    {
        CallScope scope(slot);
        pcu_b200_workspace_set_options(slot.ws, &opts);
        auto* st = (pcu_b200_nn_stats*)out_stats;
        auto* y = (const pcu_b200_cloud*)cloud;
        if (both)
            status = is_f64 ? pcu_b200_chamfer_prepared_f64(slot.ws, (const double*)a, n, y, st, (double*)out_value, (void*)stream)
                            : pcu_b200_chamfer_prepared_f32(slot.ws, (const float*)a, n, y, st, (float*)out_value, (void*)stream);
        else
            status = is_f64 ? pcu_b200_nn_stats_prepared_f64(slot.ws, (const double*)a, n, y, st, (void*)stream)
                            : pcu_b200_nn_stats_prepared_f32(slot.ws, (const float*)a, n, y, st, (void*)stream);
    }
    check(status);
}

// ---- voxel-grid down-sampling on device pointers (the Python layer owns the arrays) ----
void voxel_downsample_device(bool is_f64, uintptr_t pts, int64_t n, uintptr_t attr, int attr_cols, bool attr_is_f64,
                             std::array<double, 3> size, std::array<double, 3> lo, std::array<double, 3> hi, int min_points,
                             uintptr_t out_pts, uintptr_t out_attr, uintptr_t out_counts, uintptr_t out_rows, int device, uintptr_t stream) {
    Slot& slot = pool().get(device, stream);
    int status;
    {
        CallScope scope(slot);
        status = is_f64 ? pcu_b200_voxel_downsample_f64(slot.ws, (const double*)pts, n, (const void*)attr, attr_cols, attr_is_f64 ? 1 : 0,
                                                        size.data(), lo.data(), hi.data(), min_points, (double*)out_pts, (void*)out_attr,
                                                        (int32_t*)out_counts, (int64_t*)out_rows, (void*)stream)
                        : pcu_b200_voxel_downsample_f32(slot.ws, (const float*)pts, n, (const void*)attr, attr_cols, attr_is_f64 ? 1 : 0,
                                                        size.data(), lo.data(), hi.data(), min_points, (float*)out_pts, (void*)out_attr,
                                                        (int32_t*)out_counts, (int64_t*)out_rows, (void*)stream);
    }
    check(status);
}

void deduplicate_device(bool is_f64, uintptr_t pts, int64_t n, double epsilon, uintptr_t faces, int64_t nf, int cols, bool faces_i64,
                        uintptr_t out_pts, uintptr_t out_svi, uintptr_t out_svj, uintptr_t out_faces, uintptr_t out_counts, int device,
                        uintptr_t stream) {
    Slot& slot = pool().get(device, stream);
    int status;
    {
        CallScope scope(slot);
        status = is_f64 ? pcu_b200_deduplicate_f64(slot.ws, (const double*)pts, n, epsilon, (const void*)faces, nf, cols, faces_i64 ? 1 : 0,
                                                   (double*)out_pts, (int32_t*)out_svi, (int32_t*)out_svj, (void*)out_faces,
                                                   (int64_t*)out_counts, (void*)stream)
                        : pcu_b200_deduplicate_f32(slot.ws, (const float*)pts, n, epsilon, (const void*)faces, nf, cols, faces_i64 ? 1 : 0,
                                                   (float*)out_pts, (int32_t*)out_svi, (int32_t*)out_svj, (void*)out_faces,
                                                   (int64_t*)out_counts, (void*)stream);
    }
    check(status);
}

// ---- Poisson-disk down-sampling (src/sample_point_cloud.cpp:240-333): numpy in, int32 rows out ----
template <typename T>
py::array_t<int32_t> poisson_numpy(const py::array& v_in, double radius, int target, uint32_t seed, float tol, int device) {
    auto pts = dense<T>(v_in);
    const int64_t n = pts.shape(0);
    py::array_t<int32_t> idx({(py::ssize_t)n});
    int64_t kept = 0;
    Slot& slot = pool().get(device, kHostKey);
    int status;
    {
        CallScope scope(slot);
        status = sizeof(T) == 4 ? pcu_b200_poisson_disk_downsample_host_f32(slot.ws, (const float*)pts.data(), n, radius, target, seed, tol,
                                                                            idx.mutable_data(), &kept)
                                : pcu_b200_poisson_disk_downsample_host_f64(slot.ws, (const double*)pts.data(), n, radius, target, seed, tol,
                                                                            idx.mutable_data(), &kept);
    }
    check(status);
    idx.resize({(py::ssize_t)kept});
    return idx;
}

py::array downsample_point_cloud_poisson_disk_internal(const py::array& v, double radius, int target_num_samples, uint32_t random_seed,
                                                       float sample_num_tolerance, int device) {
    check_shapes(v, v, "v", "v");
    const Dt dt = common_dtype(v, v, "v", "v");
    const int dev = current_device_or_default(device);
    return dt == Dt::f32 ? (py::array)poisson_numpy<float>(v, radius, target_num_samples, random_seed, sample_num_tolerance, dev)
                         : (py::array)poisson_numpy<double>(v, radius, target_num_samples, random_seed, sample_num_tolerance, dev);
}

void poisson_device(bool is_f64, uintptr_t pts, int64_t n, double radius, int target, uint32_t seed, float tol, uintptr_t out_idx,
                    uintptr_t out_count, int device, uintptr_t stream) {
    Slot& slot = pool().get(device, stream);
    int status;
    {
        CallScope scope(slot);
        status = is_f64 ? pcu_b200_poisson_disk_downsample_f64(slot.ws, (const double*)pts, n, radius, target, seed, tol, (int32_t*)out_idx,
                                                               (int64_t*)out_count, (void*)stream)
                        : pcu_b200_poisson_disk_downsample_f32(slot.ws, (const float*)pts, n, radius, target, seed, tol, (int32_t*)out_idx,
                                                               (int64_t*)out_count, (void*)stream);
    }
    check(status);
}

// ---- dense pairwise distances / Sinkhorn on device pointers (the Python layer owns the arrays) ----
void pairwise_device(bool is_f64, uintptr_t a, uintptr_t b, int64_t nb, int64_t n, int64_t m, int d, int norm_kind, double p,
                     uintptr_t out, int device, uintptr_t stream) {
    Slot& slot = pool().get(device, stream);
    int status;
    {
        CallScope scope(slot);
        status = is_f64 ? pcu_b200_pairwise_distances_f64(slot.ws, (const double*)a, (const double*)b, nb, n, m, d, norm_kind, p, (double*)out, (void*)stream)
                        : pcu_b200_pairwise_distances_f32(slot.ws, (const float*)a, (const float*)b, nb, n, m, d, norm_kind, p, (float*)out, (void*)stream);
    }
    check(status);
}
void sinkhorn_device(bool is_f64, uintptr_t a, uintptr_t b, uintptr_t M, int64_t nb, int64_t n, int64_t m, double eps, int max_iters,
                     double stop_thresh, uintptr_t out_P, uintptr_t out_cost, uintptr_t out_iters, int device, uintptr_t stream) {
    Slot& slot = pool().get(device, stream);
    int status;
    {
        CallScope scope(slot);
        status = is_f64 ? pcu_b200_sinkhorn_f64(slot.ws, (const double*)a, (const double*)b, (const double*)M, nb, n, m, eps, max_iters,
                                                stop_thresh, (double*)out_P, (double*)out_cost, (int32_t*)out_iters, (void*)stream)
                        : pcu_b200_sinkhorn_f32(slot.ws, (const float*)a, (const float*)b, (const float*)M, nb, n, m, eps, max_iters,
                                                stop_thresh, (float*)out_P, (double*)out_cost, (int32_t*)out_iters, (void*)stream);
    }
    check(status);
}

// ---- raw device-pointer entry points (CUDA torch tensors) --------------------------------------
void knn_device(bool is_f64, uintptr_t query, int64_t n, uintptr_t dataset, int64_t m, int k, bool squared,
                uintptr_t out_dist, uintptr_t out_idx, uintptr_t out_n_tied, int max_points_per_leaf, int device,
                uintptr_t stream) {
    if (k <= 0) throw py::value_error("Invalid value for k (" + std::to_string(k) + ") must be greater than 0.");
    Slot& slot = pool().get(device, stream);
    pcu_b200_workspace* ws = slot.ws;
    const pcu_b200_options opts = make_options(max_points_per_leaf);
    int status;
    {
        CallScope scope(slot);
        pcu_b200_workspace_set_options(ws, &opts);
        status = is_f64 ? pcu_b200_knn_f64(ws, (const double*)query, n, (const double*)dataset, m, k, squared,
                                           (double*)out_dist, (int64_t*)out_idx, (int64_t*)out_n_tied, (void*)stream)
                        : pcu_b200_knn_f32(ws, (const float*)query, n, (const float*)dataset, m, k, squared,
                                           (float*)out_dist, (int64_t*)out_idx, (int64_t*)out_n_tied, (void*)stream);
    }
    check(status);
}

void stats_device(bool is_f64, bool both, uintptr_t a, int64_t n, uintptr_t b, int64_t m, uintptr_t out_stats,
                  uintptr_t out_value, int max_points_per_leaf, int device, uintptr_t stream) {
    Slot& slot = pool().get(device, stream);
    pcu_b200_workspace* ws = slot.ws;
    const pcu_b200_options opts = make_options(max_points_per_leaf);
    int status;
    {
        CallScope scope(slot);
        pcu_b200_workspace_set_options(ws, &opts);
        auto* st = (pcu_b200_nn_stats*)out_stats;
        if (both)
            status = is_f64 ? pcu_b200_chamfer_f64(ws, (const double*)a, n, (const double*)b, m, st, (double*)out_value, (void*)stream)
                            : pcu_b200_chamfer_f32(ws, (const float*)a, n, (const float*)b, m, st, (float*)out_value, (void*)stream);
        else
            status = is_f64 ? pcu_b200_nn_stats_f64(ws, (const double*)a, n, (const double*)b, m, st, (void*)stream)
                            : pcu_b200_nn_stats_f32(ws, (const float*)a, n, (const float*)b, m, st, (void*)stream);
    }
    check(status);
}

// Batched Chamfer on numpy inputs: x (B, n, 3), y (B, m, 3) float32 -> ((B,) float32, fp64 sum)
py::tuple batched_chamfer_numpy(const py::array& x_in, const py::array& y_in, int max_points_per_leaf, int device) {
    if (!x_in.dtype().is(py::dtype::of<float>()) || !y_in.dtype().is(py::dtype::of<float>()))
        throw py::value_error("batched_chamfer_distance: x and y must both be float32");
    if (x_in.ndim() != 3 || y_in.ndim() != 3 || x_in.shape(2) != 3 || y_in.shape(2) != 3 || x_in.shape(0) != y_in.shape(0))
        throw py::value_error("batched_chamfer_distance: x and y must have shape (B, n, 3) and (B, m, 3)");
    if (x_in.shape(0) == 0 || x_in.shape(1) == 0 || y_in.shape(1) == 0)
        throw py::value_error("Invalid input set with zero elements: x and y must have shape (B, n, 3) and (B, m, 3)");
    auto x = dense<float>(x_in);
    auto y = dense<float>(y_in);
    const int64_t B = x.shape(0), n = x.shape(1), m = y.shape(1);
    py::array_t<float> out({(py::ssize_t)B});
    double sum = 0.0;
    const int dev = current_device_or_default(device);
    Slot& slot = pool().get(dev, kHostKey);
    pcu_b200_workspace* ws = slot.ws;
    const pcu_b200_options opts = make_options(max_points_per_leaf);
    int status;
    {
        CallScope scope(slot);
        pcu_b200_workspace_set_options(ws, &opts);
        status = pcu_b200_batched_chamfer_host_f32(ws, x.data(), y.data(), B, n, m, out.mutable_data(),
                                                   &sum);
    }
    check(status);
    return py::make_tuple(out, sum);
}

void batched_chamfer_device(uintptr_t x, uintptr_t y, int64_t B, int64_t n, int64_t m, uintptr_t out_per_pair,
                            uintptr_t out_sum, int max_points_per_leaf, int device, uintptr_t stream) {
    Slot& slot = pool().get(device, stream);
    pcu_b200_workspace* ws = slot.ws;
    const pcu_b200_options opts = make_options(max_points_per_leaf);
    int status;
    {
        CallScope scope(slot);
        pcu_b200_workspace_set_options(ws, &opts);
        status = pcu_b200_batched_chamfer_f32(ws, (const float*)x, (const float*)y, B, n, m, (float*)out_per_pair,
                                              (double*)out_sum, (void*)stream);
    }
    check(status);
}

template <typename T>
py::dict debug_kd_tree_t(const py::array& pts_in, int leaf, int device) {
    auto pts = dense<T>(pts_in);
    const int64_t m = pts.shape(0);
    const int64_t cap = 2 * m + 2;
    py::array_t<int32_t> order(m), feat(cap), first(cap), last(cap), kid0(cap), kid1(cap);
    py::array_t<T> lo(cap), hi(cap);
    int64_t nn = 0;
    Slot& slot = pool().get(device, kHostKey);
    pcu_b200_workspace* ws = slot.ws;
    int status;
    if (sizeof(T) == 4)
        status = pcu_b200_debug_kd_tree_f32(ws, (const float*)pts.data(), m, leaf, order.mutable_data(), cap,
                                            feat.mutable_data(), (float*)lo.mutable_data(), (float*)hi.mutable_data(),
                                            first.mutable_data(), last.mutable_data(), kid0.mutable_data(),
                                            kid1.mutable_data(), &nn);
    else
        status = pcu_b200_debug_kd_tree_f64(ws, (const double*)pts.data(), m, leaf, order.mutable_data(), cap,
                                            feat.mutable_data(), (double*)lo.mutable_data(), (double*)hi.mutable_data(),
                                            first.mutable_data(), last.mutable_data(), kid0.mutable_data(),
                                            kid1.mutable_data(), &nn);
    check(status);
    py::dict d;
    d["order"] = order; d["feat"] = feat; d["div_lo"] = lo; d["div_hi"] = hi; d["first"] = first; d["last"] = last;
    d["kid0"] = kid0; d["kid1"] = kid1; d["n_nodes"] = nn;
    return d;
}

py::dict debug_kd_tree(const py::array& pts, int leaf, int device) {
    if (pts.ndim() != 2 || pts.shape(1) != 3 || pts.shape(0) == 0) throw py::value_error("points must be (m, 3)");
    const int dev = current_device_or_default(device);
    if (pts.dtype().is(py::dtype::of<float>())) return debug_kd_tree_t<float>(pts, leaf, dev);
    if (pts.dtype().is(py::dtype::of<double>())) return debug_kd_tree_t<double>(pts, leaf, dev);
    throw py::value_error("points must be float32 or float64");
}

void resolve_witness_device(bool is_f64, uintptr_t q, int64_t n, uintptr_t d, int64_t m, uintptr_t stats,
                            int max_points_per_leaf, int device, uintptr_t stream) {
    Slot& slot = pool().get(device, stream);
    pcu_b200_workspace* ws = slot.ws;
    const pcu_b200_options opts = make_options(max_points_per_leaf);
    int status;
    {
        CallScope scope(slot);
        pcu_b200_workspace_set_options(ws, &opts);
        status = is_f64 ? pcu_b200_resolve_witness_f64(ws, (const double*)q, n, (const double*)d, m,
                                                       (pcu_b200_nn_stats*)stats, (void*)stream)
                        : pcu_b200_resolve_witness_f32(ws, (const float*)q, n, (const float*)d, m,
                                                       (pcu_b200_nn_stats*)stats, (void*)stream);
    }
    check(status);
}

}  // namespace

PYBIND11_MODULE(_pcu_internal, mod) {
    mod.doc() = "B200-native nearest-neighbour bindings (drop-in for point_cloud_utils._pcu_internal on this path)";
    mod.def("k_nearest_neighbors", &k_nearest_neighbors, py::arg("query_points"), py::arg("dataset_points"),
            py::arg("k"), py::arg("squared_distances") = false, py::arg("max_points_per_leaf") = 10,
            py::arg("num_threads") = -1, py::arg("device") = -1,
            "Compute the k nearest neighbors (L2 distance) from each point in the query point cloud to the dataset "
            "point cloud.  Returns (dists, corrs): (n, k) arrays, squeezed to (n,) when k == 1; corrs is int64.");
    mod.def("one_sided_hausdorff_distance", &one_sided_hausdorff_distance, py::arg("source"), py::arg("target"),
            py::arg("return_index") = true, py::arg("squared_distances") = false, py::arg("max_points_per_leaf") = 10,
            py::arg("device") = -1,
            "Compute the one sided Hausdorff distance from source to target.  Returns d or (d, i, j).");
    mod.def("estimate_point_cloud_normals_knn_internal", &estimate_point_cloud_normals_knn_internal, py::arg("points"),
            py::arg("view_dirs"), py::arg("num_neighbors"), py::arg("max_points_per_leaf") = 10,
            py::arg("drop_angle_threshold") = 1.5707963267948966, py::arg("num_threads") = 0, py::arg("random_seed") = -1,
            py::arg("device") = -1,
            "Indices of the kept points and their unit normals (plane fit to the k nearest neighbours of each point).");
    mod.def("_normals_knn_device", &normals_knn_device);
    mod.def("estimate_point_cloud_normals_ball_internal", &estimate_point_cloud_normals_ball_internal, py::arg("points"),
            py::arg("view_dirs"), py::arg("radius"), py::arg("min_pts_per_ball"), py::arg("max_pts_per_ball") = -1,
            py::arg("drop_angle_threshold") = 1.5707963267948966, py::arg("max_points_per_leaf") = 10, py::arg("num_threads") = 0,
            py::arg("weight_function") = "constant", py::arg("random_seed") = -1, py::arg("device") = -1,
            "Indices of the kept points and their unit normals (plane fit to the points in a ball around each point).");
    mod.def("_normals_ball_device", &normals_ball_device);
    mod.def("_cloud_prepare", &cloud_prepare_numpy, py::arg("points"), py::arg("device") = -1, py::arg("knn_k") = 0,
            py::arg("max_points_per_leaf") = 10);
    mod.def("_cloud_prepare_device", &cloud_prepare_device, py::arg("is_f64"), py::arg("points"), py::arg("n"), py::arg("device"),
            py::arg("stream"), py::arg("knn_k") = 0, py::arg("max_points_per_leaf") = 10);
    mod.def("_knn_prepared", &knn_prepared_numpy);
    mod.def("_knn_prepared_device", &knn_prepared_device);
    mod.def("_cloud_destroy", &cloud_destroy);
    mod.def("_cloud_points", [](uintptr_t cloud) { return (uintptr_t)pcu_b200_cloud_points((const pcu_b200_cloud*)cloud); });
    mod.def("_stats_prepared", &stats_prepared_numpy);
    mod.def("_stats_prepared_device", &stats_prepared_device);
    mod.def("_voxel_downsample_device", &voxel_downsample_device);
    mod.def("_deduplicate_device", &deduplicate_device);
    mod.def("downsample_point_cloud_poisson_disk_internal", &downsample_point_cloud_poisson_disk_internal, py::arg("v"), py::arg("radius"),
            py::arg("target_num_samples"), py::arg("random_seed"), py::arg("sample_num_tolerance"), py::arg("device") = -1);
    mod.def("_poisson_device", &poisson_device);
    // (radius trials, MIS rounds) of the last Poisson-disk call on the workspace of (device, stream); stream None = numpy path
    mod.def("_poisson_stats", [](int device, py::object stream) {
        Slot& slot = pool().get(current_device_or_default(device), stream.is_none() ? kHostKey : stream.cast<uintptr_t>());
        int64_t out[2] = {0, 0};
        { CallScope scope(slot); check(pcu_b200_debug_poisson_stats(slot.ws, out)); }
        return py::make_tuple(out[0], out[1]);
    }, py::arg("device") = -1, py::arg("stream") = py::none());
    mod.def("_pairwise_device", &pairwise_device);
    mod.def("_sinkhorn_device", &sinkhorn_device);
    mod.def("morton_encode", &morton_encode, py::arg("pts"), py::arg("num_threads") = -1, py::arg("device") = -1,
            "Encode n 3D integer points into Morton codes: (n, 3) int32 / int64 -> (n,) uint64.");
    mod.def("morton_decode", &morton_decode, py::arg("codes"), py::arg("num_threads") = -1, py::arg("device") = -1,
            "Decode n Morton codes into 3D integer points: (n,) -> (n, 3) int32.");
    mod.def("morton_add", [](const py::array& a, const py::array& b, int t, int d) { return morton_addsub(a, b, t, d, false); },
            py::arg("codes_1"), py::arg("codes_2"), py::arg("num_threads") = -1, py::arg("device") = -1,
            "Add morton codes together (corresponding to adding the vectors they encode).");
    mod.def("morton_subtract", [](const py::array& a, const py::array& b, int t, int d) { return morton_addsub(a, b, t, d, true); },
            py::arg("codes_1"), py::arg("codes_2"), py::arg("num_threads") = -1, py::arg("device") = -1,
            "Subtract morton codes from each other (codes_1 - codes_2).");
    mod.def("morton_knn", &morton_knn, py::arg("codes"), py::arg("qcodes"), py::arg("k"), py::arg("sort_dist") = true,
            py::arg("device") = -1,
            "Queries a sorted array of morton encoded points to find the (approximate) k nearest neighbors: (m, min(k, n)) int64.");
    mod.def("_chamfer_stats", &chamfer_stats, py::arg("x"), py::arg("y"), py::arg("max_points_per_leaf") = 10,
            py::arg("device") = -1);
    mod.def("_batched_chamfer", &batched_chamfer_numpy, py::arg("x"), py::arg("y"), py::arg("max_points_per_leaf") = 10,
            py::arg("device") = -1);
    mod.def("_batched_chamfer_device", &batched_chamfer_device);
    mod.def("_knn_device", &knn_device);
    mod.def("_stats_device", &stats_device);
    mod.def("_resolve_witness_device", &resolve_witness_device);
    mod.def("_debug_kd_times", [](int device, py::object stream) {
        Slot& slot = pool().get(current_device_or_default(device), stream.is_none() ? kHostKey : stream.cast<uintptr_t>());
        std::array<uint64_t, 40> t{};
        { CallScope scope(slot); check(pcu_b200_debug_kd_times(slot.ws, t.data())); }
        return t;
    }, py::arg("device") = -1, py::arg("stream") = py::none());
    mod.def("_debug_kd_tree", &debug_kd_tree, py::arg("points"), py::arg("max_points_per_leaf") = 10,
            py::arg("device") = -1);
    mod.def("_stats_nbytes", []() { return (int)sizeof(pcu_b200_nn_stats); });
    mod.def("_device_count", []() { return pcu_b200_device_count(); });
    mod.def("_launch_count", []() { return (int64_t)pcu_b200_launch_count(); });
    mod.def("_abi_version", []() { return pcu_b200_abi_version(); });
    // diagnostics address a workspace by (device, stream); stream None = the numpy path's own workspace,
    // device < 0 = the device a call that names none would use
    auto key_of = [](const py::object& stream) { return stream.is_none() ? kHostKey : stream.cast<uintptr_t>(); };
    mod.def("_current_device", []() { return pcu_b200_current_device(); });
    mod.def("_grid_refinement", [key_of](int device, py::object stream) {
        float m[2] = {1.f, 1.f};
        pcu_b200_workspace_grid_refinement(pool().get(current_device_or_default(device), key_of(stream)).ws, m);
        return py::make_tuple(m[0], m[1]);
    }, py::arg("device") = -1, py::arg("stream") = py::none());
    mod.def("_workspace_bytes", [key_of](int device, py::object stream) {
        return (int64_t)pcu_b200_workspace_bytes(pool().get(current_device_or_default(device), key_of(stream)).ws);
    }, py::arg("device") = -1, py::arg("stream") = py::none());
    mod.def("_workspace_exists", [key_of](int device, py::object stream) {
        std::lock_guard<std::mutex> lock(pool().mu);
        return pool().items.count(std::make_pair(current_device_or_default(device), key_of(stream))) != 0;
    }, py::arg("device") = -1, py::arg("stream") = py::none());
    mod.def("_set_profiling", [key_of](int device, py::object stream, bool on) {
        check(pcu_b200_workspace_set_profiling(pool().get(current_device_or_default(device), key_of(stream)).ws, on ? 1 : 0));
    });
    mod.def("_last_profile", [key_of](int device, py::object stream) {
        float ms[10];
        const int n = pcu_b200_workspace_last_profile(pool().get(current_device_or_default(device), key_of(stream)).ws, ms, 10);
        py::dict d;
        for (int i = 0; i < n; ++i) d[py::str(pcu_b200_profile_stage_name(i))] = ms[i];
        return d;
    });
    mod.def("_set_defaults", [](float cell_occupancy, int disable_tie_replay, int binning, int host_staging) {
        if (host_staging < 0 || host_staging > 2) throw py::value_error("host_staging must be 0 (auto), 1 (always) or 2 (never)");
        defaults().host_staging = host_staging;
        if (disable_tie_replay < 0 || disable_tie_replay > 3) throw py::value_error("disable_tie_replay must be 0 .. 3");
        if (binning < 0 || binning > 2) throw py::value_error("binning must be 0 (auto), 1 (multi-launch) or 2 (one CTA per cloud)");
        defaults().occupancy = cell_occupancy;
        defaults().disable_replay = disable_tie_replay;
        defaults().binning = binning;
    }, py::arg("cell_occupancy") = 0.f, py::arg("disable_tie_replay") = 0, py::arg("binning") = 0, py::arg("host_staging") = 0);
    mod.def("_pinned_empty", [](py::ssize_t rows, py::ssize_t cols, bool is_f64) {
        return is_f64 ? pinned_cloud<double>(rows, cols) : pinned_cloud<float>(rows, cols);
    });
    mod.def("_release_workspaces", []() { pool().clear(); });
    mod.def("_release_pinned_results", []() { pinned_pool().clear(false); });
    // destroy workspaces and cached pinned blocks before the CUDA context goes away at interpreter exit
    py::module_::import("atexit").attr("register")(py::cpp_function([]() { pool().clear(); pinned_pool().clear(true); }));
}
