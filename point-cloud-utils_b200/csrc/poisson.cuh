// poisson.cuh -- Poisson-disk down-sampling of a point cloud (downsample_point_cloud_poisson_disk).
//
// Replaces the binding of src/sample_point_cloud.cpp:240-333, whose sampler is libigl's sequential, rand()-seeded
// blue-noise loop (fetched at build time, not in the reference tree).  The result computed here is defined instead
// as the GREEDY SEQUENTIAL MAXIMAL INDEPENDENT SET in priority order:
//     key(i) = (h(i) << 32) | i,   h(i) = mix32(seed ^ mix32(i * 0x9e3779b9 + 0x85ebca6b))
//     i and j conflict iff d2(i, j) < r2     (d2 the reference-rounded squared distance of common.cuh, r2 = fl(r * r))
//     visit the points by ascending key, accept a point iff it conflicts with no point accepted before it.
// The set is unique, so it does not depend on thread scheduling, and it is separated (no two samples conflict) and
// maximal (every other point conflicts with a sample).  Rows come out ascending.
//
// Pipeline of one call: keys -> stable radix sort of (h, row) (sort.cuh) -> the points gathered into key order, so a
// point's RANK is its priority -> per radius: the binning of grid.cuh over the ranked copy (cells no finer than half
// the radius), cell_order_kernel (normals.cuh: every cell in rank order), then the parallel greedy MIS of Blelloch,
// Fineman and Shun (SPAA 2012) on a one-byte state per rank, in ONE cooperative launch whose rounds are separated by
// grid-wide barriers:
//     an undecided point walks the LOWER-ranked points of its ball (a cell's run stops at the first rank >= its own);
//     a selected one removes it, an undecided one makes it wait for the next round, none at all selects it;
//     a point that becomes selected pushes "removed" to the higher-ranked undecided points of its ball.
// States only move forward (undecided -> selected | removed) and each final state is implied by lower-ranked final
// states alone, so a read that races with a write of the same round sees an older, still valid state: the outcome
// is the sequential one.  The lowest-ranked undecided point always decides, so the loop ends.  The push keeps the
// total work O(n * points per ball): a point is walked over by the pushes of the few samples around it instead of
// re-walking its ball every round.  Finally flags by row -> keep_count / keep_offsets (normals.cuh) -> int32 scatter.
#pragma once
#include "common.cuh"
#include "sort.cuh"
#include "normals.cuh"

namespace pcu {

using PoissonRec = SortRec<uint32_t, 1>;

constexpr unsigned char kUndecided = 0, kSelected = 1, kRemoved = 2;

__device__ __forceinline__ unsigned poisson_hash(unsigned seed, unsigned i) {
    return mix32(seed ^ mix32(i * 0x9e3779b9u + 0x85ebca6bu));
}

// record i = (h(i), i); a stable sort on h then orders by the full key (h, i)
__global__ void __launch_bounds__(kThreads) poisson_keys_kernel(long long n, unsigned seed, PoissonRec* __restrict__ recs) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    PoissonRec r;
    r.key[0] = poisson_hash(seed, (unsigned)i);
    r.idx = (uint32_t)i;
    store_rec(recs + i, r);
}

// ranked[rank] = points[row], row_of[rank] = row
template <typename T>
__global__ void __launch_bounds__(kThreads) poisson_gather_kernel(const PoissonRec* __restrict__ sorted, long long n, const T* __restrict__ pts,
                                                                  T* __restrict__ ranked, int* __restrict__ row_of) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const long long row = (long long)sorted[k].idx;
    ranked[3 * k] = pts[3 * row];
    ranked[3 * k + 1] = pts[3 * row + 1];
    ranked[3 * k + 2] = pts[3 * row + 2];
    row_of[k] = (int)row;
}

// Per-column minimum / maximum of the cloud (the bounding box of the target_num_samples search), as order-preserving
// integers: box[0..2] minima (initialised to all ones), box[3..5] maxima (initialised to zero).
template <typename T>
__global__ void __launch_bounds__(kThreads) poisson_bbox_kernel(const T* __restrict__ pts, long long n, typename Real<T>::bits_t* __restrict__ box) {
    using bits_t = typename Real<T>::bits_t;
    bits_t lo[3], hi[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) { lo[a] = ~(bits_t)0; hi[a] = (bits_t)0; }
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            T v = pts[3 * i + a];
            if (v == (T)0) v = (T)0;   // -0 and +0 are the same coordinate
            const bits_t u = ordered<T>(v);
            lo[a] = u < lo[a] ? u : lo[a];
            hi[a] = u > hi[a] ? u : hi[a];
        }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        atomicMin(box + a, lo[a]);
        atomicMax(box + 3 + a, hi[a]);
    }
}

// The cells a ball of squared radius r2 around q can touch (the box of walk_ball), and a walk over them that calls
// visit(p) for every point p of the ball with rank below (kLower) / above (!kLower) q's own, in rank order per cell,
// until visit returns false.  Cells (and rows of cells) whose wall gap already reaches r2 are skipped; the gaps add
// up in the order of the metric, so the skip is exact.
template <typename T, bool kLower, typename Visit>
__device__ __forceinline__ void walk_ranked(const Cloud<T>& cl, const GridHeader<T>& g, const Pt<T>& q, T r2, Visit&& visit) {
    using R = Real<T>;
    const T eps = sizeof(T) == 4 ? (T)1.1920929e-7 : (T)2.220446049250313e-16;
    const T reach = R::root(r2) * ((T)1 + (T)8 * eps) + (sizeof(T) == 4 ? (T)1.1754944e-38 : (T)2.2250738585072014e-308);
    int lo[3], hi[3], c[3];
    const T qv[3] = {q.x, q.y, q.z};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        lo[a] = cell_of<T>(sub_down<T>(qv[a], reach), g.origin[a], g.inv_h, g.dim[a]);
        hi[a] = cell_of<T>(add_up<T>(qv[a], reach), g.origin[a], g.inv_h, g.dim[a]);
        c[a] = cell_of<T>(qv[a], g.origin[a], g.inv_h, g.dim[a]);
    }
    const int st = g.stride;
    const T* lo_x = cl.wall_lo;           const T* hi_x = cl.wall_hi;
    const T* lo_y = cl.wall_lo + st;      const T* hi_y = cl.wall_hi + st;
    const T* lo_z = cl.wall_lo + 2 * st;  const T* hi_z = cl.wall_hi + 2 * st;
    const long long me = (long long)q.i;
    for (int z = lo[2]; z <= hi[2]; ++z) {
        const T bz = z < c[2] ? sq_gap<T>(q.z, lo_z[z + 1]) : (z > c[2] ? sq_gap<T>(q.z, hi_z[z]) : (T)0);
        if (!(bz < r2)) continue;
        for (int y = lo[1]; y <= hi[1]; ++y) {
            const T by = y < c[1] ? sq_gap<T>(q.y, lo_y[y + 1]) : (y > c[1] ? sq_gap<T>(q.y, hi_y[y]) : (T)0);
            if (!(R::add(by, bz) < r2)) continue;
            const unsigned row = (unsigned)((z * g.dim[1] + y) * g.dim[0]);
            for (int x = lo[0]; x <= hi[0]; ++x) {
                const T bx = x < c[0] ? sq_gap<T>(q.x, lo_x[x + 1]) : (x > c[0] ? sq_gap<T>(q.x, hi_x[x]) : (T)0);
                if (!(R::add(R::add(bx, by), bz) < r2)) continue;
                const unsigned a = cl.cell_start[row + x], b = cl.cell_start[row + x + 1];
                if (kLower) {
                    for (unsigned j = a; j < b; ++j) {
                        const Pt<T> p = load_pt<T>(cl.sorted + j);
                        if ((long long)p.i >= me) break;          // the rest of the cell ranks after q
                        if (dist2<T>(q.x, q.y, q.z, p.x, p.y, p.z) < r2 && !visit(p)) return;
                    }
                } else {
                    for (unsigned j = b; j-- > a;) {
                        const Pt<T> p = load_pt<T>(cl.sorted + j);
                        if ((long long)p.i <= me) break;          // the rest of the cell ranks before q
                        if (dist2<T>(q.x, q.y, q.z, p.x, p.y, p.z) < r2 && !visit(p)) return;
                    }
                }
            }
        }
    }
}

// Grid-wide barrier of a cooperative launch (every CTA is resident): bar[0] arrivals, bar[1] generation.
__device__ __forceinline__ void poisson_grid_sync(unsigned* bar) {
    __syncthreads();
    if (threadIdx.x == 0) {
        volatile unsigned* vb = bar;
        const unsigned gen = vb[1];
        __threadfence();
        if (atomicAdd(bar, 1u) == gridDim.x - 1) {
            vb[0] = 0u;
            __threadfence();
            atomicAdd(bar + 1, 1u);
        } else {
            while (vb[1] == gen) __nanosleep(64);
        }
        __threadfence();
    }
    __syncthreads();
}

// counters: 5 words, zeroed before the launch (undecided points left by a round, triple-buffered so that a round can
// clear the counter of the next one while slow CTAs may still read the previous one), then the 2 words of the grid
// barrier; rounds_out accumulates the rounds.
template <typename T>
__global__ void __launch_bounds__(kThreads, 4) poisson_mis_kernel(Cloud<T> cl, T r2, unsigned char* __restrict__ state,
                                                               unsigned* __restrict__ counters, unsigned long long* __restrict__ rounds_out) {
    __shared__ GridHeader<T> g;
    __shared__ unsigned block_left;
    if (threadIdx.x == 0) g = *cl.grid;
    __syncthreads();
    volatile unsigned char* vs = state;
    const long long n = cl.n;
    const long long stride = (long long)gridDim.x * blockDim.x;
    unsigned round = 0;
    for (;; ++round) {
        if (threadIdx.x == 0) block_left = 0u;
        if (blockIdx.x == 0 && threadIdx.x == 0) counters[(round + 1) % 3] = 0u;   // last read two barriers ago
        __syncthreads();
        unsigned left = 0u;
        for (long long pos = (long long)blockIdx.x * blockDim.x + threadIdx.x; pos < n; pos += stride) {
            const Pt<T> q = load_pt<T>(cl.sorted + pos);
            if (vs[q.i] != kUndecided) continue;
            unsigned char verdict = kSelected;
            walk_ranked<T, true>(cl, g, q, r2, [&](const Pt<T>& p) {
                const unsigned char s = vs[p.i];
                if (s == kRemoved) return true;
                verdict = s == kSelected ? kRemoved : kUndecided;
                return false;
            });
            if (verdict == kUndecided) { ++left; continue; }
            vs[q.i] = verdict;
            if (verdict == kSelected)
                walk_ranked<T, false>(cl, g, q, r2, [&](const Pt<T>& p) {
                    if (vs[p.i] == kUndecided) vs[p.i] = kRemoved;
                    return true;
                });
        }
        if (left) atomicAdd(&block_left, left);
        __syncthreads();
        if (threadIdx.x == 0 && block_left) atomicAdd(counters + round % 3, block_left);
        poisson_grid_sync(counters + 3);
        if (*(volatile unsigned*)(counters + round % 3) == 0u) break;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(rounds_out, (unsigned long long)(round + 1));
}

// keep[row_of[rank]] = state[rank] is "selected"
__global__ void __launch_bounds__(kThreads) poisson_flag_kernel(const unsigned char* __restrict__ state, const int* __restrict__ row_of, long long n,
                                                                unsigned char* __restrict__ keep) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    keep[row_of[k]] = state[k] == kSelected ? 1 : 0;
}

// after keep_count / keep_offsets: the kept rows, ascending, as int32
__global__ void __launch_bounds__(kThreads) poisson_scatter_kernel(const unsigned char* __restrict__ keep, long long n,
                                                                   const unsigned* __restrict__ block_offset, int* __restrict__ out_idx) {
    __shared__ unsigned warp_sum[kThreads / 32];
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned mine = i < n ? keep[i] : 0u;
    const unsigned ballot = __ballot_sync(0xffffffffu, mine != 0u);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) warp_sum[w] = __popc(ballot);
    __syncthreads();
    unsigned before = block_offset[blockIdx.x];
    for (int j = 0; j < w; ++j) before += warp_sum[j];
    if (mine) out_idx[before + __popc(ballot & ((1u << lane) - 1u))] = (int)i;
}

// every row (r2 not > 0: nothing conflicts; target >= n)
__global__ void __launch_bounds__(kThreads) poisson_all_rows_kernel(long long n, int* __restrict__ out_idx, long long* __restrict__ out_count) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out_idx[i] = (int)i;
    if (i == 0) *out_count = n;
}

}  // namespace pcu
