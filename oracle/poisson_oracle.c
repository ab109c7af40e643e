/* poisson_oracle.c -- TEST INFRASTRUCTURE: the Poisson-disk down-sampling result of this library, restated
 * sequentially in plain C (no reference source: the reference's sampler is libigl's, which is not in its tree).
 *
 *   key(i)  = (h(i) << 32) | i,  h(i) = mix32(seed ^ mix32(i * 0x9e3779b9 + 0x85ebca6b))
 *   i and j conflict iff d2(i, j) < r2:  d2 = ((dx*dx) + dy*dy) + dz*dz and r2 = r*r, every operation rounded in the
 *   cloud's precision T (compiled with -ffp-contract=off);
 *   the samples are the greedy independent set in ascending key order, returned as ascending rows.
 * Conflicts are found through a hash grid of the samples accepted so far, with cells no smaller than the radius
 * (widened by 1e-4 against the rounding of the cell computation), so the 27 cells around a point hold every sample it
 * can conflict with.
 *
 * target > 0: the radius search of the reference binding (src/sample_point_cloud.cpp:278-326), operation for operation
 * in T, with one addition: the doubling loop also stops once the radius cannot grow any more (zero or not finite),
 * where the reference would never end.  The radii of all trials and their sample counts are reported. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static uint32_t mix32(uint32_t h) {
    h ^= h >> 16; h *= 0x7feb352du; h ^= h >> 15; h *= 0x846ca68bu; h ^= h >> 16;
    return h;
}

static int cmp_u64(const void* a, const void* b) {
    const uint64_t x = *(const uint64_t*)a, y = *(const uint64_t*)b;
    return x < y ? -1 : (x > y ? 1 : 0);
}

/* rows in ascending key order */
static uint32_t* key_order(long long n, uint32_t seed) {
    uint64_t* keys = (uint64_t*)malloc(sizeof(uint64_t) * (size_t)n);
    uint32_t* order = (uint32_t*)malloc(sizeof(uint32_t) * (size_t)n);
    if (!keys || !order) { free(keys); free(order); return NULL; }
    for (long long i = 0; i < n; ++i) {
        const uint32_t h = mix32(seed ^ mix32((uint32_t)i * 0x9e3779b9u + 0x85ebca6bu));
        keys[i] = ((uint64_t)h << 32) | (uint64_t)(uint32_t)i;
    }
    qsort(keys, (size_t)n, sizeof(uint64_t), cmp_u64);
    for (long long k = 0; k < n; ++k) order[k] = (uint32_t)(keys[k] & 0xffffffffu);
    free(keys);
    return order;
}

typedef struct { long long c[3]; int head; int used; } Cell;

static uint64_t cell_hash(const long long c[3]) {
    uint64_t h = (uint64_t)c[0] * 0x9e3779b97f4a7c15ull ^ (uint64_t)c[1] * 0xc2b2ae3d27d4eb4full ^ (uint64_t)c[2] * 0x165667b19e3779f9ull;
    h ^= h >> 29; h *= 0xbf58476d1ce4e5b9ull; h ^= h >> 32;
    return h;
}

static Cell* find_cell(Cell* table, uint64_t mask, const long long c[3], int create) {
    for (uint64_t s = cell_hash(c) & mask;; s = (s + 1) & mask) {
        Cell* e = table + s;
        if (!e->used) {
            if (!create) return NULL;
            e->used = 1; e->c[0] = c[0]; e->c[1] = c[1]; e->c[2] = c[2]; e->head = -1;
            return e;
        }
        if (e->c[0] == c[0] && e->c[1] == c[1] && e->c[2] == c[2]) return e;
    }
}

/* one trial at radius r (in T): r2 = r * r in T; records the radius and the count */
#define TRIAL(SUF, T, r)                                                                                               \
    do {                                                                                                               \
        const T r_ = (r);                                                                                              \
        const T r2_ = r_ * r_;                                                                                         \
        count = greedy_##SUF(v, n, r2_, order, keep);                                                                  \
        if (count < 0) failed = 1;                                                                                     \
        if (radii && trials < cap) radii[trials] = (double)r_;                                                         \
        if (counts && trials < cap) counts[trials] = count;                                                            \
        ++trials;                                                                                                      \
    } while (0)

#define DEFINE_POISSON(T, SUF)                                                                                         \
static T dist2_##SUF(const T* a, const T* b) {                                                                        \
    const T dx = a[0] - b[0], dy = a[1] - b[1], dz = a[2] - b[2];                                                      \
    const T xx = dx * dx, yy = dy * dy, zz = dz * dz;                                                                  \
    const T s = xx + yy;                                                                                               \
    return s + zz;                                                                                                     \
}                                                                                                                      \
/* one radius trial: keep[row] = 1 for the samples; returns their number (-1: out of memory) */                       \
static long long greedy_##SUF(const T* v, long long n, T r2, const uint32_t* order, unsigned char* keep) {             \
    memset(keep, 0, (size_t)n);                                                                                        \
    if (!(r2 > (T)0)) { memset(keep, 1, (size_t)n); return n; }                                                        \
    double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};                          \
    for (long long i = 0; i < n; ++i)                                                                                  \
        for (int a = 0; a < 3; ++a) {                                                                                  \
            const double x = (double)v[3 * i + a];                                                                     \
            if (x < lo[a]) lo[a] = x;                                                                                  \
            if (x > hi[a]) hi[a] = x;                                                                                  \
        }                                                                                                              \
    double ext = 0.0;                                                                                                  \
    for (int a = 0; a < 3; ++a) if (hi[a] - lo[a] > ext) ext = hi[a] - lo[a];                                          \
    double h = sqrt((double)r2) * (1.0 + 1e-4);                                                                        \
    if (h < ext * 0x1p-30) h = ext * 0x1p-30;      /* cell indices stay below 2^30 */                                  \
    const int flat = !(h > 0.0) || !isfinite(h) || !isfinite(ext);                                                     \
    uint64_t slots = 64;                                                                                               \
    while (slots < 2 * (uint64_t)n) slots <<= 1;                                                                       \
    Cell* table = (Cell*)calloc((size_t)slots, sizeof(Cell));                                                          \
    int* next = (int*)malloc(sizeof(int) * (size_t)n);                                                                 \
    if (!table || !next) { free(table); free(next); return -1; }                                                       \
    long long count = 0;                                                                                               \
    for (long long k = 0; k < n; ++k) {                                                                                \
        const long long i = order[k];                                                                                  \
        const T* p = v + 3 * i;                                                                                        \
        long long c[3];                                                                                                \
        for (int a = 0; a < 3; ++a) {                                                                                  \
            const double t = flat ? 0.0 : floor(((double)p[a] - lo[a]) / h);                                           \
            c[a] = t == t ? (long long)t : 0;                                                                          \
        }                                                                                                              \
        int clash = 0;                                                                                                 \
        for (int dz = -1; dz <= 1 && !clash; ++dz)                                                                     \
            for (int dy = -1; dy <= 1 && !clash; ++dy)                                                                 \
                for (int dx = -1; dx <= 1 && !clash; ++dx) {                                                           \
                    const long long nc[3] = {c[0] + dx, c[1] + dy, c[2] + dz};                                         \
                    const Cell* e = find_cell(table, slots - 1, nc, 0);                                                \
                    for (int j = e ? e->head : -1; j >= 0; j = next[j])                                                \
                        if (dist2_##SUF(p, v + 3 * (long long)j) < r2) { clash = 1; break; }                           \
                }                                                                                                      \
        if (clash) continue;                                                                                           \
        Cell* e = find_cell(table, slots - 1, c, 1);                                                                   \
        next[i] = e->head;                                                                                             \
        e->head = (int)i;                                                                                              \
        keep[i] = 1;                                                                                                   \
        ++count;                                                                                                       \
    }                                                                                                                  \
    free(table);                                                                                                       \
    free(next);                                                                                                        \
    return count;                                                                                                      \
}                                                                                                                      \
/* Returns the number of samples (rows ascending in out_idx, capacity n); -1 on an argument error, -2 out of memory.   \
 * radii / counts (capacity cap, may be NULL): every trial's radius and sample count; *n_trials their number. */      \
long long pcu_oracle_poisson_##SUF(const T* v, long long n, double radius, int target, uint32_t seed, float tol,     \
                                   int32_t* out_idx, double* radii, long long* counts, int cap, int* n_trials) {      \
    *n_trials = 0;                                                                                                     \
    if (target <= 0 && radius <= 0.0) return -1;                                                                       \
    if (tol > 1.0 || tol <= 0.0) return -1;                                                                            \
    if (n <= 0 || n >= 0x7fffffffLL) return -1;                                                                        \
    if (target > 0 && (long long)target >= n) {                                                                        \
        for (long long i = 0; i < n; ++i) out_idx[i] = (int32_t)i;                                                     \
        return n;                                                                                                      \
    }                                                                                                                  \
    uint32_t* order = key_order(n, seed);                                                                              \
    unsigned char* keep = (unsigned char*)malloc((size_t)n);                                                           \
    if (!order || !keep) { free(order); free(keep); return -2; }                                                       \
    long long count = 0;                                                                                               \
    int trials = 0;                                                                                                    \
    int failed = 0;                                                                                                    \
    if (target <= 0) {                                                                                                 \
        TRIAL(SUF, T, (T)radius);                                                                                        \
    } else {                                                                                                           \
        const unsigned long long num_min = (unsigned long long)(int)((T)target * (T)(1.0f - tol));                     \
        const unsigned long long num_max = (unsigned long long)(int)((T)target * (T)(1.0f + tol));                     \
        T bmin[3], bmax[3];                                                                                            \
        for (int a = 0; a < 3; ++a) { bmin[a] = v[a]; bmax[a] = v[a]; }                                                \
        for (long long i = 1; i < n; ++i)                                                                              \
            for (int a = 0; a < 3; ++a) {                                                                              \
                if (v[3 * i + a] < bmin[a]) bmin[a] = v[3 * i + a];                                                    \
                if (v[3 * i + a] > bmax[a]) bmax[a] = v[3 * i + a];                                                    \
            }                                                                                                          \
        T ext[3];                                                                                                      \
        for (int a = 0; a < 3; ++a) ext[a] = bmax[a] - bmin[a];                                                        \
        const T e0 = ext[0] * ext[0], e1 = ext[1] * ext[1], e2 = ext[2] * ext[2];                                      \
        const T s01 = e0 + e1;                                                                                         \
        const T bbsize = (T)sqrt((double)(T)(s01 + e2));                                                               \
        T rmin = (T)((double)bbsize / 50.0), rmax = (T)((double)bbsize / 50.0);                                        \
        do {                                                                                                           \
            rmin = (T)((double)rmin / 2.0);                                                                            \
            TRIAL(SUF, T, rmin);                                                                                         \
        } while (!failed && (unsigned long long)count < (unsigned long long)target);                                   \
        do {                                                                                                           \
            rmax = (T)((double)rmax * 2.0);                                                                            \
            TRIAL(SUF, T, rmax);                                                                                         \
        } while (!failed && (unsigned long long)count > (unsigned long long)target && (T)((double)rmax * 2.0) > rmax); \
        int iter = 0;                                                                                                  \
        while (!failed && iter < 20 && ((unsigned long long)count < num_min || (unsigned long long)count > num_max)) { \
            iter += 1;                                                                                                 \
            const T cur = (T)((double)(T)(rmin + rmax) / 2.0);                                                         \
            TRIAL(SUF, T, cur);                                                                                          \
            if (count > (long long)target) rmin = cur;                                                                 \
            if (count < (long long)target) rmax = cur;                                                                 \
        }                                                                                                              \
    }                                                                                                                  \
    *n_trials = trials;                                                                                                \
    long long m = 0;                                                                                                   \
    if (!failed) for (long long i = 0; i < n; ++i) if (keep[i]) out_idx[m++] = (int32_t)i;                             \
    free(order);                                                                                                       \
    free(keep);                                                                                                        \
    return failed ? -2 : m;                                                                                            \
}

DEFINE_POISSON(float, f32)
DEFINE_POISSON(double, f64)
