// azb_enum.cuh — every free tree on N <= 32 vertices by index (azb_free_trees) and the exact k best of an index range by the
// c21 cost (azb_exhaustive_best).  The enumeration is defined in include/azb.h; DESIGN.md §4.10 has the design.
//
// Tables (built on the host once per handle, on first use):
//   P[r][g]  r = 0..N-1, g = 0..G-1 (G = rooted-tree ids of size <= (N-1)/2): the number of non-increasing sequences of
//            ids <= g whose sizes sum to r.  P[r][g] = P[r][g-1] + P[r - size(g)][g], P[r][-1] = (r == 0).
//   rp       the preorder parent array of every rooted tree of size <= N/2, size by size in id order.
// Unranking one sequence element: the sequences of sum r with first element < g number P[r][g-1], so the element is the
// smallest g <= bound with P[r][g] > x; the warp finds it by a 32-ary search (each lane probes one point of the interval).
#pragma once
#include <cub/device/device_radix_sort.cuh>
#include <cuda/std/tuple>

#include <algorithm>
#include <vector>

#include "azb_common.cuh"
#include "azb_cost.cuh"

#define AZB_ENUM_MAX_N 32
#define AZB_ENUM_MAX_S 16            // largest rooted tree a free tree is built from: N / 2
#define AZB_ENUM_CHUNK (1u << 22)    // trees per chunk of azb_exhaustive_best / per launch of azb_free_trees

struct AzbEnum {                      // kernel parameter: the tables of one N
    const unsigned long long *P;      // [N][G]
    const uint8_t *rp;                // rooted preorder parent arrays
    unsigned long long U;             // unicentroidal trees: indices [0, U)
    unsigned long long rpo[AZB_ENUM_MAX_S + 2];  // byte offset in rp of the arrays of size s
    uint32_t off[AZB_ENUM_MAX_S + 2];  // first id of size s (s = 1..N/2 + 1; off[N/2 + 1] = number of ids)
    uint32_t n, G, smax;              // N, columns of P, N / 2
};

struct AzbEnumCand {                  // one candidate of the running top k, sorted by (key bits, index)
    unsigned long long key;           // bits of (double)mu + lambda_1 (> 0, so the bits order like the values)
    unsigned long long idx;
};
struct AzbEnumByKey {
    __host__ __device__ cuda::std::tuple<unsigned long long &, unsigned long long &> operator()(AzbEnumCand &c) const {
        return {c.key, c.idx};
    }
};

// ---- host: counts and tables ----
// A000055(n) and the unicentroidal count U, without tables: a knapsack over every rooted tree of size <= (n-1)/2 (its
// A000081(s) types of size s, each any number of times) counts the multisets of subtrees of the centroid.
static inline void azb_enum_counts(uint32_t n, uint64_t *U, uint64_t *total) {
    std::vector<uint64_t> f(n, 0);
    f[0] = 1;
    for (uint32_t s = 1; s <= (n - 1) / 2; ++s) {
        const uint64_t types = f[s - 1];  // A000081(s): sequences of sum s - 1 over the sizes < s
        for (uint64_t t = 0; t < types; ++t)
            for (uint32_t r = s; r < n; ++r) f[r] += f[r - s];
    }
    *U = f[n - 1];
    const uint64_t half = n % 2 == 0 ? f[n / 2 - 1] : 0;  // A000081(n / 2)
    *total = *U + half * (half + 1) / 2;
}

__host__ __device__ __forceinline__ uint32_t azb_enum_size(const AzbEnum &E, uint32_t g) {
    uint32_t s = 1;
    while (s < E.smax && E.off[s + 1] <= g) ++s;
    return s;
}

// host tables; E.P / E.rp are left for the caller to point at the device copies
static inline void azb_enum_build(uint32_t n, AzbEnum &E, std::vector<unsigned long long> &P, std::vector<uint8_t> &rp) {
    E = AzbEnum{};
    E.n = n;
    E.smax = n / 2;
    const uint32_t su = (n - 1) / 2;  // largest subtree of a unique centroid
    std::vector<unsigned long long> last(n, 0);  // column g - 1
    last[0] = 1;
    std::vector<uint32_t> cnt(E.smax + 1, 0);
    E.off[1] = 0;
    // sizes up to su give the columns of P; the count of size su + 1 (= n / 2 for even n) is read off the last column
    std::vector<unsigned long long> cols;  // column-major while G is not known yet
    for (uint32_t s = 1; s <= E.smax; ++s) {
        cnt[s] = (uint32_t)last[s - 1];
        E.off[s + 1] = E.off[s] + cnt[s];
        if (s > su) break;
        for (uint32_t t = 0; t < cnt[s]; ++t) {
            for (uint32_t r = s; r < n; ++r) last[r] += last[r - s];  // in place: row r - s is already column g's
            cols.insert(cols.end(), last.begin(), last.end());
        }
    }
    E.G = E.off[su + 1];
    P.assign((size_t)n * E.G, 0ull);
    for (uint32_t g = 0; g < E.G; ++g)
        for (uint32_t r = 0; r < n; ++r) P[(size_t)r * E.G + g] = cols[(size_t)g * n + r];
    E.U = P[(size_t)(n - 1) * E.G + E.G - 1];
    // rooted preorder arrays: root 0, then each child's array in sequence order
    size_t bytes = 0;
    for (uint32_t s = 1; s <= E.smax; ++s) {
        E.rpo[s] = bytes;
        bytes += (size_t)cnt[s] * s;
    }
    E.rpo[E.smax + 1] = bytes;
    rp.assign(bytes, 0);
    for (uint32_t s = 2; s <= E.smax; ++s) {
        for (uint32_t t = 0; t < cnt[s]; ++t) {
            uint8_t *out = rp.data() + E.rpo[s] + (size_t)t * s;
            unsigned long long x = t;
            uint32_t r = s - 1, b = E.off[s] - 1, base = 1;
            while (r > 0) {
                const unsigned long long *row = P.data() + (size_t)r * E.G;
                const uint32_t g = (uint32_t)(std::upper_bound(row, row + b + 1, x) - row);
                if (g) x -= row[g - 1];
                const uint32_t cs = azb_enum_size(E, g);
                const uint8_t *src = rp.data() + E.rpo[cs] + (size_t)(g - E.off[cs]) * cs;
                out[base] = 0;
                for (uint32_t v = 1; v < cs; ++v) out[base + v] = (uint8_t)(base + src[v]);
                base += cs;
                r -= cs;
                b = g;
            }
        }
    }
}

// ---- device: one warp generates one tree ----
// the smallest g in [lo, hi] with row[g] > x (row[hi] > x): each round narrows the interval 32-fold
__device__ __forceinline__ uint32_t azb_enum_search(const unsigned long long *__restrict__ row, unsigned long long x, uint32_t lo,
                                                    uint32_t hi, int lane) {
    const uint32_t FULL = 0xffffffffu;
#pragma unroll 1
    for (;;) {
        const uint32_t stride = (hi - lo + 32u) >> 5;
        const uint32_t q = min(lo + ((uint32_t)lane + 1u) * stride - 1u, hi);  // lane 31 probes hi
        const uint32_t bal = __ballot_sync(FULL, __ldg(row + q) > x);
        const int f = __ffs(bal) - 1;
        const uint32_t nhi = __shfl_sync(FULL, q, f), prev = __shfl_sync(FULL, q, f > 0 ? f - 1 : 0);
        if (stride == 1u) return nhi;
        lo = f > 0 ? prev + 1u : lo;
        hi = nhi;
    }
}

// tree `idx` of the enumeration into par[0..N) (shared memory).  Warp-collective.
__device__ __forceinline__ void azb_enum_tree(const AzbEnum &E, unsigned long long idx, uint8_t *par, int lane) {
    const uint32_t n = E.n;
    if (idx < E.U) {
        unsigned long long x = idx;
        uint32_t r = n - 1, b = E.G - 1, base = 1;
        if (lane == 0) par[0] = 0;
#pragma unroll 1
        while (r > 0) {
            const unsigned long long *row = E.P + (size_t)r * E.G;
            const uint32_t hi = min(b, E.off[min(r, E.smax) + 1] - 1u);  // ids of size > r cannot come next
            const uint32_t g = azb_enum_search(row, x, 0u, hi, lane);
            if (g) x -= __ldg(row + g - 1);
            const uint32_t s = azb_enum_size(E, g);
            const uint8_t *src = E.rp + E.rpo[s] + (size_t)(g - E.off[s]) * s;
            if ((uint32_t)lane < s) par[base + lane] = lane == 0 ? 0 : (uint8_t)(base + __ldg(src + lane));
            base += s;
            r -= s;
            b = g;
        }
    } else {
        // bicentroidal: the pair i >= j of rooted trees of size h = N / 2 at U + i(i+1)/2 + j
        const unsigned long long rem = idx - E.U;
        unsigned long long i = (unsigned long long)((sqrt(8.0 * (double)rem + 1.0) - 1.0) * 0.5);
        while (i * (i + 1) / 2 > rem) --i;
        while ((i + 1) * (i + 2) / 2 <= rem) ++i;
        const unsigned long long j = rem - i * (i + 1) / 2;
        const uint32_t h = E.smax;
        const uint8_t *ti = E.rp + E.rpo[h] + i * h, *tj = E.rp + E.rpo[h] + j * h;
        if ((uint32_t)lane < h) {
            par[1 + lane] = lane == 0 ? 0 : (uint8_t)(1 + __ldg(tj + lane));  // tree j at 1 .. h, its root under vertex 0
            if (lane == 0) {
                par[0] = 0;
            } else {
                const uint32_t p = __ldg(ti + lane);  // tree i's other vertices at h + 1 .. N - 1
                par[h + lane] = p == 0 ? 0 : (uint8_t)(h + p);
            }
        }
    }
    __syncwarp();
}

// azb_free_trees / the parent arrays of the result: tree t is idx0 + t, or list[t].idx when list is given
__global__ void __launch_bounds__(256) azb_enum_trees_kernel(const AzbEnum E, unsigned long long idx0, const AzbEnumCand *list,
                                                             uint32_t m, uint8_t *__restrict__ out) {
    __shared__ __align__(16) uint8_t sm_par[8][64];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t nw = gridDim.x * 8u;
    uint8_t *par = sm_par[warp];
#pragma unroll 1
    for (uint32_t t = blockIdx.x * 8u + warp; t < m; t += nw) {
        azb_enum_tree(E, list ? list[t].idx : idx0 + t, par, lane);
        if ((uint32_t)lane < E.n) out[(size_t)t * E.n + lane] = par[lane];
        __syncwarp();
    }
}

// the hot path of azb_exhaustive_best: every tree of [idx0, idx0 + count) generated and costed by one warp; a tree whose
// key bits are <= *thr (the k-th best key of the earlier chunks) becomes a candidate; *n_below += trees with key < bound
template <int DEPTH>
__global__ void __launch_bounds__(256) azb_enum_best_kernel(const AzbEnum E, unsigned long long idx0, uint32_t count,
                                                            const unsigned long long *__restrict__ thr, double bound,
                                                            AzbEnumCand *__restrict__ cand, uint32_t *__restrict__ n_cand,
                                                            unsigned long long *__restrict__ n_below, uint32_t *__restrict__ err) {
    __shared__ __align__(16) uint8_t scratch_bytes[8][AZB_COST_SCRATCH_BYTES];
    __shared__ __align__(16) uint8_t sm_par[8][64];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t nw = gridDim.x * 8u;
    uint8_t *par = sm_par[warp];
    CostScratch *cs = reinterpret_cast<CostScratch *>(scratch_bytes[warp]);
    const unsigned long long T = *thr;
    unsigned long long below = 0;
    bool bad = false;
#pragma unroll 1
    for (uint32_t t = blockIdx.x * 8u + warp; t < count; t += nw) {
        azb_enum_tree(E, idx0 + t, par, lane);
        uint32_t mu = 0;
        const double l1 = azb_cost_warp<DEPTH>(E.n, par, cs, lane, &mu);
        __syncwarp();  // (the matching of the section method reads par after the warp's last barrier)
        const double key = __dadd_rn((double)mu, l1);
        below += key < bound ? 1u : 0u;
        bad |= !(l1 >= 1.4);  // ordered_edge.rs:79
        const unsigned long long bits = (unsigned long long)__double_as_longlong(key);
        if (lane == 0 && bits <= T) cand[atomicAdd(n_cand, 1u)] = AzbEnumCand{bits, idx0 + t};
    }
    if (lane == 0) {
        if (below) atomicAdd(n_below, below);
        if (bad) atomicMax(err, 5u);
    }
}
