// azb_grow.cuh — every tree on N <= 64 vertices whose c21 key (mu + lambda_1) is at most a bound (azb_trees_within),
// grown level by level: the trees on s + 1 vertices within the bound are children "tree + one leaf" of the trees on s
// vertices within it, because the key only grows from a subtree to its tree.  The set is defined in include/azb.h;
// DESIGN.md §4.11 has the design and the argument for the slack AZB_GROW_EPS.
//
// One chunk of a level (the host drives it from azb.cu):
//   expand             the s children of every tree of the chunk, leaf s under vertex v = 0..s-1
//   code               azb_tree_code_kernel (azb_best.cuh) on every child
//   sort + unique      by code (CUB), so each class of the chunk is evaluated once
//   decode             each class's canonical parent array, straight from its code
//   cost               azb_cost_kernel (azb_cost.cuh) on the canonical arrays: the key is a function of the class
//   keep               the classes with key <= the level's threshold, appended to the level's list
// The list is sorted and made unique by code whenever it could overflow and at the end of the level; it is the next
// level.  At the last level it is sorted by (key bits, code) and the first k are the result.
//
// Over several ranks (azb_comm_trees_within) each class has one owner, azb_grow_owner, and a rank holds only the classes
// it owns.  Between unique and decode a round routes the chunk's classes to their owners: count and route below write
// them as per-owner runs of 16-byte codes, the host exchanges the runs, and each rank sorts and makes unique what it
// received before it decodes, costs and keeps it.
#pragma once
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>
#include <cuda/std/tuple>

#include "azb_common.cuh"

#define AZB_GROW_CHUNK (1u << 22)  // children per chunk
#define AZB_GROW_EPS 1e-9          // slack of the levels below N (absolute, on the key)
#define AZB_GROW_MAX_WORLD 256u    // ranks azb_comm_trees_within takes: one round's codes stay below 2^31

struct AzbGrowEnt {            // one class: its code and, once evaluated, the bits of its key (> 0: they order like values)
    unsigned long long hi, lo;  // the code, as azb_tree_codes writes it (hi, lo = string bits 0..63, 64..127)
    unsigned long long key;
};
// equal codes: the unique pass keeps the first entry of each class
__host__ __device__ __forceinline__ bool operator==(const AzbGrowEnt &a, const AzbGrowEnt &b) { return a.hi == b.hi && a.lo == b.lo; }
struct AzbGrowByCode {
    __host__ __device__ cuda::std::tuple<unsigned long long &, unsigned long long &> operator()(AzbGrowEnt &e) const {
        return {e.hi, e.lo};
    }
};
struct AzbGrowByKey {
    __host__ __device__ cuda::std::tuple<unsigned long long &, unsigned long long &, unsigned long long &>
    operator()(AzbGrowEnt &e) const { return {e.key, e.hi, e.lo}; }
};

struct AzbGrowScalars {
    uint32_t n_sel, n_keep, bad, err;
    unsigned long long below;
};

// child c = t * s + v of the m trees on s vertices: tree t with the new vertex s under v (so parents[v] < v still holds)
__global__ void __launch_bounds__(256) azb_grow_expand_kernel(const uint8_t *__restrict__ par, uint32_t m, uint32_t s,
                                                              uint8_t *__restrict__ out) {
    const uint32_t n = s + 1;
    const size_t total = (size_t)m * s * n;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t c = i / n;
        const uint32_t u = (uint32_t)(i - c * n);
        out[i] = u < s ? par[(c / s) * s + u] : (uint8_t)(c % s);
    }
}

// The canonical parent array of each code (include/azb.h): the 2n-bit word read from the left, a 1 opens the next vertex
// under the current one and a 0 returns to the current vertex's parent.  Vertex 0 is the root the code was taken at,
// children come in code order, so parents[v] < v.  One thread per tree.
__global__ void __launch_bounds__(256) azb_grow_decode_kernel(const AzbGrowEnt *__restrict__ ent, uint32_t m, uint32_t n,
                                                              uint8_t *__restrict__ out) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m) return;
    const unsigned long long hi = ent[t].hi, lo = ent[t].lo;
    uint8_t *p = out + (size_t)t * n;
    p[0] = 0;
    uint32_t cur = 0, next = 1;
#pragma unroll 1
    for (uint32_t i = 1; i + 1 < 2 * n; ++i) {  // bit 0 opens the root and bit 2n - 1 closes it
        const bool one = i < 64u ? (hi >> (63u - i)) & 1ull : (lo >> (127u - i)) & 1ull;
        if (one) {
            p[next] = (uint8_t)cur;
            cur = next++;
        } else {
            cur = p[cur];
        }
    }
}

// the classes whose key (double)mu + lambda_1 is <= thr, appended at out[*n_keep] with their key bits
__global__ void __launch_bounds__(256) azb_grow_keep_kernel(const AzbGrowEnt *__restrict__ ent, const double *__restrict__ l1,
                                                            const uint32_t *__restrict__ mu, uint32_t m, double thr,
                                                            AzbGrowEnt *__restrict__ out, uint32_t *__restrict__ n_keep) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m) return;
    const double key = __dadd_rn((double)mu[t], l1[t]);
    if (key <= thr) out[atomicAdd(n_keep, 1u)] = AzbGrowEnt{ent[t].hi, ent[t].lo, (unsigned long long)__double_as_longlong(key)};
}

// *below += the entries with key < bound
__global__ void __launch_bounds__(256) azb_grow_below_kernel(const AzbGrowEnt *__restrict__ ent, uint32_t m, double bound,
                                                             unsigned long long *__restrict__ below) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = __syncthreads_count(t < m && __longlong_as_double((long long)ent[t].key) < bound);
    if (threadIdx.x == 0 && c) atomicAdd(below, (unsigned long long)c);
}

// the rank that holds a class when the growth is split over `world` ranks (include/azb.h)
__host__ __device__ __forceinline__ uint32_t azb_grow_owner(unsigned long long hi, unsigned long long lo, uint32_t world) {
    return (uint32_t)(azb_mix64(hi ^ azb_mix64(lo)) % world);
}

// counts[d] += the entries of ent[0, m) that rank d owns.  Dynamic shared memory: 4 * world bytes.
__global__ void __launch_bounds__(256) azb_grow_count_kernel(const AzbGrowEnt *__restrict__ ent, uint32_t m, uint32_t world,
                                                             unsigned long long *__restrict__ counts) {
    extern __shared__ uint32_t s_cnt[];
    for (uint32_t d = threadIdx.x; d < world; d += blockDim.x) s_cnt[d] = 0;
    __syncthreads();
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x)
        atomicAdd(&s_cnt[azb_grow_owner(ent[i].hi, ent[i].lo, world)], 1u);
    __syncthreads();
    for (uint32_t d = threadIdx.x; d < world; d += blockDim.x)
        if (s_cnt[d]) atomicAdd(&counts[d], (unsigned long long)s_cnt[d]);
}

// The codes of ent[0, m) as contiguous runs by owner: rank d's run starts at counts[0] + .. + counts[d - 1] (what
// azb_grow_count_kernel gave), and cursor[d] (zeroed before the launch) is the part of it taken so far.  Each block takes
// its slots of a run with one atomic per owner per tile of 256 entries; the order within a run is arbitrary, the
// receiver sorts.  Dynamic shared memory: 20 * world bytes.
__global__ void __launch_bounds__(256) azb_grow_route_kernel(const AzbGrowEnt *__restrict__ ent, uint32_t m, uint32_t world,
                                                             const unsigned long long *__restrict__ counts,
                                                             unsigned long long *__restrict__ cursor, ulonglong2 *__restrict__ out) {
    extern __shared__ unsigned long long s_run[];  // [world] run starts | [world] this tile's bases | [world] u32 counts
    unsigned long long *s_base = s_run + world;
    uint32_t *s_cnt = reinterpret_cast<uint32_t *>(s_base + world);
    if (threadIdx.x == 0) {
        unsigned long long run = 0;
        for (uint32_t d = 0; d < world; ++d) {
            s_run[d] = run;
            run += counts[d];
        }
    }
    for (uint32_t tile = blockIdx.x * blockDim.x; tile < m; tile += gridDim.x * blockDim.x) {
        for (uint32_t d = threadIdx.x; d < world; d += blockDim.x) s_cnt[d] = 0;
        __syncthreads();
        const uint32_t i = tile + threadIdx.x;
        unsigned long long hi = 0, lo = 0;
        uint32_t d = 0, slot = 0;
        if (i < m) {
            hi = ent[i].hi;
            lo = ent[i].lo;
            d = azb_grow_owner(hi, lo, world);
            slot = atomicAdd(&s_cnt[d], 1u);
        }
        __syncthreads();
        for (uint32_t r = threadIdx.x; r < world; r += blockDim.x)
            s_base[r] = s_run[r] + (s_cnt[r] ? atomicAdd(&cursor[r], (unsigned long long)s_cnt[r]) : 0ull);
        __syncthreads();
        if (i < m) out[s_base[d] + slot] = make_ulonglong2(hi, lo);
        __syncthreads();
    }
}
