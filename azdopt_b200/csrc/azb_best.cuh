// azb_best.cuh — the canonical tree code (azb_tree_codes) and the k best isomorphism classes among the nodes of a
// handle's trees (azb_best_trees).  The code is defined in include/azb.h; DESIGN.md §4.8 has the design.
//
// Selection, exact and deterministic (one round; the host widens M until k classes come out or every node is in):
//   hist x4 + pick x4   radix select of the M-th smallest ord(c) over every node record (first word of each 64-B record)
//   compact             every node with ord(c) <= T, in any order (atomics)
//   replay + code       the node's key replayed on its root's parents, then the code kernel
//   sort by code        (code, c, tree, node): CUB radix sort, total order, so the compaction order cannot reach the result
//   heads               the first of each code = the class value and its representative
//   sort by value       (c, code, ...): the classes in result order
#pragma once
#include <cub/device/device_radix_sort.cuh>
#include <cuda/std/tuple>

#include "azb_common.cuh"

#define AZB_CODE_WARPS 8
#define AZB_BEST_MAX_K 65536u

struct AzbBestState {  // device scratch of one selection round
    uint32_t prefix;   // high digits of the threshold chosen so far
    uint32_t rank;     // rank still to find below the prefix (1-based)
    uint32_t below;    // nodes whose key is below the prefix's bucket
    uint32_t total;    // node records of all trees
    uint32_t all;      // 1: M >= total, every node is a candidate
    uint32_t thr;      // the threshold T
    uint32_t count;    // nodes with ord(c) <= T (exact)
    uint32_t n_cand;   // compaction cursor
    uint32_t n_class;  // classes found
    uint32_t bad;      // first tree whose parent array was rejected (0xffffffff: none)
    uint32_t pad[6];
    uint32_t hist[256];
};

// one candidate / class: sorted as a whole by CUB with the decomposers below
struct AzbCand {
    unsigned long long hi, lo;  // the code: string bits 0..63, 64..127
    uint32_t c;                 // ord(c)
    uint32_t pad;
    unsigned long long id;      // tree << 20 | node (local tree: within one handle its order is the global root's)
};
struct AzbByCode {
    __host__ __device__ cuda::std::tuple<unsigned long long &, unsigned long long &, uint32_t &, unsigned long long &>
    operator()(AzbCand &k) const { return {k.hi, k.lo, k.c, k.id}; }
};
struct AzbByValue {
    __host__ __device__ cuda::std::tuple<uint32_t &, unsigned long long &, unsigned long long &, unsigned long long &>
    operator()(AzbCand &k) const { return {k.c, k.hi, k.lo, k.id}; }
};

// the 128-bit string (hi, lo) moved s bits to the right (1 <= s < 128)
__device__ __forceinline__ void azb_shr128(unsigned long long hi, unsigned long long lo, uint32_t s, unsigned long long &oh,
                                           unsigned long long &ol) {
    if (s < 64u) {
        oh = hi >> s;
        ol = (lo >> s) | (hi << (64u - s));
    } else {
        oh = 0ull;
        ol = hi >> (s - 64u);
    }
}

// ---- canonical code: one warp per tree, lane l owns vertices l and l + 32 ----
// Centres by leaf stripping on neighbour masks; then, per centre r, a breadth-first pass gives every vertex its depth and
// its parent towards r, and enc() is built one level at a time from the deepest: a child ranks itself among its siblings
// (descending code, vertex index on ties — equal codes concatenate the same either way), so its bits go to offset
// 1 + 2 * (sizes of the siblings ahead of it) in its parent's code.  Disjoint bit ranges: atomicOr order is irrelevant.
// codes[t * stride + 0/1] = the code's two words; *bad = the lowest tree with parents[v] >= v (whose code is not written).
__global__ void __launch_bounds__(AZB_CODE_WARPS * 32) azb_tree_code_kernel(const uint8_t *__restrict__ parents, uint32_t m,
                                                                            uint32_t N, unsigned long long *__restrict__ codes,
                                                                            uint32_t stride, uint32_t *__restrict__ bad) {
    __shared__ unsigned long long s_nbr[AZB_CODE_WARPS][64], s_hi[AZB_CODE_WARPS][64], s_lo[AZB_CODE_WARPS][64];
    __shared__ uint32_t s_size[AZB_CODE_WARPS][64];
    __shared__ uint8_t s_par[AZB_CODE_WARPS][64], s_rp[AZB_CODE_WARPS][64];
    const uint32_t FULL = 0xffffffffu, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t t = blockIdx.x * AZB_CODE_WARPS + warp;
    if (t >= m) return;
    unsigned long long *nbr = s_nbr[warp], *chi = s_hi[warp], *clo = s_lo[warp];
    uint32_t *size = s_size[warp];
    uint8_t *par = s_par[warp], *rp = s_rp[warp];
    const uint8_t *src = parents + (size_t)t * N;
    for (uint32_t v = lane; v < N; v += 32) par[v] = src[v];
    __syncwarp();
    bool wrong = false;
    for (uint32_t v = lane; v < N; v += 32) wrong |= v >= 1u && par[v] >= v;
    if (__any_sync(FULL, wrong)) {
        if (lane == 0) atomicMin(bad, t);
        return;
    }
    const unsigned long long all = N >= 64u ? ~0ull : ((1ull << N) - 1ull);
    unsigned long long nb[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const uint32_t v = lane + 32u * j;
        unsigned long long x = 0ull;
        if (v < N) {
            if (v) x |= 1ull << par[v];
            for (uint32_t u = v + 1; u < N; ++u) x |= (unsigned long long)(par[u] == v) << u;
            nbr[v] = x;
        }
        nb[j] = x;
    }
    // centres: strip every leaf while more than two vertices are left
    unsigned long long alive = all;
    while (__popcll(alive) > 2) {
        const bool l0 = ((alive >> lane) & 1ull) && __popcll(nb[0] & alive) <= 1;
        const bool l1 = ((alive >> (lane + 32)) & 1ull) && __popcll(nb[1] & alive) <= 1;
        alive &= ~((unsigned long long)__ballot_sync(FULL, l0) | ((unsigned long long)__ballot_sync(FULL, l1) << 32));
    }
    __syncwarp();
    unsigned long long best_hi = 0ull, best_lo = 0ull;
    for (unsigned long long cs = alive; cs; cs &= cs - 1ull) {
        const uint32_t r = __ffsll((long long)cs) - 1;
        uint32_t dep0 = r == lane ? 0u : 0xffu, dep1 = r == lane + 32u ? 0u : 0xffu;
        unsigned long long frontier = 1ull << r, seen = frontier;
        uint32_t D = 0;
        // joins v (neighbours nbv, depth dv) to the next level if it touches the frontier
        auto reach = [&](uint32_t v, unsigned long long nbv, uint32_t &dv) {
            if (v < N && !((seen >> v) & 1ull) && (nbv & frontier)) {
                dv = D + 1;
                rp[v] = (uint8_t)(__ffsll((long long)(nbv & frontier)) - 1);
                return true;
            }
            return false;
        };
        for (;;) {
            const bool n0 = reach(lane, nb[0], dep0), n1 = reach(lane + 32u, nb[1], dep1);
            const unsigned long long next = (unsigned long long)__ballot_sync(FULL, n0) | ((unsigned long long)__ballot_sync(FULL, n1) << 32);
            if (!next) break;
            seen |= next;
            frontier = next;
            ++D;
        }
        for (uint32_t v = lane; v < N; v += 32) {
            chi[v] = 1ull << 63;
            clo[v] = 0ull;
            size[v] = 1u;
        }
        __syncwarp();
        // v's code goes into its parent's at 1 + 2 * (sizes of the siblings ranked ahead of it)
        auto place = [&](uint32_t v) {
            const uint32_t p = rp[v];
            const unsigned long long hi = chi[v], lo = clo[v];
            unsigned long long sib = nbr[p] & ~(1ull << v);
            if (p != r) sib &= ~(1ull << rp[p]);
            uint32_t ahead = 0;
            for (; sib; sib &= sib - 1ull) {
                const uint32_t w = __ffsll((long long)sib) - 1;
                const unsigned long long wh = chi[w], wl = clo[w];
                if (wh > hi || (wh == hi && (wl > lo || (wl == lo && w < v)))) ahead += size[w];
            }
            unsigned long long oh, ol;
            azb_shr128(hi, lo, 1u + 2u * ahead, oh, ol);
            atomicOr(&chi[p], oh);
            atomicOr(&clo[p], ol);
            atomicAdd(&size[p], size[v]);
        };
        for (uint32_t d = D; d >= 1u; --d) {
            if (dep0 == d) place(lane);
            if (lane + 32u < N && dep1 == d) place(lane + 32u);
            __syncwarp();
        }
        const unsigned long long hi = chi[r], lo = clo[r];
        if (hi > best_hi || (hi == best_hi && lo > best_lo)) {
            best_hi = hi;
            best_lo = lo;
        }
        __syncwarp();
    }
    if (lane == 0) {
        codes[(size_t)t * stride] = best_hi;
        codes[(size_t)t * stride + 1] = best_lo;
    }
}

// ---- selection ----
// one radix digit of ord(c) over every node record whose higher digits equal the prefix; trees grid-strided over blocks
__global__ void __launch_bounds__(256) azb_best_hist_kernel(const AzbLayout L, AzbBestState *st, const uint32_t shift) {
    __shared__ uint32_t h[256];
    if (st->all) return;
    h[threadIdx.x] = 0u;
    __syncthreads();
    const uint32_t prefix = st->prefix, hmask = shift >= 24u ? 0u : (0xffffffffu << (shift + 8u));
    uint32_t n = 0;
    for (uint32_t t = blockIdx.x; t < L.B; t += gridDim.x) {
        const uint32_t nn = L.walker[(size_t)t * L.WS + WK_NNODES];
        const uint32_t *rec = reinterpret_cast<const uint32_t *>(L.node + (size_t)t * L.cap_nodes * 4);
        for (uint32_t i = threadIdx.x; i < nn; i += blockDim.x) {
            const uint32_t o = azb_f2ord(__uint_as_float(rec[(size_t)i * 16]));
            if ((o & hmask) == prefix) atomicAdd(&h[(o >> shift) & 255u], 1u);
        }
        n += nn;
    }
    __syncthreads();
    if (h[threadIdx.x]) atomicAdd(&st->hist[threadIdx.x], h[threadIdx.x]);
    if (shift == 24u && threadIdx.x == 0) atomicAdd(&st->total, n);
}

// choose the digit that holds the rank-th smallest key; after the last digit T and the count of keys <= T are exact
__global__ void azb_best_pick_kernel(AzbBestState *st, const uint32_t shift, const uint32_t M) {
    if (st->all) return;
    if (shift == 24u) {
        if (M >= st->total) {
            st->all = 1u;
            st->thr = 0xffffffffu;
            st->count = st->total;
            return;
        }
        st->rank = M;
        st->below = 0u;
    }
    uint32_t run = 0, d = 0;
    for (; d < 255u && run + st->hist[d] < st->rank; ++d) run += st->hist[d];
    st->rank -= run;
    st->below += run;
    st->prefix |= d << shift;
    if (shift == 0u) {
        st->thr = st->prefix;
        st->count = st->below + st->hist[d];
    }
    for (uint32_t i = 0; i < 256u; ++i) st->hist[i] = 0u;
}

__global__ void __launch_bounds__(256) azb_best_compact_kernel(const AzbLayout L, AzbBestState *st, AzbCand *out) {
    const uint32_t thr = st->thr, cap = st->count;
    for (uint32_t t = blockIdx.x; t < L.B; t += gridDim.x) {
        const uint32_t nn = L.walker[(size_t)t * L.WS + WK_NNODES];
        const uint32_t *rec = reinterpret_cast<const uint32_t *>(L.node + (size_t)t * L.cap_nodes * 4);
        for (uint32_t i = threadIdx.x; i < nn; i += blockDim.x) {
            const uint32_t o = azb_f2ord(__uint_as_float(rec[(size_t)i * 16]));
            if (o > thr) continue;
            const uint32_t j = atomicAdd(&st->n_cand, 1u);
            if (j < cap) out[j] = AzbCand{0ull, 0ull, o, 0u, ((unsigned long long)t << 20) | i};
        }
    }
}

// the state of each candidate: its root with its key replayed in ascending action order (finalize_argmin_state's rule);
// parents [n][N], permitted [n][W] when non-null.  One thread per candidate.
__global__ void __launch_bounds__(256) azb_best_replay_kernel(const AzbLayout L, const AzbCand *__restrict__ cand, uint32_t n,
                                                              uint8_t *__restrict__ par, uint32_t *__restrict__ perm) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t tree = (uint32_t)(cand[i].id >> 20), node = (uint32_t)(cand[i].id & 0xfffffu);
    const uint32_t *root = L.walker + (size_t)tree * L.WS + WK_HDR + L.PW + 2 * L.W;  // root parents | root permitted
    uint8_t *p = par + (size_t)i * L.N;
    uint32_t *pm = perm ? perm + (size_t)i * L.W : nullptr;
    for (uint32_t v = 0; v < L.N; ++v) p[v] = reinterpret_cast<const uint8_t *>(root)[v];
    if (pm)
        for (uint32_t w = 0; w < L.W; ++w) pm[w] = root[L.PW + w];
    const uint32_t *key = L.key + ((size_t)tree * L.cap_nodes + node) * L.W;
    for (uint32_t w = 0; w < L.W; ++w) {
        for (uint32_t word = key[w]; word; word &= word - 1u) {
            const uint32_t a = w * 32u + (__ffs(word) - 1), child = L.lut[a], first = azb_child_first_action(child);
            p[child] = (uint8_t)(a - first);
            if (pm)
                for (uint32_t q = first; q < first + child; ++q) pm[q >> 5] &= ~(1u << (q & 31u));
        }
    }
}

// after the sort by code: the first candidate of each code is its class (value and representative)
__global__ void __launch_bounds__(256) azb_best_heads_kernel(const AzbCand *__restrict__ s, uint32_t n, AzbCand *__restrict__ cls,
                                                             AzbBestState *st) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (i == 0 || s[i].hi != s[i - 1].hi || s[i].lo != s[i - 1].lo) cls[atomicAdd(&st->n_class, 1u)] = s[i];
}
