// azb_graph.cuh -- SURVEY 8(f) row 3: the c21 cost and the action kinds of CONNECTED GRAPHS held as neighbourhood
// bit sets (`ConnectedBitsetGraph<N, B32>`, graph-state/src/simple_graph/connected_bitset_graph/mod.rs), batched.
// One warp per graph, lane v = vertex v (N <= 32), everything in shared memory and registers:
//   * action kinds (`action_kinds` :134-154 over `is_cut_edge` :45-71) in the index space of
//     `AddOrDeleteEdge::action_index` (bitset_graph/space/action.rs:10-19): the bit-set BFS test on the N - 1 edges
//     of a spanning tree (the only possible cut edges), then one lane per vertex pair;
//   * matching number (`maximum_matching` :226-317 is a branch and bound; only its SIZE is read, so any exact
//     algorithm gives the same number): greedy start + Edmonds' blossom augmentation, serial on lane 0;
//   * lambda_1 (`adjacency_matrix` :200-216 with its 1e-4 diagonal, `conjecture_2_1_cost` :319-337 takes the
//     largest eigenvalue): warp-parallel Householder tridiagonalisation in f64 (lane = row), then the largest
//     eigenvalue by Sturm counts on a 32-point section per round (lane = section point).
// `azb_graph_cost64_kernel` (below) is the same row for ConnectedBitsetGraph<N, B64>, N <= 64: lane l owns vertices and
// rows l and l + 32.
// The snapshot has no NablaStateActionSpace over these graphs (SURVEY 0.1), so this is the stand-alone cost row only.
#pragma once
#include <cstdint>

#define AZG_WARPS 4

struct AzgWarpScratch {  // one per warp, carved out of dynamic shared memory: the matrix is a packed lower triangle
    double *a;
    double *u, *w, *d, *e;
    uint32_t *nbr, *kinds;
    int8_t *match, *par, *base, *queue;
};
__host__ __device__ inline uint32_t azg_tri(uint32_t n) { return (n * (n + 1) / 2 + 1u) & ~1u; }  // doubles, 16 B multiple
__host__ __device__ inline uint32_t azg_ld(uint32_t n) { return n | 1u; }  // square layout: odd row stride
__host__ __device__ inline bool azg_packed(uint32_t n) { return n > 22u; }  // the triangle costs index arithmetic and a
// divergent second loop in A u; it pays once the square would hold the kernel below ~40 resident warps per SM
__host__ __device__ inline uint32_t azg_mat_doubles(uint32_t n) { return azg_packed(n) ? azg_tri(n) : n * azg_ld(n); }
__host__ __device__ inline uint32_t azg_warp_bytes(uint32_t n) { return 8u * azg_mat_doubles(n) + 4u * 32u * 8u + 2u * 32u * 4u + 4u * 32u; }

__device__ __forceinline__ double azg_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double azg_warp_max(double v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// the bit sets are B32 (uint32_t) or B64 (uint64_t) neighbourhoods
__device__ __forceinline__ int azg_ffs(uint32_t x) { return __ffs(x); }
__device__ __forceinline__ int azg_ffs(uint64_t x) { return __ffsll((long long)x); }

// connected_bitset_graph/mod.rs:45-71
template <typename W>
__device__ __forceinline__ bool azg_is_cut_edge(const W *nbr, uint32_t v, uint32_t u) {
    W fresh = nbr[v] ^ (W(1) << u), explored = W(1) << v;
    while (fresh) {
        if (fresh >> u & 1u) return false;
        explored |= fresh;
        W next = 0u;
        for (W r = fresh; r; r &= r - 1) next |= nbr[azg_ffs(r) - 1];
        fresh = next & ~explored;
    }
    return true;
}

// Edmonds' blossom algorithm (array form), serial, on the vertices of `alive` with neighbourhoods nbr[] (already
// restricted to `alive`); match/par/base/queue live in the warp's shared scratch
template <typename W>
__device__ __forceinline__ uint32_t azg_blossom(const AzgWarpScratch &s, const W *nbr, W alive, uint32_t n) {
    int8_t *match = s.match, *par = s.par, *base = s.base, *queue = s.queue;
    uint32_t size = 0;
    for (uint32_t v = 0; v < n; ++v) match[v] = -1;
    for (W av = alive; av; av &= av - 1) {  // greedy start
        const uint32_t v = azg_ffs(av) - 1;
        if (match[v] >= 0) continue;
        for (W r = nbr[v]; r; r &= r - 1) {
            const int t = azg_ffs(r) - 1;
            if (match[t] < 0) {
                match[v] = (int8_t)t;
                match[t] = (int8_t)v;
                ++size;
                break;
            }
        }
    }
    for (W ar = alive; ar; ar &= ar - 1) {
        const uint32_t root = azg_ffs(ar) - 1;
        if (match[root] >= 0) continue;
        for (uint32_t i = 0; i < n; ++i) {
            par[i] = -1;
            base[i] = (int8_t)i;
        }
        W used = W(1) << root;
        uint32_t qh = 0, qt = 0;
        queue[qt++] = (int8_t)root;
        int found = -1;
        while (qh < qt && found < 0) {
            const int v = queue[qh++];
            for (W r = nbr[v]; r && found < 0; r &= r - 1) {
                int to = azg_ffs(r) - 1;
                if (base[v] == base[to] || match[v] == to) continue;
                if (to == (int)root || (match[to] >= 0 && par[match[to]] >= 0)) {
                    // an odd cycle: contract it onto the lowest common ancestor of v and to
                    W seen = 0u;
                    int a = v, b = to, cur;
                    for (;;) {
                        a = base[a];
                        seen |= W(1) << a;
                        if (match[a] < 0) break;
                        a = par[match[a]];
                    }
                    for (;;) {
                        b = base[b];
                        if (seen >> b & 1u) break;
                        b = par[match[b]];
                    }
                    cur = b;
                    W blossom = 0u;
                    for (int side = 0; side < 2; ++side) {
                        int x = side ? to : v, child = side ? v : to;
                        while (base[x] != cur) {
                            blossom |= W(1) << base[x];
                            blossom |= W(1) << base[match[x]];
                            par[x] = (int8_t)child;
                            child = match[x];
                            x = par[match[x]];
                        }
                    }
                    for (uint32_t i = 0; i < n; ++i)
                        if (blossom >> base[i] & 1u) {
                            base[i] = (int8_t)cur;
                            if (!(used >> i & 1u)) {
                                used |= W(1) << i;
                                queue[qt++] = (int8_t)i;
                            }
                        }
                } else if (par[to] < 0) {
                    par[to] = (int8_t)v;
                    if (match[to] < 0) {
                        found = to;
                    } else {
                        to = match[to];
                        used |= W(1) << to;
                        queue[qt++] = (int8_t)to;
                    }
                }
            }
        }
        if (found >= 0) {
            ++size;
            for (int v = found; v >= 0;) {
                const int pv = par[v], ppv = match[pv];
                match[v] = (int8_t)pv;
                match[pv] = (int8_t)v;
                v = ppv;
            }
        }
    }
    return size;
}

// out of line: the B32 kernel's call site (the B64 kernel inlines the body; a call there costs spills around it)
template <typename W>
__device__ uint32_t azg_matching_number(const AzgWarpScratch &s, const W *nbr, W alive, uint32_t n) { return azg_blossom(s, nbr, alive, n); }

// x > lambda_max of the symmetric tridiagonal (d, e)  <=>  every leading principal minor of x I - T is positive:
// p_0 = 1, p_1 = x - d_0, p_i = (x - d_{i-1}) p_{i-1} - e_{i-2}^2 p_{i-2}.  No division; |p_i| <= (2 ||T||)^32 < 1e60.
__device__ __forceinline__ bool azg_above_all(const double *d, const double *e2, uint32_t n, double x) {
    double pm = 1.0, p = __dsub_rn(x, d[0]);
    bool all = p > 0.0;
    // no early exit: the warp runs as long as its highest section point anyway, and that one never leaves early
    for (uint32_t i = 1; i < n; ++i) {
        const double pn = __fma_rn(__dsub_rn(x, d[i]), p, -__dmul_rn(e2[i - 1], pm));
        pm = p;
        p = pn;
        all = all && p > 0.0;
    }
    return all;
}

template <bool PACKED>
__global__ void __launch_bounds__(AZG_WARPS * 32)
azb_graph_cost_kernel(const uint32_t *__restrict__ nbr_g, uint32_t m, uint32_t n, uint32_t kw, double *__restrict__ l1_out,
                      uint32_t *__restrict__ mu_out, uint32_t *__restrict__ kinds_out, uint32_t *err) {
    extern __shared__ __align__(16) uint8_t azg_smem[];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t g = blockIdx.x * AZG_WARPS + warp;
    if (g >= m) return;
    AzgWarpScratch s;
    {
        uint8_t *base = azg_smem + (size_t)warp * azg_warp_bytes(n);
        s.a = reinterpret_cast<double *>(base);
        s.u = s.a + azg_mat_doubles(n);
        s.w = s.u + 32;
        s.d = s.w + 32;
        s.e = s.d + 32;
        s.nbr = reinterpret_cast<uint32_t *>(s.e + 32);
        s.kinds = s.nbr + 32;
        s.match = reinterpret_cast<int8_t *>(s.kinds + 32);
        s.par = s.match + 32;
        s.base = s.par + 32;
        s.queue = s.base + 32;
    }
    const uint32_t mine = lane < n ? nbr_g[(size_t)g * n + lane] : 0u;
    s.nbr[lane] = mine;
    s.kinds[lane] = 0u;
    __syncwarp();
    // ---- what BitsetGraph::try_from / to_connected accept: no loops, neighbours < N, symmetric (column v of the
    // relation, gathered by ballots, must equal row v); connectedness falls out of the spanning tree below
    const uint32_t full = n == 32 ? 0xffffffffu : (1u << n) - 1u;
    bool bad = (mine & ~full) || (mine >> lane & 1u);
    for (uint32_t v = 0; v < n; ++v) {
        const uint32_t column = __ballot_sync(0xffffffffu, mine >> v & 1u);
        if (lane == v) bad = bad || column != mine;
    }

    // ---- cut edges.  Only the N - 1 edges of a spanning tree can be cut edges (any other edge closes a cycle with
    // the tree), so: a breadth-first spanning tree by ballots (lane v learns its parent), then ONE round of the
    // reference's test (`is_cut_edge`), lane v on the edge to its parent, instead of one test per edge of the graph.
    uint32_t *brg = reinterpret_cast<uint32_t *>(s.u);  // brg[v]: bit u <=> vu is a cut edge (the doubles are free here)
    brg[lane] = 0u;
    int parent = -1;
    uint32_t seen = 1u;
    for (uint32_t frontier = 1u; frontier;) {
        const uint32_t cand = mine & frontier;
        const bool join = lane < n && !(seen >> lane & 1u) && cand;
        if (join) parent = __ffs(cand) - 1;
        frontier = __ballot_sync(0xffffffffu, join);
        seen |= frontier;
    }
    if (__any_sync(0xffffffffu, bad) || seen != full) {  // not a connected simple graph: report the first such input
        if (lane == 0) {
            atomicOr(err, 1u << 1);
            atomicMin(err + 1, g);
            l1_out[g] = 0.0;
            mu_out[g] = 0u;
        }
        return;
    }
    __syncwarp();
    if (parent >= 0 && azg_is_cut_edge(s.nbr, lane, (uint32_t)parent)) {
        atomicOr(&brg[lane], 1u << parent);
        atomicOr(&brg[parent], 1u << lane);
    }
    __syncwarp();

    // ---- action kinds: pair p = colex(v, u) = v (v - 1) / 2 + u, 32 pairs per round
    const uint32_t e2 = n * (n - 1) / 2;
    for (uint32_t p0 = 0; p0 < e2; p0 += 32) {
        const uint32_t p = p0 + lane;
        bool add = false, del = false;
        if (p < e2) {
            uint32_t v = (uint32_t)((1.0f + sqrtf(1.0f + 8.0f * (float)p)) * 0.5f);
            while (v * (v - 1) / 2 > p) --v;
            while (v * (v + 1) / 2 <= p) ++v;
            const uint32_t u = p - v * (v - 1) / 2;
            if (s.nbr[v] >> u & 1u) del = !(brg[v] >> u & 1u);
            else add = true;
        }
        const uint32_t wa = __ballot_sync(0xffffffffu, add), wd = __ballot_sync(0xffffffffu, del);
        if (lane == 0) {
            s.kinds[p0 >> 5] |= wa;
            const uint32_t bit = e2 + p0, sh = bit & 31u;
            s.kinds[bit >> 5] |= wd << sh;
            if (sh && (wd >> (32u - sh))) s.kinds[(bit >> 5) + 1] |= wd >> (32u - sh);
        }
        __syncwarp();
    }
    if (kinds_out && lane < kw) kinds_out[(size_t)g * kw + lane] = s.kinds[lane];

    // ---- matching number: pendant edges first (some maximum matching contains any given pendant edge, so matching a
    // leaf with its neighbour and deleting both is exact), one ballot per leaf; what is left has minimum degree 2 and
    // goes through the blossom search on lane 0.  A tree never gets there.
    uint32_t mu = 0, alive = n == 32 ? 0xffffffffu : (1u << n) - 1u;
    for (;;) {
        const bool me = alive >> lane & 1u;
        const uint32_t mynb = mine & alive;
        const uint32_t leaves = __ballot_sync(0xffffffffu, me && __popc(mynb) == 1);
        alive &= ~__ballot_sync(0xffffffffu, me && mynb == 0u);
        if (!leaves) break;
        const int v = __ffs(leaves) - 1;
        const int t = __ffs(__shfl_sync(0xffffffffu, mynb, v)) - 1;
        alive &= ~((1u << v) | (1u << t));
        ++mu;
    }
    if (alive) {
        __syncwarp();
        s.kinds[lane] = (alive >> lane & 1u) ? (mine & alive) : 0u;  // the kinds are out: their words hold the core now
        __syncwarp();
        uint32_t core = 0;
        if (lane == 0) core = azg_matching_number(s, s.kinds, alive, n);
        mu += __shfl_sync(0xffffffffu, core, 0);
    }
    __syncwarp();

    // ---- lambda_1 of A + 1e-4 I.  The matrix is symmetric: lane i keeps the lower-triangle row i (entries j <= i) at
    // a + i (i + 1) / 2; the upper part of a row is read down its column (consecutive words across lanes).
    // (n <= 22: plain square rows of n | 1 doubles, every row whole -- fewer instructions, and it fits anyway)
    double *__restrict__ arow = s.a + (PACKED ? lane * (lane + 1) / 2 : lane * azg_ld(n));
    const uint32_t jmax = PACKED ? lane : n - 1;  // last column this lane stores
    if (lane < n)
        for (uint32_t j = 0; j <= jmax; ++j) arow[j] = lane == j ? 0.0001 : ((mine >> j & 1u) ? 1.0 : 0.0);
    __syncwarp();
    for (uint32_t k = 0; k + 2 < n; ++k) {
        const bool act = lane > k && lane < n;
        const double x = act ? arow[k] : 0.0;
        const double x0 = __shfl_sync(0xffffffffu, x, k + 1);
        const double rest2 = azg_warp_sum(lane == k + 1 ? 0.0 : __dmul_rn(x, x));
        const double norm2 = __fma_rn(x0, x0, rest2);
        if (rest2 == 0.0) {  // the column is already tridiagonal
            if (lane == 0) s.e[k] = x0;
            continue;
        }
        const double alpha = x0 > 0.0 ? -__dsqrt_rn(norm2) : __dsqrt_rn(norm2);
        double u = lane == k + 1 ? __dsub_rn(x, alpha) : x;
        const double u0 = __dsub_rn(x0, alpha);
        const double un2 = __fma_rn(u0, u0, rest2);
        u = __dmul_rn(u, __ddiv_rn(1.0, __dsqrt_rn(un2)));
        s.u[lane] = u;
        __syncwarp();
        const double *__restrict__ uu = s.u;
        double q = 0.0, q1 = 0.0;
        if (act) {
            uint32_t j = k + 1;
            for (; j + 1 <= jmax; j += 2) {  // own row (up to the diagonal when packed), two partial sums
                q = __fma_rn(arow[j], uu[j], q);
                q1 = __fma_rn(arow[j + 1], uu[j + 1], q1);
            }
            if (j <= jmax) q = __fma_rn(arow[j], uu[j], q);
            if (PACKED) {
                const double *col = s.a + lane;  // A[i][j] = A[j][i] for j > i: row j starts at j (j + 1) / 2
                j = lane + 1;
                uint32_t off = j * (j + 1) / 2;
                for (; j + 1 < n; j += 2) {
                    q = __fma_rn(col[off], uu[j], q);
                    off += j + 1;
                    q1 = __fma_rn(col[off], uu[j + 1], q1);
                    off += j + 2;
                }
                if (j < n) q = __fma_rn(col[off], uu[j], q);
            }
            q = __dadd_rn(q, q1);
        }
        const double uq = azg_warp_sum(__dmul_rn(u, q));
        const double w = __fma_rn(-uq, u, q);
        s.w[lane] = w;
        __syncwarp();  // also: every column read of this step is done before the rows change
        const double *__restrict__ ww = s.w;
        if (act) {
            const double u2 = __dmul_rn(-2.0, u), w2 = __dmul_rn(-2.0, w);  // A' = A - 2 u w^T - 2 w u^T
#pragma unroll 4
            for (uint32_t j = k + 1; j <= jmax; ++j) arow[j] = __fma_rn(u2, ww[j], __fma_rn(w2, uu[j], arow[j]));
        }
        if (lane == 0) s.e[k] = alpha;
        __syncwarp();
    }
    if (lane < n) s.d[lane] = arow[lane];
    if (lane == n - 1 && n >= 2) s.e[n - 2] = arow[n - 2];
    __syncwarp();
    if (lane + 1 < n) s.u[lane] = __dmul_rn(s.e[lane], s.e[lane]);  // squared off-diagonal, once
    __syncwarp();
    // Gershgorin bracket of the spectrum, then 33-fold sections of [lo, hi] with  not above(lo), above(hi)
    double rad = 0.0, dd = -1e300;
    if (lane < n) {
        dd = s.d[lane];
        rad = (lane > 0 ? fabs(s.e[lane - 1]) : 0.0) + (lane + 1 < n ? fabs(s.e[lane]) : 0.0);
    }
    double hi = azg_warp_max(lane < n ? dd + rad : -1e300), lo = -azg_warp_max(lane < n ? rad - dd : -1e300);
    const double scale = fmax(fabs(hi), fabs(lo));
    hi = hi + fmax(scale, 1.0) * 1e-9;
    for (int round = 0; round < 16; ++round) {
        const double step = __ddiv_rn(__dsub_rn(hi, lo), 33.0);
        const double x = __dadd_rn(lo, __dmul_rn(step, (double)(lane + 1)));
        const uint32_t above = __ballot_sync(0xffffffffu, azg_above_all(s.d, s.u, n, x));
        const int first = above ? __ffs(above) - 1 : 32;
        const double nlo = first > 0 ? __shfl_sync(0xffffffffu, x, first - 1) : lo;
        const double nhi = first < 32 ? __shfl_sync(0xffffffffu, x, first & 31) : hi;
        lo = nlo;
        hi = nhi;
        if (!(__dsub_rn(hi, lo) > 4.0 * 2.220446049250313e-16 * fmax(fabs(hi), fabs(lo)))) break;
    }
    const double l1 = __dmul_rn(0.5, __dadd_rn(lo, hi));
    if (lane == 0) {
        l1_out[g] = l1;
        mu_out[g] = mu;
        if (!(l1 > 1.4)) atomicOr(err, 1u << 5);  // connected_bitset_graph/mod.rs:333 `assert!(lambda_1 > 1.4)`
    }
}

// ---- the same row for ConnectedBitsetGraph<N, B64> (N <= 64): still one warp per graph, lane l owns the vertices
// (and matrix rows) l and l + 32, so every warp-level step above runs on two values per lane.  The warps per CTA are a
// launch parameter (blockDim.x / 32): the host picks them from the shared-memory footprint, which grows with N.
#define AZG64_MAX_WARPS 4
// per warp: the matrix, u w d e [64] (u doubles as the cut-edge sets), nbr [64] u64, 128 kind words (the matching core
// reuses them as [64] u64), match par base queue [64] int8
__host__ __device__ inline uint32_t azg64_warp_bytes(uint32_t n) { return 8u * azg_mat_doubles(n) + 4u * 64u * 8u + 64u * 8u + 128u * 4u + 4u * 64u; }

template <bool PACKED>
__global__ void __launch_bounds__(AZG64_MAX_WARPS * 32)
azb_graph_cost64_kernel(const uint64_t *__restrict__ nbr_g, uint32_t m, uint32_t n, uint32_t kw, double *__restrict__ l1_out,
                        uint32_t *__restrict__ mu_out, uint32_t *__restrict__ kinds_out, uint32_t *err) {
    extern __shared__ __align__(16) uint8_t azg_smem[];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31, hi = lane + 32;
    const uint32_t g = blockIdx.x * (blockDim.x >> 5) + warp;
    if (g >= m) return;
    AzgWarpScratch s;
    uint64_t *nbr;
    {
        uint8_t *base = azg_smem + (size_t)warp * azg64_warp_bytes(n);
        s.a = reinterpret_cast<double *>(base);
        s.u = s.a + azg_mat_doubles(n);
        s.w = s.u + 64;
        s.d = s.w + 64;
        s.e = s.d + 64;
        nbr = reinterpret_cast<uint64_t *>(s.e + 64);
        s.nbr = reinterpret_cast<uint32_t *>(nbr);
        s.kinds = reinterpret_cast<uint32_t *>(nbr + 64);
        s.match = reinterpret_cast<int8_t *>(s.kinds + 128);
        s.par = s.match + 64;
        s.base = s.par + 64;
        s.queue = s.base + 64;
    }
    const uint64_t *row = nbr_g + (size_t)g * n;
    const uint64_t mine0 = lane < n ? row[lane] : 0ull, mine1 = hi < n ? row[hi] : 0ull;
    nbr[lane] = mine0;
    nbr[hi] = mine1;
    for (uint32_t w = lane; w < 128; w += 32) s.kinds[w] = 0u;
    __syncwarp();
    // ---- validation: no loops, neighbours < N, symmetric (columns v and v + 32 by two ballots each)
    const uint64_t full = n == 64 ? ~0ull : (1ull << n) - 1ull;
    bool bad = (mine0 & ~full) || (mine0 >> lane & 1u) || (mine1 & ~full) || (mine1 >> hi & 1u);
    for (uint32_t v = 0; v < 32 && v < n; ++v) {
        const uint64_t col0 = __ballot_sync(0xffffffffu, mine0 >> v & 1u) | (uint64_t)__ballot_sync(0xffffffffu, mine1 >> v & 1u) << 32;
        const uint64_t col1 = __ballot_sync(0xffffffffu, mine0 >> (v + 32) & 1u) | (uint64_t)__ballot_sync(0xffffffffu, mine1 >> (v + 32) & 1u) << 32;
        if (lane == v) bad = bad || col0 != mine0 || col1 != mine1;
    }

    // ---- cut edges: a breadth-first spanning tree by ballots on a u64 frontier, then `is_cut_edge` on its N - 1 edges
    uint64_t *brg = reinterpret_cast<uint64_t *>(s.u);
    brg[lane] = 0ull;
    brg[hi] = 0ull;
    int parent0 = -1, parent1 = -1;
    uint64_t seen = 1ull;
    for (uint64_t frontier = 1ull; frontier;) {
        const uint64_t cand0 = mine0 & frontier, cand1 = mine1 & frontier;
        const bool join0 = lane < n && !(seen >> lane & 1u) && cand0, join1 = hi < n && !(seen >> hi & 1u) && cand1;
        if (join0) parent0 = azg_ffs(cand0) - 1;
        if (join1) parent1 = azg_ffs(cand1) - 1;
        frontier = __ballot_sync(0xffffffffu, join0) | (uint64_t)__ballot_sync(0xffffffffu, join1) << 32;
        seen |= frontier;
    }
    if (__any_sync(0xffffffffu, bad) || seen != full) {
        if (lane == 0) {
            atomicOr(err, 1u << 1);
            atomicMin(err + 1, g);
            l1_out[g] = 0.0;
            mu_out[g] = 0u;
        }
        return;
    }
    __syncwarp();
    typedef unsigned long long ull;
    if (parent0 >= 0 && azg_is_cut_edge(nbr, lane, (uint32_t)parent0)) {
        atomicOr(reinterpret_cast<ull *>(&brg[lane]), 1ull << parent0);
        atomicOr(reinterpret_cast<ull *>(&brg[parent0]), 1ull << lane);
    }
    if (parent1 >= 0 && azg_is_cut_edge(nbr, hi, (uint32_t)parent1)) {
        atomicOr(reinterpret_cast<ull *>(&brg[hi]), 1ull << parent1);
        atomicOr(reinterpret_cast<ull *>(&brg[parent1]), 1ull << hi);
    }
    __syncwarp();

    // ---- action kinds: pair p = colex(v, u), 32 pairs per round (63 rounds at N = 64)
    const uint32_t e2 = n * (n - 1) / 2;
    for (uint32_t p0 = 0; p0 < e2; p0 += 32) {
        const uint32_t p = p0 + lane;
        bool add = false, del = false;
        if (p < e2) {
            uint32_t v = (uint32_t)((1.0f + sqrtf(1.0f + 8.0f * (float)p)) * 0.5f);
            while (v * (v - 1) / 2 > p) --v;
            while (v * (v + 1) / 2 <= p) ++v;
            const uint32_t u = p - v * (v - 1) / 2;
            if (nbr[v] >> u & 1u) del = !(brg[v] >> u & 1u);
            else add = true;
        }
        const uint32_t wa = __ballot_sync(0xffffffffu, add), wd = __ballot_sync(0xffffffffu, del);
        if (lane == 0) {
            s.kinds[p0 >> 5] |= wa;
            const uint32_t bit = e2 + p0, sh = bit & 31u;
            s.kinds[bit >> 5] |= wd << sh;
            if (sh && (wd >> (32u - sh))) s.kinds[(bit >> 5) + 1] |= wd >> (32u - sh);
        }
        __syncwarp();
    }
    if (kinds_out)
        for (uint32_t w = lane; w < kw; w += 32) kinds_out[(size_t)g * kw + w] = s.kinds[w];

    // ---- matching number: pendant edges by ballots, then the blossom search on lane 0 over what is left
    uint32_t mu = 0;
    uint64_t alive = full;
    for (;;) {
        const bool me0 = alive >> lane & 1u, me1 = alive >> hi & 1u;
        const uint64_t nb0 = mine0 & alive, nb1 = mine1 & alive;
        const uint64_t leaves = __ballot_sync(0xffffffffu, me0 && __popcll(nb0) == 1) |
                                (uint64_t)__ballot_sync(0xffffffffu, me1 && __popcll(nb1) == 1) << 32;
        alive &= ~(__ballot_sync(0xffffffffu, me0 && nb0 == 0ull) | (uint64_t)__ballot_sync(0xffffffffu, me1 && nb1 == 0ull) << 32);
        if (!leaves) break;
        const int v = azg_ffs(leaves) - 1;
        const int t = azg_ffs(__shfl_sync(0xffffffffu, v < 32 ? nb0 : nb1, v & 31)) - 1;
        alive &= ~((1ull << v) | (1ull << t));
        ++mu;
    }
    if (alive) {
        __syncwarp();
        uint64_t *core = reinterpret_cast<uint64_t *>(s.kinds);  // the kinds are out: their words hold the core now
        core[lane] = (alive >> lane & 1u) ? (mine0 & alive) : 0ull;
        core[hi] = (alive >> hi & 1u) ? (mine1 & alive) : 0ull;
        __syncwarp();
        uint32_t c = 0;
        if (lane == 0) c = azg_blossom(s, (const uint64_t *)core, alive, n);
        mu += __shfl_sync(0xffffffffu, c, 0);
    }
    __syncwarp();

    // ---- lambda_1 of A + 1e-4 I: Householder on rows lane and lane + 32 (packed lower triangle or square rows, as
    // above), then the Sturm sections
    double *__restrict__ arow0 = s.a + (PACKED ? lane * (lane + 1) / 2 : lane * azg_ld(n));
    double *__restrict__ arow1 = s.a + (PACKED ? hi * (hi + 1) / 2 : hi * azg_ld(n));
    const uint32_t jmax0 = PACKED ? lane : n - 1, jmax1 = PACKED ? hi : n - 1;
    if (lane < n)
        for (uint32_t j = 0; j <= jmax0; ++j) arow0[j] = lane == j ? 0.0001 : ((mine0 >> j & 1u) ? 1.0 : 0.0);
    if (hi < n)
        for (uint32_t j = 0; j <= jmax1; ++j) arow1[j] = hi == j ? 0.0001 : ((mine1 >> j & 1u) ? 1.0 : 0.0);
    __syncwarp();
    // q = (A u)_i over the columns j > k, i.e. row i (up to its diagonal when packed) and then column i below it
    auto rowdot = [&](const double *__restrict__ arow, uint32_t i, uint32_t jmax, uint32_t k, const double *__restrict__ uu) {
        double q = 0.0, q1 = 0.0;
        uint32_t j = k + 1;
        for (; j + 1 <= jmax; j += 2) {
            q = __fma_rn(arow[j], uu[j], q);
            q1 = __fma_rn(arow[j + 1], uu[j + 1], q1);
        }
        if (j <= jmax) q = __fma_rn(arow[j], uu[j], q);
        if (PACKED) {
            const double *col = s.a + i;
            j = i + 1;
            uint32_t off = j * (j + 1) / 2;
            for (; j + 1 < n; j += 2) {
                q = __fma_rn(col[off], uu[j], q);
                off += j + 1;
                q1 = __fma_rn(col[off], uu[j + 1], q1);
                off += j + 2;
            }
            if (j < n) q = __fma_rn(col[off], uu[j], q);
        }
        return __dadd_rn(q, q1);
    };
    for (uint32_t k = 0; k + 2 < n; ++k) {
        const bool act0 = lane > k && lane < n, act1 = hi > k && hi < n;
        const double x0 = act0 ? arow0[k] : 0.0, x1 = act1 ? arow1[k] : 0.0;
        const double xp = __shfl_sync(0xffffffffu, k + 1 < 32 ? x0 : x1, (k + 1) & 31);
        const double rest2 = azg_warp_sum(__dadd_rn(lane == k + 1 ? 0.0 : __dmul_rn(x0, x0), hi == k + 1 ? 0.0 : __dmul_rn(x1, x1)));
        const double norm2 = __fma_rn(xp, xp, rest2);
        if (rest2 == 0.0) {
            if (lane == 0) s.e[k] = xp;
            continue;
        }
        const double alpha = xp > 0.0 ? -__dsqrt_rn(norm2) : __dsqrt_rn(norm2);
        const double up = __dsub_rn(xp, alpha);
        const double un2 = __fma_rn(up, up, rest2), inv = __ddiv_rn(1.0, __dsqrt_rn(un2));
        const double u0 = __dmul_rn(lane == k + 1 ? __dsub_rn(x0, alpha) : x0, inv);
        const double u1 = __dmul_rn(hi == k + 1 ? __dsub_rn(x1, alpha) : x1, inv);
        s.u[lane] = u0;
        s.u[hi] = u1;
        __syncwarp();
        const double q0 = act0 ? rowdot(arow0, lane, jmax0, k, s.u) : 0.0;
        const double q1 = act1 ? rowdot(arow1, hi, jmax1, k, s.u) : 0.0;
        const double uq = azg_warp_sum(__fma_rn(u1, q1, __dmul_rn(u0, q0)));
        const double w0 = __fma_rn(-uq, u0, q0), w1 = __fma_rn(-uq, u1, q1);
        s.w[lane] = w0;
        s.w[hi] = w1;
        __syncwarp();  // also: every column read of this step is done before the rows change
        const double *__restrict__ uu = s.u, *__restrict__ ww = s.w;
        if (act0) {
            const double u2 = __dmul_rn(-2.0, u0), w2 = __dmul_rn(-2.0, w0);  // A' = A - 2 u w^T - 2 w u^T
#pragma unroll 4
            for (uint32_t j = k + 1; j <= jmax0; ++j) arow0[j] = __fma_rn(u2, ww[j], __fma_rn(w2, uu[j], arow0[j]));
        }
        if (act1) {
            const double u2 = __dmul_rn(-2.0, u1), w2 = __dmul_rn(-2.0, w1);
#pragma unroll 4
            for (uint32_t j = k + 1; j <= jmax1; ++j) arow1[j] = __fma_rn(u2, ww[j], __fma_rn(w2, uu[j], arow1[j]));
        }
        if (lane == 0) s.e[k] = alpha;
        __syncwarp();
    }
    if (lane < n) s.d[lane] = arow0[lane];
    if (hi < n) s.d[hi] = arow1[hi];
    if (lane == n - 1) s.e[n - 2] = arow0[n - 2];
    if (hi == n - 1) s.e[n - 2] = arow1[n - 2];
    __syncwarp();
    if (lane + 1 < n) s.u[lane] = __dmul_rn(s.e[lane], s.e[lane]);
    if (hi + 1 < n) s.u[hi] = __dmul_rn(s.e[hi], s.e[hi]);
    __syncwarp();
    // Gershgorin bracket, then 33-fold sections.  At N = 64 the Sturm products stay inside f64: p_i is the
    // characteristic polynomial of the leading i x i block, whose eigenvalues lie in [-64, 64], at a point x of the
    // bracket, |x| <= ||T||_inf <= 8 ||T||_2 <= 512, so |p_i| <= 576^64 < 2^590.  16 rounds shrink the bracket (width
    // < 2^11) by 33^16 > 2^80, more than the 2^61 down to 4 ulps of any lambda_1 >= 1.4 (K64: 63 needs 2^55).
    double top = -1e300, bot = -1e300;
    for (uint32_t i = lane; i < 64; i += 32)
        if (i < n) {
            const double dd = s.d[i], rad = (i > 0 ? fabs(s.e[i - 1]) : 0.0) + (i + 1 < n ? fabs(s.e[i]) : 0.0);
            top = fmax(top, dd + rad);
            bot = fmax(bot, rad - dd);
        }
    double hi_x = azg_warp_max(top), lo = -azg_warp_max(bot);
    const double scale = fmax(fabs(hi_x), fabs(lo));
    hi_x = hi_x + fmax(scale, 1.0) * 1e-9;
    for (int round = 0; round < 16; ++round) {
        const double step = __ddiv_rn(__dsub_rn(hi_x, lo), 33.0);
        const double x = __dadd_rn(lo, __dmul_rn(step, (double)(lane + 1)));
        const uint32_t above = __ballot_sync(0xffffffffu, azg_above_all(s.d, s.u, n, x));
        const int first = above ? __ffs(above) - 1 : 32;
        const double nlo = first > 0 ? __shfl_sync(0xffffffffu, x, first - 1) : lo;
        const double nhi = first < 32 ? __shfl_sync(0xffffffffu, x, first & 31) : hi_x;
        lo = nlo;
        hi_x = nhi;
        if (!(__dsub_rn(hi_x, lo) > 4.0 * 2.220446049250313e-16 * fmax(fabs(hi_x), fabs(lo)))) break;
    }
    const double l1 = __dmul_rn(0.5, __dadd_rn(lo, hi_x));
    if (lane == 0) {
        l1_out[g] = l1;
        mu_out[g] = mu;
        if (!(l1 > 1.4)) atomicOr(err, 1u << 5);
    }
}
