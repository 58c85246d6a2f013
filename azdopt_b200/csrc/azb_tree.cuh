// azb_tree.cuh — the search step: one warp owns one root's search DAG.
//
// Replaces, per root, SearchTree::roll_out_episodes (az-discrete-opt/src/nabla/tree/mod.rs:113-232) with
// next_action / revisit_choice / max_curiosity (nabla/tree/next_action.rs:11-88), add_node / add_arc / add_actions
// (nabla/tree/graph_operations.rs:8-56), cascade_new_terminal / cascade_old_node
// (nabla/tree/empty_transitions.rs:50-127), the ROTModifyParentsOnce space (graph-state/src/rooted_tree/space.rs:
// 37-125), write_vec (space.rs:91-101) and the per-tree half of the argmin scan (nabla/optimizer/mod.rs:194-221).
//
// Design notes (DESIGN.md §3-4).  The walk is a chain of dependent memory round trips, so the layout is built to
// need ONE round trip per level:
//  * an expanded node owns a block [preds | header | kids]; a kid entry carries a copy of the child's n_t, c*,
//    activity and block address, so revisit_choice never touches the children's records and the next level's
//    block can be requested as soon as the child is chosen; header, first 32 kids and first 32 predictions are
//    requested together without knowing their counts;
//  * out-arcs are stored in creation order: petgraph iterates newest-first, so "first minimum" == highest slot
//    among equal keys and the curiosity sum runs from the last slot down;
//  * a node record holds its first four in-arcs (parent, kid slot) inline, so a cascade level is one 64-byte read
//    per frontier node; the in-arc's kid slot is where the cascade refreshes the parent's copy;
//  * the transposition map BTreeMap<ActionSet, NodeIndex> is an open-addressing table keyed by the W-word mask;
//  * walker state (parents, permitted mask, path mask) sits in shared memory while the warp runs.
// A launch advances every tree that is below `target_step` by at most one step; with max_episodes != 0 a tree
// that keeps hitting terminal nodes / transpositions yields after that many episodes and finishes its step in a
// later launch (trees are independent, so results do not depend on the interleaving).
#pragma once
#include "azb_common.cuh"
#include "azb_cost.cuh"

enum { AZB_F_ADD = 1, AZB_F_ROLLOUT = 2, AZB_F_INIT = 4, AZB_F_FIRST = 8, AZB_F_MULTI = 16 };

// optional phase timing (-DAZB_PROFILE): cycles of lane 0 per phase, summed into AzbGlobals::prof
#ifdef AZB_PROFILE
#define PROF_T0() long long prof_t0 = clock64()
#define PROF_ADD(cx, ph)                                       \
    do {                                                       \
        long long prof_t1 = clock64();                         \
        if ((cx).lane == 0) (cx).ct[16 + (ph)] += (uint32_t)(prof_t1 - prof_t0); \
        prof_t0 = prof_t1;                                     \
    } while (0)
#else
#define PROF_T0() do {} while (0)
#define PROF_ADD(cx, ph) do {} while (0)
#endif
#ifdef AZB_PROFILE
__device__ unsigned long long g_flag_time[65536];  // %globaltimer when the model last raised the tree's answer flag (pick-up latency)
__device__ uint4 g_tree_prof[65536];  // per tree, last launch: cycles, episodes(resets)+1, cost evals, sqrt terms
#endif
enum { PH_SEL = 0, PH_CUR, PH_PROBE, PH_ARC, PH_CASCADE, PH_COST, PH_INSERT, PH_RESET, PH_ADD, PH_PACK, PH_LOAD, PH_STORE };

struct WarpCtx {
    uint32_t *wk;      // walker block copy [WS]
    uint8_t *par;      // parents (bytes) inside wk
    uint32_t *perm;    // permitted mask [W]
    uint32_t *keym;    // path mask [W]
    uint8_t *rpar;     // root parents
    uint32_t *rperm;   // root permitted
    uint32_t *cur;     // scratch mask [W]: current-edge mask
    uint32_t *pfx;     // scratch [W+1]
    float *lbuf;       // children's c*, creation order [LCAP]
    uint32_t *fr;      // frontier buffers [4][FRONTIER_CAP]
    uint32_t *ct;      // workload counters [16]
    CostScratch *cs;   // lambda_1 program scratch
    const uint8_t *lut;  // child vertex of every action (block-shared); behind it, while W <= 32, the [N][W] action masks
                         // of the child vertices (tree_tables_fill)
    // per-tree slabs
    uint4 *node;       // 4 x uint4 per node
    uint2 *blk;        // 8-byte units
    uint4 *blk4;       // the same arena in 16-byte units
    uint2 *inl;
    uint32_t *key;
    uint32_t *hash;
    uint32_t *casc;    // two cascade work lists of cap_nodes entries each (continuation of the shared-memory lists)
    int lane;
    uint32_t err;
    bool full_count;   // all 16 workload counters (tests, roofline pass) or only LIVE / NOOP / INS (always counted)
};

// carve a warp's shared-memory region: walker block | cur mask | prefix | counters | one region shared by the
// children's c* (selection), the cascade work lists and the cost scratch (never live together)
__device__ __forceinline__ void ctx_bind_smem(const AzbLayout &L, WarpCtx &cx, uint32_t *base, const uint8_t *lut, int lane) {
    cx.lane = lane;
    cx.err = 0;
    cx.lut = lut;
    cx.wk = base;
    cx.par = (uint8_t *)(base + WK_HDR);
    cx.perm = base + WK_HDR + L.PW;
    cx.keym = cx.perm + L.W;
    cx.rpar = (uint8_t *)(cx.keym + L.W);
    cx.rperm = cx.keym + L.W + L.PW;
    uint32_t *p = base + ((L.WS + 3u) & ~3u);
    cx.cur = p;
    p += 64;
    cx.pfx = p;
    p += 64;
    cx.ct = p;
    p += 32;
    cx.lbuf = (float *)p;
    cx.fr = p;
    cx.cs = reinterpret_cast<CostScratch *>(p);
}
// point a WarpCtx at one tree's slabs
__device__ __forceinline__ void ctx_bind_tree(const AzbLayout &L, WarpCtx &cx, uint32_t tree) {
    cx.node = L.node + (size_t)tree * L.cap_nodes * 4;
    cx.blk = L.blk + (size_t)tree * L.cap_blk;
    cx.blk4 = reinterpret_cast<uint4 *>(cx.blk);
    cx.inl = L.inl + (size_t)tree * L.cap_in;
    cx.key = L.key + (size_t)tree * L.cap_nodes * L.W;
    cx.hash = L.hash + (size_t)tree * L.cap_hash;
    cx.casc = L.casc + (size_t)tree * 2u * L.cap_nodes;
}

__device__ __forceinline__ void count(WarpCtx &cx, int which, uint32_t n) {
    if (cx.full_count && cx.lane == 0) cx.ct[which] += n;
}

__device__ __forceinline__ uint32_t nth_set_bit(uint32_t mask, uint32_t r) {
#pragma unroll 1
    for (uint32_t i = 0; i < r; ++i) mask &= mask - 1;
    return __ffs(mask) - 1;
}

// hash of a W-word action-set mask held as (k0 = word lane, k1 = word lane+32) across the warp
// (WIDE = false: W <= 32, k1 is 0 and its term is a constant)
__device__ __forceinline__ uint32_t key_hash(uint32_t k0, uint32_t k1, int lane, uint32_t W) {
    uint32_t hv = (k0 * 0x9E3779B1u + (uint32_t)lane * 0x85EBCA77u) ^ ((k1 + 0x7F4A7C15u) * 0xC2B2AE3Du);
    hv ^= hv >> 15;
    hv *= 0x2C1B3C6Du;
    hv = (uint32_t)lane < W ? hv : 0u;
    hv = __reduce_xor_sync(0xffffffffu, hv);
    hv ^= hv >> 13;
    hv *= 0x297A2D39u;
    hv ^= hv >> 16;
    return hv;
}

// transposition-table probe of a tree's table for the key (k0, k1) with hash hv (key_hash): the index of the node with
// that key, or -1 with `slot` = the empty slot where the key goes.  The search kernels and the checkpoint load's rebuild
// (azb_ckpt.cuh) share it, so a table rebuilt by inserting nodes 0..n-1 in index order is the one the search built.
template <bool WIDE>  // W > 32 (N >= 47): the key's second word per lane
__device__ __forceinline__ int hash_probe(const AzbLayout &L, const uint32_t *hash, const uint32_t *key, uint32_t k0, uint32_t k1,
                                          int lane, uint32_t hv, uint32_t &slot) {
    const uint32_t fp = hv >> 21;
    slot = hv & (L.cap_hash - 1);
    for (uint32_t probes = 0; probes < L.cap_hash; ++probes) {
        const uint32_t e = hash[slot];
        if (e == 0u) break;
        if ((e >> 21) == fp) {
            const uint32_t idx = (e & 0x1fffffu) - 1u;
            bool eq = true;
            if ((uint32_t)lane < L.W) eq = key[(size_t)idx * L.W + lane] == k0;
            if constexpr (WIDE)
                if ((uint32_t)lane + 32 < L.W) eq = eq && (key[(size_t)idx * L.W + lane + 32] == k1);
            if (__all_sync(0xffffffffu, eq)) return (int)idx;
        }
        slot = (slot + 1) & (L.cap_hash - 1);
    }
    return -1;
}
// entry of node `node` (hash hv) in the empty slot hash_probe returned
__device__ __forceinline__ void hash_insert(uint32_t *hash, uint32_t slot, uint32_t node, uint32_t hv) {
    hash[slot] = (node + 1u) | ((hv >> 21) << 21);
}

// current-edge mask of the walker state into cx.cur (rooted_tree/mod.rs:60-72)
__device__ __forceinline__ void build_cur_mask(const AzbLayout &L, WarpCtx &cx) {
#pragma unroll 1
    for (uint32_t w = cx.lane; w < L.W; w += 32) cx.cur[w] = 0u;
    __syncwarp();
#pragma unroll 1
    for (uint32_t c = 2 + cx.lane; c + 1 < L.N; c += 32) {
        uint32_t e = azb_action_index(cx.par[c], c);
        atomicOr(&cx.cur[e >> 5], 1u << (e & 31));
    }
    __syncwarp();
}

// act (rooted_tree/space.rs:56-73): set the parent, drop every action of that child, extend the path set
// fill the block-shared tables (all `n_thr` threads of the block, before the barrier that precedes their first use)
__device__ __forceinline__ void tree_tables_fill(const AzbLayout &L, uint8_t *lut, uint32_t tid, uint32_t n_thr) {
    for (uint32_t a = tid; 4u * a < L.A; a += n_thr) reinterpret_cast<uint32_t *>(lut)[a] = reinterpret_cast<const uint32_t *>(L.lut)[a];
    if (L.W <= 32u) {
        uint32_t *am = reinterpret_cast<uint32_t *>(lut + azb_lut_bytes(L.A));
        const uint32_t stride = azb_amask_stride(L.W);
        for (uint32_t i = tid; i < L.N * stride; i += n_thr) {
            const uint32_t child = i / stride, w = i - child * stride;
            uint32_t m = 0u;
            if (child >= 2u && w < L.W) {  // the actions of `child` are first .. first + child - 1 (simple_graph/edge.rs:48-65)
                const uint32_t first = azb_child_first_action(child), last = first + child, b0 = w * 32u;
                const uint32_t s = max(first, b0), e = min(last, b0 + 32u);
                if (s < e) m = (e - s == 32u ? 0xffffffffu : ((1u << (e - s)) - 1u)) << (s - b0);
            }
            am[i] = m;
        }
    }
}

// STRIDE != 0: cx.lut is the block's table pair; rows of 8 words (STRIDE 8: the tree kernels for N <= 22) or of W words
// (STRIDE -1: N <= 46)
template <int STRIDE = 0>
__device__ __forceinline__ void walker_act(const AzbLayout &L, WarpCtx &cx, uint32_t a) {
    const uint32_t child = cx.lut[a];
    const uint32_t first = azb_child_first_action(child);
    if constexpr (STRIDE != 0) {  // one mask word per lane: the child's action mask comes from the block's table
        const uint32_t w = (uint32_t)cx.lane;
        const uint32_t *amask = reinterpret_cast<const uint32_t *>(cx.lut + azb_lut_bytes(L.A));
        if (w == 0u) cx.par[child] = (uint8_t)(a - first);
        if (w < L.W) cx.perm[w] &= ~amask[child * (STRIDE > 0 ? (uint32_t)STRIDE : L.W) + w];
        if (w == (a >> 5)) cx.keym[w] |= 1u << (a & 31);
        __syncwarp();
        return;
    }
    const uint32_t last = first + child;  // exclusive
    if (cx.lane == 0) cx.par[child] = (uint8_t)(a - first);
#pragma unroll 1
    for (uint32_t w = cx.lane; w < L.W; w += 32) {
        const uint32_t b0 = w * 32, b1 = b0 + 32;
        const uint32_t s = max(first, b0), e = min(last, b1);
        if (s < e) {
            const uint32_t len = e - s;
            const uint32_t m = (len == 32 ? 0xffffffffu : ((1u << len) - 1u)) << (s - b0);
            cx.perm[w] &= ~m;
        }
        if (w == (a >> 5)) cx.keym[w] |= 1u << (a & 31);
    }
    __syncwarp();
}

__device__ __forceinline__ void walker_reset(const AzbLayout &L, WarpCtx &cx) {  // tree/mod.rs:176-178
#pragma unroll 1
    for (uint32_t i = cx.lane; i < L.PW; i += 32) ((uint32_t *)cx.par)[i] = ((const uint32_t *)cx.rpar)[i];
#pragma unroll 1
    for (uint32_t w = cx.lane; w < L.W; w += 32) {
        cx.perm[w] = cx.rperm[w];
        cx.keym[w] = 0u;
    }
    __syncwarp();
}

__device__ __forceinline__ float prior_of(const AzbLayout &L, uint32_t tree, uint32_t a, uint32_t prior_step) {
    if (L.prior_mode == 1) return azb_hash_prior(L.prior_seed, L.first_root + tree, prior_step, a);
    return L.h[(size_t)tree * L.h_ld + a];
}

// add_actions (graph_operations.rs:32-56): one prediction per legal action, ascending; g = c_s - h (04-c21-tree.rs:103).
// Allocates the node's block [preds | header | kids] and publishes its address to the node record and to the copy in
// the creator's kid entry.
template <bool WIDE>  // WIDE: W > 32 (N >= 47); otherwise the second mask word per lane is compiled out
__device__ void tree_add_actions(const AzbLayout &L, WarpCtx &cx, uint32_t tree) {
    const int lane = cx.lane;
    const uint32_t pos = cx.wk[WK_POS];
    const float c_s = __uint_as_float(cx.wk[WK_PEND_C]);
    const uint32_t prior_step = cx.wk[WK_STEP];
    // the prior row streams into shared memory (coalesced) while the legal-action mask is built
    const bool hashed = L.prior_mode == 1;
    if (!hashed) {
        const float *hrow = L.h + (size_t)tree * L.h_ld;
#pragma unroll 4
        for (uint32_t a = lane; a < L.A; a += 32) cx.lbuf[a] = __ldcg(hrow + a);  // written by other SMs in the async kernel
    }
    build_cur_mask(L, cx);
    // legal = permitted minus current edges (space.rs:75-89); counts per word -> exclusive prefix
    uint32_t l0 = (uint32_t)lane < L.W ? (cx.perm[lane] & ~cx.cur[lane]) : 0u;
    uint32_t l1 = 0u;
    if constexpr (WIDE) l1 = (uint32_t)lane + 32 < L.W ? (cx.perm[lane + 32] & ~cx.cur[lane + 32]) : 0u;
    uint32_t s0 = __popc(l0), s1 = __popc(l1);
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t0 = __shfl_up_sync(0xffffffffu, s0, d);
        if (lane >= d) s0 += t0;
        if constexpr (WIDE) {
            const uint32_t t1 = __shfl_up_sync(0xffffffffu, s1, d);
            if (lane >= d) s1 += t1;
        }
    }
    const uint32_t tot0 = __shfl_sync(0xffffffffu, s0, 31);
    uint32_t cnt = tot0;
    if constexpr (WIDE) cnt += __shfl_sync(0xffffffffu, s1, 31);
    __syncwarp();
    if ((uint32_t)lane < L.W) {
        cx.cur[lane] = l0;
        cx.pfx[lane + 1] = s0;
    }
    if constexpr (WIDE) {
        if ((uint32_t)lane + 32 < L.W) {
            cx.cur[lane + 32] = l1;
            cx.pfx[lane + 33] = tot0 + s1;
        }
    }
    if (lane == 0) cx.pfx[0] = 0u;
    __syncwarp();
    if (cnt == 0u) {  // only a root can be terminal here: it stays without a block and inactive
        if (lane == 0) cx.wk[WK_FLAGS] &= ~1u;
        __syncwarp();
        return;
    }
    uint32_t lo = cx.wk[WK_NBLK] + cnt;  // header position in units; predictions sit right below it
    lo += lo & 1u;
    const uint32_t top = lo + 2u + 2u * cnt;
    if (top > L.cap_blk || cnt > 0xffffu) {
        cx.err = 3;
        return;
    }
    const uint32_t lo2 = lo >> 1;
#pragma unroll 1
    for (uint32_t j = lane; j < cnt; j += 32) {
        // word holding the j-th legal action: largest w with pfx[w] <= j
        uint32_t a0 = 0, a1 = L.W;  // invariant pfx[a0] <= j < pfx[a1]
        while (a1 - a0 > 1) {
            uint32_t mid = (a0 + a1) >> 1;
            if (cx.pfx[mid] <= j)
                a0 = mid;
            else
                a1 = mid;
        }
        const uint32_t a = a0 * 32 + nth_set_bit(cx.cur[a0], j - cx.pfx[a0]);
        const float h = hashed ? azb_hash_prior(L.prior_seed, L.first_root + tree, prior_step, a) : cx.lbuf[a];
        if (h != h) cx.err = 4;
        const float g = __fsub_rn(c_s, h);
        cx.blk[lo - 1u - j] = make_uint2(__float_as_uint(g), a);
    }
    cx.err = __reduce_or_sync(0xffffffffu, cx.err);
    if (lane == 0) {
        cx.blk4[lo2] = make_uint4(__float_as_uint(c_s), cnt << 16, pos, 0u);
        uint32_t *rec = reinterpret_cast<uint32_t *>(cx.node + (size_t)pos * 4);
        rec[3] = cnt << 16;  // exhausted_children = 0
        rec[4] = lo2;
        const uint32_t pk = cx.wk[WK_PKIDX];
        if (pk != AZB_LO_NONE) reinterpret_cast<uint32_t *>(cx.blk4 + pk)[1] = lo2 | 0x80000000u;  // now active
        if (pos == 0u) cx.wk[WK_ROOTLO] = lo2;
        cx.wk[WK_CURLO] = lo2;
        cx.wk[WK_NBLK] = top;
        cx.wk[WK_NPREDS] += cnt;
        cx.wk[WK_FLAGS] &= ~1u;
        if (cx.full_count) cx.ct[CT_PRED] += cnt;
    }
    __syncwarp();
}

// cascade_new_terminal / cascade_old_node (empty_transitions.rs:50-127).
// The reference walks the ancestors of the arc's source level by level; every ancestor is updated exactly once with
// the same (c*, n_t of the target), and only the exhausted-children counts flow between levels.  That allows a
// two-phase form that needs far fewer dependent round trips (DESIGN.md §4.1):
//   A. value pass over ALL ancestors: the walker's own path (known, WK_PATH) is the first work list and is processed
//      in one go; in-arcs that lead off the path (transposition arcs) seed further work lists; a bitmap keeps every
//      node to one visit.  Each node gets "c* <- min / else n_t += 1 (old: n_t = max(n_t, n_t of target))" and
//      refreshes the copies held by its parents' kid entries.  A work list lives in shared memory up to
//      AZB_FRONTIER_CAP entries and continues in the tree's global scratch (L.casc, cap_nodes entries per list), so
//      no DAG shape can overflow it — the reference's BTreeMap has no limit either.
//   B. exhaustion pass: exhausted_children += 1 at the source if the arc's target is inactive; a node whose count
//      thereby reaches its prediction count became inactive and hands +1 to each of its parents.  Depth first with an
//      explicit stack: a parent is one level shallower than its child, so the stack never holds more than depth + 1
//      entries (<= N - 2), and the increments commute, so the order does not matter.
// Before a cascade every ancestor of the (active) source is active, so "inactive after the update" in the reference
// (:65-70) is exactly "became inactive in this cascade".
__device__ __forceinline__ uint32_t wl_get(const uint32_t *sh, const uint32_t *gl, uint32_t cap, uint32_t i) {
    return i < cap ? sh[i] : gl[i - cap];
}
__device__ __forceinline__ void wl_put(uint32_t *sh, uint32_t *gl, uint32_t cap, uint32_t i, uint32_t v) {
    if (i < cap)
        sh[i] = v;
    else
        gl[i - cap] = v;
}
__device__ void tree_cascade(const AzbLayout &L, WarpCtx &cx, uint32_t src, uint32_t depth, float cstar, uint32_t ntt,
                             uint32_t e0, bool old) {
    const int lane = cx.lane;
    const uint32_t FULL = 0xffffffffu, lt = (1u << lane) - 1u;
    uint32_t *wa = cx.fr, *wb = cx.fr + AZB_FRONTIER_CAP;
    uint32_t *ga = cx.casc, *gb = cx.casc + L.cap_nodes;  // the lists' continuation beyond AZB_FRONTIER_CAP entries
    uint32_t *vis = cx.fr + 3 * AZB_FRONTIER_CAP;
    const uint32_t nwords = (L.cap_nodes + 31u) >> 5;
#pragma unroll 1
    for (uint32_t w = lane; w < nwords; w += 32) vis[w] = 0u;
    __syncwarp();
    const uint32_t fcap = L.frontier_cap;  // entries a list keeps in shared memory (AZB_FRONTIER_CAP; tests shrink it)
    uint32_t ncur = depth + 1u;
#pragma unroll 1
    for (uint32_t i = lane; i < ncur; i += 32) {
        const uint32_t p = cx.wk[WK_PATH + i];
        wl_put(wa, ga, fcap, i, p);
        atomicOr(&vis[p >> 5], 1u << (p & 31));
    }
    __syncwarp();
    // ---- A. value pass
    while (ncur > 0) {
        uint32_t nnext = 0, links = 0;
        count(cx, CT_CN, ncur);
        if (ncur > fcap && lane == 0) atomicAdd(&L.g->casc_spills, 1u);  // this wave continues in the global list
        for (uint32_t base = 0; base < ncur; base += 32) {
            const uint32_t i = base + lane;
            const bool valid = i < ncur;
            uint32_t nin = 0, in_off = 0, w1 = 0, w2 = 0, w3 = 0;
            uint4 q2 = make_uint4(0, 0, 0, 0), q3 = make_uint4(0, 0, 0, 0);
            if (valid) {
                uint4 *rec = cx.node + (size_t)wl_get(wa, ga, fcap, i) * 4;
                uint4 q0 = rec[0];
                const uint4 q1 = rec[1];
                q2 = rec[2];
                q3 = rec[3];
                float cs = __uint_as_float(q0.y);
                uint32_t nt = q0.z;
                if (cs > cstar)
                    cs = cstar;
                else
                    nt += 1;
                if (old) nt = max(nt, ntt);
                q0.y = __float_as_uint(cs);
                q0.z = nt;
                rec[0] = q0;  // exhausted_children is untouched here (phase B)
                nin = q1.y;
                in_off = q1.z;
                w1 = q1.x | (((q0.w & 0xffffu) < (q0.w >> 16)) ? 0x80000000u : 0u);
                w2 = nt;
                w3 = q0.y;
                links += nin;
            }
            // parents: refresh the copy in their kid entry, enlist the ones not seen yet
            const uint32_t maxin = __reduce_max_sync(FULL, nin);
            for (uint32_t k = 0; k < maxin; ++k) {
                const bool has = valid && k < nin;
                uint32_t q = 0, kx = 0;
                if (has) {
                    if (k < 4u) {
                        q = k == 0 ? q2.x : (k == 1 ? q2.z : (k == 2 ? q3.x : q3.z));
                        kx = k == 0 ? q2.y : (k == 1 ? q2.w : (k == 2 ? q3.y : q3.w));
                    } else {
                        const uint2 ent = cx.inl[in_off + k - 4u];
                        q = ent.x;
                        kx = ent.y;
                    }
                    uint32_t *kp = reinterpret_cast<uint32_t *>(cx.blk4 + kx);
                    kp[1] = w1;
                    *reinterpret_cast<uint2 *>(kp + 2) = make_uint2(w2, w3);
                }
                bool fresh = false;
                if (has) {
                    const uint32_t bit = 1u << (q & 31);
                    fresh = (atomicOr(&vis[q >> 5], bit) & bit) == 0u;
                }
                const uint32_t bal = __ballot_sync(FULL, fresh);
                // at most cap_nodes distinct nodes are ever enlisted: the global continuation cannot overflow
                if (fresh) wl_put(wb, gb, fcap, nnext + __popc(bal & lt), q);
                nnext += __popc(bal);
            }
        }
        if (cx.full_count) {
            links = __reduce_add_sync(FULL, links);
            count(cx, CT_DCN, links);
        }
        uint32_t *t = wa;
        wa = wb;
        wb = t;
        t = ga;
        ga = gb;
        gb = t;
        ncur = nnext;
        __syncwarp();
    }
    // ---- B. exhaustion pass
    if (e0 == 0u) return;
    uint32_t *stk = cx.fr;  // (node, next in-arc, in-arc count, overflow in-arc offset) per level; the work lists are done
    uint32_t sp = 0, p = src;
    for (;;) {
        uint4 *rec = cx.node + (size_t)p * 4;
        const uint4 q0 = rec[0], q1 = rec[1];
        const uint32_t ex = (q0.w & 0xffffu) + 1u, cnt = q0.w >> 16, nin = q1.y;
        __syncwarp();
        if (lane == 0) reinterpret_cast<uint32_t *>(rec)[3] = ex | (cnt << 16);
        if (ex == cnt && nin != 0u) {  // p just became inactive: its parents' copies lose the active bit, each parent gets +1
#pragma unroll 1
            for (uint32_t k = lane; k < nin; k += 32) {
                const uint2 ent = k < 4u ? reinterpret_cast<const uint2 *>(rec + 2)[k] : cx.inl[q1.z + k - 4u];
                reinterpret_cast<uint32_t *>(cx.blk4 + ent.y)[1] = q1.x;
            }
            if (lane == 0) *reinterpret_cast<uint4 *>(stk + 4u * sp) = make_uint4(p, 0u, nin, q1.z);
            ++sp;
        }
        __syncwarp();
        if (sp == 0u) break;
        const uint4 top = *reinterpret_cast<const uint4 *>(stk + 4u * (sp - 1u));
        const uint2 ent = top.y < 4u ? reinterpret_cast<const uint2 *>(cx.node + (size_t)top.x * 4 + 2)[top.y] : cx.inl[top.w + top.y - 4u];
        __syncwarp();
        if (top.y + 1u < top.z) {
            if (lane == 0) stk[4u * (sp - 1u) + 1u] = top.y + 1u;
        } else {
            --sp;
        }
        p = ent.x;
    }
}

// the step of `tree` is complete: publish its argmin candidate (optimizer/mod.rs:203-219) and advance its clock
__device__ __forceinline__ void step_done(const AzbLayout &L, WarpCtx &cx, uint32_t tree) {
    if (cx.lane == 0) {
        const uint32_t step = cx.wk[WK_STEP];
        if (step < L.cap_steps) {
            // a release store: azb_step_poll reads this row from the host while the kernel runs, and whoever sees the
            // entry must also see the node it names (its key and record were plain stores of this warp)
            uint2 *dst = L.cand + (size_t)(step + 1u) * L.B + tree;
            asm volatile("st.release.gpu.global.v2.u32 [%0], {%1, %2};" ::"l"(dst), "r"(cx.wk[WK_CAND_C]), "r"(cx.wk[WK_CAND_NODE]) : "memory");
        } else
            cx.err = 3;
        cx.wk[WK_STEP] = step + 1u;
        cx.wk[WK_CAND_C] = 0xffffffffu;
        cx.wk[WK_CAND_NODE] = 0u;
    }
    cx.err = __reduce_or_sync(0xffffffffu, cx.err);
}

// PUCT prior weight w_j = (1 - c_s) + g_j, or +0 where negative (azb.h, AZB_SELECT_PUCT step 2)
__device__ __forceinline__ float puct_weight(float one_minus_c, uint32_t g_bits) {
    const float x = __fadd_rn(one_minus_c, __uint_as_float(g_bits));
    return x < 0.f ? 0.f : x;
}
__device__ __forceinline__ float puct_butterfly(float x) {  // every lane ends with the chunk sum of azb.h step 3
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) x = __fadd_rn(x, __shfl_xor_sync(0xffffffffu, x, m));
    return x;
}

// AZB_SELECT_PUCT in place of next_action at the active node whose block header is the 16-byte unit lo2 (the rule is
// in azb.h).  kd / pr are the first 32 kid entries / predictions, already loaded.  Returns j for Unvisited(j) with its
// prediction word in y, or -1 for Visited with the chosen kid entry's first two words in w0 / w1; sets cx.err.
// The kid of an arc'd prediction is found through the warp's scratch (cx.lbuf as u32: kid slot by action id).
__device__ __forceinline__ int puct_select(const AzbLayout &L, WarpCtx &cx, uint32_t lo2, float c_s, uint32_t n_out,
                                           uint32_t cnt, uint4 kd, uint2 pr, uint32_t &w0, uint32_t &w1, uint32_t &y) {
    const int lane = cx.lane;
    const uint32_t FULL = 0xffffffffu;
    uint32_t *kslot = reinterpret_cast<uint32_t *>(cx.lbuf);
    count(cx, CT_CUR, 1);
    count(cx, CT_CAND, cnt);
    // 1. N_s = 1 + sum_k (n_k + 1)
    uint32_t ns = 1u;
#pragma unroll 1
    for (uint32_t base = 0; base < n_out; base += 32) {
        if (base) kd = cx.blk4[lo2 + 1u + base + lane];
        const uint32_t t = base + lane;
        uint32_t v = 0u;
        if (t < n_out) {
            kslot[kd.x >> 20] = t;
            v = kd.z + 1u;
        }
        ns += __reduce_add_sync(FULL, v);
    }
    __syncwarp();
    if (ns >= (1u << 24)) {
        cx.err = 3;
        return -1;
    }
    const float sq = __fsqrt_rn(__uint2float_rn(ns));
    // 2-3. Z: butterfly per chunk, chunks folded left to right
    const float omc = __fsub_rn(1.f, c_s);
    float z = 0.f;
#pragma unroll 1
    for (uint32_t base = 0; base < cnt; base += 32) {
        if (base) pr = cx.blk[2u * lo2 - 1u - base - lane];
        const float s = puct_butterfly(base + lane < cnt ? puct_weight(omc, pr.x) : 0.f);
        z = base ? __fadd_rn(z, s) : s;
    }
    const float p0 = __fdiv_rn(1.f, __uint2float_rn(cnt));  // Z == 0
    // 4-6. scores, first maximum in ascending j
    float best = 0.f;
    int bj = -1;
    uint32_t by = 0u, bw0 = 0u, bw1 = 0u;
#pragma unroll 1
    for (uint32_t base = 0; base < cnt; base += 32) {
        if (cnt > 32u) pr = cx.blk[2u * lo2 - 1u - base - lane];
        const uint32_t j = base + lane;
        bool cand = false;
        float sc = 0.f;
        uint32_t kx = 0u, ky = 0u;
        if (j < cnt) {
            const float p = z == 0.f ? p0 : __fdiv_rn(puct_weight(omc, pr.x), z);
            float q = __uint_as_float(pr.x);
            uint32_t n1 = 1u;  // 1 + n
            cand = true;
            if ((pr.y >> 11) & 1u) {
                const uint4 kid = cx.blk4[lo2 + 1u + kslot[pr.y & 0x7ffu]];
                cand = (kid.y >> 31) != 0u;
                q = __fsub_rn(c_s, __uint_as_float(kid.w));
                n1 = kid.z + 2u;
                kx = kid.x;
                ky = kid.y;
            }
            sc = __fadd_rn(q, __fdiv_rn(__fmul_rn(__fmul_rn(L.puct_c, p), sq), __uint2float_rn(n1)));
            if (cand && sc != sc) cx.err = 4;
        }
        if (!__any_sync(FULL, cand)) continue;
        const float red = azb_ord2f(__reduce_max_sync(FULL, cand ? azb_f2ord(sc) : 0u));
        if (bj < 0 || red > best) {  // earlier chunks win ties
            const int wl = __ffs(__ballot_sync(FULL, cand && sc == red)) - 1;
            best = red;
            bj = (int)base + wl;
            by = __shfl_sync(FULL, pr.y, wl);
            bw0 = __shfl_sync(FULL, kx, wl);
            bw1 = __shfl_sync(FULL, ky, wl);
        }
    }
    cx.err = __reduce_or_sync(FULL, cx.err);
    if (cx.err) return -1;
    if (bj < 0) {
        cx.err = 6;
        return -1;
    }
    if ((by >> 11) & 1u) {
        w0 = bw0;
        w1 = bw1;
        return -1;
    }
    y = by;
    return bj;
}

// `early(cx)` is called as soon as the step's new node is known to be non-terminal — BEFORE its cost is evaluated and the
// node is inserted: the walker's state is final from that point on, so the asynchronous kernel hands the state vector to
// the model there and the cost evaluation (~5 us) and the insert overlap the model's round trip.  The lock step passes a
// no-op and packs after the walk (cx.cur still holds the current-edge mask then).
struct TreeNoEarly {
    __device__ __forceinline__ void operator()(WarpCtx &) const {}
};
// PUCT: AZB_SELECT_PUCT in place of next_action (azb.h); the default instantiations carry none of its code
template <int DEPTH, bool PUCT = false, class Early = TreeNoEarly>
__device__ void tree_rollout(const AzbLayout &L, WarpCtx &cx, uint32_t tree, uint32_t max_episodes, Early early = Early()) {
    const int lane = cx.lane;
    const uint32_t FULL = 0xffffffffu;
    uint32_t pos = cx.wk[WK_POS], depth = cx.wk[WK_DEPTH], lo2 = cx.wk[WK_CURLO];
    uint32_t guard = 0, episodes = 0;
    for (;;) {
        if (cx.err) break;
        if (++guard > 4u * L.cap_nodes + 64u) {
            cx.err = 6;
            break;
        }
        // ---- next_action (next_action.rs:11-26) at `pos`
        PROF_T0();
        bool active = lo2 != AZB_LO_NONE;
        uint4 hd = make_uint4(0, 0, 0, 0), kd = make_uint4(0, 0, 0, 0);
        uint2 pr = make_uint2(0, 0);
        if (active) {  // one round trip: header, first 32 kids, first 32 predictions (+ the root's own record)
            hd = cx.blk4[lo2];
            kd = cx.blk4[lo2 + 1u + lane];
            pr = cx.blk[2u * lo2 - 1u - lane];
            if (pos == 0u) {
                const uint4 r0 = cx.node[0];
                active = (r0.w & 0xffffu) < (r0.w >> 16);
            }
        }
        if (!active) {  // next_action.rs:12-14; only an exhausted root can be here (tree/mod.rs:220-229)
            if (depth != 0u)
                cx.err = 6;
            else {
                if (lane == 0) cx.ct[CT_NOOP] += 1u;
                step_done(L, cx, tree);
            }
            break;
        }
        const float c_s = __uint_as_float(hd.x);
        const uint32_t n_out = hd.y & 0xffffu, cnt = hd.y >> 16;
        count(cx, CT_SEL, 1);
        count(cx, CT_DSEL, n_out);
        bool visit;
        int chosen_j = -1;
        uint32_t chosen_y = 0, best_w0 = 0, best_w1 = 0;
        if constexpr (PUCT) {  // AZB_SELECT_PUCT: a kernel instantiation of its own
            chosen_j = puct_select(L, cx, lo2, c_s, n_out, cnt, kd, pr, best_w0, best_w1, chosen_y);
            if (cx.err) break;
            visit = chosen_j < 0;
        } else {
            // ---- revisit_choice (next_action.rs:28-53): first minimum of (n_t, c*) over active children, newest first
            unsigned long long best_key = ~0ull;
            int best_t = -1;
            for (uint32_t base = 0; base < n_out; base += 32) {
                if (base) kd = cx.blk4[lo2 + 1u + base + lane];
                const uint32_t t = base + lane;
                bool act_t = false;
                uint32_t oc = 0xffffffffu;
                if (t < n_out) {
                    if (n_out > 32u) cx.lbuf[t] = __uint_as_float(kd.w);  // single-chunk nodes store only if curiosity runs
                    act_t = (kd.y >> 31) != 0u;
                    oc = azb_f2ord(__uint_as_float(kd.w));
                }
                const uint32_t ntmin = __reduce_min_sync(FULL, act_t ? kd.z : 0xffffffffu);
                if (__any_sync(FULL, act_t)) {
                    const bool cand_t = act_t && kd.z == ntmin;
                    const uint32_t cmin = __reduce_min_sync(FULL, cand_t ? oc : 0xffffffffu);
                    const unsigned long long mk = ((unsigned long long)ntmin << 32) | cmin;
                    if (mk <= best_key) {  // a later chunk holds newer arcs: it wins ties
                        const uint32_t bal = __ballot_sync(FULL, cand_t && oc == cmin);
                        const int wl = 31 - __clz(bal);  // newest arc among equals
                        best_key = mk;
                        best_t = (int)base + wl;
                        best_w0 = __shfl_sync(FULL, kd.x, wl);
                        best_w1 = __shfl_sync(FULL, kd.y, wl);
                    }
                }
            }
            __syncwarp();
            PROF_ADD(cx, PH_SEL);
            const bool have_r = best_t >= 0;
            const uint32_t tol = depth < L.tol_len ? L.tol[depth] : L.tol_default;  // 04-c21-tree.rs:136-138
            visit = have_r && (uint32_t)(best_key >> 32) < tol;                    // next_action.rs:16-20
            if (!visit) {
                // ---- max_curiosity (next_action.rs:55-88)
                if (n_out <= 32u) {
                    if ((uint32_t)lane < n_out) cx.lbuf[lane] = __uint_as_float(kd.w);
                    __syncwarp();
                }
                count(cx, CT_CUR, 1);
                count(cx, CT_CAND, cnt);
    #ifdef AZB_PROFILE
                if (lane == 0) cx.ct[30] += cnt * n_out;
    #endif
                const bool no_kids = n_out == 0;
                uint32_t bk32 = 0u;
                for (uint32_t base = 0; base < cnt; base += 32) {
                    if (base) pr = cx.blk[2u * lo2 - 1u - base - lane];
                    const uint32_t j = base + lane;
                    bool cand_j = false;
                    uint32_t ov = 0u;
                    if (j < cnt && ((pr.y >> 11) & 1u) == 0u) {  // no arc yet (:68-71)
                        cand_j = true;
                        const float v = __fsub_rn(c_s, __uint_as_float(pr.x));
                        if (no_kids) {
                            if (v != v) cx.err = 4;
                            ov = azb_f2ord(v);
                        } else {
                            float cur = 0.f;
    #pragma unroll 2
                            for (int t = (int)n_out - 1; t >= 0; --t)  // newest first, left fold (:79-82)
                                cur = __fadd_rn(cur, __fsqrt_rn(fabsf(__fsub_rn(cx.lbuf[t], v))));
                            if (cur != cur) cx.err = 4;
                            ov = azb_f2ord(cur);
                        }
                    }
                    if (!__any_sync(FULL, cand_j)) continue;
                    if (no_kids) {  // first minimum (:73-75): earlier chunks win ties
                        const uint32_t red = __reduce_min_sync(FULL, cand_j ? ov : 0xffffffffu);
                        if (chosen_j < 0 || red < bk32) {
                            bk32 = red;
                            const int wl = __ffs(__ballot_sync(FULL, cand_j && ov == red)) - 1;
                            chosen_j = (int)base + wl;
                            chosen_y = __shfl_sync(FULL, pr.y, wl);
                        }
                    } else {  // last maximum (:85): later chunks win ties
                        const uint32_t red = __reduce_max_sync(FULL, cand_j ? ov : 0u);
                        if (chosen_j < 0 || red >= bk32) {
                            bk32 = red;
                            const int wl = 31 - __clz(__ballot_sync(FULL, cand_j && ov == red));
                            chosen_j = (int)base + wl;
                            chosen_y = __shfl_sync(FULL, pr.y, wl);
                        }
                    }
                }
                cx.err = __reduce_or_sync(FULL, cx.err);
                PROF_ADD(cx, PH_CUR);
                if (cx.err) break;
                if (chosen_j < 0) {
                    if (have_r)
                        visit = true;  // next_action.rs:24
                    else {
                        cx.err = 6;
                        break;
                    }
                }
            }
        }
        if (visit) {  // tree/mod.rs:139-159
            count(cx, CT_VISIT, 1);
            walker_act<(DEPTH == 3 ? 8 : DEPTH == 4 ? -1 : 0)>(L, cx, best_w0 >> 20);
            pos = best_w0 & 0xfffffu;
            lo2 = best_w1 & 0x7fffffffu;
            depth += 1;
            if (lane == 0) cx.wk[WK_PATH + depth] = pos;
            PROF_ADD(cx, PH_SEL);
            continue;
        }
        // ---- Unvisited(j) (tree/mod.rs:160-218)
        const uint32_t a = chosen_y & 0x7ffu, j = (uint32_t)chosen_j;
        count(cx, CT_PROBE, 1);
        // key of the successor = path + a; look it up
        const uint32_t k0 = (uint32_t)lane < L.W ? (cx.keym[lane] | (((a >> 5) == (uint32_t)lane) ? 1u << (a & 31) : 0u)) : 0u;
        uint32_t k1 = 0u;
        if constexpr (DEPTH == 5)  // W > 32 only for N >= 47
            k1 = (uint32_t)lane + 32 < L.W ? (cx.keym[lane + 32] | (((a >> 5) == (uint32_t)lane + 32) ? 1u << (a & 31) : 0u)) : 0u;
        const uint32_t hv = key_hash(k0, k1, lane, L.W);
        uint32_t slot;
        const int hit = hash_probe<DEPTH == 5>(L, cx.hash, cx.key, k0, k1, lane, hv, slot);
        PROF_ADD(cx, PH_PROBE);
        const uint32_t kidx = lo2 + 1u + n_out;  // this arc's kid entry (16-byte index)
        const uint32_t narcs = cx.wk[WK_NARCS];
        if (narcs >= (1u << 20)) {
            cx.err = 3;
            break;
        }
        bool reset = false, casc_old = false;
        float casc_c = 0.f;
        uint32_t casc_n = 0u, casc_e = 0u;
        if (hit >= 0) {  // transposition (tree/mod.rs:172-179)
            count(cx, CT_HIT, 1);
            uint4 *rec = cx.node + (size_t)hit * 4;
            const uint4 q0 = rec[0], q1 = rec[1];
            const bool act_o = (q0.w & 0xffffu) < (q0.w >> 16);
            const uint32_t nin = q1.y;
            if (nin >= q1.w) {  // a node of depth d has at most d parents
                cx.err = 3;
                break;
            }
            if (lane == 0) {  // add_arc (graph_operations.rs:18-30)
                cx.blk4[kidx] = make_uint4((uint32_t)hit | (a << 20), q1.x | (act_o ? 0x80000000u : 0u), q0.z, q0.y);
                reinterpret_cast<uint32_t *>(cx.blk4 + lo2)[1] = (n_out + 1u) | (cnt << 16);
                cx.blk[2u * lo2 - 1u - j].y = a | (1u << 11) | (narcs << 12);
                if (nin < 4u)
                    *reinterpret_cast<uint2 *>(reinterpret_cast<uint32_t *>(rec) + 8 + 2 * nin) = make_uint2(pos, kidx);
                else
                    cx.inl[q1.z + nin - 4u] = make_uint2(pos, kidx);
                reinterpret_cast<uint32_t *>(rec)[5] = nin + 1u;
                cx.wk[WK_NARCS] = narcs + 1u;
                if (cx.full_count) cx.ct[CT_ARC] += 1;
            }
            __syncwarp();
            PROF_ADD(cx, PH_ARC);
            casc_c = __uint_as_float(q0.y);
            casc_n = q0.z;
            casc_e = act_o ? 0u : 1u;
            casc_old = true;
            reset = true;
        } else {
            // ---- new node (tree/mod.rs:181-216)
            walker_act<(DEPTH == 3 ? 8 : DEPTH == 4 ? -1 : 0)>(L, cx, a);
            const uint32_t ndepth = depth + 1;
            // is_terminal (nabla/space/mod.rs:27-29) first: it only needs the state
            build_cur_mask(L, cx);
            bool any = false;
#pragma unroll 1
            for (uint32_t w = lane; w < L.W; w += 32) any = any || ((cx.perm[w] & ~cx.cur[w]) != 0u);
            any = __any_sync(FULL, any);
            if (any) early(cx);
            uint32_t mu = 0;
            const double l1 = azb_cost_warp<DEPTH>(L.N, cx.par, cx.cs, lane, &mu);
            if (!(l1 >= 1.4)) {  // ordered_edge.rs:79
                cx.err = 5;
                break;
            }
            const float c_new = azb_evaluate(mu, l1, L.c_lower, L.slope);
            PROF_ADD(cx, PH_COST);
            if (lane == 0) cx.ct[CT_INS] += 1u;
            const uint32_t nn = cx.wk[WK_NNODES], in_off = cx.wk[WK_INTOP];
            const uint32_t in_need = ndepth > 4u ? ndepth - 4u : 0u;
            if (nn >= L.cap_nodes || in_off + in_need > L.cap_in) {
                cx.err = 3;
                break;
            }
            if (lane < 4) {  // StateWeight::new (state_weight.rs:13-21) + the creating arc as in-arc 0
                uint4 q;
                if (lane == 0)
                    q = make_uint4(__float_as_uint(c_new), __float_as_uint(c_new), 0u, 0u);
                else if (lane == 1)
                    q = make_uint4(AZB_LO_NONE, 1u, in_off, ndepth);
                else if (lane == 2)
                    q = make_uint4(pos, kidx, 0u, 0u);
                else
                    q = make_uint4(0u, 0u, 0u, 0u);
                cx.node[(size_t)nn * 4 + lane] = q;
            }
            if ((uint32_t)lane < L.W) cx.key[(size_t)nn * L.W + lane] = k0;
            if constexpr (DEPTH == 5)
                if ((uint32_t)lane + 32 < L.W) cx.key[(size_t)nn * L.W + lane + 32] = k1;
            if (lane == 0) {
                hash_insert(cx.hash, slot, nn, hv);
                cx.wk[WK_NNODES] = nn + 1;
                cx.wk[WK_INTOP] = in_off + in_need;
                // add_arc: the child is inactive until its own add_actions (actions = 0..0)
                cx.blk4[kidx] = make_uint4(nn | (a << 20), AZB_LO_NONE, 0u, __float_as_uint(c_new));
                reinterpret_cast<uint32_t *>(cx.blk4 + lo2)[1] = (n_out + 1u) | (cnt << 16);
                cx.blk[2u * lo2 - 1u - j].y = a | (1u << 11) | (narcs << 12);
                cx.wk[WK_NARCS] = narcs + 1u;
                if (cx.full_count) cx.ct[CT_ARC] += 1;
                // argmin candidate: first minimum of c over this step's new nodes (optimizer/mod.rs:208-213)
                const uint32_t oc = azb_f2ord(c_new);
                if (oc < cx.wk[WK_CAND_C]) {
                    cx.wk[WK_CAND_C] = oc;
                    cx.wk[WK_CAND_NODE] = nn;
                }
            }
            __syncwarp();
            PROF_ADD(cx, PH_INSERT);
            if (!any) {
                count(cx, CT_TERM, 1);
                casc_c = c_new;
                casc_n = 0u;
                casc_e = 1u;
                casc_old = false;
                reset = true;
            } else {
                pos = nn;
                depth = ndepth;
                lo2 = AZB_LO_NONE;
                if (lane == 0) {
                    cx.wk[WK_PATH + ndepth] = nn;
                    cx.wk[WK_FLAGS] |= 1u;
                    cx.wk[WK_PEND_C] = __float_as_uint(c_new);
                    cx.wk[WK_PKIDX] = kidx;
                }
                if (lane == 0) cx.ct[CT_LIVE] += 1u;
                __syncwarp();
                step_done(L, cx, tree);
                break;  // tree/mod.rs:212-215
            }
        }
        if (reset) {
            // one call site for both cascades (transposition arc / new terminal node): the body is 9 KB of code
            tree_cascade(L, cx, pos, depth, casc_c, casc_n, casc_e, casc_old);
            PROF_ADD(cx, PH_CASCADE);
            walker_reset(L, cx);
            pos = 0;
            depth = 0;
            lo2 = cx.wk[WK_ROOTLO];
            count(cx, CT_RESET, 1);
            PROF_ADD(cx, PH_RESET);
            if (max_episodes && ++episodes >= max_episodes) break;  // yield: the step continues in the next launch
        }
    }
    if (lane == 0) {
        cx.wk[WK_POS] = pos;
        cx.wk[WK_DEPTH] = depth;
        cx.wk[WK_CURLO] = lo2;
    }
    __syncwarp();
}

// write_vec (rooted_tree/space.rs:91-101): [A one-hot of current edges | A permitted mask].  Both halves are bit
// masks in shared memory (cx.cur must hold the current-edge mask of the walker state: build_cur_mask).
__device__ __forceinline__ uint32_t pack_bit(const AzbLayout &L, const WarpCtx &cx, uint32_t i) {
    const uint32_t j = i < L.A ? i : i - L.A;
    const uint32_t word = i < L.A ? cx.cur[j >> 5] : cx.perm[j >> 5];
    return (word >> (j & 31)) & 1u;
}
// BF16_ONLY: the caller knows the rows go out as bf16 (the asynchronous kernel): the f32 path is compiled out
template <bool BF16_ONLY = false>
__device__ __forceinline__ void tree_pack(const AzbLayout &L, WarpCtx &cx, uint32_t tree, uint16_t *row_override = nullptr) {
    if (BF16_ONLY || L.sv16) {
        // tensor-core MLP: the row goes out as bf16 (1.0 = 0x3F80), eight entries per 128-bit store; the row pitch is
        // a multiple of 64 entries and the tail beyond 2A stays zero
        uint16_t *row = row_override ? row_override : L.sv16 + (size_t)tree * L.sv16_ld;
        const uint32_t n2 = 2 * L.A;
#pragma unroll 1
        for (uint32_t i = 8u * cx.lane; i < n2; i += 256) {
            // eight consecutive entries = eight mask bits: taken with one 64-bit shift when the chunk lies inside one
            // half of the vector (always, when A is a multiple of 8), bit by bit otherwise
            uint32_t bits = 0;
            if (i + 8u <= L.A || (i >= L.A && i + 8u <= n2)) {
                const uint32_t *m = i < L.A ? cx.cur : cx.perm;
                const uint32_t j = i < L.A ? i : i - L.A;
                const uint32_t w0 = m[j >> 5], w1 = ((j & 31u) > 24u) ? m[(j >> 5) + 1u] : 0u;
                bits = (uint32_t)((((unsigned long long)w1 << 32) | w0) >> (j & 31u)) & 0xffu;
            } else {
#pragma unroll 1
                for (uint32_t q = 0; q < 8u; ++q)
                    if (i + q < n2) bits |= pack_bit(L, cx, i + q) << q;
            }
            uint32_t w[4];
#pragma unroll
            for (int q = 0; q < 4; ++q)
                w[q] = (((bits >> (2 * q)) & 1u) * 0x3F80u) | (((bits >> (2 * q + 1)) & 1u) * 0x3F800000u);
            *reinterpret_cast<uint4 *>(row + i) = make_uint4(w[0], w[1], w[2], w[3]);
        }
        return;
    }
    if constexpr (BF16_ONLY) return;
    float *row = L.sv + (size_t)tree * L.sv_ld;
    if ((L.A & 1u) == 0u && (L.sv_ld & 3u) == 0u) {  // rows are 16-byte aligned: one 128-bit store per four entries
        for (uint32_t i = 4u * cx.lane; i < 2 * L.A; i += 128)
            *reinterpret_cast<float4 *>(row + i) =
                make_float4(pack_bit(L, cx, i) ? 1.f : 0.f, pack_bit(L, cx, i + 1) ? 1.f : 0.f,
                            pack_bit(L, cx, i + 2) ? 1.f : 0.f, pack_bit(L, cx, i + 3) ? 1.f : 0.f);
    } else {
#pragma unroll 1
        for (uint32_t i = cx.lane; i < 2 * L.A; i += 32) row[i] = pack_bit(L, cx, i) ? 1.f : 0.f;
    }
}

#ifndef AZB_TREE_MIN_BLOCKS
#define AZB_TREE_MIN_BLOCKS 7
#endif
template <int DEPTH, bool COUNT, bool PUCT = false>  // PUCT: azb_config.selection == AZB_SELECT_PUCT
__global__ void __launch_bounds__(AZB_WARPS_PER_BLOCK * 32, AZB_TREE_MIN_BLOCKS)
    azb_tree_kernel(const AzbLayout L, const uint32_t flags, const uint32_t smem_words_per_warp, const uint32_t lcap,
                    const uint32_t target_step, const uint32_t max_episodes, const uint32_t tree0,
                    const uint32_t tree_end) {
    extern __shared__ __align__(16) uint32_t smem[];
    __shared__ uint32_t s_last;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t tree = tree0 + blockIdx.x * AZB_WARPS_PER_BLOCK + warp;
    uint8_t *lut = reinterpret_cast<uint8_t *>(smem + (size_t)AZB_WARPS_PER_BLOCK * smem_words_per_warp);
    tree_tables_fill(L, lut, threadIdx.x, blockDim.x);
    __syncthreads();
    uint32_t *base = smem + (size_t)warp * smem_words_per_warp;
    if (tree < tree_end) {
        WarpCtx cx;
        cx.full_count = COUNT;
        ctx_bind_smem(L, cx, base, lut, lane);
        (void)lcap;
        ctx_bind_tree(L, cx, tree);
        uint32_t *gw = L.walker + (size_t)tree * L.WS;
        PROF_T0();
        cx.ct[lane] = 0u;
#pragma unroll 4
        for (uint32_t i = lane; i < L.WS; i += 32) cx.wk[i] = gw[i];
        __syncwarp();
        PROF_ADD(cx, PH_LOAD);

        if (flags & AZB_F_INIT) {
            // tail of par_new / par_reset_trees (optimizer/mod.rs:62-101, 340-359): state <- root, root cost, root node
            walker_reset(L, cx);
            uint32_t mu = 0;
            const double l1 = azb_cost_warp<DEPTH>(L.N, cx.par, cx.cs, lane, &mu);
            if (!(l1 >= 1.4)) cx.err = 5;
            const float c0 = azb_evaluate(mu, l1, L.c_lower, L.slope);
            if (lane < 4) {
                uint4 q = make_uint4(0u, 0u, 0u, 0u);
                if (lane == 0) q = make_uint4(__float_as_uint(c0), __float_as_uint(c0), 0u, 0u);
                if (lane == 1) q = make_uint4(AZB_LO_NONE, 0u, 0u, 0u);
                cx.node[lane] = q;
            }
            if ((uint32_t)lane < L.W) cx.key[lane] = 0u;
            if constexpr (DEPTH == 5)
                if ((uint32_t)lane + 32 < L.W) cx.key[lane + 32] = 0u;
            const uint32_t hv = key_hash(0u, 0u, lane, L.W);  // the empty path hashes like every other key
            if (lane == 0) {
                hash_insert(cx.hash, hv & (L.cap_hash - 1), 0u, hv);
                cx.wk[WK_POS] = 0;
                cx.wk[WK_DEPTH] = 0;
                cx.wk[WK_NNODES] = 1;
                cx.wk[WK_NBLK] = AZB_BLK_PAD;
                cx.wk[WK_NARCS] = 0;
                cx.wk[WK_INTOP] = 0;
                cx.wk[WK_STEP] = 0;
                cx.wk[WK_PEND_C] = __float_as_uint(c0);
                cx.wk[WK_PKIDX] = AZB_LO_NONE;
                cx.wk[WK_NPREDS] = 0;
                cx.wk[WK_ROOTLO] = AZB_LO_NONE;
                cx.wk[WK_CURLO] = AZB_LO_NONE;
                cx.wk[WK_ERR] = 0;
                cx.wk[WK_PATH] = 0;
                cx.wk[WK_FLAGS] = 1u;
                if (flags & AZB_F_FIRST) {
                    // par_new: silent argmin over the roots (optimizer/mod.rs:95-101) = candidate slot 0
                    L.cand[tree] = make_uint2(azb_f2ord(c0), 0u);
                    cx.wk[WK_CAND_C] = 0xffffffffu;
                    cx.wk[WK_CAND_NODE] = 0u;
                } else {
                    // par_reset_trees zeroes num_inspected_nodes (optimizer/mod.rs:359): the new root is looked at by
                    // the first step's argmin scan; node 0 wins ties against later nodes
                    cx.wk[WK_CAND_C] = azb_f2ord(c0);
                    cx.wk[WK_CAND_NODE] = 0u;
                }
            }
            __syncwarp();
            build_cur_mask(L, cx);
            tree_pack(L, cx, tree);
        }
        // AZB_F_MULTI (counter-hash priors only: they are computed in add_actions, so a tree never waits for anybody): the
        // warp takes its tree all the way to target_step in this one launch — the lock step without its barrier
#pragma unroll 1
        for (;;) {
            if ((flags & AZB_F_ADD) && (cx.wk[WK_FLAGS] & 1u)) tree_add_actions<DEPTH == 5>(L, cx, tree);
            PROF_ADD(cx, PH_ADD);
            if ((flags & AZB_F_ROLLOUT) && cx.err == 0 && cx.wk[WK_STEP] < target_step && !(cx.wk[WK_FLAGS] & 1u)) {
                tree_rollout<DEPTH, PUCT>(L, cx, tree, max_episodes);
#ifdef AZB_PROFILE
                prof_t0 = clock64();
#endif
                // optimizer/mod.rs:171-173 (every step, also in a multi-step launch: a tree whose later steps are no-ops
                // keeps the vector of its last live step, exactly as in the lock step)
                if (cx.err == 0 && (cx.wk[WK_FLAGS] & 1u)) tree_pack(L, cx, tree);
                PROF_ADD(cx, PH_PACK);
            }
            if (!(flags & AZB_F_MULTI) || cx.err != 0 || cx.wk[WK_STEP] >= target_step) break;
        }
#ifdef AZB_PROFILE
        prof_t0 = clock64();
#endif
        __syncwarp();
        // publish: walker block (without the root part), counters, errors, distance to the target
        const uint32_t live_words = WK_HDR + L.PW + 2 * L.W;
#pragma unroll 1
        for (uint32_t i = lane; i < live_words; i += 32) gw[i] = cx.wk[i];
        if (lane < 16) {
            const uint32_t v = (COUNT || lane == CT_INS || lane == CT_LIVE || lane == CT_NOOP) ? cx.ct[lane] : 0u;
            if (v) atomicAdd(&L.g->counters.v[lane], (unsigned long long)v);
        }
        PROF_ADD(cx, PH_STORE);
#ifdef AZB_PROFILE
        __syncwarp();
        if (lane == 0 && tree < 65536u) {
            uint32_t tot = 0;
            for (int q = 16; q < 28; ++q) tot += cx.ct[q];
            g_tree_prof[tree] = make_uint4(tot, cx.ct[CT_RESET] + 1u, cx.ct[CT_INS], cx.ct[30]);
        }
        if (lane >= 16) {
            const uint32_t v = cx.ct[lane];
            if (v) atomicAdd(&L.g->prof[lane - 16], (unsigned long long)v);
        }
#endif
        if (max_episodes != 0u && lane == 0 && (flags & AZB_F_ROLLOUT) && cx.wk[WK_STEP] < target_step)
            atomicAdd(&L.g->behind_accum, 1u);
        const uint32_t e = __reduce_or_sync(0xffffffffu, cx.err);
        if (e && lane == 0) {
            if (atomicCAS(&L.g->err, 0u, e) == 0u) {
                L.g->err_tree = tree;
                L.g->err_step = cx.wk[WK_STEP];
            }
        }
    }
    // ---- last block done: publish how many trees still have to reach the target (bounded-episode launches only)
    if (max_episodes == 0u) return;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(&L.g->blocks_done, 1u) == gridDim.x - 1) ? 1u : 0u;
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        __threadfence();
        AzbGlobals *g = L.g;
        g->n_behind = *((volatile uint32_t *)&g->behind_accum);
        g->behind_accum = 0u;
        g->blocks_done = 0u;
        __threadfence();
    }
}

// ---- par_update_argmmim_data across trees and steps (optimizer/mod.rs:194-246) -----------------------------------
// pass 1: per candidate slot, the first minimum over trees (lowest tree index wins ties)
__global__ void __launch_bounds__(256) azb_stepmin_kernel(const AzbLayout L, const uint32_t slot_lo) {
    __shared__ unsigned long long red[8];
    const uint32_t slot = slot_lo + blockIdx.x;
    const uint2 *row = L.cand + (size_t)slot * L.B;
    unsigned long long m = ~0ull;
    for (uint32_t t = threadIdx.x; t < L.B; t += blockDim.x) {
        const unsigned long long k = ((unsigned long long)row[t].x << 32) | t;
        m = k < m ? k : m;
    }
    m = warp_min_u64(m);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < 8; ++i) m = red[i] < m ? red[i] : m;
        L.stepmin[slot] = m;
    }
}

// replay a node's action set on its tree's root (optimizer/mod.rs:224-239) into g->argmin_state; one warp
__device__ void finalize_argmin_state(const AzbLayout &L, uint32_t *scratch, const uint8_t *lut, uint32_t tree,
                                      uint32_t node, int lane) {
    WarpCtx cx;
    cx.lane = lane;
    cx.full_count = false;
    cx.lut = lut;
    cx.wk = scratch;
    cx.par = (uint8_t *)(scratch + WK_HDR);
    cx.perm = scratch + WK_HDR + L.PW;
    cx.keym = cx.perm + L.W;
    const uint32_t *src = L.walker + (size_t)tree * L.WS;
#pragma unroll 1
    for (uint32_t i = lane; i < L.PW; i += 32) ((uint32_t *)cx.par)[i] = src[WK_HDR + L.PW + 2 * L.W + i];
#pragma unroll 1
    for (uint32_t w = lane; w < L.W; w += 32) {
        cx.perm[w] = src[WK_HDR + 2 * L.PW + 2 * L.W + w];
        cx.keym[w] = 0u;
    }
    __syncwarp();
    const uint32_t *key = L.key + ((size_t)tree * L.cap_nodes + node) * L.W;
    for (uint32_t w = 0; w < L.W; ++w) {
        uint32_t word = key[w];
        while (word) {
            uint32_t b = __ffs(word) - 1;
            word &= word - 1;
            walker_act(L, cx, w * 32 + b);
        }
    }
#pragma unroll 1
    for (uint32_t i = lane; i < 16; i += 32) L.g->argmin_state[i] = i < L.PW ? ((uint32_t *)cx.par)[i] : 0u;
#pragma unroll 1
    for (uint32_t w = lane; w < 61; w += 32) L.g->argmin_state[16 + w] = w < L.W ? cx.perm[w] : 0u;
}

// pass 2: walk the slots in step order with the running best; log the improving steps; rebuild the argmin state.
// slot 0 holds the roots of par_new and is silent.
__global__ void __launch_bounds__(32) azb_argmin_kernel(const AzbLayout L, const uint32_t slot_lo, const uint32_t slot_hi) {
    __shared__ uint32_t scratch[WK_HDR + 16 + 2 * 61 + 8];
    __shared__ uint8_t lut[2048];
    const int lane = threadIdx.x;
#pragma unroll 1
    for (uint32_t a = lane; a < L.A; a += 32) lut[a] = (uint8_t)azb_action_child(a);
    __syncwarp();
    AzbGlobals *g = L.g;
    uint32_t best = g->best_c, n_imp = g->n_improved, last = 0, have = 0, tree = 0, node = 0;
    for (uint32_t s = slot_lo; s < slot_hi; ++s) {
        const unsigned long long m = L.stepmin[s];
        const uint32_t oc = (uint32_t)(m >> 32);
        last = 0;
        if (oc < best) {
            best = oc;
            tree = (uint32_t)m;
            node = L.cand[(size_t)s * L.B + tree].y;
            have = 1;
            if (s != 0u) {
                last = 1;
                if (lane == 0 && n_imp < L.log_cap) {
                    L.log[n_imp].step = s - 1u;
                    L.log[n_imp].tree = tree;
                    L.log[n_imp].node = node;
                    L.log[n_imp].eval = azb_ord2f(oc);
                }
                n_imp += 1;
            }
        }
    }
    if (have) finalize_argmin_state(L, scratch, lut, tree, node, lane);
    __syncwarp();
    if (lane == 0) {
        g->best_c = best;
        g->n_improved = n_imp;
        g->improved_last = last;
        g->next_slot = slot_hi;
        if (have) {
            g->argmin_tree = tree;
            g->argmin_node = node;
        }
    }
}

// both passes for ONE slot, the slot index read from device memory: the argmin step of the single-step CUDA graph
// (azb_step(h, 1, ...)), whose kernel arguments must not change from replay to replay.  Resets n_improved first
// (the log of an azb_step call starts empty).
__global__ void __launch_bounds__(256) azb_argmin1_kernel(const AzbLayout L) {
    __shared__ unsigned long long red[8];
    __shared__ uint32_t scratch[WK_HDR + 16 + 2 * 61 + 8];
    __shared__ uint8_t lut[2048];
    AzbGlobals *g = L.g;
    const uint32_t slot = g->next_slot;
    const uint2 *row = L.cand + (size_t)slot * L.B;
    unsigned long long m = ~0ull;
    for (uint32_t t = threadIdx.x; t < L.B; t += blockDim.x) {
        const unsigned long long k = ((unsigned long long)row[t].x << 32) | t;
        m = k < m ? k : m;
    }
    m = warp_min_u64(m);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    for (uint32_t a = threadIdx.x; a < L.A; a += blockDim.x) lut[a] = (uint8_t)azb_action_child(a);
    __syncthreads();
    if (threadIdx.x >= 32) return;
    const int lane = threadIdx.x;
    for (int i = 1; i < 8; ++i) m = red[i] < m ? red[i] : m;
    const uint32_t oc = (uint32_t)(m >> 32), tree = (uint32_t)m;
    uint32_t n_imp = 0, last = 0;
    const bool better = oc < g->best_c;
    uint32_t node = 0;
    if (better) {
        node = L.cand[(size_t)slot * L.B + tree].y;
        if (slot != 0u) {
            last = 1;
            if (lane == 0) {
                L.log[0].step = slot - 1u;
                L.log[0].tree = tree;
                L.log[0].node = node;
                L.log[0].eval = azb_ord2f(oc);
            }
            n_imp = 1;
        }
        finalize_argmin_state(L, scratch, lut, tree, node, lane);
    }
    __syncwarp();
    if (lane == 0) {
        L.stepmin[slot] = m;
        if (better) {
            g->best_c = oc;
            g->argmin_tree = tree;
            g->argmin_node = node;
        }
        g->n_improved = n_imp;
        g->improved_last = last;
        g->next_slot = slot + 1u;
    }
}

// write_observations (tree/mod.rs:242-264) for every tree, plus the root vectors par_update_model packs first
// (optimizer/mod.rs:253-259).  One warp per tree; h_sa = c*_as (04-c21-tree.rs:104).  The root's kid entries carry
// everything needed.
__global__ void __launch_bounds__(128) azb_observe_kernel(const AzbLayout L, const uint32_t n_obs_tol,
                                                          float *__restrict__ obs, float *__restrict__ wts,
                                                          float *__restrict__ root_vecs) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t tree = blockIdx.x * 4 + warp;
    if (tree >= L.B) return;
    float *o = obs + (size_t)tree * L.A, *w = wts + (size_t)tree * L.A;
#pragma unroll 1
    for (uint32_t a = lane; a < L.A; a += 32) {
        o[a] = 0.f;
        w[a] = 0.f;
    }
    __syncwarp();
    const uint32_t *wk = L.walker + (size_t)tree * L.WS;
    const uint32_t lo2 = wk[WK_ROOTLO];
    if (lo2 != AZB_LO_NONE) {
        const uint4 *blk4 = reinterpret_cast<const uint4 *>(L.blk + (size_t)tree * L.cap_blk);
        const uint32_t n_out = blk4[lo2].y & 0xffffu;
#pragma unroll 1
        for (uint32_t t = lane; t < n_out; t += 32) {
            const uint4 kd = blk4[lo2 + 1u + t];
            if (!(kd.y >> 31) || kd.z >= n_obs_tol) {
                const uint32_t a = kd.x >> 20;
                o[a] = __uint_as_float(kd.w);
                w[a] = 1.0f;
            }
        }
    }
    if (root_vecs) {
        const uint8_t *rpar = (const uint8_t *)(wk + WK_HDR + L.PW + 2 * L.W);
        const uint32_t *rperm = wk + WK_HDR + 2 * L.PW + 2 * L.W;
        float *row = root_vecs + (size_t)tree * L.sv_ld;
#pragma unroll 1
        for (uint32_t i = lane; i < 2 * L.A; i += 32) {
            bool one;
            if (i < L.A) {
                const uint32_t child = azb_action_child(i);
                one = (uint32_t)rpar[child] == i - azb_child_first_action(child);
            } else {
                one = (rperm[(i - L.A) >> 5] >> ((i - L.A) & 31)) & 1u;
            }
            row[i] = one ? 1.0f : 0.0f;
        }
    }
}

// ---- par_reset_trees' modify_root (optimizer/mod.rs:284-339) with the example's policy (04-c21-tree.rs:172-206) ----
// One warp per tree, once per epoch.  n[0] is the root (the empty ActionSet is the smallest BTreeMap key):
//   c_root == c*_root (nothing better was found below this root):
//       |permitted| == k_max : a fresh random state (ROTWithActionPermissions::generate, k ~ U{k_min..k_max})
//       otherwise            : move to a uniformly chosen node with c == c_root, k ~ U{|permitted|..k_max}
//   else                     : move to a uniformly chosen node with c <= (c_root + 3 c*_root) / 4, k ~ U{k_min..k_max}
//   and in both "move" cases re-draw the permitted set (randomize_permitted_actions, modify_parent_once.rs:27-37).
// The reference draws from an unseeded thread_rng, so only the distribution is defined; here the draws come from a
// counter generator keyed by (seed, epoch, GLOBAL root index) — the same stream the oracle uses — and candidates
// are enumerated in node-index order (any fixed order gives the same uniform choice).
__device__ __forceinline__ uint32_t azb_bounded(unsigned long long r, uint32_t n) {
    return (uint32_t)(((r >> 32) * (unsigned long long)n) >> 32);
}

__global__ void __launch_bounds__(128) azb_modify_roots_kernel(const AzbLayout L, const unsigned long long seed,
                                                               const unsigned long long epoch, const uint32_t k_min,
                                                               const uint32_t k_max) {
    __shared__ uint16_t s_perm[4][2048];
    __shared__ uint32_t s_mask[4][64];
    __shared__ uint8_t s_par[4][64];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t tree = blockIdx.x * 4 + warp;
    if (tree >= L.B) return;
    const uint32_t FULL = 0xffffffffu;
    uint32_t *wk = L.walker + (size_t)tree * L.WS;
    uint32_t *g_rpar = wk + WK_HDR + L.PW + 2 * L.W, *g_rperm = g_rpar + L.PW;
    uint16_t *perm = s_perm[warp];
    uint32_t *mask = s_mask[warp];
    uint8_t *par = s_par[warp];
#pragma unroll 1
    for (uint32_t i = lane; i < L.PW; i += 32) reinterpret_cast<uint32_t *>(par)[i] = g_rpar[i];
    uint32_t kcur = 0;
#pragma unroll 1
    for (uint32_t w = lane; w < L.W; w += 32) kcur += __popc(g_rperm[w]);
    kcur = warp_sum_u32(kcur);
    __syncwarp();
    const uint4 *node = L.node + (size_t)tree * L.cap_nodes * 4;
    const uint32_t nn = wk[WK_NNODES];
    const uint4 r0 = node[0];
    const float c_root = __uint_as_float(r0.x), c_star = __uint_as_float(r0.y);
    unsigned long long s = azb_mix64(seed ^ azb_mix64(L.first_root + tree + 0x5851F42D4C957F2Dull) ^
                                     azb_mix64(epoch * 0xA24BAED4963EE407ull + 0x9FB21C651E98DF25ull));
    unsigned long long ctr = 0;
    auto next = [&]() { return azb_mix64(s + (ctr++) * 0xD1342543DE82EF95ull); };  // every lane keeps the same stream
    const bool stuck = c_root == c_star;
    uint32_t num = 0;
    uint32_t err = 0;
    if (stuck && kcur == k_max) {
        num = k_min + azb_bounded(next(), k_max - k_min + 1);
        if (lane == 0) {  // RootedOrderedTree::generate (rooted_tree/mod.rs:14-20)
            for (uint32_t i = 0; i < L.N; ++i) par[i] = 0;
        }
        __syncwarp();
        for (uint32_t i = 2; i + 1 < L.N; ++i) {
            const uint32_t p = azb_bounded(next(), i);
            if (lane == 0) par[i] = (uint8_t)p;
        }
    } else {
        if (stuck && (kcur < k_min || kcur > k_max)) err = 6;  // the reference's unreachable!() (04-c21-tree.rs:179)
        const float thr = __fdiv_rn(__fadd_rn(c_root, __fmul_rn(3.0f, c_star)), 4.0f);
        // candidates in node order: count, draw, locate
        uint32_t count = 0;
        for (uint32_t base = 0; base < nn; base += 32) {
            const uint32_t i = base + lane;
            bool cand = false;
            if (i < nn) {
                const float c = __uint_as_float(node[(size_t)i * 4].x);
                cand = stuck ? (c == c_root) : (c <= thr);
            }
            count += __popc(__ballot_sync(FULL, cand));
        }
        uint32_t chosen = 0;
        if (count == 0) {
            err = 6;  // n.choose(..).unwrap() on an empty list panics in the reference
        } else {
            const uint32_t r = azb_bounded(next(), count);
            uint32_t seen = 0;
            for (uint32_t base = 0; base < nn; base += 32) {
                const uint32_t i = base + lane;
                bool cand = false;
                if (i < nn) {
                    const float c = __uint_as_float(node[(size_t)i * 4].x);
                    cand = stuck ? (c == c_root) : (c <= thr);
                }
                const uint32_t bal = __ballot_sync(FULL, cand);
                const uint32_t here = __popc(bal);
                if (r < seen + here) {
                    chosen = base + nth_set_bit(bal, r - seen);
                    break;
                }
                seen += here;
            }
            // p.actions_taken().for_each(|a| space.act(state, a)): only the parents survive the re-draw below
            const uint32_t *key = L.key + ((size_t)tree * L.cap_nodes + chosen) * L.W;
#pragma unroll 1
            for (uint32_t w = lane; w < L.W; w += 32) {
                uint32_t word = key[w];
                while (word) {
                    const uint32_t a = w * 32 + (__ffs(word) - 1);
                    word &= word - 1;
                    const uint32_t child = azb_action_child(a);
                    par[child] = (uint8_t)(a - azb_child_first_action(child));  // distinct children: no race
                }
            }
        }
        num = stuck ? kcur + azb_bounded(next(), k_max - kcur + 1) : k_min + azb_bounded(next(), k_max - k_min + 1);
    }
    __syncwarp();
    // choose_multiple(rng, num) over 0..A as a partial Fisher-Yates (the host generator's algorithm)
#pragma unroll 1
    for (uint32_t i = lane; i < L.A; i += 32) perm[i] = (uint16_t)i;
#pragma unroll 1
    for (uint32_t w = lane; w < 64; w += 32) mask[w] = 0u;
    __syncwarp();
    if (err == 0) {
        for (uint32_t t = 0; t < num; ++t) {
            const uint32_t j = t + azb_bounded(next(), L.A - t);
            if (lane == 0) {
                const uint16_t pt = perm[t], pj = perm[j];
                perm[t] = pj;
                perm[j] = pt;
                mask[pj >> 5] |= 1u << (pj & 31);
            }
        }
        __syncwarp();
#pragma unroll 1
        for (uint32_t i = lane; i < L.PW; i += 32) g_rpar[i] = reinterpret_cast<uint32_t *>(par)[i];
#pragma unroll 1
        for (uint32_t w = lane; w < L.W; w += 32) g_rperm[w] = mask[w];
    } else if (lane == 0) {
        if (atomicCAS(&L.g->err, 0u, err) == 0u) {
            L.g->err_tree = tree;
            L.g->err_step = wk[WK_STEP];
        }
    }
}
