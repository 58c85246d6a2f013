// azb_common.cuh — device-side layout and helpers shared by every kernel.
//
// HBM layout (one slab per array, per tree contiguous; DESIGN.md §3):
//   walker [B][WS]  u32   persistent walker + root state (optimizer/mod.rs:9-14)
//   node   [B][cap_nodes] 64 B records = StateWeight (tree/state_weight.rs:4-10) + the first four in-arcs inline
//   blk    [B][cap_blk]   8 B units: one BLOCK per expanded node, laid out around its header so that one
//                         speculative, coalesced read fetches everything selection needs:
//                             [pred cnt-1 .. pred 0][header 16 B][kid 0 .. kid cnt-1]
//                         pred (8 B)  = ActionPrediction {g, a_id | has_arc | arc seq}   (tree/arc_weight.rs:11-16)
//                         kid  (16 B) = one out-arc in creation order, carrying a COPY of what revisit_choice and
//                                       the next descent step need from the child: {child | a_id, child block |
//                                       active, n_t, c*}.  Cascades keep the copies coherent through the in-arc
//                                       entries (parent, kid slot).
//   inl    [B][cap_in]    8 B  in-arcs beyond the fourth of a node ((depth-4)+ slots reserved at creation)
//   key    [B][cap_nodes][W]   ActionSet bit mask of the node (path/set.rs:5-8)
//   hash   [B][cap_hash]  u32  open-addressing transposition table: (node index + 1) | fingerprint << 21
//   casc   [B][2][cap_nodes] u32  continuation of the cascade's work lists beyond their shared-memory part
//   cand   [cap_steps+1][B] 8 B  per-step argmin candidate of every tree (slot 0 = the roots)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define AZB_WARPS_PER_BLOCK 4
#define AZB_FRONTIER_CAP 128
#define AZB_BLK_PAD 64          // units kept free in front of a tree's block arena (speculative reads)
#define AZB_LO_NONE 0x7fffffffu

// walker block word offsets
enum {
    WK_POS = 0,
    WK_DEPTH = 1,
    WK_NNODES = 2,
    WK_NBLK = 3,       // bump pointer of the block arena, in 8-byte units
    WK_NARCS = 4,
    WK_INTOP = 5,      // bump pointer of the overflow in-arc arena
    WK_FLAGS = 6,      // bit0: node `pos` awaits add_actions; bit1: root not yet seen by the argmin scan
    WK_STEP = 7,       // completed steps since init_trees
    WK_CAND_C = 8,     // first-minimum candidate of the running step: orderable c bits
    WK_CAND_NODE = 9,
    WK_PEND_C = 10,    // c of the node awaiting add_actions
    WK_PKIDX = 11,     // 16-byte index of that node's kid entry in its creator's block (AZB_LO_NONE for a root)
    WK_NPREDS = 12,    // predictions appended so far
    WK_ROOTLO = 13,    // 16-byte index of the root's block header (AZB_LO_NONE while it has none)
    WK_CURLO = 14,     // same for the walker's node
    WK_ERR = 15,
    WK_PATH = 16,      // node ids of the walker's path, root first: path[d] = node at depth d (64 words)
    WK_HDR = 80        // the state part (parents, masks, root) starts here
};

struct AzbCounters {
    unsigned long long v[16];
};
enum {
    CT_SEL = 0, CT_DSEL, CT_CUR, CT_CAND, CT_PROBE, CT_INS, CT_TERM, CT_HIT, CT_ARC, CT_PRED, CT_CN, CT_DCN, CT_RESET,
    CT_LIVE, CT_NOOP, CT_VISIT
};

struct AzbImprovementDev {
    uint32_t step, tree, node;
    float eval;
};

struct AzbGlobals {  // one per handle, in device memory
    uint32_t best_c;                // orderable bits of ArgminData.eval
    uint32_t blocks_done;           // last-block-done ticket
    uint32_t n_improved;            // improvements logged since the last azb_step call began
    uint32_t err;                   // first error code seen
    uint32_t err_tree;
    uint32_t err_step;
    uint32_t improved_last;         // 1 if the newest step of the last argmin pass improved
    uint32_t behind_accum;          // trees below the step target, accumulated by the running launch
    uint32_t n_behind;              // ... of the last finished launch
    uint32_t argmin_tree, argmin_node;
    uint32_t next_slot;             // first candidate slot the argmin pass has not consumed (device copy; single-step graph)
    uint32_t casc_spills;           // cascade waves that outgrew the shared-memory work list (diagnostic)
    uint32_t argmin_state[16 + 61]; // parents packed (16 words) + permitted (61 words)
    AzbCounters counters;
    unsigned long long prof[16];    // -DAZB_PROFILE: lane-0 cycles per phase
};

struct AzbLayout {
    uint32_t N, A, W, B, PW, WS;
    uint32_t cap_nodes, cap_blk, cap_in, cap_hash, cap_steps;
    uint32_t sv_ld, h_ld;
    float c_lower, slope;
    uint32_t tol[8];
    uint32_t tol_len, tol_default;
    uint32_t selection;   // AZB_SELECT_*: 0 = next_action, 1 = PUCT (the kernels' PUCT instantiations)
    float puct_c;
    uint32_t prior_mode, log_cap;
    uint32_t frontier_cap;  // entries of a cascade work list kept in shared memory (<= AZB_FRONTIER_CAP)
    unsigned long long first_root, prior_seed;
    const uint8_t *lut;   // child vertex of every action (A bytes, padded to a multiple of 4)
    uint32_t *walker;
    uint4 *node;
    uint2 *blk;
    uint2 *inl;
    uint32_t *key;
    uint32_t *hash;
    uint32_t *casc;       // [B][2][cap_nodes] continuation of the cascade's shared-memory work lists (rarely touched)
    uint2 *cand;
    unsigned long long *stepmin;
    float *sv;
    uint16_t *sv16;       // bf16 rows for the tensor-core MLP (null otherwise): write_vec goes there instead of sv
    uint32_t sv16_ld;
    float *h;
    AzbGlobals *g;
    AzbImprovementDev *log;
};

// ---------------------------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ unsigned long long azb_mix64(unsigned long long z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// counter-hash prior in [0,1): SURVEY.md §8d "injected priors from the same counter-based generator"
__host__ __device__ __forceinline__ float azb_hash_prior(unsigned long long seed, unsigned long long root,
                                                         unsigned long long step, uint32_t a) {
    unsigned long long r = azb_mix64(azb_mix64(seed ^ 0xA0761D6478BD642Full) + root * 0x9E3779B97F4A7C15ull +
                                     step * 0xE7037ED1A0B428DBull + (unsigned long long)a * 0x8EBC6AF09C88C6E3ull);
    return (float)(r >> 40) * 5.9604644775390625e-08f;
}

// order-preserving map f32 -> u32 (all finite values)
__host__ __device__ __forceinline__ uint32_t azb_f2ord(float f) {
#ifdef __CUDA_ARCH__
    uint32_t u = __float_as_uint(f);
#else
    uint32_t u;
    memcpy(&u, &f, 4);
#endif
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float azb_ord2f(uint32_t o) {
    uint32_t u = (o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o;
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    float f;
    memcpy(&f, &u, 4);
    return f;
#endif
}

// A.1 indexing (simple_graph/edge.rs:48-65, rooted_tree/ordered_edge.rs:35-42): action a <-> edge at colex
// position a+1; the actions of child v are the contiguous range [v(v-1)/2 - 1, v(v-1)/2 + v - 2].
__host__ __device__ __forceinline__ uint32_t azb_child_first_action(uint32_t v) { return v * (v - 1) / 2 - 1; }
// Block-shared lookup tables of the tree kernels, behind the per-warp regions: the child vertex of every action (A bytes,
// padded to 16) and — while a mask word per lane suffices (W <= 32) — for every child vertex the W-word mask of ITS actions
// (what `act` clears from the permitted set): N rows of 8 (W <= 8) or W words
__host__ __device__ __forceinline__ uint32_t azb_lut_bytes(uint32_t A) { return (A + 15u) & ~15u; }
// (rows of 8 words up to N = 22 — a shift on the walkers' path —, of W words beyond)
__host__ __device__ __forceinline__ uint32_t azb_amask_stride(uint32_t W) { return W <= 8u ? 8u : W; }
__host__ __device__ __forceinline__ uint32_t azb_amask_bytes(uint32_t N, uint32_t W) { return W <= 32u ? ((N * azb_amask_stride(W) * 4u + 15u) & ~15u) : 0u; }
__host__ __device__ __forceinline__ uint32_t azb_tables_bytes(uint32_t A, uint32_t N, uint32_t W) {
    return azb_lut_bytes(A) + azb_amask_bytes(N, W);
}
__host__ __device__ __forceinline__ uint32_t azb_action_index(uint32_t parent, uint32_t child) {
    return child * (child - 1) / 2 + parent - 1;
}
// closed form of the reference's linear search: largest v with v(v-1)/2 <= a+1
__host__ __device__ __forceinline__ uint32_t azb_action_child(uint32_t a) {
    uint32_t pos = a + 1;
    uint32_t v = (uint32_t)((1.0f + sqrtf(8.0f * (float)pos + 1.0f)) * 0.5f);
    while (v * (v - 1) / 2 > pos) --v;
    while ((v + 1) * v / 2 <= pos) ++v;
    return v;
}

#ifdef __CUDACC__
__device__ __forceinline__ unsigned long long shfl_u64(unsigned long long v, int src) {
    uint32_t lo = (uint32_t)v, hi = (uint32_t)(v >> 32);
    lo = __shfl_sync(0xffffffffu, lo, src);
    hi = __shfl_sync(0xffffffffu, hi, src);
    return ((unsigned long long)hi << 32) | lo;
}
__device__ __forceinline__ unsigned long long shfl_xor_u64(unsigned long long v, int m) {
    uint32_t lo = (uint32_t)v, hi = (uint32_t)(v >> 32);
    lo = __shfl_xor_sync(0xffffffffu, lo, m);
    hi = __shfl_xor_sync(0xffffffffu, hi, m);
    return ((unsigned long long)hi << 32) | lo;
}
__device__ __forceinline__ unsigned long long warp_min_u64(unsigned long long v) {
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
        unsigned long long o = shfl_xor_u64(v, m);
        v = o < v ? o : v;
    }
    return v;
}
__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long v) {
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
        unsigned long long o = shfl_xor_u64(v, m);
        v = o > v ? o : v;
    }
    return v;
}
__device__ __forceinline__ uint32_t warp_sum_u32(uint32_t v) {
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
    return v;
}
#endif
