// azb_async.cuh — the asynchronous form of the batched search step: ONE persistent, cooperative kernel in which
// trees never wait for each other.
//
// The reference's step (NablaOptimizer::par_roll_out_episodes, az-discrete-opt/src/nabla/optimizer/mod.rs:121-191) is
// a barrier: every tree walks until it has one new node, then ONE model call answers all of them.  Trees are
// independent (each rayon task touches only its own row, :159-189), so the barrier is an artefact of batching the
// model call, and it costs the GPU dearly: a launch lasts as long as its slowest tree (7-12 episodes) while the
// average tree needs 1.9 (profiles/README.md).  Here every CTA of ONE cooperative launch (one CTA per SM, all
// co-resident by construction, so the waits below cannot deadlock) takes one of two roles:
//   * TREE CTA (32 warps at the kernel's 64 registers).  A warp owns a fixed set of trees (tree = warp + k * n_warps).
//     It advances whichever of its trees has its priors, packs the new state vector into the next free row of a ring
//     of 128-row tiles, and moves on; it polls a per-tree flag for the answer.  Ownership is static, so a tree's arena
//     is only ever touched through one SM's L1; the priors, written by other SMs, are read with ld.cg behind one
//     acquire load of the flag.
//   * MODEL CTA (the first CTA to arrive on each of `n_workers` SMs).  Its eight warpgroups re-divide the CTA's
//     registers with setmaxnreg: warpgroup 0 (TMA producer warp + tcgen05.mma issuer warp) shrinks to 56, warpgroups
//     1-2 (eight epilogue warps) grow to 168 — four 16-column TMEM slices in flight per warp without spilling —, and
//     warpgroups 3-7 shrink to 24 and leave.  A worker takes the next full tile and runs the four Linear layers on
//     the tensor cores in passes of two 128-column blocks (per 64-deep k-block one activation tile and two weight
//     tiles, issued as ONE N = 256 MMA per k-step; the 512 TMEM columns hold two passes, so the epilogue of one pass
//     overlaps the MMAs of the next), hidden activations of width <= 512 stay in tensor memory as the next layer's A
//     operand (single worker, bf16) and the others round-trip through an L2-resident scratch, the Sigmoid head scatters f32 rows to the owning trees' prior rows
//     and the last writer raises their flags.  A tile that stays partial for `flush_ns` is topped up with dummy rows
//     and run anyway (tail of the run, tiny batches).
// Results are identical to the lock-step path: a tree's walk depends only on its own priors, and a row's forward
// pass does not depend on which tile it rides in (same K order per dot product).  Per-tree step clocks and the
// cand[step][tree] table (DESIGN.md §4.1) make the argmin pass indifferent to the interleaving.
// Every spin loop has a watchdog on %globaltimer; on expiry the kernel sets `abort` and drains.
//
// Round 1 also had a two-kernel form (tree kernel + model kernel on two streams, spinning on each other) and a
// weight-stationary model pipeline kernel.  Both are gone: separately launched kernels that wait for each other are
// not guaranteed to run at the same time (B200_PROFILING.md), and they hung under anything that serialises kernels.
#pragma once
#include "azb_mlp_tc.cuh"
#include "azb_tree.cuh"

#define AS_THREADS 1024
#define AS_WARPS 32
#define AS_EPI_WARPS 8   // two per TMEM lane quadrant, each taking AS_EPI_COLS columns of a 128-column block
#define AS_EPI_WARP0 4   // first epilogue warp: warpgroups 1 and 2 of a model CTA
#define AS_EPI_COLS (128 / (AS_EPI_WARPS / 4))      // 64
#define AS_EPI_SLICES (AS_EPI_COLS / 16)            // 16-column TMEM slices per warp and block
#define AS_EPI_CHUNKS (AS_EPI_COLS / 8)             // 16-byte chunks per staged row
#define AS_EPI_STG_BYTES (32 * AS_EPI_COLS * 2)     // staging tile per warp: [32 rows x AS_EPI_COLS bf16]
#define AS_MLP_THREADS ((2 + AS_EPI_WARPS) * 32)    // threads that meet at the model CTA's named barrier 1
// register budgets of a model CTA's warpgroups (setmaxnreg; 128 x (56 + 2 x 168 + 5 x 24) = 65 536 = 1024 x 64)
#define AS_REGS_FRONT 56
#define AS_REGS_EPI 168
#define AS_REGS_IDLE 24
#define AS_WIDE_TREE_WARPS 16   // tree warps per CTA for N >= 47 (DEPTH == 5)
#define AS_REGS_WIDE_TREE 104   // their register budget
#ifndef AS_STAGES
#define AS_STAGES 3
#endif
#define AS_ACC 2          // 128-column blocks per pass (one N = 256 MMA per k-step).  The 512 TMEM columns hold TWO passes:
                          // the epilogue drains one while the MMAs of the next run (4-block passes filled TMEM and
                          // serialised the two: MMA 24 us + epilogue 25 us per tile)
#define AS_SWEEP_GAP 1000u  // cycles between two sweeps of a tree CTA's answer flags (steal)
// a warp whose own trees all wait for their priors (no steal): AS_NAP_COUNT sleeps of AS_NAP_LONG_NS, then AS_NAP_SHORT_NS
// between polls; a warp without the sweep token (steal) naps AS_NAP_LONG_NS
#define AS_NAP_COUNT 6u
#define AS_NAP_LONG_NS 5000u
#define AS_NAP_SHORT_NS 1000u
#define AS_TILE 128
#define AS_NONE 0xffffffffu
#define AS_MAX_GROUPS 128
// cycle counters of the workers (tools/async_probe.py): only in the -DAZB_PROFILE flavour
#ifdef AZB_PROFILE
#define AS_CLK() clock64()
#else
#define AS_CLK() 0ll
#endif

struct AzbAsyncState {  // device memory, zeroed before every launch
    uint32_t abort;       // 1 watchdog, 2 tree error.  Polled by every waiting warp: alone in its 128-byte line, away
    uint32_t pad0[31];    // from the counters the atomics below keep invalidating
    uint32_t sm_flag[1024];  // first CTA to arrive on each SM (indexed by %smid)
    uint32_t mlp_claims, tree_claims;
    uint32_t row_tail;    // ring slots handed out
    uint32_t tile_head;   // tile tickets handed to MLP workers
    uint32_t tiles_done;
    uint32_t done_trees;
    uint32_t rows_real, rows_dummy;
    // worker groups: the leader's tile mailbox and the group's monotonic barriers, one 128-byte line per group (the
    // members of a group spin on their own line only)
    struct Group {
        uint32_t seq, tile, done, pad0;
        uint32_t layer[4];
        uint32_t pad1[24];
    } grp[AS_MAX_GROUPS];
};

struct AzbAsyncMaps {
    CUtensorMap ring;    // layer-0 input: [NT*128 rows][kpad0] bf16
    CUtensorMap act[3];  // hidden activations of the workers: [n_workers*128 rows][kpad[l+1]]
    CUtensorMap w[4];    // weights [rows padded to 128][kpad[l]], box 64 x 128
    CUtensorMap ws[4];   // the same weights with a box of 64 x cw[l]: one member's column slice (shared-SM form)
};

struct AzbAsyncParams {
    AzbAsyncState *st;
    uint32_t *tile_count;  // [NT] rows published into the tile, summed over its generations
    uint32_t *slot_tree;   // [NT*128] owner of every ring row (AS_NONE = dummy)
    uint32_t *tile_retired;  // [NT] generations of this ring tile the workers have finished
    uint32_t *h_flag;      // [B] rows of this tree the model has answered since the launch began
    uint16_t *ring;        // [NT*128][kpad0]
    __nv_bfloat16 *act[3];
    const float *bias[4];
    uint32_t kpad[4], npad[4];
    uint32_t wide;           // 1: bf16 operands; 2: bf16x3 (AZB_MLP_TC3) — rows hold [hi(kpad) | lo(kpad)], three k-segments
    uint32_t NT, n_workers, group, target_step, smem_words_per_warp, ring_ld;  // group = worker SMs per tile
    uint32_t tree_warps;     // tree warps per CTA (32 unless the per-warp shared memory of a large N does not fit)
    uint32_t tab_slots;      // entries of a tree CTA's scheduling table: the most trees any CTA owns
    uint32_t steal;          // 1: a free warp advances ANY runnable tree of its CTA (more trees than warps); 0: only its own
                             // (and hands the state vector to the model from inside the walk, before the cost evaluation)
    uint32_t shared_sm;      // 1: shared-SM form — every CTA walks trees with 28 warps and serves the model with its last warpgroup
    uint32_t sh_stages;      // shared-SM form: stages of a member's operand ring
    uint32_t cw[4];          // shared-SM form: output columns of layer l per group member (a multiple of 16, <= 256)
    unsigned long long timeout_ns, flush_ns;
    unsigned long long *dbg;  // optional [32] cycle counters of the workers (azb_debug_async, tools/async_probe.py); null = off
};

__device__ __forceinline__ unsigned long long as_now() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// Polls use ld.volatile (served by L2, where the atomics land), never ld.acquire.gpu: an acquire load comes with
// CCTL.IVALL — it invalidates the SM's whole L1 — and a waiting warp polls every microsecond beside 31 warps whose
// walks live on L1 hits (ncu: 160 M CCTL per 100 steps; phase cycles of the walkers 1.6-2x the lock step's).  Once a
// poll has seen its value, ONE as_ld_acquire of the same word orders what follows (PTX memory model: what the word
// guards is read or overwritten afterwards).
__device__ __forceinline__ uint32_t as_ld_volatile(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t as_ld_acquire(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// increment with release semantics at GPU scope (MEMBAR.ALL.GPU + RED: no L1 invalidation, unlike a full fence)
__device__ __forceinline__ void as_red_release_add(uint32_t *p, uint32_t v) {
    asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void as_mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc_smem_u32(bar)) : "memory");
}
// spin on test_wait (no suspend): the worker owns its SM, and try_wait's suspend/wake-up costs more than the
// wait itself at this granularity (one barrier round trip per 64-deep k-block)
__device__ __forceinline__ void as_mbar_spin(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(tc_smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void as_named_bar(uint32_t id, uint32_t threads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}
// TMA load with an L2 eviction-priority hint: the 2.5 MB of weights are re-read by every tile while gigabytes of tree
// arenas stream through the same L2, so the weight tiles are loaded evict_last
__device__ __forceinline__ uint64_t as_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void as_tma_load_2d_hint(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(
            tc_smem_u32(dst)),
        "l"(map), "r"(tc_smem_u32(bar)), "r"(c0), "r"(c1), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void as_tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void as_tmem_ld16_issue(uint32_t taddr, uint32_t (&r)[16]) {  // no wait: batch several, then wait::ld
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
// explicit shared-space accesses: the workers' shared memory arrives as a generic pointer, and ptxas then emits generic
// LD.E / ST.E for the biases and the staging tile
__device__ __forceinline__ uint4 as_lds128(uint32_t saddr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr));
    return v;
}
__device__ __forceinline__ void as_sts128(uint32_t saddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void as_fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void as_tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
        "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
        "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
// D (+)= A B^T with the A operand [128 x 16] in tensor memory (row = lane, two bf16 per column) and B in shared memory
__device__ __forceinline__ void as_umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// bias + ReLU of one 16-column TMEM slice, as eight bf16 pairs (half 1, bf16x3 only: what bf16 lost, itself rounded to bf16)
__device__ __forceinline__ void as_relu_pack(const uint32_t (&r)[16], uint32_t bias_s, uint32_t half, uint32_t *pk) {
#pragma unroll
    for (int t = 0; t < 8; t += 2) {
        const uint4 b4 = as_lds128(bias_s + 2u * t * 4u);
        float v0 = __uint_as_float(r[2 * t]) + __uint_as_float(b4.x);
        float v1 = __uint_as_float(r[2 * t + 1]) + __uint_as_float(b4.y);
        float v2 = __uint_as_float(r[2 * t + 2]) + __uint_as_float(b4.z);
        float v3 = __uint_as_float(r[2 * t + 3]) + __uint_as_float(b4.w);
        v0 = fmaxf(v0, 0.f);
        v1 = fmaxf(v1, 0.f);
        v2 = fmaxf(v2, 0.f);
        v3 = fmaxf(v3, 0.f);
        __nv_bfloat162 h01 = __floats2bfloat162_rn(v0, v1), h23 = __floats2bfloat162_rn(v2, v3);
        if (half) {
            h01 = __floats2bfloat162_rn(v0 - __low2float(h01), v1 - __high2float(h01));
            h23 = __floats2bfloat162_rn(v2 - __low2float(h23), v3 - __high2float(h23));
        }
        pk[t] = *reinterpret_cast<uint32_t *>(&h01);
        pk[t + 1] = *reinterpret_cast<uint32_t *>(&h23);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Model CTA.  Roles: warp 0 TMA producer and tile taker, warp 1 MMA issuer and TMEM owner (warpgroup 0, 56 registers),
// warps 4-11 epilogue (warpgroups 1-2, 168 registers).  Each role is its own function with its own copy of the loop
// over tiles, so that no code is shared between register budgets; they meet at named barrier 1 (AS_MLP_THREADS).
//
// Hidden layers in tensor memory.  A single worker (G = 1) with bf16 operands keeps a hidden layer of width <= 512 on
// chip: the epilogue packs it to bf16 pairs into TMEM columns [0, width / 2) (row = lane), and the next layer's MMAs read
// their A operand from there (tcgen05.mma with A in TMEM) while only weight tiles stream through the operand ring.  That
// saves the activation tile the layer would reload once per pass and the L2 round trip with its fences.  TMEM plan of a
// tile (as_a_in_tmem, as_acc_col):
//   * a layer whose input comes through shared memory runs passes of AS_ACC blocks, pass p in [256 (p & 1), + 256);
//     when it produces a TMEM hidden layer (npad <= 512, so at most two passes), pass p's epilogue writes its packed
//     columns to [128 p, 128 p + 128): in place for p = 0, over pass 0's accumulator for p = 1.  The two epilogue warps
//     of a TMEM lane quadrant meet at a pair barrier before every packed store, so neither overwrites columns the other
//     has not read yet;
//   * a layer whose input is in TMEM keeps its accumulators in [256, 512): one pass of up to AS_ACC blocks, or
//     128-column passes double-buffered in [256, 384) / [384, 512).  Its MMAs start behind h_bar, which the epilogue
//     arrives at once the whole hidden layer is stored (tcgen05.wait::st, fence, arrive) — and so once every pass of the
//     previous layer is drained.  Its own output cannot go to TMEM (it would overwrite the input its later passes read),
//     so layers alternate and a layer after a TMEM-input layer takes its input from the L2 scratch, behind layer_bar:
//     that chain also orders the MMAs that read a hidden layer before the MMAs that reuse its columns.
// G > 1 (a layer is split over SMs) and bf16x3 (hi and lo halves do not fit) keep every hand-over in L2.
struct AsWorkerShared {
    uint64_t full_bar[AS_STAGES], empty_bar[AS_STAGES], acc_full[2], acc_empty[2], layer_bar, h_bar;
    uint32_t tmem_slot, tile, epi_last;
    uint32_t bias_off[4];  // first entry of layer l's biases in the shared-memory copy
    uint32_t rowtree[AS_TILE];
};

// A GROUP of G worker SMs answers one tile together: member m computes the 128-column blocks nt = m, m + G, ... of
// every layer (a 1/G share of the weights streams through each SM's shared memory, which is what bounds a 128-row
// tile), the hidden activations meet in the group's L2-resident scratch, and the members synchronise at the three
// layer boundaries through monotonic counters in global memory.  The leader (m = 0) takes the tile.
struct AsWorkerId {
    uint32_t G, grp, mem;
};
__device__ __forceinline__ uint32_t as_blocks_of_member(uint32_t npad, const AsWorkerId &id) {
    const uint32_t n_tiles = (npad + 127u) / 128u;
    return n_tiles > id.mem ? (n_tiles - id.mem + id.G - 1u) / id.G : 0u;
}
#define AS_TILE_BYTES (AS_TILE * TC_BK * 2u)              // one 128 x 64 bf16 operand tile, 16 KB
#define AS_STAGE_BYTES ((1u + AS_ACC) * AS_TILE_BYTES)    // [A | B0 | B1]; weight-only stages (A in TMEM): up to three B tiles

// Layer l reads its A operand from TMEM (see "Hidden layers in tensor memory" above): a single worker, bf16 operands, an
// input of at most 512 columns (256 packed), and layer l - 1 did not itself read from TMEM
__device__ __forceinline__ bool as_a_in_tmem(const AzbAsyncParams &P, const uint32_t l) {
    bool in = false;  // layer 0 reads the ring
    for (uint32_t j = 1; j <= l; ++j) in = P.group == 1u && P.wide == 1u && P.kpad[j] <= 512u && !in;
    return in;
}
// 128-column blocks per pass: 128-column passes when the input is in TMEM and the layer does not fit one pass
__device__ __forceinline__ uint32_t as_pass_blocks(const bool a_tmem, const uint32_t mine) { return a_tmem && mine > AS_ACC ? 1u : AS_ACC; }
// first TMEM column of pass p's accumulator
__device__ __forceinline__ uint32_t as_acc_col(const bool a_tmem, const uint32_t p) { return a_tmem ? 256u + (p & 1u) * 128u : (p & 1u) * 256u; }

// Lane 0 of a group's first warp: the tile the group answers next (AS_NONE: leave).  The leader (member 0) waits until
// every member has finished the previous tile (its scratch is reused), takes the next ticket, waits until that tile is
// full — topping a stale partial tile up with dummy rows after flush_ns —, and posts it to the group's mailbox; the other
// members wait for the mailbox (member_nap_ns > 0: with a nanosleep between polls, for members that share their SM with
// walking trees).
__device__ __forceinline__ uint32_t as_group_next_tile(const AzbLayout &L, const AzbAsyncParams &P, const AsWorkerId id, const uint32_t seq,
                                                       const unsigned long long t_start, const uint32_t member_nap_ns) {
    AzbAsyncState *st = P.st;
    const uint32_t G = id.G, grp = id.grp, mem = id.mem;
    uint32_t q;
    if (mem == 0) {
        // ---- the previous tile must be finished by every member before its scratch is reused
        while (as_ld_volatile(&st->grp[grp].done) < G * seq && !as_ld_volatile(&st->abort)) {}
        // ---- take the next tile; wait until it is full, flush it when it stays partial, leave when all trees are done
        q = atomicAdd(&st->tile_head, 1u);
        const uint32_t *cnt_p = P.tile_count + (q % P.NT);
        const uint32_t want = AS_TILE * (q / P.NT + 1u);
        unsigned long long t_partial = 0;
        bool flushed = false;
        for (uint32_t spins = 0;; ++spins) {
            if (as_ld_volatile(cnt_p) >= want) break;
            if (as_ld_volatile(&st->abort)) {
                q = AS_NONE;
                break;
            }
            // every tree has finished the launch: its last row is already published (the rows of the last step are answered
            // in here too — no batched forward behind the kernel), so a tile no row has reached will stay empty
            const bool all_done = as_ld_volatile(&st->done_trees) >= L.B;
            const uint32_t tail = as_ld_volatile(&st->row_tail);
            if (all_done && tail <= q * AS_TILE) {
                q = AS_NONE;
                break;
            }
            if (!flushed && tail > q * AS_TILE && tail < (q + 1u) * AS_TILE) {
                const unsigned long long now = as_now();
                if (t_partial == 0) t_partial = now;
                if (all_done || now - t_partial > P.flush_ns) {
                    const uint32_t k = (q + 1u) * AS_TILE - tail;
                    const uint32_t old = atomicAdd(&st->row_tail, k);
                    for (uint32_t i = 0; i < k; ++i) P.slot_tree[(old + i) % (P.NT * AS_TILE)] = AS_NONE;
                    __threadfence();
                    for (uint32_t i = 0; i < k; ++i) atomicAdd(P.tile_count + (((old + i) / AS_TILE) % P.NT), 1u);
                    atomicAdd(&st->rows_dummy, k);
                    flushed = true;
                }
            }
            __nanosleep(100);
            if ((spins & 255u) == 255u && as_now() - t_start > P.timeout_ns) {
                atomicExch(&st->abort, 1u);
                q = AS_NONE;
                break;
            }
        }
        if (q != AS_NONE) (void)as_ld_acquire(cnt_p);  // the tile's rows and owners are read after this
        st->grp[grp].tile = q;
        __threadfence();
        atomicAdd(&st->grp[grp].seq, 1u);
    } else {
        for (uint32_t spins = 0; as_ld_volatile(&st->grp[grp].seq) <= seq; ++spins) {
            if (member_nap_ns) __nanosleep(member_nap_ns);
            if ((spins & 4095u) == 4095u && as_now() - t_start > P.timeout_ns) atomicExch(&st->abort, 1u);
            if (as_ld_volatile(&st->abort)) break;
        }
        (void)as_ld_acquire(&st->grp[grp].seq);
        q = as_ld_volatile(&st->abort) ? AS_NONE : as_ld_volatile(&st->grp[grp].tile);
    }
    return q;
}

// ---- warp 0: takes tiles for the group, feeds the operand ring by TMA
__device__ __forceinline__ void async_worker_producer(const AzbLayout &L, const AzbAsyncParams &P, const AzbAsyncMaps &M, const AsWorkerId id,
                                      uint8_t *smem, AsWorkerShared &S) {
    const uint32_t lane = threadIdx.x & 31;
    AzbAsyncState *st = P.st;
    if (lane == 0) {
        for (int s = 0; s < AS_STAGES; ++s) {
            tc_mbar_init(&S.full_bar[s], 1);
            tc_mbar_init(&S.empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            tc_mbar_init(&S.acc_full[a], 1);
            tc_mbar_init(&S.acc_empty[a], AS_EPI_WARPS);
        }
        tc_mbar_init(&S.layer_bar, 1);
        tc_mbar_init(&S.h_bar, AS_EPI_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&M.ring) : "memory");
        for (int l = 0; l < 4; ++l) asm volatile("prefetch.tensormap [%0];" ::"l"(&M.w[l]) : "memory");
        for (int l = 0; l < 3; ++l) asm volatile("prefetch.tensormap [%0];" ::"l"(&M.act[l]) : "memory");
    }
    __syncwarp();
    as_named_bar(1, AS_MLP_THREADS);
    const unsigned long long t_start = as_now();
    const uint32_t G = id.G, grp = id.grp, mem = id.mem;
    uint32_t kbc = 0, seq = 0, lbc = 0;  // ring stage counter, tiles taken, layer boundaries passed (G == 1: phase of layer_bar)
    long long d_acq = 0, d_w0 = 0, d_w1 = 0, d_busy = 0, d_tiles = 0;  // debug cycle counters (P.dbg)
    for (;;) {
        if (lane == 0) {
            const long long tq0 = AS_CLK();
            const uint32_t q = as_group_next_tile(L, P, id, seq, t_start, 0u);
            S.tile = q;
            d_acq += AS_CLK() - tq0;
        }
        __syncwarp();
        as_named_bar(1, AS_MLP_THREADS);
        const uint32_t q = S.tile;
        if (q == AS_NONE) break;
        const uint32_t ring_row0 = (q % P.NT) * AS_TILE;
        const uint32_t arrive_target = G * (seq + 1u);  // value of the group's counters once every member has arrived
        if (tc_elect_one()) {
            const long long tt0 = AS_CLK();
            d_tiles += 1;
            const uint64_t w_policy = as_policy_evict_last();
            as_fence_proxy_async();  // the tile's rows were written by tree warps through the generic proxy
            // bf16x3: a dot product runs over three k-segments, (A half, W half) = (hi,hi), (hi,lo), (lo,hi); the lo halves
            // start k_blocks blocks into a row
            const uint32_t nseg = P.wide == 2u ? 3u : 1u;
            for (uint32_t l = 0; l < 4; ++l) {
                const uint32_t k_blocks = P.kpad[l] / TC_BK, kb_all = nseg * k_blocks;
                // this member's blocks nt = mem, mem + G, ... in passes of up to AS_ACC: per k-block ONE A tile and the
                // pass's B tiles, so a tile's activations are read once per pass instead of once per block
                const uint32_t mine = as_blocks_of_member(P.npad[l], id);
                if (as_a_in_tmem(P, l)) {
                    // A is in TMEM: weight tiles only, up to three per stage (all k-blocks of a pass in order), and no
                    // layer barrier — the MMA warp waits for the hidden layer itself
                    const uint32_t pb = as_pass_blocks(true, mine);
                    for (uint32_t p0 = 0; p0 < mine; p0 += pb) {
                        const uint32_t np = min(pb, mine - p0), kps = (1u + AS_ACC) / np;
                        for (uint32_t kb = 0; kb < k_blocks; kb += kps, ++kbc) {
                            const uint32_t s = kbc % AS_STAGES, ph = (kbc / AS_STAGES) & 1u, nk = min(kps, k_blocks - kb);
                            uint8_t *dst = smem + (size_t)s * AS_STAGE_BYTES;
                            const long long tw = AS_CLK();
                            as_mbar_spin(&S.empty_bar[s], ph ^ 1u);
                            d_w0 += AS_CLK() - tw;
                            tc_mbar_expect_tx(&S.full_bar[s], nk * np * AS_TILE_BYTES);
                            for (uint32_t i = 0; i < nk; ++i)
                                for (uint32_t j = 0; j < np; ++j)
                                    as_tma_load_2d_hint(dst + (i * np + j) * AS_TILE_BYTES, &M.w[l], &S.full_bar[s], (int)((kb + i) * TC_BK),
                                                        (int)((p0 + j) * 128u), w_policy);
                        }
                    }
                    continue;
                }
                uint32_t pre = 0;  // k-blocks of the first pass whose weight tiles were requested ahead of the layer barrier
                if (l > 0) {  // this layer's input is the previous layer's output, written by all members
                    // the weights do not depend on it: while the epilogue warps still drain the previous layer, the
                    // ring's stages are free, so the first stages' B tiles go out now and only their A tiles wait
                    const uint32_t np0 = min((uint32_t)AS_ACC, mine);
                    for (; np0 && pre < min((uint32_t)AS_STAGES, k_blocks); ++pre) {
                        const uint32_t kc = kbc + pre, s = kc % AS_STAGES, ph = (kc / AS_STAGES) & 1u;
                        as_mbar_spin(&S.empty_bar[s], ph ^ 1u);
                        uint8_t *a_dst = smem + (size_t)s * AS_STAGE_BYTES;
                        tc_mbar_expect_tx(&S.full_bar[s], (1u + np0) * AS_TILE_BYTES);
                        for (uint32_t j = 0; j < np0; ++j)
                            as_tma_load_2d_hint(a_dst + (1u + j) * AS_TILE_BYTES, &M.w[l], &S.full_bar[s], (int)(pre * TC_BK),
                                                (int)((mem + j * G) * 128u), w_policy);
                    }
                    const long long tw = AS_CLK();
                    if (G == 1u) {  // a single worker: the layer boundary is a shared-memory barrier, not an L2 round trip
                        as_mbar_spin(&S.layer_bar, lbc & 1u);
                        ++lbc;
                    } else {
                        while (as_ld_volatile(&st->grp[grp].layer[l - 1]) < arrive_target && !as_ld_volatile(&st->abort)) {}
                        (void)as_ld_acquire(&st->grp[grp].layer[l - 1]);
                    }
                    d_w1 += AS_CLK() - tw;
                    as_fence_proxy_async();
                }
                const CUtensorMap *ma = l == 0 ? &M.ring : &M.act[l - 1];
                const int arow = (int)(l == 0 ? ring_row0 : grp * AS_TILE);
                for (uint32_t p0 = 0; p0 < mine; p0 += AS_ACC) {
                    const uint32_t np = min((uint32_t)AS_ACC, mine - p0);
                    for (uint32_t kb = 0; kb < kb_all; ++kb, ++kbc) {
                        const uint32_t s = kbc % AS_STAGES, ph = (kbc / AS_STAGES) & 1u;
                        const uint32_t seg = kb / k_blocks, kj = kb - seg * k_blocks;
                        const int a_col = (int)(((seg == 2u ? k_blocks : 0u) + kj) * TC_BK);
                        const int w_col = (int)(((seg == 1u ? k_blocks : 0u) + kj) * TC_BK);
                        uint8_t *a_dst = smem + (size_t)s * AS_STAGE_BYTES;
                        if (p0 == 0u && kb < pre) {  // stage claimed and its B tiles requested above: only the A tile is left
                            tc_tma_load_2d(a_dst, ma, &S.full_bar[s], a_col, arow);
                            continue;
                        }
                        const long long tw = AS_CLK();
                        as_mbar_spin(&S.empty_bar[s], ph ^ 1u);
                        d_w0 += AS_CLK() - tw;
                        tc_mbar_expect_tx(&S.full_bar[s], (1u + np) * AS_TILE_BYTES);
                        tc_tma_load_2d(a_dst, ma, &S.full_bar[s], a_col, arow);
                        for (uint32_t j = 0; j < np; ++j)
                            as_tma_load_2d_hint(a_dst + (1u + j) * AS_TILE_BYTES, &M.w[l], &S.full_bar[s], w_col,
                                                (int)((mem + (p0 + j) * G) * 128u), w_policy);
                    }
                }
            }
            d_busy += AS_CLK() - tt0;
        }
        __syncwarp();
        seq += 1u;
        as_named_bar(1, AS_MLP_THREADS);
    }
#ifdef AZB_PROFILE
    if (P.dbg && lane == 0) {  // producer: acquire, wait empty, wait layer, tile busy, tiles
        atomicAdd(P.dbg + 0, (unsigned long long)d_acq);
        atomicAdd(P.dbg + 1, (unsigned long long)d_w0);
        atomicAdd(P.dbg + 2, (unsigned long long)d_w1);
        atomicAdd(P.dbg + 3, (unsigned long long)d_busy);
        atomicAdd(P.dbg + 4, (unsigned long long)d_tiles);
    }
#endif
    as_named_bar(1, AS_MLP_THREADS);
}

// ---- warp 1: owns TMEM, issues tcgen05.mma
__device__ __forceinline__ void async_worker_mma(const AzbAsyncParams &P, const AsWorkerId id, uint8_t *smem, AsWorkerShared &S) {
    const uint32_t lane = threadIdx.x & 31;
    (void)lane;
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem_u32(&S.tmem_slot)), "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    as_named_bar(1, AS_MLP_THREADS);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = S.tmem_slot;
    const uint32_t G = id.G, mem = id.mem;
    uint32_t kbc = 0, ntc = 0, hbc = 0;  // ring stages, passes, hidden layers read from TMEM (phase of h_bar)
    long long d_w0 = 0, d_w1 = 0;
    for (;;) {
        as_named_bar(1, AS_MLP_THREADS);
        const uint32_t q = S.tile;
        if (q == AS_NONE) break;
        for (uint32_t l = 0; l < 4; ++l) {
            const uint32_t k_blocks = (P.wide == 2u ? 3u : 1u) * (P.kpad[l] / TC_BK);  // all k-segments
            const uint32_t mine = as_blocks_of_member(P.npad[l], id);
            const bool a_tmem = as_a_in_tmem(P, l);
            const uint32_t pb = as_pass_blocks(a_tmem, mine);
            for (uint32_t p0 = 0, p = 0; p0 < mine; p0 += pb, ++p, ++ntc) {
                const uint32_t np = min(pb, mine - p0);
                long long tw = AS_CLK();
                const uint32_t slot = ntc & 1u, acc_ph = (ntc >> 1) & 1u;  // barriers of this pass and their phase
                as_mbar_spin(&S.acc_empty[slot], acc_ph ^ 1u);  // the epilogue has drained the pass before last
                d_w1 += AS_CLK() - tw;
                if (a_tmem && p0 == 0u) {  // the hidden layer is in TMEM (and every pass of the previous layer drained)
                    tw = AS_CLK();
                    as_mbar_spin(&S.h_bar, hbc & 1u);
                    ++hbc;
                    d_w0 += AS_CLK() - tw;
                }
                const uint32_t tmem_acc = tmem_base + as_acc_col(a_tmem, p);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                if (a_tmem) {
                    // weight-only stages of kps k-blocks; per k-step 16 deep the A operand is 8 packed TMEM columns
                    const uint32_t kps = (1u + AS_ACC) / np, bn = min(np * 128u, P.npad[l] - p0 * 128u);
                    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((bn >> 3) << 17) | ((AS_TILE >> 4) << 24);
                    for (uint32_t kb = 0; kb < k_blocks; kb += kps, ++kbc) {
                        const uint32_t s = kbc % AS_STAGES, ph = (kbc / AS_STAGES) & 1u, nk = min(kps, k_blocks - kb);
                        tw = AS_CLK();
                        as_mbar_spin(&S.full_bar[s], ph);
                        d_w0 += AS_CLK() - tw;
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        if (tc_elect_one()) {
                            const uint32_t st_addr = tc_smem_u32(smem + (size_t)s * AS_STAGE_BYTES);
                            for (uint32_t i = 0; i < nk; ++i) {
                                const uint32_t b_addr = st_addr + i * np * AS_TILE_BYTES, ka = tmem_base + (kb + i) * (TC_BK / 2u);
#pragma unroll
                                for (uint32_t k = 0; k < TC_BK / 16; ++k)
                                    as_umma_f16_ts(tmem_acc, ka + k * 8u, tc_smem_desc(b_addr + k * 32u), idesc, ((kb + i) | k) != 0u ? 1u : 0u);
                            }
                            tc_umma_commit(&S.empty_bar[s]);
                            if (kb + nk == k_blocks) tc_umma_commit(&S.acc_full[slot]);
                        }
                        __syncwarp();
                    }
                    continue;
                }
                for (uint32_t kb = 0; kb < k_blocks; ++kb, ++kbc) {
                    const uint32_t s = kbc % AS_STAGES, ph = (kbc / AS_STAGES) & 1u;
                    tw = AS_CLK();
                    as_mbar_spin(&S.full_bar[s], ph);
                    d_w0 += AS_CLK() - tw;
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    if (tc_elect_one()) {
                        const uint32_t a_addr = tc_smem_u32(smem + (size_t)s * AS_STAGE_BYTES);
                        if (G == 1u) {
                            // adjacent 128-column blocks are adjacent in the stage and in TMEM: one N <= 256 MMA per
                            // pair reads the A tile once for both (a 128x128x16 SS-MMA is shared-memory bound)
                            for (uint32_t j = 0; j < np; j += 2) {
                                const uint32_t nt = p0 + j;
                                const uint32_t bn = min(256u, P.npad[l] - nt * 128u);
                                const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((bn >> 3) << 17) | ((AS_TILE >> 4) << 24);
                                const uint32_t b_addr = a_addr + (1u + j) * AS_TILE_BYTES;
#pragma unroll
                                for (uint32_t k = 0; k < TC_BK / 16; ++k)
                                    tc_umma_f16(tmem_acc + j * 128u, tc_smem_desc(a_addr + k * 32u), tc_smem_desc(b_addr + k * 32u),
                                                idesc, (kb | k) != 0u ? 1u : 0u);
                            }
                        } else {
                            for (uint32_t j = 0; j < np; ++j) {
                                const uint32_t nt = mem + (p0 + j) * G;
                                const uint32_t bn = min(128u, P.npad[l] - nt * 128u);
                                const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((bn >> 3) << 17) | ((AS_TILE >> 4) << 24);
                                const uint32_t b_addr = a_addr + (1u + j) * AS_TILE_BYTES;
#pragma unroll
                                for (uint32_t k = 0; k < TC_BK / 16; ++k)
                                    tc_umma_f16(tmem_acc + j * 128u, tc_smem_desc(a_addr + k * 32u), tc_smem_desc(b_addr + k * 32u),
                                                idesc, (kb | k) != 0u ? 1u : 0u);
                            }
                        }
                        tc_umma_commit(&S.empty_bar[s]);
                        if (kb + 1 == k_blocks) tc_umma_commit(&S.acc_full[slot]);
                    }
                    __syncwarp();
                }
            }
        }
        as_named_bar(1, AS_MLP_THREADS);
    }
#ifdef AZB_PROFILE
    if (P.dbg && lane == 0) {  // MMA: -, wait full, wait acc_empty
        atomicAdd(P.dbg + 5 + 1, (unsigned long long)d_w0);
        atomicAdd(P.dbg + 5 + 2, (unsigned long long)d_w1);
    }
#endif
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    as_named_bar(1, AS_MLP_THREADS);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
}

// ---- warps 4-11: TMEM -> registers -> bias + activation -> scratch / prior rows
__device__ __forceinline__ void async_worker_epilogue(const AzbLayout &L, const AzbAsyncParams &P, const AsWorkerId id, uint8_t *smem,
                                      AsWorkerShared &S) {
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t et = threadIdx.x - AS_EPI_WARP0 * 32u;  // 0 .. 255
    AzbAsyncState *st = P.st;
    // all biases into shared memory (behind the operand ring): the epilogue's only global traffic is its output
    float *s_bias = reinterpret_cast<float *>(smem + (size_t)AS_STAGES * AS_STAGE_BYTES);
    uint32_t bias_end = 0;
    for (int l = 0; l < 4; ++l) {
        if (et == 0u) S.bias_off[l] = bias_end;
        for (uint32_t i = et; i < P.npad[l]; i += AS_EPI_WARPS * 32u) s_bias[bias_end + i] = P.bias[l][i];
        bias_end += (P.npad[l] + 31u) & ~31u;
    }
    // per epilogue warp a staging tile behind the biases (coalesced activation stores)
    uint8_t *stg = reinterpret_cast<uint8_t *>(s_bias + bias_end);
    stg = (uint8_t *)(((uintptr_t)stg + 1023) & ~(uintptr_t)1023) + (warp - AS_EPI_WARP0) * AS_EPI_STG_BYTES;  // swizzle atoms: 1 KB
    as_named_bar(1, AS_MLP_THREADS);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = S.tmem_slot;
    const uint32_t G = id.G, grp = id.grp, mem = id.mem;
    // warp w may read TMEM lanes 32 (w % 4) ..; the two warps of a quadrant split each 128-column block in halves
    const uint32_t q4 = warp & 3u, part = (warp - AS_EPI_WARP0) >> 2, col0 = part * AS_EPI_COLS, row = q4 * 32u + lane;
    uint32_t ntc = 0, seq = 0;
    long long d_acq = 0, d_w0 = 0, d_w1 = 0, d_busy = 0;
    for (;;) {
        as_named_bar(1, AS_MLP_THREADS);
        const uint32_t q = S.tile;
        if (q == AS_NONE) break;
        const uint32_t ring_row0 = (q % P.NT) * AS_TILE;
        const uint32_t arrive_target = G * (seq + 1u);
        if (et < AS_TILE) S.rowtree[et] = __ldcg(P.slot_tree + ring_row0 + et);
        as_named_bar(2, AS_EPI_WARPS * 32);
        const uint32_t my_tree = S.rowtree[row];
        for (uint32_t l = 0; l < 4; ++l) {
            const float *bias = s_bias + S.bias_off[l];
            const uint32_t mine = as_blocks_of_member(P.npad[l], id);
            const bool a_tmem = as_a_in_tmem(P, l), out_tmem = l < 3u && as_a_in_tmem(P, l + 1u);
            const uint32_t pb = as_pass_blocks(a_tmem, mine);
            for (uint32_t p0 = 0, p = 0; p0 < mine; p0 += pb, ++p, ++ntc) {
                const uint32_t np = min(pb, mine - p0);
                const long long tw = AS_CLK();
                const uint32_t slot = ntc & 1u, acc_ph = (ntc >> 1) & 1u;
                as_mbar_spin(&S.acc_full[slot], acc_ph);
                const uint32_t tmem_acc = tmem_base + as_acc_col(a_tmem, p);
                const long long tb = AS_CLK();
                d_w0 += tb - tw;
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                for (uint32_t ja = 0; ja < np; ++ja) {
                    const uint32_t nt = mem + (p0 + ja) * G;
                    const uint32_t bn = min(128u, P.npad[l] - nt * 128u);
                    if (out_tmem) {
                        // the next layer's A operand: this warp's 64 columns of the block, bias + ReLU, bf16 pairs into TMEM
                        // column (nt * 128 + col0) / 2 + i of its own lanes.  Those columns belong to pass 0's accumulator;
                        // the quadrant's other warp has read its part of them once it reaches the pair barrier
                        uint32_t pk[AS_EPI_COLS / 2];
                        if (col0 < bn) {
                            uint32_t r[AS_EPI_SLICES][16];
                            const long long tl0 = AS_CLK();
#pragma unroll
                            for (uint32_t sl = 0; sl < AS_EPI_SLICES; ++sl)
                                as_tmem_ld16_issue(tmem_acc + ((q4 * 32u) << 16) + ja * 128u + col0 + sl * 16u, r[sl]);
                            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                            d_acq += AS_CLK() - tl0;
                            const uint32_t bias_s = tc_smem_u32(bias + nt * 128u + col0);
#pragma unroll
                            for (uint32_t sl = 0; sl < AS_EPI_SLICES; ++sl) as_relu_pack(r[sl], bias_s + sl * 64u, 0u, pk + sl * 8u);
                        }
                        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                        as_named_bar(4u + q4, 64u);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        if (col0 < bn) as_tmem_st32(tmem_base + ((q4 * 32u) << 16) + (nt * 128u + col0) / 2u, pk);
                    } else if (l < 3) {
                        // this warp's 64 columns of the block: four 16-column TMEM slices in flight at once, bias + ReLU,
                        // bf16 pairs into the warp's staging tile [32 rows x 128 B]; 16-byte chunks XOR-swizzled by row,
                        // so these stores and the row-wise reads below are both bank-conflict free
                        if (col0 < bn) {
                            uint32_t r[AS_EPI_SLICES][16];
                            const long long tl0 = AS_CLK();
#pragma unroll
                            for (uint32_t sl = 0; sl < AS_EPI_SLICES; ++sl)
                                as_tmem_ld16_issue(tmem_acc + ((q4 * 32u) << 16) + ja * 128u + col0 + sl * 16u, r[sl]);
                            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                            d_acq += AS_CLK() - tl0;
                            const uint32_t srow = tc_smem_u32(stg) + lane * (AS_EPI_COLS * 2u);
                            const uint32_t bias_s = tc_smem_u32(bias + nt * 128u + col0);
                            const uint32_t sw = AS_EPI_CHUNKS == 8 ? (lane & 7u) : ((lane >> 1) & 3u);  // chunk swizzle of this row
                            const uint32_t act_ld = P.wide * P.kpad[l + 1];
                            // half 0: the bf16 activations; half 1 (bf16x3 only): what bf16 lost, bf16(v - hi), stored
                            // kpad columns further into the row
                            for (uint32_t half = 0; half < P.wide; ++half) {
#pragma unroll
                                for (uint32_t sl = 0; sl < AS_EPI_SLICES; ++sl) {
                                    uint32_t pk[8];
                                    as_relu_pack(r[sl], bias_s + sl * 64u, half, pk);
                                    const uint32_t ch = 2u * sl;  // this slice's two 16-byte chunks in the staged row
                                    as_sts128(srow + ((ch ^ sw) << 4), pk[0], pk[1], pk[2], pk[3]);
                                    as_sts128(srow + (((ch + 1u) ^ sw) << 4), pk[4], pk[5], pk[6], pk[7]);
                                }
                                // the warp's [32 rows x AS_EPI_COLS columns] go out as contiguous row pieces: AS_EPI_CHUNKS lanes
                                // per row (a store per thread and row touched 32 lines per instruction and held the epilogue to
                                // ~0.4 us per 16-column slice on the LSU)
                                __syncwarp();
                                const uint32_t rr = lane / AS_EPI_CHUNKS, cc = lane % AS_EPI_CHUNKS;
                                __nv_bfloat16 *dst0 = P.act[l] + (size_t)(grp * AS_TILE + q4 * 32u) * act_ld + half * P.kpad[l + 1] +
                                                      nt * 128u + col0 + cc * 8u;
#pragma unroll
                                for (uint32_t it = 0; it < AS_EPI_CHUNKS; ++it) {
                                    const uint32_t rw = it * (32u / AS_EPI_CHUNKS) + rr;
                                    const uint32_t sw2 = AS_EPI_CHUNKS == 8 ? (rw & 7u) : ((rw >> 1) & 3u);
                                    const uint4 v = as_lds128(tc_smem_u32(stg) + rw * (AS_EPI_COLS * 2u) + ((cc ^ sw2) << 4));
                                    *reinterpret_cast<uint4 *>(dst0 + (size_t)rw * act_ld) = v;
                                }
                                __syncwarp();
                            }
                        }
                    } else {
                        // the Sigmoid head: f32 rows scattered to the owning trees' prior rows, 16 columns at a time
                        for (uint32_t c0 = col0; c0 < min(bn, col0 + (uint32_t)AS_EPI_COLS); c0 += 16) {
                            uint32_t r[16];
                            const long long tl0 = AS_CLK();
                            as_tmem_ld16(tmem_acc + ((q4 * 32u) << 16) + ja * 128u + c0, r);
                            d_acq += AS_CLK() - tl0;
                            const uint32_t nb = nt * 128u + c0;
                            float b[16];
#pragma unroll
                            for (int j = 0; j < 16; j += 4) {
                                const float4 b4 = *reinterpret_cast<const float4 *>(bias + nb + j);
                                b[j] = b4.x;
                                b[j + 1] = b4.y;
                                b[j + 2] = b4.z;
                                b[j + 3] = b4.w;
                            }
                            if (my_tree != AS_NONE) {
                                float *dst = L.h + (size_t)my_tree * L.h_ld;
                                const bool vec = (L.h_ld & 3u) == 0u;
#pragma unroll
                                for (int j = 0; j < 16; j += 4) {
                                    float o[4];
#pragma unroll
                                    for (int t = 0; t < 4; ++t) {
                                        const float v = __uint_as_float(r[j + t]) + b[j + t];
                                        o[t] = __fdividef(1.0f, 1.0f + __expf(-v));
                                    }
                                    const uint32_t n = nb + j;
                                    if (vec && n + 3u < L.A) {
                                        *reinterpret_cast<float4 *>(dst + n) = make_float4(o[0], o[1], o[2], o[3]);
                                    } else {
#pragma unroll
                                        for (int t = 0; t < 4; ++t)
                                            if (n + t < L.A) dst[n + t] = o[t];
                                    }
                                }
                            }
                        }
                    }
                }
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) as_mbar_arrive(&S.acc_empty[slot]);
                d_busy += AS_CLK() - tb;
            }
            const long long tf0 = AS_CLK();
            if (out_tmem) {  // the hidden layer is in TMEM: the MMA warp reads it behind h_bar
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) as_mbar_arrive(&S.h_bar);
                d_w1 += AS_CLK() - tf0;
                continue;
            }
            // ---- layer boundary: this member's share of the layer is stored; tell the group
            if (l < 3) as_fence_proxy_async();  // the next layer reads these stores through TMA
            // a single worker hands its hidden activations to its OWN producer warp: the cross-proxy fence, the CTA barrier
            // and the mbarrier's release/acquire are what the memory model asks for.  A GPU-scope fence is needed where
            // another SM reads them (G > 1) and before the answer flags (l == 3; it waits for every store's acknowledgement)
            if (G > 1u || l == 3u) __threadfence();
            as_named_bar(2, AS_EPI_WARPS * 32);
            if (et == 0u) {
                if (l < 3) {
                    if (G == 1u) as_mbar_arrive(&S.layer_bar);
                    else atomicAdd(&st->grp[grp].layer[l], 1u);
                } else if (atomicAdd(&st->grp[grp].done, 1u) + 1u == arrive_target) {
                    S.epi_last = 1u;  // this member is the last of the group to finish the tile
                } else {
                    S.epi_last = 0u;
                }
            }
            d_w1 += AS_CLK() - tf0;
        }
        // the tile is answered once every member is done: the last one raises the owners' flags
        as_named_bar(2, AS_EPI_WARPS * 32);
        if (S.epi_last) {
            __threadfence();
#ifdef AZB_PROFILE
            if (part == 0u && my_tree != AS_NONE && my_tree < 65536u) g_flag_time[my_tree] = as_now();
#endif
            if (part == 0u && my_tree != AS_NONE) atomicAdd(P.h_flag + my_tree, 1u);
            if (et == 0u) {
                atomicAdd(P.tile_retired + (q % P.NT), 1u);
                atomicAdd(&st->tiles_done, 1u);
            }
        }
        seq += 1u;
        as_named_bar(1, AS_MLP_THREADS);
    }
#ifdef AZB_PROFILE
    if (P.dbg && et == 0u) {  // epilogue (first warp): TMEM reads, wait acc_full, layer boundary, busy
        atomicAdd(P.dbg + 10, (unsigned long long)d_acq);
        atomicAdd(P.dbg + 11, (unsigned long long)d_w0);
        atomicAdd(P.dbg + 12, (unsigned long long)d_w1);
        atomicAdd(P.dbg + 13, (unsigned long long)d_busy);
    }
#endif
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    as_named_bar(1, AS_MLP_THREADS);
}

// Role dispatch of a model CTA (all 1024 threads enter): re-divide the registers, then run the role
__device__ __forceinline__ void async_model_cta(const AzbLayout &L, const AzbAsyncParams &P, const AzbAsyncMaps &M,
                                                const uint32_t worker, uint8_t *smem, AsWorkerShared &S) {
    const uint32_t warp = threadIdx.x >> 5, wg = warp >> 2;
    AsWorkerId id;
    id.G = P.group;
    id.grp = worker / P.group;
    id.mem = worker % P.group;
    if (wg >= 3u) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(AS_REGS_IDLE));
        return;
    }
    if (wg == 0u) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(AS_REGS_FRONT));
        if (warp == 0u) async_worker_producer(L, P, M, id, smem, S);
        else if (warp == 1u) async_worker_mma(P, id, smem, S);
        return;
    }
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(AS_REGS_EPI));
    async_worker_epilogue(L, P, id, smem, S);
}

// ---------------------------------------------------------------------------------------------------------------
// Shared-SM form (P.shared_sm; azb_config.async_workers = AZB_ASYNC_SHARED).  No SM is taken from the trees: every CTA
// walks trees with its first SH_TREE_WARPS warps, and its last warpgroup (4 warps, the kernel's 64 registers) is one
// MEMBER of a model group.  G members on G different SMs answer a 128-row tile together: member m computes the columns
// [m cw_l, (m + 1) cw_l) of every layer, so only 1/G of the weights streams through each SM's 64 B/clk L2 port — the
// port is what bounds a tile on one SM (3.9 MB per tile: 31 us) —, the hidden activations meet in the group's L2-resident
// scratch, and the members synchronise at the three layer boundaries through the group's counter line.  With G = 8 a tile
// moves 0.95 MB through each member and 18 groups are in flight on 148 SMs, which is far more model throughput than
// 4096 trees can ask for: the round trip a tree waits for shrinks while all 148 SMs keep walking.
// Roles inside the warpgroup: warp 0's elected lane takes the tile (group leader) or reads the mailbox and issues the TMA
// loads, warp 1's elected lane issues tcgen05.mma (accumulator [128 x cw_l] fp32 in TMEM, single-buffered: the next
// layer cannot start before the group barrier anyway); then all four warps drain their TMEM lane quadrant (bias, ReLU,
// bf16 through a swizzled staging tile into the scratch; the Sigmoid head scatters f32 to the owners' prior rows).
// Waits on mbarriers suspend (try_wait) and the mailbox poll naps, so an idle member costs its SM's walkers next to nothing.
#define SH_TREE_WARPS 28
#define SH_THREADS 128
#define SH_MAX_STAGES AS_STAGES  // operand ring stages (P.sh_stages <= this; fewer when a wide slice fills shared memory)
#define SH_STG_BYTES (32u * 128u)  // per-warp staging tile: 32 rows x 64 bf16
#define SH_TMEM_COLS 256u

__device__ __forceinline__ uint32_t sh_stage_bytes(const AzbAsyncParams &P) {
    const uint32_t cwmax = max(max(P.cw[0], P.cw[1]), max(P.cw[2], P.cw[3]));
    return AS_TILE_BYTES + cwmax * (TC_BK * 2u);
}

// shared-space addresses (u32) all the way in the member's issue loops: one lane runs them beside 28 walking warps, and
// every instruction on that lane's path costs ~10 cycles there
__device__ __forceinline__ void sh_mbar_wait(uint32_t bar_s, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "SH_WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra.uni SH_WAIT_DONE;\n"
        "bra.uni SH_WAIT_LOOP;\n"
        "SH_WAIT_DONE:\n"
        "}\n" ::"r"(bar_s),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void sh_mbar_expect_tx(uint32_t bar_s, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_s), "r"(bytes) : "memory");
}
__device__ __forceinline__ void sh_tma_load_2d(uint32_t dst_s, const CUtensorMap *map, uint32_t bar_s, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst_s),
                 "l"(map), "r"(bar_s), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void sh_tma_load_2d_hint(uint32_t dst_s, const CUtensorMap *map, uint32_t bar_s, int c0, int c1, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(dst_s),
        "l"(map), "r"(bar_s), "r"(c0), "r"(c1), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void sh_umma_commit(uint32_t bar_s) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_s) : "memory");
}
__device__ __forceinline__ void sh_tmem_ld16_issue(uint32_t taddr, uint32_t (&r)[16]) { as_tmem_ld16_issue(taddr, r); }

// bias + ReLU + bf16 of one 16-column TMEM slice into two 16-byte chunks of the warp's staged row
__device__ __forceinline__ void sh_relu_pack_store(const uint32_t (&r)[16], uint32_t bias_s, uint32_t half, uint32_t srow, uint32_t ch, uint32_t sw) {
    uint32_t pk[8];
    as_relu_pack(r, bias_s, half, pk);
    as_sts128(srow + ((ch ^ sw) << 4), pk[0], pk[1], pk[2], pk[3]);
    as_sts128(srow + (((ch + 1u) ^ sw) << 4), pk[4], pk[5], pk[6], pk[7]);
}

__device__ void shared_model_warpgroup(const AzbLayout &L, const AzbAsyncParams &P, const AzbAsyncMaps &M, const uint32_t member,
                                       uint8_t *smem, AsWorkerShared &S) {
    const uint32_t mt = threadIdx.x - SH_TREE_WARPS * 32u, warp = mt >> 5, lane = mt & 31u;
    AzbAsyncState *st = P.st;
    AsWorkerId id;
    id.G = P.group;
    id.grp = member / P.group;
    id.mem = member % P.group;
    const uint32_t G = id.G, grp = id.grp, mem = id.mem;
    const uint32_t stage_bytes = sh_stage_bytes(P), n_stages = P.sh_stages;
    // this member's bias slices behind the operand ring, then one staging tile per warp
    float *s_bias = reinterpret_cast<float *>(smem + (size_t)n_stages * stage_bytes);
    uint32_t bias_end = 0;
    for (uint32_t l = 0; l < 4; ++l) {
        if (mt == 0u) S.bias_off[l] = bias_end;
        for (uint32_t i = mt; i < P.cw[l]; i += SH_THREADS) {
            const uint32_t n = mem * P.cw[l] + i;
            s_bias[bias_end + i] = n < P.npad[l] ? P.bias[l][n] : 0.f;
        }
        bias_end += P.cw[l];
    }
    uint8_t *stg = reinterpret_cast<uint8_t *>(s_bias + bias_end);
    stg = (uint8_t *)(((uintptr_t)stg + 1023) & ~(uintptr_t)1023) + warp * SH_STG_BYTES;
    if (mt == 0u) {
        for (uint32_t s = 0; s < n_stages; ++s) {
            tc_mbar_init(&S.full_bar[s], 1);
            tc_mbar_init(&S.empty_bar[s], 1);
        }
        tc_mbar_init(&S.acc_full[0], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&M.ring) : "memory");
        for (int l = 0; l < 4; ++l) asm volatile("prefetch.tensormap [%0];" ::"l"(&M.ws[l]) : "memory");
        for (int l = 0; l < 3; ++l) asm volatile("prefetch.tensormap [%0];" ::"l"(&M.act[l]) : "memory");
    }
    if (warp == 1u) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem_u32(&S.tmem_slot)), "r"(SH_TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    as_named_bar(1, SH_THREADS);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = S.tmem_slot;
    const unsigned long long t_start = as_now();
    const uint32_t nseg = P.wide == 2u ? 3u : 1u;
    const uint32_t ring_s = tc_smem_u32(smem), full_s = tc_smem_u32(&S.full_bar[0]), empty_s = tc_smem_u32(&S.empty_bar[0]),
                   acc_s = tc_smem_u32(&S.acc_full[0]);
    // ring cursor of the issuing lanes (warps 0 and 1 walk the same k-block sequence): stage and phase, no divisions
    uint32_t rs = 0, rph = 0;
    uint32_t accc = 0, seq = 0;  // accumulators completed, tiles answered (uniform over the warpgroup)
    long long d_acq = 0, d_busy = 0, d_w1 = 0, d_tiles = 0, d_pe = 0, d_mf = 0, d_acc = 0, d_epi = 0, d_bar = 0;
    for (;;) {
        if (mt == 0u) {
            const long long tq0 = AS_CLK();
            S.tile = as_group_next_tile(L, P, id, seq, t_start, 200u);
            d_acq += AS_CLK() - tq0;
        }
        as_named_bar(1, SH_THREADS);
        const uint32_t q = S.tile;
        if (q == AS_NONE) break;
        const long long tt0 = AS_CLK();
        const uint32_t ring_row0 = (q % P.NT) * AS_TILE;
        const uint32_t arrive_target = G * (seq + 1u);
        const uint32_t my_tree = __ldcg(P.slot_tree + ring_row0 + mt);  // owner of this thread's row (128 threads, 128 rows)
        for (uint32_t l = 0; l < 4; ++l) {
            const uint32_t k_blocks = P.kpad[l] / TC_BK;
            const uint32_t n0 = mem * P.cw[l];
            const uint32_t bn = n0 < P.npad[l] ? min(P.cw[l], P.npad[l] - n0) : 0u;  // this member's columns of the layer
            if (warp == 0u) {
                // ===== TMA producer (one elected lane)
                if (tc_elect_one()) {
                    const uint32_t tx_bytes = AS_TILE_BYTES + P.cw[l] * (TC_BK * 2u);  // the weight box is always cw[l] rows
                    const uint64_t w_policy = as_policy_evict_last();
                    const CUtensorMap *mw = &M.ws[l];
                    uint32_t pre = 0;
                    if (l == 0u) {
                        as_fence_proxy_async();  // the tile's rows were written by tree warps through the generic proxy
                    } else {
                        // the weights do not depend on the previous layer: the first stages' B tiles go out before the
                        // group's layer barrier opens, only their A tiles wait for it
                        uint32_t ps = rs, pph = rph;
                        for (; bn && pre < min(n_stages, k_blocks); ++pre) {
                            sh_mbar_wait(empty_s + 8u * ps, pph ^ 1u);
                            sh_mbar_expect_tx(full_s + 8u * ps, tx_bytes);
                            sh_tma_load_2d_hint(ring_s + ps * stage_bytes + AS_TILE_BYTES, mw, full_s + 8u * ps, (int)(pre * TC_BK), (int)n0, w_policy);
                            if (++ps == n_stages) {
                                ps = 0;
                                pph ^= 1u;
                            }
                        }
                        const long long tw = AS_CLK();
                        const uint32_t *lp = &st->grp[grp].layer[l - 1];
                        while (as_ld_volatile(lp) < arrive_target && !as_ld_volatile(&st->abort)) {}
                        (void)as_ld_acquire(lp);
                        d_w1 += AS_CLK() - tw;
                        as_fence_proxy_async();
                    }
                    const CUtensorMap *ma = l == 0u ? &M.ring : &M.act[l - 1];
                    const int arow = (int)(l == 0u ? ring_row0 : grp * AS_TILE);
                    if (bn) {
                        uint32_t kb = 0;
                        for (uint32_t seg = 0; seg < nseg; ++seg) {
                            // bf16x3: (A half, W half) = (hi,hi), (hi,lo), (lo,hi); the lo halves start k_blocks blocks into a row
                            int a_col = (int)((seg == 2u ? k_blocks : 0u) * TC_BK), w_col = (int)((seg == 1u ? k_blocks : 0u) * TC_BK);
                            for (uint32_t kj = 0; kj < k_blocks; ++kj, ++kb, a_col += TC_BK, w_col += TC_BK) {
                                const uint32_t fb = full_s + 8u * rs, dst = ring_s + rs * stage_bytes;
                                if (kb >= pre) {  // (else: stage claimed and its B tile requested above)
                                    const long long te = AS_CLK();
                                    sh_mbar_wait(empty_s + 8u * rs, rph ^ 1u);
                                    d_pe += AS_CLK() - te;
                                    sh_mbar_expect_tx(fb, tx_bytes);
                                    sh_tma_load_2d_hint(dst + AS_TILE_BYTES, mw, fb, w_col, (int)n0, w_policy);
                                }
                                sh_tma_load_2d(dst, ma, fb, a_col, arow);
                                if (++rs == n_stages) {
                                    rs = 0;
                                    rph ^= 1u;
                                }
                            }
                        }
                    }
                }
                __syncwarp();
            } else if (warp == 1u && bn) {
                // ===== MMA issuer (one elected lane): D[128 x bn] (+)= A[128 x 64] B[bn x 64]^T per k-block, four K = 16 steps
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                if (tc_elect_one()) {
                    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((bn >> 3) << 17) | ((AS_TILE >> 4) << 24);
                    const uint32_t kb_all = nseg * k_blocks;
                    for (uint32_t kb = 0; kb < kb_all; ++kb) {
                        const long long tf = AS_CLK();
                        sh_mbar_wait(full_s + 8u * rs, rph);
                        d_mf += AS_CLK() - tf;
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        const uint32_t a_addr = ring_s + rs * stage_bytes;
                        const uint64_t adesc = tc_smem_desc(a_addr), bdesc = tc_smem_desc(a_addr + AS_TILE_BYTES);
#pragma unroll
                        for (uint32_t k = 0; k < TC_BK / 16; ++k)  // 32 bytes further along K: +2 in the descriptor's address field
                            tc_umma_f16(tmem_base, adesc + 2u * k, bdesc + 2u * k, idesc, (kb | k) != 0u ? 1u : 0u);
                        sh_umma_commit(empty_s + 8u * rs);
                        if (kb + 1u == kb_all) sh_umma_commit(acc_s);
                        if (++rs == n_stages) {
                            rs = 0;
                            rph ^= 1u;
                        }
                    }
                }
                __syncwarp();
            }
            if (bn) {
                // ===== epilogue: every warp drains its TMEM lane quadrant (rows 32 warp .. of the tile)
                const long long ta = AS_CLK();
                sh_mbar_wait(acc_s, accc & 1u);
                ++accc;
                const long long tb = AS_CLK();
                d_acc += tb - ta;
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t bias_s = tc_smem_u32(s_bias + S.bias_off[l]);
                const uint32_t tq = tmem_base + ((warp * 32u) << 16);
                if (l < 3u) {
                    const uint32_t act_ld = P.wide * P.kpad[l + 1];
                    const uint32_t stg_s = tc_smem_u32(stg), srow = stg_s + lane * 128u, sw = lane & 7u;
                    for (uint32_t c0 = 0; c0 < bn; c0 += 64u) {
                        const uint32_t ncols = min(64u, bn - c0), chunks = ncols >> 3;
                        for (uint32_t half = 0; half < P.wide; ++half) {
                            // 16-column slices in pairs: two TMEM loads in flight, one wait
#pragma unroll 1
                            for (uint32_t sl = 0; sl < (ncols >> 4); sl += 2u) {
                                uint32_t r0[16], r1[16];
                                const bool two = sl + 1u < (ncols >> 4);
                                sh_tmem_ld16_issue(tq + c0 + sl * 16u, r0);
                                if (two) sh_tmem_ld16_issue(tq + c0 + sl * 16u + 16u, r1);
                                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                                sh_relu_pack_store(r0, bias_s + (c0 + sl * 16u) * 4u, half, srow, 2u * sl, sw);
                                if (two) sh_relu_pack_store(r1, bias_s + (c0 + sl * 16u + 16u) * 4u, half, srow, 2u * sl + 2u, sw);
                            }
                            __syncwarp();
                            // the warp's [32 rows x ncols] leave as contiguous row pieces, `chunks` lanes per row
                            __nv_bfloat16 *dst0 = P.act[l] + (size_t)(grp * AS_TILE + warp * 32u) * act_ld + half * P.kpad[l + 1] + n0 + c0;
                            if (chunks == 8u) {
                                const uint32_t rr = lane >> 3, cc = lane & 7u;
#pragma unroll
                                for (uint32_t it = 0; it < 8u; ++it) {
                                    const uint32_t rw = it * 4u + rr;
                                    const uint4 v = as_lds128(stg_s + rw * 128u + ((cc ^ (rw & 7u)) << 4));
                                    *reinterpret_cast<uint4 *>(dst0 + (size_t)rw * act_ld + cc * 8u) = v;
                                }
                            } else {
#pragma unroll 1
                                for (uint32_t idx = lane; idx < 32u * chunks; idx += 32u) {
                                    const uint32_t rw = idx / chunks, cc = idx - rw * chunks;
                                    const uint4 v = as_lds128(stg_s + rw * 128u + ((cc ^ (rw & 7u)) << 4));
                                    *reinterpret_cast<uint4 *>(dst0 + (size_t)rw * act_ld + cc * 8u) = v;
                                }
                            }
                            __syncwarp();
                        }
                    }
                } else {
                    // the Sigmoid head: f32 rows scattered to the owning trees' prior rows, 16 columns at a time
                    float *dst = L.h + (size_t)(my_tree != AS_NONE ? my_tree : 0u) * L.h_ld;
                    const bool vec = (L.h_ld & 3u) == 0u;
#pragma unroll 1
                    for (uint32_t c0 = 0; c0 < bn; c0 += 16u) {
                        uint32_t r[16];
                        as_tmem_ld16(tq + c0, r);
                        if (my_tree != AS_NONE) {
#pragma unroll
                            for (int j = 0; j < 16; j += 4) {
                                const uint4 b4 = as_lds128(bias_s + (c0 + j) * 4u);
                                float o[4];
                                o[0] = __uint_as_float(r[j]) + __uint_as_float(b4.x);
                                o[1] = __uint_as_float(r[j + 1]) + __uint_as_float(b4.y);
                                o[2] = __uint_as_float(r[j + 2]) + __uint_as_float(b4.z);
                                o[3] = __uint_as_float(r[j + 3]) + __uint_as_float(b4.w);
#pragma unroll
                                for (int t = 0; t < 4; ++t) o[t] = __fdividef(1.0f, 1.0f + __expf(-o[t]));
                                const uint32_t n = n0 + c0 + j;
                                if (vec && n + 3u < L.A) {
                                    *reinterpret_cast<float4 *>(dst + n) = make_float4(o[0], o[1], o[2], o[3]);
                                } else {
#pragma unroll
                                    for (int t = 0; t < 4; ++t)
                                        if (n + t < L.A) dst[n + t] = o[t];
                                }
                            }
                        }
                    }
                }
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                d_epi += AS_CLK() - tb;
            }
            // ---- layer boundary: this member's share of the layer is stored; tell the group.  The barrier orders the 128
            // threads' stores before thread 0's fence, and the fence is cumulative: ONE L1 invalidation per boundary on an
            // SM whose other 28 warps are walking trees
            const long long tz = AS_CLK();
            if (l < 3u) as_fence_proxy_async();  // the next layer reads these stores through TMA
            as_named_bar(2, SH_THREADS);
            if (mt == 0u) {
                __threadfence();
                if (l < 3u)
                    atomicAdd(&st->grp[grp].layer[l], 1u);
                else
                    S.epi_last = atomicAdd(&st->grp[grp].done, 1u) + 1u == arrive_target ? 1u : 0u;
            }
            d_bar += AS_CLK() - tz;
        }
        // the tile is answered once every member is done: the last one raises the owners' flags
        as_named_bar(2, SH_THREADS);
        if (S.epi_last) {
            if (mt == 0u) __threadfence();  // behind the last arrival: every member's prior rows are visible before the flags
            as_named_bar(2, SH_THREADS);
            if (my_tree != AS_NONE) atomicAdd(P.h_flag + my_tree, 1u);
            if (mt == 0u) {
                atomicAdd(P.tile_retired + (q % P.NT), 1u);
                atomicAdd(&st->tiles_done, 1u);
            }
        }
        seq += 1u;
        d_tiles += 1;
        d_busy += AS_CLK() - tt0;
    }
#ifdef AZB_PROFILE
    if (P.dbg && mt == 0u) {  // acquire, producer wait-empty, wait layer, tile busy, tiles (the slots of the whole-SM producer)
        atomicAdd(P.dbg + 0, (unsigned long long)d_acq);
        atomicAdd(P.dbg + 1, (unsigned long long)d_pe);
        atomicAdd(P.dbg + 2, (unsigned long long)d_w1);
        atomicAdd(P.dbg + 3, (unsigned long long)d_busy);
        atomicAdd(P.dbg + 4, (unsigned long long)d_tiles);
    }
    if (P.dbg && mt == 32u) atomicAdd(P.dbg + 6, (unsigned long long)d_mf);
    if (P.dbg && mt == 64u) {  // a warp that only waits and drains: accumulator wait, epilogue, fence + barrier
        atomicAdd(P.dbg + 11, (unsigned long long)d_acc);
        atomicAdd(P.dbg + 13, (unsigned long long)d_epi);
        atomicAdd(P.dbg + 12, (unsigned long long)d_bar);
    }
#endif
    (void)d_acq; (void)d_busy; (void)d_w1; (void)d_tiles; (void)d_pe; (void)d_mf; (void)d_acc; (void)d_epi; (void)d_bar;
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    as_named_bar(1, SH_THREADS);
    if (warp == 1u) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(SH_TMEM_COLS) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Tree CTA.  A CTA owns a contiguous block of the batch's trees (slot i = tree0 + i), so a tree's arena is only ever seen through one
// SM's L1 — but WITHIN the CTA any free warp advances any runnable tree.  (Round 1 and the first half of round 2 gave every
// warp a fixed set of trees, warp + k * n_warps: with 8192 roots on 120 tree SMs some warps owned three trees and the
// others two, and a warp whose tree waited for its priors idled beside a neighbour with two runnable trees.)
// The CTA's scheduling table lives in shared memory, one entry per slot:
//   state  0 runnable, 1 waiting for its priors, 2 done with this launch, 3 being advanced by a warp
//   sub    rows this tree has handed to the model since the launch began (the answer flag it waits for)
//   steps  times it has been advanced (the warp takes the runnable tree that is furthest behind)
// A warp that finds nothing runnable takes the CTA's sweep token and polls the answer flags of ALL waiting slots (32 per
// ld.volatile round trip), marks the answered ones runnable behind ONE gpu-scope fence — the acquire side of the model CTAs'
// fence + atomicAdd; every tree-step used to pay its own acquire load and with it an invalidation of the SM's L1 — and
// rescans.  Warps without the token nap and rescan shared memory only, so an SM polls L2 with one warp at a time however
// many of its warps wait.
#ifdef AZB_PROFILE
#define AS_TAB_ARRAYS 6u
#else
#define AS_TAB_ARRAYS 3u
#endif
__host__ __device__ __forceinline__ size_t as_table_bytes(uint32_t slots) { return ((size_t)AS_TAB_ARRAYS * slots + 16u) * 4u; }
struct AsTreeTable {
    uint32_t *state, *sub, *steps;
    uint32_t *ctl;  // [0] slots done, [1] sweep token, [3] clock of the last sweep, [4] runnable slots (a hint)
#ifdef AZB_PROFILE
    uint32_t *run, *wait, *t0;  // 16-cycle units: cycles advancing the tree, cycles between hand-over and pick-up, time of the hand-over
#endif
};
__device__ __forceinline__ uint32_t as_lds_volatile(const uint32_t *p) { return *reinterpret_cast<const volatile uint32_t *>(p); }
__device__ __forceinline__ void as_sts_volatile(uint32_t *p, uint32_t v) { *reinterpret_cast<volatile uint32_t *>(p) = v; }

template <int DEPTH, bool COUNT, bool PUCT>
__device__ void async_tree_worker(const AzbLayout &L, const AzbAsyncParams &P, const uint32_t tree_cta,
                                  const uint32_t n_tree_ctas, uint32_t *smem, const uint32_t n_thr) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t FULL = 0xffffffffu;
    AzbAsyncState *st = P.st;
    uint8_t *lut = reinterpret_cast<uint8_t *>(smem + (size_t)P.tree_warps * P.smem_words_per_warp);
    // n_thr = the threads of the CTA that are here (the barrier counts them): all 1024, the first AS_WIDE_TREE_WARPS warps
    // for N >= 47, the first SH_TREE_WARPS warps in the shared-SM form
    tree_tables_fill(L, lut, threadIdx.x, n_thr);
    // this CTA's trees: a contiguous block of the batch, tree0 .. tree0 + n_local - 1 (<= P.tab_slots; the first B mod n CTAs
    // own one tree more)
    const uint32_t q_trees = L.B / n_tree_ctas, r_trees = L.B % n_tree_ctas;
    const uint32_t n_local = q_trees + (tree_cta < r_trees ? 1u : 0u), tree0 = tree_cta * q_trees + min(tree_cta, r_trees);
    AsTreeTable T;
    T.state = reinterpret_cast<uint32_t *>(lut + azb_tables_bytes(L.A, L.N, L.W));
    T.sub = T.state + P.tab_slots;
    T.steps = T.sub + P.tab_slots;
    T.ctl = T.steps + P.tab_slots;
#ifdef AZB_PROFILE
    T.run = T.ctl + 16;
    T.wait = T.run + P.tab_slots;
    T.t0 = T.wait + P.tab_slots;
#endif
    for (uint32_t i = threadIdx.x; i < P.tab_slots; i += n_thr) {
        T.state[i] = i < n_local ? 0u : 2u;
        T.sub[i] = 0u;
        T.steps[i] = 0u;
#ifdef AZB_PROFILE
        T.run[i] = T.wait[i] = T.t0[i] = 0u;
#endif
    }
    if (threadIdx.x < 16) T.ctl[threadIdx.x] = threadIdx.x == 4 ? n_local : 0u;  // [4]: runnable slots (a hint)
    as_named_bar(3, n_thr);
    if ((uint32_t)warp >= P.tree_warps) return;
    uint32_t *base = smem + (size_t)warp * P.smem_words_per_warp;
    WarpCtx cx;
    cx.full_count = COUNT;
    ctx_bind_smem(L, cx, base, lut, lane);
    cx.ct[lane] = 0u;
    __syncwarp();

    uint32_t my_rows = 0;  // rows this warp has handed to the model (lane 0)
    const long long t_k0 = AS_CLK();
    (void)t_k0;
    // start time for the watchdog: parked in two free words of the warp's counter block (only the idle path reads it)
    if (lane == 0) *reinterpret_cast<unsigned long long *>(cx.ct + 28) = as_now();
    __syncwarp();
    uint32_t idle = 0, naps = 0;
    const uint32_t ring_rows = P.NT * AS_TILE;
    // A warp for every tree (P.steal == 0): lane k keeps the bookkeeping of the warp's k-th own slot in registers and the
    // table is not used — a waiting warp's wake-up is one flag load, which matters: twenty idle warps per SM that run a
    // hundred instructions per microsecond each slow the walking ones by 10 % (4096 roots: 101 against 91 us per step).
    const uint32_t my_slot = (uint32_t)warp + (uint32_t)lane * P.tree_warps;
    uint32_t my_state = my_slot < n_local ? 0u : 2u;  // 0 runnable, 1 waiting for priors, 2 done
    uint32_t my_sub = 0, my_steps = 0;
    for (;;) {
        int pick;
        if (!P.steal) {
            if (my_state == 1u && as_ld_volatile(P.h_flag + tree0 + my_slot) >= my_sub) my_state = 0u;
            const uint32_t runnable = __ballot_sync(FULL, my_state == 0u);
            if (__ballot_sync(FULL, my_state != 2u) == 0u) break;
            if (runnable == 0u) {
                // every tree of this warp waits for its priors.  The round trip is tens of microseconds, so the first sleeps
                // after a walk are long and only then does the warp poll every microsecond
                __nanosleep(naps < AS_NAP_COUNT ? AS_NAP_LONG_NS : AS_NAP_SHORT_NS);
                ++naps;
                if ((++idle & 31u) == 0u) {
                    if (as_ld_volatile(&st->abort)) break;
                    if ((idle & 2047u) == 0u && as_now() - *reinterpret_cast<const unsigned long long *>(cx.ct + 28) > P.timeout_ns)
                        atomicExch(&st->abort, 1u);
                }
                continue;
            }
            // among this warp's runnable trees take the one that is furthest behind: the run ends when its slowest tree does
            const uint32_t behind = __reduce_min_sync(FULL, my_state == 0u ? my_steps : 0xffffffffu);
            const int k = __ffs(__ballot_sync(FULL, my_state == 0u && my_steps == behind)) - 1;
            pick = warp + k * (int)P.tree_warps;
            naps = 0;
            // the relaxed poll saw this tree's flag: one acquire load of it orders the prior row (read in add_actions) behind it
            if (__shfl_sync(FULL, my_sub, k) != 0u) (void)as_ld_acquire(P.h_flag + tree0 + (uint32_t)pick);
        } else {
            // ---- a runnable slot: first among this warp's HOME slots (i = warp mod tree_warps: disjoint between warps, so
            // a loaded CTA behaves like static ownership and nobody fights over a slot), the one that is furthest behind —
            // the run ends when its slowest tree does
            pick = -1;
            uint32_t behind = 0xffffffffu;
            for (uint32_t b0 = (uint32_t)warp; b0 < n_local; b0 += 32u * P.tree_warps) {
                const uint32_t i = b0 + (uint32_t)lane * P.tree_warps;
                const uint32_t st_i = i < n_local ? as_lds_volatile(T.state + i) : 2u;
                const uint32_t key = st_i == 0u ? as_lds_volatile(T.steps + i) : 0xffffffffu;
                const uint32_t m = __reduce_min_sync(FULL, key);
                if (m < behind) {
                    behind = m;
                    pick = (int)(b0 + (uint32_t)(__ffs(__ballot_sync(FULL, key == m)) - 1) * P.tree_warps);
                }
            }
            // ---- none at home: take over somebody else's (the counter of runnable slots is a hint that saves the scan)
            if (pick < 0 && (int)as_lds_volatile(T.ctl + 4) > 0) {
                const uint32_t n_chunks = (n_local + 31u) / 32u;
                for (uint32_t c = 0; c < n_chunks && pick < 0; ++c) {
                    const uint32_t i = ((c + (uint32_t)warp) % n_chunks) * 32u + lane;
                    const uint32_t ok = __ballot_sync(FULL, i < n_local && as_lds_volatile(T.state + i) == 0u);
                    if (ok) pick = (int)(i - lane) + __ffs(ok) - 1;
                }
            }
            if (pick < 0) {
                if (as_lds_volatile(T.ctl + 0) >= n_local) break;  // every tree of this CTA has finished the launch
                // ---- nothing runnable: look at the answer flags of waiting slots
                uint32_t found = 0;
                // more trees than warps: ONE warp at a time sweeps ALL waiting slots of the CTA (32 flags per ld.volatile
                // round trip), at most once per AS_SWEEP_GAP cycles; the others nap and rescan shared memory only
                uint32_t got = 0;
                if (lane == 0 && (uint32_t)clock64() - as_lds_volatile(T.ctl + 3) >= AS_SWEEP_GAP)
                    got = atomicCAS(T.ctl + 1, 0u, 1u) == 0u ? 1u : 0u;
                got = __shfl_sync(FULL, got, 0);
                if (got) {
                    for (uint32_t b0 = 0; b0 < n_local; b0 += 32) {
                        const uint32_t i = b0 + lane;
                        const bool ready = i < n_local && as_lds_volatile(T.state + i) == 1u &&
                                           as_ld_volatile(P.h_flag + tree0 + i) >= as_lds_volatile(T.sub + i);
                        const uint32_t rb = __ballot_sync(FULL, ready);
                        if (rb) {
                            // acquire side of the model CTA's (fence, atomicAdd): the prior rows of these trees are read after
                            // it (ONE acquire load per answered tree, as before — not per poll: it invalidates the SM's L1)
                            if (ready) {
                                (void)as_ld_acquire(P.h_flag + tree0 + i);
                                as_sts_volatile(T.state + i, 0u);
                            }
                            found += __popc(rb);
                        }
                    }
                    __threadfence_block();
                    __syncwarp();
                    if (lane == 0) {
                        if (found) atomicAdd(T.ctl + 4, found);
                        as_sts_volatile(T.ctl + 3, (uint32_t)clock64());
                        as_sts_volatile(T.ctl + 1, 0u);
                    }
                }
                if (found) {
                    idle = 0;
                    continue;
                }
                // Every wake-up costs issue slots next to the walking warps, and an answer is tens of microseconds away.  With
                // take-overs the CTA's idle warps wake at different times, so long naps still bring a sweep round every
                // microsecond or so; a warp that polls for itself sleeps long at first and then polls every microsecond.
                __nanosleep(AS_NAP_LONG_NS);
                if ((++idle & 7u) == 0u) {
                    if (as_ld_volatile(&st->abort)) break;
                    if ((idle & 511u) == 0u && as_now() - *reinterpret_cast<const unsigned long long *>(cx.ct + 28) > P.timeout_ns)
                        atomicExch(&st->abort, 1u);
                }
                continue;
            }
            // ---- claim it
            uint32_t ok = 0;
            if (lane == 0) ok = atomicCAS(T.state + pick, 0u, 3u) == 0u ? 1u : 0u;
            if (!__shfl_sync(FULL, ok, 0)) continue;
            if (lane == 0) atomicSub(T.ctl + 4, 1u);
            __threadfence_block();  // (behind the sweeper's store of the state)
            idle = 0;
        }
        const uint32_t tree = tree0 + (uint32_t)pick;
        const long long t_run0 = AS_CLK();
        (void)t_run0;
#ifdef AZB_PROFILE
        // pick-up latency: from the model raising the answer flag (its %globaltimer) to this warp starting the step
        if (lane == 0 && P.dbg && tree < 65536u) {
            const unsigned long long tf = *reinterpret_cast<volatile unsigned long long *>(g_flag_time + tree);
            if (tf) {
                const unsigned long long now = as_now(), dt = now > tf ? now - tf : 0ull;
                atomicAdd(P.dbg + 24, dt);
                atomicMax(P.dbg + 25, dt);
                atomicAdd(P.dbg + 26, 1ull);
                *reinterpret_cast<volatile unsigned long long *>(g_flag_time + tree) = 0ull;
            }
        }
#endif
#ifdef AZB_PROFILE
        if (lane == 0 && T.t0[pick]) T.wait[pick] += (uint32_t)(t_run0 >> 4) - T.t0[pick];
#endif
        // ---- one step of `tree` (the body of azb_tree_kernel, minus the batch barrier)
        ctx_bind_tree(L, cx, tree);
        uint32_t *gwk = L.walker + (size_t)tree * L.WS;
#pragma unroll 4
        for (uint32_t i = lane; i < L.WS; i += 32) cx.wk[i] = gwk[i];
        __syncwarp();
        if (cx.wk[WK_FLAGS] & 1u) tree_add_actions<DEPTH == 5>(L, cx, tree);
        // A new node needs priors: its state vector goes to the next ring row — or, on the last step of this launch, to
        // the tree's own row (the host runs one batched forward over those).  Called from inside the walk as soon as
        // the new node is known to be non-terminal, so the model's round trip overlaps the cost evaluation and the insert.
        bool submitted = false, last = false, in_walk = true;
        auto submit = [&](WarpCtx &c) {
            // inside the walk the step that owns this row is still open: WK_STEP advances when it completes
            last = c.wk[WK_STEP] + (in_walk ? 1u : 0u) >= P.target_step;
            uint32_t slot = 0;
            if (lane == 0) slot = atomicAdd(&st->row_tail, 1u);
            slot = __shfl_sync(FULL, slot, 0);
            // never lap a tile the workers have not retired yet (the ring is sized so that this does not spin)
            const uint32_t q = slot / AS_TILE;
            while (as_ld_volatile(P.tile_retired + (q % P.NT)) < q / P.NT && !as_ld_volatile(&st->abort)) __nanosleep(100);
            if (q >= P.NT) (void)as_ld_acquire(P.tile_retired + (q % P.NT));  // the row is overwritten after this
            const uint32_t pos = slot % ring_rows;
            tree_pack<true>(L, c, tree, P.ring + (size_t)pos * P.ring_ld);
            // the row of the launch's last step is answered in here like every other (the tree does not wait for it: its
            // priors are in place when the next launch begins); it also goes to the tree's own slot, where
            // azb_get_state_vecs and the host-model calls look for it
            if (last) tree_pack<true>(L, c, tree, nullptr);
            if (lane == 0) P.slot_tree[pos] = tree;
            // publish: every lane's part of the row crosses to the async proxy (fence.proxy.async carries a GPU-scope
            // MEMBAR), the warp barrier orders the lanes' stores before lane 0's RELEASE increment of the tile counter.
            // Not __threadfence(): that is MEMBAR.SC + CCTL.IVALL — an invalidation of the SM's whole L1, which the 32
            // walkers of the SM live on, for a fence that only has to release
            as_fence_proxy_async();
            __syncwarp();
            if (lane == 0) as_red_release_add(P.tile_count + ((slot / AS_TILE) % P.NT), 1u);
            submitted = true;
        };
        if (cx.err == 0 && cx.wk[WK_STEP] < P.target_step && !(cx.wk[WK_FLAGS] & 1u)) {
            // Early hand-over pays where a tree's own chain (walk -> model -> walk) is the bound, i.e. while there is a
            // warp for every tree; with several trees per warp (P.steal) it only lengthens the hot loop (32 768 roots:
            // -11 %), so those launches take the instantiation that submits after the walk.
            if (!P.steal)
                tree_rollout<DEPTH, PUCT>(L, cx, tree, 0u, submit);
            else
                tree_rollout<DEPTH, PUCT>(L, cx, tree, 0u);
        }
        in_walk = false;
        uint32_t new_state = 0u;
        const bool pending = (cx.wk[WK_FLAGS] & 1u) != 0u, at_target = cx.wk[WK_STEP] >= P.target_step;
        if (cx.err) {
            new_state = 2u;
        } else {
            if (pending && !submitted) submit(cx);
            if (submitted && !last)
                new_state = 1u;
            else if (at_target)
                new_state = 2u;
        }
        __syncwarp();
        const uint32_t live_words = WK_HDR + L.PW + 2 * L.W;
#pragma unroll 1
        for (uint32_t i = lane; i < live_words; i += 32) gwk[i] = cx.wk[i];
        __syncwarp();
        if (!P.steal) {
            if (my_slot == (uint32_t)pick) {
                my_state = new_state;
                if (submitted) my_sub += 1u;
                my_steps += 1u;
            }
            if (lane == 0) {
                if (submitted) my_rows += 1u;
#ifdef AZB_PROFILE
                T.sub[pick] = T.sub[pick] + (submitted ? 1u : 0u);
                T.steps[pick] += 1u;
                const long long t_end = AS_CLK();
                T.run[pick] += (uint32_t)((t_end - t_run0) >> 4);
                T.t0[pick] = (uint32_t)(t_end >> 4) | 1u;
#endif
                if (new_state == 2u) {
                    __threadfence();
                    atomicAdd(&st->done_trees, 1u);
                }
            }
        } else if (lane == 0) {
            // the next warp to advance this tree reads its walker block and arena through this SM's L1: CTA scope is enough
            if (submitted) {
                T.sub[pick] += 1u;
                my_rows += 1u;
            }
            T.steps[pick] += 1u;
#ifdef AZB_PROFILE
            const long long t_end = AS_CLK();
            T.run[pick] += (uint32_t)((t_end - t_run0) >> 4);
            T.t0[pick] = (uint32_t)(t_end >> 4) | 1u;
#endif
            __threadfence_block();
            as_sts_volatile(T.state + pick, new_state);
            if (new_state == 0u) atomicAdd(T.ctl + 4, 1u);
            if (new_state == 2u) {
                atomicAdd(T.ctl + 0, 1u);
                __threadfence();
                atomicAdd(&st->done_trees, 1u);
            }
        }
        if (cx.err) {
            if (lane == 0) {
                if (atomicCAS(&L.g->err, 0u, cx.err) == 0u) {
                    L.g->err_tree = tree;
                    L.g->err_step = cx.wk[WK_STEP];
                }
                atomicExch(&st->abort, 2u);
            }
            break;
        }
        __syncwarp();
    }
    if (lane < 16) {
        const uint32_t v = (COUNT || lane == CT_INS || lane == CT_LIVE || lane == CT_NOOP) ? cx.ct[lane] : 0u;
        if (v) atomicAdd(&L.g->counters.v[lane], (unsigned long long)v);
    }
#ifdef AZB_PROFILE
    if (lane >= 16) {  // per-phase lane-0 cycles of this warp's walks (tools/phase_probe.py)
        const uint32_t v = cx.ct[lane];
        if (v) atomicAdd(&L.g->prof[lane - 16], (unsigned long long)v);
    }
    // per tree: K-cycles walking, K-cycles waiting for priors, advances, rows — written by the last warp to leave the CTA
    __syncwarp();
    uint32_t left = 0;
    if (lane == 0) left = atomicAdd(T.ctl + 2, 1u) + 1u;
    left = __shfl_sync(FULL, left, 0);
    if (left == P.tree_warps) {
        __threadfence_block();
        for (uint32_t i = lane; i < n_local; i += 32) {
            const uint32_t tree = tree0 + i;
            const unsigned long long run = (unsigned long long)T.run[i] << 4, wait = (unsigned long long)T.wait[i] << 4;
            if (tree < 65536u) g_tree_prof[tree] = make_uint4((uint32_t)(run >> 10), (uint32_t)(wait >> 10), T.steps[i], T.sub[i]);
            if (P.dbg) {
                atomicAdd(P.dbg + 16, run);
                atomicMax(P.dbg + 17, run);
                atomicAdd(P.dbg + 19, wait);
                atomicMax(P.dbg + 20, wait);
                atomicMax(P.dbg + 21, wait + run);
            }
        }
        if (P.dbg && tree_cta == 0 && lane == 0) P.dbg[18] = (unsigned long long)(AS_CLK() - t_k0);
    }
#endif
    if (lane == 0 && my_rows) atomicAdd(&st->rows_real, my_rows);
}

template <int DEPTH, bool COUNT, bool PUCT = false>  // PUCT: azb_config.selection == AZB_SELECT_PUCT
__global__ void __launch_bounds__(AS_THREADS, 1)
    azb_async_kernel(const AzbLayout L, const AzbAsyncParams P, const __grid_constant__ AzbAsyncMaps M) {
    extern __shared__ __align__(1024) uint8_t as_smem[];
    __shared__ __align__(8) AsWorkerShared s_worker;
    __shared__ uint32_t s_role, s_idx;
    // the first CTA to arrive on each of n_workers SMs becomes that SM's model CTA; every other CTA walks trees.  The
    // launch is cooperative with one CTA per SM, so every role is resident from the start.
    if (threadIdx.x == 0 && !P.shared_sm) {
        uint32_t smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        uint32_t role = 0, idx = 0;
        if (atomicCAS(&P.st->sm_flag[smid & 1023u], 0u, 1u) == 0u) {
            const uint32_t m = atomicAdd(&P.st->mlp_claims, 1u);
            if (m < P.n_workers) {
                role = 1;
                idx = m;
            }
        }
        if (!role) idx = atomicAdd(&P.st->tree_claims, 1u);
        s_role = role;
        s_idx = idx;
    }
    __syncthreads();
    // one call site for the tree role of both forms (a second one turns the walker into a called function with spills)
    uint32_t tree_cta = s_idx, n_tree_ctas = gridDim.x - P.n_workers, n_thr = DEPTH == 5 ? AS_WIDE_TREE_WARPS * 32u : (uint32_t)AS_THREADS;
    if (P.shared_sm) {
        // shared-SM form: every CTA walks trees; its last warpgroup is one member of a model group (CTAs beyond the last
        // whole group have no model role)
        if constexpr (DEPTH != 5) {
            if ((threadIdx.x >> 5) >= SH_TREE_WARPS) {
                const size_t tree_bytes = (size_t)SH_TREE_WARPS * P.smem_words_per_warp * 4 + azb_tables_bytes(L.A, L.N, L.W) + as_table_bytes(P.tab_slots);
                uint8_t *smem = (uint8_t *)(((uintptr_t)(as_smem + tree_bytes) + 1023) & ~(uintptr_t)1023);
                if (blockIdx.x < (gridDim.x / P.group) * P.group) shared_model_warpgroup(L, P, M, blockIdx.x, smem, s_worker);
                return;
            }
            tree_cta = blockIdx.x;
            n_tree_ctas = gridDim.x;
            n_thr = SH_TREE_WARPS * 32u;
        } else {
            return;
        }
    } else if (s_role) {
        uint8_t *smem = (uint8_t *)(((uintptr_t)as_smem + 1023) & ~(uintptr_t)1023);
        async_model_cta(L, P, M, s_idx, smem, s_worker);
        return;
    } else {
        if constexpr (DEPTH == 5) {
            // N >= 47: a tree warp needs 6-10 KB of shared memory, so at most 16 of them fit (the host caps tree_warps
            // at AS_WIDE_TREE_WARPS).  Warpgroups 4-7 hand their registers over and leave; the walkers grow to 104
            // registers (128 x (4 x 104 + 4 x 24) = 65 536), which is what the Sturm-section stack program wants.
            if ((threadIdx.x >> 7) >= AS_WIDE_TREE_WARPS / 4) {
                asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(AS_REGS_IDLE));
                return;
            }
            asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(AS_REGS_WIDE_TREE));
        }
    }
    async_tree_worker<DEPTH, COUNT, PUCT>(L, P, tree_cta, n_tree_ctas, reinterpret_cast<uint32_t *>(as_smem), n_thr);
}
