/*
 * azb.h — C ABI of azdopt-b200: the B200-native replacement for ONE hot path of
 * ariasanovsky/azdopt, the batched search step of the c21 example
 * (`NablaOptimizer::par_roll_out_episodes` over `ROTModifyParentsOnce`).
 *
 * The reference has no FFI: its boundary is Rust traits plus the public methods
 * of `NablaOptimizer` (az-discrete-opt/src/nabla/optimizer/mod.rs:29-364).  Each
 * entry point below names the reference item it replaces (file:line relative to
 * the reference repository).  The space's four closures and `n_as_tol` are Rust
 * fn pointers / closures (graph-state/src/rooted_tree/space.rs:13-19,
 * graph-state/examples/04-c21-tree.rs:96-105,136-138); they cannot cross a C ABI,
 * so they travel as data in `azb_config`.
 *
 * Conventions: every function returns an `int` status (AZB_OK = 0); nothing
 * aborts.  Buffers are caller-owned host memory unless a name ends in `_dev`.
 * A handle is bound to one CUDA device and is NOT thread-safe (like the
 * reference's `&mut self`).  Row-major everywhere.
 *
 *   A  = ACTION_DIM = (N-1)(N-2)/2 - 1     (rooted_tree/space.rs:48)
 *   S  = STATE_DIM  = 2A                    (rooted_tree/space.rs:46)
 *   W  = ceil(A/32) words of an action bit mask (bit a of word a/32)
 */
#ifndef AZB_H
#define AZB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AZB_VERSION 100
#define AZB_NONE 0xFFFFFFFFu
#define AZB_MAX_VERTICES 64
#define AZB_MAX_TOL 8
#define AZB_ASYNC_AUTO 0xFFFFFFFFu  /* azb_config.async_workers: let the library pick the model SMs from the root count */
#define AZB_ASYNC_SHARED 0xFFFFFFFEu /* azb_config.async_workers: no SM is taken from the trees — every SM walks trees with 28 warps and
                                       its last warpgroup is one of 8 members of a model group (N <= 46) */

enum {
    AZB_OK = 0,
    AZB_ERR_INVALID = 1,       /* bad argument / bad config */
    AZB_ERR_CUDA = 2,          /* a CUDA call failed; see azb_last_error */
    AZB_ERR_CAPACITY = 3,      /* a per-tree arena (nodes, predictions, parents, hash, frontier) overflowed */
    AZB_ERR_NAN = 4,           /* NaN reached a comparison (the reference panics: next_action.rs:51,74,85) */
    AZB_ERR_LAMBDA = 5,        /* lambda_1 < 1.4 (the reference asserts: rooted_tree/ordered_edge.rs:79) */
    AZB_ERR_UNREACHABLE = 6,   /* inactive non-root walker (the reference's unreachable!(): tree/mod.rs:227) */
    AZB_ERR_STATE = 7          /* call order violated (e.g. step before init_trees) */
};

/* where h_theta comes from in the fused device loop */
enum {
    AZB_PRIOR_MLP = 0,      /* the built-in MLP (replaces ActionModel::write_predictions, nabla/model/dfdx.rs:69-84) */
    AZB_PRIOR_HASH = 1,     /* counter hash of (prior_seed, global root, step, action) in [0,1): parity runs */
    AZB_PRIOR_INJECTED = 2  /* rows uploaded by azb_set_priors / azb_add_actions_host */
};

/* MLP arithmetic */
enum {
    AZB_MLP_FP32 = 0,     /* fp32 CUDA-core GEMM: what cuBLAS sgemm gives the reference */
    AZB_MLP_TC = 1,       /* tcgen05 tensor cores, bf16 weights and hidden activations, fp32 accumulate */
    AZB_MLP_TC3 = 2       /* tcgen05 tensor cores at f32 accuracy: every operand as bf16 hi + lo, three products per dot
                             product (hi.hi + hi.lo + lo.hi), fp32 accumulate — within ~1e-6 of the f32 forward the
                             reference runs (nabla/model/dfdx.rs:69-84), at about three times the tensor work */
};

/* selection rule at an active node (azb_config.selection) */
enum {
    AZB_SELECT_REFERENCE = 0, /* next_action (next_action.rs:11-26): revisit_choice under n_as_tol, else max_curiosity */
    AZB_SELECT_PUCT = 1       /* AlphaZero-style PUCT argmax; defined here, it has NO reference to be checked against */
};
/* AZB_SELECT_PUCT replaces next_action at an active node s; everything after the choice (Visited -> descend,
 * Unvisited(j) -> probe, transposition, insert, cost, cascades, n_t, c*, argmin) is unchanged and n_as_tol is not
 * consulted.  Every operation is f32, round-to-nearest, in the order written, nothing fused.  c_s = the node's c; kids
 * k in creation order with action a_k, active_k, n_k (the child's n_t) and c*_k; predictions j = 0..cnt-1 in the node's
 * prediction order with a_j, g_j = c_s - h_j and has_arc_j.
 *   1. N_s = 1 + sum_k (n_k + 1) over all kids, active or not (an exact integer; AZB_ERR_CAPACITY at 2^24);
 *      sq = sqrt((float)N_s).
 *   2. w_j = (1 - c_s) + g_j, or +0 where that is negative (the model's predicted goodness 1 - h_j, up to rounding).
 *   3. Z = sum_j w_j: each chunk of 32 predictions is summed as a warp's xor butterfly does it (lane i holds
 *      w_{32c+i} or +0 beyond cnt; for m = 16, 8, 4, 2, 1: x[i] = x[i] + x[i^m]; the chunk sum is x[0]), then the
 *      chunk sums are folded left to right starting from chunk 0's.  p_j = w_j / Z, or 1 / cnt when Z == 0.
 *   4. A prediction without an arc has n = 0, q = g_j.  One with an arc to kid k (a_k == a_j) is skipped if the kid is
 *      inactive, else n = n_k + 1, q = c_s - c*_k.
 *   5. score_j = q + ((puct_c * p_j) * sq) / (float)(1 + n).
 *   6. The first maximum of score_j in ascending j wins: Visited(k) if it has an arc, else Unvisited(j).  A NaN score
 *      is AZB_ERR_NAN; no candidate at an active node is AZB_ERR_UNREACHABLE.
 * Counters per selection: n_sel += 1, d_sel += kids, n_cur += 1, n_cand += cnt (n_visit as in the reference mode). */

typedef struct azb_config {
    uint32_t struct_size;       /* sizeof(azb_config), for ABI growth */
    uint32_t n_vertices;        /* N, 5..64                                (04-c21-tree.rs:33) */
    uint32_t n_roots;           /* B on this device                        (04-c21-tree.rs:54) */
    int32_t device;             /* CUDA ordinal */
    uint64_t first_root;        /* global index of local root 0 (sharding; feeds the hash generators) */
    float c_lower;              /* C_LOWER_BOUND = 2                       (04-c21-tree.rs:58) */
    float c_upper;              /* C_UPPER_BOUND                           (04-c21-tree.rs:59-68); 0 = derive from N */
    uint32_t n_as_tol[AZB_MAX_TOL]; /* revisit budget by depth             (04-c21-tree.rs:136-138) */
    uint32_t n_as_tol_len;
    uint32_t n_as_tol_default;
    uint32_t mlp_hidden[3];     /* 512, 1024, 512                          (04-c21-tree.rs:42-44) */
    uint32_t mlp_mode;          /* AZB_MLP_* */
    uint32_t prior_mode;        /* AZB_PRIOR_* */
    uint64_t prior_seed;
    uint32_t max_steps;         /* steps between azb_init_trees calls the arenas are sized for (800: 04-c21-tree.rs:134) */
    uint32_t cap_nodes;         /* per-tree capacities; 0 = derive from max_steps */
    uint32_t cap_preds;
    uint32_t cap_parents;
    uint32_t max_episodes;      /* 0: every launch runs each tree to the end of its step (the reference's lock step).
                                   k > 0: a tree that keeps hitting terminal nodes / transpositions yields after k
                                   episodes and finishes the step in a later launch; same results, shorter launches */
    uint32_t n_groups;          /* >1: the trees of this handle advance as that many independent groups on their own
                                   CUDA streams (needs max_episodes = 0); results are identical, launches overlap */
    uint32_t async_workers;     /* > 0 (needs AZB_PRIOR_MLP + AZB_MLP_TC): azb_step(h, n >= 2) runs as ONE persistent cooperative
                                   kernel in which trees never wait for each other — the CTAs of that many SMs become
                                   tensor-core model workers that answer state vectors in 128-row tiles as they fill, all
                                   other CTAs walk trees: a CTA owns a block of the batch's trees, each warp its own while there
                                   is a warp for every tree, any free warp any runnable tree of its CTA beyond that.  Same
                                   results as the lock step (trees are independent).  0 = lock step.  AZB_ASYNC_AUTO = the
                                   measured best layout for the root count (DESIGN.md 4.4: 20 model SMs up to 4096 roots — in
                                   pairs per tile below 4096 —, 36 beyond; 16 for N >= 47), or the lock step where the
                                   asynchronous kernel does not apply (no tensor-core model, fewer than 1024 roots,
                                   max_episodes or n_groups set); azb_get_config shows the choice.  Environment, read when the
                                   handle first runs this way: AZB_ASYNC_GROUP=g (worker SMs per tile),
                                   AZB_ASYNC_STEAL=0/1 (tree scheduling inside a CTA), AZB_ASYNC_FLUSH_NS,
                                   AZB_ASYNC_TIMEOUT_MS (watchdog floor, default 2000). */
    uint32_t selection;         /* AZB_SELECT_*; 0 = the reference's next_action */
    float puct_c;               /* c_puct of AZB_SELECT_PUCT (finite, > 0; azb_config_default: 1); unused otherwise */
    uint32_t reserved[3];
} azb_config;

typedef struct azb_counters {   /* workload counters; definitions in oracle/azb_oracle.h and DESIGN.md */
    uint64_t n_sel, d_sel, n_cur, n_cand, n_probe, n_ins, n_term, n_hit, n_arc, n_pred, n_cn, d_cn, n_reset, n_live,
        n_noop, n_visit;
} azb_counters;

typedef struct azb_improvement { /* one ArgminImprovement::Improved (optimizer/mod.rs:24-27) */
    uint32_t step;               /* step index since azb_init_trees (0-based) */
    uint32_t tree;               /* local root index */
    uint32_t node;               /* node index inside that tree */
    float eval;
} azb_improvement;

typedef struct azb_handle azb_handle;

/* ---- library ---- */
int azb_version(void);
const char *azb_strerror(int code);
/* last CUDA / validation message of this handle (never NULL) */
const char *azb_last_error(const azb_handle *h);

/* ---- construction: NablaOptimizer::par_new (optimizer/mod.rs:39-118) is create + set_roots + init_trees ---- */
int azb_config_default(azb_config *cfg, uint32_t n_vertices, uint32_t n_roots);
int azb_create(const azb_config *cfg, azb_handle **out);
int azb_destroy(azb_handle *h);
int azb_get_config(const azb_handle *h, azb_config *out);   /* with derived fields filled in */

/* synthetic roots of SURVEY.md §8d, the example's distribution (04-c21-tree.rs:85,108-112;
 * rooted_tree/mod.rs:14-20; modify_parent_once.rs:14-25).  Host-only helper. */
int azb_generate_roots(uint64_t seed, uint64_t first_root, uint32_t count, uint32_t n_vertices, uint32_t k_min,
                       uint32_t k_max, uint8_t *parents /*[count*N]*/, uint32_t *permitted /*[count*W]*/);
/* roots: Vec<Space::State> (optimizer/mod.rs:9,61) */
int azb_set_roots(azb_handle *h, const uint8_t *parents /*[B*N]*/, const uint32_t *permitted /*[B*W]*/);
int azb_get_roots(azb_handle *h, uint8_t *parents, uint32_t *permitted);

/* ---- the model: NablaModel (nabla/model/mod.rs:4-8), ActionModel (nabla/model/dfdx.rs:18-53) ---- */
/* parameter block, dfdx order: for each of the 4 Linear layers weight[out][in] then bias[out], f32 */
size_t azb_mlp_num_params(const azb_handle *h);
int azb_mlp_init(azb_handle *h, uint64_t seed);             /* U(-1/sqrt(fan_in), 1/sqrt(fan_in)) */
int azb_mlp_set_params(azb_handle *h, const float *params);
int azb_mlp_get_params(azb_handle *h, float *params);
/* NablaModel::write_predictions (nabla/model/dfdx.rs:69-84): host [rows*S] -> host [rows*A]; rows <= B */
int azb_model_write_predictions(azb_handle *h, const float *states, float *predictions, uint32_t rows);

/* ---- tail of par_new / par_reset_trees (optimizer/mod.rs:62-101, 347-359): root costs, root vectors, one
 *      prior evaluation, root node + root predictions, argmin over roots.  In AZB_PRIOR_INJECTED mode the
 *      priors come from the last azb_set_priors. ---- */
int azb_set_priors(azb_handle *h, const float *priors /*[B*A]*/);
int azb_init_trees(azb_handle *h);

/* ---- the hot path: NablaOptimizer::par_roll_out_episodes (optimizer/mod.rs:121-191), n_steps times, fused on
 *      the device (no host round trip per step).  The reference reports an improvement per step
 *      (04-c21-tree.rs:143-148); `improvements` receives up to `cap` of them, `*n_improved` the total. ---- */
int azb_step(azb_handle *h, uint32_t n_steps, azb_improvement *improvements, uint32_t cap, uint32_t *n_improved);
/* enqueue only (no wait, no read-back; needs max_episodes = 0): lets several handles share one GPU concurrently.
 * azb_step(h, 0, ...) or any reading call completes the work and reports errors. */
int azb_step_enqueue(azb_handle *h, uint32_t n_steps);
/* par_roll_out_episodes' per-step return value (ArgminImprovement, optimizer/mod.rs:24-27,121-191) for steps enqueued
 * with azb_step_enqueue, one step per call in order, as soon as EVERY tree has finished that step — later steps keep
 * running (with async_workers > 0 the trees run ahead of the caller, so a loop of one call per step advances at the
 * speed of the fused loop).  *improved = 1 and *out = the record (may be null) when the step lowered the best cost
 * (the reference's rule: first minimum over trees, strictly below the running best, optimizer/mod.rs:194-246).
 * azb_step(h, 0, ...) after the last step completes the batch; it logs exactly the improvements reported here.
 * AZB_ERR_STATE when no enqueued step is left to report. */
int azb_step_poll(azb_handle *h, azb_improvement *out, int *improved);
/* same as azb_step, timed with CUDA events on the library's stream; *ms = device time of the n_steps */
int azb_step_timed(azb_handle *h, uint32_t n_steps, float *ms, uint32_t *n_improved);

/* same again, with an event between the kernels of every step: *tree_ms = summed device time of the search kernel
 * launches, *mlp_ms = of the model forward launches (roofline.achieved in bench.py divides by the former) */
int azb_step_profile(azb_handle *h, uint32_t n_steps, float *tree_ms, float *mlp_ms);

/* the same step split at the NablaModel boundary, for a host-side model (host buffers, copies included):
 *   rollout_host      = first parallel region (optimizer/mod.rs:159-174): walks + write_vec, D2H of state_vecs
 *   add_actions_host  = second region + par_update_argmmim_data (optimizer/mod.rs:177-190): H2D of h_theta */
int azb_rollout_host(azb_handle *h, float *state_vecs /*[B*S]*/);
int azb_add_actions_host(azb_handle *h, const float *h_theta /*[B*A]*/, int *improved);

/* ---- results ---- */
/* ArgminData{state, cost, eval} (log.rs:1-11; optimizer/mod.rs:361-363) */
int azb_get_argmin(azb_handle *h, uint8_t *parents /*[N]*/, uint32_t *permitted /*[W]*/, double *lambda1,
                   uint32_t *mu, float *eval);
/* The state of one node: its tree's root with the node's action set replayed in ascending order — the rebuild
 * par_update_argmmim_data does for the winning node (optimizer/mod.rs:224-239).  Does not wait for enqueued steps, so
 * an azb_step_poll record (tree, node) can be turned into ArgminData while later steps still run. */
int azb_get_node_state(azb_handle *h, uint32_t tree, uint32_t node, uint8_t *parents /*[N]*/, uint32_t *permitted /*[W]*/);
/* ---- extension (no reference item): canonical codes of trees and the k best isomorphism classes the search has
 *      evaluated.
 * The code of a tree T on N vertices (a parent array: edges {v, parents[v]} for v = 1..N-1, parents[v] < v) ignores the
 * root and the labels.  The centres are the vertices of minimum eccentricity (one or two).  For the tree rooted at r,
 * enc(v) = 1 . enc(c_1) . ... . enc(c_d) . 0 with the children ordered so that enc(c_1) >= ... >= enc(c_d)
 * lexicographically (1 > 0); every enc is a prime Dyck word, so none is a proper prefix of another and the first
 * differing bit decides.  code(T) = the maximum over the centres r of enc(r), exactly 2N bits, stored in two uint64_t
 * words: string bit i is bit 63 - i % 64 of word i / 64, unused bits 0, so comparing (word0, word1) as unsigned integers
 * compares the strings.  Two trees on N vertices have equal codes <=> they are isomorphic.
 * azb_tree_codes: the codes of M trees of the handle's N (parents[v] < v, as azb_eval_costs checks; AZB_ERR_INVALID
 * names the first tree that breaks it).  ms (may be NULL) = device time of the kernel alone; codes may be NULL. */
int azb_tree_codes(azb_handle *h, const uint8_t *parents /*[M*N]*/, uint32_t m, uint64_t *codes /*[M*2]*/, float *ms);
/* azb_best_trees: the k best isomorphism classes among ALL nodes (0..n_nodes-1) of ALL trees of the handle, at call time.
 * A class is one isomorphism class (one code) among the states of all nodes of all trees.  The value of a class is the
 * minimum c over its member nodes (at N >= 23 the cost is a labelling-dependent sectioning program, so isomorphic trees
 * may differ in the last bit of c: equal codes do not mean equal c).  The representative is, among the members whose c
 * equals the class value, the one with the smallest (first_root + tree, node), so a sharded run picks what one unsharded
 * handle would.  Classes are sorted ascending by (value, code) and the first min(k, #classes) are returned; *n_out is
 * that count.  Per class: eval = the class value; tree, node = the representative's local indices; parents, permitted =
 * exactly what azb_get_node_state(tree, node) returns; lambda1, mu = the cost kernel on the representative's parents, as
 * azb_get_argmin does (eval equals that node's stored c bits).  Any output pointer may be NULL.  The call is enqueued on
 * the library stream behind any enqueued steps and reports their errors.  AZB_ERR_STATE before azb_init_trees;
 * AZB_ERR_INVALID for k == 0 or k > 65536, and for parent arrays azb_eval_costs would reject, naming the first bad tree.
 * The call changes nothing: no tree, walker, counter, argmin or RNG state. */
int azb_best_trees(azb_handle *h, uint32_t k, uint32_t *n_out, float *eval /*[k]*/, uint64_t *codes /*[k*2]*/,
                   uint32_t *tree /*[k]*/, uint32_t *node /*[k]*/, uint8_t *parents /*[k*N]*/,
                   uint32_t *permitted /*[k*W]*/, double *lambda1 /*[k]*/, uint32_t *mu /*[k]*/);
/* ---- extension (no reference item; the reference has no checkpointing): save a handle's search and training state
 *      and resume it bit for bit in a new process, on the same or another split of the roots.
 * azb_checkpoint_save works whenever the handle is at rest after azb_init_trees / azb_reset_trees (after any completed
 * azb_step, after azb_update_model, around azb_best_trees).  Like every reading call it first runs the deferred
 * add_actions of the last step; apart from that it changes nothing (no tree, walker, counter, argmin or RNG state), so
 * two saves in a row give identical bytes.  AZB_ERR_STATE before the first azb_init_trees (or after azb_set_roots),
 * while steps enqueued with azb_step_enqueue have not been completed by azb_step(h, 0, ...), and between
 * azb_rollout_host and azb_add_actions_host.  azb_checkpoint_size gives the exact number of bytes save writes;
 * AZB_ERR_INVALID when `size` is smaller.  The buffer may be pageable.
 *
 * Blob format AZB_CKPT_FORMAT, little-endian, every section a multiple of 8 bytes:
 *   header  AZB_CKPT_HEADER_WORDS uint64 words; 32-bit values sit in the low half of their word, floats as their bits:
 *     0 AZB_CKPT_MAGIC   1 AZB_CKPT_FORMAT   2 AZB_VERSION   3 blob bytes
 *     4 n_vertices  5 c_lower  6 c_upper (derived)  7..14 n_as_tol[0..7]  15 n_as_tol_len  16 n_as_tol_default
 *     17..19 mlp_hidden  20 mlp_mode  21 prior_mode  22 prior_seed  23 selection  24 puct_c
 *     25 first_root  26 n_roots (the blob's global roots are [first_root, first_root + n_roots))
 *     27 steps_done (steps since the last init/reset)  28 resets so far (keys azb_reset_trees' draws)  29 Adam step count
 *     30..34 Adam lr, beta1, beta2, eps, l2   35 flags (bit 0: model parameters set)
 *     36 running best: orderable bits of its eval (float bits u -> u | 0x80000000 if the sign bit is clear, else ~u)
 *     37 its global root  38 its node  39..77 its state: 77 uint32 words (parents packed 4 per word in 16 words, then
 *        61 permitted-mask words) two per uint64, low half first
 *     78 n_params  79/80 model section offset/bytes  81/82 tree offset table offset/bytes  83/84 tree section offset/bytes
 *     85 model section digest  86 tree offset table digest  87..94 zero  95 digest of words 0..94
 *   model   params, Adam m, Adam v: n_params float32 each (m and v are zero before the first training step), zero-padded
 *   table   uint64[n_roots + 1]: byte offset of every tree record inside the tree section; entry n_roots = its size
 *   trees   one record per root in root order, uint32 words: the walker block (WS = 80 + 2 ceil(N/4) + 3W words: state,
 *           path, bump pointers, step clock, root parents and permitted mask) | n_nodes node records of 16 words |
 *           n_nodes keys of W words | the block arena units [64, nblk) of 2 words | the overflow in-arcs [0, intop) of 2
 *           words | a zero word if the count is odd | the record's uint64 digest.  n_nodes, nblk and intop are walker
 *           words 2, 3 and 5.  Not saved: the transposition table (rebuilt on load), cascade scratch, the consumed
 *           per-step candidates, state vectors and priors (consumed by the add_actions that ran before the save), the
 *           asynchronous kernel's ring and the workload counters.
 * Digest of n uint64 words w_0..w_{n-1} (w_i = bytes 8i..8i+7 of the section, little-endian), with
 *   mix64(z): z += 0x9E3779B97F4A7C15; z = (z ^ z >> 30) * 0xBF58476D1CE4E5B9; z = (z ^ z >> 27) * 0x94D049BB133111EB;
 *             return z ^ z >> 31                                                              (all mod 2^64)
 *   digest = mix64(S ^ n),  S = sum over i of mix64(w_i ^ (i * 0x9E3779B97F4A7C15)) mod 2^64.
 * The sum makes it independent of the order in which its terms are added; it detects corruption and truncation and is
 * not a security check.  Blocks and the overflow in-arc arena keep slots reserved for arcs not added yet; their
 * bytes are whatever the arena held, so two handles holding the same trees may write different blobs, while two saves
 * of one handle write the same bytes.
 *
 * azb_checkpoint_load rebuilds the handle's whole search and training state from one or more blobs whose ranges must
 * cover the handle's [first_root, first_root + n_roots) exactly once; a blob may reach past it (its other roots are
 * ignored) or lie outside it (only its header is read).  AZB_ERR_INVALID (azb_last_error names the field), before
 * anything is written to the device: bad magic, format, version or header digest, a blob size that differs from its
 * header's, a config field that differs from the handle's (N, c_lower, c_upper, n_as_tol, mlp_hidden, mlp_mode,
 * prior_mode, prior_seed, selection, puct_c), blobs that disagree on steps_done, resets, Adam step or config, or model
 * section, overlapping ranges, a gap in the handle's range, a bad model or table digest.  AZB_ERR_CAPACITY when the
 * handle's max_steps is below steps_done.  Everything else may differ: n_roots and first_root (resharding), device,
 * async_workers, n_groups, max_episodes, max_steps and the cap_* capacities.  A tree record that fails its digest is
 * AZB_ERR_INVALID, one that does not fit the handle's capacities AZB_ERR_CAPACITY; the message names the lowest global
 * root at fault, and the handle then behaves as before its first azb_init_trees until a load succeeds or azb_set_roots +
 * azb_init_trees run.  After a successful load: the saved roots, walkers and trees; parameters, Adam m, v, step count
 * and config; the reset count; steps_done; the running best = the first minimum by (eval, global root, node) over the
 * running bests of ALL given blobs (with one blob of the same split, exactly the saved one; resharded, every shard starts
 * from the global best, so the continued run's global best equals the uninterrupted run's, while azb_comm_argmin's owner
 * and each shard's improvement log may differ).  Workload counters restart at zero: saved + continued counters equal the
 * uninterrupted run's.  A communicator is not part of the state: attach it again with azb_comm_init. */
#define AZB_CKPT_MAGIC 0x3154504B43425A41ull /* "AZBCKPT1" */
#define AZB_CKPT_FORMAT 1
#define AZB_CKPT_HEADER_WORDS 96
int azb_checkpoint_size(azb_handle *h, uint64_t *bytes);
int azb_checkpoint_save(azb_handle *h, void *buf, uint64_t size, uint64_t *written);
int azb_checkpoint_load(azb_handle *h, const void *const *blobs, const uint64_t *sizes, uint32_t n_blobs);
/* ---- extension (no reference item): every free tree on N <= 32 vertices by index, and the exact k best of any index
 *      range by the c21 cost.
 * The enumeration.  Rooted trees carry global ids, ordered by size first (the single vertex is id 0), then by rank
 * within their size s: a rooted tree of size s is its root plus the multiset of its child subtrees, written as the
 * NON-INCREASING sequence of the children's global ids (their sizes sum to s - 1), and rank orders these sequences
 * lexicographically ascending (none is a proper prefix of another: all have the same size sum).  Size s has A000081(s)
 * ids.  A free tree on N vertices is rooted at its centroid:
 *   - unicentroidal trees take the indices [0, U): a non-increasing sequence of global ids whose sizes sum to N - 1, every
 *     size <= floor((N - 1) / 2), in lexicographically ascending order; U is the number of such sequences;
 *   - for even N the bicentroidal trees follow: the unordered pair of rooted trees of size N / 2 with in-size ranks
 *     i >= j has index U + i (i + 1) / 2 + j.
 * Labels are preorder with children visited in sequence order: the root is vertex 0, then the subtree of each element of
 * the sequence in turn, each laid out the same way (its root first, with parent the vertex it hangs from).  A bicentroidal
 * tree has the root of tree i at vertex 0, tree j at vertices 1 .. N/2 (its root at 1, parent 0), then tree i's child
 * subtrees.  So parents[v] < v, vertex 0 is a centroid, and A000055(N) indices cover every isomorphism class once.
 * Unranking: with P[r][g] = the number of non-increasing sequences of ids <= g whose sizes sum to r, the sequences of sum
 * r with first element < g number P[r][g - 1]; an index is decoded one element at a time (the smallest g with P[r][g] > x,
 * then x -= P[r][g - 1], r -= size(g)).  The handle builds P (rows r = 0..N-1, 32 x 141 083 words at N = 32) and the
 * preorder arrays of all rooted trees of size <= N/2 on first use; they and the calls' scratch count in azb_device_bytes.
 * azb_free_tree_count: A000055(n) for 5 <= n <= 32, host only.
 * azb_free_trees: the parent arrays of indices [start, start + m) of the handle's N.
 * azb_exhaustive_best: every tree of [start, start + count) through the cost kernel of azb_eval_costs; the first
 * min(k, count) sorted ascending by key = (double)mu + lambda1 (one IEEE add), ties by index.  Per entry: the index, its
 * parent array (exactly azb_free_trees'), lambda1, mu and eval = the f32 c azb_eval_costs gives for it.  *n_out = the
 * number of entries, *n_below = the number of trees of the range with key < bound (bound = sqrt(N - 1) + 1, the star's
 * key, counts the counterexamples of the conjecture).  ms = device time of the whole call.  Any output pointer may be NULL.
 * Both calls: AZB_ERR_INVALID for a handle with N > 32 and for a range that is empty (count or m = 0) or reaches past
 * A000055(N); azb_exhaustive_best also for k == 0 or k > 65536 and AZB_ERR_LAMBDA as azb_eval_costs.  They work before
 * azb_init_trees, run on the library stream and change no tree, walker, counter, argmin, model or RNG state. */
int azb_free_tree_count(uint32_t n, uint64_t *count);
int azb_free_trees(azb_handle *h, uint64_t start, uint32_t m, uint8_t *parents /*[m*N]*/);
int azb_exhaustive_best(azb_handle *h, uint64_t start, uint64_t count, uint32_t k, double bound, uint32_t *n_out,
                        uint64_t *n_below, uint64_t *index /*[k]*/, uint8_t *parents /*[k*N]*/, double *lambda1 /*[k]*/,
                        uint32_t *mu /*[k]*/, float *eval /*[k]*/, float *ms);
/* ---- extension (no reference item): every tree on the handle's N (5 <= N <= 64) vertices whose c21 key is at most a
 *      bound, found without enumerating all trees.
 * The canonical labelling of an isomorphism class is the decoding of its code (azb_tree_codes): read the 2N bits from
 * the left; the first 1 is vertex 0 (the centre the code is taken at) and becomes the current vertex; each later 1 is
 * the next unused vertex, whose parent is the current vertex, and becomes the current vertex; each 0 makes the current
 * vertex's parent current (the last 0 closes vertex 0).  So vertices are numbered in preorder, children in code order,
 * and parents[v] < v.  The key of a class is (double)mu + lambda1 (one IEEE add) with lambda1 and mu what azb_eval_costs
 * gives for the canonical labelling: from N = 23 on lambda1 depends on the labelling in its last bits, and this makes it
 * a function of the class.
 * azb_trees_within: the classes on N vertices with key <= bound (bound < 0: the key of the star K1,N-1, so the star is
 * in the set and the set is the star and every tree at least as good).  *n_within = their number, *n_below = the number
 * with key < bound, and the first min(k, n_within) sorted ascending by (key, code) are returned: per entry the code (two
 * words as azb_tree_codes), the canonical parent array, and lambda1, mu, eval exactly as azb_eval_costs gives for it;
 * *n_out = the number of entries.  ms = device time of the whole call.  Any output pointer may be NULL.
 * Method (exact): a subtree's key is below its tree's (Perron-Frobenius for lambda1, and mu cannot grow), and every tree
 * on s + 1 vertices is one on s vertices plus a leaf.  The classes on s = 5 .. N - 1 vertices with key <= bound + 1e-9
 * are grown level by level from the trees on 4 vertices, one leaf at a time, and the children of the last of them with
 * key <= bound are the result; the slack covers the rounding of lambda1 (DESIGN.md §4.11).  A level's size, not
 * A000055(N), sets the cost.
 * AZB_ERR_INVALID for k == 0, k > 65536 or a NaN bound.  AZB_ERR_CAPACITY when a level would hold more than max_level
 * classes (0: as many as fit in the device's free memory, which also bounds a larger max_level); azb_last_error names the
 * level and the classes found so far, and no output is written.  AZB_ERR_LAMBDA as azb_eval_costs.  The call works
 * before azb_init_trees, runs on the library stream, changes no tree, walker, counter, argmin, model or RNG state, and
 * its scratch counts in azb_device_bytes.  It uses this handle's GPU alone, with or without a communicator;
 * azb_comm_trees_within (below) splits the same call over the communicator's ranks. */
int azb_trees_within(azb_handle *h, double bound, uint32_t k, uint64_t max_level, uint32_t *n_out, uint64_t *n_within,
                     uint64_t *n_below, uint64_t *codes /*[k*2]*/, uint8_t *parents /*[k*N]*/, double *lambda1 /*[k]*/,
                     uint32_t *mu /*[k]*/, float *eval /*[k]*/, float *ms);
/* ---- extension (no reference item): certificates of c21 keys against a bound, with directed rounding.
 * rd / ru: one IEEE binary64 operation rounded down / up, no contraction.
 * Interval inertia count JT(T, x) for a tree T (parents[v] < v) and a binary64 point x: every vertex starts with the
 * interval [-x, -x].  For v = n-1 down to 1 the interval [l_v, u_v] of v is final when it is reached; if it contains 0
 * (or has a NaN end) the result is undecided, otherwise r_lo = rd(1/u_v), r_hi = ru(1/l_v), and then for p = parents[v]
 * l_p = rd(l_p - r_hi), u_p = ru(u_p - r_lo).  Vertex 0 is undecided if its interval contains 0.  Otherwise the count is
 * the number of v with l_v > 0.  Every exact Jacobs-Trevisan value lies in its interval and none is 0, so a decided
 * count is the number of eigenvalues of A above x: 0 proves lambda1 < x, >= 1 proves lambda1 > x.
 * mu: greedy leaf matching, v = n-1 down to 1 is matched with parents[v] when both are unmatched (exact for trees).
 * Enclosure of lambda1 from c = the cost kernel's lambda1 (a starting point only; nothing relies on it being right):
 * with d_j = 4^j ulp(c), j = 0 .. 11, lambda1_lo = rd(c - d_j) for the first j at which JT is decided with a count >= 1,
 * lambda1_hi = ru(c + d_j) for the first j at which JT is decided with a count of 0; both NaN if either is not found
 * (or c is outside [1, 2^1000)).  So lambda1_lo < lambda1 < lambda1_hi.
 * The bound as a real number: a bound >= 0 is that binary64 value; a bound < 0 is sqrt(N - 1) + 1 exactly (the star's
 * true key, not its rounded value).  t = bound - mu is enclosed in [t_lo, t_hi]: t_lo = rd(b_lo - mu), t_hi = ru(b_hi -
 * mu) with b_lo = b_hi = bound, or for the default bound b_lo = rd(rd_sqrt(N - 1) + 1), b_hi = ru(ru_sqrt(N - 1) + 1).
 * Verdict (int8): 0 = key == bound proven, only for a star (mu = 1) against the default bound or against a bound >= 0
 * with (bound - 1)^2 = N - 1; else -1 = key < bound proven (lambda1_hi <= t_lo, or JT at t_lo decided with a count of
 * 0); else +1 = key > bound proven (lambda1_lo >= t_hi, or JT at t_hi decided with a count >= 1); else 2 = open (any
 * other exact tie, or intervals too wide to decide).  Never a guess.
 * azb_certify_keys: for m trees on the handle's N vertices, the cost kernel of azb_eval_costs and then the certificate
 * of each: lambda1_lo, lambda1_hi, the greedy mu and the verdict against bound.  ms = device time of the call.  Any
 * output pointer may be NULL.  AZB_ERR_INVALID as azb_eval_costs (azb_last_error names the first bad tree) and for a
 * NaN bound; AZB_ERR_LAMBDA as azb_eval_costs.  Works before azb_init_trees, runs on the library stream, changes no
 * state, and its scratch counts in azb_device_bytes. */
int azb_certify_keys(azb_handle *h, const uint8_t *parents /*[m*N]*/, uint32_t m, double bound, double *lambda1_lo /*[m]*/,
                     double *lambda1_hi /*[m]*/, uint32_t *mu /*[m]*/, int8_t *verdict /*[m]*/, float *ms);
/* azb_trees_within_proof: azb_trees_within with the certificate above run on its way; every output but proof is bit for
 * bit what azb_trees_within gives (ms includes the certificates).  proof[5]:
 *   [0] result classes proven below the bound, [1] proven equal to it (the star), [2] proven above it (the binary64
 *   filter let them in), [3] open; these sum to n_within and are counted once per class, after the last level's merge;
 *   [4] classes dropped at any level (key not <= the level's threshold) for which key > bound was not proven: JT at t_hi
 *   counts >= 1, or else JT counts >= 1 at one of the points rd(c - 4^j ulp(c)), j = 0 .. 11, above t_hi.  A class met
 *   in several chunks of one level counts once for each, so [4] is 0 exactly when every dropped class is proven.
 * When proof[3] = proof[4] = 0 this is a theorem (DESIGN.md §4.12): exactly n_within - proof[2] trees on N vertices have
 * key <= bound, and proof[0] of them have key < bound.  Errors and state as azb_trees_within; proof may be NULL. */
int azb_trees_within_proof(azb_handle *h, double bound, uint32_t k, uint64_t max_level, uint32_t *n_out, uint64_t *n_within,
                           uint64_t *n_below, uint64_t *codes /*[k*2]*/, uint8_t *parents /*[k*N]*/, double *lambda1 /*[k]*/,
                           uint32_t *mu /*[k]*/, float *eval /*[k]*/, uint64_t *proof /*[5]*/, float *ms);
/* persistent walker state: states, paths, last_positions (optimizer/mod.rs:10-14) */
int azb_get_walkers(azb_handle *h, uint8_t *parents, uint32_t *permitted, uint32_t *path, uint32_t *pos,
                    uint32_t *path_len);
/* get_trees (optimizer/mod.rs:34-36), as a canonical dump of one SearchTree (tree/mod.rs:28-32):
 * nodes 6 x u32 {c bits, c* bits, n_t, exhausted_children, lo, hi} (state_weight.rs:4-10), keys W words per node,
 * preds 3 x u32 {a_id, g bits, edge_id|AZB_NONE} (arc_weight.rs:11-16), arcs 3 x u32 {src, dst, prediction_pos}
 * in creation order (petgraph EdgeIndex order). */
int azb_tree_sizes(azb_handle *h, uint32_t tree, uint32_t *n_nodes, uint32_t *n_arcs, uint32_t *n_preds);
int azb_dump_tree(azb_handle *h, uint32_t tree, uint32_t *nodes, uint32_t *keys, uint32_t *preds, uint32_t *arcs);
int azb_get_counters(azb_handle *h, azb_counters *out);
int azb_reset_counters(azb_handle *h);
/* full != 0 (default): all 16 workload counters; 0: only n_live, n_noop, n_ins (the timed bench pass) */
int azb_set_counter_mode(azb_handle *h, int full);
/* current state vectors / priors held on the device (state_vecs, h_theta_host: optimizer/mod.rs:15-16) */
int azb_get_state_vecs(azb_handle *h, float *state_vecs /*[B*S]*/);
int azb_get_priors(azb_handle *h, float *priors /*[B*A]*/);

/* ---- stand-alone cost kernel: Space::cost + evaluate (rooted_tree/ordered_edge.rs:72-124; 04-c21-tree.rs:96-102)
 *      for M independent trees.  ms (may be NULL) = device time of the kernel alone. ---- */
int azb_eval_costs(azb_handle *h, const uint8_t *parents /*[M*N]*/, uint32_t m, double *lambda1, uint32_t *mu,
                   float *c, float *ms);

/* ---- SURVEY 8(f) row 3: the same cost for CONNECTED GRAPHS held as neighbourhood bit sets
 *      (ConnectedBitsetGraph<N, B32>: simple_graph/connected_bitset_graph/mod.rs).  nbr[g*n + v] = neighbours of v.
 *      lambda1 = largest eigenvalue of A + 1e-4 I (adjacency_matrix :200-216, conjecture_2_1_cost :319-337),
 *      mu = matching_number (:218-317), kinds[g][ceil(n(n-1)/32)] = action_kinds (:134-154) in the index space of
 *      AddOrDeleteEdge::action_index (bitset_graph/space/action.rs:10-19): bit colex(e) set <=> Add(e) is available,
 *      bit n(n-1)/2 + colex(e) set <=> Delete(e) is (e is an edge and not a cut edge, is_cut_edge :45-71).
 *      AZB_ERR_INVALID for n outside 2..32, loops, asymmetric or disconnected input (what try_from / to_connected
 *      reject); AZB_ERR_LAMBDA where the reference asserts lambda_1 > 1.4.  Any output pointer may be NULL. ---- */
int azb_eval_graph_costs(azb_handle *h, const uint32_t *nbr /*[M*n]*/, uint32_t m, uint32_t n, double *lambda1,
                         uint32_t *mu, uint32_t *kinds, float *ms);
/* ---- the same row for ConnectedBitsetGraph<N, B64>: nbr[g*n + v] = u64 neighbourhood of v, 2 <= n <= 64.  Outputs,
 *      kinds layout (ceil(n(n-1)/32) words per graph, 126 at n = 64) and errors as above; AZB_ERR_INVALID also for
 *      n outside 2..64 and for any bit >= n (bits 32..63 included when n <= 32). ---- */
int azb_eval_graph_costs64(azb_handle *h, const uint64_t *nbr /*[M*n]*/, uint32_t m, uint32_t n, double *lambda1,
                           uint32_t *mu, uint32_t *kinds, float *ms);

/* ---- epoch boundary ("next" rows): par_update_model's observation pass (tree/mod.rs:242-264,
 *      optimizer/mod.rs:262-278) ---- */
int azb_write_observations(azb_handle *h, uint32_t n_obs_tol, float *state_vecs, float *observations,
                           float *weights);

/* ---- epoch boundary: the training step.  NablaModel::update_model (nabla/model/mod.rs:7; ActionModel:
 *      nabla/model/dfdx.rs:86-131): w_n = w / sum(w); loss = sum (forward(states) - observations)^2 * w_n; backward;
 *      Adam (04-c21-tree.rs:87-92: lr 1e-4, betas .9/.999, eps 1e-8, WeightDecay::L2(1e-6)); gradients zeroed.
 *      f32 throughout, like the reference.  Returns the loss (dfdx.rs:125,130). ---- */
int azb_adam_config(azb_handle *h, float lr, float beta1, float beta2, float eps, float l2);  /* AdamConfig */
/* update_model with host buffers [rows*S], [rows*A], [rows*A]; rows <= B */
int azb_model_update(azb_handle *h, const float *states, const float *observations, const float *action_weights,
                     uint32_t rows, float *loss);
/* test hook: loss and d loss / d params (parameter order) of the same objective, no Adam step */
int azb_model_gradients(azb_handle *h, const float *states, const float *observations, const float *action_weights,
                        uint32_t rows, float *loss, float *grads);
/* NablaOptimizer::par_update_model (optimizer/mod.rs:249-281): root vectors + observations + update_model, all on
 * the device.  With a communicator attached (below) the weight sum, the gradient and the loss are all-reduced, so
 * every rank applies the same global-batch Adam step. */
int azb_update_model(azb_handle *h, uint32_t n_obs_tol, float *loss);

/* NablaOptimizer::par_reset_trees (optimizer/mod.rs:284-360) with the example's modify_root policy
 * (04-c21-tree.rs:172-206) evaluated on the device, followed by the tail shared with par_new (= azb_init_trees):
 * a root that found nothing better moves to an equal-cost node and widens its permitted set (or is regenerated
 * once that set is at k_max); otherwise it moves to a uniformly chosen node with c <= (c + 3 c*) / 4 and re-draws
 * the permitted set.  The reference draws from an unseeded thread_rng; here every draw is a counter hash of
 * (seed, number of resets so far, GLOBAL root index), so a sharded run re-selects exactly like an unsharded one.
 * k_min / k_max = num_permitted_actions_range (0, 0 = the example's 5 ..= ACTION_DIM / 2). */
int azb_reset_trees(azb_handle *h, uint64_t seed, uint32_t k_min, uint32_t k_max);

/* ---- epoch-boundary communicator (NCCL, loaded on demand; no collective ever runs inside azb_step).  Rank 0 makes
 *      an id, the host program hands it to every rank (any out-of-band channel), each rank attaches its handle. ---- */
int azb_comm_unique_id(uint8_t *id128 /*[128]*/);
int azb_comm_init(azb_handle *h, const uint8_t *id128, int rank, int world);
int azb_comm_destroy(azb_handle *h);
/* argmin over ALL ranks' roots (the sharded form of optimizer/mod.rs:221 + argmin_data): same outputs as
 * azb_get_argmin plus the owning rank; the lowest rank wins ties */
int azb_comm_argmin(azb_handle *h, uint8_t *parents, uint32_t *permitted, double *lambda1, uint32_t *mu, float *eval,
                    int *owner_rank);
/* azb_trees_within split over the ranks of the communicator: collective (every rank calls it), with the same arguments
 * and outputs.  Every rank returns the same outputs, bit for bit what azb_trees_within returns on one handle of the same
 * N for the same bound and k, whatever the world size and each rank's chunk size: every class is costed on its
 * canonical labelling, so its key does not depend on the rank that costs it.  azb_trees_within itself stays local.
 * Ownership: a class (code hi, lo) belongs to rank mix64(hi ^ mix64(lo)) mod world (mix64 as in the checkpoint digest
 * above); a rank holds only the classes of each level it owns, the path and the star on 4 vertices start with theirs.
 * A level runs in R rounds on every rank, R = the most chunks of parents any rank has at that level (a rank with none
 * left takes part with an empty chunk).  A round: expand, code, sort and unique by code the rank's chunk; route the
 * classes by owner into per-rank runs of 16-byte codes; all-gather a record per rank (its send counts to every rank, its
 * kept-list size, its cap and its cost error word); exchange the runs with grouped NCCL sends and receives (the own run
 * is a device copy); sort and unique the received codes, then decode, cost and keep them in pieces of at most one
 * chunk.  The kept list is sorted and made unique by code as in azb_trees_within, and one more record closes the level:
 * the level's size is the sum of the kept lists, and at 0 every rank stops.  At the last level each rank sorts its
 * share by (key bits, code); n_within and n_below are sums over ranks, each rank's first min(k, share) are all-gathered
 * and merged by (key bits, code), and every rank costs the global first min(k, n_within) as azb_trees_within does.
 * Errors are agreed: the first collective all-gathers every rank's (N, bound bits, k, max_level), and every rank returns
 * AZB_ERR_INVALID (azb_last_error names the rank and the field) for k == 0, k > 65536 or a NaN bound on any rank, and
 * for an N, bound, k or max_level that differs between ranks.  AZB_ERR_CAPACITY on every rank, in the same round, when
 * the sum of the kept lists exceeds max_level or a rank's share exceeds what its device has room for (the message
 * names the level; with the same max_level this is the level where azb_trees_within stops).  AZB_ERR_LAMBDA on every
 * rank when any rank saw it.  A CUDA or NCCL failure is reported by the rank that saw it.  After an agreed refusal the
 * communicator stays usable.  AZB_ERR_STATE without azb_comm_init, AZB_ERR_INVALID on more than 256 ranks.  Works
 * before azb_init_trees, runs all NCCL work on the library stream, changes no tree, walker, counter, argmin, model or
 * RNG state; the exchange buffers come from the handle's scratch and count in azb_device_bytes. */
int azb_comm_trees_within(azb_handle *h, double bound, uint32_t k, uint64_t max_level, uint32_t *n_out, uint64_t *n_within,
                          uint64_t *n_below, uint64_t *codes /*[k*2]*/, uint8_t *parents /*[k*N]*/, double *lambda1 /*[k]*/,
                          uint32_t *mu /*[k]*/, float *eval /*[k]*/, float *ms);

/* measurement helper: `reps` NCCL all-reduces of the gradient buffer (azb_mlp_num_params floats), timed with events on
 * the library's stream; *ms = milliseconds per all-reduce */
int azb_comm_allreduce_bench(azb_handle *h, uint32_t reps, float *ms);

/* ---- measurement helpers ---- */
int azb_kernel_launches(const azb_handle *h, uint64_t *n);   /* kernels launched by this handle so far */
/* HBM held by this handle.  Every call outside the search step (the stand-alone costs, azb_get_argmin's cost, codes, best
 * trees, enumeration, azb_trees_within, checkpoints) takes its device buffers from one grow-only scratch slab, so this
 * counts the largest scratch any of them has needed so far. */
int azb_device_bytes(const azb_handle *h, uint64_t *bytes);
int azb_flush_l2(azb_handle *h);                             /* overwrite a >L2 scratch buffer */
/* cascades (cascade_new_terminal / cascade_old_node, nabla/tree/empty_transitions.rs:50-127) whose ancestor wave
 * outgrew the on-chip work list and continued in the tree's HBM scratch, since azb_create.  The reference's BTreeMap
 * frontier has no limit and neither has this path; the count exists so that tests can prove they exercised it. */
int azb_debug_cascade_spills(azb_handle *h, uint32_t *n);

#ifdef __cplusplus
}
#endif
#endif
