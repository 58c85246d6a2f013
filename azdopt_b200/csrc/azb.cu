// azb.cu — host side of libazb.so: the C ABI of include/azb.h over the sm_100a kernels in this directory.
//
// Replaces the data-parallel part of NablaOptimizer (az-discrete-opt/src/nabla/optimizer/mod.rs:39-281) for the
// c21 space.  All search state lives in HBM between calls; a step is one launch of the tree kernel plus the MLP
// forward, enqueued on the handle's stream with no host round trip.
//
// This file never includes, links or loads anything under oracle/.
#include <cuda_runtime.h>
#include <time.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <tuple>
#include <vector>

#include "../../include/azb.h"
#include "azb_common.cuh"
#include "azb_cost.cuh"
#include "azb_graph.cuh"
#include "azb_mlp.cuh"
#include "azb_mlp_tc.cuh"
#include "azb_tree.cuh"
#include "azb_train.cuh"
#include "azb_async.cuh"
#include "azb_best.cuh"
#include "azb_ckpt.cuh"
#include "azb_enum.cuh"
#include "azb_grow.cuh"
#include "azb_certify.cuh"

#include <dlfcn.h>

// ---------------------------------------------------------------------------------------------------------------
struct azb_handle {
    azb_config cfg;
    AzbLayout L;
    uint32_t N, A, W, PW, WS, S;
    uint32_t dims[5];
    size_t n_params;
    cudaStream_t stream;
    cudaEvent_t ev0, ev1;
    // model
    float *params;      // dfdx order, f32
    float *act[3];      // hidden activations of the fp32 path
    float *mlp_x, *mlp_y;
    uint16_t *sv16_save;  // azb_model_write_predictions: the walkers' bf16 state rows while their buffer serves the call
    uint32_t mlp_rows;  // rows the staging buffers hold
    AzbMlpTc tc;        // tensor-core path state (bf16 weights, activations)
    // the device scratch of every call outside the search step: one grow-only slab (scratch_grow, Carve)
    uint8_t *scratch;
    size_t scratch_cap;
    // azb_best_trees (azb_best.cuh): the selection round's state, and the cap on the first round's M that tests set
    // through AZB_TEST_BEST_CAP (0 = none)
    AzbBestState *best_st;
    uint32_t best_m_cap;
    // azb_checkpoint_* (azb_ckpt.cuh): a copy stream and its events, the chunk size tests set through AZB_TEST_CKPT_CHUNK
    // (0 = the default), and the running best's global position when a load took it from a root outside this handle's
    // range (AzbGlobals::argmin_tree is AZB_NONE then)
    cudaStream_t ckpt_stream;
    cudaEvent_t ckpt_ev[4];
    uint64_t ckpt_chunk;
    uint64_t ckpt_best_root;
    uint32_t ckpt_best_node;
    // azb_free_trees / azb_exhaustive_best (azb_enum.cuh): the enumeration tables (built on first use) and the chunk size
    // tests set through AZB_TEST_ENUM_CHUNK (0 = AZB_ENUM_CHUNK)
    AzbEnum en;
    unsigned long long *en_P;
    uint8_t *en_rp;
    uint32_t en_chunk;
    // azb_trees_within (azb_grow.cuh): children per chunk, set by tests through AZB_TEST_GROW_CHUNK (0 = AZB_GROW_CHUNK)
    uint32_t grow_chunk;
    // observations scratch
    float *obs, *obs_w;
    // training step (azb_train.cuh): gradient (parameter order), Adam moments, predictions, two dZ buffers, scalars
    float *grad, *adam_m, *adam_v, *tr_p, *tr_dz[2], *tr_x;
    double *tr_scal, *tr_part;   // [0] weight sum, [1] loss; per-block partials
    uint32_t adam_t;
    uint64_t epoch;              // azb_reset_trees calls so far (keys the root re-selection draws)
    AzbAdam adam;
    // asynchronous search kernel (azb_async.cuh)
    bool async_ready, async_ran;
    AzbAsyncParams asP;
    AzbAsyncMaps asM;
    int async_grid;
    size_t async_smem, async_zero_bytes;
    unsigned long long async_timeout_base_ns;
    // azb_step_poll: per-step results of enqueued steps while they still run (copies on their own stream)
    cudaStream_t poll_stream;
    uint2 *poll_pin;          // pinned: one candidate row [B]
    uint32_t *poll_word;      // pinned: best_c at the start of the batch
    uint32_t poll_next;       // next candidate slot to report (slot s = step s - 1)
    uint32_t poll_best;       // running best, order-preserving bits
    bool poll_best_valid;
    void *async_bufs[16];
    // epoch-boundary collectives (NCCL, loaded on demand)
    void *nccl_lib, *nccl_comm;
    int comm_rank, comm_world;
    uint32_t *comm_buf;
    void *flush_buf;
    size_t flush_bytes;
    uint64_t launches, dev_bytes;
    bool roots_set, trees_init, pending_add, first_init_done, params_set, count_full;
    bool host_add_pending;  // azb_rollout_host has run, its azb_add_actions_host has not
    int improved_last_rollout;
    uint32_t steps_done;   // steps every tree has completed since init_trees
    uint32_t argmin_from;  // first candidate slot the argmin pass has not consumed yet
    uint32_t lcap, smem_words_per_warp;
    size_t smem_bytes;
    uint32_t n_groups, group_trees;
    cudaStream_t gstream[64];
    cudaEvent_t gevent[64], fork_event;
    cudaGraphExec_t ggraph[64];   // per group: AZB_GRAPH_STEPS steps of (search kernel + model forward)
    uint32_t ggraph_key[64];      // flags | counter mode the cached graph was captured with
    cudaGraphExec_t step_graph;   // one step incl. the argmin pass and the read-back of the globals (azb_step(h, 1, ...))
    uint32_t step_graph_key;
    AzbGlobals *pin_g;            // pinned host copy of the globals' head, written by the step graph
    uint32_t *roots_pin, *roots_dev;  // azb_set_roots: pinned staging of the packed root blocks and their device copy
    cudaEvent_t roots_ev;             // the staging buffer is free again once this has passed
    AzbGlobals *pin_rg;               // pinned landing zone of read_globals / azb_get_argmin
    uint32_t *pin_abort;
    uint32_t *pin_cost;               // pinned: lambda_1 (8 bytes), mu, eval, error word of azb_get_argmin's cost evaluation
    azb_improvement *pin_log;
    char err[512];
};

static const char *k_empty = "";
extern "C" { static void azb_comm_destroy_impl(azb_handle *h); }

static int fail(azb_handle *h, int code, const char *fmt, ...) {
    if (h) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(h->err, sizeof(h->err), fmt, ap);
        va_end(ap);
    }
    return code;
}

#define CK(call)                                                                                           \
    do {                                                                                                   \
        cudaError_t e_ = (call);                                                                           \
        if (e_ != cudaSuccess)                                                                             \
            return fail(h, AZB_ERR_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

template <class T>
static cudaError_t dmalloc(azb_handle *h, T **p, size_t count) {
    size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
    cudaError_t e = cudaMalloc((void **)p, bytes);
    if (e == cudaSuccess) h->dev_bytes += bytes;
    return e;
}

// Every call outside the search step takes its device buffers from one grow-only slab on the handle (a cudaMalloc per
// call would cost more than most of these calls' kernels).  A call writes its layout once, as a function of a Carve, and
// scratch() runs it twice: without a base to size the slab, then on the slab for the pointers.  A grow frees the old
// slab, so every region a call reads after its last scratch() must come from that same layout.
struct Carve {
    uint8_t *base;
    size_t off;
    template <class T>
    T *take(size_t count) {  // the next `count` T's, 256-byte aligned
        T *p = base ? reinterpret_cast<T *>(base + off) : nullptr;
        off += (count * sizeof(T) + 255) & ~(size_t)255;
        return p;
    }
};

static int scratch_grow(azb_handle *h, size_t bytes) {
    if (bytes <= h->scratch_cap) return AZB_OK;
    if (h->scratch) {  // the library stream and the checkpoint copy stream are the only ones that use the slab
        CK(cudaStreamSynchronize(h->stream));
        if (h->ckpt_stream) CK(cudaStreamSynchronize(h->ckpt_stream));
        CK(cudaFree(h->scratch));
        h->dev_bytes -= h->scratch_cap;
    }
    h->scratch = nullptr;
    h->scratch_cap = 0;
    CK(dmalloc(h, &h->scratch, bytes));
    h->scratch_cap = bytes;
    return AZB_OK;
}

template <class Layout>
static int scratch(azb_handle *h, Layout layout) {
    Carve size{nullptr, 0};
    layout(size);
    int rc = scratch_grow(h, size.off);
    if (rc) return rc;
    Carve c{h->scratch, 0};
    layout(c);
    return AZB_OK;
}

static uint32_t isqrt_ceil(uint32_t x) {
    uint32_t s = 0;
    while ((s + 1) * (s + 1) <= x) ++s;
    return s * s == x ? s : s + 1;
}
static uint32_t next_pow2(uint32_t x) {
    uint32_t p = 1;
    while (p < x) p <<= 1;
    return p;
}
static uint32_t action_dim(uint32_t n) { return (n - 1) * (n - 2) / 2 - 1; }  // rooted_tree/space.rs:48

extern "C" {

int azb_version(void) { return AZB_VERSION; }

const char *azb_strerror(int code) {
    switch (code) {
        case AZB_OK: return "ok";
        case AZB_ERR_INVALID: return "invalid argument";
        case AZB_ERR_CUDA: return "CUDA error";
        case AZB_ERR_CAPACITY: return "per-tree arena capacity exceeded";
        case AZB_ERR_NAN: return "NaN reached a comparison";
        case AZB_ERR_LAMBDA: return "lambda_1 < 1.4";
        case AZB_ERR_UNREACHABLE: return "inactive non-root walker";
        case AZB_ERR_STATE: return "call order violated";
        default: return "unknown";
    }
}

const char *azb_last_error(const azb_handle *h) { return h ? h->err : k_empty; }

// NablaOptimizer's constants for the c21 example (graph-state/examples/04-c21-tree.rs:33-68,133-138)
int azb_config_default(azb_config *cfg, uint32_t n_vertices, uint32_t n_roots) {
    if (!cfg || n_vertices < 5 || n_vertices > AZB_MAX_VERTICES || n_roots == 0) return AZB_ERR_INVALID;
    memset(cfg, 0, sizeof(*cfg));
    cfg->struct_size = sizeof(*cfg);
    cfg->n_vertices = n_vertices;
    cfg->n_roots = n_roots;
    cfg->device = 0;
    cfg->first_root = 0;
    cfg->c_lower = 2.0f;
    cfg->c_upper = 0.0f;
    cfg->n_as_tol[0] = 200;
    cfg->n_as_tol[1] = 50;
    cfg->n_as_tol[2] = 50;
    cfg->n_as_tol_len = 3;
    cfg->n_as_tol_default = 25;
    cfg->mlp_hidden[0] = 512;
    cfg->mlp_hidden[1] = 1024;
    cfg->mlp_hidden[2] = 512;
    cfg->mlp_mode = AZB_MLP_FP32;
    cfg->prior_mode = AZB_PRIOR_MLP;
    cfg->prior_seed = 0;
    cfg->max_steps = 800;
    cfg->max_episodes = 0;
    cfg->n_groups = 1;
    cfg->selection = AZB_SELECT_REFERENCE;
    cfg->puct_c = 1.0f;
    return AZB_OK;
}

int azb_destroy(azb_handle *h) {
    if (!h) return AZB_OK;
    cudaSetDevice(h->cfg.device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->step_graph) cudaGraphExecDestroy(h->step_graph);
    for (uint32_t g = 0; g < 64; ++g)
        if (h->ggraph[g]) cudaGraphExecDestroy(h->ggraph[g]);
    if (h->nccl_comm) azb_comm_destroy_impl(h);
    for (void *p : h->async_bufs)
        if (p) cudaFree(p);
    void *ptrs[] = {h->grad, h->adam_m, h->adam_v, h->tr_p, h->tr_dz[0], h->tr_dz[1], h->tr_x, h->tr_scal, h->tr_part, h->comm_buf,
                    h->L.walker, h->L.node, h->L.blk, h->L.inl, h->L.key, h->L.hash, h->L.casc, h->L.cand, h->L.stepmin, (void *)h->L.lut, h->L.sv,
                    h->L.h, h->L.g, h->L.log, h->params, h->act[0], h->act[1], h->act[2], h->mlp_x, h->mlp_y, h->sv16_save,
                    h->scratch, h->obs, h->obs_w, h->flush_buf, h->best_st, h->en_P, h->en_rp};
    for (void *p : ptrs)
        if (p) cudaFree(p);
    azb_mlp_tc_destroy(h->tc);
    for (uint32_t g = 0; g < 64; ++g) {
        if (h->gstream[g]) cudaStreamDestroy(h->gstream[g]);
        if (h->gevent[g]) cudaEventDestroy(h->gevent[g]);
    }
    if (h->fork_event) cudaEventDestroy(h->fork_event);
    for (cudaEvent_t e : h->ckpt_ev)
        if (e) cudaEventDestroy(e);
    if (h->ckpt_stream) cudaStreamDestroy(h->ckpt_stream);
    if (h->pin_g) cudaFreeHost(h->pin_g);
    if (h->poll_pin) cudaFreeHost(h->poll_pin);
    if (h->roots_pin) cudaFreeHost(h->roots_pin);
    if (h->roots_dev) cudaFree(h->roots_dev);
    if (h->roots_ev) cudaEventDestroy(h->roots_ev);
    if (h->pin_rg) cudaFreeHost(h->pin_rg);
    if (h->pin_abort) cudaFreeHost(h->pin_abort);
    if (h->pin_cost) cudaFreeHost(h->pin_cost);
    if (h->poll_word) cudaFreeHost(h->poll_word);
    if (h->poll_stream) cudaStreamDestroy(h->poll_stream);
    if (h->pin_log) cudaFreeHost(h->pin_log);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return AZB_OK;
}

int azb_create(const azb_config *cfg_in, azb_handle **out) {
    if (!cfg_in || !out) return AZB_ERR_INVALID;
    *out = nullptr;
    if (cfg_in->struct_size != sizeof(azb_config)) return AZB_ERR_INVALID;
    azb_config cfg = *cfg_in;
    if (cfg.n_vertices < 5 || cfg.n_vertices > AZB_MAX_VERTICES || cfg.n_roots == 0) return AZB_ERR_INVALID;
    if (cfg.n_as_tol_len > AZB_MAX_TOL) return AZB_ERR_INVALID;
    if (cfg.prior_mode > AZB_PRIOR_INJECTED || cfg.mlp_mode > AZB_MLP_TC3) return AZB_ERR_INVALID;
    if (cfg.selection > AZB_SELECT_PUCT) return AZB_ERR_INVALID;
    if (cfg.selection == AZB_SELECT_PUCT && !(std::isfinite(cfg.puct_c) && cfg.puct_c > 0.0f)) return AZB_ERR_INVALID;
    azb_handle *h = new azb_handle();
    memset((void *)h, 0, sizeof(*h));
    h->err[0] = 0;
    *out = h;  // returned even on failure so that azb_last_error can be read; the caller destroys it
    {
        // a device in exclusive-process mode refuses a new context while the previous process is still being torn
        // down (seen between back-to-back benchmark processes): retry for a few seconds before giving up
        int ndev = 0;
        cudaError_t ce = cudaSuccess;
        for (int attempt = 0; attempt < 50; ++attempt) {
            ce = cudaGetDeviceCount(&ndev);
            if (ce == cudaSuccess && cfg.device >= 0 && cfg.device < ndev) {
                ce = cudaSetDevice(cfg.device);
                if (ce == cudaSuccess) ce = cudaFree(nullptr);
            }
            if (ce == cudaSuccess || ce == cudaErrorNoDevice || ce == cudaErrorInsufficientDriver) break;
            cudaGetLastError();
            struct timespec ts = {0, 100 * 1000 * 1000};
            nanosleep(&ts, nullptr);
        }
        if (ce != cudaSuccess) return fail(h, AZB_ERR_CUDA, "no usable CUDA device: %s", cudaGetErrorString(ce));
        if (cfg.device < 0 || cfg.device >= ndev) return fail(h, AZB_ERR_CUDA, "device %d of %d", cfg.device, ndev);
    }
    const uint32_t N = cfg.n_vertices, A = action_dim(N), W = (A + 31) / 32, PW = (N + 3) / 4, B = cfg.n_roots;
    if (cfg.c_upper == 0.0f) cfg.c_upper = (float)(isqrt_ceil(N - 1) + (N + 1) / 2);  // 04-c21-tree.rs:59-68
    if (!(cfg.c_upper > cfg.c_lower)) return fail(h, AZB_ERR_INVALID, "c_upper must exceed c_lower");
    if (cfg.max_steps == 0) cfg.max_steps = 800;
    if (cfg.n_groups == 0) cfg.n_groups = 1;
    if (cfg.n_groups > 64) return fail(h, AZB_ERR_INVALID, "n_groups > 64");
    if (cfg.n_groups > 1 && cfg.max_episodes) return fail(h, AZB_ERR_INVALID, "n_groups > 1 needs max_episodes = 0");
    for (int i = 0; i < 3; ++i)
        if (cfg.mlp_hidden[i] == 0) cfg.mlp_hidden[i] = i == 1 ? 1024 : 512;
    // arena growth measured with the oracle on the example's root distribution (DESIGN.md §3): at most ~1.9 nodes,
    // ~A/7 predictions (A/4 in the first steps) and ~N in-arc slots per step per tree; sized with >= 1.5x head-room,
    // overflow is reported as AZB_ERR_CAPACITY, never dropped
    if (cfg.async_workers == AZB_ASYNC_AUTO) {
        // measured on one B200 (profiles/README.md, round 2 worker sweeps): the model side needs ~2.3 M rows/s of capacity
        // per SM it gets, the tree side one warp per tree up to 4096 roots
        const bool applies = cfg.prior_mode == AZB_PRIOR_MLP && (cfg.mlp_mode == AZB_MLP_TC || cfg.mlp_mode == AZB_MLP_TC3) &&
                             cfg.max_episodes == 0 && cfg.n_groups <= 1 && cfg.n_roots >= 1024;
        if (!applies) cfg.async_workers = 0;
        else if (cfg.n_vertices >= 47) cfg.async_workers = 16;  // N = 64, 4096 roots: 8 / 16 / 24 / 32 model SMs -> 6.4 / 8.8 / 8.3 / 7.8 M
        // (session 3, `profiles/r02_dyn_*`: with free warps taking over any runnable tree of their CTA the tree side no
        // longer needs a whole number of trees per warp, and one layout serves every batch beyond 4096 roots)
        else if (cfg.n_roots <= 4096) cfg.async_workers = 20;
        else cfg.async_workers = 36;
    }
    if (cfg.cap_nodes == 0) cfg.cap_nodes = 3 * cfg.max_steps + 64;
    if (cfg.cap_preds == 0) cfg.cap_preds = 2 * A + cfg.max_steps * ((2 * A + 6) / 7);
    if (cfg.cap_parents == 0) cfg.cap_parents = cfg.cap_nodes * (N > 8 ? N - 7 : 1);  // in-arcs beyond the 4 inline ones
    if (cfg.cap_nodes > (1u << 20) - 2) return fail(h, AZB_ERR_INVALID, "cap_nodes too large");
    h->cfg = cfg;
    h->N = N;
    h->A = A;
    h->W = W;
    h->PW = PW;
    h->WS = WK_HDR + 2 * PW + 3 * W;
    h->S = 2 * A;
    h->dims[0] = h->S;
    h->dims[1] = cfg.mlp_hidden[0];
    h->dims[2] = cfg.mlp_hidden[1];
    h->dims[3] = cfg.mlp_hidden[2];
    h->dims[4] = A;
    h->n_params = 0;
    for (int l = 0; l < 4; ++l) h->n_params += (size_t)h->dims[l] * h->dims[l + 1] + h->dims[l + 1];

    CK(cudaSetDevice(cfg.device));
    CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    CK(cudaEventCreate(&h->ev0));
    CK(cudaEventCreate(&h->ev1));
    CK(cudaEventCreateWithFlags(&h->fork_event, cudaEventDisableTiming));
    CK(cudaMallocHost((void **)&h->pin_g, sizeof(AzbGlobals)));
    CK(cudaMallocHost((void **)&h->pin_log, sizeof(azb_improvement)));
    {
        // concurrent groups of trees: contiguous ranges, a multiple of 128 trees each (MLP row tiles)
        uint32_t per = (cfg.n_roots + cfg.n_groups - 1) / cfg.n_groups;
        per = (per + 127u) & ~127u;
        h->group_trees = per;
        h->n_groups = (cfg.n_roots + per - 1) / per;
        for (uint32_t g = 0; g < h->n_groups && h->n_groups > 1; ++g) {
            CK(cudaStreamCreateWithFlags(&h->gstream[g], cudaStreamNonBlocking));
            CK(cudaEventCreateWithFlags(&h->gevent[g], cudaEventDisableTiming));
        }
    }

    AzbLayout &L = h->L;
    L.N = N;
    L.A = A;
    L.W = W;
    L.B = B;
    L.PW = PW;
    L.WS = h->WS;
    L.cap_nodes = cfg.cap_nodes;
    L.cap_blk = AZB_BLK_PAD + 3 * cfg.cap_preds + 3 * cfg.cap_nodes;  // 8-byte units: preds + header + 2 per kid slot
    L.cap_blk += L.cap_blk & 1u;
    L.cap_in = cfg.cap_parents;
    L.cap_hash = next_pow2(2 * cfg.cap_nodes);
    L.cap_steps = cfg.max_steps + 8;
    L.sv_ld = h->S;
    L.h_ld = A;
    L.c_lower = cfg.c_lower;
    L.slope = 1.0f / (cfg.c_upper - cfg.c_lower);  // 04-c21-tree.rs:71
    for (uint32_t i = 0; i < 8; ++i) L.tol[i] = cfg.n_as_tol[i];
    L.tol_len = cfg.n_as_tol_len;
    L.tol_default = cfg.n_as_tol_default;
    L.selection = cfg.selection;
    L.puct_c = cfg.puct_c;
    L.prior_mode = cfg.prior_mode;
    L.log_cap = 4096;
    L.frontier_cap = AZB_FRONTIER_CAP;
    if (const char *e = getenv("AZB_TEST_FRONTIER_CAP"))  // tests: push ordinary cascades through the global continuation
        L.frontier_cap = std::min<uint32_t>(AZB_FRONTIER_CAP, std::max(1, atoi(e)));
    if (const char *e = getenv("AZB_TEST_BEST_CAP"))  // tests: force azb_best_trees through several widening rounds
        h->best_m_cap = (uint32_t)std::max(1, atoi(e));
    if (const char *e = getenv("AZB_TEST_CKPT_CHUNK"))  // tests: push checkpoints through many staging chunks
        h->ckpt_chunk = std::max<uint64_t>(8, strtoull(e, nullptr, 10));
    if (const char *e = getenv("AZB_TEST_ENUM_CHUNK"))  // tests: push azb_exhaustive_best through many threshold updates
        h->en_chunk = (uint32_t)std::max(1, atoi(e));
    if (const char *e = getenv("AZB_TEST_GROW_CHUNK"))  // tests: push azb_trees_within through many chunks and merges
        h->grow_chunk = (uint32_t)std::max(1, atoi(e));
    L.first_root = cfg.first_root;
    L.prior_seed = cfg.prior_seed;
    CK(dmalloc(h, &L.walker, (size_t)B * L.WS));
    CK(dmalloc(h, &L.node, (size_t)B * L.cap_nodes * 4));
    CK(dmalloc(h, &L.blk, (size_t)B * L.cap_blk + 128));  // + slack for the speculative 32-entry reads
    CK(dmalloc(h, &L.inl, (size_t)B * L.cap_in));
    CK(dmalloc(h, &L.key, (size_t)B * L.cap_nodes * W));
    CK(dmalloc(h, &L.hash, (size_t)B * L.cap_hash));
    CK(dmalloc(h, &L.casc, (size_t)B * 2 * L.cap_nodes));
    CK(dmalloc(h, &L.cand, (size_t)(L.cap_steps + 1) * B));
    CK(dmalloc(h, &L.stepmin, (size_t)L.cap_steps + 1));
    {
        std::vector<uint8_t> lut((A + 3) & ~3u, 0);
        for (uint32_t a = 0; a < A; ++a) lut[a] = (uint8_t)azb_action_child(a);
        uint8_t *dl = nullptr;
        CK(dmalloc(h, &dl, lut.size()));
        CK(cudaMemcpyAsync(dl, lut.data(), lut.size(), cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        L.lut = dl;
    }
    h->count_full = true;
    h->adam = AzbAdam{1e-4f, 0.9f, 0.999f, 1e-8f, 1e-6f, 1.f, 1.f};  // 04-c21-tree.rs:87-92
    CK(dmalloc(h, &L.sv, (size_t)B * L.sv_ld));
    CK(dmalloc(h, &L.h, (size_t)B * L.h_ld));
    CK(dmalloc(h, &L.g, 1));
    CK(dmalloc(h, &L.log, L.log_cap));
    CK(cudaMemsetAsync(L.walker, 0, (size_t)B * L.WS * 4, h->stream));
    CK(cudaMemsetAsync(L.sv, 0, (size_t)B * L.sv_ld * 4, h->stream));
    CK(cudaMemsetAsync(L.h, 0, (size_t)B * L.h_ld * 4, h->stream));
    AzbGlobals g0;
    memset(&g0, 0, sizeof(g0));
    g0.best_c = 0xffffffffu;
    CK(cudaMemcpyAsync(L.g, &g0, sizeof(g0), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));

    CK(dmalloc(h, &h->params, h->n_params));
    for (int i = 0; i < 3; ++i) CK(dmalloc(h, &h->act[i], (size_t)B * h->dims[i + 1]));
    if (cfg.mlp_mode == AZB_MLP_TC || cfg.mlp_mode == AZB_MLP_TC3) {
        const char *why = azb_mlp_tc_create(h->tc, B, h->dims, &h->dev_bytes, cfg.mlp_mode == AZB_MLP_TC3);
        if (why) return fail(h, AZB_ERR_CUDA, "tensor-core MLP: %s", why);
        if (cfg.prior_mode == AZB_PRIOR_MLP) {  // write_vec feeds the first GEMM directly
            L.sv16 = reinterpret_cast<uint16_t *>(h->tc.act[0]);
            L.sv16_ld = (h->tc.split ? 2u : 1u) * h->tc.kpad[0];  // bf16x3: [hi | lo]; write_vec fills hi, lo stays zero
        }
    }

    // shared memory per warp of the tree kernel: walker block + masks + children's c* + cascade frontiers
    h->lcap = (std::max<uint32_t>(A, 64) + 31) & ~31u;
    {
        // one region for: children's c* (selection) | cascade work lists + visited bitmap | cost scratch
        const uint32_t cascade_words = 3u * AZB_FRONTIER_CAP + ((L.cap_nodes + 31u) >> 5);
        const uint32_t shared_region = (std::max(std::max(h->lcap, cascade_words), azb_cost_scratch_words(h->N)) + 3u) & ~3u;
        h->smem_words_per_warp = ((L.WS + 3) & ~3u) + 64 + 64 + 32 + shared_region;
    }
    h->smem_words_per_warp = (h->smem_words_per_warp + 3u) & ~3u;
    h->smem_bytes = (size_t)AZB_WARPS_PER_BLOCK * h->smem_words_per_warp * 4 + azb_tables_bytes(A, N, h->W);  // + action->child LUT, child->action-mask table
    {
        const int sb = (int)h->smem_bytes;
        const auto attr = cudaFuncAttributeMaxDynamicSharedMemorySize;
        switch (azb_stack_depth(N) * 2 + (cfg.selection == AZB_SELECT_PUCT ? 1 : 0)) {
            case 6:
                CK(cudaFuncSetAttribute(azb_tree_kernel<3, true>, attr, sb));
                CK(cudaFuncSetAttribute(azb_tree_kernel<3, false>, attr, sb));
                break;
            case 7:
                CK(cudaFuncSetAttribute(azb_tree_kernel<3, true, true>, attr, sb));
                CK(cudaFuncSetAttribute(azb_tree_kernel<3, false, true>, attr, sb));
                break;
            case 8:
                CK(cudaFuncSetAttribute(azb_tree_kernel<4, true>, attr, sb));
                CK(cudaFuncSetAttribute(azb_tree_kernel<4, false>, attr, sb));
                break;
            case 9:
                CK(cudaFuncSetAttribute(azb_tree_kernel<4, true, true>, attr, sb));
                CK(cudaFuncSetAttribute(azb_tree_kernel<4, false, true>, attr, sb));
                break;
            case 10:
                CK(cudaFuncSetAttribute(azb_tree_kernel<5, true>, attr, sb));
                CK(cudaFuncSetAttribute(azb_tree_kernel<5, false>, attr, sb));
                break;
            default:
                CK(cudaFuncSetAttribute(azb_tree_kernel<5, true, true>, attr, sb));
                CK(cudaFuncSetAttribute(azb_tree_kernel<5, false, true>, attr, sb));
                break;
        }
    }
    return AZB_OK;
}

int azb_get_config(const azb_handle *h, azb_config *out) {
    if (!h || !out) return AZB_ERR_INVALID;
    *out = h->cfg;
    return AZB_OK;
}

// ---- synthetic roots: the example's distribution (04-c21-tree.rs:85,108-112; rooted_tree/mod.rs:14-20;
//      modify_parent_once.rs:14-25) driven by a counter hash of (seed, global root index) ----
static inline uint32_t bounded(unsigned long long r, uint32_t n) {
    return (uint32_t)(((r >> 32) * (unsigned long long)n) >> 32);
}

int azb_generate_roots(uint64_t seed, uint64_t first_root, uint32_t count, uint32_t n, uint32_t k_min, uint32_t k_max,
                       uint8_t *parents, uint32_t *permitted) {
    if (!parents || !permitted || n < 5 || n > AZB_MAX_VERTICES) return AZB_ERR_INVALID;
    const uint32_t a_dim = action_dim(n), words = (a_dim + 31) / 32;
    if (k_max == 0) k_max = a_dim / 2;
    if (k_min > k_max || k_max > a_dim) return AZB_ERR_INVALID;
    std::vector<uint32_t> perm(a_dim);
    for (uint32_t r = 0; r < count; ++r) {
        uint8_t *par = parents + (size_t)r * n;
        uint32_t *msk = permitted + (size_t)r * words;
        unsigned long long s = azb_mix64(seed ^ azb_mix64(first_root + r + 0x5851F42D4C957F2Dull));
        unsigned long long ctr = 0;
        auto next = [&]() { return azb_mix64(s + (ctr++) * 0xD1342543DE82EF95ull); };
        for (uint32_t i = 0; i < n; ++i) par[i] = 0;
        for (uint32_t i = 2; i + 1 < n; ++i) par[i] = (uint8_t)bounded(next(), i);
        uint32_t kk = k_min + bounded(next(), k_max - k_min + 1);
        for (uint32_t i = 0; i < a_dim; ++i) perm[i] = i;
        for (uint32_t i = 0; i < words; ++i) msk[i] = 0;
        for (uint32_t t = 0; t < kk; ++t) {
            uint32_t j = t + bounded(next(), a_dim - t);
            std::swap(perm[t], perm[j]);
            msk[perm[t] >> 5] |= 1u << (perm[t] & 31);
        }
    }
    return AZB_OK;
}

// root blocks [B][PW + W] (packed parents | permitted mask) -> the root part of every walker block
__global__ void azb_scatter_roots_kernel(uint32_t *__restrict__ walker, const uint32_t *__restrict__ src, uint32_t n_words,
                                         uint32_t per_root, uint32_t WS, uint32_t off) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_words) return;
    const uint32_t r = i / per_root, j = i - r * per_root;
    walker[(size_t)r * WS + off + j] = src[i];
}

int azb_set_roots(azb_handle *h, const uint8_t *parents, const uint32_t *permitted) {
    if (!h || !parents || !permitted) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    const uint32_t N = h->N, A = h->A, W = h->W, PW = h->PW, WS = h->WS, B = h->L.B, per = PW + W;
    const size_t bytes = (size_t)B * per * 4;
    // One pass over the caller's arrays validates them and packs the root part of each walker block
    // [hdr | state parents, permitted, path | ROOT parents, permitted] into a pinned staging buffer; one contiguous copy
    // and a scatter kernel put it in place (a strided copy out of pageable memory cost 0.8 ms per 4096 roots — a quarter
    // of a 20-step epoch).  The caller's buffers are free on return; nothing waits for the device here.
    if (!h->roots_pin) {
        CK(cudaMallocHost((void **)&h->roots_pin, bytes));
        CK(cudaMalloc((void **)&h->roots_dev, bytes));
        h->dev_bytes += bytes;
        CK(cudaEventCreateWithFlags(&h->roots_ev, cudaEventDisableTiming));
    } else {
        CK(cudaEventSynchronize(h->roots_ev));  // the previous call's copy has left the staging buffer
    }
    const uint32_t tail_bits = A % 32;
    for (uint32_t i = 0; i < B; ++i) {
        const uint8_t *p = parents + (size_t)i * N;
        for (uint32_t v = 1; v < N; ++v)
            if (p[v] >= v) return fail(h, AZB_ERR_INVALID, "root %u: parents[%u] = %u is not < %u", i, v, p[v], v);
        const uint32_t *m = permitted + (size_t)i * W;
        if (tail_bits && (m[W - 1] >> tail_bits)) return fail(h, AZB_ERR_INVALID, "root %u: permitted bit >= ACTION_DIM", i);
        uint32_t *dst = h->roots_pin + (size_t)i * per;
        dst[PW - 1] = 0u;
        memcpy(dst, p, N);
        memcpy(dst + PW, m, (size_t)W * 4);
    }
    CK(cudaMemcpyAsync(h->roots_dev, h->roots_pin, bytes, cudaMemcpyHostToDevice, h->stream));
    CK(cudaEventRecord(h->roots_ev, h->stream));
    const uint32_t n_words = B * per;
    azb_scatter_roots_kernel<<<(n_words + 255u) / 256u, 256, 0, h->stream>>>(h->L.walker, h->roots_dev, n_words, per, WS,
                                                                             WK_HDR + PW + 2 * W);
    CK(cudaGetLastError());
    h->launches += 1;
    h->roots_set = true;
    h->trees_init = false;
    return AZB_OK;
}

int azb_get_roots(azb_handle *h, uint8_t *parents, uint32_t *permitted) {
    if (!h || !parents || !permitted) return AZB_ERR_INVALID;
    if (!h->roots_set) return fail(h, AZB_ERR_STATE, "roots not set");
    CK(cudaSetDevice(h->cfg.device));
    const uint32_t N = h->N, W = h->W, PW = h->PW, WS = h->WS, B = h->L.B;
    std::vector<uint32_t> blk((size_t)B * (PW + W));
    CK(cudaMemcpy2DAsync(blk.data(), (size_t)(PW + W) * 4, h->L.walker + WK_HDR + PW + 2 * W, (size_t)WS * 4,
                         (size_t)(PW + W) * 4, B, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (uint32_t i = 0; i < B; ++i) {
        const uint32_t *src = blk.data() + (size_t)i * (PW + W);
        memcpy(parents + (size_t)i * N, src, N);
        memcpy(permitted + (size_t)i * W, src + PW, (size_t)W * 4);
    }
    return AZB_OK;
}

// ---- model ----
size_t azb_mlp_num_params(const azb_handle *h) { return h ? h->n_params : 0; }

int azb_mlp_set_params(azb_handle *h, const float *params) {
    if (!h || !params) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaMemcpyAsync(h->params, params, h->n_params * 4, cudaMemcpyHostToDevice, h->stream));
    if (h->tc.ready) {
        const char *why = azb_mlp_tc_load(h->tc, h->params, h->stream, &h->launches);
        if (why) return fail(h, AZB_ERR_CUDA, "tensor-core MLP: %s", why);
    }
    CK(cudaStreamSynchronize(h->stream));
    h->params_set = true;
    return AZB_OK;
}

// dfdx Linear default init: weight and bias ~ U(-1/sqrt(fan_in), 1/sqrt(fan_in)) (SURVEY.md §8d)
int azb_mlp_init(azb_handle *h, uint64_t seed) {
    if (!h) return AZB_ERR_INVALID;
    std::vector<float> p(h->n_params);
    size_t off = 0;
    for (int l = 0; l < 4; ++l) {
        const size_t cnt = (size_t)h->dims[l] * h->dims[l + 1] + h->dims[l + 1];
        const float bound = 1.0f / sqrtf((float)h->dims[l]);
        for (size_t i = 0; i < cnt; ++i) {
            unsigned long long r = azb_mix64(azb_mix64(seed + 0x1234567ull * (l + 1)) + (off + i) * 0x9E3779B97F4A7C15ull);
            float u = (float)(r >> 40) * 5.9604644775390625e-08f;
            p[off + i] = (2.0f * u - 1.0f) * bound;
        }
        off += cnt;
    }
    return azb_mlp_set_params(h, p.data());
}

int azb_mlp_get_params(azb_handle *h, float *params) {
    if (!h || !params) return AZB_ERR_INVALID;
    if (!h->params_set) return fail(h, AZB_ERR_STATE, "model parameters not set");
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaMemcpyAsync(params, h->params, h->n_params * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return AZB_OK;
}

// ActionModel::forward (nabla/model/dfdx.rs:81-83) on device rows [row0, row0 + rows)
static int mlp_forward(azb_handle *h, const float *x, uint32_t ldx, float *y, uint32_t ldy, uint32_t row0, uint32_t rows,
                       cudaStream_t stream) {
    if (h->tc.ready) {
        const bool packed = h->L.sv16 != nullptr && x == h->L.sv;  // tree_pack already wrote the bf16 rows
        const char *why = azb_mlp_tc_forward(h->tc, packed ? nullptr : x, ldx, y, ldy, row0, rows, stream, &h->launches);
        if (why) return fail(h, AZB_ERR_CUDA, "tensor-core MLP: %s", why);
        return AZB_OK;
    }
    const float *in = x + (size_t)row0 * ldx;
    uint32_t ld_in = ldx;
    const float *p = h->params;
    for (int l = 0; l < 4; ++l) {
        const uint32_t K = h->dims[l], Nout = h->dims[l + 1];
        float *outp = l < 3 ? h->act[l] + (size_t)row0 * Nout : y + (size_t)row0 * ldy;
        const uint32_t ld_out = l < 3 ? Nout : ldy;
        dim3 grid((Nout + 63) / 64, (rows + 63) / 64);
        if (l < 3)
            azb_linear_fp32_kernel<AZB_ACT_RELU><<<grid, 256, 0, stream>>>(in, ld_in, p, p + (size_t)K * Nout, outp, ld_out,
                                                                         rows, K, Nout);
        else
            azb_linear_fp32_kernel<AZB_ACT_SIGMOID><<<grid, 256, 0, stream>>>(in, ld_in, p, p + (size_t)K * Nout, outp,
                                                                            ld_out, rows, K, Nout);
        h->launches += 1;
        in = outp;
        ld_in = ld_out;
        p += (size_t)K * Nout + Nout;
    }
    CK(cudaGetLastError());
    return AZB_OK;
}

int azb_model_write_predictions(azb_handle *h, const float *states, float *predictions, uint32_t rows) {
    if (!h || !states || !predictions || rows == 0 || rows > h->L.B) return AZB_ERR_INVALID;
    if (!h->params_set) return fail(h, AZB_ERR_STATE, "model parameters not set");
    CK(cudaSetDevice(h->cfg.device));
    if (!h->mlp_x) {
        CK(dmalloc(h, &h->mlp_x, (size_t)h->L.B * h->S));
        CK(dmalloc(h, &h->mlp_y, (size_t)h->L.B * h->A));
    }
    // with AZB_PRIOR_MLP on the tensor cores the layer-0 input rows ARE the walkers' state vectors (L.sv16): they are
    // set aside while the caller's rows pass through and put back afterwards (bf16x3: both halves, so the lo half the
    // search kernels never write is zero again)
    const size_t sv16_bytes = h->L.sv16 ? (size_t)rows * h->L.sv16_ld * 2 : 0;
    if (sv16_bytes) {
        if (!h->sv16_save) CK(dmalloc(h, &h->sv16_save, (size_t)h->L.B * h->L.sv16_ld));
        CK(cudaMemcpyAsync(h->sv16_save, h->L.sv16, sv16_bytes, cudaMemcpyDeviceToDevice, h->stream));
    }
    CK(cudaMemcpyAsync(h->mlp_x, states, (size_t)rows * h->S * 4, cudaMemcpyHostToDevice, h->stream));
    int rc = mlp_forward(h, h->mlp_x, h->S, h->mlp_y, h->A, 0, rows, h->stream);
    if (rc) return rc;
    if (sv16_bytes) CK(cudaMemcpyAsync(h->L.sv16, h->sv16_save, sv16_bytes, cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaMemcpyAsync(predictions, h->mlp_y, (size_t)rows * h->A * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return AZB_OK;
}

// state_vecs (optimizer/mod.rs:15) to a host buffer; the tensor-core configuration keeps them as bf16 {0, 1} rows
static int copy_state_vecs(azb_handle *h, float *dst) {
    if (!h->L.sv16) {
        CK(cudaMemcpy2DAsync(dst, (size_t)h->S * 4, h->L.sv, (size_t)h->L.sv_ld * 4, (size_t)h->S * 4, h->L.B,
                             cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        return AZB_OK;
    }
    std::vector<uint16_t> tmp((size_t)h->L.B * h->S);
    CK(cudaMemcpy2DAsync(tmp.data(), (size_t)h->S * 2, h->L.sv16, (size_t)h->L.sv16_ld * 2, (size_t)h->S * 2, h->L.B,
                         cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (size_t i = 0; i < tmp.size(); ++i) dst[i] = tmp[i] ? 1.0f : 0.0f;
    return AZB_OK;
}

#define AZB_GRAPH_STEPS 8u

// ---- tree kernel launches ----
static int launch_tree(azb_handle *h, uint32_t flags, uint32_t target_step, int prior_mode_override = -1,
                       uint32_t tree0 = 0, uint32_t ntrees = 0xffffffffu, cudaStream_t stream = nullptr) {
    AzbLayout L = h->L;
    if (prior_mode_override >= 0) L.prior_mode = (uint32_t)prior_mode_override;
    if (!stream) stream = h->stream;
    const uint32_t tree_end = ntrees == 0xffffffffu ? L.B : std::min(L.B, tree0 + ntrees);
    const uint32_t blocks = (tree_end - tree0 + AZB_WARPS_PER_BLOCK - 1) / AZB_WARPS_PER_BLOCK;
    const dim3 block(AZB_WARPS_PER_BLOCK * 32);
    const uint32_t me = h->cfg.max_episodes;
#define AZB_LAUNCH_TREE(D, C)                                                                                             \
    do {                                                                                                                  \
        if (L.selection == AZB_SELECT_PUCT)                                                                               \
            azb_tree_kernel<D, C, true><<<blocks, block, h->smem_bytes, stream>>>(L, flags, h->smem_words_per_warp, h->lcap, \
                                                                                  target_step, me, tree0, tree_end);        \
        else                                                                                                              \
            azb_tree_kernel<D, C><<<blocks, block, h->smem_bytes, stream>>>(L, flags, h->smem_words_per_warp, h->lcap,     \
                                                                            target_step, me, tree0, tree_end);              \
    } while (0)
    switch (azb_stack_depth(h->N) * 2 + (h->count_full ? 1 : 0)) {
        case 6: AZB_LAUNCH_TREE(3, false); break;
        case 7: AZB_LAUNCH_TREE(3, true); break;
        case 8: AZB_LAUNCH_TREE(4, false); break;
        case 9: AZB_LAUNCH_TREE(4, true); break;
        case 10: AZB_LAUNCH_TREE(5, false); break;
        default: AZB_LAUNCH_TREE(5, true); break;
    }
#undef AZB_LAUNCH_TREE
    h->launches += 1;
    CK(cudaGetLastError());
    return AZB_OK;
}

static int read_globals(azb_handle *h, AzbGlobals *g) {
    // pinned landing zones: a copy into pageable memory is staged and synchronised by the driver, once per call
    if (!h->pin_rg) {
        CK(cudaMallocHost((void **)&h->pin_rg, sizeof(AzbGlobals)));
        CK(cudaMallocHost((void **)&h->pin_abort, 16));
    }
    CK(cudaMemcpyAsync(h->pin_rg, h->L.g, offsetof(AzbGlobals, argmin_state), cudaMemcpyDeviceToHost, h->stream));
    h->pin_abort[0] = 0u;
    if (h->async_ran) CK(cudaMemcpyAsync(h->pin_abort, &h->asP.st->abort, 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    memcpy(g, h->pin_rg, offsetof(AzbGlobals, argmin_state));
    const uint32_t as_abort = h->pin_abort[0];
    h->async_ran = false;
    if (as_abort == 1u) return fail(h, AZB_ERR_CUDA, "async search kernel: watchdog expired (no progress)");
    if (g->err)
        return fail(h, (int)g->err, "%s (tree %u, step %u)", azb_strerror((int)g->err), g->err_tree, g->err_step);
    return AZB_OK;
}

// read the device error word; translate it
static int check_device_error(azb_handle *h) {
    AzbGlobals g;
    return read_globals(h, &g);
}

// par_update_argmmim_data (optimizer/mod.rs:194-246) over the candidate slots [argmin_from, slot_hi): per slot the
// first minimum over trees, then the slots in step order against the running best
static int run_argmin(azb_handle *h, uint32_t slot_hi) {
    const uint32_t slot_lo = h->argmin_from;
    if (slot_hi <= slot_lo) return AZB_OK;
    azb_stepmin_kernel<<<slot_hi - slot_lo, 256, 0, h->stream>>>(h->L, slot_lo);
    azb_argmin_kernel<<<1, 32, 0, h->stream>>>(h->L, slot_lo, slot_hi);
    h->launches += 2;
    CK(cudaGetLastError());
    h->argmin_from = slot_hi;
    h->poll_next = slot_hi;
    h->poll_best_valid = false;
    return AZB_OK;
}

// the add_actions of the last rollout is fused into the NEXT step's launch; anything that reads the trees first
// runs it on its own
static int flush_pending(azb_handle *h) {
    if (!h->pending_add) return AZB_OK;
    int rc = launch_tree(h, AZB_F_ADD, h->steps_done);
    if (rc) return rc;
    h->pending_add = false;
    return AZB_OK;
}

int azb_set_priors(azb_handle *h, const float *priors) {
    if (!h || !priors) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaMemcpy2DAsync(h->L.h, (size_t)h->L.h_ld * 4, priors, (size_t)h->A * 4, (size_t)h->A * 4, h->L.B,
                         cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return AZB_OK;
}

int azb_init_trees(azb_handle *h) {
    if (!h) return AZB_ERR_INVALID;
    if (!h->roots_set) return fail(h, AZB_ERR_STATE, "azb_set_roots has not been called");
    if (h->cfg.prior_mode == AZB_PRIOR_MLP && !h->params_set) return fail(h, AZB_ERR_STATE, "model parameters not set");
    CK(cudaSetDevice(h->cfg.device));
    // SearchTree::clear (tree/mod.rs:45-49): only the transposition table needs wiping, the arenas are bump-allocated
    CK(cudaMemsetAsync(h->L.hash, 0, (size_t)h->L.B * h->L.cap_hash * 4, h->stream));
    CK(cudaMemsetAsync(&h->L.g->err, 0, 12, h->stream));
    const bool first = !h->first_init_done;
    int rc = launch_tree(h, AZB_F_INIT | (first ? (uint32_t)AZB_F_FIRST : 0u), 0);
    if (rc) return rc;
    if (h->cfg.prior_mode == AZB_PRIOR_MLP) {
        rc = mlp_forward(h, h->L.sv, h->L.sv_ld, h->L.h, h->L.h_ld, 0, h->L.B, h->stream);
        if (rc) return rc;
    }
    rc = launch_tree(h, AZB_F_ADD, 0);
    if (rc) return rc;
    h->pending_add = false;
    h->host_add_pending = false;
    h->steps_done = 0;
    h->argmin_from = first ? 0u : 1u;
    h->poll_next = 1u;
    h->poll_best_valid = false;
    if (first) {  // par_new's silent argmin over the roots (optimizer/mod.rs:95-101)
        rc = run_argmin(h, 1);
        if (rc) return rc;
    } else {
        static const uint32_t one = 1u;
        CK(cudaMemcpyAsync(&h->L.g->next_slot, &one, 4, cudaMemcpyHostToDevice, h->stream));
    }
    rc = check_device_error(h);
    if (rc) return rc;
    h->first_init_done = true;
    h->trees_init = true;
    return AZB_OK;
}


}  // extern "C"

// ---- the asynchronous search kernel (azb_async.cuh): set-up and launch -------------------------------------------
template <int D, bool C, bool PUCT>
static int async_prepare_one(azb_handle *h, int *blocks_per_sm) {
    CK(cudaFuncSetAttribute(azb_async_kernel<D, C, PUCT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->async_smem));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, azb_async_kernel<D, C, PUCT>, AS_THREADS, h->async_smem));
    return AZB_OK;
}
template <int D, bool C>
static int async_prepare_kernel(azb_handle *h, int *blocks_per_sm) {
    return h->cfg.selection == AZB_SELECT_PUCT ? async_prepare_one<D, C, true>(h, blocks_per_sm) : async_prepare_one<D, C, false>(h, blocks_per_sm);
}

static int async_create(azb_handle *h) {
    if (h->async_ready) return AZB_OK;
    if (h->cfg.prior_mode != AZB_PRIOR_MLP || !h->tc.ready)
        return fail(h, AZB_ERR_INVALID, "async_workers needs AZB_PRIOR_MLP with AZB_MLP_TC or AZB_MLP_TC3");
    if (h->cfg.max_episodes || h->n_groups > 1) return fail(h, AZB_ERR_INVALID, "async_workers excludes max_episodes / n_groups");
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, h->cfg.device));
    int coop = 0;
    CK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, h->cfg.device));
    if (!coop) return fail(h, AZB_ERR_CUDA, "cooperative launch not supported");
    uint32_t W = h->cfg.async_workers;
    const uint32_t B = h->L.B;
    // shared-SM form (azb_async.cuh): no SM is taken from the trees, the last warpgroup of every CTA is a model group member
    bool shared_sm = W == AZB_ASYNC_SHARED;
    if (const char *e = getenv("AZB_ASYNC_SHARED_SM")) shared_sm = atoi(e) != 0;
    if (shared_sm && azb_stack_depth(h->N) == 5)
        return fail(h, AZB_ERR_INVALID, "AZB_ASYNC_SHARED needs N <= 46 (larger trees take the whole SM's shared memory)");
    uint32_t group = shared_sm ? 8u : (B < 4096 ? 2u : 1u);  // pairs answer a tile faster; from 4096 roots on the model's throughput matters more
    if (const char *e = getenv("AZB_ASYNC_GROUP")) group = (uint32_t)strtoul(e, nullptr, 10);
    if (group == 0) return fail(h, AZB_ERR_INVALID, "AZB_ASYNC_GROUP must be positive");
    if (shared_sm) W = 0;
    // tree warps per CTA: 32, fewer when a large N needs more shared memory per warp (at most ~160 KB per SM, the rest is L1)
    const size_t lut_bytes = azb_tables_bytes(h->A, h->N, h->W), per_warp = (size_t)h->smem_words_per_warp * 4;
    uint32_t tree_warps = (uint32_t)std::max<size_t>(4, std::min<size_t>(AS_WARPS, (160 * 1024 - lut_bytes) / per_warp));
    if (azb_stack_depth(h->N) == 5) tree_warps = std::min<uint32_t>(tree_warps, AS_WIDE_TREE_WARPS);  // see azb_async_kernel
    if (shared_sm) tree_warps = SH_TREE_WARPS;
    // a tree CTA's scheduling table (azb_async.cuh): one entry per tree it owns
    const uint32_t n_tree_ctas_est = (uint32_t)prop.multiProcessorCount - (shared_sm ? 0u : W);
    if (!shared_sm && (int)W >= prop.multiProcessorCount) return fail(h, AZB_ERR_INVALID, "async_workers >= SM count");
    const uint32_t tab_slots = ((B + n_tree_ctas_est - 1u) / n_tree_ctas_est + 31u) & ~31u;
    const size_t tree_smem = (size_t)tree_warps * per_warp + lut_bytes + as_table_bytes(tab_slots);
    size_t bias_bytes = 0;
    for (int l = 0; l < 4; ++l) bias_bytes += (size_t)((h->tc.npad[l] + 31u) & ~31u) * 4;
    const size_t mlp_smem = (size_t)AS_STAGES * (1 + AS_ACC) * AS_TILE * TC_BK * 2 + 1024 + bias_bytes + 1024 + (size_t)AS_EPI_WARPS * AS_EPI_STG_BYTES;
    // every CTA of the one cooperative launch asks for the larger of the two roles' shared memory
    h->async_smem = std::max(tree_smem, mlp_smem);
    uint32_t cw[4] = {0, 0, 0, 0}, sh_stages = 0;
    if (shared_sm) {
        // a member's column slice of every layer: ceil(npad / G) rounded up to the MMA's N granularity
        uint32_t cwmax = 0, cwsum = 0;
        for (int l = 0; l < 4; ++l) {
            cw[l] = ((h->tc.npad[l] + group - 1u) / group + 15u) & ~15u;
            if (cw[l] > 256u) return fail(h, AZB_ERR_INVALID, "AZB_ASYNC_SHARED: %u columns per member exceed one 256-column MMA (raise AZB_ASYNC_GROUP)", cw[l]);
            cwmax = std::max(cwmax, cw[l]);
            cwsum += cw[l];
        }
        const size_t stage = (size_t)AS_TILE * TC_BK * 2 + (size_t)cwmax * TC_BK * 2;
        // trees | (1 KB alignment) operand ring | bias slices | (1 KB alignment) one staging tile per model warp
        sh_stages = SH_MAX_STAGES;
        auto need = [&](uint32_t st) { return tree_smem + 1024 + (size_t)st * stage + (size_t)cwsum * 4 + 1024 + 4u * SH_STG_BYTES; };
        while (sh_stages > 2u && need(sh_stages) > (size_t)prop.sharedMemPerBlockOptin - 2048) --sh_stages;
        h->async_smem = need(sh_stages);
    }
    int nb = 0, nb2 = 0, rc;
    switch (azb_stack_depth(h->N)) {
        case 3: rc = async_prepare_kernel<3, false>(h, &nb); if (!rc) rc = async_prepare_kernel<3, true>(h, &nb2); break;
        case 4: rc = async_prepare_kernel<4, false>(h, &nb); if (!rc) rc = async_prepare_kernel<4, true>(h, &nb2); break;
        default: rc = async_prepare_kernel<5, false>(h, &nb); if (!rc) rc = async_prepare_kernel<5, true>(h, &nb2); break;
    }
    if (rc) return rc;
    nb = std::min(nb, nb2);
    if (nb < 1) return fail(h, AZB_ERR_CUDA, "the async kernel does not fit on an SM (%zu bytes of shared memory)", h->async_smem);
    h->async_grid = nb * prop.multiProcessorCount;
    if ((int)W >= prop.multiProcessorCount || (int)W >= h->async_grid) return fail(h, AZB_ERR_INVALID, "async_workers >= SM count");
    const uint32_t n_model_groups = shared_sm ? (uint32_t)h->async_grid / group : W / group;
    if (shared_sm && (nb != 1 || n_model_groups == 0)) return fail(h, AZB_ERR_INVALID, "AZB_ASYNC_SHARED needs one CTA per SM and at least %u SMs", group);
    const uint32_t NW = (uint32_t)(h->async_grid - (int)W) * tree_warps;
    if ((uint32_t)(h->async_grid - (int)W) != n_tree_ctas_est)
        return fail(h, AZB_ERR_CUDA, "async kernel: %d CTAs where one per SM was expected", h->async_grid);
    AzbAsyncParams &P = h->asP;
    memset(&P, 0, sizeof(P));
    P.NT = 2 * ((B + AS_TILE - 1) / AS_TILE) + 2 * (shared_sm ? n_model_groups : W) + 8;
    P.n_workers = W;  // model CTAs (whole SMs)
    P.shared_sm = shared_sm ? 1u : 0u;
    for (int l = 0; l < 4; ++l) P.cw[l] = cw[l];
    P.sh_stages = sh_stages;
    P.tree_warps = tree_warps;
    P.tab_slots = tab_slots;
    // Inside a tree CTA (azb_async.cuh): up to two trees per warp a warp's own trees keep it busy exactly while the model
    // answers (walk A, walk B, A's priors are back), so static ownership loses nothing and its cheap wake-ups and the early
    // hand-over of the state vector win (6144 roots: 115 us per step against 125-133 with take-overs); beyond that — and
    // from one tree per warp on where the walk itself dominates the step (N >= 47: 16 tree warps per SM, 100+ us walks) —
    // free warps take over any runnable tree of their CTA
    P.steal = (B > 2u * NW || (azb_stack_depth(h->N) == 5 && B > NW)) ? 1u : 0u;
    if (const char *e = getenv("AZB_ASYNC_STEAL")) P.steal = atoi(e) != 0;
    // worker SMs per tile
    P.group = group;
    if (W % P.group) return fail(h, AZB_ERR_INVALID, "async_workers must be a multiple of the group size %u", P.group);
    if (n_model_groups > AS_MAX_GROUPS) return fail(h, AZB_ERR_INVALID, "more than %u model groups", (unsigned)AS_MAX_GROUPS);
    P.smem_words_per_warp = h->smem_words_per_warp;
    P.wide = h->tc.split ? 2u : 1u;
    P.ring_ld = P.wide * h->tc.kpad[0];
    h->async_timeout_base_ns = 2ull * 1000000000ull;
    if (const char *e = getenv("AZB_ASYNC_TIMEOUT_MS")) h->async_timeout_base_ns = strtoull(e, nullptr, 10) * 1000000ull;
    P.timeout_ns = h->async_timeout_base_ns;
    P.flush_ns = 4000ull;
    if (const char *e = getenv("AZB_ASYNC_FLUSH_NS")) P.flush_ns = strtoull(e, nullptr, 10);
    for (int l = 0; l < 4; ++l) {
        P.kpad[l] = h->tc.kpad[l];
        P.npad[l] = h->tc.npad[l];
        P.bias[l] = h->tc.bias[l];
    }
    int nbuf = 0;
    auto alloc = [&](void **p, size_t bytes) -> cudaError_t {
        cudaError_t e = cudaMalloc(p, bytes);
        if (e == cudaSuccess) {
            h->dev_bytes += bytes;
            h->async_bufs[nbuf++] = *p;
            e = cudaMemsetAsync(*p, 0, bytes, h->stream);
        }
        return e;
    };
    // everything a launch starts from zero sits in ONE slab (one memset per launch): state | tile counters | answer flags | debug
    {
        auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
        const size_t o_cnt = up(sizeof(AzbAsyncState)), o_ret = o_cnt + up((size_t)P.NT * 4), o_flag = o_ret + up((size_t)P.NT * 4),
                     o_dbg = o_flag + up((size_t)B * 4);
        h->async_zero_bytes = o_dbg + 32 * 8;
        uint8_t *slab = nullptr;
        CK(alloc((void **)&slab, h->async_zero_bytes));
        P.st = reinterpret_cast<AzbAsyncState *>(slab);
        P.tile_count = reinterpret_cast<uint32_t *>(slab + o_cnt);
        P.tile_retired = reinterpret_cast<uint32_t *>(slab + o_ret);
        P.h_flag = reinterpret_cast<uint32_t *>(slab + o_flag);
        P.dbg = reinterpret_cast<unsigned long long *>(slab + o_dbg);
    }
    CK(alloc((void **)&P.slot_tree, (size_t)P.NT * AS_TILE * 4));
    CK(alloc((void **)&P.ring, (size_t)P.NT * AS_TILE * P.ring_ld * 2));
    const uint32_t scratch_tiles = shared_sm ? n_model_groups : W;  // one 128-row scratch tile per group (whole-SM form: per worker)
    for (int l = 0; l < 3; ++l) CK(alloc((void **)&P.act[l], (size_t)scratch_tiles * AS_TILE * P.wide * h->tc.kpad[l + 1] * 2));
    azb_encode_fn enc = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", (void **)&enc, cudaEnableDefault, &qres) != cudaSuccess || !enc)
        return fail(h, AZB_ERR_CUDA, "cuTensorMapEncodeTiled is not available");
    const char *why = azb_tc_make_map(enc, &h->asM.ring, P.ring, (uint64_t)P.NT * AS_TILE, P.ring_ld, AS_TILE);
    for (int l = 0; l < 3 && !why; ++l)
        why = azb_tc_make_map(enc, &h->asM.act[l], P.act[l], (uint64_t)scratch_tiles * AS_TILE, P.wide * h->tc.kpad[l + 1], AS_TILE);
    for (int l = 0; l < 4 && !why; ++l)
        why = azb_tc_make_map(enc, &h->asM.w[l], h->tc.w[l], (uint64_t)(h->tc.npad[l] + 127u) / 128u * 128u, P.wide * h->tc.kpad[l], 128);
    for (int l = 0; l < 4 && !why && shared_sm; ++l)  // the same weights, fetched one member's column slice at a time
        why = azb_tc_make_map(enc, &h->asM.ws[l], h->tc.w[l], (uint64_t)(h->tc.npad[l] + 127u) / 128u * 128u, P.wide * h->tc.kpad[l], cw[l]);
    if (why) return fail(h, AZB_ERR_CUDA, "async tensor maps: %s", why);
    CK(cudaStreamSynchronize(h->stream));
    h->async_ready = true;
    return AZB_OK;
}

template <int D, bool C, bool PUCT>
static cudaError_t async_launch_sel(azb_handle *h) {
    void *args[] = {(void *)&h->L, (void *)&h->asP, (void *)&h->asM};
    return cudaLaunchCooperativeKernel((const void *)azb_async_kernel<D, C, PUCT>, dim3(h->async_grid), dim3(AS_THREADS), args,
                                       h->async_smem, h->stream);
}
template <int D, bool C>
static cudaError_t async_launch(azb_handle *h) {
    return h->cfg.selection == AZB_SELECT_PUCT ? async_launch_sel<D, C, true>(h) : async_launch_sel<D, C, false>(h);
}

// n_steps of every tree in ONE persistent cooperative kernel (tree CTAs + model CTAs), then one batched forward over
// the rows of the last step (whose add_actions is fused into the next launch, like the lock step's)
static int run_async(azb_handle *h, uint32_t n_steps) {
    int rc = async_create(h);
    if (rc) return rc;
    AzbAsyncParams &P = h->asP;
    CK(cudaMemsetAsync(P.st, 0, h->async_zero_bytes, h->stream));
    P.target_step = h->steps_done + n_steps;
    // watchdog, measured from the start of the launch: a step takes 0.1-1.2 ms at the supported sizes, so 2 s plus
    // 20 ms per step never fires on a healthy run, profiler replays included, and a stuck launch ends within seconds
    P.timeout_ns = h->async_timeout_base_ns + (unsigned long long)n_steps * 20000000ull;
    cudaError_t ce;
    switch (azb_stack_depth(h->N) * 2 + (h->count_full ? 1 : 0)) {
        case 6: ce = async_launch<3, false>(h); break;
        case 7: ce = async_launch<3, true>(h); break;
        case 8: ce = async_launch<4, false>(h); break;
        case 9: ce = async_launch<4, true>(h); break;
        case 10: ce = async_launch<5, false>(h); break;
        default: ce = async_launch<5, true>(h); break;
    }
    if (ce != cudaSuccess) return fail(h, AZB_ERR_CUDA, "async kernel launch: %s", cudaGetErrorString(ce));
    h->launches += 1;
    h->async_ran = true;
    // (the rows of the last step are answered inside the kernel too: no batched forward behind it)
    h->steps_done = P.target_step;
    h->pending_add = true;
    return AZB_OK;
}

extern "C" {

// one launch = every tree below the target advances by at most one step; then the model forward over the batch
static int enqueue_launch(azb_handle *h, uint32_t flags, uint32_t target) {
    int rc = launch_tree(h, flags, target);
    if (rc) return rc;
    if ((flags & AZB_F_ADD) && h->cfg.prior_mode == AZB_PRIOR_MLP)
        rc = mlp_forward(h, h->L.sv, h->L.sv_ld, h->L.h, h->L.h_ld, 0, h->L.B, h->stream);
    return rc;
}

static int enqueue_steps(azb_handle *h, uint32_t n_steps, uint32_t flags) {
    if (h->steps_done + n_steps > h->L.cap_steps)
        return fail(h, AZB_ERR_CAPACITY, "%u steps since azb_init_trees exceed max_steps", h->steps_done + n_steps);
    const uint32_t target = h->steps_done + n_steps;
    if (h->cfg.async_workers && n_steps >= 2 && flags == (AZB_F_ADD | AZB_F_ROLLOUT)) return run_async(h, n_steps);
    if (h->cfg.prior_mode == AZB_PRIOR_HASH && h->cfg.max_episodes == 0 && h->n_groups <= 1 && n_steps >= 2 &&
        flags == (AZB_F_ADD | AZB_F_ROLLOUT)) {
        // counter-hash priors need no model call, so nothing ties the trees together: ONE launch in which every warp takes
        // its tree through all n_steps steps (per-tree step clocks and cand[step][tree] as in the asynchronous kernel)
        int rc = launch_tree(h, flags | AZB_F_MULTI, target);
        if (rc) return rc;
        h->steps_done = target;
        h->pending_add = true;
        return AZB_OK;
    }
    if (h->cfg.max_episodes == 0 && n_steps) {
        // Lock-step launches (every tree advances exactly one step per launch).  Groups of trees advance on their own
        // streams: a group's launch only waits for its own slowest tree and its model forward overlaps the other
        // groups' walks.  AZB_GRAPH_STEPS steps of a group are replayed as one CUDA graph (the launch arguments do not
        // change from step to step), so the host issues one call per group per 8 steps instead of 5 per step.
        const bool mlp = (flags & AZB_F_ADD) && h->cfg.prior_mode == AZB_PRIOR_MLP;
        const bool grouped = h->n_groups > 1;
        if (grouped) {
            CK(cudaEventRecord(h->fork_event, h->stream));
            for (uint32_t g = 0; g < h->n_groups; ++g) CK(cudaStreamWaitEvent(h->gstream[g], h->fork_event, 0));
        }
        const uint32_t key = flags | (h->count_full ? 0x100u : 0u) | 0x1000u;
        for (uint32_t g = 0; g < h->n_groups; ++g) {
            cudaStream_t st = grouped ? h->gstream[g] : h->stream;
            const uint32_t t0 = g * h->group_trees, nt = std::min(h->group_trees, h->L.B - t0);
            auto one_step = [&]() -> int {
                int rc = launch_tree(h, flags, 0xffffffffu, -1, t0, nt, st);
                if (rc) return rc;
                if (mlp) rc = mlp_forward(h, h->L.sv, h->L.sv_ld, h->L.h, h->L.h_ld, t0, nt, st);
                return rc;
            };
            uint32_t left = n_steps;
            if (left >= AZB_GRAPH_STEPS) {
                if (!h->ggraph[g] || h->ggraph_key[g] != key) {
                    if (h->ggraph[g]) {
                        cudaGraphExecDestroy(h->ggraph[g]);
                        h->ggraph[g] = nullptr;
                    }
                    const uint64_t launches_before = h->launches;
                    cudaGraph_t graph = nullptr;
                    CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
                    int rc = AZB_OK;
                    for (uint32_t s = 0; s < AZB_GRAPH_STEPS && rc == AZB_OK; ++s) rc = one_step();
                    cudaError_t ce = cudaStreamEndCapture(st, &graph);
                    h->launches = launches_before;
                    if (rc) return rc;
                    if (ce != cudaSuccess) return fail(h, AZB_ERR_CUDA, "stream capture: %s", cudaGetErrorString(ce));
                    CK(cudaGraphInstantiate(&h->ggraph[g], graph, 0));
                    cudaGraphDestroy(graph);
                    h->ggraph_key[g] = key;
                }
                const uint64_t per_step = 1 + (mlp ? 4 : 0);
                while (left >= AZB_GRAPH_STEPS) {
                    CK(cudaGraphLaunch(h->ggraph[g], st));
                    h->launches += per_step * AZB_GRAPH_STEPS;
                    left -= AZB_GRAPH_STEPS;
                }
            }
            for (; left; --left) {
                int rc = one_step();
                if (rc) return rc;
            }
        }
        if (grouped)
            for (uint32_t g = 0; g < h->n_groups; ++g) {
                CK(cudaEventRecord(h->gevent[g], h->gstream[g]));
                CK(cudaStreamWaitEvent(h->stream, h->gevent[g], 0));
            }
        h->steps_done = target;
        h->pending_add = true;
        return AZB_OK;
    }
    for (uint32_t s = 0; s < n_steps; ++s) {
        int rc = enqueue_launch(h, flags, target);
        if (rc) return rc;
    }
    if (h->cfg.max_episodes) {
        // bounded episodes per launch: some trees may still be finishing their step
        for (;;) {
            AzbGlobals g;
            int rc = read_globals(h, &g);
            if (rc) return rc;
            if (g.n_behind == 0) break;
            for (int k = 0; k < 2; ++k) {
                rc = enqueue_launch(h, flags, target);
                if (rc) return rc;
            }
        }
    }
    h->steps_done = target;
    if (n_steps) h->pending_add = true;
    return AZB_OK;
}

// azb_step(h, 1, ...) in lock-step mode: the whole step — search kernel, model forward, argmin pass, read-back of the
// globals and of the (at most one) improvement record into pinned host memory — is ONE CUDA graph launch, so the
// per-step call of the reference's API (optimizer/mod.rs:121) costs one launch and one synchronisation.
static int step_once_graph(azb_handle *h, azb_improvement *improvements, uint32_t cap, uint32_t *n_improved) {
    const uint32_t flags = AZB_F_ADD | AZB_F_ROLLOUT;
    const bool mlp = h->cfg.prior_mode == AZB_PRIOR_MLP;
    const uint32_t key = 0x2000u | (h->count_full ? 0x100u : 0u);
    if (!h->step_graph || h->step_graph_key != key) {
        if (h->step_graph) {
            cudaGraphExecDestroy(h->step_graph);
            h->step_graph = nullptr;
        }
        const uint64_t launches_before = h->launches;
        cudaGraph_t graph = nullptr;
        CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
        int rc = launch_tree(h, flags, 0xffffffffu);
        if (rc == AZB_OK && mlp) rc = mlp_forward(h, h->L.sv, h->L.sv_ld, h->L.h, h->L.h_ld, 0, h->L.B, h->stream);
        cudaError_t cc = cudaSuccess;  // first failure inside the capture region
        if (rc == AZB_OK) {
            azb_argmin1_kernel<<<1, 256, 0, h->stream>>>(h->L);
            cc = cudaGetLastError();
            if (cc == cudaSuccess)
                cc = cudaMemcpyAsync(h->pin_g, h->L.g, offsetof(AzbGlobals, argmin_state), cudaMemcpyDeviceToHost, h->stream);
            if (cc == cudaSuccess)
                cc = cudaMemcpyAsync(h->pin_log, h->L.log, sizeof(azb_improvement), cudaMemcpyDeviceToHost, h->stream);
        }
        cudaError_t ce = cudaStreamEndCapture(h->stream, &graph);
        h->launches = launches_before;
        if (rc || cc != cudaSuccess || ce != cudaSuccess) {
            if (graph) cudaGraphDestroy(graph);
            if (rc) return rc;
            return fail(h, AZB_ERR_CUDA, "stream capture of the single-step graph: %s", cudaGetErrorString(cc != cudaSuccess ? cc : ce));
        }
        CK(cudaGraphInstantiate(&h->step_graph, graph, 0));
        cudaGraphDestroy(graph);
        h->step_graph_key = key;
    }
    // stale pinned data must not read as a result: the graph's last node rewrites both words, or the check below fires
    h->pin_g->err = 0xffffffffu;
    h->pin_g->next_slot = 0xffffffffu;
    CK(cudaGraphLaunch(h->step_graph, h->stream));
    h->launches += 2 + (mlp ? 4 : 0);
    h->steps_done += 1;
    h->argmin_from = h->steps_done + 1;
    h->poll_next = h->argmin_from;
    h->poll_best_valid = false;
    h->pending_add = true;
    CK(cudaStreamSynchronize(h->stream));
    const AzbGlobals &g = *h->pin_g;
    if (g.err == 0xffffffffu || g.next_slot != h->argmin_from)
        return fail(h, AZB_ERR_CUDA, "the single-step graph did not deliver its result (a node of the graph failed)");
    if (g.err) return fail(h, (int)g.err, "%s (tree %u, step %u)", azb_strerror((int)g.err), g.err_tree, g.err_step);
    if (n_improved) *n_improved = g.n_improved;
    if (improvements && cap && g.n_improved) improvements[0] = *h->pin_log;
    h->improved_last_rollout = (int)g.improved_last;
    return AZB_OK;
}

int azb_step(azb_handle *h, uint32_t n_steps, azb_improvement *improvements, uint32_t cap, uint32_t *n_improved) {
    if (!h) return AZB_ERR_INVALID;
    if (!h->trees_init) return fail(h, AZB_ERR_STATE, "azb_init_trees has not been called");
    CK(cudaSetDevice(h->cfg.device));
    if (n_steps == 1 && h->cfg.max_episodes == 0 && h->n_groups == 1 && h->argmin_from == h->steps_done + 1 &&
        h->steps_done + 1 <= h->L.cap_steps)
        return step_once_graph(h, improvements, cap, n_improved);
    CK(cudaMemsetAsync(&h->L.g->n_improved, 0, 4, h->stream));
    int rc = enqueue_steps(h, n_steps, AZB_F_ADD | AZB_F_ROLLOUT);
    if (rc) return rc;
    rc = run_argmin(h, h->steps_done + 1);
    if (rc) return rc;
    AzbGlobals g;
    rc = read_globals(h, &g);
    if (rc) return rc;
    if (n_improved) *n_improved = g.n_improved;
    const uint32_t take = std::min(std::min(g.n_improved, cap), h->L.log_cap);
    if (improvements && take) {
        static_assert(sizeof(AzbImprovementDev) == sizeof(azb_improvement), "log record layout");
        CK(cudaMemcpyAsync(improvements, h->L.log, (size_t)take * sizeof(azb_improvement), cudaMemcpyDeviceToHost,
                           h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    h->improved_last_rollout = (int)g.improved_last;
    return AZB_OK;
}

// enqueue n_steps without waiting (several handles on one GPU can then run concurrently); azb_step(h, 0, ...) or any
// reading call completes them
int azb_step_enqueue(azb_handle *h, uint32_t n_steps) {
    if (!h) return AZB_ERR_INVALID;
    if (!h->trees_init) return fail(h, AZB_ERR_STATE, "azb_init_trees has not been called");
    if (h->cfg.max_episodes) return fail(h, AZB_ERR_INVALID, "azb_step_enqueue needs max_episodes = 0");
    CK(cudaSetDevice(h->cfg.device));
    if (h->steps_done + n_steps > h->L.cap_steps)
        return fail(h, AZB_ERR_CAPACITY, "%u steps since azb_init_trees exceed max_steps", h->steps_done + n_steps);
    // candidate rows of these steps: "not written yet" (a tree's entry is (ord(c), node) once it has finished the step,
    // (0xffffffff, 0) for an exhausted root) — what azb_step_poll waits on
    if (n_steps)
        CK(cudaMemsetAsync(h->L.cand + (size_t)(h->steps_done + 1) * h->L.B, 0xff, (size_t)n_steps * h->L.B * sizeof(uint2), h->stream));
    return enqueue_steps(h, n_steps, AZB_F_ADD | AZB_F_ROLLOUT);
}

// The result of the next enqueued step that has not been reported yet, as soon as EVERY tree has finished that step —
// while later steps are still running (trees are independent, so on the asynchronous path they run ahead of the
// caller).  This is par_roll_out_episodes' per-step return value (optimizer/mod.rs:121-191, ArgminImprovement) at the
// speed of the fused loop: the host reads the step's candidate row (8 B per tree) on a copy stream and applies
// par_update_argmmim_data's rule itself (first minimum over trees, strictly below the running best: :194-246).
// After the last step azb_step(h, 0, ...) completes the batch (device-side argmin state, log, error check); the
// improvements it logs are exactly the ones reported here.
int azb_step_poll(azb_handle *h, azb_improvement *out, int *improved) {
    if (!h || !improved) return AZB_ERR_INVALID;
    if (!h->trees_init) return fail(h, AZB_ERR_STATE, "azb_init_trees has not been called");
    if (h->poll_next > h->steps_done || h->poll_next < h->argmin_from)
        return fail(h, AZB_ERR_STATE, "no enqueued step is waiting to be reported (azb_step_enqueue first)");
    CK(cudaSetDevice(h->cfg.device));
    const uint32_t B = h->L.B;
    if (!h->poll_stream) CK(cudaStreamCreateWithFlags(&h->poll_stream, cudaStreamNonBlocking));
    if (!h->poll_pin) CK(cudaMallocHost((void **)&h->poll_pin, (size_t)B * sizeof(uint2)));
    if (!h->poll_word) CK(cudaMallocHost((void **)&h->poll_word, 16));
    if (!h->poll_best_valid) {  // the running best is only rewritten by the argmin pass that ends a batch
        CK(cudaMemcpyAsync(h->poll_word, &h->L.g->best_c, 4, cudaMemcpyDeviceToHost, h->poll_stream));
        CK(cudaStreamSynchronize(h->poll_stream));
        h->poll_best = h->poll_word[0];
        h->poll_best_valid = true;
    }
    const uint2 *src = h->L.cand + (size_t)h->poll_next * B;
    bool finished = false;  // the enqueued work has ended: one more look at the row decides
    for (;;) {
        CK(cudaMemcpyAsync(h->poll_pin, src, (size_t)B * sizeof(uint2), cudaMemcpyDeviceToHost, h->poll_stream));
        CK(cudaStreamSynchronize(h->poll_stream));
        bool complete = true;
        for (uint32_t t = 0; t < B; ++t)
            if (h->poll_pin[t].y == 0xffffffffu) {
                complete = false;
                break;
            }
        if (complete) break;
        if (finished) {  // a tree stopped before this step (capacity, NaN, watchdog): report what the device says
            int rc = check_device_error(h);
            return rc ? rc : fail(h, AZB_ERR_CUDA, "step %u was not finished by every tree", h->poll_next - 1u);
        }
        const cudaError_t q = cudaStreamQuery(h->stream);
        if (q == cudaSuccess) finished = true;
        else if (q != cudaErrorNotReady) return fail(h, AZB_ERR_CUDA, "%s", cudaGetErrorString(q));
    }
    unsigned long long m = ~0ull;
    for (uint32_t t = 0; t < B; ++t) {
        const unsigned long long k = ((unsigned long long)h->poll_pin[t].x << 32) | t;
        m = k < m ? k : m;
    }
    const uint32_t oc = (uint32_t)(m >> 32), tree = (uint32_t)m;
    *improved = oc < h->poll_best ? 1 : 0;
    if (*improved) h->poll_best = oc;
    if (out) {
        out->step = h->poll_next - 1u;
        out->tree = tree;
        out->node = h->poll_pin[tree].y;
        out->eval = azb_ord2f(oc);
    }
    h->poll_next += 1u;
    return AZB_OK;
}

int azb_step_timed(azb_handle *h, uint32_t n_steps, float *ms, uint32_t *n_improved) {
    if (!h) return AZB_ERR_INVALID;
    if (!h->trees_init) return fail(h, AZB_ERR_STATE, "azb_init_trees has not been called");
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaMemsetAsync(&h->L.g->n_improved, 0, 4, h->stream));
    CK(cudaEventRecord(h->ev0, h->stream));
    int rc = enqueue_steps(h, n_steps, AZB_F_ADD | AZB_F_ROLLOUT);
    if (rc) return rc;
    rc = run_argmin(h, h->steps_done + 1);
    if (rc) return rc;
    CK(cudaEventRecord(h->ev1, h->stream));
    CK(cudaEventSynchronize(h->ev1));
    if (ms) CK(cudaEventElapsedTime(ms, h->ev0, h->ev1));
    AzbGlobals g;
    rc = read_globals(h, &g);
    if (rc) return rc;
    if (n_improved) *n_improved = g.n_improved;
    return AZB_OK;
}

int azb_step_profile(azb_handle *h, uint32_t n_steps, float *tree_ms, float *mlp_ms) {
    if (!h || n_steps == 0) return AZB_ERR_INVALID;
    if (!h->trees_init) return fail(h, AZB_ERR_STATE, "azb_init_trees has not been called");
    if (h->steps_done + n_steps > h->L.cap_steps) return fail(h, AZB_ERR_CAPACITY, "steps exceed max_steps");
    CK(cudaSetDevice(h->cfg.device));
    std::vector<cudaEvent_t> ev;
    auto mark = [&]() {
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, h->stream);
        ev.push_back(e);
    };
    const bool mlp = h->cfg.prior_mode == AZB_PRIOR_MLP;
    const uint32_t target = h->steps_done + n_steps;
    int rc = AZB_OK;
    mark();
    uint32_t launched = 0;
    for (;;) {
        for (uint32_t s = 0; s < n_steps && rc == AZB_OK; ++s) {
            rc = launch_tree(h, AZB_F_ADD | AZB_F_ROLLOUT, target);
            mark();
            if (rc == AZB_OK && mlp) rc = mlp_forward(h, h->L.sv, h->L.sv_ld, h->L.h, h->L.h_ld, 0, h->L.B, h->stream);
            mark();
            ++launched;
        }
        if (rc || !h->cfg.max_episodes) break;
        AzbGlobals g;
        rc = read_globals(h, &g);
        if (rc || g.n_behind == 0) break;
        n_steps = 2;  // catch-up launches
    }
    cudaStreamSynchronize(h->stream);
    double t_tree = 0, t_mlp = 0;
    if (rc == AZB_OK)
        for (uint32_t s = 0; s < launched; ++s) {
            float a = 0, b = 0;
            cudaEventElapsedTime(&a, ev[2 * s], ev[2 * s + 1]);
            cudaEventElapsedTime(&b, ev[2 * s + 1], ev[2 * s + 2]);
            t_tree += a;
            t_mlp += b;
        }
    for (auto &e : ev) cudaEventDestroy(e);
    if (rc) return rc;
    h->steps_done = target;
    h->pending_add = true;
    if (tree_ms) *tree_ms = (float)t_tree;
    if (mlp_ms) *mlp_ms = (float)t_mlp;
    rc = run_argmin(h, h->steps_done + 1);
    if (rc) return rc;
    return check_device_error(h);
}

int azb_rollout_host(azb_handle *h, float *state_vecs) {
    if (!h || !state_vecs) return AZB_ERR_INVALID;
    if (!h->trees_init) return fail(h, AZB_ERR_STATE, "azb_init_trees has not been called");
    if (h->pending_add) return fail(h, AZB_ERR_STATE, "azb_add_actions_host must follow azb_rollout_host");
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaMemsetAsync(&h->L.g->n_improved, 0, 4, h->stream));
    int rc = enqueue_steps(h, 1, AZB_F_ROLLOUT);
    if (rc) return rc;
    rc = run_argmin(h, h->steps_done + 1);
    if (rc) return rc;
    h->host_add_pending = true;
    rc = copy_state_vecs(h, state_vecs);
    if (rc) return rc;
    AzbGlobals g;
    rc = read_globals(h, &g);
    if (rc) return rc;
    h->improved_last_rollout = (int)g.improved_last;
    return AZB_OK;
}

int azb_add_actions_host(azb_handle *h, const float *h_theta, int *improved) {
    if (!h || !h_theta) return AZB_ERR_INVALID;
    if (!h->pending_add) return fail(h, AZB_ERR_STATE, "azb_rollout_host has not been called");
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaMemcpy2DAsync(h->L.h, (size_t)h->L.h_ld * 4, h_theta, (size_t)h->A * 4, (size_t)h->A * 4, h->L.B,
                         cudaMemcpyHostToDevice, h->stream));
    int rc = launch_tree(h, AZB_F_ADD, h->steps_done, AZB_PRIOR_INJECTED);
    if (rc) return rc;
    h->pending_add = false;
    h->host_add_pending = false;
    rc = check_device_error(h);
    if (rc) return rc;
    if (improved) *improved = h->improved_last_rollout;
    return AZB_OK;
}

// ---- stand-alone cost kernel ----
// the cost kernel on m trees of n vertices (azb_trees_within evaluates every level below N with it)
static void launch_cost_n(azb_handle *h, const uint8_t *dev_parents, uint32_t m, uint32_t n, double *l1, uint32_t *mu, float *c,
                          uint32_t *err) {
    const uint32_t threads = 256, blocks = (m + 7) / 8;
    switch (azb_stack_depth(n)) {
        case 3: azb_cost_kernel<3><<<blocks, threads, 0, h->stream>>>(dev_parents, m, n, h->L.c_lower, h->L.slope, l1, mu, c, err); break;
        case 4: azb_cost_kernel<4><<<blocks, threads, 0, h->stream>>>(dev_parents, m, n, h->L.c_lower, h->L.slope, l1, mu, c, err); break;
        default: azb_cost_kernel<5><<<blocks, threads, 0, h->stream>>>(dev_parents, m, n, h->L.c_lower, h->L.slope, l1, mu, c, err); break;
    }
    h->launches += 1;
}

// the cost kernel's outputs for m trees, carved from a call's scratch
struct CostOut {
    double *l1;
    uint32_t *mu;
    float *c;
    uint32_t *err;
    void take(Carve &cv, size_t m) {
        l1 = cv.take<double>(m);
        mu = cv.take<uint32_t>(m);
        c = cv.take<float>(m);
        err = cv.take<uint32_t>(1);
    }
};

// The cost kernel of azb_eval_costs on m device parent arrays of n vertices into d, then the copies of whichever of the
// parent arrays, lambda_1, mu and eval the caller asks for (the non-null destinations) and of the error word, all on the
// library stream; t0 and t1, when given, are recorded around the kernel.  The caller synchronises and maps *err.
static int cost_tail(azb_handle *h, const uint8_t *d_par, uint32_t m, uint32_t n, const CostOut &d, cudaEvent_t t0, cudaEvent_t t1,
                     uint8_t *parents, double *lambda1, uint32_t *mu, float *eval, uint32_t *err) {
    CK(cudaMemsetAsync(d.err, 0, 4, h->stream));
    if (t0) CK(cudaEventRecord(t0, h->stream));
    launch_cost_n(h, d_par, m, n, d.l1, d.mu, d.c, d.err);
    CK(cudaGetLastError());
    if (t1) CK(cudaEventRecord(t1, h->stream));
    if (parents) CK(cudaMemcpyAsync(parents, d_par, (size_t)m * n, cudaMemcpyDeviceToHost, h->stream));
    if (lambda1) CK(cudaMemcpyAsync(lambda1, d.l1, (size_t)m * 8, cudaMemcpyDeviceToHost, h->stream));
    if (mu) CK(cudaMemcpyAsync(mu, d.mu, (size_t)m * 4, cudaMemcpyDeviceToHost, h->stream));
    if (eval) CK(cudaMemcpyAsync(eval, d.c, (size_t)m * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(err, d.err, 4, cudaMemcpyDeviceToHost, h->stream));
    return AZB_OK;
}

static int eval_costs_dev(azb_handle *h, const uint8_t *parents, uint32_t m, double *lambda1, uint32_t *mu, float *c,
                          float *ms) {
    uint8_t *d_par = nullptr;
    CostOut d;
    int rc = scratch(h, [&](Carve &cv) {
        d_par = cv.take<uint8_t>((size_t)m * h->N);
        d.take(cv, m);
    });
    if (rc) return rc;
    CK(cudaMemcpyAsync(d_par, parents, (size_t)m * h->N, cudaMemcpyHostToDevice, h->stream));
    uint32_t err = 0;
    rc = cost_tail(h, d_par, m, h->N, d, h->ev0, h->ev1, nullptr, lambda1, mu, c, &err);
    if (rc) return rc;
    CK(cudaStreamSynchronize(h->stream));
    if (ms) CK(cudaEventElapsedTime(ms, h->ev0, h->ev1));
    if (err) return fail(h, (int)err, "%s", azb_strerror((int)err));
    return AZB_OK;
}

int azb_eval_costs(azb_handle *h, const uint8_t *parents, uint32_t m, double *lambda1, uint32_t *mu, float *c,
                   float *ms) {
    if (!h || !parents || m == 0) return AZB_ERR_INVALID;
    for (uint32_t i = 0; i < m; ++i)
        for (uint32_t v = 1; v < h->N; ++v)
            if (parents[(size_t)i * h->N + v] >= v)
                return fail(h, AZB_ERR_INVALID, "tree %u: parents[%u] is not < %u", i, v, v);
    CK(cudaSetDevice(h->cfg.device));
    return eval_costs_dev(h, parents, m, lambda1, mu, c, ms);
}
}  // extern "C"

// ---- certificates of c21 keys against a bound (azb_certify.cuh) ----
// the bound of azb_certify_keys and azb_trees_within_proof as the kernels take it, for trees on N vertices
static AzbCertBound cert_bound(double bound, uint32_t N) {
    AzbCertBound b{bound, N, bound < 0.0 ? 1 : 0, 0};
    uint32_t s = 0;
    while ((s + 1) * (s + 1) <= N - 1) ++s;
    // (bound - 1)^2 = N - 1 for a bound >= 0 needs N - 1 = s^2 and bound = s + 1
    b.tie = b.dflt || (s * s == N - 1 && bound == (double)(s + 1));
    return b;
}

template <class Kernel>
static int cert_smem(azb_handle *h, Kernel kernel, uint32_t n) {
    const size_t smem = azb_certify_smem(n);
    if (smem > 48 * 1024) CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return AZB_OK;
}

// azb_certify_kernel on m device parent arrays of n vertices with their lambda_1 from the cost kernel
static int launch_certify(azb_handle *h, const uint8_t *d_par, uint32_t m, uint32_t n, const double *d_l1, const AzbCertBound &b,
                          double *lo, double *hi, uint32_t *mu, int8_t *verdict, unsigned long long *tally) {
    int rc = cert_smem(h, azb_certify_kernel, n);
    if (rc) return rc;
    azb_certify_kernel<<<(m + AZB_CERT_THREADS - 1) / AZB_CERT_THREADS, AZB_CERT_THREADS, azb_certify_smem(n), h->stream>>>(
        d_par, m, n, d_l1, b, lo, hi, mu, verdict, tally);
    h->launches += 1;
    CK(cudaGetLastError());
    return AZB_OK;
}

extern "C" int azb_certify_keys(azb_handle *h, const uint8_t *parents, uint32_t m, double bound, double *lambda1_lo,
                                double *lambda1_hi, uint32_t *mu, int8_t *verdict, float *ms) {
    if (!h || !parents || m == 0) return AZB_ERR_INVALID;
    if (std::isnan(bound)) return fail(h, AZB_ERR_INVALID, "azb_certify_keys: the bound is NaN");
    const uint32_t N = h->N;
    for (uint32_t i = 0; i < m; ++i)
        for (uint32_t v = 1; v < N; ++v)
            if (parents[(size_t)i * N + v] >= v) return fail(h, AZB_ERR_INVALID, "tree %u: parents[%u] is not < %u", i, v, v);
    CK(cudaSetDevice(h->cfg.device));
    uint8_t *d_par = nullptr;
    CostOut d;
    double *d_lo = nullptr, *d_hi = nullptr;
    uint32_t *d_mu = nullptr;
    int8_t *d_v = nullptr;
    int rc = scratch(h, [&](Carve &cv) {
        d_par = cv.take<uint8_t>((size_t)m * N);
        d.take(cv, m);
        d_lo = cv.take<double>(m);
        d_hi = cv.take<double>(m);
        d_mu = cv.take<uint32_t>(m);
        d_v = cv.take<int8_t>(m);
    });
    if (rc) return rc;
    CK(cudaMemcpyAsync(d_par, parents, (size_t)m * N, cudaMemcpyHostToDevice, h->stream));
    uint32_t err = 0;
    rc = cost_tail(h, d_par, m, N, d, h->ev0, nullptr, nullptr, nullptr, nullptr, nullptr, &err);
    if (rc) return rc;
    rc = launch_certify(h, d_par, m, N, d.l1, cert_bound(bound, N), d_lo, d_hi, d_mu, d_v, nullptr);
    if (rc) return rc;
    CK(cudaEventRecord(h->ev1, h->stream));
    if (lambda1_lo) CK(cudaMemcpyAsync(lambda1_lo, d_lo, (size_t)m * 8, cudaMemcpyDeviceToHost, h->stream));
    if (lambda1_hi) CK(cudaMemcpyAsync(lambda1_hi, d_hi, (size_t)m * 8, cudaMemcpyDeviceToHost, h->stream));
    if (mu) CK(cudaMemcpyAsync(mu, d_mu, (size_t)m * 4, cudaMemcpyDeviceToHost, h->stream));
    if (verdict) CK(cudaMemcpyAsync(verdict, d_v, m, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (ms) CK(cudaEventElapsedTime(ms, h->ev0, h->ev1));
    if (err) return fail(h, (int)err, "%s", azb_strerror((int)err));
    return AZB_OK;
}
extern "C" {

// ---- stand-alone cost + action kinds of connected bitset graphs (SURVEY 8(f) row 3) ----
}  // extern "C"

// shared by the B32 and B64 entries: the scratch, the copies, the timing and the error words; `launch` enqueues the kernel
template <typename W, typename Launch>
static int eval_graph_costs_dev(azb_handle *h, const char *fn, const W *nbr, uint32_t m, uint32_t n, double *lambda1,
                                uint32_t *mu, uint32_t *kinds, float *ms, Launch launch) {
    // loops, asymmetric neighbourhoods, neighbours >= N and disconnected inputs are found by the kernel itself
    CK(cudaSetDevice(h->cfg.device));
    const uint32_t kw = (n * (n - 1) + 31) / 32;
    double *d_l1 = nullptr;
    W *d_nbr = nullptr;
    uint32_t *d_mu = nullptr, *d_kinds = nullptr, *d_err = nullptr;
    int rc = scratch(h, [&](Carve &cv) {
        d_l1 = cv.take<double>(m);
        d_nbr = cv.take<W>((size_t)m * n);
        d_mu = cv.take<uint32_t>(m);
        d_kinds = cv.take<uint32_t>((size_t)m * kw);
        d_err = cv.take<uint32_t>(2);
    });
    if (rc) return rc;
    cudaError_t ce = cudaMemcpyAsync(d_nbr, nbr, (size_t)m * n * sizeof(W), cudaMemcpyHostToDevice, h->stream);
    const uint32_t err0[2] = {0u, 0xffffffffu};  // [0] bit AZB_ERR_* per kind of failure, [1] first rejected graph
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(d_err, err0, 8, cudaMemcpyHostToDevice, h->stream);
    if (ce == cudaSuccess) ce = cudaEventRecord(h->ev0, h->stream);
    if (ce == cudaSuccess) {
        ce = launch(d_nbr, kw, d_l1, d_mu, d_kinds, d_err);
        h->launches += 1;
        if (ce == cudaSuccess) ce = cudaGetLastError();
    }
    if (ce == cudaSuccess) ce = cudaEventRecord(h->ev1, h->stream);
    uint32_t err[2] = {0u, 0u};
    if (ce == cudaSuccess && lambda1) ce = cudaMemcpyAsync(lambda1, d_l1, (size_t)m * 8, cudaMemcpyDeviceToHost, h->stream);
    if (ce == cudaSuccess && mu) ce = cudaMemcpyAsync(mu, d_mu, (size_t)m * 4, cudaMemcpyDeviceToHost, h->stream);
    if (ce == cudaSuccess && kinds) ce = cudaMemcpyAsync(kinds, d_kinds, (size_t)m * kw * 4, cudaMemcpyDeviceToHost, h->stream);
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(err, d_err, 8, cudaMemcpyDeviceToHost, h->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(h->stream);
    if (ce == cudaSuccess && ms) ce = cudaEventElapsedTime(ms, h->ev0, h->ev1);
    if (ce != cudaSuccess) return fail(h, AZB_ERR_CUDA, "%s: %s", fn, cudaGetErrorString(ce));
    if (err[0] & (1u << AZB_ERR_INVALID))
        return fail(h, AZB_ERR_INVALID, "graph %u is not a connected simple graph (a loop, a neighbour >= N, asymmetric neighbourhoods, or disconnected)", err[1]);
    if (err[0] & (1u << AZB_ERR_LAMBDA)) return fail(h, AZB_ERR_LAMBDA, "%s", azb_strerror(AZB_ERR_LAMBDA));
    return AZB_OK;
}

extern "C" {

int azb_eval_graph_costs(azb_handle *h, const uint32_t *nbr, uint32_t m, uint32_t n, double *lambda1, uint32_t *mu,
                         uint32_t *kinds, float *ms) {
    if (!h || !nbr || m == 0) return AZB_ERR_INVALID;
    if (n < 2 || n > 32) return fail(h, AZB_ERR_INVALID, "graphs have 2..32 vertices (B32 neighbourhoods), got %u", n);
    return eval_graph_costs_dev(h, "azb_eval_graph_costs", nbr, m, n, lambda1, mu, kinds, ms,
                                [&](const uint32_t *d_nbr, uint32_t kw, double *d_l1, uint32_t *d_mu, uint32_t *d_kinds, uint32_t *d_err) {
        const uint32_t blocks = (m + AZG_WARPS - 1) / AZG_WARPS, smem = AZG_WARPS * azg_warp_bytes(n);
        if (azg_packed(n)) azb_graph_cost_kernel<true><<<blocks, AZG_WARPS * 32, smem, h->stream>>>(d_nbr, m, n, kw, d_l1, d_mu, d_kinds, d_err);
        else azb_graph_cost_kernel<false><<<blocks, AZG_WARPS * 32, smem, h->stream>>>(d_nbr, m, n, kw, d_l1, d_mu, d_kinds, d_err);
        return cudaSuccess;
    });
}

}  // extern "C"

// warps per CTA of the B64 kernel: the count among 1, 2, 4 with the most resident warps per SM for this N's
// shared-memory footprint (19.5 KB per warp at N = 64, 7.6 KB at N = 33); ties go to the larger CTA
template <bool PACKED>
static cudaError_t launch_graph_cost64(azb_handle *h, const uint64_t *d_nbr, uint32_t m, uint32_t n, uint32_t kw, double *d_l1,
                                       uint32_t *d_mu, uint32_t *d_kinds, uint32_t *d_err) {
    const uint32_t bytes = azg64_warp_bytes(n);
    uint32_t warps = 1;
    int best = 0;
    for (uint32_t wc = 1; wc <= AZG64_MAX_WARPS; wc *= 2) {
        cudaError_t ce = cudaFuncSetAttribute(azb_graph_cost64_kernel<PACKED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(wc * bytes));
        int blocks = 0;
        if (ce == cudaSuccess) ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, azb_graph_cost64_kernel<PACKED>, (int)wc * 32, wc * bytes);
        if (ce != cudaSuccess) return ce;
        if (blocks * (int)wc >= best) {
            best = blocks * (int)wc;
            warps = wc;
        }
    }
    cudaError_t ce = cudaFuncSetAttribute(azb_graph_cost64_kernel<PACKED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(warps * bytes));
    if (ce != cudaSuccess) return ce;
    azb_graph_cost64_kernel<PACKED><<<(m + warps - 1) / warps, warps * 32, warps * bytes, h->stream>>>(d_nbr, m, n, kw, d_l1, d_mu, d_kinds, d_err);
    return cudaSuccess;
}

extern "C" {

int azb_eval_graph_costs64(azb_handle *h, const uint64_t *nbr, uint32_t m, uint32_t n, double *lambda1, uint32_t *mu,
                           uint32_t *kinds, float *ms) {
    if (!h || !nbr || m == 0) return AZB_ERR_INVALID;
    if (n < 2 || n > 64) return fail(h, AZB_ERR_INVALID, "graphs have 2..64 vertices (B64 neighbourhoods), got %u", n);
    // every n runs the B64 kernel, n <= 32 included: one code path, and bits 32..63 are validated like any other
    return eval_graph_costs_dev(h, "azb_eval_graph_costs64", nbr, m, n, lambda1, mu, kinds, ms,
                                [&](const uint64_t *d_nbr, uint32_t kw, double *d_l1, uint32_t *d_mu, uint32_t *d_kinds, uint32_t *d_err) {
        return azg_packed(n) ? launch_graph_cost64<true>(h, d_nbr, m, n, kw, d_l1, d_mu, d_kinds, d_err)
                             : launch_graph_cost64<false>(h, d_nbr, m, n, kw, d_l1, d_mu, d_kinds, d_err);
    });
}

// ---- results ----
int azb_get_argmin(azb_handle *h, uint8_t *parents, uint32_t *permitted, double *lambda1, uint32_t *mu, float *eval) {
    if (!h) return AZB_ERR_INVALID;
    if (!h->trees_init) return fail(h, AZB_ERR_STATE, "azb_init_trees has not been called");
    CK(cudaSetDevice(h->cfg.device));
    CostOut d;
    int rc = scratch(h, [&](Carve &cv) { d.take(cv, 1); });
    if (rc) return rc;
    if (!h->pin_rg) {
        CK(cudaMallocHost((void **)&h->pin_rg, sizeof(AzbGlobals)));
        CK(cudaMallocHost((void **)&h->pin_abort, 16));
    }
    if (!h->pin_cost) CK(cudaMallocHost((void **)&h->pin_cost, 32));
    // *cost = space.cost(state); *eval = space.evaluate(cost)  (optimizer/mod.rs:240-241): the cost kernel reads the argmin
    // state where the argmin pass left it, and everything comes back behind ONE synchronisation into pinned memory
    uint32_t *pc = h->pin_cost;
    rc = cost_tail(h, reinterpret_cast<const uint8_t *>(h->L.g->argmin_state), 1, h->N, d, nullptr, nullptr, nullptr,
                   reinterpret_cast<double *>(pc), pc + 2, reinterpret_cast<float *>(pc + 3), pc + 4);
    if (rc) return rc;
    CK(cudaMemcpyAsync(h->pin_rg, h->L.g, sizeof(AzbGlobals), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const AzbGlobals &g = *h->pin_rg;
    if (parents) memcpy(parents, g.argmin_state, h->N);
    if (permitted) memcpy(permitted, g.argmin_state + 16, (size_t)h->W * 4);
    if (h->pin_cost[4]) return fail(h, (int)h->pin_cost[4], "%s", azb_strerror((int)h->pin_cost[4]));
    if (lambda1) memcpy(lambda1, h->pin_cost, 8);
    if (mu) *mu = h->pin_cost[2];
    if (eval) memcpy(eval, h->pin_cost + 3, 4);
    return AZB_OK;
}

int azb_get_walkers(azb_handle *h, uint8_t *parents, uint32_t *permitted, uint32_t *path, uint32_t *pos,
                    uint32_t *path_len) {
    if (!h) return AZB_ERR_INVALID;
    if (!h->trees_init) return fail(h, AZB_ERR_STATE, "azb_init_trees has not been called");
    CK(cudaSetDevice(h->cfg.device));
    int rc = flush_pending(h);
    if (rc) return rc;
    const uint32_t N = h->N, W = h->W, PW = h->PW, WS = h->WS, B = h->L.B;
    std::vector<uint32_t> blk((size_t)B * WS);
    CK(cudaMemcpyAsync(blk.data(), h->L.walker, blk.size() * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (uint32_t i = 0; i < B; ++i) {
        const uint32_t *w = blk.data() + (size_t)i * WS;
        if (parents) memcpy(parents + (size_t)i * N, w + WK_HDR, N);
        if (permitted) memcpy(permitted + (size_t)i * W, w + WK_HDR + PW, (size_t)W * 4);
        if (path) memcpy(path + (size_t)i * W, w + WK_HDR + PW + W, (size_t)W * 4);
        if (pos) pos[i] = w[WK_POS];
        if (path_len) path_len[i] = w[WK_DEPTH];
    }
    return check_device_error(h);
}

int azb_tree_sizes(azb_handle *h, uint32_t tree, uint32_t *n_nodes, uint32_t *n_arcs, uint32_t *n_preds) {
    if (!h || tree >= h->L.B) return AZB_ERR_INVALID;
    if (!h->trees_init) return fail(h, AZB_ERR_STATE, "azb_init_trees has not been called");
    CK(cudaSetDevice(h->cfg.device));
    int rc = flush_pending(h);
    if (rc) return rc;
    uint32_t hdr[WK_HDR];
    CK(cudaMemcpyAsync(hdr, h->L.walker + (size_t)tree * h->WS, sizeof(hdr), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (n_nodes) *n_nodes = hdr[WK_NNODES];
    if (n_arcs) *n_arcs = hdr[WK_NARCS];
    if (n_preds) *n_preds = hdr[WK_NPREDS];
    return AZB_OK;
}

int azb_dump_tree(azb_handle *h, uint32_t tree, uint32_t *nodes, uint32_t *keys, uint32_t *preds, uint32_t *arcs) {
    if (!h || tree >= h->L.B) return AZB_ERR_INVALID;
    uint32_t nn = 0, na = 0, np = 0;
    int rc = azb_tree_sizes(h, tree, &nn, &na, &np);
    if (rc) return rc;
    const AzbLayout &L = h->L;
    uint32_t hdr[WK_HDR];
    CK(cudaMemcpyAsync(hdr, L.walker + (size_t)tree * L.WS, sizeof(hdr), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const uint32_t nblk = hdr[WK_NBLK];
    std::vector<uint32_t> nd((size_t)nn * 16);
    std::vector<uint2> blk(nblk);
    CK(cudaMemcpyAsync(nd.data(), (uint32_t *)L.node + (size_t)tree * L.cap_nodes * 16, nd.size() * 4,
                       cudaMemcpyDeviceToHost, h->stream));
    if (nblk)
        CK(cudaMemcpyAsync(blk.data(), L.blk + (size_t)tree * L.cap_blk, (size_t)nblk * 8, cudaMemcpyDeviceToHost,
                           h->stream));
    if (keys)
        CK(cudaMemcpyAsync(keys, L.key + (size_t)tree * L.cap_nodes * L.W, (size_t)nn * L.W * 4, cudaMemcpyDeviceToHost,
                           h->stream));
    CK(cudaStreamSynchronize(h->stream));
    // the reference's `predictions` Vec grows by one add_actions call at a time (graph_operations.rs:43-54): blocks
    // are bump-allocated in the same order, so ranking the blocks by address gives every node's prediction range
    std::vector<std::pair<uint32_t, uint32_t>> order;  // (lo2, node)
    for (uint32_t i = 0; i < nn; ++i) {
        const uint32_t *r = nd.data() + (size_t)i * 16;
        if ((r[3] >> 16) != 0u) order.emplace_back(r[4], i);
    }
    std::sort(order.begin(), order.end());
    std::vector<uint32_t> start(nn, 0u);
    uint32_t run = 0;
    for (auto &pr : order) {
        start[pr.second] = run;
        run += nd[(size_t)pr.second * 16 + 3] >> 16;
    }
    if (run != np) return fail(h, AZB_ERR_CAPACITY, "corrupt prediction count in tree %u (%u vs %u)", tree, run, np);
    for (uint32_t i = 0; i < nn; ++i) {
        const uint32_t *r = nd.data() + (size_t)i * 16;
        const uint32_t ex = r[3] & 0xffffu, cnt = r[3] >> 16, lo2 = r[4];
        if (nodes) {
            uint32_t *o = nodes + (size_t)i * 6;
            o[0] = r[0];
            o[1] = r[1];
            o[2] = r[2];
            o[3] = ex;
            o[4] = cnt ? start[i] : 0u;  // StateWeight::new leaves actions = 0..0 (state_weight.rs:13-21)
            o[5] = cnt ? start[i] + cnt : 0u;
        }
        if (!cnt) continue;
        const uint32_t lo = 2 * lo2;
        if (lo < cnt || lo + 2 + 2 * cnt > nblk) return fail(h, AZB_ERR_CAPACITY, "corrupt block in tree %u node %u", tree, i);
        const uint32_t n_out = blk[lo].y & 0xffffu;
        for (uint32_t j = 0; j < cnt; ++j) {
            const uint2 p = blk[lo - 1 - j];
            if (preds) {
                preds[(size_t)(start[i] + j) * 3 + 0] = p.y & 0x7ffu;
                preds[(size_t)(start[i] + j) * 3 + 1] = p.x;
                preds[(size_t)(start[i] + j) * 3 + 2] = ((p.y >> 11) & 1u) ? (p.y >> 12) : AZB_NONE;
            }
        }
        for (uint32_t t = 0; t < n_out; ++t) {
            const uint32_t w0 = blk[lo + 2 + 2 * t].x;
            const uint32_t child = w0 & 0xfffffu, a = w0 >> 20;
            uint32_t j = 0;
            while (j < cnt && (blk[lo - 1 - j].y & 0x7ffu) != a) ++j;
            if (j == cnt) return fail(h, AZB_ERR_CAPACITY, "arc without prediction in tree %u node %u", tree, i);
            const uint32_t arc = blk[lo - 1 - j].y >> 12;
            if (arc >= na) return fail(h, AZB_ERR_CAPACITY, "corrupt arc index in tree %u node %u", tree, i);
            if (arcs) {
                arcs[(size_t)arc * 3 + 0] = i;
                arcs[(size_t)arc * 3 + 1] = child;
                arcs[(size_t)arc * 3 + 2] = start[i] + j;
            }
        }
    }
    return AZB_OK;
}

int azb_get_counters(azb_handle *h, azb_counters *out) {
    if (!h || !out) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    static_assert(sizeof(azb_counters) == sizeof(AzbCounters), "counter layout");
    if (h->trees_init) {
        int rc = flush_pending(h);  // the last step's add_actions belongs to the counters it reports
        if (rc) return rc;
    }
    CK(cudaMemcpyAsync(out, &h->L.g->counters, sizeof(AzbCounters), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return AZB_OK;
}

// -DAZB_PROFILE builds only: cycles of lane 0 per phase (tools/phase_probe.py)
int azb_debug_phase_cycles(azb_handle *h, unsigned long long *out16) {
    if (!h || !out16) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaMemcpyAsync(out16, h->L.g->prof, sizeof(h->L.g->prof), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemsetAsync(h->L.g->prof, 0, sizeof(h->L.g->prof), h->stream));
#ifdef AZB_PROFILE
    {
        unsigned long long cp[8];
        CK(cudaMemcpyFromSymbol(cp, g_cost_prof, sizeof(cp)));
        for (int i = 0; i < 4; ++i) out16[12 + i] = cp[i] + (i == 3 ? cp[4] : 0ull);
        memset(cp, 0, sizeof(cp));
        CK(cudaMemcpyToSymbol(g_cost_prof, cp, sizeof(cp)));
    }
#endif
    return AZB_OK;
}

int azb_set_counter_mode(azb_handle *h, int full) {
    if (!h) return AZB_ERR_INVALID;
    h->count_full = full != 0;
    return AZB_OK;
}

#ifdef AZB_PROFILE
extern "C" int azb_debug_tree_prof(azb_handle *h, uint32_t *out4, uint32_t ntrees) {
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpyFromSymbol(out4, g_tree_prof, (size_t)ntrees * 16));
    return AZB_OK;
}
#endif

// cycle counters of the async kernel's MLP workers (last launch) + its row statistics: out[0..14] counters,
// out[15] = real rows << 32 | dummy rows
extern "C" int azb_debug_async(azb_handle *h, unsigned long long *out16) {  // out: 32 entries
    if (!h || !out16 || !h->async_ready) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(out16, h->asP.dbg, 32 * 8, cudaMemcpyDeviceToHost));
    AzbAsyncState st;
    CK(cudaMemcpy(&st, h->asP.st, sizeof(st), cudaMemcpyDeviceToHost));
    out16[15] = ((unsigned long long)st.rows_real << 32) | st.rows_dummy;
    return AZB_OK;
}

// State of one node = its tree's root with the node's action set replayed in ascending order (what
// par_update_argmmim_data does for the winning node: optimizer/mod.rs:224-239).  Runs on the poll stream from device
// data that never changes once written (root part of the walker block, the node's key), so a caller of azb_step_poll
// can turn an improvement record into ArgminData while later steps are still running.
extern "C" int azb_get_node_state(azb_handle *h, uint32_t tree, uint32_t node, uint8_t *parents, uint32_t *permitted) {
    if (!h || !parents || !permitted || tree >= h->L.B || node >= h->L.cap_nodes) return AZB_ERR_INVALID;
    if (!h->trees_init) return fail(h, AZB_ERR_STATE, "azb_init_trees has not been called");
    CK(cudaSetDevice(h->cfg.device));
    if (!h->poll_stream) CK(cudaStreamCreateWithFlags(&h->poll_stream, cudaStreamNonBlocking));
    const uint32_t W = h->W, PW = h->PW;
    std::vector<uint32_t> root(PW + W), key(W);
    const uint32_t *wk = h->L.walker + (size_t)tree * h->L.WS + WK_HDR + PW + 2 * W;  // root parents | root permitted
    CK(cudaMemcpyAsync(root.data(), wk, (size_t)(PW + W) * 4, cudaMemcpyDeviceToHost, h->poll_stream));
    CK(cudaMemcpyAsync(key.data(), h->L.key + ((size_t)tree * h->L.cap_nodes + node) * W, (size_t)W * 4, cudaMemcpyDeviceToHost,
                       h->poll_stream));
    CK(cudaStreamSynchronize(h->poll_stream));
    memcpy(parents, root.data(), h->N);
    memcpy(permitted, root.data() + PW, (size_t)W * 4);
    for (uint32_t a = 0; a < h->A; ++a) {
        if (!((key[a >> 5] >> (a & 31)) & 1u)) continue;
        const uint32_t child = azb_action_child(a), first = azb_child_first_action(child);  // act: rooted_tree/space.rs:56-73
        parents[child] = (uint8_t)(a - first);
        for (uint32_t q = first; q < first + child; ++q) permitted[q >> 5] &= ~(1u << (q & 31));
    }
    return AZB_OK;
}

// ---- the k best isomorphism classes (azb_best.cuh) ----
// the code kernel on m trees of n vertices (azb_trees_within codes every level below N with it)
static void launch_code_kernel(azb_handle *h, const uint8_t *dev_parents, uint32_t m, uint32_t n, unsigned long long *codes,
                               uint32_t stride, uint32_t *bad) {
    azb_tree_code_kernel<<<(m + AZB_CODE_WARPS - 1) / AZB_CODE_WARPS, AZB_CODE_WARPS * 32, 0, h->stream>>>(dev_parents, m, n, codes,
                                                                                                        stride, bad);
    h->launches += 1;
}

extern "C" int azb_tree_codes(azb_handle *h, const uint8_t *parents, uint32_t m, uint64_t *codes, float *ms) {
    if (!h || !parents || m == 0) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    uint8_t *d_par = nullptr;
    unsigned long long *d_codes = nullptr;
    uint32_t *d_bad = nullptr;
    int rc = scratch(h, [&](Carve &cv) {
        d_par = cv.take<uint8_t>((size_t)m * h->N);
        d_codes = cv.take<unsigned long long>((size_t)m * 2);
        d_bad = cv.take<uint32_t>(1);
    });
    if (rc) return rc;
    CK(cudaMemcpyAsync(d_par, parents, (size_t)m * h->N, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemsetAsync(d_bad, 0xff, 4, h->stream));
    CK(cudaEventRecord(h->ev0, h->stream));
    launch_code_kernel(h, d_par, m, h->N, d_codes, 2, d_bad);
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->ev1, h->stream));
    uint32_t bad = 0;
    if (codes) CK(cudaMemcpyAsync(codes, d_codes, (size_t)m * 16, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (ms) CK(cudaEventElapsedTime(ms, h->ev0, h->ev1));
    if (bad != AZB_NONE) {
        for (uint32_t v = 1; v < h->N; ++v)
            if (parents[(size_t)bad * h->N + v] >= v) return fail(h, AZB_ERR_INVALID, "tree %u: parents[%u] is not < %u", bad, v, v);
    }
    return AZB_OK;
}

// One selection round per pass of the loop: the M-th smallest ord(c) over all node records is T, every node with
// ord(c) <= T is a candidate, and the distinct codes among the candidates are classes whose value (<= T) and
// representative are exact; every class not found has a value above T.  While fewer than k classes came out and some
// node was left out, the next round asks for twice the candidates.
extern "C" int azb_best_trees(azb_handle *h, uint32_t k, uint32_t *n_out, float *eval, uint64_t *codes, uint32_t *tree,
                              uint32_t *node, uint8_t *parents, uint32_t *permitted, double *lambda1, uint32_t *mu) {
    if (!h) return AZB_ERR_INVALID;
    if (!h->trees_init) return fail(h, AZB_ERR_STATE, "azb_init_trees has not been called");
    if (k == 0 || k > AZB_BEST_MAX_K) return fail(h, AZB_ERR_INVALID, "k must be in 1..%u, got %u", AZB_BEST_MAX_K, k);
    CK(cudaSetDevice(h->cfg.device));
    // behind any enqueued steps, and their errors first (the trees may be incomplete after one)
    int rc = check_device_error(h);
    if (rc) return rc;
    if (!h->best_st) CK(dmalloc(h, &h->best_st, 1));
    const AzbLayout &L = h->L;
    const uint32_t N = h->N, W = h->W;
    const int grid = (int)std::min<uint32_t>(L.B, 1184u);
    uint32_t M = 4u * k;
    if (h->best_m_cap) M = std::min(M, h->best_m_cap);
    AzbBestState st;
    size_t tmp_bytes = 0;
    AzbCand *d_a = nullptr, *d_b = nullptr;
    uint8_t *d_par = nullptr, *d_tmp = nullptr;
    uint32_t *d_perm = nullptr;
    CostOut d_cost;
    for (;;) {
        CK(cudaMemsetAsync(h->best_st, 0, sizeof(AzbBestState), h->stream));
        CK(cudaMemsetAsync(&h->best_st->bad, 0xff, 4, h->stream));
        for (int shift = 24; shift >= 0; shift -= 8) {
            azb_best_hist_kernel<<<grid, 256, 0, h->stream>>>(L, h->best_st, (uint32_t)shift);
            azb_best_pick_kernel<<<1, 1, 0, h->stream>>>(h->best_st, (uint32_t)shift, M);
            h->launches += 2;
        }
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(&st, h->best_st, sizeof(st), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        const uint32_t C = st.count;
        if (C == 0) return fail(h, AZB_ERR_STATE, "the trees hold no node");
        size_t t1 = 0, t2 = 0;
        CK(cub::DeviceRadixSort::SortKeys(nullptr, t1, (const AzbCand *)nullptr, (AzbCand *)nullptr, C, AzbByCode{}, h->stream));
        CK(cub::DeviceRadixSort::SortKeys(nullptr, t2, (const AzbCand *)nullptr, (AzbCand *)nullptr, C, AzbByValue{}, h->stream));
        tmp_bytes = std::max(t1, t2);
        rc = scratch(h, [&](Carve &cv) {
            d_a = cv.take<AzbCand>(C);
            d_b = cv.take<AzbCand>(C);
            d_par = cv.take<uint8_t>((size_t)C * N);
            d_perm = cv.take<uint32_t>((size_t)C * W);
            d_tmp = cv.take<uint8_t>(tmp_bytes);
            d_cost.take(cv, std::min(k, C));  // the result's costs (at most k classes of at most C candidates)
        });
        if (rc) return rc;
        const uint32_t blocks = (C + 255) / 256;
        azb_best_compact_kernel<<<grid, 256, 0, h->stream>>>(L, h->best_st, d_a);
        azb_best_replay_kernel<<<blocks, 256, 0, h->stream>>>(L, d_a, C, d_par, nullptr);
        launch_code_kernel(h, d_par, C, N, reinterpret_cast<unsigned long long *>(d_a), sizeof(AzbCand) / 8, &h->best_st->bad);
        h->launches += 2;
        CK(cudaGetLastError());
        CK(cub::DeviceRadixSort::SortKeys(d_tmp, tmp_bytes, d_a, d_b, C, AzbByCode{}, h->stream));
        azb_best_heads_kernel<<<blocks, 256, 0, h->stream>>>(d_b, C, d_a, h->best_st);
        h->launches += 1;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(&st, h->best_st, sizeof(st), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        if (st.bad != 0xffffffffu) {
            // a rejected candidate keeps the all-zero code of the compaction (a code starts with 1), so it sorted first
            AzbCand c0;
            CK(cudaMemcpyAsync(&c0, d_b, sizeof(c0), cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            return fail(h, AZB_ERR_INVALID, "tree %u node %u: the replayed parent array has parents[v] >= v", (uint32_t)(c0.id >> 20),
                        (uint32_t)(c0.id & 0xfffffu));
        }
        if (st.n_class >= k || C >= st.total) break;
        M = 2u * C > C ? 2u * C : 0xffffffffu;
    }
    const uint32_t n_cls = st.n_class, n = std::min(k, n_cls);
    CK(cub::DeviceRadixSort::SortKeys(d_tmp, tmp_bytes, d_a, d_b, n_cls, AzbByValue{}, h->stream));
    azb_best_replay_kernel<<<(n + 255) / 256, 256, 0, h->stream>>>(L, d_b, n, d_par, d_perm);
    h->launches += 1;
    CK(cudaGetLastError());
    std::vector<AzbCand> cls(n);
    uint32_t cerr = 0;
    rc = cost_tail(h, d_par, n, N, d_cost, nullptr, nullptr, parents, lambda1, mu, nullptr, &cerr);
    if (rc) return rc;
    CK(cudaMemcpyAsync(cls.data(), d_b, (size_t)n * sizeof(AzbCand), cudaMemcpyDeviceToHost, h->stream));
    if (permitted) CK(cudaMemcpyAsync(permitted, d_perm, (size_t)n * W * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (cerr) return fail(h, (int)cerr, "%s", azb_strerror((int)cerr));
    for (uint32_t i = 0; i < n; ++i) {
        if (eval) eval[i] = azb_ord2f(cls[i].c);
        if (codes) {
            codes[2 * i] = cls[i].hi;
            codes[2 * i + 1] = cls[i].lo;
        }
        if (tree) tree[i] = (uint32_t)(cls[i].id >> 20);
        if (node) node[i] = (uint32_t)(cls[i].id & 0xfffffu);
    }
    if (n_out) *n_out = n;
    return AZB_OK;
}

// ---- every free tree on N <= 32 vertices by index, and the exact k best of an index range (azb_enum.cuh) ----
extern "C" int azb_free_tree_count(uint32_t n, uint64_t *count) {
    if (!count || n < 5 || n > AZB_ENUM_MAX_N) return AZB_ERR_INVALID;
    uint64_t U = 0;
    azb_enum_counts(n, &U, count);
    return AZB_OK;
}

static uint64_t enum_total(const azb_handle *h) {
    const AzbEnum &E = h->en;
    const uint64_t t = E.n % 2 == 0 ? E.off[E.smax + 1] - E.off[E.smax] : 0;  // rooted trees of size N / 2
    return E.U + t * (t + 1) / 2;
}

// the tables of the handle's N, built on the host and uploaded on first use (counted in azb_device_bytes)
static int enum_tables(azb_handle *h, const char *fn) {
    if (h->N > AZB_ENUM_MAX_N)
        return fail(h, AZB_ERR_INVALID, "%s: the enumeration covers N <= %u, the handle has N = %u", fn, AZB_ENUM_MAX_N, h->N);
    if (h->en.P) return AZB_OK;
    std::vector<unsigned long long> P;
    std::vector<uint8_t> rp;
    AzbEnum E;
    azb_enum_build(h->N, E, P, rp);
    if (!h->en_P) CK(dmalloc(h, &h->en_P, P.size()));
    if (!h->en_rp) CK(dmalloc(h, &h->en_rp, rp.size()));
    CK(cudaMemcpyAsync(h->en_P, P.data(), P.size() * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->en_rp, rp.data(), rp.size(), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    E.P = h->en_P;
    E.rp = h->en_rp;
    h->en = E;
    return AZB_OK;
}

static int enum_range(azb_handle *h, const char *fn, uint64_t start, uint64_t count) {
    const uint64_t total = enum_total(h);
    if (count == 0 || start > total || count > total - start)
        return fail(h, AZB_ERR_INVALID, "%s: %llu trees from index %llu are not all in [0, %llu)", fn, (unsigned long long)count,
                    (unsigned long long)start, (unsigned long long)total);
    return AZB_OK;
}

static int enum_sms(azb_handle *h, int *sms) {
    CK(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, h->cfg.device));
    return AZB_OK;
}

extern "C" int azb_free_trees(azb_handle *h, uint64_t start, uint32_t m, uint8_t *parents) {
    if (!h) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    int rc = enum_tables(h, "azb_free_trees");
    if (rc) return rc;
    if (!parents) return fail(h, AZB_ERR_INVALID, "azb_free_trees: parents is NULL");
    rc = enum_range(h, "azb_free_trees", start, m);
    if (rc) return rc;
    int sms = 0;
    rc = enum_sms(h, &sms);
    if (rc) return rc;
    const uint32_t N = h->N, chunk = h->en_chunk ? h->en_chunk : AZB_ENUM_CHUNK;
    uint8_t *d_par = nullptr;
    rc = scratch(h, [&](Carve &cv) { d_par = cv.take<uint8_t>((size_t)std::min(m, chunk) * N); });
    if (rc) return rc;
    for (uint32_t done = 0; done < m;) {
        const uint32_t c = std::min(chunk, m - done);
        azb_enum_trees_kernel<<<std::min<uint32_t>((c + 7) / 8, (uint32_t)sms * 16u), 256, 0, h->stream>>>(h->en, start + done, nullptr, c,
                                                                                                          d_par);
        h->launches += 1;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(parents + (size_t)done * N, d_par, (size_t)c * N, cudaMemcpyDeviceToHost, h->stream));
        done += c;
    }
    CK(cudaStreamSynchronize(h->stream));
    return AZB_OK;
}

struct AzbEnumScalars {
    unsigned long long thr;    // the k-th best key bits so far (all ones until k trees are in)
    unsigned long long below;  // trees with key < bound
    uint32_t n_cand, err;
};

// Chunks in ascending index order.  The running top k sits at the front of buffer A; a chunk's candidates (key bits <= the
// k-th best so far) land behind it, the whole is radix-sorted by (key bits, index) into B and the first k go back to A.  A
// later tree whose key equals the threshold has a larger index than all k kept ones and would lose the tie, so the
// result is the exact top k of the range.
extern "C" int azb_exhaustive_best(azb_handle *h, uint64_t start, uint64_t count, uint32_t k, double bound, uint32_t *n_out,
                                   uint64_t *n_below, uint64_t *index, uint8_t *parents, double *lambda1, uint32_t *mu, float *eval,
                                   float *ms) {
    if (!h) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    int rc = enum_tables(h, "azb_exhaustive_best");
    if (rc) return rc;
    if (k == 0 || k > AZB_BEST_MAX_K) return fail(h, AZB_ERR_INVALID, "k must be in 1..%u, got %u", AZB_BEST_MAX_K, k);
    rc = enum_range(h, "azb_exhaustive_best", start, count);
    if (rc) return rc;
    int sms = 0;
    rc = enum_sms(h, &sms);
    if (rc) return rc;
    const uint32_t N = h->N, chunk = h->en_chunk ? h->en_chunk : AZB_ENUM_CHUNK, cap = k + chunk;
    const uint32_t n_res = (uint32_t)std::min<uint64_t>(k, count);
    int bps = 0;
    if (N <= 22) CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, azb_enum_best_kernel<3>, 256, 0));
    else CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, azb_enum_best_kernel<4>, 256, 0));
    const uint32_t grid = (uint32_t)std::max(1, sms * bps);
    size_t tmp_bytes = 0;
    CK(cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, (const AzbEnumCand *)nullptr, (AzbEnumCand *)nullptr, cap, AzbEnumByKey{},
                                      h->stream));
    AzbEnumCand *d_a = nullptr, *d_b = nullptr;
    uint8_t *d_par = nullptr, *d_tmp = nullptr;
    AzbEnumScalars *d_sc = nullptr;
    CostOut d_cost;
    rc = scratch(h, [&](Carve &cv) {
        d_a = cv.take<AzbEnumCand>(cap);
        d_b = cv.take<AzbEnumCand>(cap);
        d_par = cv.take<uint8_t>((size_t)k * N);
        d_sc = cv.take<AzbEnumScalars>(1);
        d_tmp = cv.take<uint8_t>(tmp_bytes);
        d_cost.take(cv, n_res);
    });
    if (rc) return rc;
    CK(cudaEventRecord(h->ev0, h->stream));
    CK(cudaMemsetAsync(d_sc, 0, sizeof(AzbEnumScalars), h->stream));
    CK(cudaMemsetAsync(&d_sc->thr, 0xff, 8, h->stream));
    uint32_t nb = 0;  // entries of the running top k at the front of A
    for (uint64_t done = 0; done < count;) {
        const uint32_t c = (uint32_t)std::min<uint64_t>(chunk, count - done);
        const uint32_t blocks = std::min(grid, (c + 7) / 8);
        CK(cudaMemsetAsync(&d_sc->n_cand, 0, 4, h->stream));
        if (N <= 22)
            azb_enum_best_kernel<3><<<blocks, 256, 0, h->stream>>>(h->en, start + done, c, &d_sc->thr, bound, d_a + nb, &d_sc->n_cand,
                                                                   &d_sc->below, &d_sc->err);
        else
            azb_enum_best_kernel<4><<<blocks, 256, 0, h->stream>>>(h->en, start + done, c, &d_sc->thr, bound, d_a + nb, &d_sc->n_cand,
                                                                   &d_sc->below, &d_sc->err);
        h->launches += 1;
        CK(cudaGetLastError());
        uint32_t nc = 0;
        CK(cudaMemcpyAsync(&nc, &d_sc->n_cand, 4, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        done += c;
        if (nc == 0) continue;
        const uint32_t tot = nb + nc;
        CK(cub::DeviceRadixSort::SortKeys(d_tmp, tmp_bytes, d_a, d_b, tot, AzbEnumByKey{}, h->stream));
        nb = std::min(k, tot);
        CK(cudaMemcpyAsync(d_a, d_b, (size_t)nb * sizeof(AzbEnumCand), cudaMemcpyDeviceToDevice, h->stream));
        if (nb == k) CK(cudaMemcpyAsync(&d_sc->thr, &d_b[k - 1].key, 8, cudaMemcpyDeviceToDevice, h->stream));
    }
    // the result's parent arrays, and lambda_1, mu and eval from the stand-alone cost kernel (what azb_eval_costs gives)
    azb_enum_trees_kernel<<<std::min<uint32_t>((nb + 7) / 8, (uint32_t)sms * 16u), 256, 0, h->stream>>>(h->en, 0ull, d_a, nb, d_par);
    h->launches += 1;
    CK(cudaGetLastError());
    std::vector<AzbEnumCand> res(nb);
    AzbEnumScalars sc;
    uint32_t cerr = 0;
    rc = cost_tail(h, d_par, nb, N, d_cost, nullptr, h->ev1, parents, lambda1, mu, eval, &cerr);
    if (rc) return rc;
    CK(cudaMemcpyAsync(res.data(), d_a, (size_t)nb * sizeof(AzbEnumCand), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(&sc, d_sc, sizeof(sc), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (ms) CK(cudaEventElapsedTime(ms, h->ev0, h->ev1));
    if (sc.err || cerr) return fail(h, AZB_ERR_LAMBDA, "%s", azb_strerror(AZB_ERR_LAMBDA));
    if (index)
        for (uint32_t i = 0; i < nb; ++i) index[i] = res[i].idx;
    if (n_below) *n_below = sc.below;
    if (n_out) *n_out = nb;
    return AZB_OK;
}

// ---- every tree on N <= 64 vertices with key <= a bound, grown leaf by leaf (azb_grow.cuh) ----
// Level n (the classes on n vertices) is built from level n - 1 in chunks of parents; azb_grow.cuh lists the passes of
// one chunk.  The host keeps each finished level as its list of codes and lays the slab out anew for the next one: the
// level's parents decoded (LP), the chunk's buffers, and the list of kept classes (A) with the other half of its sorts (B).
//
// Sharded (azb_comm_trees_within; include/azb.h has the algorithm): a rank holds the classes of each level it owns, and
// the level runs in rounds that every rank takes part in, one chunk of its own parents each (possibly none).  A round
// routes the chunk's distinct classes to their owners, all-gathers one record per rank (WR_* below) and exchanges
// the runs; the received codes are then sorted, made unique and costed in pieces of at most one chunk.  One more record
// closes each level.  Every stop is decided from the records, so all ranks return it from the same collective.
static int comm_allgather(azb_handle *h, const unsigned long long *send, unsigned long long *recv, size_t count);
static int comm_exchange(azb_handle *h, const ulonglong2 *send, const unsigned long long *rec, ulonglong2 *recv);

// a rank's record of one round, all-gathered: send counts to every rank, then these
enum { WR_SHARE = 0, WR_CAP, WR_ERR, WR_WORDS };  // kept list at its last merge, the rank's cap on it, cost error word

// the first collective of azb_comm_trees_within: every rank's arguments and chunk; refuses on every rank what one
// rank's arguments make invalid.  chunks = every rank's children per chunk.
static int within_agree_args(azb_handle *h, double bound, uint32_t k, uint64_t max_level, uint32_t chunk,
                             std::vector<uint32_t> &chunks) {
    const uint32_t world = (uint32_t)h->comm_world;
    enum { A_N, A_BOUND, A_K, A_MAX, A_CHUNK, A_WORDS };
    unsigned long long *d_args = nullptr;
    int rc = scratch(h, [&](Carve &cv) { d_args = cv.take<unsigned long long>((size_t)A_WORDS * (world + 1)); });
    if (rc) return rc;
    unsigned long long mine[A_WORDS] = {h->N, 0, k, max_level, chunk};
    memcpy(&mine[A_BOUND], &bound, 8);
    std::vector<unsigned long long> a((size_t)A_WORDS * world);
    CK(cudaMemcpyAsync(d_args + (size_t)A_WORDS * world, mine, sizeof(mine), cudaMemcpyHostToDevice, h->stream));
    rc = comm_allgather(h, d_args + (size_t)A_WORDS * world, d_args, A_WORDS);
    if (rc) return rc;
    CK(cudaMemcpyAsync(a.data(), d_args, a.size() * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const char *name[A_WORDS] = {"N", "bound", "k", "max_level", "chunk"};
    for (uint32_t r = 0; r < world; ++r) {
        const unsigned long long *ar = a.data() + (size_t)A_WORDS * r;
        double b;
        memcpy(&b, &ar[A_BOUND], 8);
        if (ar[A_K] == 0 || ar[A_K] > AZB_BEST_MAX_K)
            return fail(h, AZB_ERR_INVALID, "azb_comm_trees_within: rank %u passes k = %llu; k must be in 1..%u", r, ar[A_K],
                        AZB_BEST_MAX_K);
        if (std::isnan(b)) return fail(h, AZB_ERR_INVALID, "azb_comm_trees_within: rank %u passes a NaN bound", r);
        for (int f = A_N; f < A_CHUNK; ++f)
            if (ar[f] != a[f])
                return fail(h, AZB_ERR_INVALID, "azb_comm_trees_within: rank %u's %s (%s 0x%llx) differs from rank 0's (0x%llx)", r,
                            name[f], f == A_BOUND ? "bits" : "value", ar[f], a[f]);
        chunks[r] = (uint32_t)ar[A_CHUNK];
    }
    return AZB_OK;
}

// The stop every rank returns after an all-gather of records (world x (world + WR_WORDS) words): a level over max_level
// (the sum of the shares), a rank's share over its cap, a cost error on any rank.
static int within_agreed_stop(azb_handle *h, const std::vector<unsigned long long> &rec, uint32_t world, uint32_t n,
                              uint64_t max_level) {
    const size_t R = world + WR_WORDS;
    unsigned long long total = 0;
    for (uint32_t r = 0; r < world; ++r) total += rec[R * r + world + WR_SHARE];
    if (max_level && total > max_level)
        return fail(h, AZB_ERR_CAPACITY,
                    "azb_comm_trees_within: level %u (trees on %u vertices) holds more than %llu classes (at least %llu found on "
                    "%u ranks; max_level %llu)",
                    n, n, (unsigned long long)max_level, total, world, (unsigned long long)max_level);
    for (uint32_t r = 0; r < world; ++r)
        if (rec[R * r + world + WR_SHARE] > rec[R * r + world + WR_CAP])
            return fail(h, AZB_ERR_CAPACITY,
                        "azb_comm_trees_within: level %u (trees on %u vertices): rank %u's share holds more than %llu classes, "
                        "the room on its device (at least %llu found; max_level %llu)",
                        n, n, r, rec[R * r + world + WR_CAP], rec[R * r + world + WR_SHARE], (unsigned long long)max_level);
    for (uint32_t r = 0; r < world; ++r)
        if (rec[R * r + world + WR_ERR]) return fail(h, AZB_ERR_LAMBDA, "%s", azb_strerror(AZB_ERR_LAMBDA));
    return AZB_OK;
}

// azb_trees_within (sharded = false: this handle alone, no collective) and azb_comm_trees_within (sharded = true);
// proof != null (azb_trees_within_proof, alone only): the same outputs and the five proof words
static int trees_within(azb_handle *h, bool sharded, double bound, uint32_t k, uint64_t max_level, uint32_t *n_out,
                        uint64_t *n_within, uint64_t *n_below, uint64_t *codes, uint8_t *parents, double *lambda1, uint32_t *mu,
                        float *eval, uint64_t *proof, float *ms) {
    CK(cudaSetDevice(h->cfg.device));
    const uint32_t N = h->N, chunk = h->grow_chunk ? h->grow_chunk : AZB_GROW_CHUNK;
    const uint32_t world = sharded ? (uint32_t)h->comm_world : 1u, me = sharded ? (uint32_t)h->comm_rank : 0u;
    const bool trace = getenv("AZB_TRACE_WITHIN") != nullptr;  // one line per level (and rank) on stderr (tools/within_probe.py)
    const size_t E = sizeof(AzbGrowEnt), R = world + WR_WORDS, tw = 2 + 3 * (size_t)k;  // tw: words of a rank's first k
    int rc = AZB_OK;
    std::vector<uint32_t> chunks(world, chunk);  // every rank's children per chunk (tests give the ranks different ones)
    if (sharded) {
        rc = within_agree_args(h, bound, k, max_level, chunk, chunks);
        if (rc) return rc;
    }
    const AzbCertBound cb = cert_bound(bound, N);  // before the default bound becomes the star's computed key
    uint64_t pw[5] = {0, 0, 0, 0, 0};             // the proof words so far
    CK(cudaEventRecord(h->ev0, h->stream));
    if (bound < 0.0) {  // the star's key on its canonical labelling: every vertex under vertex 0
        uint8_t *d_star = nullptr;
        CostOut d_cost;
        rc = scratch(h, [&](Carve &cv) {
            d_star = cv.take<uint8_t>(N);
            d_cost.take(cv, 1);
        });
        if (rc) return rc;
        CK(cudaMemsetAsync(d_star, 0, N, h->stream));
        double l1 = 0.0;
        uint32_t m1 = 0, err = 0;
        rc = cost_tail(h, d_star, 1, N, d_cost, nullptr, nullptr, nullptr, &l1, &m1, nullptr, &err);
        if (rc) return rc;
        CK(cudaStreamSynchronize(h->stream));
        if (err) return fail(h, AZB_ERR_LAMBDA, "%s", azb_strerror(AZB_ERR_LAMBDA));
        bound = (double)m1 + l1;
    }
    // the classes one level may hold: max_level, what the device has room for (per class: the list and the other half
    // of its sort, CUB's scratch, the codes and parents of the next level; the chunk's buffers set aside, and when
    // sharded the codes one round can bring with the other half of their sort and its CUB scratch), and what one CUB
    // pass takes
    const uint64_t kc_max = (uint64_t)std::max(chunk, 64u) + 64u;
    uint64_t recv_max = 0;
    if (sharded)
        for (uint32_t c : chunks) recv_max += (uint64_t)std::max(c, 64u) + 64u;
    size_t free_b = 0, total_b = 0;
    CK(cudaMemGetInfo(&free_b, &total_b));
    const uint64_t avail = (uint64_t)free_b + h->scratch_cap;
    const uint64_t set_aside = kc_max * (64 + 4 * E + 16) + recv_max * 3 * E + (256ull << 20);
    const uint64_t fit = avail > set_aside ? (avail - set_aside) / (5 * E + 64) : 0;
    const uint64_t cap_level = std::min<uint64_t>({max_level ? max_level : fit, fit, (1ull << 31) - 1 - kc_max});
    // L_4: the path (code 11100100) and the star (11010100); every tree on 5 or more vertices grows from one of them.
    // share[r] = the classes of the current level rank r holds.
    std::vector<AzbGrowEnt> lvl;
    std::vector<uint64_t> share(world, 0);
    for (const AzbGrowEnt &e : {AzbGrowEnt{0xE4ull << 56, 0ull, 0ull}, AzbGrowEnt{0xD4ull << 56, 0ull, 0ull}}) {
        const uint32_t o = azb_grow_owner(e.hi, e.lo, world);
        share[o] += 1;
        if (o == me) lvl.push_back(e);
    }
    std::vector<unsigned long long> rec(R * world);
    AzbGrowEnt *d_a = nullptr, *d_b = nullptr;
    AzbGrowScalars *d_sc = nullptr;
    uint8_t *d_res = nullptr;
    unsigned long long *d_top = nullptr;
    CostOut d_res_cost;
    size_t tmp_bytes = 0;
    uint8_t *d_tmp = nullptr;
    uint64_t nacc = 0, total = 2;
    for (uint32_t s = 4; s < N; ++s) {
        const auto t0 = std::chrono::steady_clock::now();
        const uint32_t n = s + 1, lo_bit = 128 - 2 * n;  // a code of n vertices occupies the top 2n of the 128 bits
        const bool last = n == N;
        const uint64_t ns = lvl.size();
        const uint32_t pc = std::max(1u, chunk / s), kc = pc * s;  // parents and children of a full chunk
        const uint64_t acap = std::min<uint64_t>(total * s, cap_level) + kc;
        uint32_t rounds = 0;  // the most chunks any rank has at this level
        uint64_t rmax = 0;    // sharded: the most codes one round can bring, a full chunk from every rank
        for (uint32_t r = 0; r < world; ++r) {
            const uint32_t pr = std::max(1u, chunks[r] / s);
            rounds = std::max<uint32_t>(rounds, (uint32_t)((share[r] + pr - 1) / pr));
            rmax += (uint64_t)pr * s;
        }
        if (!sharded) rmax = 0;
        size_t t[6] = {0, 0, 0, 0, 0, 0};
        CK(cub::DeviceRadixSort::SortKeys(nullptr, t[0], (const AzbGrowEnt *)nullptr, (AzbGrowEnt *)nullptr, kc, AzbGrowByCode{},
                                          lo_bit, 128, h->stream));
        CK(cub::DeviceRadixSort::SortKeys(nullptr, t[1], (const AzbGrowEnt *)nullptr, (AzbGrowEnt *)nullptr, (uint32_t)acap, AzbGrowByCode{},
                                          lo_bit, 128, h->stream));
        CK(cub::DeviceSelect::Unique(nullptr, t[2], (const AzbGrowEnt *)nullptr, (AzbGrowEnt *)nullptr, (uint32_t *)nullptr, (uint32_t)acap,
                                     h->stream));
        if (last)
            CK(cub::DeviceRadixSort::SortKeys(nullptr, t[3], (const AzbGrowEnt *)nullptr, (AzbGrowEnt *)nullptr, (uint32_t)acap, AzbGrowByKey{},
                                              h->stream));
        if (sharded) {
            CK(cub::DeviceRadixSort::SortKeys(nullptr, t[4], (const AzbGrowEnt *)nullptr, (AzbGrowEnt *)nullptr, (uint32_t)rmax,
                                              AzbGrowByCode{}, lo_bit, 128, h->stream));
            CK(cub::DeviceSelect::Unique(nullptr, t[5], (const AzbGrowEnt *)nullptr, (AzbGrowEnt *)nullptr, (uint32_t *)nullptr,
                                         (uint32_t)rmax, h->stream));
        }
        tmp_bytes = *std::max_element(t, t + 6);
        AzbGrowEnt *d_lv = nullptr, *d_e1 = nullptr, *d_e2 = nullptr, *d_r1 = nullptr, *d_r2 = nullptr;
        uint8_t *d_lp = nullptr, *d_k = nullptr;
        double *d_l1 = nullptr;
        uint32_t *d_mu = nullptr;
        float *d_c = nullptr;
        ulonglong2 *d_send = nullptr;
        unsigned long long *d_rec = nullptr, *d_cursor = nullptr, *d_proof = nullptr;
        rc = scratch(h, [&](Carve &cv) {
            d_lv = cv.take<AzbGrowEnt>(ns);
            d_lp = cv.take<uint8_t>(ns * s);
            d_k = cv.take<uint8_t>((size_t)kc * n);
            d_e1 = cv.take<AzbGrowEnt>(kc);
            d_e2 = cv.take<AzbGrowEnt>(kc);
            d_l1 = cv.take<double>(kc);
            d_mu = cv.take<uint32_t>(kc);
            d_c = cv.take<float>(kc);
            d_a = cv.take<AzbGrowEnt>(acap);
            d_b = cv.take<AzbGrowEnt>(sharded && last ? std::max<uint64_t>(acap, k) : acap);  // sharded: the merged first k
            d_sc = cv.take<AzbGrowScalars>(1);
            d_res = cv.take<uint8_t>((size_t)k * N);
            d_res_cost.take(cv, k);
            d_tmp = cv.take<uint8_t>(tmp_bytes);
            // sharded only (all empty otherwise); the received runs land in d_r2's bytes, copied out before its sort
            d_send = cv.take<ulonglong2>(sharded ? kc : 0);
            d_r1 = cv.take<AzbGrowEnt>(rmax);
            d_r2 = cv.take<AzbGrowEnt>(rmax);
            d_rec = cv.take<unsigned long long>(sharded ? R * (world + 1) : 0);
            d_cursor = cv.take<unsigned long long>(sharded ? world : 0);
            d_top = cv.take<unsigned long long>(sharded && last ? tw * (world + 1) : 0);  // count, below, first k entries
            d_proof = cv.take<unsigned long long>(proof ? 5 : 0);  // this level's proof words
        });
        if (rc) return rc;
        CK(cudaMemcpyAsync(d_lv, lvl.data(), ns * E, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemsetAsync(d_sc, 0, sizeof(AzbGrowScalars), h->stream));
        if (proof) {
            CK(cudaMemsetAsync(d_proof, 0, 5 * 8, h->stream));
            rc = cert_smem(h, azb_certify_pruned_kernel, n);
            if (rc) return rc;
        }
        if (ns) {
            azb_grow_decode_kernel<<<(uint32_t)((ns + 255) / 256), 256, 0, h->stream>>>(d_lv, (uint32_t)ns, s, d_lp);
            h->launches += 1;
            CK(cudaGetLastError());
        }
        const double thr = last ? bound : bound + AZB_GROW_EPS;
        uint64_t children = 0, evaluated = 0, sent = 0, received = 0, merged = 0;  // merged: the list's size at its last merge
        bool dirty = false;  // classes kept since that merge
        nacc = 0;
        // one entry per class, sorted by code; alone, a list over the cap ends the call here, sharded at the next record
        auto merge = [&]() -> int {
            uint32_t nu = 0;
            CK(cub::DeviceRadixSort::SortKeys(d_tmp, tmp_bytes, d_a, d_b, (uint32_t)nacc, AzbGrowByCode{}, lo_bit, 128, h->stream));
            CK(cub::DeviceSelect::Unique(d_tmp, tmp_bytes, d_b, d_a, &d_sc->n_sel, (uint32_t)nacc, h->stream));
            CK(cudaMemcpyAsync(&nu, &d_sc->n_sel, 4, cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            nacc = merged = nu;
            dirty = false;
            if (nacc > cap_level && !sharded)
                return fail(h, AZB_ERR_CAPACITY,
                            "azb_trees_within: level %u (trees on %u vertices) holds more than %llu classes (at least %llu found; "
                            "max_level %llu, room on the device for %llu)",
                            n, n, (unsigned long long)cap_level, (unsigned long long)nacc, (unsigned long long)max_level,
                            (unsigned long long)fit);
            return AZB_OK;
        };
        // sharded: route the u classes at d_e1 to their owners, all-gather the records, stop if they say so, exchange the
        // runs; *got = the distinct classes received, at d_r1
        auto exchange = [&](uint32_t u, uint32_t *got) -> int {
            unsigned long long *mine = d_rec + R * world;
            CK(cudaMemsetAsync(mine, 0, R * 8, h->stream));
            if (u) {
                const uint32_t blocks = std::min((u + 255) / 256, 1184u);
                CK(cudaMemsetAsync(d_cursor, 0, (size_t)world * 8, h->stream));
                azb_grow_count_kernel<<<blocks, 256, 4 * world, h->stream>>>(d_e1, u, world, mine);
                azb_grow_route_kernel<<<blocks, 256, 20 * world, h->stream>>>(d_e1, u, world, mine, d_cursor, d_send);
                h->launches += 2;
                CK(cudaGetLastError());
            }
            const unsigned long long tail[2] = {merged, cap_level};
            CK(cudaMemcpyAsync(mine + world + WR_SHARE, tail, sizeof(tail), cudaMemcpyHostToDevice, h->stream));
            CK(cudaMemcpyAsync(mine + world + WR_ERR, &d_sc->err, 4, cudaMemcpyDeviceToDevice, h->stream));
            int rc2 = comm_allgather(h, mine, d_rec, R);
            if (rc2) return rc2;
            CK(cudaMemcpyAsync(rec.data(), d_rec, R * world * 8, cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            rc2 = within_agreed_stop(h, rec, world, n, max_level);
            if (rc2) return rc2;
            ulonglong2 *recv = reinterpret_cast<ulonglong2 *>(d_r2);
            rc2 = comm_exchange(h, d_send, rec.data(), recv);
            if (rc2) return rc2;
            uint64_t nr = 0;
            for (uint32_t r = 0; r < world; ++r) {
                nr += rec[R * r + me];
                if (r != me) sent += rec[R * me + r], received += rec[R * r + me];
            }
            *got = 0;
            if (nr == 0) return AZB_OK;
            CK(cudaMemcpy2DAsync(d_r1, E, recv, 16, 16, nr, cudaMemcpyDeviceToDevice, h->stream));
            CK(cub::DeviceRadixSort::SortKeys(d_tmp, tmp_bytes, d_r1, d_r2, (uint32_t)nr, AzbGrowByCode{}, lo_bit, 128, h->stream));
            CK(cub::DeviceSelect::Unique(d_tmp, tmp_bytes, d_r2, d_r1, &d_sc->n_sel, (uint32_t)nr, h->stream));
            CK(cudaMemcpyAsync(got, &d_sc->n_sel, 4, cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            return AZB_OK;
        };
        uint64_t done = 0;
        for (uint32_t round = 0; round < rounds; ++round) {
            const uint32_t p = (uint32_t)std::min<uint64_t>(pc, ns - done), m = p * s;
            uint32_t u = 0;
            if (p) {
                azb_grow_expand_kernel<<<(uint32_t)std::min<size_t>(((size_t)m * n + 255) / 256, 8192), 256, 0, h->stream>>>(d_lp + done * s,
                                                                                                                         p, s, d_k);
                launch_code_kernel(h, d_k, m, n, reinterpret_cast<unsigned long long *>(d_e1), (uint32_t)(E / 8), &d_sc->bad);
                h->launches += 1;
                CK(cudaGetLastError());
                CK(cub::DeviceRadixSort::SortKeys(d_tmp, tmp_bytes, d_e1, d_e2, m, AzbGrowByCode{}, lo_bit, 128, h->stream));
                CK(cub::DeviceSelect::Unique(d_tmp, tmp_bytes, d_e2, d_e1, &d_sc->n_sel, m, h->stream));
                CK(cudaMemcpyAsync(&u, &d_sc->n_sel, 4, cudaMemcpyDeviceToHost, h->stream));
                CK(cudaStreamSynchronize(h->stream));
            }
            const AzbGrowEnt *fresh = d_e1;  // the distinct classes this rank evaluates in this round
            if (sharded) {
                rc = exchange(u, &u);
                if (rc) return rc;
                fresh = d_r1;
            }
            // decode, cost and keep, in pieces of at most one chunk (alone: the chunk, in one piece)
            for (uint32_t off = 0; off < u && merged <= cap_level; off += kc) {
                const uint32_t q = std::min(kc, u - off);
                uint32_t kept = 0;
                azb_grow_decode_kernel<<<(q + 255) / 256, 256, 0, h->stream>>>(fresh + off, q, n, d_k);
                launch_cost_n(h, d_k, q, n, d_l1, d_mu, d_c, &d_sc->err);
                CK(cudaMemsetAsync(&d_sc->n_keep, 0, 4, h->stream));
                azb_grow_keep_kernel<<<(q + 255) / 256, 256, 0, h->stream>>>(fresh + off, d_l1, d_mu, q, thr, d_a + nacc, &d_sc->n_keep);
                h->launches += 2;
                CK(cudaGetLastError());
                if (proof) {  // the classes keep dropped: key > bound proven, or proof[4]
                    azb_certify_pruned_kernel<<<(q + AZB_CERT_THREADS - 1) / AZB_CERT_THREADS, AZB_CERT_THREADS, azb_certify_smem(n),
                                                h->stream>>>(d_k, q, n, d_l1, d_mu, thr, cb, &d_proof[4]);
                    h->launches += 1;
                    CK(cudaGetLastError());
                }
                CK(cudaMemcpyAsync(&kept, &d_sc->n_keep, 4, cudaMemcpyDeviceToHost, h->stream));
                CK(cudaStreamSynchronize(h->stream));
                nacc += kept;
                evaluated += q;
                dirty = dirty || kept;
                if (dirty && nacc + kc > acap) {
                    rc = merge();
                    if (rc) return rc;
                }
            }
            children += m;
            done += p;
        }
        if (dirty) {
            rc = merge();
            if (rc) return rc;
        }
        // proof, last level: the verdict of every result class, once each (a class can be kept in several chunks, so
        // the chunks cannot count them), on its canonical labelling as the level costed it
        for (uint32_t off = 0; proof && last && off < nacc; off += kc) {
            const uint32_t q = (uint32_t)std::min<uint64_t>(kc, nacc - off);
            azb_grow_decode_kernel<<<(q + 255) / 256, 256, 0, h->stream>>>(d_a + off, q, n, d_k);
            launch_cost_n(h, d_k, q, n, d_l1, d_mu, d_c, &d_sc->err);
            h->launches += 1;
            CK(cudaGetLastError());
            rc = launch_certify(h, d_k, q, n, d_l1, cb, nullptr, nullptr, nullptr, nullptr, d_proof);
            if (rc) return rc;
        }
        if (sharded) {  // the level's closing record: every rank's share of it
            uint32_t none = 0;
            rc = exchange(0, &none);
            if (rc) return rc;
            for (uint32_t r = 0; r < world; ++r) share[r] = rec[R * r + world + WR_SHARE];
        } else {
            share[0] = nacc;
        }
        total = 0;
        for (uint64_t c : share) total += c;
        uint32_t err = 0;
        unsigned long long lp[5] = {0, 0, 0, 0, 0};
        CK(cudaMemcpyAsync(&err, &d_sc->err, 4, cudaMemcpyDeviceToHost, h->stream));
        if (proof) CK(cudaMemcpyAsync(lp, d_proof, sizeof(lp), cudaMemcpyDeviceToHost, h->stream));
        lvl.resize(last ? 0 : nacc);
        if (!last && nacc) CK(cudaMemcpyAsync(lvl.data(), d_a, nacc * E, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        if (err) return fail(h, AZB_ERR_LAMBDA, "%s", azb_strerror(AZB_ERR_LAMBDA));
        for (int w = 0; w < 5; ++w) pw[w] += lp[w];
        const double level_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (trace && !sharded)
            fprintf(stderr, "azb_trees_within: N %u level %u: %llu classes, %llu children, %llu evaluated, %.3f ms\n", N, n,
                    (unsigned long long)nacc, (unsigned long long)children, (unsigned long long)evaluated, level_ms);
        if (trace && sharded)
            fprintf(stderr,
                    "azb_comm_trees_within: N %u level %u rank %u: %llu classes owned, %llu global, %llu children, %llu codes sent, "
                    "%llu received, %llu evaluated, %.3f ms\n",
                    N, n, me, (unsigned long long)nacc, (unsigned long long)total, (unsigned long long)children,
                    (unsigned long long)sent, (unsigned long long)received, (unsigned long long)evaluated, level_ms);
        if (total == 0) break;  // no tree on more vertices is within the bound either
    }
    // the last level, by (key bits, code): count the keys below the bound, and the first k through the cost kernel of
    // azb_eval_costs on their canonical parent arrays.  Sharded, each rank sorts its share and the first k of every share
    // are merged on every rank's host, so all ranks cost the same entries.
    const uint32_t nres = (uint32_t)std::min<uint64_t>(k, total);
    std::vector<AzbGrowEnt> res(nres);
    unsigned long long below = 0;
    uint32_t cerr = 0;
    if (nres) {
        if (nacc) {
            CK(cub::DeviceRadixSort::SortKeys(d_tmp, tmp_bytes, d_a, d_b, (uint32_t)nacc, AzbGrowByKey{}, h->stream));
            azb_grow_below_kernel<<<(uint32_t)((nacc + 255) / 256), 256, 0, h->stream>>>(d_b, (uint32_t)nacc, bound, &d_sc->below);
            h->launches += 1;
            CK(cudaGetLastError());
        }
        if (sharded) {
            const unsigned long long mk = std::min<uint64_t>(k, nacc);
            unsigned long long *mine = d_top + tw * world;
            CK(cudaMemcpyAsync(mine, &mk, 8, cudaMemcpyHostToDevice, h->stream));
            CK(cudaMemcpyAsync(mine + 1, &d_sc->below, 8, cudaMemcpyDeviceToDevice, h->stream));
            if (mk) CK(cudaMemcpyAsync(mine + 2, d_b, mk * E, cudaMemcpyDeviceToDevice, h->stream));
            rc = comm_allgather(h, mine, d_top, tw);
            if (rc) return rc;
            std::vector<unsigned long long> top(tw * world);
            CK(cudaMemcpyAsync(top.data(), d_top, top.size() * 8, cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            std::vector<AzbGrowEnt> all;
            for (uint32_t r = 0; r < world; ++r) {
                const unsigned long long *tr = top.data() + tw * r;
                below += tr[1];
                for (unsigned long long i = 0; i < tr[0]; ++i) all.push_back(AzbGrowEnt{tr[2 + 3 * i], tr[3 + 3 * i], tr[4 + 3 * i]});
            }
            std::sort(all.begin(), all.end(), [](const AzbGrowEnt &a, const AzbGrowEnt &b) {
                return std::tie(a.key, a.hi, a.lo) < std::tie(b.key, b.hi, b.lo);
            });
            CK(cudaMemcpyAsync(d_b, all.data(), (size_t)nres * E, cudaMemcpyHostToDevice, h->stream));
        }
        azb_grow_decode_kernel<<<(nres + 255) / 256, 256, 0, h->stream>>>(d_b, nres, N, d_res);
        h->launches += 1;
        CK(cudaGetLastError());
        rc = cost_tail(h, d_res, nres, N, d_res_cost, nullptr, h->ev1, parents, lambda1, mu, eval, &cerr);
        if (rc) return rc;
        CK(cudaMemcpyAsync(res.data(), d_b, (size_t)nres * E, cudaMemcpyDeviceToHost, h->stream));
        if (!sharded) CK(cudaMemcpyAsync(&below, &d_sc->below, 8, cudaMemcpyDeviceToHost, h->stream));
    } else {
        CK(cudaEventRecord(h->ev1, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    if (ms) CK(cudaEventElapsedTime(ms, h->ev0, h->ev1));
    if (cerr) return fail(h, AZB_ERR_LAMBDA, "%s", azb_strerror(AZB_ERR_LAMBDA));
    if (codes)
        for (uint32_t i = 0; i < nres; ++i) {
            codes[2 * i] = res[i].hi;
            codes[2 * i + 1] = res[i].lo;
        }
    if (n_out) *n_out = nres;
    if (n_within) *n_within = total;
    if (n_below) *n_below = below;
    if (proof) memcpy(proof, pw, sizeof(pw));
    return AZB_OK;
}

extern "C" int azb_trees_within(azb_handle *h, double bound, uint32_t k, uint64_t max_level, uint32_t *n_out, uint64_t *n_within,
                                uint64_t *n_below, uint64_t *codes, uint8_t *parents, double *lambda1, uint32_t *mu, float *eval,
                                float *ms) {
    if (!h) return AZB_ERR_INVALID;
    if (k == 0 || k > AZB_BEST_MAX_K) return fail(h, AZB_ERR_INVALID, "k must be in 1..%u, got %u", AZB_BEST_MAX_K, k);
    if (std::isnan(bound)) return fail(h, AZB_ERR_INVALID, "azb_trees_within: the bound is NaN");
    return trees_within(h, false, bound, k, max_level, n_out, n_within, n_below, codes, parents, lambda1, mu, eval, nullptr, ms);
}

extern "C" int azb_trees_within_proof(azb_handle *h, double bound, uint32_t k, uint64_t max_level, uint32_t *n_out,
                                      uint64_t *n_within, uint64_t *n_below, uint64_t *codes, uint8_t *parents, double *lambda1,
                                      uint32_t *mu, float *eval, uint64_t *proof, float *ms) {
    if (!h) return AZB_ERR_INVALID;
    if (k == 0 || k > AZB_BEST_MAX_K) return fail(h, AZB_ERR_INVALID, "k must be in 1..%u, got %u", AZB_BEST_MAX_K, k);
    if (std::isnan(bound)) return fail(h, AZB_ERR_INVALID, "azb_trees_within_proof: the bound is NaN");
    uint64_t pw[5];
    return trees_within(h, false, bound, k, max_level, n_out, n_within, n_below, codes, parents, lambda1, mu, eval,
                        proof ? proof : pw, ms);
}

extern "C" int azb_comm_trees_within(azb_handle *h, double bound, uint32_t k, uint64_t max_level, uint32_t *n_out,
                                     uint64_t *n_within, uint64_t *n_below, uint64_t *codes, uint8_t *parents, double *lambda1,
                                     uint32_t *mu, float *eval, float *ms) {
    if (!h) return AZB_ERR_INVALID;
    if (!h->nccl_comm) return fail(h, AZB_ERR_STATE, "azb_comm_init has not been called");
    if (h->comm_world > AZB_GROW_MAX_WORLD)
        return fail(h, AZB_ERR_INVALID, "azb_comm_trees_within: %d ranks, at most %u", h->comm_world, AZB_GROW_MAX_WORLD);
    return trees_within(h, true, bound, k, max_level, n_out, n_within, n_below, codes, parents, lambda1, mu, eval, nullptr, ms);
}

// cascade waves that outgrew the shared-memory work list and continued in global scratch since azb_create (diagnostic;
// tests use it to prove that a dense transposition DAG really exercised that path)
extern "C" int azb_debug_cascade_spills(azb_handle *h, uint32_t *out) {
    if (!h || !out) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(out, &h->L.g->casc_spills, 4, cudaMemcpyDeviceToHost));
    return AZB_OK;
}

int azb_reset_counters(azb_handle *h) {
    if (!h) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    if (h->trees_init) {
        int rc = flush_pending(h);
        if (rc) return rc;
    }
    CK(cudaMemsetAsync(&h->L.g->counters, 0, sizeof(AzbCounters), h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return AZB_OK;
}

int azb_get_state_vecs(azb_handle *h, float *state_vecs) {
    if (!h || !state_vecs) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    return copy_state_vecs(h, state_vecs);
}

int azb_get_priors(azb_handle *h, float *priors) {
    if (!h || !priors) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaMemcpy2DAsync(priors, (size_t)h->A * 4, h->L.h, (size_t)h->L.h_ld * 4, (size_t)h->A * 4, h->L.B,
                         cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return AZB_OK;
}

// ---- epoch boundary: observations (tree/mod.rs:242-264, optimizer/mod.rs:253-278) ----
int azb_write_observations(azb_handle *h, uint32_t n_obs_tol, float *state_vecs, float *observations, float *weights) {
    if (!h || !observations || !weights) return AZB_ERR_INVALID;
    if (!h->trees_init) return fail(h, AZB_ERR_STATE, "azb_init_trees has not been called");
    CK(cudaSetDevice(h->cfg.device));
    int rc = flush_pending(h);
    if (rc) return rc;
    const uint32_t B = h->L.B;
    if (!h->obs) {
        CK(dmalloc(h, &h->obs, (size_t)B * h->A));
        CK(dmalloc(h, &h->obs_w, (size_t)B * h->A));
    }
    const uint32_t blocks = (B + 3) / 4;
    azb_observe_kernel<<<blocks, 128, 0, h->stream>>>(h->L, n_obs_tol, h->obs, h->obs_w, state_vecs ? h->L.sv : nullptr);
    h->launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(observations, h->obs, (size_t)B * h->A * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(weights, h->obs_w, (size_t)B * h->A * 4, cudaMemcpyDeviceToHost, h->stream));
    if (state_vecs)
        CK(cudaMemcpy2DAsync(state_vecs, (size_t)h->S * 4, h->L.sv, (size_t)h->L.sv_ld * 4, (size_t)h->S * 4, B,
                             cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return AZB_OK;
}


// ---- epoch boundary: the training step (nabla/model/dfdx.rs:86-131; optimizer/mod.rs:249-281) -------------------
// NCCL is loaded on demand (dlopen) so that the library has no hard dependency on it; only the epoch boundary
// communicates (SURVEY.md §8e): all-reduce of the weight sum, the gradient and the loss, all-gather of the argmins.
typedef struct { char internal[128]; } azb_nccl_uid;
typedef int (*nccl_get_uid_fn)(azb_nccl_uid *);
typedef int (*nccl_init_rank_fn)(void **, int, azb_nccl_uid, int);
typedef int (*nccl_allreduce_fn)(const void *, void *, size_t, int, int, void *, cudaStream_t);
typedef int (*nccl_allgather_fn)(const void *, void *, size_t, int, void *, cudaStream_t);
typedef int (*nccl_destroy_fn)(void *);
typedef const char *(*nccl_errstr_fn)(int);
typedef int (*nccl_send_fn)(const void *, size_t, int, int, void *, cudaStream_t);  // ncclSend / ncclRecv: buffer, count, type, peer
typedef int (*nccl_recv_fn)(void *, size_t, int, int, void *, cudaStream_t);
typedef int (*nccl_group_fn)(void);
enum { AZB_NCCL_UINT32 = 3, AZB_NCCL_UINT64 = 5, AZB_NCCL_FLOAT32 = 7, AZB_NCCL_FLOAT64 = 8, AZB_NCCL_SUM = 0 };  // nccl.h: ncclDataType_t / ncclRedOp_t

static void *nccl_open(void) {
    static void *lib = nullptr;
    if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    return lib;
}

static void azb_comm_destroy_impl(azb_handle *h) {
    if (h->nccl_comm && h->nccl_lib) {
        auto destroy = (nccl_destroy_fn)dlsym(h->nccl_lib, "ncclCommDestroy");
        if (destroy) destroy(h->nccl_comm);
    }
    h->nccl_comm = nullptr;
}

#define NCCLCK(call)                                                                                   \
    do {                                                                                               \
        int r_ = (call);                                                                               \
        if (r_ != 0) {                                                                                 \
            auto es_ = (nccl_errstr_fn)dlsym(h->nccl_lib, "ncclGetErrorString");                       \
            return fail(h, AZB_ERR_CUDA, "%s: NCCL error %d (%s)", #call, r_, es_ ? es_(r_) : "?");  \
        }                                                                                              \
    } while (0)

static int comm_allreduce(azb_handle *h, void *buf, size_t count, int dtype) {
    if (!h->nccl_comm || h->comm_world <= 1) return AZB_OK;
    auto ar = (nccl_allreduce_fn)dlsym(h->nccl_lib, "ncclAllReduce");
    if (!ar) return fail(h, AZB_ERR_CUDA, "ncclAllReduce not found");
    NCCLCK(ar(buf, buf, count, dtype, AZB_NCCL_SUM, h->nccl_comm, h->stream));
    return AZB_OK;
}

// azb_comm_trees_within: an all-gather of `count` u64 words per rank
static int comm_allgather(azb_handle *h, const unsigned long long *send, unsigned long long *recv, size_t count) {
    auto ag = (nccl_allgather_fn)dlsym(h->nccl_lib, "ncclAllGather");
    if (!ag) return fail(h, AZB_ERR_CUDA, "ncclAllGather not found");
    NCCLCK(ag(send, recv, count, AZB_NCCL_UINT64, h->nccl_comm, h->stream));
    return AZB_OK;
}

// azb_comm_trees_within: the runs of one round.  rec = the round's all-gathered records; this rank's run for rank d
// (rec[me][d] codes, runs in rank order at send) goes to d, and d's run for this rank lands at recv in rank order.  The
// own run is a device copy.
static int comm_exchange(azb_handle *h, const ulonglong2 *send, const unsigned long long *rec, ulonglong2 *recv) {
    const uint32_t world = (uint32_t)h->comm_world, me = (uint32_t)h->comm_rank;
    const size_t R = world + WR_WORDS;
    auto snd = (nccl_send_fn)dlsym(h->nccl_lib, "ncclSend");
    auto rcv = (nccl_recv_fn)dlsym(h->nccl_lib, "ncclRecv");
    auto gstart = (nccl_group_fn)dlsym(h->nccl_lib, "ncclGroupStart");
    auto gend = (nccl_group_fn)dlsym(h->nccl_lib, "ncclGroupEnd");
    if (!snd || !rcv || !gstart || !gend) return fail(h, AZB_ERR_CUDA, "ncclSend, ncclRecv, ncclGroupStart or ncclGroupEnd not found");
    unsigned long long so = 0, ro = 0, self_so = 0, self_ro = 0;
    NCCLCK(gstart());
    for (uint32_t d = 0; d < world; ++d) {
        const unsigned long long ns = rec[R * me + d], nr = rec[R * d + me];
        if (d == me) {
            self_so = so;
            self_ro = ro;
        } else {
            if (ns) NCCLCK(snd(send + so, 2 * ns, AZB_NCCL_UINT64, (int)d, h->nccl_comm, h->stream));
            if (nr) NCCLCK(rcv(recv + ro, 2 * nr, AZB_NCCL_UINT64, (int)d, h->nccl_comm, h->stream));
        }
        so += ns;
        ro += nr;
    }
    NCCLCK(gend());
    const unsigned long long own = rec[R * me + me];
    if (own) CK(cudaMemcpyAsync(recv + self_ro, send + self_so, own * 16, cudaMemcpyDeviceToDevice, h->stream));
    return AZB_OK;
}

static int train_alloc(azb_handle *h) {
    if (h->grad) return AZB_OK;
    const size_t B = h->L.B;
    uint32_t widest = h->A;
    for (int l = 1; l < 4; ++l) widest = std::max(widest, h->dims[l]);
    CK(dmalloc(h, &h->grad, h->n_params));
    CK(dmalloc(h, &h->adam_m, h->n_params));
    CK(dmalloc(h, &h->adam_v, h->n_params));
    CK(dmalloc(h, &h->tr_p, B * h->A));
    CK(dmalloc(h, &h->tr_dz[0], B * widest));
    CK(dmalloc(h, &h->tr_dz[1], B * widest));
    CK(dmalloc(h, &h->tr_scal, 4));
    CK(dmalloc(h, &h->tr_part, 1024));
    CK(cudaMemsetAsync(h->grad, 0, h->n_params * 4, h->stream));
    CK(cudaMemsetAsync(h->adam_m, 0, h->n_params * 4, h->stream));
    CK(cudaMemsetAsync(h->adam_v, 0, h->n_params * 4, h->stream));
    if (!h->obs) {
        CK(dmalloc(h, &h->obs, B * h->A));
        CK(dmalloc(h, &h->obs_w, B * h->A));
    }
    return AZB_OK;
}

// forward (f32, activations kept) + loss + backward into h->grad for device rows x[rows][ldx], o, w [rows][A];
// with a communicator the weight sum, the gradient and the loss are global sums.  Leaves the loss in tr_scal[1].
static int train_backward(azb_handle *h, const float *x, uint32_t ldx, const float *o, const float *w, uint32_t rows) {
    if (!h->params_set) return fail(h, AZB_ERR_STATE, "model parameters not set");
    int rc = train_alloc(h);
    if (rc) return rc;
    cudaStream_t st = h->stream;
    const size_t n_out = (size_t)rows * h->A;
    const uint32_t nblk = (uint32_t)std::min<size_t>(1024, (n_out + 255) / 256);
    // weight_sum = action_weights.iter().sum() (dfdx.rs:105)
    azb_sum_partial_kernel<<<nblk, 256, 0, st>>>(w, n_out, h->tr_part);
    azb_sum_final_kernel<<<1, 256, 0, st>>>(h->tr_part, nblk, h->tr_scal);
    h->launches += 2;
    rc = comm_allreduce(h, h->tr_scal, 1, AZB_NCCL_FLOAT64);
    if (rc) return rc;
    {
        // The loss divides every weight by this sum (dfdx.rs:106-110).  With no observation at all (no root child is
        // exhausted or has n_t >= n_obs_tol: short epochs) it is 0/0: the reference's step would write NaN into every
        // parameter.  Here the step is refused before anything is computed; the sum is global, so every rank of a
        // sharded run takes the same branch.
        double wsum = 0.0;
        CK(cudaMemcpyAsync(&wsum, h->tr_scal, 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (!(wsum > 0.0) || !std::isfinite(wsum))
            return fail(h, AZB_ERR_STATE, "no observations: the action weights sum to %g, the model is left unchanged", wsum);
    }
    // forward, f32 (dfdx.rs:115-116)
    {
        const float *in = x;
        uint32_t ld_in = ldx;
        const float *p = h->params;
        for (int l = 0; l < 4; ++l) {
            const uint32_t K = h->dims[l], Nout = h->dims[l + 1];
            float *outp = l < 3 ? h->act[l] : h->tr_p;
            dim3 grid((Nout + 63) / 64, (rows + 63) / 64);
            if (l < 3)
                azb_linear_fp32_kernel<AZB_ACT_RELU><<<grid, 256, 0, st>>>(in, ld_in, p, p + (size_t)K * Nout, outp, Nout, rows, K, Nout);
            else
                azb_linear_fp32_kernel<AZB_ACT_SIGMOID><<<grid, 256, 0, st>>>(in, ld_in, p, p + (size_t)K * Nout, outp, Nout, rows, K, Nout);
            h->launches += 1;
            in = outp;
            ld_in = Nout;
            p += (size_t)K * Nout + Nout;
        }
    }
    // loss and d loss / d z4 (dfdx.rs:118-126)
    azb_loss_grad_kernel<<<nblk, 256, 0, st>>>(h->tr_p, o, w, n_out, h->tr_scal, h->tr_dz[0], h->tr_part);
    azb_sum_final_kernel<<<1, 256, 0, st>>>(h->tr_part, nblk, h->tr_scal + 1);
    h->launches += 2;
    // backward, last layer first
    size_t off[5];
    off[0] = 0;
    for (int l = 0; l < 4; ++l) off[l + 1] = off[l] + (size_t)h->dims[l] * h->dims[l + 1] + h->dims[l + 1];
    int cur = 0;
    for (int l = 3; l >= 0; --l) {
        const uint32_t K = h->dims[l], Nout = h->dims[l + 1];
        const float *dz = h->tr_dz[cur];
        const float *xin = l == 0 ? x : h->act[l - 1];
        const uint32_t ld_in = l == 0 ? ldx : K;
        {   // dW[out][in] = dZ^T X
            dim3 grid((K + 63) / 64, (Nout + 63) / 64);
            azb_gemm_fp32_kernel<false, true, false><<<grid, 256, 0, st>>>(dz, Nout, xin, ld_in, h->grad + off[l], K, Nout, K, rows, nullptr, 0);
        }
        azb_colsum_kernel<<<(Nout + 31) / 32, 256, 0, st>>>(dz, Nout, rows, Nout, h->grad + off[l] + (size_t)K * Nout);
        h->launches += 2;
        if (l > 0) {  // dX = (dZ W) * relu'(input)
            dim3 grid((K + 63) / 64, (rows + 63) / 64);
            azb_gemm_fp32_kernel<true, true, true><<<grid, 256, 0, st>>>(dz, Nout, h->params + off[l], K, h->tr_dz[cur ^ 1], K, rows, K, Nout, h->act[l - 1], K);
            h->launches += 1;
            cur ^= 1;
        }
    }
    CK(cudaGetLastError());
    rc = comm_allreduce(h, h->grad, h->n_params, AZB_NCCL_FLOAT32);
    if (rc) return rc;
    return comm_allreduce(h, h->tr_scal + 1, 1, AZB_NCCL_FLOAT64);
}

// reads the (global) loss and applies the Adam step, unless the loss is not finite: a NaN gradient would destroy the
// parameters and both moment buffers for good (and, sharded, on every rank), so the step is refused and reported
static int train_finish(azb_handle *h, float *loss);

static int train_adam(azb_handle *h) {
    h->adam_t += 1;
    AzbAdam cfg = h->adam;
    cfg.bc1 = 1.0f / (1.0f - powf(cfg.beta1, (float)h->adam_t));
    cfg.bc2 = 1.0f / (1.0f - powf(cfg.beta2, (float)h->adam_t));
    const uint32_t nblk = (uint32_t)std::min<size_t>(148 * 8, (h->n_params + 255) / 256);
    azb_adam_kernel<<<nblk, 256, 0, h->stream>>>(h->params, h->grad, h->adam_m, h->adam_v, h->n_params, cfg);
    h->launches += 1;
    CK(cudaGetLastError());
    if (h->tc.ready) {
        const char *why = azb_mlp_tc_load(h->tc, h->params, h->stream, &h->launches);
        if (why) return fail(h, AZB_ERR_CUDA, "tensor-core MLP: %s", why);
    }
    return AZB_OK;
}

static int train_read_loss(azb_handle *h, float *loss) {
    double l = 0;
    CK(cudaMemcpyAsync(&l, h->tr_scal + 1, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (loss) *loss = (float)l;
    return AZB_OK;
}

static int train_finish(azb_handle *h, float *loss) {
    float l = 0.f;
    int rc = train_read_loss(h, &l);
    if (rc) return rc;
    if (loss) *loss = l;
    if (!std::isfinite(l)) {
        CK(cudaMemsetAsync(h->grad, 0, h->n_params * 4, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        return fail(h, AZB_ERR_NAN, "the loss is not finite (%g): Adam step refused, the model is left unchanged", (double)l);
    }
    return train_adam(h);
}

int azb_adam_config(azb_handle *h, float lr, float beta1, float beta2, float eps, float l2) {
    if (!h || !(lr >= 0.f) || !(beta1 >= 0.f && beta1 < 1.f) || !(beta2 >= 0.f && beta2 < 1.f)) return AZB_ERR_INVALID;
    h->adam = AzbAdam{lr, beta1, beta2, eps, l2, 1.f, 1.f};
    return AZB_OK;
}

static int train_stage_host(azb_handle *h, const float *states, const float *observations, const float *weights,
                            uint32_t rows) {
    int rc = train_alloc(h);
    if (rc) return rc;
    if (!h->tr_x) CK(dmalloc(h, &h->tr_x, (size_t)h->L.B * h->S));
    CK(cudaMemcpyAsync(h->tr_x, states, (size_t)rows * h->S * 4, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->obs, observations, (size_t)rows * h->A * 4, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->obs_w, weights, (size_t)rows * h->A * 4, cudaMemcpyHostToDevice, h->stream));
    return AZB_OK;
}

int azb_model_gradients(azb_handle *h, const float *states, const float *observations, const float *action_weights,
                        uint32_t rows, float *loss, float *grads) {
    if (!h || !states || !observations || !action_weights || rows == 0 || rows > h->L.B) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    int rc = train_stage_host(h, states, observations, action_weights, rows);
    if (rc) return rc;
    rc = train_backward(h, h->tr_x, h->S, h->obs, h->obs_w, rows);
    if (rc) return rc;
    if (grads) CK(cudaMemcpyAsync(grads, h->grad, h->n_params * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemsetAsync(h->grad, 0, h->n_params * 4, h->stream));
    return train_read_loss(h, loss);
}

int azb_model_update(azb_handle *h, const float *states, const float *observations, const float *action_weights,
                     uint32_t rows, float *loss) {
    if (!h || !states || !observations || !action_weights || rows == 0 || rows > h->L.B) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    int rc = train_stage_host(h, states, observations, action_weights, rows);
    if (rc) return rc;
    rc = train_backward(h, h->tr_x, h->S, h->obs, h->obs_w, rows);
    if (rc) return rc;
    return train_finish(h, loss);
}

int azb_update_model(azb_handle *h, uint32_t n_obs_tol, float *loss) {
    if (!h) return AZB_ERR_INVALID;
    if (!h->trees_init) return fail(h, AZB_ERR_STATE, "azb_init_trees has not been called");
    CK(cudaSetDevice(h->cfg.device));
    int rc = flush_pending(h);
    if (rc) return rc;
    rc = train_alloc(h);
    if (rc) return rc;
    // write_vec of the roots + write_observations of every tree (optimizer/mod.rs:253-278), all on the device
    azb_observe_kernel<<<(h->L.B + 3) / 4, 128, 0, h->stream>>>(h->L, n_obs_tol, h->obs, h->obs_w, h->L.sv);
    h->launches += 1;
    CK(cudaGetLastError());
    rc = train_backward(h, h->L.sv, h->L.sv_ld, h->obs, h->obs_w, h->L.B);
    if (rc) return rc;
    rc = train_finish(h, loss);
    if (rc) return rc;
    return check_device_error(h);
}

// NablaOptimizer::par_reset_trees (optimizer/mod.rs:284-360) with the example's modify_root policy
// (04-c21-tree.rs:172-206) on the device, then the tail shared with par_new (azb_init_trees)
int azb_reset_trees(azb_handle *h, uint64_t seed, uint32_t k_min, uint32_t k_max) {
    if (!h) return AZB_ERR_INVALID;
    if (!h->trees_init) return fail(h, AZB_ERR_STATE, "azb_init_trees has not been called");
    if (k_max == 0) k_max = h->A / 2;  // num_permitted_actions_range = 5..=(ACTION / 2) (04-c21-tree.rs:85)
    if (k_min == 0) k_min = 5;
    if (k_min > k_max || k_max > h->A || h->A > 2048) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    int rc = flush_pending(h);
    if (rc) return rc;
    azb_modify_roots_kernel<<<(h->L.B + 3) / 4, 128, 0, h->stream>>>(h->L, seed, h->epoch, k_min, k_max);
    h->launches += 1;
    CK(cudaGetLastError());
    h->epoch += 1;
    rc = check_device_error(h);
    if (rc) return rc;
    return azb_init_trees(h);
}

// ---- epoch-boundary communicator ----
int azb_comm_unique_id(uint8_t *id128) {
    if (!id128) return AZB_ERR_INVALID;
    void *lib = nccl_open();
    if (!lib) return AZB_ERR_CUDA;
    auto get = (nccl_get_uid_fn)dlsym(lib, "ncclGetUniqueId");
    azb_nccl_uid id;
    if (!get || get(&id) != 0) return AZB_ERR_CUDA;
    memcpy(id128, &id, 128);
    return AZB_OK;
}

int azb_comm_init(azb_handle *h, const uint8_t *id128, int rank, int world) {
    if (!h || !id128 || world < 1 || rank < 0 || rank >= world) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    if (h->nccl_comm) azb_comm_destroy_impl(h);
    h->nccl_lib = nccl_open();
    if (!h->nccl_lib) return fail(h, AZB_ERR_CUDA, "libnccl.so.2 not found: %s", dlerror());
    auto init = (nccl_init_rank_fn)dlsym(h->nccl_lib, "ncclCommInitRank");
    if (!init) return fail(h, AZB_ERR_CUDA, "ncclCommInitRank not found");
    azb_nccl_uid id;
    memcpy(&id, id128, 128);
    NCCLCK(init(&h->nccl_comm, world, id, rank));
    h->comm_rank = rank;
    h->comm_world = world;
    if (!h->comm_buf) CK(dmalloc(h, &h->comm_buf, (size_t)80 * (world + 1)));
    return AZB_OK;
}

// global argmin over all ranks' roots (optimizer/mod.rs:221 over the sharded batch): all-gather of
// {orderable eval, state}; the lowest rank wins ties (ranks own ascending blocks of roots = the first minimum)
int azb_comm_argmin(azb_handle *h, uint8_t *parents, uint32_t *permitted, double *lambda1, uint32_t *mu, float *eval,
                    int *owner_rank) {
    if (!h) return AZB_ERR_INVALID;
    if (!h->trees_init) return fail(h, AZB_ERR_STATE, "azb_init_trees has not been called");
    if (!h->nccl_comm) return fail(h, AZB_ERR_STATE, "azb_comm_init has not been called");
    CK(cudaSetDevice(h->cfg.device));
    const int world = h->comm_world;
    // record = best_c (1 word) + pad (2) + argmin_state (77 words) = 80 words, contiguous in AzbGlobals
    uint32_t *mine = h->comm_buf + (size_t)80 * world;
    CK(cudaMemcpyAsync(mine, &h->L.g->best_c, 4, cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaMemcpyAsync(mine + 3, h->L.g->argmin_state, 77 * 4, cudaMemcpyDeviceToDevice, h->stream));
    auto ag = (nccl_allgather_fn)dlsym(h->nccl_lib, "ncclAllGather");
    if (!ag) return fail(h, AZB_ERR_CUDA, "ncclAllGather not found");
    NCCLCK(ag(mine, h->comm_buf, 80, AZB_NCCL_UINT32, h->nccl_comm, h->stream));
    std::vector<uint32_t> all((size_t)80 * world);
    CK(cudaMemcpyAsync(all.data(), h->comm_buf, all.size() * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    int best = 0;
    for (int r = 1; r < world; ++r)
        if (all[(size_t)80 * r] < all[(size_t)80 * best]) best = r;
    const uint32_t *rec = all.data() + (size_t)80 * best;
    uint8_t par[AZB_MAX_VERTICES];
    memcpy(par, rec + 3, h->N);
    if (parents) memcpy(parents, par, h->N);
    if (permitted) memcpy(permitted, rec + 3 + 16, (size_t)h->W * 4);
    double l1 = 0;
    uint32_t m = 0;
    float c = 0;
    int rc = eval_costs_dev(h, par, 1, &l1, &m, &c, nullptr);
    if (rc) return rc;
    if (lambda1) *lambda1 = l1;
    if (mu) *mu = m;
    if (eval) *eval = c;
    if (owner_rank) *owner_rank = best;
    return AZB_OK;
}

// measurement helper: `reps` all-reduces of the gradient buffer (the 1 284 248 floats azb_update_model reduces once per
// epoch) back to back between two events; *ms = time per all-reduce.  The buffer holds zeros between training steps.
int azb_comm_allreduce_bench(azb_handle *h, uint32_t reps, float *ms) {
    if (!h || !ms || reps == 0) return AZB_ERR_INVALID;
    if (!h->nccl_comm) return fail(h, AZB_ERR_STATE, "azb_comm_init has not been called");
    CK(cudaSetDevice(h->cfg.device));
    int rc = train_alloc(h);
    if (rc) return rc;
    rc = comm_allreduce(h, h->grad, h->n_params, AZB_NCCL_FLOAT32);  // warm-up (channel set-up)
    if (rc) return rc;
    CK(cudaEventRecord(h->ev0, h->stream));
    for (uint32_t i = 0; i < reps && rc == AZB_OK; ++i) rc = comm_allreduce(h, h->grad, h->n_params, AZB_NCCL_FLOAT32);
    if (rc) return rc;
    CK(cudaEventRecord(h->ev1, h->stream));
    CK(cudaEventSynchronize(h->ev1));
    float t = 0.f;
    CK(cudaEventElapsedTime(&t, h->ev0, h->ev1));
    *ms = t / (float)reps;
    return AZB_OK;
}

int azb_comm_destroy(azb_handle *h) {
    if (!h) return AZB_ERR_INVALID;
    azb_comm_destroy_impl(h);
    return AZB_OK;
}

// ---- measurement helpers ----
int azb_kernel_launches(const azb_handle *h, uint64_t *n) {
    if (!h || !n) return AZB_ERR_INVALID;
    *n = h->launches;
    return AZB_OK;
}

int azb_device_bytes(const azb_handle *h, uint64_t *bytes) {
    if (!h || !bytes) return AZB_ERR_INVALID;
    *bytes = h->dev_bytes;
    return AZB_OK;
}

int azb_flush_l2(azb_handle *h) {
    if (!h) return AZB_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    if (!h->flush_buf) {
        h->flush_bytes = (size_t)256 << 20;  // > 126 MB of L2
        CK(dmalloc(h, (uint8_t **)&h->flush_buf, h->flush_bytes));
    }
    CK(cudaMemsetAsync(h->flush_buf, 0x5a, h->flush_bytes, h->stream));
    return AZB_OK;
}

}  // extern "C"

// ---- checkpoints (azb_ckpt.cuh; format in include/azb.h) ------------------------------------------------------------
enum {
    CK_MAGIC = 0, CK_FORMAT, CK_VERSION, CK_BYTES, CK_N, CK_CLO, CK_CUP, CK_TOL, CK_TOL_LEN = CK_TOL + AZB_MAX_TOL, CK_TOL_DEF,
    CK_HIDDEN, CK_MLP_MODE = CK_HIDDEN + 3, CK_PRIOR_MODE, CK_PRIOR_SEED, CK_SELECTION, CK_PUCT_C, CK_FIRST, CK_NROOTS,
    CK_STEPS, CK_EPOCH, CK_ADAM_T, CK_ADAM, CK_FLAGS = CK_ADAM + 5, CK_BEST_C, CK_BEST_ROOT, CK_BEST_NODE, CK_BEST_STATE,
    CK_NPARAMS = CK_BEST_STATE + 39, CK_MODEL_OFF, CK_MODEL_BYTES, CK_TABLE_OFF, CK_TABLE_BYTES, CK_TREES_OFF, CK_TREES_BYTES,
    CK_MODEL_DIGEST, CK_TABLE_DIGEST, CK_HDR_DIGEST = AZB_CKPT_HEADER_WORDS - 1
};
static_assert(CK_TABLE_DIGEST < CK_HDR_DIGEST, "checkpoint header layout");
static const uint64_t k_ckpt_hdr_bytes = AZB_CKPT_HEADER_WORDS * 8ull;
static const uint64_t k_ckpt_half_max = 128ull << 20;  // each of the staging area's two halves: 256 MB in all

static uint64_t ckpt_digest(const void *p, uint64_t n) {  // include/azb.h; the buffer need not be 8-byte aligned
    const uint8_t *b = static_cast<const uint8_t *>(p);
    uint64_t s = 0;
    for (uint64_t i = 0; i < n; ++i) {
        uint64_t w;
        memcpy(&w, b + 8 * i, 8);
        s += azb_ckpt_term(w, i);
    }
    return azb_mix64(s ^ n);
}
static uint32_t f2u(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    return u;
}
static uint64_t model_bytes(const azb_handle *h) { return (h->n_params * 12 + 7) & ~7ull; }

// the staging buffers: [len | offsets (B + 1 each) | CUB scratch | bad words | half 0 | half 1]; the layout up to the
// halves does not depend on their size
struct CkptSlab {
    unsigned long long *len, *off, *bad;
    void *tmp;
    size_t tmp_bytes;
    uint8_t *half[2];
};
static int ckpt_slab(azb_handle *h, uint64_t half_bytes, CkptSlab &s) {
    const size_t n = (size_t)h->L.B + 1;
    s.tmp_bytes = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, s.tmp_bytes, (const unsigned long long *)nullptr, (unsigned long long *)nullptr, (int)n,
                                     h->stream));
    int rc = scratch(h, [&](Carve &cv) {
        s.len = cv.take<unsigned long long>(n);
        s.off = cv.take<unsigned long long>(n);
        s.tmp = cv.take<uint8_t>(s.tmp_bytes);
        s.bad = cv.take<unsigned long long>(2);
        s.half[0] = cv.take<uint8_t>(half_bytes);
        s.half[1] = cv.take<uint8_t>(half_bytes);
    });
    if (rc) return rc;
    if (!h->ckpt_stream) {
        CK(cudaStreamCreateWithFlags(&h->ckpt_stream, cudaStreamNonBlocking));
        for (cudaEvent_t &e : h->ckpt_ev) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    return AZB_OK;
}

// chunks of whole records [t0, t1) with at most `half` bytes each (a record larger than that gets a chunk of its own,
// and the halves are sized for the largest record)
static uint64_t ckpt_half_bytes(const azb_handle *h, const uint64_t *off, uint32_t n) {
    uint64_t max_rec = 0;
    for (uint32_t i = 0; i < n; ++i) max_rec = std::max<uint64_t>(max_rec, off[i + 1] - off[i]);
    uint64_t half = h->ckpt_chunk ? h->ckpt_chunk : std::min<uint64_t>(k_ckpt_half_max, (off[n] - off[0] + 1) / 2);
    return std::max(half, max_rec);
}
// CTAs per record for the records [t0, t1): enough slices of AZB_CKPT_SLICE_BYTES for the largest, at most 64
static uint32_t ckpt_slices(const uint64_t *off, uint32_t t0, uint32_t t1) {
    uint64_t m = 0;
    for (uint32_t t = t0; t < t1; ++t) m = std::max<uint64_t>(m, off[t + 1] - off[t]);
    return (uint32_t)std::min<uint64_t>(64, std::max<uint64_t>(1, (m + AZB_CKPT_SLICE_BYTES - 1) / AZB_CKPT_SLICE_BYTES));
}
static std::vector<std::pair<uint32_t, uint32_t>> ckpt_chunks(const uint64_t *off, uint32_t n, uint64_t half) {
    std::vector<std::pair<uint32_t, uint32_t>> out;
    for (uint32_t t0 = 0; t0 < n;) {
        uint32_t t1 = t0 + 1;
        while (t1 < n && off[t1 + 1] - off[t0] <= half) ++t1;
        out.emplace_back(t0, t1);
        t0 = t1;
    }
    return out;
}

// the state checks of save / size, the deferred add_actions, and the offset table (host copy; device copy in s.off)
static int ckpt_prepare(azb_handle *h, std::vector<uint64_t> &off, CkptSlab &s, uint64_t half_bytes) {
    if (!h->trees_init) return fail(h, AZB_ERR_STATE, "azb_init_trees has not been called");
    if (h->host_add_pending) return fail(h, AZB_ERR_STATE, "azb_add_actions_host must follow azb_rollout_host first");
    if (h->argmin_from != h->steps_done + 1)
        return fail(h, AZB_ERR_STATE, "enqueued steps are not complete (azb_step(h, 0, ...) first)");
    CK(cudaSetDevice(h->cfg.device));
    int rc = flush_pending(h);
    if (rc) return rc;
    rc = check_device_error(h);
    if (rc) return rc;
    rc = ckpt_slab(h, half_bytes, s);
    if (rc) return rc;
    const uint32_t B = h->L.B;
    azb_ckpt_size_kernel<<<(B + 256) / 256, 256, 0, h->stream>>>(h->L, s.len);
    h->launches += 1;
    CK(cudaGetLastError());
    CK(cub::DeviceScan::ExclusiveSum(s.tmp, s.tmp_bytes, s.len, s.off, (int)B + 1, h->stream));
    h->launches += 1;
    off.resize((size_t)B + 1);
    CK(cudaMemcpyAsync(off.data(), s.off, off.size() * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return AZB_OK;
}

static uint64_t ckpt_total(const azb_handle *h, uint64_t trees_bytes) {
    return k_ckpt_hdr_bytes + model_bytes(h) + ((uint64_t)h->L.B + 1) * 8 + trees_bytes;
}

extern "C" int azb_checkpoint_size(azb_handle *h, uint64_t *bytes) {
    if (!h || !bytes) return AZB_ERR_INVALID;
    std::vector<uint64_t> off;
    CkptSlab s;
    int rc = ckpt_prepare(h, off, s, 0);
    if (rc) return rc;
    *bytes = ckpt_total(h, off.back());
    return AZB_OK;
}

extern "C" int azb_checkpoint_save(azb_handle *h, void *buf, uint64_t size, uint64_t *written) {
    if (!h || !buf) return AZB_ERR_INVALID;
    std::vector<uint64_t> off;
    CkptSlab s;
    int rc = ckpt_prepare(h, off, s, 0);
    if (rc) return rc;
    const uint32_t B = h->L.B;
    const uint64_t total = ckpt_total(h, off.back());
    if (size < total) return fail(h, AZB_ERR_INVALID, "the buffer holds %llu bytes, the checkpoint needs %llu", (unsigned long long)size,
                                  (unsigned long long)total);
    const uint64_t half = ckpt_half_bytes(h, off.data(), B);
    rc = ckpt_slab(h, half, s);  // the offsets stay where ckpt_prepare left them (a grown slab is re-filled below)
    if (rc) return rc;
    CK(cudaMemcpyAsync(s.off, off.data(), off.size() * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemsetAsync(s.len, 0, ((size_t)B + 1) * 8, h->stream));  // the digest sums
    uint8_t *out = static_cast<uint8_t *>(buf);
    const uint64_t o_model = k_ckpt_hdr_bytes, o_table = o_model + model_bytes(h), o_trees = o_table + ((uint64_t)B + 1) * 8;
    // trees: chunk c is packed into half c & 1 while chunk c - 1 goes to the host on the copy stream
    const auto chunks = ckpt_chunks(off.data(), B, half);
    cudaEvent_t *packed = h->ckpt_ev, *copied = h->ckpt_ev + 2;
    auto pack = [&](size_t c) -> int {
        if (c >= 2) CK(cudaStreamWaitEvent(h->stream, copied[c & 1], 0));
        const uint32_t t0 = chunks[c].first, t1 = chunks[c].second;
        uint32_t *stage = reinterpret_cast<uint32_t *>(s.half[c & 1]);
        azb_ckpt_pack_kernel<<<dim3(t1 - t0, ckpt_slices(off.data(), t0, t1)), AZB_CKPT_THREADS, 0, h->stream>>>(h->L, s.off, t0, off[t0],
                                                                                                           stage, s.len);
        azb_ckpt_pack_finish_kernel<<<(t1 - t0 + 255) / 256, 256, 0, h->stream>>>(h->L, s.off, t0, t1, off[t0], stage, s.len);
        h->launches += 2;
        CK(cudaGetLastError());
        CK(cudaEventRecord(packed[c & 1], h->stream));
        return AZB_OK;
    };
    if (!chunks.empty()) {
        rc = pack(0);
        if (rc) return rc;
    }
    for (size_t c = 0; c < chunks.size(); ++c) {
        if (c + 1 < chunks.size()) {
            rc = pack(c + 1);
            if (rc) return rc;
        }
        const uint32_t t0 = chunks[c].first, t1 = chunks[c].second;
        CK(cudaStreamWaitEvent(h->ckpt_stream, packed[c & 1], 0));
        CK(cudaMemcpyAsync(out + o_trees + off[t0], s.half[c & 1], off[t1] - off[t0], cudaMemcpyDeviceToHost, h->ckpt_stream));
        CK(cudaEventRecord(copied[c & 1], h->ckpt_stream));
    }
    // model, running best
    const size_t n = h->n_params;
    memset(out + o_model, 0, model_bytes(h));
    if (h->params_set) CK(cudaMemcpyAsync(out + o_model, h->params, n * 4, cudaMemcpyDeviceToHost, h->stream));
    if (h->adam_m) {
        CK(cudaMemcpyAsync(out + o_model + n * 4, h->adam_m, n * 4, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(out + o_model + n * 8, h->adam_v, n * 4, cudaMemcpyDeviceToHost, h->stream));
    }
    AzbGlobals g;
    CK(cudaMemcpyAsync(&g, h->L.g, sizeof(g), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaStreamSynchronize(h->ckpt_stream));
    memcpy(out + o_table, off.data(), off.size() * 8);
    uint64_t hw[AZB_CKPT_HEADER_WORDS];
    memset(hw, 0, sizeof(hw));
    const azb_config &cf = h->cfg;
    hw[CK_MAGIC] = AZB_CKPT_MAGIC;
    hw[CK_FORMAT] = AZB_CKPT_FORMAT;
    hw[CK_VERSION] = AZB_VERSION;
    hw[CK_BYTES] = total;
    hw[CK_N] = cf.n_vertices;
    hw[CK_CLO] = f2u(cf.c_lower);
    hw[CK_CUP] = f2u(cf.c_upper);
    for (int i = 0; i < AZB_MAX_TOL; ++i) hw[CK_TOL + i] = cf.n_as_tol[i];
    hw[CK_TOL_LEN] = cf.n_as_tol_len;
    hw[CK_TOL_DEF] = cf.n_as_tol_default;
    for (int i = 0; i < 3; ++i) hw[CK_HIDDEN + i] = cf.mlp_hidden[i];
    hw[CK_MLP_MODE] = cf.mlp_mode;
    hw[CK_PRIOR_MODE] = cf.prior_mode;
    hw[CK_PRIOR_SEED] = cf.prior_seed;
    hw[CK_SELECTION] = cf.selection;
    hw[CK_PUCT_C] = f2u(cf.puct_c);
    hw[CK_FIRST] = cf.first_root;
    hw[CK_NROOTS] = B;
    hw[CK_STEPS] = h->steps_done;
    hw[CK_EPOCH] = h->epoch;
    hw[CK_ADAM_T] = h->adam_t;
    const float adam[5] = {h->adam.lr, h->adam.beta1, h->adam.beta2, h->adam.eps, h->adam.l2};
    for (int i = 0; i < 5; ++i) hw[CK_ADAM + i] = f2u(adam[i]);
    hw[CK_FLAGS] = h->params_set ? 1u : 0u;
    hw[CK_BEST_C] = g.best_c;
    hw[CK_BEST_ROOT] = g.argmin_tree == AZB_NONE ? h->ckpt_best_root : cf.first_root + g.argmin_tree;
    hw[CK_BEST_NODE] = g.argmin_tree == AZB_NONE ? h->ckpt_best_node : g.argmin_node;
    memcpy(hw + CK_BEST_STATE, g.argmin_state, sizeof(g.argmin_state));
    hw[CK_NPARAMS] = n;
    hw[CK_MODEL_OFF] = o_model;
    hw[CK_MODEL_BYTES] = model_bytes(h);
    hw[CK_TABLE_OFF] = o_table;
    hw[CK_TABLE_BYTES] = ((uint64_t)B + 1) * 8;
    hw[CK_TREES_OFF] = o_trees;
    hw[CK_TREES_BYTES] = off.back();
    hw[CK_MODEL_DIGEST] = ckpt_digest(out + o_model, model_bytes(h) / 8);
    hw[CK_TABLE_DIGEST] = ckpt_digest(out + o_table, (uint64_t)B + 1);
    hw[CK_HDR_DIGEST] = ckpt_digest(hw, CK_HDR_DIGEST);
    memcpy(out, hw, sizeof(hw));
    if (written) *written = total;
    return AZB_OK;
}

// one blob's header, checked against itself and the handle
struct CkptBlob {
    const uint8_t *p;
    uint64_t size, first, n;
    uint64_t hw[AZB_CKPT_HEADER_WORDS];
};

static int ckpt_check_header(azb_handle *h, uint32_t i, CkptBlob &b) {
    if (b.size < k_ckpt_hdr_bytes) return fail(h, AZB_ERR_INVALID, "blob %u: %llu bytes, shorter than a header", i, (unsigned long long)b.size);
    memcpy(b.hw, b.p, k_ckpt_hdr_bytes);
    const uint64_t *w = b.hw;
    if (w[CK_MAGIC] != AZB_CKPT_MAGIC) return fail(h, AZB_ERR_INVALID, "blob %u: bad magic", i);
    if (w[CK_FORMAT] != AZB_CKPT_FORMAT) return fail(h, AZB_ERR_INVALID, "blob %u: format %llu, expected %d", i, (unsigned long long)w[CK_FORMAT], AZB_CKPT_FORMAT);
    if (w[CK_VERSION] != AZB_VERSION) return fail(h, AZB_ERR_INVALID, "blob %u: version %llu, expected %d", i, (unsigned long long)w[CK_VERSION], AZB_VERSION);
    if (ckpt_digest(w, CK_HDR_DIGEST) != w[CK_HDR_DIGEST]) return fail(h, AZB_ERR_INVALID, "blob %u: header digest", i);
    if (w[CK_BYTES] != b.size)
        return fail(h, AZB_ERR_INVALID, "blob %u: %llu bytes, its header says %llu (truncated?)", i, (unsigned long long)b.size,
                    (unsigned long long)w[CK_BYTES]);
    const azb_config &cf = h->cfg;
    struct { const char *name; uint64_t have, want; } fields[] = {
        {"n_vertices", w[CK_N], cf.n_vertices}, {"c_lower", w[CK_CLO], f2u(cf.c_lower)}, {"c_upper", w[CK_CUP], f2u(cf.c_upper)},
        {"n_as_tol_len", w[CK_TOL_LEN], cf.n_as_tol_len}, {"n_as_tol_default", w[CK_TOL_DEF], cf.n_as_tol_default},
        {"mlp_hidden[0]", w[CK_HIDDEN], cf.mlp_hidden[0]}, {"mlp_hidden[1]", w[CK_HIDDEN + 1], cf.mlp_hidden[1]},
        {"mlp_hidden[2]", w[CK_HIDDEN + 2], cf.mlp_hidden[2]}, {"mlp_mode", w[CK_MLP_MODE], cf.mlp_mode},
        {"prior_mode", w[CK_PRIOR_MODE], cf.prior_mode}, {"prior_seed", w[CK_PRIOR_SEED], cf.prior_seed},
        {"selection", w[CK_SELECTION], cf.selection}, {"puct_c", w[CK_PUCT_C], f2u(cf.puct_c)}, {"n_params", w[CK_NPARAMS], h->n_params}};
    for (const auto &f : fields)
        if (f.have != f.want) return fail(h, AZB_ERR_INVALID, "blob %u: config field %s differs from the handle's", i, f.name);
    for (uint32_t k = 0; k < cf.n_as_tol_len; ++k)
        if (w[CK_TOL + k] != cf.n_as_tol[k]) return fail(h, AZB_ERR_INVALID, "blob %u: config field n_as_tol[%u] differs from the handle's", i, k);
    b.first = w[CK_FIRST];
    b.n = w[CK_NROOTS];
    const uint64_t o_model = k_ckpt_hdr_bytes, o_table = o_model + model_bytes(h), o_trees = o_table + (b.n + 1) * 8;
    if (b.n == 0 || w[CK_MODEL_OFF] != o_model || w[CK_MODEL_BYTES] != model_bytes(h) || w[CK_TABLE_OFF] != o_table ||
        w[CK_TABLE_BYTES] != (b.n + 1) * 8 || w[CK_TREES_OFF] != o_trees || o_trees + w[CK_TREES_BYTES] != b.size)
        return fail(h, AZB_ERR_INVALID, "blob %u: section table", i);
    if (w[CK_STEPS] > 0xffffffffull || w[CK_ADAM_T] > 0xffffffffull) return fail(h, AZB_ERR_INVALID, "blob %u: step counts", i);
    return AZB_OK;
}

// everything a failed load leaves: the trees are invalid until a load succeeds or set_roots + init_trees run
static void ckpt_invalidate(azb_handle *h) {
    h->trees_init = false;
    h->first_init_done = false;
    h->pending_add = false;
    h->host_add_pending = false;
}

extern "C" int azb_checkpoint_load(azb_handle *h, const void *const *blobs, const uint64_t *sizes, uint32_t n_blobs) {
    if (!h || !blobs || !sizes || n_blobs == 0) return AZB_ERR_INVALID;
    std::vector<CkptBlob> bl(n_blobs);
    for (uint32_t i = 0; i < n_blobs; ++i) {
        if (!blobs[i]) return fail(h, AZB_ERR_INVALID, "blob %u is NULL", i);
        bl[i].p = static_cast<const uint8_t *>(blobs[i]);
        bl[i].size = sizes[i];
        int rc = ckpt_check_header(h, i, bl[i]);
        if (rc) return rc;
    }
    // one run: every blob agrees on the counters, the Adam state and the model
    const CkptBlob &b0 = bl[0];
    const uint64_t mb = model_bytes(h);
    if (ckpt_digest(b0.p + k_ckpt_hdr_bytes, mb / 8) != b0.hw[CK_MODEL_DIGEST]) return fail(h, AZB_ERR_INVALID, "blob 0: model digest");
    for (uint32_t i = 1; i < n_blobs; ++i) {
        static const struct { int w, n; const char *name; } same[] = {
            {CK_STEPS, 1, "steps_done"}, {CK_EPOCH, 1, "reset count"}, {CK_ADAM_T, 1, "Adam step"}, {CK_ADAM, 5, "Adam config"},
            {CK_FLAGS, 1, "flags"}, {CK_MODEL_DIGEST, 1, "model section"}};
        for (const auto &f : same)
            if (memcmp(bl[i].hw + f.w, b0.hw + f.w, 8 * f.n)) return fail(h, AZB_ERR_INVALID, "blob %u: %s differs from blob 0's", i, f.name);
        if (memcmp(bl[i].p + k_ckpt_hdr_bytes, b0.p + k_ckpt_hdr_bytes, mb)) return fail(h, AZB_ERR_INVALID, "blob %u: model section differs from blob 0's", i);
    }
    // ranges: pairwise disjoint, covering [F, F + B) exactly
    const uint64_t F = h->cfg.first_root, B = h->L.B;
    std::vector<uint32_t> ord(n_blobs);
    for (uint32_t i = 0; i < n_blobs; ++i) ord[i] = i;
    std::sort(ord.begin(), ord.end(), [&](uint32_t a, uint32_t b) { return bl[a].first < bl[b].first; });
    for (uint32_t k = 0; k + 1 < n_blobs; ++k)
        if (bl[ord[k]].first + bl[ord[k]].n > bl[ord[k + 1]].first)
            return fail(h, AZB_ERR_INVALID, "blobs %u and %u overlap", ord[k], ord[k + 1]);
    uint64_t covered = F;
    for (uint32_t k = 0; k < n_blobs; ++k) {
        const CkptBlob &b = bl[ord[k]];
        if (b.first + b.n <= F || b.first >= F + B) continue;
        if (b.first > covered) break;
        covered = b.first + b.n;
    }
    if (covered < F + B) return fail(h, AZB_ERR_INVALID, "no blob holds global root %llu of the handle's range", (unsigned long long)covered);
    if (b0.hw[CK_STEPS] > h->cfg.max_steps)
        return fail(h, AZB_ERR_CAPACITY, "the checkpoint is %llu steps into its epoch, max_steps is %u", (unsigned long long)b0.hw[CK_STEPS],
                    h->cfg.max_steps);
    // the offset tables of the blobs that hold some of the handle's roots
    std::vector<std::vector<uint64_t>> tables(n_blobs);
    for (uint32_t i = 0; i < n_blobs; ++i) {
        const CkptBlob &b = bl[i];
        if (b.first + b.n <= F || b.first >= F + B) continue;
        auto &t = tables[i];
        t.resize(b.n + 1);
        memcpy(t.data(), b.p + b.hw[CK_TABLE_OFF], t.size() * 8);
        if (ckpt_digest(t.data(), t.size()) != b.hw[CK_TABLE_DIGEST]) return fail(h, AZB_ERR_INVALID, "blob %u: tree offset table digest", i);
        bool ok = t[0] == 0 && t[b.n] == b.hw[CK_TREES_BYTES];
        for (uint64_t r = 0; r < b.n && ok; ++r) ok = t[r + 1] > t[r] && (t[r + 1] - t[r]) % 8 == 0;
        if (!ok) return fail(h, AZB_ERR_INVALID, "blob %u: tree offset table", i);
    }
    // the running best: first minimum by (eval, global root, node) over every blob
    uint32_t best = 0;
    for (uint32_t i = 1; i < n_blobs; ++i) {
        const uint64_t *a = bl[i].hw, *c = bl[best].hw;
        if (std::make_tuple(a[CK_BEST_C], a[CK_BEST_ROOT], a[CK_BEST_NODE]) < std::make_tuple(c[CK_BEST_C], c[CK_BEST_ROOT], c[CK_BEST_NODE])) best = i;
    }

    // ---- device: from here on a failure leaves the trees invalid
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaStreamSynchronize(h->stream));
    ckpt_invalidate(h);
    uint64_t half = 0;
    for (uint32_t i = 0; i < n_blobs; ++i)
        if (!tables[i].empty()) {
            const uint64_t lo = std::max(F, bl[i].first) - bl[i].first, hi = std::min(F + B, bl[i].first + bl[i].n) - bl[i].first;
            half = std::max(half, ckpt_half_bytes(h, tables[i].data() + lo, (uint32_t)(hi - lo)));
        }
    CkptSlab s;
    int rc = ckpt_slab(h, half, s);
    if (rc) return rc;
    static const unsigned long long none2[2] = {~0ull, ~0ull};
    CK(cudaMemcpyAsync(s.bad, none2, 16, cudaMemcpyHostToDevice, h->stream));
    cudaEvent_t *copied = h->ckpt_ev, *used = h->ckpt_ev + 2;
    for (uint32_t i = 0; i < n_blobs; ++i) {
        if (tables[i].empty()) continue;
        const CkptBlob &b = bl[i];
        const uint64_t lo = std::max(F, b.first) - b.first, hi = std::min(F + B, b.first + b.n) - b.first;
        const uint32_t cnt = (uint32_t)(hi - lo), local0 = (uint32_t)(b.first + lo - F);
        const uint64_t *t = tables[i].data() + lo;
        CK(cudaMemcpyAsync(s.off, t, ((size_t)cnt + 1) * 8, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemsetAsync(s.len, 0, ((size_t)cnt + 1) * 8, h->stream));  // the digest sums
        const uint8_t *src = b.p + b.hw[CK_TREES_OFF];
        const auto chunks = ckpt_chunks(t, cnt, half);
        // chunk c goes to half c & 1 on the copy stream while chunk c - 1 is unpacked
        auto copy = [&](size_t c) -> int {
            if (c >= 2) CK(cudaStreamWaitEvent(h->ckpt_stream, used[c & 1], 0));
            const uint32_t c0 = chunks[c].first, c1 = chunks[c].second;
            CK(cudaMemcpyAsync(s.half[c & 1], src + t[c0], t[c1] - t[c0], cudaMemcpyHostToDevice, h->ckpt_stream));
            CK(cudaEventRecord(copied[c & 1], h->ckpt_stream));
            return AZB_OK;
        };
        rc = copy(0);
        if (rc) return rc;
        for (size_t c = 0; c < chunks.size(); ++c) {
            const uint32_t c0 = chunks[c].first, c1 = chunks[c].second;
            CK(cudaStreamWaitEvent(h->stream, copied[c & 1], 0));
            const uint32_t *stage = reinterpret_cast<const uint32_t *>(s.half[c & 1]);
            azb_ckpt_unpack_kernel<<<dim3(c1 - c0, ckpt_slices(t, c0, c1)), AZB_CKPT_THREADS, 0, h->stream>>>(h->L, s.off, c0, t[c0], stage, local0,
                                                                                                       b.first + lo, s.len, s.bad);
            azb_ckpt_unpack_finish_kernel<<<(c1 - c0 + 255) / 256, 256, 0, h->stream>>>(h->L, s.off, c0, c1, t[c0], stage, b.first + lo, s.len,
                                                                                        s.bad);
            h->launches += 2;
            CK(cudaGetLastError());
            CK(cudaEventRecord(used[c & 1], h->stream));
            if (c + 1 < chunks.size()) {
                rc = copy(c + 1);
                if (rc) return rc;
            }
        }
        CK(cudaStreamSynchronize(h->ckpt_stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    unsigned long long bad[2];
    auto read_bad = [&]() -> int {
        CK(cudaMemcpyAsync(bad, s.bad, 16, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        if (bad[0] == ~0ull && bad[1] == ~0ull) return AZB_OK;
        if (bad[0] <= bad[1]) return fail(h, AZB_ERR_INVALID, "the record of global root %llu is corrupt (digest or length)", bad[0]);
        return fail(h, AZB_ERR_CAPACITY, "the record of global root %llu does not fit the handle's capacities (cap_nodes, cap_preds, cap_parents)",
                    bad[1]);
    };
    rc = read_bad();
    if (rc) return rc;
    if (azb_stack_depth(h->N) == 5)
        azb_ckpt_hash_kernel<true><<<(h->L.B + AZB_CKPT_WARPS - 1) / AZB_CKPT_WARPS, AZB_CKPT_WARPS * 32, 0, h->stream>>>(h->L, s.bad);
    else
        azb_ckpt_hash_kernel<false><<<(h->L.B + AZB_CKPT_WARPS - 1) / AZB_CKPT_WARPS, AZB_CKPT_WARPS * 32, 0, h->stream>>>(h->L, s.bad);
    h->launches += 1;
    CK(cudaGetLastError());
    rc = read_bad();
    if (rc) return rc;

    // model and Adam state
    const uint64_t *w = b0.hw;
    const size_t n = h->n_params;
    const uint8_t *model = b0.p + k_ckpt_hdr_bytes;
    if (w[CK_FLAGS] & 1u) {
        CK(cudaMemcpyAsync(h->params, model, n * 4, cudaMemcpyHostToDevice, h->stream));
        if (h->tc.ready) {
            const char *why = azb_mlp_tc_load(h->tc, h->params, h->stream, &h->launches);
            if (why) return fail(h, AZB_ERR_CUDA, "tensor-core MLP: %s", why);
        }
    }
    if (w[CK_ADAM_T] || h->adam_m) {
        rc = train_alloc(h);
        if (rc) return rc;
        CK(cudaMemcpyAsync(h->adam_m, model + n * 4, n * 4, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->adam_v, model + n * 8, n * 4, cudaMemcpyHostToDevice, h->stream));
    }
    // globals: the running best, the next candidate slot, no error, counters from zero
    AzbGlobals g;
    CK(cudaMemcpyAsync(&g, h->L.g, sizeof(g), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const uint64_t *bw = bl[best].hw;
    const uint32_t steps = (uint32_t)w[CK_STEPS];
    g.best_c = (uint32_t)bw[CK_BEST_C];
    const bool mine = bw[CK_BEST_ROOT] >= F && bw[CK_BEST_ROOT] < F + B;
    g.argmin_tree = mine ? (uint32_t)(bw[CK_BEST_ROOT] - F) : AZB_NONE;
    g.argmin_node = mine ? (uint32_t)bw[CK_BEST_NODE] : AZB_NONE;
    h->ckpt_best_root = bw[CK_BEST_ROOT];
    h->ckpt_best_node = (uint32_t)bw[CK_BEST_NODE];
    memcpy(g.argmin_state, bw + CK_BEST_STATE, sizeof(g.argmin_state));
    g.n_improved = 0;
    g.err = g.err_tree = g.err_step = 0;
    g.improved_last = 0;
    g.behind_accum = g.n_behind = g.blocks_done = 0;
    g.next_slot = steps + 1;
    memset(&g.counters, 0, sizeof(g.counters));
    CK(cudaMemcpyAsync(h->L.g, &g, sizeof(g), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (w[CK_FLAGS] & 1u) h->params_set = true;
    h->adam_t = (uint32_t)w[CK_ADAM_T];
    float adam[5];
    for (int i = 0; i < 5; ++i) memcpy(adam + i, w + CK_ADAM + i, 4);
    h->adam = AzbAdam{adam[0], adam[1], adam[2], adam[3], adam[4], 1.f, 1.f};
    h->epoch = w[CK_EPOCH];
    h->steps_done = steps;
    h->argmin_from = h->poll_next = steps + 1;
    h->poll_best_valid = false;
    h->roots_set = true;
    h->first_init_done = h->trees_init = true;
    return AZB_OK;
}
