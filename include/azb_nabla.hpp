// azb_nabla.hpp — C++ host-side mirror of the reference's optimizer surface for the c21 path, header-only, on top
// of the C ABI in azb.h.  The reference's host is Rust (nightly; no toolchain in this image), so the compiled host
// layer above the ABI is C++; INTEGRATION.md shows the Rust `extern "C"` binding a maintainer would add.
//
// Mirrors: NablaOptimizer (az-discrete-opt/src/nabla/optimizer/mod.rs:7-22,39-363), NablaModel
// (nabla/model/mod.rs:4-8), ArgminData (log.rs:1-11), ArgminImprovement (optimizer/mod.rs:24-27).
// Error behaviour: the reference panics (process abort); here every violation throws azb::Error.
#pragma once
#include <cmath>
#include <cstdint>
#include <functional>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#include "azb.h"

namespace azb {

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string &m) : std::runtime_error(m), code(c) {}
};

struct ArgminData {  // log.rs:1-11
    std::vector<uint8_t> parents;
    std::vector<uint32_t> permitted;
    double lambda_1 = 0;
    uint32_t mu = 0;
    float eval = 0;
};

// one isomorphism class of best_trees: the representative's ArgminData, the canonical code (azb.h), its tree and node
struct BestTree {
    ArgminData data;
    uint64_t code[2] = {0, 0};
    uint32_t tree = 0, node = 0;
};

// one entry of exhaustive_best: a free tree of the enumeration in azb.h, by its index
struct ExhaustiveTree {
    uint64_t index = 0;
    std::vector<uint8_t> parents;
    double lambda_1 = 0.0;
    uint32_t mu = 0;
    float eval = 0.0f;
};

// one entry of trees_within: an isomorphism class by its code, in its canonical labelling (azb.h)
struct TreeWithin {
    uint64_t code[2] = {0, 0};
    std::vector<uint8_t> parents;
    double lambda_1 = 0.0;
    uint32_t mu = 0;
    float eval = 0.0f;
};

// NablaModel (nabla/model/mod.rs:4-8) for models that live on the host
struct NablaModel {
    virtual ~NablaModel() = default;
    virtual void write_predictions(const std::vector<float> &states, std::vector<float> &predictions) = 0;
    // nabla/model/mod.rs:7: returns the loss
    virtual float update_model(const std::vector<float> & /*states*/, const std::vector<float> & /*observations*/,
                               const std::vector<float> & /*action_weights*/) { return 0.f; }
};
// nabla/model/mod.rs:10-23
struct TrivialModel : NablaModel {
    void write_predictions(const std::vector<float> &, std::vector<float> &) override {}
};

// PUCT selection (azb.h AZB_SELECT_PUCT) on a config before par_new; the reference's next_action stays the default
inline azb_config &with_puct(azb_config &cfg, float c_puct = 1.0f) {
    cfg.selection = AZB_SELECT_PUCT;
    cfg.puct_c = c_puct;
    return cfg;
}

class NablaOptimizer {
   public:
    // par_new (optimizer/mod.rs:39-118).  model == nullptr selects the built-in device MLP (ActionModel,
    // nabla/model/dfdx.rs:18-53) initialised from mlp_seed.
    static NablaOptimizer par_new(const azb_config &cfg, const std::vector<uint8_t> &root_parents,
                                  const std::vector<uint32_t> &root_permitted, NablaModel *model, uint64_t mlp_seed = 0) {
        NablaOptimizer o;
        o.cfg_ = cfg;
        o.model_ = model;
        o.cfg_.prior_mode = model ? AZB_PRIOR_INJECTED : AZB_PRIOR_MLP;
        o.ck(azb_create(&o.cfg_, &o.h_));
        o.ck(azb_get_config(o.h_, &o.cfg_));
        const uint32_t n = o.cfg_.n_vertices;
        o.a_ = (n - 1) * (n - 2) / 2 - 1;
        o.w_ = (o.a_ + 31) / 32;
        o.state_vecs_.assign((size_t)o.cfg_.n_roots * 2 * o.a_, 0.f);
        o.h_theta_.assign((size_t)o.cfg_.n_roots * o.a_, 0.f);
        if (!model) o.ck(azb_mlp_init(o.h_, mlp_seed));
        o.reseed(root_parents, root_permitted);
        return o;
    }
    // a new optimizer over cfg's roots continuing from checkpoint blobs (azb_checkpoint_load: one per rank of the saving
    // run, any number of ranks); the built-in device model only
    static NablaOptimizer resume(const azb_config &cfg, const std::vector<std::vector<uint8_t>> &blobs) {
        NablaOptimizer o;
        o.cfg_ = cfg;
        o.cfg_.prior_mode = AZB_PRIOR_MLP;
        o.ck(azb_create(&o.cfg_, &o.h_));
        o.ck(azb_get_config(o.h_, &o.cfg_));
        const uint32_t n = o.cfg_.n_vertices;
        o.a_ = (n - 1) * (n - 2) / 2 - 1;
        o.w_ = (o.a_ + 31) / 32;
        std::vector<const void *> ptrs;
        std::vector<uint64_t> sizes;
        for (const auto &b : blobs) {
            ptrs.push_back(b.data());
            sizes.push_back(b.size());
        }
        o.ck(azb_checkpoint_load(o.h_, ptrs.data(), sizes.data(), (uint32_t)blobs.size()));
        return o;
    }
    // the search and training state as a blob (azb_checkpoint_save; format in azb.h)
    std::vector<uint8_t> save_checkpoint() {
        uint64_t size = 0, written = 0;
        ck(azb_checkpoint_size(h_, &size));
        std::vector<uint8_t> blob(size);
        ck(azb_checkpoint_save(h_, blob.data(), size, &written));
        blob.resize(written);
        return blob;
    }
    NablaOptimizer(NablaOptimizer &&o) noexcept { *this = std::move(o); }
    NablaOptimizer &operator=(NablaOptimizer &&o) noexcept {
        std::swap(h_, o.h_);
        cfg_ = o.cfg_;
        model_ = o.model_;
        a_ = o.a_;
        w_ = o.w_;
        state_vecs_.swap(o.state_vecs_);
        h_theta_.swap(o.h_theta_);
        return *this;
    }
    ~NablaOptimizer() {
        if (h_) azb_destroy(h_);
    }

    // par_roll_out_episodes (optimizer/mod.rs:121-191): one batched step; the value is ArgminImprovement::Improved
    std::optional<ArgminData> par_roll_out_episodes() {
        bool improved = false;
        if (!model_) {
            uint32_t n = 0;
            ck(azb_step(h_, 1, nullptr, 0, &n));
            improved = n > 0;
        } else {
            ck(azb_rollout_host(h_, state_vecs_.data()));
            model_->write_predictions(state_vecs_, h_theta_);
            int imp = 0;
            ck(azb_add_actions_host(h_, h_theta_.data(), &imp));
            improved = imp != 0;
        }
        if (!improved) return std::nullopt;
        return argmin_data();
    }
    // the example's inner loop `for episode in 1..=episodes` (04-c21-tree.rs:142-150), fused on the device
    std::vector<azb_improvement> roll_out(uint32_t n_steps) {
        std::vector<azb_improvement> log(n_steps ? n_steps : 1);
        uint32_t n = 0;
        ck(azb_step(h_, n_steps, log.data(), (uint32_t)log.size(), &n));
        log.resize(n < log.size() ? n : log.size());
        return log;
    }
    // The example's per-step loop (04-c21-tree.rs:140-150) with the trees running ahead of the caller: on_step(step,
    // improved, record) for each of the n_steps as soon as every tree has finished that step, then the batch is
    // completed, so argmin_data() afterwards is what n_steps calls of par_roll_out_episodes would have left.
    template <class F>
    void roll_out_ahead(uint32_t n_steps, F &&on_step) {
        ck(azb_step_enqueue(h_, n_steps));
        for (uint32_t s = 0; s < n_steps; ++s) {
            azb_improvement rec{};
            int improved = 0;
            ck(azb_step_poll(h_, &rec, &improved));
            on_step(rec.step, improved != 0, rec);
        }
        uint32_t n = 0;
        ck(azb_step(h_, 0, nullptr, 0, &n));
    }
    ArgminData argmin_data() {  // optimizer/mod.rs:361-363
        ArgminData d;
        d.parents.resize(cfg_.n_vertices);
        d.permitted.resize(w_);
        ck(azb_get_argmin(h_, d.parents.data(), d.permitted.data(), &d.lambda_1, &d.mu, &d.eval));
        return d;
    }
    // the k best isomorphism classes among every node of the trees (azb_best_trees), ascending by (eval, code); call it
    // before par_reset_trees, which discards the trees
    std::vector<BestTree> best_trees(uint32_t k) {
        const size_t kk = k ? k : 1, n_v = cfg_.n_vertices;
        std::vector<float> eval(kk);
        std::vector<uint64_t> codes(2 * kk);
        std::vector<uint32_t> tree(kk), node(kk), mask(kk * w_), mu(kk);
        std::vector<uint8_t> parents(kk * n_v);
        std::vector<double> l1(kk);
        uint32_t n = 0;
        ck(azb_best_trees(h_, k, &n, eval.data(), codes.data(), tree.data(), node.data(), parents.data(), mask.data(), l1.data(),
                          mu.data()));
        std::vector<BestTree> out(n);
        for (uint32_t i = 0; i < n; ++i) {
            BestTree &b = out[i];
            b.data.parents.assign(parents.begin() + i * n_v, parents.begin() + (i + 1) * n_v);
            b.data.permitted.assign(mask.begin() + (size_t)i * w_, mask.begin() + (size_t)(i + 1) * w_);
            b.data.lambda_1 = l1[i];
            b.data.mu = mu[i];
            b.data.eval = eval[i];
            b.code[0] = codes[2 * i];
            b.code[1] = codes[2 * i + 1];
            b.tree = tree[i];
            b.node = node[i];
        }
        return out;
    }
    // the exact k best free trees of enumeration indices [start, start + count) by mu + lambda_1, ties by index
    // (azb_exhaustive_best, N <= 32; count 0 = to the end of the enumeration); bound as in azb.h (< 0: sqrt(N - 1) + 1)
    std::vector<ExhaustiveTree> exhaustive_best(uint64_t start = 0, uint64_t count = 0, uint32_t k = 100, double bound = -1.0,
                                                uint64_t *n_below = nullptr) {
        const size_t n_v = cfg_.n_vertices;
        if (count == 0) {
            uint64_t total = 0;
            if (azb_free_tree_count(cfg_.n_vertices, &total) == AZB_OK && total > start) count = total - start;
        }
        if (bound < 0.0) bound = std::sqrt((double)(n_v - 1)) + 1.0;
        const size_t kk = k ? k : 1;
        std::vector<uint64_t> index(kk);
        std::vector<uint8_t> parents(kk * n_v);
        std::vector<double> l1(kk);
        std::vector<uint32_t> mu(kk);
        std::vector<float> eval(kk);
        uint32_t n = 0;
        ck(azb_exhaustive_best(h_, start, count, k, bound, &n, n_below, index.data(), parents.data(), l1.data(), mu.data(),
                               eval.data(), nullptr));
        std::vector<ExhaustiveTree> out(n);
        for (uint32_t i = 0; i < n; ++i) {
            out[i].index = index[i];
            out[i].parents.assign(parents.begin() + i * n_v, parents.begin() + (i + 1) * n_v);
            out[i].lambda_1 = l1[i];
            out[i].mu = mu[i];
            out[i].eval = eval[i];
        }
        return out;
    }
    // every class on N vertices with mu + lambda_1 <= bound (< 0: the star's key), the first k by (key, code)
    // (azb_trees_within); max_level caps the classes of a level (0: what fits in device memory)
    std::vector<TreeWithin> trees_within(double bound = -1.0, uint32_t k = 100, uint64_t max_level = 0, uint64_t *n_within = nullptr,
                                         uint64_t *n_below = nullptr) {
        return trees_within_with(azb_trees_within, bound, k, max_level, n_within, n_below);
    }
    // trees_within split over the ranks of the attached communicator (azb_comm_trees_within): collective, every rank calls
    // it with the same arguments and gets the same result, bit for bit trees_within's on one handle
    std::vector<TreeWithin> comm_trees_within(double bound = -1.0, uint32_t k = 100, uint64_t max_level = 0,
                                              uint64_t *n_within = nullptr, uint64_t *n_below = nullptr) {
        return trees_within_with(azb_comm_trees_within, bound, k, max_level, n_within, n_below);
    }
    // trees_within with its certificate (azb_trees_within_proof): proof[5] = result classes proven below, equal, above the
    // bound (< 0: sqrt(N - 1) + 1 exactly), open, and dropped classes not proven above it; the rest as trees_within
    std::vector<TreeWithin> trees_within_proof(uint64_t proof[5], double bound = -1.0, uint32_t k = 100, uint64_t max_level = 0,
                                               uint64_t *n_within = nullptr, uint64_t *n_below = nullptr) {
        return trees_within_with(
            [proof](azb_handle *h, double b, uint32_t kk, uint64_t ml, uint32_t *n, uint64_t *nw, uint64_t *nb, uint64_t *c,
                    uint8_t *p, double *l1, uint32_t *mu, float *ev, float *ms) {
                return azb_trees_within_proof(h, b, kk, ml, n, nw, nb, c, p, l1, mu, ev, proof, ms);
            },
            bound, k, max_level, n_within, n_below);
    }
    // certificates of the keys of m trees (parents: m * N bytes) against bound (< 0: sqrt(N - 1) + 1 exactly)
    // (azb_certify_keys): verdict -1 / 0 / +1 = key below / equal to / above the bound, proven; 2 = open
    struct KeyCertificates {
        std::vector<double> lambda_1_lo, lambda_1_hi;
        std::vector<uint32_t> mu;
        std::vector<int8_t> verdict;
    };
    KeyCertificates certify_keys(const std::vector<uint8_t> &parents, double bound = -1.0) {
        const uint32_t m = (uint32_t)(parents.size() / cfg_.n_vertices);
        KeyCertificates out;
        out.lambda_1_lo.resize(m);
        out.lambda_1_hi.resize(m);
        out.mu.resize(m);
        out.verdict.resize(m);
        ck(azb_certify_keys(h_, parents.data(), m, bound, out.lambda_1_lo.data(), out.lambda_1_hi.data(), out.mu.data(),
                            out.verdict.data(), nullptr));
        return out;
    }
    template <class Fn>
    std::vector<TreeWithin> trees_within_with(Fn fn, double bound, uint32_t k, uint64_t max_level, uint64_t *n_within,
                                              uint64_t *n_below) {
        const size_t n_v = cfg_.n_vertices, kk = k ? k : 1;
        std::vector<uint64_t> codes(kk * 2);
        std::vector<uint8_t> parents(kk * n_v);
        std::vector<double> l1(kk);
        std::vector<uint32_t> mu(kk);
        std::vector<float> eval(kk);
        uint32_t n = 0;
        ck(fn(h_, bound, k, max_level, &n, n_within, n_below, codes.data(), parents.data(), l1.data(), mu.data(), eval.data(),
              nullptr));
        std::vector<TreeWithin> out(n);
        for (uint32_t i = 0; i < n; ++i) {
            out[i].code[0] = codes[2 * i];
            out[i].code[1] = codes[2 * i + 1];
            out[i].parents.assign(parents.begin() + i * n_v, parents.begin() + (i + 1) * n_v);
            out[i].lambda_1 = l1[i];
            out[i].mu = mu[i];
            out[i].eval = eval[i];
        }
        return out;
    }
    // the inputs par_update_model hands to NablaModel::update_model (optimizer/mod.rs:253-280)
    void observations(uint32_t n_obs_tol, std::vector<float> &state_vecs, std::vector<float> &obs, std::vector<float> &w) {
        state_vecs.resize((size_t)cfg_.n_roots * 2 * a_);
        obs.resize((size_t)cfg_.n_roots * a_);
        w.resize(obs.size());
        ck(azb_write_observations(h_, n_obs_tol, state_vecs.data(), obs.data(), w.data()));
    }
    // par_update_model (optimizer/mod.rs:249-281) with the built-in ActionModel: root vectors, observations, f32
    // forward/backward and the Adam step on the device (all-reduced if a communicator is attached); returns the loss
    float par_update_model(uint32_t n_obs_tol) {
        float loss = 0.f;
        if (!model_) {
            ck(azb_update_model(h_, n_obs_tol, &loss));
        } else {
            std::vector<float> sv, obs, w;
            observations(n_obs_tol, sv, obs, w);
            loss = model_->update_model(sv, obs, w);
        }
        return loss;
    }
    // par_reset_trees (optimizer/mod.rs:284-360) with the example's modify_root policy (04-c21-tree.rs:172-206) on the
    // device; k_min/k_max = num_permitted_actions_range (0,0 = 5..=ACTION/2)
    void par_reset_trees(uint64_t seed, uint32_t k_min = 0, uint32_t k_max = 0) { ck(azb_reset_trees(h_, seed, k_min, k_max)); }
    // par_reset_trees (optimizer/mod.rs:284-360) with the caller's modify_root already applied to the roots
    void par_reset_trees(const std::vector<uint8_t> &root_parents, const std::vector<uint32_t> &root_permitted) {
        reseed(root_parents, root_permitted);
    }
    azb_handle *handle() { return h_; }
    const azb_config &config() const { return cfg_; }
    uint32_t action_dim() const { return a_; }

   private:
    NablaOptimizer() = default;
    void reseed(const std::vector<uint8_t> &p, const std::vector<uint32_t> &m) {
        if (p.size() != (size_t)cfg_.n_roots * cfg_.n_vertices || m.size() != (size_t)cfg_.n_roots * w_)
            throw Error(AZB_ERR_INVALID, "root array sizes");
        ck(azb_set_roots(h_, p.data(), m.data()));
        if (model_) {  // one model call on the root vectors (optimizer/mod.rs:65-72)
            const uint32_t n = cfg_.n_vertices;
            std::fill(state_vecs_.begin(), state_vecs_.end(), 0.f);
            for (uint32_t i = 0; i < cfg_.n_roots; ++i) {
                float *v = state_vecs_.data() + (size_t)i * 2 * a_;
                for (uint32_t c = 2; c + 1 < n; ++c) v[c * (c - 1) / 2 + p[(size_t)i * n + c] - 1] = 1.f;
                for (uint32_t a = 0; a < a_; ++a)
                    if ((m[(size_t)i * w_ + (a >> 5)] >> (a & 31)) & 1u) v[a_ + a] = 1.f;
            }
            std::fill(h_theta_.begin(), h_theta_.end(), 0.f);
            model_->write_predictions(state_vecs_, h_theta_);
            ck(azb_set_priors(h_, h_theta_.data()));
        }
        ck(azb_init_trees(h_));
    }
    void ck(int rc) {
        if (rc != AZB_OK)
            throw Error(rc, std::string(azb_strerror(rc)) + ": " + (h_ ? azb_last_error(h_) : ""));
    }
    azb_handle *h_ = nullptr;
    azb_config cfg_{};
    NablaModel *model_ = nullptr;
    uint32_t a_ = 0, w_ = 0;
    std::vector<float> state_vecs_, h_theta_;
};

// ---- SURVEY 8(f) row 3: ConnectedBitsetGraph<N, B> (simple_graph/connected_bitset_graph/mod.rs:18-21) over the
// reference's two bitset words (bitset/primitive.rs): B32 (N <= 32, the default) and B64 (N <= 64) ----
using B32 = uint32_t;
using B64 = uint64_t;
template <uint32_t N, typename B = B32>
struct ConnectedBitsetGraph {
    B neighborhoods[N];  // bit u of neighborhoods[v] <=> uv is an edge
};
struct Conjecture2Dot1Cost {  // mod.rs:340-344; only matching.len() is read anywhere, so the size is what is kept
    double lambda_1;
    uint32_t matching_number;
};
// conjecture_2_1_cost (:319-337) for a batch; `action_kinds` (may be null) receives action_kinds() (:134-154) per graph
// as N (N - 1) bits in AddOrDeleteEdge::action_index order (bitset_graph/space/action.rs:10-19), padded to u32 words
template <uint32_t N>
std::vector<Conjecture2Dot1Cost> conjecture_2_1_costs(NablaOptimizer &on, const std::vector<ConnectedBitsetGraph<N>> &graphs,
                                                      std::vector<uint32_t> *action_kinds = nullptr) {
    static_assert(N >= 2 && N <= 32, "B32 neighbourhoods");
    const uint32_t m = (uint32_t)graphs.size(), kw = (N * (N - 1) + 31) / 32;
    std::vector<double> l1(m);
    std::vector<uint32_t> mu(m);
    if (action_kinds) action_kinds->assign((size_t)m * kw, 0u);
    const int rc = m ? azb_eval_graph_costs(on.handle(), &graphs[0].neighborhoods[0], m, N, l1.data(), mu.data(),
                                            action_kinds ? action_kinds->data() : nullptr, nullptr)
                     : AZB_OK;
    if (rc != AZB_OK) throw Error(rc, std::string(azb_strerror(rc)) + ": " + azb_last_error(on.handle()));
    std::vector<Conjecture2Dot1Cost> out(m);
    for (uint32_t i = 0; i < m; ++i) out[i] = {l1[i], mu[i]};
    return out;
}
// the same for ConnectedBitsetGraph<N, B64>
template <uint32_t N>
std::vector<Conjecture2Dot1Cost> conjecture_2_1_costs(NablaOptimizer &on, const std::vector<ConnectedBitsetGraph<N, B64>> &graphs,
                                                      std::vector<uint32_t> *action_kinds = nullptr) {
    static_assert(N >= 2 && N <= 64, "B64 neighbourhoods");
    const uint32_t m = (uint32_t)graphs.size(), kw = (N * (N - 1) + 31) / 32;
    std::vector<double> l1(m);
    std::vector<uint32_t> mu(m);
    if (action_kinds) action_kinds->assign((size_t)m * kw, 0u);
    const int rc = m ? azb_eval_graph_costs64(on.handle(), &graphs[0].neighborhoods[0], m, N, l1.data(), mu.data(),
                                              action_kinds ? action_kinds->data() : nullptr, nullptr)
                     : AZB_OK;
    if (rc != AZB_OK) throw Error(rc, std::string(azb_strerror(rc)) + ": " + azb_last_error(on.handle()));
    std::vector<Conjecture2Dot1Cost> out(m);
    for (uint32_t i = 0; i < m; ++i) out[i] = {l1[i], mu[i]};
    return out;
}

}  // namespace azb
