// tests/puct_oracle.cpp — TEST INFRASTRUCTURE: the CPU oracle (oracle/azb_oracle.cpp) with the PUCT selection mode of
// include/azb.h (AZB_SELECT_PUCT) in place of the reference's next_action.  The reference has no PUCT, so there is
// nothing upstream to restate: the rule is this project's own, restated here and, independently, in numpy by
// tests/pyref_puct.py.  The oracle's translation unit is compiled in unchanged; this file adds the PUCT choice and a
// copy of its walk (roll_out_episodes, tree/mod.rs:113-232) that calls it, and exports two entry points that work on
// a handle made by libazb_oracle.so (the same source and flags, so the same layout):
//   orc_puct_rollout    = orc_rollout with PUCT selection
//   orc_puct_steps_hash = orc_steps_hash with PUCT selection
// Both return the oracle's codes (1 lambda_1 < 1.4, 2 unreachable) plus 3 (N_s reached 2^24) and 4 (a NaN score).
#include "../oracle/azb_oracle.cpp"

namespace {

// PUCT in place of next_action (include/azb.h, AZB_SELECT_PUCT: the rule is defined there and has no reference).
// err (with Next::None): 3 = N_s reached 2^24, 4 = a NaN score, 2 = an active node without a candidate.
Next puct_next_action(const SearchTree &t, uint32_t pos, float c_puct, uint32_t &out, int &err, orc_counters &k) {
    const StateWeight &w = t.nodes[pos].w;
    if (!w.is_active()) return Next::None;
    ++k.n_sel;
    ++k.n_cur;
    const uint32_t cnt = w.hi - w.lo;
    k.n_cand += cnt;
    const float c_s = w.c;
    // 1. N_s = 1 + sum over all kids of (n_t + 1), exact
    uint64_t n_s = 1;
    for (uint32_t e = t.nodes[pos].next[0]; e != ORC_NONE; e = t.edges[e].next[0]) {
        ++k.d_sel;
        n_s += (uint64_t)t.nodes[t.edges[e].node[1]].w.n_t + 1u;
    }
    if (n_s >= (1u << 24)) {
        err = 3;
        return Next::None;
    }
    const float sq = std::sqrt((float)n_s);
    // 2. w_j = (1 - c_s) + g_j, +0 where negative
    const float omc = 1.0f - c_s;
    std::vector<float> wj(cnt);
    for (uint32_t j = 0; j < cnt; ++j) {
        float x = omc + t.predictions[w.lo + j].g_theta_sa;
        wj[j] = x < 0.0f ? 0.0f : x;
    }
    // 3. Z: xor-butterfly sum per 32-prediction chunk, chunk sums folded left to right
    float z = 0.0f;
    for (uint32_t base = 0; base < cnt; base += 32) {
        float x[32], y[32];
        for (uint32_t i = 0; i < 32; ++i) x[i] = base + i < cnt ? wj[base + i] : 0.0f;
        for (uint32_t m = 16; m >= 1; m >>= 1) {
            for (uint32_t i = 0; i < 32; ++i) y[i] = x[i] + x[i ^ m];
            std::copy(y, y + 32, x);
        }
        z = base == 0 ? x[0] : z + x[0];
    }
    // 4-6. first maximum of the score in ascending prediction order
    bool have = false;
    float best = 0.0f;
    uint32_t best_j = 0;
    for (uint32_t j = 0; j < cnt; ++j) {
        const ActionPrediction &p = t.predictions[w.lo + j];
        const float pj = z == 0.0f ? 1.0f / (float)cnt : wj[j] / z;
        float q = p.g_theta_sa;
        uint32_t n = 0;
        if (p.edge_id != ORC_NONE) {
            const StateWeight &cw = t.nodes[t.edges[p.edge_id].node[1]].w;
            if (!cw.is_active()) continue;
            n = cw.n_t + 1u;
            q = c_s - cw.c_t_star;
        }
        const float score = q + ((c_puct * pj) * sq) / (float)(1u + n);
        if (score != score) {
            err = 4;
            return Next::None;
        }
        if (!have || score > best) {
            have = true;
            best = score;
            best_j = w.lo + j;
        }
    }
    if (!have) {
        err = 2;
        return Next::None;
    }
    const ActionPrediction &p = t.predictions[best_j];
    if (p.edge_id != ORC_NONE) {
        out = p.edge_id;
        return Next::Visited;
    }
    out = best_j;
    return Next::Unvisited;
}

// tree/mod.rs:113-232 as in roll_out_episodes, with the PUCT choice
int roll_out_episodes_puct(SearchTree &t, const Space &space, float c_puct, const State &root, State &state, Cost &cost,
                           ActionSet &path, uint32_t &state_pos, orc_counters &k) {
    for (;;) {
        uint32_t out = 0;
        int err = 0;
        Next na = puct_next_action(t, state_pos, c_puct, out, err, k);
        if (err) return err;
        if (na == Next::Visited) {  // :139-159
            ++k.n_visit;
            uint32_t prediction_pos = t.edges[out].prediction_pos;
            uint32_t action_id = t.predictions[prediction_pos].a_id;
            path_insert(path, action_id);
            space_act(space.n, state, action_id);
            state_pos = t.edges[out].node[1];
        } else if (na == Next::Unvisited) {  // :160-218
            uint32_t prediction_pos = out;
            uint32_t action_id = t.predictions[prediction_pos].a_id;
            path_insert(path, action_id);
            ++k.n_probe;
            auto f = t.positions.find(path);
            if (f != t.positions.end()) {  // :172-179
                ++k.n_hit;
                ++k.n_arc;
                uint32_t arc = t.add_arc(state_pos, f->second, prediction_pos);
                cascade(t, arc, true, k);
                state = root;
                path.clear();
                state_pos = 0;
                ++k.n_reset;
            } else {  // :181-216
                space_act(space.n, state, action_id);
                bool bad = false;
                cost = space.cost(state, &bad);
                if (bad) return 1;
                float c_as = space.evaluate(cost);
                ++k.n_ins;
                uint32_t next_pos = t.add_node(path, StateWeight(c_as));
                ++k.n_arc;
                uint32_t arc = t.add_arc(state_pos, next_pos, prediction_pos);
                if (space_is_terminal(space.n, state)) {
                    ++k.n_term;
                    cascade(t, arc, false, k);
                    state = root;
                    path.clear();
                    state_pos = 0;
                    ++k.n_reset;
                } else {
                    state_pos = next_pos;
                    return 0;
                }
            }
        } else {  // :220-229
            if (path.empty()) return 0;
            return 2;
        }
    }
}

}  // namespace

extern "C" {

// orc_rollout (optimizer/mod.rs:159-174) with PUCT selection
int orc_puct_rollout(orc_optimizer *o, float c_puct, float *state_vecs) {
    if (!(std::isfinite(c_puct) && c_puct > 0.0f)) return 1;
    const Space &sp = o->space;
    std::fill(o->thread_err.begin(), o->thread_err.end(), 0);
    parallel_for(o->batch, o->n_threads, [&](uint32_t i, int t) {
        orc_counters &k = o->thread_counters[t];
        int rc = roll_out_episodes_puct(o->trees[i], sp, c_puct, o->roots[i], o->states[i], o->costs[i], o->paths[i],
                                        o->last_positions[i], k);
        if (rc) o->thread_err[t] = rc;
        if (!o->paths[i].empty()) {
            ++k.n_live;
            if (state_vecs) space_write_vec(sp.n, o->states[i], state_vecs + (size_t)i * 2 * sp.a_dim);
        } else {
            ++k.n_noop;
        }
    });
    for (int e : o->thread_err)
        if (e) return e;
    return 0;
}

// orc_steps_hash with PUCT selection
int orc_puct_steps_hash(orc_optimizer *o, float c_puct, uint64_t seed, uint64_t first_root, uint64_t step0,
                        uint32_t n_steps, uint32_t *improved_steps, uint32_t cap, uint32_t *n_improved) {
    const Space &sp = o->space;
    std::vector<float> priors((size_t)o->batch * sp.a_dim);
    uint32_t ni = 0;
    for (uint32_t s = 0; s < n_steps; ++s) {
        int rc = orc_puct_rollout(o, c_puct, nullptr);
        if (rc) return rc;
        parallel_for(o->batch, o->n_threads, [&](uint32_t i, int) {
            for (uint32_t a = 0; a < sp.a_dim; ++a)
                priors[(size_t)i * sp.a_dim + a] = hash_prior(seed, first_root + i, step0 + s, a);
        });
        int imp = 0;
        orc_add_actions(o, priors.data(), &imp);
        if (imp) {
            if (improved_steps && ni < cap) improved_steps[ni] = (uint32_t)(step0 + s);
            ++ni;
        }
    }
    if (n_improved) *n_improved = ni;
    return 0;
}

}  // extern "C"
