// tests/graph64_oracle.cpp — TEST INFRASTRUCTURE: the oracle's restatement of ConnectedBitsetGraph's cost and action
// kinds (simple_graph/connected_bitset_graph/mod.rs) for B64 neighbourhoods (one u64 per vertex, N <= 64), the word
// type of ConnectedBitsetGraph<N, B64>.  The oracle's translation unit is compiled in unchanged (for colex_position,
// mask_set and the Jacobi eigensolver); its B32 functions are restated here over uint64_t, line for line, so
// tests/test_oracle_graph64.py can check this copy against them on zero-extended words.
#include "../oracle/azb_oracle.cpp"

namespace {

// connected_bitset_graph/mod.rs:45-71: breadth-first search from v in G - vu; a cut edge never reaches u
bool graph64_is_cut_edge(const uint64_t *nbr, uint32_t v, uint32_t u) {
    uint64_t new_vertices = nbr[v] ^ (1ull << u);  // :52-55 add_or_remove(u)
    uint64_t explored = 1ull << v;                 // :56-57
    while (new_vertices) {                         // :58
        if (new_vertices >> u & 1u) return false;  // :59-61
        explored |= new_vertices;                  // :62
        uint64_t recent = new_vertices;            // :63
        new_vertices = 0u;                         // :64
        for (uint64_t r = recent; r; r &= r - 1) new_vertices |= nbr[__builtin_ctzll(r)];  // :65-67
        new_vertices &= ~explored;                 // :68
    }
    return true;  // :70
}

// connected_bitset_graph/mod.rs:134-154 in the index space of AddOrDeleteEdge::action_index
// (bitset_graph/space/action.rs:10-19): bit colex(e) = Add(e) is available, bit C(N,2) + colex(e) = Delete(e) is
void graph64_action_kinds(uint32_t n, const uint64_t *nbr, uint32_t *kinds) {
    const uint32_t e2 = n * (n - 1) / 2;
    for (uint32_t w = 0; w < (2 * e2 + 31) / 32; ++w) kinds[w] = 0u;
    for (uint32_t v = 0; v < n; ++v)
        for (uint32_t u = 0; u < v; ++u) {  // :139-140
            const uint32_t pos = colex_position(v, u);
            if (nbr[v] >> u & 1u) {                                            // :141
                if (!graph64_is_cut_edge(nbr, v, u)) mask_set(kinds, e2 + pos);  // :143-147 (None for a cut edge)
            } else {
                mask_set(kinds, pos);  // :149
            }
        }
}

// connected_bitset_graph/mod.rs:226-317: depth-first branch and bound over (matched edges, unvisited vertices);
// only the size of the matching is ever read on this path, so the edge lists are kept as counts.  Its bound
// popcount(unvisited) / 2 is far above the matching number of sparse graphs: from 48 vertices on it can take seconds.
uint32_t graph64_matching_number(uint32_t n, const uint64_t *nbr) {
    if (n == 0) return 0;  // :235-237
    struct Search {
        uint32_t edges;
        uint64_t unvisited;
    };
    std::vector<Search> queue;  // a VecDeque used as a stack: push_back / pop_back (:242-246)
    queue.push_back({0u, n >= 64 ? ~0ull : (1ull << n) - 1u});  // :238-243
    uint32_t matching_number = 0;                              // :244
    while (!queue.empty()) {
        Search m = queue.back();
        queue.pop_back();
        uint64_t unvisited = m.unvisited;
        uint32_t max_future = (uint32_t)__builtin_popcountll(unvisited) / 2;  // :261
        if (m.edges + max_future <= matching_number) continue;                 // :262-264
        const uint32_t next_v = 63u - (uint32_t)__builtin_clzll(unvisited);    // :269 max_unchecked
        unvisited ^= 1ull << next_v;                                           // :274
        max_future = (uint32_t)__builtin_popcountll(unvisited) / 2;            // :275
        if (m.edges + max_future > matching_number) queue.push_back({m.edges, unvisited});  // :279-285
        for (uint64_t nb = unvisited & nbr[next_v]; nb; nb &= nb - 1) {        // :286-288 ascending
            const uint32_t next_u = (uint32_t)__builtin_ctzll(nb);
            const uint32_t new_edges = m.edges + 1;                            // :289-290
            const uint64_t new_unvisited = unvisited ^ (1ull << next_u);       // :291-296
            if (new_edges > matching_number) matching_number = new_edges;      // :297-300
            max_future = (uint32_t)__builtin_popcountll(new_unvisited) / 2;    // :302
            if (new_edges + max_future > matching_number) queue.push_back({new_edges, new_unvisited});  // :303-309
        }
    }
    return matching_number;
}

// connected_bitset_graph/mod.rs:200-216 + :324-333: the largest eigenvalue of A + 1e-4 I (cyclic Jacobi, as for B32)
double graph64_lambda1(uint32_t n, const uint64_t *nbr) {
    double a[MAXN][MAXN];
    for (uint32_t i = 0; i < n; ++i)
        for (uint32_t j = 0; j < n; ++j) a[i][j] = 0.0;
    for (uint32_t i = 0; i < n; ++i) a[i][i] = 0.0001;  // :205-209 "ZERO"
    for (uint32_t v = 0; v < n; ++v)
        for (uint64_t r = nbr[v]; r; r &= r - 1) a[v][__builtin_ctzll(r)] = 1.0;  // :210-214
    return jacobi_max_eigenvalue(n, a);
}

}  // namespace

extern "C" {

int orc_graph64_is_cut_edge(uint32_t n, const uint64_t *nbr, uint32_t v, uint32_t u) {
    (void)n;
    return graph64_is_cut_edge(nbr, v, u) ? 1 : 0;
}
void orc_graph64_action_kinds(uint32_t n, const uint64_t *nbr, uint32_t *kinds) { graph64_action_kinds(n, nbr, kinds); }
uint32_t orc_graph64_matching_number(uint32_t n, const uint64_t *nbr) { return graph64_matching_number(n, nbr); }
/* lambda_1 alone: for the graphs on which the branch and bound is too slow */
double orc_graph64_lambda1(uint32_t n, const uint64_t *nbr) { return graph64_lambda1(n, nbr); }
/* conjecture_2_1_cost (:319-337): returns 1 where the reference's `assert!(lambda_1 > 1.4)` would abort */
int orc_graph64_cost(uint32_t n, const uint64_t *nbr, double *lambda1, uint32_t *mu) {
    *lambda1 = graph64_lambda1(n, nbr);
    *mu = graph64_matching_number(n, nbr);
    return *lambda1 > 1.4 ? 0 : 1;
}

}  // extern "C"
