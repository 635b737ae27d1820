// keep_oracle.cc — the keyed specification with a keep mask (DESIGN.md §3.7), sequential, for the tests.
//
// TEST INFRASTRUCTURE ONLY. The keyed oracle (oracle/rlap_oracle.cc) is compiled into this translation unit unchanged,
// so that its Philox, rank permutation, star arithmetic and emission are reused as they are; only the driver is
// restated, with the mask. With keep = NULL it is oracle_keyed_schur line for line (tests/test_oracle_keep.py checks
// that the two agree bit for bit on every mode). Built by tests/keep_oracle.py:
//     g++ -O3 -std=c++17 -shared -fPIC -o libkeep_oracle.so tests/native/keep_oracle.cc
#include "../../oracle/rlap_oracle.cc"

extern "C" {

// oracle_keyed_schur plus keep (optional, n entries): a nonzero flag protects the vertex, it is never eliminated.
// For graph g with m_g unprotected vertices: t_g = min(max(num_remove, 0), m_g) if g has a protected vertex, else
// min(max(num_remove, 0), n_g - 1). o_v = random ranks the unprotected vertices, numbered by ascending id, with the
// keyed permutation over m_g; degree / coarsen take the minimum key, the bucket and the independent-set test over the
// alive unprotected vertices only.
int64_t oracle_keyed_schur_keep(int64_t n, const int64_t* ptr, const int32_t* col, const float* w, int64_t G,
                                const int64_t* graph_ptr, const int64_t* num_remove, int o_v, int o_n, uint64_t seed,
                                uint32_t view, int flags, int32_t* out_row, int32_t* out_col, float* out_w,
                                int64_t out_cap, int64_t* stats, int32_t* order_out, const uint8_t* keep) {
    using namespace keyed;
    auto prot = [&](int64_t v) { return keep && keep[v] != 0; };
    Graph g;
    g.n = n;
    g.adj.resize((size_t)n);
    g.elim.assign((size_t)n, 0);
    g.live.assign((size_t)n, 0);
    g.deg0.assign((size_t)n, 0);
    for (int64_t v = 0; v < n; v++) {
        for (int64_t p = ptr[v]; p < ptr[v + 1]; p++) g.adj[(size_t)v].push_back(Entry{col[p], w[p]});
        g.deg0[(size_t)v] = g.live[(size_t)v] = (int32_t)(ptr[v + 1] - ptr[v]);
    }
    Philox ph{(uint32_t)seed, (uint32_t)(seed >> 32)};
    Stats st;
    if (order_out) for (int64_t v = 0; v < n; v++) order_out[v] = -1;
    for (int64_t gi = 0; gi < G; gi++) {
        int64_t b = graph_ptr[gi], e = graph_ptr[gi + 1], ng = e - b;
        // the unprotected vertices of the graph, ascending: c(v) = position in this list
        std::vector<int32_t> unprot;
        for (int64_t v = b; v < e; v++)
            if (!prot(v)) unprot.push_back((int32_t)v);
        const int64_t mg = (int64_t)unprot.size();
        // without a protected vertex one vertex always survives (the reference's cap); with one, every other may go
        int64_t t = std::min<int64_t>(std::max<int64_t>(num_remove[gi], 0), mg < ng ? mg : std::max<int64_t>(ng - 1, 0));
        if (o_v == OV_RANDOM) {
            RankPerm rp(ph, (uint32_t)gi, (flags & FLAG_SHARED_ORDER) ? 0u : view, (uint32_t)mg);
            std::vector<int32_t> by_rank((size_t)mg);
            for (int64_t c = 0; c < mg; c++) by_rank[(size_t)rp.rank((uint32_t)c)] = unprot[(size_t)c];
            for (int64_t k = 0; k < t; k++) {
                eliminate(g, by_rank[(size_t)k], o_v, o_n, flags, ph, view, st);
                if (order_out) order_out[by_rank[(size_t)k]] = (int32_t)k;
            }
            st.rounds = std::max(st.rounds, t);
        } else {
            auto open = [&](int64_t v) { return !g.elim[(size_t)v] && !prot(v); };
            int64_t rem = t, round = 0;
            while (rem > 0) {
                int32_t m = 0x7fffffff;
                for (int64_t v = b; v < e; v++)
                    if (open(v)) m = std::min(m, key_of(g, (int32_t)v));
                std::vector<int32_t> I;
                for (int64_t v = e - 1; v >= b; v--) {   // descending id = ascending tie-break
                    if (!open(v) || key_of(g, (int32_t)v) != m) continue;
                    bool ok = true;
                    for (const Entry& en : g.adj[(size_t)v])
                        if (open(en.nbr) && en.nbr > v && key_of(g, en.nbr) == m) { ok = false; break; }
                    if (ok) I.push_back((int32_t)v);
                }
                if ((int64_t)I.size() > rem) I.resize((size_t)rem);  // keep the highest ids
                for (int32_t v : I) {
                    eliminate(g, v, o_v, o_n, flags, ph, view, st);
                    if (order_out) order_out[v] = (int32_t)round;
                }
                rem -= (int64_t)I.size();
                round++;
            }
            st.rounds = std::max(st.rounds, round);
        }
    }
    // emission (A.5), canonical order: by surviving vertex, neighbours ascending
    int64_t rows = 0;
    Star s;
    for (int64_t v = 0; v < n; v++) {
        if (g.elim[(size_t)v]) continue;
        gather_star(g, (int32_t)v, s);
        for (const Merged& mm : s.m) {
            if (rows < out_cap) { out_row[rows] = mm.nbr; out_col[rows] = (int32_t)v; out_w[rows] = mm.wf; }
            rows++;
        }
    }
    if (stats) { stats[0] = st.D; stats[1] = st.F; stats[2] = st.maxlen; stats[3] = st.rounds; stats[4] = st.Draw; }
    return rows;
}

}  // extern "C"
