// oracle/rlap_oracle.cc — CPU restatement of the rLap randomized Schur-complement path.
//
// TEST INFRASTRUCTURE ONLY. Nothing under rlap_b200/ may include, link or call this file;
// it is the checker used by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg.
//
// Two restatements live here, both sequential and single threaded:
//
//  (1) "ref" mode  — oracle_ref_approximate_cholesky(): follows the reference line by line in
//      behaviour (index-based arrays instead of heap nodes) so that, given the same injected
//      seeds, it reproduces the UNMODIFIED reference (oracle/_ref) BIT FOR BIT for all 9
//      o_v x o_n combinations: rlap/csrc/reader.cc:42-61 (ingest), factorizers.cc:46-65
//      (strategy dispatch), preconditioner.cc:22-49,65-114 (flip indices, linked lists),
//      :125-246 (degree bucket queue), :248-345 (column gather / compress), :348-476 (degree),
//      :713-825 (random), :835-957 (coarsen). Parity PINNED by tests/test_oracle_pin.py against
//      oracle/_ref and the committed tests/golden/ vectors generated from it.
//
//  (2) "keyed" mode — oracle_keyed_schur(): the same algorithm re-specified so that it can be
//      executed in any dependency-respecting order (DESIGN.md §3): randomness is a pure
//      function of (seed, view, vertex, neighbour) through Philox4x32-10, neighbour order ties
//      stand where libstdc++'s std::sort leaves them (order_star), and all in-star arithmetic is done on 64-bit fixed-point weights so
//      sums are order independent. The CUDA path must match this mode bit for bit
//      (rows, columns AND fp32 weights). It shares the sampling rule (A.2: neighbour j gets one
//      fill edge to a later neighbour k drawn with probability proportional to weight, weight
//      w_j (S - C_j) / S), the coarsening rule (A.4) and the emission rule (A.5) with mode (1).
//      Statistical equivalence of (1) and (2) is tested in tests/test_oracle_keyed.py. An optional keep mask
//      (DESIGN.md §3.7) protects vertices from elimination; without one the driver is the unmasked specification.
//      Its bits are pinned by stored digests (tests/test_oracle_keyed_pin.py).
//
// Build: make -C oracle oracle   (g++ -O3 -std=c++17 -shared -fPIC)
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <cstdio>
#include <limits>
#include <random>
#include <string>
#include <vector>

// =====================================================================================
// (1) REF MODE
// =====================================================================================
namespace refmode {

struct RdStream {  // the injected stand-in for std::random_device (oracle/ref_seed_inject.h)
    uint64_t state;
    uint32_t next() {
        uint64_t z = (state += 0x9e3779b97f4a7c15ull);
        z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
        z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
        z = z ^ (z >> 31);
        return (uint32_t)(z >> 32);
    }
};

// Column-compressed adjacency after reader.cc:42-61: zero weights dropped, duplicates summed
// in order of appearance, rows ascending inside a column.
struct Csc {
    int64_t n;
    std::vector<int> outer, inner;
    std::vector<double> val;
};

static Csc ingest(const double* ei, int64_t E, int64_t n) {
    std::vector<int64_t> keep;
    keep.reserve((size_t)E);
    for (int64_t p = 0; p < E; p++)
        if (ei[p * 3 + 2] != 0) keep.push_back(p);
    // stable order by (col, row): sort indices with input position as the last key
    std::vector<int64_t> ord(keep);
    std::stable_sort(ord.begin(), ord.end(), [&](int64_t a, int64_t b) {
        int ca = (int)ei[a * 3 + 1], cb = (int)ei[b * 3 + 1];
        if (ca != cb) return ca < cb;
        return (int)ei[a * 3 + 0] < (int)ei[b * 3 + 0];
    });
    Csc A;
    A.n = n;
    A.outer.assign((size_t)n + 1, 0);
    int curc = -1, curr = -1;
    for (int64_t p : ord) {
        int r = (int)ei[p * 3 + 0], c = (int)ei[p * 3 + 1];
        double v = ei[p * 3 + 2];
        if (c == curc && r == curr) {
            A.val.back() += v;
        } else {
            A.inner.push_back(r);
            A.val.push_back(v);
            A.outer[(size_t)c + 1]++;
            curc = c; curr = r;
        }
    }
    for (int64_t i = 0; i < n; i++) A.outer[(size_t)i + 1] += A.outer[(size_t)i];
    return A;
}

// factorizers.cc:18-22: A.isApprox(A^T) with Eigen's default precision 1e-12
static bool is_symmetric(const Csc& A) {
    // transpose by counting sort
    size_t nnz = A.inner.size();
    std::vector<int> cnt((size_t)A.n + 1, 0);
    for (size_t p = 0; p < nnz; p++) cnt[(size_t)A.inner[p] + 1]++;
    for (int64_t i = 0; i < A.n; i++) cnt[(size_t)i + 1] += cnt[(size_t)i];
    std::vector<int> to(cnt), ti(nnz);
    std::vector<double> tv(nnz);
    std::vector<int> cur(cnt.begin(), cnt.end() - 1);
    for (int64_t c = 0; c < A.n; c++)
        for (int p = A.outer[(size_t)c]; p < A.outer[(size_t)c + 1]; p++) {
            int q = cur[(size_t)A.inner[(size_t)p]]++;
            ti[(size_t)q] = (int)c; tv[(size_t)q] = A.val[(size_t)p];
        }
    double d2 = 0, na = 0, nb = 0;
    for (size_t p = 0; p < nnz; p++) { na += A.val[p] * A.val[p]; nb += tv[p] * tv[p]; }
    for (int64_t c = 0; c < A.n; c++) {
        int p = A.outer[(size_t)c], pe = A.outer[(size_t)c + 1], q = to[(size_t)c], qe = to[(size_t)c + 1];
        while (p < pe || q < qe) {
            int ra = p < pe ? A.inner[(size_t)p] : 0x7fffffff, rb = q < qe ? ti[(size_t)q] : 0x7fffffff;
            double a = 0, b = 0;
            if (ra <= rb) a = A.val[(size_t)p++];
            if (rb <= ra) b = tv[(size_t)q++];
            d2 += (a - b) * (a - b);
        }
    }
    return d2 <= 1e-24 * std::min(na, nb);
}

// The linked-list sparse matrix of types.h:7-68 with element indices instead of pointers.
struct Lists {
    std::vector<double> row, val;     // types.h:14,17 (row ids are doubles in the reference)
    std::vector<int> next, reverse;   // next == self terminates a column
    std::vector<int> cols;            // head element per column
    std::vector<double> degs;
};

// preconditioner.cc:22-49 + 65-114
static Lists build_lists(const Csc& A) {
    Lists a;
    size_t nnz = A.inner.size();
    int64_t n = A.n;
    a.row.resize(nnz); a.val.resize(nnz); a.next.resize(nnz); a.reverse.resize(nnz);
    a.cols.resize((size_t)n);
    a.degs.resize((size_t)n);
    // flip index of slot (r,c) = slot of (c,r): position-wise pairing with the transpose pattern
    std::vector<int> cur(A.outer.begin(), A.outer.end() - 1);
    std::vector<int> flips(nnz);
    for (int64_t c = 0; c < n; c++)
        for (int p = A.outer[(size_t)c]; p < A.outer[(size_t)c + 1]; p++) {
            // walking columns in order visits, for every row r, its transposed slots in ascending c,
            // i.e. exactly the ascending-row order of column r
            int r = A.inner[(size_t)p];
            int q = cur[(size_t)r]++;
            flips[(size_t)q] = p;
        }
    for (int64_t i = 0; i < n; i++) {
        int s = A.outer[(size_t)i], e = A.outer[(size_t)i + 1];
        a.degs[(size_t)i] = e - s;
        if (e == s) {  // dummy self-looped element (:78-82)
            a.row.push_back(0); a.val.push_back(0);
            int id = (int)a.row.size() - 1;
            a.next.push_back(id); a.reverse.push_back(id);
            a.cols[(size_t)i] = id;
            continue;
        }
        for (int p = s; p < e; p++) {
            a.row[(size_t)p] = A.inner[(size_t)p];
            a.val[(size_t)p] = A.val[(size_t)p];
            a.next[(size_t)p] = (p == s) ? p : p - 1;  // head is the LAST entry of the column
        }
        a.cols[(size_t)i] = e - 1;
    }
    for (size_t p = 0; p < nnz; p++) a.reverse[p] = flips[p];
    return a;
}

// types.h:80-121 + preconditioner.cc:125-246
struct DegreePQ {
    std::vector<int64_t> prev, next, key;
    std::vector<char> present;
    std::vector<int64_t> lists;
    int64_t minlist, nitems, n;

    explicit DegreePQ(const std::vector<double>& degs) {
        n = (int64_t)degs.size();
        prev.assign((size_t)n, -1); next.assign((size_t)n, -1); key.assign((size_t)n, 0);
        present.assign((size_t)n, 1);
        lists.assign((size_t)(2 * n + 1), -1);
        minlist = 0;
        for (int64_t i = 0; i < n; i++) {
            int64_t k = (int64_t)degs[(size_t)i];
            int64_t head = lists[(size_t)k];
            prev[(size_t)i] = -1; next[(size_t)i] = head >= 0 ? head : -1; key[(size_t)i] = k;
            if (head >= 0) prev[(size_t)head] = i;
            lists[(size_t)k] = i;
        }
        nitems = n;
    }
    int64_t bucket(int64_t k) const { return k <= n ? k : n + k / n; }
    int64_t pop() {
        while (lists[(size_t)minlist] == -1) minlist++;
        int64_t i = lists[(size_t)minlist];
        int64_t nx = next[(size_t)i];
        lists[(size_t)minlist] = nx;
        present[(size_t)i] = 0;
        if (nx > -1) prev[(size_t)nx] = -1;
        nitems--;
        return i;
    }
    void move(int64_t i, int64_t newkey, int64_t oldlist, int64_t newlist) {
        int64_t p = prev[(size_t)i], nx = next[(size_t)i];
        if (nx > -1) prev[(size_t)nx] = p;
        if (p > -1) next[(size_t)p] = nx; else lists[(size_t)oldlist] = nx;
        int64_t head = lists[(size_t)newlist];
        if (head > -1) prev[(size_t)head] = i;
        lists[(size_t)newlist] = i;
        prev[(size_t)i] = -1; next[(size_t)i] = head; key[(size_t)i] = newkey;
    }
    void dec(int64_t i) {
        int64_t d = key[(size_t)i];
        if (d == 1) return;
        int64_t ol = bucket(d), nl = bucket(d - 1);
        if (ol != nl) { move(i, d - 1, ol, nl); if (nl < minlist) minlist = nl; }
        else key[(size_t)i] -= 1;
    }
    void inc(int64_t i) {
        int64_t d = key[(size_t)i];
        int64_t ol = bucket(d), nl = bucket(d + 1);
        if (ol != nl) move(i, d + 1, ol, nl); else key[(size_t)i] += 1;
    }
};

struct Ctx {
    Lists a;
    std::string o_n;
    RdStream rd;
    DegreePQ* pq = nullptr;           // null for the random order (no Dec on merged duplicates)
    std::vector<int> colspace;

    // preconditioner.cc:248-271
    int64_t column_length(int64_t i) {
        int ll = a.cols[(size_t)i];
        int64_t len = 0;
        auto take = [&](int e) {
            len++;
            if ((size_t)len > colspace.size()) colspace.push_back(e); else colspace[(size_t)len - 1] = e;
        };
        while (a.next[(size_t)ll] != ll) {
            if (a.val[(size_t)ll] > 0) take(ll);
            ll = a.next[(size_t)ll];
        }
        if (a.val[(size_t)ll] > 0) take(ll);
        return len;
    }
    // preconditioner.cc:273-310 (elimination) and :312-345 (emission, sc=true: no twin/PQ updates)
    int64_t compress(int64_t len, bool sc) {
        std::sort(colspace.begin(), colspace.begin() + len,
                  [&](int j, int k) { return a.row[(size_t)j] < a.row[(size_t)k]; });
        int64_t ptr = -1;
        double currow = -1;
        for (int64_t i = 0; i < len; i++) {
            int e = colspace[(size_t)i];
            if (a.row[(size_t)e] != currow) {
                currow = a.row[(size_t)e];
                ptr++;
                colspace[(size_t)ptr] = e;
            } else {
                a.val[(size_t)colspace[(size_t)ptr]] += a.val[(size_t)e];
                if (!sc) {
                    a.val[(size_t)a.reverse[(size_t)e]] = 0;
                    if (pq) pq->dec((int64_t)currow);
                }
            }
        }
        if (o_n == "asc") {
            std::sort(colspace.begin(), colspace.begin() + ptr + 1,
                      [&](int j, int k) { return a.val[(size_t)j] < a.val[(size_t)k]; });
        } else if (o_n == "desc") {
            std::sort(colspace.begin(), colspace.begin() + ptr + 1,
                      [&](int j, int k) { return a.val[(size_t)j] > a.val[(size_t)k]; });
        } else if (o_n == "random") {
            std::mt19937 gen(rd.next());
            std::shuffle(colspace.begin(), colspace.begin() + ptr + 1, gen);
        }
        return ptr + 1;
    }
    // relink the pair (ll, revj) as the fill edge (j,k) of weight w (preconditioner.cc:403-414)
    void relink(int ll, int revj, double j, double k, double w) {
        a.row[(size_t)revj] = k; a.val[(size_t)revj] = w; a.reverse[(size_t)revj] = ll;
        int khead = a.cols[(size_t)k];
        a.cols[(size_t)k] = ll;
        a.next[(size_t)ll] = khead;
        a.reverse[(size_t)ll] = revj;
        a.val[(size_t)ll] = w;
        a.row[(size_t)ll] = j;
    }
};

struct Counters { int64_t D = 0, F = 0, maxlen = 0; };

static void emit(Ctx& c, int64_t i, std::vector<double>& out) {
    int64_t len = c.column_length(i);
    len = c.compress(len, true);
    for (int64_t ii = 0; ii < len; ii++) {
        int e = c.colspace[(size_t)ii];
        out.push_back(c.a.row[(size_t)e]); out.push_back((double)i); out.push_back(c.a.val[(size_t)e]);
    }
}

// clique sampling shared by :364-432 (degree) and :727-784 (random)
static void sample_clique(Ctx& c, int64_t len, std::mt19937_64& gen, std::uniform_real_distribution<double>& ud) {
    std::vector<double> cum((size_t)len), vals((size_t)len);
    double csum = 0;
    for (int64_t ii = 0; ii < len; ii++) {
        vals[(size_t)ii] = c.a.val[(size_t)c.colspace[(size_t)ii]];
        csum += vals[(size_t)ii];
        cum[(size_t)ii] = csum;
    }
    double wdeg = csum, colScale = 1;
    for (int64_t jo = 0; jo < len - 1; jo++) {
        int ll = c.colspace[(size_t)jo];
        double w = vals[(size_t)jo] * colScale;
        double j = c.a.row[(size_t)ll];
        int revj = c.a.reverse[(size_t)ll];
        double f = w / wdeg;
        double u = ud(gen);
        double r = u * (csum - cum[(size_t)jo]) + cum[(size_t)jo];
        int64_t koff = len - 1;
        for (int64_t ki = 0; ki < len; ki++)
            if (cum[(size_t)ki] > r) { koff = ki; break; }
        double k = c.a.row[(size_t)c.colspace[(size_t)koff]];
        if (c.pq) c.pq->inc((int64_t)k);
        double nv = f * (1 - f) * wdeg;
        c.relink(ll, revj, j, k, nv);
        colScale = colScale * (1 - f);
        wdeg = wdeg * (1 - f) * (1 - f);
    }
}

static int64_t run(const double* ei, int64_t E, int64_t n, int64_t t, const std::string& o_v, const std::string& o_n_in,
                   uint64_t sample_seed, uint64_t rd_state, std::vector<double>& out, Counters& cnt, int* status) {
    Csc A = ingest(ei, E, n);
    *status = 0;
    if (!is_symmetric(A)) { *status = 1; return 0; }  // the reference prints and exit(0)s here
    Ctx c;
    c.a = build_lists(A);
    c.rd.state = rd_state;
    c.o_n = (o_v == "coarsen") ? std::string("random") : o_n_in;  // preconditioner.cc:831
    std::mt19937_64 gen(sample_seed);
    std::uniform_real_distribution<double> ud(0, 1);
    int64_t it = 1;
    if (o_v == "random") {
        // preconditioner.cc:588-613: shuffle 0..n-1, pop from the back
        std::vector<double> node_id((size_t)n);
        for (int64_t i = 0; i < n; i++) node_id[(size_t)i] = (double)i;
        {
            std::mt19937 g(c.rd.next());
            std::shuffle(node_id.begin(), node_id.end(), g);
        }
        int64_t nitems = n;
        while (it <= t && it < n) {
            int64_t i = (int64_t)node_id[(size_t)--nitems];
            int64_t len = c.column_length(i);
            cnt.D += len;
            len = c.compress(len, false);
            cnt.maxlen = std::max(cnt.maxlen, len);
            if (len > 0) cnt.F += len - 1;
            sample_clique(c, len, gen, ud);
            if (len > 0) {
                int ll = c.colspace[(size_t)len - 1];
                int revj = c.a.reverse[(size_t)ll];
                c.a.val[(size_t)ll] = 0; c.a.val[(size_t)revj] = 0;
            }
            it++;
        }
        while (nitems > 0) emit(c, (int64_t)node_id[(size_t)--nitems], out);
    } else {
        DegreePQ pq(c.a.degs);
        c.pq = &pq;
        bool coarsen = (o_v == "coarsen");
        while (it <= t && it < n) {
            int64_t i = pq.pop();
            it++;
            int64_t len = c.column_length(i);
            cnt.D += len;
            len = c.compress(len, false);
            cnt.maxlen = std::max(cnt.maxlen, len);
            if (!coarsen) {
                if (len > 0) cnt.F += len - 1;
                sample_clique(c, len, gen, ud);
                if (len > 0) {
                    int ll = c.colspace[(size_t)len - 1];
                    double j = c.a.row[(size_t)ll];
                    int revj = c.a.reverse[(size_t)ll];
                    if (it < n) pq.dec((int64_t)j);
                    c.a.val[(size_t)ll] = 0; c.a.val[(size_t)revj] = 0;
                }
            } else {
                // preconditioner.cc:851-913
                if (len < 1) continue;
                cnt.F += len - 1;
                std::vector<double> cum((size_t)len), vals((size_t)len);
                double csum = 0;
                for (int64_t ii = 0; ii < len; ii++) {
                    vals[(size_t)ii] = c.a.val[(size_t)c.colspace[(size_t)ii]];
                    csum += vals[(size_t)ii];
                    cum[(size_t)ii] = csum;
                }
                double r = ud(gen) * csum;
                int64_t koff = len - 1;
                for (int64_t ki = 0; ki < len; ki++)
                    if (cum[(size_t)ki] > r) { koff = ki; break; }
                int kpe = c.colspace[(size_t)koff];
                double k = c.a.row[(size_t)kpe];
                double wk = vals[(size_t)koff];
                c.a.val[(size_t)kpe] = 0;
                c.a.val[(size_t)c.a.reverse[(size_t)kpe]] = 0;
                pq.dec((int64_t)k);
                for (int64_t jo = 0; jo < len; jo++) {
                    if (jo == koff) continue;
                    int ll = c.colspace[(size_t)jo];
                    double w = vals[(size_t)jo];
                    double j = c.a.row[(size_t)ll];
                    int revj = c.a.reverse[(size_t)ll];
                    pq.inc((int64_t)k);
                    c.relink(ll, revj, j, k, (wk * w) / (wk + w));
                }
            }
        }
        while (pq.nitems > 0) emit(c, pq.pop(), out);
    }
    return (int64_t)out.size() / 3;
}

}  // namespace refmode

// =====================================================================================
// (2) KEYED MODE  (the specification the CUDA path implements; DESIGN.md §3)
// =====================================================================================
namespace keyed {

// Philox4x32-10 (Salmon et al., SC'11), written from the published round function.
struct Philox {
    uint32_t k0, k1;
    static inline void mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
        uint64_t p = (uint64_t)a * (uint64_t)b;
        hi = (uint32_t)(p >> 32); lo = (uint32_t)p;
    }
    void operator()(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t out[4]) const {
        uint32_t a = k0, b = k1;
        for (int r = 0; r < 10; r++) {
            uint32_t h0, l0, h1, l1;
            mulhilo(0xD2511F53u, c0, h0, l0);
            mulhilo(0xCD9E8D57u, c2, h1, l1);
            uint32_t n0 = h1 ^ c1 ^ a, n1 = l1, n2 = h0 ^ c3 ^ b, n3 = l0;
            c0 = n0; c1 = n1; c2 = n2; c3 = n3;
            a += 0x9E3779B9u; b += 0xBB67AE85u;
        }
        out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
    }
};
enum { TAG_ORDER = 1, TAG_STAR = 2, TAG_PICK = 3 };

static inline uint64_t mulhi64(uint64_t a, uint64_t b) { return (uint64_t)(((unsigned __int128)a * b) >> 64); }

// o_v = random: rank(v) = position of v in a keyed pseudo-random permutation of its graph's vertices
// (stands in for std::shuffle + pop, preconditioner.cc:588-613). 8-round balanced Feistel network over
// the smallest even-width power-of-two domain covering n_g, cycle-walked into [0, n_g); round keys come
// from Philox keyed on (seed; graph, view). The t vertices of lowest rank are eliminated in rank order.
static inline uint32_t fmix32(uint32_t h) {
    h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16;
    return h;
}
struct RankPerm {
    uint32_t rk[8];
    uint32_t hb, mask, ng;
    RankPerm(const Philox& ph, uint32_t graph, uint32_t view, uint32_t n_g) {
        uint32_t o[4];
        ph(graph, 0u, view, TAG_ORDER, o);
        for (int r = 0; r < 4; r++) rk[r] = o[r];
        ph(graph, 1u, view, TAG_ORDER, o);
        for (int r = 0; r < 4; r++) rk[4 + r] = o[r];
        uint32_t b = 2;
        while (b < 32 && ((uint64_t)1 << b) < (uint64_t)n_g) b += 2;
        hb = b / 2; mask = (hb >= 32) ? 0xffffffffu : ((1u << hb) - 1u); ng = n_g;
    }
    uint32_t perm(uint32_t x) const {
        uint32_t L = x >> hb, R = x & mask;
        for (int r = 0; r < 8; r++) {
            uint32_t t = fmix32(R * 0x9E3779B1u + rk[r]) & mask;
            uint32_t nr = L ^ t;
            L = R; R = nr;
        }
        return (L << hb) | R;
    }
    uint32_t rank(uint32_t local) const {
        uint32_t x = local;
        do { x = perm(x); } while (x >= ng);
        return x;
    }
};

enum { OV_RANDOM = 0, OV_DEGREE = 1, OV_COARSEN = 2 };
enum { ON_ASC = 0, ON_DESC = 1, ON_RANDOM = 2 };
enum { FLAG_FULL_CLIQUE = 1, FLAG_SHARED_ORDER = 2 };

struct Entry { int32_t nbr; float w; };

struct Graph {
    int64_t n;
    std::vector<std::vector<Entry>> adj;   // append-only multigraph; dead entries filtered by elim[]
    std::vector<char> elim;
    std::vector<int32_t> live;             // number of entries whose neighbour is not eliminated
    std::vector<int32_t> deg0;
};

struct Merged { int32_t nbr; uint64_t q; float wf; uint64_t shuf; uint64_t usample; };

struct Star {
    std::vector<Merged> m;
    int shift = 0;
    uint64_t S = 0;
    int64_t lraw = 0;
};

static inline int ceil_log2(int64_t x) { int h = 0; while (((int64_t)1 << h) < x) h++; return h; }

// Fixed-point image of a star: q = rint(w * 2^shift) with shift chosen from the largest weight
// and the raw entry count so that the sum of all q fits in 62 bits. Order independent.
static void gather_star(const Graph& g, int32_t i, Star& s) {
    s.m.clear();
    std::vector<Entry> raw;
    for (const Entry& e : g.adj[(size_t)i])
        if (!g.elim[(size_t)e.nbr]) raw.push_back(e);
    s.lraw = (int64_t)raw.size();
    s.S = 0;
    if (raw.empty()) return;
    float wmax = 0;
    for (const Entry& e : raw) wmax = std::max(wmax, e.w);
    int ex;
    std::frexp((double)wmax, &ex);                 // wmax = f * 2^ex, f in [0.5,1)
    s.shift = 62 - ceil_log2(s.lraw) - ex;
    std::stable_sort(raw.begin(), raw.end(), [](const Entry& a, const Entry& b) { return a.nbr < b.nbr; });
    size_t p = 0;
    while (p < raw.size()) {
        size_t e = p;
        uint64_t q = 0;
        while (e < raw.size() && raw[e].nbr == raw[p].nbr) {
            q += (uint64_t)std::llrint(std::ldexp((double)raw[e].w, s.shift));
            e++;
        }
        Merged mm;
        mm.nbr = raw[p].nbr;
        mm.q = q;
        mm.wf = (e - p == 1) ? raw[p].w : (float)std::ldexp((double)q, -s.shift);
        if (!(mm.wf > 0.0f)) mm.wf = std::numeric_limits<float>::denorm_min();   // a merged edge never vanishes on one side
        mm.shuf = 0; mm.usample = 0;
        s.m.push_back(mm);
        s.S += q;
        p = e;
    }
}

// o_n order of the merged neighbours. Ties (the rule, not the exception: every call site of the reference uses unit
// weights) stand exactly where the reference's std::sort leaves them: the column was sorted by row just before
// (preconditioner.cc:275-276), so the input is in neighbour-id order, and the very same call - libstdc++'s std::sort
// with the reference's comparator (preconditioner.cc:295-303), here on the fixed-point weights - is made on it. Up to
// 16 elements that is a stable insertion sort (ties keep the id order); above, the introsort partition loop scrambles
// equal elements in a deterministic way, which the CUDA path restates (rlap_b200/csrc/introsort.cuh, pinned against
// std::sort by tests/test_introsort.py).
static void order_star(Star& s, int o_n) {
    if (o_n == ON_ASC)
        std::sort(s.m.begin(), s.m.end(), [](const Merged& a, const Merged& b) { return a.q < b.q; });
    else if (o_n == ON_DESC)
        std::sort(s.m.begin(), s.m.end(), [](const Merged& a, const Merged& b) { return a.q > b.q; });
    else
        std::sort(s.m.begin(), s.m.end(), [](const Merged& a, const Merged& b) { return a.shuf != b.shuf ? a.shuf < b.shuf : a.nbr < b.nbr; });
}

struct Stats { int64_t D = 0, F = 0, maxlen = 0, rounds = 0, Draw = 0; };

static void add_edge(Graph& g, int32_t a, int32_t b, float w) {
    g.adj[(size_t)a].push_back(Entry{b, w});
    g.adj[(size_t)b].push_back(Entry{a, w});
    g.live[(size_t)a]++; g.live[(size_t)b]++;
}

// eliminate vertex i (A.2 / A.4 / full clique)
static void eliminate(Graph& g, int32_t i, int o_v, int o_n, int flags, const Philox& ph, uint32_t view, Stats& st) {
    Star s;
    gather_star(g, i, s);
    st.Draw += (int64_t)g.adj[(size_t)i].size();
    st.D += s.lraw;
    int64_t L = (int64_t)s.m.size();
    st.maxlen = std::max(st.maxlen, L);
    for (Merged& mm : s.m) {
        uint32_t o[4];
        ph((uint32_t)i, (uint32_t)mm.nbr, view, TAG_STAR, o);
        mm.usample = ((uint64_t)o[0] << 32) | o[1];
        mm.shuf = ((uint64_t)o[2] << 32) | o[3];
    }
    // every raw entry of i disappears from its neighbour's live count
    for (const Entry& e : g.adj[(size_t)i])
        if (!g.elim[(size_t)e.nbr]) g.live[(size_t)e.nbr]--;
    g.elim[(size_t)i] = 1;
    if (L == 0) return;
    if (flags & FLAG_FULL_CLIQUE) {
        // exact Schur complement of the star: w_ab = w_a w_b / S for every pair
        std::sort(s.m.begin(), s.m.end(), [](const Merged& a, const Merged& b) { return a.nbr < b.nbr; });
        double Sf = std::ldexp((double)s.S, -s.shift);
        for (int64_t a = 0; a < L; a++)
            for (int64_t b = a + 1; b < L; b++) {
                float w = (float)(((double)s.m[(size_t)a].wf * (double)s.m[(size_t)b].wf) / Sf);
                if (w > 0) { add_edge(g, s.m[(size_t)a].nbr, s.m[(size_t)b].nbr, w); st.F++; }
            }
        return;
    }
    if (o_v == OV_COARSEN) {
        order_star(s, ON_RANDOM);
        uint32_t o[4];
        ph((uint32_t)i, 0xffffffffu, view, TAG_PICK, o);
        uint64_t u = ((uint64_t)o[0] << 32) | o[1];
        uint64_t r = mulhi64(u, s.S), c = 0;
        int64_t koff = L - 1;
        for (int64_t k = 0; k < L; k++) { c += s.m[(size_t)k].q; if (c > r) { koff = k; break; } }
        const Merged mk = s.m[(size_t)koff];
        for (int64_t j = 0; j < L; j++) {
            if (j == koff) continue;
            const Merged& mj = s.m[(size_t)j];
            float w = (float)(((double)mk.wf * (double)mj.wf) / ((double)mk.wf + (double)mj.wf));
            if (w > 0) { add_edge(g, mj.nbr, mk.nbr, w); st.F++; }
        }
        return;
    }
    order_star(s, o_n);
    std::vector<uint64_t> C((size_t)L);
    uint64_t c = 0;
    for (int64_t k = 0; k < L; k++) { c += s.m[(size_t)k].q; C[(size_t)k] = c; }
    for (int64_t j = 0; j < L - 1; j++) {
        const Merged& mj = s.m[(size_t)j];
        uint64_t rem = s.S - C[(size_t)j];
        uint64_t r = C[(size_t)j] + mulhi64(mj.usample, rem);
        int64_t koff = (int64_t)(std::upper_bound(C.begin(), C.end(), r) - C.begin());
        if (koff >= L) koff = L - 1;
        double t1 = (double)mj.wf * (double)rem;
        float w = (float)(t1 / (double)s.S);
        if (w > 0) { add_edge(g, mj.nbr, s.m[(size_t)koff].nbr, w); st.F++; }
        else if (getenv("ORACLE_TRACE")) fprintf(stderr, "oracle: underflow at i=%d L=%lld lraw=%lld j=%d (pos %lld) k=%d wf=%g rem=%llu S=%llu\n", i, (long long)L, (long long)s.lraw, mj.nbr, (long long)j, s.m[(size_t)koff].nbr, (double)mj.wf, (unsigned long long)rem, (unsigned long long)s.S);
    }
}

static inline int32_t key_of(const Graph& g, int32_t v) {
    return g.deg0[(size_t)v] == 0 ? 0 : std::max(g.live[(size_t)v], 1);
}

}  // namespace keyed

// =====================================================================================
// C ABI (ctypes)
// =====================================================================================
extern "C" {

// ref mode. edge_info row-major [E,3] doubles. status: 0 ok, 1 asymmetric input (the reference exit(0)s).
int64_t oracle_ref_approximate_cholesky(const double* edge_info, int64_t E, int64_t n, int64_t t, const char* o_v,
                                        const char* o_n, uint64_t sample_seed, uint64_t rd_state, double** out,
                                        int64_t* counters /* D, F, maxlen */, int* status) {
    std::vector<double> o;
    refmode::Counters cnt;
    int st = 0;
    int64_t rows = refmode::run(edge_info, E, n, t, o_v, o_n, sample_seed, rd_state, o, cnt, &st);
    if (status) *status = st;
    if (counters) { counters[0] = cnt.D; counters[1] = cnt.F; counters[2] = cnt.maxlen; }
    double* buf = (double*)malloc(sizeof(double) * (o.size() + 3));
    if (!o.empty()) memcpy(buf, o.data(), sizeof(double) * o.size());
    *out = buf;
    return rows;
}

void oracle_free(void* p) { free(p); }

// Philox probe for the unit tests (known-answer vectors of Random123).
void oracle_philox4x32_10(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t* out) {
    keyed::Philox ph{k0, k1};
    ph(c0, c1, c2, c3, out);
}

// Ingest (A.1) in device formats: int32 ids / fp32 weights. Drops w == 0, sums duplicates in order
// of appearance (fp32), rows ascending. Returns nnz; ptr has n+1 entries; col/w sized >= E.
// status: 0 ok, 2 id out of range, 3 self loop.
int64_t oracle_ingest(const int64_t* src, const int64_t* dst, const float* w, int64_t E, int64_t n, int64_t* ptr,
                      int32_t* col, float* wout, int* status) {
    *status = 0;
    std::vector<int64_t> ord;
    ord.reserve((size_t)E);
    for (int64_t p = 0; p < E; p++) {
        if (src[p] < 0 || src[p] >= n || dst[p] < 0 || dst[p] >= n) { *status = 2; return 0; }
        float wv = w ? w[p] : 1.0f;
        if (wv == 0.0f) continue;
        if (src[p] == dst[p]) { *status = 3; return 0; }
        ord.push_back(p);
    }
    // owner = column (second index, as rlap/ops.py:47 + reader.cc:52-55 store it), row = first index
    std::stable_sort(ord.begin(), ord.end(), [&](int64_t a, int64_t b) {
        if (dst[a] != dst[b]) return dst[a] < dst[b];
        return src[a] < src[b];
    });
    for (int64_t i = 0; i <= n; i++) ptr[i] = 0;
    int64_t nnz = 0, curc = -1, curr = -1;
    for (int64_t p : ord) {
        float wv = w ? w[p] : 1.0f;
        if (dst[p] == curc && src[p] == curr) {
            wout[nnz - 1] += wv;
        } else {
            col[nnz] = (int32_t)src[p]; wout[nnz] = wv; nnz++;
            ptr[dst[p] + 1]++;
            curc = dst[p]; curr = src[p];
        }
    }
    for (int64_t i = 0; i < n; i++) ptr[i + 1] += ptr[i];
    return nnz;
}

// keyed mode on a coalesced CSR (ptr/col/w as produced by oracle_ingest). graph_ptr[G+1] partitions the
// vertex range into independent graphs, num_remove[G] is t per graph. One view per call.
// Output rows sorted by (col, row); returns E'. out_* must hold >= nnz entries (E' <= nnz + 0: live
// multigraph entries never exceed the input's, see DESIGN.md §3.6).
// stats: D, F, maxlen, rounds, Draw. order_out (optional, n entries): elimination round of each vertex, -1 if kept.
// keep (optional, n entries; NULL = no mask, DESIGN.md §3.7): a nonzero flag protects the vertex, it is never
// eliminated. For graph g with m_g unprotected vertices: t_g = min(max(num_remove, 0), m_g) if g has a protected vertex,
// else min(max(num_remove, 0), n_g - 1). o_v = random ranks the unprotected vertices, numbered by ascending id, with the
// keyed permutation over m_g; degree / coarsen take the minimum key, the bucket and the independent-set test over the
// alive unprotected vertices only.
int64_t oracle_keyed_schur(int64_t n, const int64_t* ptr, const int32_t* col, const float* w, int64_t G,
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
            // the t vertices of lowest rank go, in rank order: strictly sequential here; the CUDA path
            // runs any schedule that respects "lower-ranked adjacent vertex first" (SURVEY.md App. B.4)
            RankPerm rp(ph, (uint32_t)gi, (flags & FLAG_SHARED_ORDER) ? 0u : view, (uint32_t)mg);
            std::vector<int32_t> by_rank((size_t)mg);
            for (int64_t c = 0; c < mg; c++) by_rank[(size_t)rp.rank((uint32_t)c)] = unprot[(size_t)c];
            for (int64_t k = 0; k < t; k++) {
                eliminate(g, by_rank[(size_t)k], o_v, o_n, flags, ph, view, st);
                if (order_out) order_out[by_rank[(size_t)k]] = (int32_t)k;
            }
            st.rounds = std::max(st.rounds, t);
        } else {
            // degree / coarsen: rounds over the minimum-key bucket of the alive unprotected vertices (DESIGN.md §3.4)
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

extern "C" void oracle_rank_perm(uint64_t seed, uint32_t graph, uint32_t view, uint32_t n_g, uint32_t* out) {
    keyed::Philox ph{(uint32_t)seed, (uint32_t)(seed >> 32)};
    keyed::RankPerm rp(ph, graph, view, n_g);
    for (uint32_t v = 0; v < n_g; v++) out[v] = rp.rank(v);
}

// The pop order of the reference's o_v = random queue for a given injected random_device stream
// (preconditioner.cc:588-613: shuffle 0..n-1 with mt19937(rd()), pop from the back). Test helper.
extern "C" void oracle_ref_random_order(int64_t n, uint64_t rd_state, int64_t* out) {
    refmode::RdStream rd{rd_state};
    std::vector<double> node_id((size_t)n);
    for (int64_t i = 0; i < n; i++) node_id[(size_t)i] = (double)i;
    std::mt19937 g(rd.next());
    std::shuffle(node_id.begin(), node_id.end(), g);
    for (int64_t i = 0; i < n; i++) out[i] = (int64_t)node_id[(size_t)(n - 1 - i)];
}

// The o_n order of a synthetic star: merged neighbours 0..n-1 (id order) with fixed-point weights q[]. out[p] = id of
// the neighbour at position p. Test helper for the tie rule (order_star).
extern "C" void oracle_star_order(const uint64_t* q, int32_t n, int o_n, int32_t* out) {
    keyed::Star s;
    for (int32_t i = 0; i < n; i++) {
        keyed::Merged mm;
        mm.nbr = i; mm.q = q[i]; mm.wf = 1.0f; mm.shuf = 0; mm.usample = 0;
        s.m.push_back(mm);
    }
    keyed::order_star(s, o_n);
    for (int32_t i = 0; i < n; i++) out[i] = s.m[(size_t)i].nbr;
}
