// Host graph cut behind include/phmrf_gco.h: alpha-beta swap and alpha-expansion on a general
// graph with integer costs, as GCO v3.0 (Veksler, Delong; the library pygco drives) runs them:
//
//  * energy  E(l) = sum_s D[s][l_s] + sum_{edges a<b} w_ab * V[l_b][l_a]
//  * swap    one cycle visits the label pairs (a, b), a ascending and b from K-1 down to a+1;
//            expansion one cycle visits the labels in ascending order
//  * cycles  repeat while the energy of a cycle is lower than the one before, at most n_iter
//            cycles (n_iter == -1: no limit).  GCO's expansion(-1) instead runs "adaptive" cycles
//            that revisit only the labels whose expansion helped; it stops, like this, where no
//            expansion lowers the energy, but the labels may differ.  The product path runs swap.
//  * move    a binary energy over the sites the move may change (0 = alpha, 1 = beta or the
//            site's current label), minimised by the Boykov-Kolmogorov max-flow; a site takes
//            value 1 only when it can reach the sink in the residual graph.  That cut (the
//            smallest sink side of all minimum cuts) depends on the energy alone, so the labels
//            do not depend on the order in which the max-flow finds its paths.
//  * limits  a data or smooth term above GCO_MAX_ENERGYTERM (1e7), or a non-metric smooth term
//            in an expansion move, is an error.
#include <algorithm>
#include <climits>
#include <cstdint>
#include <deque>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/phmrf_gco.h"

namespace {

typedef long long cap_t;
const long long MAX_ENERGYTERM = 10000000;  // GCO_MAX_ENERGYTERM

// Boykov-Kolmogorov max-flow ("An Experimental Comparison of Min-Cut/Max-Flow Algorithms for Energy
// Minimization in Vision", PAMI 2004).  Arcs come in pairs (a, a^1); tr[i] > 0 is a residual edge
// source->i, tr[i] < 0 one i->sink.
class MaxFlow {
  public:
    void reset(int n) {
        n_ = n;
        first_.assign(n, -1);
        tr_.assign(n, 0);
        head_.clear();
        next_.clear();
        rcap_.clear();
    }
    int n_nodes() const { return n_; }
    void add_tweights(int i, cap_t cap_source, cap_t cap_sink) { tr_[i] += cap_source - cap_sink; }
    void add_edge(int i, int j, cap_t cap, cap_t rev_cap) {
        if (cap == 0 && rev_cap == 0) return;
        const int a = (int)head_.size();
        head_.push_back(j); next_.push_back(first_[i]); rcap_.push_back(cap); first_[i] = a;
        head_.push_back(i); next_.push_back(first_[j]); rcap_.push_back(rev_cap); first_[j] = a + 1;
    }
    // x = 0 (source side) or 1 (sink side) of the cut, after maxflow()
    int what_segment(int i) const { return (parent_[i] != FREE && is_sink_[i]) ? 1 : 0; }

    void maxflow() {
        const int n = n_;
        parent_.assign(n, FREE);
        next_active_.assign(n, -1);
        ts_.assign(n, 0);
        dist_.assign(n, 0);
        is_sink_.assign(n, 0);
        q_head_ = q_tail_ = -1;
        orphans_.clear();
        for (int i = 0; i < n; ++i) {
            if (tr_[i] > 0) { is_sink_[i] = 0; parent_[i] = TERMINAL; set_active(i); dist_[i] = 1; }
            else if (tr_[i] < 0) { is_sink_[i] = 1; parent_[i] = TERMINAL; set_active(i); dist_[i] = 1; }
        }
        time_ = 0;
        int current = -1;
        for (;;) {
            int i = current;
            if (i >= 0) {
                next_active_[i] = -1;
                if (parent_[i] == FREE) i = -1;
            }
            if (i < 0 && (i = pop_active()) < 0) break;
            int found = -1;  // an arc from the source tree into the sink tree
            if (!is_sink_[i]) {
                for (int a = first_[i]; a >= 0; a = next_[a]) {
                    if (!rcap_[a]) continue;
                    const int j = head_[a];
                    if (parent_[j] == FREE) {
                        is_sink_[j] = 0; parent_[j] = a ^ 1; ts_[j] = ts_[i]; dist_[j] = dist_[i] + 1; set_active(j);
                    } else if (is_sink_[j]) { found = a; break; }
                    else if (ts_[j] <= ts_[i] && dist_[j] > dist_[i]) {
                        parent_[j] = a ^ 1; ts_[j] = ts_[i]; dist_[j] = dist_[i] + 1;
                    }
                }
            } else {
                for (int a = first_[i]; a >= 0; a = next_[a]) {
                    if (!rcap_[a ^ 1]) continue;
                    const int j = head_[a];
                    if (parent_[j] == FREE) {
                        is_sink_[j] = 1; parent_[j] = a ^ 1; ts_[j] = ts_[i]; dist_[j] = dist_[i] + 1; set_active(j);
                    } else if (!is_sink_[j]) { found = a ^ 1; break; }
                    else if (ts_[j] <= ts_[i] && dist_[j] > dist_[i]) {
                        parent_[j] = a ^ 1; ts_[j] = ts_[i]; dist_[j] = dist_[i] + 1;
                    }
                }
            }
            ++time_;
            if (found >= 0) {
                next_active_[i] = i;  // i stays the node being grown
                current = i;
                augment(found);
                while (!orphans_.empty()) {
                    const int o = orphans_.front();
                    orphans_.pop_front();
                    process_orphan(o, is_sink_[o] != 0);
                }
            } else {
                current = -1;
            }
        }
    }

  private:
    static constexpr int TERMINAL = -1, ORPHAN = -2, FREE = -3;
    static constexpr int INF_D = INT_MAX;

    void set_active(int i) {
        if (next_active_[i] >= 0) return;
        if (q_tail_ >= 0) next_active_[q_tail_] = i; else q_head_ = i;
        q_tail_ = i;
        next_active_[i] = i;
    }
    int pop_active() {
        while (q_head_ >= 0) {
            const int i = q_head_;
            q_head_ = (next_active_[i] == i) ? -1 : next_active_[i];
            if (q_head_ < 0) q_tail_ = -1;
            next_active_[i] = -1;
            if (parent_[i] != FREE) return i;
        }
        return -1;
    }
    void orphan_front(int i) { parent_[i] = ORPHAN; orphans_.push_front(i); }
    void orphan_rear(int i) { parent_[i] = ORPHAN; orphans_.push_back(i); }

    void augment(int middle) {
        cap_t f = rcap_[middle];
        int i;
        for (i = head_[middle ^ 1];; i = head_[parent_[i]]) {
            const int a = parent_[i];
            if (a == TERMINAL) break;
            f = std::min(f, rcap_[a ^ 1]);
        }
        f = std::min(f, tr_[i]);
        for (i = head_[middle];; i = head_[parent_[i]]) {
            const int a = parent_[i];
            if (a == TERMINAL) break;
            f = std::min(f, rcap_[a]);
        }
        f = std::min(f, -tr_[i]);

        rcap_[middle ^ 1] += f;
        rcap_[middle] -= f;
        for (i = head_[middle ^ 1];;) {
            const int a = parent_[i];
            if (a == TERMINAL) break;
            rcap_[a] += f;
            rcap_[a ^ 1] -= f;
            if (!rcap_[a ^ 1]) orphan_front(i);
            i = head_[a];
        }
        tr_[i] -= f;
        if (!tr_[i]) orphan_front(i);
        for (i = head_[middle];;) {
            const int a = parent_[i];
            if (a == TERMINAL) break;
            rcap_[a ^ 1] += f;
            rcap_[a] -= f;
            if (!rcap_[a]) orphan_front(i);
            i = head_[a];
        }
        tr_[i] += f;
        if (!tr_[i]) orphan_front(i);
    }

    // a new parent in the orphan's own tree, or the orphan leaves the tree
    void process_orphan(int i, bool sink) {
        int best = -1, d_min = INF_D;
        for (int a0 = first_[i]; a0 >= 0; a0 = next_[a0]) {
            if (!(sink ? rcap_[a0] : rcap_[a0 ^ 1])) continue;
            int j = head_[a0];
            if ((is_sink_[j] != 0) != sink || parent_[j] == FREE) continue;
            int d = 0;  // distance of j to its terminal, or INF_D if j's origin is an orphan
            for (;;) {
                if (ts_[j] == time_) { d += dist_[j]; break; }
                const int a = parent_[j];
                ++d;
                if (a == TERMINAL) { ts_[j] = time_; dist_[j] = 1; break; }
                if (a == ORPHAN) { d = INF_D; break; }
                j = head_[a];
            }
            if (d == INF_D) continue;
            if (d < d_min) { best = a0; d_min = d; }
            for (j = head_[a0]; ts_[j] != time_; j = head_[parent_[j]]) { ts_[j] = time_; dist_[j] = d--; }
        }
        if (best >= 0) {
            parent_[i] = best;
            ts_[i] = time_;
            dist_[i] = d_min + 1;
            return;
        }
        parent_[i] = FREE;
        for (int a0 = first_[i]; a0 >= 0; a0 = next_[a0]) {
            const int j = head_[a0];
            const int a = parent_[j];
            if ((is_sink_[j] != 0) != sink || a == FREE) continue;
            if (sink ? rcap_[a0] : rcap_[a0 ^ 1]) set_active(j);
            if (a != TERMINAL && a != ORPHAN && head_[a] == i) orphan_rear(j);
        }
    }

    int n_ = 0;
    std::vector<int> first_, parent_, next_active_, ts_, dist_;
    std::vector<char> is_sink_;
    std::vector<cap_t> tr_;
    std::vector<int> head_, next_;
    std::vector<cap_t> rcap_;
    std::deque<int> orphans_;
    int q_head_ = -1, q_tail_ = -1, time_ = 0;
};

// E(x) = A at x=0, B at x=1
void add_term1(MaxFlow &g, int x, cap_t A, cap_t B) { g.add_tweights(x, B, A); }

// E(x,y) = A B / C D over (x,y) = (0,0) (0,1) / (1,0) (1,1); needs B + C >= A + D
void add_term2(MaxFlow &g, int x, int y, cap_t A, cap_t B, cap_t C, cap_t D) {
    g.add_tweights(x, D, A);
    B -= A;
    C -= D;
    if (B < 0) {
        g.add_tweights(x, 0, B);
        g.add_tweights(y, 0, -B);
        g.add_edge(x, y, 0, B + C);
    } else if (C < 0) {
        g.add_tweights(x, 0, -C);
        g.add_tweights(y, 0, C);
        g.add_edge(x, y, B + C, 0);
    } else {
        g.add_edge(x, y, B, C);
    }
}

class GeneralGraphCut {
  public:
    GeneralGraphCut(int64_t n, int K, const int32_t *unary, const int64_t *edge_ids, const int32_t *edge_w,
                    int64_t n_edges, const int32_t *smooth)
        : n_(n), K_(K), unary_(unary), smooth_(smooth), labels_(n, 0), var_(n, -1) {
        // neighbour lists (CSR, both directions)
        start_.assign(n + 1, 0);
        for (int64_t e = 0; e < n_edges; ++e) { ++start_[edge_ids[2 * e] + 1]; ++start_[edge_ids[2 * e + 1] + 1]; }
        for (int64_t s = 0; s < n; ++s) start_[s + 1] += start_[s];
        nbr_.resize(2 * n_edges);
        nw_.resize(2 * n_edges);
        std::vector<int64_t> fill(start_.begin(), start_.end() - 1);
        for (int64_t e = 0; e < n_edges; ++e) {
            const int64_t a = edge_ids[2 * e], b = edge_ids[2 * e + 1];
            nbr_[fill[a]] = b; nw_[fill[a]++] = edge_w[e];
            nbr_[fill[b]] = a; nw_[fill[b]++] = edge_w[e];
        }
    }

    std::vector<int32_t> &labels() { return labels_; }

    long long energy() const {
        long long en = 0;
        for (int64_t s = 0; s < n_; ++s) {
            en += data(s, labels_[s]);
            for (int64_t k = start_[s]; k < start_[s + 1]; ++k)
                if (nbr_[k] < s) en += (long long)nw_[k] * smooth_[labels_[s] * (int64_t)K_ + labels_[nbr_[k]]];
        }
        return en;
    }

    long long swap(int n_iter) {
        return cycles(n_iter, [this] {
            for (int a = 0; a < K_; ++a)
                for (int b = K_ - 1; b > a; --b) swap_move(a, b);
        });
    }

    long long expansion(int n_iter) {
        return cycles(n_iter, [this] {
            for (int a = 0; a < K_; ++a) expansion_move(a);
        });
    }

  private:
    template <class F>
    long long cycles(int n_iter, F one_cycle) {
        long long n_max = n_iter == -1 ? LLONG_MAX : n_iter;
        long long en = energy(), old = en + 1;
        for (long long c = 1; old > en && c <= n_max; ++c) {
            old = en;
            one_cycle();
            en = energy();
        }
        return en;
    }

    cap_t data(int64_t s, int l) const { return unary_[s * K_ + l]; }
    cap_t pair(int64_t k, int l1, int l2) const { return (cap_t)nw_[k] * smooth_[l1 * (int64_t)K_ + l2]; }

    static void check_data(cap_t e0, cap_t e1) {
        if (e0 > MAX_ENERGYTERM || e1 > MAX_ENERGYTERM)
            throw std::runtime_error("data cost term larger than GCO_MAX_ENERGYTERM (1e7): danger of integer overflow");
    }
    static void check_smooth(cap_t e0, cap_t e1, cap_t e2 = 0, cap_t e3 = 0) {
        if (e0 > MAX_ENERGYTERM || e1 > MAX_ENERGYTERM || e2 > MAX_ENERGYTERM || e3 > MAX_ENERGYTERM)
            throw std::runtime_error("smooth cost term larger than GCO_MAX_ENERGYTERM (1e7): danger of integer overflow");
    }

    // sites labelled alpha or beta choose between the two (x=0: alpha, x=1: beta)
    void swap_move(int alpha, int beta) {
        active_.clear();
        for (int64_t s = 0; s < n_; ++s)
            if (labels_[s] == alpha || labels_[s] == beta) { var_[s] = (int)active_.size(); active_.push_back(s); }
        if (active_.empty()) return;
        g_.reset((int)active_.size());
        for (int i = 0; i < (int)active_.size(); ++i) {
            const int64_t s = active_[i];
            const cap_t e0 = data(s, alpha), e1 = data(s, beta);
            check_data(e0, e1);
            add_term1(g_, i, e0, e1);
            for (int64_t k = start_[s]; k < start_[s + 1]; ++k) {
                const int64_t t = nbr_[k];
                if (var_[t] >= 0) {
                    if (t > s) continue;   // each active pair once, from its larger site
                    const cap_t e00 = pair(k, alpha, alpha), e01 = pair(k, alpha, beta), e10 = pair(k, beta, alpha),
                                e11 = pair(k, beta, beta);
                    check_smooth(e00, e01, e10, e11);
                    add_term2(g_, i, var_[t], e00, e01, e10, e11);
                } else {
                    const cap_t e0n = pair(k, alpha, labels_[t]), e1n = pair(k, beta, labels_[t]);
                    check_smooth(e0n, e1n);
                    add_term1(g_, i, e0n, e1n);
                }
            }
        }
        g_.maxflow();
        for (int i = 0; i < (int)active_.size(); ++i) {
            labels_[active_[i]] = g_.what_segment(i) == 0 ? alpha : beta;
            var_[active_[i]] = -1;
        }
    }

    // sites not labelled alpha take alpha (x=0) or keep their label (x=1)
    void expansion_move(int alpha) {
        active_.clear();
        for (int64_t s = 0; s < n_; ++s)
            if (labels_[s] != alpha) { var_[s] = (int)active_.size(); active_.push_back(s); }
        if (active_.empty()) return;
        g_.reset((int)active_.size());
        for (int i = 0; i < (int)active_.size(); ++i) {
            const int64_t s = active_[i];
            const int ls = labels_[s];
            const cap_t e0 = data(s, alpha), e1 = data(s, ls);
            check_data(e0, e1);
            add_term1(g_, i, e0, e1);
            for (int64_t k = start_[s]; k < start_[s + 1]; ++k) {
                const int64_t t = nbr_[k];
                if (var_[t] >= 0) {
                    if (t > s) continue;
                    const int lt = labels_[t];
                    const cap_t e00 = pair(k, alpha, alpha), e01 = pair(k, alpha, lt), e10 = pair(k, ls, alpha),
                                e11 = pair(k, ls, lt);
                    check_smooth(e00, e01, e10, e11);
                    if (e00 + e11 > e01 + e10)
                        throw std::runtime_error("non-submodular expansion term: smooth costs must be a metric for "
                                                 "expansion");
                    add_term2(g_, i, var_[t], e00, e01, e10, e11);
                } else {
                    const cap_t e0n = pair(k, alpha, alpha), e1n = pair(k, ls, alpha);
                    check_smooth(e0n, e1n);
                    add_term1(g_, i, e0n, e1n);
                }
            }
        }
        g_.maxflow();
        for (int i = 0; i < (int)active_.size(); ++i) {
            if (g_.what_segment(i) == 0) labels_[active_[i]] = alpha;
            var_[active_[i]] = -1;
        }
    }

    int64_t n_;
    int K_;
    const int32_t *unary_, *smooth_;
    std::vector<int32_t> labels_;
    std::vector<int> var_;
    std::vector<int64_t> start_, nbr_;
    std::vector<int32_t> nw_;
    std::vector<int64_t> active_;
    MaxFlow g_;
};

}  // namespace

static thread_local std::string g_gco_error;

extern "C" const char *phmrf_gco_last_error(void) { return g_gco_error.c_str(); }

extern "C" int phmrf_gco_cut_general_graph(int64_t n_sites, int32_t n_labels, const int32_t *unary,
                                           const int64_t *edge_ids, const int32_t *edge_w, int64_t n_edges,
                                           const int32_t *smooth, const int32_t *init_labels, int32_t n_iter,
                                           int32_t algorithm, int32_t *labels_out, long long *energy_out,
                                           long long *energy_before_out) {
    if (n_sites <= 0 || n_labels <= 0 || !unary || !smooth || !labels_out || n_edges < 0 ||
        (n_edges > 0 && (!edge_ids || !edge_w))) {
        g_gco_error = "phmrf_gco_cut_general_graph: invalid arguments";
        return -1;
    }
    // the max-flow numbers the sites of one move with an int, like GCO's 32-bit SiteID
    if (n_sites * (int64_t)n_labels >= ((int64_t)1 << 31)) {
        g_gco_error = "phmrf_gco_cut_general_graph: n_sites*n_labels overflows GCO's 32-bit indexing";
        return -1;
    }
    for (int64_t e = 0; e < n_edges; ++e) {
        const int64_t a = edge_ids[2 * e], b = edge_ids[2 * e + 1];
        if (a < 0 || b < 0 || a >= n_sites || b >= n_sites || a >= b) {
            g_gco_error = "phmrf_gco_cut_general_graph: edges must satisfy 0 <= id1 < id2 < n_sites";
            return -1;
        }
    }
    if (init_labels)
        for (int64_t i = 0; i < n_sites; ++i)
            if (init_labels[i] < 0 || init_labels[i] >= n_labels) {
                g_gco_error = "phmrf_gco_cut_general_graph: init label out of range";
                return -1;
            }
    try {
        GeneralGraphCut gc(n_sites, n_labels, unary, edge_ids, edge_w, n_edges, smooth);
        if (init_labels) std::copy(init_labels, init_labels + n_sites, gc.labels().begin());
        if (energy_before_out) *energy_before_out = gc.energy();
        const long long en = algorithm == PHMRF_GCO_EXPANSION ? gc.expansion(n_iter) : gc.swap(n_iter);
        if (energy_out) *energy_out = en;
        std::copy(gc.labels().begin(), gc.labels().end(), labels_out);
    } catch (std::exception &ex) {
        g_gco_error = std::string("GCO: ") + ex.what();
        return -1;
    } catch (...) {
        g_gco_error = "GCO: unknown exception";
        return -1;
    }
    return 0;
}
