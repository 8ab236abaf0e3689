// Symbolic analysis: elimination ordering, fill, level schedule, Ybus structure.
// See symbolic.hpp.  Pure host C++ (no CUDA), also compiled into the host-sim
// test library.
#include "symbolic.hpp"

#include <algorithm>
#include <cmath>
#include <array>
#include <map>
#include <set>
#include <stdexcept>
#include <unordered_map>

namespace opfg {
namespace {

struct Order {
    std::vector<int> pivot_node;               // node eliminated as pivot k
    std::vector<std::vector<int>> strct;       // higher-numbered neighbours (as pivot indices), sorted
    std::vector<int> level_ptr;
    double cost = 0;
    std::string name;
};

// Eliminate nodes in the sequence `seq` (a permutation) and return, per node, its
// neighbour set at elimination time.
std::vector<std::vector<int>> eliminate(const std::vector<std::set<int>>& adj0, const std::vector<int>& seq) {
    std::vector<std::set<int>> adj = adj0;
    std::vector<std::vector<int>> nb_at(adj.size());
    for (int v : seq) {
        std::vector<int> nb(adj[v].begin(), adj[v].end());
        nb_at[v] = nb;
        for (int a : nb) adj[a].erase(v);
        for (size_t i = 0; i < nb.size(); ++i)
            for (size_t j = i + 1; j < nb.size(); ++j) {
                adj[nb[i]].insert(nb[j]);
                adj[nb[j]].insert(nb[i]);
            }
        adj[v].clear();
    }
    return nb_at;
}

// classic minimum degree (ties: lowest node id)
std::vector<int> min_degree_sequence(const std::vector<std::set<int>>& adj0) {
    std::vector<std::set<int>> adj = adj0;
    const int n = (int)adj.size();
    std::vector<char> done(n, 0);
    std::vector<int> seq;
    seq.reserve(n);
    for (int step = 0; step < n; ++step) {
        int best = -1;
        size_t bd = SIZE_MAX;
        for (int v = 0; v < n; ++v)
            if (!done[v] && adj[v].size() < bd) { bd = adj[v].size(); best = v; }
        std::vector<int> nb(adj[best].begin(), adj[best].end());
        for (int a : nb) adj[a].erase(best);
        for (size_t i = 0; i < nb.size(); ++i)
            for (size_t j = i + 1; j < nb.size(); ++j) {
                adj[nb[i]].insert(nb[j]);
                adj[nb[j]].insert(nb[i]);
            }
        adj[best].clear();
        done[best] = 1;
        seq.push_back(best);
    }
    return seq;
}

// Rounds of independent low-degree sets (tree contraction: rake leaves, compress
// chains; on meshed cores: independent sets of (near-)minimum degree).  Every
// round becomes one level of the parallel schedule, so the critical path is the
// number of rounds, O(log n) for radial feeders instead of the feeder length.
std::vector<int> independent_set_sequence(const std::vector<std::set<int>>& adj0, int slack) {
    std::vector<std::set<int>> adj = adj0;
    const int n = (int)adj.size();
    std::vector<char> done(n, 0);
    std::vector<int> seq;
    seq.reserve(n);
    int remaining = n;
    while (remaining > 0) {
        size_t mind = SIZE_MAX;
        for (int v = 0; v < n; ++v)
            if (!done[v]) mind = std::min(mind, adj[v].size());
        size_t thr = std::max<size_t>(mind + (size_t)slack, 2);
        std::vector<int> cand;
        for (int v = 0; v < n; ++v)
            if (!done[v] && adj[v].size() <= thr) cand.push_back(v);
        std::stable_sort(cand.begin(), cand.end(),
                         [&](int a, int b) { return adj[a].size() < adj[b].size(); });
        std::vector<char> blocked(n, 0);
        std::vector<int> chosen;
        for (int v : cand) {
            if (blocked[v]) continue;
            chosen.push_back(v);
            blocked[v] = 1;
            for (int a : adj[v]) blocked[a] = 1;
        }
        for (int v : chosen) {
            std::vector<int> nb(adj[v].begin(), adj[v].end());
            for (int a : nb) adj[a].erase(v);
            for (size_t i = 0; i < nb.size(); ++i)
                for (size_t j = i + 1; j < nb.size(); ++j) {
                    adj[nb[i]].insert(nb[j]);
                    adj[nb[j]].insert(nb[i]);
                }
            adj[v].clear();
            done[v] = 1;
            seq.push_back(v);
            --remaining;
        }
    }
    return seq;
}

// Turn an elimination sequence into a levelled order: level = longest dependency
// path; pivots renumbered by (level, position in seq).
Order make_order(const std::vector<std::set<int>>& adj0, const std::vector<int>& seq, int threads,
                 const std::string& name, int level_cap = 0) {
    const int n = (int)adj0.size();
    auto nb_at = eliminate(adj0, seq);
    std::vector<int> pos(n);
    for (int i = 0; i < n; ++i) pos[seq[i]] = i;
    std::vector<int> level(n, 0);
    for (int i = 0; i < n; ++i) {   // seq order is a valid topological order
        int v = seq[i];
        for (int a : nb_at[v]) level[a] = std::max(level[a], level[v] + 1);
    }
    if (level_cap > 0) {
        // Balanced levels: at most `level_cap` pivots per level.  A pivot may run later than its
        // earliest level as long as everything that depends on it still fits: list scheduling by
        // latest start (the tail of a radial feeder is a chain, its leaves have slack to spare).
        int n_lv = 0;
        for (int v = 0; v < n; ++v) n_lv = std::max(n_lv, level[v] + 1);
        std::vector<int> latest(n, n_lv - 1);
        for (int i = n - 1; i >= 0; --i) {
            const int v = seq[i];
            for (int a : nb_at[v]) latest[v] = std::min(latest[v], latest[a] - 1);
        }
        std::vector<int> pending(n, 0), assigned(n, -1);   // predecessors not yet scheduled
        std::vector<std::vector<int>> preds(n);
        for (int v = 0; v < n; ++v) for (int a : nb_at[v]) { preds[a].push_back(v); pending[a]++; }
        std::vector<int> ready;
        for (int v = 0; v < n; ++v) if (!pending[v]) ready.push_back(v);
        int done = 0, round = 0;
        while (done < n) {
            std::stable_sort(ready.begin(), ready.end(), [&](int a, int b) {
                return latest[a] != latest[b] ? latest[a] < latest[b] : pos[a] < pos[b]; });
            const int take = std::min<int>((int)ready.size(), level_cap);
            std::vector<int> now(ready.begin(), ready.begin() + take);
            ready.erase(ready.begin(), ready.begin() + take);
            for (int v : now) { assigned[v] = round; ++done; }
            for (int v : now) for (int a : nb_at[v]) if (--pending[a] == 0) ready.push_back(a);
            ++round;
        }
        level = assigned;
    }
    std::vector<int> by(n);
    for (int i = 0; i < n; ++i) by[i] = seq[i];
    std::stable_sort(by.begin(), by.end(), [&](int a, int b) { return level[a] < level[b]; });
    Order o;
    o.name = name;
    o.pivot_node = by;
    std::vector<int> piv_of(n);
    for (int k = 0; k < n; ++k) piv_of[by[k]] = k;
    o.strct.resize(n);
    int nl = n ? level[by[n - 1]] + 1 : 0;
    o.level_ptr.assign(nl + 1, 0);
    for (int k = 0; k < n; ++k) {
        o.level_ptr[level[by[k]] + 1]++;
        for (int a : nb_at[by[k]]) o.strct[k].push_back(piv_of[a]);
        std::sort(o.strct[k].begin(), o.strct[k].end());
    }
    for (int l = 0; l < nl; ++l) o.level_ptr[l + 1] += o.level_ptr[l];
    // cost model (cycles): latency floor per phase + serialised item work per thread
    double cost = 0;
    const double T = threads;
    for (int l = 0; l < nl; ++l) {
        double na = o.level_ptr[l + 1] - o.level_ptr[l];
        double pairs_a = 0, nbk = 0, pairs_b = 0;
        for (int k = o.level_ptr[l]; k < o.level_ptr[l + 1]; ++k) nbk += 2.0 * o.strct[k].size();
        // pairs landing on targets of this level are not known exactly here; approximate by struct sizes
        for (int k = o.level_ptr[l]; k < o.level_ptr[l + 1]; ++k) {
            double s = (double)o.strct[k].size();
            pairs_a += s;            // updates onto later diagonals
            pairs_b += s * (s - 1);  // updates onto later off-diagonals
        }
        cost += 180 + std::ceil(na / T) * 60 + pairs_a / std::min(T, std::max(1.0, na)) * 20;   // phase A
        cost += 90 + std::ceil(nbk / T) * 30 + pairs_b / T * 20;                                   // phase B
        cost += 80 + std::ceil(na / T) * (20 + 10 * (nbk / std::max(1.0, 2 * na)));                // backward
    }
    o.cost = cost;
    return o;
}

// Breadth-first distances from `root` (-1 outside its component); returns the nodes in visiting order.
std::vector<int> bfs(const std::vector<std::set<int>>& adj, int root, std::vector<int>& dist,
                     std::vector<int>* from = nullptr) {
    dist.assign(adj.size(), -1);
    if (from) from->assign(adj.size(), -1);
    std::vector<int> seen{root};
    dist[root] = 0;
    for (size_t i = 0; i < seen.size(); ++i)
        for (int a : adj[seen[i]])
            if (dist[a] < 0) {
                dist[a] = dist[seen[i]] + 1;
                if (from) (*from)[a] = seen[i];
                seen.push_back(a);
            }
    return seen;
}

// Leaf-first order of a forest with every tree rooted at a centre (the middle of a longest path, found by
// two BFS passes): nodes by decreasing depth from their tree's centre.  Eliminating a node removes a leaf
// of what is left, so there is no fill and each pivot keeps one later neighbour (its parent), and the
// dependency chain of a tree is its radius + 1 levels: the fewest any fill-free order has, since a
// leaf-first order is a rooted tree and no root gives a lower height.  A tree with two centres takes the
// one that gives fewer levels under `level_cap`, then the lower node id.
std::vector<int> centre_rooted_sequence(const std::vector<std::set<int>>& adj, int threads, int level_cap) {
    const int n = (int)adj.size();
    std::vector<int> comp_of(n, -1), dist, from;
    std::vector<std::array<int, 2>> centres;                 // per component; [1] = -1 with one centre
    for (int v0 = 0; v0 < n; ++v0) {
        if (comp_of[v0] >= 0) continue;
        const int u = bfs(adj, v0, dist).back();             // farthest from v0: one end of a longest path
        const std::vector<int> seen = bfs(adj, u, dist, &from);
        std::vector<int> path{seen.back()};                  // the other end, walked back to u
        while (path.back() != u) path.push_back(from[path.back()]);
        const int len = (int)path.size() - 1;
        for (int v : seen) comp_of[v] = (int)centres.size();
        std::array<int, 2> c{path[len / 2], len % 2 ? path[len / 2 + 1] : -1};
        if (c[1] >= 0 && c[1] < c[0]) std::swap(c[0], c[1]);
        centres.push_back(c);
    }
    std::vector<int> root(centres.size());
    for (size_t c = 0; c < centres.size(); ++c) root[c] = centres[c][0];
    auto sequence = [&]() {
        std::vector<int> depth(n);
        for (size_t c = 0; c < centres.size(); ++c) {
            bfs(adj, root[c], dist);
            for (int v = 0; v < n; ++v) if (comp_of[v] == (int)c) depth[v] = dist[v];
        }
        std::vector<int> seq(n);
        for (int v = 0; v < n; ++v) seq[v] = v;
        std::stable_sort(seq.begin(), seq.end(), [&](int a, int b) { return depth[a] > depth[b]; });
        return seq;
    };
    if (level_cap > 0) {
        auto levels = [&]() { return (int)make_order(adj, sequence(), threads, "", level_cap).level_ptr.size() - 1; };
        int best = levels();
        for (size_t c = 0; c < centres.size(); ++c) {
            if (centres[c][1] < 0) continue;
            root[c] = centres[c][1];
            const int other = levels();
            if (other < best) best = other;
            else root[c] = centres[c][0];
        }
    }
    return sequence();
}

inline int64_t key(int i, int j) { return ((int64_t)i << 32) | (uint32_t)j; }

// graph of the non-reference buses (self loops dropped, parallel branches collapse); bus_of_node: the bus of each node
std::vector<std::set<int>> bus_graph(int nb, const std::vector<int>& bus_type, const std::vector<BranchHost>& branches,
                                     std::vector<int>& bus_of_node) {
    std::vector<int> node_of_bus(nb, -1);
    bus_of_node.clear();
    for (int b = 0; b < nb; ++b)
        if (bus_type[b] != 3) { node_of_bus[b] = (int)bus_of_node.size(); bus_of_node.push_back(b); }
    std::vector<std::set<int>> adj(bus_of_node.size());
    for (const auto& br : branches) {
        if (br.f == br.t) continue;
        int a = node_of_bus[br.f], b = node_of_bus[br.t];
        if (a >= 0 && b >= 0) { adj[a].insert(b); adj[b].insert(a); }
    }
    return adj;
}

}  // namespace

bool is_forest(int nb, const std::vector<int>& bus_type, const std::vector<BranchHost>& branches) {
    std::vector<int> bus_of_node, dist;
    const auto adj = bus_graph(nb, bus_type, branches, bus_of_node);
    const int n = (int)adj.size();
    size_t edges = 0;
    for (const auto& a : adj) edges += a.size();
    edges /= 2;
    int components = 0;
    std::vector<char> seen(n, 0);
    for (int v = 0; v < n; ++v) {
        if (seen[v]) continue;
        ++components;
        for (int u : bfs(adj, v, dist)) seen[u] = 1;
    }
    return edges == (size_t)(n - components);
}

void analyse(int nb, const std::vector<int>& bus_type, const std::vector<BranchHost>& branches,
             int ordering, int threads, Symbolic& s, int level_cap) {
    s = Symbolic();
    s.nb = nb;
    std::vector<int> bus_of_node;
    const std::vector<std::set<int>> adj = bus_graph(nb, bus_type, branches, bus_of_node);
    const int n = (int)bus_of_node.size();
    s.n = n;
    std::vector<Order> cands;
    const bool least_work = ordering == 3;     // lane-per-environment kernel: levels are irrelevant, fill is work
    if (least_work) ordering = 0;
    if (ordering == 0 || ordering == 1) cands.push_back(make_order(adj, min_degree_sequence(adj), threads, "min_degree"));
    if (ordering == 0 || ordering == 2) {
        cands.push_back(make_order(adj, independent_set_sequence(adj, 0), threads, "independent_set"));
        cands.push_back(make_order(adj, independent_set_sequence(adj, 1), threads, "independent_set+1"));
    }
    if (ordering == 4) cands.push_back(make_order(adj, centre_rooted_sequence(adj, threads, level_cap), threads, "centre_rooted", level_cap));
    if (cands.empty()) throw std::runtime_error("unknown ordering");
    const Order* best = &cands[0];
    auto work = [](const Order& o) {           // Schur-update pairs: sum over pivots of |struct|^2
        double w = 0;
        for (const auto& st : o.strct) w += (double)st.size() * (double)st.size() + 2.0 * (double)st.size();
        return w;
    };
    for (const auto& c : cands)
        if (least_work ? work(c) < work(*best) : c.cost < best->cost) best = &c;
    const Order& o = *best;
    s.ordering_name = o.name;
    s.est_cycles = o.cost;
    s.level_ptr = o.level_ptr;
    s.n_levels = (int)o.level_ptr.size() - 1;

    // internal numbering
    s.int_of_bus.assign(nb, -1);
    s.bus_of_int.assign(nb, -1);
    for (int k = 0; k < n; ++k) {
        int bus = bus_of_node[o.pivot_node[k]];
        s.int_of_bus[bus] = k;
        s.bus_of_int[k] = bus;
    }
    int nxt = n;
    for (int b = 0; b < nb; ++b)
        if (bus_type[b] == 3) { s.int_of_bus[b] = nxt; s.bus_of_int[nxt] = b; ++nxt; }

    // ---- blocks ----
    std::unordered_map<int64_t, int> blk_id;
    s.blk_row.resize(n);
    s.blk_col.resize(n);
    for (int k = 0; k < n; ++k) { blk_id[key(k, k)] = k; s.blk_row[k] = k; s.blk_col[k] = k; }
    auto add_block = [&](int i, int j) {
        int id = (int)s.blk_row.size();
        blk_id[key(i, j)] = id;
        s.blk_row.push_back(i);
        s.blk_col.push_back(j);
        return id;
    };
    for (int l = 0; l < s.n_levels; ++l) {
        for (int k = o.level_ptr[l]; k < o.level_ptr[l + 1]; ++k)
            for (int j : o.strct[k]) add_block(k, j);      // U row of pivot k
        for (int k = o.level_ptr[l]; k < o.level_ptr[l + 1]; ++k)
            for (int i : o.strct[k]) add_block(i, k);      // L column of pivot k
    }
    s.n_blocks = (int)s.blk_row.size();

    // original (Ybus) pattern among pivots
    std::set<int64_t> orig;
    for (const auto& br : branches) {
        int a = s.int_of_bus[br.f], b = s.int_of_bus[br.t];
        if (a < n && b < n && a != b) { orig.insert(key(a, b)); orig.insert(key(b, a)); }
    }
    for (int id = n; id < s.n_blocks; ++id)
        if (!orig.count(key(s.blk_row[id], s.blk_col[id]))) s.fill_ids.push_back(id);

    // ---- update pairs, generated pivot by pivot so every list is in increasing m ----
    std::vector<std::vector<int>> dl(n), dw(n), dm(n);
    std::map<int, std::pair<std::vector<int>, std::vector<int>>> opairs;   // target block -> (l ids, w ids)
    for (int m = 0; m < n; ++m) {
        const auto& st = o.strct[m];
        for (int i : st) {
            int lid = blk_id[key(i, m)];
            for (int j : st) {
                int wid = blk_id[key(m, j)];
                if (i == j) { dl[i].push_back(lid); dw[i].push_back(wid); dm[i].push_back(m); }
                else {
                    auto& p = opairs[blk_id.at(key(i, j))];
                    p.first.push_back(lid);
                    p.second.push_back(wid);
                }
            }
        }
    }
    s.dp_ptr.assign(n + 1, 0);
    for (int k = 0; k < n; ++k) {
        s.dp_ptr[k + 1] = s.dp_ptr[k] + (int)dl[k].size();
        s.dp_l.insert(s.dp_l.end(), dl[k].begin(), dl[k].end());
        s.dp_w.insert(s.dp_w.end(), dw[k].begin(), dw[k].end());
        s.dp_m.insert(s.dp_m.end(), dm[k].begin(), dm[k].end());
    }
    {   // eager gather schedule (pair lists are in increasing m, hence grouped by source level)
        std::vector<int> level_of(n, 0);
        for (int l = 0; l < s.n_levels; ++l)
            for (int k = o.level_ptr[l]; k < o.level_ptr[l + 1]; ++k) level_of[k] = l;
        s.dp_own.assign(n, 0);
        std::vector<std::vector<std::array<int, 3>>> per_phase(s.n_levels + 1);
        for (int k = 0; k < n; ++k) {
            int p = s.dp_ptr[k];
            const int pe = s.dp_ptr[k + 1];
            while (p < pe && level_of[s.dp_m[p]] < level_of[k] - 1) {
                const int ls = level_of[s.dp_m[p]], begin = p;
                while (p < pe && level_of[s.dp_m[p]] == ls) ++p;
                per_phase[ls + 1].push_back({k, begin, p - begin});
            }
            s.dp_own[k] = p;
        }
        s.eg_ptr.assign(s.n_levels + 1, 0);
        for (int l = 0; l < s.n_levels; ++l) {
            for (const auto& it : per_phase[l]) { s.eg_k.push_back(it[0]); s.eg_begin.push_back(it[1]); s.eg_count.push_back(it[2]); }
            s.eg_ptr[l + 1] = (int)s.eg_k.size();
        }
    }
    // off-diagonal items per level: every U block (needs scaling), L blocks only if they gather
    s.off_ptr.assign(s.n_levels + 1, 0);
    s.op_ptr.push_back(0);
    for (int l = 0; l < s.n_levels; ++l) {
        for (int pass = 0; pass < 2; ++pass)
            for (int k = o.level_ptr[l]; k < o.level_ptr[l + 1]; ++k)
                for (int other : o.strct[k]) {
                    int id = pass == 0 ? blk_id[key(k, other)] : blk_id[key(other, k)];
                    auto it = opairs.find(id);
                    if (pass == 1 && it == opairs.end()) continue;
                    s.off_tgt.push_back(id);
                    s.off_piv.push_back(pass == 0 ? k : -1);
                    if (it != opairs.end()) {
                        s.op_l.insert(s.op_l.end(), it->second.first.begin(), it->second.first.end());
                        s.op_w.insert(s.op_w.end(), it->second.second.begin(), it->second.second.end());
                    }
                    s.op_ptr.push_back((int)s.op_l.size());
                }
        s.off_ptr[l + 1] = (int)s.off_tgt.size();
    }
    // backward substitution lists
    s.up_ptr.assign(n + 1, 0);
    for (int k = 0; k < n; ++k) {
        for (int j : o.strct[k]) { s.up_w.push_back(blk_id[key(k, j)]); s.up_j.push_back(j); }
        s.up_ptr[k + 1] = (int)s.up_w.size();
    }

    // ---- Ybus CSR in internal numbering, diagonal first in every row ----
    std::vector<std::map<int, std::vector<std::pair<int, int>>>> rows(nb);
    for (int b = 0; b < nb; ++b) rows[s.int_of_bus[b]][s.int_of_bus[b]].push_back({b, 4});
    for (int ib = 0; ib < (int)branches.size(); ++ib) {
        const auto& br = branches[ib];
        int f = s.int_of_bus[br.f], t = s.int_of_bus[br.t];
        rows[f][f].push_back({ib, 0});
        rows[f][t].push_back({ib, 1});
        rows[t][f].push_back({ib, 2});
        rows[t][t].push_back({ib, 3});
    }
    s.y_ptr.assign(nb + 1, 0);
    s.y_diag.assign(nb, 0);
    s.yc_ptr.push_back(0);
    for (int r = 0; r < nb; ++r) {
        auto emit = [&](int c, const std::vector<std::pair<int, int>>& contrib) {
            s.y_col.push_back(c);
            int blk = -1;
            if (r < n && c < n) blk = blk_id.at(key(r, c));
            s.y_blk.push_back(blk);
            for (auto& pr : contrib) { s.yc_branch.push_back(pr.first); s.yc_role.push_back(pr.second); }
            s.yc_ptr.push_back((int)s.yc_branch.size());
        };
        s.y_diag[r] = (int)s.y_col.size();
        emit(r, rows[r][r]);
        for (auto& kv : rows[r])
            if (kv.first != r) emit(kv.first, kv.second);
        s.y_ptr[r + 1] = (int)s.y_col.size();
    }

    // ---- flop model ----
    const double nnz = (double)s.y_col.size();
    double lu = 0;
    lu += 16.0 * s.dp_l.size() + 4.0 * s.dp_l.size();      // diag Schur updates + rhs updates
    lu += 14.0 * n + 6.0 * n;                              // 2x2 inverse + t = invD*y
    lu += 16.0 * s.op_l.size();                            // off-diagonal Schur updates
    double n_u = 0;
    for (int p : s.off_piv) n_u += p >= 0;
    lu += 12.0 * n_u;                                      // W = invD * U
    lu += 8.0 * s.up_w.size();                             // backward substitution
    s.lu_flops = lu;
    s.flops_per_iter = 28.0 * nnz + 24.0 * nb + lu + 2.0 * n + 40.0 * nb;
}

void build_lane_schedule(const Symbolic& s, LaneSchedule& o) {
    o = LaneSchedule();
    const int n = s.n;
    // lower(k): pivots m < k with a block (k, m); upper(k) = the up_* list of k
    std::vector<std::vector<int>> lower(n);
    for (int m = 0; m < n; ++m)
        for (int p = s.up_ptr[m]; p < s.up_ptr[m + 1]; ++p) lower[s.up_j[p]].push_back(m);   // m ascending
    std::set<int64_t> orig;                    // blocks fed by a Ybus entry
    for (int r = 0; r < n; ++r)
        for (int e = s.y_ptr[r]; e < s.y_ptr[r + 1]; ++e)
            if (s.y_col[e] < n) orig.insert(key(r, s.y_col[e]));
    o.y_rpos.assign(s.y_ptr[n], -1);
    o.diag_pos.resize(n);
    o.fill_ptr.assign(n + 1, 0);
    o.el_ptr.assign(n + 1, 0);
    o.up_rpos.assign(s.up_w.size(), -1);
    o.el_uptr.push_back(0);
    std::vector<int> pos_of(n, -1);
    for (int k = 0; k < n; ++k) {
        const int nl = (int)lower[k].size(), nu = s.up_ptr[k + 1] - s.up_ptr[k];
        for (int a = 0; a < nl; ++a) pos_of[lower[k][a]] = a;
        pos_of[k] = nl;
        for (int a = 0; a < nu; ++a) { pos_of[s.up_j[s.up_ptr[k] + a]] = nl + 1 + a; o.up_rpos[s.up_ptr[k] + a] = nl + 1 + a; }
        o.diag_pos[k] = nl;
        o.max_row = std::max(o.max_row, nl + 1 + nu);
        for (int e = s.y_ptr[k]; e < s.y_ptr[k + 1]; ++e)
            if (s.y_col[e] < n) {
                if (pos_of[s.y_col[e]] < 0) throw std::runtime_error("lane schedule: Ybus entry outside the filled pattern");
                o.y_rpos[e] = pos_of[s.y_col[e]];
            }
        auto is_fill = [&](int c) { return !orig.count(key(k, c)); };
        for (int m : lower[k]) if (is_fill(m)) o.fill_rpos.push_back(pos_of[m]);
        for (int a = 0; a < nu; ++a) if (is_fill(s.up_j[s.up_ptr[k] + a])) o.fill_rpos.push_back(nl + 1 + a);
        o.fill_ptr[k + 1] = (int)o.fill_rpos.size();
        for (int m : lower[k]) {
            o.el_rpos.push_back(pos_of[m]);
            o.el_m.push_back(m);
            for (int p = s.up_ptr[m]; p < s.up_ptr[m + 1]; ++p) {
                const int j = s.up_j[p];
                if (pos_of[j] < 0) throw std::runtime_error("lane schedule: update target outside the filled pattern");
                o.upd_w.push_back(p);
                o.upd_rpos.push_back(pos_of[j]);
            }
            o.el_uptr.push_back((int)o.upd_w.size());
        }
        o.el_ptr[k + 1] = (int)o.el_rpos.size();
        for (int m : lower[k]) pos_of[m] = -1;
        pos_of[k] = -1;
        for (int a = 0; a < nu; ++a) pos_of[s.up_j[s.up_ptr[k] + a]] = -1;
    }
}

void factor_dc(const Symbolic& s, const std::vector<BranchHost>& branches, std::vector<double>& val, bool& ok) {
    const int n = s.n;
    val.assign(s.n_blocks, 0.0);
    std::unordered_map<int64_t, int> blk_id;
    for (int id = 0; id < s.n_blocks; ++id) blk_id[key(s.blk_row[id], s.blk_col[id])] = id;
    for (const auto& br : branches) {
        double ratio = br.tap == 0.0 ? 1.0 : br.tap;
        double b = 1.0 / br.x / ratio;
        int f = s.int_of_bus[br.f], t = s.int_of_bus[br.t];
        if (f < n) val[f] += b;
        if (t < n) val[t] += b;
        if (f < n && t < n && f != t) { val[blk_id.at(key(f, t))] -= b; val[blk_id.at(key(t, f))] -= b; }
    }
    ok = true;
    // same schedule as the device factorisation, scalar entries
    int item = 0;
    for (int l = 0; l < s.n_levels; ++l) {
        for (int k = s.level_ptr[l]; k < s.level_ptr[l + 1]; ++k) {
            double d = val[k];
            for (int p = s.dp_ptr[k]; p < s.dp_ptr[k + 1]; ++p) d -= val[s.dp_l[p]] * val[s.dp_w[p]];
            if (!(std::fabs(d) > 1e-300)) ok = false;
            val[k] = 1.0 / d;
        }
        for (; item < s.off_ptr[l + 1]; ++item) {
            int tgt = s.off_tgt[item];
            double v = val[tgt];
            for (int p = s.op_ptr[item]; p < s.op_ptr[item + 1]; ++p) v -= val[s.op_l[p]] * val[s.op_w[p]];
            if (s.off_piv[item] >= 0) v *= val[s.off_piv[item]];
            val[tgt] = v;
        }
    }
}

}  // namespace opfg
