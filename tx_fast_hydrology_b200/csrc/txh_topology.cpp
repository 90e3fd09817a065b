// txh_topology.cpp -- topology pass + dataflow schedule builder (host, exact integers).
// See txh_topology.hpp for what each artefact replaces in the reference.
#include "txh_topology.hpp"

#include <algorithm>
#include <functional>
#include <numeric>
#include <queue>

namespace txh {

// ---------------------------------------------------------------------------
// Topology
// ---------------------------------------------------------------------------
bool Topology::build(int64_t n_, const int64_t* e, std::string& err)
{
    if (n_ <= 0 || n_ >= (int64_t(1) << 30)) { err = "n out of range"; return false; }
    n = n_;
    end.resize(n);
    for (int64_t j = 0; j < n; ++j) {
        if (e[j] < 0 || e[j] >= n) { err = "endnodes entry out of range"; return false; }
        end[j] = (int32_t)e[j];
    }
    // indegree without self-loops: muskingum.py:322-330
    indeg.assign(n, 0);
    for (int64_t j = 0; j < n; ++j)
        if (end[j] != j) indeg[end[j]] += 1;
    child_off.assign(n + 1, 0);
    for (int64_t j = 0; j < n; ++j) child_off[j + 1] = child_off[j] + indeg[j];
    child.resize(child_off[n]);
    {
        std::vector<int32_t> fill(child_off.begin(), child_off.end() - 1);
        for (int64_t j = 0; j < n; ++j)
            if (end[j] != j) child[fill[end[j]]++] = (int32_t)j;   // ascending id
    }
    heads.clear();
    for (int64_t j = 0; j < n; ++j)
        if (indeg[j] == 0) heads.push_back((int32_t)j);            // muskingum.py:444

    // Kahn by level: frontier k is exactly the set of level-k reaches.
    level.assign(n, 0);
    topo.clear(); topo.reserve(n);
    level_off.clear(); level_off.push_back(0);
    {
        std::vector<int32_t> pending(indeg), frontier(heads), next;
        int32_t lv = 0;
        while (!frontier.empty()) {
            topo.insert(topo.end(), frontier.begin(), frontier.end());
            level_off.push_back((int32_t)topo.size());
            next.clear();
            for (int32_t j : frontier) {
                int32_t d = end[j];
                if (d == j) continue;
                if (level[d] < lv + 1) level[d] = lv + 1;
                if (--pending[d] == 0) next.push_back(d);
            }
            std::sort(next.begin(), next.end());
            frontier.swap(next);
            ++lv;
        }
        nlevels = lv;
    }
    if ((int64_t)topo.size() != n) { err = "network has a cycle (not a forest of in-trees)"; return false; }

    subtree.assign(n, 1);
    for (int32_t j : topo)
        if (end[j] != j) subtree[end[j]] += subtree[j];

    main_child.assign(n, -1);
    for (int64_t j = 0; j < n; ++j) {
        int32_t best = -1;
        for (int32_t k = child_off[j]; k < child_off[j + 1]; ++k) {
            int32_t c = child[k];
            if (best < 0 || level[c] > level[best]) best = c;      // ties keep the lowest id
        }
        main_child[j] = best;
    }
    path_id.assign(n, -1); path_pos.assign(n, 0); path_len.clear();
    for (int32_t j : topo) {
        int32_t m = main_child[j];
        if (m < 0) { path_id[j] = (int32_t)path_len.size(); path_pos[j] = 0; path_len.push_back(1); }
        else {
            path_id[j] = path_id[m]; path_pos[j] = path_pos[m] + 1;
            path_len[path_id[j]] = path_pos[j] + 1;
        }
    }

    // maximal unbranched chains: v continues its upstream reach's chain iff indegree[v] == 1
    chain_id.assign(n, -1); chain_pos.assign(n, 0); chain_len.clear();
    for (int64_t j = 0; j < n; ++j)
        if (indeg[j] != 1) { chain_id[j] = (int32_t)chain_len.size(); chain_len.push_back(1); }
    for (int32_t j : topo)
        if (indeg[j] == 1) {
            int32_t u = child[child_off[j]];
            chain_id[j] = chain_id[u]; chain_pos[j] = chain_pos[u] + 1;
            chain_len[chain_id[j]] = chain_pos[j] + 1;
        }

    // the reference's visit sequence: nutils.py:72-88
    visit.clear(); visit.reserve(n);
    {
        std::vector<int32_t> work(indeg);
        for (int32_t h : heads) {
            int32_t s = h, d = end[s];
            while (work[s] == 0) {
                visit.push_back(s);
                work[d] -= 1;
                s = d; d = end[s];
                if ((int64_t)visit.size() > n) break;
            }
        }
        if ((int64_t)visit.size() != n) { err = "reference walk did not visit every reach once"; return false; }
    }
    return true;
}

// ---------------------------------------------------------------------------
// Schedule
// ---------------------------------------------------------------------------
namespace {

struct Unit {
    int32_t grp;                      // row group (contiguous rows in the final layout), -1 for LINK
    int32_t kind;
    int32_t link_off, link_len;       // LINK: its entries in link_last
    int32_t side_off;                 // PRE: first side-buffer row
    std::vector<uint32_t> ins;        // input words; ROW entries hold REACH ids until positions are known
    std::vector<int32_t> A, B;        // same-step / previous-step dependencies (unit ids)
};

void sort_unique(std::vector<int32_t>& v)
{
    std::sort(v.begin(), v.end());
    v.erase(std::unique(v.begin(), v.end()), v.end());
}

}  // namespace

bool Schedule::build(const Topology& t, const SchedParams& p_in, std::string& err)
{
    SchedParams p = p_in;
    // Short segments keep the per-step work of a segment (serial in one warp) small; long networks need
    // longer ones so that the hop chain along the main stem stays short: about 100 hops along the deepest path.
    if (p.spine_cap <= 0) p.spine_cap = std::min(16, std::max(6, t.nlevels / 100));
    prm = p;
    const int64_t n = t.n;
    if (p.spine_cap < 1 || p.spine_cap > 4096 || p.pocket_cap < 1 || p.pocket_cap > 4096 ||
        p.long_path_min < 2 || p.max_slots < 0 || p.max_slots > 30 || p.link_cap < 1) {
        err = "bad schedule parameters"; return false;
    }
    std::vector<uint8_t> is_long(n);
    for (int64_t j = 0; j < n; ++j) is_long[j] = t.path_len[t.path_id[j]] >= p.long_path_min;

    // row groups: reaches in processing order + their header words
    std::vector<int32_t> g_begin, g_len, rows;
    std::vector<uint32_t> rhdr;
    rows.reserve(n); rhdr.reserve(n);
    std::vector<Unit> units;
    std::vector<int32_t> final_unit(n, -1);   // pocket reaches: their task; last reach of a segment: the path's LINK
    std::vector<int32_t> pre_unit(n, -1);     // spine reaches: the PRE unit of their segment
    std::vector<int32_t> link_reach;          // per LINK entry: last reach of the segment
    auto mk = [](int32_t grp, int32_t kind) { Unit u; u.grp = grp; u.kind = kind; u.link_off = u.link_len = 0; u.side_off = 0; return u; };
    std::vector<int32_t> push_of(n, -1);      // pocket roots feeding a spine: their side-buffer row
    n_side = 0;

    // ---- spines: long paths cut into segments (PRE + FIX each) and one LINK per path ---------
    {
        const int32_t npaths = (int32_t)t.path_len.size();
        std::vector<int32_t> poff(npaths + 1, 0);
        for (int32_t q = 0; q < npaths; ++q) poff[q + 1] = poff[q] + t.path_len[q];
        std::vector<int32_t> member(n);
        for (int64_t j = 0; j < n; ++j) member[poff[t.path_id[j]] + t.path_pos[j]] = (int32_t)j;
        std::vector<int32_t> cuts;
        for (int32_t q = 0; q < npaths; ++q) {
            const int32_t len = t.path_len[q];
            if (len < p.long_path_min) continue;
            // a reach joined by another long path starts a segment: its inflow is only known to LINK
            std::vector<int32_t> forced{0};
            for (int32_t k = 1; k < len; ++k) {
                const int32_t j = member[poff[q] + k];
                for (int32_t c = t.child_off[j]; c < t.child_off[j + 1]; ++c)
                    if (t.child[c] != t.main_child[j] && is_long[t.child[c]]) { forced.push_back(k); break; }
            }
            forced.push_back(len);
            // a segment ends when it has spine_cap reaches or side_cap pocket roots joining it: the serial work of
            // a segment per step (rows + rows handed over by other tasks) paces the whole chain downstream
            cuts.clear();
            for (size_t f = 0; f + 1 < forced.size(); ++f) {
                const int32_t a0 = forced[f], a1 = forced[f + 1];
                int32_t s0 = a0, nrows = 0, nsides = 0;
                cuts.push_back(a0);
                for (int32_t k = a0; k < a1; ++k) {
                    const int32_t j = member[poff[q] + k];
                    int32_t sk = 0;
                    for (int32_t c = t.child_off[j]; c < t.child_off[j + 1]; ++c)
                        if (t.child[c] != t.main_child[j] && !is_long[t.child[c]]) ++sk;
                    if (k > s0 && (nrows + 1 > p.spine_cap || nsides + sk > p.side_cap)) {
                        cuts.push_back(k); s0 = k; nrows = 0; nsides = 0;
                    }
                    ++nrows; nsides += sk;
                }
            }
            cuts.push_back(len);
            int32_t link_u = -1, prev_last = -1;
            for (size_t cseg = 0; cseg + 1 < cuts.size(); ++cseg) {
                const int32_t s0 = cuts[cseg], s1 = cuts[cseg + 1];
                const bool new_block = link_u < 0 || units[link_u].link_len == p.link_cap;
                if (new_block) {
                    // LINK tasks cover blocks of consecutive segments and are chained along the path
                    link_u = (int32_t)units.size();
                    units.push_back(mk(-1, TASK_LINK));
                    units[link_u].link_off = (int32_t)link_reach.size();
                }
                units[link_u].link_len += 1;
                const int32_t g = (int32_t)g_begin.size();
                g_begin.push_back((int32_t)rows.size()); g_len.push_back(s1 - s0);
                const int32_t up = (int32_t)units.size();
                units.push_back(mk(g, TASK_PRE));
                units.push_back(mk(g, TASK_FIX));
                units[up].side_off = n_side;
                std::vector<uint32_t> late;
                for (int32_t k = s0; k < s1; ++k) {
                    const int32_t j = member[poff[q] + k];
                    pre_unit[j] = up;
                    uint32_t h = 0, n_early = 0, n_first = 0;
                    const int32_t m = t.main_child[j];
                    if (k > s0) h |= HDR_ACC;
                    else if (m >= 0) { units[up + 1].ins.push_back(INW_ROW | (uint32_t)m); ++n_first; }
                    for (int32_t c = t.child_off[j]; c < t.child_off[j + 1]; ++c) {
                        const int32_t ch = t.child[c];
                        if (ch == m) continue;
                        if (is_long[ch]) {
                            if (k != s0) { err = "internal: long tributary inside a segment"; return false; }
                            units[up + 1].ins.push_back(INW_ROW | (uint32_t)ch); ++n_first;
                            late.push_back(INW_ROW | (uint32_t)ch);
                        } else { units[up].ins.push_back(INW_ROW | (uint32_t)ch); ++n_early; push_of[ch] = n_side++; }
                    }
                    if (n_early >= (1u << 13) || n_first >= (1u << 13)) { err = "confluence too wide"; return false; }
                    rows.push_back(j);
                    rhdr.push_back(h | (n_early << 6) | (n_first << 19));
                }
                const int32_t last = member[poff[q] + s1 - 1];
                final_unit[last] = link_u;
                link_reach.push_back(last);
                Unit& L = units[link_u];
                // a block's first record also takes the outflow of the previous block's last reach
                if (new_block && prev_last >= 0) late.insert(late.begin(), INW_ROW | (uint32_t)prev_last);
                L.ins.push_back(INW_ROW | (uint32_t)last);
                L.ins.push_back((uint32_t)late.size());
                L.ins.insert(L.ins.end(), late.begin(), late.end());
                prev_last = last;
            }
        }
    }
    n_spine = (int32_t)g_begin.size();

    // ---- pockets: side subtrees made of short paths only -------------------------------
    // split oversized pockets bottom-up; `closed[j]` marks roots of mini-trees
    std::vector<int32_t> open(n, 0), need(n, 0);
    std::vector<uint8_t> closed(n, 0);
    {
        std::vector<std::pair<int32_t, int32_t>> kids;
        for (int32_t j : t.topo) {
            if (is_long[j]) continue;
            int32_t total = 1;
            kids.clear();
            for (int32_t c = t.child_off[j]; c < t.child_off[j + 1]; ++c) {
                const int32_t ch = t.child[c];
                if (!closed[ch]) { kids.emplace_back(open[ch], ch); total += open[ch]; }
            }
            if (total > p.pocket_cap) {
                std::sort(kids.begin(), kids.end(), [](auto& a, auto& b) {
                    return a.first != b.first ? a.first > b.first : a.second < b.second; });
                for (auto& kv : kids) {
                    if (total <= p.pocket_cap) break;
                    closed[kv.second] = 1; total -= kv.first;
                }
            }
            open[j] = total;
            if (t.end[j] == j || is_long[t.end[j]]) closed[j] = 1;      // pocket root
        }
        // Sethi-Ullman scratch need over in-tree children
        std::vector<int32_t> nd;
        for (int32_t j : t.topo) {
            if (is_long[j]) continue;
            nd.clear();
            for (int32_t c = t.child_off[j]; c < t.child_off[j + 1]; ++c)
                if (!closed[t.child[c]]) nd.push_back(need[t.child[c]]);
            std::sort(nd.begin(), nd.end(), std::greater<int32_t>());
            int32_t v = 0;
            for (size_t i = 0; i < nd.size(); ++i) v = std::max(v, nd[i] + (int32_t)i);
            need[j] = v;
        }
    }
    // mini-tree roots and their bundling keys
    struct Mini { int64_t key; int32_t root; };
    std::vector<Mini> grpA, grpB, grpC;      // feeds a spine / isolated / feeds another mini-tree
    for (int64_t j = 0; j < n; ++j) {
        if (is_long[j] || !closed[j]) continue;
        const int32_t d = t.end[j];
        if (d == j) grpB.push_back({(int64_t)j, (int32_t)j});
        else if (is_long[d]) grpA.push_back({((int64_t)pre_unit[d] << 32) | (uint32_t)t.path_pos[d], (int32_t)j});
        else grpC.push_back({(int64_t)j, (int32_t)j});
    }
    auto by_key = [](const Mini& a, const Mini& b) { return a.key != b.key ? a.key < b.key : a.root < b.root; };
    std::sort(grpA.begin(), grpA.end(), by_key);

    // DFS emission of one mini-tree into the current unit
    std::vector<int32_t> free_slots;
    int32_t slots_hi = 0;
    std::vector<int32_t> slot_of(n, -1);
    std::function<void(int32_t)> emit_tree = [&](int32_t v) {
        std::vector<std::pair<int32_t, int32_t>> kids;     // (need, child) of in-tree children
        for (int32_t c = t.child_off[v]; c < t.child_off[v + 1]; ++c)
            if (!closed[t.child[c]]) kids.emplace_back(need[t.child[c]], t.child[c]);
        std::sort(kids.begin(), kids.end(), [](auto& a, auto& b) {
            return a.first != b.first ? a.first > b.first : a.second < b.second; });
        for (size_t i = 0; i < kids.size(); ++i) {
            emit_tree(kids[i].second);
            if (i + 1 < kids.size()) {
                // park the child's outflow: patch its header with a scratch slot if one is free
                const int32_t c = kids[i].second;
                if (!free_slots.empty()) {
                    const int32_t s = free_slots.back(); free_slots.pop_back();
                    slot_of[c] = s;
                    slots_hi = std::max(slots_hi, s + 1);
                    rhdr.back() |= (uint32_t)(s + 1) << 1;     // c is the reach just emitted
                } else {
                    row_fallbacks += 1;
                }
            }
        }
        Unit& u = units.back();
        uint32_t h = 0, nin = 0;
        if (!kids.empty()) h |= HDR_ACC;                       // last in-tree child was emitted just before v
        for (size_t i = 0; i + 1 < kids.size(); ++i) {
            const int32_t c = kids[i].second;
            if (slot_of[c] >= 0) { u.ins.push_back((uint32_t)slot_of[c]); free_slots.push_back(slot_of[c]); slot_of[c] = -1; }
            else u.ins.push_back(INW_ROW | (uint32_t)c);
            ++nin;
        }
        for (int32_t c = t.child_off[v]; c < t.child_off[v + 1]; ++c)
            if (closed[t.child[c]]) { u.ins.push_back(INW_ROW | (uint32_t)t.child[c]); ++nin; }
        if (push_of[v] >= 0) { h |= HDR_PUSH; u.ins.push_back((uint32_t)push_of[v]); }
        final_unit[v] = (int32_t)units.size() - 1;
        rows.push_back(v);
        rhdr.push_back(h | (nin << 6));
    };
    auto reset_slots = [&]() {
        free_slots.clear();
        for (int32_t s = p.max_slots - 1; s >= 0; --s) free_slots.push_back(s);
    };
    auto pack = [&](const std::vector<Mini>& grp, bool bundle, bool same_high_key) {
        int32_t cur = -1, cur_size = 0; int64_t cur_hi = -1;
        for (const Mini& m : grp) {
            const int32_t sz = open[m.root];
            const int64_t hi = m.key >> 32;
            const bool fits = bundle && cur >= 0 && cur_size + sz <= p.pocket_cap &&
                              (!same_high_key || hi == cur_hi);
            if (!fits) {
                cur = (int32_t)g_begin.size();
                g_begin.push_back((int32_t)rows.size()); g_len.push_back(0);
                units.push_back(mk(cur, TASK_POCKET));
                cur_size = 0; cur_hi = hi;
            }
            reset_slots();
            emit_tree(m.root);
            cur_size += sz;
            g_len[cur] = (int32_t)rows.size() - g_begin[cur];
        }
    };
    pack(grpC, false, false);
    pack(grpA, true, true);
    pack(grpB, true, false);
    n_pocket = (int32_t)g_begin.size() - n_spine;
    slots_used = slots_hi;
    if ((int64_t)rows.size() != n) { err = "internal: schedule does not cover every reach"; return false; }

    // ---- dependencies ------------------------------------------------------------------------
    // Who finalises a row at step s, and who is the first to overwrite it at step s+1:
    //   pocket row           : its pocket task / the same task
    //   last row of a segment: the path's LINK / the segment's PRE
    // (other spine rows are only ever read by their own segment's tasks.)
    const int32_t nu = (int32_t)units.size();
    // U reads row c (a pocket root or the last row of a segment) at step s
    auto reads_row = [&](int32_t u, int32_t c) {
        Unit& U = units[u];
        if (pre_unit[c] < 0) {
            const int32_t prod = final_unit[c];
            if (units[prod].grp == U.grp) return;                          // a row of this task itself (slot fallback)
            U.A.push_back(prod);
            units[prod].B.push_back(u);                                    // the pocket rewrites the row next step
        } else {
            U.A.push_back(final_unit[c]);                                  // final once its path's LINK has run
            units[pre_unit[c]].B.push_back(u);                             // ... rewritten by that segment's PRE
        }
    };
    for (int32_t u = 0; u < nu; ++u) {
        Unit& U = units[u];
        U.B.push_back(u);                                                  // self: one step in flight per task
        if (U.kind == TASK_PRE) U.B.push_back(u + 1);                      // rows are rewritten: own FIX must be done
        if (U.kind == TASK_FIX)                                            // its path's LINK (implies its own PRE)
            U.A.push_back(final_unit[rows[g_begin[U.grp] + g_len[U.grp] - 1]]);
        if (U.kind == TASK_LINK) {
            for (int32_t e = U.link_off; e < U.link_off + U.link_len; ++e) U.A.push_back(pre_unit[link_reach[e]]);
            size_t w = 0;
            while (w < U.ins.size()) {                                     // records: [last row][n_late][rows...]
                const uint32_t nl = U.ins[w + 1];
                w += 2;
                for (uint32_t q = 0; q < nl; ++q, ++w) reads_row(u, (int32_t)(U.ins[w] & ~INW_ROW));
            }
        } else {
            for (uint32_t x : U.ins)
                if (x & INW_ROW) reads_row(u, (int32_t)(x & ~INW_ROW));
        }
    }
    for (Unit& U : units) { sort_unique(U.A); sort_unique(U.B); }
    std::vector<std::vector<int32_t>> same(nu), next(nu);
    for (int32_t u = 0; u < nu; ++u) {
        for (int32_t a : units[u].A) same[a].push_back(u);
        for (int32_t b : units[u].B) next[b].push_back(u);
    }
    // topological order over the A-edges, longest remaining critical path first
    auto cost = [&](int32_t u) -> int64_t {
        if (units[u].kind == TASK_LINK) return 12 + 2 * units[u].link_len;
        const int32_t len = g_len[units[u].grp];
        return units[u].kind == TASK_FIX ? 12 + len / 2 : 24 + len;
    };
    std::vector<int32_t> order0; order0.reserve(nu);
    {
        std::vector<int32_t> pend(nu);
        for (int32_t u = 0; u < nu; ++u) { pend[u] = (int32_t)units[u].A.size(); if (!pend[u]) order0.push_back(u); }
        for (size_t k = 0; k < order0.size(); ++k)
            for (int32_t c : same[order0[k]]) if (--pend[c] == 0) order0.push_back(c);
        if ((int32_t)order0.size() != nu) { err = "internal: task graph has a cycle"; return false; }
    }
    std::vector<int64_t> cp(nu, 0);
    std::vector<int32_t> cpt(nu, 0);
    for (int32_t k = nu - 1; k >= 0; --k) {
        const int32_t u = order0[k];
        int64_t best = 0; int32_t bt = 0;
        for (int32_t c : same[u]) { if (cp[c] > best) best = cp[c]; if (cpt[c] > bt) bt = cpt[c]; }
        cp[u] = best + cost(u);
        cpt[u] = bt + 1;
    }
    cp_cost = 0; cp_tasks = 0;
    for (int32_t u = 0; u < nu; ++u) { cp_cost = std::max(cp_cost, cp[u]); cp_tasks = std::max(cp_tasks, cpt[u]); }
    std::vector<int32_t> order; order.reserve(nu);
    {
        auto cmp = [&](int32_t a, int32_t b) { return cp[a] != cp[b] ? cp[a] < cp[b] : a > b; };
        std::priority_queue<int32_t, std::vector<int32_t>, decltype(cmp)> pq(cmp);
        std::vector<int32_t> pend(nu);
        for (int32_t u = 0; u < nu; ++u) { pend[u] = (int32_t)units[u].A.size(); if (!pend[u]) pq.push(u); }
        while (!pq.empty()) {
            const int32_t u = pq.top(); pq.pop();
            order.push_back(u);
            for (int32_t c : same[u]) if (--pend[c] == 0) pq.push(c);
        }
    }
    std::vector<int32_t> rank(nu);
    for (int32_t k = 0; k < nu; ++k) rank[order[k]] = k;

    // ---- positions and device descriptors -------------------------------------------------
    pos_of_reach.assign(n, -1); reach_of_pos.assign(n, -1);
    hdr.assign(n, 0);
    {
        const int32_t ng = (int32_t)g_begin.size();
        std::vector<int32_t> gpos(ng, -1);
        int32_t pos = 0;
        for (int32_t k = 0; k < nu; ++k) {
            const int32_t g = units[order[k]].grp;
            if (g < 0 || gpos[g] >= 0) continue;
            gpos[g] = pos;
            for (int32_t e = g_begin[g]; e < g_begin[g] + g_len[g]; ++e, ++pos) {
                pos_of_reach[rows[e]] = pos; reach_of_pos[pos] = rows[e]; hdr[pos] = rhdr[e];
            }
        }
        tasks.assign(nu, TaskDesc{});
        inw.clear(); notify.clear(); init_ready.clear(); max_len = max_link_len = max_words = max_link_words = 0;
        link_last.resize(link_reach.size());
        for (size_t e = 0; e < link_reach.size(); ++e) link_last[e] = pos_of_reach[link_reach[e]];
        for (int32_t k = 0; k < nu; ++k) {
            const Unit& U = units[order[k]];
            TaskDesc& td = tasks[k];
            td.kind = U.kind;
            if (U.kind == TASK_LINK) { td.begin = U.link_off; td.len = U.link_len; }
            else { td.begin = gpos[U.grp]; td.len = g_len[U.grp]; }
            td.in_off = (int32_t)inw.size();
            td.side_off = U.side_off;
            if (U.kind != TASK_PRE)                                // PRE reads its inputs from the side buffer
                for (uint32_t x : U.ins) {
                    if (x & INW_ROW) x = INW_ROW | (uint32_t)pos_of_reach[x & ~INW_ROW];
                    inw.push_back(x);
                }
            td.nfy_off = (int32_t)notify.size();
            td.n_same = (int32_t)same[order[k]].size();
            td.n_next = (int32_t)next[order[k]].size();
            for (int32_t c : same[order[k]]) {
                if (rank[c] <= k) { err = "internal: producer ordered after consumer"; return false; }
                notify.push_back(rank[c]);
            }
            for (int32_t c : next[order[k]]) notify.push_back(rank[c]);
            td.n_words = (int32_t)inw.size() - td.in_off;
            if (U.kind == TASK_LINK) { max_link_len = std::max(max_link_len, td.len); max_link_words = std::max(max_link_words, td.n_words); }
            else { max_len = std::max(max_len, td.len); max_words = std::max(max_words, td.n_words); }
            td.need0 = (int32_t)U.A.size();
            td.need = (int32_t)(U.A.size() + U.B.size());
            if (td.need0 == 0) init_ready.push_back(k);
        }
    }

    // ---- window-mode tasks over the same groups -------------------------------------------
    // One task per row group.  Rows read across tasks travel through slots of a ring: every pocket
    // root read by another task, and the last row of every segment.
    {
        const int32_t ng = (int32_t)g_begin.size();
        std::vector<int32_t> grp_of(n, -1);
        for (int32_t g = 0; g < ng; ++g)
            for (int32_t e = g_begin[g]; e < g_begin[g] + g_len[g]; ++e) grp_of[rows[e]] = g;
        std::vector<int32_t> unit_pocket(ng, -1), unit_pre(ng, -1);
        for (int32_t u = 0; u < nu; ++u) {
            if (units[u].kind == TASK_POCKET) unit_pocket[units[u].grp] = u;
            if (units[u].kind == TASK_PRE) unit_pre[units[u].grp] = u;
        }
        std::vector<int32_t> slot_of_reach(n, -1);
        n_wslots = 0;
        auto slot_for = [&](int32_t c) { if (slot_of_reach[c] < 0) slot_of_reach[c] = n_wslots++; return slot_of_reach[c]; };
        struct WU { std::vector<uint32_t> words; std::vector<int32_t> prod, prod_in; int32_t n_in = 0, out_slot = -1, kind = 0; };
        std::vector<WU> wu(ng);
        std::vector<uint32_t> ghdr(rhdr);                                  // window headers, group-row order
        for (int32_t g = 0; g < ng; ++g) {
            WU& W = wu[g];
            if (unit_pocket[g] >= 0) {
                W.kind = WTASK_POCKET;
                const Unit& U = units[unit_pocket[g]];
                size_t w = 0;
                for (int32_t e = g_begin[g]; e < g_begin[g] + g_len[g]; ++e) {
                    const uint32_t h = rhdr[e];
                    const uint32_t nin = (h >> 6) & 0x1ffffffu;
                    for (uint32_t q = 0; q < nin; ++q, ++w) {
                        const uint32_t x = U.ins[w];
                        if (!(x & INW_ROW)) { W.words.push_back(x); continue; }
                        const int32_t c = (int32_t)(x & ~INW_ROW);
                        if (grp_of[c] == g) {                              // a row of this task (scratch fallback)
                            int32_t k = -1;
                            for (int32_t e2 = g_begin[g]; e2 < e; ++e2) if (rows[e2] == c) { k = e2 - g_begin[g]; break; }
                            if (k < 0) { err = "internal: own-row input not yet evaluated"; return false; }
                            W.words.push_back(WIN_OWN | (uint32_t)k);
                        } else {
                            W.words.push_back(WIN_SLOT | (uint32_t)slot_for(c));
                            W.prod.push_back(grp_of[c]);
                        }
                    }
                    if (h & HDR_PUSH) ++w;                                 // the dataflow side-buffer row: unused here
                }
                if (w != U.ins.size()) { err = "internal: pocket stream mismatch"; return false; }
            } else {
                W.kind = WTASK_SEG;
                const Unit& P = units[unit_pre[g]];
                const Unit& F = units[unit_pre[g] + 1];
                for (uint32_t x : F.ins) {                                 // rows entering the segment
                    const int32_t c = (int32_t)(x & ~INW_ROW);
                    W.words.push_back(WIN_SLOT | (uint32_t)slot_for(c));
                    W.prod_in.push_back(grp_of[c]);
                    ++W.n_in;
                }
                for (uint32_t x : P.ins) {                                 // pocket roots, in row order
                    const int32_t c = (int32_t)(x & ~INW_ROW);
                    W.words.push_back(WIN_SLOT | (uint32_t)slot_for(c));
                    W.prod.push_back(grp_of[c]);
                }
            }
            sort_unique(W.prod);
        }
        // a segment publishes its outflow only when some task reads it (every slot has exactly one reader)
        for (int32_t g = 0; g < ng; ++g)
            if (wu[g].kind == WTASK_SEG) wu[g].out_slot = slot_of_reach[rows[g_begin[g] + g_len[g] - 1]];
        // publishing rows: pocket rows with a slot get HDR_PUSH (+ the slot word after their inputs)
        for (int32_t g = 0; g < ng; ++g) {
            if (wu[g].kind != WTASK_POCKET) continue;
            std::vector<uint32_t> out;
            size_t w = 0;
            for (int32_t e = g_begin[g]; e < g_begin[g] + g_len[g]; ++e) {
                uint32_t h = rhdr[e] & ~HDR_PUSH;
                const uint32_t nin = (h >> 6) & 0x1ffffffu;
                for (uint32_t q = 0; q < nin; ++q) out.push_back(wu[g].words[w++]);
                if (slot_of_reach[rows[e]] >= 0) { h |= HDR_PUSH; out.push_back((uint32_t)slot_of_reach[rows[e]]); }
                ghdr[e] = h;
            }
            wu[g].words.swap(out);
        }
        // topological order over the producer edges, longest remaining chain first
        std::vector<std::vector<int32_t>> cons(ng);
        std::vector<std::vector<int32_t>> allprod(ng);
        for (int32_t g = 0; g < ng; ++g) {
            allprod[g] = wu[g].prod;
            allprod[g].insert(allprod[g].end(), wu[g].prod_in.begin(), wu[g].prod_in.end());
            sort_unique(allprod[g]);
            for (int32_t pr : allprod[g]) cons[pr].push_back(g);
        }
        std::vector<int64_t> wcp(ng, 0);
        std::vector<int32_t> wcpt(ng, 0), worder0;
        {
            std::vector<int32_t> pend(ng);
            for (int32_t g = 0; g < ng; ++g) { pend[g] = (int32_t)allprod[g].size(); if (!pend[g]) worder0.push_back(g); }
            for (size_t k = 0; k < worder0.size(); ++k)
                for (int32_t c : cons[worder0[k]]) if (--pend[c] == 0) worder0.push_back(c);
            if ((int32_t)worder0.size() != ng) { err = "internal: window task graph has a cycle"; return false; }
            for (int32_t k = ng - 1; k >= 0; --k) {
                const int32_t g = worder0[k];
                int64_t best = 0; int32_t bt = 0;
                for (int32_t c : cons[g]) { best = std::max(best, wcp[c]); bt = std::max(bt, wcpt[c]); }
                wcp[g] = best + 8 + g_len[g];
                wcpt[g] = bt + 1;
            }
        }
        std::vector<int32_t> worder; worder.reserve(ng);
        {
            // longest remaining chain first; among equals the lower task index
            auto cmp = [&](int32_t a, int32_t b) { return wcp[a] != wcp[b] ? wcp[a] < wcp[b] : a > b; };
            std::priority_queue<int32_t, std::vector<int32_t>, decltype(cmp)> pq(cmp);
            std::vector<int32_t> pend(ng);
            for (int32_t g = 0; g < ng; ++g) { pend[g] = (int32_t)allprod[g].size(); if (!pend[g]) pq.push(g); }
            while (!pq.empty()) {
                const int32_t g = pq.top(); pq.pop();
                worder.push_back(g);
                for (int32_t c : cons[g]) if (--pend[c] == 0) pq.push(c);
            }
        }
        std::vector<int32_t> wrank(ng);
        for (int32_t k = 0; k < ng; ++k) wrank[worder[k]] = k;
        wtasks.assign(ng, WTaskDesc{});
        whdr.assign(n, 0); winw.clear(); wprod.clear();
        w_max_len = w_max_words = w_max_prod = w_cp_tasks = w_n_own = 0;
        for (int32_t k = 0; k < ng; ++k) {
            const int32_t g = worder[k];
            const WU& W = wu[g];
            WTaskDesc& td = wtasks[k];
            td.begin = pos_of_reach[rows[g_begin[g]]]; td.len = g_len[g]; td.kind = W.kind;
            td.in_off = (int32_t)winw.size(); td.n_words = (int32_t)W.words.size();
            winw.insert(winw.end(), W.words.begin(), W.words.end());
            td.prod_off = (int32_t)wprod.size(); td.n_prod = (int32_t)(W.prod_in.size() + W.prod.size());
            for (const std::vector<int32_t>* lst : {&W.prod_in, &W.prod})
                for (int32_t pr : *lst) {
                    if (wrank[pr] >= k) { err = "internal: window producer ordered after consumer"; return false; }
                    wprod.push_back(wrank[pr]);
                }
            td.out_slot = W.out_slot; td.n_in = W.n_in;
            td.n_out = W.kind == WTASK_SEG ? 1 : 0;
            td.n_own = 0;
            for (uint32_t x : W.words) if (!(x & WIN_SLOT) && (x & WIN_OWN)) td.n_own += 1;
            w_n_own += td.n_own;
            if (W.kind == WTASK_POCKET)
                for (int32_t e = 0; e < g_len[g]; ++e) if (ghdr[g_begin[g] + e] & HDR_PUSH) td.n_out += 1;
            for (int32_t e = 0; e < g_len[g]; ++e) {
                if (pos_of_reach[rows[g_begin[g] + e]] != td.begin + e) { err = "internal: group rows not contiguous"; return false; }
                whdr[td.begin + e] = ghdr[g_begin[g] + e];
            }
            w_max_len = std::max(w_max_len, td.len); w_max_words = std::max(w_max_words, td.n_words);
            w_max_prod = std::max(w_max_prod, td.n_prod); w_cp_tasks = std::max(w_cp_tasks, wcpt[g]);
        }
    }

    // ---- position-space CSR of upstream rows + level lists -------------------------------
    up_off.assign(n + 1, 0); up_pos.resize(t.child.size());
    is_outlet_pos.assign(n, 0);
    for (int64_t q = 0; q < n; ++q) {
        const int32_t j = reach_of_pos[q];
        up_off[q + 1] = up_off[q] + (t.child_off[j + 1] - t.child_off[j]);
        int32_t w = up_off[q];
        for (int32_t c = t.child_off[j]; c < t.child_off[j + 1]; ++c) up_pos[w++] = pos_of_reach[t.child[c]];
        is_outlet_pos[q] = t.end[j] == j;
    }
    lvl_off.assign(t.level_off.begin(), t.level_off.end());
    lvl_pos.resize(n);
    for (int32_t l = 0; l < t.nlevels; ++l) {
        for (int32_t k = t.level_off[l]; k < t.level_off[l + 1]; ++k) lvl_pos[k] = pos_of_reach[t.topo[k]];
        std::sort(lvl_pos.begin() + t.level_off[l], lvl_pos.begin() + t.level_off[l + 1]);
    }
    return true;
}

}  // namespace txh

// ---------------------------------------------------------------------------
// Lane schedule (route_lane_kernel)
// ---------------------------------------------------------------------------
namespace txh {

size_t LaneSchedule::region_bytes(size_t real, size_t virt, size_t nchild, int mt)
{
    auto up16 = [](size_t x) { return (x + 15) & ~size_t(15); };
    return 16 * (size_t)mt * (real + virt + 1)   // outflows of this and the previous iteration (+ the zero row)
           + 256 * (size_t)mt * virt       // 32 steps of every incoming stream
           + 16 * virt                     // records of the virtual rows
           + up16(2 * nchild)              // children beyond the first two of a row
           + (mt > 4 ? up16(8 * (size_t)mt * real) : 0)    // p = beta i + chi o (in registers up to 4 members)
           + up16(8 * real);               // the forcing row after a row's bracket (cp.async target)
}

bool LaneSchedule::build(const Topology& t, const std::vector<int32_t>& pos_of_reach, int mt_, int cap_rows_,
                         size_t smem_budget_, int side_min, std::string& err)
{
    mt = mt_; cap_rows = cap_rows_; smem_budget = smem_budget_;
    side_min = std::max(2, side_min);
    const int64_t n = t.n;
    if (mt < 1 || mt > 16 || (mt & (mt - 1))) { err = "lane schedule: member tile must be 1, 2, 4, 8 or 16"; return false; }
    if (cap_rows < 1) { err = "lane schedule: bad row cap"; return false; }
    cap_rows = std::min(cap_rows, kLaneMaxRows);                            // one row per thread
    // weights in bytes: a real row with ~one child entry, a virtual row
    const int64_t wr = 16 * (int64_t)mt + (mt > 4 ? 8 * (int64_t)mt : 0) + 8 + 2, wv = 16 + 272 * (int64_t)mt + 2;
    const int64_t cap_bytes = (int64_t)smem_budget - 256;               // sentinel record, alignment of the parts
    if (wr + wv > cap_bytes) { err = "lane schedule: shared-memory budget too small"; return false; }

    // ---- clusters: greedy bottom-up cut of the forest into sub-trees that fit one CTA -------------------
    // The deepest child (the longest path continues through it) stays with its downstream reach as long as
    // the caps allow; side tributaries of `side_min` rows or more are always cut off -- they become clusters of
    // their own, bundled with others of the same height -- so that the chain of regions along a long path
    // (every link costs a trip through L2) stays short.
    std::vector<int64_t> open_w(n, 0);
    std::vector<int32_t> open_r(n, 0);
    std::vector<uint8_t> closed(n, 0);
    {
        std::vector<std::pair<int64_t, int32_t>> kids;
        for (int32_t j : t.topo) {
            int64_t W = wr; int32_t R = 1;
            kids.clear();
            const int32_t mainc = t.main_child[j];
            for (int32_t c = t.child_off[j]; c < t.child_off[j + 1]; ++c) {
                const int32_t ch = t.child[c];
                if (!closed[ch] && ch != mainc && open_r[ch] >= side_min) closed[ch] = 1;
                if (closed[ch]) W += wv;
                else { W += open_w[ch]; R += open_r[ch]; if (ch != mainc) kids.emplace_back(open_w[ch], ch); }
            }
            if (W > cap_bytes || R > cap_rows) {
                std::sort(kids.begin(), kids.end(), [](auto& a, auto& b) {
                    return a.first != b.first ? a.first > b.first : a.second < b.second; });
                if (mainc >= 0 && !closed[mainc]) kids.emplace_back(open_w[mainc], mainc);   // the path itself: last
                for (auto& kv : kids) {
                    if (W <= cap_bytes && R <= cap_rows) break;
                    closed[kv.second] = 1;
                    W -= kv.first - wv; R -= open_r[kv.second];
                }
                if (W > cap_bytes) { err = "lane schedule: a confluence is too wide for one region"; return false; }
            }
            open_w[j] = W; open_r[j] = R;
            if (t.end[j] == j) closed[j] = 1;
        }
    }
    // cluster of every reach, distance to the cluster's exit
    std::vector<int32_t> cl_of(n, -1), dist(n, 0), cl_root;
    for (int64_t k = n - 1; k >= 0; --k) {
        const int32_t j = t.topo[k];
        if (closed[j]) { cl_of[j] = (int32_t)cl_root.size(); cl_root.push_back(j); dist[j] = 0; }
        else { cl_of[j] = cl_of[t.end[j]]; dist[j] = dist[t.end[j]] + 1; }
    }
    const int32_t ncl = (int32_t)cl_root.size();
    // per cluster: rows, virtual rows, children entries, depth (virtual leaves included), height in the cluster graph
    std::vector<int32_t> cl_real(ncl, 0), cl_virt(ncl, 0), cl_child(ncl, 0), cl_depth(ncl, 0), cl_h(ncl, 0);
    for (int32_t j : t.topo) {                                              // upstream first: heights are final at the root
        const int32_t c = cl_of[j];
        cl_real[c] += 1;
        cl_child[c] += t.child_off[j + 1] - t.child_off[j];
        cl_depth[c] = std::max(cl_depth[c], dist[j]);
        for (int32_t e = t.child_off[j]; e < t.child_off[j + 1]; ++e) {
            const int32_t ch = t.child[e];
            if (!closed[ch]) continue;
            cl_virt[c] += 1;
            cl_depth[c] = std::max(cl_depth[c], dist[j] + 1);
            cl_h[c] = std::max(cl_h[c], cl_h[cl_of[ch]] + 1);
        }
    }
    // ---- regions: clusters of equal height bundled up to the caps; ticket order = height ascending ----------
    std::vector<int32_t> cl_order(ncl);
    std::iota(cl_order.begin(), cl_order.end(), 0);
    // among equal heights: deep clusters first (they pace their consumers), then by root id
    std::stable_sort(cl_order.begin(), cl_order.end(), [&](int32_t a, int32_t b) {
        if (cl_h[a] != cl_h[b]) return cl_h[a] < cl_h[b];
        if (cl_depth[a] != cl_depth[b]) return cl_depth[a] > cl_depth[b];
        return cl_root[a] < cl_root[b]; });
    std::vector<int32_t> reg_of_cl(ncl, -1);
    std::vector<std::vector<int32_t>> reg_cls;
    {
        size_t real = 0, virt = 0, nch = 0; int32_t cur_h = -1;
        for (int32_t c : cl_order) {
            const bool fits = !reg_cls.empty() && cl_h[c] == cur_h && real + cl_real[c] <= (size_t)cap_rows &&
                              real + virt + cl_real[c] + cl_virt[c] < 65000 &&
                              region_bytes(real + cl_real[c], virt + cl_virt[c], nch + cl_child[c], mt) <= smem_budget;
            if (!fits) {
                reg_cls.emplace_back(); real = virt = nch = 0; cur_h = cl_h[c];
                if (region_bytes(cl_real[c], cl_virt[c], cl_child[c], mt) > smem_budget) {
                    err = "lane schedule: a cluster exceeds the shared-memory budget"; return false;
                }
            }
            reg_cls.back().push_back(c);
            reg_of_cl[c] = (int32_t)reg_cls.size() - 1;
            real += cl_real[c]; virt += cl_virt[c]; nch += cl_child[c];
        }
    }
    // ---- slots: one stream per cluster root that drains into another cluster -------------------------------
    std::vector<int32_t> slot_of(n, -1);
    n_slots = 0;
    for (int32_t c = 0; c < ncl; ++c) {
        const int32_t r = cl_root[c];
        if (t.end[r] != r) slot_of[r] = n_slots++;
    }
    // ---- rows of every region ---------------------------------------------------------------------------
    const int32_t nreg = (int32_t)reg_cls.size();
    std::vector<std::vector<int32_t>> reg_rows(nreg);
    for (int64_t j = 0; j < n; ++j) reg_rows[reg_of_cl[cl_of[j]]].push_back((int32_t)j);
    regions.assign(nreg, LaneRegionDesc{});
    row_reach.clear(); row_off.clear(); row_c01.clear(); row_nx.clear(); row_xbeg.clear(); row_slot.clear(); child.clear();
    max_real = max_virt = max_child = max_extra = 0;
    max_bytes = 0;
    std::vector<int32_t> local(n, -1), off_of(n, 0);
    for (int32_t g = 0; g < nreg; ++g) {
        std::vector<int32_t>& rows = reg_rows[g];
        for (int32_t j : rows) off_of[j] = cl_depth[cl_of[j]] - dist[j];
        std::sort(rows.begin(), rows.end(), [&](int32_t a, int32_t b) {
            const bool xa = t.child_off[a + 1] - t.child_off[a] > 2, xb = t.child_off[b + 1] - t.child_off[b] > 2;
            if (xa != xb) return xb;                                        // rows with further children last
            if (off_of[a] != off_of[b]) return off_of[a] < off_of[b];
            return pos_of_reach[a] < pos_of_reach[b]; });
        LaneRegionDesc& rd = regions[g];
        rd.row_off = (int32_t)row_reach.size();
        rd.n_real = (int32_t)rows.size();
        rd.child_off = (int32_t)child.size();
        rd.height = cl_h[reg_cls[g].front()];
        for (int32_t i = 0; i < rd.n_real; ++i) local[rows[i]] = i;
        // virtual rows: one per upstream reach that belongs to another cluster, in consumer-row order
        int32_t nv = 0, extra = 0;
        for (int32_t i = 0; i < rd.n_real; ++i)
            for (int32_t e = t.child_off[rows[i]]; e < t.child_off[rows[i] + 1]; ++e) if (closed[t.child[e]]) ++nv;
        rd.n_virt = nv;
        const int32_t zero_row = rd.n_real + nv;
        std::vector<int32_t> v_off, v_slot;
        int32_t vcount = 0;
        for (int32_t i = 0; i < rd.n_real; ++i) {
            const int32_t j = rows[i];
            const int32_t off = off_of[j];
            extra = std::max(extra, off + 1);
            int32_t c01[2] = {zero_row, zero_row};
            int32_t k = 0, nx = 0;
            const int32_t xbeg = (int32_t)child.size() - rd.child_off;
            for (int32_t e = t.child_off[j]; e < t.child_off[j + 1]; ++e, ++k) {
                const int32_t ch = t.child[e];
                int32_t idx;
                if (!closed[ch]) idx = local[ch];
                else { idx = rd.n_real + vcount++; v_off.push_back(off - 1); v_slot.push_back(slot_of[ch]); }
                if (k < 2) c01[k] = idx;
                else { child.push_back((uint16_t)idx); ++nx; }
            }
            row_reach.push_back(j); row_off.push_back(off);
            row_c01.push_back(c01[0] | (c01[1] << 16));
            row_nx.push_back(nx); row_xbeg.push_back(xbeg); row_slot.push_back(slot_of[j]);
        }
        rd.n_child = (int32_t)child.size() - rd.child_off;
        for (int32_t v = 0; v < nv; ++v) {
            if (v_off[v] < 0) { err = "internal: lane skew offset below zero"; return false; }
            row_reach.push_back(-1); row_off.push_back(v_off[v]); row_c01.push_back(zero_row | (zero_row << 16));
            row_nx.push_back(0); row_xbeg.push_back(0); row_slot.push_back(v_slot[v]);
        }
        rd.n_extra = extra;
        max_real = std::max(max_real, rd.n_real); max_virt = std::max(max_virt, rd.n_virt);
        max_child = std::max(max_child, rd.n_child); max_extra = std::max(max_extra, rd.n_extra);
        const size_t bytes = region_bytes(rd.n_real, rd.n_virt, rd.n_child, mt);
        max_bytes = std::max(max_bytes, bytes);
        if (bytes > smem_budget || zero_row >= 65535) { err = "internal: lane region over budget"; return false; }
    }
    return true;
}

}  // namespace txh
