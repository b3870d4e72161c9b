// lu_symbolic.h -- symbolic analysis of the sparse LU of one inner block (plain C++17, host, set-up time only).
//
// Works on the pattern of B + B^T (Dirichlet rows make the blocks structurally nonsymmetric):
//   1. rows with identical closed adjacency are compressed into one vertex (the node-blocked dofs of s / f / fp);
//   2. nested dissection of the compressed graph: recursive bisection by BFS level structures from a pseudo-peripheral
//      vertex, the middle level trimmed to the vertices that touch both sides is the separator, leaves of <= kLeaf rows;
//   3. elimination tree, postorder, fundamental supernodes, relaxed amalgamation (the explicit zeros it stores are counted);
//   4. per supernode: the front's row list (pivot columns, then the update rows), the relative positions of its update rows
//      in the parent's front (extend-add), and for every nonzero of the block its position in a front;
//   5. a level schedule of the supernodal tree, leaves first.
// Used by sparse_lu.cu and, through tests/lu_symbolic_harness.cpp, by the CPU tests.
#pragma once
#include <algorithm>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

namespace poro {
namespace lusym {

constexpr int kLeaf = 128;   // nested dissection stops at about this many rows

struct Symbolic {
    int n = 0;
    std::vector<int> perm;            // perm[new] = old
    std::vector<int> iperm;           // iperm[old] = new
    // supernodes (numbered in postorder, pivot columns [first[s], first[s + 1]) of the permuted block)
    int nsuper = 0;
    std::vector<int> first;           // nsuper + 1
    std::vector<int> m;               // front rows: k = first[s+1] - first[s] pivot rows, then m - k update rows
    std::vector<int> parent;          // -1 at a root
    std::vector<int64_t> row_ptr;     // front row lists: row_idx[row_ptr[s] .. row_ptr[s] + m[s])
    std::vector<int> row_idx;
    std::vector<int> child_ptr, child;   // children of each supernode, ascending (the fixed extend-add order)
    std::vector<int> relmap;          // per supernode, its update rows' positions in the parent's front (indexed like upd_off)
    std::vector<int64_t> upd_off;     // nsuper + 1: offsets of the update rows (sum of m - k)
    std::vector<int64_t> front_off;   // nsuper + 1: dense m x m fronts, column-major (sum of m^2)
    std::vector<int64_t> fac_off;     // nsuper + 1: stored factor, k^2 + 2 k (m - k) per supernode
    std::vector<int64_t> nz_pos;      // per nonzero of the block (CSR order): position inside the fronts
    int nlevels = 0;
    std::vector<int> level_ptr, level_sn;   // supernodes of level l: level_sn[level_ptr[l] .. level_ptr[l+1]), leaves first
    // statistics
    int64_t nnz_l = 0, nnz_u = 0;     // stored entries: L strictly lower (unit diagonal implied), U with its diagonal
    int64_t amalg_zeros = 0;          // stored entries that the exact structure does not have
    int max_front = 0;
    double flops = 0.0;               // of the numeric factorisation (divisions + 2 per multiply-add)
};

namespace detail {

// trapezoid of a supernode with k pivot columns and m front rows: k^2 + 2 k (m - k) entries of L + U
inline int64_t stored(int64_t k, int64_t m) { return 2 * m * k - k * k; }

struct Graph {
    std::vector<int64_t> ptr;
    std::vector<int> adj;
    std::vector<int> w;               // rows per vertex
};

// nested dissection of the vertices `vs` of g; appends the elimination order to `order`
class Dissector {
  public:
    explicit Dissector(const Graph& g) : g_(g), mark_(g.w.size(), 0), lev_(g.w.size(), 0) {}
    void run(const std::vector<int>& vs, std::vector<int>& order) { recurse(vs, order, 0); }

  private:
    const Graph& g_;
    std::vector<int> mark_, lev_;     // part id of a vertex; BFS stamp (negative) of a vertex
    int stamp_ = 0, uid_ = 0;

    int64_t weight(const std::vector<int>& vs) const {
        int64_t s = 0;
        for (int v : vs) s += g_.w[v];
        return s;
    }
    // BFS inside the part marked `id` from r: fills lev_, returns the level sets
    std::vector<std::vector<int>> bfs(int r, int id) {
        std::vector<std::vector<int>> L;
        const int seen = --stamp_;        // negative stamps: visited in this BFS
        std::vector<int> cur{r};
        lev_[r] = seen;
        while (!cur.empty()) {
            L.push_back(cur);
            std::vector<int> nxt;
            for (int v : cur)
                for (int64_t q = g_.ptr[v]; q < g_.ptr[v + 1]; ++q) {
                    const int u = g_.adj[q];
                    if (mark_[u] == id && lev_[u] != seen) { lev_[u] = seen; nxt.push_back(u); }
                }
            cur.swap(nxt);
        }
        return L;
    }
    int degree_in(int v, int id) const {
        int d = 0;
        for (int64_t q = g_.ptr[v]; q < g_.ptr[v + 1]; ++q) d += mark_[g_.adj[q]] == id;
        return d;
    }
    void recurse(const std::vector<int>& vs, std::vector<int>& order, int depth) {
        if (vs.empty()) return;
        if (weight(vs) <= kLeaf || depth > 200) { order.insert(order.end(), vs.begin(), vs.end()); return; }
        const int part_id = ++uid_;
        for (int v : vs) mark_[v] = part_id;
        // pseudo-peripheral vertex: repeated BFS from a vertex of minimum degree in the last level
        int r = vs[0];
        auto L = bfs(r, part_id);
        size_t reached = 0;
        for (auto& l : L) reached += l.size();
        if (reached < vs.size()) {
            // disconnected: this component and the rest are independent (empty separator)
            std::vector<int> a, b;
            const int seen = lev_[r];
            for (int v : vs) (lev_[v] == seen ? a : b).push_back(v);
            recurse(a, order, depth + 1);
            recurse(b, order, depth + 1);
            return;
        }
        for (int it = 0; it < 8; ++it) {
            const auto& last = L.back();
            int best = last[0], bd = degree_in(best, part_id);
            for (int v : last) { int d = degree_in(v, part_id); if (d < bd) { bd = d; best = v; } }
            auto L2 = bfs(best, part_id);
            if (L2.size() <= L.size()) break;
            L.swap(L2);
            r = best;
        }
        if (L.size() < 3) { order.insert(order.end(), vs.begin(), vs.end()); return; }
        const int64_t total = weight(vs);
        int64_t acc = 0;
        size_t mid = 1;
        for (size_t l = 0; l < L.size(); ++l) {
            acc += weight(L[l]);
            if (2 * acc >= total) { mid = l; break; }
        }
        mid = std::max<size_t>(1, std::min(mid, L.size() - 2));
        const int sid = ++uid_, aid = ++uid_, bid = ++uid_;
        for (size_t l = 0; l < L.size(); ++l)
            for (int v : L[l]) mark_[v] = l < mid ? aid : (l == mid ? sid : bid);
        std::vector<int> A, B, S;
        for (size_t l = 0; l < L.size(); ++l) {
            if (l < mid) A.insert(A.end(), L[l].begin(), L[l].end());
            else if (l > mid) B.insert(B.end(), L[l].begin(), L[l].end());
        }
        // trim: a separator vertex without a neighbour on the far side joins the near side
        for (int v : L[mid]) {
            bool far = false;
            for (int64_t q = g_.ptr[v]; q < g_.ptr[v + 1] && !far; ++q) far = mark_[g_.adj[q]] == bid;
            if (far) S.push_back(v); else A.push_back(v);
        }
        if (B.empty() || S.empty()) { order.insert(order.end(), vs.begin(), vs.end()); return; }
        std::sort(A.begin(), A.end());
        std::sort(B.begin(), B.end());
        recurse(A, order, depth + 1);
        recurse(B, order, depth + 1);
        order.insert(order.end(), S.begin(), S.end());
    }
};

}  // namespace detail

// pattern of the n x n block (CSR, columns in [0, n))
inline Symbolic analyse(int n, const int64_t* rowptr, const int* col) {
    using namespace detail;
    Symbolic S;
    S.n = n;
    // ---- adjacency of B + B^T without the diagonal ----
    std::vector<int64_t> deg((size_t)n + 1, 0);
    for (int i = 0; i < n; ++i)
        for (int64_t q = rowptr[i]; q < rowptr[i + 1]; ++q) {
            const int j = col[q];
            if (j < 0 || j >= n) throw std::runtime_error("sparse LU: column index out of range");
            if (j != i) { deg[i + 1]++; deg[j + 1]++; }
        }
    for (int i = 0; i < n; ++i) deg[i + 1] += deg[i];
    std::vector<int> adj((size_t)deg[n]);
    {
        std::vector<int64_t> pos(deg.begin(), deg.end() - 1);
        for (int i = 0; i < n; ++i)
            for (int64_t q = rowptr[i]; q < rowptr[i + 1]; ++q) {
                const int j = col[q];
                if (j != i) { adj[pos[i]++] = j; adj[pos[j]++] = i; }
            }
    }
    Graph G;                          // deduplicated, sorted
    G.ptr.assign((size_t)n + 1, 0);
    for (int i = 0; i < n; ++i) {
        auto b = adj.begin() + deg[i], e = adj.begin() + deg[i + 1];
        std::sort(b, e);
        e = std::unique(b, e);
        G.ptr[i + 1] = G.ptr[i] + (e - b);
    }
    G.adj.resize((size_t)G.ptr[n]);
    for (int i = 0; i < n; ++i) {
        auto b = adj.begin() + deg[i];
        std::copy(b, b + (G.ptr[i + 1] - G.ptr[i]), G.adj.begin() + G.ptr[i]);
    }
    adj.clear(); adj.shrink_to_fit();
    // ---- compression: rows with identical closed adjacency ----
    std::vector<int> sv((size_t)n, -1), rep;       // vertex -> compressed vertex, compressed vertex -> representative row
    std::vector<std::vector<int>> members;
    {
        std::unordered_map<uint64_t, std::vector<int>> buckets;
        auto closed = [&](int i) {
            std::vector<int> c(G.adj.begin() + G.ptr[i], G.adj.begin() + G.ptr[i + 1]);
            c.insert(std::lower_bound(c.begin(), c.end(), i), i);
            return c;
        };
        for (int i = 0; i < n; ++i) {
            uint64_t h = 1469598103934665603ull;
            uint64_t s = (uint64_t)i;
            for (int64_t q = G.ptr[i]; q < G.ptr[i + 1]; ++q) s += (uint64_t)G.adj[q];
            h = (h ^ s) * 1099511628211ull;
            h = (h ^ (uint64_t)(G.ptr[i + 1] - G.ptr[i])) * 1099511628211ull;
            auto& bk = buckets[h];
            const auto ci = closed(i);
            int found = -1;
            for (int c : bk) if (closed(rep[c]) == ci) { found = c; break; }
            if (found < 0) { found = (int)rep.size(); rep.push_back(i); members.emplace_back(); bk.push_back(found); }
            sv[i] = found;
            members[found].push_back(i);
        }
    }
    const int nc = (int)rep.size();
    Graph C;
    C.w.resize((size_t)nc);
    C.ptr.assign((size_t)nc + 1, 0);
    for (int v = 0; v < nc; ++v) {
        C.w[v] = (int)members[v].size();
        const int r = rep[v];
        std::vector<int> nb;
        for (int64_t q = G.ptr[r]; q < G.ptr[r + 1]; ++q) if (sv[G.adj[q]] != v) nb.push_back(sv[G.adj[q]]);
        std::sort(nb.begin(), nb.end());
        nb.erase(std::unique(nb.begin(), nb.end()), nb.end());
        C.adj.insert(C.adj.end(), nb.begin(), nb.end());
        C.ptr[v + 1] = (int64_t)C.adj.size();
    }
    // ---- nested dissection ----
    std::vector<int> corder;
    {
        std::vector<int> all((size_t)nc);
        for (int v = 0; v < nc; ++v) all[v] = v;
        Dissector(C).run(all, corder);
    }
    std::vector<int> perm;
    perm.reserve((size_t)n);
    for (int v : corder) perm.insert(perm.end(), members[v].begin(), members[v].end());
    if ((int)perm.size() != n) throw std::runtime_error("sparse LU: nested dissection lost rows");
    // ---- elimination tree (Liu) + postorder ----
    auto etree = [&](const std::vector<int>& pm, std::vector<int>& par) {
        std::vector<int> ip((size_t)n), anc((size_t)n, -1);
        for (int k = 0; k < n; ++k) ip[pm[k]] = k;
        par.assign((size_t)n, -1);
        for (int i = 0; i < n; ++i) {
            const int o = pm[i];
            for (int64_t q = G.ptr[o]; q < G.ptr[o + 1]; ++q) {
                int r = ip[G.adj[q]];
                if (r >= i) continue;
                while (anc[r] != -1 && anc[r] != i) { const int t = anc[r]; anc[r] = i; r = t; }
                if (anc[r] == -1) { anc[r] = i; par[r] = i; }
            }
        }
    };
    std::vector<int> par;
    etree(perm, par);
    {
        std::vector<int> head((size_t)n, -1), next((size_t)n, -1), post;
        post.reserve((size_t)n);
        for (int j = n - 1; j >= 0; --j) if (par[j] >= 0) { next[j] = head[par[j]]; head[par[j]] = j; }   // ascending children
        std::vector<int> stack;
        for (int r = 0; r < n; ++r) {
            if (par[r] >= 0) continue;
            stack.push_back(r);
            while (!stack.empty()) {
                const int v = stack.back();
                if (head[v] >= 0) { const int c = head[v]; head[v] = next[c]; stack.push_back(c); }
                else { stack.pop_back(); post.push_back(v); }
            }
        }
        std::vector<int> p2((size_t)n);
        for (int k = 0; k < n; ++k) p2[k] = perm[post[k]];
        perm.swap(p2);
    }
    etree(perm, par);
    S.perm = perm;
    S.iperm.assign((size_t)n, 0);
    for (int k = 0; k < n; ++k) S.iperm[perm[k]] = k;
    const std::vector<int>& ip = S.iperm;
    // ---- column structures (kept for the last column of each fundamental supernode) ----
    std::vector<int> nchild((size_t)n, 0), cc((size_t)n, 0);
    for (int j = 0; j < n; ++j) if (par[j] >= 0) nchild[par[j]]++;
    std::vector<int> chead((size_t)n, -1), cnext((size_t)n, -1);
    for (int j = n - 1; j >= 0; --j) if (par[j] >= 0) { cnext[j] = chead[par[j]]; chead[par[j]] = j; }
    std::vector<std::vector<int>> st((size_t)n);
    std::vector<int> mark((size_t)n, -1);
    std::vector<char> linked((size_t)n, 0);       // column j and j + 1 are in one fundamental supernode
    int64_t true_entries = 0;
    for (int j = 0; j < n; ++j) {
        std::vector<int>& s = st[j];
        mark[j] = j;
        const int o = perm[j];
        for (int64_t q = G.ptr[o]; q < G.ptr[o + 1]; ++q) {
            const int i = ip[G.adj[q]];
            if (i > j && mark[i] != j) { mark[i] = j; s.push_back(i); }
        }
        for (int c = chead[j]; c >= 0; c = cnext[c])
            for (int i : st[c]) if (mark[i] != j) { mark[i] = j; s.push_back(i); }
        std::sort(s.begin(), s.end());
        cc[j] = (int)s.size();
        true_entries += 2 * (int64_t)cc[j] + 1;
        if (j > 0 && par[j - 1] == j && nchild[j] == 1 && cc[j - 1] == cc[j] + 1) {
            linked[j - 1] = 1;
            std::vector<int>().swap(st[j - 1]);    // not a last column: only its parent needed it
        }
    }
    // fundamental supernodes
    std::vector<int> ffirst, flast;
    for (int j = 0; j < n; ++j) {
        if (j == 0 || !linked[j - 1]) ffirst.push_back(j);
        if (!linked[j]) flast.push_back(j);
    }
    const int nf = (int)ffirst.size();
    std::vector<int> fsn_of((size_t)n);
    for (int s = 0; s < nf; ++s) for (int j = ffirst[s]; j <= flast[s]; ++j) fsn_of[j] = s;
    std::vector<int> fpar((size_t)nf, -1);
    for (int s = 0; s < nf; ++s) if (par[flast[s]] >= 0) fpar[s] = fsn_of[par[flast[s]]];
    // ---- relaxed amalgamation: a supernode absorbs the child whose columns immediately precede its own ----
    std::vector<int> gfirst(ffirst), gk((size_t)nf), gu((size_t)nf), grep((size_t)nf);
    std::vector<int64_t> gtrue((size_t)nf);
    for (int s = 0; s < nf; ++s) {
        gk[s] = flast[s] - ffirst[s] + 1;
        gu[s] = cc[flast[s]];
        gtrue[s] = stored(gk[s], gk[s] + gu[s]);
        grep[s] = s;
    }
    auto find = [&](int s) { while (grep[s] != s) { grep[s] = grep[grep[s]]; s = grep[s]; } return s; };
    for (int s = 0; s < nf; ++s) {
        if (fpar[s] < 0) continue;
        const int p = find(fpar[s]);
        if (flast[s] + 1 != gfirst[p]) continue;
        const int64_t k = (int64_t)gk[s] + gk[p], mm = k + gu[p];
        const int64_t st_m = stored(k, mm), z = st_m - gtrue[s] - gtrue[p];
        const bool merge = (k <= 16 && 4 * z <= st_m) || 20 * z <= st_m;
        if (!merge) continue;
        grep[s] = p;
        gfirst[p] = gfirst[s];
        gk[p] = (int)k;
        gtrue[p] += gtrue[s];
    }
    // final supernodes: the surviving groups in column order
    std::vector<int> sn_of_group((size_t)nf, -1);
    int ns = 0;
    for (int s = 0; s < nf; ++s) if (grep[s] == s) sn_of_group[s] = ns++;
    S.nsuper = ns;
    S.first.assign((size_t)ns + 1, n);
    S.m.assign((size_t)ns, 0);
    S.parent.assign((size_t)ns, -1);
    std::vector<int> last_col((size_t)ns);
    for (int s = 0; s < nf; ++s) {
        if (grep[s] != s) continue;
        const int t = sn_of_group[s];
        S.first[t] = gfirst[s];
        S.m[t] = gk[s] + gu[s];
        last_col[t] = flast[s];
        if (fpar[s] >= 0) S.parent[t] = sn_of_group[find(fpar[s])];
    }
    std::vector<int> sn_of((size_t)n);
    for (int t = 0; t < ns; ++t) for (int j = S.first[t]; j < S.first[t + 1]; ++j) sn_of[j] = t;
    // row lists
    S.row_ptr.assign((size_t)ns + 1, 0);
    for (int t = 0; t < ns; ++t) S.row_ptr[t + 1] = S.row_ptr[t] + S.m[t];
    S.row_idx.resize((size_t)S.row_ptr[ns]);
    for (int t = 0; t < ns; ++t) {
        int* r = &S.row_idx[S.row_ptr[t]];
        const int k = S.first[t + 1] - S.first[t];
        for (int q = 0; q < k; ++q) r[q] = S.first[t] + q;
        const auto& sl = st[last_col[t]];
        if ((int)sl.size() != S.m[t] - k) throw std::runtime_error("sparse LU: inconsistent supernode structure");
        std::copy(sl.begin(), sl.end(), r + k);
    }
    std::vector<std::vector<int>>().swap(st);
    // children, offsets, statistics
    S.child_ptr.assign((size_t)ns + 1, 0);
    for (int t = 0; t < ns; ++t) if (S.parent[t] >= 0) S.child_ptr[S.parent[t] + 1]++;
    for (int t = 0; t < ns; ++t) S.child_ptr[t + 1] += S.child_ptr[t];
    S.child.resize((size_t)S.child_ptr[ns]);
    {
        std::vector<int> pos(S.child_ptr.begin(), S.child_ptr.end() - 1);
        for (int t = 0; t < ns; ++t) if (S.parent[t] >= 0) S.child[pos[S.parent[t]]++] = t;
    }
    S.upd_off.assign((size_t)ns + 1, 0);
    S.front_off.assign((size_t)ns + 1, 0);
    S.fac_off.assign((size_t)ns + 1, 0);
    int64_t stored_total = 0;
    for (int t = 0; t < ns; ++t) {
        const int64_t k = S.first[t + 1] - S.first[t], mm = S.m[t];
        S.upd_off[t + 1] = S.upd_off[t] + (mm - k);
        S.front_off[t + 1] = S.front_off[t] + mm * mm;
        S.fac_off[t + 1] = S.fac_off[t] + stored(k, mm);
        stored_total += stored(k, mm);
        S.nnz_l += mm * k - k * (k + 1) / 2;
        S.nnz_u += mm * k - k * (k - 1) / 2;
        S.max_front = std::max<int>(S.max_front, (int)mm);
        for (int64_t j = 0; j < k; ++j) { const double r = (double)(mm - j - 1); S.flops += r + 2.0 * r * r; }
    }
    S.amalg_zeros = stored_total - true_entries;
    // position of a row inside supernode t's front (row must be in its list)
    auto pos_in = [&](int t, int row) -> int {
        const int k = S.first[t + 1] - S.first[t];
        if (row >= S.first[t] && row < S.first[t + 1]) return row - S.first[t];
        const int* b = &S.row_idx[S.row_ptr[t]] + k;
        const int* e = &S.row_idx[S.row_ptr[t]] + S.m[t];
        const int* it = std::lower_bound(b, e, row);
        if (it == e || *it != row) throw std::runtime_error("sparse LU: row missing from a front");
        return (int)(it - &S.row_idx[S.row_ptr[t]]);
    };
    S.relmap.resize((size_t)S.upd_off[ns]);
    for (int t = 0; t < ns; ++t) {
        const int k = S.first[t + 1] - S.first[t];
        if (S.parent[t] < 0) {
            if (S.m[t] != k) throw std::runtime_error("sparse LU: root supernode with update rows");
            continue;
        }
        for (int q = k; q < S.m[t]; ++q) S.relmap[S.upd_off[t] + q - k] = pos_in(S.parent[t], S.row_idx[S.row_ptr[t] + q]);
    }
    const int64_t nnz = rowptr[n];
    S.nz_pos.resize((size_t)nnz);
    for (int io = 0; io < n; ++io)
        for (int64_t q = rowptr[io]; q < rowptr[io + 1]; ++q) {
            const int i = ip[io], j = ip[col[q]];
            const int t = sn_of[std::min(i, j)];
            S.nz_pos[q] = S.front_off[t] + (int64_t)pos_in(t, j) * S.m[t] + pos_in(t, i);
        }
    // level schedule (children are numbered below their parent)
    std::vector<int> lvl((size_t)ns, 0);
    for (int t = 0; t < ns; ++t) if (S.parent[t] >= 0) lvl[S.parent[t]] = std::max(lvl[S.parent[t]], lvl[t] + 1);
    S.nlevels = 0;
    for (int t = 0; t < ns; ++t) S.nlevels = std::max(S.nlevels, lvl[t] + 1);
    S.level_ptr.assign((size_t)S.nlevels + 1, 0);
    for (int t = 0; t < ns; ++t) S.level_ptr[lvl[t] + 1]++;
    for (int l = 0; l < S.nlevels; ++l) S.level_ptr[l + 1] += S.level_ptr[l];
    S.level_sn.resize((size_t)ns);
    {
        std::vector<int> pos(S.level_ptr.begin(), S.level_ptr.end() - 1);
        for (int t = 0; t < ns; ++t) S.level_sn[pos[lvl[t]]++] = t;
    }
    return S;
}

}  // namespace lusym
}  // namespace poro
