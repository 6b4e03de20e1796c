// tree_host.cu -- host-side preparation of a Polya tree for the level-synchronous device kernels.
//
// The tree itself is built by the reference's Julia code (hclust -> order_nodes, src/hclust.jl:193-389;
// stays on the host by north_star) and arrives as (node_parent_idxs, node_js)
// (src/likelihood-approximation.jl:618-621) or as the 0-based left/right/leaf arrays of
// make_inverse_ptt_params (src/ptt.jl:293-309).  Here it is validated, converted to 0-based child
// pointers with the reference's rule (first child seen = RIGHT child, src/ptt.jl:104-110) and cut
// into a level-ordered schedule:
//   * "bottom" bins: forests of whole subtrees with <= bin_nodes nodes in total, one CTA each;
//   * "top": the nodes whose subtree is larger than bin_nodes, one CTA.
// Every node's arithmetic depends only on its parent (forward) or its two children (backward), so a
// level-synchronous sweep computes bit-identical values to the reference's serial index-order sweep.
#include <algorithm>
#include <cmath>
#include <chrono>
#include <climits>
#include <cstdio>
#include <cstdint>
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include <mutex>

namespace polee {

int pad_k(int K) {
    int p = 1;
    while (p < K) p <<= 1;
    return p;
}

static void make_sched(const std::vector<std::vector<int32_t>> &bins_nodes, const std::vector<int32_t> &level_of,
                       TreeSchedHost &out) {
    out.bin_lvl_ptr.assign(1, 0);
    out.lvl_off.clear();
    out.sch_node.clear();
    size_t total = 0;
    for (const auto &bn : bins_nodes) total += bn.size();
    out.sch_node.reserve(total);
    std::vector<int32_t> cnt, cur;  // reused across bins
    for (const auto &bn : bins_nodes) {
        int nl = 0;
        for (int32_t v : bn) nl = std::max(nl, level_of[v] + 1);
        cnt.assign(nl + 1, 0);
        for (int32_t v : bn) cnt[level_of[v] + 1]++;
        for (int l = 0; l < nl; ++l) cnt[l + 1] += cnt[l];
        int32_t base = (int32_t)out.sch_node.size();
        out.sch_node.resize(base + bn.size());
        cur.assign(cnt.begin(), cnt.end() - 1);
        for (int32_t v : bn) out.sch_node[base + cur[level_of[v]]++] = v;
        for (int l = 0; l <= nl; ++l) out.lvl_off.push_back(base + cnt[l]);
        out.bin_lvl_ptr.push_back((int32_t)out.lvl_off.size());
    }
}

std::string TreeHost::build_from_lrf(int64_t n_, const int32_t *left, const int32_t *right, const int32_t *leaf,
                                     int bin_nodes) {
    n = n_;
    N = 2 * n - 1;
    if (n < 1) return "tree: n must be >= 1";
    static const bool timing = getenv("POLEE_SETUP_TIMING") != nullptr && getenv("POLEE_TREE_HOST_TIMING") != nullptr;
    auto tprev = std::chrono::steady_clock::now();
    auto mark = [&](const char *what) {
        if (!timing) return;
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[polee tree host] %-26s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(t1 - tprev).count());
        tprev = t1;
    };
    nodes.assign(N, TreeNode{-1, -1, -1, -1});
    parent.assign(N, -1);
    depth.assign(N, 0);
    size.assign(N, 1);
    std::vector<char> seen_leaf(n, 0);
    int32_t k = 0;
    int64_t nleaves = 0;
    for (int64_t i = 0; i < N; ++i) {
        if (leaf[i] >= 0) {
            if (leaf[i] >= n || seen_leaf[leaf[i]]) return "tree: leaf ids are not a permutation of 1..n";
            seen_leaf[leaf[i]] = 1;
            nodes[i].leaf = leaf[i];
            ++nleaves;
            if (left[i] >= 0 || right[i] >= 0) return "tree: leaf node has children";
        } else {
            int32_t l = left[i], r = right[i];
            if (l < 0 || r < 0 || l >= N || r >= N || l == r) return "tree: internal node without two children";
            if (l <= i || r <= i) return "tree: child index must be greater than its parent's (DFS order)";
            if (parent[l] != -1 || parent[r] != -1) return "tree: node has two parents";
            parent[l] = parent[r] = (int32_t)i;
            nodes[i].left = l;
            nodes[i].right = r;
            nodes[i].k = k++;
        }
    }
    if (nleaves != n || k != n - 1) return "tree: expected n leaves and n-1 internal nodes";
    for (int64_t i = 1; i < N; ++i)
        if (parent[i] < 0) return "tree: more than one root";
    max_depth = 0;
    for (int64_t i = 1; i < N; ++i) {
        depth[i] = depth[parent[i]] + 1;
        max_depth = std::max(max_depth, (int)depth[i]);
    }
    for (int64_t i = N - 1; i >= 1; --i) size[parent[i]] += size[i];

    mark("validate + depth + size");
    // ---- DFS pre-order?  (right child = next node, left child = the node after the right subtree)
    bool preorder_nodes = n >= 2;
    for (int64_t i = 0; i < N && preorder_nodes; ++i)
        if (nodes[i].leaf < 0) preorder_nodes = nodes[i].right == i + 1 && nodes[i].left == i + 1 + size[i + 1];
    preorder = preorder_nodes && max_depth <= DFS_MAX_DEPTH;
    dnodes.clear(); drun_anc_ptr.clear(); drun_anc.clear(); dcta_k0.clear();
    dfs_max_nk = 0;
    if (preorder) {
        dnodes.assign(N + 1, DNode{-1, 0u});  // one padding record: the kernel copies records in pairs
        for (int64_t i = 0; i < N; ++i) {
            const bool is_left = i > 0 && nodes[parent[i]].left == (int32_t)i;
            dnodes[i].k_or_leaf = nodes[i].leaf >= 0 ? -1 - nodes[i].leaf : nodes[i].k;
            dnodes[i].meta = (uint32_t)depth[i] | (is_left ? 0x80000000u : 0u);
        }
        const int64_t nruns = (N + DFS_RUN - 1) / DFS_RUN;
        drun_anc_ptr.reserve(nruns + 1);
        std::vector<uint32_t> path;
        for (int64_t r = 0; r < nruns; ++r) {
            drun_anc_ptr.push_back((uint32_t)drun_anc.size());
            path.clear();
            for (int32_t v = (int32_t)(r * DFS_RUN); parent[v] >= 0; v = parent[v])
                path.push_back(((uint32_t)nodes[parent[v]].k << 1) | (nodes[parent[v]].left == v ? 1u : 0u));
            drun_anc.insert(drun_anc.end(), path.rbegin(), path.rend());
        }
        drun_anc_ptr.push_back((uint32_t)drun_anc.size());
        const int64_t nctas = (N + DFS_CTA_NODES - 1) / DFS_CTA_NODES;
        dcta_k0.reserve(nctas + 1);
        int32_t kc = 0;
        for (int64_t i = 0; i < N; ++i) {
            if (i % DFS_CTA_NODES == 0) dcta_k0.push_back(kc);
            if (nodes[i].leaf < 0) ++kc;
        }
        dcta_k0.push_back(kc);
        for (int64_t c = 0; c < nctas; ++c) dfs_max_nk = std::max(dfs_max_nk, dcta_k0[c + 1] - dcta_k0[c]);
    }

    mark("dfs-run forward inputs");
    // ---- root -> node paths, grouped (see TreeHost); not needed when the DFS-run kernel serves the tree
    ganc_ptr.clear(); ganc.clear(); gcp.clear(); nsuf_ptr.clear(); nsuf.clear();
    max_ganc = max_gsuf = 0;
    if (!preorder) {
        int64_t total = 0;
        for (int64_t i = 0; i < N; ++i) total += depth[i];
        bool ok = total <= PATH_MAX_ENTRIES && n >= 2;
        std::vector<uint32_t> path_ptr, path_ent;
        if (ok) {
            path_ptr.resize(N + 1);
            path_ent.resize((size_t)total);
            uint32_t pos = 0;
            for (int64_t i = 0; i < N; ++i) {  // parents precede their children (checked above)
                path_ptr[i] = pos;
                if (i > 0) {
                    const int32_t pa = parent[i];
                    const uint32_t pb = path_ptr[pa], pl = (uint32_t)depth[pa];
                    std::copy(path_ent.begin() + pb, path_ent.begin() + pb + pl, path_ent.begin() + pos);
                    pos += pl;
                    path_ent[pos++] = ((uint32_t)nodes[pa].k << 1) | (nodes[pa].left == (int32_t)i ? 1u : 0u);
                }
            }
            path_ptr[N] = pos;
            const int64_t ng = (N + PATH_GROUP - 1) / PATH_GROUP;
            std::vector<int32_t> local_of_k((size_t)std::max<int64_t>(n - 1, 1), -1), stamp((size_t)std::max<int64_t>(n - 1, 1), -1);
            ganc_ptr.reserve(ng + 1); gcp.reserve(ng); nsuf_ptr.reserve(N + 1);
            for (int64_t g = 0; g < ng && ok; ++g) {
                const int64_t i0 = g * PATH_GROUP, i1 = std::min<int64_t>(N, i0 + PATH_GROUP);
                uint32_t cp = (uint32_t)depth[i0];  // longest common prefix of the group's paths
                for (int64_t i = i0 + 1; i < i1; ++i) {
                    const uint32_t len = std::min<uint32_t>(cp, (uint32_t)depth[i]);
                    uint32_t c = 0;
                    while (c < len && path_ent[path_ptr[i0] + c] == path_ent[path_ptr[i] + c]) ++c;
                    cp = c;
                }
                ganc_ptr.push_back((uint32_t)ganc.size());
                gcp.push_back(cp);
                const size_t base = ganc.size(), sbase = nsuf.size();
                for (uint32_t c = 0; c < cp; ++c) ganc.push_back(path_ent[path_ptr[i0] + c]);
                for (int64_t i = i0; i < i1; ++i) {
                    nsuf_ptr.push_back((uint32_t)nsuf.size());
                    for (uint32_t c = cp; c < (uint32_t)depth[i]; ++c) {
                        const uint32_t en = path_ent[path_ptr[i] + c], k = en >> 1;
                        if (stamp[k] != (int32_t)g) {
                            stamp[k] = (int32_t)g;
                            local_of_k[k] = (int32_t)(ganc.size() - base);
                            ganc.push_back(k << 1);
                        }
                        nsuf.push_back((uint16_t)(((uint32_t)local_of_k[k] << 1) | (en & 1u)));
                    }
                }
                const int na = (int)(ganc.size() - base);
                max_ganc = std::max(max_ganc, na);
                max_gsuf = std::max(max_gsuf, (int)(nsuf.size() - sbase));
                if (na > PATH_MAX_GANC || nsuf.size() - sbase > 16384) ok = false;
            }
            ganc_ptr.push_back((uint32_t)ganc.size());
            nsuf_ptr.push_back((uint32_t)nsuf.size());
        }
        if (!ok) {
            ganc_ptr.clear(); ganc.clear(); gcp.clear(); nsuf_ptr.clear(); nsuf.clear();
            max_ganc = max_gsuf = 0;
        }
    }

    mark("root paths");
    // ---- caterpillar ("list") tree?
    caterpillar = n >= 2;
    for (int64_t i = 0; i < N && caterpillar; ++i) {
        if (nodes[i].leaf >= 0) continue;
        caterpillar = (i % 2 == 0) && nodes[i].right == i + 1 && nodes[i].left == i + 2 && nodes[i + 1].leaf >= 0;
    }
    chain_leaf.clear();
    if (caterpillar) {
        chain_leaf.resize(n);
        for (int64_t kk = 0; kk < n - 1; ++kk) chain_leaf[kk] = nodes[2 * kk + 1].leaf;
        chain_leaf[n - 1] = nodes[N - 1].leaf;
        caterpillar = nodes[N - 1].leaf >= 0;
    }

    // ---- cut: top = nodes whose subtree exceeds bin_nodes
    std::vector<char> is_top(N, 0);
    std::vector<int32_t> top_list;
    for (int64_t i = 0; i < N; ++i)
        if (size[i] > bin_nodes) {
            is_top[i] = 1;
            top_list.push_back((int32_t)i);
        }

    std::vector<int32_t> level_of(N, 0);
    std::vector<std::vector<int32_t>> bins;
    int64_t cur_fill = 0;
    std::vector<int32_t> stack;
    for (int64_t r = 0; r < N; ++r) {
        if (is_top[r] || (parent[r] >= 0 && !is_top[parent[r]])) continue;  // r is a bottom root
        if (bins.empty() || cur_fill + size[r] > bin_nodes) {
            bins.emplace_back();
            bins.back().reserve((size_t)bin_nodes);
            cur_fill = 0;
        }
        cur_fill += size[r];
        if (preorder_nodes) {  // a subtree is the contiguous index range [r, r + size): the order the stack walk below gives
            for (int32_t v = (int32_t)r; v < (int32_t)(r + size[r]); ++v) {
                level_of[v] = depth[v] - depth[r];
                bins.back().push_back(v);
            }
            continue;
        }
        stack.assign(1, (int32_t)r);
        while (!stack.empty()) {
            int32_t v = stack.back();
            stack.pop_back();
            level_of[v] = depth[v] - depth[r];
            bins.back().push_back(v);
            if (nodes[v].leaf < 0) {
                stack.push_back(nodes[v].left);
                stack.push_back(nodes[v].right);
            }
        }
    }
    mark("cut + bins");
    make_sched(bins, level_of, bottom);
    std::vector<std::vector<int32_t>> tb;
    if (!top_list.empty()) {
        tb.push_back(top_list);
        for (int32_t v : top_list) level_of[v] = depth[v];
    }
    make_sched(tb, level_of, top);

    mark("global-memory schedules");
    // ---- schedule-order records for the shared-memory kernels
    std::vector<int32_t> slot_of(N, -2);
    n_slots = 0;
    for (const auto &bn : bins)
        for (int32_t v : bn)
            if (parent[v] < 0 || is_top[parent[v]]) slot_of[v] = parent[v] < 0 ? -1 : n_slots++;
    std::vector<int32_t> local_scratch;
    auto make_ssched = [&](const std::vector<std::vector<int32_t>> &bins_nodes, bool is_top_sched, SSchedHost &out) {
        out.bin_off.assign(1, 0);
        out.bin_lvl_ptr.assign(1, 0);
        out.lvl_off.clear();
        out.recs.clear();
        out.max_bin_nodes = 0;
        out.max_bin_levels = 0;
        local_scratch.assign(N, -1);
        std::vector<int32_t> &local = local_scratch;
        size_t total = 0;
        for (const auto &bn0 : bins_nodes) total += bn0.size();
        out.recs.reserve(total + (is_top_sched ? (size_t)n_slots + 1 : 0));
        std::vector<int32_t> bn, cnt, cur, order;  // reused across bins
        for (const auto &bn0 : bins_nodes) {
            // members: the bin's nodes (+ for the top bin: the bottom roots hanging off it, as exchange leaves)
            bn.assign(bn0.begin(), bn0.end());
            if (is_top_sched)
                for (int32_t v : bn0)
                    if (nodes[v].leaf < 0)
                        for (int32_t c : {nodes[v].left, nodes[v].right})
                            if (!is_top[c]) bn.push_back(c);
            auto lvl = [&](int32_t v) { return is_top_sched ? depth[v] : level_of[v]; };
            int nl = 0;
            for (int32_t v : bn) nl = std::max(nl, lvl(v) + 1);
            cnt.assign(nl + 1, 0);
            for (int32_t v : bn) cnt[lvl(v) + 1]++;
            for (int l = 0; l < nl; ++l) cnt[l + 1] += cnt[l];
            cur.assign(cnt.begin(), cnt.end() - 1);
            order.resize(bn.size());
            for (int32_t v : bn) {
                local[v] = cur[lvl(v)]++;
                order[local[v]] = v;
            }
            const int32_t base = (int32_t)out.recs.size();
            for (int32_t v : order) {
                SNode r;
                const bool exch = is_top_sched && !is_top[v];
                if (exch) {
                    r.k_or_leaf = INT32_MIN;
                    r.left = r.right = -1;
                    r.slot = slot_of[v];
                } else if (nodes[v].leaf >= 0) {
                    r.k_or_leaf = -1 - nodes[v].leaf;
                    r.left = r.right = -1;
                    r.slot = is_top_sched ? -2 : slot_of[v];
                } else {
                    r.k_or_leaf = nodes[v].k;
                    r.left = local[nodes[v].left];
                    r.right = local[nodes[v].right];
                    r.slot = is_top_sched ? (parent[v] < 0 ? -1 : -2) : slot_of[v];
                }
                out.recs.push_back(r);
            }
            for (int l = 0; l <= nl; ++l) out.lvl_off.push_back(base + cnt[l]);
            out.bin_lvl_ptr.push_back((int32_t)out.lvl_off.size());
            out.bin_off.push_back((int32_t)out.recs.size());
            out.max_bin_nodes = std::max(out.max_bin_nodes, (int)bn.size());
            out.max_bin_levels = std::max(out.max_bin_levels, nl);
        }
    };
    make_ssched(bins, false, s_bottom);
    make_ssched(tb, true, s_top);
    mark("shared-memory schedules");
    return "";
}

std::string TreeHost::build_from_parents(int64_t n_, const int32_t *parent_idxs, const int32_t *js, int bin_nodes) {
    int64_t NN = 2 * n_ - 1;
    if (n_ < 1) return "tree: n must be >= 1";
    std::vector<int32_t> l(NN, -1), r(NN, -1), f(NN, -1);
    // src/ptt.jl:89-116 (== make_inverse_ptt_params, src/ptt.jl:293-309): first child seen is the right one
    if (parent_idxs[0] != 0) return "tree: node 1 must be the root (parent index 0)";
    for (int64_t i = 0; i < NN; ++i) {
        int32_t p = parent_idxs[i];
        if (i > 0) {
            if (p < 1 || p > NN) return "tree: parent index out of range";
            if (p - 1 >= i) return "tree: parent index must be smaller than the node's own index";
            if (r[p - 1] == -1)
                r[p - 1] = (int32_t)i;
            else if (l[p - 1] == -1)
                l[p - 1] = (int32_t)i;
            else
                return "tree: node with more than two children";
        }
        if (js[i] < 0 || js[i] > n_) return "tree: node_js out of range";
        f[i] = js[i] - 1;
    }
    return build_from_lrf(n_, l.data(), r.data(), f.data(), bin_nodes);
}

void TreeDev::release() {
    polee::dfree(nodes);
    for (TreeSchedDev *s : {&top, &bottom}) {
        polee::dfree(s->bin_lvl_ptr);
        polee::dfree(s->lvl_off);
        polee::dfree(s->sch_node);
        *s = TreeSchedDev();
    }
    polee::dfree(chain_leaf);
    chain_leaf = nullptr;
    caterpillar = false;
    polee::dfree(ganc_ptr); polee::dfree(ganc); polee::dfree(gcp); polee::dfree(nsuf_ptr); polee::dfree(nsuf);
    ganc_ptr = ganc = gcp = nsuf_ptr = nullptr;
    nsuf = nullptr;
    polee::dfree(dnodes); polee::dfree(drun_anc_ptr); polee::dfree(drun_anc); polee::dfree(dcta_k0);
    dnodes = nullptr; drun_anc_ptr = drun_anc = nullptr; dcta_k0 = nullptr;
    dfs_ctas = dfs_max_nk = 0;
    n_groups = max_ganc = max_gsuf = 0;
    for (SSchedDev *s : {&s_top, &s_bottom}) {
        polee::dfree(s->bin_off);
        polee::dfree(s->bin_lvl_ptr);
        polee::dfree(s->lvl_off);
        polee::dfree(s->recs);
        *s = SSchedDev();
    }
    nodes = nullptr;
    n = N = 0;
    n_slots = 0;
}

static cudaError_t up(const std::vector<int32_t> &v, int32_t **d) {
    *d = nullptr;
    size_t bytes = std::max<size_t>(v.size(), 1) * sizeof(int32_t);
    cudaError_t e = polee::dmalloc((void **)d, bytes);
    if (e != cudaSuccess) return e;
    if (!v.empty()) e = cudaMemcpy(*d, v.data(), v.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
    return e;
}

std::string upload_tree(const TreeHost &th, TreeDev &td) {
    td.release();
    td.n = th.n;
    td.N = th.N;
    cudaError_t e = polee::dmalloc((void **)&td.nodes, sizeof(TreeNode) * th.N);
    if (e == cudaSuccess) e = cudaMemcpy(td.nodes, th.nodes.data(), sizeof(TreeNode) * th.N, cudaMemcpyHostToDevice);
    const TreeSchedHost *hs[2] = {&th.top, &th.bottom};
    TreeSchedDev *ds[2] = {&td.top, &td.bottom};
    for (int s = 0; s < 2 && e == cudaSuccess; ++s) {
        e = up(hs[s]->bin_lvl_ptr, &ds[s]->bin_lvl_ptr);
        if (e == cudaSuccess) e = up(hs[s]->lvl_off, &ds[s]->lvl_off);
        if (e == cudaSuccess) e = up(hs[s]->sch_node, &ds[s]->sch_node);
        ds[s]->nbins = hs[s]->nbins();
    }
    const SSchedHost *hss[2] = {&th.s_top, &th.s_bottom};
    SSchedDev *dss[2] = {&td.s_top, &td.s_bottom};
    for (int s = 0; s < 2 && e == cudaSuccess; ++s) {
        e = up(hss[s]->bin_off, &dss[s]->bin_off);
        if (e == cudaSuccess) e = up(hss[s]->bin_lvl_ptr, &dss[s]->bin_lvl_ptr);
        if (e == cudaSuccess) e = up(hss[s]->lvl_off, &dss[s]->lvl_off);
        if (e == cudaSuccess) {
            size_t bytes = std::max<size_t>(hss[s]->recs.size(), 1) * sizeof(SNode);
            e = polee::dmalloc((void **)&dss[s]->recs, bytes);
            if (e == cudaSuccess && !hss[s]->recs.empty())
                e = cudaMemcpy(dss[s]->recs, hss[s]->recs.data(), hss[s]->recs.size() * sizeof(SNode), cudaMemcpyHostToDevice);
        }
        dss[s]->nbins = hss[s]->nbins();
        dss[s]->max_bin_nodes = hss[s]->max_bin_nodes;
        dss[s]->max_bin_levels = hss[s]->max_bin_levels;
    }
    if (e == cudaSuccess && !th.ganc_ptr.empty()) {
        auto upv = [&](const void *src, size_t bytes, void **dst) {
            cudaError_t ee = polee::dmalloc(dst, std::max<size_t>(bytes, 4));
            if (ee == cudaSuccess && bytes) ee = cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice);
            return ee;
        };
        e = upv(th.ganc_ptr.data(), 4 * th.ganc_ptr.size(), (void **)&td.ganc_ptr);
        if (e == cudaSuccess) e = upv(th.ganc.data(), 4 * th.ganc.size(), (void **)&td.ganc);
        if (e == cudaSuccess) e = upv(th.gcp.data(), 4 * th.gcp.size(), (void **)&td.gcp);
        if (e == cudaSuccess) e = upv(th.nsuf_ptr.data(), 4 * th.nsuf_ptr.size(), (void **)&td.nsuf_ptr);
        if (e == cudaSuccess) e = upv(th.nsuf.data(), 2 * th.nsuf.size(), (void **)&td.nsuf);
        td.n_groups = (int)th.gcp.size();
        td.max_ganc = th.max_ganc;
        td.max_gsuf = th.max_gsuf;
    }
    td.max_depth = th.max_depth;
    if (e == cudaSuccess && th.preorder) {
        auto upv = [&](const void *src, size_t bytes, void **dst) {
            cudaError_t ee = polee::dmalloc(dst, std::max<size_t>(bytes, 4));
            if (ee == cudaSuccess && bytes) ee = cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice);
            return ee;
        };
        e = upv(th.dnodes.data(), sizeof(DNode) * th.dnodes.size(), (void **)&td.dnodes);
        if (e == cudaSuccess) e = upv(th.drun_anc_ptr.data(), 4 * th.drun_anc_ptr.size(), (void **)&td.drun_anc_ptr);
        if (e == cudaSuccess) e = upv(th.drun_anc.data(), 4 * th.drun_anc.size(), (void **)&td.drun_anc);
        if (e == cudaSuccess) e = upv(th.dcta_k0.data(), 4 * th.dcta_k0.size(), (void **)&td.dcta_k0);
        td.dfs_ctas = (int)th.dcta_k0.size() - 1;
        td.dfs_max_nk = th.dfs_max_nk;
    }
    td.n_slots = th.n_slots;
    td.caterpillar = th.caterpillar;
    // read once per tree: no launch, graph-captured ones included, looks at the environment
    const char *chain_env = getenv("POLEE_CHAIN_MIN_NODES");
    td.chain_min_nodes = chain_env ? atoll(chain_env) : 4096;
    if (e == cudaSuccess && th.caterpillar) e = up(th.chain_leaf, &td.chain_leaf);
    if (e != cudaSuccess) return std::string("upload_tree: ") + cudaGetErrorString(e);
    // the pageable-memory copies above run on the legacy stream, which does not order against the handle's
    // non-blocking stream: make sure their DMA tails have landed before any kernel can read the tree
    {
        std::unique_lock<std::shared_mutex> cap(capture_mutex());
        if (cudaDeviceSynchronize() != cudaSuccess) return "upload_tree: device synchronisation failed";
    }
    return "";
}

}  // namespace polee
