// Host-only timing of TreeHost::build_from_parents (what polee_set_tree does before its upload).
//   nvcc -O3 -std=c++17 -I polee_b200/csrc -I include tools/ubench/tree_host_time.cu polee_b200/csrc/build/tree_host.o \
//        polee_b200/csrc/build/mem_cache.o -lcudart -o /tmp/tree_host_time && /tmp/tree_host_time tree.bin
// tree.bin: int32 node_parent_idxs[2n-1] followed by node_js[2n-1]
#include <chrono>
#include <cstdio>
#include <vector>
#include "common.cuh"
// FNV-1a over everything build_from_parents produces: an optimisation of the host code must leave it unchanged
static uint64_t g_h = 1469598103934665603ull;
static void mix(const void *p, size_t bytes) {
    const unsigned char *c = (const unsigned char *)p;
    for (size_t i = 0; i < bytes; ++i) { g_h ^= c[i]; g_h *= 1099511628211ull; }
}
template <typename T> static void mixv(const std::vector<T> &v) { size_t n = v.size(); mix(&n, sizeof n); if (n) mix(v.data(), n * sizeof(T)); }
static uint64_t tree_hash(const polee::TreeHost &t) {
    g_h = 1469598103934665603ull;
    mixv(t.nodes); mixv(t.parent); mixv(t.depth); mixv(t.size);
    for (const polee::TreeSchedHost *s : {&t.top, &t.bottom}) { mixv(s->bin_lvl_ptr); mixv(s->lvl_off); mixv(s->sch_node); }
    for (const polee::SSchedHost *s : {&t.s_top, &t.s_bottom}) {
        mixv(s->bin_off); mixv(s->bin_lvl_ptr); mixv(s->lvl_off); mixv(s->recs);
        mix(&s->max_bin_nodes, 4); mix(&s->max_bin_levels, 4);
    }
    mixv(t.chain_leaf); mixv(t.ganc_ptr); mixv(t.ganc); mixv(t.gcp); mixv(t.nsuf_ptr); mixv(t.nsuf);
    mixv(t.dnodes); mixv(t.drun_anc_ptr); mixv(t.drun_anc); mixv(t.dcta_k0);
    const int sc[] = {t.n_slots, (int)t.caterpillar, t.max_depth, t.max_ganc, t.max_gsuf, (int)t.preorder, t.dfs_max_nk};
    mix(sc, sizeof sc);
    return g_h;
}
int main(int argc, char **argv) {
    FILE *f = fopen(argv[1], "rb");
    if (!f) return 1;
    fseek(f, 0, SEEK_END);
    const long bytes = ftell(f);
    fseek(f, 0, SEEK_SET);
    std::vector<int32_t> buf(bytes / 4);
    if (fread(buf.data(), 4, buf.size(), f) != buf.size()) return 1;
    const int64_t N = (int64_t)buf.size() / 2, n = (N + 1) / 2;
    for (int rep = 0; rep < 6; ++rep) {
        polee::TreeHost th;
        auto t0 = std::chrono::steady_clock::now();
        std::string e = th.build_from_parents(n, buf.data(), buf.data() + N, 512);
        auto t1 = std::chrono::steady_clock::now();
        printf("rep %d: %.2f ms  err='%s' preorder=%d hash=%016llx\n", rep,
               std::chrono::duration<double, std::milli>(t1 - t0).count(), e.c_str(), (int)th.preorder,
               (unsigned long long)tree_hash(th));
    }
    return 0;
}
