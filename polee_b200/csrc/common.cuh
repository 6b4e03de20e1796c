// common.cuh -- internal declarations shared by the translation units of libpolee_b200.so.
// Nothing here is part of the ABI (that is include/polee_b200.h).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <shared_mutex>
#include <utility>
#include <string>
#include <vector>

#include "../../include/polee_b200.h"

#ifdef POLEE_WITH_NCCL
#include <nccl.h>
#endif

namespace polee {

// ------------------------------------------------------------------ error plumbing
struct Error {
    int code;
    std::string msg;
};

#define POLEE_CUDA_CHECK(h, expr)                                                          \
    do {                                                                                   \
        cudaError_t _e = (expr);                                                           \
        if (_e != cudaSuccess) {                                                           \
            return (h)->fail(POLEE_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
        }                                                                                  \
    } while (0)

// ------------------------------------------------------------------ device layouts
// K1: one tile = up to ROW_TILE rows of one row-length class of the SELL slabs.
constexpr int ROW_TILE = 256;
struct RowTile {
    uint64_t slab_off;  // element offset of (t = 0, first row of the tile) in sell_idx / sell_val
    uint32_t stride;    // rows (padded) in the class = distance between successive t
    uint32_t len;       // entries per row in this class
    uint32_t row0;      // first permuted row id of the tile
    uint32_t nrows;     // valid rows in the tile (<= ROW_TILE)
};

// ---- fused likelihood layout ("row tiles"): K1 and K2 in one pass over the matrix.
// A tile is a run of <= FT_ROWS consecutive rows (and < FT_ENTRY_WINDOW + longest-row entries), processed by one CTA;
// inside a tile the rows are re-ordered longest first and cut into groups of 32 (one warp, one lane per row).  A tile
// carries its entries twice, once per access pattern, and everything travels as one 16-byte aligned blob (one bulk
// copy):
//   header | cols u32[C] | ginfo u32[G] | dest u32[S] | valA f32[EA] | valB f32[E] | lrowB u16[E] | segptr u16[S+1] | lcolA u8[EA]
//  * row side (p = X x): group g is a dense glen x 32 slab, entry t of lane l at gbase + t * 32 + l (val 0 padding),
//    so a warp reads it conflict-free with one trip count; lcolA = index into cols, the tile's C <= 255 distinct
//    columns (a local dictionary: x of these columns is staged in shared memory once per tile); ginfo = gbase | glen << 16.
//  * column side (g += X^T w): the entries column-major with their row position, cut into S segments of <= FT_SEG
//    entries of one column (segptr); one warp sums one segment and writes one partial to slot dest[segment] of the
//    partial array, which is ordered by column, so the second stage adds contiguous runs.  w never leaves shared memory.
// ~11 bytes per entry instead of the 16 the split layouts stream (8 in K1 + 8 in K2) plus 2 x K x 4 bytes per row of w.
constexpr int FT_ROWS = 512;
constexpr uint32_t FT_ENTRY_WINDOW = 4096;
constexpr uint32_t FT_SEG = 128;
constexpr uint32_t FT_MAX_C = 255;
constexpr uint32_t FT_MAX_EA = 32767;
struct FusedHdr {
    uint32_t rows, E, C, S;  // rows, entries, distinct columns, column segments of the tile
    uint32_t row0, part0;    // first row position; index of the tile's first partial (= first segment)
    uint32_t EA, G;          // padded row-side entries, row groups
};
struct FusedTileDesc {
    uint64_t off;    // byte offset of the blob
    uint32_t bytes;  // blob size (multiple of 16)
    uint32_t pad;
};
struct BlobLayout {
    uint32_t cols, ginfo, dest, valA, valB, lrowB, segptr, lcolA, bytes;
};
__host__ __device__ inline BlobLayout blob_layout(const FusedHdr &hd) {
    BlobLayout L;
    L.cols = (uint32_t)sizeof(FusedHdr);
    L.ginfo = L.cols + ((hd.C * 4u + 15u) & ~15u);
    L.dest = L.ginfo + ((hd.G * 4u + 15u) & ~15u);
    L.valA = L.dest + ((hd.S * 4u + 15u) & ~15u);
    L.valB = L.valA + ((hd.EA * 4u + 15u) & ~15u);
    L.lrowB = L.valB + ((hd.E * 4u + 15u) & ~15u);
    L.segptr = L.lrowB + ((hd.E * 2u + 15u) & ~15u);
    L.lcolA = L.segptr + (((hd.S + 1u) * 2u + 15u) & ~15u);
    L.bytes = L.lcolA + ((hd.EA + 15u) & ~15u);
    return L;
}
// ---- equivalence-class layout ("ec"): the default likelihood layout.
// Fragments (rows) compatible with the same set of transcripts form an equivalence class -- the unit salmon / kallisto
// collapse to counts; Polee keeps every fragment's own conditional probabilities (src/rnaseq_sample.jl:104), so a class
// of R rows and L transcripts is a DENSE R x L block of Float32 values sharing ONE list of L column ids.  Position-sorted
// reads (src/rnaseq_sample.jl:399-419) make classes large (fixture: 496 classes for 19 743 rows).  The layout stores the
// column ids once per task and the values alone per entry (4 B/entry + padding instead of 8 B twice), and both sparse
// passes of a step are done on the block while it sits in shared memory, for the K draws at once:
//     p[r][k] = sum_l V[r][l] x[c_l][k]          (pAt_mul_B!,    src/sparse.jl:6-21)
//     g[c_l][k] += sum_r V[r][l] / p[r][k]       (pAt_mulinv_B!, src/sparse.jl:25-40)
// A class is cut into blocks of 32 lanes = 32 / q rows x q column slices of LH = ceil(L / q) <= 8 columns (q = 1, 2, 4,
// 8 for L <= 8, 16, 32, 64), and into tasks of <= nbt(L) blocks; one warp = one task at a time, streamed by one bulk copy:
//     EcHdr | cols u32[q LH] | dest u32[q LH] | pad to 16 | V f32[nb][LH][32]
// V element (block b, column j of the slice, lane) = value of row b * (32 / q) + lane / q, column (lane % q) * LH + j
// (0 where that column is padding): lane-major, so a warp reads a block's column j with one conflict-free 128-byte
// shared-memory read and nothing is padded when L <= 8.  dest[l] = slot of the task's partial for column l in a partial
// array ordered by column; a second small launch adds each column's partials in a fixed order (no atomics).  Classes
// with fewer than EC_MIN_ROWS rows (when that policy is on) or rows longer than EC_MAX_L go to the general layouts
// below ("rest" rows).
constexpr uint32_t EC_MAX_L = 64;
constexpr uint32_t EC_MIN_ROWS_DEFAULT = 12;
#ifndef POLEE_EC_V_BYTES
#define POLEE_EC_V_BYTES 8192
#endif
constexpr uint32_t EC_V_BYTES = POLEE_EC_V_BYTES;   // V bytes per task (<= one shared-memory stage)
constexpr uint32_t EC_MAX_NBT = 32;         // blocks per task (bounds the Float32 chains of the f32 arithmetic)
constexpr uint32_t EC_STAGE_BYTES = 16 + 2 * 4 * EC_MAX_L + EC_V_BYTES;   // 8720
__host__ __device__ inline uint32_t ec_q(uint32_t L) { return L <= 8u ? 1u : (L <= 16u ? 2u : (L <= 32u ? 4u : 8u)); }
__host__ __device__ inline uint32_t ec_lh(uint32_t L) { const uint32_t q = ec_q(L); return (L + q - 1u) / q; }
__host__ __device__ inline uint32_t ec_nbt(uint32_t L) {   // blocks per task
    const uint32_t v = EC_V_BYTES / (ec_lh(L) * 128u);
    return v < 1u ? 1u : (v > EC_MAX_NBT ? EC_MAX_NBT : v);
}
__host__ __device__ inline uint32_t ec_hdr_bytes(uint32_t L) { return (16u + 8u * ec_q(L) * ec_lh(L) + 15u) & ~15u; }
__host__ __device__ inline uint32_t ec_task_bytes(uint32_t L, uint32_t nb) { return ec_hdr_bytes(L) + nb * ec_lh(L) * 128u; }
struct EcHdr {
    uint32_t pk, nb, rows, slot0;  // L | LH << 8 | q << 16 | log2(q) << 24; blocks; valid rows; first row slot (row_of_slot / weights)
};
__host__ __device__ inline uint32_t ec_pack(uint32_t L) {
    const uint32_t q = ec_q(L), lq = q == 1u ? 0u : (q == 2u ? 1u : (q == 4u ? 2u : 3u));
    return L | (ec_lh(L) << 8) | (q << 16) | (lq << 24);
}
__host__ __device__ inline uint32_t ec_pk_l(uint32_t pk) { return pk & 0xFFu; }
__host__ __device__ inline uint32_t ec_pk_lh(uint32_t pk) { return (pk >> 8) & 0xFFu; }
__host__ __device__ inline uint32_t ec_pk_q(uint32_t pk) { return (pk >> 16) & 0xFFu; }
__host__ __device__ inline uint32_t ec_pk_lq(uint32_t pk) { return pk >> 24; }
struct EcTaskDesc {
    uint64_t off;    // byte offset of the task blob
    uint32_t bytes;  // multiple of 16
    uint32_t pad;
};
// second stage: g[col] = sum of the partials of the column, in tile order.  A unit is <= FT_UNIT partials of one
// column (KP lanes); columns with more than one unit are finished by a second small launch.
constexpr int FT_UNIT = 64;
struct FusedUnit {
    uint32_t col, begin, end;  // partials [begin, end) (the partial array is ordered by column)
    int32_t out;               // -1: writes g[col]; >= 0: writes the level-2 slot
};
struct FusedMulti {
    uint32_t col, first, count, pad;  // level-2 slots [first, first + count)
};

// K2: one warp = one segment of <= COL_SEG consecutive entries of one column (rows permuted, sorted).
constexpr int COL_SEG = 256;
struct ColSeg {
    uint32_t start;  // entry offset in csc_row / csc_val
    uint32_t len;    // low 16 bits: entries; high 16 bits: r > 0 if this segment heads a run of r segments of
                     // the same column inside one CTA item (K2_WARPS consecutive segments)
    uint32_t col;
    int32_t slot;    // of a run head: >= 0 partial slot (column spans several runs); -1: the run writes g directly
};
struct MultiCol {
    uint32_t col;
    uint32_t first_slot;
    uint32_t nslots;
    uint32_t pad;
};

// step counters living in device memory so that one captured CUDA graph can be replayed for every step
struct StepCtl {
    int step_fwd;  // 1-based step the forward kernels of the current step use
    int step_upd;  // same, as seen by the update kernel (set by k3_mid)
};

constexpr int64_t PATH_MAX_ENTRIES = 64ll << 20;  // sum of node depths up to which root paths are built
constexpr int PATH_GROUP = 128;                  // nodes per path group (one CTA)
constexpr int PATH_SLOTS = 32;                   // node slots per CTA (threads = PATH_SLOTS x KP, PATH_GROUP / PATH_SLOTS nodes each)
constexpr int PATH_MAX_GANC = 1024;              // distinct ancestors a group may have

// DFS-run forward kernel (k3d_tree_fwd): a thread walks DFS_RUN consecutive nodes of a tree stored in DFS pre-order
constexpr int DFS_RUN = 64;            // nodes per thread
constexpr int DFS_RUNS_PER_CTA = 16;   // runs per CTA (threads = DFS_RUNS_PER_CTA x KP)
constexpr int DFS_CTA_NODES = DFS_RUN * DFS_RUNS_PER_CTA;
constexpr int DFS_MAX_DEPTH = 96;      // deeper trees keep the path-product / level kernels
struct DNode {
    int32_t k_or_leaf;  // >= 0: internal node, index k; < 0: leaf, transcript = -1 - v
    uint32_t meta;      // depth | (1u << 31 if the node is its parent's LEFT child, i.e. the child that comes second)
};

// Tree node, 0-based; leaf < 0 <=> internal node (then k = index among internal nodes in node order).
struct TreeNode {
    int32_t left, right, k, leaf;
};

// Level-ordered schedule of a set of "bins" (one CTA each).  Bin b owns levels
// lvl_off[bin_lvl_ptr[b] .. bin_lvl_ptr[b+1]] (one more offset than levels) into sch_node.
struct TreeSchedHost {
    std::vector<int32_t> bin_lvl_ptr;  // nbins + 1
    std::vector<int32_t> lvl_off;      // sum(levels_b + 1)
    std::vector<int32_t> sch_node;     // node ids in (bin, level) order
    int nbins() const { return (int)bin_lvl_ptr.size() - 1; }
};

// Schedule-order records for the shared-memory tree kernels: bin b owns records bin_off[b]..bin_off[b+1],
// level-ordered; children are LOCAL positions inside the bin.
struct SNode {
    int32_t k_or_leaf;  // >= 0: internal node, index k; < 0: leaf, transcript = -1 - v; INT32_MIN: exchange leaf
    int32_t left, right;  // local positions of the children (internal nodes only)
    int32_t slot;  // level-0 nodes of bottom bins / exchange leaves of the top bin: exchange slot; -1: global root; else -2
};
struct SSchedHost {
    std::vector<int32_t> bin_off, bin_lvl_ptr, lvl_off;
    std::vector<SNode> recs;
    int max_bin_nodes = 0, max_bin_levels = 0;
    int nbins() const { return (int)bin_off.size() - 1; }
};
struct SSchedDev {
    int32_t *bin_off = nullptr, *bin_lvl_ptr = nullptr, *lvl_off = nullptr;
    SNode *recs = nullptr;
    int nbins = 0, max_bin_nodes = 0, max_bin_levels = 0;
};

struct TreeSchedDev {
    int32_t *bin_lvl_ptr = nullptr, *lvl_off = nullptr, *sch_node = nullptr;
    int nbins = 0;
};

struct TreeHost {
    int64_t n = 0, N = 0;
    std::vector<TreeNode> nodes;
    std::vector<int32_t> parent, depth, size;
    TreeSchedHost top, bottom;
    SSchedHost s_top, s_bottom;  // same cut, schedule-order records (shared-memory kernels)
    int n_slots = 0;             // exchange slots = bottom subtree roots
    bool caterpillar = false;    // list tree: internal node k at index 2k, right child = leaf at 2k+1, left = 2k+2
    std::vector<int32_t> chain_leaf;  // [n]: leaf id hanging off spine node k (k < n-1), [n-1] = the last leaf
    int max_depth = 0;
    // Root -> node paths for the path-product forward kernel, per group of PATH_GROUP consecutive nodes (neighbours in
    // DFS order share most of their ancestors): the group's distinct ancestors `ganc` -- first the gcp[g] entries of the
    // path prefix all its nodes share, root first, then the others -- as (k << 1 | 1 if the path continues into the
    // LEFT child; only meaningful in the prefix), and per node the rest of its path `nsuf` as
    // (index into the group's ganc list) << 1 | left.  Empty when the tree is too deep for it.
    std::vector<uint32_t> ganc_ptr, ganc, gcp, nsuf_ptr;
    std::vector<uint16_t> nsuf;
    int max_ganc = 0, max_gsuf = 0;  // most distinct ancestors / suffix entries of a group
    // DFS-run forward (trees in DFS pre-order, the order order_nodes emits, src/hclust.jl:361-389; then the root paths
    // above are not built): per node a DNode; per run of DFS_RUN nodes the ancestors of its first node, root first, as
    // (k << 1) | 1 if the path continues into the LEFT child; per CTA the number of internal nodes before its first node
    bool preorder = false;
    std::vector<DNode> dnodes;
    std::vector<uint32_t> drun_anc_ptr, drun_anc;
    std::vector<int32_t> dcta_k0;
    int dfs_max_nk = 0;
    // returns "" or an error text
    std::string build_from_lrf(int64_t n, const int32_t *left, const int32_t *right, const int32_t *leaf,
                               int bin_nodes);
    std::string build_from_parents(int64_t n, const int32_t *parent_idxs, const int32_t *js, int bin_nodes);
};

struct TreeDev {
    int64_t n = 0, N = 0;
    TreeNode *nodes = nullptr;
    TreeSchedDev top, bottom;
    SSchedDev s_top, s_bottom;
    int n_slots = 0;
    bool caterpillar = false;
    int32_t *chain_leaf = nullptr;
    uint32_t *ganc_ptr = nullptr, *ganc = nullptr, *gcp = nullptr, *nsuf_ptr = nullptr;  // root paths (nullptr: not built)
    uint16_t *nsuf = nullptr;
    int n_groups = 0, max_ganc = 0, max_gsuf = 0;
    DNode *dnodes = nullptr;  // DFS-run forward (nullptr: not available for this tree)
    uint32_t *drun_anc_ptr = nullptr, *drun_anc = nullptr;
    int32_t *dcta_k0 = nullptr;
    int dfs_ctas = 0, dfs_max_nk = 0, max_depth = 0;
    int64_t chain_min_nodes = 0;  // caterpillar trees of this many nodes or more take the scan kernels of tree_chain.cu
                                  // (upload_tree: POLEE_CHAIN_MIN_NODES, default 4096)
    void release();
};

std::string upload_tree(const TreeHost &th, TreeDev &td);

// The kernels that serve a tree's forward, backward and inverse passes (the rules: tree_route, tree_kernels.cu).
// polee_layout_info reports the route as its integer value, which include/polee_b200.h documents: keep the order.
enum class TreeRoute { Chain, DfsRun, PathProduct, SmemLevels, GlobalLevels };
TreeRoute tree_route(const TreeDev &td, int KP);

}  // namespace polee

// ------------------------------------------------------------------ the handle
struct polee_handle {
    polee_opts o;
    std::string err;
    int device = 0;
    int num_sms = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;  // H2D of nzval / ks overlapping the layout build
    cudaEvent_t copy_done = nullptr;
    cudaStream_t side_stream = nullptr;  // k3_mid runs beside the likelihood pass (fork / join inside the step graph)
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    int K = 0, KP = 0;  // draws, padded draws (power of two)

    // ---- matrix
    int64_t m = 0, n = 0, nnz = 0;
    int64_t m_pad = 0;          // rows in permuted order incl. class padding
    uint32_t *sell_idx = nullptr;
    float *sell_val = nullptr;
    int64_t sell_elems = 0;
    polee::RowTile *row_tiles = nullptr;
    int n_row_tiles = 0;
    uint32_t *row_perm = nullptr;  // original row -> permuted row
    float *row_weight = nullptr;   // ks per permuted row (nullable)
    uint32_t *csc_row = nullptr;
    float *csc_val = nullptr;
    polee::ColSeg *segs = nullptr;
    int n_segs = 0;
    polee::MultiCol *multi = nullptr;
    int n_multi = 0;
    int n_slots = 0;
    bool have_matrix = false;
    // fused layout (used instead of the SELL / CSC pair when `fused`)
    bool fused = false;
    unsigned char *ft_blob = nullptr;
    polee::FusedTileDesc *ft_desc = nullptr;
    int ft_tiles = 0;
    uint32_t ft_max_blob = 0, ft_max_E = 0, ft_max_rows = 0, ft_max_C = 0;
    uint32_t *ft_row_of_pos = nullptr;  // original row of every (tile-sorted) row position
    uint64_t ft_blob_bytes = 0;
    int64_t ft_parts = 0;            // (tile, column) partials
    polee::FusedUnit *ft_units = nullptr;
    int ft_nunits = 0;
    polee::FusedMulti *ft_multi = nullptr;
    int ft_nmulti = 0, ft_nlvl2 = 0;
    float *ft_row_weight = nullptr;  // ks per row, original order (nullable)
    float *ft_partial = nullptr;     // [ft_parts][KP]           (work buffer)
    double *ft_lvl2 = nullptr;       // [ft_nlvl2][KP]           (work buffer)
    int ft_grid = 0;

    // equivalence-class layout (the default; rows it cannot take go to the general layouts above as "rest" rows)
    unsigned char *ec_blob = nullptr;
    polee::EcTaskDesc *ec_desc = nullptr;
    int ec_tasks = 0;
    int64_t ec_rows = 0, ec_nnz = 0, ec_slots = 0, ec_classes = 0;  // rows / entries / padded row slots / classes it holds
    uint64_t ec_blob_bytes = 0;
    int64_t ec_parts = 0;               // (task, column) partials
    uint32_t *ec_row_of_slot = nullptr; // original row of every row slot, 0xFFFFFFFF = padding
    float *ec_slot_weight = nullptr;    // ks per row slot (nullable)
    polee::FusedUnit *ec_units = nullptr;
    int ec_nunits = 0;
    polee::FusedMulti *ec_multi = nullptr;
    int ec_nmulti = 0, ec_nlvl2 = 0;
    double *ec_partial = nullptr;       // [ec_parts][KP]   (work buffer)
    double *ec_lvl2 = nullptr;          // [ec_nlvl2][KP]   (work buffer)
    double *ec_lp_partial = nullptr;    // [ec_tasks][KP]   (work buffer)
    int ec_grid = 0;
    int ec_kind_end[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // tasks are ordered by LH, 8 first: end of each run
    int64_t gm = 0, gnnz = 0;           // rows / entries of the general ("rest") layouts; m, nnz are the whole matrix
    uint32_t *rest_row = nullptr;       // [gm] original row of every rest row (nullptr: rest = whole matrix)

    // ---- per-sample vectors
    float *efflen = nullptr;      // [n]
    float *efflen_adj = nullptr;  // Float32(n * (1/efflen))  likelihood.jl:105
    bool have_efflen = false;

    // ---- optional gene groups for gene_noninformative_prior! (likelihood.jl:114-159); only genes with >= 2 transcripts
    int64_t n_genes = 0;
    int64_t gene_n = 0;                 // n the groups were validated against
    int64_t *gene_ptr = nullptr;        // [n_genes + 1] offsets into gene_tx
    int32_t *gene_tx = nullptr;         // 0-based transcript ids
    double *gene_xl_grad = nullptr;     // [n][KP]
    double *gene_off_partial = nullptr; // [blocks][KP]
    double *gene_off = nullptr;         // [KP]
    int gene_KP = 0;

    // ---- tree
    polee::TreeHost th;
    polee::TreeDev td;
    bool have_tree = false;
    float *mu0_dev = nullptr;  // mu the fit starts from (inverse_transform! of the uniform composition), [n-1]

    // ---- parameters / ADAM state: [n-1] each
    float *mu = nullptr, *omega = nullptr, *alpha = nullptr;
    float *m_mu = nullptr, *m_omega = nullptr, *m_alpha = nullptr;
    float *v_mu = nullptr, *v_omega = nullptr, *v_alpha = nullptr;
    polee::StepCtl *d_step = nullptr;  // device step counters
    int *d_bad_step = nullptr;         // first step with a non-finite gradient, 0 = none
    unsigned int *d_leafS_counter = nullptr;  // k3_leaf_S: CTAs finished (the last one reduces; it resets the counter)
    int steps_enqueued = 0;
    polee_progress_fn progress_cb = nullptr;  // polee_set_progress
    void *progress_user = nullptr;
    int progress_every = 0;
    bool S_deferred = false;  // the forward kernel left S = sum_j x_j / efflen_j to k3_leaf_S (launched by launch_mid)
    bool reparam_ready = false;  // ys / zs0 of the next step have been produced (fused update + reparam kernel)

    // ---- per-step work buffers (layouts [item][KP])
    float *zs0 = nullptr, *zs = nullptr;  // [n-1][KP]
    double *ys = nullptr;                 // [n-1][KP]
    double *ygrad = nullptr;              // [n-1][KP]
    double *us = nullptr;                 // [N][KP]
    float2 *G = nullptr;                  // [N][KP]
    double *root_us = nullptr;            // [n_slots][KP] top -> bottom exchange (shared-memory tree kernels)
    float2 *root_G = nullptr;             // [n_slots][KP] bottom -> top exchange
    float *x = nullptr;                   // [n][KP]
    float *w = nullptr;                   // [m_pad][KP]
    double *g = nullptr;                  // [n][KP]  (all-reduced across ranks)
    float *g32 = nullptr;                 // [n][KP]  Float32 image of g for the all-reduce (multi-rank only)
    double *seg_partial = nullptr;        // [n_slots][KP]
    double *S_partial = nullptr;          // [n_tree_ctas][KP]
    double *S = nullptr;                  // [KP] sum_j x_j / efflen_j      (then lp[KP] follows in g_tail)
    double *lp_partial = nullptr;         // [n_row_tiles][KP]
    double *ladj_partial = nullptr;       // [3][n_tree_ctas + n_elem_ctas][KP]
    double *lp = nullptr;                 // [KP]
    double *elbo = nullptr;               // [num_steps]
    float *noise = nullptr;               // injected noise [steps][K][n-1]
    int64_t noise_steps = 0;
    float *grad_out = nullptr;            // [3][n-1] averaged grads (polee_lsn_draws)
    int work_KP = 0;                      // KP the work buffers were sized for
    int n_tree_ctas = 0;

    // ---- graph: one step, and STEP_GRAPH_STEPS consecutive steps (api.cu)
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t graph_exec = nullptr;
    cudaGraph_t graph_multi = nullptr;
    cudaGraphExec_t graph_multi_exec = nullptr;
    bool graph_warm = false;  // one uncaptured step has run with the current layouts
    bool pdl = true;          // step kernels launched with programmatic stream serialization (POLEE_PDL=0: plainly)

#ifdef POLEE_WITH_NCCL
    ncclComm_t comm = nullptr;
    // peer-memory all-reduce (peer_allreduce.cu): this rank's block, every rank's block as mapped here, floats per half
    void *peer_local = nullptr;
    void *peer_base[16] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                           nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    size_t peer_cap = 0;
    bool peer_ready = false;
#endif
    int nranks = 1, rank = 0;

    int fail(int code, const std::string &msg) {
        err = msg;
        return code;
    }
};

namespace polee {

int pad_k(int K);

// CALL with the padded draw count KP as the compile-time constant KPC; other KP fail the enclosing launch function
#define DISPATCH_KP(KP, CALL)                                                   \
    switch (KP) {                                                               \
        case 1: { constexpr int KPC = 1; CALL; } break;                         \
        case 2: { constexpr int KPC = 2; CALL; } break;                         \
        case 4: { constexpr int KPC = 4; CALL; } break;                         \
        case 8: { constexpr int KPC = 8; CALL; } break;                         \
        case 16: { constexpr int KPC = 16; CALL; } break;                       \
        default: return h->fail(POLEE_EINVAL, "unsupported number of MC draws (1..16)"); \
    }

// Dynamic shared memory opt-in.  The attribute is per FUNCTION and process-wide, and several handles (host threads)
// with different tile / tree sizes launch the same kernels: always raise it to the device limit, never to "what this
// launch needs", or one handle's smaller value makes another handle's launch fail.
// Copies and clears go through the handle's own (non-blocking) stream.  The legacy default stream does not order
// against it: a cudaMemset, or the DMA tail of a pageable cudaMemcpy, issued there can still be in flight when the next
// kernel of the handle starts -- harmless on an idle GPU, a data race as soon as other handles keep the GPU busy.
inline cudaError_t copy_sync(cudaStream_t st, void *dst, const void *src, size_t bytes, cudaMemcpyKind kind) {
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, kind, st);
    return e == cudaSuccess ? cudaStreamSynchronize(st) : e;
}

constexpr int MAX_SMEM_PER_CTA = 227 * 1024;  // sm_100: opt-in limit, static + dynamic
template <typename F>
inline cudaError_t allow_max_smem(F func) {
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, func);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_SMEM_PER_CTA - (int)a.sharedSizeBytes);
}

// Launch of a kernel that follows the pdl_wait() rule (device_utils.cuh) with programmatic stream serialization: it may
// start, and run its part before pdl_wait(), while the kernel before it on the stream drains.  Under stream capture the
// launch becomes a programmatic graph edge.  Only kernels that contain the wait go through here.  As with <<< >>>, a
// launch error surfaces through cudaGetLastError.
template <typename... P, typename... A>
inline void launch_pdl(const polee_handle *h, void (*kern)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                       A &&...args) {
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cfg.attrs = &attr;
    cfg.numAttrs = h->pdl ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kern, std::forward<A>(args)...);
}

// Device-wide synchronisation (explicit, or implied by cudaFree / cudaMalloc) is not permitted while ANY stream of the
// device is being captured into a graph, and it invalidates that capture -- also when the capture runs in another host
// thread on another handle.  Captures therefore hold this lock shared, device-wide operations hold it exclusively.
std::shared_mutex &capture_mutex();

// mem_cache.cu: caching device allocator (cudaMalloc / cudaFree semantics, freed blocks are kept for the next sample)
cudaError_t dmalloc(void **p, size_t bytes);
cudaError_t dfree(void *p);
void dtrim(int device);  // -1 = every device
size_t dcached_bytes(int device);
void dreport(const char *what);  // POLEE_SETUP_TIMING: allocator statistics since the last report, to stderr

// matrix_setup.cu
int setup_matrix_from_device_csc(polee_handle *h, int64_t m, int64_t n, const uint32_t *d_colptr,
                                 const uint32_t *d_rowval, const float *d_nzval, const int64_t *d_ks,
                                 const uint32_t *h_colptr_or_null, cudaEvent_t vals_ready_or_null);
void release_matrix(polee_handle *h);
// returns POLEE_OK with h->fused set, or POLEE_OK with h->fused == false when the row order has too little locality
int setup_fused_from_device_csc(polee_handle *h, int64_t m, int64_t n, int64_t nnz, const uint32_t *d_colptr,
                                const uint32_t *d_rowval, const float *d_nzval, const int64_t *d_ks,
                                const std::vector<uint32_t> &colptr, cudaEvent_t vals_ready_or_null);

// ec_setup.cu / ec_kernels.cu
struct EcRest {  // the rows the class layout did not take, as a CSC of their own (device arrays owned by the struct)
    int64_t m = 0, nnz = 0;
    uint32_t *colptr = nullptr, *rowval = nullptr;
    float *nzval = nullptr;
    int64_t *ks = nullptr;
    ~EcRest();
};
int setup_ec_from_device_csc(polee_handle *h, int64_t m, int64_t n, int64_t nnz, const uint32_t *d_colptr,
                             const uint32_t *d_rowval, const float *d_nzval, const int64_t *d_ks,
                             cudaEvent_t vals_ready_or_null, EcRest *rest);
void release_ec(polee_handle *h);
int ec_grid(polee_handle *h, int KP);
// g (+)= X_ec^T (1 / X_ec x); add_to_g: the general layouts already wrote their share of g
int launch_ec(polee_handle *h, const float *x, double *g, bool add_to_g, bool want_lp, double *lp_out, float *w_out, int KP, int K,
              bool lik_only = false);  // lik_only: the class kernel without its second stage (measurement)
void preload_ec_kernels(const polee_handle *h, int KP, int K);  // lazy-loading warm-up, see tree_kernels.cu
void preload_tree_kernels(int KP);
bool ec_math_f32(const polee_handle *h);  // opts.exact_accumulation != 2

// fused_kernels.cu
int fused_grid(polee_handle *h, int KP);
int launch_fused(polee_handle *h, const float *x, double *g, bool want_lp, double *lp_partial, float *w_out, int KP);

// sparse_kernels.cu
int launch_k1(polee_handle *h, const float *x, float *w, bool want_lp, double *lp_partial, int KP);
int launch_narrow(polee_handle *h, const double *in, float *out, size_t count);
int launch_widen(polee_handle *h, const float *in, double *out, size_t count);
int launch_k2(polee_handle *h, const float *w, double *g, int KP);
int launch_reduce_lp(polee_handle *h, const double *lp_partial, double *lp, int KP);

// tree_kernels.cu
int ensure_work_buffers(polee_handle *h, int KP);
void release_work_buffers(polee_handle *h);
int launch_reparam_fwd(polee_handle *h, int KP, int K, const float *noise, int64_t noise_steps, int want_ladj);
int launch_tree_fwd(polee_handle *h, int KP, int clamp_x, int want_S, int want_ladj);
int launch_mid(polee_handle *h, int KP, int advance, cudaStream_t st = nullptr);
int launch_tree_inv(polee_handle *h, int KP, const float *x_dev, double *us_tmp, double *ys_out, float *logu_tmp, double *ladj_out);
int launch_init_params(polee_handle *h, const double *ys0, int KP);
int launch_fill_f32(polee_handle *h, float *p, int64_t count, float v);
int launch_tree_bwd(polee_handle *h, int KP, bool with_ladj, bool apply_efflen, double *xgrad_out);
int launch_update(polee_handle *h, int KP, int K, bool do_adam, float *grad_out);
int launch_elem(polee_handle *h, int KP, int K, bool do_update, bool do_adam, bool do_reparam, const float *noise,
                int64_t noise_steps, int want_ladj, float *grad_out, int step0_fixed = -1, uint64_t seed_override = 0,
                int clamp_y = 1);
int elem_ctas(polee_handle *h, int KP);
int patch_leaf_records(polee_handle *h);
int launch_elbo(polee_handle *h, int KP, int K, bool have_lp);

// gene_prior.cu
int ensure_gene_buffers(polee_handle *h, int KP);
void release_gene_buffers(polee_handle *h);
int launch_gene_prior(polee_handle *h, int KP);
constexpr int PEER_MAX_RANKS = 16;
constexpr int PEER_ERR_TIMEOUT = -1001;  // lands in d_bad_step when a peer never arrives
void peer_release(polee_handle *h);
int launch_peer_allreduce(polee_handle *h, double *g, size_t count);
void drop_step_graph(polee_handle *h);

// tree_chain.cu (caterpillar trees)
int launch_chain_fwd(polee_handle *h, int KP, int clamp_x, const float *eff, double *Sp, int want_ladj, double *ladj_tree);
int launch_chain_bwd(polee_handle *h, int KP, bool with_ladj, const float *adj, double *xgrad_out);

}  // namespace polee
