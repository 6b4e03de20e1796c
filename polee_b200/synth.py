"""Synthetic RNASeqSample generator "polee-synth-v1" (SURVEY.md section 8d) and synthetic trees.

Used by tests (CPU, small) and bench.py (GPU, BASELINE.json shapes).  torch is used only to make the
data (on whatever device is asked for); nothing here is on the measured path.

Shape properties copied from the reference fixture (test/dataset/mBr_M_6w_1.likelihood-matrix.h5):
transcripts grouped into genes with contiguous ids; fragments emitted grouped by gene in gene order
(the reference sorts rows by genomic position, src/rnaseq_sample.jl:399-419); each fragment's transcript
set is drawn from a small per-gene pool of patterns; values f_i * exp(N(0, 1.5^2)) / efflen_j floored
just above MIN_FRAG_PROB = 1e-12 (src/constants.jl:45); every row non-empty; some empty columns.
"""
import numpy as np
import torch


def _gene_layout(n, gen, device, mean_gene_size=6.0):
    p = 1.0 / mean_gene_size
    ng = int(n / mean_gene_size * 1.5) + 16
    u = torch.rand(ng, generator=gen, device=device, dtype=torch.float64)
    sizes = 1 + torch.floor(torch.log(u.clamp_min(1e-300)) / np.log1p(-p)).to(torch.int64)
    sizes = sizes.clamp(1, 64)
    ends = torch.cumsum(sizes, 0)
    ngenes = int((ends < n).sum().item()) + 1
    sizes = sizes[:ngenes].clone()
    ends = ends[:ngenes].clone()
    if ngenes > 1:
        sizes[-1] = n - int(ends[-2].item())
    else:
        sizes[-1] = n
    starts = torch.cumsum(sizes, 0) - sizes
    return sizes, starts


def make_sample(m, n, seed=20260002, device="cpu", long_rows=False, patterns_per_gene=4, incl_prob=0.5, row_seed=None):
    """Returns dict with CSC arrays (1-based, torch int64 on `device`), nzval, efflens, gene layout.

    mean row length ~ 4 with the defaults; long_rows=True additionally turns 10 % of the rows into
    "repeat-family" rows spanning 64-512 transcripts (BASELINE config C4).

    row_seed: draw everything that belongs to the ROWS (their genes, patterns, values) from a second generator, so
    that blocks of rows made with different row_seed share the transcriptome (genes, effective lengths, abundances,
    pattern pools, repeat families) of `seed` -- how a rank makes its own block of C4 without the whole matrix ever
    existing anywhere.  None (default): one generator for everything, the sequence the golden fixtures were made with."""
    dev = torch.device(device)
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    genr = gen
    if row_seed is not None:
        genr = torch.Generator(device=dev)
        genr.manual_seed(row_seed)
    f64, i64 = torch.float64, torch.int64

    sizes, starts = _gene_layout(n, gen, dev)
    G = sizes.numel()
    gene_of_tx = torch.repeat_interleave(torch.arange(G, device=dev), sizes)
    efflen = torch.exp(7.0 + 0.8 * torch.randn(n, generator=gen, device=dev, dtype=f64)).clamp(1.0, 2e4).to(torch.float32)

    # abundance: gene weight LogNormal(0, 2), isoform split Dirichlet(0.5)
    wg = torch.exp(2.0 * torch.randn(G, generator=gen, device=dev, dtype=f64))
    gam = 0.5 * torch.randn(n, generator=gen, device=dev, dtype=f64) ** 2 + 1e-12  # Gamma(1/2, 1) = Z^2 / 2
    gsum = torch.zeros(G, device=dev, dtype=f64).index_add_(0, gene_of_tx, gam)
    theta = wg[gene_of_tx] * gam / gsum[gene_of_tx]
    gprob = torch.zeros(G, device=dev, dtype=f64).index_add_(0, gene_of_tx, theta * efflen.to(f64))
    gprob = gprob / gprob.sum()

    # fragments grouped by gene, in gene order
    cdf = torch.cumsum(gprob, 0)
    ug = torch.rand(m, generator=genr, device=dev, dtype=f64)
    row_gene = torch.searchsorted(cdf, ug).clamp_max(G - 1)
    row_gene, _ = torch.sort(row_gene)

    # per-gene pattern pool: pattern 0 = all transcripts of the gene, others random non-empty subsets
    P = patterns_per_gene
    bits = torch.rand(G, P, 64, generator=gen, device=dev) < incl_prob
    bits[:, 0, :] = True
    lane = torch.arange(64, device=dev)
    valid = lane[None, None, :] < sizes[:, None, None]
    bits &= valid
    first = torch.randint(0, 64, (G, P), generator=gen, device=dev) % sizes[:, None]
    bits[torch.arange(G, device=dev)[:, None], torch.arange(P, device=dev)[None, :], first] = True
    pat_len = bits.sum(-1).reshape(-1)                        # [G*P]
    pat_ptr = torch.cumsum(pat_len, 0) - pat_len
    nzb = bits.reshape(G * P, 64).nonzero()                   # sorted by (pattern, bit)
    pat_tx = starts[nzb[:, 0] // P] + nzb[:, 1]

    row_pat = row_gene * P + torch.randint(0, P, (m,), generator=genr, device=dev)
    row_len = pat_len[row_pat]

    fam_ptr = fam_tx = None
    if long_rows:
        F = 2048
        flen = torch.randint(64, 513, (F,), generator=gen, device=dev).clamp_max(max(1, n // 2))
        fstart = torch.randint(0, max(1, n - 4096), (F,), generator=gen, device=dev)
        fam_ptr = torch.cumsum(flen, 0) - flen
        # family f = flen[f] distinct ids in a window of 8 * flen after fstart (sorted, unique by construction)
        pos = torch.arange(int(flen.sum().item()), device=dev) - torch.repeat_interleave(fam_ptr, flen)
        jitter = torch.randint(0, 8, (pos.numel(),), generator=gen, device=dev)
        fam_tx = (torch.repeat_interleave(fstart, flen) + pos * 8 + jitter).clamp_max(n - 1)
        # clamp can create duplicates at the very end of the id range: make ids strictly increasing per family
        is_long = torch.rand(m, generator=genr, device=dev) < 0.10
        row_fam = torch.randint(0, F, (m,), generator=genr, device=dev)
        row_len = torch.where(is_long, flen[row_fam], row_len)

    row_ptr = torch.cumsum(row_len, 0) - row_len
    nnz = int(row_len.sum().item())
    ent_row = torch.repeat_interleave(torch.arange(m, device=dev), row_len)
    off = torch.arange(nnz, device=dev) - row_ptr[ent_row]
    ent_col = pat_tx[pat_ptr[row_pat[ent_row]] + off] if not long_rows else None
    if long_rows:
        base = torch.where(is_long[ent_row], fam_ptr[row_fam[ent_row]], torch.zeros((), device=dev, dtype=i64))
        col_l = fam_tx[(base + off).clamp_max(fam_tx.numel() - 1)]
        col_s = pat_tx[(pat_ptr[row_pat[ent_row]] + off).clamp_max(pat_tx.numel() - 1)]
        ent_col = torch.where(is_long[ent_row], col_l, col_s)
        # drop duplicate (row, col) pairs produced by the clamp at the end of the id range
        key = ent_row * n + ent_col
        keep = torch.ones(nnz, dtype=torch.bool, device=dev)
        keep[1:] = key[1:] != key[:-1]
        ent_row, ent_col = ent_row[keep], ent_col[keep]
        nnz = int(ent_row.numel())

    f_i = 1e-4 + (5e-3 - 1e-4) * torch.rand(m, generator=genr, device=dev, dtype=f64)
    val = f_i[ent_row] * torch.exp(1.5 * torch.randn(nnz, generator=genr, device=dev, dtype=f64)) / efflen[ent_col].to(f64)
    val = val.clamp_min(1.0001e-12).to(torch.float32)

    # CSR (row-major, ascending transcript inside a row) -> CSC: stable sort by column
    order = torch.sort(ent_col, stable=True).indices
    rowval = ent_row[order] + 1
    nzval = val[order]
    counts = torch.bincount(ent_col, minlength=n)
    colptr = torch.cat([torch.ones(1, dtype=i64, device=dev), 1 + torch.cumsum(counts, 0)])
    return {"m": m, "n": n, "nnz": nnz, "colptr": colptr, "rowval": rowval, "nzval": nzval, "efflens": efflen,
            "gene_sizes": sizes, "gene_starts": starts}


def to_numpy_sample(s):
    """CSC arrays as the uint32 / float32 numpy arrays of a Julia SparseMatrixCSC{Float32,UInt32}."""
    return {"m": s["m"], "n": s["n"], "colptr": s["colptr"].cpu().numpy().astype(np.uint32),
            "rowval": s["rowval"].cpu().numpy().astype(np.uint32), "nzval": s["nzval"].cpu().numpy(),
            "efflens": s["efflens"].cpu().numpy()}


# ------------------------------------------------------------------------------------------ trees
def tree_from_nested(root, n):
    """DFS order with the RIGHT branch first (order_nodes, src/hclust.jl:361-389) of a nested tree given as
    leaves (int, 1-based transcript id) and internal nodes (left, right) tuples -> (node_parent_idxs, node_js)."""
    N = 2 * n - 1
    pi = np.zeros(N, np.int32)
    js = np.zeros(N, np.int32)
    stack = [(root, 0)]
    pos = 0
    while stack:
        node, parent = stack.pop()
        pi[pos] = parent
        pos += 1
        if isinstance(node, tuple):
            js[pos - 1] = 0
            stack.append((node[0], pos))  # left pushed first ...
            stack.append((node[1], pos))  # ... so the right child is popped (emitted) next
        else:
            js[pos - 1] = node
    assert pos == N
    return pi, js


def balanced_tree(n, gene_sizes=None):
    """Balanced-by-gene binary tree (SURVEY 8d tree (i)): balanced over genes, then balanced inside each gene."""
    def bal(items):
        while len(items) > 1:
            nxt = [(items[i], items[i + 1]) for i in range(0, len(items) - 1, 2)]
            if len(items) % 2:
                nxt.append(items[-1])
            items = nxt
        return items[0]

    if gene_sizes is None:
        return tree_from_nested(bal(list(range(1, n + 1))), n)
    gene_sizes = [int(v) for v in np.asarray(gene_sizes)]
    assert sum(gene_sizes) == n
    genes, j = [], 1
    for sz in gene_sizes:
        genes.append(bal(list(range(j, j + sz))))
        j += sz
    return tree_from_nested(bal(genes), n)


def random_tree(n, seed=0):
    """rand_tree_nodes (src/hclust.jl:439-454): repeatedly join two random subtrees."""
    rng = np.random.default_rng(seed)
    items = list(range(1, n + 1))
    while len(items) > 1:
        i = rng.integers(len(items))
        a = items[i]
        items[i] = items[-1]
        items.pop()
        j = rng.integers(len(items))
        b = items[j]
        items[j] = (a, b)
    return tree_from_nested(items[0], n)


def spine_tree(n_spine, every):
    """(node_parent_idxs, node_js) of a caterpillar of n_spine internal nodes in which every `every`-th right-hand leaf
    is replaced by a 3-leaf subtree, in DFS pre-order.  With n_spine above 1 024 it is deep (no DFS-run inputs, more
    than 1 024 ancestors per path group, so no root-path tables) and not a caterpillar (no chain scans), and its top
    part fits in shared memory: the tree kernels' shared-memory level route."""
    pi, js = [], []

    def add(parent, leaf):
        pi.append(parent)
        js.append(leaf)
        return len(pi)                                # 1-based index of the new node

    leaves, parent = 0, 0
    for s in range(n_spine):
        me = add(parent, 0)
        if s % every == every - 1:                    # the first child of a node is its right child
            a = add(me, 0)
            add(a, leaves + 1)
            b = add(a, 0)
            add(b, leaves + 2)
            add(b, leaves + 3)
            leaves += 3
        else:
            leaves += 1
            add(me, leaves)
        parent = me
    add(parent, leaves + 1)
    return np.array(pi, np.int32), np.array(js, np.int32)
