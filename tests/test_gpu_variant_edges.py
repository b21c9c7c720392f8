"""Every kernel variant at the edges of its dispatch rule: the generic-D and rank-1 CBOW paths at odd D, long windows
through the fused kernel's four gather x scatter forms and through the gene-slab passes, and the walk sampler on graphs
whose degrees, node counts, weights, path lengths and walker counts sit on its chunk / packing / tile boundaries.

References: the C oracle bit-exact for walks; float64 NumPy restatements of the step for CBOW, at 2e-5 relative to the
largest entry for gradients and 1e-4 for vectors (tests/test_gpu_cbow.py)."""
import math

import numpy as np
import pytest

import oracle
from tests import helpers

pytestmark = pytest.mark.gpu
RTOL_GRAD, RTOL_VEC = 2e-5, 1e-4
LR, B1, B2, EPS = 0.005, 0.9, 0.999, 1e-8


@pytest.fixture(scope="module")
def g2v():
    import torch
    assert torch.cuda.is_available()
    import g2vec_b200
    return g2vec_b200


def rel_max(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


# ------------------------------------------------------------------------------------------------ CBOW
def windows(V, lens, seed, special=None):
    """CSR windows of distinct, ascending genes with the given lengths; special = {gene: count} puts those genes
    (which must be below every other gene id used) into the first `count` windows."""
    rs = np.random.RandomState(seed)
    lo = 0 if not special else max(special) + 1
    rows = [np.sort(rs.choice(np.arange(lo, V), size=l, replace=False)) for l in lens]
    for g, cnt in sorted((special or {}).items(), reverse=True):
        for i in range(cnt):
            rows[i] = np.concatenate([[g], rows[i]])
    rowptr = np.zeros(len(rows) + 1, np.int32)
    rowptr[1:] = np.cumsum([len(r) for r in rows])
    gene = np.concatenate(rows).astype(np.int32) if rows else np.zeros(0, np.int32)
    return rowptr, gene, (rs.rand(len(rows)) < 0.5).astype(np.uint8)


def step64(rowptr, gene, label, win, V, D, W0, Wo0, reduce):
    """One forward/backward of the modified CBOW (G2Vec.py:239-244) in float64 over the listed windows:
    (g_ih, g_ho, loss sum, correct count, c = X^T dO with the mean scale)."""
    W, Wo = W0.astype(np.float64), Wo0.astype(np.float64)
    g_ih = np.zeros((V, D)); g_ho = np.zeros(D); c = np.zeros(V)
    loss, nc, N = 0.0, 0, len(win)
    for n in win:
        gs = gene[rowptr[n]:rowptr[n + 1]]
        scale = 1.0 / len(gs) if (reduce == "mean" and len(gs)) else 1.0
        h = W[gs].sum(0) * scale
        o = float(h @ Wo)
        y = float(label[n])
        loss += max(o, 0.0) - o * y + math.log1p(math.exp(-abs(o)))
        nc += int((o > 0) == (y != 0))
        dO = (1.0 / (1.0 + math.exp(-o)) - y) / N
        g_ho += h * dO
        g_ih[gs] += dO * scale * Wo                                   # genes of a window are distinct
        c[gs] += dO * scale
    return g_ih, g_ho, loss, nc, c


def adam64(w, g, t=1):
    m = (1 - B1) * g
    v = (1 - B2) * g * g
    return w - LR * math.sqrt(1 - B2 ** t) / (1 - B1 ** t) * m / (np.sqrt(v) + EPS)


def updated64(W0, Wo0, g_ih, g_ho, optimizer):
    if optimizer == "adam":
        return adam64(W0.astype(np.float64), g_ih), adam64(Wo0.astype(np.float64), g_ho)
    return W0 - LR * g_ih, Wo0 - LR * g_ho


def check_step(m, ref, W0, Wo0, optimizer, acc_slot_eval=2, n_tol=2):
    """fwdbwd + evaluate have run on model m (not yet updated): gradients, loss, counts; then update and vectors."""
    import torch
    torch.cuda.synchronize()
    g_ih, g_ho, loss, nc, _ = ref
    acc = m.acc.cpu()
    assert rel_max(m.g_ih.cpu().numpy(), g_ih) < RTOL_GRAD and rel_max(m.g_ho.cpu().numpy(), g_ho) < RTOL_GRAD
    assert abs(m.loss_sum(acc) - loss) < 1e-5 * max(1.0, abs(loss))
    assert abs(int(acc[1]) - nc) <= n_tol and abs(int(acc[acc_slot_eval]) - nc) <= n_tol
    m.update()
    torch.cuda.synchronize()
    W, Wo = updated64(W0, Wo0, g_ih, g_ho, optimizer)
    assert rel_max(m.W_ih.cpu().numpy(), W) < RTOL_VEC and rel_max(m.W_ho.cpu().numpy(), Wo) < RTOL_VEC
    assert float(m.g_ih.abs().max()) == 0.0 and float(m.g_ho.abs().max()) == 0.0


GENERIC_LENS = [0, 1, 31, 32, 33, 257, 0, 1, 31, 32, 33, 257]


@pytest.mark.parametrize("optimizer,reduce", [("adam", "sum"), ("sgd", "mean")])
@pytest.mark.parametrize("D", [1, 3, 33, 129, 1000])
def test_generic_d_rows_kernel_short_and_long_windows(g2v, D, optimizer, reduce):
    """cbow_rows_generic_kernel (D not 128/256/512) and the scalar tail of cbow_update_kernel over W_ih (V*D odd for
    D = 1, 3, 33, 129): windows of 0, 1, 31, 32, 33, 257 and 4096 genes (V = 5001, so the 4096 genes are distinct)."""
    import torch
    V = 5001
    rs = np.random.RandomState(D)
    lens = GENERIC_LENS + [4096, 4095, 4096] + list(rs.randint(1, 60, size=200))
    rowptr, gene, label = windows(V, lens, seed=D)
    W0, Wo0 = helpers.init_weights(V, D, D + 1)
    win = rs.permutation(len(lens)).astype(np.int64)
    m = g2v.CbowModel(rowptr, gene, label, V, D, W0, Wo0, optimizer=optimizer, reduce=reduce, lr=LR)
    wd = torch.from_numpy(win.astype(np.int32)).cuda()
    m.fwdbwd(wd, len(win))
    m.evaluate(wd, 2)
    check_step(m, step64(rowptr, gene, label, win, V, D, W0, Wo0, reduce), W0, Wo0, optimizer)


def test_generic_d_above_the_shared_memory_limit_is_refused(g2v):
    """The generic kernel keeps 8 warps x 2 rows of D floats in shared memory (64*D bytes): D = 4000 is above the
    opt-in limit, and fwdbwd / evaluate must fail with a message instead of launching."""
    import torch
    from g2vec_b200 import _capi
    V, D = 3, 4000
    m = g2v.CbowModel(np.array([0, 2, 3], np.int32), np.array([0, 2, 1], np.int32), np.array([0, 1], np.uint8), V, D,
                      np.zeros((V, D), np.float32), np.zeros(D, np.float32))
    torch.cuda.synchronize()
    before = _capi.launch_count()
    with pytest.raises(RuntimeError, match="too large"):
        m.fwdbwd(None, 2, win_begin=0, n_win=2)
    with pytest.raises(RuntimeError, match="too large"):
        m.evaluate(None, 2, win_begin=0, n_win=2)
    assert _capi.launch_count() == before


@pytest.mark.parametrize("optimizer,reduce", [("adam", "sum"), ("sgd", "mean")])
@pytest.mark.parametrize("D", [1, 3, 33, 129, 1000])
def test_rank1_generic_d_atomic_and_csc_forms(g2v, D, optimizer, reduce):
    """Collapsed trainer at D not 128/256/512 (r1_prepare's scalar loop, r1_update_kernel<0>): genes 0..6 occur in
    exactly 1, 32, 96, 97, 128, 129 and 1000 windows -- the edges of r1_csc_reduce_kernel's 128-wide unrolled loop
    and its remainder -- and the atomic and CSC backward forms both equal the float64 step."""
    import torch
    V, N = 257, 1100
    counts = {0: 1, 1: 32, 2: 96, 3: 97, 4: 128, 5: 129, 6: 1000}
    rs = np.random.RandomState(D + 3)
    rowptr, gene, label = windows(V, list(rs.randint(0, 40, size=N)), seed=D + 3, special=counts)
    assert [int((gene == g).sum()) for g in range(7)] == [counts[g] for g in range(7)]
    W0, Wo0 = helpers.init_weights(V, D, D)
    win = np.arange(N, dtype=np.int64)
    g_ih, g_ho, loss, nc, c64 = step64(rowptr, gene, label, win, V, D, W0, Wo0, reduce)
    W, Wo = updated64(W0, Wo0, g_ih, g_ho, optimizer)
    wd = torch.arange(N, dtype=torch.int32, device="cuda")
    cs = []
    for csc in (False, True):
        m = g2v.CbowModel(rowptr, gene, label, V, D, W0, Wo0, optimizer=optimizer, reduce=reduce, lr=LR, algo="rank1")
        if csc:
            m.prepare_csc(wd)
        m.fwdbwd(wd, N)
        torch.cuda.synchronize()
        acc = m.acc.cpu()
        c = m.c.cpu().numpy().copy()
        cs.append(c)
        assert rel_max(c, c64) < RTOL_GRAD, csc
        assert abs(m.loss_sum(acc) - loss) < 1e-5 * max(1.0, abs(loss)) and abs(int(acc[1]) - nc) <= 2
        m.update()
        torch.cuda.synchronize()
        assert rel_max(m.W_ih.cpu().numpy(), W) < RTOL_VEC and rel_max(m.W_ho.cpu().numpy(), Wo) < RTOL_VEC, csc
        assert float(m.c.abs().max()) == 0.0
        s_want = m.W_ih.cpu().numpy().astype(np.float64) @ m.W_ho.cpu().numpy().astype(np.float64)
        assert np.abs(m.s.cpu().numpy() - s_want).max() < 1e-5 * max(1.0, np.abs(s_want).max())
    assert np.abs(cs[1] - cs[0]).max() <= 1e-5 * np.abs(cs[0]).max()


# lengths 33..4096 including every residue modulo R = 4 / VEC (rows per TMA-gather stage: 4, 2, 1)
LONG_LENS = [33, 34, 35, 36, 37, 63, 64, 65, 127, 128, 129, 255, 257, 1023, 1025, 2047, 4093, 4094, 4095, 4096]


@pytest.mark.parametrize("gather,scatter", [("ldg", "red"), ("tma", "red"), ("ldg", "tma"), ("tma", "tma")])
@pytest.mark.parametrize("D", [128, 256, 512])
def test_fused_kernel_long_windows_every_form(g2v, monkeypatch, D, gather, scatter):
    """cbow_rows_kernel with windows of 33..4096 genes in all four G2V_CBOW_GATHER x G2V_CBOW_SCATTER forms: the TMA
    gather's chunk loop and stage parity over many chunks, its partial last chunk, and the 32-gene LDG batches."""
    import torch
    monkeypatch.setenv("G2V_CBOW_GATHER", gather)
    monkeypatch.setenv("G2V_CBOW_SCATTER", scatter)
    V = 5001
    rs = np.random.RandomState(D)
    lens = LONG_LENS + list(rs.randint(0, 80, size=150))
    rowptr, gene, label = windows(V, lens, seed=D + len(gather) + len(scatter))
    W0, Wo0 = helpers.init_weights(V, D, 7)
    win = rs.permutation(len(lens)).astype(np.int64)
    m = g2v.CbowModel(rowptr, gene, label, V, D, W0, Wo0, lr=LR)
    wd = torch.from_numpy(win.astype(np.int32)).cuda()
    m.fwdbwd(wd, len(win))
    m.evaluate(wd, 2)
    check_step(m, step64(rowptr, gene, label, win, V, D, W0, Wo0, "sum"), W0, Wo0, "adam")


def slab_windows(V, S, seed):
    """Windows that span every slab (up to 4096 genes), windows entirely inside one slab, empty windows, short
    random ones."""
    rs = np.random.RandomState(seed)
    per = -(-V // S)
    rows = [np.sort(rs.choice(V, size=l, replace=False)) for l in [min(V, 4096), min(V, 4095), min(V, 2000)]]
    rows += [np.arange(V)] if V <= 4096 else []                      # every gene
    for s in range(S):                                               # inside slab s only (the last one is short)
        lo, hi = s * per, min(V, (s + 1) * per)
        if hi > lo:
            rows += [np.sort(rs.choice(np.arange(lo, hi), size=min(hi - lo, k), replace=False)) for k in (1, 33, 300)]
    rows += [np.zeros(0, np.int64)] * 3
    rows += [np.sort(rs.choice(V, size=l, replace=False)) for l in rs.randint(1, min(V, 80), size=200)]
    rowptr = np.zeros(len(rows) + 1, np.int32)
    rowptr[1:] = np.cumsum([len(r) for r in rows])
    return rowptr, np.concatenate(rows).astype(np.int32), (rs.rand(len(rows)) < 0.5).astype(np.uint8)


@pytest.mark.parametrize("scatter", ["red", "tma"])
@pytest.mark.parametrize("V,D,slabs,group,reduce", [(5001, 128, 7, 2, "sum"), (5001, 256, 4, 1, "mean"),
                                                    (5001, 512, 3, 3, "sum"), (37, 128, 64, 2, "sum"),
                                                    (37, 512, 37, 1, "mean")])
def test_slab_passes_long_windows_short_last_slab(g2v, monkeypatch, V, D, slabs, group, reduce, scatter):
    """csrc/g2v_cbow_slab.cu with both G2V_CBOW_SLAB_SCATTER forms (the TMA form keeps two staging rows per warp and
    waits with wait_group.read 1): V = 5001 is not a multiple of the slab count (short last slab); with
    G2V_CBOW_SLABS >= V = 37 the plan clamps to V slabs of one gene.  Against the fused kernel and float64."""
    import torch
    monkeypatch.setenv("G2V_CBOW_SLAB_SCATTER", scatter)
    monkeypatch.setenv("G2V_CBOW_SLABS", str(slabs))
    monkeypatch.setenv("G2V_CBOW_SLAB_FWD_GROUP", str(group))
    S = min(slabs, V)
    rowptr, gene, label = slab_windows(V, S, seed=V + D + slabs)
    N = len(rowptr) - 1
    W0, Wo0 = helpers.init_weights(V, D, 11)
    win = np.random.RandomState(2).permutation(N).astype(np.int64)
    wd = torch.from_numpy(win.astype(np.int32)).cuda()
    m = g2v.CbowModel(rowptr, gene, label, V, D, W0, Wo0, reduce=reduce, lr=LR)
    assert m.prepare_slabs(wd) and m._n_slabs == S
    m.fwdbwd(wd, N)
    m.evaluate(wd, 2)
    torch.cuda.synchronize()
    g_slab = m.g_ih.cpu().numpy().copy()
    monkeypatch.delenv("G2V_CBOW_SLABS")
    f = g2v.CbowModel(rowptr, gene, label, V, D, W0, Wo0, reduce=reduce, lr=LR)
    assert not f.prepare_slabs(wd)
    f.fwdbwd(wd, N)
    torch.cuda.synchronize()
    assert rel_max(g_slab, f.g_ih.cpu().numpy()) < RTOL_GRAD
    assert rel_max(m.g_ho.cpu().numpy(), f.g_ho.cpu().numpy()) < RTOL_GRAD
    check_step(m, step64(rowptr, gene, label, win, V, D, W0, Wo0, reduce), W0, Wo0, "adam")


# ----------------------------------------------------------------------------------------------- walks
def hash_fits(L, canonical):
    """Shared memory of the hash visited set (8 warps x (path + >= 3L slots)) against the B200's 227 KB opt-in."""
    lpad = (L + 31) & ~31
    if canonical:
        lpad = 32
        while lpad < L:
            lpad <<= 1
    h = 64
    while h < 3 * L:
        h <<= 1
    return 8 * 4 * (lpad + h) <= 227 * 1024


def sorted_rows(nodes, lens, pad):
    out = np.full_like(nodes, pad)
    for i, (r, n) in enumerate(zip(nodes, lens)):
        out[i, :n] = np.sort(r[:n])
    return out


def walk_variants(g2v, monkeypatch, rp, col, q, L, seed=77, group=1, walker_begin=0, walker_end=None, walker_stride=1,
                  want_layout=None):
    """Every layout (CSR arrays / {col,qw} pairs / packed edges with one or two walkers per warp) x visited set
    (bitmap / hash) x visit order / fused canonical rows, each bit-exact against the C oracle.  Returns the
    oracle's lengths."""
    import torch
    from g2vec_b200 import paths
    V = len(rp) - 1
    end = 2 * V if walker_end is None else walker_end
    want, wl = oracle.walks(rp, col, q, L, seed, group, walker_begin, end, walker_stride)
    kw = dict(seed=seed, group=group, walker_begin=walker_begin, walker_end=end, walker_stride=walker_stride)
    graphs = {}
    monkeypatch.setenv("G2V_WALK_LAYOUT", "e8")
    graphs["e8"] = g2v.WalkGraph(rp, col, qw=q)
    monkeypatch.delenv("G2V_WALK_LAYOUT")
    graphs["default"] = g2v.WalkGraph(rp, col, qw=q)
    assert graphs["e8"].layout == 1
    if want_layout is not None:
        assert graphs["default"].layout == want_layout
    forms = [("csr", "default", None), ("e8", "e8", None)]
    if graphs["default"].layout == 2:
        forms += [("e4-pair", "default", "16"), ("e4-single", "default", "32")]
    for name, gname, tile in forms:
        g = graphs[gname]
        for vis in ("bitmap", "hash"):
            for canonical in ((False,) if name == "csr" else (False, True)):
                if vis == "hash" and not hash_fits(L, canonical):
                    continue
                monkeypatch.setenv("G2V_WALK_VISITED", vis)
                if tile:
                    monkeypatch.setenv("G2V_WALK_TILE", tile)
                else:
                    monkeypatch.delenv("G2V_WALK_TILE", raising=False)
                if canonical:
                    rows, lens, key = g2v.generate_paths(g, L, 1, canonical=True, **kw)
                    _, key2 = paths._canon(torch.from_numpy(want).cuda())
                    torch.cuda.synchronize()
                    assert (lens.cpu().numpy() == wl).all(), (name, vis, "canonical")
                    assert (rows.cpu().numpy() == sorted_rows(want, wl, paths.PAD)).all(), (name, vis, "canonical")
                    assert (key.cpu().numpy() == key2.cpu().numpy()).all(), (name, vis, "key")
                else:
                    nodes, lens = g2v.generate_paths(g, L, 1, plain_csr=(name == "csr"), **kw)
                    torch.cuda.synchronize()
                    assert (lens.cpu().numpy() == wl).all() and (nodes.cpu().numpy() == want).all(), (name, vis)
    monkeypatch.delenv("G2V_WALK_VISITED", raising=False)
    monkeypatch.delenv("G2V_WALK_TILE", raising=False)
    return wl


def csr(rows, V):
    rp = np.zeros(V + 1, np.int32)
    rp[1:] = np.cumsum([len(r) for r in rows])
    return rp, (np.concatenate(rows) if rows else np.zeros(0)).astype(np.int32)


DEGREES = [0, 1, 2, 3, 4, 5, 31, 32, 33, 63, 64, 65, 127, 128, 129, 191, 192, 193, 255, 256, 257]


def degree_graph(seed=0):
    """V = 300: nodes 0..41 have degrees DEGREES twice over, the others cycle through the degrees >= 31.  Every edge
    points at a node of degree >= 31, so walks stay in a densely interlinked core: long walks leave whole
    32/64-neighbour chunks visited and the draw lands in the first chunk, in a register chunk or in the re-read
    tail."""
    V = 300
    rs = np.random.RandomState(seed)
    deg = [DEGREES[v % len(DEGREES)] if v < 2 * len(DEGREES) else DEGREES[6 + v % (len(DEGREES) - 6)] for v in range(V)]
    core = np.array([v for v in range(V) if deg[v] >= 31])
    rows = []
    for v in range(V):
        rows.append(np.sort(rs.choice(core[core != v], size=deg[v], replace=False)))
    rp, col = csr(rows, V)
    return rp, col, rs


@pytest.mark.parametrize("weights", ["pcc", "pcc-extremes", "up-to-2^24"])
def test_walk_row_degrees_at_chunk_boundaries(g2v, monkeypatch, weights):
    """Rows of 0..5, 31..33, 63..65, 127..129, 191..193, 255..257 neighbours.  PCC-range weights pack as 16+16-bit
    edges; weights exactly 32768 / 65536 still do; weights up to 2^24 (exactly 2^24 on every row of 64 and 257
    neighbours: chunk totals of 2^30, a row total above 2^32 on the long-row path) take the {col, qw} pairs."""
    rp, col, rs = degree_graph()
    E = len(col)
    if weights == "pcc":
        q = rs.randint(32769, 65537, size=E).astype(np.uint32)
    elif weights == "pcc-extremes":
        q = np.where(rs.rand(E) < 0.5, 32768, 65536).astype(np.uint32)
    else:
        q = rs.randint(1, 2**24 + 1, size=E).astype(np.uint32)
        deg = np.diff(rp)
        for v in np.nonzero((deg == 64) | (deg == 257))[0]:
            q[rp[v]:rp[v + 1]] = 2**24
    wl = walk_variants(g2v, monkeypatch, rp, col, q, 300, want_layout=2 if weights != "up-to-2^24" else 1)
    assert wl.max() > 200 and (wl == 1).any()                       # long walks and dead ends both occur


@pytest.mark.parametrize("V", [31, 32, 63, 64, 65, 95, 96])
def test_walk_small_graphs_sentinel_word(g2v, monkeypatch, V):
    """V = 0 or 31 (mod 32): the packed layout's sentinel node V is bit 0 of a new bitmap word or bit 31 of the last
    one; complete graphs minus a few edges, walks up to V nodes."""
    rs = np.random.RandomState(V)
    rows = [np.sort(rs.choice(np.delete(np.arange(V), v), size=rs.randint(V // 2, V), replace=False)) for v in range(V)]
    rp, col = csr(rows, V)
    q = rs.randint(32768, 65537, size=len(col)).astype(np.uint32)
    wl = walk_variants(g2v, monkeypatch, rp, col, q, V, walker_end=4 * V, want_layout=2)
    assert wl.max() >= V - 2


def big_sparse_graph(V, deg, seed):
    """V nodes, `deg` random out-edges each, plus edges into the highest node ids (so that node V-1 -- whose bit
    shares the sentinel's bitmap word -- is visited)."""
    rs = np.random.RandomState(seed)
    src = np.repeat(np.arange(V, dtype=np.int64), deg)
    dst = rs.randint(0, V, size=V * deg)
    hi = np.arange(V - 40, V)
    src = np.concatenate([src, rs.randint(0, V, size=4000), np.repeat(hi, 3)])
    dst = np.concatenate([dst, rs.choice(hi, size=4000), rs.randint(0, V, size=120)])
    keep = src != dst
    from g2vec_b200 import graph
    rp, col, _ = graph.csr_from_edges(src[keep], dst[keep], np.ones(int(keep.sum()), np.float32), V)
    q = rs.randint(32769, 65537, size=len(col)).astype(np.uint32)
    return rp, col, q


def test_walk_v_65535_packs_with_the_sentinel_at_0xffff(g2v, monkeypatch):
    """V = 65535 is the largest graph whose sentinel node id V fits the 16-bit column (bitmap word 2047, bit 31).  The
    bitmap (67 KB per CTA, above the 56 KB budget, so the hash set is the default here) and two walkers per warp are
    forced too; the pair kernel's own shared-memory budget then sends the launch to the one-walker kernel."""
    rp, col, q = big_sparse_graph(65535, 6, seed=1)
    wl = walk_variants(g2v, monkeypatch, rp, col, q, 40, walker_begin=3, walker_end=2 * 65535, walker_stride=7,
                       want_layout=2)
    assert wl.max() == 40


def test_walk_v_65536_takes_the_pair_layout(g2v, monkeypatch):
    """One node more and the sentinel no longer fits 16 bits: PCC-range weights must still give layout 1."""
    rp, col, q = big_sparse_graph(65536, 6, seed=2)
    wl = walk_variants(g2v, monkeypatch, rp, col, q, 40, walker_begin=1, walker_end=65536, walker_stride=5,
                       want_layout=1)
    assert wl.max() == 40


def band_graph(V, fwd=8, back=2, seed=0):
    """i -> i-back..i-1 and i+1..i+fwd: walks run forward and most reach L = 4096; the back edges point at nodes the
    walk has usually visited."""
    rows = [np.concatenate([np.arange(max(0, v - back), v), np.arange(v + 1, min(V, v + fwd + 1))]) for v in range(V)]
    rp, col = csr(rows, V)
    return rp, col, np.random.RandomState(seed).randint(32768, 65537, size=len(col)).astype(np.uint32)


@pytest.mark.parametrize("L", [31, 32, 33, 63, 64, 65, 127, 128, 129, 4095, 4096])
def test_walk_path_length_boundaries(g2v, monkeypatch, L):
    """Lpad (L rounded to 32, or to the bitonic network's power of two for canonical rows), the bitonic padding and
    the hash set of >= 3L slots, on a graph where walks reach L."""
    rp, col, q = band_graph(40000)
    n = 2000 if L < 4000 else 150
    wl = walk_variants(g2v, monkeypatch, rp, col, q, L, walker_begin=11, walker_end=11 + 97 * n, walker_stride=97,
                       want_layout=2)
    assert (wl == L).mean() > 0.8


@pytest.mark.parametrize("begin,end,stride", [(0, 1, 1), (5, 7, 1), (3, 48, 3), (100, 117, 1), (7, 436, 13),
                                              (1, 2000 * 2, 2)])
def test_walk_pair_kernel_walker_counts(g2v, monkeypatch, begin, end, stride):
    """Two walkers per warp (16-lane tiles, 16 walkers per CTA): 1, 2, 15, 17 and 33 walkers leave tiles and whole
    warps without a walker; a strided range over both repetitions."""
    rp, col, w = helpers.random_graph(2000, 20, seed=4, dead_frac=0.1)
    q = np.minimum(oracle.quantise_weights(w), 65536)             # |PCC| range: packed edges
    wl = walk_variants(g2v, monkeypatch, rp, col, q, 80, walker_begin=begin, walker_end=end, walker_stride=stride,
                       want_layout=2)
    assert len(wl) == (end - begin + stride - 1) // stride


def test_weights_above_2_to_the_24_are_refused(g2v):
    """The sampler's contract is qw <= 2^24 (32-bit chunk totals of up to 64 weights).  WalkGraph and
    g2v_walk_prepare / g2v_walk_host refuse a larger weight with a message; no walk is launched on such a graph."""
    import torch
    from g2vec_b200 import _capi
    lib = _capi.load()
    rp = np.array([0, 2, 3, 3], np.int32); col = np.array([1, 2, 0], np.int32)
    q = np.array([2**24 + 1, 40000, 50000], np.uint32)
    for bad in (q, q.view(np.int32), torch.from_numpy(q.view(np.int32)).cuda(),
                np.array([40000, 40000, -1], np.int32)):
        with pytest.raises(ValueError, match="2\\^24"):
            g2v.WalkGraph(rp, col, qw=bad)
    nodes = np.zeros((3, 4), np.int32); lens = np.zeros(3, np.int32)
    before = _capi.launch_count()
    rc = lib.g2v_walk_host(rp.ctypes.data, col.ctypes.data, q.ctypes.data, 3, 3, 4, 0, 0, 0, 3, 1,
                           nodes.ctypes.data, lens.ctypes.data)
    assert rc == 2 and b"2^24" in lib.g2v_last_error()
    assert _capi.launch_count() == before + 1                       # the weight check only
    g = g2v.WalkGraph(rp, col, qw=np.array([2**24, 40000, 50000], np.uint32))    # the limit itself is allowed
    assert g.layout == 1
