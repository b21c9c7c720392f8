"""GPU parity of HOT PATH 1 (walk sampler) against the oracle: BIT-EXACT node sequences.
All calls go through the C ABI (g2vec_b200._capi -> libg2vec_b200.so)."""
import os

import numpy as np
import pytest

import oracle
from tests import helpers

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def g2v():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import g2vec_b200
    return g2vec_b200


def run_gpu(g2v, rp, col, q, L, reps, seed, group, **kw):
    import torch
    g = g2v.WalkGraph(rp, col, qw=q)
    nodes, lens = g2v.generate_paths(g, L, reps, seed=seed, group=group, **kw)
    torch.cuda.synchronize()
    return nodes.cpu().numpy(), lens.cpu().numpy()


def test_philox_stream_is_curand_and_oracle(g2v):
    import torch
    from g2vec_b200 import _capi
    lib = _capi.load()
    for seed, sub in [(0, 0), (12345, (1 << 40) + 777), (2**63 + 5, 2**44 + 123456789)]:
        a = torch.zeros(64, dtype=torch.int64, device="cuda"); b = torch.zeros_like(a)
        _capi.check(lib.g2v_test_draws(seed, sub, 64, a.data_ptr(), 0), "g2v_test_draws")
        _capi.check(lib.g2v_test_curand_draws(seed, sub, 64, b.data_ptr(), 0), "g2v_test_curand_draws")
        torch.cuda.synchronize()
        a = a.cpu().numpy().view(np.uint64); b = b.cpu().numpy().view(np.uint64)
        assert (a == b).all(), "kernel Philox != curand Philox4_32_10"
        assert [int(x) for x in a] == [oracle.draw64(seed, sub, s) for s in range(64)]


def test_small_golden_graphs_bit_exact(g2v, golden_dir):
    z = np.load(os.path.join(golden_dir, "walk_small.npz"))
    from oracle import legacy
    for i in range(int(z["n_cases"])):
        A = z["A%d" % i]; L, iters, seed = (int(x) for x in z["meta%d" % i])
        rp, col, w = legacy.csr_from_dense(A)
        q = oracle.quantise_weights(w)
        for group in (0, 1):
            want, wl = oracle.walks(rp, col, q, L, seed, group, 0, iters * A.shape[0])
            got, gl = run_gpu(g2v, rp, col, q, L, iters, seed, group)
            assert (gl == wl).all() and (got == want).all(), "case %d group %d" % (i, group)


@pytest.mark.parametrize("L", [1, 2, 3, 80, 160])
def test_ex_graph_bit_exact(g2v, L):
    for group in (0, 1):
        rp, col, w = helpers.ex_graph(group)
        q = oracle.quantise_weights(w)
        reps = 2
        want, wl = oracle.walks(rp, col, q, L, 7, group, 0, reps * (len(rp) - 1))
        got, gl = run_gpu(g2v, rp, col, q, L, reps, 7, group)
        assert (gl == wl).all()
        assert (got == want).all()
        if L == 80:
            assert wl.max() > 30 and (wl == 1).mean() > 0.5     # long walks and singleton walks both occur


def test_high_degree_rows_take_the_tail_path(g2v):
    """Rows with more than 128 neighbours (register cache = 4 chunks of 32) and a complete graph."""
    V = 400
    A = np.zeros((V, V), dtype=np.float32)
    rs = np.random.RandomState(3)
    A[:] = (0.5 + 0.5 * rs.rand(V, V)).astype(np.float32) + np.float32(1e-4)
    np.fill_diagonal(A, 0)
    A[5, :] = 0; A[:, 9] = 0
    from oracle import legacy
    rp, col, w = legacy.csr_from_dense(A)
    q = oracle.quantise_weights(w)
    for L in (50, 400):
        want, wl = oracle.walks(rp, col, q, L, 11, 1, 0, 2 * V)
        got, gl = run_gpu(g2v, rp, col, q, L, 2, 11, 1)
        assert (gl == wl).all() and (got == want).all()
    assert wl.max() == 399       # complete graph minus the unreachable node: walks cover it


def test_random_graph_with_dead_ends_and_sharding(g2v):
    rp, col, w = helpers.random_graph(3000, 6, seed=5, dead_frac=0.3)
    q = oracle.quantise_weights(w)
    want, wl = oracle.walks(rp, col, q, 40, 99, 0, 0, 3 * 3000)
    got, gl = run_gpu(g2v, rp, col, q, 40, 3, 99, 0)
    assert (gl == wl).all() and (got == want).all()
    # any shard of the walker range reproduces its slice (counter-based RNG)
    for rank, world in [(0, 2), (1, 2), (3, 8)]:
        part, pl = run_gpu(g2v, rp, col, q, 40, 3, 99, 0, walker_begin=rank, walker_stride=world)
        assert (part == want[rank::world]).all() and (pl == wl[rank::world]).all()
    part, pl = run_gpu(g2v, rp, col, q, 40, 3, 99, 0, walker_begin=1000, walker_end=5000)
    assert (part == want[1000:5000]).all()


def test_host_entry_point_equals_device_entry_point(g2v):
    rp, col, w = helpers.ex_graph(0)
    q = oracle.quantise_weights(w)
    a, al = g2v.generate_paths_host(rp, col, q, 80, 1, seed=3, group=0)
    want, wl = oracle.walks(rp, col, q, 80, 3, 0, 0, len(rp) - 1)
    assert (a == want).all() and (al == wl).all()


def test_synthetic_10k_full_size_properties_and_oracle_sample(g2v):
    """BASELINE configs[1] graph (10k genes / 500k edges, lenPath 80, 10 repetitions): size-independent
    properties on every walk + oracle equality on a sample of walkers."""
    from g2vec_b200 import graph
    V, E, L, reps = 10_000, 500_000, 80, 10
    rp, col, w = graph.synthetic_graph(V, E, 0)
    q = graph.quantise_weights(w)
    assert (q == oracle.quantise_weights(w)).all()
    got, gl = run_gpu(g2v, rp, col, q, L, reps, 12345, 0)
    assert got.shape == (V * reps, L)
    # start nodes, padding, lengths
    assert (got[:, 0] == np.arange(V * reps) % V).all()
    assert ((got >= 0).sum(1) == gl).all() and (gl >= 1).all()
    # self-avoiding
    s = np.sort(np.where(got < 0, np.arange(L)[None, :] + V, got), axis=1)
    assert (s[:, 1:] != s[:, :-1]).all()
    # every transition is an edge of the graph
    a, b = got[:, :-1].ravel(), got[:, 1:].ravel()
    m = b >= 0
    keys = np.sort(np.repeat(np.arange(V, dtype=np.int64), np.diff(rp)) * V + col)
    tk = a[m].astype(np.int64) * V + b[m]
    pos = np.searchsorted(keys, tk)
    assert (keys[np.minimum(pos, len(keys) - 1)] == tk).all()
    # oracle on a sample of walkers
    want, wl = oracle.walks(rp, col, q, L, 12345, 0, 17, V * reps, 50)
    assert (got[17::50] == want).all() and (gl[17::50] == wl).all()


def test_hash_visited_set_path(g2v, monkeypatch):
    """Graphs too large for the per-warp bitmap use the hash set; force it on a small graph too."""
    rp, col, w = helpers.ex_graph(0)
    q = oracle.quantise_weights(w)
    want, wl = oracle.walks(rp, col, q, 80, 21, 0, 0, 2 * (len(rp) - 1))
    monkeypatch.setenv("G2V_WALK_VISITED", "hash")
    got, gl = run_gpu(g2v, rp, col, q, 80, 2, 21, 0)
    assert (got == want).all() and (gl == wl).all()
    monkeypatch.delenv("G2V_WALK_VISITED")
    from g2vec_b200 import graph
    rp, col, w = graph.synthetic_graph(120_000, 600_000, 0)                     # V > bitmap limit
    q = oracle.quantise_weights(w)
    want, wl = oracle.walks(rp, col, q, 80, 5, 1, 0, 120_000)
    got, gl = run_gpu(g2v, rp, col, q, 80, 1, 5, 1)
    assert (got == want).all() and (gl == wl).all() and wl.max() == 80 and wl.min() == 1


def sorted_rows(nodes, lens, pad):
    out = np.full_like(nodes, pad)
    for i, (r, n) in enumerate(zip(nodes, lens)):
        out[i, :n] = np.sort(r[:n])
    return out


@pytest.mark.parametrize("layout", ["csr", "e8", "e4", "e4-one-walker-per-warp"])
@pytest.mark.parametrize("vis", ["bitmap", "hash"])
def test_every_layout_and_visited_set_is_bit_exact(g2v, monkeypatch, layout, vis):
    """Every kernel instantiation: plain CSR arrays (g2v_walk_launch) / {col,qw} pairs / packed 16+16-bit edges with
    two walkers per warp (four neighbours per lane) or one (two per lane) x bitmap / hash visited set x visit order /
    fused tuple(sorted(path)) epilogue."""
    import torch
    from g2vec_b200 import paths
    monkeypatch.setenv("G2V_WALK_VISITED", vis)
    if layout == "e8":
        monkeypatch.setenv("G2V_WALK_LAYOUT", "e8")
    # packed edges + bitmap: two walkers per warp (walk_pair_kernel, default for rows that mostly fit 64 neighbours)
    # or one walker per warp; force each so that both run on every graph here, long rows included
    if layout == "e4-one-walker-per-warp":
        monkeypatch.setenv("G2V_WALK_TILE", "32")
        layout = "e4"
    elif layout == "e4":
        monkeypatch.setenv("G2V_WALK_TILE", "16")
    cases = [helpers.ex_graph(1) + (80, 2), helpers.random_graph(2000, 40, seed=1, dead_frac=0.2) + (33, 3)]
    V = 300
    A = (0.5 + 0.5 * np.random.RandomState(4).rand(V, V)).astype(np.float32) + np.float32(1e-4)
    np.fill_diagonal(A, 0)
    from oracle import legacy
    cases.append(legacy.csr_from_dense(A) + (300, 1))            # rows of 299 neighbours: register chunks + tail
    for rp, col, w, L, reps in cases:
        q = oracle.quantise_weights(w)
        n = len(rp) - 1
        want, wl = oracle.walks(rp, col, q, L, 77, 1, 0, reps * n)
        g = g2v.WalkGraph(rp, col, qw=q)
        packable = q.min() >= 32768 and q.max() <= 65536          # |PCC| in [0.5, 1] and V <= 65535
        assert g.layout == (2 if (packable and layout != "e8") else 1)
        nodes, lens = g2v.generate_paths(g, L, reps, seed=77, group=1, plain_csr=(layout == "csr"))
        torch.cuda.synchronize()
        got, gl = nodes.cpu().numpy(), lens.cpu().numpy()
        assert (gl == wl).all() and (got == want).all()
        if layout != "csr":
            # fused canonical form == sort of the visit-order rows, and its keys == g2v_paths_canonicalise's
            rows, lens2, key = g2v.generate_paths(g, L, reps, seed=77, group=1, canonical=True)
            rows2, key2 = paths._canon(nodes)
            torch.cuda.synchronize()
            assert (lens2.cpu().numpy() == wl).all()
            assert (rows.cpu().numpy() == sorted_rows(want, wl, paths.PAD)).all()
            assert (rows.cpu().numpy() == rows2.cpu().numpy()).all() and (key.cpu().numpy() == key2.cpu().numpy()).all()


def test_weights_outside_the_pcc_range_take_the_pair_layout(g2v):
    """Packed 16+16-bit edges need 32768 <= qw <= 65536; anything else (and V > 65536) uses {col, qw} pairs."""
    rp, col, w = helpers.random_graph(500, 12, seed=8, dead_frac=0.1)
    w = (w * np.random.RandomState(1).uniform(0.01, 3.0, size=len(w))).astype(np.float32)
    q = oracle.quantise_weights(w)
    assert q.min() < 32768 and q.max() > 65536
    g = g2v.WalkGraph(rp, col, qw=q)
    assert g.layout == 1
    want, wl = oracle.walks(rp, col, q, 40, 3, 0, 0, 1000)
    nodes, lens = g2v.generate_paths(g, 40, 2, seed=3, group=0)
    assert (nodes.cpu().numpy() == want).all() and (lens.cpu().numpy() == wl).all()
