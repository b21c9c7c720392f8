"""CPU-only checks: the C-ABI library builds/loads and exports every symbol the header declares, it
fails loudly without a GPU, and the host-side logic (quantisation, CSR, split, sharding, init)."""
import os
import re

import numpy as np
import pytest

import oracle
from oracle import legacy

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from g2vec_b200 import _capi
    lib = _capi.load()
    hdr = open(os.path.join(ROOT, "include", "g2vec_b200.h")).read()
    declared = set(re.findall(r"\b(g2v_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_capi.SIGNATURES), declared ^ set(_capi.SIGNATURES)
    for name in declared:
        assert hasattr(lib, name)
    assert lib.g2v_abi_version() == 2


def test_no_cpu_fallback_calls_fail_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from g2vec_b200 import _capi
    import g2vec_b200
    lib = _capi.load()
    assert lib.g2v_device_info(None, None, None, None) != 0
    assert b"no usable CUDA device" in lib.g2v_last_error()
    with pytest.raises(RuntimeError):
        g2vec_b200.WalkGraph(np.array([0, 1, 1]), np.array([1]), weights=np.array([0.7], np.float32))
    with pytest.raises(RuntimeError):
        g2vec_b200.train_cbow(np.array([0, 1, 2, 3]), np.array([0, 1, 0]), np.array([0, 1, 0]), 2, 4, 0.005, log=None)
    a = np.zeros(4, np.int32)
    rc = lib.g2v_walk_host(a.ctypes.data, a.ctypes.data, a.ctypes.data, 3, 0, 5, 0, 0, 0, 3, 1, a.ctypes.data, a.ctypes.data)
    assert rc != 0 and len(lib.g2v_last_error()) > 0


def test_walk_graph_refuses_integer_weights_above_2_to_the_24():
    """The sampler sums up to 64 weights of a row chunk in 32 bits, so qw <= 2^24 (include/g2vec_b200.h); WalkGraph
    checks it before touching a device.  int32 storage of the uint32 bits: -1 is 2^32 - 1."""
    import g2vec_b200
    rp, col = np.array([0, 2, 2, 2], np.int32), np.array([1, 2], np.int32)
    for q in (np.array([2**24 + 1, 40000], np.uint32), np.array([40000, -1], np.int32)):
        with pytest.raises(ValueError, match="2\\^24"):
            g2vec_b200.WalkGraph(rp, col, qw=q)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "g2vec_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert "libg2v_oracle" not in src and "g2v_oracle_" not in src, f


def test_quantisation_and_csr():
    from g2vec_b200 import graph
    w = np.array([0.5000069, 0.75, 0.9806, 1.0, 1e-9], dtype=np.float32)
    q = graph.quantise_weights(w)
    assert (q == oracle.quantise_weights(w)).all()
    assert q[3] == 65536 and q[4] == 1 and q[0] == 32768 + 0 or q[0] >= 32768
    with pytest.raises(ValueError):
        graph.quantise_weights(np.array([-1.0], np.float32))
    rs = np.random.RandomState(0)
    A = (rs.rand(30, 30) < 0.2) * (0.5 + 0.5 * rs.rand(30, 30))
    A = A.astype(np.float32)
    a = graph.csr_from_dense(A); b = legacy.csr_from_dense(A)
    assert all((x == y).all() for x, y in zip(a, b))
    r, c = np.nonzero(A)
    perm = rs.permutation(len(r))
    e = graph.csr_from_edges(r[perm], c[perm], A[r, c][perm], 30)
    assert all((x == y).all() for x, y in zip(e, b))
    # duplicated edge: last one wins, as adjMat[src][dest] = w does
    e2 = graph.csr_from_edges([0, 0, 1], [1, 1, 0], [0.6, 0.9, 0.7], 3)
    assert list(e2[1]) == [1, 0] and np.allclose(e2[2], [0.9, 0.7])


def test_group_csr_matches_reference_adjacency(golden_dir):
    """construct_adjMat golden (made by the reference): same kept-edge set and weights to 1e-6."""
    from g2vec_b200 import graph
    z = np.load(os.path.join(golden_dir, "pcc_small.npz"))
    for g in (0, 1):
        rp, col, w = graph.group_csr(z["expr"], z["label"], g, z["src"], z["dst"])
        A = legacy.dense_from_csr(rp, col, w)
        ref = z["adj%d" % g]
        near = np.abs(ref - 0.5) < 1e-5
        assert ((A > 0) == (ref > 0))[~near].all()
        assert np.abs(A - ref)[(A > 0) & (ref > 0)].max() < 1e-6


def test_synthetic_graph_spec():
    from g2vec_b200 import graph
    rp, col, w = graph.synthetic_graph(2000, 40000, 1)
    assert rp[-1] == 40000 and len(col) == 40000
    src = np.repeat(np.arange(2000), np.diff(rp))
    assert (src != col).all()
    key = src.astype(np.int64) * 2000 + col
    assert (np.diff(key) > 0).all()                       # distinct pairs, sorted by (src, dest)
    assert w.dtype == np.float32 and w.min() > 0.5 and w.max() <= 1.0
    rp2, col2, w2 = graph.synthetic_graph(2000, 40000, 1)
    assert (col == col2).all() and (w == w2).all()


def test_split_and_init_and_sharding():
    from g2vec_b200 import cbow
    tr, va = cbow.split_indices(1001, 3)
    otr, ova = oracle.split_indices(1001, 3)
    assert (tr == otr).all() and (va == ova).all() and len(tr) == 800
    # same permutation as the reference's in-place row shuffle of the dense pathList (SURVEY a7)
    P = np.arange(1001 * 3).reshape(1001, 3).copy()
    np.random.seed(3); np.random.shuffle(P)
    assert (P[:, 0] // 3 == np.concatenate([tr, va])).all()
    W, Wo = cbow.init_weights(500, 128, 0)
    s = 1 / np.sqrt(128)
    assert W.dtype == np.float32 and np.abs(W).max() <= 2 * s + 1e-6 and abs(W.std() / s - 0.88) < 0.02
    lens = np.random.RandomState(0).randint(1, 80, size=5000)
    idx = np.arange(5000)
    parts = [cbow.shard_by_nnz(idx, lens, 4, r) for r in range(4)]
    assert sorted(np.concatenate(parts)) == list(idx)
    work = [lens[p].sum() for p in parts]
    assert max(work) - min(work) <= 80


def test_cli_arguments_match_reference():
    from g2vec_b200 import cli
    a = cli.parse_arguments(["E", "C", "N", "R"])
    assert (a.lenPath, a.numRepetition, a.sizeHiddenlayer, a.epoch, a.learningRate, a.numBiomarker) == \
        (80, 10, 128, 500, 0.005, 50)
    a = cli.parse_arguments(["E", "C", "N", "R", "-p", "160", "-r", "3", "-s", "256", "-e", "5", "-l", "0.01", "-n", "7"])
    assert (a.lenPath, a.numRepetition, a.sizeHiddenlayer, a.epoch, a.learningRate, a.numBiomarker) == \
        (160, 3, 256, 5, 0.01, 7)


def test_writers_formats(tmp_path):
    from g2vec_b200 import cli
    p = str(tmp_path / "res")
    genes = np.array(["A1CF", "AAK1"])
    cli.write_vectors(p, genes, np.array([[0.0928071, -0.044005], [1.5, 2.25]], dtype=np.float32))
    cli.write_lgroups(p, np.array([1, 2]), genes)
    cli.write_biomarkers(p, ["AAK1"])
    assert open(p + "_vectors.txt").read() == "GeneSymbol\tV0\tV1\nA1CF\t0.092807\t-0.044005\nAAK1\t1.500000\t2.250000\n"
    assert open(p + "_lgroups.txt").read() == "GeneSymbol\tLgroup(0:good,1:poor,2:other)\nA1CF\t1\nAAK1\t2\n"
    assert open(p + "_biomarkers.txt").read() == "GeneSymbol\nAAK1\n"


def test_host_adjacency_on_all_ex_edges_matches_the_reference(golden_dir):
    """graph.group_csr (vectorised host form of construct_adjMat, G2Vec.py:370-391) on all 216 540 ex_* edges
    against the CSR the reference itself produced: same kept edges except on the 0.5 threshold, weights to 2e-6."""
    from g2vec_b200 import graph
    e = np.load(os.path.join(golden_dir, "ex_expr.npz"))
    gr = np.load(os.path.join(golden_dir, "ex_graph.npz"))
    for g in (0, 1):
        rp, col, w = graph.group_csr(e["expr"], gr["label"], g, e["src"].astype(np.int32), e["dst"].astype(np.int32))
        V = len(rp) - 1
        got = dict(zip((np.repeat(np.arange(V, dtype=np.int64), np.diff(rp)) * V + col).tolist(), w.tolist()))
        rrp, rcol, rw = gr["rowptr%d" % g], gr["col%d" % g], gr["w%d" % g]
        ref = dict(zip((np.repeat(np.arange(V, dtype=np.int64), np.diff(rrp)) * V + rcol).tolist(), rw.tolist()))
        both = set(got) & set(ref)
        assert len(both) > 25000 and max(abs(got[k] - ref[k]) for k in both) < 2e-6
        for k in set(got) ^ set(ref):
            assert abs((got.get(k) or ref.get(k)) - 0.5) < 1e-5
        assert len(set(got) ^ set(ref)) <= 2


def test_cli_steps_1_and_2_reproduce_the_readme_counts(tmp_path):
    """README.md:26-28 of the reference: n_samples 135, n_genes 7523, n_edges 216540 after the restriction."""
    from g2vec_b200 import cli
    from tests import helpers
    ef, cf, nf, genes = helpers.write_ex_tsv(tmp_path)
    data = cli.load_data(ef); clinical = cli.load_clinical(cf); network = cli.load_network(nf)
    assert data["expr"].shape[0] == 135 and data["expr"].dtype == np.float32 and "NOT_IN_NETWORK" in data["gene"]
    data["label"] = cli.match_labels(clinical, data["sample"])
    data, network = cli.restrict(data, network)
    assert data["expr"].shape == (135, 7523) and len(network["edge"]) == 216540
    assert list(data["gene"]) == sorted(data["gene"]) and (data["gene"] == genes).all()
    assert int((data["label"] == 0).sum()) == 77 and int((data["label"] == 1).sum()) == 58
    with pytest.raises(SystemExit):
        cli.match_labels({"nobody": 0}, data["sample"])
