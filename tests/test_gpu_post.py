"""--post gpu (g2vec_b200/post.py, csrc/g2v_post.cu) against the host steps 5-7 of g2vec_b200/cli.py: the "%.6f"
formatter byte for byte, the vectors file, the t-scores, k-means against scikit-learn, the empty-cluster fallback
and the command line end to end."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLT_MAX = np.finfo(np.float32).max


def _py_lines(mat):
    return "".join("".join("\t%.6f" % v for v in row) + "\n" for row in mat).encode()


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def _bits(u):
    return np.asarray(u, dtype=np.uint32).view(np.float32)


def _formatter_inputs():
    rng = np.random.default_rng(7)
    exps = np.arange(256, dtype=np.uint32) << 23
    mants = np.linspace(0, (1 << 23) - 1, 4096).astype(np.uint32)
    grid = (exps[:, None] | mants[None, :]).ravel()
    grid = np.concatenate([grid, grid | 0x80000000])
    grid = grid[((grid >> 23) & 0xff) != 0xff]                             # finite; inf / nan below
    half = (2 * rng.integers(0, 1 << 23, 1_000_000, dtype=np.int64) + 1).astype(np.float64) * 2.0 ** -7
    half = (half * rng.choice([-1.0, 1.0], half.size)).astype(np.float32)  # lowest set bit 2^-7: exact halfway
    ks = np.unique(np.concatenate([np.arange(0, 2000), rng.integers(0, 10 ** 9, 20000),
                                   [10 ** j - 1 for j in range(1, 13)], [10 ** j for j in range(1, 13)]]))
    b = ((ks + 0.5) * 1e-6).astype(np.float32)                             # k * 1e-6 + 1/2 * 1e-6, and neighbours
    bnd = np.concatenate([np.nextafter(b, np.float32(-np.inf)), b, np.nextafter(b, np.float32(np.inf))])
    bnd = np.concatenate([bnd, -bnd, np.float32([0.99999994, 4.9999999e-7, np.nextafter(np.float32(4.9999999e-7),
                                                                                         np.float32(1))])])
    special = np.concatenate([
        _bits(np.arange(1, 1 << 23, 997)), -_bits(np.arange(1, 1 << 23, 997)),   # subnormals
        np.float32([0.0, -0.0, FLT_MAX, -FLT_MAX, np.inf, -np.inf]),
        _bits([0x7fc00000, 0xffc00000, 0x7f800001, 0xff800001, 0x7fffffff, 0xffffffff, 0x7fa00000, 0xffc0beef])])
    return np.concatenate([grid.view(np.float32), half, bnd, special]).astype(np.float32)


def test_formatter_equals_python_percent_6f():
    from g2vec_b200 import post
    x = _formatter_inputs()
    D = 512
    n = -(-x.size // D) * D
    mat = np.concatenate([x, np.zeros(n - x.size, np.float32)]).reshape(-1, D)
    assert post.format_rows(_dev(mat)) == _py_lines(mat)
    assert "%.6f" % -FLT_MAX == "-" + "%.6f" % FLT_MAX and len("%.6f" % -FLT_MAX) == 47


@pytest.mark.parametrize("D,chunk", [(1, 1 << 20), (1, 37), (512, 1 << 20), (512, 3000), (3, 1), (130, 777)])
def test_formatter_widths_and_chunk_boundaries(D, chunk):
    """D = 1 and D = 512, with chunk budgets that are smaller than one line or fall inside lines: every chunk
    holds whole lines and the concatenation is the same text."""
    from g2vec_b200 import post
    x = _formatter_inputs()
    rng = np.random.default_rng(D)
    sel = x[rng.integers(0, x.size, 300 * D)].reshape(300, D)
    names = [("g%dé" % i).encode() for i in range(300)]
    want = b"".join(nm + line for nm, line in zip(names, _py_lines(sel).splitlines(keepends=True)))
    assert post.format_rows(_dev(sel), names, chunk_bytes=chunk) == want
    assert post.format_rows(_dev(sel), chunk_bytes=chunk) == _py_lines(sel)


def test_vectors_file_identical_200k_x_512(tmp_path):
    from g2vec_b200 import cli, post
    rng = np.random.default_rng(200)
    mat = (rng.standard_normal((200_000, 512)) * 0.1).astype(np.float32)
    genes = np.array(["G%06d" % i for i in range(mat.shape[0])])
    post.write_vectors(str(tmp_path / "gpu"), genes, _dev(mat))
    cli.write_vectors(str(tmp_path / "host"), genes, mat)
    a, b = (open(str(tmp_path / (p + "_vectors.txt")), "rb").read() for p in ("gpu", "host"))
    assert len(a) > 9 * 10 ** 8 and a == b


# ------------------------------------------------------------------------------------------------ t-scores
def _tscore_f64(expr, label):
    """cli.tscore's formula for every gene, in float64."""
    a, b = expr[label == 0].astype(np.float64), expr[label == 1].astype(np.float64)
    ma, mb = a.mean(0), b.mean(0)
    d1 = np.sqrt((((a - ma) ** 2).sum(0) + ((b - mb) ** 2).sum(0)) / (len(a) + len(b) - 2))
    d2 = np.sqrt(1.0 / len(a) + 1.0 / len(b))
    ok = d1 > 0
    d1 = np.where(ok, d1, 1.0)
    return np.where(ok, np.abs((ma - mb) / d1 / d2), 0.0), np.where(ok, np.maximum(np.abs(ma), np.abs(mb)) / d1 / d2, 0.0)


def test_tscores_match_host_on_ex(golden_dir):
    """Within 1e-5 of cli.tscore's formula in float64.  cli.tscores itself runs in float32 (NumPy 2 keeps
    Python-float x float32 in float32), so its mean difference cancels: against it the bound adds 4 float32 ulps
    of the larger group mean, carried through the division (up to 1.7% of a small |t| on ex_*)."""
    from g2vec_b200 import cli, post
    e = np.load(os.path.join(golden_dir, "ex_expr.npz"))
    label = np.load(os.path.join(golden_dir, "ex_graph.npz"))["label"].astype(np.int64)
    want = cli.tscores(e["expr"], label)
    got = post.tscores(_dev(e["expr"]), label).cpu().numpy()
    exact, scale = _tscore_f64(e["expr"], label)
    assert np.all(np.abs(got - exact) <= 1e-5 * exact + 1e-30)
    assert np.all(np.abs(got - want) <= 1e-5 * np.abs(want) + 4 * 2.0 ** -23 * scale)


def test_tscores_edge_cases():
    from g2vec_b200 import cli, post
    rng = np.random.default_rng(5)
    S, V = 40, 64
    expr = rng.normal(size=(S, V)).astype(np.float32)
    expr[:, :8] = np.float32([0.0, 3.0, -0.5, 1.25, 2.0 ** -10, 7.0, -2.0, 0.75])     # constant genes
    label = np.r_[np.zeros(25, int), np.ones(15, int)]
    for lab in (label, np.r_[np.zeros(39, int), [1]], np.r_[[0], np.ones(39, int)]):   # a group of one sample
        want = cli.tscores(expr, lab)
        got = post.tscores(_dev(expr), lab).cpu().numpy()
        assert (want[:8] == 0).all() and (got[:8] == 0).all()
        assert np.all(np.abs(got - want) <= 1e-5 * np.abs(want) + 1e-30)
    for lab in (np.zeros(S, int), np.ones(S, int)):                                    # all samples in one group
        with pytest.raises(ZeroDivisionError):
            cli.tscores(expr, lab)
        with pytest.raises(ZeroDivisionError):
            post.tscores(_dev(expr), lab)


# ------------------------------------------------------------------------------------------------- k-means
def _blobs(V, D, seed):
    rng = np.random.default_rng(seed)
    sizes = [V // 2, V // 3, V - V // 2 - V // 3]
    centres = rng.normal(0, 1.0, size=(3, D))
    return np.concatenate([rng.normal(c, 0.6, size=(n, D)) for c, n in zip(centres, sizes)]).astype(np.float32)[
        rng.permutation(V)]


@pytest.mark.parametrize("V,D", [(7523, 128), (20_000, 256), (200_000, 512)])
def test_kmeans_planted_clusters_equal_sklearn(V, D):
    from sklearn.cluster import KMeans, kmeans_plusplus
    from g2vec_b200 import post
    X = _blobs(V, D, V + D)
    Xd = _dev(X)
    res = post.kmeans(Xd)
    _, ids = kmeans_plusplus(X - X.mean(0), 3, random_state=0)
    assert (res.init_ids == ids).all()
    want = KMeans(n_clusters=3, random_state=0).fit(X).labels_
    assert (res.labels == want).all()
    again = post.kmeans(Xd)
    assert (again.labels == res.labels).all() and again.n_iter == res.n_iter


def test_kmeans_empty_cluster_falls_back_to_sklearn():
    from g2vec_b200 import cli, post
    rng = np.random.default_rng(3)
    pts = rng.normal(size=(2, 6)).astype(np.float32)
    X = pts[np.r_[np.zeros(120, int), np.ones(45, int)]]                # two distinct points: one cluster empties
    assert post.kmeans(_dev(X)).labels is None
    with pytest.warns(Warning):                                       # scikit-learn: fewer distinct clusters than 3
        lg, fell_back = post.find_lgroups(_dev(X))
    assert fell_back
    with pytest.warns(Warning):
        assert (lg == cli.find_lgroups(X, None, None)).all()


# ------------------------------------------------------------------------------------- the command line
RUN_GPU = r"""
import json, sys
from g2vec_b200 import cli, post
ran = []
_find = post.find_lgroups
def find(*a, **k):
    out = _find(*a, **k)
    ran.append(out[1])
    return out
post.find_lgroups = find
cli.main(sys.argv[1:])
print(json.dumps({"sklearn": "sklearn" in sys.modules, "fallback": any(ran)}))
"""


@pytest.fixture(scope="module")
def cli_runs(tmp_path_factory):
    from g2vec_b200 import cli
    from tests import helpers
    tmp = tmp_path_factory.mktemp("post_cli")
    ef, cf, nf, genes = helpers.write_ex_tsv(tmp)
    args = ["--algo", "rank1", "-r", "2", "-e", "5", "-n", "20", "--seed", "3"]
    host = str(tmp / "host")
    cli.main([ef, cf, nf, host] + args)
    gpu = str(tmp / "gpu")
    env = dict(os.environ, PYTHONPATH=ROOT)
    p = subprocess.run([sys.executable, "-c", RUN_GPU, ef, cf, nf, gpu, "--post", "gpu"] + args, cwd=ROOT, env=env,
                       capture_output=True, text=True)
    assert p.returncode == 0, p.stderr[-3000:]
    info = json.loads(p.stdout.strip().splitlines()[-1])
    return host, gpu, info, p.stdout, (ef, cf, nf)


def _read_vectors(prefix):
    lines = open(prefix + "_vectors.txt").read().splitlines()[1:]
    return np.array([[float(x) for x in ln.split("\t")[1:]] for ln in lines], dtype=np.float32), \
        np.array([ln.split("\t", 1)[0] for ln in lines])


def test_command_line_post_gpu_writes_the_host_files(cli_runs):
    from g2vec_b200 import cli
    host, gpu, info, log, (ef, cf, nf) = cli_runs
    for step in (">>> 5. Find L-groups", ">>> 6. Select biomarkers with gene scores", ">>> 7. Save results"):
        assert step in log
    assert not info["sklearn"] or info["fallback"]
    for suffix in ("_vectors.txt", "_lgroups.txt"):
        assert open(host + suffix, "rb").read() == open(gpu + suffix, "rb").read(), suffix
    bh, bg = (open(p + "_biomarkers.txt").read().splitlines() for p in (host, gpu))
    if bh != bg:
        # only a near-tie at the cut of a group may differ: the N-th and (N+1)-th host scores within 1e-6
        mat, genes = _read_vectors(host)
        data, _ = cli.restrict(cli.load_data(ef), cli.load_network(nf))
        label = cli.match_labels(cli.load_clinical(cf), data["sample"])
        lg = np.array([int(ln.split("\t")[1]) for ln in open(host + "_lgroups.txt").read().splitlines()[1:]])
        diff = set(bh) ^ set(bg)
        for i in (0, 1):
            sel = lg == i
            if not diff & set(genes[sel]):
                continue
            s = np.sort(0.5 * (cli.minmax(np.linalg.norm(mat[sel], axis=1))
                               + cli.minmax(cli.tscores(data["expr"][:, sel], label))))[::-1]
            assert abs(float(s[19]) - float(s[20])) <= 1e-6, (i, s[18:22])


def test_vectors_file_identical_on_trained_ex(cli_runs, tmp_path):
    from g2vec_b200 import cli, post
    host = cli_runs[0]
    mat, genes = _read_vectors(host)
    post.write_vectors(str(tmp_path / "g"), genes, _dev(mat))
    cli.write_vectors(str(tmp_path / "h"), genes, mat)
    assert open(str(tmp_path / "g_vectors.txt"), "rb").read() == open(str(tmp_path / "h_vectors.txt"), "rb").read()


def test_kmeans_on_trained_ex_vectors(tmp_path_factory):
    """ex_* vectors from the bit-reproducible trainer (--algo rank1 --seed 0): the GPU labels equal scikit-learn's
    on every gene where scikit-learn's float32 and float64 fits agree with each other."""
    from sklearn.cluster import KMeans
    from g2vec_b200 import cli, post
    from tests import helpers
    tmp = tmp_path_factory.mktemp("post_ex0")
    ef, cf, nf, _ = helpers.write_ex_tsv(tmp)
    cli.main([ef, cf, nf, str(tmp / "r"), "--algo", "rank1", "--seed", "0", "-r", "2", "-e", "5", "--post", "gpu"])
    mat, _ = _read_vectors(str(tmp / "r"))
    got = post.kmeans(_dev(mat)).labels
    l32 = KMeans(n_clusters=3, random_state=0).fit(mat).labels_
    l64 = KMeans(n_clusters=3, random_state=0).fit(mat.astype(np.float64)).labels_
    agree = l32 == l64
    print("ex_* rank1 seed 0: %d of %d genes outside the set where sklearn's float32 and float64 fits agree"
          % (int((~agree).sum()), agree.size))
    assert (got[agree] == l32[agree]).all()
