"""Host side of --post gpu (g2vec_b200/post.py): the option, the shared cluster-to-L-group numbering and the
k-means++ draw sequence, all without a GPU."""
import numpy as np
import pytest


def test_post_option_parses_with_host_default():
    from g2vec_b200 import cli
    a = cli.parse_arguments(["E", "C", "N", "R"])
    assert a.post == "host" and a.algo == "rows"
    assert (a.lenPath, a.numRepetition, a.sizeHiddenlayer, a.epoch, a.learningRate, a.numBiomarker) == \
        (80, 10, 128, 500, 0.005, 50)
    assert cli.parse_arguments(["E", "C", "N", "R", "--post", "gpu"]).post == "gpu"
    with pytest.raises(SystemExit):
        cli.parse_arguments(["E", "C", "N", "R", "--post", "cpu"])


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_lgroups_from_clusters_is_find_lgroups(seed):
    from sklearn.cluster import KMeans
    from g2vec_b200 import cli
    rng = np.random.default_rng(seed)
    sizes = rng.permutation([900, 300, 150])
    X = np.concatenate([rng.normal(4.0 * k, 1.0, size=(n, 8)) for k, n in enumerate(sizes)]).astype(np.float32)
    km = KMeans(n_clusters=3, random_state=0).fit(X).labels_
    got = cli.lgroups_from_clusters(km)
    assert (got == cli.find_lgroups(X, None, None)).all() and got.dtype == np.int32
    largest = np.argmax(np.bincount(km, minlength=3))
    assert (got[km == largest] == 2).all()


@pytest.mark.parametrize("shape", [(500, 16), (3000, 64), (257, 3)])
def test_kmeans_plusplus_draws_pick_sklearns_ids(shape):
    """Fed scikit-learn's own squared distances, the host draw sequence of the GPU path picks kmeans_plusplus's
    ids for random_state=0 on centred data."""
    from sklearn.cluster import kmeans_plusplus
    from sklearn.metrics.pairwise import _euclidean_distances
    from g2vec_b200 import post
    rng = np.random.default_rng(shape[0])
    X = rng.normal(size=shape).astype(np.float32)
    X[: shape[0] // 3] += 3.0
    Xc = X - X.mean(axis=0)
    norms = (Xc.astype(np.float64) ** 2).sum(1).astype(np.float32)

    def dist(ids, closest):
        d = _euclidean_distances(Xc[ids], Xc, Y_norm_squared=norms, squared=True)
        return d if closest is None else np.minimum(closest, d)

    _, want = kmeans_plusplus(Xc, 3, random_state=0)
    assert (post.kmeans_plusplus_ids(shape[0], dist, 3, 0) == want).all()
