"""CPU checks of bench.py's own pieces: the synthetic window generator of the roofline_hbm block (SURVEY 8d: distinct,
sorted genes), the counting adjacency that lets the UNMODIFIED generate_pathSet be timed on a bounded sample, and the
traffic lookup."""
import os
import sys
import time
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import bench  # noqa: E402
from oracle import ref_import  # noqa: E402


def test_synthetic_windows_are_sorted_distinct_and_reproducible():
    import torch
    rowptr, gene, label = bench.synthetic_windows(500, 3000, 80, torch.device("cpu"), seed=777)
    g = gene.view(500, 80).numpy()
    assert (np.diff(g, axis=1) > 0).all() and g.min() >= 0 and g.max() < 3000       # strictly ascending = distinct
    assert rowptr.tolist() == list(range(0, 501 * 80, 80)) and set(label.tolist()) <= {0, 1}
    r2, g2, l2 = bench.synthetic_windows(500, 3000, 80, torch.device("cpu"), seed=777)
    assert (g2 == gene).all() and (l2 == label).all()
    assert 0.3 < float(label.float().mean()) < 0.7


def test_counting_adjacency_counts_visits_and_stops_on_budget():
    from tests import helpers
    rp, col, w = helpers.random_graph(200, 6, seed=3)
    A = bench.CountingAdjacency(rp, col, w, budget_s=0.2)
    row = A[5]
    assert row.shape == (200,) and row.dtype == np.float32 and A.visits == 1
    assert (np.nonzero(row)[0] == col[rp[5]:rp[6]]).all()
    time.sleep(0.25)
    with pytest.raises(bench.CountingAdjacency.TimeUp):
        A[6]


def walk_module():
    """The reference script when it is staged; otherwise the walk port that tests/golden pins bit-exact to the
    reference's output (oracle.legacy), behind the reference's signature and its global np.random stream."""
    if ref_import.available():
        return ref_import.load()
    from oracle import legacy
    return types.SimpleNamespace(generate_pathSet=lambda adjMat, maximumLength, iterations: legacy.generate_pathSet_dense(
        adjMat, maximumLength, iterations, np.random))


def test_reference_walk_is_timed_through_its_own_function():
    from tests import helpers
    ref = walk_module()
    rp, col, w = helpers.random_graph(150, 5, seed=4)
    rate, visits, dt = bench.cpu_walk_rate(ref, [(rp, col, w)], 20, 0.5, 1)
    assert visits > 200 and 0.4 < dt < 5 and rate == pytest.approx(visits / dt)


def test_traffic_lookup_matches_only_the_captured_configuration():
    bench._RUN.update(reps=10, world=1)
    assert bench.traffic_lookup("cbow_rows_fwdbwd", "syn10k") == 67148544
    assert bench.traffic_lookup("cbow_rows_fwdbwd", "syn10k", need_reps=3) is None
    assert bench.traffic_lookup("cbow_slab_step", "stress200k", need_reps=2) == 27482516000
    bench._RUN.update(world=2)
    assert bench.traffic_lookup("cbow_rows_fwdbwd", "syn10k") is None          # captures are single-GPU
    bench._RUN.update(world=1)


def test_dump_outputs_sample_is_fixed_and_files_are_float(tmp_path):
    a = bench.sample_rows(100000, 512)
    assert len(a) == 512 and (np.diff(a) > 0).all() and (a == bench.sample_rows(100000, 512)).all()
    assert (bench.sample_rows(300, 512) == np.arange(300)).all()
    bench.write_outputs(str(tmp_path), {"W": np.ones((3, 2), np.float32), "rows": np.array([[1, 2**31 - 1]], np.int32),
                                        "keys": bench.key_words(np.array([-1, 5], dtype=np.int64))})
    W, rows, k = (np.load(str(tmp_path / (n + ".npy"))) for n in ("W", "rows", "keys"))
    assert W.dtype == np.float32 and rows.dtype == np.float64 and k.dtype == np.float64
    assert rows.tolist() == [[1, 2**31 - 1]] and k.tolist() == [[2**32 - 1, 2**32 - 1], [0, 5]]
