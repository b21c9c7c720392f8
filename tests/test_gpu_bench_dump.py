"""bench.py --dump-outputs on the ex_* workload: the files it writes are the outputs of the timed path (walks
bit-exact against the oracle, CBOW weights of the configured shape) and stay within the size budget."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
from g2vec_b200.paths import PAD
from tests import helpers

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_are_what_the_timed_path_computed(tmp_path):
    out = tmp_path / "outputs"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "ex", "--steps", "3", "--warmup", "1",
           "--no-alt-algo", "--no-cpu-baseline", "--no-e2e", "--no-hbm", "--no-strong", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3
    z = {f[:-4]: np.load(str(out / f)) for f in os.listdir(str(out))}
    assert set(z) == {"walk_index", "walk_rows", "walk_lens", "walk_keys", "cbow_W_ih", "cbow_W_ho", "cbow_accuracy"}
    assert sum(a.nbytes for a in z.values()) <= 64 << 20
    assert all(a.dtype in (np.float32, np.float64) for a in z.values())

    # walks: 10 repetitions of 7523 walkers per group, group 0 first; the sampled rows are the sorted walks
    n_walk = 10 * 7523
    idx = z["walk_index"].astype(np.int64)
    assert len(idx) == 8192 and (np.diff(idx) > 0).all() and idx[-1] < 2 * n_walk
    for g in (0, 1):
        rp, col, w = helpers.ex_graph(g)
        nodes, lens = oracle.walks(rp, col, oracle.quantise_weights(w), 80, 12345, g, 0, n_walk)
        mine = (idx >= g * n_walk) & (idx < (g + 1) * n_walk)
        wid = idx[mine] - g * n_walk
        want = np.sort(np.where(nodes[wid] < 0, PAD, nodes[wid]), axis=1)
        assert (z["walk_rows"][mine] == want).all() and (z["walk_lens"][mine] == lens[wid]).all()

    # CBOW: W_ih [V, D] and W_ho [D] after 1 + 3 eager and 1 + 3 graph steps from the seeded start
    assert z["cbow_W_ih"].shape == (7523, 128) and z["cbow_W_ho"].shape == (128,)
    assert np.isfinite(z["cbow_W_ih"]).all() and np.isfinite(z["cbow_W_ho"]).all()
    assert z["cbow_accuracy"].shape == (2,) and ((0 < z["cbow_accuracy"]) & (z["cbow_accuracy"] < 1)).all()
