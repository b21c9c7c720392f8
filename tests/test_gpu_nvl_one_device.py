"""The multi-GPU step kernels (P2P form) on ONE device: g2v_cbow_update_nvl and g2v_cbow_loop_counters_nvl take
device tables of peer pointers, so `world` replica buffer sets on one GPU stand in for the ranks.  The caller brackets
every launch with cross-GPU barriers, so ranks never overlap; launching rank 0 .. world-1 in order on one stream gives
exactly the state those barriers produce.  The NVLS multicast form (multimem.*) needs the NVSwitch and is covered only
by tests/test_gpu_multi.py.

Gradient parts are integers in [-512, 512] times 2^-24: every partial sum over up to 8 ranks is exact in float32, so
the summation order cannot matter and the N-rank step must be BIT-identical to g2v_cbow_update on the summed gradient
(both kernels call the same adam1)."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

LR, B1, B2, EPS = 0.005, 0.9, 0.999, 1e-8
SENTINEL = 7.0           # m / v outside a rank's own slice: never read, never written


@pytest.fixture(scope="module")
def lib():
    import torch
    assert torch.cuda.is_available()
    from g2vec_b200 import _capi
    return _capi.load()


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _check(rc, what):
    from g2vec_b200 import _capi
    _capi.check(rc, what)


def _ptr_table(bufs):
    import torch
    return torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device="cuda")


def owned(n, world, r):
    """Elements of the flat [W_ih | W_ho] vector that rank r updates: float4 slice r of ceil(n4 / world) float4s,
    plus the scalar tail (n % 4 elements) on the last rank."""
    n4 = n // 4
    chunk = -(-n4 // world)
    lo = min(n4, r * chunk)
    hi = min(n4, lo + chunk)
    mask = np.zeros(n, bool)
    mask[4 * lo:4 * hi] = True
    if r == world - 1:
        mask[4 * n4:] = True
    return mask


def bits(x):
    return np.ascontiguousarray(x, dtype=np.float32).view(np.int32)


SHAPES = [(257, 33), (300, 100), (64, 128)]
N_CASES = ["1", "3", "4w-1"] + ["(%d+1)*%d" % vd for vd in SHAPES]
MODES = ["adam-t1", "adam-t37", "adam-device-alpha", "sgd"]


def n_of(case, world):
    if case == "1":
        return 1, None
    if case == "3":
        return 3, None
    if case == "4w-1":
        return 4 * world - 1, None
    V, D = SHAPES[N_CASES.index(case) - 3]
    return (V + 1) * D, (V, D)


class Ranks:
    """`world` replica buffer sets + the single-GPU reference (g2v_cbow_update) on the same flat vector."""

    def __init__(self, lib, n, vd, world, adam, seed):
        import torch
        self.lib, self.n, self.vd, self.world, self.adam = lib, n, vd, world, adam
        self.rs = np.random.RandomState(seed)
        W0 = (self.rs.randn(n) * 0.1).astype(np.float32)
        dev = "cuda"
        self.g = [torch.zeros(n, dtype=torch.float32, device=dev) for _ in range(world)]
        self.w = [torch.from_numpy(W0).to(dev) for _ in range(world)]
        self.own = [owned(n, world, r) for r in range(world)]
        self.m, self.v = [], []
        for r in range(world):
            m0 = np.full(n, SENTINEL, np.float32); m0[self.own[r]] = 0.0
            self.m.append(torch.from_numpy(m0).to(dev)); self.v.append(torch.from_numpy(m0.copy()).to(dev))
        self.g_tab, self.w_tab = _ptr_table(self.g), _ptr_table(self.w)
        # reference: flat W / m / v / g; [W_ih (V*D) | W_ho (D)] views, or W_ih = the whole vector (D = 1) and a
        # separate one-element W_ho when n is not of that form
        self.W = torch.from_numpy(W0).to(dev)
        self.M, self.Vv, self.G = (torch.zeros(n, dtype=torch.float32, device=dev) for _ in range(3))
        if vd:
            V, D = vd
            self.ref = (V, D, [t[:V * D] for t in (self.W, self.M, self.Vv, self.G)],
                        [t[V * D:] for t in (self.W, self.M, self.Vv, self.G)])
        else:
            extra = [torch.zeros(1, dtype=torch.float32, device=dev) for _ in range(4)]
            self.ref = (n, 1, [self.W, self.M, self.Vv, self.G], extra)

    def gradients(self):
        """Per-rank parts: exactly representable, so every order of summation gives the same float32 sum."""
        import torch
        parts = self.rs.randint(-512, 513, size=(self.world, self.n)).astype(np.float64)
        parts[:, self.rs.rand(self.n) < 0.1] = 0.0                 # some elements get no gradient at all
        for r in range(self.world):
            self.g[r].copy_(torch.from_numpy((parts[r] * 2.0 ** -24).astype(np.float32)))
        total = (parts.sum(0) * 2.0 ** -24).astype(np.float32)
        assert (total.astype(np.float64) == parts.sum(0) * 2.0 ** -24).all()
        self.G.copy_(torch.from_numpy(total))
        return total

    def step(self, t, alpha_dev=0):
        opt = 0 if self.adam else 1
        st = _stream()
        for r in range(self.world):
            _check(self.lib.g2v_cbow_update_nvl(self.g_tab.data_ptr(), self.w_tab.data_ptr(), None, None,
                                                self.m[r].data_ptr(), self.v[r].data_ptr(), self.n, r, self.world, opt,
                                                LR, B1, B2, EPS, t, alpha_dev, st), "g2v_cbow_update_nvl")
        V, D, (w, m, v, g), (wo, mo, vo, go) = self.ref
        _check(self.lib.g2v_cbow_update(w.data_ptr(), wo.data_ptr(), m.data_ptr(), v.data_ptr(), mo.data_ptr(),
                                        vo.data_ptr(), g.data_ptr(), go.data_ptr(), V, D, opt, LR, B1, B2, EPS, t,
                                        alpha_dev, st), "g2v_cbow_update")

    def host(self):
        import torch
        torch.cuda.synchronize()
        return ([x.cpu().numpy() for x in self.g], [x.cpu().numpy() for x in self.w],
                [x.cpu().numpy() for x in self.m], [x.cpu().numpy() for x in self.v])


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("case", N_CASES)
@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
def test_nvl_update_equals_single_gpu_update_bitwise(lib, world, case, mode):
    """Reduce-scatter + Adam / SGD + all-gather over `world` replicas == g2v_cbow_update on the summed gradient, bit
    for bit, over three consecutive steps (m / v carried).  The n cover n4 = n/4 < world (n = 1, 3, 4*world-1),
    n % 4 in {1, 2, 3} (the scalar tail of the last rank) and worlds that do not divide n4."""
    import torch
    n, vd = n_of(case, world)
    adam = mode != "sgd"
    R = Ranks(lib, n, vd, world, adam, seed=world * 1000 + len(case) * 10 + MODES.index(mode))
    assert np.logical_or.reduce(R.own).all() and sum(o.sum() for o in R.own) == n     # a partition of the vector
    state = torch.tensor([1.0, 1.0, 0.0, 0.0], dtype=torch.float32, device="cuda")
    t0 = 37 if mode == "adam-t37" else 1
    prev = R.W.cpu().numpy()
    for k in range(3):
        total = R.gradients()
        adev = 0
        if mode == "adam-device-alpha":
            _check(lib.g2v_cbow_adam_tick(state.data_ptr(), LR, B1, B2, _stream()), "g2v_cbow_adam_tick")
            adev = state.data_ptr()
        R.step(t0 + k, adev)
        g, w, m, v = R.host()
        W, M, Vv = R.W.cpu().numpy(), R.M.cpu().numpy(), R.Vv.cpu().numpy()
        assert float(R.G.abs().max()) == 0.0
        for r in range(world):
            assert (g[r] == 0).all(), "rank %d gradient not zeroed (step %d)" % (r, k)
            assert (bits(w[r]) == bits(W)).all(), "rank %d weights differ from g2v_cbow_update (step %d)" % (r, k)
            off = ~R.own[r]
            assert (m[r][off] == SENTINEL).all() and (v[r][off] == SENTINEL).all(), "rank %d m/v touched outside its slice" % r
            if adam:
                assert (bits(m[r][R.own[r]]) == bits(M[R.own[r]])).all() and (bits(v[r][R.own[r]]) == bits(Vv[R.own[r]])).all()
            else:
                assert (m[r][R.own[r]] == 0).all() and (v[r][R.own[r]] == 0).all()
        moved = total != 0
        if moved.any():
            assert (W[moved] != prev[moved]).any()                 # the step did something
        if not adam:
            assert (W[~moved] == prev[~moved]).all()
        prev = W


def test_nvl_adam_against_float64_restatement(lib):
    """One Adam step of the N-rank kernel (world 3, n = 301*100, t = 37, non-zero m / v) against a float64 NumPy
    restatement of TF1 ApplyAdam: m += (g-m)(1-b1); v += (g^2-v)(1-b2); w -= lr_t m / (sqrt(v) + eps) with
    lr_t = lr sqrt(1-b2^t)/(1-b1^t).  As in TF1, beta1 / beta2 are float32 (1 - 0.999f is 0.00099998713, 217 float32
    ulps from 0.001) and so are the beta powers.  The error is counted in float32 ulps of the largest operand of the
    last add (w - update cancels near zero, so ulps of the result would measure the cancellation, not the kernel).
    Observed on a B200: w 6.92, m 1.15, v 0.91 ulps; the bounds are 16, 4 and 3.5."""
    import torch
    world, n, t = 3, 301 * 100, 37
    R = Ranks(lib, n, (300, 100), world, True, seed=5)
    rs = np.random.RandomState(6)
    m0 = (rs.randint(-512, 513, size=n) * 2.0 ** -24 * 0.3).astype(np.float32)
    v0 = ((rs.randint(0, 513, size=n) * 2.0 ** -24) ** 2 * 0.05).astype(np.float32)
    for r in range(world):
        R.m[r].copy_(torch.from_numpy(np.where(R.own[r], m0, SENTINEL).astype(np.float32)))
        R.v[r].copy_(torch.from_numpy(np.where(R.own[r], v0, SENTINEL).astype(np.float32)))
    w0 = R.W.cpu().numpy()
    g = R.gradients().astype(np.float64)
    R.step(t)
    _, w, m, v = R.host()
    mm = np.select(R.own, m); vv = np.select(R.own, v)
    b1p, b2p = np.float32(1), np.float32(1)
    for _ in range(t):
        b1p, b2p = np.float32(b1p * np.float32(B1)), np.float32(b2p * np.float32(B2))
    b1, b2 = float(np.float32(B1)), float(np.float32(B2))
    lr_t = LR * np.sqrt(1.0 - float(b2p)) / (1.0 - float(b1p))
    dm, dv = (g - m0) * (1.0 - b1), (g * g - v0) * (1.0 - b2)
    m64, v64 = m0 + dm, v0 + dv
    w64 = w0 - lr_t * m64 / (np.sqrt(v64) + EPS)

    def ulps(x32, x64, *operands):
        scale = np.max(np.abs(np.stack([np.asarray(o, np.float64) for o in operands + (x64,)])), axis=0)
        return float((np.abs(x32.astype(np.float64) - x64) / np.spacing(scale.astype(np.float32))).max())

    uw, um, uv = ulps(w[0], w64, w0), ulps(mm, m64, m0, dm), ulps(vv, v64, v0, dv)
    print("float64 ApplyAdam restatement, max error in float32 ulps: w %.3f  m %.3f  v %.3f" % (uw, um, uv))
    assert uw <= 16.0 and um <= 4.0 and uv <= 3.5


# ------------------------------------------------------------------------------------------- loop control
def rule(vals, max_steps, early_stop):
    """G2Vec.py:262-283 on the summed validation counts: `if acc_val < before_acc_val: break` (strict), cap after
    max_steps.  Returns (stop_step or -1, steps decided, before_val)."""
    before = -1
    for step, s in enumerate(vals):
        if early_stop and s < before:
            return step, step + 1, before
        before = s
        if step + 1 >= max_steps:
            return -1, step + 1, before
    return -1, len(vals), before


def run_loop(lib, acc_steps, max_steps, early_stop):
    """acc_steps [steps, world, 4]: each rank's acc per step.  Per step: loop_counters_nvl for every rank, then
    loop_decide(acc = NULL) for every rank (the cross-GPU barrier sits between the two in the product)."""
    import torch
    steps, world, _ = acc_steps.shape
    ctl = [torch.zeros(8, dtype=torch.int64, device="cuda") for _ in range(world)]
    hist = [torch.zeros(4 * (steps + 1), dtype=torch.int64, device="cuda") for _ in range(world)]
    acc = torch.from_numpy(np.ascontiguousarray(acc_steps, dtype=np.int64)).cuda()
    tab = _ptr_table(hist)
    st = _stream()
    for r in range(world):
        _check(lib.g2v_cbow_loop_init(ctl[r].data_ptr(), max_steps, int(early_stop), st), "g2v_cbow_loop_init")
    for s in range(steps):
        for r in range(world):
            _check(lib.g2v_cbow_loop_counters_nvl(ctl[r].data_ptr(), acc[s, r].data_ptr(), tab.data_ptr(), None, world,
                                                  st), "g2v_cbow_loop_counters_nvl")
        for r in range(world):
            _check(lib.g2v_cbow_loop_decide(ctl[r].data_ptr(), None, hist[r].data_ptr(), st), "g2v_cbow_loop_decide")
    torch.cuda.synchronize()
    return [c.cpu().numpy() for c in ctl], [h.cpu().numpy().reshape(-1, 4) for h in hist]


def make_acc(val, world, seed):
    """val [steps, world] validation counts; the other counters are arbitrary per-rank numbers."""
    rs = np.random.RandomState(seed)
    steps = val.shape[0]
    acc = rs.randint(0, 1000, size=(steps, world, 4)).astype(np.int64)
    acc[:, :, 0] = rs.randint(1, 2**62, size=(steps, world))          # loss-sum bits: not exchanged in this mode
    acc[:, :, 2] = val
    return acc


SCENARIOS = {
    # name: (summed-val construction, max_steps, early_stop, expected stop step or -1)
    "sum-drops-at-4": ([10, 20, 30, 40, 39, 50, 60], 100, True, 4),
    "sum-equal-is-no-drop": ([10, 20, 20, 20, 21], 100, True, -1),
    "early-stop-off": ([10, 20, 30, 5, 1, 0], 100, False, -1),
    "max-steps-cap": ([1, 2, 3, 4, 5, 6, 7], 4, True, -1),
    "drop-at-step-1": ([10, 9, 50], 100, True, 1),
}


@pytest.mark.parametrize("world", [2, 3, 5])
@pytest.mark.parametrize("name", sorted(SCENARIOS))
def test_loop_counters_nvl_decide_on_cross_rank_sums(lib, world, name):
    sums, max_steps, early, want_stop = SCENARIOS[name]
    sums = np.array(sums, np.int64)
    rs = np.random.RandomState(world)
    val = np.zeros((len(sums), world), np.int64)
    for s, tot in enumerate(sums):                                  # split each sum over the ranks at random
        cut = np.sort(rs.randint(0, tot + 1, size=world - 1))
        val[s] = np.diff(np.concatenate([[0], cut, [tot]]))
    acc = make_acc(val, world, seed=len(name) + world)
    stop, n_steps, before = rule(list(sums), max_steps, early)
    assert stop == want_stop
    ctl, hist = run_loop(lib, acc, max_steps, early)
    for r in range(world):
        assert list(ctl[r][:6]) == [1 if (stop >= 0 or n_steps >= max_steps) else 0, n_steps, stop, before, max_steps,
                                    int(early)], (r, ctl[r])
        # hist[step][1..3] = the sums over the ranks on EVERY rank; slot 0 (the loss-sum bits) is written only by
        # loop_decide with acc != NULL, so in this mode it keeps the zero of the fresh history
        for s in range(n_steps):
            assert list(hist[r][s]) == [0] + [int(acc[s, :, k].sum()) for k in (1, 2, 3)], (r, s)
        assert (hist[r][n_steps:] == 0).all()                      # steps after the stop add nothing


def test_one_rank_drops_while_the_sum_rises(lib):
    """Rank 0's own validation count falls at step 2 but the sum over the ranks rises: no early stop."""
    val = np.array([[50, 10, 10], [60, 10, 10], [40, 40, 40], [40, 41, 40]], np.int64)
    acc = make_acc(val, 3, seed=1)
    ctl, hist = run_loop(lib, acc, 100, True)
    for r in range(3):
        assert list(ctl[r][:4]) == [0, 4, -1, 121]
        assert [int(h) for h in hist[r][:4, 2]] == [70, 80, 120, 121]


def test_stopped_loop_makes_update_and_counters_no_ops(lib):
    """ctl[0] = 1 attached with g2v_cbow_loop_attach: the N-rank update and the counter exchange return at once
    (steps enqueued after the early stop inside a replayed CUDA graph); attached but not stopped, they run."""
    import torch
    world, n = 3, 4 * 37 + 3
    R = Ranks(lib, n, None, world, True, seed=3)
    R.gradients()
    ctl = torch.zeros(8, dtype=torch.int64, device="cuda")
    _check(lib.g2v_cbow_loop_init(ctl.data_ptr(), 10, 1, _stream()), "g2v_cbow_loop_init")
    hist = [torch.zeros(8, dtype=torch.int64, device="cuda") for _ in range(world)]
    tab = _ptr_table(hist)
    acc = torch.tensor([0, 5, 6, 7], dtype=torch.int64, device="cuda")
    before = R.host()
    try:
        _check(lib.g2v_cbow_loop_attach(ctl.data_ptr()), "g2v_cbow_loop_attach")
        ctl[0] = 1
        for r in range(world):
            _check(lib.g2v_cbow_update_nvl(R.g_tab.data_ptr(), R.w_tab.data_ptr(), None, None, R.m[r].data_ptr(),
                                           R.v[r].data_ptr(), n, r, world, 0, LR, B1, B2, EPS, 1, 0, _stream()),
                   "g2v_cbow_update_nvl")
            _check(lib.g2v_cbow_loop_counters_nvl(ctl.data_ptr(), acc.data_ptr(), tab.data_ptr(), None, world, _stream()),
                   "g2v_cbow_loop_counters_nvl")
        after = R.host()
        for a, b in zip(before, after):
            for x, y in zip(a, b):
                assert (bits(x) == bits(y)).all()
        assert all(int(h.abs().max()) == 0 for h in hist)
        ctl[0] = 0                                                   # attached, running: the launches do their work
        for r in range(world):
            _check(lib.g2v_cbow_update_nvl(R.g_tab.data_ptr(), R.w_tab.data_ptr(), None, None, R.m[r].data_ptr(),
                                           R.v[r].data_ptr(), n, r, world, 0, LR, B1, B2, EPS, 1, 0, _stream()),
                   "g2v_cbow_update_nvl")
            _check(lib.g2v_cbow_loop_counters_nvl(ctl.data_ptr(), acc.data_ptr(), tab.data_ptr(), None, world, _stream()),
                   "g2v_cbow_loop_counters_nvl")
        g, w, _, _ = R.host()
        assert all((x == 0).all() for x in g) and (w[0] != before[1][0]).any()
        assert all(list(h.cpu().numpy()[:4]) == [0, 5 * world, 6 * world, 7 * world] for h in hist)
    finally:
        lib.g2v_cbow_loop_attach(ctypes.c_void_p(0))
