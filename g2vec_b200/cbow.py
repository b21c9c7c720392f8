"""HOT PATH 2, host side: the modified-CBOW trainer behind the reference's call
``compute_genetovec(pathList, n_genes, hidden_size, learning_rate)`` (/root/reference/G2Vec.py:74,
217-286).  The TF1 graph (two matmuls, sigmoid BCE, Adam, accuracy; :231-251) is replaced by the
fused kernels of csrc/g2v_cbow.cu called through the C ABI; this module keeps what the reference
keeps in Python: shuffle + 80/20 split (:219-226), the epoch loop, the log lines and the early stop
(:259-284).

Multi-GPU (one process per GPU, torch.distributed/NCCL): the parameters are replicated, the
training and validation windows are sharded over the ranks, and the dense gradient is all-reduced
once per optimizer step before every rank applies the identical update.
"""
import math
import time

import numpy as np
import torch

from . import _capi


# ------------------------------------------------------------------------------ host-side pieces
def split_indices(n, seed):
    """``np.random.shuffle(pathList)`` then ``pivot = int(len * 0.8)`` (G2Vec.py:219-222), done on an
    index vector with the same legacy MT19937 stream (RandomState(seed).shuffle)."""
    perm = np.arange(n, dtype=np.int64)
    np.random.RandomState(seed).shuffle(perm)
    pivot = int(n * 0.8)
    return perm[:pivot], perm[pivot:]


def truncated_normal(shape, stddev, rng):
    """tf.truncated_normal (G2Vec.py:234-235): N(0, stddev) re-drawn while |x| > 2 stddev."""
    x = rng.standard_normal(size=shape)
    bad = np.abs(x) > 2.0
    while bad.any():
        x[bad] = rng.standard_normal(size=int(bad.sum()))
        bad = np.abs(x) > 2.0
    return (x * stddev).astype(np.float32)


def init_weights(n_genes, hidden, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    s = 1.0 / math.sqrt(hidden)
    return truncated_normal((n_genes, hidden), s, rng), truncated_normal((hidden,), s, rng)


def shard_by_nnz(idx, lens, world, rank, keep_order=False):
    """Deal window indices to ranks so every rank gets ~equal gather work: sort by length
    (descending, stable) and deal round-robin (SURVEY.md 8e).  ``keep_order`` (mini-batches): deal the
    shuffled list as it is, ``idx[rank::world]``, so that every batch stays a random sample of the list --
    batch b of the N-GPU run is then the same set of windows as batch b of the 1-GPU run."""
    if world == 1:
        return idx
    if keep_order:
        return idx[rank::world]
    order = np.argsort(-lens[idx], kind="stable")
    return idx[order][rank::world]


# ------------------------------------------------------------------------------------ the model
class CbowModel:
    """Parameters + optimizer state + scratch in HBM, and the three kernel calls."""

    def __init__(self, rowptr, gene, label, n_genes, hidden, W_ih0, W_ho0, optimizer="adam", reduce="sum",
                 lr=0.005, beta1=0.9, beta2=0.999, eps=1e-8, device=None, algo="rows", nvl_group=None):
        if not torch.cuda.is_available():
            raise RuntimeError("g2vec_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = _capi.load()
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.device = dev

        def to(a, dt):
            if isinstance(a, torch.Tensor):
                return a.to(device=dev, dtype=dt).contiguous()
            return torch.from_numpy(np.ascontiguousarray(a)).to(device=dev, dtype=dt)

        self.rowptr = to(rowptr, torch.int32)
        self.gene = to(gene, torch.int32)
        self.label = to(label, torch.uint8)
        self.V, self.D = int(n_genes), int(hidden)
        n_flat = self.V * self.D + self.D
        # rows: parameters, Adam state and gradient are flat [W_ih (V*D) | W_ho (D)] allocations.  With a process
        # group (multi-GPU) the parameters and the gradient live in symmetric memory (peer-mapped, NVLS multicast if
        # the fabric has it) and the optimizer step does the gradient exchange itself (g2v_cbow_update_nvl).
        self.nvl = None
        if algo == "rows" and nvl_group is not None:
            self.nvl = _nvl_setup(nvl_group, n_flat, dev)
        if algo == "rows":
            self.w_flat = self.nvl["w"] if self.nvl else torch.empty(n_flat, dtype=torch.float32, device=dev)
            self.W_ih = self.w_flat[:self.V * self.D].view(self.V, self.D)
            self.W_ho = self.w_flat[self.V * self.D:]
            self.W_ih.copy_(to(W_ih0, torch.float32).reshape(self.V, self.D))
            self.W_ho.copy_(to(W_ho0, torch.float32).reshape(self.D))
        else:
            self.W_ih = to(W_ih0, torch.float32).reshape(self.V, self.D).clone()
            self.W_ho = to(W_ho0, torch.float32).reshape(self.D).clone()
        self.opt = {"adam": _capi.OPT_ADAM_TF1, "sgd": _capi.OPT_SGD}[optimizer]
        self.reduce = {"sum": _capi.REDUCE_SUM, "mean": _capi.REDUCE_MEAN}[reduce]
        self.lr, self.beta1, self.beta2, self.eps = float(lr), float(beta1), float(beta2), float(eps)
        z = lambda *s: torch.zeros(*s, dtype=torch.float32, device=dev)
        if algo not in ("rows", "rank1"):
            raise ValueError("algo must be 'rows' (gather/scatter of embedding rows) or 'rank1' (collapsed)")
        self.algo = algo
        if algo == "rows":
            # one allocation [g_ih | g_ho]: a multi-GPU step all-reduces the whole gradient with ONE collective
            self.g_flat = self.nvl["g"].zero_() if self.nvl else z(n_flat)
            self.g_ih = self.g_flat[:self.V * self.D].view(self.V, self.D)
            self.g_ho = self.g_flat[self.V * self.D:]
            self.s = self.c = None
        else:                       # rank-1: s = W_ih.W_ho, c = X^T.dO; no dense gradient
            self.g_ih = None
            self.g_ho = z(int(self.lib.g2v_cbow_r1_scratch_bytes(self.D)) // 4)   # per-block partials of W_ih^T.c
            self.s, self.c = z(self.V), z(self.V)
        self.m_flat = self.v_flat = None
        if self.opt == _capi.OPT_ADAM_TF1 and algo == "rows":
            self.m_flat, self.v_flat = z(n_flat), z(n_flat)
            vd = self.V * self.D
            self.m_ih, self.v_ih = self.m_flat[:vd].view(self.V, self.D), self.v_flat[:vd].view(self.V, self.D)
            self.m_ho, self.v_ho = self.m_flat[vd:], self.v_flat[vd:]
        elif self.opt == _capi.OPT_ADAM_TF1:
            self.m_ih, self.v_ih, self.m_ho, self.v_ho = z(self.V, self.D), z(self.V, self.D), z(self.D), z(self.D)
        else:
            self.m_ih = self.v_ih = self.m_ho = self.v_ho = None
        # [loss_sum (f64 bits), n_correct_train_fwd, n_correct_val, n_correct_train] as 4 x 8 bytes
        self.acc = torch.zeros(4, dtype=torch.int64, device=dev)
        self.t = 0
        # Adam's beta1^t / beta2^t / alpha_t live on the device (TF1's beta*_power variables), advanced by
        # g2v_cbow_adam_tick: no launch of a step depends on a host-side value, so a step can be a CUDA graph
        self.hyper = torch.tensor([1.0, 1.0, 0.0, 0.0], dtype=torch.float32, device=dev)
        if algo == "rank1":
            _capi.check(self.lib.g2v_cbow_r1_prepare(self.W_ih.data_ptr(), self.W_ho.data_ptr(), self.s.data_ptr(),
                                                     self.V, self.D, self._stream()), "g2v_cbow_r1_prepare")

    def prepare_csc(self, win):
        """rank1 only: transpose the incidence of the window list ``win`` (int32 device tensor) once, so that
        fwdbwd(win, ...) over the WHOLE list forms c without atomics (deterministic, and faster when few
        genes receive many windows).  The windows are static across steps (full batch), so this is setup."""
        if self.algo != "rank1":
            return
        w = win.to(torch.int64)
        starts = self.rowptr[w].to(torch.int64)
        lens = self.rowptr[w + 1].to(torch.int64) - starts
        total = int(lens.sum())
        pos = torch.repeat_interleave(torch.arange(w.shape[0], device=self.device), lens)
        first = torch.cumsum(lens, 0) - lens
        idx = starts[pos] + (torch.arange(total, device=self.device) - first[pos])
        g = self.gene[idx].to(torch.int64)
        g, order = torch.sort(g, stable=True)
        cscptr = torch.zeros(self.V + 1, dtype=torch.int64, device=self.device)
        cscptr[1:] = torch.cumsum(torch.bincount(g, minlength=self.V), 0)
        self._csc = (win.data_ptr(), int(w.shape[0]), cscptr.to(torch.int32), pos[order].to(torch.int32),
                     torch.empty(w.shape[0], dtype=torch.float32, device=self.device))

    def prepare_slabs(self, win, win_begin=0, n_win=None):
        """rows only, tables larger than the L2 (csrc/g2v_cbow_slab.cu): record once, for the static window list
        ``win`` (int32 device tensor or None), where every window's sorted gene list crosses the gene-slab
        boundaries; fwdbwd()/evaluate() over exactly this list then run slab by slab, L2-resident."""
        if self.algo != "rows":
            return False
        import ctypes
        if not hasattr(self, "_n_slabs"):
            s = ctypes.c_int32(1)
            _capi.check(self.lib.g2v_cbow_slab_plan(self.V, self.D, ctypes.byref(s)), "g2v_cbow_slab_plan")
            self._n_slabs, self._slabs = int(s.value), {}
        n = ((win.shape[0] if win is not None else self.rowptr.shape[0] - 1) - win_begin) if n_win is None else n_win
        if self._n_slabs <= 1 or n <= 0:
            return False
        ws = torch.empty(int(self.lib.g2v_cbow_slab_workspace_bytes(int(n), self.D, self._n_slabs)), dtype=torch.uint8,
                         device=self.device)
        _capi.check(self.lib.g2v_cbow_slab_setup(self.rowptr.data_ptr(), self.gene.data_ptr(), self._ptr(win),
                                                 int(win_begin), int(n), self.V, self._n_slabs, ws.data_ptr(),
                                                 self._stream()), "g2v_cbow_slab_setup")
        self._slabs[(self._ptr(win), int(win_begin), int(n))] = ws
        return True

    def _slab_ws(self, win, win_begin, n):
        slabs = getattr(self, "_slabs", None)
        return slabs.get((self._ptr(win), int(win_begin), int(n))) if slabs else None

    def grad_tensors(self):
        """What a multi-GPU step must all-reduce (sum) between fwdbwd() and update(): nothing when update() does
        the exchange itself over NVLink (self.nvl)."""
        if self.nvl:
            return []
        return [self.g_flat] if self.algo == "rows" else [self.c]

    def exchange(self):
        if self.nvl:
            return "nvl-multicast (multimem.ld_reduce / multimem.st)" if self.nvl["g_mc"] else "nvl-p2p (peer loads / stores)"
        return "nccl all_reduce"

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    @staticmethod
    def _ptr(t):
        return 0 if t is None else t.data_ptr()

    def fwdbwd(self, win, n_total, win_begin=0, n_win=None):
        """Accumulate the gradient of the listed windows into g_ih / g_ho (loss sum -> acc[0],
        pre-update correct count -> acc[1])."""
        n = (win.shape[0] - win_begin) if n_win is None else n_win
        if self.algo == "rank1":
            csc = getattr(self, "_csc", None)
            if csc is not None and win is not None and csc[0] == win.data_ptr() and win_begin == 0 and n == csc[1]:
                rc = self.lib.g2v_cbow_r1_windows_csc(self.rowptr.data_ptr(), self.gene.data_ptr(),
                                                      self.label.data_ptr(), win.data_ptr(), int(n),
                                                      1.0 / float(n_total), self.s.data_ptr(), csc[2].data_ptr(),
                                                      csc[3].data_ptr(), csc[4].data_ptr(), self.c.data_ptr(),
                                                      self.acc.data_ptr(), self.acc.data_ptr() + 8, self.V,
                                                      self.reduce, self._stream())
                _capi.check(rc, "g2v_cbow_r1_windows_csc")
                return
            rc = self.lib.g2v_cbow_r1_windows(self.rowptr.data_ptr(), self.gene.data_ptr(), self.label.data_ptr(),
                                              self._ptr(win), int(win_begin), int(n), 1.0 / float(n_total),
                                              self.s.data_ptr(), self.c.data_ptr(), self.acc.data_ptr(),
                                              self.acc.data_ptr() + 8, self.V, self.reduce, self._stream())
            _capi.check(rc, "g2v_cbow_r1_windows")
            return
        ws = self._slab_ws(win, win_begin, n)
        if ws is not None:
            rc = self.lib.g2v_cbow_fwdbwd_slabs(self.gene.data_ptr(), self.label.data_ptr(), self._ptr(win),
                                                int(win_begin), int(n), 1.0 / float(n_total), self.W_ih.data_ptr(),
                                                self.W_ho.data_ptr(), self.g_ih.data_ptr(), self.g_ho.data_ptr(),
                                                self.acc.data_ptr(), self.acc.data_ptr() + 8, self.V, self.D,
                                                self.reduce, self._n_slabs, ws.data_ptr(), self._stream())
            _capi.check(rc, "g2v_cbow_fwdbwd_slabs")
            return
        rc = self.lib.g2v_cbow_fwdbwd(self.rowptr.data_ptr(), self.gene.data_ptr(), self.label.data_ptr(),
                                      self._ptr(win), int(win_begin), int(n), 1.0 / float(n_total),
                                      self.W_ih.data_ptr(), self.W_ho.data_ptr(), self.g_ih.data_ptr(),
                                      self.g_ho.data_ptr(), self.acc.data_ptr(), self.acc.data_ptr() + 8,
                                      self.V, self.D, self.reduce, self._stream())
        _capi.check(rc, "g2v_cbow_fwdbwd")

    def update(self):
        self.t += 1
        adev = 0
        if self.opt == _capi.OPT_ADAM_TF1:
            _capi.check(self.lib.g2v_cbow_adam_tick(self.hyper.data_ptr(), self.lr, self.beta1, self.beta2,
                                                    self._stream()), "g2v_cbow_adam_tick")
            adev = self.hyper.data_ptr()
        if self.algo == "rank1":
            rc = self.lib.g2v_cbow_r1_update(self.W_ih.data_ptr(), self.W_ho.data_ptr(), self._ptr(self.m_ih),
                                             self._ptr(self.v_ih), self._ptr(self.m_ho), self._ptr(self.v_ho),
                                             self.c.data_ptr(), self.g_ho.data_ptr(), self.s.data_ptr(), self.V,
                                             self.D, self.opt, self.lr, self.beta1, self.beta2, self.eps, self.t,
                                             adev, self._stream())
            _capi.check(rc, "g2v_cbow_r1_update")
            return
        if self.nvl:
            # gradient exchange fused with the optimizer: barrier (every rank's gradient complete) -> reduce-scatter +
            # Adam on the owned slice + all-gather of the new weights in ONE kernel -> barrier (weights delivered)
            nv = self.nvl
            nv["hg"].barrier(channel=0)
            rc = self.lib.g2v_cbow_update_nvl(nv["hg"].buffer_ptrs_dev, nv["hw"].buffer_ptrs_dev, nv["g_mc"], nv["w_mc"],
                                              self._ptr(self.m_flat), self._ptr(self.v_flat),
                                              self.V * self.D + self.D, nv["rank"], nv["world"], self.opt, self.lr,
                                              self.beta1, self.beta2, self.eps, self.t, adev, self._stream())
            _capi.check(rc, "g2v_cbow_update_nvl")
            nv["hg"].barrier(channel=1)
            return
        rc = self.lib.g2v_cbow_update(self.W_ih.data_ptr(), self.W_ho.data_ptr(), self._ptr(self.m_ih),
                                      self._ptr(self.v_ih), self._ptr(self.m_ho), self._ptr(self.v_ho),
                                      self.g_ih.data_ptr(), self.g_ho.data_ptr(), self.V, self.D, self.opt,
                                      self.lr, self.beta1, self.beta2, self.eps, self.t, adev, self._stream())
        _capi.check(rc, "g2v_cbow_update")

    def evaluate(self, win, slot, win_begin=0, n_win=None):
        """Add the number of correctly classified listed windows into acc[slot]."""
        n = (win.shape[0] - win_begin) if n_win is None else n_win
        if self.algo == "rank1":
            rc = self.lib.g2v_cbow_r1_windows(self.rowptr.data_ptr(), self.gene.data_ptr(), self.label.data_ptr(),
                                              self._ptr(win), int(win_begin), int(n), 0.0, self.s.data_ptr(), 0, 0,
                                              self.acc.data_ptr() + 8 * slot, self.V, self.reduce, self._stream())
            _capi.check(rc, "g2v_cbow_r1_windows")
            return
        ws = self._slab_ws(win, win_begin, n)
        if ws is not None:
            rc = self.lib.g2v_cbow_eval_slabs(self.gene.data_ptr(), self.label.data_ptr(), self._ptr(win),
                                              int(win_begin), int(n), self.W_ih.data_ptr(), self.W_ho.data_ptr(),
                                              self.acc.data_ptr() + 8 * slot, self.V, self.D, self.reduce,
                                              self._n_slabs, ws.data_ptr(), self._stream())
            _capi.check(rc, "g2v_cbow_eval_slabs")
            return
        rc = self.lib.g2v_cbow_eval(self.rowptr.data_ptr(), self.gene.data_ptr(), self.label.data_ptr(),
                                    self._ptr(win), int(win_begin), int(n), self.W_ih.data_ptr(),
                                    self.W_ho.data_ptr(), self.acc.data_ptr() + 8 * slot, self.V, self.D,
                                    self.reduce, self._stream())
        _capi.check(rc, "g2v_cbow_eval")

    def loss_sum(self, acc_host):
        return float(acc_host[:1].view(torch.float64)[0])


def _nvl_setup(group, n_flat, dev):
    """Symmetric-memory buffers for the parameters and the gradient (torch.distributed._symmetric_memory: peer-mapped
    allocations + signal pads for cross-GPU barriers; NVLS multicast address when the NVSwitch fabric offers it).
    Returns None -- the caller then uses NCCL -- if G2V_CBOW_NVL=0 or the rendezvous is not possible on this box."""
    import os
    import sys
    if os.environ.get("G2V_CBOW_NVL", "1") == "0":
        return None
    try:
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        w = symm.empty(n_flat, dtype=torch.float32, device=dev)
        g = symm.empty(n_flat, dtype=torch.float32, device=dev)
        hw, hg = symm.rendezvous(w, group), symm.rendezvous(g, group)
        mc = os.environ.get("G2V_CBOW_NVL_MULTICAST", "1") != "0"
        w_mc = int(hw.multicast_ptr or 0) if mc else 0       # 0: no NVLS multicast object behind this allocation
        g_mc = int(hg.multicast_ptr or 0) if mc else 0
        if not (w_mc and g_mc):
            w_mc = g_mc = 0
        return {"w": w, "g": g, "hw": hw, "hg": hg, "w_mc": w_mc, "g_mc": g_mc, "rank": dist.get_rank(group),
                "world": dist.get_world_size(group)}
    except Exception as exc:                   # no symmetric memory here: NCCL all-reduce + replicated update instead
        print("g2vec_b200: symmetric memory unavailable (%r); using NCCL for the gradient exchange" % (exc,), file=sys.stderr)
        return None


class WindowFeeder:
    """Feeds a CbowModel's context windows from pinned host memory, double-buffered.

    ``upload(k)`` enqueues, on a private copy stream, the host->device copies of the window CSR into buffer
    set k (gene ids travel as int16 when n_genes <= 32768 and are widened to int32 on the device: half the
    PCIe bytes); ``use(k)`` makes the compute stream wait for that upload and points the model at buffer set
    k; ``release(k)`` marks the set free once the step that read it has been enqueued."""

    def __init__(self, model, rowptr, gene, label):
        self.m = model
        dev = model.device
        to_np = lambda a: a.cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
        rp, ge, la = to_np(rowptr).astype(np.int32), to_np(gene), to_np(label).astype(np.uint8)
        self.narrow = model.V <= 32768
        ge = ge.astype(np.int16 if self.narrow else np.int32)
        self.pins = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in (rp, ge, la)]
        mk = lambda: [torch.empty(rp.shape[0], dtype=torch.int32, device=dev),
                      torch.empty(ge.shape[0], dtype=torch.int32, device=dev),
                      torch.empty(la.shape[0], dtype=torch.uint8, device=dev)]
        self.bufs = [mk(), mk()]
        self.stage = [torch.empty(ge.shape[0], dtype=torch.int16, device=dev) for _ in (0, 1)] if self.narrow else None
        self.stream = torch.cuda.Stream(device=dev)
        self.ready = [torch.cuda.Event(), torch.cuda.Event()]
        self.freed = [torch.cuda.Event(), torch.cuda.Event()]
        for k in (0, 1):
            self.freed[k].record(torch.cuda.current_stream(dev))
        self.h2d_bytes = int(sum(p.numel() * p.element_size() for p in self.pins))

    def upload(self, k):
        with torch.cuda.stream(self.stream):
            self.stream.wait_event(self.freed[k])            # the step that last read this set is done
            b = self.bufs[k]
            b[0].copy_(self.pins[0], non_blocking=True)
            if self.narrow:
                self.stage[k].copy_(self.pins[1], non_blocking=True)
                b[1].copy_(self.stage[k])                    # int16 -> int32 on the device
            else:
                b[1].copy_(self.pins[1], non_blocking=True)
            b[2].copy_(self.pins[2], non_blocking=True)
            self.ready[k].record(self.stream)

    def use(self, k):
        torch.cuda.current_stream(self.m.device).wait_event(self.ready[k])
        self.m.rowptr, self.m.gene, self.m.label = self.bufs[k]

    def release(self, k):
        self.freed[k].record(torch.cuda.current_stream(self.m.device))


def _dist():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist
    return None


def train_cbow(win_rowptr, win_gene, labels, n_genes, hidden, lr, max_epoch=500, seed=0, optimizer="adam",
               reduce="sum", W_ih0=None, W_ho0=None, split=None, early_stop=True, log=print, return_info=False,
               eval_train="lazy", algo="rows", batch=0, use_graph=True, device_out=False):
    """Train the modified CBOW on CSR windows and return W_ih (np.float32 [n_genes, hidden]) exactly as
    ``compute_genetovec`` does: the weights after the last step whose validation accuracy did not drop.

    ``max_epoch`` is the reference's ``--epoch`` (parsed at G2Vec.py:515 but ignored there; the loop is
    hard-coded ``range(500)`` at :262) -- the default 500 reproduces the reference.

    ``batch``: 0 (default) = full batch, one optimizer step per epoch over all training windows as the
    reference does (:262-264).  ``batch = B > 0`` is the north_star's mini-batch variant: the (already
    shuffled) training windows are cut into consecutive batches of B, one optimizer step (and, multi-GPU,
    one gradient all-reduce) per batch, loss mean over the batch; ``batch >= n_train`` equals full batch.

    ``use_graph``: on one GPU with full batch, every step after the first replays a CUDA graph of the step's
    launches (the Adam step size lives on the device, g2v_cbow_adam_tick), so the host only replays, waits
    and applies the early-stop rule.

    ``device_out``: return W_ih as a float32 CUDA tensor [n_genes, hidden] instead of a NumPy copy (the steps
    after training then run on the device, g2vec_b200.post).
    """
    dist = _dist()
    world, rank = (dist.get_world_size(), dist.get_rank()) if dist else (1, 0)
    rowptr_np = (win_rowptr.cpu().numpy() if isinstance(win_rowptr, torch.Tensor) else np.asarray(win_rowptr))
    N = rowptr_np.shape[0] - 1
    if N < 2:
        raise ValueError("need at least two context windows")
    tr, va = split_indices(N, seed) if split is None else split
    if W_ih0 is None or W_ho0 is None:
        W_ih0, W_ho0 = init_weights(n_genes, hidden, seed)
    model = CbowModel(win_rowptr, win_gene, labels, n_genes, hidden, W_ih0, W_ho0, optimizer, reduce, lr, algo=algo,
                      nvl_group=dist.group.WORLD if (dist and algo == "rows") else None)
    lens = np.diff(rowptr_np).astype(np.int64)
    n_tr, n_va = len(tr), len(va)
    full_batch = batch <= 0 or batch >= n_tr
    tr_loc = shard_by_nnz(np.asarray(tr), lens, world, rank, keep_order=not full_batch)
    va_loc = shard_by_nnz(np.asarray(va), lens, world, rank)
    dev = model.device
    tr_d = torch.from_numpy(np.ascontiguousarray(tr_loc, dtype=np.int32)).to(dev)
    va_d = torch.from_numpy(np.ascontiguousarray(va_loc, dtype=np.int32)).to(dev)

    if algo == "rank1" and (batch <= 0 or batch >= n_tr) and len(tr_loc):
        model.prepare_csc(tr_d)
    if algo == "rows" and full_batch:            # tables larger than the L2: gene-slab passes over the static lists
        model.prepare_slabs(tr_d)
        model.prepare_slabs(va_d)
    if log:
        log("     Start training the modified CBOW with early stopping")
    if max_epoch <= 0:                           # no optimizer step at all: the initial vectors
        out, hist, stop = model.W_ih, [], None
    elif full_batch:
        out, hist, stop = _device_loop(model, dist, tr_d, va_d, n_tr, n_va, len(tr_loc), len(va_loc), max_epoch,
                                       early_stop, log, eval_train, use_graph)
    else:
        out, hist, stop = _minibatch_loop(model, dist, world, tr_d, va_d, n_tr, n_va, len(tr_loc), len(va_loc),
                                          max_epoch, early_stop, log, batch)
    if log:
        log("    Optimization Finish")
    out = out.detach().clone() if device_out else out.cpu().numpy()
    if return_info:
        return out, {"history": hist, "stop_step": stop, "n_train": n_tr, "n_val": n_va, "model": model,
                     "graph": bool(getattr(model, "loop_used_graph", False)), "exchange": model.exchange() if dist else None}
    return out


class _LoopLog:
    """The host side of the reference loop body after the three session runs (G2Vec.py:268-283): log line every
    5th step, the Epoch(stop) line, the history.  Fed one step at a time with the step's counters."""

    def __init__(self, n_tr, n_va, log):
        self.n_tr, self.n_va, self.log = n_tr, n_va, log
        self.hist, self.t0 = [], time.time()
        self.before_val, self.before_tr = np.float32(-1.0), np.float32(0.0)

    def step(self, step, acc, shown, stopped_here):
        f32 = np.float32
        acc_val = f32(int(acc[2])) / f32(max(self.n_va, 1))
        acc_tr_prev = f32(int(acc[1])) / f32(max(self.n_tr, 1))      # = ACC[tr] of step-1 (SURVEY 3.2-5)
        acc_tr = f32(int(acc[3])) / f32(max(self.n_tr, 1)) if shown else None
        hist, log = self.hist, self.log
        if hist and hist[-1][2] is None:
            hist[-1] = (hist[-1][0], hist[-1][1], float(acc_tr_prev))
        if hist:
            self.before_tr = hist[-1][2]                            # ACC[tr] of the previous step (G2Vec.py:281)
        hist.append((step, float(acc_val), None if acc_tr is None else float(acc_tr)))
        if step % 5 == 0 and log:
            t1 = time.time()
            log("    - Epoch: %03d\tACC[val]=%.4f\tACC[tr]=%.4f (%.3f sec)" % (step, acc_val, acc_tr, t1 - self.t0))
            self.t0 = time.time()
        if stopped_here:
            if log:
                log("    - Epoch(stop): %03d\tACC[val]=%.4f\tACC[tr]=%.4f (%.3f sec)"
                    % (step - 1, self.before_val, self.before_tr, time.time() - self.t0))
            return True
        self.before_val = acc_val
        return False


class DeviceLoop:
    """One model's training loop state on the device (g2v_cbow_loop_*) and the launches of one iteration of the
    reference loop (G2Vec.py:262-267): snapshot + zero counters, fwd+bwd, [all-reduce], optimizer, validation
    accuracy, [training accuracy], [all-reduce of the counters], decide.  Used by train_cbow and by bench.py."""

    def __init__(self, model, dist, tr_d, va_d, n_tr, max_epoch, early_stop, snapshot=True):
        self.m, self.dist, self.tr_d, self.va_d, self.n_tr = model, dist, tr_d, va_d, n_tr
        self.n_tr_loc, self.n_va_loc = int(tr_d.shape[0]), int(va_d.shape[0])
        dev = model.device
        self.ctl = torch.zeros(8, dtype=torch.int64, device=dev)
        n_hist = max(max_epoch, 1) * 4
        # with the NVLink exchange the history lives in symmetric memory and the accuracy counters of all ranks are
        # added into it by the ranks themselves (g2v_cbow_loop_counters_nvl): no NCCL call is left in the step
        self.hist_nvl = None
        if dist and model.nvl:
            try:
                import torch.distributed._symmetric_memory as symm
                h = symm.empty(n_hist, dtype=torch.int64, device=dev)
                hh = symm.rendezvous(h, dist.group.WORLD)
                self.hist_nvl = {"h": hh, "mc": int(hh.multicast_ptr or 0) if model.nvl["g_mc"] else 0}
                self.hist_d = h
            except Exception:
                self.hist_nvl = None
        if self.hist_nvl is None:
            self.hist_d = torch.zeros(n_hist, dtype=torch.int64, device=dev)
        self.ctl_pin = torch.zeros(8, dtype=torch.int64).pin_memory()
        self.hist_pin = torch.zeros(max(max_epoch, 1) * 4, dtype=torch.int64).pin_memory()
        # snapshot buffer: W_ih before the step being decided (only an early stop ever returns it)
        self.result = model.W_ih.clone() if snapshot else None
        self.max_epoch, self.early_stop = int(max_epoch), bool(early_stop)
        self.reset()

    def _st(self):
        return torch.cuda.current_stream(self.m.device).cuda_stream

    def reset(self):
        _capi.check(self.m.lib.g2v_cbow_loop_init(self.ctl.data_ptr(), self.max_epoch, int(self.early_stop), self._st()),
                    "g2v_cbow_loop_init")
        if self.hist_nvl:
            self.hist_nvl["h"].barrier(channel=2)    # no rank is still adding into the history of the previous loop
            self.hist_d.zero_()
            self.hist_nvl["h"].barrier(channel=2)    # ... and no rank adds before every history is zero

    def attach(self):
        _capi.check(self.m.lib.g2v_cbow_loop_attach(self.ctl.data_ptr()), "g2v_cbow_loop_attach")

    def detach(self):
        _capi.check(self.m.lib.g2v_cbow_loop_attach(None), "g2v_cbow_loop_attach")

    def one(self, show, m_fb=None, m_upd=None, m_val=None):
        """Enqueue one iteration (the optional events mark the end of fwd+bwd, of the update, of the validation pass)."""
        m, lib, dist = self.m, self.m.lib, self.dist
        _capi.check(lib.g2v_cbow_loop_begin(self.ctl.data_ptr(), m.acc.data_ptr(), m.W_ih.data_ptr(),
                                            None if self.result is None else self.result.data_ptr(), m.V * m.D,
                                            self._st()), "g2v_cbow_loop_begin")
        if self.n_tr_loc:
            m.fwdbwd(self.tr_d, self.n_tr)       # acc[1] += correct predictions with the PRE-update weights
        if m_fb is not None:
            m_fb.record()
        if dist:
            for g in m.grad_tensors():
                dist.all_reduce(g)               # rows: ONE collective over [g_ih | g_ho]; rank1: c
        m.update()
        if m_upd is not None:
            m_upd.record()
        if self.n_va_loc:
            m.evaluate(self.va_d, 2)
        if m_val is not None:
            m_val.record()
        if show and self.n_tr_loc:
            m.evaluate(self.tr_d, 3)
        acc_ptr = m.acc.data_ptr()
        if self.hist_nvl:
            hn = self.hist_nvl
            _capi.check(lib.g2v_cbow_loop_counters_nvl(self.ctl.data_ptr(), acc_ptr, hn["h"].buffer_ptrs_dev, hn["mc"],
                                                       m.nvl["world"], self._st()), "g2v_cbow_loop_counters_nvl")
            hn["h"].barrier(channel=3)
            acc_ptr = None                           # decide on the sums already in hist[step]
        elif dist:
            dist.all_reduce(m.acc[1:4])
        _capi.check(lib.g2v_cbow_loop_decide(self.ctl.data_ptr(), acc_ptr, self.hist_d.data_ptr(), self._st()),
                    "g2v_cbow_loop_decide")

    def fetch(self):
        self.ctl_pin.copy_(self.ctl, non_blocking=True)
        self.hist_pin.copy_(self.hist_d, non_blocking=True)

    def capture(self, pattern):
        """The iterations of `pattern` (list of show flags) + the status read-back as one CUDA graph."""
        g = torch.cuda.CUDAGraph()
        t_before = self.m.t
        with torch.cuda.graph(g):
            for sh in pattern:
                self.one(sh)
            self.fetch()
        self.m.t = t_before                      # capture records, it does not execute
        return g


def _device_loop(model, dist, tr_d, va_d, n_tr, n_va, n_tr_loc, n_va_loc, max_epoch, early_stop, log, eval_train,
                 use_graph, chunk=5):
    """Full-batch loop of G2Vec.py:262-283 with the early-stop rule, the result snapshot and the step counter on
    the DEVICE (g2v_cbow_loop_*): the host enqueues `chunk` iterations at a time -- one CUDA-graph replay of
    4 plain iterations + 1 that also runs the training-accuracy pass -- and synchronises once per printed line
    instead of once per step.  Iterations enqueued after the stop are no-ops (every kernel tests ctl.stopped).
    Multi-GPU: the all-reduces are part of the captured graph (NCCL is capturable); if capture is refused the
    same launches run eagerly."""
    dev = model.device
    loop = DeviceLoop(model, dist, tr_d, va_d, n_tr, max_epoch, early_stop, snapshot=bool(early_stop))
    shown = lambda s: s % 5 == 0 or eval_train == "always"
    info = _LoopLog(n_tr, n_va, log)

    def consume(lo, hi):
        """Host view of steps lo..hi-1 after a sync; True when the loop is over."""
        decided, stop_step = int(loop.ctl_pin[1]), int(loop.ctl_pin[2])
        for s in range(lo, min(hi, decided)):
            if info.step(s, loop.hist_pin[4 * s:4 * s + 4], shown(s), s == stop_step):
                return True
        return bool(int(loop.ctl_pin[0]))

    loop.attach()
    graph = None
    try:
        loop.one(True); loop.fetch()             # step 0 eagerly: it also warms every kernel up before a capture
        torch.cuda.current_stream(dev).synchronize()
        done, over = 1, consume(0, 1)
        graph_failed, graph_pattern = not use_graph, None
        while not over and done < max_epoch:
            k = min(chunk, max_epoch - done)
            pattern = [shown(done + i) for i in range(k)]
            if k == chunk and not graph_failed and graph is None:
                try:
                    graph, graph_pattern = loop.capture(pattern), pattern
                except Exception:
                    if dist is None:
                        raise
                    graph_failed = True          # collectives not capturable here: same launches, eagerly
            if graph is not None and pattern == graph_pattern:
                model.t += k
                graph.replay()
            else:
                for sh in pattern:
                    loop.one(sh)
                loop.fetch()
            torch.cuda.current_stream(dev).synchronize()        # one host sync per `chunk` steps
            over = consume(done, done + k)
            done += k
        stop = int(loop.ctl_pin[2]) if int(loop.ctl_pin[2]) >= 0 else None
        if stop is None and info.hist and info.hist[-1][2] is None:
            # ACC[tr] of the last step was never needed for a log line; evaluate it once for the history
            loop.detach()
            model.acc.zero_()
            if n_tr_loc:
                model.evaluate(tr_d, 3)
            if dist:
                dist.all_reduce(model.acc[1:4])
            a = model.acc.cpu()
            last = info.hist[-1]
            info.hist[-1] = (last[0], last[1], float(np.float32(int(a[3])) / np.float32(max(n_tr, 1))))
    finally:
        loop.detach()
    model.loop_used_graph = graph is not None
    # stopped early: the snapshot taken before the dropping step (G2Vec.py:283,286); else the final weights
    return (loop.result if stop is not None else model.W_ih), info.hist, stop


def _minibatch_loop(model, dist, world, tr_d, va_d, n_tr, n_va, n_tr_loc, n_va_loc, max_epoch, early_stop, log, batch):
    """north_star's mini-batch variant: one optimizer step (and one gradient all-reduce) per batch of the shuffled
    training list, the reference's per-epoch accuracies and early stop around it; host-driven, one sync per epoch."""
    dev = model.device
    info = _LoopLog(n_tr, n_va, log)
    result = model.W_ih.clone()
    stop = None
    per = -(-batch // world)
    for step in range(max_epoch):
        model.acc.zero_()
        for lo in range(0, -(-n_tr // world), per):             # same trip count on every rank (collectives inside)
            nb = max(0, min(per, n_tr_loc - lo))
            nb_tot = nb
            if dist:
                t_nb = torch.tensor([nb], dtype=torch.int64, device=dev); dist.all_reduce(t_nb)
                nb_tot = int(t_nb[0])
            model.fwdbwd(tr_d, nb_tot, win_begin=lo, n_win=nb)
            if dist:
                for g in model.grad_tensors():
                    dist.all_reduce(g)
            model.update()
        if n_va_loc:
            model.evaluate(va_d, 2)
        if n_tr_loc:
            model.evaluate(tr_d, 3)                              # acc[1] mixes weights across batches: always evaluate
        if dist:
            dist.all_reduce(model.acc[1:4])
        acc = model.acc.cpu()                                    # the epoch's only host sync
        dropped = bool(early_stop) and (np.float32(int(acc[2])) / np.float32(max(n_va, 1))) < info.before_val
        if info.step(step, acc, True, dropped):
            stop = step
            break
        result.copy_(model.W_ih)
    return result, info.hist, stop


def compute_genetovec(pathList, n_genes, hidden_size, learning_rate, max_epoch=500, seed=0, log=print):
    """Drop-in for the reference signature (G2Vec.py:217): dense ``pathList`` [N, n_genes+1] in
    (last column = label), W_ih out."""
    from .paths import dense_pathlist_to_csr
    rowptr, gene, label = dense_pathlist_to_csr(pathList)
    return train_cbow(rowptr, gene, label, n_genes, hidden_size, learning_rate, max_epoch=max_epoch, seed=seed,
                      log=log)


def cbow_step_host(rowptr, gene, label, W_ih, W_ho, state=None, lr=0.005, t=1, optimizer="adam", reduce="sum",
                   beta1=0.9, beta2=0.999, eps=1e-8):
    """One full-batch step through ``g2v_cbow_step_host``: NumPy in, NumPy updated in place."""
    lib = _capi.load()
    rowptr = np.ascontiguousarray(rowptr, dtype=np.int32); gene = np.ascontiguousarray(gene, dtype=np.int32)
    label = np.ascontiguousarray(label, dtype=np.uint8)
    V, D = W_ih.shape
    for a in (W_ih, W_ho):
        assert a.dtype == np.float32 and a.flags.c_contiguous
    opt = {"adam": _capi.OPT_ADAM_TF1, "sgd": _capi.OPT_SGD}[optimizer]
    if opt == _capi.OPT_ADAM_TF1 and state is None:
        state = [np.zeros_like(W_ih), np.zeros_like(W_ih), np.zeros_like(W_ho), np.zeros_like(W_ho)]
    p = lambda a: 0 if a is None else a.ctypes.data
    m_ih, v_ih, m_ho, v_ho = state if state is not None else (None,) * 4
    loss = np.zeros(1, dtype=np.float64); nc = np.zeros(1, dtype=np.int64)
    rc = lib.g2v_cbow_step_host(rowptr.ctypes.data, gene.ctypes.data, label.ctypes.data, rowptr.shape[0] - 1,
                                gene.shape[0], W_ih.ctypes.data, W_ho.ctypes.data, p(m_ih), p(v_ih), p(m_ho),
                                p(v_ho), V, D, opt, {"sum": 0, "mean": 1}[reduce], lr, beta1, beta2, eps, t,
                                loss.ctypes.data, nc.ctypes.data)
    _capi.check(rc, "g2v_cbow_step_host")
    return state, float(loss[0]), int(nc[0])
