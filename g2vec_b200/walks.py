"""HOT PATH 1, host side: the walk sampler behind the reference's call
``generate_pathSet(adjMat, args.lenPath, args.numRepetition)`` (/root/reference/G2Vec.py:62,
324-352).  The work is done by ``g2v_walk_launch`` (csrc/g2v_walk.cu) on the current CUDA
device; this module only owns buffers (torch tensors) and the walker-range bookkeeping.
"""
import numpy as np
import torch

from . import _capi, graph as _graph


def _dev(device=None):
    if not torch.cuda.is_available():
        raise RuntimeError("g2vec_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)


def _to_dev(a, dtype, device):
    if isinstance(a, torch.Tensor):
        return a.to(device=device, dtype=dtype).contiguous()
    a = np.ascontiguousarray(a)
    if dtype == torch.int32 and a.dtype == np.uint32:
        a = a.view(np.int32)           # same bits; the kernel reads uint32
    return torch.from_numpy(a).to(device=device, dtype=dtype, non_blocking=True)


def _check_qw(qw):
    """Integer weights must satisfy qw <= 2^24 (include/g2vec_b200.h): the sampler sums up to 64 of them in 32 bits.
    int32 storage holds the uint32 bits, so a negative entry is a weight >= 2^31."""
    if isinstance(qw, torch.Tensor):
        top = int((qw.to(torch.int64) & 0xFFFFFFFF).max()) if qw.numel() else 0
    else:
        a = np.asarray(qw)
        top = int((a.astype(np.int64) & 0xFFFFFFFF).max()) if a.size else 0
    if top > _graph.Q_MAX:
        raise ValueError("integer edge weight %d exceeds the limit qw <= 2^24 = %d" % (top, _graph.Q_MAX))


class WalkGraph:
    """One group's directed weighted graph resident in HBM as CSR
    (rowptr int32 [V+1], col int32 [E] ascending per row, qw uint32 [E] stored as int32 bits)."""

    def __init__(self, rowptr, col, weights=None, qw=None, device=None):
        if qw is not None:
            _check_qw(qw)
        device = _dev(device)
        if qw is None:
            if weights is None:
                raise ValueError("need weights or qw")
            if isinstance(weights, torch.Tensor) and weights.is_cuda:
                # same rule as graph.quantise_weights (rint = round-half-even), kept on the device
                wd = weights.to(torch.float32).double()
                if wd.numel() and (not bool(torch.isfinite(wd).all()) or bool((wd < 0).any())):
                    raise ValueError("edge weights must be finite and non-negative")
                q = torch.round(wd * _graph.Q_ONE)
                q = torch.where((wd > 0) & (q < 1), torch.ones_like(q), q)
                if q.numel() and float(q.max()) > _graph.Q_MAX:
                    raise ValueError("edge weight too large to quantise")
                qw = q.to(torch.int32)
            else:
                qw = _graph.quantise_weights(np.asarray(weights.cpu() if isinstance(weights, torch.Tensor) else weights))
        self.rowptr = _to_dev(rowptr, torch.int32, device)
        self.col = _to_dev(col, torch.int32, device)
        self.qw = _to_dev(qw, torch.int32, device)
        self.V = int(self.rowptr.shape[0]) - 1
        self.E = int(self.col.shape[0])
        if self.qw.shape[0] != self.E:
            raise ValueError("col / weight length mismatch")
        self.device = device
        lib = _capi.load()
        self._ws = torch.zeros(max(int(lib.g2v_walk_workspace_bytes()), 64), dtype=torch.uint8, device=device)
        # packed layouts, built once per graph by g2v_walk_prepare: rows = {begin, end} pairs, edges = {col, qw}
        # pairs (layout 1) or 16+16-bit words, two neighbours per 8-byte load (layout 2: V <= 65535 and weights in
        # the |PCC| range [0.5, 1])
        import ctypes
        rb, eb = ctypes.c_size_t(0), ctypes.c_size_t(0)
        _capi.check(lib.g2v_walk_packed_bytes(self.V, self.E, ctypes.byref(rb), ctypes.byref(eb)), "g2v_walk_packed_bytes")
        self.rows = torch.empty(max(rb.value, 8), dtype=torch.uint8, device=device)
        self.edges = torch.empty(max(eb.value, 8), dtype=torch.uint8, device=device)
        lay = ctypes.c_int32(0)
        with torch.cuda.device(device):
            st = torch.cuda.current_stream().cuda_stream
            _capi.check(lib.g2v_walk_prepare(self.rowptr.data_ptr(), self.col.data_ptr(), self.qw.data_ptr(), self.V,
                                             self.E, self.rows.data_ptr(), self.edges.data_ptr(), ctypes.byref(lay),
                                             self._ws.data_ptr(), st), "g2v_walk_prepare")
        self.layout = int(lay.value)

    @classmethod
    def from_dense(cls, adjMat, device=None):
        rp, col, w = _graph.csr_from_dense(adjMat)
        return cls(rp, col, weights=w, device=device)

    def nbytes(self):
        return 4 * (self.V + 1) + 8 * self.E


def num_walkers(V, reps, begin=0, end=None, stride=1):
    end = V * reps if end is None else end
    return max(0, (end - begin + stride - 1) // stride)


def generate_paths(g, len_path, reps, seed=0, group=0, walker_begin=0, walker_end=None, walker_stride=1,
                   out=None, canonical=False, plain_csr=False):
    """Run walkers w = walker_begin + i*walker_stride < walker_end (w = rep*V + src) of graph ``g``.

    Returns (nodes int32 [n, len_path] in VISIT order padded with -1, lens int32 [n]) as device
    tensors; asynchronous on the current stream.

    ``canonical=True`` fuses ``path = tuple(sorted(path))`` (G2Vec.py:345) into the sampler: the rows come back
    sorted ascending and padded with INT32_MAX, and a third tensor holds their 64-bit keys (what
    ``paths.canonical_rows`` would otherwise compute from the visit-order rows in a second kernel).
    ``plain_csr=True`` runs the kernel on the unpacked CSR arrays through ``g2v_walk_launch``."""
    lib = _capi.load()
    end = g.V * reps if walker_end is None else walker_end
    n = num_walkers(g.V, reps, walker_begin, end, walker_stride)
    if out is None:
        nodes = torch.empty((n, len_path), dtype=torch.int32, device=g.device)
        lens = torch.empty((n,), dtype=torch.int32, device=g.device)
        key = torch.empty((n,), dtype=torch.int64, device=g.device) if canonical else None
    else:
        nodes, lens = out[0], out[1]
        key = out[2] if canonical else None
        assert nodes.shape == (n, len_path) and lens.shape == (n,) and nodes.is_contiguous()
    with torch.cuda.device(g.device):
        st = torch.cuda.current_stream().cuda_stream
        if plain_csr:
            if canonical:
                raise ValueError("canonical rows need the packed graph")
            rc = lib.g2v_walk_launch(g.rowptr.data_ptr(), g.col.data_ptr(), g.qw.data_ptr(), g.V, g.E, int(len_path),
                                     int(seed) & (2**64 - 1), int(group), int(walker_begin), int(end),
                                     int(walker_stride), nodes.data_ptr(), lens.data_ptr(), g._ws.data_ptr(), st)
        else:
            rc = lib.g2v_walk_launch_packed(g.rows.data_ptr(), g.edges.data_ptr(), g.layout, g.V, g.E, int(len_path),
                                            int(seed) & (2**64 - 1), int(group), int(walker_begin), int(end),
                                            int(walker_stride), nodes.data_ptr(), lens.data_ptr(),
                                            0 if key is None else key.data_ptr(), g._ws.data_ptr(), st)
    _capi.check(rc, "g2v_walk_launch")
    if canonical:
        return nodes, lens, key
    return nodes, lens


def generate_paths_host(rowptr, col, qw, len_path, reps, seed=0, group=0, walker_begin=0, walker_end=None,
                        walker_stride=1):
    """Same through ``g2v_walk_host``: NumPy arrays in, NumPy arrays out (the C ABI does the copies)."""
    lib = _capi.load()
    rowptr = np.ascontiguousarray(rowptr, dtype=np.int32); col = np.ascontiguousarray(col, dtype=np.int32)
    qw = np.ascontiguousarray(qw, dtype=np.uint32)
    V = rowptr.shape[0] - 1
    end = V * reps if walker_end is None else walker_end
    n = num_walkers(V, reps, walker_begin, end, walker_stride)
    # page-locked result buffers: the device->host copy of the rows then runs at PCIe speed
    nodes = torch.empty((n, len_path), dtype=torch.int32, pin_memory=True).numpy()
    lens = torch.empty((n,), dtype=torch.int32, pin_memory=True).numpy()
    rc = lib.g2v_walk_host(rowptr.ctypes.data, col.ctypes.data, qw.ctypes.data, V, col.shape[0], int(len_path),
                           int(seed) & (2**64 - 1), int(group), int(walker_begin), int(end), int(walker_stride),
                           nodes.ctypes.data, lens.ctypes.data)
    _capi.check(rc, "g2v_walk_host")
    return nodes, lens


def generate_pathSet(adjMat, maximumLength, iterations, seed=0, group=0):
    """Drop-in for the reference's ``generate_pathSet(adjMat, maximumLength, iterations)``
    (G2Vec.py:324): dense adjacency (or a WalkGraph) in, ``set`` of sorted int tuples out."""
    g = adjMat if isinstance(adjMat, WalkGraph) else WalkGraph.from_dense(adjMat)
    nodes, lens = generate_paths(g, maximumLength, iterations, seed=seed, group=group)
    nodes = nodes.cpu().numpy(); lens = lens.cpu().numpy()
    return {tuple(sorted(int(x) for x in row[:n])) for row, n in zip(nodes, lens)}
