"""The command line's steps 5-7 on the GPU (``--post gpu``): L-groups by k-means, biomarkers by gene scores, and
the vectors file, from the device-resident vectors that ``train_cbow(..., device_out=True)`` returns.

The host functions in ``cli`` stay the reference this path is compared with:
- ``find_lgroups``: KMeans(n_clusters=3, random_state=0) as scikit-learn 1.x runs it (``sklearn/cluster/_kmeans.py``):
  data centred on its float32 column mean, k-means++ with 2 + int(log k) local trials, Lloyd iterations until the
  labels stop changing or the squared centre shift is <= 1e-4 * mean per-feature variance, then one last assignment.
  The distance passes run on the device (csrc/g2v_post.cu); the random draws, the cumulative sum and the
  searchsorted run here in NumPy with scikit-learn's expressions, so the chosen initial ids are scikit-learn's.
  scikit-learn relocates a cluster that becomes empty; this path does not: it falls back to scikit-learn for that call.
  The cluster-to-L-group renumbering is ``cli.lgroups_from_clusters`` for both paths.
- ``tscores`` and the row norms are kernels; min-max, the average and the top-n use torch as plumbing.
- ``write_vectors`` formats on the device ("\\t%.6f", byte for byte as Python prints a float) in row chunks of at
  most ``chunk_bytes`` of text and writes each chunk as it comes back.

Nothing here imports scikit-learn unless the fallback runs.
"""
import numpy as np
import torch

from . import _capi
from . import cli

N_CLUSTERS = 3
MAX_ITER = 300
TOL = 1e-4
CHUNK_BYTES = 256 << 20


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def _as_device_f32(mat):
    if not isinstance(mat, torch.Tensor):
        raise TypeError("expected a CUDA tensor")
    if not mat.is_cuda:
        raise RuntimeError("g2vec_b200.post needs CUDA tensors; there is no CPU fallback")
    return mat.detach().to(torch.float32).contiguous()


# ------------------------------------------------------------------------------------- step 5: k-means
def kmeans_plusplus_ids(n_samples, dist, n_clusters=N_CLUSTERS, random_state=0, sample_weight=None):
    """k-means++ seeding of scikit-learn's ``_kmeans_plusplus``, with the distance passes delegated:
    ``dist(ids, closest)`` returns the float32 [len(ids), n_samples] squared distances of every row to the rows
    ``ids``, element-wise min'd with ``closest`` when it is not None.  Draws, potentials, cumulative sums and
    searchsorted are scikit-learn's own NumPy expressions on the same dtypes, in the same order."""
    rs = random_state if isinstance(random_state, np.random.RandomState) else np.random.RandomState(random_state)
    w = np.ones(n_samples, dtype=np.float32) if sample_weight is None else np.asarray(sample_weight)
    n_local_trials = 2 + int(np.log(n_clusters))
    center_id = rs.choice(n_samples, p=w / w.sum())
    indices = np.full(n_clusters, -1, dtype=int)
    indices[0] = center_id
    closest_dist_sq = dist(np.array([center_id]), None)[:1]            # [1, n]
    current_pot = closest_dist_sq @ w
    for c in range(1, n_clusters):
        rand_vals = rs.uniform(size=n_local_trials) * current_pot
        candidate_ids = np.searchsorted(np.cumsum(w * closest_dist_sq), rand_vals)
        np.clip(candidate_ids, None, closest_dist_sq.size - 1, out=candidate_ids)
        distance_to_candidates = dist(candidate_ids, closest_dist_sq.reshape(-1))
        candidates_pot = distance_to_candidates @ w.reshape(-1, 1)
        best = np.argmin(candidates_pot)
        current_pot = candidates_pot[best]
        closest_dist_sq = distance_to_candidates[best]
        indices[c] = candidate_ids[best]
    return indices


class KMeansResult:
    """labels (np.int32 [V], or None when a cluster became empty), the k-means++ ids, Lloyd iterations run,
    whether the labels converged strictly, and the absolute tolerance on the squared centre shift."""

    def __init__(self, labels, init_ids, n_iter, strict, tol):
        self.labels, self.init_ids, self.n_iter, self.strict, self.tol = labels, init_ids, n_iter, strict, tol


def kmeans(mat, n_clusters=N_CLUSTERS, random_state=0, max_iter=MAX_ITER, tol=TOL):
    """KMeans(n_clusters, random_state).fit(mat).labels_ on the device (see the module docstring).  Returns a
    KMeansResult; its labels are None if a cluster became empty (scikit-learn would relocate it)."""
    lib = _capi.load()
    X = _as_device_f32(mat)
    V, D = X.shape
    K = n_clusters
    if V < K:
        raise ValueError("n_samples=%d should be >= n_clusters=%d" % (V, K))
    dev, st = X.device, _stream(X)
    ws = torch.empty(int(lib.g2v_kmeans_workspace_bytes(V, D, K)), dtype=torch.uint8, device=dev)
    Xc = torch.empty_like(X)
    mean = torch.empty(D, dtype=torch.float32, device=dev)
    var = torch.empty(D, dtype=torch.float64, device=dev)
    _capi.check(lib.g2v_kmeans_center(X.data_ptr(), V, D, Xc.data_ptr(), mean.data_ptr(), var.data_ptr(),
                                      ws.data_ptr(), st), "g2v_kmeans_center")
    tol_abs = float(var.mean().item()) * tol

    out = torch.empty((8, V), dtype=torch.float32, device=dev)

    def dist(ids, closest):
        ids = np.ascontiguousarray(ids, dtype=np.int64)
        cl = None if closest is None else torch.from_numpy(np.ascontiguousarray(closest, dtype=np.float32)).to(dev)
        _capi.check(lib.g2v_kmeans_dist(Xc.data_ptr(), V, D, ids.ctypes.data, len(ids),
                                        0 if cl is None else cl.data_ptr(), out.data_ptr(), st), "g2v_kmeans_dist")
        return out[:len(ids)].cpu().numpy()

    ids = kmeans_plusplus_ids(V, dist, K, random_state)
    centres = Xc[torch.from_numpy(ids).to(dev)].contiguous()
    centres_new = torch.empty_like(centres)
    labels = torch.full((V,), -1, dtype=torch.int32, device=dev)
    labels_old = labels.clone()
    status = torch.empty(2 + 2 * K, dtype=torch.float64, device=dev)
    strict, it = False, 0
    for it in range(max_iter):
        _capi.check(lib.g2v_kmeans_lloyd_step(Xc.data_ptr(), V, D, K, centres.data_ptr(), centres_new.data_ptr(),
                                              labels_old.data_ptr(), labels.data_ptr(), status.data_ptr(),
                                              ws.data_ptr(), st), "g2v_kmeans_lloyd_step")
        s = status.cpu().numpy()
        if s[1] > 0:
            return KMeansResult(None, ids, it + 1, False, tol_abs)
        centres, centres_new = centres_new, centres
        if s[0] == 0:
            strict = True
            break
        if s[2 + K:].sum() <= tol_abs:
            break
        labels, labels_old = labels_old, labels
    if not strict:
        _capi.check(lib.g2v_kmeans_lloyd_step(Xc.data_ptr(), V, D, K, centres.data_ptr(), 0, 0, labels.data_ptr(),
                                              0, 0, st), "g2v_kmeans_lloyd_step")
    return KMeansResult(labels.cpu().numpy(), ids, it + 1, strict, tol_abs)


def find_lgroups(mat, gene_names=None, geneFreq=None):
    """cli.find_lgroups on device vectors: k-means on the device, scikit-learn's KMeans on the host only if a
    cluster became empty.  Returns (lgroup np.int32 [V], fell_back)."""
    res = kmeans(mat)
    km, fell_back = res.labels, False
    if km is None:
        from sklearn.cluster import KMeans
        km = KMeans(n_clusters=N_CLUSTERS, random_state=0).fit(mat.cpu().numpy()).labels_
        fell_back = True
    return cli.lgroups_from_clusters(km), fell_back


# ---------------------------------------------------------------------------------- step 6: gene scores
def tscores(expr, label):
    """cli.tscores for every gene at once: expr [S, V] (device, sample-major), label [S] (0 good, 1 poor).
    Returns float32 [V] on the device.  An empty group raises ZeroDivisionError, as cli.tscore does."""
    lib = _capi.load()
    x = _as_device_f32(expr)
    S, V = x.shape
    label = np.asarray(label)
    if not (label == 0).any() or not (label == 1).any():
        raise ZeroDivisionError("float division by zero")
    lab = np.where(label == 0, 0, np.where(label == 1, 1, 2)).astype(np.uint8)
    lab_d = torch.from_numpy(lab).to(x.device)
    t = torch.empty(V, dtype=torch.float32, device=x.device)
    _capi.check(lib.g2v_post_tscores(x.data_ptr(), S, V, lab_d.data_ptr(), t.data_ptr(), _stream(x)),
                "g2v_post_tscores")
    return t


def row_norms(mat):
    lib = _capi.load()
    X = _as_device_f32(mat)
    out = torch.empty(X.shape[0], dtype=torch.float32, device=X.device)
    _capi.check(lib.g2v_post_row_norms(X.data_ptr(), X.shape[0], X.shape[1], out.data_ptr(), _stream(X)),
                "g2v_post_row_norms")
    return out


def _minmax(x):
    """cli.minmax in float32: (1 - 0) / (max - min) * (x - min) + 0."""
    mn, mx = x.min(), x.max()
    return (1.0 / (mx - mn)) * (x - mn) + 0.0


def select_biomarkers(mat, expr, label, lgroup, genes, n_biomarker):
    """Step 6 of cli.main: per L-group 0 and 1, score = (minmax(||W_ih row||) + minmax(|t|)) / 2, the top
    n_biomarker genes (ties by ascending gene index, as the host's stable sort gives), names sorted."""
    X = _as_device_f32(mat)
    d_all = row_norms(X)
    t_all = tscores(expr, label)
    out = []
    lg = torch.from_numpy(np.asarray(lgroup)).to(X.device)
    for i in (0, 1):
        sel = torch.nonzero(lg == i).flatten()
        score = 0.5 * (_minmax(d_all[sel]) + _minmax(t_all[sel]))
        order = torch.sort(score, descending=True, stable=True).indices[:n_biomarker]
        top = sel[order].cpu().numpy()
        out += sorted(np.asarray(genes)[top].tolist())
    return sorted(out)


# ----------------------------------------------------------------------------------- step 7: the vectors file
def format_rows(mat, prefixes=None, chunk_bytes=CHUNK_BYTES):
    """The lines of mat [rows, D] (device) as bytes: prefix + "\\t%.6f" x D + "\\n" per row (prefixes: a list of
    bytes, or None), formatted in chunks of at most chunk_bytes as write_vectors does."""
    return b"".join(_chunks(_as_device_f32(mat), prefixes, chunk_bytes, lambda b: bytes(b)))


def _prefix_arrays(prefixes, dev):
    if prefixes is None:
        return None, None
    lens = np.fromiter((len(p) for p in prefixes), dtype=np.int64, count=len(prefixes))
    off = np.zeros(len(prefixes) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    blob = np.frombuffer(b"".join(prefixes) or b"\0", dtype=np.uint8)
    return torch.from_numpy(blob.copy()).to(dev), torch.from_numpy(off).to(dev)


def _chunks(X, prefixes, chunk_bytes, sink, timing=None):
    """Format X in row chunks of at most chunk_bytes of text (at least one row each) and hand each chunk's bytes
    (a memoryview of pinned host memory, valid during the call) to sink in order.  Two device/pinned buffer pairs:
    chunk i+1 is formatted and copied while sink writes chunk i."""
    lib = _capi.load()
    rows, D = X.shape
    dev, st = X.device, _stream(X)
    blob, poff = _prefix_arrays(prefixes, dev)
    row_bytes = torch.empty(rows, dtype=torch.int64, device=dev)
    _capi.check(lib.g2v_fmt_row_bytes(X.data_ptr(), rows, D, 0 if poff is None else poff.data_ptr(),
                                      row_bytes.data_ptr(), st), "g2v_fmt_row_bytes")
    ends = torch.cumsum(row_bytes, 0)
    ends_h = ends.cpu().numpy()
    total = int(ends_h[-1]) if rows else 0
    starts = ends - row_bytes                                    # exclusive scan: byte offset of each line
    # row chunks: each ends at the last row whose end stays within chunk_bytes of the chunk's start (>= 1 row)
    bounds, r = [0], 0
    while r < rows:
        base = int(ends_h[r - 1]) if r else 0
        nxt = int(np.searchsorted(ends_h, base + chunk_bytes, side="right"))
        r = max(nxt, r + 1)
        bounds.append(r)
    cap = max(int(ends_h[b - 1] - (ends_h[a - 1] if a else 0)) for a, b in zip(bounds[:-1], bounds[1:])) if rows else 1
    dbuf = [torch.empty(cap, dtype=torch.uint8, device=dev) for _ in range(2)]
    hbuf = [torch.empty(cap, dtype=torch.uint8, pin_memory=True) for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]
    pending = None
    for ci, (a, b) in enumerate(zip(bounds[:-1], bounds[1:])):
        k = ci & 1
        base = int(ends_h[a - 1]) if a else 0
        n = int(ends_h[b - 1]) - base
        off = (starts[a:b] - base).contiguous()
        ev0 = torch.cuda.Event(enable_timing=True) if timing is not None else None
        if ev0 is not None:
            ev0.record()
        _capi.check(lib.g2v_fmt_emit(X[a:].data_ptr(), b - a, D, 0 if blob is None else blob.data_ptr(),
                                     0 if poff is None else poff[a:].data_ptr(), off.data_ptr(),
                                     dbuf[k].data_ptr(), st), "g2v_fmt_emit")
        if ev0 is not None:
            ev1 = torch.cuda.Event(enable_timing=True)
            ev1.record()
            timing.append((ev0, ev1))
        hbuf[k][:n].copy_(dbuf[k][:n], non_blocking=True)
        done[k].record()
        if pending is not None:
            pk, pn = pending
            done[pk].synchronize()
            yield sink(memoryview(hbuf[pk].numpy())[:pn])
        pending = (k, n)
    if pending is not None:
        pk, pn = pending
        done[pk].synchronize()
        yield sink(memoryview(hbuf[pk].numpy())[:pn])
    assert total == sum(int(ends_h[b - 1] - (ends_h[a - 1] if a else 0)) for a, b in zip(bounds[:-1], bounds[1:]))


def write_vectors(prefix, genes, mat, chunk_bytes=CHUNK_BYTES, timing=None):
    """cli.write_vectors with the numbers formatted on the device: the same bytes in prefix + "_vectors.txt".
    The header goes through the same text-mode file; the gene names are encoded with that file's encoding."""
    X = _as_device_f32(mat)
    with open(prefix + "_vectors.txt", 'w') as f:
        f.write('GeneSymbol' + ''.join('\tV%d' % i for i in range(X.shape[1])) + '\n')
        f.flush()
        names = [str(g).encode(f.encoding, f.errors) for g in genes]
        if len(names) != X.shape[0]:
            raise ValueError("%d gene names for %d rows" % (len(names), X.shape[0]))
        for _ in _chunks(X, names, chunk_bytes, f.buffer.write, timing):
            pass
