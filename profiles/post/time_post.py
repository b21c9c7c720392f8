"""Steps 5-7 of the command line, --post host vs --post gpu, on seeded inputs of three shapes.

    python profiles/post/time_post.py --out profiles/post/time_post_b200.json [--shapes ex,20k,200k]

Inputs per shape: gene vectors = three Gaussian blobs of unequal size (seeded), expression [135, V] normal with the
ex_* sample labels' 0/1 split (seeded).  For each shape:
  host   cli.find_lgroups + the step-6 loop of cli.main + the three cli writers, by wall clock;
  gpu    post.find_lgroups + post.select_biomarkers + the two small writers + post.write_vectors, by wall clock
         ending in a device synchronise (median of 3 after one warm-up run), plus CUDA events per kernel phase;
         formatting (kernels and the copy to pinned memory, text discarded) is timed apart from the whole
         write_vectors call, and the file writing is the difference.
Both paths' three files are compared byte for byte before any time is reported.  Each Lloyd iteration's kernels
(assign + update + status) are timed with CUDA events on the final centres and reported as V*D*4 bytes read over
that time, against the HBM bandwidth of a 4 GiB device-to-device copy measured in the same run.  The card's name
and power limit are printed and stored with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

SHAPES = {"ex": (7523, 128), "20k": (20_000, 256), "200k": (200_000, 512)}
N_BIOMARKER = 50


def inputs(V, D, seed):
    rng = np.random.default_rng(seed)
    sizes = [V // 2, V // 3, V - V // 2 - V // 3]
    centres = rng.normal(0, 1.0, size=(3, D))
    mat = np.concatenate([rng.normal(c, 0.6, size=(n, D)) for c, n in zip(centres, sizes)]).astype(np.float32)
    mat = mat[rng.permutation(V)]
    expr = rng.normal(size=(135, V)).astype(np.float32)
    label = (rng.random(135) < 0.45).astype(np.int64)
    genes = np.array(["G%06d" % i for i in range(V)])
    return mat, expr, label, genes


def host_steps(prefix, mat, expr, label, genes):
    from g2vec_b200 import cli
    t0 = time.perf_counter()
    lgroup = cli.find_lgroups(mat, genes, None)
    t1 = time.perf_counter()
    biomarkers = []
    for i in (0, 1):
        sel = lgroup == i
        d = cli.minmax(np.linalg.norm(mat[sel], axis=1))
        t = cli.minmax(cli.tscores(expr[:, sel], label))
        score = 0.5 * (d + t)
        ranked = sorted(zip(genes[sel], score), key=lambda gs: gs[1], reverse=True)
        biomarkers += sorted(g for g, _ in ranked[:N_BIOMARKER])
    biomarkers = sorted(biomarkers)
    t2 = time.perf_counter()
    cli.write_biomarkers(prefix, biomarkers)
    cli.write_lgroups(prefix, lgroup, genes)
    t3 = time.perf_counter()
    cli.write_vectors(prefix, genes, mat)
    t4 = time.perf_counter()
    return {"step5_s": t1 - t0, "step6_s": t2 - t1, "step7_small_writers_s": t3 - t2, "step7_vectors_s": t4 - t3,
            "total_s": t4 - t0}


def gpu_steps(prefix, mat_d, expr_d, label, genes):
    import torch
    from g2vec_b200 import cli, post
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    lgroup, fell_back = post.find_lgroups(mat_d)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    biomarkers = post.select_biomarkers(mat_d, expr_d, label, lgroup, genes, N_BIOMARKER)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    cli.write_biomarkers(prefix, biomarkers)
    cli.write_lgroups(prefix, lgroup, genes)
    t3 = time.perf_counter()
    emit = []
    post.write_vectors(prefix, genes, mat_d, timing=emit)
    torch.cuda.synchronize()
    t4 = time.perf_counter()
    return {"step5_s": t1 - t0, "step6_s": t2 - t1, "step7_small_writers_s": t3 - t2, "step7_vectors_s": t4 - t3,
            "total_s": t4 - t0, "fallback": bool(fell_back),
            "emit_kernel_ms": sum(a.elapsed_time(b) for a, b in emit)}


def events_ms(fn, reps):
    import torch
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def kernel_phases(mat_d, expr_d, label, genes):
    """CUDA-event times of each phase of the GPU path, and the Lloyd iteration's bandwidth."""
    import torch
    from g2vec_b200 import _capi, post
    lib = _capi.load()
    V, D = mat_d.shape
    st = torch.cuda.current_stream().cuda_stream
    res = post.kmeans(mat_d)
    ws = torch.empty(int(lib.g2v_kmeans_workspace_bytes(V, D, 3)), dtype=torch.uint8, device="cuda")
    Xc = torch.empty_like(mat_d)
    mean = torch.empty(D, dtype=torch.float32, device="cuda")
    var = torch.empty(D, dtype=torch.float64, device="cuda")
    center = lambda: _capi.check(lib.g2v_kmeans_center(mat_d.data_ptr(), V, D, Xc.data_ptr(), mean.data_ptr(),
                                                       var.data_ptr(), ws.data_ptr(), st), "center")
    center()
    lab = torch.from_numpy(res.labels.astype(np.int64)).cuda()
    centres = torch.stack([Xc[lab == k].mean(0) for k in range(3)]).contiguous()
    cnew = torch.empty_like(centres)
    l_old = torch.from_numpy(res.labels).cuda()
    l_new = torch.empty_like(l_old)
    status = torch.empty(8, dtype=torch.float64, device="cuda")
    lloyd = lambda: _capi.check(lib.g2v_kmeans_lloyd_step(Xc.data_ptr(), V, D, 3, centres.data_ptr(), cnew.data_ptr(),
                                                          l_old.data_ptr(), l_new.data_ptr(), status.data_ptr(),
                                                          ws.data_ptr(), st), "lloyd")
    ids = np.array(res.init_ids, dtype=np.int64)
    dout = torch.empty((3, V), dtype=torch.float32, device="cuda")
    closest = torch.zeros(V, dtype=torch.float32, device="cuda")
    dist = lambda: _capi.check(lib.g2v_kmeans_dist(Xc.data_ptr(), V, D, ids.ctypes.data, 3, closest.data_ptr(),
                                                   dout.data_ptr(), st), "dist")
    lloyd_ms = events_ms(lloyd, 50)
    out = {"kmeans_n_iter": res.n_iter, "kmeans_strict": res.strict,
           "center_ms": events_ms(center, 20), "kmeanspp_dist_3cand_ms": events_ms(dist, 20),
           "lloyd_iter_ms": lloyd_ms, "lloyd_iter_bytes": V * D * 4,
           "lloyd_iter_GBps": V * D * 4 / (lloyd_ms * 1e-3) / 1e9,
           "tscores_ms": events_ms(lambda: post.tscores(expr_d, label), 20),
           "row_norms_ms": events_ms(lambda: post.row_norms(mat_d), 20)}
    t0 = time.perf_counter()
    emit = []
    n = sum(len(b) for b in post._chunks(mat_d, [g.encode() for g in genes], post.CHUNK_BYTES, lambda b: b, emit))
    torch.cuda.synchronize()
    out["format_to_pinned_s"] = time.perf_counter() - t0
    out["format_emit_kernel_ms"] = sum(a.elapsed_time(b) for a, b in emit)
    out["vectors_text_bytes"] = int(n)
    return out


def hbm_copy_GBps():
    import torch
    n = 4 << 30
    a = torch.empty(n, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    ms = events_ms(lambda: b.copy_(a), 10)
    return 2 * n / (ms * 1e-3) / 1e9


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--shapes", default="ex,20k,200k")
    args = ap.parse_args()
    import torch
    from g2vec_b200 import _capi
    _capi.load()
    info = card()
    print(json.dumps(info))
    result = {"card": info, "hbm_copy_GBps": hbm_copy_GBps(), "shapes": {}}
    print("HBM copy: %.0f GB/s" % result["hbm_copy_GBps"])
    for name in args.shapes.split(","):
        V, D = SHAPES[name]
        mat, expr, label, genes = inputs(V, D, V + D)
        mat_d, expr_d = torch.from_numpy(mat).cuda(), torch.from_numpy(expr).cuda()
        with tempfile.TemporaryDirectory() as tmp:
            host = host_steps(os.path.join(tmp, "host"), mat, expr, label, genes)
            gpu_steps(os.path.join(tmp, "gpu"), mat_d, expr_d, label, genes)           # warm-up
            runs = [gpu_steps(os.path.join(tmp, "gpu"), mat_d, expr_d, label, genes) for _ in range(3)]
            for suffix in ("_biomarkers.txt", "_lgroups.txt", "_vectors.txt"):
                with open(os.path.join(tmp, "host" + suffix), "rb") as f1, open(os.path.join(tmp, "gpu" + suffix), "rb") as f2:
                    if f1.read() != f2.read():
                        raise SystemExit("%s: %s differs between --post host and --post gpu" % (name, suffix))
        gpu = {k: float(np.median([r[k] for r in runs])) for k in runs[0] if k != "fallback"}
        gpu["fallback"] = any(r["fallback"] for r in runs)
        phases = kernel_phases(mat_d, expr_d, label, genes)
        phases["lloyd_iter_fraction_of_hbm_copy"] = phases["lloyd_iter_GBps"] / result["hbm_copy_GBps"]
        gpu["step7_file_write_s"] = gpu["step7_vectors_s"] - phases["format_to_pinned_s"]
        result["shapes"][name] = {"V": V, "D": D, "host": host, "gpu": gpu, "kernels": phases,
                                  "files_equal": True, "speedup_total": host["total_s"] / gpu["total_s"]}
        print(name, json.dumps(result["shapes"][name]))
        del mat_d, expr_d
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
