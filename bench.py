#!/usr/bin/env python
"""bench.py -- throughput of the two G2Vec hot paths on B200 (BASELINE.json metric:
"CBOW context-windows/sec and random-walk steps/sec at 1/2/4/8 B200 vs CPU ref").

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
    python bench.py --impl reference --gpus N ...          # the reference's own CPU implementation
    python bench.py ... --dump-outputs DIR                 # + the outputs of the last timed walk pass / CBOW step

--dump-outputs writes, after the timed steps of the headline workload (rank 0):
  walk_rows, walk_lens, walk_keys  generate_paths(canonical=True) of the last timed pass for a fixed sample of 8192
                                   walkers (walk_index: their rows in the group-0-then-group-1 buffer); keys as two
                                   32-bit words
  cbow_W_ih, cbow_W_ho             the weights after the last timed step of --algo (W_ih: a fixed row sample,
                                   cbow_W_ih_rows, when it exceeds 48 MiB)
  cbow_accuracy                    that step's validation and training accuracy
All inputs are seeded, so two builds run with the same arguments can be compared output for output.

One "step":  CBOW  = one iteration of the reference's training loop (G2Vec.py:262-267): a full-batch
                     optimizer step over all training windows (fwd+bwd+[all-reduce]+update) plus the
                     validation and training accuracy passes, launched exactly as g2vec_b200.train_cbow
                     launches it (g2vec_b200.cbow.DeviceLoop: early-stop bookkeeping on the device, one CUDA
                     graph replay per step);
             walks = one pass of the sampler over every walker of both patient groups.
The headline `value` is CBOW context windows/s (training windows x steps / time, both accuracy passes inside
the timed region, as the reference runs them); the walk sampler's steps/s is in the `walk` object of the same
line.  Workload at N=1: BASELINE configs[1] (synthetic 10k genes / 500k edges per group, 128-dim, lenPath 80,
10 repetitions -> 200k walkers / ~200k windows of 80 genes).  N>1: weak scaling -- every rank keeps that per-GPU
work (numRepetition = 10*N), parameters replicated, dense gradient NCCL-all-reduced once per step.

Extra blocks of the same JSON line:
  roofline       the fused fwd+bwd kernel of the headline config.  Its table + gradient (10 MB) live in the L2, so
                 the bound is the L2 / L1TEX path, and the peak it is divided by is MEASURED in the same run:
                 g2v_test_l2_rows reads / red.adds the same rows with the arithmetic removed.
  roofline_hbm   (N=1) the same kernel on BASELINE configs[4]'s table -- 200k genes x 512 = 410 MB, far beyond the
                 L2 -- on synthetic windows (SURVEY 8d: 80 distinct genes, seed 777): the single-pass kernel against
                 the measured HBM peak, and the gene-slab passes that ship for such tables (csrc/g2v_cbow_slab.cu).
  production_loop  measured: 5-step CUDA graphs of what train_cbow runs (training-accuracy pass on every 5th
                 step only, snapshot of the weights inside the graph).
  parity         (N>1) computed in-run: re-assembled walker shards == oracle on a 2000-walker sample; the
                 all-reduced gradient of a 4096-window batch vs the same batch on one rank.
  strong         strong scaling of BASELINE configs[3] (50k genes, lenPath 160) and configs[2] (20k genes, 256-dim):
                 total work fixed, walkers and windows sharded over the N ranks.

Timing: CUDA events on the launching stream, W warm-up steps, L2 flushed (256 MiB write) before every
timed step, max over ranks.  CPU baseline: the UNMODIFIED reference (oracle/_ref/G2Vec.py, staged by
__graft_entry__.build(); its TF 1.x ops on oracle/tf1_shim.py) on a bounded sample, on this box's host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "cbow_context_windows_per_sec"
UNIT = "windows/s"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--workload", default="syn10k", choices=["syn10k", "syn20k", "syn50k", "stress200k", "ex"])
    p.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    p.add_argument("--reps", type=int, default=10, help="numRepetition per GPU (weak) or in total (strong)")
    p.add_argument("--optimizer", default="adam", choices=["adam", "sgd"])
    p.add_argument("--algo", default="rows", choices=["rows", "rank1"],
                   help="CBOW formulation the headline value is measured on (rows = north_star's gather/scatter kernel)")
    p.add_argument("--no-alt-algo", action="store_true", help="do not also time the other formulation")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-hbm", action="store_true", help="skip the roofline_hbm block (N=1)")
    p.add_argument("--no-strong", action="store_true", help="skip the strong-scaling block")
    p.add_argument("--no-parity", action="store_true", help="skip the in-run parity block (N>1)")
    p.add_argument("--hbm-reps", type=int, default=2, help="numRepetition of the roofline_hbm windows (2*reps*V windows)")
    p.add_argument("--strong-workloads", nargs="*", default=["syn50k", "syn20k"])
    p.add_argument("--cpu-sample-windows", type=int, default=16384)
    p.add_argument("--cpu-walk-seconds", type=float, default=8.0)
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the headline workload's last timed walk pass and CBOW step "
                        "computed as DIR/<name>.npy (rank 0; a fixed, seeded row sample where an array is large)")
    a = p.parse_args()
    if a.steps < 1 or a.warmup < 0:
        p.error("--steps must be at least 1 and --warmup at least 0")
    return a


def workload(name):
    from g2vec_b200 import graph
    if name == "ex":
        z = np.load(os.path.join(ROOT, "tests", "golden", "ex_graph.npz"))
        gs = [(z["rowptr%d" % g], z["col%d" % g], z["w%d" % g]) for g in (0, 1)]
        return gs, 7523, 128, 80, "ex_* graphs (tests/golden/ex_graph.npz, made by the reference's construct_adjMat)"
    V, E, D, L = graph.BENCH_CONFIGS[name]
    gs = [graph.synthetic_graph(V, E, g) for g in (0, 1)]
    return gs, V, D, L, "synthetic directed ER, %d genes / %d edges per group, weights U(0.5,1)" % (V, E)


_RUN = {"reps": None, "world": 1}


def traffic_lookup(kernel, workload_name, need_reps=None):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the named kernel from the
    committed ncu capture of this same command (profiles/traffic.json); None when no capture exists for this
    workload / numRepetition / GPU count."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            e = json.load(f)[kernel][workload_name]
        reps = _RUN["reps"] if need_reps is None else need_reps
        return e["dram_bytes"] if (e.get("reps") == reps and _RUN["world"] == 1) else None
    except Exception:
        return None


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return None
        load = [x for x in sm if x > 0.5 * max(sm)] or sm
        return {"sm_mhz": float(np.median(load)), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


DUMP_BYTES = 64 << 20            # --dump-outputs: all arrays together
DUMP_WALKERS = 8192              # walker rows in the walk sample (float64, L <= 160: at most 10.5 MB)
DUMP_W_IH_BYTES = 48 << 20       # W_ih rows beyond this are sampled (stress200k: 410 MB)


def sample_rows(n, cap, seed=0):
    """Sorted indices of a fixed, seeded sample of min(n, cap) of n rows (all of them when n <= cap)."""
    if n <= cap:
        return np.arange(n, dtype=np.int64)
    return np.sort(np.random.RandomState(seed).choice(n, cap, replace=False))


def key_words(keys):
    """int64 keys -> [n, 2] (high, low) 32-bit words, which float64 holds exactly."""
    k = np.asarray(keys, dtype=np.int64).view(np.uint64)
    return np.stack([k >> np.uint64(32), k & np.uint64(0xFFFFFFFF)], axis=1)


def write_outputs(out_dir, arrays):
    """--dump-outputs: every array as out_dir/<name>.npy, integers as float64 (exact below 2^53), floats as float32."""
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32 if np.asarray(a).dtype.kind == "f" else np.float64)
        total += a.nbytes
        np.save(os.path.join(out_dir, name + ".npy"), a)
    assert total <= DUMP_BYTES, "--dump-outputs wrote %d bytes" % total
    print("bench.py: wrote %d arrays (%.1f MB) to %s" % (len(arrays), total / 1e6, out_dir), file=sys.stderr)


def synthetic_windows(N, V, L, device, seed=777):
    """SURVEY 8d: N windows of L distinct genes uniform over V, labels Bernoulli(0.5).  Sorted and distinct by
    construction: L draws from [0, V-L] sorted, plus 0..L-1."""
    import torch
    g = torch.Generator(device=device); g.manual_seed(seed)
    x = torch.randint(0, V - L + 1, (N, L), generator=g, device=device, dtype=torch.int32)
    x, _ = torch.sort(x, dim=1)
    x += torch.arange(L, device=device, dtype=torch.int32)[None, :]
    label = (torch.rand(N, generator=g, device=device) < 0.5).to(torch.uint8)
    rowptr = torch.arange(0, (N + 1) * L, L, device=device, dtype=torch.int32)
    return rowptr, x.reshape(-1).contiguous(), label


# =============================================================================== this repo's arm
def run_b200(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL announces its version on stdout when the communicator is created; keep stdout for the one JSON
        # line by pointing fd 1 at stderr while the group comes up (first collective included)
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    assert world == args.gpus, "--gpus must equal WORLD_SIZE"
    import g2vec_b200 as g2v
    from g2vec_b200 import _capi, paths, cbow
    lib = _capi.load()
    ddist = dist if world > 1 else None

    def allmax(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    def allsum(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev); dist.all_reduce(t)
        return float(t[0])

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    K, W = args.steps, args.warmup
    _RUN.update(reps=args.reps, world=world)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    peak, peak_src = peaks()

    def timed(fn, n, marks=0):
        """n steps, each: L2 flush, start event, fn(marks...), end event.  Returns per-step ms (+ inner marks)."""
        pairs = []
        for i in range(n):
            flush_buf.fill_(i & 0xFF)
            a, b = ev(), ev()
            inner = [ev() for _ in range(marks)]
            a.record(); fn(*inner) if marks else fn(); b.record()
            pairs.append((a, b, inner))
        torch.cuda.synchronize()
        tot = [a.elapsed_time(b) for a, b, _ in pairs]
        inn = [[a.elapsed_time(m) for m in inner] for a, _, inner in pairs]
        return tot, inn

    sampler = ClockSampler(local) if rank == 0 else None
    launches0 = _capi.launch_count()

    # ------------------------------------------------------------------------------------------ one pipeline
    def pipeline(wl_name, reps_total, hidden=None, want_e2e=False, want_cbow_detail=False, steps=K, warm=W, dump=None):
        """Walks -> windows -> CBOW steps for one workload; walkers rank::world, windows of the rank's own walkers.
        `dump` (a dict) receives the outputs of the last timed walk pass and of the last timed step of args.algo."""
        gs, V, D, L, desc = workload(wl_name)
        D = hidden or D
        graphs = [g2v.WalkGraph(rp, col, weights=w) for rp, col, w in gs]
        n_walk = g2v.walks.num_walkers(V, reps_total, rank, None, world)
        # both groups' rows in ONE buffer (group 0 first): the set pipeline then needs no concatenation
        all_rows = torch.empty((2 * n_walk, L), dtype=torch.int32, device=dev)
        all_lens = torch.empty((2 * n_walk,), dtype=torch.int32, device=dev)
        all_keys = torch.empty((2 * n_walk,), dtype=torch.int64, device=dev)
        outs = [(all_rows[g * n_walk:(g + 1) * n_walk], all_lens[g * n_walk:(g + 1) * n_walk],
                 all_keys[g * n_walk:(g + 1) * n_walk]) for g in (0, 1)]

        def walk_pass(canonical=True):
            for g in (0, 1):
                g2v.generate_paths(graphs[g], L, reps_total, seed=12345, group=g, walker_begin=rank, walker_stride=world,
                                   out=outs[g], canonical=canonical)

        # visit-order pass first: the byte model needs to know which visits scanned their row
        timed(lambda: walk_pass(False), max(1, warm))
        barrier()
        vt, _ = timed(lambda: walk_pass(False), min(steps, 5))
        barrier()
        visits = allsum(int(sum(int(o[1].sum()) for o in outs)))
        # algorithmic bytes of one pass: per visit 4 B (node id written); per visit that scans its row
        # (every visit but the L-th of a full-length walk) 8 B rowptr + 8 B per neighbour (col + weight)
        wbytes = 0
        for g in (0, 1):
            nodes, lens = outs[g][0], outs[g][1]
            deg = (graphs[g].rowptr[1:] - graphs[g].rowptr[:-1]).to(torch.int64)
            scan = nodes[:, :L - 1] if L > 1 else nodes[:, :0]
            m = scan >= 0
            wbytes += int(lens.sum()) * 4 + int(m.sum()) * 8 + 8 * int(deg[scan[m].to(torch.int64)].sum())
        # production pass: tuple(sorted(path)) fused into the sampler (sorted rows + keys out)
        timed(walk_pass, warm)
        barrier()
        l0 = _capi.launch_count()
        wt, _ = timed(walk_pass, steps)
        barrier()
        walk_launches = _capi.launch_count() - l0
        if dump is not None:
            # what generate_paths(canonical=True) returned in the last timed pass: sorted rows, lengths, 64-bit keys
            idx = sample_rows(2 * n_walk, DUMP_WALKERS)
            sel = torch.from_numpy(idx).to(dev)
            dump.update(walk_index=idx, walk_rows=all_rows[sel].cpu().numpy(), walk_lens=all_lens[sel].cpu().numpy(),
                        walk_keys=key_words(all_keys[sel].cpu().numpy()))
        walk_ms = allmax(float(np.mean(wt)))
        res = {"V": V, "D": D, "L": L, "desc": desc, "walk_ms": walk_ms, "walk_visit_order_ms": allmax(float(np.mean(vt))),
               "visits": visits, "walk_launches": walk_launches, "n_walk": n_walk, "wbytes": wbytes,
               "walk_gbs": wbytes / (float(np.mean(wt)) * 1e-3) / 1e9, "layout": graphs[0].layout}

        if want_e2e:
            qws = [g2v.graph.quantise_weights(w) for _, _, w in gs]
            def walk_host_pass():
                for g in (0, 1):
                    g2v.generate_paths_host(gs[g][0], gs[g][1], qws[g], L, reps_total, seed=12345, group=g,
                                            walker_begin=rank, walker_stride=world)
            walk_host_pass()
            barrier(); t0 = time.perf_counter()
            for _ in range(max(1, min(steps, 3))):
                walk_host_pass()
            barrier(); dt = allmax((time.perf_counter() - t0) / max(1, min(steps, 3)))
            csr_b = sum(4 * (len(rp)) + 8 * len(col) for rp, col, _ in gs)
            res["walk_e2e"] = {"value": visits / dt, "unit": "steps/s", "h2d_bytes_per_step": int(csr_b),
                               "d2h_bytes_per_step": int(2 * n_walk * (L + 1) * 4), "api": "g2v_walk_host (C ABI, host buffers)"}

        # ---- windows from the walks: set semantics of G2Vec.py:351,313 + CSR + geneFreq (csrc/g2v_paths.cu)
        grp = torch.cat([torch.zeros(n_walk, dtype=torch.uint8, device=dev), torch.ones(n_walk, dtype=torch.uint8, device=dev)])
        rowptr, gene, label, _code = paths.build_windows(all_rows, all_lens, all_keys, grp, V)   # sort-free set pipeline
        del all_rows, all_lens, all_keys, grp, outs
        N_loc = int(rowptr.shape[0]) - 1
        lens_np = np.diff(rowptr.cpu().numpy()).astype(np.int64)
        tr, va = cbow.split_indices(N_loc, 1000 + rank)
        n_tr_tot, n_va_tot = int(allsum(len(tr))), int(allsum(len(va)))
        W0, Wo0 = cbow.init_weights(V, D, 0)
        tr_d = torch.from_numpy(tr.astype(np.int32)).to(dev); va_d = torch.from_numpy(va.astype(np.int32)).to(dev)
        res.update(n_tr=n_tr_tot, n_va=n_va_tot, mean_len=float(lens_np.mean()), ltr=lens_np[tr], gs=gs,
                   windows=(rowptr, gene, label), tr_d=tr_d, va_d=va_d)

        def measure(algo):
            model = g2v.CbowModel(rowptr, gene, label, V, D, W0, Wo0, optimizer=args.optimizer, lr=0.005, algo=algo,
                                  nvl_group=dist.group.WORLD if (world > 1 and algo == "rows") else None)
            model.prepare_csc(tr_d)                    # rank1: transposed incidence of the static training list
            slabs = model.prepare_slabs(tr_d)          # rows, table > L2: gene-slab passes
            model.prepare_slabs(va_d)
            # the device skips every step past the loop's step cap, so the cap must exceed the longest run of steps
            # between two resets (warm-up + timed steps; the 5-step production graphs run at most steps + 10)
            loop = cbow.DeviceLoop(model, ddist, tr_d, va_d, n_tr_tot, max(512, warm + steps + 10), False)
            loop.attach()

            def snapshot():
                """The weights and the two accuracies of the last step run (dump)."""
                loop.fetch(); torch.cuda.synchronize()
                s = int(loop.ctl_pin[1]) - 1
                correct = loop.hist_pin[4 * s:4 * s + 4].numpy()
                rows = sample_rows(V, DUMP_W_IH_BYTES // (4 * D))
                dump.update(cbow_W_ih=model.W_ih[torch.from_numpy(rows).to(dev)].cpu().numpy(),
                            cbow_W_ho=model.W_ho.cpu().numpy(),
                            cbow_accuracy=np.array([correct[2] / max(n_va_tot, 1), correct[3] / max(n_tr_tot, 1)]))
                if len(rows) < V:
                    dump["cbow_W_ih_rows"] = rows
            take = dump is not None and algo == args.algo
            try:
                timed(lambda *m: loop.one(True, *m), warm, marks=3)
                barrier()
                l0 = _capi.launch_count()
                ct, marks = timed(lambda *m: loop.one(True, *m), steps, marks=3)
                barrier()
                if take:
                    snapshot()
                r = {"launches": _capi.launch_count() - l0, "eager_ms": allmax(float(np.mean(ct))),
                     "fb_ms": float(np.mean([m[0] for m in marks])),
                     "upd_ms": allmax(float(np.mean([m[1] for m in marks]))),
                     "val_ms": allmax(float(np.mean([m[2] for m in marks]))), "slabs": bool(slabs),
                     "n_slabs": getattr(model, "_n_slabs", 1), "model": model, "loop": loop,
                     "exchange": model.exchange() if world > 1 else None}
                r["step_ms"], r["graph"] = r["eager_ms"], False
                loop.reset()
                try:                                    # what train_cbow runs: the same launches as CUDA graphs
                    g_full = loop.capture([True])
                    timed(g_full.replay, warm)
                    barrier()
                    gt, _ = timed(g_full.replay, steps)
                    barrier()
                    if take:
                        snapshot()
                    r["step_ms"], r["graph"] = allmax(float(np.mean(gt))), True
                    loop.reset()
                    g_prod = loop.capture([False] * 4 + [True])
                    timed(g_prod.replay, 1)
                    barrier()
                    pt, _ = timed(g_prod.replay, max(2, steps // 5 + 1))
                    barrier()
                    r["prod_ms"] = allmax(float(np.mean(pt))) / 5.0
                except Exception as exc:                # collectives not capturable on this box: eager numbers stand
                    if world == 1:
                        raise
                    r["graph_error"] = repr(exc)[:200]
                loop.fetch(); torch.cuda.synchronize()
                r["acc_val"] = int(loop.hist_pin[2]) / max(n_va_tot, 1)
            finally:
                loop.detach()
            r["value"] = n_tr_tot / (r["step_ms"] * 1e-3)
            return r
        res["measure"] = measure
        return res

    # ------------------------------------------------------------------------------------------ headline
    reps_total = args.reps * (world if args.scaling == "weak" else 1)
    outputs = {} if (args.dump_outputs and rank == 0) else None
    P = pipeline(args.workload, reps_total, want_e2e=not args.no_e2e, dump=outputs)
    V, D, L, desc = P["V"], P["D"], P["L"], P["desc"]
    n_tr_tot, n_va_tot, ltr = P["n_tr"], P["n_va"], P["ltr"]
    rowptr, gene, label = P["windows"]
    l2_bytes = 126e6
    walkers_total = int(allsum(2 * P["n_walk"]))
    WALK = {"metric": "random_walk_steps_per_sec", "value": P["visits"] / (P["walk_ms"] * 1e-3), "unit": "steps/s",
            "ms_per_pass": P["walk_ms"], "walkers": walkers_total, "visits_per_pass": P["visits"],
            "mode": "tuple(sorted(path)) fused into the sampler (sorted rows + 64-bit keys out); graph packed as "
                    + {1: "{col, qw} pairs (8 B per edge)", 2: "16+16-bit words (4 B per edge, two neighbours per lane)"}[P["layout"]],
            "visit_order_ms_per_pass": P["walk_visit_order_ms"],
            "roofline": {"kernel": "walk_kernel", "bound": "issue", "achieved": P["walk_gbs"], "peak": peak,
                         "unit": "GB/s", "frac": P["walk_gbs"] / peak,
                         "traffic": traffic_lookup("walk", args.workload),
                         "algorithmic_bytes_per_pass": P["wbytes"],
                         "bytes_model": "4 B per visit + (8 + 8*deg) B per visit that scans its row",
                         "note": "ncu: the CSR is L2-resident (DRAM traffic 0.1 % of the algorithmic bytes) and the kernel is "
                                 "bound by instruction issue (75-87 % of the issue slots), not by bytes; the fraction of the HBM "
                                 "peak is reported because SURVEY 8d defines the walk roofline that way"},
            "e2e": P.get("walk_e2e")}
    walk_launches = P["walk_launches"]

    def l2_rows_peak(model):
        """GB/s at which the gather (LDG.128) and the scatter (RED.128) of the SAME rows run with the arithmetic
        removed: the memory-path ceiling of the fused kernel on this (L2-resident) table."""
        idx = model.gene
        n = int(idx.shape[0])
        sink = torch.zeros(1024, dtype=torch.float32, device=dev)
        scratch = torch.zeros_like(model.g_ih)
        st = lambda: torch.cuda.current_stream(dev).cuda_stream
        out = {}
        for mode, name in ((0, "gather"), (1, "red")):
            fn = lambda: _capi.check(lib.g2v_test_l2_rows(model.W_ih.data_ptr(), scratch.data_ptr(), idx.data_ptr(), n, D,
                                                          mode, sink.data_ptr(), st()), "g2v_test_l2_rows")
            timed(fn, 2)
            t, _ = timed(fn, 5)
            out[name] = n * D * 4 / (float(np.mean(t)) * 1e-3) / 1e9
        return out

    def roofline_of(algo, r):
        opt_b = (32 if args.optimizer == "adam" else 16) * V * D
        if algo == "rows":
            b = int((ltr * (8 * D + 4) + 5).sum())          # SURVEY 8d: l*(8D+4)+5 per window
            gbs = b / (r["fb_ms"] * 1e-3) / 1e9
            resident = 2 * V * D * 4 < 0.75 * l2_bytes
            out = {"kernel": ("cbow_slab_fwd_kernel + cbow_slab_bwd_kernel passes (%d gene slabs)" % r["n_slabs"]) if r["slabs"]
                             else "cbow_rows_kernel<%d,true> (fused gather/sum/logit/BCE/scatter-add)" % max(D // 128, 0),
                   "achieved": gbs, "unit": "GB/s", "kernel_ms": r["fb_ms"], "algorithmic_bytes_per_launch": b,
                   "bytes_model": "sum over this rank's training windows of l*(8D+4)+5; the optimizer epilogue "
                                  "(%d B) is a separate kernel" % opt_b,
                   "hbm_peak": peak, "frac_of_hbm_peak": gbs / peak, "peak_source": peak_src,
                   "traffic": traffic_lookup("cbow_rows_fwdbwd", args.workload)}
            if resident and D in (128, 256, 512) and not r["slabs"]:
                pk = l2_rows_peak(r["model"])
                half = float(ltr.sum()) * D * 4               # bytes gathered = bytes added
                # the gathers (L2 reads) and the REDs (L2 atomic units) of different warps overlap: the slower of the
                # two streams bounds the kernel
                l2pk = 2 * half / max(half / pk["gather"], half / pk["red"])
                out.update(bound="l2", peak=l2pk, frac=gbs / l2pk,
                           l2_peaks={"gather_GBps": pk["gather"], "red_GBps": pk["red"],
                                     "how": "g2v_test_l2_rows on the same table and the same row ids, arithmetic removed; "
                                            "the two streams overlap, so peak = bytes / max(gather bytes / gather rate, added bytes / RED rate) "
                                            "= 2 x the RED rate here: the L2 atomic units are the ceiling"},
                           note="W_ih + gradient (%.0f MB) are L2-resident at this config (ncu: DRAM traffic 0.5 %% of the "
                                "algorithmic bytes, l1tex 77 %%, lts 65 %%): the bound is the L2/L1TEX path, not HBM; "
                                "frac_of_hbm_peak is kept only for reference" % (2 * V * D * 4 / 1e6))
            elif r["slabs"]:
                out.update(bound="l2", peak=peak, frac=gbs / peak,
                           note="W_ih + gradient (%.0f MB) exceed the L2; the step runs gene slab by gene slab so that rows are "
                                "L2-resident within a pass (forward: L2 reads; backward: L2 atomic units -- ncu l1tex 87 %%, lts "
                                "61 %%, DRAM ~0): the algorithmic rate is divided by the measured HBM peak only for reference "
                                "and exceeds it; the single-pass kernel on this table is 0.74 of the HBM peak (roofline_hbm)"
                                % (2 * V * D * 4 / 1e6))
            else:
                out.update(bound="hbm", peak=peak, frac=gbs / peak,
                           note="W_ih + gradient (%.0f MB) exceed the L2" % (2 * V * D * 4 / 1e6))
            return out
        b = (28 if args.optimizer == "adam" else 12) * V * D      # update rows R/W W,m,v + prepare re-read of W
        ms = r["upd_ms"] - r["fb_ms"]
        gbs = b / (ms * 1e-3) / 1e9
        return {"kernel": "r1_update_kernel + r1_update_ho_kernel + r1_prepare_kernel (dense optimizer pass)",
                "bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                "traffic": traffic_lookup("r1_update", args.workload), "peak_source": peak_src, "kernel_ms": ms,
                "algorithmic_bytes_per_launch": b,
                "bytes_model": "28*V*D (Adam: read W,m,v + write W,m,v, then re-read W for s); the window kernels "
                               "(forward + CSC segmented sum) move only %d B (16*l+9 per window) in %.3f ms"
                               % (int((ltr * 16 + 9).sum()), r["fb_ms"])}

    main = P["measure"](args.algo)
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    main_roofline = roofline_of(args.algo, main)
    alt = "rank1" if args.algo == "rows" else "rows"
    ALT = None
    if not args.no_alt_algo:
        ALT = P["measure"](alt)
        ALT["roofline"] = roofline_of(alt, ALT)
        ALT.pop("model"); ALT.pop("loop")
        torch.cuda.empty_cache()
    model, loop = main.pop("model"), main.pop("loop")
    step_ms, upd_ms, value, acc_val, cbow_launches = main["step_ms"], main["upd_ms"], main["value"], main["acc_val"], main["launches"]

    e2e = None
    if not args.no_e2e:
        # Every step's windows come from pinned host memory.  The upload of step k+1 runs on a copy stream
        # into the other of two device buffer sets while step k computes (input double-buffering); the timed
        # region contains every copy and the per-step device->host read of the loop status + accuracy counters.
        orig = (model.rowptr, model.gene, model.label)
        feeder = g2v.WindowFeeder(model, *orig)
        loop.reset(); loop.attach()

        # one CUDA graph per device buffer set (the kernels' window pointers are baked into a graph), as in `value`
        graphs = [None, None]
        try:
            for k in (0, 1):
                feeder.upload(k); feeder.use(k)
                torch.cuda.current_stream().synchronize()
                graphs[k] = loop.capture([True])
                feeder.release(k)
        except Exception:
            if world == 1:
                raise
            graphs = [None, None]                               # collectives not capturable here: eager launches

        def e2e_run(n):
            feeder.upload(0)
            for i in range(n):
                k = i & 1
                if i + 1 < n:
                    feeder.upload(k ^ 1)
                feeder.use(k)                                   # compute stream waits for this step's upload
                if graphs[k] is not None:
                    graphs[k].replay()
                else:
                    loop.one(True); loop.fetch()
                feeder.release(k)
                torch.cuda.current_stream().synchronize()       # the accuracies are on the host
        try:
            e2e_run(2)
            barrier(); t0 = time.perf_counter()
            e2e_run(K)
            barrier(); dt = allmax((time.perf_counter() - t0) / K)
        finally:
            loop.detach()
        model.rowptr, model.gene, model.label = orig
        e2e = {"value": n_tr_tot / dt, "unit": UNIT,
               "h2d_bytes_per_step": feeder.h2d_bytes,
               "d2h_bytes_per_step": int(loop.ctl_pin.numel() * 8 + loop.hist_pin.numel() * 8),
               "api": "g2vec_b200.cbow.DeviceLoop step (C ABI kernels, one CUDA-graph replay) fed by g2vec_b200.WindowFeeder: every step's windows "
                      "are uploaded from pinned host memory (double-buffered on a copy stream, gene ids as int16 when "
                      "n_genes <= 32768) and the loop status + accuracy counters are read back every step"}
        del feeder
    windows_host = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        windows_host = (rowptr.cpu().numpy(), gene.cpu().numpy(), label.cpu().numpy())
    gs_head = P["gs"]
    mean_len = P["mean_len"]
    del model, loop, P, rowptr, gene, label
    torch.cuda.empty_cache()

    # ------------------------------------------------------------------------------------------ roofline_hbm
    hbm = None
    if world == 1 and not args.no_hbm:
        hbm = roofline_hbm(args, g2v, cbow, dev, timed, peak, peak_src, K, W)

    # ------------------------------------------------------------------------------------------ parity (N>1)
    parity = None
    if world > 1 and not args.no_parity:
        parity = parity_block(g2v, dist, rank, world, dev, gs_head, V, L)

    # ------------------------------------------------------------------------------------------ strong scaling
    strong = None
    if not args.no_strong and args.scaling == "weak" and args.workload == "syn10k":
        strong = {}
        for wl in args.strong_workloads:
            S = pipeline(wl, 10, steps=max(3, K // 2), warm=2)
            r = S["measure"]("rows")
            r.pop("model"); r.pop("loop")
            strong[wl] = {"value": r["value"], "unit": UNIT, "ms_per_step": r["step_ms"], "windows_train": S["n_tr"],
                          "graph": r["graph"], "gene_slabs": r["n_slabs"], "exchange": r["exchange"],
                          "walk": {"value": S["visits"] / (S["walk_ms"] * 1e-3), "unit": "steps/s", "ms_per_pass": S["walk_ms"]},
                          "config": "%s: %s, hidden %d, lenPath %d, numRepetition 10 in total over %d GPU(s)"
                                    % (wl, S["desc"], S["D"], S["L"], world)}
            del S, r
            torch.cuda.empty_cache()
        strong["note"] = ("strong scaling: total work fixed (10 repetitions), walkers rank::world, every rank trains on the "
                          "windows of its own walkers, one dense gradient all-reduce per step; speed-up(N) = value(N) / value(1) "
                          "from the N = 1 line of the same sweep")

    clocks = sampler.stop() if sampler else None
    total_launches = _capi.launch_count() - launches0

    # ------------------------------------------------------------------ CPU baseline (rank 0, N=1)
    cpu = walk_cpu = None
    if windows_host is not None:
        cpu, walk_cpu = cpu_baseline(args, gs_head, V, D, L, *windows_host)
    WALK["cpu_baseline"] = walk_cpu

    if rank == 0:
        prod_ms = main.get("prod_ms")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic" if args.workload != "ex" else "ex_* graphs (fixture)",
            "config": {"workload": "%s: %s, hidden %d, lenPath %d, numRepetition %d%s" % (
                           args.workload, desc, D, L, reps_total,
                           " (%d per GPU)" % args.reps if args.scaling == "weak" and world > 1 else ""),
                       "windows_train": n_tr_tot, "windows_val": n_va_tot, "mean_window_len": mean_len,
                       "optimizer": args.optimizer, "step": "fwd+bwd+update + val acc + train acc (G2Vec.py:262-267)",
                       "launch": ("one CUDA graph replay per step%s (eager launches: %.3f ms per step)"
                                  % (", NCCL all-reduces inside the graph" if world > 1 else "", main["eager_ms"]))
                                 if main.get("graph") else "eager launches",
                       "parallelism": "dp%d (windows/walkers sharded, W replicated; gradient exchange per step: %s; the 3 "
                                      "accuracy counters: %s)" % (
                                          world, main.get("exchange") or "none",
                                          "added into every rank's history over NVLS (multimem.red), no NCCL call in the step"
                                          if (main.get("exchange") or "").startswith("nvl") else "one 24-byte all_reduce"),
                       "l2": "256 MiB flush write before every timed step"},
            "train_only": {"value": n_tr_tot / (upd_ms * 1e-3), "unit": UNIT, "ms_per_step": upd_ms,
                           "note": "fwd+bwd+all-reduce+update, without the two accuracy passes (eager launches)"},
            "production_loop": None if prod_ms is None else {
                "value": n_tr_tot / (prod_ms * 1e-3), "unit": UNIT, "ms_per_step": prod_ms,
                "note": "MEASURED: 5-step CUDA graphs as g2vec_b200.train_cbow replays them -- snapshot of the weights, "
                        "fwd+bwd, update, validation accuracy every step; the training-accuracy pass of G2Vec.py:267 only on "
                        "the step that prints it (it equals the next step's training forward); early-stop rule on the "
                        "device, one host sync per 5 steps; L2 flushed before each graph"},
            "acc_val_last": acc_val,
            "e2e": e2e,
            "gpu_launches": int(cbow_launches + walk_launches),
            "gpu_launches_total_process": int(total_launches),
            "clocks": clocks,
            "roofline": main_roofline,
            "roofline_hbm": hbm,
            "parity": parity,
            "strong": strong,
            "algo": args.algo,
            "alt_algo": None if ALT is None else {
                "algo": alt, "value": ALT["value"], "unit": UNIT, "ms_per_step": ALT["step_ms"],
                "train_only_ms": ALT["upd_ms"], "acc_val_last": ALT["acc_val"], "roofline": ALT["roofline"],
                "note": "rank1 = collapsed trainer (s = W_ih.W_ho, c = X^T.dO; SURVEY 8f-3), same results up to fp32 "
                        "reassociation; rows = north_star's embedding-row gather/scatter kernel"},
            "cpu_baseline": cpu,
            "walk": WALK,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def roofline_hbm(args, g2v, cbow, dev, timed, peak, peak_src, K, W):
    """The fused CBOW kernel where it is genuinely HBM-bound: BASELINE configs[4]'s table (200k genes x 512 = 410 MB,
    3x the L2) on synthetic windows (SURVEY 8d: 80 distinct genes uniform, labels Bernoulli(0.5), seed 777)."""
    import torch
    V, D, L = 200_000, 512, 80
    N = 2 * args.hbm_reps * V
    rowptr, gene, label = synthetic_windows(N, V, L, dev)
    n_tr = int(N * 0.8)
    g = torch.Generator(device=dev); g.manual_seed(0)
    s = 1.0 / np.sqrt(D)
    W0 = (torch.randn(V, D, device=dev, generator=g) * s).clamp_(-2 * s, 2 * s)
    Wo0 = (torch.randn(D, device=dev, generator=g) * s).clamp_(-2 * s, 2 * s)
    tr = torch.randperm(N, device=dev, generator=g)[:n_tr].to(torch.int32)
    alg = n_tr * (L * (8 * D + 4) + 5)
    out = {}
    for kind in ("single_pass", "slabs"):
        if kind == "single_pass":
            os.environ["G2V_CBOW_SLABS"] = "1"
        else:
            os.environ.pop("G2V_CBOW_SLABS", None)
        m = g2v.CbowModel(rowptr, gene, label, V, D, W0, Wo0, lr=0.005)
        m.prepare_slabs(tr)
        fn = lambda: m.fwdbwd(tr, n_tr)
        timed(fn, max(W, 3))
        t, _ = timed(fn, max(K, 5))
        ms = float(np.mean(t))
        out[kind] = {"ms": ms, "achieved": alg / (ms * 1e-3) / 1e9, "n_slabs": getattr(m, "_n_slabs", 1)}
        del m
        torch.cuda.empty_cache()
    os.environ.pop("G2V_CBOW_SLABS", None)
    sp, sl = out["single_pass"], out["slabs"]
    return {"kernel": "cbow_rows_kernel<4,true> (fused gather/sum/logit/BCE/scatter-add, ONE launch per step)",
            "bound": "hbm", "achieved": sp["achieved"], "peak": peak, "unit": "GB/s", "frac": sp["achieved"] / peak,
            "kernel_ms": sp["ms"], "algorithmic_bytes_per_launch": alg, "peak_source": peak_src,
            "traffic": traffic_lookup("cbow_rows_fwdbwd", "stress200k", need_reps=args.hbm_reps),
            "config": {"workload": "CBOW only: %d synthetic windows of %d distinct genes (seed 777), %d of them training, "
                                   "V = %d, hidden %d: W_ih and the gradient are 410 MB each (L2: 126 MB)" % (N, L, n_tr, V, D),
                       "l2": "256 MiB flush write before every timed launch", "steps": max(K, 5), "warmup": max(W, 3)},
            "note": "every gathered row and every red.global.add into the gradient misses the L2 in this form: ncu of this "
                    "command shows DRAM traffic 1.30x the algorithmic bytes (the reduction is a DRAM read-modify-write)",
            "shipped": {"kernel": "cbow_slab_fwd_kernel x %d + cbow_slab_bwd_kernel x %d (gene slabs, csrc/g2v_cbow_slab.cu): "
                                  "what train_cbow runs for tables larger than the L2"
                                  % ((sl["n_slabs"] + 1) // 2, sl["n_slabs"]),
                        "bound": "l2 (forward: L2 reads; backward: L2 atomic units, ncu lts 61 % / l1tex 87 %)",
                        "ms": sl["ms"], "achieved": sl["achieved"], "unit": "GB/s", "frac_of_hbm_peak": sl["achieved"] / peak,
                        "speedup_vs_single_pass": sp["ms"] / sl["ms"],
                        "traffic": traffic_lookup("cbow_slab_step", "stress200k", need_reps=args.hbm_reps),
                        "note": "same algorithmic bytes in less time: rows are served by the L2 after their first touch in a "
                                "slab pass, so the algorithmic rate exceeds the HBM peak while DRAM traffic falls to ~0.15x the "
                                "algorithmic bytes (profiles/r2)"}}


def parity_block(g2v, dist, rank, world, dev, gs, V, L):
    """N-GPU == 1-GPU, computed in the run (outside every timed region).  The oracle is used here only as the
    checker of a 2000-walker sample, exactly as tests/ use it."""
    import torch
    out = {}
    # (a) walks: every rank runs its shard rank::world of walkers 0..1999 of group 0; rank 0 re-assembles
    n_s = 2000
    rp, col, w = gs[0]
    gr = g2v.WalkGraph(rp, col, weights=w)
    nodes, lens = g2v.generate_paths(gr, L, 1, seed=12345, group=0, walker_begin=rank, walker_end=n_s, walker_stride=world)
    per = (n_s + world - 1) // world
    pad = torch.full((per, L), -2, dtype=torch.int32, device=dev); pad[:nodes.shape[0]] = nodes
    padl = torch.full((per,), -2, dtype=torch.int32, device=dev); padl[:lens.shape[0]] = lens
    parts = [torch.empty_like(pad) for _ in range(world)]; partl = [torch.empty_like(padl) for _ in range(world)]
    dist.all_gather(parts, pad); dist.all_gather(partl, padl)
    if rank == 0:
        full = np.full((n_s, L), -2, np.int32); fl = np.full(n_s, -2, np.int32)
        for r in range(world):
            k = len(range(r, n_s, world))
            full[r::world] = parts[r][:k].cpu().numpy(); fl[r::world] = partl[r][:k].cpu().numpy()
        one_n, one_l = g2v.generate_paths(gr, L, 1, seed=12345, group=0, walker_begin=0, walker_end=n_s)
        same_1gpu = bool((one_n.cpu().numpy() == full).all() and (one_l.cpu().numpy() == fl).all())
        try:
            import oracle
            want, wl = oracle.walks(rp, col, oracle.quantise_weights(w), L, 12345, 0, 0, n_s)
            same_oracle = bool((want == full).all() and (wl == fl).all())
        except Exception as exc:                                   # no gcc on the box: the GPU comparison stands
            same_oracle = "oracle unavailable: %r" % (exc,)
        out.update(walk_sample_walkers=n_s, walk_equals_one_gpu=same_1gpu, walk_bit_exact=same_oracle)
    # (b) gradient: 4096 synthetic windows, rank r takes windows r::world, all-reduce, vs all of them on rank 0
    D, nb = 128, 4096
    rowptr, gene, label = synthetic_windows(nb, V, min(L, 80), dev, seed=4242)
    from g2vec_b200 import cbow
    W0, Wo0 = cbow.init_weights(V, D, 7)
    m = g2v.CbowModel(rowptr, gene, label, V, D, W0, Wo0)
    mine = torch.arange(rank, nb, world, dtype=torch.int32, device=dev)
    m.fwdbwd(mine, nb)
    for g in m.grad_tensors():
        dist.all_reduce(g)
    if rank == 0:
        ref = g2v.CbowModel(rowptr, gene, label, V, D, W0, Wo0)
        ref.fwdbwd(torch.arange(nb, dtype=torch.int32, device=dev), nb)
        torch.cuda.synchronize()
        err = float((m.g_flat - ref.g_flat).abs().max() / ref.g_flat.abs().max())
        out.update(grad_batch_windows=nb, grad_rel_err=err, grad_collective="one all_reduce over [g_ih | g_ho] (%d floats)"
                   % m.g_flat.numel())
    # (c) the fused exchange + optimizer kernel (g2v_cbow_update_nvl): one Adam step of the same batch sharded over
    #     the ranks vs the same step on rank 0 alone
    mn = g2v.CbowModel(rowptr, gene, label, V, D, W0, Wo0, nvl_group=dist.group.WORLD)
    if mn.nvl:                                                     # (NCCL-only runs have nothing to check here)
        mn.fwdbwd(mine, nb)
        mn.update()
        torch.cuda.synchronize()
        if rank == 0:
            ref.update()
            torch.cuda.synchronize()
            out.update(nvl_exchange=mn.exchange(),
                       nvl_update_rel_err=float((mn.w_flat - ref.w_flat).abs().max() / ref.w_flat.abs().max()))
    torch.cuda.synchronize()
    return out if rank == 0 else None


# =============================================================================== CPU side
def reference_module():
    """The UNMODIFIED reference script (oracle/_ref/G2Vec.py, or /root/reference in the build container) on the
    TF1 shim; None if it was not staged."""
    try:
        from oracle import ref_import
        return ref_import.load() if ref_import.available() else None
    except Exception:
        return None


def _cpu_windows(gs, V, L, n_windows):
    """Windows for the CPU arm, made by the oracle's walker (no GPU on this path)."""
    import oracle
    from oracle import legacy
    per = max(1, n_windows // 2)
    sets = []
    for g, (rp, col, w) in enumerate(gs):
        nodes, lens = oracle.walks(rp, col, oracle.quantise_weights(w), L, 12345, g, 0, min(per, 10 * V))
        sets.append(oracle.path_set(nodes, lens))
    rows = legacy.integrate_pathSet(sets)
    return legacy.windows_from_rows(rows)


class CountingAdjacency:
    """adjMat for the reference's generate_pathSet: `adjMat[node]` returns the dense float32 row (built on demand
    from the CSR when the [V, V] matrix would not fit), counts the calls -- one per node visit, G2Vec.py:332-334 --
    and raises TimeUp once the time budget is spent, so the unmodified function can be timed on a bounded sample."""

    class TimeUp(Exception):
        pass

    def __init__(self, rp, col, w, budget_s):
        from oracle import legacy
        V = len(rp) - 1
        self.shape = (V, V)
        self.dense = legacy.dense_from_csr(rp, col, w) if V * V * 4 <= (2 << 30) else None
        self.rp, self.col, self.w = rp, col, w
        self.visits, self.t_end, self.t0 = 0, None, None
        self.budget = budget_s

    def __getitem__(self, i):
        now = time.perf_counter()
        if self.t0 is None:
            self.t0, self.t_end = now, now + self.budget
        elif now > self.t_end:
            raise CountingAdjacency.TimeUp()
        self.visits += 1
        if self.dense is not None:
            return self.dense[i]
        row = np.zeros(self.shape[0], dtype=np.float32)
        row[self.col[self.rp[i]:self.rp[i + 1]]] = self.w[self.rp[i]:self.rp[i + 1]]
        return row


_WALK_JOB = None


def _walk_worker(seed):
    ref, rp, col, w, L, budget = _WALK_JOB
    A = CountingAdjacency(rp, col, w, budget)
    np.random.seed(seed)
    try:
        if ref is not None:
            ref.generate_pathSet(A, L, 1000)               # the reference's own function, interrupted by the budget
        else:
            from oracle import legacy
            legacy.generate_pathSet_dense(A, L, 1000, np.random.RandomState(seed))
    except CountingAdjacency.TimeUp:
        pass
    return A.visits, time.perf_counter() - A.t0


def cpu_walk_rate(ref, gs, L, budget_s, procs):
    """The reference's walk (G2Vec.py:324-352) for `budget_s` seconds per process; `procs` processes, each running the
    function on the same graph with its own np.random seed (1 = how the reference runs)."""
    global _WALK_JOB
    rp, col, w = gs[0]
    _WALK_JOB = (ref, rp, col, w, L, budget_s)
    if procs <= 1:
        res = [_walk_worker(0)]
    else:
        import multiprocessing as mp
        with mp.get_context("fork").Pool(procs) as pool:
            res = pool.map(_walk_worker, list(range(procs)))
    _WALK_JOB = None
    visits = sum(v for v, _ in res)
    dt = max(t for _, t in res)
    return visits / dt, visits, dt


def cpu_cbow_rate(ref, rowptr, gene, label, V, D, n_sample, threads):
    """Windows/s of the reference's step 4 on a sample of the workload's windows.  With the reference staged: the
    UNMODIFIED compute_genetovec (G2Vec.py:217-286; dense int32 pathList in, its own loop until its early stop) on
    oracle/tf1_shim.py, timed from its first optimizer run to its last accuracy evaluation; else the dense port."""
    import torch
    torch.set_num_threads(threads)
    N = len(rowptr) - 1
    idx = np.random.RandomState(0).permutation(N)[:min(N, n_sample)]
    if ref is not None:
        from oracle import tf1_shim
        import contextlib
        import io
        P = np.zeros((len(idx), V + 1), dtype=np.int32)
        for r, n in enumerate(idx):
            P[r, gene[rowptr[n]:rowptr[n + 1]]] = 1
        P[:, -1] = label[idx]
        best = None
        for rep in range(3):                                   # best of 3: the host cores are shared
            tf1_shim.reset(); tf1_shim.seed_initialisers(rep); np.random.seed(rep)
            with contextlib.redirect_stdout(io.StringIO()):
                ref.compute_genetovec(P.copy(), V, D, 0.005)
            tr_ = tf1_shim.trace()
            t_train = [e[2] for e in tr_ if e[0] == "train"]
            t_eval = [e[2] for e in tr_ if e[0] == "eval"]
            steps = len(t_train)
            # the first optimizer run starts one step before its timestamp: extrapolate from the later steps
            dt = (t_eval[-1] - t_train[0]) * steps / max(steps - 1 + 2.0 / 3.0, 1e-9) if steps > 1 else None
            if dt is None:
                continue
            rate = int(len(idx) * 0.8) * steps / dt
            if best is None or rate > best[0]:
                best = (rate, steps, dt)
        n_tr = int(len(idx) * 0.8)
        if best is not None:
            return best[0], n_tr, len(idx) - n_tr, "reference", ("unmodified compute_genetovec (G2Vec.py:217-286, TF 1.x ops on "
                "oracle/tf1_shim.py, torch-CPU): %d training + %d validation windows (dense int32 pathList [%d, %d]), "
                "its own loop ran %d steps to its early stop in %.1f s, best of 3"
                % (n_tr, len(idx) - n_tr, len(idx), V + 1, best[1], best[2]))
    from oracle import dense_cbow
    pivot = int(len(idx) * 0.8)
    tr, va = idx[:pivot], idx[pivot:]
    Xtr, ytr = dense_cbow.densify(rowptr, gene, label, tr, V)
    Xva, yva = dense_cbow.densify(rowptr, gene, label, va, V)
    rs = np.random.RandomState(0)
    W0 = (np.clip(rs.randn(V, D), -2, 2) / np.sqrt(D)).astype(np.float32)
    Wo0 = (np.clip(rs.randn(D), -2, 2) / np.sqrt(D)).astype(np.float32)
    model = dense_cbow.DenseCbow(W0, Wo0, 0.005)
    model.epoch(Xtr, ytr, Xva, yva)
    t0 = time.perf_counter(); n = 5
    for _ in range(n):
        model.epoch(Xtr, ytr, Xva, yva)
    dt = (time.perf_counter() - t0) / n
    return len(tr) / dt, len(tr), len(va), "port", ("dense port of the reference graph (oracle/dense_cbow.py, torch-CPU matmul): "
                                                   "%d training + %d validation windows, 5 epochs" % (len(tr), len(va)))


def cpu_baseline(args, gs, V, D, L, rowptr, gene, label):
    import torch
    ref = reference_module()
    cores = os.cpu_count() or 1
    rate, n_tr, n_va, kind, sample = cpu_cbow_rate(ref, rowptr, gene, label, V, D, args.cpu_sample_windows, cores)
    cpu = {"value": rate, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind, "sample": sample}
    wrate, visits, wdt = cpu_walk_rate(ref, gs, L, args.cpu_walk_seconds, 1)
    walk_cpu = {"value": wrate, "unit": "steps/s", "cores": 1, "kind": "reference" if ref is not None else "port",
                "sample": "%d node visits in %.1f s of %s on group 0's dense adjacency, single thread as the reference runs"
                          % (visits, wdt, "the unmodified generate_pathSet (G2Vec.py:324-352)" if ref is not None
                             else "the dense-row port (oracle/legacy.py)")}
    return cpu, walk_cpu


def run_reference(args):
    """The reference's own CPU implementation of the path, timed on this box's host cores: the UNMODIFIED
    G2Vec.py (staged into oracle/_ref by __graft_entry__.build(); its TensorFlow 1.x ops run on oracle/tf1_shim.py
    because TF cannot be installed here) -- compute_genetovec on all host threads for CBOW, generate_pathSet in one
    process per core for the walks.  Falls back to the oracle port (kind "port") only if the script is not staged."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)                               # torchrun exports OMP_NUM_THREADS=1: undo it for this arm
    K, W = args.steps, args.warmup
    ref = reference_module()
    gs, V, D, L, desc = workload(args.workload)
    rowptr, gene, label = _cpu_windows(gs, V, L, args.cpu_sample_windows)
    rate, n_tr, n_va, kind, sample = cpu_cbow_rate(ref, rowptr, gene, label, V, D, args.cpu_sample_windows, cores)
    wrate, visits, wdt = cpu_walk_rate(ref, gs, L, args.cpu_walk_seconds, cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": K,
        "warmup": W, "ms_per_step": n_tr / rate * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic" if args.workload != "ex" else "ex_* graphs (fixture)",
        "config": {"workload": "%s: %s, hidden %d, lenPath %d" % (args.workload, desc, D, L), "sample": sample,
                   "steps_note": "the reference's loop decides its own step count (early stop, G2Vec.py:276); --steps/--warmup "
                                 "do not apply; throughput = training windows x steps it ran / time, best of 3 runs"},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind, "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "walk": {"metric": "random_walk_steps_per_sec", "value": wrate, "unit": "steps/s", "cores": cores,
                 "kind": "reference" if ref is not None else "port",
                 "sample": "%d node visits in %.1f s: %s, %d processes (one per core, own np.random seed each)"
                           % (visits, wdt, "unmodified generate_pathSet (G2Vec.py:324-352)" if ref is not None
                              else "dense-row port of G2Vec.py:324-352", cores)},
    }
    print(json.dumps(line))


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
