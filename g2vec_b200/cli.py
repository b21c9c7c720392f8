"""The G2Vec command line, kept as the drop-in shell around the two B200 hot paths.

Same positionals, options, progress banners and output files as /root/reference/G2Vec.py
(parse_arguments :505-518, main :11-119, writers :127-131,159-165,203-215).  Steps 1, 2, 5, 6, 7 are
plain Python/NumPy/scikit-learn as in the reference; step 3 runs g2vec_b200.walks on the GPU and
step 4 g2vec_b200.cbow.  With ``--post gpu`` steps 5-7 run on the device (g2vec_b200.post) and write the same files;
the functions here stay the reference for them.  Two documented differences: ``--epoch`` is honoured as the cap on optimizer
steps (the reference parses it, :515, and then loops ``range(500)``, :262 -- the default 500 is the
reference behaviour), and ``--seed`` (default 0) makes runs reproducible (the reference is unseeded).
"""
import argparse
import sys
from math import sqrt

import numpy as np


def parse_arguments(argv=None):
    p = argparse.ArgumentParser(
        description="G2Vec (B200-native hot paths): network-based identification of prognostic gene "
                    "signatures. Same interface as mathcom/G2Vec G2Vec.py.")
    p.add_argument('EXPRESSION_FILE', type=str, help="Tab-delimited file for gene expression profiles.")
    p.add_argument('CLINICAL_FILE', type=str, help="Tab-delimited clinical file. LABEL=0: good prognosis, 1: poor.")
    p.add_argument('NETWORK_FILE', type=str, help="Tab-delimited file for the gene interaction network.")
    p.add_argument('RESULT_NAME', type=str, help="Prefix of *_biomarkers.txt, *_lgroups.txt and *_vectors.txt")
    p.add_argument('-p', '--lenPath', type=int, default=80, help='')
    p.add_argument('-r', '--numRepetition', type=int, default=10, help='')
    p.add_argument('-s', '--sizeHiddenlayer', type=int, default=128, help='')
    p.add_argument('-e', '--epoch', type=int, default=500, help='')
    p.add_argument('-l', '--learningRate', type=float, default=0.005, help='')
    p.add_argument('-n', '--numBiomarker', type=int, default=50, help='')
    p.add_argument('--seed', type=int, default=0, help='seed of the walk sampler, the split and the init')
    p.add_argument('--algo', choices=['rows', 'rank1'], default='rows',
                   help="CBOW kernels: 'rows' = embedding-row gather/scatter (default), 'rank1' = collapsed, "
                        "bit-reproducible trainer; same results to fp32 rounding")
    p.add_argument('--post', choices=['host', 'gpu'], default='host',
                   help="steps 5-7 (L-groups, gene scores, vectors file): 'host' = NumPy / scikit-learn (default), "
                        "'gpu' = on the device from the trained vectors (g2vec_b200.post), same files")
    return p.parse_args(argv)


# ----------------------------------------------------------------------------------- step 1: I/O
def _rows(path):
    with open(path) as f:
        return [ln.rstrip().split('\t') for ln in f]


def load_data(path):
    """Expression TSV: header = samples, rows = genes -> expr float32 [samples, genes] (G2Vec.py:478-503)."""
    rows = _rows(path)
    sample = np.array(rows[0][1:])
    gene = np.array([r[0] for r in rows[1:]])
    expr = np.array([r[1:] for r in rows[1:]], dtype=np.float32).T
    return {'sample': sample, 'expr': expr, 'gene': gene}


def load_clinical(path):
    """sample -> int label, header skipped (G2Vec.py:436-453)."""
    return {r[0]: int(r[1]) for r in _rows(path)[1:]}


def load_network(path):
    """Directed edge list [src, dest] and the gene set, header skipped (G2Vec.py:455-476)."""
    edges = _rows(path)[1:]
    genes = set()
    for e in edges:
        genes.add(e[0]); genes.add(e[1])
    return {'edge': edges, 'gene': genes}


# ------------------------------------------------------------------------- step 2: preprocessing
def match_labels(clinical, samples):
    try:
        return np.array([clinical[s] for s in samples])
    except KeyError:
        print('ERROR: There is a mismatched sample between expression data and clinical data. '
              'Please check sample names')
        sys.exit(1)


def restrict(data, network):
    """Sorted common gene list; edges with both ends in it; expression columns (G2Vec.py:393-426)."""
    common = sorted(set(network['gene']) & set(data['gene']))
    cs = set(common)
    edges = [e for e in network['edge'] if e[0] in cs and e[1] in cs]
    pos = {g: i for i, g in enumerate(data['gene'])}
    cols = [pos[g] for g in common]
    data = dict(data, expr=data['expr'][:, cols], gene=np.array(common))
    return data, {'edge': edges, 'gene': cs}


# ------------------------------------------------------------------------------ step 5: L-groups
def find_lgroups(mat, gene_names, geneFreq):
    """KMeans(3, random_state=0) on the vectors; largest cluster -> 2 (other); of the remaining two
    clusters the reference compares good/poor gene-frequency votes (G2Vec.py:167-200).  In the reference
    ``freqIdx`` is a Python list, so ``freqIdx==0`` is the scalar False and both votes are always 0
    (:172,186-187): the outcome is therefore always good = second remaining cluster, poor = first.  That
    behaviour is reproduced here so the output files match."""
    from sklearn.cluster import KMeans
    return lgroups_from_clusters(KMeans(n_clusters=3, random_state=0).fit(mat).labels_)


def lgroups_from_clusters(km):
    """Cluster ids 0..2 per gene -> L-groups, as find_lgroups numbers them (shared by --post host and gpu)."""
    km = np.asarray(km)
    sizes = [int(np.count_nonzero(km == k)) for k in range(3)]
    largest = 0
    for k in (1, 2):
        if sizes[k] > sizes[largest]:
            largest = k
    rest = [k for k in (0, 1, 2) if k != largest]
    poor_c, good_c = rest[0], rest[1]
    out = np.zeros(km.shape[0], dtype=np.int32)
    out[km == good_c] = 0
    out[km == poor_c] = 1
    out[km == largest] = 2
    return out


# ------------------------------------------------------------------------------- step 6: scoring
def minmax(x, lo=0., hi=1.):
    return (hi - lo) / (x.max() - x.min()) * (x - x.min()) + lo


def tscore(a, b):
    """abs pooled-variance t statistic between two samples (G2Vec.py:138-149)."""
    na, nb = len(a), len(b)
    sa, sb = a.std(ddof=1), b.std(ddof=1)
    d1 = sqrt(((float(na) - 1.) * sa * sa + (float(nb) - 1.) * sb * sb) / float(na + nb - 2))
    d2 = sqrt(1. / float(na) + 1. / float(nb))
    if d1 > 0. and d2 > 0.:
        return abs((a.mean() - b.mean()) / d1 / d2)
    return 0.


def tscores(expr, label):
    out = np.zeros(expr.shape[1], dtype=np.float32)
    g, p = label == 0, label == 1
    for i in range(expr.shape[1]):
        out[i] = tscore(expr[g, i], expr[p, i])
    return out


# ------------------------------------------------------------------------------- step 7: writers
def write_biomarkers(prefix, genes):
    with open(prefix + "_biomarkers.txt", 'w') as f:
        f.write("GeneSymbol\n")
        f.writelines('%s\n' % g for g in genes)


def write_lgroups(prefix, lgroup, genes):
    with open(prefix + "_lgroups.txt", 'w') as f:
        f.write('GeneSymbol\tLgroup(0:good,1:poor,2:other)\n')
        f.writelines('%s\t%d\n' % (g, k) for g, k in zip(genes, lgroup))


def write_vectors(prefix, genes, mat):
    with open(prefix + "_vectors.txt", 'w') as f:
        f.write('GeneSymbol' + ''.join('\tV%d' % i for i in range(mat.shape[1])) + '\n')
        for g, vec in zip(genes, mat):
            f.write(g + ''.join("\t%.6f" % v for v in vec) + "\n")


# ------------------------------------------------------------------------------------------ main
def _distributed():
    """One process per GPU under torchrun (RANK / WORLD_SIZE / LOCAL_RANK in the environment): NCCL group,
    device = LOCAL_RANK.  Returns (rank, world, dist or None)."""
    import os
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world <= 1:
        return 0, 1, None
    import torch
    import torch.distributed as dist
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return dist.get_rank(), world, dist


def main(argv=None):
    args = parse_arguments(argv)
    rank, world, dist = _distributed()
    import builtins
    print = builtins.print if rank == 0 else (lambda *a, **k: None)   # noqa: A001  every rank computes, rank 0 talks
    print('>>> 0. Arguments')
    print(args)

    print('>>> 1. Load data')
    data = load_data(args.EXPRESSION_FILE)
    clinical = load_clinical(args.CLINICAL_FILE)
    network = load_network(args.NETWORK_FILE)

    print('>>> 2. Preprocess data')
    data['label'] = match_labels(clinical, data['sample'])
    data, network = restrict(data, network)
    n_samples, n_genes = data['expr'].shape
    print('    n_samples: %d' % n_samples)
    print('    n_genes  : %d\t(common genes in both EXPRESSION and NETWORK)' % n_genes)
    print('    n_edges  : %d\t(edges with the common genes)' % len(network['edge']))

    print('>>> 3. Generate random paths from each group')
    print('    *** most time consuming step ***')
    from . import graph, paths, walks, cbow           # needs the GPU from here on
    idx = {g: i for i, g in enumerate(data['gene'])}
    src = np.fromiter((idx[e[0]] for e in network['edge']), dtype=np.int32, count=len(network['edge']))
    dst = np.fromiter((idx[e[1]] for e in network['edge']), dtype=np.int32, count=len(network['edge']))
    import torch
    n_total = n_genes * args.numRepetition                     # walkers per group: w = repetition * n_genes + start gene
    L = args.lenPath
    dev = torch.device("cuda", torch.cuda.current_device())
    rows = torch.empty((2 * n_total, L), dtype=torch.int32, device=dev)
    lens = torch.empty(2 * n_total, dtype=torch.int32, device=dev)
    key = torch.empty(2 * n_total, dtype=torch.int64, device=dev)
    for i, _group in enumerate(['g', 'p']):
        rp, col, w = graph.group_csr_gpu(data['expr'], data['label'], i, src, dst)
        wg = walks.WalkGraph(rp, col, weights=w)
        sl = slice(i * n_total, (i + 1) * n_total)
        if dist is None:
            # tuple(sorted(path)) is fused into the sampler: sorted rows + their 64-bit keys come back
            walks.generate_paths(wg, L, args.numRepetition, seed=args.seed, group=i, canonical=True,
                                 out=(rows[sl], lens[sl], key[sl]))
        else:
            # walkers rank, rank+world, ...: no collective during the walk (counter-based RNG); one all_gather after,
            # rows put back at their walker index so that every rank holds the 1-GPU arrays (same window order,
            # hence the same --seed split, whatever the number of GPUs)
            r_, l_, k_ = walks.generate_paths(wg, L, args.numRepetition, seed=args.seed, group=i, canonical=True,
                                              walker_begin=rank, walker_stride=world)
            rows[sl], lens[sl], key[sl] = paths.gather_walker_shards(dist, world, n_total, r_, l_, k_)
    group = torch.cat([torch.zeros(n_total, dtype=torch.uint8, device=dev), torch.ones(n_total, dtype=torch.uint8, device=dev)])
    w_rowptr, w_gene, w_label, code = paths.build_windows(rows, lens, key, group, n_genes)
    del rows, lens, key, group
    geneFreq = paths.gene_freq_dict(code, data['gene'])
    print("    n_paths : %d" % int(w_label.shape[0]))
    print("    n_genes : %d\t(genes in good or poor random paths)" % len(geneFreq))

    print(">>> 4. Compute distributed representations using modified CBOW")
    mat = cbow.train_cbow(w_rowptr, w_gene, w_label, n_genes, args.sizeHiddenlayer, args.learningRate,
                          max_epoch=args.epoch, seed=args.seed, log=print, algo=args.algo,   # print is silent off rank 0
                          device_out=args.post == 'gpu')
    genes = data['gene']
    if rank != 0:
        dist.barrier()
        dist.destroy_process_group()
        return
    if args.post == 'gpu':
        _post_gpu(args, data, mat, genes, print)
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return

    print('>>> 5. Find L-groups')
    lgroup = find_lgroups(mat, genes, geneFreq)

    print(">>> 6. Select biomarkers with gene scores")
    biomarkers = []
    for i in (0, 1):
        sel = lgroup == i
        d = minmax(np.linalg.norm(mat[sel], axis=1))
        t = minmax(tscores(data['expr'][:, sel], data['label']))
        score = 0.5 * (d + t)
        ranked = sorted(zip(genes[sel], score), key=lambda gs: gs[1], reverse=True)
        biomarkers += sorted(g for g, _ in ranked[:args.numBiomarker])
    biomarkers = sorted(biomarkers)

    print(">>> 7. Save results")
    write_biomarkers(args.RESULT_NAME, biomarkers)
    print('    %s_biomarkers.txt' % args.RESULT_NAME)
    write_lgroups(args.RESULT_NAME, lgroup, genes)
    print('    %s_lgroups.txt' % args.RESULT_NAME)
    write_vectors(args.RESULT_NAME, genes, mat)
    print('    %s_vectors.txt' % args.RESULT_NAME)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def _post_gpu(args, data, mat, genes, print):
    """Steps 5-7 with --post gpu: mat is the device tensor of the vectors; same banners and files as the host."""
    import torch
    from . import post
    print('>>> 5. Find L-groups')
    lgroup, _ = post.find_lgroups(mat)

    print(">>> 6. Select biomarkers with gene scores")
    expr = torch.from_numpy(np.ascontiguousarray(data['expr'], dtype=np.float32)).to(mat.device)
    biomarkers = post.select_biomarkers(mat, expr, data['label'], lgroup, genes, args.numBiomarker)

    print(">>> 7. Save results")
    write_biomarkers(args.RESULT_NAME, biomarkers)
    print('    %s_biomarkers.txt' % args.RESULT_NAME)
    write_lgroups(args.RESULT_NAME, lgroup, genes)
    print('    %s_lgroups.txt' % args.RESULT_NAME)
    post.write_vectors(args.RESULT_NAME, genes, mat)
    print('    %s_vectors.txt' % args.RESULT_NAME)


if __name__ == "__main__":
    main()
