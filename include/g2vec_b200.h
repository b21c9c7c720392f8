/*
 * g2vec_b200.h -- C ABI of libg2vec_b200.so: the two G2Vec hot paths as sm_100a CUDA.
 *
 * The reference (mathcom/G2Vec) has no FFI or plugin interface: its boundary for these
 * paths is two plain Python calls in main(),
 *     pathSet = generate_pathSet(adjMat, args.lenPath, args.numRepetition)     G2Vec.py:62
 *     genetovec['mat'] = compute_genetovec(pathList, n_genes, hidden, lr)      G2Vec.py:74
 * The entry points below are what a binding for those two call sites needs; the ctypes
 * binding that ships is g2vec_b200/_capi.py, and INTEGRATION.md shows the stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no exceptions, no torch types.
 *   - every function returns 0 on success, non-zero on failure; g2v_last_error() then
 *     returns a thread-local message.
 *   - `stream` is a cudaStream_t passed as void*; device entry points are asynchronous on
 *     it and never synchronise.  Buffers are owned by the caller.
 *   - `_host` entry points take HOST pointers, do their own device allocation and
 *     host<->device copies, and return after the result is back in host memory.
 *   - there is no CPU fallback: without a usable sm_100 device the calls fail.
 */
#ifndef G2VEC_B200_H
#define G2VEC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define G2V_ABI_VERSION 2

/* optimizer codes for g2v_cbow_update */
#define G2V_OPT_ADAM_TF1 0 /* tf.train.AdamOptimizer, G2Vec.py:246 (parity default) */
#define G2V_OPT_SGD 1      /* var -= lr * g (north_star variant) */

/* context reduction for the CBOW forward */
#define G2V_REDUCE_SUM 0  /* H = X.W_ih, G2Vec.py:239 (parity default) */
#define G2V_REDUCE_MEAN 1 /* H = X.W_ih / len(window) */

int g2v_abi_version(void);
const char *g2v_last_error(void);

/* Device facts (current device): SM count, compute capability, L2 bytes, and the number of
 * kernels this library has launched since load (bench.py's gpu_launches). */
int g2v_device_info(int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor, int64_t *l2_bytes);
int64_t g2v_launch_count(void);

/* ---------------------------------------------------------------------------------------
 * HOT PATH 1 -- walk sampler.  Replaces generate_pathSet / generate_randomPath,
 * G2Vec.py:324-352, for the walkers  w = walker_begin + i*walker_stride < walker_end,
 * w = rep*V + src  (rep = G2Vec.py:348 `step`, src = :349).
 *
 *   rowptr [V+1], col [E] (ascending inside a row = dense row order), qw [E]: CSR of the
 *     group's directed adjacency (rows = out-edges, G2Vec.py:390) with weights quantised to
 *     integers, 1 <= qw <= 2^24  (q = rint(|PCC| * 2^16)).  g2v_walk_prepare (and so g2v_walk_host) rejects a
 *     weight above 2^24 with an error; g2v_walk_launch does not check it.
 *   L: --lenPath, the maximum number of NODES of a path (G2Vec.py:331).  1 <= L <= 4096, and the
 *     per-CTA path + visited-set buffers must fit shared memory: always true for L <= 1365, and
 *     for any L <= 4096 while V <= ~90k (bitmap visited set); otherwise the call fails with a message.
 *   seed/group: Philox4x32-10 key and the high bits of the walker's subsequence
 *     (subsequence = group*2^40 + w, 64-bit draw s = words 2s,2s+1), so that any
 *     (walker, step) is addressable independently: results do not depend on sharding.
 *   out_nodes [n*L]: visit order of walker i in row i, padded with -1  (the reference
 *     sorts afterwards, G2Vec.py:345).  out_len [n]: nodes visited.  n = number of walkers.
 *   workspace: >= g2v_walk_workspace_bytes() bytes of device scratch (zeroed by the call).
 * ------------------------------------------------------------------------------------- */
size_t g2v_walk_workspace_bytes(void);
int g2v_walk_launch(const int32_t *rowptr, const int32_t *col, const uint32_t *qw, int32_t V,
                    int64_t E, int32_t L, uint64_t seed, uint32_t group, int64_t walker_begin,
                    int64_t walker_end, int64_t walker_stride, int32_t *out_nodes,
                    int32_t *out_len, void *workspace, void *stream);

/* Packed graph layouts (built once per graph; the graph is static across all repetitions, G2Vec.py:348-351).
 * g2v_walk_prepare turns the CSR arrays (device pointers) into
 *   rows  [V]  int32 pairs {begin, end} of each node's out-edges                (g2v_walk_packed_bytes: rows_bytes)
 *   edges      layout 1: uint32 pairs {col, qw}, rows starting at even indices: one 16-byte load brings two
 *              neighbours per lane;
 *              layout 2: uint32 col | (qw - 32768) << 16 [E] -- chosen when V <= 65535 and every
 *              32768 <= qw <= 65536 (weights |PCC| in [0.5, 1], G2Vec.py:389): one 8-byte load brings two
 *              neighbours per lane                                              (edges_bytes covers both)
 * and returns the layout chosen through *layout_out (a host int; the call synchronises the stream once).
 * g2v_walk_launch_packed is g2v_walk_launch on the packed graph.  With out_key != NULL it also performs
 * `path = tuple(sorted(path))` (G2Vec.py:345) in the same kernel: out_nodes rows are then SORTED ascending and
 * padded with INT32_MAX, and out_key [n] receives the 64-bit row key g2v_paths_canonicalise would compute. */
int g2v_walk_packed_bytes(int32_t V, int64_t E, size_t *rows_bytes, size_t *edges_bytes);
int g2v_walk_prepare(const int32_t *rowptr, const int32_t *col, const uint32_t *qw, int32_t V, int64_t E,
                     void *rows, void *edges, int32_t *layout_out, void *workspace, void *stream);
int g2v_walk_launch_packed(const void *rows, const void *edges, int32_t layout, int32_t V, int64_t E, int32_t L,
                           uint64_t seed, uint32_t group, int64_t walker_begin, int64_t walker_end,
                           int64_t walker_stride, int32_t *out_nodes, int32_t *out_len, int64_t *out_key,
                           void *workspace, void *stream);

/* Same, HOST pointers in and out (one device slab: copies in, packs, launches, copies back, frees). */
int g2v_walk_host(const int32_t *rowptr, const int32_t *col, const uint32_t *qw, int32_t V,
                  int64_t E, int32_t L, uint64_t seed, uint32_t group, int64_t walker_begin,
                  int64_t walker_end, int64_t walker_stride, int32_t *out_nodes,
                  int32_t *out_len);

/* ---------------------------------------------------------------------------------------
 * HOT PATH 2 -- modified CBOW.  Replaces the TF1 graph of compute_genetovec,
 * G2Vec.py:231-251, one optimizer step at a time; the epoch loop and the early stop
 * (G2Vec.py:262-283) stay with the host (g2vec_b200/cbow.py).
 *
 * Windows (the rows of pathList, G2Vec.py:316-320) are CSR: rowptr [N+1], gene [nnz],
 * label [N] (0 good / 1 poor).  `win` (nullable) is a list of window indices (the shuffled
 * 80/20 split of G2Vec.py:219-222); NULL means windows win_begin..win_begin+n_win-1.
 * W_ih [V*D] row-major are the gene vectors; W_ho [D].
 *
 * g2v_cbow_fwdbwd: for every listed window, gather the rows of its genes, reduce (sum),
 *   logit o = h.W_ho, dO = (sigmoid(o) - y) * inv_n_total, then ADD  dO*W_ho into
 *   g_ih[gene,:] for each gene of the window and h*dO into g_ho.  Adds the BCE loss sum
 *   into *loss_sum (double) and the count of (o > 0) == y into *n_correct.  g_ih, g_ho,
 *   loss_sum, n_correct are ACCUMULATED (device memory; the caller or g2v_cbow_update zeroes).
 * g2v_cbow_update: optimizer epilogue over W_ih and W_ho from g_ih / g_ho (after the
 *   all-reduce when multi-GPU); zeroes g_ih / g_ho for the next step.  t = 1-based step.
 * g2v_cbow_eval: forward only; adds the count of correct predictions into *n_correct.
 * ------------------------------------------------------------------------------------- */
int g2v_cbow_fwdbwd(const int32_t *rowptr, const int32_t *gene, const uint8_t *label,
                    const int32_t *win, int64_t win_begin, int64_t n_win, float inv_n_total,
                    const float *W_ih, const float *W_ho, float *g_ih, float *g_ho,
                    double *loss_sum, int64_t *n_correct, int32_t V, int32_t D, int32_t reduce,
                    void *stream);

int g2v_cbow_update(float *W_ih, float *W_ho, float *m_ih, float *v_ih, float *m_ho, float *v_ho,
                    float *g_ih, float *g_ho, int32_t V, int32_t D, int32_t optimizer, float lr,
                    float beta1, float beta2, float eps, int32_t t, const float *alpha_dev, void *stream);

/* Multi-GPU optimizer epilogue fused with the gradient exchange (one process per GPU, one node): replaces
 * ncclAllReduce(gradient) + g2v_cbow_update.  All buffers are flat [W_ih (V*D) | W_ho (D)] = n floats, the gradient
 * and the parameters in symmetric memory (same size on every rank, peer-mapped): g_ptrs_dev / w_ptrs_dev are DEVICE
 * arrays of `world` pointers (entry r = rank r's buffer as seen from this rank); g_multicast / w_multicast are the
 * NVLS multicast addresses of the same buffers, or both NULL (then peer loads/stores are used).  Rank r reduces the
 * slice r of every rank's gradient (multimem.ld_reduce or peer loads), zeroes it everywhere, applies TF1 Adam / SGD
 * to slice r of its m / v / parameters, and stores the new parameters into every rank's buffer.  The caller must
 * place a cross-GPU barrier before the call (all gradients complete) and after it (all parameters delivered). */
int g2v_cbow_update_nvl(float *const *g_ptrs_dev, float *const *w_ptrs_dev, float *g_multicast, float *w_multicast,
                        float *m_flat, float *v_flat, int64_t n, int32_t rank, int32_t world, int32_t optimizer,
                        float lr, float beta1, float beta2, float eps, int32_t t, const float *alpha_dev, void *stream);

/* Device-resident Adam step state -- TF1 keeps beta1^t / beta2^t as variables (AdamOptimizer's
 * beta1_power / beta2_power, G2Vec.py:246).  state = {beta1^t, beta2^t, alpha_t, unused}, initialised to
 * {1, 1, 0, 0}; g2v_cbow_adam_tick advances it by one step on the device.  Passing the same pointer as
 * `alpha_dev` to g2v_cbow_update / g2v_cbow_r1_update (else NULL: alpha is computed on the host from t)
 * makes every launch of a training step independent of host-side values, so the whole step can be captured
 * once in a CUDA graph and replayed (g2vec_b200/cbow.py). */
int g2v_cbow_adam_tick(float *state, float lr, float beta1, float beta2, void *stream);

int g2v_cbow_eval(const int32_t *rowptr, const int32_t *gene, const uint8_t *label,
                  const int32_t *win, int64_t win_begin, int64_t n_win, const float *W_ih,
                  const float *W_ho, int64_t *n_correct, int32_t V, int32_t D, int32_t reduce,
                  void *stream);

/* ---------------------------------------------------------------------------------------
 * Device-side control of the training loop (SURVEY.md 8f-4; G2Vec.py:262-283), so that several iterations of
 * the reference's loop can be enqueued -- or replayed as ONE CUDA graph -- without a host decision in between.
 *   ctl  [8] int64 in device memory: {stopped, step, stop_step, before_val, max_steps, early_stop, -, -}
 *        g2v_cbow_loop_init sets {0, 0, -1, -1, max_steps, early_stop}.
 *   g2v_cbow_loop_attach(ctl): from now on every CBOW kernel launched by THIS host thread first reads
 *        ctl.stopped and returns at once if it is set (attach(NULL) detaches).
 *   g2v_cbow_loop_begin: unless stopped, copies W_ih [n floats] into `snapshot` (nullable) -- the weights the
 *        reference would return if this step's validation accuracy drops (:283,:286) -- and zeroes acc[0..3].
 *   g2v_cbow_loop_decide: unless stopped, stores acc[0..3] (loss-sum bits, pre-update train correct, validation
 *        correct, train correct) in hist[step*4 ..] (acc == NULL: they are there already, see below), applies `if acc_val < before_acc_val: break` (:276) on the
 *        validation count, else before_val = count (:280); stops after max_steps; step += 1.
 * The host reads ctl / hist whenever it wants to print (every 5th step, :269) instead of after every step.
 * ------------------------------------------------------------------------------------- */
int g2v_cbow_loop_init(int64_t *ctl, int64_t max_steps, int32_t early_stop, void *stream);
int g2v_cbow_loop_attach(const int64_t *ctl);
int g2v_cbow_loop_begin(const int64_t *ctl, int64_t *acc, const float *W_ih, float *snapshot, int64_t n, void *stream);
int g2v_cbow_loop_decide(int64_t *ctl, const int64_t *acc, int64_t *hist, void *stream);
/* Multi-GPU, hist in symmetric memory (zero-initialised, same size on every rank): add this rank's acc[1..3] into
 * hist[step][1..3] of every rank (multimem.red through hist_multicast, or system-scope atomics on hist_ptrs_dev);
 * after a cross-GPU barrier call g2v_cbow_loop_decide with acc == NULL, which then decides on the summed counters
 * already in hist[step].  Replaces the all_reduce of the counters. */
int g2v_cbow_loop_counters_nvl(const int64_t *ctl, const int64_t *acc, int64_t *const *hist_ptrs_dev,
                               int64_t *hist_multicast, int32_t world, void *stream);

/* ---------------------------------------------------------------------------------------
 * HOT PATH 2 for tables larger than the L2 (csrc/g2v_cbow_slab.cu): the same step as g2v_cbow_fwdbwd /
 * g2v_cbow_eval, processed gene slab by gene slab so that the gathered rows and the gradient rows stay
 * L2-resident.  Needs windows whose gene lists are strictly ascending (tuple(sorted(path)), G2Vec.py:345).
 *
 * g2v_cbow_slab_plan: number of slabs for a [V, D] table on the current device (1 = table + gradient fit
 *   the L2 together, or D is not 128/256/512: use g2v_cbow_fwdbwd).
 * g2v_cbow_slab_workspace_bytes / g2v_cbow_slab_setup: per window list (win/win_begin/n_win as in
 *   g2v_cbow_fwdbwd; the list is static across steps, G2Vec.py:262-264), records where each window's sorted gene
 *   list crosses the slab boundaries.  Synchronises the stream once; fails on an unsorted window.
 * g2v_cbow_fwdbwd_slabs / g2v_cbow_eval_slabs: same accumulation semantics as g2v_cbow_fwdbwd / g2v_cbow_eval,
 *   for the list the workspace was set up with.
 * ------------------------------------------------------------------------------------- */
int g2v_cbow_slab_plan(int32_t V, int32_t D, int32_t *n_slabs);
size_t g2v_cbow_slab_workspace_bytes(int64_t n_win, int32_t D, int32_t n_slabs);
int g2v_cbow_slab_setup(const int32_t *rowptr, const int32_t *gene, const int32_t *win, int64_t win_begin,
                        int64_t n_win, int32_t V, int32_t n_slabs, void *workspace, void *stream);
int g2v_cbow_fwdbwd_slabs(const int32_t *gene, const uint8_t *label, const int32_t *win, int64_t win_begin,
                          int64_t n_win, float inv_n_total, const float *W_ih, const float *W_ho, float *g_ih,
                          float *g_ho, double *loss_sum, int64_t *n_correct, int32_t V, int32_t D, int32_t reduce,
                          int32_t n_slabs, void *workspace, void *stream);
int g2v_cbow_eval_slabs(const int32_t *gene, const uint8_t *label, const int32_t *win, int64_t win_begin,
                        int64_t n_win, const float *W_ih, const float *W_ho, int64_t *n_correct, int32_t V,
                        int32_t D, int32_t reduce, int32_t n_slabs, void *workspace, void *stream);

/* One full-batch step from HOST buffers: uploads the windows and the parameters/optimizer
 * state, runs fwdbwd + update, downloads the updated parameters/state, the loss sum and the
 * correct count (of the pre-update forward).  m/v may be NULL for SGD. */
int g2v_cbow_step_host(const int32_t *rowptr, const int32_t *gene, const uint8_t *label,
                       int64_t n_win, int64_t nnz, float *W_ih, float *W_ho, float *m_ih,
                       float *v_ih, float *m_ho, float *v_ho, int32_t V, int32_t D,
                       int32_t optimizer, int32_t reduce, float lr, float beta1, float beta2,
                       float eps, int32_t t, double *loss_sum, int64_t *n_correct);

/* ---------------------------------------------------------------------------------------
 * HOT PATH 2, collapsed ("rank-1") form -- SURVEY.md 8f-3.  The reference's model is linear
 * (G2Vec.py:239-240: O = (X.W_ih).W_ho), so with  s = W_ih.W_ho [V]  and  c = X^T.dO [V]
 * the same step is  o = sum_{g in window} s[g];  dW_ih[g,:] = c[g]*W_ho;  dW_ho = W_ih^T.c.
 * Same results up to float32 reassociation; 4-byte scalars per (window, gene) instead of
 * D-wide rows, and a 4*V-byte all-reduce (of c) instead of 4*V*D bytes.
 *
 * g2v_cbow_r1_prepare: s[g] = <W_ih[g,:], W_ho>.
 * g2v_cbow_r1_windows: forward over the listed windows from s; if c != NULL also the backward:
 *   c[gene] += dO for every gene of the window, loss sum and pre-update correct count
 *   accumulated as in g2v_cbow_fwdbwd.  c == NULL: accuracy pass only (g2v_cbow_eval).
 * g2v_cbow_r1_update: optimizer epilogue from c (after its all-reduce when multi-GPU): per row
 *   g = c[g]*W_ho and g_ho += c[g]*W_ih[g,:] (old W_ih), TF1 Adam / SGD on W_ih, then on W_ho,
 *   zeroes c, and refreshes s for the updated parameters.  g_ho: scratch of
 *   g2v_cbow_r1_scratch_bytes(D) bytes (per-block partial sums of W_ih^T.c, reduced in a fixed
 *   order: no floating-point atomics anywhere in this call).
 * ------------------------------------------------------------------------------------- */
int g2v_cbow_r1_prepare(const float *W_ih, const float *W_ho, float *s, int32_t V, int32_t D,
                        void *stream);
int g2v_cbow_r1_windows(const int32_t *rowptr, const int32_t *gene, const uint8_t *label,
                        const int32_t *win, int64_t win_begin, int64_t n_win, float inv_n_total,
                        const float *s, float *c, double *loss_sum, int64_t *n_correct, int32_t V,
                        int32_t reduce, void *stream);
/* Deterministic backward: the list's windows x genes incidence is also given transposed (CSC over list
 * positions: cscptr [V+1], csc_pos [nnz] = positions i in 0..n_win-1 of the windows that contain the gene).
 * dO [n_win] is scratch; c[g] += sum of dO over the gene's positions with a fixed reduction order, so
 * the step is bit-reproducible (no floating-point atomics). */
int g2v_cbow_r1_windows_csc(const int32_t *rowptr, const int32_t *gene, const uint8_t *label,
                            const int32_t *win, int64_t n_win, float inv_n_total, const float *s,
                            const int32_t *cscptr, const int32_t *csc_pos, float *dO, float *c,
                            double *loss_sum, int64_t *n_correct, int32_t V, int32_t reduce, void *stream);
size_t g2v_cbow_r1_scratch_bytes(int32_t D);
int g2v_cbow_r1_update(float *W_ih, float *W_ho, float *m_ih, float *v_ih, float *m_ho, float *v_ho,
                       float *c, float *g_ho, float *s, int32_t V, int32_t D, int32_t optimizer,
                       float lr, float beta1, float beta2, float eps, int32_t t, const float *alpha_dev,
                       void *stream);

/* ---------------------------------------------------------------------------------------
 * Upstream of the walks -- edge weighting (SURVEY.md 8f-1).  Replaces construct_adjMat /
 * compute_PCC, G2Vec.py:354-391, for one patient group.
 * g2v_pcc_zscore: expr [S*V] sample-major (rows = the group's samples, G2Vec.py:378) ->
 *   z [V*S] gene-major z-scores (population std; 0 for zero-variance genes, :359,366-367).
 * g2v_pcc_edge_weights: w[e] = |mean_s z[src[e]][s] * z[dst[e]][s]|  (G2Vec.py:362-365,385).
 * The > 0.5 threshold (:389) and the CSR assembly are done by the caller.
 * ------------------------------------------------------------------------------------- */
int g2v_pcc_zscore(const float *expr, int32_t S, int32_t V, float *z, void *stream);
int g2v_pcc_edge_weights(const float *z, int32_t S, int32_t V, const int32_t *src, const int32_t *dst,
                         int64_t E, float *w, void *stream);

/* ---------------------------------------------------------------------------------------
 * Between the two hot paths (SURVEY.md 8f-2): `tuple(sorted(path))` into a set (G2Vec.py:345,351) and
 * the removal of paths common to both groups (G2Vec.py:313).
 * g2v_paths_canonicalise: row i of nodes [n*L] (-1 or INT32_MAX padded) -> sorted [n*L] ascending with
 *   INT32_MAX padding, and a non-negative 64-bit key per row (equal rows => equal keys).
 * g2v_paths_mark: rows visited in key order (key_sorted[i] = key[perm[i]], ascending).  group == NULL:
 *   flag[i] = 1 iff row perm[i] is the first occurrence of its content (set semantics, exact: rows of a key
 *   run are compared in full).  group != NULL (0/1 per row): flag[i] = 1 iff no row of the other group has
 *   the same content (the row survives `pathSet - commonPath`).
 * ------------------------------------------------------------------------------------- */
int g2v_paths_canonicalise(const int32_t *nodes, int64_t n, int32_t L, int32_t *sorted, int64_t *key,
                           void *stream);
int g2v_paths_mark(const int32_t *rows, const int64_t *key_sorted, const int64_t *perm, const uint8_t *group,
                   int64_t n, int32_t L, uint8_t *flag, void *stream);

/* ---------------------------------------------------------------------------------------
 * Between the two hot paths, sort-free form (SURVEY.md 8f-2): from the canonical rows of BOTH groups (sorted,
 * INT32_MAX padded, with their 64-bit keys and lengths -- what g2v_walk_launch_packed writes with out_key) to the
 * trainer's input: `pathSet.add` (G2Vec.py:351), `pathSet - commonPath` (:313), the rows of integrate_pathSet
 * (:316-320) as CSR windows, and count_geneFreq (:288-308).
 * g2v_paths_set_select: keep[i] = 1 iff row i is the first occurrence of its content in its group (group[i] in
 *   {0,1}; NULL = one group) and no row of the other group has the same content.  totals (device, 3 x int64) =
 *   {rows kept, their total length, key collisions}; if collisions != 0 two different contents shared a key and the
 *   caller must use the exact sort-based functions above instead (never observed; ~n^2/2^64).
 * g2v_paths_set_emit: the kept rows in input order as CSR windows (rowptr [kept+1], gene [nnz], label [kept] = the
 *   row's group) and, if freq/code are given, code[g] = 0 / 1 / 2 / -1: more good paths / more poor / tie / gene in
 *   no kept path (freq: 2*V int32 scratch).  Synchronises the stream.
 * workspace: g2v_paths_set_workspace_bytes(n) bytes, the same buffer for both calls.
 * ------------------------------------------------------------------------------------- */
size_t g2v_paths_set_workspace_bytes(int64_t n);
int g2v_paths_set_select(const int32_t *rows, const int64_t *key, const uint8_t *group, const int32_t *len, int64_t n,
                         int32_t L, void *workspace, uint8_t *keep, int64_t *totals, void *stream);
int g2v_paths_set_emit(const int32_t *rows, const uint8_t *group, const int32_t *len, const uint8_t *keep, int64_t n,
                       int32_t L, int32_t V, const void *workspace, int64_t kept, int64_t nnz, int32_t *rowptr,
                       int32_t *gene, uint8_t *label, int32_t *freq, int8_t *code, void *stream);

/* ---------------------------------------------------------------------------------------
 * After training (csrc/g2v_post.cu): the command line's steps 5-7 on the device (--post gpu, g2vec_b200/post.py).
 *
 * Step 5, KMeans(n_clusters=3, random_state=0) as scikit-learn runs it.  X [V*D] row-major float32.
 * g2v_kmeans_workspace_bytes: device scratch for g2v_kmeans_center and g2v_kmeans_lloyd_step (one buffer serves both).
 * g2v_kmeans_center: mean [D] = float32 column mean, Xc = X - mean, var [D] (double) = per-feature population
 *   variance (scikit-learn's tol = 1e-4 * mean(var)).
 * g2v_kmeans_dist: k-means++ distance pass.  cand_host: HOST array of n_cand (1..8) row ids, read before the call
 *   returns.  out [n_cand*V]: out[k*V + i] = ||X[i] - X[cand[k]]||^2 as float32 (double accumulation), and
 *   min(closest[i], .) if closest != NULL.  The draws and the choice stay with the caller.
 * g2v_kmeans_lloyd_step: labels [V] = closest of the K (1..4) centres [K*D] (ties to the lower index), D <= 1024.
 *   centres_new != NULL: also centres_new = mean of each cluster's rows (the old centre if the cluster is empty) and
 *   status [2+2K] doubles = {rows whose label differs from labels_old (all rows if labels_old == NULL), empty clusters,
 *   count[0..K), ||new_k - old_k||^2 [0..K)}.  Fixed-order reductions, no floating-point atomics: bit-reproducible.
 *
 * Step 6: g2v_post_tscores: expr [S*V] sample-major, label [S] (0 good, 1 poor, other = neither) -> t [V] = the
 *   pooled-variance |t| of cli.tscore (ddof = 1; 0 when a group has < 2 samples or the pooled deviation is 0), in
 *   double.  g2v_post_row_norms: out [V] = ||X[r]||_2.
 *
 * Step 7, the vectors file: line r = prefix bytes [prefix_off[r], prefix_off[r+1]) (prefix_off NULL: none) +
 *   "\t%.6f" per value of X[r] (byte for byte as Python formats a float) + "\n".
 * g2v_fmt_row_bytes: row_bytes [rows] = length of each line.
 * g2v_fmt_emit: writes line r at out + offsets[r] (offsets: the caller's exclusive scan of row_bytes).
 * ------------------------------------------------------------------------------------- */
size_t g2v_kmeans_workspace_bytes(int32_t V, int32_t D, int32_t K);
int g2v_kmeans_center(const float *X, int32_t V, int32_t D, float *Xc, float *mean, double *var, void *workspace,
                      void *stream);
int g2v_kmeans_dist(const float *X, int32_t V, int32_t D, const int64_t *cand_host, int32_t n_cand,
                    const float *closest, float *out, void *stream);
int g2v_kmeans_lloyd_step(const float *X, int32_t V, int32_t D, int32_t K, const float *centres, float *centres_new,
                          const int32_t *labels_old, int32_t *labels, double *status, void *workspace, void *stream);
int g2v_post_tscores(const float *expr, int32_t S, int32_t V, const uint8_t *label, float *t, void *stream);
int g2v_post_row_norms(const float *X, int64_t V, int32_t D, float *out, void *stream);
int g2v_fmt_row_bytes(const float *X, int64_t rows, int32_t D, const int64_t *prefix_off, int64_t *row_bytes,
                      void *stream);
int g2v_fmt_emit(const float *X, int64_t rows, int32_t D, const char *prefix, const int64_t *prefix_off,
                 const int64_t *offsets, char *out, void *stream);

/* ---------------------------------------------------------------------------------------
 * Test hooks (used by tests/ only): 64-bit draws 0..n-1 of one walker subsequence from the
 * kernel's own Philox, and the same words from curand's Philox4_32_10 generator
 * (curand_init(seed, subsequence, 0)), to prove the stream is curand-compatible.
 * ------------------------------------------------------------------------------------- */
/* Measurement hook: (mode 0) read / (mode 1) red.add a constant into the rows idx[0..n_idx) of a [*, D] float
 * table, D a multiple of 128 -- the memory operations of the CBOW kernels without the arithmetic; bench.py times it
 * on an L2-resident table to get the L2 ceiling the fused kernel is compared with.  sink: >= 1024 floats. */
int g2v_test_l2_rows(const float *table, float *grad, const int32_t *idx, int64_t n_idx, int32_t D, int32_t mode,
                     float *sink, void *stream);
int g2v_test_draws(uint64_t seed, uint64_t subsequence, int32_t n, uint64_t *out_dev, void *stream);
int g2v_test_curand_draws(uint64_t seed, uint64_t subsequence, int32_t n, uint64_t *out_dev,
                          void *stream);

#ifdef __cplusplus
}
#endif
#endif /* G2VEC_B200_H */
