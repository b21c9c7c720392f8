// g2v_cbow_slab.cu -- HOT PATH 2 for embedding tables that do not fit the L2: the same gather -> sum ->
// logit -> BCE -> scatter-add step as cbow_rows_kernel (g2v_cbow.cu; G2Vec.py:239-246), processed GENE SLAB BY
// GENE SLAB so that the rows being gathered and the gradient rows being added to stay L2-resident.
//
// Why: with V*D*4 >> L2 (200k genes x 512: 410 MB against 126 MB) every gathered row and every
// red.global.add into g_ih misses; the reduction is then a DRAM read-modify-write (ncu, round 1: 272 GB of DRAM
// traffic for 210 GB algorithmic, 9 % L2 hit rate, 0.74 of the HBM peak).  The windows are static across steps
// and their gene lists are sorted (tuple(sorted(path)), G2Vec.py:345), so the genes of a window that fall into
// the slab [lo, hi) are ONE contiguous piece of its list.  slab_setup_kernel records those pieces once
// (slabptr [n_win, S+1]); then per optimizer step
//
//   forward  pass j (S_f launches)  every window adds the rows of its genes in slab group j to its partial
//                                   context sum, which lives in hbuf [n_win, D] between passes (streaming loads
//                                   and stores, evict-first); the last pass finishes the window: logit, loss,
//                                   accuracy, dO -> dO[n_win], and h*dO into g_ho
//   backward pass s (S launches)    every window adds dO*W_ho into g_ih rows of its genes in slab s
//
// During a pass the 148 SMs only touch one slab of W_ih (forward) or g_ih (backward): after its first touch a
// row is served by the L2 (each row of a slab is used N*l/V times per pass -- 256 times at the stress size), and
// DRAM sees the slab once plus the streamed hbuf/gene-id traffic.  Forward slabs may be wider than backward
// slabs (only the table has to stay resident, not table + gradient): forward group j = backward slabs
// [j*G, (j+1)*G).  The accuracy passes (g2v_cbow_eval) use the same forward passes with a 4-byte partial logit
// per window instead of hbuf.
//
// Results: same sums in a different float32 order (per window the genes are still added in ascending order; the
// partial sum is carried exactly through hbuf) -- same oracle, same tolerance as the fused kernel.
#include <stdlib.h>

#include "g2v_cbow_common.cuh"

namespace g2v {

constexpr bool kDefaultSlabScatterTma = false;   // set from the B200 measurement in profiles/r2

__device__ __forceinline__ float4 ld_stream4(const float4 *p) { return __ldcs(p); }
__device__ __forceinline__ void st_stream4(float4 *p, float4 v) { __stcs(p, v); }

// slabptr[i*(S+1) + s] = first position (absolute index into gene[]) of window i whose gene id >= s*rows_per_slab;
// entry S = end of the window.  *bad is set if a window's gene list is not strictly ascending.
__global__ void __launch_bounds__(256)
slab_setup_kernel(const int32_t *__restrict__ rowptr, const int32_t *__restrict__ gene,
                  const int32_t *__restrict__ win, int64_t win_begin, int64_t n_win, int32_t rows_per_slab, int32_t S,
                  int32_t *__restrict__ slabptr, int32_t *__restrict__ bad) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_win; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t n = win ? (int64_t)__ldg(win + win_begin + i) : win_begin + i;
        const int32_t b = __ldg(rowptr + n), e = __ldg(rowptr + n + 1);
        int32_t *sp = slabptr + i * (S + 1);
        int s = 0;
        int32_t prev = -1;
        sp[0] = b;
        for (int32_t j = b; j < e; ++j) {
            const int32_t g = __ldg(gene + j);
            if (g <= prev) *bad = 1;
            prev = g;
            while (s + 1 <= S - 1 && g >= (s + 1) * rows_per_slab) sp[++s] = j;
        }
        while (s < S) sp[++s] = e;
    }
}

// MODE 0: training forward (hbuf carries the partial context sum; LAST computes dO and g_ho)
// MODE 1: accuracy pass (obuf carries the partial logit; LAST counts correct predictions)
template <int VEC, int MODE, bool FIRST, bool LAST>
__global__ void __launch_bounds__(kCbowWarps * 32)
cbow_slab_fwd_kernel(const int32_t *__restrict__ gene, const uint8_t *__restrict__ label,
                     const int32_t *__restrict__ win, int64_t win_begin, int64_t n_win,
                     const int32_t *__restrict__ slabptr, int32_t S1, int32_t s_lo, int32_t s_hi, float inv_n,
                     const float *__restrict__ W_ih, const float *__restrict__ W_ho, float *__restrict__ hbuf,
                     float *__restrict__ obuf, float *__restrict__ dOut, float *__restrict__ g_ho,
                     double *__restrict__ loss_sum, unsigned long long *__restrict__ n_correct, int32_t reduce_mean,
                     const int32_t *__restrict__ skip) {
    G2V_SKIP_IF_STOPPED(skip);
    constexpr int D = 128 * VEC;
    constexpr int D4 = D / 4;
    constexpr int UNR = 8 / VEC;                 // 8 float4 (128 B) in flight per lane
    constexpr bool TRAIN = MODE == 0;
    __shared__ float sh_gho[(TRAIN && LAST) ? D : 1];
    __shared__ CtaAcc sh_acc;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (TRAIN && LAST) for (int i = threadIdx.x; i < D; i += blockDim.x) sh_gho[i] = 0.f;
    if (threadIdx.x == 0) { sh_acc.loss = 0.0; sh_acc.correct = 0ull; }
    __syncthreads();

    const float4 *__restrict__ W4 = reinterpret_cast<const float4 *>(W_ih);
    float4 who[VEC], gho[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
        who[v] = ldg4(reinterpret_cast<const float4 *>(W_ho) + v * 32 + lane);
        gho[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float loss_acc = 0.f;
    unsigned correct_acc = 0;

    const int64_t warps_total = (int64_t)gridDim.x * kCbowWarps;
    for (int64_t i = (int64_t)blockIdx.x * kCbowWarps + warp; i < n_win; i += warps_total) {
        const int32_t *sp = slabptr + i * S1;
        const int32_t b = __ldg(sp + s_lo), e = __ldg(sp + s_hi);
        if (!LAST && !FIRST && b == e) continue;                  // nothing of this window in the slab group
        float4 h[VEC];
        float4 *hrow = TRAIN ? reinterpret_cast<float4 *>(hbuf) + (size_t)i * D4 + lane : nullptr;
#pragma unroll
        for (int v = 0; v < VEC; ++v)
            h[v] = (TRAIN && !FIRST) ? ld_stream4(hrow + v * 32) : make_float4(0.f, 0.f, 0.f, 0.f);

        for (int32_t base = b; base < e; base += 32) {
            const int cnt = min(32, e - base);
            const int32_t g = (lane < cnt) ? __ldg(gene + base + lane) : 0;
            for (int k = 0; k < cnt; k += UNR) {
                float4 r[UNR][VEC];
#pragma unroll
                for (int u = 0; u < UNR; ++u) {
                    const int32_t gk = __shfl_sync(0xffffffffu, g, (k + u) & 31);
                    const float4 *row = W4 + (size_t)gk * D4 + lane;
#pragma unroll
                    for (int v = 0; v < VEC; ++v)
                        r[u][v] = (k + u < cnt) ? ldg4(row + v * 32) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int u = 0; u < UNR; ++u)
#pragma unroll
                    for (int v = 0; v < VEC; ++v) {
                        h[v].x += r[u][v].x; h[v].y += r[u][v].y; h[v].z += r[u][v].z; h[v].w += r[u][v].w;
                    }
            }
        }
        if (TRAIN && !LAST) {
#pragma unroll
            for (int v = 0; v < VEC; ++v) st_stream4(hrow + v * 32, h[v]);
            continue;
        }
        // whole-window length (for the mean variant): first and last entry of the window's slab table
        const int32_t len = __ldg(sp + S1 - 1) - __ldg(sp);
        const float scale = (reduce_mean && len > 0) ? 1.f / (float)len : 1.f;
        float part = 0.f;
#pragma unroll
        for (int v = 0; v < VEC; ++v)
            part += h[v].x * who[v].x + h[v].y * who[v].y + h[v].z * who[v].z + h[v].w * who[v].w;
        float o = warp_sum(part);                                 // logit of this pass's rows (TRAIN: of the whole window)
        if (!TRAIN) {
            if (!FIRST) o += obuf[i];
            if (!LAST) { if (lane == 0) obuf[i] = o; continue; }
        }
        o *= scale;
        const int64_t n = win ? (int64_t)__ldg(win + win_begin + i) : win_begin + i;
        const float y = (float)__ldg(label + n);
        if (lane == 0) {
            correct_acc += ((o > 0.f) == (y != 0.f)) ? 1u : 0u;
            if (TRAIN) loss_acc += fmaxf(o, 0.f) - o * y + log1pf(expf(-fabsf(o)));
        }
        if (TRAIN) {
            const float dO = (sigmoid_stable(o) - y) * inv_n;
            const float hs = dO * scale;                          // d cost / d (sum of rows)
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                gho[v].x += h[v].x * hs; gho[v].y += h[v].y * hs; gho[v].z += h[v].z * hs; gho[v].w += h[v].w * hs;
            }
            if (lane == 0) dOut[i] = hs;
        }
    }

    if (TRAIN && LAST) {
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            float *p = sh_gho + (v * 32 + lane) * 4;
            atomicAdd(p + 0, gho[v].x); atomicAdd(p + 1, gho[v].y);
            atomicAdd(p + 2, gho[v].z); atomicAdd(p + 3, gho[v].w);
        }
    }
    if (LAST && lane == 0) {
        if (TRAIN) atomicAdd(&sh_acc.loss, (double)loss_acc);
        atomicAdd(&sh_acc.correct, (unsigned long long)correct_acc);
    }
    __syncthreads();
    if (TRAIN && LAST) for (int i = threadIdx.x; i < D; i += blockDim.x) atomicAdd(g_ho + i, sh_gho[i]);
    if (LAST && threadIdx.x == 0) {
        if (TRAIN && loss_sum) atomicAdd(loss_sum, sh_acc.loss);
        if (n_correct) atomicAdd(n_correct, sh_acc.correct);
    }
}

// TMA = false: every lane adds its 16 bytes of the gradient row with red.global.add.v4.f32 (LSU/L1TEX path:
// VEC warp-wide RED.128 per gene row).  TMA = true: the row dO*W_ho -- the same for every gene of the
// window -- is staged once in shared memory and added into g_ih[gene,:] with ONE bulk reduction per gene
// (cp.reduce.async.bulk.global.shared::cta.add.f32, D*4 bytes, SASS UBLKRED) issued by one lane: the scatter
// leaves the LSU/L1TEX path, which is what bounds the L2-resident backward passes (ncu: l1tex 87 %).
// Two staging rows per warp, so that a window's row can be written while the previous window's bulk
// reductions are still reading theirs.
template <int VEC, bool TMA>
__global__ void __launch_bounds__(kCbowWarps * 32)
cbow_slab_bwd_kernel(const int32_t *__restrict__ gene, int64_t n_win, const int32_t *__restrict__ slabptr, int32_t S1,
                     int32_t s, const float *__restrict__ dOut, const float *__restrict__ W_ho,
                     float *__restrict__ g_ih, const int32_t *__restrict__ skip) {
    G2V_SKIP_IF_STOPPED(skip);
    constexpr int D = 128 * VEC;
    __shared__ __align__(128) float sh_row[TMA ? kCbowWarps * 2 * D : 4];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float4 who[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) who[v] = ldg4(reinterpret_cast<const float4 *>(W_ho) + v * 32 + lane);
    const int64_t warps_total = (int64_t)gridDim.x * kCbowWarps;
    int stage = 0;
    for (int64_t i = (int64_t)blockIdx.x * kCbowWarps + warp; i < n_win; i += warps_total) {
        const int32_t b = __ldg(slabptr + i * S1 + s), e = __ldg(slabptr + i * S1 + s + 1);
        if (b == e) continue;
        const float hs = __ldg(dOut + i);
        float4 gv[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) gv[v] = make_float4(who[v].x * hs, who[v].y * hs, who[v].z * hs, who[v].w * hs);
        if (TMA) {
            float *row = sh_row + (size_t)(warp * 2 + stage) * D;
            // at most one older group (the other stage) may still be reading shared memory
            asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            __syncwarp();
#pragma unroll
            for (int v = 0; v < VEC; ++v) reinterpret_cast<float4 *>(row)[v * 32 + lane] = gv[v];
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> async proxy
            __syncwarp();
            const uint32_t src = (uint32_t)__cvta_generic_to_shared(row);
            for (int32_t j = b + lane; j < e; j += 32) {
                float *dst = g_ih + (size_t)__ldg(gene + j) * D;
                asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f32 [%0], [%1], %2;"
                             ::"l"(dst), "r"(src), "n"(D * 4)
                             : "memory");
            }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            stage ^= 1;
        } else {
            for (int32_t base = b; base < e; base += 32) {
                const int cnt = min(32, e - base);
                const int32_t g = (lane < cnt) ? __ldg(gene + base + lane) : 0;
                for (int k = 0; k < cnt; ++k) {
                    const int32_t gk = __shfl_sync(0xffffffffu, g, k);
                    float *dst = g_ih + (size_t)gk * D + lane * 4;
#pragma unroll
                    for (int v = 0; v < VEC; ++v) red_add4(dst + v * 128, gv[v]);
                }
            }
        }
    }
    if (TMA) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

struct SlabLayout {            // carving of the caller's workspace
    int32_t *slabptr;          // [n_win * (S+1)]
    float *dO, *obuf;          // [n_win] each
    float *hbuf;               // [n_win * D]
};

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

static SlabLayout carve(void *ws, int64_t n_win, int32_t S) {
    char *p = reinterpret_cast<char *>(ws);
    SlabLayout l;
    l.slabptr = reinterpret_cast<int32_t *>(p); p += align256(sizeof(int32_t) * (size_t)n_win * (size_t)(S + 1));
    l.dO = reinterpret_cast<float *>(p); p += align256(sizeof(float) * (size_t)n_win);
    l.obuf = reinterpret_cast<float *>(p); p += align256(sizeof(float) * (size_t)n_win);
    l.hbuf = reinterpret_cast<float *>(p);
    return l;
}

static int fwd_group() {       // forward slab group = this many backward slabs (only the table must stay resident)
    const char *e = getenv("G2V_CBOW_SLAB_FWD_GROUP");
    const int g = e ? atoi(e) : 2;
    return g >= 1 ? g : 1;
}

template <int VEC, int MODE>
static int launch_fwd_passes(const int32_t *gene, const uint8_t *label, const int32_t *win, int64_t win_begin,
                             int64_t n_win, const SlabLayout &l, int32_t S, float inv_n, const float *W_ih,
                             const float *W_ho, float *g_ho, double *loss_sum, unsigned long long *nc, int32_t reduce,
                             cudaStream_t st) {
    const int G = fwd_group();
    const int passes = (S + G - 1) / G;
    for (int j = 0; j < passes; ++j) {
        const bool first = j == 0, last = j == passes - 1;
        const int32_t lo = j * G, hi = (j + 1) * G < S ? (j + 1) * G : S;
        int grid = 0, rc;
#define G2V_SLAB_FWD(F, L)                                                                                 \
    {                                                                                                      \
        auto kern = cbow_slab_fwd_kernel<VEC, MODE, F, L>;                                                 \
        if ((rc = rows_grid((const void *)kern, 0, n_win, &grid))) return rc;                              \
        kern<<<grid, kCbowWarps * 32, 0, st>>>(gene, label, win, win_begin, n_win, l.slabptr, S + 1, lo, hi, inv_n, \
                                               W_ih, W_ho, l.hbuf, l.obuf, l.dO, g_ho, loss_sum, nc, reduce, loop_skip_flag()); \
    }
        if (first && last) G2V_SLAB_FWD(true, true)
        else if (first) G2V_SLAB_FWD(true, false)
        else if (last) G2V_SLAB_FWD(false, true)
        else G2V_SLAB_FWD(false, false)
#undef G2V_SLAB_FWD
        G2V_CUDA_OK(cudaGetLastError());
        count_launch();
    }
    return 0;
}

template <int VEC>
static int launch_bwd_passes(const int32_t *gene, int64_t n_win, const SlabLayout &l, int32_t S, const float *W_ho,
                             float *g_ih, cudaStream_t st) {
    const char *sc = getenv("G2V_CBOW_SLAB_SCATTER");             // "red" (default) / "tma": A/B hook, see profiles/r2
    const bool tma = sc ? sc[0] == 't' : kDefaultSlabScatterTma;
    auto kern = tma ? cbow_slab_bwd_kernel<VEC, true> : cbow_slab_bwd_kernel<VEC, false>;
    int grid = 0, rc;
    if ((rc = rows_grid((const void *)kern, 0, n_win, &grid))) return rc;
    for (int s = 0; s < S; ++s) {
        kern<<<grid, kCbowWarps * 32, 0, st>>>(gene, n_win, l.slabptr, S + 1, s, l.dO, W_ho, g_ih, loop_skip_flag());
        G2V_CUDA_OK(cudaGetLastError());
        count_launch();
    }
    return 0;
}

}  // namespace g2v

using namespace g2v;

extern "C" int g2v_cbow_slab_plan(int32_t V, int32_t D, int32_t *n_slabs) {
    G2V_REQUIRE(V > 0 && D > 0 && n_slabs, "g2v_cbow_slab_plan: bad arguments");
    DeviceProps dp;
    if (device_props(&dp)) return 1;
    *n_slabs = 1;
    if (D != 128 && D != 256 && D != 512) return 0;               // the generic-D kernel has no slab form
    const double table = (double)V * D * 4.0;
    // table + gradient resident together: the fused single-pass kernel is already L2-bound
    const char *e = getenv("G2V_CBOW_SLAB_MB");                   // bytes of one BACKWARD slab of g_ih (tuning hook)
    const double slab = (e && atof(e) > 0 ? atof(e) : 32.0) * 1048576.0;
    const char *f = getenv("G2V_CBOW_SLABS");                     // force a slab count (tests)
    if (f && atoi(f) >= 1) { *n_slabs = atoi(f) > V ? V : atoi(f); return 0; }
    if (2.0 * table <= 0.75 * (double)dp.l2_bytes) return 0;
    int s = (int)((table + slab - 1) / slab);
    if (s < 2) s = 2;
    if (s > 64) s = 64;
    *n_slabs = s;
    return 0;
}

extern "C" size_t g2v_cbow_slab_workspace_bytes(int64_t n_win, int32_t D, int32_t n_slabs) {
    if (n_win <= 0 || D <= 0 || n_slabs <= 0) return 0;
    return align256(sizeof(int32_t) * (size_t)n_win * (size_t)(n_slabs + 1)) + 2 * align256(sizeof(float) * (size_t)n_win) +
           align256(sizeof(float) * (size_t)n_win * (size_t)D) + 256;
}

extern "C" int g2v_cbow_slab_setup(const int32_t *rowptr, const int32_t *gene, const int32_t *win, int64_t win_begin,
                                   int64_t n_win, int32_t V, int32_t n_slabs, void *workspace, void *stream) {
    G2V_REQUIRE(V > 0 && n_slabs >= 1 && n_win >= 0 && win_begin >= 0, "g2v_cbow_slab_setup: bad sizes");
    if (n_win == 0) return 0;
    G2V_REQUIRE(rowptr && workspace, "g2v_cbow_slab_setup: null pointer");
    DeviceProps dp;
    if (device_props(&dp)) return 1;
    cudaStream_t st = (cudaStream_t)stream;
    SlabLayout l = carve(workspace, n_win, n_slabs);
    // the "unsorted" flag borrows the first word of obuf (obuf is rewritten by every accuracy pass)
    int32_t *bad = reinterpret_cast<int32_t *>(l.obuf);
    G2V_CUDA_OK(cudaMemsetAsync(bad, 0, sizeof(int32_t), st));
    const int32_t rows_per_slab = (V + n_slabs - 1) / n_slabs;
    int64_t blocks = (n_win + 255) / 256;
    if (blocks > (int64_t)dp.sm_count * 8) blocks = (int64_t)dp.sm_count * 8;
    slab_setup_kernel<<<(unsigned)blocks, 256, 0, st>>>(rowptr, gene, win, win_begin, n_win, rows_per_slab, n_slabs,
                                                        l.slabptr, bad);
    G2V_CUDA_OK(cudaGetLastError());
    count_launch();
    int32_t h = 0;
    G2V_CUDA_OK(cudaMemcpyAsync(&h, bad, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    G2V_CUDA_OK(cudaStreamSynchronize(st));                       // setup, once per window list
    G2V_REQUIRE(h == 0, "g2v_cbow_slab_setup: a window's gene list is not strictly ascending (the slab kernels need "
                        "sorted windows, as tuple(sorted(path)) produces them)");
    return 0;
}

extern "C" int g2v_cbow_fwdbwd_slabs(const int32_t *gene, const uint8_t *label, const int32_t *win, int64_t win_begin,
                                     int64_t n_win, float inv_n_total, const float *W_ih, const float *W_ho,
                                     float *g_ih, float *g_ho, double *loss_sum, int64_t *n_correct, int32_t V,
                                     int32_t D, int32_t reduce, int32_t n_slabs, void *workspace, void *stream) {
    G2V_REQUIRE(V > 0 && n_win >= 0 && n_slabs >= 1, "g2v_cbow_fwdbwd_slabs: bad sizes");
    G2V_REQUIRE(D == 128 || D == 256 || D == 512, "g2v_cbow_fwdbwd_slabs: sizeHiddenlayer must be 128, 256 or 512 (got %d)", D);
    G2V_REQUIRE(gene && label && W_ih && W_ho && g_ih && g_ho && workspace, "g2v_cbow_fwdbwd_slabs: null pointer");
    G2V_REQUIRE(reduce == G2V_REDUCE_SUM || reduce == G2V_REDUCE_MEAN, "g2v_cbow_fwdbwd_slabs: unknown reduce %d", reduce);
    if (n_win == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    SlabLayout l = carve(workspace, n_win, n_slabs);
    unsigned long long *nc = reinterpret_cast<unsigned long long *>(n_correct);
    int rc;
#define G2V_SLAB_STEP(VEC)                                                                                          \
    {                                                                                                               \
        if ((rc = launch_fwd_passes<VEC, 0>(gene, label, win, win_begin, n_win, l, n_slabs, inv_n_total, W_ih, W_ho, \
                                            g_ho, loss_sum, nc, reduce, st))) return rc;                             \
        if ((rc = launch_bwd_passes<VEC>(gene, n_win, l, n_slabs, W_ho, g_ih, st))) return rc;                       \
    }
    if (D == 128) G2V_SLAB_STEP(1)
    else if (D == 256) G2V_SLAB_STEP(2)
    else G2V_SLAB_STEP(4)
#undef G2V_SLAB_STEP
    return 0;
}

extern "C" int g2v_cbow_eval_slabs(const int32_t *gene, const uint8_t *label, const int32_t *win, int64_t win_begin,
                                   int64_t n_win, const float *W_ih, const float *W_ho, int64_t *n_correct, int32_t V,
                                   int32_t D, int32_t reduce, int32_t n_slabs, void *workspace, void *stream) {
    G2V_REQUIRE(V > 0 && n_win >= 0 && n_slabs >= 1, "g2v_cbow_eval_slabs: bad sizes");
    G2V_REQUIRE(D == 128 || D == 256 || D == 512, "g2v_cbow_eval_slabs: sizeHiddenlayer must be 128, 256 or 512 (got %d)", D);
    G2V_REQUIRE(gene && label && W_ih && W_ho && n_correct && workspace, "g2v_cbow_eval_slabs: null pointer");
    G2V_REQUIRE(reduce == G2V_REDUCE_SUM || reduce == G2V_REDUCE_MEAN, "g2v_cbow_eval_slabs: unknown reduce %d", reduce);
    if (n_win == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    SlabLayout l = carve(workspace, n_win, n_slabs);
    unsigned long long *nc = reinterpret_cast<unsigned long long *>(n_correct);
    if (D == 128) return launch_fwd_passes<1, 1>(gene, label, win, win_begin, n_win, l, n_slabs, 0.f, W_ih, W_ho, nullptr, nullptr, nc, reduce, st);
    if (D == 256) return launch_fwd_passes<2, 1>(gene, label, win, win_begin, n_win, l, n_slabs, 0.f, W_ih, W_ho, nullptr, nullptr, nc, reduce, st);
    return launch_fwd_passes<4, 1>(gene, label, win, win_begin, n_win, l, n_slabs, 0.f, W_ih, W_ho, nullptr, nullptr, nc, reduce, st);
}
