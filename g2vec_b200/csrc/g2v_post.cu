// g2v_post.cu -- the command line's steps 5-7 on the device (--post gpu, g2vec_b200/post.py).
//
// Step 5, L-groups: KMeans(n_clusters=3, random_state=0) as scikit-learn runs it (cluster/_kmeans.py):
//   kmeans_colsum_kernel / kmeans_colfin_kernel   column mean (data centred on it) and per-feature variance (tol)
//   kmeans_dist_kernel     k-means++ distance pass: squared distance of every row to each candidate centre, running
//                          minimum with the closest distances so far.  The random draws, the cumulative sum and the
//                          searchsorted stay on the host in NumPy, so the chosen ids are scikit-learn's ids.
//   kmeans_assign_kernel   one Lloyd pass: label = closest centre (ties to the lower index), per-block partial sums
//                          of the rows of each cluster, per-block label-change count
//   kmeans_update_kernel   partial sums reduced in block order -> new centres and squared shifts
//   kmeans_status_kernel   one block: changes, empty clusters, counts and shifts for the host's stopping rule
// Every reduction has a fixed order and there are no floating-point atomics: the same input on the same device gives
// the same labels on every run.  Distances accumulate in double.
// Step 6, gene scores: per-gene |t| (pooled variance, ddof = 1) and the row L2 norms of W_ih.
// Step 7, the vectors file: "\t%.6f" per value, byte for byte as Python formats it, in two passes (bytes per row;
// emit at the caller's exclusive-scan offsets), with integer arithmetic only (see fmt_decompose).
#include "g2v_common.cuh"

namespace g2v {

constexpr int kMaxK = 4;          // clusters per call
constexpr int kMaxKmD = 1024;     // features per row for the k-means kernels (4 columns per thread of 256)
constexpr int kMaxCand = 8;       // k-means++ candidates per distance pass

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---------------------------------------------------------------- column statistics (centring and tol)
// partial[b][0][c] = sum over the block's rows of (x - shift[c]), partial[b][1][c] = sum of its square.  With
// shift = NULL (first pass) only the plain sums are used; with shift = the float32 mean (second pass) Xc = x - mean
// is written and the second moment of the centred data gives the variance without cancellation.
__global__ void __launch_bounds__(128)
kmeans_colsum_kernel(const float *__restrict__ X, int32_t V, int32_t D, const float *__restrict__ shift,
                     float *__restrict__ Xc, double *__restrict__ partial) {
    const int c = blockIdx.x * 128 + threadIdx.x;
    const int64_t per = ((int64_t)V + gridDim.y - 1) / gridDim.y;
    const int64_t r0 = (int64_t)blockIdx.y * per, r1 = min((int64_t)V, r0 + per);
    double s = 0.0, ss = 0.0;
    if (c < D) {
        const float m = shift ? shift[c] : 0.f;
        for (int64_t r = r0; r < r1; ++r) {
            const float x = __ldg(X + r * D + c) - m;
            if (Xc) Xc[r * D + c] = x;
            s += (double)x;
            ss += (double)x * (double)x;
        }
        partial[((size_t)blockIdx.y * 2 + 0) * D + c] = s;
        partial[((size_t)blockIdx.y * 2 + 1) * D + c] = ss;
    }
}

// Blocks reduced in block order.  mean_out (float32 column mean) or var_out (double population variance of the
// already centred data) is written.
__global__ void __launch_bounds__(128)
kmeans_colfin_kernel(const double *__restrict__ partial, int32_t nb, int32_t V, int32_t D, float *__restrict__ mean_out,
                     double *__restrict__ var_out) {
    const int c = blockIdx.x * 128 + threadIdx.x;
    if (c >= D) return;
    double s = 0.0, ss = 0.0;
    for (int b = 0; b < nb; ++b) {
        s += partial[((size_t)b * 2 + 0) * D + c];
        ss += partial[((size_t)b * 2 + 1) * D + c];
    }
    const double mu = s / (double)V;
    if (mean_out) mean_out[c] = (float)mu;
    if (var_out) var_out[c] = ss / (double)V - mu * mu;
}

// ---------------------------------------------------------------- k-means++ distance pass
struct CandIds { int64_t id[kMaxCand]; };

// One warp per row: out[k][i] = min(closest[i], ||X[i] - X[cand_k]||^2) as float32 (closest == NULL: no minimum).
__global__ void __launch_bounds__(256)
kmeans_dist_kernel(const float *__restrict__ X, int32_t V, int32_t D, CandIds cand, int32_t n_cand,
                   const float *__restrict__ closest, float *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < V; r += nwarps) {
        const float *x = X + r * D;
        for (int k = 0; k < n_cand; ++k) {
            const float *c = X + cand.id[k] * D;
            double acc = 0.0;
            for (int j = lane; j < D; j += 32) {
                const double d = (double)__ldg(x + j) - (double)__ldg(c + j);
                acc += d * d;
            }
            acc = warp_sum_f64(acc);
            if (lane == 0) {
                float v = (float)acc;
                if (closest) v = fminf(v, closest[r]);
                out[(int64_t)k * V + r] = v;
            }
        }
    }
}

// ---------------------------------------------------------------- Lloyd iteration
// Block = 8 warps; a tile is 8 rows, one per warp.  Each warp stages its row in shared memory while it computes the
// K distances, picks the label, and counts a change against labels_old.  After a barrier, thread t accumulates
// columns t, t+256, ... of the tile's rows into the register accumulator of their cluster (double).  Rows are visited
// in a fixed order per block, so the per-block partials -- and, reduced in block order by kmeans_update_kernel, the
// new centres -- do not depend on scheduling.  partial == NULL: labels only (scikit-learn's final E step).
__global__ void __launch_bounds__(256)
kmeans_assign_kernel(const float *__restrict__ X, int32_t V, int32_t D, int32_t K, const float *__restrict__ centres,
                     const int32_t *__restrict__ labels_old, int32_t *__restrict__ labels, double *__restrict__ partial,
                     int64_t *__restrict__ counts) {
    extern __shared__ float tile[];                 // [8][D]
    __shared__ int32_t tlab[8];
    __shared__ int32_t tchg[8];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    double acc[kMaxKmD / 256][kMaxK];
#pragma unroll
    for (int q = 0; q < kMaxKmD / 256; ++q)
#pragma unroll
        for (int k = 0; k < kMaxK; ++k) acc[q][k] = 0.0;
    int64_t cnt[kMaxK] = {0, 0, 0, 0};
    int64_t changed = 0;
    const int64_t n_tiles = ((int64_t)V + 7) / 8;
    for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const int64_t r = t * 8 + w;
        if (r < V) {
            double d[kMaxK];
#pragma unroll
            for (int k = 0; k < kMaxK; ++k) d[k] = 0.0;
            for (int j = lane; j < D; j += 32) {
                const float x = __ldg(X + r * D + j);
                tile[w * D + j] = x;
#pragma unroll
                for (int k = 0; k < kMaxK; ++k)
                    if (k < K) { const double e = (double)x - (double)__ldg(centres + k * D + j); d[k] += e * e; }
            }
            int best = 0;
            double bd = warp_sum_f64(d[0]);
#pragma unroll
            for (int k = 1; k < kMaxK; ++k)
                if (k < K) { const double v = warp_sum_f64(d[k]); if (v < bd) { bd = v; best = k; } }
            if (lane == 0) {
                labels[r] = best;
                tlab[w] = best;
                tchg[w] = labels_old ? (labels_old[r] != best) : 1;
            }
        } else if (lane == 0) {
            tlab[w] = -1;
            tchg[w] = 0;
        }
        __syncthreads();
        if (partial) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int lab = tlab[i];
                if (lab < 0) continue;
#pragma unroll
                for (int q = 0; q < kMaxKmD / 256; ++q) {
                    const int c = q * 256 + threadIdx.x;
                    if (c < D) {
                        const double x = (double)tile[i * D + c];
#pragma unroll
                        for (int k = 0; k < kMaxK; ++k) acc[q][k] += (lab == k) ? x : 0.0;
                    }
                }
            }
        }
        if (threadIdx.x == 0)
            for (int i = 0; i < 8; ++i) {
#pragma unroll
                for (int k = 0; k < kMaxK; ++k) cnt[k] += tlab[i] == k;
                changed += tchg[i];
            }
        __syncthreads();
    }
    if (!partial) return;
    // partial layout: [nb][K][D] doubles; counts: [nb][K + 1] (the last entry is the block's change count)
#pragma unroll
    for (int q = 0; q < kMaxKmD / 256; ++q) {
        const int c = q * 256 + threadIdx.x;
        if (c < D)
            for (int k = 0; k < K; ++k) partial[((size_t)blockIdx.x * K + k) * D + c] = acc[q][k];
    }
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < kMaxK; ++k)
            if (k < K) counts[(size_t)blockIdx.x * (K + 1) + k] = cnt[k];
        counts[(size_t)blockIdx.x * (K + 1) + K] = changed;
    }
}

// grid (ceil(D/32), K), block 32 columns x 8 ways: way v sums blocks v, v+8, ... in order, then the ways are added
// in order.  new = sum / count (the old centre is kept for an empty cluster, which the status reports).
__global__ void __launch_bounds__(256)
kmeans_update_kernel(const double *__restrict__ partial, const int64_t *__restrict__ counts, int32_t nb, int32_t D,
                     int32_t K, const float *__restrict__ centres, float *__restrict__ centres_new,
                     double *__restrict__ shift_sq) {
    __shared__ double sh[8][33];
    const int cl = threadIdx.x & 31, way = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + cl, k = blockIdx.y;
    double s = 0.0;
    if (c < D)
        for (int b = way; b < nb; b += 8) s += partial[((size_t)b * K + k) * D + c];
    sh[way][cl] = s;
    __syncthreads();
    if (way == 0 && c < D) {
        double tot = 0.0;
        for (int v = 0; v < 8; ++v) tot += sh[v][cl];
        int64_t n = 0;
        for (int b = 0; b < nb; ++b) n += counts[(size_t)b * (K + 1) + k];
        const float old = centres[k * D + c];
        const float nw = n > 0 ? (float)(tot / (double)n) : old;
        centres_new[k * D + c] = nw;
        const double e = (double)nw - (double)old;
        shift_sq[k * D + c] = e * e;
    }
}

// One block.  status = {label changes, empty clusters, count[0..K), shift[0..K)} in double; shift[k] is the squared
// distance between the old and the new centre k (scikit-learn's center_shift[k]**2).
__global__ void __launch_bounds__(256)
kmeans_status_kernel(const int64_t *__restrict__ counts, int32_t nb, int32_t D, int32_t K,
                     const double *__restrict__ shift_sq, double *__restrict__ status) {
    __shared__ double sh[256];
    __shared__ int64_t shn[256];
    for (int k = 0; k <= K; ++k) {
        int64_t n = 0;
        for (int b = threadIdx.x; b < nb; b += 256) n += counts[(size_t)b * (K + 1) + k];
        shn[threadIdx.x] = n;
        __syncthreads();
        if (threadIdx.x == 0) {
            int64_t tot = 0;
            for (int i = 0; i < 256; ++i) tot += shn[i];
            if (k < K) status[2 + k] = (double)tot;
            else status[0] = (double)tot;
        }
        __syncthreads();
    }
    for (int k = 0; k < K; ++k) {
        double s = 0.0;
        for (int c = threadIdx.x; c < D; c += 256) s += shift_sq[k * D + c];
        sh[threadIdx.x] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            double tot = 0.0;
            for (int i = 0; i < 256; ++i) tot += sh[i];
            status[2 + K + k] = tot;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        int empty = 0;
        for (int k = 0; k < K; ++k) empty += status[2 + k] == 0.0;
        status[1] = (double)empty;
    }
}

// ---------------------------------------------------------------- gene scores
// Block = 32 genes x 8 sample lanes, expr sample-major [S][V] as in pcc_zscore_kernel; lab[s] is 0 (good), 1 (poor)
// or anything else (sample in neither group).  cli.tscore: pooled variance with ddof = 1; 0 when the pooled deviation
// is not > 0, and 0 when a group has a single sample (its ddof = 1 std is NaN there, and so is the pooled one).
__global__ void __launch_bounds__(256)
post_tscore_kernel(const float *__restrict__ expr, int32_t S, int32_t V, const uint8_t *__restrict__ lab,
                   float *__restrict__ t) {
    __shared__ double sh[2][8][33];
    __shared__ int shn[2][8][33];
    const int gx = threadIdx.x & 31, sy = threadIdx.x >> 5;
    const int g = blockIdx.x * 32 + gx;
    double s0 = 0.0, s1 = 0.0;
    int n0 = 0, n1 = 0;
    if (g < V)
        for (int s = sy; s < S; s += 8) {
            const uint8_t l = lab[s];
            const double x = (double)expr[(size_t)s * V + g];
            if (l == 0) { s0 += x; ++n0; } else if (l == 1) { s1 += x; ++n1; }
        }
    sh[0][sy][gx] = s0; sh[1][sy][gx] = s1; shn[0][sy][gx] = n0; shn[1][sy][gx] = n1;
    __syncthreads();
    double m0 = 0.0, m1 = 0.0;
    int na = 0, nb = 0;
    for (int k = 0; k < 8; ++k) { m0 += sh[0][k][gx]; m1 += sh[1][k][gx]; na += shn[0][k][gx]; nb += shn[1][k][gx]; }
    m0 /= (double)max(na, 1);
    m1 /= (double)max(nb, 1);
    __syncthreads();
    double q0 = 0.0, q1 = 0.0;
    if (g < V)
        for (int s = sy; s < S; s += 8) {
            const uint8_t l = lab[s];
            const double x = (double)expr[(size_t)s * V + g];
            if (l == 0) q0 += (x - m0) * (x - m0); else if (l == 1) q1 += (x - m1) * (x - m1);
        }
    sh[0][sy][gx] = q0; sh[1][sy][gx] = q1;
    __syncthreads();
    if (sy != 0 || g >= V) return;
    double ss = 0.0;
    for (int k = 0; k < 8; ++k) ss += sh[0][k][gx] + sh[1][k][gx];
    float out = 0.f;
    if (na >= 2 && nb >= 2) {
        const double d1 = sqrt(ss / (double)(na + nb - 2));
        const double d2 = sqrt(1.0 / (double)na + 1.0 / (double)nb);
        if (d1 > 0.0) out = (float)fabs((m0 - m1) / d1 / d2);
    }
    t[g] = out;
}

// One warp per row: out[r] = ||X[r]||_2 (double accumulation).
__global__ void __launch_bounds__(256)
post_row_norms_kernel(const float *__restrict__ X, int64_t V, int32_t D, float *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < V; r += nwarps) {
        double acc = 0.0;
        for (int j = lane; j < D; j += 32) { const double x = (double)__ldg(X + r * D + j); acc += x * x; }
        acc = warp_sum_f64(acc);
        if (lane == 0) out[r] = (float)sqrt(acc);
    }
}

// ---------------------------------------------------------------- "%.6f" formatting
// A finite float32 is m * 2^e with m < 2^24, so N = round_half_even(|x| * 10^6) = round(m * 10^6 * 2^e) with
// P = m * 10^6 < 2^44:
//   e < 0:  N = P >> -e, rounded half to even on the exact remainder (N = 0 once 2^-e > 2 P);
//   e >= 0: N = P << e < 2^148, held in five 32-bit limbs.
// N is printed in base 10^9 chunks (short division of the limbs), with at least 7 digits and '.' before the last
// 6 -- what Python's correctly rounded '%.6f' prints.  The sign is the sign bit (-0.0 and values that round to zero
// from below print "-0.000000"); NaN of either sign prints "nan", infinities "inf" / "-inf".
struct Fmt {
    uint32_t chunk[5];   // base-10^9 digits of N, least significant first
    int n_chunks;        // >= 1
    int digits;          // decimal digits printed (>= 7)
    int kind;            // 0 finite, 1 nan, 2 inf
    bool neg;
};

__device__ __forceinline__ int dec_digits_u32(uint32_t v) {
    int n = 1;
    while (v >= 10u) { v /= 10u; ++n; }
    return n;
}

__device__ void fmt_decompose(float x, Fmt &f) {
    const uint32_t b = __float_as_uint(x);
    const uint32_t E = (b >> 23) & 0xffu, M = b & 0x7fffffu;
    f.neg = (b >> 31) != 0;
    f.kind = 0;
    f.n_chunks = 1;
    f.chunk[0] = 0;
    if (E == 0xffu) {
        f.kind = M ? 1 : 2;
        if (M) f.neg = false;
        f.digits = 0;
        return;
    }
    const uint64_t m = E ? (uint64_t)(M | 0x800000u) : (uint64_t)M;
    const int e = E ? (int)E - 150 : -149;
    const uint64_t P = m * 1000000ull;
    uint32_t limb[5] = {0, 0, 0, 0, 0};
    if (e < 0) {
        const int s = -e;
        uint64_t N = 0;
        if (s < 64) {
            N = P >> s;
            const uint64_t r = P & ((1ull << s) - 1ull), half = 1ull << (s - 1);
            if (r > half || (r == half && (N & 1ull))) ++N;
        }
        limb[0] = (uint32_t)N;
        limb[1] = (uint32_t)(N >> 32);
    } else {
        const int ws = e >> 5, bs = e & 31;
        const uint32_t p0 = (uint32_t)P, p1 = (uint32_t)(P >> 32);
        // (p1:p0) << bs spans three 32-bit words, placed at word ws
        const uint64_t lo = (uint64_t)p0 << bs;
        const uint64_t hi = (uint64_t)p1 << bs;
        const uint32_t w0 = (uint32_t)lo, w1 = (uint32_t)(lo >> 32) | (uint32_t)hi, w2 = (uint32_t)(hi >> 32);
        limb[ws] = w0;
        if (ws + 1 < 5) limb[ws + 1] = w1;
        if (ws + 2 < 5) limb[ws + 2] = w2;
    }
    // base 10^9 by repeated short division (most significant limb first)
    int top = 4;
    while (top > 0 && limb[top] == 0) --top;
    int n = 0;
    for (;;) {
        uint64_t rem = 0;
        for (int i = top; i >= 0; --i) {
            const uint64_t cur = (rem << 32) | limb[i];
            limb[i] = (uint32_t)(cur / 1000000000ull);
            rem = cur % 1000000000ull;
        }
        f.chunk[n++] = (uint32_t)rem;
        while (top > 0 && limb[top] == 0) --top;
        if (top == 0 && limb[0] == 0) break;
    }
    f.n_chunks = n;
    const int d = 9 * (n - 1) + dec_digits_u32(f.chunk[n - 1]);
    f.digits = d < 7 ? 7 : d;
}

// bytes of "\t" + the formatted value
__device__ __forceinline__ int fmt_len(const Fmt &f) {
    if (f.kind == 1) return 4;
    if (f.kind == 2) return 4 + f.neg;
    return 1 + f.neg + f.digits + 1;
}

__device__ void fmt_write(const Fmt &f, char *p) {
    *p++ = '\t';
    if (f.neg) *p++ = '-';
    if (f.kind) {
        p[0] = f.kind == 1 ? 'n' : 'i';
        p[1] = f.kind == 1 ? 'a' : 'n';
        p[2] = f.kind == 1 ? 'n' : 'f';
        return;
    }
    // digits from the least significant; position i (0 = last digit) goes before the '.' when i >= 6
    char *end = p + f.digits + 1;          // one past the last character
    int i = 0;
    for (int c = 0; c < f.n_chunks; ++c) {
        uint32_t v = f.chunk[c];
        const int nd = (c + 1 < f.n_chunks) ? 9 : max(dec_digits_u32(v), f.digits - 9 * c);
        for (int k = 0; k < nd && i < f.digits; ++k, ++i) {
            if (i == 6) *--end = '.';
            *--end = (char)('0' + v % 10u);
            v /= 10u;
        }
    }
}

// One warp per row: bytes of prefix (row's name, nullable) + "\t%.6f" x D + "\n".
__global__ void __launch_bounds__(256)
fmt_row_bytes_kernel(const float *__restrict__ X, int64_t rows, int32_t D, const int64_t *__restrict__ prefix_off,
                     int64_t *__restrict__ row_bytes) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < rows; r += nwarps) {
        uint32_t n = 0;
        for (int j = lane; j < D; j += 32) {
            Fmt f;
            fmt_decompose(__ldg(X + r * D + j), f);
            n += fmt_len(f);
        }
        n = __reduce_add_sync(0xffffffffu, n);
        if (lane == 0) row_bytes[r] = (int64_t)n + 1 + (prefix_off ? prefix_off[r + 1] - prefix_off[r] : 0);
    }
}

// One warp per row: the row's line at out + offsets[r].  Each round of 32 values is placed by a warp scan of their
// lengths.
__global__ void __launch_bounds__(256)
fmt_emit_kernel(const float *__restrict__ X, int64_t rows, int32_t D, const char *__restrict__ prefix,
                const int64_t *__restrict__ prefix_off, const int64_t *__restrict__ offsets, char *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < rows; r += nwarps) {
        char *p = out + offsets[r];
        if (prefix_off) {
            const int64_t a = prefix_off[r], n = prefix_off[r + 1] - a;
            for (int64_t i = lane; i < n; i += 32) p[i] = prefix[a + i];
            p += n;
        }
        for (int j0 = 0; j0 < D; j0 += 32) {
            const int j = j0 + lane;
            Fmt f;
            uint32_t len = 0;
            if (j < D) { fmt_decompose(__ldg(X + r * D + j), f); len = fmt_len(f); }
            const uint32_t incl = warp_inclusive_scan_u32(len, lane);
            if (j < D) fmt_write(f, p + (incl - len));
            p += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) *p = '\n';
    }
}

static int warp_grid(int64_t rows, const DeviceProps &dp) {
    const int64_t want = (rows + 7) / 8;
    return (int)max((int64_t)1, min(want, (int64_t)dp.sm_count * 16));
}

}  // namespace g2v

using namespace g2v;

// ---------------------------------------------------------------- C ABI
extern "C" size_t g2v_kmeans_workspace_bytes(int32_t V, int32_t D, int32_t K) {
    if (V <= 0 || D <= 0 || K <= 0) return 0;
    DeviceProps dp;
    const int sms = device_props(&dp) ? 160 : dp.sm_count;
    const size_t nb = (size_t)sms * 2;
    const size_t col = (size_t)sms * 2 * 2 * D * sizeof(double);
    const size_t lloyd = nb * K * D * sizeof(double) + nb * (K + 1) * sizeof(int64_t) + (size_t)K * D * sizeof(double);
    return (col > lloyd ? col : lloyd) + 256;
}

static int kmeans_blocks(int32_t V, const DeviceProps &dp) {
    return (int)max(1, min((V + 7) / 8, dp.sm_count * 2));
}

extern "C" int g2v_kmeans_center(const float *X, int32_t V, int32_t D, float *Xc, float *mean, double *var,
                                 void *workspace, void *stream) {
    G2V_REQUIRE(X && Xc && mean && var && workspace && V > 0 && D > 0, "g2v_kmeans_center: bad arguments");
    DeviceProps dp;
    if (device_props(&dp)) return 1;
    cudaStream_t st = (cudaStream_t)stream;
    const int ny = max(1, min(V, dp.sm_count * 2));
    const dim3 grid((D + 127) / 128, ny);
    double *part = (double *)workspace;
    kmeans_colsum_kernel<<<grid, 128, 0, st>>>(X, V, D, nullptr, nullptr, part);
    kmeans_colfin_kernel<<<(D + 127) / 128, 128, 0, st>>>(part, ny, V, D, mean, nullptr);
    kmeans_colsum_kernel<<<grid, 128, 0, st>>>(X, V, D, mean, Xc, part);
    kmeans_colfin_kernel<<<(D + 127) / 128, 128, 0, st>>>(part, ny, V, D, nullptr, var);
    G2V_CUDA_OK(cudaGetLastError());
    count_launch(4);
    return 0;
}

extern "C" int g2v_kmeans_dist(const float *X, int32_t V, int32_t D, const int64_t *cand_host, int32_t n_cand,
                               const float *closest, float *out, void *stream) {
    G2V_REQUIRE(X && cand_host && out && V > 0 && D > 0 && n_cand >= 1 && n_cand <= kMaxCand,
                "g2v_kmeans_dist: bad arguments (1 <= n_cand <= %d)", kMaxCand);
    CandIds c;
    for (int k = 0; k < kMaxCand; ++k) c.id[k] = 0;
    for (int k = 0; k < n_cand; ++k) {
        G2V_REQUIRE(cand_host[k] >= 0 && cand_host[k] < V, "g2v_kmeans_dist: candidate %lld out of range",
                    (long long)cand_host[k]);
        c.id[k] = cand_host[k];
    }
    DeviceProps dp;
    if (device_props(&dp)) return 1;
    kmeans_dist_kernel<<<warp_grid(V, dp), 256, 0, (cudaStream_t)stream>>>(X, V, D, c, n_cand, closest, out);
    G2V_CUDA_OK(cudaGetLastError());
    count_launch();
    return 0;
}

extern "C" int g2v_kmeans_lloyd_step(const float *X, int32_t V, int32_t D, int32_t K, const float *centres,
                                     float *centres_new, const int32_t *labels_old, int32_t *labels, double *status,
                                     void *workspace, void *stream) {
    G2V_REQUIRE(X && centres && labels && V > 0 && D > 0 && D <= kMaxKmD && K >= 1 && K <= kMaxK,
                "g2v_kmeans_lloyd_step: bad arguments (1 <= D <= %d, 1 <= K <= %d)", kMaxKmD, kMaxK);
    G2V_REQUIRE(!centres_new || (status && workspace), "g2v_kmeans_lloyd_step: centres_new needs status and workspace");
    DeviceProps dp;
    if (device_props(&dp)) return 1;
    cudaStream_t st = (cudaStream_t)stream;
    const int nb = kmeans_blocks(V, dp);
    const size_t smem = (size_t)8 * D * sizeof(float);
    if (!centres_new) {
        kmeans_assign_kernel<<<nb, 256, smem, st>>>(X, V, D, K, centres, labels_old, labels, nullptr, nullptr);
        G2V_CUDA_OK(cudaGetLastError());
        count_launch();
        return 0;
    }
    double *partial = (double *)workspace;
    int64_t *counts = (int64_t *)(partial + (size_t)nb * K * D);
    double *shift_sq = (double *)(counts + (size_t)nb * (K + 1));
    kmeans_assign_kernel<<<nb, 256, smem, st>>>(X, V, D, K, centres, labels_old, labels, partial, counts);
    kmeans_update_kernel<<<dim3((D + 31) / 32, K), 256, 0, st>>>(partial, counts, nb, D, K, centres, centres_new,
                                                                   shift_sq);
    kmeans_status_kernel<<<1, 256, 0, st>>>(counts, nb, D, K, shift_sq, status);
    G2V_CUDA_OK(cudaGetLastError());
    count_launch(3);
    return 0;
}

extern "C" int g2v_post_tscores(const float *expr, int32_t S, int32_t V, const uint8_t *label, float *t, void *stream) {
    G2V_REQUIRE(expr && label && t && S > 0 && V > 0, "g2v_post_tscores: bad arguments");
    DeviceProps dp;
    if (device_props(&dp)) return 1;
    post_tscore_kernel<<<(V + 31) / 32, 256, 0, (cudaStream_t)stream>>>(expr, S, V, label, t);
    G2V_CUDA_OK(cudaGetLastError());
    count_launch();
    return 0;
}

extern "C" int g2v_post_row_norms(const float *X, int64_t V, int32_t D, float *out, void *stream) {
    G2V_REQUIRE(X && out && V > 0 && D > 0, "g2v_post_row_norms: bad arguments");
    DeviceProps dp;
    if (device_props(&dp)) return 1;
    post_row_norms_kernel<<<warp_grid(V, dp), 256, 0, (cudaStream_t)stream>>>(X, V, D, out);
    G2V_CUDA_OK(cudaGetLastError());
    count_launch();
    return 0;
}

extern "C" int g2v_fmt_row_bytes(const float *X, int64_t rows, int32_t D, const int64_t *prefix_off,
                                 int64_t *row_bytes, void *stream) {
    G2V_REQUIRE(X && row_bytes && rows >= 0 && D > 0, "g2v_fmt_row_bytes: bad arguments");
    if (rows == 0) return 0;
    DeviceProps dp;
    if (device_props(&dp)) return 1;
    fmt_row_bytes_kernel<<<warp_grid(rows, dp), 256, 0, (cudaStream_t)stream>>>(X, rows, D, prefix_off, row_bytes);
    G2V_CUDA_OK(cudaGetLastError());
    count_launch();
    return 0;
}

extern "C" int g2v_fmt_emit(const float *X, int64_t rows, int32_t D, const char *prefix, const int64_t *prefix_off,
                            const int64_t *offsets, char *out, void *stream) {
    G2V_REQUIRE(X && offsets && out && rows >= 0 && D > 0 && (!prefix_off || prefix),
                "g2v_fmt_emit: bad arguments");
    if (rows == 0) return 0;
    DeviceProps dp;
    if (device_props(&dp)) return 1;
    fmt_emit_kernel<<<warp_grid(rows, dp), 256, 0, (cudaStream_t)stream>>>(X, rows, D, prefix, prefix_off, offsets, out);
    G2V_CUDA_OK(cudaGetLastError());
    count_launch();
    return 0;
}
