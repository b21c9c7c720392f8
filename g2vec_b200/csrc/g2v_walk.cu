// g2v_walk.cu -- HOT PATH 1: self-avoiding weighted random walks on CSR, one warp per walker.
//
// Replaces generate_pathSet / generate_randomPath (/root/reference/G2Vec.py:324-352).
// Per step of a walker at node `cur` (G2Vec.py:331-344):
//     path.append(cur)                                    -> path[] in shared memory
//     prob = adjMat[cur]; prob[path] = 0                  -> CSR row, visited test per neighbour
//     if prob.sum() > 0: cur = choice(p = prob / sum)     -> integer inverse CDF, one Philox draw
//     else: break
// and at the end `path = tuple(sorted(path))` (:345) -- optionally fused here (CANON): the path is already
// in shared memory, so the warp sorts it there (bitonic), writes the sorted row and its 64-bit key, and the
// separate canonicalise launch with its re-read of the rows disappears.
//
// Graph layouts in HBM (template LAYOUT):
//   LAY_CSR  rowptr int32 [V+1], col int32 [E], qw uint32 [E]          -- the plain C-ABI arrays (g2v_walk_launch)
//   LAY_E8   rows int2 {begin,end} [V], edges uint2 {col, qw}          -- rows start at even indices (an odd row is
//            followed by one {0, 0} pair: weight 0 masks itself), so one LDG.128 brings TWO neighbours per lane
//   LAY_E4   rows int2 [V], edges uint32 = col | (qw-32768) << 16       -- V <= 65535 and 32768 <= qw <= 65536
//            (the |PCC| in [0.5, 1] range of the reference's edges, G2Vec.py:389): one LDG.64 brings TWO
//            neighbours per lane, 64 per warp request.  Every row starts at an even index and an odd row is
//            followed by one SENTINEL word (col = V, a node that does not exist): with the bitmap visited set, bit V
//            is permanently "visited", so the pad word, and the lanes beyond the row (whose register default is the
//            sentinel word), are masked by the visited test itself -- no validity compares on the hot path
// g2v_walk_prepare packs the CSR once per graph (the graph is static across all repetitions).
//
// Per warp in shared memory: the path (written back once, coalesced) and the visited set -- a V-bit bitmap
// (one LDS per neighbour) while 8 warps' bitmaps fit in 56 KB, otherwise an open-addressing hash set of
// >= 3L slots whose size is independent of V (200k-node graphs keep full occupancy).
// Rows of at most one chunk (32 or 64 neighbours) take the short path: load, visited test, ONE warp scan that
// yields both the total and the prefix sums, draw, ballot.  Longer rows keep KC chunks in registers between the
// two passes (per-chunk totals with REDUX.SUM, then one scan inside the selected chunk) and re-read the tail.
// Philox draws are evaluated 32 steps at a time, one step per lane.  Walkers are handed out by an atomic
// ticket so that warps whose walker dead-ends early (62 % of ex_* start nodes have no out-edge) immediately
// take the next one.
//
// Integer arithmetic only on the selection path => bit-exact against oracle/g2v_oracle.c for any scan
// order:  T = sum of unvisited qw (uint64), r = mulhi64(x, T), first inclusive prefix > r.
#include <stdlib.h>
#include <string.h>

#include "g2v_common.cuh"

namespace g2v {

constexpr int kWalkWarps = 8;   // warps per CTA
constexpr int kKC = 2;          // neighbour chunks kept in registers on the long-row path
// resident CTAs per SM the kernels are compiled for: 6 (register cap 40) for the bitmap variants, 8 (cap 32) for the
// hash-set variants -- measured (profiles/r2/tune_walk_minb_r2l.txt): syn10k 1.97 ms at 6 vs 2.00 ms at 8, stress200k
// (hash set, V = 200k) 25.0 ms at 6 vs 22.0 ms at 8
#ifndef G2V_WALK_MINB_BITMAP
#define G2V_WALK_MINB_BITMAP 6
#endif
#ifndef G2V_WALK_MINB_HASH
#define G2V_WALK_MINB_HASH 8
#endif

enum { LAY_CSR = 0, LAY_E8 = 1, LAY_E4 = 2 };

// The walker's state is warp-uniform, so inside the step loop every lane stores the SAME value to the SAME shared
// word (path append, visited insert) and later reads what it stored itself: no divergence and no warp barrier on
// the instruction-bound path.  compute-sanitizer racecheck reports these same-value stores as warnings (never as
// errors).  -DG2V_WALK_STRICT_SYNC builds the formally race-free form -- lane 0 stores, __syncwarp() before the
// warp reads -- which racecheck passes with 0 hazards and which is 15 % more instructions / 20 % slower
// (profiles/r2/walk_strict_sync_r2x.txt); both forms give bit-identical walks.
#ifdef G2V_WALK_STRICT_SYNC
#define G2V_WALK_ONE_WRITER if (lane == 0)
#define G2V_WALK_STEP_SYNC() __syncwarp()
#else
#define G2V_WALK_ONE_WRITER
#define G2V_WALK_STEP_SYNC()
#endif

__device__ __forceinline__ uint32_t hash_slot(int32_t c, int shift) {
    return ((uint32_t)c * 2654435761u) >> shift;
}

// Returns q if node c is NOT in the visited set, else 0.  `hs` indexes the dynamic shared array (kept as
// an integer offset so that every access is a plain LDS/STS with a register offset).
extern __shared__ int32_t g2v_walk_smem[];
template <bool BITMAP>
__device__ __forceinline__ uint32_t unvisited_weight(int hs, uint32_t mask, int shift, int32_t c, uint32_t q) {
    if (BITMAP) {
        const uint32_t bit = ((uint32_t)g2v_walk_smem[hs + (c >> 5)] >> (c & 31)) & 1u;
        return q & (bit - 1u);                            // bit = 1 -> 0, bit = 0 -> q
    }
    uint32_t i = hash_slot(c, shift);
    while (true) {
        const int32_t x = g2v_walk_smem[hs + i];
        if (x == c) return 0u;
        if (x < 0) return q;
        i = (i + 1) & mask;
    }
}

struct WalkGraphPtrs {
    const int32_t *rows;    // LAY_CSR: rowptr [V+1];  else int2 {begin, end} [V]
    const void *edges;      // LAY_CSR: col [E];  LAY_E8: uint2 [E];  LAY_E4: uint32 [E] (+1 pad)
    const uint32_t *qw;     // LAY_CSR only
};

// One chunk of a row: lane's neighbours jb + lane*EPL + {0 .. EPL-1}, masked weights (0 = outside [b, e) or
// already visited) and node ids.  LAY_E4: jb is even (the caller aligns the first chunk down), so the pair
// is one aligned 8-byte load (rows start at even indices; the word after an odd row is a sentinel).
template <int LAYOUT, bool BITMAP>
__device__ __forceinline__ void load_chunk(const WalkGraphPtrs &g, int32_t jb, int32_t b, int32_t e, int lane, int hs,
                                           uint32_t hmask, int hshift, uint32_t sent, int32_t &c0, int32_t &c1,
                                           uint32_t &q0, uint32_t &q1) {
    (void)b;
    if (LAYOUT == LAY_E4) {
        const int32_t j = jb + 2 * lane;                                        // even: rows start at even indices
        uint2 w = make_uint2(sent, sent);                                       // lanes beyond the row: sentinel word
        // predicated load that keeps the register default (a plain `if` makes ptxas branch around the load)
        asm("{ .reg .pred p; setp.lt.s32 p, %2, %3; @p ld.global.nc.v2.u32 {%0, %1}, [%4]; }"
                     : "+r"(w.x), "+r"(w.y)
                     : "r"(j), "r"(e), "l"(reinterpret_cast<const uint32_t *>(g.edges) + j));
        c0 = (int32_t)(w.x & 0xffffu); c1 = (int32_t)(w.y & 0xffffu);
        uint32_t a0 = (w.x >> 16) + 32768u, a1 = (w.y >> 16) + 32768u;
        if (!BITMAP) {                          // the hash set knows no sentinel: explicit validity
            a0 = (j < e) ? a0 : 0u;
            a1 = (j + 1 < e) ? a1 : 0u;
        }
        q0 = unvisited_weight<BITMAP>(hs, hmask, hshift, c0, a0);               // bitmap: bit V is always set
        q1 = unvisited_weight<BITMAP>(hs, hmask, hshift, c1, a1);
    } else if (LAYOUT == LAY_E8) {
        const int32_t j = jb + 2 * lane;                                        // even: 16-byte aligned pair of {col, qw}
        uint4 w = make_uint4(0u, 0u, 0u, 0u);                                   // lanes beyond the row: weight 0
        if (j < e) w = __ldg(reinterpret_cast<const uint4 *>(g.edges) + (j >> 1));
        c0 = (int32_t)w.x; c1 = (int32_t)w.z;
        q0 = unvisited_weight<BITMAP>(hs, hmask, hshift, c0, w.y);
        q1 = unvisited_weight<BITMAP>(hs, hmask, hshift, c1, (j + 1 < e) ? w.w : 0u);   // (the pad pair has weight 0 too)
    } else {
        const int32_t j = jb + lane;
        uint32_t a0 = 0u;
        c0 = 0;
        if (j < e) {
            c0 = __ldg(reinterpret_cast<const int32_t *>(g.edges) + j);
            a0 = __ldg(g.qw + j);
        }
        q0 = unvisited_weight<BITMAP>(hs, hmask, hshift, c0, a0);
        c1 = 0; q1 = 0u;
    }
}

// Inclusive warp scan of p; the first lane whose prefix exceeds `rem` holds the chosen neighbour.
template <int EPL>
__device__ __forceinline__ int32_t pick_in_chunk(uint32_t p, uint32_t q0, int32_t c0, int32_t c1, uint32_t incl,
                                                 uint32_t rem) {
    const unsigned hit = __ballot_sync(0xffffffffu, incl > rem);
    const int32_t sel = (EPL == 2 && !(incl - p + q0 > rem)) ? c1 : c0;
    return __shfl_sync(0xffffffffu, sel, __ffs(hit) - 1);
}

template <bool BITMAP, int LAYOUT, bool CANON>
__global__ void __launch_bounds__(kWalkWarps * 32, BITMAP ? G2V_WALK_MINB_BITMAP : G2V_WALK_MINB_HASH)
walk_kernel(const WalkGraphPtrs g, int32_t V, int32_t L, int32_t Lpad, int32_t H, int32_t hshift, uint64_t seed,
            uint32_t group, int64_t walker_begin, int64_t n_walkers, int64_t walker_stride,
            int32_t *__restrict__ out_nodes, int32_t *__restrict__ out_len, unsigned long long *__restrict__ out_key,
            unsigned long long *__restrict__ ticket) {
    int32_t *const smem = g2v_walk_smem;
    constexpr int EPL = LAYOUT == LAY_CSR ? 1 : 2;      // neighbours per lane per chunk
    constexpr int CH = 32 * EPL;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int path = warp * (Lpad + H);                  // offsets into smem (ints), not pointers
    const int hs = path + Lpad;
    const uint32_t hmask = (uint32_t)H - 1u;

    constexpr bool SENT = BITMAP && LAYOUT == LAY_E4;   // bit V of the bitmap = a node that is always "visited"
    const uint32_t sent = (uint32_t)V;                   // sentinel edge word: col = V, weight field 0
    const int sw = V >> 5;
    const int32_t sbit = SENT ? (int32_t)(1u << (V & 31)) : 0;
    for (int i = lane; i < H; i += 32) smem[hs + i] = BITMAP ? ((SENT && i == sw) ? sbit : 0) : -1;
    __syncwarp();

    while (true) {
        // ------------------------------------------------------------------ take the next walker
        unsigned long long t = 0;
        if (lane == 0) t = atomicAdd(ticket, 1ull);
        t = __shfl_sync(0xffffffffu, t, 0);
        if ((int64_t)t >= n_walkers) break;
        const int64_t w = walker_begin + (int64_t)t * walker_stride;
        const uint64_t subseq = ((uint64_t)group << 40) + (uint64_t)w;
        int32_t cur = (int32_t)(w % V);
        int32_t n = 0;                                   // nodes appended = step index + 1
        uint32_t dlo = 0, dhi = 0;                       // lane holds the draw of step (s & ~31) + lane
        bool dirty = false;

        while (true) {
            G2V_WALK_ONE_WRITER smem[path + n] = cur;    // read back only after the walk (epilogue)
            const int32_t s = n++;
            if (s == L - 1) break;                       // the L-th node is appended, never expanded
            int32_t b, e;
            if (LAYOUT == LAY_CSR) {
                b = __ldg(g.rows + cur); e = __ldg(g.rows + cur + 1);
            } else {
                const int2 be = __ldg(reinterpret_cast<const int2 *>(g.rows) + cur);
                b = be.x; e = be.y;
            }
            if (b == e) break;                           // no out-edges: dead end
            if (BITMAP) {                                // visited.insert(cur)
                G2V_WALK_ONE_WRITER smem[hs + (cur >> 5)] |= (1 << (cur & 31));
            } else {
                uint32_t i = hash_slot(cur, hshift);
                while (smem[hs + i] >= 0) i = (i + 1) & hmask;
                __syncwarp();                            // every lane has found the free slot before it is filled
                G2V_WALK_ONE_WRITER smem[hs + i] = cur;
            }
            G2V_WALK_STEP_SYNC();
            dirty = true;
            if ((s & 31) == 0) {                         // 32 steps of 64-bit Philox draws at once, one per lane
                const uint64_t d = draw64(seed, subseq, (uint32_t)(s + lane));
                dlo = (uint32_t)d; dhi = (uint32_t)(d >> 32);
            }
            const uint32_t xlo = __shfl_sync(0xffffffffu, dlo, s & 31), xhi = __shfl_sync(0xffffffffu, dhi, s & 31);

            const int32_t jb0 = b;                       // (packed rows start at even indices)
            int32_t nxt;
            if (e - jb0 <= CH) {
                // ---- short row: one chunk.  One scan gives the total (lane 31) and the prefix sums.
                int32_t c0, c1; uint32_t q0, q1;
                load_chunk<LAYOUT, BITMAP>(g, jb0, b, e, lane, hs, hmask, hshift, sent, c0, c1, q0, q1);
                const uint32_t p = q0 + q1;
                const uint32_t incl = warp_inclusive_scan_u32(p, lane);
                const uint32_t T = __shfl_sync(0xffffffffu, incl, 31);            // <= 64 * 2^24 < 2^32
                if (T == 0) break;                       // every neighbour already visited
                // r = floor(x*T / 2^64) with T < 2^32: two 32x32 multiplies instead of a 64x64 high multiply
                const unsigned long long lo = (unsigned long long)xlo * T;
                const uint32_t rem = (uint32_t)(((unsigned long long)xhi * T + (lo >> 32)) >> 32);
                nxt = pick_in_chunk<EPL>(p, q0, c0, c1, incl, rem);
            } else {
                // ---- long row: pass 1 = per-chunk totals (first kKC chunks stay in registers), pass 2 = select
                uint32_t P[kKC], Q0[kKC], tot[kKC];
                int32_t C0[kKC], C1[kKC];
                unsigned long long T = 0;
#pragma unroll
                for (int k = 0; k < kKC; ++k) {
                    P[k] = 0; Q0[k] = 0; tot[k] = 0; C0[k] = 0; C1[k] = 0;
                    if (jb0 + k * CH < e) {              // warp-uniform
                        uint32_t q1;
                        load_chunk<LAYOUT, BITMAP>(g, jb0 + k * CH, b, e, lane, hs, hmask, hshift, sent, C0[k], C1[k], Q0[k], q1);
                        P[k] = Q0[k] + q1;
                        tot[k] = __reduce_add_sync(0xffffffffu, P[k]);
                        T += tot[k];
                    }
                }
                for (int32_t jb = jb0 + kKC * CH; jb < e; jb += CH) {
                    int32_t c0, c1; uint32_t q0, q1;
                    load_chunk<LAYOUT, BITMAP>(g, jb, b, e, lane, hs, hmask, hshift, sent, c0, c1, q0, q1);
                    T += __reduce_add_sync(0xffffffffu, q0 + q1);
                }
                if (T == 0) break;
                unsigned long long rem = __umul64hi(((unsigned long long)xhi << 32) | xlo, T);
                nxt = -1;
                bool found = false;
#pragma unroll
                for (int k = 0; k < kKC; ++k) {
                    if (!found && jb0 + k * CH < e) {
                        if (rem < (unsigned long long)tot[k]) {
                            const uint32_t incl = warp_inclusive_scan_u32(P[k], lane);
                            nxt = pick_in_chunk<EPL>(P[k], Q0[k], C0[k], C1[k], incl, (uint32_t)rem);
                            found = true;
                        } else {
                            rem -= tot[k];
                        }
                    }
                }
                for (int32_t jb = jb0 + kKC * CH; !found && jb < e; jb += CH) {
                    int32_t c0, c1; uint32_t q0, q1;
                    load_chunk<LAYOUT, BITMAP>(g, jb, b, e, lane, hs, hmask, hshift, sent, c0, c1, q0, q1);
                    const uint32_t p = q0 + q1;
                    const uint32_t ct = __reduce_add_sync(0xffffffffu, p);
                    if (rem < (unsigned long long)ct) {
                        const uint32_t incl = warp_inclusive_scan_u32(p, lane);
                        nxt = pick_in_chunk<EPL>(p, q0, c0, c1, incl, (uint32_t)rem);
                        found = true;
                    } else {
                        rem -= ct;
                    }
                }
            }
            cur = nxt;
        }

        // ---------------------------------------------------------------- walk finished: n nodes in smem
        G2V_WALK_STEP_SYNC();                            // (strict build: lane 0's path stores become visible)
        int32_t *row = out_nodes + (size_t)t * (size_t)L;
        if (!CANON) {
            for (int i = lane; i < L; i += 32) row[i] = (i < n) ? smem[path + i] : -1;     // visit order
        } else if (BITMAP) {
            // tuple(sorted(path)) (G2Vec.py:345) read off the visited bitmap: the set bits in index order ARE the
            // sorted path.  Lane l owns the words [l*B, (l+1)*B): count, one warp scan for its first output
            // position, then emit its bits in order (and clear the words: the next walker starts from zero).
            const int32_t lastn = smem[path + n - 1];            // the final node is appended but never inserted
            G2V_WALK_ONE_WRITER smem[hs + (lastn >> 5)] |= (1 << (lastn & 31));
            __syncwarp();
            const int B = (H + 31) >> 5, w0 = lane * B, w1 = min(H, w0 + B);
            uint32_t cnt = 0;
            for (int wi = w0; wi < w1; ++wi) cnt += __popc((uint32_t)smem[hs + wi] & ~(uint32_t)((SENT && wi == sw) ? sbit : 0));
            uint32_t pos = warp_inclusive_scan_u32(cnt, lane) - cnt;
            uint64_t h = 0;
            for (int wi = w0; wi < w1; ++wi) {
                const int32_t keepbit = (SENT && wi == sw) ? sbit : 0;
                uint32_t bits = (uint32_t)smem[hs + wi] & ~(uint32_t)keepbit;
                if (bits) smem[hs + wi] = keepbit;
                while (bits) {
                    const int32_t v = wi * 32 + (__ffs(bits) - 1);
                    bits &= bits - 1;
                    row[pos] = v;
                    h += path_key_term(v, (int)pos);
                    ++pos;
                }
            }
            for (int i = n + lane; i < L; i += 32) row[i] = kPathPad;
            h = warp_sum_u64(h);
            if (lane == 0) out_key[t] = path_key_finish(h);
            dirty = false;                                       // already cleared
        } else {
            // tuple(sorted(path)) (G2Vec.py:345): bitonic network over the next power of two, INT32_MAX padding
            int P2 = 1;
            while (P2 < n) P2 <<= 1;
            if (n > 1) {
                for (int i = n + lane; i < P2; i += 32) smem[path + i] = kPathPad;
                __syncwarp();
                for (int k = 2; k <= P2; k <<= 1)
                    for (int j = k >> 1; j > 0; j >>= 1) {
                        for (int x = lane; x < (P2 >> 1); x += 32) {
                            const int i = ((x / j) * 2 * j) + (x % j), l = i + j;
                            const bool up = (i & k) == 0;
                            const int32_t a = smem[path + i], c = smem[path + l];
                            if ((a > c) == up) { smem[path + i] = c; smem[path + l] = a; }
                        }
                        __syncwarp();
                    }
            }
            uint64_t h = 0;
            for (int i = lane; i < L; i += 32) {
                const int32_t v = (i < n) ? smem[path + i] : kPathPad;
                row[i] = v;
                if (i < n) h += path_key_term(v, i);
            }
            h = warp_sum_u64(h);
            if (lane == 0) out_key[t] = path_key_finish(h);
        }
        if (lane == 0) out_len[t] = n;
        if (dirty) {
            if (BITMAP) {                                // every lane resets the words it owns (one writer per word)
                __syncwarp();
                const int B = (H + 31) >> 5, w0 = lane * B, w1 = min(H, w0 + B);
                for (int wi = w0; wi < w1; ++wi)
                    if (smem[hs + wi] != 0) smem[hs + wi] = (SENT && wi == sw) ? sbit : 0;
            } else {
                for (int i = lane; i < H; i += 32) smem[hs + i] = -1;
            }
        }
        __syncwarp();
    }
}

// ---- two walkers per warp (packed edges + bitmap): walk_pair_kernel -----------------------------------------
// The one-walker kernel is bound by instruction issue, and most of its instructions do the same work whether 32 or
// 16 lanes take part.  Here each half-warp ("tile") owns a walker and every lane loads FOUR packed neighbours with one
// LDG.128 (rows are 16-byte aligned and sentinel-padded), so a tile still covers 64 neighbours per request and one
// instruction stream advances two walkers.  The loop is flat -- one iteration = one step of both tiles, re-converged
// by __syncwarp() -- and a tile that finishes its walk runs its epilogue / fetches the next ticket while the other
// waits, so the tiles stay in lock step for the rest of the kernel.  All warp primitives use the tile's lane mask.
// Same arithmetic as walk_kernel (integer inverse CDF, the walker's own Philox stream): bit-identical output.
__device__ __forceinline__ uint32_t tile_inclusive_scan_u32(uint32_t v, unsigned tmask) {
    // 16-lane segments: c = ((32 - 16) << 8): shfl.up clamps at the segment start and p says "source exists"
#pragma unroll
    for (int o = 1; o < 16; o <<= 1)
        asm volatile("{ .reg .pred p; .reg .u32 t; shfl.sync.up.b32 t|p, %0, %1, 0x1000, %2; @p add.u32 %0, %0, t; }"
                     : "+r"(v) : "r"(o), "r"(tmask));
    return v;
}

// full-mask 16-lane-segment scan: both tiles execute it together (converged), each within its own half
__device__ __forceinline__ uint32_t halfwarp_inclusive_scan_u32(uint32_t v) {
#pragma unroll
    for (int o = 1; o < 16; o <<= 1)
        asm volatile("{ .reg .pred p; .reg .u32 t; shfl.sync.up.b32 t|p, %0, %1, 0x1000, 0xffffffff; @p add.u32 %0, %0, t; }"
                     : "+r"(v) : "r"(o));
    return v;
}

// four packed neighbours of one lane: node ids + masked weights (sentinel / visited -> 0)
struct Quad { uint32_t c0, c1, c2, c3, q0, q1, q2, q3; };
__device__ __forceinline__ Quad load_quad(const uint4 *__restrict__ e4, int32_t j, int32_t e, bool on, uint32_t sent, int hs) {
    uint4 w = make_uint4(sent, sent, sent, sent);
    if (on && j < e) w = __ldg(e4 + (j >> 2));
    Quad r;
    r.c0 = w.x & 0xffffu; r.c1 = w.y & 0xffffu; r.c2 = w.z & 0xffffu; r.c3 = w.w & 0xffffu;
    r.q0 = unvisited_weight<true>(hs, 0u, 0, (int32_t)r.c0, (w.x >> 16) + 32768u);
    r.q1 = unvisited_weight<true>(hs, 0u, 0, (int32_t)r.c1, (w.y >> 16) + 32768u);
    r.q2 = unvisited_weight<true>(hs, 0u, 0, (int32_t)r.c2, (w.z >> 16) + 32768u);
    r.q3 = unvisited_weight<true>(hs, 0u, 0, (int32_t)r.c3, (w.w >> 16) + 32768u);
    return r;
}

template <bool CANON>
__global__ void __launch_bounds__(kWalkWarps * 32, 5)
walk_pair_kernel(const WalkGraphPtrs g, int32_t V, int32_t L, int32_t Lpad, int32_t H, uint64_t seed, uint32_t group,
                 int64_t walker_begin, int64_t n_walkers, int64_t walker_stride, int32_t *__restrict__ out_nodes,
                 int32_t *__restrict__ out_len, unsigned long long *__restrict__ out_key,
                 unsigned long long *__restrict__ ticket) {
    int32_t *const smem = g2v_walk_smem;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tile = lane >> 4, tl = lane & 15, tbase = tile << 4;
    const unsigned tmask = 0xffffu << tbase;
    const int path = (warp * 2 + tile) * (Lpad + H);
    const int hs = path + Lpad;
    const uint32_t sent = (uint32_t)V;
    const int sw = V >> 5;
    const int32_t sbit = (int32_t)(1u << (V & 31));
    const uint4 *__restrict__ e4 = reinterpret_cast<const uint4 *>(g.edges);
    for (int i = tl; i < H; i += 16) smem[hs + i] = (i == sw) ? sbit : 0;
    __syncwarp();

    bool have = false, done = false;
    unsigned long long t = 0;
    uint64_t subseq = 0;
    int32_t cur = 0, n = 0;
    uint32_t dlo = 0, dhi = 0;                           // lane tl holds the draw of step (s & ~15) + tl

    // Everything on the common path is executed by all 32 lanes together with full-mask primitives working inside
    // 16-lane segments; a tile without work carries sentinel data through it.  Only the per-walk epilogue, the Philox
    // refill and rows longer than 64 neighbours are tile-divergent sections.
    while (true) {
        const bool need = !have && !done;                // take the next walker (rare: once per walk)
        if (__any_sync(0xffffffffu, need)) {
            unsigned long long tk = 0;
            if (need && tl == 0) tk = atomicAdd(ticket, 1ull);
            tk = __shfl_sync(0xffffffffu, tk, tbase);
            if (need) {
                if ((int64_t)tk >= n_walkers) {
                    done = true;
                } else {
                    t = tk;
                    const int64_t w = walker_begin + (int64_t)tk * walker_stride;
                    subseq = ((uint64_t)group << 40) + (uint64_t)w;
                    cur = (int32_t)(w % V);
                    n = 0; have = true;
                }
            }
            if (__all_sync(0xffffffffu, done)) break;
        }

        // ------------------------------------------------------------------ one step of both tiles' walkers
        const int32_t s = n;
        if (have) { smem[path + n] = cur; ++n; }         // same value from every lane of the tile
        bool end = have && (s == L - 1);                 // the L-th node is appended, never expanded
        bool expand = have && !end;
        int32_t b = 0, e = 0;
        if (expand) {
            const int2 be = __ldg(reinterpret_cast<const int2 *>(g.rows) + cur);
            b = be.x; e = be.y;
            if (b == e) { end = true; expand = false; }  // no out-edges: dead end
        }
        if (expand) {
            smem[hs + (cur >> 5)] |= (1 << (cur & 31));  // visited.insert(cur)
            if ((s & 15) == 0) {                         // 16 steps of 64-bit Philox draws at once, one per lane
                const uint64_t d = draw64(seed, subseq, (uint32_t)(s + tl));
                dlo = (uint32_t)d; dhi = (uint32_t)(d >> 32);
            }
        }
        const int src = tbase + (s & 15);
        const uint32_t xlo = __shfl_sync(0xffffffffu, dlo, src), xhi = __shfl_sync(0xffffffffu, dhi, src);
        Quad q = load_quad(e4, b + 4 * tl, e, expand, sent, hs);
        uint32_t p = q.q0 + q.q1 + q.q2 + q.q3;
        uint32_t incl, r32;
        bool dead = false;
        if (__any_sync(0xffffffffu, expand && e - b > 64)) {
            // ---- a row longer than 64 neighbours in (at least) one tile: tile-divergent two-pass walk over its chunks
            incl = 0; r32 = 0;
            if (expand) {
                unsigned long long T = __reduce_add_sync(tmask, p);
                for (int32_t jb = b + 64; jb < e; jb += 64) {
                    const Quad x = load_quad(e4, jb + 4 * tl, e, true, sent, hs);
                    T += __reduce_add_sync(tmask, x.q0 + x.q1 + x.q2 + x.q3);
                }
                if (T == 0) {
                    dead = true;
                } else {
                    unsigned long long rem = __umul64hi(((unsigned long long)xhi << 32) | xlo, T);
                    int32_t jb = b;
                    while (true) {
                        const uint32_t ct = __reduce_add_sync(tmask, p);
                        if (rem < (unsigned long long)ct) break;
                        rem -= ct;
                        jb += 64;
                        q = load_quad(e4, jb + 4 * tl, e, true, sent, hs);
                        p = q.q0 + q.q1 + q.q2 + q.q3;
                    }
                    r32 = (uint32_t)rem;
                }
            }
            __syncwarp();
            incl = halfwarp_inclusive_scan_u32(p);
        } else {
            incl = halfwarp_inclusive_scan_u32(p);
            const uint32_t T32 = __shfl_sync(0xffffffffu, incl, tbase + 15);      // <= 64 * 2^16
            dead = expand && T32 == 0;                   // every neighbour already visited
            const unsigned long long lo = (unsigned long long)xlo * T32;
            r32 = (uint32_t)(((unsigned long long)xhi * T32 + (lo >> 32)) >> 32);
        }
        const unsigned hit = (__ballot_sync(0xffffffffu, incl > r32) >> tbase) & 0xffffu;
        const uint32_t before = incl - p;                // weight in front of this lane's four neighbours
        const uint32_t sel = (before + q.q0 > r32) ? q.c0
                           : (before + q.q0 + q.q1 > r32) ? q.c1
                           : (before + q.q0 + q.q1 + q.q2 > r32) ? q.c2 : q.c3;
        const int32_t nxt = (int32_t)__shfl_sync(0xffffffffu, sel, tbase + (hit ? __ffs(hit) - 1 : 0));
        if (dead) { end = true; expand = false; }
        if (expand) cur = nxt;

        if (end) {                                       // ---- walk finished: n nodes in smem (tile-divergent)
            int32_t *row = out_nodes + (size_t)t * (size_t)L;
            __syncwarp(tmask);
            if (!CANON) {
                for (int i = tl; i < L; i += 16) row[i] = (i < n) ? smem[path + i] : -1;
                __syncwarp(tmask);
                const int B = (H + 15) >> 4, w0 = tl * B, w1 = min(H, w0 + B);
                for (int wi = w0; wi < w1; ++wi)
                    if (smem[hs + wi] != 0) smem[hs + wi] = (wi == sw) ? sbit : 0;
            } else {
                // tuple(sorted(path)) read off the bitmap (see walk_kernel): lane tl owns the words [tl*B, (tl+1)*B)
                const int32_t lastn = smem[path + n - 1];
                smem[hs + (lastn >> 5)] |= (1 << (lastn & 31));
                __syncwarp(tmask);
                const int B = (H + 15) >> 4, w0 = tl * B, w1 = min(H, w0 + B);
                uint32_t cnt = 0;
                for (int wi = w0; wi < w1; ++wi) cnt += __popc((uint32_t)smem[hs + wi] & ~(uint32_t)((wi == sw) ? sbit : 0));
                uint32_t pos = tile_inclusive_scan_u32(cnt, tmask) - cnt;
                uint64_t h = 0;
                for (int wi = w0; wi < w1; ++wi) {
                    const int32_t keepbit = (wi == sw) ? sbit : 0;
                    uint32_t bits = (uint32_t)smem[hs + wi] & ~(uint32_t)keepbit;
                    if (bits) smem[hs + wi] = keepbit;
                    while (bits) {
                        const int32_t v = wi * 32 + (__ffs(bits) - 1);
                        bits &= bits - 1;
                        row[pos] = v;
                        h += path_key_term(v, (int)pos);
                        ++pos;
                    }
                }
                for (int i = n + tl; i < L; i += 16) row[i] = kPathPad;
#pragma unroll
                for (int o = 8; o > 0; o >>= 1) h += __shfl_xor_sync(tmask, h, o);
                if (tl == 0) out_key[t] = path_key_finish(h);
            }
            if (tl == 0) out_len[t] = n;
            have = false;
        }
        __syncwarp();                                    // both tiles start the next iteration together
    }
}

// ---- graph packing (once per graph) -------------------------------------------------------------
// flag bit 0: some weight is outside [32768, 65536] (no packed 16+16-bit layout); bit 1: some weight exceeds
// kQwMax, which the short-row path's 32-bit chunk totals (up to 64 weights) cannot hold
constexpr uint32_t kQwMax = 1u << 24;
__global__ void walk_range_kernel(const uint32_t *__restrict__ qw, int64_t E, int32_t *__restrict__ flag) {
    bool unpackable = false, too_large = false;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < E; i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t q = __ldg(qw + i);
        unpackable = unpackable || q < 32768u || q > 65536u;
        too_large = too_large || q > kQwMax;
    }
    const bool a = __any_sync(0xffffffffu, unpackable), b = __any_sync(0xffffffffu, too_large);
    if ((a || b) && (threadIdx.x & 31) == 0) atomicOr(flag, (a ? 1 : 0) | (b ? 2 : 0));
}

// LAY_E8, step 2: one warp per row copies its edges as {col, qw} pairs; an odd row is followed by a {0, 0} pair
// (the buffer is zeroed first).
__global__ void __launch_bounds__(256)
walk_pack8_edges_kernel(const int32_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                        const uint32_t *__restrict__ qw, int32_t V, const int2 *__restrict__ rows,
                        uint2 *__restrict__ e8) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t v = warp; v < V; v += nw) {
        const int32_t b = __ldg(rowptr + v), deg = __ldg(rowptr + v + 1) - b;
        const int2 r = rows[v];
        for (int k = lane; k < deg; k += 32) e8[r.x + k] = make_uint2((uint32_t)__ldg(col + b + k), __ldg(qw + b + k));
    }
}

// Packed layouts, step 1 (one block): packed begin of every row = exclusive scan of the degrees rounded up to `align`
// entries = 16 bytes (E4: four 4-byte words, E8: two 8-byte pairs), so that rows can be read with LDG.128.
__global__ void __launch_bounds__(1024)
walk_pack_rows_kernel(const int32_t *__restrict__ rowptr, int32_t V, int32_t align, int2 *__restrict__ rows) {
    const int32_t am = align - 1;                        // rows start at multiples of `align` entries (2: E8, 4: E4)
    __shared__ int32_t part[1024];
    const int per = (V + 1023) / 1024, v0 = threadIdx.x * per, v1 = min(V, v0 + per);
    int32_t sum = 0;
    for (int v = v0; v < v1; ++v) sum += (rowptr[v + 1] - rowptr[v] + am) & ~am;
    part[threadIdx.x] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        int32_t acc = 0;
        for (int t = 0; t < 1024; ++t) { const int32_t x = part[t]; part[t] = acc; acc += x; }
    }
    __syncthreads();
    int32_t pb = part[threadIdx.x];
    for (int v = v0; v < v1; ++v) {
        const int32_t deg = rowptr[v + 1] - rowptr[v];
        rows[v] = make_int2(pb, pb + deg);                            // {16-byte aligned begin, true end}
        pb += (deg + am) & ~am;
    }
}

// LAY_E4, step 2: one warp per row copies its edges as col | (qw - 32768) << 16; the row is padded with sentinel words
__global__ void __launch_bounds__(256)
walk_pack4_edges_kernel(const int32_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                        const uint32_t *__restrict__ qw, int32_t V, const int2 *__restrict__ rows,
                        uint32_t *__restrict__ e4) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t v = warp; v < V; v += nw) {
        const int32_t b = __ldg(rowptr + v), deg = __ldg(rowptr + v + 1) - b;
        const int2 r = rows[v];
        for (int k = lane; k < deg; k += 32)
            e4[r.x + k] = (uint32_t)__ldg(col + b + k) | ((__ldg(qw + b + k) - 32768u) << 16);
        if (lane < ((4 - (deg & 3)) & 3)) e4[r.y + lane] = (uint32_t)V;          // sentinel words up to the next multiple of 4
    }
}

__global__ void test_draws_kernel(uint64_t seed, uint64_t subseq, int32_t n, uint64_t *out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = draw64(seed, subseq, (uint32_t)i);
}

typedef void (*walk_kern_t)(const WalkGraphPtrs, int32_t, int32_t, int32_t, int32_t, int32_t, uint64_t, uint32_t,
                            int64_t, int64_t, int64_t, int32_t *, int32_t *, unsigned long long *,
                            unsigned long long *);

static int launch_walk(const WalkGraphPtrs &g, int layout, int32_t V, int64_t E, int32_t L, uint64_t seed,
                       uint32_t group, int64_t walker_begin, int64_t walker_end, int64_t walker_stride,
                       int32_t *out_nodes, int32_t *out_len, int64_t *out_key, void *workspace, cudaStream_t st,
                       const char *who) {
    G2V_REQUIRE(V > 0 && E >= 0, "%s: V must be > 0 and E >= 0 (V=%d E=%lld)", who, V, (long long)E);
    G2V_REQUIRE(L >= 1 && L <= 4096, "%s: lenPath must be in [1, 4096] (got %d)", who, L);
    G2V_REQUIRE(walker_stride >= 1 && walker_begin >= 0, "%s: bad walker range", who);
    G2V_REQUIRE(E < (1ll << 31), "%s: E must fit int32", who);
    const int64_t n_walkers =
        walker_end > walker_begin ? (walker_end - walker_begin + walker_stride - 1) / walker_stride : 0;
    if (n_walkers == 0) return 0;                                 // empty range: nothing to write
    G2V_REQUIRE(g.rows && out_nodes && out_len && workspace, "%s: null pointer", who);
    G2V_REQUIRE(E == 0 || (g.edges && (layout != LAY_CSR || g.qw)), "%s: null edge arrays with E > 0", who);
    G2V_REQUIRE(layout == LAY_CSR || layout == LAY_E8 || (layout == LAY_E4 && V <= 65535), "%s: bad layout %d", who, layout);
    DeviceProps dp;
    if (device_props(&dp)) return 1;
    G2V_REQUIRE(dp.cc_major == 10, "%s: needs an sm_100 device (found sm_%d%d)", who, dp.cc_major, dp.cc_minor);

    const bool canon = out_key != nullptr;
    // path buffer: L ints, rounded to 32 (visit order) or to the power of two the bitonic network needs
    int Lpad = (L + 31) & ~31;
    if (canon) { Lpad = 32; while (Lpad < L) Lpad <<= 1; }
    // visited set per walker: a V-bit bitmap when a CTA's bitmaps fit 56 KB (>= 4 CTAs per SM), else a hash set
    const int bm_words = (V + 32) / 32;                           // V + 1 bits: bit V is the packed layout's sentinel node
    const char *force = getenv("G2V_WALK_VISITED");               // test hook: "hash" / "bitmap"
    int Hh = 64, hshift = 26;                                     // hash set: >= 3L slots, power of two
    while (Hh < 3 * L) { Hh <<= 1; --hshift; }
    const size_t per_warp = (size_t)kWalkWarps * sizeof(int32_t);
    const size_t bm_smem = per_warp * (Lpad + bm_words), hash_smem = per_warp * (Lpad + Hh);
    bool bitmap = bm_smem <= 56 * 1024 || bm_smem <= hash_smem;   // occupancy first, then whichever is smaller
    if (force && force[0] == 'h') bitmap = false;
    if (force && force[0] == 'b' && bm_smem <= (size_t)dp.max_smem_optin) bitmap = true;
    const int H = bitmap ? bm_words : Hh;
    const size_t smem = per_warp * (size_t)(Lpad + H);
    G2V_REQUIRE(smem <= (size_t)dp.max_smem_optin, "%s: lenPath %d needs %zu B of shared memory", who, L, smem);
    static const walk_kern_t table[2][3][2] = {
        {{walk_kernel<false, LAY_CSR, false>, walk_kernel<false, LAY_CSR, true>},
         {walk_kernel<false, LAY_E8, false>, walk_kernel<false, LAY_E8, true>},
         {walk_kernel<false, LAY_E4, false>, walk_kernel<false, LAY_E4, true>}},
        {{walk_kernel<true, LAY_CSR, false>, walk_kernel<true, LAY_CSR, true>},
         {walk_kernel<true, LAY_E8, false>, walk_kernel<true, LAY_E8, true>},
         {walk_kernel<true, LAY_E4, false>, walk_kernel<true, LAY_E4, true>}}};
    // two walkers per warp (walk_pair_kernel): packed edges + bitmap, and both tiles' bitmaps within the 56 KB budget
    const char *ft = getenv("G2V_WALK_TILE");                    // test / A-B hook: "32" / "16" force one / two walkers per warp
    const size_t pair_smem = 2 * per_warp * (size_t)(Lpad + bm_words);
    // ... and rows that mostly fit one 64-neighbour request (longer rows take its divergent slow path; measured: syn20k,
    // mean degree 100, 7.4 ms against 6.4 ms with one walker per warp), on graphs dense enough that walks are long (on
    // the ex_* graphs, mean degree 3.4 and 62 % of the walks a single node, the per-walk epilogues diverge the tiles:
    // 0.378 ms against 0.323 ms)
#ifdef G2V_WALK_STRICT_SYNC
    const bool short_rows = false;                               // the strictly synchronised build keeps one walker per warp
#else
    const bool short_rows = (double)E <= 56.0 * (double)V && (double)E >= 8.0 * (double)V;
#endif
    if (layout == LAY_E4 && bitmap && pair_smem <= 56 * 1024 && (ft ? atoi(ft) == 16 : short_rows)) {
        auto pk = canon ? walk_pair_kernel<true> : walk_pair_kernel<false>;
        G2V_CUDA_OK(cudaFuncSetAttribute(pk, cudaFuncAttributeMaxDynamicSharedMemorySize, dp.max_smem_optin));
        G2V_CUDA_OK(cudaFuncSetAttribute(pk, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        int per_sm2 = 0;
        G2V_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm2, pk, kWalkWarps * 32, pair_smem));
        G2V_REQUIRE(per_sm2 > 0, "%s: kernel does not fit on an SM", who);
        int64_t grid2 = (int64_t)dp.sm_count * per_sm2;
        const int64_t need2 = (n_walkers + 2 * kWalkWarps - 1) / (2 * kWalkWarps);
        if (grid2 > need2) grid2 = need2;
        G2V_CUDA_OK(cudaMemsetAsync(workspace, 0, sizeof(unsigned long long), st));
        pk<<<(unsigned)grid2, kWalkWarps * 32, pair_smem, st>>>(g, V, L, Lpad, bm_words, seed, group, walker_begin, n_walkers,
                                                               walker_stride, out_nodes, out_len,
                                                               reinterpret_cast<unsigned long long *>(out_key),
                                                               (unsigned long long *)workspace);
        G2V_CUDA_OK(cudaGetLastError());
        count_launch();
        return 0;
    }
    walk_kern_t kern = table[bitmap][layout][canon];
    // per-device function attributes (set on every call: the process may have switched device)
    G2V_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, dp.max_smem_optin));
    G2V_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    int per_sm = 0;
    G2V_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kWalkWarps * 32, smem));
    G2V_REQUIRE(per_sm > 0, "%s: kernel does not fit on an SM", who);
    int64_t grid = (int64_t)dp.sm_count * per_sm;                 // persistent: whole chip resident
    const int64_t need = (n_walkers + kWalkWarps - 1) / kWalkWarps;
    if (grid > need) grid = need;
    G2V_CUDA_OK(cudaMemsetAsync(workspace, 0, sizeof(unsigned long long), st));
    kern<<<(unsigned)grid, kWalkWarps * 32, smem, st>>>(g, V, L, Lpad, H, hshift, seed, group, walker_begin, n_walkers,
                                                        walker_stride, out_nodes, out_len,
                                                        reinterpret_cast<unsigned long long *>(out_key),
                                                        (unsigned long long *)workspace);
    G2V_CUDA_OK(cudaGetLastError());
    count_launch();
    return 0;
}

}  // namespace g2v

using namespace g2v;

extern "C" size_t g2v_walk_workspace_bytes(void) { return 256; }

extern "C" int g2v_walk_launch(const int32_t *rowptr, const int32_t *col, const uint32_t *qw,
                               int32_t V, int64_t E, int32_t L, uint64_t seed, uint32_t group,
                               int64_t walker_begin, int64_t walker_end, int64_t walker_stride,
                               int32_t *out_nodes, int32_t *out_len, void *workspace,
                               void *stream) {
    WalkGraphPtrs g{rowptr, col, qw};
    return launch_walk(g, LAY_CSR, V, E, L, seed, group, walker_begin, walker_end, walker_stride, out_nodes, out_len,
                       nullptr, workspace, (cudaStream_t)stream, "g2v_walk_launch");
}

// 8-byte pairs need 8*(E + one pad pair per odd row); packed 4-byte words 4*(E + up to 3 sentinels per row + overhang)
static size_t packed_edge_bytes(int32_t V, int64_t E) {
    const size_t a = sizeof(uint2) * ((size_t)E + (size_t)V + 4), b = sizeof(uint32_t) * ((size_t)E + 3 * (size_t)V + 8);
    return a > b ? a : b;
}

extern "C" int g2v_walk_packed_bytes(int32_t V, int64_t E, size_t *rows_bytes, size_t *edges_bytes) {
    G2V_REQUIRE(V > 0 && E >= 0 && rows_bytes && edges_bytes, "g2v_walk_packed_bytes: bad arguments");
    *rows_bytes = sizeof(int2) * (size_t)V;
    *edges_bytes = packed_edge_bytes(V, E);
    return 0;
}

extern "C" int g2v_walk_prepare(const int32_t *rowptr, const int32_t *col, const uint32_t *qw, int32_t V, int64_t E,
                                void *rows, void *edges, int32_t *layout_out, void *workspace, void *stream) {
    G2V_REQUIRE(V > 0 && E >= 0 && E + 3ll * V + 8 < (1ll << 31), "g2v_walk_prepare: bad sizes (V=%d E=%lld)", V, (long long)E);
    G2V_REQUIRE(rowptr && rows && edges && layout_out && workspace && (E == 0 || (col && qw)), "g2v_walk_prepare: null pointer");
    DeviceProps dp;
    if (device_props(&dp)) return 1;
    cudaStream_t st = (cudaStream_t)stream;
    // one pass over the weights: the qw <= 2^24 contract, and whether the packed 16+16-bit layout can hold them
    int32_t *flag = reinterpret_cast<int32_t *>(workspace) + 8;   // the ticket lives in the first 8 bytes
    int32_t h = 0;
    G2V_CUDA_OK(cudaMemsetAsync(flag, 0, sizeof(int32_t), st));
    if (E > 0) {
        int64_t blocks = (E + 255) / 256;
        if (blocks > (int64_t)dp.sm_count * 8) blocks = (int64_t)dp.sm_count * 8;
        walk_range_kernel<<<(unsigned)blocks, 256, 0, st>>>(qw, E, flag);
        G2V_CUDA_OK(cudaGetLastError());
        count_launch();
    }
    G2V_CUDA_OK(cudaMemcpyAsync(&h, flag, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    G2V_CUDA_OK(cudaStreamSynchronize(st));                       // setup, once per graph
    G2V_REQUIRE((h & 2) == 0, "g2v_walk_prepare: an edge weight exceeds the limit qw <= 2^24 = %u", kQwMax);
    const char *force = getenv("G2V_WALK_LAYOUT");                // test hook: "e8" / "e4" (e4 only if eligible)
    const int layout = (V <= 65535 && !(force && force[1] == '8') && (h & 1) == 0) ? LAY_E4 : LAY_E8;
    // pads / overhang read as weight-0 (E8) or are overwritten with sentinels (E4): zero the whole buffer first
    G2V_CUDA_OK(cudaMemsetAsync(edges, 0, packed_edge_bytes(V, E), st));
    walk_pack_rows_kernel<<<1, 1024, 0, st>>>(rowptr, V, layout == LAY_E4 ? 4 : 2, reinterpret_cast<int2 *>(rows));
    G2V_CUDA_OK(cudaGetLastError());
    int64_t blocks = ((int64_t)V * 32 + 255) / 256;
    if (blocks > (int64_t)dp.sm_count * 8) blocks = (int64_t)dp.sm_count * 8;
    if (layout == LAY_E4)
        walk_pack4_edges_kernel<<<(unsigned)blocks, 256, 0, st>>>(rowptr, col, qw, V, reinterpret_cast<const int2 *>(rows),
                                                                reinterpret_cast<uint32_t *>(edges));
    else
        walk_pack8_edges_kernel<<<(unsigned)blocks, 256, 0, st>>>(rowptr, col, qw, V, reinterpret_cast<const int2 *>(rows),
                                                                reinterpret_cast<uint2 *>(edges));
    G2V_CUDA_OK(cudaGetLastError());
    count_launch(2);
    *layout_out = layout;
    return 0;
}

extern "C" int g2v_walk_launch_packed(const void *rows, const void *edges, int32_t layout, int32_t V, int64_t E,
                                      int32_t L, uint64_t seed, uint32_t group, int64_t walker_begin,
                                      int64_t walker_end, int64_t walker_stride, int32_t *out_nodes, int32_t *out_len,
                                      int64_t *out_key, void *workspace, void *stream) {
    G2V_REQUIRE(layout == LAY_E8 || layout == LAY_E4, "g2v_walk_launch_packed: layout must come from g2v_walk_prepare");
    WalkGraphPtrs g{reinterpret_cast<const int32_t *>(rows), edges, nullptr};
    return launch_walk(g, layout, V, E, L, seed, group, walker_begin, walker_end, walker_stride, out_nodes, out_len,
                       out_key, workspace, (cudaStream_t)stream, "g2v_walk_launch_packed");
}

extern "C" int g2v_walk_host(const int32_t *rowptr, const int32_t *col, const uint32_t *qw,
                             int32_t V, int64_t E, int32_t L, uint64_t seed, uint32_t group,
                             int64_t walker_begin, int64_t walker_end, int64_t walker_stride,
                             int32_t *out_nodes, int32_t *out_len) {
    G2V_REQUIRE(V > 0 && E >= 0 && L >= 1 && walker_stride >= 1, "g2v_walk_host: bad arguments");
    const int64_t n = walker_end > walker_begin ? (walker_end - walker_begin + walker_stride - 1) / walker_stride : 0;
    if (n == 0) return 0;
    // ONE device slab: rowptr | col | qw | packed rows | packed edges | nodes | len | workspace
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t Ee = (size_t)(E > 0 ? E : 1);
    const size_t o_rp = take(sizeof(int32_t) * (size_t)(V + 1)), o_col = take(sizeof(int32_t) * Ee),
                 o_qw = take(sizeof(uint32_t) * Ee), o_rows = take(sizeof(int2) * (size_t)V),
                 o_edges = take(packed_edge_bytes(V, E)), o_nodes = take(sizeof(int32_t) * (size_t)n * (size_t)L),
                 o_len = take(sizeof(int32_t) * (size_t)n), o_ws = take(g2v_walk_workspace_bytes());
    char *d = nullptr;
    int rc = 1;
    cudaStream_t st = nullptr;
    do {
        if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) break;
        if (cudaMalloc(&d, off) != cudaSuccess) break;
        if (cudaMemcpyAsync(d + o_rp, rowptr, sizeof(int32_t) * (size_t)(V + 1), cudaMemcpyHostToDevice, st) != cudaSuccess) break;
        if (E > 0) {
            if (cudaMemcpyAsync(d + o_col, col, sizeof(int32_t) * (size_t)E, cudaMemcpyHostToDevice, st) != cudaSuccess) break;
            if (cudaMemcpyAsync(d + o_qw, qw, sizeof(uint32_t) * (size_t)E, cudaMemcpyHostToDevice, st) != cudaSuccess) break;
        }
        int32_t layout = LAY_E8;
        rc = g2v_walk_prepare((int32_t *)(d + o_rp), (int32_t *)(d + o_col), (uint32_t *)(d + o_qw), V, E, d + o_rows,
                              d + o_edges, &layout, d + o_ws, st);
        if (rc) break;
        rc = g2v_walk_launch_packed(d + o_rows, d + o_edges, layout, V, E, L, seed, group, walker_begin, walker_end,
                                    walker_stride, (int32_t *)(d + o_nodes), (int32_t *)(d + o_len), nullptr, d + o_ws, st);
        if (rc) break;
        rc = 1;
        if (cudaMemcpyAsync(out_nodes, d + o_nodes, sizeof(int32_t) * (size_t)n * (size_t)L, cudaMemcpyDeviceToHost, st) != cudaSuccess) break;
        if (cudaMemcpyAsync(out_len, d + o_len, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, st) != cudaSuccess) break;
        if (cudaStreamSynchronize(st) != cudaSuccess) break;
        rc = 0;
    } while (0);
    if (rc == 1) {
        cudaError_t e = cudaGetLastError();
        set_error("g2v_walk_host: CUDA failure: %s", cudaGetErrorString(e));
    }
    cudaFree(d);
    if (st) cudaStreamDestroy(st);
    return rc;
}

extern "C" int g2v_test_draws(uint64_t seed, uint64_t subsequence, int32_t n, uint64_t *out_dev,
                              void *stream) {
    G2V_REQUIRE(n >= 0 && out_dev, "g2v_test_draws: bad arguments");
    if (n == 0) return 0;
    test_draws_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(seed, subsequence, n, out_dev);
    G2V_CUDA_OK(cudaGetLastError());
    count_launch();
    return 0;
}
