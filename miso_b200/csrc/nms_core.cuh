// nms_core.cuh — segmented greedy NMS building blocks shared by the generic
// torchvision-signature entry points (nms.cu), the fused RPN path (rpn.cu) and the fused
// detection path (detpost.cu).
//
// Reference semantics: torchvision::nms CPU (tv-csrc:ops/cpu/nms_kernel.cpp:116, restated in
// SURVEY.md Appendix B.1): areas and IoU with one fp32 rounding per operation (no FMA),
// suppression iff (double)iou > iou_threshold (strict), candidates visited in stable
// descending-score order.
//
// Pipeline over "segments" (one segment = one independent NMS problem, e.g. image x level):
//   rank    : order the elements of every segment by a unique 64-bit key (rank by counting)
//   meta    : per-segment word counts, mask offsets and a tile prefix (single block scan)
//   mask    : 64x64 IoU tiles -> one 64-bit suppression word per (row box, column block),
//             upper-triangular tiles only, persistent grid sized from the SM count
//   sweep   : one CTA per segment; serial 64-step resolve of the diagonal word, parallel OR
//             of the kept rows into the removed[] bit-vector held in shared memory
#pragma once
#include <cstdlib>
#include "common.cuh"

namespace mb {

struct SegArrays {
    int* seg_start;        // [G]   first position of segment g in the sorted arrays
    int* seg_count;        // [G]   number of live elements
    int* seg_words;        // [G]   ceil(count/64)
    long long* mask_off;   // [G]   word offset of the segment's mask rows
    long long* tile_pre;   // [G+1] exclusive prefix of T(T+1)/2
    int* keep_off;         // [G+1] exclusive prefix of T (word offset into keepbits)
    int* seg_kept;         // [G]   number of boxes kept by the sweep
    long long* totals;     // [4]   0: tiles, 1: mask words needed, 2: overflow flag, 3: spare
};

inline size_t seg_arrays_bytes(int G) {
    size_t b = 0;
    b += align_up(sizeof(int) * G, 256) * 4;              // start,count,words,kept
    b += align_up(sizeof(long long) * G, 256);            // mask_off
    b += align_up(sizeof(long long) * (G + 1), 256);      // tile_pre
    b += align_up(sizeof(int) * (G + 1), 256);            // keep_off
    b += 256;                                             // totals
    return b + 256;
}

inline SegArrays carve_seg_arrays(Carver& c, int G) {
    SegArrays s;
    s.seg_start = c.take<int>(G);
    s.seg_count = c.take<int>(G);
    s.seg_words = c.take<int>(G);
    s.seg_kept = c.take<int>(G);
    s.mask_off = c.take<long long>(G);
    s.tile_pre = c.take<long long>(G + 1);
    s.keep_off = c.take<int>(G + 1);
    s.totals = c.take<long long>(4);
    return s;
}

// ------------------------------------------------------------------------------------
// block-wide exclusive scan of one long long per thread (1024 threads), returns total
// ------------------------------------------------------------------------------------
__device__ inline long long block_excl_scan_1024(long long v, long long* sh /*[1024+32]*/, long long& total) {
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    long long x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        long long y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) sh[wid] = x;
    __syncthreads();
    if (wid == 0) {
        long long w = sh[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            long long y = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += y;
        }
        sh[32 + lane] = w;  // inclusive over warps
    }
    __syncthreads();
    long long warp_base = wid ? sh[32 + wid - 1] : 0;
    total = sh[32 + 31];
    long long r = warp_base + x - v;
    __syncthreads();
    return r;
}

// ------------------------------------------------------------------------------------
// meta: from seg_count (and, when compute_starts, a packed layout) derive everything else.
// Also evaluates torchvision's batched_nms strategy rule per image for the fused paths
// (tv:ops/boxes.py:80): trick iff 4*boxes_in_image <= trick_numel, offsets
// fl(fl(group) * fl(max_coord + 1)) (tv:ops/boxes.py:99-102); 0 otherwise.
// ------------------------------------------------------------------------------------
struct MetaRule {
    int segs_per_image;     // 0 -> no per-image rule (seg_offset not written)
    int group_base;         // group value of the first segment of an image
    long long trick_numel;  // numel threshold of the reference rule; <0 -> always vanilla
    const float* img_max;   // [num_images] max coordinate over the image's live boxes
    float* seg_offset;      // [G] out
};

static __global__ void __launch_bounds__(1024) k_seg_meta(SegArrays s, int G, int compute_starts,
                                                   long long mask_cap_words, MetaRule rule) {
    pdl_enter();
    __shared__ long long sh[64];
    __shared__ long long carry[4];
    const int tid = threadIdx.x;
    if (G <= 32) {
        // the hot-path case (image x level or image x class segments): one warp, shuffle scans, no barriers
        if (tid < 32) {
            const int n = tid < G ? s.seg_count[tid] : 0;
            const long long T = (n + 63) >> 6;
            long long v[4] = {(long long)n, (long long)n * T, T * (T + 1) / 2, T}, inc[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                inc[q] = v[q];
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const long long y = __shfl_up_sync(0xffffffffu, inc[q], o);
                    if (tid >= o) inc[q] += y;
                }
            }
            if (tid < G) {
                if (compute_starts) s.seg_start[tid] = (int)(inc[0] - v[0]);
                s.seg_words[tid] = (int)T;
                s.mask_off[tid] = inc[1] - v[1];
                s.tile_pre[tid] = inc[2] - v[2];
                s.keep_off[tid] = (int)(inc[3] - v[3]);
            }
            if (tid == 31) {
                s.tile_pre[G] = inc[2];
                s.keep_off[G] = (int)inc[3];
                s.totals[0] = inc[2];
                s.totals[1] = inc[1];
                s.totals[2] = inc[1] > mask_cap_words ? 1 : 0;
            }
        }
    } else {
    if (tid < 4) carry[tid] = 0;
    __syncthreads();
    for (int base = 0; base < G; base += 1024) {
        const int g = base + tid;
        const int n = g < G ? s.seg_count[g] : 0;
        const long long T = (n + 63) >> 6;
        long long tot;
        long long st = block_excl_scan_1024(n, sh, tot);
        const long long c0 = carry[0];
        __syncthreads();
        if (tid == 0) carry[0] = c0 + tot;
        long long mo = block_excl_scan_1024((long long)n * T, sh, tot);
        const long long c1 = carry[1];
        __syncthreads();
        if (tid == 0) carry[1] = c1 + tot;
        long long tp = block_excl_scan_1024(T * (T + 1) / 2, sh, tot);
        const long long c2 = carry[2];
        __syncthreads();
        if (tid == 0) carry[2] = c2 + tot;
        long long ko = block_excl_scan_1024(T, sh, tot);
        const long long c3 = carry[3];
        __syncthreads();
        if (tid == 0) carry[3] = c3 + tot;
        if (g < G) {
            if (compute_starts) s.seg_start[g] = (int)(c0 + st);
            s.seg_words[g] = (int)T;
            s.mask_off[g] = c1 + mo;
            s.tile_pre[g] = c2 + tp;
            s.keep_off[g] = (int)(c3 + ko);
        }
        __syncthreads();
    }
    if (tid == 0) {
        s.tile_pre[G] = carry[2];
        s.keep_off[G] = (int)carry[3];
        s.totals[0] = carry[2];
        s.totals[1] = carry[1];
        s.totals[2] = carry[1] > mask_cap_words ? 1 : 0;
    }
    }
    if (rule.segs_per_image > 0) {
        for (int g = tid; g < G; g += 1024) {
            const int img = g / rule.segs_per_image;
            long long cnt = 0;
            for (int q = 0; q < rule.segs_per_image; ++q) cnt += s.seg_count[img * rule.segs_per_image + q];
            float off = 0.0f;
            if (rule.trick_numel >= 0 && 4 * cnt <= rule.trick_numel) {
                const float grp = (float)(rule.group_base + g % rule.segs_per_image);
                off = __fmul_rn(grp, __fadd_rn(rule.img_max[img], 1.0f));
            }
            rule.seg_offset[g] = off;
        }
    }
}

// ------------------------------------------------------------------------------------
// rank by counting inside segments. Keys are unique 64-bit values (score key << 32 | tie).
// Position p of the bucketed arrays belongs to segment bseg[p] (or -1 for a hole).
// Writes skey/sbox at seg_start + rank; optional per-segment box offset (trick mode).
// ------------------------------------------------------------------------------------
constexpr int kRankThreads = 256;
constexpr int kRankSplit = 8;                              // lanes that share one key, each counting every 8th candidate
constexpr int kRankKeys = kRankThreads / kRankSplit;       // keys per CTA
constexpr int kRankTile = 2048;

static __global__ void __launch_bounds__(kRankThreads) k_rank_in_segment(
    const unsigned long long* __restrict__ bkey, const float4* __restrict__ bbox,
    const int* __restrict__ bseg, const int* __restrict__ seg_start,
    const int* __restrict__ seg_count, const float* __restrict__ seg_offset, int P,
    unsigned long long* __restrict__ skey, float4* __restrict__ sbox) {
    pdl_enter();
    __shared__ unsigned long long tile[kRankTile];
    __shared__ int s_lo, s_hi;
    const int tid = threadIdx.x, sub = tid % kRankSplit;
    const int p = blockIdx.x * kRankKeys + tid / kRankSplit;
    int g = -1, lo = 0, hi = 0;
    unsigned long long key = 0;
    if (p < P) {
        g = bseg[p];
        if (g >= 0) { lo = seg_start[g]; hi = lo + seg_count[g]; key = bkey[p]; }
    }
    if (tid == 0) { s_lo = 0x7fffffff; s_hi = 0; }
    __syncthreads();
    if (g >= 0 && sub == 0) { atomicMin(&s_lo, lo); atomicMax(&s_hi, hi); }
    __syncthreads();
    const int ulo = s_lo, uhi = s_hi;
    int rank = 0;
    for (int t0 = ulo; t0 < uhi; t0 += kRankTile) {
        const int tn = min(kRankTile, uhi - t0);
        __syncthreads();
        for (int j = tid; j < tn; j += kRankThreads) tile[j] = bkey[t0 + j];
        __syncthreads();
        const int a = max(lo, t0) - t0, b = min(hi, t0 + tn) - t0;
        int cnt = 0;
#pragma unroll 4
        for (int j = a + sub; j < b; j += kRankSplit) cnt += (tile[j] < key) ? 1 : 0;   // 8 distinct words per warp read: no conflicts
        rank += cnt;
    }
#pragma unroll
    for (int d = 1; d < kRankSplit; d <<= 1) rank += __shfl_xor_sync(0xffffffffu, rank, d);
    if (g >= 0 && sub == 0) {
        const int dst = lo + rank;
        skey[dst] = key;
        if (sbox != nullptr) {
            float4 bx = bbox[p];
            if (seg_offset != nullptr) {
                const float o = seg_offset[g];
                bx.x = __fadd_rn(bx.x, o); bx.y = __fadd_rn(bx.y, o);
                bx.z = __fadd_rn(bx.z, o); bx.w = __fadd_rn(bx.w, o);
            }
            sbox[dst] = bx;
        }
    }
}

// ------------------------------------------------------------------------------------
// IoU predicate with the reference's exact operation order.
// ------------------------------------------------------------------------------------
__device__ __forceinline__ float box_area_rn(const float4 b) {
    return __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y));
}

__device__ __forceinline__ bool iou_suppresses(const float4 a, const float area_a, const float4 b,
                                               const float area_b, const float thr_up) {
    const float xx1 = (a.x < b.x) ? b.x : a.x;   // std::max(a, b) == (a < b) ? b : a
    const float yy1 = (a.y < b.y) ? b.y : a.y;
    const float xx2 = (b.z < a.z) ? b.z : a.z;   // std::min(a, b) == (b < a) ? b : a
    const float yy2 = (b.w < a.w) ? b.w : a.w;
    float w = __fsub_rn(xx2, xx1); w = (0.0f < w) ? w : 0.0f;
    float h = __fsub_rn(yy2, yy1); h = (0.0f < h) ? h : 0.0f;
    const float inter = __fmul_rn(w, h);
    const float ovr = __fdiv_rn(inter, __fsub_rn(__fadd_rn(area_a, area_b), inter));
    return ovr >= thr_up;  // == ((double)ovr > iou_threshold); NaN -> false -> kept
}

// ------------------------------------------------------------------------------------
// mask: persistent loop over upper-triangular 64x64 tiles of all segments
// ------------------------------------------------------------------------------------
__device__ __forceinline__ float4 offset_box(float4 b, float o) {
    return make_float4(__fadd_rn(b.x, o), __fadd_rn(b.y, o), __fadd_rn(b.z, o), __fadd_rn(b.w, o));
}

// seg_offset (nullable): per-segment coordinate offset of the batched_nms coordinate trick,
// added on load (tv:ops/boxes.py:101); 0 for segments that run the per-group strategy.
static __global__ void __launch_bounds__(128) k_nms_mask(const float4* __restrict__ sbox, SegArrays s, int G,
                                                 float thr_up, unsigned long long* __restrict__ mask,
                                                 const float* __restrict__ seg_offset, int full) {
    pdl_enter();
    __shared__ float4 cbox[64];
    __shared__ float carea[64];
    // per-segment metadata of up to kMaskSegCache segments staged once per CTA: the tile -> (segment, row block, column
    // block) lookup then costs no dependent global loads (it used to be a five-deep chain of them per tile)
    constexpr int kMaskSegCache = 256;
    __shared__ long long s_pre[kMaskSegCache + 1];
    __shared__ long long s_moff[kMaskSegCache];
    __shared__ int s_cnt[kMaskSegCache], s_st[kMaskSegCache];
    __shared__ float s_off[kMaskSegCache];
    const int tid = threadIdx.x;
    if (s.totals[2] != 0) return;  // mask workspace too small: host retries with totals[1] words
    const long long total = s.totals[0];
    const bool cached = G <= kMaskSegCache;
    if (cached) {
        for (int i = tid; i <= G; i += blockDim.x) {
            s_pre[i] = s.tile_pre[i];
            if (i < G) {
                s_moff[i] = s.mask_off[i]; s_cnt[i] = s.seg_count[i]; s_st[i] = s.seg_start[i];
                s_off[i] = seg_offset != nullptr ? seg_offset[i] : 0.0f;
            }
        }
    }
    __syncthreads();
    for (long long t = blockIdx.x; t < total; t += gridDim.x) {
        // lane 0 of every warp decodes the tile (segment by binary search in the staged prefix, row block by the
        // inverse of the triangular count: float estimate, exact integer correction) and broadcasts it: no barrier,
        // and the other 31 lanes do not spend issue slots on it
        int g = 0, r = 0, c = 0;
        if ((tid & 31) == 0) {
            int lo = 0, hi = G;  // largest g with tile_pre[g] <= t
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if ((cached ? s_pre[mid] : s.tile_pre[mid]) <= t) lo = mid; else hi = mid;
            }
            g = lo;
            const long long TT = ((cached ? s_cnt[g] : s.seg_count[g]) + 63) >> 6;
            const long long tl = t - (cached ? s_pre[g] : s.tile_pre[g]);
            long long rr;
            if (TT <= 2048) {
                const float d = (float)(2 * TT + 1);
                rr = (long long)((d - sqrtf(fmaxf(d * d - 8.0f * (float)tl, 0.0f))) * 0.5f);
            } else {
                const double d = (double)(2 * TT + 1);
                rr = (long long)((d - sqrt(d * d - 8.0 * (double)tl)) * 0.5);
            }
            if (rr < 0) rr = 0;
            if (rr > TT - 1) rr = TT - 1;
            while (rr + 1 <= TT - 1 && (rr + 1) * TT - (rr + 1) * rr / 2 <= tl) ++rr;
            while (rr > 0 && rr * TT - rr * (rr - 1) / 2 > tl) --rr;
            r = (int)rr; c = (int)(rr + (tl - (rr * TT - rr * (rr - 1) / 2)));
        }
        g = __shfl_sync(0xffffffffu, g, 0); r = __shfl_sync(0xffffffffu, r, 0); c = __shfl_sync(0xffffffffu, c, 0);
        const int n = cached ? s_cnt[g] : s.seg_count[g];
        const int st = cached ? s_st[g] : s.seg_start[g];
        const long long moff = cached ? s_moff[g] : s.mask_off[g];
        const float off = cached ? s_off[g] : (seg_offset != nullptr ? seg_offset[g] : 0.0f);
        const int T = (n + 63) >> 6;
        const int ncol = min(64, n - c * 64);
        // two threads per row: thread (row, half) tests columns 32*half .. 32*half+31 and writes its own
        // 32-bit half of the mask word (little-endian halves of the 64-bit word)
        const int row = r * 64 + (tid & 63), half = tid >> 6;
        float4 a_raw = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row < n) a_raw = sbox[st + row];                 // issued together with the column box load below
        if (tid < ncol) {
            const float4 b = offset_box(sbox[st + c * 64 + tid], off);
            cbox[tid] = b;
            carea[tid] = box_area_rn(b);
        }
        __syncthreads();
        unsigned int word = 0;
        if (row < n) {
            const float4 a = offset_box(a_raw, off);
            const float area_a = box_area_rn(a);
            // Diagonal tiles carry the full symmetric word (bits j < row too): the sweep resolves a
            // 64-box block in parallel from "who suppresses me" = word & lower bits.
            const int skip = (r == c) ? (tid & 63) : -1;
            const int j0 = 32 * half, j1 = min(ncol, j0 + 32);
            if (thr_up > 0.0f) {
                // An IoU above a positive threshold needs a positive intersection, and most pairs are disjoint. Pass 1
                // marks the columns whose box overlaps this row's at all (four chained compares, no divergence: a
                // superset of "positive intersection" — degenerate boxes that slip through get IoU 0 or NaN below);
                // pass 2 runs the exact IoU only on those, each lane walking its own few set bits. With one loop a
                // warp paid for the division whenever ANY of its 32 rows overlapped the column.
                unsigned int cand = 0;
#pragma unroll 8
                for (int j = j0; j < j1; ++j) {
                    const float4 b = cbox[j];
                    if (b.x < a.z && a.x < b.z && b.y < a.w && a.y < b.w) cand |= 1u << (j - j0);
                }
                if (skip >= j0 && skip < j0 + 32) cand &= ~(1u << (skip - j0));
                while (cand) {
                    const int q = __ffs((int)cand) - 1;
                    cand &= cand - 1u;
                    if (iou_suppresses(a, area_a, cbox[j0 + q], carea[j0 + q], thr_up)) word |= 1u << q;
                }
            } else {
                for (int j = j0; j < j1; ++j)
                    if (j != skip && iou_suppresses(a, area_a, cbox[j], carea[j], thr_up)) word |= 1u << (j - j0);
            }
            // full mode (fixed-point sweep): word-major [T][n], so that the sweep's thread-per-box loads and the stores
            // here are contiguous across boxes; otherwise row-major [n][T] for the block sweeps
            const long long at = full ? (long long)c * n + row : (long long)row * T + c;
            reinterpret_cast<unsigned int*>(mask)[2 * (moff + at) + half] = word;
        }
        if (full && r != c) {
            // the fixed-point sweep reads "who suppresses me" for whole rows: IoU is symmetric, so the tile's transpose
            // fills word r of rows 64c .. 64c+63. This warp holds rows 32*(warp&1).. of columns 32*half..: one ballot
            // per column gives that column's 32 row bits; lane j keeps column j's and writes its 32-bit half.
            const int lane = tid & 31, sub = (tid >> 5) & 1;
            unsigned int tw = 0;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const unsigned int b = __ballot_sync(0xffffffffu, (word >> j) & 1u);
                if (lane == j) tw = b;
            }
            const int trow = c * 64 + 32 * half + lane;
            if (trow < n) reinterpret_cast<unsigned int*>(mask)[2 * (moff + (long long)r * n + trow) + sub] = tw;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------
// sweep: one CTA per segment. keepbits word b of segment g holds the kept flags of its
// boxes 64b..64b+63 (sorted order). max_keep > 0 stops once that many boxes are kept
// (later boxes of the segment all score lower, so they cannot enter a global top-max_keep).
// ------------------------------------------------------------------------------------
constexpr int kSweepThreads = 256;
constexpr int kSweepBigThreads = 1024;

// Generic sweep for segments of any size (the mask rows do not fit in shared memory): per 64-box block, one warp
// resolves the block from its diagonal words (parallel fixed point, see k_nms_sweep_small), then the kept rows are
// streamed from global memory one row per warp — every lane issues its whole strided share of the row before the
// first use, so a row costs one memory latency — and OR-ed into removed[] (shared memory, T words).
static __global__ void __launch_bounds__(kSweepBigThreads) k_nms_sweep(SegArrays s, const unsigned long long* __restrict__ mask,
                                                                     unsigned long long* __restrict__ keepbits, int max_keep) {
    extern __shared__ unsigned long long removed[];
    __shared__ unsigned long long diag[64];
    __shared__ unsigned long long s_keepw;
    const int g = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int kWarps = kSweepBigThreads / 32;
    const int n = s.seg_count[g];
    const int T = s.seg_words[g];
    const bool overflow = s.totals[2] != 0;
    if (n == 0 || overflow) { if (tid == 0) s.seg_kept[g] = 0; return; }
    const unsigned long long* m = mask + s.mask_off[g];
    unsigned long long* kb = keepbits + s.keep_off[g];
    for (int w = tid; w < T; w += kSweepBigThreads) removed[w] = 0;
    int kept = 0;
    for (int b = 0; b < T; ++b) {
        const int nb = min(64, n - b * 64);
        if (tid < 64) diag[tid] = tid < nb ? m[(long long)(b * 64 + tid) * T + b] : 0ull;
        __syncthreads();                               // diag ready; removed[] updates of the previous block visible
        if (warp == 0) {
            const unsigned long long invalid = nb < 64 ? ~((1ull << nb) - 1ull) : 0ull;
            unsigned long long R = removed[b] | invalid, C = 0;
            const int t0 = lane, t1 = lane + 32;
            const unsigned long long s0 = diag[t0] & ((1ull << t0) - 1ull);
            const unsigned long long s1 = diag[t1] & ((1ull << t1) - 1ull);
            while ((C | R) != ~0ull) {
                const unsigned long long D = C | R;
                bool c0 = false, r0 = false, c1 = false, r1 = false;
                if (!((D >> t0) & 1ull)) { if (s0 & C) r0 = true; else if ((s0 & ~R) == 0ull) c0 = true; }
                if (!((D >> t1) & 1ull)) { if (s1 & C) r1 = true; else if ((s1 & ~R) == 0ull) c1 = true; }
                C |= (unsigned long long)__ballot_sync(0xffffffffu, c0) | ((unsigned long long)__ballot_sync(0xffffffffu, c1) << 32);
                R |= (unsigned long long)__ballot_sync(0xffffffffu, r0) | ((unsigned long long)__ballot_sync(0xffffffffu, r1) << 32);
            }
            unsigned long long keepw = C;
            if (max_keep > 0 && kept + __popcll(keepw) > max_keep) {
                int extra = kept + __popcll(keepw) - max_keep;    // trim to exactly max_keep kept boxes in this segment
                while (extra-- > 0) keepw &= ~(1ull << (63 - __clzll(keepw)));
            }
            if (lane == 0) { s_keepw = keepw; kb[b] = keepw; }
        }
        __syncthreads();
        const unsigned long long keepw = s_keepw;
        kept += __popcll(keepw);
        if (max_keep > 0 && kept >= max_keep) {
            for (int w = b + 1 + tid; w < T; w += kSweepBigThreads) kb[w] = 0ull;
            break;
        }
        // kept row number r of this block (in bit order) goes to warp r % kWarps
        unsigned long long bits = keepw;
        for (int r = 0; bits; ++r) {
            const int t = __ffsll((long long)bits) - 1; bits &= bits - 1;
            if ((r % kWarps) != warp) continue;
            const unsigned long long* row = m + (long long)(b * 64 + t) * T;
            for (int c0 = b + 1 + lane; c0 < T; c0 += 32 * 8) {
                unsigned long long v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) { const int c = c0 + 32 * u; v[u] = c < T ? __ldg(row + c) : 0ull; }
#pragma unroll
                for (int u = 0; u < 8; ++u) if (v[u]) atomicOr(&removed[c0 + 32 * u], v[u]);
            }
        }
        // the barrier at the top of the next iteration orders these updates before the next resolve
    }
    if (tid == 0) s.seg_kept[g] = kept;
}

// ------------------------------------------------------------------------------------
// sweep for segments of up to 4096 boxes (T <= 64 words): the 64 x (T-b) tile of mask words of
// block b is staged in shared memory (next tile prefetched into registers while the current one
// is resolved); one warp resolves the block in parallel: box t is kept iff every earlier box of
// the block that overlaps it ("suppressors", the lower bits of its diagonal word) is removed, and
// removed iff one of them is kept — the lowest undecided box is always decidable, so the
// fixed point is reached in as many rounds as the longest suppression chain (typically 2-4);
// kept rows are then OR-ed into removed[] by 256 threads with shared-memory atomics.
// ------------------------------------------------------------------------------------
constexpr int kSweepSmallMaxWords = 64;

static __global__ void __launch_bounds__(kSweepThreads) k_nms_sweep_small(SegArrays s, const unsigned long long* __restrict__ mask,
                                                                        unsigned long long* __restrict__ keepbits, int max_keep) {
    __shared__ unsigned long long removed[kSweepSmallMaxWords];
    __shared__ unsigned long long tile[64 * kSweepSmallMaxWords];
    __shared__ unsigned long long s_keepw;
    constexpr int kPre = 64 * kSweepSmallMaxWords / kSweepThreads;   // tile words per thread
    const int g = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = s.seg_count[g];
    const int T = s.seg_words[g];
    if (n == 0 || s.totals[2] != 0) { if (tid == 0) s.seg_kept[g] = 0; return; }
    const unsigned long long* m = mask + s.mask_off[g];
    unsigned long long* kb = keepbits + s.keep_off[g];
    if (tid < T) removed[tid] = 0;
    unsigned long long pre[kPre];
    // tile of block b: rows 64b .. 64b+nb-1, words b .. T-1, row-major with Wn = T - b words per row.
    // Thread (warp, lane) owns rows warp, warp+8, .. and columns lane, lane+32: no index division, and a
    // warp reads up to 32 consecutive words of one row.
    static_assert(kPre == 16 && kSweepThreads == 256 && kSweepSmallMaxWords == 64, "prefetch mapping");
    auto prefetch = [&](int b) {
        const int nb = min(64, n - b * 64), Wn = T - b;
#pragma unroll
        for (int u = 0; u < kPre; ++u) {
            const int row = warp + 8 * (u >> 1), col = lane + 32 * (u & 1);
            pre[u] = (row < nb && col < Wn) ? m[(long long)(b * 64 + row) * T + b + col] : 0ull;
        }
    };
    prefetch(0);
    int kept = 0;
    for (int b = 0; b < T; ++b) {
        const int nb = min(64, n - b * 64), Wn = T - b;
#pragma unroll
        for (int u = 0; u < kPre; ++u) {
            const int row = warp + 8 * (u >> 1), col = lane + 32 * (u & 1);
            if (row < nb && col < Wn) tile[row * Wn + col] = pre[u];
        }
        __syncthreads();
        if (b + 1 < T) prefetch(b + 1);          // global loads of the next tile fly during the resolve
        if (warp == 0) {
            const unsigned long long invalid = nb < 64 ? ~((1ull << nb) - 1ull) : 0ull;
            unsigned long long R = removed[b] | invalid, C = 0;
            const int t0 = lane, t1 = lane + 32;
            const unsigned long long s0 = (t0 < nb) ? (tile[t0 * Wn] & ((1ull << t0) - 1ull)) : 0ull;
            const unsigned long long s1 = (t1 < nb) ? (tile[t1 * Wn] & ((1ull << t1) - 1ull)) : 0ull;
            while ((C | R) != ~0ull) {
                const unsigned long long D = C | R;
                bool c0 = false, r0 = false, c1 = false, r1 = false;
                if (!((D >> t0) & 1ull)) { if (s0 & C) r0 = true; else if ((s0 & ~R) == 0ull) c0 = true; }
                if (!((D >> t1) & 1ull)) { if (s1 & C) r1 = true; else if ((s1 & ~R) == 0ull) c1 = true; }
                C |= (unsigned long long)__ballot_sync(0xffffffffu, c0) | ((unsigned long long)__ballot_sync(0xffffffffu, c1) << 32);
                R |= (unsigned long long)__ballot_sync(0xffffffffu, r0) | ((unsigned long long)__ballot_sync(0xffffffffu, r1) << 32);
            }
            unsigned long long keepw = C;
            if (max_keep > 0 && kept + __popcll(keepw) > max_keep) {
                int extra = kept + __popcll(keepw) - max_keep;
                while (extra-- > 0) keepw &= ~(1ull << (63 - __clzll(keepw)));
            }
            if (lane == 0) { s_keepw = keepw; kb[b] = keepw; }
        }
        __syncthreads();
        const unsigned long long keepw = s_keepw;
        kept += __popcll(keepw);
        if (max_keep > 0 && kept >= max_keep) {
            for (int w = b + 1 + tid; w < T; w += kSweepThreads) kb[w] = 0ull;
            break;
        }
        // removed[b + col] |= OR of the kept rows' words: thread = (column, quarter of the rows)
        {
            const int col = 1 + (tid >> 2), q = tid & 3;
            if (col < Wn) {
                unsigned long long acc = 0, bits = (keepw >> (16 * q)) & 0xffffull;
                while (bits) {
                    const int t = __ffsll((long long)bits) - 1 + 16 * q; bits &= bits - 1;
                    acc |= tile[t * Wn + col];
                }
                if (acc) atomicOr(&removed[b + col], acc);
            }
        }
        __syncthreads();
    }
    if (tid == 0) s.seg_kept[g] = kept;
}

// ------------------------------------------------------------------------------------
// The same block-resolve sweep for segments of more than 4096 boxes (T > 64 words; the cross-tile seam
// NMS of a mosaic): the tile of block b (64 rows x (T - b) words) is staged in dynamic shared memory with
// cp.async; with two buffers the next tile streams in while the current block is resolved and OR-ed.
// smem: removed[Tcap] + nbuf x tile[64][Tcap] words.
// ------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(kSweepThreads) k_nms_sweep_wide(SegArrays s, const unsigned long long* __restrict__ mask,
                                                                       unsigned long long* __restrict__ keepbits, int max_keep,
                                                                       int Tcap, int nbuf) {
    extern __shared__ unsigned long long wsm[];
    __shared__ unsigned long long s_keepw;
    unsigned long long* removed = wsm;                 // [Tcap]
    unsigned long long* tiles = wsm + Tcap;            // [nbuf][64 * Tcap]
    const int g = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = s.seg_count[g];
    const int T = s.seg_words[g];
    if (n == 0 || s.totals[2] != 0) { if (tid == 0) s.seg_kept[g] = 0; return; }
    const unsigned long long* m = mask + s.mask_off[g];
    unsigned long long* kb = keepbits + s.keep_off[g];
    for (int w = tid; w < T; w += kSweepThreads) removed[w] = 0;
    // asynchronous copy of block b's tile: rows 64b .. 64b+nb-1, words b .. T-1 -> dst[row * Wn + col]
    auto stage = [&](int b, unsigned long long* dst) {
        const int nb = min(64, n - b * 64), Wn = T - b;
        for (int row = warp; row < nb; row += kSweepThreads / 32) {
            const unsigned long long* src = m + (long long)(b * 64 + row) * T + b;
            unsigned long long* d = dst + row * Wn;
            for (int col = lane; col < Wn; col += 32) {
                const unsigned da = (unsigned)__cvta_generic_to_shared(d + col);
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" :: "r"(da), "l"(src + col) : "memory");
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // ring of nbuf tile buffers: tiles b+1 .. b+nbuf-1 are in flight while block b is resolved, so the global-load
    // latency of a tile (the dominant cost of a block step) is spread over nbuf-1 steps
    const size_t tile_words = (size_t)64 * Tcap;
    for (int q = 0; q < nbuf - 1; ++q) {
        if (q < T) stage(q, tiles + q * tile_words);
        else asm volatile("cp.async.commit_group;" ::: "memory");     // keep one group per step for the wait arithmetic
    }
    if (nbuf == 1) stage(0, tiles);
    int kept = 0;
    for (int b = 0; b < T; ++b) {
        const int nb = min(64, n - b * 64), Wn = T - b;
        unsigned long long* tile = tiles + (size_t)(b % nbuf) * tile_words;
        // groups committed so far: tiles 0 .. b+nbuf-2 (one per step); tile b is complete when at most nbuf-2 are pending
        if (nbuf >= 4) asm volatile("cp.async.wait_group 2;" ::: "memory");
        else if (nbuf == 3) asm volatile("cp.async.wait_group 1;" ::: "memory");
        else asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();                                   // tile b complete and visible; buffer (b-1) % nbuf is free
        if (nbuf > 1) {
            if (b + nbuf - 1 < T) stage(b + nbuf - 1, tiles + (size_t)((b + nbuf - 1) % nbuf) * tile_words);
            else asm volatile("cp.async.commit_group;" ::: "memory");
        }
        if (warp == 0) {
            const unsigned long long invalid = nb < 64 ? ~((1ull << nb) - 1ull) : 0ull;
            unsigned long long R = removed[b] | invalid, C = 0;
            const int t0 = lane, t1 = lane + 32;
            const unsigned long long s0 = (t0 < nb) ? (tile[t0 * Wn] & ((1ull << t0) - 1ull)) : 0ull;
            const unsigned long long s1 = (t1 < nb) ? (tile[t1 * Wn] & ((1ull << t1) - 1ull)) : 0ull;
            while ((C | R) != ~0ull) {
                const unsigned long long D = C | R;
                bool c0 = false, r0 = false, c1 = false, r1 = false;
                if (!((D >> t0) & 1ull)) { if (s0 & C) r0 = true; else if ((s0 & ~R) == 0ull) c0 = true; }
                if (!((D >> t1) & 1ull)) { if (s1 & C) r1 = true; else if ((s1 & ~R) == 0ull) c1 = true; }
                C |= (unsigned long long)__ballot_sync(0xffffffffu, c0) | ((unsigned long long)__ballot_sync(0xffffffffu, c1) << 32);
                R |= (unsigned long long)__ballot_sync(0xffffffffu, r0) | ((unsigned long long)__ballot_sync(0xffffffffu, r1) << 32);
            }
            unsigned long long keepw = C;
            if (max_keep > 0 && kept + __popcll(keepw) > max_keep) {
                int extra = kept + __popcll(keepw) - max_keep;
                while (extra-- > 0) keepw &= ~(1ull << (63 - __clzll(keepw)));
            }
            if (lane == 0) { s_keepw = keepw; kb[b] = keepw; }
        }
        __syncthreads();
        const unsigned long long keepw = s_keepw;
        kept += __popcll(keepw);
        if (max_keep > 0 && kept >= max_keep) {
            for (int w = b + 1 + tid; w < T; w += kSweepThreads) kb[w] = 0ull;
            break;
        }
        // removed[b + col] |= OR of the kept rows' words: thread = (column, quarter of the rows), 64 columns per pass
        for (int c0 = 1; c0 < Wn; c0 += kSweepThreads / 4) {
            const int col = c0 + (tid >> 2), q = tid & 3;
            unsigned long long acc = 0;
            if (col < Wn) {
                unsigned long long bits = (keepw >> (16 * q)) & 0xffffull;
                while (bits) {
                    const int t = __ffsll((long long)bits) - 1 + 16 * q; bits &= bits - 1;
                    acc |= tile[t * Wn + col];
                }
            }
            acc |= __shfl_xor_sync(0xffffffffu, acc, 1);
            acc |= __shfl_xor_sync(0xffffffffu, acc, 2);
            if (q == 0 && col < Wn && acc) removed[b + col] |= acc;
        }
        if (nbuf == 1) {
            __syncthreads();                               // everyone is done with the tile before it is overwritten
            if (b + 1 < T) stage(b + 1, tiles);
        }
        // nbuf > 1: the barrier at the top of the next iteration orders this OR phase before block b+1's resolve
    }
    if (tid == 0) s.seg_kept[g] = kept;
}

// ------------------------------------------------------------------------------------
// sweep for segments of up to 1024 boxes (T <= 16 words), the RPN (image x level) and detection (image x class)
// case: greedy NMS is the unique fixed point of "kept iff every earlier overlapping box is removed; removed iff one of
// them is kept" (the lowest undecided box is always decidable), so instead of resolving 64 boxes at a time in order,
// every box of the segment iterates on it at once: thread t keeps its suppressor words (row t of the full mask, bits
// below t) in registers, the kept / removed sets live in shared memory as one 32-bit half-word per warp, and a round
// costs one barrier. Rounds = longest suppression chain of the segment (a handful for detector output; the worst case,
// a chain through all n boxes, takes n rounds and is still exact). Needs k_nms_mask(full = 1).
// ------------------------------------------------------------------------------------
constexpr int kFixThreads = 1024;
constexpr int kFixWords = kFixThreads / 64;

static __global__ void __launch_bounds__(kFixThreads) k_nms_fixpoint(SegArrays s, const unsigned long long* __restrict__ mask,
                                                                     unsigned long long* __restrict__ keepbits, int max_keep) {
    pdl_enter();
    __shared__ __align__(8) unsigned int C32[2 * kFixWords], R32[2 * kFixWords];
    const int g = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int n = s.seg_count[g];
    const int T = s.seg_words[g];
    if (n == 0 || s.totals[2] != 0) { if (t == 0) s.seg_kept[g] = 0; return; }
    const unsigned long long* m = mask + s.mask_off[g] + t;      // word-major mask: word w of box t at m[w * n]
    unsigned long long* kb = keepbits + s.keep_off[g];
    const int nw = min((warp >> 1) + 1, T);                 // words holding boxes before this warp's (warp-uniform)
    unsigned long long S[kFixWords];
#pragma unroll
    for (int w = 0; w < kFixWords; ++w) S[w] = (w < nw && t < n) ? m[(long long)w * n] : 0ull;
#pragma unroll
    for (int w = 0; w < kFixWords; ++w)
        if (w == (t >> 6)) S[w] &= (1ull << (t & 63)) - 1ull;
    bool decided = t >= n;
    {
        const unsigned int inv = __ballot_sync(0xffffffffu, decided);
        if (lane == 0) { C32[warp] = 0u; R32[warp] = inv; }
    }
    __syncthreads();
    const unsigned long long* Cw = reinterpret_cast<const unsigned long long*>(C32);
    const unsigned long long* Rw = reinterpret_cast<const unsigned long long*>(R32);
    while (true) {
        bool k = false, r = false;
        if (!decided) {
            bool hit = false, open = false;
#pragma unroll
            for (int w = 0; w < kFixWords; ++w) {
                if (w < nw) {
                    const unsigned long long c = Cw[w], rr = Rw[w];
                    hit |= (S[w] & c) != 0ull;
                    open |= (S[w] & ~rr) != 0ull;
                }
            }
            r = hit;
            k = !hit && !open;
        }
        const unsigned int bk = __ballot_sync(0xffffffffu, k), br = __ballot_sync(0xffffffffu, r);
        if (lane == 0 && (bk | br)) { C32[warp] |= bk; R32[warp] |= br; }     // a warp owns its half-word: no atomics
        decided = decided || k || r;
        // (a warp that runs ahead may publish round i+1 facts while another still reads round i: the sets only grow
        // by true facts, so any interleaving converges to the same fixed point)
        if (!__syncthreads_or(!decided)) break;
    }
    if (t == 0) {
        int kept = 0;
        for (int b = 0; b < T; ++b) {
            unsigned long long keepw = Cw[b];
            if (max_keep > 0) {
                if (kept >= max_keep) keepw = 0ull;
                else if (kept + __popcll(keepw) > max_keep) {
                    int extra = kept + __popcll(keepw) - max_keep;     // trim to exactly max_keep kept boxes
                    while (extra-- > 0) keepw &= ~(1ull << (63 - __clzll(keepw)));
                }
            }
            kb[b] = keepw;
            kept += __popcll(keepw);
        }
        s.seg_kept[g] = kept;
    }
}

// MB_NMS_SWEEP=blocks keeps the 64-box block sweeps for every segment size (development A/B switch).
// This helper and launch_mask_and_sweep are static like the kernels: each translation unit that includes this header
// launches its own copies of the sweep kernels, so it must also keep its own function-local statics (the cached switch,
// the per-device shared-memory opt-in of MB_DYN_SMEM) instead of sharing one weak definition with the other units.
static inline bool sweep_in_order() {
    static const bool v = [] { const char* e = getenv("MB_NMS_SWEEP"); return e != nullptr && e[0] == 'b'; }();
    return v;
}

inline int sweep_smem_bytes(int max_words) { return max_words * (int)sizeof(unsigned long long); }

// Host helper: launch meta + mask + sweep on prepared sorted boxes.
static inline int launch_mask_and_sweep(const float4* sbox, SegArrays s, int G, int max_seg_elems, double iou_threshold,
                                 unsigned long long* mask, unsigned long long* keepbits, int max_keep,
                                 cudaStream_t stream, const float* seg_offset = nullptr) {
    const float thr_up = strict_gt_threshold(iou_threshold);
    const bool fix = max_seg_elems <= kFixThreads && !sweep_in_order();
    MB_CUDA(launch_pdl(k_nms_mask, num_sms() * 16, 128, 0, stream, sbox, s, G, thr_up, mask, seg_offset, fix ? 1 : 0));
    if (fix) {
        MB_CUDA(launch_pdl(k_nms_fixpoint, G, kFixThreads, 0, stream, s, mask, keepbits, max_keep));
        return MB_OK;
    }
    // (the cp.async ring kernel below measured 8-12 % slower than this one at <= 4096 boxes, at every ring depth)
    if (ceil_div(max_seg_elems, 64) <= kSweepSmallMaxWords) {
        k_nms_sweep_small<<<G, kSweepThreads, 0, stream>>>(s, mask, keepbits, max_keep);
        MB_LAUNCH_CHECK();
        return MB_OK;
    }
    {   // tiled sweep with a ring of cp.async tile buffers in dynamic shared memory: removed[] + nbuf 64-row tiles
        const int Tcap = ceil_div(max_seg_elems, 64);
        int nbuf = 4;
        while (nbuf > 1 && ((long long)Tcap + 64ll * nbuf * Tcap) * 8 > 200 * 1024) --nbuf;
        const long long bytes = ((long long)Tcap + 64ll * nbuf * Tcap) * 8;
        if (bytes <= 200 * 1024) {
            MB_DYN_SMEM(k_nms_sweep_wide, (int)bytes);
            k_nms_sweep_wide<<<G, kSweepThreads, (int)bytes, stream>>>(s, mask, keepbits, max_keep, Tcap, nbuf);
            MB_LAUNCH_CHECK();
            return MB_OK;
        }
    }
    const int smem = sweep_smem_bytes(ceil_div(max_seg_elems, 64) + 1);
    if (smem > 48 * 1024) {
        if (smem > 200 * 1024) return MB_ERR_UNSUPPORTED;
        MB_DYN_SMEM(k_nms_sweep, smem);
    }
    k_nms_sweep<<<G, kSweepBigThreads, smem, stream>>>(s, mask, keepbits, max_keep);
    MB_LAUNCH_CHECK();
    return MB_OK;
}

}  // namespace mb
