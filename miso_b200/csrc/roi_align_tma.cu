// roi_align_tma.cu — MultiScaleRoIAlign forward for channels-last fp32 maps: a persistent, warp-specialised
// kernel that stages every RoI's footprint through TMA bulk copies into a shared-memory ring.
//
// Replaces tv:ops/poolers.py:147-227 + torchvision::roi_align (tv-csrc:ops/cpu/roi_align_kernel.cpp:393,
// SURVEY.md Appendix B.2) on the fast route of mb_multiscale_roi_align (sampling_ratio 2, aligned=False).
//
// Why: the gather kernel (k_roi_align_nhwc4d) was latency-bound — each warp had 9 LDG.128 in flight and waited
// for them (profiles/r1_roi_align_nhwc4d_ncu_full.txt: 35 % resident warps, 42 % of stalls on the first use
// after the loads) — and pulled every pixel 2.3x through L1 because neighbouring bins share taps. Here
//   * k_roi_geom (pre-pass, one warp per RoI, lanes = samples) writes every RoI's tap tables — level, footprint,
//     the list of touched pixel rows, per pooled row / column the distinct taps, weights and sharing pattern —
//     as one 2 KB record into the workspace: ~5 us of serial geometry per RoI that must not sit on the main
//     kernel's producer warp (measured: with the geometry inside it, the kernel's skeleton alone took 0.19 ms);
//   * k_roi_align_tma: one CTA per SM (grid = #SMs), RoIs round-robin; 16 warps: 14 consumers, 1 producer,
//     1 store warp;
//   * the producer is a pure TMA issuer: it prefetches the records of the next RoIs (bulk copy, 4-slot ring) and
//     streams the touched pixel rows of each footprint — in channels-last memory a footprint row is ONE
//     contiguous run of FW*C*4 bytes — with cp.async.bulk into a byte ring in shared memory, each row on its
//     own mbarrier; no registers are held per byte in flight and the copies run ahead across RoI boundaries;
//   * consumer warps walk the pooled rows in order; task = (bin, 128 channels), lane = 4 consecutive channels:
//     the distinct taps of the bin (3x3 typically) are LDS.128 from the ring, the 16 weight x value products
//     keep the reference order (exact mode: packed FMUL2 + FFMA2 with an opaque multiplier 1.0f, which is an
//     exactly rounded add that ptxas cannot contract with the multiply) or use FMAs;
//     rows are released (per-row "empty" mbarrier) as soon as no later pooled row needs them;
//   * the RoI's outputs are collected in shared memory in the output layout [C][PH*PW] (double buffered) and
//     leave as one bulk async copy issued by the store warp.
// Every pixel row crosses L2->SM once per RoI, and the loads are decoupled from the arithmetic.
#include <stdlib.h>

#include "common.cuh"
#include "roi_common.cuh"

namespace mb {

constexpr int kTmaConsumers = 14;
constexpr int kTmaThreads = (kTmaConsumers + 2) * 32;
constexpr int kRowSlots = 64;     // row descriptors / barriers in flight
constexpr int kMaxPool = 16;
constexpr int kGeomSlots = 4;     // records resident in shared memory (prefetched ahead of the consumers)

struct __align__(16) TmaGeom {      // one RoI's tap tables
    int mode;                // 0: zeros, 1: rows staged by TMA, 2: direct global gathers (rows wider than the ring allows)
    int nrows;               // staged rows (mode 1)
    unsigned rowbytes;       // bytes of one staged row = footprint width * C * 4
    int level;
    unsigned long long img;  // address of the image's map at the RoI's level
    unsigned long long pad2;
    int4 yidx[kMaxPool];     // 4 row slots of a pooled row: ordinals of the staged rows (mode 1) / byte offsets y*W*C*4 (mode 2)
    float4 ywa[kMaxPool];    // (h0, h0, l0, l0)
    float4 ywb[kMaxPool];    // (h1, h1, l1, l1)
    uint4 xoff[kMaxPool];    // 4 column slots of a pooled column: byte offsets inside the staged row / the map row
    float4 xwa[kMaxPool];
    float4 xwb[kMaxPool];
    int yinfo[kMaxPool];     // pattern (0..2) | valid bits << 2 | rows that must have landed << 8 | rows releasable afterwards << 16
    int xinfo[kMaxPool];     // pattern | valid bits << 2
    unsigned rowsrc[kRowSlots];   // mode 1: byte offset from img of the first footprint pixel of every staged row
};
static_assert(sizeof(TmaGeom) % 16 == 0, "records are moved with bulk copies");

// ---- mbarrier / bulk-copy primitives (PTX) ----
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// try_wait: plain (returns after a short hardware-defined time, the caller polls) or with a suspend-time hint (the
// thread sleeps in hardware until the phase completes or the hint expires; NANOSLEEP.SYNCS in SASS).
__device__ __forceinline__ bool mbar_try_wait(unsigned bar, unsigned parity) {
    unsigned ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ bool mbar_try_wait_hint(unsigned bar, unsigned parity, unsigned ns) {
    unsigned ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"(ns)
        : "memory");
    return ok != 0;
}
// A wait that cannot hang the GPU: a barrier that never completes (a protocol bug) traps after seconds.
// sleep_ns > 0: suspend-hint variant.
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity, unsigned sleep_ns = 0) {
    unsigned spins = 0;
    if (sleep_ns) {
        while (!mbar_try_wait_hint(bar, parity, sleep_ns)) {
            if (++spins > (1u << 22)) __trap();
        }
    } else {
        while (!mbar_try_wait(bar, parity)) {
            if (++spins > (1u << 24)) __trap();
        }
    }
}
__device__ __forceinline__ void st_shared(unsigned addr, float v) {
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
// Warp-level wait: one lane polls, __syncwarp() releases the others. An mbarrier operation issued by all 32 lanes
// costs ~32 cycles of the SM's shared-memory atomic path (measured: with every lane of 14 consumer warps polling,
// the barrier traffic alone bounded the kernel at ~5.7 us per RoI); shared memory has no per-thread caches, so the
// lanes released by the warp barrier read what the polling lane was allowed to read.
__device__ __forceinline__ void mbar_wait_warp(unsigned bar, unsigned parity, int lane, unsigned sleep_ns = 0) {
    if (lane == 0) mbar_wait(bar, parity, sleep_ns);
    __syncwarp();
}
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* dst, unsigned src, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n\tcp.async.bulk.commit_group;" ::"l"(dst),
                 "r"(src), "r"(bytes)
                 : "memory");
}

// one tap of 4 consecutive channels; RowT = unsigned (shared-memory address) or const char* (global)
__device__ __forceinline__ float4 tap_ld(unsigned row, unsigned off) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(row + off));
    return v;
}
__device__ __forceinline__ float4 tap_ld(const char* row, unsigned off) {
    return __ldg(reinterpret_cast<const float4*>(row + off));
}

// the reference's per-sample sum for two channels: acc + (((w1*v1 + w2*v2) + w3*v3) + w4*v4)
template <bool EXACT>
__device__ __forceinline__ float2 sample2(float2 w1, float2 w2, float2 w3, float2 w4, float2 v1, float2 v2, float2 v3,
                                          float2 v4, float2 acc, float2 ones) {
    if (EXACT) {
        // fma(p, 1.0f, t) == fl(p + t): every product and every sum is rounded once, like the CPU kernel. `ones`
        // comes from the kernel parameters, so ptxas can neither fold it nor contract the multiply into the add.
        float2 t = mul2_rn(w1, v1);
        t = fma2_rn(mul2_rn(w2, v2), ones, t);
        t = fma2_rn(mul2_rn(w3, v3), ones, t);
        t = fma2_rn(mul2_rn(w4, v4), ones, t);
        return fma2_rn(t, ones, acc);
    } else {
        return fma2_rn(w1, v1, fma2_rn(w2, v2, fma2_rn(w3, v3, fma2_rn(w4, v4, acc))));
    }
}

// the 16 weight products of a bin, w[4 * sample + corner] (each duplicated for the packed arithmetic): computed once
// per bin and shared by every 128-channel pass over it
__device__ __forceinline__ void bin_weights(const float2 (&wy)[4], const float2 (&wx)[4], float2 (&W)[16]) {
#pragma unroll
    for (int smp = 0; smp < 4; ++smp) {
        const int iy = smp >> 1, ix = smp & 1;
        const float2 hyv = wy[2 * iy], lyv = wy[2 * iy + 1], hxv = wx[2 * ix], lxv = wx[2 * ix + 1];
        W[4 * smp + 0] = mul2_rn(hyv, hxv); W[4 * smp + 1] = mul2_rn(hyv, lxv);
        W[4 * smp + 2] = mul2_rn(lyv, hxv); W[4 * smp + 3] = mul2_rn(lyv, lxv);
    }
}

// All four samples valid: the 16 taps are the product of the bin's distinct rows and columns (patterns of
// axis_pattern: 0 = both samples in one cell, 1 = they share a pixel, 2 = four pixels); each distinct pixel is loaded once.
template <bool EXACT, int PY, int PX, typename RowT>
__device__ __forceinline__ float4 bin_fast(const RowT (&rb)[4], const unsigned (&co)[4], const float2 (&W)[16], float2 ones) {
    constexpr int NR = PY == 0 ? 2 : (PY == 1 ? 3 : 4), NC = PX == 0 ? 2 : (PX == 1 ? 3 : 4);
    float4 G[NR][NC];
#pragma unroll
    for (int r = 0; r < NR; ++r)
#pragma unroll
        for (int c = 0; c < NC; ++c) G[r][c] = tap_ld(rb[r], co[c]);
    float2 lo = make_float2(0.f, 0.f), hi = make_float2(0.f, 0.f);
#pragma unroll
    for (int smp = 0; smp < 4; ++smp) {
        const int iy = smp >> 1, ix = smp & 1;
        const int yl = iy == 0 ? 0 : (PY == 0 ? 0 : (PY == 1 ? 1 : 2)), yh = iy == 0 ? 1 : (PY == 0 ? 1 : (PY == 1 ? 2 : 3));
        const int xl = ix == 0 ? 0 : (PX == 0 ? 0 : (PX == 1 ? 1 : 2)), xh = ix == 0 ? 1 : (PX == 0 ? 1 : (PX == 1 ? 2 : 3));
        const float4 v1 = G[yl][xl], v2 = G[yl][xh], v3 = G[yh][xl], v4 = G[yh][xh];
        lo = sample2<EXACT>(W[4 * smp], W[4 * smp + 1], W[4 * smp + 2], W[4 * smp + 3], make_float2(v1.x, v1.y),
                            make_float2(v2.x, v2.y), make_float2(v3.x, v3.y), make_float2(v4.x, v4.y), lo, ones);
        hi = sample2<EXACT>(W[4 * smp], W[4 * smp + 1], W[4 * smp + 2], W[4 * smp + 3], make_float2(v1.z, v1.w),
                            make_float2(v2.z, v2.w), make_float2(v3.z, v3.w), make_float2(v4.z, v4.w), hi, ones);
    }
    const float2 q = make_float2(0.25f, 0.25f);     // acc / 4 samples: exact scaling
    lo = mul2_rn(lo, q);
    hi = mul2_rn(hi, q);
    return make_float4(lo.x, lo.y, hi.x, hi.y);
}

// Any sample may be invalid (skipped like the reference does — no zero-weight multiply, so a NaN/Inf feature
// never leaks into a bin it does not belong to).
template <typename T>
__device__ __forceinline__ T slot_sel(const T (&a)[4], int i) {      // a[i] without dynamic register indexing
    return i == 0 ? a[0] : (i == 1 ? a[1] : (i == 2 ? a[2] : a[3]));
}

template <bool EXACT, typename RowT>
__device__ __forceinline__ float4 bin_generic(const RowT (&rb)[4], const unsigned (&co)[4], const float2 (&W)[16], int py, int px,
                                              int yvalid, int xvalid, float2 ones) {
    float2 lo = make_float2(0.f, 0.f), hi = make_float2(0.f, 0.f);
#pragma unroll
    for (int smp = 0; smp < 4; ++smp) {
        const int iy = smp >> 1, ix = smp & 1;
        if (!((yvalid >> iy) & 1) || !((xvalid >> ix) & 1)) continue;       // warp-uniform
        // slots of the second sample follow the axis pattern: (0,1), (1,2) or (2,3)
        const int ys = iy ? py : 0, xs = ix ? px : 0;
        const RowT rlo = slot_sel(rb, ys), rhi = slot_sel(rb, ys + 1);
        const unsigned clo = slot_sel(co, xs), chi = slot_sel(co, xs + 1);
        const float4 v1 = tap_ld(rlo, clo), v2 = tap_ld(rlo, chi);
        const float4 v3 = tap_ld(rhi, clo), v4 = tap_ld(rhi, chi);
        lo = sample2<EXACT>(W[4 * smp], W[4 * smp + 1], W[4 * smp + 2], W[4 * smp + 3], make_float2(v1.x, v1.y),
                            make_float2(v2.x, v2.y), make_float2(v3.x, v3.y), make_float2(v4.x, v4.y), lo, ones);
        hi = sample2<EXACT>(W[4 * smp], W[4 * smp + 1], W[4 * smp + 2], W[4 * smp + 3], make_float2(v1.z, v1.w),
                            make_float2(v2.z, v2.w), make_float2(v3.z, v3.w), make_float2(v4.z, v4.w), hi, ones);
    }
    const float2 q = make_float2(0.25f, 0.25f);
    lo = mul2_rn(lo, q);
    hi = mul2_rn(hi, q);
    return make_float4(lo.x, lo.y, hi.x, hi.y);
}

// One warp builds one RoI's record (lanes = samples along each axis).
__device__ __forceinline__ void build_geom(const mb_roi_align_params& p, const float* __restrict__ rois, int k,
                                           unsigned row_cap, int lane, TmaGeom& G, int* __restrict__ levels_out) {
    const unsigned full = 0xffffffffu;
    const int PH = p.pooled_h, PW = p.pooled_w, C = p.channels;
    float r[5];
    load_roi(rois, k, p, r);
    RoiGeom g;
    roi_geometry(r, p, g);
    if (levels_out != nullptr && lane == 0) levels_out[k] = g.level;
    const bool dead = g.batch < 0 || g.batch >= p.num_images;
    Tap tx = make_tap(g.start_w, g.bin_w, lane >> 1, lane & 1, 2, g.W);
    if (lane >= 2 * PW) tx.valid = 0;
    const unsigned xm = __ballot_sync(full, tx.valid != 0);
    Tap ty = make_tap(g.start_h, g.bin_h, lane >> 1, lane & 1, 2, g.H);
    if (lane >= 2 * PH) ty.valid = 0;
    const unsigned ym = __ballot_sync(full, ty.valid != 0);
    int mode = (dead || xm == 0 || ym == 0) ? 0 : 1;
    int x0 = 0, fw = 0, nrows = 0;
    if (mode != 0) {
        const int fx = __ffs(xm) - 1, lx = 31 - __clz(xm), fy = __ffs(ym) - 1, ly = 31 - __clz(ym);
        x0 = __shfl_sync(full, tx.lo, fx);
        fw = __shfl_sync(full, tx.hi, lx) - x0 + 1;
        // valid samples must be one run with non-decreasing pixel indices (bin size > 0 guarantees it);
        // anything else takes the direct route, which does not rely on it
        const int plo_x = __shfl_up_sync(full, tx.lo, 1), plo_y = __shfl_up_sync(full, ty.lo, 1);
        const int phi_x = __shfl_up_sync(full, tx.hi, 1), phi_y = __shfl_up_sync(full, ty.hi, 1);
        const bool bad = (tx.valid && lane > fx && (tx.lo < plo_x || tx.hi < phi_x)) ||
                         (ty.valid && lane > fy && (ty.lo < plo_y || ty.hi < phi_y)) ||
                         (lane >= fx && lane <= lx && !tx.valid) || (lane >= fy && lane <= ly && !ty.valid) ||
                         (tx.valid && (tx.hi < tx.lo || tx.hi > tx.lo + 1)) || (ty.valid && (ty.hi < ty.lo || ty.hi > ty.lo + 1));
        const bool irregular = __any_sync(full, bad);
        const unsigned long long rowbytes = (unsigned long long)fw * C * 4ull;
        if (irregular || fw < 1 || rowbytes > row_cap) mode = 2;
        // ---- y axis: ordinals of the touched rows ----
        const int hp_ = (lane == fy) ? -0x40000000 : phi_y;
        const bool new_lo = ty.valid && ty.lo > hp_;
        const bool new_hi = ty.valid && ty.hi > ty.lo && ty.hi > hp_;
        const int cnt = (int)new_lo + (int)new_hi;
        int incl = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int v = __shfl_up_sync(full, incl, d);
            if (lane >= d) incl += v;
        }
        const int base = incl - cnt;
        nrows = __shfl_sync(full, incl, 31);
        const int ord_lo = new_lo ? base : base - (hp_ - ty.lo + 1);
        const int ord_hi = new_hi ? base + (int)new_lo : (ty.hi == ty.lo ? ord_lo : base - 1);
        if (mode == 1) {      // byte offset of the row's first footprint pixel
            if (new_lo) G.rowsrc[base] = ((unsigned)ty.lo * (unsigned)g.W + (unsigned)x0) * (unsigned)C * 4u;
            if (new_hi) G.rowsrc[base + (int)new_lo] = ((unsigned)ty.hi * (unsigned)g.W + (unsigned)x0) * (unsigned)C * 4u;
        }
        const unsigned rowpitch = (unsigned)g.W * (unsigned)C * 4u;
        // per-sample slot values
        const int ylo_v = !ty.valid ? 0 : (mode == 1 ? ord_lo : (int)((unsigned)ty.lo * rowpitch));
        const int yhi_v = !ty.valid ? 0 : (mode == 1 ? ord_hi : (int)((unsigned)ty.hi * rowpitch));
        const unsigned xlo_v = !tx.valid ? 0u : (unsigned)(tx.lo - (mode == 1 ? x0 : 0)) * (unsigned)C * 4u;
        const unsigned xhi_v = !tx.valid ? 0u : (unsigned)(tx.hi - (mode == 1 ? x0 : 0)) * (unsigned)C * 4u;
        // lane q < PH / PW gathers its two samples (lanes 2q, 2q+1)
        const int sa = (2 * lane) & 31, sb = (2 * lane + 1) & 31;
        {   // y
            const int alo = __shfl_sync(full, ty.lo, sa), ahi = __shfl_sync(full, ty.hi, sa);
            const int blo = __shfl_sync(full, ty.lo, sb), bhi = __shfl_sync(full, ty.hi, sb);
            const int av = __shfl_sync(full, ty.valid, sa), bv = __shfl_sync(full, ty.valid, sb);
            const int a_lo = __shfl_sync(full, ylo_v, sa), a_hi = __shfl_sync(full, yhi_v, sa);
            const int b_lo = __shfl_sync(full, ylo_v, sb), b_hi = __shfl_sync(full, yhi_v, sb);
            const float ah = __shfl_sync(full, ty.h, sa), al = __shfl_sync(full, ty.l, sa);
            const float bh = __shfl_sync(full, ty.h, sb), bl = __shfl_sync(full, ty.l, sb);
            const int a_ord_hi = __shfl_sync(full, ord_hi, sa), b_ord_hi = __shfl_sync(full, ord_hi, sb);
            // first valid sample after this pooled row -> rows below its low row can be released
            const unsigned later = (2 * lane + 2 < 32) ? (ym & ~((1u << (2 * lane + 2)) - 1u)) : 0u;
            const int nxt = later ? (__ffs(later) - 1) : 0;
            const int nxt_ord = __shfl_sync(full, ord_lo, nxt);
            if (lane < PH) {
                int pat = 2;
                int4 idx = make_int4(a_lo, a_hi, b_lo, b_hi);
                if (av && bv && mode == 1) {
                    if (blo == alo && bhi == ahi) pat = 0;
                    else if (blo == ahi) { pat = 1; idx.z = b_hi; }
                }
                const int need = bv ? b_ord_hi + 1 : (av ? a_ord_hi + 1 : 0);
                const int rel = later ? nxt_ord : nrows;
                G.yidx[lane] = idx;
                G.ywa[lane] = make_float4(ah, ah, al, al);
                G.ywb[lane] = make_float4(bh, bh, bl, bl);
                G.yinfo[lane] = pat | ((av ? 1 : 0) << 2) | ((bv ? 1 : 0) << 3) | (need << 8) | (rel << 16);
            }
        }
        {   // x
            const int alo = __shfl_sync(full, tx.lo, sa), ahi = __shfl_sync(full, tx.hi, sa);
            const int blo = __shfl_sync(full, tx.lo, sb), bhi = __shfl_sync(full, tx.hi, sb);
            const int av = __shfl_sync(full, tx.valid, sa), bv = __shfl_sync(full, tx.valid, sb);
            const unsigned a_lo = __shfl_sync(full, xlo_v, sa), a_hi = __shfl_sync(full, xhi_v, sa);
            const unsigned b_lo = __shfl_sync(full, xlo_v, sb), b_hi = __shfl_sync(full, xhi_v, sb);
            const float ah = __shfl_sync(full, tx.h, sa), al = __shfl_sync(full, tx.l, sa);
            const float bh = __shfl_sync(full, tx.h, sb), bl = __shfl_sync(full, tx.l, sb);
            if (lane < PW) {
                int pat = 2;
                uint4 idx = make_uint4(a_lo, a_hi, b_lo, b_hi);
                if (av && bv && mode == 1) {
                    if (blo == alo && bhi == ahi) pat = 0;
                    else if (blo == ahi) { pat = 1; idx.z = b_hi; }
                }
                G.xoff[lane] = idx;
                G.xwa[lane] = make_float4(ah, ah, al, al);
                G.xwb[lane] = make_float4(bh, bh, bl, bl);
                G.xinfo[lane] = pat | ((av ? 1 : 0) << 2) | ((bv ? 1 : 0) << 3);
            }
        }
    }
    const char* img = reinterpret_cast<const char*>(p.features[g.level]) +
                      (dead ? 0ull : (unsigned long long)g.batch * g.H * g.W * C * 4ull);
    if (lane == 0) {
        G.mode = mode;
        G.nrows = mode == 1 ? nrows : 0;
        G.rowbytes = (unsigned)fw * (unsigned)C * 4u;
        G.level = g.level;
        G.img = reinterpret_cast<unsigned long long>(img);
        G.pad2 = 0;
    }
}

// Pre-pass: the tap tables of every RoI, one warp each, written to the workspace.
__global__ void __launch_bounds__(256) k_roi_geom(const __grid_constant__ mb_roi_align_params p, const float* __restrict__ rois,
                                                 int num_rois, unsigned row_cap, TmaGeom* __restrict__ recs,
                                                 int* __restrict__ levels_out, int dbg) {
    const int k = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (k >= num_rois) return;
    build_geom(p, rois, k, row_cap, threadIdx.x & 31, recs[k], levels_out);
    if (dbg & 16) {                        // probe: RoIs on the direct route produce zeros instead
        __syncwarp();
        if ((threadIdx.x & 31) == 0 && recs[k].mode == 2) recs[k].mode = 0;
    }
}

struct TmaSmem {          // carve-up of the dynamic shared memory (offsets in bytes)
    unsigned ring, ob, geom, rowoff, cum, rel, bars, total;
};
__host__ __device__ inline TmaSmem tma_smem_layout(unsigned ring_bytes, unsigned ob_bytes) {
    TmaSmem s;
    s.ring = 0;
    s.ob = ring_bytes;
    s.geom = s.ob + 2 * ob_bytes;
    s.rowoff = s.geom + kGeomSlots * (unsigned)sizeof(TmaGeom);
    s.cum = s.rowoff + kRowSlots * 4;
    s.rel = s.cum + kRowSlots * 4;
    s.bars = s.rel + 16 * 4;
    s.total = s.bars + (kRowSlots + 2 * kGeomSlots + 4) * 8;
    return s;
}

template <bool EXACT>
__global__ void __launch_bounds__(kTmaThreads, 1)
k_roi_align_tma(const __grid_constant__ mb_roi_align_params p, const TmaGeom* __restrict__ recs, int num_rois,
                float* __restrict__ out, unsigned ring_bytes, float2 ones, int dbg) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int PH = p.pooled_h, PW = p.pooled_w, nbins = PH * PW, C = p.channels;
    const unsigned ob_bytes = (unsigned)C * nbins * 4u;
    const TmaSmem L = tma_smem_layout(ring_bytes, ob_bytes);
    TmaGeom* geom = reinterpret_cast<TmaGeom*>(smem_raw + L.geom);
    volatile int* rowoff = reinterpret_cast<volatile int*>(smem_raw + L.rowoff);
    const unsigned s_base = smem_u32(smem_raw);
    volatile unsigned* cumtab = reinterpret_cast<volatile unsigned*>(smem_raw + L.cum);     // bytes allocated up to and including row seq
    volatile int* relcnt = reinterpret_cast<volatile int*>(smem_raw + L.rel);              // per consumer warp: rows released so far
    const unsigned b_full = s_base + L.bars, b_gfull = b_full + kRowSlots * 8;
    const unsigned b_gempty = b_gfull + kGeomSlots * 8, b_ofull = b_gempty + kGeomSlots * 8, b_ofree = b_ofull + 16;

    if (tid == 0) {
        for (int i = 0; i < kRowSlots; ++i) {
            mbar_init(b_full + 8 * i, 1);
        }
        for (int i = 0; i < kGeomSlots; ++i) {
            mbar_init(b_gfull + 8 * i, 1);
            mbar_init(b_gempty + 8 * i, kTmaConsumers);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(b_ofull + 8 * i, kTmaConsumers);
            mbar_init(b_ofree + 8 * i, 1);
        }
        for (int i = 0; i < 16; ++i) relcnt[i] = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    const unsigned slp = ((unsigned)dbg >> 8) & 0xffffu;      // probe: suspend-time hint of the waits in ns (0 = poll)
    const int my_rois = blockIdx.x < num_rois ? (num_rois - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (warp == kTmaConsumers) {
        // =========================== producer: record prefetch + TMA row copies ===========================
        // The whole warp works on one RoI: lane j owns footprint row j. Placement in the FIFO byte ring has a closed
        // form (rows of one RoI have one size and never split: n1 rows fit before the wrap, then laps of nl rows), so the
        // lanes compute their offsets and "bytes allocated so far" in parallel; a row is issued once the byte credits
        // cover it. Consumers publish "rows released" in one word per warp; one poll (a load + a 5-step shuffle min)
        // can release several rows at once. A first version with a sequential allocator and an mbarrier wait per row,
        // all on one thread, took ~550 cycles per row and bounded the whole kernel.
        int next_seq = 0;                                  // rows issued so far
        unsigned head = 0, cum_head = 0;                   // ring write offset; bytes allocated so far (mod 2^32)
        unsigned spins = 0;
        auto fetch_record = [&](int j) {          // record of this CTA's j-th RoI -> slot j % kGeomSlots
            if (j >= my_rois) return;
            const int slot = j % kGeomSlots, use = j / kGeomSlots;
            if (lane == 0) {
                if (use >= 1) mbar_wait(b_gempty + 8 * slot, (use - 1) & 1, slp);        // consumers are done with the slot's previous record
                mbar_arrive_expect_tx(b_gfull + 8 * slot, (unsigned)sizeof(TmaGeom));
                bulk_g2s(s_base + L.geom + slot * (unsigned)sizeof(TmaGeom), recs + (blockIdx.x + (size_t)j * gridDim.x),
                         (unsigned)sizeof(TmaGeom), b_gfull + 8 * slot);
            }
        };
        // Records are fetched two RoIs ahead into a 4-slot ring: the slot reused at iteration `it` held RoI it-2.
        for (int j = 0; j < kGeomSlots - 2; ++j) fetch_record(j);
        for (int it = 0; it < my_rois; ++it) {
            fetch_record(it + kGeomSlots - 2);
            const int gs = it % kGeomSlots;
            mbar_wait_warp(b_gfull + 8 * gs, (it / kGeomSlots) & 1, lane, slp);
            const TmaGeom& G = geom[gs];
            if (G.mode != 1) continue;
            const int nrows = G.nrows;
            const unsigned size = G.rowbytes;
            const char* img = reinterpret_cast<const char*>(G.img);
            const unsigned n1 = (ring_bytes - head) / size;            // rows that still fit before the ring wraps
            const unsigned nl = ring_bytes / size;                     // rows per lap after that
            const unsigned gap1 = ring_bytes - head - n1 * size, gapl = ring_bytes - nl * size;
            unsigned last_off = head, last_cum = cum_head;
            for (int j0 = 0; j0 < nrows; j0 += 32) {
                const unsigned j = (unsigned)(j0 + lane);
                bool pending = (int)j < nrows;
                unsigned off, cum_end;
                if (j < n1) { off = head + j * size; cum_end = cum_head + (j + 1) * size; }
                else {
                    const unsigned q = j - n1, lap = q / nl, pos = q - lap * nl;
                    off = pos * size;
                    cum_end = cum_head + (j + 1) * size + gap1 + lap * gapl;       // the skipped gaps are charged too
                }
                const int seq = next_seq + (int)j;
                const int slot = seq & (kRowSlots - 1);
                const unsigned src_off = pending ? G.rowsrc[j] : 0u;
                while (__any_sync(0xffffffffu, pending)) {
                    int m = lane < kTmaConsumers ? relcnt[lane] : 0x7fffffff;
#pragma unroll
                    for (int o = 16; o; o >>= 1) m = min(m, __shfl_xor_sync(0xffffffffu, m, o));
                    const unsigned cum_freed = m > 0 ? cumtab[(m - 1) & (kRowSlots - 1)] : 0u;
                    const bool ready = pending && (cum_end - cum_freed <= ring_bytes) && (seq - m < kRowSlots);
                    if (ready) {
                        cumtab[slot] = cum_end;
                        rowoff[slot] = (int)off;
                        if (dbg & 1) mbar_arrive(b_full + 8 * slot);          // probe: no copies
                        else {
                            mbar_arrive_expect_tx(b_full + 8 * slot, size);
                            bulk_g2s(s_base + L.ring + off, img + src_off, size, b_full + 8 * slot);
                        }
                        pending = false;
                    } else if (pending && ++spins > (1u << 26)) __trap();
                    __syncwarp();
                }
                const int last = min(nrows - j0, 32) - 1;               // lane of the last row of this group
                last_off = __shfl_sync(0xffffffffu, off, last);
                last_cum = __shfl_sync(0xffffffffu, cum_end, last);
            }
            head = last_off + size;
            cum_head = last_cum;
            next_seq += nrows;
        }
    } else if (warp == kTmaConsumers + 1) {
        // =========================== store warp: one bulk copy per RoI ===========================
        if (lane == 0) {
            for (int it = 0; it < my_rois; ++it) {
                const int b = it & 1;
                const size_t k = blockIdx.x + (size_t)it * gridDim.x;
                mbar_wait(b_ofull + 8 * b, (it >> 1) & 1, slp);
                if (!(dbg & 4)) bulk_s2g(out + k * C * nbins, s_base + L.ob + b * ob_bytes, ob_bytes);   // probe bit 2: no stores
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");      // the buffer may be rewritten
                mbar_arrive(b_ofree + 8 * b);
            }
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        }
    } else {
        // =========================== consumers ===========================
        // Task = one bin (ph, pw), ALL channels: the bin's control state (row waits, tap addresses, the 16 weight
        // products) is set up once and shared by the 128-channel passes (lane = 4 consecutive channels). Bins are dealt
        // round-robin to the warps and the deal continues across RoIs (49 bins over 14 warps: 4 / 3 per RoI, evened out
        // by the next RoI); warps only meet at the output hand-over.
        const int halves = (C + 127) >> 7;
        const int rot4 = lane >> 3;
        unsigned so4[4];                              // byte offsets of the rotated channel rows in the output buffer
#pragma unroll
        for (int t = 0; t < 4; ++t) so4[t] = (unsigned)(((rot4 + t) & 3) * nbins) * 4u;
        const unsigned ring_lane = s_base + L.ring + lane * 16;
        const int dph = kTmaConsumers / PW, dpw = kTmaConsumers - dph * PW;      // one task step in (ph, pw)
        const unsigned half_out = 128u * (unsigned)nbins * 4u;                    // output bytes per 128-channel pass
        int seq0 = 0;                                 // sequence number of the current RoI's first staged row
        int next_bin = warp;                          // this warp's first bin in the current RoI
        for (int it = 0; it < my_rois; ++it) {
            const int gs = it % kGeomSlots, b = it & 1, u = it >> 1;
            mbar_wait_warp(b_gfull + 8 * gs, (it / kGeomSlots) & 1, lane, slp);
            const TmaGeom& G = geom[gs];
            const int mode = G.mode, nrows = G.nrows;
            if (u >= 1) mbar_wait_warp(b_ofree + 8 * b, (u - 1) & 1, lane, slp);
            const unsigned ob_u32 = s_base + L.ob + b * ob_bytes;
            if (mode == 0) {
                float4* o4 = reinterpret_cast<float4*>(smem_raw + L.ob + b * ob_bytes);
                for (unsigned i = warp * 32 + lane; i < ob_bytes / 16; i += kTmaConsumers * 32) o4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            } else {
                int waited = 0, published = 0;
                const char* gimg = reinterpret_cast<const char*>(G.img) + lane * 16;
                int ph = next_bin / PW, pw = next_bin - ph * PW, cur_pw = -1;
                unsigned co[4];
                float2 wx[4];
                int px = 0, xv = 0;
                for (int bin = next_bin; bin < nbins; bin += kTmaConsumers) {
                    if (pw != cur_pw) {
                        cur_pw = pw;
                        const uint4 xo = G.xoff[pw];
                        const float4 xa = G.xwa[pw], xb = G.xwb[pw];
                        co[0] = xo.x; co[1] = xo.y; co[2] = xo.z; co[3] = xo.w;
                        wx[0] = make_float2(xa.x, xa.y); wx[1] = make_float2(xa.z, xa.w);
                        wx[2] = make_float2(xb.x, xb.y); wx[3] = make_float2(xb.z, xb.w);
                        const int xi = G.xinfo[pw];
                        px = xi & 3; xv = (xi >> 2) & 3;
                    }
                    const int yi = G.yinfo[ph];
                    const int need = (yi >> 8) & 0xff;
                    if (mode == 1) {
                        // Rows below the first one this bin (or any later one) needs can go — published BEFORE waiting for this
                        // bin's rows: a warp that starts at pooled row 1 must not pin row 0 while it waits (the ring may be
                        // too small to hold both), and the previous bin's taps have all been consumed (results stored).
                        const int keep_from = ph == 0 ? 0 : (G.yinfo[ph - 1] >> 16) & 0xff;
                        if (keep_from > published) {
                            __syncwarp();
                            if (lane == 0) relcnt[warp] = seq0 + keep_from;
                            published = keep_from;
                        }
                    }
                    if (mode == 1 && waited < need) {
                        if (lane == 0)
                            for (int q = waited; q < need; ++q) {
                                const int s = seq0 + q;
                                mbar_wait(b_full + 8 * (s & (kRowSlots - 1)), (s >> 6) & 1, slp);
                            }
                        __syncwarp();
                        waited = need;
                    }
                    const int4 yx = G.yidx[ph];
                    const float4 ya = G.ywa[ph], yb = G.ywb[ph];
                    const float2 wy[4] = {make_float2(ya.x, ya.y), make_float2(ya.z, ya.w), make_float2(yb.x, yb.y),
                                          make_float2(yb.z, yb.w)};
                    const int py = yi & 3, yv = (yi >> 2) & 3;
                    float2 W[16];
                    bin_weights(wy, wx, W);
                    const unsigned obin = ob_u32 + (unsigned)(4 * lane * nbins + bin) * 4u;
                    if (mode == 1) {
                        // slots of invalid samples are never read (their ordinals are 0: some staged row's offset)
                        unsigned rs[4];
                        rs[0] = ring_lane + (unsigned)rowoff[(seq0 + yx.x) & (kRowSlots - 1)];
                        rs[1] = ring_lane + (unsigned)rowoff[(seq0 + yx.y) & (kRowSlots - 1)];
                        rs[2] = ring_lane + (unsigned)rowoff[(seq0 + yx.z) & (kRowSlots - 1)];
                        rs[3] = ring_lane + (unsigned)rowoff[(seq0 + yx.w) & (kRowSlots - 1)];
                        const bool fast = yv == 3 && xv == 3;
                        const int pat = py * 3 + px;
                        for (int h = 0; h < ((dbg & 2) ? 0 : halves); ++h) {      // probe bit 1: no arithmetic
                            if (h * 128 + 4 * lane < C) {
                                float4 av;
                                if (fast) {
                                    switch (pat) {      // warp-uniform
                                        case 0: av = bin_fast<EXACT, 0, 0>(rs, co, W, ones); break;
                                        case 1: av = bin_fast<EXACT, 0, 1>(rs, co, W, ones); break;
                                        case 2: av = bin_fast<EXACT, 0, 2>(rs, co, W, ones); break;
                                        case 3: av = bin_fast<EXACT, 1, 0>(rs, co, W, ones); break;
                                        case 4: av = bin_fast<EXACT, 1, 1>(rs, co, W, ones); break;
                                        case 5: av = bin_fast<EXACT, 1, 2>(rs, co, W, ones); break;
                                        case 6: av = bin_fast<EXACT, 2, 0>(rs, co, W, ones); break;
                                        case 7: av = bin_fast<EXACT, 2, 1>(rs, co, W, ones); break;
                                        default: av = bin_fast<EXACT, 2, 2>(rs, co, W, ones); break;
                                    }
                                } else {
                                    av = bin_generic<EXACT>(rs, co, W, py, px, yv, xv, ones);
                                }
                                rotate4(av, rot4);
                                const unsigned o = obin + (unsigned)h * half_out;
                                st_shared(o + so4[0], av.x); st_shared(o + so4[1], av.y);
                                st_shared(o + so4[2], av.z); st_shared(o + so4[3], av.w);
                            }
                            rs[0] += 512u; rs[1] += 512u; rs[2] += 512u; rs[3] += 512u;      // next 128 channels of the same pixels
                        }
                    } else {
                        const char* rg[4] = {gimg + (unsigned)yx.x, gimg + (unsigned)yx.y, gimg + (unsigned)yx.z, gimg + (unsigned)yx.w};
                        for (int h = 0; h < halves; ++h) {
                            if (h * 128 + 4 * lane < C) {
                                float4 av = bin_generic<EXACT>(rg, co, W, py, px, yv, xv, ones);
                                rotate4(av, rot4);
                                const unsigned o = obin + (unsigned)h * half_out;
                                st_shared(o + so4[0], av.x); st_shared(o + so4[1], av.y);
                                st_shared(o + so4[2], av.z); st_shared(o + so4[3], av.w);
                            }
                            rg[0] += 512; rg[1] += 512; rg[2] += 512; rg[3] += 512;
                        }
                    }
                    ph += dph; pw += dpw;           // this warp's next bin
                    if (pw >= PW) { pw -= PW; ++ph; }
                }
            }
            if (mode == 1) {
                __syncwarp();
                if (lane == 0) relcnt[warp] = seq0 + nrows;      // (also for warps that had no bin in this RoI)
                seq0 += nrows;
            }
            next_bin = (next_bin >= nbins ? next_bin : next_bin + ((nbins - 1 - next_bin) / kTmaConsumers + 1) * kTmaConsumers) - nbins;
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");    // generic-proxy writes -> visible to the bulk copy
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(b_ofull + 8 * b);
                mbar_arrive(b_gempty + 8 * gs);
            }
        }
    }
}

}  // namespace mb

using namespace mb;

static long long g_tma_launches = 0;
extern "C" int64_t mb_roi_align_tma_launches(void) { return g_tma_launches; }
// SM count and opt-in shared memory per block of the current device, asked once per device
static bool tma_device_info(int& sms, int& smem) {
    static int cached_sms[64] = {}, cached_smem[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return false;
    if (cached_sms[dev] == 0) {
        int s = 0, m = 0;
        if (cudaDeviceGetAttribute(&m, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&s, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
            return false;
        cached_smem[dev] = m;
        cached_sms[dev] = s;             // racing first calls store the same values
    }
    sms = cached_sms[dev];
    smem = cached_smem[dev];
    return sms > 0;
}

// static part of the envelope (no device query): what mb_roi_align_workspace_bytes can decide
static bool tma_shape_ok(const mb_roi_align_params& p, int64_t num_rois) {
    const long long ob = (long long)p.channels * p.pooled_h * p.pooled_w * 4ll;
    return p.sampling_ratio == 2 && !p.aligned && p.channels % 4 == 0 && p.pooled_h >= 1 && p.pooled_w >= 1 &&
           p.pooled_h <= kMaxPool && p.pooled_w <= kMaxPool && num_rois > 0 && num_rois < (1ll << 31) && ob % 16 == 0 &&
           2 * ob <= 112 * 1024;
}

// bytes of workspace the TMA route needs for its per-RoI records (0: outside the envelope)
size_t mb_roi_align_tma_workspace_bytes(const mb_roi_align_params& p, int64_t num_rois) {
    return tma_shape_ok(p, num_rois) ? (size_t)num_rois * sizeof(TmaGeom) + 256 : 0;
}

// Launches the pre-pass + the TMA kernel if the configuration is inside the envelope and the workspace holds the
// records; returns 1 if launched, 0 if the caller should take the gather kernel, or an error code.
int mb_launch_roi_align_tma(const mb_roi_align_params& p, const float* rois, int64_t num_rois, float* out,
                            int32_t* levels_out, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
    int sms = 0, smem_optin = 0;
    if (!p.channels_last || !tma_shape_ok(p, num_rois) || !tma_device_info(sms, smem_optin)) return 0;
    if (workspace == nullptr || workspace_bytes < mb_roi_align_tma_workspace_bytes(p, num_rois)) return 0;
    if ((reinterpret_cast<uintptr_t>(out) & 15) != 0) return 0;
    for (int l = 0; l < p.num_levels; ++l) {
        if ((reinterpret_cast<uintptr_t>(p.features[l]) & 15) != 0) return 0;
        if ((unsigned long long)p.height[l] * p.width[l] * p.channels * 4ull >= (1ull << 31)) return 0;
    }
    const unsigned ob = (unsigned)p.channels * p.pooled_h * p.pooled_w * 4u;
    const TmaSmem fixed = tma_smem_layout(0, ob);
    if ((long long)smem_optin - (long long)fixed.total <= 0) return 0;
    const unsigned ring = ((unsigned)smem_optin - fixed.total) / 128u * 128u;
    const unsigned row_cap = ring / 5u / 16u * 16u;        // 4 rows of one pooled row + the wrap gap always fit
    if (row_cap < 8u * (unsigned)p.channels * 4u) return 0;   // ring too small to be useful: gather kernel
    const TmaSmem L = tma_smem_layout(ring, ob);
    TmaGeom* recs = reinterpret_cast<TmaGeom*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
    const int grid = (int)(num_rois < sms ? num_rois : sms);
    const float2 ones = make_float2(1.0f, 1.0f);
    const int e = p.exact ? 1 : 0;
    static const int dbg = getenv("MB_TMA_PROBE") ? atoi(getenv("MB_TMA_PROBE")) : 0;   // development probes, see tools/roi_tma_probe.py
    if (e) MB_DYN_SMEM(k_roi_align_tma<true>, smem_optin);
    else MB_DYN_SMEM(k_roi_align_tma<false>, smem_optin);
    k_roi_geom<<<(unsigned)((num_rois + 7) / 8), 256, 0, stream>>>(p, rois, (int)num_rois, row_cap, recs, levels_out, dbg);
    MB_LAUNCH_CHECK();
    if (e)
        k_roi_align_tma<true><<<grid, kTmaThreads, L.total, stream>>>(p, recs, (int)num_rois, out, ring, ones, dbg);
    else
        k_roi_align_tma<false><<<grid, kTmaThreads, L.total, stream>>>(p, recs, (int)num_rois, out, ring, ones, dbg);
    MB_LAUNCH_CHECK();
    ++g_tma_launches;
    return 1;
}
