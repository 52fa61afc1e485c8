// roi_align.cu — MultiScaleRoIAlign / roi_align forward for fp32 features (NCHW or channels-last).
//
// Replaces tv:ops/poolers.py:147-227 (per-level where/gather/roi_align/scatter loop) and
// torchvision::roi_align (tv:ops/roi_align.py:203-260 -> tv-csrc:ops/cuda/roi_align_kernel.cu:470)
// with ONE launch over all levels. Arithmetic follows the CPU kernel
// (tv-csrc:ops/cpu/roi_align_kernel.cpp:393, SURVEY.md Appendix B.2): sample coordinates are
// computed with one fp32 rounding per operation, and in `exact` mode the bilinear sum keeps the
// reference's operation order so results are bit-identical; otherwise FMAs are used (<=1e-5 rel).
//
// Kernels, fastest route first (dispatch at the bottom of the file):
//   k_roi_align_nhwc4d  channels-last maps (or NCHW maps transposed once per call by k_nchw_to_nhwc
//                       into the caller's workspace), sampling_ratio 2, <= 64 bins, C % 4 == 0:
//                       16-byte gathers straight from global memory, taps de-duplicated per bin.
//   k_roi_align_nhwc    channels-last maps k_roi_align_nhwc4d cannot take (C % 4 != 0, maps not 16-byte
//                       aligned, or one image's map of 4 GiB or more): scalar gathers.
//   k_roi_align_sr2     NCHW maps without a workspace: CTA = RoI, the footprint of 32 channels is
//                       staged NCHW -> shared memory [channel][row][col] with a plane pitch == 1
//                       (mod 32) words so that "lane = channel" tap reads hit 32 banks.
//   k_roi_align_staged  any other fixed sampling_ratio; k_roi_align_direct: adaptive sampling
//                       (sampling_ratio <= 0) or very large bins, one thread per output element.
// All of them collect a RoI's outputs in shared memory and write them as one contiguous block
// (the [K,C,PH,PW] layout makes a channel chunk of one RoI contiguous).
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "roi_common.cuh"

namespace mb {

constexpr int kRoiThreads = 256;
constexpr int kRoiWarps = kRoiThreads / 32;
constexpr int kChunk = 32;       // channels per CTA
constexpr int kMaxSamples = 64;  // sampling_ratio * pooled size per axis, staged kernel

template <bool EXACT>
__device__ __forceinline__ float bilinear4(float hy, float ly, float hx, float lx, float v1, float v2,
                                           float v3, float v4, float acc) {
    if (EXACT) {
        const float w1 = __fmul_rn(hy, hx), w2 = __fmul_rn(hy, lx), w3 = __fmul_rn(ly, hx), w4 = __fmul_rn(ly, lx);
        float t = __fmul_rn(w1, v1);
        t = __fadd_rn(t, __fmul_rn(w2, v2));
        t = __fadd_rn(t, __fmul_rn(w3, v3));
        t = __fadd_rn(t, __fmul_rn(w4, v4));
        return __fadd_rn(acc, t);
    } else {
        const float top = fmaf(lx, v2, hx * v1);
        const float bot = fmaf(lx, v4, hx * v3);
        return fmaf(hy, top, fmaf(ly, bot, acc));
    }
}

template <bool EXACT, bool SR2>
__global__ void __launch_bounds__(kRoiThreads, 4) k_roi_align_staged(const mb_roi_align_params p,
                                                                 const float* __restrict__ rois, int num_rois,
                                                                 float* __restrict__ out, int* __restrict__ levels_out,
                                                                 int stage_floats) {
    extern __shared__ __align__(16) float smem[];
    __shared__ Tap ytab[kMaxSamples], xtab[kMaxSamples];
    // sampling_ratio == 2: per output row / column, both samples packed for 128-bit broadcast loads
    __shared__ __align__(16) int4 yoff2[kMaxSamples / 2], xoff2[kMaxSamples / 2];
    __shared__ __align__(16) float4 ywt2[kMaxSamples / 2], xwt2[kMaxSamples / 2];

    const int chunks = (p.channels + kChunk - 1) / kChunk;
    const int k = blockIdx.x / chunks;
    const int c0 = (blockIdx.x % chunks) * kChunk;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int PH = p.pooled_h, PW = p.pooled_w, nbins = PH * PW;
    const int opitch = (nbins & 1) ? nbins : nbins + 1;  // odd pitch: lane=channel stores hit 32 banks
    float* out_s = smem;                       // [kChunk][opitch]
    float* patch = smem + kChunk * opitch;     // [kChunk][pitch]
    const int patch_floats = stage_floats - kChunk * opitch;

    float r[5];
    load_roi(rois, k, p, r);
    RoiGeom g;
    roi_geometry(r, p, g);  // every thread, in registers: cheaper than a broadcast through shared memory
    if (levels_out != nullptr && c0 == 0 && tid == 0) levels_out[k] = g.level;
    const int ny = PH * g.grid_h, nx = PW * g.grid_w;
    if (tid < ny) ytab[tid] = make_tap(g.start_h, g.bin_h, tid / g.grid_h, tid % g.grid_h, g.grid_h, g.H);
    if (tid >= 64 && tid < 64 + nx) {
        const int i = tid - 64;
        xtab[i] = make_tap(g.start_w, g.bin_w, i / g.grid_w, i % g.grid_w, g.grid_w, g.W);
    }
    __syncthreads();

    const bool bad_batch = g.batch < 0 || g.batch >= p.num_images;
    // Footprint columns. Sample coordinates are monotone, so invalid samples sit at the two ends:
    // the footprint runs from the first valid sample's low pixel to the last valid one's high pixel.
    int x0 = 0x7fffffff, x1 = -1;
    {
        int i = 0;
        while (i < nx && !xtab[i].valid) ++i;
        int j = nx - 1;
        while (j >= 0 && !xtab[j].valid) --j;
        if (i <= j) { x0 = xtab[i].lo; x1 = xtab[j].hi; }
    }
    const int cols = x1 - x0 + 1;
    const int c = c0 + lane;
    const bool c_ok = c < p.channels;
    const float* feat = p.features[g.level];
    const size_t plane = (size_t)g.H * g.W;
    const float* base = feat + ((size_t)(bad_batch ? 0 : g.batch) * p.channels + c0) * plane;

    int ph0 = 0;
    while (ph0 < PH) {
        // ---- choose the largest group of output rows [ph0, ph1) whose footprint fits ----
        int gy0 = 0x7fffffff, gy1 = -1, ph1 = ph0;
        bool direct = false;
        if (x1 < 0 || bad_batch) {
            ph1 = PH;  // nothing to sample: zeros
        } else {
            if (ph0 == 0) {  // common case: the whole footprint fits the staging buffer
                int i = 0;
                while (i < ny && !ytab[i].valid) ++i;
                int j = ny - 1;
                while (j >= 0 && !ytab[j].valid) --j;
                const int rows_a = (i <= j) ? ytab[j].hi - ytab[i].lo + 1 : 0;
                const int pix_a = rows_a * cols;
                if ((pix_a + ((33 - (pix_a & 31)) & 31)) * kChunk <= patch_floats) {
                    ph1 = PH;
                    if (rows_a > 0) { gy0 = ytab[i].lo; gy1 = ytab[j].hi; }
                }
            }
            while (ph1 < PH) {
                int ny0 = gy0, ny1 = gy1;
                for (int i = ph1 * g.grid_h; i < (ph1 + 1) * g.grid_h; ++i)
                    if (ytab[i].valid) { ny0 = min(ny0, ytab[i].lo); ny1 = max(ny1, ytab[i].hi); }
                const int rows_n = ny1 >= 0 ? ny1 - ny0 + 1 : 0;
                const int pix = rows_n * cols;
                const int pitch_n = pix + ((33 - (pix & 31)) & 31);
                if (pitch_n * kChunk > patch_floats) break;
                gy0 = ny0; gy1 = ny1; ++ph1;
            }
            if (ph1 == ph0) { direct = true; ph1 = ph0 + 1; }
        }
        const int rows = gy1 >= 0 ? gy1 - gy0 + 1 : 0;
        const int pix = rows * cols;
        const int pitch = pix + ((33 - (pix & 31)) & 31);

        // ---- stage the footprint. Lanes run along x (coalesced); narrow footprints pack several
        //      (channel,row) slots into one warp instruction; 8 independent loads are issued
        //      before the first store so that one warp keeps 8 rows in flight. ----
        if (!direct && rows > 0) {
            const int nch = min(kChunk, p.channels - c0);
            const int nslots = nch * rows;
            if (cols <= 32) {
                int cp2 = 1;
                while (cp2 < cols) cp2 <<= 1;
                const int rpi = 32 / cp2;                 // row slots per warp instruction
                const int sub = lane / cp2, x = lane - sub * cp2;
                const int step = kRoiWarps * rpi;         // slots per CTA iteration
                const int dcc = step / rows, drr = step - dcc * rows;
                int q = warp * rpi + sub;
                int cc = q / rows, rr = q - cc * rows;
                const float* src0 = base + (size_t)gy0 * g.W + x0 + x;
                const bool xa = x < cols;
                constexpr int U = 8;
                for (int it = 0; it < nslots; it += step * U) {
                    float v[U];
                    int so[U];
                    bool ok[U];
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        ok[u] = xa && (q < nslots);
                        so[u] = cc * pitch + rr * cols + x;
                        if (ok[u]) v[u] = __ldg(src0 + (size_t)cc * plane + rr * g.W);
                        q += step; cc += dcc; rr += drr;
                        if (rr >= rows) { rr -= rows; ++cc; }
                    }
#pragma unroll
                    for (int u = 0; u < U; ++u)
                        if (ok[u]) patch[so[u]] = v[u];
                }
            } else {
                for (int cr = warp; cr < nslots; cr += kRoiWarps) {
                    const int cc = cr / rows, rr = cr - cc * rows;
                    const float* src = base + (size_t)cc * plane + (size_t)(gy0 + rr) * g.W + x0;
                    float* dst = patch + cc * pitch + rr * cols;
                    for (int x = lane; x < cols; x += 32) dst[x] = __ldg(src + x);
                }
            }
        }
        if (SR2 && !direct && rows > 0) {   // offsets of samples outside the map are never read (skipped below)
            if (tid < ph1 - ph0) {
                const Tap a = ytab[(ph0 + tid) * 2], b = ytab[(ph0 + tid) * 2 + 1];
                yoff2[tid] = make_int4((a.lo - gy0) * cols - x0, (a.hi - gy0) * cols - x0,
                                       (b.lo - gy0) * cols - x0, (b.hi - gy0) * cols - x0);
                ywt2[tid] = make_float4(a.h, a.l, b.h, b.l);
            }
            if (tid >= 32 && tid < 32 + PW) {
                const int i = tid - 32;
                const Tap a = xtab[i * 2], b = xtab[i * 2 + 1];
                xoff2[i] = make_int4(a.lo, a.hi, b.lo, b.hi);
                xwt2[i] = make_float4(a.h, a.l, b.h, b.l);
            }
        }
        __syncthreads();

        // ---- bins of this group: warp per bin, lane per channel ----
        const int gbins = (ph1 - ph0) * PW;
        const float* sp = patch + lane * pitch;
        const float* gp = base + (size_t)lane * plane;
        for (int b = warp; b < gbins; b += kRoiWarps) {
            const int ph = ph0 + b / PW, pw = b - (b / PW) * PW;
            float acc = 0.0f;
            if (SR2 && !direct) {
                if (c_ok && rows > 0) {
                    const int4 yo = yoff2[ph - ph0], xo = xoff2[pw];
                    const float4 yw = ywt2[ph - ph0], xw = xwt2[pw];
                    // samples outside the map are skipped like the reference does, not weighted by 0 (an Inf / NaN
                    // feature elsewhere cannot leak in); the branches are warp-uniform: all lanes share the bin
                    const bool ya = ytab[2 * ph].valid, yb = ytab[2 * ph + 1].valid;
                    const bool xa = xtab[2 * pw].valid, xb = xtab[2 * pw + 1].valid;
                    // sample (iy=0, ix=0), (0,1), (1,0), (1,1) in the reference's loop order
                    if (ya && xa) acc = bilinear4<EXACT>(yw.x, yw.y, xw.x, xw.y, sp[yo.x + xo.x], sp[yo.x + xo.y], sp[yo.y + xo.x], sp[yo.y + xo.y], acc);
                    if (ya && xb) acc = bilinear4<EXACT>(yw.x, yw.y, xw.z, xw.w, sp[yo.x + xo.z], sp[yo.x + xo.w], sp[yo.y + xo.z], sp[yo.y + xo.w], acc);
                    if (yb && xa) acc = bilinear4<EXACT>(yw.z, yw.w, xw.x, xw.y, sp[yo.z + xo.x], sp[yo.z + xo.y], sp[yo.w + xo.x], sp[yo.w + xo.y], acc);
                    if (yb && xb) acc = bilinear4<EXACT>(yw.z, yw.w, xw.z, xw.w, sp[yo.z + xo.z], sp[yo.z + xo.w], sp[yo.w + xo.z], sp[yo.w + xo.w], acc);
                }
            } else if (c_ok && (direct || rows > 0)) {
                for (int iy = 0; iy < g.grid_h; ++iy) {
                    const Tap Y = ytab[ph * g.grid_h + iy];
                    if (!Y.valid) continue;
                    for (int ix = 0; ix < g.grid_w; ++ix) {
                        const Tap X = xtab[pw * g.grid_w + ix];
                        if (!X.valid) continue;
                        float v1, v2, v3, v4;
                        if (!direct) {
                            const int rlo = (Y.lo - gy0) * cols - x0, rhi = (Y.hi - gy0) * cols - x0;
                            v1 = sp[rlo + X.lo]; v2 = sp[rlo + X.hi]; v3 = sp[rhi + X.lo]; v4 = sp[rhi + X.hi];
                        } else {
                            v1 = __ldg(gp + Y.lo * g.W + X.lo); v2 = __ldg(gp + Y.lo * g.W + X.hi);
                            v3 = __ldg(gp + Y.hi * g.W + X.lo); v4 = __ldg(gp + Y.hi * g.W + X.hi);
                        }
                        acc = bilinear4<EXACT>(Y.h, Y.l, X.h, X.l, v1, v2, v3, v4, acc);
                    }
                }
            }
            out_s[lane * opitch + ph * PW + pw] = __fdiv_rn(acc, g.count);
        }
        __syncthreads();
        ph0 = ph1;
    }

    // ---- one contiguous block of min(32, C-c0)*nbins floats per (RoI, chunk) ----
    const int nch = min(kChunk, p.channels - c0);
    const int total = nch * nbins;
    float* dst = out + ((size_t)k * p.channels + c0) * nbins;
    if (opitch == nbins && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) && (total & 3) == 0) {
        const float4* s4 = reinterpret_cast<const float4*>(out_s);
        float4* d4 = reinterpret_cast<float4*>(dst);
        for (int i = tid; i < total / 4; i += kRoiThreads) d4[i] = s4[i];
    } else {
        for (int ch = warp; ch < nch; ch += kRoiWarps)
            for (int b = lane; b < nbins; b += 32) dst[ch * nbins + b] = out_s[ch * opitch + b];
    }
}

// ------------------------------------------------------------------------------------------
// sampling_ratio == 2 (the detection models): CTA = one RoI, all channels.
// Geometry, tap tables, footprint groups and a per-bin table of 16 (offset, weight) pairs are
// built ONCE per RoI; the CTA then walks the channel chunks: stage 32 planes of the footprint
// (thread = footprint pixel, loop over channels: one pointer increment per element, 8 loads in
// flight), 49 bins x 32 channels from shared memory (8 broadcast LDS.128 of the bin's table +
// 16 conflict-free LDS, products and sums in the reference's order), coalesced float4 write-out.
// ------------------------------------------------------------------------------------------
constexpr int kMaxGroups = 32;

// A sample outside the map has negative offsets in the table (kSkipTap) and is skipped like the reference does, not
// weighted by 0: an Inf / NaN feature elsewhere cannot leak in. Bins with all samples inside the map (nearly all) take
// the SKIP = false body, whose loads are not split by branches; the choice is warp-uniform (lanes are channels).
constexpr int kSkipTap = -1;

__device__ __forceinline__ bool bin_all_in(const int4* __restrict__ toff) {
    return (toff[0].x | toff[1].x | toff[2].x | toff[3].x) >= 0;
}

template <bool EXACT, bool SKIP>
__device__ __forceinline__ float bin_value(const float* sp, const int4* __restrict__ toff, const float4* __restrict__ tw) {
    float acc = 0.0f;
#pragma unroll
    for (int smp = 0; smp < 4; ++smp) {
        const int4 o = toff[smp];
        if (SKIP && o.x < 0) continue;
        const float4 wv = tw[smp];
        const float v1 = sp[o.x], v2 = sp[o.y], v3 = sp[o.z], v4 = sp[o.w];
        if (EXACT) {   // ((w1*v1 + w2*v2) + w3*v3) + w4*v4, then acc + that: the reference's order
            float t = __fmul_rn(wv.x, v1);
            t = __fadd_rn(t, __fmul_rn(wv.y, v2));
            t = __fadd_rn(t, __fmul_rn(wv.z, v3));
            t = __fadd_rn(t, __fmul_rn(wv.w, v4));
            acc = __fadd_rn(acc, t);
        } else {
            acc = fmaf(wv.x, v1, fmaf(wv.y, v2, fmaf(wv.z, v3, fmaf(wv.w, v4, acc))));
        }
    }
    return __fmul_rn(acc, 0.25f);   // acc / 4: exact scaling
}

template <bool EXACT, bool SKIP>
__device__ __forceinline__ float bin_value_smem(unsigned sbase, const int4* __restrict__ toff, const float4* __restrict__ tw) {
    // toff holds BYTE offsets; sbase is the lane's 32-bit shared address: one add per tap
    float acc = 0.0f;
#pragma unroll
    for (int smp = 0; smp < 4; ++smp) {
        const int4 o = toff[smp];
        if (SKIP && o.x < 0) continue;
        const float4 wv = tw[smp];
        float v1, v2, v3, v4;
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v1) : "r"(sbase + o.x));
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v2) : "r"(sbase + o.y));
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v3) : "r"(sbase + o.z));
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v4) : "r"(sbase + o.w));
        if (EXACT) {
            float t = __fmul_rn(wv.x, v1);
            t = __fadd_rn(t, __fmul_rn(wv.y, v2));
            t = __fadd_rn(t, __fmul_rn(wv.z, v3));
            t = __fadd_rn(t, __fmul_rn(wv.w, v4));
            acc = __fadd_rn(acc, t);
        } else {
            acc = fmaf(wv.x, v1, fmaf(wv.y, v2, fmaf(wv.z, v3, fmaf(wv.w, v4, acc))));
        }
    }
    return __fmul_rn(acc, 0.25f);
}

// scalar staging: thread = footprint pixel, channels walked with U loads in flight
template <int U>
__device__ __forceinline__ void stage_scalar(const float* src, float* dp, size_t sstep, int dstep, int cc, int nch, int NG) {
    for (; cc + (U - 1) * NG < nch; cc += U * NG) {
        float v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) v[u] = __ldg(src + u * sstep);
#pragma unroll
        for (int u = 0; u < U; ++u) dp[u * dstep] = v[u];
        src += U * sstep; dp += U * dstep;
    }
    for (; cc < nch; cc += NG) { *dp = __ldg(src); src += sstep; dp += dstep; }
}

template <bool EXACT>
__global__ void __launch_bounds__(kRoiThreads, 4) k_roi_align_sr2(const mb_roi_align_params p,
                                                                const float* __restrict__ rois,
                                                                float* __restrict__ out, int* __restrict__ levels_out,
                                                                int patch_floats, int variant) {
    extern __shared__ __align__(16) float smem[];
    __shared__ Tap ytab[32], xtab[32];
    __shared__ int grp_ph0[kMaxGroups + 1], grp_y0[kMaxGroups], grp_rows[kMaxGroups], grp_direct[kMaxGroups];
    __shared__ int s_ngroups;

    const int k = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int PH = p.pooled_h, PW = p.pooled_w, nbins = PH * PW;
    const int opitch = (nbins & 1) ? nbins : nbins + 1;
    float* out_s = smem;                                   // [kChunk][opitch]
    float* patch = out_s + kChunk * opitch;                // [kChunk][pitch]
    int4* tab_off = reinterpret_cast<int4*>(patch + patch_floats);       // [nbins][4] (16-byte aligned by construction)
    float4* tab_w = reinterpret_cast<float4*>(tab_off + nbins * 4);      // [nbins][4]

    float r[5];
    load_roi(rois, k, p, r);
    RoiGeom g;
    roi_geometry(r, p, g);
    if (levels_out != nullptr && tid == 0) levels_out[k] = g.level;
    const int ny = PH * 2, nx = PW * 2;
    if (tid < ny) ytab[tid] = make_tap(g.start_h, g.bin_h, tid >> 1, tid & 1, 2, g.H);
    if (tid >= 64 && tid < 64 + nx) xtab[tid - 64] = make_tap(g.start_w, g.bin_w, (tid - 64) >> 1, (tid - 64) & 1, 2, g.W);
    __syncthreads();

    const bool bad_batch = g.batch < 0 || g.batch >= p.num_images;
    const size_t plane = (size_t)g.H * g.W;
    const float* feat = p.features[g.level] + (size_t)(bad_batch ? 0 : g.batch) * p.channels * plane;
    // 16-byte vector staging needs every footprint row to start on a float4 boundary
    const bool vec4 = !(variant & 1) && ((g.W & 3) == 0) && ((plane & 3) == 0) && ((reinterpret_cast<uintptr_t>(feat) & 15) == 0);
    int x0 = 0, x1 = -1;
    {
        int i = 0;
        while (i < nx && !xtab[i].valid) ++i;
        int j = nx - 1;
        while (j >= 0 && !xtab[j].valid) --j;
        if (i <= j) { x0 = xtab[i].lo; x1 = xtab[j].hi; }
    }
    const bool empty = bad_batch || x1 < 0;
    if (vec4 && !empty) { x0 &= ~3; x1 |= 3; }   // W % 4 == 0, so x1 | 3 <= W - 1
    const int cols = x1 - x0 + 1;

    // ---- footprint groups: maximal runs of output rows whose rows x cols fit the staging buffer ----
    if (tid == 0) {
        int ng = 0, ph0 = 0;
        while (ph0 < PH && !empty) {
            int gy0 = 0x7fffffff, gy1 = -1, ph1 = ph0;
            while (ph1 < PH) {
                int ny0 = gy0, ny1 = gy1;
                for (int i = ph1 * 2; i < ph1 * 2 + 2; ++i)
                    if (ytab[i].valid) { ny0 = min(ny0, ytab[i].lo); ny1 = max(ny1, ytab[i].hi); }
                const int pix = (ny1 >= 0 ? ny1 - ny0 + 1 : 0) * cols;
                if ((pix + ((33 - (pix & 31)) & 31)) * kChunk > patch_floats) break;
                gy0 = ny0; gy1 = ny1; ++ph1;
            }
            const bool direct = (ph1 == ph0);
            if (direct) {  // one output row alone does not fit: gather it straight from global memory
                ph1 = ph0 + 1;
                for (int i = ph0 * 2; i < ph0 * 2 + 2; ++i)
                    if (ytab[i].valid) { gy0 = min(gy0, ytab[i].lo); gy1 = max(gy1, ytab[i].hi); }
            }
            grp_ph0[ng] = ph0; grp_y0[ng] = gy1 >= 0 ? gy0 : 0; grp_rows[ng] = gy1 >= 0 ? gy1 - gy0 + 1 : 0;
            grp_direct[ng] = direct;
            ++ng; ph0 = ph1;
        }
        grp_ph0[ng] = PH;
        s_ngroups = ng;
    }
    __syncthreads();
    const int ngroups = s_ngroups;

    // ---- per-bin tables: 4 samples x 4 corners, offsets relative to the bin's group footprint ----
    for (int e = tid; e < nbins * 4 && !empty; e += kRoiThreads) {
        const int b = e >> 2, smp = e & 3;
        const int ph = b / PW, pw = b - ph * PW;
        int gi = 0;
        while (gi + 1 < ngroups && ph >= grp_ph0[gi + 1]) ++gi;
        const Tap Y = ytab[ph * 2 + (smp >> 1)], X = xtab[pw * 2 + (smp & 1)];
        const bool ok = Y.valid && X.valid;
        const bool direct = grp_direct[gi] != 0;
        const int rs = direct ? g.W : cols;                 // row stride of the addressed buffer
        const int oy = direct ? 0 : grp_y0[gi], ox = direct ? 0 : x0;
        const int ylo = (Y.lo - oy) * rs, yhi = (Y.hi - oy) * rs;
        const int xlo = X.lo - ox, xhi = X.hi - ox;
        tab_off[e] = ok ? make_int4(4 * (ylo + xlo), 4 * (ylo + xhi), 4 * (yhi + xlo), 4 * (yhi + xhi))   // byte offsets
                        : make_int4(kSkipTap, kSkipTap, kSkipTap, kSkipTap);
        tab_w[e] = ok ? make_float4(__fmul_rn(Y.h, X.h), __fmul_rn(Y.h, X.l), __fmul_rn(Y.l, X.h), __fmul_rn(Y.l, X.l))
                      : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncthreads();

    const int nchunks = (p.channels + kChunk - 1) / kChunk;
    float* dst_roi = out + (size_t)k * p.channels * nbins;

    for (int chunk = 0; chunk < nchunks; ++chunk) {
        const int c0 = chunk * kChunk;
        const int nch = min(kChunk, p.channels - c0);
        const float* base = feat + (size_t)c0 * plane;
        if (empty) {
            for (int i = tid; i < kChunk * opitch; i += kRoiThreads) out_s[i] = 0.0f;
            __syncthreads();
        }
        for (int gi = 0; gi < ngroups; ++gi) {
            const int rows = grp_rows[gi], gy0 = grp_y0[gi];
            const bool direct = grp_direct[gi] != 0;
            const int P = rows * cols;
            const int pitch = P + ((33 - (P & 31)) & 31);
            if (!direct && P > 0) {
                if (vec4) {
                    // ---- stage, 16-byte loads: lane = (channel c%4, float4 slot). A warp instruction
                    //      reads 4 channels x 128 contiguous bytes; the four scalar stores of a float4
                    //      land on 32 distinct banks because the plane pitch is 1 (mod 32). ----
                    const int c4 = cols >> 2, P4 = rows * c4;
                    const int csub = tid & 3;
                    for (int pos4 = tid >> 2; pos4 < P4; pos4 += kRoiThreads / 4) {
                        const int rr = pos4 / c4, x4 = pos4 - rr * c4;
                        const float4* src = reinterpret_cast<const float4*>(
                            base + (size_t)csub * plane + (size_t)(gy0 + rr) * g.W + x0 + 4 * x4);
                        float* dp = patch + csub * pitch + 4 * pos4;
#pragma unroll
                        for (int half = 0; half < 2; ++half) {      // 2 x 4 loads of 16 bytes in flight
                            float4 v[4];
#pragma unroll
                            for (int u = 0; u < 4; ++u)
                                if ((half * 4 + u) * 4 + csub < nch) v[u] = __ldg(src + (size_t)(half * 4 + u) * plane);
#pragma unroll
                            for (int u = 0; u < 4; ++u)
                                if ((half * 4 + u) * 4 + csub < nch) {
                                    float* d = dp + (half * 4 + u) * 4 * pitch;
                                    d[0] = v[u].x; d[1] = v[u].y; d[2] = v[u].z; d[3] = v[u].w;
                                }
                        }
                    }
                } else {
                    // ---- stage, scalar: thread = footprint pixel (x fastest), loop over channels ----
                    const int NG = P <= kRoiThreads ? kRoiThreads / P : 1;
                    for (int pos0 = 0; pos0 < P; pos0 += kRoiThreads) {
                        int pos = pos0 + tid, grp = 0;
                        if (NG > 1) { grp = tid / P; pos = tid - grp * P; }
                        if (pos < P && grp < NG) {
                            const int rr = pos / cols, x = pos - rr * cols;
                            const float* src = base + (size_t)grp * plane + (size_t)(gy0 + rr) * g.W + x0 + x;
                            float* dp = patch + grp * pitch + pos;
                            const size_t sstep = (size_t)NG * plane;
                            const int dstep = NG * pitch;
                            if (variant & 2) stage_scalar<16>(src, dp, sstep, dstep, grp, nch, NG);
                            else stage_scalar<8>(src, dp, sstep, dstep, grp, nch, NG);
                        }
                    }
                }
            }
            __syncthreads();
            // ---- bins of this group: warp per bin, lane per channel ----
            const int b0 = grp_ph0[gi] * PW, b1 = grp_ph0[gi + 1] * PW;
            if (direct) {
                const float* gp = base + (size_t)lane * plane;            // global gathers (rare)
                if (lane < nch)
                    for (int b = b0 + warp; b < b1; b += kRoiWarps) {
                        int4 o4[4];
                        for (int q = 0; q < 4; ++q) { o4[q] = tab_off[b * 4 + q]; o4[q].x >>= 2; o4[q].y >>= 2; o4[q].z >>= 2; o4[q].w >>= 2; }
                        out_s[lane * opitch + b] = bin_all_in(o4) ? bin_value<EXACT, false>(gp, o4, tab_w + b * 4)
                                                                  : bin_value<EXACT, true>(gp, o4, tab_w + b * 4);
                    }
            } else if (P == 0) {              // no valid sample row in this group: zeros (nothing was staged)
                for (int b = b0 + warp; b < b1; b += kRoiWarps) out_s[lane * opitch + b] = 0.0f;
            } else if (lane < nch) {
                const unsigned sbase = smem_u32(patch + lane * pitch);    // 32-bit shared address: one add per tap
                for (int b = b0 + warp; b < b1; b += kRoiWarps)
                    out_s[lane * opitch + b] = bin_all_in(tab_off + b * 4)
                                                   ? bin_value_smem<EXACT, false>(sbase, tab_off + b * 4, tab_w + b * 4)
                                                   : bin_value_smem<EXACT, true>(sbase, tab_off + b * 4, tab_w + b * 4);
            }
            __syncthreads();
        }
        // ---- write out: contiguous nch*nbins floats of out[k, c0:c0+nch] ----
        float* dst = dst_roi + (size_t)c0 * nbins;
        const int total = nch * nbins;
        if (opitch == nbins && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) && (total & 3) == 0) {
            const float4* s4 = reinterpret_cast<const float4*>(out_s);
            float4* d4 = reinterpret_cast<float4*>(dst);
            for (int i = tid; i < total / 4; i += kRoiThreads) d4[i] = s4[i];
        } else {
            for (int ch = warp; ch < nch; ch += kRoiWarps)
                for (int b = lane; b < nbins; b += 32) dst[ch * nbins + b] = out_s[ch * opitch + b];
        }
        // the next chunk's bins overwrite out_s only after its own staging barrier, which every
        // thread reaches after finishing this copy
    }
}

// ------------------------------------------------------------------------------------------
// Channels-last features ([N, H, W, C] in memory): no staging at all. A tap of 32 consecutive
// channels is one 128-byte line, so "lane = channel" gathers are perfectly coalesced straight from
// global memory; the footprint of one 32-channel chunk (~330 pixels x 128 B) lives in L1 while the
// CTA's 8 warps work through the chunk's 49 bins (each pixel is touched ~2.4 times). There are no
// load/compute phases and only one barrier per chunk (output hand-over), so warps overlap their
// own global-load latency with 16 independent loads per bin.
// ------------------------------------------------------------------------------------------
// one bin of k_roi_align_nhwc: toff holds BYTE offsets of the taps' pixels from the lane's channel in the image
template <bool EXACT, bool SKIP>
__device__ __forceinline__ float bin_value_gmem(const char* gp, const int4* __restrict__ toff, const float4* __restrict__ tw) {
    float acc = 0.0f;
#pragma unroll
    for (int smp = 0; smp < 4; ++smp) {
        const int4 o = toff[smp];
        if (SKIP && o.x < 0) continue;
        const float4 wv = tw[smp];
        const float v1 = __ldg(reinterpret_cast<const float*>(gp + o.x));
        const float v2 = __ldg(reinterpret_cast<const float*>(gp + o.y));
        const float v3 = __ldg(reinterpret_cast<const float*>(gp + o.z));
        const float v4 = __ldg(reinterpret_cast<const float*>(gp + o.w));
        if (EXACT) {
            float t = __fmul_rn(wv.x, v1);
            t = __fadd_rn(t, __fmul_rn(wv.y, v2));
            t = __fadd_rn(t, __fmul_rn(wv.z, v3));
            t = __fadd_rn(t, __fmul_rn(wv.w, v4));
            acc = __fadd_rn(acc, t);
        } else {
            acc = fmaf(wv.x, v1, fmaf(wv.y, v2, fmaf(wv.z, v3, fmaf(wv.w, v4, acc))));
        }
    }
    return __fmul_rn(acc, 0.25f);
}

template <bool EXACT>
__global__ void __launch_bounds__(kRoiThreads, 4) k_roi_align_nhwc(const mb_roi_align_params p,
                                                                 const float* __restrict__ rois,
                                                                 float* __restrict__ out, int* __restrict__ levels_out) {
    extern __shared__ __align__(16) float smem[];
    __shared__ Tap ytab[32], xtab[32];
    const int k = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int PH = p.pooled_h, PW = p.pooled_w, nbins = PH * PW;
    const int opitch = (nbins & 1) ? nbins : nbins + 1;
    const int obuf = (kChunk * opitch + 3) & ~3;
    float* out_s = smem;                                               // [2][kChunk][opitch]
    int4* tab_off = reinterpret_cast<int4*>(out_s + 2 * obuf);        // [nbins][4] byte offsets of the pixel's channel vector
    float4* tab_w = reinterpret_cast<float4*>(tab_off + nbins * 4);   // [nbins][4]

    float r[5];
    load_roi(rois, k, p, r);
    RoiGeom g;
    roi_geometry(r, p, g);
    if (levels_out != nullptr && tid == 0) levels_out[k] = g.level;
    const int ny = PH * 2, nx = PW * 2;
    if (tid < ny) ytab[tid] = make_tap(g.start_h, g.bin_h, tid >> 1, tid & 1, 2, g.H);
    if (tid >= 64 && tid < 64 + nx) xtab[tid - 64] = make_tap(g.start_w, g.bin_w, (tid - 64) >> 1, (tid - 64) & 1, 2, g.W);
    __syncthreads();
    const bool bad_batch = g.batch < 0 || g.batch >= p.num_images;
    const int C = p.channels;
    float* dst_roi = out + (size_t)k * C * nbins;
    if (bad_batch) {
        for (long long i = tid; i < (long long)C * nbins; i += kRoiThreads) dst_roi[i] = 0.0f;
        return;
    }
    for (int e = tid; e < nbins * 4; e += kRoiThreads) {
        const int b = e >> 2, smp = e & 3;
        const int ph = b / PW, pw = b - ph * PW;
        const Tap Y = ytab[ph * 2 + (smp >> 1)], X = xtab[pw * 2 + (smp & 1)];
        const bool ok = Y.valid && X.valid;
        const int cb = C * 4;   // bytes per pixel
        const int ylo = Y.lo * g.W, yhi = Y.hi * g.W;
        tab_off[e] = ok ? make_int4((ylo + X.lo) * cb, (ylo + X.hi) * cb, (yhi + X.lo) * cb, (yhi + X.hi) * cb)
                        : make_int4(kSkipTap, kSkipTap, kSkipTap, kSkipTap);
        tab_w[e] = ok ? make_float4(__fmul_rn(Y.h, X.h), __fmul_rn(Y.h, X.l), __fmul_rn(Y.l, X.h), __fmul_rn(Y.l, X.l))
                      : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncthreads();
    const char* img = reinterpret_cast<const char*>(p.features[g.level]) + (size_t)g.batch * g.H * g.W * C * 4;
    const int nchunks = (C + kChunk - 1) / kChunk;
    for (int chunk = 0; chunk < nchunks; ++chunk) {
        const int c0 = chunk * kChunk;
        const int nch = min(kChunk, C - c0);
        float* ob = out_s + (chunk & 1) * obuf;
        if (lane < nch) {
            const char* gp = img + (size_t)(c0 + lane) * 4;
            for (int b = warp; b < nbins; b += kRoiWarps) {
                const int4* to = tab_off + b * 4;
                ob[lane * opitch + b] = bin_all_in(to) ? bin_value_gmem<EXACT, false>(gp, to, tab_w + b * 4)
                                                       : bin_value_gmem<EXACT, true>(gp, to, tab_w + b * 4);
            }
        }
        __syncthreads();   // the chunk's bins are complete; the other buffer is free for the next chunk
        float* dst = dst_roi + (size_t)c0 * nbins;
        const int total = nch * nbins;
        if (opitch == nbins && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) && (total & 3) == 0) {
            const float4* s4 = reinterpret_cast<const float4*>(ob);
            float4* d4 = reinterpret_cast<float4*>(dst);
            for (int i = tid; i < total / 4; i += kRoiThreads) d4[i] = s4[i];
        } else {
            for (int ch = warp; ch < nch; ch += kRoiWarps)
                for (int b = lane; b < nbins; b += 32) dst[ch * nbins + b] = ob[ch * opitch + b];
        }
        // buffer (chunk & 1) is rewritten by chunk + 2, after the barrier of chunk + 1
    }
}

constexpr int kChunk4 = 128;   // channels per pass of the 16-byte-gather kernel (lane = 4 consecutive channels)

// ------------------------------------------------------------------------------------------
// nhwc4 with de-duplicated taps. The 16 taps of a bin are the tensor product of 4 pixel rows
// {lo0, hi0, lo1, hi1} and 4 pixel columns of its two samples per axis. At the pyramid level the
// LevelMapper assigns, a RoI is 14..28 pixels across, i.e. the half-bin sample spacing is 1..2
// pixels, so most of the time hi0 == lo1 (pattern B: 3 distinct rows); boxes smaller than the
// canonical range have both samples in the same cell (pattern A: 2 rows); only the largest have 4
// distinct rows (pattern C). The per-axis pattern is found when the RoI's tables are built; the
// bin body is instantiated for the 9 (row, column) pattern pairs and loads each distinct pixel once
// (typically 3 x 3 = 9 vector loads instead of 16). The arithmetic is untouched — the same 16
// weight x value products in the reference order, fed from shared registers — so EXACT stays
// bit-identical. The kernel is bound by L1 wavefronts (profiles/), which is what this removes.
// ------------------------------------------------------------------------------------------
template <bool EXACT, int PY, int PX>
__device__ __forceinline__ float4 bin_dedup(const char* __restrict__ gp, const uint4 ro4, const uint4 co4,
                                            const float4* __restrict__ tw, const float2 ones) {
    constexpr int NR = PY == 0 ? 2 : (PY == 1 ? 3 : 4), NC = PX == 0 ? 2 : (PX == 1 ? 3 : 4);
    const unsigned ro[4] = {ro4.x, ro4.y, ro4.z, ro4.w}, co[4] = {co4.x, co4.y, co4.z, co4.w};
    float4 G[NR][NC];
#pragma unroll
    for (int r = 0; r < NR; ++r)
#pragma unroll
        for (int c = 0; c < NC; ++c) G[r][c] = __ldg(reinterpret_cast<const float4*>(gp + (ro[r] + co[c])));
    // Packed fp32x2 arithmetic (sm_100 FMUL2 / FFMA2): channels (0,1) and (2,3) of the 16-byte vector share one
    // instruction; every lane of a packed multiply is rounded to nearest exactly like the scalar operation.
    float2 lo = make_float2(0.f, 0.f), hi = make_float2(0.f, 0.f);
#pragma unroll
    for (int smp = 0; smp < 4; ++smp) {
        const int iy = smp >> 1, ix = smp & 1;
        const int yl = iy == 0 ? 0 : (PY == 0 ? 0 : (PY == 1 ? 1 : 2)), yh = iy == 0 ? 1 : (PY == 0 ? 1 : (PY == 1 ? 2 : 3));
        const int xl = ix == 0 ? 0 : (PX == 0 ? 0 : (PX == 1 ? 1 : 2)), xh = ix == 0 ? 1 : (PX == 0 ? 1 : (PX == 1 ? 2 : 3));
        // one 16-byte table read per sample; the packed operands {w, w} are built in registers (a uniform LDS.128
        // costs two L1 wavefronts, the busiest unit of this kernel, a register move costs an idle ALU slot)
        const float4 wv = tw[smp];                                    // (w1, w2, w3, w4)
        const float2 w1 = make_float2(wv.x, wv.x), w2 = make_float2(wv.y, wv.y);
        const float2 w3 = make_float2(wv.z, wv.z), w4 = make_float2(wv.w, wv.w);
        const float4 v1 = G[yl][xl], v2 = G[yl][xh], v3 = G[yh][xl], v4 = G[yh][xh];
        if (EXACT) {
            // every product and every sum rounded once, in the reference's order; the sums are packed FFMA2 with an
            // opaque multiplier 1.0f (fma(p, 1, t) == fl(p + t)), which ptxas cannot contract with the multiplies
            float2 t = mul2_rn(w1, make_float2(v1.x, v1.y));
            t = fma2_rn(mul2_rn(w2, make_float2(v2.x, v2.y)), ones, t);
            t = fma2_rn(mul2_rn(w3, make_float2(v3.x, v3.y)), ones, t);
            t = fma2_rn(mul2_rn(w4, make_float2(v4.x, v4.y)), ones, t);
            lo = fma2_rn(t, ones, lo);
            float2 u = mul2_rn(w1, make_float2(v1.z, v1.w));
            u = fma2_rn(mul2_rn(w2, make_float2(v2.z, v2.w)), ones, u);
            u = fma2_rn(mul2_rn(w3, make_float2(v3.z, v3.w)), ones, u);
            u = fma2_rn(mul2_rn(w4, make_float2(v4.z, v4.w)), ones, u);
            hi = fma2_rn(u, ones, hi);
        } else {
            lo = __ffma2_rn(w1, make_float2(v1.x, v1.y), __ffma2_rn(w2, make_float2(v2.x, v2.y),
                 __ffma2_rn(w3, make_float2(v3.x, v3.y), __ffma2_rn(w4, make_float2(v4.x, v4.y), lo))));
            hi = __ffma2_rn(w1, make_float2(v1.z, v1.w), __ffma2_rn(w2, make_float2(v2.z, v2.w),
                 __ffma2_rn(w3, make_float2(v3.z, v3.w), __ffma2_rn(w4, make_float2(v4.z, v4.w), hi))));
        }
    }
    const float2 q = make_float2(0.25f, 0.25f);
    lo = mul2_rn(lo, q); hi = mul2_rn(hi, q);
    return make_float4(lo.x, lo.y, hi.x, hi.y);
}

// one bin, samples outside the map skipped like the reference does (no zero-weight multiply: an Inf / NaN feature
// elsewhere cannot leak in); plain per-sample loads, the reference's operation order in exact mode
template <bool EXACT>
__device__ __forceinline__ float4 bin_skip_invalid(const char* __restrict__ gp, const Tap* __restrict__ ytab, const Tap* __restrict__ xtab,
                                                   int ph, int pw, unsigned rowb, unsigned colb) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int iy = 0; iy < 2; ++iy) {
        const Tap Y = ytab[2 * ph + iy];
        if (!Y.valid) continue;
        for (int ix = 0; ix < 2; ++ix) {
            const Tap X = xtab[2 * pw + ix];
            if (!X.valid) continue;
            const float4 v1 = __ldg(reinterpret_cast<const float4*>(gp + (Y.lo * rowb + X.lo * colb)));
            const float4 v2 = __ldg(reinterpret_cast<const float4*>(gp + (Y.lo * rowb + X.hi * colb)));
            const float4 v3 = __ldg(reinterpret_cast<const float4*>(gp + (Y.hi * rowb + X.lo * colb)));
            const float4 v4 = __ldg(reinterpret_cast<const float4*>(gp + (Y.hi * rowb + X.hi * colb)));
            acc.x = bilinear4<EXACT>(Y.h, Y.l, X.h, X.l, v1.x, v2.x, v3.x, v4.x, acc.x);
            acc.y = bilinear4<EXACT>(Y.h, Y.l, X.h, X.l, v1.y, v2.y, v3.y, v4.y, acc.y);
            acc.z = bilinear4<EXACT>(Y.h, Y.l, X.h, X.l, v1.z, v2.z, v3.z, v4.z, acc.z);
            acc.w = bilinear4<EXACT>(Y.h, Y.l, X.h, X.l, v1.w, v2.w, v3.w, v4.w, acc.w);
        }
    }
    return make_float4(__fmul_rn(acc.x, 0.25f), __fmul_rn(acc.y, 0.25f), __fmul_rn(acc.z, 0.25f), __fmul_rn(acc.w, 0.25f));
}

template <bool EXACT, int OCC>     // OCC = resident CTAs per SM the register budget is set for
__global__ void __launch_bounds__(kRoiThreads, OCC) k_roi_align_nhwc4d(const mb_roi_align_params p,
                                                                   const float* __restrict__ rois,
                                                                   float* __restrict__ out, int* __restrict__ levels_out,
                                                                   int rows_per_cta, const float2 ones) {
    pdl_enter();
    extern __shared__ __align__(16) float smem[];
    __shared__ Tap ytab[32], xtab[32];
    __shared__ uint4 s_ro[16], s_co[16];             // byte offsets of the distinct rows / columns of each bin row / column
    __shared__ int s_py[16], s_px[16];
    const int k = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // blockIdx.y selects a band of pooled rows (one band = the whole RoI for the 7x7 box head; the 14x14 mask
    // head runs as two bands of 7 rows so that the staged outputs of a band still fit three CTAs per SM)
    const int PH = p.pooled_h, PW = p.pooled_w, nbins_all = PH * PW;
    const int ph0 = blockIdx.y * rows_per_cta;
    const int b0 = ph0 * PW, nbins = min(rows_per_cta, PH - ph0) * PW;     // this CTA's bins: b0 .. b0 + nbins - 1
    const int opitch = (rows_per_cta * PW) | 1;
    const int obuf = (kChunk4 * opitch + 3) & ~3;                      // floats per output buffer, a multiple of 16 bytes
    float* ob = smem;                                                  // [128][opitch]
    float4* tab_w = reinterpret_cast<float4*>(ob + obuf);              // [nbins][4 samples]: (w1, w2, w3, w4)
    int* s_bin = reinterpret_cast<int*>(tab_w + rows_per_cta * PW * 4);   // [nbins] ph | pw << 8 | pattern << 16

    float r[5];
    load_roi(rois, k, p, r);
    RoiGeom g;
    roi_geometry(r, p, g);
    if (levels_out != nullptr && tid == 0 && blockIdx.y == 0) levels_out[k] = g.level;
    const int ny = PH * 2, nx = PW * 2;
    if (tid < ny) ytab[tid] = make_tap(g.start_h, g.bin_h, tid >> 1, tid & 1, 2, g.H);
    if (tid >= 64 && tid < 64 + nx) xtab[tid - 64] = make_tap(g.start_w, g.bin_w, (tid - 64) >> 1, (tid - 64) & 1, 2, g.W);
    __syncthreads();
    const int C = p.channels;
    float* dst_roi = out + (size_t)k * C * nbins_all;
    if (g.batch < 0 || g.batch >= p.num_images) {
        if (blockIdx.y == 0)
            for (long long i = tid; i < (long long)C * nbins_all; i += kRoiThreads) dst_roi[i] = 0.0f;
        return;
    }
    if (tid < PH) {
        int idx[4];
        s_py[tid] = axis_pattern(ytab[2 * tid], ytab[2 * tid + 1], idx);
        const unsigned rb = (unsigned)g.W * (unsigned)C * 4u;
        s_ro[tid] = make_uint4(idx[0] * rb, idx[1] * rb, idx[2] * rb, idx[3] * rb);
    } else if (tid >= 32 && tid < 32 + PW) {
        const int t = tid - 32;
        int idx[4];
        s_px[t] = axis_pattern(xtab[2 * t], xtab[2 * t + 1], idx);
        const unsigned cb = (unsigned)C * 4u;
        s_co[t] = make_uint4(idx[0] * cb, idx[1] * cb, idx[2] * cb, idx[3] * cb);
    }
    for (int e = tid; e < nbins * 4; e += kRoiThreads) {
        const int b = e >> 2, smp = e & 3;
        const int ph = ph0 + b / PW, pw = b % PW;
        const Tap Y = ytab[ph * 2 + (smp >> 1)], X = xtab[pw * 2 + (smp & 1)];
        const bool ok = Y.valid && X.valid;
        const float w1 = ok ? __fmul_rn(Y.h, X.h) : 0.f, w2 = ok ? __fmul_rn(Y.h, X.l) : 0.f;
        const float w3 = ok ? __fmul_rn(Y.l, X.h) : 0.f, w4 = ok ? __fmul_rn(Y.l, X.l) : 0.f;
        tab_w[e] = make_float4(w1, w2, w3, w4);
    }
    __syncthreads();
    for (int b = tid; b < nbins; b += kRoiThreads) {
        const int ph = ph0 + b / PW, pw = b % PW;
        const bool all_in = ytab[2 * ph].valid && ytab[2 * ph + 1].valid && xtab[2 * pw].valid && xtab[2 * pw + 1].valid;
        s_bin[b] = ph | (pw << 8) | ((all_in ? s_py[ph] * 3 + s_px[pw] : 9) << 16);     // 9: a sample outside the map -> skipped, not weighted by 0
    }
    __syncthreads();
    const char* img = reinterpret_cast<const char*>(p.features[g.level]) + (size_t)g.batch * g.H * g.W * C * 4;
    const int rot4 = lane >> 3;
    int so4[4];                                                        // smem row offsets in rotated order
#pragma unroll
    for (int t = 0; t < 4; ++t) so4[t] = ((rot4 + t) & 3) * opitch;
    const int nchunks = (C + kChunk4 - 1) / kChunk4;
    // With an odd bin count the staged chunk [128][nbins] IS the output layout: it leaves through one bulk
    // async copy (TMA, cp.async.bulk shared -> global) issued by one thread instead of LDS.128 + STG.128 by all
    // (a third of this kernel's L1 wavefronts). One buffer: a second one costs a resident CTA and measured slower.
    const bool bulk = gridDim.y == 1 && opitch == nbins && ((reinterpret_cast<uintptr_t>(dst_roi) & 15) == 0) &&
                      ((kChunk4 * nbins) & 3) == 0;
    for (int chunk = 0; chunk < nchunks; ++chunk) {
        const int c0 = chunk * kChunk4;
        const int nch = min(kChunk4, C - c0);
        if (bulk && chunk > 0) {            // the previous chunk's copy must have finished reading the buffer
            if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            __syncthreads();
        }
        if (4 * lane < nch) {
            const char* gp = img + (size_t)(c0 + 4 * lane) * 4;
            for (int b = warp; b < nbins; b += kRoiWarps) {
                const int info = s_bin[b];
                const uint4 ro4 = s_ro[info & 0xff], co4 = s_co[(info >> 8) & 0xff];
                const float4* tw = tab_w + b * 4;
                float4 av;
                switch (info >> 16) {      // warp-uniform
                    case 0: av = bin_dedup<EXACT, 0, 0>(gp, ro4, co4, tw, ones); break;
                    case 1: av = bin_dedup<EXACT, 0, 1>(gp, ro4, co4, tw, ones); break;
                    case 2: av = bin_dedup<EXACT, 0, 2>(gp, ro4, co4, tw, ones); break;
                    case 3: av = bin_dedup<EXACT, 1, 0>(gp, ro4, co4, tw, ones); break;
                    case 4: av = bin_dedup<EXACT, 1, 1>(gp, ro4, co4, tw, ones); break;
                    case 5: av = bin_dedup<EXACT, 1, 2>(gp, ro4, co4, tw, ones); break;
                    case 6: av = bin_dedup<EXACT, 2, 0>(gp, ro4, co4, tw, ones); break;
                    case 7: av = bin_dedup<EXACT, 2, 1>(gp, ro4, co4, tw, ones); break;
                    case 8: av = bin_dedup<EXACT, 2, 2>(gp, ro4, co4, tw, ones); break;
                    default: av = bin_skip_invalid<EXACT>(gp, ytab, xtab, info & 0xff, (info >> 8) & 0xff,
                                                         (unsigned)g.W * (unsigned)C * 4u, (unsigned)C * 4u); break;
                }
                rotate4(av, rot4);
                float* o = ob + (4 * lane) * opitch + b;
                o[so4[0]] = av.x; o[so4[1]] = av.y; o[so4[2]] = av.z; o[so4[3]] = av.w;
            }
        }
        float* dst = dst_roi + (size_t)c0 * nbins_all + b0;
        const int total = nch * nbins;
        if (bulk && (total & 3) == 0) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the async proxy
            __syncthreads();
            if (tid == 0) {
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n\tcp.async.bulk.commit_group;"
                             :: "l"(dst), "r"(smem_u32(ob)), "r"(total * 4) : "memory");
            }
            continue;
        }
        __syncthreads();
        for (int ch = warp; ch < nch; ch += kRoiWarps)
            for (int b = lane; b < nbins; b += 32) dst[ch * nbins_all + b] = ob[ch * opitch + b];
        __syncthreads();   // ob is reused by the next chunk
    }
    if (bulk && tid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // smem must outlive the copies
}

// NCHW -> channels-last transpose of one feature map ([N][C][HW] -> [N][HW][C]), 32x32 tiles through
// shared memory: reads coalesced along HW, writes coalesced along C. Used when the total footprint
// volume of the RoIs is several times the size of the pyramid: one pass over the maps (read + write)
// is then cheaper than staging every RoI's footprint from the NCHW planes.
__global__ void __launch_bounds__(256) k_nchw_to_nhwc(const float* __restrict__ in, float* __restrict__ outp, int C, int HW) {
    __shared__ float tile[32][33];
    const int n = blockIdx.z;
    const int hw0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 8 rows per pass
    const float* src = in + (size_t)n * C * HW;
    float* dst = outp + (size_t)n * C * HW;
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
        const int c = c0 + r, hw = hw0 + tx;
        if (c < C && hw < HW) tile[r][tx] = __ldg(src + (size_t)c * HW + hw);
    }
    __syncthreads();
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
        const int hw = hw0 + r, c = c0 + tx;
        if (c < C && hw < HW) dst[(size_t)hw * C + c] = tile[tx][r];
    }
}

// Direct kernel: any sampling_ratio (incl. adaptive), any pooled size. One thread per output.
__global__ void __launch_bounds__(256) k_roi_align_direct(const mb_roi_align_params p, const float* __restrict__ rois,
                                                         long long total, float* __restrict__ out,
                                                         int* __restrict__ levels_out) {
    const int PH = p.pooled_h, PW = p.pooled_w;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const int pw = (int)(idx % PW);
        const int ph = (int)((idx / PW) % PH);
        const int c = (int)((idx / ((long long)PW * PH)) % p.channels);
        const long long k = idx / ((long long)PW * PH * p.channels);
        float r[5];
        load_roi(rois, k, p, r);
        RoiGeom g;
        roi_geometry(r, p, g);
        if (levels_out != nullptr && c == 0 && ph == 0 && pw == 0) levels_out[k] = g.level;
        float acc = 0.0f;
        if (g.batch >= 0 && g.batch < p.num_images) {
            const float* plane = p.features[g.level] + ((size_t)g.batch * p.channels + c) * (size_t)g.H * g.W;
            for (int iy = 0; iy < g.grid_h; ++iy) {
                const Tap Y = make_tap(g.start_h, g.bin_h, ph, iy, g.grid_h, g.H);
                if (!Y.valid) continue;
                for (int ix = 0; ix < g.grid_w; ++ix) {
                    const Tap X = make_tap(g.start_w, g.bin_w, pw, ix, g.grid_w, g.W);
                    if (!X.valid) continue;
                    acc = bilinear4<true>(Y.h, Y.l, X.h, X.l, __ldg(plane + Y.lo * g.W + X.lo),
                                          __ldg(plane + Y.lo * g.W + X.hi), __ldg(plane + Y.hi * g.W + X.lo),
                                          __ldg(plane + Y.hi * g.W + X.hi), acc);
                }
            }
        }
        out[idx] = __fdiv_rn(acc, g.count);
    }
}

}  // namespace mb

using namespace mb;

// roi_align_tma.cu: 1 = launched, 0 = outside its envelope (take the gather kernel), else an error code
int mb_launch_roi_align_tma(const mb_roi_align_params& p, const float* rois, int64_t num_rois, float* out,
                            int32_t* levels_out, void* workspace, size_t workspace_bytes, cudaStream_t stream);
size_t mb_roi_align_tma_workspace_bytes(const mb_roi_align_params& p, int64_t num_rois);

static size_t nhwc_copy_bytes(const mb_roi_align_params& p) {
    size_t b = 0;
    for (int l = 0; l < p.num_levels; ++l)
        b += align_up((size_t)p.num_images * p.channels * p.height[l] * p.width[l] * sizeof(float), 256);
    return b;
}

// bytes of the channels-last copies of NCHW maps (0: not applicable / not worth it)
static size_t nchw_transpose_bytes(const mb_roi_align_params* pp, int64_t num_rois) {
    if (pp->channels_last || pp->sampling_ratio != 2 || pp->pooled_h > 16 || pp->pooled_w > 16 || pp->channels % 4) return 0;
    const double footprint = (double)num_rois * pp->channels * 320.0 * sizeof(float);   // ~320 pixels per RoI and channel
    const size_t maps = nhwc_copy_bytes(*pp);
    return footprint >= 1.5 * (double)maps ? maps + 256 : 0;
}

// Workspace: per-RoI tap-table records of the TMA-staged kernel (channels-last maps) and, for NCHW maps whose
// RoIs cover the pyramid several times over, room for one channels-last copy of the maps.
extern "C" size_t mb_roi_align_workspace_bytes(const mb_roi_align_params* pp, int64_t num_rois) {
    if (!pp || num_rois <= 0) return 0;
    const size_t maps = nchw_transpose_bytes(pp, num_rois);
    const size_t recs = (pp->channels_last || maps) ? mb_roi_align_tma_workspace_bytes(*pp, num_rois) : 0;
    return maps + recs;
}

extern "C" int mb_multiscale_roi_align(const mb_roi_align_params* pp, const float* rois, int64_t num_rois,
                                       float* out, int32_t* levels_out, void* workspace,
                                       size_t workspace_bytes, mb_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!pp) return MB_ERR_INVALID_ARG;
    mb_roi_align_params p = *pp;
    if (p.num_levels < 1 || p.num_levels > MB_MAX_LEVELS || p.channels < 1 || p.pooled_h < 1 || p.pooled_w < 1 ||
        p.num_images < 1 || num_rois < 0)
        return MB_ERR_INVALID_ARG;
    for (int l = 0; l < p.num_levels; ++l)
        if (!p.features[l] || p.height[l] < 1 || p.width[l] < 1) return MB_ERR_INVALID_ARG;
    if (num_rois == 0) return MB_OK;
    if (!rois || !out) return MB_ERR_INVALID_ARG;
    const int nbins = p.pooled_h * p.pooled_w;
    const long long chunks = (p.channels + kChunk - 1) / kChunk;
    const bool staged = p.sampling_ratio > 0 && p.sampling_ratio * p.pooled_h <= kMaxSamples &&
                        p.sampling_ratio * p.pooled_w <= kMaxSamples && nbins <= 512 &&
                        num_rois * chunks < (1ll << 31);
    if (!p.channels_last && workspace != nullptr && num_rois > 0) {
        // NCHW input with a workspace from mb_roi_align_workspace_bytes: transpose once, gather channels-last
        const size_t need = nchw_transpose_bytes(&p, num_rois);
        if (need != 0 && workspace_bytes >= need && (reinterpret_cast<uintptr_t>(workspace) & 15) == 0) {
            char* w = (char*)workspace;
            for (int l = 0; l < p.num_levels; ++l) {
                const int HW = p.height[l] * p.width[l];
                dim3 grid(ceil_div(HW, 32), ceil_div(p.channels, 32), p.num_images);
                k_nchw_to_nhwc<<<grid, 256, 0, stream>>>(p.features[l], (float*)w, p.channels, HW);
                MB_LAUNCH_CHECK();
                p.features[l] = (const float*)w;
                w += align_up((size_t)p.num_images * p.channels * HW * sizeof(float), 256);
            }
            p.channels_last = 1;
            workspace = (char*)workspace + need;      // what is left holds the TMA kernel's records
            workspace_bytes -= need;
        }
    }
    // route: force_gather 0 = library default, 1 = register-gather kernel, 2 = TMA-staged kernel
    static const bool tma_default = getenv("MB_ROI_TMA") && atoi(getenv("MB_ROI_TMA")) != 0;
    if (p.channels_last && (p.force_gather == 2 || (p.force_gather == 0 && tma_default))) {
        const int r = mb_launch_roi_align_tma(p, rois, num_rois, out, levels_out, workspace, workspace_bytes, stream);
        if (r == 1) return MB_OK;
        if (r != 0) return r;
    }
    if (p.channels_last) {
        if (!(p.sampling_ratio == 2 && nbins <= 256 && p.pooled_h <= 16 && p.pooled_w <= 16 && num_rois < (1ll << 31)))
            return MB_ERR_UNSUPPORTED;   // the host converts to NCHW for other configurations
        const int opitch = (nbins & 1) ? nbins : nbins + 1;
        const bool vec = p.channels % 4 == 0;
        bool aligned16 = true;
        for (int l = 0; l < p.num_levels; ++l) aligned16 = aligned16 && ((reinterpret_cast<uintptr_t>(p.features[l]) & 15) == 0);
        bool small_maps = true;   // 32-bit byte offsets inside one image
        for (int l = 0; l < p.num_levels; ++l)
            small_maps = small_maps && ((unsigned long long)p.height[l] * p.width[l] * p.channels * 4ull < (1ull << 32));
        if (vec && aligned16 && small_maps) {
            // bands of pooled rows per CTA: at most 112 bins staged at a time (7x7: one band; 14x14: two bands of 7 rows)
            const int nsplit = ceil_div(nbins, 112);
            const int rows = ceil_div(p.pooled_h, nsplit);
            const int band = rows * p.pooled_w;
            const int smemd = ((kChunk4 * (band | 1) + 3) & ~3) * (int)sizeof(float) + band * 4 * 16 + band * 4;
            dim3 grid((unsigned)num_rois, (unsigned)ceil_div(p.pooled_h, rows));
            const float2 ones = make_float2(1.0f, 1.0f);
            static const int occ_env = getenv("MB_ROI_OCC") ? atoi(getenv("MB_ROI_OCC")) : 0;      // development switch
#define MB_NHWC4D(E, O)                                                                                              \
    do {                                                                                                            \
        MB_DYN_SMEM((k_roi_align_nhwc4d<E, O>), smemd); \
        MB_CUDA(launch_pdl((k_roi_align_nhwc4d<E, O>), grid, kRoiThreads, smemd, stream, p, rois, out, levels_out, rows, ones)); \
    } while (0)
            if (p.exact) { if (occ_env == 3) MB_NHWC4D(true, 3); else MB_NHWC4D(true, 4); }
            else MB_NHWC4D(false, 4);
#undef MB_NHWC4D
            MB_LAUNCH_CHECK();
            return MB_OK;
        }
        const int obuf = (kChunk * opitch + 3) & ~3;
        const int smem = 2 * obuf * (int)sizeof(float) + nbins * 4 * 32;
        if (p.exact) {
            MB_DYN_SMEM(k_roi_align_nhwc<true>, smem);
            k_roi_align_nhwc<true><<<(int)num_rois, kRoiThreads, smem, stream>>>(p, rois, out, levels_out);
        } else {
            MB_DYN_SMEM(k_roi_align_nhwc<false>, smem);
            k_roi_align_nhwc<false><<<(int)num_rois, kRoiThreads, smem, stream>>>(p, rois, out, levels_out);
        }
        MB_LAUNCH_CHECK();
        return MB_OK;
    }
    if (staged && p.sampling_ratio == 2 && nbins <= 256 && p.pooled_h <= 16 && p.pooled_w <= 16 && num_rois < (1ll << 31)) {
        const int opitch = (nbins & 1) ? nbins : nbins + 1;
        const int variant = 2;   // bit0: no float4 staging, bit1: 16 scalar loads in flight (measured best: 2)
        const int patch_floats = kChunk * 321;   // footprint of up to 321 pixels per channel: 4 CTAs/SM at 7x7
        const int smem = (kChunk * opitch + patch_floats) * (int)sizeof(float) + nbins * 4 * 32;
        if (smem > 200 * 1024) return MB_ERR_UNSUPPORTED;
        if (p.exact) {
            MB_DYN_SMEM(k_roi_align_sr2<true>, smem);
            k_roi_align_sr2<true><<<(int)num_rois, kRoiThreads, smem, stream>>>(p, rois, out, levels_out, patch_floats, variant);
        } else {
            MB_DYN_SMEM(k_roi_align_sr2<false>, smem);
            k_roi_align_sr2<false><<<(int)num_rois, kRoiThreads, smem, stream>>>(p, rois, out, levels_out, patch_floats, variant);
        }
        MB_LAUNCH_CHECK();
        return MB_OK;
    }
    if (staged) {
        // staging buffer: outputs + a footprint of up to ~320 pixels per channel (4 CTAs/SM at 7x7)
        const int opitch = (nbins & 1) ? nbins : nbins + 1;
        const int stage_floats = kChunk * opitch + kChunk * 353;
        const int smem = stage_floats * (int)sizeof(float);
        if (smem > 200 * 1024) return MB_ERR_UNSUPPORTED;
        const int grid = (int)(num_rois * chunks);
#define MB_ROI_LAUNCH(E, S)                                                                                  \
    do {                                                                                                    \
        MB_DYN_SMEM((k_roi_align_staged<E, S>), smem); \
        k_roi_align_staged<E, S><<<grid, kRoiThreads, smem, stream>>>(p, rois, (int)num_rois, out, levels_out, stage_floats); \
    } while (0)
        const bool sr2 = p.sampling_ratio == 2;
        if (p.exact) { if (sr2) MB_ROI_LAUNCH(true, true); else MB_ROI_LAUNCH(true, false); }
        else { if (sr2) MB_ROI_LAUNCH(false, true); else MB_ROI_LAUNCH(false, false); }
#undef MB_ROI_LAUNCH
        MB_LAUNCH_CHECK();
        return MB_OK;
    }
    const long long total = num_rois * (long long)p.channels * nbins;
    const int grid = (int)min((long long)num_sms() * 32, ceil_div64(total, 256));
    k_roi_align_direct<<<grid, 256, 0, stream>>>(p, rois, total, out, levels_out);
    MB_LAUNCH_CHECK();
    return MB_OK;
}
