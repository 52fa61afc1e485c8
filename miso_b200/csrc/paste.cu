// paste.cu — paste_masks_in_image on the GPU (SURVEY.md §8f row 1).
//
// Replaces tv:models/detection/roi_heads.py:375-501 (expand_masks / expand_boxes / per-detection
// F.interpolate(bilinear, align_corners=False) / paste into a zero [R,1,H,W] tensor), which the
// reference runs as a Python loop per detection (and which the vendored engine flags:
// ref:miso/object_detection/engine/engine.py:80 "FIXME ... make paste_masks_in_image run on the GPU").
//
// One launch. CTA = (detection, band of image rows); the padded mask (M+2p)^2 sits in shared memory; a
// thread produces four consecutive pixels and writes them as one 16-byte store, so the kernel is an
// HBM write stream (R*H*W*4 bytes; 419 MB per 1024^2 image at R = 100) with arithmetic only inside
// the boxes. Arithmetic follows ATen's CPU upsample_bilinear2d as compiled with FMA contraction
// (aten/src/ATen/native/cpu/UpSampleKernel.cpp: source index = fma(scale, dst + 0.5, -0.5) clamped at
// 0, lambda = clamp(src - floor(src), 0, 1), value = fma(fma(v00, wx0, v01*wx1), wy0,
// fma(v10, wx0, v11*wx1) * wy1)): bit-identical to the reference for outputs of >= ~1600 pixels,
// within 1 ulp below (the reference's own small-output loop contracts differently).
//
// k_crop_masks (mb_crop_masks) is the same paste evaluated only at the pixels of each crop rectangle of mb_crop_plan and
// thresholded to 0 / 255 bytes: the per-crop instance masks without the [R, H, W] fp32 frame.
#include <algorithm>

#include "common.cuh"

namespace mb {

constexpr int kPasteThreads = 256;
constexpr int kPasteRows = 16;          // image rows per CTA
constexpr int kPasteMaxSide = 64;       // padded mask side kept in shared memory

struct PasteAxis {                      // one axis of one detection
    int lo, hi;                         // paste range [lo, hi) in image coordinates (empty if hi <= lo)
    int org;                            // integer box start (mask coordinate 0)
    float scale;                        // padded_side / resized_side
};

__device__ __forceinline__ void paste_axis(float b0, float b1, float mask_scale, int padded, int extent, PasteAxis& a) {
    // expand_boxes (tv:...roi_heads.py:375-391) in fp32, then .to(int64) (truncation)
    float half = __fmul_rn(__fsub_rn(b1, b0), 0.5f);
    const float ctr = __fmul_rn(__fadd_rn(b1, b0), 0.5f);
    half = __fmul_rn(half, mask_scale);
    const long long i0 = (long long)__fsub_rn(ctr, half), i1 = (long long)__fadd_rn(ctr, half);
    long long size = i1 - i0 + 1;                       // paste_mask_in_image: w = max(int(x2 - x1 + 1), 1)
    if (size < 1) size = 1;
    const long long lo = i0 > 0 ? i0 : 0, hi = (i1 + 1 < extent) ? i1 + 1 : extent;
    a.lo = (int)(lo < extent ? lo : extent);
    a.hi = (int)(hi > 0 ? hi : 0);
    a.org = (int)(i0 < -(1ll << 30) ? -(1ll << 30) : (i0 > (1ll << 30) ? (1ll << 30) : i0));   // only used inside [lo, hi)
    a.scale = __fdiv_rn((float)padded, (float)size);    // area_pixel_compute_scale: (float)input / output
}

// ATen area_pixel_compute_source_index + guard_index_and_lambda
__device__ __forceinline__ void paste_tap(float scale, int d, int padded, int& i0, int& i1, float& w0, float& w1) {
    float src = fmaf(scale, __fadd_rn((float)d, 0.5f), -0.5f);
    src = src < 0.f ? 0.f : src;
    i0 = min((int)src, padded - 1);
    w1 = fminf(fmaxf(__fsub_rn(src, (float)i0), 0.f), 1.f);
    w0 = __fsub_rn(1.0f, w1);
    i1 = i0 + (i0 < padded - 1 ? 1 : 0);
}

// ATen's bilinear value (UpSampleKernel.cpp, as compiled with FMA contraction) from two padded mask rows; every kernel
// that produces a pasted mask value calls this, so a pixel has the same bits in all of them
__device__ __forceinline__ float paste_value(const float* r0, const float* r1, int x0, int x1, float wx0, float wx1,
                                             float wy0, float wy1) {
    const float t0 = fmaf(r0[x0], wx0, __fmul_rn(r0[x1], wx1));
    const float t1 = fmaf(r1[x0], wx0, __fmul_rn(r1[x1], wx1));
    return fmaf(t0, wy0, __fmul_rn(t1, wy1));
}

__global__ void __launch_bounds__(kPasteThreads) k_paste_masks(const float* __restrict__ masks, const float4* __restrict__ boxes,
                                                               int M, int padding, float mask_scale, int H, int W,
                                                               float* __restrict__ out) {
    __shared__ float sm[kPasteMaxSide * kPasteMaxSide];
    const int r = blockIdx.y, tid = threadIdx.x;
    const int P = M + 2 * padding;
    for (int i = tid; i < P * P; i += kPasteThreads) {          // F.pad(mask, (padding,) * 4)
        const int y = i / P - padding, x = i % P - padding;
        sm[i] = (y >= 0 && y < M && x >= 0 && x < M) ? masks[(size_t)r * M * M + y * M + x] : 0.f;
    }
    const float4 b = boxes[r];
    PasteAxis ax, ay;
    paste_axis(b.x, b.z, mask_scale, P, W, ax);
    paste_axis(b.y, b.w, mask_scale, P, H, ay);
    __syncthreads();
    const int y_begin = blockIdx.x * kPasteRows, y_end = min(H, y_begin + kPasteRows);
    float* dst = out + (size_t)r * H * W;
    const bool vec = (W & 3) == 0 && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    const int groups = (W + 3) >> 2;
    for (int y = y_begin; y < y_end; ++y) {
        float* row = dst + (size_t)y * W;
        const bool live_row = y >= ay.lo && y < ay.hi && ax.hi > ax.lo;
        int y0 = 0, y1 = 0; float wy0 = 0.f, wy1 = 0.f;
        if (live_row) paste_tap(ay.scale, y - ay.org, P, y0, y1, wy0, wy1);
        const float* r0 = sm + y0 * P; const float* r1 = sm + y1 * P;
        for (int gq = tid; gq < groups; gq += kPasteThreads) {
            const int x4 = gq << 2;
            float v[4] = {0.f, 0.f, 0.f, 0.f};
            if (live_row && x4 < ax.hi && x4 + 4 > ax.lo) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int x = x4 + j;
                    if (x >= ax.lo && x < ax.hi) {
                        int x0, x1; float wx0, wx1;
                        paste_tap(ax.scale, x - ax.org, P, x0, x1, wx0, wx1);
                        v[j] = paste_value(r0, r1, x0, x1, wx0, wx1, wy0, wy1);
                    }
                }
            }
            if (vec) {
                __stcs(reinterpret_cast<float4*>(row + x4), make_float4(v[0], v[1], v[2], v[3]));   // streamed: written once, read by nobody here
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) if (x4 + j < W) row[x4 + j] = v[j];
            }
        }
    }
}

// Instance masks cut to the crop rectangles of mb_crop_plan: crop j (slot s = src[j], rectangle rc) gets
// (paste of mask s into its frame)[rc] > thr as 0 / 255 bytes, 0 where rc leaves the frame — only the crop's pixels are
// computed, never the frame. Work split of k_crop_gather: crops strided over blockIdx.x (the next crop's metadata
// prefetched), rows over the warps; the padded mask sits in shared memory, the x taps of the crop's columns are staged
// next to it once per crop (kMaskCols columns per pass), the y taps once per row. Lanes write 4-byte words between the
// row's unaligned ends.
constexpr int kMaskThreads = 256;
constexpr int kMaskCols = 1024;

struct CropMaskDev {
    int M, P, ch, rows_per_frame;
    float mask_scale, thr;
    int img_h[MB_MAX_IMAGES], img_w[MB_MAX_IMAGES];     // frame f of a NULL frame table: image f at (0, 0)
};

__global__ void __launch_bounds__(kMaskThreads) k_crop_masks(const CropMaskDev d, const float* __restrict__ probs,
                                                             const float4* __restrict__ boxes, const int4* __restrict__ frames,
                                                             const int4* __restrict__ rects, const int* __restrict__ src,
                                                             const long long* __restrict__ offsets, long long* __restrict__ totals,
                                                             unsigned char* __restrict__ out, long long capacity) {
    __shared__ float sm[kPasteMaxSide * kPasteMaxSide];
    __shared__ int2 taps[kMaskCols];       // (x0, bits of lambda1); x0 = -1: inside the frame, outside the paste box; -2: outside the frame
    const long long ncrops = totals[0];
    const bool overflow = totals[1] / d.ch > capacity;
    if (blockIdx.x == 0 && threadIdx.x == 0) totals[3] = overflow ? 1 : 0;      // caller re-runs with totals[1] / ch bytes
    if (overflow) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int nwarps = kMaskThreads / 32;
    const int M = d.M, P = d.P, pad = (P - M) / 2;
    int4 rc_next = make_int4(0, 0, 0, 0);
    int src_next = 0;
    long long off_next = 0;
    if ((long long)blockIdx.x < ncrops) { rc_next = rects[blockIdx.x]; src_next = src[blockIdx.x]; off_next = offsets[blockIdx.x]; }
    for (long long j = blockIdx.x; j < ncrops; j += gridDim.x) {
        const int4 rc = rc_next;
        const int s = src_next;
        unsigned char* dst = out + off_next / d.ch;         // every crop holds h * w * ch bytes
        const long long jn = j + gridDim.x;
        if (jn < ncrops) { rc_next = rects[jn]; src_next = src[jn]; off_next = offsets[jn]; }
        if (rc.z == 0 || rc.w == 0) continue;
        const int f = s / d.rows_per_frame;
        const int4 fr = frames ? frames[f] : make_int4(0, 0, d.img_w[f], d.img_h[f]);      // (x0, y0, w, h)
        __syncthreads();                                     // the previous crop's mask and taps are no longer read
        const float* mk = probs + (size_t)s * M * M;
        for (int i = tid; i < P * P; i += kMaskThreads) {    // F.pad(mask, (padding,) * 4)
            const int y = i / P - pad, x = i % P - pad;
            sm[i] = (y >= 0 && y < M && x >= 0 && x < M) ? mk[y * M + x] : 0.f;
        }
        const float4 b = boxes[s];
        PasteAxis ax, ay;
        paste_axis(b.x, b.z, d.mask_scale, P, fr.z, ax);
        paste_axis(b.y, b.w, d.mask_scale, P, fr.w, ay);
        for (int c0 = 0; c0 < rc.z; c0 += kMaskCols) {
            const int cn = min(kMaskCols, rc.z - c0);
            if (c0 > 0) __syncthreads();
            for (int c = tid; c < cn; c += kMaskThreads) {
                const int fx = rc.x + c0 + c - fr.x;
                int2 t = make_int2(fx >= 0 && fx < fr.z ? -1 : -2, 0);
                if (fx >= ax.lo && fx < ax.hi) {
                    int x0, x1; float w0, w1;
                    paste_tap(ax.scale, fx - ax.org, P, x0, x1, w0, w1);
                    t = make_int2(x0, __float_as_int(w1));
                }
                taps[c] = t;
            }
            __syncthreads();
            for (int r = warp; r < rc.w; r += nwarps) {
                const int fy = rc.y + r - fr.y;
                const bool in_frame = fy >= 0 && fy < fr.w;
                const bool live = fy >= ay.lo && fy < ay.hi;     // [lo, hi) lies inside the frame
                int y0 = 0, y1 = 0; float wy0 = 0.f, wy1 = 0.f;
                if (live) paste_tap(ay.scale, fy - ay.org, P, y0, y1, wy0, wy1);
                const float* r0 = sm + y0 * P; const float* r1 = sm + y1 * P;
                auto px = [&](int c) -> unsigned {
                    const int2 t = taps[c];
                    if (!in_frame || t.x == -2) return 0u;
                    float v = 0.f;                               // the paste's zero image outside the box
                    if (live && t.x >= 0) {
                        const float w1 = __int_as_float(t.y);
                        v = paste_value(r0, r1, t.x, t.x + (t.x < P - 1 ? 1 : 0), __fsub_rn(1.0f, w1), w1, wy0, wy1);
                    }
                    return v > d.thr ? 255u : 0u;
                };
                unsigned char* orow = dst + (size_t)r * rc.z + c0;
                const int head = min(cn, (int)((4u - ((unsigned)reinterpret_cast<uintptr_t>(orow) & 3u)) & 3u));
                const int nw = (cn - head) >> 2, tail = head + 4 * nw;
                if (lane < head) orow[lane] = (unsigned char)px(lane);
                for (int i = lane; i < nw; i += 32) {
                    const int c = head + 4 * i;
                    *reinterpret_cast<unsigned*>(orow + c) = px(c) | (px(c + 1) << 8) | (px(c + 2) << 16) | (px(c + 3) << 24);
                }
                if (lane < cn - tail) orow[tail + lane] = (unsigned char)px(tail + lane);
            }
        }
    }
}

// maskrcnn_inference (tv:models/detection/roi_heads.py:56-82): sigmoid of the channel the predicted label selects,
// [R, C, M, M] logits + [R] labels -> [R, 1, M, M] probabilities. One launch that reads only the selected channel
// (the reference runs sigmoid over all C channels, builds an index and gathers).
__global__ void __launch_bounds__(256) k_mask_prob(const float* __restrict__ logits, const long long* __restrict__ labels,
                                                  int num_classes, int plane, long long total, float* __restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / plane;
        const int p = (int)(i - r * plane);
        long long c = labels[r];
        if (c < 0) c += num_classes;                       // python indexing
        const float x = logits[((size_t)r * num_classes + (size_t)c) * plane + p];
        out[i] = __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-x)));
    }
}

}  // namespace mb

extern "C" int mb_mask_prob(const float* mask_logits, const int64_t* labels, int64_t num_masks, int32_t num_classes,
                            int32_t mask_side, float* out, mb_stream_t stream) {
    if (num_masks < 0 || num_classes < 1 || mask_side < 1) return MB_ERR_INVALID_ARG;
    if (num_masks == 0) return MB_OK;
    if (!mask_logits || !labels || !out) return MB_ERR_INVALID_ARG;
    const int plane = mask_side * mask_side;
    const long long total = num_masks * (long long)plane;
    const int grid = (int)min((long long)mb::num_sms() * 8, (total + 255) / 256);
    mb::k_mask_prob<<<grid, 256, 0, (cudaStream_t)stream>>>(mask_logits, (const long long*)labels, num_classes, plane, total, out);
    MB_LAUNCH_CHECK();
    return MB_OK;
}

extern "C" int mb_paste_masks(const float* masks, const float* boxes, int64_t num_masks, int32_t mask_side, int32_t padding,
                              int32_t im_h, int32_t im_w, float* out, mb_stream_t stream) {
    if (num_masks < 0 || mask_side < 1 || padding < 0 || im_h < 1 || im_w < 1) return MB_ERR_INVALID_ARG;
    if (mask_side + 2 * padding > mb::kPasteMaxSide || num_masks > 65535) return MB_ERR_UNSUPPORTED;
    if (num_masks == 0) return MB_OK;
    if (!masks || !boxes || !out) return MB_ERR_INVALID_ARG;
    // expand_masks: scale = float(M + 2 * padding) / M (a Python double), applied to fp32 tensors as an fp32 scalar
    const float mask_scale = (float)((double)(mask_side + 2 * padding) / (double)mask_side);
    dim3 grid((im_h + mb::kPasteRows - 1) / mb::kPasteRows, (unsigned)num_masks);
    mb::k_paste_masks<<<grid, mb::kPasteThreads, 0, (cudaStream_t)stream>>>(masks, reinterpret_cast<const float4*>(boxes), mask_side,
                                                                           padding, mask_scale, im_h, im_w, out);
    MB_LAUNCH_CHECK();
    return MB_OK;
}

extern "C" int mb_crop_masks(const mb_crop_params* p, const float* mask_probs, const float* paste_boxes, int32_t mask_side,
                             int32_t padding, const int32_t* frames, int32_t rows_per_frame, float mask_threshold,
                             const int32_t* rects, const int32_t* src, const int64_t* offsets, int64_t* totals,
                             uint8_t* masks_out, int64_t masks_capacity_bytes, mb_stream_t stream) {
    if (!p || mask_side < 1 || padding < 0 || rows_per_frame < 1 || masks_capacity_bytes < 0) return MB_ERR_INVALID_ARG;
    if (p->num_images < 1 || p->num_images > MB_MAX_IMAGES || p->capacity < 1 || p->channels < 1) return MB_ERR_INVALID_ARG;
    if (mask_side + 2 * padding > mb::kPasteMaxSide) return MB_ERR_UNSUPPORTED;
    if (!mask_probs || !paste_boxes || !rects || !src || !offsets || !totals || (masks_capacity_bytes > 0 && !masks_out))
        return MB_ERR_INVALID_ARG;
    if (!frames && rows_per_frame < p->capacity) return MB_ERR_INVALID_ARG;        // frame f = image f needs f < num_images
    mb::CropMaskDev d;
    d.M = mask_side; d.P = mask_side + 2 * padding; d.ch = p->channels; d.rows_per_frame = rows_per_frame;
    d.mask_scale = (float)((double)(mask_side + 2 * padding) / (double)mask_side);     // as mb_paste_masks
    d.thr = mask_threshold;
    for (int n = 0; n < MB_MAX_IMAGES; ++n) {
        const bool used = n < p->num_images;
        if (used && (p->image_h[n] < 0 || p->image_w[n] < 0)) return MB_ERR_INVALID_ARG;
        d.img_h[n] = used ? p->image_h[n] : 0; d.img_w[n] = used ? p->image_w[n] : 0;
    }
    const long long slots = (long long)p->num_images * p->capacity;
    const int grid = (int)std::min<long long>(std::max<long long>(slots, 1), (long long)mb::num_sms() * 8);
    mb::k_crop_masks<<<grid, mb::kMaskThreads, 0, (cudaStream_t)stream>>>(
        d, mask_probs, reinterpret_cast<const float4*>(paste_boxes), reinterpret_cast<const int4*>(frames),
        reinterpret_cast<const int4*>(rects), src, (const long long*)offsets, (long long*)totals, masks_out, masks_capacity_bytes);
    MB_LAUNCH_CHECK();
    return MB_OK;
}
