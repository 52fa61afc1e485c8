// train.cu — the training-side siblings of the hot path's kernels (SURVEY.md §8f row 4), so that
// `train-object-detector` (ref:miso/object_detection/engine/engine.py:33-49 -> model(images, targets)) runs the same
// data through libmisob200:
//
//   mb_box_iou            torchvision.ops.box_iou (tv:ops/boxes.py:299-330): [N,4] x [M,4] -> [N,M], the reference's
//                         operation order (area, max/min, clamp, product, (a1 + a2) - inter, division), bit-exact.
//   mb_match_encode       RegionProposalNetwork.assign_targets_to_anchors / RoIHeads.assign_targets_to_proposals
//                         (tv:models/detection/rpn.py:193-229, roi_heads.py:580-614) fused: box_iou(gt, anchors) is
//                         never materialised ([M, N] = 50 x 159 882 fp32 per image in the reference); Matcher
//                         (tv:models/detection/_utils.py:345-426: max over gt with the first maximum's index,
//                         BELOW_LOW = -1 / BETWEEN = -2, allow_low_quality_matches) and BoxCoder.encode_single
//                         (encode_boxes, _utils.py:85-127) of the matched gt box run in two passes over the anchors.
//   mb_roi_align_backward torchvision::_roi_align_backward (tv-csrc:ops/cuda/roi_align_kernel.cu, autograd wrapper
//                         tv-csrc:ops/autograd/roi_align_kernel.cpp:159): CTA = (RoI, 32-channel chunk); the RoI's
//                         footprint gradient is accumulated in shared memory (lane = channel, plane pitch odd: 32
//                         banks) and leaves as ONE atomic add per touched pixel and channel instead of the
//                         reference's 16 x bins global atomics per channel.
#include <math.h>

#include "common.cuh"
#include "roi_common.cuh"

namespace mb {

// IoU with torchvision's _box_inter_union order (a = boxes1[i], b = boxes2[j])
__device__ __forceinline__ float iou_tv(const float4 a, const float area_a, const float4 b, const float area_b) {
    const float ltx = fmaxf(a.x, b.x), lty = fmaxf(a.y, b.y);
    const float rbx = fminf(a.z, b.z), rby = fminf(a.w, b.w);
    const float w = fmaxf(__fsub_rn(rbx, ltx), 0.0f), h = fmaxf(__fsub_rn(rby, lty), 0.0f);
    const float inter = __fmul_rn(w, h);
    return __fdiv_rn(inter, __fsub_rn(__fadd_rn(area_a, area_b), inter));
}
__device__ __forceinline__ float area_tv(const float4 b) { return __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y)); }

__global__ void __launch_bounds__(256) k_box_iou(const float4* __restrict__ b1, int n1, const float4* __restrict__ b2, int n2,
                                                float* __restrict__ out) {
    const long long total = (long long)n1 * n2;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(idx / n2), j = (int)(idx - (long long)i * n2);
        const float4 a = b1[i], b = b2[j];
        out[idx] = iou_tv(a, area_tv(a), b, area_tv(b));
    }
}

// order-preserving map float -> unsigned (works for negative values too), for atomicMax
__device__ __forceinline__ unsigned ord_key(float v) {
    unsigned u = __float_as_uint(v);
    if (u == 0x80000000u) u = 0u;             // -0 == +0
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

constexpr int kMatchGtChunk = 1024;

// pass 1: per anchor the best gt (first maximum; a NaN IoU is a maximum like in torch.max) and per gt the highest
// IoU over all anchors (warp-reduced, one atomic per warp and gt)
__global__ void __launch_bounds__(256) k_match_best(const float4* __restrict__ gt, int m, const float4* __restrict__ anchors, int n,
                                                   float* __restrict__ best_val, int* __restrict__ best_idx,
                                                   unsigned* __restrict__ gt_max, int* __restrict__ gt_nan) {
    __shared__ float4 s_gt[kMatchGtChunk];
    __shared__ float s_area[kMatchGtChunk];
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = j < n;
    const float4 a = live ? anchors[j] : make_float4(0, 0, 0, 0);
    const float area_a = area_tv(a);
    float bv = -INFINITY;
    int bi = 0;
    bool have = false;
    for (int g0 = 0; g0 < m; g0 += kMatchGtChunk) {
        const int cnt = min(kMatchGtChunk, m - g0);
        __syncthreads();
        for (int i = threadIdx.x; i < cnt; i += blockDim.x) { s_gt[i] = gt[g0 + i]; s_area[i] = area_tv(s_gt[i]); }
        __syncthreads();
        for (int i = 0; i < cnt; ++i) {
            const float v = live ? iou_tv(s_gt[i], s_area[i], a, area_a) : -INFINITY;     // box_iou(gt, anchors)[g, j]
            if (live) {
                if (!have) { bv = v; bi = g0 + i; have = true; }
                else if (bv == bv && (v > bv || v != v)) { bv = v; bi = g0 + i; }          // first maximum; NaN wins once
            }
            // highest quality per gt over this warp's anchors
            const bool isn = live && v != v;
            unsigned k = (live && !isn) ? ord_key(v) : 0u;
#pragma unroll
            for (int o = 16; o; o >>= 1) k = max(k, __shfl_xor_sync(0xffffffffu, k, o));
            const unsigned anyn = __ballot_sync(0xffffffffu, isn);
            if ((threadIdx.x & 31) == 0) {
                if (k) atomicMax(&gt_max[g0 + i], k);
                if (anyn) atomicOr(&gt_nan[g0 + i], 1);
            }
        }
    }
    if (live) { best_val[j] = bv; best_idx[j] = bi; }
}

struct EncodeW { float wx, wy, ww, wh; };

// pass 2: thresholds, low-quality restoration, encode of the matched gt box
__global__ void __launch_bounds__(256) k_match_finish(const float4* __restrict__ gt, int m, const float4* __restrict__ anchors, int n,
                                                     float high, float low, int allow_low, EncodeW ew,
                                                     const float* __restrict__ best_val, const int* __restrict__ best_idx,
                                                     const unsigned* __restrict__ gt_max, const int* __restrict__ gt_nan,
                                                     long long* __restrict__ matches, float* __restrict__ vals_out,
                                                     float4* __restrict__ targets) {
    __shared__ float4 s_gt[kMatchGtChunk];
    __shared__ float s_area[kMatchGtChunk];
    __shared__ unsigned s_max[kMatchGtChunk];
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = j < n;
    const float4 a = live ? anchors[j] : make_float4(0, 0, 0, 0);
    const float area_a = area_tv(a);
    bool restore = false;
    if (allow_low) {
        for (int g0 = 0; g0 < m; g0 += kMatchGtChunk) {
            const int cnt = min(kMatchGtChunk, m - g0);
            __syncthreads();
            for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
                s_gt[i] = gt[g0 + i]; s_area[i] = area_tv(s_gt[i]);
                s_max[i] = gt_nan[g0 + i] ? 0u : gt_max[g0 + i];      // a NaN in the gt's row: its maximum is NaN, nothing equals it
            }
            __syncthreads();
            if (live)
                for (int i = 0; i < cnt; ++i) {
                    const float v = iou_tv(s_gt[i], s_area[i], a, area_a);
                    restore = restore || (v == v && s_max[i] != 0u && ord_key(v) == s_max[i]);
                }
        }
    }
    if (!live) return;
    const float v = best_val[j];
    const int bi = best_idx[j];
    long long mt = bi;
    if (v < low) mt = -1;                              // BELOW_LOW_THRESHOLD
    else if (v >= low && v < high) mt = -2;            // BETWEEN_THRESHOLDS
    if (restore) mt = bi;
    matches[j] = mt;
    if (vals_out) vals_out[j] = v;
    if (targets) {
        const float4 r = gt[mt < 0 ? 0 : (int)mt];     // gt_boxes[matched_idxs.clamp(min=0)]
        const float ew_ = __fsub_rn(a.z, a.x), eh = __fsub_rn(a.w, a.y);
        const float ecx = __fadd_rn(a.x, __fmul_rn(0.5f, ew_)), ecy = __fadd_rn(a.y, __fmul_rn(0.5f, eh));
        const float gw = __fsub_rn(r.z, r.x), gh = __fsub_rn(r.w, r.y);
        const float gcx = __fadd_rn(r.x, __fmul_rn(0.5f, gw)), gcy = __fadd_rn(r.y, __fmul_rn(0.5f, gh));
        float4 t;
        t.x = __fdiv_rn(__fmul_rn(ew.wx, __fsub_rn(gcx, ecx)), ew_);
        t.y = __fdiv_rn(__fmul_rn(ew.wy, __fsub_rn(gcy, ecy)), eh);
        t.z = __fmul_rn(ew.ww, logf(__fdiv_rn(gw, ew_)));
        t.w = __fmul_rn(ew.wh, logf(__fdiv_rn(gh, eh)));
        targets[j] = t;
    }
}

// ---------------------------------------------------------------------------------------------------------
// RoIAlign backward
// ---------------------------------------------------------------------------------------------------------
constexpr int kBwdThreads = 256;
constexpr int kBwdChunk = 32;

__global__ void __launch_bounds__(kBwdThreads) k_roi_align_backward(const float* __restrict__ grad, const float* __restrict__ rois,
                                                                   float scale, int C, int H, int W, int PH, int PW, int sr,
                                                                   int aligned, int batch, float* __restrict__ gin, int patch_floats) {
    extern __shared__ __align__(16) float bsm[];
    const int chunks = (C + kBwdChunk - 1) / kBwdChunk;
    const int k = blockIdx.x / chunks, c0 = (blockIdx.x % chunks) * kBwdChunk;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = kBwdThreads / 32;
    const float* q = rois + (size_t)k * 5;
    const int b = (int)q[0];
    if (b < 0 || b >= batch) return;
    const float off = aligned ? 0.5f : 0.0f;
    const float sw = __fsub_rn(__fmul_rn(q[1], scale), off), sh = __fsub_rn(__fmul_rn(q[2], scale), off);
    const float ew = __fsub_rn(__fmul_rn(q[3], scale), off), eh = __fsub_rn(__fmul_rn(q[4], scale), off);
    float rw = __fsub_rn(ew, sw), rh = __fsub_rn(eh, sh);
    if (!aligned) { rw = fmaxf(rw, 1.0f); rh = fmaxf(rh, 1.0f); }
    const float bin_h = __fdiv_rn(rh, (float)PH), bin_w = __fdiv_rn(rw, (float)PW);
    const int gh = sr > 0 ? sr : (int)ceilf(__fdiv_rn(rh, (float)PH)), gw = sr > 0 ? sr : (int)ceilf(__fdiv_rn(rw, (float)PW));
    const float count = (float)max(gh * gw, 1);
    // footprint of the RoI (clamped to the map): rows y0..y1, cols x0..x1
    const float ylo = sh, yhi = __fadd_rn(sh, rh), xlo = sw, xhi = __fadd_rn(sw, rw);
    int y0 = max((int)floorf(fmaxf(ylo, 0.0f)), 0), y1 = min((int)floorf(fmaxf(yhi, 0.0f)) + 1, H - 1);
    int x0 = max((int)floorf(fmaxf(xlo, 0.0f)), 0), x1 = min((int)floorf(fmaxf(xhi, 0.0f)) + 1, W - 1);
    y0 = min(y0, H - 1); x0 = min(x0, W - 1);
    const int rows = max(y1 - y0 + 1, 1), cols = max(x1 - x0 + 1, 1);
    const int pix = rows * cols;
    const int pitch = pix | 1;                               // odd plane pitch: lane = channel hits 32 banks
    const bool staged = pitch * kBwdChunk <= patch_floats;
    const int c = c0 + lane;
    const bool c_ok = c < C;
    if (staged) {
        for (int i = tid; i < pitch * kBwdChunk; i += kBwdThreads) bsm[i] = 0.0f;
        __syncthreads();
    }
    float* gplane = gin + ((size_t)b * C + c) * (size_t)H * W;
    float* sp = bsm + lane * pitch;
    const int nbins = PH * PW;
    for (int bin = warp; bin < nbins; bin += nwarps) {
        const int ph = bin / PW, pw = bin - ph * PW;
        const float g = c_ok ? grad[((size_t)k * C + c) * nbins + bin] : 0.0f;
        for (int iy = 0; iy < gh; ++iy) {
            const Tap Y = make_tap(sh, bin_h, ph, iy, gh, H);
            if (!Y.valid) continue;
            for (int ix = 0; ix < gw; ++ix) {
                const Tap X = make_tap(sw, bin_w, pw, ix, gw, W);
                if (!X.valid || !c_ok) continue;
                // the reference's order: g_i = grad * w_i / count
                const float g1 = __fdiv_rn(__fmul_rn(g, __fmul_rn(Y.h, X.h)), count), g2 = __fdiv_rn(__fmul_rn(g, __fmul_rn(Y.h, X.l)), count);
                const float g3 = __fdiv_rn(__fmul_rn(g, __fmul_rn(Y.l, X.h)), count), g4 = __fdiv_rn(__fmul_rn(g, __fmul_rn(Y.l, X.l)), count);
                const bool in = staged && Y.lo >= y0 && Y.hi <= y1 && X.lo >= x0 && X.hi <= x1;
                if (in) {
                    atomicAdd(sp + (Y.lo - y0) * cols + (X.lo - x0), g1);
                    atomicAdd(sp + (Y.lo - y0) * cols + (X.hi - x0), g2);
                    atomicAdd(sp + (Y.hi - y0) * cols + (X.lo - x0), g3);
                    atomicAdd(sp + (Y.hi - y0) * cols + (X.hi - x0), g4);
                } else {
                    atomicAdd(gplane + (size_t)Y.lo * W + X.lo, g1);
                    atomicAdd(gplane + (size_t)Y.lo * W + X.hi, g2);
                    atomicAdd(gplane + (size_t)Y.hi * W + X.lo, g3);
                    atomicAdd(gplane + (size_t)Y.hi * W + X.hi, g4);
                }
            }
        }
    }
    if (!staged) return;
    __syncthreads();
    // flush: thread = footprint pixel (x fastest -> coalesced atomics along a map row), loop over channels
    for (int cc = warp; cc < min(kBwdChunk, C - c0); cc += nwarps) {
        float* gp = gin + ((size_t)b * C + c0 + cc) * (size_t)H * W;
        const float* s = bsm + cc * pitch;
        for (int p = lane; p < pix; p += 32) {
            const float v = s[p];
            if (v != 0.0f) atomicAdd(gp + (size_t)(y0 + p / cols) * W + x0 + p % cols, v);
        }
    }
}

}  // namespace mb

using namespace mb;

extern "C" int mb_box_iou(const float* boxes1, int64_t n1, const float* boxes2, int64_t n2, float* iou_out, mb_stream_t stream) {
    if (n1 < 0 || n2 < 0 || n1 >= (1ll << 31) || n2 >= (1ll << 31)) return MB_ERR_INVALID_ARG;
    if (n1 == 0 || n2 == 0) return MB_OK;
    if (!boxes1 || !boxes2 || !iou_out) return MB_ERR_INVALID_ARG;
    const long long total = n1 * n2;
    const int grid = (int)min((long long)num_sms() * 16, ceil_div64(total, 256));
    k_box_iou<<<grid, 256, 0, (cudaStream_t)stream>>>((const float4*)boxes1, (int)n1, (const float4*)boxes2, (int)n2, iou_out);
    MB_LAUNCH_CHECK();
    return MB_OK;
}

extern "C" size_t mb_match_encode_workspace_bytes(int64_t num_gt, int64_t num_anchors) {
    if (num_gt < 0 || num_anchors < 0) return 0;
    Carver c(nullptr, 0);
    c.take<unsigned>((size_t)num_gt); c.take<int>((size_t)num_gt);
    c.take<float>((size_t)num_anchors); c.take<int>((size_t)num_anchors);
    return c.off + 256;
}

extern "C" int mb_match_encode(const float* gt_boxes, int64_t num_gt, const float* anchors, int64_t num_anchors,
                               float high_threshold, float low_threshold, int32_t allow_low_quality_matches, float wx, float wy,
                               float ww, float wh, int64_t* matches_out, float* matched_vals_out, float* targets_out,
                               void* workspace, size_t workspace_bytes, mb_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (num_gt < 1 || num_anchors < 0 || num_gt >= (1ll << 31) || num_anchors >= (1ll << 31)) return MB_ERR_INVALID_ARG;
    if (num_anchors == 0) return MB_OK;
    if (!gt_boxes || !anchors || !matches_out || !workspace) return MB_ERR_INVALID_ARG;
    if (workspace_bytes < mb_match_encode_workspace_bytes(num_gt, num_anchors)) return MB_ERR_WORKSPACE;
    Carver c(workspace, workspace_bytes);
    unsigned* gt_max = c.take<unsigned>((size_t)num_gt);
    int* gt_nan = c.take<int>((size_t)num_gt);
    float* best_val = c.take<float>((size_t)num_anchors);
    int* best_idx = c.take<int>((size_t)num_anchors);
    if (!c.ok()) return MB_ERR_WORKSPACE;
    MB_CUDA(cudaMemsetAsync(gt_max, 0, (size_t)((char*)best_val - (char*)gt_max), stream));
    const int grid = (int)ceil_div64(num_anchors, 256);
    k_match_best<<<grid, 256, 0, stream>>>((const float4*)gt_boxes, (int)num_gt, (const float4*)anchors, (int)num_anchors,
                                          best_val, best_idx, gt_max, gt_nan);
    MB_LAUNCH_CHECK();
    k_match_finish<<<grid, 256, 0, stream>>>((const float4*)gt_boxes, (int)num_gt, (const float4*)anchors, (int)num_anchors,
                                            high_threshold, low_threshold, allow_low_quality_matches, EncodeW{wx, wy, ww, wh},
                                            best_val, best_idx, gt_max, gt_nan, (long long*)matches_out, matched_vals_out,
                                            (float4*)targets_out);
    MB_LAUNCH_CHECK();
    return MB_OK;
}

extern "C" int mb_roi_align_backward(const float* grad, const float* rois, int64_t num_rois, float spatial_scale, int32_t channels,
                                     int32_t height, int32_t width, int32_t pooled_h, int32_t pooled_w, int32_t sampling_ratio,
                                     int32_t aligned, int32_t batch_size, float* grad_input, mb_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (num_rois < 0 || channels < 1 || height < 1 || width < 1 || pooled_h < 1 || pooled_w < 1 || batch_size < 1)
        return MB_ERR_INVALID_ARG;
    if (!grad_input) return MB_ERR_INVALID_ARG;
    MB_CUDA(cudaMemsetAsync(grad_input, 0, (size_t)batch_size * channels * height * width * sizeof(float), stream));
    if (num_rois == 0) return MB_OK;
    if (!grad || !rois) return MB_ERR_INVALID_ARG;
    const long long chunks = (channels + kBwdChunk - 1) / kBwdChunk;
    if (num_rois * chunks >= (1ll << 31)) return MB_ERR_UNSUPPORTED;
    const int patch_floats = kBwdChunk * 449;                 // footprints of up to 449 pixels per channel are staged
    const int smem = patch_floats * (int)sizeof(float);
    MB_DYN_SMEM(k_roi_align_backward, smem);
    k_roi_align_backward<<<(unsigned)(num_rois * chunks), kBwdThreads, smem, stream>>>(
        grad, rois, spatial_scale, channels, height, width, pooled_h, pooled_w, sampling_ratio, aligned, batch_size, grad_input,
        patch_floats);
    MB_LAUNCH_CHECK();
    return MB_OK;
}
