// morph.cu — per-crop particle measurements (morphometrics) from the instance masks of mb_crop_masks.
//
// The region of crop j is the set of non-zero bytes of its mask (h*w bytes at offsets[j] / channels, exactly the bytes
// k_crop_masks wrote), all set pixels as one region, pixels outside the crop rectangle outside it: regionprops of
// (mask > 0) with a single label. The record (MB_MORPH_FIELDS fp64, include/misob200.h) comes from exact int64 sums
// over the set pixels (A, S_r, S_c, S_rr, S_cc, S_rc, P_k) and the three counts n1, n2, n3 of regionprops' 4-connected
// perimeter codes; only the final record is floating point, so it is bit-identical for any launch shape.
//
//   k_mask_morphology  crops strided over blockIdx.x (the next crop's rect / src / offset prefetched), row bands of a
//                      crop over blockIdx.y. A band is <= kMorphBandPixels pixels of whole rows; its CTA packs the band's
//                      mask rows plus a 2-row halo into 32-bit words in shared memory (one ballot per 32 pixels) while
//                      it sums the moments and the pixel bytes of its own rows, derives erosion and border words of the
//                      band +- 1 row by shifts and funnel shifts, and counts the perimeter codes of its own rows with
//                      bit-sliced neighbour counts and popc. Sums meet by warp shuffles and shared memory, and the bands
//                      of a crop meet in the crop's workspace slot by 64-bit integer atomics: one image-sized crop is
//                      spread over many SMs and still gives the same bits.
//   k_mask_morphology_record  one thread per crop: the fp64 record from the slot's exact sums (the 128-bit and fp64
//                      arithmetic lives here, so it costs the band kernel no registers).
#include <math.h>

#include <algorithm>
#include "common.cuh"

namespace mb {

constexpr int kMorphThreads = 256;
constexpr int kMorphBandPixels = 16384;     // own pixels of one band at most (whole rows; a wider row is a band alone)
constexpr int kMorphBandRowsMax = 512;
constexpr int kMorphMaxSide = 32768;        // w, h <= 2^15: every int64 sum is exact (S_rr < 2^30 * 2^30)
constexpr int kMorphSums = 13;              // A, S_r, S_c, S_rr, S_cc, S_rc, P_0..P_3, n1, n2, n3
constexpr int kMorphSlotWords = 16;         // workspace per crop slot: the 13 sums + the band ticket, 128 bytes
// rows per band R = min(512, 16384 / w): R * ceil(w / 32) <= 1024 for every w <= 32768, so the mask words of a band
// and its halo ((R + 4) * ceil(w / 32)) and its border words ((R + 2) * ceil(w / 32)) fit these bounds
constexpr int kMorphWordsM = 1024 + 4 * (kMorphMaxSide / 32);
constexpr int kMorphWordsB = 1024 + 2 * (kMorphMaxSide / 32);
constexpr double kSqrt2 = 1.4142135623730951;               // sqrt(2.0), correctly rounded
constexpr double kPerimDiag = (1.0 + kSqrt2) / 2.0;
constexpr double kPi = 3.141592653589793;

struct MorphDev {
    int cap, ch;
    int img_w[MB_MAX_IMAGES];
    const unsigned char* img[MB_MAX_IMAGES];
};

__host__ __device__ __forceinline__ int morph_band_rows(int w) {
    const int r = kMorphBandPixels / (w > 0 ? w : 1);
    return r < 1 ? 1 : (r > kMorphBandRowsMax ? kMorphBandRowsMax : r);
}

// bit c of the result = bit c - 1 (shl1) / c + 1 (shr1) of the packed row, 0 beyond its ends
__device__ __forceinline__ unsigned shl1(const unsigned* row, int i) { return __funnelshift_l(i > 0 ? row[i - 1] : 0u, row[i], 1); }
__device__ __forceinline__ unsigned shr1(const unsigned* row, int i, int n) {
    return __funnelshift_r(row[i], i + 1 < n ? row[i + 1] : 0u, 1);
}

// per bit position, the number of set bits among a, b, c, d (0..4) as bits (s2 s1 s0)
__device__ __forceinline__ void add4(unsigned a, unsigned b, unsigned c, unsigned d, unsigned& s0, unsigned& s1, unsigned& s2) {
    const unsigned x = a ^ b, y = c ^ d, ca = a & b, cb = c & d;
    s0 = x ^ y;
    s1 = ca ^ cb ^ (x & y);            // ca, cb and x & y: never two of them without ca & cb
    s2 = ca & cb;
}

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// the record from the exact sums s[kMorphSums] of a crop at rect origin (x, y); the formulas are the ABI's
__device__ __forceinline__ void morph_record(const long long* s, int x, int y, int ch, double* __restrict__ o) {
    double f[MB_MORPH_FIELDS];
#pragma unroll
    for (int k = 0; k < MB_MORPH_FIELDS; ++k) f[k] = 0.0;
    const long long A = s[0];
    if (A > 0) {
        const double da = (double)A;
        f[0] = da;
        f[1] = ((double)s[10] + kSqrt2 * (double)s[11]) + kPerimDiag * (double)s[12];
        f[2] = (double)x + (double)s[2] / da;
        f[3] = (double)y + (double)s[1] / da;
        const __int128 a128 = A;
        const double a2 = da * da;
        const double urr = (double)(a128 * s[3] - (__int128)s[1] * s[1]) / a2;
        const double ucc = (double)(a128 * s[4] - (__int128)s[2] * s[2]) / a2;
        const double urc = (double)(a128 * s[5] - (__int128)s[1] * s[2]) / a2;
        const double a = ucc, b = -urc, c = urr;
        const double root = sqrt((a - c) * (a - c) + 4.0 * (b * b));
        double l1 = ((a + c) + root) / 2.0, l2 = ((a + c) - root) / 2.0;
        l1 = l1 > 0.0 ? l1 : 0.0;
        l2 = l2 > 0.0 ? l2 : 0.0;
        f[4] = 4.0 * sqrt(l1);
        f[5] = 4.0 * sqrt(l2);
        f[6] = a == c ? (b < 0.0 ? -kPi / 4.0 : kPi / 4.0) : 0.5 * atan2(-2.0 * b, c - a);
        f[7] = l1 == 0.0 ? 0.0 : sqrt(1.0 - l2 / l1);
        f[8] = sqrt((double)(4 * A) / kPi);
#pragma unroll
        for (int k = 0; k < 4; ++k) f[9 + k] = k < ch ? (double)s[6 + k] / da : 0.0;
    }
#pragma unroll
    for (int k = 0; k < MB_MORPH_FIELDS; ++k) o[k] = f[k];
}

// offsets are in pixel bytes (h * w * ch per crop); the mask bytes of a crop start at offset / ch. ch <= 4: no 64-bit
// division by a variable
__device__ __forceinline__ long long div_ch(long long v, int ch) { return ch == 3 ? v / 3 : v >> (ch >> 1); }

__global__ void __launch_bounds__(kMorphThreads, 6) k_mask_morphology(const MorphDev d, const unsigned char* __restrict__ masks,
                                                                   const int4* __restrict__ rects, const int* __restrict__ src,
                                                                   const long long* __restrict__ offsets,
                                                                   const long long* __restrict__ totals,
                                                                   unsigned long long* __restrict__ ws) {
    __shared__ unsigned sM[kMorphWordsM];     // mask words, crop rows lo - 2 .. hi + 1
    __shared__ unsigned sB[kMorphWordsB];     // border words (mask and not eroded), crop rows lo - 1 .. hi
    __shared__ long long sRed[kMorphThreads / 32][kMorphSums];
    __shared__ long long sTot[kMorphSums];
    if (totals[3] != 0) return;               // the masks were not written (mask buffer overflow)
    const int ncrops = (int)totals[0];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int nwarps = kMorphThreads / 32;
    const int ch = d.ch;
    int4 rc_next = make_int4(0, 0, 0, 0);
    int src_next = 0;
    long long off_next = 0;
    if ((int)blockIdx.x < ncrops) { rc_next = rects[blockIdx.x]; src_next = src[blockIdx.x]; off_next = offsets[blockIdx.x]; }
    for (int j = blockIdx.x; j < ncrops; j += gridDim.x) {
        const int4 rc = rc_next;
        const int n = src_next / d.cap;
        const unsigned char* mk = masks + div_ch(off_next, ch);
        const int jn = j + gridDim.x;
        if (jn < ncrops) { rc_next = rects[jn]; src_next = src[jn]; off_next = offsets[jn]; }
        const int w = rc.z, h = rc.w;
        const int R = morph_band_rows(w);
        const int nb = h > R ? (h + R - 1) / R : 1;
        if ((int)blockIdx.y >= nb) continue;
        const int W32 = (w + 31) >> 5;
        const unsigned char* im = d.img[n];
        const int iw = d.img_w[n];
        unsigned long long* slot = ws + (size_t)j * kMorphSlotWords;
        for (int band = blockIdx.y; band < nb; band += gridDim.y) {
            const int lo = band * R, hi = min(h, lo + R), rows = hi - lo;
            // band-local row rl = r - lo: with w * R <= 16384 every sum but S_cc fits 32 bits
            int A = 0, Srl = 0, Sc = 0, Srrl = 0, Srcl = 0, P0 = 0, P1 = 0, P2 = 0, P3 = 0;
            long long Scc = 0;
            __syncthreads();                                   // the previous band's words and sums are no longer read
            // mask rows lo - 2 .. hi + 1 -> words (zero outside the crop); moments and pixel bytes of rows lo .. hi - 1
            for (int t = warp; t < rows + 4; t += nwarps) {
                const int r = lo - 2 + t, rl = t - 2;
                unsigned* mw = sM + t * W32;
                if (r < 0 || r >= h) {
                    for (int i = lane; i < W32; i += 32) mw[i] = 0u;
                    continue;
                }
                const unsigned char* mrow = mk + (size_t)r * w;
                const bool own = r >= lo && r < hi;
                const unsigned char* prow = im + ((size_t)(rc.y + r) * iw + rc.x) * ch;
                for (int i = 0; i < W32; ++i) {
                    const int c = 32 * i + lane;
                    const bool set = c < w && __ldg(mrow + c) != 0;
                    const unsigned word = __ballot_sync(0xffffffffu, set);
                    if (lane == 0) mw[i] = word;
                    if (own && set) {
                        ++A; Srl += rl; Srrl += rl * rl; Sc += c; Srcl += rl * c; Scc += (long long)c * c;
                        const unsigned char* px = prow + c * ch;
                        P0 += __ldg(px);
                        if (ch > 1) P1 += __ldg(px + 1);
                        if (ch > 2) P2 += __ldg(px + 2);
                        if (ch > 3) P3 += __ldg(px + 3);
                    }
                }
            }
            {
                const long long v[10] = {warp_sum(A), warp_sum(Srl), warp_sum(Sc), warp_sum(Srrl), warp_sum(Scc), warp_sum(Srcl),
                                         warp_sum(P0), warp_sum(P1), warp_sum(P2), warp_sum(P3)};
                if (lane == 0) {
#pragma unroll
                    for (int k = 0; k < 10; ++k) sRed[warp][k] = v[k];
                }
            }
            __syncthreads();
            // border = mask and not eroded (4-cross erosion, outside = 0), rows lo - 1 .. hi
            for (int q = tid; q < (rows + 2) * W32; q += kMorphThreads) {
                const int t = q / W32, i = q - t * W32;
                const unsigned* m = sM + (t + 1) * W32;
                const unsigned mc = m[i];
                const unsigned e = mc & sM[t * W32 + i] & sM[(t + 2) * W32 + i] & shl1(m, i) & shr1(m, i, W32);
                sB[q] = mc & ~e;
            }
            __syncthreads();
            // perimeter codes of the border pixels of rows lo .. hi - 1: code = 1 + 2 * n4 + 10 * nd
            int n1 = 0, n2 = 0, n3 = 0;
            for (int q = tid; q < rows * W32; q += kMorphThreads) {
                const int t = q / W32, i = q - t * W32;
                const unsigned* bm = sB + (t + 1) * W32;
                const unsigned bc = bm[i];
                if (bc == 0u) continue;
                const unsigned* bu = sB + t * W32;
                const unsigned* bd = sB + (t + 2) * W32;
                unsigned f0, f1, f2, g0, g1, g2;
                add4(shl1(bm, i), shr1(bm, i, W32), bu[i], bd[i], f0, f1, f2);                              // n4
                add4(shl1(bu, i), shr1(bu, i, W32), shl1(bd, i), shr1(bd, i, W32), g0, g1, g2);              // nd
                const unsigned one4 = f0 & ~f1;                                                             // n4 == 1
                n1 += __popc(bc & f1 & ~((g0 & g1) | g2));                  // n4 in {2, 3}, nd <= 2: 5 7 15 17 25 27
                n2 += __popc(bc & ((~(f0 | f1 | f2) & ~g0 & g1) | (one4 & g0 & g1)));   // (0, 2), (1, 3): 21 33
                n3 += __popc(bc & one4 & (g0 ^ g1));                       // n4 == 1, nd in {1, 2}: 13 23
            }
            n1 = warp_sum(n1); n2 = warp_sum(n2); n3 = warp_sum(n3);
            if (lane == 0) { sRed[warp][10] = n1; sRed[warp][11] = n2; sRed[warp][12] = n3; }
            __syncthreads();
            if (tid < kMorphSums) {
                long long t = 0;
#pragma unroll
                for (int q = 0; q < nwarps; ++q) t += sRed[q][tid];
                sTot[tid] = t;
            }
            __syncthreads();
            // band-local rows -> crop rows (r = lo + rl); integer sums are order-free, so the bands of a crop meet in
            // 64-bit atomics in any order and the record kernel reads exact totals
            if (tid < kMorphSums) {
                const long long L = lo;
                long long v = sTot[tid];
                if (tid == 1) v += L * sTot[0];
                if (tid == 3) v += L * L * sTot[0] + 2 * L * sTot[1];
                if (tid == 5) v += L * sTot[2];
                if (v != 0) atomicAdd(slot + tid, (unsigned long long)v);
            }
        }
    }
}

// one thread per crop: the record from the crop's exact sums
__global__ void __launch_bounds__(256) k_mask_morphology_record(const int4* __restrict__ rects, const long long* __restrict__ totals,
                                                                const long long* __restrict__ ws, int ch, double* __restrict__ out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (totals[3] != 0 || j >= totals[0]) return;
    const int4 rc = rects[j];
    long long s[kMorphSums];
#pragma unroll
    for (int k = 0; k < kMorphSums; ++k) s[k] = ws[(size_t)j * kMorphSlotWords + k];
    morph_record(s, rc.x, rc.y, ch, out + (size_t)j * MB_MORPH_FIELDS);
}

}  // namespace mb

extern "C" size_t mb_mask_morphology_workspace_bytes(const mb_crop_params* p) {
    if (!p || p->num_images < 1 || p->capacity < 1) return 0;
    return (size_t)p->num_images * (size_t)p->capacity * mb::kMorphSlotWords * sizeof(unsigned long long);
}

extern "C" int mb_mask_morphology(const mb_crop_params* p, const uint8_t* masks, const int32_t* rects, const int32_t* src,
                                  const int64_t* offsets, const int64_t* totals, void* workspace, size_t workspace_bytes,
                                  double* out, mb_stream_t stream) {
    if (!p || !masks || !rects || !src || !offsets || !totals || !out) return MB_ERR_INVALID_ARG;
    if (p->num_images < 1 || p->num_images > MB_MAX_IMAGES || p->capacity < 1 || p->channels < 1) return MB_ERR_INVALID_ARG;
    if (p->channels > 4) return MB_ERR_UNSUPPORTED;
    mb::MorphDev d;
    d.cap = p->capacity; d.ch = p->channels;
    for (int n = 0; n < MB_MAX_IMAGES; ++n) {
        const bool used = n < p->num_images;
        if (used && (p->image_h[n] < 0 || p->image_w[n] < 0 || !p->images[n])) return MB_ERR_INVALID_ARG;
        if (used && (p->image_h[n] > mb::kMorphMaxSide || p->image_w[n] > mb::kMorphMaxSide)) return MB_ERR_UNSUPPORTED;
        d.img_w[n] = used ? p->image_w[n] : 0; d.img[n] = used ? p->images[n] : nullptr;
    }
    const size_t need = mb_mask_morphology_workspace_bytes(p);
    if (!workspace || workspace_bytes < need) return MB_ERR_WORKSPACE;
    MB_CUDA(cudaMemsetAsync(workspace, 0, need, (cudaStream_t)stream));
    // crops over x; bands of a crop over y while few crop slots leave the GPU idle (a CTA that finds its crop has no
    // band for it only pays for reading the rectangle)
    const long long slots = (long long)p->num_images * p->capacity;
    const long long fill = (long long)mb::num_sms() * 8;
    const int gx = (int)std::min<long long>(slots, fill);
    const int gy = (int)std::max<long long>(1, fill / slots);
    mb::k_mask_morphology<<<dim3(gx, gy), mb::kMorphThreads, 0, (cudaStream_t)stream>>>(
        d, masks, reinterpret_cast<const int4*>(rects), src, (const long long*)offsets, (const long long*)totals,
        (unsigned long long*)workspace);
    MB_LAUNCH_CHECK();
    mb::k_mask_morphology_record<<<(int)mb::ceil_div64(slots, 256), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const int4*>(rects), (const long long*)totals, (const long long*)workspace, d.ch, out);
    MB_LAUNCH_CHECK();
    return MB_OK;
}
