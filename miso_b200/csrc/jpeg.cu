// jpeg.cu — baseline JPEG files of the packed crops of the crop stage, one complete file per crop, byte for byte the
// file PIL (libjpeg-turbo) writes with default settings.
//
// The bytes are stated in include/misob200.h (mb_jpeg_encode) and restated on the CPU in tests/jpeg_ref.py.
//   k_jpeg_plan      one CTA: per crop its blocks in scan order (dummy blocks included) and its first block; the
//                    workspace fit of the block records
//   k_jpeg_blocks    8 threads per 8x8 block: samples read from the packed crop with the edge padding, colour
//                    conversion and h2v2 done on the fly; islow DCT (rows, then columns through shared memory);
//                    quantised DC and the bit length of the AC codes
//   k_jpeg_bits      one thread per block: the DC difference against the predecessor in scan order (dummy blocks take
//                    the DC of the block before them in their MCU), the block's bits; exclusive scan per tile of 1024
//   k_jpeg_scan      one CTA: tile bases (64-bit), per crop its data bits, chunks (kJpgChunk unstuffed bytes each) and
//                    the slot of its unstuffed stream, sized exactly; the workspace fit of the chunks and streams
//   k_jpeg_pack      8 threads per block: the coefficients again, the codes OR-ed into a shared-memory staging of the
//                    block's words; plain stores of the words whose first bit is the block's, the partial first word
//                    (owned by an earlier block) to the block record
//   k_jpeg_seam      one thread per block: the first non-owner of a word ORs its and the following blocks' partial
//                    words into it (one writer per word, no atomics)
//   k_jpeg_count     one warp per chunk: its 0xFF bytes
//   k_jpeg_layout    one CTA: chunk 0xFF prefixes, per crop header + data + stuffing + EOI, the output offsets, total and
//                    overflow flag, before anything is written
//   k_jpeg_assemble  one warp per chunk: the stuffing copy (32 words per round, warp scan of the 0xFF counts); a crop's
//                    first chunk writes the header (tables built once per CTA, h and w patched into SOF0), its last
//                    chunk the EOI
// The encoder recomputes the coefficients in k_jpeg_pack instead of storing them: 16 B of block record per block
// instead of 144 B.
#include <algorithm>

#include "common.cuh"

namespace mb {

constexpr int kJpgBlockBits = 22 + 63 * 26;                 // DC <= 11 + 11 bits, each AC <= 16 + 10
constexpr int kJpgBlockBytes = 208;                         // ceil(kJpgBlockBits / 8), a multiple of 4
constexpr int kJpgStageWords = 56;                          // staging of one block: 31 + kJpgBlockBits + 7 bits
constexpr int kJpgTile = 1024;                              // blocks per bit-offset tile
constexpr int kJpgChunk = 4096;                             // unstuffed bytes per chunk
constexpr int kJpgBlocksPerCta = 32;                        // k_jpeg_blocks / k_jpeg_pack: 8 threads per block
constexpr int kJpgHeadGray = 328, kJpgHeadColor = 623;      // SOI .. SOS
constexpr int kJpgHead = 16;                                // int64 header words of the workspace
static_assert(kJpgBlockBytes * 8 >= kJpgBlockBits && kJpgBlockBytes % 4 == 0, "block slot");
static_assert(kJpgStageWords * 32 >= 31 + kJpgBlockBits + 7, "block staging");

__device__ __constant__ unsigned char kZigzag[64] = {
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
    35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55,
    62, 63};
__device__ __constant__ unsigned char kStdQuant[2][64] = {
    {16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56, 14, 17, 22, 29, 51,
     87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92, 49, 64, 78, 87, 103, 121, 120, 101,
     72, 92, 95, 98, 112, 100, 103, 99},
    {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99, 99,
     99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
     99, 99, 99, 99, 99, 99}};
__device__ __constant__ unsigned char kDcBits[2][16] = {{0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0},
                                                        {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0}};
__device__ __constant__ unsigned char kAcBits[2][16] = {{0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d},
                                                        {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77}};
__device__ __constant__ unsigned char kAcVals[2][162] = {
    {0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14,
     0x32, 0x81, 0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09,
     0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a,
     0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65,
     0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88,
     0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9,
     0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca,
     0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea,
     0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa},
    {0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32,
     0x81, 0x08, 0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16,
     0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39,
     0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64,
     0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x82, 0x83, 0x84, 0x85, 0x86,
     0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7,
     0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8,
     0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9,
     0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa}};

__host__ __device__ inline int quant75(int std) { return min(255, max(1, (std * 50 + 50) / 100)); }

// Per-CTA tables: quantisers (natural order), zigzag position of each natural index, codes as (code << 8) | length
struct JpgTables {
    int quant[2][64];
    unsigned char zz_of[64];
    unsigned dc[2][12];
    unsigned ac[2][256];
};

__device__ void build_tables(JpgTables& t) {
    for (int i = threadIdx.x; i < 128; i += blockDim.x) t.quant[i >> 6][i & 63] = quant75(kStdQuant[i >> 6][i & 63]);
    for (int i = threadIdx.x; i < 64; i += blockDim.x) t.zz_of[kZigzag[i]] = (unsigned char)i;
    if (threadIdx.x < 4) {
        const int k = threadIdx.x & 1, ac = threadIdx.x >> 1;
        const unsigned char* bits = ac ? kAcBits[k] : kDcBits[k];
        unsigned code = 0;
        int n = 0;
        for (int len = 1; len <= 16; ++len) {
            for (int i = 0; i < bits[len - 1]; ++i, ++n, ++code) {
                const unsigned e = (code << 8) | (unsigned)len;
                if (ac) t.ac[k][kAcVals[k][n]] = e; else t.dc[k][n] = e;
            }
            code <<= 1;
        }
    }
    __syncthreads();
}

struct JpgArgs {
    const unsigned char* packed;
    const int4* rects;
    const long long* offsets;
    int src_ch, ch;
};

struct JpgRec {
    short dc, diff;      // quantised DC (k_jpeg_blocks), DC difference (k_jpeg_bits)
    unsigned off;        // bit offset within the tile (k_jpeg_bits); the AC bits before that
    unsigned edge;       // the block's bits in a first word it does not own, big-endian (k_jpeg_pack)
    unsigned pad;
};

struct JpgWs {
    long long* head;     // [kJpgHead]: 0 blocks, 1 crops, 2 workspace too small, 3 tiles, 4 chunks, 5.. offsets below
    long long* first;    // [S + 1] first block of crop j
    long long* slot;     // [S] byte offset of crop j's unstuffed stream in the slot area
    long long* cfirst;   // [S + 1] first chunk of crop j (k_jpeg_scan)
    long long* dbits;    // [S] data bits of crop j (k_jpeg_scan)
    JpgRec* recs;        // [blocks]
    long long* tiles;    // [tiles + 1] bit base of each tile, then the total
    long long* cnt;      // [chunks + 1] 0xFF bytes per chunk, then their exclusive prefix
    unsigned char* slots;
};

__host__ __device__ inline long long jpg_fixed_bytes(long long S) { return 8 * (kJpgHead + 4 * S + 2); }

__device__ inline JpgWs jpg_ws(void* ws, long long S) {
    JpgWs w;
    unsigned char* b = (unsigned char*)ws;
    w.head = (long long*)b;
    w.first = w.head + kJpgHead;
    w.slot = w.first + (S + 1);
    w.cfirst = w.slot + S;
    w.dbits = w.cfirst + (S + 1);
    w.recs = (JpgRec*)(b + w.head[5]);
    w.tiles = (long long*)(b + w.head[6]);
    w.cnt = (long long*)(b + w.head[7]);
    w.slots = b + w.head[8];
    return w;
}

__device__ inline long long jpg_blocks(int h, int w, int c) {
    if (h <= 0 || w <= 0) return 0;
    return c == 1 ? (long long)((h + 7) >> 3) * ((w + 7) >> 3) : 6ll * ((h + 15) >> 4) * ((w + 15) >> 4);
}

// Position of block q of a crop in scan order: component, block column / row in that component, dummy (jccoefct.c)
struct BlkPos {
    int comp, bx, by;
    bool dummy;
};
__device__ inline BlkPos blk_pos(int h, int w, int c, long long q) {
    if (c == 1) {
        const int nbx = (w + 7) >> 3;
        return {0, (int)(q % nbx), (int)(q / nbx), false};
    }
    const long long m = q / 6;
    const int k = (int)(q - 6 * m), mw = (w + 15) >> 4;
    const int mx = (int)(m % mw), my = (int)(m / mw);
    if (k >= 4) return {k - 3, mx, my, false};
    const int bx = 2 * mx + (k & 1), by = 2 * my + (k >> 1);
    return {0, bx, by, bx >= ((w + 7) >> 3) || by >= ((h + 7) >> 3)};
}

// long long exclusive scan over the CTA (blockDim a multiple of 32, at most 1024)
__device__ inline long long jpg_excl_scan(long long v, long long* sm, long long* total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    long long x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) sm[wid] = x;
    __syncthreads();
    long long pre = 0, all = 0;
    for (int q = 0; q < nw; ++q) {
        if (q < wid) pre += sm[q];
        all += sm[q];
    }
    __syncthreads();
    if (total) *total = all;
    return pre + x - v;
}

// first index i in [0, n) with a[i + 1] > v, for a non-decreasing a[0..n]: the crop of block / chunk v
__device__ inline long long owner_of(const long long* a, long long n, long long v) {
    long long lo = 0, hi = n;
    while (hi - lo > 1) {
        const long long mid = (lo + hi) >> 1;
        if (a[mid] <= v) lo = mid; else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(1024) k_jpeg_plan(JpgArgs a, const long long* __restrict__ totals, void* ws, size_t ws_bytes,
                                                   long long S) {
    __shared__ long long sm[32];
    __shared__ long long s_blk;
    long long* head = (long long*)ws;
    long long* first = head + kJpgHead;
    const long long ncrops = totals[2] ? 0 : totals[0];
    if (threadIdx.x == 0) s_blk = 0;
    __syncthreads();
    for (long long j0 = 0; j0 < ncrops; j0 += blockDim.x) {
        const long long j = j0 + threadIdx.x;
        long long nb = 0;
        if (j < ncrops) {
            const int4 rc = a.rects[j];
            nb = jpg_blocks(rc.w, rc.z, a.ch);
        }
        long long tb;
        const long long eb = jpg_excl_scan(nb, sm, &tb);
        if (j < ncrops) first[j] = s_blk + eb;
        __syncthreads();
        if (threadIdx.x == 0) s_blk += tb;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        // block records and tiles now; the chunk counts and the streams once k_jpeg_scan knows their sizes
        const long long nblk = s_blk, ntile = (nblk + kJpgTile - 1) / kJpgTile;
        const long long recs = (jpg_fixed_bytes(S) + 15) / 16 * 16;
        const long long tiles = recs + nblk * (long long)sizeof(JpgRec);
        const long long cnt = tiles + 8 * (ntile + 1);
        const bool fits = cnt + 8 <= (long long)ws_bytes;
        // too small: nothing is encoded, and the two words written before the layout (tiles[0], cnt[0]) stay inside
        first[fits ? ncrops : 0] = fits ? nblk : 0;
        head[0] = fits ? nblk : 0;
        head[1] = fits ? ncrops : 0;
        head[2] = fits ? 0 : 1;
        head[3] = fits ? ntile : 0;
        head[4] = 0;
        head[5] = recs; head[6] = fits ? tiles : recs; head[7] = fits ? cnt : recs + 16; head[8] = head[7];
    }
}

// ---- the coefficients of one block (8 threads: lane r = row r, then column r) ----------------------------------------
__device__ inline int descale(int x, int n) { return (x + (1 << (n - 1))) >> n; }

// jfdctint.c, one 1-D pass over d[8]; first: the row pass (outputs scaled up by PASS1_BITS)
__device__ inline void fdct8(int* d, bool first) {
    constexpr int C = 13, P = 2;
    const int t0 = d[0] + d[7], t7 = d[0] - d[7], t1 = d[1] + d[6], t6 = d[1] - d[6];
    const int t2 = d[2] + d[5], t5 = d[2] - d[5], t3 = d[3] + d[4], t4 = d[3] - d[4];
    const int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    const int sh = first ? C - P : C + P;
    d[0] = first ? (t10 + t11) << P : descale(t10 + t11, P);
    d[4] = first ? (t10 - t11) << P : descale(t10 - t11, P);
    int z1 = (t12 + t13) * 4433;                                    // FIX(0.541196100)
    d[2] = descale(z1 + t13 * 6270, sh);                            // FIX(0.765366865)
    d[6] = descale(z1 - t12 * 15137, sh);                           // FIX(1.847759065)
    z1 = t4 + t7;
    int z2 = t5 + t6, z3 = t4 + t6, z4 = t5 + t7;
    const int z5 = (z3 + z4) * 9633;                                // FIX(1.175875602)
    const int a4 = t4 * 2446, a5 = t5 * 16819, a6 = t6 * 25172, a7 = t7 * 12299;   // 0.298631336 2.053119869 3.072711026 1.501321110
    z1 *= -7373; z2 *= -20995;                                      // 0.899976223 2.562915447
    z3 = z3 * -16069 + z5; z4 = z4 * -3196 + z5;                    // 1.961570560 0.390180644
    d[7] = descale(a4 + z1 + z3, sh);
    d[5] = descale(a5 + z2 + z4, sh);
    d[3] = descale(a6 + z2 + z3, sh);
    d[1] = descale(a7 + z1 + z4, sh);
}

__device__ inline int luma(const unsigned char* p) {
    return (19595 * p[0] + 38470 * p[1] + 7471 * p[2] + 32768) >> 16;
}
__device__ inline int chroma(const unsigned char* p, int comp) {
    return comp == 1 ? (-11059 * p[0] - 21709 * p[1] + 32768 * p[2] + (128 << 16) + 32767) >> 16
                     : (32768 * p[0] - 27439 * p[1] - 5329 * p[2] + (128 << 16) + 32767) >> 16;
}

// Quantised coefficients of the block, zigzag order, into zz[64] (shared, the 8 lanes of the block's group).
// tr: 64 ints of shared scratch. All 32 lanes of the warp call it (it syncs the warp).
__device__ void block_coefs(const JpgTables& t, const unsigned char* src, int h, int w, int c, const BlkPos& p, int r,
                            int* tr, int* zz, bool live) {
    int d[8];
    if (live) {
        if (p.comp == 0) {
            const unsigned char* row = src + (long long)min(p.by * 8 + r, h - 1) * w * c;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const unsigned char* px = row + (long long)min(p.bx * 8 + k, w - 1) * c;
                d[k] = (c == 1 ? (int)px[0] : luma(px)) - 128;
            }
        } else {
            const int cy = min(p.by * 8 + r, ((h + 1) >> 1) - 1);
            const unsigned char* r0 = src + (long long)min(2 * cy, h - 1) * w * 3;
            const unsigned char* r1 = src + (long long)min(2 * cy + 1, h - 1) * w * 3;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int cx = p.bx * 8 + k;
                const long long x0 = (long long)min(2 * cx, w - 1) * 3, x1 = (long long)min(2 * cx + 1, w - 1) * 3;
                const int s = chroma(r0 + x0, p.comp) + chroma(r0 + x1, p.comp) + chroma(r1 + x0, p.comp) +
                              chroma(r1 + x1, p.comp);
                d[k] = ((s + 1 + (k & 1)) >> 2) - 128;
            }
        }
        fdct8(d, true);
#pragma unroll
        for (int k = 0; k < 8; ++k) tr[r * 8 + k] = d[k];
    }
    __syncwarp();
    if (live) {
#pragma unroll
        for (int v = 0; v < 8; ++v) d[v] = tr[v * 8 + r];
        fdct8(d, false);
        const int* q = t.quant[p.comp ? 1 : 0];
#pragma unroll
        for (int v = 0; v < 8; ++v) {
            const int dv = q[v * 8 + r] << 3, a = abs(d[v]);
            const int m = (a + (dv >> 1)) / dv;
            zz[t.zz_of[v * 8 + r]] = d[v] < 0 ? -m : m;
        }
    }
    __syncwarp();
}

__device__ inline int category(int v) { return v ? 32 - __clz(abs(v)) : 0; }

// Nonzero AC positions of the block as a 64-bit mask (bit k = zigzag position k), from the 8 lanes' values zz[8r..8r+7]
__device__ inline unsigned long long ac_mask(const int* zz, int r) {
    unsigned long long m = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) m |= (unsigned long long)(zz[8 * r + i] != 0) << (8 * r + i);
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) m |= __shfl_xor_sync(0xffffffffu, m, o);
    return m & ~1ull;
}

// Calls f(value, bits) for every AC code of the lane's positions 8r..8r+7, in order (ZRLs, code | amplitude), then
// (lane 7) the EOB when the last nonzero position is below 63.
template <typename F>
__device__ inline void ac_codes(const JpgTables& t, const int* zz, int r, int tab, unsigned long long mask, F f) {
    const unsigned zrl = t.ac[tab][0xF0];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int k = 8 * r + i, v = zz[k];
        if (k == 0 || v == 0) continue;
        const unsigned long long below = mask & ((1ull << k) - 1);
        const int prev = below ? 63 - __clzll((long long)below) : 0;
        int run = k - prev - 1;
        for (; run > 15; run -= 16) f(zrl >> 8, (int)(zrl & 255));
        const int n = category(v);
        const unsigned e = t.ac[tab][(run << 4) | n];
        const unsigned amp = (unsigned)(v < 0 ? v + (1 << n) - 1 : v) & ((1u << n) - 1);
        f(((e >> 8) << n) | amp, (int)(e & 255) + n);
    }
    if (r == 7 && (mask >> 63) == 0) {
        const unsigned eob = t.ac[tab][0];
        f(eob >> 8, (int)(eob & 255));
    }
}

struct BlkSmem {
    JpgTables t;
    int tr[kJpgBlocksPerCta][64];
    int zz[kJpgBlocksPerCta][64];
    unsigned stage[kJpgBlocksPerCta][kJpgStageWords];
};

__global__ void __launch_bounds__(256) k_jpeg_blocks(JpgArgs a, void* ws, long long S) {
    __shared__ BlkSmem sm;
    build_tables(sm.t);
    JpgWs w = jpg_ws(ws, S);
    const long long nblk = w.head[0], ncrops = w.head[1];
    const int g = threadIdx.x >> 3, r = threadIdx.x & 7;
    for (long long b0 = (long long)blockIdx.x * kJpgBlocksPerCta; b0 < nblk; b0 += (long long)gridDim.x * kJpgBlocksPerCta) {
        const long long b = b0 + g;
        const bool live = b < nblk;
        long long j = 0;
        if (live && r == 0) j = owner_of(w.first, ncrops, b);
        j = __shfl_sync(0xffffffffu, j, threadIdx.x & 24);
        int4 rc = make_int4(0, 0, 1, 1);
        BlkPos p = {0, 0, 0, true};
        if (live) { rc = a.rects[j]; p = blk_pos(rc.w, rc.z, a.ch, b - w.first[j]); }
        const unsigned char* src = a.packed + (live ? a.offsets[j] / a.src_ch * a.ch : 0);
        const bool real = live && !p.dummy;
        block_coefs(sm.t, src, rc.w, rc.z, a.ch, p, r, sm.tr[g], sm.zz[g], real);
        const unsigned long long mask = ac_mask(sm.zz[g], r);      // every lane of the warp takes part in the shuffles
        int bits = 0;
        if (real) ac_codes(sm.t, sm.zz[g], r, p.comp ? 1 : 0, mask, [&](unsigned, int n) { bits += n; });
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) bits += __shfl_xor_sync(0xffffffffu, bits, o);
        if (live && r == 0) {
            w.recs[b].dc = real ? (short)sm.zz[g][0] : 0;
            w.recs[b].off = real ? (unsigned)bits : sm.t.ac[0][0] & 255;           // a dummy block: zero AC, the EOB only
        }
        __syncwarp();
    }
}

// the block whose DC a block of the crop codes (a dummy block: the nearest real block before it in its MCU)
__device__ inline long long dc_source(int h, int w, int c, long long q) {
    while (c == 3 && blk_pos(h, w, c, q).dummy) --q;                // Y0 of an MCU is never a dummy
    return q;
}
// the previous block of the same component in scan order, or -1
__device__ inline long long dc_pred(int c, long long q) {
    if (c == 1) return q - 1;
    const long long m = q / 6;
    const int k = (int)(q - 6 * m);
    if (k >= 1 && k <= 3) return q - 1;
    if (m == 0) return -1;
    return k == 0 ? q - 3 : q - 6;
}

__global__ void __launch_bounds__(kJpgTile) k_jpeg_bits(JpgArgs a, void* ws, long long S) {
    __shared__ long long sm[32];
    __shared__ unsigned s_dc[2][12];
    JpgWs w = jpg_ws(ws, S);
    const long long nblk = w.head[0], ncrops = w.head[1], ntile = w.head[3];
    if (threadIdx.x < 2) {
        unsigned code = 0;
        int n = 0;
        for (int len = 1; len <= 16; ++len) {
            for (int i = 0; i < kDcBits[threadIdx.x][len - 1]; ++i, ++n, ++code) s_dc[threadIdx.x][n] = (code << 8) | len;
            code <<= 1;
        }
    }
    __syncthreads();
    for (long long t = blockIdx.x; t < ntile; t += gridDim.x) {
        const long long b = t * kJpgTile + threadIdx.x;
        long long bits = 0;
        if (b < nblk) {
            const long long j = owner_of(w.first, ncrops, b), f = w.first[j];
            const int4 rc = a.rects[j];
            const long long q = b - f;
            const int comp = a.ch == 1 ? 0 : (q % 6 < 4 ? 0 : (int)(q % 6) - 3);
            const long long pq = dc_pred(a.ch, q);
            const int dc = w.recs[f + dc_source(rc.w, rc.z, a.ch, q)].dc;
            const int pdc = pq < 0 ? 0 : w.recs[f + dc_source(rc.w, rc.z, a.ch, pq)].dc;
            const int diff = dc - pdc, n = category(diff);
            bits = (long long)w.recs[b].off + (s_dc[comp ? 1 : 0][n] & 255) + n;
            w.recs[b].diff = (short)diff;
        }
        long long tot;
        const long long ex = jpg_excl_scan(bits, sm, &tot);
        if (b < nblk) w.recs[b].off = (unsigned)ex;
        if (threadIdx.x == 0) w.tiles[t] = tot;
    }
}

__global__ void __launch_bounds__(1024) k_jpeg_scan(void* ws, size_t ws_bytes, long long S) {
    __shared__ long long sm[32];
    __shared__ long long s_base, s_slot;
    JpgWs w = jpg_ws(ws, S);
    const long long nblk = w.head[0], ncrops = w.head[1], ntile = w.head[3];
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (long long t0 = 0; t0 < ntile; t0 += blockDim.x) {
        const long long t = t0 + threadIdx.x;
        long long tot;
        const long long ex = jpg_excl_scan(t < ntile ? w.tiles[t] : 0, sm, &tot);
        if (t < ntile) w.tiles[t] = s_base + ex;
        __syncthreads();
        if (threadIdx.x == 0) s_base += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) { w.tiles[ntile] = s_base; s_base = 0; s_slot = 0; }
    __syncthreads();
    // k_jpeg_bits' block records hold blocks' bits to the tiles, so a block's bit offset is tiles[b / T] + off
    auto G = [&](long long b) { return b < nblk ? w.tiles[b / kJpgTile] + w.recs[b].off : w.tiles[ntile]; };
    for (long long j0 = 0; j0 < ncrops; j0 += blockDim.x) {
        const long long j = j0 + threadIdx.x;
        long long nc = 0, sb = 0;
        if (j < ncrops) {
            const long long d = G(w.first[j + 1]) - G(w.first[j]);
            w.dbits[j] = d;
            nc = ((d + 7) / 8 + kJpgChunk - 1) / kJpgChunk;
            sb = ((d + 7) / 8 + 15) / 16 * 16;
        }
        long long tot, tots;
        const long long ex = jpg_excl_scan(nc, sm, &tot);
        const long long es = jpg_excl_scan(sb, sm, &tots);
        if (j < ncrops) { w.cfirst[j] = s_base + ex; w.slot[j] = s_slot + es; }
        __syncthreads();
        if (threadIdx.x == 0) { s_base += tot; s_slot += tots; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        // the chunk counts after the tiles, then the unstuffed streams; too small: nothing is encoded
        const long long slots = (w.head[7] + 8 * (s_base + 1) + 15) / 16 * 16;
        const bool fits = !w.head[2] && slots + s_slot <= (long long)ws_bytes;
        w.cfirst[fits ? ncrops : 0] = fits ? s_base : 0;
        w.head[0] = fits ? nblk : 0;
        w.head[1] = fits ? ncrops : 0;
        w.head[2] = fits ? 0 : 1;
        w.head[4] = fits ? s_base : 0;
        w.head[8] = slots;
    }
}

__device__ inline unsigned bswap32(unsigned v) { return __byte_perm(v, 0, 0x0123); }

__global__ void __launch_bounds__(256) k_jpeg_pack(JpgArgs a, void* ws, long long S) {
    __shared__ BlkSmem sm;
    build_tables(sm.t);
    JpgWs w = jpg_ws(ws, S);
    const long long nblk = w.head[0], ncrops = w.head[1], ntile = w.head[3];
    const int g = threadIdx.x >> 3, r = threadIdx.x & 7;
    auto G = [&](long long b) { return b < nblk ? w.tiles[b / kJpgTile] + w.recs[b].off : w.tiles[ntile]; };
    for (long long b0 = (long long)blockIdx.x * kJpgBlocksPerCta; b0 < nblk; b0 += (long long)gridDim.x * kJpgBlocksPerCta) {
        const long long b = b0 + g;
        const bool live = b < nblk;
        long long j = 0;
        if (live && r == 0) j = owner_of(w.first, ncrops, b);
        j = __shfl_sync(0xffffffffu, j, threadIdx.x & 24);
        int4 rc = make_int4(0, 0, 1, 1);
        BlkPos p = {0, 0, 0, true};
        long long s = 0, e = 0;
        if (live) {
            rc = a.rects[j];
            p = blk_pos(rc.w, rc.z, a.ch, b - w.first[j]);
            const long long base = G(w.first[j]);
            s = G(b) - base;
            e = G(b + 1) - base;
            if (b + 1 == w.first[j + 1]) e = (e + 7) / 8 * 8;       // the crop's last block: 1-bits to a whole byte
        }
        const unsigned char* src = a.packed + (live ? a.offsets[j] / a.src_ch * a.ch : 0);
        for (int i = r; i < kJpgStageWords; i += 8) sm.stage[g][i] = 0;
        block_coefs(sm.t, src, rc.w, rc.z, a.ch, p, r, sm.tr[g], sm.zz[g], live && !p.dummy);
        unsigned* st = sm.stage[g];
        const int tab = p.comp ? 1 : 0;
        const unsigned long long mask = ac_mask(sm.zz[g], r);      // every lane of the warp takes part in the shuffles
        const int* zz = sm.zz[g];
        // this lane's bits: lane 0 the DC first, every lane its AC positions, lane 7 the EOB
        int n = 0;
        if (live) {
            if (r == 0) { const int dn = category(w.recs[b].diff); n += (sm.t.dc[tab][dn] & 255) + dn; }
            if (p.dummy) { if (r == 7) n += sm.t.ac[0][0] & 255; }
            else ac_codes(sm.t, zz, r, tab, mask, [&](unsigned, int k) { n += k; });
        }
        int pos = n;
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, pos, o, 8);
            if (r >= o) pos += y;
        }
        pos = pos - n + (int)(s & 31);
        auto put = [&](unsigned v, int k) {
            const int wd = pos >> 5, sh = pos & 31;
            if (sh + k <= 32) {
                atomicOr(st + wd, v << (32 - sh - k));
            } else {
                atomicOr(st + wd, v >> (sh + k - 32));
                atomicOr(st + wd + 1, v << (64 - sh - k));
            }
            pos += k;
        };
        if (live) {
            if (r == 0) {
                const int diff = w.recs[b].diff, dn = category(diff);
                const unsigned ec = sm.t.dc[tab][dn];
                const unsigned amp = (unsigned)(diff < 0 ? diff + (1 << dn) - 1 : diff) & ((1u << dn) - 1);
                put(((ec >> 8) << dn) | amp, (int)(ec & 255) + dn);
            }
            if (p.dummy) { if (r == 7) put(sm.t.ac[0][0] >> 8, (int)(sm.t.ac[0][0] & 255)); }
            else ac_codes(sm.t, zz, r, tab, mask, put);
            const long long cbits = G(b + 1) - G(w.first[j]);
            if (r == 7 && e > cbits) put((1u << (e - cbits)) - 1, (int)(e - cbits));
        }
        __syncwarp();
        if (live) {
            unsigned* out = (unsigned*)(w.slots + w.slot[j]) + (s >> 5);
            const int nw = (int)(((s & 31) + (e - s) + 31) >> 5);
            for (int i = r; i < nw; i += 8) {
                if (i == 0 && (s & 31)) w.recs[b].edge = bswap32(st[0]);      // the word's first bit is an earlier block's
                else out[i] = bswap32(st[i]);
            }
        }
        __syncwarp();
    }
}

__global__ void __launch_bounds__(256) k_jpeg_seam(void* ws, long long S) {
    JpgWs w = jpg_ws(ws, S);
    const long long nblk = w.head[0], ncrops = w.head[1], ntile = w.head[3];
    auto G = [&](long long b) { return b < nblk ? w.tiles[b / kJpgTile] + w.recs[b].off : w.tiles[ntile]; };
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < nblk; b += (long long)gridDim.x * blockDim.x) {
        const long long j = owner_of(w.first, ncrops, b), f = w.first[j], l = w.first[j + 1];
        const long long base = G(f), s = G(b) - base;
        if (!(s & 31)) continue;                                   // owns its first word
        if (b > f) {
            const long long ps = G(b - 1) - base;
            if ((ps >> 5) == (s >> 5) && (ps & 31)) continue;      // an earlier non-owner writes this word
        }
        unsigned v = 0;
        for (long long q = b; q < l; ++q) {
            const long long qs = G(q) - base;
            if ((qs >> 5) != (s >> 5)) break;
            v |= w.recs[q].edge;
        }
        unsigned* word = (unsigned*)(w.slots + w.slot[j]) + (s >> 5);
        *word |= v;
    }
}

__device__ inline int ff_bytes(unsigned v) { return __popc(__vcmpeq4(v, 0xffffffffu)) >> 3; }

__global__ void __launch_bounds__(256) k_jpeg_count(void* ws, long long S) {
    JpgWs w = jpg_ws(ws, S);
    const long long ncrops = w.head[1], nchunk = w.head[4];
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long c = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); c < nchunk; c += warps) {
        const long long j = owner_of(w.cfirst, ncrops, c);
        const long long b0 = (c - w.cfirst[j]) * kJpgChunk;
        const long long nbytes = min((long long)kJpgChunk, (w.dbits[j] + 7) / 8 - b0);
        const unsigned* src = (const unsigned*)(w.slots + w.slot[j] + b0);
        int n = 0;
        for (int i = lane; i < (nbytes + 3) / 4; i += 32) {
            unsigned v = src[i];
            const long long left = nbytes - 4ll * i;
            if (left < 4) v &= 0xffffffffu >> (8 * (4 - left));        // bytes past the data (memory order = low bytes first)
            n += ff_bytes(v);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
        if (lane == 0) w.cnt[c] = n;
    }
}

__global__ void __launch_bounds__(1024) k_jpeg_layout(void* ws, long long S, int channels, long long* __restrict__ jpeg_offsets,
                                                     long long* __restrict__ status, long long capacity) {
    __shared__ long long sm[32];
    __shared__ long long s_base;
    JpgWs w = jpg_ws(ws, S);
    const long long ncrops = w.head[1], nchunk = w.head[4];
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (long long c0 = 0; c0 < nchunk; c0 += blockDim.x) {
        const long long c = c0 + threadIdx.x;
        long long tot;
        const long long ex = jpg_excl_scan(c < nchunk ? w.cnt[c] : 0, sm, &tot);
        if (c < nchunk) w.cnt[c] = s_base + ex;
        __syncthreads();
        if (threadIdx.x == 0) s_base += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) { w.cnt[nchunk] = s_base; s_base = 0; }
    __syncthreads();
    const long long hdr = channels == 1 ? kJpgHeadGray : kJpgHeadColor;
    for (long long j0 = 0; j0 < ncrops; j0 += blockDim.x) {
        const long long j = j0 + threadIdx.x;
        long long v = 0;
        if (j < ncrops) {
            const long long bytes = (w.dbits[j] + 7) / 8;
            v = bytes ? hdr + bytes + (w.cnt[w.cfirst[j + 1]] - w.cnt[w.cfirst[j]]) + 2 : 0;
        }
        long long tot;
        const long long ex = jpg_excl_scan(v, sm, &tot);
        if (j < ncrops) jpeg_offsets[j] = s_base + ex;
        __syncthreads();
        if (threadIdx.x == 0) s_base += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const long long total = s_base;
        jpeg_offsets[ncrops] = total;
        status[0] = total;
        status[1] = w.head[2] ? 2 : (total > capacity ? 1 : 0);
    }
}

// SOI .. SOS of a file with nc components (h = w = 0); returns its length. One thread.
__device__ int build_header(unsigned char* o, int nc) {
    int n = 0;
    auto seg = [&](int marker, int len) { o[n++] = 0xFF; o[n++] = (unsigned char)marker; o[n++] = (unsigned char)(len >> 8); o[n++] = (unsigned char)len; };
    o[n++] = 0xFF; o[n++] = 0xD8;
    seg(0xE0, 16);
    const unsigned char jfif[14] = {'J', 'F', 'I', 'F', 0, 1, 1, 0, 0, 1, 0, 1, 0, 0};
    for (int i = 0; i < 14; ++i) o[n++] = jfif[i];
    for (int t = 0; t < (nc == 1 ? 1 : 2); ++t) {
        seg(0xDB, 67);
        o[n++] = (unsigned char)t;
        for (int i = 0; i < 64; ++i) o[n++] = (unsigned char)quant75(kStdQuant[t][kZigzag[i]]);
    }
    seg(0xC0, 8 + 3 * nc);
    o[n++] = 8;
    for (int i = 0; i < 4; ++i) o[n++] = 0;                      // h, w: patched per crop
    o[n++] = (unsigned char)nc;
    for (int ci = 0; ci < nc; ++ci) {
        o[n++] = (unsigned char)(ci + 1);
        o[n++] = nc == 1 ? 0x11 : (ci == 0 ? 0x22 : 0x11);
        o[n++] = (unsigned char)(ci ? 1 : 0);
    }
    for (int t = 0; t < (nc == 1 ? 1 : 2); ++t) {
        for (int ac = 0; ac < 2; ++ac) {
            const unsigned char* bits = ac ? kAcBits[t] : kDcBits[t];
            int nv = 0;
            for (int i = 0; i < 16; ++i) nv += bits[i];
            seg(0xC4, 3 + 16 + nv);
            o[n++] = (unsigned char)((ac << 4) | t);
            for (int i = 0; i < 16; ++i) o[n++] = bits[i];
            for (int i = 0; i < nv; ++i) o[n++] = ac ? kAcVals[t][i] : (unsigned char)i;
        }
    }
    seg(0xDA, 6 + 2 * nc);
    o[n++] = (unsigned char)nc;
    for (int ci = 0; ci < nc; ++ci) { o[n++] = (unsigned char)(ci + 1); o[n++] = ci ? 0x11 : 0x00; }
    o[n++] = 0; o[n++] = 63; o[n++] = 0;
    return n;
}

__global__ void __launch_bounds__(256) k_jpeg_assemble(JpgArgs a, void* ws, long long S, const long long* __restrict__ jpeg_offsets,
                                                      const long long* __restrict__ status, unsigned char* __restrict__ out) {
    __shared__ unsigned char tmpl[kJpgHeadColor];
    if (status[1]) return;
    JpgWs w = jpg_ws(ws, S);
    const long long ncrops = w.head[1], nchunk = w.head[4];
    if (threadIdx.x == 0) build_header(tmpl, a.ch);
    __syncthreads();
    const int hdr = a.ch == 1 ? kJpgHeadGray : kJpgHeadColor, sof = a.ch == 1 ? 89 : 158;
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long c = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); c < nchunk; c += warps) {
        const long long j = owner_of(w.cfirst, ncrops, c), cf = w.cfirst[j];
        const long long b0 = (c - cf) * kJpgChunk, bytes = (w.dbits[j] + 7) / 8;
        const long long nbytes = min((long long)kJpgChunk, bytes - b0);
        const unsigned* src = (const unsigned*)(w.slots + w.slot[j] + b0);
        unsigned char* file = out + jpeg_offsets[j];
        unsigned char* dst = file + hdr + b0 + (w.cnt[c] - w.cnt[cf]);
        if (c == cf) {
            const int4 rc = a.rects[j];
            for (int i = lane; i < hdr; i += 32) {
                unsigned char v = tmpl[i];
                if (i == sof + 5) v = (unsigned char)(rc.w >> 8);
                if (i == sof + 6) v = (unsigned char)rc.w;
                if (i == sof + 7) v = (unsigned char)(rc.z >> 8);
                if (i == sof + 8) v = (unsigned char)rc.z;
                file[i] = v;
            }
        }
        long long o = 0;                                          // output bytes of the earlier rounds
        for (int i0 = 0; i0 < (nbytes + 3) / 4; i0 += 32) {
            const int i = i0 + lane;
            const int nb = (int)max(0ll, min(4ll, nbytes - 4ll * i));
            unsigned v = nb ? src[i] : 0u;
            if (nb < 4) v &= nb ? 0xffffffffu >> (8 * (4 - nb)) : 0u;
            const int m = nb + ff_bytes(v);
            int x = m;
#pragma unroll
            for (int k = 1; k < 32; k <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, x, k);
                if (lane >= k) x += y;
            }
            unsigned char* d = dst + o + (x - m);
            for (int k = 0; k < nb; ++k) {
                const unsigned char byte = (unsigned char)(v >> (8 * k));
                *d++ = byte;
                if (byte == 0xFF) *d++ = 0;
            }
            o += __shfl_sync(0xffffffffu, x, 31);
        }
        if (c + 1 == w.cfirst[j + 1] && lane == 0) {
            unsigned char* eoi = out + jpeg_offsets[j + 1] - 2;
            eoi[0] = 0xFF; eoi[1] = 0xD9;
        }
    }
}

// Most blocks any crops of `pixels` pixels in total can have (tests/jpeg_ref.py max_blocks): a crop of h x w pixels
// (h + w <= h w + 1) has at most (h w) / 8 + 7/8 blocks in grey and 6 ((h w) / 16 + 15/16) in colour.
static long long jpg_max_blocks(long long pixels, long long crops, int c) {
    return c == 1 ? pixels / 8 + crops : 6 * (pixels / 16 + crops);
}

static size_t jpg_ws_bytes(long long S, long long packed, int c) {
    const long long blocks = jpg_max_blocks(packed / c, S, c);
    const long long chunks = blocks * kJpgBlockBytes / kJpgChunk + S + 1;
    return (size_t)(jpg_fixed_bytes(S) + 16 + blocks * (long long)sizeof(JpgRec) + 8 * (blocks / kJpgTile + 2) +
                    8 * (chunks + 1) + 16 + blocks * kJpgBlockBytes + 16 * S);
}

}  // namespace mb

using namespace mb;

extern "C" int64_t mb_jpeg_bound_bytes(int64_t packed_bytes, int64_t crops, int32_t channels) {
    if ((channels != 1 && channels != 3) || packed_bytes < 0 || crops < 0) return -1;
    const long long hdr = channels == 1 ? kJpgHeadGray : kJpgHeadColor;
    return crops * (hdr + 2) + 2ll * kJpgBlockBytes * jpg_max_blocks(packed_bytes / channels, crops, channels);
}

extern "C" size_t mb_jpeg_workspace_bytes(const mb_crop_params* p, int64_t packed_capacity_bytes, int32_t channels) {
    if (!p || (channels != 1 && channels != 3) || packed_capacity_bytes < 0 || p->num_images < 1 || p->capacity < 1) return 0;
    return jpg_ws_bytes((long long)p->num_images * p->capacity, packed_capacity_bytes, channels);
}

extern "C" int mb_jpeg_encode(const mb_crop_params* p, const uint8_t* packed, int32_t channels, const int32_t* rects,
                              const int64_t* offsets, const int64_t* totals, void* workspace, size_t workspace_bytes,
                              uint8_t* jpeg_out, int64_t jpeg_capacity_bytes, int64_t* jpeg_offsets_out,
                              int64_t* jpeg_status_out, mb_stream_t stream) {
    if (!p || !rects || !offsets || !totals || !workspace || !jpeg_offsets_out || !jpeg_status_out || jpeg_capacity_bytes < 0)
        return MB_ERR_INVALID_ARG;
    if ((channels != 1 && channels != 3) || p->channels < 1 || p->channels > 4) return MB_ERR_UNSUPPORTED;
    if (p->num_images < 1 || p->num_images > MB_MAX_IMAGES || p->capacity < 1) return MB_ERR_INVALID_ARG;
    for (int i = 0; i < p->num_images; ++i)
        if (p->image_h[i] > 65535 || p->image_w[i] > 65535) return MB_ERR_UNSUPPORTED;
    if (jpeg_capacity_bytes > 0 && !jpeg_out) return MB_ERR_INVALID_ARG;
    const long long S = (long long)p->num_images * p->capacity;
    if ((long long)workspace_bytes < (jpg_fixed_bytes(S) + 15) / 16 * 16 + 32) return MB_ERR_WORKSPACE;
    JpgArgs a;
    a.packed = packed; a.rects = (const int4*)rects; a.offsets = (const long long*)offsets;
    a.src_ch = p->channels; a.ch = channels;
    const cudaStream_t st = (cudaStream_t)stream;
    k_jpeg_plan<<<1, 1024, 0, st>>>(a, (const long long*)totals, workspace, workspace_bytes, S);
    MB_LAUNCH_CHECK();
    // the grids cover the most blocks / chunks the workspace can describe, capped at the persistent size
    const long long max_blocks = std::max<long long>(1, (long long)(workspace_bytes / (sizeof(JpgRec) + kJpgBlockBytes)));
    const int sms = num_sms();
    const int gb = (int)std::min<long long>(ceil_div64(max_blocks, kJpgBlocksPerCta), (long long)sms * 8);
    const int gt = (int)std::min<long long>(ceil_div64(max_blocks, kJpgTile), (long long)sms * 2);
    const int gc = (int)std::min<long long>(ceil_div64(max_blocks * kJpgBlockBytes / kJpgChunk + S + 1, 8), (long long)sms * 8);
    k_jpeg_blocks<<<gb, 256, 0, st>>>(a, workspace, S);
    MB_LAUNCH_CHECK();
    k_jpeg_bits<<<gt, kJpgTile, 0, st>>>(a, workspace, S);
    MB_LAUNCH_CHECK();
    k_jpeg_scan<<<1, 1024, 0, st>>>(workspace, workspace_bytes, S);
    MB_LAUNCH_CHECK();
    k_jpeg_pack<<<gb, 256, 0, st>>>(a, workspace, S);
    MB_LAUNCH_CHECK();
    k_jpeg_seam<<<(int)std::min<long long>(ceil_div64(max_blocks, 256), (long long)sms * 8), 256, 0, st>>>(workspace, S);
    MB_LAUNCH_CHECK();
    k_jpeg_count<<<gc, 256, 0, st>>>(workspace, S);
    MB_LAUNCH_CHECK();
    k_jpeg_layout<<<1, 1024, 0, st>>>(workspace, S, channels, (long long*)jpeg_offsets_out, (long long*)jpeg_status_out,
                                      jpeg_capacity_bytes);
    MB_LAUNCH_CHECK();
    k_jpeg_assemble<<<gc, 256, 0, st>>>(a, workspace, S, (const long long*)jpeg_offsets_out, (const long long*)jpeg_status_out,
                                        jpeg_out);
    MB_LAUNCH_CHECK();
    return MB_OK;
}
