// png.cu — lossless PNG streams of the packed crops (or masks) of the crop stage, one complete file per crop.
//
// The encoding is stated in include/misob200.h (mb_png_encode) and restated on the CPU in tests/png_ref.py.
//   k_png_plan      one CTA: per crop its filtered size h * (1 + w * c), its blocks (cuts every 32 KiB of filtered
//                   bytes) and its workspace slots; block -> crop table; the workspace fit check
//   k_png_encode    persistent grid, one CTA per block: rows filtered on the fly from the source (a warp per row:
//                   libpng's minimum-sum heuristic over the whole row, so the choice does not depend on the cut),
//                   runs by a compare with the previous byte and two CTA scans, histogram, package-merge code lengths
//                   (CTA-parallel merge by rank), zlib's code-length run coding (one thread), a per-thread bit offset
//                   scan and the bits OR-ed into shared memory; stored when not smaller; the segment goes to its slot
//                   with its raw CRC, x^(8 len) and Adler partials
//   k_png_layout    one CTA: scan of the segment sizes (plus 43 header / 22 trailer bytes per crop) to the output
//                   positions, the per-crop offsets, total and overflow flag, before anything is written
//   k_png_assemble  persistent grid, one CTA per block: copy of the segment; the crop's first block writes the
//                   signature, IHDR and IDAT header, its last block folds the crop's CRC / Adler partials (warp 0)
//                   and writes the trailer. The encoder writes to slots first because no crop's size is known until
//                   all its blocks are encoded.
#include <algorithm>

#include "common.cuh"

namespace mb {

constexpr int kPngBlock = 32768;                  // filtered bytes per deflate block
constexpr int kPngThreads = 512;                  // encoder CTA
constexpr int kPngPer = kPngBlock / kPngThreads;  // positions per encoder thread (contiguous)
constexpr int kPngCrcChunk = 72;                  // CRC bytes per thread: 512 * 72 >= the largest segment (32778)
constexpr int kPngOutWords = 8200;                // segment buffer (32800 bytes)
constexpr int kPngHead = 43, kPngTail = 22;       // bytes before the first / after the last segment of a crop
constexpr unsigned kPoly = 0xedb88320u;
constexpr unsigned kAdler = 65521u;

struct PngBlock {
    long long pos;      // output byte of the segment's first byte (k_png_layout), minus kPngHead for a crop's first block
    long long slot;     // workspace byte of the segment
    int crop, index;    // crop and block index within it
    unsigned seglen, len, crc, xpow, a, b;   // segment bytes, filtered bytes, raw CRC, x^(8 seglen), Adler partials
};

struct PngWs {
    long long* first;   // [S + 1] first block of crop j
    long long* head;    // [8]: 0 blocks, 1 crops encoded, 2 workspace too small
    PngBlock* blocks;
    unsigned char* base;
    long long rec_cap;  // block records that fit before the slot area
    long long slot_begin, bytes;
};

__host__ __device__ inline long long png_filtered(int h, int w, int c) { return (h > 0 && w > 0) ? (long long)h * (1 + (long long)w * c) : 0; }

// ---- GF(2) arithmetic of CRC-32 (zlib's crc32_combine operator) ---------------------------------------------------
__host__ __device__ inline unsigned multmodp(unsigned a, unsigned b) {
    unsigned m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = (b & 1) ? (b >> 1) ^ kPoly : b >> 1;
    }
    return p;
}
// x^(8 n) from the table x2n[k] = x^(2^k)
__device__ inline unsigned x8n(long long n, const unsigned* x2n) {
    unsigned p = 1u << 31;
    for (int k = 3; n; n >>= 1, ++k)
        if (n & 1) p = multmodp(x2n[k & 31], p);
    return p;
}
__device__ inline unsigned crc_raw_bits(unsigned c, const unsigned char* d, int n) {
    for (int i = 0; i < n; ++i) {
        c ^= d[i];
        for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ kPoly : c >> 1;
    }
    return c;
}

__device__ inline void put_bits(unsigned* out, long long pos, unsigned v, int n) {
    if (n == 0) return;
    const int w = (int)(pos >> 5), sh = (int)(pos & 31);
    atomicOr(out + w, v << sh);
    if (sh + n > 32) atomicOr(out + w + 1, v >> (32 - sh));
}

// ---- CTA scans -----------------------------------------------------------------------------------------------------
template <typename T, typename Op>
__device__ inline T cta_excl_scan(T v, T identity, Op op, T* sm, T* total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    T x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x = op(y, x);
    }
    if (lane == 31) sm[wid] = x;
    __syncthreads();
    T pre = identity, all = identity;
    for (int q = 0; q < nw; ++q) {
        if (q < wid) pre = op(pre, sm[q]);
        all = op(all, sm[q]);
    }
    T ex = __shfl_up_sync(0xffffffffu, x, 1);
    if (lane == 0) ex = identity;
    __syncthreads();
    if (total) *total = all;
    return op(pre, ex);
}

// ---- length symbols -------------------------------------------------------------------------------------------------
__device__ __constant__ short kLenBase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83,
                                             99, 115, 131, 163, 195, 227, 258};
__device__ __constant__ unsigned char kLenExtra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4,
                                                       5, 5, 5, 5, 0};
// length 3..258 -> symbol - 257 (bits 0..4), extra bits (5..7), extra value (8..12)
__device__ inline unsigned short len_entry(int l) {
    int i = 28;
    while (kLenBase[i] > l) --i;
    return (unsigned short)(i | (kLenExtra[i] << 5) | ((l - kLenBase[i]) << 8));
}

// Tokens of positions [lo, hi) of a block: f(position, is_match, value) for every position that emits one.
// carry_s: start of the run containing lo; carry_e: first run start at or after hi.
template <typename F>
__device__ inline void for_each_token(const unsigned char* d, int lo, int hi, int carry_s, int carry_e, F f) {
    int i = lo;
    while (i < hi) {
        const unsigned char v = d[i];
        const bool st = (i == 0) || d[i - 1] != v;
        const int s = st ? i : carry_s;
        int j = i + 1;
        while (j < hi && d[j] == v) ++j;
        const int e = j < hi ? j : carry_e;
        const int m = e - s - 1, full = m / 258, r = m - 258 * full;
        for (int p = i; p < j; ++p) {
            const int k = p - s;
            if (k == 0) { f(p, false, (int)v); continue; }
            const int q = k - 1;
            if (q < 258 * full) {
                if (q % 258 == 0) f(p, true, 258);
            } else if (r >= 3) {
                if (q == 258 * full) f(p, true, r);
            } else {
                f(p, false, (int)v);
            }
        }
        i = j;
    }
}

// Package-merge code lengths (all threads call it). freq[nsym] -> len[nsym]; scratch: weights 2 x (2 * nsym), leaf
// positions limit x nsym (u16), order / leaf weights nsym each.
struct PmScratch {
    unsigned* wa; unsigned* wb; unsigned short* lpos; unsigned short* order; unsigned* leaves; int* nl;
};
__device__ void package_merge(const unsigned* freq, int nsym, int limit, unsigned char* len, PmScratch s, int* sh_n) {
    const int tid = threadIdx.x;
    for (int i = tid; i < nsym; i += blockDim.x) len[i] = 0;
    if (tid == 0) {
        int n = 0;
        for (int i = 0; i < nsym; ++i) n += freq[i] > 0;
        *sh_n = n;
    }
    __syncthreads();
    const int n = *sh_n;
    if (n < 2) {
        if (tid == 0) {
            int need = 2 - n;
            for (int i = 0; i < nsym; ++i) if (freq[i] > 0) len[i] = 1;
            for (int i = 0; i < nsym && need; ++i) if (freq[i] == 0) { len[i] = 1; --need; }
        }
        __syncthreads();
        return;
    }
    for (int i = tid; i < nsym; i += blockDim.x) {
        const unsigned f = freq[i];
        if (f == 0) continue;
        int r = 0;
        for (int t = 0; t < nsym; ++t) {
            const unsigned g = freq[t];
            r += g > 0 && (g < f || (g == f && t < i));
        }
        s.order[r] = (unsigned short)i;
        s.leaves[r] = f;
    }
    __syncthreads();
    for (int i = tid; i < n; i += blockDim.x) { s.wa[i] = s.leaves[i]; s.lpos[(limit - 1) * nsym + i] = (unsigned short)i; }
    __syncthreads();
    unsigned* cur = s.wa; unsigned* nxt = s.wb;
    int cn = n;
    for (int d = limit - 1; d >= 1; --d) {
        const int np = cn / 2;
        // leaf i: before every package of equal weight
        for (int i = tid; i < n; i += blockDim.x) {
            const unsigned w = s.leaves[i];
            int lo = 0, hi = np;                            // packages with weight < w
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (cur[2 * mid] + cur[2 * mid + 1] < w) lo = mid + 1; else hi = mid; }
            nxt[i + lo] = w;
            s.lpos[(d - 1) * nsym + i] = (unsigned short)(i + lo);
        }
        for (int k = tid; k < np; k += blockDim.x) {
            const unsigned w = cur[2 * k] + cur[2 * k + 1];
            int lo = 0, hi = n;                             // leaves with weight <= w
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (s.leaves[mid] <= w) lo = mid + 1; else hi = mid; }
            nxt[k + lo] = w;
        }
        __syncthreads();
        unsigned* t = cur; cur = nxt; nxt = t;
        cn = n + np;
    }
    if (tid == 0) {
        long long k = 2 * n - 2;
        for (int d = 1; d <= limit; ++d) {
            const unsigned short* lp = s.lpos + (d - 1) * nsym;
            int lo = 0, hi = n;                             // leaves at positions < k
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (lp[mid] < k) lo = mid + 1; else hi = mid; }
            s.nl[d - 1] = lo;
            k = 2 * (k - lo);
        }
    }
    __syncthreads();
    for (int i = tid; i < n; i += blockDim.x) {
        int l = 0;
        for (int d = 0; d < limit; ++d) l += i < s.nl[d];
        len[s.order[i]] = (unsigned char)l;
    }
    __syncthreads();
}

// canonical codes, bit-reversed (all threads)
__device__ void canonical(const unsigned char* len, int nsym, unsigned short* code, int* next) {
    if (threadIdx.x == 0) {
        int cnt[16] = {0};
        for (int i = 0; i < nsym; ++i) if (len[i]) ++cnt[len[i]];
        int c = 0;
        for (int b = 1; b < 16; ++b) { c = (c + cnt[b - 1]) << 1; next[b] = c; }   // cnt[0] = 0: next[1] = 0
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nsym; i += blockDim.x) {
        const int l = len[i];
        if (!l) { code[i] = 0; continue; }
        int r = 0;
        for (int t = 0; t < i; ++t) r += len[t] == l;
        const unsigned c = (unsigned)(next[l] + r);
        code[i] = (unsigned short)(__brev(c) >> (32 - l));
    }
    __syncthreads();
}

// zlib's scan_tree / send_tree run coding of one tree's lengths (one thread): appends (symbol, extra) pairs
__device__ int tree_runs(const unsigned char* lens, int count_n, unsigned char* rs, unsigned char* rx, int nr) {
    int prevlen = -1, nextlen = lens[0], count = 0;
    int max_count = 7, min_count = 4;
    if (nextlen == 0) { max_count = 138; min_count = 3; }
    for (int n = 0; n < count_n; ++n) {
        const int curlen = nextlen;
        nextlen = n + 1 < count_n ? lens[n + 1] : 0xffff;
        if (++count < max_count && curlen == nextlen) continue;
        if (count < min_count) {
            for (int q = 0; q < count; ++q) { rs[nr] = (unsigned char)curlen; rx[nr++] = 0; }
        } else if (curlen != 0) {
            if (curlen != prevlen) { rs[nr] = (unsigned char)curlen; rx[nr++] = 0; --count; }
            rs[nr] = 16; rx[nr++] = (unsigned char)(count - 3);
        } else if (count <= 10) {
            rs[nr] = 17; rx[nr++] = (unsigned char)(count - 3);
        } else {
            rs[nr] = 18; rx[nr++] = (unsigned char)(count - 11);
        }
        count = 0; prevlen = curlen;
        if (nextlen == 0) { max_count = 138; min_count = 3; }
        else if (curlen == nextlen) { max_count = 6; min_count = 3; }
        else { max_count = 7; min_count = 4; }
    }
    return nr;
}

__device__ inline int run_xbits(int s) { return s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0; }

__device__ __constant__ unsigned char kBlOrder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

struct PngArgs {
    const unsigned char* packed;
    const int4* rects;
    const long long* offsets;
    int src_ch, ch;
};

__device__ inline PngWs png_ws(void* ws, size_t bytes, long long S) {
    PngWs w;
    unsigned char* b = (unsigned char*)ws;
    w.first = (long long*)b;
    w.head = w.first + (S + 1);
    w.blocks = (PngBlock*)(w.head + 8);
    w.base = b;
    const long long rec_off = (long long)((unsigned char*)w.blocks - b);
    w.bytes = (long long)bytes;
    w.slot_begin = 0;
    w.rec_cap = ((long long)bytes - rec_off) / (long long)sizeof(PngBlock);
    return w;
}

__global__ void __launch_bounds__(1024) k_png_plan(PngArgs a, const long long* __restrict__ totals, void* ws, size_t ws_bytes,
                                                  long long S) {
    __shared__ long long sm[32];
    __shared__ long long s_blk, s_slot;
    PngWs w = png_ws(ws, ws_bytes, S);
    const long long ncrops = (totals[2] || totals[3]) ? 0 : totals[0];
    if (threadIdx.x == 0) { s_blk = 0; s_slot = 0; }
    __syncthreads();
    auto add = [](long long x, long long y) { return x + y; };
    for (long long j0 = 0; j0 < ncrops; j0 += blockDim.x) {
        const long long j = j0 + threadIdx.x;
        long long nb = 0, sb = 0;
        if (j < ncrops) {
            const int4 rc = a.rects[j];
            const long long f = png_filtered(rc.w, rc.z, a.ch);
            nb = (f + kPngBlock - 1) / kPngBlock;
            if (nb) sb = (nb - 1) * (kPngBlock + 16) + ((f - (nb - 1) * kPngBlock + 15) / 16) * 16 + 16;
        }
        long long tb, ts;
        const long long eb = cta_excl_scan<long long>(nb, 0, add, sm, &tb);
        const long long es = cta_excl_scan<long long>(sb, 0, add, sm, &ts);
        const long long fb = s_blk + eb, fs = s_slot + es;
        if (j < ncrops) {
            w.first[j] = fb;
            // the block records of this crop (slot offsets from the end of the workspace are set once the total is known)
            for (long long q = 0; q < nb; ++q) {
                if (fb + q < w.rec_cap) {
                    PngBlock& r = w.blocks[fb + q];
                    r.crop = (int)j; r.index = (int)q;
                    r.slot = fs + q * (kPngBlock + 16);       // relative to the slot area
                }
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) { s_blk += tb; s_slot += ts; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const long long nblk = s_blk, slot_bytes = s_slot;
        const long long rec_end = (long long)((unsigned char*)(w.blocks + nblk) - w.base);
        const long long slot_begin = ((w.bytes - slot_bytes) / 16) * 16;
        const bool fits = rec_end <= slot_begin;
        w.first[fits ? ncrops : 0] = fits ? nblk : 0;
        w.head[0] = fits ? nblk : 0;
        w.head[1] = fits ? ncrops : 0;
        w.head[2] = fits ? 0 : 1;
        w.head[3] = slot_begin;
    }
}

struct EncSmem {
    unsigned char in[kPngBlock];
    unsigned out[kPngOutWords];            // also the package-merge scratch before the bits are written
    unsigned crc_tab[256];
    unsigned x2n[32];
    unsigned shift[16];
    unsigned freq[288];
    unsigned short lentab[260];
    unsigned blf[20];
    unsigned char ll[288];
    unsigned char bl[20];
    unsigned short llc[288];
    unsigned short blc[20];
    unsigned char rs[320], rx[320];
    int next[16];
    int nl[16];
    int misc[8];
    long long scan[32];
    unsigned long long scan64[32];
    unsigned scanu[32];
};

__global__ void __launch_bounds__(kPngThreads) k_png_encode(PngArgs a, void* ws, size_t ws_bytes, long long S) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    EncSmem& sm = *reinterpret_cast<EncSmem*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    PngWs w = png_ws(ws, ws_bytes, S);
    const long long nblk = w.head[0];
    unsigned char* slots = w.base + w.head[3];
    // per-CTA tables: CRC bytes, x^(2^k), x^(8 * chunk * 2^k)
    for (int l = tid; l < 259; l += blockDim.x) sm.lentab[l] = l >= 3 ? len_entry(l) : 0;
    for (int i = tid; i < 256; i += blockDim.x) {
        unsigned c = (unsigned)i;
        for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ kPoly : c >> 1;
        sm.crc_tab[i] = c;
    }
    if (tid == 0) {
        unsigned p = 1u << 30;                          // x^1
        for (int k = 0; k < 32; ++k) { sm.x2n[k] = p; p = multmodp(p, p); }
        sm.shift[0] = x8n(kPngCrcChunk, sm.x2n);
        for (int k = 1; k < 16; ++k) sm.shift[k] = multmodp(sm.shift[k - 1], sm.shift[k - 1]);
    }
    __syncthreads();
    for (long long b = blockIdx.x; b < nblk; b += gridDim.x) {
        PngBlock& rec = w.blocks[b];
        const int j = rec.crop, kb = rec.index;
        const int4 rc = a.rects[j];
        const int h = rc.w, wd = rc.z, c = a.ch;
        const long long rowb = (long long)wd * c, R = rowb + 1;
        const long long F = png_filtered(h, wd, c);
        const long long t0 = (long long)kb * kPngBlock;
        const int L = (int)min((long long)kPngBlock, F - t0);
        const unsigned char* src = a.packed + a.offsets[j] / a.src_ch * c;
        // ---- filter the rows this block covers (a warp per row) ----
        const long long r0 = t0 / R, r1 = (t0 + L - 1) / R;
        for (long long r = r0 + warp; r <= r1; r += blockDim.x >> 5) {
            const unsigned char* cur = src + r * rowb;
            const unsigned char* up = r > 0 ? cur - rowb : nullptr;
            int s0 = 0, s1 = 0, s2 = 0, s3 = 0, s4 = 0;
            auto absb = [](int v) { v &= 255; return v < 128 ? v : 256 - v; };
            for (long long x = lane; x < rowb; x += 32) {
                const int xa = cur[x], lf = x >= c ? cur[x - c] : 0, u = up ? up[x] : 0, ul = (up && x >= c) ? up[x - c] : 0;
                const int p = lf + u - ul, pa = abs(p - lf), pb = abs(p - u), pc = abs(p - ul);
                const int pr = (pa <= pb && pa <= pc) ? lf : (pb <= pc ? u : ul);
                s0 += absb(xa); s1 += absb(xa - lf); s2 += absb(xa - u); s3 += absb(xa - ((lf + u) >> 1)); s4 += absb(xa - pr);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                s0 += __shfl_xor_sync(0xffffffffu, s0, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                s2 += __shfl_xor_sync(0xffffffffu, s2, o); s3 += __shfl_xor_sync(0xffffffffu, s3, o);
                s4 += __shfl_xor_sync(0xffffffffu, s4, o);
            }
            int ft = 0, best = s0;
            if (s1 < best) { best = s1; ft = 1; }
            if (s2 < best) { best = s2; ft = 2; }
            if (s3 < best) { best = s3; ft = 3; }
            if (s4 < best) { best = s4; ft = 4; }
            const long long rs0 = r * R;
            const long long u0 = max(0ll, t0 - rs0), u1 = min(R, t0 + L - rs0);
            for (long long u = u0 + lane; u < u1; u += 32) {
                int v;
                if (u == 0) v = ft;
                else {
                    const long long x = u - 1;
                    const int xa = cur[x], lf = x >= c ? cur[x - c] : 0, uu = up ? up[x] : 0, ul = (up && x >= c) ? up[x - c] : 0;
                    if (ft == 0) v = xa;
                    else if (ft == 1) v = xa - lf;
                    else if (ft == 2) v = xa - uu;
                    else if (ft == 3) v = xa - ((lf + uu) >> 1);
                    else {
                        const int p = lf + uu - ul, pa = abs(p - lf), pb = abs(p - uu), pc = abs(p - ul);
                        v = xa - ((pa <= pb && pa <= pc) ? lf : (pb <= pc ? uu : ul));
                    }
                }
                sm.in[rs0 + u - t0] = (unsigned char)v;
            }
        }
        for (int i = tid; i < 288; i += blockDim.x) sm.freq[i] = 0;
        __syncthreads();
        // ---- runs: carry-in start and carry-out end across threads; Adler partials ----
        const int lo = min(L, tid * kPngPer), hi = min(L, lo + kPngPer);
        int fs = L, ls = -1;
        unsigned sa = 0;
        unsigned long long sb = 0;
        for (int i = lo; i < hi; ++i) {
            const unsigned char v = sm.in[i];
            if (i == 0 || sm.in[i - 1] != v) { fs = min(fs, i); ls = i; }
            sa += v;
            sb += (unsigned long long)(L - i) * v;
        }
        auto imax = [](int x, int y) { return max(x, y); };
        const int carry_s = cta_excl_scan<int>(ls, -1, imax, (int*)sm.scan, nullptr);
        // first run start after this thread's range: a min over the later threads = a max-scan of -fs in reverse order
        int carry_e;
        {
            // reverse order: thread t reads its mirror's value through shared memory
            __shared__ int rev[kPngThreads];
            rev[kPngThreads - 1 - tid] = -fs;
            __syncthreads();
            const int mine = rev[tid];
            __syncthreads();
            const int ex = cta_excl_scan<int>(mine, -L, imax, (int*)sm.scan, nullptr);  // over threads after the mirror
            rev[kPngThreads - 1 - tid] = ex;
            __syncthreads();
            carry_e = -rev[tid];
            __syncthreads();
        }
        auto add32 = [](unsigned x, unsigned y) { return x + y; };
        auto add64 = [](unsigned long long x, unsigned long long y) { return x + y; };
        unsigned ta; unsigned long long tbw;
        cta_excl_scan<unsigned>(sa, 0u, add32, sm.scanu, &ta);
        cta_excl_scan<unsigned long long>(sb, 0ull, add64, sm.scan64, &tbw);
        // ---- histogram ----
        for_each_token(sm.in, lo, hi, carry_s, carry_e, [&](int, bool m, int v) {
            atomicAdd(&sm.freq[m ? 257 + (sm.lentab[v] & 31) : v], 1u);
        });
        if (tid == 0) sm.freq[256] += 1;
        __syncthreads();
        // ---- code lengths ----
        PmScratch ps;
        ps.wa = sm.out; ps.wb = sm.out + 600; ps.leaves = sm.out + 1200; ps.order = (unsigned short*)(sm.out + 1500);
        ps.lpos = (unsigned short*)(sm.out + 1700); ps.nl = sm.nl;
        package_merge(sm.freq, 286, 15, sm.ll, ps, &sm.misc[0]);
        if (tid == 0) {
            int hlit = 257;
            for (int s = 285; s >= 257; --s) if (sm.ll[s]) { hlit = s + 1; break; }
            const unsigned char dl[2] = {1, 1};
            int nr = tree_runs(sm.ll, hlit, sm.rs, sm.rx, 0);
            nr = tree_runs(dl, 2, sm.rs, sm.rx, nr);
            for (int s = 0; s < 20; ++s) sm.blf[s] = 0;
            for (int q = 0; q < nr; ++q) sm.blf[sm.rs[q]] += 1;
            sm.misc[1] = hlit; sm.misc[2] = nr;
        }
        __syncthreads();
        package_merge(sm.blf, 19, 7, sm.bl, ps, &sm.misc[0]);
        canonical(sm.ll, 286, sm.llc, sm.next);
        canonical(sm.bl, 19, sm.blc, sm.next);
        if (tid == 0) {
            int hclen = 4;
            for (int i = 18; i >= 4; --i) if (sm.bl[kBlOrder[i]]) { hclen = i + 1; break; }
            long long bits = 3 + 5 + 5 + 4 + 3 * hclen;
            for (int q = 0; q < sm.misc[2]; ++q) bits += sm.bl[sm.rs[q]] + run_xbits(sm.rs[q]);
            sm.misc[3] = hclen; sm.misc[4] = (int)bits;
        }
        __syncthreads();
        // ---- bit offsets ----
        long long mybits = 0;
        for_each_token(sm.in, lo, hi, carry_s, carry_e, [&](int, bool m, int v) {
            if (m) { const unsigned e = sm.lentab[v]; mybits += sm.ll[257 + (e & 31)] + ((e >> 5) & 7) + 1; }
            else mybits += sm.ll[v];
        });
        long long tok_total;
        auto add = [](long long x, long long y) { return x + y; };
        const long long myoff = cta_excl_scan<long long>(mybits, 0, add, sm.scan, &tok_total);
        const long long hdr = sm.misc[4];
        const long long total = hdr + tok_total + sm.ll[256];
        const long long dyn_bytes = (total + 3 + 7) / 8 + 4;
        const bool dynamic = dyn_bytes < (long long)L + 10;
        const int seglen = dynamic ? (int)dyn_bytes : L + 10;
        for (int i = tid; i < (seglen + 3) / 4; i += blockDim.x) sm.out[i] = 0;
        __syncthreads();
        unsigned char* ob = reinterpret_cast<unsigned char*>(sm.out);
        if (dynamic) {
            if (tid == 0) {
                long long pos = 0;
                auto put = [&](unsigned v, int n) { put_bits(sm.out, pos, v, n); pos += n; };
                put(0, 1); put(2, 2); put(sm.misc[1] - 257, 5); put(1, 5); put(sm.misc[3] - 4, 4);
                for (int i = 0; i < sm.misc[3]; ++i) put(sm.bl[kBlOrder[i]], 3);
                for (int q = 0; q < sm.misc[2]; ++q) {
                    const int s = sm.rs[q];
                    put(sm.blc[s], sm.bl[s]);
                    if (run_xbits(s)) put(sm.rx[q], run_xbits(s));
                }
                put_bits(sm.out, hdr + tok_total, sm.llc[256], sm.ll[256]);
            }
            long long pos = hdr + myoff;
            for_each_token(sm.in, lo, hi, carry_s, carry_e, [&](int, bool m, int v) {
                if (m) {
                    const unsigned e = sm.lentab[v];
                    const int sym = 257 + (e & 31), xb = (e >> 5) & 7, xv = e >> 8;
                    const int n = sm.ll[sym];
                    put_bits(sm.out, pos, (unsigned)sm.llc[sym] | ((unsigned)xv << n), n + xb + 1);  // + distance code 0
                    pos += n + xb + 1;
                } else {
                    put_bits(sm.out, pos, sm.llc[v], sm.ll[v]);
                    pos += sm.ll[v];
                }
            });
            __syncthreads();
            if (tid == 0) {
                const int q = (int)((total + 3 + 7) / 8);
                ob[q] = 0; ob[q + 1] = 0; ob[q + 2] = 0xff; ob[q + 3] = 0xff;
            }
        } else {
            for (int i = tid; i < L; i += blockDim.x) ob[5 + i] = sm.in[i];
            if (tid == 0) {
                ob[0] = 0; ob[1] = (unsigned char)(L & 255); ob[2] = (unsigned char)(L >> 8);
                ob[3] = (unsigned char)(~L & 255); ob[4] = (unsigned char)((~L >> 8) & 255);
                ob[L + 5] = 0; ob[L + 6] = 0; ob[L + 7] = 0; ob[L + 8] = 0xff; ob[L + 9] = 0xff;
            }
        }
        __syncthreads();
        // ---- raw CRC of the segment: right-aligned chunks (leading zeros do not change a zero-initialised CRC) ----
        unsigned crc = 0;
        {
            const int e = seglen - (kPngThreads - 1 - tid) * kPngCrcChunk;
            const int s0 = max(0, e - kPngCrcChunk);
            for (int i = s0; i < e; ++i) crc = sm.crc_tab[(crc ^ ob[i]) & 255] ^ (crc >> 8);
        }
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            const unsigned o = __shfl_down_sync(0xffffffffu, crc, 1 << k);
            if ((lane & ((2 << k) - 1)) == 0) crc = multmodp(sm.shift[k], crc) ^ o;
        }
        if (lane == 0) sm.scanu[warp] = crc;
        unsigned xp = 0;
        if (tid == 32) xp = x8n(seglen, sm.x2n);
        // ---- segment to its slot ----
        unsigned char* dst = slots + rec.slot;
        for (int i = tid; i < (seglen + 15) / 16; i += blockDim.x)
            reinterpret_cast<uint4*>(dst)[i] = reinterpret_cast<const uint4*>(sm.out)[i];
        __syncthreads();
        if (tid == 0) {
            unsigned r = 0;
            for (int q = 0; q < (int)(blockDim.x >> 5); ++q) r = multmodp(sm.shift[5], r) ^ sm.scanu[q];
            rec.crc = r;
            rec.seglen = (unsigned)seglen;
            rec.len = (unsigned)L;
            rec.a = ta % kAdler;
            rec.b = (unsigned)(tbw % kAdler);
        }
        if (tid == 32) rec.xpow = xp;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(1024) k_png_layout(void* ws, size_t ws_bytes, long long S, long long* __restrict__ png_offsets,
                                                    long long* __restrict__ status, long long capacity) {
    __shared__ long long sm[32];
    __shared__ long long s_base;
    PngWs w = png_ws(ws, ws_bytes, S);
    const long long nblk = w.head[0], ncrops = w.head[1];
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    auto add = [](long long x, long long y) { return x + y; };
    for (long long b0 = 0; b0 < nblk; b0 += blockDim.x) {
        const long long b = b0 + threadIdx.x;
        long long v = 0;
        if (b < nblk) {
            const PngBlock& r = w.blocks[b];
            const bool last = b + 1 == nblk || w.blocks[b + 1].crop != r.crop;
            v = r.seglen + (r.index == 0 ? kPngHead : 0) + (last ? kPngTail : 0);
        }
        long long tot;
        const long long ex = cta_excl_scan<long long>(v, 0, add, sm, &tot);
        if (b < nblk) w.blocks[b].pos = s_base + ex;
        __syncthreads();
        if (threadIdx.x == 0) s_base += tot;
        __syncthreads();
    }
    const long long total = s_base;
    for (long long j = threadIdx.x; j < ncrops; j += blockDim.x) {
        const long long f = w.first[j];
        png_offsets[j] = f < nblk ? w.blocks[f].pos : total;
    }
    if (threadIdx.x == 0) {
        png_offsets[ncrops] = total;
        status[0] = total;
        status[1] = w.head[2] ? 2 : (total > capacity ? 1 : 0);
    }
}

__device__ inline void put_be32(unsigned char* p, unsigned v) {
    p[0] = (unsigned char)(v >> 24); p[1] = (unsigned char)(v >> 16); p[2] = (unsigned char)(v >> 8); p[3] = (unsigned char)v;
}

struct Fold {
    unsigned r, x, a, b, l;
};
__device__ inline Fold fold(const Fold& p, const Fold& q) {
    Fold o;
    o.r = multmodp(q.x, p.r) ^ q.r;
    o.x = multmodp(p.x, q.x);
    o.b = (unsigned)(((unsigned long long)p.b + (unsigned long long)q.l * p.a + q.b) % kAdler);
    o.a = (p.a + q.a) % kAdler;
    o.l = (p.l + q.l) % kAdler;
    return o;
}

__global__ void __launch_bounds__(256) k_png_assemble(PngArgs a, void* ws, size_t ws_bytes, long long S,
                                                     const long long* __restrict__ png_offsets, const long long* __restrict__ status,
                                                     unsigned char* __restrict__ out) {
    __shared__ unsigned x2n[32];
    PngWs w = png_ws(ws, ws_bytes, S);
    if (status[1]) return;
    const long long nblk = w.head[0];
    const unsigned char* slots = w.base + w.head[3];
    if (threadIdx.x == 0) {
        unsigned p = 1u << 30;
        for (int k = 0; k < 32; ++k) { x2n[k] = p; p = multmodp(p, p); }
    }
    __syncthreads();
    for (long long b = blockIdx.x; b < nblk; b += gridDim.x) {
        const PngBlock rec = w.blocks[b];
        const int j = rec.crop;
        const long long seg0 = rec.pos + (rec.index == 0 ? kPngHead : 0);
        const unsigned char* s = slots + rec.slot;
        unsigned char* d = out + seg0;
        for (int i = threadIdx.x; i < (int)rec.seglen; i += blockDim.x) d[i] = s[i];
        const long long first = w.first[j], nb = w.first[j + 1] - first;
        if (rec.index == 0 && threadIdx.x == 0) {
            const int4 rc = a.rects[j];
            unsigned char* hp = out + rec.pos;
            const unsigned char sig[8] = {0x89, 'P', 'N', 'G', '\r', '\n', 0x1a, '\n'};
            for (int i = 0; i < 8; ++i) hp[i] = sig[i];
            unsigned char ih[17] = {'I', 'H', 'D', 'R'};
            put_be32(ih + 4, (unsigned)rc.z); put_be32(ih + 8, (unsigned)rc.w);
            const unsigned char ct[5] = {0, 0, 4, 2, 6};
            ih[12] = 8; ih[13] = ct[a.ch]; ih[14] = 0; ih[15] = 0; ih[16] = 0;
            put_be32(hp + 8, 13);
            for (int i = 0; i < 17; ++i) hp[12 + i] = ih[i];
            put_be32(hp + 29, ~crc_raw_bits(0xffffffffu, ih, 17));
            const long long total = png_offsets[j + 1] - png_offsets[j];
            put_be32(hp + 33, (unsigned)(total - 57));
            hp[37] = 'I'; hp[38] = 'D'; hp[39] = 'A'; hp[40] = 'T'; hp[41] = 0x78; hp[42] = 0x01;
        }
        if (rec.index == nb - 1 && threadIdx.x < 32) {
            const int lane = threadIdx.x;
            const long long per = (nb + 31) / 32;
            Fold f = {0u, 1u << 31, 0u, 0u, 0u};
            for (long long q = lane * per; q < min(nb, (lane + 1) * per); ++q) {
                const PngBlock& r = w.blocks[first + q];
                f = fold(f, Fold{r.crc, r.xpow, r.a, r.b, r.len % kAdler});
            }
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                Fold g;
                g.r = __shfl_down_sync(0xffffffffu, f.r, o); g.x = __shfl_down_sync(0xffffffffu, f.x, o);
                g.a = __shfl_down_sync(0xffffffffu, f.a, o); g.b = __shfl_down_sync(0xffffffffu, f.b, o);
                g.l = __shfl_down_sync(0xffffffffu, f.l, o);
                if ((lane & (2 * o - 1)) == 0 && lane + o < 32) f = fold(f, g);
            }
            if (lane == 0) {
                const unsigned char idat[6] = {'I', 'D', 'A', 'T', 0x78, 0x01};
                Fold hf = {crc_raw_bits(0u, idat, 6), x8n(6, x2n), 0u, 0u, 0u};
                f = fold(hf, f);
                const unsigned adler = (((f.l + f.b) % kAdler) << 16) | ((1 + f.a) % kAdler);
                unsigned char* tp = d + rec.seglen;
                tp[0] = 0x03; tp[1] = 0x00;
                put_be32(tp + 2, adler);
                Fold tf = {crc_raw_bits(0u, tp, 6), x8n(6, x2n), 0u, 0u, 0u};
                f = fold(f, tf);
                put_be32(tp + 6, ~(f.r ^ multmodp(f.x, 0xffffffffu)));
                const unsigned char iend[12] = {0, 0, 0, 0, 'I', 'E', 'N', 'D', 0xae, 0x42, 0x60, 0x82};
                for (int i = 0; i < 12; ++i) tp[10 + i] = iend[i];
            }
        }
    }
}

static size_t png_ws_bytes(long long S, long long packed, int c) {
    const long long ft = packed + (packed + c - 1) / c;
    const long long blocks = S + ft / kPngBlock;
    return (size_t)((S + 1 + 8) * 8 + blocks * (long long)sizeof(PngBlock) + ft + 32 * blocks + 64);
}

}  // namespace mb

using namespace mb;

extern "C" int64_t mb_png_bound_bytes(int64_t packed_bytes, int64_t crops, int32_t channels) {
    if (channels < 1 || channels > 4 || packed_bytes < 0 || crops < 0) return -1;
    const long long ft = packed_bytes + (packed_bytes + channels - 1) / channels;
    return 75 * crops + ft + 10 * (ft / kPngBlock);
}

extern "C" size_t mb_png_workspace_bytes(const mb_crop_params* p, int64_t packed_capacity_bytes, int32_t channels) {
    if (!p || channels < 1 || channels > 4 || packed_capacity_bytes < 0 || p->num_images < 1 || p->capacity < 1) return 0;
    return png_ws_bytes((long long)p->num_images * p->capacity, packed_capacity_bytes, channels);
}

extern "C" int mb_png_encode(const mb_crop_params* p, const uint8_t* packed, int32_t channels, const int32_t* rects,
                             const int64_t* offsets, const int64_t* totals, void* workspace, size_t workspace_bytes,
                             uint8_t* png_out, int64_t png_capacity_bytes, int64_t* png_offsets_out,
                             int64_t* png_status_out, mb_stream_t stream) {
    if (!p || !rects || !offsets || !totals || !workspace || !png_offsets_out || !png_status_out || png_capacity_bytes < 0)
        return MB_ERR_INVALID_ARG;
    if (channels < 1 || channels > 4 || p->channels < 1 || p->channels > 4) return MB_ERR_UNSUPPORTED;
    if (p->num_images < 1 || p->num_images > MB_MAX_IMAGES || p->capacity < 1) return MB_ERR_INVALID_ARG;
    if (png_capacity_bytes > 0 && !png_out) return MB_ERR_INVALID_ARG;
    const long long S = (long long)p->num_images * p->capacity;
    if (workspace_bytes < png_ws_bytes(S, 0, channels)) return MB_ERR_WORKSPACE;
    PngArgs a;
    a.packed = packed; a.rects = (const int4*)rects; a.offsets = (const long long*)offsets;
    a.src_ch = p->channels; a.ch = channels;
    const cudaStream_t st = (cudaStream_t)stream;
    k_png_plan<<<1, 1024, 0, st>>>(a, (const long long*)totals, workspace, workspace_bytes, S);
    MB_LAUNCH_CHECK();
    // the grids cover the most blocks the workspace can describe, capped at the persistent size
    const long long max_blocks = std::max<long long>(1, (long long)(workspace_bytes / (sizeof(PngBlock) + 16)));
    const size_t smem = sizeof(EncSmem);
    MB_DYN_SMEM(k_png_encode, smem);
    const int ge = (int)std::min<long long>(max_blocks, (long long)num_sms() * 3);
    k_png_encode<<<ge, kPngThreads, smem, st>>>(a, workspace, workspace_bytes, S);
    MB_LAUNCH_CHECK();
    k_png_layout<<<1, 1024, 0, st>>>(workspace, workspace_bytes, S, (long long*)png_offsets_out, (long long*)png_status_out,
                                     png_capacity_bytes);
    MB_LAUNCH_CHECK();
    const int ga = (int)std::min<long long>(max_blocks, (long long)num_sms() * 8);
    k_png_assemble<<<ga, 256, 0, st>>>(a, workspace, workspace_bytes, S, (const long long*)png_offsets_out,
                                       (const long long*)png_status_out, png_out);
    MB_LAUNCH_CHECK();
    return MB_OK;
}
