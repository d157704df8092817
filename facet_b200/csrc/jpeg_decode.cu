// Baseline JPEG decoding on the device: file bytes -> upright-agnostic [n][H][W][3] uint8 frames.
//
// Replaces the decode inside `load_image_from_path` (utils/image_loading.py:90-106 of the reference:
// `Image.open(path)` ... `.convert('RGB')` through Pillow / libjpeg-turbo, then `cv2.cvtColor(RGB2BGR)`), byte-exact:
//   restart scan      finds the RSTn markers of every stream (three small kernels: count, prefix, write)
//   huffman           one thread per restart interval (ITU T.81 F.2: DC prediction restarts with the interval, so
//                     intervals are independent); a stream without DRI is one interval, i.e. one thread — correct
//                     but serial: loaders that want the GPU rate write restart markers (Pillow: restart_marker_blocks)
//   idct              dequantise + jidctint.c `jpeg_idct_islow` (13-bit constants, 2 extra bits after pass 1, the
//                     10-bit wrap of libjpeg's range-limit table), one thread per 8x8 block
//   upsample+colour   jdsample.c h2v1 / h2v2 "fancy" (triangle) upsampling with replicated edges + jdcolor.c
//                     ycc_rgb_convert (16-bit fixed point), four pixels per thread, RGB or BGR order
// Host parsing of the marker segments and the table layout: facet_b200/utils/jpeg.py.
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"
#include "kernels.h"

namespace fb {

namespace {

constexpr int kLutBits = 9;
constexpr int kStagePitch = 66;                 // int16 per staging row of the entropy decoder: 33 words, so that equal
                                                // positions of the 32 rows of a warp fall into 32 different banks

struct JpegHuff {
    uint16_t lut[1 << kLutBits];      // (length << 8) | symbol for codes of <= 9 bits, else 0
    int32_t maxcode[18];              // largest code of each length (-1: none), [17] = sentinel
    int32_t valptr[17];               // symbol index = code + valptr[length]
    uint8_t values[256];
    uint8_t pad[4];
};
struct JpegTableSet {
    uint16_t q[4][64];                // natural (row-major) order
    JpegHuff dc[4], ac[4];
};
static_assert(sizeof(JpegHuff) == 1424 && sizeof(JpegTableSet) == 11904, "layout shared with facet_b200/utils/jpeg.py");

#define FB_HD __host__ __device__ __forceinline__

__device__ const uint8_t d_zigzag[64] = {0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20,
                                     13, 6, 7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59,
                                     52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
static const uint8_t h_zigzag[64] = {0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20,
                                     13, 6, 7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59,
                                     52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
struct BitReader {
    const uint8_t* p;
    const uint8_t* end;
    uint64_t acc;
    int n;
    uint32_t w0, w1, w2;    // the aligned words at and after p, loaded ahead of their use
};

// The four bytes at p (any alignment) come from the two aligned words around p.  Three consecutive aligned words are
// kept in registers, so the word a refill needs was requested TWO refills (eight stream bytes) earlier and every fast
// refill issues one load; up to 15 bytes past the end of a stream are read (stream buffers carry that slack).
FB_HD void prefetch_words(BitReader& br) {
#ifdef __CUDA_ARCH__
    const uint32_t* w = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(br.p) & ~(uintptr_t)3);
    br.w0 = w[0];
    br.w1 = w[1];
    br.w2 = w[2];
#endif
}
FB_HD uint32_t next_be32(const BitReader& br) {
#ifdef __CUDA_ARCH__
    const uint32_t le = __funnelshift_r(br.w0, br.w1, (uint32_t)(reinterpret_cast<uintptr_t>(br.p) & 3) * 8);
    return __byte_perm(le, 0u, 0x0123);
#else
    uint32_t w = 0;
    for (int i = 0; i < 4; ++i) w = (w << 8) | (br.p + i < br.end ? br.p[i] : 0u);
    return w;
#endif
}

// Top up to > 32 buffered bits.  Fast path: the next four bytes (zeros past the end of the interval, T.81 F.2.2.5) hold no
// 0xFF (true for ~98 % of the positions) and enter the buffer as one word.  Otherwise byte by byte: inside an interval the
// only 0xFF bytes are stuffed ones, followed by 0x00.
FB_HD void refill(BitReader& br) {
    if (br.n > 32) return;
    const long long rem = br.end - br.p;
    if (rem <= 0) {
        br.acc <<= 32;
        br.n += 32;
        return;
    }
    uint32_t w = next_be32(br);
    if (rem < 4) w &= 0xFFFFFFFFu << (8 * (4 - (int)rem));       // bytes past the end of the interval count as zeros
    const uint32_t x = ~w;                                       // a 0xFF byte of w is a zero byte of x
    if (!((x - 0x01010101u) & ~x & 0x80808080u)) {
        br.acc = (br.acc << 32) | w;
        br.n += 32;
        br.p += 4;
#ifdef __CUDA_ARCH__
        br.w0 = br.w1;
        br.w1 = br.w2;
        br.w2 = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(br.p) & ~(uintptr_t)3)[2];
#endif
        return;
    }
    while (br.n <= 32) {
        uint32_t b = 0;
        if (br.p < br.end) {
            b = *br.p++;
            if (b == 0xFF && br.p < br.end && *br.p == 0x00) ++br.p;
        }
        br.acc = (br.acc << 8) | b;
        br.n += 8;
    }
    prefetch_words(br);
}
template <class R>
FB_HD uint32_t peek(const R& br, int k) { return (uint32_t)(br.acc >> (br.n - k)) & ((1u << k) - 1u); }

// One Huffman symbol (>= 16 bits buffered).  Returns -1 for a code that is not in the table.
template <class R>
FB_HD int decode_symbol(R& br, const JpegHuff& h) {
    const uint32_t e = h.lut[peek(br, kLutBits)];
    if (e) {
        br.n -= (int)(e >> 8);
        return (int)(e & 255u);
    }
    const int code16 = (int)peek(br, 16);
#pragma unroll 1
    for (int len = kLutBits + 1; len <= 16; ++len) {
        const int code = code16 >> (16 - len);
        if (code <= h.maxcode[len]) {
            br.n -= len;
            return (int)h.values[(code + h.valptr[len]) & 255];
        }
    }
    return -1;
}
FB_HD int receive_extend(BitReader& br, int s) {       // F.2.2.1 / F.2.2.4, s >= 1
    const int v = (int)peek(br, s);
    br.n -= s;
    return v < (1 << (s - 1)) ? v - (1 << s) + 1 : v;
}

struct JpegGeom {
    int width, height, ncomp;
    int hs[3], vs[3], tq[3], td[3], ta[3];
    int restart_interval, mcux, mcuy, n_intervals;
    int blocks_w[3], blocks_h[3];                 // padded block grid per component
    long long coef_comp_off[3], coef_image_stride;   // in int16 elements
    long long plane_comp_off[3], plane_image_stride; // in bytes; planes are blocks_w*8 wide, blocks_h*8 high
};

// ---- restart scan ---------------------------------------------------------------------------------------------------
constexpr int kScanThreads = 256, kScanWarpBytes = 2048, kScanChunk = (kScanThreads / 32) * kScanWarpBytes;      // 16 KB per CTA

// 0x80 in every byte of x that is zero (exact, no carries between bytes)
__device__ __forceinline__ uint32_t zero_bytes(uint32_t x) {
    const uint32_t t = (x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu;
    return ~(t | x | 0x7F7F7F7Fu);
}

// RSTn markers among the stream positions p0 .. p0+7 (a marker at p = bytes 0xFF, 0xD0..0xD7 at p, p + 1, counted when p + 1 < len):
// bit 8 j + 7 of h[j / 4 ...] — returned as two words of 0x80 flags, byte i of (lo, hi) = position p0 + i.  Nine bytes come from the
// three aligned words around s + p0 (streams carry 15 bytes of slack behind their end); SIMD-in-word compares, no branches.
__device__ __forceinline__ void rst_flags8(const uint8_t* s, long long p0, long long len, uint32_t& lo, uint32_t& hi) {
    lo = hi = 0u;
    if (p0 + 1 >= len) return;
    const uintptr_t q = reinterpret_cast<uintptr_t>(s + p0);
    const uint32_t* a = reinterpret_cast<const uint32_t*>(q & ~(uintptr_t)3);
    const uint32_t sh = (uint32_t)(q & 3) * 8;
    const uint32_t w0 = __ldg(a), w1 = __ldg(a + 1), w2 = __ldg(a + 2);
    const uint32_t b0 = __funnelshift_r(w0, w1, sh), b1 = __funnelshift_r(w1, w2, sh);       // bytes 0..3, 4..7
    const uint32_t b8 = (w2 >> sh) & 0xFFu;                                                  // byte 8
    const uint32_t y0 = __funnelshift_r(b0, b1, 8), y1 = (b1 >> 8) | (b8 << 24);            // bytes 1..4, 5..8
    lo = zero_bytes(~b0) & zero_bytes((y0 & 0xF8F8F8F8u) ^ 0xD0D0D0D0u);
    hi = zero_bytes(~b1) & zero_bytes((y1 & 0xF8F8F8F8u) ^ 0xD0D0D0D0u);
    const long long valid = len - 1 - p0;                    // positions p0 + i with i < valid count
    if (valid < 8) {
        const int v = (int)valid;
        lo &= v >= 4 ? 0xFFFFFFFFu : ((1u << (8 * v)) - 1u);
        hi &= v <= 4 ? 0u : ((1u << (8 * (v - 4))) - 1u);
    }
}

// RSTn markers (0xFF 0xD0..0xD7) of one 16 KB chunk of one stream.  A warp walks its 2 KB in 256-byte steps, 8 positions per
// lane (rst_flags8); lane order = stream order.  WRITE = false: counts[img][chunk] = number of markers; WRITE = true
// (after the prefix kernel turned counts into exclusive offsets): starts[img][1 + k] = byte after the k-th marker.
template <bool WRITE>
__global__ void __launch_bounds__(kScanThreads) jpeg_restart_scan_kernel(const uint8_t* __restrict__ bytes, const long long* __restrict__ scan_off,
                                                                         const long long* __restrict__ scan_len, int chunks, int n_intervals,
                                                                         int* __restrict__ counts, uint32_t* __restrict__ starts) {
    __shared__ int s_warp[kScanThreads / 32];
    const int img = blockIdx.y, chunk = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint8_t* s = bytes + scan_off[img];
    const long long len = scan_len[img];
    const long long w0 = (long long)chunk * kScanChunk + (long long)warp * kScanWarpBytes;
    int cnt = 0;
    for (int it = 0; it < kScanWarpBytes / 256; ++it) {
        uint32_t lo, hi;
        rst_flags8(s, w0 + it * 256 + lane * 8, len, lo, hi);
        cnt += __popc(lo) + __popc(hi);
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) s_warp[warp] = cnt;
    __syncthreads();
    if (!WRITE) {
        if (tid == 0) {
            int tot = 0;
            for (int w = 0; w < kScanThreads / 32; ++w) tot += s_warp[w];
            counts[(size_t)img * chunks + chunk] = tot;
        }
        return;
    }
    int base = counts[(size_t)img * chunks + chunk];
    for (int w = 0; w < warp; ++w) base += s_warp[w];
    if (cnt == 0) return;
    uint32_t* out = starts + (size_t)img * n_intervals + 1;
    for (int it = 0; it < kScanWarpBytes / 256; ++it) {
        const long long p0 = w0 + it * 256 + lane * 8;
        uint32_t lo, hi;
        rst_flags8(s, p0, len, lo, hi);
        const int c = __popc(lo) + __popc(hi);
        if (!__any_sync(0xffffffffu, c != 0)) continue;
        int incl = c;                                        // inclusive prefix of the lanes' counts
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int x = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += x;
        }
        int k = base + incl - c;
        for (uint32_t m = lo; m; m &= m - 1, ++k)
            if (k < n_intervals - 1) out[k] = (uint32_t)(p0 + (__ffs(m) >> 3) + 1);          // flag bit 8 i + 7 -> position p0 + i, + 2
        for (uint32_t m = hi; m; m &= m - 1, ++k)
            if (k < n_intervals - 1) out[k] = (uint32_t)(p0 + 4 + (__ffs(m) >> 3) + 1);
        base += __shfl_sync(0xffffffffu, incl, 31);
    }
}

// exclusive prefix of the per-chunk counts of one image; status[img] |= 1 when the number of markers is not n_intervals - 1
__global__ void __launch_bounds__(256) jpeg_restart_prefix_kernel(int* __restrict__ counts, int chunks, int n_intervals,
                                                                  uint32_t* __restrict__ starts, int* __restrict__ status) {
    __shared__ int s_part[256];
    const int img = blockIdx.x, tid = threadIdx.x;
    int* c = counts + (size_t)img * chunks;
    const int per = (chunks + 255) / 256;
    const int lo = min(tid * per, chunks), hi = min(lo + per, chunks);
    int sum = 0;
    for (int i = lo; i < hi; ++i) sum += c[i];
    s_part[tid] = sum;
    __syncthreads();
    for (int o = 1; o < 256; o <<= 1) {
        const int v = tid >= o ? s_part[tid - o] : 0;
        __syncthreads();
        s_part[tid] += v;
        __syncthreads();
    }
    int run = s_part[tid] - sum;
    for (int i = lo; i < hi; ++i) {
        const int v = c[i];
        c[i] = run;
        run += v;
    }
    if (tid == 255) {
        if (s_part[255] != n_intervals - 1) atomicOr(status + img, 1);
        starts[(size_t)img * n_intervals] = 0u;
    }
}

// Blocks of one MCU in scan order, 4 bits each: component (2 bits), block row and column inside the MCU (1 bit each; the
// supported sampling factors are 1 or 2).  At most 2*2 + 1 + 1 = 6 blocks.
FB_HD uint64_t mcu_layout(const JpegGeom& g, int& nblk) {
    uint64_t lay = 0;
    nblk = 0;
    for (int c = 0; c < g.ncomp; ++c)
        for (int by = 0; by < g.vs[c]; ++by)
            for (int bx = 0; bx < g.hs[c]; ++bx) {
                lay |= (uint64_t)(c | (by << 2) | (bx << 3)) << (4 * nblk);
                ++nblk;
            }
    return lay;
}

// Entropy decoding of restart interval `iv` of one stream: bytes [p0, p1) hold its MCUs (no marker inside); `zz` is the
// zigzag table.  The loop decodes ONE symbol per iteration whatever it is (DC size, AC run/size, EOB, ZRL): table, destination
// and state update are chosen by selects, so the lanes of a warp — each in its own interval — stay on the same instructions.
//
// COOP = true (the kernel): quantised coefficients go out in natural order one whole 8x8 block (128 bytes, zeros included) at
// a time.  A lane assembles its block in `stage_row` — 64 int16 of shared memory — and when it is complete the WHOLE WARP
// copies it: 32 lanes x 4 bytes = one coalesced 128-byte store per block (the rows of all lanes start at `stage_warp`, pitch
// kStagePitch).  Measured alternatives: 2-byte stores scattered into a pre-zeroed area cost 44 % of the kernel in L2
// read-modify-write traffic (plus the memset); per-lane 16-byte copies of the staged block were slower still (32 partial lines
// per store instruction).  Every lane of the warp must call this (inactive ones with active = false).
// COOP = false (the host test tool): coefficients are stored directly into a pre-zeroed area.
// Returns false on invalid Huffman data.
template <bool COOP>
FB_HD bool decode_interval(const uint8_t* p0, const uint8_t* p1, int iv, const JpegGeom& g, const JpegTableSet& T, const uint8_t* zz,
                           int16_t* cimg, bool active, int16_t* stage_warp, int lane) {
    BitReader br;
    br.p = p0;
    br.end = p1;
    br.acc = 0;
    br.n = 0;
    br.w0 = br.w1 = br.w2 = 0;
    const int total_mcus = g.mcux * g.mcuy;
    int m = g.restart_interval ? iv * g.restart_interval : 0;
    const int m1 = g.restart_interval ? (m + g.restart_interval < total_mcus ? m + g.restart_interval : total_mcus) : total_mcus;
    bool done = !active || m >= m1, ok = true;
    if (!done) prefetch_words(br);
    int nblk;
    const uint64_t lay = mcu_layout(g, nblk);
    int my = done ? 0 : m / g.mcux, mx = done ? 0 : m - my * g.mcux;
    int b = 0, k = 0;
    int pred0 = 0, pred1 = 0, pred2 = 0;
    auto block_ptr = [&](int bi, int& c) -> int16_t* {
        const int e = (int)(lay >> (4 * bi)) & 15;
        c = e & 3;
        const int row = my * g.vs[c] + ((e >> 2) & 1), col = mx * g.hs[c] + ((e >> 3) & 1);
        return cimg + g.coef_comp_off[c] + ((size_t)row * g.blocks_w[c] + col) * 64;
    };
    int c;
    int16_t* blk = block_ptr(0, c);
    int16_t* const stage_row = COOP ? stage_warp + lane * kStagePitch : nullptr;
    const JpegHuff* hd = &T.dc[g.td[c]];
    const JpegHuff* ha = &T.ac[g.ta[c]];
    for (;;) {
#ifdef __CUDA_ARCH__
        if (COOP) {
            if (!__any_sync(0xffffffffu, !done)) break;
        } else
#endif
        if (done) break;
        int16_t* flush_blk = nullptr;
        if (!done) {
            refill(br);
            const bool isdc = k == 0;
            const int sym = decode_symbol(br, isdc ? *hd : *ha);
            const int run = isdc ? 0 : sym >> 4;
            const int size = isdc ? sym : (sym & 15);
            if (sym < 0 || size > (isdc ? 11 : 15)) {
                ok = false;
                done = true;
            } else {
                int val = 0;
                if (size) {
                    const int v = (int)peek(br, size);
                    br.n -= size;
                    val = v < (1 << (size - 1)) ? v - (1 << size) + 1 : v;
                }
                int pos = 0, store = val;
                if (isdc) {
                    const int pr = (c == 0 ? pred0 : (c == 1 ? pred1 : pred2)) + val;
                    pred0 = c == 0 ? pr : pred0;
                    pred1 = c == 1 ? pr : pred1;
                    pred2 = c == 2 ? pr : pred2;
                    store = pr;
                    k = 1;
                } else if (size == 0) {
                    k = run == 15 ? k + 16 : 64;              // ZRL : EOB
                } else {
                    k += run;
                    if (k > 63) {
                        ok = false;
                        done = true;
                        k = 63;
                    }
                    pos = zz[k];
                    ++k;
                }
                if (store && ok) (COOP ? stage_row : blk)[pos] = (int16_t)store;
                if (k >= 64 && ok) {                          // block complete: next block (next MCU after the last block of this one)
                    flush_blk = blk;
                    k = 0;
                    if (++b == nblk) {
                        b = 0;
                        if (++m == m1) done = true;
                        if (++mx == g.mcux) {
                            mx = 0;
                            ++my;
                        }
                    }
                    if (!done) {
                        blk = block_ptr(b, c);
                        hd = &T.dc[g.td[c]];
                        ha = &T.ac[g.ta[c]];
                    }
                }
            }
        }
#ifdef __CUDA_ARCH__
        if (COOP) {
            // every completed block of the warp leaves as one 128-byte store; the copying lanes clear the row behind them
            unsigned mask = __ballot_sync(0xffffffffu, flush_blk != nullptr);
            while (mask) {
                const int src = __ffs(mask) - 1;
                mask &= mask - 1;
                uint32_t* dst = reinterpret_cast<uint32_t*>(__shfl_sync(0xffffffffu, reinterpret_cast<unsigned long long>(flush_blk), src));
                uint32_t* row = reinterpret_cast<uint32_t*>(stage_warp + src * kStagePitch);
                dst[lane] = row[lane];
                row[lane] = 0u;
            }
            __syncwarp();
        }
#endif
    }
    return ok;
}

// ---- entropy decoding -----------------------------------------------------------------------------------------------
constexpr int kHuffThreads = 256;
constexpr int kHuffSmem = (int)sizeof(JpegTableSet) + kHuffThreads * kStagePitch * 2;

__global__ void __launch_bounds__(kHuffThreads) jpeg_huffman_kernel(const uint8_t* __restrict__ bytes, const long long* __restrict__ scan_off,
                                                                    const long long* __restrict__ scan_len, const int* __restrict__ table_slot,
                                                                    const JpegTableSet* __restrict__ tables, const uint32_t* __restrict__ starts,
                                                                    JpegGeom g, int16_t* __restrict__ coef, int* __restrict__ status) {
    extern __shared__ __align__(16) uint8_t s_raw[];
    __shared__ uint8_t s_zz[64];
    JpegTableSet* T = reinterpret_cast<JpegTableSet*>(s_raw);
    const int img = blockIdx.y, tid = threadIdx.x;
    if (tid < 64) s_zz[tid] = d_zigzag[tid];
    {
        const uint4* src = reinterpret_cast<const uint4*>(tables + table_slot[img]);
        uint4* dst = reinterpret_cast<uint4*>(s_raw);
        for (int i = tid; i < (int)(sizeof(JpegTableSet) / 16); i += kHuffThreads) dst[i] = src[i];
    }
    __syncthreads();
    const int iv = blockIdx.x * kHuffThreads + tid;
    const bool active = iv < g.n_intervals && !(status[img] & 1);     // bit 0: restart markers do not match the header
    const uint8_t* s = bytes + scan_off[img];
    const long long len = scan_len[img];
    const uint32_t* st = starts + (size_t)img * g.n_intervals;
    const uint8_t* p0 = active ? s + st[iv] : s;
    const uint8_t* p1 = active ? ((iv + 1 < g.n_intervals) ? s + st[iv + 1] - 2 : s + len) : s;     // up to the next RSTn marker
    // staging rows of this warp (zeroed; the cooperative copy clears them again)
    int16_t* stage_warp = reinterpret_cast<int16_t*>(s_raw + sizeof(JpegTableSet)) + (tid & ~31) * kStagePitch;
    for (int i = tid & 31; i < 32 * kStagePitch / 2; i += 32) reinterpret_cast<uint32_t*>(stage_warp)[i] = 0u;
    __syncwarp();
    const bool bad = !decode_interval<true>(p0, p1, active ? iv : 0, g, *T, s_zz, coef + (size_t)img * g.coef_image_stride, active,
                                            stage_warp, tid & 31);
    if (bad) atomicOr(status + img, 2);
}

// ---- streams WITHOUT restart markers: self-synchronising parallel entropy decoding ---------------------------------------
// DC prediction and the position inside the MCU chain every symbol of such a stream to its predecessors, but Huffman streams
// SELF-SYNCHRONISE: a decoder started at a wrong bit / in a wrong state falls into step with the true symbol sequence after a
// few dozen symbols.  Scheme (after Weissenberger & Schmidt, "Massively Parallel Huffman Decoding on GPUs"):
//   1. the stuffed zero bytes are removed (jpeg_unstuff_*), so that positions are plain bit indices;
//   2. the clean stream is cut into subsequences of kSubseqBytes; thread t decodes subsequence t from a guessed state and
//      records the state at the first symbol boundary at or after the end of its subsequence (jpeg_sync_kernel, round 0);
//   3. rounds: thread t decodes again, now from the end state thread t-1 recorded; a round that changes nothing means every
//      thread started from the true state (thread 0 always does; the truth advances at least one subsequence per round, and in
//      practice everywhere within two or three rounds because of the self-synchronisation);
//   4. a prefix sum over the blocks completed per subsequence gives every thread its first block index; a last pass decodes once
//      more and stores coefficients, the DC ones as DIFFERENCES — also into a compact array, 2 bytes per block in scan order
//      (jpeg_sync_write_kernel);
//   5. a prefix sum per component over the compact array turns the differences into DC values (jpeg_dcx_segment_kernel), which
//      the inverse DCT reads instead of coefficient 0.
#ifndef FB_SUBSEQ_BYTES
#define FB_SUBSEQ_BYTES 512
#endif
constexpr int kSubseqBytes = FB_SUBSEQ_BYTES;
#ifndef FB_SYNC_ROUNDS
#define FB_SYNC_ROUNDS 24
#endif
constexpr int kSyncRounds = FB_SYNC_ROUNDS;           // rounds after round 0; a stream that still changes then is reported (status bit 2)

struct SyncState {
    long long pos;       // bit position in the clean stream (a symbol boundary)
    int b, k;            // block inside the MCU, coefficient index (0 = the DC symbol comes next)
};

struct CleanReader {
    const uint8_t* u;    // clean stream (256-byte aligned); at least 16 zero bytes follow its end
    long long next;      // next byte to load
    uint64_t acc;
    int n;
    uint32_t w0, w1, w2; // device: the aligned words at and after `next`, requested ahead of their use
};
FB_HD void cr_prefetch(CleanReader& r) {
#ifdef __CUDA_ARCH__
    const uint32_t* w = reinterpret_cast<const uint32_t*>(r.u + (r.next & ~3ll));
    r.w0 = w[0];
    r.w1 = w[1];
    r.w2 = w[2];
#endif
}
FB_HD void cr_seek(CleanReader& r, long long pos_bits) {
    r.next = pos_bits >> 3;
    r.acc = 0;
    r.n = 0;
    const int skip = (int)(pos_bits & 7);
    if (skip) {
        r.acc = r.u[r.next++] & (0xFFu >> skip);
        r.n = 8 - skip;
    }
    r.w0 = r.w1 = r.w2 = 0;
    cr_prefetch(r);
}
// no stuffing in a clean stream: whenever 32 bits fit, the next four bytes enter as one word
FB_HD void cr_refill(CleanReader& r) {
    if (r.n > 32) return;
#ifdef __CUDA_ARCH__
    const uint32_t le = __funnelshift_r(r.w0, r.w1, (uint32_t)(r.next & 3) * 8);
    const uint32_t w = __byte_perm(le, 0u, 0x0123);
    r.next += 4;
    r.w0 = r.w1;
    r.w1 = r.w2;
    r.w2 = reinterpret_cast<const uint32_t*>(r.u + (r.next & ~3ll))[2];
#else
    const uint32_t w = ((uint32_t)r.u[r.next] << 24) | ((uint32_t)r.u[r.next + 1] << 16) | ((uint32_t)r.u[r.next + 2] << 8) | (uint32_t)r.u[r.next + 3];
    r.next += 4;
#endif
    r.acc = (r.acc << 32) | w;
    r.n += 32;
}
FB_HD long long cr_pos(const CleanReader& r) { return 8 * r.next - r.n; }

// Coefficient area address of block number q of the scan (MCU by MCU, blocks of an MCU in `lay` order).
FB_HD int16_t* scan_block_ptr(int q, const JpegGeom& g, uint64_t lay, int nblk, int16_t* cimg) {
    const int m = q / nblk, bi = q - m * nblk;
    const int e = (int)(lay >> (4 * bi)) & 15, c = e & 3;
    const int my = m / g.mcux, mx = m - my * g.mcux;
    const int row = my * g.vs[c] + ((e >> 2) & 1), col = mx * g.hs[c] + ((e >> 3) & 1);
    return cimg + g.coef_comp_off[c] + ((size_t)row * g.blocks_w[c] + col) * 64;
}

// The inverse: index in scan order of the block at (brow, bcol) of component c's block grid.
FB_HD long long scan_index_of_block(const JpegGeom& g, int c, int brow, int bcol) {
    int nblk = 0, first = 0;
    for (int cc = 0; cc < g.ncomp; ++cc) {
        if (cc == c) first = nblk;
        nblk += g.hs[cc] * g.vs[cc];
    }
    const int my = brow / g.vs[c], by = brow - my * g.vs[c], mx = bcol / g.hs[c], bx = bcol - mx * g.hs[c];
    return ((long long)my * g.mcux + mx) * nblk + first + by * g.hs[c] + bx;
}

// Decode from state `st` up to the first symbol boundary at or after `limit_bits` (or the end of the data).
// WRITE = false: only the state evolves (garbage from a wrong start state is tolerated: an invalid code skips one bit, an
// overlong run ends the block).  WRITE = true: the start state is the true one; non-zero coefficients are stored into the
// pre-zeroed coefficient area (DC as the decoded difference), block q is the first one touched; returns false on invalid data.
template <bool WRITE>
FB_HD bool span_decode(const uint8_t* u, long long len_bits, SyncState st, long long limit_bits, const JpegGeom& g, const JpegTableSet& T,
                       const uint8_t* zz, uint64_t lay, int nblk, SyncState& out, int& blocks_done, int q, int total_blocks, int16_t* cimg) {
    CleanReader r;
    r.u = u;
    cr_seek(r, st.pos);
    int b = st.b, k = st.k;
    blocks_done = 0;
    bool ok = true;
    int c = (int)(lay >> (4 * b)) & 3;
    const JpegHuff* hd = &T.dc[g.td[c]];
    const JpegHuff* ha = &T.ac[g.ta[c]];
    int16_t* blk = (WRITE && q < total_blocks) ? scan_block_ptr(q, g, lay, nblk, cimg) : nullptr;
    for (;;) {
        const long long pos = cr_pos(r);
        if (pos >= limit_bits || pos >= len_bits) break;
        if (WRITE && q >= total_blocks) break;
        cr_refill(r);
        const bool isdc = k == 0;
        const int sym = decode_symbol(r, isdc ? *hd : *ha);
        if (sym < 0) {
            if (WRITE) {
                ok = false;
                break;
            }
            r.n -= 1;
            continue;
        }
        const int run = isdc ? 0 : sym >> 4;
        const int size = isdc ? (sym & 15) : (sym & 15);
        int val = 0;
        if (size) {
            const int v = (int)peek(r, size);
            r.n -= size;
            val = v < (1 << (size - 1)) ? v - (1 << size) + 1 : v;
        }
        if (isdc) {
            if (WRITE && val) blk[0] = (int16_t)val;
            k = 1;
        } else if (size == 0) {
            k = run == 15 ? k + 16 : 64;
        } else {
            k += run;
            if (k > 63) {
                if (WRITE) {
                    ok = false;
                    break;
                }
                k = 64;
            } else {
                if (WRITE) blk[zz[k]] = (int16_t)val;
                ++k;
            }
        }
        if (k >= 64) {
            k = 0;
            ++blocks_done;
            b = b + 1 == nblk ? 0 : b + 1;
            c = (int)(lay >> (4 * b)) & 3;
            hd = &T.dc[g.td[c]];
            ha = &T.ac[g.ta[c]];
            if (WRITE) {
                ++q;
                if (q < total_blocks) blk = scan_block_ptr(q, g, lay, nblk, cimg);
            }
        }
    }
    out.pos = cr_pos(r);
    out.b = b;
    out.k = k;
    return ok;
}

#ifndef FB_JPEG_HOST_TEST
// stuffed zeros (0xFF 0x00) of one 16 KB chunk.  A warp walks its 2 KB in 32-byte steps (coalesced byte loads); ballots keep
// the bytes in order.  WRITE = false counts the stuffed zeros; WRITE = true copies every other byte to its position in the
// clean stream (counts then holds the exclusive prefix of the per-chunk counts).
template <bool WRITE>
__global__ void __launch_bounds__(kScanThreads) jpeg_unstuff_kernel(const uint8_t* __restrict__ bytes, const long long* __restrict__ scan_off,
                                                                    const long long* __restrict__ scan_len, int chunks, int* __restrict__ counts,
                                                                    uint8_t* __restrict__ clean, long long clean_stride) {
    __shared__ int s_warp[kScanThreads / 32];
    const int img = blockIdx.y, chunk = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint8_t* s = bytes + scan_off[img];
    const long long len = scan_len[img];
    const long long w0 = (long long)chunk * kScanChunk + (long long)warp * kScanWarpBytes;
    // the count (both passes need it per warp): 8 positions per lane from three aligned words, SIMD-in-word compares as in rst_flags8
    int cnt = 0;
    for (int it = 0; it < kScanWarpBytes / 256; ++it) {
        const long long p0 = w0 + it * 256 + lane * 8;
        if (p0 >= len) continue;
        const uintptr_t q = reinterpret_cast<uintptr_t>(s + p0) - 1;                      // byte p0 - 1 (p0 = 0: the last header byte, masked below)
        const uint32_t* a = reinterpret_cast<const uint32_t*>(q & ~(uintptr_t)3);
        const uint32_t sh = (uint32_t)(q & 3) * 8;
        const uint32_t x0 = __ldg(a), x1 = __ldg(a + 1), x2 = __ldg(a + 2);
        const uint32_t b0 = __funnelshift_r(x0, x1, sh), b1 = __funnelshift_r(x1, x2, sh);  // bytes p0-1 .. p0+2, p0+3 .. p0+6
        const uint32_t b8 = (x2 >> sh) & 0xFFu;                                              // byte p0+7
        const uint32_t y0 = __funnelshift_r(b0, b1, 8), y1 = (b1 >> 8) | (b8 << 24);        // bytes p0 .. p0+3, p0+4 .. p0+7
        uint32_t lo = zero_bytes(~b0) & zero_bytes(y0), hi = zero_bytes(~b1) & zero_bytes(y1);   // flag byte i: position p0 + i is a stuffed zero
        if (p0 == 0) lo &= ~0xFFu;
        const long long valid = len - p0;
        if (valid < 8) {
            const int v = (int)valid;
            lo &= v >= 4 ? 0xFFFFFFFFu : ((1u << (8 * v)) - 1u);
            hi &= v <= 4 ? 0u : ((1u << (8 * (v - 4))) - 1u);
        }
        cnt += __popc(lo) + __popc(hi);
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) s_warp[warp] = cnt;
    __syncthreads();
    if (!WRITE) {
        if (tid == 0) {
            int tot = 0;
            for (int w = 0; w < kScanThreads / 32; ++w) tot += s_warp[w];
            counts[(size_t)img * chunks + chunk] = tot;
        }
        return;
    }
    long long removed = counts[(size_t)img * chunks + chunk];
    for (int w = 0; w < warp; ++w) removed += s_warp[w];
    uint8_t* out = clean + (size_t)img * clean_stride;
    for (int it = 0; it < kScanWarpBytes / 32; ++it) {
        const long long p = w0 + it * 32 + lane;
        const bool in = p < len;
        const uint8_t v = in ? s[p] : 0;
        const bool stuffed = in && p > 0 && v == 0x00 && s[p - 1] == 0xFF;
        const uint32_t m = __ballot_sync(0xffffffffu, stuffed);
        if (in && !stuffed) out[p - removed - __popc(m & ((1u << lane) - 1u))] = v;
        removed += __popc(m);
    }
}

// exclusive prefix of the per-chunk counts of one image; clean_len[img] = scan_len - number of stuffed zeros
__global__ void __launch_bounds__(256) jpeg_unstuff_prefix_kernel(int* __restrict__ counts, int chunks, const long long* __restrict__ scan_len,
                                                                  long long* __restrict__ clean_len) {
    __shared__ int s_part[256];
    const int img = blockIdx.x, tid = threadIdx.x;
    int* c = counts + (size_t)img * chunks;
    const int per = (chunks + 255) / 256;
    const int lo = min(tid * per, chunks), hi = min(lo + per, chunks);
    int sum = 0;
    for (int i = lo; i < hi; ++i) sum += c[i];
    s_part[tid] = sum;
    __syncthreads();
    for (int o = 1; o < 256; o <<= 1) {
        const int v = tid >= o ? s_part[tid - o] : 0;
        __syncthreads();
        s_part[tid] += v;
        __syncthreads();
    }
    int run = s_part[tid] - sum;
    for (int i = lo; i < hi; ++i) {
        const int v = c[i];
        c[i] = run;
        run += v;
    }
    if (tid == 255) clean_len[img] = scan_len[img] - s_part[255];
}

struct SyncArrays {
    SyncState* state[3];     // [n][T], rotating over the rounds: state at the end of every subsequence
    int* blocks;             // [n][T] blocks completed inside the subsequence
    int* first_block;        // [n][T] exclusive prefix of `blocks`
    int* changed;            // [n][kSyncRounds + 1]
    int* settled;            // [n]: 0, or 1 + the round that changed nothing (its states are the true ones)
    const long long* clean_len;
    const uint8_t* clean;
    long long clean_stride;
    int T;
    int16_t* dc;             // [n][blocks per image] DC differences / values in scan order (compact DC integration)
    long long dc_image_stride;
};

// round 0: every thread starts at the first bit of its subsequence in the guessed state (block 0, DC next) — true for thread 0.
// round r >= 1: thread t starts from what thread t-1 recorded in round r-1; skipped (states copied) once a round changed nothing.
__global__ void __launch_bounds__(128) jpeg_sync_kernel(SyncArrays A, const int* __restrict__ table_slot, const JpegTableSet* __restrict__ tables,
                                                        JpegGeom g, int round) {
    __shared__ __align__(16) uint8_t s_tab[sizeof(JpegTableSet)];
    __shared__ uint8_t s_zz[64];
    const int img = blockIdx.y, tid = threadIdx.x;
    {
        const uint4* src = reinterpret_cast<const uint4*>(tables + table_slot[img]);
        for (int i = tid; i < (int)(sizeof(JpegTableSet) / 16); i += blockDim.x) reinterpret_cast<uint4*>(s_tab)[i] = src[i];
        if (tid < 64) s_zz[tid] = d_zigzag[tid];
    }
    __syncthreads();
    const JpegTableSet& T = *reinterpret_cast<const JpegTableSet*>(s_tab);
    const int t = blockIdx.x * blockDim.x + tid;
    if (t >= A.T) return;
    const long long len_bits = 8 * A.clean_len[img];
    const SyncState* prev = A.state[(round + 2) % 3] + (size_t)img * A.T;        // round - 1
    const SyncState* prev2 = A.state[(round + 1) % 3] + (size_t)img * A.T;       // round - 2
    SyncState* cur = A.state[round % 3] + (size_t)img * A.T;
    if (round >= 2 && A.settled[img]) return;          // the whole stream is already stable: its final states stay where they are
    if (round >= 2 && t >= 1) {
        // same start state as in the previous round -> same result (only the front of corrections is decoded again)
        const SyncState a = prev[t - 1], b2 = prev2[t - 1];
        if (a.pos == b2.pos && a.b == b2.b && a.k == b2.k) {
            cur[t] = prev[t];
            return;
        }
    }
    if (round >= 1 && t == 0) {
        cur[0] = prev[0];
        return;
    }
    const long long start = (long long)t * kSubseqBytes * 8, limit = start + (long long)kSubseqBytes * 8;
    SyncState st;
    if (start >= len_bits) {
        st.pos = len_bits;
        st.b = st.k = 0;
        cur[t] = st;
        A.blocks[(size_t)img * A.T + t] = 0;
        return;
    }
    if (round == 0 || t == 0) {
        st.pos = start;
        st.b = st.k = 0;
    } else {
        st = prev[t - 1];
    }
    int nblk, done;
    const uint64_t lay = mcu_layout(g, nblk);
    SyncState out;
    span_decode<false>(A.clean + (size_t)img * A.clean_stride, len_bits, st, limit, g, T, s_zz, lay, nblk, out, done, 0, 0, nullptr);
    if (round >= 1) {
        const SyncState old = prev[t];
        if (old.pos != out.pos || old.b != out.b || old.k != out.k) atomicOr(A.changed + img * (kSyncRounds + 1) + round, 1);
    }
    cur[t] = out;
    A.blocks[(size_t)img * A.T + t] = done;
}

// after round r >= 1: a round that changed nothing settles the stream; settled[img] = r + 1 (0 = not yet)
__global__ void jpeg_sync_settle_kernel(SyncArrays A, int n, int round) {
    const int img = blockIdx.x * blockDim.x + threadIdx.x;
    if (img < n && A.settled[img] == 0 && A.changed[img * (kSyncRounds + 1) + round] == 0) A.settled[img] = round + 1;
}

// first_block[t] = number of blocks completed before subsequence t; status bit 2 when the rounds did not settle, bit 1 when the
// stream holds fewer blocks than the frame needs
__global__ void __launch_bounds__(1024) jpeg_sync_prefix_kernel(SyncArrays A, int total_blocks, int* __restrict__ status) {
    __shared__ int s_part[1024];
    const int img = blockIdx.x, tid = threadIdx.x;
    const int* nb = A.blocks + (size_t)img * A.T;
    int* fb = A.first_block + (size_t)img * A.T;
    const int per = (A.T + 1023) / 1024;
    const int lo = min(tid * per, A.T), hi = min(lo + per, A.T);
    int sum = 0;
    for (int i = lo; i < hi; ++i) sum += nb[i];
    s_part[tid] = sum;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        const int v = tid >= o ? s_part[tid - o] : 0;
        __syncthreads();
        s_part[tid] += v;
        __syncthreads();
    }
    int run = s_part[tid] - sum;
    for (int i = lo; i < hi; ++i) {
        fb[i] = run;
        run += nb[i];
    }
    if (tid == 1023) {
        if (s_part[1023] < total_blocks) atomicOr(status + img, 2);
        if (A.settled[img] == 0) atomicOr(status + img, 4);
    }
}

// Write pass.  A thread owns the blocks that START between its start state and the next thread's: it decodes (without storing)
// the block that was already in progress at its start state — that one belongs to its predecessor — and runs past the end of its
// subsequence until the block in progress there is complete.  So every block is assembled by ONE lane, in a shared-memory row,
// and leaves as ONE coalesced 128-byte store by the whole warp like in jpeg_huffman_kernel: no memset of the coefficient area,
// no 2-byte read-modify-write stores (they made this pass 3.3x as long as the same decode without stores).  DC coefficients
// are stored as differences.  `q` = number of blocks completed before the start state (jpeg_sync_prefix_kernel).
__device__ bool span_write_coop(const uint8_t* u, long long len_bits, SyncState st, long long limit_bits, bool active, const JpegGeom& g,
                                const JpegTableSet& T, const uint8_t* zz, uint64_t lay, int nblk, int q, int total_blocks, int16_t* cimg,
                                int16_t* stage_warp, int lane, int16_t* dc_img) {
    CleanReader r;
    r.u = u;
    r.next = 0;
    r.acc = 0;
    r.n = 0;
    r.w0 = r.w1 = r.w2 = 0;
    bool done = !active || q >= total_blocks, ok = true;
    if (!done) cr_seek(r, st.pos);
    int b = st.b, k = st.k;
    bool skip = k > 0;                                   // the block in progress at the start state is the predecessor's
    int c = (int)(lay >> (4 * b)) & 3;
    const JpegHuff* hd = &T.dc[g.td[c]];
    const JpegHuff* ha = &T.ac[g.ta[c]];
    int16_t* blk = done ? nullptr : scan_block_ptr(q, g, lay, nblk, cimg);
    int16_t* const stage_row = stage_warp + lane * kStagePitch;
    for (;;) {
        if (!__any_sync(0xffffffffu, !done)) break;
        int16_t* flush_blk = nullptr;
        if (!done) {
            const long long pos = cr_pos(r);
            if ((k == 0 && pos >= limit_bits) || pos >= len_bits) {
                done = true;                             // the next block starts in the next thread's span / end of the data
            } else {
                cr_refill(r);
                const bool isdc = k == 0;
                const int sym = decode_symbol(r, isdc ? *hd : *ha);
                if (sym < 0) {
                    ok = false;
                    done = true;
                } else {
                    const int run = isdc ? 0 : sym >> 4;
                    const int size = sym & 15;
                    int val = 0;
                    if (size) {
                        const int v = (int)peek(r, size);
                        r.n -= size;
                        val = v < (1 << (size - 1)) ? v - (1 << size) + 1 : v;
                    }
                    if (isdc) {
                        if (!skip && val) stage_row[0] = (int16_t)val;
                        k = 1;
                    } else if (size == 0) {
                        k = run == 15 ? k + 16 : 64;
                    } else {
                        k += run;
                        if (k > 63) {
                            ok = false;
                            done = true;
                        } else {
                            if (!skip) stage_row[zz[k]] = (int16_t)val;
                            ++k;
                        }
                    }
                    if (k >= 64 && ok) {
                        k = 0;
                        if (!skip) {
                            flush_blk = blk;
                            dc_img[q] = stage_row[0];                    // compact copy of the DC difference, scan order
                        }
                        skip = false;
                        b = b + 1 == nblk ? 0 : b + 1;
                        c = (int)(lay >> (4 * b)) & 3;
                        hd = &T.dc[g.td[c]];
                        ha = &T.ac[g.ta[c]];
                        if (++q < total_blocks) blk = scan_block_ptr(q, g, lay, nblk, cimg);
                        else done = true;
                    }
                }
            }
        }
        // every completed block of the warp leaves as one 128-byte store; the copying lanes clear the row behind them
        unsigned mask = __ballot_sync(0xffffffffu, flush_blk != nullptr);
        while (mask) {
            const int src = __ffs(mask) - 1;
            mask &= mask - 1;
            uint32_t* dst = reinterpret_cast<uint32_t*>(__shfl_sync(0xffffffffu, reinterpret_cast<unsigned long long>(flush_blk), src));
            uint32_t* row = reinterpret_cast<uint32_t*>(stage_warp + src * kStagePitch);
            dst[lane] = row[lane];
            row[lane] = 0u;
        }
        __syncwarp();
    }
    return ok;
}

constexpr int kSyncWriteThreads = 128;
constexpr int kSyncWriteSmem = (int)sizeof(JpegTableSet) + kSyncWriteThreads * kStagePitch * 2;

__global__ void __launch_bounds__(kSyncWriteThreads) jpeg_sync_write_kernel(SyncArrays A, const int* __restrict__ table_slot,
                                                                            const JpegTableSet* __restrict__ tables, JpegGeom g, int total_blocks,
                                                                            int16_t* __restrict__ coef, int* __restrict__ status) {
    extern __shared__ __align__(16) uint8_t s_raw[];
    __shared__ uint8_t s_zz[64];
    const int img = blockIdx.y, tid = threadIdx.x;
    {
        const uint4* src = reinterpret_cast<const uint4*>(tables + table_slot[img]);
        for (int i = tid; i < (int)(sizeof(JpegTableSet) / 16); i += blockDim.x) reinterpret_cast<uint4*>(s_raw)[i] = src[i];
        if (tid < 64) s_zz[tid] = d_zigzag[tid];
    }
    int16_t* stage_warp = reinterpret_cast<int16_t*>(s_raw + sizeof(JpegTableSet)) + (tid & ~31) * kStagePitch;
    for (int i = tid & 31; i < 32 * kStagePitch / 2; i += 32) reinterpret_cast<uint32_t*>(stage_warp)[i] = 0u;
    __syncthreads();
    const JpegTableSet& T = *reinterpret_cast<const JpegTableSet*>(s_raw);
    const int t = blockIdx.x * blockDim.x + tid;
    const long long len_bits = 8 * A.clean_len[img];
    const long long start = (long long)t * kSubseqBytes * 8, limit = start + (long long)kSubseqBytes * 8;
    const bool active = t < A.T && !status[img] && start < len_bits;          // warp-uniform exits only: the stores are cooperative
    SyncState st;
    st.pos = 0;
    st.b = st.k = 0;
    int q = 0;
    if (active) {
        if (t > 0) st = (A.state[(A.settled[img] - 1) % 3] + (size_t)img * A.T)[t - 1];
        q = A.first_block[(size_t)img * A.T + t];
    }
    int nblk;
    const uint64_t lay = mcu_layout(g, nblk);
    const bool ok = span_write_coop(A.clean + (size_t)img * A.clean_stride, len_bits, st, limit, active, g, T, s_zz, lay, nblk, q, total_blocks,
                                    coef + (size_t)img * g.coef_image_stride, stage_warp, tid & 31,
                                    A.dc + (size_t)img * A.dc_image_stride);
    if (!ok) atomicOr(status + img, 2);
}

// DC differences -> DC values: inclusive prefix sum over the blocks of each component in scan order.  The write pass stores
// every block's DC difference at dc[img][q], q = index of the block in scan order, so the prefix sums read and write 2 bytes per
// block contiguously instead of one 32-byte sector of the coefficient area per block (twice), and the inverse DCT takes its DC
// term from this array.  Segments of kDcxSeg MCUs: (1) segment sums (PHASE 0), (2) exclusive scan of the segment sums
// (jpeg_dc_scan_kernel), (3) prefix inside each segment (PHASE 1).  A thread owns kDcxMcus consecutive MCUs (nblk values
// each).  grid = (segments, n)
constexpr int kDcThreads = 256, kDcxMcus = 8, kDcxSeg = kDcxMcus * kDcThreads;

template <int PHASE>
__global__ void __launch_bounds__(kDcThreads) jpeg_dcx_segment_kernel(int16_t* __restrict__ dc, long long dc_image_stride, JpegGeom g, int segs,
                                                                       int* __restrict__ seg_sum) {
    __shared__ int s_part[3][kDcThreads];
    const int seg = blockIdx.x, img = blockIdx.y, tid = threadIdx.x;
    int nblk;
    const uint64_t lay = mcu_layout(g, nblk);
    const int total_mcus = g.mcux * g.mcuy;
    const int m0 = seg * kDcxSeg + tid * kDcxMcus;
    int16_t* base = dc + (size_t)img * dc_image_stride;
    int sum[3] = {0, 0, 0};
    for (int i = 0; i < kDcxMcus; ++i) {
        if (m0 + i >= total_mcus) break;
        const int16_t* v = base + (size_t)(m0 + i) * nblk;
        for (int b = 0; b < nblk; ++b) sum[(int)(lay >> (4 * b)) & 3] += v[b];
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) s_part[c][tid] = sum[c];
    __syncthreads();
    for (int o = 1; o < kDcThreads; o <<= 1) {
        int x[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) x[c] = tid >= o ? s_part[c][tid - o] : 0;
        __syncthreads();
#pragma unroll
        for (int c = 0; c < 3; ++c) s_part[c][tid] += x[c];
        __syncthreads();
    }
    int* ss = seg_sum + (size_t)img * 3 * segs;
    if (PHASE == 0) {
        if (tid == kDcThreads - 1) {
#pragma unroll
            for (int c = 0; c < 3; ++c) ss[c * segs + seg] = s_part[c][tid];
        }
        return;
    }
    int run[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) run[c] = ss[c * segs + seg] + s_part[c][tid] - sum[c];
    const bool words = (nblk & 1) == 0 && (dc_image_stride & 1) == 0;      // MCUs start on 4-byte boundaries: 32-bit loads / stores
    for (int i = 0; i < kDcxMcus; ++i) {
        if (m0 + i >= total_mcus) break;
        int16_t* v = base + (size_t)(m0 + i) * nblk;
        if (words) {
            for (int b = 0; b < nblk; b += 2) {
                const uint32_t w = *reinterpret_cast<const uint32_t*>(v + b);
                const int c0 = (int)(lay >> (4 * b)) & 3, c1 = (int)(lay >> (4 * b + 4)) & 3;
                run[c0] += (int)(int16_t)(w & 0xffffu);
                const uint32_t lo = (uint32_t)run[c0] & 0xffffu;
                run[c1] += (int)(int16_t)(w >> 16);
                *reinterpret_cast<uint32_t*>(v + b) = lo | ((uint32_t)run[c1] << 16);
            }
        } else {
            for (int b = 0; b < nblk; ++b) {
                const int c = (int)(lay >> (4 * b)) & 3;
                run[c] += v[b];
                v[b] = (int16_t)run[c];
            }
        }
    }
}

// exclusive scan of the segment sums of one image and component (a few hundred entries): one warp
__global__ void jpeg_dc_scan_kernel(int* __restrict__ seg_sum, int segs) {
    int* ss = seg_sum + (size_t)blockIdx.x * segs;
    const int lane = threadIdx.x;
    int carry = 0;
    for (int base = 0; base < segs; base += 32) {
        const int i = base + lane;
        const int v = i < segs ? ss[i] : 0;
        int inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int x = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += x;
        }
        if (i < segs) ss[i] = carry + inc - v;
        carry += __shfl_sync(0xffffffffu, inc, 31);
    }
}
#endif  // FB_JPEG_HOST_TEST

// ---- inverse DCT (jidctint.c, jpeg_idct_islow) ------------------------------------------------------------------------
constexpr int CONST_BITS = 13, PASS1_BITS = 2;
#define FIX_0_298631336 2446
#define FIX_0_390180644 3196
#define FIX_0_541196100 4433
#define FIX_0_765366865 6270
#define FIX_0_899976223 7373
#define FIX_1_175875602 9633
#define FIX_1_501321110 12299
#define FIX_1_847759065 15137
#define FIX_1_961570560 16069
#define FIX_2_053119869 16819
#define FIX_2_562915447 20995
#define FIX_3_072711026 25172

// 1-D pass on eight values (libjpeg works in `JLONG`; 32 bits are enough for 8-bit data: |input| <= 2^15 * 2^2 after
// pass 1, constants < 2^15, four-term sums), results descaled by `shift` with rounding.
FB_HD void idct8(int (&d)[8], int shift, int extra = 0) {
    int z2 = d[2], z3 = d[6];
    int z1 = (z2 + z3) * FIX_0_541196100;
    const int tmp2 = z1 + z3 * (-FIX_1_847759065);
    const int tmp3 = z1 + z2 * FIX_0_765366865;
    z2 = d[0];
    z3 = d[4];
    const int tmp0 = (z2 + z3) * (1 << CONST_BITS);
    const int tmp1 = (z2 - z3) * (1 << CONST_BITS);
    const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    int t0 = d[7], t1 = d[5], t2 = d[3], t3 = d[1];
    z1 = t0 + t3;
    z2 = t1 + t2;
    z3 = t0 + t2;
    int z4 = t1 + t3;
    const int z5 = (z3 + z4) * FIX_1_175875602;
    t0 *= FIX_0_298631336;
    t1 *= FIX_2_053119869;
    t2 *= FIX_3_072711026;
    t3 *= FIX_1_501321110;
    z1 *= -FIX_0_899976223;
    z2 *= -FIX_2_562915447;
    z3 = z3 * (-FIX_1_961570560) + z5;
    z4 = z4 * (-FIX_0_390180644) + z5;
    t0 += z1 + z3;
    t1 += z2 + z4;
    t2 += z2 + z3;
    t3 += z1 + z4;
    const int r = (1 << (shift - 1)) + extra;          // `extra` = a multiple of 1 << shift: added to every output after the shift
    d[0] = (tmp10 + t3 + r) >> shift;
    d[7] = (tmp10 - t3 + r) >> shift;
    d[1] = (tmp11 + t2 + r) >> shift;
    d[6] = (tmp11 - t2 + r) >> shift;
    d[2] = (tmp12 + t1 + r) >> shift;
    d[5] = (tmp12 - t1 + r) >> shift;
    d[3] = (tmp13 + t0 + r) >> shift;
    d[4] = (tmp13 - t0 + r) >> shift;
}

// clamp(v, 0, 255) of four values packed into one word, v0 in the low byte: two I2IP (cvt.pack.sat) on the device
FB_HD uint32_t pack4_sat_u8(int v0, int v1, int v2, int v3) {
#if defined(__CUDA_ARCH__) && __CUDA_ARCH__ >= 720
    uint32_t t, d;
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(t) : "r"(v3), "r"(v2), "r"(0));
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(v1), "r"(v0), "r"(t));
    return d;
#else
    const int v[4] = {v0, v1, v2, v3};
    uint32_t d = 0;
    for (int i = 0; i < 4; ++i) d |= (uint32_t)(v[i] < 0 ? 0 : (v[i] > 255 ? 255 : v[i])) << (8 * i);
    return d;
#endif
}

// One 8x8 block: 64 quantised coefficients (natural order) -> 8 rows of 8 samples at `out` (row pitch `pitch` bytes).
// `emit(r, s)` receives row r of the block as eight samples BEFORE the final clamp to [0, 255] (values in [-384, 639]).
template <class F>
FB_HD void idct_block_rows(const int16_t* src, const uint16_t* q, bool dc_given, int dc, F&& emit) {
    int ws[8][8];
    // dequantise; pass 1 runs down the columns
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const uint4 v = *reinterpret_cast<const uint4*>(src + 8 * r);
        const uint4 qq = *reinterpret_cast<const uint4*>(q + 8 * r);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w}, qw[4] = {qq.x, qq.y, qq.z, qq.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            ws[r][2 * j] = (int)(int16_t)(w[j] & 0xffffu) * (int)(qw[j] & 0xffffu);
            ws[r][2 * j + 1] = (int)(int16_t)(w[j] >> 16) * (int)(qw[j] >> 16);
        }
    }
    if (dc_given) ws[0][0] = dc * (int)q[0];
#pragma unroll
    for (int col = 0; col < 8; ++col) {
        int d[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) d[r] = ws[r][col];
        idct8(d, CONST_BITS - PASS1_BITS);
#pragma unroll
        for (int r = 0; r < 8; ++r) ws[r][col] = d[r];
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        int d[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) d[j] = ws[r][j];
        // libjpeg's range-limit table is indexed with the low 10 bits of the result v: wrap v to [-512, 511], then clamp(v + 128).
        // wrap(v) + 128 = ((v + 512) & 1023) - 384, and the + 512 rides the rounding constant of the pass
        idct8(d, CONST_BITS + PASS1_BITS + 3, 512 << (CONST_BITS + PASS1_BITS + 3));
#pragma unroll
        for (int j = 0; j < 8; ++j) d[j] = (d[j] & 1023) - 384;
        emit(r, d);
    }
}

FB_HD void idct_block_dc(const int16_t* src, const uint16_t* q, uint8_t* out, size_t pitch, bool dc_given, int dc) {
    idct_block_rows(src, q, dc_given, dc, [&](int r, const int (&d)[8]) {
        *reinterpret_cast<uint2*>(out + (size_t)r * pitch) = make_uint2(pack4_sat_u8(d[0], d[1], d[2], d[3]), pack4_sat_u8(d[4], d[5], d[6], d[7]));
    });
}
FB_HD void idct_block(const int16_t* src, const uint16_t* q, uint8_t* out, size_t pitch) { idct_block_dc(src, q, out, pitch, false, 0); }

// `dc` (optional): DC values in scan order (compact integration of the streams without restart markers); the block at
// (brow, bcol) of component c is block c_first + (brow % vs) * hs + bcol % hs of MCU (brow / vs) * mcux + bcol / hs.
__global__ void __launch_bounds__(128) jpeg_idct_kernel(const int16_t* __restrict__ coef, const int* __restrict__ table_slot,
                                                        const JpegTableSet* __restrict__ tables, JpegGeom g, int n,
                                                        uint8_t* __restrict__ planes, const int16_t* __restrict__ dc, long long dc_image_stride) {
    long long blocks_per_image = 0;
    for (int c = 0; c < g.ncomp; ++c) blocks_per_image += (long long)g.blocks_w[c] * g.blocks_h[c];
    const long long total = blocks_per_image * n;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int img = (int)(i / blocks_per_image);
        long long b = i - (long long)img * blocks_per_image;
        int c = 0;
        while (c + 1 < g.ncomp && b >= (long long)g.blocks_w[c] * g.blocks_h[c]) {
            b -= (long long)g.blocks_w[c] * g.blocks_h[c];
            ++c;
        }
        const int bw = g.blocks_w[c];
        const int brow = (int)(b / bw), bcol = (int)(b - (long long)brow * bw);
        const int dcv = dc ? dc[(size_t)img * dc_image_stride + scan_index_of_block(g, c, brow, bcol)] : 0;
        idct_block_dc(coef + (size_t)img * g.coef_image_stride + g.coef_comp_off[c] + b * 64, tables[table_slot[img]].q[g.tq[c]],
                      planes + (size_t)img * g.plane_image_stride + g.plane_comp_off[c] + ((size_t)brow * 8) * ((size_t)bw * 8) + (size_t)bcol * 8,
                      (size_t)bw * 8, dc != nullptr, dcv);
    }
}

// ---- chroma upsampling + colour conversion --------------------------------------------------------------------------------
constexpr int SCALEBITS = 16;
constexpr int ONE_HALF = 1 << (SCALEBITS - 1);
constexpr int kCrR = 91881, kCbB = 116130, kCrG = 46802, kCbG = 22554;        // FIX(1.40200), FIX(1.77200), FIX(0.71414), FIX(0.34414)

FB_HD int clamp8(int v) { return v < 0 ? 0 : (v > 255 ? 255 : v); }

// Six chroma samples of one plane row: columns c0-1 .. c0+4 (c0 a multiple of 4) clamped to [0, cw-1] — the replicated edge
// columns reproduce libjpeg's first / last column special cases.  One aligned word + two bytes when the row has no edge here.
FB_HD void chroma_cols(const uint8_t* row, int c0, int cw, int (&v)[6]) {
    if (c0 >= 1 && c0 + 4 <= cw - 1) {
        const uint32_t w = *reinterpret_cast<const uint32_t*>(row + c0);
        v[0] = row[c0 - 1];
        v[1] = w & 255u;
        v[2] = (w >> 8) & 255u;
        v[3] = (w >> 16) & 255u;
        v[4] = w >> 24;
        v[5] = row[c0 + 4];
    } else {
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            const int c = c0 - 1 + j;
            v[j] = row[c < 0 ? 0 : (c > cw - 1 ? cw - 1 : c)];
        }
    }
}

// YCbCr -> RGB (jdcolor.c tables as integer arithmetic) of eight consecutive pixels and their 24 output bytes at o.
template <bool BGR>
FB_HD void color_pack8(const int (&yy)[8], const int (&cbv)[8], const int (&crv)[8], bool three, uint32_t (&pk)[6]) {
    // y + ((k * (c - 128) + ONE_HALF) >> 16) = (y * 65536 + k * c + ONE_HALF - 128 k) >> 16: the - 128 and the rounding sit in one
    // constant per channel; the clamp to [0, 255] is the saturation of the packing instruction
    constexpr int kR0 = ONE_HALF - 128 * kCrR, kG0 = ONE_HALF + 128 * kCbG + 128 * kCrG, kB0 = ONE_HALF - 128 * kCbB;
    int v[24];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        int r = yy[j], gg = yy[j], b = yy[j];
        if (three) {
            r = (yy[j] * 65536 + kR0 + kCrR * crv[j]) >> SCALEBITS;
            gg = (yy[j] * 65536 + kG0 - kCbG * cbv[j] - kCrG * crv[j]) >> SCALEBITS;
            b = (yy[j] * 65536 + kB0 + kCbB * cbv[j]) >> SCALEBITS;
        }
        v[3 * j] = BGR ? b : r;
        v[3 * j + 1] = gg;
        v[3 * j + 2] = BGR ? r : b;
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) pk[i] = pack4_sat_u8(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
}

FB_HD void color_store8(const int (&yy)[8], const int (&cbv)[8], const int (&crv)[8], bool three, int bgr, int W, int x0, uint8_t* o) {
    uint32_t pk[6];
    if (bgr) color_pack8<true>(yy, cbv, crv, three, pk);
    else color_pack8<false>(yy, cbv, crv, three, pk);
    if (x0 + 8 <= W && ((reinterpret_cast<uintptr_t>(o) & 7) == 0)) {
        uint2* o64 = reinterpret_cast<uint2*>(o);
        o64[0] = make_uint2(pk[0], pk[1]);
        o64[1] = make_uint2(pk[2], pk[3]);
        o64[2] = make_uint2(pk[4], pk[5]);
    } else {
        const int nb = 3 * (W - x0 < 8 ? W - x0 : 8);
        for (int k = 0; k < nb; ++k) o[k] = (uint8_t)(pk[k >> 2] >> (8 * (k & 3)));
    }
}

// MODE 0: chroma at full resolution (4:4:4); 1: h2v1 fancy (h2v2 frames take color_pair420).  Eight consecutive pixels
// x0 .. x0+7 (x0 a multiple of 8) of row y of one image (P = its planes) -> 24 bytes at o.
template <int MODE>
FB_HD void color_group(const uint8_t* P, const JpegGeom& g, int y, int x0, int bgr, uint8_t* o) {
    static_assert(MODE == 0 || MODE == 1, "4:4:4 and h2v1 only: h2v2 frames are converted by color_pair420");
    const int W = g.width;
    const int yp = g.blocks_w[0] * 8;                                   // plane pitches (multiples of 8)
    const int cp = g.ncomp == 3 ? g.blocks_w[1] * 8 : 0;
    const int cw = MODE == 0 ? W : (W + 1) / 2;                         // downsampled chroma size (ceil(size * samp / max))
    int yy[8], cbv[8], crv[8];
    {
        const uint2 w = *reinterpret_cast<const uint2*>(P + g.plane_comp_off[0] + (size_t)y * yp + x0);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            yy[j] = (w.x >> (8 * j)) & 255u;
            yy[4 + j] = (w.y >> (8 * j)) & 255u;
        }
    }
    if (g.ncomp == 3) {
        const uint8_t* CB = P + g.plane_comp_off[1];
        const uint8_t* CR = P + g.plane_comp_off[2];
        if (MODE == 0) {
            const uint2 wb = *reinterpret_cast<const uint2*>(CB + (size_t)y * cp + x0);
            const uint2 wr = *reinterpret_cast<const uint2*>(CR + (size_t)y * cp + x0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                cbv[j] = (wb.x >> (8 * j)) & 255u;
                cbv[4 + j] = (wb.y >> (8 * j)) & 255u;
                crv[j] = (wr.x >> (8 * j)) & 255u;
                crv[4 + j] = (wr.y >> (8 * j)) & 255u;
            }
        } else {
            const int c0 = x0 >> 1;
            int sb[6], sr[6];
            chroma_cols(CB + (size_t)y * cp, c0, cw, sb);
            chroma_cols(CR + (size_t)y * cp, c0, cw, sr);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int k = 1 + (j >> 1);                     // own chroma sample: column c0 + j / 2
                const int nbk = (j & 1) ? k + 1 : k - 1;        // even pixel leans left, odd pixel leans right
                const int bias = (j & 1) ? 2 : 1;
                cbv[j] = (3 * sb[k] + sb[nbk] + bias) >> 2;
                crv[j] = (3 * sr[k] + sr[nbk] + bias) >> 2;
            }
        }
    }
    color_store8(yy, cbv, crv, g.ncomp == 3, bgr, W, x0, o);
}

// h2v2 fancy upsampling, two rows per call: rows y (even) and y + 1 share their near chroma row y / 2 and differ only in the far
// row (y / 2 - 1 above, y / 2 + 1 below, clamped: the replicated context row of jdmainct.c), so a pair needs three chroma rows
// per plane instead of four and one set of addresses.
FB_HD void color_pair420(const uint8_t* P, const JpegGeom& g, int y, int x0, int bgr, uint8_t* o) {
    const int W = g.width, H = g.height;
    const int yp = g.blocks_w[0] * 8, cp = g.blocks_w[1] * 8;
    const int cw = (W + 1) / 2, ch = (H + 1) / 2;
    const uint8_t* CB = P + g.plane_comp_off[1];
    const uint8_t* CR = P + g.plane_comp_off[2];
    const int c0 = x0 >> 1, cy = y >> 1;
    const int up = cy - 1 < 0 ? 0 : cy - 1, dn = cy + 1 > ch - 1 ? ch - 1 : cy + 1;
    int nb[6], nr[6], fb[6], fr[6];
    chroma_cols(CB + (size_t)cy * cp, c0, cw, nb);
    chroma_cols(CR + (size_t)cy * cp, c0, cw, nr);
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        nb[j] *= 3;
        nr[j] *= 3;
    }
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        if (half == 1 && y + 1 >= H) break;
        chroma_cols(CB + (size_t)(half ? dn : up) * cp, c0, cw, fb);
        chroma_cols(CR + (size_t)(half ? dn : up) * cp, c0, cw, fr);
        int yy[8], cbv[8], crv[8];
        const uint2 w = *reinterpret_cast<const uint2*>(P + g.plane_comp_off[0] + (size_t)(y + half) * yp + x0);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            yy[j] = (w.x >> (8 * j)) & 255u;
            yy[4 + j] = (w.y >> (8 * j)) & 255u;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int k = 1 + (j >> 1);
            const int nbk = (j & 1) ? k + 1 : k - 1;
            const int bias = (j & 1) ? 7 : 8;
            cbv[j] = (3 * (nb[k] + fb[k]) + nb[nbk] + fb[nbk] + bias) >> 4;
            crv[j] = (3 * (nr[k] + fr[k]) + nr[nbk] + fr[nbk] + bias) >> 4;
        }
        color_store8(yy, cbv, crv, true, bgr, W, x0, o + (size_t)half * W * 3);
    }
}

// One thread = 8 consecutive pixels of a row; blockIdx.x = image * H + row (no 64-bit divisions per thread).
template <int MODE>
__global__ void __launch_bounds__(256) jpeg_color_kernel(const uint8_t* __restrict__ planes, JpegGeom g, int n, int bgr,
                                                         uint8_t* __restrict__ out, long long out_stride) {
    const int W = g.width, H = g.height;
    const int gx = blockIdx.y * blockDim.x + threadIdx.x;
    if (gx * 8 >= W) return;
    const int img = (int)(blockIdx.x / (unsigned)H), y = (int)(blockIdx.x - (unsigned)img * (unsigned)H);
    color_group<MODE>(planes + (size_t)img * g.plane_image_stride, g, y, gx * 8, bgr,
                      out + (size_t)img * out_stride + ((size_t)y * W + gx * 8) * 3);
}


// h2v2: one thread = 8 consecutive pixels of a PAIR of rows; blockIdx.x = image * ceil(H / 2) + pair
__global__ void __launch_bounds__(256) jpeg_color420_pair_kernel(const uint8_t* __restrict__ planes, JpegGeom g, int n, int bgr,
                                                                 uint8_t* __restrict__ out, long long out_stride) {
    const int W = g.width, H = g.height;
    const unsigned pairs = (unsigned)(H + 1) >> 1;
    const int gx = blockIdx.y * blockDim.x + threadIdx.x;
    if (gx * 8 >= W) return;
    const int img = (int)(blockIdx.x / pairs), y = 2 * (int)(blockIdx.x - (unsigned)img * pairs);
    color_pair420(planes + (size_t)img * g.plane_image_stride, g, y, gx * 8, bgr, out + (size_t)img * out_stride + ((size_t)y * W + gx * 8) * 3);
}

}  // namespace

#ifndef FB_JPEG_HOST_TEST
constexpr int kSerialMcus = 1024;        // streams without restart markers up to this size take the one-thread-per-stream path

static long long selfsync_subsequences(long long max_scan_bytes) { return (max_scan_bytes + kSubseqBytes - 1) / kSubseqBytes + 1; }
static long long selfsync_clean_stride(long long max_scan_bytes) { return (max_scan_bytes + 64 + 255) & ~255ll; }

size_t jpeg_workspace_bytes(int n, int width, int height, int ncomp, int hs0, int vs0, int restart_interval, long long max_scan_bytes) {
    const int hmax = hs0, vmax = vs0;
    const long long mcux = (width + 8 * hmax - 1) / (8 * hmax), mcuy = (height + 8 * vmax - 1) / (8 * vmax);
    long long blocks = mcux * hmax * mcuy * vmax + (ncomp == 3 ? 2 * mcux * mcuy : 0);
    const long long total_mcus = mcux * mcuy;
    const long long n_iv = restart_interval > 0 ? (total_mcus + restart_interval - 1) / restart_interval : 1;
    const long long chunks = (max_scan_bytes + kScanChunk - 1) / kScanChunk + 1;
    auto al = [](long long x) { return (x + 255) & ~255ll; };
    long long total = al(blocks * 128 * n) + al(blocks * 64 * n) + al(n_iv * 4 * n) + al(chunks * 4 * n) + 256;
    if (restart_interval <= 0 && total_mcus > kSerialMcus) {
        const long long T = selfsync_subsequences(max_scan_bytes);
        total += al(selfsync_clean_stride(max_scan_bytes) * n) + al(8ll * n) + 3 * al((long long)sizeof(SyncState) * T * n) +
                 2 * al(4 * T * n) + al(4ll * (kSyncRounds + 1) * n) + al(4ll * ((n + 63) & ~63)) +
                 al(4ll * 3 * n * ((total_mcus * hmax * vmax + 2047) / 2048 + 1)) + al(2ll * blocks * n);
    }
    return (size_t)total;
}

int launch_jpeg_decode(const uint8_t* d_bytes, const long long* d_scan_off, const long long* d_scan_len, const int* d_table_slot,
                       const void* d_tables, int n, int width, int height, int ncomp, const int* hs, const int* vs, const int* tq,
                       const int* td, const int* ta, int restart_interval, long long max_scan_bytes, int bgr, void* d_workspace,
                       size_t workspace_bytes, uint8_t* d_out, long long out_stride, int* d_status, cudaStream_t stream) {
    FB_REQUIRE(d_bytes && d_scan_off && d_scan_len && d_table_slot && d_tables && d_workspace && d_out && d_status, "fb_jpeg_decode: null pointer");
    FB_REQUIRE(n >= 1 && width >= 1 && height >= 1 && width <= 65535 && height <= 65535, "fb_jpeg_decode: bad size %dx%d", width, height);
    FB_REQUIRE(ncomp == 1 || ncomp == 3, "fb_jpeg_decode: %d components (1 or 3)", ncomp);
    FB_REQUIRE(out_stride >= (long long)width * height * 3, "fb_jpeg_decode: out_stride smaller than one frame");
    JpegGeom g;
    g.width = width;
    g.height = height;
    g.ncomp = ncomp;
    for (int c = 0; c < 3; ++c) {
        g.hs[c] = c < ncomp ? hs[c] : 1;
        g.vs[c] = c < ncomp ? vs[c] : 1;
        g.tq[c] = c < ncomp ? tq[c] : 0;
        g.td[c] = c < ncomp ? td[c] : 0;
        g.ta[c] = c < ncomp ? ta[c] : 0;
        FB_REQUIRE(g.tq[c] >= 0 && g.tq[c] < 4 && g.td[c] >= 0 && g.td[c] < 4 && g.ta[c] >= 0 && g.ta[c] < 4, "fb_jpeg_decode: table id out of range");
    }
    const int hmax = g.hs[0], vmax = g.vs[0];
    FB_REQUIRE((hmax == 1 && vmax == 1) || (hmax == 2 && vmax == 1) || (hmax == 2 && vmax == 2), "fb_jpeg_decode: luma sampling %dx%d", hmax, vmax);
    FB_REQUIRE(ncomp == 1 || (g.hs[1] == 1 && g.vs[1] == 1 && g.hs[2] == 1 && g.vs[2] == 1), "fb_jpeg_decode: chroma sampling must be 1x1");
    FB_REQUIRE(ncomp == 3 || (hmax == 1 && vmax == 1), "fb_jpeg_decode: a grayscale scan has 8x8 MCUs");
    g.restart_interval = restart_interval > 0 ? restart_interval : 0;
    g.mcux = (width + 8 * hmax - 1) / (8 * hmax);
    g.mcuy = (height + 8 * vmax - 1) / (8 * vmax);
    const long long total_mcus = (long long)g.mcux * g.mcuy;
    g.n_intervals = g.restart_interval ? (int)((total_mcus + g.restart_interval - 1) / g.restart_interval) : 1;
    long long blocks = 0;
    for (int c = 0; c < 3; ++c) {
        g.blocks_w[c] = c < ncomp ? g.mcux * g.hs[c] : 0;
        g.blocks_h[c] = c < ncomp ? g.mcuy * g.vs[c] : 0;
        g.coef_comp_off[c] = blocks * 64;
        g.plane_comp_off[c] = blocks * 64;
        blocks += (long long)g.blocks_w[c] * g.blocks_h[c];
    }
    g.coef_image_stride = blocks * 64;
    g.plane_image_stride = blocks * 64;
    FB_REQUIRE(workspace_bytes >= jpeg_workspace_bytes(n, width, height, ncomp, hmax, vmax, restart_interval, max_scan_bytes),
               "fb_jpeg_decode: workspace too small");
    FB_REQUIRE((reinterpret_cast<uintptr_t>(d_workspace) & 255) == 0, "fb_jpeg_decode: workspace must be 256-byte aligned");
    auto al = [](long long x) { return (x + 255) & ~255ll; };
    uint8_t* w = reinterpret_cast<uint8_t*>(d_workspace);
    int16_t* coef = reinterpret_cast<int16_t*>(w);
    w += al(blocks * 128 * n);
    uint8_t* planes = w;
    w += al(blocks * 64 * n);
    uint32_t* starts = reinterpret_cast<uint32_t*>(w);
    w += al((long long)g.n_intervals * 4 * n);
    int* counts = reinterpret_cast<int*>(w);
    const int chunks = (int)((max_scan_bytes + kScanChunk - 1) / kScanChunk + 1);

    w += al((long long)chunks * 4 * n);
    const bool selfsync = g.restart_interval == 0 && total_mcus > kSerialMcus;
    const JpegTableSet* tables = reinterpret_cast<const JpegTableSet*>(d_tables);
    const int16_t* dc_values = nullptr;          // DC values of the self-synchronising path; the restart-marker path leaves them in coef[0]

    FB_CUDA_OK(cudaMemsetAsync(d_status, 0, sizeof(int) * n, stream));
    if (selfsync) {
        // no restart markers: unstuff, find the true decoder state at every subsequence boundary, decode, integrate the DC
        SyncArrays A;
        A.T = (int)selfsync_subsequences(max_scan_bytes);
        A.clean_stride = selfsync_clean_stride(max_scan_bytes);
        uint8_t* clean = w;
        w += al(A.clean_stride * n);
        long long* clean_len = reinterpret_cast<long long*>(w);
        w += al(8ll * n);
        for (int i = 0; i < 3; ++i) {
            A.state[i] = reinterpret_cast<SyncState*>(w);
            w += al((long long)sizeof(SyncState) * A.T * n);
        }
        A.blocks = reinterpret_cast<int*>(w);
        w += al(4ll * A.T * n);
        A.first_block = reinterpret_cast<int*>(w);
        w += al(4ll * A.T * n);
        A.changed = reinterpret_cast<int*>(w);
        w += al(4ll * (kSyncRounds + 1) * n);
        A.settled = reinterpret_cast<int*>(w);
        w += al(4ll * ((n + 63) & ~63));
        w += al(4ll * 3 * n * ((total_mcus * hmax * vmax + 2047) / 2048 + 1));          // segment sums of the DC integration
        A.dc = reinterpret_cast<int16_t*>(w);
        A.dc_image_stride = blocks;
        A.clean = clean;
        A.clean_len = clean_len;
        const int total_blocks = (int)(blocks);
        FB_REQUIRE(blocks < (1ll << 31), "fb_jpeg_decode: frame too large");
        FB_CUDA_OK(cudaMemsetAsync(clean, 0, (size_t)A.clean_stride * n, stream));
        FB_CUDA_OK(cudaMemsetAsync(A.changed, 0, sizeof(int) * (kSyncRounds + 1) * n, stream));
        FB_CUDA_OK(cudaMemsetAsync(A.settled, 0, sizeof(int) * n, stream));
        dim3 cgrid(chunks, n);
        jpeg_unstuff_kernel<false><<<cgrid, kScanThreads, 0, stream>>>(d_bytes, d_scan_off, d_scan_len, chunks, counts, clean, A.clean_stride);
        jpeg_unstuff_prefix_kernel<<<n, 256, 0, stream>>>(counts, chunks, d_scan_len, clean_len);
        jpeg_unstuff_kernel<true><<<cgrid, kScanThreads, 0, stream>>>(d_bytes, d_scan_off, d_scan_len, chunks, counts, clean, A.clean_stride);
        dim3 sgrid((A.T + 127) / 128, n);
        for (int round = 0; round <= kSyncRounds; ++round) {
            jpeg_sync_kernel<<<sgrid, 128, 0, stream>>>(A, d_table_slot, tables, g, round);
            if (round >= 1) jpeg_sync_settle_kernel<<<(n + 127) / 128, 128, 0, stream>>>(A, n, round);
        }
        jpeg_sync_prefix_kernel<<<n, 1024, 0, stream>>>(A, total_blocks, d_status);
        {
            static PerDeviceFlag w_attr_set;
            if (!w_attr_set.get()) {
                FB_CUDA_OK(cudaFuncSetAttribute(jpeg_sync_write_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSyncWriteSmem));
                w_attr_set.set();
            }
            jpeg_sync_write_kernel<<<dim3((A.T + kSyncWriteThreads - 1) / kSyncWriteThreads, n), kSyncWriteThreads, kSyncWriteSmem, stream>>>(
                A, d_table_slot, tables, g, total_blocks, coef, d_status);
        }
        // compact DC integration: prefix sums over the 2-byte-per-block copy the write pass made; the inverse DCT reads it
        const int segs = (int)((total_mcus + kDcxSeg - 1) / kDcxSeg);
        int* seg_sum = reinterpret_cast<int*>(A.settled + ((n + 63) & ~63));
        jpeg_dcx_segment_kernel<0><<<dim3(segs, n), kDcThreads, 0, stream>>>(A.dc, A.dc_image_stride, g, segs, seg_sum);
        jpeg_dc_scan_kernel<<<n * 3, 32, 0, stream>>>(seg_sum, segs);
        jpeg_dcx_segment_kernel<1><<<dim3(segs, n), kDcThreads, 0, stream>>>(A.dc, A.dc_image_stride, g, segs, seg_sum);
        dc_values = A.dc;
    } else {
        if (g.n_intervals > 1) {
            dim3 grid(chunks, n);
            jpeg_restart_scan_kernel<false><<<grid, kScanThreads, 0, stream>>>(d_bytes, d_scan_off, d_scan_len, chunks, g.n_intervals, counts, starts);
            jpeg_restart_prefix_kernel<<<n, 256, 0, stream>>>(counts, chunks, g.n_intervals, starts, d_status);
            jpeg_restart_scan_kernel<true><<<grid, kScanThreads, 0, stream>>>(d_bytes, d_scan_off, d_scan_len, chunks, g.n_intervals, counts, starts);
        } else {
            FB_CUDA_OK(cudaMemsetAsync(starts, 0, sizeof(uint32_t) * n, stream));
        }
        dim3 grid((g.n_intervals + kHuffThreads - 1) / kHuffThreads, n);
        static PerDeviceFlag attr_set;
        if (!attr_set.get()) {
            FB_CUDA_OK(cudaFuncSetAttribute(jpeg_huffman_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kHuffSmem));
            attr_set.set();
        }
        jpeg_huffman_kernel<<<grid, kHuffThreads, kHuffSmem, stream>>>(d_bytes, d_scan_off, d_scan_len, d_table_slot, tables, starts, g, coef, d_status);
    }
    {
        const long long total = blocks * n;
        long long gb = (total + 127) / 128;
        if (gb > (long long)sm_count() * 32) gb = (long long)sm_count() * 32;
        jpeg_idct_kernel<<<(unsigned)gb, 128, 0, stream>>>(coef, d_table_slot, reinterpret_cast<const JpegTableSet*>(d_tables), g, n, planes, dc_values,
                                                           blocks);
    }
    {
        const int groups = (width + 7) / 8;
        const int threads = groups >= 256 ? 256 : ((groups + 31) / 32) * 32;
        dim3 grid((unsigned)((long long)n * height), (unsigned)((groups + threads - 1) / threads));
        const int mode = ncomp == 1 ? 0 : (hmax == 1 ? 0 : (vmax == 1 ? 1 : 2));
        if (mode == 0) jpeg_color_kernel<0><<<grid, threads, 0, stream>>>(planes, g, n, bgr, d_out, out_stride);
        else if (mode == 1) jpeg_color_kernel<1><<<grid, threads, 0, stream>>>(planes, g, n, bgr, d_out, out_stride);
        else jpeg_color420_pair_kernel<<<dim3((unsigned)((long long)n * ((height + 1) / 2)), grid.y), threads, 0, stream>>>(planes, g, n, bgr, d_out, out_stride);
    }
    FB_CUDA_OK(cudaGetLastError());
    return 0;
}

#endif  // FB_JPEG_HOST_TEST

}  // namespace fb
