// TEST TOOL (not part of libfacet_b200.so): runs the __host__ __device__ bodies of csrc/jpeg_decode.cu — entropy decoding
// of every restart interval, the inverse DCT of every block, upsampling + colour conversion of every pixel group — on the
// CPU, so that tests/test_jpeg_host.py can compare them with Pillow without a GPU.  The kernels themselves (indexing,
// restart scan) are covered by tests/test_gpu_jpeg.py.
//   usage: jpeg_host_check <request file> <output file>
//   request: int32 header[32] = {width, height, ncomp, hs[3], vs[3], tq[3], td[3], restart_interval, bgr, scan_len, ta[3], selfsync, 0...}
//            then the 11904-byte table set, then scan_len bytes of entropy-coded data
#define FB_JPEG_HOST_TEST 1
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../facet_b200/csrc/jpeg_decode.cu"

namespace fb {
void set_error(const char*, ...) {}
const char* get_error() { return ""; }
int sm_count() { return 1; }
}  // namespace fb

using namespace fb;

int main(int argc, char** argv) {
    if (argc != 3) return 2;
    FILE* f = fopen(argv[1], "rb");
    if (!f) return 2;
    int32_t hdr[32];
    if (fread(hdr, 4, 32, f) != 32) return 2;
    JpegTableSet* T_ = (JpegTableSet*)aligned_alloc(16, sizeof(JpegTableSet));
    if (fread(T_, 1, sizeof(JpegTableSet), f) != sizeof(JpegTableSet)) return 2;
    const long long len = hdr[17];
    std::vector<uint8_t> scan(len + 16);
    if ((long long)fread(scan.data(), 1, len, f) != len) return 2;
    fclose(f);
    JpegGeom g;
    g.width = hdr[0];
    g.height = hdr[1];
    g.ncomp = hdr[2];
    for (int c = 0; c < 3; ++c) {
        g.hs[c] = hdr[3 + c];
        g.vs[c] = hdr[6 + c];
        g.tq[c] = hdr[9 + c];
        g.td[c] = hdr[12 + c];
    }
    for (int c = 0; c < 3; ++c) g.ta[c] = hdr[18 + c];
    g.restart_interval = hdr[15];
    const int bgr = hdr[16];
    const int hmax = g.hs[0], vmax = g.vs[0];
    g.mcux = (g.width + 8 * hmax - 1) / (8 * hmax);
    g.mcuy = (g.height + 8 * vmax - 1) / (8 * vmax);
    const long long total_mcus = (long long)g.mcux * g.mcuy;
    g.n_intervals = g.restart_interval ? (int)((total_mcus + g.restart_interval - 1) / g.restart_interval) : 1;
    long long blocks = 0;
    for (int c = 0; c < 3; ++c) {
        g.blocks_w[c] = c < g.ncomp ? g.mcux * g.hs[c] : 0;
        g.blocks_h[c] = c < g.ncomp ? g.mcuy * g.vs[c] : 0;
        g.coef_comp_off[c] = blocks * 64;
        g.plane_comp_off[c] = blocks * 64;
        blocks += (long long)g.blocks_w[c] * g.blocks_h[c];
    }
    g.coef_image_stride = g.plane_image_stride = blocks * 64;
    int16_t* coef = (int16_t*)aligned_alloc(16, (size_t)blocks * 128 + 16);
    memset(coef, 0, (size_t)blocks * 128 + 16);
    uint8_t* planes = (uint8_t*)aligned_alloc(256, ((size_t)blocks * 64 + 511) & ~(size_t)255);
    {
        // scan_index_of_block (the inverse DCT's look-up into the compact DC array) must invert scan_block_ptr
        int nblk_;
        const uint64_t lay_ = mcu_layout(g, nblk_);
        for (long long q = 0; q < blocks; ++q) {
            const int16_t* ptr = scan_block_ptr((int)q, g, lay_, nblk_, coef);
            int c = g.ncomp - 1;
            while (c > 0 && ptr < coef + g.coef_comp_off[c]) --c;
            const long long b = (ptr - (coef + g.coef_comp_off[c])) / 64;
            if (scan_index_of_block(g, c, (int)(b / g.blocks_w[c]), (int)(b % g.blocks_w[c])) != q) {
                fprintf(stderr, "scan_index_of_block does not invert scan_block_ptr at block %lld\n", q);
                return 7;
            }
        }
    }
    if (hdr[21]) {
        // self-synchronising path (streams without restart markers), the kernels' algorithm executed sequentially
        std::vector<uint8_t> clean;
        clean.reserve(len + 64);
        for (long long p = 0; p < len; ++p)
            if (!(scan[p] == 0x00 && p > 0 && scan[p - 1] == 0xFF)) clean.push_back(scan[p]);
        const long long clean_len = (long long)clean.size(), len_bits = 8 * clean_len;
        clean.resize(clean_len + 64, 0);
        const int T = (int)((clean_len + kSubseqBytes - 1) / kSubseqBytes);
        int nblk;
        const uint64_t lay = mcu_layout(g, nblk);
        std::vector<SyncState> cur(T), prev(T);
        std::vector<int> nb(T, 0), first(T, 0);
        int rounds_used = -1;
        for (int round = 0; round <= kSyncRounds; ++round) {
            bool changed = false;
            for (int t = 0; t < T; ++t) {
                const long long start = (long long)t * kSubseqBytes * 8, limit = start + (long long)kSubseqBytes * 8;
                SyncState st;
                if (round == 0 || t == 0) {
                    st.pos = start;
                    st.b = st.k = 0;
                } else {
                    st = prev[t - 1];
                }
                SyncState out;
                int done;
                span_decode<false>(clean.data(), len_bits, st, limit, g, *T_, h_zigzag, lay, nblk, out, done, 0, 0, nullptr);
                if (round >= 1 && (prev[t].pos != out.pos || prev[t].b != out.b || prev[t].k != out.k)) changed = true;
                cur[t] = out;
                nb[t] = done;
            }
            prev = cur;
            if (round >= 1 && !changed) {
                rounds_used = round;
                break;
            }
        }
        if (rounds_used < 0) {
            fprintf(stderr, "self-synchronisation did not settle in %d rounds\n", kSyncRounds);
            return 5;
        }
        fprintf(stderr, "selfsync: %d subsequences, settled after %d rounds\n", T, rounds_used);
        int run = 0;
        for (int t = 0; t < T; ++t) {
            first[t] = run;
            run += nb[t];
        }
        if (run < (int)blocks) {
            fprintf(stderr, "stream holds %d blocks, frame needs %lld\n", run, blocks);
            return 6;
        }
        for (int t = 0; t < T; ++t) {
            const long long start = (long long)t * kSubseqBytes * 8, limit = start + (long long)kSubseqBytes * 8;
            SyncState st;
            if (t == 0) {
                st.pos = 0;
                st.b = st.k = 0;
            } else {
                st = prev[t - 1];
            }
            SyncState out;
            int done;
            if (!span_decode<true>(clean.data(), len_bits, st, limit, g, *T_, h_zigzag, lay, nblk, out, done, first[t], (int)blocks, coef)) {
                fprintf(stderr, "bad Huffman data in subsequence %d\n", t);
                return 4;
            }
        }
        for (int c = 0; c < g.ncomp; ++c) {
            const int per_mcu = g.hs[c] * g.vs[c], count = g.mcux * g.mcuy * per_mcu;
            int acc = 0;
            for (int j = 0; j < count; ++j) {
                const int m = j / per_mcu, r = j - m * per_mcu, by = r / g.hs[c], bx = r - by * g.hs[c];
                const int my = m / g.mcux, mx = m - my * g.mcux;
                int16_t* p = coef + g.coef_comp_off[c] + ((size_t)(my * g.vs[c] + by) * g.blocks_w[c] + (mx * g.hs[c] + bx)) * 64;
                acc += *p;
                *p = (int16_t)acc;
            }
        }
    } else {
    // restart markers
    std::vector<uint32_t> starts(1, 0u);
    for (long long p = 0; p + 1 < len; ++p)
        if (scan[p] == 0xFF && (scan[p + 1] & 0xF8) == 0xD0) starts.push_back((uint32_t)(p + 2));
    if ((int)starts.size() != g.n_intervals) {
        fprintf(stderr, "restart markers: found %zu intervals, header says %d\n", starts.size(), g.n_intervals);
        return 3;
    }
    for (int iv = 0; iv < g.n_intervals; ++iv) {
        const uint8_t* p0 = scan.data() + starts[iv];
        const uint8_t* p1 = iv + 1 < g.n_intervals ? scan.data() + starts[iv + 1] - 2 : scan.data() + len;
        if (!decode_interval<false>(p0, p1, iv, g, *T_, h_zigzag, coef, true, nullptr, 0)) {
            fprintf(stderr, "bad Huffman data in interval %d\n", iv);
            return 4;
        }
    }
    }
    for (int c = 0; c < g.ncomp; ++c)
        for (long long b = 0; b < (long long)g.blocks_w[c] * g.blocks_h[c]; ++b) {
            const int bw = g.blocks_w[c];
            const long long brow = b / bw, bcol = b - brow * bw;
            idct_block(coef + g.coef_comp_off[c] + b * 64, T_->q[g.tq[c]], planes + g.plane_comp_off[c] + (size_t)brow * 8 * bw * 8 + (size_t)bcol * 8,
                       (size_t)bw * 8);
        }
    std::vector<uint8_t> out((size_t)g.width * (g.height + 1) * 3 + 32);
    const int mode = g.ncomp == 1 ? 0 : (hmax == 1 ? 0 : (vmax == 1 ? 1 : 2));
    for (int y = 0; y < g.height; y += mode == 2 ? 2 : 1)
        for (int x0 = 0; x0 < g.width; x0 += 8) {
            uint8_t* o = out.data() + ((size_t)y * g.width + x0) * 3;
            if (mode == 0) color_group<0>(planes, g, y, x0, bgr, o);
            else if (mode == 1) color_group<1>(planes, g, y, x0, bgr, o);
            else color_pair420(planes, g, y, x0, bgr, o);
        }
    f = fopen(argv[2], "wb");
    fwrite(out.data(), 1, (size_t)g.width * g.height * 3, f);
    fclose(f);
    return 0;
}
