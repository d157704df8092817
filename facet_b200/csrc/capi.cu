// extern "C" surface of libfacet_b200.so — see include/facet_b200.h for the contract.
#include <atomic>
#include <cstdarg>
#include <cstring>
#include <mutex>
#include <vector>

#include "../../include/facet_b200.h"
#include "common.cuh"
#include "kernels.h"

namespace fb {
int vit_forward(const fb_vit_weights* w, const float* d_clip_in, int batch, void* d_workspace, size_t workspace_bytes,
                float* d_features, float* d_embedding, float* d_aesthetic_raw, float* d_tag_sims, cudaStream_t st);
}

namespace fb {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
const char* get_error() { return g_err; }
void count_launch(int k) { g_launches.fetch_add((uint64_t)k, std::memory_order_relaxed); }

// ---- event-pair profiler -----------------------------------------------------------------------------
// A ProfScope takes (or creates) an event pair under the lock and keeps the two handles itself, so the
// destructor never indexes the shared vectors (another thread's constructor may be growing them).
namespace {
struct ProfState {
    std::mutex mu;
    std::atomic<bool> on{false};
    std::vector<cudaEvent_t> ev;     // pairs: [2*i] begin, [2*i+1] end
    std::vector<int> cat;
    size_t used = 0;
} g_prof;
}  // namespace

ProfScope::ProfScope(int c, cudaStream_t st) : slot(-1), stream(st), begin(nullptr), end(nullptr) {
    if (!g_prof.on.load(std::memory_order_relaxed)) return;
    {
        std::lock_guard<std::mutex> lk(g_prof.mu);
        if (!g_prof.on.load(std::memory_order_relaxed)) return;
        if (g_prof.used == g_prof.cat.size()) {
            cudaEvent_t a = nullptr, b = nullptr;
            if (cudaEventCreate(&a) != cudaSuccess) return;
            if (cudaEventCreate(&b) != cudaSuccess) {
                cudaEventDestroy(a);
                return;
            }
            g_prof.ev.push_back(a);
            g_prof.ev.push_back(b);
            g_prof.cat.push_back(c);
        }
        slot = (int)g_prof.used++;
        g_prof.cat[slot] = c;
        begin = g_prof.ev[2 * slot];
        end = g_prof.ev[2 * slot + 1];
    }
    cudaEventRecord(begin, stream);
}
ProfScope::~ProfScope() {
    if (slot >= 0) cudaEventRecord(end, stream);
}

int sm_count() {
    // per device ordinal: one process may drive several different GPUs
    constexpr int kMaxDev = 64;
    static std::atomic<int> cached[kMaxDev];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDev) dev = 0;
    int sms = cached[dev].load(std::memory_order_relaxed);
    if (sms == 0) {
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
        cached[dev].store(sms, std::memory_order_relaxed);
    }
    return sms;
}

}  // namespace fb

using namespace fb;

extern "C" {

int fb_abi_version(void) { return FB_ABI_VERSION; }
const char* fb_last_error(void) { return get_error(); }
uint64_t fb_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
int fb_device_sm_count(void) { return sm_count(); }

void fb_profile_enable(int on) {
    std::lock_guard<std::mutex> lk(g_prof.mu);
    g_prof.on.store(on != 0, std::memory_order_relaxed);
    g_prof.used = 0;
}

int fb_profile_read(double* ms_per_category, uint64_t* launches_per_category, int n_categories) {
    FB_REQUIRE(ms_per_category && launches_per_category && n_categories >= PROF_NCAT, "fb_profile_read: need %d categories", (int)PROF_NCAT);
    FB_CUDA_OK(cudaDeviceSynchronize());
    std::lock_guard<std::mutex> lk(g_prof.mu);
    for (int i = 0; i < n_categories; ++i) {
        ms_per_category[i] = 0.0;
        launches_per_category[i] = 0;
    }
    for (size_t i = 0; i < g_prof.used; ++i) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, g_prof.ev[2 * i], g_prof.ev[2 * i + 1]) == cudaSuccess) {
            ms_per_category[g_prof.cat[i]] += ms;
            launches_per_category[g_prof.cat[i]] += 1;
        }
    }
    g_prof.used = 0;
    return 0;
}

int fb_tech_stats_luma(const uint8_t* d_images, int n, int height, int width, int64_t image_stride, int rgb_order,
                       uint32_t* d_hist256, uint32_t* d_hs_hist, int64_t* d_sums, int force_generic, uint8_t* d_luma,
                       void* stream) {
    ProfScope ps(PROF_TECH, (cudaStream_t)stream);
    int rc = launch_tech_stats(d_images, n, height, width, (long long)image_stride, rgb_order, d_hist256, d_hs_hist,
                               reinterpret_cast<long long*>(d_sums), force_generic, d_luma, nullptr, nullptr, (cudaStream_t)stream);
    if (rc == 0) count_launch(1);
    return rc;
}

int fb_tech_stats_fused(const uint8_t* d_images, int n, int height, int width, int64_t image_stride, int rgb_order,
                        uint32_t* d_hist256, uint32_t* d_hs_hist, int64_t* d_sums, uint8_t* d_luma, uint8_t* d_box4,
                        const uint32_t* box_mult4, void* stream) {
    ProfScope ps(PROF_TECH, (cudaStream_t)stream);
    int rc = launch_tech_stats(d_images, n, height, width, (long long)image_stride, rgb_order, d_hist256, d_hs_hist,
                               reinterpret_cast<long long*>(d_sums), 0, d_luma, d_box4, box_mult4, (cudaStream_t)stream);
    if (rc == 0) count_launch(1);
    return rc;
}

int fb_tech_stats(const uint8_t* d_images, int n, int height, int width, int64_t image_stride, int rgb_order,
                  uint32_t* d_hist256, uint32_t* d_hs_hist, int64_t* d_sums, int force_generic, void* stream) {
    ProfScope ps(PROF_TECH, (cudaStream_t)stream);
    int rc = launch_tech_stats(d_images, n, height, width, (long long)image_stride, rgb_order, d_hist256, d_hs_hist,
                               reinterpret_cast<long long*>(d_sums), force_generic, nullptr, nullptr, nullptr, (cudaStream_t)stream);
    if (rc == 0) count_launch(1);
    return rc;
}

int fb_tech_derive(const uint32_t* d_hs_hist, int n, double* d_out, void* stream) {
    ProfScope ps(PROF_DERIVE, (cudaStream_t)stream);
    int rc = launch_hs_derive(d_hs_hist, n, d_out, (cudaStream_t)stream);
    if (rc == 0) count_launch(1);
    return rc;
}

int fb_tech_stats_host(const uint8_t* h_images, int n, int height, int width, int rgb_order, uint32_t* h_hist256,
                       int64_t* h_sums, double* h_derived, uint32_t* h_hs_hist) {
    FB_REQUIRE(h_images && h_hist256 && h_sums && h_derived, "fb_tech_stats_host: null pointer");
    FB_REQUIRE(n >= 1 && height >= 2 && width >= 2, "fb_tech_stats_host: need n>=1 and images of at least 2x2");
    const size_t img_bytes = (size_t)height * width * 3;
    const size_t stride = (img_bytes + 15) & ~(size_t)15;
    uint8_t* d_img = nullptr;
    uint32_t *d_h = nullptr, *d_hs = nullptr;
    long long* d_s = nullptr;
    double* d_d = nullptr;
    cudaStream_t st = nullptr;
    int rc = 0;
    auto cleanup = [&]() {
        cudaFree(d_img); cudaFree(d_h); cudaFree(d_hs); cudaFree(d_s); cudaFree(d_d);
        if (st) cudaStreamDestroy(st);
    };
#define FB_TRY(expr)                                                                              \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess) {                                                                  \
            set_error("%s failed: %s", #expr, cudaGetErrorString(_e));                            \
            cleanup();                                                                            \
            return (int)_e;                                                                       \
        }                                                                                         \
    } while (0)
    FB_TRY(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    FB_TRY(cudaMalloc(&d_img, stride * n));
    FB_TRY(cudaMalloc(&d_h, (size_t)n * 256 * 4));
    FB_TRY(cudaMalloc(&d_hs, (size_t)n * FB_HS_BINS * 4));
    FB_TRY(cudaMalloc(&d_s, (size_t)n * 4 * 8));
    FB_TRY(cudaMalloc(&d_d, (size_t)n * 4 * 8));
    if (stride == img_bytes) {
        FB_TRY(cudaMemcpyAsync(d_img, h_images, img_bytes * n, cudaMemcpyHostToDevice, st));
    } else {
        for (int i = 0; i < n; ++i)
            FB_TRY(cudaMemcpyAsync(d_img + stride * i, h_images + img_bytes * i, img_bytes, cudaMemcpyHostToDevice, st));
    }
    rc = fb_tech_stats(d_img, n, height, width, (int64_t)stride, rgb_order, d_h, d_hs, (int64_t*)d_s, 0, st);
    if (rc == 0) rc = fb_tech_derive(d_hs, n, d_d, st);
    if (rc != 0) {
        cleanup();
        return rc;
    }
    FB_TRY(cudaMemcpyAsync(h_hist256, d_h, (size_t)n * 256 * 4, cudaMemcpyDeviceToHost, st));
    FB_TRY(cudaMemcpyAsync(h_sums, d_s, (size_t)n * 4 * 8, cudaMemcpyDeviceToHost, st));
    FB_TRY(cudaMemcpyAsync(h_derived, d_d, (size_t)n * 4 * 8, cudaMemcpyDeviceToHost, st));
    if (h_hs_hist) FB_TRY(cudaMemcpyAsync(h_hs_hist, d_hs, (size_t)n * FB_HS_BINS * 4, cudaMemcpyDeviceToHost, st));
    FB_TRY(cudaStreamSynchronize(st));
#undef FB_TRY
    cleanup();
    return 0;
}

int fb_gray_hsv(const uint8_t* d_image, int height, int width, int rgb_order, uint8_t* d_gray, uint8_t* d_hsv,
                void* stream) {
    int rc = launch_gray_hsv(d_image, height, width, rgb_order, d_gray, d_hsv, (cudaStream_t)stream);
    if (rc == 0) count_launch(1);
    return rc;
}

int fb_gray_plane(const uint8_t* d_image, int height, int width, int rgb_order, uint8_t* d_gray, uint32_t* d_hist256,
                  void* stream) {
    int rc = launch_gray_plane(d_image, height, width, rgb_order, d_gray, d_hist256, (cudaStream_t)stream);
    if (rc == 0) count_launch(1);
    return rc;
}

size_t fb_canny_workspace_bytes(int height, int width) { return canny_workspace_bytes(height, width); }

int fb_canny(const uint8_t* d_gray, int height, int width, int blur, int low, int high, void* d_workspace,
             size_t workspace_bytes, uint8_t* d_edges, uint64_t* d_edge_count, void* stream) {
    ProfScope ps(PROF_OTHER, (cudaStream_t)stream);
    int rc = launch_canny(d_gray, height, width, blur, low, high, d_workspace, workspace_bytes, d_edges,
                          reinterpret_cast<unsigned long long*>(d_edge_count), (cudaStream_t)stream);
    if (rc == 0) count_launch(blur ? 5 : 4);
    return rc;
}

int fb_roi_laplacian(const uint8_t* d_image, int height, int width, int rgb_order, const int32_t* d_boxes, int k,
                     int64_t* d_out, void* stream) {
    int rc = launch_roi_laplacian(d_image, height, width, rgb_order, d_boxes, k, reinterpret_cast<long long*>(d_out),
                                  (cudaStream_t)stream);
    if (rc == 0) count_launch(1);
    return rc;
}

int fb_clip_preprocess(const uint8_t* d_images, int n, int height, int width, int64_t image_stride, int rgb_order,
                       int out_size, const int32_t* d_hp0, const int32_t* d_hcpad, int hgroups, int h_px_lo,
                       int h_span_px, const int32_t* d_vbounds, const int32_t* d_vcoef, int vk, int row0, int rows,
                       const float* mean3, const float* std3, uint8_t* d_tmp, float* d_out,
                       const int8_t* d_tc_coef, int tc_kw, int tc_limbs, const int32_t* d_tc_kb0, void* stream) {
    ProfScope ps(PROF_PREPROCESS, (cudaStream_t)stream);
    int rc = launch_clip_preprocess(d_images, n, height, width, (long long)image_stride, rgb_order, out_size, d_hp0,
                                    d_hcpad, hgroups, h_px_lo, h_span_px, d_vbounds, d_vcoef, vk, row0, rows, mean3, std3,
                                    d_tmp, d_out, d_tc_coef, tc_kw, tc_limbs, d_tc_kb0, (cudaStream_t)stream);
    if (rc == 0) count_launch(2);
    return rc;
}

int fb_phash(const uint8_t* d_images, int n, int height, int width, int64_t image_stride, int rgb_order,
             const int32_t* d_hbounds, const int32_t* d_hcoef, int hk, const int32_t* d_vbounds, const int32_t* d_vcoef, int vk,
             uint8_t* d_tmp, uint64_t* d_hashes, uint8_t* d_small, double* d_dct, uint8_t* d_luma, int luma_ready,
             const int8_t* d_tc_coef, int tc_kw, int tc_limbs, const int32_t* d_tc_kb0, void* stream) {
    ProfScope ps(PROF_OTHER, (cudaStream_t)stream);
    int rc = launch_phash(d_images, n, height, width, (long long)image_stride, rgb_order, d_hbounds, d_hcoef, hk, d_vbounds,
                          d_vcoef, vk, d_tmp, reinterpret_cast<unsigned long long*>(d_hashes), d_small, d_dct, d_luma, luma_ready,
                          d_tc_coef, tc_kw, tc_limbs, d_tc_kb0, (cudaStream_t)stream);
    if (rc == 0) count_launch(d_luma ? (luma_ready ? 2 : 3) : 2);
    return rc;
}

int fb_thumbnail(const uint8_t* d_images, int n, int height, int width, int64_t image_stride, int fx, int fy, int red_h, int red_w,
                 const uint32_t* mult4, const int32_t* d_hbounds, const int32_t* d_hcoef, int hk, const int32_t* d_vbounds,
                 const int32_t* d_vcoef, int vk, int out_h, int out_w, int swap_rb, uint8_t* d_reduced, uint8_t* d_tmp,
                 uint8_t* d_out, void* stream) {
    ProfScope ps(PROF_OTHER, (cudaStream_t)stream);
    return launch_thumbnail(d_images, n, height, width, (long long)image_stride, fx, fy, red_h, red_w, mult4, d_hbounds, d_hcoef, hk,
                            d_vbounds, d_vcoef, vk, out_h, out_w, swap_rb, d_reduced, d_tmp, d_out, 0, (cudaStream_t)stream);
}

int fb_thumbnail_from_reduced(const uint8_t* d_reduced, int n, int height, int width, int fx, int fy, int red_h, int red_w,
                              const int32_t* d_hbounds, const int32_t* d_hcoef, int hk, const int32_t* d_vbounds,
                              const int32_t* d_vcoef, int vk, int out_h, int out_w, int swap_rb, uint8_t* d_tmp, uint8_t* d_out,
                              void* stream) {
    ProfScope ps(PROF_OTHER, (cudaStream_t)stream);
    FB_REQUIRE(fx > 1 || fy > 1, "fb_thumbnail_from_reduced: no reduction in this plan");
    return launch_thumbnail(nullptr, n, height, width, (long long)height * width * 3, fx, fy, red_h, red_w, nullptr, d_hbounds,
                            d_hcoef, hk, d_vbounds, d_vcoef, vk, out_h, out_w, swap_rb, const_cast<uint8_t*>(d_reduced), d_tmp,
                            d_out, 1, (cudaStream_t)stream);
}

size_t fb_jpeg_encode_workspace_bytes(int n, int height, int width) { return jpeg_encode_workspace_bytes(n, height, width); }
size_t fb_jpeg_encode_out_stride(int height, int width, int header_bytes) { return jpeg_encode_out_stride(height, width, header_bytes); }

int fb_jpeg_encode(const uint8_t* d_rgb, int n, int height, int width, int64_t image_stride, const void* d_tables, const uint8_t* d_header,
                   int header_bytes, void* d_workspace, size_t workspace_bytes, uint8_t* d_out, int64_t out_stride, uint32_t* d_length,
                   void* stream) {
    ProfScope ps(PROF_OTHER, (cudaStream_t)stream);
    int rc = launch_jpeg_encode(d_rgb, n, height, width, (long long)image_stride, d_tables, d_header, header_bytes, d_workspace,
                                workspace_bytes, d_out, (long long)out_stride, d_length, (cudaStream_t)stream);
    if (rc == 0) count_launch(4);
    return rc;
}

int fb_orient(const uint8_t* d_src, int n, int height, int width, int64_t src_stride, int exif_orientation, int swap_rb,
              uint8_t* d_dst, int64_t dst_stride, void* stream) {
    // PIL's transpose method per EXIF orientation (ImageOps.exif_transpose) as (swap, flip_x, flip_y):
    // 1 none, 2 FLIP_LEFT_RIGHT, 3 ROTATE_180, 4 FLIP_TOP_BOTTOM, 5 TRANSPOSE, 6 ROTATE_270, 7 TRANSVERSE, 8 ROTATE_90
    static const int kMethod[9][3] = {{0, 0, 0}, {0, 0, 0}, {0, 1, 0}, {0, 1, 1}, {0, 0, 1}, {1, 0, 0}, {1, 0, 1}, {1, 1, 1}, {1, 1, 0}};
    if (exif_orientation < 1 || exif_orientation > 8) {
        fb::set_error("fb_orient: EXIF orientation %d outside 1..8", exif_orientation);
        return -1;
    }
    ProfScope ps(PROF_OTHER, (cudaStream_t)stream);
    const int* m = kMethod[exif_orientation];
    int rc = launch_orient(d_src, n, height, width, (long long)src_stride, m[0], m[1], m[2], swap_rb, d_dst,
                           (long long)dst_stride, (cudaStream_t)stream);
    if (rc == 0 && n > 0) count_launch(1);
    return rc;
}

int fb_hamming_pairs(const uint64_t* d_hashes, int64_t n, int max_distance, int part, int nparts, int32_t* d_pairs,
                     int64_t cap, uint64_t* d_count, void* stream) {
    ProfScope ps(PROF_HAMMING, (cudaStream_t)stream);
    int rc = launch_hamming_pairs(reinterpret_cast<const unsigned long long*>(d_hashes), (long long)n, max_distance,
                                  part, nparts, d_pairs, (long long)cap,
                                  reinterpret_cast<unsigned long long*>(d_count), (cudaStream_t)stream);
    if (rc == 0 && n >= 2) count_launch(1);
    return rc;
}

int fb_burst_links(const uint64_t* d_hashes, const int64_t* d_time_s, const uint8_t* d_flags, const int32_t* d_lo,
                   int64_t n, int thr, int64_t window_s, double rapid_s, int32_t* d_last_slow,
                   int32_t* d_rapid_pairs, int64_t rapid_cap, uint64_t* d_rapid_count, void* stream) {
    int rc = launch_burst_links(reinterpret_cast<const unsigned long long*>(d_hashes),
                                reinterpret_cast<const long long*>(d_time_s), d_flags, d_lo, (long long)n, thr,
                                (long long)window_s, rapid_s, d_last_slow, d_rapid_pairs, (long long)rapid_cap,
                                reinterpret_cast<unsigned long long*>(d_rapid_count), (cudaStream_t)stream);
    if (rc == 0 && n >= 1) count_launch(1);
    return rc;
}

int fb_gemm_bf16(const void* d_a, int64_t lda, const void* d_b, int64_t ldb, int m, int n, int k, int mode,
                 const float* d_bias, void* d_out, int64_t ldo, const float* d_residual, int64_t ldr, void* stream) {
    ProfScope ps(PROF_GEMM, (cudaStream_t)stream);
    int rc = launch_gemm_bf16(d_a, lda, d_b, ldb, m, n, k, mode, d_bias, d_out, ldo, d_residual, ldr, (cudaStream_t)stream);
    if (rc == 0) count_launch(1);
    return rc;
}

int fb_f32_to_bf16(const float* d_in, void* d_out_bf16, int64_t n, void* stream) {
    int rc = launch_f32_to_bf16(d_in, d_out_bf16, (long long)n, (cudaStream_t)stream);
    if (rc == 0 && n > 0) count_launch(1);
    return rc;
}

int fb_cosine_pairs(const float* d_emb_f32, const void* d_emb_bf16, int64_t n, int dim, float tau, float band,
                    int64_t row_offset, int64_t rows, int32_t* d_cand, float* d_cand_sims, int64_t cand_cap,
                    uint64_t* d_cand_count, int32_t* d_pairs, float* d_sims, int64_t cap, uint64_t* d_count, void* stream) {
    FB_REQUIRE(n >= 1 && n < (1ll << 31), "fb_cosine_pairs: n out of range");
    FB_REQUIRE(d_cand_count && d_count, "fb_cosine_pairs: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    FB_CUDA_OK(cudaMemsetAsync(d_cand_count, 0, sizeof(uint64_t), st));
    FB_CUDA_OK(cudaMemsetAsync(d_count, 0, sizeof(uint64_t), st));
    if (rows <= 0 || n < 2) return 0;
    ProfScope ps(PROF_COSINE, st);
    int rc = launch_cosine_candidates(d_emb_bf16, dim, (int)n, (int)row_offset, (int)rows, dim, tau - band, d_cand, d_cand_sims,
                                      (long long)cand_cap, reinterpret_cast<unsigned long long*>(d_cand_count), st);
    if (rc) return rc;
    rc = launch_cosine_recheck(d_emb_f32, dim, dim, d_cand, reinterpret_cast<unsigned long long*>(d_cand_count),
                               (long long)cand_cap, tau, d_pairs, d_sims, (long long)cap,
                               reinterpret_cast<unsigned long long*>(d_count), st);
    if (rc == 0) count_launch(2);
    return rc;
}

int fb_cosine_block(const void* d_a_bf16, int64_t a_rows, int64_t a_offset, const void* d_b_bf16, int64_t b_rows, int64_t b_offset, int dim,
                    float threshold, int triangle, int32_t* d_cand, float* d_cand_sims, int64_t cand_cap, uint64_t* d_cand_count,
                    void* stream) {
    FB_REQUIRE(a_offset + a_rows < (1ll << 31) && b_offset + b_rows < (1ll << 31) && d_cand_count, "fb_cosine_block: bad arguments");
    if (a_rows <= 0 || b_rows <= 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    ProfScope ps(PROF_COSINE, st);
    int rc = launch_cosine_block(d_a_bf16, (int)a_rows, (int)a_offset, d_b_bf16, (int)b_rows, (int)b_offset, dim, dim, threshold, triangle,
                                 d_cand, d_cand_sims, (long long)cand_cap, reinterpret_cast<unsigned long long*>(d_cand_count), st);
    if (rc == 0) count_launch(1);
    return rc;
}

int fb_cosine_recheck(const float* d_emb_f32, int dim, const int32_t* d_cand, const uint64_t* d_cand_count, int64_t cand_cap, float tau,
                      int32_t* d_pairs, float* d_sims, int64_t cap, uint64_t* d_count, void* stream) {
    FB_REQUIRE(d_cand_count && d_count, "fb_cosine_recheck: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    FB_CUDA_OK(cudaMemsetAsync(d_count, 0, sizeof(uint64_t), st));
    if (cand_cap <= 0) return 0;
    ProfScope ps(PROF_COSINE, st);
    int rc = launch_cosine_recheck(d_emb_f32, dim, dim, d_cand, reinterpret_cast<const unsigned long long*>(d_cand_count),
                                   (long long)cand_cap, tau, d_pairs, d_sims, (long long)cap,
                                   reinterpret_cast<unsigned long long*>(d_count), st);
    if (rc == 0) count_launch(1);
    return rc;
}

size_t fb_vit_workspace_bytes(int batch) { return vit_workspace_bytes(batch); }

int fb_vit_forward(const fb_vit_weights* w, const float* d_clip_in, int batch, void* d_workspace, size_t workspace_bytes,
                   float* d_features, float* d_embedding, float* d_aesthetic_raw, float* d_tag_sims, void* stream) {
    return vit_forward(w, d_clip_in, batch, d_workspace, workspace_bytes, d_features, d_embedding, d_aesthetic_raw,
                       d_tag_sims, (cudaStream_t)stream);
}

int fb_vit_im2col(const float* d_clip_in, int batch, void* d_out_bf16, void* stream) {
    int rc = launch_im2col_patch14(d_clip_in, batch, d_out_bf16, 0, (cudaStream_t)stream);
    if (rc == 0) count_launch(1);
    return rc;
}

int fb_vit_layernorm(const float* d_in, int64_t ld_in, int rows, const float* gamma, const float* beta,
                     const float* class_emb, const float* pos_emb, void* d_out, int64_t ld_out, int out_bf16,
                     void* stream) {
    int rc = launch_layernorm(d_in, ld_in, rows, gamma, beta, class_emb, pos_emb, d_out, ld_out, out_bf16, (cudaStream_t)stream);
    if (rc == 0) count_launch(1);
    return rc;
}

int fb_vit_attention_f16(const void* d_qkv_f16, int batch, void* d_out_f16, void* stream) {
    int rc = launch_attention_tc(d_qkv_f16, batch, d_out_f16, 1, (cudaStream_t)stream);
    if (rc == 0) count_launch(1);
    return rc;
}

int fb_embedding_heads(const float* d_vectors, int n, const float* head_w1, const float* head_b1, const float* head_w2,
                       const float* head_b2, const float* d_tag_emb, int n_tags, float* d_raw, float* d_tag_sims,
                       void* stream) {
    ProfScope ps(PROF_TAIL, (cudaStream_t)stream);
    int rc = launch_embedding_heads(d_vectors, n, head_w1, head_b1, head_w2, head_b2, d_tag_emb, n_tags, d_raw, d_tag_sims,
                                    (cudaStream_t)stream);
    if (rc == 0) count_launch(1);
    return rc;
}

size_t fb_jpeg_workspace_bytes(int n, int width, int height, int ncomp, int h0, int v0, int restart_interval, int64_t max_scan_bytes) {
    return jpeg_workspace_bytes(n, width, height, ncomp, h0, v0, restart_interval, (long long)max_scan_bytes);
}

int fb_jpeg_decode(const uint8_t* d_bytes, const int64_t* d_scan_offset, const int64_t* d_scan_bytes, const int32_t* d_table_slot,
                   const void* d_table_sets, int n, int width, int height, int ncomp, const int32_t* hs3, const int32_t* vs3,
                   const int32_t* tq3, const int32_t* td3, const int32_t* ta3, int restart_interval, int64_t max_scan_bytes, int bgr_order,
                   void* d_workspace, size_t workspace_bytes, uint8_t* d_frames, int64_t frame_stride, int32_t* d_status, void* stream) {
    FB_REQUIRE(hs3 && vs3 && tq3 && td3 && ta3, "fb_jpeg_decode: null component arrays");
    ProfScope ps(PROF_OTHER, (cudaStream_t)stream);
    int rc = launch_jpeg_decode(d_bytes, reinterpret_cast<const long long*>(d_scan_offset), reinterpret_cast<const long long*>(d_scan_bytes),
                                d_table_slot, d_table_sets, n, width, height, ncomp, hs3, vs3, tq3, td3, ta3, restart_interval,
                                (long long)max_scan_bytes, bgr_order, d_workspace, workspace_bytes, d_frames, (long long)frame_stride,
                                d_status, (cudaStream_t)stream);
    if (rc == 0) count_launch(restart_interval > 0 ? 6 : 3);
    return rc;
}

int fb_vit_attention(const void* d_qkv_bf16, int batch, void* d_out_bf16, void* stream) {
    int rc = launch_attention_tc(d_qkv_bf16, batch, d_out_bf16, 0, (cudaStream_t)stream);
    if (rc == 0) count_launch(1);
    return rc;
}

}  // extern "C"
