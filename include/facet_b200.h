/* facet_b200 — C ABI of the B200-native scoring-pass library (libfacet_b200.so).
 *
 * Every entry point takes plain pointers and sizes; there are no torch / C++ types in the
 * signatures.  Device pointers are prefixed d_, host pointers h_.  `stream` is a
 * cudaStream_t passed as void* (NULL = the legacy default stream).  All functions return 0
 * on success, a positive cudaError_t on a CUDA failure and a negative value on a contract
 * violation; fb_last_error() returns the message for the calling thread.
 *
 * Each function cites the reference interface it replaces (paths under rlorenzo/facet).
 * The Python host mirror (facet_b200/analyzers, facet_b200/processing, facet_b200/utils)
 * binds these symbols with ctypes; INTEGRATION.md shows the stub a reference maintainer adds.
 */
#ifndef FACET_B200_H_
#define FACET_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FB_ABI_VERSION 1
#define FB_HS_BINS (180 * 256)

int fb_abi_version(void);
const char* fb_last_error(void);
/* Number of kernels this library has launched in the calling process (bench gpu_launches). */
uint64_t fb_launch_count(void);
int fb_device_sm_count(void);

/* Optional CUDA-event timing of the library's own launches, per kernel family, on the launching stream
 * (used by bench.py for the roofline of the timed region).  Categories: 0 technical, 1 hs-derive,
 * 2 preprocess, 3 im2col, 4 tcgen05 GEMM, 5 layernorm, 6 attention, 7 ViT tail, 8 cosine stage,
 * 9 hamming/burst, 10 other.  fb_profile_read synchronises the device, fills the two arrays
 * (>= FB_PROFILE_CATEGORIES entries) and resets the recording. */
#define FB_PROFILE_CATEGORIES 11
void fb_profile_enable(int on);
int fb_profile_read(double* ms_per_category, uint64_t* launches_per_category, int n_categories);

/* ---------------------------------------------------------------------------------------
 * Technical metrics — replaces analyzers/image_cache.py:22-32 (ImageCache: gray, hsv,
 * Laplacian variance) and the pixel passes of analyzers/technical.py:94 (H-S calcHist),
 * :153 (luminance calcHist), :263-264/:326 (percentiles — derived from hist256),
 * :302 (Immerkaer filter2D sum).
 *
 * d_images   [n][height][width][3] uint8, interleaved, C-contiguous rows; image i starts at
 *            d_images + i*image_stride.  rgb_order = 0 for the reference's BGR arrays
 *            (utils/image_loading.py:106), 1 for RGB.
 * d_hist256  [n][256]      uint32  luminance histogram (exact counts)
 * d_hs_hist  [n][180][256] uint32  hue x saturation histogram (exact counts)
 * d_sums     [n][4]        int64   { sum Laplacian, sum Laplacian^2, sum |Immerkaer|, 0 }
 * force_generic != 0 selects the any-shape kernel (used by tests as a second opinion).
 * Outputs are overwritten.  Images must be at least 2x2 (reflect-101 borders).
 */
int fb_tech_stats(const uint8_t* d_images, int n, int height, int width, int64_t image_stride,
                  int rgb_order, uint32_t* d_hist256, uint32_t* d_hs_hist, int64_t* d_sums,
                  int force_generic, void* stream);

/* Same pass, additionally writing Pillow's luma plane (convert('L'): (19595 R + 38470 G + 7471 B + 2^15) >> 16)
 * to d_luma [n][height][width] uint8 — the input of the perceptual hash's resampler (fb_phash with
 * luma_ready = 1), so the frame is read from HBM once for both.  Needs a contiguous batch. */
int fb_tech_stats_luma(const uint8_t* d_images, int n, int height, int width, int64_t image_stride,
                       int rgb_order, uint32_t* d_hist256, uint32_t* d_hs_hist, int64_t* d_sums,
                       int force_generic, uint8_t* d_luma, void* stream);

/* Same pass with both side products of the single read of the frame (either may be NULL): d_luma as in
 * fb_tech_stats_luma, and d_box4 [n][ceil(height/4)][width/4 rounded up][3] uint8 = Pillow's ImagingReduce by (4, 4) of
 * the frame, ((sum + count/2) * multiplier) >> 24 per channel in the frame's channel order — the first step of
 * `thumb.thumbnail((640, 640), LANCZOS)` on a 24 MP frame (utils/image_transforms.py:32-50, scorer.py:1681-1686), so the
 * thumbnail needs no read of the frame of its own (fb_thumbnail_from_reduced finishes it).  box_mult4: HOST array of
 * Pillow's multipliers for the (full, right-edge, bottom-edge, corner) boxes, as for fb_thumbnail.  Shapes the fused
 * kernel does not take (width not a multiple of 8) run the separate reduction pass after the generic kernel. */
int fb_tech_stats_fused(const uint8_t* d_images, int n, int height, int width, int64_t image_stride,
                        int rgb_order, uint32_t* d_hist256, uint32_t* d_hs_hist, int64_t* d_sums,
                        uint8_t* d_luma, uint8_t* d_box4, const uint32_t* box_mult4, void* stream);

/* Per-image reductions of the H-S histogram — technical.py:97-104 (entropy) and :237
 * (mean saturation).  d_out [n][4] float64 = { entropy_bits, sum_saturation, nonzero_bins,
 * total_count }. */
int fb_tech_derive(const uint32_t* d_hs_hist, int n, double* d_out, void* stream);

/* Host-buffer convenience for the same pass (the call the reference-facing plugin makes with
 * numpy arrays): H2D copy, both kernels, D2H copy, synchronises.  h_hs_hist may be NULL. */
int fb_tech_stats_host(const uint8_t* h_images, int n, int height, int width, int rgb_order,
                       uint32_t* h_hist256, int64_t* h_sums, double* h_derived,
                       uint32_t* h_hs_hist);

/* gray [H][W] and hsv [H][W][3] uint8 planes of one image — the arrays ImageCache exposes
 * (analyzers/image_cache.py:30-31) for callers outside the technical metrics. */
int fb_gray_hsv(const uint8_t* d_image, int height, int width, int rgb_order, uint8_t* d_gray,
                uint8_t* d_hsv, void* stream);

/* Edge maps of the rule-based composition analyzer (analyzers/composition.py; called per image at
 * processing/batch_processor.py:245 `CompositionAnalyzer.detect_leading_lines(img_cv, cache=cache)` and, through
 * `get_placement_data(..., img_cv=...)`, `detect_subject_region`).
 *   fb_gray_plane  gray [H][W] uint8 = cv2.cvtColor(BGR2GRAY) (composition.py:30,210) and, when d_hist256 is not
 *                  NULL, its 256-bin histogram (np.median(gray), composition.py:33, is a closed form of it)
 *   fb_canny       blur != 0: cv2.GaussianBlur(gray, (5, 5), 0) first (composition.py:215); then
 *                  cv2.Canny(src, low, high) (composition.py:218 with 50 / 150; :36 with the median-derived
 *                  thresholds): aperture 3, L1 gradient.  d_edges [H][W] uint8, 0 or 255, bit-exact with OpenCV;
 *                  d_edge_count (device uint64, may be NULL) receives the number of edge pixels.
 *                  d_workspace: fb_canny_workspace_bytes(height, width) bytes, 256-byte aligned.
 * The sequential geometry that follows (cv2.HoughLinesP, cv2.findContours) stays with the caller. */
int fb_gray_plane(const uint8_t* d_image, int height, int width, int rgb_order, uint8_t* d_gray, uint32_t* d_hist256,
                  void* stream);
size_t fb_canny_workspace_bytes(int height, int width);
int fb_canny(const uint8_t* d_gray, int height, int width, int blur, int low, int high, void* d_workspace,
             size_t workspace_bytes, uint8_t* d_edges, uint64_t* d_edge_count, void* stream);

/* Laplacian sums of image crops — analyzers/face.py:272-279 `_get_crop_sharpness`
 * (isolation bonus, processing/batch_processor.py:254-260).  Each crop is filtered with its
 * own reflect-101 border.  d_boxes [k][4] int32 = x1,y1,x2,y2 (exclusive end, clipped by the
 * caller); d_out [k][3] int64 = { pixel count, sum Laplacian, sum Laplacian^2 }. */
int fb_roi_laplacian(const uint8_t* d_image, int height, int width, int rgb_order,
                     const int32_t* d_boxes, int k, int64_t* d_out, void* stream);

/* ---------------------------------------------------------------------------------------
 * CLIP preprocess — replaces `scorer.preprocess` (processing/scorer.py:508-510, used at
 * processing/batch_processor.py:95): torchvision Resize(shorter side, BICUBIC, antialias on
 * PIL) -> CenterCrop -> ToTensor -> Normalize.  Bit-exact with Pillow's 8-bit resampler
 * (22-bit fixed-point coefficients, horizontal pass first, uint8 intermediate).
 *
 * The caller supplies the coefficient tables (facet_b200/utils/resample.py computes them the
 * way Pillow's precompute_coeffs/normalize_coeffs_8bpc do):
 *   horizontal pass, per output column xo: d_hp0[xo] = first tap rounded down to a multiple of 4
 *   pixels, d_hcpad[4*hgroups][out] = coefficient of pixel d_hp0[xo]+i at [i][xo] (zero padded);
 *   h_px_lo (multiple of 16) / h_span_px (multiple of 16) = pixel range of a row that is staged
 *   vertical pass: d_vbounds [out][2] int32 (first tap, tap count), d_vcoef [out][vk] int32
 *   row0/rows = input rows the vertical taps touch (the only rows pass 1 produces)
 * d_tmp      scratch [n][rows][out][3] uint8 (horizontal pass output)
 * d_out      [n][3][out][out] float32, planes R,G,B, (x/255 - mean[c]) / std[c]
 * mean3/std3 are HOST pointers to 3 floats each.
 * Optional tensor-core tables (NULL/0 to skip): the horizontal pass as an exact u8 x s8 -> s32
 * tcgen05 product.  Per block j of 8 output columns, d_tc_coef holds an int8 matrix [96][tc_kw]
 * (row = limb*24 + (xo-8j)*3 + channel, column = byte - d_tc_kb0[j]) of the signed base-128 limbs of
 * the taps (tc_limbs = 3 or 4).  Used when width % 16 == 0 and the batch is contiguous; the CUDA-core
 * kernel with d_hp0/d_hcpad is the general path.
 */
int fb_clip_preprocess(const uint8_t* d_images, int n, int height, int width, int64_t image_stride,
                       int rgb_order, int out_size,
                       const int32_t* d_hp0, const int32_t* d_hcpad, int hgroups,
                       int h_px_lo, int h_span_px,
                       const int32_t* d_vbounds, const int32_t* d_vcoef, int vk,
                       int row0, int rows,
                       const float* mean3, const float* std3,
                       uint8_t* d_tmp, float* d_out,
                       const int8_t* d_tc_coef, int tc_kw, int tc_limbs, const int32_t* d_tc_kb0,
                       void* stream);

/* ---------------------------------------------------------------------------------------
 * Perceptual hash — replaces `imagehash.phash(pil_img)` (processing/batch_processor.py:216,
 * processing/scorer.py:972, processing/multi_pass.py:449): Pillow convert('L') -> resize((32,32), LANCZOS)
 * -> 2-D DCT-II -> top-left 8x8 > median, 64 bits row-major MSB first (str(ImageHash) = "%016x").
 * Coefficient tables ([32][2] bounds + [32][k] int32 taps per axis, Pillow's Lanczos taps) come from
 * facet_b200/utils/resample.py.  d_tmp scratch [n][height][32] uint8.  d_small ([n][32][32] uint8, the
 * resized luma) and d_dct ([n][64] float64, the low-frequency block) are optional debug outputs.
 * Optional tensor-core route (width % 16 == 0, contiguous batch): d_luma scratch [n][height][width] uint8
 * receives Pillow's luma plane and the horizontal Lanczos pass runs as a u8 x s8 tcgen05 product with
 * the int8 limb tables d_tc_coef [4*32][tc_kw] / d_tc_kb0 [4] (same layout as fb_clip_preprocess, one
 * channel); pass NULL/0 to use the CUDA-core kernel.  luma_ready = 1: d_luma was already filled by
 * fb_tech_stats_luma (the frame is then not read again). */
int fb_phash(const uint8_t* d_images, int n, int height, int width, int64_t image_stride, int rgb_order,
             const int32_t* d_hbounds, const int32_t* d_hcoef, int hk,
             const int32_t* d_vbounds, const int32_t* d_vcoef, int vk,
             uint8_t* d_tmp, uint64_t* d_hashes, uint8_t* d_small, double* d_dct,
             uint8_t* d_luma, int luma_ready,
             const int8_t* d_tc_coef, int tc_kw, int tc_limbs, const int32_t* d_tc_kb0,
             void* stream);

/* Photo thumbnail — the pixel work of utils/image_transforms.py:32-50 `generate_photo_thumbnail`
 * (`thumb.thumbnail((size, size), Image.Resampling.LANCZOS)`, called when a photo row is saved,
 * processing/scorer.py:1681-1686).  Pillow's algorithm, bit-exact: box reduction by (fx, fy) =
 * int(scale / reducing_gap) with ((sum + n/2) * mult) >> 24 (mult4 = multipliers of the full, right-edge,
 * bottom-edge and corner boxes), then the two-pass 8-bit Lanczos resampler on the reduced image with the
 * 22-bit taps of facet_b200/utils/thumbnail.py (d_hbounds [out_w][2], d_hcoef [out_w][hk], d_vbounds
 * [out_h][2], d_vcoef [out_h][vk]).  d_reduced [n][red_h][red_w][3] (may be NULL when fx = fy = 1),
 * d_tmp [n][red_h][out_w][3], d_out [n][out_h][out_w][3]; swap_rb reverses the channel order of the
 * output (BGR frames -> RGB thumbnails).  The JPEG encoding stays with the caller. */
int fb_thumbnail(const uint8_t* d_images, int n, int height, int width, int64_t image_stride, int fx, int fy,
                 int red_h, int red_w, const uint32_t* mult4,
                 const int32_t* d_hbounds, const int32_t* d_hcoef, int hk,
                 const int32_t* d_vbounds, const int32_t* d_vcoef, int vk,
                 int out_h, int out_w, int swap_rb, uint8_t* d_reduced, uint8_t* d_tmp, uint8_t* d_out, void* stream);

/* The two Lanczos passes of fb_thumbnail on a reduced image that already exists (d_reduced [n][red_h][red_w][3], e.g.
 * written by fb_tech_stats_fused with fx = fy = 4); height / width are those of the original frames. */
int fb_thumbnail_from_reduced(const uint8_t* d_reduced, int n, int height, int width, int fx, int fy, int red_h, int red_w,
                              const int32_t* d_hbounds, const int32_t* d_hcoef, int hk,
                              const int32_t* d_vbounds, const int32_t* d_vcoef, int vk,
                              int out_h, int out_w, int swap_rb, uint8_t* d_tmp, uint8_t* d_out, void* stream);

/* JPEG encoding of the thumbnails — the encoder half of utils/image_transforms.py:32-50 `generate_photo_thumbnail`
 * (`thumb.save(buf, format='JPEG', quality=80)`, processing/scorer.py:1681-1686), byte-exact with Pillow / libjpeg(-turbo) at its
 * defaults: YCbCr 4:2:0, standard Huffman tables, no restart markers (colour conversion, h2v2 downsampling with edge replication,
 * jpeg_fdct_islow, round-half-up quantisation, dummy blocks, Huffman coding with 0xFF stuffing and one-bit padding).
 *   d_rgb     [n][height][width][3] uint8, RGB
 *   d_tables  3328 bytes as packed by facet_b200/utils/jpeg.py `encoder_tables`: uint16 q8[2][64] (8 x quantisation value, natural
 *             order, luma / chroma), uint16 code[4][256], uint8 size[4][256] (DC luma, AC luma, DC chroma, AC chroma)
 *   d_header  the header_bytes bytes SOI .. end of the SOS header that Pillow writes for this size and quality (they do not depend
 *             on the pixels)
 *   d_out     [n] slots of out_stride >= fb_jpeg_encode_out_stride(height, width, header_bytes) bytes; d_length [n] uint32 receives
 *             the length of every stream (header + entropy-coded data + EOI)
 *   d_workspace  fb_jpeg_encode_workspace_bytes(n, height, width) bytes, 256-byte aligned */
size_t fb_jpeg_encode_workspace_bytes(int n, int height, int width);
size_t fb_jpeg_encode_out_stride(int height, int width, int header_bytes);
int fb_jpeg_encode(const uint8_t* d_rgb, int n, int height, int width, int64_t image_stride, const void* d_tables,
                   const uint8_t* d_header, int header_bytes, void* d_workspace, size_t workspace_bytes, uint8_t* d_out,
                   int64_t out_stride, uint32_t* d_length, void* stream);

/* ---------------------------------------------------------------------------------------
 * Frame orientation — the pixel work of utils/image_loading.py:101-106 for frames already in device
 * memory: ImageOps.exif_transpose (PIL transpose method chosen by EXIF tag 0x0112: 2 FLIP_LEFT_RIGHT,
 * 3 ROTATE_180, 4 FLIP_TOP_BOTTOM, 5 TRANSPOSE, 6 ROTATE_270, 7 TRANSVERSE, 8 ROTATE_90, 1 none)
 * followed, when swap_rb, by cv2.cvtColor(RGB2BGR).  d_src [n][height][width][3], d_dst
 * [n][height'][width'][3] with (height', width') = (width, height) for orientations 5..8; strides in
 * bytes between images; d_dst must not alias d_src. */
int fb_orient(const uint8_t* d_src, int n, int height, int width, int64_t src_stride, int exif_orientation, int swap_rb,
              uint8_t* d_dst, int64_t dst_stride, void* stream);

/* ---------------------------------------------------------------------------------------
 * JPEG decoding — replaces the decode of `load_image_from_path` (utils/image_loading.py:90-106: `Image.open(path)`,
 * `.convert('RGB')` through Pillow / libjpeg-turbo, `cv2.cvtColor(RGB2BGR)`), byte-exact with Pillow's output:
 * Huffman decoding (one thread per restart interval; streams without restart markers above 1024 MCUs by
 * self-synchronising parallel decoding), dequantisation + libjpeg's `jpeg_idct_islow`, h2v1 / h2v2 "fancy" chroma
 * upsampling, `ycc_rgb_convert`.  One call decodes a batch of streams of EQUAL geometry (size,
 * components, sampling factors, restart interval); tables may differ per stream.
 *
 * d_bytes         the streams' bytes, concatenated anywhere in one device buffer
 * d_scan_offset   [n] int64: offset of each stream's entropy-coded segment (first byte after the SOS header) in d_bytes
 * d_scan_bytes    [n] int64: length of that segment (up to, not including, the EOI marker)
 * d_table_slot    [n] int32: index of the stream's table set in d_table_sets
 * d_table_sets    table sets as laid out by facet_b200/utils/jpeg.py `pack_tables` (11904 bytes each: uint16 q[4][64]
 *                 in row-major order, then 4 DC and 4 AC Huffman tables: uint16 lut[512] (9-bit lookahead,
 *                 length << 8 | symbol), int32 maxcode[18], int32 valptr[17], uint8 values[256], 4 bytes padding)
 * hs3 .. ta3      HOST arrays of 3 ints: sampling factors, quantisation / DC / AC table ids per component
 *                 (luma 1x1, 2x1 or 2x2 with 1x1 chroma; ncomp = 1 uses entry 0 with 1x1)
 * restart_interval  MCUs per restart interval (DRI), 0 = none
 * d_frames        [n][height][width][3] uint8, BGR when bgr_order (what the analyzers take) else RGB
 * d_status        [n] int32: 0 ok, bit 0 = restart markers do not match the header, bit 1 = invalid / truncated Huffman data,
 *                 bit 2 = the self-synchronisation rounds did not settle (48 rounds)
 * The orientation (EXIF) is not applied here: fb_orient does that on the decoded frames. */
size_t fb_jpeg_workspace_bytes(int n, int width, int height, int ncomp, int h0, int v0, int restart_interval, int64_t max_scan_bytes);
int fb_jpeg_decode(const uint8_t* d_bytes, const int64_t* d_scan_offset, const int64_t* d_scan_bytes, const int32_t* d_table_slot,
                   const void* d_table_sets, int n, int width, int height, int ncomp, const int32_t* hs3, const int32_t* vs3,
                   const int32_t* tq3, const int32_t* td3, const int32_t* ta3, int restart_interval, int64_t max_scan_bytes, int bgr_order,
                   void* d_workspace, size_t workspace_bytes, uint8_t* d_frames, int64_t frame_stride, int32_t* d_status, void* stream);

/* ---------------------------------------------------------------------------------------
 * Duplicate / burst grouping — replaces the O(N^2) loop of utils/duplicate.py:94-119 and the
 * pairwise predicate of processing/scorer.py:1943-1968.
 *
 * fb_hamming_pairs: all pairs (i, j), i < j, i in this part's rows, with
 * popcount(h[i]^h[j]) <= max_distance.  The upper-triangle tiles of the pair matrix are dealt to the
 * parts round-robin (tile t of the row-major enumeration belongs to part t % nparts; tiles are 256 x 256
 * hashes up to n = 65536 and 2048 x 2048 above), so a triangular problem balances across GPUs to within
 * one tile and small sets still spread over every part.  d_pairs [cap][2] int32 receives the pairs in
 * no particular order; *d_count (uint64, device) receives how many pairs exist — if it exceeds cap the
 * list is truncated and the caller retries with a larger buffer.
 */
int fb_hamming_pairs(const uint64_t* d_hashes, int64_t n, int max_distance, int part, int nparts,
                     int32_t* d_pairs, int64_t cap, uint64_t* d_count, void* stream);

/* fb_burst_links: for photo i (rows in the reference's ORDER BY date_taken order) the largest
 * b in [d_lo[i], i) that satisfies the "slow" rule |t_i - t_b| <= window_s && hamming <= thr
 * (scorer.py:1962-1965), or -1.  Candidates of the "rapid" rule (|dt| <= rapid_s &&
 * hamming <= 2*thr, scorer.py:1957-1960) are appended to d_rapid_pairs [(i,b)] so the host can
 * apply the shares_person check.  d_flags[i]: bit0 = date parsed (scorer.py:1946-1952),
 * bit1 = hash present (scorer.py:1927-1929).  d_lo[i] is a host-computed lower bound of the
 * window (any b < d_lo[i] is farther than window_s from i). */
int fb_burst_links(const uint64_t* d_hashes, const int64_t* d_time_s, const uint8_t* d_flags,
                   const int32_t* d_lo, int64_t n, int thr, int64_t window_s, double rapid_s,
                   int32_t* d_last_slow, int32_t* d_rapid_pairs, int64_t rapid_cap,
                   uint64_t* d_rapid_count, void* stream);

/* Cosine mode of the similarity stage (north_star kernel 3): all pairs (i<j), i in
 * [row_offset, row_offset+rows), with <e_i, e_j> >= tau on the stored L2-normalised float32
 * embeddings (formula sites models/tagger.py:99-101, api/routers/gallery.py:465-471; grouping as
 * utils/duplicate.py).  The N x N product runs as a bf16 tcgen05 GEMM whose epilogue emits
 * candidates with sim >= tau - band into d_cand; they are then re-scored from d_emb_f32 with float64
 * accumulation (pair kept iff double(dot) >= double(tau): order-independent to ~1e-13, unlike a float32 dot)
 * and the survivors written to d_pairs [(i,j)] / d_sims (the dot rounded to float32).  Counts above the capacities mean the
 * lists were truncated (caller retries with larger buffers).  band >= 2^-8 is loss-free. */
int fb_f32_to_bf16(const float* d_in, void* d_out_bf16, int64_t n, void* stream);
int fb_cosine_pairs(const float* d_emb_f32, const void* d_emb_bf16, int64_t n, int dim, float tau, float band,
                    int64_t row_offset, int64_t rows, int32_t* d_cand, float* d_cand_sims, int64_t cand_cap,
                    uint64_t* d_cand_count, int32_t* d_pairs, float* d_sims, int64_t cap, uint64_t* d_count,
                    void* stream);

/* The two halves of fb_cosine_pairs as separate calls, for the multi-GPU flow (utils/duplicate.py `cosine_pairs_sharded`):
 * the scan needs only bf16 rows, so the all-gather of the float32 rows (twice the bytes) runs on the NCCL stream WHILE the
 * scan computes; the recheck waits for it.
 * fb_cosine_block scans one shard-against-shard block and emits (i, j, bf16 sim) with sim >= threshold (= tau - band): the
 * a_rows rows at d_a_bf16 (global row index a_offset + i) against the b_rows rows at d_b_bf16 (global index b_offset + j), both
 * [rows][dim] bf16 with row pitch dim.  triangle != 0 keeps only global column > global row (the block of a shard against
 * itself); rectangular blocks report every hit as (global row, global column) — the caller orders the pair.  Candidates are
 * APPENDED: d_cand_count is not reset, so a rank's blocks fill one list.  A rank can scan its own shard against itself while
 * the all-gather of the other shards is still in flight.
 * fb_cosine_recheck keeps the candidates whose float64-accumulated dot product of the float32 rows is >= tau. */
int fb_cosine_block(const void* d_a_bf16, int64_t a_rows, int64_t a_offset, const void* d_b_bf16, int64_t b_rows,
                    int64_t b_offset, int dim, float threshold, int triangle, int32_t* d_cand, float* d_cand_sims,
                    int64_t cand_cap, uint64_t* d_cand_count, void* stream);
int fb_cosine_recheck(const float* d_emb_f32, int dim, const int32_t* d_cand, const uint64_t* d_cand_count, int64_t cand_cap, float tau,
                      int32_t* d_pairs, float* d_sims, int64_t cap, uint64_t* d_count, void* stream);

/* ---------------------------------------------------------------------------------------
 * CLIP ViT-L/14 image tower + heads — replaces `self.model.encode_image(inputs)`,
 * `F.normalize(features)`, `self.aesthetic_head(features.float())`
 * (processing/scorer.py:661-664; twins at :596, :610 and processing/multi_pass.py:523) and the
 * tag similarity `image_features @ self.text_embeddings.T` (models/tagger.py:99-101).
 *
 * fb_gemm_bf16: C[M,N] = A[M,K] * B[N,K]^T on tcgen05 tensor cores, A/B bf16 row-major
 * (K-major; a PyTorch Linear weight [out,in] is B as is), K % 64 == 0, N % 32 == 0.
 * Epilogue modes: 0 bf16 out = acc + bias; 1 bf16 out = gelu_erf(acc + bias);
 * 2 f32 out = acc + bias + residual (out may alias residual); 3 f32 out = acc (+ bias). */
#define FB_GEMM_BIAS_BF16 0
#define FB_GEMM_BIAS_GELU_BF16 1
#define FB_GEMM_BIAS_RESIDUAL_F32 2
#define FB_GEMM_F32 3
#define FB_GEMM_F16_FLAG 16   /* OR into mode: operands and 16-bit outputs are IEEE fp16 instead of bf16 */
int fb_gemm_bf16(const void* d_a, int64_t lda, const void* d_b, int64_t ldb, int m, int n, int k, int mode,
                 const float* d_bias, void* d_out, int64_t ldo, const float* d_residual, int64_t ldr,
                 void* stream);

/* Device pointers of one packed ViT-L/14 (width 1024, 24 layers, 16 heads, MLP 4096, patch 14,
 * 224 px, 257 tokens, output 768).  GEMM weights are bf16 [out][in]; everything else fp32. */
typedef struct fb_vit_layer {
    const float *ln1_g, *ln1_b, *ln2_g, *ln2_b;
    const void *w_qkv;  const float *b_qkv;    /* [3072][1024] bf16, [3072] */
    const void *w_out;  const float *b_out;    /* [1024][1024] */
    const void *w_fc;   const float *b_fc;     /* [4096][1024] */
    const void *w_proj; const float *b_proj;   /* [1024][4096] */
    /* LayerNorm fold (optional, all six or none; used when fb_vit_weights.fused_ln != 0): the two LayerNorms of the block are
     * folded into the GEMMs that consume them.  w_*_ln = the weight with LayerNorm's gain on its input columns
     * (W[n][k] * gamma[k], 16-bit), s_* [n] = sum_k of those 16-bit values, c_* [n] = sum_k beta[k] * W[n][k] + b[n].  The
     * residual GEMM in front writes the 16-bit copy of the residual stream and per-row sums; LayerNorm(x) W^T + b is then
     * rstd_r * (x16 W_ln^T - mean_r * s) + c in the consumer's epilogue: no LayerNorm pass over the residual stream. */
    const void *w_qkv_ln; const float *s_qkv; const float *c_qkv;
    const void *w_fc_ln;  const float *s_fc;  const float *c_fc;
} fb_vit_layer;

typedef struct fb_vit_weights {
    const void *w_patch;                       /* [1024][640] bf16: conv1 weight flattened (c,ky,kx), zero padded */
    const float *class_emb;                    /* [1024] */
    const float *pos_emb;                      /* [257][1024] */
    const float *ln_pre_g, *ln_pre_b, *ln_post_g, *ln_post_b;
    const float *proj;                         /* [1024][768] fp32 */
    const float *head_w1, *head_b1;            /* aesthetic head Linear(768,256): [256][768], [256] (scorer.py:578-582) */
    const float *head_w2, *head_b2;            /* Linear(256,1): [256], [1] */
    const float *tag_emb;                      /* [n_tags][768] L2-normalised text embeddings (tagger.py:73) or NULL */
    int n_tags;
    int f16;                                   /* 0: 16-bit weights/activations are bf16; 1: IEEE fp16 (the reference runs
                                                  `.half()` on CUDA, processing/scorer.py:515) */
    int n_layers;                              /* 24 */
    const fb_vit_layer *layers;                /* HOST array of n_layers entries */
    int fused_ln;                              /* != 0: use the layers' LayerNorm-fold fields (see fb_vit_layer) */
} fb_vit_weights;

size_t fb_vit_workspace_bytes(int batch);

/* d_clip_in [batch][3][224][224] float32 (output of fb_clip_preprocess).  Outputs (device):
 * d_features [batch][768] un-normalised, d_embedding [batch][768] L2-normalised,
 * d_aesthetic_raw [batch] (the reference maps it with clip((raw+1)*5, 0, 10), scorer.py:669),
 * d_tag_sims [batch][n_tags] (may be NULL when n_tags == 0). */
int fb_vit_forward(const fb_vit_weights* w, const float* d_clip_in, int batch, void* d_workspace,
                   size_t workspace_bytes, float* d_features, float* d_embedding, float* d_aesthetic_raw,
                   float* d_tag_sims, void* stream);

/* Individual stages (exposed for tests and for callers that schedule the tower themselves). */
int fb_vit_im2col(const float* d_clip_in, int batch, void* d_out_bf16, void* stream);
int fb_vit_layernorm(const float* d_in, int64_t ld_in, int rows, const float* gamma, const float* beta,
                     const float* class_emb, const float* pos_emb, void* d_out, int64_t ld_out,
                     int out_bf16 /* 0 fp32, 1 bf16, 2 fp16 */, void* stream);
int fb_vit_attention(const void* d_qkv_bf16, int batch, void* d_out_bf16, void* stream);      /* tcgen05 */
int fb_vit_attention_f16(const void* d_qkv_f16, int batch, void* d_out_f16, void* stream);     /* tcgen05, fp16 operands */

/* Heads on stored embeddings (no tower) — replaces the two per-image calls of the reference that start from the
 * 3072-byte `clip_embedding` BLOB: `Facet.score_from_embedding` (processing/scorer.py:620-629, the MLP head on the
 * vector as stored) and `CLIPTagger.get_tags_from_embedding`'s product (models/tagger.py:99-101, emb @ T^T).
 * d_vectors [n][768] float32.  d_raw [n] (NULL to skip the head; head_* as in fb_vit_weights) and
 * d_tag_sims [n][n_tags] (n_tags = 0 to skip). */
int fb_embedding_heads(const float* d_vectors, int n, const float* head_w1, const float* head_b1, const float* head_w2,
                       const float* head_b2, const float* d_tag_emb, int n_tags, float* d_raw, float* d_tag_sims,
                       void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FACET_B200_H_ */
