// Horizontal pass of Pillow's 8-bit resampler as an exact int8 tensor-core product.
//
// Part of `scorer.preprocess` (processing/scorer.py:508-510).  For a block of 8 output columns the
// pass is  tmp[row, xo, c] = clip8((2^21 + sum_x img[row, x, c] * k[xo, x]) >> 22), i.e. a matrix product
// of the image rows (uint8, interleaved channels, K = byte offset inside the block's window) with a
// banded coefficient matrix.  Coefficients are 22-bit fixed point, so they are split into signed base-128
// limbs (int8): the product is evaluated exactly with tcgen05.mma.kind::i8 (u8 x s8 -> s32) and the limbs
// are recombined in the epilogue.
//   A  image bytes [n*H rows][W*3] uint8, K-major, TMA boxes of 128 rows x 128 bytes (128-byte swizzle)
//   B  per column block j: [96][KW] int8, row = limb*24 + (xo-8j)*3 + c, K = byte - kb0[j]   (host table)
//   D  [128 rows][96] int32 in TMEM (two buffers), epilogue: one thread per row, 24 output bytes
// Persistent CTAs, 6 warps: TMA producer, MMA issuer, 4 epilogue warps; 6-stage mbarrier ring.
// Two schedules:
//   resident  (resample_h_tc_resident_kernel) a CTA keeps ONE column block for the whole launch: its coefficient matrix
//             (72 KB for the CLIP resize of a 24 MP frame) is loaded into shared memory once and only image rows stream
//             through an 8-stage ring.  CTA c works on block c % nblk and on every (grid / nblk)-th 128-row tile, so the
//             CTAs that read overlapping windows of the same rows run at the same time (L2 hits).  The streaming schedule
//             re-loaded the coefficients with every tile: 72 of the 168 KB per tile, and the L2 -> shared-memory path
//             (about 64 B / clk / SM) is what bounds this pass.
//   streaming (resample_h_tc_kernel) tile = (rows, block), coefficients loaded with every tile: shapes whose coefficient
//             matrix does not fit beside the ring, or with more blocks than SMs.
#include "common.cuh"
#include "kernels.h"
#include "tc_common.cuh"

namespace fb {

namespace {

constexpr int RM = 128, RKB = 128, RSTAGES = 6;
constexpr int kABytesR = RM * RKB;        // 16 KB
constexpr int kThreadsR = 192;
constexpr int kNB = 8;                    // output columns per block
constexpr int kPrec = 32 - 8 - 2;
template <int CH> struct RCfg {
    static constexpr int RN = CH == 3 ? 96 : 32;          // coefficient rows per block: limb * (8*CH) + (xo-8j)*CH + c, padded
    static constexpr int kBBytes = RN * RKB;
    static constexpr int kStage = kABytesR + kBBytes;
    static constexpr int kSmem = RSTAGES * kStage + 1024 + 256;
};

struct ResampleTcArgs {
    int n_img, H, row0, rows;             // rows [row0, row0+rows) of every image are produced
    int out;                              // output columns (multiple of 8)
    int kblocks;                          // KW / 128
    int limbs;                            // 3 or 4
    const int* kb0;                       // [out/8] first byte of each block's window (multiple of 16)
    uint8_t* tmp;                         // [n][rows][out][CH]
};

// kind::i8: D = s32 (c_format 2), A = unsigned 8 bit (0), B = signed 8 bit (1), both K-major
__host__ __device__ constexpr uint32_t make_idesc_u8s8(int m, int n) {
    return (2u << 4) | (0u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}

template <int CH>
__global__ void __launch_bounds__(kThreadsR, 1)
resample_h_tc_kernel(const __grid_constant__ CUtensorMap tmap_img, const __grid_constant__ CUtensorMap tmap_coef, ResampleTcArgs p) {
    constexpr int RN = RCfg<CH>::RN;
    constexpr int kStageR = RCfg<CH>::kStage;
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment by pointer arithmetic on the shared pointer (a round trip through an integer would
    // make every later access a generic LD/ST instead of LDS/STS)
    uint8_t* smem = smem_raw + ((1024u - ((uint32_t)__cvta_generic_to_shared(smem_raw) & 1023u)) & 1023u);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + RSTAGES * kStageR);
    uint64_t* full_bar = bars;
    uint64_t* empty_bar = bars + RSTAGES;
    uint64_t* tmem_full = bars + 2 * RSTAGES;
    uint64_t* tmem_empty = bars + 2 * RSTAGES + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * RSTAGES + 4);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nblk = p.out / kNB;
    const int mtiles_img = (p.rows + RM - 1) / RM;
    const int num_tiles = p.n_img * mtiles_img * nblk;

    if (threadIdx.x == 0) {
        for (int s = 0; s < RSTAGES; ++s) {
            tc::mbar_init(&full_bar[s], 1);
            tc::mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            tc::mbar_init(&tmem_full[a], 1);
            tc::mbar_init(&tmem_empty[a], 4);
        }
        tc::mbar_fence_init();
        tc::fence_proxy_async();
        tc::tma_prefetch_desc(&tmap_img);
        tc::tma_prefetch_desc(&tmap_coef);
    }
    if (warp == 1) tc::tmem_alloc(tmem_slot, 256);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // tile -> (image, m-tile inside the image, column block); column block fastest: 28 blocks share the rows in L2
    auto decode = [&](int tile, int& img, int& mt, int& blk) {
        blk = tile % nblk;
        const int t2 = tile / nblk;
        mt = t2 % mtiles_img;
        img = t2 / mtiles_img;
    };

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                int img, mt, blk;
                decode(tile, img, mt, blk);
                const int grow = img * p.H + p.row0 + mt * RM;     // first global row of the tile
                const int kb0 = __ldg(p.kb0 + blk);
                for (int kb = 0; kb < p.kblocks; ++kb) {
                    tc::mbar_wait(&empty_bar[stage], phase ^ 1);
                    uint8_t* sa = smem + stage * kStageR;
                    tc::mbar_expect_tx(&full_bar[stage], kStageR);
                    tc::tma_load_2d(&tmap_img, &full_bar[stage], sa, kb0 + kb * RKB, grow);
                    tc::tma_load_2d(&tmap_coef, &full_bar[stage], sa + kABytesR, kb * RKB, blk * RN);
                    if (++stage == RSTAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = make_idesc_u8s8(RM, RN);
            int stage = 0, iter = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++iter) {
                const int acc = iter & 1;
                tc::mbar_wait(&tmem_empty[acc], ((iter >> 1) & 1) ^ 1);
                tc::tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * 128;
                for (int kb = 0; kb < p.kblocks; ++kb) {
                    tc::mbar_wait(&full_bar[stage], phase);
                    tc::tc_fence_after();
                    const uint32_t sa = tc::smem_u32(smem + stage * kStageR);
                    const uint64_t da = tc::make_desc_k_sw128(sa);
                    const uint64_t db = tc::make_desc_k_sw128(sa + kABytesR);
#pragma unroll
                    for (int k = 0; k < RKB / 32; ++k) umma_i8(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
                    tc::umma_commit(&empty_bar[stage]);
                    if (++stage == RSTAGES) { stage = 0; phase ^= 1; }
                }
                tc::umma_commit(&tmem_full[acc]);
            }
        }
    } else {
        const int quarter = warp & 3;
        int iter = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++iter) {
            int img, mt, blk;
            decode(tile, img, mt, blk);
            const int acc = iter & 1;
            tc::mbar_wait(&tmem_full[acc], (iter >> 1) & 1);
            tc::tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * 128;
            const int r_in = mt * RM + quarter * 32 + lane;
            if (CH == 3) {
                uint32_t d0[32], d1[32], d2[32];
                tc::tmem_ld_32x32(taddr, d0);
                tc::tmem_ld_32x32(taddr + 32, d1);
                tc::tmem_ld_32x32(taddr + 64, d2);
                tc::tmem_ld_wait();
                tc::tc_fence_before();
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(&tmem_empty[acc]);
                // columns: limb L occupies [24 L, 24 L + 24); 96 values = d0 | d1 | d2
                auto col = [&](int c) -> uint32_t { return c < 32 ? d0[c] : (c < 64 ? d1[c - 32] : d2[c - 64]); };
                if (r_in < p.rows) {
                    uint32_t packed[6];
#pragma unroll
                    for (int w = 0; w < 6; ++w) packed[w] = 0u;
#pragma unroll
                    for (int i = 0; i < 24; ++i) {
                        uint32_t v = col(i) + (col(24 + i) << 7) + (col(48 + i) << 14) + (1u << (kPrec - 1));
                        if (p.limbs == 4) v += col(72 + i) << 21;
                        int s = (int)v >> kPrec;
                        s = s < 0 ? 0 : (s > 255 ? 255 : s);
                        packed[i >> 2] |= (uint32_t)s << (8 * (i & 3));
                    }
                    uint8_t* dst = p.tmp + (((size_t)img * p.rows + r_in) * p.out + (size_t)blk * kNB) * 3;
                    uint2* d8 = reinterpret_cast<uint2*>(dst);
                    d8[0] = make_uint2(packed[0], packed[1]);
                    d8[1] = make_uint2(packed[2], packed[3]);
                    d8[2] = make_uint2(packed[4], packed[5]);
                }
            } else {
                uint32_t d0[32];
                tc::tmem_ld_32x32(taddr, d0);
                tc::tmem_ld_wait();
                tc::tc_fence_before();
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(&tmem_empty[acc]);
                if (r_in < p.rows) {
                    uint32_t packed[2] = {0u, 0u};
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        uint32_t v = d0[i] + (d0[8 + i] << 7) + (d0[16 + i] << 14) + (1u << (kPrec - 1));
                        if (p.limbs == 4) v += d0[24 + i] << 21;
                        int s = (int)v >> kPrec;
                        s = s < 0 ? 0 : (s > 255 ? 255 : s);
                        packed[i >> 2] |= (uint32_t)s << (8 * (i & 3));
                    }
                    *reinterpret_cast<uint2*>(p.tmp + ((size_t)img * p.rows + r_in) * p.out + (size_t)blk * kNB) = make_uint2(packed[0], packed[1]);
                }
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    if (warp == 1) tc::tmem_dealloc(tmem_base, 256);
}

constexpr int kResMaxStages = 8;

struct ResidentArgs {
    ResampleTcArgs a;
    int stages;                           // A stages in the ring (4..8)
    int ngroups;                          // gridDim.x / nblk: CTAs per column block
};

// Resident-coefficient schedule (see the file header).  Shared memory: [kblocks][RN][128] int8 coefficients | A ring | barriers.
template <int CH>
__global__ void __launch_bounds__(kThreadsR, 1)
resample_h_tc_resident_kernel(const __grid_constant__ CUtensorMap tmap_img, const __grid_constant__ CUtensorMap tmap_coef, ResidentArgs q) {
    constexpr int RN = RCfg<CH>::RN;
    constexpr int kBSlab = RN * RKB;
    const ResampleTcArgs& p = q.a;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - ((uint32_t)__cvta_generic_to_shared(smem_raw) & 1023u)) & 1023u);
    uint8_t* smem_b = smem;
    uint8_t* smem_a = smem + p.kblocks * kBSlab;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_a + q.stages * kABytesR);
    uint64_t* full_bar = bars;
    uint64_t* empty_bar = bars + kResMaxStages;
    uint64_t* tmem_full = bars + 2 * kResMaxStages;
    uint64_t* tmem_empty = bars + 2 * kResMaxStages + 2;
    uint64_t* b_full = bars + 2 * kResMaxStages + 4;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kResMaxStages + 5);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nblk = p.out / kNB;
    const int mtiles_img = (p.rows + RM - 1) / RM;
    const int total_m = p.n_img * mtiles_img;
    const int blk = blockIdx.x % nblk, group = blockIdx.x / nblk;

    if (threadIdx.x == 0) {
        for (int s = 0; s < q.stages; ++s) {
            tc::mbar_init(&full_bar[s], 1);
            tc::mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            tc::mbar_init(&tmem_full[a], 1);
            tc::mbar_init(&tmem_empty[a], 4);
        }
        tc::mbar_init(b_full, 1);
        tc::mbar_fence_init();
        tc::fence_proxy_async();
        tc::tma_prefetch_desc(&tmap_img);
        tc::tma_prefetch_desc(&tmap_coef);
    }
    if (warp == 1) tc::tmem_alloc(tmem_slot, 256);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            // the block's coefficient matrix, once
            tc::mbar_expect_tx(b_full, (uint32_t)(p.kblocks * kBSlab));
            for (int kb = 0; kb < p.kblocks; ++kb) tc::tma_load_2d(&tmap_coef, b_full, smem_b + kb * kBSlab, kb * RKB, blk * RN);
            const int kb0 = __ldg(p.kb0 + blk);
            int stage = 0;
            uint32_t phase = 0;
            for (int mtg = group; mtg < total_m; mtg += q.ngroups) {
                const int img = mtg / mtiles_img, mt = mtg - img * mtiles_img;
                const int grow = img * p.H + p.row0 + mt * RM;
                for (int kb = 0; kb < p.kblocks; ++kb) {
                    tc::mbar_wait(&empty_bar[stage], phase ^ 1);
                    tc::mbar_expect_tx(&full_bar[stage], kABytesR);
                    tc::tma_load_2d(&tmap_img, &full_bar[stage], smem_a + stage * kABytesR, kb0 + kb * RKB, grow);
                    if (++stage == q.stages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = make_idesc_u8s8(RM, RN);
            int stage = 0, iter = 0;
            uint32_t phase = 0;
            tc::mbar_wait(b_full, 0);
            for (int mtg = group; mtg < total_m; mtg += q.ngroups, ++iter) {
                const int acc = iter & 1;
                tc::mbar_wait(&tmem_empty[acc], ((iter >> 1) & 1) ^ 1);
                tc::tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * 128;
                for (int kb = 0; kb < p.kblocks; ++kb) {
                    tc::mbar_wait(&full_bar[stage], phase);
                    tc::tc_fence_after();
                    const uint64_t da = tc::make_desc_k_sw128(tc::smem_u32(smem_a + stage * kABytesR));
                    const uint64_t db = tc::make_desc_k_sw128(tc::smem_u32(smem_b + kb * kBSlab));
#pragma unroll
                    for (int k = 0; k < RKB / 32; ++k) umma_i8(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
                    tc::umma_commit(&empty_bar[stage]);
                    if (++stage == q.stages) { stage = 0; phase ^= 1; }
                }
                tc::umma_commit(&tmem_full[acc]);
            }
        }
    } else {
        const int quarter = warp & 3;
        int iter = 0;
        for (int mtg = group; mtg < total_m; mtg += q.ngroups, ++iter) {
            const int img = mtg / mtiles_img, mt = mtg - img * mtiles_img;
            const int acc = iter & 1;
            tc::mbar_wait(&tmem_full[acc], (iter >> 1) & 1);
            tc::tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * 128;
            const int r_in = mt * RM + quarter * 32 + lane;
            if (CH == 3) {
                uint32_t d0[32], d1[32], d2[32];
                tc::tmem_ld_32x32(taddr, d0);
                tc::tmem_ld_32x32(taddr + 32, d1);
                tc::tmem_ld_32x32(taddr + 64, d2);
                tc::tmem_ld_wait();
                tc::tc_fence_before();
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(&tmem_empty[acc]);
                auto col = [&](int c) -> uint32_t { return c < 32 ? d0[c] : (c < 64 ? d1[c - 32] : d2[c - 64]); };
                if (r_in < p.rows) {
                    uint32_t packed[6];
#pragma unroll
                    for (int w = 0; w < 6; ++w) packed[w] = 0u;
#pragma unroll
                    for (int i = 0; i < 24; ++i) {
                        uint32_t v = col(i) + (col(24 + i) << 7) + (col(48 + i) << 14) + (1u << (kPrec - 1));
                        if (p.limbs == 4) v += col(72 + i) << 21;
                        int sv = (int)v >> kPrec;
                        sv = sv < 0 ? 0 : (sv > 255 ? 255 : sv);
                        packed[i >> 2] |= (uint32_t)sv << (8 * (i & 3));
                    }
                    uint8_t* dst = p.tmp + (((size_t)img * p.rows + r_in) * p.out + (size_t)blk * kNB) * 3;
                    uint2* d8 = reinterpret_cast<uint2*>(dst);
                    d8[0] = make_uint2(packed[0], packed[1]);
                    d8[1] = make_uint2(packed[2], packed[3]);
                    d8[2] = make_uint2(packed[4], packed[5]);
                }
            } else {
                uint32_t d0[32];
                tc::tmem_ld_32x32(taddr, d0);
                tc::tmem_ld_wait();
                tc::tc_fence_before();
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(&tmem_empty[acc]);
                if (r_in < p.rows) {
                    uint32_t packed[2] = {0u, 0u};
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        uint32_t v = d0[i] + (d0[8 + i] << 7) + (d0[16 + i] << 14) + (1u << (kPrec - 1));
                        if (p.limbs == 4) v += d0[24 + i] << 21;
                        int sv = (int)v >> kPrec;
                        sv = sv < 0 ? 0 : (sv > 255 ? 255 : sv);
                        packed[i >> 2] |= (uint32_t)sv << (8 * (i & 3));
                    }
                    *reinterpret_cast<uint2*>(p.tmp + ((size_t)img * p.rows + r_in) * p.out + (size_t)blk * kNB) = make_uint2(packed[0], packed[1]);
                }
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    if (warp == 1) tc::tmem_dealloc(tmem_base, 256);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int make_tmap_u8_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t row_stride, uint32_t box_rows) {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(ptr);
    }
    FB_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {row_stride};
    cuuint32_t box[2] = {128, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    FB_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(u8) failed with CUresult %d", (int)r);
    return 0;
}

}  // namespace

// Returns 1 when the tensor-core path does not apply (caller falls back to the CUDA-core kernel), 0 on success.
// channels = 3: d_images is [n][H][W][3] interleaved; channels = 1: a [n][H][W] uint8 plane.
int launch_resample_h_tc(const uint8_t* d_images, int n, int H, int W, long long image_stride, int out_size, const int8_t* d_coef,
                         int kw, int limbs, const int* d_kb0, int row0, int rows, uint8_t* d_tmp, int channels,
                         cudaStream_t stream) {
    if (!d_coef || !d_kb0 || kw <= 0) return 1;
    if ((W % 16) != 0 || (reinterpret_cast<uintptr_t>(d_images) & 15) != 0 || image_stride != (long long)H * W * channels) return 1;
    if (out_size % kNB != 0 || (kw % RKB) != 0 || (limbs != 3 && limbs != 4) || (channels != 1 && channels != 3)) return 1;
    if ((reinterpret_cast<uintptr_t>(d_tmp) & 7) != 0) return 1;
    const int RN = channels == 3 ? RCfg<3>::RN : RCfg<1>::RN;
    CUtensorMap ta, tb;
    int rc = make_tmap_u8_2d(&ta, d_images, (uint64_t)n * H, (uint64_t)W * channels, (uint64_t)W * channels, RM);
    if (rc) return rc;
    rc = make_tmap_u8_2d(&tb, d_coef, (uint64_t)(out_size / kNB) * RN, (uint64_t)kw, (uint64_t)kw, RN);
    if (rc) return rc;
    ResampleTcArgs p;
    p.n_img = n; p.H = H; p.row0 = row0; p.rows = rows; p.out = out_size; p.kblocks = kw / RKB; p.limbs = limbs;
    p.kb0 = d_kb0; p.tmp = d_tmp;
    static PerDeviceFlag attr_set;
    if (!attr_set.get()) {
        FB_CUDA_OK(cudaFuncSetAttribute(resample_h_tc_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, RCfg<3>::kSmem));
        FB_CUDA_OK(cudaFuncSetAttribute(resample_h_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, RCfg<1>::kSmem));
        attr_set.set();
    }
    // resident-coefficient schedule when the block's coefficient matrix fits beside a ring of >= 4 image stages
    {
        const int nblk = out_size / kNB;
        const int total_m = n * ((rows + RM - 1) / RM);
        const long long b_bytes = (long long)p.kblocks * RN * RKB;
        const long long room = 227ll * 1024 - 1024 /*alignment*/ - 256 /*barriers*/ - b_bytes;
        int stages = (int)(room / kABytesR);
        if (stages > kResMaxStages) stages = kResMaxStages;
        int ngroups = sm_count() / nblk;
        if (ngroups > total_m) ngroups = total_m;
        if (stages >= 4 && ngroups >= 1) {
            ResidentArgs q;
            q.a = p;
            q.stages = stages;
            q.ngroups = ngroups;
            const int smem = (int)(b_bytes + (long long)stages * kABytesR + 1024 + 256);
            // the attribute only ever grows: set it to the largest size a launch may ask for
            static PerDeviceFlag res_attr_set;
            if (!res_attr_set.get()) {
                FB_CUDA_OK(cudaFuncSetAttribute(resample_h_tc_resident_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
                FB_CUDA_OK(cudaFuncSetAttribute(resample_h_tc_resident_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
                res_attr_set.set();
            }
            if (channels == 3) resample_h_tc_resident_kernel<3><<<nblk * ngroups, kThreadsR, smem, stream>>>(ta, tb, q);
            else resample_h_tc_resident_kernel<1><<<nblk * ngroups, kThreadsR, smem, stream>>>(ta, tb, q);
            FB_CUDA_OK(cudaGetLastError());
            return 0;
        }
    }
    const int tiles = n * ((rows + RM - 1) / RM) * (out_size / kNB);
    const int grid = tiles < sm_count() ? tiles : sm_count();
    if (channels == 3) resample_h_tc_kernel<3><<<grid, kThreadsR, RCfg<3>::kSmem, stream>>>(ta, tb, p);
    else resample_h_tc_kernel<1><<<grid, kThreadsR, RCfg<1>::kSmem, stream>>>(ta, tb, p);
    FB_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace fb
