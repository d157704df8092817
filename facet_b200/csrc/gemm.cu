// bf16 GEMM on the 5th-generation tensor cores: C[M,N] = A[M,K] * B[N,K]^T (+ fused epilogue).
//
// This is the GEMM under the CLIP ViT-L/14 image tower that the reference runs through
// open_clip / cuBLAS (`self.model.encode_image`, processing/scorer.py:662): QKV, attention
// out-projection, MLP fc / proj and the patch-embedding convolution (as an im2col GEMM), and the
// cosine all-pairs GEMM of the similarity stage.  Both operands are K-major (PyTorch Linear
// weights [out,in] are already "B[N,K]").
//
// Structure (one persistent CTA per SM, 320 threads):
//   warp 0      TMA producer, mbarrier ring, 128-byte swizzle
//   warp 1      tcgen05.mma issuer (one elected lane), fp32 accumulators in TMEM, two 256-column
//               accumulator buffers so tile i+1 overlaps the epilogue of i
//   warps 2..9  epilogue: tcgen05.ld (32 lanes x 32 columns), bias / GELU / residual / threshold,
//               per-warp shared-memory transpose, 16-byte global stores of full row segments
// Two forms of the same kernel (template parameter CL2):
//   single CTA  128x256 tile, 128x64 A box + 256x64 B box per stage, 4 stages (patch embedding, similarity)
//   CTA pair    clusters of two CTAs, tcgen05.mma.cta_group::2 on a 256x256 tile: each CTA loads its 128 rows
//               of A and half of B (32 KB per stage), 6 stages; the leader CTA issues the MMAs for both (the
//               ViT-layer GEMMs: QKV, out-projection, fc, proj)
#include <map>
#include <mutex>
#include <tuple>

#include "common.cuh"
#include "kernels.h"
#include "tc_common.cuh"

namespace fb {

namespace {

constexpr int BM = 128, BN = 256, BK = 64, STAGES = 4;
constexpr int kABytes = BM * BK * 2;     // 16 KB
constexpr int kBBytes = BN * BK * 2;     // 32 KB
constexpr int kStageBytes = kABytes + kBBytes;
constexpr int kEpiPitch = 80;                               // bytes per staged row (64 B of bf16 + 16 B pad: conflict-free)
// Epilogue warps per CTA: 8, each on 128 of the tile's 256 columns.  Round-2 experiment (profiles/r2_gemm_gelu_epilogue.txt):
// the erf-GELU epilogue of the CTA-pair form with 16 warps (four per scheduler, 64 columns each, five TMA stages, the
// accumulator handed back before any of the math) is within 2 % of the 8-warp form, and knock-out builds show its cost is
// proportional to the FMA-pipe instruction count of the erf polynomial (not MUFU, not latency): -DFB_GELU_EPI_WARPS=16
// builds that variant.
#ifndef FB_GELU_EPI_WARPS
#define FB_GELU_EPI_WARPS 8
#endif
#ifndef FB_GELU_EARLY_RELEASE
#define FB_GELU_EARLY_RELEASE 1
#endif
#ifndef FB_GELU_STAGES
#define FB_GELU_STAGES 5
#endif
__host__ __device__ constexpr bool bf16_out_mode(int mode) { return mode == FB_GEMM_BIAS_BF16 || mode == FB_GEMM_BIAS_GELU_BF16; }
__host__ __device__ constexpr int epi_warps(int mode, bool cl2) { return (mode == FB_GEMM_BIAS_GELU_BF16 && cl2) ? FB_GELU_EPI_WARPS : 8; }
__host__ __device__ constexpr int gemm_threads(int mode, bool cl2) { return 64 + 32 * epi_warps(mode, cl2); }
__host__ __device__ constexpr int gemm_stages(int mode, bool cl2) { return cl2 ? (epi_warps(mode, cl2) == 16 ? FB_GELU_STAGES : 6) : STAGES; }
__host__ __device__ constexpr int gemm_stage_bytes(bool cl2) { return kABytes + (cl2 ? kBBytes / 2 : kBBytes); }
__host__ __device__ constexpr int gemm_smem_bytes(int mode, bool cl2) {
    return gemm_stages(mode, cl2) * gemm_stage_bytes(cl2) + epi_warps(mode, cl2) * (32 * kEpiPitch + 1024) + 1024 /*alignment slack*/ +
           256 /*barriers*/;
}

struct GemmArgs {
    int M, N, K;
    int mode;             // FB_GEMM_*
    const float* bias;    // [N] or nullptr
    void* out;            // bf16 or f32, row-major
    long long ldo;        // elements
    const float* residual;
    long long ldr;
    // FB_GEMM_THRESHOLD_PAIRS: candidates (row_offset + row, col_offset + col) with acc >= tau and, when tri_on, global
    // column > global row (a diagonal block of the all-pairs scan); rectangular blocks (tri_on = 0) report every hit
    float tau;
    int row_offset;
    int col_offset;
    int tri_on;
    int* pairs;
    float* pair_sims;
    long long pair_cap;
    unsigned long long* pair_count;
    int f16;              // operands (and 16-bit outputs) are fp16 instead of bf16
    // LayerNorm fold (csrc/vit_forward.cu).  Producer side, FB_GEMM_BIAS_RESIDUAL_F32: besides the fp32 residual stream the
    // epilogue writes a 16-bit copy of it (the A operand of the next GEMM) and, per row and per 128-column slice, the sum and the
    // sum of squares of the new values.  Consumer side, FB_GEMM_BIAS_BF16 / _GELU_BF16: the A operand is that raw copy and the
    // weights carry the LayerNorm gain, so LayerNorm(x) W^T + b = rstd_r (acc - mean_r s_n) + c_n with s_n = sum_k gamma_k W_nk
    // and c_n = sum_k beta_k W_nk + b_n (passed as `bias`); mean / rstd come from the producer's row sums.
    void* out16;          // [M][ldo16] 16-bit copy of the output, or nullptr
    long long ldo16;
    float* row_stats;     // producer: [M][ln_slots][2] (sum, sum of squares); consumer: the same array, read
    int ln_slots;         // slices per row (N / 128 of the producer)
    const float* ln_s;    // consumer: [N] column sums of the folded weights, or nullptr (no fold)
    int ln_width;         // consumer: number of elements a row of the normalised operand has (1024)
};

// Exact (erf) GELU, nn.GELU() of the reference tower.  erf via Abramowitz & Stegun 7.1.26 (|error| <= 1.5e-7,
// i.e. fp32 noise; checked against scipy over [-8, 8]): 2 MUFU + 9 FMA instead of erff's ~45 instructions.
//   0.5 x (1 + erf(x / sqrt 2)) = 0.5 x + 0.5 |x| erf(|x| / sqrt 2)
__device__ __forceinline__ float gelu_erf(float x) {
#if defined(FB_GELU_KO) && FB_GELU_KO == 1      /* knock-out: the polynomial without the two MUFU operations */
    {
        const float z = fabsf(x) * 0.70710678118654752440f;
        float t = fmaf(0.3275911f, z, 1.0f);
        float p = fmaf(1.061405429f, t, -1.453152027f);
        p = fmaf(p, t, 1.421413741f);
        p = fmaf(p, t, -0.284496736f);
        p = fmaf(p, t, 0.254829592f);
        p *= t;
        float e = -z * z * 1.4426950408889634f;
        const float hx = 0.5f * x;
        return fmaf(fabsf(hx), fmaf(-p, e, 1.0f), hx);
    }
#elif defined(FB_GELU_KO) && FB_GELU_KO == 2    /* knock-out: the two MUFU operations without the polynomial */
    {
        float t, e;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(x));
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x));
        return t + e;
    }
#elif defined(FB_GELU_KO) && FB_GELU_KO == 3    /* knock-out: half the polynomial, one MUFU */
    {
        const float z = fabsf(x) * 0.70710678118654752440f;
        float t;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.0f)));
        float p = fmaf(1.061405429f, t, -1.453152027f);
        p = fmaf(p, t, 1.421413741f);
        const float hx = 0.5f * x;
        return fmaf(fabsf(hx), p, hx);
    }
#endif
    const float z = fabsf(x) * 0.70710678118654752440f;
    float t;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.0f)));
    float p = fmaf(1.061405429f, t, -1.453152027f);
    p = fmaf(p, t, 1.421413741f);
    p = fmaf(p, t, -0.284496736f);
    p = fmaf(p, t, 0.254829592f);
    p *= t;
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-z * z * 1.4426950408889634f));
    const float hx = 0.5f * x;
    return fmaf(fabsf(hx), fmaf(-p, e, 1.0f), hx);
}

// CL2: launched as clusters of two CTAs (a CTA pair) that compute one 256x256 tile with tcgen05.mma.cta_group::2:
// each CTA loads its own 128 rows of A and HALF of the B tile (32 KB per k-block instead of 48 KB), so six
// stages fit where four did and the TMA pipeline covers the L2 latency.  The leader CTA issues the MMAs for
// both; its full barriers collect the bytes of both CTAs' loads, its commits free the stages and publish the
// accumulators in both CTAs, and both CTAs' epilogue warps hand the accumulator back to the leader.
template <int MODE, bool F16, bool CL2>
__global__ void __launch_bounds__(gemm_threads(MODE, CL2), 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, GemmArgs p) {
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment by pointer arithmetic on the shared pointer (a round trip through an integer would
    // make every later access a generic LD/ST instead of LDS/STS)
    uint8_t* smem = smem_raw + ((1024u - ((uint32_t)__cvta_generic_to_shared(smem_raw) & 1023u)) & 1023u);
    constexpr int kEpiWarps = epi_warps(MODE, CL2);
    constexpr int kEpiStageBytes = kEpiWarps * 32 * kEpiPitch;             // per-warp 32x32 bf16 transpose buffers
    constexpr int kEpiBiasBytes = kEpiWarps * 1024;                        // per-warp copy of the bias (and LayerNorm-fold column sum) values of its columns
    constexpr int kColsPerWarp = BN / (kEpiWarps / 4);                     // 128, or 64 with 16 epilogue warps
    constexpr int kChunks = kColsPerWarp / 32;
    constexpr int NS = gemm_stages(MODE, CL2);                             // pipeline stages
    constexpr int SB = gemm_stage_bytes(CL2);                              // stage bytes
    static_assert(gemm_smem_bytes(MODE, CL2) <= 227 * 1024, "shared memory budget");
    uint8_t* epi_stage = smem + NS * SB;
    uint8_t* epi_bias = epi_stage + kEpiStageBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + NS * SB + kEpiStageBytes + kEpiBiasBytes);
    uint64_t* full_bar = bars;                   // [NS]
    uint64_t* empty_bar = bars + NS;             // [NS]
    uint64_t* tmem_full = bars + 2 * NS;         // [2]
    uint64_t* tmem_empty = bars + 2 * NS + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * NS + 4);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int tiles_n = (p.N + BN - 1) / BN;
    const int tiles_m = (p.M + BM - 1) / BM;
    const int crank = CL2 ? (int)tc::cluster_ctarank() : 0;
    // CL2 walks pairs of tile rows: pair t -> tile rows 2 (t / tiles_n) + rank, tile column t % tiles_n
    const int num_tiles = CL2 ? ((tiles_m + 1) / 2) * tiles_n : tiles_m * tiles_n;
    const int tile_first = CL2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int tile_step = CL2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    const int kblocks = p.K / BK;
    // similarity mode only needs tiles that contain an element with col > global row
    constexpr bool tri = (MODE == FB_GEMM_THRESHOLD_PAIRS);
#define FB_TILE_SKIPPED(m0_, n0_) (tri && p.tri_on && ((n0_) + p.col_offset + BN <= (m0_) + p.row_offset + 1))
    // Tile order.  Plain GEMMs walk row-major (their B operand is a weight matrix that stays in L2).  The
    // similarity scan has a B operand far larger than L2, so its tiles are walked in groups of kGroupM tile
    // rows, column by column: the CTAs running at any moment share kGroupM A tiles and every B tile is used
    // kGroupM times while it is hot in L2 (HBM traffic per tile / kGroupM).
    constexpr int kGroupM = 16;
#define FB_TILE_COORDS(tile_, m0_, n0_)                                             \
    int m0_, n0_;                                                                   \
    if (tri) {                                                                      \
        const int per_group_ = kGroupM * tiles_n;                                   \
        const int g_ = (tile_) / per_group_;                                        \
        const int w_ = (tile_) - g_ * per_group_;                                   \
        const int gm_ = min(kGroupM, tiles_m - g_ * kGroupM);                       \
        m0_ = (g_ * kGroupM + w_ % gm_) * BM;                                       \
        n0_ = (w_ / gm_) * BN;                                                      \
    } else if (CL2) {                                                               \
        m0_ = (2 * ((tile_) / tiles_n) + crank) * BM;                               \
        n0_ = ((tile_) % tiles_n) * BN;                                             \
    } else {                                                                        \
        m0_ = ((tile_) / tiles_n) * BM;                                             \
        n0_ = ((tile_) % tiles_n) * BN;                                             \
    }

    if (threadIdx.x == 0) {
        for (int s = 0; s < NS; ++s) {
            tc::mbar_init(&full_bar[s], CL2 ? 2 : 1);         // pair: one arrive.expect_tx per CTA
            tc::mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            tc::mbar_init(&tmem_full[a], 1);
            tc::mbar_init(&tmem_empty[a], CL2 ? 2 * kEpiWarps : kEpiWarps);
        }
        tc::mbar_fence_init();
        tc::fence_proxy_async();
    }
    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&tmap_a);
        tc::tma_prefetch_desc(&tmap_b);
    }
    if (warp == 1) {
        if (CL2) tc::tmem_alloc_pair(tmem_slot, 512);
        else tc::tmem_alloc(tmem_slot, 512);
    }
    tc::tc_fence_before();
    __syncthreads();
    if (CL2) tc::cluster_sync_all();     // the peer's barriers are initialised before anything is multicast to them
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = tile_first; tile < num_tiles; tile += tile_step) {
                FB_TILE_COORDS(tile, m0, n0)
                if (FB_TILE_SKIPPED(m0, n0)) continue;
                for (int kb = 0; kb < kblocks; ++kb) {
                    tc::mbar_wait(&empty_bar[stage], phase ^ 1);
                    uint8_t* sa = smem + stage * SB;
                    if (CL2) {
                        // both CTAs report their bytes to the leader's full barrier; tmap_b has a 128-row box here and
                        // this CTA holds rows [n0 + 128 rank, +128) of the B tile
                        const uint32_t lead_bar = tc::mapa_u32(tc::smem_u32(&full_bar[stage]), 0u);
                        tc::mbar_expect_tx_cluster(lead_bar, SB);
                        tc::tma_load_2d_pair(&tmap_a, lead_bar, sa, kb * BK, m0);
                        tc::tma_load_2d_pair(&tmap_b, lead_bar, sa + kABytes, kb * BK, n0 + crank * (BN / 2));
                    } else {
                        tc::mbar_expect_tx(&full_bar[stage], SB);
                        tc::tma_load_2d(&tmap_a, &full_bar[stage], sa, kb * BK, m0);
                        tc::tma_load_2d(&tmap_b, &full_bar[stage], sa + kABytes, kb * BK, n0);
                    }
                    if (++stage == NS) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0 && crank == 0) {            // pair: the leader issues for both CTAs
            const uint32_t idesc = tc::make_idesc16<F16>(CL2 ? 2 * BM : BM, BN);
            int stage = 0;
            uint32_t phase = 0;
            int iter = 0;
            for (int tile = tile_first; tile < num_tiles; tile += tile_step) {
                FB_TILE_COORDS(tile, m0, n0)
                if (FB_TILE_SKIPPED(m0, n0)) continue;
                const int acc = iter & 1;
                tc::mbar_wait(&tmem_empty[acc], ((iter >> 1) & 1) ^ 1);
                tc::tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                for (int kb = 0; kb < kblocks; ++kb) {
                    tc::mbar_wait(&full_bar[stage], phase);
                    tc::tc_fence_after();
                    const uint32_t sa = tc::smem_u32(smem + stage * SB);
                    const uint64_t da = tc::make_desc_k_sw128(sa);
                    const uint64_t db = tc::make_desc_k_sw128(sa + kABytes);
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k) {
                        // advancing K by 16 bf16 = 32 bytes inside the 128-byte swizzle row: +2 in the address field
                        if (CL2) tc::umma_bf16_pair(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
                        else tc::umma_bf16(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
                    }
                    // frees the smem stage when the MMAs retire (pair: in both CTAs)
                    if (CL2) tc::umma_commit_pair(&empty_bar[stage], (uint16_t)3);
                    else tc::umma_commit(&empty_bar[stage]);
                    if (++stage == NS) { stage = 0; phase ^= 1; }
                }
                // accumulator complete (pair: published to both CTAs' epilogues)
                if (CL2) tc::umma_commit_pair(&tmem_full[acc], (uint16_t)3);
                else tc::umma_commit(&tmem_full[acc]);
                ++iter;
            }
        }
    } else {
        // ===== epilogue =====
        const int ew = warp - 2;
        const int quarter = warp & 3;          // TMEM lanes [32*quarter, +32) are the ones this warp may read
        const int half = ew >> 2;              // which kColsPerWarp of the 256 accumulator columns
        uint8_t* stg = epi_stage + ew * (32 * kEpiPitch);
        float* bias_s = reinterpret_cast<float*>(epi_bias + ew * 1024);
        float* lns_s = bias_s + 128;
        const bool ln_fold = bf16_out_mode(MODE) && p.ln_s != nullptr;
        constexpr bool bf16_out = (MODE == FB_GEMM_BIAS_BF16 || MODE == FB_GEMM_BIAS_GELU_BF16);
        int iter = 0;
        for (int tile = tile_first; tile < num_tiles; tile += tile_step) {
            FB_TILE_COORDS(tile, m0, n0)
            if (FB_TILE_SKIPPED(m0, n0)) continue;
            const int acc = iter & 1;
            const int rbase = m0 + quarter * 32;
            const int row = rbase + lane;
            const bool row_ok = row < p.M;
            const int ncol0 = n0 + half * kColsPerWarp;
            // bias of this warp's 128 columns -> smem, while the MMAs of the tile are still running
            __syncwarp();
            {
                float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (p.bias && lane * 4 < kColsPerWarp && ncol0 + lane * 4 < p.N) b4 = __ldg(reinterpret_cast<const float4*>(p.bias + ncol0 + lane * 4));
                if (lane * 4 < kColsPerWarp) *reinterpret_cast<float4*>(bias_s + lane * 4) = b4;
                if (ln_fold && lane * 4 < kColsPerWarp) {
                    float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (ncol0 + lane * 4 < p.N) s4 = __ldg(reinterpret_cast<const float4*>(p.ln_s + ncol0 + lane * 4));
                    *reinterpret_cast<float4*>(lns_s + lane * 4) = s4;
                }
            }
            // LayerNorm fold: mean and 1 / std of this thread's row from the producer's per-slice sums (fixed order)
            float ln_mean = 0.f, ln_rstd = 1.f;
            if (ln_fold && row_ok) {
                const float* st2 = p.row_stats + (size_t)row * p.ln_slots * 2;
                float sx = 0.f, sq = 0.f;
                for (int i = 0; i < p.ln_slots; ++i) {
                    const float2 v2 = *reinterpret_cast<const float2*>(st2 + 2 * i);
                    sx += v2.x;
                    sq += v2.y;
                }
                const float inv_w = 1.0f / (float)p.ln_width;
                ln_mean = sx * inv_w;
                ln_rstd = rsqrtf(fmaxf(sq * inv_w - ln_mean * ln_mean, 0.f) + 1e-5f);
            }
            // producer side: running (sum, sum of squares) of the rows this lane sees after the transpose: rows (lane >> 2) + 8 j
            float st_s[4] = {0.f, 0.f, 0.f, 0.f}, st_q[4] = {0.f, 0.f, 0.f, 0.f};
            __syncwarp();
            tc::mbar_wait(&tmem_full[acc], (iter >> 1) & 1);
            tc::tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BN + half * kColsPerWarp;

            // coalesced residual prefetch for chunk c: lane -> row (lane>>2)+8j, 16-byte piece (lane&3) of each 64-byte half
            auto prefetch_res = [&](float4 (&rr)[8], int c) {
                if (MODE != FB_GEMM_BIAS_RESIDUAL_F32) return;
                const int col0 = ncol0 + c * 32;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const int rl = (lane >> 2) + 8 * (q & 3);
                    rr[q] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (rbase + rl < p.M && col0 < p.N)
                        rr[q] = *reinterpret_cast<const float4*>(p.residual + (size_t)(rbase + rl) * p.ldr + col0 + 16 * (q >> 2) + 4 * (lane & 3));
                }
            };
            auto process = [&](const uint32_t (&v)[32], int c, const float4 (&rr)[8]) {
                const int col0 = ncol0 + c * 32;
                if (MODE == FB_GEMM_THRESHOLD_PAIRS) {
                    const int grow = p.row_offset + row;
                    const int gcol0 = p.col_offset + col0;
                    // candidates are rare: one max over the lane's 32 values decides whether to look at them at all
                    float vmax = __uint_as_float(v[0]);
#pragma unroll
                    for (int j = 1; j < 32; ++j) vmax = fmaxf(vmax, __uint_as_float(v[j]));
                    if (row_ok && (!p.tri_on || gcol0 + 31 > grow) && vmax >= p.tau) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const float sim = __uint_as_float(v[j]);
                            const int col = col0 + j;
                            if (sim >= p.tau && (!p.tri_on || gcol0 + j > grow) && col < p.N) {
                                const unsigned long long pos = atomicAdd(p.pair_count, 1ull);
                                if ((long long)pos < p.pair_cap) {
                                    p.pairs[2 * pos] = grow;
                                    p.pairs[2 * pos + 1] = gcol0 + j;
                                    p.pair_sims[pos] = sim;
                                }
                            }
                        }
                    }
                    return;
                }
                if (col0 >= p.N) return;          // warp-uniform
                float f[32];
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 b4 = *reinterpret_cast<const float4*>(bias_s + c * 32 + j);
                    if (ln_fold) {
                        const float4 s4 = *reinterpret_cast<const float4*>(lns_s + c * 32 + j);
                        f[j] = fmaf(ln_rstd, fmaf(-ln_mean, s4.x, __uint_as_float(v[j])), b4.x);
                        f[j + 1] = fmaf(ln_rstd, fmaf(-ln_mean, s4.y, __uint_as_float(v[j + 1])), b4.y);
                        f[j + 2] = fmaf(ln_rstd, fmaf(-ln_mean, s4.z, __uint_as_float(v[j + 2])), b4.z);
                        f[j + 3] = fmaf(ln_rstd, fmaf(-ln_mean, s4.w, __uint_as_float(v[j + 3])), b4.w);
                    } else {
                        f[j] = __uint_as_float(v[j]) + b4.x;
                        f[j + 1] = __uint_as_float(v[j + 1]) + b4.y;
                        f[j + 2] = __uint_as_float(v[j + 2]) + b4.z;
                        f[j + 3] = __uint_as_float(v[j + 3]) + b4.w;
                    }
                }
                if (MODE == FB_GEMM_BIAS_GELU_BF16) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = gelu_erf(f[j]);
                }
                // thread = row holds 32 consecutive outputs.  Transpose through the per-warp smem buffer so that
                // 4 lanes write 64 contiguous bytes of one row (full sectors) instead of 32 rows x 16 bytes.
                if (bf16_out) {
                    __syncwarp();
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        *reinterpret_cast<uint4*>(stg + lane * kEpiPitch + 16 * j) =
                            make_uint4(tc::pack16<F16>(f[8 * j], f[8 * j + 1]), tc::pack16<F16>(f[8 * j + 2], f[8 * j + 3]),
                                       tc::pack16<F16>(f[8 * j + 4], f[8 * j + 5]), tc::pack16<F16>(f[8 * j + 6], f[8 * j + 7]));
                    __syncwarp();
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int rl = (lane >> 2) + 8 * j;
                        const uint4 val = *reinterpret_cast<const uint4*>(stg + rl * kEpiPitch + 16 * (lane & 3));
                        if (rbase + rl < p.M)
                            *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out) + (size_t)(rbase + rl) * p.ldo + col0 + 8 * (lane & 3)) = val;
                    }
                } else {
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh) {
                        __syncwarp();
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            *reinterpret_cast<float4*>(stg + lane * kEpiPitch + 16 * j) =
                                make_float4(f[16 * hh + 4 * j], f[16 * hh + 4 * j + 1], f[16 * hh + 4 * j + 2], f[16 * hh + 4 * j + 3]);
                        __syncwarp();
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const int rl = (lane >> 2) + 8 * j;
                            float4 val = *reinterpret_cast<const float4*>(stg + rl * kEpiPitch + 16 * (lane & 3));
                            if (rbase + rl < p.M) {
                                if (MODE == FB_GEMM_BIAS_RESIDUAL_F32) {
                                    const float4 r4 = rr[hh * 4 + j];
                                    val.x += r4.x; val.y += r4.y; val.z += r4.z; val.w += r4.w;
                                    if (p.out16) {
                                        *reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(p.out16) + (size_t)(rbase + rl) * p.ldo16 + col0 + 16 * hh + 4 * (lane & 3)) =
                                            make_uint2(tc::pack16<F16>(val.x, val.y), tc::pack16<F16>(val.z, val.w));
                                        st_s[j] += (val.x + val.y) + (val.z + val.w);
                                        st_q[j] += fmaf(val.x, val.x, val.y * val.y) + fmaf(val.z, val.z, val.w * val.w);
                                    }
                                }
                                *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + (size_t)(rbase + rl) * p.ldo + col0 + 16 * hh + 4 * (lane & 3)) = val;
                            }
                        }
                    }
                }
            };

            if (MODE == FB_GEMM_BIAS_GELU_BF16 && kChunks == 2 && FB_GELU_EARLY_RELEASE) {
                // 16 warps x 64 columns: the whole slice of the accumulator fits in registers, so the TMEM buffer goes
                // back to the MMA issuer before any of the erf-GELU math (the next-but-one tile no longer waits for it)
                uint32_t va[32], vb[32];
                float4 rz[8];
                tc::tmem_ld_32x32(taddr, va);
                tc::tmem_ld_32x32(taddr + 32, vb);
                tc::tmem_ld_wait();
                tc::tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if (CL2) tc::mbar_arrive_cluster(tc::mapa_u32(tc::smem_u32(&tmem_empty[acc]), 0u));
                    else tc::mbar_arrive(&tmem_empty[acc]);
                }
                process(va, 0, rz);
                process(vb, 1, rz);
            } else if (MODE == FB_GEMM_BIAS_GELU_BF16) {
                // erf-GELU is register hungry: one register set, chunk after chunk
                uint32_t va[32];
                float4 rz[8];
#pragma unroll 1
                for (int c = 0; c < kChunks; ++c) {
                    tc::tmem_ld_32x32(taddr + 32 * c, va);
                    tc::tmem_ld_wait();
                    if (c == kChunks - 1) {
                        tc::tc_fence_before();
                        __syncwarp();
                        if (lane == 0) {
                            if (CL2) tc::mbar_arrive_cluster(tc::mapa_u32(tc::smem_u32(&tmem_empty[acc]), 0u));   // the leader waits for both CTAs
                            else tc::mbar_arrive(&tmem_empty[acc]);
                        }
                    }
                    process(va, c, rz);
                }
            } else if (MODE == FB_GEMM_BIAS_RESIDUAL_F32) {
                static_assert(MODE == FB_GEMM_BIAS_GELU_BF16 || kChunks == 4, "these epilogues walk four 32-column chunks");
                // one accumulator register set, two residual sets: the (coalesced) residual loads of chunk
                // c+1 are in flight while chunk c is added and stored
                uint32_t va[32];
                float4 ra[8], rb[8];
                prefetch_res(ra, 0);
                tc::tmem_ld_32x32(taddr, va);
                prefetch_res(rb, 1);
                tc::tmem_ld_wait();
                process(va, 0, ra);
                tc::tmem_ld_32x32(taddr + 32, va);
                prefetch_res(ra, 2);
                tc::tmem_ld_wait();
                process(va, 1, rb);
                tc::tmem_ld_32x32(taddr + 64, va);
                prefetch_res(rb, 3);
                tc::tmem_ld_wait();
                process(va, 2, ra);
                tc::tmem_ld_32x32(taddr + 96, va);
                tc::tmem_ld_wait();
                tc::tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                            if (CL2) tc::mbar_arrive_cluster(tc::mapa_u32(tc::smem_u32(&tmem_empty[acc]), 0u));   // the leader waits for both CTAs
                            else tc::mbar_arrive(&tmem_empty[acc]);
                        }
                process(va, 3, rb);
                if (p.out16) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        float a = st_s[j], b = st_q[j];
                        a += __shfl_xor_sync(0xffffffffu, a, 1);
                        b += __shfl_xor_sync(0xffffffffu, b, 1);
                        a += __shfl_xor_sync(0xffffffffu, a, 2);
                        b += __shfl_xor_sync(0xffffffffu, b, 2);
                        const int rl = (lane >> 2) + 8 * j;
                        if ((lane & 3) == 0 && rbase + rl < p.M && ncol0 < p.N)
                            *reinterpret_cast<float2*>(p.row_stats + ((size_t)(rbase + rl) * p.ln_slots + (ncol0 >> 7)) * 2) = make_float2(a, b);
                    }
                }
            } else {
                // two register sets: the tcgen05.ld of chunk c+1 is in flight while chunk c is processed
                uint32_t va[32], vb[32];
                float4 ra[8], rb[8];
                tc::tmem_ld_32x32(taddr, va);
                prefetch_res(ra, 0);
                tc::tmem_ld_wait();
                tc::tmem_ld_32x32(taddr + 32, vb);
                prefetch_res(rb, 1);
                process(va, 0, ra);
                tc::tmem_ld_wait();
                tc::tmem_ld_32x32(taddr + 64, va);
                prefetch_res(ra, 2);
                process(vb, 1, rb);
                tc::tmem_ld_wait();
                tc::tmem_ld_32x32(taddr + 96, vb);
                prefetch_res(rb, 3);
                process(va, 2, ra);
                tc::tmem_ld_wait();
                // the accumulator is in registers now: hand the TMEM buffer back before the last chunk's math
                tc::tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                            if (CL2) tc::mbar_arrive_cluster(tc::mapa_u32(tc::smem_u32(&tmem_empty[acc]), 0u));   // the leader waits for both CTAs
                            else tc::mbar_arrive(&tmem_empty[acc]);
                        }
                process(vb, 3, rb);
            }
            ++iter;
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    if (CL2) tc::cluster_sync_all();     // the peer may still arrive on this CTA's barriers until it is done too
    if (warp == 1) {
        if (CL2) tc::tmem_dealloc_pair(tmem_base, 512);
        else tc::tmem_dealloc(tmem_base, 512);
    }
}

// ---- tensor-map encoding through the driver entry point (no link against libcuda) ------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    });
    return fn;
}

}  // namespace

int make_tmap_bf16_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t row_stride_elems,
                      uint32_t box_rows, uint32_t box_cols) {
    EncodeTiledFn fn = encode_fn();
    FB_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
    FB_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0 && (row_stride_elems * 2) % 16 == 0,
               "TMA needs a 16-byte aligned base and row pitch");
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {row_stride_elems * 2};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    FB_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return 0;
}

// Clusters of two CTAs that can be co-resident for a kernel (the persistent grid must not exceed it).
template <typename K>
static int max_cluster_pairs(K kernel, int threads, int smem_bytes, int* out) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * sm_count(), 1, 1);
    cfg.blockDim = dim3(threads, 1, 1);
    cfg.dynamicSmemBytes = smem_bytes;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n = 0;
    FB_CUDA_OK(cudaOccupancyMaxActiveClusters(&n, kernel, &cfg));
    *out = n;
    return 0;
}

template <typename K>
static int launch_cluster2(K kernel, int pairs, int threads, int smem_bytes, const CUtensorMap& ta, const CUtensorMap& tb, const GemmArgs& p,
                           cudaStream_t stream) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * pairs, 1, 1);
    cfg.blockDim = dim3(threads, 1, 1);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    FB_CUDA_OK(cudaLaunchKernelEx(&cfg, kernel, ta, tb, p));
    return 0;
}

static int launch_gemm_common(const void* d_a, long long lda, const void* d_b, long long ldb, GemmArgs p, cudaStream_t stream) {
    // clusters of two with a multicast B tile: the ViT-layer GEMMs (large M, B = weights)
    const bool cl2 = p.mode != FB_GEMM_THRESHOLD_PAIRS && p.mode != FB_GEMM_F32 && p.M >= 4 * BM && p.N % BN == 0;
    CUtensorMap ta, tb;
    int rc = make_tmap_bf16_2d(&ta, d_a, (uint64_t)p.M, (uint64_t)p.K, (uint64_t)lda, BM, BK);
    if (rc) return rc;
    rc = make_tmap_bf16_2d(&tb, d_b, (uint64_t)p.N, (uint64_t)p.K, (uint64_t)ldb, cl2 ? BN / 2 : BN, BK);
    if (rc) return rc;
    const int tiles_m = (p.M + BM - 1) / BM, tiles_n = (p.N + BN - 1) / BN;
    const int tiles = tiles_m * tiles_n;
    const int grid = tiles < sm_count() ? tiles : sm_count();
#define FB_LAUNCH_MODE(MODE_)                                                                                          \
    case MODE_: {                                                                                                      \
        static PerDeviceFlag attr_set;                                                                                  \
        constexpr int threads_ = gemm_threads(MODE_, false), smem_ = gemm_smem_bytes(MODE_, false);                    \
        if (!attr_set.get()) {                                                                                               \
            FB_CUDA_OK(cudaFuncSetAttribute(gemm_bf16_kernel<MODE_, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_)); \
            FB_CUDA_OK(cudaFuncSetAttribute(gemm_bf16_kernel<MODE_, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_)); \
            attr_set.set();                                                                                           \
        }                                                                                                              \
        if (p.f16) gemm_bf16_kernel<MODE_, true, false><<<grid, threads_, smem_, stream>>>(ta, tb, p);                 \
        else gemm_bf16_kernel<MODE_, false, false><<<grid, threads_, smem_, stream>>>(ta, tb, p);                      \
        break;                                                                                                         \
    }
// Kernel attributes and the co-resident cluster count are per device (one process may drive several GPUs): a
// PerDeviceFlag plus one pair count per device ordinal, the same pattern as sm_count().
#define FB_LAUNCH_MODE_CL2(MODE_)                                                                                      \
    case MODE_: {                                                                                                      \
        static PerDeviceFlag attr_set;                                                                                 \
        static std::atomic<int> max_pairs_dev[64];                                                                     \
        constexpr int threads_ = gemm_threads(MODE_, true), smem_ = gemm_smem_bytes(MODE_, true);                      \
        if (!attr_set.get()) {                                                                                         \
            FB_CUDA_OK(cudaFuncSetAttribute(gemm_bf16_kernel<MODE_, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_)); \
            FB_CUDA_OK(cudaFuncSetAttribute(gemm_bf16_kernel<MODE_, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_)); \
            int a_ = 0, b_ = 0;                                                                                        \
            rc = max_cluster_pairs(gemm_bf16_kernel<MODE_, false, true>, threads_, smem_, &a_);                        \
            if (rc) return rc;                                                                                         \
            rc = max_cluster_pairs(gemm_bf16_kernel<MODE_, true, true>, threads_, smem_, &b_);                         \
            if (rc) return rc;                                                                                         \
            max_pairs_dev[PerDeviceFlag::device()].store(a_ < b_ ? a_ : b_, std::memory_order_relaxed);                \
            attr_set.set();                                                                                            \
        }                                                                                                              \
        const int max_pairs = max_pairs_dev[PerDeviceFlag::device()].load(std::memory_order_relaxed);                  \
        const int work_ = ((tiles_m + 1) / 2) * tiles_n;                                                               \
        const int pairs_ = work_ < max_pairs ? work_ : max_pairs;                                                      \
        FB_REQUIRE(pairs_ >= 1, "fb_gemm_bf16: no cluster of two CTAs fits on this device");                          \
        rc = p.f16 ? launch_cluster2(gemm_bf16_kernel<MODE_, true, true>, pairs_, threads_, smem_, ta, tb, p, stream)  \
                   : launch_cluster2(gemm_bf16_kernel<MODE_, false, true>, pairs_, threads_, smem_, ta, tb, p, stream);\
        if (rc) return rc;                                                                                             \
        break;                                                                                                         \
    }
    if (cl2) {
        switch (p.mode) {
            FB_LAUNCH_MODE_CL2(FB_GEMM_BIAS_BF16)
            FB_LAUNCH_MODE_CL2(FB_GEMM_BIAS_GELU_BF16)
            FB_LAUNCH_MODE_CL2(FB_GEMM_BIAS_RESIDUAL_F32)
            default:
                FB_REQUIRE(false, "fb_gemm_bf16: unknown epilogue mode %d", p.mode);
        }
    } else {
        switch (p.mode) {
            FB_LAUNCH_MODE(FB_GEMM_BIAS_BF16)
            FB_LAUNCH_MODE(FB_GEMM_BIAS_GELU_BF16)
            FB_LAUNCH_MODE(FB_GEMM_BIAS_RESIDUAL_F32)
            FB_LAUNCH_MODE(FB_GEMM_F32)
            FB_LAUNCH_MODE(FB_GEMM_THRESHOLD_PAIRS)
            default:
                FB_REQUIRE(false, "fb_gemm_bf16: unknown epilogue mode %d", p.mode);
        }
    }
#undef FB_LAUNCH_MODE
#undef FB_LAUNCH_MODE_CL2
    FB_CUDA_OK(cudaGetLastError());
    return 0;
}

// Candidate pairs of one block of the all-pairs scan: the m rows at d_a (global row index a_offset + i) against the n rows at
// d_b (global index b_offset + j).  triangle != 0 keeps only global column > global row (a block on the diagonal);
// the candidate counter is NOT reset, so the blocks of one scan append to the same list.
int launch_cosine_block(const void* d_a_bf16, int m, int a_offset, const void* d_b_bf16, int n, int b_offset, long long ld, int k, float tau,
                        int triangle, int* d_pairs, float* d_sims, long long cap, unsigned long long* d_count, cudaStream_t stream) {
    FB_REQUIRE(d_a_bf16 && d_b_bf16 && d_pairs && d_sims && d_count, "fb_cosine_block: null pointer");
    FB_REQUIRE(n >= 1 && m >= 1 && a_offset >= 0 && b_offset >= 0, "fb_cosine_block: bad block");
    FB_REQUIRE(k >= BK && k % BK == 0, "fb_cosine_block: embedding dim must be a multiple of %d", BK);
    GemmArgs p{};
    p.M = m; p.N = n; p.K = k; p.mode = FB_GEMM_THRESHOLD_PAIRS;
    p.tau = tau; p.row_offset = a_offset; p.col_offset = b_offset; p.tri_on = triangle ? 1 : 0;
    p.pairs = d_pairs; p.pair_sims = d_sims; p.pair_cap = cap; p.pair_count = d_count;
    return launch_gemm_common(d_a_bf16, ld, d_b_bf16, ld, p, stream);
}

// Candidate pairs of the cosine similarity stage: rows [row_offset, row_offset+m) of E against all n rows.
int launch_cosine_candidates(const void* d_emb_bf16, long long ld, int n, int row_offset, int m, int k, float tau,
                             int* d_pairs, float* d_sims, long long cap, unsigned long long* d_count,
                             cudaStream_t stream) {
    FB_REQUIRE(n >= 1 && m >= 1 && row_offset >= 0 && row_offset + m <= n, "fb_cosine_pairs: bad row range");
    const __nv_bfloat16* a = reinterpret_cast<const __nv_bfloat16*>(d_emb_bf16) + (size_t)row_offset * ld;
    return launch_cosine_block(a, m, row_offset, d_emb_bf16, n, 0, ld, k, tau, 1, d_pairs, d_sims, cap, d_count, stream);
}

int launch_gemm_bf16_ln(const void* d_a, long long lda, const void* d_b, long long ldb, int M, int N, int K, int mode,
                        const float* d_bias, void* d_out, long long ldo, const float* d_residual, long long ldr,
                        const GemmLnFold* ln, cudaStream_t stream) {
    FB_REQUIRE(d_a && d_b && d_out, "fb_gemm_bf16: null pointer");
    FB_REQUIRE(M >= 1 && N >= 1 && K >= BK && K % BK == 0, "fb_gemm_bf16: K must be a positive multiple of %d (got %d)", BK, K);
    FB_REQUIRE(N % 32 == 0, "fb_gemm_bf16: N must be a multiple of 32 (got %d)", N);
    const int f16 = (mode & FB_GEMM_F16_FLAG) ? 1 : 0;
    mode &= ~FB_GEMM_F16_FLAG;
    FB_REQUIRE(mode >= 0 && mode <= 3, "fb_gemm_bf16: unknown epilogue mode %d", mode);
    FB_REQUIRE(mode != FB_GEMM_BIAS_RESIDUAL_F32 || d_residual, "fb_gemm_bf16: residual pointer required");
    const int out_elt = (mode == FB_GEMM_BIAS_BF16 || mode == FB_GEMM_BIAS_GELU_BF16) ? 2 : 4;
    FB_REQUIRE((reinterpret_cast<uintptr_t>(d_out) & 15) == 0 && (ldo * out_elt) % 16 == 0, "fb_gemm_bf16: output not 16-byte aligned");
    FB_REQUIRE(!d_bias || (reinterpret_cast<uintptr_t>(d_bias) & 15) == 0, "fb_gemm_bf16: bias not 16-byte aligned");
    FB_REQUIRE(!d_residual || ((reinterpret_cast<uintptr_t>(d_residual) & 15) == 0 && (ldr * 4) % 16 == 0), "fb_gemm_bf16: residual not aligned");
    GemmArgs p{};
    p.M = M; p.N = N; p.K = K; p.mode = mode; p.bias = d_bias; p.out = d_out; p.ldo = ldo;
    p.residual = d_residual; p.ldr = ldr; p.f16 = f16;
    if (ln) {
        if (mode == FB_GEMM_BIAS_RESIDUAL_F32) {
            FB_REQUIRE(ln->out16 && ln->row_stats && ln->ln_slots * 128 == N && (ln->ldo16 * 2) % 8 == 0 &&
                       (reinterpret_cast<uintptr_t>(ln->out16) & 7) == 0 && (reinterpret_cast<uintptr_t>(ln->row_stats) & 7) == 0,
                       "LayerNorm fold (producer): needs the 16-bit copy, the row sums and N = 128 * slots");
            p.out16 = ln->out16; p.ldo16 = ln->ldo16; p.row_stats = ln->row_stats; p.ln_slots = ln->ln_slots;
        } else {
            FB_REQUIRE((mode == FB_GEMM_BIAS_BF16 || mode == FB_GEMM_BIAS_GELU_BF16) && ln->ln_s && ln->row_stats && ln->ln_slots >= 1 &&
                       ln->ln_width >= 1 && d_bias && (reinterpret_cast<uintptr_t>(ln->ln_s) & 15) == 0,
                       "LayerNorm fold (consumer): needs the column sums, the folded bias and the row sums");
            p.ln_s = ln->ln_s; p.row_stats = ln->row_stats; p.ln_slots = ln->ln_slots; p.ln_width = ln->ln_width;
        }
    }
    return launch_gemm_common(d_a, lda, d_b, ldb, p, stream);
}

int launch_gemm_bf16(const void* d_a, long long lda, const void* d_b, long long ldb, int M, int N, int K, int mode,
                     const float* d_bias, void* d_out, long long ldo, const float* d_residual, long long ldr,
                     cudaStream_t stream) {
    return launch_gemm_bf16_ln(d_a, lda, d_b, ldb, M, N, K, mode, d_bias, d_out, ldo, d_residual, ldr, nullptr, stream);
}

}  // namespace fb
