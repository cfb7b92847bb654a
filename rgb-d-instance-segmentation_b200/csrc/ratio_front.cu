// K4a+K4b fused: the multi-scale stem AND the point-wise middle of EnhancedDepthImageRatioPredictor.forward
// (reference mask2former/utils/custom_model.py:1458-1470) as ONE tcgen05 kernel on CTA pairs:
//     ms  = ReLU(BN(cat[Conv3x3, Conv5x5, Conv7x7](depth)))           CM:1458-1463   GEMM 1: K = 256 (row-im2col), N = 192
//     f   = ReLU(BN(Conv1x1_{192->128}(ms)))                           CM:1466        GEMM 2: K = 192, N = 128
//     a   = sigmoid(Conv1x1_{64->128}(ReLU(Conv1x1_{128->64}(f))))     CM:1469        GEMM 3: K = 128, N = 64; GEMM 4: K = 64, N = 128
//     out = f * a                                                       CM:1470
// Only the 128-byte/pixel row-im2col operand streams in (TMA ring) and the 128-channel bf16 result leaves (TMA store):
// the 192-channel stem output, f and the attention hidden layer live in TENSOR MEMORY as packed bf16 and feed the next
// GEMM as its A operand (tcgen05.mma with A in TMEM).  All four weight matrices (176 KB) stay resident in shared
// memory, split by output rows between the two CTAs of a pair (cta_group::2, M = 256 = two 128-pixel tiles).
//
// The epilogues are bound by the TMEM read rate (~64 B/clk/SM: 512 accumulator columns per tile = 4096 cycles) while
// the MMAs need 2816 cycles per tile, so TWO tile chains are kept in flight per CTA, each with its own eight epilogue
// warps.  Three MMA-issuing threads (stem GEMMs; chain 0; chain 1) each block on exactly the barrier they need.  TMEM columns (480 of 512):
//     P_c = 192*c .. +192   chain c:  acc1 [0,192) -> acc2 [0,128) | f bf16 [128,192) -> acc3 [0,64) | relu bf16 [160,192)
//                                      -> acc4 [0,128)          (each reuse only after the previous owner was consumed)
//     Q   = [384,480)       ms as bf16 (A operand of GEMM 2), shared by both chains (the other chain's GEMM 2 must be done)
// f is also stashed in shared memory (the output staging tile) for the final gating, so it is read from TMEM only once.
#include "common.cuh"
#include "rgbd_b200.h"
#include "tc_ptx.cuh"
#include "tma_host.cuh"

namespace {

constexpr int kBlockM = 128;
constexpr int kThreads = 640;                 // 4 control warps + 2 chains x 8 epilogue warps
constexpr int kChainThreads = 256;            // epilogue threads per chain: two warps (column halves) per TMEM lane quarter
constexpr int kSliceBytes = kBlockM * 128;    // 16 KB
// Stem operand, two layouts (template parameter EM):
//  EM = false  R (B,H+6,W,64): row-im2col written by ratio_stem_pack (128 B per pixel and row); 4 K-slices of 64 per tile
//  EM = true   E (B,2,H+6,Wp,4): the depth image itself, channels-last with c padded to 4 (8 B per pixel) and zero borders,
//              in two copies shifted by one pixel.  The 8 dx taps x 4 channels of a pixel are 64 CONTIGUOUS bytes of E, so a
//              tensor map whose pixel dimension has a 16-byte stride (two pixels) under a 64-byte inner box is the im2col
//              along x for free (overlapping strides are legal for tiled TMA: profiles/micro/tma_overlap.cu); copy 0 serves
//              the even pixels, copy 1 the odd ones (16-byte alignment).  7 K-blocks of 32 (one per row tap, 64-byte swizzle),
//              tile rows 0..63 = even pixels, 64..127 = odd pixels; the output store uses pixel-stride-2 tensor maps.
//              HBM: the 1.27 GB R tensor (batch 32) is replaced by 0.16 GB that stays in L2.
template <bool EM> struct StemCfg;
template <> struct StemCfg<false> { static constexpr int kBlocks = 4, kStageBytes = 16384, kStages = 4, kW1Block = 96 * 128, kMmaPerBlock = 4, kRowBytes = 128; };
template <> struct StemCfg<true> { static constexpr int kBlocks = 7, kStageBytes = 8192, kStages = 9, kW1Block = 96 * 64, kMmaPerBlock = 2, kRowBytes = 64; };
constexpr int kMaxStages = 12;
constexpr int kW2Half = 3 * 64 * 128;         //          64 of 128 rows x 3 K-slices      24 KB
constexpr int kW3Half = 2 * 32 * 128;         //          32 of  64 rows x 2 K-slices       8 KB
constexpr int kW4Half = 1 * 64 * 128;         //          64 of 128 rows x 1 K-slice        8 KB
constexpr int kWRest = kW2Half + kW3Half + kW4Half;
constexpr int kStashBytes = 2 * kSliceBytes;  // per chain: 128 pixels x 128 channels bf16 (f, then out)
constexpr uint32_t kColQ = 384;

struct FrontParams {
    int n_img, tiles_x, tiles_y, BX, BY, total_tiles;
    const float* sh1;
    const float* sh2;
    const float* sh3;
    const float* sh4;
};

struct alignas(16) FrontCtl {
    uint64_t full[kMaxStages];
    uint64_t empty[kMaxStages];
    uint64_t w_full;
    uint64_t acc_full[2][4];      // [chain][GEMM 1..4]   multicast commit -> both CTAs
    uint64_t x_ready[2][3];       // [chain][after E1..E3] epilogue threads of BOTH CTAs (counted in the leader)
    uint64_t p_free[2];           // acc4 of the chain was read: its P columns may be overwritten by the next GEMM 1
    uint32_t tmem_base;
    uint32_t pad;
};

__device__ __forceinline__ void decode(const FrontParams& p, int t, int& img, int& ty, int& tx) {
    ty = t % p.tiles_y; t /= p.tiles_y;       // walk down columns: the 4 row taps of the stem re-hit L2
    tx = t % p.tiles_x;
    img = t / p.tiles_x;
}

template <bool EM>
__global__ void __launch_bounds__(kThreads, 1)
ratio_front_kernel(const __grid_constant__ CUtensorMap tmap_r, const __grid_constant__ CUtensorMap tmap_r1,
                   const __grid_constant__ CUtensorMap tmap_w1, const __grid_constant__ CUtensorMap tmap_w2,
                   const __grid_constant__ CUtensorMap tmap_w3, const __grid_constant__ CUtensorMap tmap_w4,
                   const __grid_constant__ CUtensorMap tmap_out, const __grid_constant__ CUtensorMap tmap_out1,
                   const __grid_constant__ FrontParams p) {
    using Cfg = StemCfg<EM>;
    constexpr int kStages = Cfg::kStages, kStageBytes = Cfg::kStageBytes, kW1Half = Cfg::kBlocks * Cfg::kW1Block;
    constexpr int kWBytes = kW1Half + kWRest;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* s_w1 = smem;
    uint8_t* s_w2 = s_w1 + kW1Half;
    uint8_t* s_w3 = s_w2 + kW2Half;
    uint8_t* s_w4 = s_w3 + kW3Half;
    uint8_t* s_ring = s_w4 + kW4Half;
    uint8_t* s_stash = s_ring + kStages * kStageBytes;
    FrontCtl* ctl = reinterpret_cast<FrontCtl*>(s_stash + 2 * kStashBytes);
    float* s_sh1 = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(ctl) + sizeof(FrontCtl));
    float* s_sh2 = s_sh1 + 192;
    float* s_sh3 = s_sh2 + 128;
    float* s_sh4 = s_sh3 + 64;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = tc::cluster_ctarank();
    const bool leader = rank == 0;
    for (int i = threadIdx.x; i < 192; i += blockDim.x) {
        s_sh1[i] = p.sh1[i];
        if (i < 128) {
            s_sh2[i] = p.sh2[i];
            s_sh4[i] = p.sh4[i];
        }
        if (i < 64) s_sh3[i] = p.sh3[i];
    }
    if (warp == 0 && lane == 0) {
        tc::prefetch_tmap(&tmap_r);
        if (EM) tc::prefetch_tmap(&tmap_r1);
        if (EM) tc::prefetch_tmap(&tmap_out1);
        tc::prefetch_tmap(&tmap_w1);
        tc::prefetch_tmap(&tmap_w2);
        tc::prefetch_tmap(&tmap_w3);
        tc::prefetch_tmap(&tmap_w4);
        tc::prefetch_tmap(&tmap_out);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < kStages; ++s) {
            tc::mbar_init(&ctl->full[s], 1);
            tc::mbar_init(&ctl->empty[s], 1);
        }
        tc::mbar_init(&ctl->w_full, 1);
        for (int c = 0; c < 2; ++c) {
            for (int g = 0; g < 4; ++g) tc::mbar_init(&ctl->acc_full[c][g], 1);
            for (int g = 0; g < 3; ++g) tc::mbar_init(&ctl->x_ready[c][g], 2 * (kChainThreads / 32));   // one arrive per warp
            tc::mbar_init(&ctl->p_free[c], 2 * (kChainThreads / 32));
        }
        tc::fence_barrier_init();
    }
    tc::cluster_sync_all();
    if (warp == 2) tc::tmem_alloc_2cta(&ctl->tmem_base, 512);
    tc::tc_fence_before();
    tc::cluster_sync_all();
    tc::tc_fence_after();
    const uint32_t tmem = ctl->tmem_base;

    // work units = pairs of adjacent tiles (2u, 2u+1); chain c of the cluster takes its units u_begin + 2i + c
    const int n_units = (p.total_tiles + 1) / 2;
    const int n_clusters = gridDim.x / 2, cid = blockIdx.x / 2;
    const int per = n_units / n_clusters, rem = n_units % n_clusters;
    const int u_begin = cid * per + min(cid, rem);
    const int n_mine = per + (cid < rem ? 1 : 0);
    const int n_a = (n_mine + 1) / 2, n_b = n_mine / 2;

    if (warp == 0 && lane == 0) {
        // ================= TMA producer: resident weight halves, then the row-im2col slices =================
        if (leader) tc::mbar_expect_tx(&ctl->w_full, 2u * kWBytes);
        for (int j = 0; j < Cfg::kBlocks; ++j)
            tc::tma_load_2d_2cta(s_w1 + j * Cfg::kW1Block, &tmap_w1, &ctl->w_full, j * (Cfg::kRowBytes / 2), (int)rank * 96);
        for (int j = 0; j < 3; ++j) tc::tma_load_2d_2cta(s_w2 + j * (64 * 128), &tmap_w2, &ctl->w_full, j * 64, (int)rank * 64);
        for (int j = 0; j < 2; ++j) tc::tma_load_2d_2cta(s_w3 + j * (32 * 128), &tmap_w3, &ctl->w_full, j * 64, (int)rank * 32);
        tc::tma_load_2d_2cta(s_w4, &tmap_w4, &ctl->w_full, 0, (int)rank * 64);
        int stage = 0;
        uint32_t phase = 0;
        for (int n = 0; n < n_mine; ++n) {
            int img, ty, tx;
            decode(p, 2 * (u_begin + n) + (int)rank, img, ty, tx);
            for (int j = 0; j < Cfg::kBlocks; ++j) {
                tc::mbar_wait(&ctl->empty[stage], phase ^ 1);
                if (leader) tc::mbar_expect_tx(&ctl->full[stage], 2u * kStageBytes);
                if (EM) {       // row tap dy = j: E row y + j; even pixels from copy 0, odd pixels from copy 1 (64 pixel pairs each)
                    tc::tma_load_4d_2cta(s_ring + stage * kStageBytes, &tmap_r, &ctl->full[stage], 0, tx * 64, ty + j, img);
                    tc::tma_load_4d_2cta(s_ring + stage * kStageBytes + kStageBytes / 2, &tmap_r1, &ctl->full[stage], 0, tx * 64,
                                         ty + j, img);
                } else {        // slice j holds taps dy = 2j, 2j+1: rows y + 2j of R
                    tc::tma_load_4d_2cta(s_ring + stage * kStageBytes, &tmap_r, &ctl->full[stage], 0, tx * p.BX, ty * p.BY + 2 * j, img);
                }
                if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1 && leader) {
        // ================= MMA issuer 1 (leader): the stem GEMMs of both chains, in the tile order of the TMA ring ======
        // The tensor pipe executes MMAs in issue order, so a whole GEMM 1 (1536 cycles) queued at once would park the other
        // chain's short GEMMs 2-4 behind it: issue one K-slice (384 cycles), wait until it has executed, issue the next.
        const uint32_t idesc192 = tc::make_idesc_bf16(2 * kBlockM, 192);
        tc::mbar_wait(&ctl->w_full, 0);
        tc::tc_fence_after();
        int stage = 0;
        uint32_t phase = 0;
        for (int n = 0; n < n_mine; ++n) {
            const int c = n & 1, i = n >> 1;
            tc::mbar_wait(&ctl->p_free[c], (uint32_t)((i & 1) ^ 1));      // acc4 of the chain's previous tile was read
            tc::tc_fence_after();
            const uint32_t d = tmem + (uint32_t)(c * 192);
            for (int j = 0; j < Cfg::kBlocks; ++j) {
                tc::mbar_wait(&ctl->full[stage], phase);
                tc::tc_fence_after();
                const uint64_t adesc = tc::make_kmajor_desc(tc::smem_u32(s_ring + stage * kStageBytes), Cfg::kRowBytes);
                const uint64_t bdesc = tc::make_kmajor_desc(tc::smem_u32(s_w1 + j * Cfg::kW1Block), Cfg::kRowBytes);
                if (tc::elect_one()) {
#pragma unroll
                    for (int k = 0; k < Cfg::kMmaPerBlock; ++k)
                        tc::umma_bf16_2cta(d, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc192, (j | k) != 0);
                    tc::umma_commit_2cta(&ctl->empty[stage]);
                    if (j == Cfg::kBlocks - 1) tc::umma_commit_2cta(&ctl->acc_full[c][0]);
                }
                __syncwarp();
                // throttle: at most ~384 cycles of stem MMAs queued ahead of the other chain's short GEMMs
                if (j != Cfg::kBlocks - 1 && (!EM || (j & 1))) tc::mbar_wait(&ctl->empty[stage], phase);
                if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
        }
    } else if ((warp == 2 || warp == 3) && leader) {
        // whole warp runs the (uniform) control flow so the descriptors stay in uniform registers; one elected lane issues
        // ================= MMA issuers 2/3 (leader): GEMMs 2-4 of chain 0 / chain 1, A operand in tensor memory ==========
        const int c = warp - 2;
        const uint32_t idesc128 = tc::make_idesc_bf16(2 * kBlockM, 128);
        const uint32_t idesc64 = tc::make_idesc_bf16(2 * kBlockM, 64);
        const uint32_t d = tmem + (uint32_t)(c * 192);
        const uint64_t w2d = tc::make_kmajor_desc(tc::smem_u32(s_w2), 128);
        const uint64_t w3d = tc::make_kmajor_desc(tc::smem_u32(s_w3), 128);
        const uint64_t w4d = tc::make_kmajor_desc(tc::smem_u32(s_w4), 128);
        tc::mbar_wait(&ctl->w_full, 0);
        tc::tc_fence_after();
        const int n_c = c == 0 ? n_a : n_b;
        for (int i = 0; i < n_c; ++i) {
            const uint32_t ph = (uint32_t)(i & 1);
            // GEMM 2: acc2 = ms(bf16, TMEM Q) . W2^T   (K = 192: 12 MMAs, A advances 8 columns, B 32 bytes / 8 KB per slice)
            tc::mbar_wait(&ctl->x_ready[c][0], ph);
            tc::tc_fence_after();
            if (tc::elect_one()) {
#pragma unroll
                for (int k = 0; k < 12; ++k)
                    tc::umma_bf16_ts_2cta(d, tmem + kColQ + (uint32_t)(k * 8), w2d + (uint64_t)((k >> 2) * ((64 * 128) >> 4) + (k & 3) * 2),
                                      idesc128, k != 0);
                tc::umma_commit_2cta(&ctl->acc_full[c][1]);
            }
            __syncwarp();
            // GEMM 3: acc3 = f(bf16, TMEM P+128) . W3^T   (K = 128: 8 MMAs)
            tc::mbar_wait(&ctl->x_ready[c][1], ph);
            tc::tc_fence_after();
            if (tc::elect_one()) {
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    tc::umma_bf16_ts_2cta(d, d + 128u + (uint32_t)(k * 8), w3d + (uint64_t)((k >> 2) * ((32 * 128) >> 4) + (k & 3) * 2), idesc64,
                                      k != 0);
                tc::umma_commit_2cta(&ctl->acc_full[c][2]);
            }
            __syncwarp();
            // GEMM 4: acc4 = relu(.)(bf16, TMEM P+160) . W4^T   (K = 64: 4 MMAs)
            tc::mbar_wait(&ctl->x_ready[c][2], ph);
            tc::tc_fence_after();
            if (tc::elect_one()) {
#pragma unroll
                for (int k = 0; k < 4; ++k) tc::umma_bf16_ts_2cta(d, d + 160u + (uint32_t)(k * 8), w4d + (uint64_t)(k * 2), idesc128, k != 0);
                tc::umma_commit_2cta(&ctl->acc_full[c][3]);
            }
            __syncwarp();
        }
    } else if (warp >= 4) {
        // ================= epilogue: chain c = warps 4..11 / 12..19; a thread owns one pixel row and every other
        // 32-column chunk (h = column half), so two warps work on each TMEM lane quarter of a chain =================
        const int c = (warp - 4) >> 3;
        const int h = ((warp - 4) >> 2) & 1;
        const int q = warp & 3;
        const int row = q * 32 + lane;
        const uint32_t P = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(c * 192);
        const uint32_t Q = tmem + ((uint32_t)(q * 32) << 16) + kColQ;
        uint8_t* stash = s_stash + c * kStashBytes;
        const bool issuer = (warp == 4 + 8 * c) && lane == 0;
        const int bar_id = 1 + c;
        uint32_t x_remote[3], p_free_remote;
        for (int g = 0; g < 3; ++g) x_remote[g] = tc::mapa(tc::smem_u32(&ctl->x_ready[c][g]), 0);
        p_free_remote = tc::mapa(tc::smem_u32(&ctl->p_free[c]), 0);
        const int n_c = c == 0 ? n_a : n_b;
        for (int i = 0; i < n_c; ++i) {
            const uint32_t ph = (uint32_t)(i & 1);
            int img, ty, tx;
            decode(p, 2 * (u_begin + 2 * i + c) + (int)rank, img, ty, tx);

            // ---- E1: ms = relu(acc1 + sh1) -> bf16 -> TMEM Q (shared: the other chain's GEMM 2 must have read it)
            tc::mbar_wait_sleep(&ctl->acc_full[c][0], ph);
            if (c == 1) tc::mbar_wait_sleep(&ctl->acc_full[0][1], ph);
            else if (i > 0) tc::mbar_wait_sleep(&ctl->acc_full[1][1], ph ^ 1);
            tc::tc_fence_after();
#pragma unroll 1
            for (int k = h; k < 6; k += 2) {
                uint32_t v[32];
                tc::tmem_ld_32x32(P + k * 32, v);
                tc::tmem_ld_wait();
                uint32_t o[16];
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4) {
                    const float4 b = *reinterpret_cast<const float4*>(s_sh1 + k * 32 + j4 * 4);
                    o[j4 * 2] = tc::pack_bf16x2_relu(__uint_as_float(v[j4 * 4]) + b.x, __uint_as_float(v[j4 * 4 + 1]) + b.y);
                    o[j4 * 2 + 1] = tc::pack_bf16x2_relu(__uint_as_float(v[j4 * 4 + 2]) + b.z, __uint_as_float(v[j4 * 4 + 3]) + b.w);
                }
                tc::tmem_st_32x16(Q + k * 16, o);
            }
            tc::tmem_st_wait();
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive_cluster_tmem(x_remote[0]);
            // the stash must be free before E2 overwrites it: checked HERE, inside the wait for GEMM 2, not after it
            if (issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // previous TMA store has read the stash
            asm volatile("bar.sync %0, 256;" ::"r"(bar_id) : "memory");

            // ---- E2: f = relu(acc2 + sh2) -> bf16 -> TMEM P+128 (A of GEMM 3) and the shared-memory stash (gating)
            tc::mbar_wait_sleep(&ctl->acc_full[c][1], ph);
            tc::tc_fence_after();
#pragma unroll 1
            for (int k = h; k < 4; k += 2) {
                uint32_t v[32];
                tc::tmem_ld_32x32(P + k * 32, v);
                tc::tmem_ld_wait();
                uint32_t o[16];
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4) {
                    const float4 b = *reinterpret_cast<const float4*>(s_sh2 + k * 32 + j4 * 4);
                    o[j4 * 2] = tc::pack_bf16x2_relu(__uint_as_float(v[j4 * 4]) + b.x, __uint_as_float(v[j4 * 4 + 1]) + b.y);
                    o[j4 * 2 + 1] = tc::pack_bf16x2_relu(__uint_as_float(v[j4 * 4 + 2]) + b.z, __uint_as_float(v[j4 * 4 + 3]) + b.w);
                }
                tc::tmem_st_32x16(P + 128 + k * 16, o);
                uint8_t* rowp = stash + (k >> 1) * kSliceBytes + row * 128;
#pragma unroll
                for (int g4 = 0; g4 < 4; ++g4) {
                    const int piece = ((k & 1) * 4 + g4) ^ (row & 7);
                    *reinterpret_cast<uint4*>(rowp + piece * 16) = make_uint4(o[g4 * 4], o[g4 * 4 + 1], o[g4 * 4 + 2], o[g4 * 4 + 3]);
                }
            }
            tc::tmem_st_wait();
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive_cluster_tmem(x_remote[1]);

            // ---- E3: relu(acc3 + b3) -> bf16 -> TMEM P+160 (A of GEMM 4)
            tc::mbar_wait_sleep(&ctl->acc_full[c][2], ph);
            tc::tc_fence_after();
#pragma unroll 1
            for (int k = h; k < 2; k += 2) {
                uint32_t v[32];
                tc::tmem_ld_32x32(P + k * 32, v);
                tc::tmem_ld_wait();
                uint32_t o[16];
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4) {
                    const float4 b = *reinterpret_cast<const float4*>(s_sh3 + k * 32 + j4 * 4);
                    o[j4 * 2] = tc::pack_bf16x2_relu(__uint_as_float(v[j4 * 4]) + b.x, __uint_as_float(v[j4 * 4 + 1]) + b.y);
                    o[j4 * 2 + 1] = tc::pack_bf16x2_relu(__uint_as_float(v[j4 * 4 + 2]) + b.z, __uint_as_float(v[j4 * 4 + 3]) + b.w);
                }
                tc::tmem_st_32x16(P + 160 + k * 16, o);
            }
            tc::tmem_st_wait();
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive_cluster_tmem(x_remote[2]);

            // ---- E4: out = sigmoid(acc4 + b4) * f(stash) -> bf16 -> stash -> TMA store
            tc::mbar_wait_sleep(&ctl->acc_full[c][3], ph);
            tc::tc_fence_after();
            // both accumulator chunks go to registers first, so the chain's TMEM columns are released (and the stem
            // GEMM of its next tile starts) BEFORE the sigmoid / gating math, which is bound by the MUFU pipe
            uint32_t va[32], vb[32];
            tc::tmem_ld_32x32(P + h * 32, va);
            tc::tmem_ld_32x32(P + (h + 2) * 32, vb);
            tc::tmem_ld_wait();
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive_cluster_tmem(p_free_remote);
            auto gate = [&](const int k, const uint32_t (&v)[32]) {
                uint8_t* rowp = stash + (k >> 1) * kSliceBytes + row * 128;
#pragma unroll
                for (int g4 = 0; g4 < 4; ++g4) {
                    const int piece = ((k & 1) * 4 + g4) ^ (row & 7);
                    const uint4 fq = *reinterpret_cast<const uint4*>(rowp + piece * 16);
                    const uint32_t fw[4] = {fq.x, fq.y, fq.z, fq.w};
                    const float4 b0 = *reinterpret_cast<const float4*>(s_sh4 + k * 32 + g4 * 8);
                    const float4 b1 = *reinterpret_cast<const float4*>(s_sh4 + k * 32 + g4 * 8 + 4);
                    const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                    uint32_t w[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int j = g4 * 4 + e;                  // packed pair index: columns 2j, 2j+1
                        const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&fw[e]));
                        const float a = tc::fast_sigmoid(__uint_as_float(v[2 * j]) + bb[2 * e]);
                        const float b = tc::fast_sigmoid(__uint_as_float(v[2 * j + 1]) + bb[2 * e + 1]);
                        w[e] = tc::pack_bf16x2(a * f.x, b * f.y);
                    }
                    *reinterpret_cast<uint4*>(rowp + piece * 16) = make_uint4(w[0], w[1], w[2], w[3]);
                }
            };
            gate(h, va);
            gate(h + 2, vb);
            tc::fence_proxy_async();
            asm volatile("bar.sync %0, 256;" ::"r"(bar_id) : "memory");
            if (issuer) {
                for (int g2 = 0; g2 < 2; ++g2) {
                    if (EM) {   // tile rows 0..63 = even pixels, 64..127 = odd pixels: pixel-stride-2 maps
                        tc::tma_store_4d(&tmap_out, stash + g2 * kSliceBytes, g2 * 64, tx * 64, ty, img);
                        tc::tma_store_4d(&tmap_out1, stash + g2 * kSliceBytes + kSliceBytes / 2, g2 * 64, tx * 64, ty, img);
                    } else {
                        tc::tma_store_4d(&tmap_out, stash + g2 * kSliceBytes, g2 * 64, tx * p.BX, ty * p.BY, img);
                    }
                }
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
        }
        if (issuer) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }

    tc::tc_fence_before();
    tc::cluster_sync_all();
    if (warp == 2) {
        tc::tc_fence_after();
        tc::tmem_dealloc_2cta(tmem, 512);
    }
}

template <bool EM>
int launch_front(const CUtensorMap& m_r, const CUtensorMap& m_r1, const CUtensorMap& m_w1, const CUtensorMap& m_w2,
                 const CUtensorMap& m_w3, const CUtensorMap& m_w4, const CUtensorMap& m_out, const CUtensorMap& m_out1,
                 const FrontParams& p, cudaStream_t stream) {
    using Cfg = StemCfg<EM>;
    const int smem_bytes = 1024 + Cfg::kBlocks * Cfg::kW1Block + kWRest + Cfg::kStages * Cfg::kStageBytes + 2 * kStashBytes +
                           (int)sizeof(FrontCtl) + (192 + 128 + 64 + 128) * 4 + 64;
    RgbdDeviceInfo di;
    if (int rc = rgbd_device_info(&di)) return rc;
    const int num_sms = di.num_sms;
    RGBD_ONCE_PER_DEVICE(di.device, {
        RGBD_CHECK_CUDA(cudaFuncSetAttribute(ratio_front_kernel<EM>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    });
    const int n_units = (p.total_tiles + 1) / 2;
    int clusters = num_sms / 2;
    if (clusters > n_units) clusters = n_units;
    return launch_kernel(ratio_front_kernel<EM>, 2 * clusters, kThreads, smem_bytes, true, stream, m_r, m_r1, m_w1, m_w2, m_w3,
                         m_w4, m_out, m_out1, p);
}

}  // namespace

extern "C" int rgbd_ratio_front(const void* r_bf16, const void* w1_bf16, const void* w2_bf16, const void* w3_bf16,
                                const void* w4_bf16, const float* sh1, const float* sh2, const float* sh3, const float* sh4,
                                void* out_bf16, int B, int H, int W, int bx, int by, int compact_operand, rgbd_stream_t stream) {
    RGBD_CHECK_ARG(r_bf16 && w1_bf16 && w2_bf16 && w3_bf16 && w4_bf16 && sh1 && sh2 && sh3 && sh4 && out_bf16,
                   "ratio_front: null pointer");
    RGBD_CHECK_ARG(B >= 1 && H >= 1 && W >= 1, "ratio_front: bad geometry");
    RGBD_CHECK_ARG(bx >= 1 && by >= 1 && bx * by == kBlockM && bx <= 256 && by <= 256, "ratio_front: box must cover 128 pixels");
    if (compact_operand)
        RGBD_CHECK_ARG(bx == kBlockM && by == 1 && W % 2 == 0, "ratio_front: the compact operand needs a 128x1 box and an even width");
    const char* who = "ratio_front";
    const CUtensorMapSwizzle sw64 = CU_TENSOR_MAP_SWIZZLE_64B, sw128 = CU_TENSOR_MAP_SWIZZLE_128B;
    CUtensorMap m_r, m_r1, m_w1, m_w2, m_w3, m_w4, m_out, m_out1;
    // (n, k) weight matrices: boxes of 64 K elements x n/2 rows (one CTA's half)
    if (int rc = encode_bf16_map(&m_w2, who, w2_bf16, {192, 128}, {192 * 2}, {64, 64}, sw128)) return rc;
    if (int rc = encode_bf16_map(&m_w3, who, w3_bf16, {128, 64}, {128 * 2}, {64, 32}, sw128)) return rc;
    if (int rc = encode_bf16_map(&m_w4, who, w4_bf16, {64, 128}, {64 * 2}, {64, 64}, sw128)) return rc;
    if (compact_operand) {
        // pixel-pair views: dims (inner, pairs, rows, images) with a 2-pixel stride in dimension 1 (overlapping when the inner
        // extent exceeds it: the sliding window over x)
        const int Wp = rgbd_ratio_stem_compact_width(W);
        const long long row_bytes = (long long)Wp * 8, plane = (long long)(H + 6) * row_bytes;
        const uint8_t* e = reinterpret_cast<const uint8_t*>(r_bf16);
        if (int rc = encode_bf16_map(&m_r, who, e, {32, W / 2, H + 6, B}, {16, row_bytes, 2 * plane}, {32, 64, 1, 1}, sw64)) return rc;
        if (int rc = encode_bf16_map(&m_r1, who, e + plane, {32, W / 2, H + 6, B}, {16, row_bytes, 2 * plane}, {32, 64, 1, 1}, sw64))
            return rc;
        if (int rc = encode_bf16_map(&m_w1, who, w1_bf16, {224, 192}, {224 * 2}, {32, 96}, sw64)) return rc;   // 32-element K blocks
        uint8_t* o = reinterpret_cast<uint8_t*>(out_bf16);
        const long long o_row = (long long)W * 256, o_img = (long long)H * W * 256;
        if (int rc = encode_bf16_map(&m_out, who, o, {128, W / 2, H, B}, {512, o_row, o_img}, {64, 64, 1, 1}, sw128)) return rc;
        if (int rc = encode_bf16_map(&m_out1, who, o + 256, {128, W / 2, H, B}, {512, o_row, o_img}, {64, 64, 1, 1}, sw128)) return rc;
    } else {
        const long long r_row = 64 * 2 * (long long)W, o_row = 128 * 2 * (long long)W;
        if (int rc = encode_bf16_map(&m_r, who, r_bf16, {64, W, H + 6, B}, {64 * 2, r_row, r_row * (H + 6)}, {64, bx, by, 1}, sw128))
            return rc;
        if (int rc = encode_bf16_map(&m_out, who, out_bf16, {128, W, H, B}, {128 * 2, o_row, o_row * H}, {64, bx, by, 1}, sw128))
            return rc;
        if (int rc = encode_bf16_map(&m_w1, who, w1_bf16, {256, 192}, {256 * 2}, {64, 96}, sw128)) return rc;
        m_r1 = m_r;
        m_out1 = m_out;
    }
    FrontParams p;
    p.n_img = B; p.BX = bx; p.BY = by;
    p.tiles_x = ceil_div(W, bx);
    p.tiles_y = ceil_div(H, by);
    const long long total = (long long)B * p.tiles_x * p.tiles_y;
    RGBD_CHECK_ARG(total < (1ll << 30), "ratio_front: too many tiles");
    p.total_tiles = (int)total;
    p.sh1 = sh1; p.sh2 = sh2; p.sh3 = sh3; p.sh4 = sh4;
    return compact_operand ? launch_front<true>(m_r, m_r1, m_w1, m_w2, m_w3, m_w4, m_out, m_out1, p, (cudaStream_t)stream)
                           : launch_front<false>(m_r, m_r1, m_w1, m_w2, m_w3, m_w4, m_out, m_out1, p, (cudaStream_t)stream);
}
