// K4b: the point-wise middle of EnhancedDepthImageRatioPredictor.forward (reference
// mask2former/utils/custom_model.py:1466-1470) fused into ONE tcgen05 kernel per 128-pixel tile:
//     f  = ReLU(BN(Conv1x1_{192->128}(ms)))          feature_fusion      (CM:1466; BN scale folded into W2)
//     a  = sigmoid(Conv1x1_{64->128}(ReLU(Conv1x1_{128->64}(f))))   attention (CM:1469)
//     out = f * a                                                     (CM:1470)
// Three chained GEMMs per tile (K = 192, 128, 64).  The intermediate activations never leave the SM:
// the epilogue warps write them back into TENSOR MEMORY as packed bf16 (tcgen05.st) and the next GEMM
// reads its A operand straight from TMEM (tcgen05.mma with the A operand in tensor memory); all three weight matrices
// (80 KB) stay resident in shared memory; only the 192-channel input tile streams in through a TMA ring
// and the 128-channel result leaves through swizzled staging + TMA stores.  HBM traffic per pixel:
// 384 B in + 256 B out instead of the 1.4 KB of three separate layers.
//
// TMEM columns: acc2 [0,128) | f as bf16 [128,192) | acc3 [192,256) | relu(.) as bf16 [256,288) | acc4 [288,416).
#include "common.cuh"
#include "rgbd_b200.h"
#include "tc_ptx.cuh"
#include "tma_host.cuh"

namespace {

constexpr int kBlockM = 128;
constexpr int kThreads = 384;               // 4 control warps + 8 epilogue warps (two per TMEM lane quarter)
constexpr int kStages = 6;                 // 16 KB each: two tiles of three 64-channel slices
constexpr int kSliceBytes = kBlockM * 128; // 16 KB
constexpr int kW2Bytes = 3 * 128 * 128;    // 48 KB
constexpr int kW3Bytes = 2 * 64 * 128;     // 16 KB
constexpr int kW4Bytes = 1 * 128 * 128;    // 16 KB
constexpr int kStagingBytes = 2 * kSliceBytes;
constexpr uint32_t kColAcc2 = 0, kColX2 = 128, kColAcc3 = 192, kColX3 = 256, kColAcc4 = 288;

struct ChainParams {
    int n_img, tiles_x, tiles_y, BX, BY, total_tiles;
    const float* sh2;
    const float* sh3;
    const float* sh4;
};

struct alignas(16) ChainCtl {
    uint64_t full[kStages];
    uint64_t empty[kStages];
    uint64_t w_full;
    uint64_t acc2_full, acc3_full, acc4_full;
    uint64_t x2_ready, x3_ready;
    uint32_t tmem_base;
    uint32_t pad;
};

__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(acc)
        : "memory");
}

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}

__global__ void __launch_bounds__(kThreads, 1)
ratio_chain_kernel(const __grid_constant__ CUtensorMap tmap_x1, const __grid_constant__ CUtensorMap tmap_w2,
                   const __grid_constant__ CUtensorMap tmap_w3, const __grid_constant__ CUtensorMap tmap_w4,
                   const __grid_constant__ CUtensorMap tmap_out, const __grid_constant__ ChainParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* s_w2 = smem;
    uint8_t* s_w3 = s_w2 + kW2Bytes;
    uint8_t* s_w4 = s_w3 + kW3Bytes;
    uint8_t* s_ring = s_w4 + kW4Bytes;
    uint8_t* s_staging = s_ring + kStages * kSliceBytes;
    ChainCtl* ctl = reinterpret_cast<ChainCtl*>(s_staging + kStagingBytes);
    float* s_sh2 = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(ctl) + sizeof(ChainCtl));
    float* s_sh3 = s_sh2 + 128;
    float* s_sh4 = s_sh3 + 64;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < 128; i += blockDim.x) {
        s_sh2[i] = p.sh2[i];
        s_sh4[i] = p.sh4[i];
        if (i < 64) s_sh3[i] = p.sh3[i];
    }
    if (warp == 0 && lane == 0) {
        tc::prefetch_tmap(&tmap_x1);
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
        tc::mbar_init(&ctl->acc2_full, 1);
        tc::mbar_init(&ctl->acc3_full, 1);
        tc::mbar_init(&ctl->acc4_full, 1);
        tc::mbar_init(&ctl->x2_ready, 256);
        tc::mbar_init(&ctl->x3_ready, 256);
        tc::fence_barrier_init();
    }
    if (warp == 2) tc::tmem_alloc(&ctl->tmem_base, 512);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = ctl->tmem_base;

    const int per = p.total_tiles / gridDim.x, rem = p.total_tiles % gridDim.x;
    const int t_begin = blockIdx.x * per + min((int)blockIdx.x, rem);
    const int t_end = t_begin + per + ((int)blockIdx.x < rem ? 1 : 0);

    if (warp == 0 && lane == 0) {
        // ================= TMA producer =================
        tc::mbar_expect_tx(&ctl->w_full, kW2Bytes + kW3Bytes + kW4Bytes);
        for (int j = 0; j < 3; ++j) tc::tma_load_2d(s_w2 + j * (128 * 128), &tmap_w2, &ctl->w_full, j * 64, 0);
        for (int j = 0; j < 2; ++j) tc::tma_load_2d(s_w3 + j * (64 * 128), &tmap_w3, &ctl->w_full, j * 64, 0);
        tc::tma_load_2d(s_w4, &tmap_w4, &ctl->w_full, 0, 0);
        int stage = 0;
        uint32_t phase = 0;
        for (int t = t_begin; t < t_end; ++t) {
            int mt = t;
            const int tx = mt % p.tiles_x; mt /= p.tiles_x;
            const int ty = mt % p.tiles_y;
            const int img = mt / p.tiles_y;
            for (int j = 0; j < 3; ++j) {
                tc::mbar_wait(&ctl->empty[stage], phase ^ 1);
                tc::mbar_expect_tx(&ctl->full[stage], kSliceBytes);
                tc::tma_load_4d(s_ring + stage * kSliceBytes, &tmap_x1, &ctl->full[stage], j * 64, tx * p.BX, ty * p.BY, img);
                if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1 && lane == 0) {
        // ================= MMA issuer =================
        const uint32_t idesc128 = tc::make_idesc_bf16(kBlockM, 128);
        const uint32_t idesc64 = tc::make_idesc_bf16(kBlockM, 64);
        tc::mbar_wait(&ctl->w_full, 0);
        int stage = 0;
        uint32_t phase = 0, tphase = 0;
        for (int t = t_begin; t < t_end; ++t) {
            // GEMM 2: acc2 = X1 . W2^T   (A from the smem ring, 3 slices x 4 MMAs)
            for (int j = 0; j < 3; ++j) {
                tc::mbar_wait(&ctl->full[stage], phase);
                tc::tc_fence_after();
                const uint64_t adesc = tc::make_kmajor_desc(tc::smem_u32(s_ring + stage * kSliceBytes), 128);
                const uint64_t bdesc = tc::make_kmajor_desc(tc::smem_u32(s_w2 + j * (128 * 128)), 128);
                for (int k = 0; k < 4; ++k)
                    tc::umma_bf16(tmem + kColAcc2, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc128, (j | k) != 0);
                tc::umma_commit(&ctl->empty[stage]);
                if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
            tc::umma_commit(&ctl->acc2_full);
            // GEMM 3: acc3 = f(bf16, TMEM) . W3^T   (K = 128 -> 8 MMAs, A advances 8 columns per MMA)
            tc::mbar_wait(&ctl->x2_ready, tphase);
            tc::tc_fence_after();
            for (int k = 0; k < 8; ++k) {
                const uint64_t bdesc = tc::make_kmajor_desc(tc::smem_u32(s_w3 + (k >> 2) * (64 * 128)), 128) + (uint64_t)((k & 3) * 2);
                umma_bf16_ts(tmem + kColAcc3, tmem + kColX2 + (uint32_t)(k * 8), bdesc, idesc64, k != 0);
            }
            tc::umma_commit(&ctl->acc3_full);
            // GEMM 4: acc4 = relu(.)(bf16, TMEM) . W4^T   (K = 64 -> 4 MMAs)
            tc::mbar_wait(&ctl->x3_ready, tphase);
            tc::tc_fence_after();
            for (int k = 0; k < 4; ++k) {
                const uint64_t bdesc = tc::make_kmajor_desc(tc::smem_u32(s_w4), 128) + (uint64_t)(k * 2);
                umma_bf16_ts(tmem + kColAcc4, tmem + kColX3 + (uint32_t)(k * 8), bdesc, idesc128, k != 0);
            }
            tc::umma_commit(&ctl->acc4_full);
            tphase ^= 1;
        }
    } else if (warp >= 4) {
        // ================= epilogue =================
        const int q = warp & 3;
        const int half = (warp - 4) >> 2;           // chunks k = half, half+2 (E2, E4) / k = half (E3)
        const int row = q * 32 + lane;
        const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16);
        uint32_t tphase = 0;
        for (int t = t_begin; t < t_end; ++t) {
            int mt = t;
            const int tx = mt % p.tiles_x; mt /= p.tiles_x;
            const int ty = mt % p.tiles_y;
            const int img = mt / p.tiles_y;

            // ---- E2: f = relu(acc2*sc2 + sh2) -> bf16 -> TMEM
            tc::mbar_wait(&ctl->acc2_full, tphase);
            tc::tc_fence_after();
#pragma unroll 1
            for (int k = half; k < 4; k += 2) {
                uint32_t v[32];
                tc::tmem_ld_32x32(lane_base + kColAcc2 + k * 32, v);
                tc::tmem_ld_wait();
                uint32_t o[16];
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4) {
                    const float4 b = *reinterpret_cast<const float4*>(s_sh2 + k * 32 + j4 * 4);
                    o[j4 * 2] = tc::pack_bf16x2_relu(__uint_as_float(v[j4 * 4]) + b.x, __uint_as_float(v[j4 * 4 + 1]) + b.y);
                    o[j4 * 2 + 1] = tc::pack_bf16x2_relu(__uint_as_float(v[j4 * 4 + 2]) + b.z, __uint_as_float(v[j4 * 4 + 3]) + b.w);
                }
                tc::tmem_st_32x16(lane_base + kColX2 + k * 16, o);
            }
            tc::tmem_st_wait();
            tc::tc_fence_before();
            tc::mbar_arrive(&ctl->x2_ready);

            // ---- E3: relu(acc3 + b3) -> bf16 -> TMEM
            tc::mbar_wait(&ctl->acc3_full, tphase);
            tc::tc_fence_after();
            {
                const int k = half;
                uint32_t v[32];
                tc::tmem_ld_32x32(lane_base + kColAcc3 + k * 32, v);
                tc::tmem_ld_wait();
                uint32_t o[16];
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4) {
                    const float4 b = *reinterpret_cast<const float4*>(s_sh3 + k * 32 + j4 * 4);
                    o[j4 * 2] = tc::pack_bf16x2_relu(__uint_as_float(v[j4 * 4]) + b.x, __uint_as_float(v[j4 * 4 + 1]) + b.y);
                    o[j4 * 2 + 1] = tc::pack_bf16x2_relu(__uint_as_float(v[j4 * 4 + 2]) + b.z, __uint_as_float(v[j4 * 4 + 3]) + b.w);
                }
                tc::tmem_st_32x16(lane_base + kColX3 + k * 16, o);
            }
            tc::tmem_st_wait();
            tc::tc_fence_before();
            tc::mbar_arrive(&ctl->x3_ready);

            // ---- E4: out = sigmoid(acc4 + b4) * f -> bf16 -> swizzled staging -> TMA store
            tc::mbar_wait(&ctl->acc4_full, tphase);
            tc::tc_fence_after();
            if (warp == 4 && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            asm volatile("bar.sync 1, 256;" ::: "memory");
#pragma unroll 1
            for (int k = half; k < 4; k += 2) {
                uint32_t v[32], g[16];
                tc::tmem_ld_32x32(lane_base + kColAcc4 + k * 32, v);
                tc::tmem_ld_32x16(lane_base + kColX2 + k * 16, g);
                tc::tmem_ld_wait();
                uint8_t* rowp = s_staging + (k >> 1) * kSliceBytes + row * 128;
#pragma unroll
                for (int g4 = 0; g4 < 4; ++g4) {
                    uint32_t w[4];
                    const float4 b0 = *reinterpret_cast<const float4*>(s_sh4 + k * 32 + g4 * 8);
                    const float4 b1 = *reinterpret_cast<const float4*>(s_sh4 + k * 32 + g4 * 8 + 4);
                    const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int j = g4 * 4 + e;                  // packed pair index: columns 2j, 2j+1
                        const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&g[j]));
                        const float a = tc::fast_sigmoid(__uint_as_float(v[2 * j]) + bb[2 * e]);
                        const float b = tc::fast_sigmoid(__uint_as_float(v[2 * j + 1]) + bb[2 * e + 1]);
                        w[e] = tc::pack_bf16x2(a * f.x, b * f.y);
                    }
                    const int piece = ((k & 1) * 4 + g4) ^ (row & 7);
                    *reinterpret_cast<uint4*>(rowp + piece * 16) = make_uint4(w[0], w[1], w[2], w[3]);
                }
            }
            tc::tc_fence_before();
            tc::fence_proxy_async();
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if (warp == 4 && lane == 0) {
                for (int g2 = 0; g2 < 2; ++g2)
                    tc::tma_store_4d(&tmap_out, s_staging + g2 * kSliceBytes, g2 * 64, tx * p.BX, ty * p.BY, img);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
            tphase ^= 1;
        }
        if (warp == 4 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }

    tc::tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem, 512);
    }
}

}  // namespace

extern "C" int rgbd_ratio_chain(const void* x1_bf16, const void* w2_bf16, const void* w3_bf16, const void* w4_bf16,
                                const float* sh2, const float* sh3, const float* sh4, void* out_bf16,
                                int B, int H, int W, int bx, int by, rgbd_stream_t stream) {
    RGBD_CHECK_ARG(x1_bf16 && w2_bf16 && w3_bf16 && w4_bf16 && sh2 && sh3 && sh4 && out_bf16, "ratio_chain: null pointer");
    RGBD_CHECK_ARG(B >= 1 && H >= 1 && W >= 1, "ratio_chain: bad geometry");
    RGBD_CHECK_ARG(bx >= 1 && by >= 1 && bx * by == kBlockM && bx <= 256 && by <= 256, "ratio_chain: box must cover 128 pixels");
    const char* who = "ratio_chain";
    const CUtensorMapSwizzle sw128 = CU_TENSOR_MAP_SWIZZLE_128B;
    const long long x1_row = 192 * 2 * (long long)W, o_row = 128 * 2 * (long long)W;
    CUtensorMap m_x1, m_w2, m_w3, m_w4, m_out;
    if (int rc = encode_bf16_map(&m_x1, who, x1_bf16, {192, W, H, B}, {192 * 2, x1_row, x1_row * H}, {64, bx, by, 1}, sw128)) return rc;
    if (int rc = encode_bf16_map(&m_out, who, out_bf16, {128, W, H, B}, {128 * 2, o_row, o_row * H}, {64, bx, by, 1}, sw128)) return rc;
    // (n, k) weight matrices, one box of 64 K elements x all n rows
    if (int rc = encode_bf16_map(&m_w2, who, w2_bf16, {192, 128}, {192 * 2}, {64, 128}, sw128)) return rc;
    if (int rc = encode_bf16_map(&m_w3, who, w3_bf16, {128, 64}, {128 * 2}, {64, 64}, sw128)) return rc;
    if (int rc = encode_bf16_map(&m_w4, who, w4_bf16, {64, 128}, {64 * 2}, {64, 128}, sw128)) return rc;
    ChainParams p;
    p.n_img = B; p.BX = bx; p.BY = by;
    p.tiles_x = ceil_div(W, bx);
    p.tiles_y = ceil_div(H, by);
    const long long total = (long long)B * p.tiles_x * p.tiles_y;
    RGBD_CHECK_ARG(total < (1ll << 31), "ratio_chain: too many tiles");
    p.total_tiles = (int)total;
    p.sh2 = sh2; p.sh3 = sh3; p.sh4 = sh4;
    const int smem_bytes = 1024 + kW2Bytes + kW3Bytes + kW4Bytes + kStages * kSliceBytes + kStagingBytes +
                           (int)sizeof(ChainCtl) + (128 + 128 + 64 + 128) * 4 + 64;
    RgbdDeviceInfo di;
    if (int rc = rgbd_device_info(&di)) return rc;
    const int num_sms = di.num_sms;
    RGBD_ONCE_PER_DEVICE(di.device, {
        RGBD_CHECK_CUDA(cudaFuncSetAttribute(ratio_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    });
    const int grid = p.total_tiles < num_sms ? p.total_tiles : num_sms;
    ratio_chain_kernel<<<grid, kThreads, smem_bytes, (cudaStream_t)stream>>>(m_x1, m_w2, m_w3, m_w4, m_out, p);
    RGBD_CHECK_LAUNCH();
    return RGBD_OK;
}
