// K3b: backward of a DSAM stage (autograd of reference mask2former/utils/custom_model.py:683-696; SURVEY H11).
//   Out = sum_t Conv_t(p_t * F) + Proj(F) (+ bias, + residual)          3x3 stride 2 pad 1 (or 1x1 stride 1)
//   dW_t[n,c,dy,dx] = sum_{b,oy,ox} G[b,n,oy,ox] * (p_t*F)[b,c,2oy+dy-1,2ox+dx-1]        (wgrad, this file)
//   db_t[n]         = sum_{b : region t used} sum_{oy,ox} G[b,n,oy,ox]                    (this file)
//   dF              = sum_t p_t * ConvT_t(G) + ProjT(G)   -> conv_gemm.cu, epilogue mode 3 (masked segment sum)
//
// wgrad is a GEMM whose reduction dimension is the OUTPUT PIXELS: M = C_out rows of G^T, N = C_in rows of the
// masked input, K = B*Ho*Wo.  Both operands are staged pixel-contiguous (bf16, "NCHW") with the SAME row pitch, so
// a K block is 64 consecutive flattened pixels (one 128-byte swizzled TMA row per channel); a filter tap is a
// constant shift of the flattened index inside the tap's parity plane (rows: -pitch; columns: a pre-shifted copy
// of the plane, because TMA needs a 16-byte aligned innermost start) and out-of-range pixels are zero-filled
// (= conv padding; the pitch padding of G is zero, so pad columns never contribute).  One CTA tile = (segment, tap, 128 output channels, BLOCK_N input
// channels, image range); tcgen05.mma accumulates in TMEM over the whole K loop; the epilogue adds the fp32 tile
// into dW with red.global (split-K over images keeps all SMs busy).
#include "common.cuh"
#include "rgbd_b200.h"
#include "tc_ptx.cuh"
#include "tma_host.cuh"
#include <stdlib.h>

namespace {

constexpr int kBlockM = 128;
constexpr int kThreads = 224;          // warp 0 TMA, warp 1 MMA, warp 2 TMEM alloc/dealloc (never diverges), warps 3-6 epilogue
constexpr int kMaxStagesW = 8;

struct WgradParams {
    int B, Ho, Wo, Wp, k_blocks;
    int n_seg, n_par, taps;
    int m_tiles, n_tiles, BLOCK_N, ksplit;
    int N_out, Cp, stages;
    int taps_tbl[9][2];                // (plane, flattened pixel offset) per tap
    float* dw;                         // [N_out][n_seg][taps][Cp]
    int total_tiles;
};

struct alignas(16) WCtl {
    uint64_t full[kMaxStagesW];
    uint64_t empty[kMaxStagesW];
    uint64_t acc_full;
    uint64_t acc_empty;
    uint32_t tmem_base;
    uint32_t pad[3];
};

__device__ __forceinline__ void decode_wtile(const WgradParams& p, int t, int& ks, int& seg, int& tap, int& mt, int& nt) {
    nt = t % p.n_tiles; t /= p.n_tiles;
    mt = t % p.m_tiles; t /= p.m_tiles;
    tap = t % p.taps; t /= p.taps;
    seg = t % p.n_seg;
    ks = t / p.n_seg;
}

__global__ void __launch_bounds__(kThreads, 1)
dsam_wgrad_kernel(const __grid_constant__ CUtensorMap tmap_g, const __grid_constant__ CUtensorMap tmap_x,
                  const __grid_constant__ WgradParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    const int a_bytes = kBlockM * 128, b_bytes = p.BLOCK_N * 128, stage_bytes = a_bytes + b_bytes;
    WCtl* ctl = reinterpret_cast<WCtl*>(smem + (size_t)p.stages * stage_bytes);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        tc::prefetch_tmap(&tmap_g);
        tc::prefetch_tmap(&tmap_x);
        for (int s = 0; s < p.stages; ++s) {
            tc::mbar_init(&ctl->full[s], 1);
            tc::mbar_init(&ctl->empty[s], 1);
        }
        tc::mbar_init(&ctl->acc_full, 1);
        tc::mbar_init(&ctl->acc_empty, 128);
        tc::fence_barrier_init();
    }
    if (warp == 2) tc::tmem_alloc(&ctl->tmem_base, 256);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = ctl->tmem_base;

    if (warp == 0 && lane == 0) {
        int stage = 0;
        uint32_t phase = 0;
        for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x) {
            int ks, seg, tap, mt, nt;
            decode_wtile(p, t, ks, seg, tap, mt, nt);
            const int b0 = (int)(((long long)p.B * ks) / p.ksplit), b1 = (int)(((long long)p.B * (ks + 1)) / p.ksplit);
            const int par = p.taps_tbl[tap][0], off = p.taps_tbl[tap][1];
            for (int b = b0; b < b1; ++b) {
                const int plane = (b * p.n_seg + seg) * p.n_par + par;
                for (int kb = 0; kb < p.k_blocks; ++kb) {
                    tc::mbar_wait(&ctl->empty[stage], phase ^ 1);
                    uint8_t* sa = smem + (size_t)stage * stage_bytes;
                    tc::mbar_expect_tx(&ctl->full[stage], (uint32_t)stage_bytes);
                    tc::tma_load_3d(sa, &tmap_g, &ctl->full[stage], kb * 64, mt * kBlockM, b);
                    tc::tma_load_3d(sa + a_bytes, &tmap_x, &ctl->full[stage], kb * 64 + off, nt * p.BLOCK_N, plane);
                    if (++stage == p.stages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // whole warp in uniform control flow, one elected lane issues (descriptors stay in uniform registers)
        const uint32_t idesc = tc::make_idesc_bf16(kBlockM, p.BLOCK_N);
        int stage = 0;
        uint32_t phase = 0, aphase = 0;
        for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x) {
            int ks, seg, tap, mt, nt;
            decode_wtile(p, t, ks, seg, tap, mt, nt);
            const int b0 = (int)(((long long)p.B * ks) / p.ksplit), b1 = (int)(((long long)p.B * (ks + 1)) / p.ksplit);
            const int n_kblocks = (b1 - b0) * p.k_blocks;
            tc::mbar_wait(&ctl->acc_empty, aphase ^ 1);
            tc::tc_fence_after();
            for (int j = 0; j < n_kblocks; ++j) {
                tc::mbar_wait(&ctl->full[stage], phase);
                tc::tc_fence_after();
                const uint32_t sa = tc::smem_u32(smem + (size_t)stage * stage_bytes);
                const uint64_t adesc = tc::make_kmajor_desc(sa, 128), bdesc = tc::make_kmajor_desc(sa + a_bytes, 128);
                if (tc::elect_one()) {
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        tc::umma_bf16(tmem, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (j | k) != 0);
                    tc::umma_commit(&ctl->empty[stage]);
                }
                __syncwarp();
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
            if (tc::elect_one()) tc::umma_commit(&ctl->acc_full);
            __syncwarp();
            aphase ^= 1;
        }
    } else if (warp >= 3) {
        const int q = warp & 3;                    // TMEM lane quarter of this warp
        const int row = q * 32 + lane;
        uint32_t aphase = 0;
        for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x) {
            int ks, seg, tap, mt, nt;
            decode_wtile(p, t, ks, seg, tap, mt, nt);
            const int b0 = (int)(((long long)p.B * ks) / p.ksplit), b1 = (int)(((long long)p.B * (ks + 1)) / p.ksplit);
            tc::mbar_wait(&ctl->acc_full, aphase);
            tc::tc_fence_after();
            const int n = mt * kBlockM + row;
            for (int k = 0; k < (p.BLOCK_N >> 5); ++k) {
                uint32_t v[32];
                tc::tmem_ld_32x32(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(k * 32), v);
                tc::tmem_ld_wait();
                if (n < p.N_out && b1 > b0) {
                    float* dst = p.dw + (((size_t)n * p.n_seg + seg) * p.taps + tap) * p.Cp + nt * p.BLOCK_N + k * 32;
#pragma unroll
                    for (int j = 0; j < 32; ++j) atomicAdd(dst + j, __uint_as_float(v[j]));
                }
            }
            tc::tc_fence_before();
            tc::mbar_arrive(&ctl->acc_empty);
            aphase ^= 1;
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        __syncwarp();
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem, 256);
    }
}

// ---- operand staging ---------------------------------------------------------------------------------------
// G (B,N,Ho,Wo) fp32 -> bf16 with the row pitch padded to a multiple of 8 pixels (TMA strides are 16-byte units)
__global__ void __launch_bounds__(256) cast_pitched_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst,
                                                           long long rows, int W, int Wp) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = rows * Wp;
    if (i >= total) return;
    const long long r = i / Wp;
    const int x = (int)(i - r * Wp);
    dst[i] = __float2bfloat16(x < W ? src[r * W + x] : 0.f);
}

// masked, parity-split, pixel-contiguous input: out[b][seg][par][c][y2][x2 (pitch W2p)] = bf16(F[b][c][y][x] * bit(code,seg)).
// TMA needs the innermost (x) start coordinate 16-byte aligned, so the x-1 tap cannot be a box shifted by one pixel:
// planes 4 and 5 are copies of the px=1 planes (py=0 / py=1) shifted right by one pixel (x2 -> x2+1).
__global__ void __launch_bounds__(256) dsam_pack_t_kernel(const float* __restrict__ feat, const uint8_t* __restrict__ codes,
                                                          __nv_bfloat16* __restrict__ out, int C, int Cp, int H, int W,
                                                          int H2, int W2p, int n_seg, int masked_segs, int split) {
    const int b = blockIdx.z, c = blockIdx.y;
    const int n_par = split ? 6 : 1;
    const size_t plane = (size_t)H * W;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < H * W; i += gridDim.x * blockDim.x) {
        const int y = i / W, x = i - y * W;
        const float v = feat[((size_t)b * C + c) * plane + i];
        const unsigned code = codes[(size_t)b * plane + i];
        const int par = split ? ((y & 1) * 2 + (x & 1)) : 0;
        const int yy = split ? (y >> 1) : y, xx = split ? (x >> 1) : x;
        for (int s = 0; s < n_seg; ++s) {
            const bool keep = s >= masked_segs || ((code >> s) & 1u);
            const __nv_bfloat16 h = __float2bfloat16(keep ? v : 0.f);
            const size_t pl = ((size_t)b * n_seg + s) * n_par;
            out[(((pl + par) * Cp + c) * H2 + yy) * W2p + xx] = h;
            if (split && (x & 1) && xx + 1 < W2p)
                out[(((pl + 4 + (y & 1)) * Cp + c) * H2 + yy) * W2p + xx + 1] = h;
        }
    }
}

// db_t[n] += sum_{oy,ox} G[b,n,:,:] for every region t the image uses (t < variant[b])
__global__ void __launch_bounds__(256) dsam_dbias_kernel(const float* __restrict__ g, const int* __restrict__ variant,
                                                         float* __restrict__ db, int N, int HW, int n_bias) {
    const int b = blockIdx.y, n = blockIdx.x;
    const float* src = g + ((size_t)b * N + n) * HW;
    float s = 0.f;
    for (int i = threadIdx.x; i < HW; i += blockDim.x) s += src[i];
    __shared__ float red[8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float tot = 0.f;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += red[w];
        const int nb = variant ? variant[b] : n_bias;
        for (int t = 0; t < n_bias && t < nb; ++t) atomicAdd(db + (size_t)t * N + n, tot);
    }
}

}  // namespace

extern "C" int rgbd_cast_bf16_pitched(const float* src, void* dst_bf16, long long rows, int W, int W_pitch,
                                      rgbd_stream_t stream) {
    RGBD_CHECK_ARG(src && dst_bf16 && rows >= 1 && W >= 1 && W_pitch >= W && W_pitch % 8 == 0, "cast_bf16_pitched: bad arguments");
    const long long total = rows * W_pitch;
    cast_pitched_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(src, (__nv_bfloat16*)dst_bf16, rows, W,
                                                                                         W_pitch);
    RGBD_CHECK_LAUNCH();
    return RGBD_OK;
}

extern "C" int rgbd_dsam_pack_t(const float* feat, const uint8_t* codes, void* out_bf16, int B, int C, int C_pad, int H, int W,
                                int W2_pitch, int n_seg, int masked_segs, int parity_split, rgbd_stream_t stream) {
    RGBD_CHECK_ARG(feat && codes && out_bf16, "dsam_pack_t: null pointer");
    RGBD_CHECK_ARG(B >= 1 && C >= 1 && C_pad >= C && H >= 1 && W >= 1 && W2_pitch % 8 == 0, "dsam_pack_t: bad geometry");
    const int H2 = parity_split ? (H + 1) / 2 : H;
    RGBD_CHECK_ARG(W2_pitch >= (parity_split ? (W + 1) / 2 : W), "dsam_pack_t: pitch too small");
    dim3 grid(min(ceil_div(H * W, 256), 64), C, B);
    dsam_pack_t_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(feat, codes, (__nv_bfloat16*)out_bf16, C, C_pad, H, W, H2,
                                                              W2_pitch, n_seg, masked_segs, parity_split ? 1 : 0);
    RGBD_CHECK_LAUNCH();
    return RGBD_OK;
}

extern "C" int rgbd_dsam_dbias(const float* g, const int* variant, float* db, int B, int N, int HW, int n_bias,
                               rgbd_stream_t stream) {
    RGBD_CHECK_ARG(g && db && B >= 1 && N >= 1 && HW >= 1 && n_bias >= 1, "dsam_dbias: bad arguments");
    RGBD_CHECK_CUDA(cudaMemsetAsync(db, 0, sizeof(float) * (size_t)n_bias * N, (cudaStream_t)stream));
    dsam_dbias_kernel<<<dim3(N, B), 256, 0, (cudaStream_t)stream>>>(g, variant, db, N, HW, n_bias);
    RGBD_CHECK_LAUNCH();
    return RGBD_OK;
}

extern "C" int rgbd_dsam_wgrad(const void* g_bf16, int g_w_pitch, const void* xt_bf16, int x_w_pitch, int x_h, float* dw,
                               int B, int N_out, int C_pad, int Ho, int Wo, int n_seg, int parity_split,
                               rgbd_stream_t stream) {
    RGBD_CHECK_ARG(g_bf16 && xt_bf16 && dw, "dsam_wgrad: null pointer");
    RGBD_CHECK_ARG(B >= 1 && N_out >= 1 && C_pad >= 32 && C_pad % 32 == 0 && Ho >= 1 && Wo >= 1 && n_seg >= 1 && n_seg <= 8,
                   "dsam_wgrad: bad geometry");
    RGBD_CHECK_ARG(g_w_pitch % 8 == 0 && x_w_pitch % 8 == 0 && g_w_pitch >= Wo, "dsam_wgrad: row pitches must be multiples of 8");
    WgradParams p;
    p.B = B; p.Ho = Ho; p.Wo = Wo; p.N_out = N_out; p.Cp = C_pad;
    p.n_seg = n_seg;
    p.n_par = parity_split ? 6 : 1;
    p.taps = parity_split ? 9 : 1;
    RGBD_CHECK_ARG(g_w_pitch == x_w_pitch && x_h >= Ho, "dsam_wgrad: G and X^T must share the row pitch (got %d / %d)", g_w_pitch,
                   x_w_pitch);
    p.Wp = g_w_pitch;
    p.k_blocks = ceil_div(Ho * p.Wp, 64);
    for (int tap = 0; tap < p.taps; ++tap) {
        int par = 0, off = 0;
        if (parity_split) {
            const int dy = tap / 3, dx = tap % 3;           // input row 2*oy+dy-1: dy=0 -> odd plane, row oy-1; 1 -> even, oy; 2 -> odd, oy
            const int py = dy == 1 ? 0 : 1, px = dx == 1 ? 0 : 1;
            par = dx == 0 ? 4 + py : py * 2 + px;           // dx == 0 reads pixel x2-1: the right-shifted copy of the px=1 plane
            off = dy == 0 ? -p.Wp : 0;
        }
        p.taps_tbl[tap][0] = par; p.taps_tbl[tap][1] = off;
    }
    p.BLOCK_N = C_pad <= 256 ? C_pad : 0;
    if (!p.BLOCK_N)
        for (int bn = 256; bn >= 32; bn -= 32)
            if (C_pad % bn == 0) { p.BLOCK_N = bn; break; }
    p.n_tiles = C_pad / p.BLOCK_N;
    p.m_tiles = ceil_div(N_out, kBlockM);
    RgbdDeviceInfo di;
    if (int rc = rgbd_device_info(&di)) return rc;
    const int num_sms = di.num_sms, max_smem = di.max_smem;
    RGBD_ONCE_PER_DEVICE(di.device, {
        RGBD_CHECK_CUDA(cudaFuncSetAttribute(dsam_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
    });
    const int base_tiles = p.n_seg * p.taps * p.m_tiles * p.n_tiles;
    int ksplit = 1;
    while (ksplit * 2 <= B && base_tiles * ksplit < 2 * num_sms) ksplit *= 2;
    p.ksplit = ksplit;
    p.total_tiles = base_tiles * ksplit;
    p.dw = dw;
    const int stage_bytes = kBlockM * 128 + p.BLOCK_N * 128;
    int stages = (max_smem - 2048 - (int)sizeof(WCtl)) / stage_bytes;
    if (stages > kMaxStagesW) stages = kMaxStagesW;
    RGBD_CHECK_ARG(stages >= 2, "dsam_wgrad: not enough shared memory");
    p.stages = stages;
    // channel-major operands: (pixels, channels, planes), pixels innermost
    CUtensorMap m_g, m_x;
    const long long g_pix = (long long)Ho * g_w_pitch, x_pix = (long long)x_h * x_w_pitch;
    if (int rc = encode_bf16_map(&m_g, "dsam_wgrad", g_bf16, {g_pix, N_out, B}, {g_pix * 2, g_pix * 2 * N_out}, {64, kBlockM, 1},
                                 CU_TENSOR_MAP_SWIZZLE_128B))
        return rc;
    if (int rc = encode_bf16_map(&m_x, "dsam_wgrad", xt_bf16, {x_pix, C_pad, B * n_seg * p.n_par},
                                 {x_pix * 2, x_pix * 2 * C_pad}, {64, p.BLOCK_N, 1}, CU_TENSOR_MAP_SWIZZLE_128B))
        return rc;
    RGBD_CHECK_CUDA(cudaMemsetAsync(dw, 0, sizeof(float) * (size_t)N_out * n_seg * p.taps * C_pad, (cudaStream_t)stream));
    int smem_bytes = 1024 + stages * stage_bytes + (int)sizeof(WCtl) + 64;
    if (smem_bytes < 120 * 1024) smem_bytes = 120 * 1024;     // one CTA per SM (TMEM allocation)
    const int grid = p.total_tiles < num_sms ? p.total_tiles : num_sms;
    dsam_wgrad_kernel<<<grid, kThreads, smem_bytes, (cudaStream_t)stream>>>(m_g, m_x, p);
    RGBD_CHECK_LAUNCH();
    return RGBD_OK;
}
