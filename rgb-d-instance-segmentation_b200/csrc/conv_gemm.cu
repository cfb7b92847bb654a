// K3/K4 core: implicit-GEMM convolution on the 5th-generation tensor cores (tcgen05 + TMEM + TMA).
//
// One persistent, warp-specialised kernel serves every dense contraction on the E-DSAM path:
//   * DSAModule.forward (reference mask2former/utils/custom_model.py:683-696): the five 3x3 stride-2
//     convolutions of a stage are ONE GEMM with K = 45*C_in over the K-concatenated operand
//     [p0*F | p1*F | p2*F | p3*F | F] (SURVEY.md section 8a row 9);
//   * EnhancedDepthImageRatioPredictor.forward (CM:1458-1473): the multi-scale 3x3/5x5/7x7 stem (as one
//     7x7 conv over a row-im2col tensor), the 1x1 fusion / attention convs and the 3x3 128->256 conv.
//
// A operand: a bf16 channels-last activation tensor addressed as a 4-D TMA tensor (c, x, y, plane).
// A "K slice" is 64 (or 32) channels of one filter tap: (c0, dx, dy, dplane) offsets added to the tile's
// base coordinate; out-of-bounds rows are zero-filled by TMA (= conv zero padding).  B operand: packed
// bf16 weights [N][K] (K-major), K ordered like the slice table.  D: fp32 accumulators in TMEM,
// 128 pixels x BLOCK_N channels, double buffered so the epilogue of tile i overlaps the MMAs of i+1.
//
// Warp roles (384 threads): warp 0 = TMA producer, warp 1 = MMA issuer (one thread), warp 2 = TMEM
// allocator, warps 4-11 = epilogue, two per TMEM lane quarter (TMEM -> registers -> fused scale/shift/activation -> global).
// Epilogues: (0) bf16 channels-last store with optional gating multiply, (1) fp32 NCHW store with
// optional residual add, (2) adaptive-average-pool accumulation (the 256-channel map of the ratio
// predictor is never written: CM:1412-1416 BN/ReLU/AdaptiveAvgPool2d(4) are fused here).
#include "common.cuh"
#include "rgbd_b200.h"
#include "tc_ptx.cuh"
#include "tma_host.cuh"

namespace {

constexpr int kBlockM = 128;
constexpr int kMaxStages = 12;
constexpr int kMaxSlices = 1024;
constexpr int kThreads = 384;        // 4 control warps + 8 epilogue warps
constexpr int kEpiThreads = 256;
constexpr int kEpiWarps = kEpiThreads / 32;   // arrivals per CTA on tmem_empty: one per epilogue warp
constexpr int kTmemCols = 512;
constexpr int kAccStages = 2;        // accumulator buffers in tensor memory: the epilogue of tile t overlaps the MMAs of tile t+1

struct KParams {
    int n_img, tiles_x, tiles_y, BX, BY, out_w, out_h;
    int n_slices, kb_bytes, stages;
    int N, N_pad, BLOCK_N, n_tiles_n;
    int plane_per_img, tile_order;
    const int4* slices;
    int epi_mode, act;
    const float* scale;
    const float* shift;
    const int* variant;
    const __nv_bfloat16* gate;
    void* out;
    const float* residual;
    long long* pool;          // fixed-point (1/RGBD_POOL_FIXED_ONE) cell sums: order-independent integer atomics
    long long* pool_sq;       // act 3 (statistics pass of a train-mode BatchNorm): cell sums of the SQUARED values
    int cells_y, cells_x;
    int total_tiles;
    int staging_bytes;    // epi_mode 0: swizzled bf16 output tile staged for TMA stores
    int gate_bytes;       // epi_mode 0 with gate: TMA-loaded gate tile (same layout)
    int b_resident;       // whole weight matrix stays in shared memory (single N tile); the ring carries A only
    int b_res_bytes;
    const uint8_t* codes;     // epilogue mode 3: region codes at the resolution of dX
    int in_h, in_w, m3_py, m3_px, m3_stride, m3_masked_segs, m3_n_seg;
    int dsam_taps;            // dsam_fwd_kernel: 9 (3x3 stride 2 on parity planes)
    // epilogue mode 1: also emit the result as the NEXT DSAM stage's bf16 parity-split operand (what rgbd_dsam_pack would
    // build from the fp32 output), so the cascade needs no pack kernel between its stages
    __nv_bfloat16* next_op;
    const uint8_t* next_codes;
    int next_c_pad, next_n_seg, next_masked_segs;
    int c_blocks, sa_stages, a_stage_bytes;   // conv3x3_kernel: 64-channel blocks, A-ring depth, bytes per A stage
};

struct alignas(16) SmemCtl {
    uint64_t full[kMaxStages];
    uint64_t empty[kMaxStages];
    uint64_t tmem_full[kAccStages];
    uint64_t tmem_empty[kAccStages];
    uint64_t gate_full;
    uint64_t gate_empty;
    uint64_t b_full;
    uint64_t a_full[4];       // conv3x3_kernel: separate ring for the (128+2)-pixel A tiles
    uint64_t a_empty[4];
    uint64_t masked_full[2];  // dsam_fwd_kernel: the masked copies of an A group are written (both CTAs of the pair)
    uint64_t masked_empty[2]; // ... and consumed by the pair's MMAs
    uint32_t tmem_base;
    uint32_t pad[3];
};

__device__ __forceinline__ void decode_tile(const KParams& p, int t, int& img, int& ty, int& tx, int& nt) {
    nt = t % p.n_tiles_n;
    int mt = t / p.n_tiles_n;
    if (p.tile_order == 0) {
        tx = mt % p.tiles_x; mt /= p.tiles_x;
        ty = mt % p.tiles_y;
        img = mt / p.tiles_y;
    } else {
        ty = mt % p.tiles_y; mt /= p.tiles_y;
        tx = mt % p.tiles_x;
        img = mt / p.tiles_x;
    }
}

struct EpiCtx {
    uint8_t* s_staging;
    uint8_t* s_gate;
    SmemCtl* ctl;
    float* s_scale;
    float* s_shift;
    uint32_t tmem_base;
    int t_begin, t_end, warp, lane;   // work units [t_begin, t_end): tiles, or tile PAIRS when pair_rank >= 0
    int pair_rank;                    // -1: one CTA per tile; 0/1: rank of this CTA in a CTA pair (see pair_tile)
    uint32_t tmem_empty_remote[kAccStages];   // shared::cluster addresses of the leader's tmem_empty barriers (0: arrive locally)
};

// Slot and mbarrier phase of a ring of buffers; the phase flips each time the slot wraps to 0.
struct Ring {
    int i = 0;
    uint32_t ph = 0;
    __device__ __forceinline__ void next(int n) {
        if (++i == n) { i = 0; ph ^= 1; }
    }
};

// tile of CTA `rank` in pair unit u: the two CTAs take adjacent M tiles of the SAME N tile (they share the B operand)
__device__ __forceinline__ int pair_tile(const KParams& p, int u, int rank) {
    return (2 * (u / p.n_tiles_n) + rank) * p.n_tiles_n + (u % p.n_tiles_n);
}

__device__ __forceinline__ void pool_add(long long* dst, float v) {
    atomicAdd(reinterpret_cast<unsigned long long*>(dst), (unsigned long long)__double2ll_rn((double)v * RGBD_POOL_FIXED_ONE));
}

// ACT 3 = "statistics": identity here; the pooled epilogue additionally accumulates the squares into pool_sq
template <int ACT>
__device__ __forceinline__ float act_fn(float x) {
    if (ACT == 1) return fmaxf(x, 0.f);
    if (ACT == 2) return tc::fast_sigmoid(x);
    return x;
}

// Epilogue warps 4..11: TMEM -> registers -> y = act(acc*scale + shift) -> mode-specific output.
// MODE and ACT are compile-time so the per-element code is branch-free and the loads are batched.
template <int MODE, int ACT, bool SCALE>
__device__ __forceinline__ void epilogue_loop(const KParams& p, const EpiCtx& c, const CUtensorMap* tmap_out) {
    SmemCtl* ctl = c.ctl;
    const int warp = c.warp, lane = c.lane;
    const int q = warp & 3;                    // TMEM lane quarter (a warp may only touch lanes 32*(warp%4)..)
    const int half = (warp - 4) >> 2;          // two warps per quarter: chunks k = half, half+2, ...
    const int row = q * 32 + lane;
    const int lx = row % p.BX, ly = row / p.BX;
    const int n_chunks = p.BLOCK_N >> 5;
    const int epi_tid = (int)threadIdx.x - 128;   // 0..255
    Ring buf;                                  // accumulator buffer
    uint32_t gphase = 0;
    float acc[8];                              // pooled-mode running sums (lane L owns column 32*k + L)
    float acc_sq[8];                           // ... of the squares (ACT 3 only; dead code otherwise)
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = acc_sq[k] = 0.f;
    int cur_key = -1, cur_nt = 0;
    const int cell_h = p.cells_y ? p.out_h / p.cells_y : 1, cell_w = p.cells_x ? p.out_w / p.cells_x : 1;
    const int ncells = p.cells_y * p.cells_x;
    int ss_key = -1;                           // (variant, nt) whose scale/shift currently sit in shared memory

    for (int unit = c.t_begin; unit < c.t_end; ++unit) {
        const int t = c.pair_rank < 0 ? unit : pair_tile(p, unit, c.pair_rank);
        int img, ty, tx, nt;
        decode_tile(p, t, img, ty, tx, nt);
        const int ox = tx * p.BX + lx, oy = ty * p.BY + ly;
        const bool valid = ox < p.out_w && oy < p.out_h && img < p.n_img;   // img >= n_img: padding tile of an odd pair

        // scale / shift of this (variant, N tile) -> shared memory (reloaded only when they change)
        const int var = (p.variant && img < p.n_img) ? __ldg(p.variant + img) : 0;
        const int want = var * p.n_tiles_n + nt;
        if (MODE != 3 && want != ss_key) {
            asm volatile("bar.sync 2, 256;" ::: "memory");          // everyone is done with the old table
            for (int i = epi_tid; i < p.BLOCK_N; i += kEpiThreads) {
                if (p.scale) c.s_scale[i] = __ldg(p.scale + nt * p.BLOCK_N + i);
                c.s_shift[i] = __ldg(p.shift + (size_t)var * p.N_pad + nt * p.BLOCK_N + i);
            }
            asm volatile("bar.sync 2, 256;" ::: "memory");
            ss_key = want;
        }

        tc::mbar_wait(&ctl->tmem_full[buf.i], buf.ph);
        tc::tc_fence_after();
        const uint32_t taddr0 = c.tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf.i * p.BLOCK_N);

        int key = -1;
        bool uniform = false;
        if (MODE == 2) {
            key = valid ? img * ncells + (oy / cell_h) * p.cells_x + (ox / cell_w) : -1;
            const unsigned vm = __ballot_sync(0xffffffffu, valid);
            const int leader_key = vm ? __shfl_sync(0xffffffffu, key, __ffs(vm) - 1) : -1;
            uniform = __all_sync(0xffffffffu, !valid || key == leader_key);
            if (uniform && vm && (leader_key != cur_key || nt != cur_nt)) {
                if (cur_key >= 0) {
#pragma unroll
                    for (int kk = 0; kk < 8; ++kk) {
                        if (kk < n_chunks && (kk & 1) == half) {
                            pool_add(p.pool + (size_t)cur_key * p.N_pad + cur_nt * p.BLOCK_N + kk * 32 + lane, acc[kk]);
                            acc[kk] = 0.f;
                            if (ACT == 3) {
                                pool_add(p.pool_sq + (size_t)cur_key * p.N_pad + cur_nt * p.BLOCK_N + kk * 32 + lane, acc_sq[kk]);
                                acc_sq[kk] = 0.f;
                            }
                        }
                    }
                }
                cur_key = leader_key;
                cur_nt = nt;
            }
            if (!vm) uniform = false;
        }
        if (MODE == 0) {
            if (p.gate_bytes) tc::mbar_wait(&ctl->gate_full, gphase);
            // the previous tile's TMA stores must have finished reading the staging buffer
            if (warp == 4 && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            asm volatile("bar.sync 1, 256;" ::: "memory");
        }

        if (MODE == 3) {
            // dF tile: columns are (segment, 32 channels); each warp half owns 16 channels and sums the
            // segments under the region masks of the INPUT pixel (y, x) = (oy*stride+py, ox*stride+px)
            const int y = oy * p.m3_stride + p.m3_py, x = ox * p.m3_stride + p.m3_px;
            const bool ok = valid && y < p.in_h && x < p.in_w;
            const unsigned code = ok ? p.codes[((size_t)img * p.in_h + y) * p.in_w + x] : 0u;
            float a16[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) a16[j] = 0.f;
            for (int sgm = 0; sgm < p.m3_n_seg; ++sgm) {
                uint32_t v16[16];
                tc::tmem_ld_32x16(taddr0 + (uint32_t)(sgm * 32 + half * 16), v16);
                tc::tmem_ld_wait();
                const bool keep = sgm >= p.m3_masked_segs || ((code >> sgm) & 1u);
                if (keep) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) a16[j] += __uint_as_float(v16[j]);
                }
            }
            if (ok) {
                const size_t plane = (size_t)p.in_h * p.in_w;
                const size_t base = (size_t)img * p.N * plane + (size_t)y * p.in_w + x;
                float* o = reinterpret_cast<float*>(p.out);
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int ch = nt * 32 + half * 16 + j;
                    if (ch < p.N) {
                        float r = a16[j];
                        if (p.residual) r += __ldg(p.residual + base + (size_t)ch * plane);
                        o[base + (size_t)ch * plane] = r;
                    }
                }
            }
        }
#pragma unroll 1
        for (int k = (MODE == 3 ? n_chunks : half); k < n_chunks; k += 2) {
            uint32_t v[32];
            tc::tmem_ld_32x32(taddr0 + (uint32_t)(k * 32), v);
            float sh[32], f[32];
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
                const float4 b = *reinterpret_cast<const float4*>(c.s_shift + k * 32 + j4 * 4);
                sh[j4 * 4] = b.x; sh[j4 * 4 + 1] = b.y; sh[j4 * 4 + 2] = b.z; sh[j4 * 4 + 3] = b.w;
            }
            if (SCALE) {
                float sc[32];
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4) {
                    const float4 a = *reinterpret_cast<const float4*>(c.s_scale + k * 32 + j4 * 4);
                    sc[j4 * 4] = a.x; sc[j4 * 4 + 1] = a.y; sc[j4 * 4 + 2] = a.z; sc[j4 * 4 + 3] = a.w;
                }
                tc::tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = fmaf(__uint_as_float(v[j]), sc[j], sh[j]);
            } else {
                tc::tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]) + sh[j];
            }
            const int n0 = nt * p.BLOCK_N + k * 32;
            // ReLU of the channels-last store is fused into the bf16 pack below
            if (!(MODE == 0 && ACT == 1)) {
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = act_fn<ACT>(f[j]);
            }

            if (MODE == 0) {
                // stage the bf16 tile in shared memory (128B-swizzled rows of 64 channels) for TMA stores
                const int grp = k >> 1;
                uint8_t* rowp = c.s_staging + grp * (kBlockM * 128) + row * 128;
                if (p.gate_bytes) {
                    if (ACT == 1) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
                    }
                    const uint8_t* grow = c.s_gate + grp * (kBlockM * 128) + row * 128;
#pragma unroll
                    for (int g4 = 0; g4 < 4; ++g4) {
                        const int piece = ((k & 1) * 4 + g4) ^ (row & 7);
                        const uint4 gv = *reinterpret_cast<const uint4*>(grow + piece * 16);
                        const __nv_bfloat162* g2 = reinterpret_cast<const __nv_bfloat162*>(&gv);
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            float2 gf = __bfloat1622float2(g2[e]);
                            f[g4 * 8 + e * 2] *= gf.x;
                            f[g4 * 8 + e * 2 + 1] *= gf.y;
                        }
                    }
                }
#pragma unroll
                for (int g4 = 0; g4 < 4; ++g4) {
                    uint4 o;
                    if (ACT == 1 && !p.gate_bytes) {
                        o.x = tc::pack_bf16x2_relu(f[g4 * 8 + 0], f[g4 * 8 + 1]);
                        o.y = tc::pack_bf16x2_relu(f[g4 * 8 + 2], f[g4 * 8 + 3]);
                        o.z = tc::pack_bf16x2_relu(f[g4 * 8 + 4], f[g4 * 8 + 5]);
                        o.w = tc::pack_bf16x2_relu(f[g4 * 8 + 6], f[g4 * 8 + 7]);
                    } else {
                        o.x = tc::pack_bf16x2(f[g4 * 8 + 0], f[g4 * 8 + 1]);
                        o.y = tc::pack_bf16x2(f[g4 * 8 + 2], f[g4 * 8 + 3]);
                        o.z = tc::pack_bf16x2(f[g4 * 8 + 4], f[g4 * 8 + 5]);
                        o.w = tc::pack_bf16x2(f[g4 * 8 + 6], f[g4 * 8 + 7]);
                    }
                    const int piece = ((k & 1) * 4 + g4) ^ (row & 7);
                    *reinterpret_cast<uint4*>(rowp + piece * 16) = o;
                }
            } else if (MODE == 1) {
                if (valid) {
                    const size_t plane = (size_t)p.out_h * p.out_w;
                    const size_t base = (size_t)img * p.N * plane + (size_t)oy * p.out_w + ox;
                    float* o = reinterpret_cast<float*>(p.out);
                    if (p.residual) {
                        float r[32];
#pragma unroll
                        for (int j = 0; j < 32; ++j) r[j] = (n0 + j < p.N) ? __ldg(p.residual + base + (size_t)(n0 + j) * plane) : 0.f;
#pragma unroll
                        for (int j = 0; j < 32; ++j) f[j] += r[j];
                    }
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (n0 + j < p.N) o[base + (size_t)(n0 + j) * plane] = f[j];
                    if (p.next_op && n0 < p.next_c_pad) {
                        uint4 v4[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            uint32_t* w = reinterpret_cast<uint32_t*>(&v4[e]);
#pragma unroll
                            for (int t = 0; t < 4; ++t) {
                                const int j = e * 8 + t * 2;
                                w[t] = tc::pack_bf16x2(n0 + j < p.N ? f[j] : 0.f, n0 + j + 1 < p.N ? f[j + 1] : 0.f);
                            }
                        }
                        const int H2 = (p.out_h + 1) >> 1, W2 = (p.out_w + 1) >> 1;
                        const int par = (oy & 1) * 2 + (ox & 1);
                        const unsigned code = p.next_masked_segs ? p.next_codes[((size_t)img * p.out_h + oy) * p.out_w + ox] : 0u;
                        const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
                        for (int sg = 0; sg < p.next_n_seg; ++sg) {
                            const bool keep = sg >= p.next_masked_segs || ((code >> sg) & 1u);
                            const size_t pl = ((size_t)img * p.next_n_seg + sg) * 4 + par;
                            uint4* dst = reinterpret_cast<uint4*>(p.next_op + ((pl * H2 + (oy >> 1)) * W2 + (ox >> 1)) * p.next_c_pad + n0);
#pragma unroll
                            for (int e = 0; e < 4; ++e) dst[e] = keep ? v4[e] : zero;
                        }
                    }
                }
            } else {
                if (uniform) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = valid ? f[j] : 0.f;
                    float g[32];
                    if (ACT == 3) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) g[j] = f[j] * f[j];
                    }
#pragma unroll
                    for (int s = 16; s >= 1; s >>= 1) {
                        const bool upper = (lane & s) != 0;
#pragma unroll
                        for (int i = 0; i < s; ++i) {
                            const float send = upper ? f[i] : f[i + s];
                            const float keep = upper ? f[i + s] : f[i];
                            f[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
                            if (ACT == 3) {
                                const float send2 = upper ? g[i] : g[i + s];
                                const float keep2 = upper ? g[i + s] : g[i];
                                g[i] = keep2 + __shfl_xor_sync(0xffffffffu, send2, s);
                            }
                        }
                    }
#pragma unroll
                    for (int kk = 0; kk < 8; ++kk)
                        if (kk == k) {
                            acc[kk] += f[0];
                            if (ACT == 3) acc_sq[kk] += g[0];
                        }
                } else if (valid) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        pool_add(p.pool + (size_t)key * p.N_pad + n0 + j, f[j]);
                        if (ACT == 3) pool_add(p.pool_sq + (size_t)key * p.N_pad + n0 + j, f[j] * f[j]);
                    }
                }
            }
        }
        tc::tc_fence_before();
        // one arrive per warp, CTA-scope release: the payload is tensor memory (read complete: tcgen05.wait::ld above,
        // ordered by the tcgen05 fence); a cluster-scope release per thread costs a MEMBAR.ALL.GPU + ERRBAR each
        __syncwarp();
        if (lane == 0) {
            if (c.tmem_empty_remote[buf.i]) tc::mbar_arrive_cluster_tmem(c.tmem_empty_remote[buf.i]);
            else tc::mbar_arrive(&ctl->tmem_empty[buf.i]);
        }
        buf.next(kAccStages);
        if (MODE == 0) {
            if (p.gate_bytes) {
                tc::mbar_arrive(&ctl->gate_empty);
                gphase ^= 1;
            }
            tc::fence_proxy_async();               // generic-proxy smem writes -> visible to the TMA engine
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if (warp == 4 && lane == 0) {
                for (int g = 0; g < (p.BLOCK_N >> 6); ++g)
                    tc::tma_store_4d(tmap_out, c.s_staging + g * (kBlockM * 128), nt * p.BLOCK_N + g * 64, tx * p.BX,
                                     ty * p.BY, img);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
        }
    }
    if (MODE == 0 && warp == 4 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    if (MODE == 2 && cur_key >= 0) {
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)
            if (kk < n_chunks && (kk & 1) == half) {
                pool_add(p.pool + (size_t)cur_key * p.N_pad + cur_nt * p.BLOCK_N + kk * 32 + lane, acc[kk]);
                if (ACT == 3) pool_add(p.pool_sq + (size_t)cur_key * p.N_pad + cur_nt * p.BLOCK_N + kk * 32 + lane, acc_sq[kk]);
            }
    }
}

// ---- the frame shared by the GEMM kernels ---------------------------------------------------------------------------------
enum GemmKind { kGemm, kGemmPair, kConv3x3, kConv3x3Pair, kDsam };

constexpr int kTile = kBlockM * 128;         // 16 KB: 128 pixels x 64 bf16 channels
constexpr int kDsamThreads = 512;            // dsam_fwd_kernel: 4 control warps + 8 epilogue warps + 4 mask warps
constexpr int kDsamRaw = 3;                  // dsam_fwd_kernel: raw (unmasked) tile ring, prefetched ahead of the masking

// Dynamic shared memory of a GEMM kernel from its 1024-aligned start: a kernel-specific head (conv_gemm_kernel: the resident
// weights; the 3x3 kernels: the ring of A tiles; dsam_fwd_kernel: the raw tiles and two groups of masked copies), the operand
// ring of p.stages slots, the staged output tile and the gate tile (epilogue mode 0), the barriers, the slice table and the
// scale / shift tables.  The host sizes the launch and the kernel places its buffers with this one function.
// Addr: uint8_t* from the aligned start in a kernel, size_t from 0 on the host.
template <typename Addr>
struct SmemLayout {
    Addr ring;                               // the operand ring
    int stage;                               // bytes per ring slot
    Addr staging, gate, ctl, slices, scale, shift, end;
};

template <typename Addr>
__host__ __device__ __forceinline__ SmemLayout<Addr> smem_layout(GemmKind kind, const KParams& p, Addr base) {
    SmemLayout<Addr> L;
    switch (kind) {
    case kGemm:
        L.ring = base + p.b_res_bytes;
        L.stage = kBlockM * p.kb_bytes + (p.b_resident ? 0 : p.BLOCK_N * p.kb_bytes);
        break;
    case kGemmPair:                          // A tile + this CTA's half of the B K block
        L.ring = base;
        L.stage = kBlockM * p.kb_bytes + (p.BLOCK_N / 2) * p.kb_bytes;
        break;
    case kConv3x3:
    case kConv3x3Pair:                       // B tiles (a CTA pair: half of each per CTA)
        L.ring = base + (size_t)p.sa_stages * p.a_stage_bytes;
        L.stage = (kind == kConv3x3 ? p.BLOCK_N : p.BLOCK_N / 2) * 128;
        break;
    case kDsam:                              // half weight tiles
        L.ring = base + (size_t)(kDsamRaw + 2 * p.m3_masked_segs) * kTile;
        L.stage = (p.BLOCK_N / 2) * 128;
        break;
    }
    L.staging = L.ring + (size_t)p.stages * L.stage;
    L.gate = L.staging + p.staging_bytes;
    L.ctl = L.gate + p.gate_bytes;
    L.slices = L.ctl + sizeof(SmemCtl);
    L.scale = L.slices + (size_t)p.n_slices * sizeof(int4);
    L.shift = L.scale + (size_t)p.BLOCK_N * sizeof(float);
    L.end = L.shift + (size_t)p.BLOCK_N * sizeof(float);
    return L;
}

// dynamic shared memory aligned to 1024 bytes (the period of the 128B swizzle); keeps the shared address space
__device__ __forceinline__ uint8_t* smem_base() {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    return smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
}

// Prologue of a GEMM kernel; PAIR: the CTA pair of a cluster runs tcgen05 cta_group::2.  Warp 0 prefetches the tensor maps,
// warp 1 initialises the operand ring's barriers and the accumulator buffers' barriers (tmem_empty: one arrive per epilogue
// warp of every CTA) and fences them together with the kernel's own, which the same thread initialised before the call;
// warp 2 allocates the tensor memory.  Returns its base address.
template <bool PAIR>
__device__ __forceinline__ uint32_t gemm_prologue(SmemCtl* ctl, const KParams& p, const CUtensorMap* tmap_a,
                                                  const CUtensorMap* tmap_b, const CUtensorMap* tmap_out,
                                                  const CUtensorMap* tmap_gate) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        tc::prefetch_tmap(tmap_a);
        tc::prefetch_tmap(tmap_b);
        if (p.staging_bytes) tc::prefetch_tmap(tmap_out);
        if (p.gate_bytes) tc::prefetch_tmap(tmap_gate);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < p.stages; ++s) {
            tc::mbar_init(&ctl->full[s], 1);
            tc::mbar_init(&ctl->empty[s], 1);
        }
        for (int s = 0; s < kAccStages; ++s) {
            tc::mbar_init(&ctl->tmem_full[s], 1);
            tc::mbar_init(&ctl->tmem_empty[s], (PAIR ? 2 : 1) * kEpiWarps);
        }
        tc::fence_barrier_init();
    }
    if (PAIR) {
        tc::cluster_sync_all();              // the barriers of both CTAs exist before any remote use
        if (warp == 2) tc::tmem_alloc_2cta(&ctl->tmem_base, kTmemCols);
        tc::tc_fence_before();
        tc::cluster_sync_all();
    } else {
        if (warp == 2) tc::tmem_alloc(&ctl->tmem_base, kTmemCols);
        tc::tc_fence_before();
        __syncthreads();
    }
    tc::tc_fence_after();
    return ctl->tmem_base;
}

// Contiguous range [begin, end) of work units of this CTA (PAIR: of this CTA pair): tiles, or pair units (see pair_tile).
// Contiguous ranges keep the pooled epilogue's partial sums in registers across tiles.
template <bool PAIR>
__device__ __forceinline__ void work_range(const KParams& p, int& begin, int& end) {
    const int units = PAIR ? ((p.total_tiles / p.n_tiles_n + 1) / 2) * p.n_tiles_n : p.total_tiles;
    const int n = PAIR ? (int)gridDim.x / 2 : (int)gridDim.x, id = PAIR ? (int)blockIdx.x / 2 : (int)blockIdx.x;
    const int per = units / n, rem = units % n;
    begin = id * per + min(id, rem);
    end = begin + per + (id < rem ? 1 : 0);
}

// the epilogue warps' view; in a CTA pair they release the accumulator on the leader's tmem_empty barriers
template <bool PAIR>
__device__ __forceinline__ EpiCtx epi_ctx(const SmemLayout<uint8_t*>& L, SmemCtl* ctl, uint32_t tmem_base, int begin, int end) {
    EpiCtx c{L.staging, L.gate, ctl, reinterpret_cast<float*>(L.scale), reinterpret_cast<float*>(L.shift), tmem_base, begin, end,
             (int)threadIdx.x >> 5, (int)threadIdx.x & 31, -1, {0u, 0u}};
    if (PAIR) {
        c.pair_rank = (int)tc::cluster_ctarank();
        for (int b = 0; b < kAccStages; ++b) c.tmem_empty_remote[b] = tc::mapa(tc::smem_u32(&ctl->tmem_empty[b]), 0);
    }
    return c;
}

template <bool PAIR>
__device__ __forceinline__ void gemm_teardown(uint32_t tmem_base) {
    tc::tc_fence_before();
    if (PAIR) tc::cluster_sync_all();        // the peer's smem / TMEM stay alive until the leader's MMAs are done
    else __syncthreads();
    if ((threadIdx.x >> 5) == 2) {
        tc::tc_fence_after();
        if (PAIR) tc::tmem_dealloc_2cta(tmem_base, kTmemCols);
        else tc::tmem_dealloc(tmem_base, kTmemCols);
    }
}

// Every GEMM kernel takes the same parameters: A and B maps, the output and gate maps of epilogue mode 0 (placeholders
// otherwise) and the parameter block.
template <bool STATS>
__global__ void __launch_bounds__(kThreads, 1)
conv_gemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                 const __grid_constant__ CUtensorMap tmap_out, const __grid_constant__ CUtensorMap tmap_gate,
                 const __grid_constant__ KParams p) {
    uint8_t* smem = smem_base();
    const SmemLayout<uint8_t*> L = smem_layout(kGemm, p, smem);
    const int a_bytes = kBlockM * p.kb_bytes;
    const int b_bytes = p.BLOCK_N * p.kb_bytes;
    uint8_t* s_bres = smem;                                                  // resident weights (b_resident)
    uint8_t* s_ring = L.ring;
    uint8_t* s_gate = L.gate;
    SmemCtl* ctl = reinterpret_cast<SmemCtl*>(L.ctl);
    int4* s_slices = reinterpret_cast<int4*>(L.slices);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < p.n_slices; i += blockDim.x) s_slices[i] = p.slices[i];
    if (warp == 1 && lane == 0) {
        tc::mbar_init(&ctl->b_full, 1);
        tc::mbar_init(&ctl->gate_full, 1);
        tc::mbar_init(&ctl->gate_empty, kEpiThreads);
    }
    const uint32_t tmem_base = gemm_prologue<false>(ctl, p, &tmap_a, &tmap_b, &tmap_out, &tmap_gate);
    int t_begin, t_end;
    work_range<false>(p, t_begin, t_end);

    if (warp == 0 && lane == 0) {
        // ================= TMA producer =================
        Ring st;
        uint32_t gphase = 0;
        if (p.b_resident) {
            tc::mbar_expect_tx(&ctl->b_full, (uint32_t)p.b_res_bytes);
            for (int j = 0; j < p.n_slices; ++j)
                tc::tma_load_2d(s_bres + (size_t)j * b_bytes, &tmap_b, &ctl->b_full, j * (p.kb_bytes >> 1), 0);
        }
        for (int t = t_begin; t < t_end; ++t) {
            int img, ty, tx, nt;
            decode_tile(p, t, img, ty, tx, nt);
            const int x0 = tx * p.BX, y0 = ty * p.BY, pl0 = img * p.plane_per_img;
            if (p.gate_bytes) {
                tc::mbar_wait(&ctl->gate_empty, gphase ^ 1);
                tc::mbar_expect_tx(&ctl->gate_full, (uint32_t)p.gate_bytes);
                for (int g = 0; g < (p.BLOCK_N >> 6); ++g)
                    tc::tma_load_4d(s_gate + g * (kBlockM * 128), &tmap_gate, &ctl->gate_full, nt * p.BLOCK_N + g * 64, x0,
                                    y0, img);
                gphase ^= 1;
            }
            for (int j = 0; j < p.n_slices; ++j) {
                tc::mbar_wait(&ctl->empty[st.i], st.ph ^ 1);
                uint8_t* sa = s_ring + (size_t)st.i * L.stage;
                uint8_t* sb = sa + a_bytes;
                tc::mbar_expect_tx(&ctl->full[st.i], (uint32_t)L.stage);
                const int4 sl = s_slices[j];
                tc::tma_load_4d(sa, &tmap_a, &ctl->full[st.i], sl.x, x0 + sl.y, y0 + sl.z, pl0 + sl.w);
                if (!p.b_resident)
                    tc::tma_load_2d(sb, &tmap_b, &ctl->full[st.i], j * (p.kb_bytes >> 1), nt * p.BLOCK_N);
                st.next(p.stages);
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer: whole warp in uniform control flow, one elected lane issues =================
        const uint32_t idesc = tc::make_idesc_bf16(kBlockM, p.BLOCK_N);
        const int k_per_block = p.kb_bytes >> 5;           // UMMA_K = 16 bf16 = 32 bytes
        Ring st, buf;
        if (p.b_resident) tc::mbar_wait(&ctl->b_full, 0);
        for (int t = t_begin; t < t_end; ++t) {
            tc::mbar_wait(&ctl->tmem_empty[buf.i], buf.ph ^ 1);
            tc::tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(buf.i * p.BLOCK_N);
            for (int j = 0; j < p.n_slices; ++j) {
                tc::mbar_wait(&ctl->full[st.i], st.ph);
                tc::tc_fence_after();
                const uint32_t sa = tc::smem_u32(s_ring + (size_t)st.i * L.stage);
                const uint32_t sb = p.b_resident ? tc::smem_u32(s_bres + (size_t)j * b_bytes) : sa + a_bytes;
                const uint64_t adesc = tc::make_kmajor_desc(sa, p.kb_bytes);
                const uint64_t bdesc = tc::make_kmajor_desc(sb, p.kb_bytes);
                if (tc::elect_one()) {
                    for (int k = 0; k < k_per_block; ++k)
                        tc::umma_bf16(d_tmem, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (j | k) != 0);
                    tc::umma_commit(&ctl->empty[st.i]);
                    if (j == p.n_slices - 1) tc::umma_commit(&ctl->tmem_full[buf.i]);
                }
                __syncwarp();
                st.next(p.stages);
            }
            buf.next(kAccStages);
        }
    } else if (warp >= 4) {
        // ================= epilogue =================
        const EpiCtx c = epi_ctx<false>(L, ctl, tmem_base, t_begin, t_end);
        const bool sc = p.scale != nullptr;
        if (p.epi_mode == 0) {
            if (p.act == 2) epilogue_loop<0, 2, false>(p, c, &tmap_out);
            else if (p.act == 1 && sc) epilogue_loop<0, 1, true>(p, c, &tmap_out);
            else if (p.act == 1) epilogue_loop<0, 1, false>(p, c, &tmap_out);
            else if (sc) epilogue_loop<0, 0, true>(p, c, &tmap_out);
            else epilogue_loop<0, 0, false>(p, c, &tmap_out);
        } else if (p.epi_mode == 1) {
            if (sc) epilogue_loop<1, 0, true>(p, c, &tmap_out);
            else epilogue_loop<1, 0, false>(p, c, &tmap_out);
        } else if (p.epi_mode == 3) {
            epilogue_loop<3, 0, false>(p, c, &tmap_out);
        } else {
            if (STATS) epilogue_loop<2, 3, false>(p, c, &tmap_out);
            else if (sc) epilogue_loop<2, 1, true>(p, c, &tmap_out);
            else epilogue_loop<2, 1, false>(p, c, &tmap_out);
        }
    }
    gemm_teardown<false>(tmem_base);
}


// 3x3 stride-1 pad-1 convolution with shared-memory reuse of the A operand across the three dx taps
// (reference CM:1412-1416, the 128->256 conv that carries 84 % of the ratio predictor's FLOPs).
// For every (dy, 64-channel block) ONE tile of 130 pixels (x0-1 .. x0+128) is loaded; the MMAs of tap dx read it
// through a descriptor whose start address is advanced by dx rows of 128 bytes (the 128B swizzle is a function of
// the absolute shared-memory address, profiles/r01_notes.md).  Per output tile the SM receives 6 A tiles instead
// of 18, i.e. 676 KB instead of 864 KB over its 64 B/clk L2 port (MMA time: 9216 cycles = 590 KB at 64 B/clk).
template <bool STATS>
__global__ void __launch_bounds__(kThreads, 1)
conv3x3_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
               const __grid_constant__ CUtensorMap tmap_out, const __grid_constant__ CUtensorMap tmap_gate,
               const __grid_constant__ KParams p) {
    uint8_t* smem = smem_base();
    const SmemLayout<uint8_t*> L = smem_layout(kConv3x3, p, smem);
    uint8_t* s_a = smem;
    uint8_t* s_b = L.ring;
    SmemCtl* ctl = reinterpret_cast<SmemCtl*>(L.ctl);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < p.sa_stages; ++s) {
            tc::mbar_init(&ctl->a_full[s], 1);
            tc::mbar_init(&ctl->a_empty[s], 1);
        }
        tc::mbar_init(&ctl->gate_full, 1);
        tc::mbar_init(&ctl->gate_empty, kEpiThreads);
    }
    const uint32_t tmem_base = gemm_prologue<false>(ctl, p, &tmap_a, &tmap_b, &tmap_out, &tmap_gate);
    int t_begin, t_end;
    work_range<false>(p, t_begin, t_end);

    if (warp == 0 && lane == 0) {
        // ================= TMA producer =================
        Ring ra, rb;
        for (int t = t_begin; t < t_end; ++t) {
            int img, ty, tx, nt;
            decode_tile(p, t, img, ty, tx, nt);
            const int x0 = tx * p.BX, y0 = ty;
            for (int dy = 0; dy < 3; ++dy) {
                for (int cb = 0; cb < p.c_blocks; ++cb) {
                    tc::mbar_wait(&ctl->a_empty[ra.i], ra.ph ^ 1);
                    tc::mbar_expect_tx(&ctl->a_full[ra.i], (uint32_t)((kBlockM + 2) * 128));
                    tc::tma_load_4d(s_a + (size_t)ra.i * p.a_stage_bytes, &tmap_a, &ctl->a_full[ra.i], cb * 64, x0 - 1, y0 + dy - 1, img);
                    ra.next(p.sa_stages);
                    for (int dx = 0; dx < 3; ++dx) {
                        tc::mbar_wait(&ctl->empty[rb.i], rb.ph ^ 1);
                        tc::mbar_expect_tx(&ctl->full[rb.i], (uint32_t)L.stage);
                        tc::tma_load_2d(s_b + (size_t)rb.i * L.stage, &tmap_b, &ctl->full[rb.i],
                                        ((dy * 3 + dx) * p.c_blocks + cb) * 64, nt * p.BLOCK_N);
                        rb.next(p.stages);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer: whole warp in uniform control flow, one elected lane issues =================
        const uint32_t idesc = tc::make_idesc_bf16(kBlockM, p.BLOCK_N);
        Ring ra, rb, buf;
        for (int t = t_begin; t < t_end; ++t) {
            tc::mbar_wait(&ctl->tmem_empty[buf.i], buf.ph ^ 1);
            tc::tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(buf.i * p.BLOCK_N);
            uint32_t first = 0;                 // 0 until the tile's first MMA (overwrites the accumulator)
            for (int dy = 0; dy < 3; ++dy) {
                for (int cb = 0; cb < p.c_blocks; ++cb) {
                    tc::mbar_wait(&ctl->a_full[ra.i], ra.ph);
                    const uint32_t a_base = tc::smem_u32(s_a + (size_t)ra.i * p.a_stage_bytes);
                    for (int dx = 0; dx < 3; ++dx) {
                        tc::mbar_wait(&ctl->full[rb.i], rb.ph);
                        tc::tc_fence_after();
                        const uint64_t adesc = tc::make_kmajor_desc(a_base + (uint32_t)(dx * 128), 128);
                        const uint64_t bdesc = tc::make_kmajor_desc(tc::smem_u32(s_b + (size_t)rb.i * L.stage), 128);
                        if (tc::elect_one()) {
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                tc::umma_bf16(d_tmem, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (first | k) ? 1u : 0u);
                            tc::umma_commit(&ctl->empty[rb.i]);
                            if (dx == 2) {
                                tc::umma_commit(&ctl->a_empty[ra.i]);
                                if (dy == 2 && cb == p.c_blocks - 1) tc::umma_commit(&ctl->tmem_full[buf.i]);
                            }
                        }
                        __syncwarp();
                        first = 1;
                        rb.next(p.stages);
                    }
                    ra.next(p.sa_stages);
                }
            }
            buf.next(kAccStages);
        }
    } else if (warp >= 4) {
        const EpiCtx c = epi_ctx<false>(L, ctl, tmem_base, t_begin, t_end);
        const bool sc = p.scale != nullptr;
        if (p.epi_mode == 0) {
            if (p.act == 1 && !sc) epilogue_loop<0, 1, false>(p, c, &tmap_out);
            else epilogue_loop<0, 0, false>(p, c, &tmap_out);
        } else if (p.epi_mode == 1) {
            epilogue_loop<1, 0, false>(p, c, &tmap_out);
        } else {
            if (STATS) epilogue_loop<2, 3, false>(p, c, &tmap_out);
            else if (sc) epilogue_loop<2, 1, true>(p, c, &tmap_out);
            else epilogue_loop<2, 1, false>(p, c, &tmap_out);
        }
    }
    gemm_teardown<false>(tmem_base);
}

// DSAModule.forward (CM:683-696) without the five-fold masked operand in HBM: the UNMASKED feature tile of a
// (tap, 64-channel block) is loaded once by TMA; four "mask warps" write the region-masked copies
// (mask_t * F = the tile with the rows of pixels outside region t zeroed, region bits from the pooled code of the
// INPUT pixel the tap reads) into shared memory; the MMA then runs the five K blocks [p0*F | p1*F | p2*F | p3*F | F]
// against the five weight tiles.  Versus conv_gemm on a pre-masked operand this loads 128 + 5*BLOCK_N/2 TMA rows per
// 5 K blocks instead of 5*(128 + BLOCK_N/2) and the pack kernel writes one copy instead of five.  CTA pairs
// (cta_group::2): every CTA masks its own tile, the weight tiles are split between the two CTAs.
__global__ void __launch_bounds__(kDsamThreads, 1)
dsam_fwd_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                const __grid_constant__ CUtensorMap tmap_out, const __grid_constant__ CUtensorMap tmap_gate,
                const __grid_constant__ KParams p) {
    uint8_t* smem = smem_base();
    const SmemLayout<uint8_t*> L = smem_layout(kDsam, p, smem);
    const int n_seg = p.m3_n_seg;                              // 5: four masked segments + the projection copy
    const int n_msk = p.m3_masked_segs;
    uint8_t* s_rawt = smem;                                    // kDsamRaw raw tiles (TMA targets; also the projection operand)
    uint8_t* s_msk = s_rawt + kDsamRaw * kTile;                // 2 groups x n_msk masked copies
    uint8_t* s_b = L.ring;
    SmemCtl* ctl = reinterpret_cast<SmemCtl*>(L.ctl);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = tc::cluster_ctarank();
    const bool leader = rank == 0;
    if (warp == 1 && lane == 0) {
        for (int r = 0; r < kDsamRaw; ++r) {
            tc::mbar_init(&ctl->a_full[r], 1);                 // raw tile landed (local TMA)
            tc::mbar_init(&ctl->a_empty[r], 1);                // released by the pair's MMAs (multicast commit)
        }
        for (int g = 0; g < 2; ++g) {
            tc::mbar_init(&ctl->masked_full[g], 2 * 4);        // one arrive per mask warp of BOTH CTAs (counted in the leader)
            tc::mbar_init(&ctl->masked_empty[g], 1);           // multicast commit
        }
    }
    const uint32_t tmem_base = gemm_prologue<true>(ctl, p, &tmap_a, &tmap_b, &tmap_out, &tmap_gate);
    int u_begin, u_end;
    work_range<true>(p, u_begin, u_end);
    const int groups_per_tile = p.dsam_taps * p.c_blocks;

    if (warp == 0 && lane == 0) {
        // ================= TMA producer: weight tiles =================
        Ring rb;
        for (int u = u_begin; u < u_end; ++u) {
            const int nt = pair_tile(p, u, (int)rank) % p.n_tiles_n;
            for (int gi = 0; gi < groups_per_tile; ++gi) {
                for (int sg = 0; sg < n_seg; ++sg) {
                    tc::mbar_wait(&ctl->empty[rb.i], rb.ph ^ 1);
                    if (leader) tc::mbar_expect_tx(&ctl->full[rb.i], 2u * (uint32_t)L.stage);
                    tc::tma_load_2d_2cta(s_b + (size_t)rb.i * L.stage, &tmap_b, &ctl->full[rb.i], (gi * n_seg + sg) * 64,
                                         nt * p.BLOCK_N + (int)rank * (p.BLOCK_N / 2));
                    rb.next(p.stages);
                }
            }
        }
    } else if (warp == 3 && lane == 0) {
        // ================= TMA producer: raw feature tiles (own ring, runs ahead of the masking) =================
        Ring raw;
        for (int u = u_begin; u < u_end; ++u) {
            int img, ty, tx, nt;
            decode_tile(p, pair_tile(p, u, (int)rank), img, ty, tx, nt);
            const int x0 = tx * p.BX, y0 = ty * p.BY;
            for (int tap = 0; tap < p.dsam_taps; ++tap) {
                const int dy = tap / 3, dx = tap % 3;
                // input row 2*oy+dy-1: dy=0 -> odd plane, row oy-1; dy=1 -> even plane, row oy; dy=2 -> odd plane, row oy
                const int par = (dy == 1 ? 0 : 2) + (dx == 1 ? 0 : 1);
                const int yo = dy == 0 ? -1 : 0, xo = dx == 0 ? -1 : 0;
                for (int cb = 0; cb < p.c_blocks; ++cb) {
                    tc::mbar_wait(&ctl->a_empty[raw.i], raw.ph ^ 1);
                    tc::mbar_expect_tx(&ctl->a_full[raw.i], kTile);
                    tc::tma_load_4d(s_rawt + (size_t)raw.i * kTile, &tmap_a, &ctl->a_full[raw.i], cb * 64, x0 + xo, y0 + yo, img * 4 + par);
                    raw.next(kDsamRaw);
                }
            }
        }
    } else if (warp == 1 && leader) {
        // ================= MMA issuer (leader): the whole warp runs the uniform control flow so the descriptors stay in
        // uniform registers (no per-MMA ELECT/R2UR waterfall); one elected lane issues =================
        const uint32_t idesc = tc::make_idesc_bf16(2 * kBlockM, p.BLOCK_N);
        Ring grp, raw, rb, buf;
        for (int u = u_begin; u < u_end; ++u) {
            tc::mbar_wait(&ctl->tmem_empty[buf.i], buf.ph ^ 1);
            tc::tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(buf.i * p.BLOCK_N);
            uint32_t first = 0;                                 // 0 until the tile's first MMA (overwrites the accumulator)
            for (int gi = 0; gi < groups_per_tile; ++gi) {
                tc::mbar_wait(&ctl->masked_full[grp.i], grp.ph);   // both CTAs: raw tile landed and masked copies written
                tc::tc_fence_after();
                for (int sg = 0; sg < n_seg; ++sg) {
                    tc::mbar_wait(&ctl->full[rb.i], rb.ph);
                    tc::tc_fence_after();
                    const uint8_t* a_tile = sg < n_msk ? s_msk + (size_t)(grp.i * n_msk + sg) * kTile : s_rawt + (size_t)raw.i * kTile;
                    const uint64_t adesc = tc::make_kmajor_desc(tc::smem_u32(a_tile), 128);
                    const uint64_t bdesc = tc::make_kmajor_desc(tc::smem_u32(s_b + (size_t)rb.i * L.stage), 128);
                    if (tc::elect_one()) {
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            tc::umma_bf16_2cta(d_tmem, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (first | k) ? 1u : 0u);
                        tc::umma_commit_2cta(&ctl->empty[rb.i]);
                        if (sg == n_seg - 1) {
                            tc::umma_commit_2cta(&ctl->masked_empty[grp.i]);
                            tc::umma_commit_2cta(&ctl->a_empty[raw.i]);
                            if (gi == groups_per_tile - 1) tc::umma_commit_2cta(&ctl->tmem_full[buf.i]);
                        }
                    }
                    __syncwarp();
                    first = 1;
                    rb.next(p.stages);
                }
                grp.next(2);
                raw.next(kDsamRaw);
            }
            buf.next(kAccStages);
        }
    } else if (warp >= 12) {
        // ================= mask warps: masked copies of the raw tile =================
        const int row = (warp - 12) * 32 + lane;               // pixel row of the tile
        const int lx = row % p.BX, ly = row / p.BX;
        const uint32_t masked_full_remote[2] = {tc::mapa(tc::smem_u32(&ctl->masked_full[0]), 0),
                                                tc::mapa(tc::smem_u32(&ctl->masked_full[1]), 0)};
        Ring grp, raw;
        for (int u = u_begin; u < u_end; ++u) {
            int img, ty, tx, nt;
            decode_tile(p, pair_tile(p, u, (int)rank), img, ty, tx, nt);
            const int oy = ty * p.BY + ly, ox = tx * p.BX + lx;
            const bool img_ok = img < p.n_img;
            for (int tap = 0; tap < p.dsam_taps; ++tap) {
                const int iy = 2 * oy + tap / 3 - 1, ix = 2 * ox + tap % 3 - 1;
                unsigned code = 0;
                if (img_ok && iy >= 0 && iy < p.in_h && ix >= 0 && ix < p.in_w)
                    code = p.codes[((size_t)img * p.in_h + iy) * p.in_w + ix];
                for (int cb = 0; cb < p.c_blocks; ++cb) {
                    tc::mbar_wait(&ctl->a_full[raw.i], raw.ph);
                    const uint8_t* src = s_rawt + (size_t)raw.i * kTile + row * 128;
                    uint4 v[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = *reinterpret_cast<const uint4*>(src + (((j + row) & 7) << 4));   // rotated: bank-conflict free
                    tc::mbar_wait(&ctl->masked_empty[grp.i], grp.ph ^ 1);
                    const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
                    for (int sg = 0; sg < n_msk; ++sg) {
                        uint8_t* dst = s_msk + (size_t)(grp.i * n_msk + sg) * kTile + row * 128;
                        const bool keep = (code >> sg) & 1u;
#pragma unroll
                        for (int j = 0; j < 8; ++j) *reinterpret_cast<uint4*>(dst + (((j + row) & 7) << 4)) = keep ? v[j] : zero;
                    }
                    tc::fence_proxy_async();                   // generic-proxy writes -> visible to the tensor core's smem reads
                    __syncwarp();
                    // one arrive per warp, CTA-scope release: the copies are read by THIS CTA's tensor core (async proxy,
                    // ordered by the fence above); the remote barrier only signals the leader's MMA thread
                    if (lane == 0) tc::mbar_arrive_cluster_tmem(masked_full_remote[grp.i]);
                    grp.next(2);
                    raw.next(kDsamRaw);
                }
            }
        }
    } else if (warp >= 4 && warp < 12) {
        const EpiCtx c = epi_ctx<true>(L, ctl, tmem_base, u_begin, u_end);
        epilogue_loop<1, 0, false>(p, c, &tmap_out);
    }
    gemm_teardown<true>(tmem_base);
}

// conv_gemm_kernel on CTA pairs (tcgen05 cta_group::2) for the DSAM stages (epilogue modes 1 and 3): the two CTAs of a
// cluster take adjacent M tiles of the same N tile, so each stages only half of every B (weight) K block.
__global__ void __launch_bounds__(kThreads, 1)
conv_gemm_2cta_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                      const __grid_constant__ CUtensorMap tmap_out, const __grid_constant__ CUtensorMap tmap_gate,
                      const __grid_constant__ KParams p) {
    uint8_t* smem = smem_base();
    const SmemLayout<uint8_t*> L = smem_layout(kGemmPair, p, smem);
    const int a_bytes = kBlockM * p.kb_bytes;
    SmemCtl* ctl = reinterpret_cast<SmemCtl*>(L.ctl);
    int4* s_slices = reinterpret_cast<int4*>(L.slices);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = tc::cluster_ctarank();
    const bool leader = rank == 0;
    for (int i = threadIdx.x; i < p.n_slices; i += blockDim.x) s_slices[i] = p.slices[i];
    const uint32_t tmem_base = gemm_prologue<true>(ctl, p, &tmap_a, &tmap_b, &tmap_out, &tmap_gate);
    int u_begin, u_end;
    work_range<true>(p, u_begin, u_end);

    if (warp == 0 && lane == 0) {
        Ring st;
        for (int u = u_begin; u < u_end; ++u) {
            int img, ty, tx, nt;
            decode_tile(p, pair_tile(p, u, (int)rank), img, ty, tx, nt);
            const int x0 = tx * p.BX, y0 = ty * p.BY, pl0 = img * p.plane_per_img;
            for (int j = 0; j < p.n_slices; ++j) {
                tc::mbar_wait(&ctl->empty[st.i], st.ph ^ 1);
                uint8_t* sa = L.ring + (size_t)st.i * L.stage;
                if (leader) tc::mbar_expect_tx(&ctl->full[st.i], 2u * (uint32_t)L.stage);
                const int4 sl = s_slices[j];
                tc::tma_load_4d_2cta(sa, &tmap_a, &ctl->full[st.i], sl.x, x0 + sl.y, y0 + sl.z, pl0 + sl.w);
                tc::tma_load_2d_2cta(sa + a_bytes, &tmap_b, &ctl->full[st.i], j * (p.kb_bytes >> 1),
                                     nt * p.BLOCK_N + (int)rank * (p.BLOCK_N / 2));
                st.next(p.stages);
            }
        }
    } else if (warp == 1 && leader) {
        // whole warp in uniform control flow, one elected lane issues (descriptors stay in uniform registers)
        const uint32_t idesc = tc::make_idesc_bf16(2 * kBlockM, p.BLOCK_N);
        const int k_per_block = p.kb_bytes >> 5;
        Ring st, buf;
        for (int u = u_begin; u < u_end; ++u) {
            tc::mbar_wait(&ctl->tmem_empty[buf.i], buf.ph ^ 1);
            tc::tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(buf.i * p.BLOCK_N);
            for (int j = 0; j < p.n_slices; ++j) {
                tc::mbar_wait(&ctl->full[st.i], st.ph);
                tc::tc_fence_after();
                const uint32_t sa = tc::smem_u32(L.ring + (size_t)st.i * L.stage);
                const uint64_t adesc = tc::make_kmajor_desc(sa, p.kb_bytes);
                const uint64_t bdesc = tc::make_kmajor_desc(sa + a_bytes, p.kb_bytes);
                if (tc::elect_one()) {
                    for (int k = 0; k < k_per_block; ++k)
                        tc::umma_bf16_2cta(d_tmem, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (j | k) != 0);
                    tc::umma_commit_2cta(&ctl->empty[st.i]);
                    if (j == p.n_slices - 1) tc::umma_commit_2cta(&ctl->tmem_full[buf.i]);
                }
                __syncwarp();
                st.next(p.stages);
            }
            buf.next(kAccStages);
        }
    } else if (warp >= 4) {
        const EpiCtx c = epi_ctx<true>(L, ctl, tmem_base, u_begin, u_end);
        if (p.epi_mode == 3) epilogue_loop<3, 0, false>(p, c, &tmap_out);
        else if (p.scale) epilogue_loop<1, 0, true>(p, c, &tmap_out);
        else epilogue_loop<1, 0, false>(p, c, &tmap_out);
    }
    gemm_teardown<true>(tmem_base);
}

// The same 3x3 convolution on a CTA PAIR (tcgen05 cta_group::2): the two CTAs of a cluster work on two consecutive
// output tiles (rows y, y+1 of one column strip) as ONE M=256 MMA.  Each CTA stages its own A tiles and only HALF of
// every B tile (128 of the 256 output channels); the tensor cores of both SMs read both halves.  Per tile the SM's
// L2 inbound drops from 676 KB to 388 KB (64 B/clk port; 9216 MMA cycles = 590 KB) and its shared-memory operand
// reads from 96 to 64 B/clk, so the kernel becomes MMA-bound.  Leader (cluster rank 0) issues the MMAs; both CTAs
// issue TMA loads (bytes counted on the leader's barriers) and run their own epilogue on their own TMEM half.
template <bool STATS>
__global__ void __launch_bounds__(kThreads, 1)
conv3x3_2cta_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                    const __grid_constant__ CUtensorMap tmap_out, const __grid_constant__ CUtensorMap tmap_gate,
                    const __grid_constant__ KParams p) {
    uint8_t* smem = smem_base();
    const SmemLayout<uint8_t*> L = smem_layout(kConv3x3Pair, p, smem);
    uint8_t* s_a = smem;
    uint8_t* s_b = L.ring;
    SmemCtl* ctl = reinterpret_cast<SmemCtl*>(L.ctl);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = tc::cluster_ctarank();
    const bool leader = rank == 0;
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < p.sa_stages; ++s) {
            tc::mbar_init(&ctl->a_full[s], 1);
            tc::mbar_init(&ctl->a_empty[s], 1);
        }
    }
    const uint32_t tmem_base = gemm_prologue<true>(ctl, p, &tmap_a, &tmap_b, &tmap_out, &tmap_gate);
    // pairs of tiles (2u, 2u+1) are split contiguously over the clusters (one N tile)
    int u_begin, u_end;
    work_range<true>(p, u_begin, u_end);

    if (warp == 0 && lane == 0) {
        // ================= TMA producer (both CTAs) =================
        Ring ra, rb;
        for (int u = u_begin; u < u_end; ++u) {
            int img, ty, tx, nt;
            decode_tile(p, pair_tile(p, u, (int)rank), img, ty, tx, nt);
            const int x0 = tx * p.BX, y0 = ty;
            for (int dy = 0; dy < 3; ++dy) {
                for (int cb = 0; cb < p.c_blocks; ++cb) {
                    tc::mbar_wait(&ctl->a_empty[ra.i], ra.ph ^ 1);
                    if (leader) tc::mbar_expect_tx(&ctl->a_full[ra.i], 2u * (uint32_t)((kBlockM + 2) * 128));
                    tc::tma_load_4d_2cta(s_a + (size_t)ra.i * p.a_stage_bytes, &tmap_a, &ctl->a_full[ra.i], cb * 64, x0 - 1,
                                         y0 + dy - 1, img);
                    ra.next(p.sa_stages);
                    for (int dx = 0; dx < 3; ++dx) {
                        tc::mbar_wait(&ctl->empty[rb.i], rb.ph ^ 1);
                        if (leader) tc::mbar_expect_tx(&ctl->full[rb.i], 2u * (uint32_t)L.stage);
                        tc::tma_load_2d_2cta(s_b + (size_t)rb.i * L.stage, &tmap_b, &ctl->full[rb.i],
                                             ((dy * 3 + dx) * p.c_blocks + cb) * 64, (int)rank * (p.BLOCK_N / 2));
                        rb.next(p.stages);
                    }
                }
            }
        }
    } else if (warp == 1 && leader) {
        // ================= MMA issuer (leader CTA only): whole warp in uniform control flow, one elected lane issues (keeps the
        // descriptors in uniform registers: no per-MMA ELECT/R2UR waterfall) =================
        const uint32_t idesc = tc::make_idesc_bf16(2 * kBlockM, p.BLOCK_N);
        Ring ra, rb, buf;
        for (int u = u_begin; u < u_end; ++u) {
            tc::mbar_wait(&ctl->tmem_empty[buf.i], buf.ph ^ 1);
            tc::tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(buf.i * p.BLOCK_N);
            uint32_t started = 0;
            for (int dy = 0; dy < 3; ++dy) {
                for (int cb = 0; cb < p.c_blocks; ++cb) {
                    tc::mbar_wait(&ctl->a_full[ra.i], ra.ph);
                    const uint32_t a_base = tc::smem_u32(s_a + (size_t)ra.i * p.a_stage_bytes);
                    for (int dx = 0; dx < 3; ++dx) {
                        tc::mbar_wait(&ctl->full[rb.i], rb.ph);
                        tc::tc_fence_after();
                        const uint64_t adesc = tc::make_kmajor_desc(a_base + (uint32_t)(dx * 128), 128);
                        const uint64_t bdesc = tc::make_kmajor_desc(tc::smem_u32(s_b + (size_t)rb.i * L.stage), 128);
                        if (tc::elect_one()) {
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                tc::umma_bf16_2cta(d_tmem, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc,
                                                   (started | k) ? 1u : 0u);
                            tc::umma_commit_2cta(&ctl->empty[rb.i]);
                            if (dx == 2) {
                                tc::umma_commit_2cta(&ctl->a_empty[ra.i]);
                                if (dy == 2 && cb == p.c_blocks - 1) tc::umma_commit_2cta(&ctl->tmem_full[buf.i]);
                            }
                        }
                        __syncwarp();
                        started = 1;
                        rb.next(p.stages);
                    }
                    ra.next(p.sa_stages);
                }
            }
            buf.next(kAccStages);
        }
    } else if (warp >= 4) {
        // ================= epilogue (both CTAs, each on its own 128 TMEM lanes) =================
        const EpiCtx c = epi_ctx<true>(L, ctl, tmem_base, u_begin, u_end);
        if (STATS) epilogue_loop<2, 3, false>(p, c, &tmap_out);
        else if (p.scale) epilogue_loop<2, 1, true>(p, c, &tmap_out);
        else epilogue_loop<2, 1, false>(p, c, &tmap_out);
    }
    gemm_teardown<true>(tmem_base);
}

// ---- host side ------------------------------------------------------------------------------
using GemmKernel = void (*)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, KParams);

// the statistics epilogue (act 3, train-mode BatchNorm) lives in its own instantiations: it needs 17 more registers, which
// the inference kernels should not pay for
GemmKernel gemm_kernel(GemmKind kind, bool stats) {
    switch (kind) {
    case kGemm:
        if (stats) return conv_gemm_kernel<true>;
        return conv_gemm_kernel<false>;
    case kGemmPair:
        return conv_gemm_2cta_kernel;
    case kConv3x3:
        if (stats) return conv3x3_kernel<true>;
        return conv3x3_kernel<false>;
    case kConv3x3Pair:
        if (stats) return conv3x3_2cta_kernel<true>;
        return conv3x3_2cta_kernel<false>;
    case kDsam:
        break;
    }
    return dsam_fwd_kernel;
}

}  // namespace

extern "C" int rgbd_conv_gemm(const rgbd_conv_gemm_desc* d, rgbd_stream_t stream) {
    // ---- validate
    RGBD_CHECK_ARG(d, "conv_gemm: null descriptor");
    RGBD_CHECK_ARG(d->a && d->w && (d->slices || d->conv3x3_reuse || d->dsam_masked), "conv_gemm: null operand pointer");
    RGBD_CHECK_ARG(d->kb_elems == 64 || d->kb_elems == 32, "conv_gemm: kb_elems must be 64 or 32 (got %d)", d->kb_elems);
    RGBD_CHECK_ARG(d->a_c % 8 == 0 && d->a_c >= d->kb_elems, "conv_gemm: A channel count %d must be a multiple of 8 and >= kb", d->a_c);
    RGBD_CHECK_ARG(d->bx >= 1 && d->by >= 1 && d->bx * d->by == kBlockM && d->bx <= 256 && d->by <= 256,
                   "conv_gemm: box %dx%d must cover exactly %d pixels", d->bx, d->by, kBlockM);
    RGBD_CHECK_ARG(d->conv3x3_reuse || d->dsam_masked || (d->n_slices >= 1 && d->n_slices <= kMaxSlices), "conv_gemm: n_slices %d out of range",
                   d->n_slices);
    if (d->conv3x3_reuse)
        RGBD_CHECK_ARG(d->kb_elems == 64 && d->bx == kBlockM && d->by == 1 && d->a_c % 64 == 0 && d->plane_per_img == 1,
                       "conv_gemm: the 3x3 A-reuse path needs kb=64, a 128x1 box, C %% 64 == 0 and one plane per image");
    RGBD_CHECK_ARG(d->n_pad % 32 == 0 && d->block_n % 32 == 0 && d->block_n >= 32 && d->block_n <= 256 &&
                       d->n_pad % d->block_n == 0 && d->n <= d->n_pad && d->n >= 1,
                   "conv_gemm: bad N tiling (N=%d N_pad=%d BLOCK_N=%d)", d->n, d->n_pad, d->block_n);
    RGBD_CHECK_ARG(d->epi_mode >= 0 && d->epi_mode <= 3, "conv_gemm: bad epilogue mode %d", d->epi_mode);
    RGBD_CHECK_ARG(d->shift || d->epi_mode == 3, "conv_gemm: shift table is required");
    if (d->dsam_masked)
        RGBD_CHECK_ARG(d->epi_mode == 1 && d->kb_elems == 64 && d->a_c % 64 == 0 && d->plane_per_img == 4 && d->codes &&
                           d->m3_n_seg >= 2 && d->m3_n_seg <= 5 && d->m3_masked_segs == d->m3_n_seg - 1 && d->in_h >= 1 &&
                           d->in_w >= 1 && !d->conv3x3_reuse && (d->block_n / 2) % 16 == 0 &&
                           (long long)d->n_img * ceil_div(d->out_w, d->bx) * ceil_div(d->out_h, d->by) >= 2,
                       "conv_gemm: dsam_masked needs epilogue mode 1, kb=64, C %% 64 == 0, 4 parity planes, codes, "
                       "2..5 segments and at least two pixel tiles");
    if (d->next_operand)
        RGBD_CHECK_ARG(d->epi_mode == 1 && d->next_c_pad >= d->n && d->next_c_pad % 32 == 0 && d->next_n_seg >= 1 &&
                           d->next_n_seg <= 8 && d->next_masked_segs >= 0 && d->next_masked_segs <= 4 &&
                           d->next_masked_segs <= d->next_n_seg && (d->next_masked_segs == 0 || d->next_codes),
                       "conv_gemm: next_operand needs epilogue mode 1 and the next stage's packing geometry");
    if (d->epi_mode == 3)
        RGBD_CHECK_ARG(d->codes && d->m3_n_seg >= 1 && d->m3_n_seg <= 8 && d->block_n == 32 * d->m3_n_seg && d->in_h >= 1 &&
                           d->in_w >= 1 && (d->m3_stride == 1 || d->m3_stride == 2) && !d->conv3x3_reuse,
                       "conv_gemm: epilogue mode 3 needs codes, block_n == 32*n_seg and the dX geometry");
    RGBD_CHECK_ARG(d->n_img >= 1 && d->out_w >= 1 && d->out_h >= 1, "conv_gemm: bad output geometry");
    if (d->epi_mode == 2) {
        RGBD_CHECK_ARG(d->pool && d->cells_x >= 1 && d->cells_y >= 1, "conv_gemm: pool epilogue needs pool buffer and cells");
        RGBD_CHECK_ARG(d->out_w % d->cells_x == 0 && d->out_h % d->cells_y == 0,
                       "conv_gemm: fused average pooling needs H,W divisible by the %dx%d cell grid (got %dx%d)",
                       d->cells_y, d->cells_x, d->out_h, d->out_w);
        RGBD_CHECK_ARG(d->act == 1 || (d->act == 3 && d->pool_sq && !d->scale),
                       "conv_gemm: the pooled epilogue takes act 1 (ReLU) or act 3 (statistics: needs pool_sq, no scale)");
    } else {
        RGBD_CHECK_ARG(d->act != 3, "conv_gemm: act 3 (statistics) belongs to epilogue mode 2");
        RGBD_CHECK_ARG(d->out, "conv_gemm: null output");
    }
    if (d->epi_mode == 0)
        RGBD_CHECK_ARG(d->block_n % 64 == 0, "conv_gemm: the channels-last epilogue needs BLOCK_N %% 64 == 0 (got %d)", d->block_n);
    RGBD_CHECK_ARG(d->epi_mode == 0 || !d->gate, "conv_gemm: gate is only supported by epilogue mode 0");

    // ---- plan: kernel, buffers, stage count, grid
    const int kb_bytes = d->kb_elems * 2;
    KParams p;
    p.n_img = d->n_img;
    p.BX = d->bx; p.BY = d->by;
    p.out_w = d->out_w; p.out_h = d->out_h;
    p.tiles_x = ceil_div(d->out_w, d->bx);
    p.tiles_y = ceil_div(d->out_h, d->by);
    p.n_slices = (d->conv3x3_reuse || d->dsam_masked) ? 0 : d->n_slices;
    p.dsam_taps = 9;
    p.next_op = reinterpret_cast<__nv_bfloat16*>(d->next_operand);
    p.next_codes = reinterpret_cast<const uint8_t*>(d->next_codes);
    p.next_c_pad = d->next_c_pad; p.next_n_seg = d->next_n_seg; p.next_masked_segs = d->next_masked_segs;
    p.kb_bytes = kb_bytes;
    p.c_blocks = d->a_c / 64;
    p.N = d->n; p.N_pad = d->n_pad; p.BLOCK_N = d->block_n; p.n_tiles_n = d->n_pad / d->block_n;
    p.plane_per_img = d->plane_per_img;
    p.tile_order = d->tile_order;
    p.slices = reinterpret_cast<const int4*>(d->slices);
    p.epi_mode = d->epi_mode; p.act = d->act;
    p.scale = d->scale; p.shift = d->shift; p.variant = d->variant;
    p.gate = reinterpret_cast<const __nv_bfloat16*>(d->gate);
    p.out = d->out; p.residual = d->residual; p.pool = d->pool; p.pool_sq = d->pool_sq;
    p.cells_y = d->cells_y; p.cells_x = d->cells_x;
    p.codes = reinterpret_cast<const uint8_t*>(d->codes);
    p.in_h = d->in_h; p.in_w = d->in_w; p.m3_py = d->m3_py; p.m3_px = d->m3_px; p.m3_stride = d->m3_stride;
    p.m3_masked_segs = d->m3_masked_segs; p.m3_n_seg = d->m3_n_seg;
    const long long total = (long long)p.n_img * p.tiles_x * p.tiles_y * p.n_tiles_n;
    RGBD_CHECK_ARG(total < (1ll << 31), "conv_gemm: too many tiles");
    p.total_tiles = (int)total;
    const int total_m = p.total_tiles / p.n_tiles_n;
    p.b_resident = 0; p.b_res_bytes = 0;
    p.staging_bytes = d->epi_mode == 0 ? (p.BLOCK_N / 64) * kBlockM * 128 : 0;
    p.gate_bytes = (d->epi_mode == 0 && d->gate) ? p.staging_bytes : 0;
    p.sa_stages = 0; p.a_stage_bytes = 0;
    GemmKind kind;
    if (d->conv3x3_reuse) {
        p.gate_bytes = 0;                                 // the 3x3 kernels take no gate
        p.sa_stages = 3;
        p.a_stage_bytes = 17 * 1024;                      // (128+2) rows x 128 B, rounded up to the swizzle period
        const bool pair = d->epi_mode == 2 && p.n_tiles_n == 1 && p.BLOCK_N % 32 == 0 && (p.BLOCK_N / 2) % 8 == 0 && p.total_tiles >= 2;
        kind = pair ? kConv3x3Pair : kConv3x3;
    } else if (d->dsam_masked) {
        kind = kDsam;
    } else {
        const int b_total = p.n_slices * p.BLOCK_N * kb_bytes;
        p.b_resident = (p.n_tiles_n == 1 && b_total <= 100 * 1024) ? 1 : 0;
        p.b_res_bytes = p.b_resident ? b_total : 0;
        const bool pair = (d->epi_mode == 1 || d->epi_mode == 3) && !p.b_resident && total_m >= 2 && (p.BLOCK_N / 2) % 16 == 0;
        kind = pair ? kGemmPair : kGemm;
    }
    const bool pair = kind == kGemmPair || kind == kConv3x3Pair || kind == kDsam;
    const bool stats = d->epi_mode == 2 && d->act == 3;

    RgbdDeviceInfo di;
    if (int rc = rgbd_device_info(&di)) return rc;
    const int num_sms = di.num_sms, max_smem = di.max_smem;
    RGBD_ONCE_PER_DEVICE(di.device, {
        for (int k = kGemm; k <= kDsam; ++k)
            for (int st = 0; st < 2; ++st)
                RGBD_CHECK_CUDA(cudaFuncSetAttribute(gemm_kernel((GemmKind)k, st), cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
    });
    // dynamic shared memory: the layout, the alignment slack and 64 bytes
    p.stages = 0;
    const SmemLayout<size_t> fixed = smem_layout(kind, p, (size_t)0);
    p.stages = (max_smem - 1024 - (int)fixed.end - 64) / fixed.stage;
    if (p.stages > kMaxStages) p.stages = kMaxStages;
    RGBD_CHECK_ARG(p.stages >= 2, "conv_gemm: not enough shared memory for 2 pipeline stages");
    int smem_bytes = 1024 + (int)smem_layout(kind, p, (size_t)0).end + 64;
    // the slice-table kernels always take (almost) the whole SM so exactly one CTA (and its 512 TMEM columns) is resident
    if ((kind == kGemm || kind == kGemmPair) && smem_bytes < 160 * 1024) smem_bytes = 160 * 1024;
    int grid = p.total_tiles < num_sms ? p.total_tiles : num_sms;
    if (pair) {
        const int n_units = ((total_m + 1) / 2) * p.n_tiles_n;
        const int clusters = num_sms / 2 < n_units ? num_sms / 2 : n_units;
        grid = 2 * clusters;
    }

    // ---- encode the tensor maps
    const CUtensorMapSwizzle swz = kb_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    const long long a_px = 2ll * d->a_c, a_row = a_px * d->a_x;
    CUtensorMap tmap_a, tmap_b;
    if (int rc = encode_bf16_map(&tmap_a, "conv_gemm(A)", d->a, {d->a_c, d->a_x, d->a_y, d->a_planes}, {a_px, a_row, a_row * d->a_y},
                                 {d->kb_elems, d->conv3x3_reuse ? d->bx + 2 : d->bx, d->by, 1}, swz))
        return rc;
    // B: [N_pad][K], K-major; a CTA pair stages half of the BLOCK_N rows in each CTA
    const long long k_total = d->conv3x3_reuse ? 9ll * d->a_c
                              : d->dsam_masked ? 9ll * d->a_c * d->m3_n_seg : (long long)d->n_slices * d->kb_elems;
    if (int rc = encode_bf16_map(&tmap_b, "conv_gemm(B)", d->w, {k_total, d->n_pad}, {k_total * 2},
                                 {d->kb_elems, pair ? p.BLOCK_N / 2 : p.BLOCK_N}, swz))
        return rc;
    CUtensorMap tmap_out = tmap_a, tmap_gate = tmap_a;   // placeholders unless epilogue mode 0 uses them
    if (d->epi_mode == 0) {
        const long long o_px = 2ll * d->n_pad, o_row = o_px * d->out_w;
        if (int rc = encode_bf16_map(&tmap_out, "conv_gemm(out)", d->out, {d->n_pad, d->out_w, d->out_h, d->n_img},
                                     {o_px, o_row, o_row * d->out_h}, {64, d->bx, d->by, 1}, CU_TENSOR_MAP_SWIZZLE_128B))
            return rc;
        if (d->gate)
            if (int rc = encode_bf16_map(&tmap_gate, "conv_gemm(gate)", d->gate, {d->n_pad, d->out_w, d->out_h, d->n_img},
                                         {o_px, o_row, o_row * d->out_h}, {64, d->bx, d->by, 1}, CU_TENSOR_MAP_SWIZZLE_128B))
                return rc;
    }

    return launch_kernel(gemm_kernel(kind, stats), grid, kind == kDsam ? kDsamThreads : kThreads, smem_bytes, pair,
                         (cudaStream_t)stream, tmap_a, tmap_b, tmap_out, tmap_gate, p);
}
