// Swin window attention (inference), the inner op of the stock backbone that PRODUCES the hot path's input pyramid
// (reference call site mask2former/utils/custom_model.py:330 `self.encoder(rgb).feature_maps`; transformers
// SwinSelfAttention.forward): per (window, head)
//     out = softmax(q k^T / sqrt(d) + relative_position_bias[head] + shift_mask[window]) v          49 x 49 scores, d = 32
// The stock path runs it as bmm -> div -> add -> add -> softmax -> cast -> bmm -> permute-copy over a (windows*heads, 49, 49)
// score tensor (0.4 GB in fp32 at the first stage of a 32-frame batch): ~9 of the backbone's 35 ms.  Here one warp owns one
// (window, head): K and V are staged in shared memory as fp32, every lane owns one query row (two for rows >= 32) and runs an
// online softmax over 8-key chunks in registers; scores are never written.  58 GFLOP for the whole Swin-T at batch 32 -- CUDA-core
// work, bound by the FMA issue rate, not by memory.
#include "common.cuh"
#include "rgbd_b200.h"

namespace {

constexpr int kHd = 32;          // head dimension of every Swin variant (embed_dim / heads)
constexpr int kMaxN = 64;        // tokens per window (7 x 7 = 49; up to 8 x 8)
constexpr int kWarps = 4;

constexpr int kTabPitch = 64;    // floats per row of the additive table (256-byte rows: a quad's 8 bytes x 4 = one 32-byte sector)

// add[w][h][r][c] = bias[h][r][c] + mask[w][r][c] for c < N, -inf for the padded columns: the one additive term of the scores,
// laid out so that the score fragments' (row, 2 adjacent columns) reads are aligned 8-byte loads
__global__ void __launch_bounds__(256) window_attention_table_kernel(const float* __restrict__ bias, const float* __restrict__ mask,
                                                                    float* __restrict__ add, int nW, int heads, int N) {
    const long long n = (long long)nW * heads * N * kTabPitch;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int c = (int)(i % kTabPitch);
    const long long row = i / kTabPitch;
    const int r = (int)(row % N);
    const int h = (int)((row / N) % heads);
    const long long w = row / ((long long)N * heads);
    float x = -INFINITY;
    if (c < N) {
        x = bias[((size_t)h * N + r) * N + c];
        if (mask) x += mask[((size_t)w * N + r) * N + c];
    }
    add[i] = x;
}

struct Ld {
    static __device__ __forceinline__ void row(const float* p, float (&x)[kHd]) {
#pragma unroll
        for (int i = 0; i < kHd / 4; ++i) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(p) + i);
            x[4 * i] = v.x; x[4 * i + 1] = v.y; x[4 * i + 2] = v.z; x[4 * i + 3] = v.w;
        }
    }
    static __device__ __forceinline__ float one(const float* p) { return __ldg(p); }
    static __device__ __forceinline__ void store(float* p, const float (&x)[kHd]) {
#pragma unroll
        for (int i = 0; i < kHd / 4; ++i) reinterpret_cast<float4*>(p)[i] = make_float4(x[4 * i], x[4 * i + 1], x[4 * i + 2], x[4 * i + 3]);
    }
};

__global__ void __launch_bounds__(kWarps * 32) window_attention_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                                     const float* __restrict__ v, const float* __restrict__ add,
                                                                     float* __restrict__ out, long long n_units, int heads, int N,
                                                                     int nW, float sqrt_d) {
    extern __shared__ float s_kv[];                          // per warp: K [N][32], V [N][32] as fp32
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long unit = (long long)blockIdx.x * kWarps + warp;
    if (unit >= n_units) return;
    const long long win = unit / heads;                      // b_ = image * nW + window
    const int h = (int)(unit % heads);
    const int C = heads * kHd;
    float* sk = s_kv + (size_t)warp * 2 * N * kHd;
    float* sv = sk + N * kHd;
    const float* kb = k + (size_t)win * N * C + h * kHd;
    const float* vb = v + (size_t)win * N * C + h * kHd;
    for (int i = lane; i < N * kHd; i += 32) {
        const int j = i >> 5, d = i & 31;
        sk[i] = Ld::one(kb + (size_t)j * C + d);
        sv[i] = Ld::one(vb + (size_t)j * C + d);
    }
    __syncwarp();
    const float* add_wh = add + ((size_t)(win % nW) * heads + h) * N * kTabPitch;
    for (int r = lane; r < N; r += 32) {
        float qv[kHd], o[kHd];
        Ld::row(q + ((size_t)win * N + r) * C + h * kHd, qv);
#pragma unroll
        for (int d = 0; d < kHd; ++d) o[d] = 0.f;
        float m = -INFINITY, l = 0.f;
        const float* arow = add_wh + (size_t)r * kTabPitch;
        for (int j0 = 0; j0 < N; j0 += 8) {
            float s[8];
            float cmax = -INFINITY;
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
                const int j = j0 + jj;
                s[jj] = -INFINITY;
                if (j < N) {
                    const float4* kr = reinterpret_cast<const float4*>(sk + j * kHd);
                    float acc = 0.f;
#pragma unroll
                    for (int d4 = 0; d4 < kHd / 4; ++d4) {
                        const float4 kk = kr[d4];
                        acc = fmaf(qv[4 * d4], kk.x, acc);
                        acc = fmaf(qv[4 * d4 + 1], kk.y, acc);
                        acc = fmaf(qv[4 * d4 + 2], kk.z, acc);
                        acc = fmaf(qv[4 * d4 + 3], kk.w, acc);
                    }
                    const float sc = acc / sqrt_d + __ldg(arow + j);
                    s[jj] = sc;
                    cmax = fmaxf(cmax, sc);
                }
            }
            const float m_new = fmaxf(m, cmax);
            const float corr = __expf(m - m_new);              // 0 on the first chunk (m = -inf)
            l *= corr;
#pragma unroll
            for (int d = 0; d < kHd; ++d) o[d] *= corr;
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
                const int j = j0 + jj;
                if (j < N) {
                    const float p = __expf(s[jj] - m_new);
                    l += p;
                    const float4* vr = reinterpret_cast<const float4*>(sv + j * kHd);
#pragma unroll
                    for (int d4 = 0; d4 < kHd / 4; ++d4) {
                        const float4 vv = vr[d4];
                        o[4 * d4] = fmaf(p, vv.x, o[4 * d4]);
                        o[4 * d4 + 1] = fmaf(p, vv.y, o[4 * d4 + 1]);
                        o[4 * d4 + 2] = fmaf(p, vv.z, o[4 * d4 + 2]);
                        o[4 * d4 + 3] = fmaf(p, vv.w, o[4 * d4 + 3]);
                    }
                }
            }
            m = m_new;
        }
        const float inv = 1.0f / l;
#pragma unroll
        for (int d = 0; d < kHd; ++d) o[d] *= inv;
        Ld::store(out + ((size_t)win * N + r) * C + h * kHd, o);
    }
}

// ---- bf16 inputs: warp-level tensor-core path (mma.sync m16n8k16, the FlashAttention-2 register choreography) ----------
// The CUDA-core kernel above re-reads K and V from shared memory once per query row (1 568 LDS.128 per (window, head)): it is
// bound by the LSU issue rate at ~10 TFLOP/s (1.18 ms for the first Swin-T stage of a 32-frame batch).  Here a warp stages K and V
// as bf16 (rows padded to 80 bytes: conflict-free ldmatrix), and per 16-row tile of queries runs S = Q K^T (16 MMAs, fp32
// accumulators), adds bias + shift mask, takes the softmax over the <= 64 keys in registers (a row lives in the four lanes of a
// quad: two shuffles per reduction), repacks P as the A operand and runs O = P V (16 MMAs).  This is 49 x 49 x 32 work per unit:
// far too small for a tcgen05 / TMEM pipeline (M = 128 tiles, one issuing thread), which is why it stays on mma.sync.
constexpr int kPitch = 40;                                   // bf16 elements per staged row (80 bytes)

__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const void* p) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t (&r)[4], const void* p) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
    const __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&t);
}

__global__ void __launch_bounds__(kWarps * 32) window_attention_mma_kernel(const __nv_bfloat16* __restrict__ q,
                                                                          const __nv_bfloat16* __restrict__ k,
                                                                          const __nv_bfloat16* __restrict__ v,
                                                                          const float* __restrict__ add_tab,
                                                                          __nv_bfloat16* __restrict__ out, long long n_units, int heads,
                                                                          int N, int nW, float sqrt_d) {
    __shared__ __align__(16) __nv_bfloat16 s_all[kWarps][2][kMaxN * kPitch];     // K, V per warp: 2 x 5 KB (Q fragments come straight from global)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    long long unit = (long long)blockIdx.x * kWarps + warp;
    if (unit >= n_units) return;                             // whole warps leave together
    const long long win = unit / heads;
    const int h = (int)(unit % heads);
    const int C = heads * kHd;
    __nv_bfloat16* sk = s_all[warp][0];
    __nv_bfloat16* sv = s_all[warp][1];
    const size_t base = (size_t)win * N * C + h * kHd;
    for (int i = lane; i < kMaxN * 4; i += 32) {            // 64 rows x four 16-byte pieces per tensor; rows >= N are zero
        const int r = i >> 2, piece = i & 3;
        uint4 b = make_uint4(0u, 0u, 0u, 0u), c = b;
        if (r < N) {
            const size_t o = base + (size_t)r * C + piece * 8;
            b = __ldg(reinterpret_cast<const uint4*>(k + o));
            c = __ldg(reinterpret_cast<const uint4*>(v + o));
        }
        *reinterpret_cast<uint4*>(sk + r * kPitch + piece * 8) = b;
        *reinterpret_cast<uint4*>(sv + r * kPitch + piece * 8) = c;
    }
    __syncwarp();
    const int g = lane >> 2, t = lane & 3;
    const float* add_wh = add_tab + ((size_t)(win % nW) * heads + h) * N * kTabPitch;
    const int n_mt = (N + 15) >> 4, n_nt = (N + 7) >> 3;      // 16-row query tiles, 8-key tiles actually needed
    const int n_kk = (N + 15) >> 4;                           // 16-key steps of P V
    // ldmatrix source rows for this lane: A operand (x4: rows 0-7 / 8-15 at k 0-7, then at k 8-15), B operand from K ([key][d]:
    // x4 = one 8-key tile at d 0-7 / 8-15 / 16-23 / 24-31), B operand from V ([key][d], transposed: x4 = keys 0-7 / 8-15 at
    // d 0-7, then at d 8-15)
    const int kb_row = lane & 7, kb_col = (lane >> 3) * 8;
    const int vb_row = (lane & 7) + ((lane >> 3) & 1) * 8, vb_col = (lane >> 4) * 8;
    const float inv_sqrt_d = 1.0f / sqrt_d;
    // A fragments of Q straight from global: a0 = (row g, d 2t..), a1 = (row g + 8, same), a2 / a3 = the same rows at d + 8
    auto load_q = [&](int mt, uint32_t (&qa)[2][4]) {
        const int qr0 = mt * 16 + g, qr1 = qr0 + 8;
        const uint32_t* p0 = reinterpret_cast<const uint32_t*>(q + base + (size_t)qr0 * C) + t;
        const uint32_t* p1 = reinterpret_cast<const uint32_t*>(q + base + (size_t)qr1 * C) + t;
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            qa[ks][0] = qr0 < N ? __ldg(p0 + ks * 8) : 0u;
            qa[ks][1] = qr1 < N ? __ldg(p1 + ks * 8) : 0u;
            qa[ks][2] = qr0 < N ? __ldg(p0 + ks * 8 + 4) : 0u;
            qa[ks][3] = qr1 < N ? __ldg(p1 + ks * 8 + 4) : 0u;
        }
    };
    uint32_t qa[2][4], qn[2][4];
    load_q(0, qa);
    for (int mt = 0; mt < n_mt; ++mt) {
        // everything this tile reads from global is requested BEFORE its MMAs: the additive term (bias + shift mask, -inf for
        // padded keys / rows; one aligned 8-byte load per row and key tile from the padded table) of the 32 score elements this lane owns, and the next tile's Q fragments
        const int r0 = mt * 16 + g, r1 = r0 + 8;
        const bool ok0 = r0 < N, ok1 = r1 < N;
        float add[8][4];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            float2 a0 = make_float2(-INFINITY, -INFINITY), a1 = a0;
            if (ok0) a0 = __ldg(reinterpret_cast<const float2*>(add_wh + r0 * kTabPitch + nt * 8 + 2 * t));
            if (ok1) a1 = __ldg(reinterpret_cast<const float2*>(add_wh + r1 * kTabPitch + nt * 8 + 2 * t));
            add[nt][0] = a0.x; add[nt][1] = a0.y; add[nt][2] = a1.x; add[nt][3] = a1.y;
        }
        if (mt + 1 < n_mt) load_q(mt + 1, qn);
        float sc[8][4];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
            if (nt < n_nt) {
                uint32_t kb[4];
                ldsm_x4(kb, sk + (nt * 8 + kb_row) * kPitch + kb_col);
                mma_bf16(sc[nt], qa[0], kb[0], kb[1]);
                mma_bf16(sc[nt], qa[1], kb[2], kb[3]);
            }
        }
        // scores of rows r0 = 16 mt + g and r1 = r0 + 8, columns 8 nt + 2 t + {0, 1}
        float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
            for (int e = 0; e < 4; ++e) sc[nt][e] = fmaf(sc[nt][e], inv_sqrt_d, add[nt][e]);
            mx0 = fmaxf(mx0, fmaxf(sc[nt][0], sc[nt][1]));
            mx1 = fmaxf(mx1, fmaxf(sc[nt][2], sc[nt][3]));
        }
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
        if (!ok0) mx0 = 0.f;                                   // padded rows: exp(-inf - 0) = 0 everywhere, never stored
        if (!ok1) mx1 = 0.f;
        float l0 = 0.f, l1 = 0.f;
        uint32_t pa[4][4];                                     // P as A operand: 16 rows x 16 keys per kk
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const float p00 = __expf(sc[nt][0] - mx0), p01 = __expf(sc[nt][1] - mx0);
            const float p10 = __expf(sc[nt][2] - mx1), p11 = __expf(sc[nt][3] - mx1);
            l0 += p00 + p01;
            l1 += p10 + p11;
            pa[nt >> 1][(nt & 1) * 2] = pack2(p00, p01);
            pa[nt >> 1][(nt & 1) * 2 + 1] = pack2(p10, p11);
        }
        l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
        l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
        l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
        l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
        float oc[4][4];
#pragma unroll
        for (int dt = 0; dt < 4; ++dt) oc[dt][0] = oc[dt][1] = oc[dt][2] = oc[dt][3] = 0.f;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            if (kk < n_kk) {
#pragma unroll
                for (int dp = 0; dp < 2; ++dp) {               // two 8-wide d tiles per ldmatrix.x4.trans
                    uint32_t vb[4];
                    ldsm_x4_trans(vb, sv + (kk * 16 + vb_row) * kPitch + dp * 16 + vb_col);
                    mma_bf16(oc[2 * dp], pa[kk], vb[0], vb[1]);
                    mma_bf16(oc[2 * dp + 1], pa[kk], vb[2], vb[3]);
                }
            }
        }
        const float i0 = ok0 ? 1.0f / l0 : 0.f, i1 = ok1 ? 1.0f / l1 : 0.f;
#pragma unroll
        for (int dt = 0; dt < 4; ++dt) {
            const int c = dt * 8 + 2 * t;
            if (ok0) *reinterpret_cast<uint32_t*>(out + base + (size_t)r0 * C + c) = pack2(oc[dt][0] * i0, oc[dt][1] * i0);
            if (ok1) *reinterpret_cast<uint32_t*>(out + base + (size_t)r1 * C + c) = pack2(oc[dt][2] * i1, oc[dt][3] * i1);
        }
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
#pragma unroll
            for (int e = 0; e < 4; ++e) qa[ks][e] = qn[ks][e];
    }
}

// ---- masked cross-attention of the Mask2Former transformer decoder (inference, bf16) -----------------------------------------
// nn.MultiheadAttention.forward as transformers' Mask2FormerMaskedAttentionDecoderLayer calls it (the consumer of the pixel
// decoder's multi-scale features behind CM:383): 100 queries attend to the S = 300 / 1 200 / 4 800 pixels of one feature level
// under a BOOLEAN mask (True = may not attend; the mask rgbd_attention_mask writes).  The stock path materialises an additive
// -inf mask, the (batch*heads, 100, S) score tensor in float32 (0.5 GB at S = 4 800), its softmax and a bf16 copy: ~1.7 ms per
// layer at the finest level.  Here one CTA owns one (image, head): four warps x 32 query rows, the keys stream through shared
// memory in tiles of 64 (register prefetch of the next tile), FlashAttention-2 online softmax with the mask bytes read in the
// score fragments' own layout (two adjacent keys = one 2-byte load).
constexpr int kKeyTile = 64;

__global__ void __launch_bounds__(128) masked_cross_attention_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ k,
                                                                    const __nv_bfloat16* __restrict__ v, const uint8_t* __restrict__ mask,
                                                                    __nv_bfloat16* __restrict__ out, int B, int H, int L, int S,
                                                                    float scale) {
    __shared__ __align__(16) __nv_bfloat16 s_k[kKeyTile * kPitch];
    __shared__ __align__(16) __nv_bfloat16 s_v[kKeyTile * kPitch];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int bh = blockIdx.x, b = bh / H, h = bh % H;
    const int E = H * kHd;
    const int row_base = blockIdx.y * 128 + warp * 32;        // this warp's 32 query rows (two 16-row tiles)
    const int g = lane >> 2, t = lane & 3;
    const size_t tok = (size_t)B * E;                          // elements between consecutive tokens of (len, batch, embed) tensors
    const size_t col0 = (size_t)b * E + h * kHd;

    uint32_t qa[2][2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
        const int r0 = row_base + mt * 16 + g, r1 = r0 + 8;
        const uint32_t* p0 = reinterpret_cast<const uint32_t*>(q + (size_t)r0 * tok + col0) + t;
        const uint32_t* p1 = reinterpret_cast<const uint32_t*>(q + (size_t)r1 * tok + col0) + t;
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            qa[mt][ks][0] = r0 < L ? __ldg(p0 + ks * 8) : 0u;
            qa[mt][ks][1] = r1 < L ? __ldg(p1 + ks * 8) : 0u;
            qa[mt][ks][2] = r0 < L ? __ldg(p0 + ks * 8 + 4) : 0u;
            qa[mt][ks][3] = r1 < L ? __ldg(p1 + ks * 8 + 4) : 0u;
        }
    }
    float oc[2][4][4];
    float m_run[2][2], l_run[2][2];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
        m_run[mt][0] = m_run[mt][1] = -INFINITY;
        l_run[mt][0] = l_run[mt][1] = 0.f;
#pragma unroll
        for (int dt = 0; dt < 4; ++dt) oc[mt][dt][0] = oc[mt][dt][1] = oc[mt][dt][2] = oc[mt][dt][3] = 0.f;
    }
    // staging: 64 keys x four 16-byte pieces per tensor = 256 pieces, two per thread and tensor
    const int st_row = threadIdx.x >> 1, st_piece = (threadIdx.x & 1) * 2;
    uint4 pk[2], pv[2];
    auto fetch = [&](int key0) {
        const int key = key0 + st_row;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            pk[i] = make_uint4(0u, 0u, 0u, 0u);
            pv[i] = pk[i];
            if (key < S) {
                const size_t o = (size_t)key * tok + col0 + (st_piece + i) * 8;
                pk[i] = __ldg(reinterpret_cast<const uint4*>(k + o));
                pv[i] = __ldg(reinterpret_cast<const uint4*>(v + o));
            }
        }
    };
    const int kb_row = lane & 7, kb_col = (lane >> 3) * 8;
    const int vb_row = (lane & 7) + ((lane >> 3) & 1) * 8, vb_col = (lane >> 4) * 8;
    const uint8_t* mask_bh = mask + (size_t)bh * L * S;
    const int n_tiles = (S + kKeyTile - 1) / kKeyTile;
    fetch(0);
    for (int kt = 0; kt < n_tiles; ++kt) {
        __syncthreads();                                       // everyone is done reading the previous tile
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            *reinterpret_cast<uint4*>(s_k + st_row * kPitch + (st_piece + i) * 8) = pk[i];
            *reinterpret_cast<uint4*>(s_v + st_row * kPitch + (st_piece + i) * 8) = pv[i];
        }
        __syncthreads();
        if (kt + 1 < n_tiles) fetch((kt + 1) * kKeyTile);      // in flight while this tile is computed
        const int key0 = kt * kKeyTile;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
            const int r0 = row_base + mt * 16 + g, r1 = r0 + 8;
            // mask bytes of this lane's score elements: (row, keys key0 + 8 nt + 2 t + {0, 1}) = one 2-byte load
            uint32_t mk[8];
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                const int c = key0 + nt * 8 + 2 * t;
                uint32_t m0 = 0x0101u, m1 = 0x0101u;          // out of range = masked
                if (c < S) {                                   // S is even (checked on the host): c + 1 < S as well
                    if (r0 < L) m0 = __ldg(reinterpret_cast<const unsigned short*>(mask_bh + (size_t)r0 * S + c));
                    if (r1 < L) m1 = __ldg(reinterpret_cast<const unsigned short*>(mask_bh + (size_t)r1 * S + c));
                }
                mk[nt] = m0 | (m1 << 16);
            }
            float sc[8][4];
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
                uint32_t kb[4];
                ldsm_x4(kb, s_k + (nt * 8 + kb_row) * kPitch + kb_col);
                mma_bf16(sc[nt], qa[mt][0], kb[0], kb[1]);
                mma_bf16(sc[nt], qa[mt][1], kb[2], kb[3]);
            }
            float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                sc[nt][0] = (mk[nt] & 0x000000ffu) ? -INFINITY : sc[nt][0] * scale;
                sc[nt][1] = (mk[nt] & 0x0000ff00u) ? -INFINITY : sc[nt][1] * scale;
                sc[nt][2] = (mk[nt] & 0x00ff0000u) ? -INFINITY : sc[nt][2] * scale;
                sc[nt][3] = (mk[nt] & 0xff000000u) ? -INFINITY : sc[nt][3] * scale;
                mx0 = fmaxf(mx0, fmaxf(sc[nt][0], sc[nt][1]));
                mx1 = fmaxf(mx1, fmaxf(sc[nt][2], sc[nt][3]));
            }
            mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
            mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
            mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
            mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
            const float mn0 = fmaxf(m_run[mt][0], mx0), mn1 = fmaxf(m_run[mt][1], mx1);
            const float ms0 = mn0 == -INFINITY ? 0.f : mn0, ms1 = mn1 == -INFINITY ? 0.f : mn1;   // all keys masked so far
            const float c0 = __expf(m_run[mt][0] - ms0), c1 = __expf(m_run[mt][1] - ms1);
            m_run[mt][0] = mn0;
            m_run[mt][1] = mn1;
            float l0 = 0.f, l1 = 0.f;
            uint32_t pa[4][4];
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                const float p00 = __expf(sc[nt][0] - ms0), p01 = __expf(sc[nt][1] - ms0);
                const float p10 = __expf(sc[nt][2] - ms1), p11 = __expf(sc[nt][3] - ms1);
                l0 += p00 + p01;
                l1 += p10 + p11;
                pa[nt >> 1][(nt & 1) * 2] = pack2(p00, p01);
                pa[nt >> 1][(nt & 1) * 2 + 1] = pack2(p10, p11);
            }
            l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
            l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
            l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
            l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
            l_run[mt][0] = l_run[mt][0] * c0 + l0;
            l_run[mt][1] = l_run[mt][1] * c1 + l1;
#pragma unroll
            for (int dt = 0; dt < 4; ++dt) {
                oc[mt][dt][0] *= c0; oc[mt][dt][1] *= c0;
                oc[mt][dt][2] *= c1; oc[mt][dt][3] *= c1;
            }
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
                for (int dp = 0; dp < 2; ++dp) {
                    uint32_t vb[4];
                    ldsm_x4_trans(vb, s_v + (kk * 16 + vb_row) * kPitch + dp * 16 + vb_col);
                    mma_bf16(oc[mt][2 * dp], pa[kk], vb[0], vb[1]);
                    mma_bf16(oc[mt][2 * dp + 1], pa[kk], vb[2], vb[3]);
                }
            }
        }
    }
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
        const int r0 = row_base + mt * 16 + g, r1 = r0 + 8;
        const float i0 = l_run[mt][0] > 0.f ? 1.0f / l_run[mt][0] : 0.f, i1 = l_run[mt][1] > 0.f ? 1.0f / l_run[mt][1] : 0.f;
#pragma unroll
        for (int dt = 0; dt < 4; ++dt) {
            const int c = dt * 8 + 2 * t;
            if (r0 < L) *reinterpret_cast<uint32_t*>(out + (size_t)r0 * tok + col0 + c) = pack2(oc[mt][dt][0] * i0, oc[mt][dt][1] * i0);
            if (r1 < L) *reinterpret_cast<uint32_t*>(out + (size_t)r1 * tok + col0 + c) = pack2(oc[mt][dt][2] * i1, oc[mt][dt][3] * i1);
        }
    }
}

}  // namespace

extern "C" size_t rgbd_window_attention_workspace_bytes(int N, int heads, int n_mask_windows) {
    if (N < 1 || heads < 1) return 0;
    return (size_t)(n_mask_windows > 0 ? n_mask_windows : 1) * heads * N * kTabPitch * sizeof(float);
}

extern "C" int rgbd_window_attention(const void* q, const void* k, const void* v, int dtype, const float* bias, const float* mask,
                                     void* out, long long n_windows, int N, int heads, int head_dim, int n_mask_windows,
                                     void* workspace, rgbd_stream_t stream) {
    RGBD_CHECK_ARG(q && k && v && bias && out && workspace, "window_attention: null pointer");
    RGBD_CHECK_ARG(dtype == RGBD_DTYPE_F32 || dtype == RGBD_DTYPE_BF16, "window_attention: q / k / v are f32 or bf16");
    RGBD_CHECK_ARG(head_dim == kHd, "window_attention: head dimension must be %d (got %d)", kHd, head_dim);
    RGBD_CHECK_ARG(N >= 1 && N <= kMaxN, "window_attention: 1..%d tokens per window (got %d)", kMaxN, N);
    RGBD_CHECK_ARG(n_windows >= 1 && heads >= 1, "window_attention: bad sizes");
    RGBD_CHECK_ARG(!mask || (n_mask_windows >= 1 && n_windows % n_mask_windows == 0),
                   "window_attention: the window count must be a multiple of the mask's window count");
    const int nW = mask ? n_mask_windows : 1;
    const long long n_units = n_windows * heads;
    const long long blocks = (n_units + kWarps - 1) / kWarps;
    RGBD_CHECK_ARG(blocks <= 0x7fffffffLL, "window_attention: too many windows");
    const size_t smem = (size_t)kWarps * 2 * N * kHd * sizeof(float);
    RgbdDeviceInfo di;
    if (int rc = rgbd_device_info(&di)) return rc;
    RGBD_ONCE_PER_DEVICE(di.device, {
        RGBD_CHECK_CUDA(cudaFuncSetAttribute(window_attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             kWarps * 2 * kMaxN * kHd * (int)sizeof(float)));
    });
    cudaStream_t s = (cudaStream_t)stream;
    float* add = reinterpret_cast<float*>(workspace);
    const long long n_tab = (long long)nW * heads * N * kTabPitch;
    window_attention_table_kernel<<<(unsigned)((n_tab + 255) / 256), 256, 0, s>>>(bias, mask, add, nW, heads, N);
    RGBD_CHECK_LAUNCH();
    const float sqrt_d = sqrtf((float)head_dim);
    if (dtype == RGBD_DTYPE_BF16)
        window_attention_mma_kernel<<<(unsigned)blocks, kWarps * 32, 0, s>>>(
            (const __nv_bfloat16*)q, (const __nv_bfloat16*)k, (const __nv_bfloat16*)v, add, (__nv_bfloat16*)out, n_units, heads, N, nW, sqrt_d);
    else
        window_attention_kernel<<<(unsigned)blocks, kWarps * 32, smem, s>>>((const float*)q, (const float*)k, (const float*)v, add,
                                                                                  (float*)out, n_units, heads, N, nW, sqrt_d);
    RGBD_CHECK_LAUNCH();
    return RGBD_OK;
}

extern "C" int rgbd_masked_cross_attention(const void* q_bf16, const void* k_bf16, const void* v_bf16, const uint8_t* mask, void* out_bf16,
                                           int B, int heads, int L, int S, int head_dim, rgbd_stream_t stream) {
    RGBD_CHECK_ARG(q_bf16 && k_bf16 && v_bf16 && mask && out_bf16, "masked_cross_attention: null pointer");
    RGBD_CHECK_ARG(head_dim == kHd, "masked_cross_attention: head dimension must be %d (got %d)", kHd, head_dim);
    RGBD_CHECK_ARG(B >= 1 && heads >= 1 && L >= 1 && S >= 2 && S % 2 == 0, "masked_cross_attention: S must be even, sizes positive");
    RGBD_CHECK_ARG((long long)B * heads <= 0x7fffffffLL && (L + 127) / 128 <= 65535, "masked_cross_attention: too many CTAs");
    masked_cross_attention_kernel<<<dim3((unsigned)(B * heads), (unsigned)((L + 127) / 128)), 128, 0, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)q_bf16, (const __nv_bfloat16*)k_bf16, (const __nv_bfloat16*)v_bf16, mask, (__nv_bfloat16*)out_bf16, B, heads, L, S,
        1.0f / sqrtf((float)head_dim));
    RGBD_CHECK_LAUNCH();
    return RGBD_OK;
}
