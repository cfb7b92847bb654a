// K5: instance post-processing on the device (SURVEY 8f-3).  Replaces the HuggingFace routine the reference calls on the
// model outputs, `image_processor.post_process_instance_segmentation(outputs, threshold, target_sizes,
// return_binary_maps=True)` (reference mask2former/utils/model_essential_part.py:86-91, mask2former/predictor.py:34-36,
// 701-703), for a batch of same-sized images and without a host round trip per query:
//   1. postproc_select_kernel   softmax over the classes, top-Q of the Q*C (query, label) scores (bitonic sort in
//                               shared memory; defined order: score descending, flat index ascending on ties)
//   2. postproc_grid_kernel     per candidate: bilinear 384x384 upsample of its mask logits evaluated on the fly in
//                               separable form (torch's align_corners=False source-index arithmetic, operation for
//                               operation), pixel count of (logit > 0), sum of sigmoid over those pixels (deterministic
//                               two-level sum) and the SIGN BITMAP of the grid (18 KB per candidate);
//      postproc_stats_kernel    point-wise fallback for very tall logit planes, and the non-emptiness of the
//                               nearest-resized target mask when the target is smaller than the grid
//   3. postproc_finalize_kernel mask score = sum / (count + 1e-6), score = class score * mask score, keep rule
//                               (non-empty and score >= threshold), compact slots in candidate order
//   4. postproc_paint_kernel    binary masks of the kept segments at the target size (nearest sample of the 384 grid's sign
//                               bitmap written by pass 2), and the painted segmentation map (id of the last kept segment
//                               covering a pixel)
// The 384x384 upsampled logits (59 MB per image for 100 queries) are never materialised.
// rgbd_label_map_rle: run-length encoding of the painted map (HF `return_coco_annotation=True`) in four sync-free passes.
// rgbd_instance_rle: pycocotools' compressed RLE string of every kept segment, from the same encoder run on the transposed
// map, then a size, scan, base and emit pass over the runs; no host synchronisation either.
// rgbd_mask_iou: pairwise mask IoU (the evaluator's torchmetrics `iou_type="segm"` core) with 16-byte loads + popcount.
// Compiled with -fmad=false: the interpolation is written as separate multiplies and adds like ATen's kernel.
#include "common.cuh"
#include "rgbd_b200.h"

namespace {

constexpr int kGrid = 384;          // HF: "Scale back to preprocessed image size - (384, 384) for all models"
constexpr int kChunk = 4096;        // grid points per CTA in the stats pass
static_assert((kGrid * kGrid) % kChunk == 0 && kChunk % 256 == 0, "whole chunks, whole warps");
constexpr int kMaxSort = 8192;      // Q*C candidates sorted in shared memory

struct PostGeom {
    int B, Q, C1, h, w, Ht, Wt;
    float rh, rw;                   // h / 384, w / 384          (torch: area_pixel_compute_scale)
    float sy, sx;                   // 384 / Ht, 384 / Wt        (nearest: floor(dst * scale))
};

// value of the bilinearly upsampled (384 x 384, align_corners=False) logit plane at grid point (gy, gx)
__device__ __forceinline__ float grid_logit(const float* __restrict__ plane, const PostGeom& g, int gy, int gx) {
    float fy = __fsub_rn(__fmul_rn(g.rh, __fadd_rn((float)gy, 0.5f)), 0.5f);
    float fx = __fsub_rn(__fmul_rn(g.rw, __fadd_rn((float)gx, 0.5f)), 0.5f);
    fy = fy < 0.f ? 0.f : fy;
    fx = fx < 0.f ? 0.f : fx;
    const int y0 = (int)fy, x0 = (int)fx;
    const int y1 = y0 + (y0 < g.h - 1 ? 1 : 0), x1 = x0 + (x0 < g.w - 1 ? 1 : 0);
    const float ly1 = __fsub_rn(fy, (float)y0), ly0 = __fsub_rn(1.f, ly1);
    const float lx1 = __fsub_rn(fx, (float)x0), lx0 = __fsub_rn(1.f, lx1);
    const float v00 = __ldg(plane + (size_t)y0 * g.w + x0), v01 = __ldg(plane + (size_t)y0 * g.w + x1);
    const float v10 = __ldg(plane + (size_t)y1 * g.w + x0), v11 = __ldg(plane + (size_t)y1 * g.w + x1);
    const float top = __fadd_rn(__fmul_rn(lx0, v00), __fmul_rn(lx1, v01));
    const float bot = __fadd_rn(__fmul_rn(lx0, v10), __fmul_rn(lx1, v11));
    return __fadd_rn(__fmul_rn(ly0, top), __fmul_rn(ly1, bot));
}

// target pixel -> grid point (torch "nearest": min(floor(dst * scale), in - 1))
__device__ __forceinline__ int nearest_src(int dst, float scale) {
    const int s = (int)floorf(__fmul_rn((float)dst, scale));
    return s < kGrid - 1 ? s : kGrid - 1;
}

__global__ void __launch_bounds__(256) postproc_select_kernel(const float* __restrict__ cls, PostGeom g, int n_sort,
                                                              float* __restrict__ sel_score, int* __restrict__ sel_query,
                                                              int* __restrict__ sel_label) {
    extern __shared__ unsigned long long keys[];
    const int b = blockIdx.x, C = g.C1 - 1;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int i = threadIdx.x; i < n_sort; i += blockDim.x) keys[i] = 0ull;
    __syncthreads();
    for (int q = warp; q < g.Q; q += nw) {
        const float* row = cls + ((size_t)b * g.Q + q) * g.C1;
        float mx = -INFINITY;
        for (int c = lane; c < g.C1; c += 32) mx = fmaxf(mx, row[c]);
#pragma unroll
        for (int k = 16; k > 0; k >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, k));
        float sum = 0.f;
        for (int c = lane; c < g.C1; c += 32) sum += expf(row[c] - mx);
#pragma unroll
        for (int k = 16; k > 0; k >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, k);
        for (int c = lane; c < C; c += 32) {
            const float p = expf(row[c] - mx) / sum;
            const unsigned flat = (unsigned)(q * C + c);
            keys[flat] = ((unsigned long long)__float_as_uint(p) << 32) | (unsigned long long)(0xFFFFFFFFu - flat);
        }
    }
    __syncthreads();
    // bitonic sort, descending
    for (int k = 2; k <= n_sort; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n_sort; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned long long a = keys[i], c2 = keys[ixj];
                    const bool desc = (i & k) == 0;
                    if (desc ? a < c2 : a > c2) {
                        keys[i] = c2;
                        keys[ixj] = a;
                    }
                }
            }
            __syncthreads();
        }
    }
    for (int j = threadIdx.x; j < g.Q; j += blockDim.x) {
        const unsigned long long kk = keys[j];
        const unsigned flat = 0xFFFFFFFFu - (unsigned)(kk & 0xFFFFFFFFull);
        sel_score[(size_t)b * g.Q + j] = __uint_as_float((unsigned)(kk >> 32));
        sel_query[(size_t)b * g.Q + j] = (int)(flat / (unsigned)C);
        sel_label[(size_t)b * g.Q + j] = (int)(flat % (unsigned)C);
    }
}

// blockIdx.x < n_chunk_grid: statistics over a chunk of the 384x384 grid; the remaining blocks: any(mask) over a chunk of
// the target pixels
__global__ void __launch_bounds__(256) postproc_stats_kernel(const float* __restrict__ masks, PostGeom g,
                                                             const int* __restrict__ sel_query, int n_chunk_grid,
                                                             unsigned* __restrict__ part_cnt, float* __restrict__ part_sum,
                                                             unsigned* __restrict__ any_target, unsigned* __restrict__ bitmap) {
    const int j = blockIdx.y, b = blockIdx.z;
    const int q = sel_query[(size_t)b * g.Q + j];
    const float* plane = masks + ((size_t)b * g.Q + q) * g.h * g.w;
    __shared__ unsigned s_cnt[8];
    __shared__ float s_sum[8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if ((int)blockIdx.x < n_chunk_grid) {
        unsigned cnt = 0;
        float sum = 0.f;
        const int base = blockIdx.x * kChunk;
        for (int i = threadIdx.x; i < kChunk; i += blockDim.x) {
            const int pt = base + i;                        // kGrid^2 is a multiple of kChunk: no partial chunk, warps stay whole
            const float v = grid_logit(plane, g, pt / kGrid, pt % kGrid);
            if (v > 0.f) {
                ++cnt;
                sum += 1.0f / (1.0f + expf(-v));
            }
            if (bitmap) {                                   // 32 consecutive grid points per warp -> one word of the sign bitmap
                const unsigned word = __ballot_sync(0xffffffffu, v > 0.f);
                if (lane == 0) bitmap[((size_t)b * g.Q + j) * (kGrid * (kGrid / 32)) + (pt >> 5)] = word;
            }
        }
#pragma unroll
        for (int k = 16; k > 0; k >>= 1) {
            cnt += __shfl_xor_sync(0xffffffffu, cnt, k);
            sum += __shfl_xor_sync(0xffffffffu, sum, k);
        }
        if (lane == 0) {
            s_cnt[warp] = cnt;
            s_sum[warp] = sum;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned c = 0;
            float s = 0.f;
            for (int k = 0; k < 8; ++k) {
                c += s_cnt[k];
                s += s_sum[k];
            }
            const size_t o = ((size_t)b * g.Q + j) * n_chunk_grid + blockIdx.x;
            part_cnt[o] = c;
            part_sum[o] = s;
        }
    } else {
        const int base = ((int)blockIdx.x - n_chunk_grid) * kChunk;
        const int n_t = g.Ht * g.Wt;
        bool any = false;
        for (int i = threadIdx.x; i < kChunk; i += blockDim.x) {
            const int pt = base + i;
            if (pt >= n_t) break;
            const float v = grid_logit(plane, g, nearest_src(pt / g.Wt, g.sy), nearest_src(pt % g.Wt, g.sx));
            any |= v > 0.f;
        }
        if (__syncthreads_or(any ? 1 : 0) && threadIdx.x == 0) atomicOr(&any_target[(size_t)b * g.Q + j], 1u);
    }
}

// Grid pass, separable form (used when a band's source rows fit in shared memory).  ATen's bilinear value is
//   ly0 * (lx0 * v[y0][x0] + lx1 * v[y0][x1]) + ly1 * (lx0 * v[y1][x0] + lx1 * v[y1][x1]):
// the bracketed horizontal interpolations depend on (source row, grid column) only, so a CTA computes them ONCE for the source
// rows its band of 32 grid rows touches (12 rows for 120 -> 384) and every grid point costs two multiplies and an add -- the same
// operations in the same order as `grid_logit`, hence bit-identical.  Besides the (count, sigmoid sum) partials it writes the
// SIGN BITMAP of the grid (384 x 12 words per candidate), which the mask pass reads instead of re-evaluating the bilinear.
constexpr int kBand = 32;
constexpr int kBands = kGrid / kBand;
constexpr int kWordsPerRow = kGrid / 32;
__global__ void __launch_bounds__(256) postproc_grid_kernel(const float* __restrict__ masks, PostGeom g,
                                                            const int* __restrict__ sel_query, int rows_cap,
                                                            unsigned* __restrict__ part_cnt, float* __restrict__ part_sum,
                                                            unsigned* __restrict__ bitmap) {
    extern __shared__ float s_t[];                          // rows_cap x kGrid horizontal interpolations
    __shared__ int s_x0[kGrid], s_x1[kGrid];
    __shared__ float s_lx0[kGrid], s_lx1[kGrid];
    __shared__ unsigned s_cnt[8];
    __shared__ float s_sum[8];
    const int band = blockIdx.x, j = blockIdx.y, b = blockIdx.z;
    const int q = sel_query[(size_t)b * g.Q + j];
    const float* plane = masks + ((size_t)b * g.Q + q) * g.h * g.w;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int gx = threadIdx.x; gx < kGrid; gx += blockDim.x) {
        float fx = __fsub_rn(__fmul_rn(g.rw, __fadd_rn((float)gx, 0.5f)), 0.5f);
        fx = fx < 0.f ? 0.f : fx;
        const int x0 = (int)fx;
        s_x0[gx] = x0;
        s_x1[gx] = x0 + (x0 < g.w - 1 ? 1 : 0);
        const float lx1 = __fsub_rn(fx, (float)x0);
        s_lx1[gx] = lx1;
        s_lx0[gx] = __fsub_rn(1.f, lx1);
    }
    auto src_row = [&](int gy, int& y0, int& y1, float& ly0, float& ly1) {
        float fy = __fsub_rn(__fmul_rn(g.rh, __fadd_rn((float)gy, 0.5f)), 0.5f);
        fy = fy < 0.f ? 0.f : fy;
        y0 = (int)fy;
        y1 = y0 + (y0 < g.h - 1 ? 1 : 0);
        ly1 = __fsub_rn(fy, (float)y0);
        ly0 = __fsub_rn(1.f, ly1);
    };
    int y_lo, y_hi, t0, t1;
    float f0, f1;
    src_row(band * kBand, y_lo, t1, f0, f1);
    src_row(band * kBand + kBand - 1, t0, y_hi, f0, f1);
    const int rows = y_hi - y_lo + 1;                       // <= rows_cap (checked on the host)
    __syncthreads();
    for (int i = threadIdx.x; i < rows * kGrid; i += blockDim.x) {
        const int r = i / kGrid, gx = i - r * kGrid;
        const float* row = plane + (size_t)(y_lo + r) * g.w;
        s_t[i] = __fadd_rn(__fmul_rn(s_lx0[gx], __ldg(row + s_x0[gx])), __fmul_rn(s_lx1[gx], __ldg(row + s_x1[gx])));
    }
    __syncthreads();
    unsigned cnt = 0;
    float sum = 0.f;
    unsigned* bm = bitmap + ((size_t)b * g.Q + j) * (kGrid * kWordsPerRow);
    for (int gl = warp; gl < kBand; gl += 8) {
        const int gy = band * kBand + gl;
        int y0, y1;
        float ly0, ly1;
        src_row(gy, y0, y1, ly0, ly1);
        const float* top = s_t + (y0 - y_lo) * kGrid;
        const float* bot = s_t + (y1 - y_lo) * kGrid;
#pragma unroll 4
        for (int k = 0; k < kWordsPerRow; ++k) {
            const int gx = k * 32 + lane;
            const float v = __fadd_rn(__fmul_rn(ly0, top[gx]), __fmul_rn(ly1, bot[gx]));
            const bool pos = v > 0.f;
            if (pos) {
                ++cnt;
                sum += 1.0f / (1.0f + expf(-v));
            }
            const unsigned word = __ballot_sync(0xffffffffu, pos);
            if (lane == 0) bm[gy * kWordsPerRow + k] = word;
        }
    }
#pragma unroll
    for (int k = 16; k > 0; k >>= 1) {
        cnt += __shfl_xor_sync(0xffffffffu, cnt, k);
        sum += __shfl_xor_sync(0xffffffffu, sum, k);
    }
    if (lane == 0) {
        s_cnt[warp] = cnt;
        s_sum[warp] = sum;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned c = 0;
        float sm = 0.f;
        for (int k = 0; k < 8; ++k) {
            c += s_cnt[k];
            sm += s_sum[k];
        }
        const size_t o = ((size_t)b * g.Q + j) * kBands + band;
        part_cnt[o] = c;
        part_sum[o] = sm;
    }
}

__global__ void __launch_bounds__(256) postproc_finalize_kernel(PostGeom g, float threshold, int n_chunk_grid,
                                                                const float* __restrict__ sel_score,
                                                                const int* __restrict__ sel_query,
                                                                const int* __restrict__ sel_label,
                                                                const unsigned* __restrict__ part_cnt,
                                                                const float* __restrict__ part_sum,
                                                                const unsigned* __restrict__ any_target, int* __restrict__ slot,
                                                                int* __restrict__ inv_slot, int* __restrict__ out_labels, float* __restrict__ out_scores,
                                                                int* __restrict__ out_query, int* __restrict__ out_count) {
    extern __shared__ float s_pred[];           // Q predicted scores, then Q keep flags
    int* s_keep = reinterpret_cast<int*>(s_pred + g.Q);
    const int b = blockIdx.x;
    for (int j = threadIdx.x; j < g.Q; j += blockDim.x) {
        const size_t o = ((size_t)b * g.Q + j) * n_chunk_grid;
        unsigned cnt = 0;
        float sum = 0.f;
        for (int k = 0; k < n_chunk_grid; ++k) {   // fixed order: deterministic
            cnt += part_cnt[o + k];
            sum += part_sum[o + k];
        }
        const float mask_score = sum / ((float)cnt + 1e-6f);
        const float pred = sel_score[(size_t)b * g.Q + j] * mask_score;
        s_pred[j] = pred;
        // nearest UPsampling visits every grid point, so the target mask is empty iff the grid mask is
        const bool nonempty = (g.Ht >= kGrid && g.Wt >= kGrid) ? cnt != 0u : any_target[(size_t)b * g.Q + j] != 0u;
        s_keep[j] = (nonempty && pred >= threshold) ? 1 : 0;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int n = 0;
        for (int j = 0; j < g.Q; ++j) {
            if (s_keep[j]) {
                slot[(size_t)b * g.Q + j] = n;
                inv_slot[(size_t)b * g.Q + n] = j;
                out_labels[(size_t)b * g.Q + n] = sel_label[(size_t)b * g.Q + j];
                out_scores[(size_t)b * g.Q + n] = s_pred[j];
                out_query[(size_t)b * g.Q + n] = sel_query[(size_t)b * g.Q + j];
                ++n;
            } else {
                slot[(size_t)b * g.Q + j] = -1;
            }
        }
        for (int k = n; k < g.Q; ++k) {
            out_labels[(size_t)b * g.Q + k] = -1;
            out_scores[(size_t)b * g.Q + k] = 0.f;
            out_query[(size_t)b * g.Q + k] = -1;
        }
        out_count[b] = n;
    }
}

// One thread = four consecutive target pixels of one image, for ALL kept segments: the pixel -> grid-point mapping is computed
// once, every segment costs a few bit extractions from its sign bitmap (L1/L2-resident: 18 KB per candidate) and one 4-byte
// store; the painted map keeps the highest slot whose bit is set ("last kept segment wins") in a register -- no atomics, no
// fill pass.  (Per-segment CTAs with an atomicMax per positive pixel took 3/4 of the post-processing time.)
__global__ void __launch_bounds__(256) postproc_paint_kernel(PostGeom g, const int* __restrict__ inv_slot,
                                                             const int* __restrict__ out_count,
                                                             const unsigned* __restrict__ bitmap, uint8_t* __restrict__ out_masks,
                                                             int* __restrict__ seg) {
    const int b = blockIdx.y;
    const int n_t = g.Ht * g.Wt;
    const int p0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (p0 >= n_t) return;
    const int n = n_t - p0 < 4 ? n_t - p0 : 4;
    int wi[4], sh[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int pt = p0 + (e < n ? e : 0);
        const int gy = nearest_src(pt / g.Wt, g.sy), gx = nearest_src(pt % g.Wt, g.sx);
        wi[e] = gy * (kGrid / 32) + (gx >> 5);
        sh[e] = gx & 31;
    }
    int painted[4] = {-1, -1, -1, -1};
    const int count = out_count[b];
    const bool vec = n == 4 && (n_t & 3) == 0;
    for (int sl = 0; sl < count; ++sl) {
        const unsigned* bm = bitmap + ((size_t)b * g.Q + inv_slot[(size_t)b * g.Q + sl]) * (kGrid * (kGrid / 32));
        unsigned packed = 0;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const unsigned bit = (__ldg(bm + wi[e]) >> sh[e]) & 1u;
            packed |= bit << (8 * e);
            if (bit) painted[e] = sl;
        }
        uint8_t* dst = out_masks + ((size_t)b * g.Q + sl) * n_t + p0;
        if (vec) {
            *reinterpret_cast<unsigned*>(dst) = packed;
        } else {
            for (int e = 0; e < n; ++e) dst[e] = (uint8_t)((packed >> (8 * e)) & 1u);
        }
    }
    if (seg) {
        int* sp = seg + (size_t)b * n_t + p0;
        if (vec) {
            *reinterpret_cast<int4*>(sp) = make_int4(painted[0], painted[1], painted[2], painted[3]);
        } else {
            for (int e = 0; e < n; ++e) sp[e] = painted[e];
        }
    }
}

// ---- run-length encoding of int32 label maps (HF `convert_segmentation_to_rle`: per value present, ascending, the maximal
// row-major runs as [start_1, len_1, ...] with 1-based starts).  Label k = id + 1 of id in [-1, L).  Each warp owns a subtile
// of kRleSub consecutive pixels of one image and walks it in rounds of 32 pixels, lane order = pixel order.  A run STARTS at p
// when p == 0 or seg[p-1] != seg[p] and ENDS at p when p == N-1 or seg[p+1] != seg[p].
//   1. rle_count_kernel  starts per (label, subtile) -> table (B, K, n_sub); pixels outside [-1, L) are counted and skipped
//   2. rle_scan_kernel   per image, exclusive scan of the table in label-major (label, subtile) order, in place: the first
//                        start of label k in subtile s goes to slot table[b,k,s] relative to the image; offsets (B, K+1)
//   3. rle_base_kernel   exclusive scan of the per-image totals -> base (B+1)
//   4. rle_emit_kernel   slot of a start = cursor + (same-label starts in the lower lanes); the end of a run at p takes
//                        (starts of its label at positions <= p) - 1, so a start and its end meet in one slot even when they
//                        fall in different subtiles.  The cursor per (label, subtile) is owned by one warp: no atomics decide
//                        an order, and the output depends on the input alone.
constexpr int kRleWarps = 4;
constexpr int kRleRounds = 32;
constexpr int kRleSub = 32 * kRleRounds;        // pixels per warp
constexpr int kRleMaxLabels = 4096;

__device__ __forceinline__ bool rle_label(int v, int L, int& k) {
    k = v + 1;
    return v >= -1 && v < L;
}

__global__ void __launch_bounds__(kRleWarps * 32) rle_count_kernel(const int* __restrict__ seg, int N, int K, int n_sub,
                                                                   int* __restrict__ table, int* __restrict__ bad) {
    extern __shared__ int s_rle[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int s = blockIdx.x * kRleWarps + warp, b = blockIdx.y;
    if (s >= n_sub) return;
    int* hist = s_rle + warp * K;
    for (int k = lane; k < K; k += 32) hist[k] = 0;
    __syncwarp();
    const int* img = seg + (size_t)b * N;
    unsigned n_bad = 0;
    for (int r = 0; r < kRleRounds; ++r) {
        const int p = s * kRleSub + r * 32 + lane;
        if (s * kRleSub + r * 32 >= N) break;                      // warp-uniform
        int k = -1;
        bool start = false, ok = false;
        if (p < N) {
            const int v = __ldg(img + p);
            ok = rle_label(v, K - 1, k);
            start = ok && (p == 0 || __ldg(img + p - 1) != v);
        }
        n_bad += __popc(__ballot_sync(0xffffffffu, p < N && !ok));
        if (!__ballot_sync(0xffffffffu, start)) continue;         // most rounds of a real map: no run starts here
        // one key for every lane that takes no part: __match_any_sync costs grow with the number of distinct keys
        const unsigned grp = __match_any_sync(0xffffffffu, start ? k : -1);
        if (start && (__ffs(grp) - 1) == lane) hist[k] += __popc(grp);
        __syncwarp();
    }
    __syncwarp();
    for (int k = lane; k < K; k += 32) table[((size_t)b * K + k) * n_sub + s] = hist[k];
    if (lane == 0 && n_bad) atomicAdd(bad, (int)n_bad);            // a count, not an order
}

constexpr int kScanThreads = 1024;
constexpr int kScanItems = 8;

// Exclusive scan of one value per thread over a block of kScanThreads threads; `total` = the block's sum in every thread.
// Ends with a barrier, so s_warp (kScanThreads / 32 ints) can be reused by the next call.
__device__ __forceinline__ int block_exclusive_scan(int x, int* s_warp, int& total) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int incl = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += y;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = s_warp[lane];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, w, d);
            if (lane >= d) w += y;
        }
        s_warp[lane] = w;
    }
    __syncthreads();
    const int ex = (warp ? s_warp[warp - 1] : 0) + incl - x;
    total = s_warp[kScanThreads / 32 - 1];
    __syncthreads();
    return ex;
}

__global__ void __launch_bounds__(kScanThreads) rle_scan_kernel(int K, int n_sub, int* __restrict__ table,
                                                                int* __restrict__ offsets) {
    __shared__ int s_warp[kScanThreads / 32];
    const int b = blockIdx.x;
    const long long M = (long long)K * n_sub;
    int* t = table + (size_t)b * M;
    int* off = offsets + (size_t)b * (K + 1);
    int carry = 0;
    for (long long c0 = 0; c0 < M; c0 += (long long)kScanThreads * kScanItems) {
        const long long i0 = c0 + (long long)threadIdx.x * kScanItems;
        int v[kScanItems], sum = 0;
#pragma unroll
        for (int e = 0; e < kScanItems; ++e) {
            v[e] = i0 + e < M ? t[i0 + e] : 0;
            sum += v[e];
        }
        int total;
        int run = carry + block_exclusive_scan(sum, s_warp, total);
#pragma unroll
        for (int e = 0; e < kScanItems; ++e) {
            const long long i = i0 + e;
            if (i < M) {
                t[i] = run;
                if (i % n_sub == 0) off[i / n_sub] = run;
            }
            run += v[e];
        }
        carry += total;
    }
    if (threadIdx.x == 0) off[K] = carry;
}

__global__ void __launch_bounds__(kScanThreads) rle_base_kernel(int B, int K, const int* __restrict__ offsets,
                                                                int* __restrict__ base) {
    __shared__ int s_warp[kScanThreads / 32];
    int carry = 0;
    for (int c0 = 0; c0 < B; c0 += kScanThreads) {
        const int i = c0 + threadIdx.x;
        int total;
        const int ex = block_exclusive_scan(i < B ? offsets[(size_t)i * (K + 1) + K] : 0, s_warp, total);
        if (i < B) base[i] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) base[B] = carry;
}

__global__ void __launch_bounds__(kRleWarps * 32) rle_emit_kernel(const int* __restrict__ seg, int N, int K, int n_sub,
                                                                  const int* __restrict__ table, const int* __restrict__ base,
                                                                  int2* __restrict__ runs) {
    extern __shared__ int s_rle[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int s = blockIdx.x * kRleWarps + warp, b = blockIdx.y;
    if (s >= n_sub) return;
    int* cur = s_rle + warp * K;
    const int b0 = base[b];
    for (int k = lane; k < K; k += 32) cur[k] = b0 + table[((size_t)b * K + k) * n_sub + s];
    __syncwarp();
    const int* img = seg + (size_t)b * N;
    const unsigned le = 0xffffffffu >> (31 - lane);                // lanes <= this one
    for (int r = 0; r < kRleRounds; ++r) {
        const int p = s * kRleSub + r * 32 + lane;
        if (s * kRleSub + r * 32 >= N) break;                      // warp-uniform
        int k = -1;
        bool start = false, end = false;
        if (p < N) {
            const int v = __ldg(img + p);
            if (rle_label(v, K - 1, k)) {
                start = p == 0 || __ldg(img + p - 1) != v;
                end = p == N - 1 || __ldg(img + p + 1) != v;
            }
        }
        if (!__ballot_sync(0xffffffffu, start || end)) continue;  // warp-uniform: nothing to write this round
        const unsigned grp = __match_any_sync(0xffffffffu, (start || end) ? k : -1);
        const unsigned starts = grp & __ballot_sync(0xffffffffu, start);
        int c = 0;
        if (start || end) {
            c = cur[k];
            const int slot = c + __popc(starts & le) - 1;
            if (start) runs[slot].x = p + 1;
            if (end) runs[slot].y = p + 1;
        }
        __syncwarp();
        if ((start || end) && (__ffs(grp) - 1) == lane) cur[k] = c + __popc(starts);
        __syncwarp();
    }
}

struct RleLayout {
    int K, n_sub;
    size_t table, total;
};

// The argument rules of rgbd_label_map_rle; the workspace query applies them too (0 bytes = invalid).
bool rle_args_ok(int B, int H, int W, int L) {
    return B >= 1 && H >= 1 && W >= 1 && L >= 0 && L <= kRleMaxLabels && B <= 65535 &&
           (long long)B * H * W < (1ll << 31);
}

RleLayout rle_layout(int B, int H, int W, int L) {   // valid arguments only (rle_args_ok)
    RleLayout l;
    l.K = L + 1;
    l.n_sub = ceil_div(H * W, kRleSub);
    l.table = 0;
    l.total = ((size_t)B * l.K * l.n_sub * 4 + 255) / 256 * 256;
    return l;
}

// ---- pycocotools RLE of the segments of a painted map (`pycocotools.mask.encode` of (map == s) in Fortran order, then
// `rleToString`).  The map is transposed, so the label-major runs the rle_* kernels find in it are the 1-runs of each
// segment in column-major order (position q = x*H + y).  Then, per image, one ITEM per run plus one TAIL item per
// segment s in [0, L): with the image's run indices j counted from o1 = (its first non-background run), run j of segment s
// is item (j - o1 + s) and the tail of s is item (offsets_r[s+2] - o1 + s), so items are placed without a search.
// Run m of a segment gives counts 2m (zeros before it) and 2m+1 (its length); the tail gives count 2R = h*w - end_{R-1}
// when that is > 0 (the whole [h*w] of an empty segment).  Each item reads its run and the two before it in the segment,
// which is all the string's deltas (x - c[i-2] for i > 2) need, so a segment with h*w/2 runs is spread over threads.
//   coco_transpose_kernel  (B,H,W) -> (B,W,H), 32x32 shared tiles with a padded row
//   rgbd_label_map_rle     the four rle_* kernels on the transposed map, into the workspace
//   coco_size_kernel       characters per item -> pos (B, H*W + L); run lengths of segments s >= count[b] -> bad
//   coco_scan_kernel       per image, exclusive scan of pos in place over its items; total -> offsets[b, L]
//   rle_base_kernel        exclusive scan of the per-image totals -> base (B+1)
//   coco_emit_kernel       writes each item's characters at base[b] + pos; the first item of s writes offsets[b, s]
constexpr int kCocoTile = 32;
constexpr int kCocoThreads = 256;

__global__ void __launch_bounds__(kCocoTile * 8) coco_transpose_kernel(const int* __restrict__ seg, int H, int W,
                                                                       int tiles_w, int* __restrict__ seg_t) {
    __shared__ int tile[kCocoTile][kCocoTile + 1];                 // +1: the column reads hit 32 different banks
    const int b = blockIdx.y;
    const int ty = blockIdx.x / tiles_w, tx = blockIdx.x - ty * tiles_w;
    const int* src = seg + (size_t)b * H * W;
    int* dst = seg_t + (size_t)b * H * W;
    const int x = tx * kCocoTile + threadIdx.x;
    for (int r = threadIdx.y; r < kCocoTile; r += 8) {
        const int y = ty * kCocoTile + r;
        if (y < H && x < W) tile[r][threadIdx.x] = __ldg(src + (size_t)y * W + x);
    }
    __syncthreads();
    const int y = ty * kCocoTile + threadIdx.x;
    for (int r = threadIdx.y; r < kCocoTile; r += 8) {
        const int xo = tx * kCocoTile + r;
        if (xo < W && y < H) dst[(size_t)xo * H + y] = tile[threadIdx.x][r];
    }
}

// rleToString: 5-bit groups, low bits first, 0x20 = more follow, +48.  Returns the number of characters; writes them when
// `out` is given.
__device__ __forceinline__ int coco_put(int x, uint8_t* out) {
    int n = 0;
    bool more = true;
    while (more) {
        int c = x & 0x1f;
        x >>= 5;                                                   // arithmetic: negative deltas end at x == -1
        more = (c & 0x10) ? x != -1 : x != 0;
        if (more) c |= 0x20;
        if (out) out[n] = (uint8_t)(c + 48);
        ++n;
    }
    return n;
}

// The counts of item t of image b as (up to) two string values, in order.  Returns the number of values (0, 1 or 2) and
// sets the segment, whether this is the segment's first item, and the length of the run (0 for a tail).
struct CocoItem {
    int n_val, val[2], s, item, run_len;
    bool first;
};

__device__ __forceinline__ CocoItem coco_item(int t, int N, int L, const int* __restrict__ off_r, const int2* __restrict__ runs,
                                              const int* __restrict__ img_t) {
    CocoItem it;
    const int o1 = off_r[1], n_runs = off_r[L + 1] - o1;
    int m, R;                                                      // run index in the segment; runs of the segment
    int2 cur = make_int2(0, 0);
    if (t < n_runs) {
        cur = runs[o1 + t];
        it.s = __ldg(img_t + cur.x - 1);
        m = o1 + t - off_r[it.s + 1];
        R = m + 1;
        it.item = t + it.s;
        it.run_len = cur.y - cur.x + 1;
    } else {
        it.s = t - n_runs;
        R = off_r[it.s + 2] - off_r[it.s + 1];
        m = R;                                                     // the tail sits where run R would
        it.item = off_r[it.s + 2] - o1 + it.s;
        it.run_len = 0;
    }
    it.first = m == 0;
    const int j0 = off_r[it.s + 1];                                // run m of the segment is runs[j0 + m]
    const int2 p1 = m >= 1 ? runs[j0 + m - 1] : make_int2(0, 0);
    const int2 p2 = m >= 2 ? runs[j0 + m - 2] : make_int2(0, 0);
    const int gap1 = p1.x - 1 - p2.y;                              // zeros before run m-1 (count 2m-2), when m >= 1
    if (t < n_runs) {
        const int gap = cur.x - 1 - p1.y;                          // count 2m
        it.val[0] = m >= 2 ? gap - gap1 : gap;                     // delta when 2m > 2
        it.val[1] = m >= 1 ? it.run_len - (p1.y - p1.x + 1) : it.run_len;   // count 2m+1: delta when 2m+1 > 2
        it.n_val = 2;
    } else {
        const int tail = N - p1.y;                                 // count 2R: trailing zeros, h*w for an empty segment
        it.val[0] = R >= 2 ? tail - gap1 : tail;
        it.n_val = tail > 0 ? 1 : 0;
    }
    return it;
}

// image b's valid segment count: count[b] when it lies in [0, L], else 0 (and coco_scan_kernel counts it in bad)
__device__ __forceinline__ int coco_n_segments(const int* __restrict__ count, int b, int L) {
    const int n = count[b];
    return n >= 0 && n <= L ? n : 0;
}

__global__ void __launch_bounds__(kCocoThreads) coco_size_kernel(int N, int L, const int* __restrict__ count,
                                                                 const int* __restrict__ off_r, const int* __restrict__ base_r,
                                                                 const int2* __restrict__ runs, const int* __restrict__ seg_t,
                                                                 int* __restrict__ pos, int* __restrict__ bad) {
    const int b = blockIdx.y;
    const int t = blockIdx.x * kCocoThreads + threadIdx.x;
    const int* o = off_r + (size_t)b * (L + 2);
    const int n_items = o[L + 1] - o[1] + L;
    int n_bad = 0;
    if (t < n_items) {
        const CocoItem it = coco_item(t, N, L, o, runs + base_r[b], seg_t + (size_t)b * N);
        int n = 0;
        if (it.s < coco_n_segments(count, b, L)) {
#pragma unroll
            for (int v = 0; v < 2; ++v) n += v < it.n_val ? coco_put(it.val[v], nullptr) : 0;
        } else {
            n_bad = it.run_len;                                    // painted pixels of an id >= count[b]
        }
        pos[(size_t)b * (N + L) + it.item] = n;
    }
#pragma unroll
    for (int k = 16; k > 0; k >>= 1) n_bad += __shfl_xor_sync(0xffffffffu, n_bad, k);
    if ((threadIdx.x & 31) == 0 && n_bad) atomicAdd(bad, n_bad);    // a count, not an order
}

// rle_scan_kernel's pattern over the image's items only: a checkerboard has ~h*w/2 of them, a real map a few per column
__global__ void __launch_bounds__(kScanThreads) coco_scan_kernel(int N, int L, const int* __restrict__ count,
                                                                 const int* __restrict__ off_r, int* __restrict__ pos,
                                                                 int* __restrict__ offsets, int* __restrict__ bad) {
    __shared__ int s_warp[kScanThreads / 32];
    const int b = blockIdx.x;
    const int* o = off_r + (size_t)b * (L + 2);
    const int n_items = o[L + 1] - o[1] + L;
    int* p = pos + (size_t)b * (N + L);
    int carry = 0;
    for (int c0 = 0; c0 < n_items; c0 += kScanThreads * kScanItems) {
        const int i0 = c0 + threadIdx.x * kScanItems;
        int v[kScanItems], sum = 0;
#pragma unroll
        for (int e = 0; e < kScanItems; ++e) {
            v[e] = i0 + e < n_items ? p[i0 + e] : 0;
            sum += v[e];
        }
        int total;
        int run = carry + block_exclusive_scan(sum, s_warp, total);
#pragma unroll
        for (int e = 0; e < kScanItems; ++e) {
            if (i0 + e < n_items) p[i0 + e] = run;
            run += v[e];
        }
        carry += total;
    }
    if (threadIdx.x == 0) {
        offsets[(size_t)b * (L + 1) + L] = carry;
        if (count[b] < 0 || count[b] > L) atomicAdd(bad, 1);
    }
}

__global__ void __launch_bounds__(kCocoThreads) coco_emit_kernel(int N, int L, const int* __restrict__ count,
                                                                 const int* __restrict__ off_r, const int* __restrict__ base_r,
                                                                 const int2* __restrict__ runs, const int* __restrict__ seg_t,
                                                                 const int* __restrict__ pos, const int* __restrict__ base,
                                                                 int* __restrict__ offsets, uint8_t* __restrict__ chars) {
    const int b = blockIdx.y;
    const int t = blockIdx.x * kCocoThreads + threadIdx.x;
    const int* o = off_r + (size_t)b * (L + 2);
    if (t >= o[L + 1] - o[1] + L) return;
    const CocoItem it = coco_item(t, N, L, o, runs + base_r[b], seg_t + (size_t)b * N);
    const int at = pos[(size_t)b * (N + L) + it.item];
    if (it.first) offsets[(size_t)b * (L + 1) + it.s] = at;
    if (it.s >= coco_n_segments(count, b, L)) return;
    uint8_t* dst = chars + base[b] + at;
#pragma unroll
    for (int v = 0; v < 2; ++v) dst += v < it.n_val ? coco_put(it.val[v], dst) : 0;
}

struct CocoLayout {
    RleLayout rle;
    size_t seg_t, rle_ws, off_r, base_r, runs, pos, total;
};

// The argument rules of rgbd_instance_rle: those of rgbd_label_map_rle, and the character capacity (a count takes at most 7
// characters, an image at most 2*H*W + L counts) must index with int32.
bool coco_args_ok(int B, int H, int W, int L) {
    return rle_args_ok(B, H, W, L) && 7ll * B * (2ll * H * W + L) < (1ll << 31);
}

size_t coco_capacity(int B, int H, int W, int L) { return 7ull * B * (2ull * H * W + L); }

CocoLayout coco_layout(int B, int H, int W, int L) {   // valid arguments only (coco_args_ok)
    CocoLayout l;
    l.rle = rle_layout(B, W, H, L);
    const size_t N = (size_t)H * W;
    size_t o = 0;
    auto take = [&](size_t bytes) {
        const size_t at = o;
        o += (bytes + 255) / 256 * 256;
        return at;
    };
    l.seg_t = take((size_t)B * N * 4);
    l.rle_ws = take(l.rle.total);
    l.off_r = take((size_t)B * (L + 2) * 4);
    l.base_r = take((size_t)(B + 1) * 4);
    l.runs = take((size_t)B * N * 8);
    l.pos = take((size_t)B * (N + L) * 4);
    l.total = o;
    return l;
}

__global__ void __launch_bounds__(256) fill_int_kernel(int* __restrict__ p, size_t n, int v) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}

// one CTA per (pred, gt) pair; masks are bytes holding 0 / 1
__global__ void __launch_bounds__(256) mask_iou_kernel(const uint8_t* __restrict__ pred, const uint8_t* __restrict__ gt,
                                                       long long n, float* __restrict__ iou, int G) {
    const int p = blockIdx.y, gi = blockIdx.x;
    const uint8_t* a = pred + (size_t)p * n;
    const uint8_t* c = gt + (size_t)gi * n;
    unsigned inter = 0, na = 0, nc = 0;
    const bool vec = (n % 16 == 0) && ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(c)) % 16 == 0);
    if (vec) {
        const uint4* a4 = reinterpret_cast<const uint4*>(a);
        const uint4* c4 = reinterpret_cast<const uint4*>(c);
        for (long long i = threadIdx.x; i < n / 16; i += blockDim.x) {
            const uint4 x = __ldg(a4 + i), y = __ldg(c4 + i);
            inter += __popc(x.x & y.x & 0x01010101u) + __popc(x.y & y.y & 0x01010101u) + __popc(x.z & y.z & 0x01010101u) +
                     __popc(x.w & y.w & 0x01010101u);
            na += __popc(x.x & 0x01010101u) + __popc(x.y & 0x01010101u) + __popc(x.z & 0x01010101u) + __popc(x.w & 0x01010101u);
            nc += __popc(y.x & 0x01010101u) + __popc(y.y & 0x01010101u) + __popc(y.z & 0x01010101u) + __popc(y.w & 0x01010101u);
        }
    } else {
        for (long long i = threadIdx.x; i < n; i += blockDim.x) {
            const unsigned x = a[i] & 1u, y = c[i] & 1u;
            inter += x & y;
            na += x;
            nc += y;
        }
    }
    __shared__ unsigned s[3][8];
#pragma unroll
    for (int k = 16; k > 0; k >>= 1) {
        inter += __shfl_xor_sync(0xffffffffu, inter, k);
        na += __shfl_xor_sync(0xffffffffu, na, k);
        nc += __shfl_xor_sync(0xffffffffu, nc, k);
    }
    if ((threadIdx.x & 31) == 0) {
        s[0][threadIdx.x >> 5] = inter;
        s[1][threadIdx.x >> 5] = na;
        s[2][threadIdx.x >> 5] = nc;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned i2 = 0, a2 = 0, c2 = 0;
        for (int k = 0; k < 8; ++k) {
            i2 += s[0][k];
            a2 += s[1][k];
            c2 += s[2][k];
        }
        const unsigned uni = a2 + c2 - i2;
        iou[(size_t)p * G + gi] = uni ? (float)((double)i2 / (double)uni) : 0.f;
    }
}

int next_pow2(int v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

struct WsLayout {
    size_t sel_score, sel_query, sel_label, part_cnt, part_sum, any_target, slot, inv_slot, bitmap, total;
};

WsLayout ws_layout(int B, int Q) {
    const int n_chunk = ceil_div(kGrid * kGrid, kChunk);
    WsLayout l;
    size_t o = 0;
    auto take = [&](size_t bytes) {
        const size_t at = o;
        o += (bytes + 255) / 256 * 256;
        return at;
    };
    l.sel_score = take((size_t)B * Q * 4);
    l.sel_query = take((size_t)B * Q * 4);
    l.sel_label = take((size_t)B * Q * 4);
    l.part_cnt = take((size_t)B * Q * n_chunk * 4);
    l.part_sum = take((size_t)B * Q * n_chunk * 4);
    l.any_target = take((size_t)B * Q * 4);
    l.slot = take((size_t)B * Q * 4);
    l.inv_slot = take((size_t)B * Q * 4);
    l.bitmap = take((size_t)B * Q * kGrid * (kGrid / 32) * 4);
    l.total = o;
    return l;
}

}  // namespace

extern "C" size_t rgbd_postprocess_workspace_bytes(int B, int Q) {
    if (B < 1 || Q < 1) return 0;
    return ws_layout(B, Q).total;
}

extern "C" int rgbd_postprocess_instances(const float* class_logits, const float* mask_logits, int B, int Q, int C1, int h,
                                          int w, int Ht, int Wt, float threshold, void* workspace, uint8_t* out_masks,
                                          int* out_labels, float* out_scores, int* out_query, int* out_count,
                                          int* out_segmentation, rgbd_stream_t stream) {
    RGBD_CHECK_ARG(class_logits && mask_logits && workspace && out_masks && out_labels && out_scores && out_query && out_count,
                   "postprocess: null pointer");
    RGBD_CHECK_ARG(B >= 1 && Q >= 1 && C1 >= 2 && h >= 1 && w >= 1 && Ht >= 1 && Wt >= 1, "postprocess: bad geometry");
    const int n_cand = Q * (C1 - 1);
    RGBD_CHECK_ARG(n_cand <= kMaxSort, "postprocess: Q*(C) = %d candidates exceed the in-shared-memory sort (%d)", n_cand, kMaxSort);
    RGBD_CHECK_ARG(Q <= 4096, "postprocess: at most 4096 queries");
    cudaStream_t s = (cudaStream_t)stream;
    PostGeom g;
    g.B = B; g.Q = Q; g.C1 = C1; g.h = h; g.w = w; g.Ht = Ht; g.Wt = Wt;
    g.rh = (float)h / (float)kGrid; g.rw = (float)w / (float)kGrid;
    g.sy = (float)kGrid / (float)Ht; g.sx = (float)kGrid / (float)Wt;
    const WsLayout l = ws_layout(B, Q);
    uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
    float* sel_score = reinterpret_cast<float*>(ws + l.sel_score);
    int* sel_query = reinterpret_cast<int*>(ws + l.sel_query);
    int* sel_label = reinterpret_cast<int*>(ws + l.sel_label);
    unsigned* part_cnt = reinterpret_cast<unsigned*>(ws + l.part_cnt);
    float* part_sum = reinterpret_cast<float*>(ws + l.part_sum);
    unsigned* any_target = reinterpret_cast<unsigned*>(ws + l.any_target);
    int* slot = reinterpret_cast<int*>(ws + l.slot);
    int* inv_slot = reinterpret_cast<int*>(ws + l.inv_slot);
    unsigned* bitmap = reinterpret_cast<unsigned*>(ws + l.bitmap);

    const int n_sort = next_pow2(n_cand < Q ? Q : n_cand);
    RgbdDeviceInfo di;
    if (int rc = rgbd_device_info(&di)) return rc;
    RGBD_ONCE_PER_DEVICE(di.device, {
        RGBD_CHECK_CUDA(cudaFuncSetAttribute(postproc_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSort * 8));
    });
    postproc_select_kernel<<<B, 256, (size_t)n_sort * 8, s>>>(class_logits, g, n_sort, sel_score, sel_query, sel_label);
    RGBD_CHECK_LAUNCH();
    RGBD_CHECK_CUDA(cudaMemsetAsync(any_target, 0, (size_t)B * Q * 4, s));
    int n_chunk_grid = ceil_div(kGrid * kGrid, kChunk);
    const int n_chunk_t = (Ht >= kGrid && Wt >= kGrid) ? 0 : ceil_div(Ht * Wt, kChunk);
    // source rows one band of grid rows can touch: floor(rh * 31) + 3 bounds y1(last) - y0(first) + 1
    const int rows_cap = (int)((double)g.rh * (kBand - 1)) + 3;
    const size_t band_smem = (size_t)rows_cap * kGrid * sizeof(float);
    if (band_smem <= 64 * 1024) {
        RGBD_ONCE_PER_DEVICE(di.device, {
            RGBD_CHECK_CUDA(cudaFuncSetAttribute(postproc_grid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        });
        postproc_grid_kernel<<<dim3(kBands, Q, B), 256, band_smem, s>>>(mask_logits, g, sel_query, rows_cap, part_cnt, part_sum, bitmap);
        RGBD_CHECK_LAUNCH();
        if (n_chunk_t) {          // downsampled targets: any(mask) over the target pixels (the grid chunks of this launch are empty)
            postproc_stats_kernel<<<dim3(n_chunk_t, Q, B), 256, 0, s>>>(mask_logits, g, sel_query, 0, part_cnt, part_sum, any_target,
                                                                       nullptr);
            RGBD_CHECK_LAUNCH();
        }
        n_chunk_grid = kBands;
    } else {                      // very tall logit planes: point-wise evaluation
        postproc_stats_kernel<<<dim3(n_chunk_grid + n_chunk_t, Q, B), 256, 0, s>>>(mask_logits, g, sel_query, n_chunk_grid, part_cnt,
                                                                                   part_sum, any_target, bitmap);
        RGBD_CHECK_LAUNCH();
    }
    postproc_finalize_kernel<<<B, 256, (size_t)Q * 8, s>>>(g, threshold, n_chunk_grid, sel_score, sel_query, sel_label, part_cnt,
                                                           part_sum, any_target, slot, inv_slot, out_labels, out_scores, out_query,
                                                           out_count);
    RGBD_CHECK_LAUNCH();
    RGBD_CHECK_ARG(B <= 65535, "postprocess: at most 65535 images per call");
    postproc_paint_kernel<<<dim3(ceil_div(Ht * Wt, 256 * 4), B), 256, 0, s>>>(g, inv_slot, out_count, bitmap, out_masks, out_segmentation);
    RGBD_CHECK_LAUNCH();
    return RGBD_OK;
}

extern "C" size_t rgbd_label_map_rle_workspace_bytes(int B, int H, int W, int L) {
    return rle_args_ok(B, H, W, L) ? rle_layout(B, H, W, L).total : 0;
}

extern "C" int rgbd_label_map_rle(const int* seg, int B, int H, int W, int L, void* workspace, int* offsets, int* base,
                                  int* runs, int* bad_count, rgbd_stream_t stream) {
    RGBD_CHECK_ARG(seg && workspace && offsets && base && runs && bad_count, "label_map_rle: null pointer");
    RGBD_CHECK_ARG(B >= 1 && H >= 1 && W >= 1, "label_map_rle: bad geometry B=%d H=%d W=%d", B, H, W);
    RGBD_CHECK_ARG(L >= 0 && L <= kRleMaxLabels, "label_map_rle: L = %d labels outside [0, %d]", L, kRleMaxLabels);
    RGBD_CHECK_ARG((long long)B * H * W < (1ll << 31), "label_map_rle: B*H*W must be below 2^31");
    RGBD_CHECK_ARG(B <= 65535, "label_map_rle: at most 65535 images per call");
    cudaStream_t s = (cudaStream_t)stream;
    const RleLayout l = rle_layout(B, H, W, L);
    const int N = H * W;
    int* table = reinterpret_cast<int*>(reinterpret_cast<uint8_t*>(workspace) + l.table);
    const size_t smem = (size_t)kRleWarps * l.K * sizeof(int);
    RgbdDeviceInfo di;
    if (int rc = rgbd_device_info(&di)) return rc;
    RGBD_ONCE_PER_DEVICE(di.device, {
        const int cap = kRleWarps * (kRleMaxLabels + 1) * (int)sizeof(int);
        RGBD_CHECK_CUDA(cudaFuncSetAttribute(rle_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
        RGBD_CHECK_CUDA(cudaFuncSetAttribute(rle_emit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
    });
    const dim3 grid(ceil_div(l.n_sub, kRleWarps), B);
    RGBD_CHECK_CUDA(cudaMemsetAsync(bad_count, 0, sizeof(int), s));
    rle_count_kernel<<<grid, kRleWarps * 32, smem, s>>>(seg, N, l.K, l.n_sub, table, bad_count);
    RGBD_CHECK_LAUNCH();
    rle_scan_kernel<<<B, kScanThreads, 0, s>>>(l.K, l.n_sub, table, offsets);
    RGBD_CHECK_LAUNCH();
    rle_base_kernel<<<1, kScanThreads, 0, s>>>(B, l.K, offsets, base);
    RGBD_CHECK_LAUNCH();
    rle_emit_kernel<<<grid, kRleWarps * 32, smem, s>>>(seg, N, l.K, l.n_sub, table, base, reinterpret_cast<int2*>(runs));
    RGBD_CHECK_LAUNCH();
    return RGBD_OK;
}

extern "C" size_t rgbd_instance_rle_workspace_bytes(int B, int H, int W, int L) {
    return coco_args_ok(B, H, W, L) ? coco_layout(B, H, W, L).total : 0;
}

extern "C" size_t rgbd_instance_rle_capacity(int B, int H, int W, int L) {
    return coco_args_ok(B, H, W, L) ? coco_capacity(B, H, W, L) : 0;
}

extern "C" int rgbd_instance_rle(const int* seg, const int* count, int B, int H, int W, int L, void* workspace, int* offsets,
                                 int* base, uint8_t* chars, int* bad_count, rgbd_stream_t stream) {
    RGBD_CHECK_ARG(seg && count && workspace && offsets && base && chars && bad_count, "instance_rle: null pointer");
    RGBD_CHECK_ARG(B >= 1 && H >= 1 && W >= 1, "instance_rle: bad geometry B=%d H=%d W=%d", B, H, W);
    RGBD_CHECK_ARG(L >= 0 && L <= kRleMaxLabels, "instance_rle: L = %d labels outside [0, %d]", L, kRleMaxLabels);
    RGBD_CHECK_ARG(B <= 65535, "instance_rle: at most 65535 images per call");
    RGBD_CHECK_ARG(coco_args_ok(B, H, W, L), "instance_rle: 7*B*(2*H*W + L) characters must be below 2^31");
    cudaStream_t s = (cudaStream_t)stream;
    const CocoLayout l = coco_layout(B, H, W, L);
    uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
    int* seg_t = reinterpret_cast<int*>(ws + l.seg_t);
    int* off_r = reinterpret_cast<int*>(ws + l.off_r);
    int* base_r = reinterpret_cast<int*>(ws + l.base_r);
    int* runs = reinterpret_cast<int*>(ws + l.runs);
    int* pos = reinterpret_cast<int*>(ws + l.pos);
    const int N = H * W;
    const int tiles_w = ceil_div(W, kCocoTile);
    coco_transpose_kernel<<<dim3(tiles_w * ceil_div(H, kCocoTile), B), dim3(kCocoTile, 8), 0, s>>>(seg, H, W, tiles_w, seg_t);
    RGBD_CHECK_LAUNCH();
    // the column-major runs: the label encoder on the (W, H) maps; it zeroes bad_count and counts ids outside [-1, L)
    if (int rc = rgbd_label_map_rle(seg_t, B, W, H, L, ws + l.rle_ws, off_r, base_r, runs, bad_count, stream)) return rc;
    const dim3 grid(ceil_div(N + L, kCocoThreads), B);
    const int2* runs2 = reinterpret_cast<const int2*>(runs);
    coco_size_kernel<<<grid, kCocoThreads, 0, s>>>(N, L, count, off_r, base_r, runs2, seg_t, pos, bad_count);
    RGBD_CHECK_LAUNCH();
    coco_scan_kernel<<<B, kScanThreads, 0, s>>>(N, L, count, off_r, pos, offsets, bad_count);
    RGBD_CHECK_LAUNCH();
    rle_base_kernel<<<1, kScanThreads, 0, s>>>(B, L, offsets, base);
    RGBD_CHECK_LAUNCH();
    coco_emit_kernel<<<grid, kCocoThreads, 0, s>>>(N, L, count, off_r, base_r, runs2, seg_t, pos, base, offsets, chars);
    RGBD_CHECK_LAUNCH();
    return RGBD_OK;
}

extern "C" int rgbd_mask_iou(const uint8_t* pred_masks, const uint8_t* gt_masks, int P, int G, long long pixels, float* iou,
                             rgbd_stream_t stream) {
    RGBD_CHECK_ARG(iou && pixels >= 1 && P >= 0 && G >= 0, "mask_iou: bad arguments");
    if (P == 0 || G == 0) return RGBD_OK;
    RGBD_CHECK_ARG(pred_masks && gt_masks, "mask_iou: null pointer");
    RGBD_CHECK_ARG(P <= 65535, "mask_iou: at most 65535 predictions per call");
    mask_iou_kernel<<<dim3(G, P), 256, 0, (cudaStream_t)stream>>>(pred_masks, gt_masks, pixels, iou, G);
    RGBD_CHECK_LAUNCH();
    return RGBD_OK;
}
