// Host side of the tcgen05 kernels: bf16 TMA tensor maps and launches on 2-CTA clusters.
#pragma once
#include "common.cuh"
#include <cuda.h>
#include <utility>

// Encodes a bf16 tiled tensor map of rank R: `dims` innermost first, `strides` the byte strides of dims 1..R-1, `box` the
// tile one TMA copy moves.  Element strides 1, 256-byte L2 promotion, out-of-bounds elements read as zero.  A failure is
// reported under the caller's name `who`.
template <int R>
int encode_bf16_map(CUtensorMap* m, const char* who, const void* base, const long long (&dims)[R],
                    const long long (&strides)[R - 1], const int (&box)[R], CUtensorMapSwizzle swizzle) {
    typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                      const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                      CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static const EncodeTiledFn encode = [] {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess ||
            qres != cudaDriverEntryPointSuccess)
            fn = nullptr;
        return (EncodeTiledFn)fn;
    }();
    if (!encode) {
        rgbd_set_error("%s: cuTensorMapEncodeTiled is not available from the driver", who);
        return RGBD_ERR_CUDA;
    }
    cuuint64_t d[R], s[R];
    cuuint32_t b[R], e[R];
    for (int i = 0; i < R; ++i) {
        d[i] = (cuuint64_t)dims[i];
        if (i + 1 < R) s[i] = (cuuint64_t)strides[i];
        b[i] = (cuuint32_t)box[i];
        e[i] = 1;
    }
    const CUresult r = encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, R, const_cast<void*>(base), d, s, b, e,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        rgbd_set_error("%s: cuTensorMapEncodeTiled failed with %d", who, (int)r);
        return RGBD_ERR_CUDA;
    }
    return RGBD_OK;
}

// kernel<<<grid, threads, smem, stream>>>(args...); with `pair` the grid (even) runs as clusters of two CTAs, the unit of
// tcgen05 cta_group::2.
template <typename... Params, typename... Args>
int launch_kernel(void (*kernel)(Params...), int grid, int threads, int smem, bool pair, cudaStream_t stream, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pair ? 1 : 0;
    RGBD_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...));
    return RGBD_OK;
}
