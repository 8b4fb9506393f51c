// Shared types and host helpers of the tcgen05 NatureCNN kernels (included by net_tc.cu and the tc_*.cuh kernel files).
#pragma once
#include <cuda.h>            // CUtensorMap types only; the encoder is resolved at run time (no libcuda link)
#include <cstring>
#include "common.cuh"
#include "tc_common.cuh"

namespace b200rl {
using namespace tc;
typedef __nv_bfloat16 bf16;

__device__ __forceinline__ int4 ldg16(const void* p) { return __ldg(reinterpret_cast<const int4*>(p)); }

// ---- host: tensor maps for row-major bf16 matrices (cuTensorMapEncodeTiled resolved through the runtime)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static int make_tmap_2d(CUtensorMap* tm, const void* base, int64_t rows, int64_t cols, int box_rows, const char* what) {
    if (!g_encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
        if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn)
            return fail(B200RL_ERR_CUDA, "%s: cuTensorMapEncodeTiled not available (%s)", what, cudaGetErrorString(e));
        g_encode = reinterpret_cast<EncodeTiledFn>(fn);
    }
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
    const cuuint32_t box[2] = {64u, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1u, 1u};
    CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(B200RL_ERR_CUDA, "%s: cuTensorMapEncodeTiled failed (%d)", what, (int)r);
    return B200RL_OK;
}

// [n_images][rows_per_image][cols] bf16, box = [1][box_rows][64]: rows past an image's end are zero-filled
static int make_tmap_3d(CUtensorMap* tm, const void* base, int64_t n_images, int64_t rows_per_image, int64_t cols, int box_rows,
                        const char* what) {
    if (!g_encode) {
        CUtensorMap dummy;
        int rc = make_tmap_2d(&dummy, base, 128, 64, 8, what);      // resolves the driver entry point
        if (rc) return rc;
    }
    const cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows_per_image, (cuuint64_t)n_images};
    const cuuint64_t strides[2] = {(cuuint64_t)cols * 2, (cuuint64_t)rows_per_image * (cuuint64_t)cols * 2};
    const cuuint32_t box[3] = {64u, (cuuint32_t)box_rows, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(B200RL_ERR_CUDA, "%s: cuTensorMapEncodeTiled (3-D) failed (%d)", what, (int)r);
    return B200RL_OK;
}

// uint8 [n_images][rows_per_image][cols] (row pitch `pitch` bytes), box = [1][box_rows][box_cols]; swizzle = the box
// width (64 B or 128 B rows), none otherwise.  Out-of-range rows / columns are
// zero-filled.
static int make_tmap_3d_u8(CUtensorMap* tm, const void* base, int64_t n_images, int64_t rows_per_image, int64_t cols, int64_t pitch,
                           int box_rows, int box_cols, const char* what) {
    if (!g_encode) {
        CUtensorMap dummy;
        int rc = make_tmap_2d(&dummy, base, 128, 64, 8, what);      // resolves the driver entry point
        if (rc) return rc;
    }
    const cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows_per_image, (cuuint64_t)n_images};
    const cuuint64_t strides[2] = {(cuuint64_t)pitch, (cuuint64_t)rows_per_image * (cuuint64_t)pitch};
    const cuuint32_t box[3] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE,
                          box_cols == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : (box_cols == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE),
                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(B200RL_ERR_CUDA, "%s: cuTensorMapEncodeTiled (u8 3-D) failed (%d)", what, (int)r);
    return B200RL_OK;
}

// uint8 frames [n_images][441 positions][64 ch] read as [n_images][221 pair rows][128 B] (image stride 28 224 B), box =
// [1][box_rows][128 B], SWIZZLE_128B; rows >= 221 are zero-filled
static int make_tmap_pairs_u8(CUtensorMap* tm, const void* base, int64_t n_images, const char* what, int box_rows = 144) {
    if (!g_encode) {
        CUtensorMap dummy;
        int rc = make_tmap_2d(&dummy, base, 128, 64, 8, what);
        if (rc) return rc;
    }
    const cuuint64_t dims[3] = {128u, 221u, (cuuint64_t)n_images};
    const cuuint64_t strides[2] = {128u, 28224u};
    const cuuint32_t box[3] = {128u, (cuuint32_t)box_rows, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(B200RL_ERR_CUDA, "%s: cuTensorMapEncodeTiled (u8 pair rows) failed (%d)", what, (int)r);
    return B200RL_OK;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device (per-context) attribute: cache the opt-in per device
struct SmemAttrCache {
    size_t v[64] = {};
    template <class F>
    int ensure(F* func, size_t smem, const char* what) {
        int dev = 0;
        cudaGetDevice(&dev);
        const bool cached = dev >= 0 && dev < 64;
        if (cached && smem <= v[dev]) return B200RL_OK;
        cudaError_t e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return fail(B200RL_ERR_CUDA, "%s: smem attribute (%zu B): %s", what, smem, cudaGetErrorString(e));
        if (cached) v[dev] = smem;
        return B200RL_OK;
    }
};

static int g_num_sms = 0;
static int num_sms() {
    if (g_num_sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        if (cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || g_num_sms <= 0) g_num_sms = 148;
    }
    return g_num_sms;
}

}  // namespace b200rl
