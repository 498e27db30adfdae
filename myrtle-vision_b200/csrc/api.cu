// api.cu — error reporting, launch counter and host-side TMA descriptor construction.
#include <stdarg.h>

#include "common.cuh"
#include "../../include/mv_b200.h"

namespace mv {

static thread_local char g_err[512] = "";
int64_t g_launches = 0;
int* g_overflow = nullptr;      // device int registered with mv_set_overflow_flag (NULL: no overflow reporting)

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int check_cuda(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return 0;
    set_error("CUDA error in %s: %s", what, cudaGetErrorString(e));
    return 1;
}

// cuTensorMapEncodeTiled is a driver entry point; fetch it through the runtime so the
// library carries no link-time dependency on libcuda (it must load on a CPU-only box).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn) return fn;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || p == nullptr) {
        set_error("cuTensorMapEncodeTiled unavailable: %s", cudaGetErrorString(e));
        return nullptr;
    }
    fn = reinterpret_cast<EncodeTiledFn>(p);
    return fn;
}

static CUtensorMapDataType tmap_dtype(int dtype, int* esz) {
    switch (dtype) {
        case MV_F16: *esz = 2; return CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
        default: *esz = 4; return CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
    }
}

int make_tmap_2d(CUtensorMap* map, const void* ptr, int dtype, uint64_t rows, uint64_t cols,
                 uint64_t ld, uint32_t box_rows, uint32_t box_cols) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return 1;
    int esz;
    CUtensorMapDataType dt = tmap_dtype(dtype, &esz);
    MV_CHECK(reinterpret_cast<uintptr_t>(ptr) % 16 == 0, "TMA: base pointer not 16-byte aligned");
    MV_CHECK((ld * esz) % 16 == 0, "TMA: row pitch %llu B not a multiple of 16", (unsigned long long)(ld * esz));
    MV_CHECK(box_cols * esz == 128, "TMA: box inner extent must be 128 B for SWIZZLE_128B");
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {ld * esz};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, dt, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MV_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(2d) failed with %d (rows=%llu cols=%llu ld=%llu box=%ux%u)",
             int(r), (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld, box_rows, box_cols);
    return 0;
}

// un-swizzled 2-D boxes (epilogue operands read row by row by the CUDA cores)
int make_tmap_2d_plain(CUtensorMap* map, const void* ptr, int dtype, uint64_t rows, uint64_t cols,
                       uint64_t ld, uint32_t box_rows, uint32_t box_cols, int swizzle64) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return 1;
    int esz;
    CUtensorMapDataType dt = tmap_dtype(dtype, &esz);
    MV_CHECK(reinterpret_cast<uintptr_t>(ptr) % 16 == 0, "TMA: base pointer not 16-byte aligned");
    MV_CHECK((ld * esz) % 16 == 0, "TMA: row pitch %llu B not a multiple of 16", (unsigned long long)(ld * esz));
    MV_CHECK((box_cols * esz) % 16 == 0, "TMA: box inner extent must be a multiple of 16 B");
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {ld * esz};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, dt, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MV_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(2d, plain) failed with %d", int(r));
    return 0;
}

int make_tmap_3d(CUtensorMap* map, const void* ptr, int dtype, uint64_t d0, uint64_t d1,
                 uint64_t d2, uint64_t stride1, uint64_t stride2, uint32_t box0, uint32_t box1,
                 uint32_t box2) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return 1;
    int esz;
    CUtensorMapDataType dt = tmap_dtype(dtype, &esz);
    MV_CHECK(reinterpret_cast<uintptr_t>(ptr) % 16 == 0, "TMA: base pointer not 16-byte aligned");
    MV_CHECK((stride1 * esz) % 16 == 0 && (stride2 * esz) % 16 == 0, "TMA: strides not multiples of 16 B");
    MV_CHECK(box0 * esz == 128, "TMA: box inner extent must be 128 B for SWIZZLE_128B");
    cuuint64_t dims[3] = {d0, d1, d2};
    cuuint64_t strides[2] = {stride1 * esz, stride2 * esz};
    cuuint32_t box[3] = {box0, box1, box2};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(map, dt, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MV_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(3d) failed with %d", int(r));
    return 0;
}

}  // namespace mv

extern "C" const char* mv_last_error(void) { return mv::g_err; }
extern "C" int mv_version(void) { return 105; }
extern "C" int mv_set_overflow_flag(int* flag_dev) { mv::g_overflow = flag_dev; return 0; }
extern "C" int64_t mv_launch_count(void) { return mv::g_launches; }
