// fdes_b200 -- host side of the TMA column tiles: CUtensorMap descriptors for [images][N][N]
// complex64 arrays, boxes of [BR rows][CW columns] (col_pipe.cuh).  The driver entry point is
// resolved through the runtime (cudaGetDriverEntryPoint), so the library links only libcudart.
#include "sweep_vtable.h"
#include <cuda.h>
#include <cuda_runtime.h>
#include <cstring>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

namespace fdes {

namespace {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn()
{
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p ||
            q != cudaDriverEntryPointSuccess)
            throw std::runtime_error("cuTensorMapEncodeTiled is not available from this driver");
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}
struct Entry { int dev; const void* base; int N, nimg, CW, BR; CUtensorMap map; };
std::mutex g_mutex;
std::vector<Entry> g_cache;
}  // namespace

void tile_map(CUtensorMap_st* out, const void* base, int N, int nimg, int CW, int BR)
{
    int dev = 0;
    CK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_mutex);
    for (const Entry& e : g_cache)
        if (e.base == base && e.N == N && e.nimg == nimg && e.CW == CW && e.BR == BR && e.dev == dev) { *out = e.map; return; }
    if (g_cache.size() >= 512) g_cache.clear();   // descriptors are 128 bytes; a bounded cache is enough
    Entry e{dev, base, N, nimg, CW, BR, {}};
    const cuuint64_t dims[3] = {(cuuint64_t)N, (cuuint64_t)N, (cuuint64_t)nimg};
    const cuuint64_t strides[2] = {(cuuint64_t)N * 8, (cuuint64_t)N * N * 8};    // bytes, dimensions 1 and 2
    const cuuint32_t box[3] = {(cuuint32_t)CW, (cuuint32_t)BR, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    const int rowb = CW * 8;
    const CUtensorMapSwizzle swz = rowb >= 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                 : rowb == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                 : rowb == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
    // complex64 elements travel as opaque 8-byte words
    const CUresult r = encode_fn()(&e.map, CU_TENSOR_MAP_DATA_TYPE_UINT64, 3, const_cast<void*>(base), dims, strides, box, estr,
                                   CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        throw std::runtime_error("cuTensorMapEncodeTiled failed with code " + std::to_string((int)r) + " for N = " +
                                 std::to_string(N) + ", tile width " + std::to_string(CW));
    g_cache.push_back(e);
    *out = e.map;
}

}  // namespace fdes
