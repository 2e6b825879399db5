// tma_util.cu -- host half of tma_util.cuh: tensor-map encoding (one driver entry-point lookup), the tensor-map cache of
// the tendency kernels, the SM count.
#include "tma_util.cuh"
#include <map>
#include <mutex>
#include <tuple>

namespace ob {
namespace tmau {

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

template <class FT>
bool encode(CUtensorMap* out, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides,
            const cuuint32_t* box) {
    static const EncodeFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess ||
            qr != cudaDriverEntryPointSuccess)
            return (EncodeFn) nullptr;
        return (EncodeFn)p;
    }();
    if (!fn) return false;
    const cuuint32_t es[5] = {1, 1, 1, 1, 1};
    return fn(out, sizeof(FT) == 8 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, rank,
              const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
              CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
template bool encode<float>(CUtensorMap*, const void*, int, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*);
template bool encode<double>(CUtensorMap*, const void*, int, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*);

typedef std::tuple<const void*, int, int, int, int, int, int> MapKey;
static std::map<MapKey, CUtensorMap>& map_cache() { static std::map<MapKey, CUtensorMap> c; return c; }
static std::mutex& map_mutex() { static std::mutex m; return m; }

template <class FT>
CUtensorMap make_map(const GridD<FT>& g, const FT* base, int box_x, int box_y) {
    std::lock_guard<std::mutex> lk(map_mutex());
    auto& cache = map_cache();
    auto key = std::make_tuple((const void*)base, g.S[0], g.S[1], g.S[2], (int)sizeof(FT), box_x, box_y);
    auto it = cache.find(key);
    if (it != cache.end()) return it->second;
    CUtensorMap m;
    cuuint64_t dims[3] = {(cuuint64_t)g.S[0], (cuuint64_t)g.S[1], (cuuint64_t)g.S[2]};
    cuuint64_t strides[2] = {(cuuint64_t)g.S[0] * sizeof(FT), (cuuint64_t)g.S[0] * g.S[1] * sizeof(FT)};
    cuuint32_t box[3] = {(cuuint32_t)box_x, (cuuint32_t)box_y, 1};
    if (!encode<FT>(&m, base, 3, dims, strides, box)) throw Error("cuTensorMapEncodeTiled unavailable or failed");
    cache[key] = m;
    return m;
}
template CUtensorMap make_map<float>(const GridD<float>&, const float*, int, int);
template CUtensorMap make_map<double>(const GridD<double>&, const double*, int, int);

void evict_maps(const void* base, size_t bytes) {
    std::lock_guard<std::mutex> lk(map_mutex());
    auto& cache = map_cache();
    const char* lo = (const char*)base;
    const char* hi = lo + bytes;
    for (auto it = cache.begin(); it != cache.end();) {
        const char* p = (const char*)std::get<0>(it->first);
        if (p >= lo && p < hi) it = cache.erase(it); else ++it;
    }
}
size_t cached_maps() {
    std::lock_guard<std::mutex> lk(map_mutex());
    return map_cache().size();
}

int sm_count() {
    static const int n = [] {
        int dev = 0, sms = 0;
        OB_CUDA(cudaGetDevice(&dev));
        OB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        return sms;
    }();
    return n;
}

}  // namespace tmau
}  // namespace ob
