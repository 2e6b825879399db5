// tma_util.cuh -- PTX helpers (mbarrier, cp.async.bulk, cp.async.bulk.tensor) of the TMA-staged kernels: the tendency
// kernels (tendency_tma.cu, tendency_fused.cu) and the FFT passes (fft_tma.cuh, fft_xtma.cuh).  The host half, in
// tma_util.cu: tensor-map encoding, the tensor-map cache and the SM count.
#pragma once
#include "common.cuh"
#include <cuda.h>

namespace ob {
namespace tmau {

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// after the last mbar_init, before the barriers are used (by the other threads or the async proxy)
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    unsigned ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* tm, int x, int y, int z, unsigned long long* bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(smem_u32(dst)), "l"(tm), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* tm, int x, int y, int z, int w, unsigned long long* bar) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
        ::"r"(smem_u32(dst)), "l"(tm), "r"(x), "r"(y), "r"(z), "r"(w), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* tm, int x, int y, int z, const void* src) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%1, %2, %3}], [%4];"
                 ::"l"(tm), "r"(x), "r"(y), "r"(z), "r"(smem_u32(src)) : "memory");
}
// 1-D bulk copy of `bytes` contiguous bytes (a multiple of 16, both addresses 16-byte aligned)
__device__ __forceinline__ void bulk_load(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// tiled tensor map over `base` (element type FT), rank `rank`: dims[rank], byte strides of dims 1..rank-1, box[rank];
// element strides 1, no interleave, no swizzle, L2 promotion 128B, no out-of-bounds fill.  False if the driver lacks the
// tiled-encode entry point or rejects the map.
template <class FT>
bool encode(CUtensorMap* out, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides,
            const cuuint32_t* box);

// 3-D tiled map over a field in the internal layout (common.cuh), box (box_x, box_y, 1); throws if it cannot be encoded.
// Encodings are cached per (address, extents, element size, box); evict_maps() drops the entries of a freed allocation
// (called by the field destructor, so a recycled address can never meet a stale entry and the cache stays bounded).
template <class FT> CUtensorMap make_map(const GridD<FT>& g, const FT* base, int box_x, int box_y);
void evict_maps(const void* base, size_t bytes);
size_t cached_maps();

// multiprocessor count of the device (queried once: the devices of a process are one model), for persistent grids
int sm_count();

}  // namespace tmau
}  // namespace ob
