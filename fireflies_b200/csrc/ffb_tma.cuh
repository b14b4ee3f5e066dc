// mbarrier / TMA (cp.async.bulk.tensor) helpers for sm_100a and the host-side tensor-map encoder lookup.
// Not part of the public ABI.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

namespace ffb {
namespace tma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!done);
}
// true in exactly one lane of a converged warp.  With this predicate (instead of `lane == 0`) the compiler issues the
// uniform-datapath TMA instruction once under the elected predicate; under an ordinary divergent branch it wraps every
// UTMALDG in an ELECT / BRA.U.ANY loop over the active lanes.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// one box of a rank-3 tensor map -> shared memory; completion is signalled on `bar` as transaction bytes
__device__ __forceinline__ void load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int x, int y, int z) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(x), "r"(y), "r"(z) : "memory");
}

// shared memory -> one box of a rank-3 tensor map (texels outside the tensor are clipped); bulk-group completion
__device__ __forceinline__ void store_3d(const CUtensorMap* map, const void* src, int x, int y, int z) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4}], [%1];"
                 ::"l"(map), "r"(smem_u32(src)), "r"(x), "r"(y), "r"(z) : "memory");
}
__device__ __forceinline__ void store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// the sources of all but the newest N committed store groups have been read: their shared memory may be overwritten
template <int N>
__device__ __forceinline__ void store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
// generic-proxy shared-memory writes of this thread become visible to the async proxy (TMA)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// fp32 [d2, d1, d0] row-major tensor (d0 innermost), box {b0, b1, 1}.  Returns false when TMA cannot describe it
// (unaligned base, row pitch not a multiple of 16 bytes, or no driver entry point).
inline bool encode_f32_3d(CUtensorMap* map, const float* base, uint64_t d0, uint64_t d1, uint64_t d2, uint32_t b0, uint32_t b1,
                          CUtensorMapSwizzle swizzle) {
    memset(map, 0, sizeof(*map));
    EncodeTiledFn enc = get_encode();
    if (!enc || !base || (reinterpret_cast<uintptr_t>(base) & 15) != 0 || (d0 & 3) != 0) return false;
    cuuint64_t gdim[3] = {d0, d1, d2};
    cuuint64_t gstr[2] = {d0 * 4, d0 * d1 * 4};
    cuuint32_t box[3] = {b0, b1, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace tma
}  // namespace ffb
