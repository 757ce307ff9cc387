// imgcorr_tma.cuh — the TMA / mbarrier primitives every staged kernel uses (inline PTX for sm_100a) and the host-side
// tensor-map encoder.  cuTensorMapEncodeTiled is taken from the driver at run time (cudaGetDriverEntryPoint), so
// libimgcorr.so does not link libcuda and still loads on a box without a GPU.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <mutex>

namespace imgcorr {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// make freshly initialised barriers visible to the async proxy (TMA) before first use
__device__ __forceinline__ void mbar_init_fence() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
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
// tiled bulk tensor loads global -> shared, completion counted in bytes on `bar`.
// Rules that bit us: the box must start on a 16-byte boundary of the row (x * element size % 16 == 0), its width must
// be a multiple of 16 bytes, each box dimension <= 256, the shared destination 128-byte aligned.  Out-of-bounds parts
// of a box are zero-filled (and still count towards the transaction bytes).
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* tm, uint64_t* bar, int x, int y) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(tm), "r"(smem_u32(bar)), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* tm, uint64_t* bar, int x, int y, int z) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(dst)), "l"(tm), "r"(smem_u32(bar)), "r"(x), "r"(y), "r"(z) : "memory");
}

// the same with an L2 eviction-priority hint (the 64-bit policy words createpolicy.fractional produces for fraction 1.0):
// calibration maps are re-read by every launch and should outlive the frames that stream through L2 once
constexpr uint64_t L2_EVICT_NORMAL = 0x1000000000000000ull, L2_EVICT_FIRST = 0x12F0000000000000ull, L2_EVICT_LAST = 0x14F0000000000000ull;
__device__ __forceinline__ void tma_load_2d_hint(void* dst, const CUtensorMap* tm, uint64_t* bar, int x, int y, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(dst)), "l"(tm), "r"(smem_u32(bar)), "r"(x), "r"(y), "l"(policy) : "memory");
}
__device__ __forceinline__ void tma_load_3d_hint(void* dst, const CUtensorMap* tm, uint64_t* bar, int x, int y, int z, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;"
        ::"r"(smem_u32(dst)), "l"(tm), "r"(smem_u32(bar)), "r"(x), "r"(y), "r"(z), "l"(policy) : "memory");
}
// plain (1-D) bulk copy global -> shared, 16-byte aligned, size a multiple of 16 bytes, completion on `bar`
__device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ---- host ---------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_tensorMapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                             const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                             CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline PFN_tensorMapEncodeTiled tensor_map_encoder() {
    static PFN_tensorMapEncodeTiled fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (PFN_tensorMapEncodeTiled)p;
    }
    return fn;
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) and the occupancy answer are per DEVICE: a process may hold contexts on
// several devices (imgcorr_ctx_create(device, ...)), so both are cached per (device, kernel) under a lock.  Returns the
// resident CTAs per SM (>= 1), 0 with *err set on failure.
inline int blocks_per_sm_cached(const void* kern, int threads, size_t smem, cudaError_t* err) {
    constexpr int MAXDEV = 64, MAXK = 256;
    struct Entry { const void* k; int per_sm[MAXDEV]; };
    static Entry table[MAXK];
    static int used = 0;
    static std::mutex mu;
    int dev = 0;
    *err = cudaGetDevice(&dev);
    if (*err != cudaSuccess) return 0;
    std::lock_guard<std::mutex> lock(mu);
    int slot = -1;
    for (int s = 0; s < used; ++s) if (table[s].k == kern) { slot = s; break; }
    if (slot < 0 && used < MAXK) { slot = used++; table[slot].k = kern; for (int d = 0; d < MAXDEV; ++d) table[slot].per_sm[d] = 0; }
    if (slot >= 0 && dev < MAXDEV && table[slot].per_sm[dev]) return table[slot].per_sm[dev];
    *err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (*err != cudaSuccess) return 0;
    int n = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, threads, smem);
    if (n < 1) n = 1;
    if (slot >= 0 && dev < MAXDEV) table[slot].per_sm[dev] = n;
    return n;
}

// dense row-major [N][H][W] (N == 0: [H][W], rank 2) of `esz`-byte elements, box = boxw x boxh (x 1)
inline bool make_tensor_map(CUtensorMap* tm, CUtensorMapDataType dt, size_t esz, const void* ptr, int W, int H, int N,
                            int boxw, int boxh, int boxd = 1) {
    PFN_tensorMapEncodeTiled enc = tensor_map_encoder();
    if (!enc) return false;
    cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)(N > 0 ? N : 1)};
    cuuint64_t strides[2] = {(cuuint64_t)W * esz, (cuuint64_t)W * H * esz};
    cuuint32_t box[3] = {(cuuint32_t)boxw, (cuuint32_t)boxh, (cuuint32_t)boxd};
    cuuint32_t estr[3] = {1, 1, 1};
    const int rank = N > 0 ? 3 : 2;
    return enc(tm, dt, rank, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace imgcorr
