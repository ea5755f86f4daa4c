// TMA plumbing shared by the pipelined kernels: mbarrier + bulk-tensor-copy wrappers (device) and tensor-map
// construction through the driver entry point (host; no link-time dependency on libcuda).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>

namespace pm {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done = 0;
    for (unsigned spin = 0; !done; ++spin) {
        asm volatile(
            "{\n.reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (spin > (1u << 26)) __trap();  // a tile that never lands is a bug: fail loudly instead of hanging the GPU
    }
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
// generic-proxy writes to shared memory -> visible to the async proxy (TMA loads and stores, tensor-core operand reads);
// also needed before a TMA load overwrites a box that threads have written into
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

typedef CUresult (*pm_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                       const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                       CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static pm_encode_tiled_fn encode_tiled() {
    static pm_encode_tiled_fn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (pm_encode_tiled_fn)p;
        tried = true;
    }
    return fn;
}

// 2-D map of a row-major [rows][cols] matrix with [box_rows][box_cols] boxes; in shared memory the box is dense, or
// (swizzle128: box rows of exactly 128 bytes, destination 1024-byte aligned) has its 16-byte chunks XOR-ed with
// (row & 7) -- the bank-conflict-free layout the tensor-core tiles use.
// cuTensorMapEncodeTiled costs tens of microseconds on the host, which a launch-bound (un-captured) step cannot
// afford per kernel: maps are memoised on (address, shape, box, swizzle). A map holds no ownership, so an entry
// stays valid when the caching allocator hands the same block out again.
struct TensorMapKey {
    const void* base;
    size_t rows, cols;
    unsigned box_rows, box_cols, esz, swz, l2_256;
    bool operator==(const TensorMapKey& o) const {
        return base == o.base && rows == o.rows && cols == o.cols && box_rows == o.box_rows && box_cols == o.box_cols &&
               esz == o.esz && swz == o.swz && l2_256 == o.l2_256;
    }
};

template <typename T>
static bool make_map_2d(CUtensorMap* map, const void* base, size_t rows, size_t cols, unsigned box_rows, unsigned box_cols,
                        int swizzle128 /* 0 none, 1 SWIZZLE_128B (16-byte chunks), 2 SWIZZLE_128B_ATOM_32B (32-byte chunks), 3 SWIZZLE_64B */,
                        bool l2_256 = false /* L2 promotion: 256-byte DRAM fetches instead of 128 */) {
    constexpr int SLOTS = 128;
    static std::mutex mu;
    static TensorMapKey keys[SLOTS];
    static CUtensorMap maps[SLOTS];
    static bool used[SLOTS];
    static unsigned next = 0;
    const TensorMapKey key{base, rows, cols, box_rows, box_cols, (unsigned)sizeof(T), (unsigned)swizzle128, (unsigned)l2_256};
    std::lock_guard<std::mutex> lock(mu);
    for (int i = 0; i < SLOTS; ++i)
        if (used[i] && keys[i] == key) {
            *map = maps[i];
            return true;
        }
    pm_encode_tiled_fn enc = encode_tiled();
    if (enc == nullptr) return false;
    const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)cols * sizeof(T)};
    const cuuint32_t box[2] = {box_cols, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUtensorMapDataType dt = sizeof(T) == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    if (enc(map, dt, 2, const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            swizzle128 == 3   ? CU_TENSOR_MAP_SWIZZLE_64B
            : swizzle128 == 2 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B
            : swizzle128      ? CU_TENSOR_MAP_SWIZZLE_128B
                              : CU_TENSOR_MAP_SWIZZLE_NONE,
            l2_256 ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B : CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return false;
    const unsigned slot = next++ % SLOTS;
    keys[slot] = key, maps[slot] = *map, used[slot] = true;
    return true;
}

// round a shared-memory pointer up to a multiple of `a` bytes (a power of two); callers allocate the slack
__device__ __forceinline__ unsigned char* smem_align(unsigned char* p, unsigned a) {
    return p + ((a - (smem_u32(p) & (a - 1))) & (a - 1));
}

}  // namespace pm
