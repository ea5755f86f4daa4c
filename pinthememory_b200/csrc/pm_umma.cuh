// tcgen05 (5th-generation tensor core) plumbing for the 1x1-convolution GEMMs: TMEM allocation, shared-memory
// matrix descriptors, the instruction descriptor, single-thread MMA issue, commit -> mbarrier, TMEM -> register
// loads, and the TMA store / reduce-add path of the epilogue. Inline PTX only (sm_100a); no CUTLASS.
#pragma once
#include "pm_tma.cuh"

namespace pm {

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- TMEM: 512 columns x 128 lanes x 32 bit per SM. One warp allocates and the same warp frees. ----------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {  // whole warp, ncols = 2^n >= 32
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// ---- shared-memory matrix descriptor (64 bit), 128-byte-row swizzled layouts -----------------------------------
//   bits  0-13 start address >> 4      bits 16-29 leading byte offset >> 4     bits 32-45 stride byte offset >> 4
//   bits 46-47 version (1 on sm_100)   bits 61-63 layout type: 2 = SWIZZLE_128B (16-byte chunk ^ row%8),
//                                                              1 = SWIZZLE_128B_BASE32B (32-byte chunk ^ row%4)
// K-major operand  [rows][128 bytes of K], type 2: 8-row groups are `sbo` apart (1024 when dense); lbo unused (1).
// MN-major operand [K rows][128 bytes of M/N]: 128-byte chunks along M/N are `lbo` apart;
//   16-bit elements, type 2: 8-row K groups `sbo` apart;
//   32-bit elements (TF32) MUST use type 1: 4-row K groups `sbo` apart (the only MN-major layout tf32 has).
// These are what a TMA box with 128-byte rows writes with CU_TENSOR_MAP_SWIZZLE_128B / _128B_ATOM_32B
// (tile base 1024-byte aligned).
constexpr uint32_t UMMA_SW128 = 2, UMMA_SW128_BASE32B = 1, UMMA_SW64 = 4;  // SW64: [rows][64 bytes], 8-row groups 512 B
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                              uint32_t layout = UMMA_SW128) {
    uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)layout << 61;
    return d;
}

// ---- instruction descriptor (32 bit): fp32 accumulate, A/B format, major-ness, N>>3, M>>4 --------------------
constexpr uint32_t UMMA_FMT_BF16 = 1, UMMA_FMT_TF32 = 2;
__host__ __device__ constexpr uint32_t umma_idesc(uint32_t fmt, bool a_mn_major, bool b_mn_major, int M, int N) {
    return (1u << 4) | (fmt << 7) | (fmt << 10) | ((a_mn_major ? 1u : 0u) << 15) | ((b_mn_major ? 1u : 0u) << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// D[tmem] (+)= A[smem] . B[smem]; issued by ONE thread on behalf of the CTA
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
// mbarrier arrives when every MMA issued so far by this thread has completed (implies fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- SM pairs (cta_group::2): the two CTAs of a 2-CTA cluster run one MMA of M = 256 -------------------------------
// Rank 0 (the leader) issues every MMA. A's rows 0-127 come from the leader's shared memory and rows 128-255 from the
// peer's, B's first N/2 rows from the leader and the last N/2 from the peer, each at the same shared-memory offset as
// the descriptors name; each CTA's TMEM receives its own 128 rows of D. Every tcgen05 instruction of such a kernel uses
// cta_group::2; alloc, relinquish and dealloc are executed by one warp in EACH CTA of the pair.
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
// every thread of every CTA of the cluster; orders shared-memory (and mbarrier) accesses across the cluster
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_dst, uint32_t ncols) {  // whole warp, in both CTAs
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {  // whole warp, in both CTAs
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_tf32_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
// one arrival on the mbarrier at `bar`'s offset in every CTA of `cta_mask` once the pair MMAs issued so far have completed
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     smem_u32(bar)),
                 "h"(cta_mask)
                 : "memory");
}
// arrive on the mbarrier at `bar`'s offset in cluster CTA `cta` (release at CTA scope, as a local arrive: a cluster-scope
// release here costs microseconds per arrival and serialises the split warps -- measured, 3xTF32 wgrad 72 -> 78 us)
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
    asm volatile(
        "{\n.reg .b32 ra;\nmapa.shared::cluster.u32 ra, %0, %1;\n"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n}" ::"r"(smem_u32(bar)),
        "r"(cta)
        : "memory");
}

// 32 lanes x 32 consecutive columns: thread = lane (row of D), r[j] = column j. Warp w may only touch lanes
// 32*(w%4) .. 32*(w%4)+31. Follow with tmem_ld_wait() before using r.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- TMA store / reduce-add of a shared-memory box into a 2-D tensor map (bulk async-group completion) -------
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, int c0, int c1, const void* src) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(map)),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* map, int c0, int c1, const void* src) {
    asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(map)),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {  // <= N groups still READING their shared-memory source
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait() {  // <= N groups not yet complete (writes performed)
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

}  // namespace pm
