// The two 1x1 convolutions of the memory module as tcgen05 GEMMs (SURVEY.md 8f row 1).
//
// Reference: `self.output[0] = Conv2d(2C -> C, 1x1, bias=False)` (memory.py:103-104, applied at :334) and
// `Writingnet.writefeat[0] = Conv2d(C -> C, 1x1, bias=False)` (memory.py:74-75, applied at :84 / :214), plus their
// autograd (input gradient, weight gradient). On NCHW activations a 1x1 convolution is, per image b,
//     Y[b] (M x hw) = A (M x K) . X[b] (K x hw)           A = weight  (forward), weight^T (input gradient)
//     dW   (M x N)  = sum_b dY[b] (M x hw) . X[b]^T (hw x N)                         (weight gradient)
// with the PIXEL axis contiguous. Both run on the 5th-generation tensor cores:
//   * operands are staged by TMA (`cp.async.bulk.tensor.2d`, SWIZZLE_128B boxes with 128-byte rows) into a
//     shared-memory ring; the activation tile of the first form is an MN-major UMMA operand (pixels contiguous),
//     the weight tile a K-major one; in the weight-gradient form both activations are K-major (K = pixels);
//   * one elected thread issues `tcgen05.mma` (M = 128 rows of output channels, N = the pixel tile / the input
//     channels), accumulators live in TMEM (fp32, double-buffered where they fit), `tcgen05.commit` releases ring
//     slots and hands finished accumulators to the epilogue warps through mbarriers;
//   * fp32 I/O computes in 3xTF32 (hi.hi + hi.lo + lo.hi, hi = x rounded to nearest TF32, lo = x - hi exact in
//     fp32): plain TF32 (2^-11 per product) cannot hold the 1e-5 parity bar. The weights are
//     split once per call by `conv1x1_prep_kernel`; the activation tiles are split in shared memory by four
//     transform warps (same swizzled offset in a second buffer, so no layout change). bf16 I/O is one
//     `kind::f16` pass straight from the TMA tiles. PM_F32_TF32 (torch's TF32 switches on) is one `kind::tf32` pass
//     on fp32 tiles the transform warps round to nearest TF32 in place (element type Tf32OnePass);
//   * epilogue warps read TMEM with `tcgen05.ld` (thread = output channel, registers = 32 consecutive pixels), so
//     the per-channel sum and sum of squares of the BatchNorm that follows are thread-local register sums
//     (fp64 across tiles, one atomicAdd per channel per CTA); the tile goes out through a swizzled shared-memory
//     stage and a TMA store (or TMA reduce-add when the caller accumulates into an existing gradient).
#include "pm_common.cuh"
#include "pm_umma.cuh"
#include "pm_internal.h"

namespace pm {

constexpr int GEMM_THREADS = 320;  // warp 0 TMA producer, 1 MMA issuer (+TMEM owner), 2-5 epilogue, 6-9 operand split
constexpr int GEMM_RING_BYTES = 192 * 1024;
constexpr int TILE_A_BYTES = 128 * 128;  // one 128-row K-major operand block: [128 rows][128 bytes]

// fp32 I/O computed in ONE kind::tf32 pass (PM_F32_TF32): the element type of the kernels that run it. BN = the launch
// forms dz in its operand path (pm_conv1x1_dgrad_bnbwd), which needs a second activation buffer per stage.
template <bool BN>
struct Tf32OnePass {
    float v;
};

// SPLIT: 3xTF32 (hi/lo operands, three MMAs per K step); XFORM: the transform warps touch every activation tile (split or
// round it, or form dz); XBUF: activation buffers per stage; BNB: may form dz; MAXST: ring stages at most
template <typename T>
struct GemmTraits;
template <>
struct GemmTraits<float> {
    static constexpr int PXC = 32;   // elements per 128-byte row
    static constexpr int UK = 8;     // K per tcgen05.mma (32 bytes)
    static constexpr uint32_t FMT = UMMA_FMT_TF32;
    static constexpr bool SPLIT = true, XFORM = true, BNB = true;
    static constexpr int XBUF = 2, MAXST = 4;
};
template <bool BN>
struct GemmTraits<Tf32OnePass<BN>> {
    static constexpr int PXC = 32;
    static constexpr int UK = 8;
    static constexpr uint32_t FMT = UMMA_FMT_TF32;
    static constexpr bool SPLIT = false, XFORM = true, BNB = BN;
    // without lo buffers a stage is half as large: up to 6 fit the ring (the barrier block holds 4 x 6 + 2 x 2 words)
    static constexpr int XBUF = BN ? 2 : 1, MAXST = 6;
};
template <>
struct GemmTraits<__nv_bfloat16> {
    static constexpr int PXC = 64;
    static constexpr int UK = 16;
    static constexpr uint32_t FMT = UMMA_FMT_BF16;
    static constexpr bool SPLIT = false, XFORM = false, BNB = false;
    static constexpr int XBUF = 1, MAXST = 4;
};

template <typename T>
__device__ __forceinline__ void umma_issue(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
    if constexpr (sizeof(T) == 4) umma_tf32(d, a, b, idesc, acc);
    else umma_bf16(d, a, b, idesc, acc);
}

// hi = x rounded to nearest TF32 (10 mantissa bits), lo = x - hi (exact in fp32, either sign) for `n4` float4 of a
// staged tile: hi is written back in place, lo at the same offsets of `lo`. The tensor core TRUNCATES an fp32
// container to TF32, so leaving the raw value as "hi" would make every lo non-negative relative to x and the dropped
// lo.lo products a coherent bias (~2^-22 per product, measured 2e-6 on the GEMM); with round-to-nearest the residuals
// are symmetric and half as large.
// lo = x - trunc_tf32(x) only (the tensor core truncates the untouched fp32 container itself): one shared-memory write
// per element instead of two. Measured on the GEMMs: the same error as the round-to-nearest split (the 2e-6 that
// remains grows linearly with K -- it is the tensor core's truncating fp32 accumulation, not the split), so the
// activation tiles, which are split in the inner loop, take this one; the weights (split once per call) are rounded.
__device__ __forceinline__ void split_tile_trunc(const float4* __restrict__ raw, float4* __restrict__ lo, int n4, int t,
                                                 int nthreads) {
    for (int i = t; i < n4; i += nthreads) {
        const float4 v = raw[i];
        float4 l;
        l.x = v.x - __uint_as_float(__float_as_uint(v.x) & 0xffffe000u);
        l.y = v.y - __uint_as_float(__float_as_uint(v.y) & 0xffffe000u);
        l.z = v.z - __uint_as_float(__float_as_uint(v.z) & 0xffffe000u);
        l.w = v.w - __uint_as_float(__float_as_uint(v.w) & 0xffffe000u);
        lo[i] = l;
    }
}
__device__ __forceinline__ float tf32_rn(float x) { return __uint_as_float((__float_as_uint(x) + 0x00001000u) & 0xffffe000u); }
// one-pass TF32: the activation tile rounded to nearest TF32 in place. Left raw, the tensor core would truncate it, which
// lowers every operand's magnitude by up to one TF32 ulp (2^-10 relative): a bias, not noise -- a weight gradient, whose
// operands are both activations, would come out scaled down by a few 1e-4. Rounded, the errors are symmetric and cancel.
__device__ __forceinline__ void round_tile(float4* __restrict__ raw, int n4, int t, int nthreads) {
    for (int i = t; i < n4; i += nthreads) {
        float4 v = raw[i];
        v.x = tf32_rn(v.x), v.y = tf32_rn(v.y), v.z = tf32_rn(v.z), v.w = tf32_rn(v.w);
        raw[i] = v;
    }
}
__device__ __forceinline__ void split_tile(float4* __restrict__ raw, float4* __restrict__ lo, int n4, int t, int nthreads) {
    for (int i = t; i < n4; i += nthreads) {
        const float4 v = raw[i];
        float4 h, l;
        h.x = tf32_rn(v.x), h.y = tf32_rn(v.y), h.z = tf32_rn(v.z), h.w = tf32_rn(v.w);
        l.x = v.x - h.x, l.y = v.y - h.y, l.z = v.z - h.z, l.w = v.w - h.w;
        lo[i] = l;
        raw[i] = h;
    }
}

// ---- BatchNorm backward in the operand path of the input-gradient GEMM (fp32) ---------------------------------------
// The input gradient of conv -> BatchNorm (-> ReLU) is W^T . dz with dz = gamma*invstd*(g - dbeta/n - xhat*dgamma/n),
// g = dy*(y > 0), xhat = (z - mean)*invstd: an element-wise function of the incoming gradient dy and the saved
// convolution output z. Instead of a separate pass that reads both and writes dz (bn_bwd_apply, 42 us at cfg 2) the
// producer loads the dy tile AND the z tile of a stage, the operand-split warps -- which touch every element anyway --
// form dz in place (raw fp32 = the "hi" operand in the dy buffer, dz - trunc(dz) = "lo" in the z buffer) and one of
// them hands the dz tile to the TMA unit as a store, because the weight-gradient GEMM needs it too. The ReLU gate is
// recomputed from z with the forward's own expression (no mask load); only for blocks without a residual.
struct BnBwdArgs {
    const float *mean, *invstd, *gamma, *beta, *dgamma, *dbeta;  // per conv-output channel; mean == nullptr: off
    float inv_n;
    int training, relu;
};

// SPLIT (3xTF32): dz -> dy buffer (the "hi" operand and the stored tile), dz - trunc(dz) -> z buffer ("lo").
// one pass: tf32_rn(dz) -> dy buffer (the operand), dz -> z buffer (the stored tile keeps every fp32 bit).
template <int KB, bool SPLIT>
__device__ __forceinline__ void bnbwd_tile(float4* __restrict__ dy_hi, float4* __restrict__ z_lo, int n4, int t, int nthreads,
                                           int ch0, const BnBwdArgs& bn) {
    // 8 float4 per 128-byte row, KB rows per 32-pixel chunk: float4 i belongs to row (i >> 3) % KB. With 128 threads and
    // KB = 16 a thread stays on ONE row (t >> 3) for the whole tile: its channel's coefficients are loaded once.
    constexpr bool FIXED = (KB == 16);
    float is = 0.f, mu = 0.f, sc = 0.f, sh = 0.f, k1 = 0.f, k2 = 0.f;
    auto coef = [&](int c) {
        is = __ldg(bn.invstd + c), mu = __ldg(bn.mean + c);
        sc = is * __ldg(bn.gamma + c), sh = __ldg(bn.beta + c) - mu * sc;  // the forward's affine (bn_apply_kernel), same expression
        k1 = bn.training ? __ldg(bn.dbeta + c) * bn.inv_n : 0.f, k2 = bn.training ? __ldg(bn.dgamma + c) * bn.inv_n : 0.f;
    };
    if (FIXED) coef(ch0 + ((t >> 3) % KB));
    for (int i = t; i < n4; i += nthreads) {
        if (!FIXED) coef(ch0 + ((i >> 3) % KB));
        const float4 g = dy_hi[i], z = z_lo[i];
        float4 d, l;
#define PM_BNBWD_ONE(f)                                                                  \
        {                                                                                \
            const float gv = (!bn.relu || fmaf(z.f, sc, sh) > 0.f) ? g.f : 0.f;          \
            const float xh = (z.f - mu) * is;                                            \
            d.f = sc * (gv - k1 - xh * k2);                                              \
            if (SPLIT) l.f = d.f - __uint_as_float(__float_as_uint(d.f) & 0xffffe000u);  \
            else l.f = d.f, d.f = tf32_rn(d.f);                                          \
        }
        PM_BNBWD_ONE(x) PM_BNBWD_ONE(y) PM_BNBWD_ONE(z) PM_BNBWD_ONE(w)
#undef PM_BNBWD_ONE
        dy_hi[i] = d;
        z_lo[i] = l;
    }
}

// =================================================================================================================
// Form 1: Y[b] = A . X[b]   (forward convolution and input gradient)
//   mapX  : [B*K rows][hw] activations, box [KB rows][PXC pixels]           (MN-major B operand)
//   mapAh : [Mpad rows][K] weights (fp32: TF32 "hi" part; bf16: the weight), box [128 rows][KB]   (K-major A operand)
//   mapAl : fp32 only, the "lo" part
//   mapY  : [B*M rows][hw] output, box [32 rows][PXC pixels]
//   CTA tile: MT x 128 output rows (starting at 128*m_tile0) x NT pixels of one image; persistent over tiles.
// =================================================================================================================
template <typename T, int MT, int NT, int KB, bool ORD = false>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
    conv1x1_nn_kernel(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapAh,
                      const __grid_constant__ CUtensorMap mapAl, const __grid_constant__ CUtensorMap mapY, int K, int M,
                      int m_tile0, int tiles_per_img, int total_tiles, int accumulate, double* __restrict__ stats,
                      const float* __restrict__ ep_scale, const float* __restrict__ ep_shift, int ep_relu,
                      const __grid_constant__ CUtensorMap mapZ, const __grid_constant__ CUtensorMap mapDZ, const BnBwdArgs bn) {
    using TR = GemmTraits<T>;
    constexpr int PXC = TR::PXC, UK = TR::UK, KSTEPS = KB / UK;
    const bool bnbwd = TR::BNB && bn.mean != nullptr;  // X = dy, Z = saved conv output: dz formed in the split stage
    constexpr int NCH = NT / PXC;                      // 128-byte pixel chunks per tile
    constexpr int XCHUNK = KB * 128;                   // bytes of one [KB rows][128 B] chunk
    constexpr int XBYTES = NCH * XCHUNK;               // = NT * KB * sizeof(T)
    constexpr int NOPA = TR::SPLIT ? 2 : 1, XB = TR::XBUF;  // weight operands (hi[, lo]), activation buffers
    // weight block: [128 rows][KB channels] K-major; 128-byte rows use SWIZZLE_128B, 64-byte rows SWIZZLE_64B
    constexpr int AROW = KB * (int)sizeof(T);
    static_assert(AROW == 128 || AROW == 64, "weight rows must be 64 or 128 bytes");
    constexpr int TILE_A = 128 * AROW;
    constexpr uint32_t ASWZ = AROW == 128 ? UMMA_SW128 : UMMA_SW64, ASBO = 8 * AROW;
    constexpr int STAGE = XB * XBYTES + NOPA * MT * TILE_A;
    constexpr int STAGES = (GEMM_RING_BYTES / STAGE) > TR::MAXST ? TR::MAXST : (GEMM_RING_BYTES / STAGE);
    constexpr int ACC = (512 / (MT * NT)) >= 2 ? 2 : 1;  // accumulator stages in TMEM
    constexpr uint32_t TX = XBYTES + NOPA * MT * TILE_A;
    static_assert(STAGES >= 2, "ring too small");
    static_assert(MT * NT <= 512, "accumulators exceed TMEM");
    constexpr uint32_t IDESC = umma_idesc(TR::FMT, false, true, 128, NT);

    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = smem_align(smem_raw, 1024);
    unsigned char* stg = smem + STAGES * STAGE;                 // 4 warps x 2 x [32 rows][128 B]
    uint64_t* bars = reinterpret_cast<uint64_t*>(stg + 4 * 2 * 4096);
    uint64_t* full = bars;                 // [STAGES] TMA landed
    uint64_t* empty = bars + STAGES;       // [STAGES] MMAs of the stage retired
    uint64_t* xfull = bars + 2 * STAGES;   // [STAGES] activation tile transformed (fp32)
    uint64_t* accf = bars + 3 * STAGES;    // [ACC] accumulator complete
    uint64_t* acce = accf + ACC;           // [ACC] accumulator drained
    uint64_t* sfree = acce + ACC;          // [STAGES] the dz store of the stage has left shared memory (bnbwd only)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sfree + STAGES);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int i = 0; i < STAGES; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], 1);
            mbar_init(&xfull[i], 4);  // one arrival per operand-split warp
            mbar_init(&sfree[i], 1);
        }
        for (int i = 0; i < ACC; ++i) {
            mbar_init(&accf[i], 1);
            mbar_init(&acce[i], 128);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        prefetch_tmap(&mapX);
        prefetch_tmap(&mapAh);
        prefetch_tmap(&mapY);
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const int nkb = (K + KB - 1) / KB;
    const int tile0 = blockIdx.x, tile_stride = gridDim.x;  // persistent CTAs: tiles tile0, tile0 + tile_stride, ...

    if (warp == 0) {
        if (lane == 0) {  // ---------------------------------------------------------------- TMA producer
            uint32_t it = 0;
            for (int tile = tile0; tile < total_tiles; tile += tile_stride) {
                const int b = tile / tiles_per_img, px0 = (tile - b * tiles_per_img) * NT;
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = it % STAGES;
                    mbar_wait(&empty[s], ((it / STAGES) & 1) ^ 1);
                    if (bnbwd) mbar_wait(&sfree[s], ((it / STAGES) & 1) ^ 1);
                    unsigned char* st = smem + s * STAGE;
                    mbar_expect_tx(&full[s], TX + (bnbwd ? (uint32_t)XBYTES : 0u));
#pragma unroll
                    for (int c = 0; c < NCH; ++c) tma_load_2d(st + c * XCHUNK, &mapX, px0 + c * PXC, b * K + kb * KB, &full[s]);
                    if (bnbwd) {  // the saved convolution output of the same block lands where "lo" will be written
#pragma unroll
                        for (int c = 0; c < NCH; ++c)
                            tma_load_2d(st + XBYTES + c * XCHUNK, &mapZ, px0 + c * PXC, b * K + kb * KB, &full[s]);
                    }
                    unsigned char* sa = st + XB * XBYTES;
#pragma unroll
                    for (int j = 0; j < NOPA * MT; ++j) {  // weight blocks: [hi of every row tile | lo of every row tile]
                        const int mt = j % MT;
                        tma_load_2d(sa + j * TILE_A, j < MT ? &mapAh : &mapAl, kb * KB, (m_tile0 + mt) * 128, &full[s]);
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {  // ---------------------------------------------------------------- MMA issuer
            uint32_t it = 0, tc = 0;
            for (int tile = tile0; tile < total_tiles; tile += tile_stride, ++tc) {
                const int a = tc % ACC;
                mbar_wait(&acce[a], ((tc / ACC) & 1) ^ 1);
                tc_fence_after();
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    mbar_wait(&full[s], ph);
                    if (TR::XFORM) mbar_wait(&xfull[s], ph);
                    tc_fence_after();
                    const uint32_t sx = smem_u32(smem + s * STAGE);
                    const uint32_t sa = sx + XB * XBYTES;
                    int ksteps = (K - kb * KB) / UK;
                    if (ksteps > KSTEPS) ksteps = KSTEPS;
                    for (int ks = 0; ks < ksteps; ++ks) {
                        // X: MN-major, 128-byte pixel chunks XCHUNK apart, 8-row K groups 1024 bytes apart
                        // tf32 has one MN-major layout: 32-byte swizzle atoms, K groups of 4 rows (512 bytes apart)
                        constexpr uint32_t XL = sizeof(T) == 4 ? UMMA_SW128_BASE32B : UMMA_SW128;
                        constexpr uint32_t XSBO = sizeof(T) == 4 ? 512u : 1024u;
                        const uint64_t bh = umma_desc(sx + ks * (UK * 128), XCHUNK, XSBO, XL);
                        const uint64_t bl = umma_desc(sx + XBYTES + ks * (UK * 128), XCHUNK, XSBO, XL);
                        const uint32_t first = (kb | ks) ? 1u : 0u;
#pragma unroll
                        for (int mt = 0; mt < MT; ++mt) {
                            const uint32_t d = tmem + (uint32_t)((a * MT + mt) * NT);
                            const uint64_t ah = umma_desc(sa + mt * TILE_A + ks * 32, 16, ASBO, ASWZ);
                            if (TR::SPLIT) {
                                const uint64_t al = umma_desc(sa + (MT + mt) * TILE_A + ks * 32, 16, ASBO, ASWZ);
                                umma_issue<T>(d, al, bh, IDESC, first);
                                umma_issue<T>(d, ah, bl, IDESC, 1u);
                                umma_issue<T>(d, ah, bh, IDESC, 1u);
                            } else {
                                umma_issue<T>(d, ah, bh, IDESC, first);
                            }
                        }
                    }
                    umma_commit(&empty[s]);
                }
                umma_commit(&accf[a]);
            }
        }
    } else if (warp < 6) {  // ------------------------------------------------------------------ epilogue
        const int q = warp & 3;  // TMEM lane quarter this warp may read
        unsigned char* mystg = stg + q * 2 * 4096;
        int bi = 0;
        double sum[MT], sq[MT];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) sum[mt] = 0.0, sq[mt] = 0.0;
        uint32_t tc = 0;
        for (int tile = tile0; tile < total_tiles; tile += tile_stride, ++tc) {
            const int b = tile / tiles_per_img, px0 = (tile - b * tiles_per_img) * NT;
            const int a = tc % ACC;
            mbar_wait(&accf[a], (tc / ACC) & 1);
            tc_fence_after();
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
                const int row0 = (m_tile0 + mt) * 128 + q * 32;
                if (row0 >= M) continue;  // padded rows
                // optional per-row affine (+ ReLU) of the output: the eval-mode BatchNorm (+ ReLU) that follows the
                // convolution, folded into the epilogue (this thread's row = one output channel)
                const float sc = ep_scale != nullptr ? __ldg(ep_scale + row0 + lane) : 1.f;
                const float sh = ep_scale != nullptr ? __ldg(ep_shift + row0 + lane) : 0.f;
                float ts = 0.f, tq = 0.f;
                const uint32_t ta0 = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)((a * MT + mt) * NT);
                // stage one 32-row x 128-byte chunk in shared memory (swizzled) and hand it to the TMA unit
                auto emit = [&](const uint4 (&out)[8], int c) {
                    unsigned char* buf = mystg + bi * 4096;
                    bi ^= 1;
                    if (lane == 0) bulk_wait_read<1>();  // the store issued two chunks ago has left this buffer
                    __syncwarp();
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        *reinterpret_cast<uint4*>(buf + lane * 128 + ((j ^ (lane & 7)) << 4)) = out[j];
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        if (accumulate) tma_reduce_add_2d(&mapY, px0 + c * PXC, b * M + row0, buf);
                        else tma_store_2d(&mapY, px0 + c * PXC, b * M + row0, buf);
                        bulk_commit();
                    }
                };
                if constexpr (sizeof(T) == 4) {
                    // software pipeline over the chunks: the TMEM load of chunk c+1 is in flight while chunk c is reduced,
                    // staged and stored (tcgen05.wait::ld waits for everything outstanding, so exactly one load is)
                    auto process = [&](uint32_t (&r)[32], int c) {
                        if (ep_scale != nullptr) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) {
                                float v = fmaf(__uint_as_float(r[j]), sc, sh);
                                if (ep_relu) v = fmaxf(v, 0.f);
                                r[j] = __float_as_uint(v);
                            }
                        }
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const float v = __uint_as_float(r[j]);
                            ts += v;
                            tq = fmaf(v, v, tq);
                        }
                        uint4 out[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) out[j] = make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
                        emit(out, c);
                    };
                    uint32_t ra[32], rb[32];
                    tmem_ld32(ta0, ra);
#pragma unroll 1
                    for (int c = 0; c < NCH; c += 2) {
                        tmem_ld_wait();
                        if (c + 1 < NCH) tmem_ld32(ta0 + (uint32_t)((c + 1) * PXC), rb);
                        process(ra, c);
                        if (c + 1 < NCH) {
                            tmem_ld_wait();
                            if (c + 2 < NCH) tmem_ld32(ta0 + (uint32_t)((c + 2) * PXC), ra);
                            process(rb, c + 1);
                        }
                    }
                } else {
#pragma unroll 1
                    for (int c = 0; c < NCH; ++c) {
                        const uint32_t ta = ta0 + (uint32_t)(c * PXC);
                        uint4 out[8];
                        uint32_t r0[32], r1[32];
                        tmem_ld32(ta, r0);
                        tmem_ld32(ta + 32, r1);
                        tmem_ld_wait();
                        if (ep_scale != nullptr) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) {
                                float v0 = fmaf(__uint_as_float(r0[j]), sc, sh), v1 = fmaf(__uint_as_float(r1[j]), sc, sh);
                                if (ep_relu) v0 = fmaxf(v0, 0.f), v1 = fmaxf(v1, 0.f);
                                r0[j] = __float_as_uint(v0), r1[j] = __float_as_uint(v1);
                            }
                        }
                        uint32_t pk[32];
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const __nv_bfloat162 p0 = __floats2bfloat162_rn(__uint_as_float(r0[2 * j]), __uint_as_float(r0[2 * j + 1]));
                            const __nv_bfloat162 p1 = __floats2bfloat162_rn(__uint_as_float(r1[2 * j]), __uint_as_float(r1[2 * j + 1]));
                            pk[j] = *reinterpret_cast<const uint32_t*>(&p0);
                            pk[16 + j] = *reinterpret_cast<const uint32_t*>(&p1);
                            const float2 f0 = __bfloat1622float2(p0), f1 = __bfloat1622float2(p1);
                            ts += (f0.x + f0.y) + (f1.x + f1.y);
                            tq = fmaf(f0.x, f0.x, fmaf(f0.y, f0.y, fmaf(f1.x, f1.x, fmaf(f1.y, f1.y, tq))));
                        }
#pragma unroll
                        for (int j = 0; j < 8; ++j) out[j] = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
                        emit(out, c);
                    }
                }
                sum[mt] += (double)ts;
                sq[mt] += (double)tq;
            }
            tc_fence_before();
            mbar_arrive(&acce[a]);
        }
        if (lane == 0) bulk_wait<0>();
        if (stats != nullptr) {
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
                const int row = (m_tile0 + mt) * 128 + q * 32 + lane;
                if (row < M) {
                    if constexpr (ORD) {  // ordered instantiation: stats is the partial scratch, this CTA's slot is [blockIdx.x]
                        stats[(size_t)blockIdx.x * 2 * M + row] = sum[mt];
                        stats[(size_t)blockIdx.x * 2 * M + M + row] = sq[mt];
                    } else {
                        atomicAdd(&stats[row], sum[mt]);
                        atomicAdd(&stats[M + row], sq[mt]);
                    }
                }
            }
        }
    } else {  // ---------------------------------------------------------- operand transform (fp32 only)
        if constexpr (TR::XFORM) {
            const int t = threadIdx.x - 6 * 32;
            uint32_t it = 0;
            for (int tile = tile0; tile < total_tiles; tile += tile_stride) {
                const int b = tile / tiles_per_img, px0 = (tile - b * tiles_per_img) * NT;
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = it % STAGES;
                    mbar_wait(&full[s], (it / STAGES) & 1);
                    unsigned char* st = smem + s * STAGE;
                    if (bnbwd) bnbwd_tile<KB, TR::SPLIT>(reinterpret_cast<float4*>(st), reinterpret_cast<float4*>(st + XBYTES), XBYTES / 16, t, 128, kb * KB, bn);
                    else if (TR::SPLIT) split_tile_trunc(reinterpret_cast<float4*>(st), reinterpret_cast<float4*>(st + XBYTES), XBYTES / 16, t, 128);
                    else round_tile(reinterpret_cast<float4*>(st), XBYTES / 16, t, 128);
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&xfull[s]);
                    if (bnbwd && t == 0) {
                        // once all four split warps have arrived the dz tile is complete: this thread stores it (the
                        // weight-gradient GEMM reads it later) while the MMAs consume the same buffers; the stage may be
                        // refilled once the MMAs AND this store have read it
                        mbar_wait(&xfull[s], (it / STAGES) & 1);
#pragma unroll
                        for (int c = 0; c < NCH; ++c)   // (the fp32 dz: in the dy buffer for 3xTF32, in the z buffer for one pass)
                            tma_store_2d(&mapDZ, px0 + c * PXC, b * K + kb * KB, st + (TR::SPLIT ? 0 : XBYTES) + c * XCHUNK);
                        bulk_commit();
                        bulk_wait_read<1>();  // every store but the one just issued has left shared memory
                        if (it > 0) mbar_arrive(&sfree[(it - 1) % STAGES]);
                    }
                }
            }
            if (bnbwd && t == 0) bulk_wait<0>();  // the last dz tiles are in global memory before the kernel ends
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem, 512);
    }
}

template <typename T, int MT, int NT, int KB>
constexpr size_t nn_smem_bytes() {
    using TR = GemmTraits<T>;
    constexpr int NOPA = TR::SPLIT ? 2 : 1;
    constexpr int STAGE = TR::XBUF * NT * KB * (int)sizeof(T) + NOPA * MT * 128 * KB * (int)sizeof(T);
    constexpr int STAGES = (GEMM_RING_BYTES / STAGE) > TR::MAXST ? TR::MAXST : (GEMM_RING_BYTES / STAGE);
    return (size_t)STAGES * STAGE + 4 * 2 * 4096 + 256 + 1024;
}

template <typename T, int MT, int NT, int KB, bool ORD = false>
static int launch_nn(const void* X, const void* Ah, const void* Al, void* Y, double* stats, int B, int K, int M, int Mpad,
                     int hw, int m_tile0, int accumulate, const float* ep_scale, const float* ep_shift, int ep_relu,
                     cudaStream_t st, const void* Z = nullptr, void* DZ = nullptr, const BnBwdArgs* bnargs = nullptr) {
    using TR = GemmTraits<T>;
    CUtensorMap mX, mAh, mAl, mY, mZ, mDZ;
    BnBwdArgs bn{};
    if (bnargs != nullptr && Z != nullptr && DZ != nullptr) {
        if (!TR::BNB || K % KB != 0) return PM_ERR_SHAPE;
        bn = *bnargs;
        if (!make_map_2d<T>(&mZ, Z, (size_t)B * K, hw, KB, TR::PXC, 2)) return PM_ERR_ALIGN;
        if (!make_map_2d<T>(&mDZ, DZ, (size_t)B * K, hw, KB, TR::PXC, 2)) return PM_ERR_ALIGN;
    }
    constexpr int ASW = KB * (int)sizeof(T) == 128 ? 1 : 3;  // TMA swizzle of the weight boxes: 128-byte or 64-byte rows
    if (!make_map_2d<T>(&mX, X, (size_t)B * K, hw, KB, TR::PXC, sizeof(T) == 4 ? 2 : 1)) return PM_ERR_ALIGN;
    if (!make_map_2d<T>(&mAh, Ah, Mpad, K, 128, KB, ASW)) return PM_ERR_ALIGN;
    if (TR::SPLIT) {
        if (!make_map_2d<T>(&mAl, Al, Mpad, K, 128, KB, ASW)) return PM_ERR_ALIGN;
    } else {
        mAl = mAh;
    }
    if (!make_map_2d<T>(&mY, Y, (size_t)B * M, hw, 32, TR::PXC, true)) return PM_ERR_ALIGN;
    if (bn.mean == nullptr) mZ = mX, mDZ = mX;  // unused
    const int tiles_per_img = (hw + NT - 1) / NT, total = B * tiles_per_img;
    const size_t smem = nn_smem_bytes<T, MT, NT, KB>();
    const int grid = total < 148 ? total : 148;
    cudaError_t e = cudaFuncSetAttribute(conv1x1_nn_kernel<T, MT, NT, KB, ORD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    conv1x1_nn_kernel<T, MT, NT, KB, ORD><<<grid, GEMM_THREADS, smem, st>>>(mX, mAh, mAl, mY, K, M, m_tile0, tiles_per_img, total,
                                                                      accumulate, stats, ep_scale, ep_shift, ep_relu, mZ, mDZ, bn);
    e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

// =================================================================================================================
// Form 2: dW (M x N) = sum over (b, pixel) of dY[b] . X[b]^T   (weight gradient). Both operands K-major (K = pixels).
//   mapG : [B*M rows][hw] output gradient, box [128 rows][PXC pixels]      (A operand)
//   mapX : [B*Ntot rows][hw] layer input,  box [NW/2 rows][PXC pixels], NI = N / NW boxes per stage   (B operand);
//          this launch covers input channels n0 .. n0+N-1 (N <= 288) of the Ntot
//   grid : (2 * ceil(mtiles / 2), pixel chunks of every image) in clusters of 2 along x (a launch with the pair along y
//          is refused as a cluster misconfiguration): SM pair p runs row tiles 2p (rank 0, the leader) and 2p+1 (rank 1)
//          of one chunk as M = 256 cta_group::2 MMAs. Each CTA stages its own 128 dY rows and HALF of every X box (rows
//          NW/2 * rank ..), so X crosses L2 -> SM once per chunk and a stage is 34 KB per operand set instead of 52. Each CTA writes its [128][N] partial to `part`
//          part[(chunk * Mpad + row) * N + col]; wgrad_reduce_kernel sums the chunks. With an odd number of row tiles
//          the last pair's rank 1 has rows >= Mpad: it loads, splits and takes part in the MMAs, and stores nothing.
//   protocol: each CTA's producer fills its own stage (local full[s]) once the leader's commit has released it (local
//          empty[s]); its split warps (bf16: one relay thread) wait on full[s] and arrive on the LEADER's xfull[s]; the
//          leader's MMA thread waits on xfull[s] only and commits to empty[s] -- and after the last block to accf --
//          of both CTAs at once (multicast). Before exit each producer waits for the last commits on its empty
//          barriers, so no arrival is still in flight towards a CTA that has left the SM.
// =================================================================================================================
constexpr int WG_NMAX = 288;

template <typename T>
__host__ __device__ constexpr int wgrad_stage_bytes() {
    return (GemmTraits<T>::SPLIT ? 2 : 1) * (TILE_A_BYTES + WG_NMAX / 2 * 128);
}
template <typename T>
__host__ __device__ constexpr int wgrad_stages() {  // 3 in 3xTF32 (68 KB stages), 6 in one pass and bf16 (34 KB)
    return (212992 / wgrad_stage_bytes<T>()) > 6 ? 6 : (212992 / wgrad_stage_bytes<T>());
}

template <typename T>
__device__ __forceinline__ void umma_issue_pair(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
    if constexpr (sizeof(T) == 4) umma_tf32_pair(d, a, b, idesc, acc);
    else umma_bf16_pair(d, a, b, idesc, acc);
}

template <typename T>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
    conv1x1_wgrad_kernel(const __grid_constant__ CUtensorMap mapG, const __grid_constant__ CUtensorMap mapX, int M, int N,
                         int Ntot, int n0, int NW, int hw, int chunks_per_img, int blocks_per_chunk, float* __restrict__ part,
                         int Mpad) {
    using TR = GemmTraits<T>;
    constexpr int PXC = TR::PXC, UK = TR::UK, KSTEPS = PXC / UK;
    constexpr int NOPA = TR::SPLIT ? 2 : 1;
    constexpr int BBYTES = WG_NMAX / 2 * 128;  // this CTA's half of the widest X block
    constexpr int STAGE = wgrad_stage_bytes<T>();
    constexpr int STAGES = wgrad_stages<T>();
    static_assert(STAGES >= 2, "ring too small");

    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = smem_align(smem_raw, 1024);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE);
    uint64_t* full = bars;                 // [STAGES] this CTA's TMA landed
    uint64_t* empty = bars + STAGES;       // [STAGES] the pair MMAs of the stage retired (leader's multicast commit)
    uint64_t* xfull = bars + 2 * STAGES;   // [STAGES] leader only: both CTAs' tiles split (or landed, bf16)
    uint64_t* accf = bars + 3 * STAGES;    // accumulator complete (leader's multicast commit)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accf + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    if (threadIdx.x == 0) {
        for (int i = 0; i < STAGES; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], 1);
            mbar_init(&xfull[i], TR::XFORM ? 8 : 2);  // one arrival per split warp (bf16: per relay thread) of either CTA
        }
        mbar_init(accf, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        prefetch_tmap(&mapG);
        prefetch_tmap(&mapX);
    }
    if (warp == 1) tmem_alloc_pair(tmem_slot, 512);
    tc_fence_before();
    cluster_sync();  // both CTAs' barriers initialised before either arrives on the other's
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    const int mt = blockIdx.x, chunk = blockIdx.y;
    const int b = chunk / chunks_per_img, cb0 = (chunk - b * chunks_per_img) * blocks_per_chunk;
    const int nblk_img = (hw + PXC - 1) / PXC;
    int nkb = nblk_img - cb0;  // >= 1: every chunk of wgrad_split starts inside its image
    if (nkb > blocks_per_chunk) nkb = blocks_per_chunk;
    const int NI = N / NW, NH = NW / 2;
    const uint32_t TX = TILE_A_BYTES + (uint32_t)(NI * NH) * 128;

    if (warp == 0) {
        if (lane == 0) {
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % STAGES;
                mbar_wait(&empty[s], ((kb / STAGES) & 1) ^ 1);
                unsigned char* st = smem + s * STAGE;
                mbar_expect_tx(&full[s], TX);
                const int px = (cb0 + kb) * PXC;
                tma_load_2d(st, &mapG, px, b * M + mt * 128, &full[s]);
                for (int j = 0; j < NI; ++j)
                    tma_load_2d(st + NOPA * TILE_A_BYTES + j * NH * 128, &mapX, px, b * Ntot + n0 + j * NW + (int)rank * NH, &full[s]);
            }
            for (int kb = nkb; kb < nkb + STAGES; ++kb) mbar_wait(&empty[kb % STAGES], ((kb / STAGES) & 1) ^ 1);
        }
    } else if (warp == 1) {
        if (lane == 0 && rank == 0) {
            const uint32_t IDESC = umma_idesc(TR::FMT, false, false, 256, NW);
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % STAGES;
                mbar_wait(&xfull[s], (kb / STAGES) & 1);
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + s * STAGE);
                const uint32_t sb = sa + NOPA * TILE_A_BYTES;
#pragma unroll
                for (int ks = 0; ks < KSTEPS; ++ks) {
                    const uint64_t ah = umma_desc(sa + ks * 32, 16, 1024);
                    const uint64_t al = umma_desc(sa + TILE_A_BYTES + ks * 32, 16, 1024);
                    const uint32_t first = (kb | ks) ? 1u : 0u;
                    for (int j = 0; j < NI; ++j) {
                        const uint32_t d = tmem + (uint32_t)(j * NW);
                        const uint64_t bh = umma_desc(sb + j * NH * 128 + ks * 32, 16, 1024);
                        if (TR::SPLIT) {
                            const uint64_t bl = umma_desc(sb + BBYTES + j * NH * 128 + ks * 32, 16, 1024);
                            umma_issue_pair<T>(d, al, bh, IDESC, first);
                            umma_issue_pair<T>(d, ah, bl, IDESC, 1u);
                            umma_issue_pair<T>(d, ah, bh, IDESC, 1u);
                        } else {
                            umma_issue_pair<T>(d, ah, bh, IDESC, first);
                        }
                    }
                }
                umma_commit_pair(&empty[s], 0x3);
            }
            umma_commit_pair(accf, 0x3);
        }
    } else if (warp < 6) {
        const int q = warp & 3;
        mbar_wait(accf, 0);  // (also on an idle rank 1: the MMAs writing its TMEM and reading its tiles are complete)
        tc_fence_after();
        if (mt * 128 < Mpad) {
            float* dst = part + ((size_t)chunk * Mpad + mt * 128 + q * 32 + lane) * N;
            for (int c = 0; c < N / 32; ++c) {
                uint32_t r[32];
                tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(c * 32), r);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    *reinterpret_cast<uint4*>(dst + c * 32 + 4 * j) = make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
            }
        }
    } else if constexpr (TR::XFORM) {
        const int t = threadIdx.x - 6 * 32;
        for (int kb = 0; kb < nkb; ++kb) {
            const int s = kb % STAGES;
            mbar_wait(&full[s], (kb / STAGES) & 1);
            unsigned char* st = smem + s * STAGE;
            if (TR::SPLIT) {
                split_tile_trunc(reinterpret_cast<float4*>(st), reinterpret_cast<float4*>(st + TILE_A_BYTES), TILE_A_BYTES / 16, t, 128);
                split_tile_trunc(reinterpret_cast<float4*>(st + 2 * TILE_A_BYTES), reinterpret_cast<float4*>(st + 2 * TILE_A_BYTES + BBYTES),
                                 NI * NH * 8, t, 128);
            } else {
                round_tile(reinterpret_cast<float4*>(st), TILE_A_BYTES / 16, t, 128);
                round_tile(reinterpret_cast<float4*>(st + TILE_A_BYTES), NI * NH * 8, t, 128);
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(&xfull[s], 0);
        }
    } else if (warp == 6 && lane == 0) {  // bf16: the tiles go to the tensor core as they landed; relay "landed" to the leader
        for (int kb = 0; kb < nkb; ++kb) {
            const int s = kb % STAGES;
            mbar_wait(&full[s], (kb / STAGES) & 1);
            mbar_arrive_remote(&xfull[s], 0);
        }
    }
    tc_fence_before();
    cluster_sync();  // the leader's MMAs, the peer's arrivals and every commit are done in both CTAs
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc_pair(tmem, 512);
    }
}

// dW[m][n] (+)= sum over chunks of part[chunk][m][n]. 256 threads = 32 float4 columns x 8 chunk groups: every thread
// keeps its share of the chunk loads in flight, the groups meet in shared memory (fixed order: deterministic).
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float* __restrict__ part, float* __restrict__ dW, int M, int N,
                                                           int Mpad, int ldw, int col0, int nchunks, int accumulate) {
    __shared__ float4 red[8][32];
    const int col = threadIdx.x & 31, grp = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + col;  // float4 index in [M][N/4]
    const int n4 = N / 4, total = M * n4;
    const int m = i < total ? i / n4 : 0, c = i < total ? i - m * n4 : 0;
    const float4* p = reinterpret_cast<const float4*>(part) + (size_t)m * n4 + c;
    const size_t stride = (size_t)Mpad * n4;
    float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0;
    if (i < total) {
        int j = grp;
#pragma unroll 4
        for (; j + 8 < nchunks; j += 16) {
            const float4 v0 = __ldg(p + (size_t)j * stride), v1 = __ldg(p + (size_t)(j + 8) * stride);
            a0.x += v0.x, a0.y += v0.y, a0.z += v0.z, a0.w += v0.w;
            a1.x += v1.x, a1.y += v1.y, a1.z += v1.z, a1.w += v1.w;
        }
        if (j < nchunks) {
            const float4 v0 = __ldg(p + (size_t)j * stride);
            a0.x += v0.x, a0.y += v0.y, a0.z += v0.z, a0.w += v0.w;
        }
    }
    red[grp][col] = make_float4(a0.x + a1.x, a0.y + a1.y, a0.z + a1.z, a0.w + a1.w);
    __syncthreads();
    if (grp == 0 && i < total) {
        float4 r = red[0][col];
#pragma unroll
        for (int g = 1; g < 8; ++g) {
            const float4 v = red[g][col];
            r.x += v.x, r.y += v.y, r.z += v.z, r.w += v.w;
        }
        float* o = dW + (size_t)m * ldw + col0 + 4 * c;
        if (accumulate) r.x += o[0], r.y += o[1], r.z += o[2], r.w += o[3];
        *reinterpret_cast<float4*>(o) = r;
    }
}

template <typename T>
constexpr size_t wgrad_smem_bytes() {
    return (size_t)wgrad_stages<T>() * wgrad_stage_bytes<T>() + 256 + 1024;
}

static void wgrad_split(int B, int M, int hw, int pxc, int* chunks_per_img, int* blocks_per_chunk) {
    const int mtiles = (M + 127) / 128, nblk = (hw + pxc - 1) / pxc;
    int want = 148 / (mtiles * B);
    if (want < 1) want = 1;
    if (want > nblk) want = nblk;
    const int bpc = (nblk + want - 1) / want;
    *blocks_per_chunk = bpc;
    *chunks_per_img = (nblk + bpc - 1) / bpc;
}

template <typename T>
static int launch_wgrad(const void* dY, const void* X, float* part, float* dW, int B, int M, int Ntot, int n0, int N, int hw,
                        int accumulate, cudaStream_t st) {
    using TR = GemmTraits<T>;
    const int NI = N > 256 ? 2 : 1, NW = N / NI;
    // the pair instruction (M = 256) takes N % 16 == 0, N <= 256, and each CTA stages NW/2 rows of X in 8-row swizzle atoms
    if (N % NI || NW % 16 || NW > 256) return PM_ERR_SHAPE;
    const int Mpad = (M + 127) / 128 * 128, mtiles = Mpad / 128;
    int cpi, bpc;
    wgrad_split(B, M, hw, TR::PXC, &cpi, &bpc);
    CUtensorMap mG, mX;
    // 256-byte L2 promotion: a chunk walks its rows 128 bytes (one block) at a time, so every DRAM access also brings in
    // the block after it (measured: one pass 54.5 -> 50.7 us at 256x288, the other forms unchanged)
    if (!make_map_2d<T>(&mG, dY, (size_t)B * M, hw, 128, TR::PXC, true, true)) return PM_ERR_ALIGN;
    if (!make_map_2d<T>(&mX, X, (size_t)B * Ntot, hw, NW / 2, TR::PXC, true, true)) return PM_ERR_ALIGN;
    const size_t smem = wgrad_smem_bytes<T>();
    cudaError_t e = cudaFuncSetAttribute(conv1x1_wgrad_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2, attr[0].val.clusterDim.y = 1, attr[0].val.clusterDim.z = 1;  // SM pairs: row tiles 2p, 2p+1
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((mtiles + 1) / 2 * 2, B * cpi);
    cfg.blockDim = dim3(GEMM_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    e = cudaLaunchKernelEx(&cfg, conv1x1_wgrad_kernel<T>, mG, mX, M, N, Ntot, n0, NW, hw, cpi, bpc, part, Mpad);
    if (e != cudaSuccess) return (int)e;
    const int n4 = M * (N / 4);
    wgrad_reduce_kernel<<<(n4 + 31) / 32, 256, 0, st>>>(part, dW, M, N, Mpad, Ntot, n0, B * cpi, accumulate);
    e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

// A[m][k] = W[m][k] (transpose = 0, W is [M][K]) or W[k][m] (transpose = 1, W is [K][M]); rows M..Mpad-1 are zero.
// fp32: hi = W rounded to nearest TF32, lo = W - hi (both fp32 [Mpad][K]; lo == nullptr: one-pass TF32, hi only);
// bf16: hi = bf16(W).
template <typename T>
__global__ void conv1x1_prep_kernel(const float* __restrict__ W, int M, int K, int Mpad, int transpose, T* __restrict__ hi,
                                    T* __restrict__ lo) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Mpad * K) return;
    const int m = i / K, k = i - m * K;
    const float v = m < M ? (transpose ? W[(size_t)k * M + m] : W[(size_t)m * K + k]) : 0.f;
    if constexpr (sizeof(T) == 4) {
        const float h = tf32_rn(v);
        hi[i] = h;
        if (lo != nullptr) lo[i] = v - h;
    } else {
        hi[i] = __float2bfloat16_rn(v);
    }
}

// both operand layouts of one weight in ONE launch (blockIdx.y = 0: A = W, 1: A = W^T): the transposed operand of the
// input-gradient GEMM is produced next to the forward one instead of by a second launch in the backward pass
template <typename T>
__global__ void conv1x1_prep_both_kernel(const float* __restrict__ W, int R, int S, T* __restrict__ hi, T* __restrict__ lo,
                                         T* __restrict__ hiT, T* __restrict__ loT, double* __restrict__ zero,
                                         int zero_n) {
    // the statistics buffer of the BatchNorm that follows the forward GEMM is zeroed here (this launch precedes the GEMM
    // on the same stream) instead of by a fill kernel of its own
    if (blockIdx.x == 0 && blockIdx.y == 0)
        for (int z = threadIdx.x; z < zero_n; z += blockDim.x) zero[z] = 0.0;
    const int tr = blockIdx.y;
    const int M = tr ? S : R, K = tr ? R : S, Mpad = (M + 127) / 128 * 128;
    T* h_out = tr ? hiT : hi;
    T* l_out = tr ? loT : lo;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Mpad * K) return;
    const int m = i / K, k = i - m * K;
    const float v = m < M ? (tr ? W[(size_t)k * M + m] : W[(size_t)m * K + k]) : 0.f;
    if constexpr (sizeof(T) == 4) {
        const float h = tf32_rn(v);
        h_out[i] = h;
        if (l_out != nullptr) l_out[i] = v - h;
    } else {
        h_out[i] = __float2bfloat16_rn(v);
    }
}

}  // namespace pm

using namespace pm;

extern "C" {

int pm_conv1x1_prep_both(const float* W, int R, int S, int dtype, void* A_hi, void* A_lo, void* At_hi, void* At_lo, double* zero,
                         int zero_n, void* stream) {
    if (!W || !A_hi || !At_hi || (dtype == PM_F32 && (!A_lo || !At_lo))) return PM_ERR_NULL;
    if (dtype != PM_F32 && dtype != PM_BF16 && dtype != PM_F32_TF32) return PM_ERR_DTYPE;
    if (R <= 0 || S <= 0 || zero_n < 0 || (zero_n > 0 && !zero)) return PM_ERR_SHAPE;
    const int n0 = (R + 127) / 128 * 128 * S, n1 = (S + 127) / 128 * 128 * R, n = n0 > n1 ? n0 : n1;
    cudaStream_t st = (cudaStream_t)stream;
    const dim3 grid((n + 255) / 256, 2);
    if (dtype == PM_F32)
        conv1x1_prep_both_kernel<float><<<grid, 256, 0, st>>>(W, R, S, (float*)A_hi, (float*)A_lo, (float*)At_hi, (float*)At_lo, zero, zero_n);
    else if (dtype == PM_F32_TF32)
        conv1x1_prep_both_kernel<float><<<grid, 256, 0, st>>>(W, R, S, (float*)A_hi, nullptr, (float*)At_hi, nullptr, zero, zero_n);
    else
        conv1x1_prep_both_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(W, R, S, (__nv_bfloat16*)A_hi, nullptr, (__nv_bfloat16*)At_hi, nullptr, zero, zero_n);
    PM_CHECK_LAUNCH();
    return 0;
}

int pm_conv1x1_prep(const float* W, int M, int K, int transpose, int dtype, void* A_hi, void* A_lo, void* stream) {
    if (!W || !A_hi || (dtype == PM_F32 && !A_lo)) return PM_ERR_NULL;
    if (dtype != PM_F32 && dtype != PM_BF16 && dtype != PM_F32_TF32) return PM_ERR_DTYPE;
    if (M <= 0 || K <= 0) return PM_ERR_SHAPE;
    const int Mpad = (M + 127) / 128 * 128, n = Mpad * K;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == PM_F32)
        conv1x1_prep_kernel<float><<<(n + 255) / 256, 256, 0, st>>>(W, M, K, Mpad, transpose, (float*)A_hi, (float*)A_lo);
    else if (dtype == PM_F32_TF32)
        conv1x1_prep_kernel<float><<<(n + 255) / 256, 256, 0, st>>>(W, M, K, Mpad, transpose, (float*)A_hi, nullptr);
    else
        conv1x1_prep_kernel<__nv_bfloat16><<<(n + 255) / 256, 256, 0, st>>>(W, M, K, Mpad, transpose, (__nv_bfloat16*)A_hi, nullptr);
    PM_CHECK_LAUNCH();
    return 0;
}

extern "C++" {  // (templates inside the extern "C" block)
// the fp32 tile shapes: 256-pixel tiles and 16-channel blocks -- a tile pulls the weights of its row tiles through the
// SM's L2 port once per 256 pixels instead of once per 128 (the measured bound of the 128-pixel version); small maps keep
// 128-pixel tiles so that more than a handful of SMs get work
template <typename T, bool ORD>
static int launch_f32_tiles(bool wide, int mt, const void* X, const void* A_hi, const void* A_lo, void* Y, double* stats, int B,
                            int K, int M, int Mpad, int hw, int t0, int accumulate, const float* ep_scale, const float* ep_shift,
                            int ep_relu, cudaStream_t st, const void* Z, void* DZ, const BnBwdArgs* bn) {
    if (wide)
        return mt == 2 ? launch_nn<T, 2, 256, 16, ORD>(X, A_hi, A_lo, Y, stats, B, K, M, Mpad, hw, t0, accumulate, ep_scale, ep_shift, ep_relu, st, Z, DZ, bn)
                       : launch_nn<T, 1, 256, 16, ORD>(X, A_hi, A_lo, Y, stats, B, K, M, Mpad, hw, t0, accumulate, ep_scale, ep_shift, ep_relu, st, Z, DZ, bn);
    return mt == 2 ? launch_nn<T, 2, 128, 32, ORD>(X, A_hi, A_lo, Y, stats, B, K, M, Mpad, hw, t0, accumulate, ep_scale, ep_shift, ep_relu, st, Z, DZ, bn)
                   : launch_nn<T, 1, 128, 32, ORD>(X, A_hi, A_lo, Y, stats, B, K, M, Mpad, hw, t0, accumulate, ep_scale, ep_shift, ep_relu, st, Z, DZ, bn);
}

template <bool ORD = false>
static int conv1x1_fwd_impl(const void* X, const void* A_hi, const void* A_lo, void* Y, double* stats, int B, int K, int M, int hw,
                            int accumulate, const float* ep_scale, const float* ep_shift, int ep_relu, int dtype, void* stream,
                            const void* Z = nullptr, void* DZ = nullptr, const BnBwdArgs* bn = nullptr) {
    if (!X || !A_hi || !Y || (dtype == PM_F32 && !A_lo) || ((ep_scale == nullptr) != (ep_shift == nullptr))) return PM_ERR_NULL;
    if (dtype != PM_F32 && dtype != PM_BF16 && dtype != PM_F32_TF32) return PM_ERR_DTYPE;
    const bool f32 = dtype != PM_BF16;
    const int esz = f32 ? 4 : 2, uk = f32 ? 8 : 16;
    if (B <= 0 || hw <= 0 || K <= 0 || M <= 0 || K % uk || M % 32 || M > 512) return PM_ERR_SHAPE;
    if ((hw * esz) % 16 || ((uintptr_t)X | (uintptr_t)Y | (uintptr_t)A_hi | (uintptr_t)A_lo) % 16) return PM_ERR_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    const int Mpad = (M + 127) / 128 * 128, mtiles = Mpad / 128;
    // two 128-row tiles per CTA where possible (the activation tile is read once for both), then the remainder
    for (int t0 = 0; t0 < mtiles; t0 += 2) {
        const int mt = mtiles - t0 >= 2 ? 2 : 1;
        int rc;
        const bool wide = (long long)B * ((hw + 255) / 256) >= 96;
        if (f32) {
            // fused BatchNorm backward: the FIRST launch forms dz from (X = dy, Z) in its operand path and stores it to DZ
            // (every launch walks all K operand channels of its pixel tiles); the remaining row tiles read DZ
            const bool first = bn != nullptr && t0 == 0;
            const void* Xin = (bn != nullptr && t0 > 0) ? DZ : X;
            const void* Zi = first ? Z : nullptr;
            void* DZo = first ? DZ : nullptr;
            const BnBwdArgs* bi = first ? bn : nullptr;
            if (dtype == PM_F32)
                rc = launch_f32_tiles<float, ORD>(wide, mt, Xin, A_hi, A_lo, Y, stats, B, K, M, Mpad, hw, t0, accumulate, ep_scale, ep_shift, ep_relu, st, Zi, DZo, bi);
            else if (bi == nullptr)
                rc = launch_f32_tiles<Tf32OnePass<false>, ORD>(wide, mt, Xin, A_hi, A_hi, Y, stats, B, K, M, Mpad, hw, t0, accumulate, ep_scale, ep_shift, ep_relu, st, Zi, DZo, bi);
            else   // (only pm_conv1x1_dgrad_bnbwd forms dz, never with ordered statistics)
                rc = launch_f32_tiles<Tf32OnePass<true>, false>(wide, mt, Xin, A_hi, A_hi, Y, stats, B, K, M, Mpad, hw, t0, accumulate, ep_scale, ep_shift, ep_relu, st, Zi, DZo, bi);
        } else {
            rc = mt == 2 ? launch_nn<__nv_bfloat16, 2, 128, 64, ORD>(X, A_hi, A_lo, Y, stats, B, K, M, Mpad, hw, t0, accumulate, ep_scale, ep_shift, ep_relu, st)
                         : launch_nn<__nv_bfloat16, 1, 128, 64, ORD>(X, A_hi, A_lo, Y, stats, B, K, M, Mpad, hw, t0, accumulate, ep_scale, ep_shift, ep_relu, st);
        }
        if (rc) return rc;
    }
    return 0;
}
}  // extern "C++"

int pm_conv1x1_fwd(const void* X, const void* A_hi, const void* A_lo, void* Y, double* stats, int B, int K, int M, int hw,
                   int accumulate, int dtype, void* stream) {
    return conv1x1_fwd_impl(X, A_hi, A_lo, Y, stats, B, K, M, hw, accumulate, nullptr, nullptr, 0, dtype, stream);
}

// CTAs of the forward GEMM: each stores one [sum | sum of squares] partial in the ordered variant
static int conv1x1_fwd_ctas(int B, int hw, int dtype) {
    const bool wide = dtype != PM_BF16 && (long long)B * ((hw + 255) / 256) >= 96;   // as conv1x1_fwd_impl chooses NT
    const long long total = (long long)B * ((hw + (wide ? 255 : 127)) / (wide ? 256 : 128));
    return (int)(total < 148 ? total : 148);
}

int pm_conv1x1_stats_scratch_bytes(int B, int M, int hw, int dtype) {
    if (dtype != PM_F32 && dtype != PM_BF16 && dtype != PM_F32_TF32) return PM_ERR_DTYPE;
    if (B <= 0 || hw <= 0 || M <= 0 || M % 32 || M > 512) return PM_ERR_SHAPE;
    return conv1x1_fwd_ctas(B, hw, dtype) * 2 * M * (int)sizeof(double);
}

int pm_conv1x1_fwd_ordered(const void* X, const void* A_hi, const void* A_lo, void* Y, double* stats, double* scratch, int B,
                           int K, int M, int hw, int dtype, void* stream) {
    if (!stats || !scratch) return PM_ERR_NULL;
    if (((uintptr_t)stats | (uintptr_t)scratch) & 7) return PM_ERR_ALIGN;
    // every CTA stores its fp64 [sum | sq] rows to `scratch` (all row tiles of one call share the grid), then one
    // fixed-order reduction adds them into stats
    if (int rc = conv1x1_fwd_impl<true>(X, A_hi, A_lo, Y, scratch, B, K, M, hw, 0, nullptr, nullptr, 0, dtype, stream)) return rc;
    return pm::reduce_partials_f64(stats, scratch, conv1x1_fwd_ctas(B, hw, dtype), 2LL * M, (cudaStream_t)stream);
}

int pm_conv1x1_dgrad_bnbwd(const void* dY, const void* Z, const void* A_hi, const void* A_lo, void* dX, void* dZ,
                           const float* mean, const float* invstd, const float* gamma, const float* beta, const float* dgamma,
                           const float* dbeta, int relu, int training, int B, int K, int M, int hw, int dtype, void* stream) {
    if (!Z || !dZ || !mean || !invstd || !gamma || !beta || !dgamma || !dbeta) return PM_ERR_NULL;
    if (dtype != PM_F32 && dtype != PM_F32_TF32) return PM_ERR_DTYPE;  // the operand path transforms fp32 tiles; bf16 keeps the separate pass
    if (K % 32 || ((uintptr_t)Z | (uintptr_t)dZ) % 16) return PM_ERR_ALIGN;
    BnBwdArgs bn{mean, invstd, gamma, beta, dgamma, dbeta, 1.f / ((float)B * (float)hw), training, relu};
    return conv1x1_fwd_impl(dY, A_hi, A_lo, dX, nullptr, B, K, M, hw, 0, nullptr, nullptr, 0, dtype, stream, Z, dZ, &bn);
}

int pm_conv1x1_fwd_affine(const void* X, const void* A_hi, const void* A_lo, void* Y, const float* scale, const float* shift,
                          int relu, int B, int K, int M, int hw, int dtype, void* stream) {
    if (!scale || !shift) return PM_ERR_NULL;
    return conv1x1_fwd_impl(X, A_hi, A_lo, Y, nullptr, B, K, M, hw, 0, scale, shift, relu, dtype, stream);
}

int pm_conv1x1_wgrad_workspace_floats(int B, int M, int N, int hw, int dtype) {
    if (B <= 0 || M <= 0 || N <= 0 || hw <= 0) return 0;
    int cpi, bpc;
    wgrad_split(B, M, hw, (dtype == PM_F32 || dtype == PM_F32_TF32) ? 32 : 64, &cpi, &bpc);
    const int Mpad = (M + 127) / 128 * 128;
    const int nmax = N > WG_NMAX ? WG_NMAX : N;
    return B * cpi * Mpad * nmax;
}

int pm_conv1x1_wgrad(const void* dY, const void* X, float* workspace, float* dW, int B, int M, int N, int hw, int accumulate,
                     int dtype, void* stream) {
    if (!dY || !X || !workspace || !dW) return PM_ERR_NULL;
    if (dtype != PM_F32 && dtype != PM_BF16 && dtype != PM_F32_TF32) return PM_ERR_DTYPE;
    const int esz = dtype == PM_BF16 ? 2 : 4;
    if (B <= 0 || hw <= 0 || M <= 0 || N <= 0 || M % 32 || N % 32 || M > 512 || N > 1024) return PM_ERR_SHAPE;
    if ((hw * esz) % 16 || ((uintptr_t)X | (uintptr_t)dY | (uintptr_t)workspace | (uintptr_t)dW) % 16) return PM_ERR_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    // column blocks of at most WG_NMAX input channels (TMEM: 128 lanes x 512 columns; ring: 3 x 68 KB); blocks wider
    // than 256 channels take two N/2-wide instructions, so they must be multiples of 32 channels
    for (int n0 = 0; n0 < N;) {
        int nb = N - n0;
        if (nb > WG_NMAX) nb = 256;
        const int rc = dtype == PM_F32        ? launch_wgrad<float>(dY, X, workspace, dW, B, M, N, n0, nb, hw, accumulate, st)
                       : dtype == PM_F32_TF32 ? launch_wgrad<Tf32OnePass<false>>(dY, X, workspace, dW, B, M, N, n0, nb, hw, accumulate, st)
                                              : launch_wgrad<__nv_bfloat16>(dY, X, workspace, dW, B, M, N, n0, nb, hw, accumulate, st);
        if (rc) return rc;
        n0 += nb;
    }
    return 0;
}

}  // extern "C"
