// Shared device helpers for the pinmem-b200 kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pinmem_b200.h"

#define PM_IGNORE_LABEL 255
#define PM_NORM_EPS 1e-12f  // F.normalize eps (reference memory.py:215,239,319)

#define PM_CHECK_LAUNCH()                                   \
    do {                                                    \
        cudaError_t e__ = cudaGetLastError();               \
        if (e__ != cudaSuccess) return (int)e__;            \
    } while (0)

namespace pm {

template <typename T>
__device__ __forceinline__ float ldf(const T* p);
template <>
__device__ __forceinline__ float ldf<float>(const float* p) {
    return __ldg(p);
}
template <>
__device__ __forceinline__ float ldf<__nv_bfloat16>(const __nv_bfloat16* p) {
    return __bfloat162float(__ldg(p));
}
template <typename T>
__device__ __forceinline__ void stf(T* p, float v);
template <>
__device__ __forceinline__ void stf<float>(float* p, float v) {
    *p = v;
}
template <>
__device__ __forceinline__ void stf<__nv_bfloat16>(__nv_bfloat16* p, float v) {
    *p = __float2bfloat16_rn(v);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// ---- Ampere-style async copies (LDGSTS): 16-byte global -> shared, zero-filled when !valid ----------
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src, bool valid) {
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    int bytes = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(gmem_src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}

// Load one [ROWS x 32 pixel] tile of an NCHW map into shared memory (dense rows of 32 elements) with
// 16-byte async copies. `base` points at element (row 0, pixel 0 of the image); rows are `hw` apart.
// Requires hw % (16/sizeof(T)) == 0 and 16-byte aligned base (checked by the host dispatcher).
template <typename T, int ROWS, int NTHREADS>
__device__ __forceinline__ void tile_load_async(T* smem_tile, const T* __restrict__ base, int hw, int px0) {
    constexpr int EPC = 16 / (int)sizeof(T);  // elements per 16-byte chunk
    constexpr int CPR = 32 / EPC;             // chunks per tile row
    static_assert(NTHREADS % CPR == 0, "thread count must be a multiple of the chunks per row");
    const int ch = threadIdx.x % CPR;
    const int px = px0 + ch * EPC;
    const bool valid = px < hw;
    const T* src = base + (size_t)(threadIdx.x / CPR) * hw + (valid ? px : 0);
    const size_t step = (size_t)(NTHREADS / CPR) * hw;
    T* dst = smem_tile + (threadIdx.x / CPR) * 32 + ch * EPC;
    for (int row = threadIdx.x / CPR; row < ROWS; row += NTHREADS / CPR) {
        cp_async16(dst, src, valid);
        src += step;
        dst += (NTHREADS / CPR) * 32;
    }
}

// Same tile, but the 16-byte chunks of every row are XOR-swizzled so that a warp whose lanes are CHANNELS
// (32 consecutive rows) can read one chunk per lane with LDS.128 without bank conflicts:
// physical chunk = chunk ^ swz(row), swz(row) = (row / (128 / row_bytes)) & (chunks_per_row - 1).
template <typename T>
__device__ __forceinline__ int tile_swz(int row) {
    constexpr int CPR = 32 * (int)sizeof(T) / 16;
    constexpr int RPL = 128 / (32 * (int)sizeof(T));  // rows per 128-byte bank window
    return (row / RPL) & (CPR - 1);
}
template <typename T, int ROWS, int NTHREADS>
__device__ __forceinline__ void tile_load_async_swz(T* smem_tile, const T* __restrict__ base, int hw, int px0) {
    constexpr int EPC = 16 / (int)sizeof(T);
    constexpr int CPR = 32 / EPC;
    static_assert(NTHREADS % CPR == 0, "thread count must be a multiple of the chunks per row");
    const int ch = threadIdx.x % CPR;
    const int px = px0 + ch * EPC;
    const bool valid = px < hw;
    const T* src = base + (size_t)(threadIdx.x / CPR) * hw + (valid ? px : 0);
    const size_t step = (size_t)(NTHREADS / CPR) * hw;
    for (int row = threadIdx.x / CPR; row < ROWS; row += NTHREADS / CPR) {
        cp_async16(smem_tile + row * 32 + (ch ^ tile_swz<T>(row)) * EPC, src, valid);
        src += step;
    }
}

// fp32 tile for the tensor-core (mma.sync) contraction: 16-byte chunk c of row r is stored at chunk c ^ (r & 7)
// -- the TMA SWIZZLE_128B pattern, so the same tile can be filled by cp.async or by a tensor-map box. The A-fragment
// loads of m16n8k8 (lanes = 8 pixels x 4 rows 2t+h of an 8-row step) then hit 32 distinct banks. A lane that wants
// pixel `px` of row `r` reads word mma_tile_pos(px, r & 7).
__device__ __forceinline__ int mma_tile_pos(int px, int swz) { return (((px >> 2) ^ swz) << 2) | (px & 3); }
template <int ROWS, int NTHREADS>
__device__ __forceinline__ void tile_load_async_mma(float* smem_tile, const float* __restrict__ base, int hw, int px0) {
    static_assert(NTHREADS % 8 == 0, "thread count must be a multiple of the chunks per row");
    const int ch = threadIdx.x % 8;
    const int px = px0 + ch * 4;
    const bool valid = px < hw;
    const float* src = base + (size_t)(threadIdx.x / 8) * hw + (valid ? px : 0);
    const size_t step = (size_t)(NTHREADS / 8) * hw;
    for (int row = threadIdx.x / 8; row < ROWS; row += NTHREADS / 8) {
        cp_async16(smem_tile + row * 32 + ((ch ^ (row & 7)) << 2), src, valid);
        src += step;
    }
}

// hi/lo split for 3xTF32. The tensor core ignores the low 13 mantissa bits of a TF32 operand, so the raw fp32
// bits serve as "hi" (= x truncated to 10 mantissa bits) and lo = x - trunc(x) is exact in fp32: one LOP3 and one
// FADD per value (cvt.rna.tf32 is emulated with ~5 instructions on sm_100 and bought nothing measurable).
__device__ __forceinline__ unsigned tf32_hi(float x) { return __float_as_uint(x); }
__device__ __forceinline__ unsigned tf32_lo(float x) {
    return __float_as_uint(x - __uint_as_float(__float_as_uint(x) & 0xffffe000u));
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], unsigned a0, unsigned a1, unsigned a2, unsigned a3, unsigned b0,
                                         unsigned b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// ---- BatchNorm per-channel step and element expression, shared by every kernel that forms a normalised value ---------
// (pm_bn.cu's normalise pass and the writing net's fused class-sum / write-backward kernels): one source, so the writing
// net's features, and the ReLU gate they imply, are the same bits whichever kernel forms them.
struct BnFinalize {  // stats == nullptr: mean / invstd are given
    const double* stats;
    const double* n_dev;  // NULL, or the element count on the device (SyncBatchNorm: the all-reduced global count)
    double n;
    float eps, momentum;
    float *mean_out, *invstd_out, *running_mean, *running_var;
    long long* num_batches_tracked;  // NULL, or nn.BatchNorm2d's counter: bumped here instead of by a torch add kernel
};
// mean and 1/sqrt(var + eps) of channel c from the convolution epilogue's fp64 [sum | sum of squares]; `publish`: also store
// them for the backward and update the running statistics (exactly one thread per channel and call may publish)
__device__ __forceinline__ void bn_finalize_channel(const BnFinalize& fin, int c, int C, bool publish, float& mu, float& is) {
    const double n = fin.n_dev != nullptr ? *fin.n_dev : fin.n;
    const double m = fin.stats[c] / n;
    double var = fin.stats[C + c] / n - m * m;
    if (var < 0.0) var = 0.0;
    mu = (float)m;
    is = (float)(1.0 / sqrt(var + (double)fin.eps));
    if (publish) {
        fin.mean_out[c] = mu;
        fin.invstd_out[c] = is;
        if (fin.running_mean != nullptr) {  // PyTorch: running_var takes the unbiased estimate
            const double unb = n > 1.0 ? var * n / (n - 1.0) : var;
            fin.running_mean[c] = (float)((1.0 - fin.momentum) * fin.running_mean[c] + fin.momentum * m);
            fin.running_var[c] = (float)((1.0 - fin.momentum) * fin.running_var[c] + fin.momentum * unb);
        }
    }
}
// y = z * sc + sh is the normalise + affine: sc = invstd * gamma, sh = beta - mean * sc
__device__ __forceinline__ void bn_scale_shift(float mu, float is, float gamma, float beta, float& sc, float& sh) {
    sc = is * gamma;
    sh = beta - mu * sc;
}
__device__ __forceinline__ float bn_affine(float z, float sc, float sh) { return fmaf(z, sc, sh); }
// the writing net's output relu(x + BN(z)) (reference memory.py:84-86)
__device__ __forceinline__ float bn_res_relu(float z, float sc, float sh, float x) { return fmaxf(bn_affine(z, sc, sh) + x, 0.f); }

__device__ __forceinline__ float to_float(float v) { return v; }
__device__ __forceinline__ float to_float(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float tile_get(const float* t, int row, int px) { return t[row * 32 + px]; }
__device__ __forceinline__ float tile_get(const __nv_bfloat16* t, int row, int px) {
    return __bfloat162float(t[row * 32 + px]);
}

// Bilinear (align_corners=True) source index of output index `dst`: PyTorch computes
// src = scale * dst in fp32, i0 = floor(src) clamped to in-1, lambda = src - i0.
__device__ __forceinline__ int src_index(float scale, int dst, int n_in, float* lambda) {
    float src = scale * (float)dst;
    int i0 = (int)src;
    if (i0 > n_in - 1) i0 = n_in - 1;
    float l = src - (float)i0;
    *lambda = fminf(fmaxf(l, 0.f), 1.f);
    return i0;
}

// ATen's align_corners=True source index and lambda (upsample_bilinear2d_out_frame): src = scale * dst in fp32,
// i0 = trunc(src) clamped to n_in - 1, lambda = src - i0. Round-to-nearest intrinsics keep nvcc from contracting them
// into an FFMA, so the tap set is exactly torch's.
__device__ __forceinline__ int tap(float scale, int dst, int n_in, float* lambda) {
    const float src = __fmul_rn(scale, (float)dst);
    int i0 = (int)src;
    if (i0 > n_in - 1) i0 = n_in - 1;
    *lambda = __fsub_rn(src, (float)i0);
    return i0;
}

// ATen's interpolated value h0λ·(w0λ·a + w1λ·b) + h1λ·(w0λ·c + w1λ·d) as nvcc contracts it in torch's sm_100 build
// (fp32 and bf16 instantiations alike): fma(h0, fma(w0, a, w1 * b), h1 * fma(w0, c, w1 * d)).
__device__ __forceinline__ float lerp4(float h0, float h1, float w0, float w1, float a, float b, float c, float d) {
    return __fmaf_rn(h0, __fmaf_rn(w0, a, __fmul_rn(w1, b)), __fmul_rn(h1, __fmaf_rn(w0, c, __fmul_rn(w1, d))));
}
__device__ __forceinline__ float2 lerp4(float2 h0, float2 h1, float2 w0, float2 w1, float2 a, float2 b, float2 c, float2 d) {
    return __ffma2_rn(h0, __ffma2_rn(w0, a, __fmul2_rn(w1, b)), __fmul2_rn(h1, __ffma2_rn(w0, c, __fmul2_rn(w1, d))));
}

// The (<=4) label taps a feature pixel samples when the (K+1)-channel one-hot label map is
// bilinearly down-sampled to the feature grid (reference memory.py:220-223). Equal classes
// are merged; unused slots get weight 0. Class K is the ignore slot.
struct LabelTaps {
    int cls[4];
    float w[4];
};

__device__ __forceinline__ int map_label(long long v, int K) {
    return (v >= 0 && v < K) ? (int)v : K;  // 255 (and anything out of range) -> ignore slot
}

// `lab` is one image's label map: int64 class ids as the reference hands them over (u8 = 0), or the packed uint8
// class map of pm_labels_pack (u8 = 1: 0..K-1, K = ignore).
__device__ __forceinline__ int fetch_label(const void* __restrict__ lab, size_t i, int u8, int K) {
    if (u8) {
        const int v = (int)__ldg(reinterpret_cast<const unsigned char*>(lab) + i);
        return v < K ? v : K;
    }
    return map_label(__ldg(reinterpret_cast<const long long*>(lab) + i), K);
}
__device__ __forceinline__ const void* label_image(const void* labels, size_t image_offset, int u8) {
    return reinterpret_cast<const char*>(labels) + image_offset * (u8 ? 1 : 8);
}

__device__ __forceinline__ LabelTaps label_taps(const void* __restrict__ lab, int u8, int Hm, int Wm, int fy,
                                                int fx, float sy, float sx, int K) {
    float ly, lx;
    int y0 = src_index(sy, fy, Hm, &ly), x0 = src_index(sx, fx, Wm, &lx);
    int y1 = y0 + (y0 < Hm - 1 ? 1 : 0), x1 = x0 + (x0 < Wm - 1 ? 1 : 0);
    LabelTaps t;
    t.cls[0] = fetch_label(lab, (size_t)y0 * Wm + x0, u8, K);
    t.cls[1] = fetch_label(lab, (size_t)y0 * Wm + x1, u8, K);
    t.cls[2] = fetch_label(lab, (size_t)y1 * Wm + x0, u8, K);
    t.cls[3] = fetch_label(lab, (size_t)y1 * Wm + x1, u8, K);
    // PyTorch: out = h0l*(w0l*a + w1l*b) + h1l*(w0l*c + w1l*d)
    float hy0 = 1.f - ly, hx0 = 1.f - lx;
    t.w[0] = hy0 * hx0;
    t.w[1] = hy0 * lx;
    t.w[2] = ly * hx0;
    t.w[3] = ly * lx;
#pragma unroll
    for (int j = 1; j < 4; ++j)
#pragma unroll
        for (int i = 0; i < j; ++i)
            if (t.w[j] != 0.f && t.cls[j] == t.cls[i] && t.w[i] != 0.f) {
                t.w[i] += t.w[j];
                t.w[j] = 0.f;
            }
    return t;
}

// Move the non-zero taps to the front (entry 0 is non-zero for every real pixel: the weights sum to 1);
// returns how many are non-zero. Static indices only (a 3-pass bubble), so it stays in registers.
__device__ __forceinline__ int compact_taps(LabelTaps& t) {
#pragma unroll
    for (int pass = 0; pass < 3; ++pass)
#pragma unroll
        for (int j = 0; j < 3 - pass; ++j)
            if (t.w[j] == 0.f && t.w[j + 1] != 0.f) {
                t.w[j] = t.w[j + 1];
                t.cls[j] = t.cls[j + 1];
                t.w[j + 1] = 0.f;
            }
    int n = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) n += (t.w[j] != 0.f) ? 1 : 0;
    return n;
}

// ---- column sums of score_query's backward (pm_score.cu: pm_score_bwd; pm_exchange.cu: the global read's exchange)
// SB_PARTS CTAs each leave one fp64 partial per column ([SB_PARTS][32] doubles); the column sum is formed in ONE fixed
// order everywhere: group j (0..SB_GROUPS-1) adds partials j, j + SB_GROUPS, ... in ascending order, then the groups are
// added in ascending order. sb_group_sum is one group's term.
constexpr int SB_PARTS = 148, SB_GROUPS = 8;
__device__ __forceinline__ double sb_group_sum(const double* part, int k, int j) {
    double a = 0.0;
    for (int i = j; i < SB_PARTS; i += SB_GROUPS) a += __ldcg(part + (size_t)i * 32 + k);
    return a;
}

// ---- cross-rank flags in the symmetric peer buffer (pm_write.cu: the sharded update; pm_exchange.cu: the global read).
// flags[kind][row 0..31][rank 0..15] (u32, monotone epochs) at PM_PEER_FLAG_OFF; kinds 0..3 belong to the update kernels,
// 4..7 to the read exchanges, rows 0..7 of kind 8 (PM_PEER_BN_FLAG_OFF) to the SyncBatchNorm exchanges (pm_bn_exchange.cu).
struct PeerCtx {
    const unsigned long long* bufs;  // device array [world] of symmetric-buffer base addresses; nullptr = not sharded
    int rank, world;
    unsigned* epoch;                 // device counter of this kernel's launches (one per kernel kind)
};

__device__ __forceinline__ unsigned* peer_flag(unsigned long long base, int kind, int row, int rank) {
    return reinterpret_cast<unsigned*>(base + PM_PEER_FLAG_OFF) + ((kind * 32 + row) * 16 + rank);
}
// all threads of the CTA call both; data written by this CTA before peer_signal is visible to the peers after their wait
__device__ __forceinline__ void peer_signal(const PeerCtx& p, int kind, int row, unsigned e) {
    __threadfence_system();
    __syncthreads();
    if ((int)threadIdx.x < p.world) {
        unsigned* f = peer_flag(p.bufs[threadIdx.x], kind, row, p.rank);
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f), "r"(e) : "memory");
    }
}
__device__ __forceinline__ void peer_wait(const PeerCtx& p, int kind, int row, unsigned e) {
    if ((int)threadIdx.x < p.world) {
        const unsigned* f = peer_flag(p.bufs[p.rank], kind, row, threadIdx.x);
        unsigned v = 0;
        for (unsigned spin = 0;; ++spin) {
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
            if ((int)(v - e) >= 0) break;
            if (spin > (1u << 27)) __trap();  // a peer that never arrives (crashed rank): fail loudly, do not hang the GPU
            __nanosleep(32);
        }
    }
    __syncthreads();
}

}  // namespace pm
