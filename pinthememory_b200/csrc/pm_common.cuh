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

}  // namespace pm
