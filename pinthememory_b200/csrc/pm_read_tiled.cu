// Memory read, pipelined variants (the fast path when hw is a multiple of the 16-byte chunk).
//
// Persistent CTAs (2 per SM) walk tiles of 32 consecutive pixels x all C channels. Each tile is brought
// into shared memory by TMA (the ds pass of the backward: 16-byte async copies, LDGSTS) into a 2-stage ring,
// so the next tile streams from HBM while the current one is consumed and the feature values never occupy
// registers. The 8 warps split the channels, a lane owns one pixel (conflict-free column reads of the dense [C][32] tile), the
// K x C memory sits transposed in shared memory (Mt[c][KP]: a channel's K values are five broadcast
// 128-bit loads) and all multiply-adds are packed FFMA2 (fp32x2), which is what reaches the fp32 peak
// on sm_100 (profiles/microbench/ffma2.cu: 65.9 vs 46.8 TFLOP/s for scalar FFMA).

#include "pm_common.cuh"
#include "pm_tma.cuh"
#include "pm_internal.h"

namespace pm {

constexpr int TP = 32;        // pixels per tile (= lanes)
constexpr int TL_THREADS = 256;
constexpr int TL_WARPS = 8;

__device__ __forceinline__ float2 f2(float a, float b) { return make_float2(a, b); }

template <int C, int KP>
__device__ __forceinline__ void load_Mt(float* Mt, const float* __restrict__ M, int K) {
    constexpr int PER = (C * KP + TL_THREADS - 1) / TL_THREADS;
    float v[PER];
#pragma unroll
    for (int r = 0; r < PER; ++r) {  // all loads in flight before the first store
        const int i = threadIdx.x + r * TL_THREADS;
        const int c = i / KP, k = i - c * KP;
        v[r] = (i < C * KP && k < K) ? __ldg(M + (size_t)k * C + c) : 0.f;
    }
#pragma unroll
    for (int r = 0; r < PER; ++r) {
        const int i = threadIdx.x + r * TL_THREADS;
        if (i < C * KP) Mt[i] = v[r];
    }
}

// dots of this warp's CW channels of tile `xt` (column `lane`) with the memory: a2[k/2] += x * Mt[c][k]
template <typename T, int CW, int KP>
__device__ __forceinline__ void tile_dots(const T* xt, const float* Mt, int c0, int lane, float2 (&a2)[KP / 2],
                                          float& n2) {
    const T* xcol = xt + c0 * 32 + lane;
    const float4* mbase = reinterpret_cast<const float4*>(Mt + c0 * KP);
#pragma unroll
    for (int j = 0; j < CW; ++j) {
        const float xv = to_float(xcol[j * 32]);
        const float2 x2 = f2(xv, xv);
        n2 = fmaf(xv, xv, n2);
        const float4* mrow = mbase + j * (KP / 4);
#pragma unroll
        for (int q = 0; q < KP / 4; ++q) {
            const float4 m = mrow[q];
            a2[2 * q] = __ffma2_rn(x2, f2(m.x, m.y), a2[2 * q]);
            a2[2 * q + 1] = __ffma2_rn(x2, f2(m.z, m.w), a2[2 * q + 1]);
        }
    }
}

// ---- tensor-core variant of the same contraction (fp32 tiles, CW % 8 == 0) -----------------------------------
// S[32 px][KP] (+)= X[32 px][CW ch] . Mt[CW ch][KP] with mma.sync m16n8k8 TF32 and 3xTF32 error compensation
// (a = a_hi + a_lo, b = b_hi + b_lo; a_lo.b_hi + a_hi.b_lo + a_hi.b_hi in an fp32 accumulator): fp32-level
// accuracy at 93 TFLOP/s effective (profiles/microbench/mma_tf32.cu), operands reused inside the tensor core
// instead of one broadcast shared-memory load per FMA pair. The k index of an MMA is a free permutation, so
// k = t maps to channel 2t and k = t+4 to channel 2t+1 of an 8-channel step: with that choice the B fragments
// read the existing Mt[c][KP=20] rows without bank conflicts, and the A fragments read the chunk-swizzled tile
// (tile_load_async_mma, or a SWIZZLE_128B TMA box) without bank conflicts. Writes this warp's partial sums straight into part / pn.
template <int CW, int KP>
__device__ __forceinline__ void tile_dots_mma(const float* xt, const float* Mt, int c0, int lane, float* part_w,
                                              float* pn_w) {
    constexpr int NT = (KP + 7) / 8;
    const int g = lane >> 2, t = lane & 3;
    float acc[2][NT][4];
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
        for (int n = 0; n < NT; ++n) acc[m][n][0] = acc[m][n][1] = acc[m][n][2] = acc[m][n][3] = 0.f;
    float n2[4] = {0.f, 0.f, 0.f, 0.f};
    int pos[4];  // rows c0+8ks+2t+h (c0 % 8 == 0): swizzle (row & 7) = 2t + h; h = 1 flips bit 0 of the chunk = word ^ 4
#pragma unroll
    for (int r = 0; r < 4; ++r) pos[r] = mma_tile_pos(g + 8 * r, 2 * t);
#pragma unroll
    for (int ks = 0; ks < CW / 8; ++ks) {
        const float* r0 = xt + (c0 + 8 * ks + 2 * t) * 32;
        const float* mrow = Mt + (c0 + 8 * ks + 2 * t) * KP + g;
        unsigned ahi[4][2], alo[4][2];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const float v = r0[h * 32 + (pos[r] ^ (4 * h))];
                n2[r] = fmaf(v, v, n2[r]);
                ahi[r][h] = tf32_hi(v);
                alo[r][h] = tf32_lo(v);
            }
        }
#pragma unroll
        for (int n = 0; n < NT; ++n) {
            // slots >= KP of the last 8-slot step do not exist (their accumulators are never stored): read zeros instead
            // of the next row's first slots -- past the end of Mt for the last channel
            const bool in = (8 * n + 8 <= KP) || (8 * n + g < KP);
            const float b0 = in ? mrow[8 * n] : 0.f, b1 = in ? mrow[KP + 8 * n] : 0.f;
            const unsigned b0h = tf32_hi(b0), b1h = tf32_hi(b1);
            const unsigned b0l = tf32_lo(b0), b1l = tf32_lo(b1);
#pragma unroll
            for (int m = 0; m < 2; ++m) {
                mma_tf32(acc[m][n], alo[2 * m][0], alo[2 * m + 1][0], alo[2 * m][1], alo[2 * m + 1][1], b0h, b1h);
                mma_tf32(acc[m][n], ahi[2 * m][0], ahi[2 * m + 1][0], ahi[2 * m][1], ahi[2 * m + 1][1], b0l, b1l);
                mma_tf32(acc[m][n], ahi[2 * m][0], ahi[2 * m + 1][0], ahi[2 * m][1], ahi[2 * m + 1][1], b0h, b1h);
            }
        }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        n2[r] += __shfl_xor_sync(0xffffffffu, n2[r], 1);
        n2[r] += __shfl_xor_sync(0xffffffffu, n2[r], 2);
        if (t == 0 && pn_w != nullptr) pn_w[g + 8 * r] = n2[r];
    }
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
        for (int n = 0; n < NT; ++n) {
            const int slot = 8 * n + 2 * t;
            if (slot < KP) {
                *reinterpret_cast<float2*>(part_w + (g + 16 * m) * KP + slot) = make_float2(acc[m][n][0], acc[m][n][1]);
                *reinterpret_cast<float2*>(part_w + (g + 8 + 16 * m) * KP + slot) = make_float2(acc[m][n][2], acc[m][n][3]);
            }
        }
}

// Second contraction of the read on the tensor core: cout[32 px][CW ch] = P[32 px][K] . M[K][CW ch] for this
// warp's channels, written straight to the second half of u (NCHW). A fragments come from p_sm[px][KP] (stride 20:
// conflict-free), B fragments from Mt[c][KP] (same pattern); slots >= KP of the last 8-slot step are zero.
template <typename T, int CW, int KP>
__device__ __forceinline__ void tile_weighted_sum_mma(const float* p_sm, const float* Mt, int c0, int lane, T* uc,
                                                      int hw, int nvalid) {
    constexpr int NKS = (KP + 7) / 8, NNT = CW / 8;
    const int g = lane >> 2, t = lane & 3;
    unsigned ahi[2][NKS][4], alo[2][NKS][4];
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
        for (int ks = 0; ks < NKS; ++ks)
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int px = g + 16 * m + 8 * (e & 1), slot = 8 * ks + t + 4 * (e >> 1);
                const float v = (slot < KP) ? p_sm[px * KP + slot] : 0.f;
                ahi[m][ks][e] = tf32_hi(v);
                alo[m][ks][e] = tf32_lo(v);
            }
#pragma unroll
    for (int n = 0; n < NNT; ++n) {
        float acc[2][4];
#pragma unroll
        for (int m = 0; m < 2; ++m) acc[m][0] = acc[m][1] = acc[m][2] = acc[m][3] = 0.f;
        const float* mrow = Mt + (c0 + 8 * n + g) * KP + t;
#pragma unroll
        for (int ks = 0; ks < NKS; ++ks) {
            const float b0 = mrow[8 * ks], b1 = (8 * ks + 4 < KP) ? mrow[8 * ks + 4] : 0.f;  // KP % 4 == 0
            const unsigned b0h = tf32_hi(b0), b1h = tf32_hi(b1), b0l = tf32_lo(b0), b1l = tf32_lo(b1);
#pragma unroll
            for (int m = 0; m < 2; ++m) {
                mma_tf32(acc[m], alo[m][ks][0], alo[m][ks][1], alo[m][ks][2], alo[m][ks][3], b0h, b1h);
                mma_tf32(acc[m], ahi[m][ks][0], ahi[m][ks][1], ahi[m][ks][2], ahi[m][ks][3], b0l, b1l);
                mma_tf32(acc[m], ahi[m][ks][0], ahi[m][ks][1], ahi[m][ks][2], ahi[m][ks][3], b0h, b1h);
            }
        }
        // c0:(px g, ch 2t) c1:(px g, ch 2t+1) c2:(px g+8, ch 2t) c3:(px g+8, ch 2t+1)   (+16m px, +8n ch)
        T* base = uc + (size_t)(8 * n + 2 * t) * hw;
#pragma unroll
        for (int m = 0; m < 2; ++m) {
            const int pa = g + 16 * m, pb = pa + 8;
            if (pa < nvalid) {
                stf(base + pa, acc[m][0]);
                stf(base + hw + pa, acc[m][1]);
            }
            if (pb < nvalid) {
                stf(base + pb, acc[m][2]);
                stf(base + hw + pb, acc[m][3]);
            }
        }
    }
}

// ---- bf16 tiles on the tensor core (mma.sync m16n8k16, fp32 accumulate) ------------------------------------------
// The tile is [C][32 px] bf16 (64-byte rows) in the TMA SWIZZLE_64B layout: 16-byte chunk c of row r sits at chunk
// c ^ ((r >> 1) & 3), so the eight 16-byte rows of an 8-channel x 8-pixel block fall into eight distinct bank groups
// and `ldmatrix.trans` -- which hands thread (g, t) the pair (channel 2t, 2t+1) of pixel g, exactly the A fragment of
// a [pixels x channels] operand -- reads a block in one wavefront. The memory is the B operand, kept in shared memory
// as bf16 pairs over channels, split hi + lo (M = hi + lo to 2^-17), so the only rounding left is the feature map's own.
__device__ __forceinline__ int bf16_tile_off(int row, int px) {  // element offset of (row, px) in a SWIZZLE_64B tile
    return row * 32 + ((((px >> 3) ^ ((row >> 1) & 3)) << 3) | (px & 7));
}
__device__ __forceinline__ void ldmatrix_x4_trans(unsigned (&r)[4], uint32_t saddr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(saddr));
}
__device__ __forceinline__ void mma_bf16(float (&c)[4], const unsigned (&a)[4], unsigned b0, unsigned b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ unsigned pack_bf16(float lo, float hi) {  // lo -> bits 0..15
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<unsigned*>(&v);
}
__device__ __forceinline__ float bf16_lo_f(unsigned w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16_hi_f(unsigned w) { return __uint_as_float(w & 0xffff0000u); }

template <int KP>
struct MbLayout {
    static constexpr int NT = (KP + 7) / 8;
    // row stride in words: rows t = 0..3 (and 4..7) of a B-fragment load must land in distinct 8-bank groups
    static constexpr int LD = (NT == 3) ? 24 : 40;
};
// Mb_hi / Mb_lo [C/2][LD] words: word (cp, k) = bf16 pair (M[k][2cp], M[k][2cp+1])
template <int C, int KP>
__device__ __forceinline__ void load_Mb(unsigned* Mb_hi, unsigned* Mb_lo, const float* __restrict__ M, int K) {
    constexpr int LD = MbLayout<KP>::LD;
    for (int i = threadIdx.x; i < (C / 2) * LD; i += TL_THREADS) {
        const int cp = i / LD, k = i - cp * LD;
        float a = 0.f, b = 0.f;
        if (k < K) {
            const float2 v = __ldg(reinterpret_cast<const float2*>(M + (size_t)k * C) + cp);
            a = v.x, b = v.y;
        }
        const float ah = __bfloat162float(__float2bfloat16_rn(a)), bh = __bfloat162float(__float2bfloat16_rn(b));
        Mb_hi[i] = pack_bf16(ah, bh);
        Mb_lo[i] = pack_bf16(a - ah, b - bh);
    }
}

// S[32 px][KP] = X[32 px][CW ch] . M^T for this warp's CW channels (CW % 16 == 0) + the partial squared norms
template <int CW, int KP>
__device__ __forceinline__ void tile_dots_mma_bf16(const __nv_bfloat16* xt, const unsigned* Mb_hi, const unsigned* Mb_lo,
                                                   int c0, int lane, float* part_w, float* pn_w) {
    constexpr int NT = MbLayout<KP>::NT, LD = MbLayout<KP>::LD;
    const int g = lane >> 2, t = lane & 3;
    float acc[2][NT][4];
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
        for (int n = 0; n < NT; ++n) acc[m][n][0] = acc[m][n][1] = acc[m][n][2] = acc[m][n][3] = 0.f;
    float n2[4] = {0.f, 0.f, 0.f, 0.f};  // pixels g, g+8, g+16, g+24
    const uint32_t xbase = smem_u32(xt);
    const int mj = lane >> 3, rr = lane & 7;  // ldmatrix: this lane addresses row rr of matrix mj
#pragma unroll
    for (int ks = 0; ks < CW / 16; ++ks) {
        const int cb = c0 + 16 * ks;
        unsigned a[2][4];
#pragma unroll
        for (int m = 0; m < 2; ++m) {
            const int row = cb + (mj >> 1) * 8 + rr, chunk = 2 * m + (mj & 1);
            ldmatrix_x4_trans(a[m], xbase + (uint32_t)(row * 64 + ((chunk ^ ((row >> 1) & 3)) << 4)));
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float lo = bf16_lo_f(a[m][e]), hi = bf16_hi_f(a[m][e]);
                n2[2 * m + (e & 1)] = fmaf(lo, lo, fmaf(hi, hi, n2[2 * m + (e & 1)]));
            }
        }
        const unsigned* bh = Mb_hi + ((cb >> 1) + t) * LD + g;
        const unsigned* bl = Mb_lo + ((cb >> 1) + t) * LD + g;
#pragma unroll
        for (int n = 0; n < NT; ++n) {
            const unsigned b0h = bh[8 * n], b1h = bh[4 * LD + 8 * n], b0l = bl[8 * n], b1l = bl[4 * LD + 8 * n];
#pragma unroll
            for (int m = 0; m < 2; ++m) {
                mma_bf16(acc[m][n], a[m], b0l, b1l);
                mma_bf16(acc[m][n], a[m], b0h, b1h);
            }
        }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        n2[r] += __shfl_xor_sync(0xffffffffu, n2[r], 1);
        n2[r] += __shfl_xor_sync(0xffffffffu, n2[r], 2);
        if (t == 0 && pn_w != nullptr) pn_w[g + 8 * r] = n2[r];
    }
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
        for (int n = 0; n < NT; ++n) {
            const int slot = 8 * n + 2 * t;
            if (slot < KP) {
                *reinterpret_cast<float2*>(part_w + (g + 16 * m) * KP + slot) = make_float2(acc[m][n][0], acc[m][n][1]);
                *reinterpret_cast<float2*>(part_w + (g + 8 + 16 * m) * KP + slot) = make_float2(acc[m][n][2], acc[m][n][3]);
            }
        }
}

template <typename T, int CW>
struct UseMma {
    static constexpr bool value = false;
};
template <int CW>
struct UseMma<float, CW> {
    static constexpr bool value = (CW % 8 == 0);
};
template <int CW>
struct UseMma<__nv_bfloat16, CW> {
    static constexpr bool value = (CW % 16 == 0);
};

// dispatch: load one tile for the dots phase in the layout the chosen contraction wants
template <typename T, int C, int NTHREADS, bool MMA>
__device__ __forceinline__ void dots_tile_load(T* smem_tile, const T* __restrict__ base, int hw, int px0) {
    static_assert(!MMA || sizeof(T) == 4, "the cp.async tensor-core layout is the fp32 one");
    if constexpr (MMA) tile_load_async_mma<C, NTHREADS>(reinterpret_cast<float*>(smem_tile), reinterpret_cast<const float*>(base), hw, px0);
    else tile_load_async<T, C, NTHREADS>(smem_tile, base, hw, px0);
}

template <int KP>
__device__ __forceinline__ void store_partial(float* part, int wid, int lane, const float2 (&a2)[KP / 2]) {
    float4* d = reinterpret_cast<float4*>(part + ((size_t)wid * TP + lane) * KP);
#pragma unroll
    for (int q = 0; q < KP / 4; ++q) d[q] = make_float4(a2[2 * q].x, a2[2 * q].y, a2[2 * q + 1].x, a2[2 * q + 1].y);
}

// --------------------------------------------------------------------------------------------- forward

// exp(x) for x <= 0 (softmax terms after the maximum is subtracted): ex2.approx of x*log2(e) -- 2 instructions instead of
// expf's ~10; the terms that matter have |x| of a few units, where the product's rounding is ~1e-7 relative (the read-loss
// kernels have always computed their softmax this way)
__device__ __forceinline__ float fexp_nonpos(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x * 1.4426950408889634f));
    return y;
}

// The x tiles arrive as tensor-map boxes (SWIZZLE_128B / SWIZZLE_64B for the tensor-core layouts, dense otherwise) on an
// mbarrier ring. `x` itself is not read; it stays in the parameter list because the offsets of the parameters after it
// steer ptxas: without it the bf16 tensor-core instantiations are scheduled differently (C = 128, K > 19: 87 registers
// instead of 80).
template <typename T, int C, int KP, int NSTAGE>
__global__ void __launch_bounds__(TL_THREADS, 2)
    read_fwd_tiled_kernel(const __grid_constant__ CUtensorMap tm_x, const T* __restrict__ x,
                          const float* __restrict__ M, const float* __restrict__ gum_m,
                          const float* __restrict__ gum_q, T* __restrict__ u, float* __restrict__ s_out,
                          float* __restrict__ p_out, float* __restrict__ colpart, int hw, int K, int tiles_per_img,
                          int ntiles, int planes) {
    // planes == 0: u = [q ; p.M], 2C channels. planes == 1: u = [q ; p as PM_PLANES score planes], C + PM_PLANES
    // channels (planes >= K are zero): the 1x1 convolution that follows is then W1.q + (W2.M^T).p, a (C+32)-wide
    // GEMM instead of a 2C-wide one, and its input gradient hands dp back directly.
    constexpr int CW = C / TL_WARPS, NI = (KP + 7) / 8;
    const int UC = planes ? C + PM_PLANES : 2 * C;
    constexpr bool MMA = UseMma<T, CW>::value;
    extern __shared__ __align__(16) unsigned char smraw[];
    float* Mt = reinterpret_cast<float*>(smraw);  // [C][KP]
    float* part = Mt + C * KP;                    // [8][TP][KP]
    float* pn = part + TL_WARPS * TP * KP;        // [8][TP]
    float* s_sm = pn + TL_WARPS * TP;             // [TP][KP]
    float* p_sm = s_sm + TP * KP;                 // [TP][KP]
    float* invr = p_sm + TP * KP;                 // [TP]
    constexpr bool MMA16 = MMA && sizeof(T) == 2;
    constexpr int MB_WORDS = MMA16 ? (C / 2) * MbLayout<KP>::LD : 0;
    unsigned* Mb_hi = reinterpret_cast<unsigned*>(invr + TP);  // [C/2][LD] x 2: the memory as bf16 pairs (bf16 tiles only)
    unsigned* Mb_lo = Mb_hi + MB_WORDS;
    // [NSTAGE][C][TP]; 1 KB aligned for the swizzled TMA boxes (the launcher allocates the slack)
    T* xs = reinterpret_cast<T*>(smem_align(reinterpret_cast<unsigned char*>(Mb_lo + MB_WORDS), 1024));
    __shared__ __align__(8) uint64_t full[NSTAGE];

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    int tile = blockIdx.x;
    auto issue = [&](int t, int s) {  // one thread
        const int b = t / tiles_per_img, px0 = (t - b * tiles_per_img) * TP;
        mbar_expect_tx(&full[s], (uint32_t)(C * TP * sizeof(T)));
        tma_load_2d(xs + s * C * TP, &tm_x, px0, b * C, &full[s]);
    };
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < NSTAGE; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#pragma unroll
        for (int s = 0; s < NSTAGE; ++s)
            if (tile + s * (int)gridDim.x < ntiles) issue(tile + s * gridDim.x, s);
    }
    load_Mt<C, KP>(Mt, M, K);
    if constexpr (MMA16) load_Mb<C, KP>(Mb_hi, Mb_lo, M, K);
    float cm[NI], cl[NI];  // running column (max, sum) of this thread's slots for score_query
#pragma unroll
    for (int i = 0; i < NI; ++i) cm[i] = -INFINITY, cl[i] = 0.f;

    int stage = 0;
    unsigned phase = 0;
    for (; tile < ntiles; tile += gridDim.x) {
        __syncthreads();  // Mt and the mbarriers are set up
        mbar_wait(&full[stage], phase);
        const T* xt = xs + stage * C * TP;
        const int b = tile / tiles_per_img, px0 = (tile - b * tiles_per_img) * TP;
        const int nvalid = min(TP, hw - px0);
        const size_t n0g = (size_t)b * hw + px0;
        if constexpr (MMA16) {
            tile_dots_mma_bf16<CW, KP>(reinterpret_cast<const __nv_bfloat16*>(xt), Mb_hi, Mb_lo, wid * CW, lane,
                                       part + wid * TP * KP, pn + wid * TP);
        } else if constexpr (MMA) {
            tile_dots_mma<CW, KP>(reinterpret_cast<const float*>(xt), Mt, wid * CW, lane, part + wid * TP * KP,
                                  pn + wid * TP);
        } else {
            float2 a2[KP / 2];
#pragma unroll
            for (int i = 0; i < KP / 2; ++i) a2[i] = f2(0.f, 0.f);
            float n2 = 0.f;
            tile_dots<T, CW, KP>(xt, Mt, wid * CW, lane, a2, n2);
            store_partial<KP>(part, wid, lane, a2);
            pn[wid * TP + lane] = n2;
        }
        __syncthreads();
        {  // cross-warp reduction + softmax over slots: 8 threads per pixel, slots j, j+8, j+16(, j+24)
            const int px = tid >> 3, j = tid & 7;
            float n2 = 0.f;
#pragma unroll
            for (int w = 0; w < TL_WARPS; ++w) n2 += pn[w * TP + px];
            const float ir = 1.f / fmaxf(sqrtf(n2), PM_NORM_EPS);
            const bool valid = px < nvalid;
            float sv[NI], z[NI], mx = -INFINITY;
#pragma unroll
            for (int i = 0; i < NI; ++i) {
                const int k = j + 8 * i;
                float acc = 0.f;
                if (k < KP) {
#pragma unroll
                    for (int w = 0; w < TL_WARPS; ++w) acc += part[((size_t)w * TP + px) * KP + k];
                }
                sv[i] = acc * ir;
                float g = 0.f;
                if (gum_m != nullptr && valid && k < K) g = __ldg(gum_m + (n0g + px) * K + k);
                z[i] = (k < K) ? sv[i] + g : -INFINITY;
                mx = fmaxf(mx, z[i]);
            }
            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 4));
            float sum = 0.f;
#pragma unroll
            for (int i = 0; i < NI; ++i) {
                z[i] = (j + 8 * i < K) ? fexp_nonpos(z[i] - mx) : 0.f;
                sum += z[i];
            }
            sum += __shfl_xor_sync(0xffffffffu, sum, 1);
            sum += __shfl_xor_sync(0xffffffffu, sum, 2);
            sum += __shfl_xor_sync(0xffffffffu, sum, 4);
            const float inv = 1.f / sum;
#pragma unroll
            for (int i = 0; i < NI; ++i) {
                const int k = j + 8 * i;
                if (k < KP) {
                    s_sm[px * KP + k] = (k < K) ? sv[i] : 0.f;
                    p_sm[px * KP + k] = z[i] * inv;
                }
                if (colpart != nullptr && valid && k < K) {
                    float zq = sv[i];
                    if (gum_q != nullptr) zq += __ldg(gum_q + (n0g + px) * K + k);
                    if (zq > cm[i]) {
                        cl[i] = cl[i] * fexp_nonpos(cm[i] - zq) + 1.f;
                        cm[i] = zq;
                    } else {
                        cl[i] += fexp_nonpos(zq - cm[i]);
                    }
                }
            }
            if (j == 0) invr[px] = ir;
        }
        __syncthreads();
        for (int o = tid; o < nvalid * (KP / 4); o += TL_THREADS)
            reinterpret_cast<float4*>(s_out + n0g * KP)[o] = reinterpret_cast<const float4*>(s_sm)[o];
        for (int o = tid; o < nvalid * K; o += TL_THREADS) {
            const int px = o / K, k = o - px * K;
            p_out[n0g * K + o] = p_sm[px * KP + k];
        }
        if (planes) {
            for (int r = wid; r < PM_PLANES; r += TL_WARPS) {
                const float v = (r < K) ? p_sm[lane * KP + r] : 0.f;
                if (lane < nvalid) stf(u + ((size_t)b * UC + C + r) * hw + px0 + lane, v);
            }
        }
        if constexpr (MMA16) {  // bf16: two channel rows x 16 pixel pairs per store instruction (2 x 64 bytes)
            if (!planes)
                tile_weighted_sum_mma<T, CW, KP>(p_sm, Mt, wid * CW, lane,
                                                 u + ((size_t)b * UC + C + wid * CW) * hw + px0, hw, nvalid);
            const int half = lane >> 4, pp = (lane & 15) * 2;
            const float ir0 = invr[pp], ir1 = invr[pp + 1];
            if (pp < nvalid) {  // hw % 8 == 0: a pixel pair is valid or not as a whole
                const unsigned* xw = reinterpret_cast<const unsigned*>(xt);
                unsigned* uq = reinterpret_cast<unsigned*>(u + ((size_t)b * UC + wid * CW + half) * hw + px0 + pp);
#pragma unroll
                for (int j = 0; j < CW / 2; ++j) {
                    const int row = wid * CW + 2 * j + half;
                    const unsigned v = xw[bf16_tile_off(row, pp) >> 1];
                    *uq = pack_bf16(bf16_lo_f(v) * ir0, bf16_hi_f(v) * ir1);
                    uq += hw;  // two rows of bf16 = hw 32-bit words
                }
            }
        } else if constexpr (MMA) {  // u = [q ; p.M]: p.M on the tensor core, q = x/|x| element-wise
            if (!planes)
                tile_weighted_sum_mma<T, CW, KP>(p_sm, Mt, wid * CW, lane,
                                                 u + ((size_t)b * UC + C + wid * CW) * hw + px0, hw, nvalid);
            const float ir = invr[lane];
            if (lane < nvalid) {
                T* uq = u + ((size_t)b * UC + wid * CW) * hw + px0 + lane;
#pragma unroll
                for (int j = 0; j < CW; ++j) {
                    stf(uq, to_float(xt[(wid * CW + j) * 32 + mma_tile_pos(lane, j & 7)]) * ir);  // CW % 8 == 0
                    uq += hw;
                }
            }
        } else {  // u = [q ; p.M]
            float2 p2[KP / 2];
            const float4* pr = reinterpret_cast<const float4*>(p_sm + lane * KP);
#pragma unroll
            for (int q = 0; q < KP / 4; ++q) {
                const float4 v = pr[q];
                p2[2 * q] = f2(v.x, v.y);
                p2[2 * q + 1] = f2(v.z, v.w);
            }
            const float ir = invr[lane];
            const bool v = lane < nvalid;
            T* uq = u + ((size_t)b * UC + wid * CW) * hw + px0 + lane;
            const size_t chw = (size_t)C * hw;
            const T* xcol = xt + wid * CW * 32 + lane;
            const float4* mbase = reinterpret_cast<const float4*>(Mt + wid * CW * KP);
            if (planes) {
#pragma unroll
                for (int j = 0; j < CW; ++j) {
                    if (v) stf(uq, to_float(xcol[j * 32]) * ir);
                    uq += hw;
                }
            } else {
#pragma unroll
                for (int j = 0; j < CW; ++j) {
                    const float4* mrow = mbase + j * (KP / 4);
                    float2 acc = f2(0.f, 0.f);
#pragma unroll
                    for (int q = 0; q < KP / 4; ++q) {
                        const float4 m = mrow[q];
                        acc = __ffma2_rn(p2[2 * q], f2(m.x, m.y), acc);
                        acc = __ffma2_rn(p2[2 * q + 1], f2(m.z, m.w), acc);
                    }
                    const float xq = to_float(xcol[j * 32]) * ir;
                    if (v) {
                        stf(uq, xq);
                        stf(uq + chw, acc.x + acc.y);
                    }
                    uq += hw;
                }
            }
        }
        __syncthreads();  // every read of this stage is done: refill it
        const int next = tile + NSTAGE * gridDim.x;
        if (tid == 0 && next < ntiles) issue(next, stage);
        if (++stage == NSTAGE) stage = 0, phase ^= 1u;
    }

    if (colpart != nullptr) {  // per-CTA column (max,sum) partials, same layout as colsoftmax_stats_kernel
        __syncthreads();
        float* scr = part;  // [NI][2][256]
#pragma unroll
        for (int i = 0; i < NI; ++i) {
            scr[(i * 2 + 0) * TL_THREADS + tid] = cm[i];
            scr[(i * 2 + 1) * TL_THREADS + tid] = cl[i];
        }
        __syncthreads();
        if (tid < K) {
            const int j = tid & 7, i = tid >> 3;
            float Mx = -INFINITY;
            for (int px = 0; px < TP; ++px) Mx = fmaxf(Mx, scr[(i * 2 + 0) * TL_THREADS + px * 8 + j]);
            float L = 0.f;
            for (int px = 0; px < TP; ++px) {
                const float mi = scr[(i * 2 + 0) * TL_THREADS + px * 8 + j];
                if (mi > -INFINITY) L += scr[(i * 2 + 1) * TL_THREADS + px * 8 + j] * expf(mi - Mx);
            }
            colpart[(size_t)blockIdx.x * 64 + tid] = Mx;
            colpart[(size_t)blockIdx.x * 64 + 32 + tid] = L;
        }
        // The last CTA to get here combines the gridDim.x partial rows into the final column maximum and 1/sum (row
        // PM_COLPART_ROWS) -- what used to be a separate one-CTA launch between this kernel and the normalising pass.
        // Ticket = first word of row PM_COLPART_ROWS + 1: zero on entry (caller), left zero.
        __shared__ int s_last;
        __threadfence();
        __syncthreads();
        if (tid == 0) {
            unsigned* ticket = reinterpret_cast<unsigned*>(colpart + (size_t)(PM_COLPART_ROWS + 1) * 64);
            s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
        }
        __syncthreads();
        if (s_last) {
            __threadfence();
            // thread (k = tid % 32, r0 = tid / 32): rows r0, r0 + 8, ..; loads in batches of 8 independent L2 hits
            const int k = tid & 31, r0 = tid >> 5;
            float Mx = -INFINITY, L = 0.f;
            const int G = (int)gridDim.x;
            for (int rb = r0; rb < G; rb += 8 * 8) {
                float pmx[8], pl[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int r = rb + 8 * j;
                    pmx[j] = (r < G && k < K) ? __ldcg(colpart + (size_t)r * 64 + k) : -INFINITY;
                    pl[j] = (r < G && k < K) ? __ldcg(colpart + (size_t)r * 64 + 32 + k) : 0.f;
                }
                float bm = Mx;
#pragma unroll
                for (int j = 0; j < 8; ++j) bm = fmaxf(bm, pmx[j]);
                if (bm > -INFINITY) {
                    L *= expf(Mx - bm);  // Mx = -inf: L is 0 and exp(-inf) = 0
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        if (pmx[j] > -INFINITY) L += pl[j] * expf(pmx[j] - bm);
                    Mx = bm;
                }
            }
            float* scr = part;  // [8][2][32]
            __syncthreads();
            scr[(r0 * 2 + 0) * 32 + k] = Mx;
            scr[(r0 * 2 + 1) * 32 + k] = L;
            __syncthreads();
            if (tid < K) {
                float Mt_ = -INFINITY;
#pragma unroll
                for (int i = 0; i < 8; ++i) Mt_ = fmaxf(Mt_, scr[(i * 2) * 32 + tid]);
                float Ls = 0.f;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float mi = scr[(i * 2) * 32 + tid];
                    if (mi > -INFINITY) Ls += scr[(i * 2 + 1) * 32 + tid] * expf(mi - Mt_);
                }
                colpart[(size_t)PM_COLPART_ROWS * 64 + tid] = Mt_;
                colpart[(size_t)PM_COLPART_ROWS * 64 + 32 + tid] = 1.f / Ls;
            }
            if (tid == 0) *reinterpret_cast<unsigned*>(colpart + (size_t)(PM_COLPART_ROWS + 1) * 64) = 0u;
        }
    }
}

template <typename T, int C, int KP>
int launch_read_fwd_tiled(const void* x, const float* M, const float* gum_m, const float* gum_q, void* u, float* s,
                          float* p, float* colpart, int B, int hw, int K, int planes, cudaStream_t st) {
    constexpr int NSTAGE = 2;
    constexpr bool MMA = UseMma<T, C / TL_WARPS>::value;  // the tensor-core layouts are swizzled
    constexpr bool MMA16 = MMA && sizeof(T) == 2;
    const size_t smem = sizeof(float) * ((size_t)C * KP + TL_WARPS * TP * KP + TL_WARPS * TP + 2 * TP * KP + TP) +
                        (MMA16 ? sizeof(unsigned) * 2 * (C / 2) * MbLayout<KP>::LD : 0) +
                        sizeof(T) * (size_t)NSTAGE * C * TP + 1024;
    const int tiles = (hw + TP - 1) / TP, ntiles = B * tiles;
    int grid = 2 * 148;
    if (grid > ntiles) grid = ntiles;
    CUtensorMap tm_x;
    // fp32 tiles: 128-byte rows, SWIZZLE_128B; bf16 tiles: 64-byte rows, SWIZZLE_64B
    if (!make_map_2d<T>(&tm_x, x, (size_t)B * C, hw, C, TP, MMA16 ? 3 : (MMA ? 1 : 0))) return PM_ERR_ALIGN;
    auto kern = read_fwd_tiled_kernel<T, C, KP, NSTAGE>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    kern<<<grid, TL_THREADS, smem, st>>>(tm_x, (const T*)x, M, gum_m, gum_q, (T*)u, s, p, colpart, hw, K, tiles, ntiles, planes);
    cudaError_t le = cudaGetLastError();
    return le == cudaSuccess ? 0 : (int)le;
}

// -------------------------------------------------------------------------------- backward, part A: ds
// ds = p * (M.dc - p.(M.dc)) + g_loss/(V*T) * ds_rl  per pixel: the forward's first phase applied to the
// dc half of du, then the softmax backward by 8 threads per pixel. Writes the [N][KP] score-gradient
// buffer that part B (and the dM kernel) consume.

template <typename T, int C, int KP, int NSTAGE>
__global__ void __launch_bounds__(TL_THREADS, 2)
    read_bwd_ds_tiled_kernel(const T* __restrict__ du, const float* __restrict__ M, const float* __restrict__ p_in,
                             const float* __restrict__ ds_rl, const float* __restrict__ g_loss,
                             const float* __restrict__ rl_out, float* __restrict__ ds_out, int hw, int K,
                             int tiles_per_img, int ntiles) {
    constexpr int CW = C / TL_WARPS, NI = (KP + 7) / 8;
    constexpr bool MMA = UseMma<T, CW>::value && sizeof(T) == 4;  // (the bf16 tensor-core path exists in the forward only)
    extern __shared__ __align__(16) unsigned char smraw[];
    float* Mt = reinterpret_cast<float*>(smraw);  // [C][KP]
    float* part = Mt + C * KP;                    // [8][TP][KP]
    float* ds_sm = part + TL_WARPS * TP * KP;     // [TP][KP]
    T* xs = reinterpret_cast<T*>(ds_sm + TP * KP);  // [NSTAGE][C][TP]  (dc tiles)

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    int tile = blockIdx.x;
#pragma unroll
    for (int s = 0; s < NSTAGE; ++s) {
        const int t = tile + s * gridDim.x;
        if (t < ntiles) {
            const int b = t / tiles_per_img, px0 = (t - b * tiles_per_img) * TP;
            dots_tile_load<T, C, TL_THREADS, MMA>(xs + s * C * TP, du + ((size_t)b * 2 * C + C) * hw, hw, px0);
        }
        cp_async_commit();
    }
    load_Mt<C, KP>(Mt, M, K);
    float scale = 0.f;
    if (ds_rl != nullptr && g_loss != nullptr && rl_out != nullptr) scale = __ldg(g_loss) * __ldg(rl_out + 1);

    int stage = 0;
    for (; tile < ntiles; tile += gridDim.x) {
        const int b = tile / tiles_per_img, px0 = (tile - b * tiles_per_img) * TP;
        const int nvalid = min(TP, hw - px0);
        const size_t n0g = (size_t)b * hw + px0;
        // this thread's share of p and ds_rl (pixel tid>>3, slots j, j+8, ..): fetched before the dots
        const int px = tid >> 3, j = tid & 7;
        const bool valid = px < nvalid;
        float pk[NI], rl[NI];
#pragma unroll
        for (int i = 0; i < NI; ++i) {
            const int k = j + 8 * i;
            pk[i] = (valid && k < K) ? __ldg(p_in + (n0g + px) * K + k) : 0.f;
            rl[i] = (valid && k < K && scale != 0.f) ? __ldg(ds_rl + (n0g + px) * KP + k) : 0.f;
        }
        cp_async_wait<NSTAGE - 1>();
        __syncthreads();
        const T* xt = xs + stage * C * TP;
        if constexpr (MMA) {
            tile_dots_mma<CW, KP>(reinterpret_cast<const float*>(xt), Mt, wid * CW, lane, part + wid * TP * KP, nullptr);
        } else {
            float2 a2[KP / 2];
#pragma unroll
            for (int i = 0; i < KP / 2; ++i) a2[i] = f2(0.f, 0.f);
            float n2 = 0.f;
            tile_dots<T, CW, KP>(xt, Mt, wid * CW, lane, a2, n2);
            store_partial<KP>(part, wid, lane, a2);
        }
        __syncthreads();
        {
            float dp[NI], dot = 0.f;
#pragma unroll
            for (int i = 0; i < NI; ++i) {
                const int k = j + 8 * i;
                float acc = 0.f;
                if (k < KP) {
#pragma unroll
                    for (int w = 0; w < TL_WARPS; ++w) acc += part[((size_t)w * TP + px) * KP + k];
                }
                dp[i] = acc;
                dot = fmaf(pk[i], acc, dot);
            }
            dot += __shfl_xor_sync(0xffffffffu, dot, 1);
            dot += __shfl_xor_sync(0xffffffffu, dot, 2);
            dot += __shfl_xor_sync(0xffffffffu, dot, 4);
#pragma unroll
            for (int i = 0; i < NI; ++i) {
                const int k = j + 8 * i;
                if (k < KP) ds_sm[px * KP + k] = fmaf(scale, rl[i], pk[i] * (dp[i] - dot));
            }
        }
        __syncthreads();  // ds_sm complete; every read of this stage and of `part` is done
        for (int o = tid; o < nvalid * (KP / 4); o += TL_THREADS)
            reinterpret_cast<float4*>(ds_out + n0g * KP)[o] = reinterpret_cast<const float4*>(ds_sm)[o];
        const int next = tile + NSTAGE * gridDim.x;
        if (next < ntiles) {
            const int nb = next / tiles_per_img, npx0 = (next - nb * tiles_per_img) * TP;
            dots_tile_load<T, C, TL_THREADS, MMA>(xs + stage * C * TP, du + ((size_t)nb * 2 * C + C) * hw, hw, npx0);
        }
        cp_async_commit();
        stage = (stage + 1 == NSTAGE) ? 0 : stage + 1;
        // ds_sm is rewritten only after the next iteration's two barriers
    }
    cp_async_wait<0>();
}

// planes mode of part A: dp[n][k] = du[b][C + k][px]; ds = p * (dp - p.dp) + g_loss/(V*T) * ds_rl, one thread per pixel
template <typename T, int KP>
__global__ void __launch_bounds__(256)
    read_bwd_ds_planes_kernel(const T* __restrict__ du, const float* __restrict__ p_in, const float* __restrict__ ds_rl,
                              const float* __restrict__ g_loss, const float* __restrict__ rl_out,
                              float* __restrict__ ds_out, int hw, int C, int K, int UC, long long N) {
    const long long n = (long long)blockIdx.x * 256 + threadIdx.x;
    if (n >= N) return;
    const int b = (int)(n / hw), px = (int)(n - (long long)b * hw);
    const T* dp = du + ((size_t)b * UC + C) * hw + px;
    float scale = 0.f;
    if (ds_rl != nullptr && g_loss != nullptr && rl_out != nullptr) scale = __ldg(g_loss) * __ldg(rl_out + 1);
    float pk[KP], d[KP], dot = 0.f;
#pragma unroll
    for (int k = 0; k < KP; ++k) {
        pk[k] = (k < K) ? __ldg(p_in + (size_t)n * K + k) : 0.f;
        d[k] = (k < K) ? ldf(dp + (size_t)k * hw) : 0.f;
        dot = fmaf(pk[k], d[k], dot);
    }
    float4* out = reinterpret_cast<float4*>(ds_out + (size_t)n * KP);
    const float4* rl = reinterpret_cast<const float4*>(ds_rl + (size_t)n * KP);
#pragma unroll
    for (int q = 0; q < KP / 4; ++q) {
        float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
        if (scale != 0.f) r = __ldg(rl + q);
        float4 o;
        o.x = (4 * q + 0 < K) ? fmaf(scale, r.x, pk[4 * q + 0] * (d[4 * q + 0] - dot)) : 0.f;
        o.y = (4 * q + 1 < K) ? fmaf(scale, r.y, pk[4 * q + 1] * (d[4 * q + 1] - dot)) : 0.f;
        o.z = (4 * q + 2 < K) ? fmaf(scale, r.z, pk[4 * q + 2] * (d[4 * q + 2] - dot)) : 0.f;
        o.w = (4 * q + 3 < K) ? fmaf(scale, r.w, pk[4 * q + 3] * (d[4 * q + 3] - dot)) : 0.f;
        out[q] = o;
    }
}

// -------------------------------------------------------------------------------- backward, part B: dx
// dq = dq0 + ds.M ; q = x/|x| ; dx = (dq - q (q.dq)) / |x|. One CTA per SM, 16 warps x (C/16) channels, lanes = pixels.
// The x and dq0 tiles of a stage arrive as two 2-D tensor-map boxes ([C rows][32 pixels] of the [B*C, hw] / [B*UC, hw]
// matrices) and the ds rows as one 1-D bulk copy, all completing on an mbarrier per stage that one thread issues (3
// instructions). The kernel is LSU / shared-memory-pipe bound (DESIGN.md 6), and the async proxy keeps the tile fill off
// that pipe. Columns past the end of an image row are zero-filled by the TMA unit.

constexpr int DX_THREADS = 512, DX_WARPS = 16;

template <typename T, int C, int KP, int NSTAGE>
__global__ void __launch_bounds__(DX_THREADS, 1)
    read_bwd_dx_tma_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_du,
                           const float* __restrict__ M, const float* __restrict__ ds, T* __restrict__ dx,
                           const T* __restrict__ dx_add, int hw, int K, int tiles_per_img, int ntiles, int UC) {
    constexpr int CW = C / DX_WARPS;
    extern __shared__ __align__(1024) unsigned char smraw_[];
    __shared__ __align__(8) uint64_t full[NSTAGE];
    // TMA destinations want 128-byte alignment: round the dynamic window up ourselves (1 KB of slack is allocated)
    unsigned char* smraw = smraw_ + ((1024u - (smem_u32(smraw_) & 1023u)) & 1023u);
    T* xs = reinterpret_cast<T*>(smraw);                                   // [NSTAGE][2][C][TP]: x tile, dq0 tile
    float* dss = reinterpret_cast<float*>(xs + (size_t)NSTAGE * 2 * C * TP);  // [NSTAGE][TP][KP]
    float* Mt = dss + NSTAGE * TP * KP;                                    // [C][KP]
    float* pn = Mt + C * KP;                                               // [16][TP]
    float* pd = pn + DX_WARPS * TP;                                        // [16][TP]

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < NSTAGE; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    auto issue = [&](int t, int s) {  // one thread
        const int b = t / tiles_per_img, px0 = (t - b * tiles_per_img) * TP;
        const int nvalid = min(TP, hw - px0);
        const uint32_t ds_bytes = (uint32_t)(nvalid * KP * sizeof(float));
        T* base = xs + (size_t)s * 2 * C * TP;
        mbar_expect_tx(&full[s], (uint32_t)(2 * C * TP * sizeof(T)) + ds_bytes);
        tma_load_2d(base, &tm_x, px0, b * C, &full[s]);
        tma_load_2d(base + C * TP, &tm_du, px0, b * UC, &full[s]);
        bulk_load_1d(dss + s * TP * KP, ds + ((size_t)b * hw + px0) * KP, ds_bytes, &full[s]);
    };
    int tile = blockIdx.x;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < NSTAGE; ++s) {
            const int t = tile + s * gridDim.x;
            if (t < ntiles) issue(t, s);
        }
    }
    for (int i = tid; i < C * KP; i += DX_THREADS) {
        const int c = i / KP, k = i - c * KP;
        Mt[i] = (k < K) ? __ldg(M + (size_t)k * C + c) : 0.f;
    }
    __syncthreads();

    int stage = 0;
    unsigned phase = 0;
    for (; tile < ntiles; tile += gridDim.x) {
        mbar_wait(&full[stage], phase);
        const T* xt = xs + (size_t)stage * 2 * C * TP;
        const T* qt = xt + C * TP;
        const int b = tile / tiles_per_img, px0 = (tile - b * tiles_per_img) * TP;
        const int nvalid = min(TP, hw - px0);
        const T* xcol = xt + wid * CW * 32 + lane;
        const T* qcol = qt + wid * CW * 32 + lane;
        const size_t o0 = ((size_t)b * C + wid * CW) * hw + px0 + lane;
        float av[CW];  // a second gradient of x (the write branch's), summed here instead of by an add kernel
#pragma unroll
        for (int j = 0; j < CW; ++j) av[j] = (dx_add != nullptr && lane < nvalid) ? ldf(dx_add + o0 + (size_t)j * hw) : 0.f;
        float xv[CW], n2 = 0.f;
#pragma unroll
        for (int j = 0; j < CW; ++j) {
            xv[j] = to_float(xcol[j * 32]);
            n2 = fmaf(xv[j], xv[j], n2);
        }
        pn[wid * TP + lane] = n2;
        float2 s2[KP / 2];
        {
            const float4* sr = reinterpret_cast<const float4*>(dss + stage * TP * KP + lane * KP);
#pragma unroll
            for (int q = 0; q < KP / 4; ++q) {
                float4 v = sr[q];
                if (lane >= nvalid) v = make_float4(0.f, 0.f, 0.f, 0.f);  // rows past the image end are not copied
                s2[2 * q] = f2(v.x, v.y);
                s2[2 * q + 1] = f2(v.z, v.w);
            }
        }
        float dq[CW];
        const float4* mbase = reinterpret_cast<const float4*>(Mt + wid * CW * KP);
#pragma unroll
        for (int j = 0; j < CW; ++j) {
            const float4* mrow = mbase + j * (KP / 4);
            float2 acc = f2(to_float(qcol[j * 32]), 0.f);
#pragma unroll
            for (int q = 0; q < KP / 4; ++q) {
                const float4 m = mrow[q];
                acc = __ffma2_rn(s2[2 * q], f2(m.x, m.y), acc);
                acc = __ffma2_rn(s2[2 * q + 1], f2(m.z, m.w), acc);
            }
            dq[j] = acc.x + acc.y;
        }
        __syncthreads();
        float nn = 0.f;
#pragma unroll
        for (int w = 0; w < DX_WARPS; ++w) nn += pn[w * TP + lane];
        const float nrm = sqrtf(nn), ir = 1.f / fmaxf(nrm, PM_NORM_EPS);
        float dot = 0.f;
#pragma unroll
        for (int j = 0; j < CW; ++j) {
            xv[j] *= ir;  // q
            dot = fmaf(xv[j], dq[j], dot);
        }
        pd[wid * TP + lane] = dot;
        __syncthreads();  // also: every read of this stage's tiles is done
        const int next = tile + NSTAGE * gridDim.x;
        if (tid == 0 && next < ntiles) issue(next, stage);
        dot = 0.f;
#pragma unroll
        for (int w = 0; w < DX_WARPS; ++w) dot += pd[w * TP + lane];
        if (nrm <= PM_NORM_EPS) dot = 0.f;
        if (lane < nvalid) {
            T* dxp = dx + o0;
#pragma unroll
            for (int j = 0; j < CW; ++j) {
                stf(dxp, (dq[j] - xv[j] * dot) * ir + av[j]);
                dxp += hw;
            }
        }
        if (++stage == NSTAGE) stage = 0, phase ^= 1u;
    }
}


// ---------------------------------------------------------------- backward, part B for bf16 maps on the tensor core
// Same arithmetic; what changes is who does it. The K-slot contraction dq = dq0 + ds . M runs on mma.sync m16n8k16
// (ds and M split bf16 hi + lo, three products, fp32 accumulate: 2^-16 relative), the x and dq0 values arrive as
// `ldmatrix.trans` fragments in the accumulator layout (no 2-byte shared-memory loads, no conversions per element),
// the result is packed back in place over the dq0 tile with `stmatrix.trans` and leaves as ONE TMA store per tile.
// 8 warps x C/8 channels, 2 CTAs per SM. One barrier pair per tile: |x|^2 and x.dq are reduced together
// (q.dq = x.dq / |x|).
__device__ __forceinline__ void stmatrix_x4_trans(uint32_t saddr, const unsigned (&r)[4]) {
    asm volatile("stmatrix.sync.aligned.m8n8.x4.trans.shared.b16 [%0], {%1,%2,%3,%4};" ::"r"(saddr), "r"(r[0]), "r"(r[1]),
                 "r"(r[2]), "r"(r[3])
                 : "memory");
}
__device__ __forceinline__ void tma_store_tile_2d(const CUtensorMap* map, const void* src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(map)),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1)
                 : "memory");
}

constexpr int DXB_THREADS = 256, DXB_WARPS = 8;

template <int C, int KP, int NSTAGE>
__global__ void __launch_bounds__(DXB_THREADS, 2)
    read_bwd_dx_bf16_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_du,
                            const __grid_constant__ CUtensorMap tm_dx, const float* __restrict__ M,
                            const float* __restrict__ ds, int hw, int K, int tiles_per_img, int ntiles, int UC) {
    using T = __nv_bfloat16;
    constexpr int CW = C / DXB_WARPS, NN = CW / 8, KS = 2, LDK = C + 8;  // LDK % 32 == 8
    static_assert(CW % 8 == 0 && KP <= 32, "channel slice must be whole 8-channel blocks");
    extern __shared__ __align__(1024) unsigned char smraw_[];
    __shared__ __align__(8) uint64_t full[NSTAGE];
    unsigned char* smraw = smraw_ + ((1024u - (smem_u32(smraw_) & 1023u)) & 1023u);
    T* xs = reinterpret_cast<T*>(smraw);                                      // [NSTAGE][2][C][TP]: x tile, dq0 tile
    float* dss = reinterpret_cast<float*>(xs + (size_t)NSTAGE * 2 * C * TP);   // [NSTAGE][TP][KP]
    unsigned* Mk_hi = reinterpret_cast<unsigned*>(dss + NSTAGE * TP * KP);     // [16][LDK]: (M[2kp][c], M[2kp+1][c])
    unsigned* Mk_lo = Mk_hi + 8 * KS * LDK;
    float* pn = reinterpret_cast<float*>(Mk_lo + 8 * KS * LDK);                // [8][TP]
    float* pd = pn + DXB_WARPS * TP;                                           // [8][TP]

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < NSTAGE; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    auto issue = [&](int tl, int s) {  // one thread
        const int b = tl / tiles_per_img, px0 = (tl - b * tiles_per_img) * TP;
        const int nvalid = min(TP, hw - px0);
        const uint32_t ds_bytes = (uint32_t)(nvalid * KP * sizeof(float));
        T* base = xs + (size_t)s * 2 * C * TP;
        mbar_expect_tx(&full[s], (uint32_t)(2 * C * TP * sizeof(T)) + ds_bytes);
        tma_load_2d(base, &tm_x, px0, b * C, &full[s]);
        tma_load_2d(base + C * TP, &tm_du, px0, b * UC, &full[s]);
        bulk_load_1d(dss + s * TP * KP, ds + ((size_t)b * hw + px0) * KP, ds_bytes, &full[s]);
    };
    int tile = blockIdx.x;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < NSTAGE; ++s) {
            const int tl = tile + s * gridDim.x;
            if (tl < ntiles) issue(tl, s);
        }
    }
    for (int i = tid; i < 8 * KS * C; i += DXB_THREADS) {
        const int kp = i / C, c = i - kp * C;
        const float a = (2 * kp < K) ? __ldg(M + (size_t)(2 * kp) * C + c) : 0.f;
        const float b = (2 * kp + 1 < K) ? __ldg(M + (size_t)(2 * kp + 1) * C + c) : 0.f;
        const float ah = __bfloat162float(__float2bfloat16_rn(a)), bh = __bfloat162float(__float2bfloat16_rn(b));
        Mk_hi[kp * LDK + c] = pack_bf16(ah, bh);
        Mk_lo[kp * LDK + c] = pack_bf16(a - ah, b - bh);
    }
    __syncthreads();

    const int c0 = wid * CW;
    const int mj = lane >> 3, rr = lane & 7;  // ldmatrix / stmatrix: this lane addresses row rr of matrix mj
    int stage = 0, pending = -1;              // `pending`: stage whose tile was handed to the TMA store last iteration
    unsigned phase = 0;
    for (; tile < ntiles; tile += gridDim.x) {
        if (tid == 0 && pending >= 0) {  // refill the previous stage once its store has finished reading shared memory
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            const int next = tile + (NSTAGE - 1) * (int)gridDim.x;
            if (next < ntiles) issue(next, pending);
        }
        mbar_wait(&full[stage], phase);
        T* xt = xs + (size_t)stage * 2 * C * TP;
        T* qt = xt + C * TP;
        const int b = tile / tiles_per_img, px0 = (tile - b * tiles_per_img) * TP;
        const int nvalid = min(TP, hw - px0);
        // A fragments of ds [32 px][32 slots]: a[m][ks] = rows g+16m / g+8+16m, slots 16ks+2t(+1) / +8
        unsigned ahi[2][KS][4], alo[2][KS][4];
        {
            const float* dsr = dss + stage * TP * KP;
#pragma unroll
            for (int m = 0; m < 2; ++m)
#pragma unroll
                for (int ks = 0; ks < KS; ++ks)
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int px = g + 16 * m + 8 * (e & 1), k = 16 * ks + 2 * t + 8 * (e >> 1);
                        float2 v = make_float2(0.f, 0.f);
                        if (k < KP && px < nvalid) v = *reinterpret_cast<const float2*>(dsr + px * KP + k);  // KP even
                        const float hx = __bfloat162float(__float2bfloat16_rn(v.x)), hy = __bfloat162float(__float2bfloat16_rn(v.y));
                        ahi[m][ks][e] = pack_bf16(hx, hy);
                        alo[m][ks][e] = pack_bf16(v.x - hx, v.y - hy);
                    }
        }
        float dq[NN][2][4];      // [n][m][c-fragment]
        unsigned xr[NN][4];      // x fragments: block j = pixels 8j..8j+7, halves = channels 2t, 2t+1 of the n-th block
        float n2[4] = {0.f, 0.f, 0.f, 0.f}, xd[4] = {0.f, 0.f, 0.f, 0.f};  // pixels g + 8j
#pragma unroll
        for (int n = 0; n < NN; ++n) {
            const int row = c0 + 8 * n + rr;
            const uint32_t off = (uint32_t)(row * 64 + ((mj ^ ((row >> 1) & 3)) << 4));
            unsigned qr[4];
            ldmatrix_x4_trans(xr[n], smem_u32(xt) + off);
            ldmatrix_x4_trans(qr, smem_u32(qt) + off);
#pragma unroll
            for (int m = 0; m < 2; ++m) {
                dq[n][m][0] = bf16_lo_f(qr[2 * m]), dq[n][m][1] = bf16_hi_f(qr[2 * m]);
                dq[n][m][2] = bf16_lo_f(qr[2 * m + 1]), dq[n][m][3] = bf16_hi_f(qr[2 * m + 1]);
            }
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
                const int cidx = (8 * ks + t) * LDK + c0 + 8 * n + g;
                const unsigned b0h = Mk_hi[cidx], b1h = Mk_hi[cidx + 4 * LDK], b0l = Mk_lo[cidx], b1l = Mk_lo[cidx + 4 * LDK];
#pragma unroll
                for (int m = 0; m < 2; ++m) {
                    mma_bf16(dq[n][m], alo[m][ks], b0h, b1h);
                    mma_bf16(dq[n][m], ahi[m][ks], b0l, b1l);
                    mma_bf16(dq[n][m], ahi[m][ks], b0h, b1h);
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float x0 = bf16_lo_f(xr[n][j]), x1 = bf16_hi_f(xr[n][j]);
                const float d0 = dq[n][j >> 1][2 * (j & 1)], d1 = dq[n][j >> 1][2 * (j & 1) + 1];
                n2[j] = fmaf(x0, x0, fmaf(x1, x1, n2[j]));
                xd[j] = fmaf(x0, d0, fmaf(x1, d1, xd[j]));
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            n2[j] += __shfl_xor_sync(0xffffffffu, n2[j], 1);
            n2[j] += __shfl_xor_sync(0xffffffffu, n2[j], 2);
            xd[j] += __shfl_xor_sync(0xffffffffu, xd[j], 1);
            xd[j] += __shfl_xor_sync(0xffffffffu, xd[j], 2);
            if (t == 0) pn[wid * TP + g + 8 * j] = n2[j], pd[wid * TP + g + 8 * j] = xd[j];
        }
        __syncthreads();
        float ir[4], cf[4];  // 1/|x| and (x.dq)/|x|^2 of pixels g + 8j
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float nn = 0.f, dd = 0.f;
#pragma unroll
            for (int w = 0; w < DXB_WARPS; ++w) nn += pn[w * TP + g + 8 * j], dd += pd[w * TP + g + 8 * j];
            const float nrm = sqrtf(nn);
            ir[j] = 1.f / fmaxf(nrm, PM_NORM_EPS);
            cf[j] = (nrm <= PM_NORM_EPS) ? 0.f : dd * ir[j] * ir[j];  // F.normalize clamps: no projection below eps
        }
#pragma unroll
        for (int n = 0; n < NN; ++n) {
            unsigned o[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float x0 = bf16_lo_f(xr[n][j]), x1 = bf16_hi_f(xr[n][j]);
                const float d0 = dq[n][j >> 1][2 * (j & 1)], d1 = dq[n][j >> 1][2 * (j & 1) + 1];
                o[j] = pack_bf16((d0 - x0 * cf[j]) * ir[j], (d1 - x1 * cf[j]) * ir[j]);
            }
            const int row = c0 + 8 * n + rr;
            stmatrix_x4_trans(smem_u32(qt) + (uint32_t)(row * 64 + ((mj ^ ((row >> 1) & 3)) << 4)), o);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();  // the dx tile is complete in shared memory; every read of this stage is done
        if (tid == 0) {
            tma_store_tile_2d(&tm_dx, qt, px0, b * C);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        (void)nvalid;
        pending = stage;
        if (++stage == NSTAGE) stage = 0, phase ^= 1u;
    }
    if (tid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

template <typename T, int C, int KP>
int launch_read_bwd_tiled(const void* du, const void* x, const float* M, const float* p, const float* ds_rl,
                          const float* g_loss, const float* rl_out, void* dx, const void* dx_add, float* ds, int B, int hw,
                          int K, int planes, cudaStream_t st) {
    constexpr int NSTAGE = 2;
    const int tiles = (hw + TP - 1) / TP, ntiles = B * tiles;
    const int UC = planes ? C + PM_PLANES : 2 * C;
    if (planes) {  // dp comes back from the convolution as planes [C, C+K) of du: per-pixel softmax backward only
        const long long N = (long long)B * hw;
        read_bwd_ds_planes_kernel<T, KP><<<(unsigned)((N + 255) / 256), 256, 0, st>>>((const T*)du, p, ds_rl, g_loss, rl_out,
                                                                                    ds, hw, C, K, UC, N);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return (int)e;
    } else {
        const size_t smem = sizeof(float) * ((size_t)C * KP + TL_WARPS * TP * KP + TP * KP) +
                            sizeof(T) * (size_t)NSTAGE * C * TP;
        auto kern = read_bwd_ds_tiled_kernel<T, C, KP, NSTAGE>;
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        int grid = 2 * 148;
        if (grid > ntiles) grid = ntiles;
        kern<<<grid, TL_THREADS, smem, st>>>((const T*)du, M, p, ds_rl, g_loss, rl_out, ds, hw, K, tiles, ntiles);
        e = cudaGetLastError();
        if (e != cudaSuccess) return (int)e;
    }
    CUtensorMap tm_x, tm_du;
    cudaError_t e;
    if constexpr (sizeof(T) == 2 && (C == 128 || C == 256)) {
        if (dx_add == nullptr) {
            CUtensorMap tm_dx;
            if (!make_map_2d<T>(&tm_x, x, (size_t)B * C, hw, C, TP, 3) || !make_map_2d<T>(&tm_du, du, (size_t)B * UC, hw, C, TP, 3) ||
                !make_map_2d<T>(&tm_dx, dx, (size_t)B * C, hw, C, TP, 3))
                return PM_ERR_ALIGN;
            constexpr int NS = 2;
            const size_t sm = sizeof(T) * (size_t)NS * 2 * C * TP + sizeof(float) * ((size_t)NS * TP * KP + 2 * DXB_WARPS * TP) +
                              sizeof(unsigned) * 2 * 16 * (C + 8) + 1024;
            auto kern = read_bwd_dx_bf16_kernel<C, KP, NS>;
            e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
            if (e != cudaSuccess) return (int)e;
            int g2 = 2 * 148;
            if (g2 > ntiles) g2 = ntiles;
            kern<<<g2, DXB_THREADS, sm, st>>>(tm_x, tm_du, tm_dx, M, ds, hw, K, tiles, ntiles, UC);
            e = cudaGetLastError();
            return e == cudaSuccess ? 0 : (int)e;
        }
    }
    if (!make_map_2d<T>(&tm_x, x, (size_t)B * C, hw, C, TP, false) || !make_map_2d<T>(&tm_du, du, (size_t)B * UC, hw, C, TP, false))
        return PM_ERR_ALIGN;
    const size_t smem = sizeof(float) * ((size_t)C * KP + 2 * DX_WARPS * TP + (size_t)NSTAGE * TP * KP) +
                        sizeof(T) * (size_t)NSTAGE * 2 * C * TP + 1024;
    auto kern = read_bwd_dx_tma_kernel<T, C, KP, NSTAGE>;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    int grid = 148;
    if (grid > ntiles) grid = ntiles;
    kern<<<grid, DX_THREADS, smem, st>>>(tm_x, tm_du, M, ds, (T*)dx, (const T*)dx_add, hw, K, tiles, ntiles, UC);
    e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

#define PM_TILED_SWITCH_C(T, KP, FN, ...)                   \
    switch (C) {                                            \
        case 32: return FN<T, 32, KP>(__VA_ARGS__);         \
        case 64: return FN<T, 64, KP>(__VA_ARGS__);         \
        case 128: return FN<T, 128, KP>(__VA_ARGS__);       \
        case 256: return FN<T, 256, KP>(__VA_ARGS__);       \
        default: return PM_ERR_CHANNELS;                    \
    }

bool tiled_ok(const void* p0, const void* p1, const void* p2, int hw, int dtype) {
    const int epc = dtype == PM_F32 ? 4 : 8;
    return (hw % epc) == 0 && (((uintptr_t)p0 | (uintptr_t)p1 | (uintptr_t)p2) & 15) == 0;
}

int read_fwd_tiled(const void* x, const float* M, const float* gum_m, const float* gum_q, void* u, float* s, float* p,
                   float* colpart, int B, int C, int hw, int K, int dtype, int planes, cudaStream_t st) {
    if (dtype == PM_F32) {
        if (K <= 19) { PM_TILED_SWITCH_C(float, 20, launch_read_fwd_tiled, x, M, gum_m, gum_q, u, s, p, colpart, B, hw, K, planes, st) }
        else { PM_TILED_SWITCH_C(float, 32, launch_read_fwd_tiled, x, M, gum_m, gum_q, u, s, p, colpart, B, hw, K, planes, st) }
    } else {
        if (K <= 19) { PM_TILED_SWITCH_C(__nv_bfloat16, 20, launch_read_fwd_tiled, x, M, gum_m, gum_q, u, s, p, colpart, B, hw, K, planes, st) }
        else { PM_TILED_SWITCH_C(__nv_bfloat16, 32, launch_read_fwd_tiled, x, M, gum_m, gum_q, u, s, p, colpart, B, hw, K, planes, st) }
    }
}

int read_bwd_tiled(const void* du, const void* x, const float* M, const float* p, const float* ds_rl,
                   const float* g_loss, const float* rl_out, void* dx, const void* dx_add, float* ds, int B, int C, int hw,
                   int K, int dtype, int planes, cudaStream_t st) {
    if (dtype == PM_F32) {
        if (K <= 19) { PM_TILED_SWITCH_C(float, 20, launch_read_bwd_tiled, du, x, M, p, ds_rl, g_loss, rl_out, dx, dx_add, ds, B, hw, K, planes, st) }
        else { PM_TILED_SWITCH_C(float, 32, launch_read_bwd_tiled, du, x, M, p, ds_rl, g_loss, rl_out, dx, dx_add, ds, B, hw, K, planes, st) }
    } else {
        if (K <= 19) { PM_TILED_SWITCH_C(__nv_bfloat16, 20, launch_read_bwd_tiled, du, x, M, p, ds_rl, g_loss, rl_out, dx, dx_add, ds, B, hw, K, planes, st) }
        else { PM_TILED_SWITCH_C(__nv_bfloat16, 32, launch_read_bwd_tiled, du, x, M, p, ds_rl, g_loss, rl_out, dx, dx_add, ds, B, hw, K, planes, st) }
    }
}

}  // namespace pm
