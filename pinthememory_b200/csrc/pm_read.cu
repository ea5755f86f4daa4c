// Memory read: forward, backward, dM, and the NHWC get_score similarity.
//
// Layout idea (all three big kernels): features stay NCHW, so for a fixed channel the pixels of one
// image are contiguous. A CTA owns a tile of P=64 consecutive pixels of one image and all C channels;
// its 8 warps split the channels (CW = C/8 each) and every lane owns two pixels (lane, lane+32), so
// each channel row is fetched with two fully coalesced 128-byte (fp32) warp loads and every memory
// value pulled from shared memory feeds two FMAs. The K x C memory lives transposed in shared memory
// (Mt[c][k], k padded to KP so a channel's K values are 16-byte vectors, broadcast to the warp).
// Per-pixel quantities that need all channels (|x|^2 and the K similarities) are reduced across the
// 8 warps through shared memory.
#include "pm_common.cuh"
#include "pm_internal.h"

namespace pm {

constexpr int RD_THREADS = 256;
constexpr int RD_WARPS = 8;
constexpr int RD_P = 64;

template <int C, int KP>
__device__ __forceinline__ void load_memory_transposed(float* Mt, const float* __restrict__ M, int K) {
    for (int i = threadIdx.x; i < C * KP; i += RD_THREADS) {
        int c = i / KP, k = i - c * KP;
        Mt[i] = (k < K) ? __ldg(M + (size_t)k * C + c) : 0.f;
    }
}

// Sum the 8 per-warp partial [P][KP] blocks into block 0 and the 8 partial |x|^2 into inv-norms.
template <int KP>
__device__ __forceinline__ void reduce_partials(float* part, const float* pn, float* invr, float* rnorm) {
    for (int o = threadIdx.x; o < RD_P * KP; o += RD_THREADS) {
        float sum = 0.f;
#pragma unroll
        for (int w = 0; w < RD_WARPS; ++w) sum += part[w * RD_P * KP + o];
        part[o] = sum;
    }
    if (threadIdx.x < RD_P) {
        float n2 = 0.f;
#pragma unroll
        for (int w = 0; w < RD_WARPS; ++w) n2 += pn[w * RD_P + threadIdx.x];
        float n = sqrtf(n2);
        invr[threadIdx.x] = 1.f / fmaxf(n, PM_NORM_EPS);
        if (rnorm) rnorm[threadIdx.x] = n;
    }
}

// ------------------------------------------------------------------------------------------ forward

template <typename T, int CW, int KP>
__global__ void __launch_bounds__(RD_THREADS) read_fwd_kernel(const T* __restrict__ x, const float* __restrict__ M,
                                                              const float* __restrict__ gum, T* __restrict__ u,
                                                              float* __restrict__ s_out, float* __restrict__ p_out,
                                                              int hw, int K, int tiles_per_img) {
    constexpr int C = CW * RD_WARPS, P = RD_P;
    extern __shared__ __align__(16) float smem[];
    float* Mt = smem;                   // [C][KP]
    float* part = Mt + C * KP;          // [8][P][KP]
    float* pn = part + RD_WARPS * P * KP;  // [8][P]
    float* invr = pn + RD_WARPS * P;    // [P]

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int b = blockIdx.x / tiles_per_img, px0 = (blockIdx.x - b * tiles_per_img) * P;
    const int nvalid = min(P, hw - px0);
    const bool v0 = lane < nvalid, v1 = lane + 32 < nvalid;

    // issue all feature loads first (2*CW independent coalesced loads per thread)
    const T* xb = x + ((size_t)b * C + wid * CW) * hw + px0 + lane;
    float xv0[CW], xv1[CW];
#pragma unroll
    for (int j = 0; j < CW; ++j) {
        xv0[j] = v0 ? ldf(xb + (size_t)j * hw) : 0.f;
        xv1[j] = v1 ? ldf(xb + (size_t)j * hw + 32) : 0.f;
    }
    load_memory_transposed<C, KP>(Mt, M, K);
    __syncthreads();

    float a0[KP], a1[KP], n0 = 0.f, n1 = 0.f;
#pragma unroll
    for (int k = 0; k < KP; ++k) a0[k] = a1[k] = 0.f;
#pragma unroll
    for (int j = 0; j < CW; ++j) {
        const float4* mrow = reinterpret_cast<const float4*>(Mt + (wid * CW + j) * KP);
        n0 = fmaf(xv0[j], xv0[j], n0);
        n1 = fmaf(xv1[j], xv1[j], n1);
#pragma unroll
        for (int q = 0; q < KP / 4; ++q) {
            float4 m = mrow[q];
            a0[4 * q + 0] = fmaf(xv0[j], m.x, a0[4 * q + 0]);
            a0[4 * q + 1] = fmaf(xv0[j], m.y, a0[4 * q + 1]);
            a0[4 * q + 2] = fmaf(xv0[j], m.z, a0[4 * q + 2]);
            a0[4 * q + 3] = fmaf(xv0[j], m.w, a0[4 * q + 3]);
            a1[4 * q + 0] = fmaf(xv1[j], m.x, a1[4 * q + 0]);
            a1[4 * q + 1] = fmaf(xv1[j], m.y, a1[4 * q + 1]);
            a1[4 * q + 2] = fmaf(xv1[j], m.z, a1[4 * q + 2]);
            a1[4 * q + 3] = fmaf(xv1[j], m.w, a1[4 * q + 3]);
        }
    }
    {
        float4* d0 = reinterpret_cast<float4*>(part + ((size_t)wid * P + lane) * KP);
        float4* d1 = reinterpret_cast<float4*>(part + ((size_t)wid * P + lane + 32) * KP);
#pragma unroll
        for (int q = 0; q < KP / 4; ++q) {
            d0[q] = make_float4(a0[4 * q], a0[4 * q + 1], a0[4 * q + 2], a0[4 * q + 3]);
            d1[q] = make_float4(a1[4 * q], a1[4 * q + 1], a1[4 * q + 2], a1[4 * q + 3]);
        }
        pn[wid * P + lane] = n0;
        pn[wid * P + lane + 32] = n1;
    }
    __syncthreads();
    reduce_partials<KP>(part, pn, invr, nullptr);
    __syncthreads();

    // per-pixel softmax over the K slots (64 threads), raw s and p staged for coalesced write-out
    float* s_sm = part + P * KP;      // [P][KP]  (partial block 1, already consumed)
    float* p_sm = part + 2 * P * KP;  // [P][K] dense
    if (tid < P) {
        const float ir = invr[tid];
        const size_t n = (size_t)b * hw + px0 + tid;
        float z[KP], mx = -INFINITY;
#pragma unroll
        for (int k = 0; k < KP; ++k) {
            float sv = part[tid * KP + k] * ir;
            s_sm[tid * KP + k] = (k < K) ? sv : 0.f;
            float g = (gum != nullptr && k < K && tid < nvalid) ? __ldg(gum + n * K + k) : 0.f;
            z[k] = (k < K) ? sv + g : -INFINITY;
            mx = fmaxf(mx, z[k]);
        }
        float sum = 0.f;
#pragma unroll
        for (int k = 0; k < KP; ++k) {
            z[k] = (k < K) ? expf(z[k] - mx) : 0.f;
            sum += z[k];
        }
        const float inv = 1.f / sum;
#pragma unroll
        for (int k = 0; k < KP; ++k)
            if (k < K) p_sm[tid * K + k] = z[k] * inv;
    }
    __syncthreads();

    {
        const size_t n0g = (size_t)b * hw + px0;
        for (int o = tid; o < nvalid * KP; o += RD_THREADS) s_out[n0g * KP + o] = s_sm[o];
        for (int o = tid; o < nvalid * K; o += RD_THREADS) p_out[n0g * K + o] = p_sm[o];
    }

    // u = [q ; p.M]
    float p0[KP], p1[KP];
#pragma unroll
    for (int k = 0; k < KP; ++k) {
        p0[k] = (k < K) ? p_sm[lane * K + k] : 0.f;
        p1[k] = (k < K) ? p_sm[(lane + 32) * K + k] : 0.f;
    }
    const float ir0 = invr[lane], ir1 = invr[lane + 32];
    T* uq = u + ((size_t)b * 2 * C + wid * CW) * hw + px0 + lane;
    T* uc = uq + (size_t)C * hw;
#pragma unroll
    for (int j = 0; j < CW; ++j) {
        const float4* mrow = reinterpret_cast<const float4*>(Mt + (wid * CW + j) * KP);
        float c0 = 0.f, c1 = 0.f;
#pragma unroll
        for (int q = 0; q < KP / 4; ++q) {
            float4 m = mrow[q];
            c0 = fmaf(p0[4 * q + 0], m.x, c0);
            c0 = fmaf(p0[4 * q + 1], m.y, c0);
            c0 = fmaf(p0[4 * q + 2], m.z, c0);
            c0 = fmaf(p0[4 * q + 3], m.w, c0);
            c1 = fmaf(p1[4 * q + 0], m.x, c1);
            c1 = fmaf(p1[4 * q + 1], m.y, c1);
            c1 = fmaf(p1[4 * q + 2], m.z, c1);
            c1 = fmaf(p1[4 * q + 3], m.w, c1);
        }
        if (v0) {
            stf(uq + (size_t)j * hw, xv0[j] * ir0);
            stf(uc + (size_t)j * hw, c0);
        }
        if (v1) {
            stf(uq + (size_t)j * hw + 32, xv1[j] * ir1);
            stf(uc + (size_t)j * hw + 32, c1);
        }
    }
}

// ----------------------------------------------------------------------------------------- backward

template <typename T, int CW, int KP>
__global__ void __launch_bounds__(RD_THREADS) read_bwd_kernel(const T* __restrict__ du, const T* __restrict__ x,
                                                              const float* __restrict__ M,
                                                              const float* __restrict__ p_in,
                                                              const float* __restrict__ ds_rl,
                                                              const float* __restrict__ g_loss,
                                                              const float* __restrict__ rl_out, T* __restrict__ dx,
                                                              float* __restrict__ ds_out, int hw, int K,
                                                              int tiles_per_img) {
    constexpr int C = CW * RD_WARPS, P = RD_P;
    extern __shared__ __align__(16) float smem[];
    float* Mt = smem;
    float* part = Mt + C * KP;
    float* pn = part + RD_WARPS * P * KP;
    float* invr = pn + RD_WARPS * P;
    float* rnorm = invr + P;

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int b = blockIdx.x / tiles_per_img, px0 = (blockIdx.x - b * tiles_per_img) * P;
    const int nvalid = min(P, hw - px0);
    const bool v0 = lane < nvalid, v1 = lane + 32 < nvalid;

    const T* xb = x + ((size_t)b * C + wid * CW) * hw + px0 + lane;
    const T* dqb = du + ((size_t)b * 2 * C + wid * CW) * hw + px0 + lane;
    const T* dcb = dqb + (size_t)C * hw;
    float xv0[CW], xv1[CW], g0[CW], g1[CW];  // g*: first dc, later dq
#pragma unroll
    for (int j = 0; j < CW; ++j) {
        xv0[j] = v0 ? ldf(xb + (size_t)j * hw) : 0.f;
        xv1[j] = v1 ? ldf(xb + (size_t)j * hw + 32) : 0.f;
        g0[j] = v0 ? ldf(dcb + (size_t)j * hw) : 0.f;
        g1[j] = v1 ? ldf(dcb + (size_t)j * hw + 32) : 0.f;
    }
    load_memory_transposed<C, KP>(Mt, M, K);
    __syncthreads();

    // dp[k] = M[k] . dc   (partial over this warp's channels), |x|^2
    {
        float a0[KP], a1[KP], n0 = 0.f, n1 = 0.f;
#pragma unroll
        for (int k = 0; k < KP; ++k) a0[k] = a1[k] = 0.f;
#pragma unroll
        for (int j = 0; j < CW; ++j) {
            const float4* mrow = reinterpret_cast<const float4*>(Mt + (wid * CW + j) * KP);
            n0 = fmaf(xv0[j], xv0[j], n0);
            n1 = fmaf(xv1[j], xv1[j], n1);
#pragma unroll
            for (int q = 0; q < KP / 4; ++q) {
                float4 m = mrow[q];
                a0[4 * q + 0] = fmaf(g0[j], m.x, a0[4 * q + 0]);
                a0[4 * q + 1] = fmaf(g0[j], m.y, a0[4 * q + 1]);
                a0[4 * q + 2] = fmaf(g0[j], m.z, a0[4 * q + 2]);
                a0[4 * q + 3] = fmaf(g0[j], m.w, a0[4 * q + 3]);
                a1[4 * q + 0] = fmaf(g1[j], m.x, a1[4 * q + 0]);
                a1[4 * q + 1] = fmaf(g1[j], m.y, a1[4 * q + 1]);
                a1[4 * q + 2] = fmaf(g1[j], m.z, a1[4 * q + 2]);
                a1[4 * q + 3] = fmaf(g1[j], m.w, a1[4 * q + 3]);
            }
        }
        float4* d0 = reinterpret_cast<float4*>(part + ((size_t)wid * P + lane) * KP);
        float4* d1 = reinterpret_cast<float4*>(part + ((size_t)wid * P + lane + 32) * KP);
#pragma unroll
        for (int q = 0; q < KP / 4; ++q) {
            d0[q] = make_float4(a0[4 * q], a0[4 * q + 1], a0[4 * q + 2], a0[4 * q + 3]);
            d1[q] = make_float4(a1[4 * q], a1[4 * q + 1], a1[4 * q + 2], a1[4 * q + 3]);
        }
        pn[wid * P + lane] = n0;
        pn[wid * P + lane + 32] = n1;
    }
    // the dq half of du is not needed until after the softmax backward: fetch it now
#pragma unroll
    for (int j = 0; j < CW; ++j) {
        g0[j] = v0 ? ldf(dqb + (size_t)j * hw) : 0.f;
        g1[j] = v1 ? ldf(dqb + (size_t)j * hw + 32) : 0.f;
    }
    __syncthreads();
    reduce_partials<KP>(part, pn, invr, rnorm);
    __syncthreads();

    // ds = p * (dp - p.dp) + scale * ds_rl     (64 threads)
    float* ds_sm = part + P * KP;  // [P][KP]
    if (tid < P) {
        const size_t n = (size_t)b * hw + px0 + tid;
        const bool valid = tid < nvalid;
        float scale = 0.f;
        if (ds_rl != nullptr && g_loss != nullptr && rl_out != nullptr) scale = __ldg(g_loss) * __ldg(rl_out + 1);
        float pk[KP], dot = 0.f;
#pragma unroll
        for (int k = 0; k < KP; ++k) {
            pk[k] = (k < K && valid) ? __ldg(p_in + n * K + k) : 0.f;
            dot = fmaf(pk[k], part[tid * KP + k], dot);
        }
#pragma unroll
        for (int k = 0; k < KP; ++k) {
            float d = pk[k] * (part[tid * KP + k] - dot);
            if (scale != 0.f && k < K && valid) d = fmaf(scale, __ldg(ds_rl + n * KP + k), d);
            ds_sm[tid * KP + k] = (k < K) ? d : 0.f;
        }
    }
    __syncthreads();
    if (ds_out != nullptr) {
        const size_t n0g = (size_t)b * hw + px0;
        for (int o = tid; o < nvalid * KP; o += RD_THREADS) ds_out[n0g * KP + o] = ds_sm[o];
    }

    // dq = dq0 + ds.M ; dx = (dq - q (q.dq)) / |x|
    float s0[KP], s1[KP];
    {
        const float4* r0 = reinterpret_cast<const float4*>(ds_sm + lane * KP);
        const float4* r1 = reinterpret_cast<const float4*>(ds_sm + (lane + 32) * KP);
#pragma unroll
        for (int q = 0; q < KP / 4; ++q) {
            float4 a = r0[q], c = r1[q];
            s0[4 * q] = a.x, s0[4 * q + 1] = a.y, s0[4 * q + 2] = a.z, s0[4 * q + 3] = a.w;
            s1[4 * q] = c.x, s1[4 * q + 1] = c.y, s1[4 * q + 2] = c.z, s1[4 * q + 3] = c.w;
        }
    }
    const float ir0 = invr[lane], ir1 = invr[lane + 32];
    float dot0 = 0.f, dot1 = 0.f;
#pragma unroll
    for (int j = 0; j < CW; ++j) {
        const float4* mrow = reinterpret_cast<const float4*>(Mt + (wid * CW + j) * KP);
        float c0 = g0[j], c1 = g1[j];
#pragma unroll
        for (int q = 0; q < KP / 4; ++q) {
            float4 m = mrow[q];
            c0 = fmaf(s0[4 * q + 0], m.x, c0);
            c0 = fmaf(s0[4 * q + 1], m.y, c0);
            c0 = fmaf(s0[4 * q + 2], m.z, c0);
            c0 = fmaf(s0[4 * q + 3], m.w, c0);
            c1 = fmaf(s1[4 * q + 0], m.x, c1);
            c1 = fmaf(s1[4 * q + 1], m.y, c1);
            c1 = fmaf(s1[4 * q + 2], m.z, c1);
            c1 = fmaf(s1[4 * q + 3], m.w, c1);
        }
        g0[j] = c0;
        g1[j] = c1;
        xv0[j] *= ir0;  // q
        xv1[j] *= ir1;
        dot0 = fmaf(xv0[j], c0, dot0);
        dot1 = fmaf(xv1[j], c1, dot1);
    }
    float* pd = pn;  // reuse [8][P]
    pd[wid * P + lane] = dot0;
    pd[wid * P + lane + 32] = dot1;
    __syncthreads();
    dot0 = dot1 = 0.f;
#pragma unroll
    for (int w = 0; w < RD_WARPS; ++w) {
        dot0 += pd[w * P + lane];
        dot1 += pd[w * P + lane + 32];
    }
    // F.normalize clamps the norm at eps: below it the projection term has no gradient
    if (rnorm[lane] <= PM_NORM_EPS) dot0 = 0.f;
    if (rnorm[lane + 32] <= PM_NORM_EPS) dot1 = 0.f;
    T* dxb = dx + ((size_t)b * C + wid * CW) * hw + px0 + lane;
#pragma unroll
    for (int j = 0; j < CW; ++j) {
        if (v0) stf(dxb + (size_t)j * hw, (g0[j] - xv0[j] * dot0) * ir0);
        if (v1) stf(dxb + (size_t)j * hw + 32, (g1[j] - xv1[j] * dot1) * ir1);
    }
}

// --------------------------------------------------------------------------------------- dM (case C)
// Reduction over pixels, so here a thread owns a CHANNEL (all K accumulators in registers) and walks the
// pixels of a transposed tile in shared memory. Persistent CTAs; one vector RED per CTA at the end.

constexpr int DM_P = 32;

template <typename T, int C, int KP, bool ORD = false>
__global__ void __launch_bounds__(C) read_bwd_dM_kernel(const T* __restrict__ du, const T* __restrict__ x,
                                                         const float* __restrict__ p_in, const float* __restrict__ ds,
                                                         float* __restrict__ dM, int hw, int K, int tiles_per_img,
                                                         int ntiles) {
    constexpr int P = DM_P, LD = P + 1, NW = C / 32;
    extern __shared__ __align__(16) float smem[];
    float* xt = smem;             // [C][LD]
    float* dct = xt + C * LD;     // [C][LD]
    float* p_sm = dct + C * LD;   // [P][KP]
    float* ds_sm = p_sm + P * KP; // [P][KP]
    float* pn = ds_sm + P * KP;   // [NW][P]
    float* invr = pn + NW * P;    // [P]

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    float acc[KP];
#pragma unroll
    for (int k = 0; k < KP; ++k) acc[k] = 0.f;

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int b = tile / tiles_per_img, px0 = (tile - b * tiles_per_img) * P;
        const int nvalid = min(P, hw - px0);
        const bool v = lane < nvalid;
        const T* xb = x + (size_t)b * C * hw + px0 + lane;
        const T* dcb = du ? du + ((size_t)b * 2 * C + C) * hw + px0 + lane : nullptr;
        float n2 = 0.f;
        for (int c = wid; c < C; c += NW) {
            float xv = v ? ldf(xb + (size_t)c * hw) : 0.f;
            float dv = (v && dcb) ? ldf(dcb + (size_t)c * hw) : 0.f;
            n2 = fmaf(xv, xv, n2);
            xt[c * LD + lane] = xv;
            dct[c * LD + lane] = dv;
        }
        pn[wid * P + lane] = n2;
        const size_t n0g = (size_t)b * hw + px0;
        for (int o = tid; o < P * KP; o += C) {
            int px = o / KP, k = o - px * KP;
            bool ok = px < nvalid && k < K;
            p_sm[o] = ok ? __ldg(p_in + (n0g + px) * K + k) : 0.f;
            ds_sm[o] = ok ? __ldg(ds + (n0g + px) * KP + k) : 0.f;
        }
        __syncthreads();
        if (tid < P) {
            float s = 0.f;
            for (int w = 0; w < NW; ++w) s += pn[w * P + tid];
            invr[tid] = 1.f / fmaxf(sqrtf(s), PM_NORM_EPS);
        }
        __syncthreads();
        for (int px = 0; px < P; ++px) {
            const float q = xt[tid * LD + px] * invr[px];
            const float d = dct[tid * LD + px];
            const float4* pr = reinterpret_cast<const float4*>(p_sm + px * KP);
            const float4* sr = reinterpret_cast<const float4*>(ds_sm + px * KP);
#pragma unroll
            for (int qd = 0; qd < KP / 4; ++qd) {
                float4 pv = pr[qd], sv = sr[qd];
                acc[4 * qd + 0] = fmaf(pv.x, d, fmaf(sv.x, q, acc[4 * qd + 0]));
                acc[4 * qd + 1] = fmaf(pv.y, d, fmaf(sv.y, q, acc[4 * qd + 1]));
                acc[4 * qd + 2] = fmaf(pv.z, d, fmaf(sv.z, q, acc[4 * qd + 2]));
                acc[4 * qd + 3] = fmaf(pv.w, d, fmaf(sv.w, q, acc[4 * qd + 3]));
            }
        }
        __syncthreads();
    }
    if constexpr (ORD) {  // ordered instantiation: dM is the partial scratch, this CTA's [K][C] slot is [blockIdx.x]
        float* dst = dM + (size_t)blockIdx.x * K * C;
#pragma unroll
        for (int k = 0; k < KP; ++k)
            if (k < K) dst[(size_t)k * C + tid] = acc[k];
    } else {
#pragma unroll
        for (int k = 0; k < KP; ++k)
            if (k < K) atomicAdd(dM + (size_t)k * C + tid, acc[k]);
    }
}

// ----------------------------------------------------------------------- get_score on an NHWC query
// One warp per pixel: lanes stride the contiguous channels, K warp reductions.
template <int KP>
__global__ void __launch_bounds__(256) score_nhwc_kernel(const float* __restrict__ q, const float* __restrict__ M,
                                                         float* __restrict__ s, int N, int C, int K) {
    extern __shared__ __align__(16) float Msm[];  // [K][C]
    for (int i = threadIdx.x; i < K * C; i += blockDim.x) Msm[i] = __ldg(M + i);
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int n = blockIdx.x * nw + wid; n < N; n += gridDim.x * nw) {
        float acc[KP];
#pragma unroll
        for (int k = 0; k < KP; ++k) acc[k] = 0.f;
        for (int c = lane; c < C; c += 32) {
            float v = __ldg(q + (size_t)n * C + c);
#pragma unroll
            for (int k = 0; k < KP; ++k)
                if (k < K) acc[k] = fmaf(v, Msm[k * C + c], acc[k]);
        }
#pragma unroll
        for (int k = 0; k < KP; ++k) {
            float r = warp_sum(acc[k]);
            if (lane == 0) s[(size_t)n * KP + k] = (k < K) ? r : 0.f;
        }
    }
}

// ------------------------------------------------------------------------------------------ dispatch

template <int KP>
constexpr size_t read_smem_bytes(int C) {
    return sizeof(float) * ((size_t)C * KP + (size_t)RD_WARPS * RD_P * KP + RD_WARPS * RD_P + 2 * RD_P);
}

template <typename T, int CW, int KP>
int launch_read_fwd(const void* x, const float* M, const float* gum, void* u, float* s, float* p, int B, int hw,
                    int K, cudaStream_t st) {
    constexpr int C = CW * RD_WARPS;
    const size_t smem = read_smem_bytes<KP>(C);
    auto kern = read_fwd_kernel<T, CW, KP>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const int tiles = (hw + RD_P - 1) / RD_P;
    kern<<<B * tiles, RD_THREADS, smem, st>>>((const T*)x, M, gum, (T*)u, s, p, hw, K, tiles);
    PM_CHECK_LAUNCH();
    return 0;
}

template <typename T, int CW, int KP>
int launch_read_bwd(const void* du, const void* x, const float* M, const float* p, const float* ds_rl,
                    const float* g_loss, const float* rl_out, void* dx, float* ds, int B, int hw, int K,
                    cudaStream_t st) {
    constexpr int C = CW * RD_WARPS;
    const size_t smem = read_smem_bytes<KP>(C);
    auto kern = read_bwd_kernel<T, CW, KP>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const int tiles = (hw + RD_P - 1) / RD_P;
    kern<<<B * tiles, RD_THREADS, smem, st>>>((const T*)du, (const T*)x, M, p, ds_rl, g_loss, rl_out, (T*)dx, ds, hw,
                                               K, tiles);
    PM_CHECK_LAUNCH();
    return 0;
}

template <typename T, int C, int KP>
int launch_read_bwd_dM(const void* du, const void* x, const float* p, const float* ds, float* dM, int B, int hw,
                       int K, cudaStream_t st, float* part = nullptr, int* ncta = nullptr) {
    constexpr int LD = DM_P + 1;
    const size_t smem = sizeof(float) * ((size_t)2 * C * LD + 2 * DM_P * KP + (C / 32) * DM_P + DM_P);
    auto kern = part ? read_bwd_dM_kernel<T, C, KP, true> : read_bwd_dM_kernel<T, C, KP>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const int tiles = (hw + DM_P - 1) / DM_P, ntiles = B * tiles;
    const int grid = ntiles < 148 ? ntiles : 148;
    if (part) dM = part, *ncta = grid;
    kern<<<grid, C, smem, st>>>((const T*)du, (const T*)x, p, ds, dM, hw, K, tiles, ntiles);
    PM_CHECK_LAUNCH();
    return 0;
}

}  // namespace pm

#define PM_DISPATCH_CW(T, KP, FN, ...)                   \
    switch (C) {                                         \
        case 32: return pm::FN<T, 4, KP>(__VA_ARGS__);   \
        case 64: return pm::FN<T, 8, KP>(__VA_ARGS__);   \
        case 128: return pm::FN<T, 16, KP>(__VA_ARGS__); \
        case 256: return pm::FN<T, 32, KP>(__VA_ARGS__); \
        default: return PM_ERR_CHANNELS;                 \
    }
#define PM_DISPATCH_C(T, KP, FN, ...)                     \
    switch (C) {                                          \
        case 32: return pm::FN<T, 32, KP>(__VA_ARGS__);   \
        case 64: return pm::FN<T, 64, KP>(__VA_ARGS__);   \
        case 128: return pm::FN<T, 128, KP>(__VA_ARGS__); \
        case 256: return pm::FN<T, 256, KP>(__VA_ARGS__); \
        default: return PM_ERR_CHANNELS;                  \
    }
#define PM_DISPATCH(MACRO, FN, ...)                                            \
    do {                                                                       \
        if (dtype == PM_F32) {                                                 \
            if (K <= 19) { MACRO(float, 20, FN, __VA_ARGS__) }                 \
            else { MACRO(float, 32, FN, __VA_ARGS__) }                         \
        } else if (dtype == PM_BF16) {                                         \
            if (K <= 19) { MACRO(__nv_bfloat16, 20, FN, __VA_ARGS__) }         \
            else { MACRO(__nv_bfloat16, 32, FN, __VA_ARGS__) }                 \
        }                                                                      \
        return PM_ERR_DTYPE;                                                   \
    } while (0)

static int check_common(int B, int C, int h, int w, int K, int dtype) {
    if (dtype != PM_F32 && dtype != PM_BF16) return PM_ERR_DTYPE;
    if (C != 32 && C != 64 && C != 128 && C != 256) return PM_ERR_CHANNELS;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (B <= 0 || h <= 0 || w <= 0 || (long long)B * h * w > 0x7fffffffLL / 64) return PM_ERR_SHAPE;
    return 0;
}

static int read_fwd_generic(const void* x, const float* M, const float* gumbel_m, void* u, float* s, float* score_m,
                            int B, int C, int h, int w, int K, int dtype, void* stream) {
    PM_DISPATCH(PM_DISPATCH_CW, launch_read_fwd, x, M, gumbel_m, u, s, score_m, B, h * w, K, (cudaStream_t)stream);
}

extern "C" int pm_read_fwd(const void* x, const float* M, const float* gumbel_m, const float* gumbel_q, void* u,
                           float* s, float* score_m, float* col_partials, int B, int C, int h, int w, int K, int dtype,
                           void* stream) {
    if (!x || !M || !u || !s || !score_m) return PM_ERR_NULL;
    if (int e = check_common(B, C, h, w, K, dtype)) return e;
    if (((uintptr_t)s & 15) != 0) return PM_ERR_ALIGN;
    if (pm::tiled_ok(x, u, s, h * w, dtype))
        return pm::read_fwd_tiled(x, M, gumbel_m, gumbel_q, u, s, score_m, col_partials, B, C, h * w, K, dtype, 0,
                                  (cudaStream_t)stream);
    // generic path (any hw / alignment): un-pipelined kernel, column statistics in a separate launch
    if (int e = read_fwd_generic(x, M, gumbel_m, u, s, score_m, B, C, h, w, K, dtype, stream)) return e;
    if (col_partials) return pm::colsoftmax_stats(s, gumbel_q, col_partials, B * h * w, K, (cudaStream_t)stream);
    return 0;
}

extern "C" int pm_read_bwd(const void* du, const void* x, const float* M, const float* score_m, const float* ds_rl,
                           const float* g_loss, const float* rl_out, void* dx, float* ds, int B, int C, int h, int w,
                           int K, int dtype, void* stream) {
    if (!du || !x || !M || !score_m || !dx) return PM_ERR_NULL;
    if (int e = check_common(B, C, h, w, K, dtype)) return e;
    if (((uintptr_t)ds & 15) != 0 || ((uintptr_t)ds_rl & 15) != 0) return PM_ERR_ALIGN;
    if (ds != nullptr && pm::tiled_ok(du, x, dx, h * w, dtype))
        return pm::read_bwd_tiled(du, x, M, score_m, ds_rl, g_loss, rl_out, dx, nullptr, ds, B, C, h * w, K, dtype, 0,
                                  (cudaStream_t)stream);
    PM_DISPATCH(PM_DISPATCH_CW, launch_read_bwd, du, x, M, score_m, ds_rl, g_loss, rl_out, dx, ds, B, h * w, K,
                (cudaStream_t)stream);
}

extern "C" int pm_read_planes(void) { return PM_PLANES; }

extern "C" int pm_read_fwd_planes(const void* x, const float* M, const float* gumbel_m, const float* gumbel_q, void* u,
                                  float* s, float* score_m, float* col_partials, int B, int C, int h, int w, int K,
                                  int dtype, void* stream) {
    if (!x || !M || !u || !s || !score_m) return PM_ERR_NULL;
    if (int e = check_common(B, C, h, w, K, dtype)) return e;
    if (((uintptr_t)s & 15) != 0 || !pm::tiled_ok(x, u, s, h * w, dtype)) return PM_ERR_ALIGN;
    return pm::read_fwd_tiled(x, M, gumbel_m, gumbel_q, u, s, score_m, col_partials, B, C, h * w, K, dtype, 1,
                              (cudaStream_t)stream);
}

extern "C" int pm_read_bwd_planes(const void* du, const void* x, const float* M, const float* score_m,
                                  const float* ds_rl, const float* g_loss, const float* rl_out, void* dx,
                                  const void* dx_add, float* ds, int B, int C, int h, int w, int K, int dtype,
                                  void* stream) {
    if (!du || !x || !M || !score_m || !dx || !ds) return PM_ERR_NULL;
    if (int e = check_common(B, C, h, w, K, dtype)) return e;
    if (((uintptr_t)ds & 15) != 0 || ((uintptr_t)ds_rl & 15) != 0 || !pm::tiled_ok(du, x, dx, h * w, dtype))
        return PM_ERR_ALIGN;
    return pm::read_bwd_tiled(du, x, M, score_m, ds_rl, g_loss, rl_out, dx, dx_add, ds, B, C, h * w, K, dtype, 1,
                              (cudaStream_t)stream);
}

extern "C" int pm_read_bwd_dM(const void* du, const void* x, const float* score_m, const float* ds, float* dM, int B,
                              int C, int h, int w, int K, int dtype, void* stream) {
    if (!x || !score_m || !ds || !dM) return PM_ERR_NULL;  // du NULL: only the ds (x) q term (planes mode)
    if (int e = check_common(B, C, h, w, K, dtype)) return e;
    PM_DISPATCH(PM_DISPATCH_C, launch_read_bwd_dM, du, x, score_m, ds, dM, B, h * w, K, (cudaStream_t)stream);
}

extern "C" int pm_read_bwd_dM_scratch_bytes(int B, int C, int h, int w, int K) {
    if (C != 32 && C != 64 && C != 128 && C != 256) return PM_ERR_CHANNELS;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (B <= 0 || h <= 0 || w <= 0 || (long long)B * h * w > 0x7fffffffLL / 64) return PM_ERR_SHAPE;
    const long long ntiles = (long long)B * ((h * w + pm::DM_P - 1) / pm::DM_P);
    return (int)((ntiles < 148 ? ntiles : 148) * K * C * (long long)sizeof(float));
}

extern "C" int pm_read_bwd_dM_ordered(const void* du, const void* x, const float* score_m, const float* ds, float* dM,
                                      float* scratch, int B, int C, int h, int w, int K, int dtype, void* stream) {
    if (!x || !score_m || !ds || !dM || !scratch) return PM_ERR_NULL;
    if (int e = check_common(B, C, h, w, K, dtype)) return e;
    if ((uintptr_t)scratch & 15) return PM_ERR_ALIGN;
    int ncta = 0;
    // every CTA stores its [K][C] partial to `scratch`, then one fixed-order reduction adds them into dM
    const int rc = [&]() -> int {
        PM_DISPATCH(PM_DISPATCH_C, launch_read_bwd_dM, du, x, score_m, ds, dM, B, h * w, K, (cudaStream_t)stream, scratch,
                    &ncta);
    }();
    if (rc) return rc;
    return pm::reduce_partials_f32(dM, scratch, ncta, (long long)K * C, (cudaStream_t)stream);
}

extern "C" int pm_score_nhwc(const float* q, const float* M, float* s, int N, int C, int K, void* stream) {
    if (!q || !M || !s) return PM_ERR_NULL;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (N <= 0 || C <= 0 || C > 2048) return PM_ERR_SHAPE;
    const size_t smem = sizeof(float) * (size_t)K * C;
    int grid = (N + 7) / 8;
    if (grid > 148 * 8) grid = 148 * 8;
    cudaError_t e;
    if (K <= 19) {
        e = cudaFuncSetAttribute(pm::score_nhwc_kernel<20>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        pm::score_nhwc_kernel<20><<<grid, 256, smem, (cudaStream_t)stream>>>(q, M, s, N, C, K);
    } else {
        e = cudaFuncSetAttribute(pm::score_nhwc_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        pm::score_nhwc_kernel<32><<<grid, 256, smem, (cudaStream_t)stream>>>(q, M, s, N, C, K);
    }
    PM_CHECK_LAUNCH();
    return 0;
}
