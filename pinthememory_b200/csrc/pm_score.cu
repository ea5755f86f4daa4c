// Score-side kernels: the dim-0 (over all pixels) softmax and the feature-cohesion read loss.
#include "pm_common.cuh"
#include "pm_internal.h"

namespace pm {

// ------------------------------------------------------------------ score_query: softmax over pixels
// memory.py:183/186. Two small launches: per-CTA online (max, sum) per column, then normalise.
// Threads per CTA = K * floor(256/K) so a thread's column is fixed while its flat index strides rows.

constexpr int CS_MAXG = PM_COLPART_ROWS;

__global__ void __launch_bounds__(256) colsoftmax_stats_kernel(const float* __restrict__ s, const float* __restrict__ g,
                                                               float* __restrict__ partial, int N, int K, int KP,
                                                               int rows_per_cta) {
    __shared__ float sm_m[256], sm_l[256];
    const int t = threadIdx.x, k = t % K, r0 = t / K, rstep = blockDim.x / K;
    const int start = blockIdx.x * rows_per_cta, end = min(N, start + rows_per_cta);
    float m = -INFINITY, l = 0.f;
    for (int r = start + r0; r < end; r += rstep) {
        float z = __ldg(s + (size_t)r * KP + k);
        if (g != nullptr) z += __ldg(g + (size_t)r * K + k);
        if (z > m) {
            l = l * expf(m - z) + 1.f;
            m = z;
        } else {
            l += expf(z - m);
        }
    }
    sm_m[t] = m;
    sm_l[t] = l;
    __syncthreads();
    if (t < K) {
        float M = -INFINITY;
        for (int i = 0; i < rstep; ++i) M = fmaxf(M, sm_m[i * K + t]);
        float L = 0.f;
        for (int i = 0; i < rstep; ++i) {
            float mi = sm_m[i * K + t];
            if (mi > -INFINITY) L += sm_l[i * K + t] * expf(mi - M);
        }
        partial[(size_t)blockIdx.x * 64 + t] = M;
        partial[(size_t)blockIdx.x * 64 + 32 + t] = L;
    }
}

// Combine the PM_COLPART_ROWS per-CTA (max, sum) partials of every column ONCE (one CTA) into the final column maximum and
// 1/sum, stored in row PM_COLPART_ROWS of the partials buffer ([0..32) max, [32..64) 1/sum). The apply kernel that follows
// then runs on as many small CTAs as there are rows to normalise (the round-1 version re-combined the 296 x 64 partials
// in every one of its <= 296 CTAs: 75 KB of L2 reads and a dependent latency chain per CTA, 18 us for 11 MB of work).
__global__ void __launch_bounds__(256) colsoftmax_combine_kernel(float* __restrict__ partial, int K) {  // all PM_COLPART_ROWS rows
    __shared__ float sm_m[256], sm_l[256];
    const int t = threadIdx.x, k = t % K, r0 = t / K, rstep = blockDim.x / K;
    constexpr int MAXJ = (CS_MAXG + 7) / 8;  // rstep >= 8 for K <= 31
    float pm_[MAXJ], pl_[MAXJ];
#pragma unroll
    for (int j = 0; j < MAXJ; ++j) {  // all loads issued before the first use (independent L2 hits)
        const int i = r0 + j * rstep;
        const bool ok = i < CS_MAXG;
        pm_[j] = ok ? __ldcg(partial + (size_t)i * 64 + k) : -INFINITY;
        pl_[j] = ok ? __ldcg(partial + (size_t)i * 64 + 32 + k) : 0.f;
    }
    float M = -INFINITY, L = 0.f;
#pragma unroll
    for (int j = 0; j < MAXJ; ++j) M = fmaxf(M, pm_[j]);
#pragma unroll
    for (int j = 0; j < MAXJ; ++j)
        if (pm_[j] > -INFINITY) L += pl_[j] * expf(pm_[j] - M);
    sm_m[t] = M;
    sm_l[t] = L;
    __syncthreads();
    if (t < K) {
        float Mx = -INFINITY;
        for (int i = 0; i < rstep; ++i) Mx = fmaxf(Mx, sm_m[i * K + t]);
        float Ls = 0.f;
        for (int i = 0; i < rstep; ++i) {
            const float mi = sm_m[i * K + t];
            if (mi > -INFINITY) Ls += sm_l[i * K + t] * expf(mi - Mx);
        }
        partial[(size_t)CS_MAXG * 64 + t] = Mx;
        partial[(size_t)CS_MAXG * 64 + 32 + t] = 1.f / Ls;
    }
}

__global__ void __launch_bounds__(256) colsoftmax_apply_kernel(const float* __restrict__ s, const float* __restrict__ g,
                                                               const float* __restrict__ partial,
                                                               float* __restrict__ out, int N, int K, int KP,
                                                               int rows_per_cta) {
    const int t = threadIdx.x, k = t % K, r0 = t / K, rstep = blockDim.x / K;
    const float M = __ldg(partial + (size_t)CS_MAXG * 64 + k), il = __ldg(partial + (size_t)CS_MAXG * 64 + 32 + k);
    const int start = blockIdx.x * rows_per_cta, end = min(N, start + rows_per_cta);
    for (int r = start + r0; r < end; r += rstep) {
        float z = __ldg(s + (size_t)r * KP + k);
        if (g != nullptr) z += __ldg(g + (size_t)r * K + k);
        out[(size_t)r * K + k] = expf(z - M) * il;
    }
}

// -------------------------------------------------------- score_memory for the external get_score path
// Row softmax of s (+ gumbel_m) -> dense [N,K]. (Inside Memory_sup.forward this is fused in read_fwd.)
template <int KP>
__global__ void __launch_bounds__(256) rowsoftmax_kernel(const float* __restrict__ s, const float* __restrict__ g,
                                                         float* __restrict__ out, int N, int K) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    float z[KP], mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < KP; ++k) {
        z[k] = (k < K) ? __ldg(s + (size_t)n * KP + k) + (g ? __ldg(g + (size_t)n * K + k) : 0.f) : -INFINITY;
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
        if (k < K) out[(size_t)n * K + k] = z[k] * inv;
}

}  // namespace pm

extern "C" int pm_score_stride(int K) { return K <= 19 ? 20 : 32; }
extern "C" int pm_colsoftmax_workspace_floats(int K) { return (pm::CS_MAXG + 2) * 64; }  // + the combined row + the ticket row

namespace pm {
int colsoftmax_stats(const float* s, const float* gumbel_q, float* partial, int N, int K, cudaStream_t st) {
    const int KP = pm_score_stride(K), tpb = K * (256 / K);
    const int rows_per_cta = (N + CS_MAXG - 1) / CS_MAXG;  // CTAs past the end write (-inf, 0)
    colsoftmax_stats_kernel<<<CS_MAXG, tpb, 0, st>>>(s, gumbel_q, partial, N, K, KP, rows_per_cta);
    colsoftmax_combine_kernel<<<1, tpb, 0, st>>>(partial, K);  // -> row PM_COLPART_ROWS: column maximum, 1/sum
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}
}  // namespace pm

extern "C" int pm_colsoftmax_apply(const float* s, const float* gumbel_q, const float* col_partials, float* score_q,
                                   int N, int K, void* stream) {
    if (!s || !score_q || !col_partials) return PM_ERR_NULL;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (N <= 0) return PM_ERR_SHAPE;
    const int KP = pm_score_stride(K), tpb = K * (256 / K), rstep = tpb / K;
    // the combined row (column maximum, 1/sum) was left by pm_read_fwd[_planes] / the statistics pass
    const int rows_per_cta = rstep * 5;   // 5 rows per thread: ~1100 small CTAs at cfg 2
    const int G = (N + rows_per_cta - 1) / rows_per_cta;
    pm::colsoftmax_apply_kernel<<<G, tpb, 0, (cudaStream_t)stream>>>(s, gumbel_q, col_partials, score_q, N, K, KP,
                                                                       rows_per_cta);
    PM_CHECK_LAUNCH();
    return 0;
}

extern "C" int pm_colsoftmax(const float* s, const float* gumbel_q, float* score_q, float* workspace, int N, int K,
                             void* stream) {
    if (!s || !score_q || !workspace) return PM_ERR_NULL;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (N <= 0) return PM_ERR_SHAPE;
    if (int e = pm::colsoftmax_stats(s, gumbel_q, workspace, N, K, (cudaStream_t)stream)) return e;
    return pm_colsoftmax_apply(s, gumbel_q, workspace, score_q, N, K, stream);
}

extern "C" int pm_rowsoftmax(const float* s, const float* gumbel_m, float* score_m, int N, int K, void* stream) {
    if (!s || !score_m) return PM_ERR_NULL;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (N <= 0) return PM_ERR_SHAPE;
    const int grid = (N + 255) / 256;
    if (K <= 19)
        pm::rowsoftmax_kernel<20><<<grid, 256, 0, (cudaStream_t)stream>>>(s, gumbel_m, score_m, N, K);
    else
        pm::rowsoftmax_kernel<32><<<grid, 256, 0, (cudaStream_t)stream>>>(s, gumbel_m, score_m, N, K);
    PM_CHECK_LAUNCH();
    return 0;
}

// ------------------------------------------------------------------ backward of the two softmaxes
// E[n,k] = p_m (g_m - sum_j p_m g_m)[n,k] + p_q[n,k] (g_q[n,k] - c[k]) + scale * ds_rl[n,k],  c[k] = sum_n p_q g_q [n,k].
// The column sums c are a reduction over every pixel, formed in a fixed order in fp64: SB_PARTS CTAs each sum a fixed
// pixel range (thread partials, then the CTA's threads in index order) and store one double per column; every CTA of the
// element-wise pass adds the SB_PARTS partials in CTA order itself (<= 37 KB of L2 reads per CTA), so the result does not
// depend on scheduling and the two passes need no arrival counter or zeroed state.

namespace pm {

// (SB_PARTS, SB_GROUPS and the summation order: pm_common.cuh, sb_group_sum)

__global__ void __launch_bounds__(256) score_bwd_colsum_kernel(const float* __restrict__ p, const float* __restrict__ g,
                                                               double* __restrict__ part, int N, int K, int rows_per_cta) {
    __shared__ double red[256];
    const int t = threadIdx.x, k = t % K, r0 = t / K, rstep = blockDim.x / K;
    const int start = blockIdx.x * rows_per_cta, end = min(N, start + rows_per_cta);
    double acc = 0.0;
    // thread t reads flat elements start*K + t + i*rstep*K: the CTA's accesses are contiguous
    for (int r = start + r0; r < end; r += rstep)
        acc += (double)__ldg(p + (size_t)r * K + k) * (double)__ldg(g + (size_t)r * K + k);
    red[t] = acc;
    __syncthreads();
    if (t < K) {
        double c = 0.0;
        for (int i = 0; i < rstep; ++i) c += red[i * K + t];
        part[(size_t)blockIdx.x * 32 + t] = c;
    }
}

// GLOBAL: `part` is the double[32] of global column sums pm_read_exchange_bwd left (the global read of a sharded run)
template <int KP, bool GLOBAL = false>
__global__ void __launch_bounds__(256)
    score_bwd_apply_kernel(const float* __restrict__ score_q, const float* __restrict__ g_q, const float* __restrict__ score_m,
                           const float* __restrict__ g_m, const float* __restrict__ ds_rl, const float* __restrict__ g_loss,
                           const float* __restrict__ rl_out, const double* __restrict__ part, float* __restrict__ E, int N,
                           int K) {
    __shared__ double red[SB_GROUPS][32];
    __shared__ float cq[32];
    const int t = threadIdx.x;
    if (GLOBAL && g_q != nullptr) {
        if (t < 32) cq[t] = t < K ? (float)__ldcg(part + t) : 0.f;
        __syncthreads();
    } else if (g_q != nullptr) {
        // c[k]: SB_GROUPS groups of 32 threads, one group term each (sb_group_sum), then the groups in ascending order
        static_assert(SB_GROUPS * 32 == 256, "one group of 32 threads per group term");
        const int k = t & 31, j = t >> 5;
        red[j][k] = k < K ? sb_group_sum(part, k, j) : 0.0;
        __syncthreads();
        if (t < 32) {
            double c = 0.0;
#pragma unroll
            for (int i = 0; i < SB_GROUPS; ++i) c += red[i][t];
            cq[t] = (float)c;
        }
        __syncthreads();
    }
    float scale = 0.f;
    if (ds_rl != nullptr && g_loss != nullptr && rl_out != nullptr) scale = __ldg(g_loss) * __ldg(rl_out + 1);
    for (long long n = (long long)blockIdx.x * 256 + t; n < N; n += (long long)gridDim.x * 256) {
        float e[KP];
#pragma unroll
        for (int k = 0; k < KP; ++k) e[k] = 0.f;
        if (g_m != nullptr) {
            float pm_[KP], dot = 0.f;
#pragma unroll
            for (int k = 0; k < KP; ++k) {
                pm_[k] = (k < K) ? __ldg(score_m + (size_t)n * K + k) : 0.f;
                e[k] = (k < K) ? __ldg(g_m + (size_t)n * K + k) : 0.f;
                dot = fmaf(pm_[k], e[k], dot);
            }
#pragma unroll
            for (int k = 0; k < KP; ++k) e[k] = pm_[k] * (e[k] - dot);
        }
        if (g_q != nullptr) {
#pragma unroll
            for (int k = 0; k < KP; ++k)
                if (k < K) e[k] = fmaf(__ldg(score_q + (size_t)n * K + k), __ldg(g_q + (size_t)n * K + k) - cq[k], e[k]);
        }
        if (scale != 0.f) {
            const float4* rl = reinterpret_cast<const float4*>(ds_rl + (size_t)n * KP);
#pragma unroll
            for (int q = 0; q < KP / 4; ++q) {
                const float4 r = __ldg(rl + q);
                e[4 * q + 0] = fmaf(scale, r.x, e[4 * q + 0]);
                e[4 * q + 1] = fmaf(scale, r.y, e[4 * q + 1]);
                e[4 * q + 2] = fmaf(scale, r.z, e[4 * q + 2]);
                e[4 * q + 3] = fmaf(scale, r.w, e[4 * q + 3]);
            }
        }
        float4* out = reinterpret_cast<float4*>(E + (size_t)n * KP);
#pragma unroll
        for (int q = 0; q < KP / 4; ++q)
            out[q] = make_float4(4 * q + 0 < K ? e[4 * q + 0] : 0.f, 4 * q + 1 < K ? e[4 * q + 1] : 0.f,
                                 4 * q + 2 < K ? e[4 * q + 2] : 0.f, 4 * q + 3 < K ? e[4 * q + 3] : 0.f);
    }
}

// ------------------------------------------------------------------ backward of get_score's s = q.M^T
// dq[n,c] = sum_k E[n,k] M[k,c];  dM[k,c] = sum_n E[n,k] q[n,c]. One thread per channel (M's column in registers), a CTA
// walks a fixed pixel range in 32-pixel tiles of E staged in shared memory; its dM partial goes to scratch and
// reduce_partials_f32 adds the partials in CTA order.

constexpr int SNB_TILE = 32, SNB_CTAS = 296;

static int snb_grid(int N) { return min(SNB_CTAS, (N + SNB_TILE - 1) / SNB_TILE); }

template <int KP>
__global__ void __launch_bounds__(256)
    score_nhwc_bwd_kernel(const float* __restrict__ q, const float* __restrict__ M, const float* __restrict__ E,
                          float* __restrict__ dq, float* __restrict__ part, int N, int C, int K, int rows_per_cta) {
    __shared__ __align__(16) float Es[SNB_TILE * KP];
    const int start = blockIdx.x * rows_per_cta, end = min(N, start + rows_per_cta);
    for (int c0 = 0; c0 < C; c0 += blockDim.x) {
        const int c = c0 + threadIdx.x;
        const bool cv = c < C;
        float m[KP], acc[KP];
#pragma unroll
        for (int k = 0; k < KP; ++k) {
            m[k] = (dq && cv && k < K) ? __ldg(M + (size_t)k * C + c) : 0.f;
            acc[k] = 0.f;
        }
        for (int n0 = start; n0 < end; n0 += SNB_TILE) {
            const int np = min(SNB_TILE, end - n0);
            __syncthreads();
            for (int i = threadIdx.x; i < np * (KP / 4); i += blockDim.x)
                reinterpret_cast<float4*>(Es)[i] = __ldg(reinterpret_cast<const float4*>(E + (size_t)n0 * KP) + i);
            __syncthreads();
            if (!cv) continue;
            for (int i = 0; i < np; ++i) {
                const size_t n = (size_t)(n0 + i);
                const float qv = part ? __ldg(q + n * C + c) : 0.f;
                float d = 0.f;
#pragma unroll
                for (int k = 0; k < KP; ++k) {
                    const float e = Es[i * KP + k];
                    d = fmaf(e, m[k], d);
                    acc[k] = fmaf(e, qv, acc[k]);
                }
                if (dq) dq[n * C + c] = d;
            }
        }
        if (part && cv) {
#pragma unroll
            for (int k = 0; k < KP; ++k)
                if (k < K) part[((size_t)blockIdx.x * K + k) * C + c] = acc[k];
        }
    }
}

}  // namespace pm

extern "C" int pm_score_bwd_workspace_floats(int K) { return pm::SB_PARTS * 32 * 2; }  // SB_PARTS x 32 doubles

extern "C" int pm_score_bwd(const float* score_q, const float* g_q, const float* score_m, const float* g_m,
                            const float* ds_rl, const float* g_loss, const float* rl_out, float* E, float* workspace, int N,
                            int K, void* stream) {
    if (!E || (g_q && (!score_q || !workspace)) || (g_m && !score_m)) return PM_ERR_NULL;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (N <= 0) return PM_ERR_SHAPE;
    if (((uintptr_t)E & 15) || ((uintptr_t)ds_rl & 15) || ((uintptr_t)workspace & 7)) return PM_ERR_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    double* part = reinterpret_cast<double*>(workspace);
    if (g_q) {
        const int rows_per_cta = (N + pm::SB_PARTS - 1) / pm::SB_PARTS;  // CTAs past the end store 0
        pm::score_bwd_colsum_kernel<<<pm::SB_PARTS, K * (256 / K), 0, st>>>(score_q, g_q, part, N, K, rows_per_cta);
        PM_CHECK_LAUNCH();
    }
    const int grid = min((N + 255) / 256, 148 * 4);
    if (K <= 19)
        pm::score_bwd_apply_kernel<20><<<grid, 256, 0, st>>>(score_q, g_q, score_m, g_m, ds_rl, g_loss, rl_out, part, E, N, K);
    else
        pm::score_bwd_apply_kernel<32><<<grid, 256, 0, st>>>(score_q, g_q, score_m, g_m, ds_rl, g_loss, rl_out, part, E, N, K);
    PM_CHECK_LAUNCH();
    return 0;
}

extern "C" int pm_score_nhwc_bwd_scratch_bytes(int N, int C, int K) {
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (N <= 0 || C <= 0 || C > 2048) return PM_ERR_SHAPE;
    const long long b = (long long)pm::snb_grid(N) * K * C * (long long)sizeof(float);
    return b > 0x7fffffffLL ? PM_ERR_SHAPE : (int)b;
}

extern "C" int pm_score_nhwc_bwd(const float* q, const float* M, const float* E, float* dq, float* dM, float* scratch, int N,
                                 int C, int K, void* stream) {
    if (!E || (dq && !M) || (dM && (!q || !scratch))) return PM_ERR_NULL;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (N <= 0 || C <= 0 || C > 2048) return PM_ERR_SHAPE;
    if ((uintptr_t)E & 15) return PM_ERR_ALIGN;
    if (!dq && !dM) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int G = pm::snb_grid(N), rows_per_cta = (N + G - 1) / G;
    const int tpb = min(256, (C + 31) / 32 * 32);
    float* part = dM ? scratch : nullptr;
    if (K <= 19)
        pm::score_nhwc_bwd_kernel<20><<<G, tpb, 0, st>>>(q, M, E, dq, part, N, C, K, rows_per_cta);
    else
        pm::score_nhwc_bwd_kernel<32><<<G, tpb, 0, st>>>(q, M, E, dq, part, N, C, K, rows_per_cta);
    PM_CHECK_LAUNCH();
    if (dM) return pm::reduce_partials_f32(dM, scratch, G, (long long)K * C, st);
    return 0;
}

extern "C" int pm_score_bwd_partials(const float* score_q, const float* g_q, float* workspace, int N, int K, void* stream) {
    if (!score_q || !g_q || !workspace) return PM_ERR_NULL;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (N <= 0) return PM_ERR_SHAPE;
    if ((uintptr_t)workspace & 7) return PM_ERR_ALIGN;
    const int rows_per_cta = (N + pm::SB_PARTS - 1) / pm::SB_PARTS;
    pm::score_bwd_colsum_kernel<<<pm::SB_PARTS, K * (256 / K), 0, (cudaStream_t)stream>>>(
        score_q, g_q, reinterpret_cast<double*>(workspace), N, K, rows_per_cta);
    PM_CHECK_LAUNCH();
    return 0;
}

extern "C" int pm_score_bwd_global(const float* score_q, const float* g_q, const float* score_m, const float* g_m,
                                   const float* ds_rl, const float* g_loss, const float* rl_out, const double* colsums, float* E,
                                   int N, int K, void* stream) {
    if (!E || (g_q && (!score_q || !colsums)) || (g_m && !score_m)) return PM_ERR_NULL;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (N <= 0) return PM_ERR_SHAPE;
    if (((uintptr_t)E & 15) || ((uintptr_t)ds_rl & 15) || ((uintptr_t)colsums & 7)) return PM_ERR_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = min((N + 255) / 256, 148 * 4);
    if (K <= 19)
        pm::score_bwd_apply_kernel<20, true><<<grid, 256, 0, st>>>(score_q, g_q, score_m, g_m, ds_rl, g_loss, rl_out, colsums, E,
                                                                   N, K);
    else
        pm::score_bwd_apply_kernel<32, true><<<grid, 256, 0, st>>>(score_q, g_q, score_m, g_m, ds_rl, g_loss, rl_out, colsums, E,
                                                                   N, K);
    PM_CHECK_LAUNCH();
    return 0;
}
