// BatchNorm (+ residual, + ReLU) of the module's two 1x1-conv blocks, NCHW, training and eval mode.
//
// Reference: `self.output = Sequential(Conv2d 1x1, BatchNorm2d, ReLU)` (memory.py:103-107) and
// `Writingnet: relu(x + BatchNorm2d(Conv2d 1x1(x)))` (memory.py:74-87). The 1x1 convolutions stay library
// GEMMs; everything after them -- batch statistics, running-stat update, normalise + affine (+ residual)
// + ReLU, and the whole backward through those -- is done here in four streaming passes instead of
// cuDNN's BN kernels plus separate add / ReLU / threshold-backward element-wise kernels:
//   bn_stats      : per channel sum, sum of squares  -> mean, 1/sqrt(var+eps), running stats   (reads x)
//   bn_apply      : y = relu((x-mean)*invstd*gamma + beta + residual)                          (reads x[,res], writes y)
//   bn_bwd_reduce : g = dy*(y>0); dbeta = sum g, dgamma = sum g*xhat                           (reads dy,y,x)
//   bn_bwd_apply  : dx = gamma*invstd*(g - mean(g) - xhat*mean(g*xhat)); dres = g              (reads dy,y,x, writes dx[,dres])
// A channel's data is B contiguous rows of hw elements; rows are read with 16-byte vectors when hw allows.
#include "pm_common.cuh"

namespace pm {

constexpr int BN_THREADS = 512;

template <typename T>
struct Vec4;
template <>
struct Vec4<float> {
    float4 v;
    __device__ __forceinline__ void load(const float* p) { v = *reinterpret_cast<const float4*>(p); }
    __device__ __forceinline__ void store(float* p) const { *reinterpret_cast<float4*>(p) = v; }
    __device__ __forceinline__ float get(int i) const { return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w; }
    __device__ __forceinline__ void set(int i, float f) {
        if (i == 0) v.x = f;
        else if (i == 1) v.y = f;
        else if (i == 2) v.z = f;
        else v.w = f;
    }
};
template <>
struct Vec4<__nv_bfloat16> {
    uint2 v;
    __device__ __forceinline__ void load(const __nv_bfloat16* p) { v = *reinterpret_cast<const uint2*>(p); }
    __device__ __forceinline__ void store(__nv_bfloat16* p) const { *reinterpret_cast<uint2*>(p) = v; }
    __device__ __forceinline__ float get(int i) const {
        const unsigned w = i < 2 ? v.x : v.y;
        return __uint_as_float((i & 1) ? (w & 0xffff0000u) : (w << 16));
    }
    __device__ __forceinline__ void set(int i, float f) {
        const unsigned b = (unsigned)__bfloat16_as_ushort(__float2bfloat16_rn(f));
        unsigned& w = i < 2 ? v.x : v.y;
        w = (i & 1) ? ((w & 0x0000ffffu) | (b << 16)) : ((w & 0xffff0000u) | b);
    }
};

// 16-byte bf16 vector (8 elements): the width at which the bf16 passes move as many bytes per load as the fp32 ones
struct Vec8bf {
    uint4 v;
    __device__ __forceinline__ void load(const __nv_bfloat16* p) { v = *reinterpret_cast<const uint4*>(p); }
    __device__ __forceinline__ void store(__nv_bfloat16* p) const { *reinterpret_cast<uint4*>(p) = v; }
    __device__ __forceinline__ float get(int i) const {
        const unsigned w = (i >> 1) == 0 ? v.x : (i >> 1) == 1 ? v.y : (i >> 1) == 2 ? v.z : v.w;
        return __uint_as_float((i & 1) ? (w & 0xffff0000u) : (w << 16));
    }
    __device__ __forceinline__ void set(int i, float f) {
        const unsigned b = (unsigned)__bfloat16_as_ushort(__float2bfloat16_rn(f));
        unsigned& w = (i >> 1) == 0 ? v.x : (i >> 1) == 1 ? v.y : (i >> 1) == 2 ? v.z : v.w;
        w = (i & 1) ? ((w & 0x0000ffffu) | (b << 16)) : ((w & 0xffff0000u) | b);
    }
};
// VN = elements per thread and load: 4 (float4 / 8-byte bf16) or 8 (16-byte bf16); 0 = scalar path
template <typename T, int VN>
struct VecSel {
    typedef Vec4<T> type;
};
template <>
struct VecSel<__nv_bfloat16, 8> {
    typedef Vec8bf type;
};
// bits of the VN elements of vector j of a row out of the packed mask (1 bit per element, 32 per word)
template <int VN>
__device__ __forceinline__ unsigned mask_bits(const unsigned* __restrict__ words, int j) {
    constexpr int LPW = 32 / VN;  // vectors per word
    return (__ldg(words + j / LPW) >> (VN * (j % LPW))) & ((1u << VN) - 1u);
}

__device__ __forceinline__ double block_sum_double(double v, double* red) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if (lane == 0) red[wid] = v;
    __syncthreads();
    double t = 0.0;
    for (int i = 0; i < BN_THREADS / 32; ++i) t += red[i];
    return t;
}

// one CTA per channel
template <typename T, int VN>
__global__ void __launch_bounds__(BN_THREADS) bn_stats_kernel(const T* __restrict__ x, int B, int C, int hw, float eps,
                                                              float* __restrict__ mean, float* __restrict__ invstd,
                                                              float* __restrict__ running_mean,
                                                              float* __restrict__ running_var, float momentum) {
    __shared__ double red[BN_THREADS / 32];
    const int c = blockIdx.x;
    float s = 0.f, q = 0.f;
    if constexpr (VN != 0) {
        const int nv = hw / VN, total = B * nv;
#pragma unroll 4
        for (int i = threadIdx.x; i < total; i += BN_THREADS) {
            const int b = i / nv, j = i - b * nv;
            typename VecSel<T, VN>::type v;
            v.load(x + ((size_t)b * C + c) * hw + VN * j);
#pragma unroll
            for (int e = 0; e < VN; ++e) {
                const float f = v.get(e);
                s += f;
                q = fmaf(f, f, q);
            }
        }
    } else {
        const int total = B * hw;
        for (int i = threadIdx.x; i < total; i += BN_THREADS) {
            const int b = i / hw, j = i - b * hw;
            const float f = ldf(x + ((size_t)b * C + c) * hw + j);
            s += f;
            q = fmaf(f, f, q);
        }
    }
    const double S = block_sum_double((double)s, red);
    const double Q = block_sum_double((double)q, red);
    if (threadIdx.x == 0) {
        const double n = (double)B * (double)hw;
        const double m = S / n;
        double var = Q / n - m * m;
        if (var < 0.0) var = 0.0;
        mean[c] = (float)m;
        invstd[c] = (float)(1.0 / sqrt(var + (double)eps));
        if (running_mean != nullptr) {  // PyTorch: running_var takes the unbiased estimate
            const double unb = n > 1.0 ? var * n / (n - 1.0) : var;
            running_mean[c] = (float)((1.0 - momentum) * running_mean[c] + momentum * m);
            running_var[c] = (float)((1.0 - momentum) * running_var[c] + momentum * unb);
        }
    }
}

// one CTA per (b, c) row (BnFinalize: pm_common.cuh)
template <typename T, int VN>
__global__ void __launch_bounds__(256) bn_apply_kernel(const T* __restrict__ x, const float* __restrict__ mean,
                                                       const float* __restrict__ invstd, const float* __restrict__ gamma,
                                                       const float* __restrict__ beta, const T* __restrict__ residual,
                                                       T* __restrict__ y, unsigned* __restrict__ relu_mask, int relu,
                                                       int C, int hw, BnFinalize fin) {
    const int row = blockIdx.x, c = row % C;
    float mu, is;
    if (fin.stats != nullptr) {
        // batch statistics straight from the convolution epilogue's fp64 (sum, sum of squares): every CTA finalises its
        // own channel (two loads, a division and a square root) instead of waiting for a finalise launch; the CTAs of
        // image 0 publish mean / invstd for the backward and update the running statistics
        bn_finalize_channel(fin, c, C, row < C && threadIdx.x == 0, mu, is);
        if (row == 0 && threadIdx.x == 0 && fin.num_batches_tracked != nullptr) *fin.num_batches_tracked += 1;
    } else {
        mu = mean[c], is = invstd[c];
    }
    float sc, sh;
    bn_scale_shift(mu, is, gamma[c], beta[c], sc, sh);
    const size_t base = (size_t)row * hw;
    if constexpr (VN != 0) {
        // relu_mask (optional): 1 bit per element, bit = output > 0, 32 elements per word, rows padded to whole
        // words: the backward reads it instead of y (1/32 of the bytes). The loop is warp-uniform so that the
        // 32 / VN lanes that share a word can OR their bit groups with one REDUX.
        constexpr int LPW = 32 / VN;
        const int nv = hw / VN, wpr = (nv + LPW - 1) / LPW, lane = threadIdx.x & 31;
        const unsigned gmask = ((LPW == 32) ? 0xffffffffu : ((1u << LPW) - 1u)) << (lane & ~(LPW - 1));
        for (int j0 = 0; j0 < nv; j0 += 256) {
            const int j = j0 + threadIdx.x;
            unsigned nib = 0u;
            if (j < nv) {
                typename VecSel<T, VN>::type v, r, o;
                v.load(x + base + VN * j);
                if (residual) r.load(residual + base + VN * j);
#pragma unroll
                for (int e = 0; e < VN; ++e) {
                    float f = bn_affine(v.get(e), sc, sh);
                    if (residual) f += r.get(e);  // with relu: bn_res_relu, the writing net's fused kernels' expression
                    nib |= (f > 0.f ? 1u : 0u) << e;
                    o.set(e, relu ? fmaxf(f, 0.f) : f);
                }
                o.store(y + base + VN * j);
            }
            if (relu_mask != nullptr) {
                const unsigned word = __reduce_or_sync(gmask, nib << (VN * (lane & (LPW - 1))));
                if ((lane & (LPW - 1)) == 0 && j < nv) relu_mask[(size_t)row * wpr + j / LPW] = word;
            }
        }
    } else {
        for (int j = threadIdx.x; j < hw; j += 256) {
            float f = bn_affine(ldf(x + base + j), sc, sh);
            if (residual) f += ldf(residual + base + j);
            stf(y + base + j, relu ? fmaxf(f, 0.f) : f);
        }
    }
}

// dbeta = sum g, dgamma = sum g * xhat, g = dy * (y > 0 if relu), with one CTA per (b, c) ROW -- the access pattern of
// bn_bwd_apply, which streams at ~90 % of the copy peak where one CTA per channel reaches ~50 %: each CTA reads two
// contiguous rows front to back. A row's two
// partial sums go to `partials` [B][C][2] (doubles); the CTA that completes a channel (per-channel arrival counter) adds
// the B partials in image order -- deterministic -- and RESETS the counter, so the scratch only has to be zeroed when it is
// allocated, not per call.
template <typename T, int VN>
__global__ void __launch_bounds__(256) bn_bwd_reduce_rows_kernel(const T* __restrict__ dy, const T* __restrict__ y,
                                                                 const unsigned* __restrict__ relu_mask,
                                                                 const T* __restrict__ x, const float* __restrict__ mean,
                                                                 const float* __restrict__ invstd, int relu,
                                                                 float* __restrict__ dgamma, float* __restrict__ dbeta, int B,
                                                                 int C, int hw, double* __restrict__ partials,
                                                                 unsigned* __restrict__ counters) {
    __shared__ double red[16];
    const int row = blockIdx.x, c = row % C;
    const float m = mean[c], is = invstd[c];
    const size_t base = (size_t)row * hw;
    float sg = 0.f, sgx = 0.f;
    if constexpr (VN != 0) {
        const int nv = hw / VN, wpr = (nv + 32 / VN - 1) / (32 / VN);
#pragma unroll 3
        for (int j = threadIdx.x; j < nv; j += 256) {
            typename VecSel<T, VN>::type g, yy, xx;
            g.load(dy + base + VN * j);
            xx.load(x + base + VN * j);
            unsigned bits = (1u << VN) - 1u;
            if (relu) {
                if (relu_mask != nullptr) {
                    bits = mask_bits<VN>(relu_mask + (size_t)row * wpr, j);
                } else {
                    yy.load(y + base + VN * j);
                    bits = 0u;
#pragma unroll
                    for (int e = 0; e < VN; ++e) bits |= (yy.get(e) > 0.f ? 1u : 0u) << e;
                }
            }
#pragma unroll
            for (int e = 0; e < VN; ++e) {
                const float gv = ((bits >> e) & 1u) ? g.get(e) : 0.f;
                sg += gv;
                sgx = fmaf(gv, (xx.get(e) - m) * is, sgx);
            }
        }
    } else {
        for (int j = threadIdx.x; j < hw; j += 256) {
            const float gv = (!relu || ldf(y + base + j) > 0.f) ? ldf(dy + base + j) : 0.f;
            sg += gv;
            sgx = fmaf(gv, (ldf(x + base + j) - m) * is, sgx);
        }
    }
    // block sums (256 threads = 8 warps): both values in one round
    double a = (double)sg, q = (double)sgx;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        q += __shfl_xor_sync(0xffffffffu, q, o);
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) red[wid] = a, red[8 + wid] = q;
    __syncthreads();
    if (threadIdx.x == 0) {
        a = q = 0.0;
        for (int i = 0; i < 8; ++i) a += red[i], q += red[8 + i];
        partials[(size_t)row * 2] = a;
        partials[(size_t)row * 2 + 1] = q;
        __threadfence();
        if (atomicAdd(counters + c, 1u) == (unsigned)B - 1) {
            __threadfence();
            a = q = 0.0;
            for (int b = 0; b < B; ++b) {
                a += __ldcg(partials + ((size_t)b * C + c) * 2);
                q += __ldcg(partials + ((size_t)b * C + c) * 2 + 1);
            }
            dbeta[c] = (float)a;
            dgamma[c] = (float)q;
            counters[c] = 0u;  // ready for the next call on this scratch
        }
    }
}

// one CTA per (b, c) row: dx = gamma*invstd*(g - [training] (dbeta + xhat*dgamma)/n); dres = g
template <typename T, int VN>
__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(const T* __restrict__ dy, const T* __restrict__ y,
                                                           const unsigned* __restrict__ relu_mask,
                                                           const T* __restrict__ x, const float* __restrict__ mean,
                                                           const float* __restrict__ invstd, const float* __restrict__ gamma,
                                                           const float* __restrict__ dgamma, const float* __restrict__ dbeta,
                                                           int relu, int training, float inv_n, T* __restrict__ dx,
                                                           T* __restrict__ dres, int C, int hw) {
    const int row = blockIdx.x, c = row % C;
    const float m = mean[c], is = invstd[c], gi = gamma[c] * is;
    const float k1 = training ? dbeta[c] * inv_n : 0.f, k2 = training ? dgamma[c] * inv_n : 0.f;
    const size_t base = (size_t)row * hw;
    if constexpr (VN != 0) {
        const int nv = hw / VN, wpr = (nv + 32 / VN - 1) / (32 / VN);
        for (int j = threadIdx.x; j < nv; j += 256) {
            typename VecSel<T, VN>::type g, yy, xx, o, r;
            g.load(dy + base + VN * j);
            xx.load(x + base + VN * j);
            unsigned bits = (1u << VN) - 1u;
            if (relu) {
                if (relu_mask != nullptr) {
                    bits = mask_bits<VN>(relu_mask + (size_t)row * wpr, j);
                } else {
                    yy.load(y + base + VN * j);
                    bits = 0u;
#pragma unroll
                    for (int e = 0; e < VN; ++e) bits |= (yy.get(e) > 0.f ? 1u : 0u) << e;
                }
            }
#pragma unroll
            for (int e = 0; e < VN; ++e) {
                const float gv = ((bits >> e) & 1u) ? g.get(e) : 0.f;
                const float xh = (xx.get(e) - m) * is;
                o.set(e, gi * (gv - k1 - xh * k2));
                r.set(e, gv);
            }
            o.store(dx + base + VN * j);
            if (dres) r.store(dres + base + VN * j);
        }
    } else {
        for (int j = threadIdx.x; j < hw; j += 256) {
            const float gv = (!relu || ldf(y + base + j) > 0.f) ? ldf(dy + base + j) : 0.f;
            const float xh = (ldf(x + base + j) - m) * is;
            stf(dx + base + j, gi * (gv - k1 - xh * k2));
            if (dres) stf(dres + base + j, gv);
        }
    }
}

// vector width of the streaming loops: 4 (fp32: 16-byte rows; bf16: 8-byte), 8 (bf16, 16-byte rows), 0 = scalar
static int vec_ok(int hw, const void* a, const void* b, const void* c, const void* d, const void* e, int dtype) {
    const uintptr_t all = (uintptr_t)a | (uintptr_t)b | (uintptr_t)c | (uintptr_t)d | (uintptr_t)e;
    if (dtype != PM_F32 && hw % 8 == 0 && (all & 15) == 0) return 8;
    const uintptr_t m = dtype == PM_F32 ? 15 : 7;
    return (hw % 4 == 0 && (all & m) == 0) ? 4 : 0;
}

// mean / invstd / running statistics from the fp64 (sum, sum of squares) pairs the convolution epilogue produced
__global__ void bn_finalize_kernel(const double* __restrict__ stats, int C, double n, float eps, float* __restrict__ mean,
                                   float* __restrict__ invstd, float* __restrict__ running_mean,
                                   float* __restrict__ running_var, float momentum) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double m = stats[c] / n;
    double var = stats[C + c] / n - m * m;
    if (var < 0.0) var = 0.0;
    mean[c] = (float)m;
    invstd[c] = (float)(1.0 / sqrt(var + (double)eps));
    if (running_mean != nullptr) {
        const double unb = n > 1.0 ? var * n / (n - 1.0) : var;
        running_mean[c] = (float)((1.0 - momentum) * running_mean[c] + momentum * m);
        running_var[c] = (float)((1.0 - momentum) * running_var[c] + momentum * unb);
    }
}

}  // namespace pm


static int bn_check(int B, int C, int hw, int dtype) {
    if (dtype != PM_F32 && dtype != PM_BF16) return PM_ERR_DTYPE;
    if (B <= 0 || C <= 0 || hw <= 0 || (long long)B * C > 0x7fffffffLL || (long long)B * hw > 0x7fffffffLL)
        return PM_ERR_SHAPE;
    return 0;
}

namespace pm {
// eval-mode BatchNorm as a per-channel affine: scale = gamma / sqrt(var + eps), shift = beta - mean * scale
__global__ void bn_eval_affine_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                                      const float* __restrict__ mean, const float* __restrict__ var, float eps, int C,
                                      float* __restrict__ scale, float* __restrict__ shift) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float sc = gamma[c] * rsqrtf(var[c] + eps);
    scale[c] = sc;
    shift[c] = fmaf(-mean[c], sc, beta[c]);
}
}  // namespace pm

extern "C" int pm_bn_eval_affine(const float* gamma, const float* beta, const float* running_mean, const float* running_var,
                                 float eps, int C, float* scale, float* shift, void* stream) {
    if (!gamma || !beta || !running_mean || !running_var || !scale || !shift) return PM_ERR_NULL;
    if (C <= 0) return PM_ERR_SHAPE;
    pm::bn_eval_affine_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(gamma, beta, running_mean, running_var, eps, C,
                                                                                 scale, shift);
    PM_CHECK_LAUNCH();
    return 0;
}

extern "C" int pm_bn_finalize(const double* stats, int C, double count, float eps, float* mean, float* invstd,
                              float* running_mean, float* running_var, float momentum, void* stream) {
    if (!stats || !mean || !invstd || ((running_mean == nullptr) != (running_var == nullptr))) return PM_ERR_NULL;
    if (C <= 0 || count <= 0.0) return PM_ERR_SHAPE;
    pm::bn_finalize_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(stats, C, count, eps, mean, invstd, running_mean,
                                                                              running_var, momentum);
    PM_CHECK_LAUNCH();
    return 0;
}

extern "C" int pm_bn_stats(const void* x, int B, int C, int hw, int dtype, float eps, float* mean, float* invstd,
                           float* running_mean, float* running_var, float momentum, void* stream) {
    if (!x || !mean || !invstd || ((running_mean == nullptr) != (running_var == nullptr))) return PM_ERR_NULL;
    if (int e = bn_check(B, C, hw, dtype)) return e;
    const int vec = pm::vec_ok(hw, x, nullptr, nullptr, nullptr, nullptr, dtype);
#define X_(T) (const T*)x
    if (dtype == PM_F32) {
        if (vec) pm::bn_stats_kernel<float, 4><<<C, pm::BN_THREADS, 0, (cudaStream_t)stream>>>(X_(float), B, C, hw, eps, mean, invstd, running_mean, running_var, momentum);
        else pm::bn_stats_kernel<float, 0><<<C, pm::BN_THREADS, 0, (cudaStream_t)stream>>>(X_(float), B, C, hw, eps, mean, invstd, running_mean, running_var, momentum);
    } else {
        if (vec == 8) pm::bn_stats_kernel<__nv_bfloat16, 8><<<C, pm::BN_THREADS, 0, (cudaStream_t)stream>>>(X_(__nv_bfloat16), B, C, hw, eps, mean, invstd, running_mean, running_var, momentum);
        else if (vec) pm::bn_stats_kernel<__nv_bfloat16, 4><<<C, pm::BN_THREADS, 0, (cudaStream_t)stream>>>(X_(__nv_bfloat16), B, C, hw, eps, mean, invstd, running_mean, running_var, momentum);
        else pm::bn_stats_kernel<__nv_bfloat16, 0><<<C, pm::BN_THREADS, 0, (cudaStream_t)stream>>>(X_(__nv_bfloat16), B, C, hw, eps, mean, invstd, running_mean, running_var, momentum);
    }
#undef X_
    PM_CHECK_LAUNCH();
    return 0;
}

extern "C" int pm_bn_mask_words(int B, int C, int hw) { return hw % 4 == 0 ? B * C * ((hw / 4 + 7) / 8) : 0; }

static int bn_apply_impl(const void* x, const float* mean, const float* invstd, const float* gamma, const float* beta,
                         const void* residual, void* y, uint32_t* relu_mask, int relu, int B, int C, int hw, int dtype,
                         pm::BnFinalize fin, void* stream);

extern "C" int pm_bn_apply(const void* x, const float* mean, const float* invstd, const float* gamma, const float* beta,
                           const void* residual, void* y, uint32_t* relu_mask, int relu, int B, int C, int hw, int dtype,
                           void* stream) {
    if (!mean || !invstd) return PM_ERR_NULL;
    return bn_apply_impl(x, mean, invstd, gamma, beta, residual, y, relu_mask, relu, B, C, hw, dtype,
                         pm::BnFinalize{nullptr, nullptr, 0.0, 0.f, 0.f, nullptr, nullptr, nullptr, nullptr, nullptr}, stream);
}

extern "C" int pm_bn_apply_stats(const void* x, const double* stats, double count, float eps, const float* gamma,
                                 const float* beta, const void* residual, void* y, uint32_t* relu_mask, int relu,
                                 float* mean_out, float* invstd_out, float* running_mean, float* running_var, float momentum,
                                 const double* count_dev, long long* num_batches_tracked, int B, int C, int hw, int dtype,
                                 void* stream) {
    if (!stats || !mean_out || !invstd_out || ((running_mean == nullptr) != (running_var == nullptr))) return PM_ERR_NULL;
    if (!(count > 0.0)) return PM_ERR_SHAPE;
    return bn_apply_impl(x, nullptr, nullptr, gamma, beta, residual, y, relu_mask, relu, B, C, hw, dtype,
                         pm::BnFinalize{stats, count_dev, count, eps, momentum, mean_out, invstd_out, running_mean, running_var, num_batches_tracked},
                         stream);
}

static int bn_apply_impl(const void* x, const float* mean, const float* invstd, const float* gamma, const float* beta,
                         const void* residual, void* y, uint32_t* relu_mask, int relu, int B, int C, int hw, int dtype,
                         pm::BnFinalize fin, void* stream) {
    if (!x || !gamma || !beta || !y) return PM_ERR_NULL;
    if (int e = bn_check(B, C, hw, dtype)) return e;
    const int vec = pm::vec_ok(hw, x, residual, y, nullptr, nullptr, dtype);
    if (relu_mask != nullptr && !vec) return PM_ERR_ALIGN;  // the packed mask exists only on the vector path
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == PM_F32) {
        if (vec) pm::bn_apply_kernel<float, 4><<<B * C, 256, 0, st>>>((const float*)x, mean, invstd, gamma, beta, (const float*)residual, (float*)y, relu_mask, relu, C, hw, fin);
        else pm::bn_apply_kernel<float, 0><<<B * C, 256, 0, st>>>((const float*)x, mean, invstd, gamma, beta, (const float*)residual, (float*)y, relu_mask, relu, C, hw, fin);
    } else {
        typedef __nv_bfloat16 bf;
        if (vec == 8) pm::bn_apply_kernel<bf, 8><<<B * C, 256, 0, st>>>((const bf*)x, mean, invstd, gamma, beta, (const bf*)residual, (bf*)y, relu_mask, relu, C, hw, fin);
        else if (vec) pm::bn_apply_kernel<bf, 4><<<B * C, 256, 0, st>>>((const bf*)x, mean, invstd, gamma, beta, (const bf*)residual, (bf*)y, relu_mask, relu, C, hw, fin);
        else pm::bn_apply_kernel<bf, 0><<<B * C, 256, 0, st>>>((const bf*)x, mean, invstd, gamma, beta, (const bf*)residual, (bf*)y, relu_mask, relu, C, hw, fin);
    }
    PM_CHECK_LAUNCH();
    return 0;
}

/* BatchNorm backward sums with one CTA per (image, channel) row (bn_bwd_reduce_rows_kernel). scratch:
 * pm_bn_bwd_rows_scratch_bytes(B, C) bytes, 8-byte aligned, zeroed ONCE when allocated (the kernel leaves its arrival
 * counters at zero); one scratch per stream that may run this concurrently. */
extern "C" int pm_bn_bwd_rows_scratch_bytes(int B, int C) { return (B > 0 && C > 0) ? B * C * 2 * 8 + C * 4 : 0; }
extern "C" int pm_bn_bwd_reduce_rows(const void* dy, const void* y, const uint32_t* relu_mask, const void* x, const float* mean,
                                     const float* invstd, int relu, float* dgamma, float* dbeta, int B, int C, int hw, int dtype,
                                     void* scratch, void* stream) {
    if (!dy || !x || !mean || !invstd || !dgamma || !dbeta || (relu && !y && !relu_mask)) return PM_ERR_NULL;
    if (!scratch || ((uintptr_t)scratch & 7)) return PM_ERR_NULL;
    if (int e = bn_check(B, C, hw, dtype)) return e;
    const int vec = pm::vec_ok(hw, dy, y, x, nullptr, nullptr, dtype);
    if (relu && !y && !vec) return PM_ERR_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    double* partials = (double*)scratch;
    unsigned* counters = (unsigned*)(partials + (size_t)B * C * 2);
    const int grid = B * C;
    if (dtype == PM_F32) {
        if (vec) pm::bn_bwd_reduce_rows_kernel<float, 4><<<grid, 256, 0, st>>>((const float*)dy, (const float*)y, relu_mask, (const float*)x, mean, invstd, relu, dgamma, dbeta, B, C, hw, partials, counters);
        else pm::bn_bwd_reduce_rows_kernel<float, 0><<<grid, 256, 0, st>>>((const float*)dy, (const float*)y, relu_mask, (const float*)x, mean, invstd, relu, dgamma, dbeta, B, C, hw, partials, counters);
    } else {
        typedef __nv_bfloat16 bf;
        if (vec == 8) pm::bn_bwd_reduce_rows_kernel<bf, 8><<<grid, 256, 0, st>>>((const bf*)dy, (const bf*)y, relu_mask, (const bf*)x, mean, invstd, relu, dgamma, dbeta, B, C, hw, partials, counters);
        else if (vec) pm::bn_bwd_reduce_rows_kernel<bf, 4><<<grid, 256, 0, st>>>((const bf*)dy, (const bf*)y, relu_mask, (const bf*)x, mean, invstd, relu, dgamma, dbeta, B, C, hw, partials, counters);
        else pm::bn_bwd_reduce_rows_kernel<bf, 0><<<grid, 256, 0, st>>>((const bf*)dy, (const bf*)y, relu_mask, (const bf*)x, mean, invstd, relu, dgamma, dbeta, B, C, hw, partials, counters);
    }
    PM_CHECK_LAUNCH();
    return 0;
}

extern "C" int pm_bn_bwd_apply(const void* dy, const void* y, const uint32_t* relu_mask, const void* x, const float* mean,
                               const float* invstd, const float* gamma, const float* dgamma, const float* dbeta, int relu,
                               int training, void* dx, void* dres, int B, int C, int hw, int dtype, void* stream) {
    if (!dy || !x || !mean || !invstd || !gamma || !dgamma || !dbeta || !dx || (relu && !y && !relu_mask))
        return PM_ERR_NULL;
    if (int e = bn_check(B, C, hw, dtype)) return e;
    const int vec = pm::vec_ok(hw, dy, y, x, dx, dres, dtype);
    if (relu && !y && !vec) return PM_ERR_ALIGN;
    const float inv_n = 1.f / ((float)B * (float)hw);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == PM_F32) {
        if (vec) pm::bn_bwd_apply_kernel<float, 4><<<B * C, 256, 0, st>>>((const float*)dy, (const float*)y, relu_mask, (const float*)x, mean, invstd, gamma, dgamma, dbeta, relu, training, inv_n, (float*)dx, (float*)dres, C, hw);
        else pm::bn_bwd_apply_kernel<float, 0><<<B * C, 256, 0, st>>>((const float*)dy, (const float*)y, relu_mask, (const float*)x, mean, invstd, gamma, dgamma, dbeta, relu, training, inv_n, (float*)dx, (float*)dres, C, hw);
    } else {
        typedef __nv_bfloat16 bf;
        if (vec == 8) pm::bn_bwd_apply_kernel<bf, 8><<<B * C, 256, 0, st>>>((const bf*)dy, (const bf*)y, relu_mask, (const bf*)x, mean, invstd, gamma, dgamma, dbeta, relu, training, inv_n, (bf*)dx, (bf*)dres, C, hw);
        else if (vec) pm::bn_bwd_apply_kernel<bf, 4><<<B * C, 256, 0, st>>>((const bf*)dy, (const bf*)y, relu_mask, (const bf*)x, mean, invstd, gamma, dgamma, dbeta, relu, training, inv_n, (bf*)dx, (bf*)dres, C, hw);
        else pm::bn_bwd_apply_kernel<bf, 0><<<B * C, 256, 0, st>>>((const bf*)dy, (const bf*)y, relu_mask, (const bf*)x, mean, invstd, gamma, dgamma, dbeta, relu, training, inv_n, (bf*)dx, (bf*)dres, C, hw);
    }
    PM_CHECK_LAUNCH();
    return 0;
}
