// Segmentation validation metrics in one pass over the label map: for every label pixel the bilinearly up-sampled
// (align_corners=True) class logits, their argmax, the cross-entropy term and one confusion-matrix increment.
//
// Reference: the validation loop train.py:847-939 and the whole-image eval eval.py:277-286,304-337 -- the head's output
// up-sampled to label size (deepv3plus.py:575-578, mynn.py:57-62), criterion on it, `argmax`, `.cpu()` and NumPy
// `fast_hist` (utils/misc.py:65-73: bincount(K * label + pred) over the labels in [0,K)). The [B,K,Hm,Wm] map never
// exists and nothing leaves the device.
//
// Interpolation matches ATen's upsample_bilinear2d_out_frame bit for bit: src = scale * dst (fp32), i0 = trunc(src),
// lambda = src - i0, and value = fma(h0, fma(w0, a, w1 * b), h1 * fma(w0, c, w1 * d)) -- the contraction nvcc made of
// `h0λ·(w0λ·a + w1λ·b) + h1λ·(w0λ·c + w1λ·d)` in torch's sm_100 build. Written with explicit round-to-nearest
// intrinsics so the compiler cannot contract it differently here. Equal sizes copy (torch does too).
//
// A CTA owns a TY x TX tile of label pixels of one image. In up-sampling mode it first stages the logits of the tile's
// footprint in shared memory pixel-major ([px][KP], KP = 4 mod 8 so that the 16-byte loads of a quarter-warp hit
// distinct banks), transposed from NCHW on the way in. Per pixel: K interpolated values in registers, a running
// argmax with strict '>' (the first maximal class wins, as torch.argmax), the sum of exp2((v - max) * log2 e), and the
// labelled class's value recomputed from shared memory with the same expression. Confusion increments go to per-CTA
// uint32 bins through warp aggregation (match.any on the bin); each non-zero bin is flushed once per CTA.
#include "pm_common.cuh"

namespace pm {
namespace se {

constexpr int THREADS = 256, TY = 16, TX = 32, PPT = TY * TX / THREADS;  // label pixels per thread
constexpr float PAD = -1e30f;                                             // padded class slots: never the max, exp -> 0

__device__ __forceinline__ float ex2a(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float lg2a(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

template <typename T>
__device__ __forceinline__ float ld_logit(const T* p);
template <>
__device__ __forceinline__ float ld_logit<float>(const float* p) { return __ldg(p); }
template <>
__device__ __forceinline__ float ld_logit<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }

template <typename T, int KP, bool IDENT>
__global__ void __launch_bounds__(THREADS)
    seg_eval_kernel(const T* __restrict__ logits, const void* __restrict__ labels, int u8, int K, int h, int w, int Hm,
                    int Wm, float sy, float sx, unsigned long long* __restrict__ conf, unsigned char* __restrict__ pred,
                    unsigned long long* __restrict__ ws, float* __restrict__ out) {
    extern __shared__ __align__(16) float s_px[];   // [footprint px][KP] (up-sampling mode only)
    __shared__ unsigned bins[31 * 31];
    __shared__ float red_loss[THREADS / 32];
    __shared__ unsigned red_cnt[THREADS / 32][2];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int b = blockIdx.z, Y0 = blockIdx.y * TY, X0 = blockIdx.x * TX;
    const size_t plane = (size_t)h * w;
    const T* lg = logits + (size_t)b * K * plane;

    // footprint of the tile on the logit grid (rows ry0..ry0+nr-1, columns rx0..rx0+nc-1)
    int ry0 = 0, rx0 = 0, nc = 1;
    if (!IDENT) {
        float l;
        ry0 = tap(sy, Y0, h, &l);
        const int ry1 = min(tap(sy, min(Y0 + TY, Hm) - 1, h, &l) + 1, h - 1);
        rx0 = tap(sx, X0, w, &l);
        const int rx1 = min(tap(sx, min(X0 + TX, Wm) - 1, w, &l) + 1, w - 1);
        const int nr = ry1 - ry0 + 1;
        nc = rx1 - rx0 + 1;
        const int npx = nr * nc;
        for (int i = tid; i < KP * npx; i += THREADS) {
            const int k = i / npx, p = i - k * npx;
            const int r = p / nc, c = p - r * nc;
            s_px[p * KP + k] = k < K ? ld_logit(lg + (size_t)k * plane + (size_t)(ry0 + r) * w + rx0 + c) : PAD;
        }
    }
    for (int i = tid; i < K * K; i += THREADS) bins[i] = 0u;
    __syncthreads();

    const void* lab_img = label_image(labels, (size_t)b * Hm * Wm, u8);
    unsigned char* pred_img = pred ? pred + (size_t)b * Hm * Wm : nullptr;
    float loss = 0.f;   // natural-log units
    unsigned nvalid = 0, nbad = 0;
#pragma unroll 1
    for (int it = 0; it < PPT; ++it) {   // warp-uniform trip count: every lane reaches the match below
        const int idx = tid + it * THREADS;
        const int Y = Y0 + idx / TX, X = X0 + idx % TX;
        const bool live = Y < Hm && X < Wm;
        int key = -1;
        if (live) {
            const size_t li = (size_t)Y * Wm + X;
            const long long raw = u8 ? (long long)__ldg(reinterpret_cast<const unsigned char*>(lab_img) + li)
                                     : __ldg(reinterpret_cast<const long long*>(lab_img) + li);
            const bool valid = raw >= 0 && raw < K;
            nbad += (!valid && raw != PM_IGNORE_LABEL) ? 1u : 0u;
            float v[KP];
            float h0 = 1.f, h1 = 0.f, w0 = 1.f, w1 = 0.f;
            const float *pa = nullptr, *pb = nullptr, *pc = nullptr, *pd = nullptr;
            if (IDENT) {
                const T* p = lg + li;
#pragma unroll
                for (int k = 0; k < KP; ++k) v[k] = k < K ? ld_logit(p + (size_t)k * plane) : PAD;
            } else {
                float ly, lx;
                const int y0 = tap(sy, Y, h, &ly), x0 = tap(sx, X, w, &lx);
                const int dy = y0 < h - 1 ? nc * KP : 0, dx = x0 < w - 1 ? KP : 0;
                h1 = ly, h0 = __fsub_rn(1.f, ly), w1 = lx, w0 = __fsub_rn(1.f, lx);
                pa = s_px + ((y0 - ry0) * nc + (x0 - rx0)) * KP;
                pb = pa + dx, pc = pa + dy, pd = pc + dx;
                const float2 H0 = make_float2(h0, h0), H1 = make_float2(h1, h1), W0 = make_float2(w0, w0),
                             W1 = make_float2(w1, w1);
#pragma unroll
                for (int q = 0; q < KP / 4; ++q) {
                    const float4 a = reinterpret_cast<const float4*>(pa)[q], bq = reinterpret_cast<const float4*>(pb)[q];
                    const float4 c = reinterpret_cast<const float4*>(pc)[q], d = reinterpret_cast<const float4*>(pd)[q];
                    const float2 lo = lerp4(H0, H1, W0, W1, make_float2(a.x, a.y), make_float2(bq.x, bq.y),
                                            make_float2(c.x, c.y), make_float2(d.x, d.y));
                    const float2 hi = lerp4(H0, H1, W0, W1, make_float2(a.z, a.w), make_float2(bq.z, bq.w),
                                            make_float2(c.z, c.w), make_float2(d.z, d.w));
                    v[4 * q] = lo.x, v[4 * q + 1] = lo.y, v[4 * q + 2] = hi.x, v[4 * q + 3] = hi.y;
                }
            }
            float m = v[0];
            int arg = 0;
#pragma unroll
            for (int k = 1; k < KP; ++k)
                if (v[k] > m) m = v[k], arg = k;
            if (pred_img) pred_img[li] = (unsigned char)arg;
            if (valid) {
                const int y = (int)raw;
                const float vy = IDENT ? ld_logit(lg + li + (size_t)y * plane)
                                       : lerp4(h0, h1, w0, w1, pa[y], pb[y], pc[y], pd[y]);
                constexpr float L2E = 1.4426950408889634f;
                const float2 m2 = make_float2(-m, -m), l2e = make_float2(L2E, L2E);
                float2 s2 = make_float2(0.f, 0.f);
#pragma unroll
                for (int k = 0; k < KP; k += 2) {
                    const float2 t = __fmul2_rn(__fadd2_rn(make_float2(v[k], v[k + 1]), m2), l2e);
                    s2 = __fadd2_rn(s2, make_float2(ex2a(t.x), ex2a(t.y)));
                }
                loss += (m - vy) + 0.6931471805599453f * lg2a(s2.x + s2.y);
                ++nvalid;
                key = y * K + arg;
            }
        }
        // confident models put most lanes of a warp on one (mostly diagonal) bin: one shared atomic per distinct bin
        const unsigned peers = __match_any_sync(0xffffffffu, key);
        if (key >= 0 && (int)(__ffs(peers) - 1) == lane) atomicAdd(&bins[key], (unsigned)__popc(peers));
    }

    loss = warp_sum(loss);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        nvalid += __shfl_xor_sync(0xffffffffu, nvalid, o);
        nbad += __shfl_xor_sync(0xffffffffu, nbad, o);
    }
    if (lane == 0) red_loss[wid] = loss, red_cnt[wid][0] = nvalid, red_cnt[wid][1] = nbad;
    __syncthreads();
    for (int i = tid; i < K * K; i += THREADS)
        if (bins[i]) atomicAdd(conf + i, (unsigned long long)bins[i]);
    if (tid == 0) {
        float tl = 0.f;
        unsigned tv = 0, tb = 0;
        for (int i = 0; i < THREADS / 32; ++i) tl += red_loss[i], tv += red_cnt[i][0], tb += red_cnt[i][1];
        if (tv) {
            atomicAdd(reinterpret_cast<double*>(ws + PM_SEG_WS_LOSS_SUM), (double)tl);
            atomicAdd(ws + PM_SEG_WS_VALID, (unsigned long long)tv);
        }
        if (tb) atomicAdd(ws + PM_SEG_WS_BAD, (unsigned long long)tb);
        __threadfence();
        const unsigned long long nblocks = (unsigned long long)gridDim.x * gridDim.y * gridDim.z;
        if (atomicAdd(ws + PM_SEG_WS_COUNTER, 1ULL) == nblocks - 1) {
            __threadfence();
            const unsigned long long V = atomicAdd(ws + PM_SEG_WS_VALID, 0ULL);
            const double sum = __longlong_as_double((long long)atomicAdd(ws + PM_SEG_WS_LOSS_SUM, 0ULL));
            out[0] = (float)(sum / (double)V);   // V == 0 -> 0/0 = NaN like torch
        }
    }
}

// Largest footprint (in logit rows or columns) of a TILE-long run of output indices, with the kernel's own arithmetic.
int footprint(float scale, int n_out, int n_in, int tile) {
    int mx = 1;
    for (int o0 = 0; o0 < n_out; o0 += tile) {
        const int a = min((int)(scale * (float)o0), n_in - 1);
        const int z = min(min((int)(scale * (float)(min(o0 + tile, n_out) - 1)), n_in - 1) + 1, n_in - 1);
        mx = max(mx, z - a + 1);
    }
    return mx;
}

template <typename T, int KP>
int launch(const void* logits, const void* labels, int u8, int B, int K, int h, int w, int Hm, int Wm, int64_t* conf,
           uint8_t* pred, void* ws, float* out, cudaStream_t st) {
    const dim3 grid((Wm + TX - 1) / TX, (Hm + TY - 1) / TY, B);
    auto* c = reinterpret_cast<unsigned long long*>(conf);
    auto* wsq = reinterpret_cast<unsigned long long*>(ws);
    if (h == Hm && w == Wm) {
        seg_eval_kernel<T, KP, true><<<grid, THREADS, 0, st>>>((const T*)logits, labels, u8, K, h, w, Hm, Wm, 0.f, 0.f, c, pred,
                                                               wsq, out);
    } else {
        // PyTorch's align_corners scale, (in - 1) / (out - 1) in fp32, 0 when out == 1
        const float sy = Hm > 1 ? (float)(h - 1) / (float)(Hm - 1) : 0.f;
        const float sx = Wm > 1 ? (float)(w - 1) / (float)(Wm - 1) : 0.f;
        const size_t smem = (size_t)footprint(sy, Hm, h, TY) * footprint(sx, Wm, w, TX) * KP * sizeof(float);
        auto kern = seg_eval_kernel<T, KP, false>;
        if (smem > 48 * 1024) {
            const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return (int)e;
        }
        kern<<<grid, THREADS, smem, st>>>((const T*)logits, labels, u8, K, h, w, Hm, Wm, sy, sx, c, pred, wsq, out);
    }
    PM_CHECK_LAUNCH();
    return 0;
}

template <typename T>
int dispatch(const void* logits, const void* labels, int u8, int B, int K, int h, int w, int Hm, int Wm, int64_t* conf,
             uint8_t* pred, void* ws, float* out, cudaStream_t st) {
    // KP = 4 mod 8: a quarter-warp's 16-byte loads of 8 different pixels cover all 32 banks once
    if (K <= 4) return launch<T, 4>(logits, labels, u8, B, K, h, w, Hm, Wm, conf, pred, ws, out, st);
    if (K <= 12) return launch<T, 12>(logits, labels, u8, B, K, h, w, Hm, Wm, conf, pred, ws, out, st);
    if (K <= 20) return launch<T, 20>(logits, labels, u8, B, K, h, w, Hm, Wm, conf, pred, ws, out, st);
    if (K <= 28) return launch<T, 28>(logits, labels, u8, B, K, h, w, Hm, Wm, conf, pred, ws, out, st);
    return launch<T, 36>(logits, labels, u8, B, K, h, w, Hm, Wm, conf, pred, ws, out, st);
}

}  // namespace se
}  // namespace pm

extern "C" int pm_seg_eval(const void* logits, int dtype, int B, int K, int h, int w, const void* labels, int labels_are_u8,
                           int Hm, int Wm, int64_t* confusion, uint8_t* pred, void* ws, float* out, void* stream) {
    if (!logits || !labels || !confusion || !ws || !out) return PM_ERR_NULL;
    if (dtype != PM_F32 && dtype != PM_BF16) return PM_ERR_DTYPE;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (B <= 0 || h <= 0 || w <= 0 || Hm < h || Wm < w || B > 65535 || Hm > 65535 * pm::se::TY) return PM_ERR_SHAPE;
    if (((uintptr_t)confusion & 7) || ((uintptr_t)ws & 7)) return PM_ERR_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    const int u8 = labels_are_u8 ? 1 : 0;
    if (dtype == PM_F32)
        return pm::se::dispatch<float>(logits, labels, u8, B, K, h, w, Hm, Wm, confusion, pred, ws, out, st);
    return pm::se::dispatch<__nv_bfloat16>(logits, labels, u8, B, K, h, w, Hm, Wm, confusion, pred, ws, out, st);
}
