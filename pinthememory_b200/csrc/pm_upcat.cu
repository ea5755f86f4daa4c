// Decoder up-sample + concat of the DeepLabV3+ head (network/deepv3plus.py:569-572):
//     dec0 = cat([bot_fine(low_level), Upsample(dec0_up, low_level.size()[2:])], 1)
// with Upsample = F.interpolate(bilinear, align_corners=True) (mynn.py:57-62).
//
// Forward: one kernel writes out[B, Cf+Cc, H, W] -- planes [0,Cf) copied from fine[B,Cf,H,W], planes [Cf,Cf+Cc)
// up-sampled from coarse[B,Cc,h,w] -- so the up-sampled map is never materialised on its own and never re-read by a
// cat. The interpolation is ATen's upsample_bilinear2d_out_frame bit for bit (tap / lerp4 of pm_common.cuh, one
// round-to-nearest store for bf16); equal sizes copy, as torch does. Coarse taps come through L1/L2 (a coarse plane is
// 9 KB at 48x48), stores are 16-byte vectors on the 16-byte grid of the output with scalar head and tail elements.
//
// Backward: d_coarse = Wy^T G Wx, the exact transpose of the forward's sparse map (the fp32 weights of the forward's
// own taps, duplicated taps at the last row / column included), read from the coarse-channel slice of the incoming
// gradient in place (batch stride (Cf+Cc)*H*W). A CTA owns a TI x TJ tile of one d_coarse plane. Phase 1 reduces along
// Y: u[i][x] = sum_y wy(y,i) g[y][x] over the output rows feeding coarse row i, lanes along x (coalesced loads), into
// shared memory. Phase 2 reduces along X: thread (i,j) sums wx(x,j) u[i][x] over the output columns feeding coarse
// column j and stores d_coarse[i][j] once. Every sum runs in fp32 in ascending y, then ascending x: no atomics, so the
// result does not depend on scheduling. The row and column ranges come from the forward's tap arithmetic (binary search
// on the monotone source index), so both directions use the same tap set.
#include "pm_common.cuh"

namespace pm {
namespace uc {

constexpr int THREADS = 256;
constexpr int FWD_ELEMS = 4096;   // output elements per forward CTA (about 16 per thread)
constexpr int BWD_ITEMS = 256;    // d_coarse elements per backward CTA (one per thread)
constexpr int BWD_XCHUNK = 1024;  // output columns per phase-1 pass
constexpr int BWD_SMEM_FLOATS = 8192;   // phase-1 tile bound (32 KB): TI * XC <= this

__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T>
__device__ __forceinline__ T from_f(float v);
template <>
__device__ __forceinline__ float from_f<float>(float v) { return v; }
template <>
__device__ __forceinline__ __nv_bfloat16 from_f<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// First output index o in [0, n_out) whose source index is >= t (n_out if none); the source index is monotone in o.
__device__ __forceinline__ int first_tap_at_least(float scale, int n_out, int n_in, int t) {
    int lo = 0, hi = n_out;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        float l;
        if (tap(scale, mid, n_in, &l) >= t) hi = mid;
        else lo = mid + 1;
    }
    return lo;
}

template <typename T>
struct RowTaps {
    const T* r0;   // coarse row y0
    const T* r1;   // coarse row y0 + h1p
    float h0, h1;
};

template <typename T>
__device__ __forceinline__ RowTaps<T> row_taps(const T* plane, float sy, int y, int h, int w) {
    float ly;
    const int y0 = tap(sy, y, h, &ly);
    RowTaps<T> r;
    r.r0 = plane + (size_t)y0 * w;
    r.r1 = r.r0 + (y0 < h - 1 ? w : 0);
    r.h1 = ly;
    r.h0 = __fsub_rn(1.f, ly);
    return r;
}

template <typename T>
__device__ __forceinline__ float interp(const RowTaps<T>& r, float sx, int x, int w) {
    float lx;
    const int x0 = tap(sx, x, w, &lx);
    const int dx = x0 < w - 1 ? 1 : 0;
    const float w1 = lx, w0 = __fsub_rn(1.f, lx);
    return lerp4(r.h0, r.h1, w0, w1, to_f(__ldg(r.r0 + x0)), to_f(__ldg(r.r0 + x0 + dx)), to_f(__ldg(r.r1 + x0)),
                 to_f(__ldg(r.r1 + x0 + dx)));
}

// grid (row bands, Cf + Cc, B); `rows` output rows per band.
template <typename T>
__global__ void __launch_bounds__(THREADS)
    upcat_fwd_kernel(const T* __restrict__ fine, const T* __restrict__ coarse, T* __restrict__ out, int Cf, int Cc, int h,
                     int w, int H, int W, int rows, float sy, float sx) {
    constexpr int VEC = 16 / (int)sizeof(T);
    const int p = blockIdx.y, b = blockIdx.z;
    const size_t HW = (size_t)H * W;
    const int e0 = blockIdx.x * rows * W, e1 = min(blockIdx.x * rows + rows, H) * W;   // flat range in the plane
    T* dst = out + ((size_t)b * (Cf + Cc) + p) * HW;
    const bool copy = p < Cf || (h == H && w == W);
    const T* src = p < Cf ? fine + ((size_t)b * Cf + p) * HW : coarse + ((size_t)b * Cc + (p - Cf)) * ((size_t)h * w);
    // elements before the first 16-byte boundary of the output at or after e0, then whole vectors, then the tail
    const int head = min((int)((((unsigned)-(uintptr_t)(dst + e0)) & 15u) / sizeof(T)), e1 - e0);
    const int v0 = e0 + head, nvec = (e1 - v0) / VEC, t0 = v0 + nvec * VEC;

    if (copy) {
        const bool vsrc = (((uintptr_t)(src + v0)) & 15u) == 0;
        for (int v = threadIdx.x; v < nvec; v += THREADS) {
            const int e = v0 + v * VEC;
            uint4 val;
            if (vsrc) {
                val = __ldg(reinterpret_cast<const uint4*>(src + e));
            } else {
                T tmp[VEC];
#pragma unroll
                for (int k = 0; k < VEC; ++k) tmp[k] = src[e + k];
                val = *reinterpret_cast<const uint4*>(tmp);
            }
            *reinterpret_cast<uint4*>(dst + e) = val;
        }
        const int t = threadIdx.x;
        if (t < head) dst[e0 + t] = src[e0 + t];
        if (t < e1 - t0) dst[t0 + t] = src[t0 + t];
        return;
    }

    for (int v = threadIdx.x; v < nvec; v += THREADS) {
        const int e = v0 + v * VEC;
        int y = e / W, x = e - y * W;
        RowTaps<T> r = row_taps(src, sy, y, h, w);
        __align__(16) T res[VEC];
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
            res[k] = from_f<T>(interp(r, sx, x, w));
            if (++x == W && k + 1 < VEC) {   // a vector that runs into the next row (W not a multiple of VEC)
                x = 0;
                r = row_taps(src, sy, ++y, h, w);
            }
        }
        *reinterpret_cast<uint4*>(dst + e) = *reinterpret_cast<const uint4*>(res);
    }
    const int t = threadIdx.x;
    const int e = t < head ? e0 + t : (t < head + (e1 - t0) ? t0 + t - head : -1);
    if (e >= 0) {
        const int y = e / W, x = e - y * W;
        dst[e] = from_f<T>(interp(row_taps(src, sy, y, h, w), sx, x, w));
    }
}

// grid (row bands * column tiles, Cc, B). A CTA owns coarse rows [i0, i0+TI) x columns [j0, j0+TJ) of one plane;
// dynamic shared memory: TI x XC floats (phase-1 tile of one column chunk).
template <typename T>
__global__ void __launch_bounds__(THREADS)
    upcat_bwd_kernel(const T* __restrict__ g, T* __restrict__ dc, int Cf, int Cc, int h, int w, int H, int W, int TI,
                     int TJ, int ntj, int XC, float sy, float sx) {
    extern __shared__ float s_u[];   // [TI][XC]
    __shared__ int s_rows[BWD_ITEMS + 2];
    const int tid = threadIdx.x, c = blockIdx.y, b = blockIdx.z;
    const int i0 = (blockIdx.x / ntj) * TI, j0 = (blockIdx.x % ntj) * TJ;
    const int ni = min(TI, h - i0), nj = min(TJ, w - j0);
    const T* gp = g + ((size_t)b * (Cf + Cc) + Cf + c) * ((size_t)H * W);

    // the output rows feeding coarse row i are those with source row i-1 (weight h1) or i (h0, and h1 where h1p = 0):
    // [s_rows[i-i0], s_rows[i-i0+2]) with s_rows[k] = first row whose source row is >= i0+k-1
    for (int k = tid; k < ni + 2; k += THREADS) s_rows[k] = first_tap_at_least(sy, H, h, i0 + k - 1);

    // this thread's phase-2 element and the output columns feeding it (same rule along x)
    const int ti = tid / TJ, tj = tid - ti * TJ;
    const bool mine = ti < ni && tj < nj;
    const int i = i0 + ti, j = j0 + tj;
    int xs = 0, xe = 0;
    if (mine) {
        xs = first_tap_at_least(sx, W, w, j - 1);
        xe = first_tap_at_least(sx, W, w, j + 1);
    }
    const int X0 = first_tap_at_least(sx, W, w, j0 - 1), X1 = first_tap_at_least(sx, W, w, j0 + nj);
    __syncthreads();

    float acc = 0.f;
    for (int xc = X0; xc < X1; xc += XC) {
        const int nx = min(XC, X1 - xc);
        // phase 1: u[k][x] = sum over the rows feeding coarse row i0+k, ascending
        for (int it = tid; it < ni * nx; it += THREADS) {
            const int k = it / nx, xi = it - k * nx;
            const int ic = i0 + k, ya = s_rows[k], yb = s_rows[k + 2];
            const T* col = gp + xc + xi;
            float u = 0.f;
#pragma unroll 4
            for (int y = ya; y < yb; ++y) {
                float ly;
                const int y0 = tap(sy, y, h, &ly);
                const float gv = to_f(__ldg(col + (size_t)y * W));
                if (y0 == ic) u = __fmaf_rn(__fsub_rn(1.f, ly), gv, u);
                if (y0 + (y0 < h - 1 ? 1 : 0) == ic) u = __fmaf_rn(ly, gv, u);
            }
            s_u[k * XC + xi] = u;
        }
        __syncthreads();
        // phase 2: d[i][j] += sum over this chunk's columns feeding coarse column j, ascending
        if (mine) {
            const float* ur = s_u + ti * XC;
            const int xa = max(xs, xc), xb = min(xe, xc + nx);
            for (int x = xa; x < xb; ++x) {
                float lx;
                const int x0 = tap(sx, x, w, &lx);
                const float uv = ur[x - xc];
                if (x0 == j) acc = __fmaf_rn(__fsub_rn(1.f, lx), uv, acc);
                if (x0 + (x0 < w - 1 ? 1 : 0) == j) acc = __fmaf_rn(lx, uv, acc);
            }
        }
        __syncthreads();
    }
    if (mine) dc[((size_t)b * Cc + c) * ((size_t)h * w) + (size_t)i * w + j] = from_f<T>(acc);
}

template <typename T>
int launch_fwd(const void* fine, const void* coarse, void* out, int B, int Cf, int Cc, int h, int w, int H, int W,
               cudaStream_t st) {
    const int rows = max(1, FWD_ELEMS / W);
    const dim3 grid((H + rows - 1) / rows, Cf + Cc, B);
    // PyTorch's align_corners scale, (in - 1) / (out - 1) in fp32, 0 when out == 1
    const float sy = H > 1 ? (float)(h - 1) / (float)(H - 1) : 0.f;
    const float sx = W > 1 ? (float)(w - 1) / (float)(W - 1) : 0.f;
    upcat_fwd_kernel<T><<<grid, THREADS, 0, st>>>((const T*)fine, (const T*)coarse, (T*)out, Cf, Cc, h, w, H, W, rows, sy,
                                                  sx);
    PM_CHECK_LAUNCH();
    return 0;
}

template <typename T>
int launch_bwd(const void* g, void* dc, int B, int Cf, int Cc, int h, int w, int H, int W, cudaStream_t st) {
    const int rx = (W + w - 1) / w;                     // output columns per coarse column, rounded up
    const int TJ = min(w, max(1, BWD_ITEMS / rx));      // about BWD_ITEMS output columns per tile
    const int XC = min(W, BWD_XCHUNK);
    const int TI = min(min(h, max(1, BWD_ITEMS / TJ)), max(1, BWD_SMEM_FLOATS / XC));
    const int nti = (h + TI - 1) / TI, ntj = (w + TJ - 1) / TJ;
    const float sy = H > 1 ? (float)(h - 1) / (float)(H - 1) : 0.f;
    const float sx = W > 1 ? (float)(w - 1) / (float)(W - 1) : 0.f;
    const size_t smem = (size_t)TI * XC * sizeof(float);   // <= BWD_SMEM_FLOATS floats: no opt-in needed
    upcat_bwd_kernel<T><<<dim3(nti * ntj, Cc, B), THREADS, smem, st>>>((const T*)g, (T*)dc, Cf, Cc, h, w, H, W, TI, TJ, ntj,
                                                                       XC, sy, sx);
    PM_CHECK_LAUNCH();
    return 0;
}

int check_shape(int dtype, int B, int Cf, int Cc, int h, int w, int H, int W) {
    if (dtype != PM_F32 && dtype != PM_BF16) return PM_ERR_DTYPE;
    if (B <= 0 || Cc <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0 || Cf < 0 || H < h || W < w) return PM_ERR_SHAPE;
    // grid.y = channel planes, grid.z = images; flat plane offsets are int
    if (B > 65535 || (long long)Cf + Cc > 65535 || (long long)H * W > 0x7fffffffLL) return PM_ERR_SHAPE;
    return PM_OK;
}

}  // namespace uc
}  // namespace pm

extern "C" int pm_upcat_fwd(const void* fine, const void* coarse, void* out, int dtype, int B, int Cf, int Cc, int h, int w,
                            int H, int W, void* stream) {
    if ((!fine && Cf > 0) || !coarse || !out) return PM_ERR_NULL;
    const int s = pm::uc::check_shape(dtype, B, Cf, Cc, h, w, H, W);
    if (s != PM_OK) return s;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == PM_F32) return pm::uc::launch_fwd<float>(fine, coarse, out, B, Cf, Cc, h, w, H, W, st);
    return pm::uc::launch_fwd<__nv_bfloat16>(fine, coarse, out, B, Cf, Cc, h, w, H, W, st);
}

extern "C" int pm_upcat_bwd(const void* g, void* d_coarse, int dtype, int B, int Cf, int Cc, int h, int w, int H, int W,
                            void* stream) {
    if (!g || !d_coarse) return PM_ERR_NULL;
    const int s = pm::uc::check_shape(dtype, B, Cf, Cc, h, w, H, W);
    if (s != PM_OK) return s;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == PM_F32) return pm::uc::launch_bwd<float>(g, d_coarse, B, Cf, Cc, h, w, H, W, st);
    return pm::uc::launch_bwd<__nv_bfloat16>(g, d_coarse, B, Cf, Cc, h, w, H, W, st);
}
