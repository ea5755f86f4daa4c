// Fixed-order combination of per-CTA partials: the second half of the ordered (bitwise reproducible) entry points.
//
// The kernels whose default instantiations flush per-CTA partials with float atomics (class sums, BatchNorm statistics,
// dM, the read-loss tap tiles) have an ordered instantiation that STORES each CTA's partial to scratch instead. Every CTA
// already visits its tiles in a fixed order, so each partial is reproducible; the kernels below add the partials in
// ascending CTA order, so the result does not depend on which CTA finished first.
#include "pm_common.cuh"
#include "pm_internal.h"

namespace pm {

// dst[i] += sum_g part[g * n + i], g ascending. One thread per element; the loads of a group of 8 partials are issued
// before their adds so that a thread keeps several loads in flight.
template <typename T>
__global__ void __launch_bounds__(256) reduce_partials_kernel(T* __restrict__ dst, const T* __restrict__ part, int G, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    T acc = 0;
    int g = 0;
    for (; g + 8 <= G; g += 8) {
        T v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = __ldg(part + (size_t)(g + j) * n + i);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc += v[j];
    }
    for (; g < G; ++g) acc += __ldg(part + (size_t)g * n + i);
    dst[i] += acc;
}

template <typename T>
static int reduce_partials(T* dst, const T* part, int G, long long n, cudaStream_t st) {
    if (G <= 0 || n <= 0) return 0;
    const long long blocks = (n + 255) / 256;
    reduce_partials_kernel<T><<<(unsigned)blocks, 256, 0, st>>>(dst, part, G, n);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

int reduce_partials_f32(float* dst, const float* part, int G, long long n, cudaStream_t st) {
    return reduce_partials<float>(dst, part, G, n, st);
}
int reduce_partials_f64(double* dst, const double* part, int G, long long n, cudaStream_t st) {
    return reduce_partials<double>(dst, part, G, n, st);
}

// ds_rl of every feature pixel from the stored (TY+1) x (TX+1) tap tiles of the read-loss kernels: the owner tile's entry,
// then the halo entries of the tile above, the tile to the left and the diagonal tile, in that order. Block 0 also adds
// the CTAs' loss partials in CTA order and finalises out[0] = loss_sum / V, out[1] = 1 / (V*T) (V from the histogram
// in ws), as the last CTA of the atomic kernels does.
__global__ void __launch_bounds__(256)
    readloss_gather_kernel(const float* __restrict__ tiles, const float* __restrict__ lossp, int ncta, int h, int w, int KP,
                           int TY, int TX, int tiles_x, int tiles_y, int K, float temperature, long long n4,
                           float* __restrict__ ds_rl, unsigned long long* __restrict__ ws, float* __restrict__ out) {
    const int LDX = TX + 1, q4 = KP / 4;
    const size_t tile_elems = (size_t)(TY + 1) * LDX * KP;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
        const long long e = i / q4;
        const int q = (int)(i - e * q4);
        const int fx = (int)(e % w);
        const long long r = e / w;
        const int fy = (int)(r % h), b = (int)(r / h);
        const int tyi = fy / TY, txi = fx / TX, ly = fy - tyi * TY, lx = fx - txi * TX;
        auto at = [&](int ty, int tx, int yy, int xx) {
            const size_t t = (size_t)((b * tiles_y + ty) * tiles_x + tx);
            return __ldg(reinterpret_cast<const float4*>(tiles + t * tile_elems + (size_t)(yy * LDX + xx) * KP) + q);
        };
        float4 v = at(tyi, txi, ly, lx);
        if (ly == 0 && tyi > 0) {
            const float4 a = at(tyi - 1, txi, TY, lx);
            v.x += a.x, v.y += a.y, v.z += a.z, v.w += a.w;
        }
        if (lx == 0 && txi > 0) {
            const float4 a = at(tyi, txi - 1, ly, TX);
            v.x += a.x, v.y += a.y, v.z += a.z, v.w += a.w;
        }
        if (ly == 0 && lx == 0 && tyi > 0 && txi > 0) {
            const float4 a = at(tyi - 1, txi - 1, TY, TX);
            v.x += a.x, v.y += a.y, v.z += a.z, v.w += a.w;
        }
        reinterpret_cast<float4*>(ds_rl)[i] = v;
    }
    if (blockIdx.x != 0) return;
    __shared__ double red[256];
    double part = 0.0;
    for (int g = threadIdx.x; g < ncta; g += blockDim.x) part += (double)__ldg(lossp + g) * 0.6931471805599453;
    red[threadIdx.x] = part;
    __syncthreads();
    if (threadIdx.x == 0) {
        double sum = 0.0;
        for (int t = 0; t < (int)blockDim.x; ++t) sum += red[t];
        unsigned long long V = 0;
        for (int k = 0; k < K; ++k) V += ws[PM_WS_HIST + k];
        ws[PM_WS_LOSS_SUM] = (unsigned long long)__double_as_longlong(sum);
        out[0] = (float)(sum / (double)V);  // V == 0 -> 0/0 = NaN like torch
        out[1] = (float)(1.0 / ((double)V * (double)temperature));
    }
}

int readloss_gather(const float* tiles, const float* lossp, int ncta, int B, int h, int w, int KP, int TY, int TX, int tiles_x,
                    int tiles_y, int K, float temperature, float* ds_rl, unsigned long long* ws, float* out, cudaStream_t st) {
    const long long n4 = (long long)B * h * w * (KP / 4);
    long long blocks = (n4 + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    readloss_gather_kernel<<<(unsigned)blocks, 256, 0, st>>>(tiles, lossp, ncta, h, w, KP, TY, TX, tiles_x, tiles_y, K,
                                                              temperature, n4, ds_rl, ws, out);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

}  // namespace pm
