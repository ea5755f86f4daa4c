// Feature-cohesion read loss, fourth kernel: warps that own their cells end to end.
//
// The third kernel (a thread per label row, since removed) had the right instruction mix in its label loop but spent
// more than half of its time in per-CTA phases: tile load -> barrier -> rows -> barrier -> y-weighting -> barrier -> flush
// -> reduction -> ticket, at two CTAs per SM (profiles/r2f_ncu_full.txt, DESIGN.md section 6). Here nothing is CTA-wide
// until the very last instruction:
//   * a warp = 16 neighbouring cells of one cell row x 2 lanes per cell; each lane of a pair carries HALF of the 20 slots
//     (float2 slot pairs 2j + half): E, ratio, the two row sums and the four tap accumulators are 5 float2 each = 80
//     registers, so the kernel stays at 128 registers (16 warps per SM) while a thread still walks ALL label rows of its
//     cell -- tap accumulators live in registers for the whole cell, no row records, no y-weighting pass;
//   * the only cross-lane traffic in the label loop is one shuffle per pixel (the two half sums of the softmax);
//   * each warp stages its own [2][17][20] tile (stabilised by the warp's maximum, padded slots at -1e20) and its own
//     fixed-point one-hot tile in shared memory, synchronised with __syncwarp only;
//   * at the end of the cell row, right-hand taps move to the neighbouring cell's lanes by shuffle and every lane flushes
//     its left-hand taps with 8-byte REDs; the block meets once, for the loss sum and the last-CTA ticket.
#include "pm_common.cuh"
#include <cstdlib>

namespace pm {
namespace rc {

constexpr int THREADS = 128, WARPS = THREADS / 32, CPW = 16, KP = 20, NJ = 5;  // cells per warp; float2 slot pairs per lane
constexpr int TCOLS = CPW + 1;
constexpr int TILE_F = 2 * TCOLS * KP;       // floats of a warp's similarity tile (680)
constexpr int OSTR = 21;                    // words per feature pixel in the one-hot tile (odd: 16 cells hit 16 banks)
constexpr int OTILE_W = 720;                // >= 2 * TCOLS * OSTR = 714, a multiple of 4
constexpr int CHUNK = 3, SEG = 9;

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
__device__ __forceinline__ float rcpa(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ int bil_index(float scale, int dst, int n_in) {
    const int i0 = (int)(scale * (float)dst);
    return i0 > n_in - 1 ? n_in - 1 : i0;
}
__device__ __forceinline__ int first_ge(int c, float scale, int n_out, int n_in) {
    if (c <= 0) return 0;
    if (c > n_in - 1 || scale <= 0.f) return n_out;
    int y = (int)ceilf((float)c / scale);
    y = max(0, min(y, n_out));
    while (y > 0 && bil_index(scale, y - 1, n_in) >= c) --y;
    while (y < n_out && bil_index(scale, y, n_in) < c) ++y;
    return y;
}
__device__ __forceinline__ float2 shfl_xor2(float2 v, int m) {
    return make_float2(__shfl_xor_sync(0xffffffffu, v.x, m), __shfl_xor_sync(0xffffffffu, v.y, m));
}

__device__ __forceinline__ void red_shared_add(unsigned addr, unsigned v) {
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

struct RowCtx {
    float sx, cxf, hy, lamy, fscale;
    int Xa, ncols, nc_max, K, half;
    const unsigned char* lrow;
    unsigned o_cell;    // shared-memory byte address of the one-hot tile at (row 0, this cell's column)
};

// One label row of a cell for this lane's five slot pairs. A = stabilised logits at the cell's left edge, Bc = right - left.
template <bool EXACT>
__device__ __forceinline__ void row_pixels(const float2 (&A)[NJ], const float2 (&Bc)[NJ], const RowCtx& c, float2 (&G00)[NJ],
                                           float2 (&G01)[NJ], float2 (&G10)[NJ], float2 (&G11)[NJ], float& lossacc) {
    int labs[SEG];
#pragma unroll
    for (int i = 0; i < SEG; ++i) labs[i] = (i < c.ncols) ? (int)__ldg(c.lrow + i) : 255;
    float2 E[NJ], Rt[NJ], R0[NJ], R1[NJ];
    const float lam_first = fminf(fmaxf(c.sx * (float)c.Xa - c.cxf, 0.f), 1.f);
    const float2 lf2 = make_float2(lam_first, lam_first), sx2 = make_float2(c.sx, c.sx);
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
        if (!EXACT) {
            const float2 e0 = __ffma2_rn(lf2, Bc[i], A[i]), rr = __fmul2_rn(sx2, Bc[i]);
            E[i] = make_float2(ex2a(e0.x), ex2a(e0.y));
            Rt[i] = make_float2(ex2a(rr.x), ex2a(rr.y));
        } else {
            E[i] = A[i];
            Rt[i] = Bc[i];
        }
        R0[i] = R1[i] = make_float2(0.f, 0.f);
    }
    // one-hot term: the pair splits the PIXELS (half 0 the even ones, half 1 the odd ones); the lane that owns a pixel adds
    // its four fixed-point tap weights to the labelled class's column -- four native shared atomics and no run-length
    // bookkeeping (which cost more instructions than the atomics it saved)
    const float wt = c.hy * c.fscale, wb = c.lamy * c.fscale;
    for (int S0 = 0; S0 < c.nc_max; S0 += SEG) {
        if (S0 > 0) {
#pragma unroll
            for (int i = 0; i < SEG; ++i) labs[i] = (S0 + i < c.ncols) ? (int)__ldg(c.lrow + S0 + i) : 255;
        }
#pragma unroll
        for (int g = 0; g < SEG / CHUNK; ++g) {
            const int X0 = S0 + g * CHUNK;
            if (X0 >= c.nc_max) break;
            float lamx[CHUNK], hx[CHUNK];
#pragma unroll
            for (int i = 0; i < CHUNK; ++i) {
                lamx[i] = fminf(fmaxf(c.sx * (float)(c.Xa + X0 + i) - c.cxf, 0.f), 1.f);
                hx[i] = 1.f - lamx[i];
            }
#pragma unroll
            for (int i = 0; i < CHUNK; ++i) {
                const bool valid = labs[g * CHUNK + i] < c.K;
                float pshift = 0.f;
                float2 e[NJ];
                if (EXACT) {
                    float m = -INFINITY;
#pragma unroll
                    for (int q = 0; q < NJ; ++q) {
                        e[q] = __ffma2_rn(make_float2(lamx[i], lamx[i]), Rt[q], E[q]);
                        m = fmaxf(m, fmaxf(e[q].x, e[q].y));
                    }
                    m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 1));
                    pshift = m;
#pragma unroll
                    for (int q = 0; q < NJ; ++q) e[q] = make_float2(ex2a(e[q].x - m), ex2a(e[q].y - m));
                }
                const float2* ev = EXACT ? e : E;
                float2 s01 = __fadd2_rn(ev[0], ev[1]), s23 = __fadd2_rn(ev[2], ev[3]);
                s01 = __fadd2_rn(__fadd2_rn(s01, s23), ev[4]);
                float sum = s01.x + s01.y;
                sum += __shfl_xor_sync(0xffffffffu, sum, 1);   // the other half of the slots
                const float vf = valid ? 1.f : 0.f;
                // each pixel's loss is counted by half 0 only
                lossacc = fmaf(c.half ? 0.f : vf, pshift + lg2a(sum), lossacc);
                const float inv = rcpa(sum) * vf;
                const float2 ihx = make_float2(inv * hx[i], inv * hx[i]), ilx = make_float2(inv * lamx[i], inv * lamx[i]);
#pragma unroll
                for (int q = 0; q < NJ; ++q) {
                    R0[q] = __ffma2_rn(ev[q], ihx, R0[q]);
                    R1[q] = __ffma2_rn(ev[q], ilx, R1[q]);
                }
                if (!EXACT) {
#pragma unroll
                    for (int q = 0; q < NJ; ++q) E[q] = __fmul2_rn(E[q], Rt[q]);
                }
            }
#pragma unroll
            for (int i = 0; i < CHUNK; ++i) {
                const int cls = labs[g * CHUNK + i];
                if (cls < c.K && ((X0 + i) & 1) == c.half) {
                    // (the address lives in ONE register: left to itself the compiler re-derives the tile pointer from the
                    // CTA's shared window for every pixel, 12 integer instructions)
                    const unsigned p = c.o_cell + 4u * (unsigned)cls;
                    red_shared_add(p, __float2uint_rn(wt * hx[i]));
                    red_shared_add(p + 4 * OSTR, __float2uint_rn(wt * lamx[i]));
                    red_shared_add(p + 4 * TCOLS * OSTR, __float2uint_rn(wb * hx[i]));
                    red_shared_add(p + 4 * (TCOLS * OSTR + OSTR), __float2uint_rn(wb * lamx[i]));
                }
            }
        }
    }
    const float2 hy2 = make_float2(c.hy, c.hy), ly2 = make_float2(c.lamy, c.lamy);
#pragma unroll
    for (int q = 0; q < NJ; ++q) {
        G00[q] = __ffma2_rn(R0[q], hy2, G00[q]);
        G01[q] = __ffma2_rn(R1[q], hy2, G01[q]);
        G10[q] = __ffma2_rn(R0[q], ly2, G10[q]);
        G11[q] = __ffma2_rn(R1[q], ly2, G11[q]);
    }
}

__global__ void __launch_bounds__(THREADS, 4)
    readloss_cells_kernel(const float* __restrict__ s, const unsigned char* __restrict__ lab8, float inv_T, float temperature, int h,
                          int w, int Hm, int Wm, int K, float sy, float sx, int tiles_x, int RS, int nitems, float fscale,
                          float* __restrict__ ds_rl, unsigned long long* __restrict__ ws, float* __restrict__ out) {
    __shared__ __align__(16) float s_tiles[WARPS][TILE_F];
    __shared__ __align__(16) unsigned o_tiles[WARPS][OTILE_W];
    __shared__ float red[WARPS];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int cell = lane >> 1, half = lane & 1;
    float* s_tile = s_tiles[wid];
    unsigned* o_tile = o_tiles[wid];
    float lossacc = 0.f;  // log2 units

    const int item = blockIdx.x * WARPS + wid;   // (image, cell row, block of 16 cells, row split)
    if (item < nitems) {
        // RS > 1 (few cells: output stride 16, small batches): the label rows of a cell row are dealt round-robin to RS warps,
        // each with its own tiles; their taps meet in the global REDs like those of neighbouring cells
        const int rsp = item % RS, it2 = item / RS;
        const int tx_i = it2 % tiles_x, rest = it2 / tiles_x;
        const int cy = rest % h, b = rest / h;
        const int fx0 = tx_i * CPW, cx = fx0 + cell;
        const float c2 = inv_T * 1.4426950408889634f;

        // ---- the warp's tile: z' = s * c2 - max(tile), padded slots at -1e20; zeroed one-hot tile; geometry
        float4 v[6];
        float tmax = -INFINITY, tmin = INFINITY;
#pragma unroll
        for (int r = 0; r < 6; ++r) {
            const int i = lane + 32 * r;
            v[r] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < TILE_F / 4) {
                const int e = i / (KP / 4), q = i - e * (KP / 4);
                const int ty = e / TCOLS, tx = e - ty * TCOLS;
                const int fy = min(cy + ty, h - 1), fx = min(fx0 + tx, w - 1);
                float4 t = __ldg(reinterpret_cast<const float4*>(s + ((size_t)(b * h + fy) * w + fx) * KP) + q);
                t.x *= c2, t.y *= c2, t.z *= c2, t.w *= c2;
                if (4 * q + 0 < K) tmax = fmaxf(tmax, t.x), tmin = fminf(tmin, t.x); else t.x = -1e20f;
                if (4 * q + 1 < K) tmax = fmaxf(tmax, t.y), tmin = fminf(tmin, t.y); else t.y = -1e20f;
                if (4 * q + 2 < K) tmax = fmaxf(tmax, t.z), tmin = fminf(tmin, t.z); else t.z = -1e20f;
                if (4 * q + 3 < K) tmax = fmaxf(tmax, t.w), tmin = fminf(tmin, t.w); else t.w = -1e20f;
                if (!(t.x == t.x && t.y == t.y && t.z == t.z && t.w == t.w)) tmin = -INFINITY;  // NaN: exact path
                v[r] = t;
            }
            if (i < OTILE_W / 4) reinterpret_cast<uint4*>(o_tile)[i] = make_uint4(0u, 0u, 0u, 0u);
        }
        // one first_ge per lane: half 0 finds the cell's first label column, half 1 its end; the pair swaps
        const int xe = first_ge(cx + half, sx, Wm, w);
        const int xo = __shfl_xor_sync(0xffffffffu, xe, 1);
        const int Xa = half ? xo : xe, Xb = half ? xe : xo;
        const int ye = first_ge(min(cy + half, h), sy, Hm, h);
        const int yo = __shfl_xor_sync(0xffffffffu, ye, 1);
        const int Ya = half ? yo : ye, Yb = half ? ye : yo;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            tmax = fmaxf(tmax, __shfl_xor_sync(0xffffffffu, tmax, o));
            tmin = fminf(tmin, __shfl_xor_sync(0xffffffffu, tmin, o));
        }
        const bool exact = !(tmax - tmin < 60.f);
#pragma unroll
        for (int r = 0; r < 6; ++r) {
            const int i = lane + 32 * r;
            if (i < TILE_F / 4) {
                const int q = i % (KP / 4);
                float4 t = v[r];
                if (4 * q + 0 < K) t.x -= tmax;
                if (4 * q + 1 < K) t.y -= tmax;
                if (4 * q + 2 < K) t.z -= tmax;
                if (4 * q + 3 < K) t.w -= tmax;
                reinterpret_cast<float4*>(s_tile)[i] = t;
            }
        }
        __syncwarp();

        const int ncols = Xb - Xa;  // 0 for cells beyond the map
        const int nc_max = __reduce_max_sync(0xffffffffu, ncols);
        float2 G00[NJ], G01[NJ], G10[NJ], G11[NJ];
#pragma unroll
        for (int q = 0; q < NJ; ++q) G00[q] = G01[q] = G10[q] = G11[q] = make_float2(0.f, 0.f);
        RowCtx rc;
        rc.sx = sx, rc.cxf = (float)cx, rc.fscale = fscale, rc.Xa = Xa, rc.ncols = ncols, rc.nc_max = nc_max, rc.K = K, rc.half = half;
        rc.o_cell = (unsigned)__cvta_generic_to_shared(o_tile + cell * OSTR);
        asm volatile("mov.u32 %0, %0;" : "+r"(rc.o_cell));   // opaque: keeps the compiler from re-deriving it per pixel
        // this lane's slot pairs of the four taps: float2 index 2j + half of each 20-float pixel record
        const float2* t00 = reinterpret_cast<const float2*>(s_tile + cell * KP) + half;
        const float2 *t01 = t00 + KP / 2, *t10 = t00 + TCOLS * (KP / 2), *t11 = t10 + KP / 2;
        const unsigned char* lab_b = lab8 + (size_t)b * Hm * Wm + Xa;
        for (int Y = Ya + rsp; Y < Yb; Y += RS) {
            const float lamy = fminf(fmaxf(sy * (float)Y - (float)cy, 0.f), 1.f);
            rc.lamy = lamy, rc.hy = 1.f - lamy;
            rc.lrow = lab_b + (size_t)Y * Wm;
            const float2 ly2 = make_float2(lamy, lamy), neg1 = make_float2(-1.f, -1.f);
            float2 A[NJ], Bc[NJ];
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                const float2 a = t00[2 * j], bq = t01[2 * j], c = t10[2 * j], d = t11[2 * j];
                const float2 l = __ffma2_rn(ly2, __ffma2_rn(a, neg1, c), a);
                const float2 r = __ffma2_rn(ly2, __ffma2_rn(bq, neg1, d), bq);
                A[j] = l;
                Bc[j] = __ffma2_rn(l, neg1, r);
            }
            if (!exact) row_pixels<false>(A, Bc, rc, G00, G01, G10, G11, lossacc);
            else row_pixels<true>(A, Bc, rc, G00, G01, G10, G11, lossacc);
        }
        __syncwarp();   // the pair's one-hot atomics are complete

        // ---- minus the one-hot weights; the loss gets -<one-hot weights, z'> (every tile element counted once: a lane
        //      counts its left-hand taps, the last cell also its right-hand ones)
        {
            const float inv_fs = 1.f / fscale;
            // a tile element is handled once: by the active cell whose LEFT tap it is, or -- column 16, or the clamped
            // column behind the map's last cell -- as the RIGHT tap of the cell that has no active neighbour
            const bool active = cx < w, lastc = active && (cell == CPW - 1 || cx == w - 1);
            float zy = 0.f;
            const unsigned* o00 = o_tile + cell * OSTR + 2 * half;   // this lane's slots 4j + 2*half, +1 of the four taps
            const unsigned *o01 = o00 + OSTR, *o10 = o00 + TCOLS * OSTR, *o11 = o10 + OSTR;
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                const float2 fa = make_float2((float)o00[4 * j] * inv_fs, (float)o00[4 * j + 1] * inv_fs);
                const float2 fb = make_float2((float)o01[4 * j] * inv_fs, (float)o01[4 * j + 1] * inv_fs);
                const float2 fc = make_float2((float)o10[4 * j] * inv_fs, (float)o10[4 * j + 1] * inv_fs);
                const float2 fd = make_float2((float)o11[4 * j] * inv_fs, (float)o11[4 * j + 1] * inv_fs);
                const float2 sa = t00[2 * j], sb = t01[2 * j], sc = t10[2 * j], sd = t11[2 * j];
                if (active) {
                    zy = fmaf(fa.x, sa.x, fmaf(fa.y, sa.y, zy));
                    zy = fmaf(fc.x, sc.x, fmaf(fc.y, sc.y, zy));
                }
                if (lastc) {
                    zy = fmaf(fb.x, sb.x, fmaf(fb.y, sb.y, zy));
                    zy = fmaf(fd.x, sd.x, fmaf(fd.y, sd.y, zy));
                }
                G00[j].x -= fa.x, G00[j].y -= fa.y;
                G10[j].x -= fc.x, G10[j].y -= fc.y;
                if (lastc) {
                    G01[j].x -= fb.x, G01[j].y -= fb.y;
                    G11[j].x -= fd.x, G11[j].y -= fd.y;
                }
            }
            lossacc -= zy;
        }
        // ---- right-hand taps go to the next cell's lanes (same half: two lanes up); then 8-byte REDs
        const int fyT = cy, fyB = min(cy + 1, h - 1);
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const float2 rt = make_float2(__shfl_up_sync(0xffffffffu, G01[j].x, 2), __shfl_up_sync(0xffffffffu, G01[j].y, 2));
            const float2 rb = make_float2(__shfl_up_sync(0xffffffffu, G11[j].x, 2), __shfl_up_sync(0xffffffffu, G11[j].y, 2));
            if (cell > 0) {
                G00[j].x += rt.x, G00[j].y += rt.y;
                G10[j].x += rb.x, G10[j].y += rb.y;
            }
        }
        if (cx < w) {
            const int fxL = cx, fxR = min(cx + 1, w - 1);
            float2* dT = reinterpret_cast<float2*>(ds_rl + ((size_t)(b * h + fyT) * w + fxL) * KP) + half;
            float2* dB = reinterpret_cast<float2*>(ds_rl + ((size_t)(b * h + fyB) * w + fxL) * KP) + half;
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                if (G00[j].x != 0.f || G00[j].y != 0.f) atomicAdd(dT + 2 * j, G00[j]);
                if (G10[j].x != 0.f || G10[j].y != 0.f) atomicAdd(dB + 2 * j, G10[j]);
            }
            // the right-hand taps of the warp's last cell -- or of the map's last column -- have no lane to go to
            if (cell == CPW - 1 || cx == w - 1) {
                float2* eT = reinterpret_cast<float2*>(ds_rl + ((size_t)(b * h + fyT) * w + fxR) * KP) + half;
                float2* eB = reinterpret_cast<float2*>(ds_rl + ((size_t)(b * h + fyB) * w + fxR) * KP) + half;
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    if (G01[j].x != 0.f || G01[j].y != 0.f) atomicAdd(eT + 2 * j, G01[j]);
                    if (G11[j].x != 0.f || G11[j].y != 0.f) atomicAdd(eB + 2 * j, G11[j]);
                }
            }
        }
    }
    // ---- the block meets once: loss sum and last-CTA ticket
    lossacc = warp_sum(lossacc);
    if (lane == 0) red[wid] = lossacc;
    __syncthreads();
    if (tid == 0) {
        float tot = 0.f;
        for (int i = 0; i < WARPS; ++i) tot += red[i];
        atomicAdd(reinterpret_cast<double*>(ws + PM_WS_LOSS_SUM), (double)tot * 0.6931471805599453);
        __threadfence();
        const unsigned long long ticket = atomicAdd(ws + PM_WS_COUNTER, 1ULL);
        if (ticket == (unsigned long long)gridDim.x - 1) {
            __threadfence();
            unsigned long long V = 0;
            for (int k = 0; k < K; ++k) V += atomicAdd(ws + PM_WS_HIST + k, 0ULL);
            const double sum = __longlong_as_double((long long)atomicAdd(ws + PM_WS_LOSS_SUM, 0ULL));
            out[0] = (float)(sum / (double)V);  // V == 0 -> 0/0 = NaN like torch
            out[1] = (float)(1.0 / ((double)V * (double)temperature));
        }
    }
}

}  // namespace rc
}  // namespace pm

// 0 = launched, positive = CUDA error, -1 = shape outside the fixed-point range of the one-hot tile
int pm_readloss_cells_launch(const float* s, const uint8_t* lab8, float temperature, int B, int h, int w, int Hm, int Wm, int K,
                             float* ds_rl, void* ws, float* out, cudaStream_t st) {
    using namespace pm::rc;
    const float sy = Hm > 1 ? (float)(h - 1) / (float)(Hm - 1) : 0.f;
    const float sx = Wm > 1 ? (float)(w - 1) / (float)(Wm - 1) : 0.f;
    const int rmax = h > 1 ? (Hm - 1) / (h - 1) + 2 : Hm, cmax = w > 1 ? (Wm - 1) / (w - 1) + 2 : Wm;
    const double bound = 4.0 * (double)rmax * (double)cmax;
    int bits = 0;
    while (bits < 30 && (double)(1ull << (bits + 1)) * bound <= 4294967296.0) ++bits;
    if (bits < 16) return -1;
    const float fscale = (float)(1u << bits);
    const int tiles_x = (w + CPW - 1) / CPW;
    long long nitems = (long long)B * h * tiles_x;
    int RS = 1;   // row split: at least ~1.5 waves of 16 warps per SM
    static int sms = 0;
    if (sms == 0 && cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0) != cudaSuccess) sms = 148;
    while (RS < 4 && nitems * RS < 24LL * sms && 4 * (RS * 2) <= rmax - 1) RS *= 2;
    nitems *= RS;
    if (nitems > 0x7fffffffLL) return -1;
    const int grid = (int)((nitems + WARPS - 1) / WARPS);
    readloss_cells_kernel<<<grid, THREADS, 0, st>>>(s, lab8, 1.f / temperature, temperature, h, w, Hm, Wm, K, sy, sx, tiles_x,
                                                    RS, (int)nitems, fscale, ds_rl, (unsigned long long*)ws, out);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}
