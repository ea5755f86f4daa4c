// Feature-cohesion read loss, forward (+ the gradient w.r.t. the similarities, + label histogram).
//
// readloss = CE(bilinear_up(s/T -> [Hm,Wm], align_corners=True), labels; ignore 255), mean over valid
// label pixels (reference memory.py:173-176) -- computed per label pixel on the fly, the [B,K,Hm,Wm]
// logits never exist.
//
// A "cell" (cy,cx) is the set of label pixels whose four bilinear taps are the feature pixels
// (cy,cx),(cy,cx+1),(cy+1,cx),(cy+1,cx+1); inside a cell every logit is bilinear in (lambda_y, lambda_x).
// Two threads (lane pair) own a cell, each half of the K slots (keeps the 4 x K/2 gradient accumulators in
// registers at 2 CTAs/SM); a thread walks the cell's label rows (optionally 1/RS of them), per row forms
// z_k(lambda_x) = A_k + lambda_x * B_k, and per pixel spends K/2 FFMA (packed FFMA2), K/2 ex2, one shuffle
// for the softmax denominator and 4 x K/4 FFMA2 for the tap gradients. Loop bounds are warp-uniform
// (out-of-range pixels are predicated off) so the warp never diverges around the shuffles. Labels are
// fetched a chunk of 8 pixels ahead. The one-hot part of the gradient, the label histogram and the
// "- logit[label]" term of the loss need a dynamic class index: they are run-length accumulated in
// registers and flushed to thread-private shared-memory columns (no atomics). Cells merge into the CTA's tap tile in conflict-free phases; the tile is flushed to ds_rl
// with 16-byte vector REDs (only tile borders are shared between CTAs). The last CTA divides by V.
//
// Softmax stabiliser: the maximum over the cell's 4 taps x K slots bounds every logit in the cell, so it
// is subtracted once per cell (folded into A_k) instead of a per-pixel max; cells whose tap spread is
// large enough for that to underflow (> 60 in log2 units: tiny T or un-normalised queries) additionally
// take the per-pixel max.
#include "pm_common.cuh"
#include "pm_internal.h"

namespace pm {

// cells per CTA along x: template parameter TX = 32, or 16 when a 32-wide tiling would leave >= 16 columns of the
// last tile empty (w = 48, the OS16 shape: 64 thread columns for 48 cells); a warp is 16 lane pairs = 16 cells of one
// cell row in both cases, so all its lanes share the cell row and the row split.
constexpr int RL_THREADS = 256;    // 128 cells x 2 slot halves
constexpr int RL_CHUNK = 3;        // label pixels fetched ahead (cells are 8-9 / 16-17 pixels wide: 3 divides 9 and 18)

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float lg2_approx(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ int bil_index(float scale, int dst, int n_in) {
    int i0 = (int)(scale * (float)dst);
    return i0 > n_in - 1 ? n_in - 1 : i0;
}
// smallest dst in [0, n_out] whose bilinear source index is >= c
__device__ __forceinline__ int first_ge(int c, float scale, int n_out, int n_in) {
    if (c <= 0) return 0;
    if (c > n_in - 1 || scale <= 0.f) return n_out;
    int y = (int)ceilf((float)c / scale);
    y = max(0, min(y, n_out));
    while (y > 0 && bil_index(scale, y - 1, n_in) >= c) --y;
    while (y < n_out && bil_index(scale, y, n_in) < c) ++y;
    return y;
}

// ORD = true (ordered instantiation): ds_rl is the tile scratch and `out` the per-CTA loss partials; each CTA stores its
// whole tap tile and its loss to slot [blockIdx.x] instead of adding them with atomics (readloss_gather combines them)
template <int KP, int RL_TX, bool ORD = false>
__global__ void __launch_bounds__(RL_THREADS, 2)
    readloss_kernel(const float* __restrict__ s, const long long* __restrict__ labels, float inv_T, float temperature,
                    int h, int w, int Hm, int Wm, int K, float sy, float sx, int RS, int TYC, int tiles_x, int tiles_y,
                    float* __restrict__ ds_rl, unsigned long long* __restrict__ ws, float* __restrict__ out) {
    constexpr int KH = KP / 2, NH2 = KH / 2, NT = RL_THREADS, RL_LDX = RL_TX + 1;
    extern __shared__ __align__(16) float smem[];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int tile_elems = (TYC + 1) * RL_LDX * KP;
    float* s_tile = smem;                                         // [(TYC+1)][33][KP]
    float* ds_tile = s_tile + tile_elems;                         // same shape
    float* priv = ds_tile + tile_elems;                           // [4][KH][NT] one-hot tap weights
    int* pcnt = reinterpret_cast<int*>(priv + 4 * KH * NT);       // [KP][NT/2] label counts (slot-half 0 threads)
    int* hist_sm = pcnt + KP * (NT / 2);                          // [KP]
    float* red = reinterpret_cast<float*>(hist_sm + KP);          // [8]

    int bid = blockIdx.x;
    const int tx_i = bid % tiles_x;
    bid /= tiles_x;
    const int ty_i = bid % tiles_y, b = bid / tiles_y;
    const int fy0 = ty_i * TYC, fx0 = tx_i * RL_TX;

    for (int i = tid; i < tile_elems; i += NT) {
        int e = i / KP, k = i - e * KP;
        int ty = e / RL_LDX, tx = e - ty * RL_LDX;
        int fy = min(fy0 + ty, h - 1), fx = min(fx0 + tx, w - 1);
        s_tile[i] = __ldg(s + ((size_t)(b * h + fy) * w + fx) * KP + k);
        ds_tile[i] = 0.f;
    }
    for (int i = tid; i < 4 * KH * NT; i += NT) priv[i] = 0.f;
    for (int i = tid; i < KP * (NT / 2); i += NT) pcnt[i] = 0;
    if (tid < KP) hist_sm[tid] = 0;
    __syncthreads();

    const int half = tid & 1, pair = tid >> 1;
    const int cxl = pair % RL_TX, rest = pair / RL_TX;  // rest in [0, TYC*RS)
    const int cyl = rest / RS, split = rest - cyl * RS;
    const int cy = fy0 + cyl, cx = fx0 + cxl;
    const bool active = (cy < h) && (cx < w);
    const int ly0 = cyl, ly1 = min(cy + 1, h - 1) - fy0;
    const int lx0 = cxl, lx1 = min(cx + 1, w - 1) - fx0;
    const int k0 = half * KH;  // first slot of this thread

    float2 G00[NH2], G01[NH2], G10[NH2], G11[NH2];
#pragma unroll
    for (int i = 0; i < NH2; ++i) G00[i] = G01[i] = G10[i] = G11[i] = make_float2(0.f, 0.f);
    float lossacc = 0.f;  // in log2 units
    float* pv = priv + tid;        // element (tap, kk) at pv[(tap*KH + kk)*NT]
    int* pc = pcnt + pair;         // element k at pc[k*(NT/2)]

    // Loop bounds are made warp-uniform (max over the lanes, out-of-range pixels predicated off) so the
    // whole warp stays converged and the pair shuffles can use the full mask.
    int Ya = 0, Yb = 0, Xa = 0, Xb = 0;
    if (active) {
        Ya = first_ge(cy, sy, Hm, h), Yb = first_ge(cy + 1, sy, Hm, h);
        Xa = first_ge(cx, sx, Wm, w), Xb = first_ge(cx + 1, sx, Wm, w);
    }
    const int nr_lane = (Yb - Ya - split + RS - 1) / RS;  // rows this thread owns (<= 0: none)
    const int nr_max = __reduce_max_sync(0xffffffffu, max(nr_lane, 0));
    const int nc_max = __reduce_max_sync(0xffffffffu, Xb - Xa);
    const float c2 = inv_T * 1.4426950408889634f;
    // taps of this cell (inactive lanes read tap (0,0): finite values, results never merged)
    const int tl0 = active ? ly0 : 0, tl1 = active ? ly1 : 0, tx0 = active ? lx0 : 0, tx1 = active ? lx1 : 0;
    const float* t00 = s_tile + (tl0 * RL_LDX + tx0) * KP + k0;
    const float* t01 = s_tile + (tl0 * RL_LDX + tx1) * KP + k0;
    const float* t10 = s_tile + (tl1 * RL_LDX + tx0) * KP + k0;
    const float* t11 = s_tile + (tl1 * RL_LDX + tx1) * KP + k0;
    float shift;  // softmax stabiliser (log2 units): max over the cell's taps and slots
    bool pxmax;
    {
        float m = -INFINITY, n = INFINITY;
#pragma unroll
        for (int i = 0; i < KH; ++i) {
            if (k0 + i < K) {
                m = fmaxf(m, fmaxf(fmaxf(t00[i], t01[i]), fmaxf(t10[i], t11[i])));
                n = fminf(n, fminf(fminf(t00[i], t01[i]), fminf(t10[i], t11[i])));
            }
        }
        shift = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 1)) * c2;
        const float lo = fminf(n, __shfl_xor_sync(0xffffffffu, n, 1)) * c2;
        // spread too large for the per-cell stabiliser (tiny T / un-normalised queries; also NaN/inf)
        pxmax = __any_sync(0xffffffffu, !(shift - lo < 60.f));
    }
    // run-length state of the one-hot / histogram part
    int cur = -1, cnt = 0;
    float o00 = 0.f, o01 = 0.f, o10 = 0.f, o11 = 0.f;
    const long long* lab_b = labels + (size_t)b * Hm * Wm;
    const float cxf = (float)cx, cyf = (float)cy;

    for (int r = 0; r < nr_max; ++r) {
        const int Y = Ya + split + r * RS;
        const bool rowok = active && Y < Yb;
        const float lamy = fminf(fmaxf(sy * (float)Y - cyf, 0.f), 1.f);
        const float hy = 1.f - lamy;
        float2 A[NH2], Bc[NH2];
#pragma unroll
        for (int i = 0; i < NH2; ++i) {
            const float2 v00 = reinterpret_cast<const float2*>(t00)[i], v01 = reinterpret_cast<const float2*>(t01)[i];
            const float2 v10 = reinterpret_cast<const float2*>(t10)[i], v11 = reinterpret_cast<const float2*>(t11)[i];
            float l0 = fmaf(lamy, v10.x - v00.x, v00.x), l1 = fmaf(lamy, v11.x - v01.x, v01.x);
            A[i].x = fmaf(l0, c2, -shift), Bc[i].x = (l1 - l0) * c2;
            l0 = fmaf(lamy, v10.y - v00.y, v00.y), l1 = fmaf(lamy, v11.y - v01.y, v01.y);
            A[i].y = fmaf(l0, c2, -shift), Bc[i].y = (l1 - l0) * c2;
            if (k0 + 2 * i >= K) A[i].x = -INFINITY, Bc[i].x = 0.f;
            if (k0 + 2 * i + 1 >= K) A[i].y = -INFINITY, Bc[i].y = 0.f;
        }
        // labels are interpreted by their low 32 bits (little endian int64)
        const int* lrow = reinterpret_cast<const int*>(lab_b + (size_t)(rowok ? Y : 0) * Wm + Xa);
        const int ncols = rowok ? Xb - Xa : 0;
        // per-row accumulators of p*(1-lambda_x) and p*lambda_x; split over the two tap rows at row end
        float2 R0[NH2], R1[NH2];
#pragma unroll
        for (int q = 0; q < NH2; ++q) R0[q] = R1[q] = make_float2(0.f, 0.f);
        float ox0 = 0.f, ox1 = 0.f;  // one-hot counterparts for the current run (this row only)
        for (int X0 = 0; X0 < nc_max; X0 += RL_CHUNK) {
            int lab[RL_CHUNK];
#pragma unroll
            for (int i = 0; i < RL_CHUNK; ++i) lab[i] = (X0 + i < ncols) ? __ldg(lrow + 2 * (X0 + i)) : -1;
#pragma unroll
            for (int i = 0; i < RL_CHUNK; ++i) {
                if (X0 + i >= nc_max) break;  // warp-uniform
                const bool ok = X0 + i < ncols;
                const int labi = lab[i];
                const unsigned ucls = (unsigned)labi;
                const bool valid = ok && ucls < (unsigned)K;
                const int cls = (int)min(ucls, (unsigned)K);
                const float lamx = fminf(fmaxf(sx * (float)(Xa + X0 + i) - cxf, 0.f), 1.f);
                float2 e[NH2];
#pragma unroll
                for (int q = 0; q < NH2; ++q) e[q] = __ffma2_rn(make_float2(lamx, lamx), Bc[q], A[q]);
                float pshift = shift;
                if (pxmax) {  // warp-uniform
                    float m = -INFINITY;
#pragma unroll
                    for (int q = 0; q < NH2; ++q) m = fmaxf(m, fmaxf(e[q].x, e[q].y));
                    m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 1));
                    pshift += m;
#pragma unroll
                    for (int q = 0; q < NH2; ++q) e[q].x -= m, e[q].y -= m;
                }
                float2 sum2 = make_float2(0.f, 0.f);
#pragma unroll
                for (int q = 0; q < NH2; ++q) {
                    e[q].x = ex2_approx(e[q].x);
                    e[q].y = ex2_approx(e[q].y);
                    sum2 = __fadd2_rn(sum2, e[q]);
                }
                float sum = sum2.x + sum2.y;
                sum += __shfl_xor_sync(0xffffffffu, sum, 1);
                if (valid && half == 0) lossacc += pshift + lg2_approx(sum);
                const float inv = valid ? rcp_approx(sum) : 0.f;
                const float hx = 1.f - lamx;
                const float ihx = inv * hx, ilx = inv * lamx;
#pragma unroll
                for (int q = 0; q < NH2; ++q) {
                    R0[q] = __ffma2_rn(e[q], make_float2(ihx, ihx), R0[q]);
                    R1[q] = __ffma2_rn(e[q], make_float2(ilx, ilx), R1[q]);
                }
                // one-hot part + histogram: run-length accumulate, flush to the private columns on a change
                if (ok && cls != cur) {
                    if (cur >= 0) {
                        if (half == 0) pc[cur * (NT / 2)] += cnt;
                        const int kk = cur - k0;
                        if (kk >= 0 && kk < KH && cur < K) {
                            pv[(0 * KH + kk) * NT] += fmaf(hy, ox0, o00);
                            pv[(1 * KH + kk) * NT] += fmaf(hy, ox1, o01);
                            pv[(2 * KH + kk) * NT] += fmaf(lamy, ox0, o10);
                            pv[(3 * KH + kk) * NT] += fmaf(lamy, ox1, o11);
                        }
                    }
                    cnt = 0;
                    o00 = o01 = o10 = o11 = 0.f;
                    ox0 = ox1 = 0.f;
                    cur = cls;
                }
                if (ok && !valid && labi != PM_IGNORE_LABEL && half == 0) atomicAdd(ws + PM_WS_BAD, 1ULL);
                cnt += ok ? 1 : 0;
                ox0 += ok ? hx : 0.f;
                ox1 += ok ? lamx : 0.f;
            }
        }
        // end of row: fold the row accumulators into the four taps
        o00 = fmaf(hy, ox0, o00), o01 = fmaf(hy, ox1, o01);
        o10 = fmaf(lamy, ox0, o10), o11 = fmaf(lamy, ox1, o11);
        {
            const float2 hy2 = make_float2(hy, hy), ly2 = make_float2(lamy, lamy);
#pragma unroll
            for (int q = 0; q < NH2; ++q) {
                G00[q] = __ffma2_rn(R0[q], hy2, G00[q]);
                G01[q] = __ffma2_rn(R1[q], hy2, G01[q]);
                G10[q] = __ffma2_rn(R0[q], ly2, G10[q]);
                G11[q] = __ffma2_rn(R1[q], ly2, G11[q]);
            }
        }
    }
    if (active) {
        if (cur >= 0) {
            if (half == 0) pc[cur * (NT / 2)] += cnt;
            const int kk = cur - k0;
            if (kk >= 0 && kk < KH && cur < K) {
                pv[(0 * KH + kk) * NT] += o00;
                pv[(1 * KH + kk) * NT] += o01;
                pv[(2 * KH + kk) * NT] += o10;
                pv[(3 * KH + kk) * NT] += o11;
            }
        }
        // minus the logit of the labelled class: sum_px z_y = c2 * sum_{tap,k} onehot_weight[tap][k] * tap[k];
        // then subtract the one-hot part from the tap gradients
        float zy = 0.f;
#pragma unroll
        for (int q = 0; q < NH2; ++q) {
            const float a0 = pv[(0 * KH + 2 * q) * NT], a1 = pv[(0 * KH + 2 * q + 1) * NT];
            const float b0 = pv[(1 * KH + 2 * q) * NT], b1 = pv[(1 * KH + 2 * q + 1) * NT];
            const float c0 = pv[(2 * KH + 2 * q) * NT], c1 = pv[(2 * KH + 2 * q + 1) * NT];
            const float d0 = pv[(3 * KH + 2 * q) * NT], d1 = pv[(3 * KH + 2 * q + 1) * NT];
            zy = fmaf(a0, t00[2 * q], fmaf(a1, t00[2 * q + 1], zy));
            zy = fmaf(b0, t01[2 * q], fmaf(b1, t01[2 * q + 1], zy));
            zy = fmaf(c0, t10[2 * q], fmaf(c1, t10[2 * q + 1], zy));
            zy = fmaf(d0, t11[2 * q], fmaf(d1, t11[2 * q + 1], zy));
            G00[q].x -= a0, G00[q].y -= a1;
            G01[q].x -= b0, G01[q].y -= b1;
            G10[q].x -= c0, G10[q].y -= c1;
            G11[q].x -= d0, G11[q].y -= d1;
        }
        lossacc = fmaf(-c2, zy, lossacc);
        // fold degenerate taps (last row / column clamp onto themselves)
        if (ly1 == ly0) {
#pragma unroll
            for (int q = 0; q < NH2; ++q) {
                G00[q] = __fadd2_rn(G00[q], G10[q]), G01[q] = __fadd2_rn(G01[q], G11[q]);
                G10[q] = G11[q] = make_float2(0.f, 0.f);
            }
        }
        if (lx1 == lx0) {
#pragma unroll
            for (int q = 0; q < NH2; ++q) {
                G00[q] = __fadd2_rn(G00[q], G01[q]), G10[q] = __fadd2_rn(G10[q], G11[q]);
                G01[q] = G11[q] = make_float2(0.f, 0.f);
            }
        }
    } else {
        lossacc = 0.f;
    }

    // merge into the tap tile: within one (tap, split) phase every active thread owns distinct addresses
    for (int sp = 0; sp < RS; ++sp) {
#pragma unroll
        for (int tap = 0; tap < 4; ++tap) {
            const bool fold = (tap >= 2 && ly1 == ly0) || ((tap & 1) && lx1 == lx0);
            if (active && split == sp && !fold) {
                const int ly = (tap >= 2) ? ly1 : ly0, lx = (tap & 1) ? lx1 : lx0;
                float2* dst = reinterpret_cast<float2*>(ds_tile + (ly * RL_LDX + lx) * KP + k0);
#pragma unroll
                for (int q = 0; q < NH2; ++q) {
                    const float2 g = tap == 0 ? G00[q] : tap == 1 ? G01[q] : tap == 2 ? G10[q] : G11[q];
                    float2 v = dst[q];
                    v.x += g.x, v.y += g.y;
                    dst[q] = v;
                }
            }
            __syncthreads();
        }
    }
    if constexpr (ORD) {
        float4* dst = reinterpret_cast<float4*>(ds_rl + (size_t)blockIdx.x * tile_elems);
        for (int i = tid; i < tile_elems / 4; i += NT) dst[i] = reinterpret_cast<const float4*>(ds_tile)[i];
    } else {
        // flush taps that exist (clamped duplicates were folded and stay zero)
        for (int i = tid; i < tile_elems / 4; i += NT) {
            int e = i / (KP / 4), q = i - e * (KP / 4);
            int ty = e / RL_LDX, tx = e - ty * RL_LDX;
            int fy = fy0 + ty, fx = fx0 + tx;
            if (fy < h && fx < w) {
                float4 v = reinterpret_cast<const float4*>(ds_tile)[i];
                if (v.x != 0.f || v.y != 0.f || v.z != 0.f || v.w != 0.f)
                    atomicAdd(reinterpret_cast<float4*>(ds_rl + ((size_t)(b * h + fy) * w + fx) * KP) + q, v);
            }
        }
    }
    // label histogram + loss sum
    for (int k = 0; k <= K; ++k) {
        int c = __reduce_add_sync(0xffffffffu, half == 0 ? pc[k * (NT / 2)] : 0);
        if (lane == 0 && c != 0) atomicAdd(hist_sm + k, c);
    }
    lossacc = warp_sum(lossacc);
    if (lane == 0) red[wid] = lossacc;
    __syncthreads();
    if (tid == 0) {
        float tot = 0.f;
        for (int i = 0; i < NT / 32; ++i) tot += red[i];
        if constexpr (ORD) out[blockIdx.x] = tot;
        else atomicAdd(reinterpret_cast<double*>(ws + PM_WS_LOSS_SUM), (double)tot * 0.6931471805599453);
    }
    if (tid <= K && hist_sm[tid] != 0) atomicAdd(ws + PM_WS_HIST + tid, (unsigned long long)hist_sm[tid]);
    if constexpr (ORD) return;
    // last CTA: readloss = loss_sum / V ; scale = 1 / (V*T)
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        unsigned long long ticket = atomicAdd(ws + PM_WS_COUNTER, 1ULL);
        if (ticket == (unsigned long long)gridDim.x - 1) {
            __threadfence();
            unsigned long long V = 0;
            for (int k = 0; k < K; ++k) V += atomicAdd(ws + PM_WS_HIST + k, 0ULL);
            double sum = __longlong_as_double((long long)atomicAdd(ws + PM_WS_LOSS_SUM, 0ULL));
            out[0] = (float)(sum / (double)V);  // V == 0 -> 0/0 = NaN like torch
            out[1] = (float)(1.0 / ((double)V * (double)temperature));
        }
    }
}

// row-split factor and tiling of the first kernel (shared by the launch and the ordered variant's scratch size)
static void rl_tiling(int B, int h, int w, int Hm, int RL_TX, int* RS_out, int* TYC_out, int* tiles_x, int* tiles_y) {
    // row-split factor: enough threads to fill the chip when there are few cells
    const long long cells = (long long)B * h * w;
    const int rows_per_cell = h > 1 ? (Hm + h - 2) / (h - 1) : Hm;
    int RS = 1;
    while (RS < 4 && cells * RS * 2 < 148LL * 512 && RS * 2 <= rows_per_cell) RS *= 2;
    const int TYC = (RL_THREADS / 2 / RL_TX) / RS;
    *RS_out = RS, *TYC_out = TYC;
    *tiles_x = (w + RL_TX - 1) / RL_TX, *tiles_y = (h + TYC - 1) / TYC;
}

// cells per CTA along x (see RL_THREADS)
static int rl_tx(int w) { return (w + 31) / 32 * 32 - w >= 16 ? 16 : 32; }

template <int KP, int RL_TX, bool ORD>
static int launch_readloss_tx(const float* s, const long long* labels, float temperature, int B, int h, int w, int Hm,
                           int Wm, int K, float* ds_rl, unsigned long long* ws, float* out, cudaStream_t st) {
    // PyTorch's align_corners scale: (in-1)/(out-1) in fp32, 0 when out == 1
    const float sy = Hm > 1 ? (float)(h - 1) / (float)(Hm - 1) : 0.f;
    const float sx = Wm > 1 ? (float)(w - 1) / (float)(Wm - 1) : 0.f;
    int RS, TYC, tiles_x, tiles_y;
    rl_tiling(B, h, w, Hm, RL_TX, &RS, &TYC, &tiles_x, &tiles_y);
    const size_t smem = sizeof(float) * ((size_t)2 * (TYC + 1) * (RL_TX + 1) * KP + (size_t)4 * (KP / 2) * RL_THREADS +
                                         (size_t)KP * (RL_THREADS / 2) + KP + 8);
    const long long grid = (long long)B * tiles_x * tiles_y;
    if (grid > 0x7fffffffLL) return PM_ERR_SHAPE;
    auto kern = readloss_kernel<KP, RL_TX, ORD>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    kern<<<(int)grid, RL_THREADS, smem, st>>>(s, labels, 1.f / temperature, temperature, h, w, Hm, Wm, K, sy, sx, RS,
                                              TYC, tiles_x, tiles_y, ds_rl, ws, out);
    e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

template <int KP, bool ORD = false>
static int launch_readloss(const float* s, const long long* labels, float temperature, int B, int h, int w, int Hm,
                           int Wm, int K, float* ds_rl, unsigned long long* ws, float* out, cudaStream_t st) {
    if (rl_tx(w) == 16) return launch_readloss_tx<KP, 16, ORD>(s, labels, temperature, B, h, w, Hm, Wm, K, ds_rl, ws, out, st);
    return launch_readloss_tx<KP, 32, ORD>(s, labels, temperature, B, h, w, Hm, Wm, K, ds_rl, ws, out, st);
}

long long readloss8_scratch_bytes(int B, int h, int w, int Hm, int Wm);   // pm_readloss8.cu

struct RlGeometry {
    int TX, TYC, tiles_x, tiles_y;
    long long grid, tile_elems;
};
static RlGeometry rl_geometry(int B, int h, int w, int Hm, int KP) {
    RlGeometry g;
    int RS;
    g.TX = rl_tx(w);
    rl_tiling(B, h, w, Hm, g.TX, &RS, &g.TYC, &g.tiles_x, &g.tiles_y);
    g.grid = (long long)B * g.tiles_x * g.tiles_y;
    g.tile_elems = (long long)(g.TYC + 1) * (g.TX + 1) * KP;
    return g;
}

}  // namespace pm

extern "C" int pm_readloss_fwd(const float* s, const int64_t* labels, float temperature, int B, int h, int w, int Hm,
                               int Wm, int K, float* ds_rl, void* ws, float* out, void* stream) {
    if (!s || !labels || !ds_rl || !ws || !out) return PM_ERR_NULL;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (B <= 0 || h <= 0 || w <= 0 || Hm <= 0 || Wm <= 0 || !(temperature > 0.f)) return PM_ERR_SHAPE;
    if (((uintptr_t)s & 15) || ((uintptr_t)ds_rl & 15) || ((uintptr_t)ws & 7)) return PM_ERR_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    const long long* lab = (const long long*)labels;
    unsigned long long* w64 = (unsigned long long*)ws;
    if (K <= 19) return pm::launch_readloss<20>(s, lab, temperature, B, h, w, Hm, Wm, K, ds_rl, w64, out, st);
    return pm::launch_readloss<32>(s, lab, temperature, B, h, w, Hm, Wm, K, ds_rl, w64, out, st);
}

extern "C" int pm_readloss_scratch_bytes(int B, int h, int w, int Hm, int Wm, int K, int packed) {
    if (K < 1 || K > (packed ? 19 : 31)) return PM_ERR_SLOTS;
    if (B <= 0 || h <= 0 || w <= 0 || Hm <= 0 || Wm <= 0) return PM_ERR_SHAPE;
    long long bytes;
    if (packed) {
        bytes = pm::readloss8_scratch_bytes(B, h, w, Hm, Wm);
    } else {
        const pm::RlGeometry g = pm::rl_geometry(B, h, w, Hm, K <= 19 ? 20 : 32);
        bytes = (g.grid * g.tile_elems + (g.grid + 3) / 4 * 4) * (long long)sizeof(float);
    }
    return bytes > 0x7fffffffLL ? PM_ERR_SHAPE : (int)bytes;
}

extern "C" int pm_readloss_fwd_ordered(const float* s, const int64_t* labels, float temperature, int B, int h, int w, int Hm,
                                       int Wm, int K, float* ds_rl, void* ws, float* out, float* scratch, void* stream) {
    if (!s || !labels || !ds_rl || !ws || !out || !scratch) return PM_ERR_NULL;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (B <= 0 || h <= 0 || w <= 0 || Hm <= 0 || Wm <= 0 || !(temperature > 0.f)) return PM_ERR_SHAPE;
    if (((uintptr_t)s & 15) || ((uintptr_t)ds_rl & 15) || ((uintptr_t)ws & 7) || ((uintptr_t)scratch & 15)) return PM_ERR_ALIGN;
    const cudaStream_t st = (cudaStream_t)stream;
    const long long* lab = (const long long*)labels;
    unsigned long long* w64 = (unsigned long long*)ws;
    const int KP = K <= 19 ? 20 : 32;
    const pm::RlGeometry g = pm::rl_geometry(B, h, w, Hm, KP);
    if (g.grid > 0x7fffffffLL) return PM_ERR_SHAPE;
    float* lossp = scratch + (size_t)g.grid * g.tile_elems;
    const int rc = KP == 20 ? pm::launch_readloss<20, true>(s, lab, temperature, B, h, w, Hm, Wm, K, scratch, w64, lossp, st)
                            : pm::launch_readloss<32, true>(s, lab, temperature, B, h, w, Hm, Wm, K, scratch, w64, lossp, st);
    if (rc) return rc;
    return pm::readloss_gather(scratch, lossp, (int)g.grid, B, h, w, KP, g.TYC, g.TX, g.tiles_x, g.tiles_y, K, temperature,
                               ds_rl, w64, out, st);
}
