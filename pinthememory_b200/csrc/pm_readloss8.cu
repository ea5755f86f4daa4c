// Feature-cohesion read loss on the packed uint8 class map (pm_labels_pack), second-generation kernel.
//
// readloss = CE(bilinear_up(s/T -> [Hm,Wm], align_corners=True), labels; ignore 255), mean over valid label pixels
// (reference memory.py:173-176), plus d(loss_sum)/d(s/T) scattered back to the feature pixels -- computed per label
// pixel on the fly, the [B,K,Hm,Wm] logits never exist. Same cell decomposition as pm_readloss.cu (a "cell" = the
// label pixels whose four bilinear taps are feature pixels (cy,cx)..(cy+1,cx+1)); what changed is the work per pixel:
//   * ONE thread owns a cell with all KP = 20 slots in registers (the first kernel paired two threads per cell and
//     paid the label logic, the lambda arithmetic and a shuffle twice per pixel);
//   * inside a cell row every logit is linear in lambda_x, and lambda_x advances by the constant `sx` per label pixel,
//     so exp2(z_k) is a GEOMETRIC sequence along the row: E_k <- E_k * r_k with r_k = exp2(c * sx * B_k). Two `ex2`
//     per slot per ROW replace one per slot per PIXEL (the MUFU pipe is 16 lanes/clk/SM: 20 per pixel was a 20 us
//     floor on its own) and the FFMA that formed the exponent disappears;
//   * labels are one byte per pixel from the packed map, the histogram / valid count / bad-label count come from the
//     pack pass, so the per-pixel label work is a byte load, a compare and the run-length bookkeeping of the one-hot
//     term.
// Per pixel that is ~60 instructions in one thread instead of ~2 x 91 (363 thread-instructions per label pixel measured
// on the first kernel, profiles/r1f_ncu_full.txt). The exact per-pixel path is kept for cells whose tap spread is too
// large for the per-cell stabiliser (tiny temperatures, un-normalised logits of the head's main loss).
//
// Accuracy of the recurrence: ex2.approx is 2^-22 relative and every step multiplies, so after i steps the error of a
// probability is ~ (i + 1) * 2.4e-7 (i <= 8 at output stride 8, <= 16 at stride 16); measured against the oracle the
// loss and ds_rl stay below 3e-6 (tests/test_gpu_parity.py). The weights lambda_x / lambda_y themselves are computed
// exactly as PyTorch does (fp32 `scale * dst`, floor, clamp).
#include "pm_common.cuh"
#include "pm_internal.h"

namespace pm {

constexpr int RL8_THREADS = 128;  // one cell (or one row-split of a cell) per thread; 2 CTAs per SM (249 registers) so that
                                  // one CTA's tile load / merge / flush phases overlap the other's label loop
constexpr int RL8_TX = 32;        // cells per CTA along x (a warp = 32 cells of one cell row, same row split)
constexpr int RL8_KP = 20;        // padded slot count of the score rows (K <= 19)

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
__device__ __forceinline__ int bil_index8(float scale, int dst, int n_in) {
    int i0 = (int)(scale * (float)dst);
    return i0 > n_in - 1 ? n_in - 1 : i0;
}
// smallest dst in [0, n_out] whose bilinear source index is >= c
__device__ __forceinline__ int first_ge8(int c, float scale, int n_out, int n_in) {
    if (c <= 0) return 0;
    if (c > n_in - 1 || scale <= 0.f) return n_out;
    int y = (int)ceilf((float)c / scale);
    y = max(0, min(y, n_out));
    while (y > 0 && bil_index8(scale, y - 1, n_in) >= c) --y;
    while (y < n_out && bil_index8(scale, y, n_in) < c) ++y;
    return y;
}

struct RunState {  // run-length state of the one-hot term: current class and its tap weights so far
    int cur;
    float o00, o01, o10, o11;
};
struct CellCtx {
    const float2 *t00, *t01, *t10, *t11;  // the cell's four taps in the shared-memory tile
    const unsigned char* lab_b;
    int Ya, Yb, Xa, Xb, split, RS, Wm, K, nr_max, nc_max;
    bool active;
    float sx, sy, cxf, cyf, c2, shift;
};

constexpr int RL8_CHUNK = 3;  // label pixels per unrolled group (cells are 8-9 / 16-17 pixels wide: 3 divides 9 and 18)

// All label rows of one cell (or of its row split). EXACT = false: geometric recurrence along the row; EXACT = true:
// per-pixel exponent, per-pixel maximum (cells whose tap spread defeats the per-cell stabiliser). Each group of
// RL8_CHUNK pixels first runs the branch-free softmax part for all its pixels (independent dependency chains for the
// scheduler to interleave), then the run-length bookkeeping of the one-hot term, which branches.
template <bool EXACT>
__device__ __forceinline__ void cell_rows(const CellCtx& c, RunState& rs, float* __restrict__ pv, float2 (&G00)[RL8_KP / 2],
                                          float2 (&G01)[RL8_KP / 2], float2 (&G10)[RL8_KP / 2], float2 (&G11)[RL8_KP / 2],
                                          float& lossacc) {
    constexpr int KP = RL8_KP, NH = KP / 2, NT = RL8_THREADS;
    const int K = c.K;
    const float lam_first = fminf(fmaxf(c.sx * (float)c.Xa - c.cxf, 0.f), 1.f);
    for (int r = 0; r < c.nr_max; ++r) {
        const int Y = c.Ya + c.split + r * c.RS;
        const bool rowok = c.active && Y < c.Yb;
        const float lamy = fminf(fmaxf(c.sy * (float)Y - c.cyf, 0.f), 1.f);
        const float hy = 1.f - lamy;
        // z_k(lambda_x) = A_k + lambda_x * B_k (log2 units, stabilised). EXACT: E = A, Rt = B. Otherwise E = exp2(z) at
        // the row's first pixel and Rt = exp2(sx * B), the per-pixel ratio.
        float2 E[NH], Rt[NH];
#pragma unroll
        for (int i = 0; i < NH; ++i) {
            const float2 v00 = c.t00[i], v01 = c.t01[i], v10 = c.t10[i], v11 = c.t11[i];
            float l0 = fmaf(lamy, v10.x - v00.x, v00.x), l1 = fmaf(lamy, v11.x - v01.x, v01.x);
            float Ax = fmaf(l0, c.c2, -c.shift), Bx = (l1 - l0) * c.c2;
            l0 = fmaf(lamy, v10.y - v00.y, v00.y), l1 = fmaf(lamy, v11.y - v01.y, v01.y);
            float Ay = fmaf(l0, c.c2, -c.shift), By = (l1 - l0) * c.c2;
            if (2 * i >= K) Ax = -INFINITY, Bx = 0.f;
            if (2 * i + 1 >= K) Ay = -INFINITY, By = 0.f;
            if (!EXACT) {
                E[i] = make_float2(ex2a(fmaf(lam_first, Bx, Ax)), ex2a(fmaf(lam_first, By, Ay)));
                Rt[i] = make_float2(ex2a(c.sx * Bx), ex2a(c.sx * By));
            } else {
                E[i] = make_float2(Ax, Ay);
                Rt[i] = make_float2(Bx, By);
            }
        }
        const unsigned char* lrow = c.lab_b + (size_t)(rowok ? Y : 0) * c.Wm + c.Xa;
        const int ncols = rowok ? c.Xb - c.Xa : 0;
        float2 R0[NH], R1[NH];  // row accumulators of p*(1-lambda_x) and p*lambda_x
#pragma unroll
        for (int q = 0; q < NH; ++q) R0[q] = R1[q] = make_float2(0.f, 0.f);
        float ox0 = 0.f, ox1 = 0.f;  // one-hot counterparts for the current run (this row only)
        int labn[RL8_CHUNK];        // labels of the NEXT group (fetched one group ahead)
#pragma unroll
        for (int i = 0; i < RL8_CHUNK; ++i) labn[i] = (i < ncols) ? (int)__ldg(lrow + i) : 255;
        for (int X0 = 0; X0 < c.nc_max; X0 += RL8_CHUNK) {   // warp-uniform; pixels past a lane's row are predicated off
            int lab[RL8_CHUNK];
            float lamx[RL8_CHUNK], hx[RL8_CHUNK];
#pragma unroll
            for (int i = 0; i < RL8_CHUNK; ++i) {
                lab[i] = labn[i];
                const int xn = X0 + RL8_CHUNK + i;
                labn[i] = (xn < ncols) ? (int)__ldg(lrow + xn) : 255;
                lamx[i] = fminf(fmaxf(c.sx * (float)(c.Xa + X0 + i) - c.cxf, 0.f), 1.f);
                hx[i] = 1.f - lamx[i];
            }
            // ---- softmax part, branch-free
#pragma unroll
            for (int i = 0; i < RL8_CHUNK; ++i) {
                const bool valid = lab[i] < K;  // 0..K-1 real class; K = ignore; 255 = outside this lane's row
                float pshift = c.shift;
                float2 e[NH];
                if (EXACT) {
                    float m = -INFINITY;
#pragma unroll
                    for (int q = 0; q < NH; ++q) {
                        e[q] = __ffma2_rn(make_float2(lamx[i], lamx[i]), Rt[q], E[q]);
                        m = fmaxf(m, fmaxf(e[q].x, e[q].y));
                    }
                    pshift += m;
#pragma unroll
                    for (int q = 0; q < NH; ++q) e[q] = make_float2(ex2a(e[q].x - m), ex2a(e[q].y - m));
                }
                const float2* ev = EXACT ? e : E;
                float2 s01 = __fadd2_rn(ev[0], ev[1]), s23 = __fadd2_rn(ev[2], ev[3]), s45 = __fadd2_rn(ev[4], ev[5]);
                float2 s67 = __fadd2_rn(ev[6], ev[7]), s89 = __fadd2_rn(ev[8], ev[9]);
                s01 = __fadd2_rn(s01, s23), s45 = __fadd2_rn(s45, s67);
                s01 = __fadd2_rn(__fadd2_rn(s01, s45), s89);
                const float sum = s01.x + s01.y;
                if (valid) lossacc += pshift + lg2a(sum);
                const float inv = valid ? rcpa(sum) : 0.f;
                const float2 ihx = make_float2(inv * hx[i], inv * hx[i]), ilx = make_float2(inv * lamx[i], inv * lamx[i]);
#pragma unroll
                for (int q = 0; q < NH; ++q) {
                    R0[q] = __ffma2_rn(ev[q], ihx, R0[q]);
                    R1[q] = __ffma2_rn(ev[q], ilx, R1[q]);
                }
                if (!EXACT) {
#pragma unroll
                    for (int q = 0; q < NH; ++q) E[q] = __fmul2_rn(E[q], Rt[q]);
                }
            }
            // ---- one-hot term: run-length accumulate, flush to the private columns when the class changes
#pragma unroll
            for (int i = 0; i < RL8_CHUNK; ++i) {
                const int cls = lab[i];
                const bool ok = cls != 255;
                if (ok && cls != rs.cur) {
                    if (rs.cur >= 0 && rs.cur < K) {
                        pv[(0 * KP + rs.cur) * NT] += fmaf(hy, ox0, rs.o00);
                        pv[(1 * KP + rs.cur) * NT] += fmaf(hy, ox1, rs.o01);
                        pv[(2 * KP + rs.cur) * NT] += fmaf(lamy, ox0, rs.o10);
                        pv[(3 * KP + rs.cur) * NT] += fmaf(lamy, ox1, rs.o11);
                    }
                    rs.o00 = rs.o01 = rs.o10 = rs.o11 = 0.f;
                    ox0 = ox1 = 0.f;
                    rs.cur = cls;
                }
                ox0 += ok ? hx[i] : 0.f;
                ox1 += ok ? lamx[i] : 0.f;
            }
        }
        // end of row: fold the row accumulators into the four taps
        rs.o00 = fmaf(hy, ox0, rs.o00), rs.o01 = fmaf(hy, ox1, rs.o01);
        rs.o10 = fmaf(lamy, ox0, rs.o10), rs.o11 = fmaf(lamy, ox1, rs.o11);
        {
            const float2 hy2 = make_float2(hy, hy), ly2 = make_float2(lamy, lamy);
#pragma unroll
            for (int q = 0; q < NH; ++q) {
                G00[q] = __ffma2_rn(R0[q], hy2, G00[q]);
                G01[q] = __ffma2_rn(R1[q], hy2, G01[q]);
                G10[q] = __ffma2_rn(R0[q], ly2, G10[q]);
                G11[q] = __ffma2_rn(R1[q], ly2, G11[q]);
            }
        }
    }
}

// ORD = true (ordered instantiation): ds_rl is the tile scratch and `out` the per-CTA loss partials; each CTA stores its
// whole tap tile and its loss to slot [blockIdx.x] instead of adding them with atomics (readloss_gather combines them)
template <bool ORD = false>
__global__ void __launch_bounds__(RL8_THREADS, 2)
    readloss8_kernel(const float* __restrict__ s, const unsigned char* __restrict__ lab8, float inv_T, float temperature, int h,
                     int w, int Hm, int Wm, int K, float sy, float sx, int RS, int TYC, int tiles_x, int tiles_y,
                     float* __restrict__ ds_rl, unsigned long long* __restrict__ ws, float* __restrict__ out) {
    constexpr int KP = RL8_KP, NH = KP / 2, NT = RL8_THREADS, LDX = RL8_TX + 1;
    extern __shared__ __align__(16) float smem[];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int tile_elems = (TYC + 1) * LDX * KP;
    float* s_tile = smem;                    // [(TYC+1)][33][KP] similarities of the tile's feature pixels
    float* ds_tile = s_tile + tile_elems;    // same shape: gradient taps
    float* priv = ds_tile + tile_elems;      // [4][KP][NT] one-hot tap weights, thread-private columns
    float* red = priv + 4 * KP * NT;         // [8]

    int bid = blockIdx.x;
    const int tx_i = bid % tiles_x;
    bid /= tiles_x;
    const int ty_i = bid % tiles_y, b = bid / tiles_y;
    const int fy0 = ty_i * TYC, fx0 = tx_i * RL8_TX;

    for (int i = tid; i < tile_elems; i += NT) {
        const int e = i / KP, k = i - e * KP;
        const int ty = e / LDX, tx = e - ty * LDX;
        const int fy = min(fy0 + ty, h - 1), fx = min(fx0 + tx, w - 1);
        s_tile[i] = __ldg(s + ((size_t)(b * h + fy) * w + fx) * KP + k);
        ds_tile[i] = 0.f;
    }
    for (int i = tid; i < KP * NT; i += NT) reinterpret_cast<float4*>(priv)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncthreads();

    const int cxl = tid % RL8_TX, rest = tid / RL8_TX;  // rest in [0, TYC*RS)
    const int cyl = rest / RS, split = rest - cyl * RS;
    const int cy = fy0 + cyl, cx = fx0 + cxl;
    const bool active = (cy < h) && (cx < w);
    const int ly0 = cyl, ly1 = min(cy + 1, h - 1) - fy0;
    const int lx0 = cxl, lx1 = min(cx + 1, w - 1) - fx0;

    float2 G00[NH], G01[NH], G10[NH], G11[NH];
#pragma unroll
    for (int i = 0; i < NH; ++i) G00[i] = G01[i] = G10[i] = G11[i] = make_float2(0.f, 0.f);
    float lossacc = 0.f;  // log2 units
    float* pv = priv + tid;  // element (tap, k) at pv[(tap*KP + k)*NT]

    int Ya = 0, Yb = 0, Xa = 0, Xb = 0;
    if (active) {
        Ya = first_ge8(cy, sy, Hm, h), Yb = first_ge8(cy + 1, sy, Hm, h);
        Xa = first_ge8(cx, sx, Wm, w), Xb = first_ge8(cx + 1, sx, Wm, w);
    }
    // warp-uniform loop bounds (out-of-range pixels predicated off)
    const int nr_lane = (Yb - Ya - split + RS - 1) / RS;
    const int nr_max = __reduce_max_sync(0xffffffffu, max(nr_lane, 0));
    const int nc_max = __reduce_max_sync(0xffffffffu, Xb - Xa);
    const float c2 = inv_T * 1.4426950408889634f;
    const int tl0 = active ? ly0 : 0, tl1 = active ? ly1 : 0, tx0 = active ? lx0 : 0, tx1 = active ? lx1 : 0;
    const float2* t00 = reinterpret_cast<const float2*>(s_tile + (tl0 * LDX + tx0) * KP);
    const float2* t01 = reinterpret_cast<const float2*>(s_tile + (tl0 * LDX + tx1) * KP);
    const float2* t10 = reinterpret_cast<const float2*>(s_tile + (tl1 * LDX + tx0) * KP);
    const float2* t11 = reinterpret_cast<const float2*>(s_tile + (tl1 * LDX + tx1) * KP);
    float shift;  // softmax stabiliser (log2 units): max over the cell's taps and slots
    bool pxmax;
    {
        float m = -INFINITY, n = INFINITY;
#pragma unroll
        for (int i = 0; i < NH; ++i) {
            const float2 a = t00[i], bq = t01[i], c = t10[i], d = t11[i];
            if (2 * i < K) {
                m = fmaxf(m, fmaxf(fmaxf(a.x, bq.x), fmaxf(c.x, d.x)));
                n = fminf(n, fminf(fminf(a.x, bq.x), fminf(c.x, d.x)));
            }
            if (2 * i + 1 < K) {
                m = fmaxf(m, fmaxf(fmaxf(a.y, bq.y), fmaxf(c.y, d.y)));
                n = fminf(n, fminf(fminf(a.y, bq.y), fminf(c.y, d.y)));
            }
        }
        shift = m * c2;
        // spread too large for the per-cell stabiliser (tiny T / un-normalised logits; also NaN/inf): exact path
        pxmax = __any_sync(0xffffffffu, !(shift - n * c2 < 60.f));
    }
    // run-length state of the one-hot term
    RunState rs;
    rs.cur = -1, rs.o00 = rs.o01 = rs.o10 = rs.o11 = 0.f;
    const unsigned char* lab_b = lab8 + (size_t)b * Hm * Wm;
    CellCtx cc;
    cc.t00 = t00, cc.t01 = t01, cc.t10 = t10, cc.t11 = t11;
    cc.lab_b = lab_b, cc.Ya = Ya, cc.Yb = Yb, cc.Xa = Xa, cc.Xb = Xb, cc.split = split, cc.RS = RS, cc.Wm = Wm, cc.K = K;
    cc.nr_max = nr_max, cc.nc_max = nc_max, cc.active = active;
    cc.sx = sx, cc.sy = sy, cc.cxf = (float)cx, cc.cyf = (float)cy, cc.c2 = c2, cc.shift = shift;
    if (!pxmax) cell_rows<false>(cc, rs, pv, G00, G01, G10, G11, lossacc);
    else cell_rows<true>(cc, rs, pv, G00, G01, G10, G11, lossacc);
    const int cur = rs.cur;
    const float o00 = rs.o00, o01 = rs.o01, o10 = rs.o10, o11 = rs.o11;

    if (active) {
        if (cur >= 0 && cur < K) {
            pv[(0 * KP + cur) * NT] += o00;
            pv[(1 * KP + cur) * NT] += o01;
            pv[(2 * KP + cur) * NT] += o10;
            pv[(3 * KP + cur) * NT] += o11;
        }
        // minus the logit of the labelled class: sum_px z_y = c2 * sum_{tap,k} onehot_weight[tap][k] * tap[k];
        // then subtract the one-hot part from the tap gradients
        float zy = 0.f;
#pragma unroll
        for (int q = 0; q < NH; ++q) {
            const float a0 = pv[(0 * KP + 2 * q) * NT], a1 = pv[(0 * KP + 2 * q + 1) * NT];
            const float b0 = pv[(1 * KP + 2 * q) * NT], b1 = pv[(1 * KP + 2 * q + 1) * NT];
            const float c0 = pv[(2 * KP + 2 * q) * NT], c1 = pv[(2 * KP + 2 * q + 1) * NT];
            const float d0 = pv[(3 * KP + 2 * q) * NT], d1 = pv[(3 * KP + 2 * q + 1) * NT];
            const float2 v00 = t00[q], v01 = t01[q], v10 = t10[q], v11 = t11[q];
            zy = fmaf(a0, v00.x, fmaf(a1, v00.y, zy));
            zy = fmaf(b0, v01.x, fmaf(b1, v01.y, zy));
            zy = fmaf(c0, v10.x, fmaf(c1, v10.y, zy));
            zy = fmaf(d0, v11.x, fmaf(d1, v11.y, zy));
            G00[q].x -= a0, G00[q].y -= a1;
            G01[q].x -= b0, G01[q].y -= b1;
            G10[q].x -= c0, G10[q].y -= c1;
            G11[q].x -= d0, G11[q].y -= d1;
        }
        lossacc = fmaf(-c2, zy, lossacc);
        // fold degenerate taps (last row / column clamp onto themselves)
        if (ly1 == ly0) {
#pragma unroll
            for (int q = 0; q < NH; ++q) {
                G00[q] = __fadd2_rn(G00[q], G10[q]), G01[q] = __fadd2_rn(G01[q], G11[q]);
                G10[q] = G11[q] = make_float2(0.f, 0.f);
            }
        }
        if (lx1 == lx0) {
#pragma unroll
            for (int q = 0; q < NH; ++q) {
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
                float2* dst = reinterpret_cast<float2*>(ds_tile + (ly * LDX + lx) * KP);
#pragma unroll
                for (int q = 0; q < NH; ++q) {
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
            const int e = i / (KP / 4), q = i - e * (KP / 4);
            const int ty = e / LDX, tx = e - ty * LDX;
            const int fy = fy0 + ty, fx = fx0 + tx;
            if (fy < h && fx < w) {
                const float4 v = reinterpret_cast<const float4*>(ds_tile)[i];
                if (v.x != 0.f || v.y != 0.f || v.z != 0.f || v.w != 0.f)
                    atomicAdd(reinterpret_cast<float4*>(ds_rl + ((size_t)(b * h + fy) * w + fx) * KP) + q, v);
            }
        }
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
    if constexpr (ORD) return;
    // last CTA: readloss = loss_sum / V ; scale = 1 / (V*T)   (V from the histogram pm_labels_pack left in ws)
    __threadfence();
    __syncthreads();
    if (tid == 0) {
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

struct Rl8Geometry {
    float sy, sx;
    int RS, TYC, tiles_x, tiles_y;
    long long grid, tile_elems;  // CTAs; floats of one CTA's (TYC+1) x (RL8_TX+1) x RL8_KP tap tile
};

static Rl8Geometry rl8_geometry(int B, int h, int w, int Hm, int Wm) {
    Rl8Geometry g;
    // PyTorch's align_corners scale: (in-1)/(out-1) in fp32, 0 when out == 1
    g.sy = Hm > 1 ? (float)(h - 1) / (float)(Hm - 1) : 0.f;
    g.sx = Wm > 1 ? (float)(w - 1) / (float)(Wm - 1) : 0.f;
    // row-split factor: enough CTAs to fill the chip when there are few cells (output stride 16, small batches)
    const long long cells = (long long)B * h * w;
    const int rows_per_cell = h > 1 ? (Hm + h - 2) / (h - 1) : Hm;
    g.RS = 1;
    while (g.RS < 4 && cells * g.RS < 4LL * 148 * RL8_THREADS && g.RS * 2 <= rows_per_cell) g.RS *= 2;
    g.TYC = (RL8_THREADS / RL8_TX) / g.RS;
    g.tiles_x = (w + RL8_TX - 1) / RL8_TX, g.tiles_y = (h + g.TYC - 1) / g.TYC;
    g.grid = (long long)B * g.tiles_x * g.tiles_y;
    g.tile_elems = (long long)(g.TYC + 1) * (RL8_TX + 1) * RL8_KP;
    return g;
}

template <bool ORD>
static int launch_readloss8(const float* s, const uint8_t* lab8, float temperature, int B, int h, int w, int Hm, int Wm, int K,
                            float* ds_rl, unsigned long long* ws, float* out, cudaStream_t st) {
    const Rl8Geometry g = rl8_geometry(B, h, w, Hm, Wm);
    const size_t smem = sizeof(float) * ((size_t)2 * g.tile_elems + (size_t)4 * RL8_KP * RL8_THREADS + 8);
    if (g.grid > 0x7fffffffLL) return PM_ERR_SHAPE;
    cudaError_t e = cudaFuncSetAttribute(readloss8_kernel<ORD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    readloss8_kernel<ORD><<<(int)g.grid, RL8_THREADS, smem, st>>>(s, lab8, 1.f / temperature, temperature, h, w, Hm, Wm, K, g.sy,
                                                                  g.sx, g.RS, g.TYC, g.tiles_x, g.tiles_y, ds_rl, ws, out);
    e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

long long readloss8_scratch_bytes(int B, int h, int w, int Hm, int Wm) {
    const Rl8Geometry g = rl8_geometry(B, h, w, Hm, Wm);
    return (g.grid * g.tile_elems + (g.grid + 3) / 4 * 4) * (long long)sizeof(float);
}

}  // namespace pm

// cells kernel (pm_readloss10.cu): 0 = launched, -1 = shape outside its fixed-point range
int pm_readloss_cells_launch(const float* s, const uint8_t* lab8, float temperature, int B, int h, int w, int Hm, int Wm, int K,
                             float* ds_rl, void* ws, float* out, cudaStream_t st);

extern "C" int pm_readloss_fwd8(const float* s, const uint8_t* lab8, float temperature, int B, int h, int w, int Hm, int Wm,
                                int K, float* ds_rl, void* ws, float* out, void* stream) {
    if (!s || !lab8 || !ds_rl || !ws || !out) return PM_ERR_NULL;
    if (K < 1 || K > 19) return PM_ERR_SLOTS;
    if (B <= 0 || h <= 0 || w <= 0 || Hm <= 0 || Wm <= 0 || !(temperature > 0.f)) return PM_ERR_SHAPE;
    if (((uintptr_t)s & 15) || ((uintptr_t)ds_rl & 15) || ((uintptr_t)ws & 7)) return PM_ERR_ALIGN;
    const int minratio = 3;   // narrower cells (label map < 3x the feature map) keep the one-thread-per-cell kernel
    if (w > 1 && (Wm - 1) / (w - 1) >= minratio) {
        const int rc = pm_readloss_cells_launch(s, lab8, temperature, B, h, w, Hm, Wm, K, ds_rl, ws, out, (cudaStream_t)stream);
        if (rc >= 0) return rc;
    }
    return pm::launch_readloss8<false>(s, lab8, temperature, B, h, w, Hm, Wm, K, ds_rl, (unsigned long long*)ws, out,
                                       (cudaStream_t)stream);
}

extern "C" int pm_readloss_fwd8_ordered(const float* s, const uint8_t* lab8, float temperature, int B, int h, int w, int Hm,
                                        int Wm, int K, float* ds_rl, void* ws, float* out, float* scratch, void* stream) {
    if (!s || !lab8 || !ds_rl || !ws || !out || !scratch) return PM_ERR_NULL;
    if (K < 1 || K > 19) return PM_ERR_SLOTS;
    if (B <= 0 || h <= 0 || w <= 0 || Hm <= 0 || Wm <= 0 || !(temperature > 0.f)) return PM_ERR_SHAPE;
    if (((uintptr_t)s & 15) || ((uintptr_t)ds_rl & 15) || ((uintptr_t)ws & 7) || ((uintptr_t)scratch & 15)) return PM_ERR_ALIGN;
    // readloss8_kernel takes every shape; the cells kernel is never used here (its warps scatter with REDs)
    using namespace pm;
    const Rl8Geometry g = rl8_geometry(B, h, w, Hm, Wm);
    if (g.grid > 0x7fffffffLL) return PM_ERR_SHAPE;
    float* lossp = scratch + (size_t)g.grid * g.tile_elems;
    const cudaStream_t st = (cudaStream_t)stream;
    if (int rc = launch_readloss8<true>(s, lab8, temperature, B, h, w, Hm, Wm, K, scratch, (unsigned long long*)ws, lossp, st))
        return rc;
    return readloss_gather(scratch, lossp, (int)g.grid, B, h, w, RL8_KP, g.TYC, RL8_TX, g.tiles_x, g.tiles_y, K, temperature,
                           ds_rl, (unsigned long long*)ws, out, st);
}
