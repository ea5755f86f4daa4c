// Memory write, pipelined variants (fast path when hw is a multiple of the 16-byte chunk).

#include "pm_common.cuh"
#include "pm_tma.cuh"
#include "pm_internal.h"

namespace pm {

// ----------------------------------------------------------------------------- class sums (forward)
// Same algorithm as write_reduce_kernel (thread = channel, warp-uniform class index, run-length register
// accumulator, private column of a CTA-resident [K+1][C+4] tile, one vector RED per touched class row),
// but the [C][32] feature tile arrives through a 2-stage ring of 16-byte async copies and is stored with
// XOR-swizzled chunks, so a thread reads 4 (fp32) / 8 (bf16) pixels of its channel per conflict-free
// LDS.128; the label taps of the NEXT tile are fetched while the current one is reduced.

template <typename T, int C, int KP, bool ORD = false>
__global__ void __launch_bounds__(C) write_reduce_tiled_kernel(const T* __restrict__ f, const void* __restrict__ labels, int lab_u8,
                                                                float* __restrict__ SD, int h, int w, int Hm, int Wm,
                                                                int K, float sy, float sx, int tiles_per_img,
                                                                int ntiles) {
    constexpr int NSTAGE = 2, EPC = 16 / (int)sizeof(T), CPR = 32 / EPC, NW = C / 32, CS = C + 4;
    extern __shared__ __align__(16) unsigned char smraw[];
    float* S_tile = reinterpret_cast<float*>(smraw);               // [KP][CS]
    float* pn = S_tile + KP * CS;                                   // [NW][32]
    float* invr = pn + NW * 32;                                     // [32]
    float4* ent = reinterpret_cast<float4*>(invr + 32);             // [2][32][4] (class bits, w/|f|, w, -)
    unsigned* multi = reinterpret_cast<unsigned*>(ent + 2 * 32 * 4);  // [2] + pad
    T* ft = reinterpret_cast<T*>(multi + 4);                        // [NSTAGE][C][32], swizzled chunks

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, hw = h * w;
    for (int i = tid; i < KP * CS; i += C) S_tile[i] = 0.f;
    int cur = -1;
    unsigned seen = 0u;
    float acc = 0.f, accD = 0.f;

    auto tile_coords = [&](int t, int& b, int& px0) {
        b = t / tiles_per_img;
        px0 = (t - b * tiles_per_img) * 32;
    };
    auto store_entries = [&](int buf, const LabelTaps& t, int n) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
            ent[(buf * 32 + lane) * 4 + j] = make_float4(__int_as_float(t.cls[j]), 0.f, t.w[j], 0.f);
        const unsigned m = __ballot_sync(0xffffffffu, n > 1);
        if (lane == 0) multi[buf] = m;
    };
    auto taps_for = [&](int t) {
        LabelTaps r;
        int b, px0;
        tile_coords(t, b, px0);
        const int px = px0 + lane;
        if (t < ntiles && px < hw) {
            const int fy = px / w, fx = px - fy * w;
            r = label_taps(label_image(labels, (size_t)b * Hm * Wm, lab_u8), lab_u8, Hm, Wm, fy, fx, sy, sx, K);
        } else {
            r.cls[0] = r.cls[1] = r.cls[2] = r.cls[3] = K;
            r.w[0] = r.w[1] = r.w[2] = r.w[3] = 0.f;
        }
        return r;
    };

    int tile = blockIdx.x;
#pragma unroll
    for (int s = 0; s < NSTAGE; ++s) {
        const int t = tile + s * gridDim.x;
        if (t < ntiles) {
            int b, px0;
            tile_coords(t, b, px0);
            tile_load_async_swz<T, C, C>(ft + s * C * 32, f + (size_t)b * C * hw, hw, px0);
        }
        cp_async_commit();
    }
    if (wid == 0) {
        LabelTaps t0 = taps_for(tile);
        const int n = compact_taps(t0);
        store_entries(0, t0, n);
    }

    int stage = 0, ebuf = 0;
    for (; tile < ntiles; tile += gridDim.x) {
        // raw taps of the next tile: loads are issued now, consumed at the end of this iteration
        LabelTaps tn;
        if (wid == 0) tn = taps_for(tile + gridDim.x);
        cp_async_wait<NSTAGE - 1>();
        __syncthreads();
        const T* xt = ft + stage * C * 32;
        int b, px0;
        tile_coords(tile, b, px0);
        const int nvalid = min(32, hw - px0);
        {  // |f|^2 per pixel: lanes = pixels, each warp sums C/NW of the C rows
            float n2 = 0.f;
            if (NW % 8 == 0) {
                // rows wid, wid+NW, ... share one swizzle phase: the lane's offset inside a row is constant
                const int pc = ((lane / EPC) ^ tile_swz<T>(wid)) * EPC + (lane % EPC);
                const T* col = xt + wid * 32 + pc;
#pragma unroll 8
                for (int i = 0; i < C / NW; ++i) {
                    const float v = to_float(col[i * NW * 32]);
                    n2 = fmaf(v, v, n2);
                }
            } else {
#pragma unroll 8
                for (int c = wid; c < C; c += NW) {
                    const int pc = ((lane / EPC) ^ tile_swz<T>(c)) * EPC + (lane % EPC);
                    const float v = to_float(xt[c * 32 + pc]);
                    n2 = fmaf(v, v, n2);
                }
            }
            pn[wid * 32 + lane] = n2;
        }
        __syncthreads();
        if (tid < 32) {
            float sacc = 0.f;
#pragma unroll
            for (int i = 0; i < NW; ++i) sacc += pn[i * 32 + tid];
            const float ir = 1.f / fmaxf(sqrtf(sacc), PM_NORM_EPS);
            float4* e4 = ent + (ebuf * 32 + tid) * 4;  // fold 1/|f| into the tap weights of this pixel
#pragma unroll
            for (int j = 0; j < 4; ++j) e4[j].y = e4[j].z * ir;
        }
        __syncthreads();
        {
            const unsigned mm = multi[ebuf];
            const float4* eb = ent + ebuf * 32 * 4;
            const int swz = tile_swz<T>(tid);
            // entries are warp-uniform; a zero-weight entry (pixel past the end of the image) adds zeros
            auto add_entry = [&](const float4 en, float val) {
                const int cls = __float_as_int(en.x);
                if (cls != cur) {
                    if (cur >= 0) {
                        S_tile[cur * CS + tid] += acc;
                        if (tid == 0) S_tile[cur * CS + C] += accD;
                    }
                    acc = 0.f;
                    accD = 0.f;
                    cur = cls;
                    seen |= 1u << cls;
                }
                acc = fmaf(en.y, val, acc);
                accD += en.z;
            };
#pragma unroll 1
            for (int q = 0; q < CPR; ++q) {
                float v[EPC];
                if (sizeof(T) == 4) {
                    const float4 r = reinterpret_cast<const float4*>(xt + tid * 32)[q ^ swz];
                    v[0] = r.x, v[1] = r.y, v[2] = r.z, v[3] = r.w;
                } else {
                    const uint4 r = reinterpret_cast<const uint4*>(xt + tid * 32)[q ^ swz];
                    const unsigned rr[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        v[(2 * i) % EPC] = __uint_as_float(rr[i] << 16);
                        v[(2 * i + 1) % EPC] = __uint_as_float(rr[i] & 0xffff0000u);
                    }
                }
#pragma unroll
                for (int j = 0; j < EPC; ++j) {
                    const int px = q * EPC + j;
                    add_entry(eb[px * 4], v[j]);
                    if ((mm >> px) & 1u) {  // warp-uniform: this pixel straddles classes
#pragma unroll 1
                        for (int e = 1; e < 4; ++e) {
                            const float4 en = eb[px * 4 + e];
                            if (en.z != 0.f) add_entry(en, v[j]);
                        }
                    }
                }
            }
        }
        __syncthreads();  // stage and entry buffer consumed
        const int next = tile + NSTAGE * gridDim.x;
        if (next < ntiles) {
            int nb, npx0;
            tile_coords(next, nb, npx0);
            tile_load_async_swz<T, C, C>(ft + stage * C * 32, f + (size_t)nb * C * hw, hw, npx0);
        }
        cp_async_commit();
        if (wid == 0) {
            const int n = compact_taps(tn);
            store_entries(ebuf ^ 1, tn, n);
        }
        stage = (stage + 1 == NSTAGE) ? 0 : stage + 1;
        ebuf ^= 1;
    }
    cp_async_wait<0>();
    if (cur >= 0) {
        S_tile[cur * CS + tid] += acc;
        if (tid == 0) S_tile[cur * CS + C] += accD;
    }
    __syncthreads();
    if constexpr (ORD) {  // ordered instantiation: SD is the partial scratch, this CTA's slot is [blockIdx.x]
        float4* dst = reinterpret_cast<float4*>(SD + (size_t)blockIdx.x * (K + 1) * CS);
        for (int i = tid; i < (K + 1) * CS / 4; i += C) dst[i] = reinterpret_cast<const float4*>(S_tile)[i];
    } else {
        for (int k = 0; k <= K; ++k) {
            if (!((seen >> k) & 1u)) continue;
            for (int i = tid; i < CS / 4; i += C)
                atomicAdd(reinterpret_cast<float4*>(SD + (size_t)k * CS) + i,
                          reinterpret_cast<const float4*>(S_tile + k * CS)[i]);
        }
    }
}

// ---- tensor-core variant (fp32): S[class][channel] += Omega^T[class][px] . V[px][channel] -----------------------
// The class sums ARE a skinny GEMM (the reference computes them with torch.matmul, memory.py:227): per tile of
// 32 pixels, M = classes (one or two 16-row tiles), N = channels (each warp 32 = four 8-column tiles), K = pixels.
// mma.sync m16n8k8 TF32 with 3xTF32 compensation (see pm_read_tiled.cu); accumulators stay in registers across
// all tiles of the persistent CTA. The soft label weights of a tile are expanded to a dense [32 px][40] table
// in shared memory (row stride 40: conflict-free A fragments), B fragments come straight from the
// chunk-swizzled f tile (conflict-free) and are scaled by 1/|f| on the fly. Cost no longer depends on how
// fragmented the label map is (the run-length kernel above degenerates on noisy labels).

// The tiles arrive as SWIZZLE_128B tensor-map boxes (16-byte chunk c of row r at chunk c ^ (r & 7)) on an mbarrier ring.
//
// BN = true (the writing net's fused forward, pm_write_reduce_bn_fwd): the boxes are the convolution output z and the
// writing net's input x, and f = relu(x + BN(z)) is formed in place over the z box before the unchanged body runs, so
// f never exists in global memory. Each CTA finalises the C channels' statistics in its prologue; CTA 0 publishes
// mean / invstd and the running statistics and bumps the batch counter. A 2-stage ring of (z, x) pairs (128 KB at C = 256)
// would leave one CTA per SM; instead there is one z box and one x box, each on its own barrier, and the x box is refilled
// with the next tile as soon as f is formed, so half of the next tile streams in under the class sums (two CTAs per SM).
template <int C>
__host__ __device__ constexpr size_t wr_mma_ring_floats(int nstage) {  // the tile ring, which is also the [32][C+4] class-sum tile at the end
    return (size_t)nstage * C * 32 > (size_t)32 * (C + 4) ? (size_t)nstage * C * 32 : (size_t)32 * (C + 4);
}
template <int C, bool BN>
constexpr size_t wr_mma_smem_bytes() {
    constexpr size_t ring = (wr_mma_ring_floats<C>(BN ? 1 : 2) + 255) / 256 * 256;  // x box 1 KB aligned behind it
    return sizeof(float) * (ring + (BN ? (size_t)C * 32 + 2 * C : 0) + 32 * 40 + (C / 32) * 32 + 32 + 4) + 1024;
}

template <int C, int KP, bool ORD = false, bool BN = false>
__global__ void __launch_bounds__(C) write_reduce_mma_kernel(const __grid_constant__ CUtensorMap tm_f,
                                                              const __grid_constant__ CUtensorMap tm_x,
                                                              const void* __restrict__ labels, int lab_u8,
                                                              float* __restrict__ SD, int h, int w, int Hm, int Wm,
                                                              int K, float sy, float sx, int tiles_per_img,
                                                              int ntiles, const float* __restrict__ gamma,
                                                              const float* __restrict__ beta, BnFinalize fin) {
    constexpr int NSTAGE = BN ? 1 : 2, NW = C / 32, CS = C + 4, OMLD = 40;
    extern __shared__ __align__(16) unsigned char smraw_[];
    __shared__ __align__(8) uint64_t full[NSTAGE];
    __shared__ __align__(8) uint64_t fullx;            // BN: the x box has a barrier of its own (refilled before the z box)
    unsigned char* smraw = smem_align(smraw_, 1024);  // the swizzled TMA boxes need 1 KB alignment
    float* ft = reinterpret_cast<float*>(smraw);       // [NSTAGE][C][32] swizzled; reused as S_tile [32][CS] at the end
    constexpr size_t RING = (wr_mma_ring_floats<C>(NSTAGE) + 255) / 256 * 256;
    float* xs = ft + RING;                             // BN: [C][32] swizzled x box
    float* scs = xs + (BN ? C * 32 : 0);               // BN: [C] scale, [C] shift of the normalise
    float* shs = scs + (BN ? C : 0);
    float* om = shs + (BN ? C : 0);                    // [32 px][OMLD] dense label weights of the current tile
    float* pn = om + 32 * OMLD;                        // [NW][32]
    float* invr = pn + NW * 32;                        // [32]
    unsigned* cmask = reinterpret_cast<unsigned*>(invr + 32);  // [4]

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, hw = h * w;
    const int g = lane >> 2, t = lane & 3;
    float acc[2][4][4];
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
        for (int n = 0; n < 4; ++n) acc[m][n][0] = acc[m][n][1] = acc[m][n][2] = acc[m][n][3] = 0.f;
    float Dacc = 0.f;  // lane = class, partial over this warp's pixels
    unsigned seen = 0u;

    auto tile_coords = [&](int tl, int& b, int& px0) {
        b = tl / tiles_per_img;
        px0 = (tl - b * tiles_per_img) * 32;
    };
    auto taps_for = [&](int tl) {
        LabelTaps r;
        int b, px0;
        tile_coords(tl, b, px0);
        const int px = px0 + lane;
        if (tl < ntiles && px < hw) {
            const int fy = px / w, fx = px - fy * w;
            r = label_taps(label_image(labels, (size_t)b * Hm * Wm, lab_u8), lab_u8, Hm, Wm, fy, fx, sy, sx, K);
        } else {
            r.cls[0] = r.cls[1] = r.cls[2] = r.cls[3] = K;
            r.w[0] = r.w[1] = r.w[2] = r.w[3] = 0.f;
        }
        return r;
    };

    int tile = blockIdx.x;
    auto issue = [&](int tl, int s) {  // one thread
        int b, px0;
        tile_coords(tl, b, px0);
        if constexpr (BN) fence_proxy_async_smem();  // f was written over the z box of the previous tile
        mbar_expect_tx(&full[s], (uint32_t)(C * 32 * sizeof(float)));
        tma_load_2d(ft + s * C * 32, &tm_f, px0, b * C, &full[s]);
    };
    auto issue_x = [&](int tl) {  // one thread (BN)
        int b, px0;
        tile_coords(tl, b, px0);
        fence_proxy_async_smem();
        mbar_expect_tx(&fullx, (uint32_t)(C * 32 * sizeof(float)));
        tma_load_2d(xs, &tm_x, px0, b * C, &fullx);
    };
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < NSTAGE; ++s) mbar_init(&full[s], 1);
        if constexpr (BN) mbar_init(&fullx, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#pragma unroll
        for (int s = 0; s < NSTAGE; ++s)
            if (tile + s * (int)gridDim.x < ntiles) issue(tile + s * gridDim.x, s);
        if constexpr (BN)
            if (tile < ntiles) issue_x(tile);
    }
    if constexpr (BN) {  // thread = channel (blockDim == C)
        float mu, is;
        bn_finalize_channel(fin, tid, C, blockIdx.x == 0, mu, is);
        bn_scale_shift(mu, is, gamma[tid], beta[tid], scs[tid], shs[tid]);
        if (blockIdx.x == 0 && tid == 0 && fin.num_batches_tracked != nullptr) *fin.num_batches_tracked += 1;
    }
    LabelTaps tcur;
    if (wid == 0) tcur = taps_for(tile);

    int stage = 0;
    unsigned phase = 0;
    for (; tile < ntiles; tile += gridDim.x) {
        LabelTaps tnext;
        if (wid == 0) tnext = taps_for(tile + gridDim.x);  // loads in flight across this tile
        __syncthreads();
        mbar_wait(&full[stage], phase);
        float* xt = ft + stage * C * 32;
        if constexpr (BN) {  // f over the z box: both boxes share the swizzle, so element i of either is channel i / 32
            mbar_wait(&fullx, phase);
#pragma unroll 4
            for (int i = tid; i < C * 8; i += C) {
                const int c = i >> 3;
                const float sc = scs[c], sh = shs[c];
                float4 z = reinterpret_cast<const float4*>(xt)[i];
                const float4 x = reinterpret_cast<const float4*>(xs)[i];
                z.x = bn_res_relu(z.x, sc, sh, x.x), z.y = bn_res_relu(z.y, sc, sh, x.y);
                z.z = bn_res_relu(z.z, sc, sh, x.z), z.w = bn_res_relu(z.w, sc, sh, x.w);
                reinterpret_cast<float4*>(xt)[i] = z;
            }
            __syncthreads();  // x box consumed: the next tile's x streams in under this tile's class sums
            if (tid == 0 && tile + (int)gridDim.x < ntiles) issue_x(tile + gridDim.x);
        }
        for (int i = tid; i < 32 * OMLD / 4; i += C) reinterpret_cast<float4*>(om)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        {  // |f|^2 per pixel: lanes = pixels, each warp sums 32 of the C rows (rows wid, wid+NW, .. share a swizzle
           // phase when NW % 8 == 0)
            float n2 = 0.f;
            if (NW % 8 == 0) {
                const float* col = xt + wid * 32 + (((lane >> 2) ^ (wid & 7)) << 2) + (lane & 3);
#pragma unroll 8
                for (int i = 0; i < C / NW; ++i) {
                    const float v = col[i * NW * 32];
                    n2 = fmaf(v, v, n2);
                }
            } else {
                for (int c = wid; c < C; c += NW) {
                    const float v = xt[c * 32 + (((lane >> 2) ^ (c & 7)) << 2) + (lane & 3)];
                    n2 = fmaf(v, v, n2);
                }
            }
            pn[wid * 32 + lane] = n2;
        }
        __syncthreads();
        if (wid == 0) {
            float sacc = 0.f;
#pragma unroll
            for (int i = 0; i < NW; ++i) sacc += pn[i * 32 + lane];
            invr[lane] = 1.f / fmaxf(sqrtf(sacc), PM_NORM_EPS);
            unsigned m = 0u;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (tcur.w[j] != 0.f) {  // merged taps: distinct classes per pixel
                    om[lane * OMLD + tcur.cls[j]] = tcur.w[j];
                    m |= 1u << tcur.cls[j];
                }
            m = __reduce_or_sync(0xffffffffu, m);
            if (lane == 0) cmask[0] = m;
        }
        __syncthreads();
        const unsigned cm = cmask[0];
        seen |= cm;
        const bool hi_tile = (cm >> 16) != 0u;  // classes 16.. present in this tile (warp-uniform)
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
            const float ir0 = invr[8 * ks + t], ir1 = invr[8 * ks + t + 4];
            unsigned ah[2][4], al[2][4];
#pragma unroll
            for (int m = 0; m < 2; ++m) {
                if (m == 0 || hi_tile) {
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const float v = om[(8 * ks + t + 4 * (e >> 1)) * OMLD + 16 * m + g + 8 * (e & 1)];
                        ah[m][e] = tf32_hi(v);
                        al[m][e] = tf32_lo(v);
                    }
                }
            }
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                const float* row = xt + (wid * 32 + 8 * n + g) * 32 + t;
                const float b0 = row[((2 * ks) ^ g) << 2] * ir0, b1 = row[((2 * ks + 1) ^ g) << 2] * ir1;
                const unsigned b0h = tf32_hi(b0), b1h = tf32_hi(b1), b0l = tf32_lo(b0), b1l = tf32_lo(b1);
#pragma unroll
                for (int m = 0; m < 2; ++m) {
                    if (m == 0 || hi_tile) {
                        mma_tf32(acc[m][n], al[m][0], al[m][1], al[m][2], al[m][3], b0h, b1h);
                        mma_tf32(acc[m][n], ah[m][0], ah[m][1], ah[m][2], ah[m][3], b0l, b1l);
                        mma_tf32(acc[m][n], ah[m][0], ah[m][1], ah[m][2], ah[m][3], b0h, b1h);
                    }
                }
            }
        }
        {  // soft counts: lane = class, every warp sums its own 32/NW pixels (combined at the end)
#pragma unroll
            for (int px = wid; px < 32; px += NW) Dacc += om[px * OMLD + lane];
        }
        __syncthreads();  // stage and label table consumed
        const int next = tile + NSTAGE * gridDim.x;
        if (tid == 0 && next < ntiles) issue(next, stage);
        if (wid == 0) tcur = tnext;
        if (++stage == NSTAGE) stage = 0, phase ^= 1u;
    }
    __syncthreads();
    // accumulators -> shared [32][CS] (over the tile ring), then one vector RED per touched class row
    float* S_tile = ft;
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
        for (int n = 0; n < 4; ++n) {
            const int ch = wid * 32 + 8 * n + 2 * t;
            *reinterpret_cast<float2*>(S_tile + (16 * m + g) * CS + ch) = make_float2(acc[m][n][0], acc[m][n][1]);
            *reinterpret_cast<float2*>(S_tile + (16 * m + g + 8) * CS + ch) = make_float2(acc[m][n][2], acc[m][n][3]);
        }
    pn[wid * 32 + lane] = Dacc;  // pn is free now
    __syncthreads();
    if (wid == 0) {
        float d = 0.f;
#pragma unroll
        for (int i = 0; i < NW; ++i) d += pn[i * 32 + lane];
        S_tile[lane * CS + C] = d;
        S_tile[lane * CS + C + 1] = S_tile[lane * CS + C + 2] = S_tile[lane * CS + C + 3] = 0.f;
    }
    __syncthreads();
    if constexpr (ORD) {  // ordered instantiation: SD is the partial scratch, this CTA's slot is [blockIdx.x]
        float4* dst = reinterpret_cast<float4*>(SD + (size_t)blockIdx.x * (K + 1) * CS);
        for (int i = tid; i < (K + 1) * CS / 4; i += C) dst[i] = reinterpret_cast<const float4*>(S_tile)[i];
    } else {
        for (int k = 0; k <= K; ++k) {
            if (!((seen >> k) & 1u)) continue;
            for (int i = tid; i < CS / 4; i += C)
                atomicAdd(reinterpret_cast<float4*>(SD + (size_t)k * CS) + i,
                          reinterpret_cast<const float4*>(S_tile + k * CS)[i]);
        }
    }
}

// ---- tensor-core variant for bf16 maps: mma.sync m16n8k16, fp32 accumulate ---------------------------------------
// Same GEMM. The f tile ([C][32 px] bf16, TMA SWIZZLE_64B) IS the B operand: a 32-bit word of a channel row holds the
// pixel pair (2t, 2t+1) an m16n8k16 B fragment wants, and with the 64-byte swizzle the eight rows of a fragment load
// fall into distinct bank groups. 1/|f| scales the A operand (the label weights of the pixel) instead of the features,
// so the bf16 feature values enter the product unrounded; A is split hi + lo (two MMAs).
template <int C, int KP, bool ORD = false>
__global__ void __launch_bounds__(C) write_reduce_mma16_kernel(const __grid_constant__ CUtensorMap tm_f,
                                                                const void* __restrict__ labels, int lab_u8,
                                                                float* __restrict__ SD, int h, int w, int Hm, int Wm, int K,
                                                                float sy, float sx, int tiles_per_img, int ntiles) {
    using T = __nv_bfloat16;
    constexpr int NSTAGE = 2, NW = C / 32, CS = C + 4, OMLD = 40;
    extern __shared__ __align__(16) unsigned char smraw_[];
    __shared__ __align__(8) uint64_t full[NSTAGE];
    unsigned char* smraw = smem_align(smraw_, 1024);
    T* ft = reinterpret_cast<T*>(smraw);  // [NSTAGE][C][32] swizzled; the region is reused as S_tile [32][CS] fp32 at the end
    constexpr size_t RING_B = sizeof(T) * NSTAGE * C * 32 > sizeof(float) * 32 * CS ? sizeof(T) * NSTAGE * C * 32 : sizeof(float) * 32 * CS;
    float* om = reinterpret_cast<float*>(smraw + RING_B);  // [32 px][OMLD] dense label weights of the current tile
    float* pn = om + 32 * OMLD;                            // [NW][32]
    float* invr = pn + NW * 32;                            // [32]
    unsigned* cmask = reinterpret_cast<unsigned*>(invr + 32);

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, hw = h * w;
    const int g = lane >> 2, t = lane & 3;
    float acc[2][4][4];
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
        for (int n = 0; n < 4; ++n) acc[m][n][0] = acc[m][n][1] = acc[m][n][2] = acc[m][n][3] = 0.f;
    float Dacc = 0.f;
    unsigned seen = 0u;

    auto tile_coords = [&](int tl, int& b, int& px0) {
        b = tl / tiles_per_img;
        px0 = (tl - b * tiles_per_img) * 32;
    };
    auto taps_for = [&](int tl) {
        LabelTaps r;
        int b, px0;
        tile_coords(tl, b, px0);
        const int px = px0 + lane;
        if (tl < ntiles && px < hw) {
            const int fy = px / w, fx = px - fy * w;
            r = label_taps(label_image(labels, (size_t)b * Hm * Wm, lab_u8), lab_u8, Hm, Wm, fy, fx, sy, sx, K);
        } else {
            r.cls[0] = r.cls[1] = r.cls[2] = r.cls[3] = K;
            r.w[0] = r.w[1] = r.w[2] = r.w[3] = 0.f;
        }
        return r;
    };
    int tile = blockIdx.x;
    auto issue = [&](int tl, int s) {  // one thread
        int b, px0;
        tile_coords(tl, b, px0);
        mbar_expect_tx(&full[s], (uint32_t)(C * 32 * sizeof(T)));
        tma_load_2d(ft + (size_t)s * C * 32, &tm_f, px0, b * C, &full[s]);
    };
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < NSTAGE; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#pragma unroll
        for (int s = 0; s < NSTAGE; ++s)
            if (tile + s * (int)gridDim.x < ntiles) issue(tile + s * gridDim.x, s);
    }
    LabelTaps tcur;
    if (wid == 0) tcur = taps_for(tile);

    int stage = 0;
    unsigned phase = 0;
    for (; tile < ntiles; tile += gridDim.x) {
        LabelTaps tnext;
        if (wid == 0) tnext = taps_for(tile + gridDim.x);
        __syncthreads();
        mbar_wait(&full[stage], phase);
        const T* xt = ft + (size_t)stage * C * 32;
        const unsigned* xw = reinterpret_cast<const unsigned*>(xt);
        for (int i = tid; i < 32 * OMLD / 4; i += C) reinterpret_cast<float4*>(om)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        {  // |f|^2 per pixel: lane l sums pixel pair (2(l&15), +1) over the rows wid*32 + 2i + (l>>4); halves combined below
            const int half = lane >> 4, pp = (lane & 15) * 2;
            float na = 0.f, nb = 0.f;
#pragma unroll 8
            for (int i = 0; i < 16; ++i) {
                const int row = wid * 32 + 2 * i + half;
                const unsigned v = xw[(row * 32 + ((((pp >> 3) ^ ((row >> 1) & 3)) << 3) | (pp & 7))) >> 1];
                const float lo = __uint_as_float(v << 16), hi = __uint_as_float(v & 0xffff0000u);
                na = fmaf(lo, lo, na), nb = fmaf(hi, hi, nb);
            }
            na += __shfl_xor_sync(0xffffffffu, na, 16);
            nb += __shfl_xor_sync(0xffffffffu, nb, 16);
            if (half == 0) pn[wid * 32 + pp] = na, pn[wid * 32 + pp + 1] = nb;
        }
        __syncthreads();
        if (wid == 0) {
            float sacc = 0.f;
#pragma unroll
            for (int i = 0; i < NW; ++i) sacc += pn[i * 32 + lane];
            invr[lane] = 1.f / fmaxf(sqrtf(sacc), PM_NORM_EPS);
            unsigned m = 0u;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (tcur.w[j] != 0.f) {
                    om[lane * OMLD + tcur.cls[j]] = tcur.w[j];
                    m |= 1u << tcur.cls[j];
                }
            m = __reduce_or_sync(0xffffffffu, m);
            if (lane == 0) cmask[0] = m;
        }
        __syncthreads();
        const unsigned cm = cmask[0];
        seen |= cm;
        const bool hi_tile = (cm >> 16) != 0u;
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {  // 16 pixels per step
            // A[class][px]: a0 = (class g, px 2t,2t+1), a1 = (class g+8, ..), a2 = (class g, px 2t+8,..), a3 = (class g+8, ..)
            unsigned ah[2][4], al[2][4];
#pragma unroll
            for (int m = 0; m < 2; ++m) {
                if (m == 0 || hi_tile) {
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int px = 16 * ks + 2 * t + 8 * (e >> 1), cls = 16 * m + g + 8 * (e & 1);
                        const float v0 = om[px * OMLD + cls] * invr[px], v1 = om[(px + 1) * OMLD + cls] * invr[px + 1];
                        const float h0 = __bfloat162float(__float2bfloat16_rn(v0)), h1 = __bfloat162float(__float2bfloat16_rn(v1));
                        __nv_bfloat162 hh = __floats2bfloat162_rn(h0, h1), ll = __floats2bfloat162_rn(v0 - h0, v1 - h1);
                        ah[m][e] = *reinterpret_cast<unsigned*>(&hh);
                        al[m][e] = *reinterpret_cast<unsigned*>(&ll);
                    }
                }
            }
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                const int row = wid * 32 + 8 * n + g, sw = (row >> 1) & 3;
                const unsigned b0 = xw[row * 16 + (((2 * ks) ^ sw) << 2) + t], b1 = xw[row * 16 + (((2 * ks + 1) ^ sw) << 2) + t];
#pragma unroll
                for (int m = 0; m < 2; ++m) {
                    if (m == 0 || hi_tile) {
                        asm volatile(
                            "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                            : "+f"(acc[m][n][0]), "+f"(acc[m][n][1]), "+f"(acc[m][n][2]), "+f"(acc[m][n][3])
                            : "r"(al[m][0]), "r"(al[m][1]), "r"(al[m][2]), "r"(al[m][3]), "r"(b0), "r"(b1));
                        asm volatile(
                            "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                            : "+f"(acc[m][n][0]), "+f"(acc[m][n][1]), "+f"(acc[m][n][2]), "+f"(acc[m][n][3])
                            : "r"(ah[m][0]), "r"(ah[m][1]), "r"(ah[m][2]), "r"(ah[m][3]), "r"(b0), "r"(b1));
                    }
                }
            }
        }
        {
#pragma unroll
            for (int px = wid; px < 32; px += NW) Dacc += om[px * OMLD + lane];
        }
        __syncthreads();
        const int next = tile + NSTAGE * gridDim.x;
        if (tid == 0 && next < ntiles) issue(next, stage);
        if (wid == 0) tcur = tnext;
        if (++stage == NSTAGE) stage = 0, phase ^= 1u;
    }
    __syncthreads();
    float* S_tile = reinterpret_cast<float*>(smraw);
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
        for (int n = 0; n < 4; ++n) {
            const int ch = wid * 32 + 8 * n + 2 * t;
            *reinterpret_cast<float2*>(S_tile + (16 * m + g) * CS + ch) = make_float2(acc[m][n][0], acc[m][n][1]);
            *reinterpret_cast<float2*>(S_tile + (16 * m + g + 8) * CS + ch) = make_float2(acc[m][n][2], acc[m][n][3]);
        }
    pn[wid * 32 + lane] = Dacc;
    __syncthreads();
    if (wid == 0) {
        float d = 0.f;
#pragma unroll
        for (int i = 0; i < NW; ++i) d += pn[i * 32 + lane];
        S_tile[lane * CS + C] = d;
        S_tile[lane * CS + C + 1] = S_tile[lane * CS + C + 2] = S_tile[lane * CS + C + 3] = 0.f;
    }
    __syncthreads();
    if constexpr (ORD) {  // ordered instantiation: SD is the partial scratch, this CTA's slot is [blockIdx.x]
        float4* dst = reinterpret_cast<float4*>(SD + (size_t)blockIdx.x * (K + 1) * CS);
        for (int i = tid; i < (K + 1) * CS / 4; i += C) dst[i] = reinterpret_cast<const float4*>(S_tile)[i];
    } else {
        for (int k = 0; k <= K; ++k) {
            if (!((seen >> k) & 1u)) continue;
            for (int i = tid; i < CS / 4; i += C)
                atomicAdd(reinterpret_cast<float4*>(SD + (size_t)k * CS) + i, reinterpret_cast<const float4*>(S_tile + k * CS)[i]);
        }
    }
}

template <int C, int KP>
int launch_write_reduce_mma16(const void* f, const void* labels, int lab_u8, float* SD, int B, int h, int w, int Hm, int Wm,
                              int K, cudaStream_t st, float* part, int* ncta) {
    using T = __nv_bfloat16;
    const size_t ring = sizeof(T) * (size_t)2 * C * 32, stile = sizeof(float) * (size_t)32 * (C + 4);
    const size_t smem = sizeof(float) * (32 * 40 + (C / 32) * 32 + 32 + 4) + (ring > stile ? ring : stile) + 1024;
    const int hw = h * w, tiles = (hw + 31) / 32, ntiles = B * tiles;
    const float sy = h > 1 ? (float)(Hm - 1) / (float)(h - 1) : 0.f;
    const float sx = w > 1 ? (float)(Wm - 1) / (float)(w - 1) : 0.f;
    CUtensorMap tm_f;
    if (!make_map_2d<T>(&tm_f, f, (size_t)B * C, hw, C, 32, 3)) return PM_ERR_ALIGN;
    auto kern = part ? write_reduce_mma16_kernel<C, KP, true> : write_reduce_mma16_kernel<C, KP>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    int per_sm = 1;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, C, smem);
    if (e != cudaSuccess) return (int)e;
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 4) per_sm = 4;
    int grid = 148 * per_sm;
    if (grid > ntiles) grid = ntiles;
    if (part) {
        if (grid > PM_ORD_CTAS) grid = PM_ORD_CTAS;
        SD = part, *ncta = grid;
    }
    kern<<<grid, C, smem, st>>>(tm_f, labels, lab_u8, SD, h, w, Hm, Wm, K, sy, sx, tiles, ntiles);
    e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

// BN: f is relu(x + BN(z)) of the z map `f` and the x map `x` (see write_reduce_mma_kernel)
template <int C, int KP, bool BN = false>
int launch_write_reduce_mma(const void* f, const void* labels, int lab_u8, float* SD, int B, int h, int w, int Hm, int Wm, int K,
                            cudaStream_t st, float* part, int* ncta, const void* x = nullptr, const float* gamma = nullptr,
                            const float* beta = nullptr, BnFinalize fin = BnFinalize{}) {
    const size_t smem = wr_mma_smem_bytes<C, BN>();
    const int hw = h * w, tiles = (hw + 31) / 32, ntiles = B * tiles;
    const float sy = h > 1 ? (float)(Hm - 1) / (float)(h - 1) : 0.f;
    const float sx = w > 1 ? (float)(Wm - 1) / (float)(w - 1) : 0.f;
    CUtensorMap tm_f, tm_x;
    if (!make_map_2d<float>(&tm_f, f, (size_t)B * C, hw, C, 32, true)) return PM_ERR_ALIGN;
    if (!make_map_2d<float>(&tm_x, BN ? x : f, (size_t)B * C, hw, C, 32, true)) return PM_ERR_ALIGN;
    auto kern = part ? write_reduce_mma_kernel<C, KP, true, BN> : write_reduce_mma_kernel<C, KP, false, BN>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    int per_sm = 1;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, C, smem);
    if (e != cudaSuccess) return (int)e;
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 4) per_sm = 4;
    int grid = 148 * per_sm;
    if (grid > ntiles) grid = ntiles;
    if (part) {
        if (grid > PM_ORD_CTAS) grid = PM_ORD_CTAS;
        SD = part, *ncta = grid;
    }
    kern<<<grid, C, smem, st>>>(tm_f, tm_x, labels, lab_u8, SD, h, w, Hm, Wm, K, sy, sx, tiles, ntiles, gamma, beta, fin);
    e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

template <typename T, int C, int KP>
int launch_write_reduce_tiled(const void* f, const void* labels, int lab_u8, float* SD, int B, int h, int w, int Hm, int Wm,
                              int K, cudaStream_t st, float* part, int* ncta) {
    const size_t smem = sizeof(float) * ((size_t)KP * (C + 4) + (C / 32) * 32 + 32) + sizeof(float4) * 2 * 32 * 4 + 16 +
                        sizeof(T) * (size_t)2 * C * 32;
    auto kern = part ? write_reduce_tiled_kernel<T, C, KP, true> : write_reduce_tiled_kernel<T, C, KP>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const int hw = h * w, tiles = (hw + 31) / 32, ntiles = B * tiles;
    int per_sm = (int)(220 * 1024 / (smem + 1024));
    if (per_sm > 2048 / C) per_sm = 2048 / C;
    if (per_sm < 1) per_sm = 1;
    int grid = 148 * per_sm;
    if (grid > ntiles) grid = ntiles;
    if (part) {
        if (grid > PM_ORD_CTAS) grid = PM_ORD_CTAS;
        SD = part, *ncta = grid;
    }
    const float sy = h > 1 ? (float)(Hm - 1) / (float)(h - 1) : 0.f;
    const float sx = w > 1 ? (float)(Wm - 1) / (float)(w - 1) : 0.f;
    kern<<<grid, C, smem, st>>>((const T*)f, labels, lab_u8, SD, h, w, Hm, Wm, K, sy, sx, tiles, ntiles);
    e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

// ---------------------------------------------------------------------------- write backward (to f)
// dv[n] = sum_taps w * dS[class]; df = (dv - v (v.dv)) / |f|, v = f/|f|. Persistent CTAs, 2 per SM (measured:
// one 16-warp CTA with a 5-stage ring is 45% slower -- the per-tile barriers need a second CTA to hide
// behind, bytes in flight are not the limit); the [C][32] tiles of f arrive as 2-D tensor-map boxes on a
// 2-stage mbarrier ring (one thread issues a stage), lanes = pixels, 8 warps split the channels,
// dS sits in shared memory with row stride C+1 (lanes with different classes hit different banks). The
// label taps of the next tile are fetched by warp 0 while the current tile is processed.

//
// BN = true (the writing net's fused backward, pm_write_bwd_bn, fp32): the boxes are z and x of the writing net
// f = relu(x + BN(z)); f is formed over the x box with the forward's expression (same bits, same gate), and the kernel
// stores g = df * [f > 0] -- the residual gradient and the BatchNorm's output gradient -- instead of df. It also leaves
// this CTA's per-channel (sum g, sum g * xhat) in part[blockIdx.x] (lane sums over the tile, added over the CTA's tiles
// in tile order), which bn_sums_finalize_kernel adds in CTA order. One stage of two boxes keeps two CTAs per SM.
constexpr int WBT_THREADS = 256, WBT_WARPS = 8, WBT_STAGES = 2;

// v[i] summed over the 32 lanes, scattered: lane l returns the total of v[l % N] (N <= 32, a power of two). Full butterfly
// sums over the lane bits >= N, then a halving exchange: N - 1 shuffles for N values instead of 5 N.
template <int N>
__device__ __forceinline__ float lane_reduce_scatter(float (&v)[N], int lane) {
#pragma unroll
    for (int o = 16; o >= N; o >>= 1)
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], o);
#pragma unroll
    for (int s = N / 2; s >= 1; s >>= 1) {
        const bool up = (lane & s) != 0;
#pragma unroll
        for (int i = 0; i < s; ++i) {
            const float send = up ? v[i] : v[i + s], keep = up ? v[i + s] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
        }
    }
    return v[0];
}

template <typename T, int C, int KP, bool BN = false>
__global__ void __launch_bounds__(WBT_THREADS, 2)
    write_bwd_tiled_kernel(const __grid_constant__ CUtensorMap tm_f, const __grid_constant__ CUtensorMap tm_x,
                           const float* __restrict__ dS, const void* __restrict__ labels, int lab_u8,
                           T* __restrict__ df, int h, int w, int Hm, int Wm, int K, float sy, float sx,
                           int tiles_per_img, int ntiles, const float* __restrict__ mean, const float* __restrict__ invstd,
                           const float* __restrict__ gamma, const float* __restrict__ beta, float* __restrict__ part) {
    constexpr int NSTAGE = BN ? 1 : WBT_STAGES, CW = C / WBT_WARPS, LDS_ = C + 1;
    extern __shared__ __align__(16) unsigned char smraw[];
    float* dSs = reinterpret_cast<float*>(smraw);      // [KP][C+1]; rows >= K are zero (ignore class)
    float* pn = dSs + KP * LDS_;                        // [8][32]
    float* pd = pn + WBT_WARPS * 32;                    // [8][32]
    float* bnc = pd + WBT_WARPS * 32;                   // BN: [4][C] scale, shift, mean, invstd
    float2* ent = reinterpret_cast<float2*>(bnc + (BN ? 4 * C : 0) + ((KP * LDS_) & 1));  // [2][32][4]
    T* ft = reinterpret_cast<T*>(smem_align(reinterpret_cast<unsigned char*>(ent + 2 * 32 * 4), 128));  // [NSTAGE][C][32]
    T* xs = ft + NSTAGE * C * 32;                       // BN: [C][32] x box, overwritten with f
    __shared__ __align__(8) uint64_t full[NSTAGE];

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, hw = h * w;
    auto tile_coords = [&](int t, int& b, int& px0) {
        b = t / tiles_per_img;
        px0 = (t - b * tiles_per_img) * 32;
    };
    auto taps_for = [&](int t) {
        LabelTaps r;
        int b, px0;
        tile_coords(t, b, px0);
        const int px = px0 + lane;
        if (t < ntiles && px < hw) {
            const int fy = px / w, fx = px - fy * w;
            r = label_taps(label_image(labels, (size_t)b * Hm * Wm, lab_u8), lab_u8, Hm, Wm, fy, fx, sy, sx, K);
        } else {
            r.cls[0] = r.cls[1] = r.cls[2] = r.cls[3] = K;
            r.w[0] = r.w[1] = r.w[2] = r.w[3] = 0.f;
        }
        return r;
    };
    auto store_entries = [&](int buf, const LabelTaps& t) {
#pragma unroll
        for (int j = 0; j < 4; ++j) ent[(buf * 32 + lane) * 4 + j] = make_float2(__int_as_float(t.cls[j]), t.w[j]);
    };

    int tile = blockIdx.x;
    auto issue = [&](int t, int s) {  // one thread
        int b, px0;
        tile_coords(t, b, px0);
        if constexpr (BN) fence_proxy_async_smem();  // f was written over the x box of the previous tile
        mbar_expect_tx(&full[s], (uint32_t)((BN ? 2 : 1) * C * 32 * sizeof(T)));
        tma_load_2d(ft + s * C * 32, &tm_f, px0, b * C, &full[s]);
        if constexpr (BN) tma_load_2d(xs, &tm_x, px0, b * C, &full[s]);
    };
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < NSTAGE; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#pragma unroll
        for (int s = 0; s < NSTAGE; ++s)
            if (tile + s * (int)gridDim.x < ntiles) issue(tile + s * gridDim.x, s);
    }
    for (int i = tid; i < KP * LDS_; i += WBT_THREADS) {
        const int k = i / LDS_, c = i - k * LDS_;
        dSs[i] = (k < K && c < C) ? __ldg(dS + (size_t)k * C + c) : 0.f;
    }
    if constexpr (BN) {
        for (int c = tid; c < C; c += WBT_THREADS) {
            const float mu = mean[c], is = invstd[c];
            bn_scale_shift(mu, is, gamma[c], beta[c], bnc[c], bnc[C + c]);
            bnc[2 * C + c] = mu, bnc[3 * C + c] = is;
        }
    }
    float accg = 0.f, accgx = 0.f;  // BN: lane l's channel wid * CW + l % CW
    if (wid == 0) {
        LabelTaps t0 = taps_for(tile);
        compact_taps(t0);
        store_entries(0, t0);
    }

    int stage = 0, ebuf = 0;
    unsigned phase = 0;
    for (; tile < ntiles; tile += gridDim.x) {
        LabelTaps tn;
        if (wid == 0) tn = taps_for(tile + gridDim.x);  // loads in flight across this tile
        __syncthreads();  // dS / tap entries of this tile visible
        mbar_wait(&full[stage], phase);
        const T* xt = ft + stage * C * 32;
        int b, px0;
        tile_coords(tile, b, px0);
        const int nvalid = min(32, hw - px0);
        if constexpr (BN) {  // f over the x box; each thread forms (and later reads) only its own column
            T* fc = xs + wid * CW * 32 + lane;
            const T* zc = xt + wid * CW * 32 + lane;
#pragma unroll
            for (int j = 0; j < CW; ++j) {
                const int c = wid * CW + j;
                fc[j * 32] = bn_res_relu(zc[j * 32], bnc[c], bnc[C + c], fc[j * 32]);
            }
        }
        // this pixel's taps
        int cls[4];
        float wt[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float2 e = ent[(ebuf * 32 + lane) * 4 + j];
            cls[j] = __float_as_int(e.x);
            wt[j] = e.y;
        }
        const bool multi = wt[1] != 0.f;
        const T* fcol = (BN ? xs : xt) + wid * CW * 32 + lane;
        const float* r0 = dSs + cls[0] * LDS_ + wid * CW;
        float dv[CW], n2 = 0.f, dotf = 0.f;
#pragma unroll
        for (int j = 0; j < CW; ++j) {
            const float fv = to_float(fcol[j * 32]);
            n2 = fmaf(fv, fv, n2);
            dv[j] = wt[0] * r0[j];
        }
        if (multi) {  // pixel straddles classes (rare for real label maps)
            const float* r1 = dSs + cls[1] * LDS_ + wid * CW;
            const float* r2 = dSs + cls[2] * LDS_ + wid * CW;
            const float* r3 = dSs + cls[3] * LDS_ + wid * CW;
#pragma unroll
            for (int j = 0; j < CW; ++j) dv[j] = fmaf(wt[1], r1[j], fmaf(wt[2], r2[j], fmaf(wt[3], r3[j], dv[j])));
        }
#pragma unroll
        for (int j = 0; j < CW; ++j) dotf = fmaf(to_float(fcol[j * 32]), dv[j], dotf);
        pn[wid * 32 + lane] = n2;
        pd[wid * 32 + lane] = dotf;
        __syncthreads();
        float nn = 0.f, dd = 0.f;
#pragma unroll
        for (int i = 0; i < WBT_WARPS; ++i) {
            nn += pn[i * 32 + lane];
            dd += pd[i * 32 + lane];
        }
        const float nrm = sqrtf(nn), ir = 1.f / fmaxf(nrm, PM_NORM_EPS);
        // v.dv = ir * (f.dv); df = (dv - v (v.dv)) * ir = dv*ir - f * (ir^3 * f.dv)
        const float coef = (nrm <= PM_NORM_EPS) ? 0.f : ir * ir * ir * dd;
        if constexpr (BN) {
            const T* zc = xt + wid * CW * 32 + lane;
            float gx[CW];
#pragma unroll
            for (int j = 0; j < CW; ++j) {
                const int c = wid * CW + j;
                const float fv = fcol[j * 32];
                const float g = (fv > 0.f && lane < nvalid) ? fmaf(-coef, fv, dv[j] * ir) : 0.f;
                dv[j] = g;
                gx[j] = g * ((zc[j * 32] - bnc[2 * C + c]) * bnc[3 * C + c]);
            }
            if (lane < nvalid) {
                T* gp = df + ((size_t)b * C + wid * CW) * hw + px0 + lane;
#pragma unroll
                for (int j = 0; j < CW; ++j) {
                    stf(gp, dv[j]);
                    gp += hw;
                }
            }
            accg += lane_reduce_scatter<CW>(dv, lane);
            accgx += lane_reduce_scatter<CW>(gx, lane);
        } else if (lane < nvalid) {
            T* dfp = df + ((size_t)b * C + wid * CW) * hw + px0 + lane;
#pragma unroll
            for (int j = 0; j < CW; ++j) {
                stf(dfp, fmaf(-coef, to_float(fcol[j * 32]), dv[j] * ir));
                dfp += hw;
            }
        }
        __syncthreads();  // stage, entries and pn/pd consumed
        const int next = tile + NSTAGE * gridDim.x;
        if (tid == 0 && next < ntiles) issue(next, stage);
        if (wid == 0) {
            compact_taps(tn);
            store_entries(ebuf ^ 1, tn);
        }
        if (++stage == NSTAGE) stage = 0, phase ^= 1u;
        ebuf ^= 1;
    }
    if constexpr (BN) {
        if (lane < CW) {
            part[(size_t)blockIdx.x * 2 * C + wid * CW + lane] = accg;
            part[(size_t)blockIdx.x * 2 * C + C + wid * CW + lane] = accgx;
        }
    }
}

// dbeta[c] = sum_g part[g][0][c], dgamma[c] = sum_g part[g][1][c] over the G CTA partials of write_bwd_tiled_kernel<BN>,
// in fp64 and a fixed order: warp w adds the partials g = w, w + 16, ... in ascending order, then thread l of warp 0 adds
// the 16 warp sums in warp order. A block takes 32 consecutive entries of the [2][C] row.
__global__ void __launch_bounds__(512) bn_sums_finalize_kernel(const float* __restrict__ part, int G, int C,
                                                               float* __restrict__ dgamma, float* __restrict__ dbeta) {
    __shared__ double red[16][32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, e = blockIdx.x * 32 + lane;
    double a = 0.0;
    if (e < 2 * C) {
#pragma unroll 4
        for (int g = wid; g < G; g += 16) a += (double)__ldg(part + (size_t)g * 2 * C + e);
    }
    red[wid][lane] = a;
    __syncthreads();
    if (wid == 0 && e < 2 * C) {
        double t = 0.0;
#pragma unroll
        for (int i = 0; i < 16; ++i) t += red[i][lane];
        if (e < C) dbeta[e] = (float)t;
        else dgamma[e - C] = (float)t;
    }
}

// CTAs of the write backward (two per SM); also the number of BatchNorm partials the BN instantiation leaves
constexpr int WBT_GRID = 2 * 148;

// BN: `f` is z, `x` the writing net's input; df receives g; part [grid][2][C] the CTA partials, then dgamma / dbeta
template <typename T, int C, int KP, bool BN = false>
int launch_write_bwd_tiled(const float* dS, const void* f, const void* labels, int lab_u8, void* df, int B, int h, int w, int Hm,
                           int Wm, int K, cudaStream_t st, const void* x = nullptr, const float* mean = nullptr,
                           const float* invstd = nullptr, const float* gamma = nullptr, const float* beta = nullptr,
                           float* part = nullptr, float* dgamma = nullptr, float* dbeta = nullptr) {
    const size_t smem = sizeof(float) * ((size_t)KP * (C + 1) + 2 * WBT_WARPS * 32 + (BN ? 4 * C : 0) + 1) +
                        sizeof(float2) * 2 * 32 * 4 + sizeof(T) * (size_t)(BN ? 2 : WBT_STAGES) * C * 32 + 128;
    const int hw = h * w, tiles = (hw + 31) / 32, ntiles = B * tiles;
    int grid = WBT_GRID;
    if (grid > ntiles) grid = ntiles;
    const float sy = h > 1 ? (float)(Hm - 1) / (float)(h - 1) : 0.f;
    const float sx = w > 1 ? (float)(Wm - 1) / (float)(w - 1) : 0.f;
    CUtensorMap tm_f, tm_x;
    if (!make_map_2d<T>(&tm_f, f, (size_t)B * C, hw, C, 32, false)) return PM_ERR_ALIGN;
    if (!make_map_2d<T>(&tm_x, BN ? x : f, (size_t)B * C, hw, C, 32, false)) return PM_ERR_ALIGN;
    auto kern = write_bwd_tiled_kernel<T, C, KP, BN>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    kern<<<grid, WBT_THREADS, smem, st>>>(tm_f, tm_x, dS, labels, lab_u8, (T*)df, h, w, Hm, Wm, K, sy, sx, tiles, ntiles, mean,
                                          invstd, gamma, beta, part);
    e = cudaGetLastError();
    if (e != cudaSuccess || !BN) return e == cudaSuccess ? 0 : (int)e;
    bn_sums_finalize_kernel<<<(2 * C + 31) / 32, 512, 0, st>>>(part, grid, C, dgamma, dbeta);
    e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

#define PM_WT_SWITCH_C(T, KP, FN, ...)                \
    switch (C) {                                      \
        case 32: return FN<T, 32, KP>(__VA_ARGS__);   \
        case 64: return FN<T, 64, KP>(__VA_ARGS__);   \
        case 128: return FN<T, 128, KP>(__VA_ARGS__); \
        case 256: return FN<T, 256, KP>(__VA_ARGS__); \
        default: return PM_ERR_CHANNELS;              \
    }

int write_reduce_tiled(const void* f, const void* labels, int lab_u8, float* SD, int B, int C, int h, int w, int Hm, int Wm,
                       int K, int dtype, cudaStream_t st, float* part, int* ncta) {
    if (dtype == PM_F32) {
        switch (C) {  // tensor-core variant for every fp32 case (K + 1 <= 32 classes fit two 16-row MMA tiles)
            case 32: return launch_write_reduce_mma<32, 32>(f, labels, lab_u8, SD, B, h, w, Hm, Wm, K, st, part, ncta);
            case 64: return launch_write_reduce_mma<64, 32>(f, labels, lab_u8, SD, B, h, w, Hm, Wm, K, st, part, ncta);
            case 128: return launch_write_reduce_mma<128, 32>(f, labels, lab_u8, SD, B, h, w, Hm, Wm, K, st, part, ncta);
            case 256: return launch_write_reduce_mma<256, 32>(f, labels, lab_u8, SD, B, h, w, Hm, Wm, K, st, part, ncta);
            default: return PM_ERR_CHANNELS;
        }
    } else {
        switch (C) {  // tensor-core variant (whole 32-channel warps, >= 64 threads for the tile loads)
            case 64: return launch_write_reduce_mma16<64, 32>(f, labels, lab_u8, SD, B, h, w, Hm, Wm, K, st, part, ncta);
            case 128: return launch_write_reduce_mma16<128, 32>(f, labels, lab_u8, SD, B, h, w, Hm, Wm, K, st, part, ncta);
            case 256: return launch_write_reduce_mma16<256, 32>(f, labels, lab_u8, SD, B, h, w, Hm, Wm, K, st, part, ncta);
            case 32: break;  // the run-length FFMA2 kernel
            default: return PM_ERR_CHANNELS;
        }
        if (K <= 19) return launch_write_reduce_tiled<__nv_bfloat16, 32, 20>(f, labels, lab_u8, SD, B, h, w, Hm, Wm, K, st, part, ncta);
        return launch_write_reduce_tiled<__nv_bfloat16, 32, 32>(f, labels, lab_u8, SD, B, h, w, Hm, Wm, K, st, part, ncta);
    }
}

int write_bwd_tiled(const float* dS, const void* f, const void* labels, int lab_u8, void* df, int B, int C, int h, int w, int Hm,
                    int Wm, int K, int dtype, cudaStream_t st) {
    if (dtype == PM_F32) {
        if (K <= 19) { PM_WT_SWITCH_C(float, 20, launch_write_bwd_tiled, dS, f, labels, lab_u8, df, B, h, w, Hm, Wm, K, st) }
        else { PM_WT_SWITCH_C(float, 32, launch_write_bwd_tiled, dS, f, labels, lab_u8, df, B, h, w, Hm, Wm, K, st) }
    } else {
        if (K <= 19) { PM_WT_SWITCH_C(__nv_bfloat16, 20, launch_write_bwd_tiled, dS, f, labels, lab_u8, df, B, h, w, Hm, Wm, K, st) }
        else { PM_WT_SWITCH_C(__nv_bfloat16, 32, launch_write_bwd_tiled, dS, f, labels, lab_u8, df, B, h, w, Hm, Wm, K, st) }
    }
}

int write_reduce_bn(const float* z, const float* x, const void* labels, int lab_u8, float* SD, int B, int C, int h, int w, int Hm,
                    int Wm, int K, const float* gamma, const float* beta, const BnFinalize& fin, cudaStream_t st, float* part,
                    int* ncta) {
    switch (C) {
        case 32: return launch_write_reduce_mma<32, 32, true>(z, labels, lab_u8, SD, B, h, w, Hm, Wm, K, st, part, ncta, x, gamma, beta, fin);
        case 64: return launch_write_reduce_mma<64, 32, true>(z, labels, lab_u8, SD, B, h, w, Hm, Wm, K, st, part, ncta, x, gamma, beta, fin);
        case 128: return launch_write_reduce_mma<128, 32, true>(z, labels, lab_u8, SD, B, h, w, Hm, Wm, K, st, part, ncta, x, gamma, beta, fin);
        case 256: return launch_write_reduce_mma<256, 32, true>(z, labels, lab_u8, SD, B, h, w, Hm, Wm, K, st, part, ncta, x, gamma, beta, fin);
        default: return PM_ERR_CHANNELS;
    }
}

int write_bwd_bn_scratch_floats(int C) { return WBT_GRID * 2 * C; }

#define PM_WBN_SWITCH_C(KP)                                                                                                  \
    switch (C) {                                                                                                             \
        case 32: return launch_write_bwd_tiled<float, 32, KP, true>(dS, z, labels, lab_u8, g, B, h, w, Hm, Wm, K, st, x, mean, invstd, gamma, beta, part, dgamma, dbeta);   \
        case 64: return launch_write_bwd_tiled<float, 64, KP, true>(dS, z, labels, lab_u8, g, B, h, w, Hm, Wm, K, st, x, mean, invstd, gamma, beta, part, dgamma, dbeta);   \
        case 128: return launch_write_bwd_tiled<float, 128, KP, true>(dS, z, labels, lab_u8, g, B, h, w, Hm, Wm, K, st, x, mean, invstd, gamma, beta, part, dgamma, dbeta); \
        case 256: return launch_write_bwd_tiled<float, 256, KP, true>(dS, z, labels, lab_u8, g, B, h, w, Hm, Wm, K, st, x, mean, invstd, gamma, beta, part, dgamma, dbeta); \
        default: return PM_ERR_CHANNELS;                                                                                     \
    }

int write_bwd_bn(const float* dS, const float* z, const float* x, const void* labels, int lab_u8, const float* mean,
                 const float* invstd, const float* gamma, const float* beta, float* g, float* dgamma, float* dbeta, float* part,
                 int B, int C, int h, int w, int Hm, int Wm, int K, cudaStream_t st) {
    if (K <= 19) { PM_WBN_SWITCH_C(20) }
    else { PM_WBN_SWITCH_C(32) }
}

}  // namespace pm
