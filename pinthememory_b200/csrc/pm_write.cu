// Memory write: label-masked per-class segmented reduction, momentum update (+ both write losses),
// and their backward kernels.
#include "pm_common.cuh"
#include "pm_internal.h"

namespace pm {

// ----------------------------------------------------------------------------- class sums (forward)
// S[k] = sum_n omega[n,k] f[n]/|f[n]|, D[k] = sum_n omega[n,k]; omega = the <=4 bilinear label taps of
// feature pixel n. A reduction over pixels: a thread owns one CHANNEL and walks the pixels of a
// transposed [C][32+1] tile in shared memory. Class indices are warp-uniform (broadcast from shared
// memory), so each thread keeps a register accumulator for the current class (run-length: label maps
// are piecewise constant) and spills it into its private column of the CTA's [K+1][C+4] tile only when
// the class changes -- no atomics in the loop. CTAs are persistent; one vector RED per touched class
// row at the end.

constexpr int WR_P = 32;

template <typename T, int C, int KP, bool ORD = false>
__global__ void __launch_bounds__(C) write_reduce_kernel(const T* __restrict__ f, const void* __restrict__ labels, int lab_u8,
                                                          float* __restrict__ SD, int h, int w, int Hm, int Wm, int K,
                                                          float sy, float sx, int tiles_per_img, int ntiles) {
    constexpr int P = WR_P, LD = P + 1, NW = C / 32, CS = C + 4;
    extern __shared__ __align__(16) float smem[];
    float* S_tile = smem;                 // [KP][CS]
    float* ft = S_tile + KP * CS;         // [C][LD]
    float* pn = ft + C * LD;              // [NW][P]
    float* invr = pn + NW * P;            // [P]
    float2* ent = reinterpret_cast<float2*>(invr + P);  // [P][4] (class bits, weight)

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, hw = h * w;
    for (int i = tid; i < KP * CS; i += C) S_tile[i] = 0.f;
    int cur = -1;
    unsigned seen = 0u;
    float acc = 0.f, accD = 0.f;

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int b = tile / tiles_per_img, px0 = (tile - b * tiles_per_img) * P;
        const int nvalid = min(P, hw - px0);
        const bool v = lane < nvalid;
        const T* fb = f + (size_t)b * C * hw + px0 + lane;
        float n2 = 0.f;
#pragma unroll 8
        for (int c = wid; c < C; c += NW) {
            float fv = v ? ldf(fb + (size_t)c * hw) : 0.f;
            n2 = fmaf(fv, fv, n2);
            ft[c * LD + lane] = fv;
        }
        pn[wid * P + lane] = n2;
        if (tid < P) {
            LabelTaps t;
            if (tid < nvalid) {
                int px = px0 + tid, fy = px / w, fx = px - fy * w;
                t = label_taps(label_image(labels, (size_t)b * Hm * Wm, lab_u8), lab_u8, Hm, Wm, fy, fx, sy, sx, K);
            } else {
                t.cls[0] = t.cls[1] = t.cls[2] = t.cls[3] = K;
                t.w[0] = t.w[1] = t.w[2] = t.w[3] = 0.f;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) ent[tid * 4 + j] = make_float2(__int_as_float(t.cls[j]), t.w[j]);
        }
        __syncthreads();
        if (tid < P) {
            float s = 0.f;
#pragma unroll
            for (int i = 0; i < NW; ++i) s += pn[i * P + tid];
            invr[tid] = 1.f / fmaxf(sqrtf(s), PM_NORM_EPS);
        }
        __syncthreads();
        for (int px = 0; px < nvalid; ++px) {
            const float val = ft[tid * LD + px] * invr[px];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float2 e = ent[px * 4 + j];
                if (e.y != 0.f) {  // warp-uniform
                    const int cls = __float_as_int(e.x);
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
                    acc = fmaf(e.y, val, acc);
                    accD += e.y;
                }
            }
        }
        __syncthreads();
    }
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

// ---------------------------------------------------------------------------- write backward (to f)
// dv[n] = sum_k omega[n,k] dS[k]; df = (dv - v (v.dv)) / |f|. Per-pixel map, so the read kernels' mapping:
// CTA = 64 pixels x C channels, 8 warps split channels, a lane owns pixels (lane, lane+32). dS sits in
// shared memory with row stride C+1 so lanes with different classes hit different banks.

constexpr int WB_THREADS = 256, WB_WARPS = 8, WB_P = 64;

template <typename T, int CW, int KP>
__global__ void __launch_bounds__(WB_THREADS) write_bwd_kernel(const float* __restrict__ dS, const T* __restrict__ f,
                                                               const void* __restrict__ labels, int lab_u8,
                                                               T* __restrict__ df, int h, int w, int Hm, int Wm, int K,
                                                               float sy, float sx, int tiles_per_img) {
    constexpr int C = CW * WB_WARPS, P = WB_P, LDS_ = C + 1;
    extern __shared__ __align__(16) float smem[];
    float* dSs = smem;              // [K+1][C+1]; row K (ignore) is zero
    float* pn = dSs + KP * LDS_;    // [8][P]
    float* invr = pn + WB_WARPS * P;
    float* rnorm = invr + P;

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, hw = h * w;
    const int b = blockIdx.x / tiles_per_img, px0 = (blockIdx.x - b * tiles_per_img) * P;
    const int nvalid = min(P, hw - px0);
    const bool v0 = lane < nvalid, v1 = lane + 32 < nvalid;

    const T* fb = f + ((size_t)b * C + wid * CW) * hw + px0 + lane;
    float a0[CW], a1[CW], d0[CW], d1[CW];
    float n0 = 0.f, n1 = 0.f;
#pragma unroll
    for (int j = 0; j < CW; ++j) {
        a0[j] = v0 ? ldf(fb + (size_t)j * hw) : 0.f;
        a1[j] = v1 ? ldf(fb + (size_t)j * hw + 32) : 0.f;
    }
    for (int i = tid; i < KP * LDS_; i += WB_THREADS) {
        int k = i / LDS_, c = i - k * LDS_;
        dSs[i] = (k < K && c < C) ? __ldg(dS + (size_t)k * C + c) : 0.f;
    }
    LabelTaps t0, t1;
    {
        const void* lab_b = label_image(labels, (size_t)b * Hm * Wm, lab_u8);
        int px = px0 + (v0 ? lane : 0), fy = px / w, fx = px - fy * w;
        t0 = label_taps(lab_b, lab_u8, Hm, Wm, fy, fx, sy, sx, K);
        px = px0 + (v1 ? lane + 32 : 0), fy = px / w, fx = px - fy * w;
        t1 = label_taps(lab_b, lab_u8, Hm, Wm, fy, fx, sy, sx, K);
    }
#pragma unroll
    for (int j = 0; j < CW; ++j) {
        n0 = fmaf(a0[j], a0[j], n0);
        n1 = fmaf(a1[j], a1[j], n1);
    }
    pn[wid * P + lane] = n0;
    pn[wid * P + lane + 32] = n1;
    __syncthreads();
    if (tid < P) {
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < WB_WARPS; ++i) s += pn[i * P + tid];
        float n = sqrtf(s);
        rnorm[tid] = n;
        invr[tid] = 1.f / fmaxf(n, PM_NORM_EPS);
    }
    __syncthreads();
    const float ir0 = invr[lane], ir1 = invr[lane + 32];
    float dot0 = 0.f, dot1 = 0.f;
    const float* r00 = dSs + t0.cls[0] * LDS_ + wid * CW;
    const float* r01 = dSs + t0.cls[1] * LDS_ + wid * CW;
    const float* r02 = dSs + t0.cls[2] * LDS_ + wid * CW;
    const float* r03 = dSs + t0.cls[3] * LDS_ + wid * CW;
    const float* r10 = dSs + t1.cls[0] * LDS_ + wid * CW;
    const float* r11 = dSs + t1.cls[1] * LDS_ + wid * CW;
    const float* r12 = dSs + t1.cls[2] * LDS_ + wid * CW;
    const float* r13 = dSs + t1.cls[3] * LDS_ + wid * CW;
#pragma unroll
    for (int j = 0; j < CW; ++j) {
        float dv0 = t0.w[0] * r00[j];
        dv0 = fmaf(t0.w[1], r01[j], dv0);
        dv0 = fmaf(t0.w[2], r02[j], dv0);
        dv0 = fmaf(t0.w[3], r03[j], dv0);
        float dv1 = t1.w[0] * r10[j];
        dv1 = fmaf(t1.w[1], r11[j], dv1);
        dv1 = fmaf(t1.w[2], r12[j], dv1);
        dv1 = fmaf(t1.w[3], r13[j], dv1);
        a0[j] *= ir0;  // v
        a1[j] *= ir1;
        d0[j] = dv0;
        d1[j] = dv1;
        dot0 = fmaf(a0[j], dv0, dot0);
        dot1 = fmaf(a1[j], dv1, dot1);
    }
    __syncthreads();  // pn reuse
    pn[wid * P + lane] = dot0;
    pn[wid * P + lane + 32] = dot1;
    __syncthreads();
    dot0 = dot1 = 0.f;
#pragma unroll
    for (int i = 0; i < WB_WARPS; ++i) {
        dot0 += pn[i * P + lane];
        dot1 += pn[i * P + lane + 32];
    }
    if (rnorm[lane] <= PM_NORM_EPS) dot0 = 0.f;
    if (rnorm[lane + 32] <= PM_NORM_EPS) dot1 = 0.f;
    T* dfb = df + ((size_t)b * C + wid * CW) * hw + px0 + lane;
#pragma unroll
    for (int j = 0; j < CW; ++j) {
        if (v0) stf(dfb + (size_t)j * hw, (d0[j] - a0[j] * dot0) * ir0);
        if (v1) stf(dfb + (size_t)j * hw + 32, (d1[j] - a1[j] * dot1) * ir1);
    }
}

// --------------------------------------------------------------------------- momentum update + losses
// K x C is 19 x 256: pure latency work. One CTA per memory row (grid = K, 256 threads, thread = channel), every
// thread keeping its channel of ALL K rows in registers, so the K x K products (classifier logits, Gram) are
// per-thread multiplies followed by one batched block reduction, and nothing is re-read from shared memory
// (the first version -- one CTA, operands in shared memory -- was shared-memory-bandwidth bound: 25 us).
// Cross-row results meet in a small zero-initialised `aux` buffer; the last CTA to arrive finalises.
// Branch-free replacement of the reference's per-slot python loop with its 19 host syncs (memory.py:233-237).

constexpr int UP_THREADS = 256, UP_WARPS = 8, UP_KMAX = 32;

// Transpose-reduce 32 per-lane values across the warp in 31 shuffles (instead of 32 x 5): at every step a lane
// keeps the half of its values whose index bit matches its lane bit and adds the partner's copy of that half.
// On return v[0] of lane l is the warp total of value l.
__device__ __forceinline__ void warp_reduce32(float (&v)[32]) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const bool hi = (lane & off) != 0;
#pragma unroll
        for (int j = 0; j < off; ++j) {
            const float mine = hi ? v[j + off] : v[j];
            const float theirs = hi ? v[j] : v[j + off];
            v[j] = mine + __shfl_xor_sync(0xffffffffu, theirs, off);
        }
    }
}

// CTA total of 32 per-thread values: out[l] (l < 32) valid for every thread after the call. scratch: [UP_WARPS][32]
__device__ __forceinline__ void block_reduce32(float (&v)[32], float* scratch, float* out) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    warp_reduce32(v);
    scratch[wid * 32 + lane] = v[0];
    __syncthreads();
    if (wid == 0) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < UP_WARPS; ++w) t += scratch[w * 32 + lane];
        out[lane] = t;
    }
    __syncthreads();
}

// ---- the sharded update's exchange, fused into the update kernels over NVLink peer memory --------------------------
// Every rank owns one "symmetric" buffer (allocated and exchanged by torch.distributed._symmetric_memory on the host
// side; `bufs` is the device array of all ranks' base addresses, peer-mapped) laid out as
//   [0, PM_PEER_DS_OFF)            SD  : this rank's class sums|counts [K+1, C+4] (pm_write_reduce_fwd adds into it)
//   [PM_PEER_DS_OFF, FLAG_OFF)     dS  : this rank's gradient w.r.t. the class sums [K, C]
//   [PM_PEER_FLAG_OFF, ...)        flags[kind 0..3][row 0..31][rank 0..15] (u32, monotone epochs)
// CTA i of the update kernels is the only one that touches row-slot i: it raises flag (kind, i, my rank) = epoch in
// EVERY peer's buffer (st.release.sys), spins on its own copies until all ranks have raised theirs (ld.acquire.sys),
// then reads the operand straight out of the peers' buffers and sums in rank order -- the same order on every rank,
// so the updated memory is bit-identical across ranks. A second flag round ("done") at the end of the kernel keeps a
// rank from zeroing / overwriting its buffer for the next step while a slower peer still reads it. No NCCL launch,
// no extra kernel: ~21 KB per rank cross NVSwitch inside the kernel that needs them.
// (PeerCtx, peer_signal and peer_wait: pm_common.cuh)

// aux layout (floats, zeroed by the caller): [0] arrival counter (as unsigned), [2 .. 2+32) per-row CE term,
// [34 .. 34+32) per-row positive off-diagonal Gram sum
template <bool PEER>
__global__ void __launch_bounds__(UP_THREADS) update_fwd_kernel(const float* __restrict__ SD, PeerCtx peer,
                                                                float* __restrict__ SD_sum, const float* __restrict__ M_old,
                                                                float momentum, const float* __restrict__ W,
                                                                const float* __restrict__ bias, float* __restrict__ M_new,
                                                                float* __restrict__ losses, float* __restrict__ saved,
                                                                float* __restrict__ aux, int C, int K) {
    __shared__ float scratch[UP_WARPS * 32];
    __shared__ float red[32], red2[32], invn[32];
    const int tid = threadIdx.x, lane = tid & 31, i = blockIdx.x, CS = C + 4;
    const bool on = tid < C;
    // this thread's channel of every row; all loads are issued before the first use
    float m[UP_KMAX], wv[UP_KMAX], sd[UP_KMAX], dk[UP_KMAX];
    unsigned epoch = 0;
    if (PEER) {  // every rank's class sums are complete (its write_reduce kernel precedes this one in stream order)
        epoch = *peer.epoch + 1;
        peer_signal(peer, 0, i, epoch);
        peer_wait(peer, 0, i, epoch);
    }
#pragma unroll
    for (int k = 0; k < UP_KMAX; ++k) {
        const bool ok = k < K && on;
        m[k] = ok ? __ldg(M_old + (size_t)k * C + tid) : 0.f;
        wv[k] = ok ? __ldg(W + (size_t)k * C + tid) : 0.f;
        if (!PEER) {
            dk[k] = ok ? __ldg(SD + (size_t)k * CS + C) : 0.f;
            sd[k] = ok ? __ldg(SD + (size_t)k * CS + tid) : 0.f;
        } else {
            dk[k] = sd[k] = 0.f;
        }
    }
    if (PEER) {
        // CTA i gathers ROW i over the ranks in rank order, straight out of their buffers (volatile loads: peer memory is
        // not cached locally, and the flags above ordered these reads after the peers' writes), leaves the sum in
        // SD_sum (local) and releases the peers; the K CTAs of THIS rank then meet on a local counter and every CTA reads
        // all summed rows from SD_sum -- one row per CTA crosses NVLink instead of K.
        float si = 0.f, di = 0.f, rowK = 0.f, rowKc = 0.f;
        for (int r = 0; r < peer.world; ++r) {
            const volatile float* P = reinterpret_cast<const volatile float*>(peer.bufs[r]);
            if (on) si += P[(size_t)i * CS + tid];
            if (tid == 0) di += P[(size_t)i * CS + C];
            if (i == 0) {  // the ignore row only feeds last_class_sums
                if (on) rowK += P[(size_t)K * CS + tid];
                if (tid == 0) rowKc += P[(size_t)K * CS + C];
            }
        }
        if (on) SD_sum[(size_t)i * CS + tid] = si;
        if (tid == 0) SD_sum[(size_t)i * CS + C] = di;
        if (i == 0 && on) SD_sum[(size_t)K * CS + tid] = rowK;
        if (i == 0 && tid == 0) SD_sum[(size_t)K * CS + C] = rowKc;
        peer_signal(peer, 1, i, epoch);  // done reading the peers' sums (also: __threadfence_system + __syncthreads)
        if (tid == 0) {                   // local grid barrier: all K rows of SD_sum are written
            unsigned* cnt = reinterpret_cast<unsigned*>(aux) + 1;
            atomicAdd(cnt, 1u);
            for (unsigned spin = 0; atomicAdd(cnt, 0u) < (unsigned)K; ++spin)
                if (spin > (1u << 27)) __trap();
            __threadfence();
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < UP_KMAX; ++k) {
            const bool ok = k < K && on;
            dk[k] = ok ? __ldcg(SD_sum + (size_t)k * CS + C) : 0.f;
            sd[k] = ok ? __ldcg(SD_sum + (size_t)k * CS + tid) : 0.f;
        }
    }
    float d_own = 0.f;
#pragma unroll
    for (int k = 0; k < UP_KMAX; ++k)
        if (k == i) d_own = dk[k];
#pragma unroll
    for (int k = 0; k < UP_KMAX; ++k) {
        m[k] = (dk[k] != 0.f) ? fmaf((1.f - momentum) / dk[k], sd[k], momentum * m[k]) : m[k];
        sd[k] = m[k] * m[k];
    }
    block_reduce32(sd, scratch, red);  // red[k] = |M'_k|^2
    if (tid < 32) invn[tid] = 1.f / fmaxf(sqrtf(red[tid]), PM_NORM_EPS);
    __syncthreads();
#pragma unroll
    for (int k = 0; k < UP_KMAX; ++k) m[k] *= invn[k];
    float mi = 0.f;
#pragma unroll
    for (int k = 0; k < UP_KMAX; ++k)
        if (k == i) mi = m[k];
    if (on) M_new[(size_t)i * C + tid] = mi;
    if (tid == 0) {
        saved[i] = sqrtf(red[i]);
        saved[K + i] = d_own;
    }
    // row i of the classifier logits (red) and of the Gram matrix (red2)
#pragma unroll
    for (int k = 0; k < UP_KMAX; ++k) {
        wv[k] *= mi;
        sd[k] = mi * m[k];
    }
    __syncthreads();  // red / invn consumed
    block_reduce32(wv, scratch, red);
    block_reduce32(sd, scratch, red2);
    if (tid < 32) {  // CE term and positive off-diagonal Gram sum of row i
        const float z = lane < K ? red[lane] + __ldg(bias + lane) : -INFINITY;
        const float mx = warp_max(z);
        const float sum = warp_sum(lane < K ? expf(z - mx) : 0.f);
        const float zii = __shfl_sync(0xffffffffu, z, i);
        const float g = (lane < K && lane != i) ? fmaxf(red2[lane], 0.f) : 0.f;
        const float gsum = warp_sum(g);
        unsigned t = 0;
        if (lane == 0) {
            aux[2 + i] = mx + logf(sum) - zii;
            aux[2 + UP_KMAX + i] = gsum;
            __threadfence();
            t = atomicAdd(reinterpret_cast<unsigned*>(aux), 1u);
        }
        t = __shfl_sync(0xffffffffu, t, 0);
        if (t == (unsigned)K - 1) {  // last row to arrive: fixed-order (shuffle tree) sums -> deterministic losses
            __threadfence();
            const float c = warp_sum(lane < K ? __ldcg(aux + 2 + lane) : 0.f);
            const float d = warp_sum(lane < K ? __ldcg(aux + 2 + UP_KMAX + lane) : 0.f);
            if (lane == 0) {
                losses[0] = d / (float)(K * (K - 1));
                losses[1] = c / (float)K;
                if (PEER) *peer.epoch = epoch;  // every CTA has read the counter (it arrived above); next launch sees epoch
            }
        }
    }
    if (PEER) peer_wait(peer, 1, i, epoch);  // no peer still reads this rank's sums: the buffer may be zeroed again
}

// aux layout (floats, zeroed by the caller): [0] arrival counter, [32 .. 32 + K*32) dz rows
template <bool PEER>
__global__ void __launch_bounds__(UP_THREADS) update_bwd_kernel(const float* __restrict__ dM_new, const float* __restrict__ g_div,
                                                                const float* __restrict__ g_cls, const float* __restrict__ M_new,
                                                                const float* __restrict__ saved, const float* __restrict__ W,
                                                                const float* __restrict__ bias, float momentum,
                                                                float* __restrict__ dS, PeerCtx peer, float* __restrict__ dW,
                                                                float* __restrict__ db, float* __restrict__ aux, int C,
                                                                int K) {
    __shared__ float scratch[UP_WARPS * 32];
    __shared__ float red[32], red2[32];
    __shared__ float dzs[UP_KMAX * UP_KMAX];
    __shared__ int is_last;
    const int tid = threadIdx.x, lane = tid & 31, i = blockIdx.x;
    const bool on = tid < C;
    const float gd = g_div ? __ldg(g_div) : 0.f, gc = g_cls ? __ldg(g_cls) : 0.f;
    float m[UP_KMAX], wv[UP_KMAX], pz[UP_KMAX], pg[UP_KMAX];
#pragma unroll
    for (int k = 0; k < UP_KMAX; ++k) {
        m[k] = (k < K && on) ? __ldg(M_new + (size_t)k * C + tid) : 0.f;
        wv[k] = (k < K && on) ? __ldg(W + (size_t)k * C + tid) : 0.f;
    }
    const float up = (dM_new != nullptr && on) ? __ldg(dM_new + (size_t)i * C + tid) : 0.f;
    const float nrm = saved[i], Dn = saved[K + i];
    float mi = 0.f;
#pragma unroll
    for (int k = 0; k < UP_KMAX; ++k)
        if (k == i) mi = m[k];
#pragma unroll
    for (int k = 0; k < UP_KMAX; ++k) {
        pz[k] = mi * wv[k];
        pg[k] = mi * m[k];
    }
    block_reduce32(pz, scratch, red);
    block_reduce32(pg, scratch, red2);
    if (tid < 32) {  // dz_i = g_cls (softmax(z_i) - e_i) / K ; Gram indicator scaled by g_div 2/(K(K-1))
        const float z = lane < K ? red[lane] + __ldg(bias + lane) : -INFINITY;
        const float mx = warp_max(z);
        const float e = lane < K ? expf(z - mx) : 0.f;
        const float sum = warp_sum(e);
        const float dz = lane < K ? (gc / (float)K) * (e / sum - (lane == i ? 1.f : 0.f)) : 0.f;
        const float g = red2[lane];
        // the reference zeroes only cos < 0 (memory.py:269-271)
        const float gi = (lane < K && lane != i && g >= 0.f) ? gd * 2.f / (float)(K * (K - 1)) : 0.f;
        red[lane] = dz;
        red2[lane] = gi;
        aux[32 + i * UP_KMAX + lane] = dz;
    }
    __syncthreads();
    // dM''_i[c], projection through the normalisation, scale into dS_i
    float a = up;
#pragma unroll
    for (int k = 0; k < UP_KMAX; ++k) {
        a = fmaf(red2[k], m[k], a);
        a = fmaf(red[k], wv[k], a);
    }
    float dot = warp_sum(a * mi);
    if (lane == 0) scratch[tid >> 5] = dot;
    __syncthreads();
    dot = 0.f;
#pragma unroll
    for (int w = 0; w < UP_WARPS; ++w) dot += scratch[w];
    {
        const float inv = 1.f / fmaxf(nrm, PM_NORM_EPS);
        const float coef = (Dn != 0.f) ? (1.f - momentum) / Dn : 0.f;
        const float dmp = (nrm <= PM_NORM_EPS) ? a * inv : (a - mi * dot) * inv;
        if (!PEER) {
            if (on) dS[(size_t)i * C + tid] = coef * dmp;
        } else {
            // this rank's share goes into its symmetric buffer; row i is then summed over the ranks (rank order) out of
            // the peers' buffers into dS -- the gradient of the GLOBAL class sums, identical on every rank
            const unsigned epoch = *peer.epoch + 1;
            float* mine = reinterpret_cast<float*>(peer.bufs[peer.rank] + PM_PEER_DS_OFF);
            if (on) mine[(size_t)i * C + tid] = coef * dmp;
            peer_signal(peer, 2, i, epoch);
            peer_wait(peer, 2, i, epoch);
            float acc = 0.f;
            for (int r = 0; r < peer.world; ++r) {
                const volatile float* P = reinterpret_cast<const volatile float*>(peer.bufs[r] + PM_PEER_DS_OFF);
                if (on) acc += P[(size_t)i * C + tid];
            }
            if (on) dS[(size_t)i * C + tid] = acc;
            peer_signal(peer, 3, i, epoch);
            peer_wait(peer, 3, i, epoch);   // nobody still reads this rank's row: the next launch may overwrite it
        }
    }
    // the last row to arrive turns the dz rows into dW = dz^T M_new and db
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const unsigned t = atomicAdd(reinterpret_cast<unsigned*>(aux), 1u);
        is_last = (t == (unsigned)K - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        for (int q = tid; q < K * UP_KMAX; q += UP_THREADS) dzs[q] = __ldcg(aux + 32 + q);
        __syncthreads();
        for (int j = 0; j < K; ++j) {
            float acc = 0.f;
#pragma unroll
            for (int k = 0; k < UP_KMAX; ++k) acc = fmaf(k < K ? dzs[k * UP_KMAX + j] : 0.f, m[k], acc);
            if (on) dW[(size_t)j * C + tid] = acc;
        }
        if (tid < K) {
            float acc = 0.f;
            for (int k = 0; k < K; ++k) acc += dzs[k * UP_KMAX + tid];
            db[tid] = acc;
        }
        if (PEER && tid == 0) *peer.epoch = *peer.epoch + 1;  // last CTA: every other CTA has read the counter already
    }
}

// ------------------------------------------------------------------------------------------ dispatch

template <typename T, int C, int KP>
int launch_write_reduce(const void* f, const void* labels, int lab_u8, float* SD, int B, int h, int w, int Hm, int Wm, int K,
                        cudaStream_t st, float* part, int* ncta) {
    constexpr int LD = WR_P + 1, CS = C + 4;
    const size_t smem = sizeof(float) * ((size_t)KP * CS + (size_t)C * LD + (C / 32) * WR_P + WR_P + 8 * WR_P);
    auto kern = part ? write_reduce_kernel<T, C, KP, true> : write_reduce_kernel<T, C, KP>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const int hw = h * w, tiles = (hw + WR_P - 1) / WR_P, ntiles = B * tiles;
    int grid = 148 * 2;
    if (grid > ntiles) grid = ntiles;
    if (part) SD = part, *ncta = grid;  // (grid <= PM_ORD_CTAS already)
    // down-sampling the label map to the feature grid: scale = (Hm-1)/(h-1)  (in = labels, out = features)
    const float sy = h > 1 ? (float)(Hm - 1) / (float)(h - 1) : 0.f;
    const float sx = w > 1 ? (float)(Wm - 1) / (float)(w - 1) : 0.f;
    kern<<<grid, C, smem, st>>>((const T*)f, labels, lab_u8, SD, h, w, Hm, Wm, K, sy, sx, tiles, ntiles);
    PM_CHECK_LAUNCH();
    return 0;
}

template <typename T, int CW, int KP>
int launch_write_bwd(const float* dS, const void* f, const void* labels, int lab_u8, void* df, int B, int h, int w, int Hm,
                     int Wm, int K, cudaStream_t st) {
    constexpr int C = CW * WB_WARPS;
    const size_t smem = sizeof(float) * ((size_t)KP * (C + 1) + WB_WARPS * WB_P + 2 * WB_P);
    auto kern = write_bwd_kernel<T, CW, KP>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const int hw = h * w, tiles = (hw + WB_P - 1) / WB_P;
    const float sy = h > 1 ? (float)(Hm - 1) / (float)(h - 1) : 0.f;
    const float sx = w > 1 ? (float)(Wm - 1) / (float)(w - 1) : 0.f;
    kern<<<B * tiles, WB_THREADS, smem, st>>>(dS, (const T*)f, labels, lab_u8, (T*)df, h, w, Hm, Wm, K, sy,
                                               sx, tiles);
    PM_CHECK_LAUNCH();
    return 0;
}

}  // namespace pm

#define PMW_DISPATCH_CW(T, KP, FN, ...)                  \
    switch (C) {                                         \
        case 32: return pm::FN<T, 4, KP>(__VA_ARGS__);   \
        case 64: return pm::FN<T, 8, KP>(__VA_ARGS__);   \
        case 128: return pm::FN<T, 16, KP>(__VA_ARGS__); \
        case 256: return pm::FN<T, 32, KP>(__VA_ARGS__); \
        default: return PM_ERR_CHANNELS;                 \
    }
#define PMW_DISPATCH_C(T, KP, FN, ...)                    \
    switch (C) {                                          \
        case 32: return pm::FN<T, 32, KP>(__VA_ARGS__);   \
        case 64: return pm::FN<T, 64, KP>(__VA_ARGS__);   \
        case 128: return pm::FN<T, 128, KP>(__VA_ARGS__); \
        case 256: return pm::FN<T, 256, KP>(__VA_ARGS__); \
        default: return PM_ERR_CHANNELS;                  \
    }
#define PMW_DISPATCH(MACRO, FN, ...)                                   \
    do {                                                               \
        if (dtype == PM_F32) {                                         \
            if (K <= 19) { MACRO(float, 20, FN, __VA_ARGS__) }         \
            else { MACRO(float, 32, FN, __VA_ARGS__) }                 \
        } else if (dtype == PM_BF16) {                                 \
            if (K <= 19) { MACRO(__nv_bfloat16, 20, FN, __VA_ARGS__) } \
            else { MACRO(__nv_bfloat16, 32, FN, __VA_ARGS__) }         \
        }                                                              \
        return PM_ERR_DTYPE;                                           \
    } while (0)

static int check_write(int B, int C, int h, int w, int Hm, int Wm, int K, int dtype) {
    if (dtype != PM_F32 && dtype != PM_BF16) return PM_ERR_DTYPE;
    if (C != 32 && C != 64 && C != 128 && C != 256) return PM_ERR_CHANNELS;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (B <= 0 || h <= 0 || w <= 0 || Hm <= 0 || Wm <= 0 || (long long)B * h * w > 0x7fffffffLL / 64)
        return PM_ERR_SHAPE;
    return 0;
}

static int write_reduce_any(const void* f, const void* labels, int lab_u8, float* SD, int B, int C, int h, int w, int Hm,
                            int Wm, int K, int dtype, void* stream, float* part = nullptr, int* ncta = nullptr) {
    if (!f || !labels || !SD) return PM_ERR_NULL;
    if (int e = check_write(B, C, h, w, Hm, Wm, K, dtype)) return e;
    if ((uintptr_t)SD & 15) return PM_ERR_ALIGN;
    if (pm::tiled_ok(f, nullptr, nullptr, h * w, dtype))
        return pm::write_reduce_tiled(f, labels, lab_u8, SD, B, C, h, w, Hm, Wm, K, dtype, (cudaStream_t)stream, part, ncta);
    PMW_DISPATCH(PMW_DISPATCH_C, launch_write_reduce, f, labels, lab_u8, SD, B, h, w, Hm, Wm, K, (cudaStream_t)stream, part,
                 ncta);
}

// ordered: every CTA stores its [K+1][C+4] tile to `scratch`, then one fixed-order reduction adds them into SD
static int write_reduce_ordered(const void* f, const void* labels, int lab_u8, float* SD, float* scratch, int B, int C, int h,
                                int w, int Hm, int Wm, int K, int dtype, void* stream) {
    if (!scratch) return PM_ERR_NULL;
    if ((uintptr_t)scratch & 15) return PM_ERR_ALIGN;
    int ncta = 0;
    if (int rc = write_reduce_any(f, labels, lab_u8, SD, B, C, h, w, Hm, Wm, K, dtype, stream, scratch, &ncta)) return rc;
    return pm::reduce_partials_f32(SD, scratch, ncta, (long long)(K + 1) * (C + 4), (cudaStream_t)stream);
}

static int write_bwd_any(const float* dS, const void* f, const void* labels, int lab_u8, void* df, int B, int C, int h, int w,
                         int Hm, int Wm, int K, int dtype, void* stream) {
    if (!dS || !f || !labels || !df) return PM_ERR_NULL;
    if (int e = check_write(B, C, h, w, Hm, Wm, K, dtype)) return e;
    if (pm::tiled_ok(f, df, nullptr, h * w, dtype))
        return pm::write_bwd_tiled(dS, f, labels, lab_u8, df, B, C, h, w, Hm, Wm, K, dtype, (cudaStream_t)stream);
    PMW_DISPATCH(PMW_DISPATCH_CW, launch_write_bwd, dS, f, labels, lab_u8, df, B, h, w, Hm, Wm, K, (cudaStream_t)stream);
}

extern "C" int pm_write_reduce_fwd(const void* f, const int64_t* labels, float* SD, int B, int C, int h, int w, int Hm,
                                   int Wm, int K, int dtype, void* stream) {
    return write_reduce_any(f, labels, 0, SD, B, C, h, w, Hm, Wm, K, dtype, stream);
}
extern "C" int pm_write_reduce_fwd8(const void* f, const uint8_t* lab8, float* SD, int B, int C, int h, int w, int Hm,
                                    int Wm, int K, int dtype, void* stream) {
    return write_reduce_any(f, lab8, 1, SD, B, C, h, w, Hm, Wm, K, dtype, stream);
}
extern "C" int pm_write_reduce_scratch_bytes(int B, int C, int h, int w, int K) {
    if (C != 32 && C != 64 && C != 128 && C != 256) return PM_ERR_CHANNELS;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (B <= 0 || h <= 0 || w <= 0 || (long long)B * h * w > 0x7fffffffLL / 64) return PM_ERR_SHAPE;
    const long long ntiles = (long long)B * ((h * w + 31) / 32);   // 32-pixel tiles in every variant
    const long long ncta = ntiles < pm::PM_ORD_CTAS ? ntiles : pm::PM_ORD_CTAS;
    return (int)(ncta * (K + 1) * (C + 4) * (long long)sizeof(float));
}
extern "C" int pm_write_reduce_fwd_ordered(const void* f, const int64_t* labels, float* SD, float* scratch, int B, int C, int h,
                                           int w, int Hm, int Wm, int K, int dtype, void* stream) {
    return write_reduce_ordered(f, labels, 0, SD, scratch, B, C, h, w, Hm, Wm, K, dtype, stream);
}
extern "C" int pm_write_reduce_fwd8_ordered(const void* f, const uint8_t* lab8, float* SD, float* scratch, int B, int C, int h,
                                            int w, int Hm, int Wm, int K, int dtype, void* stream) {
    return write_reduce_ordered(f, lab8, 1, SD, scratch, B, C, h, w, Hm, Wm, K, dtype, stream);
}
extern "C" int pm_write_bwd(const float* dS, const void* f, const int64_t* labels, void* df, int B, int C, int h, int w,
                            int Hm, int Wm, int K, int dtype, void* stream) {
    return write_bwd_any(dS, f, labels, 0, df, B, C, h, w, Hm, Wm, K, dtype, stream);
}
extern "C" int pm_write_bwd8(const float* dS, const void* f, const uint8_t* lab8, void* df, int B, int C, int h, int w,
                             int Hm, int Wm, int K, int dtype, void* stream) {
    return write_bwd_any(dS, f, lab8, 1, df, B, C, h, w, Hm, Wm, K, dtype, stream);
}

// the writing net's fused passes (fp32, pipelined kernels only: 16-byte rows and pointers)
static int write_bn_fwd_any(const void* z, const void* x, const void* labels, int lab_u8, float* SD, float* scratch,
                            const double* stats, double count, const double* count_dev, float eps, const float* gamma,
                            const float* beta, float* mean_out, float* invstd_out, float* running_mean, float* running_var,
                            float momentum, long long* num_batches_tracked, int B, int C, int h, int w, int Hm, int Wm, int K,
                            void* stream) {
    if (!z || !x || !labels || !SD || !stats || !gamma || !beta || !mean_out || !invstd_out ||
        ((running_mean == nullptr) != (running_var == nullptr)))
        return PM_ERR_NULL;
    if (int e = check_write(B, C, h, w, Hm, Wm, K, PM_F32)) return e;
    if (!(count > 0.0)) return PM_ERR_SHAPE;
    if (((uintptr_t)SD | (uintptr_t)scratch) & 15) return PM_ERR_ALIGN;
    if (!pm::tiled_ok(z, x, nullptr, h * w, PM_F32)) return PM_ERR_ALIGN;
    const pm::BnFinalize fin{stats, count_dev, count, eps, momentum, mean_out, invstd_out, running_mean, running_var,
                             num_batches_tracked};
    cudaStream_t st = (cudaStream_t)stream;
    int ncta = 0;
    if (int rc = pm::write_reduce_bn((const float*)z, (const float*)x, labels, lab_u8, SD, B, C, h, w, Hm, Wm, K, gamma, beta,
                                     fin, st, scratch, scratch ? &ncta : nullptr))
        return rc;
    return scratch ? pm::reduce_partials_f32(SD, scratch, ncta, (long long)(K + 1) * (C + 4), st) : 0;
}
extern "C" int pm_write_reduce_bn_fwd(const void* z, const void* x, const void* labels, int lab_u8, float* SD, const double* stats,
                                      double count, const double* count_dev, float eps, const float* gamma, const float* beta,
                                      float* mean_out, float* invstd_out, float* running_mean, float* running_var, float momentum,
                                      long long* num_batches_tracked, int B, int C, int h, int w, int Hm, int Wm, int K,
                                      void* stream) {
    return write_bn_fwd_any(z, x, labels, lab_u8, SD, nullptr, stats, count, count_dev, eps, gamma, beta, mean_out, invstd_out,
                            running_mean, running_var, momentum, num_batches_tracked, B, C, h, w, Hm, Wm, K, stream);
}
extern "C" int pm_write_reduce_bn_fwd_ordered(const void* z, const void* x, const void* labels, int lab_u8, float* SD,
                                              float* scratch, const double* stats, double count, const double* count_dev, float eps,
                                              const float* gamma, const float* beta, float* mean_out, float* invstd_out,
                                              float* running_mean, float* running_var, float momentum,
                                              long long* num_batches_tracked, int B, int C, int h, int w, int Hm, int Wm, int K,
                                              void* stream) {
    if (!scratch) return PM_ERR_NULL;
    return write_bn_fwd_any(z, x, labels, lab_u8, SD, scratch, stats, count, count_dev, eps, gamma, beta, mean_out, invstd_out,
                            running_mean, running_var, momentum, num_batches_tracked, B, C, h, w, Hm, Wm, K, stream);
}
extern "C" int pm_write_bwd_bn_scratch_bytes(int C) {
    if (C != 32 && C != 64 && C != 128 && C != 256) return PM_ERR_CHANNELS;
    return pm::write_bwd_bn_scratch_floats(C) * (int)sizeof(float);
}
extern "C" int pm_write_bwd_bn(const float* dS, const void* z, const void* x, const void* labels, int lab_u8, const float* mean,
                               const float* invstd, const float* gamma, const float* beta, void* g, float* dgamma, float* dbeta,
                               float* scratch, int B, int C, int h, int w, int Hm, int Wm, int K, void* stream) {
    if (!dS || !z || !x || !labels || !mean || !invstd || !gamma || !beta || !g || !dgamma || !dbeta || !scratch)
        return PM_ERR_NULL;
    if (int e = check_write(B, C, h, w, Hm, Wm, K, PM_F32)) return e;
    if (!pm::tiled_ok(z, x, g, h * w, PM_F32) || ((uintptr_t)scratch & 15)) return PM_ERR_ALIGN;
    return pm::write_bwd_bn(dS, (const float*)z, (const float*)x, labels, lab_u8, mean, invstd, gamma, beta, (float*)g, dgamma,
                            dbeta, scratch, B, C, h, w, Hm, Wm, K, (cudaStream_t)stream);
}

extern "C" int pm_update_aux_floats(int K) { return 32 + K * pm::UP_KMAX + 68; }

extern "C" int pm_update_fwd(const float* SD, const float* M_old, float momentum, const float* W_cls,
                             const float* b_cls, float* M_new, float* losses, float* saved, float* aux, int C, int K,
                             void* stream) {
    if (!SD || !M_old || !W_cls || !b_cls || !M_new || !losses || !saved || !aux) return PM_ERR_NULL;
    if (C != 32 && C != 64 && C != 128 && C != 256) return PM_ERR_CHANNELS;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    pm::update_fwd_kernel<false><<<K, pm::UP_THREADS, 0, (cudaStream_t)stream>>>(SD, pm::PeerCtx{nullptr, 0, 1, nullptr}, nullptr,
                                                                                 M_old, momentum, W_cls, b_cls, M_new, losses,
                                                                                 saved, aux, C, K);
    PM_CHECK_LAUNCH();
    return 0;
}

extern "C" int pm_peer_buffer_bytes(void) { return PM_PEER_BYTES; }

extern "C" int pm_update_fwd_peer(const void* peer_bufs, int rank, int world, unsigned* epoch, float* SD_sum,
                                  const float* M_old, float momentum, const float* W_cls, const float* b_cls, float* M_new,
                                  float* losses, float* saved, float* aux, int C, int K, void* stream) {
    if (!peer_bufs || !epoch || !M_old || !W_cls || !b_cls || !M_new || !losses || !saved || !aux) return PM_ERR_NULL;
    if (C != 32 && C != 64 && C != 128 && C != 256) return PM_ERR_CHANNELS;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (world < 1 || world > 16 || rank < 0 || rank >= world) return PM_ERR_SHAPE;
    pm::PeerCtx p{(const unsigned long long*)peer_bufs, rank, world, epoch};
    pm::update_fwd_kernel<true><<<K, pm::UP_THREADS, 0, (cudaStream_t)stream>>>(nullptr, p, SD_sum, M_old, momentum, W_cls, b_cls,
                                                                                M_new, losses, saved, aux, C, K);
    PM_CHECK_LAUNCH();
    return 0;
}

extern "C" int pm_update_bwd(const float* dM_new, const float* g_div, const float* g_cls, const float* M_new,
                             const float* saved, const float* W_cls, const float* b_cls, float momentum, float* dS,
                             float* dW_cls, float* db_cls, float* aux, int C, int K, void* stream) {
    if (!M_new || !saved || !W_cls || !b_cls || !dS || !dW_cls || !db_cls || !aux) return PM_ERR_NULL;
    if (C != 32 && C != 64 && C != 128 && C != 256) return PM_ERR_CHANNELS;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    pm::update_bwd_kernel<false><<<K, pm::UP_THREADS, 0, (cudaStream_t)stream>>>(dM_new, g_div, g_cls, M_new, saved, W_cls, b_cls,
                                                                                 momentum, dS, pm::PeerCtx{nullptr, 0, 1, nullptr},
                                                                                 dW_cls, db_cls, aux, C, K);
    PM_CHECK_LAUNCH();
    return 0;
}

extern "C" int pm_update_bwd_peer(const void* peer_bufs, int rank, int world, unsigned* epoch, const float* dM_new,
                                  const float* g_div, const float* g_cls, const float* M_new, const float* saved,
                                  const float* W_cls, const float* b_cls, float momentum, float* dS, float* dW_cls,
                                  float* db_cls, float* aux, int C, int K, void* stream) {
    if (!peer_bufs || !epoch || !M_new || !saved || !W_cls || !b_cls || !dS || !dW_cls || !db_cls || !aux) return PM_ERR_NULL;
    if (C != 32 && C != 64 && C != 128 && C != 256) return PM_ERR_CHANNELS;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (world < 1 || world > 16 || rank < 0 || rank >= world) return PM_ERR_SHAPE;
    pm::PeerCtx p{(const unsigned long long*)peer_bufs, rank, world, epoch};
    pm::update_bwd_kernel<true><<<K, pm::UP_THREADS, 0, (cudaStream_t)stream>>>(dM_new, g_div, g_cls, M_new, saved, W_cls, b_cls,
                                                                                momentum, dS, p, dW_cls, db_cls, aux, C, K);
    PM_CHECK_LAUNCH();
    return 0;
}

extern "C" int pm_version(void) { return PM_ABI_VERSION; }

extern "C" const char* pm_status_string(int code) {
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    switch (code) {
        case PM_OK: return "ok";
        case PM_ERR_NULL: return "a required pointer is NULL";
        case PM_ERR_DTYPE: return "dtype must be PM_F32 (0) or PM_BF16 (1); PM_F32_TF32 (2) only for the pm_conv1x1_* entries";
        case PM_ERR_CHANNELS: return "C (mem_dim) must be one of 32, 64, 128, 256";
        case PM_ERR_SLOTS: return "K (mem_slot) must be in 1..31";
        case PM_ERR_SHAPE: return "a dimension is <= 0 or too large";
        case PM_ERR_ALIGN: return "a pointer is not aligned as documented";
        default: return "unknown pinmem_b200 status";
    }
}
