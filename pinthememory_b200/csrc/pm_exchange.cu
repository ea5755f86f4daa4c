// Global-batch read for sharded runs: the read loss (memory.py:173-176) and score_query (memory.py:183,186-187) over the
// concatenated batch of all ranks. Each rank contributes one small row (layout: include/pinmem_b200.h, PM_READ_ROW_FLOATS);
// a one-CTA kernel combines the rows of all ranks in rank order, reading them either straight out of the peers' symmetric
// buffers over NVLink (flags kinds 4..7, pm_common.cuh) or out of a local [world][row] tensor an NCCL all-gather filled.
// Both paths run the same combine code, so the result and its bit-identity across ranks do not depend on the path.
#include "pm_common.cuh"
#include "pm_internal.h"

namespace pm {

constexpr int RX_THREADS = 64;  // threads 0..31: one column each; thread 32: the scalars
constexpr int RX_FWD = 4, RX_FWD_DONE = 5, RX_BWD = 6, RX_BWD_DONE = 7;

static_assert(PM_PEER_FLAG_OFF + 8 * 32 * 16 * 4 <= PM_PEER_READ_FWD_OFF, "read rows overlap the flag area");
static_assert(PM_PEER_READ_FWD_OFF + PM_READ_ROW_FLOATS * 4 <= PM_PEER_READ_BWD_OFF, "read rows overlap");
static_assert(PM_PEER_READ_BWD_OFF + PM_READ_ROW_FLOATS * 4 <= PM_PEER_BYTES, "read rows past the peer buffer");

// ---- forward row: [0,32) column maximum, [32,64) column sum, doubles at float 64: read-loss sum, valid count V
__device__ __forceinline__ void fwd_pack(const float* __restrict__ colpart, const unsigned long long* __restrict__ ws,
                                         float* row, int K) {
    const int t = threadIdx.x;
    if (t < K) {
        row[t] = __ldcg(colpart + (size_t)PM_COLPART_ROWS * 64 + t);
        row[32 + t] = 1.f / __ldcg(colpart + (size_t)PM_COLPART_ROWS * 64 + 32 + t);
    }
    if (t == 32) {
        double loss = 0.0, V = 0.0;
        if (ws != nullptr) {  // every read-loss kernel leaves the fp64 loss sum and the label histogram here
            loss = __longlong_as_double((long long)__ldcg(ws + PM_WS_LOSS_SUM));
            unsigned long long v = 0;
            for (int k = 0; k < K; ++k) v += __ldcg(ws + PM_WS_HIST + k);
            V = (double)v;
        }
        double* d = reinterpret_cast<double*>(row + 64);
        d[0] = loss;
        d[1] = V;
    }
}

// rows(r) -> row of rank r; m = max_r m_r, S = sum_r S_r exp(m_r - m) (rank order, fp32, the column softmax's expf)
template <typename Rows>
__device__ __forceinline__ void fwd_combine(Rows rows, int world, float* __restrict__ colpart, float temperature,
                                            float* __restrict__ out, int K) {
    const int t = threadIdx.x;
    if (t < K) {
        float m = -INFINITY;
        for (int r = 0; r < world; ++r) m = fmaxf(m, rows(r)[t]);
        float S = 0.f;
        for (int r = 0; r < world; ++r) {
            const float mr = rows(r)[t];
            if (mr > -INFINITY) S += rows(r)[32 + t] * expf(mr - m);
        }
        colpart[(size_t)PM_COLPART_ROWS * 64 + t] = m;
        colpart[(size_t)PM_COLPART_ROWS * 64 + 32 + t] = 1.f / S;
    }
    if (t == 32 && out != nullptr) {
        double loss = 0.0, V = 0.0;
        for (int r = 0; r < world; ++r) {
            const volatile double* d = reinterpret_cast<const volatile double*>(rows(r) + 64);
            loss += d[0];
            V += d[1];
        }
        out[0] = (float)(loss / V);  // V == 0 -> 0/0 = NaN like torch (no valid pixel in the whole global batch)
        out[1] = (float)(1.0 / (V * (double)temperature));
    }
}

// ---- backward row: doubles [0] upstream gradient of readloss, [1, 1+K) the rank's column sums c_k
__device__ __forceinline__ void bwd_pack(const double* __restrict__ part, const float* __restrict__ g_loss, double* row, int K) {
    const int t = threadIdx.x;
    if (t < K) {
        // the order of pm_score_bwd's own combine (pm_common.cuh): the group terms, then the groups in ascending order
        double c = 0.0;
        if (part != nullptr)
            for (int j = 0; j < SB_GROUPS; ++j) c += sb_group_sum(part, t, j);
        row[1 + t] = c;
    }
    if (t == 32) row[0] = g_loss != nullptr ? (double)__ldg(g_loss) : 0.0;
}

template <typename Rows>
__device__ __forceinline__ void bwd_combine(Rows rows, int world, float* __restrict__ g_loss_sum, double* __restrict__ colsums,
                                            int K) {
    const int t = threadIdx.x;
    if (t < 32) {
        double c = 0.0;
        if (t < K)
            for (int r = 0; r < world; ++r) c += rows(r)[1 + t];
        colsums[t] = c;
    }
    if (t == 32) {
        double g = 0.0;
        for (int r = 0; r < world; ++r) g += rows(r)[0];
        *g_loss_sum = (float)g;
    }
}

__device__ __forceinline__ const volatile float* peer_row_f(const PeerCtx& p, int r, int off) {
    return reinterpret_cast<const volatile float*>(p.bufs[r] + off);
}

// The "done" round of launch e-1 is waited for at the START of launch e (before the row is overwritten), so a launch
// returns as soon as it has combined; epoch 0 (nothing before) passes at once on the zeroed flags.
__global__ void __launch_bounds__(RX_THREADS) read_xchg_fwd_peer_kernel(PeerCtx p, float* __restrict__ colpart,
                                                                        const unsigned long long* __restrict__ ws,
                                                                        float temperature, float* __restrict__ out, int K) {
    const unsigned e = *p.epoch + 1;
    peer_wait(p, RX_FWD_DONE, 0, e - 1);
    fwd_pack(colpart, ws, reinterpret_cast<float*>(p.bufs[p.rank] + PM_PEER_READ_FWD_OFF), K);
    peer_signal(p, RX_FWD, 0, e);
    peer_wait(p, RX_FWD, 0, e);
    fwd_combine([&](int r) { return peer_row_f(p, r, PM_PEER_READ_FWD_OFF); }, p.world, colpart, temperature, out, K);
    peer_signal(p, RX_FWD_DONE, 0, e);
    if (threadIdx.x == 0) *p.epoch = e;
}

__global__ void __launch_bounds__(RX_THREADS) read_xchg_fwd_gathered_kernel(const float* __restrict__ gathered, int world,
                                                                            float* __restrict__ colpart, float temperature,
                                                                            float* __restrict__ out, int K) {
    fwd_combine([&](int r) { return gathered + (size_t)r * PM_READ_ROW_FLOATS; }, world, colpart, temperature, out, K);
}

__global__ void __launch_bounds__(RX_THREADS) read_row_fwd_kernel(const float* __restrict__ colpart,
                                                                  const unsigned long long* __restrict__ ws,
                                                                  float* __restrict__ row, int K) {
    fwd_pack(colpart, ws, row, K);
}

__global__ void __launch_bounds__(RX_THREADS) read_xchg_bwd_peer_kernel(PeerCtx p, const double* __restrict__ part,
                                                                        const float* __restrict__ g_loss,
                                                                        float* __restrict__ g_loss_sum,
                                                                        double* __restrict__ colsums, int K) {
    const unsigned e = *p.epoch + 1;
    peer_wait(p, RX_BWD_DONE, 0, e - 1);
    bwd_pack(part, g_loss, reinterpret_cast<double*>(p.bufs[p.rank] + PM_PEER_READ_BWD_OFF), K);
    peer_signal(p, RX_BWD, 0, e);
    peer_wait(p, RX_BWD, 0, e);
    bwd_combine([&](int r) { return reinterpret_cast<const volatile double*>(p.bufs[r] + PM_PEER_READ_BWD_OFF); }, p.world,
                g_loss_sum, colsums, K);
    peer_signal(p, RX_BWD_DONE, 0, e);
    if (threadIdx.x == 0) *p.epoch = e;
}

__global__ void __launch_bounds__(RX_THREADS) read_xchg_bwd_gathered_kernel(const double* __restrict__ gathered, int world,
                                                                            float* __restrict__ g_loss_sum,
                                                                            double* __restrict__ colsums, int K) {
    bwd_combine([&](int r) { return gathered + (size_t)r * (PM_READ_ROW_FLOATS / 2); }, world, g_loss_sum, colsums, K);
}

__global__ void __launch_bounds__(RX_THREADS) read_row_bwd_kernel(const double* __restrict__ part,
                                                                  const float* __restrict__ g_loss, double* __restrict__ row,
                                                                  int K) {
    bwd_pack(part, g_loss, row, K);
}

}  // namespace pm

static int rx_check(const void* peer_bufs, int rank, int world, const unsigned* epoch, const float* gathered, int K) {
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (world < 1 || world > 16) return PM_ERR_SHAPE;
    if (peer_bufs) {
        if (!epoch) return PM_ERR_NULL;
        if (rank < 0 || rank >= world) return PM_ERR_SHAPE;
    } else if (!gathered) {
        return PM_ERR_NULL;
    } else if ((uintptr_t)gathered & 15) {
        return PM_ERR_ALIGN;
    }
    return 0;
}

extern "C" int pm_read_row_fwd(const float* col_partials, const void* ws, float* row, int K, void* stream) {
    if (!col_partials || !row) return PM_ERR_NULL;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (((uintptr_t)row & 15) || ((uintptr_t)ws & 7)) return PM_ERR_ALIGN;
    pm::read_row_fwd_kernel<<<1, pm::RX_THREADS, 0, (cudaStream_t)stream>>>(
        col_partials, (const unsigned long long*)ws, row, K);
    PM_CHECK_LAUNCH();
    return 0;
}

extern "C" int pm_read_row_bwd(const float* partials, const float* g_loss, float* row, int K, void* stream) {
    if (!row) return PM_ERR_NULL;
    if (K < 1 || K > 31) return PM_ERR_SLOTS;
    if (((uintptr_t)row & 15) || ((uintptr_t)partials & 7)) return PM_ERR_ALIGN;
    pm::read_row_bwd_kernel<<<1, pm::RX_THREADS, 0, (cudaStream_t)stream>>>((const double*)partials, g_loss, (double*)row, K);
    PM_CHECK_LAUNCH();
    return 0;
}

extern "C" int pm_read_exchange_fwd(const void* peer_bufs, int rank, int world, unsigned* epoch, const float* gathered,
                                    float* col_partials, const void* ws, float temperature, float* out, int K, void* stream) {
    if (!col_partials || (!ws != !out)) return PM_ERR_NULL;
    if (int e = rx_check(peer_bufs, rank, world, epoch, gathered, K)) return e;
    if ((uintptr_t)ws & 7) return PM_ERR_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    if (peer_bufs) {
        pm::PeerCtx p{(const unsigned long long*)peer_bufs, rank, world, epoch};
        pm::read_xchg_fwd_peer_kernel<<<1, pm::RX_THREADS, 0, st>>>(p, col_partials, (const unsigned long long*)ws, temperature,
                                                                    out, K);
    } else {
        pm::read_xchg_fwd_gathered_kernel<<<1, pm::RX_THREADS, 0, st>>>(gathered, world, col_partials, temperature, out, K);
    }
    PM_CHECK_LAUNCH();
    return 0;
}

extern "C" int pm_read_exchange_bwd(const void* peer_bufs, int rank, int world, unsigned* epoch, const float* gathered,
                                    const float* partials, const float* g_loss, float* g_loss_sum, double* colsums, int K,
                                    void* stream) {
    if (!g_loss_sum || !colsums) return PM_ERR_NULL;
    if (int e = rx_check(peer_bufs, rank, world, epoch, gathered, K)) return e;
    if (((uintptr_t)partials & 7) || ((uintptr_t)colsums & 7)) return PM_ERR_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    if (peer_bufs) {
        pm::PeerCtx p{(const unsigned long long*)peer_bufs, rank, world, epoch};
        pm::read_xchg_bwd_peer_kernel<<<1, pm::RX_THREADS, 0, st>>>(p, (const double*)partials, g_loss, g_loss_sum, colsums, K);
    } else {
        pm::read_xchg_bwd_gathered_kernel<<<1, pm::RX_THREADS, 0, st>>>((const double*)gathered, world, g_loss_sum, colsums, K);
    }
    PM_CHECK_LAUNCH();
    return 0;
}
