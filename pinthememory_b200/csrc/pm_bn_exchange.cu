// SyncBatchNorm over the module's symmetric peer buffers: the two cross-rank sums of the layers convert_sync_batchnorm makes
// of memory.py:76 and :105 (train.py:95, --syncbn). The forward sums the GEMM epilogue's fp64 [sum | sum of squares] and the
// pixel counts, the backward the (dgamma, dbeta) the input gradient needs. One CTA per launch, the read exchange's protocol
// (pm_exchange.cu): rows and flags are laid out in include/pinmem_b200.h, every sum runs over the ranks in rank order in fp64.
#include "pm_common.cuh"

namespace pm {

constexpr int BX_THREADS = 256;
constexpr int BX_KIND = 8;  // flag kind of these exchanges: row 2x arrival, 2x + 1 "done" of exchange x = 2 * slot + direction

static_assert(PM_PEER_FLAG_OFF + BX_KIND * 32 * 16 * 4 == PM_PEER_BN_FLAG_OFF, "kind 8 of the flag area is the BN flag block");
static_assert(PM_PEER_BN_FLAG_OFF + 8 * 16 * 4 <= PM_PEER_READ_FWD_OFF, "BN flags overlap the read rows");
static_assert(PM_PEER_READ_BWD_OFF + PM_READ_ROW_FLOATS * 4 <= PM_PEER_BN_FWD_OFF, "BN rows overlap the read rows");
static_assert(PM_PEER_BN_FWD_OFF + 2 * PM_BN_FWD_ROW_BYTES <= PM_PEER_BN_BWD_OFF, "BN forward rows overlap");
static_assert(PM_PEER_BN_BWD_OFF + 2 * PM_BN_BWD_ROW_BYTES <= PM_PEER_BYTES, "BN rows past the peer buffer");
static_assert((2 * PM_BN_MAX_C + 1) * 8 <= PM_BN_FWD_ROW_BYTES && 2 * PM_BN_MAX_C * 4 <= PM_BN_BWD_ROW_BYTES, "BN rows too small");
static_assert(PM_PEER_BN_FWD_OFF % 16 == 0 && PM_PEER_BN_BWD_OFF % 16 == 0 && PM_BN_FWD_ROW_BYTES % 16 == 0 &&
                  PM_BN_BWD_ROW_BYTES % 16 == 0,
              "BN rows must be 16-byte aligned");

// The "done" round of launch e-1 is waited for at the start of launch e, before the row is overwritten (pm_exchange.cu).
__global__ void __launch_bounds__(BX_THREADS) bn_xchg_fwd_kernel(PeerCtx p, int slot, double* __restrict__ stats, double count,
                                                                 int M) {
    const int x = 2 * slot;
    const int off = PM_PEER_BN_FWD_OFF + slot * PM_BN_FWD_ROW_BYTES;
    const int n = 2 * M + 1;
    const unsigned e = *p.epoch + 1;
    peer_wait(p, BX_KIND, 2 * x + 1, e - 1);
    double* row = reinterpret_cast<double*>(p.bufs[p.rank] + off);
    for (int i = threadIdx.x; i < n; i += BX_THREADS) row[i] = i < 2 * M ? stats[i] : count;
    peer_signal(p, BX_KIND, 2 * x, e);
    peer_wait(p, BX_KIND, 2 * x, e);
    for (int i = threadIdx.x; i < n; i += BX_THREADS) {
        double s = 0.0;
        for (int r = 0; r < p.world; ++r) s += reinterpret_cast<const volatile double*>(p.bufs[r] + off)[i];
        stats[i] = s;
    }
    peer_signal(p, BX_KIND, 2 * x + 1, e);
    if (threadIdx.x == 0) *p.epoch = e;
}

__global__ void __launch_bounds__(BX_THREADS) bn_xchg_bwd_kernel(PeerCtx p, int slot, const float* __restrict__ dgamma,
                                                                 const float* __restrict__ dbeta,
                                                                 const double* __restrict__ count_global, double local_count,
                                                                 float* __restrict__ sg, float* __restrict__ sb, int M) {
    const int x = 2 * slot + 1;
    const int off = PM_PEER_BN_BWD_OFF + slot * PM_BN_BWD_ROW_BYTES;
    const unsigned e = *p.epoch + 1;
    peer_wait(p, BX_KIND, 2 * x + 1, e - 1);
    float* row = reinterpret_cast<float*>(p.bufs[p.rank] + off);
    for (int i = threadIdx.x; i < 2 * M; i += BX_THREADS) row[i] = i < M ? dgamma[i] : dbeta[i - M];
    peer_signal(p, BX_KIND, 2 * x, e);
    peer_wait(p, BX_KIND, 2 * x, e);
    // the input-gradient passes divide by the LOCAL pixel count: hand them the global sums scaled by local / global
    const double scale = local_count / *count_global;
    for (int i = threadIdx.x; i < 2 * M; i += BX_THREADS) {
        double s = 0.0;
        for (int r = 0; r < p.world; ++r) s += (double)reinterpret_cast<const volatile float*>(p.bufs[r] + off)[i];
        const float v = (float)(s * scale);
        if (i < M)
            sg[i] = v;
        else
            sb[i - M] = v;
    }
    peer_signal(p, BX_KIND, 2 * x + 1, e);
    if (threadIdx.x == 0) *p.epoch = e;
}

}  // namespace pm

static int bx_check(const void* peer_bufs, int rank, int world, const unsigned* epoch, int slot, int M) {
    if (!peer_bufs || !epoch) return PM_ERR_NULL;
    if (M < 1 || M > PM_BN_MAX_C) return PM_ERR_SHAPE;
    if (world < 2 || world > 16 || rank < 0 || rank >= world) return PM_ERR_SHAPE;
    if (slot != 0 && slot != 1) return PM_ERR_SHAPE;
    return 0;
}

extern "C" int pm_bn_exchange_fwd(const void* peer_bufs, int rank, int world, unsigned* epoch, int slot, double* stats,
                                  double count, int M, void* stream) {
    if (!stats) return PM_ERR_NULL;
    if (int e = bx_check(peer_bufs, rank, world, epoch, slot, M)) return e;
    if ((uintptr_t)stats & 7) return PM_ERR_ALIGN;
    pm::PeerCtx p{(const unsigned long long*)peer_bufs, rank, world, epoch};
    pm::bn_xchg_fwd_kernel<<<1, pm::BX_THREADS, 0, (cudaStream_t)stream>>>(p, slot, stats, count, M);
    PM_CHECK_LAUNCH();
    return 0;
}

extern "C" int pm_bn_exchange_bwd(const void* peer_bufs, int rank, int world, unsigned* epoch, int slot, const float* dgamma,
                                  const float* dbeta, const double* count_global, double local_count, float* sg, float* sb, int M,
                                  void* stream) {
    if (!dgamma || !dbeta || !count_global || !sg || !sb) return PM_ERR_NULL;
    if (int e = bx_check(peer_bufs, rank, world, epoch, slot, M)) return e;
    if (((uintptr_t)count_global & 7) || (((uintptr_t)dgamma | (uintptr_t)dbeta | (uintptr_t)sg | (uintptr_t)sb) & 3))
        return PM_ERR_ALIGN;
    pm::PeerCtx p{(const unsigned long long*)peer_bufs, rank, world, epoch};
    pm::bn_xchg_bwd_kernel<<<1, pm::BX_THREADS, 0, (cudaStream_t)stream>>>(p, slot, dgamma, dbeta, count_global, local_count,
                                                                           sg, sb, M);
    PM_CHECK_LAUNCH();
    return 0;
}
