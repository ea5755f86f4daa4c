// Internal cross-file declarations (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace pm {

// true when the pipelined (TMA / 16-byte async copy) kernels can be used for these feature pointers
bool tiled_ok(const void* p0, const void* p1, const void* p2, int hw, int dtype);

int read_fwd_tiled(const void* x, const float* M, const float* gum_m, const float* gum_q, void* u, float* s, float* p,
                   float* colpart, int B, int C, int hw, int K, int dtype, int planes, cudaStream_t st);

// needs a [N][stride] ds buffer (never NULL); dx_add: NULL, or a second gradient of x to sum into dx
int read_bwd_tiled(const void* du, const void* x, const float* M, const float* p, const float* ds_rl,
                   const float* g_loss, const float* rl_out, void* dx, const void* dx_add, float* ds, int B, int C, int hw,
                   int K, int dtype, int planes, cudaStream_t st);

// part != NULL: the ordered instantiation stores each CTA's [K+1][C+4] tile to part[blockIdx.x] and sets *ncta to the
// grid size (at most PM_ORD_CTAS) instead of adding into SD
int write_reduce_tiled(const void* f, const void* labels, int lab_u8, float* SD, int B, int C, int h, int w, int Hm, int Wm,
                       int K, int dtype, cudaStream_t st, float* part = nullptr, int* ncta = nullptr);

// CTA cap of the ordered class-sum kernels: bounds their partial scratch (persistent CTAs take the tiles in turn)
constexpr int PM_ORD_CTAS = 296;

// pm_ordered.cu: dst[i] += sum_g part[g*n + i] with g ascending
int reduce_partials_f32(float* dst, const float* part, int G, long long n, cudaStream_t st);
int reduce_partials_f64(double* dst, const double* part, int G, long long n, cudaStream_t st);
// ds_rl and the loss of the ordered read-loss kernels from their stored tap tiles ([ncta][(TY+1)][(TX+1)][KP]) and
// per-CTA loss partials (log2 units)
int readloss_gather(const float* tiles, const float* lossp, int ncta, int B, int h, int w, int KP, int TY, int TX, int tiles_x,
                    int tiles_y, int K, float temperature, float* ds_rl, unsigned long long* ws, float* out, cudaStream_t st);

int write_bwd_tiled(const float* dS, const void* f, const void* labels, int lab_u8, void* df, int B, int C, int h, int w, int Hm,
                    int Wm, int K, int dtype, cudaStream_t st);

struct BnFinalize;
// pm_write_tiled.cu, fp32: the writing net's fused class sums (f = relu(x + BN(z)) formed from the z and x maps; `fin` finalises
// the statistics, CTA 0 publishes them) and write backward (g = df * [f > 0] into g, then dgamma / dbeta from the per-CTA
// partials in `part`, write_bwd_bn_scratch_floats(C) floats)
int write_reduce_bn(const float* z, const float* x, const void* labels, int lab_u8, float* SD, int B, int C, int h, int w, int Hm,
                    int Wm, int K, const float* gamma, const float* beta, const BnFinalize& fin, cudaStream_t st,
                    float* part = nullptr, int* ncta = nullptr);
int write_bwd_bn_scratch_floats(int C);
int write_bwd_bn(const float* dS, const float* z, const float* x, const void* labels, int lab_u8, const float* mean,
                 const float* invstd, const float* gamma, const float* beta, float* g, float* dgamma, float* dbeta, float* part,
                 int B, int C, int h, int w, int Hm, int Wm, int K, cudaStream_t st);

// fills `partial` ([PM_COLPART_ROWS][64]: max at [k], sum at [32+k]) from s (+ gumbel_q) and combines them (row PM_COLPART_ROWS)
int colsoftmax_stats(const float* s, const float* gumbel_q, float* partial, int N, int K, cudaStream_t st);

}  // namespace pm
