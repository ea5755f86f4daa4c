/*
 * pinmem_b200.h -- C ABI of the B200 (sm_100a) categorical-memory kernels.
 *
 * This is the drop-in boundary of the hot path named by BASELINE.json: the reference's
 * `network/memory.py::Memory_sup` (read, get_score, write, diversityloss, classification_loss).
 * The reference is pure PyTorch, so there is no FFI to replace; each entry point below is what a
 * maintainer's binding (ctypes, see INTEGRATION.md) calls instead of the cited eager torch lines.
 * Paths are relative to the reference tree.
 *
 * Conventions
 *   - every function returns 0 on success, a NEGATIVE pm_status on a rejected argument and a POSITIVE
 *     cudaError_t if the launch failed; nothing throws, nothing allocates, nothing synchronises.
 *   - all pointers are DEVICE pointers owned by the caller (PyTorch's caching allocator in the shipped
 *     host side); `stream` is a cudaStream_t passed as void*.
 *   - feature-sized tensors (x, u, f, du, dx, df) are NCHW-contiguous in `dtype` (PM_F32 or PM_BF16);
 *     memory, scores, sums, losses and every accumulation are fp32; labels are int64 [B,Hm,Wm] with
 *     255 = ignore (transforms/transforms.py:95-97).
 *   - C (mem_dim) must be one of 32, 64, 128, 256; K (mem_slot) must be 1..31.
 *   - N = B*h*w. "Score buffers" internal to the path (s, ds_rl, ds) have a padded row stride
 *     pm_score_stride(K) floats so rows are 16-byte aligned; user-visible scores are dense [N,K].
 */
#ifndef PINMEM_B200_H
#define PINMEM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum pm_dtype { PM_F32 = 0, PM_BF16 = 1 };

enum pm_status {
    PM_OK = 0,
    PM_ERR_NULL = -1,      /* a required pointer is NULL */
    PM_ERR_DTYPE = -2,     /* dtype not PM_F32 / PM_BF16 */
    PM_ERR_CHANNELS = -3,  /* C not in {32,64,128,256} */
    PM_ERR_SLOTS = -4,     /* K not in 1..31 */
    PM_ERR_SHAPE = -5,     /* a dimension is <= 0 or too large */
    PM_ERR_ALIGN = -6      /* a pointer is not aligned as documented */
};

/* 64-bit words of the read-loss workspace (`ws`, zero it before pm_readloss_fwd). */
enum pm_readloss_ws_layout {
    PM_WS_LOSS_SUM = 0, /* double: sum over valid label pixels of (LSE - logit[y])            */
    PM_WS_COUNTER = 1,  /* uint64: CTA arrival counter                                         */
    PM_WS_BAD = 2,      /* int64: label values outside [0,K) u {255} (counted as ignore)       */
    PM_WS_HIST = 4,     /* int64[K+1]: label histogram, bin K = ignore; sum(bins<K) = V        */
    PM_WS_WORDS = 40
};

/* Rows of the per-CTA column-softmax partials ([PM_COLPART_ROWS + 2][64] floats; row PM_COLPART_ROWS = combined column
 * maximum | 1/sum, row PM_COLPART_ROWS + 1 = arrival ticket of the fused combine: ZERO on entry, left zero). */
#define PM_COLPART_ROWS 296

/* Bumped with every prototype change; the binding refuses a library whose pm_version() differs. */
#define PM_ABI_VERSION 208
int pm_version(void);
const char* pm_status_string(int code);
/* Row stride (floats) of the internal score buffers for K slots: 20 for K<=19, else 32. */
int pm_score_stride(int K);
/* Floats of the column-softmax partials buffer ((PM_COLPART_ROWS + 2) * 64, layout above). */
int pm_colsoftmax_workspace_floats(int K);

/*
 * Memory read, forward. Replaces memory.py:319-320 (normalise + NCHW->NHWC), :171 (q.M^T),
 * :181-187 dim=1 [gumbel-]softmax, :328 (p.M), :330-332 (cat + NHWC->NCHW).
 *   x        [B,C,h,w] dtype          M         [K,C] fp32
 *   gumbel_m [N,K] fp32 or NULL       (the noise of F.gumbel_softmax(score, dim=1), memory.py:184)
 *   gumbel_q [N,K] fp32 or NULL       (the noise of the dim=0 call, memory.py:183; only used for col_partials)
 *   u        [B,2C,h,w] dtype out     = [x/|x| ; softmax_k(s+g).M]
 *   s        [N,stride] fp32 out      raw similarities (internal score buffer)
 *   score_m  [N,K] fp32 out           softmax over slots (score_memory)
 *   col_partials  NULL, or pm_colsoftmax_workspace_floats(K) floats whose LAST 64 (the ticket row) the caller has
 *                 ZEROED: per-CTA (max,sum) of every column of s + gumbel_q -- the first pass of the dim-0 softmax
 *                 fused into this kernel -- and, from the last CTA to finish, their combination (column maximum and
 *                 1/sum); feed it to pm_colsoftmax_apply.
 */
int pm_read_fwd(const void* x, const float* M, const float* gumbel_m, const float* gumbel_q, void* u, float* s,
                float* score_m, float* col_partials, int B, int C, int h, int w, int K, int dtype, void* stream);

/*
 * score_query = softmax over ALL N pixels (dim 0) of s (+ gumbel_q). memory.py:183/186.
 *   s [N,stride] fp32, gumbel_q [N,K] fp32 or NULL, score_q [N,K] fp32 out,
 *   workspace: pm_colsoftmax_workspace_floats(K) floats of scratch.
 */
int pm_colsoftmax(const float* s, const float* gumbel_q, float* score_q, float* workspace, int N, int K,
                  void* stream);
/* Second pass only: normalise with the combined column statistics pm_read_fwd[_planes] left in col_partials (one
 * launch; the round-1 library combined the partials in a launch of its own here). */
int pm_colsoftmax_apply(const float* s, const float* gumbel_q, const float* col_partials, float* score_q, int N,
                        int K, void* stream);

/*
 * Feature-cohesion (read) loss, forward, plus everything its backward needs. Replaces
 * memory.py:173-176: s/T -> bilinear up-sample (align_corners=True) to [Hm,Wm] -> CrossEntropy
 * (ignore 255, mean over valid pixels) WITHOUT materialising the [B,K,Hm,Wm] logits.
 *   s      [N,stride] fp32          labels [B,Hm,Wm] int64
 *   ds_rl  [N,stride] fp32, ZEROED by the caller; receives sum over label pixels of
 *          bilinear^T (softmax(logits) - onehot(y)) (i.e. d loss_sum / d (s/T))
 *   ws     PM_WS_WORDS 64-bit words, ZEROED by the caller (layout above)
 *   out    float[2] out: out[0] = readloss = loss_sum / V (NaN when V == 0, like torch),
 *                        out[1] = 1 / (V*T)  (scale of ds_rl in the backward)
 */
int pm_readloss_fwd(const float* s, const int64_t* labels, float temperature, int B, int h, int w, int Hm,
                    int Wm, int K, float* ds_rl, void* ws, float* out, void* stream);

/*
 * Memory read, backward (autograd of the lines pm_read_fwd + pm_readloss_fwd replace).
 *   du       [B,2C,h,w] dtype     upstream gradient of u
 *   x, M, score_m                  as in the forward (score_m carries the gumbel noise implicitly)
 *   ds_rl    [N,stride] fp32 or NULL; g_loss: device float* (upstream grad of readloss) or NULL;
 *   rl_out   the `out` array of pm_readloss_fwd (its [1] is the scale) or NULL
 *   dx       [B,C,h,w] dtype out
 *   ds       [N,stride] fp32 out or NULL: total gradient w.r.t. the similarities (input of pm_read_bwd_dM).
 *            Pass a buffer: the pipelined two-kernel path (score gradients, then dx) needs it as scratch;
 *            with NULL the slower single-kernel generic path runs.
 */
int pm_read_bwd(const void* du, const void* x, const float* M, const float* score_m, const float* ds_rl,
                const float* g_loss, const float* rl_out, void* dx, float* ds, int B, int C, int h, int w,
                int K, int dtype, void* stream);

/*
 * "Score-plane" variants of the read for the case where u feeds a bias-free 1x1 convolution, i.e. the
 * reference's self.output[0] (memory.py:103-104, 330-334). There conv(W, [q ; p.M]) = W1.q + (W2.M^T).p with
 * W = [W1 | W2], so instead of materialising c = p.M (C channels) the read hands the convolution
 *   u' [B, C + PM_PLANES, h, w] = [ q ; score_memory as PM_PLANES channel planes (planes >= K are zero) ]
 * and the caller convolves with W' = [W1 | W2.M^T | 0]: a (C+32)-wide GEMM instead of a 2C-wide one, 85 MB of u
 * instead of 151 MB at cfg 2, and the convolution's input gradient du' = [dq0 ; dp planes] already contains
 * dp = M.dc, so the backward skips that contraction. Same arguments as pm_read_fwd / pm_read_bwd otherwise.
 * Only on the pipelined path: returns PM_ERR_ALIGN unless h*w is a multiple of 4 (fp32) / 8 (bf16) and the
 * feature pointers are 16-byte aligned (callers fall back to pm_read_fwd then). ds must not be NULL.
 */
#define PM_PLANES 32
int pm_read_planes(void); /* = PM_PLANES */
int pm_read_fwd_planes(const void* x, const float* M, const float* gumbel_m, const float* gumbel_q, void* u,
                       float* s, float* score_m, float* col_partials, int B, int C, int h, int w, int K, int dtype,
                       void* stream);
int pm_read_bwd_planes(const void* du, const void* x, const float* M, const float* score_m, const float* ds_rl,
                       const float* g_loss, const float* rl_out, void* dx, const void* dx_add, float* ds, int B, int C,
                       int h, int w, int K, int dtype, void* stream);
/*   dx_add   NULL, or [B,C,h,w] dtype: a second gradient of x (the write branch's, when query feeds both the read and
 *            the writing net) that the kernel sums into dx -- the accumulation autograd would otherwise do with an
 *            element-wise add of three feature-sized tensors. */

/*
 * The folded weight of the score-plane read and its gradient w.r.t. W (both fp32, row-major):
 *   Wp [Co, C + PM_PLANES] = [ W[:, :C] | W[:, C:] . M^T | 0 ]        W [Co, 2C], M [K, C]
 *   dW [Co, 2C]            = [ dWp[:, :C] | dWp[:, C:C+K] . M ]
 * (the gradient w.r.t. M, needed only when m_items carries graph, is one small matmul left to the caller).
 */
int pm_fold_weight_fwd(const float* W, const float* M, float* Wp, int Co, int C, int K, void* stream);
int pm_fold_weight_bwd(const float* dWp, const float* M, float* dW, int Co, int C, int K, void* stream);

/*
 * Gradient w.r.t. the memory when m_items carries graph (meta-test read, train.py:558,570):
 * dM = sum_n score_m[n]^T dc[n] + ds[n]^T q[n].  dM [K,C] fp32 must be ZEROED by the caller.
 * du NULL: only the second term (score-plane mode, where the first term reaches M through W2.M^T in autograd).
 */
int pm_read_bwd_dM(const void* du, const void* x, const float* score_m, const float* ds, float* dM, int B,
                   int C, int h, int w, int K, int dtype, void* stream);

/*
 * get_score on an already normalised NHWC query (external call at train.py:894): s = q.M^T.
 *   q [N,C] fp32 (channels contiguous), M [K,C] fp32, s [N,stride] fp32 out.
 */
int pm_score_nhwc(const float* q, const float* M, float* s, int N, int C, int K, void* stream);

/*
 * score_memory for that external get_score path: dense [N,K] row softmax of s (+ gumbel_m), memory.py:184/187.
 */
int pm_rowsoftmax(const float* s, const float* gumbel_m, float* score_m, int N, int K, void* stream);

/*
 * Memory write, class sums. Replaces memory.py:215 (normalise), :220-223 (255->K, one_hot(K+1),
 * float, bilinear down-sample to [h,w], align_corners=True), :226-231 (per-class sums and counts).
 *   f   [B,C,h,w] dtype (output of the writing net)      labels [B,Hm,Wm] int64
 *   SD  [K+1, C+4] fp32, ZEROED by the caller; rows = classes (row K = ignore), columns 0..C-1 =
 *       sum_n omega[n,k] f[n]/|f[n]|, column C = soft count sum_n omega[n,k], columns C+1..C+3 unused.
 *   This [K+1,C+4] buffer is what a sharded run all-reduces (SURVEY.md 8e).
 */
int pm_write_reduce_fwd(const void* f, const int64_t* labels, float* SD, int B, int C, int h, int w, int Hm,
                        int Wm, int K, int dtype, void* stream);

/*
 * Momentum update + re-normalisation + both write losses. Replaces memory.py:233-239 (branch-free:
 * no host sync per slot), :264-272 (diversityloss), :259-262 (classification_loss).
 *   SD [K+1,C+4], M_old [K,C], W_cls [K,C], b_cls [K] fp32
 *   M_new [K,C] out (unit rows), losses float[2] out = {div, cls},
 *   saved float[2K] out = {|M'_k| (pre-normalisation norms), D_k} for the backward,
 *   aux: pm_update_aux_floats(K) floats of scratch, ZEROED by the caller (one CTA per row; rows meet there).
 */
int pm_update_aux_floats(int K);
int pm_update_fwd(const float* SD, const float* M_old, float momentum, const float* W_cls, const float* b_cls,
                  float* M_new, float* losses, float* saved, float* aux, int C, int K, void* stream);

/*
 * Backward of pm_update_fwd.
 *   dM_new [K,C] or NULL (gradient arriving at the new memory), g_losses: device float[2] = upstream
 *   grads of {div, cls} (either pointer may be NULL = 0), M_new, saved, W_cls, b_cls as in the forward.
 *   dS [K,C] out (gradient w.r.t. the class sums; zero rows for absent classes; this is what a sharded
 *   run all-reduces in the backward), dW_cls [K,C] out, db_cls [K] out.
 */
int pm_update_bwd(const float* dM_new, const float* g_div, const float* g_cls, const float* M_new,
                  const float* saved, const float* W_cls, const float* b_cls, float momentum, float* dS,
                  float* dW_cls, float* db_cls, float* aux /* zeroed, pm_update_aux_floats(K) */, int C, int K,
                  void* stream);

/*
 * Memory write, backward to the write feature: dv[n] = sum_k omega[n,k] dS[k];
 * df = (dv - v (v.dv)) / |f|.   dS [K,C] fp32, f and labels as in the forward, df [B,C,h,w] dtype out.
 */
int pm_write_bwd(const float* dS, const void* f, const int64_t* labels, void* df, int B, int C, int h, int w,
                 int Hm, int Wm, int K, int dtype, void* stream);

/*
 * BatchNorm2d (+ residual, + ReLU) of the module's two 1x1-conv blocks, NCHW (x, y, residual, dy, dx, dres are
 * [B,C,hw] in `dtype`; statistics and affine parameters fp32 [C]). Replaces, for `self.output`
 * (memory.py:103-107) and `Writingnet` (memory.py:74-87), the BatchNorm2d / add / ReLU modules that follow
 * the 1x1 convolution (the convolution itself stays a library GEMM).
 *   pm_bn_stats       batch mean and 1/sqrt(biased var + eps) per channel; if running_mean/var are given they
 *                     are updated in place with `momentum` (unbiased variance), like nn.BatchNorm2d in training
 *   pm_bn_apply       y = [relu]((x - mean) * invstd * gamma + beta [+ residual]); optionally also a packed ReLU
 *                     mask (1 bit per element, pm_bn_mask_words(B,C,hw) uint32 words; needs hw % 4 == 0) that the
 *                     backward passes read instead of y
 *   pm_bn_bwd_reduce  g = dy * (y > 0 if relu) (from relu_mask if given, else from y);  dbeta = sum g,  dgamma = sum g * xhat
 *   pm_bn_bwd_apply   dx = gamma * invstd * (g - [training](dbeta + xhat * dgamma) / (B*hw));  dres = g (or NULL)
 */
int pm_bn_stats(const void* x, int B, int C, int hw, int dtype, float eps, float* mean, float* invstd,
                float* running_mean, float* running_var, float momentum, void* stream);
int pm_bn_mask_words(int B, int C, int hw);
int pm_bn_apply(const void* x, const float* mean, const float* invstd, const float* gamma, const float* beta,
                const void* residual, void* y, uint32_t* relu_mask, int relu, int B, int C, int hw, int dtype,
                void* stream);
/* The same with the statistics finalised in the kernel: `stats` = the fp64 [sum | sum of squares] per channel that
 * pm_conv1x1_fwd's epilogue produced, `count` = B*h*w. Every CTA derives mean / invstd of its channel itself; mean_out /
 * invstd_out [C] (for the backward) and the running statistics (momentum update, unbiased variance; may be NULL) are
 * written once per channel. Replaces pm_bn_finalize + pm_bn_apply (one launch less between the GEMM and its consumer). */
int pm_bn_apply_stats(const void* x, const double* stats, double count, float eps, const float* gamma, const float* beta,
                      const void* residual, void* y, uint32_t* relu_mask, int relu, float* mean_out, float* invstd_out,
                      float* running_mean, float* running_var, float momentum, const double* count_dev,
                      long long* num_batches_tracked, int B, int C, int hw, int dtype, void* stream);
/*   num_batches_tracked  NULL, or nn.BatchNorm2d's int64 counter: incremented by one by this launch (the module's own side
 *              effect, torch/nn/modules/batchnorm.py) instead of by an element-wise kernel of its own.
 *   count_dev  NULL, or the element count in device memory, used instead of `count`: SyncBatchNorm (the reference under
 *              --syncbn, train.py:95) all-reduces [stats | count] over the ranks and normalises with the global statistics
 *              without a device->host read. */
int pm_bn_bwd_reduce(const void* dy, const void* y, const uint32_t* relu_mask, const void* x, const float* mean,
                     const float* invstd, int relu, float* dgamma, float* dbeta, int B, int C, int hw, int dtype,
                     void* stream);
/* pm_bn_bwd_reduce with every channel split over 4 CTAs (256 channels alone are 1.7 waves of long serial loops on 148
 * SMs); scratch: pm_bn_bwd_scratch_bytes(C) bytes, ZEROED by the caller; partials are added in split order (deterministic). */
int pm_bn_bwd_scratch_bytes(int C);
int pm_bn_bwd_reduce_split(const void* dy, const void* y, const uint32_t* relu_mask, const void* x, const float* mean,
                           const float* invstd, int relu, float* dgamma, float* dbeta, int B, int C, int hw, int dtype,
                           void* scratch, void* stream);
/* pm_bn_bwd_reduce with one CTA per (image, channel) row -- bn_bwd_apply's access pattern, ~1.6x the bandwidth of one CTA
 * per channel. scratch: pm_bn_bwd_rows_scratch_bytes(B, C) bytes, 8-byte aligned, zeroed ONCE when allocated (the kernel
 * leaves its arrival counters at zero); the B row partials of a channel are added in image order (deterministic). Use one
 * scratch per stream that may run this entry concurrently. */
int pm_bn_bwd_rows_scratch_bytes(int B, int C);
int pm_bn_bwd_reduce_rows(const void* dy, const void* y, const uint32_t* relu_mask, const void* x, const float* mean,
                          const float* invstd, int relu, float* dgamma, float* dbeta, int B, int C, int hw, int dtype,
                          void* scratch, void* stream);
int pm_bn_bwd_apply(const void* dy, const void* y, const uint32_t* relu_mask, const void* x, const float* mean,
                    const float* invstd, const float* gamma, const float* dgamma, const float* dbeta, int relu,
                    int training, void* dx, void* dres, int B, int C, int hw, int dtype, void* stream);

/*
 * The two 1x1 convolutions themselves (memory.py:74-75 `Writingnet.writefeat[0]`, memory.py:103-104 `self.output[0]`,
 * both bias-free, applied at memory.py:84/214 and :334) and their autograd, as tcgen05 GEMMs on NCHW activations
 * (csrc/pm_gemm.cu). Per image b:   Y[b] (M x hw) = A (M x K) . X[b] (K x hw).
 *   dtype PM_F32 computes in 3xTF32 (error-compensated, ~fp32 accuracy), PM_BF16 in bf16 with fp32 accumulation.
 *
 *   pm_conv1x1_prep   A = W (transpose = 0, W is [M,K] fp32) or W^T (transpose = 1, W is [K,M] fp32), padded with
 *                     zero rows to Mpad = ceil(M/128)*128. PM_F32: A_hi, A_lo are fp32 [Mpad,K] (the TF32 split);
 *                     PM_BF16: A_hi is bf16 [Mpad,K], A_lo unused. transpose = 0 prepares the forward convolution,
 *                     transpose = 1 its input gradient (dX[b] = W^T . dY[b]).
 *   pm_conv1x1_fwd    X [B,K,hw], Y [B,M,hw] in `dtype`; A_hi/A_lo from pm_conv1x1_prep. accumulate != 0 adds into Y
 *                     (TMA reduce-add; gradient accumulation). stats: NULL, or double[2*M] ZEROED by the caller that
 *                     receives per-row sum and sum of squares of Y over (b, pixel) -- the batch statistics of the
 *                     BatchNorm2d that follows (memory.py:76,105), see pm_bn_finalize.
 *                     K % 8 == 0 (PM_F32) / 16 (PM_BF16), M % 32 == 0, M <= 512, hw * sizeof(dtype) % 16 == 0.
 *   pm_conv1x1_wgrad  dW [M,N] fp32 (+)= sum_b dY[b] (M x hw) . X[b]^T (hw x N); dY [B,M,hw], X [B,N,hw] in `dtype`;
 *                     workspace: pm_conv1x1_wgrad_workspace_floats(B,M,N,hw,dtype) floats of scratch (split-K partials).
 *                     M % 32 == 0, N % 32 == 0.
 *   pm_bn_finalize    mean/invstd (fp32 [C]) and the running-stat update from the fp64 sums pm_conv1x1_fwd produced;
 *                     count = B*hw. Same arithmetic as pm_bn_stats.
 */
int pm_conv1x1_prep(const float* W, int M, int K, int transpose, int dtype, void* A_hi, void* A_lo, void* stream);
/* pm_conv1x1_prep for BOTH operand layouts of one weight W [R,S] in one launch: (A_hi, A_lo) = W (M = R, K = S), the forward
 * operand, and (At_hi, At_lo) = W^T (M = S, K = R), the operand of the input-gradient GEMM. zero / zero_n: optional
 * double buffer cleared by the same launch (the statistics buffer pm_conv1x1_fwd's epilogue adds into). */
int pm_conv1x1_prep_both(const float* W, int R, int S, int dtype, void* A_hi, void* A_lo, void* At_hi, void* At_lo, double* zero,
                         int zero_n, void* stream);
int pm_conv1x1_fwd(const void* X, const void* A_hi, const void* A_lo, void* Y, double* stats, int B, int K, int M,
                   int hw, int accumulate, int dtype, void* stream);
/* Y[b] = [relu](scale[m] * (A . X[b]) + shift[m]): the convolution with the eval-mode BatchNorm2d (+ ReLU) that follows it
 * (memory.py:103-107 with running statistics: scale = gamma / sqrt(var + eps), shift = beta - mean * scale) folded into
 * the GEMM epilogue -- the inference read (BASELINE config 5) then has no separate normalise pass. scale, shift fp32 [M]. */
int pm_bn_eval_affine(const float* gamma, const float* beta, const float* running_mean, const float* running_var, float eps,
                      int C, float* scale, float* shift, void* stream);
/*
 * Input gradient of conv1x1 -> BatchNorm (-> ReLU) with the BatchNorm backward in the GEMM's operand path (fp32, blocks
 * WITHOUT a residual: self.output, memory.py:103-107): dX[b] = W^T . dz[b], dz = gamma*invstd*(g - dbeta/n - xhat*dgamma/n),
 * g = dY*(y > 0). Replaces pm_bn_bwd_apply + pm_conv1x1_fwd on the transposed weight: the producer loads the dY tile and the
 * tile of the saved convolution output Z, the operand-split warps form dz in place (the ReLU gate is recomputed from Z with
 * the forward's expression) and the dz tiles are stored to dZ [B,K,hw] for the weight-gradient GEMM.
 *   dY, Z, dZ [B,K,hw] fp32 (K = the convolution's OUTPUT channels)      A_hi/A_lo = pm_conv1x1_prep(W, transpose = 1)
 *   dX [B,M,hw] fp32 (M = the convolution's INPUT channels)              mean/invstd/gamma/beta [K], dgamma/dbeta [K] =
 *   the sums pm_bn_bwd_reduce produced; training = 0: eval-mode BatchNorm (dz = gamma*invstd*g); n = B*hw.
 */
int pm_conv1x1_dgrad_bnbwd(const void* dY, const void* Z, const void* A_hi, const void* A_lo, void* dX, void* dZ,
                           const float* mean, const float* invstd, const float* gamma, const float* beta, const float* dgamma,
                           const float* dbeta, int relu, int training, int B, int K, int M, int hw, int dtype, void* stream);
int pm_conv1x1_fwd_affine(const void* X, const void* A_hi, const void* A_lo, void* Y, const float* scale, const float* shift,
                          int relu, int B, int K, int M, int hw, int dtype, void* stream);
int pm_conv1x1_wgrad_workspace_floats(int B, int M, int N, int hw, int dtype);
int pm_conv1x1_wgrad(const void* dY, const void* X, float* workspace, float* dW, int B, int M, int N, int hw,
                     int accumulate, int dtype, void* stream);
int pm_bn_finalize(const double* stats, int C, double count, float eps, float* mean, float* invstd,
                   float* running_mean, float* running_var, float momentum, void* stream);

/*
 * The two write losses on an ARBITRARY memory, for the reference's public methods `diversityloss(mem)`
 * (memory.py:264-272) and `classification_loss(mem)` (memory.py:259-262); inside write() they are fused into
 * pm_update_fwd / pm_update_bwd. mem [K,C] fp32 (rows need not be unit length), W_cls [K,C] / b_cls [K] or both NULL
 * (divergence loss only).
 *   fwd: out float[2] = {div, cls}; gram [K*K] and prob [K*K] (softmax rows of the classifier) are kept for the backward
 *        (either may be NULL when no backward follows).
 *   bwd: g_div / g_cls device scalars (NULL = 0); dmem [K,C] out; dW_cls [K,C], db_cls [K] out or NULL.
 */
int pm_memory_losses_fwd(const float* mem, const float* W_cls, const float* b_cls, int K, int C, float* out, float* gram,
                         float* prob, void* stream);
int pm_memory_losses_bwd(const float* mem, const float* W_cls, const float* gram, const float* prob, const float* g_div,
                         const float* g_cls, int K, int C, float* dmem, float* dW_cls, float* db_cls, void* stream);

/*
 * One pass over the labels for the whole step (csrc/pm_labels.cu). Replaces memory.py:220 (`tempmask[tempmask == 255]
 * = memory_size`) and the label side of CrossEntropyLoss(ignore_index=255) (memory.py:117,176).
 *   labels   [n] int64 (labels_are_u8 = 0) or uint8 (labels_are_u8 = 1): class ids 0..K-1, 255 = ignore
 *   lab8     [n] uint8 out: class id, K for ignore. Values outside [0,K) u {255} -- torch's one_hot / CE would raise a
 *            device assert on them -- also map to K and are COUNTED in ws[PM_WS_BAD].
 *   ws       the PM_WS_WORDS 64-bit words of the read-loss workspace, ZEROED by the caller: receives the bit-exact
 *            label histogram (ws[PM_WS_HIST + k], bin K = ignore) and the bad-label count.
 * pm_readloss_fwd8 is pm_readloss_fwd on that packed map (K <= 19): pass the SAME ws after pm_labels_pack (it reads the
 * histogram for the number of valid pixels and adds the loss sum and its CTA counter).
 */
int pm_labels_pack(const void* labels, int labels_are_u8, long long n, int K, uint8_t* lab8, void* ws, void* stream);
int pm_readloss_fwd8(const float* s, const uint8_t* lab8, float temperature, int B, int h, int w, int Hm, int Wm, int K,
                     float* ds_rl, void* ws, float* out, void* stream);
/* pm_write_reduce_fwd / pm_write_bwd on the packed map (1 byte per label pixel instead of 8). */
int pm_write_reduce_fwd8(const void* f, const uint8_t* lab8, float* SD, int B, int C, int h, int w, int Hm, int Wm, int K,
                         int dtype, void* stream);
int pm_write_bwd8(const float* dS, const void* f, const uint8_t* lab8, void* df, int B, int C, int h, int w, int Hm, int Wm,
                  int K, int dtype, void* stream);

/*
 * The sharded update with its exchange FUSED into the update kernels over NVLink peer memory (SURVEY.md 8e: the one
 * collective of the path is the all-reduce of the [K+1,C+4] class sums|counts before the update, and -- its autograd
 * mirror -- of the [K,C] gradient w.r.t. the sums). Instead of an NCCL launch before pm_update_fwd and another after
 * pm_update_bwd, every rank keeps a "symmetric" buffer of PM_PEER_BYTES (host side: torch.distributed._symmetric_memory;
 * `peer_bufs` is the DEVICE array of all ranks' buffer addresses as peer-mapped pointers):
 *   bytes [0, PM_PEER_DS_OFF)     this rank's sums|counts  -- pm_write_reduce_fwd[8] accumulates straight into it
 *                                 (zero it first)
 *   bytes [PM_PEER_DS_OFF, ...)   this rank's dS share     -- written by pm_update_bwd_peer itself
 *   bytes [PM_PEER_FLAG_OFF, ...) arrival flags, zeroed once at allocation
 * CTA i raises a flag in every peer's buffer, waits for all ranks' flags, reads row i (forward: all rows) out of the
 * peers' buffers and sums in rank order -- identical on every rank, so the new memory is bit-identical across ranks.
 * `epoch`: one device uint32 per kernel kind (two in total), zeroed at allocation, owned by the kernels.
 * SD_sum [K+1,C+4] (may be NULL) receives the all-reduced sums|counts; dS [K,C] the all-reduced gradient.
 * Every rank of the group must launch the same sequence of these two kernels (they spin on each other, bounded: a peer
 * that never arrives traps instead of hanging).
 */
#define PM_PEER_DS_OFF 36864
#define PM_PEER_FLAG_OFF 73728
#define PM_PEER_BYTES 131072
int pm_peer_buffer_bytes(void);
int pm_update_fwd_peer(const void* peer_bufs, int rank, int world, unsigned* epoch, float* SD_sum, const float* M_old,
                       float momentum, const float* W_cls, const float* b_cls, float* M_new, float* losses, float* saved,
                       float* aux, int C, int K, void* stream);
int pm_update_bwd_peer(const void* peer_bufs, int rank, int world, unsigned* epoch, const float* dM_new, const float* g_div,
                       const float* g_cls, const float* M_new, const float* saved, const float* W_cls, const float* b_cls,
                       float momentum, float* dS, float* dW_cls, float* db_cls, float* aux, int C, int K, void* stream);

/* 64-bit words of the segmentation-metrics workspace (`ws`, zero it before every pm_seg_eval call). */
enum pm_seg_eval_ws_layout {
    PM_SEG_WS_LOSS_SUM = 0, /* double: sum over valid label pixels of (LSE - logit[y])                   */
    PM_SEG_WS_VALID = 1,    /* uint64: V, label pixels with a class id in [0,K)                           */
    PM_SEG_WS_BAD = 2,      /* uint64: label values outside [0,K) u {255} (excluded like 255, and counted) */
    PM_SEG_WS_COUNTER = 3,  /* uint64: CTA arrival ticket                                                 */
    PM_SEG_WS_WORDS = 4
};

/*
 * Segmentation validation metrics (csrc/pm_segeval.cu). Replaces, per validation batch, the up-sampling of the head's
 * output to label size (network/deepv3plus.py:575-578, mynn.py:57-62), the criterion on it, `argmax` and the host-side
 * `fast_hist` (utils/misc.py:65-73) of the validation loop (train.py:847-939) and the whole-image eval
 * (eval.py:277-286,304-337) -- the [B,K,Hm,Wm] logits are never written and nothing is copied to the host.
 *   logits     [B,K,h,w] NCHW in `dtype`; bilinearly up-sampled (align_corners=True) to [Hm,Wm] with ATen's arithmetic,
 *              used as they are when h == Hm and w == Wm. Hm >= h, Wm >= w, K in 1..31.
 *   labels     [B,Hm,Wm] int64 (labels_are_u8 = 0) or uint8 (1); 255 = ignore. Values outside [0,K) are excluded from
 *              the confusion matrix and the loss (fast_hist's mask); those other than 255 are counted in ws[PM_SEG_WS_BAD].
 *   confusion  [K,K] int64, ACCUMULATED: confusion[label][pred] += 1 per label pixel with a valid label.
 *   pred       [B,Hm,Wm] uint8 out (argmax, first maximal class; written for every pixel, ignored ones included) or NULL.
 *   ws         PM_SEG_WS_WORDS 64-bit words, ZEROED by the caller (layout above).
 *   out        float[1] out: mean cross-entropy over the valid label pixels (NaN when there is none, like torch).
 */
int pm_seg_eval(const void* logits, int dtype, int B, int K, int h, int w, const void* labels, int labels_are_u8, int Hm,
                int Wm, int64_t* confusion, uint8_t* pred, void* ws, float* out, void* stream);

/*
 * Decoder up-sample + concat (csrc/pm_upcat.cu). Replaces the DeepLabV3+ decoder step after the memory module
 * (network/deepv3plus.py:569-572): `Upsample(dec0_up, low_level.size()[2:])` (mynn.py:57-62, bilinear,
 * align_corners=True) and `torch.cat([dec0_fine, dec0_up], 1)` -- the up-sampled map is written straight into its
 * channels of the concatenated output and never exists on its own.
 *   fine    [B,Cf,H,W] NCHW in `dtype` (may be NULL when Cf == 0; Cf = 0 is a plain up-sample)
 *   coarse  [B,Cc,h,w] NCHW in `dtype`; H >= h, W >= w (up-sampling only)
 *   out     [B,Cf+Cc,H,W] out: planes [0,Cf) = fine, planes [Cf,Cf+Cc) = coarse up-sampled with ATen's arithmetic
 *           (upsample_bilinear2d_out_frame bit for bit; equal sizes copy).
 * B <= 65535 and Cf + Cc <= 65535 (grid limits), H * W < 2^31.
 */
int pm_upcat_fwd(const void* fine, const void* coarse, void* out, int dtype, int B, int Cf, int Cc, int h, int w, int H, int W,
                 void* stream);
/*
 * Backward of pm_upcat_fwd with respect to `coarse`. Replaces upsample_bilinear2d_backward (atomics, registered as
 * non-deterministic) after the copy of the gradient's coarse-channel slice made by cat's backward.
 *   g         [B,Cf+Cc,H,W] NCHW in `dtype`: the gradient of `out`; only its planes [Cf,Cf+Cc) are read, in place.
 *   d_coarse  [B,Cc,h,w] out: the exact transpose of the forward's interpolation (the same taps and fp32 weights),
 *             accumulated in fp32 in a fixed order and stored once per element: bitwise reproducible.
 * The gradient of `fine` is g's planes [0,Cf) as they are (what cat's backward returns); no kernel touches it.
 */
int pm_upcat_bwd(const void* g, void* d_coarse, int dtype, int B, int Cf, int Cc, int h, int w, int H, int W, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PINMEM_B200_H */
