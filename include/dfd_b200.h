/* dfd_b200.h — C ABI of libdfd_b200.so: the sm_100a device kernels behind the data-parallel train / validate
 * step of TARTRL/Deepfake_Detection (dfd/runners/train.py:610-649, :713-746).
 *
 * The reference has NO native/FFI layer (SURVEY.md section 2.1): every entry point below replaces a stock
 * PyTorch op (ATen / cuDNN / cuBLAS dispatch) that the reference's nn.Module tree issues on the hot path; the
 * citation on each function is the reference call site it stands in for.  INTEGRATION.md shows the binding a
 * maintainer adds on the reference side (ctypes, because the reference is pure Python).
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer owned by the caller (no ownership transfer);
 *   - activations are NHWC, 16-bit: dt = DFD_DT_BF16 (0) or DFD_DT_FP16 (1); parameters, gradients, BN
 *     statistics, SE vectors, logits and the loss are fp32; channel counts are multiples of 8;
 *   - `stream` is a cudaStream_t; kernels are enqueued on it and nothing synchronises the host;
 *   - return value: 0 on success, negative DFD_ERR_* otherwise (dfd_last_error() gives the message); the
 *     Python host raises RuntimeError, the reference's only error convention;
 *   - per-channel statistics buffers hold DFD_STAT_SLOTS (= dfd_stat_slots() = 8) interleaved fp64 copies,
 *     i.e. [8][C] doubles, accumulated with atomics and zeroed by the caller once per step.
 */
#ifndef DFD_B200_H
#define DFD_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define DFD_OK 0
#define DFD_ERR_ARG (-1)
#define DFD_ERR_CUDA (-2)
#define DFD_ERR_UNSUPPORTED (-3)

#define DFD_DT_BF16 0
#define DFD_DT_FP16 1

#define DFD_ACT_NONE 0
#define DFD_ACT_SWISH 1
#define DFD_ACT_RELU 2

/* ---- runtime ---------------------------------------------------------------------------------------- */
const char* dfd_last_error(void);
int dfd_abi_version(void);
int dfd_stat_slots(void);
/* optimizer.zero_grad() (train.py:631) and per-step scratch clearing */
int dfd_memset_async(void* p, int value, long long bytes, void* stream);

/* ---- pointwise (1x1) convolution: nn.Conv2d via create_conv2d, efficientnet_blocks.py:165,277,299,
 *      efficientnet.py:292, resnet.py:192,199 -------------------------------------------------------- */
/* C[M,N] = A[M,K] * B[N,K]^T on tcgen05 (TMA in/out, TMEM accumulators). Forward: A = input [N*H*W, Cin],
 * B = weight [Cout, Cin]. Input gradient: A = dY [N*H*W, Cout], B = weight^T [Cin, Cout].
 * dsum/dsq (optional): per-column sum / sum of squares of the stored C for the following BatchNorm. */
int dfd_gemm_tn(const void* A, const void* B, void* C, long long M, int N, int K, int dt, double* dsum, double* dsq,
                const void* fin, void* stream);
/* `fin` (optional; here and on dfd_gemm_tn_rowpack / dfd_dwconv_fwd): device pointer to a BnFinDesc (csrc/bn_finalize.cuh) -
 * the LAST CTA of the launch then finalises the BatchNorm behind the convolution (what dfd_bn_finalize does in its own
 * one-block launch): scale / shift / mean / rstd and the running statistics. The backward producers (dfd_act_bwd,
 * dfd_bn_bwd_reduce, dfd_dwconv_bwd) take a BnBwdFinDesc the same way (what dfd_bn_bwd_finalize does). NULL: no finalisation. */
/* Small-K variant (Cin = 16 / 24 / 32 pointwise convs and their input gradients): `pack` consecutive rows of A are read
 * as one row of pack*K values against the block-diagonal weight Bd[pack*N, pack*K] built by dfd_blockdiag_weights; the
 * result is byte-identical row-major C[M,N], statistics are folded back onto the N channels. Requires M % pack == 0. */
int dfd_gemm_tn_rowpack(const void* A, const void* Bd, void* C, long long M, int N, int K, int pack, int dt,
                        double* dsum, double* dsq, const void* fin, void* stream);
/* table: device array of { const void* src; void* dst; int N; int K; int pack; int _pad; } */
int dfd_blockdiag_weights(const void* table, int count, int dt, void* stream);
/* same contract on the warp-level mma.sync path (+ optional residual `add` [M,N]); cross-check / fallback */
int dfd_gemm_tn_mma(const void* A, const void* B, void* C, const void* add, long long M, int N, int K, int dt,
                    double* dsum, double* dsq, void* stream);
/* weight gradient dW[Nw,Kw] (fp32, accumulated) += G[M,Nw]^T * X[M,Kw]  (autograd of the conv, train.py:634) */
int dfd_gemm_wgrad_mma(const void* G, const void* X, float* dW, long long M, int Nw, int Kw, int dt, void* stream);
/* the same contract on tcgen05: both operands MN-major straight from NHWC memory (TMA 128-byte swizzle boxes), fp32
 * accumulator in TMEM over a contiguous range of rows per CTA, one red.global.add flush */
int dfd_gemm_wgrad(const void* G, const void* X, float* dW, long long M, int Nw, int Kw, int dt, void* ws, long long ws_bytes,
                   void* stream);
/* ws (optional): ORDER-DETERMINISTIC mode - split z stores its fp32 partial matrix at ws[z][Nw][Kw] with plain stores, dW is
 * not touched, and dfd_ordered_reduce adds the dfd_gemm_wgrad_splits(M, Nw, Kw) partials into dW in split order afterwards
 * (ws_bytes >= splits * Nw * Kw * 4). NULL: red.global.add from every split straight into dW, in arrival order. */
int dfd_gemm_wgrad_splits(long long M, int Nw, int Kw);
/* dst[i] += sum_{p < parts} src[p * stride + i], i < n, partials added in index order. table: device array of
 * { const float* src; float* dst; long long n; long long stride; int parts; int _pad; } (n % 4 == 0, 16-byte aligned);
 * blocks_x = CTAs per entry (a CTA covers 256 float4 per trip of an entry with <= 64 parts, 8 float4 per trip otherwise);
 * first_dst (the lowest gradient address written) is informational for host-side planners. */
int dfd_ordered_reduce(const void* table, int count, const float* first_dst, int blocks_x, void* stream);

/* ---- depthwise k x k convolution: nn.Conv2d(groups=C), efficientnet_blocks.py:152-153,283-285 -------- */
int dfd_dwconv_fwd(const void* x, const float* scale, const float* shift, const float* w, void* out, int N, int H,
                   int W, int C, int k, int stride, int act_in, int dt, double* dsum, double* dsq, const void* fin,
                   void* stream);
int dfd_dwconv_dgrad(const void* gy, const void* yout, const float* cA, const float* cB, const float* cC,
                     const float* w, const void* xin, const float* scale, const float* shift, const float* mean,
                     const float* rstd, const void* add, void* gx, int N, int H, int W, int C, int k, int stride,
                     int mode, int dt, double* s1, double* s2, void* stream);
int dfd_dwconv_wgrad(const void* x, const float* scale, const float* shift, const void* gy, const void* yout,
                     const float* cA, const float* cB, const float* cC, float* dW, int N, int H, int W, int C, int k,
                     int stride, int dt, void* stream);
/* dfd_dwconv_dgrad + dfd_dwconv_wgrad of one depthwise stage in a single pass over dy: the autograd backward of conv_dw
 * (+ bn1/act1 behind it when scale != NULL, efficientnet_blocks.py:283-285, 277-281; scale == NULL: DS block,
 * efficientnet_blocks.py:152-153, gx = dgrad (+ add)), dW accumulated into `dW` */
int dfd_dwconv_bwd(const void* gy, const void* yout, const float* cA, const float* cB, const float* cC,
                   const float* w, const void* xin, const float* scale, const float* shift, const float* mean,
                   const float* rstd, const void* add, void* gx, float* dW, int N, int H, int W, int C, int k,
                   int stride, int dt, double* s1, double* s2, void* ws, long long ws_bytes, const void* fin, void* stream);
/* ws (optional): ORDER-DETERMINISTIC dW - CTA (tile x, channel block y, image group z) stores its partial at
 * ws[y][x * groups + z][B * k*k] laid out like dW[By .. By+B)[k*k], B = dfd_dwconv_block_channels(C), and
 * dfd_ordered_reduce adds the dfd_dwconv_bwd_parts(...) = tiles * groups partials of every channel block into dW in slot order
 * afterwards (ws_bytes >= ceil(C/B) * parts * B*k*k * 4). NULL: fp32 atomics into dW. */
int dfd_dwconv_bwd_parts(int N, int H, int W, int C, int k, int stride);
/* channels per CTA of the depthwise kernels for a layer of C channels (64, or 32 / 16 where 64-channel blocks would leave a
 * fifth or more of the lanes idle): the slot width and the channel-block size of the ws layout above */
int dfd_dwconv_block_channels(int C);

/* ---- stem convolution: conv_stem 3x3 s2 (efficientnet.py:275,321) / conv1 7x7 s2 (resnet.py:379,451) ---- */
int dfd_stem_fwd(const void* x_nchw, const float* w, void* out_nhwc, int N, int Cin, int H, int W, int Cout, int k,
                 int stride, int pad, int dt, double* dsum, double* dsq, void* stream);
int dfd_stem_wgrad(const void* x_nchw, const void* g, const void* y, const float* cA, const float* cB,
                   const float* cC, float* dW, int N, int Cin, int H, int W, int Cout, int k, int stride, int pad,
                   int dt, void* stream);

/* stem as a GEMM (round-1 perf path): im2col of the NCHW image, column order (ci,kh,kw) == OIHW flattening, K padded to
 * Kp % 8 == 0; weights padded to [Cout, Kp]; fp32 gradient un-padded (accumulating) into the OIHW arena */
int dfd_stem_im2col(const void* x_nchw, void* cols, int N, int Cin, int H, int W, int k, int stride, int pad, int Kp, int dt,
                    void* stream);
int dfd_pad_weight(const void* src16, void* dst16, int O, int taps, int Kp, int dt, void* stream);
int dfd_unpad_grad(const float* g_padded, float* g_accum, int O, int taps, int Kp, void* stream);

/* ---- dense k x k convolution, max-pool, ReLU tail (ResNet: resnet.py:129-136,150-175,195-260,379-382,450-468).
 *      Product path: the IMPLICIT GEMMs further down (dfd_conv_tc, dfd_conv_wgrad_tc, dfd_conv_dgrad_s2_tc,
 *      dfd_conv1x1_dgrad_add) for every 3x3 and strided 1x1 convolution; the materialised formulation below (conv = im2col ->
 *      dfd_gemm_tn; dgrad = dfd_gemm_tn -> col2im; wgrad on the im2col matrix) serves the 7x7 stem, channel counts that are
 *      not multiples of 64, and the bit-exact cross-checks in the tests.
 *      Column order of the im2col matrix / packed weights: (kh, kw, ci). ------------------------------------------- */
int dfd_im2col(const void* x, void* cols, int N, int H, int W, int C, int k, int stride, int pad, int dt, void* stream);
int dfd_col2im(const void* dcols, const void* add, void* dx, int N, int H, int W, int C, int k, int stride, int pad, int dt,
               void* stream);
/* table: device array of { const void* src_OIHW16; void* dst_OHWI16; void* dstT_HWI_O16; void* dstD_IH'W'O16 (flipped taps);
 *                          int O; int I; int k; int pad; }  - dstT / dstD may be null */
int dfd_repack_weights(const void* table, int count, int dt, void* stream);
/* Dense k x k convolution, stride 1, padding (k-1)/2, as an IMPLICIT GEMM on tcgen05 (no im2col matrix in memory): the TMA
 * producer loads, per tap and 64-channel block, the NHWC input box shifted by the tap through a 4-D tensor map; out-of-image
 * rows arrive as zeros (= the padding). Replaces nn.Conv2d 3x3 stride 1 of BasicBlock / Bottleneck (resnet.py:129-136,195-197):
 *   forward: x = input [N,H,W,Cin],  wpk = dst_OHWI16,             y [N,H,W,Cout]; dsum/dsq = BatchNorm statistics of y
 *   dgrad  : x = dY    [N,H,W,Cout], wpk = dstD (flipped, [Cin]..), y = dX [N,H,W,Cin]  (call with Cin/Cout exchanged)
 * Cin % 64 == 0, Cout % 64 == 0. H, W = INPUT extents; stride 1 or 2 (2: the TMA box walks the input with element strides
 * {1, 2, 2, 1}; forward / weight gradient only - the strided input gradient stays dfd_gemm_tn + dfd_col2im); k = 1 with
 * stride 2 is the strided 1x1 downsample convolution (resnet.py:249-260) without its gather. */
int dfd_conv_tc(const void* x, const void* wpk, void* y, int N, int H, int W, int Cin, int Cout, int k, int stride, int dt,
                double* dsum, double* dsq, const void* fin, void* stream);
/* Weight gradient of the same convolution, also an implicit GEMM (MN-major tcgen05 operands straight from the NHWC tensors,
 * one pipeline stage = one patch of <= 64 output pixels, its input box shifted by the tap): dW_OHWI fp32 [Cout][kh][kw][Cin]
 * += sum_pixels dY[pixel, co] * x[pixel + tap, ci]. `ws` / `ws_bytes` as for dfd_gemm_wgrad: when given, the split partials
 * (dfd_conv_wgrad_splits x Cout x k*k*Cin floats) are written there for dfd_ordered_reduce and dW is left alone. */
int dfd_conv_wgrad_tc(const void* dy, const void* x, float* dW_ohwi, int N, int H, int W, int Cin, int Cout, int k, int stride,
                      int dt, void* ws, long long ws_bytes, void* stream);
int dfd_conv_wgrad_splits(int N, int H, int W, int Cin, int Cout, int k, int stride);
/* Input gradient of a 3x3, stride-2, padding-1 convolution (the autograd dgrad of resnet.py:195-197 with stride 2) as four
 * implicit GEMMs, one per parity class of the input pixels (1, 2, 2 and 4 taps), each storing through a strided tensor-map
 * view of dx: dx [N,H,W,Cin] is written exactly once, no column matrix, no col2im. dy [N,Ho,Wo,Cout]; wpkD = the tap-flipped
 * [Cin][kh'][kw'][Cout] layout of dfd_repack_weights. Cin % 64 == 0, Cout % 64 == 0. */
int dfd_conv_dgrad_s2_tc(const void* dy, const void* wpkD, void* dx, int N, int H, int W, int Cin, int Cout, int dt, void* stream);
/* Input gradient of a 1x1 convolution with stride 1 or 2 (downsample branch, resnet.py:249-260) ADDED into dx [N,H,W,Cin],
 * which already holds the main-path gradient: dx[n, s*a, s*b, :] += dY[n,a,b,:] * W - an implicit GEMM whose output map is
 * the stride-s pixel view of dx and whose epilogue is a TMA reduction store (16-bit add in L2). wT = transposed [Cin][Cout]
 * weight (dfd_transpose_weights). Replaces dfd_gemm_tn + dfd_col2im / dfd_add_inplace. */
int dfd_conv1x1_dgrad_add(const void* dy, const void* wT, void* dx, int N, int H, int W, int Cin, int Cout, int stride, int dt,
                          void* stream);
int dfd_unpack_grad(const float* g_ohwi, float* g_oihw_accum, int O, int I, int k, void* stream);
int dfd_maxpool_fwd(const void* x, void* out, void* argmax_u8, int N, int H, int W, int C, int dt, void* stream);
int dfd_maxpool_bwd(const void* gy, const void* argmax_u8, void* gx, int N, int H, int W, int C, int dt, void* stream);
int dfd_relu_bwd(const void* g, const void* out, void* gm, long long numel, int dt, void* stream);
int dfd_pool_bwd(const float* dpooled, void* dout, int N, long long hw, int C, int dt, void* stream);

/* ---- BatchNorm2d (train + eval), Swish, SE gating, residual, global pool and their backward:
 *      efficientnet_blocks.py:104-110,154,166,180-194,280-348; layers/activations.py:19-33;
 *      efficientnet.py:323-343; resnet.py:154-173 ---------------------------------------------------- */
int dfd_colstats(const void* y, int n, long long hw, int C, int dt, double* dsum, double* dsq, void* stream);
int dfd_bn_finalize(const double* dsum, const double* dsq, double count, const float* gamma, const float* beta,
                    float* running_mean, float* running_var, long long* num_batches_tracked, float momentum,
                    float eps, int training, int C, float* scale, float* shift, float* mean, float* rstd,
                    void* stream);
int dfd_bn_act(const void* y, const float* scale, const float* shift, const float* gate, const void* res, void* out,
               int n, long long hw, int C, int act, int res_mode, int dt, void* stream);
/* pooled[n,c] = mean_hw act(scale*y + shift). `partial` (optional, max_chunks * n * C floats): when the batch alone cannot
 * fill the GPU, every image is reduced by up to max_chunks CTAs whose partial sums are added in a fixed order (the
 * forward stays bit-reproducible); NULL / max_chunks <= 1: one CTA per image */
int dfd_pool(const void* y, const float* scale, const float* shift, float* pooled, int n, long long hw, int C,
             int act, int dt, float* partial, int max_chunks, void* stream);
int dfd_bn_bwd_reduce(const void* g, const void* y, const void* out, const float* mean, const float* rstd, int n,
                      long long hw, int C, int dt, double* s1, double* s2, const void* fin, void* stream);
/* ReLU backward (and the residual add of the block above: g2 optional) fused into the reduction (ResNet block tail):
 * gm = round16(g + g2) * (out > 0) is stored and reduced in one pass */
int dfd_relu_bn_bwd_reduce(const void* g, const void* g2, const void* y, const void* out, void* gm, const float* mean,
                           const float* rstd, int n, long long hw, int C, int dt, double* s1, double* s2, void* stream);
int dfd_bn_bwd_finalize(const double* s1, const double* s2, double count, const float* gamma, const float* mean,
                        const float* rstd, float* dgamma, float* dbeta, float* cA, float* cB, float* cC, int C,
                        void* stream);
int dfd_bn_bwd_apply(const void* g, const void* y, const void* out, const float* cA, const float* cB,
                     const float* cC, void* dy, int n, long long hw, int C, int dt, void* stream);
int dfd_se_bwd_reduce(const void* da, const void* y, const float* scale, const float* shift, float* draw, int n,
                      long long hw, int C, int dt, void* stream);
int dfd_act_bwd(const void* da, const void* y, const float* scale, const float* shift, const float* mean,
                const float* rstd, const float* gate, const float* dpool, void* gu, int n, long long hw, int C,
                int act, int dt, double* s1, double* s2, const void* fin, void* stream);
int dfd_add_inplace(void* a, const void* b, long long numel, int dt, void* stream);

/* ---- squeeze-excite FCs: SqueezeExcite.forward, efficientnet_blocks.py:104-110 ------------------------ */
int dfd_se_fc_fwd(const float* pooled, const float* Wr, const float* br, const float* We, const float* be,
                  float* gate, int N, int C, int Cse, void* stream);
int dfd_se_fc_bwd(const float* draw, const float* pooled, const float* Wr, const float* br, const float* We,
                  const float* be, float* d_e, float* r, float* d_rpre, float* dpool, float* dWr, float* dbr,
                  float* dWe, float* dbe, int N, int C, int Cse, void* stream);

/* SE parameter gradients from the per-image vectors of the backward chain: dWe += d_e^T r, dbe += sum d_e,
 * dWr += d_rpre^T pooled, dbr += sum d_rpre (split partials in fixed slots, added in order) */
int dfd_se_fc_wgrad(const float* d_e, const float* r, const float* d_rpre, const float* pooled, float* dWr, float* dbr,
                    float* dWe, float* dbe, int N, int C, int Cse, void* stream);
/* Fused forms (one launch each; the CTA that completes an image's reduction carries on with that image's FC chain, which is
 * latency-bound and hides in the tail of the streaming kernel):
 *   dfd_pool_se      = dfd_pool + dfd_se_fc_fwd            (squeeze + excite gate)
 *   dfd_se_bwd_chain = dfd_se_bwd_reduce + the per-image part of dfd_se_fc_bwd   (dfd_se_fc_wgrad follows) */
int dfd_pool_se(const void* y, const float* scale, const float* shift, float* pooled, const float* Wr, const float* br,
                const float* We, const float* be, float* gate, int n, long long hw, int C, int Cse, int act, int dt,
                int max_chunks, void* stream);
int dfd_se_bwd_chain(const void* da, const void* y, const float* scale, const float* shift, float* draw, const float* pooled,
                     const float* Wr, const float* br, const float* We, const float* be, float* d_e, float* r, float* d_rpre,
                     float* dpool, int n, long long hw, int C, int Cse, int dt, void* stream);

/* ---- classifier + loss + accuracy: nn.Linear (efficientnet.py:348, resnet.py:467), LabelSmoothing /
 *      SoftTarget / nn.CrossEntropyLoss (loss/cross_entropy.py:20-36, train.py:509-520), accuracy
 *      (utils.py:170-186).  Any class count 1 <= K <= DFD_HEAD_KMAX; the loss needs K >= 2.
 *   K == 2: one CTA per image, softmax-CE computed as sigmoid-BCE on z1 - z0 (exactly equal).
 *   K != 2: fp32 shared-memory tile products for the logits, dpooled and dW, and one CTA per image for the softmax-CE
 *           (lse = max + log sum exp(z - max); targets t_k = smoothing/K + (1 - smoothing)[k == y], or the soft row),
 *           top-1 (first index of the row max; the label of a soft row is its first argmax) and dL/dlogits.
 *   Every output is one sum in a fixed order (no atomics, no split partials), so results are bit-reproducible. Logits-only
 *   calls with K = 3..32 sum over F in a different order than before DFD_HEAD_KMAX existed (last-bit differences).
 *   Labels are clamped into [0, K-1]. K > DFD_HEAD_KMAX, or a loss with K < 2, returns DFD_ERR_UNSUPPORTED.
 *   dfd_head_bwd: dpooled = dlogits W (overwritten); dW += dlogits^T pooled, db += sum_n dlogits (accumulated). ----- */
#define DFD_HEAD_KMAX 4096
int dfd_head_max_classes(void);
int dfd_head_fwd(const float* pooled, const float* W, const float* b, float* logits, int N, int F, int K,
                 const long long* target_i64, const float* target_soft, float smoothing, float loss_scale,
                 const float* loss_scale_dev, float* loss_acc, float* correct_acc, float* dlogits, void* stream);
int dfd_head_bwd(const float* dlogits, const float* pooled, const float* W, float* dW, float* db, float* dpooled,
                 int N, int F, int K, void* stream);

/* ---- the step's non-activation inputs (csrc/input.cu) ------------------------------------------------------------ */
/* PrefetchLoader.__iter__, dfd/timm/data/loader.py:243-256: uint8 NCHW batch -> 16-bit NCHW, (x - mean255[c]) / std255[c]
 * in fp32 with one rounding (mean255 / std255: device float[C] = mean*255 / std*255 repeated per frame, loader.py:229-230) */
int dfd_input_normalize(const void* x_u8, const float* mean255, const float* std255, void* out, int N, int C, int H, int W,
                        int dt, void* stream);
/* drop_path (layers/drop.py:84-100) and F.dropout (efficientnet.py:346-347) masks, already divided by keep_prob.
 * table: device array of { float* out; long long rows; int width; float keep_prob; int stream; int _pad; } - one random
 * draw per row, replicated over `width`; state: device int64 [seed, step] of the counter-based generator */
int dfd_rng_masks(const void* table, int count, const long long* state, void* stream);
int dfd_rng_tick(long long* state, void* stream);
int dfd_mul_f32(float* a, const float* b, long long n, void* stream);

/* ---- optimizers over the flat fp32 parameter arena: create_optimizer, optim_factory.py:26-100;
 *      RMSpropTF rmsprop_tf.py:57-122; AdamW adamw.py:55-117; apex AMP loss scaling train.py:353,632-634 ---- */
/* effective gradient scale = grad_scale * (*gscale_dev if non-null): 1/world for the DDP mean, 1/loss_scale on device.
 * lr_dev (optional, device float): when non-null it overrides `lr` - the schedulers mutate param_groups[i]['lr'] every
 * update (scheduler/scheduler.py:81-85), and a device-resident value lets one captured CUDA graph survive that.
 * step_dev (optional, device int): Adam's step count for the bias corrections, advanced by dfd_opt_tick. */
int dfd_sgd_step(float* p, const float* g, float* m, long long n, float lr, float momentum, float wd, int nesterov,
                 float grad_scale, const float* gscale_dev, const int* skip, void* p16, int dt, const float* lr_dev,
                 void* stream);
int dfd_adam_step(float* p, const float* g, float* m, float* v, long long n, float lr, float b1, float b2, float eps,
                  float wd, int decoupled, int step, float grad_scale, const float* gscale_dev, const int* skip, void* p16,
                  int dt, const float* lr_dev, const int* step_dev, void* stream);
int dfd_rmsprop_tf_step(float* p, const float* g, float* sq, float* mom, long long n, float lr, float alpha,
                        float eps, float wd, float momentum, float grad_scale, const float* gscale_dev, const int* skip,
                        void* p16, int dt, const float* lr_dev, void* stream);
/* *step_dev += 1 unless *skip (fp16 overflow): a skipped step does not advance Adam's bias correction (apex semantics) */
int dfd_opt_tick(int* step_dev, const int* skip, void* stream);
/* dst[0..n) = v0..v(n-1), n <= 8: host scalars (learning rates) to device memory, values carried in the launch itself */
int dfd_set_floats(float* dst, int n, float v0, float v1, float v2, float v3, float v4, float v5, float v6, float v7,
                   void* stream);
/* ModelEma.update (dfd/timm/utils.py:329-340) over the flat parameter / buffer arenas: ema = ema*decay + (1-decay)*model;
 * the int64 num_batches_tracked entries follow the reference's float arithmetic + truncating copy_ */
int dfd_ema_update(float* ema, const float* p, long long n, long long* ema_i64, const long long* p_i64, int n_i64,
                   float decay, void* stream);
int dfd_cast_arena(const float* p, void* p16, long long n, int dt, void* stream);
int dfd_check_finite(const float* g, long long n, int* flag, void* stream);
int dfd_update_loss_scale(int* flag, float* scale, int* good_steps, int interval, float* inv_scale_out,
                          void* stream);
/* table: device array of { const void* src; void* dst; int O; int I; } — dst[I,O] = transpose(src[O,I]) */
int dfd_transpose_weights(const void* table, int count, int dt, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DFD_B200_H */
