/* C ABI of the B200-native ConvLSTM / UNet-block hot path (libb200convlstm.so).
 *
 * The reference (dordanino12/unet-convlstm) has no native interface: its hot path is the Python
 * nn.Module code in train/unet.py, which lowers to ATen library kernels.  Each entry point below
 * names the reference lines whose arithmetic it replaces.  Conventions:
 *   - every pointer is a device pointer owned by the caller (the multi-tensor entry points take HOST arrays of
 *     device pointers and say so); nothing is allocated or freed here except one 4-byte watchdog flag per device
 *     and one 4-byte step counter per (device, stream) that runs a timestep-persistent kernel, and the split-K
 *     workspace per (device, stream) of the split weight gradients and b200_*_splitk_tc (kept for the process);
 *   - calls on distinct streams may be made concurrently from different threads;
 *   - activations are NHWC ("channels last"), bf16 on the tensor-core path (*_tc), fp32 or bf16 on
 *     the generic SIMT path; a sequence tensor is [T][B][H][W][C];
 *   - `stream` is a cudaStream_t passed as void*; kernels are launched on it, no hidden sync;
 *   - return value 0 = success, negative = B200_ERR_* below; b200_last_error() gives the text.
 *     No exception ever crosses this boundary.
 */
#ifndef B200_CONVLSTM_H
#define B200_CONVLSTM_H

#ifdef __cplusplus
extern "C" {
#endif

#define B200_OK 0
#define B200_ERR_SHAPE -1
#define B200_ERR_ALIGN -2
#define B200_ERR_CUDA -3
#define B200_ERR_ARG -4
#define B200_ERR_PIPELINE -5

/* Text of the last error raised on the calling thread. */
const char* b200_last_error(void);
/* Reads and clears the device watchdog flag (non-zero: id of the mbarrier a kernel timed out on). */
int b200_device_error(void);

/* TMA tensor maps are cached per (base pointer, dims, strides, box) inside the library: counters since load. */
int b200_tmap_cache_stats(long long* hits, long long* misses);

/* 1 if the tcgen05 path can tile this problem (else use the *_simt entry points). */
int b200_conv_tc_supported(int B, int H, int W, int C0, int C1, int N, int lstm);

/* Convolution over the virtual concat [src0 ; src1] (nn.Conv2d(.., k, padding=k//2), unet.py:19,70-71;
 * the torch.cat of unet.py:28 and :98 is never materialised).  wpacked: bf16 [k*k][N][C0+C1].
 * Output columns [0,split) go to dst0 (row stride ld0), [split,N) to dst1 (row stride ld1). */
int b200_conv_tc_fwd(const void* src0, int C0, const void* src1, int C1, int T, int B, int H, int W,
                     const void* wpacked, const float* bias, int N, int ksize, void* dst0,
                     long long ld0, int split, void* dst1, long long ld1, int out_fp32, int relu,
                     int accumulate, void* stream);

/* The first half of a DoubleConv stage (unet.py:70-71): the same convolution with the training-mode
 * nn.BatchNorm2d batch statistics of its output fused into the epilogue.  dst: bf16 [T][B][H][W][N]
 * (contiguous); stat_sum / stat_sumsq: fp64 [T][N], zeroed here and filled with the per-(t, channel) sum
 * and sum of squares over (B, H, W) of the stored (bf16) outputs -- the input of b200_bn_finalize, so
 * b200_bn_stats and its extra pass over dst are not needed. */
int b200_conv_bnstats_tc_fwd(const void* src0, int C0, const void* src1, int C1, int T, int B, int H, int W,
                             const void* wpacked, const float* bias, int N, int ksize, void* dst,
                             double* stat_sum, double* stat_sumsq, void* stream);

/* Inference form of one half of a DoubleConv stage (Conv3x3 + eval-mode BatchNorm2d + ReLU, unet.py:70-71 with
 * model.eval()): out = relu(conv(x) * scale[n] + shift[n]), the BatchNorm folded into the GEMM epilogue
 * (scale = gamma / sqrt(running_var + eps), shift = beta + (conv_bias - running_mean) * scale), so the
 * pre-activation tensor and the two normalisation passes of the training path do not exist.  dst: bf16. */
int b200_conv_affine_relu_tc_fwd(const void* src0, int C0, const void* src1, int C1, int T, int B, int H, int W,
                                 const void* wpacked, const float* scale, const float* shift, int N, int ksize,
                                 void* dst, int relu, void* stream);

/* nn.ConvTranspose2d(Cin, Cout, 2, stride=2) + F.pad to the skip size (Up, unet.py:90-97) in one kernel: the
 * GEMM [P, Cin] x [Cin, 4*Cout] (wpacked: bf16 [1][4*Cout (tap, co)][Cin]) whose epilogue adds bias[co] and
 * writes column block `tap` of input pixel (h, w) to output pixel (2h + tap/2 + oy, 2w + tap%2 + ox) of
 * y: bf16 [T][B][Hd][Wd][Cout], (oy, ox) = ((Hd-2H)/2, (Wd-2W)/2); y must be zero-filled when Hd > 2H or Wd > 2W. */
int b200_convT2x2_tc_fwd(const void* x, int Cin, int T, int B, int H, int W, const void* wpacked, const float* bias,
                         int Cout, void* y, int Hd, int Wd, void* stream);

/* One ConvLSTM cell step, ConvLSTMCell.forward (unet.py:21-36): gate conv over [x ; h_prev] fused
 * with sigmoid/tanh and the c/h update.  wpacked: bf16 [k*k][4*Ch gate-interleaved][Cin+Ch];
 * bias_packed fp32 [4*Ch] in the same row order (b200_pack_lstm_weights).  h_prev / c_prev may be
 * NULL (zero state, unet.py:23-25).  gates_out (bf16 [P][4][Ch], activated i,f,g,o) may be NULL. */
int b200_convlstm_cell_fwd_tc(const void* x, int Cin, const void* h_prev, int Ch, int B, int H, int W,
                              const void* wpacked, const float* bias_packed, const float* c_prev,
                              float* c_next, void* h_next, void* gates_out, int ksize, void* stream);

/* Whole-sequence forward of one ConvLSTM layer, the t-loop of ConvLSTM.forward (unet.py:52-57), as ONE
 * timestep-persistent cooperative kernel: the grid iterates over t = 0..T-1, h_t / c_t stay in the
 * (L2-resident) state buffers, a grid-wide counter separates the steps, no host round trip per step.
 * x_seq: bf16 [T][B][H][W][Cin]; h_all: bf16 [T+1][B][H][W][Ch], slot 0 = initial state (ignored when
 * have_h0 == 0: zero state, unet.py:23-25), slot t+1 = h_t; c_all: fp32 [T+1][...] likewise;
 * gates: bf16 [T][P][4][Ch] activated i,f,g,o (kept for BPTT), or NULL (gate recompute, see
 * b200_convlstm_gates_recompute_tc).  Also uses one 4-byte per-device step
 * counter owned by the library. */
int b200_convlstm_seq_fwd_tc(const void* x_seq, int Cin, void* h_all, int Ch, int T, int B, int H, int W,
                             const void* wpacked, const float* bias_packed, float* c_all, void* gates,
                             int have_h0, int ksize, void* stream);

/* ---- Split K for single-frame problems with few M tiles (streaming inference, one frame at a time: at B = 1 and
 * 4x4 .. 16x16 pixels the tensor-core tiling has a single M tile, so the unsplit launch occupies a handful of SMs and
 * each CTA walks the whole K = 9 x (C0 + C1) loop alone).  The implicit GEMM of b200_conv_tc_fwd (1-CTA kernel) runs
 * `splits` contiguous ranges of its (tap, 64-channel chunk) k-blocks side by side; each range stores fp32 partial sums
 * [P][N] (P = B*H*W) to its own slice of a library-owned per-(device, stream) workspace, and a second kernel adds the
 * slices in split order -- no atomics, the result does not depend on which split finishes first -- and applies the
 * epilogue.  Two kernel launches per call.  The workspace grows on the first call of a larger shape on a stream and
 * never during a CUDA-graph capture (that call fails instead).  bf16 only.
 * b200_splitk_splits: the number of splits the library recommends for a bf16 convolution of that shape (1 = do not
 * split; see csrc/capi.cu for the rule and the measurement behind it). */
int b200_splitk_splits(int B, int H, int W, int C0, int C1, int N, int ksize);
/* b200_convlstm_cell_fwd_tc split over K: arguments as there, without gates_out (inference keeps no gates). */
int b200_convlstm_cell_fwd_splitk_tc(const void* x, int Cin, const void* h_prev, int Ch, int B, int H, int W,
                                     const void* wpacked, const float* bias_packed, const float* c_prev, float* c_next,
                                     void* h_next, int splits, int ksize, void* stream);
/* b200_conv_affine_relu_tc_fwd of one frame (T = 1) split over K: dst = relu?(conv * scale + shift), bf16 or fp32
 * (out_fp32); scale / shift may be NULL (1 / 0), which leaves the plain convolution. */
int b200_conv_affine_relu_splitk_tc(const void* src0, int C0, const void* src1, int C1, int B, int H, int W,
                                    const void* wpacked, const float* scale, const float* shift, int N, int ksize,
                                    void* dst, int out_fp32, int relu, int splits, void* stream);

/* ---- "tf32" precision mode (north_star: "bf16/TF32 inputs with fp32 accumulation"; the reference's own GPU numerics:
 * torch enables TF32 in cuDNN convolutions by default).  Same implicit GEMM as the *_tc entry points with fp32 tensors
 * everywhere: sources, packed weights ([k*k][N][C0+C1], gate-interleaved for the cell), outputs, h and the activated
 * gates; the products are tcgen05 kind::tf32 (10-bit mantissa), the accumulation fp32.  Channel counts must be
 * multiples of 8 (K blocks of 32 / 16 / 8 channels = rows of 128 / 64 / 32 bytes). ---- */
int b200_conv_tf32_supported(int B, int H, int W, int C0, int C1, int N, int lstm);
int b200_conv_tf32_fwd(const float* src0, int C0, const float* src1, int C1, int T, int B, int H, int W,
                       const float* wpacked, const float* bias, int N, int ksize, float* dst0, long long ld0, int split,
                       float* dst1, long long ld1, int relu, int accumulate, void* stream);
/* Weight gradient in the tf32 mode: dw += ..., arguments and reduction as b200_wgrad_tc with fp32 dz / src. */
int b200_wgrad_tf32_supported(int B, int H, int W, int Nz, int Csrc);
int b200_wgrad_tf32(const float* dz, int Nz, const float* src, int Csrc, int T, int B, int H, int W, int ksize, float* dw,
                    long long ldk, int koff, void* stream);
/* One fused ConvLSTM cell step (unet.py:21-36) in the tf32 mode; arguments as b200_convlstm_cell_fwd_tc. */
int b200_convlstm_cell_fwd_tf32(const float* x, int Cin, const float* h_prev, int Ch, int B, int H, int W,
                                const float* wpacked, const float* bias_packed, const float* c_prev, float* c_next,
                                float* h_next, float* gates_out, int ksize, void* stream);

/* Gate recompute for BPTT (north_star "gate-gradient recompute"; the reference's autograd instead keeps the four
 * activated gates of every step, unet.py:29-33): the activated gates of ALL T steps from the stored x_t, h_{t-1}
 * (h_all slot t) and c_{t-1} (c_all slot t) in one tensor-core launch -- the steps are independent once the states
 * are known.  Same arithmetic as the forward kernel; writes only gates_out (bf16 [T][P][4][Ch]), which may be the
 * buffer the gate-gradient kernel then overwrites with dz.  With a zero initial state slot 0 of h_all / c_all must
 * hold zeros. */
int b200_convlstm_gates_recompute_tc(const void* x_seq, int Cin, const void* h_all, int Ch, int T, int B, int H, int W,
                                     const void* wpacked, const float* bias_packed, const float* c_all, void* gates_out,
                                     int ksize, void* stream);

/* Whole-sequence BPTT data path of one ConvLSTM layer -- the autograd of the t-loop of ConvLSTM.forward
 * (unet.py:52-57) -- as ONE timestep-persistent cooperative kernel running t = T-1 .. 0.  Step t is the
 * data-gradient convolution of dz_t (wd_packed: bf16 [k*k flipped][Cin+Ch][4*Ch]) into [dx_t ; dh_{t-1}];
 * the dh columns never leave the epilogue registers: they are added to the upstream dh_seq[t-1] and go
 * through the gate-gradient math of step t-1 (autograd of unet.py:30-35), which writes dz_{t-1} (the next
 * step's GEMM operand) and dL/dc_{t-2}.  dz_all: bf16 [T][P][4*Ch] (i|f|g|o), slot T-1 filled by the caller
 * (b200_lstm_gates_bwd), the other slots here -- afterwards it is the dz operand of the weight gradient.
 * gates: bf16 [T][P][4][Ch]; c_all: fp32 [T+1][P][Ch]; dh_seq: bf16 [T][P][Ch] or NULL; dc_buf: fp32
 * [2][P][Ch], slot (T-1)&1 filled by the caller, slot 0 holds dL/dc_{-1} on return; dx_seq: bf16
 * [T][P][Cin] or NULL (not needed); dh0: bf16 [P][Ch] or NULL (gradient of the initial hidden state). */
int b200_convlstm_seq_bwd_tc(void* dz_all, const void* wd_packed, const void* gates, const float* c_all,
                             const void* dh_seq, float* dc_buf, void* dx_seq, void* dh0, int Cin, int Ch,
                             int T, int B, int H, int W, int have_h0, int ksize, void* stream);

/* Weight gradient of a convolution, summed over all T*B images (autograd of nn.Conv2d, unet.py:19
 * and :70-71; for the ConvLSTM this is the BPTT sum over timesteps):
 *   dw[tap][n][koff + k] += sum_{t,p} dz[t,p,n] * src[t, p+tap, k]
 * dz: bf16 [T][B][H][W][Nz], src: bf16 [T][B][H][W][Csrc], dw: fp32 [k*k][Nz][ldk]; columns outside
 * [koff, koff + Csrc) are not touched.  The reduction over t,p is split; each split stores its partial sums to its own
 * slice of the per-stream workspace and a second kernel adds the slices to dw in split order, at any split count
 * (one included): the result does not depend on which split finishes first. */
int b200_wgrad_tc(const void* dz, int Nz, const void* src, int Csrc, int T, int B, int H, int W,
                  int ksize, float* dw, long long ldk, int koff, void* stream);
/* The kernel b200_wgrad_tc (in_fp32 = 0) or b200_wgrad_tf32 (in_fp32 = 1) runs for this problem and its number of
 * reduction splits, without launching anything: plan[0] = 0 wgrad_tc, 1 wgrad_tc2, 2 wgrad_halo; plan[1] = splits. */
int b200_wgrad_plan(int Nz, int Csrc, int T, int B, int H, int W, int ksize, long long ldk, int koff, int in_fp32,
                    int* plan);

/* 1 if b200_wgrad_tc can tile this problem. */
int b200_wgrad_tc_supported(int B, int H, int W, int Nz, int Csrc);

/* ---- generic CUDA-core convolutions: the fp32 check mode (dtype_fp32 = 1, 1e-5 parity with the
 * reference's fp32 arithmetic) and shapes the tcgen05 path cannot tile (dtype_fp32 = 0: bf16 storage).
 * Same math and packed-weight layout as the *_tc entry points; IMG = T*B images. ---- */
int b200_conv_simt_fwd(const void* src0, int C0, const void* src1, int C1, int IMG, int H, int W,
                       const void* w, const float* bias, int N, int ksize, void* dst0, long long ld0,
                       int split, void* dst1, long long ld1, int dtype_fp32, int out_fp32, int relu,
                       void* stream);
int b200_wgrad_simt(const void* dz, int Nz, const void* src, int Csrc, int IMG, int H, int W, int ksize,
                    float* dw, long long ldk, int koff, int dtype_fp32, void* stream);

/* ---- BatchNorm2d + ReLU of DoubleConv (unet.py:70-71), statistics per (t, channel) over the P = B*H*W
 * pixels of one timestep because the reference calls the block once per timestep (unet.py:179-182,
 * :196-202).  x, y, dy, dx: [T][P][C]; sum / sumsq / sum_g / sum_gx: double [T][C] workspaces. ---- */
int b200_bn_stats(const void* x, int T, long long P, int C, int dtype_fp32, double* sum, double* sumsq,
                  void* stream);
/* training: mean/rstd/scale/shift [T][C] from the sums and T sequential momentum updates of the running
 * estimates (unbiased variance); eval: scale/shift [1][C] from the running estimates. */
int b200_bn_finalize(const double* sum, const double* sumsq, int T, long long n, int C, const float* gamma,
                     const float* beta, float* running_mean, float* running_var, float eps, float momentum,
                     int training, float* mean, float* rstd, float* scale, float* shift, void* stream);
/* y = relu(x*scale[t][c] + shift[t][c]); tstride = C (training) or 0 (eval) */
int b200_bn_relu_apply(const void* x, const float* scale, const float* shift, void* y, int T, long long P, int C,
                       int tstride, int relu, int dtype_fp32, void* stream);
/* autograd of BatchNorm2d+ReLU: g = dy*[y>0]; sum_g = sum g, sum_gx = sum g*xhat */
int b200_bn_relu_bwd_reduce(const void* x, const void* dy, const float* mean, const float* rstd,
                            const float* scale, const float* shift, int T, long long P, int C, int tstride,
                            int dtype_fp32, double* sum_g, double* sum_gx, void* stream);
/* also yields the gradient of the preceding conv's bias, dconv_bias = sum_pixels dx (may be NULL): it is
 * identically zero in training mode and scale*sum_g in eval mode (scale: [C], the eval-mode scale) */
int b200_bn_bwd_finalize(const double* sum_g, const double* sum_gx, int T, long long n, int C, int training,
                         const float* scale, float* coef1, float* coef2, float* dgamma, float* dbeta,
                         float* dconv_bias, int accumulate, void* stream);
/* dx = scale*(g - coef1 - xhat*coef2) */
int b200_bn_relu_bwd_apply(const void* x, const void* dy, const float* mean, const float* rstd,
                           const float* scale, const float* shift, const float* coef1, const float* coef2,
                           void* dx, int T, long long P, int C, int tstride, int dtype_fp32, void* stream);

/* nn.MaxPool2d(2) of Down (unet.py:81) and its backward (first maximum in scan order gets the gradient). */
int b200_maxpool2_fwd(const void* x, void* y, long long IMG, int H, int W, int C, int dtype_fp32, void* stream);
int b200_maxpool2_bwd(const void* x, const void* dy, void* dx, long long IMG, int H, int W, int C,
                      int accumulate, int dtype_fp32, void* stream);

/* BatchNorm2d + ReLU + MaxPool2d(2) in one pass for a DoubleConv output that feeds both a skip connection and the
 * next Down stage (unet.py:70-71 -> :81, :179-182): y = relu(x*scale+shift) [T][B][H][W][C] and pooled = maxpool2x2(y)
 * [T][B][H/2][W/2][C].  H and W even.  The backward pair takes the two gradients of y -- dy through the skip connection
 * (may be NULL) and dp through the pool -- and replaces b200_maxpool2_bwd + b200_bn_relu_bwd_reduce / _apply; results
 * are bit-identical to the separate entry points. */
int b200_bn_relu_apply_pool(const void* x, const float* scale, const float* shift, void* y, void* pooled, int T,
                            long long B, int H, int W, int C, int tstride, int dtype_fp32, void* stream);
int b200_bn_relu_pool_bwd_reduce(const void* x, const void* dy, const void* dp, const float* mean, const float* rstd,
                                 const float* scale, const float* shift, int T, long long B, int H, int W, int C,
                                 int tstride, int dtype_fp32, double* sum_g, double* sum_gx, void* stream);
int b200_bn_relu_pool_bwd_apply(const void* x, const void* dy, const void* dp, const float* mean, const float* rstd,
                                const float* scale, const float* shift, const float* coef1, const float* coef2,
                                void* dx, int T, long long B, int H, int W, int C, int tstride, int dtype_fp32,
                                void* stream);

/* BatchNorm2d + ReLU + the 1x1 OutConv with ONE output channel in one pass (the last DoubleConv feeding `outc`,
 * unet.py:70-71 -> :104, :202-203): out[t][p] = b + sum_c relu(x*scale+shift)[t][p][c] * w[c], fp32; the activation is
 * never written.  C / 8 (bf16) or C / 4 (fp32) must be a power of two <= 32.  Backward: the data gradient of the 1x1
 * convolution is dout[p] * w[c], formed inside the two BatchNorm-backward passes; the reduction pass also yields the
 * OutConv weight gradient dw[c] = sum_{t,p} dout * y (sum_dw: fp64 workspace [C]; dw fp32 [C], may be NULL).  These
 * replace b200_bn_relu_apply + b200_outconv_fwd and b200_outconv_bwd + b200_bn_relu_bwd_reduce / _apply. */
int b200_bn_relu_outconv_fwd(const void* x, const float* scale, const float* shift, const float* w, const float* b,
                             float* out, int T, long long P, int C, int tstride, int dtype_fp32, void* stream);
int b200_bn_relu_outconv_bwd_reduce(const void* x, const float* dout, const float* w, const float* mean,
                                    const float* rstd, const float* scale, const float* shift, int T, long long P, int C,
                                    int tstride, int dtype_fp32, double* sum_g, double* sum_gx, double* sum_dw, float* dw,
                                    void* stream);
int b200_bn_relu_outconv_bwd_apply(const void* x, const float* dout, const float* w, const float* mean, const float* rstd,
                                   const float* scale, const float* shift, const float* coef1, const float* coef2,
                                   void* dx, int T, long long P, int C, int tstride, int dtype_fp32, void* stream);

/* ConvLSTM gate math when it is not fused into the GEMM epilogue (unet.py:29-35).  z: fp32 [P][4*Ch]
 * pre-activations in the reference's chunk order i|f|g|o; gates: [P][4][Ch] activated. */
int b200_lstm_gates_fwd(const float* z, const float* c_prev, void* gates, float* c_next, void* h_next,
                        long long P, int Ch, int dtype_fp32, void* stream);
/* One BPTT step of the gate math (autograd of unet.py:30-35): dh = dh_a + dh_b (either may be NULL),
 * dc_next may be NULL; writes dz [P][4*Ch] (i|f|g|o) and dc_prev. */
int b200_lstm_gates_bwd(const void* gates, const float* c_prev, const float* c_next, const void* dh_a,
                        const void* dh_b, const float* dc_next, void* dz, float* dc_prev, long long P, int Ch,
                        int dtype_fp32, void* stream);

/* out[c] (+)= sum_rows x[row][c]  (bias gradients); workspace: double [C] */
int b200_colsum(const void* x, long long rows, int C, int dtype_fp32, double* workspace, float* out,
                int accumulate, void* stream);

/* OutConv (1x1 conv, unet.py:101-107): y fp32 [P][O]; backward: dx (may be NULL), dw [O][C], db [O];
 * workspace: double [max(C,O)] */
int b200_outconv_fwd(const void* x, const float* w, const float* b, float* y, long long P, int C, int O,
                     int dtype_fp32, void* stream);
int b200_outconv_bwd(const void* x, const float* w, const float* dy, long long P, int C, int O, int dtype_fp32,
                     void* dx, double* workspace, float* dw, float* db, int accumulate, void* stream);

/* SpatialAttention (unet.py:113-125; TemporalUNetDualView(use_attention=True) applies it to the bottleneck output):
 *   y = x * a,  a = sigmoid(conv_k([mean_c x ; amax_c x]))   (2 -> 1 channels, padding k/2, no bias; k = 1, 3, 5 or 7)
 * per image of x [IMG][H][W][C] (bf16, or fp32 if dtype_fp32; y and dx alike).  w: fp32 [2][k][k] (nn.Conv2d weight
 * [1, 2, k, k]), read from device memory at run time.  Forward writes pooled fp32 [IMG][H][W][2] (mean, max) and a fp32
 * [IMG][H][W], both inputs of the backward.  Backward, given dy: with ds = (sum_c dy*x) * (1-a) * a and (dmean, dmax) the
 * transposed convolution of ds,
 *   dx = dy*a + dmean / C + [x == max] * dmax / (number of channels equal to the max)     (dx may be NULL: not computed)
 *   dw = sum over pixels of ds * pooled at the tap's pixel                               (dw may be NULL: not computed)
 * the max split evenly among ties as torch.amax's backward does.  ws: fp32 workspace of 2*P + ceil(P / 2048) * 2*k*k
 * floats, P = IMG*H*W; dw is summed per range of 2048 pixels and the ranges added in order: no atomics, run-to-run
 * bit-identical.  16-byte accesses when C * element size is a multiple of 16 and the activation pointers are 16-byte
 * aligned, scalar ones otherwise.  pooled must be 8-byte aligned (the backward reads it as float2; B200_ERR_ALIGN
 * otherwise).  Kernel launches: 2 forward; backward 2, +1 with dx, +2 with dw (the sums and splitk_reduce). */
int b200_spatial_attention_fwd(const void* x, const float* w, long long IMG, int H, int W, int C, int ksize,
                               int dtype_fp32, float* pooled, float* a, void* y, void* stream);
int b200_spatial_attention_bwd(const void* x, const void* dy, const float* w, const float* pooled, const float* a,
                               long long IMG, int H, int W, int C, int ksize, int dtype_fp32, float* ws, void* dx,
                               float* dw, void* stream);

/* Pixel shuffle of ConvTranspose2d(k=2, stride=2) (unet.py:90) with the F.pad offsets of unet.py:95-97:
 * z [IMG][H][W][4][C] (+bias) <-> y [IMG][Hd][Wd][C] at (2h+i+oy, 2w+j+ox), tap = 2i+j. */
int b200_shuffle2x2(const void* src, void* dst, const float* bias, long long IMG, int H, int W, int C, int Hd,
                    int Wd, int oy, int ox, int unshuffle, int dtype_fp32, void* stream);

/* dst[i . dst_strides] (+)= src[i . src_strides] over a 5-D index space (layout changes at the module
 * boundary: NCHW <-> NHWC; weight packing OIHW <-> [tap][N][K]).  Strides in elements. */
int b200_strided_copy(const void* src, int src_fp32, void* dst, int dst_fp32, const long long* dims,
                      const long long* src_strides, const long long* dst_strides, int accumulate, void* stream);

/* Weight layout changes, once per weight and optimizer step.  src: the reference's parameter layout, fp32
 * [A][B][taps] with the tap index fastest (Conv2d OIHW: A = Cout, B = Cin; ConvTranspose2d IOHW: A = Cin, B = Cout).
 * b200_pack_weight writes the GEMM operand dst (bf16, or fp32 if dst_fp32):
 *     a_contig = 0:  dst[tap' * tap_pitch + pa(a) * row_pitch + b]      (K-major B operand of the forward conv)
 *     a_contig = 1:  dst[tap' * tap_pitch + b * row_pitch + pa(a)]      (data-gradient weights)
 * tap' = taps-1-tap if flip else tap; pa = the gate interleave of the fused ConvLSTM kernel when perm_ch = Ch != 0
 * (row g*Ch + nt*cht + j -> (nt*4 + g)*cht + j, unet.py:19,29 rows blocked i,f,g,o), identity otherwise.  Padding
 * rows / columns of dst are the caller's (zero-filled beforehand).
 * b200_unpack_wgrad is the way back for weight gradients: packed fp32 [taps][A][ldb] -> dst fp32 [A][B][taps]. */
int b200_pack_weight(const float* src, int A, int B, int taps, void* dst, int dst_fp32, int a_contig, int flip,
                     long long tap_pitch, long long row_pitch, int perm_ch, int perm_cht, void* stream);
int b200_unpack_wgrad(const float* packed, int A, int B, int taps, long long ldb, float* dst, void* stream);

/* The reference's training loss `compute_loss` (main.py:28-72): weighted L1 (weight 1 + 4|y|^3) + 0.005 x the
 * spatial-gradient loss on the [H-1, W-1] crop; with a mask (float 0/1, same shape) the means are masked and
 * carry the 1e-8 epsilon of main.py:42,65, with mask == NULL they are plain means (main.py:45,67).
 * y_pred / y / mask / d_y_pred: fp32 [IMG][H][W] (any leading shape flattened to IMG); sums: fp64 [6] workspace
 * written by the forward pass and read by the backward pass; loss: one fp32 on the device; grad_out: one fp32 on
 * the device (NULL = 1).  Two passes over the maps instead of ~25 + ~40 element-wise launches. */
int b200_wl1_grad_loss_fwd(const float* y_pred, const float* y, const float* mask, long long IMG, int H, int W,
                           double* sums, float* loss, void* stream);
int b200_wl1_grad_loss_bwd(const float* y_pred, const float* y, const float* mask, long long IMG, int H, int W,
                           const double* sums, const float* grad_out, float* d_y_pred, void* stream);

/* Error metrics of the reference's train / evaluate loops (main.py:110-145, :166-199): both maps are de-normalised
 * like NPZSequenceDataset.denormalize (unet.py:306-327; transform 0 = identity, 1 = asinh, 2 = signed_log) and
 * acc[0..3] += {sum |d|, sum d^2, sum d, count} over the pixels with mask != 0 (mask == NULL: all pixels).
 * y_pred / y / mask: fp32 [n]; acc: fp64 [4] on the device, zeroed by the caller at the start of an epoch and read
 * once at its end (MAE = acc0/acc3, RMSE = sqrt(acc1/acc3), ME = acc2/acc3). */
int b200_denorm_metrics_accum(const float* y_pred, const float* y, const float* mask, long long n, int transform,
                              double trans_min, double trans_max, double y_scale, double* acc, void* stream);

/* One training batch of the reference's NPZSequenceDataset (unet.py:393-401 + default_collate) from the raw dataset
 * kept in device memory, in one launch: for b < B, row n = idx[b] (idx: int64 [B] on the device),
 *   mask[b,t,0] = X[n,t,0] > 1.1f;  x[b,t,c] = X[n,t,c] / (float)norm_const (IEEE fp32 division);
 *   y[b,t,0]    = 2 * (tr(clip(Y[n,t,0])) - trans_min) / trans_range - 1, rounded once to fp32,
 * where clip (if clip != 0) bounds by [min_vel, max_vel] like np.clip, tr is transform 0 = identity, 1 = asinh(v /
 * y_scale), 2 = sign(v) * log1p(|v| / y_scale), and trans_range = trans_max - trans_min as the caller computed it.
 * The dtypes follow NumPy: fp64_transform = 1 runs clip, transform and affine map in fp64 (np.float64 clip bounds),
 * fp64_affine = 1 only the affine map (np.float64 trans_min); otherwise every step is fp32 with the constants rounded to
 * fp32.  X: fp32 [N][T][Cx][H][W], Y: fp32 [N][T][1][H][W]; x: fp32 [B][T][Cx][H][W], y / mask: fp32 [B][T][1][H][W],
 * all contiguous.  16-byte accesses when H*W % 4 == 0 and the bases are 16-byte aligned, scalar ones otherwise.  An idx
 * outside [0, N) is never read: its item comes out as x = y = NaN, mask = 0 (callers check indices beforehand). */
int b200_sequence_batch(const float* X, const float* Y, long long N, int T, int Cx, int H, int W, const void* idx, int B,
                        double norm_const, int clip, double min_vel, double max_vel, int transform, double y_scale,
                        double trans_min, double trans_range, int fp64_transform, int fp64_affine, float* x, float* y,
                        float* mask, void* stream);

/* Gradient clipping + AdamW of the reference's step (main.py:106 clip_grad_norm_(params, 1.0); main.py:275
 * torch.optim.AdamW) over a LIST of fp32 tensors.  The pointer arrays (params, grads, ...) and numel live in HOST
 * memory and hold n device pointers / element counts; they are copied into the kernel parameters (48 tensors per
 * launch), so they may be freed as soon as the call returns.
 *   b200_grad_sqnorm_multi : *sqnorm (fp64, device) = sum over all tensors of g^2
 *   b200_grad_clip_multi   : g *= min(1, max_norm / (sqrt(*sqnorm) + 1e-6)) in place (clip_grad_norm_ semantics)
 *   b200_adamw_multi       : decoupled weight decay + Adam moments + bias-corrected update, torch.optim.AdamW
 *                            arithmetic (amsgrad = False, maximize = False); `step` is the 1-based update count.
 *                            sqnorm != NULL and max_norm > 0 folds the clip coefficient into the gradient read
 *                            (the gradients themselves are left unscaled). */
int b200_grad_sqnorm_multi(int n, const void* const* grads, const long long* numel, double* sqnorm, void* stream);
int b200_grad_clip_multi(int n, void* const* grads, const long long* numel, const double* sqnorm, float max_norm,
                         void* stream);
int b200_adamw_multi(int n, void* const* params, const void* const* grads, void* const* exp_avg,
                     void* const* exp_avg_sq, const long long* numel, float lr, float beta1, float beta2, float eps,
                     float weight_decay, long long step, const double* sqnorm, float max_norm, void* stream);
/* AdamW (main.py:275) of convolution weights [A][B][taps] fp32 (OIHW: A = Cout, B = Cin; IOHW for ConvTranspose2d) that also
 * emits the GEMM-operand copies of the UPDATED weights -- SURVEY section 8 f1, "fused AdamW that also emits the packed bf16
 * weights": same arithmetic as b200_adamw_multi (bit-identical), then up to two destinations per weight in the layouts
 * of b200_pack_weight.  b200_adamw_pack_multi: n weights in one launch per 16; host tables like b200_adamw_multi,
 * dims = [n][3] {A, B, taps}, dst0 / dst1 = [n] device pointers (NULL = unused), geom0 / geom1 = [n][7]
 * {dst_fp32, a_contig, flip, tap_pitch, row_pitch, perm_ch, perm_cht} as in b200_pack_weight.  b200_adamw_pack: one
 * weight, the same through scalar arguments. */
int b200_adamw_pack_multi(int n, void* const* params, const void* const* grads, void* const* exp_avg,
                          void* const* exp_avg_sq, const long long* dims, float lr, float beta1, float beta2, float eps,
                          float weight_decay, long long step, const double* sqnorm, float max_norm, void* const* dst0,
                          const long long* geom0, void* const* dst1, const long long* geom1, void* stream);
int b200_adamw_pack(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int A, int B, int taps,
                    float lr, float beta1, float beta2, float eps, float weight_decay, long long step,
                    const double* sqnorm, float max_norm, void* dst0, int dst0_fp32, int a_contig0, int flip0,
                    long long tap_pitch0, long long row_pitch0, int perm_ch0, int perm_cht0, void* dst1, int dst1_fp32,
                    int a_contig1, int flip1, long long tap_pitch1, long long row_pitch1, int perm_ch1, int perm_cht1,
                    void* stream);

#ifdef __cplusplus
}
#endif
#endif
