// Launchers of the HBM-bound kernels (pointwise.cu) and of the generic SIMT convolutions
// (conv_simt.cu).  dtype_fp32: 1 = fp32 storage (check mode), 0 = bf16 storage.
#pragma once
#include "common.cuh"

namespace b200 {

int launch_bn_stats(const void* x, int T, long long P, int C, int dtype_fp32, double* sum, double* sumsq,
                    cudaStream_t stream);
int launch_colsum(const void* x, long long rows, int C, int dtype_fp32, double* out, cudaStream_t stream);
int launch_bn_relu_bwd_reduce(const void* x, const void* dy, const float* mean, const float* rstd,
                              const float* scale, const float* shift, int T, long long P, int C, int tstride,
                              int dtype_fp32, double* sum_g, double* sum_gx, cudaStream_t stream);
int launch_outconv_wgrad(const void* x, const float* dy, long long P, int C, int O, int o, int dtype_fp32,
                         double* out, cudaStream_t stream);
int launch_bn_finalize(const double* sum, const double* sumsq, int T, long long n, int C, const float* gamma,
                       const float* beta, float* running_mean, float* running_var, float eps, float momentum,
                       int training, float* mean, float* rstd, float* scale, float* shift, cudaStream_t stream);
int launch_bn_bwd_finalize(const double* sum_g, const double* sum_gx, int T, long long n, int C, int training,
                           const float* scale, float* coef1, float* coef2, float* dgamma, float* dbeta,
                           float* dconv_bias, int accumulate, cudaStream_t stream);
int launch_cast_double(const double* src, float* dst, int n, int accumulate, cudaStream_t stream);
int launch_bn_relu_apply(const void* x, const float* scale, const float* shift, void* y, int T, long long P, int C,
                         int tstride, int relu, int dtype_fp32, cudaStream_t stream);
int launch_bn_relu_bwd_apply(const void* x, const void* dy, const float* mean, const float* rstd, const float* scale,
                             const float* shift, const float* coef1, const float* coef2, void* dx, int T,
                             long long P, int C, int tstride, int dtype_fp32, cudaStream_t stream);
int launch_maxpool2_fwd(const void* x, void* y, long long IMG, int H, int W, int C, int dtype_fp32,
                        cudaStream_t stream);
int launch_maxpool2_bwd(const void* x, const void* dy, void* dx, long long IMG, int H, int W, int C, int accumulate,
                        int dtype_fp32, cudaStream_t stream);
int launch_bn_relu_apply_pool(const void* x, const float* scale, const float* shift, void* y, void* pooled, int T,
                              long long B, int H, int W, int C, int tstride, int dtype_fp32, cudaStream_t stream);
int launch_bn_relu_pool_bwd_reduce(const void* x, const void* dy, const void* dp, const float* mean, const float* rstd,
                                   const float* scale, const float* shift, int T, long long B, int H, int W, int C,
                                   int tstride, int dtype_fp32, double* sum_g, double* sum_gx, cudaStream_t stream);
int launch_bn_relu_pool_bwd_apply(const void* x, const void* dy, const void* dp, const float* mean, const float* rstd,
                                  const float* scale, const float* shift, const float* coef1, const float* coef2,
                                  void* dx, int T, long long B, int H, int W, int C, int tstride, int dtype_fp32,
                                  cudaStream_t stream);
int launch_bn_relu_outconv_fwd(const void* x, const float* scale, const float* shift, const float* w, const float* b,
                               float* out, int T, long long P, int C, int tstride, int dtype_fp32, cudaStream_t stream);
int launch_bn_relu_outconv_bwd_reduce(const void* x, const float* dout, const float* w, const float* mean, const float* rstd,
                                      const float* scale, const float* shift, int T, long long P, int C, int tstride,
                                      int dtype_fp32, double* sum_g, double* sum_gx, double* sum_dw, float* dw,
                                      cudaStream_t stream);
int launch_bn_relu_outconv_bwd_apply(const void* x, const float* dout, const float* w, const float* mean, const float* rstd,
                                     const float* scale, const float* shift, const float* coef1, const float* coef2,
                                     void* dx, int T, long long P, int C, int tstride, int dtype_fp32,
                                     cudaStream_t stream);
int launch_lstm_gates_fwd(const float* z, const float* c_prev, void* gates, float* c_next, void* h_next, long long P,
                          int Ch, int dtype_fp32, cudaStream_t stream);
int launch_lstm_gates_bwd(const void* gates, const float* c_prev, const float* c_next, const void* dh_a,
                          const void* dh_b, const float* dc_next, void* dz, float* dc_prev, long long P, int Ch,
                          int dtype_fp32, cudaStream_t stream);
int launch_outconv_fwd(const void* x, const float* w, const float* b, float* y, long long P, int C, int O,
                       int dtype_fp32, cudaStream_t stream);
int launch_outconv_dgrad(const float* dy, const float* w, void* dx, long long P, int C, int O, int dtype_fp32,
                         cudaStream_t stream);
int launch_shuffle2x2(const void* src, void* dst, const float* bias, long long IMG, int H, int W, int C, int Hd,
                      int Wd, int oy, int ox, int unshuffle, int dtype_fp32, cudaStream_t stream);
int launch_strided_copy(const void* src, int src_fp32, void* dst, int dst_fp32, const long long* dims,
                        const long long* sstr, const long long* dstr, int accumulate, cudaStream_t stream);
// split-K reduction epilogues: ws = `splits` fp32 slices [P][N] (N = 4*Ch for the cell), added in split order
int launch_splitk_lstm_cell(const float* ws, int splits, long long P, int Ch, int cht, const float* bias,
                            const float* c_prev, float* c_next, void* h_next, cudaStream_t stream);
int launch_splitk_affine(const float* ws, int splits, long long P, int N, const float* scale, const float* shift, int relu,
                         void* y, int out_fp32, cudaStream_t stream);

// ---- conv_simt.cu ----
struct ConvSimtParams {
    const void* src0;
    const void* src1;
    const void* w;      // [taps][N][C0+C1], same element type as the sources
    const float* bias;  // [N] or nullptr
    void* dst0;
    void* dst1;
    int IMG, H, W;      // IMG = T*B images
    int C0, C1, N, ksize, pad;
    int split;          // columns [0,split) -> dst0, [split,N) -> dst1
    long long ld0, ld1;
    int relu;
    int out_fp32;       // 1: fp32 output, 0: output in the source element type
};
int launch_conv_simt(const ConvSimtParams& p, int dtype_fp32, cudaStream_t stream);

struct WgradSimtParams {
    const void* dz;
    const void* src;
    float* dw;          // [taps][Nz][ldk], accumulated into (caller zero-fills)
    int IMG, H, W;
    int Nz, Csrc, ksize, pad;
    long long ldk;
    int koff;
    long long m_per_block;
    long long split_stride;  // with more than one pixel split: dw is the split-K workspace, split z at dw + z * split_stride
};
int launch_wgrad_simt(WgradSimtParams p, int dtype_fp32, cudaStream_t stream);

}  // namespace b200
