// Parameters of the tcgen05 implicit-GEMM convolution (conv_tc.cu).
#pragma once
#include "common.cuh"

namespace b200 {

enum ConvEpilogue : int {
    EPI_STORE = 0,  // out = acc (+bias) (+relu) -> bf16 / fp32, optionally split over two tensors
    EPI_LSTM = 1,   // gate-interleaved N tile: sigma/tanh gate math + c/h update (unet.py:29-35)
    EPI_LSTM_BWD = 2,  // BPTT: data-gradient conv of dz_t -> [dx_t ; dh_{t-1}], the dh columns go straight
                       // into the gate-gradient math of step t-1 (autograd of unet.py:30-35) -> dz_{t-1}
};

struct ConvTcParams {
    // problem
    int T, B, H, W;   // T groups of B images of H x W pixels (NHWC)
    int C0, C1;       // channels of source 0 / source 1 (C1 == 0: single source)
    int N;            // GEMM N (output channels; 4*Ch for the LSTM epilogue)
    int ksize, pad;   // square filter size (odd) and padding
    int kc;           // channels per K block (bf16: 64 / 32 / 16; fp32 operands: 32 / 16 / 8 -- rows of 128 / 64 / 32 bytes)
    int in_fp32;      // 1: sources and packed weights are fp32 and the MMA is tcgen05 kind::tf32 (the "tf32" precision
                      // mode: fp32 storage, TF32 tensor-core products, fp32 accumulation); 0: bf16, kind::f16
    int state_fp32;   // EPI_LSTM with in_fp32: h_next / gates_out are fp32 tensors
    int wK;           // row length of the packed weights (0: C0 + C1)
    // M tiling
    int Wt, Ht, Bt;
    int tiles_w, tiles_h, tiles_b;
    int num_m_tiles, num_n_tiles;
    // EPI_STORE
    void* dst0;
    void* dst1;
    long long ld0, ld1;  // row strides (elements)
    int split;           // columns [0,split) -> dst0, [split,N) -> dst1
    int out_fp32;        // 0: bf16, 1: fp32
    int relu;
    int accumulate;      // fp32 only: dst += value
    const float* bias;   // [N] (packed order) or nullptr
    const float* scale;  // [N] or nullptr: out = acc * scale + bias (eval-mode BatchNorm folded into the conv)
    // split K (EPI_STORE, fp32 output, no bias / scale / relu): split z = blockIdx.z accumulates the k-blocks
    // [z * kb_split, (z + 1) * kb_split) of the (tap, channel chunk) loop and stores its partial sums at
    // dst0 + z * split_stride.  kb_split = 0: the whole K loop, one split (every other launch).
    int kb_split;
    long long split_stride;
    // fused 2x2 pixel shuffle (ConvTranspose2d k=2 s=2 as a GEMM, unet.py:90-97; bf16 output, dst0 only):
    // column n = tap * shuf_C + co of input pixel (img, h, w) goes to output pixel
    // (2h + tap/2 + shuf_oy, 2w + tap%2 + shuf_ox) of a [IMG][shuf_Hd][shuf_Wd][shuf_C] tensor; bias is [shuf_C]
    int shuf_C, shuf_Hd, shuf_Wd, shuf_oy, shuf_ox;
    // fused BatchNorm statistics (bf16 output only): per (t, column) sum and sum of squares of the
    // stored (bf16-rounded) outputs are added to stat_sum / stat_sumsq [T][N] (caller zeroes them)
    double* stat_sum;
    double* stat_sumsq;
    // EPI_LSTM  (Ch = N/4; packed column = (n_tile*4 + gate)*CHT + j)
    const float* c_prev;        // [P, Ch] fp32 or nullptr (zeros)
    float* c_next;              // [P, Ch] fp32
    __nv_bfloat16* h_next;      // [P, Ch] bf16
    __nv_bfloat16* gates_out;   // [P, 4, Ch] bf16 post-activation i,f,g,o or nullptr
    // timestep-persistent mode (EPI_LSTM): seq_T > 0 -> the kernel loops over seq_T steps; source 0 is
    // x_seq [T], source 1 is h_all [T+1] (slot t = h_{t-1}), c_prev/c_next/h_next/gates_out point at
    // slot 0 / slot 1 / slot 1 / step 0 of their sequence buffers
    int seq_T;
    int seq_have_h0;
    // EPI_LSTM_BWD (always timestep-persistent, t = seq_T-1 .. 0).  N = Cin + Ch, source 0 = dz_all.
    int bwd_Cin, bwd_Ch;
    int bwd_alternate;               // set by the launcher: N tiles split evenly into a dx half and a dh half
    long long bwd_P;                 // pixels per timestep (B*H*W)
    const __nv_bfloat16* bwd_gates;  // [T][P][4][Ch] activated i,f,g,o
    const float* bwd_c_all;          // [T+1][P][Ch]
    const __nv_bfloat16* bwd_dh_seq; // [T][P][Ch] upstream dL/dh_t or nullptr
    float* bwd_dc;                   // [2][P][Ch] ping-pong: slot (t & 1) holds dL/dc_{t-1} produced at step t
    __nv_bfloat16* bwd_dz_all;       // [T][P][4*Ch] (i|f|g|o): slot T-1 is filled by the caller, the rest here
    __nv_bfloat16* bwd_dx_seq;       // [T][P][Cin] or nullptr
    __nv_bfloat16* bwd_dh0;          // [P][Ch] dL/dh_{-1} or nullptr
    unsigned* sync_ctr;
    int* err_flag;
};

// Launches the kernel for one problem.  All pointers are device pointers; maps are built per call.
int launch_conv_tc(const void* src0, const void* src1, const void* wpacked, ConvTcParams p, int epi,
                   cudaStream_t stream);

// Split-K form of launch_conv_tc (1-CTA kernel, EPI_STORE): `splits` K ranges of whole k-blocks, one per
// blockIdx.z, each storing fp32 partial sums [P][N] (P = T*B*H*W) to ws + z * P * N.  Returns the number of
// splits actually launched (every split gets at least one k-block) in *splits_out.
int launch_conv_tc_splitk(const void* src0, const void* src1, const void* wpacked, ConvTcParams p, int splits,
                          float* ws, int* splits_out, cudaStream_t stream);
// k-blocks of the implicit GEMM over [src0 ; src1] (taps x channel chunks), as launch_conv_tc will tile it.
int conv_tc_num_kb(int C0, int C1, int ksize);

// Whole-sequence forward of one ConvLSTM layer in ONE cooperative launch (see ConvTcParams::seq_T).
int launch_convlstm_seq_tc(const void* x_seq, const void* h_all, const void* wpacked, ConvTcParams p,
                           cudaStream_t stream);

// Whole-sequence BPTT data path of one ConvLSTM layer in ONE cooperative launch (EPI_LSTM_BWD).
int launch_convlstm_seq_bwd_tc(const void* wd_packed, ConvTcParams p, cudaStream_t stream);

// conv_halo.cu: 3x3 convolution with the activation tile loaded once per output tile (narrow layers).
bool conv_halo_supported(int IMG, int H, int W, int C0, int C1, int N, int ksize);
int launch_conv_halo(const void* src0, const void* src1, const void* wpacked, int IMG, int H, int W, int C0, int C1,
                     int N, const float* bias, void* dst0, long long ld0, int split, void* dst1, long long ld1,
                     int out_fp32, int relu, int accumulate, double* stat_sum, double* stat_sumsq, int imgs_per_t,
                     const float* scale, cudaStream_t stream);

// conv_tc2.cu: the same convolution on a CTA pair (tcgen05 cta_group::2, M = 256 per pair), plain store epilogue.
bool conv_tc2_supported(const ConvTcParams& p);
int launch_conv_tc2(const void* src0, const void* src1, const void* wpacked, ConvTcParams p, int epi, cudaStream_t stream);

// Picks BLOCK_N for a given GEMM N (multiple of 16).  LSTM epilogue needs N % 64 == 0.
int pick_block_n(int N, int epi);

}  // namespace b200
