// C-ABI entry points (declared in include/b200_convlstm.h): argument checks + kernel launches.
// Nothing here allocates device memory; no exception crosses the boundary.
#include "../../include/b200_convlstm.h"
#include "common.cuh"
#include "conv_tc.cuh"
#include "pointwise.cuh"

#include <stdlib.h>

using namespace b200;

namespace b200 {
int launch_wgrad_tc(const void* dz, int Nz, const void* src, int Csrc, int T, int B, int H, int W,
                    int ksize, float* dw, long long ldk, int koff, cudaStream_t stream, int in_fp32 = 0);
// wgrad_halo.cu: 64-channel 3x3 layers, source tile loaded once per pixel block
bool wgrad_halo_supported(int Nz, int Csrc, int B, int H, int W, int ksize);
int launch_wgrad_halo(const void* dz, int Nz, const void* src, int Csrc, int T, int B, int H, int W, float* dw,
                      long long ldk, int koff, cudaStream_t stream);
// wgrad_tc2.cu: narrow sources on a CTA pair (tcgen05 cta_group::2)
bool wgrad_tc2_supported(int Nz, int Csrc, int ksize);
int launch_wgrad_tc2(const void* dz, int Nz, const void* src, int Csrc, int T, int B, int H, int W, int ksize, float* dw,
                     long long ldk, int koff, cudaStream_t stream);
}

extern "C" int b200_device_error(void) {
    int* f = device_error_flag();
    if (!f) return 0;
    // the flag lives in pinned host memory mapped into the device: readable even after a trap
    const int v = *static_cast<volatile int*>(f);
    if (v != 0) *static_cast<volatile int*>(f) = 0;
    return v;
}

extern "C" int b200_tmap_cache_stats(long long* hits, long long* misses) {
    unsigned long long h = 0, m = 0;
    tmap_cache_stats(&h, &m);
    if (hits) *hits = static_cast<long long>(h);
    if (misses) *misses = static_cast<long long>(m);
    return B200_OK;
}

extern "C" int b200_conv_tc_supported(int B, int H, int W, int C0, int C1, int N, int lstm) {
    MTile mt;
    if (!plan_mtile(B, H, W, 128, &mt)) return 0;
    if (C0 <= 0 || C0 % 16 != 0 || C1 % 16 != 0) return 0;
    if (pick_block_n(N, lstm ? EPI_LSTM : EPI_STORE) == 0) return 0;
    return 1;
}

static int conv_tc_fwd_impl(const void* src0, int C0, const void* src1, int C1, int T, int B, int H,
                           int W, const void* wpacked, const float* bias, int N, int ksize,
                           void* dst0, long long ld0, int split, void* dst1, long long ld1,
                           int out_fp32, int relu, int accumulate, double* stat_sum, double* stat_sumsq,
                           const float* scale, void* stream) {
    if (!src0 || !wpacked || !dst0 || T <= 0 || N <= 0 || (ksize & 1) == 0) {
        set_last_error("b200_conv_tc_fwd: bad arguments");
        return B200_ERR_ARG;
    }
    if (split < 0 || split > N || (split < N && !dst1) || split % 16 != 0 || ld0 % 8 != 0 ||
        (split < N && ld1 % 8 != 0)) {
        set_last_error("b200_conv_tc_fwd: bad split/ld (split=%d N=%d ld0=%lld ld1=%lld)", split, N, ld0,
                       ld1);
        return B200_ERR_ARG;
    }
    if (accumulate && !out_fp32) {
        set_last_error("b200_conv_tc_fwd: accumulate requires fp32 output");
        return B200_ERR_ARG;
    }
    // narrow layers are bound by the L2 -> smem fill rate of the per-tap activation boxes: use the halo
    // kernel (activation tile loaded once per output tile).  B200_CONV_HALO=0 disables, =2 forces it
    // for every shape it supports.
    static const int halo_mode = [] {
        const char* e = getenv("B200_CONV_HALO");
        return e ? atoi(e) : 1;
    }();
    // CTA-pair kernel (conv_tc2.cu, tcgen05 cta_group::2).  B200_CONV_2CTA: 0 = never, 1 (default) = everywhere
    // except the N <= 64 layers the halo kernel takes (measured, profiles/r01_conv_2cta_ab.txt: 1.04-1.16x on the
    // N >= 128 shapes, 0.78x at K64->N64 where loading the activation tile once matters more), 2 = always.
    static const int pair_mode = [] {
        const char* e = getenv("B200_CONV_2CTA");
        return e ? atoi(e) : 1;
    }();
    ConvTcParams pp = {};
    pp.T = T; pp.B = B; pp.H = H; pp.W = W;
    pp.C0 = C0; pp.C1 = C1; pp.N = N; pp.ksize = ksize;
    pp.dst0 = dst0; pp.dst1 = dst1; pp.ld0 = ld0; pp.ld1 = ld1; pp.split = split;
    pp.out_fp32 = out_fp32; pp.relu = relu; pp.accumulate = accumulate; pp.bias = bias;
    pp.stat_sum = stat_sum; pp.stat_sumsq = stat_sumsq; pp.scale = scale;
    const bool halo_takes = halo_mode > 0 && ksize == 3 && (N <= 128 || halo_mode >= 2) &&
                            conv_halo_supported(T * B, H, W, C0, C1, N, ksize);
    if (pair_mode > 0 && conv_tc2_supported(pp) && (pair_mode >= 2 || !(halo_takes && N <= 64)))
        return launch_conv_tc2(src0, src1, wpacked, pp, EPI_STORE, static_cast<cudaStream_t>(stream));
    if (halo_mode > 0 && ksize == 3 && (N <= 128 || halo_mode >= 2) &&
        conv_halo_supported(T * B, H, W, C0, C1, N, ksize))
        return launch_conv_halo(src0, src1, wpacked, T * B, H, W, C0, C1, N, bias, dst0, ld0, split, dst1, ld1,
                                out_fp32, relu, accumulate, stat_sum, stat_sumsq, B, scale,
                                static_cast<cudaStream_t>(stream));
    ConvTcParams p = {};
    p.T = T; p.B = B; p.H = H; p.W = W;
    p.C0 = C0; p.C1 = C1; p.N = N; p.ksize = ksize;
    p.dst0 = dst0; p.dst1 = dst1; p.ld0 = ld0; p.ld1 = ld1; p.split = split;
    p.out_fp32 = out_fp32; p.relu = relu; p.accumulate = accumulate; p.bias = bias;
    p.stat_sum = stat_sum; p.stat_sumsq = stat_sumsq; p.scale = scale;
    return launch_conv_tc(src0, src1, wpacked, p, EPI_STORE, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_conv_tc_fwd(const void* src0, int C0, const void* src1, int C1, int T, int B, int H,
                                int W, const void* wpacked, const float* bias, int N, int ksize,
                                void* dst0, long long ld0, int split, void* dst1, long long ld1,
                                int out_fp32, int relu, int accumulate, void* stream) {
    return conv_tc_fwd_impl(src0, C0, src1, C1, T, B, H, W, wpacked, bias, N, ksize, dst0, ld0, split, dst1, ld1,
                            out_fp32, relu, accumulate, nullptr, nullptr, nullptr, stream);
}

extern "C" int b200_conv_bnstats_tc_fwd(const void* src0, int C0, const void* src1, int C1, int T, int B, int H,
                                        int W, const void* wpacked, const float* bias, int N, int ksize, void* dst,
                                        double* stat_sum, double* stat_sumsq, void* stream) {
    if (!stat_sum || !stat_sumsq) {
        set_last_error("b200_conv_bnstats_tc_fwd: statistics buffers are required");
        return B200_ERR_ARG;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    B200_CUDA_CHECK(cudaMemsetAsync(stat_sum, 0, sizeof(double) * T * N, st));
    B200_CUDA_CHECK(cudaMemsetAsync(stat_sumsq, 0, sizeof(double) * T * N, st));
    return conv_tc_fwd_impl(src0, C0, src1, C1, T, B, H, W, wpacked, bias, N, ksize, dst, N, N, nullptr, 0,
                            /*out_fp32=*/0, /*relu=*/0, /*accumulate=*/0, stat_sum, stat_sumsq, nullptr, stream);
}

extern "C" int b200_conv_affine_relu_tc_fwd(const void* src0, int C0, const void* src1, int C1, int T, int B, int H,
                                           int W, const void* wpacked, const float* scale, const float* shift, int N,
                                           int ksize, void* dst, int relu, void* stream) {
    if (!scale || !shift) {
        set_last_error("b200_conv_affine_relu_tc_fwd: scale and shift are required");
        return B200_ERR_ARG;
    }
    return conv_tc_fwd_impl(src0, C0, src1, C1, T, B, H, W, wpacked, shift, N, ksize, dst, N, N, nullptr, 0,
                            /*out_fp32=*/0, relu, /*accumulate=*/0, nullptr, nullptr, scale, stream);
}

extern "C" int b200_convT2x2_tc_fwd(const void* x, int Cin, int T, int B, int H, int W, const void* wpacked,
                                    const float* bias, int Cout, void* y, int Hd, int Wd, void* stream) {
    if (!x || !wpacked || !y || Cin <= 0 || Cout <= 0 || Cout % 16 != 0 || Hd < 2 * H || Wd < 2 * W) {
        set_last_error("b200_convT2x2_tc_fwd: bad arguments (Cout must be a multiple of 16, Hd >= 2H, Wd >= 2W)");
        return B200_ERR_ARG;
    }
    ConvTcParams p = {};
    p.T = T; p.B = B; p.H = H; p.W = W;
    p.C0 = Cin; p.C1 = 0; p.N = 4 * Cout; p.ksize = 1;
    p.dst0 = y; p.ld0 = Cout; p.split = 4 * Cout;
    p.bias = bias;
    p.shuf_C = Cout; p.shuf_Hd = Hd; p.shuf_Wd = Wd;
    p.shuf_oy = (Hd - 2 * H) / 2; p.shuf_ox = (Wd - 2 * W) / 2;  // centred like F.pad (unet.py:95-97)
    // CTA-pair kernel by default (low-K GEMM: 8 epilogue warps per CTA drain the tile); B200_CONV_2CTA=0 -> 1 CTA
    static const int pair_mode = [] {
        const char* e = getenv("B200_CONV_2CTA");
        return e ? atoi(e) : 1;
    }();
    if (pair_mode > 0 && conv_tc2_supported(p))
        return launch_conv_tc2(x, nullptr, wpacked, p, EPI_STORE, static_cast<cudaStream_t>(stream));
    return launch_conv_tc(x, nullptr, wpacked, p, EPI_STORE, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_convlstm_cell_fwd_tc(const void* x, int Cin, const void* h_prev, int Ch, int B, int H,
                                         int W, const void* wpacked, const float* bias_packed,
                                         const float* c_prev, float* c_next, void* h_next,
                                         void* gates_out, int ksize, void* stream) {
    if (!x || !wpacked || !c_next || !h_next || Ch <= 0 || Cin <= 0) {
        set_last_error("b200_convlstm_cell_fwd_tc: bad arguments");
        return B200_ERR_ARG;
    }
    ConvTcParams p = {};
    p.T = 1; p.B = B; p.H = H; p.W = W;
    p.C0 = Cin; p.C1 = h_prev ? Ch : 0;
    p.N = 4 * Ch; p.ksize = ksize;
    p.wK = Cin + Ch;
    p.bias = bias_packed;
    p.c_prev = c_prev; p.c_next = c_next;
    p.h_next = static_cast<__nv_bfloat16*>(h_next);
    p.gates_out = static_cast<__nv_bfloat16*>(gates_out);
    // With h_prev == NULL (zero initial state, unet.py:23-25) the h half of K is skipped; the
    // packed weight rows still span Cin+Ch columns, so the weight map must keep the full K.
    return launch_conv_tc(x, h_prev, wpacked, p, EPI_LSTM, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_convlstm_seq_fwd_tc(const void* x_seq, int Cin, void* h_all, int Ch, int T, int B, int H, int W,
                                        const void* wpacked, const float* bias_packed, float* c_all, void* gates,
                                        int have_h0, int ksize, void* stream) {
    if (!x_seq || !h_all || !wpacked || !c_all || Ch <= 0 || Cin <= 0 || T <= 0) {
        set_last_error("b200_convlstm_seq_fwd_tc: bad arguments");
        return B200_ERR_ARG;
    }
    const long long slot = static_cast<long long>(B) * H * W * Ch;
    ConvTcParams p = {};
    p.T = 1; p.B = B; p.H = H; p.W = W;
    p.C0 = Cin; p.C1 = Ch;
    p.N = 4 * Ch; p.ksize = ksize;
    p.wK = Cin + Ch;
    p.bias = bias_packed;
    p.c_prev = c_all;
    p.c_next = c_all + slot;
    p.h_next = static_cast<__nv_bfloat16*>(h_all) + slot;
    p.gates_out = static_cast<__nv_bfloat16*>(gates);
    p.seq_T = T;
    p.seq_have_h0 = have_h0;
    // B200_LSTM_2CTA (default 1): the CTA-pair kernel (conv_tc2.cu, tcgen05 cta_group::2); 0: the 1-CTA kernel
    static const int pair_mode = [] {
        const char* e = getenv("B200_LSTM_2CTA");
        return e ? atoi(e) : 1;
    }();
    if (pair_mode > 0) return launch_conv_tc2(x_seq, h_all, wpacked, p, EPI_LSTM, static_cast<cudaStream_t>(stream));
    return launch_convlstm_seq_tc(x_seq, h_all, wpacked, p, static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------------------
// Split K for single-frame GEMMs with few M tiles (streaming inference, unet_convlstm_b200/stream.py)
// ------------------------------------------------------------------------------------------------
// Rule (b200_splitk_splits): split only when the 1-CTA tiling has at most SPLITK_MAX_M_TILES M tiles and all its
// tiles together occupy at most 1 / SPLITK_SM_SHARE of the SMs; then S = SMs / tiles (about one wave of tiles x S
// CTAs), capped so that every split keeps at least SPLITK_MIN_KB k-blocks (one k-block = one tap x 64 channels).
// Measured on a B200 at 1000 W (tools/bench_infer.py --stream, profiles/stream_infer_b200.txt): the split cell and
// folded convs of the 4x4 / 8x8 / 16x16 levels at B = 1 and 8 run 1.3-2.1x faster than the unsplit launch; below
// ~16 k-blocks per split the cell loses again (8x8 Ch 512, B = 1: S = 8 1.61x, S = 16 1.39x; 16x16 Ch 256: S = 4
// 1.30x, S = 8 1.20x; at B = 8 S = 16 falls to 0.27-0.60x), so 16 is the minimum -- within ~5 % of the best S at
// every measured shape.  Shapes with more M tiles (16x16 at B = 8, every level at B = 64) were not measured split
// and stay unsplit.
static constexpr int SPLITK_MAX_M_TILES = 4;
static constexpr int SPLITK_SM_SHARE = 4;
static constexpr int SPLITK_MIN_KB = 16;

extern "C" int b200_splitk_splits(int B, int H, int W, int C0, int C1, int N, int ksize) {
    MTile mt;
    if (!plan_mtile(B, H, W, 128, &mt) || C0 <= 0 || C0 % 16 != 0 || C1 % 16 != 0 || (ksize & 1) == 0) return 1;
    const int block_n = pick_block_n(N, EPI_STORE);
    if (block_n == 0) return 1;
    const int m_tiles = mt.tiles_w * mt.tiles_h * mt.tiles_b;
    const int tiles = m_tiles * ((N + block_n - 1) / block_n);
    if (m_tiles > SPLITK_MAX_M_TILES || tiles * SPLITK_SM_SHARE > num_sms()) return 1;
    int s = num_sms() / tiles;
    const int by_k = conv_tc_num_kb(C0, C1, ksize) / SPLITK_MIN_KB;
    if (s > by_k) s = by_k;
    return s >= 2 ? s : 1;
}

static float* splitk_ws_or_error(const char* who, cudaStream_t st, int splits, long long P, int N) {
    float* ws = splitk_workspace(st, static_cast<size_t>(splits) * P * N);
    if (!ws)
        set_last_error("%s: no split-K workspace (cudaMalloc failed, or it would have to grow during a CUDA-graph "
                       "capture: run the same shape once on this stream before capturing)", who);
    return ws;
}

extern "C" int b200_convlstm_cell_fwd_splitk_tc(const void* x, int Cin, const void* h_prev, int Ch, int B, int H, int W,
                                                const void* wpacked, const float* bias_packed, const float* c_prev,
                                                float* c_next, void* h_next, int splits, int ksize, void* stream) {
    if (!x || !wpacked || !c_next || !h_next || Ch <= 0 || Cin <= 0 || splits < 1 || (ksize & 1) == 0) {
        set_last_error("b200_convlstm_cell_fwd_splitk_tc: bad arguments");
        return B200_ERR_ARG;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ConvTcParams p = {};
    p.T = 1; p.B = B; p.H = H; p.W = W;
    p.C0 = Cin; p.C1 = h_prev ? Ch : 0;   // zero state: the h half of K is skipped, as in the unsplit cell
    p.N = 4 * Ch; p.ksize = ksize;
    p.wK = Cin + Ch;
    const long long P = static_cast<long long>(B) * H * W;
    float* ws = splitk_ws_or_error("b200_convlstm_cell_fwd_splitk_tc", st, splits, P, p.N);
    if (!ws) return B200_ERR_CUDA;
    int S = 0;
    int rc = launch_conv_tc_splitk(x, h_prev, wpacked, p, splits, ws, &S, st);
    if (rc != B200_OK) return rc;
    const int cht = Ch % 64 == 0 ? 64 : (Ch % 32 == 0 ? 32 : 16);   // the gate interleave of b200_pack_weight
    return launch_splitk_lstm_cell(ws, S, P, Ch, cht, bias_packed, c_prev, c_next, h_next, st);
}

extern "C" int b200_conv_affine_relu_splitk_tc(const void* src0, int C0, const void* src1, int C1, int B, int H, int W,
                                               const void* wpacked, const float* scale, const float* shift, int N,
                                               int ksize, void* dst, int out_fp32, int relu, int splits, void* stream) {
    if (!src0 || !wpacked || !dst || N <= 0 || splits < 1 || (ksize & 1) == 0 || (C1 > 0 && !src1)) {
        set_last_error("b200_conv_affine_relu_splitk_tc: bad arguments");
        return B200_ERR_ARG;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ConvTcParams p = {};
    p.T = 1; p.B = B; p.H = H; p.W = W;
    p.C0 = C0; p.C1 = C1; p.N = N; p.ksize = ksize;
    const long long P = static_cast<long long>(B) * H * W;
    float* ws = splitk_ws_or_error("b200_conv_affine_relu_splitk_tc", st, splits, P, N);
    if (!ws) return B200_ERR_CUDA;
    int S = 0;
    int rc = launch_conv_tc_splitk(src0, src1, wpacked, p, splits, ws, &S, st);
    if (rc != B200_OK) return rc;
    return launch_splitk_affine(ws, S, P, N, scale, shift, relu, dst, out_fp32, st);
}

// ------------------------------------------------------------------------------------------------
// "tf32" precision mode: fp32 tensors, tcgen05 kind::tf32 products, fp32 accumulation
// ------------------------------------------------------------------------------------------------
extern "C" int b200_conv_tf32_supported(int B, int H, int W, int C0, int C1, int N, int lstm) {
    MTile mt;
    if (!plan_mtile(B, H, W, 128, &mt)) return 0;
    if (C0 <= 0 || C0 % 8 != 0 || C1 % 8 != 0) return 0;
    if (pick_block_n(N, lstm ? EPI_LSTM : EPI_STORE) == 0) return 0;
    return 1;
}

extern "C" int b200_conv_tf32_fwd(const float* src0, int C0, const float* src1, int C1, int T, int B, int H, int W,
                                  const float* wpacked, const float* bias, int N, int ksize, float* dst0, long long ld0,
                                  int split, float* dst1, long long ld1, int relu, int accumulate, void* stream) {
    if (!src0 || !wpacked || !dst0 || T <= 0 || N <= 0 || (ksize & 1) == 0) {
        set_last_error("b200_conv_tf32_fwd: bad arguments");
        return B200_ERR_ARG;
    }
    if (split < 0 || split > N || (split < N && !dst1) || split % 16 != 0 || ld0 % 4 != 0 || (split < N && ld1 % 4 != 0)) {
        set_last_error("b200_conv_tf32_fwd: bad split/ld (split=%d N=%d ld0=%lld ld1=%lld)", split, N, ld0, ld1);
        return B200_ERR_ARG;
    }
    ConvTcParams p = {};
    p.T = T; p.B = B; p.H = H; p.W = W;
    p.C0 = C0; p.C1 = C1; p.N = N; p.ksize = ksize;
    p.dst0 = dst0; p.dst1 = dst1; p.ld0 = ld0; p.ld1 = ld1;
    p.split = split;
    p.out_fp32 = 1; p.relu = relu; p.accumulate = accumulate;
    p.bias = bias;
    p.in_fp32 = 1;
    return launch_conv_tc(src0, src1, wpacked, p, EPI_STORE, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_convlstm_cell_fwd_tf32(const float* x, int Cin, const float* h_prev, int Ch, int B, int H, int W,
                                           const float* wpacked, const float* bias_packed, const float* c_prev,
                                           float* c_next, float* h_next, float* gates_out, int ksize, void* stream) {
    if (!x || !wpacked || !c_next || !h_next || Ch <= 0 || Cin <= 0) {
        set_last_error("b200_convlstm_cell_fwd_tf32: bad arguments");
        return B200_ERR_ARG;
    }
    ConvTcParams p = {};
    p.T = 1; p.B = B; p.H = H; p.W = W;
    p.C0 = Cin; p.C1 = h_prev ? Ch : 0;
    p.N = 4 * Ch; p.ksize = ksize;
    p.wK = Cin + Ch;
    p.bias = bias_packed;
    p.c_prev = c_prev; p.c_next = c_next;
    p.h_next = reinterpret_cast<__nv_bfloat16*>(h_next);       // fp32 tensors: see ConvTcParams::state_fp32
    p.gates_out = reinterpret_cast<__nv_bfloat16*>(gates_out);
    p.in_fp32 = 1; p.state_fp32 = 1;
    return launch_conv_tc(x, h_prev, wpacked, p, EPI_LSTM, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_convlstm_gates_recompute_tc(const void* x_seq, int Cin, const void* h_all, int Ch, int T, int B, int H,
                                                int W, const void* wpacked, const float* bias_packed, const float* c_all,
                                                void* gates_out, int ksize, void* stream) {
    if (!x_seq || !h_all || !wpacked || !c_all || !gates_out || Ch <= 0 || Cin <= 0 || T <= 0) {
        set_last_error("b200_convlstm_gates_recompute_tc: bad arguments");
        return B200_ERR_ARG;
    }
    // all T steps at once: with h_{t-1} and c_{t-1} stored, the gate pre-activations of different steps are independent
    ConvTcParams p = {};
    p.T = T; p.B = B; p.H = H; p.W = W;
    p.C0 = Cin; p.C1 = Ch;
    p.N = 4 * Ch; p.ksize = ksize;
    p.wK = Cin + Ch;
    p.bias = bias_packed;
    p.c_prev = c_all;            // slot t = c_{t-1}
    p.c_next = nullptr;          // state outputs are not rewritten
    p.h_next = nullptr;
    p.gates_out = static_cast<__nv_bfloat16*>(gates_out);
    return launch_conv_tc2(x_seq, h_all, wpacked, p, EPI_LSTM, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_convlstm_seq_bwd_tc(void* dz_all, const void* wd_packed, const void* gates, const float* c_all,
                                        const void* dh_seq, float* dc_buf, void* dx_seq, void* dh0, int Cin, int Ch,
                                        int T, int B, int H, int W, int have_h0, int ksize, void* stream) {
    if (!dz_all || !wd_packed || !gates || !c_all || !dc_buf || Cin <= 0 || Ch <= 0 || T <= 0 || (ksize & 1) == 0) {
        set_last_error("b200_convlstm_seq_bwd_tc: bad arguments");
        return B200_ERR_ARG;
    }
    ConvTcParams p = {};
    p.T = 1; p.B = B; p.H = H; p.W = W;
    p.C0 = 4 * Ch; p.C1 = 0;
    p.N = Cin + Ch; p.ksize = ksize;
    p.seq_T = T;
    p.seq_have_h0 = have_h0;
    p.bwd_Cin = Cin; p.bwd_Ch = Ch;
    p.bwd_P = static_cast<long long>(B) * H * W;
    p.bwd_gates = static_cast<const __nv_bfloat16*>(gates);
    p.bwd_c_all = c_all;
    p.bwd_dh_seq = static_cast<const __nv_bfloat16*>(dh_seq);
    p.bwd_dc = dc_buf;
    p.bwd_dz_all = static_cast<__nv_bfloat16*>(dz_all);
    p.bwd_dx_seq = static_cast<__nv_bfloat16*>(dx_seq);
    p.bwd_dh0 = static_cast<__nv_bfloat16*>(dh0);
    return launch_convlstm_seq_bwd_tc(wd_packed, p, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_wgrad_tc(const void* dz, int Nz, const void* src, int Csrc, int T, int B, int H, int W,
                             int ksize, float* dw, long long ldk, int koff, void* stream) {
    if (!dz || !src || !dw || Nz <= 0 || Csrc <= 0 || (ksize & 1) == 0 || koff < 0 || koff + Csrc > ldk) {
        set_last_error("b200_wgrad_tc: bad arguments");
        return B200_ERR_ARG;
    }
    // B200_WGRAD_HALO (default 1): the halo kernel (wgrad_halo.cu) for the 64-channel 3x3 layers -- source tile
    // loaded once per pixel block, taps as shifted MN-major descriptors: 820 -> 1090 TFLOP/s at Nz = 64, 64x64
    static const int halo_mode = [] {
        const char* e = getenv("B200_WGRAD_HALO");
        return e ? atoi(e) : 1;
    }();
    if (halo_mode > 0 && (ldk % 4) == 0 && (koff % 4) == 0 && wgrad_halo_supported(Nz, Csrc, B, H, W, ksize))
        return launch_wgrad_halo(dz, Nz, src, Csrc, T, B, H, W, dw, ldk, koff, static_cast<cudaStream_t>(stream));
    // B200_WGRAD_2CTA: the CTA-pair kernel (wgrad_tc2.cu).  0 = never, 1 (default) = where it measured faster or
    // equal (profiles/r01_wgrad_2cta_ab.txt): every wide-source shape it supports (1.00-1.19x) and 64-channel sources
    // with dz >= 128 channels (912 -> 1100 TFLOP/s; at Nz = 64 both kernels sit at the L2 -> SM fill limit of the
    // nine tap-shifted source boxes: 778 vs 762), 2 = wherever it can run.
    static const int pair_mode = [] {
        const char* e = getenv("B200_WGRAD_2CTA");
        return e ? atoi(e) : 1;
    }();
    if (pair_mode > 0 && (pair_mode >= 2 || Csrc > 64 || (Csrc == 64 && Nz >= 128)) && (ldk % 4) == 0 && (koff % 4) == 0 &&
        wgrad_tc2_supported(Nz, Csrc, ksize))
        return launch_wgrad_tc2(dz, Nz, src, Csrc, T, B, H, W, ksize, dw, ldk, koff, static_cast<cudaStream_t>(stream));
    return launch_wgrad_tc(dz, Nz, src, Csrc, T, B, H, W, ksize, dw, ldk, koff,
                           static_cast<cudaStream_t>(stream));
}

// "tf32" precision mode: the weight gradient from fp32 dz / src on tcgen05 kind::tf32 (MN-major operands, 32 pixels per
// pipeline stage); 1-CTA kernel only
extern "C" int b200_wgrad_tf32_supported(int B, int H, int W, int Nz, int Csrc) {
    MTile mt;
    if (!plan_mtile(B, H, W, 32, &mt)) return 0;
    if (Nz <= 0 || Csrc <= 0 || Nz % 32 != 0 || Csrc % 32 != 0) return 0;   // 128-byte pixel rows (see wgrad_tc.cu)
    return 1;
}

extern "C" int b200_wgrad_tf32(const float* dz, int Nz, const float* src, int Csrc, int T, int B, int H, int W, int ksize,
                               float* dw, long long ldk, int koff, void* stream) {
    if (!dz || !src || !dw || Nz <= 0 || Csrc <= 0 || (ksize & 1) == 0 || koff < 0 || koff + Csrc > ldk) {
        set_last_error("b200_wgrad_tf32: bad arguments");
        return B200_ERR_ARG;
    }
    return launch_wgrad_tc(dz, Nz, src, Csrc, T, B, H, W, ksize, dw, ldk, koff, static_cast<cudaStream_t>(stream), 1);
}

extern "C" int b200_wgrad_tc_supported(int B, int H, int W, int Nz, int Csrc) {
    MTile mt;
    if (!plan_mtile(B, H, W, 64, &mt)) return 0;
    if (Nz <= 0 || Csrc <= 0 || Nz % 16 != 0 || Csrc % 16 != 0) return 0;
    return 1;
}

// ------------------------------------------------------------------------------------------------
// generic SIMT convolutions (fp32 check mode; shapes the tensor-core path cannot tile)
// ------------------------------------------------------------------------------------------------
extern "C" int b200_conv_simt_fwd(const void* src0, int C0, const void* src1, int C1, int IMG, int H, int W,
                                  const void* w, const float* bias, int N, int ksize, void* dst0, long long ld0,
                                  int split, void* dst1, long long ld1, int dtype_fp32, int out_fp32, int relu,
                                  void* stream) {
    if (!src0 || !w || !dst0 || IMG <= 0 || H <= 0 || W <= 0 || C0 <= 0 || C1 < 0 || N <= 0 || (ksize & 1) == 0 ||
        (C1 > 0 && !src1) || split < 0 || split > N || (split < N && !dst1)) {
        set_last_error("b200_conv_simt_fwd: bad arguments");
        return B200_ERR_ARG;
    }
    ConvSimtParams p = {};
    p.src0 = src0; p.src1 = src1; p.w = w; p.bias = bias; p.dst0 = dst0; p.dst1 = dst1;
    p.IMG = IMG; p.H = H; p.W = W; p.C0 = C0; p.C1 = C1; p.N = N; p.ksize = ksize; p.pad = ksize / 2;
    p.split = split; p.ld0 = ld0; p.ld1 = ld1; p.relu = relu; p.out_fp32 = out_fp32 || dtype_fp32;
    return launch_conv_simt(p, dtype_fp32, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_wgrad_simt(const void* dz, int Nz, const void* src, int Csrc, int IMG, int H, int W, int ksize,
                               float* dw, long long ldk, int koff, int dtype_fp32, void* stream) {
    if (!dz || !src || !dw || Nz <= 0 || Csrc <= 0 || (ksize & 1) == 0 || koff < 0 || koff + Csrc > ldk) {
        set_last_error("b200_wgrad_simt: bad arguments");
        return B200_ERR_ARG;
    }
    WgradSimtParams p = {};
    p.dz = dz; p.src = src; p.dw = dw; p.IMG = IMG; p.H = H; p.W = W; p.Nz = Nz; p.Csrc = Csrc;
    p.ksize = ksize; p.pad = ksize / 2; p.ldk = ldk; p.koff = koff;
    return launch_wgrad_simt(p, dtype_fp32, static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------------------
// BatchNorm + ReLU
// ------------------------------------------------------------------------------------------------
#define B200_REQUIRE(cond, name)                          \
    do {                                                  \
        if (!(cond)) {                                    \
            set_last_error(name ": bad arguments");       \
            return B200_ERR_ARG;                          \
        }                                                 \
    } while (0)

extern "C" int b200_bn_stats(const void* x, int T, long long P, int C, int dtype_fp32, double* sum, double* sumsq,
                             void* stream) {
    B200_REQUIRE(x && sum && sumsq && T > 0 && P > 0 && C > 0, "b200_bn_stats");
    return launch_bn_stats(x, T, P, C, dtype_fp32, sum, sumsq, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_bn_finalize(const double* sum, const double* sumsq, int T, long long n, int C,
                                const float* gamma, const float* beta, float* running_mean, float* running_var,
                                float eps, float momentum, int training, float* mean, float* rstd, float* scale,
                                float* shift, void* stream) {
    B200_REQUIRE(gamma && beta && running_mean && running_var && mean && rstd && scale && shift && C > 0 &&
                     (!training || (sum && sumsq && T > 0 && n > 0)),
                 "b200_bn_finalize");
    return launch_bn_finalize(sum, sumsq, T, n, C, gamma, beta, running_mean, running_var, eps, momentum, training,
                              mean, rstd, scale, shift, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_bn_relu_apply(const void* x, const float* scale, const float* shift, void* y, int T, long long P,
                                  int C, int tstride, int relu, int dtype_fp32, void* stream) {
    B200_REQUIRE(x && scale && shift && y && T > 0 && P > 0 && C > 0, "b200_bn_relu_apply");
    return launch_bn_relu_apply(x, scale, shift, y, T, P, C, tstride, relu, dtype_fp32,
                                static_cast<cudaStream_t>(stream));
}

extern "C" int b200_bn_relu_bwd_reduce(const void* x, const void* dy, const float* mean, const float* rstd,
                                       const float* scale, const float* shift, int T, long long P, int C,
                                       int tstride, int dtype_fp32, double* sum_g, double* sum_gx, void* stream) {
    B200_REQUIRE(x && dy && mean && rstd && scale && shift && sum_g && sum_gx && T > 0 && P > 0 && C > 0,
                 "b200_bn_relu_bwd_reduce");
    return launch_bn_relu_bwd_reduce(x, dy, mean, rstd, scale, shift, T, P, C, tstride, dtype_fp32, sum_g, sum_gx,
                                     static_cast<cudaStream_t>(stream));
}

extern "C" int b200_bn_bwd_finalize(const double* sum_g, const double* sum_gx, int T, long long n, int C,
                                    int training, const float* scale, float* coef1, float* coef2, float* dgamma,
                                    float* dbeta, float* dconv_bias, int accumulate, void* stream) {
    B200_REQUIRE(sum_g && sum_gx && scale && coef1 && coef2 && dgamma && dbeta && T > 0 && n > 0 && C > 0,
                 "b200_bn_bwd_finalize");
    return launch_bn_bwd_finalize(sum_g, sum_gx, T, n, C, training, scale, coef1, coef2, dgamma, dbeta, dconv_bias,
                                  accumulate, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_bn_relu_bwd_apply(const void* x, const void* dy, const float* mean, const float* rstd,
                                      const float* scale, const float* shift, const float* coef1,
                                      const float* coef2, void* dx, int T, long long P, int C, int tstride,
                                      int dtype_fp32, void* stream) {
    B200_REQUIRE(x && dy && mean && rstd && scale && shift && coef1 && coef2 && dx && T > 0 && P > 0 && C > 0,
                 "b200_bn_relu_bwd_apply");
    return launch_bn_relu_bwd_apply(x, dy, mean, rstd, scale, shift, coef1, coef2, dx, T, P, C, tstride, dtype_fp32,
                                    static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------------------
// max-pool, ConvLSTM gate math, reductions, 1x1 output conv, pixel shuffle, strided copy
// ------------------------------------------------------------------------------------------------
extern "C" int b200_maxpool2_fwd(const void* x, void* y, long long IMG, int H, int W, int C, int dtype_fp32,
                                 void* stream) {
    B200_REQUIRE(x && y && IMG > 0 && H > 0 && W > 0 && C > 0, "b200_maxpool2_fwd");
    return launch_maxpool2_fwd(x, y, IMG, H, W, C, dtype_fp32, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_maxpool2_bwd(const void* x, const void* dy, void* dx, long long IMG, int H, int W, int C,
                                 int accumulate, int dtype_fp32, void* stream) {
    B200_REQUIRE(x && dy && dx && IMG > 0 && H > 0 && W > 0 && C > 0, "b200_maxpool2_bwd");
    return launch_maxpool2_bwd(x, dy, dx, IMG, H, W, C, accumulate, dtype_fp32, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_bn_relu_apply_pool(const void* x, const float* scale, const float* shift, void* y, void* pooled,
                                       int T, long long B, int H, int W, int C, int tstride, int dtype_fp32,
                                       void* stream) {
    B200_REQUIRE(x && scale && shift && y && pooled && T > 0 && B > 0 && H > 0 && W > 0 && C > 0, "b200_bn_relu_apply_pool");
    if ((H & 1) || (W & 1)) {
        set_last_error("b200_bn_relu_apply_pool: H and W must be even (got %dx%d)", H, W);
        return B200_ERR_SHAPE;
    }
    return launch_bn_relu_apply_pool(x, scale, shift, y, pooled, T, B, H, W, C, tstride, dtype_fp32,
                                     static_cast<cudaStream_t>(stream));
}

extern "C" int b200_bn_relu_pool_bwd_reduce(const void* x, const void* dy, const void* dp, const float* mean,
                                            const float* rstd, const float* scale, const float* shift, int T,
                                            long long B, int H, int W, int C, int tstride, int dtype_fp32,
                                            double* sum_g, double* sum_gx, void* stream) {
    B200_REQUIRE(x && dp && mean && rstd && scale && shift && sum_g && sum_gx && T > 0 && B > 0 && H > 0 && W > 0 && C > 0,
                 "b200_bn_relu_pool_bwd_reduce");
    if ((H & 1) || (W & 1)) {
        set_last_error("b200_bn_relu_pool_bwd_reduce: H and W must be even (got %dx%d)", H, W);
        return B200_ERR_SHAPE;
    }
    return launch_bn_relu_pool_bwd_reduce(x, dy, dp, mean, rstd, scale, shift, T, B, H, W, C, tstride, dtype_fp32, sum_g,
                                          sum_gx, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_bn_relu_pool_bwd_apply(const void* x, const void* dy, const void* dp, const float* mean,
                                           const float* rstd, const float* scale, const float* shift,
                                           const float* coef1, const float* coef2, void* dx, int T, long long B, int H,
                                           int W, int C, int tstride, int dtype_fp32, void* stream) {
    B200_REQUIRE(x && dp && mean && rstd && scale && shift && coef1 && coef2 && dx && T > 0 && B > 0 && H > 0 && W > 0 && C > 0,
                 "b200_bn_relu_pool_bwd_apply");
    if ((H & 1) || (W & 1)) {
        set_last_error("b200_bn_relu_pool_bwd_apply: H and W must be even (got %dx%d)", H, W);
        return B200_ERR_SHAPE;
    }
    return launch_bn_relu_pool_bwd_apply(x, dy, dp, mean, rstd, scale, shift, coef1, coef2, dx, T, B, H, W, C, tstride,
                                         dtype_fp32, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_bn_relu_outconv_fwd(const void* x, const float* scale, const float* shift, const float* w,
                                        const float* b, float* out, int T, long long P, int C, int tstride,
                                        int dtype_fp32, void* stream) {
    B200_REQUIRE(x && scale && shift && w && out && T > 0 && P > 0 && C > 0, "b200_bn_relu_outconv_fwd");
    return launch_bn_relu_outconv_fwd(x, scale, shift, w, b, out, T, P, C, tstride, dtype_fp32,
                                      static_cast<cudaStream_t>(stream));
}

extern "C" int b200_bn_relu_outconv_bwd_reduce(const void* x, const float* dout, const float* w, const float* mean,
                                               const float* rstd, const float* scale, const float* shift, int T,
                                               long long P, int C, int tstride, int dtype_fp32, double* sum_g,
                                               double* sum_gx, double* sum_dw, float* dw, void* stream) {
    B200_REQUIRE(x && dout && w && mean && rstd && scale && shift && sum_g && sum_gx && sum_dw && T > 0 && P > 0 && C > 0,
                 "b200_bn_relu_outconv_bwd_reduce");
    return launch_bn_relu_outconv_bwd_reduce(x, dout, w, mean, rstd, scale, shift, T, P, C, tstride, dtype_fp32, sum_g,
                                             sum_gx, sum_dw, dw, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_bn_relu_outconv_bwd_apply(const void* x, const float* dout, const float* w, const float* mean,
                                              const float* rstd, const float* scale, const float* shift,
                                              const float* coef1, const float* coef2, void* dx, int T, long long P,
                                              int C, int tstride, int dtype_fp32, void* stream) {
    B200_REQUIRE(x && dout && w && mean && rstd && scale && shift && coef1 && coef2 && dx && T > 0 && P > 0 && C > 0,
                 "b200_bn_relu_outconv_bwd_apply");
    return launch_bn_relu_outconv_bwd_apply(x, dout, w, mean, rstd, scale, shift, coef1, coef2, dx, T, P, C, tstride,
                                            dtype_fp32, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_lstm_gates_fwd(const float* z, const float* c_prev, void* gates, float* c_next, void* h_next,
                                   long long P, int Ch, int dtype_fp32, void* stream) {
    B200_REQUIRE(z && gates && c_next && h_next && P > 0 && Ch > 0, "b200_lstm_gates_fwd");
    return launch_lstm_gates_fwd(z, c_prev, gates, c_next, h_next, P, Ch, dtype_fp32,
                                 static_cast<cudaStream_t>(stream));
}

extern "C" int b200_lstm_gates_bwd(const void* gates, const float* c_prev, const float* c_next, const void* dh_a,
                                   const void* dh_b, const float* dc_next, void* dz, float* dc_prev, long long P,
                                   int Ch, int dtype_fp32, void* stream) {
    B200_REQUIRE(gates && c_next && dz && dc_prev && P > 0 && Ch > 0, "b200_lstm_gates_bwd");
    return launch_lstm_gates_bwd(gates, c_prev, c_next, dh_a, dh_b, dc_next, dz, dc_prev, P, Ch, dtype_fp32,
                                 static_cast<cudaStream_t>(stream));
}

extern "C" int b200_colsum(const void* x, long long rows, int C, int dtype_fp32, double* workspace, float* out,
                           int accumulate, void* stream) {
    B200_REQUIRE(x && workspace && out && rows > 0 && C > 0, "b200_colsum");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc = launch_colsum(x, rows, C, dtype_fp32, workspace, st);
    if (rc != B200_OK) return rc;
    return launch_cast_double(workspace, out, C, accumulate, st);
}

extern "C" int b200_outconv_fwd(const void* x, const float* w, const float* b, float* y, long long P, int C, int O,
                                int dtype_fp32, void* stream) {
    B200_REQUIRE(x && w && y && P > 0 && C > 0 && O > 0, "b200_outconv_fwd");
    return launch_outconv_fwd(x, w, b, y, P, C, O, dtype_fp32, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_outconv_bwd(const void* x, const float* w, const float* dy, long long P, int C, int O,
                                int dtype_fp32, void* dx, double* workspace, float* dw, float* db, int accumulate,
                                void* stream) {
    B200_REQUIRE(x && w && dy && workspace && P > 0 && C > 0 && O > 0, "b200_outconv_bwd");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc = B200_OK;
    if (dx) {
        rc = launch_outconv_dgrad(dy, w, dx, P, C, O, dtype_fp32, st);
        if (rc != B200_OK) return rc;
    }
    if (dw) {
        for (int o = 0; o < O; ++o) {
            rc = launch_outconv_wgrad(x, dy, P, C, O, o, dtype_fp32, workspace, st);
            if (rc != B200_OK) return rc;
            rc = launch_cast_double(workspace, dw + static_cast<long long>(o) * C, C, accumulate, st);
            if (rc != B200_OK) return rc;
        }
    }
    if (db) {
        rc = launch_colsum(dy, P, O, 1, workspace, st);
        if (rc != B200_OK) return rc;
        rc = launch_cast_double(workspace, db, O, accumulate, st);
    }
    return rc;
}

extern "C" int b200_shuffle2x2(const void* src, void* dst, const float* bias, long long IMG, int H, int W, int C,
                               int Hd, int Wd, int oy, int ox, int unshuffle, int dtype_fp32, void* stream) {
    B200_REQUIRE(src && dst && IMG > 0 && H > 0 && W > 0 && C > 0 && Hd > 0 && Wd > 0, "b200_shuffle2x2");
    return launch_shuffle2x2(src, dst, bias, IMG, H, W, C, Hd, Wd, oy, ox, unshuffle, dtype_fp32,
                             static_cast<cudaStream_t>(stream));
}

extern "C" int b200_strided_copy(const void* src, int src_fp32, void* dst, int dst_fp32, const long long* dims,
                                 const long long* src_strides, const long long* dst_strides, int accumulate,
                                 void* stream) {
    B200_REQUIRE(src && dst && dims && src_strides && dst_strides, "b200_strided_copy");
    for (int i = 0; i < 5; ++i)
        if (dims[i] < 0) {
            set_last_error("b200_strided_copy: negative dimension");
            return B200_ERR_ARG;
        }
    return launch_strided_copy(src, src_fp32, dst, dst_fp32, dims, src_strides, dst_strides, accumulate,
                               static_cast<cudaStream_t>(stream));
}
