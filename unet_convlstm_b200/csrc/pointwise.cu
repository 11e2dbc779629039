// HBM-bound kernels of the hot path: BatchNorm statistics / apply / backward, ReLU, 2x2 max-pool,
// the ConvLSTM gate math (forward when not fused into the GEMM epilogue, and the BPTT gate
// gradients), the 1x1 output convolution, pixel (un)shuffle for the 2x2 transposed convolution and
// a generic strided copy used for layout changes and weight (un)packing.
//
// Conventions: activations are NHWC; a sequence tensor is [T][P][C] with P = B*H*W pixels.  Every
// kernel is templated on the storage type (float: fp32 check mode, __nv_bfloat16: bf16 mode) and on
// the vector width V: 16-byte accesses (V = 4 floats / 8 bf16) when the channel count and the
// pointers allow it, scalar accesses (V = 1) otherwise.  Reductions over pixels keep per-thread
// partial sums in registers (double in the fp32 mode), combine them through shared memory and
// finish with one double-precision atomic per channel and block.
#include "pointwise.cuh"

#include <type_traits>

namespace b200 {

// ------------------------------------------------------------------------------------------------
// vector load / store helpers
// ------------------------------------------------------------------------------------------------
template <typename T, int V>
__device__ __forceinline__ void ldv(const T* __restrict__ p, float (&f)[V]) {
    if constexpr (V == 1) {
        if constexpr (std::is_same<T, float>::value)
            f[0] = p[0];
        else
            f[0] = __bfloat162float(p[0]);
    } else if constexpr (std::is_same<T, float>::value) {
#pragma unroll
        for (int i = 0; i < V / 4; ++i) {
            const float4 t = reinterpret_cast<const float4*>(p)[i];
            f[4 * i] = t.x;
            f[4 * i + 1] = t.y;
            f[4 * i + 2] = t.z;
            f[4 * i + 3] = t.w;
        }
    } else {
        static_assert(V % 8 == 0 || V == 1, "bf16 vectors are 8 wide");
#pragma unroll
        for (int i = 0; i < V / 8; ++i) {
            const uint4 t = reinterpret_cast<const uint4*>(p)[i];
            const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                f[8 * i + 2 * j] = __uint_as_float(w[j] << 16);
                f[8 * i + 2 * j + 1] = __uint_as_float(w[j] & 0xffff0000u);
            }
        }
    }
}

// Raw (not yet converted) vector of V elements: lets a loop issue several independent 16-byte loads
// before the first conversion, so enough bytes are in flight to cover the HBM latency.
template <typename T, int V>
struct RawVec {
    static constexpr int NW = (V == 1) ? 1 : 4;
    uint32_t w[NW];
};
template <typename T, int V>
__device__ __forceinline__ void ld_raw(const T* __restrict__ p, RawVec<T, V>& r) {
    if constexpr (V == 1) {
        if constexpr (std::is_same<T, float>::value)
            r.w[0] = __float_as_uint(p[0]);
        else
            r.w[0] = static_cast<uint32_t>(*reinterpret_cast<const unsigned short*>(p)) << 16;
    } else {
        const uint4 t = *reinterpret_cast<const uint4*>(p);
        r.w[0] = t.x; r.w[1] = t.y; r.w[2] = t.z; r.w[3] = t.w;
    }
}
template <typename T, int V>
__device__ __forceinline__ void unpack_raw(const RawVec<T, V>& r, float (&f)[V]) {
    if constexpr (V == 1) {
        f[0] = __uint_as_float(r.w[0]);
    } else if constexpr (std::is_same<T, float>::value) {
        static_assert(V == 4, "fp32 vectors are 4 wide");
#pragma unroll
        for (int j = 0; j < 4; ++j) f[j] = __uint_as_float(r.w[j]);
    } else {
        static_assert(V == 8, "bf16 vectors are 8 wide");
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            f[2 * j] = __uint_as_float(r.w[j] << 16);
            f[2 * j + 1] = __uint_as_float(r.w[j] & 0xffff0000u);
        }
    }
}

__device__ __forceinline__ uint32_t pack2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}

template <typename T, int V>
__device__ __forceinline__ void stv(T* __restrict__ p, const float (&f)[V]) {
    if constexpr (V == 1) {
        if constexpr (std::is_same<T, float>::value)
            p[0] = f[0];
        else
            p[0] = __float2bfloat16_rn(f[0]);
    } else if constexpr (std::is_same<T, float>::value) {
#pragma unroll
        for (int i = 0; i < V / 4; ++i)
            reinterpret_cast<float4*>(p)[i] = make_float4(f[4 * i], f[4 * i + 1], f[4 * i + 2], f[4 * i + 3]);
    } else {
#pragma unroll
        for (int i = 0; i < V / 8; ++i)
            reinterpret_cast<uint4*>(p)[i] =
                make_uint4(pack2(f[8 * i], f[8 * i + 1]), pack2(f[8 * i + 2], f[8 * i + 3]),
                           pack2(f[8 * i + 4], f[8 * i + 5]), pack2(f[8 * i + 6], f[8 * i + 7]));
    }
}

template <typename T>
static int pick_vec(int C, std::initializer_list<const void*> ptrs) {
    constexpr int V = std::is_same<T, float>::value ? 4 : 8;
    if (C % V != 0) return 1;
    for (const void* p : ptrs)
        if (p && (reinterpret_cast<uintptr_t>(p) & 15)) return 1;
    return V;
}

static inline unsigned grid_for(long long work, int per_block, int max_blocks) {
    long long g = (work + per_block - 1) / per_block;
    if (g > max_blocks) g = max_blocks;
    if (g < 1) g = 1;
    return static_cast<unsigned>(g);
}

// ------------------------------------------------------------------------------------------------
// column reductions over pixels:  out[t][c] = sum_p f(t, p, c)
// ------------------------------------------------------------------------------------------------
struct ReduceGeom {
    int T;
    long long P;  // rows per t
    int C;
    int cvb;            // channel vectors per block
    int rows_per_iter;  // 256 / cvb
    long long rows_per_block;
};

// Op::load(frag, t, row, c) fetches the raw operands of V channels starting at c of one row;
// Op::accum(state, frag, a0, a1) adds their contribution.  The row loop loads ColredTraits<Op>::U rows ahead;
// ColredTraits<Op>::BLOCKS = resident blocks per SM the bf16 instantiation is compiled for (an Op whose "row" is a
// 2x2 pixel window holds nine 16-byte vectors per row: one row in flight, two blocks per SM).
template <typename Op>
struct ColredTraits {
    static constexpr int U = 4;
    static constexpr int BLOCKS = 4;
};
template <typename T, int V, typename Acc, typename Op>
__global__ void __launch_bounds__(256, (std::is_same<T, float>::value ? 2 : ColredTraits<Op>::BLOCKS)) colreduce_kernel(const Op op, const ReduceGeom g, double* __restrict__ out0,
                                                        double* __restrict__ out1) {
    constexpr int COLRED_U = ColredTraits<Op>::U;
    __shared__ Acc red[2][256 * (V > 4 ? 4 : V)];  // reduced in two halves when V == 8
    const int tid = threadIdx.x;
    const int r = tid / g.cvb;
    const int cv = tid - r * g.cvb;
    const int c = (blockIdx.y * g.cvb + cv) * V;
    const int t = blockIdx.z;
    const bool active = (r < g.rows_per_iter) && (c < g.C);
    const long long p_begin = static_cast<long long>(blockIdx.x) * g.rows_per_block;
    long long p_end = p_begin + g.rows_per_block;
    if (p_end > g.P) p_end = g.P;

    Acc a0[V], a1[V];
#pragma unroll
    for (int j = 0; j < V; ++j) a0[j] = a1[j] = Acc(0);
    if (active) {
        typename Op::template State<V> st;  // per-thread coefficients, loaded once
        op.template init<V>(t, c, st);
        const long long step = g.rows_per_iter;
        long long p = p_begin + r;
        // main loop: COLRED_U independent rows per trip, every load issued before the first use
        for (; p + (COLRED_U - 1) * step < p_end; p += COLRED_U * step) {
            typename Op::template Frag<T, V> fr[COLRED_U];
#pragma unroll
            for (int u = 0; u < COLRED_U; ++u) op.template load<T, V>(fr[u], t, p + u * step, c);
#pragma unroll
            for (int u = 0; u < COLRED_U; ++u) op.template accum<T, V, Acc>(st, fr[u], a0, a1);
        }
        for (; p < p_end; p += step) {
            typename Op::template Frag<T, V> fr;
            op.template load<T, V>(fr, t, p, c);
            op.template accum<T, V, Acc>(st, fr, a0, a1);
        }
    }
    // combine the rows_per_iter partial sums of each channel
    constexpr int HV = V > 4 ? 4 : V;
#pragma unroll
    for (int half = 0; half < V / HV; ++half) {
        __syncthreads();
#pragma unroll
        for (int j = 0; j < HV; ++j) {
            red[0][tid * HV + j] = a0[half * HV + j];
            red[1][tid * HV + j] = a1[half * HV + j];
        }
        __syncthreads();
        if (r == 0 && c < g.C) {
#pragma unroll
            for (int j = 0; j < HV; ++j) {
                double s0 = 0.0, s1 = 0.0;
                for (int rr = 0; rr < g.rows_per_iter; ++rr) {
                    s0 += static_cast<double>(red[0][(rr * g.cvb + cv) * HV + j]);
                    s1 += static_cast<double>(red[1][(rr * g.cvb + cv) * HV + j]);
                }
                const long long o = static_cast<long long>(t) * g.C + c + half * HV + j;
                op.post(t, c + half * HV + j, s0, s1);
                atomicAdd(out0 + o, s0);
                if (out1) atomicAdd(out1 + o, s1);
            }
        }
    }
}

template <typename T, typename Op>
static int launch_colreduce(const Op& op, int T_, long long P, int C, int V, double* out0, double* out1,
                            cudaStream_t stream) {
    ReduceGeom g;
    g.T = T_;
    g.P = P;
    g.C = C;
    const int CV = C / V;
    g.cvb = CV < 256 ? CV : 256;
    g.rows_per_iter = 256 / g.cvb;
    const unsigned gy = (CV + g.cvb - 1) / g.cvb;
    // at most 8 blocks per SM in total (= two full waves at 4 resident blocks per SM; rounding UP here gave 1200 blocks
    // on 1184 slots at T = 20, i.e. a third, almost empty wave: ncu showed the SMs idle for 21 % of the kernel), at
    // least 4 iterations per thread
    long long want_x = (2LL * ColredTraits<Op>::BLOCKS * num_sms()) / ((long long)gy * T_);
    long long max_x = (P + 4LL * g.rows_per_iter - 1) / (4LL * g.rows_per_iter);
    if (want_x > max_x) want_x = max_x;
    if (want_x < 1) want_x = 1;
    g.rows_per_block = (P + want_x - 1) / want_x;
    const unsigned gx = static_cast<unsigned>((P + g.rows_per_block - 1) / g.rows_per_block);
    dim3 grid(gx, gy, T_);
    using Acc = typename std::conditional<std::is_same<T, float>::value, double, float>::type;
    if (V == 1)
        colreduce_kernel<T, 1, Acc, Op><<<grid, 256, 0, stream>>>(op, g, out0, out1);
    else if constexpr (std::is_same<T, float>::value)
        colreduce_kernel<T, 4, Acc, Op><<<grid, 256, 0, stream>>>(op, g, out0, out1);
    else
        colreduce_kernel<T, 8, Acc, Op><<<grid, 256, 0, stream>>>(op, g, out0, out1);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// ---- BatchNorm statistics: sum x, sum x^2 (nn.BatchNorm2d training forward, unet.py:70-71) ----
struct NoState {
    template <int V>
    struct State {};
    template <int V>
    __device__ __forceinline__ void init(int, int, State<V>&) const {}
    __device__ __forceinline__ void post(int, int, double&, double&) const {}
};

struct StatsOp : NoState {
    const void* x;
    long long P;
    int C;
    template <typename T, int V>
    struct Frag {
        RawVec<T, V> x;
    };
    template <typename T, int V>
    __device__ __forceinline__ void load(Frag<T, V>& fr, int t, long long p, int c) const {
        ld_raw<T, V>(static_cast<const T*>(x) + (static_cast<long long>(t) * P + p) * C + c, fr.x);
    }
    template <typename T, int V, typename Acc>
    __device__ __forceinline__ void accum(const State<V>&, const Frag<T, V>& fr, Acc (&a0)[V], Acc (&a1)[V]) const {
        float f[V];
        unpack_raw<T, V>(fr.x, f);
#pragma unroll
        for (int j = 0; j < V; ++j) {
            a0[j] += Acc(f[j]);
            a1[j] += Acc(f[j]) * Acc(f[j]);
        }
    }
};

int launch_bn_stats(const void* x, int T_, long long P, int C, int dtype_fp32, double* sum, double* sumsq,
                    cudaStream_t stream) {
    B200_CUDA_CHECK(cudaMemsetAsync(sum, 0, sizeof(double) * T_ * C, stream));
    B200_CUDA_CHECK(cudaMemsetAsync(sumsq, 0, sizeof(double) * T_ * C, stream));
    StatsOp op;
    op.x = x; op.P = P; op.C = C;
    if (dtype_fp32) return launch_colreduce<float>(op, T_, P, C, pick_vec<float>(C, {x}), sum, sumsq, stream);
    return launch_colreduce<__nv_bfloat16>(op, T_, P, C, pick_vec<__nv_bfloat16>(C, {x}), sum, sumsq, stream);
}

// ---- plain column sum (bias gradients) ----
struct ColsumOp : NoState {
    const void* x;
    int C;
    template <typename T, int V>
    struct Frag {
        RawVec<T, V> x;
    };
    template <typename T, int V>
    __device__ __forceinline__ void load(Frag<T, V>& fr, int, long long p, int c) const {
        ld_raw<T, V>(static_cast<const T*>(x) + p * C + c, fr.x);
    }
    template <typename T, int V, typename Acc>
    __device__ __forceinline__ void accum(const State<V>&, const Frag<T, V>& fr, Acc (&a0)[V], Acc (&)[V]) const {
        float f[V];
        unpack_raw<T, V>(fr.x, f);
#pragma unroll
        for (int j = 0; j < V; ++j) a0[j] += Acc(f[j]);
    }
};

int launch_colsum(const void* x, long long rows, int C, int dtype_fp32, double* out, cudaStream_t stream) {
    B200_CUDA_CHECK(cudaMemsetAsync(out, 0, sizeof(double) * C, stream));
    ColsumOp op;
    op.x = x; op.C = C;
    if (dtype_fp32) return launch_colreduce<float>(op, 1, rows, C, pick_vec<float>(C, {x}), out, nullptr, stream);
    return launch_colreduce<__nv_bfloat16>(op, 1, rows, C, pick_vec<__nv_bfloat16>(C, {x}), out, nullptr, stream);
}

// ---- BatchNorm+ReLU backward reduction: sum g, sum g*xhat with g = dy * [relu active] ----
struct BnBwdReduceOp {
    const void* x;    // pre-BN conv output
    const void* dy;   // gradient w.r.t. the ReLU output
    const float* mean;   // [Ts][C]
    const float* rstd;   // [Ts][C]
    const float* scale;  // [Ts][C]
    const float* shift;  // [Ts][C]
    long long P;
    int C;
    int tstride;  // C in training mode, 0 in eval mode (one set of statistics for every t)
    // Only the ReLU mask needs coefficients inside the loop: the kernel accumulates sum g and sum g*x and
    // the block epilogue turns the second into sum g*xhat = rstd * (sum g*x - mean * sum g) in fp64.
    template <int V>
    struct State {
        float sc[V], sh[V];
    };
    template <int V>
    __device__ __forceinline__ void init(int t, int c, State<V>& st) const {
#pragma unroll
        for (int j = 0; j < V; ++j) {
            const int i = t * tstride + c + j;
            st.sc[j] = __ldg(scale + i);
            st.sh[j] = __ldg(shift + i);
        }
    }
    __device__ __forceinline__ void post(int t, int c, double& s0, double& s1) const {
        const int i = t * tstride + c;
        s1 = static_cast<double>(__ldg(rstd + i)) * (s1 - static_cast<double>(__ldg(mean + i)) * s0);
    }
    template <typename T, int V>
    struct Frag {
        RawVec<T, V> x, d;
    };
    template <typename T, int V>
    __device__ __forceinline__ void load(Frag<T, V>& fr, int t, long long p, int c) const {
        const long long off = (static_cast<long long>(t) * P + p) * C + c;
        ld_raw<T, V>(static_cast<const T*>(x) + off, fr.x);
        ld_raw<T, V>(static_cast<const T*>(dy) + off, fr.d);
    }
    template <typename T, int V, typename Acc>
    __device__ __forceinline__ void accum(const State<V>& st, const Frag<T, V>& fr, Acc (&a0)[V],
                                          Acc (&a1)[V]) const {
        float fx[V], fd[V];
        unpack_raw<T, V>(fr.x, fx);
        unpack_raw<T, V>(fr.d, fd);
#pragma unroll
        for (int j = 0; j < V; ++j) {
            const float yv = fmaf(fx[j], st.sc[j], st.sh[j]);
            const float gq = yv > 0.f ? fd[j] : 0.f;
            a0[j] += Acc(gq);
            a1[j] += Acc(gq) * Acc(fx[j]);
        }
    }
};

int launch_bn_relu_bwd_reduce(const void* x, const void* dy, const float* mean, const float* rstd,
                              const float* scale, const float* shift, int T_, long long P, int C, int tstride,
                              int dtype_fp32, double* sum_g, double* sum_gx, cudaStream_t stream) {
    B200_CUDA_CHECK(cudaMemsetAsync(sum_g, 0, sizeof(double) * T_ * C, stream));
    B200_CUDA_CHECK(cudaMemsetAsync(sum_gx, 0, sizeof(double) * T_ * C, stream));
    BnBwdReduceOp op{x, dy, mean, rstd, scale, shift, P, C, tstride};
    if (dtype_fp32)
        return launch_colreduce<float>(op, T_, P, C, pick_vec<float>(C, {x, dy}), sum_g, sum_gx, stream);
    return launch_colreduce<__nv_bfloat16>(op, T_, P, C, pick_vec<__nv_bfloat16>(C, {x, dy}), sum_g, sum_gx, stream);
}

// ---- 1x1 output conv weight gradient: dw[o][c] = sum_p dy[p][o] * x[p][c] (OutConv, unet.py:104) ----
struct OutconvWgradOp : NoState {
    const void* x;
    const float* dy;  // [P][O] fp32
    int C, O, o;
    template <typename T, int V>
    struct Frag {
        RawVec<T, V> x;
        float d;
    };
    template <typename T, int V>
    __device__ __forceinline__ void load(Frag<T, V>& fr, int, long long p, int c) const {
        ld_raw<T, V>(static_cast<const T*>(x) + p * C + c, fr.x);
        fr.d = __ldg(dy + p * O + o);
    }
    template <typename T, int V, typename Acc>
    __device__ __forceinline__ void accum(const State<V>&, const Frag<T, V>& fr, Acc (&a0)[V], Acc (&)[V]) const {
        float f[V];
        unpack_raw<T, V>(fr.x, f);
#pragma unroll
        for (int j = 0; j < V; ++j) a0[j] += Acc(fr.d) * Acc(f[j]);
    }
};

int launch_outconv_wgrad(const void* x, const float* dy, long long P, int C, int O, int o, int dtype_fp32,
                         double* out, cudaStream_t stream) {
    B200_CUDA_CHECK(cudaMemsetAsync(out, 0, sizeof(double) * C, stream));
    OutconvWgradOp op;
    op.x = x; op.dy = dy; op.C = C; op.O = O; op.o = o;
    if (dtype_fp32) return launch_colreduce<float>(op, 1, P, C, pick_vec<float>(C, {x}), out, nullptr, stream);
    return launch_colreduce<__nv_bfloat16>(op, 1, P, C, pick_vec<__nv_bfloat16>(C, {x}), out, nullptr, stream);
}

// ------------------------------------------------------------------------------------------------
// BatchNorm finalisation (tiny kernels: one thread per channel, sequential over t)
// ------------------------------------------------------------------------------------------------
// Training: per-call (= per-timestep, unet.py:179-182) batch statistics, biased variance for the
// normalisation, T sequential momentum updates of the running estimates with the unbiased variance.
// Eval: scale/shift from the running estimates (Ts = 1).
__global__ void bn_finalize_kernel(const double* __restrict__ sum, const double* __restrict__ sumsq, int T_,
                                   long long n, int C, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float* running_mean, float* running_var,
                                   float eps, float momentum, int training, float* __restrict__ mean,
                                   float* __restrict__ rstd, float* __restrict__ scale, float* __restrict__ shift) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float gm = gamma[c], bt = beta[c];
    if (!training) {
        const float m = running_mean[c];
        const float rs = static_cast<float>(1.0 / sqrt(static_cast<double>(running_var[c]) + eps));
        mean[c] = m;
        rstd[c] = rs;
        scale[c] = gm * rs;
        shift[c] = bt - m * gm * rs;
        return;
    }
    // running statistics are optional (track_running_stats=False); momentum < 0 encodes nn.BatchNorm2d(momentum=None),
    // the cumulative moving average: momentum = -(n0 + 1) with n0 = num_batches_tracked before this call, and the
    // update factor of step t is 1 / (n0 + t + 1)
    const bool track = running_mean != nullptr && running_var != nullptr;
    double rm = track ? running_mean[c] : 0.0, rv = track ? running_var[c] : 0.0;
    for (int t = 0; t < T_; ++t) {
        const double m = sum[t * C + c] / n;
        double var = sumsq[t * C + c] / n - m * m;
        if (var < 0) var = 0;
        const double rs = 1.0 / sqrt(var + eps);
        mean[t * C + c] = static_cast<float>(m);
        rstd[t * C + c] = static_cast<float>(rs);
        const float sc = static_cast<float>(gm * rs);
        scale[t * C + c] = sc;
        shift[t * C + c] = static_cast<float>(bt - m * gm * rs);
        const double unb = n > 1 ? var * (static_cast<double>(n) / (n - 1)) : var;
        // fp32 rounding after each update, like the reference's fp32 buffers
        const double f = momentum >= 0.f ? static_cast<double>(momentum) : 1.0 / (static_cast<double>(-momentum) + t);
        rm = static_cast<float>((1.0 - f) * rm + f * m);
        rv = static_cast<float>((1.0 - f) * rv + f * unb);
    }
    if (track) {
        running_mean[c] = static_cast<float>(rm);
        running_var[c] = static_cast<float>(rv);
    }
}

int launch_bn_finalize(const double* sum, const double* sumsq, int T_, long long n, int C, const float* gamma,
                       const float* beta, float* running_mean, float* running_var, float eps, float momentum,
                       int training, float* mean, float* rstd, float* scale, float* shift, cudaStream_t stream) {
    bn_finalize_kernel<<<(C + 127) / 128, 128, 0, stream>>>(sum, sumsq, T_, n, C, gamma, beta, running_mean,
                                                            running_var, eps, momentum, training, mean, rstd,
                                                            scale, shift);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// coef1 = sum_g / n, coef2 = sum_gx / n (zero in eval mode); dgamma += sum_t sum_gx, dbeta += sum_t sum_g
// dconv_bias = sum over pixels of dz = scale * (sum_g - n*coef1 - coef2 * sum xhat): identically zero in
// training mode (sum xhat = 0, n*coef1 = sum_g); scale * sum_g with running statistics (eval mode).
__global__ void bn_bwd_finalize_kernel(const double* __restrict__ sum_g, const double* __restrict__ sum_gx, int T_,
                                       long long n, int C, int training, const float* __restrict__ scale,
                                       float* __restrict__ coef1, float* __restrict__ coef2,
                                       float* __restrict__ dgamma, float* __restrict__ dbeta,
                                       float* __restrict__ dconv_bias, int accumulate) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double dg = 0, db = 0;
    for (int t = 0; t < T_; ++t) {
        const double sg = sum_g[t * C + c], sgx = sum_gx[t * C + c];
        dg += sgx;
        db += sg;
        coef1[t * C + c] = training ? static_cast<float>(sg / n) : 0.f;
        coef2[t * C + c] = training ? static_cast<float>(sgx / n) : 0.f;
    }
    const float dcb = training ? 0.f : static_cast<float>(scale[c] * db);
    if (accumulate) {
        dgamma[c] += static_cast<float>(dg);
        dbeta[c] += static_cast<float>(db);
        if (dconv_bias) dconv_bias[c] += dcb;
    } else {
        dgamma[c] = static_cast<float>(dg);
        dbeta[c] = static_cast<float>(db);
        if (dconv_bias) dconv_bias[c] = dcb;
    }
}

int launch_bn_bwd_finalize(const double* sum_g, const double* sum_gx, int T_, long long n, int C, int training,
                           const float* scale, float* coef1, float* coef2, float* dgamma, float* dbeta,
                           float* dconv_bias, int accumulate, cudaStream_t stream) {
    bn_bwd_finalize_kernel<<<(C + 127) / 128, 128, 0, stream>>>(sum_g, sum_gx, T_, n, C, training, scale, coef1,
                                                                coef2, dgamma, dbeta, dconv_bias, accumulate);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

__global__ void cast_double_kernel(const double* __restrict__ src, float* __restrict__ dst, int n, int accumulate) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float v = static_cast<float>(src[i]);
    dst[i] = accumulate ? dst[i] + v : v;
}

int launch_cast_double(const double* src, float* dst, int n, int accumulate, cudaStream_t stream) {
    cast_double_kernel<<<(n + 255) / 256, 256, 0, stream>>>(src, dst, n, accumulate);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// ------------------------------------------------------------------------------------------------
// element-wise kernels over [T][P][C]
// ------------------------------------------------------------------------------------------------
// Row-loop geometry shared by the BatchNorm apply kernels: like colreduce, a thread owns a fixed vector
// of V channels of one timestep, so the per-(t, channel) coefficients are loaded ONCE into registers
// and the loop over pixels only touches the activations (an earlier version re-read six coefficient
// arrays per element and was L1-bound at 56 % of HBM peak, profiles/r01_ncu_bn_relu_bwd_apply.txt).
static ReduceGeom rowloop_geom(int T_, long long P, int C, int V, dim3* grid) {
    ReduceGeom g;
    g.T = T_;
    g.P = P;
    g.C = C;
    const int CV = C / V;
    g.cvb = CV < 256 ? CV : 256;
    g.rows_per_iter = 256 / g.cvb;
    const unsigned gy = (CV + g.cvb - 1) / g.cvb;
    long long want_x = (16LL * num_sms() + (long long)gy * T_ - 1) / ((long long)gy * T_);
    long long max_x = (P + 8LL * g.rows_per_iter - 1) / (8LL * g.rows_per_iter);
    if (want_x > max_x) want_x = max_x;
    if (want_x < 1) want_x = 1;
    g.rows_per_block = (P + want_x - 1) / want_x;
    *grid = dim3(static_cast<unsigned>((P + g.rows_per_block - 1) / g.rows_per_block), gy, T_);
    return g;
}

// y = relu(x * scale[t][c] + shift[t][c])   (BatchNorm2d + ReLU, unet.py:70-71)
template <typename T, int V>
__global__ void __launch_bounds__(256) bn_relu_apply_kernel(const T* __restrict__ x, const float* __restrict__ scale,
                                                            const float* __restrict__ shift, T* __restrict__ y,
                                                            const ReduceGeom g, int tstride, int relu) {
    const int tid = threadIdx.x;
    const int r = tid / g.cvb;
    const int cv = tid - r * g.cvb;
    const int c = (blockIdx.y * g.cvb + cv) * V;
    const int t = blockIdx.z;
    if (r >= g.rows_per_iter || c >= g.C) return;
    float sc[V], sh[V];
#pragma unroll
    for (int j = 0; j < V; ++j) {
        sc[j] = __ldg(scale + t * tstride + c + j);
        sh[j] = __ldg(shift + t * tstride + c + j);
    }
    const long long p_begin = static_cast<long long>(blockIdx.x) * g.rows_per_block;
    long long p_end = p_begin + g.rows_per_block;
    if (p_end > g.P) p_end = g.P;
    const long long base = static_cast<long long>(t) * g.P;
#pragma unroll 4
    for (long long p = p_begin + r; p < p_end; p += g.rows_per_iter) {
        const long long off = (base + p) * g.C + c;
        float f[V];
        ldv<T, V>(x + off, f);
#pragma unroll
        for (int j = 0; j < V; ++j) {
            f[j] = fmaf(f[j], sc[j], sh[j]);
            if (relu) f[j] = fmaxf(f[j], 0.f);
        }
        stv<T, V>(y + off, f);
    }
}

int launch_bn_relu_apply(const void* x, const float* scale, const float* shift, void* y, int T_, long long P, int C,
                         int tstride, int relu, int dtype_fp32, cudaStream_t stream) {
    auto go = [&](auto tag, int V) {
        using T = decltype(tag);
        dim3 grid;
        const ReduceGeom g = rowloop_geom(T_, P, C, V, &grid);
        const T* xs = static_cast<const T*>(x);
        T* ys = static_cast<T*>(y);
        if (V == 1)
            bn_relu_apply_kernel<T, 1><<<grid, 256, 0, stream>>>(xs, scale, shift, ys, g, tstride, relu);
        else if constexpr (std::is_same<T, float>::value)
            bn_relu_apply_kernel<T, 4><<<grid, 256, 0, stream>>>(xs, scale, shift, ys, g, tstride, relu);
        else
            bn_relu_apply_kernel<T, 8><<<grid, 256, 0, stream>>>(xs, scale, shift, ys, g, tstride, relu);
    };
    if (dtype_fp32)
        go(float(), pick_vec<float>(C, {x, y}));
    else
        go(__nv_bfloat16(), pick_vec<__nv_bfloat16>(C, {x, y}));
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// dx = scale * (g - coef1 - xhat * coef2),  g = dy * [x*scale+shift > 0],  xhat = (x - mean) * rstd
template <typename T, int V>
__global__ void __launch_bounds__(256, (std::is_same<T, float>::value ? 2 : 4))
bn_relu_bwd_apply_kernel(const T* __restrict__ x, const T* __restrict__ dy, const float* __restrict__ mean,
                         const float* __restrict__ rstd, const float* __restrict__ scale,
                         const float* __restrict__ shift, const float* __restrict__ coef1,
                         const float* __restrict__ coef2, T* __restrict__ dx, const ReduceGeom g, int tstride) {
    const int tid = threadIdx.x;
    const int r = tid / g.cvb;
    const int cv = tid - r * g.cvb;
    const int c = (blockIdx.y * g.cvb + cv) * V;
    const int t = blockIdx.z;
    if (r >= g.rows_per_iter || c >= g.C) return;
    // dx = scale * (g - c1 - (x - mean) * rstd * c2)  =  scale * g + ka * x + kb   (g = dy where ReLU is active)
    float sc[V], sh[V], ka[V], kb[V];
#pragma unroll
    for (int j = 0; j < V; ++j) {
        const int ps = t * tstride + c + j, pc = t * g.C + c + j;
        sc[j] = __ldg(scale + ps);
        sh[j] = __ldg(shift + ps);
        const float rc2 = __ldg(rstd + ps) * __ldg(coef2 + pc);
        ka[j] = -sc[j] * rc2;
        kb[j] = sc[j] * (rc2 * __ldg(mean + ps) - __ldg(coef1 + pc));
    }
    const long long p_begin = static_cast<long long>(blockIdx.x) * g.rows_per_block;
    long long p_end = p_begin + g.rows_per_block;
    if (p_end > g.P) p_end = g.P;
    const long long base = static_cast<long long>(t) * g.P;
    auto apply = [&](const RawVec<T, V>& rx, const RawVec<T, V>& rd, long long off) {
        float fx[V], fd[V];
        unpack_raw<T, V>(rx, fx);
        unpack_raw<T, V>(rd, fd);
#pragma unroll
        for (int j = 0; j < V; ++j) {
            const float yv = fmaf(fx[j], sc[j], sh[j]);
            const float gq = yv > 0.f ? fd[j] : 0.f;
            fd[j] = fmaf(sc[j], gq, fmaf(ka[j], fx[j], kb[j]));
        }
        stv<T, V>(dx + off, fd);
    };
    // U independent rows per trip: all 2U loads are issued before the first use
    constexpr int U = 4;
    const long long step = g.rows_per_iter;
    long long p = p_begin + r;
    for (; p + (U - 1) * step < p_end; p += U * step) {
        RawVec<T, V> rx[U], rd[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long off = (base + p + u * step) * g.C + c;
            ld_raw<T, V>(x + off, rx[u]);
            ld_raw<T, V>(dy + off, rd[u]);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) apply(rx[u], rd[u], (base + p + u * step) * g.C + c);
    }
    for (; p < p_end; p += step) {
        const long long off = (base + p) * g.C + c;
        RawVec<T, V> rx, rd;
        ld_raw<T, V>(x + off, rx);
        ld_raw<T, V>(dy + off, rd);
        apply(rx, rd, off);
    }
}

int launch_bn_relu_bwd_apply(const void* x, const void* dy, const float* mean, const float* rstd, const float* scale,
                             const float* shift, const float* coef1, const float* coef2, void* dx, int T_,
                             long long P, int C, int tstride, int dtype_fp32, cudaStream_t stream) {
    auto go = [&](auto tag, int V) {
        using T = decltype(tag);
        dim3 grid;
        const ReduceGeom g = rowloop_geom(T_, P, C, V, &grid);
        const T* xs = static_cast<const T*>(x);
        const T* ds = static_cast<const T*>(dy);
        T* os = static_cast<T*>(dx);
        if (V == 1)
            bn_relu_bwd_apply_kernel<T, 1><<<grid, 256, 0, stream>>>(xs, ds, mean, rstd, scale, shift, coef1, coef2, os, g, tstride);
        else if constexpr (std::is_same<T, float>::value)
            bn_relu_bwd_apply_kernel<T, 4><<<grid, 256, 0, stream>>>(xs, ds, mean, rstd, scale, shift, coef1, coef2, os, g, tstride);
        else
            bn_relu_bwd_apply_kernel<T, 8><<<grid, 256, 0, stream>>>(xs, ds, mean, rstd, scale, shift, coef1, coef2, os, g, tstride);
    };
    if (dtype_fp32)
        go(float(), pick_vec<float>(C, {x, dy, dx}));
    else
        go(__nv_bfloat16(), pick_vec<__nv_bfloat16>(C, {x, dy, dx}));
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// ---- 2x2 max-pool (nn.MaxPool2d(2), unet.py:81): floor(H/2) x floor(W/2) ----
template <typename T, int V>
__global__ void __launch_bounds__(256) maxpool2_fwd_kernel(const T* __restrict__ x, T* __restrict__ y, long long nvec,
                                                           int H, int W, int Ho, int Wo, int CV) {
    for (long long v = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; v < nvec;
         v += static_cast<long long>(gridDim.x) * blockDim.x) {
        long long r = v;
        const int cv = static_cast<int>(r % CV);
        r /= CV;
        const int wo = static_cast<int>(r % Wo);
        r /= Wo;
        const int ho = static_cast<int>(r % Ho);
        const long long img = r / Ho;
        const T* base = x + (((img * H + 2 * ho) * W + 2 * wo) * CV + cv) * V;
        float a[V], b[V], c[V], d[V];
        ldv<T, V>(base, a);
        ldv<T, V>(base + static_cast<long long>(CV) * V, b);
        ldv<T, V>(base + static_cast<long long>(W) * CV * V, c);
        ldv<T, V>(base + static_cast<long long>(W + 1) * CV * V, d);
#pragma unroll
        for (int j = 0; j < V; ++j) a[j] = fmaxf(fmaxf(a[j], b[j]), fmaxf(c[j], d[j]));
        stv<T, V>(y + v * V, a);
    }
}

int launch_maxpool2_fwd(const void* x, void* y, long long IMG, int H, int W, int C, int dtype_fp32,
                        cudaStream_t stream) {
    const int Ho = H / 2, Wo = W / 2;
    if (Ho == 0 || Wo == 0) return B200_OK;
    auto go = [&](auto tag, int V) {
        using T = decltype(tag);
        const long long nvec = IMG * Ho * Wo * (C / V);
        const unsigned grid = grid_for(nvec, 256 * 2, num_sms() * 16);
        const T* xs = static_cast<const T*>(x);
        T* ys = static_cast<T*>(y);
        if (V == 1)
            maxpool2_fwd_kernel<T, 1><<<grid, 256, 0, stream>>>(xs, ys, nvec, H, W, Ho, Wo, C);
        else if constexpr (std::is_same<T, float>::value)
            maxpool2_fwd_kernel<T, 4><<<grid, 256, 0, stream>>>(xs, ys, nvec, H, W, Ho, Wo, C / 4);
        else
            maxpool2_fwd_kernel<T, 8><<<grid, 256, 0, stream>>>(xs, ys, nvec, H, W, Ho, Wo, C / 8);
    };
    if (dtype_fp32)
        go(float(), pick_vec<float>(C, {x, y}));
    else
        go(__nv_bfloat16(), pick_vec<__nv_bfloat16>(C, {x, y}));
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// Backward: the FIRST maximum in window scan order (0,0),(0,1),(1,0),(1,1) receives the gradient
// (ATen max_pool2d_with_indices).  dx (+)= routed gradient; rows/columns beyond 2*Ho / 2*Wo are
// untouched (the caller zero-fills dx when not accumulating and H or W is odd).
template <typename T, int V>
__global__ void __launch_bounds__(256) maxpool2_bwd_kernel(const T* __restrict__ x, const T* __restrict__ dy,
                                                           T* __restrict__ dx, long long nvec, int H, int W, int Ho,
                                                           int Wo, int CV, int accumulate) {
    for (long long v = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; v < nvec;
         v += static_cast<long long>(gridDim.x) * blockDim.x) {
        long long r = v;
        const int cv = static_cast<int>(r % CV);
        r /= CV;
        const int wo = static_cast<int>(r % Wo);
        r /= Wo;
        const int ho = static_cast<int>(r % Ho);
        const long long img = r / Ho;
        const long long o00 = (((img * H + 2 * ho) * W + 2 * wo) * CV + cv) * V;
        const long long offs[4] = {o00, o00 + static_cast<long long>(CV) * V, o00 + static_cast<long long>(W) * CV * V,
                                   o00 + static_cast<long long>(W + 1) * CV * V};
        float q[4][V], g[V];
#pragma unroll
        for (int k = 0; k < 4; ++k) ldv<T, V>(x + offs[k], q[k]);
        ldv<T, V>(dy + v * V, g);
        int arg[V];
#pragma unroll
        for (int j = 0; j < V; ++j) {
            float m = q[0][j];
            int a = 0;
#pragma unroll
            for (int k = 1; k < 4; ++k)
                if (q[k][j] > m) {
                    m = q[k][j];
                    a = k;
                }
            arg[j] = a;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float o[V];
            if (accumulate) ldv<T, V>(dx + offs[k], o);
#pragma unroll
            for (int j = 0; j < V; ++j) {
                const float add = arg[j] == k ? g[j] : 0.f;
                o[j] = accumulate ? o[j] + add : add;
            }
            stv<T, V>(dx + offs[k], o);
        }
    }
}

int launch_maxpool2_bwd(const void* x, const void* dy, void* dx, long long IMG, int H, int W, int C, int accumulate,
                        int dtype_fp32, cudaStream_t stream) {
    const int Ho = H / 2, Wo = W / 2;
    const size_t esz = dtype_fp32 ? 4 : 2;
    if (!accumulate && ((H & 1) || (W & 1)))
        B200_CUDA_CHECK(cudaMemsetAsync(dx, 0, static_cast<size_t>(IMG) * H * W * C * esz, stream));
    if (Ho == 0 || Wo == 0) return B200_OK;
    auto go = [&](auto tag, int V) {
        using T = decltype(tag);
        const long long nvec = IMG * Ho * Wo * (C / V);
        const unsigned grid = grid_for(nvec, 256, num_sms() * 16);
        const T* xs = static_cast<const T*>(x);
        const T* ds = static_cast<const T*>(dy);
        T* os = static_cast<T*>(dx);
        if (V == 1)
            maxpool2_bwd_kernel<T, 1><<<grid, 256, 0, stream>>>(xs, ds, os, nvec, H, W, Ho, Wo, C, accumulate);
        else if constexpr (std::is_same<T, float>::value)
            maxpool2_bwd_kernel<T, 4><<<grid, 256, 0, stream>>>(xs, ds, os, nvec, H, W, Ho, Wo, C / 4, accumulate);
        else
            maxpool2_bwd_kernel<T, 8><<<grid, 256, 0, stream>>>(xs, ds, os, nvec, H, W, Ho, Wo, C / 8, accumulate);
    };
    if (dtype_fp32)
        go(float(), pick_vec<float>(C, {x, dy, dx}));
    else
        go(__nv_bfloat16(), pick_vec<__nv_bfloat16>(C, {x, dy, dx}));
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// ------------------------------------------------------------------------------------------------
// BatchNorm + ReLU + 2x2 max-pool in ONE pass, forward and backward: the DoubleConv output of an encoder stage
// feeds a skip connection AND the MaxPool2d of the next Down (unet.py:70-71, 81, 179-182).  Separately that is
// apply (read z, write y) + pool (read y, write pooled) forward and pool-backward (read y, g_skip, g_pool, write g) +
// BatchNorm-backward sums (read z, g) + apply (read z, g, write dz) backward: 3.25 + 8.25 passes over the full-size
// tensor; fused it is 2.25 + 5.5.  A "row" of the row loop is one 2x2 window (H and W even; the host falls back to
// the separate kernels otherwise).  Results are bit-identical to the separate kernels: the maximum is taken over
// the values as they are STORED (rounded to T), ties go to the first pixel in scan order (ATen
// max_pool2d_with_indices), and the summed gradient g_skip + routed g_pool is rounded to T like the stored one was.
// ------------------------------------------------------------------------------------------------
struct WinGeom {
    int H, W, Ho, Wo;  // Ho = H / 2, Wo = W / 2
    long long P;       // pixels per timestep = B * H * W
    long long Pw;      // windows per timestep = B * Ho * Wo
    int C;
};

// window w of a timestep -> index of its top-left pixel inside that timestep
__device__ __forceinline__ long long win_pixel(long long w, const WinGeom& q) {
    const long long r = w / q.Wo;
    const int wo = static_cast<int>(w - r * q.Wo);
    const long long b = r / q.Ho;
    const int ho = static_cast<int>(r - b * q.Ho);
    return (b * q.H + 2 * ho) * q.W + 2 * wo;
}

// v as a store to T rounds it
template <typename T>
__device__ __forceinline__ float as_stored(float v) {
    if constexpr (std::is_same<T, float>::value)
        return v;
    else
        return __bfloat162float(__float2bfloat16_rn(v));
}

template <typename T, int V>
__global__ void __launch_bounds__(256) bn_relu_apply_pool_kernel(const T* __restrict__ x, const float* __restrict__ scale,
                                                                 const float* __restrict__ shift, T* __restrict__ y,
                                                                 T* __restrict__ pooled, const ReduceGeom g,
                                                                 const WinGeom q, int tstride) {
    const int tid = threadIdx.x;
    const int r = tid / g.cvb;
    const int cv = tid - r * g.cvb;
    const int c = (blockIdx.y * g.cvb + cv) * V;
    const int t = blockIdx.z;
    if (r >= g.rows_per_iter || c >= g.C) return;
    float sc[V], sh[V];
#pragma unroll
    for (int j = 0; j < V; ++j) {
        sc[j] = __ldg(scale + t * tstride + c + j);
        sh[j] = __ldg(shift + t * tstride + c + j);
    }
    const long long w_begin = static_cast<long long>(blockIdx.x) * g.rows_per_block;
    long long w_end = w_begin + g.rows_per_block;
    if (w_end > g.P) w_end = g.P;
    const long long base = static_cast<long long>(t) * q.P;
    const long long wbase = static_cast<long long>(t) * q.Pw;
    const long long dk[4] = {0, q.C, static_cast<long long>(q.W) * q.C, static_cast<long long>(q.W + 1) * q.C};
#pragma unroll 2
    for (long long w = w_begin + r; w < w_end; w += g.rows_per_iter) {
        const long long off = (base + win_pixel(w, q)) * q.C + c;
        RawVec<T, V> rx[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) ld_raw<T, V>(x + off + dk[k], rx[k]);
        float m[V];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float f[V];
            unpack_raw<T, V>(rx[k], f);
#pragma unroll
            for (int j = 0; j < V; ++j) {
                f[j] = fmaxf(fmaf(f[j], sc[j], sh[j]), 0.f);
                m[j] = k == 0 ? f[j] : fmaxf(m[j], f[j]);  // rounding is monotonic: max of the stored = stored max
            }
            stv<T, V>(y + off + dk[k], f);
        }
        stv<T, V>(pooled + (wbase + w) * q.C + c, m);
    }
}

static WinGeom win_geom(long long B, int H, int W, int C) {
    WinGeom q;
    q.H = H; q.W = W; q.Ho = H / 2; q.Wo = W / 2;
    q.P = B * H * W;
    q.Pw = B * q.Ho * q.Wo;
    q.C = C;
    return q;
}

int launch_bn_relu_apply_pool(const void* x, const float* scale, const float* shift, void* y, void* pooled, int T_,
                              long long B, int H, int W, int C, int tstride, int dtype_fp32, cudaStream_t stream) {
    const WinGeom q = win_geom(B, H, W, C);
    auto go = [&](auto tag, int V) {
        using T = decltype(tag);
        dim3 grid;
        const ReduceGeom g = rowloop_geom(T_, q.Pw, C, V, &grid);
        const T* xs = static_cast<const T*>(x);
        T* ys = static_cast<T*>(y);
        T* ps = static_cast<T*>(pooled);
        if (V == 1)
            bn_relu_apply_pool_kernel<T, 1><<<grid, 256, 0, stream>>>(xs, scale, shift, ys, ps, g, q, tstride);
        else if constexpr (std::is_same<T, float>::value)
            bn_relu_apply_pool_kernel<T, 4><<<grid, 256, 0, stream>>>(xs, scale, shift, ys, ps, g, q, tstride);
        else
            bn_relu_apply_pool_kernel<T, 8><<<grid, 256, 0, stream>>>(xs, scale, shift, ys, ps, g, q, tstride);
    };
    if (dtype_fp32)
        go(float(), pick_vec<float>(C, {x, y, pooled}));
    else
        go(__nv_bfloat16(), pick_vec<__nv_bfloat16>(C, {x, y, pooled}));
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// The gradient that reaches the ReLU output of the four pixels of a window: g_k = stored(g_skip_k + [k == argmax] g_pool)
// (g_skip may be absent).  arg[] is found on the stored activations, exactly as maxpool2_bwd_kernel finds it on y.
// Returns the argmax of channel j in bits [2j, 2j+2).
template <typename T, int V>
__device__ __forceinline__ unsigned window_argmax(const RawVec<T, V> (&rx)[4], const float (&sc)[V], const float (&sh)[V]) {
    float best[V];
    int arg[V];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        float f[V];
        unpack_raw<T, V>(rx[k], f);
#pragma unroll
        for (int j = 0; j < V; ++j) {
            const float yv = as_stored<T>(fmaxf(fmaf(f[j], sc[j], sh[j]), 0.f));
            if (k == 0) {
                best[j] = yv;
                arg[j] = 0;
            } else if (yv > best[j]) {
                best[j] = yv;
                arg[j] = k;
            }
        }
    }
    unsigned bits = 0;
#pragma unroll
    for (int j = 0; j < V; ++j) bits |= static_cast<unsigned>(arg[j]) << (2 * j);
    return bits;
}

struct BnBwdReducePoolOp {
    const void* x;    // pre-BN conv output [T][P][C]
    const void* dy;   // gradient w.r.t. the ReLU output through the skip connection, or nullptr
    const void* dp;   // gradient w.r.t. the pooled output [T][Pw][C]
    const float* mean;
    const float* rstd;
    const float* scale;
    const float* shift;
    WinGeom q;
    int tstride;
    template <int V>
    struct State {
        float sc[V], sh[V];
    };
    template <int V>
    __device__ __forceinline__ void init(int t, int c, State<V>& st) const {
#pragma unroll
        for (int j = 0; j < V; ++j) {
            const int i = t * tstride + c + j;
            st.sc[j] = __ldg(scale + i);
            st.sh[j] = __ldg(shift + i);
        }
    }
    __device__ __forceinline__ void post(int t, int c, double& s0, double& s1) const {
        const int i = t * tstride + c;
        s1 = static_cast<double>(__ldg(rstd + i)) * (s1 - static_cast<double>(__ldg(mean + i)) * s0);
    }
    template <typename T, int V>
    struct Frag {
        RawVec<T, V> x[4], d[4], p;
    };
    template <typename T, int V>
    __device__ __forceinline__ void load(Frag<T, V>& fr, int t, long long w, int c) const {
        const long long off = (static_cast<long long>(t) * q.P + win_pixel(w, q)) * q.C + c;
        const long long dk[4] = {0, q.C, static_cast<long long>(q.W) * q.C, static_cast<long long>(q.W + 1) * q.C};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            ld_raw<T, V>(static_cast<const T*>(x) + off + dk[k], fr.x[k]);
            if (dy) {
                ld_raw<T, V>(static_cast<const T*>(dy) + off + dk[k], fr.d[k]);
            } else {
#pragma unroll
                for (int i = 0; i < RawVec<T, V>::NW; ++i) fr.d[k].w[i] = 0u;
            }
        }
        ld_raw<T, V>(static_cast<const T*>(dp) + (static_cast<long long>(t) * q.Pw + w) * q.C + c, fr.p);
    }
    template <typename T, int V, typename Acc>
    __device__ __forceinline__ void accum(const State<V>& st, const Frag<T, V>& fr, Acc (&a0)[V], Acc (&a1)[V]) const {
        const unsigned arg = window_argmax<T, V>(fr.x, st.sc, st.sh);
        float fp[V];
        unpack_raw<T, V>(fr.p, fp);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float fx[V], fd[V];
            unpack_raw<T, V>(fr.x[k], fx);
            unpack_raw<T, V>(fr.d[k], fd);
#pragma unroll
            for (int j = 0; j < V; ++j) {
                const float gk = as_stored<T>(fd[j] + (((arg >> (2 * j)) & 3u) == static_cast<unsigned>(k) ? fp[j] : 0.f));
                const float yv = fmaf(fx[j], st.sc[j], st.sh[j]);
                const float gq = yv > 0.f ? gk : 0.f;
                a0[j] += Acc(gq);
                a1[j] += Acc(gq) * Acc(fx[j]);
            }
        }
    }
};
template <>
struct ColredTraits<BnBwdReducePoolOp> {
    static constexpr int U = 1;
    static constexpr int BLOCKS = 2;
};

int launch_bn_relu_pool_bwd_reduce(const void* x, const void* dy, const void* dp, const float* mean, const float* rstd,
                                   const float* scale, const float* shift, int T_, long long B, int H, int W, int C,
                                   int tstride, int dtype_fp32, double* sum_g, double* sum_gx, cudaStream_t stream) {
    B200_CUDA_CHECK(cudaMemsetAsync(sum_g, 0, sizeof(double) * T_ * C, stream));
    B200_CUDA_CHECK(cudaMemsetAsync(sum_gx, 0, sizeof(double) * T_ * C, stream));
    BnBwdReducePoolOp op{x, dy, dp, mean, rstd, scale, shift, win_geom(B, H, W, C), tstride};
    if (dtype_fp32)
        return launch_colreduce<float>(op, T_, op.q.Pw, C, pick_vec<float>(C, {x, dy, dp}), sum_g, sum_gx, stream);
    return launch_colreduce<__nv_bfloat16>(op, T_, op.q.Pw, C, pick_vec<__nv_bfloat16>(C, {x, dy, dp}), sum_g, sum_gx, stream);
}

// dz of the four pixels of each window: dx = scale * g + ka * x + kb as in bn_relu_bwd_apply_kernel
template <typename T, int V>
__global__ void __launch_bounds__(256, 2)
bn_relu_pool_bwd_apply_kernel(const T* __restrict__ x, const T* __restrict__ dy, const T* __restrict__ dp,
                              const float* __restrict__ mean, const float* __restrict__ rstd,
                              const float* __restrict__ scale, const float* __restrict__ shift,
                              const float* __restrict__ coef1, const float* __restrict__ coef2, T* __restrict__ dx,
                              const ReduceGeom g, const WinGeom q, int tstride) {
    const int tid = threadIdx.x;
    const int r = tid / g.cvb;
    const int cv = tid - r * g.cvb;
    const int c = (blockIdx.y * g.cvb + cv) * V;
    const int t = blockIdx.z;
    if (r >= g.rows_per_iter || c >= g.C) return;
    float sc[V], sh[V], ka[V], kb[V];
#pragma unroll
    for (int j = 0; j < V; ++j) {
        const int ps = t * tstride + c + j, pc = t * g.C + c + j;
        sc[j] = __ldg(scale + ps);
        sh[j] = __ldg(shift + ps);
        const float rc2 = __ldg(rstd + ps) * __ldg(coef2 + pc);
        ka[j] = -sc[j] * rc2;
        kb[j] = sc[j] * (rc2 * __ldg(mean + ps) - __ldg(coef1 + pc));
    }
    const long long w_begin = static_cast<long long>(blockIdx.x) * g.rows_per_block;
    long long w_end = w_begin + g.rows_per_block;
    if (w_end > g.P) w_end = g.P;
    const long long base = static_cast<long long>(t) * q.P;
    const long long wbase = static_cast<long long>(t) * q.Pw;
    const long long dk[4] = {0, q.C, static_cast<long long>(q.W) * q.C, static_cast<long long>(q.W + 1) * q.C};
    for (long long w = w_begin + r; w < w_end; w += g.rows_per_iter) {
        const long long off = (base + win_pixel(w, q)) * q.C + c;
        RawVec<T, V> rx[4], rd[4], rp;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            ld_raw<T, V>(x + off + dk[k], rx[k]);
            if (dy) {
                ld_raw<T, V>(dy + off + dk[k], rd[k]);
            } else {
#pragma unroll
                for (int i = 0; i < RawVec<T, V>::NW; ++i) rd[k].w[i] = 0u;
            }
        }
        ld_raw<T, V>(dp + (wbase + w) * q.C + c, rp);
        const unsigned arg = window_argmax<T, V>(rx, sc, sh);
        float fp[V];
        unpack_raw<T, V>(rp, fp);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float fx[V], fd[V];
            unpack_raw<T, V>(rx[k], fx);
            unpack_raw<T, V>(rd[k], fd);
#pragma unroll
            for (int j = 0; j < V; ++j) {
                const float gk = as_stored<T>(fd[j] + (((arg >> (2 * j)) & 3u) == static_cast<unsigned>(k) ? fp[j] : 0.f));
                const float yv = fmaf(fx[j], sc[j], sh[j]);
                const float gq = yv > 0.f ? gk : 0.f;
                fd[j] = fmaf(sc[j], gq, fmaf(ka[j], fx[j], kb[j]));
            }
            stv<T, V>(dx + off + dk[k], fd);
        }
    }
}

int launch_bn_relu_pool_bwd_apply(const void* x, const void* dy, const void* dp, const float* mean, const float* rstd,
                                  const float* scale, const float* shift, const float* coef1, const float* coef2,
                                  void* dx, int T_, long long B, int H, int W, int C, int tstride, int dtype_fp32,
                                  cudaStream_t stream) {
    const WinGeom q = win_geom(B, H, W, C);
    auto go = [&](auto tag, int V) {
        using T = decltype(tag);
        dim3 grid;
        const ReduceGeom g = rowloop_geom(T_, q.Pw, C, V, &grid);
        const T* xs = static_cast<const T*>(x);
        const T* ds = static_cast<const T*>(dy);
        const T* ps = static_cast<const T*>(dp);
        T* os = static_cast<T*>(dx);
        if (V == 1)
            bn_relu_pool_bwd_apply_kernel<T, 1><<<grid, 256, 0, stream>>>(xs, ds, ps, mean, rstd, scale, shift, coef1, coef2, os, g, q, tstride);
        else if constexpr (std::is_same<T, float>::value)
            bn_relu_pool_bwd_apply_kernel<T, 4><<<grid, 256, 0, stream>>>(xs, ds, ps, mean, rstd, scale, shift, coef1, coef2, os, g, q, tstride);
        else
            bn_relu_pool_bwd_apply_kernel<T, 8><<<grid, 256, 0, stream>>>(xs, ds, ps, mean, rstd, scale, shift, coef1, coef2, os, g, q, tstride);
    };
    if (dtype_fp32)
        go(float(), pick_vec<float>(C, {x, dy, dp, dx}));
    else
        go(__nv_bfloat16(), pick_vec<__nv_bfloat16>(C, {x, dy, dp, dx}));
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// ------------------------------------------------------------------------------------------------
// BatchNorm + ReLU + the 1x1 output convolution in one pass (the last DoubleConv feeds OutConv with out_channels = 1,
// unet.py:70-71 -> :104, :202-203).  Forward: out[p] = b + sum_c relu(x*scale+shift)[p][c] * w[c]; the 64-channel
// full-resolution activation is NEVER written.  Backward: the data gradient of the 1x1 convolution is the rank-1
// product dout[p] * w[c], so the BatchNorm-backward passes form it on the fly instead of reading a stored tensor, and
// the weight gradient dw[c] = sum_p dout[p] * y[p][c] rides along in the reduction pass with y recomputed.  Separately
// that is apply (r + w) + outconv (r) forward and outconv wgrad (r) + dgrad (w) + BatchNorm sums (2r) + apply (2r + w)
// backward = 10 passes over the largest activation tensor of the network; fused it is 1 + 1 + 2.  The activation and the
// data gradient of the 1x1 convolution are never stored, so they are not rounded to T either (the separate kernels round
// both to bf16 on the way through HBM): the fused results sit closer to exact arithmetic by those two roundings.
// A pixel's C / V channel vectors sit in C / V consecutive lanes (a power of two <= 32).
// ------------------------------------------------------------------------------------------------
template <typename T, int V>
__global__ void __launch_bounds__(256) bn_relu_outconv_fwd_kernel(const T* __restrict__ x, const float* __restrict__ scale,
                                                                  const float* __restrict__ shift, const float* __restrict__ w,
                                                                  const float* __restrict__ b, float* __restrict__ out,
                                                                  const ReduceGeom g, int tstride) {
    const int tid = threadIdx.x;
    const int r = tid / g.cvb;       // g.cvb == C / V divides 32: the lanes of one pixel are one aligned shuffle group
    const int cv = tid - r * g.cvb;
    const int c = cv * V;
    const int t = blockIdx.z;
    float sc[V], sh[V], wv[V];
#pragma unroll
    for (int j = 0; j < V; ++j) {
        sc[j] = __ldg(scale + t * tstride + c + j);
        sh[j] = __ldg(shift + t * tstride + c + j);
        wv[j] = __ldg(w + c + j);
    }
    const float bias = b ? __ldg(b) : 0.f;
    const long long p_begin = static_cast<long long>(blockIdx.x) * g.rows_per_block;
    long long p_end = p_begin + g.rows_per_block;
    if (p_end > g.P) p_end = g.P;
    const long long base = static_cast<long long>(t) * g.P;
    constexpr int U = 4;
    const long long step = g.rows_per_iter;
    // block-uniform trip count: every lane takes part in the shuffles
    for (long long p0 = p_begin; p0 < p_end; p0 += U * step) {
        RawVec<T, V> rx[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long p = p0 + u * step + r;
            if (p < p_end) ld_raw<T, V>(x + (base + p) * g.C + c, rx[u]);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long p = p0 + u * step + r;
            float acc = 0.f;
            if (p < p_end) {
                float f[V];
                unpack_raw<T, V>(rx[u], f);
#pragma unroll
                for (int j = 0; j < V; ++j) acc = fmaf(fmaxf(fmaf(f[j], sc[j], sh[j]), 0.f), wv[j], acc);
            }
            for (int s = g.cvb >> 1; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
            if (p < p_end && cv == 0) out[base + p] = acc + bias;
        }
    }
}

static bool outconv_fusable(int C, int V) {
    const int cv = C / V;
    return C % V == 0 && cv >= 1 && cv <= 32 && (cv & (cv - 1)) == 0;
}

// rows per block for the pixel-group kernels: cvb = C / V exactly (no idle threads), grid ~16 blocks per SM
static ReduceGeom pixgroup_geom(int T_, long long P, int C, int V, dim3* grid) {
    ReduceGeom g;
    g.T = T_;
    g.P = P;
    g.C = C;
    g.cvb = C / V;
    g.rows_per_iter = 256 / g.cvb;
    long long want_x = (16LL * num_sms() + T_ - 1) / T_;
    long long max_x = (P + 8LL * g.rows_per_iter - 1) / (8LL * g.rows_per_iter);
    if (want_x > max_x) want_x = max_x;
    if (want_x < 1) want_x = 1;
    g.rows_per_block = (P + want_x - 1) / want_x;
    *grid = dim3(static_cast<unsigned>((P + g.rows_per_block - 1) / g.rows_per_block), 1, T_);
    return g;
}

int launch_bn_relu_outconv_fwd(const void* x, const float* scale, const float* shift, const float* w, const float* b,
                               float* out, int T_, long long P, int C, int tstride, int dtype_fp32, cudaStream_t stream) {
    auto go = [&](auto tag, int V) -> int {
        using T = decltype(tag);
        if (!outconv_fusable(C, V)) {
            set_last_error("b200_bn_relu_outconv_fwd: C / %d must be a power of two <= 32 (C = %d)", V, C);
            return B200_ERR_SHAPE;
        }
        dim3 grid;
        const ReduceGeom g = pixgroup_geom(T_, P, C, V, &grid);
        const T* xs = static_cast<const T*>(x);
        if (V == 1)
            bn_relu_outconv_fwd_kernel<T, 1><<<grid, 256, 0, stream>>>(xs, scale, shift, w, b, out, g, tstride);
        else if constexpr (std::is_same<T, float>::value)
            bn_relu_outconv_fwd_kernel<T, 4><<<grid, 256, 0, stream>>>(xs, scale, shift, w, b, out, g, tstride);
        else
            bn_relu_outconv_fwd_kernel<T, 8><<<grid, 256, 0, stream>>>(xs, scale, shift, w, b, out, g, tstride);
        return B200_OK;
    };
    const int rc = dtype_fp32 ? go(float(), pick_vec<float>(C, {x})) : go(__nv_bfloat16(), pick_vec<__nv_bfloat16>(C, {x}));
    if (rc != B200_OK) return rc;
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// sum_g[t][c] = sum_p g, sum_gx[t][c] = sum_p g * xhat (as BnBwdReduceOp) with g = dout[p] * w[c] * [relu active], and
// dw[c] += sum_p dout[p] * y[p][c] over ALL t.  Same block / thread layout as colreduce_kernel.  One 16-byte vector and
// one scalar per row: eight rows in flight per thread at two blocks per SM (ncu of the first version, four rows at
// three blocks: 2.7 TB/s with the warps waiting on their loads).
template <typename T, int V, typename Acc>
__global__ void __launch_bounds__(256, 2)
bn_relu_outconv_bwd_reduce_kernel(const T* __restrict__ x, const float* __restrict__ dout, const float* __restrict__ w,
                                  const float* __restrict__ mean, const float* __restrict__ rstd,
                                  const float* __restrict__ scale, const float* __restrict__ shift, const ReduceGeom g,
                                  int tstride, double* __restrict__ sum_g, double* __restrict__ sum_gx,
                                  double* __restrict__ sum_dw) {
    constexpr int HV = V > 4 ? 4 : V;
    __shared__ Acc red[3][256 * HV];
    const int tid = threadIdx.x;
    const int r = tid / g.cvb;
    const int cv = tid - r * g.cvb;
    const int c = cv * V;
    const int t = blockIdx.z;
    const long long p_begin = static_cast<long long>(blockIdx.x) * g.rows_per_block;
    long long p_end = p_begin + g.rows_per_block;
    if (p_end > g.P) p_end = g.P;
    const long long base = static_cast<long long>(t) * g.P;
    float sc[V], sh[V], wv[V];
    Acc a0[V], a1[V], a2[V];
#pragma unroll
    for (int j = 0; j < V; ++j) {
        sc[j] = __ldg(scale + t * tstride + c + j);
        sh[j] = __ldg(shift + t * tstride + c + j);
        wv[j] = __ldg(w + c + j);
        a0[j] = a1[j] = a2[j] = Acc(0);
    }
    auto accum = [&](const RawVec<T, V>& rx, float d) {
        float fx[V];
        unpack_raw<T, V>(rx, fx);
#pragma unroll
        for (int j = 0; j < V; ++j) {
            const float yv = fmaf(fx[j], sc[j], sh[j]);
            const float gq = yv > 0.f ? d * wv[j] : 0.f;
            a0[j] += Acc(gq);
            a1[j] += Acc(gq) * Acc(fx[j]);
            a2[j] += Acc(d) * Acc(fmaxf(yv, 0.f));
        }
    };
    constexpr int U = 8;
    const long long step = g.rows_per_iter;
    long long p = p_begin + r;
    for (; p + (U - 1) * step < p_end; p += U * step) {
        RawVec<T, V> rx[U];
        float d[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            ld_raw<T, V>(x + (base + p + u * step) * g.C + c, rx[u]);
            d[u] = __ldg(dout + base + p + u * step);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) accum(rx[u], d[u]);
    }
    for (; p < p_end; p += step) {
        RawVec<T, V> rx;
        ld_raw<T, V>(x + (base + p) * g.C + c, rx);
        accum(rx, __ldg(dout + base + p));
    }
#pragma unroll
    for (int half = 0; half < V / HV; ++half) {
        __syncthreads();
#pragma unroll
        for (int j = 0; j < HV; ++j) {
            red[0][tid * HV + j] = a0[half * HV + j];
            red[1][tid * HV + j] = a1[half * HV + j];
            red[2][tid * HV + j] = a2[half * HV + j];
        }
        __syncthreads();
        if (r == 0) {
#pragma unroll
            for (int j = 0; j < HV; ++j) {
                double s0 = 0.0, s1 = 0.0, s2 = 0.0;
                for (int rr = 0; rr < g.rows_per_iter; ++rr) {
                    s0 += static_cast<double>(red[0][(rr * g.cvb + cv) * HV + j]);
                    s1 += static_cast<double>(red[1][(rr * g.cvb + cv) * HV + j]);
                    s2 += static_cast<double>(red[2][(rr * g.cvb + cv) * HV + j]);
                }
                const int cc = c + half * HV + j;
                const int i = t * tstride + cc;
                s1 = static_cast<double>(__ldg(rstd + i)) * (s1 - static_cast<double>(__ldg(mean + i)) * s0);
                atomicAdd(sum_g + static_cast<long long>(t) * g.C + cc, s0);
                atomicAdd(sum_gx + static_cast<long long>(t) * g.C + cc, s1);
                atomicAdd(sum_dw + cc, s2);
            }
        }
    }
}

int launch_bn_relu_outconv_bwd_reduce(const void* x, const float* dout, const float* w, const float* mean, const float* rstd,
                                      const float* scale, const float* shift, int T_, long long P, int C, int tstride,
                                      int dtype_fp32, double* sum_g, double* sum_gx, double* sum_dw, float* dw,
                                      cudaStream_t stream) {
    B200_CUDA_CHECK(cudaMemsetAsync(sum_g, 0, sizeof(double) * T_ * C, stream));
    B200_CUDA_CHECK(cudaMemsetAsync(sum_gx, 0, sizeof(double) * T_ * C, stream));
    B200_CUDA_CHECK(cudaMemsetAsync(sum_dw, 0, sizeof(double) * C, stream));
    auto go = [&](auto tag, int V) -> int {
        using T = decltype(tag);
        using Acc = typename std::conditional<std::is_same<T, float>::value, double, float>::type;
        if (!outconv_fusable(C, V)) {
            set_last_error("b200_bn_relu_outconv_bwd_reduce: C / %d must be a power of two <= 32 (C = %d)", V, C);
            return B200_ERR_SHAPE;
        }
        ReduceGeom g;
        g.T = T_; g.P = P; g.C = C;
        g.cvb = C / V;
        g.rows_per_iter = 256 / g.cvb;
        // two full waves at two resident blocks per SM, at least 8 iterations per thread (see launch_colreduce)
        long long want_x = (4LL * num_sms()) / T_;
        long long max_x = (P + 8LL * g.rows_per_iter - 1) / (8LL * g.rows_per_iter);
        if (want_x > max_x) want_x = max_x;
        if (want_x < 1) want_x = 1;
        g.rows_per_block = (P + want_x - 1) / want_x;
        dim3 grid(static_cast<unsigned>((P + g.rows_per_block - 1) / g.rows_per_block), 1, T_);
        const T* xs = static_cast<const T*>(x);
        if (V == 1)
            bn_relu_outconv_bwd_reduce_kernel<T, 1, Acc><<<grid, 256, 0, stream>>>(xs, dout, w, mean, rstd, scale, shift, g, tstride, sum_g, sum_gx, sum_dw);
        else if constexpr (std::is_same<T, float>::value)
            bn_relu_outconv_bwd_reduce_kernel<T, 4, Acc><<<grid, 256, 0, stream>>>(xs, dout, w, mean, rstd, scale, shift, g, tstride, sum_g, sum_gx, sum_dw);
        else
            bn_relu_outconv_bwd_reduce_kernel<T, 8, Acc><<<grid, 256, 0, stream>>>(xs, dout, w, mean, rstd, scale, shift, g, tstride, sum_g, sum_gx, sum_dw);
        return B200_OK;
    };
    const int rc = dtype_fp32 ? go(float(), pick_vec<float>(C, {x})) : go(__nv_bfloat16(), pick_vec<__nv_bfloat16>(C, {x}));
    if (rc != B200_OK) return rc;
    B200_CUDA_CHECK(cudaGetLastError());
    return dw ? launch_cast_double(sum_dw, dw, C, 0, stream) : B200_OK;
}

// dx = scale * g + ka * x + kb as bn_relu_bwd_apply_kernel, g = stored(dout[p] * w[c]) where the ReLU is active
template <typename T, int V>
__global__ void __launch_bounds__(256, (std::is_same<T, float>::value ? 2 : 3))
bn_relu_outconv_bwd_apply_kernel(const T* __restrict__ x, const float* __restrict__ dout, const float* __restrict__ w,
                                 const float* __restrict__ mean, const float* __restrict__ rstd,
                                 const float* __restrict__ scale, const float* __restrict__ shift,
                                 const float* __restrict__ coef1, const float* __restrict__ coef2, T* __restrict__ dx,
                                 const ReduceGeom g, int tstride) {
    const int tid = threadIdx.x;
    const int r = tid / g.cvb;
    const int cv = tid - r * g.cvb;
    const int c = (blockIdx.y * g.cvb + cv) * V;
    const int t = blockIdx.z;
    if (r >= g.rows_per_iter || c >= g.C) return;
    float sc[V], sh[V], ka[V], kb[V], wv[V];
#pragma unroll
    for (int j = 0; j < V; ++j) {
        const int ps = t * tstride + c + j, pc = t * g.C + c + j;
        sc[j] = __ldg(scale + ps);
        sh[j] = __ldg(shift + ps);
        wv[j] = __ldg(w + c + j);
        const float rc2 = __ldg(rstd + ps) * __ldg(coef2 + pc);
        ka[j] = -sc[j] * rc2;
        kb[j] = sc[j] * (rc2 * __ldg(mean + ps) - __ldg(coef1 + pc));
    }
    const long long p_begin = static_cast<long long>(blockIdx.x) * g.rows_per_block;
    long long p_end = p_begin + g.rows_per_block;
    if (p_end > g.P) p_end = g.P;
    const long long base = static_cast<long long>(t) * g.P;
    auto apply = [&](const RawVec<T, V>& rx, float d, long long off) {
        float fx[V], fd[V];
        unpack_raw<T, V>(rx, fx);
#pragma unroll
        for (int j = 0; j < V; ++j) {
            const float yv = fmaf(fx[j], sc[j], sh[j]);
            const float gq = yv > 0.f ? d * wv[j] : 0.f;
            fd[j] = fmaf(sc[j], gq, fmaf(ka[j], fx[j], kb[j]));
        }
        stv<T, V>(dx + off, fd);
    };
    constexpr int U = 4;
    const long long step = g.rows_per_iter;
    long long p = p_begin + r;
    for (; p + (U - 1) * step < p_end; p += U * step) {
        RawVec<T, V> rx[U];
        float d[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            ld_raw<T, V>(x + (base + p + u * step) * g.C + c, rx[u]);
            d[u] = __ldg(dout + base + p + u * step);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) apply(rx[u], d[u], (base + p + u * step) * g.C + c);
    }
    for (; p < p_end; p += step) {
        RawVec<T, V> rx;
        ld_raw<T, V>(x + (base + p) * g.C + c, rx);
        apply(rx, __ldg(dout + base + p), (base + p) * g.C + c);
    }
}

int launch_bn_relu_outconv_bwd_apply(const void* x, const float* dout, const float* w, const float* mean, const float* rstd,
                                     const float* scale, const float* shift, const float* coef1, const float* coef2,
                                     void* dx, int T_, long long P, int C, int tstride, int dtype_fp32,
                                     cudaStream_t stream) {
    auto go = [&](auto tag, int V) {
        using T = decltype(tag);
        dim3 grid;
        const ReduceGeom g = rowloop_geom(T_, P, C, V, &grid);
        const T* xs = static_cast<const T*>(x);
        T* os = static_cast<T*>(dx);
        if (V == 1)
            bn_relu_outconv_bwd_apply_kernel<T, 1><<<grid, 256, 0, stream>>>(xs, dout, w, mean, rstd, scale, shift, coef1, coef2, os, g, tstride);
        else if constexpr (std::is_same<T, float>::value)
            bn_relu_outconv_bwd_apply_kernel<T, 4><<<grid, 256, 0, stream>>>(xs, dout, w, mean, rstd, scale, shift, coef1, coef2, os, g, tstride);
        else
            bn_relu_outconv_bwd_apply_kernel<T, 8><<<grid, 256, 0, stream>>>(xs, dout, w, mean, rstd, scale, shift, coef1, coef2, os, g, tstride);
    };
    if (dtype_fp32)
        go(float(), pick_vec<float>(C, {x, dx}));
    else
        go(__nv_bfloat16(), pick_vec<__nv_bfloat16>(C, {x, dx}));
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// ------------------------------------------------------------------------------------------------
// ConvLSTM gate math (ConvLSTMCell.forward, unet.py:29-35) and its BPTT gradient
// ------------------------------------------------------------------------------------------------
template <bool FAST>
__device__ __forceinline__ float act_tanh(float x) {
    if constexpr (FAST) {
        float y;
        asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
        return y;
    } else {
        return tanhf(x);
    }
}
template <bool FAST>
__device__ __forceinline__ float act_sigmoid(float x) {
    if constexpr (FAST)
        return fmaf(0.5f, act_tanh<true>(0.5f * x), 0.5f);
    else
        return 1.f / (1.f + expf(-x));
}

// z: [P][4*Ch] fp32 pre-activations (bias included), gate-major i|f|g|o like the reference's chunk.
// gates: [P][4][Ch] activated; c fp32; h in the storage type.
template <typename T, int V, bool FAST>
__global__ void __launch_bounds__(256) lstm_gates_fwd_kernel(const float* __restrict__ z, const float* __restrict__ c_prev,
                                                             T* __restrict__ gates, float* __restrict__ c_next,
                                                             T* __restrict__ h_next, long long nvec, int Ch) {
    const int CV = Ch / V;
    for (long long v = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; v < nvec;
         v += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long p = v / CV;
        const int c = static_cast<int>(v - p * CV) * V;
        float zi[V], zf[V], zg[V], zo[V], cp[V];
        const float* zr = z + p * 4 * Ch + c;
        ldv<float, V>(zr, zi);
        ldv<float, V>(zr + Ch, zf);
        ldv<float, V>(zr + 2 * Ch, zg);
        ldv<float, V>(zr + 3 * Ch, zo);
        if (c_prev) {
            ldv<float, V>(c_prev + p * Ch + c, cp);
        } else {
#pragma unroll
            for (int j = 0; j < V; ++j) cp[j] = 0.f;
        }
        float cn[V], hn[V];
#pragma unroll
        for (int j = 0; j < V; ++j) {
            zi[j] = act_sigmoid<FAST>(zi[j]);
            zf[j] = act_sigmoid<FAST>(zf[j]);
            zg[j] = act_tanh<FAST>(zg[j]);
            zo[j] = act_sigmoid<FAST>(zo[j]);
            cn[j] = fmaf(zf[j], cp[j], zi[j] * zg[j]);
            hn[j] = zo[j] * act_tanh<FAST>(cn[j]);
        }
        T* gr = gates + p * 4 * Ch + c;
        stv<T, V>(gr, zi);
        stv<T, V>(gr + Ch, zf);
        stv<T, V>(gr + 2 * Ch, zg);
        stv<T, V>(gr + 3 * Ch, zo);
        stv<float, V>(c_next + p * Ch + c, cn);
        stv<T, V>(h_next + p * Ch + c, hn);
    }
}

int launch_lstm_gates_fwd(const float* z, const float* c_prev, void* gates, float* c_next, void* h_next, long long P,
                          int Ch, int dtype_fp32, cudaStream_t stream) {
    if (dtype_fp32) {
        const int V = pick_vec<float>(Ch, {z, c_prev, gates, c_next, h_next});
        const long long nvec = P * (Ch / V);
        const unsigned grid = grid_for(nvec, 256, num_sms() * 16);
        if (V == 4)
            lstm_gates_fwd_kernel<float, 4, false><<<grid, 256, 0, stream>>>(z, c_prev, static_cast<float*>(gates), c_next, static_cast<float*>(h_next), nvec, Ch);
        else
            lstm_gates_fwd_kernel<float, 1, false><<<grid, 256, 0, stream>>>(z, c_prev, static_cast<float*>(gates), c_next, static_cast<float*>(h_next), nvec, Ch);
    } else {
        const int V = pick_vec<__nv_bfloat16>(Ch, {z, c_prev, gates, c_next, h_next});
        const long long nvec = P * (Ch / V);
        const unsigned grid = grid_for(nvec, 256, num_sms() * 16);
        auto* g = static_cast<__nv_bfloat16*>(gates);
        auto* h = static_cast<__nv_bfloat16*>(h_next);
        if (V == 8)
            lstm_gates_fwd_kernel<__nv_bfloat16, 8, true><<<grid, 256, 0, stream>>>(z, c_prev, g, c_next, h, nvec, Ch);
        else
            lstm_gates_fwd_kernel<__nv_bfloat16, 1, true><<<grid, 256, 0, stream>>>(z, c_prev, g, c_next, h, nvec, Ch);
    }
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// Gate gradients of one BPTT step (autograd of unet.py:30-35):
//   dh = dh_a + dh_b;  tc = tanh(c_next);  do = dh*tc;  dc = dc_next + dh*o*(1-tc^2)
//   di = dc*g; dg = dc*i; df = dc*c_prev; dc_prev = dc*f
//   dz = [di*i*(1-i), df*f*(1-f), dg*(1-g^2), do*o*(1-o)]      ([P][4*Ch], gate-major)
template <typename T, int V, bool FAST>
__global__ void __launch_bounds__(256)
lstm_gates_bwd_kernel(const T* __restrict__ gates, const float* __restrict__ c_prev, const float* __restrict__ c_next,
                      const T* __restrict__ dh_a, const T* __restrict__ dh_b, const float* __restrict__ dc_next,
                      T* __restrict__ dz, float* __restrict__ dc_prev, long long nvec, int Ch) {
    const int CV = Ch / V;
    for (long long v = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; v < nvec;
         v += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long p = v / CV;
        const int c = static_cast<int>(v - p * CV) * V;
        float gi[V], gf[V], gg[V], go[V], cp[V], cn[V], dh[V], dc[V];
        const T* gr = gates + p * 4 * Ch + c;
        ldv<T, V>(gr, gi);
        ldv<T, V>(gr + Ch, gf);
        ldv<T, V>(gr + 2 * Ch, gg);
        ldv<T, V>(gr + 3 * Ch, go);
        const long long so = p * Ch + c;
        if (c_prev) {
            ldv<float, V>(c_prev + so, cp);
        } else {
#pragma unroll
            for (int j = 0; j < V; ++j) cp[j] = 0.f;
        }
        ldv<float, V>(c_next + so, cn);
        if (dh_a) {
            ldv<T, V>(dh_a + so, dh);
        } else {
#pragma unroll
            for (int j = 0; j < V; ++j) dh[j] = 0.f;
        }
        if (dh_b) {
            float t2[V];
            ldv<T, V>(dh_b + so, t2);
#pragma unroll
            for (int j = 0; j < V; ++j) dh[j] += t2[j];
        }
        if (dc_next) {
            ldv<float, V>(dc_next + so, dc);
        } else {
#pragma unroll
            for (int j = 0; j < V; ++j) dc[j] = 0.f;
        }
        float zi[V], zf[V], zg[V], zo[V], dcp[V];
#pragma unroll
        for (int j = 0; j < V; ++j) {
            const float tc = act_tanh<FAST>(cn[j]);
            const float d_o = dh[j] * tc;
            const float d_c = fmaf(dh[j] * go[j], 1.f - tc * tc, dc[j]);
            zi[j] = d_c * gg[j] * gi[j] * (1.f - gi[j]);
            zf[j] = d_c * cp[j] * gf[j] * (1.f - gf[j]);
            zg[j] = d_c * gi[j] * (1.f - gg[j] * gg[j]);
            zo[j] = d_o * go[j] * (1.f - go[j]);
            dcp[j] = d_c * gf[j];
        }
        T* zr = dz + p * 4 * Ch + c;
        stv<T, V>(zr, zi);
        stv<T, V>(zr + Ch, zf);
        stv<T, V>(zr + 2 * Ch, zg);
        stv<T, V>(zr + 3 * Ch, zo);
        stv<float, V>(dc_prev + so, dcp);
    }
}

int launch_lstm_gates_bwd(const void* gates, const float* c_prev, const float* c_next, const void* dh_a,
                          const void* dh_b, const float* dc_next, void* dz, float* dc_prev, long long P, int Ch,
                          int dtype_fp32, cudaStream_t stream) {
    if (dtype_fp32) {
        using T = float;
        const int V = pick_vec<T>(Ch, {gates, c_prev, c_next, dh_a, dh_b, dc_next, dz, dc_prev});
        const long long nvec = P * (Ch / V);
        const unsigned grid = grid_for(nvec, 256, num_sms() * 16);
        if (V == 4)
            lstm_gates_bwd_kernel<T, 4, false><<<grid, 256, 0, stream>>>(static_cast<const T*>(gates), c_prev, c_next, static_cast<const T*>(dh_a), static_cast<const T*>(dh_b), dc_next, static_cast<T*>(dz), dc_prev, nvec, Ch);
        else
            lstm_gates_bwd_kernel<T, 1, false><<<grid, 256, 0, stream>>>(static_cast<const T*>(gates), c_prev, c_next, static_cast<const T*>(dh_a), static_cast<const T*>(dh_b), dc_next, static_cast<T*>(dz), dc_prev, nvec, Ch);
    } else {
        using T = __nv_bfloat16;
        const int V = pick_vec<T>(Ch, {gates, c_prev, c_next, dh_a, dh_b, dc_next, dz, dc_prev});
        const long long nvec = P * (Ch / V);
        const unsigned grid = grid_for(nvec, 256, num_sms() * 16);
        if (V == 8)
            lstm_gates_bwd_kernel<T, 8, true><<<grid, 256, 0, stream>>>(static_cast<const T*>(gates), c_prev, c_next, static_cast<const T*>(dh_a), static_cast<const T*>(dh_b), dc_next, static_cast<T*>(dz), dc_prev, nvec, Ch);
        else
            lstm_gates_bwd_kernel<T, 1, true><<<grid, 256, 0, stream>>>(static_cast<const T*>(gates), c_prev, c_next, static_cast<const T*>(dh_a), static_cast<const T*>(dh_b), dc_next, static_cast<T*>(dz), dc_prev, nvec, Ch);
    }
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// ------------------------------------------------------------------------------------------------
// 1x1 output convolution (OutConv, unet.py:101-107): y[p][o] = b[o] + sum_c x[p][c] w[o][c]  (fp32 out)
// A group of L lanes (power of two) owns one pixel; lanes stride over the channel vectors.
// ------------------------------------------------------------------------------------------------
template <typename T, int V>
__global__ void __launch_bounds__(256) outconv_fwd_kernel(const T* __restrict__ x, const float* __restrict__ w,
                                                          const float* __restrict__ b, float* __restrict__ y,
                                                          long long P, int C, int O, int L) {
    const int CV = C / V;
    const int lane = threadIdx.x & (L - 1);
    const int G = 32 / L;  // pixel groups per warp
    const int gidx = (threadIdx.x & 31) / L;
    const long long warp = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
    // warp-uniform trip count: every lane takes part in the shuffles
    for (long long base = warp * G; base < P; base += nwarps * G) {
        const long long p = base + gidx;
        const bool valid = p < P;
        for (int o = 0; o < O; ++o) {
            float acc = 0.f;
            if (valid) {
                for (int cv = lane; cv < CV; cv += L) {
                    float f[V];
                    ldv<T, V>(x + p * C + cv * V, f);
#pragma unroll
                    for (int j = 0; j < V; ++j) acc = fmaf(f[j], __ldg(w + o * C + cv * V + j), acc);
                }
            }
            for (int s = L >> 1; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
            if (valid && lane == 0) y[p * O + o] = acc + (b ? b[o] : 0.f);
        }
    }
}

static int pow2_floor(int x) {
    int p = 1;
    while (p * 2 <= x) p *= 2;
    return p;
}

int launch_outconv_fwd(const void* x, const float* w, const float* b, float* y, long long P, int C, int O,
                       int dtype_fp32, cudaStream_t stream) {
    auto go = [&](auto tag, int V) {
        using T = decltype(tag);
        int L = pow2_floor(C / V);
        if (L > 32) L = 32;
        // P rounded up to whole warps so that every lane of a shuffle group stays in the loop together
        const unsigned grid = grid_for(P * L, 256, num_sms() * 16);
        const T* xs = static_cast<const T*>(x);
        if (V == 1)
            outconv_fwd_kernel<T, 1><<<grid, 256, 0, stream>>>(xs, w, b, y, P, C, O, L);
        else if constexpr (std::is_same<T, float>::value)
            outconv_fwd_kernel<T, 4><<<grid, 256, 0, stream>>>(xs, w, b, y, P, C, O, L);
        else
            outconv_fwd_kernel<T, 8><<<grid, 256, 0, stream>>>(xs, w, b, y, P, C, O, L);
    };
    if (dtype_fp32)
        go(float(), pick_vec<float>(C, {x}));
    else
        go(__nv_bfloat16(), pick_vec<__nv_bfloat16>(C, {x}));
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// dx[p][c] = sum_o dy[p][o] * w[o][c]
template <typename T, int V>
__global__ void __launch_bounds__(256) outconv_dgrad_kernel(const float* __restrict__ dy, const float* __restrict__ w,
                                                            T* __restrict__ dx, long long nvec, int C, int O) {
    const int CV = C / V;
    for (long long v = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; v < nvec;
         v += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long p = v / CV;
        const int c = static_cast<int>(v - p * CV) * V;
        float f[V];
#pragma unroll
        for (int j = 0; j < V; ++j) f[j] = 0.f;
        for (int o = 0; o < O; ++o) {
            const float d = __ldg(dy + p * O + o);
#pragma unroll
            for (int j = 0; j < V; ++j) f[j] = fmaf(d, __ldg(w + o * C + c + j), f[j]);
        }
        stv<T, V>(dx + v * V, f);
    }
}

int launch_outconv_dgrad(const float* dy, const float* w, void* dx, long long P, int C, int O, int dtype_fp32,
                         cudaStream_t stream) {
    auto go = [&](auto tag, int V) {
        using T = decltype(tag);
        const long long nvec = P * (C / V);
        const unsigned grid = grid_for(nvec, 256 * 2, num_sms() * 16);
        T* os = static_cast<T*>(dx);
        if (V == 1)
            outconv_dgrad_kernel<T, 1><<<grid, 256, 0, stream>>>(dy, w, os, nvec, C, O);
        else if constexpr (std::is_same<T, float>::value)
            outconv_dgrad_kernel<T, 4><<<grid, 256, 0, stream>>>(dy, w, os, nvec, C, O);
        else
            outconv_dgrad_kernel<T, 8><<<grid, 256, 0, stream>>>(dy, w, os, nvec, C, O);
    };
    if (dtype_fp32)
        go(float(), pick_vec<float>(C, {dx}));
    else
        go(__nv_bfloat16(), pick_vec<__nv_bfloat16>(C, {dx}));
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// ------------------------------------------------------------------------------------------------
// pixel shuffle for ConvTranspose2d(k=2, stride=2) (unet.py:90) and the F.pad of unet.py:95-97
//   shuffle  : z [IMG][H][W][4][C] (+bias[c])  ->  y [IMG][Hd][Wd][C] at (2h+i+oy, 2w+j+ox); tap = i*2+j
//   unshuffle: the inverse gather (backward)
// ------------------------------------------------------------------------------------------------
template <typename T, int V, bool UNSHUFFLE>
__global__ void __launch_bounds__(256) shuffle2x2_kernel(const T* __restrict__ src, T* __restrict__ dst,
                                                         const float* __restrict__ bias, long long nvec, int H, int W,
                                                         int Hd, int Wd, int oy, int ox, int CV) {
    for (long long v = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; v < nvec;
         v += static_cast<long long>(gridDim.x) * blockDim.x) {
        long long r = v;
        const int cv = static_cast<int>(r % CV);
        r /= CV;
        const int tap = static_cast<int>(r & 3);
        r >>= 2;
        const int w = static_cast<int>(r % W);
        r /= W;
        const int h = static_cast<int>(r % H);
        const long long img = r / H;
        const int yy = 2 * h + (tap >> 1) + oy, xx = 2 * w + (tap & 1) + ox;
        const long long big = (((img * Hd + yy) * Wd + xx) * CV + cv) * V;
        float f[V];
        if (UNSHUFFLE) {
            if (yy >= 0 && yy < Hd && xx >= 0 && xx < Wd) {
                ldv<T, V>(src + big, f);
            } else {
#pragma unroll
                for (int j = 0; j < V; ++j) f[j] = 0.f;
            }
            stv<T, V>(dst + v * V, f);
        } else {
            if (yy >= 0 && yy < Hd && xx >= 0 && xx < Wd) {
                ldv<T, V>(src + v * V, f);
                if (bias) {
#pragma unroll
                    for (int j = 0; j < V; ++j) f[j] += __ldg(bias + cv * V + j);
                }
                stv<T, V>(dst + big, f);
            }
        }
    }
}

int launch_shuffle2x2(const void* src, void* dst, const float* bias, long long IMG, int H, int W, int C, int Hd,
                      int Wd, int oy, int ox, int unshuffle, int dtype_fp32, cudaStream_t stream) {
    auto go = [&](auto tag, int V) {
        using T = decltype(tag);
        const long long nvec = IMG * H * W * 4 * (C / V);
        const unsigned grid = grid_for(nvec, 256 * 2, num_sms() * 16);
        const T* s = static_cast<const T*>(src);
        T* d = static_cast<T*>(dst);
        if (unshuffle) {
            if (V == 1)
                shuffle2x2_kernel<T, 1, true><<<grid, 256, 0, stream>>>(s, d, bias, nvec, H, W, Hd, Wd, oy, ox, C);
            else if constexpr (std::is_same<T, float>::value)
                shuffle2x2_kernel<T, 4, true><<<grid, 256, 0, stream>>>(s, d, bias, nvec, H, W, Hd, Wd, oy, ox, C / 4);
            else
                shuffle2x2_kernel<T, 8, true><<<grid, 256, 0, stream>>>(s, d, bias, nvec, H, W, Hd, Wd, oy, ox, C / 8);
        } else {
            if (V == 1)
                shuffle2x2_kernel<T, 1, false><<<grid, 256, 0, stream>>>(s, d, bias, nvec, H, W, Hd, Wd, oy, ox, C);
            else if constexpr (std::is_same<T, float>::value)
                shuffle2x2_kernel<T, 4, false><<<grid, 256, 0, stream>>>(s, d, bias, nvec, H, W, Hd, Wd, oy, ox, C / 4);
            else
                shuffle2x2_kernel<T, 8, false><<<grid, 256, 0, stream>>>(s, d, bias, nvec, H, W, Hd, Wd, oy, ox, C / 8);
        }
    };
    if (dtype_fp32)
        go(float(), pick_vec<float>(C, {src, dst}));
    else
        go(__nv_bfloat16(), pick_vec<__nv_bfloat16>(C, {src, dst}));
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// ------------------------------------------------------------------------------------------------
// generic 5-D strided copy with type conversion: dst[i . dstride] (+)= src[i . sstride]
// used for NCHW <-> NHWC layout changes at the module boundary and for weight (un)packing
// ------------------------------------------------------------------------------------------------
struct Copy5 {
    long long dims[5];
    long long ss[5];
    long long ds[5];
};

template <typename TS, typename TD>
__global__ void __launch_bounds__(256) strided_copy_kernel(const TS* __restrict__ src, TD* __restrict__ dst,
                                                           const Copy5 g, long long n, int accumulate) {
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        long long r = i, so = 0, dofs = 0;
#pragma unroll
        for (int d = 4; d >= 0; --d) {
            const long long k = r % g.dims[d];
            r /= g.dims[d];
            so += k * g.ss[d];
            dofs += k * g.ds[d];
        }
        float f[1], o[1];
        ldv<TS, 1>(src + so, f);
        if (accumulate) {
            ldv<TD, 1>(dst + dofs, o);
            f[0] += o[0];
        }
        stv<TD, 1>(dst + dofs, f);
    }
}

int launch_strided_copy(const void* src, int src_fp32, void* dst, int dst_fp32, const long long* dims,
                        const long long* sstr, const long long* dstr, int accumulate, cudaStream_t stream) {
    Copy5 g;
    long long n = 1;
    for (int i = 0; i < 5; ++i) {
        g.dims[i] = dims[i];
        g.ss[i] = sstr[i];
        g.ds[i] = dstr[i];
        n *= dims[i];
    }
    if (n == 0) return B200_OK;
    const unsigned grid = grid_for(n, 256 * 4, num_sms() * 16);
    using B = __nv_bfloat16;
    if (src_fp32 && dst_fp32)
        strided_copy_kernel<float, float><<<grid, 256, 0, stream>>>(static_cast<const float*>(src), static_cast<float*>(dst), g, n, accumulate);
    else if (src_fp32)
        strided_copy_kernel<float, B><<<grid, 256, 0, stream>>>(static_cast<const float*>(src), static_cast<B*>(dst), g, n, accumulate);
    else if (dst_fp32)
        strided_copy_kernel<B, float><<<grid, 256, 0, stream>>>(static_cast<const B*>(src), static_cast<float*>(dst), g, n, accumulate);
    else
        strided_copy_kernel<B, B><<<grid, 256, 0, stream>>>(static_cast<const B*>(src), static_cast<B*>(dst), g, n, accumulate);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// ------------------------------------------------------------------------------------------------
// Split-K reduction epilogues (conv_tc.cu launch_conv_tc_splitk): ws holds `splits` slices [P][N] of fp32 partial
// sums; every thread adds the slices of one output vector in split order (no atomics, so the result does not depend on
// the order in which the splits finished), then applies what the unsplit GEMM epilogue would have applied.
// ------------------------------------------------------------------------------------------------

// ConvLSTM step (the EPI_LSTM epilogue of conv_tc.cu, unet.py:29-35): the N = 4*Ch columns are gate-interleaved in
// blocks of cht hidden channels (column (nt*4 + g)*cht + j, like bias_packed); h_next bf16, c_next fp32, no gates.
__global__ void __launch_bounds__(256) splitk_lstm_cell_kernel(const float* __restrict__ ws, int splits, long long P,
                                                               int Ch, int cht, const float* __restrict__ bias,
                                                               const float* __restrict__ c_prev,
                                                               float* __restrict__ c_next,
                                                               __nv_bfloat16* __restrict__ h_next) {
    constexpr int V = 8;
    const int CV = Ch / V;
    const long long nvec = P * CV;
    const long long slice = P * 4LL * Ch;
    for (long long v = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; v < nvec;
         v += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long p = v / CV;
        const int ch = static_cast<int>(v - p * CV) * V;
        const int nt = ch / cht;
        const int col = nt * 4 * cht + (ch - nt * cht);  // gate g at col + g * cht
        const float* r = ws + p * 4LL * Ch + col;
        float z[4][V];
#pragma unroll
        for (int g = 0; g < 4; ++g) ldv<float, V>(r + g * cht, z[g]);
        for (int s = 1; s < splits; ++s) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                float t[V];
                ldv<float, V>(r + s * slice + g * cht, t);
#pragma unroll
                for (int j = 0; j < V; ++j) z[g][j] += t[j];
            }
        }
        if (bias) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                float b[V];
                ldv<float, V>(bias + col + g * cht, b);
#pragma unroll
                for (int j = 0; j < V; ++j) z[g][j] += b[j];
            }
        }
        float cp[V];
        if (c_prev) {
            ldv<float, V>(c_prev + p * Ch + ch, cp);
        } else {
#pragma unroll
            for (int j = 0; j < V; ++j) cp[j] = 0.f;
        }
        float cn[V], hn[V];
#pragma unroll
        for (int j = 0; j < V; ++j) {
            const float gi = act_sigmoid<true>(z[0][j]);
            const float gf = act_sigmoid<true>(z[1][j]);
            const float gg = act_tanh<true>(z[2][j]);
            const float go = act_sigmoid<true>(z[3][j]);
            cn[j] = fmaf(gf, cp[j], gi * gg);
            hn[j] = go * act_tanh<true>(cn[j]);
        }
        stv<float, V>(c_next + p * Ch + ch, cn);
        stv<__nv_bfloat16, V>(h_next + p * Ch + ch, hn);
    }
}

int launch_splitk_lstm_cell(const float* ws, int splits, long long P, int Ch, int cht, const float* bias,
                            const float* c_prev, float* c_next, void* h_next, cudaStream_t stream) {
    if (Ch % 16 != 0 || (cht != 16 && cht != 32 && cht != 64) || Ch % cht != 0) {
        set_last_error("splitk_lstm_cell: Ch=%d / cht=%d not supported", Ch, cht);
        return B200_ERR_SHAPE;
    }
    for (const void* q : {static_cast<const void*>(ws), static_cast<const void*>(bias), static_cast<const void*>(c_prev),
                          static_cast<const void*>(c_next), static_cast<const void*>(h_next)})
        if (reinterpret_cast<uintptr_t>(q) & 15) {
            set_last_error("splitk_lstm_cell: pointers must be 16-byte aligned");
            return B200_ERR_ALIGN;
        }
    const long long nvec = P * (Ch / 8);
    splitk_lstm_cell_kernel<<<grid_for(nvec, 256, num_sms() * 16), 256, 0, stream>>>(
        ws, splits, P, Ch, cht, bias, c_prev, c_next, static_cast<__nv_bfloat16*>(h_next));
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// Convolution with eval-mode BatchNorm folded in (the EPI_STORE epilogue with scale): y = sum * scale + shift, optional
// ReLU; scale / shift may be NULL (1 / 0).  y: bf16 or fp32 [P][N].
template <typename TD>
__global__ void __launch_bounds__(256) splitk_affine_kernel(const float* __restrict__ ws, int splits, long long P, int N,
                                                            const float* __restrict__ scale,
                                                            const float* __restrict__ shift, int relu,
                                                            TD* __restrict__ y) {
    constexpr int V = 8;
    const int NV = N / V;
    const long long nvec = P * NV;
    const long long slice = P * static_cast<long long>(N);
    for (long long v = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; v < nvec;
         v += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long p = v / NV;
        const int n = static_cast<int>(v - p * NV) * V;
        const float* r = ws + p * N + n;
        float f[V];
        ldv<float, V>(r, f);
        for (int s = 1; s < splits; ++s) {
            float t[V];
            ldv<float, V>(r + s * slice, t);
#pragma unroll
            for (int j = 0; j < V; ++j) f[j] += t[j];
        }
        if (scale) {
            float a[V];
            ldv<float, V>(scale + n, a);
#pragma unroll
            for (int j = 0; j < V; ++j) f[j] *= a[j];
        }
        if (shift) {
            float b[V];
            ldv<float, V>(shift + n, b);
#pragma unroll
            for (int j = 0; j < V; ++j) f[j] += b[j];
        }
        if (relu) {
#pragma unroll
            for (int j = 0; j < V; ++j) f[j] = fmaxf(f[j], 0.f);
        }
        stv<TD, V>(y + p * N + n, f);
    }
}

int launch_splitk_affine(const float* ws, int splits, long long P, int N, const float* scale, const float* shift, int relu,
                         void* y, int out_fp32, cudaStream_t stream) {
    if (N % 16 != 0) {
        set_last_error("splitk_affine: N=%d is not a multiple of 16", N);
        return B200_ERR_SHAPE;
    }
    for (const void* q : {static_cast<const void*>(ws), static_cast<const void*>(scale), static_cast<const void*>(shift),
                          static_cast<const void*>(y)})
        if (reinterpret_cast<uintptr_t>(q) & 15) {
            set_last_error("splitk_affine: pointers must be 16-byte aligned");
            return B200_ERR_ALIGN;
        }
    const long long nvec = P * (N / 8);
    const unsigned grid = grid_for(nvec, 256, num_sms() * 16);
    if (out_fp32)
        splitk_affine_kernel<float><<<grid, 256, 0, stream>>>(ws, splits, P, N, scale, shift, relu, static_cast<float*>(y));
    else
        splitk_affine_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(ws, splits, P, N, scale, shift, relu,
                                                                     static_cast<__nv_bfloat16*>(y));
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

}  // namespace b200
