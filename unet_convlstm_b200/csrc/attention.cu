// SpatialAttention (reference unet.py:113-125) on channels-last images x [IMG][H][W][C]:
//   y = x * sigmoid(conv_k([mean_c x ; amax_c x]))      conv: 2 inputs, 1 output, padding k/2, no bias, k in {1,3,5,7}
// and its backward with ATen's semantics (amax splits its gradient evenly among tied maxima).
//
// The convolution has K = 2k^2 <= 98, so none of this is tensor-core work: the kernels are HBM-bound passes over the
// activation tensor, one warp per pixel (its C channels are contiguous), reading bf16 or fp32 and computing in fp32.
//   forward:  attn_pool_kernel      mean / max over C                              reads x
//             attn_apply_kernel     the k x k convolution of the pooled map at the warp's pixel, sigmoid -> a[p],
//                                   y = x * a[p] (bf16: rounded once from the fp32 product)   reads x, writes y
//   backward: attn_bwd_reduce_kernel  da = sum_c g*x, ds = da*(1-a)*a, the number of tied maxima   reads g, x
//             attn_bwd_dx_kernel      the transposed convolution of ds at the warp's pixel, then
//                                     dx = g*a + dmean / C + [x == max] * dmax / ties              reads g, x, writes dx
//             attn_wgrad_kernel       dw partial sums over fixed pixel ranges, added in range order by splitk_reduce
//                                     into the zeroed dw
// The convolution runs per pixel inside the warp that owns the pixel (lanes split the 2k^2 taps, a butterfly sum gives
// every lane the same bits), so a and dpooled need no pass of their own.  Every sum has a fixed order: results are
// run-to-run bit-identical, with no atomics.
#include <math.h>

#include "../../include/b200_convlstm.h"
#include "common.cuh"

namespace b200 {

namespace {

constexpr int kWarps = 8;               // pixels per 256-thread block
constexpr int kUnroll = 4;              // 16-byte loads a lane issues before it uses them
constexpr int kWgradThreads = 256;
constexpr int kWgradPixels = 2048;      // pixels per weight-gradient partial sum (b200_spatial_attention_bwd)

// 16 bytes of activations <-> fp32 values
template <typename T>
struct Pack16;
template <>
struct Pack16<float> {
    static constexpr int N = 4;
    __device__ static float get(const uint4& u, int i) {
        return __uint_as_float(i == 0 ? u.x : i == 1 ? u.y : i == 2 ? u.z : u.w);
    }
    __device__ static uint4 put(const float* f) {
        return make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]), __float_as_uint(f[3]));
    }
    __device__ static float load1(const float* p) { return __ldg(p); }
    __device__ static void store1(float* p, float v) { *p = v; }
};
template <>
struct Pack16<__nv_bfloat16> {
    static constexpr int N = 8;
    __device__ static float get(const uint4& u, int i) {
        const unsigned w = (i >> 1) == 0 ? u.x : (i >> 1) == 1 ? u.y : (i >> 1) == 2 ? u.z : u.w;
        return __uint_as_float((i & 1) ? (w & 0xffff0000u) : (w << 16));
    }
    __device__ static unsigned pair(float lo, float hi) {
        const __nv_bfloat162 b = __floats2bfloat162_rn(lo, hi);
        return *reinterpret_cast<const unsigned*>(&b);
    }
    __device__ static uint4 put(const float* f) {
        return make_uint4(pair(f[0], f[1]), pair(f[2], f[3]), pair(f[4], f[5]), pair(f[6], f[7]));
    }
    __device__ static float load1(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }
    __device__ static void store1(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

struct Geo {
    long long NP;   // IMG * H * W pixels
    int H, W, C, k;
};

// Sum over the taps of the warp's pixel p of w[c][ky][kx] * src[c-plane value at the tap's pixel].  transposed = 0: the
// forward convolution of the pooled map (src = pooled [NP][2], tap pixel (y + ky - r, x + kx - r)); transposed = 1: its
// data gradient from ds (src = ds [NP], tap pixel (y - ky + r, x - kx + r)), one sum per input plane.  Lanes take taps
// lane, lane + 32, ...; the butterfly leaves the same value in every lane.
template <int TRANSPOSED>
__device__ __forceinline__ void tap_sums(const float* __restrict__ w, const float* __restrict__ src, long long p,
                                         const Geo& g, int lane, float& s0, float& s1) {
    const int HW = g.H * g.W;
    const long long img0 = (p / HW) * HW;
    const int pix = static_cast<int>(p - img0);
    const int py = pix / g.W, px = pix - py * g.W;
    const int taps = g.k * g.k, r = g.k / 2;
    s0 = 0.f;
    s1 = 0.f;
    for (int t = lane; t < 2 * taps; t += 32) {
        const int c = t >= taps;
        const int tt = t - c * taps;
        const int ky = tt / g.k, kx = tt - ky * g.k;
        const int iy = TRANSPOSED ? py - ky + r : py + ky - r;
        const int ix = TRANSPOSED ? px - kx + r : px + kx - r;
        if (iy < 0 || iy >= g.H || ix < 0 || ix >= g.W) continue;
        const long long q = img0 + iy * g.W + ix;
        const float v = TRANSPOSED ? __ldg(src + q) : __ldg(src + 2 * q + c);
        if (c) s1 = fmaf(__ldg(w + t), v, s1);
        else s0 = fmaf(__ldg(w + t), v, s0);
    }
    s0 = warp_sum(s0);
    s1 = warp_sum(s1);
}

// pooled[p] = {sum_c x / C, max_c x}
template <typename T, bool VEC>
__global__ void __launch_bounds__(32 * kWarps) attn_pool_kernel(const T* __restrict__ x, Geo g, float* __restrict__ pooled) {
    using P = Pack16<T>;
    const long long p = static_cast<long long>(blockIdx.x) * kWarps + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (p >= g.NP) return;
    const T* xp = x + p * g.C;
    float s = 0.f, m = -INFINITY;
    if (VEC) {
        const uint4* xv = reinterpret_cast<const uint4*>(xp);
        const int nv = g.C / P::N;
        for (int v0 = lane; v0 < nv; v0 += 32 * kUnroll) {
            uint4 u[kUnroll];
#pragma unroll
            for (int j = 0; j < kUnroll; ++j)
                if (v0 + 32 * j < nv) u[j] = __ldg(xv + v0 + 32 * j);
#pragma unroll
            for (int j = 0; j < kUnroll; ++j) {
                if (v0 + 32 * j >= nv) break;
#pragma unroll
                for (int e = 0; e < P::N; ++e) {
                    const float f = P::get(u[j], e);
                    s += f;
                    m = fmaxf(m, f);
                }
            }
        }
    } else {
        for (int c = lane; c < g.C; c += 32) {
            const float f = P::load1(xp + c);
            s += f;
            m = fmaxf(m, f);
        }
    }
    s = warp_sum(s);
    m = warp_max(m);
    if (lane == 0) {
        pooled[2 * p] = s / static_cast<float>(g.C);
        pooled[2 * p + 1] = m;
    }
}

// a[p] = sigmoid(conv(pooled)[p]); y = x * a[p]
template <typename T, bool VEC>
__global__ void __launch_bounds__(32 * kWarps) attn_apply_kernel(const T* __restrict__ x, const float* __restrict__ w,
                                                                  const float* __restrict__ pooled, Geo g,
                                                                  float* __restrict__ a, T* __restrict__ y) {
    using P = Pack16<T>;
    const long long p = static_cast<long long>(blockIdx.x) * kWarps + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (p >= g.NP) return;
    float s0, s1;
    tap_sums<0>(w, pooled, p, g, lane, s0, s1);
    const float av = 1.f / (1.f + expf(-(s0 + s1)));
    if (lane == 0) a[p] = av;
    const T* xp = x + p * g.C;
    T* yp = y + p * g.C;
    if (VEC) {
        const uint4* xv = reinterpret_cast<const uint4*>(xp);
        uint4* yv = reinterpret_cast<uint4*>(yp);
        const int nv = g.C / P::N;
        for (int v0 = lane; v0 < nv; v0 += 32 * kUnroll) {
            uint4 u[kUnroll];
#pragma unroll
            for (int j = 0; j < kUnroll; ++j)
                if (v0 + 32 * j < nv) u[j] = __ldg(xv + v0 + 32 * j);
#pragma unroll
            for (int j = 0; j < kUnroll; ++j) {
                if (v0 + 32 * j >= nv) break;
                float f[P::N];
#pragma unroll
                for (int e = 0; e < P::N; ++e) f[e] = P::get(u[j], e) * av;
                yv[v0 + 32 * j] = P::put(f);
            }
        }
    } else {
        for (int c = lane; c < g.C; c += 32) P::store1(yp + c, P::load1(xp + c) * av);
    }
}

// ds[p] = (sum_c g*x) * (1 - a) * a  (ATen's sigmoid_backward order); ties[p] = #{c : x == max}
template <typename T, bool VEC>
__global__ void __launch_bounds__(32 * kWarps) attn_bwd_reduce_kernel(const T* __restrict__ x, const T* __restrict__ dy,
                                                                       const float* __restrict__ pooled,
                                                                       const float* __restrict__ a, Geo g,
                                                                       float* __restrict__ ds, float* __restrict__ ties) {
    using P = Pack16<T>;
    const long long p = static_cast<long long>(blockIdx.x) * kWarps + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (p >= g.NP) return;
    const float mx = __ldg(pooled + 2 * p + 1);
    const T* xp = x + p * g.C;
    const T* gp = dy + p * g.C;
    float s = 0.f;
    int n = 0;
    if (VEC) {
        const uint4* xv = reinterpret_cast<const uint4*>(xp);
        const uint4* gv = reinterpret_cast<const uint4*>(gp);
        const int nv = g.C / P::N;
        for (int v0 = lane; v0 < nv; v0 += 32 * kUnroll) {
            uint4 ux[kUnroll], ug[kUnroll];
#pragma unroll
            for (int j = 0; j < kUnroll; ++j)
                if (v0 + 32 * j < nv) {
                    ux[j] = __ldg(xv + v0 + 32 * j);
                    ug[j] = __ldg(gv + v0 + 32 * j);
                }
#pragma unroll
            for (int j = 0; j < kUnroll; ++j) {
                if (v0 + 32 * j >= nv) break;
#pragma unroll
                for (int e = 0; e < P::N; ++e) {
                    const float xf = P::get(ux[j], e);
                    s = fmaf(P::get(ug[j], e), xf, s);
                    n += xf == mx;
                }
            }
        }
    } else {
        for (int c = lane; c < g.C; c += 32) {
            const float xf = P::load1(xp + c);
            s = fmaf(P::load1(gp + c), xf, s);
            n += xf == mx;
        }
    }
    s = warp_sum(s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
    if (lane == 0) {
        const float av = __ldg(a + p);
        ds[p] = s * (1.f - av) * av;
        ties[p] = static_cast<float>(n);
    }
}

// dx = g*a + dmean / C + [x == max] * (dmax / ties)
template <typename T, bool VEC>
__global__ void __launch_bounds__(32 * kWarps) attn_bwd_dx_kernel(const T* __restrict__ x, const T* __restrict__ dy,
                                                                   const float* __restrict__ w,
                                                                   const float* __restrict__ pooled,
                                                                   const float* __restrict__ a,
                                                                   const float* __restrict__ ds,
                                                                   const float* __restrict__ ties, Geo g,
                                                                   T* __restrict__ dx) {
    using P = Pack16<T>;
    const long long p = static_cast<long long>(blockIdx.x) * kWarps + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (p >= g.NP) return;
    float dmean, dmax;
    tap_sums<1>(w, ds, p, g, lane, dmean, dmax);
    const float qm = dmean / static_cast<float>(g.C);
    const float qx = dmax / __ldg(ties + p);
    const float mx = __ldg(pooled + 2 * p + 1);
    const float av = __ldg(a + p);
    const T* xp = x + p * g.C;
    const T* gp = dy + p * g.C;
    T* dp = dx + p * g.C;
    if (VEC) {
        const uint4* xv = reinterpret_cast<const uint4*>(xp);
        const uint4* gv = reinterpret_cast<const uint4*>(gp);
        uint4* dv = reinterpret_cast<uint4*>(dp);
        const int nv = g.C / P::N;
        for (int v0 = lane; v0 < nv; v0 += 32 * kUnroll) {
            uint4 ux[kUnroll], ug[kUnroll];
#pragma unroll
            for (int j = 0; j < kUnroll; ++j)
                if (v0 + 32 * j < nv) {
                    ux[j] = __ldg(xv + v0 + 32 * j);
                    ug[j] = __ldg(gv + v0 + 32 * j);
                }
#pragma unroll
            for (int j = 0; j < kUnroll; ++j) {
                if (v0 + 32 * j >= nv) break;
                float f[P::N];
#pragma unroll
                for (int e = 0; e < P::N; ++e)
                    f[e] = P::get(ug[j], e) * av + qm + (P::get(ux[j], e) == mx ? qx : 0.f);
                dv[v0 + 32 * j] = P::put(f);
            }
        }
    } else {
        for (int c = lane; c < g.C; c += 32)
            P::store1(dp + c, P::load1(gp + c) * av + qm + (P::load1(xp + c) == mx ? qx : 0.f));
    }
}

// part[blockIdx.x][c][ky][kx] = sum over the block's kWgradPixels pixels p of ds[p] * pooled_c[tap pixel of p].  Each
// thread keeps the 2k^2 sums of its own pixels (p0 + tid, p0 + tid + 256, ...) in registers; warps add their lanes'
// sums with a butterfly, then thread t adds the 8 warps' sums of tap t in warp order.
template <int K>
__global__ void __launch_bounds__(kWgradThreads) attn_wgrad_kernel(const float* __restrict__ ds,
                                                                  const float* __restrict__ pooled, Geo g,
                                                                  float* __restrict__ part) {
    constexpr int TAPS = K * K, R = K / 2;
    __shared__ float red[kWgradThreads / 32][2 * TAPS];
    float acc[2 * TAPS];
#pragma unroll
    for (int t = 0; t < 2 * TAPS; ++t) acc[t] = 0.f;
    const int HW = g.H * g.W;
    const long long p0 = static_cast<long long>(blockIdx.x) * kWgradPixels;
    for (int i = threadIdx.x; i < kWgradPixels; i += kWgradThreads) {
        const long long p = p0 + i;
        if (p >= g.NP) break;
        const long long img0 = (p / HW) * HW;
        const int pix = static_cast<int>(p - img0);
        const int py = pix / g.W, px = pix - py * g.W;
        const float d = __ldg(ds + p);
#pragma unroll
        for (int ky = 0; ky < K; ++ky) {
            const int iy = py + ky - R;
            if (iy < 0 || iy >= g.H) continue;
#pragma unroll
            for (int kx = 0; kx < K; ++kx) {
                const int ix = px + kx - R;
                if (ix < 0 || ix >= g.W) continue;
                const float2 v = __ldg(reinterpret_cast<const float2*>(pooled) + img0 + iy * g.W + ix);
                acc[ky * K + kx] = fmaf(d, v.x, acc[ky * K + kx]);
                acc[TAPS + ky * K + kx] = fmaf(d, v.y, acc[TAPS + ky * K + kx]);
            }
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int t = 0; t < 2 * TAPS; ++t) {
        const float v = warp_sum(acc[t]);
        if (lane == 0) red[warp][t] = v;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < 2 * TAPS; t += kWgradThreads) {
        float s = red[0][t];
#pragma unroll
        for (int w = 1; w < kWgradThreads / 32; ++w) s += red[w][t];
        part[static_cast<long long>(blockIdx.x) * 2 * TAPS + t] = s;
    }
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int check_geo(const char* who, long long IMG, int H, int W, int C, int ksize, Geo* g) {
    if (ksize != 1 && ksize != 3 && ksize != 5 && ksize != 7) {
        set_last_error("%s: kernel size %d is not supported (1, 3, 5 or 7)", who, ksize);
        return B200_ERR_SHAPE;
    }
    if (IMG <= 0 || H <= 0 || W <= 0 || C <= 0) {
        set_last_error("%s: sizes must be positive (IMG=%lld H=%d W=%d C=%d)", who, IMG, H, W, C);
        return B200_ERR_SHAPE;
    }
    const long long HW = static_cast<long long>(H) * W;
    const long long NP = IMG * HW;
    if (HW > 0x7fffffffLL || (NP + kWarps - 1) / kWarps > 0x7fffffffLL) {
        set_last_error("%s: %lld pixels are too many", who, NP);
        return B200_ERR_SHAPE;
    }
    *g = Geo{NP, H, W, C, ksize};
    return B200_OK;
}

template <typename T>
int launch_fwd(const void* x, const float* w, const Geo& g, float* pooled, float* a, void* y, cudaStream_t st) {
    const bool vec = (static_cast<long long>(g.C) * sizeof(T)) % 16 == 0 && aligned16(x) && aligned16(y);
    const unsigned blocks = static_cast<unsigned>((g.NP + kWarps - 1) / kWarps);
    const T* xt = static_cast<const T*>(x);
    T* yt = static_cast<T*>(y);
    if (vec) {
        attn_pool_kernel<T, true><<<blocks, 32 * kWarps, 0, st>>>(xt, g, pooled);
        attn_apply_kernel<T, true><<<blocks, 32 * kWarps, 0, st>>>(xt, w, pooled, g, a, yt);
    } else {
        attn_pool_kernel<T, false><<<blocks, 32 * kWarps, 0, st>>>(xt, g, pooled);
        attn_apply_kernel<T, false><<<blocks, 32 * kWarps, 0, st>>>(xt, w, pooled, g, a, yt);
    }
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

template <typename T>
int launch_bwd(const void* x, const void* dy, const float* w, const float* pooled, const float* a, const Geo& g,
               float* ws, void* dx, float* dw, cudaStream_t st) {
    const bool vec = (static_cast<long long>(g.C) * sizeof(T)) % 16 == 0 && aligned16(x) && aligned16(dy) &&
                     (dx == nullptr || aligned16(dx));
    const unsigned blocks = static_cast<unsigned>((g.NP + kWarps - 1) / kWarps);
    const T* xt = static_cast<const T*>(x);
    const T* gt = static_cast<const T*>(dy);
    T* dxt = static_cast<T*>(dx);
    float* ds = ws;
    float* ties = ws + g.NP;
    if (vec) attn_bwd_reduce_kernel<T, true><<<blocks, 32 * kWarps, 0, st>>>(xt, gt, pooled, a, g, ds, ties);
    else attn_bwd_reduce_kernel<T, false><<<blocks, 32 * kWarps, 0, st>>>(xt, gt, pooled, a, g, ds, ties);
    B200_CUDA_CHECK(cudaGetLastError());
    if (dx) {
        if (vec) attn_bwd_dx_kernel<T, true><<<blocks, 32 * kWarps, 0, st>>>(xt, gt, w, pooled, a, ds, ties, g, dxt);
        else attn_bwd_dx_kernel<T, false><<<blocks, 32 * kWarps, 0, st>>>(xt, gt, w, pooled, a, ds, ties, g, dxt);
        B200_CUDA_CHECK(cudaGetLastError());
    }
    if (dw) {
        const long long splits = (g.NP + kWgradPixels - 1) / kWgradPixels;
        float* part = ws + 2 * g.NP;
        const unsigned nb = static_cast<unsigned>(splits);
        switch (g.k) {
            case 1: attn_wgrad_kernel<1><<<nb, kWgradThreads, 0, st>>>(ds, pooled, g, part); break;
            case 3: attn_wgrad_kernel<3><<<nb, kWgradThreads, 0, st>>>(ds, pooled, g, part); break;
            case 5: attn_wgrad_kernel<5><<<nb, kWgradThreads, 0, st>>>(ds, pooled, g, part); break;
            default: attn_wgrad_kernel<7><<<nb, kWgradThreads, 0, st>>>(ds, pooled, g, part); break;
        }
        B200_CUDA_CHECK(cudaGetLastError());
        const int cols = 2 * g.k * g.k;
        B200_CUDA_CHECK(cudaMemsetAsync(dw, 0, cols * sizeof(float), st));
        return splitk_reduce(part, static_cast<int>(splits), 1, cols, dw, cols, 0, st);
    }
    return B200_OK;
}

}  // namespace

}  // namespace b200

using namespace b200;

extern "C" int b200_spatial_attention_fwd(const void* x, const float* w, long long IMG, int H, int W, int C, int ksize,
                                          int dtype_fp32, float* pooled, float* a, void* y, void* stream) {
    if (!x || !w || !pooled || !a || !y) {
        set_last_error("b200_spatial_attention_fwd: null pointer");
        return B200_ERR_ARG;
    }
    Geo g;
    const int rc = check_geo("b200_spatial_attention_fwd", IMG, H, W, C, ksize, &g);
    if (rc != B200_OK) return rc;
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    return dtype_fp32 ? launch_fwd<float>(x, w, g, pooled, a, y, st)
                      : launch_fwd<__nv_bfloat16>(x, w, g, pooled, a, y, st);
}

extern "C" int b200_spatial_attention_bwd(const void* x, const void* dy, const float* w, const float* pooled,
                                          const float* a, long long IMG, int H, int W, int C, int ksize, int dtype_fp32,
                                          float* ws, void* dx, float* dw, void* stream) {
    if (!x || !dy || !w || !pooled || !a || !ws) {
        set_last_error("b200_spatial_attention_bwd: null pointer");
        return B200_ERR_ARG;
    }
    Geo g;
    const int rc = check_geo("b200_spatial_attention_bwd", IMG, H, W, C, ksize, &g);
    if (rc != B200_OK) return rc;
    if (reinterpret_cast<uintptr_t>(pooled) & 7u) {
        set_last_error("b200_spatial_attention_bwd: pooled must be 8-byte aligned (read as float2)");
        return B200_ERR_ALIGN;
    }
    if ((g.NP + kWgradPixels - 1) / kWgradPixels > 0x7fffffffLL) {
        set_last_error("b200_spatial_attention_bwd: %lld pixels are too many", g.NP);
        return B200_ERR_SHAPE;
    }
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    return dtype_fp32 ? launch_bwd<float>(x, dy, w, pooled, a, g, ws, dx, dw, st)
                      : launch_bwd<__nv_bfloat16>(x, dy, w, pooled, a, g, ws, dx, dw, st);
}
