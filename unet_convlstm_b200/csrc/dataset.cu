// Batch assembly of the reference's NPZSequenceDataset (train/unet.py:393-401) from the raw arrays kept in device
// memory: for every batch item b (dataset row n = idx[b]), timestep t and pixel,
//   mask = X[n,t,0] > 1.1f                 (torch compares the fp32 tensor with the Python float in fp32, on raw X)
//   x    = X[n,t,c] / norm_const           (IEEE fp32 division, as torch's CPU division by the scalar)
//   y    = affine(transform(clip(Y[n,t])))  in the dtypes NumPy 2 (NEP 50) evaluates them in, rounded once to fp32.
// The reference runs this in NumPy on the host one sequence at a time and copies every batch to the device; here one
// launch per batch reads 12 bytes and writes 16 bytes per pixel-timestep (Cx = 2): HBM-bound.
//
// Which dtype each step of y runs in depends on the types of the dataset's constants, which the caller inspects:
//   fp64_transform: np.clip with np.float64 bounds promotes the fp32 item to float64, so the clip, the transform and
//                   the affine map all run in fp64.  NPZSequenceDataset never makes such bounds (explicit ones are
//                   Python floats, np.percentile of the fp32 Y is np.float32); a dataset object given np.float64 ones does;
//   fp64_affine:    trans_min / trans_max - trans_min are np.float64 (explicit constants with asinh / signed_log):
//                   the fp32 transform is promoted to float64 for the affine map;
//   neither:        Python-float or np.float32 constants are weak / fp32 and everything stays fp32.
// Division, subtraction and scaling go through the _rn intrinsics so that no FMA contraction can fuse them.
#include <type_traits>

#include "../../include/b200_convlstm.h"
#include "common.cuh"

namespace b200 {

struct SeqBatchCfg {
    float norm, lo32, hi32, scale32, tmin32, den32;
    double lo64, hi64, scale64, tmin64, den64;
    int clip, transform, fp64_transform, fp64_affine;  // transform: 0 identity, 1 asinh, 2 signed_log
};

// np.sign(v) * np.log1p(np.abs(v) / s): sign(+-0) = +-0 times log1p(0) = 0, sign(NaN) = NaN
__device__ __forceinline__ float signed_log32(float v, float s) {
    const float sg = v > 0.f ? 1.f : (v < 0.f ? -1.f : v);
    return __fmul_rn(sg, log1pf(__fdiv_rn(fabsf(v), s)));
}
__device__ __forceinline__ double signed_log64(double v, double s) {
    const double sg = v > 0.0 ? 1.0 : (v < 0.0 ? -1.0 : v);
    return __dmul_rn(sg, log1p(__ddiv_rn(fabs(v), s)));
}

// 2 * (t - trans_min) / (trans_max - trans_min) - 1.0, evaluated left to right like NumPy
__device__ __forceinline__ float affine64(double t, const SeqBatchCfg& c) {
    return __double2float_rn(__dsub_rn(__ddiv_rn(__dmul_rn(2.0, __dsub_rn(t, c.tmin64)), c.den64), 1.0));
}

__device__ __forceinline__ float seq_y(float raw, const SeqBatchCfg& c) {
    if (c.fp64_transform) {
        double v = raw;
        // np.clip = minimum(maximum(v, lo), hi): a NaN stays NaN, lo > hi gives hi
        if (c.clip) {
            v = v < c.lo64 ? c.lo64 : v;
            v = v > c.hi64 ? c.hi64 : v;
        }
        if (c.transform == 1) v = asinh(__ddiv_rn(v, c.scale64));
        else if (c.transform == 2) v = signed_log64(v, c.scale64);
        return affine64(v, c);
    }
    float v = raw;
    if (c.clip) {
        v = v < c.lo32 ? c.lo32 : v;
        v = v > c.hi32 ? c.hi32 : v;
    }
    if (c.transform == 1) v = asinhf(__fdiv_rn(v, c.scale32));
    else if (c.transform == 2) v = signed_log32(v, c.scale32);
    if (c.fp64_affine) return affine64(static_cast<double>(v), c);
    return __fsub_rn(__fdiv_rn(__fmul_rn(2.f, __fsub_rn(v, c.tmin32)), c.den32), 1.f);
}

// Elementwise over the V floats of a float or float4, with no local array (an array accessed through a vector cast
// goes to local memory)
template <class F>
__device__ __forceinline__ float vmap(float v, F f) { return f(v); }
template <class F>
__device__ __forceinline__ float4 vmap(float4 v, F f) { return make_float4(f(v.x), f(v.y), f(v.z), f(v.w)); }

// One thread per V consecutive pixels of one (b, t); blockIdx.y walks the B*T (item, timestep) pairs.  V = 4: 16-byte
// loads and stores (H*W % 4 == 0 and 16-byte aligned bases); V = 1: the scalar path for any other size.
// An index outside [0, N) reads nothing: its item is written as x = y = NaN, mask = 0 (the Python wrapper refuses such
// indices before they reach the device; this only keeps a stray index from reading out of bounds).
// 256 threads a block, at most 64 registers: with __launch_bounds__(256) instead, ptxas kept 64 registers but spilled
// 16 bytes around the slow-path calls of the IEEE division in the float4 path; with this cap it spills nothing.
template <int V>
__global__ void __maxnreg__(64) sequence_batch_kernel(const float* __restrict__ X, const float* __restrict__ Y,
                                                      const long long* __restrict__ idx, long long N, int T, int Cx,
                                                      long long HW, int BT, SeqBatchCfg c, float* __restrict__ x,
                                                      float* __restrict__ y, float* __restrict__ mask) {
    using VT = typename std::conditional<V == 4, float4, float>::type;
    const long long HWv = HW / V;
    const long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (q >= HWv) return;
    for (int bt = blockIdx.y; bt < BT; bt += gridDim.y) {
        const int b = bt / T, t = bt - b * T;
        const long long n = __ldg(idx + b);
        const bool ok = n >= 0 && n < N;
        const long long nt = n * T + t;
        // y first: its transform may call the slow-path subroutines of the IEEE division and the libm functions, and
        // nothing of the x / mask part is live across those calls yet
        VT* yo = reinterpret_cast<VT*>(y + static_cast<long long>(bt) * HW) + q;
        if (ok) {
            const VT yraw = __ldg(reinterpret_cast<const VT*>(Y + nt * HW) + q);
            *yo = vmap(yraw, [&c](float e) { return seq_y(e, c); });
        } else {
            *yo = vmap(VT{}, [](float) { return __int_as_float(0x7fc00000); });
        }
        VT* xo = reinterpret_cast<VT*>(x + static_cast<long long>(bt) * Cx * HW) + q;
        VT* mo = reinterpret_cast<VT*>(mask + static_cast<long long>(bt) * HW) + q;
        if (!ok) {
            for (int ch = 0; ch < Cx; ++ch) xo[ch * HWv] = vmap(VT{}, [](float) { return __int_as_float(0x7fc00000); });
            *mo = VT{};
            continue;
        }
        const VT* xi = reinterpret_cast<const VT*>(X + nt * Cx * HW) + q;
        const float norm = c.norm;
        for (int ch = 0; ch < Cx; ++ch) {
            const VT v = __ldg(xi + ch * HWv);
            if (ch == 0) *mo = vmap(v, [](float e) { return e > 1.1f ? 1.f : 0.f; });
            xo[ch * HWv] = vmap(v, [norm](float e) { return __fdiv_rn(e, norm); });
        }
    }
}

}  // namespace b200

using namespace b200;

extern "C" int b200_sequence_batch(const float* X, const float* Y, long long N, int T, int Cx, int H, int W,
                                   const void* idx, int B, double norm_const, int clip, double min_vel, double max_vel,
                                   int transform, double y_scale, double trans_min, double trans_range,
                                   int fp64_transform, int fp64_affine, float* x, float* y, float* mask, void* stream) {
    if (!X || !Y || !idx || !x || !y || !mask) {
        set_last_error("b200_sequence_batch: null pointer");
        return B200_ERR_ARG;
    }
    if (N <= 0 || T <= 0 || Cx <= 0 || H <= 0 || W <= 0 || B <= 0) {
        set_last_error("b200_sequence_batch: sizes must be positive (N=%lld T=%d Cx=%d H=%d W=%d B=%d)", N, T, Cx, H, W, B);
        return B200_ERR_SHAPE;
    }
    if (transform < 0 || transform > 2) {
        set_last_error("b200_sequence_batch: unknown transform code %d (0 identity, 1 asinh, 2 signed_log)", transform);
        return B200_ERR_ARG;
    }
    if ((clip != 0 && clip != 1) || (fp64_transform != 0 && fp64_transform != 1) ||
        (fp64_affine != 0 && fp64_affine != 1) || (fp64_transform && !fp64_affine)) {
        set_last_error("b200_sequence_batch: clip / fp64_transform / fp64_affine must be 0 or 1, and an fp64 transform "
                       "implies an fp64 affine map");
        return B200_ERR_ARG;
    }
    const long long BT = static_cast<long long>(B) * T;
    if (BT > 0x7fffffffLL) {
        set_last_error("b200_sequence_batch: B*T = %lld too large", BT);
        return B200_ERR_SHAPE;
    }
    SeqBatchCfg c;
    c.norm = static_cast<float>(norm_const);
    c.lo32 = static_cast<float>(min_vel);
    c.hi32 = static_cast<float>(max_vel);
    c.scale32 = static_cast<float>(y_scale);
    c.tmin32 = static_cast<float>(trans_min);
    c.den32 = static_cast<float>(trans_range);
    c.lo64 = min_vel;
    c.hi64 = max_vel;
    c.scale64 = y_scale;
    c.tmin64 = trans_min;
    c.den64 = trans_range;
    c.clip = clip;
    c.transform = transform;
    c.fp64_transform = fp64_transform;
    c.fp64_affine = fp64_affine;

    const long long HW = static_cast<long long>(H) * W;
    const auto aligned = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
    const bool vec = HW % 4 == 0 && aligned(X) && aligned(Y) && aligned(x) && aligned(y) && aligned(mask);
    const long long per_bt = vec ? HW / 4 : HW;
    const long long gx = (per_bt + 255) / 256;
    if (gx > 0x7fffffffLL) {
        set_last_error("b200_sequence_batch: H*W = %lld too large", HW);
        return B200_ERR_SHAPE;
    }
    const dim3 grid(static_cast<unsigned>(gx), static_cast<unsigned>(BT < 65535 ? BT : 65535));
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long* ip = static_cast<const long long*>(idx);
    if (vec)
        sequence_batch_kernel<4><<<grid, 256, 0, st>>>(X, Y, ip, N, T, Cx, HW, static_cast<int>(BT), c, x, y, mask);
    else
        sequence_batch_kernel<1><<<grid, 256, 0, st>>>(X, Y, ip, N, T, Cx, HW, static_cast<int>(BT), c, x, y, mask);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}
