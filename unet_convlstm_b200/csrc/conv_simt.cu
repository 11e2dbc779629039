// Generic CUDA-core (SIMT) convolution kernels: fp32 accumulate, fp32 or bf16 storage.
//
// These serve two purposes:
//   1. the "fp32 check mode" of the hot path (north_star: 1e-5 relative parity with the reference's
//      fp32 arithmetic, which the bf16 tensor-core path cannot meet by construction);
//   2. shapes the tcgen05 path cannot tile (first UNet conv with Cin = 2, channel counts that are
//      not multiples of 16, spatial sizes that are not TMA-box friendly, kernel_size != 3 ...).
// Same math and the same packed-weight layout ([tap][N][K]) as conv_tc.cu / wgrad_tc.cu.
#include "pointwise.cuh"

namespace b200 {

template <typename T>
__device__ __forceinline__ float ld_as_float(const T* p);
template <>
__device__ __forceinline__ float ld_as_float<float>(const float* p) { return *p; }
template <>
__device__ __forceinline__ float ld_as_float<__nv_bfloat16>(const __nv_bfloat16* p) {
    return __bfloat162float(*p);
}
template <typename T>
__device__ __forceinline__ void st_from_float(T* p, float v);
template <>
__device__ __forceinline__ void st_from_float<float>(float* p, float v) { *p = v; }
template <>
__device__ __forceinline__ void st_from_float<__nv_bfloat16>(__nv_bfloat16* p, float v) {
    *p = __float2bfloat16_rn(v);
}


// out[m, n] = sum_{kk} A[m, kk] * Wp[tap(kk)][n][c(kk)],  kk = tap*Ct + c
template <typename T>
__global__ void __launch_bounds__(256) conv_simt_kernel(const ConvSimtParams p) {
    __shared__ float As[16][64 + 4];
    __shared__ float Bs[16][64 + 4];
    const int Ct = p.C0 + p.C1;
    const int Kflat = p.ksize * p.ksize * Ct;
    const long long M = static_cast<long long>(p.IMG) * p.H * p.W;
    const long long m0 = static_cast<long long>(blockIdx.x) * 64;
    const int n0 = blockIdx.y * 64;
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const T* s0 = static_cast<const T*>(p.src0);
    const T* s1 = static_cast<const T*>(p.src1);
    const T* w = static_cast<const T*>(p.w);

    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    // each thread stages 4 A and 4 B elements per K chunk; (row, kq) fixed across chunks
    int a_row[4], a_kq[4], a_h[4], a_w[4];
    long long a_img[4];
    bool a_ok[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int e = tid + i * 256;
        a_row[i] = e >> 4;
        a_kq[i] = e & 15;
        const long long m = m0 + a_row[i];
        a_ok[i] = m < M;
        const long long mm = a_ok[i] ? m : 0;
        a_w[i] = static_cast<int>(mm % p.W);
        a_h[i] = static_cast<int>((mm / p.W) % p.H);
        a_img[i] = mm / (static_cast<long long>(p.W) * p.H);
    }

    for (int k0 = 0; k0 < Kflat; k0 += 16) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int kk = k0 + a_kq[i];
            float va = 0.f, vb = 0.f;
            if (kk < Kflat) {
                const int tap = kk / Ct;
                const int c = kk - tap * Ct;
                const int ky = tap / p.ksize, kx = tap - ky * p.ksize;
                const int hh = a_h[i] + ky - p.pad, ww = a_w[i] + kx - p.pad;
                if (a_ok[i] && hh >= 0 && hh < p.H && ww >= 0 && ww < p.W) {
                    const long long pix = (a_img[i] * p.H + hh) * p.W + ww;
                    va = (c < p.C0) ? ld_as_float(s0 + pix * p.C0 + c)
                                    : ld_as_float(s1 + pix * p.C1 + (c - p.C0));
                }
                const int n = n0 + a_row[i];
                if (n < p.N) vb = ld_as_float(w + (static_cast<long long>(tap) * p.N + n) * Ct + c);
            }
            As[a_kq[i]][a_row[i]] = va;
            Bs[a_kq[i]][a_row[i]] = vb;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            float a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[k][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Bs[k][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }

#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const long long m = m0 + ty * 4 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n >= p.N) continue;
            float v = acc[i][j];
            if (p.bias) v += p.bias[n];
            if (p.relu) v = fmaxf(v, 0.f);
            const bool second = n >= p.split;
            const long long off = second ? m * p.ld1 + (n - p.split) : m * p.ld0 + n;
            void* base = second ? p.dst1 : p.dst0;
            if (p.out_fp32)
                static_cast<float*>(base)[off] = v;
            else
                st_from_float(static_cast<T*>(base) + off, v);
        }
    }
}

int launch_conv_simt(const ConvSimtParams& p, int dtype_fp32, cudaStream_t stream) {
    const long long M = static_cast<long long>(p.IMG) * p.H * p.W;
    dim3 grid(static_cast<unsigned>((M + 63) / 64), static_cast<unsigned>((p.N + 63) / 64));
    if (dtype_fp32)
        conv_simt_kernel<float><<<grid, 256, 0, stream>>>(p);
    else
        conv_simt_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(p);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// ------------------------------------------------------------------------------------------------
// weight gradient:  dw[tap][n][koff + c] += sum_m dz[m, n] * src[m + tap, c]
// tile: 64 flattened (tap, c) rows x 64 n columns, reduction over a slice of the pixels per block
// ------------------------------------------------------------------------------------------------

template <typename T>
__global__ void __launch_bounds__(256) wgrad_simt_kernel(const WgradSimtParams p) {
    __shared__ float As[16][64 + 4];  // [pixel][flattened (tap,c)]
    __shared__ float Bs[16][64 + 4];  // [pixel][n]
    const int Kflat = p.ksize * p.ksize * p.Csrc;
    const long long M = static_cast<long long>(p.IMG) * p.H * p.W;
    const int kk0 = blockIdx.x * 64;
    const int n0 = blockIdx.y * 64;
    const long long m_begin = static_cast<long long>(blockIdx.z) * p.m_per_block;
    const long long m_end = min(m_begin + p.m_per_block, M);
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const T* dz = static_cast<const T*>(p.dz);
    const T* src = static_cast<const T*>(p.src);

    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    // staging assignment: element e = tid + i*256 -> (pixel row r = e / 64, column q = e % 64)
    for (long long mb = m_begin; mb < m_end; mb += 16) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int e = tid + i * 256;
            const int r = e >> 6, q = e & 63;
            const long long m = mb + r;
            float va = 0.f, vb = 0.f;
            if (m < m_end) {
                const int n = n0 + q;
                if (n < p.Nz) vb = ld_as_float(dz + m * p.Nz + n);
                const int kk = kk0 + q;
                if (kk < Kflat) {
                    const int tap = kk / p.Csrc;
                    const int c = kk - tap * p.Csrc;
                    const int ky = tap / p.ksize, kx = tap - ky * p.ksize;
                    const int w_ = static_cast<int>(m % p.W);
                    const int h_ = static_cast<int>((m / p.W) % p.H);
                    const long long img = m / (static_cast<long long>(p.W) * p.H);
                    const int hh = h_ + ky - p.pad, ww = w_ + kx - p.pad;
                    if (hh >= 0 && hh < p.H && ww >= 0 && ww < p.W)
                        va = ld_as_float(src + ((img * p.H + hh) * p.W + ww) * p.Csrc + c);
                }
            }
            As[r][q] = va;
            Bs[r][q] = vb;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            float a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[k][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Bs[k][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int kk = kk0 + ty * 4 + i;
        if (kk >= Kflat) continue;
        const int tap = kk / p.Csrc;
        const int c = kk - tap * p.Csrc;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n >= p.Nz) continue;
            float* o = p.dw + blockIdx.z * p.split_stride + (static_cast<long long>(tap) * p.Nz + n) * p.ldk + p.koff + c;
            if (gridDim.z > 1)
                *o = acc[i][j];
            else
                *o += acc[i][j];
        }
    }
}

int launch_wgrad_simt(WgradSimtParams p, int dtype_fp32, cudaStream_t stream) {
    const long long M = static_cast<long long>(p.IMG) * p.H * p.W;
    const int Kflat = p.ksize * p.ksize * p.Csrc;
    const unsigned gx = (Kflat + 63) / 64, gy = (p.Nz + 63) / 64;
    long long want = (4LL * num_sms() + gx * gy - 1) / (gx * gy);
    long long max_z = (M + 255) / 256;
    if (want > max_z) want = max_z;
    if (want < 1) want = 1;
    if (want > 65535) want = 65535;
    p.m_per_block = ((M + want - 1) / want + 15) / 16 * 16;
    const unsigned gz = static_cast<unsigned>((M + p.m_per_block - 1) / p.m_per_block);
    float* const dw = p.dw;
    const long long ldk = p.ldk;
    const int koff = p.koff;
    p.split_stride = 0;
    if (gz > 1) {
        p.split_stride = static_cast<long long>(Kflat) * p.Nz;
        p.dw = splitk_workspace(stream, gz * static_cast<size_t>(p.split_stride));
        if (!p.dw) {
            set_last_error("wgrad_simt: no split-K workspace (cudaMalloc failed, or growth during graph capture)");
            return B200_ERR_CUDA;
        }
        p.ldk = p.Csrc;
        p.koff = 0;
    }
    dim3 grid(gx, gy, gz);
    if (dtype_fp32)
        wgrad_simt_kernel<float><<<grid, 256, 0, stream>>>(p);
    else
        wgrad_simt_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(p);
    B200_CUDA_CHECK(cudaGetLastError());
    if (gz == 1) return B200_OK;
    return splitk_reduce(p.dw, gz, static_cast<long long>(p.ksize) * p.ksize * p.Nz, p.Csrc, dw, ldk, koff, stream);
}

}  // namespace b200
