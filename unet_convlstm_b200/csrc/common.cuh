// Shared host/device declarations for the b200 ConvLSTM / UNet-block kernels.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

// Status codes returned through the C ABI (include/b200_convlstm.h).
#define B200_OK 0
#define B200_ERR_SHAPE -1       // shape not supported by this entry point (caller may use *_simt)
#define B200_ERR_ALIGN -2       // pointer / leading dimension misaligned
#define B200_ERR_CUDA -3        // a CUDA runtime / driver call failed (see b200_last_error)
#define B200_ERR_ARG -4         // inconsistent arguments
#define B200_ERR_PIPELINE -5    // device-side pipeline watchdog fired

namespace b200 {

void set_last_error(const char* fmt, ...);

#define B200_CUDA_CHECK(expr)                                                                 \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            b200::set_last_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr,                \
                                 cudaGetErrorString(_e));                                     \
            return B200_ERR_CUDA;                                                             \
        }                                                                                     \
    } while (0)

int num_sms();

// first() is true once per device (and call site): cudaFuncSetAttribute settings belong to the device that was
// current when they were made, so a process driving several GPUs has to repeat them on each.
struct PerDeviceOnce {
    bool done[64] = {};
    bool first() {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;
        if (done[dev]) return false;
        done[dev] = true;
        return true;
    }
};
int* device_error_flag();  // one int in device memory, zero unless a watchdog fired
unsigned* device_sync_counter(cudaStream_t stream);  // step counter of the timestep-persistent kernels, per (device, stream)

// Split-K weight gradients without atomics, so that the result does not depend on the order in which the reduction
// splits finish: every split stores its partial dW [rows][cols] to its own slice of a per-(device, stream) workspace,
// then splitk_reduce adds the slices to dw[r * ldk + koff + c] in split order.
// Grows on demand and is kept for the life of the process; nullptr if cudaMalloc fails or if it would have to grow
// while the stream is being captured into a CUDA graph.
float* splitk_workspace(cudaStream_t stream, size_t floats);
int splitk_reduce(const float* ws, int splits, long long rows, int cols, float* dw, long long ldk, int koff,
                  cudaStream_t stream);

// ---- TMA tensor-map construction (driver entry point resolved at run time, no libcuda link) ----
// Activation map over a bf16 NHWC tensor viewed as {C, W, H, B, T}; box = {box_c, Wt, Ht, Bt, 1}.
int make_act_tmap(CUtensorMap* out, const void* base, int C, int W, int H, int B, int T, int box_c,
                  int Wt, int Ht, int Bt, int esize = 2, int atom32 = 0);
// General 5-D bf16 map with explicit element strides between dimensions (dims[0] is contiguous).
int make_tmap_5d(CUtensorMap* out, const void* base, const uint64_t dims[5],
                 const uint64_t strides_elems[4], const uint32_t box[5], int esize = 2, int atom32 = 0);
// Weight map over bf16 [taps][rows][K] viewed as {K, rows, taps}; box = {box_k, box_rows, 1}.
int make_w_tmap(CUtensorMap* out, const void* base, int K, int rows, int taps, int box_k,
                int box_rows, int esize = 2);

// hits / misses of the tensor-map cache since the library was loaded
void tmap_cache_stats(unsigned long long* hits, unsigned long long* misses);

// M-tile geometry: 128 output pixels = Wt x Ht x Bt box (w fastest).  Returns false if the
// spatial shape cannot be tiled by the tensor-core path.
struct MTile {
    int Wt, Ht, Bt;
    int tiles_w, tiles_h, tiles_b;
};
bool plan_mtile(int B, int H, int W, int rows, MTile* mt);

}  // namespace b200
