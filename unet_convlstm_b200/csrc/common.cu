// Host-side utilities: error reporting, device properties, TMA tensor-map encoding.
#include "common.cuh"

#include <signal.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include <map>
#include <mutex>
#include <vector>

namespace b200 {

static thread_local char g_last_error[512] = "";

void set_last_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_last_error, sizeof(g_last_error), fmt, ap);
    va_end(ap);
}
const char* last_error() { return g_last_error; }

int num_sms() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
            n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

// pinned, device-mapped host memory (UVA: same pointer on both sides): the host can still read the barrier id
// after a watchdog trap has killed the context -- including from the SIGABRT handler below, which is how the id
// reaches stderr when the sticky error surfaces inside a destructor (std::terminate) rather than as an exception
static int* g_err_flags[64] = {nullptr};
static std::mutex g_err_mu;
static void (*g_prev_abort)(int) = nullptr;

static void abort_reporter(int sig) {
    for (int d = 0; d < 64; ++d) {
        int* f = g_err_flags[d];
        if (f && *static_cast<volatile int*>(f) != 0) {
            char buf[96];
            int n = snprintf(buf, sizeof(buf), "b200: device %d watchdog flag = %d (see csrc/ptx.cuh mbar_wait tags)\n", d,
                             *static_cast<volatile int*>(f));
            if (n > 0) (void)!write(2, buf, size_t(n));
        }
    }
    signal(sig, g_prev_abort ? g_prev_abort : SIG_DFL);
    raise(sig);
}

int* device_error_flag() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> lk(g_err_mu);
    if (!g_err_flags[dev]) {
        int* p = nullptr;
        if (cudaHostAlloc(&p, sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) return nullptr;
        *p = 0;
        g_err_flags[dev] = p;
        static bool installed = false;
        if (!installed) {
            installed = true;
            void (*prev)(int) = signal(SIGABRT, abort_reporter);
            g_prev_abort = (prev == SIG_ERR || prev == SIG_IGN) ? nullptr : prev;
        }
    }
    return g_err_flags[dev];
}

unsigned* device_sync_counter(cudaStream_t stream) {
    // One counter per (device, stream): two timestep-persistent kernels on different streams may run side by side.
    // The counters of a device come from ONE pool allocated the first time the device launches such a kernel; a
    // stream seen for the first time later only takes the next slot -- no cudaMalloc, no synchronous memset (every
    // launch resets its counter with cudaMemsetAsync on its own stream), so a launch on a new stream is legal inside
    // a CUDA-graph capture (ADVICE r01: the capture stream of torch.cuda.graph is never the warm-up stream).
    constexpr int SLOTS = 256;
    struct Pool {
        unsigned* base = nullptr;
        int used = 0;
        std::map<cudaStream_t, unsigned*> by_stream;
    };
    static Pool pools[64];
    static std::mutex mu;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> lk(mu);
    Pool& pool = pools[dev];
    auto it = pool.by_stream.find(stream);
    if (it != pool.by_stream.end()) return it->second;
    if (!pool.base) {
        unsigned* p = nullptr;
        if (cudaMalloc(&p, SLOTS * 32) != cudaSuccess) return nullptr;  // 32 bytes apart: one L2 sector per counter
        pool.base = p;
    }
    if (pool.used == SLOTS) return nullptr;
    unsigned* slot = pool.base + 8 * pool.used++;
    pool.by_stream[stream] = slot;
    return slot;
}

float* splitk_workspace(cudaStream_t stream, size_t floats) {
    struct Buf {
        float* ptr = nullptr;
        size_t floats = 0;
        std::vector<float*> retired;
    };
    static std::map<std::pair<int, cudaStream_t>, Buf> bufs;
    static std::mutex mu;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    std::lock_guard<std::mutex> lk(mu);
    Buf& b = bufs[{dev, stream}];
    if (b.floats < floats) {
        // no allocation inside a CUDA-graph capture: an eager call of the same shape must size the buffer first
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(stream, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone) return nullptr;
        // the old buffer stays allocated: launches already enqueued, or captured into a graph, still use it; growing
        // at least twofold bounds what is kept to the size of the current buffer
        if (b.ptr) b.retired.push_back(b.ptr);
        if (floats < 2 * b.floats) floats = 2 * b.floats;
        b.ptr = nullptr;
        b.floats = 0;
        void* p = nullptr;
        if (cudaMalloc(&p, floats * sizeof(float)) != cudaSuccess) return nullptr;
        b.ptr = static_cast<float*>(p);
        b.floats = floats;
    }
    return b.ptr;
}

__global__ void splitk_reduce_kernel(const float* __restrict__ ws, int splits, long long rows, int cols,
                                     float* __restrict__ dw, long long ldk, int koff) {
    const long long n = rows * cols;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        float s = ws[i];
        for (int k = 1; k < splits; ++k) s += ws[k * n + i];
        const long long r = i / cols;
        dw[r * ldk + koff + (i - r * cols)] += s;
    }
}

int splitk_reduce(const float* ws, int splits, long long rows, int cols, float* dw, long long ldk, int koff,
                  cudaStream_t stream) {
    const long long n = rows * cols;
    long long blocks = (n + 255) / 256;
    if (blocks > 8LL * num_sms()) blocks = 8LL * num_sms();
    splitk_reduce_kernel<<<static_cast<unsigned>(blocks), 256, 0, stream>>>(ws, splits, rows, cols, dw, ldk, koff);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// ----------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &p, 12000, cudaEnableDefault,
                                             &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    });
    return fn;
}

static CUtensorMapSwizzle swizzle_for_bytes(int inner_bytes) {
    switch (inner_bytes) {
        case 128: return CU_TENSOR_MAP_SWIZZLE_128B;
        case 64: return CU_TENSOR_MAP_SWIZZLE_64B;
        case 32: return CU_TENSOR_MAP_SWIZZLE_32B;
        default: return CU_TENSOR_MAP_SWIZZLE_NONE;
    }
}

// ----------------------------------------------------------------------------------------------
// Tensor-map cache (SURVEY.md section 8b: "TMA descriptors cached per (ptr, shape)").  A training step encodes the
// same ~300 maps again every step (the caching allocator hands out the same addresses); the 128-byte CUtensorMap is a
// pure function of (base, dims, strides, box), so a direct-mapped table keyed by those replaces the driver call by one
// compare.  Collisions simply re-encode.
// ----------------------------------------------------------------------------------------------
struct TmapKey {
    const void* base;
    uint64_t d[5];
    uint64_t s[4];
    uint32_t b[5];
    uint32_t rank;
    bool operator==(const TmapKey& o) const { return memcmp(this, &o, sizeof(TmapKey)) == 0; }
};
struct TmapSlot {
    TmapKey key;
    CUtensorMap map;
    bool used;
};
static constexpr int TMAP_SLOTS = 2048;
static TmapSlot* g_tmap_cache = nullptr;
static std::mutex g_tmap_mu;
static unsigned long long g_tmap_hits = 0, g_tmap_misses = 0;

static uint64_t tmap_hash(const TmapKey& k) {
    const uint64_t* w = reinterpret_cast<const uint64_t*>(&k);
    uint64_t h = 1469598103934665603ull;
    for (size_t i = 0; i < sizeof(TmapKey) / 8; ++i) h = (h ^ w[i]) * 1099511628211ull;
    return h ^ (h >> 29);
}
static bool tmap_lookup(const TmapKey& k, CUtensorMap* out) {
    std::lock_guard<std::mutex> lk(g_tmap_mu);
    if (!g_tmap_cache) g_tmap_cache = static_cast<TmapSlot*>(calloc(TMAP_SLOTS, sizeof(TmapSlot)));
    if (!g_tmap_cache) return false;
    TmapSlot& sl = g_tmap_cache[tmap_hash(k) % TMAP_SLOTS];
    if (sl.used && sl.key == k) {
        *out = sl.map;
        ++g_tmap_hits;
        return true;
    }
    ++g_tmap_misses;
    return false;
}
static void tmap_store(const TmapKey& k, const CUtensorMap& m) {
    std::lock_guard<std::mutex> lk(g_tmap_mu);
    if (!g_tmap_cache) return;
    TmapSlot& sl = g_tmap_cache[tmap_hash(k) % TMAP_SLOTS];
    sl.key = k;
    sl.map = m;
    sl.used = true;
}
void tmap_cache_stats(unsigned long long* hits, unsigned long long* misses) {
    std::lock_guard<std::mutex> lk(g_tmap_mu);
    *hits = g_tmap_hits;
    *misses = g_tmap_misses;
}

int make_tmap_5d(CUtensorMap* out, const void* base, const uint64_t dims[5],
                 const uint64_t strides_elems[4], const uint32_t box[5], int esize, int atom32) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) {
        set_last_error("cuTensorMapEncodeTiled entry point not available");
        return B200_ERR_CUDA;
    }
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) {
        set_last_error("TMA base pointer %p not 16-byte aligned", base);
        return B200_ERR_ALIGN;
    }
    TmapKey key;
    memset(&key, 0, sizeof(key));
    key.base = base;
    key.rank = 5u | (uint32_t(esize) << 8) | (uint32_t(atom32) << 16);
    for (int i = 0; i < 5; ++i) { key.d[i] = dims[i]; key.b[i] = box[i]; }
    for (int i = 0; i < 4; ++i) key.s[i] = strides_elems[i];
    if (tmap_lookup(key, out)) return B200_OK;
    cuuint64_t gdim[5], gstr[4];
    cuuint32_t bx[5], estr[5];
    for (int i = 0; i < 5; ++i) {
        gdim[i] = dims[i];
        bx[i] = box[i];
        estr[i] = 1;
    }
    for (int i = 0; i < 4; ++i) {
        gstr[i] = strides_elems[i] * uint64_t(esize);  // bf16 (2) or fp32 (4)
        if (gstr[i] % 16 != 0) {
            set_last_error("TMA stride %d = %llu bytes not a multiple of 16", i,
                           (unsigned long long)gstr[i]);
            return B200_ERR_ALIGN;
        }
    }
    CUresult r = fn(out, esize == 4 ? CU_TENSOR_MAP_DATA_TYPE_TFLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5,
                    const_cast<void*>(base), gdim, gstr, bx,
                    estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    // atom32: the 128-byte swizzle on 32-byte atoms (4-row period) -- what an MN-major operand of 32-bit
                    // elements needs (UMMA layout type SWIZZLE_128B_BASE32B, wgrad_tc.cu tf32 mode)
                    atom32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : swizzle_for_bytes(int(box[0]) * esize),
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_last_error(
            "cuTensorMapEncodeTiled(5d) failed: %d dims={%llu,%llu,%llu,%llu,%llu} box={%u,%u,%u,%u,%u}",
            int(r), (unsigned long long)gdim[0], (unsigned long long)gdim[1],
            (unsigned long long)gdim[2], (unsigned long long)gdim[3], (unsigned long long)gdim[4],
            bx[0], bx[1], bx[2], bx[3], bx[4]);
        return B200_ERR_CUDA;
    }
    tmap_store(key, *out);
    return B200_OK;
}

int make_act_tmap(CUtensorMap* out, const void* base, int C, int W, int H, int B, int T, int box_c,
                  int Wt, int Ht, int Bt, int esize, int atom32) {
    uint64_t dims[5] = {uint64_t(C), uint64_t(W), uint64_t(H), uint64_t(B), uint64_t(T)};
    uint64_t str[4] = {uint64_t(C), uint64_t(C) * W, uint64_t(C) * W * H, uint64_t(C) * W * H * B};
    uint32_t box[5] = {uint32_t(box_c), uint32_t(Wt), uint32_t(Ht), uint32_t(Bt), 1u};
    return make_tmap_5d(out, base, dims, str, box, esize, atom32);
}

int make_w_tmap(CUtensorMap* out, const void* base, int K, int rows, int taps, int box_k,
                int box_rows, int esize) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) {
        set_last_error("cuTensorMapEncodeTiled entry point not available");
        return B200_ERR_CUDA;
    }
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || ((K * esize) % 16) != 0) {
        set_last_error("weight TMA map: base %p / K=%d misaligned", base, K);
        return B200_ERR_ALIGN;
    }
    TmapKey key;
    memset(&key, 0, sizeof(key));
    key.base = base;
    key.rank = 3u | (uint32_t(esize) << 8);
    key.d[0] = uint64_t(K); key.d[1] = uint64_t(rows); key.d[2] = uint64_t(taps);
    key.b[0] = uint32_t(box_k); key.b[1] = uint32_t(box_rows); key.b[2] = 1;
    if (tmap_lookup(key, out)) return B200_OK;
    cuuint64_t gdim[3] = {cuuint64_t(K), cuuint64_t(rows), cuuint64_t(taps)};
    cuuint64_t gstr[2] = {cuuint64_t(K) * esize, cuuint64_t(K) * esize * rows};
    cuuint32_t bx[3] = {cuuint32_t(box_k), cuuint32_t(box_rows), 1u};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(out, esize == 4 ? CU_TENSOR_MAP_DATA_TYPE_TFLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3,
                    const_cast<void*>(base), gdim, gstr, bx,
                    estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for_bytes(box_k * esize),
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_last_error("cuTensorMapEncodeTiled(3d weights) failed: %d K=%d rows=%d taps=%d box={%d,%d}",
                       int(r), K, rows, taps, box_k, box_rows);
        return B200_ERR_CUDA;
    }
    tmap_store(key, *out);
    return B200_OK;
}

static bool is_pow2(int x) { return x > 0 && (x & (x - 1)) == 0; }
static int pow2_ceil(int x) {
    int p = 1;
    while (p < x) p <<= 1;
    return p;
}

bool plan_mtile(int B, int H, int W, int rows, MTile* mt) {
    if (B <= 0 || H <= 0 || W <= 0) return false;
    int Wt;
    if (W >= rows) {
        if (W % rows != 0) return false;
        Wt = rows;
    } else {
        if (!is_pow2(W)) return false;
        Wt = W;
    }
    int Ht = rows / Wt;
    int hp = pow2_ceil(H);
    if (Ht > hp) Ht = hp;
    int Bt = rows / (Wt * Ht);
    if (Bt > 256 || Ht > 256 || Wt > 256) return false;
    mt->Wt = Wt;
    mt->Ht = Ht;
    mt->Bt = Bt;
    mt->tiles_w = W / Wt;
    mt->tiles_h = (H + Ht - 1) / Ht;
    mt->tiles_b = (B + Bt - 1) / Bt;
    return true;
}

}  // namespace b200

extern "C" const char* b200_last_error(void) { return b200::last_error(); }
