// Weight gradient of the 64-channel 3x3 layers with the source tile loaded ONCE per pixel block ("halo" variant of
// wgrad_tc.cu's stacked mode; the wgrad counterpart of conv_halo.cu).
//
//   dW[tap][n][koff + c] (+)= sum_{t, pixel p} dz[t, p, n] * src[t, p + tap, c]          (Csrc = 64, 3x3)
//
// wgrad_tc.cu loads one tap-shifted source box per tap: nine 8 KB boxes per 64 pixels, and at 64 channels the
// kernel sits at the L2 -> shared-memory fill limit (profiles/r01_wgrad_2cta_ab.txt).  Here a pixel block is
// Ht = 128 / W whole image rows; ONE TMA box {64 channels, W + 2, Ht + 2} starting at (w, h) = (-1, h0 - 1) brings
// the block with its halo (out-of-bounds fill = zero padding) as (W + 2) * (Ht + 2) rows of 128 bytes.  The pixels of
// an MMA K step (16 consecutive pixels of one image row) shifted by tap (ky, kx) are 16 CONSECUTIVE rows of that tile
// starting at row (hl + ky) * (W + 2) + w + kx, so every tap is just a different start address of the MN-major A
// descriptor (the 128-byte swizzle is a function of the absolute shared-memory address, as conv_halo.cu relies on),
// and two taps are stacked along M = 128 with the descriptor's leading-dimension offset = the distance between them.
// Source traffic per 128 pixels drops from 18 x 8 KB to one 33 KB box; the dz box is shared by all nine taps
// (five M = 128 accumulators of 64 columns in TMEM).
//
// 16-channel sources (the UNet's first layer: 2 input channels zero-padded to 16): rows of 32 bytes, 32-byte swizzle;
// the M = 128 operand has eight 16-channel slots, three of which hold the taps (0,kx) (1,kx) (2,kx) of one kx --
// equally spaced by one tile row pitch, which is what a single leading-dimension offset can express -- so three
// MMAs (kx = 0, 1, 2) per K step; the other five slots read rows past the taps and are never stored.
//
// Warp roles: warp 0 TMA producer, warp 1 MMA issuer, warp 2 TMEM allocator, warps 4-7 epilogue (transposed fp32
// stores; split-K partials go to the workspace slices, as in wgrad_tc.cu).
#include "common.cuh"
#include "ptx.cuh"

namespace b200 {

static constexpr int WH_THREADS = 256;
static constexpr int WH_RB = 128;     // pixels per block
static constexpr int WH_STAGES = 4;    // at most (barrier layout); p.stages are used
static constexpr int WH_GROUPS = 5;   // tap pairs (0,1) (2,3) (4,5) (6,7) (8,-)
static constexpr int WH_DZ_BYTES = WH_RB * 128;

struct WgradHaloParams {
    int T, B, H, W;
    int Nz;
    int Cs;            // source channels: 64 or 16
    int Ht;            // image rows per block = 128 / W
    int P;             // padded tile width W + 2
    int blocks_per_img;
    int num_rblocks, rb_per_split, splits;
    int s_tiles;       // Nz / 64
    uint32_t src_bytes, src_stage_bytes;
    int stages;        // pipeline depth that fits in shared memory (3 or 4)
    float* dw;         // the split-K workspace, split s at dw + s * split_stride
    long long ldk;
    int koff;
    long long split_stride;
    int* err_flag;
};

__global__ void __launch_bounds__(WH_THREADS, 1)
wgrad_halo_kernel(const __grid_constant__ CUtensorMap tm_dz, const __grid_constant__ CUtensorMap tm_src,
                  const WgradHaloParams p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t stage_bytes = p.src_stage_bytes + WH_DZ_BYTES;
    const uint32_t bar_base = smem_base + p.stages * stage_bytes;
    auto full = [&](int s) { return bar_base + 8u * s; };
    auto empty = [&](int s) { return bar_base + 8u * (WH_STAGES + s); };
    const uint32_t tfull = bar_base + 8u * (2 * WH_STAGES);
    const uint32_t tempty = tfull + 8u;
    const uint32_t tmem_ptr_addr = tfull + 16u;
    volatile uint32_t* tmem_ptr_gen =
        reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_ptr_addr - smem_u32(smem_raw)));

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const int lane = threadIdx.x & 31;
    const int total_units = p.s_tiles * p.splits;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tm_dz);
        prefetch_tmap(&tm_src);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < WH_STAGES; ++s) {
            mbar_init(full(s), 1);
            mbar_init(empty(s), 1);
        }
        mbar_init(tfull, 1);
        mbar_init(tempty, 4);
        fence_mbar_init();
    }
    if (warp == 2) {
        tmem_alloc(tmem_ptr_addr, 512);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_gen;

    if (warp == 0) {
        // =================================== TMA producer ===================================
        int stage = 0;
        uint32_t phase = 0;
        for (int unit = blockIdx.x; unit < total_units; unit += gridDim.x) {
            const int split = unit / p.s_tiles;
            const int s0 = (unit - split * p.s_tiles) * 64;
            const int rb_begin = split * p.rb_per_split;
            const int rb_end = min(rb_begin + p.rb_per_split, p.num_rblocks);
            int m = rb_begin;
            int hb = m % p.blocks_per_img;
            m /= p.blocks_per_img;
            int b = m % p.B;
            int t = m / p.B;
            for (int rb = rb_begin; rb < rb_end; ++rb) {
                mbar_wait(empty(stage), phase ^ 1u, p.err_flag, 6000 + 500 + stage);
                if (elect_one()) {
                    const uint32_t fb = full(stage);
                    const uint32_t dst = smem_base + stage * stage_bytes;
                    const int h0 = hb * p.Ht;
                    mbar_arrive_expect_tx(fb, p.src_bytes + WH_DZ_BYTES);
                    tma_load_5d(dst, &tm_src, fb, 0, -1, h0 - 1, b, t);                   // source block with its halo
                    tma_load_5d(dst + p.src_stage_bytes, &tm_dz, fb, s0, 0, h0, b, t);    // 64 dz channels of the block
                }
                __syncwarp();
                if (++stage == p.stages) {
                    stage = 0;
                    phase ^= 1u;
                }
                if (++hb == p.blocks_per_img) {
                    hb = 0;
                    if (++b == p.B) {
                        b = 0;
                        ++t;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // =================================== MMA issuer =====================================
        const uint32_t idesc = make_idesc_bf16(128, 64, 1, 1);  // both operands MN-major
        const uint32_t row_lo = 128u >> 4;                      // one pixel row of the dz tile = 128 bytes
        const uint32_t srow = p.Cs * 2;                         // one pixel row of the source tile: 128 or 32 bytes
        const uint32_t srow_lo = srow >> 4;
        const uint32_t ltS = p.Cs == 64 ? 2u : 6u;              // 128-byte / 32-byte swizzle
        // A descriptors: the leading-dimension offset is the distance between the stacked taps
        const uint64_t hiA_near = make_smem_desc(0, srow, 8u * srow, ltS);            // (ky, kx) , (ky, kx + 1)
        const uint64_t hiA_wrap = make_smem_desc(0, p.W * srow, 8u * srow, ltS);      // (ky, 2)  , (ky + 1, 0)
        const uint64_t hiA_col = make_smem_desc(0, p.P * srow, 8u * srow, ltS);       // (0, kx), (1, kx), (2, kx), ...
        const uint64_t hiB = make_smem_desc(0, WH_DZ_BYTES, 1024, 2);
        const int steps_per_row = p.W >> 4;
        const uint32_t smem_lo = (smem_base & 0x3FFFFu) >> 4;
        int stage = 0;
        uint32_t phase = 0, pt = 0;
        for (int unit = blockIdx.x; unit < total_units; unit += gridDim.x) {
            const int split = unit / p.s_tiles;
            const int rb_begin = split * p.rb_per_split;
            const int rb_end = min(rb_begin + p.rb_per_split, p.num_rblocks);
            mbar_wait(tempty, pt ^ 1u, p.err_flag, 6000 + 700);
            tc_fence_after();
            uint32_t accum = 0;
            for (int rb = rb_begin; rb < rb_end; ++rb) {
                mbar_wait(full(stage), phase, p.err_flag, 6000 + 600 + stage);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t src_lo = smem_lo + stage * (stage_bytes >> 4);
                    const uint32_t dz_lo = src_lo + (p.src_stage_bytes >> 4);
                    int hl = 0, wstep = 0;
                    for (int ks = 0; ks < WH_RB / 16; ++ks) {
                        const uint64_t bdesc = hiB | (dz_lo + ks * 16 * row_lo);
                        const uint32_t row0 = hl * p.P + wstep * 16;  // tile row of tap (0, 0) for this K step
                        if (p.Cs == 64) {
                            // tap pairs: (0,0)(0,1) | (0,2)(1,0) | (1,1)(1,2) | (2,0)(2,1) | (2,2)(-)
                            umma_bf16(tmem_base + 0 * 64, hiA_near | (src_lo + (row0) * srow_lo), bdesc, idesc, accum);
                            umma_bf16(tmem_base + 1 * 64, hiA_wrap | (src_lo + (row0 + 2) * srow_lo), bdesc, idesc, accum);
                            umma_bf16(tmem_base + 2 * 64, hiA_near | (src_lo + (row0 + p.P + 1) * srow_lo), bdesc, idesc, accum);
                            umma_bf16(tmem_base + 3 * 64, hiA_near | (src_lo + (row0 + 2 * p.P) * srow_lo), bdesc, idesc, accum);
                            umma_bf16(tmem_base + 4 * 64, hiA_near | (src_lo + (row0 + 2 * p.P + 2) * srow_lo), bdesc, idesc, accum);
                        } else {
                            // tap columns: slots 0..2 of the M operand = (0,kx) (1,kx) (2,kx), one MMA per kx
                            umma_bf16(tmem_base + 0 * 64, hiA_col | (src_lo + (row0) * srow_lo), bdesc, idesc, accum);
                            umma_bf16(tmem_base + 1 * 64, hiA_col | (src_lo + (row0 + 1) * srow_lo), bdesc, idesc, accum);
                            umma_bf16(tmem_base + 2 * 64, hiA_col | (src_lo + (row0 + 2) * srow_lo), bdesc, idesc, accum);
                        }
                        accum = 1u;
                        if (++wstep == steps_per_row) {
                            wstep = 0;
                            ++hl;
                        }
                    }
                    umma_commit(empty(stage));
                }
                __syncwarp();
                accum = 1u;
                if (++stage == p.stages) {
                    stage = 0;
                    phase ^= 1u;
                }
            }
            if (elect_one()) umma_commit(tfull);
            __syncwarp();
            pt ^= 1u;
        }
    } else if (warp >= 4) {
        // =================================== epilogue =======================================
        const int q = static_cast<int>(threadIdx.x >> 5) - 4;
        const int r = q * 32 + lane;
        // accumulator row = (slot, source channel): 64 channels -> 2 slots (the tap pair), 16 channels -> 8 slots of
        // which 0..2 are the taps (ky = slot) of the group's kx
        const int gi = p.Cs == 64 ? (r >> 6) : (r >> 4);
        const int c = p.Cs == 64 ? (r & 63) : (r & 15);
        const int ngroups = p.Cs == 64 ? WH_GROUPS : 3;
        uint32_t pt = 0;
        for (int unit = blockIdx.x; unit < total_units; unit += gridDim.x) {
            const int split = unit / p.s_tiles;
            const int s0 = (unit - split * p.s_tiles) * 64;
            mbar_wait(tfull, pt, p.err_flag, 6000 + 800);
            pt ^= 1u;
            tc_fence_after();
            for (int g = 0; g < ngroups; ++g) {
                const int tp = p.Cs == 64 ? 2 * g + gi : gi * 3 + g;
                const bool valid = p.Cs == 64 ? tp < 9 : gi < 3;
                float* row = p.dw + split * p.split_stride + (static_cast<long long>(valid ? tp : 0) * p.Nz + s0) * p.ldk + p.koff + c;
                const uint32_t t_row = tmem_base + g * 64 + (uint32_t(q * 32) << 16);
#pragma unroll 1
                for (int c16 = 0; c16 < 4; ++c16) {
                    uint32_t v[16];
                    tmem_ld16(t_row + c16 * 16, v);
                    tmem_ld_wait();
                    if (!valid) continue;
                    float* o = row + static_cast<long long>(c16) * 16 * p.ldk;  // transposed: lanes = source channels
#pragma unroll
                    for (int j = 0; j < 16; ++j) o[j * p.ldk] = __uint_as_float(v[j]);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

bool wgrad_halo_supported(int Nz, int Csrc, int B, int H, int W, int ksize) {
    if ((Csrc != 64 && Csrc != 16) || ksize != 3 || Nz % 64 != 0) return false;
    if (!(W == 16 || W == 32 || W == 64 || W == 128)) return false;
    const int Ht = WH_RB / W;
    return H % Ht == 0 && B > 0;
}

// Tiling and reduction split of a launch: every field of p except the pointers, the output layout and the stages.
static int plan_wgrad_halo(int Nz, int Csrc, int T, int B, int H, int W, WgradHaloParams* pp) {
    if (!wgrad_halo_supported(Nz, Csrc, B, H, W, 3)) {
        set_last_error("wgrad_halo: shape not supported");
        return B200_ERR_SHAPE;
    }
    WgradHaloParams& p = *pp;
    p = {};
    p.T = T; p.B = B; p.H = H; p.W = W; p.Nz = Nz; p.Cs = Csrc;
    p.Ht = WH_RB / W;
    p.P = W + 2;
    p.blocks_per_img = H / p.Ht;
    p.num_rblocks = T * B * p.blocks_per_img;
    p.s_tiles = Nz / 64;
    p.src_bytes = static_cast<uint32_t>(p.P) * (p.Ht + 2) * static_cast<uint32_t>(Csrc * 2);
    p.src_stage_bytes = (p.src_bytes + 1023u) & ~1023u;
    const int nsm = num_sms();
    int max_splits = (p.num_rblocks + 3) / 4;
    if (max_splits > 4 * nsm) max_splits = 4 * nsm;
    if (max_splits < 1) max_splits = 1;
    int best = 1;
    double best_cost = 1e30;
    for (int s = 1; s <= max_splits; ++s) {
        const long long units = static_cast<long long>(p.s_tiles) * s;
        const double cost = static_cast<double>((units + nsm - 1) / nsm) / s;
        if (cost < best_cost * 0.97) {
            best_cost = cost;
            best = s;
        }
    }
    p.rb_per_split = (p.num_rblocks + best - 1) / best;
    p.splits = (p.num_rblocks + p.rb_per_split - 1) / p.rb_per_split;
    return B200_OK;
}

int wgrad_halo_splits(int Nz, int Csrc, int T, int B, int H, int W) {
    WgradHaloParams p;
    const int rc = plan_wgrad_halo(Nz, Csrc, T, B, H, W, &p);
    return rc == B200_OK ? p.splits : rc;
}

// dw += the weight gradient, at any split count (see launch_wgrad_tc)
int launch_wgrad_halo(const void* dz, int Nz, const void* src, int Csrc, int T, int B, int H, int W, float* dw,
                      long long ldk, int koff, cudaStream_t stream) {
    WgradHaloParams p;
    int rc = plan_wgrad_halo(Nz, Csrc, T, B, H, W, &p);
    if (rc != B200_OK) return rc;
    const int nsm = num_sms();
    p.split_stride = 9LL * Nz * Csrc;
    p.dw = splitk_workspace(stream, static_cast<size_t>(p.splits) * p.split_stride);
    if (!p.dw) {
        set_last_error("%s: no split-K workspace (cudaMalloc failed, or growth during graph capture)", __func__);
        return B200_ERR_CUDA;
    }
    p.ldk = Csrc;
    p.koff = 0;
    p.err_flag = device_error_flag();

    CUtensorMap tz, ts;
    rc = make_act_tmap(&tz, dz, Nz, W, H, B, T, 64, W, p.Ht, 1);
    if (rc != B200_OK) return rc;
    rc = make_act_tmap(&ts, src, Csrc, W, H, B, T, Csrc, p.P, p.Ht + 2, 1);
    if (rc != B200_OK) return rc;
    const int stage_bytes = static_cast<int>(p.src_stage_bytes + WH_DZ_BYTES);
    // The MMAs read source-tile rows past the loaded box: the unused second tap of the (2,2) pair (64 channels), and
    // slots 3..7 of the M operand, which sit 3P..7P rows after the taps (16 channels).  Those rows are never stored,
    // but they must lie inside the shared-memory allocation.  From a stage other than the last they fall into the next
    // stage; the last stage needs `tail` bytes after it, which also hold the barriers (256 bytes).  The 16-channel
    // first layer at W = 128 (P = 130, one image row per block) reads 3.5 KB past its stage: without this tail the
    // last stage read past the end of shared memory and the launch stopped with an illegal-address error.
    const int row0_max = (p.Ht - 1) * p.P + W - 16;  // tile row of tap (0, 0) in the last K step of a block
    const int read_end = (Csrc == 64 ? row0_max + 2 * p.P + 2 + 1 + 16 : row0_max + 2 + 7 * p.P + 16) * Csrc * 2;
    const int tail = read_end - stage_bytes > 256 ? read_end - stage_bytes : 256;
    p.stages = (227 * 1024 - 1024 - tail) / stage_bytes;
    if (p.stages > WH_STAGES) p.stages = WH_STAGES;
    if (p.stages < 2) {
        set_last_error("wgrad_halo: tile does not fit in shared memory");
        return B200_ERR_SHAPE;
    }
    const int smem = p.stages * stage_bytes + 1024 + tail;
    static PerDeviceOnce attr_once;  // kernel attributes are per device
    if (attr_once.first()) {
        B200_CUDA_CHECK(cudaFuncSetAttribute(wgrad_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        // the whole unified L1/shared array as shared memory: the kernel itself only needs its ring, but the
        // remainder lets HBM-bound blocks of another stream (BatchNorm sums: 9 KB static) share the SM when the
        // weight gradient runs on the background stream (with the default carve-out the next step is 196 KB)
        B200_CUDA_CHECK(cudaFuncSetAttribute(wgrad_halo_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                             cudaSharedmemCarveoutMaxShared));
    }
    const int total = p.s_tiles * p.splits;
    const int grid = total < nsm ? total : nsm;
    wgrad_halo_kernel<<<grid, WH_THREADS, smem, stream>>>(tz, ts, p);
    B200_CUDA_CHECK(cudaGetLastError());
    return splitk_reduce(p.dw, p.splits, 9LL * Nz, Csrc, dw, ldk, koff, stream);
}

}  // namespace b200
