// Weight-gradient GEMM on the sm_100a tensor cores (conv backward-weight, batched over the
// whole sequence / frame batch):
//
//   dW[tap][n][koff + c] (+)= sum_{t, pixel p} dz[t, p, n] * src[t, p + tap, c]
//
// i.e. the autograd weight gradient of nn.Conv2d (reference train/unet.py:19 for the ConvLSTM
// gate conv -- summed over all T timesteps of BPTT --, :70-71 for the UNet blocks).
//
// Both operands are read straight from their NHWC tensors, where the *channel* index is
// contiguous and the pixel (reduction) index is strided: both UMMA operands are therefore
// "MN-major".  A TMA box {cw channels, Wt, Ht, Bt} (64 pixels) lands in smem as [pixel][cw] rows
// with the 128/64/32-byte swizzle, which is exactly the canonical MN-major layout
//     ((8 elem, cw/8, m), (8 pixels, k)) : ((1, 8, LBO), (cw, SBO))
// with SBO = 8 pixel rows and LBO = one whole box (next channel chunk).  The tap shift and the
// zero padding are the TMA coordinates / out-of-bounds fill of the source box, as in conv_tc.cu.
//
// The kernel is bound by the L2 -> shared-memory fill rate, not by the tensor pipe, so it is
// organised to load as few bytes per MMA as possible:
//   * dz does not depend on the tap.  One dz box (the "shared" operand S) is loaded per 64-pixel
//     block and re-used by up to GU taps / tap groups, each with its own TMEM accumulator
//     (GU * BLOCK_N <= 512 columns); only the tap-shifted source boxes (the "varying" operand V)
//     are loaded per tap.  S and V live in two independent smem rings.
//   * Normal mode: A = dz (M = 128 dz channels), B = source channels (N <= 256).
//   * Stacked mode (source with 16/32/64 channels, the full-resolution UNet layers): an M tile of
//     128 dz channels would be half empty, so the roles are swapped: A = G = 128/Csrc tap-shifted
//     source boxes stacked along M (rows = (tap, source channel)), B = dz channels (N).
//
// Work units = (reduction split) x (tap-group set, S tile, V tile); every split, a single one too, stores its
// partial sums to its own workspace slice and splitk_reduce (common.cu) adds them to dw in split order, so the
// result is the same from run to run and is added to dw at any split count.
// Warp roles: warp 0 TMA producer, warp 1 MMA issuer, warp 2 TMEM allocator, warps 4-7 epilogue.
#include "common.cuh"
#include "ptx.cuh"

namespace b200 {

static constexpr int WG_BLOCK_M = 128;
static constexpr int WG_RB = 64;  // pixels per pipeline stage
static constexpr int WG_THREADS = 320;  // warps 0,2,3,8,9 TMA producers, 1 MMA issuer, 4-7 epilogue

struct WgradParams {
    int T, B, H, W;
    int Nz;          // channels of dz (rows of dW)
    int Csrc;        // channels of the source (columns written)
    int ksize, pad, taps;
    int cwS, cwV;    // channel chunk widths (64/32/16) of dz / source boxes
    int Wt, Ht, Bt, tiles_w, tiles_h, tiles_b;  // 64-pixel box geometry
    int num_rblocks; // T * tiles_w * tiles_h * tiles_b
    int rb_per_split, splits;
    int G;           // taps per group (stacked mode: 128 / Csrc; normal mode: 1)
    int ngroups;     // ceil(taps / G)
    int GU;          // groups (accumulators) per unit
    int ngsets;      // ceil(ngroups / GU)
    int s_tiles, v_tiles, out_tiles;
    float* dw;       // the split-K workspace, split s at dw + s * split_stride: [taps][Nz][ldk = Csrc], koff = 0
    long long ldk;
    int koff;
    long long split_stride;
    int* err_flag;
    int in_fp32;     // 1: dz and src are fp32 tensors, tcgen05 kind::tf32 (the "tf32" precision mode); a pipeline stage
                     // then holds 32 pixels instead of 64 -- the same bytes, the same four MMAs (K = 8 pixels each)
};

template <int BLOCK_N, bool STACKED>
struct WgCfg {
    static constexpr int A_BYTES = WG_BLOCK_M * WG_RB * 2;  // 16 KB: the M = 128 operand
    static constexpr int B_BYTES = BLOCK_N * WG_RB * 2;
    static constexpr int V_BYTES = STACKED ? A_BYTES : B_BYTES;  // varying (source) operand
    static constexpr int S_BYTES = STACKED ? B_BYTES : A_BYTES;  // shared (dz) operand
    static constexpr int SV = STACKED ? (BLOCK_N == 256 ? 6 : 8) : (BLOCK_N == 256 ? 5 : (BLOCK_N == 128 ? 6 : 8));
    static constexpr int SS = STACKED ? (BLOCK_N == 64 ? 4 : 3) : (BLOCK_N == 256 ? 3 : 4);
    static constexpr int MAX_GU = 512 / BLOCK_N;
    static constexpr int SMEM_BYTES = SV * V_BYTES + SS * S_BYTES + 1024 + 256;
};

struct WgUnit {
    int split, gset, s0, v0, scols, vcols, ngr;
};

template <int BLOCK_N, bool STACKED>
__device__ __forceinline__ WgUnit wg_decode(const WgradParams& p, int unit) {
    WgUnit u;
    u.split = unit / p.out_tiles;
    int ot = unit - u.split * p.out_tiles;
    const int vt = ot % p.v_tiles;
    ot /= p.v_tiles;
    const int st = ot % p.s_tiles;
    u.gset = ot / p.s_tiles;
    if (STACKED) {
        u.s0 = st * BLOCK_N;  // dz channels are the N operand
        u.scols = min(BLOCK_N, p.Nz - u.s0);
        u.v0 = 0;
        u.vcols = WG_BLOCK_M;
    } else {
        u.s0 = st * WG_BLOCK_M;  // dz channels are the M operand
        u.scols = min(WG_BLOCK_M, p.Nz - u.s0);
        u.v0 = vt * BLOCK_N;
        u.vcols = min(BLOCK_N, p.Csrc - u.v0);
    }
    u.ngr = min(p.GU, p.ngroups - u.gset * p.GU);
    return u;
}

template <int BLOCK_N, bool STACKED>
__global__ void __launch_bounds__(WG_THREADS, 1)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap tm_dz, const __grid_constant__ CUtensorMap tm_src,
                const WgradParams p) {
    using Cfg = WgCfg<BLOCK_N, STACKED>;
    constexpr int SV = Cfg::SV, SS = Cfg::SS;

    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t v_base = smem_base;
    const uint32_t s_base = smem_base + SV * Cfg::V_BYTES;
    const uint32_t bar_base = s_base + SS * Cfg::S_BYTES;
    auto vfull = [&](int s) { return bar_base + 8u * s; };
    auto vempty = [&](int s) { return bar_base + 8u * (SV + s); };
    auto sfull = [&](int s) { return bar_base + 8u * (2 * SV + s); };
    auto sempty = [&](int s) { return bar_base + 8u * (2 * SV + SS + s); };
    const uint32_t tfull = bar_base + 8u * (2 * SV + 2 * SS);
    const uint32_t tempty = tfull + 8u;
    const uint32_t tmem_ptr_addr = tfull + 16u;
    volatile uint32_t* tmem_ptr_gen =
        reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_ptr_addr - smem_u32(smem_raw)));

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);  // provably warp-uniform: role branches use the uniform datapath
    const int lane = threadIdx.x & 31;
    const int total_units = p.out_tiles * p.splits;
    // A operand (M = 128): stacked -> source boxes, normal -> dz boxes
    const int cwA = STACKED ? p.cwV : p.cwS;
    const int cwB = STACKED ? p.cwS : p.cwV;
    // bytes of one box = (pixels per stage) x (channel chunk) x (element size): 64 x cw x 2 (bf16) = 32 x cw x 4 (fp32)
    const uint32_t esize = p.in_fp32 ? 4u : 2u;
    const uint32_t boxA_bytes = 128u * cwA;
    const uint32_t boxB_bytes = 128u * cwB;
    const uint32_t boxS_bytes = STACKED ? boxB_bytes : boxA_bytes;
    const uint32_t boxV_bytes = STACKED ? boxA_bytes : boxB_bytes;
    const int cwS = p.cwS, cwV = p.cwV;
    int tmem_cols = 32;
    while (tmem_cols < p.GU * BLOCK_N) tmem_cols <<= 1;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tm_dz);
        prefetch_tmap(&tm_src);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < SV; ++s) {
            mbar_init(vfull(s), 1);
            mbar_init(vempty(s), 1);
        }
        for (int s = 0; s < SS; ++s) {
            mbar_init(sfull(s), 1);
            mbar_init(sempty(s), 1);
        }
        mbar_init(tfull, 1);
        mbar_init(tempty, 4);
        fence_mbar_init();
    }
    if (warp == 2) {
        tmem_alloc(tmem_ptr_addr, tmem_cols);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_gen;

    if (warp == 0 || warp == 2 || warp == 3 || warp >= 8) {
        // =================================== TMA producers ==================================
        // The warp runs converged and ONE elected lane (elect.sync) issues every copy of a stage in one
        // straight-line block of UTMALDGs; under a divergent per-lane guard ptxas wraps each copy in an
        // ELECT/branch loop.  All coordinates are warp-uniform: the first tap of every group is
        // decoded once per unit (registers, the group loop is unrolled), the pixel-block coordinates
        // are carried by nested counters (no divisions in the loop).
        //
        // FIVE producer warps share the issue work (profiles/r01_ncu_wgrad_producer_bound.txt: with one
        // producer the 11 copies per 64-pixel block of the 64-channel layers cost ~2500 cycles of issue
        // against ~1000 cycles of MMA): the tap groups of a block are dealt round-robin, producer 0 also
        // loads the dz boxes.  Every producer walks the same stage sequence (sv, pv), waits for every
        // stage to be free and fills the stages of its own groups.
        constexpr int NPROD = 5;
        const int pid = warp == 0 ? 0 : (warp < 8 ? warp - 1 : warp - 5);  // warps 0,2,3,8,9 -> 0..4
        constexpr int MAX_GU = Cfg::MAX_GU;
        int turn = 0;  // producer that fills the next ring position
        // at most SV warps take turns (the parity argument at the vempty wait needs SV >= the number of warps dealt to);
        // with a shorter ring the remaining producer warps own nothing and never touch a barrier
        constexpr int NTURN = SV < NPROD ? SV : NPROD;
        int sv = 0, ss = 0;
        uint32_t pv = 0, ps = 0;
        for (int unit = blockIdx.x; unit < total_units; unit += gridDim.x) {
            const WgUnit u = wg_decode<BLOCK_N, STACKED>(p, unit);
            const int boxesS = (u.scols + cwS - 1) / cwS;
            const int boxesV = STACKED ? p.G : (u.vcols + cwV - 1) / cwV;
            const int rb_begin = u.split * p.rb_per_split;
            const int rb_end = min(rb_begin + p.rb_per_split, p.num_rblocks);
            // first tap (kx, ky) of every group of this unit
            int gkx[MAX_GU], gky[MAX_GU];
#pragma unroll
            for (int g = 0; g < MAX_GU; ++g) {
                const int tp = (u.gset * p.GU + g) * p.G;
                gky[g] = tp / p.ksize;
                gkx[g] = tp - gky[g] * p.ksize;
            }
            const uint32_t s_tx = boxesS * boxS_bytes, v_tx = boxesV * boxV_bytes;
            // pixel-block counters
            int m = rb_begin;
            int wt = m % p.tiles_w;
            m /= p.tiles_w;
            int ht = m % p.tiles_h;
            m /= p.tiles_h;
            int bt = m % p.tiles_b;
            int t = m / p.tiles_b;
            for (int rb = rb_begin; rb < rb_end; ++rb) {
                const int w0 = wt * p.Wt, h0 = ht * p.Ht, b0 = bt * p.Bt;
                // shared operand: the dz box(es) of this pixel block
                if (pid == 0) {
                    mbar_wait(sempty(ss), ps ^ 1u, p.err_flag, 4000 + 500 + ss);
                    if (elect_one()) {
                        mbar_arrive_expect_tx(sfull(ss), s_tx);
                        uint32_t dst = s_base + ss * Cfg::S_BYTES;
                        int sc = u.s0;
                        for (int i = 0; i < boxesS; ++i, dst += boxS_bytes, sc += cwS)
                            tma_load_5d(dst, &tm_dz, sfull(ss), sc, w0, h0, b0, t);
                    }
                    __syncwarp();
                    if (++ss == SS) {
                        ss = 0;
                        ps ^= 1u;
                    }
                }
                // varying operand: one stage per tap group
#pragma unroll
                for (int g = 0; g < MAX_GU; ++g) {
                    if (g < u.ngr) {
                        // The stages of the ring are dealt to NTURN producer warps ROUND-ROBIN OVER THE RING POSITION (`turn`),
                        // not over the group index g as in round 1, and a producer waits only for the stages it fills.
                        // A parity wait on vempty(sv) is unambiguous iff the waiter is neither a lap behind nor a lap
                        // ahead of the barrier.  The owner of position q (lap L) cannot be behind: completion L + 1 of
                        // that stage needs ITS fill.  It cannot be ahead: it filled position q - NTURN after the MMA
                        // warp consumed q - NTURN - SV >= q - 2 SV (NTURN <= SV), i.e. at least L - 1 completions.
                        // Round 1 dealt by g and made every producer wait on every stage: in units with fewer groups
                        // than producers a warp owned nothing, nothing held it, it fell a lap behind, its parity
                        // aliased and the kernel hung (watchdog 4523 / 4800, profiles/r02_fault_root_cause.md).
                        if (turn == pid) {
                        mbar_wait(vempty(sv), pv ^ 1u, p.err_flag, 4000 + 520 + sv);
                        if (elect_one()) {
                            const uint32_t fb = vfull(sv);
                            mbar_arrive_expect_tx(fb, v_tx);
                            uint32_t dst = v_base + sv * Cfg::V_BYTES;
                            if (STACKED) {
                                // G consecutive taps; taps beyond the filter repeat the last one (their
                                // rows are never stored)
                                int kx = gkx[g], ky = gky[g];
                                for (int i = 0; i < boxesV; ++i, dst += boxV_bytes) {
                                    tma_load_5d(dst, &tm_src, fb, 0, w0 + kx - p.pad, h0 + ky - p.pad, b0, t);
                                    if (ky * p.ksize + kx + 1 < p.taps) {
                                        if (++kx == p.ksize) {
                                            kx = 0;
                                            ++ky;
                                        }
                                    }
                                }
                            } else {
                                const int cw = w0 + gkx[g] - p.pad, chh = h0 + gky[g] - p.pad;
                                int c = u.v0;
                                for (int i = 0; i < boxesV; ++i, dst += boxV_bytes, c += cwV)
                                    tma_load_5d(dst, &tm_src, fb, c, cw, chh, b0, t);
                            }
                        }
                        __syncwarp();
                        }
                        if (++turn == NTURN) turn = 0;
                        if (++sv == SV) {
                            sv = 0;
                            pv ^= 1u;
                        }
                    }
                }
                if (++wt == p.tiles_w) {
                    wt = 0;
                    if (++ht == p.tiles_h) {
                        ht = 0;
                        if (++bt == p.tiles_b) {
                            bt = 0;
                            ++t;
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // =================================== MMA issuer =====================================
        // converged warp, one elected lane issues (see the producer): back-to-back UTCHMMA
        // swizzle span = bytes of one pixel row of a box (cw channels): 128 / 64 / 32
        const uint32_t rowA = cwA * esize, rowB = cwB * esize;
        const uint32_t ltA = (rowA == 128) ? 2u : (rowA == 64 ? 4u : 6u);
        const uint32_t ltB = (rowB == 128) ? 2u : (rowB == 64 ? 4u : 6u);
        // descriptor = constant high part | (smem address >> 4); one MMA K step = 32 bytes of pixels per channel row
        // = 16 bf16 pixels (two 8-row atoms) or 8 fp32 pixels (one atom) further down the box: 32 * cw bytes either way
        // tf32: MN-major operands of 32-bit elements use the 128-byte swizzle on 32-byte atoms (UMMA layout type 1,
        // SWIZZLE_128B_BASE32B; TMA CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B): 128-byte pixel rows (32 channels), swizzle
        // period and stride-byte-offset = 4 pixel rows
        const bool tf32 = p.in_fp32 != 0;
        const uint64_t hiA = tf32 ? make_smem_desc(0, boxA_bytes, 4u * rowA, 1u) : make_smem_desc(0, boxA_bytes, 8u * rowA, ltA);
        const uint64_t hiB = tf32 ? make_smem_desc(0, boxB_bytes, 4u * rowB, 1u) : make_smem_desc(0, boxB_bytes, 8u * rowB, ltB);
        const uint32_t stepA = (32u * cwA) >> 4, stepB = (32u * cwB) >> 4;
        const uint32_t v_lo0 = (v_base & 0x3FFFFu) >> 4, s_lo0 = (s_base & 0x3FFFFu) >> 4;
        int sv = 0, ss = 0;
        uint32_t pv = 0, ps = 0, pt = 0;
        for (int unit = blockIdx.x; unit < total_units; unit += gridDim.x) {
            const WgUnit u = wg_decode<BLOCK_N, STACKED>(p, unit);
            const int ncols = STACKED ? u.scols : u.vcols;
            const int nmma = ((ncols + cwB - 1) / cwB) * cwB;  // whole loaded boxes
            const uint32_t idesc = tf32 ? make_idesc_tf32(WG_BLOCK_M, nmma, 1, 1) : make_idesc_bf16(WG_BLOCK_M, nmma, 1, 1);
            const int rb_begin = u.split * p.rb_per_split;
            const int rb_end = min(rb_begin + p.rb_per_split, p.num_rblocks);
            mbar_wait(tempty, pt ^ 1u, p.err_flag, 4000 + 700);
            tc_fence_after();
            uint32_t accum = 0;
            for (int rb = rb_begin; rb < rb_end; ++rb) {
                mbar_wait(sfull(ss), ps, p.err_flag, 4000 + 600 + ss);
                const uint32_t s_lo = s_lo0 + ss * (Cfg::S_BYTES >> 4);
                uint32_t d_tmem = tmem_base;
                for (int g = 0; g < u.ngr; ++g, d_tmem += BLOCK_N) {
                    mbar_wait(vfull(sv), pv, p.err_flag, 4000 + 620 + sv);
                    tc_fence_after();
                    if (elect_one()) {
                        const uint32_t v_lo = v_lo0 + sv * (Cfg::V_BYTES >> 4);
                        const uint64_t adesc = hiA | (STACKED ? v_lo : s_lo);
                        const uint64_t bdesc = hiB | (STACKED ? s_lo : v_lo);
                        if (tf32) {
                            umma_tf32(d_tmem, adesc, bdesc, idesc, accum);
                            umma_tf32(d_tmem, adesc + stepA, bdesc + stepB, idesc, 1u);
                            umma_tf32(d_tmem, adesc + 2 * stepA, bdesc + 2 * stepB, idesc, 1u);
                            umma_tf32(d_tmem, adesc + 3 * stepA, bdesc + 3 * stepB, idesc, 1u);
                        } else {
                            umma_bf16(d_tmem, adesc, bdesc, idesc, accum);
                            umma_bf16(d_tmem, adesc + stepA, bdesc + stepB, idesc, 1u);
                            umma_bf16(d_tmem, adesc + 2 * stepA, bdesc + 2 * stepB, idesc, 1u);
                            umma_bf16(d_tmem, adesc + 3 * stepA, bdesc + 3 * stepB, idesc, 1u);
                        }
                        umma_commit(vempty(sv));
                    }
                    __syncwarp();
                    if (++sv == SV) {
                        sv = 0;
                        pv ^= 1u;
                    }
                }
                accum = 1u;
                if (elect_one()) umma_commit(sempty(ss));  // after the MMAs of every group that read this dz box
                __syncwarp();
                if (++ss == SS) {
                    ss = 0;
                    ps ^= 1u;
                }
            }
            if (elect_one()) umma_commit(tfull);
            __syncwarp();
            pt ^= 1u;
        }
    } else if (warp >= 4 && warp < 8) {
        // =================================== epilogue =======================================
        const int q = warp - 4;
        const int r = q * 32 + lane;
        uint32_t pt = 0;
        for (int unit = blockIdx.x; unit < total_units; unit += gridDim.x) {
            const WgUnit u = wg_decode<BLOCK_N, STACKED>(p, unit);
            const int ncols = STACKED ? u.scols : u.vcols;
            mbar_wait(tfull, pt, p.err_flag, 4000 + 800);
            pt ^= 1u;
            tc_fence_after();
            for (int g = 0; g < u.ngr; ++g) {
                const int grp = u.gset * p.GU + g;
                bool valid;
                float* row;
                if (STACKED) {
                    // row r = (tap within the group, source channel); column = dz channel
                    const int gi = r / p.Csrc, c = r - gi * p.Csrc;
                    const int tp = grp * p.G + gi;
                    valid = tp < p.taps;
                    row = p.dw + u.split * p.split_stride + (static_cast<long long>(tp) * p.Nz + u.s0) * p.ldk + p.koff + c;
                } else {
                    const int n = u.s0 + r;
                    valid = n < p.Nz;
                    row = p.dw + u.split * p.split_stride + (static_cast<long long>(grp) * p.Nz + n) * p.ldk + p.koff + u.v0;
                }
                const uint32_t t_row = tmem_base + g * BLOCK_N + (uint32_t(q * 32) << 16);
#pragma unroll 1
                for (int c16 = 0; c16 * 16 < ncols; ++c16) {
                    uint32_t v[16];
                    tmem_ld16(t_row + c16 * 16, v);
                    tmem_ld_wait();
                    if (!valid) continue;
                    if (STACKED) {
                        // transposed store: consecutive lanes hold consecutive source channels
                        float* o = row + static_cast<long long>(c16) * 16 * p.ldk;
#pragma unroll
                        for (int j = 0; j < 16; ++j) o[j * p.ldk] = __uint_as_float(v[j]);
                    } else {
                        float* o = row + c16 * 16;
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            reinterpret_cast<float4*>(o)[j] =
                                make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                            __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
                    }
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
        tmem_dealloc(tmem_base, tmem_cols);
    }
}

template <int BLOCK_N, bool STACKED>
static int launch_wgrad_impl(const CUtensorMap& tz, const CUtensorMap& ts, const WgradParams& p,
                             cudaStream_t stream) {
    using Cfg = WgCfg<BLOCK_N, STACKED>;
    auto kern = wgrad_tc_kernel<BLOCK_N, STACKED>;
    static PerDeviceOnce attr_once;  // kernel attributes are per device
    if (attr_once.first()) {
        B200_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             Cfg::SMEM_BYTES));
        // the whole unified L1/shared array as shared memory: the kernel itself only needs its ring, but the
        // remainder lets HBM-bound blocks of another stream (BatchNorm sums: 9 KB static) share the SM when the
        // weight gradient runs on the background stream (with the default carve-out the next step is 196 KB)
        B200_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout,
                                             cudaSharedmemCarveoutMaxShared));
    }
    int total = p.out_tiles * p.splits;
    int grid = total < num_sms() ? total : num_sms();
    kern<<<grid, WG_THREADS, Cfg::SMEM_BYTES, stream>>>(tz, ts, p);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// widest channel chunk whose pixel row is 128 / 64 / 32 bytes
static int chunk_width(int C, int esize) {
    for (int bytes = 128; bytes >= 32; bytes >>= 1)
        if (C % (bytes / esize) == 0) return bytes / esize;
    return 0;
}

// Tiling and reduction split of a launch: every field of p except the pointers and the output layout.
static int plan_wgrad_tc(int Nz, int Csrc, int T, int B, int H, int W, int ksize, int in_fp32, WgradParams* pp,
                         MTile* pmt, bool* pstacked, int* pblock_n) {
    const int esize = in_fp32 ? 4 : 2;
    const int rb_pixels = 128 / esize;   // pixels per pipeline stage: 64 (bf16) or 32 (fp32)
    WgradParams& p = *pp;
    MTile& mt = *pmt;
    p = {};
    p.in_fp32 = in_fp32;
    p.T = T; p.B = B; p.H = H; p.W = W;
    p.Nz = Nz; p.Csrc = Csrc; p.ksize = ksize; p.pad = ksize / 2; p.taps = ksize * ksize;
    p.cwS = chunk_width(Nz, esize);
    p.cwV = chunk_width(Csrc, esize);
    if (in_fp32 && (p.cwS != 32 || p.cwV != 32)) p.cwS = p.cwV = 0;   // tf32: 128-byte pixel rows only (32 channels)
    if (p.cwS == 0 || p.cwV == 0) {
        set_last_error("wgrad_tc: channels Nz=%d Csrc=%d not multiples of %d", Nz, Csrc, 32 / esize);
        return B200_ERR_SHAPE;
    }
    if (!plan_mtile(B, H, W, rb_pixels, &mt)) {
        set_last_error("wgrad_tc: spatial shape B=%d H=%d W=%d cannot be tiled", B, H, W);
        return B200_ERR_SHAPE;
    }
    p.Wt = mt.Wt; p.Ht = mt.Ht; p.Bt = mt.Bt;
    p.tiles_w = mt.tiles_w; p.tiles_h = mt.tiles_h; p.tiles_b = mt.tiles_b;
    p.num_rblocks = T * mt.tiles_w * mt.tiles_h * mt.tiles_b;
    // few source channels: stack G taps of the source along M, dz becomes the N operand
    // (the stacked source box is ONE channel chunk: its pixel row must fit the 128-byte swizzle span)
    const bool stacked = (Csrc * esize == 32 || Csrc * esize == 64 || Csrc * esize == 128) && p.taps > 1;
    int& block_n = *pblock_n;
    *pstacked = stacked;
    if (stacked) {
        p.G = WG_BLOCK_M / Csrc;
        p.cwV = Csrc;
        block_n = Nz > 128 ? 256 : (Nz > 64 ? 128 : 64);
        p.s_tiles = (Nz + block_n - 1) / block_n;
        p.v_tiles = 1;
    } else {
        p.G = 1;
        block_n = Csrc > 128 ? 256 : (Csrc > 64 ? 128 : 64);
        p.s_tiles = (Nz + WG_BLOCK_M - 1) / WG_BLOCK_M;
        p.v_tiles = (Csrc + block_n - 1) / block_n;
    }
    p.ngroups = (p.taps + p.G - 1) / p.G;
    p.GU = 512 / block_n;
    if (p.GU > p.ngroups) p.GU = p.ngroups;
    // balance the group sets (e.g. 9 taps, at most 4 accumulators -> 3+3+3 rather than 4+4+1)
    p.ngsets = (p.ngroups + p.GU - 1) / p.GU;
    p.GU = (p.ngroups + p.ngsets - 1) / p.ngsets;
    p.out_tiles = p.ngsets * p.s_tiles * p.v_tiles;
    // reduction split: the split count that minimises (waves of CTAs) / split, smallest such count;
    // at least 8 reduction blocks per unit
    const int nsm = num_sms();
    int max_splits = (p.num_rblocks + 7) / 8;
    if (max_splits > 4 * nsm) max_splits = 4 * nsm;
    if (max_splits < 1) max_splits = 1;
    int best = 1;
    double best_cost = 1e30;
    for (int s = 1; s <= max_splits; ++s) {
        const long long units = static_cast<long long>(p.out_tiles) * s;
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

int wgrad_tc_splits(int Nz, int Csrc, int T, int B, int H, int W, int ksize, int in_fp32) {
    WgradParams p;
    MTile mt;
    bool stacked;
    int block_n;
    const int rc = plan_wgrad_tc(Nz, Csrc, T, B, H, W, ksize, in_fp32, &p, &mt, &stacked, &block_n);
    return rc == B200_OK ? p.splits : rc;
}

// dw += the weight gradient, at any split count: every split stores its partial sums to its own workspace slice and
// splitk_reduce adds the slices to dw.  in_fp32: dz / src are fp32 tensors and the products are TF32 (see
// WgradParams::in_fp32).
int launch_wgrad_tc(const void* dz, int Nz, const void* src, int Csrc, int T, int B, int H, int W,
                    int ksize, float* dw, long long ldk, int koff, cudaStream_t stream, int in_fp32) {
    const int esize = in_fp32 ? 4 : 2;
    if ((ldk % 4) != 0 || (koff % 4) != 0) {
        set_last_error("wgrad_tc: ldk/koff must be multiples of 4");
        return B200_ERR_ALIGN;
    }
    WgradParams p;
    MTile mt;
    bool stacked;
    int block_n;
    int rc = plan_wgrad_tc(Nz, Csrc, T, B, H, W, ksize, in_fp32, &p, &mt, &stacked, &block_n);
    if (rc != B200_OK) return rc;
    p.split_stride = static_cast<long long>(p.taps) * Nz * Csrc;
    p.dw = splitk_workspace(stream, static_cast<size_t>(p.splits) * p.split_stride);
    if (!p.dw) {
        set_last_error("%s: no split-K workspace (cudaMalloc failed, or growth during graph capture)", __func__);
        return B200_ERR_CUDA;
    }
    p.ldk = Csrc;
    p.koff = 0;
    p.err_flag = device_error_flag();

    CUtensorMap tz, ts;
    rc = make_act_tmap(&tz, dz, Nz, W, H, B, T, p.cwS, mt.Wt, mt.Ht, mt.Bt, esize, in_fp32);
    if (rc != B200_OK) return rc;
    rc = make_act_tmap(&ts, src, Csrc, W, H, B, T, p.cwV, mt.Wt, mt.Ht, mt.Bt, esize, in_fp32);
    if (rc != B200_OK) return rc;
    if (stacked) {
        switch (block_n) {
            case 256: rc = launch_wgrad_impl<256, true>(tz, ts, p, stream); break;
            case 128: rc = launch_wgrad_impl<128, true>(tz, ts, p, stream); break;
            default: rc = launch_wgrad_impl<64, true>(tz, ts, p, stream); break;
        }
    } else {
        switch (block_n) {
            case 256: rc = launch_wgrad_impl<256, false>(tz, ts, p, stream); break;
            case 128: rc = launch_wgrad_impl<128, false>(tz, ts, p, stream); break;
            default: rc = launch_wgrad_impl<64, false>(tz, ts, p, stream); break;
        }
    }
    if (rc != B200_OK) return rc;
    return splitk_reduce(p.dw, p.splits, static_cast<long long>(p.taps) * Nz, Csrc, dw, ldk, koff, stream);
}

}  // namespace b200
