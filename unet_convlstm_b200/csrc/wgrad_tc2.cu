// Weight-gradient GEMM on a CTA PAIR (tcgen05 cta_group::2): the 2-SM variants of wgrad_tc.cu.
//
// NORMAL mode (wide sources): A = dz, the pair covers 256 dz channels (CTA r its own 128), B = source channels,
// each CTA loads HALF of the source tile of every tap -- the varying operand, nine tap-shifted copies of it per
// pixel block, is what the 1-CTA kernel spends its L2 -> SM bandwidth on.
//
// STACKED mode (source with 16 / 32 / 64 channels):
//
//   dW[tap][n][koff + c] (+)= sum_{t, pixel p} dz[t, p, n] * src[t, p + tap, c]
//
// wgrad_tc.cu stacks G = 128 / Csrc tap-shifted source boxes along M (rows = (tap, source channel)) and uses
// the dz channels as N; at N = 64 that MMA is bound by the shared-memory read of its A operand, and the nine
// taps of a 64-channel layer need five of them per 16 pixels.  Here the pair stacks 2G taps along M = 256 --
// CTA r holds the boxes of taps (2*group + r)*G .. +G-1 -- and each CTA loads only HALF of the dz tile
// (BLOCK_N / 2 channels), so a 64-channel layer needs three M = 256 MMAs per 16 pixels instead of five
// M = 128 ones, each dz byte crosses L2 -> SM once per pair, and the per-SM shared-memory read per MMA drops
// from A + B to A + B/2.
//
// Pipeline (barriers at the same shared-memory offset in both CTAs): sfull / vfull live in the leader (two
// arrive.expect_tx, both CTAs' cta_group::2 TMA copies complete on them); sempty / vempty / tfull are signalled in
// both CTAs by the leader's multicast tcgen05.commit; tempty collects the epilogue warps of the pair.  Work units,
// reduction splits (with their workspace slices), the five producer warps and the transposed fp32 store epilogue are
// those of wgrad_tc.cu.
#include "common.cuh"
#include <stdlib.h>

#include "ptx.cuh"

namespace b200 {

static constexpr int W2_BLOCK_M = 128;  // rows per CTA
static constexpr int W2_RB = 128;       // pixels per pipeline stage (8 MMA K steps): halves the barrier round trips
                                        // and TMA issues per pixel -- the 1-CTA kernel's bottleneck on these layers
static constexpr int W2_THREADS = 320;  // warps 0,2,3,8,9 producers, 1 MMA issuer (leader), 4-7 epilogue

struct Wgrad2Params {
    int T, B, H, W;
    int Nz, Csrc;
    int ksize, pad, taps;
    int cwS;                    // channel width of one dz box
    int cwV;                    // channel width of one source box
    int Wt, Ht, Bt, tiles_w, tiles_h, tiles_b;
    int num_rblocks, rb_per_split, splits;
    int G;                      // taps per CTA and group (128 / Csrc); a pair group has 2G taps
    int ngroups, GU, ngsets;
    int gset_inner;             // unit order: tap sets fastest (1) or slowest (0)
    int s_tiles, v_tiles, out_tiles;
    float* dw;                  // the split-K workspace, split s at dw + s * split_stride
    long long ldk;
    int koff;
    long long split_stride;
    int* err_flag;
};

template <int BLOCK_N, bool STACKED>
struct Wg2Cfg {
    static constexpr int A_BYTES = W2_BLOCK_M * W2_RB * 2;     // this CTA's 128 M rows: 32 KB
    static constexpr int B_BYTES = (BLOCK_N / 2) * W2_RB * 2;  // this CTA's half of the N operand
    static constexpr int V_BYTES = STACKED ? A_BYTES : B_BYTES;  // varying (source) operand
    static constexpr int S_BYTES = STACKED ? B_BYTES : A_BYTES;  // shared (dz) operand
    static constexpr int SV = STACKED ? ((BLOCK_N == 256) ? 4 : 5) : ((BLOCK_N == 256) ? 4 : (BLOCK_N == 128 ? 6 : 8));
    static constexpr int SS = STACKED ? ((BLOCK_N == 256) ? 2 : 3) : ((BLOCK_N == 256) ? 2 : 3);
    static constexpr int MAX_GU = 512 / BLOCK_N;
    static constexpr int SMEM_BYTES = SV * V_BYTES + SS * S_BYTES + 1024 + 512;
};

struct Wg2Unit {
    int split, gset, s0, v0, ngr;
};

template <int BLOCK_N, bool STACKED>
__device__ __forceinline__ Wg2Unit wg2_decode(const Wgrad2Params& p, int unit) {
    Wg2Unit u;
    u.split = unit / p.out_tiles;
    int ot = unit - u.split * p.out_tiles;
    int vt, st;
    if (p.gset_inner) {
        // tap sets fastest: the pairs resident at the same time then cover ALL taps of a few (dz tile, source tile)
        // pairs -- the taps read the same source bytes (shifted windows) and the same dz tile -- instead of one tap
        // set of every tile, which re-reads the whole dz range once per tap set (5 x at the temporal cell's shape)
        u.gset = ot % p.ngsets;
        ot /= p.ngsets;
        vt = ot % p.v_tiles;
        st = ot / p.v_tiles;
    } else {
        vt = ot % p.v_tiles;
        ot /= p.v_tiles;
        st = ot % p.s_tiles;
        u.gset = ot / p.s_tiles;
    }
    u.s0 = st * (STACKED ? BLOCK_N : 2 * W2_BLOCK_M);  // stacked: dz channels are N; normal: 256 dz rows per pair
    u.v0 = vt * BLOCK_N;
    u.ngr = min(p.GU, p.ngroups - u.gset * p.GU);
    return u;
}

template <int BLOCK_N, bool STACKED>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(W2_THREADS, 1)
wgrad_tc2_kernel(const __grid_constant__ CUtensorMap tm_dz, const __grid_constant__ CUtensorMap tm_src,
                 const Wgrad2Params p) {
    using Cfg = Wg2Cfg<BLOCK_N, STACKED>;
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

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int num_clusters = gridDim.x >> 1;
    const int cluster_id = blockIdx.x >> 1;
    const int total_units = p.out_tiles * p.splits;
    // A operand (this CTA's 128 M rows): stacked -> G source boxes (one per tap), normal -> dz boxes
    const int cwA = STACKED ? p.cwV : p.cwS;
    const int cwB = STACKED ? p.cwS : p.cwV;
    const uint32_t boxA_bytes = W2_RB * cwA * 2;
    const uint32_t boxB_bytes = W2_RB * cwB * 2;
    const uint32_t boxS_bytes = STACKED ? boxB_bytes : boxA_bytes;
    const uint32_t boxV_bytes = STACKED ? boxA_bytes : boxB_bytes;
    const int boxesS = (STACKED ? BLOCK_N / 2 : W2_BLOCK_M) / p.cwS;  // dz boxes per CTA and pixel block
    const int boxesV = STACKED ? p.G : (BLOCK_N / 2) / p.cwV;         // source boxes per CTA and group
    int tmem_cols = 32;
    while (tmem_cols < p.GU * BLOCK_N) tmem_cols <<= 1;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tm_dz);
        prefetch_tmap(&tm_src);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < SV; ++s) {
            mbar_init(vfull(s), 2);   // one arrive.expect_tx per CTA (leader's copy is the one used)
            mbar_init(vempty(s), 1);  // multicast commit
        }
        for (int s = 0; s < SS; ++s) {
            mbar_init(sfull(s), 2);
            mbar_init(sempty(s), 1);
        }
        mbar_init(tfull, 1);
        mbar_init(tempty, 8);  // 4 epilogue warps of each CTA (leader's copy is the one used)
        fence_mbar_init();
    }
    if (warp == 2) {
        tmem_alloc2(tmem_ptr_addr, tmem_cols);
        tmem_relinquish2();
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_gen;

    if (warp == 0 || warp == 2 || warp == 3 || warp >= 8) {
        // =================================== TMA producers (both CTAs) ==================================
        constexpr int NPROD = 5;
        const int pid = warp == 0 ? 0 : (warp < 8 ? warp - 1 : warp - 5);
        constexpr int MAX_GU = Cfg::MAX_GU;
        const uint32_t vfull0_l = map_to_cta(vfull(0), 0), sfull0_l = map_to_cta(sfull(0), 0);
        int turn = 0;  // producer that fills the next ring position
        // at most SV warps take turns (the parity argument at the vempty wait needs SV >= the number of warps dealt to);
        // with a shorter ring the remaining producer warps own nothing and never touch a barrier
        constexpr int NTURN = SV < NPROD ? SV : NPROD;
        int sv = 0, ss = 0;
        uint32_t pv = 0, ps = 0;
        for (int unit = cluster_id; unit < total_units; unit += num_clusters) {
            const Wg2Unit u = wg2_decode<BLOCK_N, STACKED>(p, unit);
            const int rb_begin = u.split * p.rb_per_split;
            const int rb_end = min(rb_begin + p.rb_per_split, p.num_rblocks);
            // first tap (kx, ky) of this CTA's part of every group of this unit
            int gkx[MAX_GU], gky[MAX_GU];
#pragma unroll
            for (int g = 0; g < MAX_GU; ++g) {
                const int tp = STACKED ? min(((u.gset * p.GU + g) * 2 + static_cast<int>(rank)) * p.G, p.taps - 1)
                                       : min(u.gset * p.GU + g, p.taps - 1);
                gky[g] = tp / p.ksize;
                gkx[g] = tp - gky[g] * p.ksize;
            }
            const uint32_t s_tx = boxesS * boxS_bytes, v_tx = boxesV * boxV_bytes;
            // this CTA's dz channels: stacked -> its half of the N tile, normal -> its 128 of the pair's 256 M rows
            const int sc0 = u.s0 + static_cast<int>(rank) * (STACKED ? BLOCK_N / 2 : W2_BLOCK_M);
            const int vc0 = u.v0 + static_cast<int>(rank) * (BLOCK_N / 2);  // normal: its half of the source tile
            int m = rb_begin;
            int wt = m % p.tiles_w;
            m /= p.tiles_w;
            int ht = m % p.tiles_h;
            m /= p.tiles_h;
            int bt = m % p.tiles_b;
            int t = m / p.tiles_b;
            for (int rb = rb_begin; rb < rb_end; ++rb) {
                const int w0 = wt * p.Wt, h0 = ht * p.Ht, b0 = bt * p.Bt;
                if (pid == 0) {
                    mbar_wait(sempty(ss), ps ^ 1u, p.err_flag, 5000 + 500 + ss);
                    if (elect_one()) {
                        const uint32_t fb = sfull0_l + 8u * ss;
                        mbar_arrive_expect_tx_cluster(fb, s_tx);
                        uint32_t dst = s_base + ss * Cfg::S_BYTES;
                        int sc = sc0;
                        for (int i = 0; i < boxesS; ++i, dst += boxS_bytes, sc += p.cwS)
                            tma2_load_5d(dst, &tm_dz, fb, sc, w0, h0, b0, t);
                    }
                    __syncwarp();
                    if (++ss == SS) {
                        ss = 0;
                        ps ^= 1u;
                    }
                }
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
                            mbar_wait(vempty(sv), pv ^ 1u, p.err_flag, 5000 + 520 + sv);
                            if (elect_one()) {
                                const uint32_t fb = vfull0_l + 8u * sv;
                                mbar_arrive_expect_tx_cluster(fb, v_tx);
                                uint32_t dst = v_base + sv * Cfg::V_BYTES;
                                if (STACKED) {
                                    // G consecutive taps; taps beyond the filter repeat the last one (never stored)
                                    int kx = gkx[g], ky = gky[g];
                                    for (int i = 0; i < boxesV; ++i, dst += boxV_bytes) {
                                        tma2_load_5d(dst, &tm_src, fb, 0, w0 + kx - p.pad, h0 + ky - p.pad, b0, t);
                                        if (ky * p.ksize + kx + 1 < p.taps) {
                                            if (++kx == p.ksize) {
                                                kx = 0;
                                                ++ky;
                                            }
                                        }
                                    }
                                } else {
                                    const int cw = w0 + gkx[g] - p.pad, chh = h0 + gky[g] - p.pad;
                                    int c = vc0;
                                    for (int i = 0; i < boxesV; ++i, dst += boxV_bytes, c += p.cwV)
                                        tma2_load_5d(dst, &tm_src, fb, c, cw, chh, b0, t);
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
        // =================================== MMA issuer (leader CTA only) ===============================
        if (leader) {
            const uint32_t ltA = (cwA == 64) ? 2u : (cwA == 32 ? 4u : 6u);
            const uint32_t ltB = (cwB == 64) ? 2u : (cwB == 32 ? 4u : 6u);
            const uint64_t hiA = make_smem_desc(0, boxA_bytes, 8u * cwA * 2, ltA);
            const uint64_t hiB = make_smem_desc(0, boxB_bytes, 8u * cwB * 2, ltB);
            const uint32_t stepA = (16u * cwA * 2) >> 4, stepB = (16u * cwB * 2) >> 4;
            const uint32_t v_lo0 = (v_base & 0x3FFFFu) >> 4, s_lo0 = (s_base & 0x3FFFFu) >> 4;
            const uint32_t idesc = make_idesc_bf16(2 * W2_BLOCK_M, BLOCK_N, 1, 1);
            int sv = 0, ss = 0;
            uint32_t pv = 0, ps = 0, pt = 0;
            for (int unit = cluster_id; unit < total_units; unit += num_clusters) {
                const Wg2Unit u = wg2_decode<BLOCK_N, STACKED>(p, unit);
                const int rb_begin = u.split * p.rb_per_split;
                const int rb_end = min(rb_begin + p.rb_per_split, p.num_rblocks);
                mbar_wait(tempty, pt ^ 1u, p.err_flag, 5000 + 700);
                tc_fence_after();
                uint32_t accum = 0;
                for (int rb = rb_begin; rb < rb_end; ++rb) {
                    mbar_wait(sfull(ss), ps, p.err_flag, 5000 + 600 + ss);
                    const uint32_t s_lo = s_lo0 + ss * (Cfg::S_BYTES >> 4);
                    uint32_t d_tmem = tmem_base;
                    for (int g = 0; g < u.ngr; ++g, d_tmem += BLOCK_N) {
                        mbar_wait(vfull(sv), pv, p.err_flag, 5000 + 620 + sv);
                        tc_fence_after();
                        if (elect_one()) {
                            const uint32_t v_lo = v_lo0 + sv * (Cfg::V_BYTES >> 4);
                            const uint64_t adesc = hiA | (STACKED ? v_lo : s_lo);
                            const uint64_t bdesc = hiB | (STACKED ? s_lo : v_lo);
                            umma2_bf16(d_tmem, adesc, bdesc, idesc, accum);
#pragma unroll
                            for (int k = 1; k < W2_RB / 16; ++k)
                                umma2_bf16(d_tmem, adesc + k * stepA, bdesc + k * stepB, idesc, 1u);
                            umma2_commit_both(vempty(sv));
                        }
                        __syncwarp();
                        if (++sv == SV) {
                            sv = 0;
                            pv ^= 1u;
                        }
                    }
                    accum = 1u;
                    if (elect_one()) umma2_commit_both(sempty(ss));
                    __syncwarp();
                    if (++ss == SS) {
                        ss = 0;
                        ps ^= 1u;
                    }
                }
                if (elect_one()) umma2_commit_both(tfull);
                __syncwarp();
                pt ^= 1u;
            }
        }
    } else if (warp >= 4 && warp < 8) {
        // =================================== epilogue (both CTAs, own TMEM lanes) =======================
        const int q = warp - 4;
        const int r = q * 32 + lane;
        const uint32_t tempty_l = map_to_cta(tempty, 0);
        uint32_t pt = 0;
        for (int unit = cluster_id; unit < total_units; unit += num_clusters) {
            const Wg2Unit u = wg2_decode<BLOCK_N, STACKED>(p, unit);
            const int ncols = STACKED ? min(BLOCK_N, p.Nz - u.s0) : min(BLOCK_N, p.Csrc - u.v0);
            mbar_wait(tfull, pt, p.err_flag, 5000 + 800);
            pt ^= 1u;
            tc_fence_after();
            for (int g = 0; g < u.ngr; ++g) {
                const int grp = u.gset * p.GU + g;
                bool valid;
                float* row;
                if (STACKED) {
                    // row r of this CTA = (tap within its G taps, source channel); column = dz channel
                    const int gi = r / p.Csrc, c = r - gi * p.Csrc;
                    const int tp = (grp * 2 + static_cast<int>(rank)) * p.G + gi;
                    valid = tp < p.taps;
                    row = p.dw + u.split * p.split_stride + (static_cast<long long>(valid ? tp : 0) * p.Nz + u.s0) * p.ldk + p.koff + c;
                } else {
                    // row r of this CTA = dz channel; column = source channel
                    const int n = u.s0 + static_cast<int>(rank) * W2_BLOCK_M + r;
                    valid = n < p.Nz;
                    row = p.dw + u.split * p.split_stride + (static_cast<long long>(grp) * p.Nz + (valid ? n : 0)) * p.ldk + p.koff + u.v0;
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
            if (lane == 0) mbar_arrive_cluster(tempty_l);
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc2(tmem_base, tmem_cols);
    }
}

template <int BLOCK_N, bool STACKED>
static int launch_wgrad2_impl(const CUtensorMap& tz, const CUtensorMap& ts, const Wgrad2Params& p, cudaStream_t stream) {
    using Cfg = Wg2Cfg<BLOCK_N, STACKED>;
    auto kern = wgrad_tc2_kernel<BLOCK_N, STACKED>;
    static PerDeviceOnce attr_once;  // kernel attributes are per device
    if (attr_once.first()) {
        B200_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        // the whole unified L1/shared array as shared memory: the kernel itself only needs its ring, but the
        // remainder lets HBM-bound blocks of another stream (BatchNorm sums: 9 KB static) share the SM when the
        // weight gradient runs on the background stream (with the default carve-out the next step is 196 KB)
        B200_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout,
                                             cudaSharedmemCarveoutMaxShared));
    }
    const int total = p.out_tiles * p.splits;
    const int max_clusters = num_sms() / 2;
    const int clusters = total < max_clusters ? total : max_clusters;
    kern<<<2 * clusters, W2_THREADS, Cfg::SMEM_BYTES, stream>>>(tz, ts, p);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

static bool w2_stacked(int Csrc, int ksize) { return (Csrc == 16 || Csrc == 32 || Csrc == 64) && ksize * ksize > 1; }

// Stacked mode: narrow sources, dz width a multiple of its N tile.  Normal mode: dz channels in pairs of 128 and a
// source width that is a multiple of its N tile (the ConvLSTM weight gradients and the deep UNet layers).
bool wgrad_tc2_supported(int Nz, int Csrc, int ksize) {
    if (w2_stacked(Csrc, ksize)) {
        const int block_n = Nz > 128 ? 256 : (Nz > 64 ? 128 : 64);
        return Nz % block_n == 0;
    }
    if (Csrc < 64 || Nz % (2 * W2_BLOCK_M) != 0) return false;
    const int block_n = Csrc > 128 ? 256 : (Csrc > 64 ? 128 : 64);
    return Csrc % block_n == 0;
}

// Tiling and reduction split of a launch: every field of p except the pointers and the output layout.
static int plan_wgrad_tc2(int Nz, int Csrc, int T, int B, int H, int W, int ksize, Wgrad2Params* pp, MTile* pmt,
                          int* pblock_n) {
    Wgrad2Params& p = *pp;
    MTile& mt = *pmt;
    int& block_n = *pblock_n;
    p = {};
    p.T = T; p.B = B; p.H = H; p.W = W;
    p.Nz = Nz; p.Csrc = Csrc; p.ksize = ksize; p.pad = ksize / 2; p.taps = ksize * ksize;
    const bool stacked = w2_stacked(Csrc, ksize);
    if (!plan_mtile(B, H, W, W2_RB, &mt)) {
        set_last_error("wgrad_tc2: spatial shape B=%d H=%d W=%d cannot be tiled", B, H, W);
        return B200_ERR_SHAPE;
    }
    if (stacked) {
        block_n = Nz > 128 ? 256 : (Nz > 64 ? 128 : 64);
        p.cwS = (block_n / 2) < 64 ? (block_n / 2) : 64;
        p.cwV = Csrc;
        p.G = W2_BLOCK_M / Csrc;
        p.s_tiles = Nz / block_n;
        p.v_tiles = 1;
        p.ngroups = (p.taps + 2 * p.G - 1) / (2 * p.G);
    } else {
        block_n = Csrc > 128 ? 256 : (Csrc > 64 ? 128 : 64);
        p.cwS = 64;
        p.cwV = (block_n / 2) < 64 ? (block_n / 2) : 64;
        p.G = 1;
        p.s_tiles = Nz / (2 * W2_BLOCK_M);
        p.v_tiles = Csrc / block_n;
        p.ngroups = p.taps;
    }
    p.Wt = mt.Wt; p.Ht = mt.Ht; p.Bt = mt.Bt;
    p.tiles_w = mt.tiles_w; p.tiles_h = mt.tiles_h; p.tiles_b = mt.tiles_b;
    p.num_rblocks = T * mt.tiles_w * mt.tiles_h * mt.tiles_b;
    p.GU = 512 / block_n;
    if (p.GU > p.ngroups) p.GU = p.ngroups;
    p.ngsets = (p.ngroups + p.GU - 1) / p.GU;
    p.GU = (p.ngroups + p.ngsets - 1) / p.ngsets;
    p.out_tiles = p.ngsets * p.s_tiles * p.v_tiles;
    {
        static const int order = [] { const char* e = getenv("B200_WGRAD_TAPS_INNER"); return e ? atoi(e) : 1; }();
        p.gset_inner = order;
    }
    // reduction split over the clusters (see wgrad_tc.cu): fewest waves per split, at least 4 blocks per unit
    const int ncl = num_sms() / 2;
    int max_splits = (p.num_rblocks + 3) / 4;
    if (max_splits > 4 * ncl) max_splits = 4 * ncl;
    if (max_splits < 1) max_splits = 1;
    int best = 1;
    double best_cost = 1e30;
    for (int s = 1; s <= max_splits; ++s) {
        const long long units = static_cast<long long>(p.out_tiles) * s;
        const double cost = static_cast<double>((units + ncl - 1) / ncl) / s;
        if (cost < best_cost * 0.97) {
            best_cost = cost;
            best = s;
        }
    }
    p.rb_per_split = (p.num_rblocks + best - 1) / best;
    p.splits = (p.num_rblocks + p.rb_per_split - 1) / p.rb_per_split;
    return B200_OK;
}

int wgrad_tc2_splits(int Nz, int Csrc, int T, int B, int H, int W, int ksize) {
    Wgrad2Params p;
    MTile mt;
    int block_n;
    const int rc = plan_wgrad_tc2(Nz, Csrc, T, B, H, W, ksize, &p, &mt, &block_n);
    return rc == B200_OK ? p.splits : rc;
}

// dw += the weight gradient, at any split count (see launch_wgrad_tc)
int launch_wgrad_tc2(const void* dz, int Nz, const void* src, int Csrc, int T, int B, int H, int W, int ksize, float* dw,
                     long long ldk, int koff, cudaStream_t stream) {
    Wgrad2Params p;
    MTile mt;
    int block_n;
    int rc = plan_wgrad_tc2(Nz, Csrc, T, B, H, W, ksize, &p, &mt, &block_n);
    if (rc != B200_OK) return rc;
    const bool stacked = w2_stacked(Csrc, ksize);
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
    rc = make_act_tmap(&tz, dz, Nz, W, H, B, T, p.cwS, mt.Wt, mt.Ht, mt.Bt);
    if (rc != B200_OK) return rc;
    rc = make_act_tmap(&ts, src, Csrc, W, H, B, T, p.cwV, mt.Wt, mt.Ht, mt.Bt);
    if (rc != B200_OK) return rc;
    if (stacked) {
        switch (block_n) {
            case 256: rc = launch_wgrad2_impl<256, true>(tz, ts, p, stream); break;
            case 128: rc = launch_wgrad2_impl<128, true>(tz, ts, p, stream); break;
            default: rc = launch_wgrad2_impl<64, true>(tz, ts, p, stream); break;
        }
    } else {
        switch (block_n) {
            case 256: rc = launch_wgrad2_impl<256, false>(tz, ts, p, stream); break;
            case 128: rc = launch_wgrad2_impl<128, false>(tz, ts, p, stream); break;
            default: rc = launch_wgrad2_impl<64, false>(tz, ts, p, stream); break;
        }
    }
    if (rc != B200_OK) return rc;
    return splitk_reduce(p.dw, p.splits, static_cast<long long>(p.taps) * Nz, Csrc, dw, ldk, koff, stream);
}

}  // namespace b200
