// Implicit-GEMM convolution on the sm_100a tensor cores.
//
//   out[p, n] = sum_{tap, k} in[p + tap, k] * Wp[tap][n][k]          (zero padding)
//
// GEMM view: M = 128 output pixels per tile (a Wt x Ht x Bt box of the NHWC tensor), N = BLOCK_N
// output channels, K = taps x (C0 + C1) input channels.  The input is the *virtual* concatenation of
// two NHWC tensors (x_t and h_{t-1} of the ConvLSTM cell, reference train/unet.py:28; the skip and
// the up-sampled tensor of an Up block, unet.py:98): each K block comes from one TMA box of one of
// the two tensors, so no concatenated copy ever exists.  Zero padding is the TMA out-of-bounds
// fill: the box of tap (ky,kx) starts at (w0+kx-pad, h0+ky-pad), possibly negative.
//
// Warp roles (256 threads, one CTA per SM, persistent over tiles):
//   warp 0   TMA producer           : A box + B box per K block into a STAGES-deep smem ring
//   warp 1   MMA issuer (1 thread)  : tcgen05.mma kind::f16, fp32 accumulators in TMEM (2 stages)
//   warp 2   TMEM allocator
//   warps 4-7 epilogue              : tcgen05.ld -> bias / gate math -> global stores
//
// Epilogues:
//   EPI_STORE  bias, optional ReLU, bf16 or fp32 output, optionally split over two destination
//              tensors (dgrad of the virtual concat: [dx ; dh]).
//   EPI_LSTM   the N tile holds the four gates of CHT hidden channels (weights are packed
//              gate-interleaved), so i,f,g,o of a (pixel, channel) sit in one thread's TMEM lane:
//              sigma,sigma,tanh,sigma, c' = f*c + i*g, h' = o*tanh(c')  (unet.py:29-35) are applied
//              in registers and only h' (bf16), c' (fp32) and the activated gates (bf16, for BPTT)
//              are written; the 4*Ch pre-activations never reach HBM.
#include "conv_tc.cuh"
#include "ptx.cuh"

#include <stdlib.h>

namespace b200 {

static constexpr int BLOCK_M = 128;
static constexpr int EPI_WARP0 = 4;
// Epilogue warps: 4 (one per TMEM lane quarter) for the plain store and the forward cell update; 8 for the
// BPTT epilogue, whose per-element operand loads (gates, c, dc, dh: ~34 bytes) are latency bound -- two
// warps share a lane quarter and split the columns of the tile.
template <int EPI>
struct EpiCfg {
    static constexpr int WARPS = (EPI == EPI_LSTM_BWD) ? 8 : 4;
    static constexpr int THREADS = (EPI_WARP0 + WARPS) * 32;
};

template <int BLOCK_N>
struct TcCfg {
    static constexpr int A_BYTES = BLOCK_M * 128;  // at kc = 64 (bf16)
    static constexpr int B_BYTES = BLOCK_N * 128;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int STAGES = (BLOCK_N == 256) ? 4 : (BLOCK_N == 128 ? 6 : 8);
    static constexpr int TMEM_COLS = 2 * BLOCK_N;  // double-buffered accumulator
    static constexpr int STAT_BYTES = 4 * 2 * BLOCK_N * 4;  // BatchNorm partial sums, one row per epilogue warp
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/ + STAT_BYTES;
};

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}

// Spin (bounded) until the grid-wide step counter reaches `target`.  Safe only under a cooperative
// launch, where every CTA of the grid is resident.
__device__ __forceinline__ void grid_wait(const unsigned* ctr, unsigned target, int* err_flag) {
    const long long t0 = clock64();
    unsigned v;
    do {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory");
        if (v >= target) break;
        if (clock64() - t0 > 8000000000LL) {
            if (err_flag) *reinterpret_cast<volatile int*>(err_flag) = 1900;
            __threadfence_system();
            asm volatile("trap;");
        }
    } while (true);
}

struct TileCoord {
    int n0, t, b0, h0, w0;
};

__device__ __forceinline__ TileCoord decode_tile(const ConvTcParams& p, int tile, int block_n) {
    TileCoord tc;
    int nt = tile / p.num_m_tiles;
    int m = tile - nt * p.num_m_tiles;
    tc.n0 = nt * block_n;
    int wt = m % p.tiles_w;
    m /= p.tiles_w;
    int ht = m % p.tiles_h;
    m /= p.tiles_h;
    int bt = m % p.tiles_b;
    tc.t = m / p.tiles_b;
    tc.w0 = wt * p.Wt;
    tc.h0 = ht * p.Ht;
    tc.b0 = bt * p.Bt;
    return tc;
}

template <int BLOCK_N, int EPI>
__global__ void __launch_bounds__(EpiCfg<EPI>::THREADS, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tm_a0, const __grid_constant__ CUtensorMap tm_a1,
               const __grid_constant__ CUtensorMap tm_b, const ConvTcParams p) {
    using Cfg = TcCfg<BLOCK_N>;
    constexpr int STAGES = Cfg::STAGES;

    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_base = smem_base + STAGES * Cfg::STAGE_BYTES;
    // barrier layout (8 B each): full[STAGES], empty[STAGES], tfull[2], tempty[2], then tmem ptr
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
    auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + s); };
    auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + 2 + s); };
    const uint32_t tmem_ptr_addr = bar_base + 8u * (2 * STAGES + 4);
    volatile uint32_t* tmem_ptr_gen =
        reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_ptr_addr - smem_u32(smem_raw)));
    // [4 epilogue warps][2][BLOCK_N] floats after the 256-byte barrier area
    float* stat_smem = reinterpret_cast<float*>(smem_raw + (bar_base + 256u - smem_u32(smem_raw)));

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);  // provably warp-uniform: role branches use the uniform datapath
    const int lane = threadIdx.x & 31;

    const int taps = p.ksize * p.ksize;
    const int chunks0 = p.C0 / p.kc;
    const int chunks1 = p.C1 / p.kc;
    const int chunks = chunks0 + chunks1;
    const int num_kb = taps * chunks;
    // K range of this CTA (split K, see ConvTcParams::kb_split): k-blocks [kb_lo, kb_hi) of the (tap, chunk) loop
    const int kb_lo = p.kb_split > 0 ? static_cast<int>(blockIdx.z) * p.kb_split : 0;
    const int kb_hi = p.kb_split > 0 ? min(kb_lo + p.kb_split, num_kb) : num_kb;
    const int total_tiles = p.num_m_tiles * p.num_n_tiles;
    // timestep-persistent mode (EPI_LSTM only): the kernel iterates over the whole sequence, h_t and
    // c_t stay in the L2-resident state buffers and a grid-wide counter separates the steps
    const bool seq = p.seq_T > 0;
    const int nsteps = seq ? p.seq_T : 1;
    // BPTT runs the sequence backwards; a tile whose columns nobody needs is skipped by all three roles
    // (dx columns without a dx_seq buffer; dh columns at t = 0 without a dh0 buffer)
    auto step_t = [&](int step) { return (EPI == EPI_LSTM_BWD) ? p.seq_T - 1 - step : step; };
    // i-th tile of this CTA: -2 = no more tiles, -1 = nothing in this slot.  Default: blockIdx.x + i * grid.
    // BPTT (p.bwd_alternate): the N tiles split into a dh half (heavy gate-gradient epilogue) and a dx half
    // (plain store); a CTA alternates between them, heavy first, so that a heavy epilogue always overlaps
    // the main loop of a light tile and the last tile of a step is a light one.
    const int half_tiles = (p.num_n_tiles >> 1) * p.num_m_tiles;
    const int alt_iters = 2 * ((half_tiles + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x));
    auto tile_at = [&](int i) {
        if (EPI == EPI_LSTM_BWD && p.bwd_alternate) {
            if (i >= alt_iters) return -2;
            const int u = (i >> 1) * static_cast<int>(gridDim.x) + static_cast<int>(blockIdx.x);
            if (u >= half_tiles) return -1;
            return ((i & 1) ? 0 : half_tiles) + u;
        }
        const int t = static_cast<int>(blockIdx.x) + i * static_cast<int>(gridDim.x);
        return t < total_tiles ? t : -2;
    };
    auto tile_active = [&](int t, int n0) {
        if constexpr (EPI != EPI_LSTM_BWD) return true;
        if (n0 + BLOCK_N <= p.bwd_Cin) return p.bwd_dx_seq != nullptr;
        if (n0 >= p.bwd_Cin) return t > 0 || p.bwd_dh0 != nullptr;
        return true;
    };
    const uint32_t esize = p.in_fp32 ? 4u : 2u;  // operand element size: bf16 (kind::f16) or fp32 read as TF32 (kind::tf32)
    const uint32_t a_bytes = BLOCK_M * p.kc * esize;
    const uint32_t b_bytes = BLOCK_N * p.kc * esize;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tm_a0);
        if (p.C1 > 0) prefetch_tmap(&tm_a1);
        prefetch_tmap(&tm_b);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full_bar(s), 1);
            mbar_init(empty_bar(s), 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(tfull_bar(s), 1);
            mbar_init(tempty_bar(s), EpiCfg<EPI>::WARPS);  // one arrive per epilogue warp
        }
        fence_mbar_init();
    }
    if (warp == 2) {
        tmem_alloc(tmem_ptr_addr, Cfg::TMEM_COLS);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_gen;

    if (warp == 0) {
        // =================================== TMA producer ===================================
        // The whole warp runs the loop converged and ONE elected lane (elect.sync) issues the copies:
        // ptxas then emits straight-line UTMALDG code; under a divergent `lane == 0` guard it wraps
        // every copy in an ELECT / branch loop, which made the N = 64 tiles (a K block is only 128
        // tensor-pipe cycles) issue-bound (profiles/r01_ncu_conv_halo_issue_loop.txt).  The (tap,
        // channel-chunk) index is carried by nested counters, never derived by division.
        int stage = 0;
        uint32_t phase = 0;
        uint32_t a_dst = smem_base;
        const uint32_t tx_bytes = a_bytes + b_bytes;
        for (int step = 0; step < nsteps; ++step) {
            const int chunks_t = (seq && step == 0 && !p.seq_have_h0) ? chunks0 : chunks;
            if (seq && step > 0) {
                // h_{t-1} was written by the epilogue warps of every CTA in the previous step
                if (lane == 0) grid_wait(p.sync_ctr, gridDim.x * step, p.err_flag);
                __syncwarp();
                fence_proxy_async_all();  // every lane: whichever one is elected issues the TMA reads
            }
            for (int ti = 0;; ++ti) {
                const int tile = tile_at(ti);
                if (tile == -2) break;
                if (tile < 0) continue;
                TileCoord tc = decode_tile(p, tile, BLOCK_N);
                if (seq) tc.t = step_t(step);
                if (!tile_active(tc.t, tc.n0)) continue;
                int ky = 0, kx = 0, kbi = 0;
                for (int tap = 0; tap < taps; ++tap) {
                    const int cw = tc.w0 + kx - p.pad, chh = tc.h0 + ky - p.pad;
                    int kofs = 0;
                    for (int c = 0; c < chunks_t; ++c, kofs += p.kc, ++kbi) {
                        if (kbi < kb_lo || kbi >= kb_hi) continue;  // outside this split's K range (warp-uniform)
                        mbar_wait(empty_bar(stage), phase ^ 1u, p.err_flag, 1000 + 100 + stage);
                        if (elect_one()) {
                            const uint32_t fb = full_bar(stage);
                            mbar_arrive_expect_tx(fb, tx_bytes);
                            if (c < chunks0)
                                tma_load_5d(a_dst, &tm_a0, fb, kofs, cw, chh, tc.b0, tc.t);
                            else
                                tma_load_5d(a_dst, &tm_a1, fb, kofs - p.C0, cw, chh, tc.b0, tc.t);
                            tma_load_3d(a_dst + Cfg::A_BYTES, &tm_b, fb, kofs, tc.n0, tap);
                        }
                        __syncwarp();
                        a_dst += Cfg::STAGE_BYTES;
                        if (++stage == STAGES) {
                            stage = 0;
                            phase ^= 1u;
                            a_dst = smem_base;
                        }
                    }
                    if (++kx == p.ksize) {
                        kx = 0;
                        ++ky;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // =================================== MMA issuer =====================================
        // converged warp, one elected lane issues (see the producer): back-to-back UTCHMMA
        const bool tf32 = p.in_fp32 != 0;
        const uint32_t idesc = tf32 ? make_idesc_tf32(BLOCK_M, BLOCK_N, 0, 0) : make_idesc_bf16(BLOCK_M, BLOCK_N, 0, 0);
        // K-major swizzled operand tiles: rows of kc*esize bytes (128 / 64 / 32), 8-row atoms => SBO = 8 * row bytes
        const uint32_t row_bytes = p.kc * esize;
        const uint32_t layout_type = (row_bytes == 128) ? 2u : (row_bytes == 64 ? 4u : 6u);
        const uint32_t sbo = 8u * row_bytes;
        const int mma_per_kb = row_bytes / 32;  // one MMA = 32 bytes of K: 16 bf16 or 8 tf32
        // descriptor = constant high part | (smem address >> 4); only the address changes per stage
        const uint64_t desc_hi = make_smem_desc(0, 16, sbo, layout_type);
        int stage = 0;
        uint32_t phase = 0;
        int acc = 0;
        uint32_t acc_phase = 0;
        uint32_t a_lo = (smem_base & 0x3FFFFu) >> 4;
        const uint32_t a_lo0 = a_lo;
        constexpr uint32_t STAGE_LO = Cfg::STAGE_BYTES >> 4, B_LO = Cfg::A_BYTES >> 4;
        for (int step = 0; step < nsteps; ++step) {
            const int num_kb_t = min(kb_hi, (seq && step == 0 && !p.seq_have_h0) ? taps * chunks0 : num_kb);
            for (int ti = 0;; ++ti) {
                const int tile = tile_at(ti);
                if (tile == -2) break;
                if (tile < 0) continue;
                if constexpr (EPI == EPI_LSTM_BWD) {
                    if (!tile_active(step_t(step), (tile / p.num_m_tiles) * BLOCK_N)) continue;
                }
                mbar_wait(tempty_bar(acc), acc_phase ^ 1u, p.err_flag, 1000 + 300 + acc);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
                uint32_t accum = 0;
                for (int kb = kb_lo; kb < num_kb_t; ++kb) {
                    mbar_wait(full_bar(stage), phase, p.err_flag, 1000 + 200 + stage);
                    tc_fence_after();
                    if (elect_one()) {
                        const uint64_t adesc = desc_hi | a_lo;
                        const uint64_t bdesc = desc_hi | (a_lo + B_LO);
                        if (tf32) {
                            for (int k = 0; k < mma_per_kb; ++k)
                                umma_tf32(d_tmem, adesc + uint64_t(2 * k), bdesc + uint64_t(2 * k), idesc,
                                          k == 0 ? accum : 1u);
                        } else if (mma_per_kb == 4) {
                            // advance 16 bf16 = 32 B along K inside the swizzled row: +2 in >>4 units
                            umma_bf16(d_tmem, adesc, bdesc, idesc, accum);
                            umma_bf16(d_tmem, adesc + 2, bdesc + 2, idesc, 1u);
                            umma_bf16(d_tmem, adesc + 4, bdesc + 4, idesc, 1u);
                            umma_bf16(d_tmem, adesc + 6, bdesc + 6, idesc, 1u);
                        } else {
                            for (int k = 0; k < mma_per_kb; ++k)
                                umma_bf16(d_tmem, adesc + uint64_t(2 * k), bdesc + uint64_t(2 * k), idesc,
                                          k == 0 ? accum : 1u);
                        }
                        umma_commit(empty_bar(stage));  // frees the smem slot when the MMAs retire
                    }
                    __syncwarp();
                    accum = 1u;
                    a_lo += STAGE_LO;
                    if (++stage == STAGES) {
                        stage = 0;
                        phase ^= 1u;
                        a_lo = a_lo0;
                    }
                }
                if (elect_one()) umma_commit(tfull_bar(acc));  // accumulator complete -> epilogue
                __syncwarp();
                if (++acc == 2) {
                    acc = 0;
                    acc_phase ^= 1u;
                }
            }
        }
    } else if (warp >= EPI_WARP0) {
        // =================================== epilogue =======================================
        const int ew = static_cast<int>(threadIdx.x >> 5) - EPI_WARP0;  // epilogue warp (vector-register copy)
        const int q = ew & 3;             // TMEM lane quarter == warp % 4
        const int chalf = ew >> 2;        // column half of the tile (always 0 with 4 epilogue warps)
        constexpr int C16_PER_WARP = BLOCK_N / 16 / (EpiCfg<EPI>::WARPS / 4);
        const int r = q * 32 + lane;     // row of the M tile
        const int wi = r % p.Wt;
        const int hi = (r / p.Wt) % p.Ht;
        const int bi = r / (p.Wt * p.Ht);
        int acc = 0;
        uint32_t acc_phase = 0;
        // fused BatchNorm statistics: every epilogue warp keeps the partial sums of its 32 rows in its
        // own shared-memory row (plain read-modify-write by the owning lane: no atomics, no barriers) and
        // flushes them (fp64 atomics) whenever the (t, N tile) key changes -- tiles are ordered N tile,
        // t, image, row, so a warp flushes ~T times per N tile
        const bool do_stats = (EPI == EPI_STORE) && p.stat_sum != nullptr;
        float* stat_row = stat_smem + q * (2 * BLOCK_N);
        int stat_t = -1, stat_n0 = 0;
        auto stat_flush = [&]() {
            __syncwarp();
            for (int i = lane; i < 2 * BLOCK_N; i += 32) {
                const float v = stat_row[i];
                stat_row[i] = 0.f;
                const int col = stat_n0 + (i % BLOCK_N);
                if (col < p.N && stat_t >= 0)
                    atomicAdd((i < BLOCK_N ? p.stat_sum : p.stat_sumsq) + static_cast<long long>(stat_t) * p.N + col,
                              static_cast<double>(v));
            }
            __syncwarp();
        };
        if (do_stats) stat_flush();  // zeroes the buffer (stat_t < 0: nothing is added)
        for (int step = 0; step < nsteps; ++step) {
        const bool zero_state = seq && step == 0 && !p.seq_have_h0;
        for (int ti = 0;; ++ti) {
                const int tile = tile_at(ti);
                if (tile == -2) break;
                if (tile < 0) continue;
            TileCoord tc = decode_tile(p, tile, BLOCK_N);
            if (seq) tc.t = step_t(step);
            if (!tile_active(tc.t, tc.n0)) continue;
            if (do_stats && (tc.t != stat_t || tc.n0 != stat_n0)) {
                if (stat_t >= 0) stat_flush();
                stat_t = tc.t;
                stat_n0 = tc.n0;
            }
            const bool valid = (tc.h0 + hi < p.H) && (tc.b0 + bi < p.B);
            const long long pix =
                ((static_cast<long long>(tc.t) * p.B + tc.b0 + bi) * p.H + tc.h0 + hi) * p.W + tc.w0 + wi;
            if constexpr (EPI == EPI_LSTM_BWD) {
                // The gate-gradient operands of this tile (gates, c, dc, upstream dh: ~34 bytes per element,
                // cold in HBM) are known before the accumulator is: pull them into L2 while the main loop of
                // the tile is still running, so the epilogue's dependent loads are L2 hits.
                const int cb = max(tc.n0, p.bwd_Cin) - p.bwd_Cin;
                const int ce = min(tc.n0 + BLOCK_N, p.N) - p.bwd_Cin;
                if (valid && ce > cb && tc.t > 0) {
                    const int Ch = p.bwd_Ch;
                    const long long pin = pix - static_cast<long long>(tc.t) * p.bwd_P;
                    const long long sp = static_cast<long long>(tc.t - 1) * p.bwd_P + pin;
                    const char* gr = reinterpret_cast<const char*>(p.bwd_gates + sp * (4LL * Ch) + cb);
                    const char* c0 = reinterpret_cast<const char*>(p.bwd_c_all + sp * Ch + cb);
                    const char* c1 = reinterpret_cast<const char*>(p.bwd_c_all + (sp + p.bwd_P) * Ch + cb);
                    const char* dcp = reinterpret_cast<const char*>(
                        p.bwd_dc + (static_cast<long long>(tc.t & 1) * p.bwd_P + pin) * Ch + cb);
                    const int nb2 = (ce - cb) * 2, nb4 = (ce - cb) * 4;
                    for (int o = 0; o < nb2; o += 128) {
#pragma unroll
                        for (int gq = 0; gq < 4; ++gq) prefetch_l2(gr + gq * Ch * 2 + o);
                        if (p.bwd_dh_seq) prefetch_l2(reinterpret_cast<const char*>(p.bwd_dh_seq + sp * Ch + cb) + o);
                    }
                    for (int o = 0; o < nb4; o += 128) {
                        if (tc.t > 1 || p.seq_have_h0) prefetch_l2(c0 + o);
                        prefetch_l2(c1 + o);
                        prefetch_l2(dcp + o);
                    }
                }
            }
            mbar_wait(tfull_bar(acc), acc_phase, p.err_flag, 1000 + 400 + acc);
            tc_fence_after();
            const uint32_t t_row = tmem_base + acc * BLOCK_N + (uint32_t(q * 32) << 16);

            if constexpr (EPI == EPI_STORE) {
#pragma unroll 1
                for (int c16 = 0; c16 < BLOCK_N / 16; ++c16) {
                    const int ncol = tc.n0 + c16 * 16;
                    if (ncol >= p.N) break;  // warp-uniform
                    uint32_t v[16];
                    tmem_ld16(t_row + c16 * 16, v);
                    tmem_ld_wait();
                    if (do_stats) {
                        // statistics of the values as stored (bias added, rounded to bf16); rows outside
                        // the tensor contribute nothing
                        float s1[16], s2[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            float x = __uint_as_float(v[j]);
                            if (p.bias) x += __ldg(p.bias + ncol + j);
                            x = valid ? __bfloat162float(__float2bfloat16_rn(x)) : 0.f;
                            s1[j] = x;
                            s2[j] = x * x;
                        }
                        warp_colsum16(s1, lane);
                        warp_colsum16(s2, lane);
                        if ((lane & 1) == 0) {
                            const int col = c16 * 16 + stat_col(lane);
                            stat_row[col] += s1[0];
                            stat_row[BLOCK_N + col] += s2[0];
                        }
                    }
                    if (valid) {
                        float f[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(v[j]);
                        if (p.scale) {
#pragma unroll
                            for (int j = 0; j < 16; ++j) f[j] *= __ldg(p.scale + ncol + j);
                        }
                        if (p.bias) {
                            const float* bp = p.bias + (p.shuf_C > 0 ? ncol % p.shuf_C : ncol);
#pragma unroll
                            for (int j = 0; j < 16; ++j) f[j] += __ldg(bp + j);
                        }
                        if (p.relu) {
#pragma unroll
                            for (int j = 0; j < 16; ++j) f[j] = fmaxf(f[j], 0.f);
                        }
                        if (p.shuf_C > 0) {
                            // ConvTranspose 2x2 stride 2: the tap block of this column chunk selects the output
                            // pixel of the 2x2 patch (no separate pixel-shuffle pass)
                            const int tap = ncol / p.shuf_C, co = ncol - tap * p.shuf_C;
                            const long long img = static_cast<long long>(tc.t) * p.B + tc.b0 + bi;
                            const long long orow = (img * p.shuf_Hd + 2 * (tc.h0 + hi) + (tap >> 1) + p.shuf_oy) * p.shuf_Wd +
                                                   2 * (tc.w0 + wi) + (tap & 1) + p.shuf_ox;
                            // shuf_C is a multiple of 16: every piece is 32-byte aligned
                            st_bf16x16(static_cast<__nv_bfloat16*>(p.dst0) + orow * p.shuf_C + co, f);
                            continue;
                        }
                        const bool second = ncol >= p.split;
                        const long long off = second ? pix * p.ld1 + (ncol - p.split)
                                                     : pix * p.ld0 + ncol + blockIdx.z * p.split_stride;
                        void* base = second ? p.dst1 : p.dst0;
                        if (p.out_fp32) {
                            float4* o = reinterpret_cast<float4*>(static_cast<float*>(base) + off);
                            if (p.accumulate) {
#pragma unroll
                                for (int j = 0; j < 4; ++j) {
                                    float4 old = o[j];
                                    o[j] = make_float4(old.x + f[4 * j], old.y + f[4 * j + 1],
                                                       old.z + f[4 * j + 2], old.w + f[4 * j + 3]);
                                }
                            } else {
#pragma unroll
                                for (int j = 0; j < 4; ++j)
                                    o[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
                            }
                        } else {
                            uint4* o = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(base) + off);
                            o[0] = make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]),
                                              pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
                            o[1] = make_uint4(pack_bf16x2(f[8], f[9]), pack_bf16x2(f[10], f[11]),
                                              pack_bf16x2(f[12], f[13]), pack_bf16x2(f[14], f[15]));
                        }
                    }
                }
            } else if constexpr (EPI == EPI_LSTM_BWD) {
                // ---- BPTT step: [dx_t ; dh_{t-1}] columns; the dh columns feed the gate gradients of
                //      step t-1 (autograd of reference train/unet.py:30-35) without leaving the registers ----
                const int Cin = p.bwd_Cin, Ch = p.bwd_Ch;
                const long long pin = pix - static_cast<long long>(tc.t) * p.bwd_P;  // pixel within the step
                const int tp = tc.t - 1;                                              // gate-gradient step
#pragma unroll 1
                for (int c16 = chalf * C16_PER_WARP; c16 < (chalf + 1) * C16_PER_WARP; ++c16) {
                    const int ncol = tc.n0 + c16 * 16;
                    if (ncol >= p.N) break;  // warp-uniform
                    if (ncol < Cin ? p.bwd_dx_seq == nullptr : (tp < 0 && p.bwd_dh0 == nullptr)) continue;
                    uint32_t v[16];
                    tmem_ld16(t_row + c16 * 16, v);
                    tmem_ld_wait();
                    if (!valid) continue;
                    auto st16 = [](__nv_bfloat16* dst, const float* s) {
                        uint4* o = reinterpret_cast<uint4*>(dst);
                        o[0] = make_uint4(pack_bf16x2(s[0], s[1]), pack_bf16x2(s[2], s[3]),
                                          pack_bf16x2(s[4], s[5]), pack_bf16x2(s[6], s[7]));
                        o[1] = make_uint4(pack_bf16x2(s[8], s[9]), pack_bf16x2(s[10], s[11]),
                                          pack_bf16x2(s[12], s[13]), pack_bf16x2(s[14], s[15]));
                    };
                    auto ld16 = [](const __nv_bfloat16* src, float* d) {
                        const uint4* q4 = reinterpret_cast<const uint4*>(src);
#pragma unroll
                        for (int h2 = 0; h2 < 2; ++h2) {
                            const uint4 u = q4[h2];
                            const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                d[8 * h2 + 2 * j] = __uint_as_float(w[j] << 16);
                                d[8 * h2 + 2 * j + 1] = __uint_as_float(w[j] & 0xffff0000u);
                            }
                        }
                    };
                    auto ld16f = [](const float* src, float* d) {
                        const float4* q4 = reinterpret_cast<const float4*>(src);
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const float4 u = q4[j];
                            d[4 * j] = u.x; d[4 * j + 1] = u.y; d[4 * j + 2] = u.z; d[4 * j + 3] = u.w;
                        }
                    };
                    float dh[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) dh[j] = __uint_as_float(v[j]);
                    if (ncol < Cin) {
                        st16(p.bwd_dx_seq + pix * Cin + ncol, dh);
                        continue;
                    }
                    const int ch = ncol - Cin;
                    if (tp < 0) {
                        st16(p.bwd_dh0 + pin * Ch + ch, dh);  // dL/dh_{-1}: gradient of the initial state
                        continue;
                    }
                    const long long sp = static_cast<long long>(tp) * p.bwd_P + pin;  // (step t-1, pixel)
                    if (p.bwd_dh_seq) {
                        float up[16];
                        ld16(p.bwd_dh_seq + sp * Ch + ch, up);
#pragma unroll
                        for (int j = 0; j < 16; ++j) dh[j] += up[j];
                    }
                    float gi[16], gf[16], gg[16], go[16], cp[16], cn[16], dc[16];
                    const __nv_bfloat16* gr = p.bwd_gates + sp * (4LL * Ch) + ch;
                    ld16(gr, gi);
                    ld16(gr + Ch, gf);
                    ld16(gr + 2 * Ch, gg);
                    ld16(gr + 3 * Ch, go);
                    if (tp > 0 || p.seq_have_h0) {
                        ld16f(p.bwd_c_all + sp * Ch + ch, cp);
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; ++j) cp[j] = 0.f;  // zero initial state (unet.py:23-25)
                    }
                    ld16f(p.bwd_c_all + (sp + p.bwd_P) * Ch + ch, cn);
                    ld16f(p.bwd_dc + (static_cast<long long>(tc.t & 1) * p.bwd_P + pin) * Ch + ch, dc);
                    float zi[16], zf[16], zg[16], zo[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const float tch = fast_tanh(cn[j]);
                        const float d_o = dh[j] * tch;
                        const float d_c = fmaf(dh[j] * go[j], 1.f - tch * tch, dc[j]);
                        zi[j] = d_c * gg[j] * gi[j] * (1.f - gi[j]);
                        zf[j] = d_c * cp[j] * gf[j] * (1.f - gf[j]);
                        zg[j] = d_c * gi[j] * (1.f - gg[j] * gg[j]);
                        zo[j] = d_o * go[j] * (1.f - go[j]);
                        dc[j] = d_c * gf[j];
                    }
                    __nv_bfloat16* zr = p.bwd_dz_all + sp * (4LL * Ch) + ch;
                    st16(zr, zi);
                    st16(zr + Ch, zf);
                    st16(zr + 2 * Ch, zg);
                    st16(zr + 3 * Ch, zo);
                    float4* dco = reinterpret_cast<float4*>(p.bwd_dc + (static_cast<long long>(tp & 1) * p.bwd_P + pin) * Ch + ch);
#pragma unroll
                    for (int j = 0; j < 4; ++j) dco[j] = make_float4(dc[4 * j], dc[4 * j + 1], dc[4 * j + 2], dc[4 * j + 3]);
                }
            } else {
                // ---- fused LSTM cell update (reference train/unet.py:29-35) ----
                constexpr int CHT = BLOCK_N / 4;
                const int Ch = p.N >> 2;
                const int ch0 = (tc.n0 >> 2);  // first hidden channel of this N tile
#pragma unroll 1
                for (int j0 = 0; j0 < CHT; j0 += 16) {
                    uint32_t vi[16], vf[16], vg[16], vo[16];
                    tmem_ld16(t_row + 0 * CHT + j0, vi);
                    tmem_ld16(t_row + 1 * CHT + j0, vf);
                    tmem_ld16(t_row + 2 * CHT + j0, vg);
                    tmem_ld16(t_row + 3 * CHT + j0, vo);
                    tmem_ld_wait();
                    if (valid) {
                        const int ch = ch0 + j0;
                        const long long coff = pix * Ch + ch;
                        float cp[16];
                        if (p.c_prev && !zero_state) {
                            const float4* c4 = reinterpret_cast<const float4*>(p.c_prev + coff);
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                float4 t4 = c4[j];
                                cp[4 * j] = t4.x;
                                cp[4 * j + 1] = t4.y;
                                cp[4 * j + 2] = t4.z;
                                cp[4 * j + 3] = t4.w;
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 16; ++j) cp[j] = 0.f;
                        }
                        float gi[16], gf[16], gg[16], go[16], cn[16], hn[16];
                        const float* bp = p.bias ? p.bias + tc.n0 + j0 : nullptr;
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            float zi = __uint_as_float(vi[j]);
                            float zf = __uint_as_float(vf[j]);
                            float zg = __uint_as_float(vg[j]);
                            float zo = __uint_as_float(vo[j]);
                            if (bp) {
                                zi += __ldg(bp + j);
                                zf += __ldg(bp + CHT + j);
                                zg += __ldg(bp + 2 * CHT + j);
                                zo += __ldg(bp + 3 * CHT + j);
                            }
                            if (p.state_fp32) {
                                // tf32 mode: full-precision gate functions.  The BPTT derivative s(1-s) is formed from
                                // the stored gate, so an absolute error of 2^-12 (tanh.approx) in a saturated gate is a
                                // relative error of percents in its gradient -- fine next to bf16 storage, not here.
                                gi[j] = 1.f / (1.f + expf(-zi));
                                gf[j] = 1.f / (1.f + expf(-zf));
                                gg[j] = tanhf(zg);
                                go[j] = 1.f / (1.f + expf(-zo));
                                cn[j] = fmaf(gf[j], cp[j], gi[j] * gg[j]);
                                hn[j] = go[j] * tanhf(cn[j]);
                            } else {
                                gi[j] = fast_sigmoid(zi);
                                gf[j] = fast_sigmoid(zf);
                                gg[j] = fast_tanh(zg);
                                go[j] = fast_sigmoid(zo);
                                cn[j] = fmaf(gf[j], cp[j], gi[j] * gg[j]);
                                hn[j] = go[j] * fast_tanh(cn[j]);
                            }
                        }
                        if (p.c_next) {
                            float4* co = reinterpret_cast<float4*>(p.c_next + coff);
#pragma unroll
                            for (int j = 0; j < 4; ++j)
                                co[j] = make_float4(cn[4 * j], cn[4 * j + 1], cn[4 * j + 2], cn[4 * j + 3]);
                        }
                        if (p.state_fp32) {
                            // "tf32" precision mode: h and the activated gates are fp32 tensors
                            auto st16f = [](float* dst, const float* sv) {
                                float4* o = reinterpret_cast<float4*>(dst);
#pragma unroll
                                for (int j = 0; j < 4; ++j) o[j] = make_float4(sv[4 * j], sv[4 * j + 1], sv[4 * j + 2], sv[4 * j + 3]);
                            };
                            if (p.h_next) st16f(reinterpret_cast<float*>(p.h_next) + coff, hn);
                            if (p.gates_out) {
                                float* gb = reinterpret_cast<float*>(p.gates_out) + pix * (4LL * Ch) + ch;
                                st16f(gb, gi);
                                st16f(gb + Ch, gf);
                                st16f(gb + 2 * Ch, gg);
                                st16f(gb + 3 * Ch, go);
                            }
                            continue;
                        }
                        if (p.h_next) {
                            uint4* ho = reinterpret_cast<uint4*>(p.h_next + coff);
                            ho[0] = make_uint4(pack_bf16x2(hn[0], hn[1]), pack_bf16x2(hn[2], hn[3]),
                                               pack_bf16x2(hn[4], hn[5]), pack_bf16x2(hn[6], hn[7]));
                            ho[1] = make_uint4(pack_bf16x2(hn[8], hn[9]), pack_bf16x2(hn[10], hn[11]),
                                               pack_bf16x2(hn[12], hn[13]), pack_bf16x2(hn[14], hn[15]));
                        }
                        if (p.gates_out) {
                            __nv_bfloat16* gb = p.gates_out + pix * (4LL * Ch) + ch;
                            auto st16 = [](__nv_bfloat16* dst, const float* s) {
                                uint4* o = reinterpret_cast<uint4*>(dst);
                                o[0] = make_uint4(pack_bf16x2(s[0], s[1]), pack_bf16x2(s[2], s[3]),
                                                  pack_bf16x2(s[4], s[5]), pack_bf16x2(s[6], s[7]));
                                o[1] = make_uint4(pack_bf16x2(s[8], s[9]), pack_bf16x2(s[10], s[11]),
                                                  pack_bf16x2(s[12], s[13]), pack_bf16x2(s[14], s[15]));
                            };
                            st16(gb, gi);
                            st16(gb + Ch, gf);
                            st16(gb + 2 * Ch, gg);
                            st16(gb + 3 * Ch, go);
                        }
                    }
                }
            }
            // release the accumulator stage back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty_bar(acc));
            if (++acc == 2) {
                acc = 0;
                acc_phase ^= 1u;
            }
        }
        if (do_stats && stat_t >= 0) {
            stat_flush();
            stat_t = -1;
        }
        if (seq && step + 1 < nsteps) {
            // publish h_t / c_t of this CTA's tiles, then signal the grid-wide step counter
            asm volatile("bar.sync 1, %0;" ::"n"(EpiCfg<EPI>::WARPS * 32) : "memory");
            if (threadIdx.x == EPI_WARP0 * 32) {
                // A CTA without an active tile in this step has not been held back by its producer: it must
                // not signal step s before every CTA has finished step s-1 (the counter only counts arrivals)
                if (step > 0) grid_wait(p.sync_ctr, gridDim.x * step, p.err_flag);
                __threadfence();
                atomicAdd(p.sync_ctr, 1u);
            }
        }
        }
    }

    // ---- teardown ----
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------------
int pick_block_n(int N, int epi) {
    if (epi == EPI_LSTM) {
        int Ch = N / 4;
        if (Ch % 64 == 0) return 256;
        if (Ch % 32 == 0) return 128;
        if (Ch % 16 == 0) return 64;
        return 0;
    }
    if (N % 16 != 0) return 0;
    if (N >= 256 || N > 128) return 256;
    if (N > 64) return 128;
    return 64;
}

template <int BLOCK_N, int EPI>
static int launch_impl(const CUtensorMap& ta0, const CUtensorMap& ta1, const CUtensorMap& tb,
                       const ConvTcParams& p, cudaStream_t stream, int splits = 1) {
    using Cfg = TcCfg<BLOCK_N>;
    auto kern = conv_tc_kernel<BLOCK_N, EPI>;
    static PerDeviceOnce attr_once;  // kernel attributes are per device
    if (attr_once.first()) {
        B200_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             Cfg::SMEM_BYTES));
    }
    int total = p.num_m_tiles * p.num_n_tiles;
    int grid = total < num_sms() ? total : num_sms();
    if (p.seq_T > 0) {
        // the steps are separated by a grid-wide counter: every CTA must be resident -> cooperative launch
        B200_CUDA_CHECK(cudaMemsetAsync(p.sync_ctr, 0, sizeof(unsigned), stream));
        void* args[] = {const_cast<CUtensorMap*>(&ta0), const_cast<CUtensorMap*>(&ta1),
                        const_cast<CUtensorMap*>(&tb), const_cast<ConvTcParams*>(&p)};
        B200_CUDA_CHECK(cudaLaunchCooperativeKernel(reinterpret_cast<const void*>(kern), dim3(grid),
                                                    dim3(EpiCfg<EPI>::THREADS), args, Cfg::SMEM_BYTES, stream));
        return B200_OK;
    }
    kern<<<dim3(grid, 1, splits), EpiCfg<EPI>::THREADS, Cfg::SMEM_BYTES, stream>>>(ta0, ta1, tb, p);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// K-block width: the widest of 128 / 64 / 32-byte rows that divides both channel counts (0: none does)
static int pick_kc(int C0, int C1, int esize) {
    const int kc_max = 128 / esize, kc_min = 32 / esize;
    int kc = kc_max;
    while (kc >= kc_min && ((C0 % kc) != 0 || (C1 % kc) != 0)) kc >>= 1;
    return (kc < kc_min || C0 <= 0) ? 0 : kc;
}

int conv_tc_num_kb(int C0, int C1, int ksize) {
    const int kc = pick_kc(C0, C1, 2);
    return kc ? ksize * ksize * (C0 / kc + C1 / kc) : 0;
}

int launch_conv_tc_splitk(const void* src0, const void* src1, const void* wpacked, ConvTcParams p, int splits,
                          float* ws, int* splits_out, cudaStream_t stream) {
    const int num_kb = conv_tc_num_kb(p.C0, p.C1, p.ksize);
    if (num_kb == 0 || splits < 1 || p.seq_T > 0 || p.in_fp32) {
        set_last_error("conv_tc_splitk: bf16 single-step problems with channel counts in multiples of 16 only");
        return B200_ERR_SHAPE;
    }
    p.kb_split = (num_kb + splits - 1) / splits;
    *splits_out = (num_kb + p.kb_split - 1) / p.kb_split;  // no empty split
    p.split_stride = static_cast<long long>(p.T) * p.B * p.H * p.W * p.N;
    p.dst0 = ws; p.ld0 = p.N; p.split = p.N; p.dst1 = nullptr; p.ld1 = 0;
    p.out_fp32 = 1; p.relu = 0; p.accumulate = 0;
    p.bias = nullptr; p.scale = nullptr; p.stat_sum = nullptr; p.stat_sumsq = nullptr; p.shuf_C = 0;
    return launch_conv_tc(src0, src1, wpacked, p, EPI_STORE, stream);
}

int launch_convlstm_seq_tc(const void* x_seq, const void* h_all, const void* wpacked, ConvTcParams p,
                           cudaStream_t stream) {
    p.sync_ctr = device_sync_counter(stream);
    if (!p.sync_ctr || p.seq_T <= 0) {
        set_last_error("convlstm_seq_tc: no step counter / bad sequence length");
        return B200_ERR_ARG;
    }
    return launch_conv_tc(x_seq, h_all, wpacked, p, EPI_LSTM, stream);
}

int launch_convlstm_seq_bwd_tc(const void* wd_packed, ConvTcParams p, cudaStream_t stream) {
    p.sync_ctr = device_sync_counter(stream);
    if (!p.sync_ctr || p.seq_T <= 0 || !p.bwd_dz_all || !p.bwd_gates || !p.bwd_c_all || !p.bwd_dc) {
        set_last_error("convlstm_seq_bwd_tc: missing buffers / bad sequence length");
        return B200_ERR_ARG;
    }
    if (p.bwd_Cin % 16 != 0 || p.bwd_Ch % 16 != 0) {
        set_last_error("convlstm_seq_bwd_tc: Cin=%d Ch=%d must be multiples of 16", p.bwd_Cin, p.bwd_Ch);
        return B200_ERR_SHAPE;
    }
    return launch_conv_tc(p.bwd_dz_all, nullptr, wd_packed, p, EPI_LSTM_BWD, stream);
}

int launch_conv_tc(const void* src0, const void* src1, const void* wpacked, ConvTcParams p, int epi,
                   cudaStream_t stream) {
    if (p.C1 > 0 && !src1) {
        set_last_error("conv_tc: C1 > 0 but src1 is null");
        return B200_ERR_ARG;
    }
    const int Ct = p.wK > 0 ? p.wK : p.C0 + p.C1;
    const int esize = p.in_fp32 ? 4 : 2;
    const int kc = pick_kc(p.C0, p.C1, esize);   // K-block rows of 128 .. 32 bytes
    if (kc == 0) {
        set_last_error("conv_tc: channel counts C0=%d C1=%d are not multiples of %d", p.C0, p.C1, 32 / esize);
        return B200_ERR_SHAPE;
    }
    if (p.kb_split > 0 && (epi != EPI_STORE || p.seq_T > 0 || !p.out_fp32 || p.bias || p.scale || p.relu ||
                           p.accumulate || p.stat_sum || p.shuf_C > 0 || p.split != p.N)) {
        set_last_error("conv_tc: split K stores plain fp32 partial sums (no bias, scale, relu, statistics or shuffle)");
        return B200_ERR_ARG;
    }
    const int splits = p.kb_split > 0 ? (p.ksize * p.ksize * (p.C0 / kc + p.C1 / kc) + p.kb_split - 1) / p.kb_split : 1;
    if (p.in_fp32 && (epi == EPI_LSTM_BWD || p.seq_T > 0 || p.stat_sum || p.shuf_C > 0 || !(p.out_fp32 || epi == EPI_LSTM))) {
        set_last_error("conv_tc: the tf32 mode covers plain fp32-output convolutions and the single-step fused cell");
        return B200_ERR_ARG;
    }
    p.kc = kc;
    const int block_n = pick_block_n(p.N, epi);
    if (block_n == 0) {
        set_last_error("conv_tc: N=%d not supported for epilogue %d", p.N, epi);
        return B200_ERR_SHAPE;
    }
    MTile mt;
    if (!plan_mtile(p.B, p.H, p.W, BLOCK_M, &mt)) {
        set_last_error("conv_tc: spatial shape B=%d H=%d W=%d cannot be tiled", p.B, p.H, p.W);
        return B200_ERR_SHAPE;
    }
    p.Wt = mt.Wt;
    p.Ht = mt.Ht;
    p.Bt = mt.Bt;
    p.tiles_w = mt.tiles_w;
    p.tiles_h = mt.tiles_h;
    p.tiles_b = mt.tiles_b;
    const int map_T = p.seq_T > 0 ? p.seq_T : p.T;
    if (p.seq_T > 0) p.T = 1;  // tiles of ONE step; the kernel iterates over the steps itself
    p.num_m_tiles = p.T * mt.tiles_w * mt.tiles_h * mt.tiles_b;
    p.num_n_tiles = (p.N + block_n - 1) / block_n;
    static const bool alt_ok = [] {
        const char* e = getenv("B200_BWD_ALTERNATE");  // developer switch (A/B of the tile order)
        return !e || atoi(e) != 0;
    }();
    p.bwd_alternate = (alt_ok && epi == EPI_LSTM_BWD && (p.num_n_tiles & 1) == 0 &&
                       p.bwd_Cin == (p.num_n_tiles / 2) * block_n) ? 1 : 0;
    p.pad = p.ksize / 2;
    p.err_flag = device_error_flag();

    CUtensorMap ta0, ta1, tb;
    int rc = make_act_tmap(&ta0, src0, p.C0, p.W, p.H, p.B, map_T, kc, mt.Wt, mt.Ht, mt.Bt, esize);
    if (rc != B200_OK) return rc;
    if (p.C1 > 0) {
        rc = make_act_tmap(&ta1, src1, p.C1, p.W, p.H, p.B, map_T, kc, mt.Wt, mt.Ht, mt.Bt, esize);
        if (rc != B200_OK) return rc;
    } else {
        ta1 = ta0;
    }
    // rows beyond N inside the last N tile are TMA out-of-bounds reads => zero filled
    rc = make_w_tmap(&tb, wpacked, Ct, p.N, p.ksize * p.ksize, kc, block_n, esize);
    if (rc != B200_OK) return rc;

    if (epi == EPI_LSTM) {
        switch (block_n) {
            case 256: return launch_impl<256, EPI_LSTM>(ta0, ta1, tb, p, stream);
            case 128: return launch_impl<128, EPI_LSTM>(ta0, ta1, tb, p, stream);
            default: return launch_impl<64, EPI_LSTM>(ta0, ta1, tb, p, stream);
        }
    }
    if (epi == EPI_LSTM_BWD) {
        switch (block_n) {
            case 256: return launch_impl<256, EPI_LSTM_BWD>(ta0, ta1, tb, p, stream);
            case 128: return launch_impl<128, EPI_LSTM_BWD>(ta0, ta1, tb, p, stream);
            default: return launch_impl<64, EPI_LSTM_BWD>(ta0, ta1, tb, p, stream);
        }
    }
    switch (block_n) {
        case 256: return launch_impl<256, EPI_STORE>(ta0, ta1, tb, p, stream, splits);
        case 128: return launch_impl<128, EPI_STORE>(ta0, ta1, tb, p, stream, splits);
        default: return launch_impl<64, EPI_STORE>(ta0, ta1, tb, p, stream, splits);
    }
}

}  // namespace b200
