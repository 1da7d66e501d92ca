// tcgen05 / TMEM implicit-GEMM convolution kernels for sm_100a.
//
// One kernel family covers every dense contraction of the Pix2Pix U-Net + PatchGAN hot path
// (reference call sites: models/pix2pix.py:63-69 Conv2d(4,2,1), :99-105 ConvTranspose2d(4,2,1),
// models/wrapper.py:229-233 discriminator convs):
//
//   igemm_fprop_kernel : out[pix, co] = act( bias[co] + sum_{tap, ci} A[pix + tap, ci] * Wp[co, tap, ci] )
//       A is an NHWC bf16 tensor seen through a 5-D TMA map (C', W', P, H', N).  A stride-2 4x4
//       convolution uses the "parity split" view C' = 2C, W' = W/2, P = 2, H' = H/2, so every tap is
//       a dense, unit-stride box and zero padding is the TMA out-of-bounds fill.  A transposed
//       convolution runs as 4 sub-pixel phases (blockIdx.z), each a 2x2 unit-stride conv.  The same
//       kernel therefore also is Conv dgrad (== ConvT fprop) and ConvT dgrad (== Conv fprop).
//   igemm_wgrad_kernel : dW[tap][cu][cs] += sum_pix U[pix, cu] * S[pix + tap, cs]
//       both operands MN-major straight out of the NHWC activations / gradients.
//
// Tile: M = 128 pixels (TMEM lanes), N = n_tile channels (TMEM columns), K-block = 64 channels
// (one SWIZZLE_128B row).  Warp roles: 0 = TMA producer, 1 = MMA issuer, 2 = TMEM allocator,
// 4..11 (fprop; 4..7 wgrad) = epilogue (TMEM -> registers -> global; fprop bf16 tiles through a shared-memory box and a
// TMA store).
#include <stdio.h>
#include <stdlib.h>

#include "pai_common.cuh"
#include "pai_epilogue.cuh"
#include "pai_kernels.h"

namespace pai {

// Optional role timing (build.sh -DPAI_PROFILE_ROLES): CTA 0 prints how its TMA producer, MMA issuer and one epilogue
// warp split their cycles between waiting and working -- the measurement that says which role starves the tensor pipe.
#ifdef PAI_PROFILE_ROLES
#define ROLE_T0() const long long _t0 = clock64()
#define ROLE_ADD(var) var += clock64() - _t0
#else
#define ROLE_T0()
#define ROLE_ADD(var)
#endif

static constexpr int kThreads = 256;       // wgrad: 4 control/idle warps + 4 epilogue warps
static constexpr int kFpropThreads = 384;  // fprop: 4 control/idle warps + 8 epilogue warps
static constexpr int kMaxStages = 8;

struct __align__(8) PipeSmem {
    uint64_t full[kMaxStages];
    uint64_t empty[kMaxStages];
    uint64_t acc_full[2];
    uint64_t acc_empty[2];
    uint64_t mask_full[8];        // fprop, masked: per epilogue warp, its TMA load of saved activations has landed
    uint32_t tmem_base;
};

// =============================================================================================
// Persistent: one CTA per SM walks tiles t = blockIdx.x, blockIdx.x + gridDim.x, ...  The fp32
// accumulator is double-buffered in TMEM so the epilogue of tile i overlaps the MMAs of tile i+1.
// Tile order: output-channel tile fastest, so CTAs running at the same time share the A tile in L2.
//
// PAIR = true: the kernel runs as 2-CTA clusters (the two SMs of a TPC).  A pair owns an M = 256 tile: each CTA stages its
// own 128 pixels of A and HALF of the weight tile (n_tile / 2 rows), the leader CTA issues tcgen05.mma.cta_group::2 and
// the accumulator rows of each half land in that CTA's own TMEM, so every SM pulls a third less operand data through L2
// per FLOP (the large layers are L2 -> SM bound, profiles/r1_igemm_fprop_step_summary.txt) and one instruction stream
// drives two tensor cores.  `full` barriers live in the leader (both CTAs' TMA loads complete on them), `empty` /
// `acc_full` are signalled in both CTAs by multicast commits, both epilogues release the leader's `acc_empty`.
template <bool PAIR, bool MASKED>
__global__ void __launch_bounds__(kFpropThreads, 1)
igemm_fprop_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                   const __grid_constant__ IgemmOutMaps om, const IgemmFpropParams p) {
    pdl_launch_dependents();
    extern __shared__ uint8_t smem_raw[];
    __shared__ PipeSmem ps;
    // per epilogue warp: 32 rows x 128 B in the SWIZZLE_128B layout (16-byte chunk c of row r at c ^ (r & 7)), the source
    // box of its TMA stores (and the destination of its TMA loads of saved activations)
    __shared__ __align__(1024) uint4 stage_buf[8][32 * 8];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_tile = p.n_tile;
    const bool fused = p.fused_phases != 0;
    const uint32_t rank = PAIR ? cluster_ctarank() : 0u;    // 0 = leader (issues the MMAs)
    const int cta_n = PAIR ? n_tile / 2 : n_tile;           // weight-tile rows staged by this CTA
    const uint32_t a_bytes = 128 * 128;
    const uint32_t b_bytes = (uint32_t)cta_n * 128;
    // A pipeline stage holds p.ksub (1 or 2) 64-channel K blocks, each [A box | weight box(es)]: the MMA-issuing thread
    // pays its per-stage costs (barrier wait, fence, commit, loop) once per 8 MMAs instead of once per 4
    const int ksub = p.ksub;
    const uint32_t sub_bytes = a_bytes + (fused ? 4 : 1) * b_bytes;
    const uint32_t stage_bytes = (uint32_t)ksub * sub_bytes;
    const int stages = p.stages;
    const int num_kb = (fused ? 9 : p.ntaps) * p.kc_per_tap;
    const int acc_n = fused ? 4 * n_tile : n_tile;          // accumulator columns per tile
    const uint32_t acc_cols = tmem_cols_for(acc_n);
    // p.m_tiles counts the units a worker walks: 128-pixel tiles, or (PAIR) pairs of them
    const int total_tiles = p.n_tiles * p.m_tiles * p.phases * p.splitk;
    const int worker = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int workers = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tm_a);
        tma_prefetch_desc(&tm_b);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&ps.full[s], 1);
            mbar_init(&ps.empty[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&ps.acc_full[a], 1);
            mbar_init(&ps.acc_empty[a], PAIR ? 16 : 8);       // one arrival per epilogue warp (and CTA)
        }
        if (MASKED)
            for (int w = 0; w < 8; ++w) mbar_init(&ps.mask_full[w], 1);
        mbar_fence_init();
    }
    if (warp == 2) {
        if (PAIR)
            tmem_alloc_pair(&ps.tmem_base, 2 * acc_cols);
        else
            tmem_alloc(&ps.tmem_base, 2 * acc_cols);
    }
    tc_fence_before();
    if (PAIR)
        cluster_sync_all();          // the peer's barriers are initialised before anything remote touches them
    else
        __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = ps.tmem_base;
    pdl_wait();      // everything above overlapped the previous kernel's tail; its outputs are visible from here on

    long long prof_wait = 0, prof_wait2 = 0, prof_total = 0, prof_fence = 0, prof_issue = 0, prof_commit = 0;
    (void)prof_wait, (void)prof_wait2, (void)prof_total, (void)prof_fence, (void)prof_issue, (void)prof_commit;
    // TMA producers: warps 0, 2 and 3 deal the k-blocks round-robin.  One elected thread needs ~250 cycles per
    // cp.async.bulk.tensor (coordinate set-up, barrier wait, issue) -- measured with -DPAI_PROFILE_ROLES: a single
    // producer was busy 78 % of the kernel and the MMA thread waited on it -- while an N = 128 k-block is only 256 cycles
    // of tensor time.
    const int pidx = warp == 0 ? 0 : (warp == 2 ? 1 : (warp == 3 ? 2 : -1));
    if (pidx >= 0) {
        if (elect_one()) {
            constexpr int P = 3;
            int g = 0, mine = pidx;              // running k-block count of this CTA / the next one this thread loads
            int stage = pidx;
            uint32_t phase = 0;
            while (stage >= stages) stage -= stages, phase ^= 1;
            const int brow = PAIR ? (int)rank * cta_n : 0;     // this CTA's half of the weight tile
#ifdef PAI_PROFILE_ROLES
            const long long tstart = clock64();
#endif
            for (int t = worker; t < total_tiles; t += workers) {
                int ks, tt, nt, r, mt, phase_idx, tw, th, tn;
                p.fd_splitk.divmod(t, tt, ks);
                p.fd_n_tiles.divmod(tt, r, nt);
                p.fd_m_tiles.divmod(r, phase_idx, mt);
                if (PAIR) mt = 2 * mt + (int)rank;       // an odd tile count leaves the last peer tile out of bounds: zero fill
                p.fd_tiles_w.divmod(mt, mt, tw);
                p.fd_tiles_h.divmod(mt, tn, th);
                const int w0 = tw * p.bw, h0 = th * p.bh, n0 = tn * p.bn;
                const int col0 = nt * n_tile;
                const int kb_begin = num_kb * ks / p.splitk, kb_end = num_kb * (ks + 1) / p.splitk;
                const int g_end = g + (kb_end - kb_begin) / ksub;        // stages of this tile (host: ksub | k-blocks)
                // this worker's next tile: its activation boxes are prefetched into L2 box by box alongside the loads
                int pw0 = 0, ph0 = 0, pn0 = 0, pphase = 0;
                const bool pf = p.prefetch_taps != 0 && t + workers < total_tiles;
                if (pf) {
                    int r2, m2, tw2, th2, tn2;
                    p.fd_n_tiles.divmod(p.fd_splitk.quot(t + workers), r2, tn2);
                    p.fd_m_tiles.divmod(r2, pphase, m2);
                    if (PAIR) m2 = 2 * m2 + (int)rank;
                    p.fd_tiles_w.divmod(m2, m2, tw2);
                    p.fd_tiles_h.divmod(m2, tn2, th2);
                    pw0 = tw2 * p.bw, ph0 = th2 * p.bh, pn0 = tn2 * p.bn;
                }
                for (; mine < g_end; mine += P) {
                    const int kb0 = kb_begin + (mine - g) * ksub;
                    {
                        ROLE_T0();
                        mbar_wait(&ps.empty[stage], phase ^ 1);
                        ROLE_ADD(prof_wait);
                    }
                    uint8_t* st = smem + (size_t)stage * stage_bytes;
                    int tap, kc;
                    p.fd_kc.divmod(kb0, tap, kc);                // fused: tap = box index 0..8 (ksub | kc_per_tap)
                    const int nu = fused ? p.box_nu[tap] : 1;
                    const uint32_t tx = (uint32_t)ksub * (a_bytes + nu * b_bytes);
                    if (!PAIR || rank == 0) mbar_expect_tx(&ps.full[stage], PAIR ? 2 * tx : tx);
                    for (int j = 0; j < ksub; ++j) {
                        uint8_t* sa = st + (size_t)j * sub_bytes;
                        uint8_t* sb = sa + a_bytes;
                        const int kb = kb0 + j;
                        if (fused) {
                            const int kcj = kc + j;
                            if (PAIR)
                                tma_load_5d_pair(sa, &tm_a, &ps.full[stage], kcj * 64, w0 + p.box_w[tap], 0, h0 + p.box_h[tap], n0);
                            else
                                tma_load_5d(sa, &tm_a, &ps.full[stage], kcj * 64, w0 + p.box_w[tap], 0, h0 + p.box_h[tap], n0);
                            if (pf && ((p.prefetch_taps >> tap) & 1u))
                                tma_prefetch_5d(&tm_a, kcj * 64, pw0 + p.box_w[tap], 0, ph0 + p.box_h[tap], pn0);
                            if (PAIR && p.box_merge[tap]) {
                                // one MMA of N = 64 * nu: the N dimension of a cta_group::2 tile is split [first half |
                                // second half] between the two CTAs, so this CTA stages the WHOLE 64-row weight boxes of
                                // its half of the users (two 32-row loads each) instead of half of every box
                                const int per = nu >> 1;
                                for (int v = 0; v < per; ++v) {
                                    const int pt = p.box_users[tap][(int)rank * per + v], ph = pt >> 2, tp = pt & 3;
                                    for (int hr = 0; hr < 2; ++hr)
                                        tma_load_2d_pair(sb + (2 * v + hr) * b_bytes, &tm_b, &ps.full[stage],
                                                         (tp * p.kc_per_tap + kcj) * 64, ph * p.b_rows_per_phase + hr * cta_n);
                                }
                            } else {
                                for (int u = 0; u < nu; ++u) {
                                    const int pt = p.box_users[tap][u], ph = pt >> 2, tp = pt & 3;
                                    if (PAIR)
                                        tma_load_2d_pair(sb + u * b_bytes, &tm_b, &ps.full[stage], (tp * p.kc_per_tap + kcj) * 64,
                                                         ph * p.b_rows_per_phase + brow);
                                    else
                                        tma_load_2d(sb + u * b_bytes, &tm_b, &ps.full[stage], (tp * p.kc_per_tap + kcj) * 64,
                                                    ph * p.b_rows_per_phase);
                                }
                            }
                        } else {
                            int tapj, kcj;
                            p.fd_kc.divmod(kb, tapj, kcj);
                            const int ti = phase_idx * p.ntaps + tapj;
                            if (pf && ((p.prefetch_taps >> tapj) & 1u)) {
                                const int tj = pphase * p.ntaps + tapj;
                                tma_prefetch_5d(&tm_a, p.tap_c[tj] + kcj * 64, pw0 + p.tap_w[tj], p.tap_p[tj], ph0 + p.tap_h[tj], pn0);
                            }
                            if (PAIR) {
                                tma_load_5d_pair(sa, &tm_a, &ps.full[stage], p.tap_c[ti] + kcj * 64, w0 + p.tap_w[ti], p.tap_p[ti],
                                                 h0 + p.tap_h[ti], n0);
                                tma_load_2d_pair(sb, &tm_b, &ps.full[stage], kb * 64, phase_idx * p.b_rows_per_phase + col0 + brow);
                            } else {
                                tma_load_5d(sa, &tm_a, &ps.full[stage], p.tap_c[ti] + kcj * 64, w0 + p.tap_w[ti], p.tap_p[ti],
                                            h0 + p.tap_h[ti], n0);
                                tma_load_2d(sb, &tm_b, &ps.full[stage], kb * 64, phase_idx * p.b_rows_per_phase + col0);
                            }
                        }
                    }
                    stage += P;
                    while (stage >= stages) stage -= stages, phase ^= 1;
                }
                g = g_end;
            }
#ifdef PAI_PROFILE_ROLES
            if (blockIdx.x == 0 && pidx == 0) printf("[roles] producer 0 of 3: total %lld cyc, waiting for empty stages %lld\n", clock64() - tstart, prof_wait);
#endif
        }
    } else if (warp == 1) {
        if (rank == 0) {
            // MMA issuer.  The WHOLE warp walks the loops -- warp-uniform control flow lets the compiler keep the stage
            // counter, barrier addresses and descriptor words in uniform registers -- and one elected lane issues.  The
            // issuing thread is the critical path of every N <= 128 layer (a lone warp pays the full latency of each
            // dependent instruction: -DPAI_PROFILE_ROLES showed ~290 cycles per stage outside the MMAs against 256
            // cycles of tensor work, and 700 per stage in the phase-fused mode), so everything that does not depend on
            // the stage is computed once per tile or per box and the per-stage work is: wait, fence, two 32-bit
            // descriptor words, the MMAs, the commit.
            const uint32_t idesc = umma_idesc_bf16(PAIR ? 256 : 128, n_tile, 0, 0);
            const uint32_t idesc_n2 = umma_idesc_bf16(PAIR ? 256 : 128, fused ? 2 * n_tile : n_tile, 0, 0);
            const uint32_t idesc_n4 = umma_idesc_bf16(PAIR ? 256 : 128, fused ? 4 * n_tile : n_tile, 0, 0);
            const uint32_t full0 = smem_u32(&ps.full[0]), empty0 = smem_u32(&ps.empty[0]);
            const uint32_t acc_full0 = smem_u32(&ps.acc_full[0]), acc_empty0 = smem_u32(&ps.acc_empty[0]);
            const uint32_t a_lo0 = umma_desc_lo_kmajor(smem_u32(smem));
            const uint32_t stage_units = stage_bytes >> 4, sub_units = sub_bytes >> 4, a_units = a_bytes >> 4, b_units = b_bytes >> 4;
            const int kmma = p.kmma, kc_per_tap = p.kc_per_tap, splitk = p.splitk;
            int stage = 0;
            uint32_t phase = 0;
            int it = 0;
#ifdef PAI_PROFILE_ROLES
            const long long tstart = clock64();
#endif
            for (int t = worker; t < total_tiles; t += workers, ++it) {
                const int a = it & 1;
                const uint32_t acc_phase = (it >> 1) & 1;
                {
                    ROLE_T0();
                    mbar_wait_u32(acc_empty0 + 8 * a, acc_phase ^ 1);   // epilogue has drained this accumulator
                    ROLE_ADD(prof_wait2);
                }
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + a * acc_cols;
                if (fused) {
                    // 9 boxes x kc_per_tap channel blocks, box-major (the producers' order); the centre box comes first
                    // and starts all four accumulators, so everything after its first channel block accumulates
                    for (int box = 0; box < 9; ++box) {
                        const int nu = p.box_nu[box];
                        const bool merged = p.box_merge[box] != 0;
                        const int groups = merged ? 1 : nu;
                        const uint32_t idesc_u = merged ? (nu == 2 ? idesc_n2 : idesc_n4) : idesc;
                        const uint32_t td0 = tmem_d + p.box_col[box][0] * n_tile, td1 = tmem_d + p.box_col[box][1] * n_tile;
                        const uint32_t td2 = tmem_d + p.box_col[box][2] * n_tile, td3 = tmem_d + p.box_col[box][3] * n_tile;
                        for (int kc = 0; kc < kc_per_tap; kc += ksub) {
                            {
                                ROLE_T0();
                                mbar_wait_u32(full0 + 8 * stage, phase);
                                ROLE_ADD(prof_wait);
                            }
                            tc_fence_after();
                            if (elect_one()) {
                                for (int j = 0; j < ksub; ++j) {
                                    const uint32_t a_lo = a_lo0 + stage * stage_units + j * sub_units, b_lo = a_lo + a_units;
                                    const uint32_t acc = (box | kc | j) != 0;
                                    umma_kblock_lo<PAIR, 4>(td0, a_lo, b_lo, idesc_u, acc);
                                    if (groups > 1) umma_kblock_lo<PAIR, 4>(td1, a_lo, b_lo + b_units, idesc_u, acc);
                                    if (groups > 2) {      // only with PAI_NO_PHASE_MERGE: the centre box as 4 N = 64 MMAs
                                        umma_kblock_lo<PAIR, 4>(td2, a_lo, b_lo + 2 * b_units, idesc_u, acc);
                                        umma_kblock_lo<PAIR, 4>(td3, a_lo, b_lo + 3 * b_units, idesc_u, acc);
                                    }
                                }
                                umma_commit_u32<PAIR>(empty0 + 8 * stage);     // frees the stage (in both CTAs)
                            }
                            if (++stage == stages) {
                                stage = 0;
                                phase ^= 1;
                            }
                        }
                    }
                } else {
                    const int ks = t - p.fd_splitk.quot(t) * splitk;
                    const int kb_begin = num_kb * ks / splitk, kb_end = num_kb * (ks + 1) / splitk;
                    if (kmma == 4) {
                        for (int kb = kb_begin; kb < kb_end; kb += ksub) {
                            {
                                ROLE_T0();
                                mbar_wait_u32(full0 + 8 * stage, phase);
                                ROLE_ADD(prof_wait);
                            }
                            tc_fence_after();
                            const uint32_t a_lo = a_lo0 + stage * stage_units, b_lo = a_lo + a_units;
                            if (elect_one()) {
                                umma_kblock_lo<PAIR, 4>(tmem_d, a_lo, b_lo, idesc, kb != kb_begin);
                                if (ksub > 1) umma_kblock_lo<PAIR, 4>(tmem_d, a_lo + sub_units, b_lo + sub_units, idesc, 1u);
                                umma_commit_u32<PAIR>(empty0 + 8 * stage);
                            }
                            if (++stage == stages) {
                                stage = 0;
                                phase ^= 1;
                            }
                        }
                    } else {
                        // thin im2col operands: one K block of which only the first 16 * kmma columns hold data (ksub == 1)
                        for (int kb = kb_begin; kb < kb_end; ++kb) {
                            mbar_wait_u32(full0 + 8 * stage, phase);
                            tc_fence_after();
                            const uint32_t a_lo = a_lo0 + stage * stage_units, b_lo = a_lo + a_units;
                            if (elect_one()) {
                                const uint32_t acc = kb != kb_begin;
                                if (kmma == 1)
                                    umma_kblock_lo<PAIR, 1>(tmem_d, a_lo, b_lo, idesc, acc);
                                else if (kmma == 2)
                                    umma_kblock_lo<PAIR, 2>(tmem_d, a_lo, b_lo, idesc, acc);
                                else
                                    umma_kblock_lo<PAIR, 3>(tmem_d, a_lo, b_lo, idesc, acc);
                                umma_commit_u32<PAIR>(empty0 + 8 * stage);
                            }
                            if (++stage == stages) {
                                stage = 0;
                                phase ^= 1;
                            }
                        }
                    }
                }
                if (elect_one()) umma_commit_u32<PAIR>(acc_full0 + 8 * a);      // the epilogue(s) may read the tile
            }
#ifdef PAI_PROFILE_ROLES
            if (blockIdx.x == 0 && elect_one())
                printf("[roles] mma: total %lld cyc, waiting for full stages %lld, for a drained accumulator %lld, tiles %d, k-blocks/tile %d; unfused: fence %lld issue %lld commit %lld\n",
                       clock64() - tstart, prof_wait, prof_wait2, it, num_kb / p.splitk, prof_fence, prof_issue, prof_commit);
#endif
        }
    } else if (warp >= 4) {
        // 8 epilogue warps: warp w may read TMEM lanes (w % 4) * 32 .. +31, so the two warps of a lane quarter
        // split the work items (64-column chunk x output, or 16-column steps on the generic path) between them
        const int q = warp & 3;
        const int half = (warp - 4) >> 2;
        const int r = q * 32 + lane;
        // this lane's row (TMEM lane r) inside the pixel box, packed w | h << 8 | n << 16 (each < 128): six separate
        // position registers, live across the whole tile loop, made the epilogue spill at the 168-register cap
        const int rpos = (r % p.bw) | (((r / p.bw) % p.bh) << 8) | ((r / (p.bw * p.bh)) << 16);
        const int n_out = p.out2 != nullptr ? 2 : 1;
        // The warp's 32 rows are one box of the pixel grid (rows run w-fastest over the power-of-two bw x bh x bn tile box):
        // its corner inside the tile box is lane 0's row position.  The bf16 path writes a 64-channel chunk of them with ONE TMA store of the
        // staging tile -- per-lane shared-memory reads and global stores share the MIO pipe with the barrier traffic of
        // the producer and MMA warps, and slowed the main loop (profiles/r2_igemm_ablation.txt) -- and the TMA clips the
        // rows and channels outside the output.
        const int qpos = __shfl_sync(0xffffffffu, rpos, 0);
        uint4* tile = stage_buf[warp - 4];
        uint32_t mask_phase = 0;
        // BatchNorm / bias-gradient column sums: this lane's 8 channels (chunk lane % 8) of rows i * 4 + lane / 8, carried
        // in registers ACROSS tiles and reduced over the 4 row groups + added to the CTA's partial row only when the
        // warp moves to other columns or runs out of tiles (before: 32 shared-memory loads and 4 reductions per chunk)
        // (only where the warp stays on ONE 64-channel block -- N <= 128 or the phase-fused tiles; elsewhere the chunk's
        // sums are reduced and added right after its stores)
        const bool st_persist = fused || acc_n <= 128;
        float st_sum[8], st_sq[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) st_sum[j] = st_sq[j] = 0.f;
        int st_col = -1;                               // first channel of the 64 the accumulators belong to
        // reduce over the 4 row groups (lanes l, l^8, l^16, l^24 hold the same channels) and add to the CTA's partial row
        auto reduce_add = [&](float (&su)[8], float (&sq)[8], int col) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                su[j] += __shfl_xor_sync(0xffffffffu, su[j], 8);
                su[j] += __shfl_xor_sync(0xffffffffu, su[j], 16);
                sq[j] += __shfl_xor_sync(0xffffffffu, sq[j], 8);
                sq[j] += __shfl_xor_sync(0xffffffffu, sq[j], 16);
            }
            if (lane < 8) {
                float* bp = p.bn_part + (size_t)blockIdx.x * (2 * p.cout) + col + lane * 8;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    atomicAdd(bp + j, su[j]);
                    atomicAdd(bp + p.cout + j, sq[j]);
                }
            }
        };
        auto flush_stats = [&]() {
            if (st_col < 0) return;
            reduce_add(st_sum, st_sq, st_col);
#pragma unroll
            for (int j = 0; j < 8; ++j) st_sum[j] = st_sq[j] = 0.f;
            st_col = -1;
        };
        int it = 0;
        for (int t = worker; t < total_tiles; t += workers, ++it) {
            int nt, rr, mt, phase_idx, tw, th, tn;
            const int tt = p.fd_splitk.quot(t);
            p.fd_n_tiles.divmod(tt, rr, nt);
            p.fd_m_tiles.divmod(rr, phase_idx, mt);
            if (PAIR) mt = 2 * mt + (int)rank;
            p.fd_tiles_w.divmod(mt, mt, tw);
            p.fd_tiles_h.divmod(mt, tn, th);
            const int col0 = nt * n_tile;
            const int gw = tw * p.bw + (rpos & 255), gh = th * p.bh + ((rpos >> 8) & 255), gn = tn * p.bn + (rpos >> 16);
            const bool row_ok = (gw < p.gw) && (gh < p.gh) && (gn < p.gn);
            const int a = it & 1;
            const uint32_t acc_phase = (it >> 1) & 1;
            const bool fast = p.tma_out && (n_tile & 63) == 0 && col0 + n_tile <= p.cout &&
                              (p.bias == nullptr || (reinterpret_cast<uintptr_t>(p.bias) & 15) == 0);
            // (the fused-phase mode is only launched when this holds: cout == n_tile == 64, bf16 output)
            // the warp's box on the grid
            const int bw0 = tw * p.bw + (qpos & 255), bh0 = th * p.bh + ((qpos >> 8) & 255), bn0 = tn * p.bn + (qpos >> 16);
            // fused activation backward: lane 0 TMA-loads the saved activations of the warp's chunk c (the output's box
            // in the saved tensor; zeros outside it) into the staging tile once the previous store has read it -- the
            // first chunk while the MMAs of the tile are still running, the next one behind the current chunk's store
            const bool masked = MASKED && p.mask_src != nullptr && fast;   // (MASKED: the instantiation of pai_conv4x4_dgrad_act)
            auto mask_load = [&](int c) {
                __syncwarp();                   // every lane is done reading the tile
                if (lane == 0) {
                    bulk_wait_group_read0();
                    mbar_expect_tx(&ps.mask_full[warp - 4], 32 * 128);
                    tma_load_4d(tile, &om.aux[fused ? c >> 6 : phase_idx], &ps.mask_full[warp - 4], col0 + (fused ? 0 : c),
                                bw0, bh0, bn0);
                }
            };
            if (masked && 64 * half < acc_n) mask_load(64 * half);
            {
                ROLE_T0();
                mbar_wait(&ps.acc_full[a], acc_phase);
                ROLE_ADD(prof_wait);
            }
#ifdef PAI_PROFILE_ROLES
            const long long twork = clock64();
#endif
            tc_fence_after();
            const uint32_t tmem_d = tmem_base + a * acc_cols + ((uint32_t)(q * 32) << 16);
            // The accumulator is handed back as soon as this warp's LAST chunk sits in registers -- before its bias /
            // statistics / store work -- with a relaxed arrival (2 x 8 warps release a pair's accumulators, 8 otherwise).
            bool released = false;
            auto release_acc = [&]() {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {                        // (every lane fenced its TMEM reads before the __syncwarp)
                    if (PAIR)
                        mbar_arrive_leader_relaxed(&ps.acc_empty[a]);
                    else
                        mbar_arrive_relaxed(&ps.acc_empty[a]);
                }
                released = true;
            };
            if (fast) {
                // ---- bf16 path: 64 channels of the warp's 32 rows are packed into the swizzled staging tile, which one
                // TMA store writes out; lane 0 issues every store of the warp and owns its bulk async-groups
                // rows of the tile inside the output grid, for the column sums (bit i: row i of the warp's 32)
                const uint32_t rows_ok = __ballot_sync(0xffffffffu, row_ok);
                int item = 0;
                const int n_items = (acc_n >> 6) * n_out;
                const int last_item = ((n_items - 1) & 1) == half ? n_items - 1 : n_items - 2;   // of this warp (< 0: none)
                for (int c = 0; c < acc_n; c += 64) {
                    // fused phases: chunk c is phase (column block) c/64 of the same 64 output channels
                    const int oc = fused ? 0 : c;
                    for (int which = 0; which < n_out; ++which, ++item) {
                        if ((item & 1) != half) continue;
                        uint32_t v[64];
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            tmem_ld_16(tmem_d + (uint32_t)(c + 16 * j), *reinterpret_cast<uint32_t(*)[16]>(&v[16 * j]));
                        tmem_ld_wait();
                        if (item == last_item) release_acc();
                        const int act = which == 0 ? p.act : p.act2;
                        const float* bias_c = p.bias != nullptr ? p.bias + col0 + oc : nullptr;
                        if (masked) {
                            mbar_wait(&ps.mask_full[warp - 4], mask_phase);
                            mask_phase ^= 1;
                            mask_pack(v, p.mask_slope, tile, lane);
                        } else {
                            if (lane == 0) bulk_wait_group_read0();     // the previous store has read the tile
                            __syncwarp();
                            // activation / bias dispatch hoisted out of the 64-element loop
                            if (act == PAI_ACT_LEAKY)
                                bias_act_pack<PAI_ACT_LEAKY>(v, bias_c, p.slope, tile, lane);
                            else if (act == PAI_ACT_RELU)
                                bias_act_pack<PAI_ACT_RELU>(v, bias_c, p.slope, tile, lane);
                            else if (act == PAI_ACT_TANH)
                                bias_act_pack<PAI_ACT_TANH>(v, bias_c, p.slope, tile, lane);
                            else
                                bias_act_pack<PAI_ACT_NONE>(v, bias_c, p.slope, tile, lane);
                        }
                        fence_proxy_async_smem();
                        __syncwarp();
                        if (lane == 0) {
                            tma_store_4d(which == 0 ? &om.out[fused ? c >> 6 : phase_idx] : &om.aux[0], tile, col0 + oc,
                                         bw0, bh0, bn0);
                            bulk_commit_group();
                        }
                        const bool stats = p.bn_part != nullptr && which == 0;
                        if (stats) {
                            if (st_persist && st_col != col0 + oc) {
                                flush_stats();
                                st_col = col0 + oc;
                            }
                            // this chunk's column sums over the rows inside the grid: exactly the stored bf16 values
                            float cs[8], cq[8];
#pragma unroll
                            for (int j = 0; j < 8; ++j) cs[j] = cq[j] = 0.f;
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                const int row = i * 4 + (lane >> 3), ch = lane & 7;
                                if ((rows_ok >> row) & 1u) {
                                    const uint4 val = tile[row * 8 + (ch ^ (row & 7))];
                                    const __nv_bfloat162* hv = reinterpret_cast<const __nv_bfloat162*>(&val);
#pragma unroll
                                    for (int j = 0; j < 4; ++j) {
                                        const float2 f = __bfloat1622float2(hv[j]);
                                        cs[2 * j] += f.x;
                                        cs[2 * j + 1] += f.y;
                                        cq[2 * j] = fmaf(f.x, f.x, cq[2 * j]);
                                        cq[2 * j + 1] = fmaf(f.y, f.y, cq[2 * j + 1]);
                                    }
                                }
                            }
                            if (st_persist) {
#pragma unroll
                                for (int j = 0; j < 8; ++j) st_sum[j] += cs[j], st_sq[j] += cq[j];
                            } else {
                                reduce_add(cs, cq, col0 + oc);
                            }
                        }
                        if (masked && c + 128 < acc_n) mask_load(c + 128);   // this warp's next chunk
                    }
                }
            } else {
                // ---- generic path (fp32 output, narrow or ragged tiles, split-K accumulation, unaligned bf16 rows)
                const long long off = p.out_phase_off[phase_idx] + (long long)gn * p.out_sn + (long long)gh * p.out_sh +
                                      (long long)gw * p.out_sw + col0;
                const long long off2 = (long long)gn * p.out2_sn + (long long)gh * p.out2_sh + (long long)gw * p.out2_sw + col0;
                const bool vec_ok = ((p.cout & 7) == 0) && ((off & 7) == 0) && ((off2 & 7) == 0);
                int step = 0;
                for (int cc = 0; cc < n_tile; cc += 16, ++step) {
                    if ((step & 1) != half) continue;
                    uint32_t v[16];
                    __syncwarp();
                    tmem_ld_16(tmem_d + (uint32_t)cc, v);
                    tmem_ld_wait();
                    if (!row_ok || col0 + cc >= p.cout) continue;
                    float f[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        float x = __uint_as_float(v[j]);
                        if (p.bias != nullptr && col0 + cc + j < p.cout) x += __ldg(p.bias + col0 + cc + j);
                        f[j] = x;
                    }
                    if (p.accumulate) {
                        float* o = reinterpret_cast<float*>(p.out) + off + cc;
                        if (col0 + cc + 16 <= p.cout && ((off + cc) & 3) == 0) {
#pragma unroll
                            for (int j = 0; j < 16; j += 4) red_add_v4(o + j, f[j], f[j + 1], f[j + 2], f[j + 3]);
                        } else {
#pragma unroll
                            for (int j = 0; j < 16; ++j)
                                if (col0 + cc + j < p.cout) atomicAdd(o + j, f[j]);
                        }
                    } else if (p.out_f32) {
                        float* o = reinterpret_cast<float*>(p.out) + off + cc;
                        if (col0 + cc + 16 <= p.cout && ((off + cc) & 3) == 0 && p.act == PAI_ACT_NONE) {
#pragma unroll
                            for (int j = 0; j < 16; j += 4)
                                *reinterpret_cast<float4*>(o + j) = make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
                        } else {
#pragma unroll
                            for (int j = 0; j < 16; ++j)
                                if (col0 + cc + j < p.cout) o[j] = apply_act(f[j], p.act, p.slope);
                        }
                    } else {
                        store_bf16_16(reinterpret_cast<__nv_bfloat16*>(p.out) + off + cc, f, p.act, p.slope,
                                      vec_ok && col0 + cc + 16 <= p.cout, p.cout - (col0 + cc));
                    }
                    if (p.out2 != nullptr)
                        store_bf16_16(reinterpret_cast<__nv_bfloat16*>(p.out2) + off2 + cc, f, p.act2, p.slope,
                                      vec_ok && col0 + cc + 16 <= p.cout, p.cout - (col0 + cc));
                }
            }
            if (!released) release_acc();
#ifdef PAI_PROFILE_ROLES
            prof_total += clock64() - twork;
#endif
        }
        if (p.bn_part != nullptr) flush_stats();
        if (lane == 0) bulk_wait_group0();      // the output is written before the CTA exits (and dependents launch)
#ifdef PAI_PROFILE_ROLES
        if (blockIdx.x == 0 && threadIdx.x == 128)
            printf("[roles] epilogue warp 4: waiting for a full accumulator %lld cyc, working %lld cyc over %d tiles\n", prof_wait, prof_total, it);
#endif
    }
    tc_fence_before();
    if (PAIR)
        cluster_sync_all();      // neither CTA may exit (or free TMEM) while the other's MMAs / barriers still reference it
    else
        __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        if (PAIR)
            tmem_dealloc_pair(tmem_base, 2 * acc_cols);
        else
            tmem_dealloc(tmem_base, 2 * acc_cols);
    }
}

// =============================================================================================
// wgrad (stream-K, persistent): dW[tap][cu][cs] += sum over pixels of U[pix, cu] * S[pix + tap, cs]
//
// GEMM view: M = cu (mb 128-row blocks per tile), N = up to 256 columns made of `nbt` 64-channel
// blocks that may belong to different taps (so narrow layers still run N = 256 and share the U tile
// between taps), K = pixels in 64-pixel boxes.  Work unit = (tile, k-block); the units are dealt out in
// equal contiguous ranges to one CTA per SM, so every SM gets the same amount of MMA work regardless
// of the tile count; a CTA flushes its accumulators with vector reductions (red.global.add.v4.f32)
// whenever its range leaves a tile.  mb = 2 keeps two 128 x 256 fp32 accumulators (all 512 TMEM
// columns) on one B tile: 128 FLOP per byte staged from L2 instead of 85.
__global__ void __launch_bounds__(kThreads, 1)
igemm_wgrad_kernel(const __grid_constant__ CUtensorMap tm_u, const __grid_constant__ CUtensorMap tm_s,
                   const IgemmWgradParams p) {
    pdl_launch_dependents();
    extern __shared__ uint8_t smem_raw[];
    __shared__ PipeSmem ps;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int mb = p.mb, nbt = p.nbt;
    const uint32_t blk_bytes = 64 * 128;  // one [64 pixels x 64 channels] box
    const uint32_t a_bytes = 2 * mb * blk_bytes;
    const uint32_t stage_bytes = a_bytes + nbt * blk_bytes;
    const int stages = p.stages;
    const int n_cols = nbt * 64;
    const uint32_t tmem_cols = tmem_cols_for(mb * 256);

    const long long units = (long long)p.tiles * p.kblocks;
    const long long u_begin = units * blockIdx.x / gridDim.x, u_end = units * (blockIdx.x + 1) / gridDim.x;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tm_u);
        tma_prefetch_desc(&tm_s);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&ps.full[s], 1);
            mbar_init(&ps.empty[s], 1);
        }
        mbar_init(&ps.acc_full[0], 1);
        mbar_init(&ps.acc_empty[0], 4);
        mbar_fence_init();
    }
    if (warp == 2) tmem_alloc(&ps.tmem_base, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = ps.tmem_base;
    pdl_wait();

    // three TMA producer warps deal the work units round-robin (see igemm_fprop_kernel: one thread cannot issue the up
    // to 8 boxes of a stage as fast as the tensor core consumes them)
    const int pidx = warp == 0 ? 0 : (warp == 2 ? 1 : (warp == 3 ? 2 : -1));
    if (pidx >= 0) {
        if (elect_one()) {
            constexpr int P = 3;
            int stage = pidx;
            uint32_t phase = 0;
            while (stage >= stages) stage -= stages, phase ^= 1;
            for (long long u = u_begin + pidx; u < u_end; u += P) {
                const int tile = (int)(u / p.kblocks);
                int mt = (int)(u - (long long)tile * p.kblocks);
                const int ng = tile % p.n_groups, cu0 = (tile / p.n_groups) * 128 * mb;
                const int tw = mt % p.tiles_w;
                mt /= p.tiles_w;
                const int th = mt % p.tiles_h;
                const int tn = mt / p.tiles_h;
                const int w0 = tw * p.bw, h0 = th * p.bh, n0 = tn * p.bn;
                mbar_wait(&ps.empty[stage], phase ^ 1);
                uint8_t* sa = smem + (size_t)stage * stage_bytes;
                uint8_t* sb = sa + a_bytes;
                mbar_expect_tx(&ps.full[stage], stage_bytes);
                for (int i = 0; i < 2 * mb; ++i)   // rows >= cu are TMA zero fill and never stored
                    tma_load_5d(sa + i * blk_bytes, &tm_u, &ps.full[stage], cu0 + i * 64, w0, 0, h0, n0);
                for (int nb = 0; nb < nbt; ++nb) {
                    const int blk = ng * nbt + nb, tap = blk / p.cs_blocks, cb = blk - tap * p.cs_blocks;
                    tma_load_5d(sb + nb * blk_bytes, &tm_s, &ps.full[stage], p.tap_c[tap] + cb * 64, w0 + p.tap_w[tap],
                                p.tap_p[tap], h0 + p.tap_h[tap], n0);
                }
                stage += P;
                while (stage >= stages) stage -= stages, phase ^= 1;
            }
        }
    } else if (warp == 1) {
        if (elect_one()) {
            const uint32_t idesc = umma_idesc_bf16(128, n_cols, 1, 1);
            int stage = 0;
            uint32_t phase = 0;
            int seg = 0;
            long long u = u_begin;
            while (u < u_end) {
                const long long tile_end = (u / p.kblocks + 1) * p.kblocks;
                const long long seg_end = tile_end < u_end ? tile_end : u_end;
                mbar_wait(&ps.acc_empty[0], (seg & 1) ^ 1);    // epilogue drained the previous segment
                tc_fence_after();
                bool first = true;
                for (; u < seg_end; ++u) {
                    mbar_wait(&ps.full[stage], phase);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + (size_t)stage * stage_bytes);
                    const uint32_t sb = sa + a_bytes;
                    const uint64_t db0 = umma_desc_mnmajor_sw128(sb, blk_bytes);
                    for (int a = 0; a < mb; ++a) {     // 16 pixels (= 16 rows of 128 B = 128 16-byte units) per MMA
                        const uint64_t da0 = umma_desc_mnmajor_sw128(sa + a * 2 * blk_bytes, blk_bytes);
                        const uint32_t td = tmem_base + a * 256;
                        umma_bf16_ss(td, da0, db0, idesc, !first);
                        umma_bf16_acc(td, da0 + 128, db0 + 128, idesc);
                        umma_bf16_acc(td, da0 + 256, db0 + 256, idesc);
                        umma_bf16_acc(td, da0 + 384, db0 + 384, idesc);
                    }
                    first = false;
                    umma_commit(&ps.empty[stage]);
                    if (++stage == stages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                umma_commit(&ps.acc_full[0]);
                ++seg;
            }
        }
    } else if (warp >= 4) {
        const int q = warp & 3;
        const int r = q * 32 + lane;
        int seg = 0;
        long long u = u_begin;
        while (u < u_end) {
            const int tile = (int)(u / p.kblocks);
            const long long tile_end = (long long)(tile + 1) * p.kblocks;
            u = tile_end < u_end ? tile_end : u_end;
            const int ng = tile % p.n_groups, cu0 = (tile / p.n_groups) * 128 * mb;
            mbar_wait(&ps.acc_full[0], seg & 1);
            tc_fence_after();
            for (int a = 0; a < mb; ++a) {
                const int row = cu0 + a * 128 + r;
                const bool row_ok = row < p.cu;
                for (int nb = 0; nb < nbt; ++nb) {
                    const int blk = ng * nbt + nb, tap = blk / p.cs_blocks, cb = blk - tap * p.cs_blocks;
                    float* o = p.out + ((size_t)tap * p.cu + row) * (size_t)p.cs + cb * 64;
#pragma unroll
                    for (int c = 0; c < 64; c += 16) {
                        uint32_t v[16];
                        __syncwarp();
                        tmem_ld_16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * 256 + nb * 64 + c), v);
                        tmem_ld_wait();
                        if (row_ok) {
#pragma unroll
                            for (int j = 0; j < 16; j += 4)
                                red_add_v4(o + c + j, __uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                                           __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_relaxed(&ps.acc_empty[0]);   // relaxed: must not wait for the reductions above
            ++seg;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, tmem_cols);
    }
}

// =============================================================================================
// host launchers
static int pick_stages(size_t stage_bytes, size_t budget) {
    int s = (int)(budget / stage_bytes);
    if (s > kMaxStages) s = kMaxStages;
    if (s < 2) s = 2;
    return s;
}

// The 2-CTA form pays off when the layer has enough 256-pixel tiles to fill the machine; it needs a weight tile that
// splits into two UMMA-legal halves and no split-K.  PAI_NO_CTA_PAIR=1 forces the 1-CTA kernel (A/B measurements).
bool igemm_fprop_use_pair(int n_tile, long long m_tiles, int n_tiles, int phases, int splitk) {
    static const bool off = getenv("PAI_NO_CTA_PAIR") != nullptr;
    if (off || splitk > 1 || n_tile % 32 != 0) return false;
    return ((m_tiles + 1) / 2) * n_tiles * phases >= 74;
}

int launch_igemm_fprop(const CUtensorMap& tm_a, const CUtensorMap& tm_b, const IgemmOutMaps& om, IgemmFpropParams p,
                       int m_tiles, int n_tiles, int phases, cudaStream_t stream) {
    const bool pair = p.pair != 0;
    const size_t sub_bytes = 128 * 128 + (size_t)(p.fused_phases ? 4 : 1) * (pair ? p.n_tile / 2 : p.n_tile) * 128;
    if (p.kmma <= 0 || p.kmma > 4) p.kmma = 4;
    if (p.splitk < 1) p.splitk = 1;
    // two K blocks per pipeline stage when every tile (and split-K slice) has an even number of them and at least three
    // such stages fit: halves the per-stage work of the MMA-issuing thread.  PAI_IGEMM_KSUB=1 forces single blocks.
    {
        static const char* env = getenv("PAI_IGEMM_KSUB");
        const int num_kb = (p.fused_phases ? 9 : p.ntaps) * p.kc_per_tap;
        const bool even = p.fused_phases ? p.kc_per_tap % 2 == 0 : num_kb % (2 * p.splitk) == 0;
        p.ksub = (even && p.kmma == 4 && 3 * 2 * sub_bytes <= 192 * 1024 && !(env && env[0] == '1')) ? 2 : 1;
    }
    const size_t stage_bytes = sub_bytes * p.ksub;
    p.stages = pick_stages(stage_bytes, 192 * 1024);
    p.prefetch_taps = 0;
    // opt-in (PAI_L2_PREFETCH=1): measured on every layer of the batch-64 step, it changes nothing -- the loop is not
    // waiting on DRAM latency (DESIGN.md 4.1)
    if (getenv("PAI_L2_PREFETCH") != nullptr && p.splitk == 1) {
        if (p.fused_phases) {
            p.prefetch_taps = 1u;                       // the centre box
        } else {
            for (int t = 0; t < p.ntaps && t < 32; ++t) {
                bool first = true;                      // first tap of its (channel offset, parity) class
                for (int u = 0; u < t; ++u) first = first && !(p.tap_c[u] == p.tap_c[t] && p.tap_p[u] == p.tap_p[t]);
                if (first) p.prefetch_taps |= 1u << t;
            }
        }
    }
    p.m_tiles = pair ? (m_tiles + 1) / 2 : m_tiles, p.n_tiles = n_tiles, p.phases = phases;
    const size_t smem = stage_bytes * p.stages + 1024;
    static DeviceOnce once;
    const int dev = current_device(), num_sms = persistent_ctas(dev);
    if (num_sms < 0) return -1;
    if (once.need(dev)) {
        PAI_CUDA_OK(cudaFuncSetAttribute(igemm_fprop_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 194 * 1024));
        PAI_CUDA_OK(cudaFuncSetAttribute(igemm_fprop_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 194 * 1024));
        PAI_CUDA_OK(cudaFuncSetAttribute(igemm_fprop_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 194 * 1024));
        PAI_CUDA_OK(cudaFuncSetAttribute(igemm_fprop_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 194 * 1024));
        once.mark(dev);
    }
    if (p.splitk < 1) p.splitk = 1;
    PAI_REQUIRE(!pair || (p.splitk == 1 && p.n_tile % 32 == 0), "igemm fprop: the CTA-pair kernel needs n_tile %% 32 == 0 and no split-K");
    p.fd_splitk = make_fastdiv(p.splitk), p.fd_n_tiles = make_fastdiv(n_tiles), p.fd_m_tiles = make_fastdiv(p.m_tiles);
    p.fd_tiles_w = make_fastdiv(p.tiles_w), p.fd_tiles_h = make_fastdiv(p.tiles_h), p.fd_kc = make_fastdiv(p.kc_per_tap);
    const long long total = (long long)p.m_tiles * n_tiles * phases * p.splitk;
    int grid;
    if (pair) {
        const long long pairs = total < num_sms / 2 ? total : num_sms / 2;
        grid = (int)(2 * pairs);
    } else {
        grid = (int)(total < num_sms ? total : num_sms);
    }
    if (p.mask_src != nullptr)
        PAI_REQUIRE(!p.out_f32 && p.splitk == 1 && !p.accumulate && (p.n_tile & 63) == 0 && p.cout % p.n_tile == 0 &&
                        (p.cout & 7) == 0 && p.bias == nullptr && p.act == PAI_ACT_NONE && p.out2 == nullptr &&
                        (reinterpret_cast<uintptr_t>(p.mask_src) & 15) == 0 && p.tma_out,
                    "igemm fprop: the fused activation backward needs a plain bf16 output with 16 B aligned rows, "
                    "cout %% 64 == 0 and no split-K (cout=%d n_tile=%d splitk=%d)", p.cout, p.n_tile, p.splitk);
    if (p.bn_part != nullptr) {
        // the statistics ride on the coalesced bf16 epilogue: whole 64-channel chunks, one output, no split-K
        PAI_REQUIRE(!p.out_f32 && p.splitk == 1 && !p.accumulate && (p.n_tile & 63) == 0 && p.cout % p.n_tile == 0 &&
                        (p.cout & 7) == 0 && p.bn_rows >= grid,
                    "igemm fprop: fused BatchNorm statistics need a bf16 output with cout %% 64 == 0, no split-K and "
                    "%d partial rows (cout=%d n_tile=%d splitk=%d rows=%d)", grid, p.cout, p.n_tile, p.splitk, p.bn_rows);
    }
    const int cl = pair ? 2 : 1;
    const dim3 g((unsigned)grid), b(kFpropThreads);
    if (pair && p.mask_src != nullptr)
        PAI_CUDA_OK(launch_pdl(igemm_fprop_kernel<true, true>, g, b, smem, stream, cl, tm_a, tm_b, om, p));
    else if (pair)
        PAI_CUDA_OK(launch_pdl(igemm_fprop_kernel<true, false>, g, b, smem, stream, cl, tm_a, tm_b, om, p));
    else if (p.mask_src != nullptr)
        PAI_CUDA_OK(launch_pdl(igemm_fprop_kernel<false, true>, g, b, smem, stream, cl, tm_a, tm_b, om, p));
    else
        PAI_CUDA_OK(launch_pdl(igemm_fprop_kernel<false, false>, g, b, smem, stream, cl, tm_a, tm_b, om, p));
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

// split-K finish: y = act(ws + bias) over a dense fp32 workspace [pixels][cout]
__global__ void __launch_bounds__(256)
splitk_finish_kernel(const float* __restrict__ ws, long long total, int cout, const float* __restrict__ bias, int act,
                     float slope, void* __restrict__ y, int y_ld, int y_f32) {
    pdl_launch_dependents();
    pdl_wait();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long pix = i / cout;
        const int c = (int)(i - pix * cout);
        float v = ws[i];
        if (bias != nullptr) v += bias[c];
        v = apply_act(v, act, slope);
        if (y_f32)
            reinterpret_cast<float*>(y)[pix * y_ld + c] = v;
        else
            reinterpret_cast<__nv_bfloat16*>(y)[pix * y_ld + c] = __float2bfloat16_rn(v);
    }
}

int launch_splitk_finish(const float* ws, long long pixels, int cout, const float* bias, int act, float slope, void* y,
                         int y_ld, int y_f32, cudaStream_t stream) {
    const long long total = pixels * cout;
    long long blocks = (total + 255) / 256;
    const int sms = sm_count(current_device());
    if (sms < 0) return -1;
    if (blocks > sms * 8) blocks = sms * 8;
    PAI_CUDA_OK(launch_pdl(splitk_finish_kernel, dim3((unsigned)blocks), dim3(256), 0, stream, 1, ws, total, cout, bias, act, slope, y, y_ld, y_f32));
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int launch_igemm_wgrad(const CUtensorMap& tm_u, const CUtensorMap& tm_s, IgemmWgradParams p, cudaStream_t stream) {
    const size_t stage_bytes = (size_t)(2 * p.mb + p.nbt) * 8192;
    p.stages = pick_stages(stage_bytes, 196 * 1024);
    const size_t smem = stage_bytes * p.stages + 1024;
    static DeviceOnce once;
    const int dev = current_device(), num_sms = persistent_ctas(dev);
    if (num_sms < 0) return -1;
    if (once.need(dev)) {
        PAI_CUDA_OK(cudaFuncSetAttribute(igemm_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        once.mark(dev);
    }
    const long long units = (long long)p.tiles * p.kblocks;
    // at least ~4 k-blocks per CTA so the pipeline fill / accumulator flush is amortised
    long long grid = units / 4 > p.tiles ? units / 4 : p.tiles;
    if (grid > num_sms) grid = num_sms;
    if (grid < 1) grid = 1;
    if (p.max_ctas > 0 && grid > p.max_ctas) grid = p.max_ctas;
    PAI_CUDA_OK(launch_pdl(igemm_wgrad_kernel, dim3((unsigned)grid), dim3(kThreads), smem, stream, 1, tm_u, tm_s, p));
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace pai
