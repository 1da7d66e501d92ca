// Internal launcher interfaces shared by the .cu translation units (not part of the C-ABI).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pai_b200.h"

namespace pai {

// Unsigned division by a runtime constant without the ~20-instruction hardware sequence:
// q = (umulhi(n, mul) + n) >> shift, exact for n < 2^31.
struct FastDiv {
    uint32_t mul, shift, div;
#ifdef __CUDACC__
    __device__ __forceinline__ int quot(int n) const { return (int)((__umulhi((uint32_t)n, mul) + (uint32_t)n) >> shift); }
    __device__ __forceinline__ void divmod(int n, int& q, int& r) const {
        q = quot(n);
        r = n - q * (int)div;
    }
#endif
};
inline FastDiv make_fastdiv(int d) {
    FastDiv f;
    f.div = (uint32_t)d;
    uint32_t s = 0;
    while ((1u << s) < (uint32_t)d) ++s;
    f.shift = s;
    f.mul = (uint32_t)(((1ull << 32) * ((1ull << s) - (uint64_t)d)) / (uint64_t)d + 1);
    return f;
}

struct IgemmFpropParams {
    int bw, bh, bn;            // TMA box on the pixel grid, bw*bh*bn == 128
    int tiles_w, tiles_h;      // tiles along w / h (tiles along n follow from gridDim.y)
    int gw, gh, gn;            // valid pixel-grid extents (rows outside are not stored)
    int n_tile;                // output channels per CTA (multiple of 16, <= 256)
    int cout;                  // valid output channels
    int kc_per_tap, ntaps;     // 64-channel K blocks per tap, taps per phase
    int stages;
    int ksub;                  // 64-channel K blocks per pipeline stage (1 or 2), chosen by launch_igemm_fprop
    // Optional (PAI_L2_PREFETCH=1) L2 prefetch of the NEXT tile's activation boxes while this tile is loaded (bit t: tap /
    // box t is prefetched; one tap per parity class is enough, the others are shifted copies of the same lines).  An
    // experiment that ruled DRAM latency out as the limit of the narrow layers: no layer moved.  Filled by launch_igemm_fprop.
    unsigned prefetch_taps;
    int m_tiles, n_tiles, phases;  // tile grid walked by the persistent CTAs
    int tap_c[16], tap_w[16], tap_p[16], tap_h[16];  // per (phase * ntaps + tap): A-box coordinate offsets
    int b_rows_per_phase;      // rows of the packed weight matrix per phase (cout_pad)
    long long out_sn, out_sh, out_sw;  // output element strides per pixel-grid step
    long long out_phase_off[4];
    const float* bias;
    int act;
    float slope;
    int out_f32;
    void* out;
    // optional second bf16 output with its own activation and pixel strides (same grid mapping)
    void* out2;
    int act2;
    long long out2_sn, out2_sh, out2_sw;
    FastDiv fd_splitk, fd_n_tiles, fd_m_tiles, fd_tiles_w, fd_tiles_h, fd_kc;   // filled by launch_igemm_fprop
    // phase-fused transposed convolution (cout_pad == n_tile == 64): one tile owns the 4 sub-pixel phases of its
    // input pixels; the 9 distinct activation boxes (dy, dx in {-1,0,1}) of a channel block are staged once and each
    // feeds the 1, 2 or 4 (phase, tap) MMAs that read it (instead of 16 separate box loads)
    int fused_phases;
    int box_w[9], box_h[9];            // box coordinate offsets
    int box_users[9][4];               // phase * 4 + tap of every MMA fed by the box, -1 terminated, in column order
    // The accumulator of phase ph sits in TMEM column block box_col = {0, 1, 3, 2}[ph] (out_phase_off is indexed by
    // column block).  A box whose users occupy CONSECUTIVE column blocks feeds ONE MMA of N = 64 * users (box_merge):
    // an N = 64 SS-mode MMA reads 6 KB of operands for 32 clocks of tensor work -- more than shared memory delivers --
    // while N = 256 reads 12 KB for 128 clocks.  The centre box (all 4 phases) comes first, so every later MMA accumulates.
    int box_nu[9], box_col[9][4], box_merge[9];
    int kmma;                  // MMA k-steps (16 channels each) issued per 64-channel K block: 4, or fewer when only the
                               // first 16 * kmma columns of the (single) K block hold data (thin im2col operands)
    // BatchNorm statistics from the epilogue (coalesced bf16 path only): every CTA adds the per-channel sum and sum of
    // squares of the bf16-rounded outputs it stores to its own row bn_part[blockIdx.x][2 * cout] (zeroed by the caller)
    float* bn_part;
    int bn_rows;
    // activation backward folded into a data-gradient GEMM (coalesced bf16 path): out = acc * act'(mask_src) with the
    // LeakyReLU / ReLU derivative taken from the sign of the saved activation at the SAME location as the output element
    const void* mask_src;
    float mask_slope;
    int pair;                  // run as 2-CTA clusters (cta_group::2, M = 256): tm_b's box must hold n_tile / 2 rows
    int splitk;                // K slices per output tile (>1: partial sums are accumulated into fp32 `out`)
    int accumulate;            // generic fp32 path adds into `out` (red.add) instead of storing
    // the IgemmOutMaps of the launch describe `out` (and `out2` / `mask_src`): 64-channel chunks of bf16 tiles go out as
    // TMA stores.  Set by the host only where those maps exist (bf16 output, 16-byte aligned base and rows).
    int tma_out;
};

// TMA maps of the bf16 outputs of an igemm fprop launch: 4-D (C, W, H, N) views of `out` + out_phase_off[j] with the
// output's strides, extents (cout, gw, gh, gn) -- TMA clips ragged pixel tiles and channel tails -- and a box of one
// epilogue warp's 32 accumulator rows x 64 channels, SWIZZLE_128B (the layout of the warp's staging tile).
//   out[j]: column block j of a phase-fused tile, phase j otherwise (the index of out_phase_off)
//   aux[j]: the saved activations of a masked data gradient at the same positions (mask_src + out_phase_off[j]);
//           or aux[0] = `out2` with its own strides
struct IgemmOutMaps {
    CUtensorMap out[4];
    CUtensorMap aux[4];
};

struct IgemmWgradParams {
    int bw, bh, bn;            // pixel box, bw*bh*bn == 64
    int tiles_w, tiles_h, tiles_n;
    int kblocks;               // tiles_w * tiles_h * tiles_n 64-pixel K blocks
    int mb;                    // 128-row blocks of cu per tile (1 or 2)
    int nbt;                   // 64-channel B blocks per tile (N = 64 * nbt <= 256)
    int cs_blocks;             // cs / 64
    int n_groups;              // ntaps * cs_blocks / nbt
    int tiles;                 // ceil(cu / (128 * mb)) * n_groups
    int max_ctas;              // 0 = one per SM; the legacy `splitk` argument caps the CTA count (tests)
    int cu, cs;                // channel counts of the unshifted / shifted operand
    int stages;
    int tap_c[16], tap_w[16], tap_p[16], tap_h[16];
    float* out;                // [ntaps][cu][cs] fp32, accumulated with vector reductions
};

bool igemm_fprop_use_pair(int n_tile, long long m_tiles, int n_tiles, int phases, int splitk);
int launch_igemm_fprop(const CUtensorMap& tm_a, const CUtensorMap& tm_b, const IgemmOutMaps& om, IgemmFpropParams p,
                       int m_tiles, int n_tiles, int phases, cudaStream_t stream);
// y[pix * ld + c] = act(ws[pix * c_count + c] + bias[c]) for a dense fp32 split-K workspace
int launch_splitk_finish(const float* ws, long long pixels, int cout, const float* bias, int act, float slope, void* y,
                         int y_ld, int y_f32, cudaStream_t stream);
int launch_igemm_wgrad(const CUtensorMap& tm_u, const CUtensorMap& tm_s, IgemmWgradParams p, cudaStream_t stream);

}  // namespace pai
