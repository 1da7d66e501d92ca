// C-ABI entry points (include/pai_b200.h): argument validation, TMA tensor-map construction and
// tap tables for the implicit-GEMM kernels in igemm.cu.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <cudaTypedefs.h>

#include "pai_common.cuh"
#include "pai_kernels.h"

namespace pai {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
    set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
    return -1;
}

int current_device() {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) {
        cuda_fail(e, "cudaGetDevice");
        return -1;
    }
    return dev;
}

bool pdl_enabled() {
    static const bool on = getenv("PAI_PDL") != nullptr;       // opt-in: measured 0.5-1 % SLOWER on the graph-replayed step
    return on;
}

int sm_count(int dev) {
    static int cached[64] = {0};
    if (dev < 0) return -1;
    int v = __atomic_load_n(&cached[dev & 63], __ATOMIC_ACQUIRE);
    if (v > 0) return v;
    cudaError_t e = cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess || v <= 0) {
        cuda_fail(e, "cudaDeviceGetAttribute(MultiProcessorCount)");
        return -1;
    }
    __atomic_store_n(&cached[dev & 63], v, __ATOMIC_RELEASE);
    return v;
}

static int g_reserved_sms = 0;

int persistent_ctas(int dev) {
    const int sms = sm_count(dev);
    if (sms < 0) return sms;
    int n = sms - __atomic_load_n(&g_reserved_sms, __ATOMIC_RELAXED);
    if (n < 2) n = 2;
    return n & ~1;          // CTA pairs
}

static PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
    static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
    if (fn == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
    }
    return fn;
}

int encode_tmap_bf16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                     const uint64_t* strides_bytes, const uint32_t* box) {
    auto fn = get_encode();
    PAI_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled driver entry point unavailable");
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base),
                    reinterpret_cast<const cuuint64_t*>(dims), reinterpret_cast<const cuuint64_t*>(strides_bytes),
                    reinterpret_cast<const cuuint32_t*>(box), estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (%d): rank %d dims [%llu %llu %llu %llu %llu] box [%u %u %u %u %u]",
                  (int)r, rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
                  (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0),
                  (unsigned long long)(rank > 4 ? dims[4] : 0), box[0], rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0,
                  rank > 3 ? box[3] : 0, rank > 4 ? box[4] : 0);
        return -3;
    }
    return 0;
}

static int pow2_ge(int v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

struct PixBox {
    int bw, bh, bn, tiles_w, tiles_h, tiles_n;
};
// Splits `m` (128 or 64) GEMM rows over a (w, h, n) box of the pixel grid.
static PixBox pick_box(int gw, int gh, int gn, int m) {
    PixBox b;
    b.bw = pow2_ge(gw) < m ? pow2_ge(gw) : m;
    int rest = m / b.bw;
    b.bh = pow2_ge(gh) < rest ? pow2_ge(gh) : rest;
    b.bn = rest / b.bh;
    b.tiles_w = (gw + b.bw - 1) / b.bw;
    b.tiles_h = (gh + b.bh - 1) / b.bh;
    b.tiles_n = (gn + b.bn - 1) / b.bn;
    return b;
}

// 5-D views of an NHWC bf16 tensor: (C', W', P, H', N).
static int map_unit(CUtensorMap* m, const void* base, int n, int h, int w, int c, int ld, const PixBox& b) {
    uint64_t dims[5] = {(uint64_t)c, (uint64_t)w, 1, (uint64_t)h, (uint64_t)n};
    uint64_t str[4] = {(uint64_t)ld * 2, (uint64_t)w * ld * 2, (uint64_t)w * ld * 2, (uint64_t)h * w * ld * 2};
    uint32_t box[5] = {64, (uint32_t)b.bw, 1, (uint32_t)b.bh, (uint32_t)b.bn};
    return encode_tmap_bf16(m, base, 5, dims, str, box);
}
// parity-split view for "input = 2*o - 1 + k" access: column 2*wq+px -> (c + px*C, wq), row 2*hq+py -> (py, hq)
static int map_split(CUtensorMap* m, const void* base, int n, int h, int w, int c, const PixBox& b) {
    uint64_t dims[5] = {(uint64_t)2 * c, (uint64_t)w / 2, 2, (uint64_t)h / 2, (uint64_t)n};
    uint64_t str[4] = {(uint64_t)2 * c * 2, (uint64_t)w * c * 2, (uint64_t)2 * w * c * 2, (uint64_t)h * w * c * 2};
    uint32_t box[5] = {64, (uint32_t)b.bw, 1, (uint32_t)b.bh, (uint32_t)b.bn};
    return encode_tmap_bf16(m, base, 5, dims, str, box);
}
// k in 0..3 of a stride-2, pad-1 access -> (quotient offset, parity)
static void s2_tap(int k, int* q, int* par) {
    static const int Q[4] = {-1, 0, 0, 1}, P[4] = {1, 0, 1, 0};
    *q = Q[k];
    *par = P[k];
}
// ConvTranspose2d(4,2,1) sub-pixel phases: T[parity][t] = (k, d)
static const int kTd[2][2] = {{0, -1}, {1, 0}};

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// 4-D (C, W, H, N) view of a bf16 tensor on the output pixel grid of an igemm fprop launch (element strides sw, sh, sn),
// box = the 32 accumulator rows of one epilogue warp x 64 channels.  The 128 rows of a tile run w-fastest over the
// power-of-two bw x bh x bn pixel box, so a warp's 32 rows are always the box {64, min(bw, 32), ...}.
static int map_out(CUtensorMap* m, const void* base, int cout, int gw, int gh, int gn, long long sw, long long sh,
                   long long sn, const PixBox& b) {
    const int bw = b.bw < 32 ? b.bw : 32, bh = b.bh < 32 / bw ? b.bh : 32 / bw, bn = 32 / (bw * bh);
    // a size-1 H dimension may have stride 0 (pointwise rows); TMA wants a non-zero multiple of 16 bytes
    if (sh == 0) sh = (long long)gw * sw;
    uint64_t dims[4] = {(uint64_t)cout, (uint64_t)gw, (uint64_t)gh, (uint64_t)gn};
    uint64_t str[3] = {(uint64_t)sw * 2, (uint64_t)sh * 2, (uint64_t)sn * 2};
    uint32_t box[4] = {64, (uint32_t)bw, (uint32_t)bh, (uint32_t)bn};
    return encode_tmap_bf16(m, base, 4, dims, str, box);
}

// Output maps of a launch (IgemmOutMaps) for `nmaps` phases / column blocks of p.out, from the strides and phase offsets
// already in `p` (and maps of p.out2 or p.mask_src).  Without 16-byte aligned bf16 rows there are none and every tile
// takes the generic epilogue (p.tma_out stays 0).
static int map_outputs(IgemmOutMaps* om, IgemmFpropParams& p, int nmaps, const PixBox& b) {
    p.tma_out = 0;
    const bool ok = !p.out_f32 && !p.accumulate && (p.cout & 7) == 0 && aligned16(p.out) && p.out_sw % 8 == 0 &&
                    p.out_sh % 8 == 0 && p.out_sn % 8 == 0 &&
                    (p.out2 == nullptr || (aligned16(p.out2) && p.out2_sw % 8 == 0 && p.out2_sh % 8 == 0 && p.out2_sn % 8 == 0));
    if (!ok) return 0;
    for (int j = 0; j < nmaps; ++j) {
        PAI_REQUIRE(p.out_phase_off[j] % 8 == 0, "igemm fprop: phase offset %lld is not 16 B aligned", p.out_phase_off[j]);
        int rc = map_out(&om->out[j], static_cast<const __nv_bfloat16*>(p.out) + p.out_phase_off[j], p.cout, p.gw, p.gh,
                         p.gn, p.out_sw, p.out_sh, p.out_sn, b);
        if (rc) return rc;
        if (p.mask_src != nullptr) {
            rc = map_out(&om->aux[j], static_cast<const __nv_bfloat16*>(p.mask_src) + p.out_phase_off[j], p.cout, p.gw,
                         p.gh, p.gn, p.out_sw, p.out_sh, p.out_sn, b);
            if (rc) return rc;
        }
    }
    if (p.out2 != nullptr) {
        int rc = map_out(&om->aux[0], p.out2, p.cout, p.gw, p.gh, p.gn, p.out2_sw, p.out2_sh, p.out2_sn, b);
        if (rc) return rc;
    }
    p.tma_out = 1;
    return 0;
}

// Output-channel tile: the widest of 256/128/64/32/16 that divides cout_pad while still giving every
// SM a tile (wider tiles re-read the activations less often from L2).
static int auto_n_tile(int cout_pad, long long m_tiles_x_phases) {
    static const int cand[5] = {256, 128, 64, 32, 16};
    int best = 0;
    for (int i = 0; i < 5; ++i) {
        if (cout_pad % cand[i]) continue;
        if (best == 0) best = cand[i];
        if (m_tiles_x_phases * (cout_pad / cand[i]) >= 148) return cand[i];
        best = cand[i] >= 128 ? cand[i] : best;      // small problems: do not go below 128 just to add CTAs
        if (cand[i] <= 128) break;
    }
    return best;
}

// Split-K factor for layers too small to give every SM an output tile (the <= 8x8 levels of the U-Net):
// the K loop (taps x channel blocks) is cut into slices that run on different SMs and meet in an fp32
// workspace.  Returns 1 when the layer has enough tiles or no workspace was supplied.
static int pick_splitk(const void* ws, long long tiles, int num_kb) {
    if (ws == nullptr || tiles > 74 || num_kb < 8) return 1;
    long long s = 148 / tiles;
    if (s > num_kb / 2) s = num_kb / 2;
    return s < 2 ? 1 : (int)s;
}

}  // namespace pai

using namespace pai;

extern "C" {

const char* pai_last_error(void) { return g_err; }
int pai_version(void) { return 100; }

int pai_reserve_sms(int n) {
    PAI_REQUIRE(n >= 0 && n <= 64, "pai_reserve_sms: reservation must be in 0..64 (got %d)", n);
    __atomic_store_n(&g_reserved_sms, n, __ATOMIC_RELAXED);
    return 0;
}

static int conv4x4_fprop_impl(const void* x, int n, int h, int w, int cin, int x_ld, const void* w_packed, int cout,
                              int cout_pad, int stride, const float* bias, int act, float slope, void* y, int y_ld,
                              int y_f32, int n_tile, float* splitk_ws, float* bn_part, int bn_rows, void* stream,
                              void* y2 = nullptr, int y2_ld = 0, int act2 = PAI_ACT_NONE) {
    PAI_REQUIRE(x && w_packed && y, "pai_conv4x4_fprop: null pointer");
    PAI_REQUIRE(stride == 1 || stride == 2, "pai_conv4x4_fprop: stride must be 1 or 2 (got %d)", stride);
    PAI_REQUIRE(cin > 0 && cin % 64 == 0, "pai_conv4x4_fprop: cin must be a multiple of 64 (got %d)", cin);
    PAI_REQUIRE(cout_pad % 16 == 0 && cout <= cout_pad, "pai_conv4x4_fprop: bad cout %d / cout_pad %d", cout, cout_pad);
    PAI_REQUIRE(aligned16(x) && aligned16(w_packed) && x_ld % 8 == 0, "pai_conv4x4_fprop: x / w must be 16 B aligned");
    int ho, wo;
    if (stride == 2) {
        PAI_REQUIRE(h % 2 == 0 && w % 2 == 0 && x_ld == cin, "pai_conv4x4_fprop: stride 2 needs even h,w and dense x");
        ho = h / 2;
        wo = w / 2;
    } else {
        PAI_REQUIRE(h >= 2 && w >= 2, "pai_conv4x4_fprop: stride 1 needs h,w >= 2");
        ho = h - 1;
        wo = w - 1;
    }
    PixBox b = pick_box(wo, ho, n, 128);
    if (n_tile <= 0) n_tile = auto_n_tile(cout_pad, (long long)b.tiles_w * b.tiles_h * b.tiles_n);
    PAI_REQUIRE(n_tile >= 16 && n_tile <= 256 && n_tile % 16 == 0 && cout_pad % n_tile == 0,
                "pai_conv4x4_fprop: bad n_tile %d for cout_pad %d", n_tile, cout_pad);
    CUtensorMap tm_a, tm_b;
    int rc = stride == 2 ? map_split(&tm_a, x, n, h, w, cin, b) : map_unit(&tm_a, x, n, h, w, cin, x_ld, b);
    if (rc) return rc;
    const int m_tiles = b.tiles_w * b.tiles_h * b.tiles_n;
    const int splitk = pick_splitk(splitk_ws, (long long)m_tiles * (cout_pad / n_tile), 16 * (cin / 64));
    const bool pair = igemm_fprop_use_pair(n_tile, m_tiles, cout_pad / n_tile, 1, splitk);
    uint64_t bd[2] = {(uint64_t)16 * cin, (uint64_t)cout_pad};
    uint64_t bs[1] = {(uint64_t)16 * cin * 2};
    uint32_t bb[2] = {64, (uint32_t)(pair ? n_tile / 2 : n_tile)};
    rc = encode_tmap_bf16(&tm_b, w_packed, 2, bd, bs, bb);
    if (rc) return rc;

    IgemmFpropParams p;
    memset(&p, 0, sizeof(p));
    IgemmOutMaps om;
    memset(&om, 0, sizeof(om));
    p.pair = pair;
    p.bw = b.bw, p.bh = b.bh, p.bn = b.bn, p.tiles_w = b.tiles_w, p.tiles_h = b.tiles_h;
    p.gw = wo, p.gh = ho, p.gn = n;
    p.n_tile = n_tile, p.cout = cout, p.kc_per_tap = cin / 64, p.ntaps = 16;
    for (int ky = 0; ky < 4; ++ky)
        for (int kx = 0; kx < 4; ++kx) {
            int t = ky * 4 + kx;
            if (stride == 2) {
                int qx, px, qy, py;
                s2_tap(kx, &qx, &px);
                s2_tap(ky, &qy, &py);
                p.tap_c[t] = px * cin, p.tap_w[t] = qx, p.tap_p[t] = py, p.tap_h[t] = qy;
            } else {
                p.tap_c[t] = 0, p.tap_w[t] = kx - 1, p.tap_p[t] = 0, p.tap_h[t] = ky - 1;
            }
        }
    p.b_rows_per_phase = cout_pad;
    p.bn_part = bn_part, p.bn_rows = bn_rows;
    p.splitk = splitk;
    if (p.splitk > 1) {
        p.out_sn = (long long)ho * wo * cout, p.out_sh = (long long)wo * cout, p.out_sw = cout;
        p.out_f32 = 1, p.accumulate = 1, p.out = splitk_ws;
        int rc2 = launch_igemm_fprop(tm_a, tm_b, om, p, m_tiles, cout_pad / n_tile, 1, (cudaStream_t)stream);
        if (rc2) return rc2;
        return launch_splitk_finish(splitk_ws, (long long)n * ho * wo, cout, bias, act, slope, y, y_ld, y_f32,
                                    (cudaStream_t)stream);
    }
    p.out_sn = (long long)ho * wo * y_ld, p.out_sh = (long long)wo * y_ld, p.out_sw = y_ld;
    p.bias = bias, p.act = act, p.slope = slope, p.out_f32 = y_f32, p.out = y;
    if (y2 != nullptr) {
        PAI_REQUIRE(!y_f32 && y2_ld % 8 == 0 && aligned16(y2) && aligned16(y) && y_ld % 8 == 0 && cout % 64 == 0,
                    "pai_conv4x4_fprop_dual: two bf16 outputs need cout %% 64 == 0 and 16 B aligned rows");
        p.out2 = y2, p.act2 = act2;
        p.out2_sn = (long long)ho * wo * y2_ld, p.out2_sh = (long long)wo * y2_ld, p.out2_sw = y2_ld;
    }
    rc = map_outputs(&om, p, 1, b);
    if (rc) return rc;
    return launch_igemm_fprop(tm_a, tm_b, om, p, m_tiles, cout_pad / n_tile, 1, (cudaStream_t)stream);
}

int pai_conv4x4_fprop_dual(const void* x, int n, int h, int w, int cin, int x_ld, const void* w_packed, int cout,
                           int cout_pad, int stride, const float* bias, int act, float slope, void* y, int y_ld, void* y2,
                           int y2_ld, int act2, int n_tile, void* stream) {
    PAI_REQUIRE(y2 != nullptr, "pai_conv4x4_fprop_dual: null second output");
    return conv4x4_fprop_impl(x, n, h, w, cin, x_ld, w_packed, cout, cout_pad, stride, bias, act, slope, y, y_ld, 0, n_tile,
                              nullptr, nullptr, 0, stream, y2, y2_ld, act2);
}

int pai_conv4x4_fprop(const void* x, int n, int h, int w, int cin, int x_ld, const void* w_packed, int cout,
                      int cout_pad, int stride, const float* bias, int act, float slope, void* y, int y_ld,
                      int y_f32, int n_tile, float* splitk_ws, void* stream) {
    return conv4x4_fprop_impl(x, n, h, w, cin, x_ld, w_packed, cout, cout_pad, stride, bias, act, slope, y, y_ld, y_f32,
                              n_tile, splitk_ws, nullptr, 0, stream);
}
int pai_conv4x4_fprop_bnstats(const void* x, int n, int h, int w, int cin, int x_ld, const void* w_packed, int cout,
                              int cout_pad, int stride, const float* bias, void* y, int y_ld, int n_tile,
                              float* bn_partials, int bn_rows, void* stream) {
    PAI_REQUIRE(bn_partials != nullptr && bn_rows > 0, "pai_conv4x4_fprop_bnstats: null partial-sum buffer");
    return conv4x4_fprop_impl(x, n, h, w, cin, x_ld, w_packed, cout, cout_pad, stride, bias, PAI_ACT_NONE, 0.f, y, y_ld, 0,
                              n_tile, nullptr, bn_partials, bn_rows, stream);
}

static int convT4x4s2_fprop_impl(const void* x, int n, int h, int w, int cin, int x_ld, const void* w_packed, int cout,
                                 int cout_pad, const float* bias, int act, float slope, void* y, int y_ld, int y_f32,
                                 int n_tile, float* splitk_ws, float* bn_part, int bn_rows, void* stream,
                                 const void* mask_src = nullptr, float mask_slope = 0.f) {
    PAI_REQUIRE(x && w_packed && y, "pai_convT4x4s2_fprop: null pointer");
    PAI_REQUIRE(cin > 0 && cin % 64 == 0, "pai_convT4x4s2_fprop: cin must be a multiple of 64 (got %d)", cin);
    PAI_REQUIRE(cout_pad % 16 == 0 && cout <= cout_pad, "pai_convT4x4s2_fprop: bad cout %d / cout_pad %d", cout, cout_pad);
    PAI_REQUIRE(aligned16(x) && aligned16(w_packed) && x_ld % 8 == 0 && x_ld >= cin,
                "pai_convT4x4s2_fprop: x / w must be 16 B aligned");
    PixBox b = pick_box(w, h, n, 128);
    if (n_tile <= 0) n_tile = auto_n_tile(cout_pad, 4LL * b.tiles_w * b.tiles_h * b.tiles_n);
    PAI_REQUIRE(n_tile >= 16 && n_tile <= 256 && n_tile % 16 == 0 && cout_pad % n_tile == 0,
                "pai_convT4x4s2_fprop: bad n_tile %d for cout_pad %d", n_tile, cout_pad);
    CUtensorMap tm_a, tm_b;
    int rc = map_unit(&tm_a, x, n, h, w, cin, x_ld, b);
    if (rc) return rc;
    const int m_tiles = b.tiles_w * b.tiles_h * b.tiles_n;
    const int splitk = pick_splitk(splitk_ws, 4LL * m_tiles * (cout_pad / n_tile), 4 * (cin / 64));
    // phase fusion for the 64-channel layers (dec6, the data gradients of enc1 / D1): the activation tile is the
    // L2-bound operand there, and 9 boxes per channel block instead of 16 feed all four phases
    const bool fuse = splitk == 1 && cout == 64 && cout_pad == 64 && n_tile == 64 && !y_f32 && y_ld % 8 == 0 &&
                      aligned16(y) && (bias == nullptr || aligned16(bias)) && getenv("PAI_NO_PHASE_FUSION") == nullptr;
    const bool pair = fuse ? igemm_fprop_use_pair(n_tile, m_tiles, 1, 1, 1)
                           : igemm_fprop_use_pair(n_tile, m_tiles, cout_pad / n_tile, 4, splitk);
    uint64_t bd[2] = {(uint64_t)4 * cin, (uint64_t)4 * cout_pad};
    uint64_t bs[1] = {(uint64_t)4 * cin * 2};
    uint32_t bb[2] = {64, (uint32_t)(pair ? n_tile / 2 : n_tile)};
    rc = encode_tmap_bf16(&tm_b, w_packed, 2, bd, bs, bb);
    if (rc) return rc;

    IgemmFpropParams p;
    memset(&p, 0, sizeof(p));
    IgemmOutMaps om;
    memset(&om, 0, sizeof(om));
    p.pair = pair;
    p.bw = b.bw, p.bh = b.bh, p.bn = b.bn, p.tiles_w = b.tiles_w, p.tiles_h = b.tiles_h;
    p.gw = w, p.gh = h, p.gn = n;
    p.n_tile = n_tile, p.cout = cout, p.kc_per_tap = cin / 64, p.ntaps = 4;
    for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px)
            for (int ty = 0; ty < 2; ++ty)
                for (int tx = 0; tx < 2; ++tx) {
                    int i = (py * 2 + px) * 4 + ty * 2 + tx;
                    p.tap_c[i] = 0, p.tap_w[i] = kTd[px][tx], p.tap_p[i] = 0, p.tap_h[i] = kTd[py][ty];
                }
    p.b_rows_per_phase = cout_pad;
    p.bn_part = bn_part, p.bn_rows = bn_rows;
    p.mask_src = mask_src, p.mask_slope = mask_slope;
    const long long wo = 2LL * w;
    p.splitk = splitk;
    const long long ld = p.splitk > 1 ? cout : y_ld;
    p.out_sn = 4LL * h * w * ld, p.out_sh = 2 * wo * ld, p.out_sw = 2LL * ld;
    for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px) p.out_phase_off[py * 2 + px] = (py * wo + px) * ld;
    if (fuse) {
        p.fused_phases = 1;
        static const int col_of_phase[4] = {0, 1, 3, 2};      // 3 of the 4 two-phase boxes get adjacent column blocks
        static const int box_order[9] = {4, 0, 1, 2, 3, 5, 6, 7, 8};   // centre (dy = dx = 0) first
        const bool merge_ok = getenv("PAI_NO_PHASE_MERGE") == nullptr;
        for (int bi = 0; bi < 9; ++bi) {
            const int bx = box_order[bi];
            const int dy = bx / 3 - 1, dx = bx % 3 - 1;
            p.box_h[bi] = dy, p.box_w[bi] = dx;
            int nu = 0;
            for (int col = 0; col < 4; ++col)            // users in column order
                for (int ph = 0; ph < 4; ++ph) {
                    if (col_of_phase[ph] != col) continue;
                    const int py = ph >> 1, px = ph & 1;
                    for (int ty = 0; ty < 2; ++ty)
                        for (int tx = 0; tx < 2; ++tx)
                            if (kTd[py][ty] == dy && kTd[px][tx] == dx) {
                                p.box_users[bi][nu] = ph * 4 + ty * 2 + tx;
                                p.box_col[bi][nu] = col;
                                ++nu;
                            }
                }
            p.box_nu[bi] = nu;
            bool consecutive = nu > 1;
            for (int u = 1; u < nu; ++u) consecutive = consecutive && p.box_col[bi][u] == p.box_col[bi][u - 1] + 1;
            p.box_merge[bi] = merge_ok && consecutive;
            for (; nu < 4; ++nu) p.box_users[bi][nu] = -1, p.box_col[bi][nu] = 0;
        }
        for (int py = 0; py < 2; ++py)
            for (int px = 0; px < 2; ++px) p.out_phase_off[col_of_phase[py * 2 + px]] = (py * wo + px) * ld;
        p.bias = bias, p.act = act, p.slope = slope, p.out_f32 = 0, p.out = y;
        rc = map_outputs(&om, p, 4, b);
        if (rc) return rc;
        return launch_igemm_fprop(tm_a, tm_b, om, p, m_tiles, 1, 1, (cudaStream_t)stream);
    }
    if (p.splitk > 1) {
        p.out_f32 = 1, p.accumulate = 1, p.out = splitk_ws;
        int rc2 = launch_igemm_fprop(tm_a, tm_b, om, p, m_tiles, cout_pad / n_tile, 4, (cudaStream_t)stream);
        if (rc2) return rc2;
        return launch_splitk_finish(splitk_ws, 4LL * n * h * w, cout, bias, act, slope, y, y_ld, y_f32,
                                    (cudaStream_t)stream);
    }
    p.bias = bias, p.act = act, p.slope = slope, p.out_f32 = y_f32, p.out = y;
    rc = map_outputs(&om, p, 4, b);
    if (rc) return rc;
    return launch_igemm_fprop(tm_a, tm_b, om, p, m_tiles, cout_pad / n_tile, 4, (cudaStream_t)stream);
}

int pai_convT4x4s2_fprop(const void* x, int n, int h, int w, int cin, int x_ld, const void* w_packed, int cout,
                         int cout_pad, const float* bias, int act, float slope, void* y, int y_ld, int y_f32,
                         int n_tile, float* splitk_ws, void* stream) {
    return convT4x4s2_fprop_impl(x, n, h, w, cin, x_ld, w_packed, cout, cout_pad, bias, act, slope, y, y_ld, y_f32, n_tile,
                                 splitk_ws, nullptr, 0, stream);
}
int pai_convT4x4s2_fprop_bnstats(const void* x, int n, int h, int w, int cin, int x_ld, const void* w_packed, int cout,
                                 int cout_pad, const float* bias, void* y, int y_ld, int n_tile, float* bn_partials,
                                 int bn_rows, void* stream) {
    PAI_REQUIRE(bn_partials != nullptr && bn_rows > 0, "pai_convT4x4s2_fprop_bnstats: null partial-sum buffer");
    return convT4x4s2_fprop_impl(x, n, h, w, cin, x_ld, w_packed, cout, cout_pad, bias, PAI_ACT_NONE, 0.f, y, y_ld, 0,
                                 n_tile, nullptr, bn_partials, bn_rows, stream);
}

int pai_conv4x4_dgrad_act(const void* gy, int n, int h, int w, int cout, int gy_ld, const void* w_packed_dgrad, int cin,
                          int cin_pad, const void* saved_act, float slope, void* gx, int gx_ld, int n_tile,
                          float* colsum_partials, int rows, void* stream) {
    PAI_REQUIRE(saved_act != nullptr, "pai_conv4x4_dgrad_act: null saved activation");
    PAI_REQUIRE(colsum_partials == nullptr || rows > 0, "pai_conv4x4_dgrad_act: bad partial-sum buffer");
    return convT4x4s2_fprop_impl(gy, n, h, w, cout, gy_ld, w_packed_dgrad, cin, cin_pad, nullptr, PAI_ACT_NONE, 0.f, gx,
                                 gx_ld, 0, n_tile, nullptr, colsum_partials, rows, stream, saved_act, slope);
}

// stride: 2 = parity-split taps, 1 = unit-stride 4x4 taps, 0 = pointwise (a single tap at offset 0)
static int wgrad_common(const void* u, int un, int uh, int uw, int cu, int u_ld, const void* s, int sh, int sw,
                        int cs, int s_ld, int stride, float* dw, int splitk, cudaStream_t stream, const char* who) {
    PAI_REQUIRE(u && s && dw, "%s: null pointer", who);
    PAI_REQUIRE(cu % 64 == 0 && cs % 64 == 0, "%s: channel counts (%d rows, %d cols) must be multiples of 64", who, cu,
                cs);
    PAI_REQUIRE(aligned16(u) && aligned16(s) && u_ld % 8 == 0 && s_ld % 8 == 0, "%s: operands must be 16 B aligned",
                who);
    PixBox b = pick_box(uw, uh, un, 64);
    CUtensorMap tm_u, tm_s;
    int rc = map_unit(&tm_u, u, un, uh, uw, cu, u_ld, b);
    if (rc) return rc;
    if (stride == 2) {
        PAI_REQUIRE(s_ld == cs && sh % 2 == 0 && sw % 2 == 0, "%s: the stride-2 operand must be dense with even h,w",
                    who);
        rc = map_split(&tm_s, s, un, sh, sw, cs, b);
    } else {
        rc = map_unit(&tm_s, s, un, sh, sw, cs, s_ld, b);
    }
    if (rc) return rc;
    IgemmWgradParams p;
    memset(&p, 0, sizeof(p));
    p.bw = b.bw, p.bh = b.bh, p.bn = b.bn, p.tiles_w = b.tiles_w, p.tiles_h = b.tiles_h, p.tiles_n = b.tiles_n;
    p.cu = cu, p.cs = cs, p.out = dw;
    for (int ky = 0; ky < 4; ++ky)
        for (int kx = 0; kx < 4; ++kx) {
            int t = ky * 4 + kx;
            if (stride == 2) {
                int qx, px, qy, py;
                s2_tap(kx, &qx, &px);
                s2_tap(ky, &qy, &py);
                p.tap_c[t] = px * cs, p.tap_w[t] = qx, p.tap_p[t] = py, p.tap_h[t] = qy;
            } else if (stride == 1) {
                p.tap_c[t] = 0, p.tap_w[t] = kx - 1, p.tap_p[t] = 0, p.tap_h[t] = ky - 1;
            }   // stride 0: the single tap stays at offset 0
        }
    if (stride == 3)   // 3x3, stride 1, padding 1
        for (int t = 0; t < 9; ++t) p.tap_c[t] = 0, p.tap_w[t] = t % 3 - 1, p.tap_p[t] = 0, p.tap_h[t] = t / 3 - 1;
    const int ntaps = stride == 0 ? 1 : (stride == 3 ? 9 : 16);
    p.kblocks = b.tiles_w * b.tiles_h * b.tiles_n;
    p.cs_blocks = cs / 64;
    const int nb_total = ntaps * p.cs_blocks;
    p.nbt = nb_total % 4 == 0 ? 4 : (nb_total % 2 == 0 ? 2 : 1);
    p.n_groups = nb_total / p.nbt;
    p.mb = cu > 128 ? 2 : 1;
    p.tiles = ((cu + 128 * p.mb - 1) / (128 * p.mb)) * p.n_groups;
    p.max_ctas = splitk > 0 ? splitk * p.tiles : 0;
    return launch_igemm_wgrad(tm_u, tm_s, p, stream);
}

int pai_conv4x4_wgrad(const void* x, int n, int h, int w, int cin, int x_ld, const void* gy, int cout, int gy_ld,
                      int stride, float* dw, int splitk, void* stream) {
    PAI_REQUIRE(stride == 1 || stride == 2, "pai_conv4x4_wgrad: stride must be 1 or 2");
    const int ho = stride == 2 ? h / 2 : h - 1, wo = stride == 2 ? w / 2 : w - 1;
    return wgrad_common(gy, n, ho, wo, cout, gy_ld, x, h, w, cin, x_ld, stride, dw, splitk, (cudaStream_t)stream,
                        "pai_conv4x4_wgrad");
}

int pai_pointwise_wgrad(const void* u, long long m, int cu, int u_ld, const void* s, int cs, int s_ld, float* dw,
                        int splitk, void* stream) {
    PAI_REQUIRE(m > 0 && m < (1LL << 31), "pai_pointwise_wgrad: bad row count");
    // rows are independent: one [1, 1, m] pixel row cut into 64-pixel boxes (a ragged tail is TMA zero fill)
    return wgrad_common(u, 1, 1, (int)m, cu, u_ld, s, 1, (int)m, cs, s_ld, 0, dw, splitk, (cudaStream_t)stream,
                        "pai_pointwise_wgrad");
}

int pai_pointwise_gemm(const void* x, long long m, int cin, int x_ld, const void* w_packed, int cout, int cout_pad,
                       const float* bias, int act, float slope, void* y, int y_ld, int y_f32, void* y2, int y2_ld,
                       int act2, int n_tile, int k_valid, void* stream) {
    PAI_REQUIRE(x && w_packed && y, "pai_pointwise_gemm: null pointer");
    PAI_REQUIRE(k_valid == 0 || (cin == 64 && k_valid > 0 && k_valid <= 64 && k_valid % 16 == 0),
                "pai_pointwise_gemm: k_valid (%d) needs cin == 64 and a multiple of 16", k_valid);
    PAI_REQUIRE(cin > 0 && cin % 64 == 0, "pai_pointwise_gemm: cin must be a multiple of 64 (got %d)", cin);
    PAI_REQUIRE(cout_pad % 16 == 0 && cout <= cout_pad, "pai_pointwise_gemm: bad cout %d / cout_pad %d", cout, cout_pad);
    PAI_REQUIRE(aligned16(x) && aligned16(w_packed) && x_ld % 8 == 0 && x_ld >= cin, "pai_pointwise_gemm: alignment");
    PAI_REQUIRE(m > 0 && m < (1LL << 31), "pai_pointwise_gemm: bad row count %lld", m);
    // one [1, 1, m] pixel row cut into 128-row tiles; a ragged last tile is TMA zero fill and is not stored
    const int wbox = (int)m, n = 1;
    PixBox b = pick_box(wbox, 1, n, 128);
    if (n_tile <= 0) n_tile = auto_n_tile(cout_pad, (long long)b.tiles_w * b.tiles_h * b.tiles_n);
    PAI_REQUIRE(n_tile >= 16 && n_tile <= 256 && n_tile % 16 == 0 && cout_pad % n_tile == 0,
                "pai_pointwise_gemm: bad n_tile %d for cout_pad %d", n_tile, cout_pad);
    CUtensorMap tm_a, tm_b;
    int rc = map_unit(&tm_a, x, n, 1, wbox, cin, x_ld, b);
    if (rc) return rc;
    uint64_t bd[2] = {(uint64_t)cin, (uint64_t)cout_pad};
    uint64_t bs[1] = {(uint64_t)cin * 2};
    uint32_t bb[2] = {64, (uint32_t)n_tile};
    rc = encode_tmap_bf16(&tm_b, w_packed, 2, bd, bs, bb);
    if (rc) return rc;
    IgemmFpropParams p;
    memset(&p, 0, sizeof(p));
    IgemmOutMaps om;
    memset(&om, 0, sizeof(om));
    p.bw = b.bw, p.bh = b.bh, p.bn = b.bn, p.tiles_w = b.tiles_w, p.tiles_h = b.tiles_h;
    p.gw = wbox, p.gh = 1, p.gn = n;
    p.n_tile = n_tile, p.cout = cout, p.kc_per_tap = cin / 64, p.ntaps = 1;
    p.b_rows_per_phase = cout_pad;
    p.out_sn = (long long)wbox * y_ld, p.out_sh = 0, p.out_sw = y_ld;
    p.out2_sn = (long long)wbox * y2_ld, p.out2_sh = 0, p.out2_sw = y2_ld;
    p.bias = bias, p.act = act, p.slope = slope, p.out_f32 = y_f32, p.out = y, p.out2 = y2, p.act2 = act2;
    p.kmma = k_valid > 0 ? k_valid / 16 : 4;
    rc = map_outputs(&om, p, 1, b);
    if (rc) return rc;
    return launch_igemm_fprop(tm_a, tm_b, om, p, b.tiles_w * b.tiles_h * b.tiles_n, cout_pad / n_tile, 1,
                              (cudaStream_t)stream);
}

int pai_convT4x4s2_wgrad(const void* x, int n, int h, int w, int cin, int x_ld, const void* gy, int cout, int gy_ld,
                         float* dw, int splitk, void* stream) {
    return wgrad_common(x, n, h, w, cin, x_ld, gy, 2 * h, 2 * w, cout, gy_ld, 2, dw, splitk, (cudaStream_t)stream,
                        "pai_convT4x4s2_wgrad");
}

int pai_conv3x3_fprop(const void* x, int n, int h, int w, int cin, int x_ld, const void* w_packed, int cout,
                      int cout_pad, const float* bias, int act, float slope, void* y, int y_ld, int y_f32, int n_tile,
                      float* splitk_ws, void* stream) {
    PAI_REQUIRE(x && w_packed && y, "pai_conv3x3_fprop: null pointer");
    PAI_REQUIRE(cin > 0 && cin % 64 == 0, "pai_conv3x3_fprop: cin must be a multiple of 64 (got %d)", cin);
    PAI_REQUIRE(cout_pad % 16 == 0 && cout <= cout_pad, "pai_conv3x3_fprop: bad cout %d / cout_pad %d", cout, cout_pad);
    PAI_REQUIRE(aligned16(x) && aligned16(w_packed) && x_ld % 8 == 0 && x_ld >= cin, "pai_conv3x3_fprop: alignment");
    PixBox b = pick_box(w, h, n, 128);
    if (n_tile <= 0) n_tile = auto_n_tile(cout_pad, (long long)b.tiles_w * b.tiles_h * b.tiles_n);
    PAI_REQUIRE(n_tile >= 16 && n_tile <= 256 && n_tile % 16 == 0 && cout_pad % n_tile == 0,
                "pai_conv3x3_fprop: bad n_tile %d for cout_pad %d", n_tile, cout_pad);
    CUtensorMap tm_a, tm_b;
    int rc = map_unit(&tm_a, x, n, h, w, cin, x_ld, b);
    if (rc) return rc;
    uint64_t bd[2] = {(uint64_t)9 * cin, (uint64_t)cout_pad};
    uint64_t bs[1] = {(uint64_t)9 * cin * 2};
    uint32_t bb[2] = {64, (uint32_t)n_tile};
    rc = encode_tmap_bf16(&tm_b, w_packed, 2, bd, bs, bb);
    if (rc) return rc;
    IgemmFpropParams p;
    memset(&p, 0, sizeof(p));
    IgemmOutMaps om;
    memset(&om, 0, sizeof(om));
    p.bw = b.bw, p.bh = b.bh, p.bn = b.bn, p.tiles_w = b.tiles_w, p.tiles_h = b.tiles_h;
    p.gw = w, p.gh = h, p.gn = n;
    p.n_tile = n_tile, p.cout = cout, p.kc_per_tap = cin / 64, p.ntaps = 9;
    for (int t = 0; t < 9; ++t) p.tap_c[t] = 0, p.tap_w[t] = t % 3 - 1, p.tap_p[t] = 0, p.tap_h[t] = t / 3 - 1;
    p.b_rows_per_phase = cout_pad;
    const int m_tiles = b.tiles_w * b.tiles_h * b.tiles_n;
    p.splitk = pick_splitk(splitk_ws, (long long)m_tiles * (cout_pad / n_tile), 9 * (cin / 64));
    if (p.splitk > 1) {
        p.out_sn = (long long)h * w * cout, p.out_sh = (long long)w * cout, p.out_sw = cout;
        p.out_f32 = 1, p.accumulate = 1, p.out = splitk_ws;
        int rc2 = launch_igemm_fprop(tm_a, tm_b, om, p, m_tiles, cout_pad / n_tile, 1, (cudaStream_t)stream);
        if (rc2) return rc2;
        return launch_splitk_finish(splitk_ws, (long long)n * h * w, cout, bias, act, slope, y, y_ld, y_f32,
                                    (cudaStream_t)stream);
    }
    p.out_sn = (long long)h * w * y_ld, p.out_sh = (long long)w * y_ld, p.out_sw = y_ld;
    p.bias = bias, p.act = act, p.slope = slope, p.out_f32 = y_f32, p.out = y;
    rc = map_outputs(&om, p, 1, b);
    if (rc) return rc;
    return launch_igemm_fprop(tm_a, tm_b, om, p, m_tiles, cout_pad / n_tile, 1, (cudaStream_t)stream);
}

int pai_conv3x3_wgrad(const void* x, int n, int h, int w, int cin, int x_ld, const void* gy, int cout, int gy_ld,
                      float* dw, void* stream) {
    return wgrad_common(gy, n, h, w, cout, gy_ld, x, h, w, cin, x_ld, 3, dw, 0, (cudaStream_t)stream,
                        "pai_conv3x3_wgrad");
}

}  // extern "C"
