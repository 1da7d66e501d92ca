// Direct (CUDA-core) kernels for the four degenerate layers of the hot path, which are HBM-bound and
// have a 1- or 2-wide channel dimension that cannot feed a 64-channel TMA/UMMA K-block:
//   enc0  Conv2d(1, 64, 4, 2, 1)            models/pix2pix.py:141-147
//   D0    Conv2d(2, 64, 4, 2, 1)+LeakyReLU  models/wrapper.py:196-206,229 (input = cat([x, y], 1))
//   dec7  ConvTranspose2d(128, 1, 4, 2, 1)  models/pix2pix.py:186-192   (data / weight gradient)
// plus the im2col / col2im halves of the Attention U-Net's first and last layers with 1-4 image planes.
//   D4    Conv2d(512, 1, 4, 1, 1, no bias)  models/wrapper.py:233       (data / weight gradient)
//
//   pai_smallc_conv_fprop:  out[n,oy,ox,c] = act(bias[c] + sum_{t,j} plane_j[n, s*oy+dy_t, s*ox+dx_t] * W[c][t][j])
//   pai_smallc_conv_wgrad:  dW[c][t][j]   += sum_{n,y,x} A[n,y,x,c] * plane_j[n, s*y+dy_t, s*x+dx_t]
// with (dy_t, dx_t) = (ky-1, kx-1), or (1-ky, 1-kx) when `flip` (gradient of a stride-1 conv).
// Planes are single-channel fp32 images (the network input, target, prediction, or a 1-channel
// gradient); the wide operand is NHWC bf16.
#include "pai_common.cuh"
#include "pai_kernels.h"

namespace pai {

static constexpr int kDcThreads = 256;

struct SmallConvGeom {
    int n, ih, iw;   // plane (fine) grid
    int oh, ow;      // wide-tensor (coarse) grid
    int stride, flip, cin, c;
};

__device__ __forceinline__ void tap_offset(int t, int flip, int* dy, int* dx) {
    const int ky = t >> 2, kx = t & 3;
    *dy = flip ? 1 - ky : ky - 1;
    *dx = flip ? 1 - kx : kx - 1;
}

// thread <-> (8 channels, 4 consecutive output columns): the 4 x (3*STRIDE+4) input patch of each plane
// sits in registers and every shared-memory weight vector is reused for 4 pixels.
template <int STRIDE, int FLIP>
__global__ void __launch_bounds__(kDcThreads)
smallc_fprop_kernel(const float* __restrict__ p0, const float* __restrict__ p1, SmallConvGeom g,
                    const float* __restrict__ w /* [c][16][cin] */, const float* __restrict__ bias,
                    __nv_bfloat16* __restrict__ o1, int ld1, int act1, __nv_bfloat16* __restrict__ o2, int ld2,
                    int act2, float slope) {
    constexpr int PX = 4, COLS = 3 * STRIDE + 4;
    extern __shared__ float ws[];  // [16][cin][c]
    for (int i = threadIdx.x; i < g.c * 16 * g.cin; i += kDcThreads) {
        const int ch = i / (16 * g.cin), r = i - ch * 16 * g.cin;
        ws[r * g.c + ch] = w[i];
    }
    __syncthreads();
    const int cv = g.c >> 3;
    const int gx = (g.ow + PX - 1) / PX;
    const unsigned total = (unsigned)g.n * g.oh * gx * cv;   // < 2^31, checked by the launcher
    for (unsigned idx = blockIdx.x * kDcThreads + threadIdx.x; idx < total; idx += gridDim.x * kDcThreads) {
        const int vec = (int)(idx % (unsigned)cv);
        unsigned rest = idx / (unsigned)cv;
        const int ox0 = (int)(rest % (unsigned)gx) * PX;
        rest /= (unsigned)gx;
        const int oy = (int)(rest % (unsigned)g.oh);
        const int n = (int)(rest / (unsigned)g.oh);
        float acc[PX][8];
#pragma unroll
        for (int j = 0; j < PX; ++j)
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[j][i] = bias != nullptr ? bias[vec * 8 + i] : 0.f;
        const int iy0 = FLIP ? oy - 2 : oy * STRIDE - 1;
        const int ix0 = FLIP ? ox0 - 2 : ox0 * STRIDE - 1;
        const size_t plane_off = (size_t)n * g.ih * g.iw;
        for (int pl = 0; pl < g.cin; ++pl) {
            const float* __restrict__ src = (pl == 0 ? p0 : p1) + plane_off;
            float in[4][COLS];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int iy = iy0 + r;
                const bool rok = iy >= 0 && iy < g.ih;
#pragma unroll
                for (int cidx = 0; cidx < COLS; ++cidx) {
                    const int ix = ix0 + cidx;
                    in[r][cidx] = (rok && ix >= 0 && ix < g.iw) ? __ldg(src + (size_t)iy * g.iw + ix) : 0.f;
                }
            }
#pragma unroll
            for (int ky = 0; ky < 4; ++ky)
#pragma unroll
                for (int kx = 0; kx < 4; ++kx) {
                    const float* wr = ws + ((ky * 4 + kx) * g.cin + pl) * g.c + vec * 8;
                    const float4 wa = *reinterpret_cast<const float4*>(wr);
                    const float4 wb = *reinterpret_cast<const float4*>(wr + 4);
                    const float wv[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
                    const int r = FLIP ? 3 - ky : ky;
#pragma unroll
                    for (int j = 0; j < PX; ++j) {
                        const float v = in[r][FLIP ? j + 3 - kx : STRIDE * j + kx];
#pragma unroll
                        for (int i = 0; i < 8; ++i) acc[j][i] = fmaf(v, wv[i], acc[j][i]);
                    }
                }
        }
        const long long pix0 = ((long long)n * g.oh + oy) * g.ow + ox0;
#pragma unroll
        for (int j = 0; j < PX; ++j) {
            if (ox0 + j >= g.ow) break;
            uint4 u;
            __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float a = acc[j][2 * i], b = acc[j][2 * i + 1];
                if (act1 == PAI_ACT_LEAKY) a = a > 0.f ? a : a * slope, b = b > 0.f ? b : b * slope;
                if (act1 == PAI_ACT_RELU) a = fmaxf(a, 0.f), b = fmaxf(b, 0.f);
                h[i] = __floats2bfloat162_rn(a, b);
            }
            *reinterpret_cast<uint4*>(o1 + (pix0 + j) * ld1 + vec * 8) = u;
            if (o2 != nullptr) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    float a = acc[j][2 * i], b = acc[j][2 * i + 1];
                    if (act2 == PAI_ACT_LEAKY) a = a > 0.f ? a : a * slope, b = b > 0.f ? b : b * slope;
                    if (act2 == PAI_ACT_RELU) a = fmaxf(a, 0.f), b = fmaxf(b, 0.f);
                    h[i] = __floats2bfloat162_rn(a, b);
                }
                *reinterpret_cast<uint4*>(o2 + (pix0 + j) * ld2 + vec * 8) = u;
            }
        }
    }
}

// thread <-> (8 channels, 4 taps); a block covers kDcThreads / (4 * c/8) pixels per iteration
__global__ void __launch_bounds__(kDcThreads)
smallc_wgrad_kernel(const __nv_bfloat16* __restrict__ a, int lda, const float* __restrict__ p0,
                    const float* __restrict__ p1, SmallConvGeom g, float* __restrict__ dw /* [c][16][cin] */) {
    extern __shared__ float red[];  // [kDcThreads][8*4*cin]
    const int cv = g.c >> 3;
    const int tpp = cv * 4;                  // threads per pixel
    const int sub = threadIdx.x % tpp;
    const int vec = sub % cv, tg = sub / cv;  // channel vector, tap group (taps 4*tg .. 4*tg+3)
    const int ppb = kDcThreads / tpp;
    float acc[8][4][2];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int t = 0; t < 4; ++t) acc[i][t][0] = acc[i][t][1] = 0.f;
    const unsigned total = (unsigned)g.n * g.oh * g.ow;      // < 2^30, checked by the launcher
    const unsigned step = gridDim.x * ppb;
    // two pixels per iteration: all loads of both are issued before the FMAs (memory-level parallelism)
    for (unsigned pixa = blockIdx.x * ppb + threadIdx.x / tpp; pixa < total; pixa += 2 * step) {
        uint4 u[2];
        float v[2][4][2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const unsigned pix = pixa + q * step;
            const bool ok = pix < total;
            u[q] = ok ? *reinterpret_cast<const uint4*>(a + (size_t)pix * lda + vec * 8) : make_uint4(0, 0, 0, 0);
            const int ox = (int)(pix % (unsigned)g.ow);
            const unsigned row = pix / (unsigned)g.ow;
            const int oy = (int)(row % (unsigned)g.oh);
            const int n = (int)(row / (unsigned)g.oh);
            const size_t plane_off = (size_t)n * g.ih * g.iw;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                int dy, dx;
                tap_offset(tg * 4 + t, g.flip, &dy, &dx);
                const int iy = oy * g.stride + dy, ix = ox * g.stride + dx;
                const bool in_ok = ok && iy >= 0 && iy < g.ih && ix >= 0 && ix < g.iw;
                const size_t o = plane_off + (size_t)iy * g.iw + ix;
                v[q][t][0] = in_ok ? __ldg(p0 + o) : 0.f;
                v[q][t][1] = (in_ok && g.cin == 2) ? __ldg(p1 + o) : 0.f;
            }
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u[q]);
            float av[8];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float2 f = __bfloat1622float2(h[i]);
                av[2 * i] = f.x, av[2 * i + 1] = f.y;
            }
#pragma unroll
            for (int t = 0; t < 4; ++t)
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    acc[i][t][0] = fmaf(av[i], v[q][t][0], acc[i][t][0]);
                    if (g.cin == 2) acc[i][t][1] = fmaf(av[i], v[q][t][1], acc[i][t][1]);
                }
        }
    }
    const int per = 32 * g.cin;  // values per thread
    float* mine = red + (size_t)threadIdx.x * per;
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            mine[(i * 4 + t) * g.cin] = acc[i][t][0];
            if (g.cin == 2) mine[(i * 4 + t) * g.cin + 1] = acc[i][t][1];
        }
    __syncthreads();
    // outputs of this block: tpp * per values, each summed over the ppb pixel replicas
    for (int o = threadIdx.x; o < tpp * per; o += kDcThreads) {
        const int s = o / per, e = o - s * per;  // sub-thread, element
        float sum = 0.f;
        for (int r = 0; r < ppb; ++r) sum += red[(size_t)(r * tpp + s) * per + e];
        const int svec = s % cv, stg = s / cv;
        const int i = e / (4 * g.cin), t = (e / g.cin) % 4, j = e % g.cin;
        atomicAdd(dw + ((size_t)(svec * 8 + i) * 16 + stg * 4 + t) * g.cin + j, sum);
    }
}

// Base pointers of up to 4 fp32 planes; plane j of image n is the [ih, iw] image at p[j] + n * img.
struct PlaneRefs {
    const float* p[4];
    long long img;
};
__device__ __forceinline__ const float* plane_ref(const PlaneRefs& r, int j) {
    return j == 0 ? r.p[0] : j == 1 ? r.p[1] : j == 2 ? r.p[2] : r.p[3];   // no dynamic indexing of the parameter block
}

// im2col of 1 to 4 single-channel fp32 planes into a 64-channel bf16 NHWC tensor on the coarse grid, tap-major:
// col[n,oy,ox, t*cin + j] = plane_j[n, s*oy+dy_t, s*ox+dx_t]  (0 outside the image), rows are 64 channels wide.
// It turns the 1-4 channel wide convolutions into plain tensor-core GEMMs (pai_pointwise_gemm / _wgrad).
__global__ void __launch_bounds__(kDcThreads)
im2col4x4_kernel(PlaneRefs pl, SmallConvGeom g, __nv_bfloat16* __restrict__ col) {
    // 2 * cin vectors of 8 channels per pixel hold data; the padding up to 64 channels is NOT written (the GEMMs that
    // read col skip it: k_valid of pai_pointwise_gemm, discarded columns of pai_pointwise_wgrad) -- up to 4x less
    // store traffic than zero-filling the 128-byte rows
    const unsigned nvec = 2u * (unsigned)g.cin;
    const unsigned total = (unsigned)g.n * g.oh * g.ow * nvec;
    for (unsigned idx = blockIdx.x * kDcThreads + threadIdx.x; idx < total; idx += gridDim.x * kDcThreads) {
        const int vec = (int)(idx % nvec);
        const unsigned pix = idx / nvec;
        const int ox = (int)(pix % (unsigned)g.ow);
        const unsigned row = pix / (unsigned)g.ow;
        const int oy = (int)(row % (unsigned)g.oh);
        const int n = (int)(row / (unsigned)g.oh);
        const long long plane_off = (long long)n * pl.img;
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int ch = vec * 8 + i;
            const int t = ch / g.cin;
            const int j = ch - t * g.cin;
            int dy, dx;
            tap_offset(t, g.flip, &dy, &dx);
            const int iy = oy * g.stride + dy, ix = ox * g.stride + dx;
            float x = 0.f;
            if (iy >= 0 && iy < g.ih && ix >= 0 && ix < g.iw) x = __ldg(plane_ref(pl, j) + plane_off + (long long)iy * g.iw + ix);
            v[i] = x;
        }
        uint4 u;
        __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
        for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
        *reinterpret_cast<uint4*>(col + (size_t)pix * 64 + vec * 8) = u;
    }
}

// col2im of a transposed 4x4 stride-2 convolution with np (1..4) output channels, plane-major partial products:
// out_o[n, 2a+py, 2b+px] = act(bias[o] + sum_{(ky,dy) in T[py]} sum_{(kx,dx) in T[px]} P[n, a+dy, b+dx, o*16 + ky*4+kx])
// P: fp32 [n, h, w, ldp] (the 16*np per-tap partial products of pai_pointwise_gemm); thread <-> output pixel.
// Output plane o of image n is the [2h, 2w] image at out + n*img + o*ps.
__global__ void __launch_bounds__(kDcThreads)
col2im4x4s2_kernel(const float* __restrict__ P, int ldp, int n, int h, int w, const float* __restrict__ bias,
                   int act, float* __restrict__ out, int np, long long img, long long ps) {
    const unsigned total = (unsigned)n * np * 4 * h * w;
    const int ow = 2 * w, oh = 2 * h;
    for (unsigned idx = blockIdx.x * kDcThreads + threadIdx.x; idx < total; idx += gridDim.x * kDcThreads) {
        const int x = (int)(idx % (unsigned)ow);
        const unsigned r = idx / (unsigned)ow;
        const int y = (int)(r % (unsigned)oh);
        const unsigned pl = r / (unsigned)oh;
        const int img_i = (int)(pl / (unsigned)np), o = (int)(pl % (unsigned)np);
        const int a = y >> 1, py = y & 1, b = x >> 1, px = x & 1;
        // T[0] = {(k=1,d=0),(k=3,d=-1)}, T[1] = {(k=0,d=+1),(k=2,d=0)}
        const int ky0 = py ? 0 : 1, dy0 = py ? 1 : 0, ky1 = py ? 2 : 3, dy1 = py ? 0 : -1;
        const int kx0 = px ? 0 : 1, dx0 = px ? 1 : 0, kx1 = px ? 2 : 3, dx1 = px ? 0 : -1;
        float s = bias != nullptr ? bias[o] : 0.f;
        const float* base = P + (size_t)img_i * h * w * ldp + o * 16;
#define PAI_TAP(ky, dy, kx, dx)                                                            \
    if (a + (dy) >= 0 && a + (dy) < h && b + (dx) >= 0 && b + (dx) < w)                    \
        s += __ldg(base + ((size_t)(a + (dy)) * w + (b + (dx))) * ldp + (ky) * 4 + (kx));
        PAI_TAP(ky0, dy0, kx0, dx0) PAI_TAP(ky0, dy0, kx1, dx1) PAI_TAP(ky1, dy1, kx0, dx0) PAI_TAP(ky1, dy1, kx1, dx1)
#undef PAI_TAP
        if (act == PAI_ACT_TANH) s = tanhf(s);
        out[(long long)img_i * img + (long long)o * ps + (long long)y * ow + x] = s;
    }
}

}  // namespace pai

using namespace pai;

extern "C" {

static int launch_im2col4x4(const PlaneRefs& pl, int cin, int n, int ih, int iw, int oh, int ow, int stride, int flip,
                            void* col, void* stream) {
    SmallConvGeom g{n, ih, iw, oh, ow, stride, flip, cin, 64};
    long long blocks = ((long long)n * oh * ow * 2 * cin + kDcThreads - 1) / kDcThreads;
    if (blocks > 148 * 16) blocks = 148 * 16;
    im2col4x4_kernel<<<(int)blocks, kDcThreads, 0, (cudaStream_t)stream>>>(pl, g, (__nv_bfloat16*)col);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_im2col4x4(const float* plane0, const float* plane1, int cin, int n, int ih, int iw, int oh, int ow, int stride,
                  int flip, void* col, void* stream) {
    PAI_REQUIRE(plane0 && col && (cin == 1 || (cin == 2 && plane1)), "pai_im2col4x4: bad planes / cin=%d", cin);
    PAI_REQUIRE((long long)n * oh * ow * 8 < (1LL << 31), "pai_im2col4x4: tensor too large");
    const PlaneRefs pl{{plane0, plane1, nullptr, nullptr}, (long long)ih * iw};
    return launch_im2col4x4(pl, cin, n, ih, iw, oh, ow, stride, flip, col, stream);
}

int pai_im2col4x4_planes(const float* planes, int np, long long plane_stride, int n, int ih, int iw, int oh, int ow,
                         int stride, int flip, void* col, void* stream) {
    PAI_REQUIRE(planes && col, "pai_im2col4x4_planes: null pointer");
    PAI_REQUIRE(np >= 1 && np <= 4, "pai_im2col4x4_planes: plane count %d outside 1..4", np);
    PAI_REQUIRE(n > 0 && ih > 0 && iw > 0 && oh > 0 && ow > 0 && plane_stride >= (long long)ih * iw,
                "pai_im2col4x4_planes: bad size / plane stride %lld", plane_stride);
    PAI_REQUIRE((reinterpret_cast<uintptr_t>(planes) & 3) == 0 && (reinterpret_cast<uintptr_t>(col) & 15) == 0,
                "pai_im2col4x4_planes: alignment");
    PAI_REQUIRE((long long)n * oh * ow * 8 < (1LL << 31), "pai_im2col4x4_planes: tensor too large");
    PlaneRefs pl{{planes, planes, planes, planes}, np * plane_stride};
    for (int j = 1; j < np; ++j) pl.p[j] = planes + j * plane_stride;
    return launch_im2col4x4(pl, np, n, ih, iw, oh, ow, stride, flip, col, stream);
}

static void col2im4x4s2_launch(const float* p, int ldp, int n, int h, int w, const float* bias, int act, float* out,
                               int np, long long img, long long ps, void* stream) {
    long long blocks = ((long long)n * np * 4 * h * w + kDcThreads - 1) / kDcThreads;
    if (blocks > 148 * 16) blocks = 148 * 16;
    col2im4x4s2_kernel<<<(int)blocks, kDcThreads, 0, (cudaStream_t)stream>>>(p, ldp, n, h, w, bias, act, out, np, img, ps);
}

int pai_col2im4x4s2(const float* p, int ldp, int n, int h, int w, const float* bias, int act, float* out,
                    void* stream) {
    PAI_REQUIRE(p && out && ldp >= 16, "pai_col2im4x4s2: null pointer / ldp < 16");
    PAI_REQUIRE((long long)n * 4 * h * w < (1LL << 31), "pai_col2im4x4s2: tensor too large");
    const long long hw4 = 4LL * h * w;
    col2im4x4s2_launch(p, ldp, n, h, w, bias, act, out, 1, hw4, hw4, stream);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_col2im4x4s2_planes(const float* p, int ldp, int n, int h, int w, const float* bias, int act, float* out, int np,
                           long long plane_stride, void* stream) {
    PAI_REQUIRE(p && out, "pai_col2im4x4s2_planes: null pointer");
    PAI_REQUIRE(np >= 1 && np <= 4, "pai_col2im4x4s2_planes: plane count %d outside 1..4", np);
    PAI_REQUIRE(n > 0 && h > 0 && w > 0 && ldp >= 16 * np && plane_stride >= 4LL * h * w,
                "pai_col2im4x4s2_planes: bad size, ldp %d < 16 * planes or plane stride %lld", ldp, plane_stride);
    PAI_REQUIRE((reinterpret_cast<uintptr_t>(p) & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 3) == 0,
                "pai_col2im4x4s2_planes: alignment");
    PAI_REQUIRE((long long)n * np * 4 * h * w < (1LL << 31), "pai_col2im4x4s2_planes: tensor too large");
    col2im4x4s2_launch(p, ldp, n, h, w, bias, act, out, np, np * plane_stride, plane_stride, stream);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_smallc_conv_fprop(const float* plane0, const float* plane1, int cin, int n, int ih, int iw, int oh, int ow,
                          int stride, int flip, const float* w, const float* bias, int c, void* out1, int ld1,
                          int act1, void* out2, int ld2, int act2, float slope, void* stream) {
    PAI_REQUIRE(plane0 && w && out1 && (cin == 1 || (cin == 2 && plane1)), "pai_smallc_conv_fprop: bad planes / cin=%d", cin);
    PAI_REQUIRE(c > 0 && c % 8 == 0 && ld1 % 8 == 0 && (out2 == nullptr || ld2 % 8 == 0) && (stride == 1 || stride == 2),
                "pai_smallc_conv_fprop: c=%d must be a multiple of 8, stride 1|2", c);
    const size_t smem = sizeof(float) * 16 * cin * c;
    PAI_REQUIRE(smem <= 96 * 1024, "pai_smallc_conv_fprop: weights do not fit shared memory (c=%d)", c);
    PAI_REQUIRE((stride == 2 && !flip) || (stride == 1 && flip),
                "pai_smallc_conv_fprop: supported geometries are (stride 2, flip 0) and (stride 1, flip 1)");
    static DeviceOnce attr_once;
    const int attr_dev = current_device();
    if (attr_dev < 0) return -1;
    if (attr_once.need(attr_dev)) {
        PAI_CUDA_OK(cudaFuncSetAttribute(smallc_fprop_kernel<2, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        PAI_CUDA_OK(cudaFuncSetAttribute(smallc_fprop_kernel<1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        attr_once.mark(attr_dev);
    }
    SmallConvGeom g{n, ih, iw, oh, ow, stride, flip, cin, c};
    PAI_REQUIRE((long long)n * oh * ow * (c / 8) < (1LL << 31), "pai_smallc_conv_fprop: tensor too large");
    const long long total = (long long)n * oh * ((ow + 3) / 4) * (c / 8);
    long long blocks = (total + kDcThreads - 1) / kDcThreads;
    if (blocks > 148 * 8) blocks = 148 * 8;
    if (stride == 2)
        smallc_fprop_kernel<2, 0><<<(int)blocks, kDcThreads, smem, (cudaStream_t)stream>>>(
            plane0, plane1, g, w, bias, (__nv_bfloat16*)out1, ld1, act1, (__nv_bfloat16*)out2, ld2, act2, slope);
    else
        smallc_fprop_kernel<1, 1><<<(int)blocks, kDcThreads, smem, (cudaStream_t)stream>>>(
            plane0, plane1, g, w, bias, (__nv_bfloat16*)out1, ld1, act1, (__nv_bfloat16*)out2, ld2, act2, slope);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_smallc_conv_wgrad(const void* a, int lda, int c, const float* plane0, const float* plane1, int cin, int n,
                          int ih, int iw, int oh, int ow, int stride, int flip, float* dw, void* stream) {
    PAI_REQUIRE(a && plane0 && dw && (cin == 1 || (cin == 2 && plane1)), "pai_smallc_conv_wgrad: bad planes / cin=%d", cin);
    const int cv = c / 8;
    PAI_REQUIRE(c > 0 && c % 8 == 0 && lda % 8 == 0 && cv * 4 <= kDcThreads && kDcThreads % (cv * 4) == 0,
                "pai_smallc_conv_wgrad: c=%d must be a multiple of 8 with (c/2) | 256", c);
    const size_t smem = sizeof(float) * kDcThreads * 32 * cin;
    static DeviceOnce attr_once;
    const int attr_dev = current_device();
    if (attr_dev < 0) return -1;
    if (attr_once.need(attr_dev)) {
        PAI_CUDA_OK(cudaFuncSetAttribute(smallc_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        attr_once.mark(attr_dev);
    }
    SmallConvGeom g{n, ih, iw, oh, ow, stride, flip, cin, c};
    PAI_REQUIRE((long long)n * oh * ow < (1LL << 30), "pai_smallc_conv_wgrad: tensor too large");
    const int ppb = kDcThreads / (cv * 4);
    long long blocks = ((long long)n * oh * ow + ppb - 1) / ppb;
    // every block ends with (threads per pixel) * 32 * cin atomics: wide layers (c = 512: one pixel per block
    // iteration) get one block per SM, narrow ones a few waves
    const long long cap = ppb == 1 ? 148 : 148 * 6;
    if (blocks > cap) blocks = cap;
    cudaStream_t st = (cudaStream_t)stream;
    smallc_wgrad_kernel<<<(int)blocks, kDcThreads, smem, st>>>((const __nv_bfloat16*)a, lda, plane0, plane1, g, dw);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // extern "C"
