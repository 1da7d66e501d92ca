// Layer kernels of the Residual / Attention / Trans U-Net variants that are not dense contractions
// (those run on the implicit-GEMM kernels of igemm.cu).  All are HBM-bound streams over NHWC bf16
// tensors with 8-channel (16-byte) vectors; 1-channel tensors (network input / output, attention
// logits) are fp32 planes [n, h, w].
//
// Reference call sites:
//   nn.MaxPool2d(2) / nn.Upsample(scale_factor=2)         models/res_unet.py:196,228; models/trans_unet.py
//   residual add (+ReLU)                                   models/res_unet.py:90,129-130,170-171
//   x * attention                                          models/attention_unet.py:96
//   Conv2d(C, 64, 3, padding=1) / Conv2d(64, C, 3, padding=1) (+Tanh), C = 1..4   models/res_unet.py:263,312-320
//   Conv2d(C/2, 1, 1) of the attention gate                models/attention_unet.py:85-89
//   Conv2d(128, 128, 3, padding=1, groups=32) (ResNeXt)    models/res_unet.py:150-156
#include "pai_common.cuh"
#include "pai_kernels.h"

namespace pai {

static constexpr int kLyThreads = 256;

struct V8 {
    float v[8];
};
__device__ __forceinline__ V8 ld8(const __nv_bfloat16* p) {
    const uint4 u = *reinterpret_cast<const uint4*>(p);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
    V8 r;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 f = __bfloat1622float2(h[i]);
        r.v[2 * i] = f.x;
        r.v[2 * i + 1] = f.y;
    }
    return r;
}
__device__ __forceinline__ void st8(__nv_bfloat16* p, const V8& r) {
    uint4 u;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(r.v[2 * i], r.v[2 * i + 1]);
    *reinterpret_cast<uint4*>(p) = u;
}
static int ly_grid(long long items) {
    long long b = (items + kLyThreads - 1) / kLyThreads;
    if (b > 148LL * 16) b = 148LL * 16;
    return b < 1 ? 1 : (int)b;
}
__device__ __forceinline__ float act_apply(float v, int act, float slope) {
    if (act == PAI_ACT_LEAKY) return fmaxf(v, v * slope);
    if (act == PAI_ACT_RELU) return fmaxf(v, 0.f);
    if (act == PAI_ACT_TANH) return tanhf(v);
    return v;
}

// ---------------------------------------------------------------------------------------------
// MaxPool2d(2): y[n,oy,ox,:] = max of the 2x2 window; backward routes the gradient to the first maximum
// in row-major window order (PyTorch's tie rule).
__global__ void __launch_bounds__(kLyThreads)
maxpool2_fwd_kernel(const __nv_bfloat16* __restrict__ x, int n, int h, int w, int c, int ldx,
                    __nv_bfloat16* __restrict__ y, int ldy) {
    const int cv = c >> 3, oh = h >> 1, ow = w >> 1;
    const long long total = (long long)n * oh * ow * cv;
    for (long long i = (long long)blockIdx.x * kLyThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kLyThreads) {
        const int vec = (int)(i % cv);
        long long r = i / cv;
        const int ox = (int)(r % ow);
        r /= ow;
        const int oy = (int)(r % oh);
        const int b = (int)(r / oh);
        const __nv_bfloat16* src = x + (((long long)b * h + 2 * oy) * w + 2 * ox) * ldx + vec * 8;
        const V8 a = ld8(src), bq = ld8(src + ldx), cq = ld8(src + (long long)w * ldx), d = ld8(src + (long long)(w + 1) * ldx);
        V8 o;
#pragma unroll
        for (int k = 0; k < 8; ++k) o.v[k] = fmaxf(fmaxf(a.v[k], bq.v[k]), fmaxf(cq.v[k], d.v[k]));
        st8(y + (((long long)b * oh + oy) * ow + ox) * ldy + vec * 8, o);
    }
}
__global__ void __launch_bounds__(kLyThreads)
maxpool2_bwd_kernel(const __nv_bfloat16* __restrict__ x, int n, int h, int w, int c, int ldx,
                    const __nv_bfloat16* __restrict__ gy, int ldgy, __nv_bfloat16* __restrict__ gx, int ldgx) {
    const int cv = c >> 3, oh = h >> 1, ow = w >> 1;
    const long long total = (long long)n * oh * ow * cv;
    for (long long i = (long long)blockIdx.x * kLyThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kLyThreads) {
        const int vec = (int)(i % cv);
        long long r = i / cv;
        const int ox = (int)(r % ow);
        r /= ow;
        const int oy = (int)(r % oh);
        const int b = (int)(r / oh);
        const long long p00 = (((long long)b * h + 2 * oy) * w + 2 * ox);
        const __nv_bfloat16* src = x + p00 * ldx + vec * 8;
        const V8 a = ld8(src), bq = ld8(src + ldx), cq = ld8(src + (long long)w * ldx), d = ld8(src + (long long)(w + 1) * ldx);
        const V8 g = ld8(gy + (((long long)b * oh + oy) * ow + ox) * ldgy + vec * 8);
        V8 o[4];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float m = fmaxf(fmaxf(a.v[k], bq.v[k]), fmaxf(cq.v[k], d.v[k]));
            const int which = a.v[k] == m ? 0 : (bq.v[k] == m ? 1 : (cq.v[k] == m ? 2 : 3));
#pragma unroll
            for (int q = 0; q < 4; ++q) o[q].v[k] = which == q ? g.v[k] : 0.f;
        }
        __nv_bfloat16* dst = gx + p00 * ldgx + vec * 8;
        st8(dst, o[0]);
        st8(dst + ldgx, o[1]);
        st8(dst + (long long)w * ldgx, o[2]);
        st8(dst + (long long)(w + 1) * ldgx, o[3]);
    }
}

// Upsample(scale_factor=2, nearest): y[n,2a+i,2b+j,:] = x[n,a,b,:]; backward sums the 2x2 block.
__global__ void __launch_bounds__(kLyThreads)
upsample2_fwd_kernel(const __nv_bfloat16* __restrict__ x, int n, int h, int w, int c, int ldx,
                     __nv_bfloat16* __restrict__ y, int ldy) {
    const int cv = c >> 3;
    const long long total = (long long)n * h * w * cv;
    for (long long i = (long long)blockIdx.x * kLyThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kLyThreads) {
        const int vec = (int)(i % cv);
        long long r = i / cv;
        const int a = (int)(r % w);
        r /= w;
        const int b = (int)(r % h);
        const int nn = (int)(r / h);
        const uint4 u = *reinterpret_cast<const uint4*>(x + (((long long)nn * h + b) * w + a) * ldx + vec * 8);
        __nv_bfloat16* dst = y + (((long long)nn * 2 * h + 2 * b) * (2 * w) + 2 * a) * ldy + vec * 8;
        *reinterpret_cast<uint4*>(dst) = u;
        *reinterpret_cast<uint4*>(dst + ldy) = u;
        *reinterpret_cast<uint4*>(dst + (long long)2 * w * ldy) = u;
        *reinterpret_cast<uint4*>(dst + (long long)(2 * w + 1) * ldy) = u;
    }
}
__global__ void __launch_bounds__(kLyThreads)
upsample2_bwd_kernel(const __nv_bfloat16* __restrict__ gy, int n, int h, int w, int c, int ldgy,
                     __nv_bfloat16* __restrict__ gx, int ldgx) {
    const int cv = c >> 3;
    const long long total = (long long)n * h * w * cv;
    for (long long i = (long long)blockIdx.x * kLyThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kLyThreads) {
        const int vec = (int)(i % cv);
        long long r = i / cv;
        const int a = (int)(r % w);
        r /= w;
        const int b = (int)(r % h);
        const int nn = (int)(r / h);
        const __nv_bfloat16* src = gy + (((long long)nn * 2 * h + 2 * b) * (2 * w) + 2 * a) * ldgy + vec * 8;
        const V8 p = ld8(src), q = ld8(src + ldgy), s = ld8(src + (long long)2 * w * ldgy), t = ld8(src + (long long)(2 * w + 1) * ldgy);
        V8 o;
#pragma unroll
        for (int k = 0; k < 8; ++k) o.v[k] = (p.v[k] + q.v[k]) + (s.v[k] + t.v[k]);
        st8(gx + (((long long)nn * h + b) * w + a) * ldgx + vec * 8, o);
    }
}

// stride-2 subsampling (the 1x1 stride-2 projection of the Trans U-Net encoder, trans_unet.py:208-216):
// y[n,a,b,:] = x[n,2a,2b,:]; backward scatters into a zeroed tensor.
__global__ void __launch_bounds__(kLyThreads)
subsample2_kernel(const __nv_bfloat16* __restrict__ x, int n, int h, int w, int c, int ldx, __nv_bfloat16* __restrict__ y,
                  int ldy, int scatter) {
    const int cv = c >> 3, oh = h >> 1, ow = w >> 1;
    const long long total = (long long)n * oh * ow * cv;
    for (long long i = (long long)blockIdx.x * kLyThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kLyThreads) {
        const int vec = (int)(i % cv);
        long long r = i / cv;
        const int ox = (int)(r % ow);
        r /= ow;
        const int oy = (int)(r % oh);
        const int b = (int)(r / oh);
        const long long fine = (((long long)b * h + 2 * oy) * w + 2 * ox), coarse = (((long long)b * oh + oy) * ow + ox);
        if (!scatter)   // x fine -> y coarse
            *reinterpret_cast<uint4*>(y + coarse * ldy + vec * 8) = *reinterpret_cast<const uint4*>(x + fine * ldx + vec * 8);
        else            // x coarse (gradient) -> y fine (pre-zeroed)
            *reinterpret_cast<uint4*>(y + fine * ldy + vec * 8) = *reinterpret_cast<const uint4*>(x + coarse * ldx + vec * 8);
    }
}

// out = act(a + b) (b nullable) over [m, c]
__global__ void __launch_bounds__(kLyThreads)
add_act_kernel(const __nv_bfloat16* __restrict__ a, int lda, const __nv_bfloat16* __restrict__ b, int ldb, long long m,
               int c, int act, float slope, __nv_bfloat16* __restrict__ out, int ldo) {
    const int cv = c >> 3;
    const long long total = m * cv;
    for (long long i = (long long)blockIdx.x * kLyThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kLyThreads) {
        const int vec = (int)(i % cv);
        const long long pix = i / cv;
        V8 x = ld8(a + pix * lda + vec * 8);
        if (b != nullptr) {
            const V8 y = ld8(b + pix * ldb + vec * 8);
#pragma unroll
            for (int k = 0; k < 8; ++k) x.v[k] += y.v[k];
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) x.v[k] = act_apply(x.v[k], act, slope);
        st8(out + pix * ldo + vec * 8, x);
    }
}

// row scaling by a per-pixel fp32 factor: out[p, :] = act(x[p, :] * s[p]);  backward: gx = g * s * act',
// gs[p] = sum_c g * act' * x  (one warp per pixel group; 8 lanes share a pixel when c = 64, ...)
__global__ void __launch_bounds__(kLyThreads)
scale_rows_fwd_kernel(const __nv_bfloat16* __restrict__ x, int ldx, const float* __restrict__ s, long long m, int c,
                      int act, __nv_bfloat16* __restrict__ out, int ldo) {
    const int cv = c >> 3;
    const long long total = m * cv;
    for (long long i = (long long)blockIdx.x * kLyThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kLyThreads) {
        const int vec = (int)(i % cv);
        const long long pix = i / cv;
        V8 v = ld8(x + pix * ldx + vec * 8);
        const float f = s[pix];
#pragma unroll
        for (int k = 0; k < 8; ++k) v.v[k] = act_apply(v.v[k] * f, act, 0.f);
        st8(out + pix * ldo + vec * 8, v);
    }
}
// nn.Dropout2d on NHWC: out[n, p, c] = x[n, p, c] * mask[n, c]  (mask = 0 or 1 / (1 - p_drop) per (sample, channel));
// the backward is the same multiplication applied to the gradient.
__global__ void __launch_bounds__(kLyThreads)
scale_channels_kernel(const __nv_bfloat16* __restrict__ x, int ldx, const float* __restrict__ mask, long long m,
                      long long hw, int c, __nv_bfloat16* __restrict__ out, int ldo) {
    const int cv = c >> 3;
    const long long total = m * cv;
    for (long long i = (long long)blockIdx.x * kLyThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kLyThreads) {
        const int vec = (int)(i % cv);
        const long long pix = i / cv;
        V8 v = ld8(x + pix * ldx + vec * 8);
        const float* mk = mask + (pix / hw) * c + vec * 8;
#pragma unroll
        for (int k = 0; k < 8; ++k) v.v[k] *= mk[k];
        st8(out + pix * ldo + vec * 8, v);
    }
}
// one warp per pixel: lanes stride over the channel vectors, shuffle-reduce the dot product
__global__ void __launch_bounds__(kLyThreads)
scale_rows_bwd_kernel(const __nv_bfloat16* __restrict__ x, int ldx, const float* __restrict__ s,
                      const __nv_bfloat16* __restrict__ g, int ldg, long long m, int c, int act,
                      __nv_bfloat16* __restrict__ gx, int ldgx, float* __restrict__ gs) {
    const int cv = c >> 3, lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * kLyThreads + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * kLyThreads) >> 5;
    for (long long pix = warp; pix < m; pix += nwarps) {
        const float f = s[pix];
        float dot = 0.f;
        for (int vec = lane; vec < cv; vec += 32) {
            const V8 xv = ld8(x + pix * ldx + vec * 8);
            V8 gv = ld8(g + pix * ldg + vec * 8);
            V8 o;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                if (act == PAI_ACT_RELU && !(xv.v[k] * f > 0.f)) gv.v[k] = 0.f;
                o.v[k] = gv.v[k] * f;
                dot = fmaf(gv.v[k], xv.v[k], dot);
            }
            st8(gx + pix * ldgx + vec * 8, o);
        }
        dot = warp_sum(dot);
        if (lane == 0) gs[pix] = dot;
    }
}

// ---------------------------------------------------------------------------------------------
// P-plane (1 <= P <= 4) <-> C-channel k x k convolutions (stride 1, zero padding `pad`), taps t = ky*k + kx at offset
// (ky - pad, kx - pad), negated when `flip`.  Plane j of image b is the fp32 [h, w] image at base + b*img + j*ps
// (NCHW [n, P, h, w]: ps = h*w, img = P*h*w; a 1-plane [n, h, w] tensor is img = h*w).
//   plane_to_wide:  out[p, c]  = act(bias[c] + sum_j sum_t plane_j[p + off_t] * w[c][j][t])
//   wide_to_plane:  out_o[p]   = act(bias[o] + sum_t sum_c x[p + off_t, c] * w[o][t][c])      (o < P)
//   plane_wide_wgrad: dw[c][j][t] += sum_p wide[p, c] * plane_j[p + off_t]
// With P = 1 every kernel issues the FMAs of the original 1-plane kernels in the same order, so the 1-plane entry
// points (which call these kernels) give the same bits as before.
__global__ void __launch_bounds__(kLyThreads)
plane_to_wide_kernel(const float* __restrict__ planes, long long img, long long ps, int np, int n, int h, int w, int k,
                     int pad, int flip, const float* __restrict__ wt /* [c][np][k*k] */, const float* __restrict__ bias,
                     int c, int act, float slope, __nv_bfloat16* __restrict__ out, int ldo) {
    extern __shared__ float wsm[];   // [np*k*k][c]
    const int taps = k * k, rows = np * taps;
    for (int i = threadIdx.x; i < c * rows; i += kLyThreads) wsm[(i % rows) * c + i / rows] = wt[i];
    __syncthreads();
    const int cv = c >> 3;
    const long long total = (long long)n * h * w * cv;
    for (long long i = (long long)blockIdx.x * kLyThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kLyThreads) {
        const int vec = (int)(i % cv);
        long long r = i / cv;
        const int x0 = (int)(r % w);
        r /= w;
        const int y0 = (int)(r % h);
        const int b = (int)(r / h);
        V8 acc;
#pragma unroll
        for (int q = 0; q < 8; ++q) acc.v[q] = bias != nullptr ? bias[vec * 8 + q] : 0.f;
        for (int j = 0; j < np; ++j) {
            const float* src = planes + (long long)b * img + (long long)j * ps;
            for (int t = 0; t < taps; ++t) {
                int dy = t / k - pad, dx = t % k - pad;
                if (flip) dy = -dy, dx = -dx;
                const int yy = y0 + dy, xx = x0 + dx;
                if (yy < 0 || yy >= h || xx < 0 || xx >= w) continue;
                const float v = __ldg(src + (long long)yy * w + xx);
                const float* wr = wsm + (j * taps + t) * c + vec * 8;
#pragma unroll
                for (int q = 0; q < 8; ++q) acc.v[q] = fmaf(v, wr[q], acc.v[q]);
            }
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) acc.v[q] = act_apply(acc.v[q], act, slope);
        st8(out + (((long long)b * h + y0) * w + x0) * ldo + vec * 8, acc);
    }
}

// 8 lanes per pixel (channel vectors strided by 8), shuffle reduce; all P output planes from one read of x
template <int P>
__global__ void __launch_bounds__(kLyThreads)
wide_to_plane_kernel(const __nv_bfloat16* __restrict__ x, int n, int h, int w, int c, int ldx, int k, int pad,
                     const float* __restrict__ wt /* [P][k*k][c] */, const float* __restrict__ bias, int act,
                     float* __restrict__ out, long long img, long long ps) {
    const int cv = c >> 3, sub = threadIdx.x & 7, taps = k * k;
    const long long total = (long long)n * h * w;
    const long long g0 = ((long long)blockIdx.x * kLyThreads + threadIdx.x) >> 3;
    const long long ng = ((long long)gridDim.x * kLyThreads) >> 3;
    const long long rounds = (total + ng - 1) / ng;
    for (long long it = 0; it < rounds; ++it) {
        const long long p = g0 + it * ng;
        float acc[P];
#pragma unroll
        for (int o = 0; o < P; ++o) acc[o] = 0.f;
        int x0 = 0, y0 = 0, b = 0;
        if (p < total) {
            x0 = (int)(p % w);
            y0 = (int)((p / w) % h);
            b = (int)(p / ((long long)w * h));
            for (int t = 0; t < taps; ++t) {
                const int yy = y0 + t / k - pad, xx = x0 + t % k - pad;
                if (yy < 0 || yy >= h || xx < 0 || xx >= w) continue;
                const __nv_bfloat16* src = x + (((long long)b * h + yy) * w + xx) * ldx;
                for (int vec = sub; vec < cv; vec += 8) {
                    const V8 v = ld8(src + vec * 8);
#pragma unroll
                    for (int o = 0; o < P; ++o) {
                        const float* wr = wt + ((long long)o * taps + t) * c + vec * 8;
#pragma unroll
                        for (int q = 0; q < 8; ++q) acc[o] = fmaf(v.v[q], __ldg(wr + q), acc[o]);
                    }
                }
            }
        }
#pragma unroll
        for (int o = 0; o < P; ++o) {
            acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], 1);
            acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], 2);
            acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], 4);
        }
        if (p < total && sub == 0) {
            float* dst = out + (long long)b * img + (long long)y0 * w + x0;
#pragma unroll
            for (int o = 0; o < P; ++o) dst[(long long)o * ps] = act_apply(acc[o] + (bias != nullptr ? bias[o] : 0.f), act, 0.f);
        }
    }
}

// thread <-> (pixel, 8 channels); per-thread partial sums for all taps (<= 9) of ONE plane, block reduce, atomics.
// The planes are spread over the grid (block = pixel block * np + plane), so a thread never holds more than
// TAPS x 8 accumulators whatever np is; the np blocks of a pixel block run side by side and share the wide reads in L2.
template <int TAPS>
__global__ void __launch_bounds__(kLyThreads)
plane_wide_wgrad_kernel(const float* __restrict__ planes, long long img, long long ps, int np,
                        const __nv_bfloat16* __restrict__ wide, int ldw, int n, int h, int w, int c, int k, int pad,
                        int flip, float* __restrict__ dw /* [c][np][TAPS] */) {
    __shared__ float red[kLyThreads * 8];
    const int cv = c >> 3;
    const int vec = threadIdx.x % cv;
    const int ppb = kLyThreads / cv;
    const int j = (int)(blockIdx.x % (unsigned)np);
    const long long blk = blockIdx.x / (unsigned)np, nblk = gridDim.x / (unsigned)np;
    const float* src = planes + (long long)j * ps;
    float acc[TAPS][8];
#pragma unroll
    for (int t = 0; t < TAPS; ++t)
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[t][q] = 0.f;
    const long long total = (long long)n * h * w;
    for (long long p = blk * ppb + threadIdx.x / cv; p < total; p += nblk * ppb) {
        const int x0 = (int)(p % w);
        const int y0 = (int)((p / w) % h);
        const int b = (int)(p / ((long long)w * h));
        const V8 v = ld8(wide + p * ldw + vec * 8);
#pragma unroll
        for (int t = 0; t < TAPS; ++t) {
            int dy = t / k - pad, dx = t % k - pad;
            if (flip) dy = -dy, dx = -dx;
            const int yy = y0 + dy, xx = x0 + dx;
            const float s = (yy >= 0 && yy < h && xx >= 0 && xx < w) ? __ldg(src + (long long)b * img + (long long)yy * w + xx) : 0.f;
#pragma unroll
            for (int q = 0; q < 8; ++q) acc[t][q] = fmaf(v.v[q], s, acc[t][q]);
        }
    }
#pragma unroll
    for (int t = 0; t < TAPS; ++t) {
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 8; ++q) red[threadIdx.x * 8 + q] = acc[t][q];
        __syncthreads();
        for (int i = threadIdx.x; i < cv * 8; i += kLyThreads) {
            const int vv = i >> 3, q = i & 7;
            float s = 0.f;
            for (int r = vv; r < kLyThreads; r += cv) s += red[r * 8 + q];
            atomicAdd(dw + ((long long)i * np + j) * TAPS + t, s);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Grouped 3x3 convolution with 4 input and 4 output channels per group (ResNeXt, cardinality 32 x 4):
// a thread owns 8 consecutive channels = two whole groups of one pixel.
//   fprop:  y[p, co] = bias[co] + sum_t sum_{j<4} x[p + off_t, 4*(co/4) + j] * w[co][t][j]
//   (dgrad is the same kernel on gy with the taps flipped and w transposed within each group)
//   wgrad:  dw[co][t][j] += sum_p gy[p, co] * x[p + off_t, 4*(co/4) + j]
__global__ void __launch_bounds__(kLyThreads)
gconv4_fprop_kernel(const __nv_bfloat16* __restrict__ x, int n, int h, int w, int c, int ldx,
                    const float* __restrict__ wt /* [c][9][4] */, const float* __restrict__ bias,
                    __nv_bfloat16* __restrict__ y, int ldy) {
    extern __shared__ float wsm[];   // [9][c][4]
    for (int i = threadIdx.x; i < c * 36; i += kLyThreads) {
        const int co = i / 36, r = i - co * 36, t = r >> 2, j = r & 3;
        wsm[(t * c + co) * 4 + j] = wt[i];
    }
    __syncthreads();
    const int cv = c >> 3;
    const long long total = (long long)n * h * w * cv;
    for (long long i = (long long)blockIdx.x * kLyThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kLyThreads) {
        const int vec = (int)(i % cv);
        long long r = i / cv;
        const int x0 = (int)(r % w);
        r /= w;
        const int y0 = (int)(r % h);
        const int b = (int)(r / h);
        V8 acc;
#pragma unroll
        for (int q = 0; q < 8; ++q) acc.v[q] = bias != nullptr ? bias[vec * 8 + q] : 0.f;
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            const int yy = y0 + t / 3 - 1, xx = x0 + t % 3 - 1;
            if (yy < 0 || yy >= h || xx < 0 || xx >= w) continue;
            const V8 v = ld8(x + (((long long)b * h + yy) * w + xx) * ldx + vec * 8);
            const float4* wr = reinterpret_cast<const float4*>(wsm + ((long long)t * c + vec * 8) * 4);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const float4 ww = wr[q];
                const int base = (q >> 2) * 4;
                acc.v[q] = fmaf(v.v[base], ww.x, fmaf(v.v[base + 1], ww.y, fmaf(v.v[base + 2], ww.z, fmaf(v.v[base + 3], ww.w, acc.v[q]))));
            }
        }
        st8(y + (((long long)b * h + y0) * w + x0) * ldy + vec * 8, acc);
    }
}

// grid (pixel blocks, 3 tap rows): thread <-> (pixel lane, 8 channels = 2 groups); the three taps dx = -1, 0, +1 of the
// row share one load of the output gradient (3 instead of 9 passes over gy, all four 16-byte loads of a pixel in
// flight together), 96 partial sums per thread, block reduce per tap
__global__ void __launch_bounds__(kLyThreads)
gconv4_wgrad_kernel(const __nv_bfloat16* __restrict__ x, int ldx, const __nv_bfloat16* __restrict__ gy, int ldg, int n,
                    int h, int w, int c, float* __restrict__ dw /* [c][9][4] */) {
    __shared__ float red[kLyThreads * 33];
    const int dy = (int)blockIdx.y - 1;
    const int cv = c >> 3;
    const int vec = threadIdx.x % cv;
    const int ppb = kLyThreads / cv;
    float acc[3][8][4];
#pragma unroll
    for (int t = 0; t < 3; ++t)
#pragma unroll
        for (int q = 0; q < 8; ++q)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[t][q][j] = 0.f;
    const long long total = (long long)n * h * w;
    const uint4 zero = make_uint4(0, 0, 0, 0);
    for (long long p = (long long)blockIdx.x * ppb + threadIdx.x / cv; p < total; p += (long long)gridDim.x * ppb) {
        const int x0 = (int)(p % w);
        const int y0 = (int)((p / w) % h);
        const int yy = y0 + dy;
        if (yy < 0 || yy >= h) continue;
        const __nv_bfloat16* xr = x + (p + (long long)dy * w) * ldx + vec * 8;
        const uint4 rg = *reinterpret_cast<const uint4*>(gy + p * ldg + vec * 8);
        uint4 rx[3];
        rx[0] = x0 > 0 ? *reinterpret_cast<const uint4*>(xr - ldx) : zero;
        rx[1] = *reinterpret_cast<const uint4*>(xr);
        rx[2] = x0 + 1 < w ? *reinterpret_cast<const uint4*>(xr + ldx) : zero;
        V8 g;
        {
            const __nv_bfloat162* hg = reinterpret_cast<const __nv_bfloat162*>(&rg);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float2 f = __bfloat1622float2(hg[i]);
                g.v[2 * i] = f.x, g.v[2 * i + 1] = f.y;
            }
        }
#pragma unroll
        for (int t = 0; t < 3; ++t) {
            V8 v;
            const __nv_bfloat162* hv = reinterpret_cast<const __nv_bfloat162*>(&rx[t]);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float2 f = __bfloat1622float2(hv[i]);
                v.v[2 * i] = f.x, v.v[2 * i + 1] = f.y;
            }
#pragma unroll
            for (int q = 0; q < 8; ++q)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[t][q][j] = fmaf(g.v[q], v.v[(q >> 2) * 4 + j], acc[t][q][j]);
        }
    }
#pragma unroll
    for (int t = 0; t < 3; ++t) {
#pragma unroll
        for (int q = 0; q < 8; ++q)
#pragma unroll
            for (int j = 0; j < 4; ++j) red[threadIdx.x * 33 + q * 4 + j] = acc[t][q][j];
        __syncthreads();
        const int tap = ((int)blockIdx.y) * 3 + t;
        for (int i = threadIdx.x; i < cv * 32; i += kLyThreads) {
            const int vv = i >> 5, e = i & 31;          // e = q*4 + j
            float s = 0.f;
            for (int r = vv; r < kLyThreads; r += cv) s += red[r * 33 + e];
            const int co = vv * 8 + (e >> 2), j = e & 3;
            atomicAdd(dw + ((long long)co * 9 + tap) * 4 + j, s);
        }
        __syncthreads();
    }
}

static bool v8_ok(int c, const void* p, int ld) {
    return c > 0 && c % 8 == 0 && ld % 8 == 0 && (reinterpret_cast<uintptr_t>(p) & 15) == 0;
}
static bool cv_divides_block(int c) { return (c >> 3) <= kLyThreads && kLyThreads % (c >> 3) == 0; }

}  // namespace pai

using namespace pai;
typedef __nv_bfloat16 bf16;

extern "C" {

int pai_maxpool2_fwd(const void* x, int n, int h, int w, int c, int ldx, void* y, int ldy, void* stream) {
    PAI_REQUIRE(x && y && n > 0 && h % 2 == 0 && w % 2 == 0, "pai_maxpool2_fwd: null pointer or odd size %dx%d", h, w);
    PAI_REQUIRE(v8_ok(c, x, ldx) && v8_ok(c, y, ldy), "pai_maxpool2_fwd: c=%d must be a multiple of 8, 16 B aligned", c);
    maxpool2_fwd_kernel<<<ly_grid((long long)n * (h / 2) * (w / 2) * (c / 8)), kLyThreads, 0, (cudaStream_t)stream>>>(
        (const bf16*)x, n, h, w, c, ldx, (bf16*)y, ldy);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_maxpool2_bwd(const void* x, int n, int h, int w, int c, int ldx, const void* gy, int ldgy, void* gx, int ldgx,
                     void* stream) {
    PAI_REQUIRE(x && gy && gx && n > 0 && h % 2 == 0 && w % 2 == 0, "pai_maxpool2_bwd: null pointer or odd size");
    PAI_REQUIRE(v8_ok(c, x, ldx) && v8_ok(c, gy, ldgy) && v8_ok(c, gx, ldgx), "pai_maxpool2_bwd: bad channels / alignment");
    maxpool2_bwd_kernel<<<ly_grid((long long)n * (h / 2) * (w / 2) * (c / 8)), kLyThreads, 0, (cudaStream_t)stream>>>(
        (const bf16*)x, n, h, w, c, ldx, (const bf16*)gy, ldgy, (bf16*)gx, ldgx);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_upsample2_fwd(const void* x, int n, int h, int w, int c, int ldx, void* y, int ldy, void* stream) {
    PAI_REQUIRE(x && y && n > 0, "pai_upsample2_fwd: null pointer");
    PAI_REQUIRE(v8_ok(c, x, ldx) && v8_ok(c, y, ldy), "pai_upsample2_fwd: bad channels / alignment");
    upsample2_fwd_kernel<<<ly_grid((long long)n * h * w * (c / 8)), kLyThreads, 0, (cudaStream_t)stream>>>(
        (const bf16*)x, n, h, w, c, ldx, (bf16*)y, ldy);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_upsample2_bwd(const void* gy, int n, int h, int w, int c, int ldgy, void* gx, int ldgx, void* stream) {
    PAI_REQUIRE(gy && gx && n > 0, "pai_upsample2_bwd: null pointer");
    PAI_REQUIRE(v8_ok(c, gy, ldgy) && v8_ok(c, gx, ldgx), "pai_upsample2_bwd: bad channels / alignment");
    upsample2_bwd_kernel<<<ly_grid((long long)n * h * w * (c / 8)), kLyThreads, 0, (cudaStream_t)stream>>>(
        (const bf16*)gy, n, h, w, c, ldgy, (bf16*)gx, ldgx);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_subsample2(const void* x, int n, int h, int w, int c, int ldx, void* y, int ldy, int scatter, void* stream) {
    PAI_REQUIRE(x && y && n > 0 && h % 2 == 0 && w % 2 == 0, "pai_subsample2: null pointer or odd size");
    PAI_REQUIRE(v8_ok(c, x, ldx) && v8_ok(c, y, ldy), "pai_subsample2: bad channels / alignment");
    subsample2_kernel<<<ly_grid((long long)n * (h / 2) * (w / 2) * (c / 8)), kLyThreads, 0, (cudaStream_t)stream>>>(
        (const bf16*)x, n, h, w, c, ldx, (bf16*)y, ldy, scatter);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_add_act(const void* a, int lda, const void* b, int ldb, long long m, int c, int act, float slope, void* out,
                int ldo, void* stream) {
    PAI_REQUIRE(a && out && m > 0, "pai_add_act: null pointer");
    PAI_REQUIRE(v8_ok(c, a, lda) && (b == nullptr || v8_ok(c, b, ldb)) && v8_ok(c, out, ldo), "pai_add_act: bad channels / alignment");
    add_act_kernel<<<ly_grid(m * (c / 8)), kLyThreads, 0, (cudaStream_t)stream>>>((const bf16*)a, lda, (const bf16*)b, ldb, m,
                                                                                 c, act, slope, (bf16*)out, ldo);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_scale_rows_fwd(const void* x, int ldx, const float* s, long long m, int c, int act, void* out, int ldo,
                       void* stream) {
    PAI_REQUIRE(x && s && out && m > 0, "pai_scale_rows_fwd: null pointer");
    PAI_REQUIRE(v8_ok(c, x, ldx) && v8_ok(c, out, ldo), "pai_scale_rows_fwd: bad channels / alignment");
    scale_rows_fwd_kernel<<<ly_grid(m * (c / 8)), kLyThreads, 0, (cudaStream_t)stream>>>((const bf16*)x, ldx, s, m, c, act,
                                                                                        (bf16*)out, ldo);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_scale_channels(const void* x, int ldx, const float* mask, int n, long long hw, int c, void* out, int ldo,
                       void* stream) {
    PAI_REQUIRE(x && mask && out && n > 0 && hw > 0, "pai_scale_channels: null pointer / empty input");
    PAI_REQUIRE(v8_ok(c, x, ldx) && v8_ok(c, out, ldo), "pai_scale_channels: bad channels / alignment");
    scale_channels_kernel<<<ly_grid((long long)n * hw * (c / 8)), kLyThreads, 0, (cudaStream_t)stream>>>(
        (const bf16*)x, ldx, mask, (long long)n * hw, hw, c, (bf16*)out, ldo);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_scale_rows_bwd(const void* x, int ldx, const float* s, const void* g, int ldg, long long m, int c, int act,
                       void* gx, int ldgx, float* gs, void* stream) {
    PAI_REQUIRE(x && s && g && gx && gs && m > 0, "pai_scale_rows_bwd: null pointer");
    PAI_REQUIRE(v8_ok(c, x, ldx) && v8_ok(c, g, ldg) && v8_ok(c, gx, ldgx), "pai_scale_rows_bwd: bad channels / alignment");
    scale_rows_bwd_kernel<<<ly_grid(m * 32), kLyThreads, 0, (cudaStream_t)stream>>>((const bf16*)x, ldx, s, (const bf16*)g, ldg,
                                                                                   m, c, act, (bf16*)gx, ldgx, gs);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
static bool planes_ok(int np, long long ps, int h, int w, const void* p) {
    return np >= 1 && np <= 4 && ps >= (long long)h * w && (reinterpret_cast<uintptr_t>(p) & 3) == 0;
}
static int launch_plane_to_wide(const char* who, const float* planes, long long img, long long ps, int np, int n, int h,
                                int w, int k, int pad, int flip, const float* wt, const float* bias, int c, int act,
                                float slope, void* out, int ldo, void* stream) {
    PAI_REQUIRE(v8_ok(c, out, ldo) && c * np * k * k * 4 <= 48 * 1024, "%s: bad channels / alignment", who);
    plane_to_wide_kernel<<<ly_grid((long long)n * h * w * (c / 8)), kLyThreads, c * np * k * k * sizeof(float),
                           (cudaStream_t)stream>>>(planes, img, ps, np, n, h, w, k, pad, flip, wt, bias, c, act, slope,
                                                   (bf16*)out, ldo);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
static int launch_wide_to_plane(const void* x, int n, int h, int w, int c, int ldx, int k, int pad, const float* wt,
                                const float* bias, int act, float* out, int np, long long img, long long ps, void* stream) {
    const int grid = ly_grid((long long)n * h * w * 8);
    cudaStream_t st = (cudaStream_t)stream;
    switch (np) {
        case 1: wide_to_plane_kernel<1><<<grid, kLyThreads, 0, st>>>((const bf16*)x, n, h, w, c, ldx, k, pad, wt, bias, act, out, img, ps); break;
        case 2: wide_to_plane_kernel<2><<<grid, kLyThreads, 0, st>>>((const bf16*)x, n, h, w, c, ldx, k, pad, wt, bias, act, out, img, ps); break;
        case 3: wide_to_plane_kernel<3><<<grid, kLyThreads, 0, st>>>((const bf16*)x, n, h, w, c, ldx, k, pad, wt, bias, act, out, img, ps); break;
        default: wide_to_plane_kernel<4><<<grid, kLyThreads, 0, st>>>((const bf16*)x, n, h, w, c, ldx, k, pad, wt, bias, act, out, img, ps); break;
    }
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
static int launch_plane_wide_wgrad(const char* who, const float* planes, long long img, long long ps, int np,
                                   const void* wide, int ldw, int n, int h, int w, int c, int k, int pad, int flip,
                                   float* dw, void* stream) {
    PAI_REQUIRE(k == 1 || k == 3, "%s: k must be 1 or 3 (got %d)", who, k);
    PAI_REQUIRE(v8_ok(c, wide, ldw) && cv_divides_block(c), "%s: bad channels / alignment (c=%d)", who, c);
    const long long ppb = kLyThreads / (c / 8);
    long long blocks = ((long long)n * h * w + ppb - 1) / ppb;
    if (blocks > 148 * 4) blocks = 148 * 4;
    blocks *= np;
    if (k == 1)
        plane_wide_wgrad_kernel<1><<<(int)blocks, kLyThreads, 0, (cudaStream_t)stream>>>(planes, img, ps, np, (const bf16*)wide,
                                                                                       ldw, n, h, w, c, k, pad, flip, dw);
    else
        plane_wide_wgrad_kernel<9><<<(int)blocks, kLyThreads, 0, (cudaStream_t)stream>>>(planes, img, ps, np, (const bf16*)wide,
                                                                                       ldw, n, h, w, c, k, pad, flip, dw);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_conv_plane_to_wide(const float* plane, int n, int h, int w, int k, int pad, int flip, const float* wt,
                           const float* bias, int c, int act, float slope, void* out, int ldo, void* stream) {
    PAI_REQUIRE(plane && wt && out && n > 0 && k >= 1 && k <= 4, "pai_conv_plane_to_wide: null pointer or k=%d", k);
    const long long hw = (long long)h * w;
    return launch_plane_to_wide("pai_conv_plane_to_wide", plane, hw, hw, 1, n, h, w, k, pad, flip, wt, bias, c, act, slope,
                                out, ldo, stream);
}
int pai_conv_planes_to_wide(const float* planes, int np, long long plane_stride, int n, int h, int w, int k, int pad,
                            int flip, const float* wt, const float* bias, int c, int act, float slope, void* out, int ldo,
                            void* stream) {
    PAI_REQUIRE(planes && wt && out, "pai_conv_planes_to_wide: null pointer");
    PAI_REQUIRE(np >= 1 && np <= 4, "pai_conv_planes_to_wide: plane count %d outside 1..4", np);
    PAI_REQUIRE(n > 0 && h > 0 && w > 0 && k >= 1 && k <= 4, "pai_conv_planes_to_wide: bad size or k=%d", k);
    PAI_REQUIRE(planes_ok(np, plane_stride, h, w, planes), "pai_conv_planes_to_wide: plane stride %lld / alignment",
                plane_stride);
    return launch_plane_to_wide("pai_conv_planes_to_wide", planes, np * plane_stride, plane_stride, np, n, h, w, k, pad, flip,
                                wt, bias, c, act, slope, out, ldo, stream);
}
int pai_conv_wide_to_plane(const void* x, int n, int h, int w, int c, int ldx, int k, int pad, const float* wt,
                           const float* bias, int act, float* out, void* stream) {
    PAI_REQUIRE(x && wt && out && n > 0 && k >= 1 && k <= 4, "pai_conv_wide_to_plane: null pointer or k=%d", k);
    PAI_REQUIRE(v8_ok(c, x, ldx), "pai_conv_wide_to_plane: bad channels / alignment");
    const long long hw = (long long)h * w;
    return launch_wide_to_plane(x, n, h, w, c, ldx, k, pad, wt, bias, act, out, 1, hw, hw, stream);
}
int pai_conv_wide_to_planes(const void* x, int n, int h, int w, int c, int ldx, int k, int pad, const float* wt,
                            const float* bias, int act, float* out, int np, long long plane_stride, void* stream) {
    PAI_REQUIRE(x && wt && out, "pai_conv_wide_to_planes: null pointer");
    PAI_REQUIRE(np >= 1 && np <= 4, "pai_conv_wide_to_planes: plane count %d outside 1..4", np);
    PAI_REQUIRE(n > 0 && h > 0 && w > 0 && k >= 1 && k <= 4, "pai_conv_wide_to_planes: bad size or k=%d", k);
    PAI_REQUIRE(v8_ok(c, x, ldx) && planes_ok(np, plane_stride, h, w, out),
                "pai_conv_wide_to_planes: bad channels / plane stride / alignment");
    return launch_wide_to_plane(x, n, h, w, c, ldx, k, pad, wt, bias, act, out, np, np * plane_stride, plane_stride, stream);
}
int pai_conv_plane_wide_wgrad(const float* plane, const void* wide, int ldw, int n, int h, int w, int c, int k, int pad,
                              int flip, float* dw, void* stream) {
    PAI_REQUIRE(plane && wide && dw && n > 0, "pai_conv_plane_wide_wgrad: null pointer");
    const long long hw = (long long)h * w;
    return launch_plane_wide_wgrad("pai_conv_plane_wide_wgrad", plane, hw, hw, 1, wide, ldw, n, h, w, c, k, pad, flip, dw,
                                   stream);
}
int pai_conv_planes_wide_wgrad(const float* planes, int np, long long plane_stride, const void* wide, int ldw, int n,
                               int h, int w, int c, int k, int pad, int flip, float* dw, void* stream) {
    PAI_REQUIRE(planes && wide && dw, "pai_conv_planes_wide_wgrad: null pointer");
    PAI_REQUIRE(np >= 1 && np <= 4, "pai_conv_planes_wide_wgrad: plane count %d outside 1..4", np);
    PAI_REQUIRE(n > 0 && h > 0 && w > 0, "pai_conv_planes_wide_wgrad: empty input");
    PAI_REQUIRE(planes_ok(np, plane_stride, h, w, planes), "pai_conv_planes_wide_wgrad: plane stride %lld / alignment",
                plane_stride);
    return launch_plane_wide_wgrad("pai_conv_planes_wide_wgrad", planes, np * plane_stride, plane_stride, np, wide, ldw, n,
                                   h, w, c, k, pad, flip, dw, stream);
}
int pai_gconv4_3x3_fprop(const void* x, int n, int h, int w, int c, int ldx, const float* wt, const float* bias, void* y,
                         int ldy, void* stream) {
    PAI_REQUIRE(x && wt && y && n > 0, "pai_gconv4_3x3_fprop: null pointer");
    PAI_REQUIRE(v8_ok(c, x, ldx) && v8_ok(c, y, ldy) && c * 36 * 4 <= 96 * 1024, "pai_gconv4_3x3_fprop: bad channels / alignment");
    static DeviceOnce attr_once;
    const int attr_dev = current_device();
    if (attr_dev < 0) return -1;
    if (attr_once.need(attr_dev)) {
        PAI_CUDA_OK(cudaFuncSetAttribute(gconv4_fprop_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        attr_once.mark(attr_dev);
    }
    gconv4_fprop_kernel<<<ly_grid((long long)n * h * w * (c / 8)), kLyThreads, c * 36 * sizeof(float), (cudaStream_t)stream>>>(
        (const bf16*)x, n, h, w, c, ldx, wt, bias, (bf16*)y, ldy);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_gconv4_3x3_wgrad(const void* x, int ldx, const void* gy, int ldg, int n, int h, int w, int c, float* dw,
                         void* stream) {
    PAI_REQUIRE(x && gy && dw && n > 0, "pai_gconv4_3x3_wgrad: null pointer");
    PAI_REQUIRE(v8_ok(c, x, ldx) && v8_ok(c, gy, ldg) && cv_divides_block(c), "pai_gconv4_3x3_wgrad: bad channels / alignment");
    const long long ppb = kLyThreads / (c / 8);
    long long blocks = ((long long)n * h * w + ppb - 1) / ppb;
    if (blocks > 148 * 4) blocks = 148 * 4;
    gconv4_wgrad_kernel<<<dim3((int)blocks, 3), kLyThreads, 0, (cudaStream_t)stream>>>((const bf16*)x, ldx, (const bf16*)gy,
                                                                                      ldg, n, h, w, c, dw);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // extern "C"
