// fp32 check path (north star: "generator outputs within 1e-5 with the fp32 accumulate check path").
//
// Plain CUDA-core kernels on fp32 NCHW tensors in the reference's own layouts -- no bf16 rounding anywhere, one
// thread per output element, fp32 FMA accumulation in a fixed order.  They are the slow, exact twin of the
// tcgen05 path: tests run the same drop-in modules through them (pai_b200.engine.check_path()) to show that the
// index math / layer wiring reproduces the reference (models/pix2pix.py:46-111,198-216, models/wrapper.py:196-238)
// to fp32 rounding, which separates "bf16 operand noise" from "wrong arithmetic" in the 1e-2 bf16 parity bound.
// Forward and backward (data / weight / bias gradients, BatchNorm and activation backward); never used by a training
// or benchmark path.
#include "pai_common.cuh"
#include "pai_kernels.h"

namespace pai {
namespace {

__device__ __forceinline__ float check_act(float v, int act, float slope) {
    switch (act) {
        case PAI_ACT_LEAKY: return v > 0.f ? v : v * slope;
        case PAI_ACT_RELU: return fmaxf(v, 0.f);
        case PAI_ACT_TANH: return tanhf(v);
        case PAI_ACT_SIGMOID: return 1.f / (1.f + expf(-v));
        case PAI_ACT_GELU: return 0.5f * v * (1.f + erff(v * 0.70710678118654752f));
        default: return v;
    }
}

// y[n,co,oy,ox] = bias[co] + sum_{ci,ky,kx} pre(x[n,ci,oy*s-p+ky,ox*s-p+kx]) * w[co,ci-ci0,ky,kx]   (nn.Conv2d)
// with groups: ci runs over the cin/groups input channels of co's group, starting at ci0 (groups = 1: all of them).
// Acc = float: fp32 FMA chain (pai_check_conv2d_f32); Acc = double: the exact fp32 products summed in double, same order
// (pai_check_conv2d_grouped_f32).
template <typename Acc>
__global__ void check_conv2d_kernel(const float* __restrict__ x, int n, int cin, int h, int w,
                                    const float* __restrict__ wt, int cout, int k, int stride, int pad, int groups,
                                    const float* __restrict__ bias, int pre_act, float slope, int ho, int wo,
                                    float* __restrict__ y) {
    const int cin_g = cin / groups, cout_g = cout / groups;
    const long long total = (long long)n * cout * ho * wo;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int ox = (int)(i % wo);
        const int oy = (int)((i / wo) % ho);
        const int co = (int)((i / ((long long)wo * ho)) % cout);
        const int b = (int)(i / ((long long)wo * ho * cout));
        const int ci0 = (co / cout_g) * cin_g;
        Acc acc = bias != nullptr ? (Acc)bias[co] : (Acc)0;
        for (int ci = ci0; ci < ci0 + cin_g; ++ci) {
            const float* xp = x + ((size_t)b * cin + ci) * h * w;
            const float* wp = wt + ((size_t)co * cin_g + (ci - ci0)) * k * k;
            for (int ky = 0; ky < k; ++ky) {
                const int iy = oy * stride - pad + ky;
                if (iy < 0 || iy >= h) continue;
                for (int kx = 0; kx < k; ++kx) {
                    const int ix = ox * stride - pad + kx;
                    if (ix < 0 || ix >= w) continue;
                    acc = fma((Acc)check_act(xp[(size_t)iy * w + ix], pre_act, slope), (Acc)wp[ky * k + kx], acc);
                }
            }
        }
        y[i] = (float)acc;
    }
}

// y[n,co,oy,ox] = bias[co] + sum_{ci,ky,kx : oy = iy*s - p + ky} pre(x[n,ci,iy,ix]) * w[ci,co-co0,ky,kx]
// (nn.ConvTranspose2d; with groups, ci runs over the input channels of co's group)
template <typename Acc>
__global__ void check_convT2d_kernel(const float* __restrict__ x, int n, int cin, int h, int w,
                                     const float* __restrict__ wt, int cout, int k, int stride, int pad, int groups,
                                     const float* __restrict__ bias, int pre_act, float slope, int ho, int wo,
                                     float* __restrict__ y) {
    const int cin_g = cin / groups, cout_g = cout / groups;
    const long long total = (long long)n * cout * ho * wo;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int ox = (int)(i % wo);
        const int oy = (int)((i / wo) % ho);
        const int co = (int)((i / ((long long)wo * ho)) % cout);
        const int b = (int)(i / ((long long)wo * ho * cout));
        const int grp = co / cout_g, ci0 = grp * cin_g;
        Acc acc = bias != nullptr ? (Acc)bias[co] : (Acc)0;
        for (int ci = ci0; ci < ci0 + cin_g; ++ci) {
            const float* xp = x + ((size_t)b * cin + ci) * h * w;
            const float* wp = wt + ((size_t)ci * cout_g + (co - grp * cout_g)) * k * k;
            for (int ky = 0; ky < k; ++ky) {
                const int ty = oy + pad - ky;
                if (ty < 0 || ty % stride) continue;
                const int iy = ty / stride;
                if (iy >= h) continue;
                for (int kx = 0; kx < k; ++kx) {
                    const int tx = ox + pad - kx;
                    if (tx < 0 || tx % stride) continue;
                    const int ix = tx / stride;
                    if (ix >= w) continue;
                    acc = fma((Acc)check_act(xp[(size_t)iy * w + ix], pre_act, slope), (Acc)wp[ky * k + kx], acc);
                }
            }
        }
        y[i] = (float)acc;
    }
}

// nn.BatchNorm2d on fp32 NCHW, one CTA per channel.  training: biased batch variance for the normalisation, unbiased
// for running_var, running = (1 - momentum) * running + momentum * batch (models/pix2pix.py:70,106 defaults).
__global__ void check_bn_kernel(const float* __restrict__ x, int n, int c, int hw, const float* __restrict__ gamma,
                                const float* __restrict__ beta, float* __restrict__ running_mean,
                                float* __restrict__ running_var, int training, float eps, float momentum,
                                float* __restrict__ y) {
    __shared__ double red[256];
    __shared__ float s_mean, s_inv;
    const int ch = blockIdx.x, tid = threadIdx.x;
    const long long cnt = (long long)n * hw;
    if (training) {
        double s = 0.0;
        for (long long i = tid; i < cnt; i += blockDim.x) s += x[((size_t)(i / hw) * c + ch) * hw + (i % hw)];
        red[tid] = s;
        __syncthreads();
        for (int o = blockDim.x / 2; o > 0; o >>= 1) {
            if (tid < o) red[tid] += red[tid + o];
            __syncthreads();
        }
        const double mean = red[0] / (double)cnt;
        __syncthreads();
        double q = 0.0;
        for (long long i = tid; i < cnt; i += blockDim.x) {
            const double d = (double)x[((size_t)(i / hw) * c + ch) * hw + (i % hw)] - mean;
            q += d * d;
        }
        red[tid] = q;
        __syncthreads();
        for (int o = blockDim.x / 2; o > 0; o >>= 1) {
            if (tid < o) red[tid] += red[tid + o];
            __syncthreads();
        }
        if (tid == 0) {
            const double var = red[0] / (double)cnt;
            s_mean = (float)mean;
            s_inv = 1.f / sqrtf((float)var + eps);
            if (running_mean != nullptr) {
                const double unbiased = cnt > 1 ? red[0] / (double)(cnt - 1) : var;
                running_mean[ch] = (1.f - momentum) * running_mean[ch] + momentum * (float)mean;
                running_var[ch] = (1.f - momentum) * running_var[ch] + momentum * (float)unbiased;
            }
        }
    } else if (tid == 0) {
        s_mean = running_mean[ch];
        s_inv = 1.f / sqrtf(running_var[ch] + eps);
    }
    __syncthreads();
    const float mean = s_mean, inv = s_inv, g = gamma[ch], b = beta[ch];
    for (long long i = tid; i < cnt; i += blockDim.x) {
        const size_t o = ((size_t)(i / hw) * c + ch) * hw + (i % hw);
        y[o] = (x[o] - mean) * inv * g + b;
    }
}

__global__ void check_act_kernel(const float* __restrict__ x, long long count, int act, float slope, float* __restrict__ y) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x)
        y[i] = check_act(x[i], act, slope);
}

// dW of nn.Conv2d (transposed = 0, dw [cout,cin/groups,k,k]) or nn.ConvTranspose2d (transposed = 1,
// dw [cin,cout/groups,k,k]): one CTA per weight (out-channel, in-channel) pair, k*k <= 16 taps per thread, positions
// strided over the CTA; the per-thread partial sums in Acc (float: pai_check_conv2d_wgrad_f32; double, the exact fp32
// products: pai_check_conv2d_wgrad_grouped_f32), then a double tree reduction across the CTA.
//   conv : dW[co,ci,ky,kx] = sum_{b,oy,ox} g[b,co,oy,ox] * pre(x[b,ci,oy*s-p+ky,ox*s-p+kx])
//   convT: dW[ci,co,ky,kx] = sum_{b,iy,ix} pre(x[b,ci,iy,ix]) * g[b,co,iy*s-p+ky,ix*s-p+kx]
template <typename Acc>
__global__ void check_conv_wgrad_kernel(const float* __restrict__ x, int n, int cin, int h, int w,
                                        const float* __restrict__ g, int cout, int ho, int wo, int k, int stride, int pad,
                                        int groups, int pre_act, float slope, int transposed, float* __restrict__ dw) {
    __shared__ double red[64];
    const int cin_g = cin / groups, cout_g = cout / groups;
    int co, ci;
    if (transposed) {
        ci = blockIdx.x / cout_g;
        co = (ci / cin_g) * cout_g + blockIdx.x % cout_g;
    } else {
        co = blockIdx.x % cout;
        ci = (co / cout_g) * cin_g + blockIdx.x / cout;
    }
    // "small" grid = the tensor indexed directly by the loop, "big" = the one read at s*pos - p + k
    const float* small = transposed ? x : g;
    const float* big = transposed ? g : x;
    const int sc = transposed ? ci : co, sC = transposed ? cin : cout, sh = transposed ? h : ho, sw = transposed ? w : wo;
    const int bc = transposed ? co : ci, bC = transposed ? cout : cin, bh = transposed ? ho : h, bw = transposed ? wo : w;
    Acc acc[16];
    for (int t = 0; t < 16; ++t) acc[t] = (Acc)0;
    const long long cnt = (long long)n * sh * sw;
    for (long long i = threadIdx.x; i < cnt; i += blockDim.x) {
        const int px = (int)(i % sw), py = (int)((i / sw) % sh), b = (int)(i / ((long long)sw * sh));
        float sv = small[(((size_t)b * sC + sc) * sh + py) * sw + px];
        if (transposed) sv = check_act(sv, pre_act, slope);
        const float* bp = big + ((size_t)b * bC + bc) * bh * bw;
        for (int ky = 0; ky < k; ++ky) {
            const int yy = py * stride - pad + ky;
            if (yy < 0 || yy >= bh) continue;
            for (int kx = 0; kx < k; ++kx) {
                const int xx = px * stride - pad + kx;
                if (xx < 0 || xx >= bw) continue;
                float bv = bp[(size_t)yy * bw + xx];
                if (!transposed) bv = check_act(bv, pre_act, slope);
                acc[ky * k + kx] = fma((Acc)sv, (Acc)bv, acc[ky * k + kx]);
            }
        }
    }
    float* out = dw + (transposed ? ((size_t)ci * cout_g + co % cout_g) : ((size_t)co * cin_g + ci % cin_g)) * k * k;
    for (int t = 0; t < k * k; ++t) {
        red[threadIdx.x] = (double)acc[t];
        __syncthreads();
        for (int o = blockDim.x / 2; o > 0; o >>= 1) {
            if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
            __syncthreads();
        }
        if (threadIdx.x == 0) out[t] = (float)red[0];
        __syncthreads();
    }
}

// sums[ch] = sum over (n, hw) of g[n, ch, :]   (bias gradients), one CTA per channel
__global__ void check_chansum_kernel(const float* __restrict__ g, int n, int c, int hw, float* __restrict__ sums) {
    __shared__ double red[256];
    const int ch = blockIdx.x, tid = threadIdx.x;
    const long long cnt = (long long)n * hw;
    double s = 0.0;
    for (long long i = tid; i < cnt; i += blockDim.x) s += g[((size_t)(i / hw) * c + ch) * hw + (i % hw)];
    red[tid] = s;
    __syncthreads();
    for (int o = blockDim.x / 2; o > 0; o >>= 1) {
        if (tid < o) red[tid] += red[tid + o];
        __syncthreads();
    }
    if (tid == 0) sums[ch] = (float)red[0];
}

// train-mode nn.BatchNorm2d backward, one CTA per channel:
// dx = gamma * invstd * (g - mean(g) - xhat * mean(g * xhat)),  dgamma = sum g * xhat,  dbeta = sum g
__global__ void check_bn_bwd_kernel(const float* __restrict__ x, const float* __restrict__ g, int n, int c, int hw,
                                    const float* __restrict__ gamma, float eps, float* __restrict__ dx,
                                    float* __restrict__ dgamma, float* __restrict__ dbeta) {
    __shared__ double red[256];
    __shared__ double s_val[4];
    const int ch = blockIdx.x, tid = threadIdx.x;
    const long long cnt = (long long)n * hw;
    auto at = [&](long long i) { return ((size_t)(i / hw) * c + ch) * hw + (i % hw); };
    auto reduce = [&](double v, int slot) {
        red[tid] = v;
        __syncthreads();
        for (int o = blockDim.x / 2; o > 0; o >>= 1) {
            if (tid < o) red[tid] += red[tid + o];
            __syncthreads();
        }
        if (tid == 0) s_val[slot] = red[0];
        __syncthreads();
    };
    double s = 0.0;
    for (long long i = tid; i < cnt; i += blockDim.x) s += x[at(i)];
    reduce(s, 0);
    const double mean = s_val[0] / (double)cnt;
    double q = 0.0;
    for (long long i = tid; i < cnt; i += blockDim.x) {
        const double d = (double)x[at(i)] - mean;
        q += d * d;
    }
    reduce(q, 1);
    const float inv = 1.f / sqrtf((float)(s_val[1] / (double)cnt) + eps);
    double sg = 0.0, sgx = 0.0;
    for (long long i = tid; i < cnt; i += blockDim.x) {
        const size_t o = at(i);
        const double xh = ((double)x[o] - mean) * (double)inv;
        sg += g[o];
        sgx += (double)g[o] * xh;
    }
    reduce(sg, 2);
    reduce(sgx, 3);
    const double mg = s_val[2] / (double)cnt, mgx = s_val[3] / (double)cnt;
    const float gm = gamma[ch];
    for (long long i = tid; i < cnt; i += blockDim.x) {
        const size_t o = at(i);
        const double xh = ((double)x[o] - mean) * (double)inv;
        dx[o] = (float)((double)gm * (double)inv * ((double)g[o] - mg - xh * mgx));
    }
    if (tid == 0) {
        dgamma[ch] = (float)s_val[3];
        dbeta[ch] = (float)s_val[2];
    }
}

// dx = g * act'(x) with x the value the activation was applied to
__global__ void check_act_bwd_kernel(const float* __restrict__ x, const float* __restrict__ g, long long count, int act,
                                     float slope, float* __restrict__ dx) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
        const float v = x[i];
        float d = 1.f;
        if (act == PAI_ACT_LEAKY) d = v > 0.f ? 1.f : slope;
        else if (act == PAI_ACT_RELU) d = v > 0.f ? 1.f : 0.f;
        else if (act == PAI_ACT_TANH) { const float t = tanhf(v); d = 1.f - t * t; }
        else if (act == PAI_ACT_SIGMOID) { const float s = 1.f / (1.f + expf(-v)); d = s * (1.f - s); }
        else if (act == PAI_ACT_GELU)     // d/dv [v * Phi(v)] = Phi(v) + v * phi(v)
            d = 0.5f * (1.f + erff(v * 0.70710678118654752f)) + v * 0.39894228040143268f * expf(-0.5f * v * v);
        dx[i] = g[i] * d;
    }
}

// ---- resampling (fp32 NCHW, all n*c planes of [h, w] alike)
// nn.MaxPool2d(2): the first maximum of the 2x2 window in row-major order wins (torch: v > max || isnan(v))
__device__ __forceinline__ int check_argmax4(const float* p, int w) {
    int idx = 0;
    float m = p[0];
    const float v[3] = {p[1], p[w], p[w + 1]};
    for (int t = 0; t < 3; ++t)
        if (v[t] > m || isnan(v[t])) { m = v[t]; idx = t + 1; }
    return idx;
}

__global__ void check_maxpool2_kernel(const float* __restrict__ x, long long planes, int h, int w, int ho, int wo,
                                      float* __restrict__ y) {
    const long long total = planes * ho * wo;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int ox = (int)(i % wo), oy = (int)((i / wo) % ho);
        const float* p = x + (size_t)(i / ((long long)wo * ho)) * h * w + (size_t)(2 * oy) * w + 2 * ox;
        const int a = check_argmax4(p, w);
        y[i] = p[(a >> 1) * w + (a & 1)];
    }
}

// one thread per INPUT element: it receives g of its window iff it is that window's argmax (no atomics)
__global__ void check_maxpool2_bwd_kernel(const float* __restrict__ x, const float* __restrict__ g, long long planes, int h,
                                          int w, int ho, int wo, float* __restrict__ dx) {
    const long long total = planes * h * w;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int ix = (int)(i % w), iy = (int)((i / w) % h);
        const long long pl = i / ((long long)w * h);
        const int oy = iy >> 1, ox = ix >> 1;
        float d = 0.f;
        if (oy < ho && ox < wo) {
            const int a = check_argmax4(x + (size_t)pl * h * w + (size_t)(2 * oy) * w + 2 * ox, w);
            if (a == ((iy & 1) << 1 | (ix & 1))) d = g[((size_t)pl * ho + oy) * wo + ox];
        }
        dx[i] = d;
    }
}

// nn.Upsample(scale_factor=2) (nearest): y[2h, 2w]
__global__ void check_upsample2_kernel(const float* __restrict__ x, long long planes, int h, int w, float* __restrict__ y) {
    const long long total = planes * 4 * h * w;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int ox = (int)(i % (2 * w)), oy = (int)((i / (2 * w)) % (2 * h));
        y[i] = x[(size_t)(i / (4LL * w * h)) * h * w + (size_t)(oy >> 1) * w + (ox >> 1)];
    }
}

// dx[iy,ix] = g[2iy,2ix] + g[2iy,2ix+1] + g[2iy+1,2ix] + g[2iy+1,2ix+1], summed in that order
__global__ void check_upsample2_bwd_kernel(const float* __restrict__ g, long long planes, int h, int w, float* __restrict__ dx) {
    const long long total = planes * h * w;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int ix = (int)(i % w), iy = (int)((i / w) % h);
        const float* p = g + (size_t)(i / ((long long)w * h)) * 4 * h * w + (size_t)(2 * iy) * (2 * w) + 2 * ix;
        dx[i] = ((p[0] + p[1]) + p[2 * w]) + p[2 * w + 1];
    }
}

// ---- row-major [m, d] layers of the ViT bottleneck
__device__ double check_block_sum(double v, double* red) {       // blockDim.x == 256; every thread gets the sum
    red[threadIdx.x] = v;
    __syncthreads();
    for (int o = blockDim.x / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    const double s = red[0];
    __syncthreads();
    return s;
}

// nn.LayerNorm(d) over each row, one CTA per row: mean and biased variance in double, y = (x - mean) * rstd * g + b
__global__ void check_layernorm_kernel(const float* __restrict__ x, int d, const float* __restrict__ gamma,
                                       const float* __restrict__ beta, float eps, float* __restrict__ y,
                                       float* __restrict__ mean_out, float* __restrict__ rstd_out) {
    __shared__ double red[256];
    const float* xr = x + (size_t)blockIdx.x * d;
    double s = 0.0;
    for (int j = threadIdx.x; j < d; j += blockDim.x) s += xr[j];
    const double mean = check_block_sum(s, red) / d;
    double q = 0.0;
    for (int j = threadIdx.x; j < d; j += blockDim.x) {
        const double t = (double)xr[j] - mean;
        q += t * t;
    }
    const float var = (float)(check_block_sum(q, red) / d);
    const float mf = (float)mean, inv = 1.f / sqrtf(var + eps);
    for (int j = threadIdx.x; j < d; j += blockDim.x) y[(size_t)blockIdx.x * d + j] = (xr[j] - mf) * inv * gamma[j] + beta[j];
    if (threadIdx.x == 0) {
        mean_out[blockIdx.x] = mf;
        rstd_out[blockIdx.x] = inv;
    }
}

// dx = rstd * (g*gamma - mean(g*gamma) - xhat * mean(g*gamma*xhat)) per row (one CTA per row, double reductions)
__global__ void check_layernorm_bwd_kernel(const float* __restrict__ x, const float* __restrict__ g, int d,
                                           const float* __restrict__ gamma, const float* __restrict__ mean,
                                           const float* __restrict__ rstd, float* __restrict__ dx) {
    __shared__ double red[256];
    const size_t r = (size_t)blockIdx.x * d;
    const double mu = mean[blockIdx.x], rs = rstd[blockIdx.x];
    double a = 0.0, b = 0.0;
    for (int j = threadIdx.x; j < d; j += blockDim.x) {
        const double gg = (double)g[r + j] * gamma[j];
        a += gg;
        b += gg * (((double)x[r + j] - mu) * rs);
    }
    const double ma = check_block_sum(a, red) / d, mb = check_block_sum(b, red) / d;
    for (int j = threadIdx.x; j < d; j += blockDim.x) {
        const double xh = ((double)x[r + j] - mu) * rs;
        dx[r + j] = (float)(rs * ((double)g[r + j] * gamma[j] - ma - xh * mb));
    }
}

// dgamma[j] = sum_r g[r,j] * xhat[r,j],  dbeta[j] = sum_r g[r,j]: one thread per column, rows in order, in double
__global__ void check_layernorm_wgrad_kernel(const float* __restrict__ x, const float* __restrict__ g, int m, int d,
                                             const float* __restrict__ mean, const float* __restrict__ rstd,
                                             float* __restrict__ dgamma, float* __restrict__ dbeta) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= d) return;
    double sg = 0.0, sgx = 0.0;
    for (int r = 0; r < m; ++r) {
        const double gv = g[(size_t)r * d + j];
        sg += gv;
        sgx += gv * (((double)x[(size_t)r * d + j] - (double)mean[r]) * (double)rstd[r]);
    }
    dgamma[j] = (float)sgx;
    dbeta[j] = (float)sg;
}

// nn.Linear (the exact fp32 products summed in double, in order), w [out, in]:  transpose = 0: y[r,o] = b[o] + sum_i x[r,i] w[o,i]   (x [m,in],  y [m,out])
//                          transpose = 1: y[r,i] = sum_o x[r,o] w[o,i]            (x [m,out], y [m,in]: the data gradient)
__global__ void check_linear_kernel(const float* __restrict__ x, int m, int in, int out, const float* __restrict__ wt,
                                    const float* __restrict__ bias, int transpose, float* __restrict__ y) {
    const int ycols = transpose ? in : out, red = transpose ? out : in;
    const long long total = (long long)m * ycols;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % ycols);
        const float* xr = x + (size_t)(i / ycols) * red;
        double acc = bias != nullptr ? bias[c] : 0.0;
        if (transpose)
            for (int o = 0; o < red; ++o) acc = fma((double)xr[o], (double)wt[(size_t)o * in + c], acc);
        else
            for (int k = 0; k < red; ++k) acc = fma((double)xr[k], (double)wt[(size_t)c * in + k], acc);
        y[i] = (float)acc;
    }
}

// dW[o,i] = sum_r g[r,o] x[r,i] (one thread per weight element, rows in order, in double); dbias[o] = sum_r g[r,o]
__global__ void check_linear_wgrad_kernel(const float* __restrict__ x, const float* __restrict__ g, int m, int in, int out,
                                          float* __restrict__ dw, float* __restrict__ dbias) {
    const long long total = (long long)out * in;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int o = (int)(t / in), i = (int)(t % in);
        double acc = 0.0;
        for (int r = 0; r < m; ++r) acc += (double)g[(size_t)r * out + o] * (double)x[(size_t)r * in + i];
        dw[t] = (float)acc;
        if (dbias != nullptr && i == 0) {
            double s = 0.0;
            for (int r = 0; r < m; ++r) s += g[(size_t)r * out + o];
            dbias[o] = (float)s;
        }
    }
}

// ---- multi-head attention over the sequence axis of qkv [S*B, 3E] (row = s*B + b; Q | K | V; head h = columns
// [h*hd, (h+1)*hd) of each), the layout of the tensor-core path (csrc/transformer.cu).  probs [B*H, S, S].
// One thread per (b*H + h, query i): scores summed in double, softmax with max subtraction, the normaliser in double.
__global__ void check_attn_probs_kernel(const float* __restrict__ qkv, int S, int B, int H, int hd, float scale,
                                        float* __restrict__ probs) {
    const long long total = (long long)B * H * S;
    const int E = H * hd;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(t % S), bh = (int)(t / S), b = bh / H, h = bh % H;
        const float* q = qkv + ((size_t)i * B + b) * 3 * E + h * hd;
        float* p = probs + (size_t)t * S;
        float mx = -INFINITY;
        for (int j = 0; j < S; ++j) {
            const float* k = qkv + ((size_t)j * B + b) * 3 * E + E + h * hd;
            double acc = 0.0;
            for (int c = 0; c < hd; ++c) acc = fma((double)q[c], (double)k[c], acc);
            p[j] = (float)acc * scale;
            mx = fmaxf(mx, p[j]);
        }
        double sum = 0.0;
        for (int j = 0; j < S; ++j) {
            p[j] = expf(p[j] - mx);
            sum += p[j];
        }
        for (int j = 0; j < S; ++j) p[j] = (float)(p[j] / sum);
    }
}

// out[i*B+b, h*hd+c] = sum_j P[bh,i,j] V[j*B+b, h*hd+c]
__global__ void check_attn_out_kernel(const float* __restrict__ qkv, const float* __restrict__ probs, int S, int B, int H,
                                      int hd, float* __restrict__ out) {
    const int E = H * hd;
    const long long total = (long long)S * B * E;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int col = (int)(t % E), row = (int)(t / E), i = row / B, b = row % B, h = col / hd;
        const float* p = probs + (((size_t)b * H + h) * S + i) * S;
        double acc = 0.0;
        for (int j = 0; j < S; ++j) acc = fma((double)p[j], (double)qkv[((size_t)j * B + b) * 3 * E + 2 * E + col], acc);
        out[t] = (float)acc;
    }
}

// dS[bh,i,j] = P[i,j] * (dP[i,j] - sum_j' P[i,j'] dP[i,j']) with dP[i,j] = dout[i] . V[j]; one thread per (bh, i)
__global__ void check_attn_ds_kernel(const float* __restrict__ qkv, const float* __restrict__ probs,
                                     const float* __restrict__ dout, int S, int B, int H, int hd, float* __restrict__ ds) {
    const long long total = (long long)B * H * S;
    const int E = H * hd;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(t % S), bh = (int)(t / S), b = bh / H, h = bh % H;
        const float* go = dout + ((size_t)i * B + b) * E + h * hd;
        const float* p = probs + (size_t)t * S;
        float* d = ds + (size_t)t * S;
        double dot = 0.0;
        for (int j = 0; j < S; ++j) {
            const float* v = qkv + ((size_t)j * B + b) * 3 * E + 2 * E + h * hd;
            double acc = 0.0;
            for (int c = 0; c < hd; ++c) acc = fma((double)go[c], (double)v[c], acc);
            d[j] = (float)acc;
            dot += (double)p[j] * acc;
        }
        for (int j = 0; j < S; ++j) d[j] = p[j] * (float)((double)d[j] - dot);
    }
}

// d(qkv), one thread per element:  dQ[i] = scale sum_j dS[i,j] K[j],  dK[j] = scale sum_i dS[i,j] Q[i],
// dV[j] = sum_i P[i,j] dout[i]
__global__ void check_attn_dqkv_kernel(const float* __restrict__ qkv, const float* __restrict__ probs,
                                       const float* __restrict__ ds, const float* __restrict__ dout, int S, int B, int H,
                                       int hd, float scale, float* __restrict__ dqkv) {
    const int E = H * hd;
    const long long total = (long long)S * B * 3 * E;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int col3 = (int)(t % (3 * E)), row = (int)(t / (3 * E)), s = row / B, b = row % B;
        const int part = col3 / E, col = col3 % E, h = col / hd;
        const size_t bh = (size_t)b * H + h;
        double acc = 0.0;
        if (part == 0) {
            for (int j = 0; j < S; ++j) acc = fma((double)ds[(bh * S + s) * S + j], (double)qkv[((size_t)j * B + b) * 3 * E + E + col], acc);
            acc *= scale;
        } else if (part == 1) {
            for (int i = 0; i < S; ++i) acc = fma((double)ds[(bh * S + i) * S + s], (double)qkv[((size_t)i * B + b) * 3 * E + col], acc);
            acc *= scale;
        } else {
            for (int i = 0; i < S; ++i) acc = fma((double)probs[(bh * S + i) * S + s], (double)dout[((size_t)i * B + b) * E + col], acc);
        }
        dqkv[t] = (float)acc;
    }
}

int grid_for(long long total) {
    long long g = (total + 255) / 256;
    return (int)(g < 148 * 32 ? (g > 0 ? g : 1) : 148 * 32);
}

template <typename Acc>
int check_conv_launch(const float* x, int n, int cin, int h, int w, const float* wt, int cout, int k, int stride, int pad,
                      int groups, int ho, int wo, const float* bias, int pre_act, float slope, int transposed, float* y,
                      cudaStream_t st) {
    const long long total = (long long)n * cout * ho * wo;
    if (transposed)
        check_convT2d_kernel<Acc><<<grid_for(total), 256, 0, st>>>(x, n, cin, h, w, wt, cout, k, stride, pad, groups, bias,
                                                                  pre_act, slope, ho, wo, y);
    else
        check_conv2d_kernel<Acc><<<grid_for(total), 256, 0, st>>>(x, n, cin, h, w, wt, cout, k, stride, pad, groups, bias,
                                                                 pre_act, slope, ho, wo, y);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace
}  // namespace pai

using namespace pai;

extern "C" {

int pai_check_conv2d_grouped_f32(const float* x, int n, int cin, int h, int w, const float* wt, int cout, int k,
                                 int stride, int pad, int groups, int out_pad, const float* bias, int pre_act, float slope,
                                 int transposed, float* y, void* stream) {
    PAI_REQUIRE(x && wt && y, "pai_check_conv2d_grouped_f32: null pointer");
    PAI_REQUIRE(n >= 0 && cin > 0 && cout > 0 && h > 0 && w > 0 && k > 0 && stride > 0 && pad >= 0,
                "pai_check_conv2d_grouped_f32: bad shape n=%d cin=%d cout=%d %dx%d k=%d stride=%d pad=%d", n, cin, cout, h, w,
                k, stride, pad);
    PAI_REQUIRE(groups > 0 && cin % groups == 0 && cout % groups == 0,
                "pai_check_conv2d_grouped_f32: groups=%d must divide cin=%d and cout=%d", groups, cin, cout);
    PAI_REQUIRE(out_pad >= 0 && (transposed ? out_pad < stride : out_pad == 0),
                "pai_check_conv2d_grouped_f32: output padding %d (transposed only, < stride %d)", out_pad, stride);
    const int ho = transposed ? (h - 1) * stride - 2 * pad + k + out_pad : (h + 2 * pad - k) / stride + 1;
    const int wo = transposed ? (w - 1) * stride - 2 * pad + k + out_pad : (w + 2 * pad - k) / stride + 1;
    PAI_REQUIRE(ho > 0 && wo > 0, "pai_check_conv2d_grouped_f32: empty output (%dx%d)", ho, wo);
    if (n == 0) return 0;
    return check_conv_launch<double>(x, n, cin, h, w, wt, cout, k, stride, pad, groups, ho, wo, bias, pre_act, slope,
                                     transposed, y, (cudaStream_t)stream);
}

int pai_check_conv2d_f32(const float* x, int n, int cin, int h, int w, const float* wt, int cout, int k, int stride,
                         int pad, const float* bias, int pre_act, float slope, int transposed, float* y, void* stream) {
    PAI_REQUIRE(x && wt && y, "pai_check_conv2d_f32: null pointer");
    PAI_REQUIRE(n >= 0 && cin > 0 && cout > 0 && h > 0 && w > 0 && k > 0 && stride > 0 && pad >= 0,
                "pai_check_conv2d_f32: bad shape n=%d cin=%d cout=%d %dx%d k=%d stride=%d pad=%d", n, cin, cout, h, w, k,
                stride, pad);
    const int ho = transposed ? (h - 1) * stride - 2 * pad + k : (h + 2 * pad - k) / stride + 1;
    const int wo = transposed ? (w - 1) * stride - 2 * pad + k : (w + 2 * pad - k) / stride + 1;
    PAI_REQUIRE(ho > 0 && wo > 0, "pai_check_conv2d_f32: empty output (%dx%d)", ho, wo);
    if (n == 0) return 0;
    return check_conv_launch<float>(x, n, cin, h, w, wt, cout, k, stride, pad, 1, ho, wo, bias, pre_act, slope, transposed,
                                    y, (cudaStream_t)stream);
}

int pai_check_batchnorm_f32(const float* x, int n, int c, int hw, const float* gamma, const float* beta,
                            float* running_mean, float* running_var, int training, float eps, float momentum, float* y,
                            void* stream) {
    PAI_REQUIRE(x && gamma && beta && y, "pai_check_batchnorm_f32: null pointer");
    PAI_REQUIRE(training || (running_mean && running_var), "pai_check_batchnorm_f32: eval mode needs running statistics");
    PAI_REQUIRE(n >= 0 && c > 0 && hw > 0, "pai_check_batchnorm_f32: bad shape");
    if (n == 0) return 0;
    check_bn_kernel<<<c, 256, 0, (cudaStream_t)stream>>>(x, n, c, hw, gamma, beta, running_mean, running_var, training,
                                                        eps, momentum, y);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_check_conv2d_wgrad_grouped_f32(const float* x, int n, int cin, int h, int w, const float* g, int cout, int k,
                                       int stride, int pad, int groups, int out_pad, int pre_act, float slope, int transposed,
                                       float* dw, float* dbias, void* stream) {
    PAI_REQUIRE(x && g && dw, "pai_check_conv2d_wgrad_grouped_f32: null pointer");
    PAI_REQUIRE(n > 0 && cin > 0 && cout > 0 && h > 0 && w > 0 && k > 0 && k <= 4 && stride > 0 && pad >= 0,
                "pai_check_conv2d_wgrad_grouped_f32: bad shape n=%d cin=%d cout=%d %dx%d k=%d stride=%d pad=%d", n, cin, cout,
                h, w, k, stride, pad);
    PAI_REQUIRE(groups > 0 && cin % groups == 0 && cout % groups == 0,
                "pai_check_conv2d_wgrad_grouped_f32: groups=%d must divide cin=%d and cout=%d", groups, cin, cout);
    PAI_REQUIRE(out_pad >= 0 && (transposed ? out_pad < stride : out_pad == 0),
                "pai_check_conv2d_wgrad_grouped_f32: output padding %d (transposed only, < stride %d)", out_pad, stride);
    const int ho = transposed ? (h - 1) * stride - 2 * pad + k + out_pad : (h + 2 * pad - k) / stride + 1;
    const int wo = transposed ? (w - 1) * stride - 2 * pad + k + out_pad : (w + 2 * pad - k) / stride + 1;
    PAI_REQUIRE(ho > 0 && wo > 0, "pai_check_conv2d_wgrad_grouped_f32: empty output (%dx%d)", ho, wo);
    cudaStream_t st = (cudaStream_t)stream;
    check_conv_wgrad_kernel<double><<<cin / groups * cout, 64, 0, st>>>(x, n, cin, h, w, g, cout, ho, wo, k, stride, pad, groups,
                                                                pre_act, slope, transposed, dw);
    PAI_CUDA_OK(cudaGetLastError());
    if (dbias != nullptr) {
        check_chansum_kernel<<<cout, 256, 0, st>>>(g, n, cout, ho * wo, dbias);
        PAI_CUDA_OK(cudaGetLastError());
    }
    return 0;
}

int pai_check_conv2d_wgrad_f32(const float* x, int n, int cin, int h, int w, const float* g, int cout, int k, int stride,
                               int pad, int pre_act, float slope, int transposed, float* dw, float* dbias, void* stream) {
    PAI_REQUIRE(x && g && dw, "pai_check_conv2d_wgrad_f32: null pointer");
    PAI_REQUIRE(n > 0 && cin > 0 && cout > 0 && k > 0 && k <= 4 && stride > 0 && pad >= 0, "pai_check_conv2d_wgrad_f32: bad shape");
    const int ho = transposed ? (h - 1) * stride - 2 * pad + k : (h + 2 * pad - k) / stride + 1;
    const int wo = transposed ? (w - 1) * stride - 2 * pad + k : (w + 2 * pad - k) / stride + 1;
    cudaStream_t st = (cudaStream_t)stream;
    check_conv_wgrad_kernel<float><<<cin * cout, 64, 0, st>>>(x, n, cin, h, w, g, cout, ho, wo, k, stride, pad, 1, pre_act, slope,
                                                       transposed, dw);
    PAI_CUDA_OK(cudaGetLastError());
    if (dbias != nullptr) {
        check_chansum_kernel<<<cout, 256, 0, st>>>(g, n, cout, ho * wo, dbias);
        PAI_CUDA_OK(cudaGetLastError());
    }
    return 0;
}

int pai_check_batchnorm_bwd_f32(const float* x, const float* g, int n, int c, int hw, const float* gamma, float eps,
                                float* dx, float* dgamma, float* dbeta, void* stream) {
    PAI_REQUIRE(x && g && gamma && dx && dgamma && dbeta && n > 0 && c > 0 && hw > 0, "pai_check_batchnorm_bwd_f32: bad arguments");
    check_bn_bwd_kernel<<<c, 256, 0, (cudaStream_t)stream>>>(x, g, n, c, hw, gamma, eps, dx, dgamma, dbeta);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_check_act_bwd_f32(const float* x, const float* g, long long count, int act, float slope, float* dx, void* stream) {
    PAI_REQUIRE(x && g && dx && count >= 0, "pai_check_act_bwd_f32: bad arguments");
    if (count == 0) return 0;
    check_act_bwd_kernel<<<grid_for(count), 256, 0, (cudaStream_t)stream>>>(x, g, count, act, slope, dx);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_check_act_f32(const float* x, long long count, int act, float slope, float* y, void* stream) {
    PAI_REQUIRE(x && y && count >= 0, "pai_check_act_f32: bad arguments");
    if (count == 0) return 0;
    check_act_kernel<<<grid_for(count), 256, 0, (cudaStream_t)stream>>>(x, count, act, slope, y);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_check_maxpool2_f32(const float* x, int n, int c, int h, int w, float* y, void* stream) {
    PAI_REQUIRE(x && y, "pai_check_maxpool2_f32: null pointer");
    PAI_REQUIRE(n >= 0 && c > 0 && h >= 2 && w >= 2, "pai_check_maxpool2_f32: bad shape n=%d c=%d %dx%d", n, c, h, w);
    const long long total = (long long)n * c * (h / 2) * (w / 2);
    if (total == 0) return 0;
    check_maxpool2_kernel<<<grid_for(total), 256, 0, (cudaStream_t)stream>>>(x, (long long)n * c, h, w, h / 2, w / 2, y);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_check_maxpool2_bwd_f32(const float* x, const float* g, int n, int c, int h, int w, float* dx, void* stream) {
    PAI_REQUIRE(x && g && dx, "pai_check_maxpool2_bwd_f32: null pointer");
    PAI_REQUIRE(n >= 0 && c > 0 && h >= 2 && w >= 2, "pai_check_maxpool2_bwd_f32: bad shape n=%d c=%d %dx%d", n, c, h, w);
    const long long total = (long long)n * c * h * w;
    if (total == 0) return 0;
    check_maxpool2_bwd_kernel<<<grid_for(total), 256, 0, (cudaStream_t)stream>>>(x, g, (long long)n * c, h, w, h / 2, w / 2,
                                                                                 dx);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_check_upsample2_f32(const float* x, int n, int c, int h, int w, float* y, void* stream) {
    PAI_REQUIRE(x && y, "pai_check_upsample2_f32: null pointer");
    PAI_REQUIRE(n >= 0 && c > 0 && h > 0 && w > 0, "pai_check_upsample2_f32: bad shape n=%d c=%d %dx%d", n, c, h, w);
    const long long total = 4LL * n * c * h * w;
    if (total == 0) return 0;
    check_upsample2_kernel<<<grid_for(total), 256, 0, (cudaStream_t)stream>>>(x, (long long)n * c, h, w, y);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_check_upsample2_bwd_f32(const float* g, int n, int c, int h, int w, float* dx, void* stream) {
    PAI_REQUIRE(g && dx, "pai_check_upsample2_bwd_f32: null pointer");
    PAI_REQUIRE(n >= 0 && c > 0 && h > 0 && w > 0, "pai_check_upsample2_bwd_f32: bad shape n=%d c=%d %dx%d", n, c, h, w);
    const long long total = (long long)n * c * h * w;
    if (total == 0) return 0;
    check_upsample2_bwd_kernel<<<grid_for(total), 256, 0, (cudaStream_t)stream>>>(g, (long long)n * c, h, w, dx);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_check_layernorm_f32(const float* x, int m, int d, const float* gamma, const float* beta, float eps, float* y,
                            float* mean, float* rstd, void* stream) {
    PAI_REQUIRE(x && gamma && beta && y && mean && rstd, "pai_check_layernorm_f32: null pointer");
    PAI_REQUIRE(m >= 0 && d > 0 && eps >= 0.f, "pai_check_layernorm_f32: bad shape m=%d d=%d", m, d);
    if (m == 0) return 0;
    check_layernorm_kernel<<<m, 256, 0, (cudaStream_t)stream>>>(x, d, gamma, beta, eps, y, mean, rstd);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_check_layernorm_bwd_f32(const float* x, const float* g, int m, int d, const float* gamma, const float* mean,
                                const float* rstd, float* dx, float* dgamma, float* dbeta, void* stream) {
    PAI_REQUIRE(x && g && gamma && mean && rstd && dx && dgamma && dbeta, "pai_check_layernorm_bwd_f32: null pointer");
    PAI_REQUIRE(m > 0 && d > 0, "pai_check_layernorm_bwd_f32: bad shape m=%d d=%d", m, d);
    cudaStream_t st = (cudaStream_t)stream;
    check_layernorm_bwd_kernel<<<m, 256, 0, st>>>(x, g, d, gamma, mean, rstd, dx);
    PAI_CUDA_OK(cudaGetLastError());
    check_layernorm_wgrad_kernel<<<(d + 255) / 256, 256, 0, st>>>(x, g, m, d, mean, rstd, dgamma, dbeta);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_check_linear_f32(const float* x, int m, int in, int out, const float* w, const float* bias, int transpose, float* y,
                         void* stream) {
    PAI_REQUIRE(x && w && y, "pai_check_linear_f32: null pointer");
    PAI_REQUIRE(m >= 0 && in > 0 && out > 0, "pai_check_linear_f32: bad shape m=%d in=%d out=%d", m, in, out);
    PAI_REQUIRE(!(transpose && bias), "pai_check_linear_f32: the transposed product (data gradient) takes no bias");
    const long long total = (long long)m * (transpose ? in : out);
    if (total == 0) return 0;
    check_linear_kernel<<<grid_for(total), 256, 0, (cudaStream_t)stream>>>(x, m, in, out, w, bias, transpose, y);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_check_linear_wgrad_f32(const float* x, const float* g, int m, int in, int out, float* dw, float* dbias,
                               void* stream) {
    PAI_REQUIRE(x && g && dw, "pai_check_linear_wgrad_f32: null pointer");
    PAI_REQUIRE(m > 0 && in > 0 && out > 0, "pai_check_linear_wgrad_f32: bad shape m=%d in=%d out=%d", m, in, out);
    check_linear_wgrad_kernel<<<grid_for((long long)out * in), 256, 0, (cudaStream_t)stream>>>(x, g, m, in, out, dw, dbias);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_check_attention_f32(const float* qkv, int s, int b, int heads, int head_dim, float* probs, float* out,
                            void* stream) {
    PAI_REQUIRE(qkv && probs && out, "pai_check_attention_f32: null pointer");
    PAI_REQUIRE(s > 0 && b > 0 && heads > 0 && head_dim > 0,
                "pai_check_attention_f32: bad shape s=%d b=%d heads=%d head_dim=%d", s, b, heads, head_dim);
    cudaStream_t st = (cudaStream_t)stream;
    const long long rows = (long long)b * heads * s;
    check_attn_probs_kernel<<<grid_for(rows), 256, 0, st>>>(qkv, s, b, heads, head_dim, 1.f / sqrtf((float)head_dim), probs);
    PAI_CUDA_OK(cudaGetLastError());
    check_attn_out_kernel<<<grid_for(rows * head_dim), 256, 0, st>>>(qkv, probs, s, b, heads, head_dim, out);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

int pai_check_attention_bwd_f32(const float* qkv, const float* probs, const float* dout, int s, int b, int heads,
                                int head_dim, float* ds_work, float* dqkv, void* stream) {
    PAI_REQUIRE(qkv && probs && dout && ds_work && dqkv, "pai_check_attention_bwd_f32: null pointer");
    PAI_REQUIRE(s > 0 && b > 0 && heads > 0 && head_dim > 0,
                "pai_check_attention_bwd_f32: bad shape s=%d b=%d heads=%d head_dim=%d", s, b, heads, head_dim);
    cudaStream_t st = (cudaStream_t)stream;
    const long long rows = (long long)b * heads * s;
    check_attn_ds_kernel<<<grid_for(rows), 256, 0, st>>>(qkv, probs, dout, s, b, heads, head_dim, ds_work);
    PAI_CUDA_OK(cudaGetLastError());
    check_attn_dqkv_kernel<<<grid_for(rows * 3 * head_dim), 256, 0, st>>>(qkv, probs, ds_work, dout, s, b, heads, head_dim,
                                                                          1.f / sqrtf((float)head_dim), dqkv);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // extern "C"
