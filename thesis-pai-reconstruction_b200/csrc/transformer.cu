// Kernels of the Trans U-Net's ViT bottleneck (models/trans_unet.py:120-175): nn.LayerNorm,
// nn.TransformerEncoderLayer(d, 8 heads, d_ff=2048, activation="gelu", post-norm) stacked 12 times.
// The Linear layers run on the tensor-core pointwise GEMM (igemm.cu); here are the row-wise and attention parts.
//
// Tokens are rows of a [m, d] bf16 matrix.  The reference builds the encoder layer WITHOUT batch_first and feeds
// it [n, patches, d], so self-attention runs over the BATCH axis: sequence length S = n (images of the batch on
// this GPU), "batch" B = patches (SURVEY.md Q4).  Row index = s * B + b.
#include "pai_common.cuh"
#include "pai_dropout.cuh"
#include "pai_kernels.h"

namespace pai {

__device__ __forceinline__ float block_sum(float v, float* red /* [32] */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float t = 0.f;
    for (int i = 0; i < nw; ++i) t += red[i];
    return t;
}

// ---- LayerNorm over the last dimension: one CTA per row --------------------------------------
__global__ void __launch_bounds__(256)
layernorm_fwd_kernel(const __nv_bfloat16* __restrict__ x, int d, const float* __restrict__ gamma,
                     const float* __restrict__ beta, float eps, __nv_bfloat16* __restrict__ y,
                     float* __restrict__ mean, float* __restrict__ rstd) {
    __shared__ float red[32];
    const long long row = blockIdx.x;
    const __nv_bfloat16* xr = x + row * d;
    float s = 0.f;
    for (int i = threadIdx.x; i < d; i += blockDim.x) s += __bfloat162float(xr[i]);
    const float mu = block_sum(s, red) / d;
    float q = 0.f;
    for (int i = threadIdx.x; i < d; i += blockDim.x) {
        const float c = __bfloat162float(xr[i]) - mu;
        q = fmaf(c, c, q);
    }
    const float rs = rsqrtf(block_sum(q, red) / d + eps);
    for (int i = threadIdx.x; i < d; i += blockDim.x)
        y[row * d + i] = __float2bfloat16_rn((__bfloat162float(xr[i]) - mu) * rs * gamma[i] + beta[i]);
    if (threadIdx.x == 0) {
        mean[row] = mu;
        rstd[row] = rs;
    }
}
// dx = rstd * (g*gamma - mean(g*gamma) - xhat * mean(g*gamma*xhat))
__global__ void __launch_bounds__(256)
layernorm_bwd_dx_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ g, int d,
                        const float* __restrict__ gamma, const float* __restrict__ mean,
                        const float* __restrict__ rstd, __nv_bfloat16* __restrict__ dx) {
    __shared__ float red[32];
    const long long row = blockIdx.x;
    const float mu = mean[row], rs = rstd[row];
    float a = 0.f, b = 0.f;
    for (int i = threadIdx.x; i < d; i += blockDim.x) {
        const float gg = __bfloat162float(g[row * d + i]) * gamma[i];
        const float xh = (__bfloat162float(x[row * d + i]) - mu) * rs;
        a += gg;
        b = fmaf(gg, xh, b);
    }
    const float ma = block_sum(a, red) / d;
    const float mb = block_sum(b, red) / d;
    for (int i = threadIdx.x; i < d; i += blockDim.x) {
        const float gg = __bfloat162float(g[row * d + i]) * gamma[i];
        const float xh = (__bfloat162float(x[row * d + i]) - mu) * rs;
        dx[row * d + i] = __float2bfloat16_rn(rs * (gg - ma - xh * mb));
    }
}
// dgamma[i] = sum_rows g*xhat, dbeta[i] = sum_rows g: thread <-> column, rows split over blockIdx.y
__global__ void __launch_bounds__(256)
layernorm_bwd_affine_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ g, long long m, int d,
                            const float* __restrict__ mean, const float* __restrict__ rstd, float* __restrict__ dgamma,
                            float* __restrict__ dbeta) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= d) return;
    float a = 0.f, b = 0.f;
    for (long long r = blockIdx.y; r < m; r += gridDim.y) {
        const float gg = __bfloat162float(g[r * d + col]);
        a = fmaf(gg, (__bfloat162float(x[r * d + col]) - mean[r]) * rstd[r], a);
        b += gg;
    }
    atomicAdd(dgamma + col, a);
    atomicAdd(dbeta + col, b);
}

// ---- GELU (exact, erf) -------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gelu_fwd_kernel(const __nv_bfloat16* __restrict__ x, long long n, __nv_bfloat16* __restrict__ y) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float v = __bfloat162float(x[i]);
        y[i] = __float2bfloat16_rn(0.5f * v * (1.f + erff(v * 0.70710678118654752f)));
    }
}
__global__ void __launch_bounds__(256)
gelu_bwd_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ g, long long n,
                __nv_bfloat16* __restrict__ dx) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float v = __bfloat162float(x[i]);
        const float cdf = 0.5f * (1.f + erff(v * 0.70710678118654752f));
        const float pdf = 0.3989422804014327f * __expf(-0.5f * v * v);
        dx[i] = __float2bfloat16_rn(__bfloat162float(g[i]) * (cdf + v * pdf));
    }
}

// ---- dropout fused into the row-wise kernels (pai_dropout.cuh; one thread per 4 consecutive elements) ---------
// mask of the attention block's / feed-forward's output: z = x + y * M / (1-p) (bf16, the residual sum the backward
// reads), out = LayerNorm(z).  One CTA per row; zs[d] holds the row of z.
__global__ void __launch_bounds__(256)
add_dropout_layernorm_fwd_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ y, int d,
                                 const long long* __restrict__ key, int site, uint32_t thr, float dscale,
                                 const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                 __nv_bfloat16* __restrict__ z, __nv_bfloat16* __restrict__ out,
                                 float* __restrict__ mean, float* __restrict__ rstd) {
    extern __shared__ float zs[];
    __shared__ float red[32];
    const long long row = blockIdx.x;
    const unsigned long long k = (unsigned long long)*key;
    float s = 0.f;
    for (int c = threadIdx.x * 4; c < d; c += blockDim.x * 4) {
        const long long e = row * d + c;
        const uint4 r = dropout_bits((unsigned long long)e >> 2, site, k);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const __nv_bfloat16 zb = __float2bfloat16_rn(
                __bfloat162float(x[e + q]) + __bfloat162float(y[e + q]) * dropout_factor(dropout_word(r, q), thr, dscale));
            z[e + q] = zb;
            zs[c + q] = __bfloat162float(zb);
            s += zs[c + q];
        }
    }
    const float mu = block_sum(s, red) / d;       // block_sum's barriers also publish zs
    float qs = 0.f;
    for (int i = threadIdx.x; i < d; i += blockDim.x) {
        const float c = zs[i] - mu;
        qs = fmaf(c, c, qs);
    }
    const float rs = rsqrtf(block_sum(qs, red) / d + eps);
    for (int i = threadIdx.x; i < d; i += blockDim.x)
        out[row * d + i] = __float2bfloat16_rn((zs[i] - mu) * rs * gamma[i] + beta[i]);
    if (threadIdx.x == 0) {
        mean[row] = mu;
        rstd[row] = rs;
    }
}
// LayerNorm backward dz as layernorm_bwd_dx_kernel, plus the dropout branch's dy = dz * M / (1-p)
__global__ void __launch_bounds__(256)
layernorm_bwd_dx_dropout_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ g, int d,
                                const float* __restrict__ gamma, const float* __restrict__ mean,
                                const float* __restrict__ rstd, const long long* __restrict__ key, int site,
                                uint32_t thr, float dscale, __nv_bfloat16* __restrict__ dx, __nv_bfloat16* __restrict__ dy) {
    __shared__ float red[32];
    const long long row = blockIdx.x;
    const float mu = mean[row], rs = rstd[row];
    float a = 0.f, b = 0.f;
    for (int i = threadIdx.x; i < d; i += blockDim.x) {
        const float gg = __bfloat162float(g[row * d + i]) * gamma[i];
        const float xh = (__bfloat162float(x[row * d + i]) - mu) * rs;
        a += gg;
        b = fmaf(gg, xh, b);
    }
    const float ma = block_sum(a, red) / d;
    const float mb = block_sum(b, red) / d;
    const unsigned long long k = (unsigned long long)*key;
    for (int c = threadIdx.x * 4; c < d; c += blockDim.x * 4) {
        const long long e = row * d + c;
        const uint4 r = dropout_bits((unsigned long long)e >> 2, site, k);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float gg = __bfloat162float(g[e + q]) * gamma[c + q];
            const float xh = (__bfloat162float(x[e + q]) - mu) * rs;
            const float v = rs * (gg - ma - xh * mb);
            dx[e + q] = __float2bfloat16_rn(v);
            dy[e + q] = __float2bfloat16_rn(v * dropout_factor(dropout_word(r, q), thr, dscale));
        }
    }
}
// y = GELU(x) * M / (1-p) over n4 groups of 4 elements
__global__ void __launch_bounds__(256)
gelu_dropout_fwd_kernel(const __nv_bfloat16* __restrict__ x, long long n4, const long long* __restrict__ key, int site,
                        uint32_t thr, float dscale, __nv_bfloat16* __restrict__ y) {
    const unsigned long long k = (unsigned long long)*key;
    for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < n4; g += (long long)gridDim.x * blockDim.x) {
        const uint4 r = dropout_bits((unsigned long long)g, site, k);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float v = __bfloat162float(x[4 * g + q]);
            const float gl = 0.5f * v * (1.f + erff(v * 0.70710678118654752f));
            y[4 * g + q] = __float2bfloat16_rn(gl * dropout_factor(dropout_word(r, q), thr, dscale));
        }
    }
}
// dx = g * M / (1-p) * GELU'(x)
__global__ void __launch_bounds__(256)
gelu_dropout_bwd_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ g, long long n4,
                        const long long* __restrict__ key, int site, uint32_t thr, float dscale,
                        __nv_bfloat16* __restrict__ dx) {
    const unsigned long long k = (unsigned long long)*key;
    for (long long gi = (long long)blockIdx.x * blockDim.x + threadIdx.x; gi < n4; gi += (long long)gridDim.x * blockDim.x) {
        const uint4 r = dropout_bits((unsigned long long)gi, site, k);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const long long i = 4 * gi + q;
            const float v = __bfloat162float(x[i]);
            const float cdf = 0.5f * (1.f + erff(v * 0.70710678118654752f));
            const float pdf = 0.3989422804014327f * __expf(-0.5f * v * v);
            const float gd = __bfloat162float(g[i]) * dropout_factor(dropout_word(r, q), thr, dscale);
            dx[i] = __float2bfloat16_rn(gd * (cdf + v * pdf));
        }
    }
}
// the mask itself (0 = dropped, 1 = kept), for tests and RNG checks
__global__ void __launch_bounds__(256)
dropout_mask_kernel(const long long* __restrict__ key, int site, long long n, uint32_t thr, uint8_t* __restrict__ out) {
    const unsigned long long k = (unsigned long long)*key;
    const long long n4 = (n + 3) >> 2;
    for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < n4; g += (long long)gridDim.x * blockDim.x) {
        const uint4 r = dropout_bits((unsigned long long)g, site, k);
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (4 * g + q < n) out[4 * g + q] = dropout_word(r, q) >= thr ? 1 : 0;
    }
}

// ---- multi-head self-attention over the sequence axis S -----------------------------------------
// Dropout on the attention probabilities (site 0 of a layer): element (bh, i, j) has the linear index (bh*S + i)*S + j
// of probs.  Key, site, threshold and 1/(1-p) travel together; DROP = false compiles the plain kernels.
struct DropArgs {
    const long long* key;
    int site;
    uint32_t thr;
    float scale;
};

// v[j] *= dropout factor of element base + j, j < len; block-cooperative, 4 consecutive elements per Philox call
__device__ __forceinline__ void dropout_span(float* v, long long base, int len, unsigned long long key, const DropArgs& da) {
    const long long g1 = (base + len - 1) >> 2;
    for (long long g = (base >> 2) + threadIdx.x; g <= g1; g += blockDim.x) {
        const uint4 r = dropout_bits((unsigned long long)g, da.site, key);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const long long j = g * 4 + q - base;
            if (j >= 0 && j < len) v[j] *= dropout_factor(dropout_word(r, q), da.thr, da.scale);
        }
    }
}

// qkv: [S*B, 3*E] bf16 (row = s*B + b; columns [0,E) = Q, [E,2E) = K, [2E,3E) = V), E = H*hd.
// One CTA per (query i, b*H + h).  probs: [B*H, S, S] fp32 (saved for backward, never dropped).  S <= 1024.
template <bool DROP>
__device__ __forceinline__ void
attn_fwd_body(const __nv_bfloat16* __restrict__ qkv, int S, int B, int H, int hd, float scale,
              float* __restrict__ probs, __nv_bfloat16* __restrict__ out /* [S*B, E] */, const DropArgs& da) {
    extern __shared__ float sm[];        // q[hd] | p[S]
    float* qs = sm;
    float* ps = sm + hd;
    __shared__ float red[32];
    const int i = blockIdx.x, bh = blockIdx.y, b = bh / H, h = bh % H;
    const int E = H * hd;
    const long long ld = 3LL * E;
    const __nv_bfloat16* qrow = qkv + ((long long)i * B + b) * ld + h * hd;
    for (int t = threadIdx.x; t < hd; t += blockDim.x) qs[t] = __bfloat162float(qrow[t]);
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int j = warp; j < S; j += nw) {
        const __nv_bfloat16* krow = qkv + ((long long)j * B + b) * ld + E + h * hd;
        float acc = 0.f;
        for (int t = lane; t < hd; t += 32) acc = fmaf(qs[t], __bfloat162float(krow[t]), acc);
        acc = warp_sum(acc);
        if (lane == 0) ps[j] = acc * scale;
    }
    __syncthreads();
    float mx = -INFINITY;
    for (int j = threadIdx.x; j < S; j += blockDim.x) mx = fmaxf(mx, ps[j]);
    {   // block max
        float v = mx;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
        if (lane == 0) red[warp] = v;
        __syncthreads();
        v = red[0];
        for (int w = 1; w < nw; ++w) v = fmaxf(v, red[w]);
        mx = v;
    }
    float sum = 0.f;
    for (int j = threadIdx.x; j < S; j += blockDim.x) {
        const float e = __expf(ps[j] - mx);
        ps[j] = e;
        sum += e;
    }
    const float inv = 1.f / block_sum(sum, red);
    for (int j = threadIdx.x; j < S; j += blockDim.x) {
        ps[j] *= inv;
        probs[((long long)bh * S + i) * S + j] = ps[j];
    }
    __syncthreads();
    if (DROP) {
        dropout_span(ps, ((long long)bh * S + i) * S, S, (unsigned long long)*da.key, da);
        __syncthreads();
    }
    for (int t = threadIdx.x; t < hd; t += blockDim.x) {
        float acc = 0.f;
        for (int j = 0; j < S; ++j)
            acc = fmaf(ps[j], __bfloat162float(qkv[((long long)j * B + b) * ld + 2 * E + h * hd + t]), acc);
        out[((long long)i * B + b) * E + h * hd + t] = __float2bfloat16_rn(acc);
    }
}
__global__ void __launch_bounds__(128)
attn_fwd_kernel(const __nv_bfloat16* __restrict__ qkv, int S, int B, int H, int hd, float scale,
                float* __restrict__ probs, __nv_bfloat16* __restrict__ out) {
    attn_fwd_body<false>(qkv, S, B, H, hd, scale, probs, out, DropArgs{});
}
// out = (P o M / (1-p)) V
__global__ void __launch_bounds__(128)
attn_fwd_dropout_kernel(const __nv_bfloat16* __restrict__ qkv, int S, int B, int H, int hd, float scale,
                        float* __restrict__ probs, __nv_bfloat16* __restrict__ out, DropArgs da) {
    attn_fwd_body<true>(qkv, S, B, H, hd, scale, probs, out, da);
}
// backward, query side: dS[i, :] = P[i, :] * (dP[i, :] - sum_j P dP), dP[i, j] = dO_i . V_j (times M_ij / (1-p) with
// dropout);  dQ_i = scale * sum_j dS_ij K_j
template <bool DROP>
__device__ __forceinline__ void
attn_bwd_q_body(const __nv_bfloat16* __restrict__ qkv, const __nv_bfloat16* __restrict__ dout, int S, int B, int H,
                int hd, float scale, const float* __restrict__ probs, float* __restrict__ ds /* [B*H, S, S] */,
                __nv_bfloat16* __restrict__ dqkv /* [S*B, 3E] */, const DropArgs& da) {
    extern __shared__ float sm[];        // do[hd] | dsrow[S]
    float* dos = sm;
    float* dsr = sm + hd;
    __shared__ float red[32];
    const int i = blockIdx.x, bh = blockIdx.y, b = bh / H, h = bh % H;
    const int E = H * hd;
    const long long ld = 3LL * E;
    for (int t = threadIdx.x; t < hd; t += blockDim.x)
        dos[t] = __bfloat162float(dout[((long long)i * B + b) * E + h * hd + t]);
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const float* prow = probs + ((long long)bh * S + i) * S;
    for (int j = warp; j < S; j += nw) {
        const __nv_bfloat16* vrow = qkv + ((long long)j * B + b) * ld + 2 * E + h * hd;
        float acc = 0.f;
        for (int t = lane; t < hd; t += 32) acc = fmaf(dos[t], __bfloat162float(vrow[t]), acc);
        acc = warp_sum(acc);
        if (lane == 0) dsr[j] = acc;
    }
    __syncthreads();
    if (DROP) {
        dropout_span(dsr, ((long long)bh * S + i) * S, S, (unsigned long long)*da.key, da);
        __syncthreads();
    }
    float part = 0.f;
    for (int j = threadIdx.x; j < S; j += blockDim.x) part = fmaf(prow[j], dsr[j], part);
    const float delta = block_sum(part, red);
    for (int j = threadIdx.x; j < S; j += blockDim.x) {
        const float v = prow[j] * (dsr[j] - delta);
        dsr[j] = v;
        ds[((long long)bh * S + i) * S + j] = v;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < hd; t += blockDim.x) {
        float acc = 0.f;
        for (int j = 0; j < S; ++j)
            acc = fmaf(dsr[j], __bfloat162float(qkv[((long long)j * B + b) * ld + E + h * hd + t]), acc);
        dqkv[((long long)i * B + b) * ld + h * hd + t] = __float2bfloat16_rn(acc * scale);
    }
}
__global__ void __launch_bounds__(128)
attn_bwd_q_kernel(const __nv_bfloat16* __restrict__ qkv, const __nv_bfloat16* __restrict__ dout, int S, int B, int H,
                  int hd, float scale, const float* __restrict__ probs, float* __restrict__ ds,
                  __nv_bfloat16* __restrict__ dqkv) {
    attn_bwd_q_body<false>(qkv, dout, S, B, H, hd, scale, probs, ds, dqkv, DropArgs{});
}
__global__ void __launch_bounds__(128)
attn_bwd_q_dropout_kernel(const __nv_bfloat16* __restrict__ qkv, const __nv_bfloat16* __restrict__ dout, int S, int B,
                          int H, int hd, float scale, const float* __restrict__ probs, float* __restrict__ ds,
                          __nv_bfloat16* __restrict__ dqkv, DropArgs da) {
    attn_bwd_q_body<true>(qkv, dout, S, B, H, hd, scale, probs, ds, dqkv, da);
}
// backward, key/value side: dK_j = scale * sum_i dS_ij Q_i;  dV_j = sum_i P_ij dO_i (P_ij M_ij / (1-p) with dropout:
// the column's elements are S apart, so each regenerates its own Philox block)
template <bool DROP>
__device__ __forceinline__ void
attn_bwd_kv_body(const __nv_bfloat16* __restrict__ qkv, const __nv_bfloat16* __restrict__ dout, int S, int B, int H,
                 int hd, float scale, const float* __restrict__ probs, const float* __restrict__ ds,
                 __nv_bfloat16* __restrict__ dqkv, const DropArgs& da) {
    extern __shared__ float sm[];        // pcol[S] | dscol[S]
    float* pc = sm;
    float* dc = sm + S;
    const int j = blockIdx.x, bh = blockIdx.y, b = bh / H, h = bh % H;
    const int E = H * hd;
    const long long ld = 3LL * E;
    for (int i = threadIdx.x; i < S; i += blockDim.x) {
        const long long idx = ((long long)bh * S + i) * S + j;
        pc[i] = probs[idx];
        dc[i] = ds[idx];
        if (DROP) {
            const uint4 r = dropout_bits((unsigned long long)idx >> 2, da.site, (unsigned long long)*da.key);
            pc[i] *= dropout_factor(dropout_word(r, (int)(idx & 3)), da.thr, da.scale);
        }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < hd; t += blockDim.x) {
        float dk = 0.f, dv = 0.f;
        for (int i = 0; i < S; ++i) {
            dk = fmaf(dc[i], __bfloat162float(qkv[((long long)i * B + b) * ld + h * hd + t]), dk);
            dv = fmaf(pc[i], __bfloat162float(dout[((long long)i * B + b) * E + h * hd + t]), dv);
        }
        dqkv[((long long)j * B + b) * ld + E + h * hd + t] = __float2bfloat16_rn(dk * scale);
        dqkv[((long long)j * B + b) * ld + 2 * E + h * hd + t] = __float2bfloat16_rn(dv);
    }
}
__global__ void __launch_bounds__(128)
attn_bwd_kv_kernel(const __nv_bfloat16* __restrict__ qkv, const __nv_bfloat16* __restrict__ dout, int S, int B, int H,
                   int hd, float scale, const float* __restrict__ probs, const float* __restrict__ ds,
                   __nv_bfloat16* __restrict__ dqkv) {
    attn_bwd_kv_body<false>(qkv, dout, S, B, H, hd, scale, probs, ds, dqkv, DropArgs{});
}
__global__ void __launch_bounds__(128)
attn_bwd_kv_dropout_kernel(const __nv_bfloat16* __restrict__ qkv, const __nv_bfloat16* __restrict__ dout, int S, int B,
                           int H, int hd, float scale, const float* __restrict__ probs, const float* __restrict__ ds,
                           __nv_bfloat16* __restrict__ dqkv, DropArgs da) {
    attn_bwd_kv_body<true>(qkv, dout, S, B, H, hd, scale, probs, ds, dqkv, da);
}

}  // namespace pai

using namespace pai;
typedef __nv_bfloat16 bf16;

extern "C" {

int pai_layernorm_fwd(const void* x, long long m, int d, const float* gamma, const float* beta, float eps, void* y,
                      float* mean, float* rstd, void* stream) {
    PAI_REQUIRE(x && gamma && beta && y && mean && rstd && m > 0 && d > 0, "pai_layernorm_fwd: null pointer / empty input");
    layernorm_fwd_kernel<<<(unsigned)m, 256, 0, (cudaStream_t)stream>>>((const bf16*)x, d, gamma, beta, eps, (bf16*)y, mean, rstd);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_layernorm_bwd(const void* x, const void* g, long long m, int d, const float* gamma, const float* mean,
                      const float* rstd, void* dx, float* dgamma, float* dbeta, void* stream) {
    PAI_REQUIRE(x && g && gamma && mean && rstd && dx && dgamma && dbeta && m > 0, "pai_layernorm_bwd: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    layernorm_bwd_dx_kernel<<<(unsigned)m, 256, 0, st>>>((const bf16*)x, (const bf16*)g, d, gamma, mean, rstd, (bf16*)dx);
    PAI_CUDA_OK(cudaGetLastError());
    PAI_CUDA_OK(cudaMemsetAsync(dgamma, 0, sizeof(float) * d, st));
    PAI_CUDA_OK(cudaMemsetAsync(dbeta, 0, sizeof(float) * d, st));
    int ry = (int)(m < 32 ? m : 32);
    layernorm_bwd_affine_kernel<<<dim3((d + 255) / 256, ry), 256, 0, st>>>((const bf16*)x, (const bf16*)g, m, d, mean, rstd,
                                                                          dgamma, dbeta);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_gelu_fwd(const void* x, long long n, void* y, void* stream) {
    PAI_REQUIRE(x && y && n > 0, "pai_gelu_fwd: null pointer");
    long long b = (n + 255) / 256;
    if (b > 148 * 16) b = 148 * 16;
    gelu_fwd_kernel<<<(int)b, 256, 0, (cudaStream_t)stream>>>((const bf16*)x, n, (bf16*)y);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_gelu_bwd(const void* x, const void* g, long long n, void* dx, void* stream) {
    PAI_REQUIRE(x && g && dx && n > 0, "pai_gelu_bwd: null pointer");
    long long b = (n + 255) / 256;
    if (b > 148 * 16) b = 148 * 16;
    gelu_bwd_kernel<<<(int)b, 256, 0, (cudaStream_t)stream>>>((const bf16*)x, (const bf16*)g, n, (bf16*)dx);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_attn_fwd(const void* qkv, int s, int b, int heads, int head_dim, float* probs, void* out, void* stream) {
    PAI_REQUIRE(qkv && probs && out && s > 0 && b > 0 && heads > 0 && head_dim > 0, "pai_attn_fwd: null pointer / empty");
    PAI_REQUIRE((head_dim + s) * 4 <= 48 * 1024, "pai_attn_fwd: head_dim + sequence too large for shared memory");
    attn_fwd_kernel<<<dim3(s, b * heads), 128, (head_dim + s) * sizeof(float), (cudaStream_t)stream>>>(
        (const bf16*)qkv, s, b, heads, head_dim, 1.f / sqrtf((float)head_dim), probs, (bf16*)out);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_attn_bwd(const void* qkv, const void* dout, int s, int b, int heads, int head_dim, const float* probs,
                 float* ds_work, void* dqkv, void* stream) {
    PAI_REQUIRE(qkv && dout && probs && ds_work && dqkv && s > 0, "pai_attn_bwd: null pointer / empty");
    PAI_REQUIRE((head_dim + s) * 4 <= 48 * 1024 && 2 * s * 4 <= 48 * 1024, "pai_attn_bwd: sizes too large for shared memory");
    cudaStream_t st = (cudaStream_t)stream;
    const float scale = 1.f / sqrtf((float)head_dim);
    attn_bwd_q_kernel<<<dim3(s, b * heads), 128, (head_dim + s) * sizeof(float), st>>>(
        (const bf16*)qkv, (const bf16*)dout, s, b, heads, head_dim, scale, probs, ds_work, (bf16*)dqkv);
    PAI_CUDA_OK(cudaGetLastError());
    attn_bwd_kv_kernel<<<dim3(s, b * heads), 128, 2 * s * sizeof(float), st>>>(
        (const bf16*)qkv, (const bf16*)dout, s, b, heads, head_dim, scale, probs, ds_work, (bf16*)dqkv);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}


// ---- train-mode dropout of the encoder layer (sites: layer*4 + {0 attention probs, 1 attention output,
// 2 after GELU, 3 feed-forward output}); key is a device pointer to the forward's 64-bit key
#define PAI_DROPOUT_ARGS_OK(name)                                                                          \
    PAI_REQUIRE(key != nullptr, name ": null key pointer");                                                \
    PAI_REQUIRE(p > 0.f && p < 1.f, name ": dropout probability %g outside (0, 1)", (double)p)

static long long dropout_grid(long long n4) {
    const long long b = (n4 + 255) / 256;
    return b > 148 * 16 ? 148 * 16 : b;
}

int pai_dropout_mask(const long long* key, int site, long long n, float p, void* out, void* stream) {
    PAI_DROPOUT_ARGS_OK("pai_dropout_mask");
    PAI_REQUIRE(out && n > 0 && site >= 0, "pai_dropout_mask: null pointer / empty / negative site");
    dropout_mask_kernel<<<(int)dropout_grid((n + 3) / 4), 256, 0, (cudaStream_t)stream>>>(key, site, n, dropout_threshold(p),
                                                                                          (uint8_t*)out);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_attn_fwd_dropout(const void* qkv, int s, int b, int heads, int head_dim, const long long* key, int site, float p,
                         float* probs, void* out, void* stream) {
    PAI_DROPOUT_ARGS_OK("pai_attn_fwd_dropout");
    PAI_REQUIRE(qkv && probs && out && s > 0 && b > 0 && heads > 0 && head_dim > 0 && site >= 0,
                "pai_attn_fwd_dropout: null pointer / empty");
    PAI_REQUIRE((head_dim + s) * 4 <= 48 * 1024, "pai_attn_fwd_dropout: head_dim + sequence too large for shared memory");
    const DropArgs da{key, site, dropout_threshold(p), 1.f / (1.f - p)};
    attn_fwd_dropout_kernel<<<dim3(s, b * heads), 128, (head_dim + s) * sizeof(float), (cudaStream_t)stream>>>(
        (const bf16*)qkv, s, b, heads, head_dim, 1.f / sqrtf((float)head_dim), probs, (bf16*)out, da);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_attn_bwd_dropout(const void* qkv, const void* dout, int s, int b, int heads, int head_dim, const long long* key,
                         int site, float p, const float* probs, float* ds_work, void* dqkv, void* stream) {
    PAI_DROPOUT_ARGS_OK("pai_attn_bwd_dropout");
    PAI_REQUIRE(qkv && dout && probs && ds_work && dqkv && s > 0 && b > 0 && heads > 0 && head_dim > 0 && site >= 0,
                "pai_attn_bwd_dropout: null pointer / empty");
    PAI_REQUIRE((head_dim + s) * 4 <= 48 * 1024 && 2 * s * 4 <= 48 * 1024,
                "pai_attn_bwd_dropout: sizes too large for shared memory");
    cudaStream_t st = (cudaStream_t)stream;
    const float scale = 1.f / sqrtf((float)head_dim);
    const DropArgs da{key, site, dropout_threshold(p), 1.f / (1.f - p)};
    attn_bwd_q_dropout_kernel<<<dim3(s, b * heads), 128, (head_dim + s) * sizeof(float), st>>>(
        (const bf16*)qkv, (const bf16*)dout, s, b, heads, head_dim, scale, probs, ds_work, (bf16*)dqkv, da);
    PAI_CUDA_OK(cudaGetLastError());
    attn_bwd_kv_dropout_kernel<<<dim3(s, b * heads), 128, 2 * s * sizeof(float), st>>>(
        (const bf16*)qkv, (const bf16*)dout, s, b, heads, head_dim, scale, probs, ds_work, (bf16*)dqkv, da);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_add_dropout_layernorm_fwd(const void* x, const void* y, long long m, int d, const long long* key, int site, float p,
                                  const float* gamma, const float* beta, float eps, void* z, void* out, float* mean,
                                  float* rstd, void* stream) {
    PAI_DROPOUT_ARGS_OK("pai_add_dropout_layernorm_fwd");
    PAI_REQUIRE(x && y && gamma && beta && z && out && mean && rstd && m > 0 && d > 0 && site >= 0,
                "pai_add_dropout_layernorm_fwd: null pointer / empty input");
    PAI_REQUIRE(d % 4 == 0 && d * 4 <= 48 * 1024, "pai_add_dropout_layernorm_fwd: d must be a multiple of 4, at most 12288");
    add_dropout_layernorm_fwd_kernel<<<(unsigned)m, 256, d * sizeof(float), (cudaStream_t)stream>>>(
        (const bf16*)x, (const bf16*)y, d, key, site, dropout_threshold(p), 1.f / (1.f - p), gamma, beta, eps, (bf16*)z,
        (bf16*)out, mean, rstd);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_layernorm_bwd_dropout(const void* z, const void* g, long long m, int d, const float* gamma, const float* mean,
                              const float* rstd, const long long* key, int site, float p, void* dz, void* dy,
                              float* dgamma, float* dbeta, void* stream) {
    PAI_DROPOUT_ARGS_OK("pai_layernorm_bwd_dropout");
    PAI_REQUIRE(z && g && gamma && mean && rstd && dz && dy && dgamma && dbeta && m > 0 && d > 0 && site >= 0,
                "pai_layernorm_bwd_dropout: null pointer / empty input");
    PAI_REQUIRE(d % 4 == 0, "pai_layernorm_bwd_dropout: d must be a multiple of 4");
    cudaStream_t st = (cudaStream_t)stream;
    layernorm_bwd_dx_dropout_kernel<<<(unsigned)m, 256, 0, st>>>((const bf16*)z, (const bf16*)g, d, gamma, mean, rstd, key,
                                                                 site, dropout_threshold(p), 1.f / (1.f - p), (bf16*)dz,
                                                                 (bf16*)dy);
    PAI_CUDA_OK(cudaGetLastError());
    PAI_CUDA_OK(cudaMemsetAsync(dgamma, 0, sizeof(float) * d, st));
    PAI_CUDA_OK(cudaMemsetAsync(dbeta, 0, sizeof(float) * d, st));
    int ry = (int)(m < 32 ? m : 32);
    layernorm_bwd_affine_kernel<<<dim3((d + 255) / 256, ry), 256, 0, st>>>((const bf16*)z, (const bf16*)g, m, d, mean, rstd,
                                                                          dgamma, dbeta);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_gelu_dropout_fwd(const void* x, long long n, const long long* key, int site, float p, void* y, void* stream) {
    PAI_DROPOUT_ARGS_OK("pai_gelu_dropout_fwd");
    PAI_REQUIRE(x && y && n > 0 && site >= 0, "pai_gelu_dropout_fwd: null pointer / empty input");
    PAI_REQUIRE(n % 4 == 0, "pai_gelu_dropout_fwd: n must be a multiple of 4");
    gelu_dropout_fwd_kernel<<<(int)dropout_grid(n / 4), 256, 0, (cudaStream_t)stream>>>(
        (const bf16*)x, n / 4, key, site, dropout_threshold(p), 1.f / (1.f - p), (bf16*)y);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}
int pai_gelu_dropout_bwd(const void* x, const void* g, long long n, const long long* key, int site, float p, void* dx,
                         void* stream) {
    PAI_DROPOUT_ARGS_OK("pai_gelu_dropout_bwd");
    PAI_REQUIRE(x && g && dx && n > 0 && site >= 0, "pai_gelu_dropout_bwd: null pointer / empty input");
    PAI_REQUIRE(n % 4 == 0, "pai_gelu_dropout_bwd: n must be a multiple of 4");
    gelu_dropout_bwd_kernel<<<(int)dropout_grid(n / 4), 256, 0, (cudaStream_t)stream>>>(
        (const bf16*)x, (const bf16*)g, n / 4, key, site, dropout_threshold(p), 1.f / (1.f - p), (bf16*)dx);
    PAI_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // extern "C"
