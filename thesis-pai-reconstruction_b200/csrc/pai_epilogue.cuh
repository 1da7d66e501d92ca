// Epilogue helpers shared by the tcgen05 kernels (igemm.cu, thin.cu): TMEM accumulator rows -> bias / activation ->
// bf16 -> XOR-swizzled (SWIZZLE_128B) shared-memory tile -> global memory (a TMA store in igemm.cu, coalesced 128-byte
// row segments in thin.cu).
#pragma once
#include "pai_common.cuh"
#include "pai_kernels.h"

namespace pai {

__device__ __forceinline__ uint32_t tmem_cols_for(int n) {
    uint32_t c = 32;
    while ((int)c < n) c <<= 1;
    return c;
}

__device__ __forceinline__ float apply_act(float v, int act, float slope) {
    if (act == PAI_ACT_LEAKY) return v > 0.f ? v : v * slope;
    if (act == PAI_ACT_RELU) return fmaxf(v, 0.f);
    if (act == PAI_ACT_TANH) return tanhf(v);
    return v;
}

__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d)
                 : "memory");
}

// 16 consecutive channels of one pixel -> bf16, vectorised when aligned and fully inside the tensor
__device__ __forceinline__ void store_bf16_16(__nv_bfloat16* o, const float (&f)[16], int act, float slope, bool vec,
                                              int valid) {
    if (vec) {
        uint32_t w[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            __nv_bfloat162 h = __floats2bfloat162_rn(apply_act(f[2 * j], act, slope), apply_act(f[2 * j + 1], act, slope));
            w[j] = *reinterpret_cast<uint32_t*>(&h);
        }
        reinterpret_cast<uint4*>(o)[0] = make_uint4(w[0], w[1], w[2], w[3]);
        reinterpret_cast<uint4*>(o)[1] = make_uint4(w[4], w[5], w[6], w[7]);
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j)
            if (j < valid) o[j] = __float2bfloat16_rn(apply_act(f[j], act, slope));
    }
}

// 64 fp32 accumulator columns of one row -> (+bias) -> activation -> bf16 -> one XOR-swizzled 128-byte row
// of the warp's transpose tile.  ACT is a template parameter so the element loop carries no dispatch.
template <int ACT>
__device__ __forceinline__ float act_t(float v, float slope) {
    if (ACT == PAI_ACT_LEAKY) return fmaxf(v, v * slope);      // slope in (0, 1)
    if (ACT == PAI_ACT_RELU) return fmaxf(v, 0.f);
    if (ACT == PAI_ACT_TANH) return tanhf(v);
    return v;
}
template <int ACT>
__device__ __forceinline__ void bias_act_pack(const uint32_t (&v)[64], const float* __restrict__ bias, float slope,
                                              uint4* tile, int lane) {
#pragma unroll
    for (int ch = 0; ch < 8; ++ch) {
        float f[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) f[k] = __uint_as_float(v[8 * ch + k]);
        if (bias != nullptr) {
            const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + 8 * ch));
            const float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + 8 * ch) + 1);
            f[0] += b0.x, f[1] += b0.y, f[2] += b0.z, f[3] += b0.w;
            f[4] += b1.x, f[5] += b1.y, f[6] += b1.z, f[7] += b1.w;
        }
        uint32_t w[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            __nv_bfloat162 h = __floats2bfloat162_rn(act_t<ACT>(f[2 * k], slope), act_t<ACT>(f[2 * k + 1], slope));
            w[k] = *reinterpret_cast<uint32_t*>(&h);
        }
        tile[lane * 8 + (ch ^ (lane & 7))] = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// out = acc * (saved > 0 ? 1 : slope): the activation backward of the layer whose data gradient this GEMM produces.
// Works in place: the tile already holds this lane's row of 64 saved activations in the same swizzled layout (a TMA
// load of the output's box from the saved tensor; zeros for rows outside it), and each 16-byte slot is replaced by the
// product it gates.
__device__ __forceinline__ void mask_pack(const uint32_t (&v)[64], float slope, uint4* tile, int lane) {
#pragma unroll
    for (int ch = 0; ch < 8; ++ch) {
        const uint4 m = tile[lane * 8 + (ch ^ (lane & 7))];
        const __nv_bfloat162* mh = reinterpret_cast<const __nv_bfloat162*>(&m);
        uint32_t w[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float2 mf = __bfloat1622float2(mh[k]);
            const float a = __uint_as_float(v[8 * ch + 2 * k]) * (mf.x > 0.f ? 1.f : slope);
            const float b = __uint_as_float(v[8 * ch + 2 * k + 1]) * (mf.y > 0.f ? 1.f : slope);
            __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
            w[k] = *reinterpret_cast<uint32_t*>(&h);
        }
        tile[lane * 8 + (ch ^ (lane & 7))] = make_uint4(w[0], w[1], w[2], w[3]);
    }
}


// byte offset of 16-byte chunk `c` (0..7) of row `r` inside a SWIZZLE_128B tile with 128-byte rows (tile base aligned to
// 1024 B): the layout a TMA box with a 64-element bf16 inner dimension writes and the K-major UMMA descriptors read
__device__ __forceinline__ uint32_t sw128_off(int r, int c) { return (uint32_t)r * 128u + (uint32_t)((c ^ (r & 7)) << 4); }

// generic-proxy shared-memory writes -> visible to the async proxy (tcgen05.mma / TMA reads of that memory)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

}  // namespace pai
