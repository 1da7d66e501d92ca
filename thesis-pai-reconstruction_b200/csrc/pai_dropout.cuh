// Counter-based dropout masks (Philox4x32-10, Salmon et al., SC'11).  A mask is never stored: a kernel that applies
// dropout regenerates the bits of its elements from (element index, site, key), so the backward sees exactly the
// forward's mask.  Element idx of site `site` under the 64-bit key `key`:
//   r = word (idx & 3) of philox4x32_10(counter = (lo32(idx >> 2), hi32(idx >> 2), site, 0), key = (lo32, hi32))
//   dropped iff r < thr, thr = min(2^32 - 1, llround(p * 2^32)) computed once on the host in double precision;
//   kept elements are multiplied by 1 / (1 - p) (fp32).
// oracle/vit_dropout_ref.py restates this rule in numpy.
#pragma once
#include <math.h>
#include <stdint.h>

namespace pai {

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), hi1 = __umulhi(0xCD9E8D57u, c.z);
        const uint32_t lo0 = 0xD2511F53u * c.x, lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

// The random words of elements 4g .. 4g+3 of dropout site `site`.
__device__ __forceinline__ uint4 dropout_bits(unsigned long long g, int site, unsigned long long key) {
    return philox4x32_10(make_uint4((uint32_t)g, (uint32_t)(g >> 32), (uint32_t)site, 0u),
                         make_uint2((uint32_t)key, (uint32_t)(key >> 32)));
}

__device__ __forceinline__ uint32_t dropout_word(const uint4& r, int q) {
    return q == 0 ? r.x : q == 1 ? r.y : q == 2 ? r.z : r.w;
}

// multiplier of an element whose random word is r: 0 (dropped) or 1 / (1 - p)
__device__ __forceinline__ float dropout_factor(uint32_t r, uint32_t thr, float scale) {
    return r < thr ? 0.f : scale;
}

inline uint32_t dropout_threshold(float p) {
    const long long t = llround((double)p * 4294967296.0);
    return t > 0xffffffffLL ? 0xffffffffu : (uint32_t)t;
}

}  // namespace pai
