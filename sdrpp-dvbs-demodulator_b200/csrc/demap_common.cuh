// K1 device helpers shared by demap_kernel / demap_idx_kernel (demapper.cu) and demap_vcm_kernel (vcm.cu): one
// payload symbol -> its LLR bytes at their deinterleaved places.  Both kernels must produce the same bytes.
#pragma once
#include <climits>
#include <cstdint>

#include "demapper.cuh"

namespace s2 {

// int(double) as the x86 host does it (cvttsd2si): out-of-range and NaN give INT_MIN
__device__ __forceinline__ int host_trunc(double v) {
    if (!(v > -2147483649.0 && v < 2147483648.0)) return INT_MIN;
    return __double2int_rz(v);
}
__device__ __forceinline__ int lut_index(float s) {
    int x = host_trunc(((double)s / 1.5) * 256 + 128);
    return min(max(x, 0), 255);
}
__device__ __forceinline__ int halving_clamp(float x) {
    while (x < -127 || x > 127) {
        x *= 0.5f;
        if (!isfinite(x)) return 0;   // (int8_t)(int)inf/nan on the host: low byte of INT_MIN
    }
    return (int)x;
}

// LLR bytes of symbol s to their deinterleaved places (S2Deinterleaver::deinterleave, s2_deinterleaver.cpp:72-136)
__device__ __forceinline__ void store_llrs(const DemapDev& d, int8_t* o, int s, const int8_t (&b)[5]) {
    if (d.constellation == 0) {           // QPSK: the pair is swapped, no column interleave
        *reinterpret_cast<uint16_t*>(o + 2 * s) = (uint16_t)((uint8_t)b[1] | ((uint16_t)(uint8_t)b[0] << 8));
        return;
    }
#pragma unroll
    for (int k = 0; k < 5; ++k)
        if (k < d.bits) {
            int col = (d.reversed_cols) ? (2 - k) : k;
            o[col * d.nsym + s] = b[k];
        }
}

// soft bits of one (descrambled) symbol: the LUT gather, or for 32APSK the reference's per-symbol expf / logf
__device__ __forceinline__ void demap_symbol(const DemapDev& d, float2 v, int8_t (&b)[5]) {
    if (d.constellation != 3) {
        uint32_t w = __ldg(&d.lut[lut_index(v.x) * 256 + lut_index(v.y)]);
        b[0] = (int8_t)(w & 0xFF);
        b[1] = (int8_t)((w >> 8) & 0xFF);
        b[2] = (int8_t)((w >> 16) & 0xFF);
        b[3] = (int8_t)(w >> 24);
    } else {
        float re = (v.x * d.amp) * d.prescale, im = (v.y * d.amp) * d.prescale;
        float acc[10];
#pragma unroll
        for (int k = 0; k < 10; ++k) acc[k] = 0.f;
        for (int i = 0; i < 32; ++i) {
            float dr = re - d.pts[2 * i], di = im - d.pts[2 * i + 1];
            float e = expf(-sqrtf(__fadd_rn(__fmul_rn(dr, dr), __fmul_rn(di, di))));
#pragma unroll
            for (int jb = 0; jb < 5; ++jb) {
                if ((i >> jb) & 1) acc[2 * jb + 1] += e;
                else acc[2 * jb] += e;
            }
        }
#pragma unroll
        for (int jb = 0; jb < 5; ++jb)
            b[4 - jb] = (int8_t)halving_clamp((logf(acc[2 * jb + 1]) - logf(acc[2 * jb])) * d.sca);
    }
}

}  // namespace s2
