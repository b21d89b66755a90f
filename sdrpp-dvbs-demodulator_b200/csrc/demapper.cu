// K1 -- see demapper.cuh.
#include "demapper.cuh"
#include "demap_common.cuh"

#include <algorithm>

namespace s2 {
namespace {

// gridDim.y is limited to 65535: frames beyond that are taken by the same blocks in further rounds, while the symbol
// index stays in x so that neighbouring threads load neighbouring symbols
constexpr int kMaxGridY = 65535;

__global__ void __launch_bounds__(256) demap_kernel(const __grid_constant__ DemapDev d, const float2* __restrict__ in,
                                                    int nframes, int8_t* __restrict__ out) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= d.nsym) return;
    const int raw = 90 + s + (d.pilots ? 36 * (s / 1440) : 0);
    for (int frame = blockIdx.y; frame < nframes; frame += gridDim.y) {
        float2 v = __ldg(&in[(size_t)frame * d.plframe_syms + raw]);
        if (d.rn) {   // exact: quarter turns only swap and negate
            const int r = __ldg(&d.rn[raw - 90]);
            const float2 u = v;
            if (r == 1) v = make_float2(u.y, -u.x);
            else if (r == 2) v = make_float2(-u.x, -u.y);
            else if (r == 3) v = make_float2(-u.y, u.x);
        }
        int8_t* o = out + (size_t)frame * d.N;
        int8_t b[5];
        demap_symbol(d, v, b);
        store_llrs(d, o, s, b);
    }
}

// Same gather from the two 8-bit LUT coordinates per symbol that the host computed (dvbs2fec_quantize_plframes:
// the reference's own index arithmetic, constellation.cpp:295-310, after pilot removal and PL descrambling):
// 2 bytes per symbol over PCIe instead of 8, identical LLRs.
__global__ void __launch_bounds__(256) demap_idx_kernel(const __grid_constant__ DemapDev d, const uchar2* __restrict__ idx,
                                                        int nframes, int8_t* __restrict__ out) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= d.nsym) return;
    for (int frame = blockIdx.y; frame < nframes; frame += gridDim.y) {
        const uchar2 xy = __ldg(&idx[(size_t)frame * d.nsym + s]);
        const uint32_t w = __ldg(&d.lut[(int)xy.x * 256 + (int)xy.y]);
        int8_t b[5] = {(int8_t)(w & 0xFF), (int8_t)((w >> 8) & 0xFF), (int8_t)((w >> 16) & 0xFF), (int8_t)(w >> 24), 0};
        store_llrs(d, out + (size_t)frame * d.N, s, b);
    }
}

}  // namespace

int demap_launch(const DemapDev& d, const float* plframes, int nframes, int8_t* llr_out, cudaStream_t stream) {
    if (nframes <= 0) return 0;
    dim3 grid((d.nsym + 255) / 256, std::min(nframes, kMaxGridY));
    demap_kernel<<<grid, 256, 0, stream>>>(d, reinterpret_cast<const float2*>(plframes), nframes, llr_out);
    return (int)cudaGetLastError();
}

int demap_idx_launch(const DemapDev& d, const uint8_t* idx, int nframes, int8_t* llr_out, cudaStream_t stream) {
    if (nframes <= 0) return 0;
    if (!d.lut) return (int)cudaErrorInvalidValue;   // 32APSK has no LUT
    dim3 grid((d.nsym + 255) / 256, std::min(nframes, kMaxGridY));
    demap_idx_kernel<<<grid, 256, 0, stream>>>(d, reinterpret_cast<const uchar2*>(idx), nframes, llr_out);
    return (int)cudaGetLastError();
}

}  // namespace s2
