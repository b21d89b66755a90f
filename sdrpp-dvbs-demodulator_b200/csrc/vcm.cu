// VCM / ACM kernels -- see vcm.cuh.
#include "vcm.cuh"

#include <algorithm>

#include "../../include/dvbs2fec.h"
#include "demap_common.cuh"

namespace s2 {
namespace {

constexpr int kMaxGrid = 65535;   // frames in gridDim.y (x for the scatter): further frames are taken in further rounds
constexpr int kGatherWords = 4;   // 8-byte words per thread and block row of the gather

// One thread per payload symbol of the chunk's largest frame; blockIdx.y walks the frames.  Each frame reads its
// configuration's DemapDev from the device table (the rn field there is unused: the handle's sequence is passed in).
__global__ void __launch_bounds__(256) demap_vcm_kernel(const DemapDev* __restrict__ table, const uint8_t* __restrict__ rn,
                                                        const float2* __restrict__ in, long long in_shift,
                                                        const VcmFrame* __restrict__ frames, int nframes,
                                                        int8_t* __restrict__ out) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    for (int frame = blockIdx.y; frame < nframes; frame += gridDim.y) {
        const VcmFrame& f = frames[frame];
        if (f.pos < 0) continue;   // DUMMY PLFRAME: never read
        const DemapDev& d = table[f.cfg];
        if (s >= d.nsym) continue;
        const int raw = 90 + s + (d.pilots ? 36 * (s / 1440) : 0);
        float2 v = __ldg(&in[f.in_off - in_shift + raw]);
        if (rn) {   // exact: quarter turns only swap and negate
            const int r = __ldg(&rn[raw - 90]);
            const float2 u = v;
            if (r == 1) v = make_float2(u.y, -u.x);
            else if (r == 2) v = make_float2(-u.x, -u.y);
            else if (r == 3) v = make_float2(-u.y, u.x);
        }
        int8_t b[5];
        demap_symbol(d, v, b);
        store_llrs(d, out + f.llr_off, s, b);
    }
}

// LLR rows into their group rows.  Frame starts are multiples of 8 bytes apart (16 200 / 64 800): 8-byte words when
// both ends are aligned, bytes otherwise.
__global__ void __launch_bounds__(256) vcm_gather_kernel(const int8_t* __restrict__ in, long long in_shift,
                                                         const VcmFrame* __restrict__ frames, int nframes,
                                                         int8_t* __restrict__ out) {
    for (int frame = blockIdx.y; frame < nframes; frame += gridDim.y) {
        const VcmFrame& f = frames[frame];
        if (f.pos < 0) continue;
        const int8_t* src = in + (f.in_off - in_shift);
        int8_t* dst = out + f.llr_off;
        const int base = blockIdx.x * blockDim.x * kGatherWords;   // in words
        if ((((uintptr_t)src | (uintptr_t)dst) & 7) == 0) {
            const int words = f.nbytes >> 3;
#pragma unroll
            for (int k = 0; k < kGatherWords; ++k) {
                const int w = base + k * blockDim.x + threadIdx.x;
                if (w < words) reinterpret_cast<uint2*>(dst)[w] = __ldg(&reinterpret_cast<const uint2*>(src)[w]);
            }
        } else {
            for (int k = 0; k < 8 * kGatherWords; ++k) {
                const int x = 8 * base + k * blockDim.x + threadIdx.x;
                if (x < f.nbytes) dst[x] = src[x];
            }
        }
    }
}

// BBFRAMEs and records back to input order; the caller's BBFRAME offsets are unaligned (normal 1/4: 2001 bytes)
__global__ void __launch_bounds__(256) vcm_scatter_kernel(const VcmFrame* __restrict__ frames, int nframes,
                                                          const uint8_t* __restrict__ bb, const dvbs2fec_result* __restrict__ res,
                                                          uint8_t* __restrict__ bb_out, long long bb_shift,
                                                          dvbs2fec_result* __restrict__ res_out, unsigned long long tag_base) {
    for (int frame = blockIdx.x; frame < nframes; frame += gridDim.x) {
        const VcmFrame& f = frames[frame];
        if (f.pos >= 0 && bb_out) {
            const uint8_t* src = bb + f.bb_src;
            uint8_t* dst = bb_out + (f.bb_dst - bb_shift);
            for (int x = threadIdx.x; x < f.kb; x += blockDim.x) dst[x] = src[x];
        }
        if (threadIdx.x == 0 && res_out) {
            dvbs2fec_result r;
            if (f.pos >= 0) {
                r = res[f.pos];
            } else {
                r.ldpc_iters = 0;
                r.bch_corr = 0;
                r.flags = DVBS2FEC_FLAG_DUMMY;
            }
            r.tag = tag_base + (unsigned long long)frame;
            res_out[frame] = r;
        }
    }
}

}  // namespace

int demap_vcm_launch(const DemapDev* table, const uint8_t* rn, const float* in, long long in_shift, const VcmFrame* frames,
                     int nframes, int nsym_max, int8_t* llr, cudaStream_t stream) {
    if (nframes <= 0 || nsym_max <= 0) return 0;
    dim3 grid((nsym_max + 255) / 256, std::min(nframes, kMaxGrid));
    demap_vcm_kernel<<<grid, 256, 0, stream>>>(table, rn, reinterpret_cast<const float2*>(in), in_shift, frames, nframes, llr);
    return (int)cudaGetLastError();
}

int vcm_gather_launch(const int8_t* in, long long in_shift, const VcmFrame* frames, int nframes, int n_max, int8_t* llr,
                      cudaStream_t stream) {
    if (nframes <= 0 || n_max <= 0) return 0;
    const int per_block = 256 * kGatherWords * 8;
    dim3 grid((n_max + per_block - 1) / per_block, std::min(nframes, kMaxGrid));
    vcm_gather_kernel<<<grid, 256, 0, stream>>>(in, in_shift, frames, nframes, llr);
    return (int)cudaGetLastError();
}

int vcm_scatter_launch(const VcmFrame* frames, int nframes, const uint8_t* bb, const void* results, uint8_t* bb_out,
                       long long bb_shift, void* results_out, unsigned long long tag_base, cudaStream_t stream) {
    if (nframes <= 0) return 0;
    vcm_scatter_kernel<<<std::min(nframes, kMaxGrid), 256, 0, stream>>>(
        frames, nframes, bb, static_cast<const dvbs2fec_result*>(results), bb_out, bb_shift,
        static_cast<dvbs2fec_result*>(results_out), tag_base);
    return (int)cudaGetLastError();
}

}  // namespace s2
