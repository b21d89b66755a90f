// VCM / ACM batches: frames of different MODCOD, frame size and pilot setting in one call (dvbs2fec_decode_*vcm*).
//
// The host splits a call into chunks of at most max_batch frames and groups the frames of a chunk by LDPC code.
// Each group runs the per-configuration kernels (K2 ldpc_launch, K3 bch_launch) on a plain [n][N] array; the kernels
// here move frames between the caller's packed, input-ordered buffers and those group arrays:
//   * demap_vcm_kernel: PLFRAME symbols -> each frame's LLR row in its group (K1's arithmetic, demap_common.cuh);
//   * vcm_gather_kernel: LLR input -> the same rows;
//   * vcm_scatter_kernel: BBFRAMEs and result records from group order back to input order, dummy frames' records too.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "demapper.cuh"

namespace s2 {

constexpr int kVcmConfigs = 29 * 4;   // demap table index of (modcod, short, pilots): modcod * 4 + short * 2 + pilots

struct VcmFrame {          // one frame of a call, built on the host
    long long in_off;      // symbols: complex sample of the PLFRAME's start in the input; LLRs: byte offset
    long long llr_off;     // byte offset of its LLR row in the chunk's grouped LLR buffer
    long long bb_src;      // byte offset of its BBFRAME in the chunk's grouped BBFRAME buffer
    long long bb_dst;      // byte offset of its BBFRAME in the caller's packed output
    int cfg;               // demap table index
    int nbytes;            // N: LLR bytes
    int pos;               // its record in the chunk's grouped result buffer; -1: DUMMY PLFRAME
    int kb;                // kbch / 8
};

// nsym_max: largest payload symbol count of the chunk; in_shift / bb_shift: subtracted from in_off / bb_dst (a host
// call holds one chunk of the input and output at a time).  rn: PL scrambling sequence or nullptr.  cudaError_t as int.
int demap_vcm_launch(const DemapDev* table, const uint8_t* rn, const float* in, long long in_shift, const VcmFrame* frames,
                     int nframes, int nsym_max, int8_t* llr, cudaStream_t stream);
int vcm_gather_launch(const int8_t* in, long long in_shift, const VcmFrame* frames, int nframes, int n_max, int8_t* llr,
                      cudaStream_t stream);
// results: dvbs2fec_result records in group order -> results_out[frame], tag = tag_base + frame
int vcm_scatter_launch(const VcmFrame* frames, int nframes, const uint8_t* bb, const void* results, uint8_t* bb_out,
                       long long bb_shift, void* results_out, unsigned long long tag_base, cudaStream_t stream);

}  // namespace s2
