// K2 -- DVB-S2 LDPC layered offset-min-sum decoder for sm_100a: the host interface of the kernels in ldpc_v2.cuh
// (one thread per check row) and ldpc_v2l.cuh (two threads per row, for the codes with many links per check).
//
// What it must reproduce bit-for-bit (SURVEY.md spec S-LDPC): LDPCDecoder::operator()
// (xdsopl-ldpc-pabr/layered_decoder.hh:121-133) driven per frame the way BBFrameLDPC::decode does
// (codings/bbframe_ldpc.cpp:123-139), with OffsetMinSumAlgorithm<SIMD<int8_t,W>,NormalUpdate,2>
// (algorithms.hh:206-277).  In brief:
//
//   * a CTA owns a PAIR of frames: frame A in the low and frame B in the high 16-bit lane of every register, so
//     the check-node maths runs on the native s16x2 / u16x2 SIMD instructions;
//   * row j of every layer belongs to thread j (360 threads), or to threads 2j and 2j+1 (720).  Rows of one layer
//     that share a data bit are split into dependency levels (s2_codes.cpp) separated by a barrier, which keeps the
//     sequential row order of the reference exactly;
//   * data-bit LLRs and the layer descriptors live in shared memory; messages, parity-bit LLRs and the bit planes
//     of the termination test stream through a per-CTA workspace in global memory;
//   * each frame of the pair stops on its own (iteration count, frozen state), as the reference's
//     lane-0 / blocks=1 call does for a single frame.
//
// Details and measurements: ldpc_v2.cuh, ldpc_v2l.cuh and DESIGN.md section 4.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace s2 {

constexpr int kBitWords = 13;           // 360 hard bits = 12 words (last holds 8) + one zero pad word
constexpr int16_t kLdpcItersNoInput = -2;   // iters_out value of a frame whose streamed input never arrived

struct LdpcPlan;                        // the kernel parameter block and launch choice, built once per configuration

struct LdpcDev {
    int N, K, R, q;
    int ngroups;   // K / 360
    int max_cnt;   // data links per row (max over layers)
    int sg;        // uint4 message slot-groups per row in the workspace: ldpc_slot_groups_for(max_cnt, lanes2)
    bool occ3;     // kernel variant compiled for one more CTA per SM than the default (ldpc_ctas_wanted3(code index))
    bool lanes2;   // two threads per row (ldpc_v2l.cuh) instead of one (ldpc_v2.cuh): ldpc_use_lanes2(code index)
    const LdpcPlan* plan;   // ldpc_prepare(); owned by the caller of ldpc_prepare (ldpc_release)
    // HOST pointers: copied into the kernel parameter block (constant bank) at every launch
    const uint32_t* links;       // per layer: (group << 16) | shift
    const int* layer_off;        // [q + 1]
    const uint8_t* layer_nlev;   // [q]
    // DEVICE pointer
    const uint8_t* row_level;    // [q * 360] dependency level of row (i,j) inside layer i
};
bool ldpc_ctas_wanted3(int code_index);     // measured per code, see ldpc_decoder.cu
bool ldpc_use_lanes2(int code_index);       // likewise
// uint4 message slot-groups per row of the kernel instantiation that serves max_cnt data links (0 = unsupported)
int ldpc_slot_groups_for(int max_cnt, bool lanes2);
// Builds the parameter block (layer tables, barrier elision) and opts the kernel in to the device's full
// shared memory, once; ldpc_launch then only patches the per-launch pointers.  Returns cudaError_t as int.
int ldpc_prepare(LdpcDev& code);
void ldpc_release(LdpcDev& code);

struct LdpcArgs {
    LdpcDev code;
    const int8_t* llr_in;   // [nframes][N]
    int nframes;
    int max_trials;
    uint8_t* hard_out;      // [nframes][hard_stride] MSB-first hard decisions of the K systematic bits
    int hard_stride;        // bytes per frame in hard_out (>= K/8)
    int16_t* iters_out;     // [nframes]        iterations executed, -1 = never converged
    int8_t* llr_out;        // [nframes][N] or nullptr: posterior LLRs (what the reference leaves in place)
    uint8_t* workspace;     // gridDim.x * ldpc_workspace_bytes(code)
    unsigned int* work_counter;  // zeroed before launch
    const unsigned int* arrived; // nullptr, or a device word the input copy raises: frames of llr_in delivered so far
};

inline size_t ldpc_workspace_bytes(const LdpcDev& c) {
    // message records, parity LLR pairs, the bit planes of the full termination test, per-thread constants
    const size_t b = (size_t)c.q * c.sg * 360 * 16 + (((size_t)c.R * 2 + 15) & ~(size_t)15) +
                     (size_t)2 * (c.ngroups + c.q) * kBitWords * 4 + 32 + (size_t)768 * 16;
    return (b + 255) & ~(size_t)255;
}
inline size_t ldpc_smem_bytes(const LdpcDev& c) {
    // LLR pairs + the 361 pty[q-1][.] pairs handed between neighbouring threads + layer descriptors
    if (c.lanes2) return (size_t)c.K * 2 + 768 + (size_t)c.q * (4 + 2 * ((2 * ((c.max_cnt + 1) / 2) + 3) & ~3)) * 4 + 64;
    return (size_t)c.K * 2 + 768 + (size_t)c.q * ((1 + 2 * c.max_cnt + 3) & ~3) * 4 + 64;
}

// returns cudaError_t as int; launches the kernel instantiation ldpc_prepare chose
int ldpc_launch(const LdpcArgs& args, int grid, cudaStream_t stream);
int ldpc_max_ctas_per_sm(const LdpcDev& code);

}  // namespace s2
