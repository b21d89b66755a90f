// Internal to the LDPC decoder: the kernel parameter block and the table types through which the instantiation
// translation units (ldpc2_inst_*.cu and ldpc2l_inst_*.cu, compiled in parallel) hand their kernels to ldpc_decoder.cu.
#pragma once
#include <cstdint>

namespace s2 {

// Layer tables ride in the kernel parameter (constant bank): uniform, indexed by layer.
constexpr int kMaxLinks = 656;   // B5 (n3/5) has 648 table entries, the largest
constexpr int kMaxLayers = 136;  // B1 (n1/4) has q = 135
struct LdpcParams2 {
    int N, K, R, q, ngroups, sg;
    int nframes, max_trials, hard_stride, pad_;
    long long wait_budget;            // SM clocks a CTA waits for streamed input before it reports kLdpcItersNoInput
    const int8_t* llr_in;
    uint8_t* hard_out;
    int16_t* iters_out;
    int8_t* llr_out;
    uint8_t* workspace;
    unsigned long long ws_stride;
    unsigned int* work_counter;
    const unsigned int* arrived;
    const uint8_t* row_level;
    uint16_t layer_off[kMaxLayers + 1];
    uint8_t layer_nlev[kMaxLayers];
    uint8_t layer_sync[kMaxLayers];   // 1: a CTA barrier must follow this layer
    uint8_t link_group[kMaxLinks];    // data-bit group g of the link; its LLR pairs start at byte 720 g of the shared array
    uint16_t link_add[kMaxLinks];     // 720 - 2 * shift: row j reads byte 720 g + ((2 j + link_add) mod 720)
};
static_assert(sizeof(LdpcParams2) <= 4096, "kernel parameter block must stay within the 4 KB constant window");

using KernelFn2 = void (*)(const LdpcParams2);
// one thread per row (ldpc_v2.cuh)
struct Variant2 {
    int cnt;
    // [streamed input][one more CTA per SM]
    KernelFn2 uniform[2][2];   // every layer has exactly cnt data links per row (all normal codes, 5 short ones)
    KernelFn2 ragged[2][2];    // layers with fewer links exist (short 1/4, 1/2, 3/4, 4/5, 5/6)
};
// one entry per distinct "max data links per row" among the 21 codes, ascending, spread over four translation units
extern const Variant2 kLdpc2VariantsA[], kLdpc2VariantsB[], kLdpc2VariantsC[], kLdpc2VariantsD[];
extern const int kLdpc2VariantsA_n, kLdpc2VariantsB_n, kLdpc2VariantsC_n, kLdpc2VariantsD_n;

// two threads per row (ldpc_v2l.cuh), for the codes with many links per check
struct VariantL {
    int cnt;
    KernelFn2 uniform[2];   // [streamed input]
    KernelFn2 ragged[2];
};
extern const VariantL kLdpc2lVariantsA[], kLdpc2lVariantsB[];
extern const int kLdpc2lVariantsA_n, kLdpc2lVariantsB_n;

}  // namespace s2
