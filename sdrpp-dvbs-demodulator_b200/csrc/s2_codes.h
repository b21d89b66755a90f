// DVB-S2 code parameters and the host-side expansion of the EN 302 307 address tables into the
// layered schedule the CUDA decoder runs.
//
// Reference behaviour mirrored here (cited for parity review, nothing is shared with it):
//   * MODCOD -> constellation / rate / slots / gamma     codings/modcod_to_cfg.cpp:5-140
//   * table iterator + layered permutation               xdsopl-ldpc-pabr/ldpc.hh:25-109,
//                                                        layered_decoder.hh:79-120
//   * BCH parameters per rate                            codings/bbframe_bch.cpp:39-193
#pragma once
#include <cstdint>
#include <vector>

namespace s2 {

constexpr int kGroup = 360;  // EN 302 307: parity addresses repeat with period 360
constexpr int kNumCodes = 21;

// Same numbering as the reference's dvbs2_code_rate_t (dvbs2/dvbs2.h:11-25).
enum Rate { R1_4 = 0, R1_3, R2_5, R1_2, R3_5, R2_3, R3_4, R4_5, R5_6, R7_8, R8_9, R9_10 };
// dvbs2_constellation_t (dvbs2/dvbs2.h:33-39)
enum Constellation { QPSK = 0, PSK8 = 1, APSK16 = 2, APSK32 = 3 };

struct ModcodCfg {
    int modcod;
    bool shortframes, pilots;
    Constellation constellation;
    int bits;         // bits per symbol
    Rate rate;
    int slots;        // 90-symbol data slots per PLFRAME
    float g1, g2;     // APSK ring ratios (0 where unused)
    int code;         // index into code table (0..20), -1 when the standard has no such code
};
// false for modcod outside 1..28 (the reference throws, modcod_to_cfg.cpp:10-11,134-135)
bool modcod_config(int modcod, bool shortframes, bool pilots, ModcodCfg* out);
// complex samples of a PLFRAME of this configuration: PLHEADER, payload and (with pilots) a pilot block of 36 after
// every 16 slots but the last
int plframe_symbols(const ModcodCfg& mc);

struct LayerLink {
    uint16_t group;  // data-bit group g: bits 360g .. 360g+359
    uint16_t shift;  // row j of this layer touches bit 360g + ((j - shift) mod 360)
};

// One LDPC code, expanded.  Row (i, j) (layer i, row j) is the reference's check q*j + i.
struct LdpcCode {
    const char* name;
    int index;
    bool shortframe;
    Rate rate;
    int N, K, R, q;
    int kbch, bch_t, bch_m;          // outer code: kbch info bits, t errors, GF(2^m)
    int links_total;                 // TABLE::LINKS_TOTAL (incl. 2R-1 parity links)
    int max_cnt;                     // max data links per check (= LINKS_MAX_CN - 2)
    std::vector<int> layer_off;      // [q+1] offsets into links
    std::vector<LayerLink> links;    // per layer: its data links, ascending group
    std::vector<uint8_t> layer_nlev; // [q] number of dependency levels in the layer (note N6)
    std::vector<uint8_t> row_level;  // [q*360] level of row (i,j) inside its layer
    int sum_levels;                  // sum of layer_nlev = barriers per iteration
};

// Built once, on first use (thread-safe).
const LdpcCode& ldpc_code(int index);
int code_index(bool shortframe, int rate);  // -1 when there is no table (SURVEY note N4)

// Raw table access for the encoder: calls fn(bit, check) for every data edge, bits ascending.
struct RawTable {
    int N, K, nruns;
    int deg[3], len[3];
    const uint16_t* addr;
};
const RawTable& raw_table(int index);

}  // namespace s2
