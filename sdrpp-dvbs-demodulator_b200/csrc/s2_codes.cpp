// Host-side DVB-S2 code tables: see s2_codes.h.
#include "s2_codes.h"

#include <algorithm>
#include <cstring>
#include <mutex>

namespace s2 {

namespace {

struct RawDesc {
    const char* tag;
    const char* name;
    int N, K, nruns;
    int deg[3], len[3];
    int off;
};

#define S2_CODE(tag, name, N, K, nruns, d0, l0, d1, l1, d2, l2, off) \
    {#tag, name, N, K, nruns, {d0, d1, d2}, {l0, l1, l2}, off},
const RawDesc kRaw[kNumCodes] = {
#include "s2_ldpc_addr.inc"
};
#undef S2_CODE
#define S2_CODE(...)
#define S2_ADDR_POOL
const uint16_t kS2AddrPool[] = {
#include "s2_ldpc_addr.inc"
};
#undef S2_ADDR_POOL
#undef S2_CODE

// code table order: B1..B11 (normal) then C1..C10 (short)
const int kNormalIdx[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, -1, 9, 10};
const int kShortIdx[12] = {11, 12, 13, 14, 15, 16, 17, 18, 19, -1, 20, -1};
const Rate kRateOfCode[kNumCodes] = {R1_4, R1_3, R2_5, R1_2, R3_5, R2_3, R3_4, R4_5, R5_6, R8_9, R9_10,
                                     R1_4, R1_3, R2_5, R1_2, R3_5, R2_3, R3_4, R4_5, R5_6, R8_9};

std::once_flag g_once[kNumCodes];
LdpcCode g_codes[kNumCodes];
RawTable g_rawtab[kNumCodes];
std::once_flag g_raw_once;

void build(int idx) {
    const RawDesc& rd = kRaw[idx];
    LdpcCode& c = g_codes[idx];
    c.name = rd.name;
    c.index = idx;
    c.shortframe = idx >= 11;
    c.rate = kRateOfCode[idx];
    c.N = rd.N;
    c.K = rd.K;
    c.R = rd.N - rd.K;
    c.q = c.R / kGroup;
    // outer code (EN 302 307 table 5a/5b): t = 12 except normal 2/3, 5/6 (10) and 8/9, 9/10 (8)
    if (c.shortframe) {
        c.bch_t = 12;
        c.bch_m = 14;
        c.kbch = c.K - 168;
    } else {
        c.bch_m = 16;
        c.bch_t = (c.rate == R2_3 || c.rate == R5_6) ? 10 : (c.rate == R8_9 || c.rate == R9_10) ? 8 : 12;
        c.kbch = c.K - 16 * c.bch_t;
    }
    // A table entry x of group g contributes, to layer (x mod q), the link
    // row j -> bit 360 g + ((j - x div q) mod 360).
    std::vector<std::vector<LayerLink>> per_layer(c.q);
    const uint16_t* row = kS2AddrPool + rd.off;
    int g = 0, ndata = 0;
    for (int r = 0; r < rd.nruns; ++r)
        for (int k = 0; k < rd.len[r]; ++k, ++g) {
            for (int d = 0; d < rd.deg[r]; ++d) {
                int x = row[d];
                per_layer[x % c.q].push_back(LayerLink{(uint16_t)g, (uint16_t)(x / c.q)});
                ndata += kGroup;
            }
            row += rd.deg[r];
        }
    c.links_total = ndata + 2 * c.R - 1;
    c.layer_off.assign(c.q + 1, 0);
    c.max_cnt = 0;
    for (int i = 0; i < c.q; ++i) {
        auto& v = per_layer[i];
        std::stable_sort(v.begin(), v.end(), [](const LayerLink& a, const LayerLink& b) { return a.group < b.group; });
        c.layer_off[i + 1] = c.layer_off[i] + (int)v.size();
        c.max_cnt = std::max(c.max_cnt, (int)v.size());
        c.links.insert(c.links.end(), v.begin(), v.end());
    }
    // Dependency levels inside a layer: rows are visited j = 0..359 by the sequential decoder; two rows
    // that touch the same data bit must keep that order, all others commute.  level(j) = 1 + max level
    // of earlier rows sharing a bit.  (Parity links never collide inside a layer.)
    c.layer_nlev.assign(c.q, 1);
    c.row_level.assign((size_t)c.q * kGroup, 0);
    c.sum_levels = 0;
    std::vector<int> next_level(c.K);
    for (int i = 0; i < c.q; ++i) {
        const LayerLink* L = &c.links[c.layer_off[i]];
        int cnt = c.layer_off[i + 1] - c.layer_off[i];
        for (int k = 0; k < cnt; ++k)
            std::fill(next_level.begin() + kGroup * L[k].group, next_level.begin() + kGroup * (L[k].group + 1), 0);
        int nlev = 1;
        for (int j = 0; j < kGroup; ++j) {
            int lvl = 0;
            for (int k = 0; k < cnt; ++k) {
                int b = kGroup * L[k].group + (j - L[k].shift + kGroup) % kGroup;
                lvl = std::max(lvl, next_level[b]);
            }
            for (int k = 0; k < cnt; ++k) {
                int b = kGroup * L[k].group + (j - L[k].shift + kGroup) % kGroup;
                next_level[b] = lvl + 1;
            }
            c.row_level[(size_t)i * kGroup + j] = (uint8_t)lvl;
            nlev = std::max(nlev, lvl + 1);
        }
        c.layer_nlev[i] = (uint8_t)nlev;
        c.sum_levels += nlev;
    }
}

}  // namespace

int code_index(bool shortframe, int rate) {
    if (rate < 0 || rate > 11) return -1;
    return shortframe ? kShortIdx[rate] : kNormalIdx[rate];
}

const LdpcCode& ldpc_code(int index) {
    std::call_once(g_once[index], build, index);
    return g_codes[index];
}

const RawTable& raw_table(int index) {
    std::call_once(g_raw_once, [] {
        for (int i = 0; i < kNumCodes; ++i) {
            RawTable& t = g_rawtab[i];
            t.N = kRaw[i].N;
            t.K = kRaw[i].K;
            t.nruns = kRaw[i].nruns;
            for (int k = 0; k < 3; ++k) {
                t.deg[k] = kRaw[i].deg[k];
                t.len[k] = kRaw[i].len[k];
            }
            t.addr = kS2AddrPool + kRaw[i].off;
        }
    });
    return g_rawtab[index];
}

bool modcod_config(int modcod, bool shortframes, bool pilots, ModcodCfg* out) {
    // EN 302 307 table 12 (MODCOD field); ring ratios from tables 9 and 10.
    struct Row { Constellation c; Rate r; float g1, g2; };
    static const Row rows[29] = {
        {QPSK, R1_4, 0, 0},  // 0: dummy frame, rejected below
        {QPSK, R1_4, 0, 0}, {QPSK, R1_3, 0, 0}, {QPSK, R2_5, 0, 0}, {QPSK, R1_2, 0, 0}, {QPSK, R3_5, 0, 0},
        {QPSK, R2_3, 0, 0}, {QPSK, R3_4, 0, 0}, {QPSK, R4_5, 0, 0}, {QPSK, R5_6, 0, 0}, {QPSK, R8_9, 0, 0},
        {QPSK, R9_10, 0, 0},
        {PSK8, R3_5, 0, 0}, {PSK8, R2_3, 0, 0}, {PSK8, R3_4, 0, 0}, {PSK8, R5_6, 0, 0}, {PSK8, R8_9, 0, 0},
        {PSK8, R9_10, 0, 0},
        {APSK16, R2_3, 3.15f, 0}, {APSK16, R3_4, 2.85f, 0}, {APSK16, R4_5, 2.75f, 0}, {APSK16, R5_6, 2.70f, 0},
        {APSK16, R8_9, 2.60f, 0}, {APSK16, R9_10, 2.57f, 0},
        {APSK32, R3_4, 2.84f, 5.27f}, {APSK32, R4_5, 2.72f, 4.87f}, {APSK32, R5_6, 2.64f, 4.64f},
        {APSK32, R8_9, 2.54f, 4.33f}, {APSK32, R9_10, 2.53f, 4.30f},
    };
    if (modcod < 1 || modcod > 28) return false;
    const Row& r = rows[modcod];
    out->modcod = modcod;
    out->shortframes = shortframes;
    out->pilots = pilots;
    out->constellation = r.c;
    out->bits = 2 + (int)r.c;
    out->rate = r.r;
    out->g1 = r.g1;
    out->g2 = r.g2;
    int n = shortframes ? 16200 : 64800;
    out->slots = n / out->bits / 90;
    out->code = code_index(shortframes, r.r);
    return true;
}

int plframe_symbols(const ModcodCfg& mc) {
    const int nsym = mc.slots * 90;
    return 90 + nsym + (mc.pilots ? 36 * ((nsym - 1) / 1440) : 0);
}

}  // namespace s2
