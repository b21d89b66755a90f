// K2 host side -- see ldpc_decoder.cuh for the interface and ldpc_v2.cuh / ldpc_v2l.cuh for the kernels.
// Reference semantics: SURVEY.md spec S-LDPC (layered_decoder.hh:23-74,121-133; algorithms.hh:235-256,261-276;
// bbframe_ldpc.cpp:123-139).
#include "ldpc_decoder.cuh"
#include "ldpc_variants.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

namespace s2 {

// Everything a launch needs that depends only on the configured code: built by ldpc_prepare, read by ldpc_launch.
struct LdpcPlan {
    int threads = 0;
    KernelFn2 fn2[2] = {nullptr, nullptr};   // [streamed]
    LdpcParams2 p2;
    size_t smem = 0;
};

namespace {

int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return e ? atoi(e) : dflt;
}

const Variant2* pick2(int max_cnt) {
    const Variant2* parts[4] = {kLdpc2VariantsA, kLdpc2VariantsB, kLdpc2VariantsC, kLdpc2VariantsD};
    const int counts[4] = {kLdpc2VariantsA_n, kLdpc2VariantsB_n, kLdpc2VariantsC_n, kLdpc2VariantsD_n};
    for (int k = 0; k < 4; ++k)
        for (int i = 0; i < counts[k]; ++i)
            if (parts[k][i].cnt >= max_cnt) return &parts[k][i];
    return nullptr;
}
const VariantL* pickl(int max_cnt) {
    const VariantL* parts[2] = {kLdpc2lVariantsA, kLdpc2lVariantsB};
    const int counts[2] = {kLdpc2lVariantsA_n, kLdpc2lVariantsB_n};
    for (int k = 0; k < 2; ++k)
        for (int i = 0; i < counts[k]; ++i)
            if (parts[k][i].cnt == max_cnt) return &parts[k][i];
    return nullptr;
}
bool is_uniform(const LdpcDev& c, int cnt) {
    bool uniform = cnt == c.max_cnt;
    for (int i = 0; i < c.q && uniform; ++i) uniform = (c.layer_off[i + 1] - c.layer_off[i]) == cnt;
    return uniform;
}
KernelFn2 pick_fn2(const LdpcDev& c, bool streamed) {
    if (c.lanes2) {
        const VariantL* v = pickl(c.max_cnt);
        if (!v) return nullptr;
        return (is_uniform(c, v->cnt) && v->uniform[0]) ? v->uniform[streamed] : v->ragged[streamed];
    }
    const Variant2* v = pick2(c.max_cnt);
    if (!v) return nullptr;
    const int oc = c.occ3 ? 1 : 0;
    return (is_uniform(c, v->cnt) && v->uniform[0][0]) ? v->uniform[streamed][oc] : v->ragged[streamed][oc];
}

// Opt every launch of `fn` in to the device's full dynamic shared memory.  The value is the same for every
// code that shares a kernel instantiation, so handles configured for different MODCODs can launch concurrently
// from different host threads without racing on the function attribute.
template <typename Fn>
cudaError_t allow_max_smem(Fn fn) {
    int dev = 0, optin = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e != cudaSuccess) return e;
    cudaFuncAttributes fa;
    e = cudaFuncGetAttributes(&fa, fn);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)fa.sharedSizeBytes);
}

// Barrier elision.  The reference visits rows strictly in order, but two rows commute unless they touch a common
// bit.  Parity bits chain rows of the same thread only (kept in registers), except pty[q-1][j-1] (layer 0 of thread
// j, layer q-1 of thread j-1).  Data bits are shared between threads, group by group: a barrier is needed before a
// layer exactly when it touches a 360-bit group that some layer since the last barrier touched; level-scheduled
// layers are always fenced on both sides.
void plan_barriers(const LdpcDev& c, uint8_t* layer_sync) {
    std::vector<char> seen(c.ngroups, 0);
    bool any = false;
    for (int i = 0; i < c.q; ++i) {
        const bool multi = c.layer_nlev[i] > 1;
        bool conflict = multi;
        for (int k = c.layer_off[i]; k < c.layer_off[i + 1] && !conflict; ++k) conflict = seen[c.links[k] >> 16] != 0;
        if (i > 0 && conflict) {
            layer_sync[i - 1] = 1;
            any = any || (i - 1 <= c.q - 3);
            std::fill(seen.begin(), seen.end(), 0);
        }
        layer_sync[i] = 0;
        for (int k = c.layer_off[i]; k < c.layer_off[i + 1]; ++k) seen[c.links[k] >> 16] = 1;
        if (multi) {
            layer_sync[i] = 1;
            any = any || (i <= c.q - 3);
            std::fill(seen.begin(), seen.end(), 0);
        }
    }
    if (c.q > 0) layer_sync[c.q - 1] = 1;   // end of the pass
    if (!any) layer_sync[0] = 1;            // pty[q-1][j-1]: stored in layer 0, read (by thread j-1) in layer q-1 / prefetched in q-2
}

}  // namespace

// Codes that run faster with one more resident CTA per SM than the default and the register allocation squeezed
// accordingly (three CTAs / 56 registers for CNT <= 9, two CTAs / 80 registers above): their shared memory
// allows it.  Index = code table order B1..B11, C1..C10.
bool ldpc_ctas_wanted3(int code_index) {
    static const bool table[21] = {true,  true,  true,  true,  false, false, false, false, false, false, false,
                                   true,  true,  true,  true,  true,  true,  true,  true,  true,  false};
    static const int force = env_int("DVBS2FEC_LDPC_OCC3", -1);
    if (force >= 0) return force != 0;
    return code_index >= 0 && code_index < 21 && table[code_index];
}

int ldpc_slot_groups_for(int max_cnt, bool lanes2) {
    if (!lanes2) {
        const Variant2* v = pick2(max_cnt);
        return v ? (v->cnt + 2 + 7) / 8 : 0;
    }
    if (!pickl(max_cnt)) return 0;
    const int dh = (max_cnt + 1) / 2 + 1;     // slots per half row
    return 2 * ((dh + 7) / 8);
}

// Codes that run faster with two threads per row (ldpc_v2l.cuh).  Measured with tools/modcod_sweep.py (2048 normal /
// 8192 short frames, fixed noise) against the one-thread-per-row kernel: n3/4 -8 %, n4/5 -8 %, n5/6 -9 %, n8/9 -11 %,
// n9/10 -15 %, s5/6 -14 %, s8/9 -11 % time; the codes with up to eleven data links per row lose 5-30 % (the two
// shuffles and the longer minimum chain outweigh the shorter level steps).  DVBS2FEC_LDPC_LANES2=0|1 overrides (1:
// every code that has such a kernel).  Index = code table order B1..B11, C1..C10.
bool ldpc_use_lanes2(int code_index) {
    static const bool table[21] = {false, false, false, false, false, false, true,  true,  true,  true,  true,
                                   false, false, false, false, false, false, false, false, true,  true};
    static const int force = env_int("DVBS2FEC_LDPC_LANES2", -1);
    if (force >= 0) return force != 0;
    return code_index >= 0 && code_index < 21 && table[code_index];
}

int ldpc_prepare(LdpcDev& c) {
    ldpc_release(c);
    if (c.q < 1 || c.q > kMaxLayers) return (int)cudaErrorInvalidValue;
    const int nlinks = c.layer_off[c.q];
    if (nlinks > kMaxLinks) return (int)cudaErrorInvalidValue;
    LdpcPlan* pl = new LdpcPlan();
    pl->fn2[0] = pick_fn2(c, false);
    pl->fn2[1] = pick_fn2(c, true);
    pl->threads = c.lanes2 ? 720 : 360;   // v2::kLdpcThreads2 / v2::kThreads
    if (!pl->fn2[0] || !pl->fn2[1] || ldpc_slot_groups_for(c.max_cnt, c.lanes2) != c.sg) {
        delete pl;
        return (int)cudaErrorInvalidValue;
    }
    LdpcParams2& p = pl->p2;
    memset(&p, 0, sizeof(p));
    p.N = c.N; p.K = c.K; p.R = c.R; p.q = c.q; p.ngroups = c.ngroups; p.sg = c.sg;
    p.ws_stride = ldpc_workspace_bytes(c);
    p.row_level = c.row_level;
    p.wait_budget = (long long)env_int("DVBS2FEC_STREAM_WAIT_S", 20) * 2000000000ll;
    for (int i = 0; i <= c.q; ++i) p.layer_off[i] = (uint16_t)c.layer_off[i];
    for (int i = 0; i < c.q; ++i) p.layer_nlev[i] = c.layer_nlev[i];
    plan_barriers(c, p.layer_sync);
    for (int i = 0; i < nlinks; ++i) {
        const uint32_t g = c.links[i] >> 16, sh = c.links[i] & 0xFFFFu;
        p.link_group[i] = (uint8_t)g;
        p.link_add[i] = (uint16_t)(720u - 2u * sh);
    }
    cudaError_t e = cudaSuccess;
    for (int st = 0; st < 2 && e == cudaSuccess; ++st) e = allow_max_smem(pl->fn2[st]);
    if (e != cudaSuccess) {
        delete pl;
        return (int)e;
    }
    pl->smem = ldpc_smem_bytes(c);
    c.plan = pl;
    return 0;
}

void ldpc_release(LdpcDev& c) {
    delete c.plan;
    c.plan = nullptr;
}

int ldpc_max_ctas_per_sm(const LdpcDev& c) {
    if (!c.plan) return 0;
    int n = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, c.plan->fn2[0], c.plan->threads, c.plan->smem);
    return n;
}

int ldpc_launch(const LdpcArgs& a, int grid, cudaStream_t stream) {
    const LdpcPlan* pl = a.code.plan;
    if (!pl) return (int)cudaErrorInvalidValue;
    const int st = a.arrived ? 1 : 0;
    LdpcParams2 p = pl->p2;
    p.nframes = a.nframes; p.max_trials = a.max_trials; p.hard_stride = a.hard_stride;
    p.llr_in = a.llr_in; p.hard_out = a.hard_out; p.iters_out = a.iters_out; p.llr_out = a.llr_out;
    p.workspace = a.workspace; p.work_counter = a.work_counter; p.arrived = a.arrived;
    pl->fn2[st]<<<grid, pl->threads, pl->smem, stream>>>(p);
    return (int)cudaGetLastError();
}

}  // namespace s2
