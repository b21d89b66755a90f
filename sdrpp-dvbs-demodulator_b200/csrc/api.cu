// C ABI of libdvbs2fec.so (include/dvbs2fec.h): handle, per-GPU contexts, the frame-batching
// queue and the by-frame multi-GPU dispatcher.  Everything that computes runs in the CUDA kernels
// (ldpc_decoder.cu, bch_decoder.cu, demapper.cu); there is no CPU fallback -- without a device every
// compute entry point returns DVBS2FEC_ENODEV.
#include "../../include/dvbs2fec.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <climits>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <deque>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>
#include <emmintrin.h>

#include "abi_util.h"
#include "bch_decoder.cuh"
#include "demapper.cuh"
#include "host_tables.h"
#include "ldpc_decoder.cuh"
#include "s2_codes.h"
#include "ts_parser.cuh"
#include "vcm.cuh"

using namespace s2;

namespace {
thread_local char g_err[512] = "";
}  // namespace

int s2::fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

namespace {

constexpr int kStages = 4; // page-locked staging batches per handle (frame queue)
constexpr int kPiece = 256; // frames per piece of a streamed input copy
constexpr int kSlots = 2;  // double buffering per device: copy of batch k+1 overlaps kernels of batch k

// what a decode call gets per frame
enum class Input { llr, sym, idx };   // LLRs, PLFRAME symbols, LUT coordinates of the payload symbols

struct Slot {
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    // streamed LLR input: pieces go out on their own stream while the LDPC kernel is already running
    cudaStream_t copy = nullptr;
    cudaEvent_t armed = nullptr;
    DevBuf<unsigned int> arrived;        // frames delivered so far (device word the kernel polls)
    DevBuf<uint8_t> ts;                  // fused TS output of the batch (queue, TS mode)
    DevBuf<int> ts_len;
    PinBuf<unsigned int> arrived_vals;   // the values the copy engine writes there, one per piece
    DevBuf<int8_t> llr;
    DevBuf<float> sym;
    DevBuf<uint8_t> idx;                 // LUT coordinates per payload symbol (quantised symbols path)
    DevBuf<uint8_t> hard;
    DevBuf<int16_t> iters;
    DevBuf<int16_t> corr;
    DevBuf<uint8_t> bb;
    DevBuf<dvbs2fec_result> res;
    DevBuf<uint8_t> workspace;
    DevBuf<unsigned int> counter;
    PinBuf<uint8_t> h_in;
    PinBuf<uint8_t> h_bb;
    PinBuf<dvbs2fec_result> h_res;
    // VCM calls: the chunk's input as it arrives (host entries), its packed output (host entries), the frame records
    DevBuf<uint8_t> vin;
    DevBuf<uint8_t> vbb;
    DevBuf<dvbs2fec_result> vres;
    DevBuf<VcmFrame> vmeta;
    PinBuf<VcmFrame> h_vmeta;
    bool vmeta_copying = false;          // device entry: `armed` marks the end of the last copy out of h_vmeta
    // pending copy-out of a staged batch
    uint8_t* user_bb = nullptr;
    dvbs2fec_result* user_res = nullptr;
    int pending = 0;
    size_t bb_bytes = 0;
    bool staged_out = true;
};

struct BchTabDev {
    DevBuf<uint16_t> crc, basis;
};

struct CodeTables {  // what the kernels of one LDPC code need on one device; ldpc.links points into links
    LdpcDev ldpc{};
    BchDev bch{};
    int grid = 0;
    int hard_stride = 0;
    std::vector<uint32_t> links;
    DevBuf<uint8_t> row_level;
    ~CodeTables() { ldpc_release(ldpc); }
};

struct DevCtx {
    int device = 0;
    int sms = 0;
    // [0,kSlots): synchronous entry points; [kSlots,2 kSlots): the frame queue's worker; [2 kSlots]: the device entry
    // point (dvbs2fec_decode_batch_device), whose users on different streams are chained through slot.done
    Slot slot[2 * kSlots + 1];
    std::mutex dev_mu;
    bool dev_used = false;
    // prepared codes by code index (prepare_code); entries stay where they are while others are added
    std::map<int, CodeTables> codes;
    std::map<int, BchTabDev> bch;           // key m*100+t
    DevBuf<uint16_t> gf_log[2], gf_exp[2];  // [0]: m=14, [1]: m=16
    DevBuf<uint8_t> prbs;
    DevBuf<uint8_t> pl_rn;                  // PL scrambling sequence of the handle's Gold code (empty: off)
    std::map<int, DevBuf<uint32_t>> luts;   // key modcod constellation/gamma: modcod number
    // current configuration; the queue worker reaches the code only through cur
    const CodeTables* cur = nullptr;
    DemapDev demap{};
    // VCM calls: demap records by (modcod, short, pilots) -- see vcm.cuh
    DevBuf<DemapDev> vcm_demap;
    bool vcm_demap_ok[kVcmConfigs] = {};
    ~DevCtx() {   // the buffers free themselves after this, with the device current
        cudaSetDevice(device);
        for (int k = 0; k < 2 * kSlots + 1; ++k) {
            Slot& s = slot[k];
            if (s.copy && !(k >= 1 && k < kSlots)) {   // (slots 1..kSlots-1 borrow slot 0's)
                cudaStreamSynchronize(s.copy);
                cudaStreamDestroy(s.copy);
            }
            if (s.stream) {
                cudaStreamSynchronize(s.stream);
                cudaStreamDestroy(s.stream);
            }
            if (s.done) cudaEventDestroy(s.done);
            if (s.armed) cudaEventDestroy(s.armed);
        }
    }
};

}  // namespace

// BBFRAME -> TS parser object (row 8(f)-1); entry points further down
struct dvbs2fec_ts_parser {
    int device = 0;
    int kb = 0, max_dfl = 0;
    cudaStream_t stream = nullptr;
    DevBuf<TsState> state;
    DevBuf<TsPlan> plan;
    DevBuf<uint32_t> meta;
    DevBuf<uint8_t> bb, out;
    PinBuf<int> h_produced;
    // GSE branch (ts_parser.cu): reassembly state and buffers persist, the rest is per-call scratch
    int gse_pool = 0;                  // < 0: GSE frames are only counted; 0: default sizing; > 0: packets per device-side call
    DevBuf<GseState> gstate;
    DevBuf<uint8_t> gbuf, g_sync;
    DevBuf<int> g_doff, g_before, g_nxt, g_aux, g_aux2;
    DevBuf<GseDesc> g_desc;
    DevBuf<GseOut> g_out;
    DevBuf<uint32_t> g_crc0, g_xpow;
    ~dvbs2fec_ts_parser() {
        cudaSetDevice(device);
        if (stream) {
            cudaStreamSynchronize(stream);
            cudaStreamDestroy(stream);
        }
    }
};

struct dvbs2fec_handle {
    dvbs2fec_config cfg{};
    std::vector<std::unique_ptr<DevCtx>> devs;
    ModcodCfg mc{};
    const LdpcCode* code = nullptr;
    int max_trials = 25;
    int plsyms = 0;
    int last_launches = 0;
    int pl_codenum = -1;                // Gold code of the PL descrambler in K1, -1 = inputs are descrambled
    // fused TS output of the queue (dvbs2fec_set_ts_output): K6 runs behind K3 on the device
    bool ts_output = false;
    dvbs2fec_ts_parser* ts = nullptr;
    cudaEvent_t ts_done = nullptr;      // K6 of the previous batch has finished (its state carries over)
    bool configured = false;
    bool profiling = false;
    struct Span { int kind; cudaEvent_t a, b; };
    std::vector<Span> spans;
    std::mutex span_mu;
    // ---- queue
    std::mutex mu;
    std::mutex submit_mu;               // serialises producers (the reference has one per instance)
    std::condition_variable cv_work, cv_done;
    std::thread worker;
    bool stop = false, flush_req = false, busy = false;
    bool acquired = false;              // a producer is writing a frame straight into the batch being filled
    // Frames wait in page-locked staging batches ("stages"): submit copies a frame straight into the stage being
    // filled, the worker hands a full (or timed-out) stage to the GPUs with asynchronous copies in both
    // directions, collect copies BBFRAMEs out of finished stages.  Stages cycle free -> fill -> ready -> inflight
    // -> done -> free; at most kSlots are in flight, so the copy-in of one overlaps the kernels of the other.
    struct Stage {
        PinBuf<uint8_t> in, bb, ts;
        PinBuf<dvbs2fec_result> res;
        PinBuf<int> ts_len;
        int ts_taken = 0, res_taken = 0;
        bool has_ts = false;
        std::vector<uint64_t> tags;
        int n = 0, taken = 0, cap = 0;
        Input kind = Input::llr;
        int rc = 0;
        size_t kb = 0, in_bytes = 0;
        std::atomic<int> outstanding{0};   // device shares still running
        std::chrono::steady_clock::time_point first;
    };
    struct ShareDone { dvbs2fec_handle* h; int stage; };
    Stage stages[kStages];
    ShareDone share_done[kStages];
    std::deque<int> st_free, st_ready, st_inflight, st_done;
    int st_fill = -1;
    uint64_t launch_seq = 0;
    ~dvbs2fec_handle() {
        {
            std::unique_lock<std::mutex> lk(mu);
            stop = true;
            cv_work.notify_all();
        }
        if (worker.joinable()) worker.join();
        for (auto& d : devs) {   // work enqueued on caller-owned streams by the device entry point, before anything goes
            cudaSetDevice(d->device);
            cudaDeviceSynchronize();
        }
        dvbs2fec_ts_destroy(ts);
        if (ts_done) cudaEventDestroy(ts_done);
        for (auto& sp : spans) {
            cudaEventDestroy(sp.a);
            cudaEventDestroy(sp.b);
        }
    }
};

static int ts_args(dvbs2fec_ts_parser* p, const uint8_t* d_bb, int cnt, uint8_t* d_out, int out_cap, int* d_produced, TsArgs* out);

namespace {

// LDPC plan, grid, hard stride and link words of code c on device d into T
int prepare_ldpc(DevCtx& d, const LdpcCode& c, CodeTables& T) {
    CU(T.row_level.reserve(c.row_level.size()));
    CU(upload(T.row_level.p, c.row_level.data(), c.row_level.size()));
    for (const LayerLink& l : c.links) T.links.push_back(((uint32_t)l.group << 16) | l.shift);
    T.hard_stride = ((c.K / 8) + 15) & ~15;
    LdpcDev& L = T.ldpc;
    L.N = c.N; L.K = c.K; L.R = c.R; L.q = c.q;
    L.ngroups = c.K / kGroup;
    L.max_cnt = c.max_cnt;
    L.lanes2 = ldpc_use_lanes2(c.index) && ldpc_slot_groups_for(c.max_cnt, true) > 0;
    L.sg = ldpc_slot_groups_for(c.max_cnt, L.lanes2);
    L.occ3 = ldpc_ctas_wanted3(c.index);
    if (!L.sg) return fail(DVBS2FEC_EINVAL, "no LDPC kernel for %d links per row", c.max_cnt);
    L.links = T.links.data();
    L.layer_off = c.layer_off.data();
    L.layer_nlev = c.layer_nlev.data();
    L.row_level = T.row_level.p;
    if (int e = ldpc_prepare(L)) return fail(DVBS2FEC_ECUDA, "LDPC kernel set-up: %s", cudaGetErrorString((cudaError_t)e));
    int per_sm = ldpc_max_ctas_per_sm(L);
    if (per_sm <= 0) return fail(DVBS2FEC_ENODEV, "LDPC kernel does not fit on device %d (%s)", d.device,
                                 cudaGetErrorString(cudaGetLastError()));
    T.grid = d.sms * per_sm;
    return 0;
}

// BCH, GF and BB scrambler tables of code c on device d into B
int prepare_bch(DevCtx& d, const LdpcCode& c, BchDev& B) {
    const int m = c.bch_m, t = c.bch_t, fi = (m == 16);
    const GfHost& gf = gf_host(m);
    if (!d.gf_log[fi].p) {
        CU(d.gf_log[fi].reserve(gf.log.size()));
        CU(d.gf_exp[fi].reserve(gf.exp.size()));
        CU(upload(d.gf_log[fi].p, gf.log.data(), gf.log.size() * 2));
        CU(upload(d.gf_exp[fi].p, gf.exp.data(), gf.exp.size() * 2));
    }
    BchTabDev& bt = d.bch[m * 100 + t];
    if (!bt.crc.p) {
        const BchHost& bh = bch_host(m, t);
        CU(bt.crc.reserve(bh.crc.size()));
        CU(bt.basis.reserve(bh.basis.size()));
        CU(upload(bt.crc.p, bh.crc.data(), bh.crc.size() * 2));
        CU(upload(bt.basis.p, bh.basis.data(), bh.basis.size() * 2));
    }
    if (!d.prbs.p) {
        const auto& seq = bb_prbs();
        CU(d.prbs.reserve(seq.size()));
        CU(upload(d.prbs.p, seq.data(), seq.size()));
    }
    B.gf.m = m; B.gf.N = gf.N; B.gf.log = d.gf_log[fi].p; B.gf.exp = d.gf_exp[fi].p;
    B.t = t; B.nbch = c.K; B.kbch = c.kbch;
    B.prefix = gf.N - c.K;
    B.crc = bt.crc.p; B.basis = bt.basis.p; B.prbs = d.prbs.p;
    return 0;
}

// Code ci on device d, prepared on first use (LDPC plan and grid, BCH record, hard stride, link words) -- the one
// store of prepared codes for the single-MODCOD configuration and VCM calls alike
int prepare_code(DevCtx& d, int ci, const CodeTables** out) {
    auto it = d.codes.find(ci);
    if (it == d.codes.end()) {
        it = d.codes.try_emplace(ci).first;
        const LdpcCode& c = ldpc_code(ci);
        int rc = prepare_ldpc(d, c, it->second);
        if (!rc) rc = prepare_bch(d, c, it->second.bch);
        if (rc) {
            d.codes.erase(it);
            return rc;
        }
    }
    *out = &it->second;
    return 0;
}

// demapper record of configuration mc (code c, plsyms complex samples per PLFRAME) on device d into D
int prepare_demap(DevCtx& d, const ModcodCfg& mc, const LdpcCode& c, int plsyms, const uint8_t* rn, DemapDev& D) {
    ConstellationHost ch = make_constellation(mc.constellation, mc.g1, mc.g2);
    D.constellation = (int)mc.constellation;
    D.bits = mc.bits;
    D.N = c.N;
    D.nsym = c.N / mc.bits;
    D.reversed_cols = (mc.constellation == PSK8 && mc.rate == R3_5);
    D.pilots = mc.pilots;
    D.plframe_syms = plsyms;
    D.amp = ch.amp; D.prescale = ch.prescale; D.sca = ch.sca;
    for (int i = 0; i < 32; ++i) {
        D.pts[2 * i] = i < ch.states ? ch.re[i] : 0.f;
        D.pts[2 * i + 1] = i < ch.states ? ch.im[i] : 0.f;
    }
    D.lut = nullptr;
    D.rn = rn;
    if (mc.constellation != APSK32) {
        int key = (mc.constellation == APSK16) ? mc.modcod : (int)mc.constellation;  // 16APSK: one LUT per gamma
        DevBuf<uint32_t>& lut = d.luts[key];
        if (!lut.p) {
            std::vector<uint32_t> tab = demap_lut(ch);
            CU(lut.reserve(tab.size()));
            CU(upload(lut.p, tab.data(), tab.size() * 4));
        }
        D.lut = lut.p;
    }
    return 0;
}

int setup_device_tables(dvbs2fec_handle* h, DevCtx& d) {
    CU(cudaSetDevice(d.device));
    if (int rc = prepare_code(d, h->code->index, &d.cur)) return rc;
    return prepare_demap(d, h->mc, *h->code, h->plsyms, h->pl_codenum >= 0 ? d.pl_rn.p : nullptr, d.demap);
}

size_t input_frame_bytes(const dvbs2fec_handle* h, Input kind) {
    return kind == Input::sym ? (size_t)h->plsyms * 8 : kind == Input::idx ? (size_t)(h->code->N / h->mc.bits) * 2 : (size_t)h->code->N;
}

// where a batch of input of this kind goes in slot s
void* slot_input(Slot& s, Input kind) {
    return kind == Input::sym ? (void*)s.sym.p : kind == Input::idx ? (void*)s.idx.p : (void*)s.llr.p;
}

int reserve_slot(dvbs2fec_handle* h, DevCtx& d, Slot& s, int nframes, Input kind, bool host_staging) {
    const LdpcCode& c = *h->code;
    CU(cudaSetDevice(d.device));
    CU(s.llr.reserve((size_t)nframes * c.N));
    if (kind == Input::sym) CU(s.sym.reserve((size_t)nframes * h->plsyms * 2));
    if (kind == Input::idx) CU(s.idx.reserve((size_t)nframes * input_frame_bytes(h, Input::idx)));
    CU(s.hard.reserve((size_t)nframes * d.cur->hard_stride));
    CU(s.iters.reserve(nframes));
    CU(s.corr.reserve(nframes));
    CU(s.bb.reserve((size_t)nframes * (c.kbch / 8)));
    CU(s.res.reserve(nframes));
    CU(s.workspace.reserve((size_t)d.cur->grid * ldpc_workspace_bytes(d.cur->ldpc)));
    CU(s.counter.reserve(1));
    if (host_staging) {
        size_t in_bytes = (size_t)nframes * input_frame_bytes(h, kind);
        CU(s.h_in.reserve(in_bytes));
        CU(s.h_bb.reserve((size_t)nframes * (c.kbch / 8)));
        CU(s.h_res.reserve(nframes));
    }
    return 0;
}

// kernel-time spans for dvbs2fec_kernel_times (kind 0 demap, 1 LDPC, 2 BCH); several threads (one per GPU, the queue
// worker) may add some
struct SpanMark {
    dvbs2fec_handle* h;
    cudaStream_t st;
    dvbs2fec_handle::Span cur{0, nullptr, nullptr};
    void operator()(int kind, bool begin) {
        if (!h->profiling) return;
        if (begin) {
            cur = dvbs2fec_handle::Span{kind, nullptr, nullptr};
            cudaEventCreate(&cur.a);
            cudaEventCreate(&cur.b);
            cudaEventRecord(cur.a, st);
        } else {
            cudaEventRecord(cur.b, st);
            std::lock_guard<std::mutex> lk(h->span_mu);
            h->spans.push_back(cur);
        }
    }
};

// The argument blocks of LDPC and BCH for n frames of code T in slot s: the fields that depend on the code and the slot.
// The frames' hard decisions start at byte hard_off of s.hard, their iteration counts at entry `at` of s.iters, and
// LDPC hands them out through work counter k (a VCM chunk places the frames of each code so).
LdpcArgs ldpc_args(const dvbs2fec_handle* h, const CodeTables& T, const Slot& s, const int8_t* llr, int n,
                   size_t hard_off = 0, int at = 0, int k = 0) {
    LdpcArgs la{};
    la.code = T.ldpc;
    la.llr_in = llr;
    la.nframes = n;
    la.max_trials = h->max_trials;
    la.hard_out = s.hard.p + hard_off;
    la.hard_stride = T.hard_stride;
    la.iters_out = s.iters.p + at;
    la.workspace = s.workspace.p;
    la.work_counter = s.counter.p + k;
    return la;
}
BchArgs bch_args(const CodeTables& T, const Slot& s, int n, size_t hard_off = 0, int at = 0) {
    BchArgs ba{};
    ba.code = T.bch;
    ba.hard = s.hard.p + hard_off;
    ba.hard_stride = T.hard_stride;
    ba.nframes = n;
    ba.ldpc_iters = s.iters.p + at;
    ba.descramble = 1;
    return ba;
}
int ldpc_grid(const CodeTables& T, int n) { return std::min(T.grid, (n + 1) / 2); }

// LDPC then BCH/descramble on st for n frames of code T, placed in slot s as ldpc_args says: BBFRAMEs to bb, records
// (tags tag_base + i) to res
int enqueue_ldpc_bch(dvbs2fec_handle* h, const CodeTables& T, Slot& s, cudaStream_t st, int* launches, const int8_t* llr,
                     int n, const unsigned int* arrived, uint8_t* bb, dvbs2fec_result* res, unsigned long long tag_base,
                     size_t hard_off = 0, int at = 0, int k = 0) {
    SpanMark mark{h, st};
    CU(cudaMemsetAsync(s.counter.p + k, 0, sizeof(unsigned int), st));
    LdpcArgs la = ldpc_args(h, T, s, llr, n, hard_off, at, k);
    la.arrived = arrived;
    mark(1, true);
    int e = ldpc_launch(la, ldpc_grid(T, n), st);
    mark(1, false);
    if (e) return fail(DVBS2FEC_ECUDA, "ldpc launch: %s", cudaGetErrorString((cudaError_t)e));
    ++*launches;
    BchArgs ba = bch_args(T, s, n, hard_off, at);
    ba.tag_base = tag_base;
    ba.bb_out = bb;
    ba.results = res;
    mark(2, true);
    e = bch_launch(ba, st);
    mark(2, false);
    if (e) return fail(DVBS2FEC_ECUDA, "bch launch: %s", cudaGetErrorString((cudaError_t)e));
    ++*launches;
    return 0;
}

// enqueue demap (symbol and coordinate input) + LDPC + BCH/descramble for n frames of the current code already on
// the device
int enqueue_chain(dvbs2fec_handle* h, DevCtx& d, Slot& s, Input kind, const void* in, int n, uint8_t* d_bb,
                  dvbs2fec_result* d_res, cudaStream_t st, int* launches, uint64_t tag_base,
                  const unsigned int* arrived = nullptr) {
    const int8_t* llr = static_cast<const int8_t*>(in);
    if (kind != Input::llr) {
        SpanMark mark{h, st};
        mark(0, true);
        int e = kind == Input::sym ? demap_launch(d.demap, static_cast<const float*>(in), n, s.llr.p, st)
                                   : demap_idx_launch(d.demap, static_cast<const uint8_t*>(in), n, s.llr.p, st);
        mark(0, false);
        if (e) return fail(DVBS2FEC_ECUDA, "demap launch: %s", cudaGetErrorString((cudaError_t)e));
        llr = s.llr.p;
        ++*launches;
    }
    return enqueue_ldpc_bch(h, *d.cur, s, st, launches, llr, n, arrived, d_bb, d_res, tag_base);
}

// Streamed LLR input.  arm: zero the arrival word on the copy stream and make the compute stream wait for that,
// so the kernel launched next can never see a stale count.  feed: copy the frames piece by piece, raising the
// arrival word behind every piece (copies on one stream complete in order).  The LDPC kernel hands out frame
// pairs in order and waits for the word to cover a pair before loading it, so decoding starts when the first
// piece has landed instead of after the whole batch.  Rule: every copy a kernel will wait for is enqueued BEFORE
// the kernel is launched -- a spinning kernel must never depend on a host call that is still to come (that call
// could block behind the kernel, e.g. in lazy module loading or cudaFree).
int arm_streamed_input(Slot& s, int nframes) {
    CU(s.arrived.reserve(1));
    CU(s.arrived_vals.reserve((size_t)(nframes + kPiece - 1) / kPiece + 1));
    CU(cudaMemsetAsync(s.arrived.p, 0, sizeof(unsigned int), s.copy));
    CU(cudaEventRecord(s.armed, s.copy));
    CU(cudaStreamWaitEvent(s.stream, s.armed, 0));
    return 0;
}
int feed_streamed_input(Slot& s, const uint8_t* src, int nframes, size_t frame_bytes, bool src_pinned) {
    for (int f0 = 0, k = 0; f0 < nframes; f0 += kPiece, ++k) {
        const int n = std::min(kPiece, nframes - f0);
        const uint8_t* from = src + (size_t)f0 * frame_bytes;
        if (!src_pinned) {   // pageable caller memory goes through the slot's page-locked staging buffer
            memcpy(s.h_in.p + (size_t)f0 * frame_bytes, from, (size_t)n * frame_bytes);
            from = s.h_in.p + (size_t)f0 * frame_bytes;
        }
        CU(cudaMemcpyAsync(s.llr.p + (size_t)f0 * frame_bytes, from, (size_t)n * frame_bytes, cudaMemcpyHostToDevice, s.copy));
        s.arrived_vals.p[k] = (unsigned int)(f0 + n);
        CU(cudaMemcpyAsync(s.arrived.p, &s.arrived_vals.p[k], sizeof(unsigned int), cudaMemcpyHostToDevice, s.copy));
    }
    return 0;
}

bool is_pinned(const void* p) {
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

int finish_slot(dvbs2fec_handle* h, Slot& s) {
    if (!s.pending) return 0;
    CU(cudaEventSynchronize(s.done));
    if (s.user_bb && s.staged_out) memcpy(s.user_bb, s.h_bb.p, s.bb_bytes);
    if (s.user_res && s.staged_out) memcpy(s.user_res, s.h_res.p, (size_t)s.pending * sizeof(dvbs2fec_result));
    s.pending = 0;
    return 0;
}

// The end of a chunk of a synchronous call: its outputs (bb_bytes of BBFRAMEs, m records) go to the caller, straight
// into page-locked caller memory or else through the slot's staging (finish_slot copies them out), and the slot is
// pending until `done`.
int chunk_out(Slot& s, uint8_t* user_bb, const uint8_t* d_bb, size_t bb_bytes, dvbs2fec_result* user_res,
              const dvbs2fec_result* d_res, int m, bool pin_out) {
    s.user_bb = user_bb;
    s.user_res = user_res;
    s.staged_out = !pin_out;
    if (user_bb && bb_bytes) CU(cudaMemcpyAsync(pin_out ? user_bb : s.h_bb.p, d_bb, bb_bytes, cudaMemcpyDeviceToHost, s.stream));
    if (user_res)
        CU(cudaMemcpyAsync(pin_out ? (void*)user_res : (void*)s.h_res.p, d_res, (size_t)m * sizeof(dvbs2fec_result),
                           cudaMemcpyDeviceToHost, s.stream));
    CU(cudaEventRecord(s.done, s.stream));
    s.pending = m;
    s.bb_bytes = bb_bytes;
    return 0;
}

// Error exit of the synchronous entry points: nothing asynchronous may outlive the call -- copies into the caller's
// buffers that were already enqueued are waited for, and no slot keeps a pointer to them (a later call would copy into
// freed memory).
struct HostSlotsAbort {
    DevCtx& d;
    bool armed = true;
    ~HostSlotsAbort() {
        if (!armed) return;
        char keep[sizeof(g_err)];
        memcpy(keep, g_err, sizeof keep);
        for (int k = 0; k < kSlots; ++k) {
            Slot& s = d.slot[k];
            cudaStreamSynchronize(s.copy);
            cudaStreamSynchronize(s.stream);
            s.pending = 0;
            s.user_bb = nullptr;
            s.user_res = nullptr;
        }
        cudaGetLastError();
        memcpy(g_err, keep, sizeof keep);
    }
};

// frames [0, n) of one device's share, host buffers in and out
int run_device_share(dvbs2fec_handle* h, DevCtx& d, Input kind, const void* input, int n, uint8_t* bb,
                     dvbs2fec_result* res, uint64_t tag0, int* launches) {
    if (n <= 0) return 0;
    CU(cudaSetDevice(d.device));
    const LdpcCode& c = *h->code;
    const size_t kb = c.kbch / 8;
    const size_t in_frame_bytes = input_frame_bytes(h, kind);
    const uint8_t* in = static_cast<const uint8_t*>(input);
    const int chunk = std::min(h->cfg.max_batch, n);
    for (int k = 0; k < kSlots; ++k) {
        int rc = reserve_slot(h, d, d.slot[k], chunk, kind, true);
        if (rc) return rc;
    }
    // caller buffers that are already page-locked are used directly; pageable ones are staged
    const bool pin_in = is_pinned(in);
    const bool pin_out = (!bb || is_pinned(bb)) && (!res || is_pinned(res));
    int which = 0, rc = 0;
    HostSlotsAbort abort_guard{d};
    for (int f0 = 0; f0 < n; f0 += chunk, which ^= 1) {
        Slot& s = d.slot[which];
        const int m = std::min(chunk, n - f0);
        if ((rc = finish_slot(h, s))) return rc;
        const uint8_t* src = in + (size_t)f0 * in_frame_bytes;
        void* dst = slot_input(s, kind);
        if (kind == Input::llr) {   // the kernel starts on the first piece
            if ((rc = arm_streamed_input(s, m))) return rc;
            if ((rc = feed_streamed_input(s, src, m, in_frame_bytes, pin_in))) return rc;
            rc = enqueue_chain(h, d, s, kind, dst, m, s.bb.p, s.res.p, s.stream, launches, tag0 + f0, s.arrived.p);
        } else {
            if (!pin_in) {
                memcpy(s.h_in.p, src, (size_t)m * in_frame_bytes);
                src = s.h_in.p;
            }
            CU(cudaMemcpyAsync(dst, src, (size_t)m * in_frame_bytes, cudaMemcpyHostToDevice, s.stream));
            rc = enqueue_chain(h, d, s, kind, dst, m, s.bb.p, s.res.p, s.stream, launches, tag0 + f0);
        }
        if (rc) return rc;
        rc = chunk_out(s, bb ? bb + (size_t)f0 * kb : nullptr, s.bb.p, (size_t)m * kb, res ? res + f0 : nullptr, s.res.p, m, pin_out);
        if (rc) return rc;
    }
    for (int k = 0; k < kSlots; ++k)
        if ((rc = finish_slot(h, d.slot[k]))) return rc;
    abort_guard.armed = false;
    return 0;
}

int decode_host(dvbs2fec_handle* h, Input kind, const void* in, int n, uint8_t* bb, dvbs2fec_result* res) {
    if (!h || !h->configured) return fail(DVBS2FEC_EINVAL, "set_modcod has not been called");
    if (n < 0 || !in) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (kind == Input::idx && h->mc.constellation == APSK32) return fail(DVBS2FEC_EINVAL, "32APSK has no LUT in the reference: send symbols");
    if (h->devs.empty()) return fail(DVBS2FEC_ENODEV, "no CUDA device");
    const int nd = (int)h->devs.size();
    const size_t kb = h->code->kbch / 8;
    const size_t in_stride = input_frame_bytes(h, kind);
    h->last_launches = 0;
    if (nd == 1) {
        int launches = 0;
        int rc = run_device_share(h, *h->devs[0], kind, in, n, bb, res, 0, &launches);
        h->last_launches = launches;
        return rc;
    }
    // by-frame sharding: contiguous shares, one host thread per GPU, no cross-GPU exchange
    std::vector<std::thread> th;
    std::vector<int> rcs(nd, 0), ln(nd, 0);
    std::vector<std::string> errs(nd);
    int per = (n + nd - 1) / nd;
    for (int k = 0; k < nd; ++k) {
        int f0 = std::min(n, k * per), f1 = std::min(n, f0 + per);
        th.emplace_back([=, &rcs, &ln, &errs] {
            rcs[k] = run_device_share(h, *h->devs[k], kind, static_cast<const uint8_t*>(in) + (size_t)f0 * in_stride, f1 - f0,
                                      bb ? bb + (size_t)f0 * kb : nullptr, res ? res + f0 : nullptr, (uint64_t)f0, &ln[k]);
            if (rcs[k]) errs[k] = g_err;
        });
    }
    for (auto& t : th) t.join();
    for (int k = 0; k < nd; ++k) {
        h->last_launches += ln[k];
        if (rcs[k]) return fail(rcs[k], "device %d: %s", h->devs[k]->device, errs[k].c_str());
    }
    return 0;
}

// stream callback at the end of one device's share of a stage (no CUDA calls allowed in here)
void CUDART_CB stage_share_done(void* arg) {
    auto* a = static_cast<dvbs2fec_handle::ShareDone*>(arg);
    if (a->h->stages[a->stage].outstanding.fetch_sub(1) == 1) {
        std::lock_guard<std::mutex> lk(a->h->mu);
        a->h->cv_work.notify_all();
    }
}

// hand stage `st` to the GPUs: contiguous shares by frame, everything asynchronous on slot kSlots + which
void launch_stage(dvbs2fec_handle* h, int st, int which) {
    dvbs2fec_handle::Stage& S = h->stages[st];
    const int nd = (int)h->devs.size();
    const int per = (S.n + nd - 1) / nd;
    int shares = 0;
    for (int k = 0; k < nd; ++k) shares += std::min(S.n, k * per) < S.n;
    S.outstanding.store(shares);
    S.rc = 0;
    h->last_launches = 0;
    for (int k = 0; k < nd; ++k) {
        const int f0 = std::min(S.n, k * per), f1 = std::min(S.n, f0 + per), m = f1 - f0;
        if (m <= 0) continue;
        DevCtx& d = *h->devs[k];
        Slot& s = d.slot[kSlots + which];
        auto body = [&]() -> int {
            int rc = reserve_slot(h, d, s, std::max(m, h->cfg.max_batch), S.kind, false);
            if (rc) return rc;
            // plain copy-in on the slot's stream: with two batches in flight per handle (and other handles' work
            // beside them) the copy of one batch already overlaps the kernels of another, and a kernel that
            // starts early and waits for streamed input would only hold SMs that a neighbour could use
            // (measured: 8 handles at max_batch 4096, 588 k frames/s plain vs 405 k streamed)
            void* dst = slot_input(s, S.kind);
            CU(cudaMemcpyAsync(dst, S.in.p + (size_t)f0 * S.in_bytes, (size_t)m * S.in_bytes, cudaMemcpyHostToDevice, s.stream));
            rc = enqueue_chain(h, d, s, S.kind, dst, m, s.bb.p, s.res.p, s.stream, &h->last_launches, (uint64_t)f0);
            if (rc) return rc;
            CU(cudaMemcpyAsync(S.bb.p + (size_t)f0 * S.kb, s.bb.p, (size_t)m * S.kb, cudaMemcpyDeviceToHost, s.stream));
            CU(cudaMemcpyAsync(S.res.p + f0, s.res.p, (size_t)m * sizeof(dvbs2fec_result), cudaMemcpyDeviceToHost, s.stream));
            if (S.has_ts) {   // K6 behind K3, on the BBFRAMEs still in device memory; its state runs through all batches
                dvbs2fec_ts_parser* tp = h->ts;
                const int ts_cap = (int)((size_t)m * S.kb + 376);   // room for everything: see dvbs2fec_ts_work
                CU(s.ts.reserve((size_t)std::max(m, h->cfg.max_batch) * S.kb + 376));
                CU(s.ts_len.reserve(1));
                CU(cudaStreamWaitEvent(s.stream, h->ts_done, 0));
                const int saved_pool = tp->gse_pool;
                tp->gse_pool = -1;   // the fused queue output is TS only (GSE frames are counted): its room is sized for TS
                TsArgs ta;
                rc = ts_args(tp, s.bb.p, m, s.ts.p, ts_cap, s.ts_len.p, &ta);
                tp->gse_pool = saved_pool;
                if (rc) return rc;
                int e = ts_launch(ta, s.stream);
                if (e) return fail(DVBS2FEC_ECUDA, "ts launch: %s", cudaGetErrorString((cudaError_t)e));
                h->last_launches += 3;
                CU(cudaEventRecord(h->ts_done, s.stream));
                CU(cudaMemcpyAsync(S.ts.p, s.ts.p, (size_t)ts_cap, cudaMemcpyDeviceToHost, s.stream));
                CU(cudaMemcpyAsync(S.ts_len.p, s.ts_len.p, sizeof(int), cudaMemcpyDeviceToHost, s.stream));
            }
            CU(cudaLaunchHostFunc(s.stream, stage_share_done, &h->share_done[st]));
            return 0;
        };
        int rc = body();
        if (rc) {   // this share never got its completion callback; what it did enqueue still writes into the stage
            S.rc = rc;
            cudaStreamSynchronize(s.stream);
            cudaGetLastError();
            S.outstanding.fetch_sub(1);
        }
    }
}

void worker_main(dvbs2fec_handle* h) {
    std::unique_lock<std::mutex> lk(h->mu);
    const auto latency = std::chrono::microseconds(h->cfg.max_latency_us);
    for (;;) {
        // publish finished stages in launch order
        bool published = false;
        while (!h->st_inflight.empty() && h->stages[h->st_inflight.front()].outstanding.load() == 0) {
            h->st_done.push_back(h->st_inflight.front());
            h->st_inflight.pop_front();
            published = true;
        }
        if (published) h->cv_done.notify_all();
        // next stage to launch: a full one, else the one being filled once it is old enough (or on flush)
        int st = -1;
        if ((int)h->st_inflight.size() < kSlots) {
            if (!h->st_ready.empty()) {
                st = h->st_ready.front();
                h->st_ready.pop_front();
            } else if (h->st_fill >= 0 && h->stages[h->st_fill].n > 0 && !h->acquired &&
                       (h->flush_req || std::chrono::steady_clock::now() >= h->stages[h->st_fill].first + latency)) {
                st = h->st_fill;
                h->st_fill = -1;
            }
        }
        if (st >= 0) {
            h->st_inflight.push_back(st);
            const int which = (int)(h->launch_seq++ % kSlots);
            lk.unlock();
            launch_stage(h, st, which);
            lk.lock();
            continue;
        }
        if (h->stop) return;
        const bool filling = h->st_fill >= 0 && h->stages[h->st_fill].n > 0;
        if (!filling && h->st_ready.empty() && h->st_inflight.empty()) {
            h->flush_req = false;
            h->cv_done.notify_all();
        }
        if (filling && !h->acquired && (int)h->st_inflight.size() < kSlots)
            h->cv_work.wait_until(lk, h->stages[h->st_fill].first + latency);
        else
            h->cv_work.wait(lk);
    }
}

void drain_queue(dvbs2fec_handle* h) {
    std::unique_lock<std::mutex> lk(h->mu);
    if (!h->worker.joinable()) return;
    h->flush_req = true;
    h->cv_work.notify_all();
    h->cv_done.wait(lk, [h] {
        return h->st_ready.empty() && h->st_inflight.empty() && (h->st_fill < 0 || h->stages[h->st_fill].n == 0);
    });
    h->flush_req = false;
}

// ---------------------------------------------------------------- VCM / ACM batches (vcm.cuh)
struct VcmDesc {   // one frame of a call; code -1: DUMMY PLFRAME
    int cfg, code, plsyms, nsym, N, kb;
};
struct VcmGroup {  // the frames of one LDPC code inside a chunk, in input order
    int code, cnt, p0;                  // p0: first record in group order
    size_t llr_off, hard_off, bb_off;   // byte offsets of the group in the chunk's scratch
};
struct VcmChunk {
    int f0, f1;
    bool fast;                          // one code, no dummy frame: nothing to reorder
    int nsym_max, n_max;
    std::vector<VcmGroup> groups;       // largest first
};
struct VcmPlan {
    std::vector<VcmDesc> fr;
    std::vector<int64_t> sym_off, llr_off, bb_off;   // [n + 1]
    std::vector<VcmFrame> rec;                       // [n]
    std::vector<VcmChunk> chunks;
    size_t llr_bytes = 0, hard_bytes = 0, bb_bytes = 0, workspace = 0, in_max = 0, out_max = 0;   // per chunk, maximum
    int max_chunk = 0;
};

constexpr int kDummySyms = 90 + 36 * 90;   // DUMMY PLFRAME: header + 36 slots

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// validates every descriptor and fills the layout; nothing else is touched on error
int vcm_parse(int n, const int32_t* desc, VcmPlan& P) {
    if (n < 0) return fail(DVBS2FEC_EINVAL, "frame count %d is negative", n);
    if (n > 0 && !desc) return fail(DVBS2FEC_EINVAL, "desc is NULL");
    P.fr.resize(n);
    P.sym_off.assign(n + 1, 0);
    P.llr_off.assign(n + 1, 0);
    P.bb_off.assign(n + 1, 0);
    for (int i = 0; i < n; ++i) {
        const int modcod = desc[4 * i];
        const bool sh = desc[4 * i + 1] != 0, pi = desc[4 * i + 2] != 0;
        VcmDesc& f = P.fr[i];
        if (modcod == 0) {
            f = VcmDesc{0, -1, kDummySyms, 0, 0, 0};
        } else {
            ModcodCfg mc;
            if (modcod < 0 || modcod > 28 || !modcod_config(modcod, sh, pi, &mc) || mc.code < 0)
                return fail(DVBS2FEC_EINVAL, "frame %d: MODCOD %d with %s frames has no LDPC code", i, modcod,
                            sh ? "short" : "normal");
            const LdpcCode& c = ldpc_code(mc.code);
            f = VcmDesc{modcod * 4 + sh * 2 + pi, mc.code, plframe_symbols(mc), c.N / mc.bits, c.N, c.kbch / 8};
        }
        P.sym_off[i + 1] = P.sym_off[i] + f.plsyms;
        P.llr_off[i + 1] = P.llr_off[i] + f.N;
        P.bb_off[i + 1] = P.bb_off[i] + f.kb;
    }
    return 0;
}

// Prepares every code and (symbol input) demap record the call uses, then splits it into chunks of at most chunk
// frames and lays out each chunk's groups and frame records.
int vcm_plan(dvbs2fec_handle* h, DevCtx& d, VcmPlan& P, bool sym, int chunk) {
    CU(cudaSetDevice(d.device));
    const int n = (int)P.fr.size();
    bool code_seen[kNumCodes] = {}, cfg_seen[kVcmConfigs] = {};
    for (const VcmDesc& f : P.fr)
        if (f.code >= 0) code_seen[f.code] = cfg_seen[f.cfg] = true;
    for (int ci = 0; ci < kNumCodes; ++ci) {
        if (!code_seen[ci]) continue;
        const CodeTables* T = nullptr;
        if (int rc = prepare_code(d, ci, &T)) return rc;
        P.workspace = std::max(P.workspace, (size_t)T->grid * ldpc_workspace_bytes(T->ldpc));
    }
    if (sym) {
        CU(d.vcm_demap.reserve(kVcmConfigs));
        for (int cfg = 0; cfg < kVcmConfigs; ++cfg) {
            if (!cfg_seen[cfg] || d.vcm_demap_ok[cfg]) continue;
            ModcodCfg mc;
            modcod_config(cfg / 4, (cfg & 2) != 0, (cfg & 1) != 0, &mc);
            DemapDev D{};
            if (int rc = prepare_demap(d, mc, ldpc_code(mc.code), plframe_symbols(mc), nullptr, D)) return rc;
            CU(upload(d.vcm_demap.p + cfg, &D, sizeof D));
            d.vcm_demap_ok[cfg] = true;
        }
    }
    P.rec.resize(n);
    for (int f0 = 0; f0 < n; f0 += chunk) {
        VcmChunk c{f0, std::min(n, f0 + chunk), false, 0, 0, {}};
        int gi[kNumCodes];
        std::fill(gi, gi + kNumCodes, -1);
        bool dummy = false;
        for (int f = c.f0; f < c.f1; ++f) {
            const int code = P.fr[f].code;
            if (code < 0) {
                dummy = true;
                continue;
            }
            if (gi[code] < 0) {
                gi[code] = (int)c.groups.size();
                c.groups.push_back(VcmGroup{code, 0, 0, 0, 0, 0});
            }
            ++c.groups[gi[code]].cnt;
        }
        std::stable_sort(c.groups.begin(), c.groups.end(), [](const VcmGroup& a, const VcmGroup& b) { return a.cnt > b.cnt; });
        c.fast = c.groups.size() == 1 && !dummy;
        size_t lo = 0, ho = 0, bo = 0;
        int p = 0;
        for (size_t g = 0; g < c.groups.size(); ++g) {
            VcmGroup& G = c.groups[g];
            const LdpcCode& lc = ldpc_code(G.code);
            gi[G.code] = (int)g;
            G.p0 = p;
            G.llr_off = lo;
            G.hard_off = ho;
            G.bb_off = bo;
            lo += align256((size_t)G.cnt * lc.N);
            ho += (size_t)G.cnt * d.codes.at(G.code).hard_stride;
            bo += align256((size_t)G.cnt * (lc.kbch / 8));
            p += G.cnt;
        }
        int fill[kNumCodes] = {};
        for (int f = c.f0; f < c.f1; ++f) {
            const VcmDesc& D = P.fr[f];
            VcmFrame& r = P.rec[f];
            r.in_off = sym ? P.sym_off[f] : P.llr_off[f];
            r.bb_dst = P.bb_off[f];
            r.cfg = D.cfg;
            r.nbytes = D.N;
            r.kb = D.kb;
            r.pos = -1;
            r.llr_off = r.bb_src = 0;
            if (D.code < 0) continue;
            const VcmGroup& G = c.groups[gi[D.code]];
            const int i = fill[D.code]++;
            r.pos = G.p0 + i;
            r.llr_off = (long long)(G.llr_off + (size_t)i * D.N);
            r.bb_src = (long long)(G.bb_off + (size_t)i * D.kb);
            c.nsym_max = std::max(c.nsym_max, D.nsym);
            c.n_max = std::max(c.n_max, D.N);
        }
        if (sym || !c.fast) P.llr_bytes = std::max(P.llr_bytes, lo);   // a fast chunk of LLRs is decoded where it lies
        P.hard_bytes = std::max(P.hard_bytes, ho);
        P.bb_bytes = std::max(P.bb_bytes, bo);
        P.in_max = std::max(P.in_max, sym ? (size_t)(P.sym_off[c.f1] - P.sym_off[c.f0]) * 8 : (size_t)(P.llr_off[c.f1] - P.llr_off[c.f0]));
        P.out_max = std::max(P.out_max, (size_t)(P.bb_off[c.f1] - P.bb_off[c.f0]));
        P.max_chunk = std::max(P.max_chunk, c.f1 - c.f0);
        P.chunks.push_back(std::move(c));
    }
    return 0;
}

// scratch of slot s for the plan; host: also the staging of the chunk's input and output, records per chunk
int vcm_reserve(Slot& s, const VcmPlan& P, bool host) {
    CU(s.llr.reserve(P.llr_bytes));
    CU(s.hard.reserve(P.hard_bytes));
    CU(s.iters.reserve(P.max_chunk));
    CU(s.bb.reserve(P.bb_bytes));
    CU(s.res.reserve(P.max_chunk));
    CU(s.workspace.reserve(P.workspace));
    CU(s.counter.reserve(kNumCodes));
    const size_t nrec = host ? (size_t)P.max_chunk : P.rec.size();
    CU(s.vmeta.reserve(nrec));
    CU(s.h_vmeta.reserve(nrec));
    if (host) {
        CU(s.vin.reserve(P.in_max));
        CU(s.vbb.reserve(P.out_max));
        CU(s.vres.reserve(P.max_chunk));
        CU(s.h_in.reserve(P.in_max));
        CU(s.h_bb.reserve(P.out_max));
        CU(s.h_res.reserve(P.max_chunk));
    }
    return 0;
}

// Enqueues one chunk on st.  in: the input, in_off - in_shift indexes it (complex samples or bytes); rec: the chunk's
// records on the device; bb_out / res_out: BBFRAMEs at bb_off - bb_shift and the records of frames f0.. (may be null).
// Launches: demap or gather (unless the chunk is a fast one of LLRs, or all dummy), LDPC and BCH per code, scatter
// (unless fast): 2k + 2 for k codes, 2 / 3 for a fast chunk of LLRs / symbols, 1 for a chunk of dummy frames.
int vcm_chunk(dvbs2fec_handle* h, DevCtx& d, Slot& s, const VcmPlan& P, const VcmChunk& c, bool sym, const void* in,
              long long in_shift, const VcmFrame* rec, uint8_t* bb_out, long long bb_shift, dvbs2fec_result* res_out,
              cudaStream_t st, int* launches) {
    SpanMark mark{h, st};
    const int m = c.f1 - c.f0;
    const int8_t* llr = s.llr.p;
    if (!c.groups.empty()) {
        int e = 0;
        if (sym) {
            mark(0, true);
            e = demap_vcm_launch(d.vcm_demap.p, h->pl_codenum >= 0 ? d.pl_rn.p : nullptr, static_cast<const float*>(in), in_shift,
                                 rec, m, c.nsym_max, s.llr.p, st);
            mark(0, false);
            ++*launches;
        } else if (!c.fast) {
            mark(0, true);
            e = vcm_gather_launch(static_cast<const int8_t*>(in), in_shift, rec, m, c.n_max, s.llr.p, st);
            mark(0, false);
            ++*launches;
        } else {
            llr = static_cast<const int8_t*>(in) + (P.llr_off[c.f0] - in_shift);
        }
        if (e) return fail(DVBS2FEC_ECUDA, "VCM demap / gather launch: %s", cudaGetErrorString((cudaError_t)e));
    }
    for (size_t g = 0; g < c.groups.size(); ++g) {
        const VcmGroup& G = c.groups[g];
        // a fast chunk is in input order: straight into the caller's buffers
        uint8_t* bb = c.fast ? (bb_out ? bb_out + (P.bb_off[c.f0] - bb_shift) : nullptr) : s.bb.p + G.bb_off;
        dvbs2fec_result* res = c.fast ? res_out : s.res.p + G.p0;
        int rc = enqueue_ldpc_bch(h, d.codes.at(G.code), s, st, launches, llr + G.llr_off, G.cnt, nullptr, bb, res,
                                  c.fast ? (unsigned long long)c.f0 : 0, G.hard_off, G.p0, (int)g);
        if (rc) return rc;
    }
    if (!c.fast) {
        mark(2, true);
        int e = vcm_scatter_launch(rec, m, s.bb.p, s.res.p, bb_out, bb_shift, res_out, (unsigned long long)c.f0, st);
        mark(2, false);
        if (e) return fail(DVBS2FEC_ECUDA, "VCM scatter launch: %s", cudaGetErrorString((cudaError_t)e));
        ++*launches;
    }
    return 0;
}

// host buffers: chunk by chunk through the two synchronous slots, like run_device_share (no streamed input)
int vcm_host(dvbs2fec_handle* h, int n, const int32_t* desc, const void* in, bool sym, uint8_t* bb, dvbs2fec_result* res) {
    if (!h) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    VcmPlan P;
    if (int rc = vcm_parse(n, desc, P)) return rc;
    if (!in && (sym ? P.sym_off[n] : P.llr_off[n]) > 0) return fail(DVBS2FEC_EINVAL, "input is NULL");
    if (h->devs.empty()) return fail(DVBS2FEC_ENODEV, "no CUDA device");
    h->last_launches = 0;
    if (n == 0) return 0;
    DevCtx& d = *h->devs[0];
    if (int rc = vcm_plan(h, d, P, sym, std::max(h->cfg.max_batch, 1))) return rc;
    for (int k = 0; k < kSlots; ++k)
        if (int rc = vcm_reserve(d.slot[k], P, true)) return rc;
    const bool pin_in = is_pinned(in);
    const bool pin_out = (!bb || is_pinned(bb)) && (!res || is_pinned(res));
    const std::vector<int64_t>& in_off = sym ? P.sym_off : P.llr_off;
    const size_t unit = sym ? 8 : 1;
    int which = 0, rc = 0, launches = 0;
    HostSlotsAbort abort_guard{d};
    for (const VcmChunk& c : P.chunks) {
        Slot& s = d.slot[which];
        which ^= 1;
        const int m = c.f1 - c.f0;
        if ((rc = finish_slot(h, s))) return rc;
        const size_t in_bytes = (size_t)(in_off[c.f1] - in_off[c.f0]) * unit;
        const uint8_t* src = static_cast<const uint8_t*>(in) + (size_t)in_off[c.f0] * unit;
        if (!pin_in && in_bytes) {
            memcpy(s.h_in.p, src, in_bytes);
            src = s.h_in.p;
        }
        if (in_bytes) CU(cudaMemcpyAsync(s.vin.p, src, in_bytes, cudaMemcpyHostToDevice, s.stream));
        if (sym || !c.fast) {
            memcpy(s.h_vmeta.p, &P.rec[c.f0], (size_t)m * sizeof(VcmFrame));
            CU(cudaMemcpyAsync(s.vmeta.p, s.h_vmeta.p, (size_t)m * sizeof(VcmFrame), cudaMemcpyHostToDevice, s.stream));
        }
        rc = vcm_chunk(h, d, s, P, c, sym, s.vin.p, in_off[c.f0], s.vmeta.p, bb ? s.vbb.p : nullptr, P.bb_off[c.f0],
                       res ? s.vres.p : nullptr, s.stream, &launches);
        if (rc) return rc;
        rc = chunk_out(s, bb ? bb + P.bb_off[c.f0] : nullptr, s.vbb.p, (size_t)(P.bb_off[c.f1] - P.bb_off[c.f0]),
                       res ? res + c.f0 : nullptr, s.vres.p, m, pin_out);
        if (rc) return rc;
    }
    for (int k = 0; k < kSlots; ++k)
        if ((rc = finish_slot(h, d.slot[k]))) return rc;
    abort_guard.armed = false;
    h->last_launches = launches;
    return 0;
}

// The bracket of the device entry points.  They have their own slot (LDPC workspace, hard decisions, work counter),
// never shared with the synchronous entry points.  Calls may come on different streams: each one waits for the
// previous user of the slot (begin) before it touches it, so they are serialised on the device (not on the host) and
// none of them can race on it, and marks its own end (end) after its last enqueue, also when it fails part-way.
struct DeviceCall {
    DevCtx& d;
    cudaStream_t st;
    Slot& s = d.slot[2 * kSlots];
    std::lock_guard<std::mutex> serial{d.dev_mu};
    int begin() {
        if (d.dev_used) CU(cudaStreamWaitEvent(st, s.done, 0));
        return 0;
    }
    int end(int rc) {
        CU(cudaEventRecord(s.done, st));
        d.dev_used = true;
        return rc;
    }
};

// device buffers, through the device entry points' bracket
int vcm_device(dvbs2fec_handle* h, int n, const int32_t* desc, const void* d_in, bool sym, uint8_t* d_bb,
               dvbs2fec_result* d_res, void* cuda_stream) {
    if (!h) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    VcmPlan P;
    if (int rc = vcm_parse(n, desc, P)) return rc;
    if (!d_in && (sym ? P.sym_off[n] : P.llr_off[n]) > 0) return fail(DVBS2FEC_EINVAL, "input is NULL");
    if (h->devs.empty()) return fail(DVBS2FEC_ENODEV, "no CUDA device");
    DevCtx& d = *h->devs[0];
    DeviceCall call{d, (cudaStream_t)cuda_stream};
    Slot& s = call.s;
    cudaStream_t st = call.st;
    h->last_launches = 0;
    if (n == 0) return 0;
    if (int rc = vcm_plan(h, d, P, sym, std::max(h->cfg.max_batch, 1))) return rc;
    // the records go out of a page-locked buffer that the previous call's copy may still be reading
    if (s.vmeta_copying) CU(cudaEventSynchronize(s.armed));
    s.vmeta_copying = false;
    if (int rc = vcm_reserve(s, P, false)) return rc;
    if (int rc = call.begin()) return rc;
    bool need_rec = sym;
    for (const VcmChunk& c : P.chunks) need_rec |= !c.fast;
    if (need_rec) {
        memcpy(s.h_vmeta.p, P.rec.data(), (size_t)n * sizeof(VcmFrame));
        CU(cudaMemcpyAsync(s.vmeta.p, s.h_vmeta.p, (size_t)n * sizeof(VcmFrame), cudaMemcpyHostToDevice, st));
        CU(cudaEventRecord(s.armed, st));
        s.vmeta_copying = true;
    }
    int rc = 0;
    for (size_t k = 0; k < P.chunks.size() && !rc; ++k) {
        const VcmChunk& c = P.chunks[k];
        rc = vcm_chunk(h, d, s, P, c, sym, d_in, 0, s.vmeta.p + c.f0, d_bb, 0, d_res ? d_res + c.f0 : nullptr, st,
                       &h->last_launches);
    }
    return call.end(rc);
}

// frames of the current configuration in device buffers, enqueued on the caller's stream chunk by chunk
int decode_device(dvbs2fec_handle* h, Input kind, const void* d_in, int n, uint8_t* d_bb, dvbs2fec_result* d_res,
                  void* cuda_stream) {
    if (!h || !h->configured || !d_in || n < 0) return fail(DVBS2FEC_EINVAL, "bad arguments");
    DevCtx& d = *h->devs[0];
    DeviceCall call{d, (cudaStream_t)cuda_stream};
    if (int rc = call.begin()) return rc;
    const int chunk = std::min(n, std::max(h->cfg.max_batch, 1));
    int rc = reserve_slot(h, d, call.s, chunk, Input::llr, false);
    if (rc) return rc;
    const size_t kb = h->code->kbch / 8, in_bytes = input_frame_bytes(h, kind);
    h->last_launches = 0;
    for (int f0 = 0; f0 < n && !rc; f0 += chunk) {
        int m = std::min(chunk, n - f0);
        rc = enqueue_chain(h, d, call.s, kind, static_cast<const uint8_t*>(d_in) + (size_t)f0 * in_bytes, m,
                           d_bb ? d_bb + (size_t)f0 * kb : nullptr, d_res ? d_res + f0 : nullptr, call.st, &h->last_launches,
                           (uint64_t)f0);
    }
    return call.end(rc);
}

}  // namespace

extern "C" {

const char* dvbs2fec_last_error(void) { return g_err; }

int dvbs2fec_create(const dvbs2fec_config* cfg, dvbs2fec_handle** out) {
    if (!out) return fail(DVBS2FEC_EINVAL, "out is NULL");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(DVBS2FEC_ENODEV, "no CUDA device: %s", cudaGetErrorString(cudaGetLastError()));
    std::unique_ptr<dvbs2fec_handle> h(new dvbs2fec_handle());
    if (cfg) h->cfg = *cfg;
    if (h->cfg.max_batch <= 0) h->cfg.max_batch = 1024;
    if (h->cfg.max_latency_us <= 0) h->cfg.max_latency_us = 2000;
    if (h->cfg.max_trials <= 0) h->cfg.max_trials = 25;
    h->max_trials = h->cfg.max_trials;
    std::vector<int> ids;
    if (h->cfg.n_devices <= 0) {
        int cur = 0;
        cudaGetDevice(&cur);
        ids.push_back(cur);
    } else {
        for (int i = 0; i < h->cfg.n_devices && i < 8; ++i) ids.push_back(h->cfg.devices[i]);
    }
    for (int id : ids) {
        if (id < 0 || id >= ndev) return fail(DVBS2FEC_EINVAL, "device %d out of range (%d present)", id, ndev);
        std::unique_ptr<DevCtx> d(new DevCtx());
        d->device = id;
        CU(cudaSetDevice(id));
        cudaDeviceProp prop;
        CU(cudaGetDeviceProperties(&prop, id));
        if (prop.major < 10)
            return fail(DVBS2FEC_ENODEV, "device %d is sm_%d%d; this library carries sm_100a code only", id, prop.major,
                        prop.minor);
        d->sms = prop.multiProcessorCount;
        for (int k = 0; k < 2 * kSlots + 1; ++k) {
            CU(cudaStreamCreateWithFlags(&d->slot[k].stream, cudaStreamNonBlocking));
            CU(cudaEventCreateWithFlags(&d->slot[k].done, cudaEventDisableTiming));
            // The two slots of the synchronous host path share ONE input-copy stream: their chunks then cross PCIe one
            // after the other, in the order the kernels consume them.  With a stream each, the copy engines interleave
            // the two transfers, the first kernel is fed at half the link rate (slower than it decodes) and the call
            // takes a third longer (measured: e2e 17.4 -> see profiles/r02_bench_line.json).
            if (k >= 1 && k < kSlots)
                d->slot[k].copy = d->slot[0].copy;
            else
                CU(cudaStreamCreateWithFlags(&d->slot[k].copy, cudaStreamNonBlocking));
            CU(cudaEventCreateWithFlags(&d->slot[k].armed, cudaEventDisableTiming));
        }
        h->devs.push_back(std::move(d));
    }
    for (int k = 0; k < kStages; ++k) {
        h->share_done[k] = {h.get(), k};
        h->st_free.push_back(k);
    }
    *out = h.release();
    return 0;
}

void dvbs2fec_destroy(dvbs2fec_handle* h) { delete h; }

int dvbs2fec_set_modcod(dvbs2fec_handle* h, int modcod, int shortframes, int pilots, int max_trials) {
    if (!h) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    ModcodCfg mc;
    if (!modcod_config(modcod, shortframes != 0, pilots != 0, &mc))
        return fail(DVBS2FEC_EINVAL, "MODCOD %d is outside 1..28", modcod);
    if (mc.code < 0)
        return fail(DVBS2FEC_EINVAL, "MODCOD %d has no %s-frame LDPC code in EN 302 307", modcod,
                    shortframes ? "short" : "normal");
    drain_queue(h);
    h->mc = mc;
    h->code = &ldpc_code(mc.code);
    if (max_trials > 0) h->max_trials = max_trials;
    h->plsyms = plframe_symbols(mc);
    for (auto& d : h->devs) {
        int rc = setup_device_tables(h, *d);
        if (rc) return rc;
    }
    h->configured = true;
    if (h->ts_output) {   // like setFrameSize on a MODCOD change: the parser starts over
        int rc = dvbs2fec_ts_set_frame_size(h->ts, h->code->kbch);
        if (rc) return rc;
    }
    return 0;
}

int dvbs2fec_set_pl_scrambling(dvbs2fec_handle* h, int codenum) {
    if (!h) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    if (codenum > 262141) return fail(DVBS2FEC_EINVAL, "Gold code number %d outside 0..262141", codenum);
    drain_queue(h);
    h->pl_codenum = codenum < 0 ? -1 : codenum;
    for (auto& dp : h->devs) {
        DevCtx& d = *dp;
        CU(cudaSetDevice(d.device));
        if (codenum >= 0) {
            // longest PLFRAME payload: 64800 / 2 symbols + 22 pilot blocks of 36
            std::vector<uint8_t> rn = pl_scrambling_rn(codenum, 32400 + 36 * 22 + 8);
            CU(d.pl_rn.reserve(rn.size()));
            CU(upload(d.pl_rn.p, rn.data(), rn.size()));
        }
        d.demap.rn = codenum >= 0 ? d.pl_rn.p : nullptr;
    }
    return 0;
}

int dvbs2fec_kbch(const dvbs2fec_handle* h) { return (h && h->configured) ? h->code->kbch : DVBS2FEC_EINVAL; }
int dvbs2fec_kldpc(const dvbs2fec_handle* h) { return (h && h->configured) ? h->code->K : DVBS2FEC_EINVAL; }
int dvbs2fec_nldpc(const dvbs2fec_handle* h) { return (h && h->configured) ? h->code->N : DVBS2FEC_EINVAL; }
int dvbs2fec_plframe_symbols(const dvbs2fec_handle* h) { return (h && h->configured) ? h->plsyms : DVBS2FEC_EINVAL; }
int dvbs2fec_last_launch_count(const dvbs2fec_handle* h) { return h ? h->last_launches : 0; }

int dvbs2fec_set_profiling(dvbs2fec_handle* h, int on) {
    if (!h) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    h->profiling = on != 0;
    return 0;
}
int dvbs2fec_kernel_times(dvbs2fec_handle* h, float* demap_ms, float* ldpc_ms, float* bch_ms, int* launches) {
    if (!h) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    float acc[3] = {0, 0, 0};
    int n = 0;
    std::vector<dvbs2fec_handle::Span> spans;
    {
        std::lock_guard<std::mutex> lk(h->span_mu);
        spans.swap(h->spans);
    }
    for (auto& sp : spans) {
        float ms = 0;
        CU(cudaEventSynchronize(sp.b));
        CU(cudaEventElapsedTime(&ms, sp.a, sp.b));
        acc[sp.kind] += ms;
        cudaEventDestroy(sp.a);
        cudaEventDestroy(sp.b);
        ++n;
    }
    if (demap_ms) *demap_ms = acc[0];
    if (ldpc_ms) *ldpc_ms = acc[1];
    if (bch_ms) *bch_ms = acc[2];
    if (launches) *launches = n;
    return 0;
}

int dvbs2fec_bb_to_soft(dvbs2fec_handle* h, const float* plframes, int n, int8_t* llr_out) {
    if (!h || !h->configured || !plframes || !llr_out || n < 0) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (n == 0) return 0;
    DevCtx& d = *h->devs[0];
    Slot& s = d.slot[0];
    int rc = reserve_slot(h, d, s, n, Input::sym, false);
    if (rc) return rc;
    CU(cudaMemcpyAsync(s.sym.p, plframes, (size_t)n * h->plsyms * 8, cudaMemcpyHostToDevice, s.stream));
    int e = demap_launch(d.demap, s.sym.p, n, s.llr.p, s.stream);
    if (e) return fail(DVBS2FEC_ECUDA, "demap launch: %s", cudaGetErrorString((cudaError_t)e));
    CU(cudaMemcpyAsync(llr_out, s.llr.p, (size_t)n * h->code->N, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    return 0;
}

int dvbs2fec_ldpc_decode(dvbs2fec_handle* h, int8_t* frames, int n, int max_trials, int16_t* iters) {
    if (!h || !h->configured || !frames || n < 0) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (n == 0) return 0;
    DevCtx& d = *h->devs[0];
    Slot& s = d.slot[0];
    int rc = reserve_slot(h, d, s, n, Input::llr, false);
    if (rc) return rc;
    const size_t bytes = (size_t)n * h->code->N;
    CU(cudaMemcpyAsync(s.llr.p, frames, bytes, cudaMemcpyHostToDevice, s.stream));
    CU(cudaMemsetAsync(s.counter.p, 0, sizeof(unsigned int), s.stream));
    LdpcArgs la = ldpc_args(h, *d.cur, s, s.llr.p, n);
    if (max_trials > 0) la.max_trials = max_trials;
    la.llr_out = s.llr.p;  // in place, like BBFrameLDPC::decode
    int e = ldpc_launch(la, ldpc_grid(*d.cur, n), s.stream);
    if (e) return fail(DVBS2FEC_ECUDA, "ldpc launch: %s", cudaGetErrorString((cudaError_t)e));
    CU(cudaMemcpyAsync(frames, s.llr.p, bytes, cudaMemcpyDeviceToHost, s.stream));
    if (iters) CU(cudaMemcpyAsync(iters, s.iters.p, (size_t)n * 2, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    return 0;
}

int dvbs2fec_bch_decode(dvbs2fec_handle* h, uint8_t* frames, int n, int16_t* corrections) {
    if (!h || !h->configured || !frames || n < 0) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (n == 0) return 0;
    DevCtx& d = *h->devs[0];
    Slot& s = d.slot[0];
    int rc = reserve_slot(h, d, s, n, Input::llr, false);
    if (rc) return rc;
    const size_t nb = h->code->K / 8, stride = d.cur->hard_stride;
    CU(cudaMemsetAsync(s.hard.p, 0, (size_t)n * stride, s.stream));
    CU(cudaMemcpy2DAsync(s.hard.p, stride, frames, nb, nb, n, cudaMemcpyHostToDevice, s.stream));
    BchArgs ba = bch_args(*d.cur, s, n);
    ba.corr_out = s.corr.p;
    ba.descramble = 0;
    int e = bch_launch(ba, s.stream);
    if (e) return fail(DVBS2FEC_ECUDA, "bch launch: %s", cudaGetErrorString((cudaError_t)e));
    CU(cudaMemcpy2DAsync(frames, nb, s.hard.p, stride, nb, n, cudaMemcpyDeviceToHost, s.stream));
    if (corrections) CU(cudaMemcpyAsync(corrections, s.corr.p, (size_t)n * 2, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    return 0;
}

int dvbs2fec_descramble(dvbs2fec_handle* h, uint8_t* frames, int stride, int n) {
    if (!h || !h->configured || !frames || n < 0 || stride < h->code->kbch / 8) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (n == 0) return 0;
    DevCtx& d = *h->devs[0];
    Slot& s = d.slot[0];
    CU(cudaSetDevice(d.device));
    CU(s.bb.reserve((size_t)n * stride));
    CU(cudaMemcpyAsync(s.bb.p, frames, (size_t)n * stride, cudaMemcpyHostToDevice, s.stream));
    int e = descramble_launch(s.bb.p, stride, n, h->code->kbch, d.prbs.p, s.stream);
    if (e) return fail(DVBS2FEC_ECUDA, "descramble launch: %s", cudaGetErrorString((cudaError_t)e));
    CU(cudaMemcpyAsync(frames, s.bb.p, (size_t)n * stride, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    return 0;
}

int dvbs2fec_decode_batch(dvbs2fec_handle* h, const int8_t* llr, int n, uint8_t* bb_out, dvbs2fec_result* results) {
    return decode_host(h, Input::llr, llr, n, bb_out, results);
}
int dvbs2fec_decode_plframes(dvbs2fec_handle* h, const float* plframes, int n, uint8_t* bb_out,
                             dvbs2fec_result* results) {
    return decode_host(h, Input::sym, plframes, n, bb_out, results);
}

int dvbs2fec_quantize_plframes(const dvbs2fec_handle* h, const float* plframes, int n, uint8_t* idx_out) {
    if (!h || !h->configured || !plframes || !idx_out || n < 0) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (h->mc.constellation == APSK32) return fail(DVBS2FEC_EINVAL, "32APSK has no LUT in the reference: send symbols");
    const int nsym = h->code->N / h->mc.bits;
    std::vector<uint8_t> rn;
    if (h->pl_codenum >= 0) rn = pl_scrambling_rn(h->pl_codenum, nsym + 36 * 22 + 8);
    auto coord = [](float s) {   // constellation.cpp:295-302 / 304-310: int(double) truncation (cvttsd2si), then the clamp
        const double v = ((double)s / 1.5) * 256 + 128;
        int x = (v > -2147483649.0 && v < 2147483648.0) ? (int)v : INT_MIN;
        return (uint8_t)(x < 0 ? 0 : x >= 256 ? 255 : x);
    };
    for (int f = 0; f < n; ++f) {
        const float* in = plframes + (size_t)f * h->plsyms * 2;
        uint8_t* out = idx_out + (size_t)f * nsym * 2;
        for (int s = 0; s < nsym; ++s) {
            const int raw = 90 + s + (h->mc.pilots ? 36 * (s / 1440) : 0);
            float re = in[2 * raw], im = in[2 * raw + 1];
            if (!rn.empty()) {   // S2Scrambling::descramble: quarter turns only swap and negate
                const float a = re, b = im;
                switch (rn[raw - 90]) {
                case 1: re = b; im = -a; break;
                case 2: re = -a; im = -b; break;
                case 3: re = -b; im = a; break;
                default: break;
                }
            }
            out[2 * s] = coord(re);
            out[2 * s + 1] = coord(im);
        }
    }
    return 0;
}

int dvbs2fec_decode_plframes_idx(dvbs2fec_handle* h, const uint8_t* idx, int n, uint8_t* bb_out, dvbs2fec_result* results) {
    return decode_host(h, Input::idx, idx, n, bb_out, results);
}

int dvbs2fec_decode_batch_device(dvbs2fec_handle* h, const int8_t* d_llr, int n, uint8_t* d_bb_out,
                                 dvbs2fec_result* d_results, void* cuda_stream) {
    return decode_device(h, Input::llr, d_llr, n, d_bb_out, d_results, cuda_stream);
}

// PLFRAME symbols already on the device (e.g. what dvbs2fec_pll_process_device left there): demapper, LDPC, BCH and
// descrambler enqueued on the caller's stream, nothing crosses PCIe.  Shares the device entry point's scratch.
int dvbs2fec_decode_plframes_device(dvbs2fec_handle* h, const float* d_plframes, int n, uint8_t* d_bb_out,
                                    dvbs2fec_result* d_results, void* cuda_stream) {
    return decode_device(h, Input::sym, d_plframes, n, d_bb_out, d_results, cuda_stream);
}

int dvbs2fec_vcm_layout(int n, const int32_t* desc, int64_t* sym_off, int64_t* llr_off, int64_t* bb_off) {
    VcmPlan P;
    if (int rc = vcm_parse(n, desc, P)) return rc;
    if (sym_off) std::copy(P.sym_off.begin(), P.sym_off.end(), sym_off);
    if (llr_off) std::copy(P.llr_off.begin(), P.llr_off.end(), llr_off);
    if (bb_off) std::copy(P.bb_off.begin(), P.bb_off.end(), bb_off);
    return 0;
}
int dvbs2fec_decode_vcm(dvbs2fec_handle* h, int n, const int32_t* desc, const int8_t* llr, uint8_t* bb_out,
                        dvbs2fec_result* results) {
    return vcm_host(h, n, desc, llr, false, bb_out, results);
}
int dvbs2fec_decode_plframes_vcm(dvbs2fec_handle* h, int n, const int32_t* desc, const float* plframes, uint8_t* bb_out,
                                 dvbs2fec_result* results) {
    return vcm_host(h, n, desc, plframes, true, bb_out, results);
}
int dvbs2fec_decode_vcm_device(dvbs2fec_handle* h, int n, const int32_t* desc, const int8_t* d_llr, uint8_t* d_bb_out,
                               dvbs2fec_result* d_results, void* cuda_stream) {
    return vcm_device(h, n, desc, d_llr, false, d_bb_out, d_results, cuda_stream);
}
int dvbs2fec_decode_plframes_vcm_device(dvbs2fec_handle* h, int n, const int32_t* desc, const float* d_plframes,
                                        uint8_t* d_bb_out, dvbs2fec_result* d_results, void* cuda_stream) {
    return vcm_device(h, n, desc, d_plframes, true, d_bb_out, d_results, cuda_stream);
}

// Copy into a staging batch with non-temporal stores: the CPU never reads these bytes again (the copy engine does), so
// they need not displace the producer's working set from its caches, and the lines are written without being read
// first.  Measured with tools/mixed_stream on the 4-GPU box: see profiles/r02_mixed_stream_*.json.
static void stream_copy(void* dst_v, const void* src_v, size_t n) {
    uint8_t* dst = static_cast<uint8_t*>(dst_v);
    const uint8_t* src = static_cast<const uint8_t*>(src_v);
    const size_t head = std::min(n, (size_t)((16 - ((uintptr_t)dst & 15)) & 15));
    memcpy(dst, src, head);
    dst += head; src += head; n -= head;
    const size_t body = n & ~(size_t)63;
    for (size_t i = 0; i < body; i += 64) {
        const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + i));
        const __m128i b = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + i + 16));
        const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + i + 32));
        const __m128i d = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + i + 48));
        _mm_stream_si128(reinterpret_cast<__m128i*>(dst + i), a);
        _mm_stream_si128(reinterpret_cast<__m128i*>(dst + i + 16), b);
        _mm_stream_si128(reinterpret_cast<__m128i*>(dst + i + 32), c);
        _mm_stream_si128(reinterpret_cast<__m128i*>(dst + i + 48), d);
    }
    memcpy(dst + body, src + body, n - body);
    _mm_sfence();
}

// The slot of the next frame in the staging batch being filled (opening a batch if need be).  Called with h->mu held
// through `lk`, which is dropped while page-locked memory is allocated.
static int acquire_slot(dvbs2fec_handle* h, std::unique_lock<std::mutex>& lk, Input kind, uint8_t** slot) {
    if (!h->worker.joinable()) h->worker = std::thread(worker_main, h);
    if (h->st_fill >= 0 && h->stages[h->st_fill].n > 0 && h->stages[h->st_fill].kind != kind) {
        h->st_ready.push_back(h->st_fill);   // a batch holds one kind of input: close the pending one
        h->st_fill = -1;
        h->cv_work.notify_all();
    }
    if (h->st_fill < 0) {
        if (h->st_free.empty()) return fail(DVBS2FEC_EAGAIN, "queue full");
        const int idx = h->st_free.front();
        h->st_free.pop_front();
        dvbs2fec_handle::Stage& S = h->stages[idx];
        S.cap = h->cfg.max_batch * (int)h->devs.size();
        S.kb = h->code->kbch / 8;
        S.in_bytes = input_frame_bytes(h, kind);
        S.kind = kind;
        S.n = S.taken = 0;
        S.ts_taken = 0;
        S.res_taken = 0;
        S.has_ts = h->ts_output;
        S.tags.clear();
        // page-locked allocation may synchronise with the device, and stream callbacks take h->mu: allocate unlocked
        // (submit_mu keeps other producers out, and a stage that is on no list is invisible to worker and collect)
        lk.unlock();
        cudaError_t e = cudaSetDevice(h->devs[0]->device);
        if (e == cudaSuccess) e = S.in.reserve((size_t)S.cap * S.in_bytes);
        if (e == cudaSuccess) e = S.bb.reserve((size_t)S.cap * S.kb);
        if (e == cudaSuccess) e = S.res.reserve(S.cap);
        if (e == cudaSuccess && S.has_ts) e = S.ts.reserve((size_t)S.cap * S.kb + 376);
        if (e == cudaSuccess && S.has_ts) e = S.ts_len.reserve(1);
        lk.lock();
        if (e != cudaSuccess) {
            h->st_free.push_back(idx);
            return fail(DVBS2FEC_ECUDA, "page-locked staging: %s", cudaGetErrorString(e));
        }
        h->st_fill = idx;
    }
    dvbs2fec_handle::Stage& S = h->stages[h->st_fill];
    *slot = S.in.p + (size_t)S.n * S.in_bytes;
    return 0;
}
// the frame in the acquired slot is complete (h->mu held)
static void commit_slot(dvbs2fec_handle* h, uint64_t tag) {
    dvbs2fec_handle::Stage& S = h->stages[h->st_fill];
    S.tags.push_back(tag);
    if (++S.n == 1) {
        S.first = std::chrono::steady_clock::now();
        h->cv_work.notify_all();   // arms the latency deadline
    }
    if (S.n == S.cap) {
        h->st_ready.push_back(h->st_fill);
        h->st_fill = -1;
        h->cv_work.notify_all();
    }
}

static int submit_common(dvbs2fec_handle* h, Input kind, const void* frame, uint64_t tag) {
    if (!h || !h->configured) return fail(DVBS2FEC_EINVAL, "set_modcod has not been called");
    std::lock_guard<std::mutex> producer(h->submit_mu);
    std::unique_lock<std::mutex> lk(h->mu);
    if (h->acquired) return fail(DVBS2FEC_EINVAL, "a frame acquired with dvbs2fec_acquire_* has not been committed");
    uint8_t* slot = nullptr;
    int rc = acquire_slot(h, lk, kind, &slot);
    if (rc) return rc;
    stream_copy(slot, frame, h->stages[h->st_fill].in_bytes);
    commit_slot(h, tag);
    return 0;
}

static int acquire_common(dvbs2fec_handle* h, Input kind, void** slot) {
    if (!h || !h->configured || !slot) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (kind == Input::idx && h->mc.constellation == APSK32) return fail(DVBS2FEC_EINVAL, "32APSK has no LUT in the reference: send symbols");
    std::lock_guard<std::mutex> producer(h->submit_mu);
    std::unique_lock<std::mutex> lk(h->mu);
    if (h->acquired) return fail(DVBS2FEC_EINVAL, "the previous frame has not been committed");
    uint8_t* p = nullptr;
    int rc = acquire_slot(h, lk, kind, &p);
    if (rc) return rc;
    h->acquired = true;   // the worker leaves the batch alone until the commit (see worker_main)
    *slot = p;
    return 0;
}

int dvbs2fec_submit_llr(dvbs2fec_handle* h, const int8_t* llr, uint64_t tag) {
    if (!llr) return fail(DVBS2FEC_EINVAL, "llr is NULL");
    return submit_common(h, Input::llr, llr, tag);
}
int dvbs2fec_submit_plframe(dvbs2fec_handle* h, const float* plframe, int nsym, uint64_t tag) {
    if (!plframe || !h || !h->configured || nsym != h->plsyms)
        return fail(DVBS2FEC_EINVAL, "plframe must hold dvbs2fec_plframe_symbols() complex samples");
    return submit_common(h, Input::sym, plframe, tag);
}

int dvbs2fec_submit_plframe_idx(dvbs2fec_handle* h, const uint8_t* idx, uint64_t tag) {
    if (!idx || !h || !h->configured) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (h->mc.constellation == APSK32) return fail(DVBS2FEC_EINVAL, "32APSK has no LUT in the reference: send symbols");
    return submit_common(h, Input::idx, idx, tag);
}

int dvbs2fec_acquire_llr(dvbs2fec_handle* h, int8_t** slot) { return acquire_common(h, Input::llr, reinterpret_cast<void**>(slot)); }
int dvbs2fec_acquire_plframe(dvbs2fec_handle* h, float** slot) { return acquire_common(h, Input::sym, reinterpret_cast<void**>(slot)); }
int dvbs2fec_acquire_plframe_idx(dvbs2fec_handle* h, uint8_t** slot) { return acquire_common(h, Input::idx, reinterpret_cast<void**>(slot)); }
int dvbs2fec_commit(dvbs2fec_handle* h, uint64_t tag) {
    if (!h || !h->configured) return fail(DVBS2FEC_EINVAL, "bad arguments");
    std::lock_guard<std::mutex> producer(h->submit_mu);
    std::unique_lock<std::mutex> lk(h->mu);
    if (!h->acquired || h->st_fill < 0) return fail(DVBS2FEC_EINVAL, "no frame has been acquired");
    h->acquired = false;
    commit_slot(h, tag);
    h->cv_work.notify_all();   // the batch may be due (latency deadline, flush) and was held back for this frame
    return 0;
}

// collect: wait up to timeout_us (< 0: for ever) for a finished stage (h->mu held through lk)
static void wait_for_done(dvbs2fec_handle* h, std::unique_lock<std::mutex>& lk, int timeout_us) {
    if (!h->st_done.empty() || timeout_us == 0) return;
    auto ready = [h] { return !h->st_done.empty(); };
    if (timeout_us < 0)
        h->cv_done.wait(lk, ready);
    else
        h->cv_done.wait_for(lk, std::chrono::microseconds(timeout_us), ready);
}
// the record of frame i of a finished stage; a stage that failed to launch has decoded nothing
static dvbs2fec_result stage_record(const dvbs2fec_handle::Stage& S, int i) {
    dvbs2fec_result r = S.res.p[i];
    r.tag = S.tags[i];
    if (S.rc) {
        r.ldpc_iters = -1;
        r.bch_corr = -1;
        r.flags = DVBS2FEC_FLAG_LDPC_FAIL | DVBS2FEC_FLAG_BCH_FAIL;
    }
    return r;
}

int dvbs2fec_collect(dvbs2fec_handle* h, uint8_t* bb_out, dvbs2fec_result* results, int max, int timeout_us) {
    if (!h || !h->configured || max < 0) return fail(DVBS2FEC_EINVAL, "bad arguments");
    std::unique_lock<std::mutex> lk(h->mu);
    wait_for_done(h, lk, timeout_us);
    int n = 0;
    const size_t kb = h->code->kbch / 8;
    while (n < max && !h->st_done.empty()) {
        dvbs2fec_handle::Stage& S = h->stages[h->st_done.front()];
        const int k = std::min(max - n, S.n - S.taken);
        if (bb_out) {
            if (S.kb == kb)
                memcpy(bb_out + (size_t)n * kb, S.bb.p + (size_t)S.taken * kb, (size_t)k * kb);
            else   // frames of the MODCOD before a set_modcod call: as many bytes as fit the current frame size
                for (int i = 0; i < k; ++i) memcpy(bb_out + (size_t)(n + i) * kb, S.bb.p + (size_t)(S.taken + i) * S.kb, std::min(kb, S.kb));
        }
        if (results)
            for (int i = 0; i < k; ++i) results[n + i] = stage_record(S, S.taken + i);
        S.taken += k;
        n += k;
        if (S.taken == S.n) {
            h->st_free.push_back(h->st_done.front());
            h->st_done.pop_front();
        }
    }
    return n;
}

int dvbs2fec_set_ts_output(dvbs2fec_handle* h, int on) {
    if (!h) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    if (on && h->devs.size() != 1)
        return fail(DVBS2FEC_EINVAL, "TS output needs a single-device handle (the parser state runs through the frames in order)");
    drain_queue(h);
    {
        std::lock_guard<std::mutex> lk(h->mu);
        if (!h->st_done.empty()) return fail(DVBS2FEC_EAGAIN, "collect the finished frames before switching the output kind");
    }
    if (on && !h->ts) {
        int rc = dvbs2fec_ts_create(h->devs[0]->device, &h->ts);
        if (rc) return rc;
        CU(cudaEventCreateWithFlags(&h->ts_done, cudaEventDisableTiming));
    }
    h->ts_output = on != 0;
    if (on && h->configured) return dvbs2fec_ts_set_frame_size(h->ts, h->code->kbch);
    return 0;
}

int dvbs2fec_collect_ts(dvbs2fec_handle* h, uint8_t* ts_out, int cap, dvbs2fec_result* results, int max_results,
                        int* nresults, int timeout_us) {
    if (nresults) *nresults = 0;
    if (!h || !h->configured || !ts_out || cap < 0 || max_results < 0) return fail(DVBS2FEC_EINVAL, "bad arguments");
    std::unique_lock<std::mutex> lk(h->mu);
    wait_for_done(h, lk, timeout_us);
    int bytes = 0, nres = 0;
    while (!h->st_done.empty()) {
        dvbs2fec_handle::Stage& S = h->stages[h->st_done.front()];
        if (!S.has_ts) return fail(DVBS2FEC_EINVAL, "frames decoded before dvbs2fec_set_ts_output: use dvbs2fec_collect");
        const int total = S.rc ? 0 : *S.ts_len.p;
        const int take = std::min(total - S.ts_taken, (cap - bytes) / 188 * 188);
        memcpy(ts_out + bytes, S.ts.p + S.ts_taken, (size_t)take);
        S.ts_taken += take;
        bytes += take;
        if (S.ts_taken < total) break;   // no room for the rest: next call
        if (results) {                   // the batch's records follow its last packets, as many as fit
            const int k = std::min(max_results - nres, S.n - S.res_taken);
            for (int i = S.res_taken; i < S.res_taken + k; ++i) results[nres++] = stage_record(S, i);
            S.res_taken += k;
            if (S.res_taken < S.n) break;   // the rest of the records: next call
        }
        h->st_free.push_back(h->st_done.front());
        h->st_done.pop_front();
    }
    if (nresults) *nresults = nres;
    return bytes;
}

int dvbs2fec_flush(dvbs2fec_handle* h) {
    if (!h) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    drain_queue(h);
    return 0;
}

void* dvbs2fec_alloc_pinned(size_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) return nullptr;
    return p;
}
void dvbs2fec_free_pinned(void* p) {
    if (p) cudaFreeHost(p);
}

// ---------------------------------------------------------------- BBFRAME -> TS (row 8(f)-1)
int dvbs2fec_ts_create(int device, dvbs2fec_ts_parser** out) {
    if (!out) return fail(DVBS2FEC_EINVAL, "out is NULL");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(DVBS2FEC_ENODEV, "no CUDA device: %s", cudaGetErrorString(cudaGetLastError()));
    if (device < 0 || device >= ndev) return fail(DVBS2FEC_EINVAL, "device %d out of range (%d present)", device, ndev);
    std::unique_ptr<dvbs2fec_ts_parser> p(new dvbs2fec_ts_parser());
    p->device = device;
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
    CU(p->state.reserve(1));
    CU(p->h_produced.reserve(4));
    CU(cudaMemset(p->state.p, 0, sizeof(TsState)));
    CU(p->gstate.reserve(1));
    CU(cudaMemset(p->gstate.p, 0, sizeof(GseState)));
    CU(p->gbuf.reserve((size_t)2 * 3 * kGseBuf));
    *out = p.release();
    return 0;
}

void dvbs2fec_ts_destroy(dvbs2fec_ts_parser* p) { delete p; }

int dvbs2fec_ts_set_frame_size(dvbs2fec_ts_parser* p, int kbch_bits) {
    if (!p || kbch_bits < 88 || kbch_bits > 65535 || kbch_bits % 8) return fail(DVBS2FEC_EINVAL, "bad frame size");
    CU(cudaSetDevice(p->device));
    p->kb = kbch_bits / 8;
    p->max_dfl = kbch_bits - 80;
    CU(cudaMemsetAsync(p->state.p, 0, sizeof(TsState), p->stream));
    CU(cudaStreamSynchronize(p->stream));
    return 0;
}

}  // extern "C"

// scratch that every call needs, and the argument block of the kernels
static int ts_args(dvbs2fec_ts_parser* p, const uint8_t* d_bb, int cnt, uint8_t* d_out, int out_cap, int* d_produced, TsArgs* out) {
    CU(p->plan.reserve(std::max(cnt, 1)));
    CU(p->meta.reserve(std::max(cnt, 1)));
    TsArgs a{};
    a.bb = d_bb;
    a.cnt = cnt;
    a.kb = p->kb;
    a.max_dfl = p->max_dfl;
    a.out = d_out;
    a.out_cap = out_cap;
    a.state = p->state.p;
    a.plan = p->plan.p;
    a.meta = p->meta.p;
    a.produced_out = d_produced;
    if (p->gse_pool >= 0) {
        CU(p->g_sync.reserve(std::max(cnt, 1)));
        CU(p->g_doff.reserve(cnt + 1));
        CU(p->g_before.reserve(cnt + 1));
        a.gse.state = p->gstate.p;
        a.gse.buf = p->gbuf.p;
        a.gse.entry_sync = p->g_sync.p;
        a.gse.doff = p->g_doff.p;
        a.gse.before = p->g_before.p;
    }
    *out = a;
    return 0;
}
static int gse_pool(dvbs2fec_ts_parser* p, int cap, TsArgs* a) {
    cap = std::max(cap, 1);
    CU(p->g_desc.reserve(cap)); CU(p->g_out.reserve(cap)); CU(p->g_crc0.reserve(cap)); CU(p->g_xpow.reserve(cap));
    CU(p->g_nxt.reserve(cap)); CU(p->g_aux.reserve(cap)); CU(p->g_aux2.reserve(cap));
    a->gse.desc = p->g_desc.p; a->gse.out = p->g_out.p; a->gse.crc0 = p->g_crc0.p; a->gse.xpow = p->g_xpow.p;
    a->gse.nxt = p->g_nxt.p; a->gse.aux = p->g_aux.p; a->gse.aux2 = p->g_aux2.p;
    a->gse.cap = cap;
    return 0;
}

extern "C" {

int dvbs2fec_ts_work_device(dvbs2fec_ts_parser* p, const uint8_t* d_bbframes, int cnt, uint8_t* d_tsframes,
                            int buffer_outsize, int* d_produced, void* stream) {
    if (!p || !p->kb) return fail(DVBS2FEC_EINVAL, "set_frame_size has not been called");
    if (cnt < 0 || (cnt && !d_bbframes) || !d_tsframes || buffer_outsize < 0) return fail(DVBS2FEC_EINVAL, "bad arguments");
    CU(cudaSetDevice(p->device));
    TsArgs a;
    int rc = ts_args(p, d_bbframes, cnt, d_tsframes, buffer_outsize, d_produced, &a);
    if (rc) return rc;
    int e = ts_launch(a, (cudaStream_t)stream);
    if (e) return fail(DVBS2FEC_ECUDA, "ts launch: %s", cudaGetErrorString((cudaError_t)e));
    if (a.gse.state) {
        // The host cannot know here whether the call holds GSE frames: the GSE pass is enqueued behind the TS pass and
        // every kernel of it returns at once unless the plan kernel deferred the call (a few microseconds of launches).
        // The descriptor pool is sized in advance; a call with more GSE packets than that is refused (kTsNoSpace).
        if ((rc = gse_pool(p, p->gse_pool > 0 ? p->gse_pool : 64 * cnt + 1024, &a))) return rc;
        e = gse_launch_count(a, (cudaStream_t)stream);
        if (!e) e = gse_launch_rest(a, (cudaStream_t)stream);
        if (e) return fail(DVBS2FEC_ECUDA, "gse launch: %s", cudaGetErrorString((cudaError_t)e));
    }
    return 0;
}

int dvbs2fec_ts_work(dvbs2fec_ts_parser* p, const uint8_t* bbframes, int cnt, uint8_t* tsframes, int buffer_outsize) {
    if (!p || !p->kb) return fail(DVBS2FEC_EINVAL, "set_frame_size has not been called");
    if (cnt < 0 || (cnt && !bbframes) || !tsframes || buffer_outsize < 0) return fail(DVBS2FEC_EINVAL, "bad arguments");
    CU(cudaSetDevice(p->device));
    const size_t in_bytes = (size_t)cnt * p->kb;
    // A call emits at most in_bytes - 10 cnt + 187 bytes of TS (every frame spends 10 bytes on its BBHEADER; one unit
    // may have been carried in).  With in_bytes + 376 bytes of room no test of the room rule (:176,208-211) can fail,
    // so a larger caller buffer is equivalent to that much -- and the kernels are told the size that is really
    // allocated.  GSE: PDUs begun in earlier calls may complete in this one, at most one per reassembly slot.
    const size_t gse_extra = p->gse_pool >= 0 ? 3 * (size_t)(kGseBuf + 4) : 0;
    const size_t out_alloc = std::min((size_t)buffer_outsize, in_bytes + 376 + gse_extra);
    CU(p->bb.reserve(std::max<size_t>(in_bytes, 1)));
    CU(p->out.reserve(std::max<size_t>(out_alloc, 1)));
    if (in_bytes) CU(cudaMemcpyAsync(p->bb.p, bbframes, in_bytes, cudaMemcpyHostToDevice, p->stream));
    TsArgs a;
    int rc = ts_args(p, p->bb.p, cnt, p->out.p, (int)out_alloc, nullptr, &a);
    if (rc) return rc;
    int e = ts_launch(a, p->stream);
    if (e) return fail(DVBS2FEC_ECUDA, "ts launch: %s", cudaGetErrorString((cudaError_t)e));
    // produced and phase lie next to each other in TsState
    CU(cudaMemcpyAsync(p->h_produced.p, &p->state.p->produced, 2 * sizeof(int), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaStreamSynchronize(p->stream));
    if (p->h_produced.p[1] == 1) {
        // the call holds GSE frames and was deferred: count the packets, size the pool, run the GSE pass
        TsArgs c = a;
        c.gse.cap = 0x7FFFFFFF;
        e = gse_launch_count(c, p->stream);
        if (e) return fail(DVBS2FEC_ECUDA, "gse launch: %s", cudaGetErrorString((cudaError_t)e));
        CU(cudaMemcpyAsync(p->h_produced.p + 2, &p->gstate.p->ndesc_wanted, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
        CU(cudaStreamSynchronize(p->stream));
        if ((rc = gse_pool(p, p->h_produced.p[2], &a))) return rc;
        e = gse_launch_rest(a, p->stream);
        if (e) return fail(DVBS2FEC_ECUDA, "gse launch: %s", cudaGetErrorString((cudaError_t)e));
        CU(cudaMemcpyAsync(p->h_produced.p, &p->state.p->produced, 2 * sizeof(int), cudaMemcpyDeviceToHost, p->stream));
        CU(cudaStreamSynchronize(p->stream));
    }
    const int produced = *p->h_produced.p;
    if (produced == kTsNoSpace)
        return fail(DVBS2FEC_ENOSPC, "GSE output does not fit into %d bytes (the reference writes PDUs without a room test)", buffer_outsize);
    if (produced > 0) {
        CU(cudaMemcpyAsync(tsframes, p->out.p, (size_t)produced, cudaMemcpyDeviceToHost, p->stream));
        CU(cudaStreamSynchronize(p->stream));
    }
    return produced;
}

int dvbs2fec_ts_set_gse(dvbs2fec_ts_parser* p, int max_packets_per_call) {
    if (!p) return fail(DVBS2FEC_EINVAL, "parser is NULL");
    p->gse_pool = max_packets_per_call;
    return 0;
}

int dvbs2fec_ts_gse_stats(dvbs2fec_ts_parser* p, int* last_gse_crc_err, int* pdus, int* crc_errors, int* malformed,
                          int* dropped) {
    if (!p) return fail(DVBS2FEC_EINVAL, "parser is NULL");
    CU(cudaSetDevice(p->device));
    GseState g;
    CU(cudaMemcpy(&g, p->gstate.p, sizeof g, cudaMemcpyDeviceToHost));
    if (last_gse_crc_err) *last_gse_crc_err = g.last_crc_err;
    if (pdus) *pdus = g.pdus;
    if (crc_errors) *crc_errors = g.crc_errors;
    if (malformed) *malformed = g.malformed;
    if (dropped) *dropped = g.dropped;
    return 0;
}

int dvbs2fec_ts_stats(dvbs2fec_ts_parser* p, dvbs2fec_bbheader* last_header, int* last_bb_cnt, int* last_bb_proc,
                      int* gse_frames) {
    if (!p) return fail(DVBS2FEC_EINVAL, "parser is NULL");
    CU(cudaSetDevice(p->device));
    TsState s;
    CU(cudaMemcpy(&s, p->state.p, sizeof s, cudaMemcpyDeviceToHost));
    if (last_header) {
        const uint8_t* b = s.last_header;   // BBHeader(uint8_t*) (bbframe_ts_parser.h:52-64)
        dvbs2fec_bbheader h{};
        h.ts_gs = b[0] >> 6;
        h.sis_mis = (b[0] >> 5) & 1;
        h.ccm_acm = (b[0] >> 4) & 1;
        h.issyi = (b[0] >> 3) & 1;
        h.npd = (b[0] >> 2) & 1;
        h.ro = b[0] & 3;
        h.isi = h.sis_mis == 0 ? b[1] : 0;
        h.upl = (uint16_t)((b[2] << 8) | b[3]);
        h.dfl = (uint16_t)((b[4] << 8) | b[5]);
        h.sync = b[6];
        h.syncd = (uint16_t)((b[7] << 8) | b[8]);
        *last_header = h;
    }
    if (last_bb_cnt) *last_bb_cnt = s.last_bb_cnt;
    if (last_bb_proc) *last_bb_proc = s.last_bb_proc;
    if (gse_frames) *gse_frames = s.gse_frames;
    return s.have_header;
}


int dvbs2fec_encode_fecframe(int modcod, int shortframes, const uint8_t* bbframe, uint8_t* code_bits) {
    ModcodCfg mc;
    if (!bbframe || !code_bits || !modcod_config(modcod, shortframes != 0, false, &mc) || mc.code < 0)
        return fail(DVBS2FEC_EINVAL, "unsupported MODCOD/frame size");
    const LdpcCode& c = ldpc_code(mc.code);
    std::vector<uint8_t> frame(c.K / 8, 0);
    const auto& prbs = bb_prbs();
    for (int i = 0; i < c.kbch / 8; ++i) frame[i] = bbframe[i] ^ prbs[i];
    bch_encode(bch_host(c.bch_m, c.bch_t), frame.data(), c.kbch);
    std::vector<uint8_t> bits(c.K);
    for (int i = 0; i < c.K; ++i) bits[i] = (frame[i >> 3] >> (7 - (i & 7))) & 1;
    ldpc_encode_bits(mc.code, bits.data(), code_bits);
    return 0;
}

int dvbs2fec_modulate(int modcod, int shortframes, int pilots, const uint8_t* code_bits, float* plframe) {
    ModcodCfg mc;
    if (!code_bits || !plframe || !modcod_config(modcod, shortframes != 0, pilots != 0, &mc) || mc.code < 0)
        return fail(DVBS2FEC_EINVAL, "unsupported MODCOD/frame size");
    const LdpcCode& c = ldpc_code(mc.code);
    ConstellationHost ch = make_constellation(mc.constellation, mc.g1, mc.g2);
    const int nsym = c.N / mc.bits;
    memset(plframe, 0, (size_t)plframe_symbols(mc) * 8);
    std::vector<uint8_t> tx(c.N);
    for (int n = 0; n < c.N; ++n) tx[interleaved_position(mc, n)] = code_bits[n] & 1;
    for (int s = 0; s < nsym; ++s) {
        int raw = 90 + s + (mc.pilots ? 36 * (s / 1440) : 0);
        map_symbol(ch, &tx[(size_t)s * mc.bits], &plframe[2 * raw]);
    }
    return 0;
}

int dvbs2fec_modcod_info(int modcod, int shortframes, int pilots, int* nldpc, int* kldpc, int* kbch, int* bch_t,
                         int* bits_per_symbol, int* plframe_symbols, int* links_total) {
    ModcodCfg mc;
    if (!modcod_config(modcod, shortframes != 0, pilots != 0, &mc) || mc.code < 0)
        return fail(DVBS2FEC_EINVAL, "unsupported MODCOD/frame size");
    const LdpcCode& c = ldpc_code(mc.code);
    if (nldpc) *nldpc = c.N;
    if (kldpc) *kldpc = c.K;
    if (kbch) *kbch = c.kbch;
    if (bch_t) *bch_t = c.bch_t;
    if (bits_per_symbol) *bits_per_symbol = mc.bits;
    if (plframe_symbols) *plframe_symbols = s2::plframe_symbols(mc);
    if (links_total) *links_total = c.links_total;
    return 0;
}

}  // extern "C"
