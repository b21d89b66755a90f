// C ABI of the PL front end (include/dvbs2fec.h, "upstream of the decode stage"): dvbs2fec_plsync_* -- PL frame
// synchronisation, PLHEADER demodulation / PLS decoding, coarse frequency error.  Kernels: pl_sync.cu.
#include "../../include/dvbs2fec.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <vector>

#include <cuda_runtime.h>

#include "abi_util.h"
#include "host_tables.h"
#include "pl_sync.cuh"

using namespace s2;

namespace {

// s2_sof / s2_plscodes (dvbs2/s2_defs.h:16-87) with the reference's float expressions
void build_tables(PlTables& t) {
    const uint32_t sof_value = 0x18d2e82u;
    for (int s = 0; s < 26; ++s) {
        const int bit = (sof_value >> (25 - s)) & 1, angle = bit * 2 + (s & 1);
        t.sof[s].x = 1 * cosf((float)(M_PI / 4 + 2 * M_PI * angle / 4));
        t.sof[s].y = 1 * sinf((float)(M_PI / 4 + 2 * M_PI * angle / 4));
    }
    const uint32_t G[6] = {0x55555555u, 0x33333333u, 0x0f0f0f0fu, 0x00ff00ffu, 0x0000ffffu, 0xffffffffu};
    for (int index = 0; index < 128; ++index) {
        uint32_t y = 0;
        for (int row = 0; row < 6; ++row)
            if ((index >> (6 - row)) & 1) y ^= G[row];
        unsigned long long code = 0;
        for (int bit = 31; bit >= 0; --bit) {
            const unsigned long long yi = (y >> bit) & 1;
            code = (index & 1) ? ((code << 2) | (yi << 1) | (yi ^ 1)) : ((code << 2) | (yi << 1) | yi);
        }
        code ^= 0x719d83c953422dfaull;
        t.codewords[index] = code;
        for (int i = 0; i < 64; ++i) {
            const int yi = (int)((code >> (63 - i)) & 1), nyi = yi ^ (i & 1);
            t.pls[index][i].x = (float)(1 * (1 - 2 * nyi)) / sqrtf(2);
            t.pls[index][i].y = (float)(1 * (1 - 2 * yi)) / sqrtf(2);
        }
    }
}

int raw_frame_size(int slot_num, int pilots) {   // dvbs2_pl_sync.cpp:15-30
    int rfs = (slot_num + 1) * 90;
    if (pilots) {
        int raw = (rfs - 90) / 90, cnt = 1;
        raw -= 16;
        while (raw > 16) {
            raw -= 16;
            ++cnt;
        }
        rfs += cnt * 36;
    }
    return rfs;
}
}  // namespace

struct dvbs2fec_plsync {
    int device = 0;
    cudaStream_t stream = nullptr;
    int rfs = 0;
    int cur = 0;               // work buffer holding the carried symbols
    int pend_ub = 0;           // upper bound of the symbols carried over (exact after a synchronous call)
    bool pend_exact = true;
    DevBuf<float2> work[2], out, frames_in, hdr_out;
    DevBuf<float> metric, fed_out;
    DevBuf<int> starts;
    DevBuf<PlSyncState> st;
    DevBuf<PlHdrState> hst;
    DevBuf<PlHdrResult> hres;
    DevBuf<PlTables> tab;
    DevBuf<uint8_t> rn;           // the coarse FED's PL scrambling sequence, of Gold code rn_codenum
    int rn_codenum = -2;
    PlSyncState h_st{};
    // S2PLLBlock (K8)
    DevBuf<PllState> pst;
    DevBuf<float> perr, pll_state;
    DevBuf<float2> pll_in, pll_out;
    DevBuf<uint8_t> pll_rn;       // the loop's own sequence: a FED call with another code must not change what a queued loop reads
    DevBuf<uint8_t> pll_jobs;
    PllArgs pll{};            // configuration part; buffers are filled in per call
    bool pll_ready = false;
    int pll_sequential = 0;      // 0: pipelined speculative kernel, 1: sequential walk, 2: one-warp speculative kernel
    ~dvbs2fec_plsync() {
        cudaSetDevice(device);
        if (stream) {
            cudaStreamSynchronize(stream);
            cudaStreamDestroy(stream);
        }
    }
};

extern "C" {

int dvbs2fec_plsync_create(int device, dvbs2fec_plsync** out) {
    if (!out) return fail(DVBS2FEC_EINVAL, "out is NULL");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(DVBS2FEC_ENODEV, "no CUDA device");
    if (device < 0 || device >= ndev) return fail(DVBS2FEC_EINVAL, "device out of range");
    std::unique_ptr<dvbs2fec_plsync> p(new dvbs2fec_plsync());
    p->device = device;
    if (const char* e = getenv("DVBS2FEC_PLL_MODE")) p->pll_sequential = (atoi(e) == 1 || atoi(e) == 2) ? atoi(e) : 0;      // A/B measurements
    p->h_st.current_position = -1;   // (dvbs2_pl_sync.h:38-40)
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
    CU(p->st.reserve(1));
    CU(p->hst.reserve(1));
    CU(p->tab.reserve(1));
    std::unique_ptr<PlTables> t(new PlTables());
    build_tables(*t);
    CU(upload(p->tab.p, t.get(), sizeof(PlTables)));
    CU(cudaMemset(p->hst.p, 0, sizeof(PlHdrState)));
    CU(p->pst.reserve(1));
    CU(cudaMemset(p->pst.p, 0, sizeof(PllState)));
    CU(cudaDeviceSynchronize());      // device memsets are asynchronous; the handle's streams do not wait for the default stream
    *out = p.release();
    return 0;
}

void dvbs2fec_plsync_destroy(dvbs2fec_plsync* p) { delete p; }

int dvbs2fec_plsync_set_params(dvbs2fec_plsync* p, int slot_num, int pilots) {
    if (!p || slot_num < 1 || slot_num > 4096) return fail(DVBS2FEC_EINVAL, "bad slot count");
    CU(cudaSetDevice(p->device));
    p->rfs = raw_frame_size(slot_num, pilots);
    return dvbs2fec_plsync_reset(p);
}

int dvbs2fec_plsync_reset(dvbs2fec_plsync* p) {
    if (!p || !p->rfs) return fail(DVBS2FEC_EINVAL, "set_params has not been called");
    CU(cudaSetDevice(p->device));
    // reset() (dvbs2_pl_sync.cpp:37-45) clears the gathering state; the public members keep their values
    PlSyncState s = p->h_st;
    s.state = 0; s.best_pos = 0; s.pend = 0; s.nframes = 0; s.cur = 0;
    p->h_st = s;
    p->pend_ub = 0;
    p->pend_exact = true;
    p->cur = 0;
    CU(cudaMemcpyAsync(p->st.p, &p->h_st, sizeof s, cudaMemcpyHostToDevice, p->stream));
    CU(cudaStreamSynchronize(p->stream));
    return 0;
}

int dvbs2fec_plsync_raw_frame_size(const dvbs2fec_plsync* p) { return p ? p->rfs : DVBS2FEC_EINVAL; }

// common part: `count` new symbols are already behind the carried ones in work[cur]
static int plsync_run(dvbs2fec_plsync* p, int count, const float2* d_append, float2* d_out, int* d_nframes, int max_frames, cudaStream_t st) {
    CU(p->metric.reserve((size_t)2 * p->rfs + count + 1));
    CU(p->starts.reserve((size_t)max_frames + 1));
    PlSyncArgs a{};
    a.work = p->work[p->cur].p;
    a.work_next = p->work[p->cur ^ 1].p;
    a.append = d_append;
    a.count = count;
    a.rfs = p->rfs;
    a.metric = p->metric.p;
    a.starts = p->starts.p;
    a.max_frames = max_frames;
    a.out = d_out;
    a.st = p->st.p;
    a.nframes_out = d_nframes;
    int e = plsync_launch(a, p->pend_ub, st);
    if (e) return fail(DVBS2FEC_ECUDA, "%s", cudaGetErrorString((cudaError_t)e));
    p->cur ^= 1;
    return 0;
}

int dvbs2fec_plsync_process(dvbs2fec_plsync* p, int count, const float* in, float* out) {
    if (!p || !p->rfs) return fail(DVBS2FEC_EINVAL, "set_params has not been called");
    if (count < 0 || (count && !in) || !out) return fail(DVBS2FEC_EINVAL, "bad arguments");
    CU(cudaSetDevice(p->device));
    if (!p->pend_exact) {   // device-buffer calls came before: ask the device how many symbols it carries
        CU(cudaDeviceSynchronize());
        CU(cudaMemcpy(&p->h_st, p->st.p, sizeof(PlSyncState), cudaMemcpyDeviceToHost));
        p->pend_ub = p->h_st.pend;
        p->pend_exact = true;
    }
    const size_t need = (size_t)p->pend_ub + count + 1;
    CU(p->work[p->cur].grow(need, p->pend_ub, p->stream));
    CU(p->work[p->cur ^ 1].reserve(std::max(need, (size_t)2 * p->rfs + 1)));
    const int max_frames = (int)((p->pend_ub + (size_t)count) / p->rfs) + 1;
    CU(p->out.reserve((size_t)max_frames * p->rfs));
    if (count) CU(cudaMemcpyAsync(p->work[p->cur].p + p->pend_ub, in, (size_t)count * sizeof(float2), cudaMemcpyHostToDevice, p->stream));
    int rc = plsync_run(p, count, nullptr, p->out.p, nullptr, max_frames, p->stream);
    if (rc) return rc;
    CU(cudaMemcpyAsync(&p->h_st, p->st.p, sizeof(PlSyncState), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaStreamSynchronize(p->stream));
    p->pend_ub = p->h_st.pend;
    const size_t n = (size_t)p->h_st.nframes * p->rfs;
    if (n) {
        CU(cudaMemcpyAsync(out, p->out.p, n * sizeof(float2), cudaMemcpyDeviceToHost, p->stream));
        CU(cudaStreamSynchronize(p->stream));
    }
    return (int)n;
}

int dvbs2fec_plsync_process_device(dvbs2fec_plsync* p, int count, const float* d_in, float* d_out, int max_frames, int* d_nframes,
                                   void* stream) {
    if (!p || !p->rfs) return fail(DVBS2FEC_EINVAL, "set_params has not been called");
    if (count < 0 || (count && !d_in) || !d_out || max_frames < 0) return fail(DVBS2FEC_EINVAL, "bad arguments");
    CU(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    // fewer than two frames are ever carried over: sized for that, the buffers only grow with the caller's block size
    const size_t need = (size_t)2 * p->rfs + count + 1;
    if (need > p->work[p->cur].cap || need > p->work[p->cur ^ 1].cap) {
        // buffers grow only here, with everything enqueued so far finished
        CU(cudaStreamSynchronize(st));
        CU(p->work[p->cur].grow(need, p->pend_ub, p->stream));
        CU(p->work[p->cur ^ 1].reserve(need));
    }
    // Without a look at the device the number of carried symbols is only bounded: fewer than two frames (a window
    // plus the realignment it asked for).  The kernels take the exact count from the device state, and the first
    // of them puts the new symbols behind the carried ones.
    const int lmax = p->pend_ub + count;
    const int room = std::min(max_frames, lmax / p->rfs + 1);
    int rc = plsync_run(p, count, reinterpret_cast<const float2*>(d_in), reinterpret_cast<float2*>(d_out), d_nframes, room, st);
    if (rc) return rc;
    p->pend_ub = std::min(lmax, 2 * p->rfs);
    p->pend_exact = false;
    return 0;
}

int dvbs2fec_plsync_stats(dvbs2fec_plsync* p, int* current_position, double* best_match, int* pending) {
    if (!p) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    CU(cudaSetDevice(p->device));
    CU(cudaMemcpy(&p->h_st, p->st.p, sizeof(PlSyncState), cudaMemcpyDeviceToHost));
    if (current_position) *current_position = p->h_st.current_position;
    if (best_match) *best_match = p->h_st.best_match;
    if (pending) *pending = p->h_st.pend;
    return p->h_st.nframes;
}

int dvbs2fec_plhdr_set_params(dvbs2fec_plsync* p, float loop_bw) {
    if (!p) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    CU(cudaSetDevice(p->device));
    // S2PLHDRDemod::init (dvbs2_plhdr_demod.cpp:5-12): criticallyDamped(loop_bw * 0.03f), phase = freq = 0
    PlHdrState s{};
    const float bw = loop_bw * 0.03f;
    const float damp = (float)(sqrt(2.0) / 2.0);
    const float den = (float)(1.0 + 2.0 * damp * bw + bw * bw);
    s.alpha = (4 * damp * bw) / den;
    s.beta = (4 * bw * bw) / den;
    CU(upload(p->hst.p, &s, sizeof s));
    return 0;
}

int dvbs2fec_plhdr_process_device(dvbs2fec_plsync* p, int nframes, const float* d_frames, float* d_headers, int32_t* d_results,
                                  void* stream) {
    if (!p || !p->rfs || nframes < 0 || (nframes && (!d_frames || !d_headers || !d_results))) return fail(DVBS2FEC_EINVAL, "bad arguments");
    CU(cudaSetDevice(p->device));
    static_assert(sizeof(PlHdrResult) == 4 * sizeof(int32_t), "result record is four ints");
    int e = plhdr_launch(reinterpret_cast<const float2*>(d_frames), nframes, p->rfs, reinterpret_cast<float2*>(d_headers),
                         reinterpret_cast<PlHdrResult*>(d_results), p->hst.p, p->tab.p, (cudaStream_t)stream);
    if (e) return fail(DVBS2FEC_ECUDA, "%s", cudaGetErrorString((cudaError_t)e));
    return 0;
}

int dvbs2fec_plhdr_process(dvbs2fec_plsync* p, int nframes, const float* frames, float* headers, int32_t* results, float* loop_state) {
    if (!p || !p->rfs || nframes < 0 || (nframes && (!frames || !headers || !results))) return fail(DVBS2FEC_EINVAL, "bad arguments");
    CU(cudaSetDevice(p->device));
    CU(p->frames_in.reserve((size_t)std::max(nframes, 1) * p->rfs));
    CU(p->hdr_out.reserve((size_t)std::max(nframes, 1) * kPlHeader));
    CU(p->hres.reserve(std::max(nframes, 1)));
    if (nframes) {
        CU(cudaMemcpyAsync(p->frames_in.p, frames, (size_t)nframes * p->rfs * sizeof(float2), cudaMemcpyHostToDevice, p->stream));
        int rc = dvbs2fec_plhdr_process_device(p, nframes, reinterpret_cast<const float*>(p->frames_in.p), reinterpret_cast<float*>(p->hdr_out.p),
                                               reinterpret_cast<int32_t*>(p->hres.p), p->stream);
        if (rc) return rc;
        CU(cudaMemcpyAsync(headers, p->hdr_out.p, (size_t)nframes * kPlHeader * sizeof(float2), cudaMemcpyDeviceToHost, p->stream));
        CU(cudaMemcpyAsync(results, p->hres.p, (size_t)nframes * sizeof(PlHdrResult), cudaMemcpyDeviceToHost, p->stream));
    }
    PlHdrState s;
    CU(cudaMemcpyAsync(&s, p->hst.p, sizeof s, cudaMemcpyDeviceToHost, p->stream));
    CU(cudaStreamSynchronize(p->stream));
    if (loop_state) {
        loop_state[0] = s.phase;
        loop_state[1] = s.freq;
    }
    return nframes;
}

static int fed_tables(dvbs2fec_plsync* p, int pilots, int codenum) {
    if (pilots && p->rn_codenum != codenum) {
        if (codenum < 0 || codenum > 262141) return fail(DVBS2FEC_EINVAL, "Gold code number outside 0..262141");
        std::vector<uint8_t> rn = pl_scrambling_rn(codenum, 131072);
        CU(p->rn.reserve(rn.size()));
        CU(upload(p->rn.p, rn.data(), rn.size()));
        p->rn_codenum = codenum;
    }
    return 0;
}

int dvbs2fec_coarse_fed_device(dvbs2fec_plsync* p, int nframes, const float* d_frames, int pilots, int pls_code, int codenum, float* d_err,
                               void* stream) {
    if (!p || !p->rfs || nframes < 0 || (nframes && (!d_frames || !d_err))) return fail(DVBS2FEC_EINVAL, "bad arguments");
    CU(cudaSetDevice(p->device));
    int rc = fed_tables(p, pilots, codenum);
    if (rc) return rc;
    int e = fed_launch(reinterpret_cast<const float2*>(d_frames), nframes, p->rfs, pilots, pls_code, p->rn.p, p->tab.p, d_err, (cudaStream_t)stream);
    if (e) return fail(DVBS2FEC_ECUDA, "%s", cudaGetErrorString((cudaError_t)e));
    return 0;
}

int dvbs2fec_coarse_fed(dvbs2fec_plsync* p, int nframes, const float* frames, int pilots, int pls_code, int codenum, float* err) {
    if (!p || !p->rfs || nframes < 0 || (nframes && (!frames || !err))) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (!nframes) return 0;
    CU(cudaSetDevice(p->device));
    CU(p->frames_in.reserve((size_t)nframes * p->rfs));
    CU(p->fed_out.reserve(nframes));
    CU(cudaMemcpyAsync(p->frames_in.p, frames, (size_t)nframes * p->rfs * sizeof(float2), cudaMemcpyHostToDevice, p->stream));
    int rc = dvbs2fec_coarse_fed_device(p, nframes, reinterpret_cast<const float*>(p->frames_in.p), pilots, pls_code, codenum, p->fed_out.p, p->stream);
    if (rc) return rc;
    CU(cudaMemcpyAsync(err, p->fed_out.p, (size_t)nframes * sizeof(float), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaStreamSynchronize(p->stream));
    return nframes;
}

// ---------------------------------------------------------------------------------------------- S2PLLBlock (K8)
int dvbs2fec_pll_set_params(dvbs2fec_plsync* p, float loop_bw, int modcod, int shortframes, int pilots, int codenum) {
    if (!p) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    ModcodCfg cfg;
    if (!modcod_config(modcod, shortframes != 0, pilots != 0, &cfg)) return fail(DVBS2FEC_EINVAL, "modcod outside 1..28");
    if (codenum < 0 || codenum > 262141) return fail(DVBS2FEC_EINVAL, "Gold code number outside 0..262141");
    CU(cudaSetDevice(p->device));
    {   // the loop descrambles every payload symbol, pilots or not
        const std::vector<uint8_t> rn = pl_scrambling_rn(codenum, 131072);
        CU(p->pll_rn.reserve(rn.size()));
        CU(upload(p->pll_rn.p, rn.data(), rn.size()));
    }
    // PhaseControlLoop<float>::criticallyDamped(loop_bw, alpha, beta) (dvbs2_pll.cpp:10)
    PllState s{};
    CU(cudaMemcpy(&s, p->pst.p, sizeof s, cudaMemcpyDeviceToHost));
    const float bw = loop_bw;
    const float damp = (float)(sqrt(2.0) / 2.0);
    const float den = (float)(1.0 + 2.0 * damp * bw + bw * bw);
    s.alpha = (4 * damp * bw) / den;
    s.beta = (4 * bw * bw) / den;
    CU(upload(p->pst.p, &s, sizeof s));
    PllArgs& a = p->pll;
    a = PllArgs{};
    a.pilot_cnt = 0;
    if (pilots) {   // S2PLLBlock::update (dvbs2_pll.h:47-59): counted from the slot number (SURVEY.md note N2)
        int raw_size = (cfg.slots - 90) / 90;
        a.pilot_cnt = 1;
        raw_size -= 16;
        while (raw_size > 16) {
            raw_size -= 16;
            a.pilot_cnt++;
        }
    }
    a.total = (cfg.slots + 1) * 90 + a.pilot_cnt * 36;
    a.divisor = (float)(cfg.slots + 1) * 90 + a.pilot_cnt * 36;
    a.pls_code = (modcod << 2 | (shortframes ? 2 : 0) | (pilots ? 1 : 0)) & 127;
    const ConstellationHost c = make_constellation(cfg.constellation, cfg.g1, cfg.g2);
    a.amp = c.amp;
    a.prescale = c.prescale;
    a.states = c.states;
    for (int i = 0; i < c.states; ++i) {
        a.pts[2 * i] = c.re[i];
        a.pts[2 * i + 1] = c.im[i];
    }
    if (cfg.constellation != APSK32) {   // the reference has no table for 32APSK (constellation.cpp:294,319-321)
        const std::vector<float> lut = demap_phase_lut(c);
        CU(p->perr.reserve(lut.size()));
        CU(upload(p->perr.p, lut.data(), lut.size() * sizeof(float)));
        a.perr_lut = p->perr.p;
    }
    a.rn = p->pll_rn.p;
    a.tab = p->tab.p;
    a.st = p->pst.p;
    p->pll_ready = true;
    return 0;
}

int dvbs2fec_pll_reset(dvbs2fec_plsync* p) {
    if (!p) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    CU(cudaSetDevice(p->device));
    PllState s{};
    CU(cudaMemcpy(&s, p->pst.p, sizeof s, cudaMemcpyDeviceToHost));
    s.phase = 0;
    s.freq = 0;
    CU(upload(p->pst.p, &s, sizeof s));
    return 0;
}

int dvbs2fec_pll_set_state(dvbs2fec_plsync* p, float phase, float freq) {
    if (!p) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    CU(cudaSetDevice(p->device));
    PllState s{};
    CU(cudaMemcpy(&s, p->pst.p, sizeof s, cudaMemcpyDeviceToHost));
    s.phase = phase;
    s.freq = freq;
    CU(upload(p->pst.p, &s, sizeof s));
    return 0;
}

int dvbs2fec_pll_set_sequential(dvbs2fec_plsync* p, int on) {
    if (!p) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    p->pll_sequential = (on == 1 || on == 2) ? on : 0;
    return 0;
}

int dvbs2fec_pll_frame_symbols(const dvbs2fec_plsync* p) { return (p && p->pll_ready) ? p->pll.total : DVBS2FEC_EINVAL; }

int dvbs2fec_pll_process_device(dvbs2fec_plsync* p, int nframes, int frame_stride, const float* d_frames, float* d_out, float* d_state,
                                void* stream) {
    if (!p || !p->pll_ready) return fail(DVBS2FEC_EINVAL, "dvbs2fec_pll_set_params has not been called");
    if (nframes < 0 || frame_stride < p->pll.total || (nframes && (!d_frames || !d_out))) return fail(DVBS2FEC_EINVAL, "bad arguments");
    CU(cudaSetDevice(p->device));
    PllArgs a = p->pll;
    a.frames = reinterpret_cast<const float2*>(d_frames);
    a.out = reinterpret_cast<float2*>(d_out);
    a.nframes = nframes;
    a.rfs = frame_stride;
    a.state_out = d_state;
    int e = pll_launch(a, p->pll_sequential, (cudaStream_t)stream);
    if (e) return fail(DVBS2FEC_ECUDA, "%s", cudaGetErrorString((cudaError_t)e));
    return 0;
}

int dvbs2fec_pll_process(dvbs2fec_plsync* p, int nframes, int frame_stride, const float* frames, float* out, float* state) {
    if (!p || !p->pll_ready) return fail(DVBS2FEC_EINVAL, "dvbs2fec_pll_set_params has not been called");
    if (nframes < 0 || frame_stride < p->pll.total || (nframes && (!frames || !out))) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (!nframes) return 0;
    CU(cudaSetDevice(p->device));
    const size_t n = (size_t)nframes * frame_stride;
    CU(p->pll_in.reserve(n));
    CU(p->pll_out.reserve(n));
    CU(p->pll_state.reserve((size_t)3 * nframes));
    CU(cudaMemcpyAsync(p->pll_in.p, frames, n * sizeof(float2), cudaMemcpyHostToDevice, p->stream));
    // (symbols behind the ones process() handles are not touched by the reference either: hand back the caller's own)
    CU(cudaMemcpyAsync(p->pll_out.p, out, n * sizeof(float2), cudaMemcpyHostToDevice, p->stream));
    int rc = dvbs2fec_pll_process_device(p, nframes, frame_stride, reinterpret_cast<const float*>(p->pll_in.p),
                                         reinterpret_cast<float*>(p->pll_out.p), p->pll_state.p, p->stream);
    if (rc) return rc;
    CU(cudaMemcpyAsync(out, p->pll_out.p, n * sizeof(float2), cudaMemcpyDeviceToHost, p->stream));
    if (state) CU(cudaMemcpyAsync(state, p->pll_state.p, (size_t)3 * nframes * sizeof(float), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaStreamSynchronize(p->stream));
    return nframes;
}

int dvbs2fec_pll_process_multi_device(int nstreams, dvbs2fec_plsync* const* objs, int nframes, int frame_stride,
                                      const float* const* d_frames, float* const* d_out, void* stream) {
    if (nstreams < 1 || nstreams > 4096 || !objs || !d_frames || !d_out || nframes < 0) return fail(DVBS2FEC_EINVAL, "bad arguments");
    std::vector<PllArgs> jobs((size_t)nstreams);
    for (int k = 0; k < nstreams; ++k) {
        dvbs2fec_plsync* p = objs[k];
        if (!p || !p->pll_ready || p->device != objs[0]->device || frame_stride < p->pll.total || !d_frames[k] || !d_out[k])
            return fail(DVBS2FEC_EINVAL, "stream not configured, on another device, or stride shorter than its frame");
        PllArgs a = p->pll;
        a.frames = reinterpret_cast<const float2*>(d_frames[k]);
        a.out = reinterpret_cast<float2*>(d_out[k]);
        a.nframes = nframes;
        a.rfs = frame_stride;
        a.state_out = nullptr;
        jobs[(size_t)k] = a;
    }
    if (!nframes) return 0;
    dvbs2fec_plsync* p0 = objs[0];
    CU(cudaSetDevice(p0->device));
    cudaStream_t st = (cudaStream_t)stream;
    // the job records travel through the first object's scratch (stream-ordered: the copy is enqueued before the kernel)
    CU(cudaStreamSynchronize(st));   // a previous multi call on this stream may still read the scratch
    CU(p0->pll_jobs.reserve((size_t)nstreams * sizeof(PllArgs)));
    CU(cudaMemcpyAsync(p0->pll_jobs.p, jobs.data(), jobs.size() * sizeof(PllArgs), cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));   // `jobs` is pageable host memory
    int e = pll_launch_multi(reinterpret_cast<const PllArgs*>(p0->pll_jobs.p), nstreams, st);
    if (e) return fail(DVBS2FEC_ECUDA, "%s", cudaGetErrorString((cudaError_t)e));
    return 0;
}

int dvbs2fec_pll_rounds(dvbs2fec_plsync* p) {
    if (!p) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    CU(cudaSetDevice(p->device));
    PllState s{};
    CU(cudaMemcpy(&s, p->pst.p, sizeof s, cudaMemcpyDeviceToHost));
    return (int)s.rounds;
}

}  // extern "C"
