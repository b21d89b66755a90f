// The decode stage of the reference's DVB-S2 module as one call: DVBS2Demod::process (dvbs2/module_dvbs2_demod.cpp:300-367)
// behind its sample-domain front end (AGC, RRC, clock recovery, frequency shifter -- SDR++ DSP, out of scope):
//   symbols -> PL sync (K7) -> per frame: coarse frequency error (K7), payload phase loop with PL descrambling (K8),
//   PLHEADER demodulation (K7), demapper (K1), LDPC (K2), BCH + BB descrambler (K3) -> BBFRAMEs
// Symbols go up once; frames, derotated symbols, LLRs and hard decisions never leave the device.  The objects are the
// library's own C-ABI handles; this file strings their device entry points together on one stream, in the reference's
// order.  Two things the reference's loop does are left to the caller because they belong to its sample-domain side: the
// coarse frequency error is handed back per frame (the module feeds it to its frequency shifter, :302-313, which acts on
// LATER samples anyway), and nothing waits for 16 frames before decoding (SURVEY.md note N1).
#include "../../include/dvbs2fec.h"

#include <algorithm>
#include <memory>

#include <cuda_runtime.h>

#include "abi_util.h"

using namespace s2;

struct dvbs2fec_s2_demod {
    int device = 0;
    dvbs2fec_handle* fec = nullptr;
    dvbs2fec_plsync* pl = nullptr;
    dvbs2fec_ts_parser* ts = nullptr;      // BBFRAME -> TS / GSE (K6), for dvbs2fec_s2_demod_process_ts
    cudaStream_t stream = nullptr;
    int modcod = 0, shortframes = 0, pilots = 0, codenum = 0, rfs = 0, kb = 0;
    DevBuf<float> d_x, d_fr, d_pl, d_hsym, d_fed;
    DevBuf<uint8_t> d_bb, d_ts;
    DevBuf<dvbs2fec_result> d_res;
    DevBuf<int32_t> d_hdr;
    DevBuf<int> d_n;
    int last_frames = 0;
    ~dvbs2fec_s2_demod() {
        cudaSetDevice(device);
        if (stream) {
            cudaStreamSynchronize(stream);
            cudaStreamDestroy(stream);
        }
        dvbs2fec_plsync_destroy(pl);
        dvbs2fec_ts_destroy(ts);
        dvbs2fec_destroy(fec);
    }
};

extern "C" {

void dvbs2fec_s2_demod_destroy(dvbs2fec_s2_demod* p) { delete p; }

int dvbs2fec_s2_demod_create(const dvbs2fec_config* cfg, dvbs2fec_s2_demod** out) {
    if (!out) return fail(DVBS2FEC_EINVAL, "out is NULL");
    *out = nullptr;
    std::unique_ptr<dvbs2fec_s2_demod> p(new dvbs2fec_s2_demod());
    dvbs2fec_config c{};
    if (cfg) c = *cfg;
    if (c.n_devices > 1) return fail(DVBS2FEC_EINVAL, "one stream of symbols is a recurrence (PL sync, phase loops): one device");
    int dev = 0;
    if (c.n_devices == 1) dev = c.devices[0];
    else if (cudaGetDevice(&dev) != cudaSuccess) return fail(DVBS2FEC_ENODEV, "no CUDA device");
    c.n_devices = 1;
    c.devices[0] = dev;
    if (c.max_batch <= 0) c.max_batch = 1024;
    p->device = dev;
    int rc = dvbs2fec_create(&c, &p->fec);
    if (!rc) rc = dvbs2fec_plsync_create(dev, &p->pl);
    if (!rc) rc = dvbs2fec_ts_create(dev, &p->ts);
    if (rc) return rc;
    CU(cudaSetDevice(dev));
    CU(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
    CU(p->d_n.reserve(1));
    *out = p.release();
    return 0;
}

int dvbs2fec_s2_demod_set_params(dvbs2fec_s2_demod* p, int modcod, int shortframes, int pilots, int max_trials, float pll_loop_bw,
                                 float plhdr_loop_bw, int codenum) {
    if (!p) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    int nldpc = 0, bits = 0, plsyms = 0;
    int rc = dvbs2fec_modcod_info(modcod, shortframes, pilots, &nldpc, nullptr, nullptr, nullptr, &bits, &plsyms, nullptr);
    if (rc) return rc;
    CU(cudaSetDevice(p->device));
    CU(cudaStreamSynchronize(p->stream));
    rc = dvbs2fec_set_modcod(p->fec, modcod, shortframes, pilots, max_trials);      // DVBS2Demod::setDemodParams (:118-168)
    if (!rc) rc = dvbs2fec_set_pl_scrambling(p->fec, -1);                            // the phase loop hands over descrambled symbols
    if (!rc) rc = dvbs2fec_plsync_set_params(p->pl, nldpc / bits / 90, pilots);
    if (!rc) rc = dvbs2fec_plhdr_set_params(p->pl, plhdr_loop_bw);
    if (!rc) rc = dvbs2fec_pll_set_params(p->pl, pll_loop_bw, modcod, shortframes, pilots, codenum);
    if (rc) return rc;
    p->modcod = modcod; p->shortframes = !!shortframes; p->pilots = !!pilots; p->codenum = codenum;
    p->rfs = dvbs2fec_plsync_raw_frame_size(p->pl);
    p->kb = dvbs2fec_kbch(p->fec) / 8;
    rc = dvbs2fec_ts_set_frame_size(p->ts, p->kb * 8);      // BBFrameTSParser::setFrameSize (main.cpp, on a MODCOD change)
    if (rc) return rc;
    if (p->rfs != plsyms || dvbs2fec_pll_frame_symbols(p->pl) > p->rfs) return fail(DVBS2FEC_EINVAL, "frame sizes of the stages disagree");
    return 0;
}

int dvbs2fec_s2_demod_reset(dvbs2fec_s2_demod* p) {
    if (!p || !p->rfs) return fail(DVBS2FEC_EINVAL, "set_params has not been called");
    CU(cudaSetDevice(p->device));
    CU(cudaStreamSynchronize(p->stream));
    int rc = dvbs2fec_plsync_reset(p->pl);
    if (!rc) rc = dvbs2fec_pll_reset(p->pl);
    return rc;
}

int dvbs2fec_s2_demod_bbframe_bytes(const dvbs2fec_s2_demod* p) { return p ? p->kb : 0; }
int dvbs2fec_s2_demod_max_frames(const dvbs2fec_s2_demod* p, int count) { return p && p->rfs ? count / p->rfs + 2 : 0; }

}  // extern "C"

namespace {
// symbols in host memory -> BBFRAMEs, results, frequency errors and PLHEADER fields on the device (enqueued, not waited for);
// returns the number of frames
int stage_to_device(dvbs2fec_s2_demod* p, int count, const float* syms) {
    const int room = count / p->rfs + 2;      // fewer than two frames are ever carried over
    CU(cudaSetDevice(p->device));
    cudaStream_t st = p->stream;
    const size_t fsz = (size_t)room * p->rfs * 2;
    CU(p->d_x.reserve((size_t)2 * count));
    CU(p->d_fr.reserve(fsz));
    if (fsz > p->d_pl.cap) {
        CU(p->d_pl.reserve(fsz));
        CU(cudaMemsetAsync(p->d_pl.p, 0, fsz * sizeof(float), st));      // symbols behind the ones the loop handles are never written
    }
    CU(p->d_hsym.reserve((size_t)room * 180));
    CU(p->d_bb.reserve((size_t)room * p->kb));
    CU(p->d_res.reserve((size_t)room));
    CU(p->d_fed.reserve((size_t)room));
    CU(p->d_hdr.reserve((size_t)room * 4));
    CU(cudaMemcpyAsync(p->d_x.p, syms, sizeof(float) * 2 * count, cudaMemcpyHostToDevice, st));
    int rc = dvbs2fec_plsync_process_device(p->pl, count, p->d_x.p, p->d_fr.p, room, p->d_n.p, st);      // :300
    if (rc) return rc;
    int n = 0;
    CU(cudaMemcpyAsync(&n, p->d_n.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (n <= 0) return 0;
    const int pls_code = p->modcod << 2 | p->shortframes << 1 | p->pilots;
    rc = dvbs2fec_coarse_fed_device(p->pl, n, p->d_fr.p, p->pilots, pls_code, p->codenum, p->d_fed.p, st);      // :302
    if (!rc) rc = dvbs2fec_pll_process_device(p->pl, n, p->rfs, p->d_fr.p, p->d_pl.p, nullptr, st);             // :314
    if (!rc) rc = dvbs2fec_plhdr_process_device(p->pl, n, p->d_fr.p, p->d_hsym.p, p->d_hdr.p, st);                // :315
    if (!rc) rc = dvbs2fec_decode_plframes_device(p->fec, p->d_pl.p, n, p->d_bb.p, p->d_res.p, st);               // :316, 334-366
    if (rc) return rc;
    return n;
}

int copy_side_outputs(dvbs2fec_s2_demod* p, int n, dvbs2fec_result* results, float* fed_err, int32_t* plhdr) {
    cudaStream_t st = p->stream;
    if (results) CU(cudaMemcpyAsync(results, p->d_res.p, sizeof(dvbs2fec_result) * n, cudaMemcpyDeviceToHost, st));
    if (fed_err) CU(cudaMemcpyAsync(fed_err, p->d_fed.p, sizeof(float) * n, cudaMemcpyDeviceToHost, st));
    if (plhdr) CU(cudaMemcpyAsync(plhdr, p->d_hdr.p, sizeof(int32_t) * 4 * n, cudaMemcpyDeviceToHost, st));
    return 0;
}
}  // namespace

extern "C" {

int dvbs2fec_s2_demod_process(dvbs2fec_s2_demod* p, int count, const float* syms, uint8_t* bb_out, int max_frames, dvbs2fec_result* results,
                              float* fed_err, int32_t* plhdr) {
    if (!p || !p->rfs) return fail(DVBS2FEC_EINVAL, "set_params has not been called");
    if (count < 0 || (count && !syms) || !bb_out) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (max_frames < count / p->rfs + 2) return fail(DVBS2FEC_EINVAL, "max_frames < count / raw_frame_size + 2 (dvbs2fec_s2_demod_max_frames)");
    if (!count) return 0;
    const int n = stage_to_device(p, count, syms);
    if (n <= 0) return n;
    cudaStream_t st = p->stream;
    CU(cudaMemcpyAsync(bb_out, p->d_bb.p, (size_t)n * p->kb, cudaMemcpyDeviceToHost, st));
    int rc = copy_side_outputs(p, n, results, fed_err, plhdr);
    if (rc) return rc;
    CU(cudaStreamSynchronize(st));
    return n;
}

int dvbs2fec_s2_demod_process_ts(dvbs2fec_s2_demod* p, int count, const float* syms, uint8_t* ts_out, int ts_cap, int max_frames, int* nframes,
                                 dvbs2fec_result* results, float* fed_err, int32_t* plhdr) {
    if (!p || !p->rfs) return fail(DVBS2FEC_EINVAL, "set_params has not been called");
    if (count < 0 || (count && !syms) || !ts_out || ts_cap <= 0) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if ((results || fed_err || plhdr) && max_frames < count / p->rfs + 2)
        return fail(DVBS2FEC_EINVAL, "max_frames < count / raw_frame_size + 2 (dvbs2fec_s2_demod_max_frames)");
    if (nframes) *nframes = 0;
    if (!count) return 0;
    const int n = stage_to_device(p, count, syms);
    if (n <= 0) return n;
    if (nframes) *nframes = n;
    cudaStream_t st = p->stream;
    CU(p->d_ts.reserve((size_t)ts_cap));
    int rc = dvbs2fec_ts_work_device(p->ts, p->d_bb.p, n, p->d_ts.p, ts_cap, p->d_n.p, st);      // main.cpp:538: ts_parser.work(...)
    if (rc) return rc;
    int produced = 0;
    CU(cudaMemcpyAsync(&produced, p->d_n.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    rc = copy_side_outputs(p, n, results, fed_err, plhdr);
    if (rc) return rc;
    CU(cudaStreamSynchronize(st));
    if (produced < 0) return fail(produced, "TS / GSE output does not fit ts_cap");
    if (produced) {
        CU(cudaMemcpyAsync(ts_out, p->d_ts.p, (size_t)produced, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    return produced;
}

}  // extern "C"
