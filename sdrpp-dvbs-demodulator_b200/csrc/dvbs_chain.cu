// The decode stage of the reference's DVB-S module as one call: DVBSDemod::process (dvbs/module_dvbs_demod.cpp:78-119)
// behind its sample-domain front end (demod.process: AGC, RRC, clock and carrier recovery -- SDR++ DSP, out of scope):
//   symbols -> soft bits (K11 sts) -> punctured Viterbi decoder (K11) -> TS deframer (K10) -> deinterleaver, RS(204,188),
//   descrambler (K9) -> 188-byte TS packets
// with every intermediate buffer on the device.  The objects are the library's own C-ABI handles; this file only strings
// their device entry points together the way the module does, its frame stride included (it walks the deframer's frames
// with a stride of 204 bytes instead of 1632, module_dvbs_demod.cpp:87; frame_stride selects that or back-to-back frames).
#include "../../include/dvbs2fec.h"

#include <algorithm>
#include <memory>

#include <cuda_runtime.h>

#include "abi_util.h"

using namespace s2;

struct dvbs2fec_dvbs_demod {
    int device = 0, frame_stride = 204;
    dvbs2fec_dvbs_viterbi* vit = nullptr;
    dvbs2fec_dvbs_deframer* def = nullptr;
    dvbs2fec_dvbs_outer* outer = nullptr;
    DevBuf<float> d_syms;
    DevBuf<int8_t> d_soft;
    DevBuf<uint8_t> d_bits;      // persists: what the decoder leaves unwritten (rate 5/6) is what was there
    DevBuf<uint8_t> d_frames, d_ts;
    DevBuf<int32_t> d_err;
    int errors[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int frames_found = 0, frames_done = 0;
    ~dvbs2fec_dvbs_demod() {
        cudaSetDevice(device);
        dvbs2fec_dvbs_viterbi_destroy(vit);
        dvbs2fec_dvbs_deframer_destroy(def);
        dvbs2fec_dvbs_outer_destroy(outer);
    }
};

extern "C" {

void dvbs2fec_dvbs_demod_destroy(dvbs2fec_dvbs_demod* p) { delete p; }

int dvbs2fec_dvbs_demod_create(int device, float ber_threshold, int max_outsync, int frame_stride, dvbs2fec_dvbs_demod** out) {
    if (!out) return fail(DVBS2FEC_EINVAL, "out is NULL");
    *out = nullptr;
    if (frame_stride != 204 && frame_stride != 1632) return fail(DVBS2FEC_EINVAL, "frame_stride is 204 (as the module) or 1632 (back-to-back frames)");
    std::unique_ptr<dvbs2fec_dvbs_demod> p(new dvbs2fec_dvbs_demod());
    p->device = device;
    p->frame_stride = frame_stride;
    int rc = dvbs2fec_dvbs_viterbi_create(device, ber_threshold, max_outsync, &p->vit);
    if (!rc) rc = dvbs2fec_dvbs_deframer_create(device, &p->def);
    if (!rc) rc = dvbs2fec_dvbs_outer_create(device, &p->outer);
    if (rc) return rc;
    *out = p.release();
    return 0;
}

int dvbs2fec_dvbs_demod_reset(dvbs2fec_dvbs_demod* p) {
    if (!p) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    int rc = dvbs2fec_dvbs_viterbi_reset(p->vit);
    if (!rc) rc = dvbs2fec_dvbs_deframer_reset(p->def);
    if (!rc) rc = dvbs2fec_dvbs_outer_reset(p->outer);
    if (rc) return rc;
    CU(cudaSetDevice(p->device));
    if (p->d_bits.p) CU(cudaMemset(p->d_bits.p, 0, p->d_bits.cap));
    CU(cudaDeviceSynchronize());
    std::fill(p->errors, p->errors + 8, 0);
    p->frames_found = p->frames_done = 0;
    return 0;
}

int dvbs2fec_dvbs_demod_process(dvbs2fec_dvbs_demod* p, int count, const float* syms, uint8_t* out, int out_cap) {
    if (!p || count < 0 || out_cap < 0 || (count && !syms) || (out_cap && !out)) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (!count) return 0;
    if (count > (1 << 23)) return fail(DVBS2FEC_EINVAL, "more than 2^23 symbols in one call");
    CU(cudaSetDevice(p->device));
    const size_t nsoft_max = (size_t)2 * count + 8192;
    CU(p->d_syms.reserve((size_t)2 * count));
    CU(p->d_soft.reserve(nsoft_max));
    const size_t had = p->d_bits.cap;      // d_bits grows without forgetting, and from zeros
    CU(p->d_bits.grow(nsoft_max, had, nullptr));
    if (p->d_bits.cap > had) CU(cudaMemset(p->d_bits.p + had, 0, p->d_bits.cap - had));
    CU(cudaMemcpy(p->d_syms.p, syms, sizeof(float) * 2 * count, cudaMemcpyHostToDevice));
    CU(cudaDeviceSynchronize());      // a pageable copy and a memset return early; the stages' own streams do not wait for the default stream
    const int nsoft = dvbs2fec_dvbs_sts_process_device(p->vit, count, p->d_syms.p, p->d_soft.p);      // :80
    if (nsoft <= 0) return nsoft;
    const int nbits = dvbs2fec_dvbs_viterbi_process_device(p->vit, nsoft, p->d_soft.p, p->d_bits.p);      // :81
    if (nbits <= 0) return nbits;
    // :82 -- a frame needs 13056 new bits unless sync patterns overlap; room for one frame per 1632 bits and a few more
    const int max_frames = nbits / 1632 + 8;
    CU(p->d_frames.reserve((size_t)max_frames * 1632));
    int rc = dvbs2fec_dvbs_deframer_work_device(p->def, p->d_bits.p, nbits, p->d_frames.p, max_frames, nullptr, nullptr);
    if (rc) return rc;
    int found = 0;
    const int nframes = dvbs2fec_dvbs_deframer_stats(p->def, nullptr, nullptr, &found);      // synchronises
    if (nframes < 0) return nframes;
    p->frames_found = found;
    p->frames_done = nframes;
    if (!nframes) return 0;
    if ((long long)nframes * 8 * 188 > out_cap) return fail(DVBS2FEC_ENOSPC, "TS output does not fit out_cap");
    CU(p->d_ts.reserve((size_t)nframes * 8 * 188));
    CU(p->d_err.reserve((size_t)nframes * 8));
    const int nb = dvbs2fec_dvbs_outer_process_device(p->outer, nframes, p->frame_stride, p->d_frames.p, p->d_ts.p, p->d_err.p, nullptr);      // :85-100
    if (nb < 0) return nb;
    CU(cudaMemcpy(out, p->d_ts.p, (size_t)nframes * 8 * 188, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(p->errors, p->d_err.p + (size_t)(nframes - 1) * 8, sizeof(int) * 8, cudaMemcpyDeviceToHost));
    return nframes * 8 * 188;
}

int dvbs2fec_dvbs_demod_stats(dvbs2fec_dvbs_demod* p, float* viterbi_ber, int* viterbi_lock, int* viterbi_rate, float* rs_avg, int* deframer_err,
                              int* frames_found, int* frames_done) {
    if (!p) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    int rc = dvbs2fec_dvbs_viterbi_stats(p->vit, viterbi_ber, viterbi_lock, viterbi_rate, nullptr, nullptr, nullptr);      // :101-113
    if (rc) return rc;
    if (rs_avg) {      // :114 (integer division, as there)
        int s = 0;
        for (int i = 0; i < 8; ++i) s += p->errors[i];
        *rs_avg = (float)(s / 8);
    }
    if (deframer_err) {      // :115
        int a = 0, b = 0;
        rc = dvbs2fec_dvbs_deframer_stats(p->def, &a, &b, nullptr);
        if (rc < 0) return rc;
        *deframer_err = std::min(a, b);
    }
    if (frames_found) *frames_found = p->frames_found;
    if (frames_done) *frames_done = p->frames_done;
    return 0;
}

}  // extern "C"
