// K9: the outer decoder of the DVB-S chain on the device (SURVEY.md 8(f) rank 4, the byte-domain half): the body of
// the frame loop of DVBSDemod::process (dvbs/module_dvbs_demod.cpp:91-106) for a whole batch of frames --
//   convolutional deinterleaver   dvbs/dvbs_interleaving.h:30-40,57-70   (I = 12, M = 17)
//   8 x RS(204,188) per frame     dvbs/dvbs_reedsolomon.h:18-48 over the vendored libcorrect
//                                 (common/correct/reed-solomon/decode.c:12-27,31-124,128-145,147-228,303-376)
//   energy-dispersal descrambler  dvbs/dvbs_scrambling.h:16-45
//   8 x 188 bytes out             module_dvbs_demod.cpp:102-105
// and the C ABI dvbs2fec_dvbs_outer_* around it.
//
// The reference runs this one frame after the other with three pieces of state; each of them becomes a parallel
// step here:
//   * the deinterleaver's FIFOs are fixed delays -- byte n of the (logical) input stream comes out 204 (11 - n % 12)
//     bytes later -- so every output byte is one gather, from this call's frames or from the 2244 bytes of history
//     kept on the device;
//   * the Reed-Solomon decoder works on one packet at a time (a warp per packet: syndromes across lanes, libcorrect's
//     Berlekamp-Massey restated step by step in one lane, root search and error values across lanes) -- but the
//     wrapper hands a packet it could not decode the PREVIOUS packet's output (it compares libcorrect's return value
//     with 1 instead of -1, dvbs_reedsolomon.h:33-36, and libcorrect leaves the output buffer alone on failure).  That
//     is a "last packet that decoded at or before me" relation: a max-scan over the packets;
//   * the descrambler's register is loaded by an inverted sync byte and otherwise runs on: the sequence byte a data
//     byte meets depends on the distance to the last packet that began with 0xB8 -- a second max-scan -- and is then
//     a look-up in the 32767-byte table of the generator's period.
// Results are bit-identical to the reference's (tests/test_gpu_dvbs.py against the oracle, which
// tests/test_dvbs_oracle.py pins to the compiled reference).
#include "../../include/dvbs2fec.h"

#include <cstring>
#include <memory>
#include <vector>

#include <cuda_runtime.h>

#include "abi_util.h"

using namespace s2;

namespace {

constexpr int kFrame = 1632;        // 8 x 204
constexpr int kPkt = 204;
constexpr int kHist = 2244;         // longest FIFO: 11 x 204 bytes of stream
constexpr int kPeriod = 32767;      // 2^15 - 1

struct OuterState {
    uint8_t hist[2][kHist + 4];     // the last kHist bytes of the logical input stream
    uint8_t obuf[2][192];           // DVBSReedSolomon::obuffer[51..239)
    int cur;                        // which hist / obuf is current
    int prbs_off;                   // clocks since the descrambler was loaded, at the start of the next packet; -1: never
    int prbs_next;                  // value for the next call (set by the scan kernel, committed with cur)
};

struct GfTables {
    uint8_t exp[512];
    uint8_t log[256];
};

// ---------------------------------------------------------------------------------------------- deinterleaver
// logical stream S: [history][window 0][window 1]... where window k = frames[k * stride .. + 1632)
__device__ __forceinline__ uint8_t stream_byte(const uint8_t* frames, int stride, const uint8_t* hist, long long idx) {
    if (idx < 0) return hist[kHist + idx];
    const long long w = idx / kFrame;
    return frames[w * stride + (idx - w * kFrame)];
}

__global__ void __launch_bounds__(256) deint_kernel(const uint8_t* __restrict__ frames, int nframes, int stride, OuterState* st,
                                                    uint8_t* __restrict__ D) {
    const long long total = (long long)nframes * kFrame;
    const uint8_t* hist = st->hist[st->cur];
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n < total) {
        const int m = (int)(n % kFrame);
        D[n] = stream_byte(frames, stride, hist, n - kPkt * (11 - m % 12));
    } else if (n < total + kHist) {      // the history the next call starts with
        const int i = (int)(n - total);
        st->hist[st->cur ^ 1][i] = stream_byte(frames, stride, hist, total - kHist + i);
    }
}

// ---------------------------------------------------------------------------------------------- Reed-Solomon
struct WarpScratch {
    uint8_t syn[16];
    uint8_t loc[40], last[40];
    uint8_t roots[36];
    uint8_t omega[16];
    int order, nroots;
};

__device__ __forceinline__ uint8_t gmul(const GfTables& g, uint8_t l, uint8_t r) { return (!l || !r) ? 0 : g.exp[g.log[l] + g.log[r]]; }
__device__ __forceinline__ uint8_t gdiv(const GfTables& g, uint8_t l, uint8_t r) { return (!l || !r) ? 0 : g.exp[255 + g.log[l] - g.log[r]]; }
// polynomial_eval_lut (polynomial.c:113-132): powers of v counted with logs in 1..255 (log[1] = 255)
__device__ __forceinline__ uint8_t peval(const GfTables& g, const uint8_t* c, int order, uint8_t v) {
    if (v == 0) return c[0];
    uint8_t res = 0;
    unsigned acc = 255;
    const unsigned vlog = g.log[v];
    for (int i = 0; i <= order; ++i) {
        if (c[i]) res ^= g.exp[g.log[c[i]] + acc];
        acc += vlog;
        if (acc > 255) acc -= 255;
    }
    return res;
}

// one warp per packet, eight packets (one frame) per CTA
__global__ void __launch_bounds__(256) rs_kernel(const uint8_t* __restrict__ D, int npackets, const GfTables* __restrict__ gtab,
                                                 uint8_t* __restrict__ dec, uint8_t* __restrict__ ok) {
    __shared__ GfTables g;
    __shared__ WarpScratch ws[8];
    for (int i = threadIdx.x; i < (int)sizeof(GfTables); i += blockDim.x) reinterpret_cast<uint8_t*>(&g)[i] = reinterpret_cast<const uint8_t*>(gtab)[i];
    __syncthreads();
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int p = blockIdx.x * 8 + wid;
    if (p >= npackets) return;
    const uint8_t* pk = D + (size_t)p * kPkt;
    uint8_t* out = dec + (size_t)p * 188;
    WarpScratch& w = ws[wid];
    // the message part goes out as received; corrections are XORed in afterwards
    for (int k = lane; k < 188; k += 32) out[k] = pk[k];
    // syndromes S_j = sum_i c_i alpha^(i j), c_i = packet byte 203 - i (decode.c:317-331; the 51 leading bytes are zero)
    uint32_t s[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) s[j] = 0;
    for (int i = lane; i < kPkt; i += 32) {
        const uint8_t c = pk[203 - i];
        if (c) {
            unsigned e = g.log[c];               // log c + i j, kept below 255 + 255
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                s[j] ^= g.exp[e];
                e += (unsigned)i;
                if (e >= 255) e -= 255;
                if (e >= 255) e -= 255;          // (log c up to 255, i up to 203)
            }
        }
    }
    uint32_t any = 0;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) s[j] ^= __shfl_xor_sync(0xFFFFFFFFu, s[j], off);
        any |= s[j];
    }
    if (!any) {                                   // all syndromes zero: the message as received (decode.c:333-340)
        if (lane == 0) ok[p] = 1;
        return;
    }
    if (lane < 16) {
        uint32_t mine = 0;
#pragma unroll
        for (int j = 0; j < 16; ++j) mine = (lane == j) ? s[j] : mine;
        w.syn[lane] = (uint8_t)mine;
    }
    __syncwarp();
    if (lane == 0) {   // Berlekamp-Massey exactly as libcorrect runs it (decode.c:31-124)
        uint8_t* loc = w.loc;
        uint8_t* last = w.last;
        for (int i = 0; i < 40; ++i) loc[i] = last[i] = 0;
        loc[0] = last[0] = 1;
        unsigned loc_order = 0, last_order = 0, numerrors = 0, delay = 1;
        uint8_t last_disc = 1;
        for (unsigned i = 0; i < 16; ++i) {
            uint8_t disc = w.syn[i];
            for (unsigned j = 1; j <= numerrors; ++j) disc ^= gmul(g, loc[j], w.syn[i - j]);
            if (!disc) {
                delay++;
                continue;
            }
            if (2 * numerrors <= i) {
                for (int j = (int)last_order; j >= 0; --j) last[j + delay] = gdiv(g, gmul(g, last[j], disc), last_disc);
                for (int j = (int)delay - 1; j >= 0; --j) last[j] = 0;
                for (unsigned j = 0; j <= last_order + delay; ++j) {
                    const uint8_t t = loc[j];
                    loc[j] ^= last[j];
                    last[j] = t;
                }
                const unsigned t = loc_order;
                loc_order = last_order + delay;
                last_order = t;
                numerrors = i + 1 - numerrors;
                last_disc = disc;
                delay = 1;
                continue;
            }
            for (int j = (int)last_order; j >= 0; --j) loc[j + delay] ^= gdiv(g, gmul(g, last[j], disc), last_disc);
            if (last_order + delay > loc_order) loc_order = last_order + delay;
            delay++;
        }
        w.order = (int)loc_order;
    }
    __syncwarp();
    const int order = w.order;
    // roots of the locator among all 256 field elements, ascending (decode.c:128-145)
    int nroots = 0;
    for (int t = 0; t < 8; ++t) {
        const int v = t * 32 + lane;
        const bool root = peval(g, w.loc, order, (uint8_t)v) == 0;
        const unsigned m = __ballot_sync(0xFFFFFFFFu, root);
        if (root) {
            const int at = nroots + __popc(m & ((1u << lane) - 1));
            if (at < 36) w.roots[at] = (uint8_t)v;
        }
        nroots += __popc(m);
    }
    if (nroots != order) {                        // too many errors: libcorrect returns -1 and writes nothing (:353-357)
        if (lane == 0) ok[p] = 0;
        return;
    }
    // error evaluator = locator * S(x) mod x^16 (decode.c:147-160), one coefficient per lane
    if (lane < 16) {
        uint8_t o = 0;
        for (int i = 0; i <= order && i <= lane; ++i) o ^= gmul(g, w.loc[i], w.syn[lane - i]);
        w.omega[lane] = o;
    }
    __syncwarp();
    // error values (Forney, :162-198) and locations (:200-228), one root per lane
    if (lane < order) {
        const uint8_t root = w.roots[lane];
        // derivative of the locator at the root (polynomial.c:74-87): the odd-power coefficients, shifted down
        uint8_t der = 0;
        {
            unsigned acc = 255;
            const unsigned vlog = g.log[root];
            for (int i = 0; i <= order - 1; ++i) {
                const uint8_t c = ((i + 1) & 1) ? w.loc[i + 1] : 0;
                if (c) der ^= g.exp[g.log[c] + acc];
                acc += vlog;
                if (acc > 255) acc -= 255;
            }
        }
        const uint8_t inv = g.exp[(255 - g.log[root]) % 255];              // field_pow(root, first_consecutive_root - 1)
        const uint8_t val = gmul(g, inv, gdiv(g, peval(g, w.omega, 15, root), der));
        const unsigned where = g.log[gdiv(g, 1, root)];                     // coefficient index; log[1] = 255 (field.h)
        // coefficient i is packet byte 203 - i; only the message bytes (0..187) leave this kernel
        if (where >= 16 && where <= 203) out[203 - where] ^= val;
    }
    if (lane == 0) ok[p] = 1;
}

// ---------------------------------------------------------------------------------------------- the two scans
// src[p]: last packet <= p that decoded (-1: the buffer the call inherited); eff[p]: clocks since the descrambler was
// loaded when byte 1 of packet p meets it (-1: never loaded).  One CTA; every thread owns a run of packets.
__global__ void __launch_bounds__(1024) scan_kernel(const uint8_t* __restrict__ dec, const uint8_t* __restrict__ ok, int npackets, OuterState* st,
                                                    int* __restrict__ src, int* __restrict__ eff) {
    __shared__ int sm[1024];
    const int tid = threadIdx.x;
    const int per = (npackets + 1023) / 1024;
    const int lo = min(tid * per, npackets), hi = min(lo + per, npackets);
    auto exclusive_max = [&](int mine) -> int {   // max over the threads before this one (-1 if none)
        sm[tid] = mine;
        __syncthreads();
        for (int off = 1; off < 1024; off <<= 1) {
            const int o = tid >= off ? sm[tid - off] : -1;
            __syncthreads();
            sm[tid] = max(sm[tid], o);
            __syncthreads();
        }
        const int r = tid ? sm[tid - 1] : -1;
        __syncthreads();
        return r;
    };
    int last = -1;
    for (int p = lo; p < hi; ++p)
        if (ok[p]) last = p;
    int run = exclusive_max(last);
    const uint8_t* inherited = st->obuf[st->cur];
    int lastr = -1;
    for (int p = lo; p < hi; ++p) {
        if (ok[p]) run = p;
        src[p] = run;
        const uint8_t b0 = run >= 0 ? dec[(size_t)run * 188] : inherited[0];
        if (b0 == 0xB8) lastr = p;                // DVBSScrambling::descramble loads the register here (:34-35)
    }
    int runr = exclusive_max(lastr);
    const int c0 = st->prbs_off;
    int e = -1;
    for (int p = lo; p < hi; ++p) {
        const uint8_t b0 = src[p] >= 0 ? dec[(size_t)src[p] * 188] : inherited[0];
        if (b0 == 0xB8) runr = p;
        if (runr >= 0) e = (int)(((long long)(p - runr) * 1504) % kPeriod);
        else e = c0 >= 0 ? (int)((c0 + 8 + (long long)p * 1504) % kPeriod) : -1;
        eff[p] = e;
    }
    if (hi == npackets && lo < hi) st->prbs_next = e >= 0 ? (e + 1496) % kPeriod : -1;
}

// ---------------------------------------------------------------------------------------------- output
__global__ void __launch_bounds__(256) out_kernel(const uint8_t* __restrict__ D, const uint8_t* __restrict__ dec, const int* __restrict__ src,
                                                  const int* __restrict__ eff, int npackets, OuterState* st, const uint8_t* __restrict__ prbs,
                                                  uint8_t* __restrict__ out, int32_t* __restrict__ errors) {
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int p = blockIdx.x * 8 + wid;
    if (p >= npackets) return;
    const uint8_t* data = src[p] >= 0 ? dec + (size_t)src[p] * 188 : st->obuf[st->cur];
    const uint8_t* rx = D + (size_t)p * kPkt;
    const int e = eff[p];
    int err = 0;
    for (int k = lane; k < 188; k += 32) {
        const uint8_t d = data[k];
        err += d != rx[k];
        uint8_t o = 0x47;
        if (k) o = e >= 0 ? (uint8_t)(d ^ prbs[(e + 8 * (k - 1)) % kPeriod]) : d;
        out[(size_t)p * 188 + k] = o;
        if (p == npackets - 1) st->obuf[st->cur ^ 1][k] = d;     // what the next call inherits
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) err += __shfl_xor_sync(0xFFFFFFFFu, err, off);
    if (lane == 0 && errors) errors[p] = err;                    // DVBSReedSolomon::decode's return value (:38-47)
}

__global__ void commit_kernel(OuterState* st) {
    st->cur ^= 1;
    st->prbs_off = st->prbs_next;
}

}  // namespace

struct dvbs2fec_dvbs_outer {
    int device = 0;
    cudaStream_t stream = nullptr;
    DevBuf<OuterState> st;
    DevBuf<GfTables> gf;
    DevBuf<uint8_t> prbs, D, dec, ok, in, out;
    DevBuf<int> src, eff;
    DevBuf<int32_t> err;
    ~dvbs2fec_dvbs_outer() {
        cudaSetDevice(device);
        if (stream) {
            cudaStreamSynchronize(stream);
            cudaStreamDestroy(stream);
        }
    }
};

extern "C" {

int dvbs2fec_dvbs_outer_reset(dvbs2fec_dvbs_outer* p) {
    if (!p) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    CU(cudaSetDevice(p->device));
    OuterState s;
    memset(&s, 0, sizeof s);            // FIFOs and obuffer zeroed (dvbs_interleaving.h:30-40, dvbs_reedsolomon.h:20-22), reg = 0
    s.prbs_off = -1;
    s.prbs_next = -1;
    CU(upload(p->st.p, &s, sizeof s));
    return 0;
}

int dvbs2fec_dvbs_outer_create(int device, dvbs2fec_dvbs_outer** out) {
    if (!out) return fail(DVBS2FEC_EINVAL, "out is NULL");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(DVBS2FEC_ENODEV, "no CUDA device");
    if (device < 0 || device >= ndev) return fail(DVBS2FEC_EINVAL, "device out of range");
    std::unique_ptr<dvbs2fec_dvbs_outer> p(new dvbs2fec_dvbs_outer());
    p->device = device;
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
    CU(p->st.reserve(1));
    CU(p->gf.reserve(1));
    CU(p->prbs.reserve(kPeriod + 1));
    // GF(256) as libcorrect builds it (field.h:24-45): x^8 + x^4 + x^3 + x^2 + 1, exp doubled, log[1] = 255
    GfTables g;
    memset(&g, 0, sizeof g);
    unsigned e = 1;
    g.exp[0] = 1;
    for (unsigned i = 1; i < 512; ++i) {
        e *= 2;
        if (e > 255) e ^= 0x11d;
        g.exp[i] = (uint8_t)e;
        if (i < 256) g.log[e] = (uint8_t)i;
    }
    CU(upload(p->gf.p, &g, sizeof g));
    // one period of the dispersal generator from its load value 0xa9 (dvbs_scrambling.h:16-28): entry o = the byte
    // prbs(8) returns after o clocks
    std::vector<uint8_t> bits(kPeriod + 8), tab(kPeriod + 1);
    int reg = 0xa9;
    for (int i = 0; i < kPeriod + 8; ++i) {
        const int fb = ((reg >> 13) ^ (reg >> 14)) & 1;
        reg = ((reg << 1) | fb) & 0x7fff;
        bits[(size_t)i] = (uint8_t)fb;
    }
    for (int o = 0; o < kPeriod; ++o) {
        int b = 0;
        for (int k = 0; k < 8; ++k) b = (b << 1) | bits[(size_t)(o + k)];
        tab[(size_t)o] = (uint8_t)b;
    }
    CU(upload(p->prbs.p, tab.data(), kPeriod));
    int rc = dvbs2fec_dvbs_outer_reset(p.get());
    if (rc) return rc;
    *out = p.release();
    return 0;
}

void dvbs2fec_dvbs_outer_destroy(dvbs2fec_dvbs_outer* p) { delete p; }

int dvbs2fec_dvbs_outer_process_device(dvbs2fec_dvbs_outer* p, int nframes, int frame_stride, const uint8_t* d_frames, uint8_t* d_out,
                                       int32_t* d_errors, void* stream) {
    if (!p || nframes < 0 || frame_stride < 1 || (nframes && (!d_frames || !d_out))) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (!nframes) return 0;
    if (nframes > (1 << 20)) return fail(DVBS2FEC_EINVAL, "more than 2^20 frames in one call");
    CU(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int np = nframes * 8;
    if ((size_t)nframes * kFrame > p->D.cap || (size_t)np > p->ok.cap) {
        CU(cudaStreamSynchronize(st));    // scratch grows only with everything enqueued so far finished
        CU(p->D.reserve((size_t)nframes * kFrame));
        CU(p->dec.reserve((size_t)np * 188));
        CU(p->ok.reserve(np));
        CU(p->src.reserve(np));
        CU(p->eff.reserve(np));
    }
    const long long cells = (long long)nframes * kFrame + kHist;
    deint_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, st>>>(d_frames, nframes, frame_stride, p->st.p, p->D.p);
    rs_kernel<<<nframes, 256, 0, st>>>(p->D.p, np, p->gf.p, p->dec.p, p->ok.p);
    scan_kernel<<<1, 1024, 0, st>>>(p->dec.p, p->ok.p, np, p->st.p, p->src.p, p->eff.p);
    out_kernel<<<nframes, 256, 0, st>>>(p->D.p, p->dec.p, p->src.p, p->eff.p, np, p->st.p, p->prbs.p, d_out, d_errors);
    commit_kernel<<<1, 1, 0, st>>>(p->st.p);
    CU(cudaGetLastError());
    return 0;
}

int dvbs2fec_dvbs_outer_process(dvbs2fec_dvbs_outer* p, int nframes, int frame_stride, const uint8_t* frames, uint8_t* out, int32_t* errors) {
    if (!p || nframes < 0 || frame_stride < 1 || (nframes && (!frames || !out))) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (!nframes) return 0;
    CU(cudaSetDevice(p->device));
    const size_t in_bytes = (size_t)(nframes - 1) * frame_stride + kFrame, np = (size_t)nframes * 8;
    CU(p->in.reserve(in_bytes));
    CU(p->out.reserve(np * 188));
    CU(p->err.reserve(np));
    CU(cudaMemcpyAsync(p->in.p, frames, in_bytes, cudaMemcpyHostToDevice, p->stream));
    int rc = dvbs2fec_dvbs_outer_process_device(p, nframes, frame_stride, p->in.p, p->out.p, p->err.p, p->stream);
    if (rc) return rc;
    CU(cudaMemcpyAsync(out, p->out.p, np * 188, cudaMemcpyDeviceToHost, p->stream));
    if (errors) CU(cudaMemcpyAsync(errors, p->err.p, np * sizeof(int32_t), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaStreamSynchronize(p->stream));
    return nframes * 8 * 188;
}

}  // extern "C"
