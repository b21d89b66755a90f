// K10: the TS deframer of the DVB-S chain on the device (SURVEY.md 8(f) rank 4): DVBS_TS_Deframer::work
// (dvbs/dvbs_ts_deframer.cpp:44-101) and the C ABI dvbs2fec_dvbs_deframer_* around it.
//
// The reference pushes every bit of the Viterbi decoder's output (one bit per byte) into a window of 8 x 204 x 8 bits
// by moving the whole 13056-byte array, packs the eight sync bytes of the window and counts how many of their 64 bits
// differ from B8 47 47 47 47 47 47 47; at most 8 -> the window goes out as a frame of 1632 bytes, at least 56 (at most 8
// against the inverted pattern) -> it goes out inverted.  Every window position is independent of every other:
//   pack     the bits of the call, behind the 13055 carried over from the call before, into 32-bit words;
//   detect   a thread per window position: eight funnel shifts and population counts; the hits of a block of 256
//            positions are compacted in order;
//   collect  one CTA scans the per-block counts and strings the hits together in stream order;
//   frames   a CTA per frame: 408 words by funnel shift (inverted where the pattern was), stored byte-swapped;
//   carry    the last 13055 bits for the next call.
// Input bytes are taken as their lowest bit (the decoder delivers 0 or 1; the reference ORs whole bytes into its
// packing, which is the same thing for 0 / 1).  The reference's window is allocated uninitialised; here -- as in the
// oracle and in the harness around the compiled reference -- it starts from zeros.
#include "../../include/dvbs2fec.h"

#include <cstring>
#include <memory>

#include <cuda_runtime.h>

#include "abi_util.h"

using namespace s2;

namespace {

constexpr int kWindow = 13056;          // bits: 8 packets x 204 bytes x 8
constexpr int kCarry = kWindow - 1;     // bits kept from call to call
constexpr int kDetect = 256;

struct DeframerState {
    int nframes;        // frames the last call found (before the caller's limit)
    int written;        // ... and wrote
    int errors_nor, errors_inv;   // public members (dvbs_ts_deframer.h:24-25)
};

__device__ __forceinline__ uint32_t stream_bit(const uint8_t* hist, const uint8_t* in, int size, long long idx) {
    if (idx < kCarry) return hist[idx] & 1u;
    idx -= kCarry;
    return idx < size ? (in[idx] & 1u) : 0u;
}

__global__ void __launch_bounds__(256) pack_kernel(const uint8_t* __restrict__ hist, const uint8_t* __restrict__ in, int size, uint32_t* __restrict__ W,
                                                   int nwords) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nwords) return;
    uint32_t v = 0;
    const long long base = 32ll * w;
#pragma unroll 8
    for (int k = 0; k < 32; ++k) v = v << 1 | stream_bit(hist, in, size, base + k);
    W[w] = v;      // bit 31 = the first bit
}

// 32 bits of the packed stream starting at bit offset o
__device__ __forceinline__ uint32_t bits32(const uint32_t* __restrict__ W, long long o) {
    const long long w = o >> 5;
    return __funnelshift_l(W[w + 1], W[w], (unsigned)(o & 31));
}

__global__ void __launch_bounds__(kDetect) detect_kernel(const uint32_t* __restrict__ W, int size, uint32_t* __restrict__ blockhits, int* __restrict__ counts) {
    __shared__ int warp_base[kDetect / 32];
    const int s = blockIdx.x * kDetect + threadIdx.x;     // window start in the packed stream = index of the newest bit in the call
    bool hit = false;
    uint32_t rec = 0;
    if (s < size) {
        int t_nor = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const uint32_t b = bits32(W, (long long)s + 1632ll * i) >> 24;
            t_nor += __popc(b ^ (i == 0 ? 0xB8u : 0x47u));
        }
        // against the inverted pattern the count is 64 - t_nor (0x47 = ~0xB8): the two tests (:76,88) exclude each other
        if (t_nor <= 8) { hit = true; rec = (uint32_t)s | (uint32_t)t_nor << 24; }
        else if (64 - t_nor <= 8) { hit = true; rec = (uint32_t)s | (uint32_t)(64 - t_nor) << 24 | 0x80000000u; }
    }
    const unsigned m = __ballot_sync(0xFFFFFFFFu, hit);
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) warp_base[wid] = __popc(m);
    __syncthreads();
    int base = 0, total = 0;
    for (int k = 0; k < kDetect / 32; ++k) {
        if (k < wid) base += warp_base[k];
        total += warp_base[k];
    }
    if (hit) blockhits[(size_t)blockIdx.x * kDetect + base + __popc(m & ((1u << lane) - 1))] = rec;
    if (threadIdx.x == 0) counts[blockIdx.x] = total;
}

__global__ void __launch_bounds__(1024) collect_kernel(const uint32_t* __restrict__ blockhits, const int* __restrict__ counts, int nblocks, int max_frames,
                                                       uint32_t* __restrict__ hits, DeframerState* st, int* nframes_out) {
    __shared__ int sm[1024];
    __shared__ int carry;
    __shared__ uint32_t last_rec;
    const int tid = threadIdx.x;
    if (tid == 0) { carry = 0; last_rec = 0xFFFFFFFFu; }
    __syncthreads();
    for (int b0 = 0; b0 < nblocks; b0 += 1024) {
        const int b = b0 + tid;
        const int c = b < nblocks ? counts[b] : 0;
        sm[tid] = c;
        __syncthreads();
        for (int off = 1; off < 1024; off <<= 1) {
            const int o = tid >= off ? sm[tid - off] : 0;
            __syncthreads();
            sm[tid] += o;
            __syncthreads();
        }
        const int start = carry + sm[tid] - c;
        for (int k = 0; k < c; ++k)
            if (start + k < max_frames) hits[start + k] = blockhits[(size_t)b * kDetect + k];
        __syncthreads();
        if (tid == 1023) carry += sm[1023];
        __syncthreads();
    }
    // the public error counters are those of the last window that matched, written or not (:83-84,95-96)
    if (tid == 0) {
        for (int b = nblocks - 1; b >= 0; --b)
            if (counts[b]) { last_rec = blockhits[(size_t)b * kDetect + counts[b] - 1]; break; }
        st->nframes = carry;
        st->written = min(carry, max_frames);
        if (last_rec != 0xFFFFFFFFu) {
            const int e = (int)((last_rec >> 24) & 0x7F);
            st->errors_nor = (last_rec & 0x80000000u) ? 0 : e;
            st->errors_inv = (last_rec & 0x80000000u) ? e : 0;
        }
        if (nframes_out) *nframes_out = st->written;
    }
}

__global__ void __launch_bounds__(416) frames_kernel(const uint32_t* __restrict__ W, const uint32_t* __restrict__ hits, const DeframerState* st,
                                                     uint32_t* __restrict__ out) {
    const int f = blockIdx.x;
    if (f >= st->written) return;
    const uint32_t rec = hits[f];
    const long long s = rec & 0xFFFFFFu;
    const uint32_t inv = (rec & 0x80000000u) ? 0xFFFFFFFFu : 0u;
    const int j = threadIdx.x;
    if (j < 408) out[(size_t)f * 408 + j] = __byte_perm(bits32(W, s + 32ll * j) ^ inv, 0, 0x0123);   // first bit = MSB of byte 0
}

__global__ void __launch_bounds__(256) carry_kernel(const uint8_t* __restrict__ hist, const uint8_t* __restrict__ in, int size, uint8_t* __restrict__ next) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < kCarry) next[i] = (uint8_t)stream_bit(hist, in, size, (long long)size + i);
}

}  // namespace

struct dvbs2fec_dvbs_deframer {
    int device = 0;
    cudaStream_t stream = nullptr;
    DevBuf<DeframerState> st;
    DevBuf<uint8_t> hist[2];
    int cur = 0;
    DevBuf<uint32_t> W, blockhits, hits, out;
    DevBuf<int> counts;
    DevBuf<uint8_t> in;
    ~dvbs2fec_dvbs_deframer() {
        cudaSetDevice(device);
        if (stream) {
            cudaStreamSynchronize(stream);
            cudaStreamDestroy(stream);
        }
    }
};

extern "C" {

int dvbs2fec_dvbs_deframer_reset(dvbs2fec_dvbs_deframer* p) {
    if (!p) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    CU(cudaSetDevice(p->device));
    CU(cudaMemset(p->st.p, 0, sizeof(DeframerState)));
    CU(cudaMemset(p->hist[0].p, 0, kWindow));
    CU(cudaMemset(p->hist[1].p, 0, kWindow));
    CU(cudaDeviceSynchronize());      // device memsets are asynchronous, and the callers' streams do not wait for the default stream
    p->cur = 0;
    return 0;
}

int dvbs2fec_dvbs_deframer_create(int device, dvbs2fec_dvbs_deframer** out) {
    if (!out) return fail(DVBS2FEC_EINVAL, "out is NULL");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(DVBS2FEC_ENODEV, "no CUDA device");
    if (device < 0 || device >= ndev) return fail(DVBS2FEC_EINVAL, "device out of range");
    std::unique_ptr<dvbs2fec_dvbs_deframer> p(new dvbs2fec_dvbs_deframer());
    p->device = device;
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
    CU(p->st.reserve(1));
    CU(p->hist[0].reserve(kWindow));
    CU(p->hist[1].reserve(kWindow));
    int rc = dvbs2fec_dvbs_deframer_reset(p.get());
    if (rc) return rc;
    *out = p.release();
    return 0;
}

void dvbs2fec_dvbs_deframer_destroy(dvbs2fec_dvbs_deframer* p) { delete p; }

int dvbs2fec_dvbs_deframer_work_device(dvbs2fec_dvbs_deframer* p, const uint8_t* d_bits, int size, uint8_t* d_frames, int max_frames,
                                       int32_t* d_nframes, void* stream) {
    if (!p || size < 0 || max_frames < 0 || (size && !d_bits) || (max_frames && !d_frames)) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (size >= (1 << 24)) return fail(DVBS2FEC_EINVAL, "more than 2^24 - 1 bits in one call");
    if ((reinterpret_cast<uintptr_t>(d_frames) & 3u) != 0) return fail(DVBS2FEC_EINVAL, "frame buffer must be 4-byte aligned");
    CU(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (!size) {
        if (d_nframes) CU(cudaMemsetAsync(d_nframes, 0, sizeof(int), st));
        return 0;
    }
    const int nwords = (kCarry + size + 31) / 32 + 2, nblocks = (size + kDetect - 1) / kDetect;
    if ((size_t)nwords > p->W.cap || (size_t)nblocks > p->counts.cap || (size_t)max_frames + 1 > p->hits.cap) {
        CU(cudaStreamSynchronize(st));
        CU(p->W.reserve((size_t)nwords));
        CU(p->blockhits.reserve((size_t)nblocks * kDetect));
        CU(p->counts.reserve((size_t)nblocks));
        CU(p->hits.reserve((size_t)max_frames + 1));
    }
    const uint8_t* hist = p->hist[p->cur].p;
    pack_kernel<<<(nwords + 255) / 256, 256, 0, st>>>(hist, d_bits, size, p->W.p, nwords);
    detect_kernel<<<nblocks, kDetect, 0, st>>>(p->W.p, size, p->blockhits.p, p->counts.p);
    collect_kernel<<<1, 1024, 0, st>>>(p->blockhits.p, p->counts.p, nblocks, max_frames, p->hits.p, p->st.p, d_nframes);
    if (max_frames) frames_kernel<<<max_frames, 416, 0, st>>>(p->W.p, p->hits.p, p->st.p, reinterpret_cast<uint32_t*>(d_frames));
    carry_kernel<<<(kCarry + 255) / 256, 256, 0, st>>>(hist, d_bits, size, p->hist[p->cur ^ 1].p);
    CU(cudaGetLastError());
    p->cur ^= 1;
    return 0;
}

int dvbs2fec_dvbs_deframer_work(dvbs2fec_dvbs_deframer* p, const uint8_t* bits, int size, uint8_t* frames, int max_frames) {
    if (!p || size < 0 || max_frames < 0 || (size && !bits) || (max_frames && !frames)) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (!size) return 0;
    CU(cudaSetDevice(p->device));
    // a frame cannot follow another in less than one bit; the caller's limit bounds what is written
    CU(p->in.reserve((size_t)size));
    CU(p->out.reserve((size_t)max_frames * 408 + 1));
    CU(cudaMemcpyAsync(p->in.p, bits, (size_t)size, cudaMemcpyHostToDevice, p->stream));
    int rc = dvbs2fec_dvbs_deframer_work_device(p, p->in.p, size, reinterpret_cast<uint8_t*>(p->out.p), max_frames, nullptr, p->stream);
    if (rc) return rc;
    DeframerState s;
    CU(cudaMemcpyAsync(&s, p->st.p, sizeof s, cudaMemcpyDeviceToHost, p->stream));
    CU(cudaStreamSynchronize(p->stream));
    if (s.written) {
        CU(cudaMemcpyAsync(frames, p->out.p, (size_t)s.written * 1632, cudaMemcpyDeviceToHost, p->stream));
        CU(cudaStreamSynchronize(p->stream));
    }
    return s.written;
}

int dvbs2fec_dvbs_deframer_stats(dvbs2fec_dvbs_deframer* p, int* errors_nor, int* errors_inv, int* found) {
    if (!p) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    CU(cudaSetDevice(p->device));
    DeframerState s;
    CU(cudaMemcpy(&s, p->st.p, sizeof s, cudaMemcpyDeviceToHost));
    if (errors_nor) *errors_nor = s.errors_nor;
    if (errors_inv) *errors_inv = s.errors_inv;
    if (found) *found = s.nframes;
    return s.written;
}

}  // extern "C"
