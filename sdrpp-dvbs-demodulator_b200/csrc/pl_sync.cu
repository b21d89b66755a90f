// K7: PL sync, PLHEADER demodulation, coarse frequency error.  See pl_sync.cuh.
//
// PL sync.  The reference gathers raw_frame_size symbols, slides a differential correlator over every position of
// that window (26 SOF + 32 PLS-code terms of conj(x[n-1]) x[n], dvbs2_pl_sync.cpp:109-143), realigns on the best
// position and goes on with the next window -- where the next window starts depends on the position just found.
// Here the correlation magnitude is computed for EVERY position of the call's symbols at once (a thread per
// position, the differential products shared through shared memory), and one CTA then walks the windows in
// order, each step a block-wide arg-max over values that are already there.  Frames are copied out by a third
// kernel, which also moves the symbols that stay behind to the front of the next call's work buffer.
// Every float operation is the reference's, in its order, without fused multiply-add (__fmul_rn / __fadd_rn).
#include "pl_sync.cuh"

#include <algorithm>

namespace s2 {
namespace {

constexpr int kMetricThreads = 256;
constexpr int kChainThreads = 1024;
constexpr uint32_t kSofValue = 0x18d2e82u;
constexpr unsigned long long kPlsScrambling = 0x719d83c953422dfaull;

__device__ __forceinline__ float2 cmul_rn(float2 a, float2 b) {   // complex_t::operator*
    return make_float2(__fsub_rn(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)), __fadd_rn(__fmul_rn(a.y, b.x), __fmul_rn(a.x, b.y)));
}
__device__ __forceinline__ float2 conj2(float2 a) { return make_float2(a.x, -a.y); }
__device__ __forceinline__ float camp_rn(float2 a) { return __fsqrt_rn(__fadd_rn(__fmul_rn(a.x, a.x), __fmul_rn(a.y, a.y))); }

// bit i set: term i is added (correlate_sof_diff, :167-181); PLS: bit i set (i odd): term i is subtracted (:183-193)
__host__ __device__ constexpr uint32_t sof_plus_mask() {
    uint32_t dsof = kSofValue ^ (kSofValue >> 1), m = 0;
    for (int i = 0; i < 26; ++i)
        if (((dsof >> (25 - i)) ^ (uint32_t)i) & 1u) m |= 1u << i;
    return m;
}
__host__ __device__ constexpr unsigned long long pls_minus_mask() {
    unsigned long long dscr = kPlsScrambling ^ (kPlsScrambling >> 1), m = 0;
    for (int i = 1; i < 64; i += 2)
        if ((dscr >> (63 - i)) & 1ull) m |= 1ull << i;
    return m;
}

__global__ void __launch_bounds__(256) plsync_append_kernel(const PlSyncArgs a) {
    float2* dst = a.work + a.st->pend;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < a.count; i += gridDim.x * 256) dst[i] = a.append[i];
}

// metric[n] = |d| when d.im > 0, else 0, for the 90 symbols starting at n (:109-131: "difference > best_match &&
// d.im > 0" with best_match starting at 0 -- a position with metric 0 can never win)
__global__ void __launch_bounds__(kMetricThreads) plsync_metric_kernel(const PlSyncArgs a) {
    __shared__ float2 sx[kMetricThreads + kPlHeader];
    __shared__ float2 sd[kMetricThreads + kPlHeader];
    const int L = a.st->pend + a.count;
    const int npos = L - (kPlHeader - 1);
    const int n0 = blockIdx.x * kMetricThreads, tid = threadIdx.x;
    if (n0 >= npos) return;
    for (int i = tid; i < kMetricThreads + kPlHeader; i += kMetricThreads) sx[i] = n0 + i < L ? a.work[n0 + i] : make_float2(0.f, 0.f);
    __syncthreads();
    // volk_32fc_conjugate_32fc + volk_32fc_x2_multiply_32fc (:112-113): conj(x[n-1]) x[n], product as VOLK's generic kernel
    for (int i = tid + 1; i < kMetricThreads + kPlHeader; i += kMetricThreads) {
        const float ar = sx[i - 1].x, ai = -sx[i - 1].y, br = sx[i].x, bi = sx[i].y;
        sd[i] = make_float2(__fsub_rn(__fmul_rn(ar, br), __fmul_rn(ai, bi)), __fadd_rn(__fmul_rn(ar, bi), __fmul_rn(ai, br)));
    }
    __syncthreads();
    const int n = n0 + tid;
    if (n >= npos) return;
    constexpr uint32_t sof_plus = sof_plus_mask();
    constexpr unsigned long long pls_minus = pls_minus_mask();
    float2 csof = make_float2(0.f, 0.f), cpls = make_float2(0.f, 0.f);
#pragma unroll
    for (int i = 1; i < 26; ++i) {   // term 0 is (0 + 0i) x[n]: adds nothing
        const float2 d = sd[tid + i];
        if ((sof_plus >> i) & 1u) { csof.x = __fadd_rn(csof.x, d.x); csof.y = __fadd_rn(csof.y, d.y); }
        else { csof.x = __fsub_rn(csof.x, d.x); csof.y = __fsub_rn(csof.y, d.y); }
    }
#pragma unroll
    for (int i = 1; i < 64; i += 2) {
        const float2 d = sd[tid + 26 + i];
        if ((pls_minus >> i) & 1ull) { cpls.x = __fsub_rn(cpls.x, d.x); cpls.y = __fsub_rn(cpls.y, d.y); }
        else { cpls.x = __fadd_rn(cpls.x, d.x); cpls.y = __fadd_rn(cpls.y, d.y); }
    }
    const float2 c0 = make_float2(__fadd_rn(csof.x, cpls.x), __fadd_rn(csof.y, cpls.y));   // best when b7 == 0 (pilots off)
    const float2 c1 = make_float2(__fsub_rn(csof.x, cpls.x), __fsub_rn(csof.y, cpls.y));   // best when b7 == 1
    const float2 c = camp_rn(c0) > camp_rn(c1) ? c0 : c1;
    const float k = 1.0f / (26 - 1 + 64 / 2);
    const float2 d = make_float2(__fmul_rn(c.x, k), __fmul_rn(c.y, k));
    a.metric[n] = d.y > 0.f ? camp_rn(d) : 0.f;
}

// internal_process (:102-165) over all windows the call completes.  starts[max_frames] receives the first symbol
// that stays behind.
__global__ void __launch_bounds__(kChainThreads) plsync_chain_kernel(const PlSyncArgs a) {
    __shared__ float s_val[32];
    __shared__ int s_idx[32];
    PlSyncState* S = a.st;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int L = S->pend + a.count, rfs = a.rfs;
    int s = 0, state = S->state, best_pos = S->best_pos, nfr = 0, curpos = S->current_position;
    double best_match = S->best_match;
    __syncthreads();   // everybody has read the state before thread 0 rewrites it
    for (;;) {
        if (state == 0) {
            if (s + rfs > L) break;
            // first position of the largest metric (the reference takes a later one only when strictly larger)
            float bv = 0.f;
            int bi = 0;
            for (int i = tid; i < rfs - kPlHeader; i += kChainThreads) {
                const float v = a.metric[s + i];
                if (v > bv) { bv = v; bi = i; }
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const float ov = __shfl_down_sync(0xFFFFFFFFu, bv, off);
                const int oi = __shfl_down_sync(0xFFFFFFFFu, bi, off);
                if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
            }
            __syncthreads();   // s_val / s_idx of the previous round have been read
            if (lane == 0) { s_val[warp] = bv; s_idx[warp] = bi; }
            __syncthreads();
            bv = s_val[lane];
            bi = s_idx[lane];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const float ov = __shfl_down_sync(0xFFFFFFFFu, bv, off);
                const int oi = __shfl_down_sync(0xFFFFFFFFu, bi, off);
                if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
            }
            bv = __shfl_sync(0xFFFFFFFFu, bv, 0);
            bi = __shfl_sync(0xFFFFFFFFu, bi, 0);
            best_pos = bv > 0.f ? bi : 0;
            best_match = (double)bv;
            if (bv > 0.f) curpos = bi;
            if (best_pos != 0) {   // (:145-150) gather best_pos more symbols, then deliver the realigned frame
                state = 1;
                continue;
            }
            if (tid == 0 && nfr < a.max_frames) a.starts[nfr] = s;
            ++nfr;
            s += rfs;
        } else {
            if (s + rfs + best_pos > L) break;
            if (tid == 0 && nfr < a.max_frames) a.starts[nfr] = s + best_pos;
            ++nfr;
            s += rfs + best_pos;
            best_pos = 0;
            state = 0;
        }
    }
    if (tid == 0) {
        nfr = min(nfr, a.max_frames);
        a.starts[a.max_frames] = s;
        S->state = state;
        S->best_pos = best_pos;
        S->pend = L - s;
        S->current_position = curpos;
        S->best_match = best_match;
        S->nframes = nfr;
        if (a.nframes_out) *a.nframes_out = nfr;
    }
}

// k < max_frames: frame k -> out; k == max_frames: what stays behind -> front of the next work buffer.  k runs from
// blockIdx.y in steps of gridDim.y, which is at most 65535.
__global__ void __launch_bounds__(256) plsync_copy_kernel(const PlSyncArgs a, int pend_before_upper) {
    const int nfr = a.st->nframes;
    for (int k = blockIdx.y; k <= a.max_frames; k += gridDim.y) {
        if (k < a.max_frames) {
            if (k >= nfr) continue;
            const float2* src = a.work + a.starts[k];
            float2* dst = a.out + (size_t)k * a.rfs;
            for (int i = blockIdx.x * 256 + threadIdx.x; i < a.rfs; i += gridDim.x * 256) dst[i] = src[i];
        } else {
            const float2* src = a.work + a.starts[a.max_frames];
            const int n = a.st->pend;
            for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) a.work_next[i] = src[i];
        }
    }
}

// ---------------------------------------------------------------------------------------------- PLHEADER
// PhaseControlLoop<float>::advance with the limits of S2PLHDRDemod::init (dvbs2_plhdr_demod.cpp:10)
__device__ __forceinline__ void pcl_advance(float& phase, float& freq, float alpha, float beta, float error) {
    const float pi = 3.1415926535f;
    freq = __fadd_rn(freq, __fmul_rn(beta, error));
    if (freq > pi) freq = pi;
    else if (freq < -pi) freq = -pi;
    phase = __fadd_rn(phase, __fadd_rn(freq, __fmul_rn(alpha, error)));
    const float delta = __fsub_rn(pi, -pi);
    while (phase > pi) phase = __fsub_rn(phase, delta);
    while (phase < -pi) phase = __fadd_rn(phase, delta);
}

__global__ void __launch_bounds__(32) plhdr_kernel(const float2* frames, int nframes, int rfs, float2* headers_out, PlHdrResult* res,
                                                   PlHdrState* st, const PlTables* tab) {
    const int lane = threadIdx.x;
    float phase = st->phase, freq = st->freq;
    const float alpha = st->alpha, beta = st->beta;
    const float2 rot = make_float2((float)cos(-M_PI / 4), (float)sin(-M_PI / 4));
    for (int f = 0; f < nframes; ++f) {
        const float2* x = frames + (size_t)f * rfs;
        unsigned long long plheader = 0;
        for (int i = 0; i < kPlHeader; ++i) {   // every lane runs the loop (the values are warp-uniform), lane 0 stores
            const float2 t = cmul_rn(x[i], make_float2(cosf(-phase), sinf(-phase)));
            const float error = __fsub_rn(__fmul_rn(t.x > 0.f ? 1.f : -1.f, t.y), __fmul_rn(t.y > 0.f ? 1.f : -1.f, t.x));
            const float2 o = (i & 1) ? make_float2(-t.x, t.y) : make_float2(t.y, t.x);
            if (lane == 0) headers_out[(size_t)f * kPlHeader + i] = o;
            if (i >= 26) plheader = plheader << 1 | (unsigned long long)!(cmul_rn(o, rot).x > 0.f);
            pcl_advance(phase, freq, alpha, beta, error);
        }
        phase = __fadd_rn(phase, __fmul_rn(freq, (float)(rfs - 91)));
        pcl_advance(phase, freq, alpha, beta, 0.f);
        // closest of the 128 codewords over bits 59..0 (checkSyncMarker, :69-79), the first one among equals
        int bd = 64, bc = 0;
        for (int c = lane; c < 128; c += 32) {
            const int d = __popcll((tab->codewords[c] ^ plheader) & ((1ull << 60) - 1));
            if (d < bd) { bd = d; bc = c; }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const int od = __shfl_xor_sync(0xFFFFFFFFu, bd, off), oc = __shfl_xor_sync(0xFFFFFFFFu, bc, off);
            if (od < bd || (od == bd && oc < bc)) { bd = od; bc = oc; }
        }
        if (lane == 0) res[f] = PlHdrResult{(bc >> 2) & 31, (bc & 2) >> 1, bc & 1, bc};
    }
    if (lane == 0) {
        st->phase = phase;
        st->freq = freq;
    }
}

// ---------------------------------------------------------------------------------------------- coarse FED
__global__ void __launch_bounds__(128) fed_kernel(const float2* frames, int nframes, int rfs, int pilots, int pls_code, const uint8_t* rn,
                                                  const PlTables* tab, float* err_out) {
    const int f = blockIdx.x * 128 + threadIdx.x;
    if (f >= nframes) return;
    const float2* frame = frames + (size_t)f * rfs;
    const float2* sof = tab->sof;
    const float2* pl = tab->pls[pls_code & 127];
    float err = 0.f, symcnt = 90 - 2;
    auto term = [](float2 a, float2 b, float2 c, float2 d) { return cmul_rn(cmul_rn(cmul_rn(a, conj2(b)), conj2(c)), d).y; };
    for (int i = 0; i < 26 - 2; ++i) err = __fadd_rn(err, term(frame[i + 2], sof[i + 2], frame[i], sof[i]));
    err = __fadd_rn(err, term(frame[24 + 2], pl[24 - 26 + 2], frame[24], sof[24]));
    err = __fadd_rn(err, term(frame[25 + 2], pl[25 - 26 + 2], frame[25], sof[25]));
    for (int i = 26; i < 90 - 2; ++i) err = __fadd_rn(err, term(frame[i + 2], pl[i - 26 + 2], frame[i], pl[i - 26]));
    if (pilots) {
        float2 t1 = make_float2(0.f, 0.f), t2 = make_float2(0.f, 0.f);
        const float2 ref = make_float2(0.707f, 0.707f);
        for (int blk = 0; blk < ((rfs / 90 - 1) / 16) - 1; ++blk) {
            const int startsym = 90 * 17 + blk * (90 * 16 + 37);   // (sic, dvbs2_fed.h:29)
            int pos = startsym - 90;
            for (int i = 0; i < 36; ++i) {
                const float2 p = frame[startsym + i];
                float2 d;
                switch (rn[pos++]) {   // S2Scrambling::descramble (s2_scrambling.cpp:37-58)
                case 3: d = make_float2(-p.y, p.x); break;
                case 2: d = make_float2(-p.x, -p.y); break;
                case 1: d = make_float2(p.y, -p.x); break;
                default: d = p; break;
                }
                if (i >= 2) err = __fadd_rn(err, term(d, ref, t2, ref));
                t2 = t1;
                t1 = d;
            }
            symcnt = __fadd_rn(symcnt, 36 - 2);
        }
    }
    err_out[f] = __fdiv_rn(err, symcnt);
}

}  // namespace

int plsync_launch(const PlSyncArgs& a, int pend_upper_bound, cudaStream_t stream) {
    const int lmax = pend_upper_bound + a.count;
    if (a.append && a.count > 0) plsync_append_kernel<<<std::min((a.count + 255) / 256, 1184), 256, 0, stream>>>(a);
    if (lmax >= kPlHeader) plsync_metric_kernel<<<(lmax - kPlHeader + 1 + kMetricThreads - 1) / kMetricThreads, kMetricThreads, 0, stream>>>(a);
    plsync_chain_kernel<<<1, kChainThreads, 0, stream>>>(a);
    plsync_copy_kernel<<<dim3(16, std::min(a.max_frames + 1, 65535)), 256, 0, stream>>>(a, pend_upper_bound);
    return (int)cudaGetLastError();
}

int plhdr_launch(const float2* frames, int nframes, int rfs, float2* headers_out, PlHdrResult* res, PlHdrState* st, const PlTables* tab,
                 cudaStream_t stream) {
    if (nframes > 0) plhdr_kernel<<<1, 32, 0, stream>>>(frames, nframes, rfs, headers_out, res, st, tab);
    return (int)cudaGetLastError();
}

int fed_launch(const float2* frames, int nframes, int rfs, int pilots, int pls_code, const uint8_t* rn, const PlTables* tab, float* err_out,
               cudaStream_t stream) {
    if (nframes > 0) fed_kernel<<<(nframes + 127) / 128, 128, 0, stream>>>(frames, nframes, rfs, pilots, pls_code, rn, tab, err_out);
    return (int)cudaGetLastError();
}

}  // namespace s2
