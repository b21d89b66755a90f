// K11: the inner decoder of the DVB-S chain on the device (SURVEY.md 8(f) rank 4): DVBSymToSoftBlock::process
// (dvbs/dvbs_syms_to_soft.cpp:26-42), DVBSVitBlock::process (dvbs/dvbs_vit.cpp:6-13) and behind it the self-locking
// punctured K = 7 decoder viterbi::Viterbi_DVBS (dvbs/viterbi_all.cpp:75-318) with its CCDecoder (the bundled generic
// butterfly, dvbs/viterbi/volk_k7_r2_generic_fixed.h:42-115, traceback cc_decoder.cpp:242-283), CCEncoder re-encoding
// BER test, the depuncturers (dvbs/depunc.h, viterbi_all.h:93-151) and rotate_soft / signed_soft_to_unsigned.
//
// How the reference's strictly sequential object becomes a batch:
//  * every work() call decodes ONE block of 8192 soft bits with freshly biased metrics; the only thing a decoder carries
//    from call to call is the state its traceback reached at the block's end (6 bits).  So a batch is a set of decode
//    TASKS chained through one small integer each.  A guess kernel runs the last 326 trellis steps of every task from
//    flat metrics and traces 6 steps back -- survivors have long merged by then, so that is the carried state in all
//    but pathological inputs; the decode kernel runs every task in parallel from its predecessor's guess; a check
//    compares each task's start with what its predecessor really reached and repeats the tasks that were wrong until
//    nothing changes.  The result is the sequential result, not an approximation.
//  * a task = a warp: lane i owns butterfly i (states 2i, 2i+1 as the two 16-bit halves of one register), the two
//    inputs come by shuffle, add-compare-select is a packed 16-bit minimum with the reference's 8-bit wrap-around kept
//    by masking, decisions leave by ballot, the per-step renormalisation is a warp min-reduction; the traceback is cut
//    into 32 pieces, one per lane, each started 128 steps early from an arbitrary state and accepted only if every
//    piece began where the piece above it ended (otherwise the task is walked back step by step).
//  * the lock search (52 candidate decodes per call: 2 phases x 26 rate / puncturing-shift branches) is the same kind
//    of task; a CTA per block replays the reference's buffer writes in shared memory so that every candidate sees
//    the stale bytes the reference's decoders read past their depunctured input (viterbi_all.cpp:89,107,127,167).
//  * the state machine (lock / count bad calls / give up the lock) runs on the host over the per-block BER counts; a
//    batch is computed under the assumption that the state at its start lasts, and cut where that stops being true.
// Results are bit-identical to the reference's -- decoded bits, BER, lock parameters after every call -- including what
// it does wrong (rate 5/6 decodes 6799 of 6826 steps per call and leaves the other output bits unwritten; rate 2/3
// decodes a step of stale data every third call): tests/test_gpu_vit.py against the oracle, which
// tests/test_vit_oracle.py pins to the compiled reference (bundled generic kernel; a reference built against a VOLK
// with the "spiral" kernel runs that instead and is unpinned).
#include "../../include/dvbs2fec.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <vector>

#include <cuda_runtime.h>

#include "abi_util.h"

using s2::DevBuf;
using s2::fail;

namespace {

constexpr int kBuf = 8192;            // VIT_BUF_SIZE (dvbs/dvbs_defines.h)
constexpr int kTest = 2048;           // TEST_BITS_LENGTH
constexpr int kGuessSteps = 326;      // trellis steps the guess kernel runs (320 + the 6 behind the block)
constexpr int kSearchTasks = 52;
constexpr int kWarm = 128;            // traceback steps a lane runs above its piece before its bits count
constexpr int kMaxSearchBlocks = 64, kMaxSyncBlocks = 8192;
enum { R12, R23, R34, R56, R78 };
const int kShifts[5] = {2, 6, 2, 12, 4};
const float kRatio[5] = {2.5f, 3.5f, 5.0f, 8.0f, 10.0f};
// frame sizes and BER lengths as the constructor's double arithmetic truncates them (viterbi_all.cpp:17-33,92,110,130,150,170)
const int kFsBer[5] = {kTest / 2, (int)(kTest * 1.334 / 2), (int)(kTest * 1.5 / 2), (int)(kTest * 1.66 / 2), (int)(kTest * 1.75 / 2)};
const int kFsMain[5] = {kBuf / 2, 10924 / 2, (int)(kBuf * 1.5 / 2), (int)(kBuf * 1.66 / 2), (int)(kBuf * 1.75 / 2)};
const int kBerLen[5] = {kTest, (int)(kTest * 1.25), (int)(kTest * 1.5), (int)(kTest * 1.66), (int)(kTest * 1.75)};

inline int pad16(int n) { return (n + 15) & ~15; }

struct VTask {
    uint32_t img;        // byte offset of the input image (16-byte aligned)
    uint32_t out;        // byte offset of the decoded bits
    uint32_t dec;        // offset of the decision words (uint2 units)
    int nsteps, fs;      // d_veclen, d_frame_size
    int pred, start;     // decoder chain: task whose end state I start from; or (pred < 0) start itself, -1 = flat 31s (first use)
    int enc_pred, enc_state, enc_fs;   // re-encoder chain: its register holds the last 6 bits it saw
    int ber_len;
    int stale_task, stale_bit;         // rate 5/6: get_ber reads re-encoded bit 3398, which only rate 7/8 ever writes; -2: not read
    int is78;
};
struct VResult {
    int guess, start_used, retval, need;
    int errors, total, enc_end, bit3398;
};

// ---------------------------------------------------------------------------------------------------- soft bits
// rotate_soft (rotation.cpp:9-42, phases 0 and 90) + signed_soft_to_unsigned (utils.cpp:11-20) of soft bit idx of a block
__device__ __forceinline__ uint32_t soft_u8(const int8_t* __restrict__ blk, int idx, int phase) {
    int v;
    if (phase == 0) v = blk[idx];
    else if (idx & 1) { v = blk[idx - 1]; v = -(v == -128 ? -127 : v); }
    else v = blk[idx + 1];
    if (v == -128) v = -127;
    const uint32_t u = (uint32_t)(v + 127) & 0xFFu;
    return u == 128u ? 127u : u;
}

// a depuncturing pattern: the output slots of one period, each with the input (index within the period) it is emitted
// with and whether it is that input or the erasure next to it; prefix[a] = slots before input a
struct Pattern { int pin, pout; int8_t owner[14]; int8_t era[14]; int8_t prefix[9]; };
enum { P23 = 0, P56 = 1, P34 = 2, P78 = 4, kPatterns = 8 };
__constant__ Pattern cPat[kPatterns];

// slot q of the stream that starts with input 0 at phase a: the input index it carries, -1 for an erasure, -2 when
// nin inputs do not reach that far
__device__ __forceinline__ int pat_source(const Pattern& P, int a, int q, int nin) {
    const int qq = q + P.prefix[a];
    const int per = qq / P.pout, w = qq - per * P.pout;
    const int idx = per * P.pin + P.owner[w] - a;
    if (idx >= nin) return -2;
    return P.era[w] ? -1 : idx;
}
__host__ __device__ inline int pat_count(const Pattern& P, int a, int nin) {
    const int n = a + nin;
    return (n / P.pin) * P.pout + P.prefix[n % P.pin] - P.prefix[a];
}

// ---- lock search: the 52 candidate inputs of one block (viterbi_all.cpp:79-189) --------------------------------------------
struct SearchLayout { int img[26]; int nread[26]; int rate[26]; int shift[26]; int per_phase; };
__constant__ SearchLayout cSearch;

__global__ void __launch_bounds__(256) search_image_kernel(const int8_t* __restrict__ in, const int8_t* __restrict__ prev_in, int have_prev,
                                                           uint8_t* __restrict__ images, uint32_t block_stride) {
    __shared__ uint8_t buf[kTest + 3600];      // ber_soft_buffer followed by ber_depunc_buffer (viterbi_all.h:78-79)
    uint8_t* bsoft = buf;
    uint8_t* bdep = buf + kTest;
    const int b = blockIdx.x, tid = threadIdx.x;
    const int8_t* blk = in + (size_t)b * kBuf;
    // what the previous search left in ber_depunc_buffer: its last candidate, rate 7/8 shift 3 at phase 90 (3584 bytes);
    // behind that nothing is ever written (zeros from construction)
    const int8_t* pblk = b > 0 ? in + (size_t)(b - 1) * kBuf : prev_in;
    const bool hp = b > 0 || have_prev;
    for (int q = tid; q < 3600; q += 256) {
        uint32_t v = 0;
        if (hp && q < 3584) {
            const int src = pat_source(cPat[P78 + 3], 0, q, kTest);
            v = src >= 0 ? soft_u8(pblk, src, 1) : 128u;
        }
        bdep[q] = (uint8_t)v;
    }
    uint8_t* out = images + (size_t)b * block_stride;
    for (int phase = 0; phase < 2; ++phase) {
        __syncthreads();
        for (int i = tid; i < kTest; i += 256) bsoft[i] = (uint8_t)soft_u8(blk, i, phase);
        __syncthreads();
        for (int c = 0; c < 26; ++c) {
            const int r = cSearch.rate[c], sh = cSearch.shift[c], nread = cSearch.nread[c];
            uint8_t* img = out + phase * cSearch.per_phase + cSearch.img[c];
            if (r == R12) {       // decoder input = ber_soft_buffer + shift, running 12 / 13 bytes into the buffer behind
                for (int p = tid; p < nread; p += 256) img[p] = buf[p + sh];
                __syncthreads();      // the next candidate writes where this one read its last bytes
                continue;
            }
            int lead = 0, a = 0, oo;
            const Pattern* P;
            if (r == R23) { P = &cPat[P23]; lead = sh > 2; a = sh % 3; }
            else if (r == R56) { P = &cPat[P56]; lead = sh > 5; a = sh % 6; }
            else if (r == R34) P = &cPat[P34 + sh];
            else P = &cPat[P78 + sh];
            oo = lead + pat_count(*P, a, kTest);
            for (int q = tid; q < oo; q += 256) {
                uint32_t v = 128u;
                if (q >= lead) {
                    const int src = pat_source(*P, a, q - lead, kTest);
                    if (src >= 0) v = bsoft[src];
                }
                bdep[q] = (uint8_t)v;
            }
            __syncthreads();
            for (int p = tid; p < nread; p += 256) img[p] = bdep[p];
            __syncthreads();
        }
    }
}

// ---- locked: the decoder input of every block (viterbi_all.cpp:196-250) -------------------------------------------------
struct ContDesc { int lead, c, oo, stale_src[2]; };      // Depunc23 / Depunc56 ::depunc_cont state at the block's start
struct ContRec { int buf_val, v[2]; };                   // ... what the block leaves behind: the byte held back, depunc_buffer[10922..10923]

// byte p (< oo) of what depunc_cont wrote for block k
__device__ uint32_t cont_value(const Pattern& P, const ContDesc* __restrict__ desc, const int8_t* __restrict__ in, int phase, int k, int p,
                               int carried_buf) {
    const ContDesc d = desc[k];
    if (p == 0 && d.lead) {
        if (k == 0) return (uint32_t)carried_buf;
        const ContDesc e = desc[k - 1];      // the byte block k - 1 held back: its last one (never its own lead)
        const int src = pat_source(P, e.c, e.oo - 1 - e.lead, kBuf);
        return src >= 0 ? soft_u8(in + (size_t)(k - 1) * kBuf, src, phase) : 128u;
    }
    const int src = pat_source(P, d.c, p - d.lead, kBuf);
    return src >= 0 ? soft_u8(in + (size_t)k * kBuf, src, phase) : 128u;
}

__global__ void __launch_bounds__(256) sync_image_kernel(const int8_t* __restrict__ in, int rate, int phase, int shift, int nread,
                                                         const ContDesc* __restrict__ desc, ContRec* __restrict__ rec, int carried_buf, int carried_v0,
                                                         int carried_v1, uint8_t* __restrict__ images, uint32_t block_stride) {
    const int k = blockIdx.x;
    const int8_t* blk = in + (size_t)k * kBuf;
    uint8_t* img = images + (size_t)k * block_stride;
    const int carried_v[2] = {carried_v0, carried_v1};
    for (int p = blockIdx.y * 256 + threadIdx.x; p < nread; p += gridDim.y * 256) {
        uint32_t v = 128u;      // soft_buffer / depunc_buffer are set to 128 when the lock is taken (:99-100)
        if (rate == R12) {
            if (p + shift < kBuf) v = soft_u8(blk, p + shift, phase);
        } else if (rate == R34 || rate == R78) {
            const int src = pat_source(cPat[(rate == R34 ? P34 : P78) + shift], 0, p, kBuf);
            if (src >= 0) v = soft_u8(blk, src, phase);
        } else {
            const Pattern& P = cPat[rate == R23 ? P23 : P56];
            if (p < desc[k].oo) v = cont_value(P, desc, in, phase, k, p, carried_buf);
            else if (rate == R23 && (p == 10922 || p == 10923)) {      // what an earlier call left there
                const int j = desc[k].stale_src[p - 10922];
                v = j >= 0 ? cont_value(P, desc, in, phase, j, p, carried_buf) : (uint32_t)carried_v[p - 10922];
            }
        }
        img[p] = (uint8_t)v;
    }
    if (rec && blockIdx.y == 0 && threadIdx.x < 3) {
        const Pattern& P = cPat[rate == R23 ? P23 : P56];
        const ContDesc d = desc[k];
        if (threadIdx.x == 0) rec[k].buf_val = (int)cont_value(P, desc, in, phase, k, d.oo - 1, carried_buf);
        else {
            const int i = threadIdx.x - 1, p = 10922 + i;
            int v = 128;
            if (rate == R23) {
                const int j = p < d.oo ? k : d.stale_src[i];
                v = j >= 0 ? (int)cont_value(P, desc, in, phase, j, p, carried_buf) : carried_v[i];
            }
            rec[k].v[i] = v;
        }
    }
}

// ---- the decoder proper: CCDecoder::work (cc_decoder.cpp:295-316) for one task per warp ----------------------------------
// mode 0: guess (last kGuessSteps steps from flat metrics, 6 steps of traceback); 1: decode from the predecessor's guess;
// 2: decode again where the check found the start wrong
__device__ __forceinline__ uint32_t acs_step(uint32_t y, uint32_t Pj, int lane, uint32_t selx, uint32_t selm, uint32_t& w0, uint32_t& w1) {
    const uint32_t a = __shfl_sync(0xFFFFFFFFu, y, lane >> 1), b = __shfl_sync(0xFFFFFFFFu, y, 16 + (lane >> 1));
    const uint32_t x0 = __byte_perm(a, 0, selx), x1 = __byte_perm(b, 0, selx);      // X[i] and X[i + 32] in both halves
    const uint32_t bm = __byte_perm(Pj, 0, selm);                                    // this butterfly's branch metric
    const uint32_t mp = bm * 0xFFFF0001u + (63u << 16);                              // metric | (63 - metric) << 16
    const uint32_t mq = 63u * 0x10001u - mp;                                         // (63 - metric) | metric << 16
    const uint32_t q0 = (x0 + mp) & 0x00FF00FFu;                                     // m0 | m2 << 16, each wrapped to 8 bits as the reference's
    const uint32_t q1 = (x1 + mq) & 0x00FF00FFu;                                     // m1 | m3 << 16
    uint32_t yn = __vminu2(q0, q1);
    const uint32_t e = yn ^ q1;                                                      // a half is 0 where m1 (m3) was taken: m0 >= m1 (m2 >= m3)
    w0 = __ballot_sync(0xFFFFFFFFu, (e & 0xFFFFu) == 0);
    w1 = __ballot_sync(0xFFFFFFFFu, (e & 0xFFFF0000u) == 0);
    const uint32_t m = __reduce_min_sync(0xFFFFFFFFu, min(yn & 0xFFFFu, yn >> 16));  // renormalize (:25-38)
    return yn - m * 0x10001u;
}

__global__ void __launch_bounds__(128) acs_kernel(const VTask* __restrict__ tasks, VResult* __restrict__ res, int ntasks, int mode,
                                                  const uint8_t* __restrict__ images, uint2* __restrict__ decpool, uint8_t* __restrict__ decoded, int* __restrict__ walks) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= ntasks) return;
    const VTask t = tasks[warp];
    int start = 0;
    if (mode == 1) start = t.pred >= 0 ? res[t.pred].guess : t.start;
    else if (mode == 2) {
        if (!res[warp].need) return;
        start = res[warp].start_used;
    }
    // Branchtab (cc_decoder.cpp:127-134): 255 where the parity of (2 i) & polynomial is odd
    const int b0 = __popc((2 * lane) & 79) & 1, b1 = __popc((2 * lane) & 109) & 1;
    const uint32_t selm = 0x4440u | (uint32_t)(b0 * 2 + b1);
    const uint32_t selx = (lane & 1) ? 0x4242u : 0x4040u;
    uint32_t y;
    if (mode == 0) y = 0;
    else if (start < 0) y = 31u * 0x10001u;                       // init_viterbi_unbiased (:189-201)
    else y = ((2 * lane == start) ? 0u : 63u) | ((2 * lane + 1 == start) ? 0u : 63u) << 16;      // init_viterbi (:170-187)
    const uint8_t* img = images + t.img;
    uint2* dec = decpool + t.dec;
    const int s0 = mode == 0 ? max(0, t.nsteps - kGuessSteps) : 0;
    for (int base = s0; base < t.nsteps; base += 32) {
        const int s = base + lane;
        uint32_t P = 0;
        if (s < t.nsteps) {
            const uint32_t sy = *reinterpret_cast<const unsigned short*>(img + 2 * s);
            const uint32_t a = sy & 0xFFu, b = sy >> 8;
            // (1 + (Branchtab0 ^ sym0) + (Branchtab1 ^ sym1)) >> 1 >> 2 for the four Branchtab combinations (:60-63)
            P = ((1u + a + b) >> 3) | ((1u + a + (255u ^ b)) >> 3) << 8 | ((1u + (255u ^ a) + b) >> 3) << 16 | ((1u + (255u ^ a) + (255u ^ b)) >> 3) << 24;
        }
        const int cnt = min(32, t.nsteps - base);
        uint32_t w0, w1;      // bit i of w0 / w1: decision of state 2 i / 2 i + 1; lane 0 stores them (the store pipe has room, the integer pipe has not)
        if (cnt == 32) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                y = acs_step(y, __shfl_sync(0xFFFFFFFFu, P, j), lane, selx, selm, w0, w1);
                if (lane == 0) dec[base + j] = make_uint2(w0, w1);
            }
        } else {
            for (int j = 0; j < cnt; ++j) {
                y = acs_step(y, __shfl_sync(0xFFFFFFFFu, P, j), lane, selx, selm, w0, w1);
                if (lane == 0) dec[base + j] = make_uint2(w0, w1);
            }
        }
    }
    __syncwarp();
    // find_endstate (:203-220): the first state with the smallest metric -- 0 after the renormalisation
    const uint32_t zero = __ballot_sync(0xFFFFFFFFu, (y & 0xFFFFu) == 0 || (y >> 16) == 0);
    const int L = __ffs(zero) - 1;
    const uint32_t yl = __shfl_sync(0xFFFFFFFFu, y, L);
    int state = 2 * L + ((yl & 0xFFFFu) == 0 ? 0 : 1);
    // chainback_viterbi (:242-283) with tailsize 6: bit n comes from the decisions of step n + 6
    if (mode == 0) {
        for (int n = t.fs - 1; n >= t.fs - 6; --n) {
            const uint2 w = dec[n + 6];
            const int k = (((state & 1) ? w.y : w.x) >> (state >> 1)) & 1;
            state = (state >> 1) | (k << 5);
        }
        if (lane == 0) res[warp].guess = state;
        return;
    }
    int retval = 0;
    uint8_t* out = decoded + t.out;
    // Traceback in 32 pieces, one per lane.  The lane of the top piece starts from the end state; every other lane starts
    // kWarm steps above its piece from state 0 -- tracebacks from different states run into the same path within a few
    // constraint lengths -- and the pieces are right if every lane arrived, at the top of its piece, at the state the lane
    // above ended in (then they are the sequential traceback, by induction from the top).  If one did not: the walk below.
    const int PL = ((t.fs + 31) / 32 + 15) & ~15;
    const int T = (t.fs - 1) / PL;
    const int seg_lo = lane * PL, seg_hi = min(seg_lo + PL, t.fs);
    const bool active = lane <= T;
    int st = state, warm_state = -1, retv = 0;
    auto back = [&](int m) {
        const uint2 w = dec[m + 6];
        const int k = (((st & 1) ? w.y : w.x) >> (st >> 1)) & 1;
        st = (st >> 1) | (k << 5);
        return (uint32_t)k;
    };
    if (active && lane < T) {
        const int nw = min(seg_hi - 1 + kWarm, t.fs - 1);
        st = nw == t.fs - 1 ? state : 0;
        for (int m = nw; m >= seg_hi; --m) back(m);
        warm_state = st;
    }
    if (active)
        for (int c = (seg_hi - 1) & ~15; c >= seg_lo; c -= 16) {
            uint32_t r[4] = {0, 0, 0, 0};
#pragma unroll
            for (int i = 15; i >= 0; --i)
                if (c + i < seg_hi) {
                    r[i >> 2] |= back(c + i) << (8 * (i & 3));
                    if (c + i == t.fs - 6) retv = st;
                }
            *reinterpret_cast<uint4*>(out + c) = make_uint4(r[0], r[1], r[2], r[3]);      // (the task's bits end on a 16-byte boundary of their own)
        }
    const int above = __shfl_down_sync(0xFFFFFFFFu, st, 1);
    const bool ok = !active || lane == T || warm_state == above;
    if (__all_sync(0xFFFFFFFFu, ok)) retval = __shfl_sync(0xFFFFFFFFu, retv, (t.fs - 6) / PL);
    else {
        for (int n0 = (t.fs - 1) & ~31; n0 >= 0; n0 -= 32) {
            const int n = n0 + lane;
            uint2 w = make_uint2(0, 0);
            if (n < t.fs) w = dec[n + 6];
            const int jtop = min(31, t.fs - 1 - n0);
            uint32_t mybit = 0;
            for (int j = jtop; j >= 0; --j) {
                const uint32_t wx = __shfl_sync(0xFFFFFFFFu, w.x, j), wy = __shfl_sync(0xFFFFFFFFu, w.y, j);
                const int k = (((state & 1) ? wy : wx) >> (state >> 1)) & 1;
                state = (state >> 1) | (k << 5);
                if (lane == j) mybit = k;
                if (n0 + j == t.fs - 6) retval = state;
            }
            if (n < t.fs) out[n] = (uint8_t)mybit;
        }
        if (lane == 0) atomicAdd(walks, 1);
    }
    if (lane == 0) {
        res[warp].retval = retval;
        res[warp].start_used = start;
        res[warp].need = 0;
    }
}

// a task started from the right state if that is where its predecessor's traceback ended
__global__ void mark_kernel(const VTask* __restrict__ tasks, VResult* __restrict__ res, int ntasks, int* __restrict__ flag) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ntasks) return;
    const int p = tasks[t].pred;
    if (p < 0) return;
    const int truth = res[p].retval;
    if (res[t].start_used != truth) {
        res[t].start_used = truth;
        res[t].need = 1;
        atomicAdd(flag, 1);
    }
}

// ---- CCEncoder::work + get_ber (cc_encoder.cpp:92-104, viterbi_all.cpp:60-73) per task -----------------------------------
__device__ __forceinline__ uint32_t enc_reg(const uint8_t* __restrict__ bits, int ii, uint32_t st6) {
    uint32_t reg = 0;
#pragma unroll
    for (int k = 0; k < 7; ++k) {
        const int i = ii - k;
        const uint32_t bit = i >= 0 ? (bits[i] & 1u) : ((st6 >> (-i - 1)) & 1u);
        reg |= bit << k;
    }
    return reg;
}
__device__ __forceinline__ uint32_t last6(const uint8_t* __restrict__ bits, int fs) {
    uint32_t v = 0;
    for (int k = 0; k < 6; ++k) v |= (bits[fs - 1 - k] & 1u) << k;
    return v;
}
__global__ void __launch_bounds__(128) ber_kernel(const VTask* __restrict__ tasks, VResult* __restrict__ res, int ntasks,
                                                  const uint8_t* __restrict__ images, const uint8_t* __restrict__ decoded) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= ntasks) return;
    const VTask t = tasks[warp];
    const uint8_t* bits = decoded + t.out;
    uint32_t st6 = (uint32_t)t.enc_state & 63u;
    if (t.enc_pred >= 0) st6 = last6(decoded + tasks[t.enc_pred].out, tasks[t.enc_pred].enc_fs);
    uint32_t stale = (uint32_t)t.stale_bit & 1u;
    if (t.stale_task >= 0) stale = __popc(enc_reg(decoded + tasks[t.stale_task].out, 1699, 0) & 79u) & 1u;
    const uint8_t* raw = images + t.img;
    int errors = 0, total = 0;
    for (int i = lane; i < t.ber_len; i += 32) {
        const uint32_t r = raw[i];
        if (r == 128u) continue;
        const int ii = i >> 1;
        uint32_t e = stale;
        if (ii < t.enc_fs) e = __popc(enc_reg(bits, ii, st6) & ((i & 1) ? 109u : 79u)) & 1u;
        errors += (int)((r > 127u) != (e != 0));
        total++;
    }
    errors = __reduce_add_sync(0xFFFFFFFFu, errors);
    total = __reduce_add_sync(0xFFFFFFFFu, total);
    if (lane == 0) {
        res[warp].errors = errors;
        res[warp].total = total;
        res[warp].enc_end = (int)last6(bits, t.enc_fs);
        res[warp].bit3398 = t.is78 ? (int)(__popc(enc_reg(bits, 1699, 0) & 79u) & 1u) : 0;
    }
}

// decoded bits of the accepted blocks -> the caller's stream
struct EmitDesc { uint32_t src; int n; long long dst; };
__global__ void __launch_bounds__(256) emit_kernel(const EmitDesc* __restrict__ d, const uint8_t* __restrict__ decoded, uint8_t* __restrict__ out) {
    const EmitDesc e = d[blockIdx.x];
    for (int i = threadIdx.x; i < e.n; i += 256) out[e.dst + i] = decoded[e.src + i];
}

// ---- DVBSymToSoftBlock::process ----------------------------------------------------------------------------------------
__device__ __forceinline__ int8_t sts_clamp(float x) {      // dvbs_syms_to_soft.cpp:8-14
    if (x < -127.0f) return -127;
    if (x > 127.0f) return 127;
    return (int8_t)x;
}
__global__ void __launch_bounds__(256) sts_kernel(const float* __restrict__ syms, int nsoft_in, const int8_t* __restrict__ carry, int fill, int nout,
                                                  int8_t* __restrict__ out, int8_t* __restrict__ carry_next) {
    const int total = fill + nsoft_in;
    for (int p = blockIdx.x * 256 + threadIdx.x; p < total; p += gridDim.x * 256) {
        const int8_t v = p < fill ? carry[p] : sts_clamp(syms[p - fill] * 100);
        if (p < nout) out[p] = v;
        else carry_next[p - nout] = v;
    }
}

void build_patterns(Pattern* P) {
    memset(P, 0, sizeof(Pattern) * kPatterns);
    auto fill = [](Pattern& p, int pin, std::initializer_list<std::pair<int, int>> slots) {      // (owner, erasure)
        p.pin = pin;
        p.pout = (int)slots.size();
        int i = 0;
        for (auto s : slots) { p.owner[i] = (int8_t)s.first; p.era[i] = (int8_t)s.second; ++i; }
        for (int a = 0; a <= pin; ++a) {
            int n = 0;
            while (n < p.pout && p.owner[n] < a) ++n;
            p.prefix[a] = (int8_t)n;
        }
    };
    fill(P[P23], 3, {{0, 0}, {1, 0}, {1, 1}, {2, 0}});                                                      // depunc.h:22-33
    fill(P[P56], 6, {{0, 0}, {1, 0}, {1, 1}, {2, 0}, {3, 0}, {3, 1}, {4, 1}, {4, 0}, {5, 0}, {5, 1}});      // depunc.h:105-133
    fill(P[P34 + 0], 4, {{0, 0}, {1, 0}, {2, 1}, {2, 0}, {3, 0}, {3, 1}});                                  // viterbi_all.h:93-113
    fill(P[P34 + 1], 4, {{0, 1}, {0, 0}, {1, 0}, {1, 1}, {2, 0}, {3, 0}});
    for (int sh = 0; sh < 4; ++sh) {                                                                        // viterbi_all.h:115-151
        Pattern& p = P[P78 + sh];
        p.pin = 8;
        int n = 0;
        for (int i = 0; i < 4; ++i) {
            const int a = 2 * i, b = 2 * i + 1;
            switch ((i + sh) % 4) {
            case 0: p.owner[n] = a; p.era[n++] = 0; p.owner[n] = b; p.era[n++] = 0; break;
            case 1: p.owner[n] = a; p.era[n++] = 1; p.owner[n] = a; p.era[n++] = 0; p.owner[n] = b; p.era[n++] = 1; p.owner[n] = b; p.era[n++] = 0; break;
            default: p.owner[n] = a; p.era[n++] = 1; p.owner[n] = a; p.era[n++] = 0; p.owner[n] = b; p.era[n++] = 0; p.owner[n] = b; p.era[n++] = 1; break;
            }
        }
        p.pout = n;
        for (int a = 0; a <= 8; ++a) {
            int m = 0;
            while (m < p.pout && p.owner[m] < a) ++m;
            p.prefix[a] = (int8_t)m;
        }
    }
}

struct DepuncState { int is_first = 0, changing_shift = 0, got_extra = 0, buf = 128; };

}  // namespace

struct dvbs2fec_dvbs_viterbi {
    int device = 0;
    cudaStream_t stream = nullptr;
    float thr = 0.15f, max_outsync = 20;
    // Viterbi_DVBS members (viterbi_all.h:43-54)
    int state = 0, rate = 0, phase = 0, shift = 0, invalid = 0;
    float ber = 10, bers[5][2][12];
    // what the ten decoders, five re-encoders and two depuncturers carry from call to call
    int dec_ber_start[5], dec_main_start[5], enc_state[5] = {0, 0, 0, 0, 0}, stale_bit = 0;
    DepuncState dp[5];
    int stale23[2] = {128, 128};
    DevBuf<int8_t> d_last_search;      // first 2048 soft bits of the last block the search ran on
    int have_last_search = 0;
    int search_batch = 1;
    int max_sync_blocks = kMaxSyncBlocks;      // DVBS2FEC_VIT_MAX_BATCH overrides (tests: batches cut inside a call)
    long long n_tasks = 0, n_repeated = 0, n_passes = 0;      // diagnostics: decode tasks run, tasks repeated from a corrected start, check passes
    Pattern pat[kPatterns];
    SearchLayout lay;
    int search_img_stride = 0, search_steps = 0, search_out = 0;
    // device pools
    DevBuf<int8_t> d_in;
    DevBuf<uint8_t> d_out, images, decoded;
    DevBuf<uint2> decpool;
    DevBuf<VTask> tasks;
    DevBuf<VResult> res;
    DevBuf<ContDesc> desc;
    DevBuf<ContRec> rec;
    DevBuf<EmitDesc> emit;
    DevBuf<int> flag;
    std::vector<VTask> h_tasks;
    std::vector<VResult> h_res;
    std::vector<ContDesc> h_desc;
    std::vector<ContRec> h_rec;
    std::vector<EmitDesc> h_emit;
    // DVBSymToSoftBlock
    DevBuf<int8_t> sts_carry[2];
    int sts_cur = 0, sts_fill = 0;
    DevBuf<float> d_syms;
    DevBuf<int8_t> d_soft;
    ~dvbs2fec_dvbs_viterbi() {
        cudaSetDevice(device);
        if (stream) {
            cudaStreamSynchronize(stream);
            cudaStreamDestroy(stream);
        }
    }
};

namespace {

using Vit = dvbs2fec_dvbs_viterbi;

// guess, decode, check (repeat what started wrong), BER; results to the host
int run_tasks(Vit* v, int ntasks) {
    cudaStream_t st = v->stream;
    CU(v->tasks.reserve((size_t)ntasks));
    CU(v->res.reserve((size_t)ntasks));
    CU(cudaMemcpyAsync(v->tasks.p, v->h_tasks.data(), sizeof(VTask) * ntasks, cudaMemcpyHostToDevice, st));
    const int grid = (ntasks + 3) / 4;
    acs_kernel<<<grid, 128, 0, st>>>(v->tasks.p, v->res.p, ntasks, 0, v->images.p, v->decpool.p, v->decoded.p, v->flag.p + 1);
    acs_kernel<<<grid, 128, 0, st>>>(v->tasks.p, v->res.p, ntasks, 1, v->images.p, v->decpool.p, v->decoded.p, v->flag.p + 1);
    v->h_res.resize(ntasks);
    v->n_tasks += ntasks;
    for (int pass = 0;; ++pass) {
        int flag = 0;
        CU(cudaMemsetAsync(v->flag.p, 0, sizeof(int), st));
        mark_kernel<<<(ntasks + 255) / 256, 256, 0, st>>>(v->tasks.p, v->res.p, ntasks, v->flag.p);
        ber_kernel<<<grid, 128, 0, st>>>(v->tasks.p, v->res.p, ntasks, v->images.p, v->decoded.p);
        CU(cudaMemcpyAsync(&flag, v->flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(v->h_res.data(), v->res.p, sizeof(VResult) * ntasks, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        v->n_passes++;
        if (!flag) break;
        v->n_repeated += flag;
        if (pass > ntasks) return fail(DVBS2FEC_ECUDA, "viterbi: start-state check does not settle");
        acs_kernel<<<grid, 128, 0, st>>>(v->tasks.p, v->res.p, ntasks, 2, v->images.p, v->decpool.p, v->decoded.p, v->flag.p + 1);
    }
    CU(cudaGetLastError());
    return 0;
}

// the lock search on n blocks, assuming none of them locks; returns how many blocks were consumed WITHOUT output (the block
// that takes the lock is not consumed: it is decoded next)
int run_search(Vit* v, const int8_t* d_in, int n, int* consumed) {
    cudaStream_t st = v->stream;
    const SearchLayout& L = v->lay;
    CU(v->images.reserve((size_t)n * v->search_img_stride));
    CU(v->decpool.reserve((size_t)n * v->search_steps));
    CU(v->decoded.reserve((size_t)n * v->search_out));
    search_image_kernel<<<n, 256, 0, st>>>(d_in, v->d_last_search.p, v->have_last_search, v->images.p, (uint32_t)v->search_img_stride);
    v->h_tasks.resize((size_t)n * kSearchTasks);
    int last_of_rate[5];      // task index of the latest candidate of each rate
    for (int r = 0; r < 5; ++r) last_of_rate[r] = -1;
    for (int b = 0; b < n; ++b) {
        uint32_t dec = (uint32_t)((size_t)b * v->search_steps), out = (uint32_t)((size_t)b * v->search_out);
        for (int phase = 0; phase < 2; ++phase)
            for (int c = 0; c < 26; ++c) {
                const int ti = b * kSearchTasks + phase * 26 + c, r = L.rate[c];
                VTask& t = v->h_tasks[ti];
                t.img = (uint32_t)((size_t)b * v->search_img_stride + phase * L.per_phase + L.img[c]);
                t.out = out;
                t.dec = dec;
                t.fs = kFsBer[r];
                t.nsteps = t.fs + 6;
                out += pad16(t.fs);
                dec += t.nsteps;
                t.pred = last_of_rate[r];
                t.start = v->dec_ber_start[r];
                t.enc_pred = last_of_rate[r];
                t.enc_state = v->enc_state[r];
                t.enc_fs = t.fs;
                t.ber_len = kBerLen[r];
                t.stale_task = r == R56 ? last_of_rate[R78] : -2;
                t.stale_bit = v->stale_bit;
                t.is78 = r == R78;
                last_of_rate[r] = ti;
            }
    }
    int rc = run_tasks(v, n * kSearchTasks);
    if (rc) return rc;
    int b = 0;
    bool locked = false;
    for (; b < n && !locked; ++b) {
        v->ber = 10;
        for (int phase = 0; phase < 2; ++phase)
            for (int c = 0; c < 26; ++c) {
                const int ti = b * kSearchTasks + phase * 26 + c, r = L.rate[c], sh = L.shift[c];
                const VResult& R = v->h_res[ti];
                const float ber = ((float)R.errors / (float)R.total) * kRatio[r];
                v->bers[r][phase][sh] = ber;
                v->dec_ber_start[r] = R.retval;
                v->enc_state[r] = R.enc_end;
                if (r == R78) v->stale_bit = R.bit3398;
                if (ber < v->thr) {      // every candidate under the threshold takes the lock; the last one keeps it (:94-105 ...)
                    v->ber = ber;
                    v->state = 1;
                    v->phase = phase;
                    v->shift = sh;
                    v->invalid = 0;
                    v->rate = r;
                    if (r == R23 || r == R56) { v->dp[r].changing_shift = sh; v->dp[r].is_first = sh > (r == R23 ? 2 : 5); }
                    v->stale23[0] = v->stale23[1] = 128;      // memset(depunc_buffer, 128)
                    locked = true;
                }
            }
    }
    // b blocks went through the search; the last of them is what ber_depunc_buffer now derives from
    CU(cudaMemcpyAsync(v->d_last_search.p, d_in + (size_t)(b - 1) * kBuf, kTest, cudaMemcpyDeviceToDevice, st));
    v->have_last_search = 1;
    *consumed = locked ? b - 1 : b;
    return 0;
}

// decode n blocks at the lock, assuming it holds; *accepted = blocks whose result stands (the lock may be given up after one)
int run_sync(Vit* v, const int8_t* d_in, int n, uint8_t* d_out, long long* oidx, int* accepted) {
    cudaStream_t st = v->stream;
    const int r = v->rate, fs = kFsMain[r], nsteps = fs + 6, nread = 2 * nsteps, stride = pad16(nread), ostride = pad16(fs);
    CU(v->images.reserve((size_t)n * stride));
    CU(v->decpool.reserve((size_t)n * nsteps));
    CU(v->decoded.reserve((size_t)n * ostride));
    const bool cont = r == R23 || r == R56;
    std::vector<DepuncState> after(n);
    std::vector<int> szs(n, kBuf);
    v->h_desc.assign(n, ContDesc{0, 0, 0, {-1, -1}});
    if (cont) {      // Depunc23 / Depunc56 ::depunc_cont (depunc.h:43-76,143-186): the bookkeeping, block by block
        DepuncState d = v->dp[r];
        const Pattern& P = v->pat[r == R23 ? P23 : P56];
        int writer[2] = {-1, -1};
        for (int k = 0; k < n; ++k) {
            ContDesc& D = v->h_desc[k];
            D.lead = d.is_first || d.got_extra;
            d.is_first = d.got_extra = 0;
            D.c = d.changing_shift % P.pin;
            D.oo = D.lead + pat_count(P, D.c, kBuf);
            d.changing_shift = D.c + kBuf;
            for (int i = 0; i < 2; ++i) {
                if (D.oo > 10922 + i) writer[i] = k;
                D.stale_src[i] = writer[i];
            }
            szs[k] = D.oo;
            if (D.oo % 2 == 1) { szs[k] = D.oo - 1; d.got_extra = 1; }
            after[k] = d;
        }
        CU(v->desc.reserve((size_t)n));
        CU(v->rec.reserve((size_t)n));
        CU(cudaMemcpyAsync(v->desc.p, v->h_desc.data(), sizeof(ContDesc) * n, cudaMemcpyHostToDevice, st));
    } else if (r == R34) std::fill(szs.begin(), szs.end(), kBuf / 2 * 3);
    else if (r == R78) std::fill(szs.begin(), szs.end(), kBuf / 8 * 14);
    sync_image_kernel<<<dim3(n, 8), 256, 0, st>>>(d_in, r, v->phase, v->shift, nread, cont ? v->desc.p : nullptr, cont ? v->rec.p : nullptr, v->dp[r].buf,
                                                   v->stale23[0], v->stale23[1], v->images.p, (uint32_t)stride);
    v->h_tasks.resize(n);
    for (int k = 0; k < n; ++k) {
        VTask& t = v->h_tasks[k];
        t.img = (uint32_t)((size_t)k * stride);
        t.out = (uint32_t)((size_t)k * ostride);
        t.dec = (uint32_t)((size_t)k * nsteps);
        t.fs = fs;
        t.nsteps = nsteps;
        t.pred = k - 1;
        t.start = v->dec_main_start[r];
        t.enc_pred = k - 1;
        t.enc_state = v->enc_state[r];
        t.enc_fs = kFsBer[r];
        t.ber_len = kBerLen[r];
        t.stale_task = -2;
        t.stale_bit = v->stale_bit;
        t.is78 = r == R78;
    }
    int rc = run_tasks(v, n);
    if (rc) return rc;
    if (cont) {
        v->h_rec.resize(n);
        CU(cudaMemcpyAsync(v->h_rec.data(), v->rec.p, sizeof(ContRec) * n, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    v->h_emit.clear();
    int k = 0;
    for (; k < n && v->state == 1; ++k) {
        const VResult& R = v->h_res[k];
        v->ber = ((float)R.errors / (float)R.total) * kRatio[r];
        v->dec_main_start[r] = R.retval;
        v->enc_state[r] = R.enc_end;
        if (r == R78) v->stale_bit = R.bit3398;
        if (cont) {
            const int held = v->dp[r].buf;
            v->dp[r] = after[k];
            v->dp[r].buf = szs[k] != v->h_desc[k].oo ? v->h_rec[k].buf_val : held;      // an odd count: the last byte waits for the next call
            if (r == R23) { v->stale23[0] = v->h_rec[k].v[0]; v->stale23[1] = v->h_rec[k].v[1]; }
        }
        const int out_n = szs[k] / 2;
        v->h_emit.push_back(EmitDesc{v->h_tasks[k].out, std::min(fs, out_n), *oidx});      // the decoder writes its frame size; what lies
        *oidx += out_n;                                                                     // behind out_n the next block overwrites
        if (v->ber > v->thr) {      // :268-277
            v->invalid++;
            if ((float)v->invalid > v->max_outsync) v->state = 0;
        } else
            v->invalid = 0;
    }
    *accepted = k;
    if (k) {
        CU(v->emit.reserve((size_t)k));
        CU(cudaMemcpyAsync(v->emit.p, v->h_emit.data(), sizeof(EmitDesc) * k, cudaMemcpyHostToDevice, st));
        emit_kernel<<<k, 256, 0, st>>>(v->emit.p, v->decoded.p, d_out);
        CU(cudaStreamSynchronize(st));      // h_emit is reused by the next batch
    }
    CU(cudaGetLastError());
    return 0;
}

}  // namespace

extern "C" {

int dvbs2fec_dvbs_viterbi_reset(dvbs2fec_dvbs_viterbi* v) {
    if (!v) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    CU(cudaSetDevice(v->device));
    v->state = v->rate = v->phase = v->shift = v->invalid = 0;
    v->ber = 10;
    for (int r = 0; r < 5; ++r) {
        v->dec_ber_start[r] = v->dec_main_start[r] = -1;
        v->enc_state[r] = 0;
        v->dp[r] = DepuncState();
        for (int p = 0; p < 2; ++p)
            for (int s = 0; s < 12; ++s) v->bers[r][p][s] = 10;
    }
    v->stale_bit = 0;
    v->stale23[0] = v->stale23[1] = 128;
    v->have_last_search = 0;
    v->search_batch = 1;
    v->sts_fill = 0;
    return 0;
}

int dvbs2fec_dvbs_viterbi_create(int device, float ber_threshold, int max_outsync, dvbs2fec_dvbs_viterbi** out) {
    if (!out) return fail(DVBS2FEC_EINVAL, "out is NULL");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(DVBS2FEC_ENODEV, "no CUDA device");
    if (device < 0 || device >= ndev) return fail(DVBS2FEC_EINVAL, "device out of range");
    std::unique_ptr<Vit> v(new Vit());
    v->device = device;
    v->thr = ber_threshold;
    v->max_outsync = (float)max_outsync;
    if (const char* e = getenv("DVBS2FEC_VIT_MAX_BATCH")) v->max_sync_blocks = std::max(1, std::min(atoi(e), kMaxSyncBlocks));
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&v->stream, cudaStreamNonBlocking));
    build_patterns(v->pat);
    CU(cudaMemcpyToSymbol(cPat, v->pat, sizeof(Pattern) * kPatterns));
    // the 26 candidates of one phase in the order the reference tries them
    SearchLayout& L = v->lay;
    int c = 0, off = 0, steps = 0, outb = 0;
    for (int r = 0; r < 5; ++r)
        for (int s = 0; s < kShifts[r]; ++s, ++c) {
            L.rate[c] = r;
            L.shift[c] = s;
            L.nread[c] = 2 * (kFsBer[r] + 6);
            L.img[c] = off;
            off += pad16(L.nread[c]);
            steps += kFsBer[r] + 6;
            outb += pad16(kFsBer[r]);
        }
    L.per_phase = off;
    v->search_img_stride = 2 * off;
    v->search_steps = 2 * steps;
    v->search_out = 2 * outb;
    CU(cudaMemcpyToSymbol(cSearch, &L, sizeof L));
    CU(v->d_last_search.reserve(kTest));
    CU(v->flag.reserve(2));
    CU(cudaMemset(v->flag.p, 0, 2 * sizeof(int)));      // [0] tasks that started wrong in this pass, [1] tracebacks that fell back to the walk
    CU(cudaDeviceSynchronize());
    CU(v->sts_carry[0].reserve(kBuf));
    CU(v->sts_carry[1].reserve(kBuf));
    int rc = dvbs2fec_dvbs_viterbi_reset(v.get());
    if (rc) return rc;
    *out = v.release();
    return 0;
}

void dvbs2fec_dvbs_viterbi_destroy(dvbs2fec_dvbs_viterbi* v) { delete v; }

int dvbs2fec_dvbs_viterbi_process_device(dvbs2fec_dvbs_viterbi* v, int count, const int8_t* d_in, uint8_t* d_out) {
    if (!v || count < 0 || (count && (!d_in || !d_out))) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (count % kBuf) return fail(DVBS2FEC_EINVAL, "count must be a multiple of 8192 soft bits (VIT_BUF_SIZE)");
    CU(cudaSetDevice(v->device));
    const int nb = count / kBuf;
    int pos = 0;
    long long oidx = 0;
    while (pos < nb) {
        if (v->state == 0) {
            const int n = std::min({nb - pos, v->search_batch, kMaxSearchBlocks});
            int consumed = 0;
            int rc = run_search(v, d_in + (size_t)pos * kBuf, n, &consumed);
            if (rc) return rc;
            pos += consumed;
            v->search_batch = v->state == 1 ? 1 : std::min(v->search_batch * 4, kMaxSearchBlocks);
        }
        if (v->state == 1 && pos < nb) {
            const int n = std::min(nb - pos, v->max_sync_blocks);
            int accepted = 0;
            int rc = run_sync(v, d_in + (size_t)pos * kBuf, n, d_out, &oidx, &accepted);
            if (rc) return rc;
            pos += accepted;
        }
    }
    if (oidx > 0x7FFFFFFF) return fail(DVBS2FEC_EINVAL, "more than 2^31 - 1 output bits in one call");
    return (int)oidx;
}

int dvbs2fec_dvbs_viterbi_process(dvbs2fec_dvbs_viterbi* v, int count, const int8_t* in, uint8_t* out) {
    if (!v || count < 0 || (count && (!in || !out))) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (count % kBuf) return fail(DVBS2FEC_EINVAL, "count must be a multiple of 8192 soft bits (VIT_BUF_SIZE)");
    if (!count) return 0;
    CU(cudaSetDevice(v->device));
    CU(v->d_in.reserve((size_t)count));
    CU(v->d_out.reserve((size_t)count));
    CU(cudaMemcpyAsync(v->d_in.p, in, (size_t)count, cudaMemcpyHostToDevice, v->stream));
    // the bytes the reference leaves unwritten (rate 5/6) keep what the caller's buffer holds
    CU(cudaMemcpyAsync(v->d_out.p, out, (size_t)count, cudaMemcpyHostToDevice, v->stream));
    const int n = dvbs2fec_dvbs_viterbi_process_device(v, count, v->d_in.p, v->d_out.p);
    if (n <= 0) return n;
    CU(cudaMemcpyAsync(out, v->d_out.p, (size_t)n, cudaMemcpyDeviceToHost, v->stream));
    CU(cudaStreamSynchronize(v->stream));
    return n;
}

int dvbs2fec_dvbs_viterbi_stats(dvbs2fec_dvbs_viterbi* v, float* ber, int* state, int* rate, int* phase, int* shift, int* invalid) {
    if (!v) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    float b = v->ber;
    if (v->state != 1) {      // Viterbi_DVBS::ber (:282-313): the best candidate of the last search
        b = 10;
        for (int r = 0; r < 5; ++r)
            for (int p = 0; p < 2; ++p)
                for (int s = 0; s < kShifts[r]; ++s)
                    if (b > v->bers[r][p][s]) b = v->bers[r][p][s];
    }
    if (ber) *ber = b;
    if (state) *state = v->state;
    if (rate) *rate = v->rate;
    if (phase) *phase = v->phase;
    if (shift) *shift = v->shift;
    if (invalid) *invalid = v->invalid;
    return 0;
}

int dvbs2fec_dvbs_viterbi_counters(dvbs2fec_dvbs_viterbi* v, long long* tasks, long long* repeated, long long* passes, long long* walks) {
    if (!v) return fail(DVBS2FEC_EINVAL, "handle is NULL");
    if (walks) {
        int w = 0;
        CU(cudaSetDevice(v->device));
        CU(cudaMemcpy(&w, v->flag.p + 1, sizeof(int), cudaMemcpyDeviceToHost));
        *walks = w;
    }
    if (tasks) *tasks = v->n_tasks;
    if (repeated) *repeated = v->n_repeated;
    if (passes) *passes = v->n_passes;
    return 0;
}

int dvbs2fec_dvbs_sts_process_device(dvbs2fec_dvbs_viterbi* v, int count, const float* d_syms, int8_t* d_out) {
    if (!v || count < 0 || (count && (!d_syms || !d_out))) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (!count) return 0;
    CU(cudaSetDevice(v->device));
    const int total = v->sts_fill + 2 * count, nout = total / kBuf * kBuf;
    sts_kernel<<<std::min((total + 255) / 256, 1184), 256, 0, v->stream>>>(d_syms, 2 * count, v->sts_carry[v->sts_cur].p, v->sts_fill, nout, d_out,
                                                                            v->sts_carry[v->sts_cur ^ 1].p);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(v->stream));
    v->sts_cur ^= 1;
    v->sts_fill = total - nout;
    return nout;
}

int dvbs2fec_dvbs_sts_process(dvbs2fec_dvbs_viterbi* v, int count, const float* syms, int8_t* out) {
    if (!v || count < 0 || (count && (!syms || !out))) return fail(DVBS2FEC_EINVAL, "bad arguments");
    if (!count) return 0;
    CU(cudaSetDevice(v->device));
    CU(v->d_syms.reserve((size_t)2 * count));
    CU(v->d_soft.reserve((size_t)2 * count + kBuf));
    CU(cudaMemcpyAsync(v->d_syms.p, syms, sizeof(float) * 2 * count, cudaMemcpyHostToDevice, v->stream));
    const int n = dvbs2fec_dvbs_sts_process_device(v, count, v->d_syms.p, v->d_soft.p);
    if (n <= 0) return n;
    CU(cudaMemcpyAsync(out, v->d_soft.p, (size_t)n, cudaMemcpyDeviceToHost, v->stream));
    CU(cudaStreamSynchronize(v->stream));
    return n;
}

}  // extern "C"
