// K2, second generation: the LDPC layered offset-min-sum kernel rebuilt around the measured issue rates of sm_100a
// (profiles/r02_onchip_peaks.json: every integer/SIMD instruction shares the ALU pipe at 2 warp-instructions per
// clock per SM; IMAD/HFMA2 run beside it on the FMA pipe at another 2).  Same decomposition as the first kernel --
// a CTA owns a PAIR of frames (frame A in the low, frame B in the high 16-bit lane of every register), thread j
// owns row j of every layer, dependency levels keep the reference's sequential row order -- but the row update is
// written for the ALU pipe budget (about 15 ALU-pipe instructions per edge pair instead of 29) and everything
// around it is reorganised:
//
//   * messages are stored as beta = 32 - m (1..64, a non-negative byte), so that "LLR - message" is a carry-free
//     32-bit add on the FMA pipe followed by one VIADDMNMX.RELU (subtract 32, clamp to the int8 range), and the new
//     message leaves the sign step already in that form (no two's-complement negations anywhere);
//   * the conditional negation by the outgoing sign is  (om ^ mask) + [negative]  with the [negative] bit taken from
//     the mask by one multiplication (mask * 0xFFFEFFFF, FMA pipe), folded with the +32 bias of the message;
//   * exclusive minima come from alternating prefix/suffix minima combined with three-input VIMNMX3 (2D - 2
//     instructions for D links instead of 3D - 6);
//   * link addresses are  min(x, x - 720)  in unsigned arithmetic (one VIADDMNMX.U32) instead of compare/select;
//   * there is no "one frame finished" code path: a frame's results are written out the moment it stops and its
//     lane simply keeps computing until the pair is done;
//   * column j of the q x 360 parity matrix is CONTIGUOUS in the input frame (v[K + q j + i],
//     layered_decoder.hh:124-126) and thread j is its only consumer; the pair load transposes it once, with
//     coalesced loads and stores, into the workspace words every pass reads (layer-major, one word per row);
//   * the next pair is claimed when the first frame of the current one stops, and its frames are prefetched into L2;
//   * LDPCDecoder::bad is screened: after every pass thread j tests row (q-1, j), whose parity LLRs it still holds
//     in registers; only when all 360 rows of that layer pass for a live frame does the full bit-plane test run.
//     Any bad row makes bad() true (layered_decoder.hh:28-45), so the screen never changes a result.
//
// Reference semantics (SURVEY.md spec S-LDPC): layered_decoder.hh:23-74,121-133; algorithms.hh:235-256,261-276;
// generic.hh:15-18; bbframe_ldpc.cpp:123-139.  Included by the instantiation units ldpc2_inst_*.cu only.
#pragma once
#include "ldpc_decoder.cuh"
#include "ldpc_variants.h"

#include <type_traits>

namespace s2 {
namespace v2 {

// One thread per row and none to spare: 360 threads = eleven warps and a quarter.  (With 384 threads the 24 extra
// ones either need a "row exists" predicate everywhere or shadow row 359, which racecheck rightly flags.)
constexpr int kThreads = 360;

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}
__device__ __forceinline__ uint32_t minu2(uint32_t a, uint32_t b) {
    uint32_t d;
    asm("min.u16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
}
__device__ __forceinline__ uint32_t min3u2(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("{.reg .b32 t; min.u16x2 t, %1, %2; min.u16x2 %0, t, %3;}" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
// (a + b) per 16-bit lane, then min with c, then max with 0: one VIADDMNMX.S16x2.RELU
__device__ __forceinline__ uint32_t addmin_relu(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("{.reg .b32 t; add.s16x2 t, %1, %2; min.s16x2.relu %0, t, %3;}" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t addmin(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("{.reg .b32 t; add.s16x2 t, %1, %2; min.s16x2 %0, t, %3;}" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
// min(x + c, x) in unsigned arithmetic: one VIADDMNMX.U32
__device__ __forceinline__ uint32_t addmin_u32(uint32_t x, uint32_t c) {
    uint32_t d;
    asm("{.reg .b32 t; add.u32 t, %1, %2; min.u32 %0, t, %1;}" : "=r"(d) : "r"(x), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) {
    uint16_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_u16(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"((uint16_t)v));
}

// two packed bytes [A, B] (low half of w) -> zero-extended 16-bit lanes, and back
__device__ __forceinline__ uint32_t unpack_lo(uint32_t w) { return prmt(w, 0, 0x4140); }
__device__ __forceinline__ uint32_t unpack_hi(uint32_t w) { return prmt(w, 0, 0x4342); }
__device__ __forceinline__ uint32_t pack_pair(uint32_t x) { return prmt(x, 0, 0x4420); }
__device__ __forceinline__ uint32_t pack_two(uint32_t x0, uint32_t x1) { return prmt(x0, x1, 0x6420); }
// 0xFFFF in every lane whose low byte has bit 7 set
__device__ __forceinline__ uint32_t lane_mask7(uint32_t x) { return prmt(x, 0, 0xAA88); }

constexpr uint32_t kC128 = 0x00800080u, kC255 = 0x00FF00FFu, kM32 = 0xFFE0FFE0u, kP32 = 0x00200020u;
constexpr uint32_t kP63 = 0x003F003Fu, kP64 = 0x00400040u, kAllOnes = 0xFFFFFFFFu;

// ex[k] = min over all a[c], c != k  (per 16-bit lane), in 2D - 2 VIMNMX(3) instructions.
// P[i] = min(a[0..i]) is kept for odd i, S[i] = min(a[i..D-1]) for even i (D odd: S[D-1] = a[D-1]; D even:
// S[D-2] = min(a[D-2], a[D-1])); every ex[k] is then one instruction over at most three terms.
template <int D>
__device__ __forceinline__ void exclusive_min(const uint32_t (&a)[D], uint32_t (&ex)[D]) {
    static_assert(D >= 3, "a check has at least three links");
    uint32_t P[D], S[D + 2];
#pragma unroll
    for (int i = 1; i < D; i += 2) P[i] = (i == 1) ? minu2(a[0], a[1]) : min3u2(P[i - 2], a[i - 1], a[i]);
    constexpr int top = (D & 1) ? D - 1 : D - 2;
    S[top] = (D & 1) ? a[D - 1] : minu2(a[D - 2], a[D - 1]);
#pragma unroll
    for (int i = top - 2; i >= 0; i -= 2) S[i] = min3u2(a[i], a[i + 1], S[i + 2]);
#pragma unroll
    for (int k = 0; k < D; ++k) {
        uint32_t t[4];
        int n = 0;
        if (k & 1) {                       // left = a[0..k-1], k - 1 even
            if (k >= 3) t[n++] = P[k - 2];
            t[n++] = a[k - 1];
        } else if (k >= 2) {
            t[n++] = P[k - 1];
        }
        if (k + 1 <= D - 1) {              // right = a[k+1..D-1]
            if (((k + 1) & 1) == 0 && k + 1 <= top) {
                t[n++] = S[k + 1];
            } else {
                t[n++] = a[k + 1];
                if (k + 2 <= top) t[n++] = S[k + 2];
            }
        }
        ex[k] = (n == 1) ? t[0] : (n == 2) ? minu2(t[0], t[1]) : min3u2(t[0], t[1], t[2]);
    }
}

// One check row for both frames of the pair (all quantities per 16-bit lane; LLRs are offset binary u = llr + 128).
//   off[]  : shared-memory addresses of the row's data-link LLR pairs
//   mw[]   : the row's message bytes beta = 32 - m, two slots (of two frames) per word; slot c < CNT = data link c,
//            slot CNT = own parity bit, slot CNT + 1 = second parity bit                        (in/out)
//   pown, psec : the two parity LLRs, unpacked                                                  (in/out)
// FIRST : first pass, all messages are zero (layered_decoder.hh:23-27) and mw[] is write-only.
// RAGGED: only the first cnt data links exist in this layer; the others act as a link whose LLR is +127 with no
//         write-back: |t| >= 96 never decides a minimum that the clamp to 32 lets through and its sign is +.
//         The missing second parity link of row (0,0) is the same thing (the caller passes psec = 255).
// Maths per link (algorithms.hh:235-256,273-276; layered_decoder.hh:55-70):
//   t = sat8(llr - m)            tu = clamp(u + beta - 32, 0, 255)
//   a = |t|                      (the reference's max(|max(t,-127)|-1, 0) is monotone in a, applied after the minimum)
//   ex = min of a over the other links;  om = clamp(ex - 1, 0, 32)
//   m' = -om if an odd number of the other t is negative, else min(om, 31);  llr' = sat8(t + m')
// keep: word whose upper half is stored in the upper half of the last message word when the number of slots is odd
//       (the record's spare bytes; the caller keeps the row level there).
// m1  : 0xFFFFFFFF in a register the compiler cannot see through, so that 64 - bm is issued as a multiply-add on
//       the FMA pipe (as a subtraction ptxas puts it on the ALU pipe, which is the one this kernel saturates).
template <int CNT, bool FIRST, bool RAGGED>
__device__ __forceinline__ void row_update(const uint32_t (&off)[CNT], int cnt, uint32_t (&mw)[(CNT + 3) / 2],
                                           uint32_t& pown, uint32_t& psec, uint32_t keep, uint32_t m1) {
    constexpr int D = CNT + 2;
    uint32_t tu[D], a[D], ex[D];
    // bit 7 of tu is set for t >= 0.  The product of the OTHER signs of link k is negative iff
    // bit7(sx ^ tu_k) ^ ((D - 1) & 1), sx = XOR of all tu; the constant is folded into the start value.
    uint32_t sx = ((D - 1) & 1) ? kC128 : 0u;
#pragma unroll
    for (int c = 0; c < D; ++c) {
        uint32_t u;
        if (c < CNT)
            u = (!RAGGED || c < cnt) ? unpack_lo(lds_u16(off[c])) : kC255;
        else
            u = (c == CNT) ? pown : psec;
        uint32_t t = u;
        if (!FIRST) {
            const uint32_t beta = (c & 1) ? unpack_hi(mw[c >> 1]) : unpack_lo(mw[c >> 1]);
            t = addmin_relu(u + beta, kM32, kC255);
        }
        tu[c] = t;
        a[c] = __vabsdiffu4(t, kC128);
        sx ^= t;
    }
    exclusive_min<D>(a, ex);
    const uint32_t ssx = lane_mask7(sx);
    uint32_t prev = 0;
#pragma unroll
    for (int c = 0; c < D; ++c) {
        const uint32_t om = addmin_relu(ex[c], kAllOnes, kP32);        // clamp(ex - 1, 0, 32)
        const uint32_t neg = lane_mask7(tu[c]) ^ ssx;                  // 0xFFFF: outgoing sign is -
        const uint32_t bias = neg * 0xFFFEFFFFu + kP32;                // 32 + [neg] per lane (0xFFFF * 0xFFFEFFFF = 1)
        const uint32_t bm = addmin(om ^ neg, bias, kP63);              // m' + 32 = 32 - om | min(32 + om, 63)
        const uint32_t un = addmin_relu(tu[c] + bm, kM32, kC255);      // llr' = sat8(t + m')
        uint32_t beta;                                                 // 32 - m' = 64 - bm
        asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(beta) : "r"(bm), "r"(m1), "r"(kP64));
        if (c < CNT) {
            if (!RAGGED || c < cnt) sts_u16(off[c], pack_pair(un));
        } else if (c == CNT) {
            pown = un;
        } else {
            psec = un;
        }
        if (c & 1)
            mw[c >> 1] = pack_two(prev, beta);
        else if (c == D - 1)
            mw[c >> 1] = prmt(beta, keep, 0x7620);      // beta.A, beta.B, keep.byte2, keep.byte3
        prev = beta;
    }
}

// ---- the termination test on bit planes (full form; see the screen in the kernel) -----------------------------

// bits [o, o+32) of the 360-periodic extension of a 360-bit vector stored in 12 words (+1 zero word)
// (the planes live in the CTA's workspace in global memory: L2-coherent accesses)
__device__ __forceinline__ uint32_t win360(const uint32_t* H, int o) {
    int w = o >> 5, s = o & 31;
    uint32_t r = __funnelshift_r(__ldcg(H + w), __ldcg(H + w + 1), s);
    int over = o + 32 - 360;
    if (over > 0) r |= __ldcg(H) << (32 - over);
    return r;
}
// Hard decisions + zero test of 8 consecutive offset-binary LLR pairs (one uint4: A0 B0 A1 B1 ...).
// Returns bits 0-7 = "A_k negative", bits 8-15 = "B_k negative"; clears bit 7 of byte f (and f + 2) of nzacc
// for every zero LLR of frame f.
__device__ __forceinline__ uint32_t harvest8(uint4 w, uint32_t& nzacc) {
    const uint32_t k80 = 0x80808080u;
    nzacc &= __vabsdiffu4(w.x, k80) + 0x7F7F7F7Fu;
    nzacc &= __vabsdiffu4(w.y, k80) + 0x7F7F7F7Fu;
    nzacc &= __vabsdiffu4(w.z, k80) + 0x7F7F7F7Fu;
    nzacc &= __vabsdiffu4(w.w, k80) + 0x7F7F7F7Fu;
    uint32_t a0 = prmt(w.x, w.y, 0x6420), b0 = prmt(w.x, w.y, 0x7531);
    uint32_t a1 = prmt(w.z, w.w, 0x6420), b1 = prmt(w.z, w.w, 0x7531);
    auto mask4 = [](uint32_t x) { return (((~x & 0x80808080u) >> 7) * 0x00204081u >> 21) & 0xFu; };
    return mask4(a0) | (mask4(a1) << 4) | (mask4(b0) << 8) | (mask4(b1) << 12);
}
// bit planes of n360 groups of 360 LLR pairs starting at src: plane A at H[g*13 words], plane B at
// H[(gstride + g)*13 words], byte k of a group = bits 8k..8k+7
template <bool GLOBAL, int THREADS>
__device__ __forceinline__ void harvest_planes(const uint4* src, int n360, uint32_t* H, int gstride, int tid,
                                               uint32_t& nzacc) {
    uint8_t* Hb = reinterpret_cast<uint8_t*>(H);
    for (int t = tid; t < n360 * 45; t += THREADS) {
        uint4 w = GLOBAL ? __ldcg(src + t) : src[t];
        uint32_t bits = harvest8(w, nzacc);
        int g = t / 45, k = t - g * 45;
        __stcg(&Hb[g * (kBitWords * 4) + k], (uint8_t)bits);
        __stcg(&Hb[(gstride + g) * (kBitWords * 4) + k], (uint8_t)(bits >> 8));
    }
}

// The full LDPCDecoder::bad (layered_decoder.hh:28-45) for both frames of the pair: a row is bad when its sign product
// is not positive, i.e. odd parity of hard decisions or any zero LLR.  Hard decisions are gathered into bit planes
// (parity part from the workspace, where load_pair staged it before the first pass), each layer's 360 checks are then
// 12 words of rotate-and-XOR.  Returns bit f set when frame f is bad.  All threads of the CTA call it.
template <int THREADS>
__device__ __noinline__ int full_test(const LdpcParams2& p, const uint16_t* wpty, uint32_t* HP, uint32_t* HD,
                                      const uint4* vdata4, int* s_bad) {
    const int tid = threadIdx.x, q = p.q;
    uint32_t nzacc = 0xFFFFFFFFu;
    harvest_planes<true, THREADS>(reinterpret_cast<const uint4*>(wpty), q, HP, q, tid, nzacc);
    harvest_planes<false, THREADS>(vdata4, p.ngroups, HD, p.ngroups, tid, nzacc);
    if (tid < 2) s_bad[tid] = 0;
    __syncthreads();
    if (~nzacc & 0x00800080u) atomicOr(&s_bad[0], 1);
    if (~nzacc & 0x80008000u) atomicOr(&s_bad[1], 1);
    for (int task = tid; task < q * 12; task += THREADS) {
        const int ii = task / 12, w = task - ii * 12;
        const int loff = p.layer_off[ii], cnt = (int)p.layer_off[ii + 1] - loff;
        uint32_t sA = __ldcg(&HP[ii * kBitWords + w]), sB = __ldcg(&HP[(q + ii) * kBitWords + w]);
        if (ii > 0) {
            sA ^= __ldcg(&HP[(ii - 1) * kBitWords + w]);
            sB ^= __ldcg(&HP[(q + ii - 1) * kBitWords + w]);
        } else {  // row (0,j) uses pty[q-1][j-1], row (0,0) has no second parity link
            const uint32_t* ta = &HP[(q - 1) * kBitWords];
            const uint32_t* tb = &HP[(2 * q - 1) * kBitWords];
            sA ^= (__ldcg(ta + w) << 1) | (w ? __ldcg(ta + w - 1) >> 31 : 0u);
            sB ^= (__ldcg(tb + w) << 1) | (w ? __ldcg(tb + w - 1) >> 31 : 0u);
        }
        for (int c = 0; c < cnt; ++c) {
            // bit (32 w + b) of the row vector is data bit (32 w + b - shift) mod 360 of the group
            int o = 32 * w + (int)(p.link_add[loff + c] >> 1) - 360;   // (720 - 2 shift) / 2 - 360 = -shift
            o += (o < 0) ? 360 : 0;
            const int g = p.link_group[loff + c];
            sA ^= win360(&HD[g * kBitWords], o);
            sB ^= win360(&HD[(p.ngroups + g) * kBitWords], o);
        }
        if (w == 11) {
            sA &= 0xFFu;
            sB &= 0xFFu;
        }
        if (sA) atomicOr(&s_bad[0], 1);
        if (sB) atomicOr(&s_bad[1], 1);
    }
    __syncthreads();
    return (s_bad[0] ? 1 : 0) | (s_bad[1] ? 2 : 0);
}

// Results of the frames that stop here (bit f of fin): iteration count, MSB-first hard decisions of the K systematic
// bits (module_dvbs2_demod.cpp:357-360) straight from the LLR pairs (8 pairs = one uint4 give one byte of each frame),
// optionally the posterior LLRs (what BBFrameLDPC::decode leaves in place; before the first pass the staged input).
template <int THREADS>
__device__ __noinline__ void emit_results(const LdpcParams2& p, int fin, const int (&res)[2], int fa, int fb,
                                          const uint16_t* wpty, const uint4* vdata4) {
    const int tid = threadIdx.x, q = p.q, K = p.K, N = p.N, R = p.R;
    const int kbytes = K / 8;
    for (int b = tid; b < kbytes; b += THREADS) {
        uint32_t nz = 0xFFFFFFFFu;
        const uint32_t bits = harvest8(vdata4[b], nz);
        if (fin & 1) p.hard_out[(size_t)fa * p.hard_stride + b] = (uint8_t)(__brev(bits & 0xFFu) >> 24);
        if (fin & 2) p.hard_out[(size_t)fb * p.hard_stride + b] = (uint8_t)(__brev((bits >> 8) & 0xFFu) >> 24);
    }
    for (int f = 0; f < 2; ++f) {
        if (!(fin >> f & 1)) continue;
        const int fr = f ? fb : fa;
        if (tid == 0) p.iters_out[fr] = (int16_t)res[f];
        if (p.llr_out) {
            int8_t* lo = p.llr_out + (size_t)fr * N;
            const uint8_t* vb = reinterpret_cast<const uint8_t*>(vdata4) + f;
            for (int x = tid; x < K; x += THREADS) lo[x] = (int8_t)(vb[2 * x] ^ 0x80u);
            for (int x = tid; x < R; x += THREADS) {
                const int jj = x / q, ii = x - jj * q;
                lo[K + x] = (int8_t)((__ldcg(&wpty[360 * ii + jj]) >> (8 * f)) ^ 0x80u);
            }
        }
    }
}

// 8 LLRs of frame A and the same 8 of frame B -> 8 LLR pairs in offset binary (A in the even bytes)
__device__ __forceinline__ uint4 interleave8(uint2 a, uint2 b) {
    uint4 o;
    o.x = prmt(a.x, b.x, 0x5140) ^ 0x80808080u;
    o.y = prmt(a.x, b.x, 0x7362) ^ 0x80808080u;
    o.z = prmt(a.y, b.y, 0x5140) ^ 0x80808080u;
    o.w = prmt(a.y, b.y, 0x7362) ^ 0x80808080u;
    return o;
}
template <bool STREAMED>
__device__ __forceinline__ uint2 ld_in8(const int8_t* frame, int x) {   // 8 bytes at frame + 8 x (frames are 8-byte aligned)
    const uint2* s = reinterpret_cast<const uint2*>(frame) + x;
    // streamed: the copy engine is still writing other frames of this buffer -> L2-coherent loads
    return STREAMED ? __ldcg(s) : __ldg(s);
}

// Pair load.  Parity part: pty[i][j] = v[K + q j + i] (column j of the q x 360 parity matrix is contiguous in the
// frame, layered_decoder.hh:124-126), and every pass reads it as wpty[i * 360 + j] (packed offset-binary pair, A in the
// low byte), i.e. transposed.  Both frames' parity bytes are read with coalesced 8-byte loads into vdata (which the
// systematic part fills only afterwards), interleaved, and written out transposed with coalesced 16-bit stores: a
// strided gather of single bytes straight from the frames would touch a sector per lane and per layer.  vdata holds
// 2K bytes, the parity pairs of the frame 2R: below rate 1/2 this goes in chunks of columns, a multiple of 8 columns
// each so that every chunk starts 8-byte aligned.  Then the systematic LLRs -> vdata (A in even bytes, B in odd).
// All threads of the CTA call it; the caller's barrier publishes vdata, the ones in here publish wpty.
template <bool STREAMED, int THREADS>
__device__ __noinline__ void load_pair(const LdpcParams2& p, const int8_t* inA, const int8_t* inB, uint16_t* vdata,
                                       uint16_t* wpty) {
    static_assert(THREADS % 360 == 0, "a whole number of threads per column");
    const int tid = threadIdx.x, q = p.q, K = p.K;
    uint4* v4 = reinterpret_cast<uint4*>(vdata);
    const int8_t* ptA = inA + K;
    const int8_t* ptB = inB + K;
    const int cols = min(360, (K / q) & ~7);
    const int jj = tid % 360, i0 = tid / 360;          // this thread's column in a chunk and first layer
    for (int j0 = 0; j0 < 360; j0 += cols) {
        const int nc = min(cols, 360 - j0);
        const int b8 = q * j0 / 8;
        for (int x = tid; x < q * nc / 8; x += THREADS) v4[x] = interleave8(ld_in8<STREAMED>(ptA, b8 + x), ld_in8<STREAMED>(ptB, b8 + x));
        __syncthreads();
        if (jj < nc)
            for (int i = i0; i < q; i += THREADS / 360) __stcg(&wpty[i * 360 + j0 + jj], vdata[jj * q + i]);
        __syncthreads();
    }
    for (int x = tid; x < K / 8; x += THREADS) v4[x] = interleave8(ld_in8<STREAMED>(inA, x), ld_in8<STREAMED>(inB, x));
}

// Take the next pair from the launch's counter ahead of time (the caller keeps it for its next round) and prefetch
// both of its frames into L2, so that its load_pair reads from L2 instead of HBM.  Streamed input is prefetched only
// when the copy engine has already delivered it; there is no waiting here.  cp.async.bulk.prefetch wants a 16-byte
// aligned address and size; a short frame (16 200 bytes) of odd index starts 8 bytes off, so the range is widened to
// 16-byte boundaries -- at most 15 bytes either side, inside the same mapped page as the frame's own bytes.
// The last grid's worth of pairs is left to be handed out when a CTA is actually free (kNoPair): a pair claimed
// ahead starts only after the slower frame of the current pair, which at the end of a launch lengthens its drain.
constexpr unsigned kNoPair = 0xFFFFFFFFu;   // no pair claimed ahead
template <bool STREAMED>
__device__ __noinline__ unsigned claim_next_pair(const LdpcParams2& p, unsigned npairs) {
    if (*reinterpret_cast<const volatile unsigned*>(p.work_counter) + gridDim.x >= npairs) return kNoPair;
    const unsigned np = atomicAdd(p.work_counter, 1u);
    if (np < npairs) {
        const unsigned f0 = 2u * np, nf = min(2u, (unsigned)p.nframes - f0);
        if (!STREAMED || *reinterpret_cast<const volatile unsigned*>(p.arrived) >= f0 + nf) {
            const size_t b = reinterpret_cast<size_t>(p.llr_in + (size_t)f0 * p.N);
            const size_t lo = b & ~(size_t)15, hi = (b + (size_t)nf * p.N + 15) & ~(size_t)15;
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(lo), "r"((unsigned)(hi - lo)) : "memory");
        }
    }
    return np;
}

// Streamed input: block until the copy engine has delivered `need` frames.  Returns false when the host never
// sent them (the caller marks the pair as failed instead of hanging or trapping the context).
static __device__ __noinline__ bool wait_arrived(const unsigned int* arrived_ptr, unsigned need, long long budget) {
    const volatile unsigned* arrived = arrived_ptr;
    const long long t0 = clock64();
    while (*arrived < need) {
        __nanosleep(500);
        if (clock64() - t0 > budget) return false;
    }
    return true;
}

template <int CNT, bool RAGGED, bool STREAMED, int OCC>
__global__ void __launch_bounds__(kThreads, OCC) ldpc_v2_kernel(const __grid_constant__ LdpcParams2 p) {
    constexpr int SLOTS = CNT + 2;
    constexpr int MW = (SLOTS + 1) / 2;     // message words per row in registers
    constexpr int SG = (SLOTS + 7) / 8;     // uint4 groups per row in the workspace
    static_assert(16 * SG >= 2 * SLOTS + 2, "the message record needs two spare bytes (row level)");
    constexpr int DW = (1 + 2 * CNT + 3) & ~3;   // words per layer descriptor (multiple of 4: read with 128-bit loads)
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const int q = p.q, K = p.K, N = p.N, R = p.R;
    uint16_t* vdata = reinterpret_cast<uint16_t*>(smem_raw);
    uint16_t* X = reinterpret_cast<uint16_t*>(smem_raw + (size_t)K * 2);      // X[j + 1] = pty[q-1][j], X[0] unused
    // Layer descriptors, built once per CTA: word 0 = levels | barrier-after << 8 | data links << 16, then per data
    // link the shared-memory address of its group's first LLR pair and 720 - 2 shift.  One or a few 128-bit loads per
    // layer replace a dozen dependent constant-bank reads and the arithmetic on them.
    uint32_t* desc = reinterpret_cast<uint32_t*>(smem_raw + (size_t)K * 2 + 768);
    __shared__ unsigned int s_pair;
    __shared__ int s_bad[2];

    const int tid = threadIdx.x;
    const int j = tid;     // this thread's row in every layer
    const uint32_t vbase = (uint32_t)__cvta_generic_to_shared(vdata);
    uint32_t dbase = (uint32_t)__cvta_generic_to_shared(desc);
    uint32_t j2 = 2u * (uint32_t)j;
    uint32_t xaddr = (uint32_t)__cvta_generic_to_shared(X) + j2;   // shared address of X[j]
    uint32_t m1 = 0xFFFFFFFFu;
    uint4* wmsg = reinterpret_cast<uint4*>(p.workspace + (size_t)blockIdx.x * p.ws_stride);
    uint16_t* wpty = reinterpret_cast<uint16_t*>(p.workspace + (size_t)blockIdx.x * p.ws_stride + (size_t)q * SG * 360 * 16);
    // bit planes of the full termination test (hard decisions, 360 bits per group in 13 words): in the workspace too --
    // with the screen the full test runs about twice per frame, and without the planes a third CTA fits on the SM
    uint32_t* HD = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(wpty) + (((size_t)R * 2 + 15) & ~(size_t)15));  // [2][ngroups][13]
    uint32_t* HP = HD + 2 * p.ngroups * kBitWords;                                                                       // [2][q][13]
    {   // Per-thread constants that ptxas would otherwise rematerialise from %tid and the shared-window base in every
        // layer (it does so under the register limit of the three-CTA variants): a round trip through memory makes
        // them plain values.  The words lie behind the bit planes in this CTA's workspace.
        volatile uint4* opq = reinterpret_cast<volatile uint4*>(HP + 2 * q * kBitWords + 4) + tid;
        opq->x = j2; opq->y = xaddr; opq->z = dbase; opq->w = m1;
        j2 = opq->x; xaddr = opq->y; dbase = opq->z; m1 = opq->w;
    }
    for (int x = tid; x < q * DW; x += kThreads) {
        const int i = x / DW, w = x - i * DW;
        const int loff = p.layer_off[i], cnt = (int)p.layer_off[i + 1] - loff;
        uint32_t v = 0;
        if (w == 0) {
            v = (uint32_t)p.layer_nlev[i] | (uint32_t)p.layer_sync[i] << 8 | (uint32_t)cnt << 16;
        } else if (w <= 2 * CNT) {
            const int c = (w - 1) >> 1;
            const int k = loff + (c < cnt ? c : 0);
            v = ((w - 1) & 1) ? (uint32_t)p.link_add[k] : vbase + 720u * p.link_group[k];
        }
        desc[x] = v;
    }
    const int npairs = (p.nframes + 1) >> 1;

    // zero the bit planes once: bytes 45..51 of every 360-bit group are never written and must read as 0
    for (int x = tid; x < 2 * (p.ngroups + q) * kBitWords; x += kThreads) __stcg(&HD[x], 0u);
    __shared__ unsigned int s_next;   // pair claimed (and prefetched) while the current one still ran, or kNoPair
    if (tid == 0) s_next = kNoPair;

    for (;;) {
        __syncthreads();
        if (tid == 0) {
            unsigned np = s_next;
            if (np == kNoPair) np = atomicAdd(p.work_counter, 1u);
            s_next = kNoPair;
            if (STREAMED && np < (unsigned)npairs) {
                // the copy engine raises *arrived behind every piece of frames it has delivered (same stream, so the
                // data is in memory before the count); pairs are handed out in frame order, so every waiter waits
                // for a copy that is already queued
                if (!wait_arrived(p.arrived, min(2u * np + 2u, (unsigned)p.nframes), p.wait_budget)) np |= 0x80000000u;
                __threadfence();
            }
            s_pair = np;
        }
        __syncthreads();
        const unsigned pair_word = s_pair;
        const unsigned pair = pair_word & 0x7FFFFFFFu;
        if (pair >= (unsigned)npairs) break;
        const int fa = 2 * pair, fb = 2 * pair + 1;
        const bool hasB = fb < p.nframes;
        if (STREAMED && (pair_word & 0x80000000u)) {   // input never arrived: report, do not hang
            if (tid == 0) {
                p.iters_out[fa] = kLdpcItersNoInput;
                if (hasB) p.iters_out[fb] = kLdpcItersNoInput;
            }
            continue;
        }
        const int8_t* inA = p.llr_in + (size_t)fa * N;
        const int8_t* inB = p.llr_in + (size_t)(hasB ? fb : fa) * N;

        // ---- load: parity LLR pairs -> workspace (transposed), systematic LLRs -> shared, offset binary
        load_pair<STREAMED, kThreads>(p, inA, inB, vdata, wpty);
        uint32_t pown = 0, psec = 0;      // unpacked parity LLRs of the row being worked on
        {
            const uint32_t last = __ldcg(wpty + (q - 1) * 360 + j);
            X[j + 1] = (uint16_t)last;
            pown = unpack_lo(last);
            psec = unpack_lo(__ldcg(wpty + (q - 2) * 360 + j));
        }
        if (tid == 0) X[0] = 0xFFFFu;

        int live = hasB ? 3 : 1;          // bit f set: frame f still iterating
        uint32_t off[CNT];                // shared-memory addresses of the data links of the current layer
        uint32_t lw0 = 0;                 // word 0 of the current layer's descriptor
        auto link_addresses = [&](int i) {
            uint32_t dw[DW];
#pragma unroll
            for (int x = 0; x < DW; x += 4)
                asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(dw[x]), "=r"(dw[x + 1]), "=r"(dw[x + 2]), "=r"(dw[x + 3])
                             : "r"(dbase + (uint32_t)(i * DW + x) * 4u));
            lw0 = dw[0];
#pragma unroll
            for (int c = 0; c < CNT; ++c)   // address of pair (j - shift) mod 360 of the group: the wrap is min(x, x - 720), unsigned
                off[c] = dw[1 + 2 * c] + addmin_u32(j2 + dw[2 + 2 * c], (uint32_t)-720);
        };
        // Screen of LDPCDecoder::bad: row (q-1, j) with the parity LLRs in pown (pty[q-1][j]) and psec (pty[q-2][j]).
        // Returns bit f set when the row is bad for frame f (sign product not positive or a zero LLR).
        auto screen = [&]() -> int {
            link_addresses(q - 1);
            const int cnt = (int)(lw0 >> 16);
            uint32_t sx = pown ^ psec, mn = minu2(__vabsdiffu4(pown, kC128), __vabsdiffu4(psec, kC128));
            int nl = 2;
#pragma unroll
            for (int c = 0; c < CNT; ++c) {
                if (!RAGGED || c < cnt) {
                    const uint32_t u = unpack_lo(lds_u16(off[c]));
                    sx ^= u;
                    mn = minu2(mn, __vabsdiffu4(u, kC128));
                    ++nl;
                }
            }
            // bit 7 set = non-negative; the row is good iff no LLR is zero and the number of negative ones is even
            if (nl & 1) sx ^= kC128;
            int bad = 0;
            if ((sx & 0x80u) || (mn & 0xFFFFu) == 0) bad |= 1;
            if ((sx & 0x800000u) || (mn >> 16) == 0) bad |= 2;
            return bad;
        };

        __syncthreads();
        int scr = screen();
        int res[2] = {-1, -1};
        for (int n = 0;; ++n) {
            // ---- LDPCDecoder::bad (layered_decoder.hh:28-45): screen first, full bit-plane test only when the
            //      screen found nothing for a frame that is still iterating
            int bad = (__syncthreads_or(scr & 1) ? 1 : 0) | (__syncthreads_or(scr & 2) ? 2 : 0);
            if (live & ~bad)
                bad = full_test<kThreads>(p, wpty, HP, HD, reinterpret_cast<const uint4*>(vdata), s_bad);
            // ---- while (bad() && --trials >= 0) update();  (layered_decoder.hh:127-128), per frame
            int fin = 0;
            for (int f = 0; f < 2; ++f) {
                if (!(live >> f & 1)) continue;
                if (!(bad >> f & 1)) {
                    res[f] = n;
                    fin |= 1 << f;
                } else if (n == p.max_trials) {
                    fin |= 1 << f;    // still bad after max_trials updates: -1
                }
            }
            if (fin) {
                emit_results<kThreads>(p, fin, res, fa, fb, wpty, reinterpret_cast<const uint4*>(vdata));
                // the first frame of the pair to stop: take the next pair now and start its frames towards L2 (the
                // other frame near the threshold runs more passes, which hide the HBM latency); not near the launch's end
                if (tid == 0 && s_next == kNoPair) s_next = claim_next_pair<STREAMED>(p, (unsigned)npairs);
                live &= ~fin;
                // the other frame goes on: nobody may start the next pass (it overwrites the LLRs and the parity
                // words in the workspace) while a slower warp is still reading them out
                if (live) __syncthreads();
            }
            if (!live) break;

            // ---- LDPCDecoder::update (layered_decoder.hh:46-74): one pass over all layers.  The first pass (all
            //      messages zero, row levels from the table) is its own instantiation of the loop.
            auto pass = [&](auto first_tag) {
                constexpr bool FIRST = decltype(first_tag)::value;
                uint32_t mw[MW];
                uint4 nxt[SG];
                uint32_t pnext = 0;    // parity LLR pair of the next layer's own parity bit
                uint32_t pprev = 0;
#pragma unroll
                for (int x = 0; x < MW; ++x) mw[x] = 0;
                // running pointers: this thread's message record and own parity LLR pair of the layer being worked on
                uint4* rp = wmsg + j;
                uint16_t* pp = wpty + j;
                psec = unpack_lo(lds_u16(xaddr));    // X[j] = pty[q-1][j-1]; thread 0 reads the +127 stand-in of the missing link
                pnext = __ldcg(pp);
                if (!FIRST) {
#pragma unroll
                    for (int s = 0; s < SG; ++s) nxt[s] = __ldcg(rp + s * 360);
                }
                // Dependency level of this thread's row inside the layer.  The first pass takes it from the table in
                // global memory and leaves it in the top byte of the row's message record (the record has at least two
                // spare bytes), so the later passes get it with the messages: no separate load whose scoreboard slot
                // the prefetches would share.
                uint32_t lev_next = (FIRST && p.layer_nlev[0] > 1) ? (uint32_t)p.row_level[j] << 24 : 0u;
                for (int i = 0; i < q; ++i) {
                    // everything loaded during the previous layer is consumed HERE, before this layer's prefetches
                    uint32_t keep = lev_next;          // top byte: the row's level
                    if (!FIRST) {
#pragma unroll
                        for (int s = 0; s < SG; ++s) {
                            if (4 * s + 0 < MW) mw[4 * s + 0] = nxt[s].x;
                            if (4 * s + 1 < MW) mw[4 * s + 1] = nxt[s].y;
                            if (4 * s + 2 < MW) mw[4 * s + 2] = nxt[s].z;
                            if (4 * s + 3 < MW) mw[4 * s + 3] = nxt[s].w;
                        }
                        keep = nxt[SG - 1].w;
                    }
                    // pty[q-1][j] was updated in layer 0 by thread j+1 (at least one barrier ago: layer_sync)
                    pown = unpack_lo(i == q - 1 ? lds_u16(xaddr + 2) : pnext);   // X[j + 1]
                    if (i + 1 < q) {   // prefetch the next layer's row while this one computes
                        pnext = __ldcg(pp + 360);
                        if (!FIRST) {
#pragma unroll
                            for (int s = 0; s < SG; ++s) nxt[s] = __ldcg(rp + (SG + s) * 360);
                        }
                    }
                    link_addresses(i);
                    const int cnt = RAGGED ? (int)(lw0 >> 16) : CNT;
                    const int nlev = (int)(lw0 & 0xFFu);
                    if (FIRST) lev_next = (i + 1 < q && p.layer_nlev[i + 1] > 1) ? (uint32_t)p.row_level[(i + 1) * 360 + j] << 24 : 0u;
                    if (nlev == 1) {
                        row_update<CNT, FIRST, RAGGED>(off, cnt, mw, pown, psec, keep, m1);
                        // barriers separate layers only where a later layer touches a bit group that a layer since the
                        // last barrier also touches (rows on disjoint bits commute)
                        if (lw0 & 0x100u) __syncthreads();
                    } else {
                        const int mylev = (int)(keep >> 24);
                        for (int lvl = 0; lvl < nlev; ++lvl) {
                            if (mylev == lvl) row_update<CNT, FIRST, RAGGED>(off, cnt, mw, pown, psec, keep, m1);
                            __syncthreads();
                        }
                    }
                    // write the row's messages back; retire the parity LLR that just got its last update
#pragma unroll
                    for (int s = 0; s < SG; ++s) {
                        uint4 o;
                        o.x = (4 * s + 0 < MW) ? mw[4 * s + 0] : 0u;
                        o.y = (4 * s + 1 < MW) ? mw[4 * s + 1] : 0u;
                        o.z = (4 * s + 2 < MW) ? mw[4 * s + 2] : 0u;
                        o.w = (4 * s + 3 < MW) ? mw[4 * s + 3] : 0u;
                        if (s == SG - 1 && 4 * s + 3 >= MW) o.w = keep & 0xFF000000u;   // (else row_update kept it)
                        __stcg(rp + s * 360, o);
                    }
                    if (i == 0)
                        sts_u16(xaddr, pack_pair(psec));      // X[j] = pty[q-1][j-1], updated again in layer q-1 (X[0]: scratch of thread 0)
                    else
                        __stcg(pp - 360, (uint16_t)pack_pair(psec));
                    pprev = psec;
                    psec = pown;
                    rp += SG * 360;
                    pp += 360;
                }
                // after the last layer: pprev = pty[q-2][j] (stored above), pown = pty[q-1][j], both final for this pass
                psec = pprev;
                {
                    const uint16_t pk = (uint16_t)pack_pair(pown);
                    sts_u16(xaddr + 2, pk);
                    __stcg(pp - 360, pk);
                }
            };
            if (n == 0) pass(std::true_type{});
            else pass(std::false_type{});
            __syncthreads();
            scr = screen();
        }
    }
}

}  // namespace v2
}  // namespace s2

#define S2_V2_K4(c, r) {{v2::ldpc_v2_kernel<c, r, false, (c <= 9 ? 2 : 1)>, v2::ldpc_v2_kernel<c, r, false, (c <= 9 ? 3 : 2)>}, \
                        {v2::ldpc_v2_kernel<c, r, true, (c <= 9 ? 2 : 1)>, v2::ldpc_v2_kernel<c, r, true, (c <= 9 ? 3 : 2)>}}
#define S2_V2_N4 {{nullptr, nullptr}, {nullptr, nullptr}}
#define V2U(c) {c, S2_V2_K4(c, false), S2_V2_N4}
#define V2B(c) {c, S2_V2_K4(c, false), S2_V2_K4(c, true)}
#define V2R(c) {c, S2_V2_N4, S2_V2_K4(c, true)}
