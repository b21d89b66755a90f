// K2, two lanes per row: the second-generation LDPC kernel (ldpc_v2.cuh) for the codes with many links per check
// (high rates: 10 to 30 links).  There one thread per row means a row body of several hundred dependent instructions,
// 117+ registers, one CTA of twelve warps per SM -- and every dependency level of a conflicted layer (SURVEY.md note
// N6; up to 90 levels in one layer) costs that whole latency while eleven warps wait.  Here a row is shared by two
// adjacent threads (736 threads, 23 warps per CTA):
//
//   * half h of row j owns the data links d = h, h + 2, h + 4, ... and ONE parity link (h = 0: the row's own parity
//     bit pty[i][j], h = 1: the second one, pty[i-1][j]), so both halves run the same instruction stream;
//   * the check-node reduction crosses the pair with two warp shuffles (the other half's minimum |t| and sign XOR:
//     BASELINE.json's "warp shuffles for the check-node min1/min2 reduction"), the own parity LLR moves to the other
//     half for the next layer with a third;
//   * everything else -- beta = 32 - m messages, layer descriptors in shared memory, screened termination test,
//     results written when a frame stops -- is the one-lane kernel's, and the arithmetic per link is identical
//     (same primitives in the same order per bit), so the two kernels produce the same bytes.
//
// A level step is half as long, registers per thread drop below 80 and twice as many warps hide the rest.
// Reference semantics: as ldpc_v2.cuh.  Included by ldpc2l_inst_*.cu only.
#pragma once
#include "ldpc_v2.cuh"

namespace s2 {
namespace v2 {

constexpr int kLdpcThreads2 = 720;   // one thread per half row: 22 warps and a half

// One half of a check row for both frames of the pair.
//   off[]  : shared-memory addresses of this half's data links (slot s = link 2 s + h)
//   cntl   : how many of them exist in this layer for this half
//   mw[]   : this half's message bytes beta = 32 - m; slot 0 = the parity link, slots 1.. = data links      (in/out)
//   preg   : the half's parity LLR, unpacked                                                                  (in/out)
// The other half's contribution to the minimum and to the sign product arrives by __shfl_xor.
template <int NL, bool FIRST, bool RAGGED>
__device__ __forceinline__ void row_update2(const uint32_t (&off)[NL], int cntl, uint32_t (&mw)[(NL + 2) / 2], uint32_t& preg,
                                            uint32_t keep, uint32_t m1, unsigned lanes) {
    constexpr int DH = NL + 1;            // slots of this half
    uint32_t tu[DH], a[DH];
    // sign bookkeeping as in row_update: both halves together hold 2 DH slots (absent ones count as +)
    uint32_t sx = ((2 * DH - 1) & 1) ? kC128 : 0u;
#pragma unroll
    for (int s = 0; s < DH; ++s) {
        uint32_t u;
        if (s == 0)
            u = preg;
        else
            u = (!RAGGED || s - 1 < cntl) ? unpack_lo(lds_u16(off[s - 1])) : kC255;
        uint32_t t = u;
        if (!FIRST) {
            const uint32_t beta = (s & 1) ? unpack_hi(mw[s >> 1]) : unpack_lo(mw[s >> 1]);
            t = addmin_relu(u + beta, kM32, kC255);
        }
        tu[s] = t;
        a[s] = __vabsdiffu4(t, kC128);
        sx ^= t;
    }
    // prefix / suffix minima of this half, the other half's total by shuffle
    uint32_t P[DH], S[DH];
    P[0] = a[0];
#pragma unroll
    for (int s = 1; s < DH; ++s) P[s] = minu2(P[s - 1], a[s]);
    S[DH - 1] = a[DH - 1];
#pragma unroll
    for (int s = DH - 2; s >= 0; --s) S[s] = minu2(S[s + 1], a[s]);
    const uint32_t other = __shfl_xor_sync(lanes, P[DH - 1], 1);   // (both halves of a row are always in `lanes` together)
    sx ^= __shfl_xor_sync(lanes, sx, 1) ^ (((2 * DH - 1) & 1) ? kC128 : 0u);   // (the start value only once)
    const uint32_t ssx = lane_mask7(sx);
    uint32_t prev = 0;
#pragma unroll
    for (int s = 0; s < DH; ++s) {
        uint32_t ex;
        if (s == 0)
            ex = minu2(S[1], other);
        else if (s == DH - 1)
            ex = minu2(P[DH - 2], other);
        else
            ex = min3u2(P[s - 1], S[s + 1], other);
        const uint32_t om = addmin_relu(ex, kAllOnes, kP32);
        const uint32_t neg = lane_mask7(tu[s]) ^ ssx;
        const uint32_t bias = neg * 0xFFFEFFFFu + kP32;
        const uint32_t bm = addmin(om ^ neg, bias, kP63);
        const uint32_t un = addmin_relu(tu[s] + bm, kM32, kC255);
        uint32_t beta;
        asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(beta) : "r"(bm), "r"(m1), "r"(kP64));
        if (s == 0) {
            preg = un;
        } else if (!RAGGED || s - 1 < cntl) {
            sts_u16(off[s - 1], pack_pair(un));
        }
        if (s & 1)
            mw[s >> 1] = pack_two(prev, beta);
        else if (s == DH - 1)
            mw[s >> 1] = prmt(beta, keep, 0x7620);
        prev = beta;
    }
}

template <int CNT, bool RAGGED, bool STREAMED>
__global__ void __launch_bounds__(kLdpcThreads2, 1) ldpc_v2l_kernel(const __grid_constant__ LdpcParams2 p) {
    constexpr int T = kLdpcThreads2;
    constexpr int NL = (CNT + 1) / 2;        // data link slots per half
    constexpr int DH = NL + 1;               // + the parity link
    constexpr int MW = (DH + 1) / 2;         // message words per half row in registers
    constexpr int SG = (DH + 7) / 8;         // uint4 groups per half row in the workspace
    static_assert(16 * SG >= 2 * DH + 2, "the message record needs two spare bytes (row level)");
    constexpr int HW = (2 * NL + 3) & ~3;    // descriptor words per half (multiple of 4)
    constexpr int DW = 4 + 2 * HW;           // words per layer descriptor: header, half 0 links, half 1 links
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const int q = p.q, K = p.K, N = p.N, R = p.R;
    uint16_t* vdata = reinterpret_cast<uint16_t*>(smem_raw);
    uint16_t* X = reinterpret_cast<uint16_t*>(smem_raw + (size_t)K * 2);      // X[j + 1] = pty[q-1][j], X[0] unused
    uint32_t* desc = reinterpret_cast<uint32_t*>(smem_raw + (size_t)K * 2 + 768);
    __shared__ unsigned int s_pair;
    __shared__ int s_bad[2];

    const int tid = threadIdx.x;
    const int h = tid & 1;
    const int j = tid >> 1;
    const unsigned wl = __activemask();      // this warp's lanes (the CTA's last warp is half a warp)
    const int slot_t = 2 * j + h;            // index of this half row in the workspace records
    const uint32_t vbase = (uint32_t)__cvta_generic_to_shared(vdata);
    uint32_t dbase = (uint32_t)__cvta_generic_to_shared(desc) + 16u + (uint32_t)h * HW * 4u;
    uint32_t j2 = 2u * (uint32_t)j;
    uint32_t xaddr = (uint32_t)__cvta_generic_to_shared(X) + j2;   // shared address of X[j]
    uint32_t m1 = 0xFFFFFFFFu;
    uint4* wmsg = reinterpret_cast<uint4*>(p.workspace + (size_t)blockIdx.x * p.ws_stride);
    uint16_t* wpty = reinterpret_cast<uint16_t*>(p.workspace + (size_t)blockIdx.x * p.ws_stride + (size_t)q * 2 * SG * 360 * 16);
    uint32_t* HD = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(wpty) + (((size_t)R * 2 + 15) & ~(size_t)15));  // [2][ngroups][13]
    uint32_t* HP = HD + 2 * p.ngroups * kBitWords;                                                                       // [2][q][13]
    {   // per-thread constants through memory, so that ptxas keeps them instead of recomputing them in every layer
        volatile uint4* opq = reinterpret_cast<volatile uint4*>(HP + 2 * q * kBitWords + 4) + tid;
        opq->x = j2; opq->y = xaddr; opq->z = dbase; opq->w = m1;
        j2 = opq->x; xaddr = opq->y; dbase = opq->z; m1 = opq->w;
    }
    // layer descriptors: header (levels | barrier-after << 8 | data links << 16), then per half its links' group
    // address and 720 - 2 shift
    for (int x = tid; x < q * DW; x += T) {
        const int i = x / DW, w = x - i * DW;
        const int loff = p.layer_off[i], cnt = (int)p.layer_off[i + 1] - loff;
        uint32_t v = 0;
        if (w == 0) {
            v = (uint32_t)p.layer_nlev[i] | (uint32_t)p.layer_sync[i] << 8 | (uint32_t)cnt << 16;
        } else if (w >= 4) {
            const int hh = (w - 4) / HW, e = (w - 4) - hh * HW;
            const int s = e >> 1, d = 2 * s + hh;
            if (s < NL) {
                const int k = loff + (d < cnt ? d : 0);
                v = (e & 1) ? (uint32_t)p.link_add[k] : vbase + 720u * p.link_group[k];
            }
        }
        desc[x] = v;
    }
    const int npairs = (p.nframes + 1) >> 1;
    for (int x = tid; x < 2 * (p.ngroups + q) * kBitWords; x += T) __stcg(&HD[x], 0u);
    __shared__ unsigned int s_next;   // pair claimed (and prefetched) while the current one still ran, or kNoPair
    if (tid == 0) s_next = kNoPair;

    for (;;) {
        __syncthreads();
        if (tid == 0) {
            unsigned np = s_next;
            if (np == kNoPair) np = atomicAdd(p.work_counter, 1u);
            s_next = kNoPair;
            if (STREAMED && np < (unsigned)npairs) {
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
        if (STREAMED && (pair_word & 0x80000000u)) {
            if (tid == 0) {
                p.iters_out[fa] = kLdpcItersNoInput;
                if (hasB) p.iters_out[fb] = kLdpcItersNoInput;
            }
            continue;
        }
        const int8_t* inA = p.llr_in + (size_t)fa * N;
        const int8_t* inB = p.llr_in + (size_t)(hasB ? fb : fa) * N;

        load_pair<STREAMED, T>(p, inA, inB, vdata, wpty);
        // this half's parity LLR of row (q-1, j): h = 0 pty[q-1][j], h = 1 pty[q-2][j] (for the screen before pass 1)
        uint32_t preg;
        {
            const uint32_t w = __ldcg(wpty + (q - 1 - h) * 360 + j);
            if (h == 0) X[j + 1] = (uint16_t)w;
            preg = unpack_lo(w);
        }
        if (tid == 0) X[0] = 0xFFFFu;

        int live = hasB ? 3 : 1;
        uint32_t off[NL];
        uint32_t lw0 = 0;
        auto link_addresses = [&](int i) {
            uint32_t dw[HW];
            const uint32_t lb = dbase + (uint32_t)(i * DW) * 4u;
            lw0 = lds_u32(lb - 16u - (uint32_t)h * HW * 4u);
#pragma unroll
            for (int x = 0; x < HW; x += 4)
                asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(dw[x]), "=r"(dw[x + 1]), "=r"(dw[x + 2]), "=r"(dw[x + 3])
                             : "r"(lb + (uint32_t)x * 4u));
#pragma unroll
            for (int s = 0; s < NL; ++s) off[s] = dw[2 * s] + addmin_u32(j2 + dw[2 * s + 1], (uint32_t)-720);
        };
        // data links of this half in a layer with cnt data links: d = h, h + 2, ... < cnt
        auto half_links = [&](int cnt) { return (cnt - h + 1) >> 1; };
        auto screen = [&]() -> int {
            link_addresses(q - 1);
            const int cntl = half_links((int)(lw0 >> 16));
            uint32_t sx = preg, mn = __vabsdiffu4(preg, kC128);
            int nl = 1;
#pragma unroll
            for (int s = 0; s < NL; ++s) {
                if (s < cntl) {
                    const uint32_t u = unpack_lo(lds_u16(off[s]));
                    sx ^= u;
                    mn = minu2(mn, __vabsdiffu4(u, kC128));
                    ++nl;
                }
            }
            if (nl & 1) sx ^= kC128;
            sx ^= __shfl_xor_sync(wl, sx, 1);
            mn = minu2(mn, __shfl_xor_sync(wl, mn, 1));
            int bad = 0;
            if ((sx & 0x80u) || (mn & 0xFFFFu) == 0) bad |= 1;
            if ((sx & 0x800000u) || (mn >> 16) == 0) bad |= 2;
            return bad;
        };

        __syncthreads();
        int scr = screen();
        int res[2] = {-1, -1};
        for (int n = 0;; ++n) {
            int bad = (__syncthreads_or(scr & 1) ? 1 : 0) | (__syncthreads_or(scr & 2) ? 2 : 0);
            if (live & ~bad)
                bad = full_test<T>(p, wpty, HP, HD, reinterpret_cast<const uint4*>(vdata), s_bad);
            int fin = 0;
            for (int f = 0; f < 2; ++f) {
                if (!(live >> f & 1)) continue;
                if (!(bad >> f & 1)) {
                    res[f] = n;
                    fin |= 1 << f;
                } else if (n == p.max_trials) {
                    fin |= 1 << f;
                }
            }
            if (fin) {
                emit_results<T>(p, fin, res, fa, fb, wpty, reinterpret_cast<const uint4*>(vdata));
                if (tid == 0 && s_next == kNoPair) s_next = claim_next_pair<STREAMED>(p, (unsigned)npairs);   // as ldpc_v2_kernel
                live &= ~fin;
                // the other frame goes on: nobody may start the next pass (it overwrites the LLRs and the parity
                // words in the workspace) while a slower warp is still reading them out
                if (live) __syncthreads();
            }
            if (!live) break;

            auto pass = [&](auto first_tag) {
                constexpr bool FIRST = decltype(first_tag)::value;
                uint32_t mw[MW];
                uint4 nxt[SG];
                uint32_t pnext = 0;
#pragma unroll
                for (int x = 0; x < MW; ++x) mw[x] = 0;
                uint4* rp = wmsg + slot_t;
                uint16_t* pp = wpty + j;
                // h = 1 starts with pty[q-1][j-1] (X[j]; thread 0's is the +127 stand-in of the missing link)
                if (h == 1) preg = unpack_lo(lds_u16(xaddr));
                pnext = __ldcg(pp);
                if (!FIRST) {
#pragma unroll
                    for (int s = 0; s < SG; ++s) nxt[s] = __ldcg(rp + s * 720);
                }
                uint32_t lev_next = (FIRST && p.layer_nlev[0] > 1) ? (uint32_t)p.row_level[j] << 24 : 0u;
                for (int i = 0; i < q; ++i) {
                    uint32_t keep = lev_next;
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
                    if (h == 0)     // the row's own parity bit
                        preg = unpack_lo(i == q - 1 ? lds_u16(xaddr + 2) : pnext);   // X[j + 1]
                    if (i + 1 < q) {
                        pnext = __ldcg(pp + 360);
                        if (!FIRST) {
#pragma unroll
                            for (int s = 0; s < SG; ++s) nxt[s] = __ldcg(rp + (SG + s) * 720);
                        }
                    }
                    link_addresses(i);
                    const int cntl = RAGGED ? half_links((int)(lw0 >> 16)) : (h == 0 ? (CNT + 1) / 2 : CNT / 2);
                    const int nlev = (int)(lw0 & 0xFFu);
                    if (FIRST) lev_next = (i + 1 < q && p.layer_nlev[i + 1] > 1) ? (uint32_t)p.row_level[(i + 1) * 360 + j] << 24 : 0u;
                    constexpr bool kPartial = RAGGED || (CNT & 1);   // some half has fewer links than NL
                    if (nlev == 1) {
                        row_update2<NL, FIRST, kPartial>(off, cntl, mw, preg, keep, m1, wl);
                        if (lw0 & 0x100u) __syncthreads();
                    } else {
                        const int mylev = (int)(keep >> 24);
                        for (int lvl = 0; lvl < nlev; ++lvl) {
                            const unsigned lanes = __ballot_sync(wl, mylev == lvl);
                            if (mylev == lvl) row_update2<NL, FIRST, kPartial>(off, cntl, mw, preg, keep, m1, lanes);
                            __syncthreads();
                        }
                    }
#pragma unroll
                    for (int s = 0; s < SG; ++s) {
                        uint4 o;
                        o.x = (4 * s + 0 < MW) ? mw[4 * s + 0] : 0u;
                        o.y = (4 * s + 1 < MW) ? mw[4 * s + 1] : 0u;
                        o.z = (4 * s + 2 < MW) ? mw[4 * s + 2] : 0u;
                        o.w = (4 * s + 3 < MW) ? mw[4 * s + 3] : 0u;
                        if (s == SG - 1 && (4 * s + 3 >= MW || !(DH & 1))) o.w = (o.w & 0x00FFFFFFu) | (keep & 0xFF000000u);
                        __stcg(rp + s * 720, o);
                    }
                    // h = 1 retires the parity LLR that just got its last update; h = 0 hands pty[i][j] to h = 1
                    if (h == 1) {
                        if (i == 0)
                            sts_u16(xaddr, pack_pair(preg));           // X[j] = pty[q-1][j-1], updated again in layer q-1
                        else
                            __stcg(pp - 360, (uint16_t)pack_pair(preg));
                    }
                    const uint32_t other = __shfl_xor_sync(wl, preg, 1);
                    if (h == 1 && i + 1 < q) preg = other;
                    rp += 2 * SG * 360;
                    pp += 360;
                }
                // after the last layer: h = 0 holds pty[q-1][j], h = 1 pty[q-2][j] (stored above), both final
                if (h == 0) {
                    const uint16_t pk = (uint16_t)pack_pair(preg);
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

#define S2_V2L_K2(c, r) {v2::ldpc_v2l_kernel<c, r, false>, v2::ldpc_v2l_kernel<c, r, true>}
#define S2_V2L_N2 {nullptr, nullptr}
#define V2LU(c) {c, S2_V2L_K2(c, false), S2_V2L_N2}
#define V2LR(c) {c, S2_V2L_N2, S2_V2L_K2(c, true)}
