// K3/K4/K5 -- see bch_decoder.cuh.
#include "bch_decoder.cuh"

#include <algorithm>

namespace s2 {
namespace {

constexpr int kWarps = 4;             // frames per CTA
constexpr int kMaxT = 12;

struct ResultRec {                    // mirrors dvbs2fec_result (include/dvbs2fec.h)
    unsigned long long tag;
    short ldpc_iters;
    short bch_corr;
    unsigned int flags;
};

__device__ __forceinline__ uint32_t gf_mul(const GfDev& f, uint32_t a, uint32_t b) {
    if (!a || !b) return 0;
    int s = (int)f.log[a] + (int)f.log[b];
    if (s >= f.N) s -= f.N;
    return f.exp[s];
}
__device__ __forceinline__ uint32_t gf_div(const GfDev& f, uint32_t a, uint32_t b) {  // b != 0
    if (!a) return 0;
    int s = (int)f.log[a] - (int)f.log[b];
    if (s < 0) s += f.N;
    return f.exp[s];
}
// a * alpha^e, 0 <= e < N
__device__ __forceinline__ uint32_t gf_mul_exp(const GfDev& f, uint32_t a, int e) {
    if (!a) return 0;
    int s = (int)f.log[a] + e;
    if (s >= f.N) s -= f.N;
    return f.exp[s];
}

__device__ __forceinline__ uint32_t warp_xor(uint32_t v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v ^= __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}

__global__ void __launch_bounds__(kWarps * 32) bch_kernel(const __grid_constant__ BchArgs a) {
    extern __shared__ __align__(16) uint8_t smem[];
    const BchDev& c = a.code;
    const GfDev& f = c.gf;
    const int t = c.t, NR = 2 * c.t, m = f.m;
    uint16_t* s_crc = reinterpret_cast<uint16_t*>(smem);            // [t][256]
    uint16_t* s_basis = s_crc + kMaxT * 256;                        // [t][16]
    uint8_t* s_frames = reinterpret_cast<uint8_t*>(s_basis + kMaxT * 16);
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t* fr = s_frames + (size_t)wid * a.hard_stride;
    __shared__ uint16_t s_synd[kWarps][24];
    __shared__ uint16_t s_lambda[kWarps][26];
    __shared__ uint16_t s_ev[kWarps][26];
    __shared__ int s_loc[kWarps][26];
    __shared__ int s_nloc[kWarps];

    for (int x = threadIdx.x; x < t * 256; x += blockDim.x) s_crc[x] = c.crc[x];
    for (int x = threadIdx.x; x < t * 16; x += blockDim.x) s_basis[x] = c.basis[x];
    __syncthreads();

    const int nbytes = c.nbch >> 3, kbytes = c.kbch >> 3;
    for (int frame = blockIdx.x * kWarps + wid; frame < a.nframes; frame += gridDim.x * kWarps) {
        uint8_t* gfr = a.hard + (size_t)frame * a.hard_stride;
        // ---- stage the codeword (hard decisions of the K_ldpc = nbch systematic bits)
        for (int x = lane; x < a.hard_stride / 16; x += 32)
            reinterpret_cast<uint4*>(fr)[x] = reinterpret_cast<const uint4*>(gfr)[x];
        __syncwarp();

        // ---- syndromes S_i = c(alpha^i), i = 1..2t.  Odd i: remainder of this lane's byte chunk modulo
        //      the minimal polynomial of alpha^i, mapped into the field, weighted by alpha^(i * bits
        //      that follow the chunk), XOR-reduced over lanes.  Even i: S_2i = S_i^2 (binary code).
        const int chunk = (nbytes + 31) >> 5;
        const int beg = min(lane * chunk, nbytes), end = min(beg + chunk, nbytes);
        uint32_t r[kMaxT];
#pragma unroll
        for (int k = 0; k < kMaxT; ++k) r[k] = 0;
        const uint32_t rmask = (1u << m) - 1u;
        for (int x = beg; x < end; ++x) {
            uint32_t byte = fr[x];
#pragma unroll
            for (int k = 0; k < kMaxT; ++k)
                if (k < t) {
                    // r <- (r x^8 + byte) mod m_k(x);  crc[idx] = (idx x^m) mod m_k(x)
                    uint32_t idx = r[k] >> (m - 8);
                    r[k] = (((r[k] << 8) & rmask) | byte) ^ s_crc[k * 256 + idx];
                }
        }
        const int bits_after = 8 * (nbytes - end);
        uint32_t so[kMaxT];
#pragma unroll
        for (int k = 0; k < kMaxT; ++k) {
            so[k] = 0;
            if (k < t) {
                uint32_t v = 0;
                for (int b = 0; b < m; ++b)
                    if ((r[k] >> b) & 1u) v ^= s_basis[k * 16 + b];
                int e = (int)(((long long)(2 * k + 1) * bits_after) % f.N);
                so[k] = warp_xor(gf_mul_exp(f, v, e));
            }
        }
        if (lane == 0) {
#pragma unroll
            for (int k = 0; k < kMaxT; ++k)
                if (k < t) s_synd[wid][2 * k] = (uint16_t)so[k];        // synd[i] = c(alpha^(i+1))
            for (int i = 2; i <= NR; i += 2) {                           // S_i = S_(i/2)^2
                uint32_t h = s_synd[wid][i / 2 - 1];
                s_synd[wid][i - 1] = (uint16_t)gf_mul(f, h, h);
            }
        }
        __syncwarp();
        uint32_t any = 0;
        if (lane < NR) any = s_synd[wid][lane];
        any = __ballot_sync(0xFFFFFFFFu, any != 0);

        int corr = 0;
        if (any) {
            // ---- Berlekamp-Massey (reed_solomon_error_correction.hh:225-276), coefficient i on lane i
            uint32_t C = (lane == 0), B = (lane == 0);
            int L = 0, mm = 1;
            for (int n = 0; n < NR; ++n) {
                uint32_t term = 0;
                if (lane == 0) term = s_synd[wid][n];
                else if (lane <= L) term = gf_mul(f, C, s_synd[wid][n - lane]);
                uint32_t d = warp_xor(term);
                if (!d) {
                    ++mm;
                } else {
                    uint32_t Bs = __shfl_sync(0xFFFFFFFFu, B, (lane - mm) & 31);
                    uint32_t T = (lane < mm || lane > NR) ? C : (gf_mul(f, d, Bs) ^ C);
                    if (2 * L <= n) {
                        L = n + 1 - L;
                        B = (lane <= NR) ? gf_div(f, C, d) : 0u;
                        mm = 1;
                    } else {
                        ++mm;
                    }
                    C = (lane <= NR) ? T : 0u;
                }
            }
            // trim trailing zero coefficients (:301-307)
            unsigned nzmask = __ballot_sync(0xFFFFFFFFu, C != 0 && lane <= L);
            int deg = nzmask ? 31 - __clz(nzmask) : -1;
            if (lane <= NR) s_lambda[wid][lane] = (uint16_t)C;
            if (lane == 0) s_nloc[wid] = 0;
            __syncwarp();
            bool fail = deg < 0;
            int count = 0;
            if (!fail && deg > 0) {
                // degree-2 closed form of the reference refuses the all-ones half-trace argument
                // (reed_solomon_error_correction.hh:80-83,111-122): keep that observable behaviour
                bool quirk = false;
                if (deg == 2) {
                    uint32_t l0 = s_lambda[wid][0], l1 = s_lambda[wid][1], l2 = s_lambda[wid][2];
                    if (!l1 || !l0) quirk = true;
                    else quirk = gf_div(f, gf_mul(f, l2, l0), gf_mul(f, l1, l1)) == (uint32_t)f.N;
                }
                if (!quirk) {
                    // ---- root search over the nbch real positions: position p (full-length index
                    //      prefix + p) is a root iff Lambda(alpha^(prefix + p + 1)) == 0  (:39-61)
                    int idx[kMaxT + 1];
                    int step[kMaxT + 1];
                    const uint32_t l0 = s_lambda[wid][0];
#pragma unroll
                    for (int jj = 1; jj <= kMaxT; ++jj) {
                        idx[jj] = -1;
                        step[jj] = 0;
                        if (jj <= deg) {
                            uint32_t lj = s_lambda[wid][jj];
                            if (lj) {
                                long long e = (long long)jj * (c.prefix + 1 + lane) + f.log[lj];
                                idx[jj] = (int)(e % f.N);
                                step[jj] = (32 * jj) % f.N;
                            }
                        }
                    }
                    for (int p0 = 0; p0 < c.nbch; p0 += 32) {
                        uint32_t sum = l0;
#pragma unroll
                        for (int jj = 1; jj <= kMaxT; ++jj)
                            if (jj <= deg && idx[jj] >= 0) {
                                sum ^= f.exp[idx[jj]];
                                idx[jj] += step[jj];
                                if (idx[jj] >= f.N) idx[jj] -= f.N;
                            }
                        int p = p0 + lane;
                        if (p < c.nbch && sum == 0) {
                            int slot = atomicAdd(&s_nloc[wid], 1);
                            if (slot < 26) s_loc[wid][slot] = c.prefix + p;
                        }
                    }
                    __syncwarp();
                    count = s_nloc[wid];
                }
                if (count < deg) fail = true;
            }
            if (!fail && deg > 0) {
                // ---- Forney (:137-204), FCR = 1: evaluator = (S * Lambda) mod x^NR, up to degree count
                int top = min(count, NR - 1);
                uint32_t ev = 0;
                if (lane <= top) {
                    for (int jj = 0; jj <= lane; ++jj)
                        ev ^= gf_mul(f, s_synd[wid][lane - jj], s_lambda[wid][jj]);
                }
                unsigned evmask = __ballot_sync(0xFFFFFFFFu, ev != 0);
                int evdeg = evmask ? 31 - __clz(evmask) : -1;
                if (lane <= top) s_ev[wid][lane] = (uint16_t)ev;
                __syncwarp();
                uint32_t mag = 0;
                int loc = 0;
                if (lane < count) {
                    loc = s_loc[wid][lane];
                    int root = loc + 1;                       // locations[i] * Index(1)
                    if (root >= f.N) root -= f.N;
                    int tmp = root;
                    uint32_t eval = s_ev[wid][0];
                    for (int jj = 1; jj <= evdeg; ++jj) {
                        eval ^= gf_mul_exp(f, s_ev[wid][jj], tmp);
                        tmp += root;
                        if (tmp >= f.N) tmp -= f.N;
                    }
                    if (eval) {
                        uint32_t deriv = s_lambda[wid][1];
                        int root2 = 2 * root;
                        if (root2 >= f.N) root2 -= f.N;
                        int tmp2 = root2;
                        for (int jj = 3; jj <= count; jj += 2) {
                            deriv ^= gf_mul_exp(f, s_lambda[wid][jj], tmp2);
                            tmp2 += root2;
                            if (tmp2 >= f.N) tmp2 -= f.N;
                        }
                        int e = (int)f.log[eval] - (int)f.log[deriv];   // log[0] = N mirrors index(0)
                        if (e < 0) e += f.N;
                        mag = f.exp[e];
                    }
                }
                unsigned big = __ballot_sync(0xFFFFFFFFu, lane < count && mag > 1);
                if (big) {
                    fail = true;                              // magnitude > 1 (:116-120 of the BCH driver)
                } else {
                    if (lane < count && mag) {
                        int bit = loc - c.prefix;             // codeword bit index
                        atomicXor(reinterpret_cast<unsigned int*>(fr) + (bit >> 5),
                                  0x80u >> (bit & 7) << (8 * ((bit >> 3) & 3)));
                    }
                    corr = __popc(__ballot_sync(0xFFFFFFFFu, lane < count && mag != 0));
                }
            }
            if (fail) corr = -1;
            __syncwarp();
        }

        // ---- outputs: corrected codeword back in place, descrambled BBFRAME, per-frame record
        if (any && corr > 0) {
            for (int x = lane; x < a.hard_stride / 16; x += 32)
                reinterpret_cast<uint4*>(gfr)[x] = reinterpret_cast<const uint4*>(fr)[x];
        }
        if (a.bb_out) {
            uint8_t* o = a.bb_out + (size_t)frame * kbytes;
            if (a.descramble)
                for (int x = lane; x < kbytes; x += 32) o[x] = fr[x] ^ c.prbs[x];
            else
                for (int x = lane; x < kbytes; x += 32) o[x] = fr[x];
        }
        if (lane == 0) {
            int it = a.ldpc_iters ? a.ldpc_iters[frame] : 0;
            if (a.corr_out) a.corr_out[frame] = (int16_t)corr;
            if (a.results) {
                ResultRec rr;
                rr.tag = a.tags ? a.tags[frame] : a.tag_base + (unsigned long long)frame;
                rr.ldpc_iters = (short)it;
                rr.bch_corr = (short)corr;
                rr.flags = (it < 0 ? 1u : 0u) | (corr < 0 ? 2u : 0u);
                if (a.descramble) {
                    // BBHEADER CRC-8 as the downstream parser checks it (bbframe_ts_parser.cpp:66-80): bit-serial,
                    // MSB first, reflected polynomial 0xAB over the first 80 descrambled bits; valid iff it ends at 0
                    uint32_t crc = 0;
                    for (int n = 0; n < 80; ++n) {
                        uint32_t byte = fr[n >> 3] ^ c.prbs[n >> 3];
                        uint32_t b = ((byte >> (7 - (n & 7))) & 1u) ^ (crc & 1u);
                        crc >>= 1;
                        if (b) crc ^= 0xABu;
                    }
                    if (crc) rr.flags |= 4u;
                }
                reinterpret_cast<ResultRec*>(a.results)[frame] = rr;
            }
        }
        __syncwarp();
    }
}

// gridDim.y is at most 65535: each block row takes frames blockIdx.y, blockIdx.y + gridDim.y, ...
__global__ void descramble_kernel(uint8_t* frames, int stride, int nframes, int kbytes, const uint8_t* prbs) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= kbytes) return;
    const uint8_t p = prbs[x];
    for (int f = blockIdx.y; f < nframes; f += gridDim.y) frames[(size_t)f * stride + x] ^= p;
}

}  // namespace

int bch_launch(const BchArgs& a, cudaStream_t stream) {
    if (a.nframes <= 0) return 0;
    if (a.code.t > kMaxT || (a.hard_stride & 15)) return (int)cudaErrorInvalidValue;
    size_t smem = (size_t)kMaxT * 256 * 2 + kMaxT * 16 * 2 + (size_t)kWarps * a.hard_stride;
    int grid = (a.nframes + kWarps - 1) / kWarps;
    if (grid > 148 * 16) grid = 148 * 16;
    bch_kernel<<<grid, kWarps * 32, smem, stream>>>(a);
    return (int)cudaGetLastError();
}

int descramble_launch(uint8_t* frames, int stride, int nframes, int kbch, const uint8_t* prbs, cudaStream_t stream) {
    if (nframes <= 0) return 0;
    int kbytes = kbch / 8;
    dim3 grid((kbytes + 255) / 256, std::min(nframes, 65535));
    descramble_kernel<<<grid, 256, 0, stream>>>(frames, stride, nframes, kbytes, prbs);
    return (int)cudaGetLastError();
}

}  // namespace s2
