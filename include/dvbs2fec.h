/* dvbs2fec -- C ABI of the B200 DVB-S2 decode stage (libdvbs2fec.so).
 *
 * This is the drop-in boundary for the decode stage of the SDR++ dvbs_demodulator module: the
 * calls below replace the five host objects DVBS2Demod::process drives at
 * src/demod/dvbs2/module_dvbs2_demod.cpp:334-367 (S2BBToSoft, BBFrameLDPC, the repack loop,
 * BBFrameBCH, BBFrameDescrambler).  Plain C types only, opaque handle, caller-owned buffers,
 * negative return = error (never an exception), one handle per demodulator instance; handles are
 * independent and may be used from different threads concurrently (one thread per handle).
 *
 * Every entry point cites the reference interface it stands in for (paths relative to the
 * reference's src/demod/).  INTEGRATION.md shows the ~30-line patch that binds them.
 */
#ifndef DVBS2FEC_H
#define DVBS2FEC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DVBS2FEC_OK 0
#define DVBS2FEC_EINVAL (-22)   /* bad argument / unsupported MODCOD+frame-size (reference: get_dvbs2_cfg throws,
                                   codings/modcod_to_cfg.cpp:10-11,134-135; no LDPC table: bbframe_ldpc.cpp:67-68,105-106) */
#define DVBS2FEC_ENODEV (-19)   /* no usable CUDA device / kernels missing: the library never falls back to the CPU */
#define DVBS2FEC_ECUDA (-5)     /* a CUDA call failed; dvbs2fec_last_error() has the text */
#define DVBS2FEC_EAGAIN (-11)   /* queue full (submit) */
#define DVBS2FEC_ENOSPC (-28)   /* BBFRAME parser: GSE output does not fit the caller's buffer / descriptor pool */

#define DVBS2FEC_FLAG_LDPC_FAIL 1u /* LDPC never met all parity checks (BBFrameLDPC::decode returned -1) */
#define DVBS2FEC_FLAG_BCH_FAIL 2u  /* BBFrameBCH::decode returned -1 */
#define DVBS2FEC_FLAG_BBHEADER_CRC_FAIL 4u /* CRC-8 over the 80 BBHEADER bits is non-zero: BBFrameTSParser::work would
                                              drop this frame (dvbs2/bbframe_ts_parser.cpp:66-80,121-134) */
#define DVBS2FEC_FLAG_DUMMY 8u     /* VCM calls: the frame is a DUMMY PLFRAME (modcod 0); nothing was decoded */

typedef struct dvbs2fec_handle dvbs2fec_handle;

typedef struct {
    int32_t n_devices;      /* 0 = the calling thread's current CUDA device (cudaGetDevice; device 0 unless the caller chose another);
                               otherwise devices[0..n_devices) share the frames of every batch */
    int32_t devices[8];
    int32_t max_batch;      /* frames per kernel launch and per device (default 1024) */
    int32_t max_latency_us; /* submit/collect queue: launch a partial batch after this long (default 2000) */
    int32_t max_trials;     /* default LDPC iteration cap (reference: DVBS2_DEMOD_LDPC_RETRIES, main.cpp:65) */
    int32_t reserved[4];
} dvbs2fec_config;

/* Per-frame outcome; mirrors the fields DVBS2Demod exposes to the GUI (module_dvbs2_demod.h:86-87). */
typedef struct {
    uint64_t tag;        /* caller's tag (submit) or frame index (batch calls) */
    int16_t ldpc_iters;  /* iterations executed, 0 = input already a codeword, -1 = not converged (bbframe_ldpc.cpp:135-138) */
    int16_t bch_corr;    /* corrected bit errors, -1 = uncorrectable (bose_chaudhuri_hocquenghem_decoder.hh:116-142) */
    uint32_t flags;      /* DVBS2FEC_FLAG_* */
} dvbs2fec_result;

/* ctor/dtor of the decoder objects (DVBS2Demod::init, module_dvbs2_demod.cpp:7-91).  cfg may be NULL. */
int dvbs2fec_create(const dvbs2fec_config* cfg, dvbs2fec_handle** out);
void dvbs2fec_destroy(dvbs2fec_handle* h);
const char* dvbs2fec_last_error(void);

/* DVBS2Demod::setDemodParams (module_dvbs2_demod.h:60, .cpp:118-168) + get_dvbs2_cfg
 * (codings/modcod_to_cfg.cpp:5-140): modcod 1..28.  Queued frames of the previous MODCOD are
 * decoded and kept for collect() first.  max_trials <= 0 keeps the configured default. */
int dvbs2fec_set_modcod(dvbs2fec_handle* h, int modcod, int shortframes, int pilots, int max_trials);

/* PL descrambling inside the demapper (S2Scrambling, dvbs2/codings/s2_scrambling.h:12-45; the reference runs it in
 * S2PLLBlock::process, dvbs2_pll.cpp:37-44, on the phase-corrected symbol): codenum = Gold code number
 * 0..262141 -> PLFRAME inputs are taken as still PL-scrambled and every symbol after the 90 header symbols
 * (pilots count) is turned back by Rn * 90 degrees before demapping; codenum < 0 (default) -> inputs are already
 * descrambled.  Survives dvbs2fec_set_modcod; frames already queued are decoded with the previous setting. */
int dvbs2fec_set_pl_scrambling(dvbs2fec_handle* h, int codenum);

/* getKBCH (module_dvbs2_demod.h:80), BBFrameLDPC::dataSize (codings/bbframe_ldpc.h:48), frame length. Bits. */
int dvbs2fec_kbch(const dvbs2fec_handle* h);
int dvbs2fec_kldpc(const dvbs2fec_handle* h);
int dvbs2fec_nldpc(const dvbs2fec_handle* h);
/* complex samples per PLFRAME handed to the demapper: 90 header + payload (+ pilot blocks) */
int dvbs2fec_plframe_symbols(const dvbs2fec_handle* h);

/* ---- stage-level calls: one-to-one with the reference objects, HOST buffers, synchronous ---- */

/* S2BBToSoft::process (dvbs2/dvbs2_bb_to_soft.cpp:7-33): n PLFRAMEs of dvbs2fec_plframe_symbols()
 * complex floats each (header at [0,90), PL-descrambled) -> n x N int8 LLRs, deinterleaved. */
int dvbs2fec_bb_to_soft(dvbs2fec_handle* h, const float* plframes, int n, int8_t* llr_out);
/* BBFrameLDPC::decode (codings/bbframe_ldpc.cpp:123-139), once per frame: n x N LLRs are replaced by the
 * posterior LLRs; iters[i] = its return value for frame i. */
int dvbs2fec_ldpc_decode(dvbs2fec_handle* h, int8_t* frames, int n, int max_trials, int16_t* iters);
/* BBFrameBCH::decode (codings/bbframe_bch.cpp:380-405): n x (K_ldpc/8) bytes corrected in place. */
int dvbs2fec_bch_decode(dvbs2fec_handle* h, uint8_t* frames, int n, int16_t* corrections);
/* BBFrameDescrambler::work (codings/bbframe_descramble.cpp:138-143): first kbch/8 bytes of each
 * stride-byte frame XORed in place. */
int dvbs2fec_descramble(dvbs2fec_handle* h, uint8_t* frames, int stride, int n);

/* ---- whole decode stage, synchronous (module_dvbs2_demod.cpp:349-366 for n frames) ---- */

/* n x N int8 LLRs (host) -> n x kbch/8 BBFRAME bytes (host) + per-frame results.  This is the parity
 * boundary: bit-exact with the reference decoder applied to each frame. */
int dvbs2fec_decode_batch(dvbs2fec_handle* h, const int8_t* llr, int n, uint8_t* bb_out, dvbs2fec_result* results);
/* same, starting from PLFRAME symbols (module_dvbs2_demod.cpp:334-366) */
int dvbs2fec_decode_plframes(dvbs2fec_handle* h, const float* plframes, int n, uint8_t* bb_out,
                             dvbs2fec_result* results);
/* Quantised symbols path for the LUT constellations (QPSK, 8PSK, 16APSK).  The reference demapper reduces every
 * symbol to two 8-bit LUT coordinates before it looks anything up (constellation_t::demod_soft_lut,
 * common/dsp/demod/constellation.cpp:295-310).  dvbs2fec_quantize_plframes does exactly that on the host -- pilot
 * removal and PL descrambling (dvbs2fec_set_pl_scrambling) included, header dropped -- and writes 2 bytes per payload
 * symbol (N / bits_per_symbol symbols per frame); dvbs2fec_decode_plframes_idx / dvbs2fec_submit_plframe_idx take
 * those instead of 8-byte complex floats: a quarter of the PCIe traffic, bit-identical LLRs.  32APSK has no LUT in
 * the reference (:294,319-321): DVBS2FEC_EINVAL, send symbols. */
int dvbs2fec_quantize_plframes(const dvbs2fec_handle* h, const float* plframes, int n, uint8_t* idx_out);
int dvbs2fec_decode_plframes_idx(dvbs2fec_handle* h, const uint8_t* idx, int n, uint8_t* bb_out, dvbs2fec_result* results);
/* device-resident variant on the handle's first device: all pointers are device pointers, work is
 * enqueued on `cuda_stream` (a cudaStream_t; NULL = default stream) and NOT synchronised.  The call owns a
 * scratch area of its own (never shared with the synchronous entry points); calls issued on different streams
 * are chained on the device through an event, so they may be issued freely but do not overlap each other.  The
 * caller must keep d_llr, d_bb_out and d_results alive until its stream has passed the enqueued work. */
int dvbs2fec_decode_batch_device(dvbs2fec_handle* h, const int8_t* d_llr, int n, uint8_t* d_bb_out,
                                 dvbs2fec_result* d_results, void* cuda_stream);
/* same from PLFRAME symbols on the device (dvbs2fec_plframe_symbols complex floats per frame, as PL sync / the payload
 * phase loop leave them: dvbs2fec_plsync_process_device, dvbs2fec_pll_process_device): demapper, LDPC, BCH, descrambler
 * without a host copy of the symbols (S2BBToSoft::process onwards, module_dvbs2_demod.cpp:334-366) */
int dvbs2fec_decode_plframes_device(dvbs2fec_handle* h, const float* d_plframes, int n, uint8_t* d_bb_out,
                                    dvbs2fec_result* d_results, void* cuda_stream);
/* number of kernel launches the last decode_batch* / decode_*vcm* call on this handle enqueued */
int dvbs2fec_last_launch_count(const dvbs2fec_handle* h);
/* measurement aid: with profiling on, every kernel launch of decode_batch_device is bracketed by CUDA
 * events on its stream; kernel_times() waits for them and returns the summed device time per kernel
 * (ms) and the number of launches since the previous call.  VCM calls count their gather into demap_ms and their
 * scatter into bch_ms. */
int dvbs2fec_set_profiling(dvbs2fec_handle* h, int on);
int dvbs2fec_kernel_times(dvbs2fec_handle* h, float* demap_ms, float* ldpc_ms, float* bch_ms, int* launches);

/* ---- VCM / ACM: frames of different MODCOD, frame size and pilot setting in one call ----
 * desc holds four int32 per frame, laid out like the results of dvbs2fec_plhdr_process so that they can be passed
 * straight in: modcod (0..28), shortframes, pilots, and a fourth field that is ignored.  modcod 0 is a DUMMY PLFRAME:
 * 90 + 36 * 90 = 3330 symbols, no LLRs, no BBFRAME bytes; its result has ldpc_iters = 0, bch_corr = 0 and
 * DVBS2FEC_FLAG_DUMMY.  Any other frame without an LDPC code (modcod outside 0..28, short frames at rate 9/10) fails
 * the whole call with DVBS2FEC_EINVAL before anything is written; the error text names the frame.
 * Frames are packed back to back in input order: dvbs2fec_plframe_symbols(frame) complex floats, nldpc(frame) LLR
 * bytes and kbch(frame) / 8 BBFRAME bytes each (no alignment: normal 1/4 is 2001 bytes).  One result per frame,
 * tag = the frame's index in the call. */

/* n + 1 prefix offsets of that layout into each non-NULL array: sym_off in complex samples, llr_off and bb_off in
 * bytes.  Needs no handle or device. */
int dvbs2fec_vcm_layout(int n, const int32_t* desc, int64_t* sym_off, int64_t* llr_off, int64_t* bb_off);
/* dvbs2fec_decode_batch / dvbs2fec_decode_plframes for a VCM batch: host buffers, synchronous.  desc is in host memory
 * in all four calls (the host groups the frames by LDPC code and sizes the launches from it).  The calls use the
 * handle's max_trials and dvbs2fec_set_pl_scrambling setting (the PL descrambling sequence restarts at every frame),
 * run on the handle's first device, need no dvbs2fec_set_modcod and leave the configured MODCOD as it was.  A call
 * runs in chunks of at most max_batch frames; inside a chunk the frames of each LDPC code are decoded by one launch. */
int dvbs2fec_decode_vcm(dvbs2fec_handle* h, int n, const int32_t* desc, const int8_t* llr, uint8_t* bb_out,
                        dvbs2fec_result* results);
int dvbs2fec_decode_plframes_vcm(dvbs2fec_handle* h, int n, const int32_t* desc, const float* plframes, uint8_t* bb_out,
                                 dvbs2fec_result* results);
/* the same on device buffers, enqueued on `cuda_stream` and not synchronised, sharing the scratch and the ordering of
 * dvbs2fec_decode_batch_device */
int dvbs2fec_decode_vcm_device(dvbs2fec_handle* h, int n, const int32_t* desc, const int8_t* d_llr, uint8_t* d_bb_out,
                               dvbs2fec_result* d_results, void* cuda_stream);
int dvbs2fec_decode_plframes_vcm_device(dvbs2fec_handle* h, int n, const int32_t* desc, const float* d_plframes,
                                        uint8_t* d_bb_out, dvbs2fec_result* d_results, void* cuda_stream);

/* ---- frame-batching queue between PL sync and the decoder (replaces simd_packer,
 *      module_dvbs2_demod.cpp:343-347): frames come back in submission order ---- */
int dvbs2fec_submit_llr(dvbs2fec_handle* h, const int8_t* llr, uint64_t tag);
int dvbs2fec_submit_plframe(dvbs2fec_handle* h, const float* plframe, int nsym, uint64_t tag);
int dvbs2fec_submit_plframe_idx(dvbs2fec_handle* h, const uint8_t* idx, uint64_t tag);   /* see dvbs2fec_quantize_plframes */
/* Zero-copy submit: acquire hands out the place of the next frame inside the page-locked batch being filled
 * (nldpc bytes / plframe_symbols complex floats / 2 bytes per payload symbol), the producer -- the demapper, the
 * PLL loop, a socket read -- writes its output there instead of into a buffer of its own, commit queues it.  One
 * frame at a time per handle; the batch is not launched while a frame is being written.  Saves the copy of
 * submit_* (64.8 KB per normal frame), which is what limits a multi-GPU handle fed by few host threads. */
int dvbs2fec_acquire_llr(dvbs2fec_handle* h, int8_t** slot);
int dvbs2fec_acquire_plframe(dvbs2fec_handle* h, float** slot);
int dvbs2fec_acquire_plframe_idx(dvbs2fec_handle* h, uint8_t** slot);
int dvbs2fec_commit(dvbs2fec_handle* h, uint64_t tag);
/* up to max frames; bb_out receives kbch/8 bytes per frame.  timeout_us: 0 = poll, <0 = wait for one. */
int dvbs2fec_collect(dvbs2fec_handle* h, uint8_t* bb_out, dvbs2fec_result* results, int max, int timeout_us);
/* force the partial batch through (DVBS2Demod::reset / tempStop) */
int dvbs2fec_flush(dvbs2fec_handle* h);

/* Fused TS output (SURVEY 8(f) rank 1 behind the queue): with on != 0 the worker runs the BBFRAME -> TS kernels on
 * the device right behind the BCH kernel -- BBFrameTSParser::work (dvbs2/bbframe_ts_parser.cpp:100-212) as
 * main.cpp:538 applies it to the decoded frames, parser state running through all frames of the handle in
 * submission order and starting over at dvbs2fec_set_modcod like setFrameSize.  Single-device handles only.
 * Frames are then taken with dvbs2fec_collect_ts instead of dvbs2fec_collect. */
int dvbs2fec_set_ts_output(dvbs2fec_handle* h, int on);
/* TS packets of finished frames, in order: returns the bytes written (a multiple of 188, <= cap).  results
 * (optional, room for max_results records) receives one record per frame, in submission order, each batch's
 * records following its last packets (as many as fit; the rest with the next call); *nresults the count. */
int dvbs2fec_collect_ts(dvbs2fec_handle* h, uint8_t* ts_out, int cap, dvbs2fec_result* results, int max_results,
                        int* nresults, int timeout_us);

/* pinned host memory for zero-staging transfers (optional) */
void* dvbs2fec_alloc_pinned(size_t bytes);
void dvbs2fec_free_pinned(void* p);

/* ---- downstream of the decode stage: BBFRAME -> MPEG-TS packets (SURVEY.md 8(f) rank 1) ----
 * Mirrors BBFrameTSParser (dvbs2/bbframe_ts_parser.h:67-108) as main.cpp:538 uses it.  The parser is its own
 * object, like the reference's; its state (sync, unfinished packet, GSE reassembly) lives on the device between calls. */
typedef struct dvbs2fec_ts_parser dvbs2fec_ts_parser;
typedef struct dvbs2fec_bbheader { /* BBHeader (bbframe_ts_parser.h:37-65) */
    uint8_t ts_gs, sis_mis, ccm_acm, issyi, npd, ro, isi, sync;
    uint16_t upl, dfl, syncd, reserved;
} dvbs2fec_bbheader;
int dvbs2fec_ts_create(int device, dvbs2fec_ts_parser** out);
void dvbs2fec_ts_destroy(dvbs2fec_ts_parser* p);
/* BBFrameTSParser::setFrameSize (bbframe_ts_parser.cpp:31-43): kbch in bits; resets the parser state */
int dvbs2fec_ts_set_frame_size(dvbs2fec_ts_parser* p, int kbch_bits);
/* BBFrameTSParser::work (bbframe_ts_parser.cpp:100-392): cnt BBFRAMEs of kbch/8 bytes in; out come 188-byte packets
 * for TS frames (ts_gs = 11, :171-212) and GRE-wrapped PDUs for GSE frames (ts_gs = 01, :213-389: complete PDUs and
 * PDUs reassembled from Start/Continuation/End fragments in three FragID slots, CRC-32 checked), in frame order.
 * Returns the number of bytes written or a negative error.  Host buffers.  Where the reference is undefined the
 * call is defined: GSE packets whose lengths lead outside the input are reported (malformed) and end the walk of
 * their frame; a call with GSE frames whose output does not fit buffer_outsize returns DVBS2FEC_ENOSPC with nothing
 * written (the reference writes PDUs without a room test); >= 188 unconsumed bytes behind the TS room rule drop sync. */
int dvbs2fec_ts_work(dvbs2fec_ts_parser* p, const uint8_t* bbframes, int cnt, uint8_t* tsframes, int buffer_outsize);
/* same on device buffers (e.g. straight from dvbs2fec_decode_batch_device), asynchronous on `stream`;
 * d_produced (optional, device int) receives the byte count (DVBS2FEC_ENOSPC as above, also when the call holds
 * more GSE packets than the descriptor pool: see dvbs2fec_ts_set_gse) */
int dvbs2fec_ts_work_device(dvbs2fec_ts_parser* p, const uint8_t* d_bbframes, int cnt, uint8_t* d_tsframes,
                            int buffer_outsize, int* d_produced, void* stream);
/* GSE branch: max_packets_per_call < 0 -> GSE frames are accepted and counted but not unpacked; 0 (default) ->
 * unpacked, descriptor pool sized exactly (host-buffer call) or 64 packets per frame + 1024 (device-buffer call,
 * which cannot ask the device first); > 0 -> pool of that many packets for device-buffer calls.  The reassembly
 * state survives dvbs2fec_ts_set_frame_size like the reference's. */
int dvbs2fec_ts_set_gse(dvbs2fec_ts_parser* p, int max_packets_per_call);
/* last_gse_crc_err (bbframe_ts_parser.h:73) and counters of the last call that held GSE frames: PDUs delivered,
 * reassemblies that failed the CRC-32, frames with a malformed packet chain, fragments without a slot */
int dvbs2fec_ts_gse_stats(dvbs2fec_ts_parser* p, int* last_gse_crc_err, int* pdus, int* crc_errors, int* malformed,
                          int* dropped);
/* public members after work() (bbframe_ts_parser.h:72-76): last_header (returns 0 if no frame was accepted
 * yet, 1 otherwise), last_bb_cnt, last_bb_proc; gse_frames = accepted GSE frames in the last call */
int dvbs2fec_ts_stats(dvbs2fec_ts_parser* p, dvbs2fec_bbheader* last_header, int* last_bb_cnt, int* last_bb_proc,
                      int* gse_frames);

/* ---- upstream of the decode stage: PL frame synchronisation, PLHEADER demodulation, coarse frequency error
 *      (SURVEY.md 8(f) rank 3), as DVBS2Demod::process drives them per block of clock-recovered symbols
 *      (dvbs2/module_dvbs2_demod.cpp:300-316).  Complex symbols are interleaved float pairs (re, im).  One object
 *      holds the state of S2PLSyncBlock and S2PLHDRDemod of one demodulator; it lives on the device between calls. ---- */
typedef struct dvbs2fec_plsync dvbs2fec_plsync;
int dvbs2fec_plsync_create(int device, dvbs2fec_plsync** out);
void dvbs2fec_plsync_destroy(dvbs2fec_plsync* p);
/* S2PLSyncBlock::init / setParams (dvbs2/dvbs2_pl_sync.cpp:10-35,47-76): slots of 90 payload symbols per frame and
 * pilots -> raw_frame_size; the gathering state starts over.  reset (:37-45) only does the latter. */
int dvbs2fec_plsync_set_params(dvbs2fec_plsync* p, int slot_num, int pilots);
int dvbs2fec_plsync_reset(dvbs2fec_plsync* p);
int dvbs2fec_plsync_raw_frame_size(const dvbs2fec_plsync* p);
/* S2PLSyncBlock::process (dvbs2/dvbs2_pl_sync.cpp:80-165): count symbols in; every frame completed by them comes out,
 * raw_frame_size symbols each, starting at the position the PLHEADER correlator chose.  Returns the number of symbols
 * written (a multiple of raw_frame_size; out needs room for count + raw_frame_size).  Host buffers, synchronous. */
int dvbs2fec_plsync_process(dvbs2fec_plsync* p, int count, const float* in, float* out);
/* same on device buffers, asynchronous on `stream`: at most max_frames frames are written to d_out, their number to
 * d_nframes (optional device int) */
int dvbs2fec_plsync_process_device(dvbs2fec_plsync* p, int count, const float* d_in, float* d_out, int max_frames,
                                   int* d_nframes, void* stream);
/* public members after process (dvbs2_pl_sync.h:38-40): current_position, best_match; pending = symbols gathered
 * but not delivered yet.  Returns the frames the last call delivered. */
int dvbs2fec_plsync_stats(dvbs2fec_plsync* p, int* current_position, double* best_match, int* pending);
/* S2PLHDRDemod::init (dvbs2/dvbs2_plhdr_demod.cpp:5-12): loop bandwidth; phase and frequency start at 0 */
int dvbs2fec_plhdr_set_params(dvbs2fec_plsync* p, float loop_bw);
/* S2PLHDRDemod::process (dvbs2/dvbs2_plhdr_demod.cpp:33-67), once per frame in order: nframes frames of raw_frame_size
 * symbols in; headers = 90 phase-corrected header symbols per frame (what process() leaves in out[0..90));
 * results = four ints per frame: detect_modcod, detect_shortframes, detect_pilots, PLS index; loop_state (optional)
 * = phase and frequency of the loop after the last frame.  The sin/cos of the loop are evaluated on the device:
 * header symbols and loop state agree with the reference to float rounding (tests: 1e-4), the PLS fields exactly
 * wherever no header symbol lies within that distance of a decision boundary. */
int dvbs2fec_plhdr_process(dvbs2fec_plsync* p, int nframes, const float* frames, float* headers, int32_t* results,
                           float* loop_state);
int dvbs2fec_plhdr_process_device(dvbs2fec_plsync* p, int nframes, const float* d_frames, float* d_headers,
                                  int32_t* d_results, void* stream);
/* dvbs2_pilot_coarse_fed (dvbs2/dvbs2_fed.h:7-48) for nframes frames: one float per frame (what module_dvbs2_demod.cpp
 * :302 feeds back into the frequency shifter).  pls_code = PLS index of the configured MODCOD (S2PLLBlock::pls_code),
 * codenum = Gold code of the PL scrambler (pilot blocks are descrambled; ignored without pilots). */
int dvbs2fec_coarse_fed(dvbs2fec_plsync* p, int nframes, const float* frames, int pilots, int pls_code, int codenum,
                        float* err);
int dvbs2fec_coarse_fed_device(dvbs2fec_plsync* p, int nframes, const float* d_frames, int pilots, int pls_code,
                               int codenum, float* d_err, void* stream);

/* ---- the payload phase loop (SURVEY.md 8(f) rank 2): S2PLLBlock, between PL sync and the demapper
 *      (dvbs2/module_dvbs2_demod.cpp:332).  Part of the same object: it shares the PLHEADER tables and the PL
 *      scrambling sequence, and its state (pcl.phase, pcl.freq) lives on the device between calls. ---- */
/* S2PLLBlock::init + the members DVBS2Demod::init / setDemodParams set (dvbs2_pll.cpp:5-14, module_dvbs2_demod.cpp:59-65,
 * 146-151): loop bandwidth -> criticallyDamped coefficients, constellation of the MODCOD (with its phase-error table),
 * frame_slot_count, pls_code = modcod << 2 | shortframes << 1 | pilots, update() (pilot_cnt counted as the reference
 * counts it, dvbs2_pll.h:47-59); codenum = Gold code of the PL scrambler.  The loop state is kept (the reference
 * only re-creates the constellation); dvbs2fec_pll_reset zeroes phase and frequency (dvbs2_pll.cpp:16-23). */
int dvbs2fec_pll_set_params(dvbs2fec_plsync* p, float loop_bw, int modcod, int shortframes, int pilots, int codenum);
int dvbs2fec_pll_reset(dvbs2fec_plsync* p);
/* hand the loop a state (a host-side loop that ran so far, or a test): pcl.phase, pcl.freq */
int dvbs2fec_pll_set_state(dvbs2fec_plsync* p, float phase, float freq);
/* 0 (default): six warps take the blocks of 32 symbols in turn, each speculating its block from the state its predecessor
 * published a tick earlier; 1: walk the loop one symbol at a time in one thread, as the reference does (the yardstick: the
 * speculative kernels produce the same bits -- tests/test_gpu_pll.py -- and are several times faster); 2: one warp, block
 * after block (the first speculative kernel) */
int dvbs2fec_pll_set_sequential(dvbs2fec_plsync* p, int on);
/* symbols process() handles per frame: (frame_slot_count + 1) * 90 + pilot_cnt * 36 */
int dvbs2fec_pll_frame_symbols(const dvbs2fec_plsync* p);
/* S2PLLBlock::process (dvbs2_pll.cpp:34-86) for nframes consecutive frames of the stream, frame_stride symbols apart
 * (raw_frame_size as PL sync delivers them; at least dvbs2fec_pll_frame_symbols): derotated header symbols and
 * derotated, PL-descrambled payload symbols out, same stride; state (optional) = pcl.phase, pcl.freq and the block's
 * public `error` after every frame (3 floats each).  Returns nframes.  sin / cos / atan2 are the device's: symbols and
 * state agree with the reference to float rounding (tests: 2e-4), everything else is the reference's arithmetic. */
int dvbs2fec_pll_process(dvbs2fec_plsync* p, int nframes, int frame_stride, const float* frames, float* out, float* state);
/* same on device buffers, asynchronous on `stream`; d_state optional (3 floats per frame) */
int dvbs2fec_pll_process_device(dvbs2fec_plsync* p, int nframes, int frame_stride, const float* d_frames, float* d_out,
                                float* d_state, void* stream);
/* Several independent streams (transponders) in one launch, a CTA of six warps each: objs[k] processes nframes frames from
 * d_frames[k] into d_out[k] (device buffers, same frame_stride; all objects on the same device and configured).
 * Frames of one stream are a recurrence and cannot overlap; streams can. */
int dvbs2fec_pll_process_multi_device(int nstreams, dvbs2fec_plsync* const* objs, int nframes, int frame_stride,
                                      const float* const* d_frames, float* const* d_out, void* stream);
/* diagnostic: evaluation rounds the last call needed (two per block of 32 symbols is the minimum) */
int dvbs2fec_pll_rounds(dvbs2fec_plsync* p);

/* ---- the decode stage of the DVB-S2 module in one call: DVBS2Demod::process (dvbs2/module_dvbs2_demod.cpp:300-367) behind
 *      its sample-domain front end.  count clock-recovered symbols (re, im) -> PL sync -> per frame: coarse frequency
 *      error, payload phase loop (with PL descrambling), PLHEADER demodulation, demapper, LDPC, BCH, BB descrambler ->
 *      BBFRAMEs of kbch / 8 bytes, in stream order.  Symbols cross PCIe once; everything between them and the BBFRAMEs
 *      stays on the device, on one stream, stage after stage in the reference's order.  One device (a stream of symbols
 *      is a recurrence).  Left to the caller: feeding fed_err to its frequency shifter (:302-313).  Not reproduced: the
 *      module's wait for 16 frames before it decodes (SURVEY.md note N1) -- every frame a call completes is decoded by it. ---- */
typedef struct dvbs2fec_s2_demod dvbs2fec_s2_demod;
int dvbs2fec_s2_demod_create(const dvbs2fec_config* cfg, dvbs2fec_s2_demod** out);
void dvbs2fec_s2_demod_destroy(dvbs2fec_s2_demod* p);
/* DVBS2Demod::setDemodParams (:118-168) and the loop bandwidths / Gold code DVBS2Demod::init hands its blocks (:59-65);
 * the PL sync state starts over, the phase loops keep their state (as the reference's do) */
int dvbs2fec_s2_demod_set_params(dvbs2fec_s2_demod* p, int modcod, int shortframes, int pilots, int max_trials, float pll_loop_bw,
                                 float plhdr_loop_bw, int codenum);
/* S2PLSyncBlock::reset + S2PLLBlock::reset */
int dvbs2fec_s2_demod_reset(dvbs2fec_s2_demod* p);
int dvbs2fec_s2_demod_bbframe_bytes(const dvbs2fec_s2_demod* p);            /* kbch / 8 */
int dvbs2fec_s2_demod_max_frames(const dvbs2fec_s2_demod* p, int count);    /* frames a call with count symbols can complete */
/* returns the frames completed and decoded (<= max_frames, which must be at least dvbs2fec_s2_demod_max_frames(count));
 * bb_out: max_frames * kbch / 8 bytes; optional per frame: results, fed_err (dvbs2_pilot_coarse_fed's value), plhdr (four
 * ints: detect_modcod, detect_shortframes, detect_pilots, PLS index).  Host buffers, synchronous. */
int dvbs2fec_s2_demod_process(dvbs2fec_s2_demod* p, int count, const float* syms, uint8_t* bb_out, int max_frames,
                              dvbs2fec_result* results, float* fed_err, int32_t* plhdr);
/* the same with the BBFRAME parser behind it (BBFrameTSParser::work as main.cpp:538 calls it on the module's output; K6
 * on the device, its state kept in the handle): 188-byte TS packets / GRE-wrapped GSE PDUs out, at most ts_cap bytes (the
 * parser's buffer_outsize); returns the bytes written, *nframes (optional) = frames decoded.  The per-frame outputs are
 * optional; with any of them max_frames must be at least dvbs2fec_s2_demod_max_frames(count). */
int dvbs2fec_s2_demod_process_ts(dvbs2fec_s2_demod* p, int count, const float* syms, uint8_t* ts_out, int ts_cap, int max_frames,
                                 int* nframes, dvbs2fec_result* results, float* fed_err, int32_t* plhdr);

/* ---- DVB-S legacy chain, the byte-domain half (SURVEY.md 8(f) rank 4): the body of the frame loop of
 *      DVBSDemod::process (dvbs/module_dvbs_demod.cpp:91-106) -- convolutional deinterleaver
 *      (DVBSInterleaving::deinterleave, dvbs/dvbs_interleaving.h:57-70), eight RS(204,188) decodes (DVBSReedSolomon::decode,
 *      dvbs/dvbs_reedsolomon.h:27-47, over the vendored libcorrect), energy-dispersal descrambler
 *      (DVBSScrambling::descramble, dvbs/dvbs_scrambling.h:30-43), 8 x 188 bytes out -- for a batch of frames.
 *      One object holds what the three reference objects hold between frames (FIFO contents, the decoder's output
 *      buffer, the descrambler register); it lives on the device.  Bit-identical to the reference, its observable
 *      quirks included: a packet libcorrect gives up on comes out as the previous decoded packet, and errors[] is what
 *      DVBSReedSolomon::decode returns (bytes in which the received message differs from what comes out; never -1). ---- */
typedef struct dvbs2fec_dvbs_outer dvbs2fec_dvbs_outer;
int dvbs2fec_dvbs_outer_create(int device, dvbs2fec_dvbs_outer** out);
void dvbs2fec_dvbs_outer_destroy(dvbs2fec_dvbs_outer* p);
/* back to the state of freshly constructed objects */
int dvbs2fec_dvbs_outer_reset(dvbs2fec_dvbs_outer* p);
/* nframes frames of 8 x 204 bytes as the TS deframer delivers them; frame k starts at frames + k * frame_stride
 * (1632 for back-to-back frames; the reference module itself steps by 204, module_dvbs_demod.cpp:91 -- give it that
 * to reproduce it), so frames must hold (nframes - 1) * frame_stride + 1632 bytes.  out: nframes * 8 * 188 bytes of TS
 * packets; errors (optional): nframes * 8 ints.  Returns the bytes written.  Host buffers, synchronous. */
int dvbs2fec_dvbs_outer_process(dvbs2fec_dvbs_outer* p, int nframes, int frame_stride, const uint8_t* frames, uint8_t* out,
                                int32_t* errors);
/* same on device buffers, asynchronous on `stream` */
int dvbs2fec_dvbs_outer_process_device(dvbs2fec_dvbs_outer* p, int nframes, int frame_stride, const uint8_t* d_frames,
                                       uint8_t* d_out, int32_t* d_errors, void* stream);

/* ---- K10: DVBS_TS_Deframer::work (dvbs/dvbs_ts_deframer.cpp:44-101, dvbs_ts_deframer.h:17-70; the module calls it
 *      through DVBSDefra::process, dvbs/dvbs_defra.cpp:5-9).  Input: the Viterbi decoder's output, one bit per byte;
 *      output: every window of 8 x 204 x 8 bits whose eight sync bytes differ from B8 47 47 47 47 47 47 47 in at most 8
 *      bits, as a frame of 1632 bytes (inverted where the inverted pattern matched), in stream order.  The window persists
 *      over calls (it starts from zeros; the reference's is allocated uninitialised).  Every window position is tested
 *      at once on the device; bit-identical to the reference. ---- */
typedef struct dvbs2fec_dvbs_deframer dvbs2fec_dvbs_deframer;
int dvbs2fec_dvbs_deframer_create(int device, dvbs2fec_dvbs_deframer** out);
void dvbs2fec_dvbs_deframer_destroy(dvbs2fec_dvbs_deframer* p);
int dvbs2fec_dvbs_deframer_reset(dvbs2fec_dvbs_deframer* p);
/* size bits (< 2^24) -> at most max_frames frames of 1632 bytes; returns the number of frames written (the reference
 * writes all it finds: give max_frames >= the frames the call can hold to reproduce it).  Host buffers, synchronous. */
int dvbs2fec_dvbs_deframer_work(dvbs2fec_dvbs_deframer* p, const uint8_t* bits, int size, uint8_t* frames, int max_frames);
/* same on device buffers (d_frames 4-byte aligned), asynchronous on `stream`; the count goes to *d_nframes (optional) */
int dvbs2fec_dvbs_deframer_work_device(dvbs2fec_dvbs_deframer* p, const uint8_t* d_bits, int size, uint8_t* d_frames,
                                       int max_frames, int32_t* d_nframes, void* stream);
/* the public members errors_nor / errors_inv (dvbs_ts_deframer.h:24-25) after the last call, the frames it found
 * (before max_frames); returns the frames it wrote.  Synchronises the device. */
int dvbs2fec_dvbs_deframer_stats(dvbs2fec_dvbs_deframer* p, int* errors_nor, int* errors_inv, int* found);

/* ---- K11: the inner decoder of the DVB-S chain -- DVBSVitBlock::process (dvbs/dvbs_vit.cpp:6-13) over
 *      viterbi::Viterbi_DVBS (dvbs/viterbi_all.h:33-163, viterbi_all.cpp:75-318) as the module constructs it
 *      (module_dvbs_demod.cpp:23: phases 0 and 90 degrees, 8192 soft bits per work() call; ber_threshold 0.15 and
 *      max_outsync 20 there), and DVBSymToSoftBlock::process (dvbs/dvbs_syms_to_soft.cpp:26-42) in front of it.
 *      Self-locking punctured K = 7 decoder: searches rate (1/2, 2/3, 3/4, 5/6, 7/8), constellation phase and puncturing
 *      shift by decoding + re-encoding 2048 soft bits on every candidate, then decodes block after block until max_outsync
 *      blocks in a row fail the BER test.  All blocks of a call are decoded at once on the device; decoded bits, BER and
 *      lock parameters are bit-identical to the reference running its bundled generic butterfly kernel
 *      (dvbs/viterbi/volk_k7_r2_generic_fixed.h), its quirks included (see csrc/dvbs_viterbi.cu).  The members the
 *      reference reads before writing them start from zeros. ---- */
typedef struct dvbs2fec_dvbs_viterbi dvbs2fec_dvbs_viterbi;
int dvbs2fec_dvbs_viterbi_create(int device, float ber_threshold, int max_outsync, dvbs2fec_dvbs_viterbi** out);
void dvbs2fec_dvbs_viterbi_destroy(dvbs2fec_dvbs_viterbi* v);
int dvbs2fec_dvbs_viterbi_reset(dvbs2fec_dvbs_viterbi* v);
/* count signed soft bits (a multiple of 8192; the reference reads past its input otherwise) -> decoded bits, one per
 * byte; returns how many (0 while searching).  out must hold count bytes; bytes the reference leaves unwritten (27 of
 * every 6826 at rate 5/6) keep the caller's content.  Unlike the reference the input is not rotated in place.  Host
 * buffers, synchronous. */
int dvbs2fec_dvbs_viterbi_process(dvbs2fec_dvbs_viterbi* v, int count, const int8_t* in, uint8_t* out);
/* same on device buffers (no PCIe traffic but the per-block BER counts); synchronous: the lock state machine runs on the host.
 * The work runs on a stream of the handle's: d_in must be complete when the call is made, d_out is complete when it returns.
 * A handle is used by one thread at a time (as the reference's object is). */
int dvbs2fec_dvbs_viterbi_process_device(dvbs2fec_dvbs_viterbi* v, int count, const int8_t* d_in, uint8_t* d_out);
/* Viterbi_DVBS::ber(), getState() (0 searching, 1 locked), rate() (0..4 = 1/2, 2/3, 3/4, 5/6, 7/8) and the lock's phase
 * (0 / 1 = 0 / 90 degrees), puncturing shift and count of bad blocks; any pointer may be NULL */
int dvbs2fec_dvbs_viterbi_stats(dvbs2fec_dvbs_viterbi* v, float* ber, int* state, int* rate, int* phase, int* shift, int* invalid);
/* diagnostics since create: decode tasks run (one per block when locked, 52 per block while searching), tasks that had to
 * be repeated because the start state guessed for them was not the one their predecessor reached, check passes, and
 * tracebacks whose 32 parallel pieces did not join up and were walked step by step instead */
int dvbs2fec_dvbs_viterbi_counters(dvbs2fec_dvbs_viterbi* v, long long* tasks, long long* repeated, long long* passes, long long* walks);
/* DVBSymToSoftBlock::process: count symbols (re, im) -> clamp(re * 100), clamp(im * 100) in chunks of 8192 soft bits; what
 * does not fill a chunk waits in the handle; returns the soft bits written (out: 2 * count + 8192 bytes) */
int dvbs2fec_dvbs_sts_process(dvbs2fec_dvbs_viterbi* v, int count, const float* syms, int8_t* out);
int dvbs2fec_dvbs_sts_process_device(dvbs2fec_dvbs_viterbi* v, int count, const float* d_syms, int8_t* d_out);

/* ---- the decode stage of the DVB-S module in one call: DVBSDemod::process (dvbs/module_dvbs_demod.cpp:78-119) behind its
 *      sample-domain front end (demod.process, SDR++ DSP: not part of this library).  count complex symbols (re, im) ->
 *      soft bits -> Viterbi (K11) -> TS deframer (K10) -> deinterleaver / RS(204,188) / descrambler (K9) -> TS packets of
 *      188 bytes; every intermediate buffer stays on the device.  frame_stride: 204 walks the deframer's frames the way
 *      the module does (module_dvbs_demod.cpp:87 steps by 204 bytes instead of 1632), 1632 takes them back to back.
 *      Returns the TS bytes written (a multiple of 1504) or DVBS2FEC_ENOSPC.  At most nbits / 1632 + 8 frames per call are
 *      taken from the deframer (it finds one per 13056 bits in a stream that is not built to fool it); frames_found tells. ---- */
typedef struct dvbs2fec_dvbs_demod dvbs2fec_dvbs_demod;
int dvbs2fec_dvbs_demod_create(int device, float ber_threshold, int max_outsync, int frame_stride, dvbs2fec_dvbs_demod** out);
void dvbs2fec_dvbs_demod_destroy(dvbs2fec_dvbs_demod* p);
int dvbs2fec_dvbs_demod_reset(dvbs2fec_dvbs_demod* p);
int dvbs2fec_dvbs_demod_process(dvbs2fec_dvbs_demod* p, int count, const float* syms, uint8_t* out, int out_cap);
/* stats_viterbi_ber / _lock / _rate (0..4), stats_rs_avg, stats_deframer_err (module_dvbs_demod.cpp:101-115) and the frames
 * the deframer found / the call decoded; any pointer may be NULL */
int dvbs2fec_dvbs_demod_stats(dvbs2fec_dvbs_demod* p, float* viterbi_ber, int* viterbi_lock, int* viterbi_rate, float* rs_avg,
                              int* deframer_err, int* frames_found, int* frames_done);

/* ---- in-tree transmitter for synthetic input (not part of the reference's decode path) ---- */
/* bbframe: kbch/8 bytes -> code_bits: N bytes of 0/1 (BB scramble, BCH, LDPC; EN 302 307 5.2-5.3) */
int dvbs2fec_encode_fecframe(int modcod, int shortframes, const uint8_t* bbframe, uint8_t* code_bits);
/* code_bits -> PLFRAME symbols (90 zero header symbols, bit interleave, mapping; pilots as 0+0j) */
int dvbs2fec_modulate(int modcod, int shortframes, int pilots, const uint8_t* code_bits, float* plframe);
/* static facts about a MODCOD: returns 0 or DVBS2FEC_EINVAL */
int dvbs2fec_modcod_info(int modcod, int shortframes, int pilots, int* nldpc, int* kldpc, int* kbch, int* bch_t,
                         int* bits_per_symbol, int* plframe_symbols, int* links_total);

#ifdef __cplusplus
}
#endif
#endif /* DVBS2FEC_H */
