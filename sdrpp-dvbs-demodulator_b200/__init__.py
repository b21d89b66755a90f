"""Host-side mirror of the SDR++ dvbs_demodulator decode-stage objects over libdvbs2fec.so.

The compute path is the CUDA library only (csrc/, built in-tree for sm_100a by ``build()``); this
module is a thin ctypes binding whose class and method names follow the reference objects that
``DVBS2Demod::process`` drives (src/demod/dvbs2/module_dvbs2_demod.cpp:334-367):

    S2BBToSoft.process        dvbs2/dvbs2_bb_to_soft.h:19
    BBFrameLDPC.decode        dvbs2/codings/bbframe_ldpc.h:48-53
    BBFrameBCH.decode         dvbs2/codings/bbframe_bch.h:81-85
    BBFrameDescrambler.work   dvbs2/codings/bbframe_descramble.h:42
    DVBS2Decoder              the whole stage (setDemodParams + batch decode + queue)

There is no CPU fallback: if the shared library is missing or no B200 is visible every call raises.
The directory name contains hyphens; import it with ``importlib.import_module("sdrpp-dvbs-demodulator_b200")``.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdvbs2fec.so")
INCLUDE = os.path.join(os.path.dirname(_HERE), "include", "dvbs2fec.h")

EINVAL, ENODEV, ECUDA, EAGAIN, ENOSPC = -22, -19, -5, -11, -28
FLAG_LDPC_FAIL, FLAG_BCH_FAIL, FLAG_BBHEADER_CRC_FAIL, FLAG_DUMMY = 1, 2, 4, 8

# reference dvbs2_code_rate_t numbering (dvbs2/dvbs2.h:11-25)
RATE_NAMES = {0: "1/4", 1: "1/3", 2: "2/5", 3: "1/2", 4: "3/5", 5: "2/3", 6: "3/4", 7: "4/5", 8: "5/6", 10: "8/9", 11: "9/10"}


class DVBS2FecError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("dvbs2fec error %d: %s" % (code, msg))
        self.code = code


class Config(C.Structure):
    _fields_ = [("n_devices", C.c_int32), ("devices", C.c_int32 * 8), ("max_batch", C.c_int32),
                ("max_latency_us", C.c_int32), ("max_trials", C.c_int32), ("reserved", C.c_int32 * 4)]


class BBHeader(C.Structure):
    """dvbs2fec_bbheader == BBHeader (dvbs2/bbframe_ts_parser.h:37-65)"""
    _fields_ = [(n, C.c_uint8) for n in ("ts_gs", "sis_mis", "ccm_acm", "issyi", "npd", "ro", "isi", "sync")] + \
               [(n, C.c_uint16) for n in ("upl", "dfl", "syncd", "reserved")]


class Result(C.Structure):
    _fields_ = [("tag", C.c_uint64), ("ldpc_iters", C.c_int16), ("bch_corr", C.c_int16), ("flags", C.c_uint32)]


RESULT_DTYPE = np.dtype([("tag", np.uint64), ("ldpc_iters", np.int16), ("bch_corr", np.int16), ("flags", np.uint32)])

_lib = None


def build(verbose=False):
    """Compile libdvbs2fec.so for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    out = None if verbose else subprocess.DEVNULL
    subprocess.check_call(["make", "-C", _HERE, "-j8"], stdout=out)
    return LIB_PATH


def lib():
    """The loaded C-ABI library.  Raises if it has not been built -- there is nothing to fall back to."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DVBS2FecError(ENODEV, "%s is missing: run build() / `make -C %s` first" % (LIB_PATH, _HERE))
    L = C.CDLL(LIB_PATH)
    vp, ip = C.c_void_p, C.POINTER(C.c_int)
    L.dvbs2fec_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.dvbs2fec_destroy.argtypes = [vp]
    L.dvbs2fec_destroy.restype = None
    L.dvbs2fec_last_error.restype = C.c_char_p
    L.dvbs2fec_set_modcod.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int]
    for f in ("dvbs2fec_kbch", "dvbs2fec_kldpc", "dvbs2fec_nldpc", "dvbs2fec_plframe_symbols", "dvbs2fec_last_launch_count",
              "dvbs2fec_flush"):
        getattr(L, f).argtypes = [vp]
    L.dvbs2fec_bb_to_soft.argtypes = [vp, vp, C.c_int, vp]
    L.dvbs2fec_ldpc_decode.argtypes = [vp, vp, C.c_int, C.c_int, vp]
    L.dvbs2fec_bch_decode.argtypes = [vp, vp, C.c_int, vp]
    L.dvbs2fec_descramble.argtypes = [vp, vp, C.c_int, C.c_int]
    L.dvbs2fec_decode_batch.argtypes = [vp, vp, C.c_int, vp, vp]
    L.dvbs2fec_decode_plframes.argtypes = [vp, vp, C.c_int, vp, vp]
    L.dvbs2fec_decode_batch_device.argtypes = [vp, vp, C.c_int, vp, vp, vp]
    L.dvbs2fec_decode_plframes_device.argtypes = [vp, vp, C.c_int, vp, vp, vp]
    L.dvbs2fec_quantize_plframes.argtypes = [vp, vp, C.c_int, vp]
    L.dvbs2fec_decode_plframes_idx.argtypes = [vp, vp, C.c_int, vp, vp]
    L.dvbs2fec_submit_plframe_idx.argtypes = [vp, vp, C.c_uint64]
    for f in ("dvbs2fec_acquire_llr", "dvbs2fec_acquire_plframe", "dvbs2fec_acquire_plframe_idx"):
        getattr(L, f).argtypes = [vp, C.POINTER(vp)]
    L.dvbs2fec_commit.argtypes = [vp, C.c_uint64]
    L.dvbs2fec_set_profiling.argtypes = [vp, C.c_int]
    L.dvbs2fec_kernel_times.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float), ip]
    L.dvbs2fec_submit_llr.argtypes = [vp, vp, C.c_uint64]
    L.dvbs2fec_submit_plframe.argtypes = [vp, vp, C.c_int, C.c_uint64]
    L.dvbs2fec_collect.argtypes = [vp, vp, vp, C.c_int, C.c_int]
    L.dvbs2fec_alloc_pinned.argtypes = [C.c_size_t]
    L.dvbs2fec_alloc_pinned.restype = vp
    L.dvbs2fec_free_pinned.argtypes = [vp]
    L.dvbs2fec_free_pinned.restype = None
    L.dvbs2fec_encode_fecframe.argtypes = [C.c_int, C.c_int, vp, vp]
    L.dvbs2fec_modulate.argtypes = [C.c_int, C.c_int, C.c_int, vp, vp]
    L.dvbs2fec_modcod_info.argtypes = [C.c_int, C.c_int, C.c_int, ip, ip, ip, ip, ip, ip, ip]
    L.dvbs2fec_set_pl_scrambling.argtypes = [vp, C.c_int]
    L.dvbs2fec_set_ts_output.argtypes = [vp, C.c_int]
    L.dvbs2fec_collect_ts.argtypes = [vp, vp, C.c_int, vp, C.c_int, ip, C.c_int]
    L.dvbs2fec_ts_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.dvbs2fec_ts_destroy.argtypes = [vp]
    L.dvbs2fec_ts_destroy.restype = None
    L.dvbs2fec_ts_set_frame_size.argtypes = [vp, C.c_int]
    L.dvbs2fec_ts_work.argtypes = [vp, vp, C.c_int, vp, C.c_int]
    L.dvbs2fec_ts_work_device.argtypes = [vp, vp, C.c_int, vp, C.c_int, vp, vp]
    L.dvbs2fec_ts_stats.argtypes = [vp, C.POINTER(BBHeader), ip, ip, ip]
    L.dvbs2fec_ts_set_gse.argtypes = [vp, C.c_int]
    L.dvbs2fec_ts_gse_stats.argtypes = [vp, ip, ip, ip, ip, ip]
    L.dvbs2fec_plsync_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.dvbs2fec_plsync_destroy.argtypes = [vp]
    L.dvbs2fec_plsync_destroy.restype = None
    L.dvbs2fec_plsync_set_params.argtypes = [vp, C.c_int, C.c_int]
    L.dvbs2fec_plsync_reset.argtypes = [vp]
    L.dvbs2fec_plsync_raw_frame_size.argtypes = [vp]
    L.dvbs2fec_plsync_process.argtypes = [vp, C.c_int, vp, vp]
    L.dvbs2fec_plsync_process_device.argtypes = [vp, C.c_int, vp, vp, C.c_int, vp, vp]
    L.dvbs2fec_plsync_stats.argtypes = [vp, ip, C.POINTER(C.c_double), ip]
    L.dvbs2fec_plhdr_set_params.argtypes = [vp, C.c_float]
    L.dvbs2fec_plhdr_process.argtypes = [vp, C.c_int, vp, vp, vp, vp]
    L.dvbs2fec_plhdr_process_device.argtypes = [vp, C.c_int, vp, vp, vp, vp]
    L.dvbs2fec_coarse_fed.argtypes = [vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, vp]
    L.dvbs2fec_coarse_fed_device.argtypes = [vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, vp, vp]
    L.dvbs2fec_pll_set_params.argtypes = [vp, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int]
    L.dvbs2fec_pll_reset.argtypes = [vp]
    L.dvbs2fec_pll_frame_symbols.argtypes = [vp]
    L.dvbs2fec_pll_process.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp]
    L.dvbs2fec_pll_process_device.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, vp]
    L.dvbs2fec_pll_rounds.argtypes = [vp]
    L.dvbs2fec_dvbs_outer_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.dvbs2fec_dvbs_outer_destroy.argtypes = [vp]
    L.dvbs2fec_dvbs_outer_destroy.restype = None
    L.dvbs2fec_dvbs_outer_reset.argtypes = [vp]
    L.dvbs2fec_dvbs_outer_process.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp]
    L.dvbs2fec_dvbs_outer_process_device.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, vp]
    L.dvbs2fec_dvbs_deframer_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.dvbs2fec_dvbs_deframer_destroy.argtypes = [vp]
    L.dvbs2fec_dvbs_deframer_destroy.restype = None
    L.dvbs2fec_dvbs_deframer_reset.argtypes = [vp]
    L.dvbs2fec_dvbs_deframer_work.argtypes = [vp, vp, C.c_int, vp, C.c_int]
    L.dvbs2fec_dvbs_deframer_work_device.argtypes = [vp, vp, C.c_int, vp, C.c_int, vp, vp]
    L.dvbs2fec_dvbs_deframer_stats.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.dvbs2fec_dvbs_viterbi_create.argtypes = [C.c_int, C.c_float, C.c_int, C.POINTER(vp)]
    L.dvbs2fec_dvbs_viterbi_destroy.argtypes = [vp]
    L.dvbs2fec_dvbs_viterbi_destroy.restype = None
    L.dvbs2fec_dvbs_viterbi_reset.argtypes = [vp]
    L.dvbs2fec_dvbs_viterbi_process.argtypes = [vp, C.c_int, vp, vp]
    L.dvbs2fec_dvbs_viterbi_process_device.argtypes = [vp, C.c_int, vp, vp]
    L.dvbs2fec_dvbs_viterbi_stats.argtypes = [vp, C.POINTER(C.c_float)] + [C.POINTER(C.c_int)] * 5
    L.dvbs2fec_dvbs_viterbi_counters.argtypes = [vp] + [C.POINTER(C.c_longlong)] * 4
    L.dvbs2fec_dvbs_sts_process.argtypes = [vp, C.c_int, vp, vp]
    L.dvbs2fec_dvbs_sts_process_device.argtypes = [vp, C.c_int, vp, vp]
    L.dvbs2fec_s2_demod_create.argtypes = [vp, C.POINTER(vp)]
    L.dvbs2fec_s2_demod_destroy.argtypes = [vp]
    L.dvbs2fec_s2_demod_destroy.restype = None
    L.dvbs2fec_s2_demod_set_params.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int]
    L.dvbs2fec_s2_demod_reset.argtypes = [vp]
    L.dvbs2fec_s2_demod_bbframe_bytes.argtypes = [vp]
    L.dvbs2fec_s2_demod_max_frames.argtypes = [vp, C.c_int]
    L.dvbs2fec_s2_demod_process.argtypes = [vp, C.c_int, vp, vp, C.c_int, vp, vp, vp]
    L.dvbs2fec_s2_demod_process_ts.argtypes = [vp, C.c_int, vp, vp, C.c_int, C.c_int, C.POINTER(C.c_int), vp, vp, vp]
    L.dvbs2fec_dvbs_demod_create.argtypes = [C.c_int, C.c_float, C.c_int, C.c_int, C.POINTER(vp)]
    L.dvbs2fec_dvbs_demod_destroy.argtypes = [vp]
    L.dvbs2fec_dvbs_demod_destroy.restype = None
    L.dvbs2fec_dvbs_demod_reset.argtypes = [vp]
    L.dvbs2fec_dvbs_demod_process.argtypes = [vp, C.c_int, vp, vp, C.c_int]
    L.dvbs2fec_dvbs_demod_stats.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_float),
                                            C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.dvbs2fec_pll_set_state.argtypes = [vp, C.c_float, C.c_float]
    L.dvbs2fec_pll_set_sequential.argtypes = [vp, C.c_int]
    L.dvbs2fec_pll_process_multi_device.argtypes = [C.c_int, vp, C.c_int, C.c_int, vp, vp, vp]
    L.dvbs2fec_vcm_layout.argtypes = [C.c_int, vp, vp, vp, vp]
    L.dvbs2fec_decode_vcm.argtypes = [vp, C.c_int, vp, vp, vp, vp]
    L.dvbs2fec_decode_plframes_vcm.argtypes = [vp, C.c_int, vp, vp, vp, vp]
    L.dvbs2fec_decode_vcm_device.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp]
    L.dvbs2fec_decode_plframes_vcm_device.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp]
    _lib = L
    return L


def _check(rc):
    if rc < 0:
        raise DVBS2FecError(rc, lib().dvbs2fec_last_error().decode(errors="replace"))
    return rc


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def modcod_info(modcod, shortframes=False, pilots=False):
    """MODCOD facts (get_dvbs2_cfg, codings/modcod_to_cfg.cpp:5-140, plus code parameters)."""
    v = [C.c_int() for _ in range(7)]
    _check(lib().dvbs2fec_modcod_info(modcod, int(shortframes), int(pilots), *[C.byref(x) for x in v]))
    keys = ("nldpc", "kldpc", "kbch", "bch_t", "bits", "plframe_symbols", "links_total")
    return dict(zip(keys, (x.value for x in v)))


def encode_fecframe(modcod, shortframes, bbframe):
    """In-tree transmitter: kbch/8 payload bytes -> N code bits (uint8 0/1)."""
    info = modcod_info(modcod, shortframes)
    bb = np.ascontiguousarray(bbframe, np.uint8)
    assert bb.size == info["kbch"] // 8
    out = np.zeros(info["nldpc"], np.uint8)
    _check(lib().dvbs2fec_encode_fecframe(modcod, int(shortframes), _ptr(bb), _ptr(out)))
    return out


def modulate(modcod, shortframes, pilots, code_bits):
    """In-tree transmitter: N code bits -> PLFRAME complex64 (header and pilots left at 0)."""
    info = modcod_info(modcod, shortframes, pilots)
    bits = np.ascontiguousarray(code_bits, np.uint8)
    out = np.zeros(info["plframe_symbols"] * 2, np.float32)
    _check(lib().dvbs2fec_modulate(modcod, int(shortframes), int(pilots), _ptr(bits), _ptr(out)))
    return out.view(np.complex64)


def _vcm_desc(desc):
    """frame descriptors as dvbs2fec_plhdr_process returns them: int32 [n][4] = modcod, shortframes, pilots, (ignored)"""
    return np.ascontiguousarray(desc, np.int32).reshape(-1, 4)


def vcm_layout(desc):
    """packed layout of a VCM batch: (sym_off, llr_off, bb_off), n + 1 int64 prefix offsets each -- complex samples of
    the PLFRAMEs, LLR bytes, BBFRAME bytes.  Raises DVBS2FecError (EINVAL) on a descriptor without a code."""
    d = _vcm_desc(desc)
    offs = [np.zeros(len(d) + 1, np.int64) for _ in range(3)]
    _check(lib().dvbs2fec_vcm_layout(len(d), _ptr(d), *[_ptr(o) for o in offs]))
    return tuple(offs)


class DVBS2Decoder:
    """One decode-stage instance (== one DVBS2Demod's FEC objects).  ``devices`` shards every batch by frame."""

    def __init__(self, devices=None, max_batch=1024, max_latency_us=2000, max_trials=25):
        cfg = Config()
        if devices:
            cfg.n_devices = len(devices)
            for i, d in enumerate(devices):
                cfg.devices[i] = d
        cfg.max_batch, cfg.max_latency_us, cfg.max_trials = max_batch, max_latency_us, max_trials
        self._h = C.c_void_p()
        _check(lib().dvbs2fec_create(C.byref(cfg), C.byref(self._h)))
        self.configured = False

    def close(self):
        if getattr(self, "_h", None):
            lib().dvbs2fec_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # DVBS2Demod::setDemodParams (module_dvbs2_demod.h:60)
    def setDemodParams(self, modcod, shortframes=False, pilots=False, max_ldpc_trials=0):
        _check(lib().dvbs2fec_set_modcod(self._h, modcod, int(shortframes), int(pilots), max_ldpc_trials))
        self.modcod, self.shortframes, self.pilots = modcod, bool(shortframes), bool(pilots)
        self.N = lib().dvbs2fec_nldpc(self._h)
        self.K = lib().dvbs2fec_kldpc(self._h)
        self.kbch = lib().dvbs2fec_kbch(self._h)
        self.plframe_symbols = lib().dvbs2fec_plframe_symbols(self._h)
        self.configured = True
        return self

    set_modcod = setDemodParams

    def set_pl_scrambling(self, codenum):
        """S2Scrambling(codenum) inside the demapper; -1: PLFRAMEs arrive descrambled (default)"""
        _check(lib().dvbs2fec_set_pl_scrambling(self._h, codenum))

    def getKBCH(self):
        return self.kbch

    # ---- stage-level (host numpy arrays) ----
    def bb_to_soft(self, plframes):
        x = np.ascontiguousarray(plframes).view(np.float32).reshape(-1, self.plframe_symbols * 2)
        out = np.zeros((x.shape[0], self.N), np.int8)
        _check(lib().dvbs2fec_bb_to_soft(self._h, _ptr(x), x.shape[0], _ptr(out)))
        return out

    def ldpc_decode(self, frames, max_trials=0):
        """frames: (n, N) int8, decoded IN PLACE like BBFrameLDPC::decode; returns int16 iterations per frame."""
        assert frames.dtype == np.int8 and frames.flags.c_contiguous and frames.shape[-1] == self.N
        n = frames.size // self.N
        iters = np.zeros(n, np.int16)
        _check(lib().dvbs2fec_ldpc_decode(self._h, _ptr(frames), n, max_trials, _ptr(iters)))
        return iters

    def bch_decode(self, frames):
        """frames: (n, K/8) uint8 corrected IN PLACE like BBFrameBCH::decode; returns int16 corrections per frame."""
        assert frames.dtype == np.uint8 and frames.flags.c_contiguous and frames.shape[-1] == self.K // 8
        n = frames.size // (self.K // 8)
        corr = np.zeros(n, np.int16)
        _check(lib().dvbs2fec_bch_decode(self._h, _ptr(frames), n, _ptr(corr)))
        return corr

    def descramble(self, frames):
        assert frames.dtype == np.uint8 and frames.flags.c_contiguous and frames.ndim == 2
        _check(lib().dvbs2fec_descramble(self._h, _ptr(frames), frames.shape[1], frames.shape[0]))
        return frames

    # ---- whole stage ----
    def decode_batch(self, llr):
        x = np.ascontiguousarray(llr, np.int8).reshape(-1, self.N)
        bb = np.zeros((x.shape[0], self.kbch // 8), np.uint8)
        res = np.zeros(x.shape[0], RESULT_DTYPE)
        _check(lib().dvbs2fec_decode_batch(self._h, _ptr(x), x.shape[0], _ptr(bb), _ptr(res)))
        return bb, res

    def decode_plframes(self, plframes):
        x = np.ascontiguousarray(plframes).view(np.float32).reshape(-1, self.plframe_symbols * 2)
        bb = np.zeros((x.shape[0], self.kbch // 8), np.uint8)
        res = np.zeros(x.shape[0], RESULT_DTYPE)
        _check(lib().dvbs2fec_decode_plframes(self._h, _ptr(x), x.shape[0], _ptr(bb), _ptr(res)))
        return bb, res

    def quantize_plframes(self, plframes):
        """PLFRAME symbols -> two LUT coordinates per payload symbol (uint8 [n][N / bits][2]), on the host"""
        x = np.ascontiguousarray(plframes).view(np.float32).reshape(-1, self.plframe_symbols * 2)
        nsym = self.N // modcod_info(self.modcod, self.shortframes)["bits"]
        out = np.zeros((x.shape[0], nsym, 2), np.uint8)
        _check(lib().dvbs2fec_quantize_plframes(self._h, _ptr(x), x.shape[0], _ptr(out)))
        return out

    def decode_plframes_idx(self, idx):
        x = np.ascontiguousarray(idx, np.uint8)
        n = x.shape[0]
        bb = np.zeros((n, self.kbch // 8), np.uint8)
        res = np.zeros(n, RESULT_DTYPE)
        _check(lib().dvbs2fec_decode_plframes_idx(self._h, _ptr(x), n, _ptr(bb), _ptr(res)))
        return bb, res

    def acquire_llr(self):
        """zero-copy submit: a writable int8 view of the next frame's place in the page-locked batch; commit(tag) queues it"""
        p = C.c_void_p()
        _check(lib().dvbs2fec_acquire_llr(self._h, C.byref(p)))
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_int8)), shape=(self.N,))

    def commit(self, tag=0):
        _check(lib().dvbs2fec_commit(self._h, tag))

    def submit_plframe_idx(self, idx, tag=0):
        x = np.ascontiguousarray(idx, np.uint8)
        _check(lib().dvbs2fec_submit_plframe_idx(self._h, _ptr(x), tag))

    def decode_batch_raw(self, llr_ptr, n, bb_ptr, res_ptr):
        """Host pointers (e.g. pinned buffers); synchronous."""
        _check(lib().dvbs2fec_decode_batch(self._h, llr_ptr, n, bb_ptr, res_ptr))

    def decode_batch_device(self, d_llr_ptr, n, d_bb_ptr, d_res_ptr, stream_ptr=0):
        """Device pointers on this decoder's first device; enqueues on ``stream_ptr`` and returns."""
        _check(lib().dvbs2fec_decode_batch_device(self._h, d_llr_ptr, n, d_bb_ptr, d_res_ptr, stream_ptr))

    def decode_plframes_device(self, d_plframes_ptr, n, d_bb_ptr, d_res_ptr, stream_ptr=0):
        """PLFRAME symbols on the device (plframe_symbols complex floats per frame) -> BBFRAMEs on the device"""
        _check(lib().dvbs2fec_decode_plframes_device(self._h, d_plframes_ptr, n, d_bb_ptr, d_res_ptr, stream_ptr))

    # ---- VCM / ACM batches: any MODCOD, frame size and pilot setting per frame (no setDemodParams needed) ----
    def decode_vcm(self, desc, llr):
        """desc: int32 [n][4] (modcod 0 = DUMMY PLFRAME); llr: the frames' LLRs packed back to back (vcm_layout).
        -> (packed BBFRAME bytes, bb_off [n + 1], results [n])"""
        d = _vcm_desc(desc)
        _, llr_off, bb_off = vcm_layout(d)
        x = np.ascontiguousarray(llr, np.int8).reshape(-1)
        assert x.size == llr_off[-1], (x.size, llr_off[-1])
        bb = np.zeros(bb_off[-1], np.uint8)
        res = np.zeros(len(d), RESULT_DTYPE)
        _check(lib().dvbs2fec_decode_vcm(self._h, len(d), _ptr(d), _ptr(x), _ptr(bb), _ptr(res)))
        return bb, bb_off, res

    def decode_plframes_vcm(self, desc, plframes):
        """desc as decode_vcm; plframes: the PLFRAMEs packed back to back (complex64, vcm_layout's sym_off)"""
        d = _vcm_desc(desc)
        sym_off, _, bb_off = vcm_layout(d)
        x = np.ascontiguousarray(plframes).view(np.float32).reshape(-1)
        assert x.size == 2 * sym_off[-1], (x.size, 2 * sym_off[-1])
        bb = np.zeros(bb_off[-1], np.uint8)
        res = np.zeros(len(d), RESULT_DTYPE)
        _check(lib().dvbs2fec_decode_plframes_vcm(self._h, len(d), _ptr(d), _ptr(x), _ptr(bb), _ptr(res)))
        return bb, bb_off, res

    def decode_vcm_device(self, desc, d_llr_ptr, d_bb_ptr, d_res_ptr, stream_ptr=0):
        """desc in host memory, the rest device pointers (vcm_layout sizes them); enqueues on ``stream_ptr`` and returns"""
        d = _vcm_desc(desc)
        _check(lib().dvbs2fec_decode_vcm_device(self._h, len(d), _ptr(d), d_llr_ptr, d_bb_ptr, d_res_ptr, stream_ptr))

    def decode_plframes_vcm_device(self, desc, d_plframes_ptr, d_bb_ptr, d_res_ptr, stream_ptr=0):
        d = _vcm_desc(desc)
        _check(lib().dvbs2fec_decode_plframes_vcm_device(self._h, len(d), _ptr(d), d_plframes_ptr, d_bb_ptr, d_res_ptr, stream_ptr))

    def set_profiling(self, on):
        _check(lib().dvbs2fec_set_profiling(self._h, int(on)))

    def kernel_times(self):
        """(demap_ms, ldpc_ms, bch_ms, launches) summed since the previous call; waits for the events."""
        a, b, c, n = C.c_float(), C.c_float(), C.c_float(), C.c_int()
        _check(lib().dvbs2fec_kernel_times(self._h, C.byref(a), C.byref(b), C.byref(c), C.byref(n)))
        return a.value, b.value, c.value, n.value

    def last_launch_count(self):
        return lib().dvbs2fec_last_launch_count(self._h)

    # ---- queue ----
    def submit_llr(self, llr, tag):
        x = np.ascontiguousarray(llr, np.int8)
        assert x.size == self.N
        _check(lib().dvbs2fec_submit_llr(self._h, _ptr(x), tag))

    def submit_plframe(self, plframe, tag):
        x = np.ascontiguousarray(plframe).view(np.float32)
        _check(lib().dvbs2fec_submit_plframe(self._h, _ptr(x), x.size // 2, tag))

    def collect(self, max_frames, timeout_us=0):
        bb = np.zeros((max_frames, self.kbch // 8), np.uint8)
        res = np.zeros(max_frames, RESULT_DTYPE)
        n = _check(lib().dvbs2fec_collect(self._h, _ptr(bb), _ptr(res), max_frames, timeout_us))
        return bb[:n], res[:n]

    def flush(self):
        _check(lib().dvbs2fec_flush(self._h))

    def set_ts_output(self, on=True):
        """queue delivers TS packets (BBFrameTSParser::work fused behind the decoder) instead of BBFRAMEs"""
        _check(lib().dvbs2fec_set_ts_output(self._h, int(on)))

    def collect_ts(self, cap=65536 * 10, max_results=4096, timeout_us=0):
        ts = np.zeros(max(cap, 1), np.uint8)
        res = np.zeros(max_results, RESULT_DTYPE)
        nres = C.c_int()
        n = _check(lib().dvbs2fec_collect_ts(self._h, _ptr(ts), cap, _ptr(res), max_results, C.byref(nres), timeout_us))
        return ts[:n], res[:nres.value]


class _StageObject:
    """Common part of the per-stage mirrors: each owns a decoder configured for (framesize, rate)."""

    # first MODCOD that uses a given rate (any constellation gives the same FEC objects)
    _MODCOD_OF_RATE = {0: 1, 1: 2, 2: 3, 3: 4, 4: 5, 5: 6, 6: 7, 7: 8, 8: 9, 10: 10, 11: 11}

    def __init__(self, framesize_short, rate, decoder=None, max_trials=25):
        if rate not in self._MODCOD_OF_RATE:
            raise DVBS2FecError(EINVAL, "code rate %r has no DVB-S2 LDPC table" % (rate,))
        self.dec = decoder or DVBS2Decoder(max_trials=max_trials)
        self.dec.setDemodParams(self._MODCOD_OF_RATE[rate], bool(framesize_short), False)


class BBFrameLDPC(_StageObject):
    """codings/bbframe_ldpc.h:32-60"""

    def dataSize(self):
        return self.dec.K

    def decode(self, frame, max_trials):
        """frame: N int8 LLRs, replaced in place by the posterior LLRs; returns iterations or -1."""
        f = frame.reshape(1, -1)
        return int(self.dec.ldpc_decode(f, max_trials)[0])


class BBFrameBCH(_StageObject):
    """codings/bbframe_bch.h:33-88"""

    def dataSize(self):
        return self.dec.kbch

    def decode(self, frame):
        """frame: K_ldpc/8 bytes corrected in place; returns corrections or -1."""
        return int(self.dec.bch_decode(frame.reshape(1, -1))[0])


class BBFrameDescrambler(_StageObject):
    """codings/bbframe_descramble.h:28-44"""

    def work(self, frame):
        self.dec.descramble(frame.reshape(1, -1))
        return 0


class S2BBToSoft:
    """dvbs2/dvbs2_bb_to_soft.h:16-48: PLFRAME symbols -> deinterleaved int8 LLRs."""

    def __init__(self, modcod, shortframes=False, pilots=False, decoder=None):
        self.dec = decoder or DVBS2Decoder()
        self.dec.setDemodParams(modcod, shortframes, pilots)

    def process(self, plframe):
        return self.dec.bb_to_soft(plframe)[0]


class BBFrameTSParser:
    """dvbs2/bbframe_ts_parser.h:67-108 on the device: BBFRAMEs in; 188-byte TS packets and GRE-wrapped GSE PDUs
    out.  Parser state (sync, unfinished packet, GSE reassembly) persists between work() calls like the reference's."""

    def __init__(self, device=0):
        self._p = C.c_void_p()
        _check(lib().dvbs2fec_ts_create(device, C.byref(self._p)))
        self.last_header = BBHeader()
        self.last_bb_cnt = self.last_bb_proc = self.gse_frames = 0
        self.last_gse_crc_err = 0
        self.gse_counters = dict(pdus=0, crc_errors=0, malformed=0, dropped=0)
        self.have_header = False

    def close(self):
        if getattr(self, "_p", None):
            lib().dvbs2fec_ts_destroy(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def setFrameSize(self, bbframe_size):
        _check(lib().dvbs2fec_ts_set_frame_size(self._p, bbframe_size))
        self.kbch = bbframe_size

    def _stats(self):
        a, b, g = C.c_int(), C.c_int(), C.c_int()
        self.have_header = bool(_check(lib().dvbs2fec_ts_stats(self._p, C.byref(self.last_header), C.byref(a), C.byref(b), C.byref(g))))
        self.last_bb_cnt, self.last_bb_proc, self.gse_frames = a.value, b.value, g.value
        v = [C.c_int() for _ in range(5)]
        _check(lib().dvbs2fec_ts_gse_stats(self._p, *[C.byref(x) for x in v]))
        self.last_gse_crc_err = v[0].value
        self.gse_counters = dict(pdus=v[1].value, crc_errors=v[2].value, malformed=v[3].value, dropped=v[4].value)

    def set_gse(self, max_packets_per_call=0):
        """< 0: GSE frames are only counted; 0: unpacked (default); > 0: descriptor pool for work_device"""
        _check(lib().dvbs2fec_ts_set_gse(self._p, max_packets_per_call))

    def work(self, bbframes, cnt=None, buffer_outsize=65536 * 10):
        """returns the TS bytes produced (uint8 array), like work()'s tsframes[:return value]"""
        x = np.ascontiguousarray(bbframes, np.uint8)
        if cnt is None:
            cnt = x.size // (self.kbch // 8)
        out = np.zeros(max(buffer_outsize, 1), np.uint8)
        n = _check(lib().dvbs2fec_ts_work(self._p, _ptr(x), cnt, _ptr(out), buffer_outsize))
        self._stats()
        return out[:n]

    def work_device(self, d_bb_ptr, cnt, d_out_ptr, buffer_outsize, d_produced_ptr=0, stream_ptr=0):
        _check(lib().dvbs2fec_ts_work_device(self._p, d_bb_ptr, cnt, d_out_ptr, buffer_outsize, d_produced_ptr, stream_ptr))


class S2PLSyncBlock:
    """dvbs2/dvbs2_pl_sync.h:11-66 on the device, together with the PLHEADER demodulator (S2PLHDRDemod,
    dvbs2/dvbs2_plhdr_demod.h:13-49) and the coarse frequency error detector (dvbs2/dvbs2_fed.h:7-48) that
    DVBS2Demod::process runs on its output.  Symbols are complex64 arrays."""

    def __init__(self, slot_num, pilots, device=0, loop_bw=0.004):
        self._p = C.c_void_p()
        _check(lib().dvbs2fec_plsync_create(device, C.byref(self._p)))
        self.setParams(slot_num, pilots)
        _check(lib().dvbs2fec_plhdr_set_params(self._p, loop_bw))
        self.current_position, self.best_match, self.pending = -1, 0.0, 0

    def close(self):
        if getattr(self, "_p", None):
            lib().dvbs2fec_plsync_destroy(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def setParams(self, slot_num, pilots):
        _check(lib().dvbs2fec_plsync_set_params(self._p, slot_num, int(pilots)))
        self.raw_frame_size = _check(lib().dvbs2fec_plsync_raw_frame_size(self._p))

    def reset(self):
        _check(lib().dvbs2fec_plsync_reset(self._p))

    def stats(self):
        a, b, c = C.c_int(), C.c_double(), C.c_int()
        n = _check(lib().dvbs2fec_plsync_stats(self._p, C.byref(a), C.byref(b), C.byref(c)))
        self.current_position, self.best_match, self.pending = a.value, b.value, c.value
        return n

    def process(self, symbols):
        x = np.ascontiguousarray(symbols, np.complex64)
        out = np.zeros(len(x) + 2 * self.raw_frame_size, np.complex64)
        n = _check(lib().dvbs2fec_plsync_process(self._p, len(x), _ptr(x), _ptr(out)))
        self.stats()
        return out[:n]

    def process_device(self, d_in_ptr, count, d_out_ptr, max_frames, d_nframes_ptr=0, stream_ptr=0):
        _check(lib().dvbs2fec_plsync_process_device(self._p, count, d_in_ptr, d_out_ptr, max_frames, d_nframes_ptr, stream_ptr))

    def plhdr_set_params(self, loop_bw):
        _check(lib().dvbs2fec_plhdr_set_params(self._p, loop_bw))

    def plhdr_process(self, frames):
        """frames [n][raw_frame_size] -> (headers [n][90] complex64, results [n][4] int32 = modcod, shortframes, pilots,
        PLS index, loop state (phase, freq))"""
        x = np.ascontiguousarray(frames, np.complex64).reshape(-1, self.raw_frame_size)
        n = len(x)
        hdr = np.zeros((n, 90), np.complex64)
        res = np.zeros((n, 4), np.int32)
        loop = np.zeros(2, np.float32)
        _check(lib().dvbs2fec_plhdr_process(self._p, n, _ptr(x), _ptr(hdr), _ptr(res), _ptr(loop)))
        return hdr, res, loop

    def coarse_fed(self, frames, pilots, pls_code, codenum=0):
        x = np.ascontiguousarray(frames, np.complex64).reshape(-1, self.raw_frame_size)
        err = np.zeros(len(x), np.float32)
        _check(lib().dvbs2fec_coarse_fed(self._p, len(x), _ptr(x), int(pilots), pls_code, codenum, _ptr(err)))
        return err

    # ---- S2PLLBlock (dvbs2/dvbs2_pll.h:17-78): the payload phase loop, same device object ----
    def pll_set_params(self, loop_bw, modcod, shortframes=False, pilots=False, codenum=0):
        _check(lib().dvbs2fec_pll_set_params(self._p, loop_bw, modcod, int(shortframes), int(pilots), codenum))
        self.pll_frame_symbols = _check(lib().dvbs2fec_pll_frame_symbols(self._p))

    def pll_reset(self):
        _check(lib().dvbs2fec_pll_reset(self._p))

    def pll_set_state(self, phase, freq):
        _check(lib().dvbs2fec_pll_set_state(self._p, phase, freq))

    def pll_set_sequential(self, on):
        _check(lib().dvbs2fec_pll_set_sequential(self._p, int(on)))

    def pll_process(self, frames, frame_stride=None):
        """frames [n][frame_stride] complex64 (consecutive frames of the stream) -> (out [n][frame_stride], of which the
        first pll_frame_symbols of every frame are written; state [n][3] = pcl.phase, pcl.freq, error after each frame)"""
        stride = frame_stride or self.raw_frame_size
        x = np.ascontiguousarray(frames, np.complex64).reshape(-1, stride)
        out = np.zeros_like(x)
        st = np.zeros((len(x), 3), np.float32)
        _check(lib().dvbs2fec_pll_process(self._p, len(x), stride, _ptr(x), _ptr(out), _ptr(st)))
        return out, st

    def pll_process_device(self, d_frames_ptr, nframes, frame_stride, d_out_ptr, d_state_ptr=0, stream_ptr=0):
        _check(lib().dvbs2fec_pll_process_device(self._p, nframes, frame_stride, d_frames_ptr, d_out_ptr, d_state_ptr, stream_ptr))

    def pll_rounds(self):
        return _check(lib().dvbs2fec_pll_rounds(self._p))


def pll_process_multi_device(blocks, d_frames_ptrs, nframes, frame_stride, d_out_ptrs, stream_ptr=0):
    """dvbs2fec_pll_process_multi_device: one launch for several S2PLSyncBlock objects (independent streams)"""
    n = len(blocks)
    objs = (C.c_void_p * n)(*[b._p for b in blocks])
    fin = (C.c_void_p * n)(*d_frames_ptrs)
    fout = (C.c_void_p * n)(*d_out_ptrs)
    _check(lib().dvbs2fec_pll_process_multi_device(n, objs, nframes, frame_stride, fin, fout, stream_ptr))


class DVBSOuterDecoder:
    """The frame loop body of DVBSDemod::process (dvbs/module_dvbs_demod.cpp:91-106) on the device: DVBSInterleaving
    .deinterleave, 8 x DVBSReedSolomon.decode, DVBSScrambling.descramble, 8 x 188 bytes out, for a batch of frames."""

    def __init__(self, device=0):
        self._p = C.c_void_p()
        _check(lib().dvbs2fec_dvbs_outer_create(device, C.byref(self._p)))

    def close(self):
        if getattr(self, "_p", None):
            lib().dvbs2fec_dvbs_outer_destroy(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self):
        _check(lib().dvbs2fec_dvbs_outer_reset(self._p))

    def process(self, frames, nframes, frame_stride=1632):
        """-> (TS packets [nframes * 8][188], errors [nframes * 8])"""
        x = np.ascontiguousarray(frames, np.uint8).reshape(-1)
        if nframes and len(x) < (nframes - 1) * frame_stride + 1632:
            raise ValueError("input shorter than (nframes - 1) * frame_stride + 1632 bytes")
        out = np.zeros((nframes * 8, 188), np.uint8)
        err = np.zeros(nframes * 8, np.int32)
        _check(lib().dvbs2fec_dvbs_outer_process(self._p, nframes, frame_stride, _ptr(x), _ptr(out), _ptr(err)))
        return out, err

    def process_device(self, d_frames_ptr, nframes, frame_stride, d_out_ptr, d_errors_ptr=0, stream_ptr=0):
        _check(lib().dvbs2fec_dvbs_outer_process_device(self._p, nframes, frame_stride, d_frames_ptr, d_out_ptr, d_errors_ptr, stream_ptr))


class DVBSTSDeframer:
    """deframing::DVBS_TS_Deframer (dvbs/dvbs_ts_deframer.h:17-70) on the device: work() takes the Viterbi decoder's
    unpacked bits and returns the frames of 8 x 204 bytes it finds; errors_nor / errors_inv as the reference's members."""

    def __init__(self, device=0):
        self._p = C.c_void_p()
        _check(lib().dvbs2fec_dvbs_deframer_create(device, C.byref(self._p)))

    def close(self):
        if getattr(self, "_p", None):
            lib().dvbs2fec_dvbs_deframer_destroy(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self):
        _check(lib().dvbs2fec_dvbs_deframer_reset(self._p))

    def work(self, bits, max_frames=None):
        """-> frames [n][1632]"""
        x = np.ascontiguousarray(bits, np.uint8).reshape(-1)
        if max_frames is None:
            max_frames = len(x) // 64 + 2
        out = np.zeros((max_frames, 1632), np.uint8)
        n = _check(lib().dvbs2fec_dvbs_deframer_work(self._p, _ptr(x), len(x), _ptr(out), max_frames))
        return out[:n].copy()

    def work_device(self, d_bits_ptr, size, d_frames_ptr, max_frames, d_nframes_ptr=0, stream_ptr=0):
        _check(lib().dvbs2fec_dvbs_deframer_work_device(self._p, d_bits_ptr, size, d_frames_ptr, max_frames, d_nframes_ptr, stream_ptr))

    def stats(self):
        """-> (errors_nor, errors_inv, frames found by the last call)"""
        a, b, c = C.c_int(), C.c_int(), C.c_int()
        _check(lib().dvbs2fec_dvbs_deframer_stats(self._p, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value


class DVBSViterbi:
    """DVBSVitBlock over viterbi::Viterbi_DVBS (dvbs/dvbs_vit.cpp:6-13, dvbs/viterbi_all.h:33-163) on the device, plus
    DVBSymToSoftBlock (dvbs/dvbs_syms_to_soft.cpp:26-42) in front of it."""
    RATES = ("1/2", "2/3", "3/4", "5/6", "7/8")

    def __init__(self, ber_threshold=0.15, max_outsync=20, device=0):
        self._p = C.c_void_p()
        _check(lib().dvbs2fec_dvbs_viterbi_create(device, ber_threshold, max_outsync, C.byref(self._p)))

    def close(self):
        if getattr(self, "_p", None):
            lib().dvbs2fec_dvbs_viterbi_destroy(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self):
        _check(lib().dvbs2fec_dvbs_viterbi_reset(self._p))

    def process(self, softs, out=None):
        """signed soft bits (a multiple of 8192) -> decoded bits, one per byte.  `out` (len(softs) bytes) is the buffer the
        bits are written into: what the reference leaves unwritten at rate 5/6 keeps its content"""
        x = np.ascontiguousarray(softs, np.int8).reshape(-1)
        if out is None:
            out = np.zeros(len(x), np.uint8)
        n = _check(lib().dvbs2fec_dvbs_viterbi_process(self._p, len(x), _ptr(x), _ptr(out)))
        return out[:n]

    def process_device(self, d_in_ptr, count, d_out_ptr):
        return _check(lib().dvbs2fec_dvbs_viterbi_process_device(self._p, count, d_in_ptr, d_out_ptr))

    def stats(self):
        """-> (ber, state, rate, phase, shift, invalid)"""
        b = C.c_float()
        v = [C.c_int() for _ in range(5)]
        _check(lib().dvbs2fec_dvbs_viterbi_stats(self._p, C.byref(b), *[C.byref(i) for i in v]))
        return (b.value,) + tuple(i.value for i in v)

    def counters(self):
        """-> (decode tasks run, tasks repeated from a corrected start state, check passes, tracebacks walked step by step)"""
        v = [C.c_longlong() for _ in range(4)]
        _check(lib().dvbs2fec_dvbs_viterbi_counters(self._p, *[C.byref(i) for i in v]))
        return tuple(i.value for i in v)

    def syms_to_soft(self, syms):
        """complex symbols -> soft bits, in chunks of 8192 (the rest waits for the next call)"""
        x = np.ascontiguousarray(syms).view(np.float32).reshape(-1) if np.iscomplexobj(syms) else np.ascontiguousarray(syms, np.float32).reshape(-1)
        n = len(x) // 2
        out = np.zeros(2 * n + 8192, np.int8)
        k = _check(lib().dvbs2fec_dvbs_sts_process(self._p, n, _ptr(x), _ptr(out)))
        return out[:k]


class DVBSDemod:
    """The decode stage of dsp::dvbs::DVBSDemod::process (dvbs/module_dvbs_demod.cpp:78-119) behind demod.process: symbols
    -> TS packets, on the device.  frame_stride=204 is the module's own walk over the deframer's frames, 1632 back to back."""

    def __init__(self, ber_threshold=0.15, max_outsync=20, frame_stride=204, device=0):
        self._p = C.c_void_p()
        _check(lib().dvbs2fec_dvbs_demod_create(device, ber_threshold, max_outsync, frame_stride, C.byref(self._p)))

    def close(self):
        if getattr(self, "_p", None):
            lib().dvbs2fec_dvbs_demod_destroy(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self):
        _check(lib().dvbs2fec_dvbs_demod_reset(self._p))

    def process(self, syms):
        """complex symbols -> TS packets [n][188]"""
        x = np.ascontiguousarray(syms).view(np.float32).reshape(-1) if np.iscomplexobj(syms) else np.ascontiguousarray(syms, np.float32).reshape(-1)
        n = len(x) // 2
        out = np.zeros(((2 * n + 8192) // 1632 + 8) * 1504, np.uint8)
        k = _check(lib().dvbs2fec_dvbs_demod_process(self._p, n, _ptr(x), _ptr(out), len(out)))
        return out[:k].reshape(-1, 188).copy()

    def stats(self):
        """-> dict(viterbi_ber, viterbi_lock, viterbi_rate, rs_avg, deframer_err, frames_found, frames_done)"""
        b, r = C.c_float(), C.c_float()
        i = [C.c_int() for _ in range(5)]
        _check(lib().dvbs2fec_dvbs_demod_stats(self._p, C.byref(b), C.byref(i[0]), C.byref(i[1]), C.byref(r), C.byref(i[2]), C.byref(i[3]), C.byref(i[4])))
        return dict(viterbi_ber=b.value, viterbi_lock=i[0].value, viterbi_rate=i[1].value, rs_avg=r.value, deframer_err=i[2].value,
                    frames_found=i[3].value, frames_done=i[4].value)


class DVBS2DemodStage:
    """The decode stage of dsp::dvbs2::DVBS2Demod::process (dvbs2/module_dvbs2_demod.cpp:300-367) behind its sample-domain
    front end, on the device: symbols -> PL sync -> coarse FED, phase loop, PLHEADER demodulation, demapper, LDPC, BCH,
    descrambler -> BBFRAMEs."""

    def __init__(self, device=None, max_batch=1024, max_trials=25):
        cfg = Config()
        if device is not None:
            cfg.n_devices, cfg.devices[0] = 1, device
        cfg.max_batch, cfg.max_trials = max_batch, max_trials
        self._p = C.c_void_p()
        _check(lib().dvbs2fec_s2_demod_create(C.byref(cfg), C.byref(self._p)))

    def close(self):
        if getattr(self, "_p", None):
            lib().dvbs2fec_s2_demod_destroy(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def setDemodParams(self, modcod, shortframes, pilots, max_trials=25, pll_loop_bw=0.004, plhdr_loop_bw=0.004, codenum=0):
        _check(lib().dvbs2fec_s2_demod_set_params(self._p, modcod, int(shortframes), int(pilots), max_trials, pll_loop_bw, plhdr_loop_bw, codenum))
        self.kb = lib().dvbs2fec_s2_demod_bbframe_bytes(self._p)

    def reset(self):
        _check(lib().dvbs2fec_s2_demod_reset(self._p))

    def process(self, syms):
        """complex symbols -> (bbframes [n][kbch / 8], results [n], coarse frequency errors [n], PLHEADER fields [n][4])"""
        x = np.ascontiguousarray(syms, np.complex64)
        m = lib().dvbs2fec_s2_demod_max_frames(self._p, len(x))
        bb = np.zeros((m, self.kb), np.uint8)
        res = np.zeros(m, RESULT_DTYPE)
        fed = np.zeros(m, np.float32)
        hdr = np.zeros((m, 4), np.int32)
        n = _check(lib().dvbs2fec_s2_demod_process(self._p, len(x), _ptr(x), _ptr(bb), m, _ptr(res), _ptr(fed), _ptr(hdr)))
        return bb[:n], res[:n], fed[:n], hdr[:n]

    def process_ts(self, syms, ts_cap=65536 * 10):
        """complex symbols -> (TS / GSE output bytes of BBFrameTSParser::work on the decoded BBFRAMEs, frames decoded)"""
        x = np.ascontiguousarray(syms, np.complex64)
        out = np.zeros(ts_cap, np.uint8)
        nfr = C.c_int()
        n = _check(lib().dvbs2fec_s2_demod_process_ts(self._p, len(x), _ptr(x), _ptr(out), ts_cap, 0, C.byref(nfr), None, None, None))
        return out[:n], nfr.value
