"""VCM / ACM batches: frames of any MODCOD, frame size and pilot setting, and DUMMY PLFRAMEs, in one call
(`dvbs2fec_decode_vcm`, `dvbs2fec_decode_plframes_vcm` and their `_device` forms).

The reference is the per-configuration path, which the demapper, LDPC and BCH tests pin to the oracle: every frame's
BBFRAME bytes, LDPC iterations, BCH corrections and flags must equal what a handle configured for that frame alone
(`setDemodParams(config)` + `decode_plframes`) returns.  The pool holds two noisy frames of each of the 104
configurations -- one well above the code's threshold, one near it -- and NaN-filled DUMMY PLFRAMEs, in a seeded order
that changes the code, constellation or frame size at nearly every step.  A sample is also checked against the oracle
chain directly."""
import ctypes as C

import numpy as np
import pytest

import orclib
from fec import pkg, MODCODS
from test_gpu_demapper import configurations, oracle_chain, oracle_llrs, payload_positions, pl_scramble

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

# Es/N0 (dB) at which each MODCOD's normal frames reach quasi-error-free operation, EN 302 307 Table 13
THRESHOLD = {1: -2.35, 2: -1.24, 3: -0.30, 4: 1.00, 5: 2.23, 6: 3.10, 7: 4.03, 8: 4.68, 9: 5.18, 10: 6.20, 11: 6.42,
             12: 5.50, 13: 6.62, 14: 7.91, 15: 9.35, 16: 10.69, 17: 10.98, 18: 8.97, 19: 10.21, 20: 11.03, 21: 11.61,
             22: 12.89, 23: 13.13, 24: 12.73, 25: 13.64, 26: 14.28, 27: 15.69, 28: 16.05}
MARGINS = (3.0, 0.5)          # dB above the threshold: a clean frame and one near it (short frames get 0.5 dB more)
DUMMY_SYMS = 90 + 36 * 90
N_DUMMY = 24
CODENUM = 77777               # Gold code of the PL-scrambled runs


class Pool:
    def __init__(self, seed=5):
        rng = np.random.default_rng(seed)
        items = []
        for modcod, short, pilots in configurations():
            info = pkg.modcod_info(modcod, short, pilots)
            pos, _ = payload_positions(info["nldpc"] // info["bits"], pilots)
            for margin in MARGINS:
                bits = pkg.encode_fecframe(modcod, short, rng.integers(0, 256, info["kbch"] // 8, dtype=np.uint8))
                tx = pkg.modulate(modcod, short, pilots, bits)
                es = float(np.mean(np.abs(tx[pos]) ** 2))
                esn0 = THRESHOLD[modcod] + margin + (0.5 if short else 0.0)
                sigma = np.sqrt(es / (2 * 10 ** (esn0 / 10)))
                noise = rng.normal(0, sigma, (len(tx), 2)).astype(np.float32).view(np.complex64).reshape(-1)
                items.append(((modcod, int(short), int(pilots)), (tx + noise).astype(np.complex64)))
        items += [(None, np.full(DUMMY_SYMS, np.nan + 1j * np.nan, np.complex64)) for _ in range(N_DUMMY)]
        order = rng.permutation(len(items))
        self.cfg = [items[i][0] for i in order]
        self.syms = [items[i][1] for i in order]
        self.desc = np.array([(0, 0, 0, 0) if c is None else (c[0], c[1], c[2], 0) for c in self.cfg], np.int32)
        self.dummy = np.array([c is None for c in self.cfg])
        self.by_cfg = {}
        for i, c in enumerate(self.cfg):
            if c is not None:
                self.by_cfg.setdefault(c, []).append(i)
        self.n = len(self.cfg)
        self.ref = {}

    def reference(self, dec, codenum):
        """per-configuration results; codenum >= 0: the frames PL-scrambled with that Gold code"""
        n = self.n
        syms, llr, bb = list(self.syms), [np.zeros(0, np.int8)] * n, [np.zeros(0, np.uint8)] * n
        its, cor = np.zeros(n, np.int16), np.zeros(n, np.int16)
        flags = np.full(n, pkg.FLAG_DUMMY, np.uint32)
        dec.set_pl_scrambling(codenum)
        for cfg, idx in self.by_cfg.items():
            dec.setDemodParams(cfg[0], bool(cfg[1]), bool(cfg[2]), 25)
            x = np.stack([self.syms[i] for i in idx])
            if codenum >= 0:
                x = pl_scramble(x.view(np.float32).reshape(len(idx), -1, 2), codenum).reshape(len(idx), -1).view(np.complex64)
            b, r = dec.decode_plframes(x)
            soft = dec.bb_to_soft(x)
            for k, i in enumerate(idx):
                syms[i], llr[i], bb[i] = x[k], soft[k], b[k]
                its[i], cor[i], flags[i] = r["ldpc_iters"][k], r["bch_corr"][k], r["flags"][k]
        dec.set_pl_scrambling(-1)
        self.ref[codenum] = dict(syms=np.concatenate(syms), llr=np.concatenate(llr), bb=np.concatenate(bb), iters=its,
                                 corr=cor, flags=flags)
        return self.ref[codenum]


@pytest.fixture(scope="module")
def pool():
    p = Pool()
    dec = pkg.DVBS2Decoder(max_batch=64, max_trials=25)
    p.reference(dec, -1)
    p.reference(dec, CODENUM)
    dec.close()
    return p


def assert_results(pool, want, bb, res, what):
    n = pool.n
    assert np.array_equal(res["tag"], np.arange(n)), what
    assert np.array_equal(res["ldpc_iters"], want["iters"]), (what, np.flatnonzero(res["ldpc_iters"] != want["iters"]))
    assert np.array_equal(res["bch_corr"], want["corr"]), (what, np.flatnonzero(res["bch_corr"] != want["corr"]))
    assert np.array_equal(res["flags"], want["flags"]), (what, np.flatnonzero(res["flags"] != want["flags"]))
    assert np.array_equal(bb, want["bb"]), what


def run_device(dec, pool, sym, inp, stream):
    """one device call on `stream` from device copies of the packed input; returns host copies of the outputs"""
    _, _, bb_off = pkg.vcm_layout(pool.desc)
    d_in = torch.from_numpy(inp.view(np.uint8).copy()).cuda()
    d_bb = torch.full((int(bb_off[-1]),), 0xA5, dtype=torch.uint8, device="cuda")
    d_res = torch.full((pool.n, 16), 0xA5, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    f = dec.decode_plframes_vcm_device if sym else dec.decode_vcm_device
    f(pool.desc, d_in.data_ptr(), d_bb.data_ptr(), d_res.data_ptr(), stream.cuda_stream)
    stream.synchronize()
    return d_bb.cpu().numpy(), d_res.cpu().numpy().view(pkg.RESULT_DTYPE).reshape(-1)


@pytest.mark.parametrize("max_batch", [7, 4096])
def test_vcm_matches_the_per_configuration_path(pool, max_batch):
    """all four entry points on a handle that was never configured; max_batch 7 puts chunk edges inside groups and
    leaves some chunks with a single code (the path without reordering), 4096 holds the whole pool.  Then PL-scrambled
    on the same handle."""
    assert pool.n == 2 * 104 + N_DUMMY
    dec = pkg.DVBS2Decoder(max_batch=max_batch, max_trials=25)
    st = torch.cuda.Stream()
    plain, scr = pool.ref[-1], pool.ref[CODENUM]
    bb, bb_off, res = dec.decode_vcm(pool.desc, plain["llr"])
    assert np.array_equal(bb_off, pkg.vcm_layout(pool.desc)[2])
    assert_results(pool, plain, bb, res, "decode_vcm")
    bb, _, res = dec.decode_plframes_vcm(pool.desc, plain["syms"])
    assert_results(pool, plain, bb, res, "decode_plframes_vcm")
    assert_results(pool, plain, *run_device(dec, pool, False, plain["llr"], st), "decode_vcm_device")
    assert_results(pool, plain, *run_device(dec, pool, True, plain["syms"], st), "decode_plframes_vcm_device")
    dec.set_pl_scrambling(CODENUM)
    bb, _, res = dec.decode_plframes_vcm(pool.desc, scr["syms"])
    assert_results(pool, scr, bb, res, "decode_plframes_vcm, PL scrambled")
    assert_results(pool, scr, *run_device(dec, pool, True, scr["syms"], st), "decode_plframes_vcm_device, PL scrambled")
    # LLR input does not depend on the PL scrambling
    bb, _, res = dec.decode_vcm(pool.desc, plain["llr"])
    assert_results(pool, plain, bb, res, "decode_vcm with PL scrambling set")
    dec.close()
    # the pool exercises what it is meant to: iteration counts vary, both outcomes occur
    its = plain["iters"][~pool.dummy]
    assert len(np.unique(its)) > 5
    assert (its == np.min(its)).mean() < 0.9


def test_sample_against_the_oracle(pool):
    """16 frames of LUT constellations straight against orc_bb_to_soft + orc_decode_frame (32APSK's LLRs are within a
    tolerance of the oracle's, not equal: its chain is checked in test_gpu_demapper)"""
    dec = pkg.DVBS2Decoder(max_batch=4096, max_trials=25)
    bb, bb_off, res = dec.decode_plframes_vcm(pool.desc, pool.ref[-1]["syms"])
    dec.close()
    cand = [i for i in range(pool.n) if not pool.dummy[i] and MODCODS[pool.cfg[i][0]][0] != 3]
    pick = np.random.default_rng(9).choice(cand, 16, replace=False)
    for i in pick:
        modcod, short, pilots = pool.cfg[i]
        info = pkg.modcod_info(modcod, bool(short), bool(pilots))
        pos, _ = payload_positions(info["nldpc"] // info["bits"], pilots)
        payload = pool.syms[i].view(np.float32).reshape(-1, 2)[pos]
        llr = oracle_llrs(modcod, short, payload[None])
        wbb, wits, wcor, wflags = oracle_chain(short, MODCODS[modcod][2], llr)
        assert (res["ldpc_iters"][i], res["bch_corr"][i], res["flags"][i]) == (wits[0], wcor[0], wflags[0]), (i, pool.cfg[i])
        assert np.array_equal(bb[bb_off[i]:bb_off[i + 1]], wbb[0]), (i, pool.cfg[i])


def test_device_calls_interleaved_with_decode_batch_device(pool):
    """VCM device calls on one stream, CCM device calls of the same handle on another: each gets its own results"""
    cfg = (4, 0, 0)
    idx = pool.by_cfg[cfg]
    dec = pkg.DVBS2Decoder(max_batch=64, max_trials=25)
    dec.setDemodParams(4, False, False, 25)
    _, llr_off, bb_off = pkg.vcm_layout(pool.desc)
    ccm_llr = np.stack([pool.ref[-1]["llr"][llr_off[i]:llr_off[i + 1]] for i in idx] * 8)
    want_bb, want_res = dec.decode_batch(ccm_llr)
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    d_ccm = torch.from_numpy(ccm_llr).cuda()
    d_sym = torch.from_numpy(pool.ref[-1]["syms"].view(np.uint8).copy()).cuda()
    outs = []
    torch.cuda.synchronize()
    for k in range(3):
        a_bb = torch.full(want_bb.shape, 0xA5, dtype=torch.uint8, device="cuda")
        a_res = torch.full((len(ccm_llr), 16), 0xA5, dtype=torch.uint8, device="cuda")
        b_bb = torch.full((int(bb_off[-1]),), 0xA5, dtype=torch.uint8, device="cuda")
        b_res = torch.full((pool.n, 16), 0xA5, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        dec.decode_batch_device(d_ccm.data_ptr(), len(ccm_llr), a_bb.data_ptr(), a_res.data_ptr(), sa.cuda_stream)
        dec.decode_plframes_vcm_device(pool.desc, d_sym.data_ptr(), b_bb.data_ptr(), b_res.data_ptr(), sb.cuda_stream)
        outs.append((a_bb, a_res, b_bb, b_res))
    torch.cuda.synchronize()
    for a_bb, a_res, b_bb, b_res in outs:
        assert np.array_equal(a_bb.cpu().numpy(), want_bb)
        assert np.array_equal(a_res.cpu().numpy().view(pkg.RESULT_DTYPE).reshape(-1), want_res)
        assert_results(pool, pool.ref[-1], b_bb.cpu().numpy(), b_res.cpu().numpy().view(pkg.RESULT_DTYPE).reshape(-1),
                       "interleaved VCM device call")
    dec.close()


def test_vcm_call_leaves_the_configuration_alone(pool):
    cfg = (13, 1, 1)   # 8PSK 2/3 short, pilots
    idx = pool.by_cfg[cfg]
    dec = pkg.DVBS2Decoder(max_batch=16, max_trials=25)
    dec.setDemodParams(13, True, True, 25)
    x = np.stack([pool.syms[i] for i in idx])
    bb1, res1 = dec.decode_plframes(x)
    llr1 = dec.bb_to_soft(x)
    bb, _, res = dec.decode_plframes_vcm(pool.desc, pool.ref[-1]["syms"])
    assert_results(pool, pool.ref[-1], bb, res, "VCM call on a configured handle")
    bb2, res2 = dec.decode_plframes(x)
    assert np.array_equal(bb1, bb2) and np.array_equal(res1, res2)
    assert np.array_equal(llr1, dec.bb_to_soft(x))
    assert (dec.N, dec.kbch) == (pkg.lib().dvbs2fec_nldpc(dec._h), pkg.lib().dvbs2fec_kbch(dec._h))
    dec.close()


BAD = [(29, 0, 0), (31, 0, 0), (-1, 0, 0), (11, 1, 0), (28, 1, 1)]


def test_bad_input_is_refused_and_nothing_is_written(pool):
    L = pkg.lib()
    dec = pkg.DVBS2Decoder(max_batch=7, max_trials=25)
    vp = C.c_void_p
    good = np.array([[4, 0, 0, 0], [0, 0, 0, 0], [13, 1, 1, 0]], np.int32)
    _, llr_off, bb_off = pkg.vcm_layout(good)
    sym = np.zeros(2 * 100000, np.float32)
    llr = np.zeros(int(llr_off[-1]), np.int8)
    bb = np.full(int(bb_off[-1]) + 64, 0x5A, np.uint8)
    res = np.zeros(8, pkg.RESULT_DTYPE)
    res.view(np.uint8)[:] = 0x5A
    d_in = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    d_bb = torch.full((int(bb_off[-1]) + 64,), 0x5A, dtype=torch.uint8, device="cuda")
    d_res = torch.full((8, 16), 0x5A, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    calls = [lambda n, d, i: L.dvbs2fec_decode_vcm(dec._h, n, d, i if i is None else llr.ctypes.data_as(vp), bb.ctypes.data_as(vp), res.ctypes.data_as(vp)),
             lambda n, d, i: L.dvbs2fec_decode_plframes_vcm(dec._h, n, d, i if i is None else sym.ctypes.data_as(vp), bb.ctypes.data_as(vp), res.ctypes.data_as(vp)),
             lambda n, d, i: L.dvbs2fec_decode_vcm_device(dec._h, n, d, i if i is None else d_in.data_ptr(), d_bb.data_ptr(), d_res.data_ptr(), None),
             lambda n, d, i: L.dvbs2fec_decode_plframes_vcm_device(dec._h, n, d, i if i is None else d_in.data_ptr(), d_bb.data_ptr(), d_res.data_ptr(), None)]
    for k, call in enumerate(calls):
        for bad in BAD:
            d = np.concatenate([good, [[bad[0], bad[1], bad[2], 0]], good]).astype(np.int32)
            assert call(len(d), d.ctypes.data_as(vp), 1) == pkg.EINVAL, (k, bad)
            assert "frame 3" in L.dvbs2fec_last_error().decode(), (k, bad)
        assert call(-1, good.ctypes.data_as(vp), 1) == pkg.EINVAL, k
        assert call(3, None, 1) == pkg.EINVAL, k
        assert call(3, good.ctypes.data_as(vp), None) == pkg.EINVAL, k
        assert pkg.lib().dvbs2fec_decode_vcm(None, 3, good.ctypes.data_as(vp), llr.ctypes.data_as(vp), None, None) == pkg.EINVAL
    torch.cuda.synchronize()
    assert (bb == 0x5A).all() and (res.view(np.uint8) == 0x5A).all()
    assert (d_bb.cpu().numpy() == 0x5A).all() and (d_res.cpu().numpy() == 0x5A).all()
    # the handle still decodes
    bb, _, res = dec.decode_plframes_vcm(pool.desc, pool.ref[-1]["syms"])
    assert_results(pool, pool.ref[-1], bb, res, "after refused calls")
    dec.close()


def launches(dec, desc, sym, syms, llr):
    if sym:
        dec.decode_plframes_vcm(desc, syms)
    else:
        dec.decode_vcm(desc, llr)
    return dec.last_launch_count()


def test_launch_count_follows_the_number_of_codes(pool):
    """DESIGN §3: per chunk of k codes 2k + 2 launches (demap or gather, LDPC and BCH per code, scatter); a chunk of
    one code and no dummy frame takes 2 (LLRs) or 3 (symbols); a chunk of dummy frames 1.  Not the number of frames."""
    dec = pkg.DVBS2Decoder(max_batch=4096, max_trials=25)
    ref = pool.ref[-1]
    sym_off, llr_off, _ = pkg.vcm_layout(pool.desc)

    def sub(idx):
        idx = list(idx)
        return (pool.desc[idx], np.concatenate([ref["syms"][sym_off[i]:sym_off[i + 1]] for i in idx]),
                np.concatenate([ref["llr"][llr_off[i]:llr_off[i + 1]] for i in idx]))

    three = [i for i in range(pool.n) if pool.cfg[i] is not None and pool.cfg[i][:2] in ((4, 0), (13, 1), (19, 0))]
    dummies = list(np.flatnonzero(pool.dummy))
    codes = {(MODCODS[pool.cfg[i][0]][2], pool.cfg[i][1]) for i in three}
    k = len(codes)
    assert k == 3
    for sym in (False, True):
        for reps in (1, 3):
            desc, s, l = sub(three * reps + dummies[:2])
            assert launches(dec, desc, sym, s, l) == 2 * k + 2, (sym, reps)
        one = [i for i in range(pool.n) if pool.cfg[i] is not None and pool.cfg[i][:2] == (4, 0)]
        for reps in (1, 5):
            desc, s, l = sub(one * reps)
            assert launches(dec, desc, sym, s, l) == (3 if sym else 2), (sym, reps)
        desc, s, l = sub(dummies)
        assert launches(dec, desc, sym, s, l) == 1
    # two chunks: the counts add up
    dec.close()
    dec = pkg.DVBS2Decoder(max_batch=len(three) + 2, max_trials=25)
    desc, s, l = sub(three + dummies[:2] + one)
    assert launches(dec, desc, False, s, l) == (2 * k + 2) + 2
    dec.close()


def test_more_than_65535_frames_in_one_call():
    """65 600 frames in one device call (one chunk): all DUMMY but every 500th, a QPSK 1/2 short frame.  The demap
    launch's y dimension and the scatter's x dimension are capped at 65 535 and loop."""
    n = 65600
    desc = np.zeros((n, 4), np.int32)
    real = np.arange(0, n, 500)
    desc[real, 0], desc[real, 1] = 4, 1
    sym_off, llr_off, bb_off = pkg.vcm_layout(desc)
    rng = np.random.default_rng(21)
    ref = pkg.DVBS2Decoder(max_batch=256, max_trials=25)
    ref.setDemodParams(4, True, False, 25)
    info = pkg.modcod_info(4, True, False)
    frames = []
    for k in range(8):
        bits = pkg.encode_fecframe(4, True, rng.integers(0, 256, info["kbch"] // 8, dtype=np.uint8))
        tx = pkg.modulate(4, True, False, bits)
        frames.append(tx + rng.normal(0, 0.45 if k % 2 else 0.3, (len(tx), 2)).astype(np.float32).view(np.complex64).reshape(-1))
    frames = np.stack(frames).astype(np.complex64)
    which = np.arange(len(real)) % len(frames)
    want_bb, want_res = ref.decode_plframes(frames[which])
    llr = ref.bb_to_soft(frames)
    ref.close()
    dev = torch.device("cuda", 0)
    d_frames = torch.from_numpy(frames.view(np.float32)).to(dev)
    d_llr_frames = torch.from_numpy(llr).to(dev)
    d_sym = torch.full((2 * int(sym_off[-1]),), float("nan"), dtype=torch.float32, device=dev)
    d_llr = torch.empty(int(llr_off[-1]), dtype=torch.int8, device=dev)
    for j, i in enumerate(real):
        d_sym[2 * sym_off[i]:2 * sym_off[i + 1]] = d_frames[which[j]]
        d_llr[llr_off[i]:llr_off[i + 1]] = d_llr_frames[which[j]]
    dec = pkg.DVBS2Decoder(max_batch=n, max_trials=25)
    st = torch.cuda.current_stream()
    for sym, src in ((True, d_sym), (False, d_llr)):
        d_bb = torch.full((int(bb_off[-1]),), 0xA5, dtype=torch.uint8, device=dev)
        d_res = torch.full((n, 16), 0xA5, dtype=torch.uint8, device=dev)
        f = dec.decode_plframes_vcm_device if sym else dec.decode_vcm_device
        f(desc, src.data_ptr(), d_bb.data_ptr(), d_res.data_ptr(), st.cuda_stream)
        torch.cuda.synchronize()
        res = d_res.cpu().numpy().view(pkg.RESULT_DTYPE).reshape(-1)
        assert np.array_equal(res["tag"], np.arange(n)), sym
        dummy = np.ones(n, bool)
        dummy[real] = False
        assert (res["ldpc_iters"][dummy] == 0).all() and (res["bch_corr"][dummy] == 0).all(), sym
        assert (res["flags"][dummy] == pkg.FLAG_DUMMY).all(), sym
        for field in ("ldpc_iters", "bch_corr", "flags"):
            assert np.array_equal(res[field][real], want_res[field]), (sym, field)
        assert np.array_equal(d_bb.cpu().numpy(), want_bb.reshape(-1)), sym
        assert dec.last_launch_count() == 4, sym
    dec.close()
