"""K7 (PLHEADER decoding, coarse frequency error, PL sync) and K8 (the payload phase loop) against the CPU oracle on every
PLS code, every geometry (slots 36 .. 360, pilots off / on) and every (MODCOD, frame size, pilots) configuration, and the
one-call stage on every geometry.  The constructions are checked against the oracle alone in
tests/test_pl_frontend_model.py.

Bit for bit:
* PLHEADER decoding with the loop at rest: header symbols on the pi/2-BPSK diagonals make the loop error exactly 0, so
  headers, loop state and PLS fields equal the oracle's exactly, and the hard decisions spell any word: all 128
  codewords, bits 63..60 flipped, 1..13 errors, ties across the kernel's lane split (the lowest index wins), symbols on
  the decision boundary (the reference's unfused `> 0`), random words with ties of three;
* the coarse FED for every PLS code on every geometry, the pilots flag independent of the code, the Gold code changing
  between calls;
* the phase loop open (alpha = beta = 0): output symbols and per-frame phase and frequency for all 104 configurations;
  the mean error too, except for 32APSK, whose error is CUDA's atan2f against glibc's (held to a bound from the ulps of
  the per-symbol errors and of the running sum).  The mean error is one float per frame: it pins each table cell a
  probe visits to about an ulp of that sum, not to its last bit;
* the speculative kernels against the sequential walk, multi-stream against single-stream calls, the one-call stage
  against the stages called one by one, PL sync frame positions and metrics.
To tolerance: noisy PLHEADERs (1e-4, PLS fields exact), the closed phase loop (the bar of tests/test_gpu_pll.py).
`test_fed_does_not_change_the_loops_scrambling_sequence` holds the loop's PL descrambling to the code it was configured
with, whatever code the FED is called with in between."""
import numpy as np
import pytest

import orclib
import plstream
from fec import pkg, MODCODS
from test_gpu_demapper import configurations, oracle_constellation
from test_gpu_pll import MEDIAN_SYM, TOL_SYM
from test_plsync_oracle import OrcSync, f32
from test_pl_frontend_model import (GEOMETRIES, crafted_words, decode, fields, float_sum, header_frames, noisy_header_plan,
                                    open_loop_errors, open_loop_frames, oracle_pll, oracle_plhdr, pll_geometry, pll_sequence)

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def bits(x):
    return np.ascontiguousarray(x).view(np.uint32)


def cuts(n, rng, k=5):
    """uneven call boundaries over n frames"""
    return [0] + sorted(set(int(c) for c in rng.integers(1, n, k))) + [n]


def plhdr_device(g, frames, stream):
    """dvbs2fec_plhdr_process_device on torch buffers -> (headers, results)"""
    n, rfs = frames.shape
    d_fr = torch.from_numpy(f32(frames).copy()).cuda()
    d_h = torch.zeros(n * 180, dtype=torch.float32, device="cuda")
    d_r = torch.zeros(n * 4, dtype=torch.int32, device="cuda")
    pkg._check(pkg.lib().dvbs2fec_plhdr_process_device(g._p, n, d_fr.data_ptr(), d_h.data_ptr(), d_r.data_ptr(), stream.cuda_stream))
    stream.synchronize()
    return d_h.cpu().numpy().view(np.complex64).reshape(n, 90), d_r.cpu().numpy().reshape(n, 4)


# ------------------------------------------------------------------------------------------------ 1. PLHEADER, exact
@pytest.mark.parametrize("gi", [0, 3], ids=lambda gi: "%d-%s" % (GEOMETRIES[gi][0], "pilots" if GEOMETRIES[gi][1] else "nopilots"))
def test_plhdr_crafted_words_bit_for_bit(gi):
    slots, pilots = GEOMETRIES[gi]
    words, kinds, _ = crafted_words()
    rng = np.random.default_rng(30 + gi)
    g = pkg.S2PLSyncBlock(slots, pilots, loop_bw=0.004)
    rfs = g.raw_frame_size
    fr, o = header_frames(words, rfs, rng)
    want_h, want_r, want_l = oracle_plhdr(fr, rfs)
    want = decode(words)
    assert np.array_equal(want_r, fields(want)[:, :3])
    got_h, got_r = [], []
    c = cuts(len(fr), rng)
    for a, b in zip(c[:-1], c[1:]):
        h, r, loop = g.plhdr_process(fr[a:b])
        got_h.append(h)
        got_r.append(r)
        assert np.array_equal(bits(loop), bits(want_l[b - 1])), (a, b)
    got_h, got_r = np.concatenate(got_h), np.concatenate(got_r)
    assert np.array_equal(bits(got_h), bits(want_h)) and np.array_equal(bits(got_h), bits(o))
    bad = np.flatnonzero((got_r != fields(want)).any(axis=1))
    assert not len(bad), [(kinds[i], int(want[i]), got_r[i].tolist()) for i in bad[:10]]
    g.close()


def test_plhdr_4096_frames_in_one_call_and_in_pieces_and_on_device_buffers():
    words, _, _ = crafted_words()
    rng = np.random.default_rng(4096)
    words = words[rng.integers(0, len(words), 4096)]
    slots, pilots = GEOMETRIES[0]
    g = pkg.S2PLSyncBlock(slots, pilots)
    rfs = g.raw_frame_size
    fr, o = header_frames(words, rfs, rng)
    want = fields(decode(words))
    h1, r1, l1 = g.plhdr_process(fr)
    assert np.array_equal(r1, want) and np.array_equal(bits(h1), bits(o)) and not bits(l1).any()
    c = cuts(4096, rng, 9)
    parts = [g.plhdr_process(fr[a:b]) for a, b in zip(c[:-1], c[1:])]
    assert np.array_equal(np.concatenate([p[1] for p in parts]), r1)
    assert np.array_equal(bits(np.concatenate([p[0] for p in parts])), bits(h1))
    h3, r3 = plhdr_device(g, fr, torch.cuda.Stream())
    assert np.array_equal(r3, r1) and np.array_equal(bits(h3), bits(h1))
    g.close()


# ------------------------------------------------------------------------------------------------ 2. PLHEADER, noisy
@pytest.mark.parametrize("gi", range(16), ids=lambda gi: "%d-%s" % (GEOMETRIES[gi][0], "pilots" if GEOMETRIES[gi][1] else "nopilots"))
def test_plhdr_noisy_every_code(gi):
    """the codes gi, gi + 16, ... (all 128 over the 16 geometries), three frames each at Es/N0 3 and 10 dB, own phase and
    carrier offsets, in uneven calls: headers and loop state within 1e-4 of the oracle, PLS fields exact and equal to the
    transmitted code"""
    slots, pilots = GEOMETRIES[gi]
    codes, fr, rng = noisy_header_plan(gi)
    g = pkg.S2PLSyncBlock(slots, pilots, loop_bw=0.004)
    rfs = g.raw_frame_size
    assert fr.shape[1] == rfs
    want_h, want_r, want_l = oracle_plhdr(fr, rfs)
    got_h, got_r = [], []
    c = cuts(len(fr), rng)
    for a, b in zip(c[:-1], c[1:]):
        h, r, loop = g.plhdr_process(fr[a:b])
        got_h.append(h)
        got_r.append(r)
        assert np.allclose(loop, want_l[b - 1], atol=1e-4), (a, b, loop, want_l[b - 1])
    got_h, got_r = np.concatenate(got_h), np.concatenate(got_r)
    rot = np.complex64(complex(np.float32(np.cos(-np.pi / 4)), np.float32(np.sin(-np.pi / 4))))
    for k in np.flatnonzero((got_r[:, :3] != want_r).any(axis=1)):      # which hard decisions differed
        dev_bits, orc_bits = (got_h[k, 26:] * rot).real > 0, (want_h[k, 26:] * rot).real > 0
        pytest.fail("frame %d: fields %s, oracle %s; decisions differ at header symbols %s" % (
            k, got_r[k].tolist(), want_r[k].tolist(), (26 + np.flatnonzero(dev_bits != orc_bits)).tolist()))
    assert np.array_equal(got_r, fields(codes))
    assert np.abs(got_h - want_h).max() < 1e-4
    g.close()


# ------------------------------------------------------------------------------------------------ 3. coarse FED
FED_CODENUMS = (0, 1, 131071, 262141, 7, 40507, 99999, 200000)


@pytest.mark.parametrize("gi", range(16), ids=lambda gi: "%d-%s" % (GEOMETRIES[gi][0], "pilots" if GEOMETRIES[gi][1] else "nopilots"))
def test_coarse_fed_every_code(gi):
    """all 128 PLS codes on one handle, the pilots flag independent of the code's own pilots bit, the Gold code
    changing from one pilots call to the next: bit for bit with orc_coarse_fed; and on torch buffers"""
    slots, pilots = GEOMETRIES[gi]
    rng = np.random.default_rng(1300 + gi)
    g = pkg.S2PLSyncBlock(slots, pilots)
    rfs = g.raw_frame_size
    x = plstream.stream((gi * 9) & 127, slots, pilots, 3, rng, esn0_db=8.0, lead=0, cfo=2e-4, codenum=FED_CODENUMS[gi % 8])
    frames = x.reshape(3, rfs)
    rn = {c: plstream.pl_rn(c) for c in FED_CODENUMS}
    o = orclib.oracle()
    k = gi
    for code in rng.permutation(128):
        fp = int((code >> 3) ^ code ^ gi) & 1
        cn = FED_CODENUMS[k % 8]
        k += fp
        want = np.array([o.orc_coarse_fed(f32(f), rfs, fp, int(code), rn[cn]) for f in frames], np.float32)
        got = g.coarse_fed(frames, fp, int(code), cn)
        assert np.array_equal(bits(got), bits(want)), (int(code), fp, cn)
    st = torch.cuda.Stream()
    d_fr = torch.from_numpy(f32(frames).copy()).cuda()
    d_err = torch.zeros(3, dtype=torch.float32, device="cuda")
    for code, fp, cn in ((gi, 1, 262141), (127 - gi, 0, 0), (64 + gi, 1, 131071)):
        pkg._check(pkg.lib().dvbs2fec_coarse_fed_device(g._p, 3, d_fr.data_ptr(), fp, code, cn, d_err.data_ptr(), st.cuda_stream))
        st.synchronize()
        want = np.array([o.orc_coarse_fed(f32(f), rfs, fp, code, rn[cn]) for f in frames], np.float32)
        assert np.array_equal(bits(d_err.cpu().numpy()), bits(want)), (code, fp, cn)
    g.close()


# ------------------------------------------------------------------------------------------------ 4. FED vs loop
def test_fed_does_not_change_the_loops_scrambling_sequence():
    """the loop descrambles with the Gold code it was configured with, whatever code the coarse FED used in between"""
    rng = np.random.default_rng(44)
    cfg = (4, False, True)
    slots, total, stride, _ = pll_geometry(cfg)
    fr = closed_loop_frames(cfg, 3, 1, rng)
    g = pkg.S2PLSyncBlock(slots, True)
    assert g.raw_frame_size == stride
    g.pll_set_params(0.004, 4, False, True, 3)
    g.pll_set_state(0.1, 1e-4)
    a, sa = g.pll_process(fr)
    g.coarse_fed(fr, True, 4 << 2 | 1, 77)
    g.pll_set_state(0.1, 1e-4)
    b, sb = g.pll_process(fr)
    assert np.array_equal(bits(a), bits(b)) and np.array_equal(bits(sa), bits(sb))

    # device entry points: the loop enqueued on a stream, the FED with another code called behind it
    st = torch.cuda.Stream()
    many = np.concatenate([fr] * 8)
    g.pll_set_state(0.1, 1e-4)
    want, _ = g.pll_process(many)
    d_in = torch.from_numpy(f32(many).copy()).cuda()
    d_out = torch.zeros_like(d_in)
    d_err = torch.zeros(len(many), dtype=torch.float32, device="cuda")
    g.pll_set_state(0.1, 1e-4)
    g.pll_process_device(d_in.data_ptr(), len(many), stride, d_out.data_ptr(), 0, st.cuda_stream)
    pkg._check(pkg.lib().dvbs2fec_coarse_fed_device(g._p, len(many), d_in.data_ptr(), 1, 4 << 2 | 1, 262141, d_err.data_ptr(), st.cuda_stream))
    st.synchronize()
    got = d_out.cpu().numpy().view(np.complex64).reshape(len(many), stride)
    assert np.array_equal(bits(got[:, :total]), bits(want[:, :total]))
    g.close()


# ------------------------------------------------------------------------------------------------ 5. phase loop
SEQ = pll_sequence()
# closed loop, per constellation.  8PSK runs 4 dB above tests/test_gpu_pll.py: over a normal frame at 12 dB, noise puts
# enough symbols next to a decision boundary that a kick of alpha * pi / 4 moved 3-4 % of the symbols beyond 1e-3 (B200)
ESN0 = {0: 8.0, 1: 16.0, 2: 16.0, 3: 20.0}


def step_id(i):
    modcod, short, pilots = SEQ[i]
    return "%03d-mc%02d-%s-%s" % (i, modcod, "short" if short else "normal", "pilots" if pilots else "nopilots")


def closed_loop_frames(cfg, codenum, nframes, rng, esn0=None, cfo=2e-5):
    """consecutive PLFRAMEs [n][PLFRAME length] of coded random BBFRAMEs (in-tree encoder and modulator), header and
    unmodulated pilots as the transmitter sends them, PL scrambled, with a carrier offset, a phase offset and noise"""
    modcod, short, pilots = cfg
    const = MODCODS[modcod][0]
    kb = pkg.modcod_info(modcod, short)["kbch"] // 8
    pls = modcod << 2 | int(short) << 1 | int(pilots)
    rn = plstream.pl_rn(codenum)
    out = []
    for _ in range(nframes):
        sym = pkg.modulate(modcod, short, pilots, pkg.encode_fecframe(modcod, short, rng.integers(0, 256, kb, dtype=np.uint8))).view(np.complex64).copy()
        body = sym[90:]
        amp = np.float32(np.sqrt(np.mean(np.abs(body) ** 2)))
        if pilots:
            k = np.arange(len(body)) % (1440 + 36)
            body[k >= 1440] = (1 + 1j) / np.sqrt(2) * amp
        out.append(np.concatenate([plstream.plheader(pls) * amp, body * np.array([1, 1j, -1, -1j])[rn[:len(body)]]]))
    x = np.stack(out).astype(np.complex64)
    n = np.arange(x.size).reshape(x.shape)
    x = x * np.exp(1j * (0.2 + 2 * np.pi * cfo * n))
    sigma = np.abs(x[0, :90]).mean() * np.sqrt(0.5 / 10 ** ((ESN0[const] if esn0 is None else esn0) / 10))
    return (x + sigma * (rng.normal(size=x.shape) + 1j * rng.normal(size=x.shape))).astype(np.complex64)


@pytest.fixture(scope="module")
def loop():
    g = pkg.S2PLSyncBlock(36, False)
    yield g
    g.close()


def codenum_of(step):
    return (0, 1, 131071, 262141)[step] if step < 4 else (step * 40507 + 11) % 262142


@pytest.mark.parametrize("step", range(len(SEQ)), ids=step_id)
def test_phase_loop_configuration(loop, step):
    cfg = SEQ[step]
    modcod, short, pilots = cfg
    slots, total, stride, div = pll_geometry(cfg)
    codenum = codenum_of(step)
    g = loop
    rng = np.random.default_rng(5000 + step)

    # open loop: alpha = beta = 0 from (0, 0)
    fr = open_loop_frames(cfg)
    g.pll_set_params(0.0, modcod, short, pilots, codenum)
    assert g.pll_frame_symbols == total
    g.pll_set_state(0.0, 0.0)
    got, st = g.pll_process(fr, frame_stride=stride)
    want, ws = oracle_pll(cfg, 0.0, codenum, fr)
    assert np.array_equal(bits(got[:, :total]), bits(want)), "open loop: output symbols"
    assert not bits(got[:, total:]).any()
    assert np.array_equal(bits(st[:, :2]), bits(ws[:, :2])) and not bits(st[:, :2]).any(), "open loop: phase / frequency"
    if MODCODS[modcod][0] != 3:
        assert np.array_equal(bits(st[:, 2]), bits(ws[:, 2])), ("open loop: mean error", st[:, 2], ws[:, 2])
    else:
        e = open_loop_errors(cfg, fr)
        s = float_sum(e)
        tol = (4 * np.spacing(np.abs(e)).sum(axis=1) + e.shape[1] * np.spacing(np.abs(s).max(axis=1))) / div + np.spacing(np.abs(ws[:, 2]))
        assert np.all(np.abs(st[:, 2] - ws[:, 2]) <= tol), ("open loop, 32APSK: mean error", st[:, 2], ws[:, 2], tol)

    # closed loop: every frame from the oracle's state
    fr = closed_loop_frames(cfg, codenum, 2, rng)
    g.pll_set_params(0.004, modcod, short, pilots, codenum)
    ws = np.zeros(3, np.float32)
    o = orclib.oracle()
    _, ctype, _, g1, g2 = MODCODS[modcod]
    h = o.orc_pll_create(0.004, ctype, g1, g2, slots, int(pilots), modcod << 2 | int(short) << 1 | int(pilots), codenum)
    try:
        buf = np.zeros(2 * stride, np.float32)
        for f in range(len(fr)):
            g.pll_set_state(float(ws[0]), float(ws[1]))
            got, st = g.pll_process(fr[f:f + 1], frame_stride=stride)
            o.orc_pll_process(h, f32(fr[f]), buf, ws)
            want = buf[:2 * total].view(np.complex64)
            dev = np.abs(got[0, :total] - want)
            assert dev[:64].max() < 5e-6, (f, dev[:64].max())
            assert np.median(dev) < MEDIAN_SYM and np.mean(dev > TOL_SYM) < 0.02, (f, np.median(dev), np.mean(dev > TOL_SYM))
            dphi = abs((st[0, 0] - ws[0] + np.pi) % (2 * np.pi) - np.pi)
            assert dphi < 2e-2 and abs(st[0, 1] - ws[1]) < 1e-4 and abs(st[0, 2] - ws[2]) < 1e-4, (f, st[0], ws)
    finally:
        o.orc_pll_destroy(h)

    # speculative pipeline (0) == one-warp kernel (2) == sequential walk (1): in lock, and out of lock (noise and a carrier
    # offset beyond the +-0.01 pi clamp)
    wild = closed_loop_frames(cfg, codenum, 1, rng, esn0=0.0, cfo=6e-3)
    for frames in (fr, wild):
        res = []
        for mode in (1, 0, 2):
            g.pll_set_sequential(mode)
            g.pll_set_state(0.3, -2e-3)
            res.append(g.pll_process(frames, frame_stride=stride))
        g.pll_set_sequential(0)
        for k in (1, 2):
            assert np.array_equal(bits(res[0][0]), bits(res[k][0])) and np.array_equal(bits(res[0][1]), bits(res[k][1])), k


MULTI = [(4, False, False), (12, True, True), (18, False, True), (19, True, False), (20, False, False), (21, True, True),
         (22, False, True), (23, False, False), (24, True, True), (28, False, False), (1, True, True), (14, False, True),
         (11, False, True), (27, True, False)]


def test_multi_stream_every_table():
    """one launch over streams of every phase-error table, both frame sizes, pilots on and off, at a common stride:
    each stream equals its single-stream call bit for bit"""
    assert {(MODCODS[m][0], MODCODS[m][3], MODCODS[m][4]) for m, _, _ in MULTI} >= {(MODCODS[m][0], MODCODS[m][3], 0.0) for m in range(1, 24)}
    assert {(s, p) for _, s, p in MULTI} == {(False, False), (False, True), (True, False), (True, True)}
    rng = np.random.default_rng(77)
    stride = max(pll_geometry(c)[2] for c in MULTI)
    blocks, ins, outs, want = [], [], [], []
    for k, cfg in enumerate(MULTI):
        fr = closed_loop_frames(cfg, 17 * k, 2, rng)
        fr = np.pad(fr, ((0, 0), (0, stride - fr.shape[1])))
        g = pkg.S2PLSyncBlock(36, False)
        g.pll_set_params(0.004, *cfg, 17 * k)
        w, _ = g.pll_process(fr, frame_stride=stride)
        g.pll_reset()
        blocks.append(g)
        want.append(w)
        ins.append(torch.from_numpy(f32(fr).copy()).cuda())
        outs.append(torch.zeros_like(ins[-1]))
    pkg.pll_process_multi_device(blocks, [t.data_ptr() for t in ins], 2, stride, [t.data_ptr() for t in outs],
                                 torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    for cfg, g, w, o in zip(MULTI, blocks, want, outs):
        assert np.array_equal(bits(o.cpu().numpy()), bits(w)), cfg
        g.close()


# ------------------------------------------------------------------------------------------------ 6. PL sync
@pytest.mark.parametrize("case", [(36, True, 12.0, 6), (45, False, 3.0, 7), (45, True, 8.0, 8), (60, False, 16.0, 9), (60, True, 1.0, 10),
                                  (144, False, 6.0, 11), (180, False, 2.0, 12), (180, True, 10.0, 13), (240, False, 5.0, 14),
                                  (240, True, 0.0, 15)])
def test_sync_matches_oracle_remaining_geometries(case):
    """as tests/test_gpu_plsync.py::test_sync_matches_oracle, on the ten geometries it does not run"""
    slots, pilots, esn0, seed = case
    rng = np.random.default_rng(40 + seed)
    x = plstream.stream(11 << 2 | pilots, slots, pilots, 6, rng, esn0_db=esn0, lead=int(rng.integers(1, 3000)), cfo=2e-5 * seed)
    o = OrcSync(slots, pilots)
    g = pkg.S2PLSyncBlock(slots, pilots)
    assert g.raw_frame_size == o.rfs
    c = sorted(set(int(c) for c in rng.integers(0, len(x), 9)) | {0, len(x)})
    for a, b in zip(c[:-1], c[1:]):
        want, got = o.process(x[a:b]), g.process(x[a:b])
        assert len(want) == len(got) and np.array_equal(bits(want), bits(got))
        assert (g.current_position, g.best_match) == o.stats()[1:]
    g.close()


# ------------------------------------------------------------------------------------------------ 7. one-call stage
# One MODCOD per geometry, then until every 16APSK and 32APSK gamma has been used.  With pilots on, S2PLLBlock handles
# (slots + 1) * 90 + 36 symbols of a frame (one pilot block, counted from the slot number: SURVEY.md note N2), so the
# symbols behind them reach the demapper neither derotated nor descrambled; the 8/9 and 9/10 codes do not survive that
# loss, so they run here with pilots off.
STAGE = [(4, False, False), (7, False, True), (1, True, False), (10, True, True), (12, False, False), (15, False, True),
         (13, True, False), (16, True, True), (23, False, False), (18, False, True), (19, True, False), (20, True, True),
         (28, False, False), (24, False, True), (25, True, False), (26, True, True),
         (21, False, False), (22, True, False), (27, False, False),
         (2, True, True), (11, False, False), (14, False, False), (17, False, False), (5, True, False)]
STAGE_ESN0 = {0: 14.0, 1: 18.0, 2: 22.0, 3: 26.0}


def test_stage_cases_cover_every_geometry_and_gamma():
    geo = set()
    for m, s, p in STAGE:
        info = pkg.modcod_info(m, s, p)
        geo.add((info["nldpc"] // info["bits"] // 90, p))
    assert geo == set(GEOMETRIES)
    assert {m for m, _, _ in STAGE} >= set(range(18, 29))


@pytest.mark.parametrize("k", range(len(STAGE)), ids=lambda k: "mc%02d-%s-%s" % (STAGE[k][0], "short" if STAGE[k][1] else "normal",
                                                                                 "pilots" if STAGE[k][2] else "nopilots"))
def test_s2_demod_stage_every_geometry(k):
    """dvbs2fec_s2_demod_process over two calls cut inside a frame: BBFRAMEs, results, FED values and PLHEADER fields
    equal, bit for bit, to the stages called one after the other through their host entry points; the transmitted
    payloads come back"""
    modcod, short, pilots = STAGE[k]
    codenum = (k * 7919) % 262142
    rng = np.random.default_rng(600 + k)
    n = 5
    dec = pkg.DVBS2Decoder(max_batch=16)
    dec.setDemodParams(modcod, short, pilots, 25)
    info = pkg.modcod_info(modcod, short, pilots)
    pay = rng.integers(0, 256, (n, dec.kbch // 8), dtype=np.uint8)
    pls = modcod << 2 | int(short) << 1 | int(pilots)
    rn = plstream.pl_rn(codenum)
    frames = []
    for i in range(n):
        sym = pkg.modulate(modcod, short, pilots, pkg.encode_fecframe(modcod, short, pay[i])).view(np.complex64).copy()
        body = sym[90:]
        amp = np.float32(np.sqrt(np.mean(np.abs(body) ** 2)))
        if pilots:
            j = np.arange(len(body)) % (1440 + 36)
            body[j >= 1440] = (1 + 1j) / np.sqrt(2) * amp
        frames.append(np.concatenate([plstream.plheader(pls) * amp, body * np.array([1, 1j, -1, -1j])[rn[:len(body)]]]))
    amp = np.abs(frames[0][:90]).mean()
    x = np.concatenate([0.3 * amp * (rng.normal(size=1500) + 1j * rng.normal(size=1500))] + frames + [frames[0][:300]]).astype(np.complex64)
    x = x * np.exp(1j * (0.4 + 2 * np.pi * 1.5e-5 * np.arange(len(x))))
    sigma = amp * np.sqrt(0.5 / 10 ** (STAGE_ESN0[MODCODS[modcod][0]] / 10))
    x = (x + sigma * (rng.normal(size=len(x)) + 1j * rng.normal(size=len(x)))).astype(np.complex64)
    rfs = info["plframe_symbols"]
    cut = 1500 + 2 * rfs + rfs // 3          # inside the third frame
    slots = info["nldpc"] // info["bits"] // 90
    h = pkg.S2PLSyncBlock(slots, pilots)
    assert h.raw_frame_size == rfs
    h.plhdr_set_params(0.004)
    h.pll_set_params(0.004, modcod, short, pilots, codenum)
    want = []
    for seg in (x[:cut], x[cut:]):
        fr = h.process(seg).reshape(-1, rfs)
        if not len(fr):
            want.append(None)
            continue
        fed = h.coarse_fed(fr, pilots, pls, codenum)
        out, _ = h.pll_process(fr)
        _, hres, _ = h.plhdr_process(fr)
        bb, res = dec.decode_plframes(out.view(np.float32).reshape(len(fr), -1))
        want.append((bb, res, np.asarray(fed, np.float32), hres))
    h.close()
    g = pkg.DVBS2DemodStage(max_batch=16)
    g.setDemodParams(modcod, short, pilots, 25, 0.004, 0.004, codenum)
    got_bb = []
    for seg, w in zip((x[:cut], x[cut:]), want):
        bb, res, fed, hres = g.process(seg)
        if w is None:
            assert len(bb) == 0
            continue
        assert np.array_equal(bb, w[0])
        for key in ("ldpc_iters", "bch_corr", "flags"):
            assert np.array_equal(res[key], w[1][key]), key
        assert np.array_equal(bits(fed), bits(w[2])) and np.array_equal(hres, w[3])
        got_bb.append(bb)
    got_bb = np.concatenate(got_bb)
    assert len(got_bb) >= n - 1
    good = sum(any(np.array_equal(b, p) for p in pay) for b in got_bb)
    assert good >= len(got_bb) - 1, (good, len(got_bb))      # (the first frame: the loop may still be pulling in)
    g.close()
    dec.close()
