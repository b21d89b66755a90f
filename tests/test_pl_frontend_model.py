"""Host-only half of tests/test_gpu_pl_frontend.py: the constructions the GPU test feeds the PL front end (K7 PLHEADER
decoding, K8 payload phase loop), checked against the CPU oracle alone, so that what the GPU test expects is right
before a device is involved.

* the 128 PLS codewords restated here equal the ones the oracle's header symbols carry;
* the crafted PLHEADER words (clean, bits 63..60 flipped, 1..13 errors, ties, random words) decode through
  `orc_plhdr_process` to the index the GPU test expects, and the ties are ties;
* the payload phase loop's pilot rule (positions k % 1474 >= 1439 of the payload are judged against the diagonals) and
  its frame length per geometry;
* with the loop open (alpha = beta = 0), the oracle's mean error is the float32 sum, in order, of the phase-error table
  cells (32APSK: of `orc_demod_phase_error_calc`) of the probes, divided by the divisor."""
import numpy as np
import pytest

import orclib
import plstream
from fec import pkg, MODCODS
from test_gpu_demapper import configurations, lut_coords, odd_values, oracle_constellation

A = np.float32(0.70710677)          # pi/2-BPSK diagonal: float(cos(pi/4))
MASK60 = np.uint64((1 << 60) - 1)   # checkSyncMarker compares bits 59..0
GEOMETRIES = [(s, p) for s in (36, 45, 60, 90, 144, 180, 240, 360) for p in (False, True)]


# ------------------------------------------------------------------------------------------------ PLHEADER words
def codewords():
    """EN 302 307 §5.5.2.4: the 32-bit first-order Reed-Muller word of the PLS code's 6 MSBs, each bit repeated (b0 = 0)
    or followed by its inverse (b0 = 1), scrambled with 0x719d83c953422dfa"""
    G = (0x55555555, 0x33333333, 0x0F0F0F0F, 0x00FF00FF, 0x0000FFFF, 0xFFFFFFFF)
    out = np.zeros(128, np.uint64)
    for c in range(128):
        y = 0
        for row in range(6):
            if (c >> (6 - row)) & 1:
                y ^= G[row]
        w = 0
        for bit in range(31, -1, -1):
            yi = (y >> bit) & 1
            w = (w << 2) | (yi << 1) | (yi ^ (c & 1))
        out[c] = w ^ 0x719D83C953422DFA
    return out


CODEWORDS = codewords()


def distances(words):
    """[n] words -> [n][128] Hamming distances to the codewords over bits 59..0"""
    return np.bitwise_count((np.asarray(words, np.uint64)[:, None] ^ CODEWORDS[None, :]) & MASK60).astype(np.int32)


def decode(words):
    """the reference's decision: the first codeword among those nearest over bits 59..0"""
    return np.argmin(distances(words), axis=1)


def fields(c):
    c = np.asarray(c, np.int32)
    return np.stack([(c >> 2) & 31, (c >> 1) & 1, c & 1, c], axis=-1)


def _tie(c1, c2, rng):
    """a word at equal distance from codewords c1 and c2 and no nearer to any other: from c1, half of the bits in 59..0
    where they differ are moved to c2 (odd distance: one fewer, plus one bit where both agree)"""
    diff = [b for b in range(60) if (int(CODEWORDS[c1] ^ CODEWORDS[c2]) >> b) & 1]
    same = [b for b in range(60) if b not in diff]
    for _ in range(200):
        flip = list(rng.choice(diff, len(diff) // 2, replace=False))
        if len(diff) % 2:
            flip.append(int(rng.choice(same)))
        w = int(CODEWORDS[c1])
        for b in flip:
            w ^= 1 << int(b)
        d = distances([w])[0]
        if d[c1] == d[c2] == d.min():
            return np.uint64(w)
    raise AssertionError("no tie found for %d, %d" % (c1, c2))


# pairs whose tie crosses the kernel's lane split (codeword c is held by lane c % 32 as its (c // 32)-th candidate)
LANE_PAIRS = [(c, c + 32) for c in range(96)] + [(c, c + 64) for c in range(0, 64, 7)] + \
             [(1, 64), (31, 32), (33, 96), (2, 99), (63, 64), (95, 96), (5, 66), (40, 97), (0, 127), (30, 65)]


def crafted_words(seed=11):
    """(words [n] uint64, kind [n] str, partner pairs [n][2] (ties) or -1) -- every codeword clean, with bits 63..60
    flipped, with 1..13 errors in 59..0; ties on LANE_PAIRS and three random pairs per codeword (each codeword is the
    lower index of some ties and the higher of others); random words, among which ties of three or more"""
    rng = np.random.default_rng(seed)
    words, kinds, pairs = [], [], []

    def add(w, kind, pair=(-1, -1)):
        words.append(np.uint64(w)); kinds.append(kind); pairs.append(pair)

    for c in range(128):
        add(CODEWORDS[c], "clean")
        add(CODEWORDS[c] ^ np.uint64(int(rng.integers(1, 16)) << 60), "bits 63..60")
        add(CODEWORDS[c] ^ np.uint64(0xF << 60), "bits 63..60")
        for k in (1 + c % 13, 13):
            e = 0
            for b in rng.choice(60, k, replace=False):
                e |= 1 << int(b)
            add(CODEWORDS[c] ^ np.uint64(e), "%d errors" % k)
    # (a pair at distance 60 -- the PLS codes that differ in the frame-size bit only -- has no word nearer to both than
    # to every other codeword)
    near = distances(CODEWORDS) <= 32
    ties = [p for p in LANE_PAIRS if near[p]]
    for c in range(128):
        for o in rng.choice([x for x in range(128) if x != c and near[c, x]], 3, replace=False):
            ties.append((min(c, int(o)), max(c, int(o))))
    for c1, c2 in ties:
        add(_tie(c1, c2, rng), "tie", (c1, c2))
    for w in rng.integers(0, 2 ** 63, 400, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, 400, dtype=np.uint64):
        add(w, "random")
    return np.array(words, np.uint64), np.array(kinds), np.array(pairs, np.int32)


def header_symbols(words, rng):
    """words [n] -> header symbols [n][90] that, with the loop at phase 0, come out as pi/2-BPSK diagonal points whose
    hard decisions spell the word (bit 63 first): a 0 bit is o = (a, a); a 1 bit is (-a, -a), (a, -a) or (-a, a) -- the
    last two on the decision boundary, where cmul(o, rot).re is exactly 0.  The kernel's output mapping is inverted
    (odd i: o = (-t.re, t.im); even i: o = (t.im, t.re)).  Every t is a diagonal point, so the loop error is exactly 0."""
    words = np.asarray(words, np.uint64)
    n = len(words)
    bits = ((words[:, None] >> np.arange(63, -1, -1, dtype=np.uint64)) & np.uint64(1)).astype(bool)
    o = np.empty((n, 90, 2), np.float32)
    o[:, :26] = rng.choice(np.array([A, -A], np.float32), (n, 26, 2))
    ones = np.array([[-A, -A], [A, -A], [-A, A]], np.float32)
    o[:, 26:] = np.where(bits[..., None], ones[rng.integers(0, 3, (n, 64))], np.array([A, A], np.float32))
    t = np.empty_like(o)
    odd = (np.arange(90) & 1) == 1
    t[:, odd, 0], t[:, odd, 1] = -o[:, odd, 0], o[:, odd, 1]
    t[:, ~odd, 0], t[:, ~odd, 1] = o[:, ~odd, 1], o[:, ~odd, 0]
    return np.ascontiguousarray(t).view(np.complex64)[..., 0], np.ascontiguousarray(o).view(np.complex64)[..., 0]


def header_frames(words, rfs, rng):
    """PLFRAMEs [n][rfs] with the crafted header and NaN behind it (the PLHEADER decoder reads the first 90 symbols)"""
    t, o = header_symbols(words, rng)
    fr = np.full((len(words), rfs), np.complex64(complex(np.nan, np.nan)), np.complex64)
    fr[:, :90] = t
    return fr, o


def oracle_plhdr(frames, rfs, bw=0.004, h=None):
    """orc_plhdr_process over the frames in order -> (headers [n][90], fields [n][3], loop state after each [n][2])"""
    o = orclib.oracle()
    own = h is None
    if own:
        h = o.orc_plhdr_create(bw)
    n = len(frames)
    hd, res, loop = np.zeros((n, 90), np.complex64), np.zeros((n, 3), np.int32), np.zeros((n, 2), np.float32)
    for k in range(n):
        o.orc_plhdr_process(h, rfs, np.ascontiguousarray(frames[k]).view(np.float32), hd[k].view(np.float32), res[k], loop[k])
    if own:
        o.orc_plhdr_destroy(h)
    return hd, res, loop


def noisy_header_stream(slots, pilots, codes, rng, esn0=(3.0, 10.0), max_cfo=1e-4, max_phase=0.4):
    """PLFRAMEs [n][rfs] of the given PLS codes (QPSK payload, PL scrambled with code 0), each with its own phase offset
    and carrier offset (up to max_cfo cycles per symbol, from the frame's first symbol) and Gaussian noise at alternating
    Es/N0"""
    rn = plstream.pl_rn(0)
    rfs = orclib.oracle().orc_raw_frame_size(slots, int(pilots))
    out = np.empty((len(codes), rfs), np.complex64)
    n = np.arange(rfs)
    for k, c in enumerate(codes):
        x = plstream.plframe(int(c), slots, pilots, rng, rn)
        assert len(x) == rfs
        x = x * np.exp(1j * (rng.uniform(-max_phase, max_phase) + 2 * np.pi * rng.uniform(-max_cfo, max_cfo) * n))
        sigma = np.sqrt(0.5 / 10 ** (esn0[k % len(esn0)] / 10))
        out[k] = x + sigma * (rng.normal(size=rfs) + 1j * rng.normal(size=rfs))
    return out


def noisy_header_plan(gi, seed=0):
    """geometry gi of GEOMETRIES: its share of the 128 codes (gi, gi + 16, ...), three frames each, shuffled"""
    rng = np.random.default_rng(900 + 16 * seed + gi)
    codes = rng.permutation(np.repeat(np.arange(gi, 128, 16), 3))
    slots, pilots = GEOMETRIES[gi]
    return codes, noisy_header_stream(slots, pilots, codes, rng), rng


# ------------------------------------------------------------------------------------------------ payload phase loop
def pll_key(cfg):
    """what selects the loop's phase-error table: constellation and gammas"""
    const, _, _, g1, g2 = MODCODS[cfg[0]]
    return const, g1, g2


def pll_sequence():
    """the 104 configurations, the phase-error table (constellation or gamma) changing at every step, then the first one
    again (greedy: the largest group left that differs from the previous step)"""
    groups = {}
    for c in configurations():
        groups.setdefault(pll_key(c), []).append(c)
    seq, last = [], max(groups, key=lambda k: (len(groups[k]), k))   # start elsewhere: the repeat must differ from the end
    while any(groups.values()):
        k = max((k for k, g in groups.items() if g and k != last), key=lambda k: (len(groups[k]), k))
        seq.append(groups[k].pop(0))
        last = k
    return seq + [seq[0]]


def pll_geometry(cfg):
    """(slots, symbols the loop handles per frame, PLFRAME length, divisor) of a configuration: S2PLLBlock counts one
    pilot block for every slot count below 1620 (dvbs2_pll.h:47-59)"""
    modcod, short, pilots = cfg
    info = pkg.modcod_info(modcod, short, pilots)
    slots = info["nldpc"] // info["bits"] // 90
    total = (slots + 1) * 90 + (36 if pilots else 0)
    return slots, total, info["plframe_symbols"], np.float32((slots + 1) * 90 + (36 if pilots else 0))


def diagonal_positions(total, pilots):
    """payload positions (from the first payload symbol) the reference's pilot counter judges against the diagonals:
    k % 1474 >= 1439, pilots only"""
    k = np.arange(total - 90)
    return (k % 1474 >= 1439) if pilots else np.zeros(total - 90, bool)


def lut_probes(rng):
    """every cell centre; the floats just below, at and above each of the 257 cell edges on either axis (the other
    coordinate a random centre); finite odd values on either axis.  No inf or NaN: x * (-0) makes NaN of them, and NaN
    payload bits are not specified"""
    c = ((np.arange(256) - 127.5) / 256 * 1.5).astype(np.float32)
    x, y = np.meshgrid(c, c, indexing="ij")
    v = odd_values()
    v = v[np.isfinite(v)]
    out = [np.stack([x.ravel(), y.ravel()], axis=1), np.stack([v, rng.choice(c, len(v))], axis=1), np.stack([rng.choice(c, len(v)), v], axis=1)]
    return np.concatenate(out).astype(np.float32)


_OPEN = {}


def open_loop_frames(cfg):
    """probe frames [n][PLFRAME length] complex64 of a configuration, for the loop with alpha = beta = 0 at phase 0:
    the oracle's own PLHEADER of the configuration's PLS code; at the diagonal positions (a, -a) or (-a, a) -- exactly on
    a diagonal after any descrambling (error exactly 0) but, in the table, in a cell with a nonzero error, so a shifted
    window changes the error sum; elsewhere the probes.  LUT configurations sharing a table share the probes of
    lut_probes() between them; 32APSK gets noisy constellation symbols and points of a grid over +-1.5.  NaN behind the
    symbols the loop reads."""
    if cfg in _OPEN:
        return _OPEN[cfg]
    key = pll_key(cfg)
    group = [c for c in configurations() if pll_key(c) == key]
    rng = np.random.default_rng(4242 + 7 * cfg[0])
    slots_n = {c: int((~diagonal_positions(pll_geometry(c)[1], c[2])).sum()) for c in group}
    if key[0] == 3:
        want = {c: slots_n[c] for c in group}
        probes = None
    else:
        probes = rng.permutation(lut_probes(rng))
        rounds = -(-len(probes) // sum(slots_n.values()))
        need = rounds * sum(slots_n.values())
        probes = np.concatenate([probes, probes[rng.integers(0, len(probes), need - len(probes))]])
    at = 0
    for c in group:
        modcod, short, pilots = c
        slots, total, stride, _ = pll_geometry(c)
        diag = diagonal_positions(total, pilots)
        if probes is not None:
            nfr = rounds
            pay = probes[at: at + nfr * slots_n[c]].reshape(nfr, slots_n[c], 2)
            at += nfr * slots_n[c]
        else:
            nfr = 2
            kb = pkg.modcod_info(modcod, short)["kbch"] // 8
            pay = np.empty((nfr, slots_n[c], 2), np.float32)
            for f in range(nfr):
                s = pkg.modulate(modcod, short, False, pkg.encode_fecframe(modcod, short, rng.integers(0, 256, kb, dtype=np.uint8)))
                s = s.view(np.float32).reshape(-1, 2)[90: 90 + slots_n[c]]
                pay[f] = s + rng.normal(0, 0.05 * (f + 1), s.shape)
                grid = rng.uniform(-1.5, 1.5, (slots_n[c] // 4, 2))
                pay[f, 3::4][: len(grid)] = grid[: len(pay[f, 3::4])]
        pls = modcod << 2 | int(short) << 1 | int(pilots)
        fr = np.full((nfr, stride, 2), np.nan, np.float32)
        fr[:, :90] = plstream.plheader(pls).view(np.float32).reshape(90, 2)
        body = np.empty((nfr, total - 90, 2), np.float32)
        s = rng.choice(np.array([-1, 1], np.float32), (nfr, int(diag.sum())))
        body[:, diag, 0], body[:, diag, 1] = s * A, -s * A
        body[:, ~diag] = pay
        fr[:, 90:total] = body
        _OPEN[c] = np.ascontiguousarray(fr).view(np.complex64)[..., 0]
    return _OPEN[cfg]


def oracle_pll(cfg, bw, codenum, frames, state=None):
    """orc_pll_create with the MODCOD's own gammas, frames in order -> (outputs [n][total], states [n][3]); `state`:
    a list of (phase, freq) to start each frame from instead of carrying the loop over (None: carried over)"""
    modcod, short, pilots = cfg
    _, ctype, _, g1, g2 = MODCODS[modcod]
    slots, total, _, _ = pll_geometry(cfg)
    o = orclib.oracle()
    h = o.orc_pll_create(bw, ctype, g1, g2, slots, int(pilots), modcod << 2 | int(short) << 1 | int(pilots), codenum)
    try:
        assert (slots + 1) * 90 + o.orc_pll_pilot_cnt(h) * 36 == total
        outs, sts = np.zeros((len(frames), total), np.complex64), np.zeros((len(frames), 3), np.float32)
        buf = np.zeros(2 * frames.shape[1], np.float32)
        for k in range(len(frames)):
            assert o.orc_pll_process(h, np.ascontiguousarray(frames[k]).view(np.float32), buf, sts[k]) == total
            outs[k] = buf[: 2 * total].view(np.complex64)
        return outs, sts
    finally:
        o.orc_pll_destroy(h)


def open_loop_errors(cfg, frames):
    """per-symbol errors [n][total] of the open loop at phase 0: 0 for header and diagonal positions; the oracle's
    table cell of the probe (lut_coords: the reference's double index), or orc_demod_phase_error_calc for 32APSK"""
    modcod, short, pilots = cfg
    slots, total, _, _ = pll_geometry(cfg)
    diag = diagonal_positions(total, pilots)
    pay = np.ascontiguousarray(frames[:, 90:total]).view(np.float32).reshape(len(frames), total - 90, 2)
    e = np.zeros((len(frames), total), np.float32)
    c = oracle_constellation(modcod)
    o = orclib.oracle()
    if MODCODS[modcod][0] == 3:
        for f in range(len(frames)):
            e[f, 90:][~diag] = [o.orc_demod_phase_error_calc(c, float(a), float(b)) for a, b in pay[f][~diag]]
    else:
        lut = np.ctypeslib.as_array(o.orc_const_phase_lut(c), shape=(256, 256)).copy()
        ix = lut_coords(pay).astype(np.intp)
        e[:, 90:] = np.where(diag[None], np.float32(0), lut[ix[..., 0], ix[..., 1]])
    return e


def float_sum(e):
    """the reference's running float sum, in order"""
    return np.cumsum(e, axis=-1, dtype=np.float32)


# ------------------------------------------------------------------------------------------------ tests
def test_codewords_are_the_oracles():
    o = orclib.oracle()
    for c in range(128):
        h = plstream.plheader(c)[26:]
        assert np.all(np.abs(np.abs(h.imag) - np.float32(1 / np.sqrt(2))) < 1e-7)
        bits = (h.imag < 0).astype(np.uint64)        # im = (1 - 2 y_i) / sqrt 2
        assert int((bits << np.arange(63, -1, -1, dtype=np.uint64)).sum()) == int(CODEWORDS[c]) == o.orc_pls_codeword(c), c
    d = distances(CODEWORDS)
    assert (np.diag(d) == 0).all() and d[~np.eye(128, dtype=bool)].min() >= 28      # 13 errors in 59..0 still decode


def test_crafted_words_decode_through_the_oracle():
    words, kinds, pairs = crafted_words()
    rng = np.random.default_rng(1)
    for slots, pilots in (GEOMETRIES[0], GEOMETRIES[3]):
        rfs = orclib.oracle().orc_raw_frame_size(slots, int(pilots))
        fr, o = header_frames(words, rfs, rng)
        hd, res, loop = oracle_plhdr(fr, rfs)
        assert np.array_equal(hd.view(np.uint32), o.view(np.uint32))     # the loop stays at rest: headers exact
        assert not loop.view(np.uint32).any()
        want = decode(words)
        assert np.array_equal(res, fields(want)[:, :3])
    idx = np.arange(128)
    assert np.array_equal(want[kinds == "clean"], idx)
    assert np.array_equal(want[kinds == "bits 63..60"], np.repeat(idx, 2))
    assert np.array_equal(want[np.char.endswith(kinds, "errors")], np.repeat(idx, 2))
    assert {k for k in kinds if k.endswith("errors")} == {"%d errors" % k for k in range(1, 14)}
    tie = kinds == "tie"
    d = distances(words[tie])
    for row, (c1, c2), w in zip(d, pairs[tie], want[tie]):
        m = np.flatnonzero(row == row.min())
        assert c1 in m and c2 in m and w == m[0]
    # every codeword is the lower index of a tie and the higher one of another; ties that cross lanes both ways
    assert set(pairs[tie][:, 0]) | set(pairs[tie][:, 1]) == set(range(128))
    lane = pairs[tie] % 32
    assert (lane[:, 0] == lane[:, 1]).any() and (lane[:, 0] > lane[:, 1]).any() and (lane[:, 0] < lane[:, 1]).any()
    d = distances(words)
    assert max(np.count_nonzero(r == r.min()) for r in d) >= 3                    # a tie among three or more
    # the boundary symbols are there, and they decide 1 as the reference's `> 0` does
    assert np.any(np.isclose(o[:, 26:].real, A) & np.isclose(o[:, 26:].imag, -A))
    assert np.any(np.isclose(o[:, 26:].real, -A) & np.isclose(o[:, 26:].imag, A))


def test_noisy_headers_decode_to_the_transmitted_codes_in_the_oracle():
    """the GPU test's noisy frames: every code 0..127, the oracle decodes each to the transmitted code"""
    seen = set()
    for gi, (slots, pilots) in enumerate(GEOMETRIES):
        codes, fr, _ = noisy_header_plan(gi)
        rfs = fr.shape[1]
        _, res, _ = oracle_plhdr(fr, rfs)
        assert np.array_equal(res, fields(codes)[:, :3]), (slots, pilots)
        seen |= set(codes.tolist())
    assert seen == set(range(128))


def test_pll_sequence_changes_the_table_at_every_step():
    seq = pll_sequence()
    assert sorted(seq[:-1]) == sorted(configurations()) and len(seq) == 105 and seq[-1] == seq[0]
    assert all(pll_key(a) != pll_key(b) for a, b in zip(seq, seq[1:]))
    assert len({pll_key(c) for c in seq}) == 8 + 5      # eight tables, five 32APSK gamma pairs


@pytest.mark.parametrize("slots,pilots", GEOMETRIES)
def test_pilot_rule_and_frame_length(slots, pilots):
    """S2PLLBlock handles (slots + 1) * 90 symbols plus one pilot block of 36 (pilot_cnt is 1 for every slot count used by
    DVB-S2); a probe at payload position k is judged against the diagonals exactly where k % 1474 >= 1439"""
    o = orclib.oracle()
    h = o.orc_pll_create(0.0, 1, 0.0, 0.0, slots, int(pilots), 4 << 2 | int(pilots), 0)
    try:
        assert o.orc_pll_pilot_cnt(h) == int(pilots)
        total = (slots + 1) * 90 + 36 * int(pilots)
        c = oracle_constellation(4)
        lut = np.ctypeslib.as_array(o.orc_const_phase_lut(c), shape=(256, 256))
        diag = diagonal_positions(total, pilots)
        probe = np.array([[0.5, 0.2]], np.float32)
        e_lut = lut[tuple(lut_coords(probe)[0].astype(np.intp))]
        assert e_lut != 0
        base = np.full((total, 2), A, np.float32)     # (a, a): zero error in the table and against the diagonals
        base[:90] = plstream.plheader(4 << 2 | int(pilots)).view(np.float32).reshape(90, 2)
        ks = sorted({0, 1438, 1439, 1440, 1472, 1473, 1474, 2912, 2913, 2947, 2948, total - 91} & set(range(total - 90)))
        st, out = np.zeros(3, np.float32), np.zeros(2 * total, np.float32)
        for k in ks:
            fr = base.copy()
            fr[90 + k] = probe
            o.orc_pll_process(h, fr.reshape(-1), out, st)
            is_lut = st[2] == np.float32(e_lut / np.float32(total))
            assert is_lut != diag[k], (k, st[2], e_lut)
    finally:
        o.orc_pll_destroy(h)


@pytest.mark.parametrize("cfg", configurations(), ids=lambda c: "mc%02d-%s-%s" % (c[0], "short" if c[1] else "normal", "pilots" if c[2] else "nopilots"))
def test_open_loop_model(cfg):
    """the oracle's open loop (alpha = beta = 0) on the probe frames: outputs are the input descrambled, phase and
    frequency stay exactly 0, and the mean error of each frame is the float32 running sum of open_loop_errors over the
    divisor, bit for bit"""
    fr = open_loop_frames(cfg)
    slots, total, stride, div = pll_geometry(cfg)
    assert fr.shape[1] == stride and np.isfinite(fr[:, :total]).all() and np.isnan(fr[:, total:]).all()
    outs, sts = oracle_pll(cfg, 0.0, 5, fr)
    assert not sts[:, :2].view(np.uint32).any()
    rn = plstream.pl_rn(5)[: total - 90]
    assert np.array_equal(outs[:, 90:], fr[:, 90:total] * np.array([1, -1j, -1, 1j], np.complex64)[rn])   # descrambled, not rotated
    e = open_loop_errors(cfg, fr)
    want = float_sum(e)[:, -1] / div
    assert np.array_equal(sts[:, 2].view(np.uint32), want.astype(np.float32).view(np.uint32)), (sts[:, 2], want)
    diag = diagonal_positions(total, cfg[2])
    if cfg[2]:
        # the diagonal symbols sit in cells whose table error is not 0: a window shifted by one changes the sum
        if MODCODS[cfg[0]][0] != 3:
            o = orclib.oracle()
            lut = np.ctypeslib.as_array(o.orc_const_phase_lut(oracle_constellation(cfg[0])), shape=(256, 256))
            ix = lut_coords(np.ascontiguousarray(fr[:, 90:total]).view(np.float32).reshape(len(fr), -1, 2)).astype(np.intp)
            first = np.flatnonzero(diag)[0]
            assert np.all(lut[ix[:, first, 0], ix[:, first, 1]] != 0)


def test_open_loop_probes_cover_every_cell_and_edge():
    """over the configurations sharing a table, the probes visit every cell centre and every edge value"""
    groups = {}
    for c in configurations():
        if MODCODS[c[0]][0] != 3:
            groups.setdefault(pll_key(c), []).append(c)
    assert len(groups) == 8
    edge = ((np.arange(257) - 128) * 1.5 / 256).astype(np.float32)
    need = np.concatenate([edge, np.nextafter(edge, np.float32(-np.inf)), np.nextafter(edge, np.float32(np.inf))]).view(np.uint32)
    for key, cfgs in groups.items():
        pay = []
        for c in cfgs:
            _, total, _, _ = pll_geometry(c)
            diag = diagonal_positions(total, c[2])
            pay.append(np.ascontiguousarray(open_loop_frames(c)[:, 90:total][:, ~diag]).view(np.float32).reshape(-1, 2))
        pay = np.concatenate(pay)
        ix = lut_coords(pay).astype(np.int32)
        assert len(np.unique(ix[:, 0] * 256 + ix[:, 1])) == 65536, key
        for axis in (0, 1):
            assert np.isin(need, pay[:, axis].view(np.uint32)).all(), (key, axis)
