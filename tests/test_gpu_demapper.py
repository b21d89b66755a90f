"""K1, the demapper (`demap_kernel` / `demap_idx_kernel`), against the CPU oracle on every (MODCOD, frame size, pilots)
configuration: the 104 that `set_modcod` accepts (28 MODCODs x normal / short x pilots off / on, minus the short 9/10 rates).

One decoder runs the whole matrix, in an order in which the constellation, the 16APSK gamma or the frame size changes at
every step, and the first configuration runs again at the end: a LUT or demapper descriptor left over from the previous
MODCOD, or cached under the wrong key, fails a step.  Per configuration:

* the reference is the oracle's `orc_bb_to_soft` (pilots off).  Pilots-on frames reach it with the pilot blocks removed
  by this file's own statement of EN 302 307 §5.5.3; the PLHEADER and every pilot position are poisoned (NaN, or a
  corner-cell value) so that reading one of them changes an LLR;
* QPSK / 8PSK / 16APSK: all 65 536 LUT cell centres, shuffled over deinterleaver columns and pilot-block offsets, plus
  the floats just below, at and above each of the 257 cell edges of either axis and odd values (+-0, subnormals,
  far outside the grid, +-inf, NaN): LLR bytes bit for bit, and `quantize_plframes` against the same double
  expression in numpy.  Together the steps pin all eight distinct host-built LUTs, through the device;
* 32APSK (no LUT: per-symbol expf / logf): the DESIGN §1 tolerance on noisy frames at several sigma, on a grid over
  +-1.5 on each axis, and on a radial far field from 1.5x to 4x the outer ring, which crosses the band where the exp
  terms become subnormal and then zero.  LDPC, BCH and BBFRAME behind the device LLRs equal the oracle run on those LLRs;
* two noisy frames through `decode_plframes` against the oracle chain, and through
  `decode_plframes_idx(quantize_plframes(x))`;
* all of it again PL-scrambled with `set_pl_scrambling(codenum)`: the same LLRs, coordinates and frames.

`test_launches_of_more_than_65535_frames` runs the three entry points whose launches put frames in the grid's y
dimension with 65 600 frames in one launch."""
import ctypes as C

import numpy as np
import pytest

import orclib
from fec import pkg, MODCODS

SHORT_9_10 = {11, 17, 23, 28}   # 9/10 has no short-frame code (EN 302 307 Table 5b)
SIGMAS = {0: (0.14, 0.17), 1: (0.14, 0.20), 2: (0.08, 0.12)}   # noisy frames of the whole-stage check, per constellation
SIGMAS_32APSK = (0.02, 0.05, 0.08, 0.11)
CODENUMS = (0, 1, 131071, 262141)   # PL scrambling code numbers of the first steps; later steps spread over 0..262141


def configurations():
    """(modcod, short, pilots) for which modcod_info answers, in enumeration order"""
    out = []
    for modcod in range(1, 29):
        for short in (False, True):
            for pilots in (False, True):
                try:
                    pkg.modcod_info(modcod, short, pilots)
                except pkg.DVBS2FecError:
                    continue
                out.append((modcod, short, pilots))
    return out


def table_key(cfg):
    """what selects the demapper's tables: the constellation, the 16APSK gamma, the frame size"""
    modcod, short, _ = cfg
    const, _, _, g1, _ = MODCODS[modcod]
    return const, g1 if const == 2 else 0.0, short


def ordered(cfgs):
    """every configuration once, the table key changing at every step (greedy: the largest group left that differs
    from the previous step), then the first one again"""
    groups = {}
    for c in cfgs:
        groups.setdefault(table_key(c), []).append(c)
    for g in groups.values():   # pilots alternate inside a group as well
        g.sort(key=lambda c: (c[2], c[0]))
        g[:] = [x for pair in zip(g[: len(g) // 2], g[len(g) // 2:]) for x in pair] + g[2 * (len(g) // 2):]
    seq, last = [], max(groups, key=lambda k: (len(groups[k]), k))   # start elsewhere: the repeat must differ from the end
    while any(groups.values()):
        k = max((k for k, g in groups.items() if g and k != last), key=lambda k: (len(groups[k]), k))
        seq.append(groups[k].pop(0))
        last = k
    return seq + [seq[0]]


SEQUENCE = ordered(configurations())


def step_id(i):
    modcod, short, pilots = SEQUENCE[i]
    return "%03d-mc%02d-%s-%s" % (i, modcod, "short" if short else "normal", "pilots" if pilots else "nopilots")


def payload_positions(nsym, pilots):
    """raw PLFRAME positions of the payload symbols, and the PLFRAME length (EN 302 307 §5.5.3): the 90-symbol PLHEADER,
    then slots of 90 symbols; with pilots, a block of 36 pilot symbols follows every 16th slot except the last slot"""
    slots = nsym // 90
    assert slots * 90 == nsym
    pos, raw = [], 90
    for j in range(slots):
        pos.append(np.arange(raw, raw + 90))
        raw += 90
        if pilots and (j + 1) % 16 == 0 and j + 1 < slots:
            raw += 36
    return np.concatenate(pos), raw


def assemble(payload, pos, total):
    """payload symbols [n][nsym][2] -> PLFRAMEs [n][total][2]; the header and the pilot positions are poisoned: NaN in
    even frames, a corner-cell value in odd ones"""
    out = np.empty((len(payload), total, 2), np.float32)
    out[0::2] = np.nan
    out[1::2] = (0.74, -0.74)
    out[:, pos] = payload
    return out


def lut_coords(v):
    """the LUT index of each coordinate: int((double)v / 1.5 * 256 + 128) as x86 truncates it (out of range and NaN give
    INT_MIN), clamped to 0..255 (constellation.cpp:295-310)"""
    d = v.astype(np.float64) / 1.5 * 256 + 128
    ok = (d > -2147483649.0) & (d < 2147483648.0)
    x = np.where(ok, np.trunc(np.where(ok, d, 0.0)), -2.0 ** 31)
    return np.clip(x, 0, 255).astype(np.uint8)


def cell_centres():
    """the centre of each of the 256 x 256 LUT cells, ((k - 128 + 0.5) / 256) * 1.5 on each axis (exact in float32)"""
    c = ((np.arange(256) - 127.5) / 256 * 1.5).astype(np.float32)
    x, y = np.meshgrid(c, c, indexing="ij")
    return np.stack([x.ravel(), y.ravel()], axis=1)


def odd_values():
    """per axis: the float just below, at and just above each of the 257 cell edges, and values where index arithmetic
    goes wrong (signed zeros, subnormals, far outside the grid, infinities, NaN of either sign)"""
    edge = ((np.arange(257) - 128) * 1.5 / 256).astype(np.float32)   # exact: multiples of 3 / 512
    v = [edge, np.nextafter(edge, np.float32(-np.inf)), np.nextafter(edge, np.float32(np.inf))]
    tiny = np.float32(np.finfo(np.float32).smallest_subnormal)
    small = [0.0, tiny, 2 * tiny, np.finfo(np.float32).tiny, np.nextafter(np.finfo(np.float32).tiny, np.float32(0))]
    big = [1.5, 30.0, 3e30, np.finfo(np.float32).max, np.inf]
    mag = np.array(small + big, np.float32)
    v += [mag, -mag, np.array([np.nan, -np.nan], np.float32)]
    v = np.concatenate(v).astype(np.float32)
    _, keep = np.unique(v.view(np.uint32), return_index=True)
    return v[np.sort(keep)]


def odd_symbols(rng, n):
    """n symbols: every odd value once as re and once as im next to another odd value, the rest random pairs of them"""
    v = odd_values()
    assert 2 * len(v) <= n
    a = np.stack([v, rng.choice(v, len(v))], axis=1)
    b = np.stack([rng.choice(v, len(v)), v], axis=1)
    rest = rng.choice(v, (n - 2 * len(v), 2))
    return rng.permutation(np.concatenate([a, b, rest]).astype(np.float32))


def fill_frames(syms, nsym, rng):
    """shuffle symbols into whole frames [n][nsym][2], padding the last frame with repeats"""
    nf = -(-len(syms) // nsym)
    pad = syms[rng.integers(0, len(syms), nf * nsym - len(syms))]
    return rng.permutation(np.concatenate([syms, pad])).reshape(nf, nsym, 2)


_CONSTELLATIONS = {}
_RN = {}


def oracle_constellation(modcod):
    _, ctype, _, g1, g2 = MODCODS[modcod]
    if (ctype, g1, g2) not in _CONSTELLATIONS:
        _CONSTELLATIONS[(ctype, g1, g2)] = orclib.oracle().orc_const_create(ctype, g1, g2)
    return _CONSTELLATIONS[(ctype, g1, g2)]


def oracle_llrs(modcod, short, payload):
    """orc_bb_to_soft (S2BBToSoft::process, pilots off) on each frame's payload symbols behind a 90-symbol header"""
    const, _, rate, _, _ = MODCODS[modcod]
    c = oracle_constellation(modcod)
    n, nsym, _ = payload.shape
    buf = np.zeros((90 + nsym, 2), np.float32)
    out = np.zeros((n, nsym * orclib.oracle().orc_const_bits(c)), np.int8)
    for i in range(n):
        buf[90:] = payload[i]
        orclib.oracle().orc_bb_to_soft(c, const, int(short), rate, buf.reshape(-1), out[i])
    return out


def oracle_chain(short, rate, llr):
    """orc_decode_frame (LDPC, BCH, BB descrambler) -> BBFRAME bytes, iterations, corrections, flags"""
    o = orclib.oracle()
    kb = orclib.code_params(int(short), rate)["kbch"] // 8
    bb = np.zeros((len(llr), kb), np.uint8)
    its = np.zeros(len(llr), np.int16)
    cor = np.zeros(len(llr), np.int16)
    for i in range(len(llr)):
        a, b = C.c_int(), C.c_int()
        o.orc_decode_frame(int(short), rate, llr[i].copy(), 25, bb[i], C.byref(a), C.byref(b))
        its[i], cor[i] = a.value, b.value
    crc_bad = np.array([o.orc_bbheader_crc8(np.ascontiguousarray(bb[i])) != 0 for i in range(len(llr))])
    flags = (its < 0) * pkg.FLAG_LDPC_FAIL + (cor < 0) * pkg.FLAG_BCH_FAIL + crc_bad * pkg.FLAG_BBHEADER_CRC_FAIL
    return bb, its, cor, flags.astype(np.uint32)


def assert_stage_equal(got, want, what):
    bb, res = got
    wbb, wits, wcor, wflags = want
    assert np.array_equal(res["ldpc_iters"], wits), (what, res["ldpc_iters"], wits)
    assert np.array_equal(res["bch_corr"], wcor), (what, res["bch_corr"], wcor)
    assert np.array_equal(res["flags"], wflags), (what, res["flags"], wflags)
    assert np.array_equal(res["tag"], np.arange(len(bb))), what
    assert np.array_equal(bb, wbb), what


def as_tuple(bb, res):
    return bb, res["ldpc_iters"], res["bch_corr"], res["flags"]


def pl_scramble(frames, codenum):
    """S2Scrambling::scramble (oracle restatement) over everything after the header, pilots included"""
    o = orclib.oracle()
    if codenum not in _RN:
        _RN[codenum] = np.zeros(131072, np.uint8)
        o.orc_pl_rn(codenum, _RN[codenum])
    out = frames.copy()
    nsym = frames.shape[1] - 90
    buf = np.zeros(2 * nsym, np.float32)
    for i in range(len(frames)):
        o.orc_pl_scramble(_RN[codenum], np.ascontiguousarray(frames[i, 90:]).reshape(-1), nsym, buf)
        out[i, 90:] = buf.reshape(-1, 2)
    return out


def noisy_payload(modcod, short, pilots, pos, sigmas, rng):
    """payload symbols of coded frames (random BBFRAMEs, in-tree encoder and modulator) plus Gaussian noise"""
    kb = pkg.modcod_info(modcod, short)["kbch"] // 8
    out = []
    for s in sigmas:
        bits = pkg.encode_fecframe(modcod, short, rng.integers(0, 256, kb, dtype=np.uint8))
        tx = pkg.modulate(modcod, short, pilots, bits).view(np.float32).reshape(-1, 2)
        out.append(tx[pos] + rng.normal(0, s, (len(pos), 2)).astype(np.float32))
    return np.stack(out)


def within_tolerance(got, want, payload, outer, what):
    """DESIGN §1, 32APSK: |dLLR| <= 1 LSB on at most 0.5 % of the LLRs.  Beyond 1.5x the outer ring, where the LLRs
    reach the halving clamp's steps at 127 * 2^k and exp(-dist) becomes subnormal, a last-bit difference between CUDA's
    and glibc's expf / logf may change a byte by more: on at most 1e-5 of the LLRs (measured on a B200: 2 of 84 million
    LLRs from 1x to 4x the outer ring, by 17; up to 60 in other samples)."""
    d = np.abs(got.astype(np.int16) - want.astype(np.int16))
    nsym = payload.shape[1]
    far = np.tile(np.hypot(payload[..., 0], payload[..., 1]) > 1.5 * outer, (1, got.shape[1] // nsym))   # LLR j: symbol j % nsym
    frac, big = np.count_nonzero(d) / d.size, d > 1
    assert frac <= 0.005, (what, "share of LLRs that differ", frac)
    assert not big[~far].any(), (what, "near the constellation, max |dLLR|", int(d[~far].max()))
    assert np.count_nonzero(big) <= 1e-5 * d.size, (what, "LLRs that differ by more than 1", np.count_nonzero(big), d.size)


# ------------------------------------------------------------------------------------------------ host-only checks
def test_configuration_matrix():
    cfgs = configurations()
    assert len(cfgs) == 104
    missing = {(m, s, p) for m in range(1, 29) for s in (False, True) for p in (False, True)} - set(cfgs)
    assert missing == {(m, True, p) for m in SHORT_9_10 for p in (False, True)}
    for modcod, short, pilots in cfgs:
        info = pkg.modcod_info(modcod, short, pilots)
        slots = info["nldpc"] // info["bits"] // 90
        assert info["plframe_symbols"] == 90 + 90 * slots + (36 * ((slots - 1) // 16) if pilots else 0)
        pos, total = payload_positions(info["nldpc"] // info["bits"], pilots)
        assert total == info["plframe_symbols"] and len(pos) == 90 * slots
        assert MODCODS[modcod][0] == info["bits"] - 2
    assert sorted(SEQUENCE[:-1]) == sorted(cfgs) and SEQUENCE[-1] == SEQUENCE[0]
    assert all(table_key(a) != table_key(b) for a, b in zip(SEQUENCE, SEQUENCE[1:]))
    # all eight LUTs (QPSK, 8PSK, six 16APSK gammas) and both frame sizes of each
    luts = {table_key(c)[:2] for c in cfgs if MODCODS[c[0]][0] != 3}
    assert len(luts) == 8


def test_symbols_of_the_lut_checks():
    """the cell centres hit every cell once; each edge value lands on the side of the edge it is meant to"""
    idx = lut_coords(cell_centres())
    assert len(np.unique(idx[:, 0].astype(np.int32) * 256 + idx[:, 1])) == 65536
    edge = ((np.arange(257) - 128) * 1.5 / 256).astype(np.float32)
    below, above = np.nextafter(edge, np.float32(-np.inf)), np.nextafter(edge, np.float32(np.inf))
    k = np.arange(1, 256)
    assert np.array_equal(lut_coords(above[1:256]), k)
    # below an edge is the cell before it, except below 0: 128 - 2**-149 / 1.5 * 256 rounds to 128 in double
    assert np.array_equal(lut_coords(below[1:256]), np.where(k == 128, 128, k - 1))
    at = lut_coords(edge)
    assert ((at == np.clip(np.arange(257), 0, 255)) | (at == np.arange(257) - 1)).all()
    v = odd_values()
    assert len(v) == 3 * 257 + 22 - 3 and np.isnan(v).sum() == 2
    # beyond int32 the x86 conversion gives INT_MIN, so huge positive values land in cell 0 like NaN
    assert lut_coords(np.array([np.nan, -np.inf, -3e30, np.inf, 3e30, 30, -0.0], np.float32)).tolist() == [0, 0, 0, 0, 0, 255, 128]


# ------------------------------------------------------------------------------------------------ on the device
@pytest.fixture(scope="module")
def dec():
    d = pkg.DVBS2Decoder(max_batch=64, max_trials=25)
    yield d
    d.close()
    for c in _CONSTELLATIONS.values():
        orclib.oracle().orc_const_destroy(c)
    _CONSTELLATIONS.clear()


def check_lut_configuration(dec, modcod, short, pilots, pos, total, codenum, rng):
    const, _, rate, _, _ = MODCODS[modcod]
    nsym = len(pos)
    payload = np.concatenate([fill_frames(cell_centres(), nsym, rng), odd_symbols(rng, nsym)[None]])
    x = assemble(payload, pos, total)
    want = oracle_llrs(modcod, short, payload)
    assert np.array_equal(dec.bb_to_soft(x), want)
    want_idx = lut_coords(payload)
    assert np.array_equal(dec.quantize_plframes(x), want_idx)

    noisy = assemble(noisy_payload(modcod, short, pilots, pos, SIGMAS[const], rng), pos, total)
    want_stage = oracle_chain(short, rate, oracle_llrs(modcod, short, noisy[:, pos]))
    got = dec.decode_plframes(noisy)
    assert_stage_equal(got, want_stage, "decode_plframes")
    assert_stage_equal(dec.decode_plframes_idx(dec.quantize_plframes(noisy)), as_tuple(*got), "decode_plframes_idx")

    dec.set_pl_scrambling(codenum)
    try:
        xs = pl_scramble(x, codenum)
        assert np.array_equal(dec.bb_to_soft(xs), want), codenum
        assert np.array_equal(dec.quantize_plframes(xs), want_idx), codenum
        ns = pl_scramble(noisy, codenum)
        assert_stage_equal(dec.decode_plframes(ns), as_tuple(*got), "decode_plframes, PL scrambled")
        assert_stage_equal(dec.decode_plframes_idx(dec.quantize_plframes(ns)), as_tuple(*got), "decode_plframes_idx, PL scrambled")
    finally:
        dec.set_pl_scrambling(-1)


def check_32apsk_configuration(dec, modcod, short, pilots, pos, total, codenum, rng):
    _, _, rate, _, _ = MODCODS[modcod]
    nsym = len(pos)
    noisy = noisy_payload(modcod, short, pilots, pos, SIGMAS_32APSK, rng)
    tx = noisy_payload(modcod, short, pilots, pos, (0.0,), rng)[0]
    outer = float(np.hypot(tx[:, 0], tx[:, 1]).max())
    g = np.linspace(-1.5, 1.5, 256, dtype=np.float32)
    grid = np.stack(np.meshgrid(g, g, indexing="ij"), axis=2).reshape(-1, 2)
    grid = fill_frames(np.concatenate([grid, odd_symbols(rng, nsym)]), nsym, rng)
    r = outer * np.repeat(np.linspace(1.5, 4.0, 1024), 256)
    phi = rng.uniform(0, 2 * np.pi, r.size)
    far = fill_frames(np.stack([r * np.cos(phi), r * np.sin(phi)], axis=1).astype(np.float32), nsym, rng)

    sets = {"noisy": noisy, "grid": grid, "far field": far}
    frames = {k: assemble(v, pos, total) for k, v in sets.items()}
    got = {k: dec.bb_to_soft(f) for k, f in frames.items()}
    for k in sets:
        within_tolerance(got[k], oracle_llrs(modcod, short, sets[k]), sets[k], outer, k)

    # the decoder behind the float demapper is exact: the oracle's chain on the device's own LLRs
    stage = dec.decode_plframes(frames["noisy"])
    assert_stage_equal(stage, oracle_chain(short, rate, got["noisy"]), "decode_plframes")
    with pytest.raises(pkg.DVBS2FecError):
        dec.quantize_plframes(frames["noisy"])

    dec.set_pl_scrambling(codenum)
    try:
        for k, f in frames.items():
            assert np.array_equal(dec.bb_to_soft(pl_scramble(f, codenum)), got[k]), (k, codenum)
        assert_stage_equal(dec.decode_plframes(pl_scramble(frames["noisy"], codenum)), as_tuple(*stage), "decode_plframes, PL scrambled")
    finally:
        dec.set_pl_scrambling(-1)


@pytest.mark.gpu
@pytest.mark.parametrize("step", range(len(SEQUENCE)), ids=step_id)
def test_demapper_against_oracle(dec, step):
    modcod, short, pilots = SEQUENCE[step]
    info = pkg.modcod_info(modcod, short, pilots)
    pos, total = payload_positions(info["nldpc"] // info["bits"], pilots)
    dec.setDemodParams(modcod, short, pilots)
    assert (dec.N, dec.plframe_symbols) == (info["nldpc"], total)
    codenum = CODENUMS[step] if step < len(CODENUMS) else (step * 40507 + 11) % 262142
    rng = np.random.default_rng(7000 + 64 * modcod + 2 * short + pilots)
    if MODCODS[modcod][0] == 3:
        check_32apsk_configuration(dec, modcod, short, pilots, pos, total, codenum, rng)
    else:
        check_lut_configuration(dec, modcod, short, pilots, pos, total, codenum, rng)


# ------------------------------------------------------------------------------------------------ > 65 535 frames
def tiled(base, n):
    """frame i of the batch is base[i % len(base)]"""
    return np.tile(base, (-(-n // len(base)),) + (1,) * (base.ndim - 1))[:n]


def assert_tiled(out, base):
    m = len(base)
    for f0 in range(0, len(out), 700 * m):
        part = out[f0: f0 + 700 * m]
        k = len(part) // m
        assert np.array_equal(part[: k * m].reshape((k,) + base.shape), np.broadcast_to(base, (k,) + base.shape)), f0
        assert np.array_equal(part[k * m:], base[: len(part) - k * m]), f0


@pytest.mark.gpu
def test_launches_of_more_than_65535_frames():
    """one launch of 65 600 frames through the entry points whose frames go in the grid's y dimension: frames past
    65 535 are demapped, descrambled and decoded like the same frames at low indices"""
    n = 65600
    rng = np.random.default_rng(65600)

    # bb_to_soft: short 32APSK 9/10 is the smallest PLFRAME (3 330 symbols)
    dec = pkg.DVBS2Decoder(max_batch=1024)
    try:
        dec.setDemodParams(24, True, False)
        assert dec.plframe_symbols == 3330
        pos, total = payload_positions(3240, False)
        base = assemble(noisy_payload(24, True, False, pos, (0.01, 0.03, 0.05, 0.07, 0.1, 0.3, 3.0), rng), pos, total)
        want = dec.bb_to_soft(base)
        x = tiled(base, n)
        got = dec.bb_to_soft(x)
        del x
        assert_tiled(got, want)
        del got

        # descramble: short-frame BBFRAMEs against numpy XOR with the PRBS
        dec.setDemodParams(4, True, False)
        prbs = np.zeros(dec.K // 8, np.uint8)
        orclib.oracle().orc_descramble(1, 3, prbs)
        fr = rng.integers(0, 256, (n, dec.K // 8), dtype=np.uint8)
        want = fr ^ prbs
        assert np.array_equal(dec.descramble(fr), want)
    finally:
        dec.close()

    # decode_plframes_idx on a handle whose batch is one launch of 65 600 frames: short 8PSK 2/3
    dec = pkg.DVBS2Decoder(max_batch=n)
    try:
        dec.setDemodParams(13, True, False)
        pos, total = payload_positions(5400, False)
        noisy = assemble(noisy_payload(13, True, False, pos, (0.05, 0.1, 0.14, 0.18, 0.2, 0.22, 0.5), rng), pos, total)
        idx = dec.quantize_plframes(noisy)
        wbb, wres = dec.decode_plframes_idx(idx)
        assert len(set(wres["ldpc_iters"].tolist())) >= 3
        bb, res = dec.decode_plframes_idx(tiled(idx, n))
        assert dec.last_launch_count() >= 2 and np.array_equal(res["tag"], np.arange(n))
        assert_tiled(bb, wbb)
        for k in ("ldpc_iters", "bch_corr", "flags"):
            assert_tiled(res[k], wres[k])
    finally:
        dec.close()
