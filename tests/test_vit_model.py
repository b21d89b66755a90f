"""The numpy model of K11's speculation (tests/vit_model.py) against the CPU oracle, and the seeded input families that
drive each of K11's fallbacks: a wrong start-state guess (a repeated task), a traceback whose 32 pieces disagree (a task
walked back step by step), and a cascade of repeats (a batch that needs three or more check passes).
tests/test_gpu_vit_speculation.py sends the same families to the GPU and asserts the counters the model predicts; this
file makes sure those predictions are not all zero."""
import numpy as np
import pytest

import dvbs_stream
import vit_model as M
from test_vit_oracle import OrcViterbi
from vit_model import FAMILIES, LOCK_SHIFT, model_family

B = M.K_BUF


@pytest.mark.parametrize("rate", range(5))
@pytest.mark.parametrize("phase", [0, 1])
def test_model_matches_oracle_on_locked_streams(rate, phase):
    """decoded bits (and so the chained end states) equal the oracle's, one batch of five locked blocks after the lock,
    with -128 and saturated runs inside the noisy code word"""
    rng = np.random.default_rng(rate * 2 + phase)
    bits = rng.integers(0, 2, 8000 * 6, dtype=np.uint8)
    s = dvbs_stream.inner_softs(bits, rate, rng, sigma=[12.0, 10.0, 9.0, 7.0, 5.0][rate], phase=phase, lead=2)[:5 * B].copy()
    s[2 * B + 100:2 * B + 400] = -128
    s[3 * B + 50:3 * B + 900:3] = 127
    s[4 * B:4 * B + 200] = -128
    s[5 * B - 300:] = 127
    o = OrcViterbi(0.15, 1000)
    want = o.process(s, fill=9)
    st = o.stats()
    assert st[1:5] == (1, rate, phase, LOCK_SHIFT[rate])
    L = M.LockedStream(rate, phase, st[4])
    b, outn, _ = L.run([s[k * B:(k + 1) * B] for k in range(5)])
    assert np.array_equal(M.assemble(b, outn, 9), want)
    # the end state the next block starts from is the last six decoded bits of the block (retval at n = fs - 6)
    assert L.start == int(sum(int(b[-1][M.FS_MAIN[rate] - 6 + j]) << (5 - j) for j in range(6)))


def test_model_clean_stream_needs_no_fallback():
    """on a noisy but clean code word every guess is right and every 32-piece traceback is accepted: the fallbacks the
    families below provoke are not the model's default"""
    rng = np.random.default_rng(3)
    clean = dvbs_stream.inner_softs(rng.integers(0, 2, 4096 * 4, dtype=np.uint8), 0, rng, sigma=8.0)[:3 * B]
    L = M.LockedStream(0, 0, 0)
    _, _, c = L.run([clean[k * B:(k + 1) * B] for k in range(3)])
    assert (c["tasks"], c["repeats"], c["passes"], c["walks"]) == (3, 0, 1, 0)


def test_families_drive_every_speculative_path():
    """each family at every rate and both phases: model bits equal the oracle's, and together the families repeat tasks
    (zeros: at every rate and phase), walk tasks, and build a cascade of >= 3 check passes (sat at 2/3 and 7/8, phase
    90: both saturated blocks end where their guesses did not; the -128 block, decoded again from its corrected start,
    ends in yet another state, so the clean block behind it is repeated twice).  Runs of soft 0 and midpoints of two
    code words make the warm-up from state 0 miss the path (walks); soft 0 at the end of a block makes the guess from
    flat metrics miss the end state at every rate.  Midpoint tails of 1200 soft bits leave the guess right: the tie
    rule picks the code word the decoder was already on."""
    tot = dict(repeats=0, walks=0, cascades=0)
    for kind in FAMILIES:
        for rate in range(5):
            for phase in (0, 1):
                s, st, want, got, c = model_family(kind, rate, phase)
                assert st[1:5] == (1, rate, phase, LOCK_SHIFT[rate]), (kind, rate, phase, st)
                assert np.array_equal(got, want), (kind, rate, phase)
                if kind == "zeros":
                    assert c["repeats"] >= 1, (rate, phase, c)
                if kind == "sat" and phase == 1 and rate in (1, 4):
                    assert c["passes"] >= 3, (rate, c)
                tot["repeats"] += c["repeats"]
                tot["walks"] += c["walks"]
                tot["cascades"] += c["passes"] >= 3
    assert tot["repeats"] >= 10 and tot["walks"] >= 40 and tot["cascades"] >= 2, tot
