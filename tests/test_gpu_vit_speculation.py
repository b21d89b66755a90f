"""K11 (csrc/dvbs_viterbi.cu) where its speculation fails and across every lock transition, bit for bit against the
oracle (decoded bits, and the lock state after every call).  The speculation counters of
dvbs2fec_dvbs_viterbi_counters are checked against tests/vit_model.py, so that a repeat pass, a cascade of repeats or a
walked traceback that goes wrong -- or never runs -- fails here."""
import numpy as np
import pytest

import dvbs_stream
import vit_model as M
from fec import pkg
from vit_model import FAMILIES, model_family
from test_vit_oracle import OrcViterbi, same_stats

pytestmark = pytest.mark.gpu

B = M.K_BUF
SIGMA = [12.0, 10.0, 9.0, 7.0, 5.0]
# soft bits of noise in front of a signal, and the shift the search then locks at: 2/3 and 5/6 lock with
# shift > period - 1, so depunc_cont starts with the byte it held back (dp.buf), which survives a lost lock
LEAD = {0: (0, 0), 1: (1, 5), 2: (2, 1), 3: (5, 7), 4: (2, 3)}
TOTAL = dict(tasks=0, repeats=0, passes=0, walks=0)


@pytest.fixture(autouse=True, scope="module")
def _report_totals():
    """the counter deltas this file asserted, summed (shown with -s)"""
    yield
    print("\nK11 counter deltas asserted:", TOTAL)


def _delta(g, c0):
    c = g.counters()
    d = tuple(a - b for a, b in zip(c, c0))
    for k, v in zip(("tasks", "repeats", "passes", "walks"), d):
        TOTAL[k] += v
    return d


def sig(rate, n, rng, lead=None):
    bits = rng.integers(0, 2, 8192 * n, dtype=np.uint8)
    return dvbs_stream.inner_softs(bits, rate, rng, sigma=SIGMA[rate], lead=LEAD[rate][0] if lead is None else lead)[:n * B]


def noise(n, rng):
    return np.clip(np.rint(rng.normal(0, 40, n * B)), -128, 127).astype(np.int8)


def oracle_blocks(o, s, fill):
    """the oracle block by block -> (output of the whole stream, stats after every block)"""
    out, stats = [], []
    for k in range(len(s) // B):
        out.append(o.process(s[k * B:(k + 1) * B], fill=fill))
        stats.append(o.stats())
    return np.concatenate(out), stats


# ---- 1. forced paths, exact counters ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", FAMILIES)
def test_forced_speculation_paths_match_oracle_and_model(kind):
    """lock on a clean block, then five adversarial blocks in one call at every rate and both phases (max_outsync 1000
    keeps them at the lock): bits and stats equal the oracle, the counter deltas of the second call equal the model's
    run_tasks -- tasks, repeats, check passes, walks"""
    seen = dict(repeats=0, walks=0, cascade=0)
    for rate in range(5):
        for phase in (0, 1):
            s, st, want, model_out, c = model_family(kind, rate, phase)
            g = pkg.DVBSViterbi(0.15, 1000)
            g.process(s[:B])
            assert same_stats(g.stats(), st), (rate, phase)
            c0 = g.counters()
            got = g.process(s[B:], out=np.full(5 * B, 3, np.uint8))
            assert np.array_equal(got, want), (kind, rate, phase)
            assert np.array_equal(got, model_out)
            o = OrcViterbi(0.15, 1000)
            o.process(s)
            assert same_stats(g.stats(), o.stats()) and g.stats()[1] == 1
            assert _delta(g, c0) == (5, c["repeats"], c["passes"], c["walks"]), (kind, rate, phase, c)
            seen["repeats"] += c["repeats"]
            seen["walks"] += c["walks"]
            seen["cascade"] += c["passes"] >= 3
            g.close()
    if kind == "zeros":
        assert seen["repeats"] >= 10 and seen["walks"] > 0
    if kind == "sat":
        assert seen["cascade"] >= 2
    if kind in ("tail", "ambig"):
        assert seen["walks"] >= 10


# ---- 2. lock transitions -----------------------------------------------------------------------------------------------------
def held_byte_episode(rate, rng):
    """signal at 2/3 or 5/6 for 3, 4 or 5 blocks, then the 3 noise blocks that lose the lock (max_outsync 2), with the
    length chosen so that the byte Depunc23/56 holds back when the lock is lost is a soft bit, not an erasure (128, what
    a reset depuncturer holds) -> (blocks, that byte)"""
    s, nz = sig(rate, 5, rng), noise(3, rng)
    for n in (3, 4, 5):
        L = M.LockedStream(rate, 0, LEAD[rate][1])
        ep = np.concatenate([s[:n * B], nz])
        for k in range(n + 3):
            L.image(ep[k * B:(k + 1) * B])
        if L.buf != 128:
            return ep, L.buf
    raise AssertionError("no episode length leaves a soft bit held back")


def transition_stream(r1, r2, rng):
    """signal r1, noise until the lock is lost, signal r2.  When r2 is 2/3 or 5/6 its depuncturer must carry a soft bit
    into the re-lock: an r2 episode that leaves one comes first (when r1 is r2, that episode is r1's).
    -> (stream, [(block, rate) of every lock], the byte the r2 re-lock reads first, or None)"""
    parts, locks, held, k = [], [], None, 0
    episodes = [r2, r1] if r2 in M.PERIOD and r1 != r2 else [r1]
    for r in episodes:
        if r in M.PERIOD and r == r2:
            ep, held = held_byte_episode(r, rng)
        else:
            ep = np.concatenate([sig(r, 3, rng), noise(3, rng)])
        parts.append(ep)
        locks.append((k, r))
        k += len(ep) // B
    parts.append(sig(r2, 3, rng))
    locks.append((k, r2))
    return np.concatenate(parts), locks, held


@pytest.mark.parametrize("r1", range(5))
def test_lock_transitions_match_oracle(r1):
    """signal at r1, noise until the lock is given up (max_outsync 2), signal at r2, for every r2: in one call and
    block by block.  2/3 and 5/6 re-lock with shift > period - 1, so depunc_cont starts with the byte Depunc23/56 held
    back when the lock was lost; the streams make that byte a soft bit, so a depuncturer that forgot it (128) reads a
    different first byte and counts one more BER position.  7/8 -> 5/6 reads the re-encoded bit 3398 the 7/8 lock left."""
    for r2 in range(5):
        rng = np.random.default_rng(600 + 5 * r1 + r2)
        s, locks, held = transition_stream(r1, r2, rng)
        want, stats = oracle_blocks(OrcViterbi(0.15, 2), s, 7)
        for blk, r in locks:
            assert stats[blk][1:5] == (1, r, 0, LEAD[r][1]) and (blk == 0 or stats[blk - 1][1] == 0), (r1, r2, blk)
        if r2 in M.PERIOD:
            assert held is not None and held != 128 and LEAD[r2][1] > M.PERIOD[r2] - 1
        g = pkg.DVBSViterbi(0.15, 2)
        assert np.array_equal(g.process(s, out=np.full(len(s), 7, np.uint8)), want), (r1, r2)
        assert same_stats(g.stats(), stats[-1])
        g.reset()
        o = 0
        for k in range(len(s) // B):
            got = g.process(s[k * B:(k + 1) * B], out=np.full(B, 7, np.uint8))
            assert np.array_equal(got, want[o:o + len(got)]), (r1, r2, k)
            o += len(got)
            assert same_stats(g.stats(), stats[k]), (r1, r2, k)
        assert o == len(want)
        g.close()


# ---- 3. batch cuts -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rate", range(5))
def test_batch_cuts_match_oracle(rate, monkeypatch):
    """decode batches of 1, 2, 3 and 7 blocks: the depuncturers' carried state (the held byte, rate 2/3's stale bytes
    10922/10923 and its stale step every third call) crosses every batch joint; the lock is given up inside a batch"""
    rng = np.random.default_rng(700 + rate)
    s = np.concatenate([sig(rate, 8, rng), noise(3, rng), sig(rate, 6, rng)])
    want, stats = oracle_blocks(OrcViterbi(0.15, 2), s, 5)
    assert stats[10][1] == 0 and stats[11][1] == 1
    for mb in (1, 2, 3, 7):
        monkeypatch.setenv("DVBS2FEC_VIT_MAX_BATCH", str(mb))
        g = pkg.DVBSViterbi(0.15, 2)
        c0 = g.counters()
        assert np.array_equal(g.process(s, out=np.full(len(s), 5, np.uint8)), want), mb
        assert same_stats(g.stats(), stats[-1]), mb
        assert _delta(g, c0)[0] == plan_tasks([(0, 0)] + stats[:-1], stats, [len(s) // B], mb)[0], mb
        g.close()


# ---- 4. search batches ---------------------------------------------------------------------------------------------------------
def plan_tasks(stats_before, stats_after, calls, max_sync=8192):
    """the tasks run_tasks runs, from the oracle's per-block lock state: 52 per searched block of each search batch
    (1, 4, 16, 64 blocks; the blocks behind the locking one are searched and thrown away), then each sync batch"""
    sb, base, out = 1, 0, []
    for nb in calls:
        pos, t = 0, 0
        while pos < nb:
            if stats_before[base + pos][1] == 0:
                n = min(nb - pos, sb, 64)
                t += 52 * n
                lock = next((b for b in range(pos, pos + n) if stats_after[base + b][1] == 1), None)
                if lock is None:
                    pos += n
                    sb = min(sb * 4, 64)
                    continue
                pos, sb = lock, 1
            n = min(nb - pos, max_sync)
            t += n
            lost = next((b for b in range(pos, pos + n) if stats_after[base + b][1] == 0), None)
            pos = pos + n if lost is None else lost + 1
        out.append(t)
        base += nb
    return out


@pytest.mark.parametrize("at", [1, 2, 4, 5, 12, 20, 21, 50, 84])
def test_search_batches_match_oracle(at):
    """noise, then a signal that locks as the first, a middle or the last block of the 4-, 16- or 64-block search batch
    (the blocks behind the locking one are searched, thrown away and decoded at the lock); the first call ends two
    blocks behind that batch, so the second call carries the lock over.  Tasks equal the plan."""
    rng = np.random.default_rng(800 + at)
    rate = at % 5
    end = 4 if at <= 4 else 20 if at <= 20 else 84      # last block of the search batch that holds `at`
    s = np.concatenate([noise(at, rng), sig(rate, end - at + 4, rng)])
    want, stats = oracle_blocks(OrcViterbi(), s, 0)
    assert all(st[1] == 0 for st in stats[:at]) and stats[at][1:3] == (1, rate)
    calls = [end + 2, len(s) // B - end - 2]
    plan = plan_tasks([(0, 0)] + stats[:-1], stats, calls)
    g = pkg.DVBSViterbi()
    got, lo = [], 0
    for nb, p in zip(calls, plan):
        c0 = g.counters()
        got.append(g.process(s[lo * B:(lo + nb) * B]))
        assert _delta(g, c0)[0] == p, (at, nb)
        assert same_stats(g.stats(), stats[lo + nb - 1])
        lo += nb
    assert np.array_equal(np.concatenate(got), want)
    g.close()


def test_two_candidates_under_the_threshold():
    """threshold 0.3: a clean rate 1/2 block passes its own candidate and the last one, rate 7/8 phase 90 shift 3, which
    keeps the lock.  Two noise blocks first, so the clean block is the middle block of the 4-block search batch."""
    rng = np.random.default_rng(900)
    clean = dvbs_stream.inner_softs(rng.integers(0, 2, 8000 * 4, dtype=np.uint8), 0, rng)[:3 * B]
    s = np.concatenate([noise(2, rng), clean])
    # the same stream at threshold 0.15 locks at rate 1/2 on that block: the candidates of a block do not depend on the
    # threshold while no earlier block has locked, so the rate 1/2 candidate is under 0.15 < 0.3 in the stream below too
    _, low = oracle_blocks(OrcViterbi(0.15, 20), s, 0)
    assert low[0][1] == low[1][1] == 0 and low[2][1:5] == (1, 0, 0, 0)
    want, stats = oracle_blocks(OrcViterbi(0.3, 20), s, 0)
    assert stats[0][1] == stats[1][1] == 0 and stats[2][1:5] == (1, 4, 1, 3)
    g = pkg.DVBSViterbi(0.3, 20)
    c0 = g.counters()
    assert np.array_equal(g.process(s), want) and same_stats(g.stats(), stats[-1])
    plan = plan_tasks([(0, 0)] + stats[:-1], stats, [5])[0]
    assert plan == 52 * (1 + 4) + 3 and _delta(g, c0)[0] == plan
    g.close()


# ---- 5. process_device ---------------------------------------------------------------------------------------------------------
def test_process_device_matches_oracle():
    """torch int8 / uint8 CUDA buffers: rate 5/6 leaves 27 bits per block unwritten, which keep the sentinel exactly as the
    oracle's buffer keeps its fill; nothing is written behind the returned count"""
    import torch
    rng = np.random.default_rng(1000)
    s = np.concatenate([noise(2, rng), sig(3, 6, rng)])
    want, stats = oracle_blocks(OrcViterbi(), s, 0xA5)
    g = pkg.DVBSViterbi()
    d_in = torch.from_numpy(s).cuda()
    d_out = torch.full((len(s),), 0xA5, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()      # the handle runs on its own stream: the copy and the fill are done before it starts
    n = g.process_device(d_in.data_ptr(), len(s), d_out.data_ptr())
    torch.cuda.synchronize()
    out = d_out.cpu().numpy()
    assert n == len(want) and np.array_equal(out[:n], want)
    assert np.all(out[n:] == 0xA5)
    assert np.sum(want == 0xA5) >= 27 * 5
    assert same_stats(g.stats(), stats[-1])
    g.close()
