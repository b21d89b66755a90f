"""TEST INFRASTRUCTURE -- a numpy model of how K11 (csrc/dvbs_viterbi.cu) computes a locked batch, so that tests can
predict its speculation counters (tasks, repeats, check passes, walks) and build inputs that drive each fallback.

It restates, on top of the oracle's ccdec_work (oracle/oracle_vit.c:58-93), vectorised over the tasks of a batch:
  acs()            the reference's butterfly: uint8 metrics that wrap, the tie rule m0 >= m1, renormalisation, the
                   decision bits of every step
  guess()          acs_kernel mode 0: the last kGuessSteps steps from zero metrics, find_endstate, 6 traceback steps
  decode()         acs_kernel modes 1 / 2 from a given start state (-1: unbiased 31s, else 63 with 0 at the start):
                   the sequential traceback (bits, retval) and whether the 32-piece traceback is accepted or the task
                   is walked back step by step
  run_batch()      run_tasks: mode 1 from the predecessor's guess, then mark_kernel / mode 2 until nothing is flagged
  LockedStream     Viterbi_DVBS::work at the lock (viterbi_all.cpp:196-250) for all five rates: rotate_to_unsigned,
                   depuncture_34 / depuncture_78, Depunc23 / Depunc56::depunc_cont with the byte it holds back, and
                   the soft / depunc buffers that persist from block to block -- the decoder image of every block
  family()         seeded inputs that drive each fallback: a wrong guess, a walked traceback, a cascade of repeats
The lock search (search_image_kernel's replay of stale buffers) is not modelled."""
import numpy as np

import dvbs_stream
from test_vit_oracle import OrcViterbi

K_BUF = 8192
K_GUESS = 326        # kGuessSteps
K_WARM = 128         # kWarm
FS_MAIN = [K_BUF // 2, 10924 // 2, int(K_BUF * 1.5 / 2), int(K_BUF * 1.66 / 2), int(K_BUF * 1.75 / 2)]
PERIOD = {1: 3, 3: 6}       # Depunc23, Depunc56


def _parity(v):
    return np.array([bin(int(x)).count("1") & 1 for x in v], np.uint8)


_I = np.arange(32)
G0 = (_parity((2 * _I) & 79) * 255).astype(np.uint8)      # Branchtab (cc_decoder.cpp:127-134)
G1 = (_parity((2 * _I) & 109) * 255).astype(np.uint8)


def acs(img, nsteps, start, first=0):
    """img [T, >= 2 nsteps] uint8 decoder input; start [T]: -1 unbiased 31s, -2 zeros (guess), else the biased start
    state.  -> (decisions [nsteps, T, 64] bool, end state [T]) after steps first..nsteps-1"""
    img = np.asarray(img, np.uint8)
    T = img.shape[0]
    start = np.asarray(start)
    x = np.full((T, 64), 63, np.uint8)
    x[start == -1] = 31
    x[start == -2] = 0
    hot = start >= 0
    x[np.nonzero(hot)[0], start[hot]] = 0
    a = img[:, 2 * first:2 * nsteps:2].T[:, :, None]
    b = img[:, 2 * first + 1:2 * nsteps:2].T[:, :, None]
    met = ((1 + (G0 ^ a).astype(np.int32) + (G1 ^ b)) >> 3).astype(np.uint8)      # [steps, T, 32]
    inv = (63 - met).astype(np.uint8)
    dec = np.zeros((nsteps, T, 64), bool)
    y = np.empty((T, 64), np.uint8)
    for s in range(first, nsteps):
        m, q = met[s - first], inv[s - first]
        lo, hi = x[:, :32], x[:, 32:]
        m0, m1, m2, m3 = lo + m, hi + q, lo + q, hi + m      # uint8: wraps like the reference's unsigned char
        d0, d1 = m0 >= m1, m2 >= m3
        y[:, 0::2] = np.where(d0, m1, m0)
        y[:, 1::2] = np.where(d1, m3, m2)
        y -= y.min(1, keepdims=True)
        dec[s, :, 0::2] = d0
        dec[s, :, 1::2] = d1
        x, y = y, x
    return dec, x.argmin(1)      # find_endstate: the first smallest metric


def _back(dec, n, st):
    k = dec[n + 6, np.arange(len(st)), st].astype(np.int64)
    return (st >> 1) | (k << 5), k


def guess(img, fs):
    """acs_kernel mode 0 -> the guessed end state (retval) of every task"""
    nsteps = fs + 6
    dec, st = acs(img, nsteps, np.full(len(img), -2), max(0, nsteps - K_GUESS))
    for n in range(fs - 1, fs - 7, -1):
        st, _ = _back(dec, n, st)
    return st


def pieces_ok(dec, end, fs):
    """acs_kernel's acceptance rule (dvbs_viterbi.cu:315-345): does the 32-piece traceback stand?  -> bool [T]"""
    T = len(end)
    PL = ((fs + 31) // 32 + 15) & ~15
    top = (fs - 1) // PL
    lanes = np.arange(top + 1)
    seg_lo = lanes * PL
    seg_hi = np.minimum(seg_lo + PL, fs)
    nw = np.minimum(seg_hi - 1 + K_WARM, fs - 1)
    nw[top] = fs - 1
    st = np.where((nw == fs - 1)[None, :], end[:, None], 0).astype(np.int64)      # [T, lanes]
    warm = np.full((T, top + 1), -1, np.int64)
    rows = np.arange(T)[:, None]
    for j in range(int((nw - seg_lo).max()) + 1):
        m = nw - j
        live = m >= seg_lo
        if not live.any():
            break
        mm = np.where(live, m, 0)
        at = (m == seg_hi - 1) & (lanes < top)
        warm[:, at] = st[:, at]
        k = dec[(mm + 6)[None, :], rows, st].astype(np.int64)
        st = np.where(live[None, :], (st >> 1) | (k << 5), st)
    return np.all(warm[:, :top] == st[:, 1:top + 1], axis=1)


def decode(img, fs, start):
    """acs_kernel modes 1 / 2 -> (bits [T, fs] uint8, retval [T], walked [T] bool)"""
    dec, end = acs(img, fs + 6, start)
    st = end.astype(np.int64)
    bits = np.zeros((len(st), fs), np.uint8)
    ret = None
    for n in range(fs - 1, -1, -1):
        st, k = _back(dec, n, st)
        bits[:, n] = k
        if n == fs - 6:
            ret = st.copy()
    return bits, ret, ~pieces_ok(dec, end.astype(np.int64), fs)


def run_batch(imgs, fs, start):
    """run_tasks over tasks chained k - 1 -> k, task 0 starting from `start`.
    -> (bits [n, fs], retval [n], dict(tasks, repeats, passes, walks, walked=[task indices walked, once per decode]))"""
    imgs = np.asarray(imgs, np.uint8)
    n = len(imgs)
    g = guess(imgs, fs)
    used = np.concatenate([[start], g[:-1]]).astype(np.int64)
    bits, ret, walked = decode(imgs, fs, used)
    c = dict(tasks=n, repeats=0, passes=0, walks=int(walked.sum()), walked=list(np.nonzero(walked)[0]), rounds=[])
    while True:
        c["passes"] += 1
        flag = np.nonzero(used[1:] != ret[:-1])[0] + 1
        if not len(flag):
            break
        c["repeats"] += len(flag)
        c["rounds"].append(list(flag))
        used[flag] = ret[flag - 1]
        b2, r2, w2 = decode(imgs[flag], fs, used[flag])
        bits[flag], ret[flag] = b2, r2
        c["walks"] += int(w2.sum())
        c["walked"] += list(flag[w2])
    return bits, ret, c


# ---- the decoder input at the lock (viterbi_all.cpp:196-250) ----------------------------------------------------------
def rotate_to_unsigned(x, phase):
    """rotate_soft (phases 0 and 90) + signed_soft_to_unsigned of one block"""
    x = np.asarray(x, np.int16)
    x = np.where(x == -128, -127, x)
    a, b = x[0::2], x[1::2]
    if phase == 1:
        a, b = b, -a
    out = np.empty(len(x), np.int16)
    out[0::2], out[1::2] = a + 127, b + 127
    out = out.astype(np.uint8)
    out[out == 128] = 127
    return out


def _spread(vals, counts, vpos):
    """every input value emitted with counts[i] slots, the value at offset vpos[i] of its slots, 128 elsewhere"""
    off = np.cumsum(counts) - counts
    out = np.full(int(counts.sum()), 128, np.uint8)
    out[off + vpos] = vals
    return out


def depuncture_34(soft, shift):
    i = np.arange(len(soft) // 2)
    plain = (shift != 0) ^ (i % 2 == 0)
    return _pairs(soft.reshape(-1, 2), np.where(plain, 2, 4), np.where(plain, 0, 1), np.where(plain, 1, 2))


def _pairs(pairs, cnt, pa, pb):
    """pair i emitted as cnt[i] slots with its a at pa[i], its b at pb[i], 128 elsewhere"""
    off = np.cumsum(cnt) - cnt
    out = np.full(int(cnt.sum()), 128, np.uint8)
    out[off + pa] = pairs[:, 0]
    out[off + pb] = pairs[:, 1]
    return out


def depuncture_78(soft, shift):
    i = np.arange(len(soft) // 2)
    ph = (i + shift) % 4
    cnt = np.where(ph == 0, 2, 4)
    pa = np.where(ph == 0, 0, 1)
    pb = np.where(ph == 0, 1, np.where(ph == 1, 3, 2))
    return _pairs(soft.reshape(-1, 2), cnt, pa, pb)


def depunc_emit(period, ph, vals):
    """Depunc23 / Depunc56 depunc_emit for inputs at phases ph"""
    if period == 3:
        cnt, vpos = np.where(ph == 1, 2, 1), np.zeros(len(ph), np.int64)
    else:
        cnt = np.where((ph == 0) | (ph == 2), 1, 2)
        vpos = (ph == 4).astype(np.int64)
    return _spread(vals, cnt, vpos)


class LockedStream:
    """Viterbi_DVBS at the lock, block by block: the decoder image of every block and the decoder's start state.
    `dp` = Depunc23 / Depunc56 state that survives from before the lock (got_extra, buf); `start` = the main decoder's
    carried start state (-1 on its first use)"""

    def __init__(self, rate, phase, shift, start=-1, got_extra=0, buf=128):
        self.rate, self.phase, self.shift, self.start = rate, phase, shift, start
        self.fs = FS_MAIN[rate]
        self.nread = 2 * (self.fs + 6)
        self.soft = np.full(4 * K_BUF, 128, np.uint8)       # memset at the lock
        self.dbuf = np.full(4 * K_BUF, 128, np.uint8)
        if rate in PERIOD:
            self.period = PERIOD[rate]
            self.cs, self.is_first = shift, int(shift > self.period - 1)      # depunc_set_shift
        self.got_extra, self.buf = got_extra, buf

    def image(self, block):
        """-> (decoder image of the block [nread], out_n = the output bits the call reports)"""
        self.soft[:K_BUF] = rotate_to_unsigned(block, self.phase)
        r = self.rate
        if r == 0:
            return self.soft[self.shift:self.shift + self.nread].copy(), K_BUF // 2
        if r == 2:
            o = depuncture_34(self.soft[:K_BUF], self.shift)
        elif r == 4:
            o = depuncture_78(self.soft[:K_BUF], self.shift)
        else:      # depunc_cont
            lead = []
            if self.is_first or self.got_extra:
                lead = [self.buf]
                self.is_first = self.got_extra = 0
            self.cs %= self.period
            ph = (self.cs + np.arange(K_BUF)) % self.period
            self.cs += K_BUF
            o = np.concatenate([np.array(lead, np.uint8), depunc_emit(self.period, ph, self.soft[:K_BUF])])
            if len(o) % 2 == 1:
                self.buf = int(o[-1])
                self.got_extra = 1
                self.dbuf[:len(o)] = o
                return self.dbuf[:self.nread].copy(), (len(o) - 1) // 2
        self.dbuf[:len(o)] = o
        return self.dbuf[:self.nread].copy(), len(o) // 2

    def run(self, blocks):
        """one batch of locked blocks (a sync batch of run_sync) -> (per-block bits, per-block out_n, counters)"""
        imgs, outn = zip(*[self.image(b) for b in blocks])
        bits, ret, c = run_batch(np.stack(imgs), self.fs, self.start)
        self.start = int(ret[-1])
        return bits, list(outn), c


def assemble(bits, outn, fill=0):
    """the output stream of a call, as orc_vit_process writes it: every block writes its frame size, the next starts
    out_n further on; what no block writes keeps `fill`"""
    total = int(sum(outn))
    out = np.full(total + K_BUF, fill, np.uint8)
    o = 0
    for b, n in zip(bits, outn):
        out[o:o + len(b)] = b
        o += n
    return out[:total]


# ---- seeded inputs that drive each fallback (tests/test_vit_model.py shows that they do) ----------------------------------
FAMILIES = ["zeros", "tail", "ambig", "sat"]


def _two_codewords(rate, phase, seed, nblk):
    """two unrelated code words (different encoder states everywhere) of one rate, puncturing phase and rotation"""
    rng = np.random.default_rng(seed)
    n = 8000 * (nblk + 1)
    a, b = rng.integers(0, 2, n, dtype=np.uint8), rng.integers(0, 2, n, dtype=np.uint8)
    sa = dvbs_stream.inner_softs(a, rate, np.random.default_rng(seed + 1), phase=phase, lead=2)[:nblk * K_BUF]
    sb = dvbs_stream.inner_softs(b, rate, np.random.default_rng(seed + 1), phase=phase, lead=2)[:nblk * K_BUF]
    return sa, sb


def family(kind, rate, phase, seed=0):
    """six blocks: block 0 a clean code word that locks the decoder at (rate, phase, shift 4 / 4 / 1 / 4 / 3), then:
      zeros  soft 0 (every branch metric 31 or 32) in blocks 2 (700 soft bits in the middle) and 3 (its last 800)
      tail   the last 1200 soft bits of blocks 2 and 4 the midpoint of two code words with different encoder states
      ambig  blocks 2..4 the midpoint of the two code words throughout
      sat    block 2 all +127, block 3 all -128 (saturated: the 8-bit metrics wrap, -128 becomes -127)"""
    sa, sb = _two_codewords(rate, phase, 10 * rate + phase + 1000 * seed, 6)
    mid = ((sa.astype(np.int16) + sb) // 2).astype(np.int8)
    s = sa.copy()
    if kind == "zeros":
        s[2 * K_BUF + 3000:2 * K_BUF + 3700] = 0
        s[4 * K_BUF - 800:4 * K_BUF] = 0
    elif kind == "tail":
        for k in (2, 4):
            s[(k + 1) * K_BUF - 1200:(k + 1) * K_BUF] = mid[(k + 1) * K_BUF - 1200:(k + 1) * K_BUF]
    elif kind == "ambig":
        s[2 * K_BUF:5 * K_BUF] = mid[2 * K_BUF:5 * K_BUF]
    elif kind == "sat":
        s[2 * K_BUF:3 * K_BUF] = 127
        s[3 * K_BUF:4 * K_BUF] = -128
    return s


LOCK_SHIFT = [0, 4, 1, 4, 3]


def model_family(kind, rate, phase):
    """-> (stream, lock stats after block 0, oracle output of blocks 1..5 with fill 3, model output, model counters of
    blocks 1..5 as one locked batch)"""
    s = family(kind, rate, phase)
    o = OrcViterbi(0.15, 1000)
    o.process(s[:K_BUF])
    st = o.stats()
    want = o.process(s[K_BUF:], fill=3)
    L = LockedStream(st[2], st[3], st[4])
    L.run([s[:K_BUF]])
    bits, outn, c = L.run([s[k * K_BUF:(k + 1) * K_BUF] for k in range(1, 6)])
    return s, st, want, assemble(bits, outn, 3), c
