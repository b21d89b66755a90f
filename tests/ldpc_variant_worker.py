"""Helpers of tests/test_gpu_ldpc_variants.py, and the subprocess that decodes under one set of LDPC overrides.

The kernel-choice overrides (DVBS2FEC_LDPC_LANES2, _OCC3, _V2, _CHAINS, DVBS2FEC_CHAIN_MINLEV) are read once per
process, so every environment of the variant matrix runs in a process of its own:

    python tests/ldpc_variant_worker.py ORACLE.npz REPORT.json

decodes, for every code in ORACLE.npz, a large batch tiled from the code's M oracle frames through four entry
points, compares every position in-process and writes a small JSON report (mismatch counts, the first mismatch,
the LDPC kernels launched).  Not collected by pytest (no test_ prefix)."""
import json
import os
import re
import sys
import tempfile
import time

import numpy as np

import orclib
from orclib import code_params

# ---- tiled batches -------------------------------------------------------------------------------------------------
# Position p of a batch holds frame (STEP * p + SHIFT) mod M of the code's M oracle frames.  M is an odd prime and
# gcd(STEP, M) = 1, so two positions hold the same frame only if they are a multiple of M apart: the pair partner,
# the next pair, a streamed piece (256 frames), a 255-frame chunk and a whole grid's worth of pairs all hold other
# frames, and every frame lands in lane A (even position) and lane B (odd position) of a pair.
M = 31
STEP = 7
SHIFT = 5
# offsets at which a kernel or the host plan could confuse one frame with another: pair partner, next pair, half a
# streamed piece, a 255-frame chunk, a streamed piece, and one grid / one grid's worth of pairs at 2 and 3 CTAs per SM
# on a 148-SM B200
CONFUSABLE_OFFSETS = (1, 2, 3, 128, 255, 256, 296, 444, 510, 592, 888)


def tile(n, m=M, step=STEP, shift=SHIFT):
    """frame index of every position of an n-frame batch"""
    return (step * np.arange(n, dtype=np.int64) + shift) % m


def batch_size(sms):
    """odd, and at least 8 frames per CTA of the largest grid (3 CTAs per SM): every CTA decodes four pairs or more"""
    n = 8 * sms * 3
    return n + 1 if n % 2 == 0 else n


# ---- kernel choice model -------------------------------------------------------------------------------------------
# (max data links per check, every layer has that many) per code; the code tables are built in s2_codes.cpp and
# test_ldpc_variant_model.py checks these against the oracle's schedule
CODE_LINKS = {
    (0, 0): (2, True), (0, 1): (3, True), (0, 2): (4, True), (0, 3): (5, True), (0, 4): (9, True), (0, 5): (8, True),
    (0, 6): (12, True), (0, 7): (16, True), (0, 8): (20, True), (0, 10): (25, True), (0, 11): (28, True),
    (1, 0): (2, False), (1, 1): (3, True), (1, 2): (4, True), (1, 3): (5, False), (1, 4): (9, True), (1, 5): (8, True),
    (1, 6): (11, False), (1, 7): (11, False), (1, 8): (17, False), (1, 10): (25, True),
}
# compiled instantiations, cnt -> forms ("U" every layer has cnt links, "R" ragged): ldpc_inst_*.cu and
# ldpc2_inst_*.cu (one thread per row) list the same set, ldpc2l_inst_*.cu (two threads per row) its own
ONE_LANE = {2: "UR", 3: "U", 4: "U", 5: "UR", 8: "U", 9: "U", 11: "R", 12: "U", 16: "U", 17: "R", 20: "U", 25: "U", 28: "U"}
TWO_LANES = {8: "U", 9: "U", 11: "R", 12: "U", 16: "U", 17: "R", 20: "U", 25: "U", 28: "U"}


def has_two_lanes(code):
    return CODE_LINKS[code][0] in TWO_LANES


def selected_shape(code, lanes2):
    """(CNT, uniform form) that pick / pickl and is_uniform (ldpc_decoder.cu) choose for the code"""
    max_cnt, uniform = CODE_LINKS[code]
    table = TWO_LANES if lanes2 else ONE_LANE
    cnt = max_cnt if lanes2 else min(c for c in table if c >= max_cnt)
    use_u = uniform and cnt == max_cnt and "U" in table[cnt]
    assert use_u or "R" in table[cnt], (code, cnt)
    return cnt, use_u


def occupancy(cnt, occ3):
    return (3 if cnt <= 9 else 2) if occ3 else (2 if cnt <= 9 else 1)


def instantiation(code, v2, lanes2, occ3, chains, streamed):
    """the kernel a code launches, as parse_kernel spells it"""
    lanes2 = v2 and lanes2 and has_two_lanes(code)
    cnt, use_u = selected_shape(code, lanes2)
    if lanes2:
        return ("ldpc_v2l_kernel", cnt, not use_u, streamed)
    if v2:
        return ("ldpc_v2_kernel", cnt, not use_u, streamed, occupancy(cnt, occ3))
    return ("ldpc_pair_kernel", cnt, use_u, streamed, chains, occupancy(cnt, occ3))


def reachable_instantiations():
    """every instantiation some code selects under some combination of the overrides"""
    out = set()
    for code in CODE_LINKS:
        for st in (False, True):
            for occ3 in (False, True):
                out.add(instantiation(code, True, False, occ3, False, st))
                out.add(instantiation(code, True, True, occ3, False, st))
                for ch in (False, True):
                    out.add(instantiation(code, False, False, occ3, ch, st))
    return out


def compiled_instantiations():
    out = set()
    for st in (False, True):
        for cnt, forms in ONE_LANE.items():
            for f in forms:
                rg = f == "R"
                for occ3 in (False, True):
                    out.add(("ldpc_v2_kernel", cnt, rg, st, occupancy(cnt, occ3)))
                    for ch in (False, True):
                        out.add(("ldpc_pair_kernel", cnt, not rg, st, ch, occupancy(cnt, occ3)))
        for cnt, forms in TWO_LANES.items():
            for f in forms:
                out.add(("ldpc_v2l_kernel", cnt, f == "R", st))
    return out


_KERNEL_RE = re.compile(r"\b(ldpc_pair_kernel|ldpc_v2l_kernel|ldpc_v2_kernel)<([^<>]*)>")


def parse_kernel(name):
    """('ldpc_v2_kernel', 9, False, True, 3) from 'void s2::v2::ldpc_v2_kernel<9, false, true, 3>(s2::LdpcParams2)'"""
    m = _KERNEL_RE.search(name)
    if not m:
        return None
    args = []
    for a in m.group(2).split(","):
        a = a.strip()
        args.append(a == "true" if a in ("true", "false") else int(a.rstrip("uUlL")))
    return (m.group(1), *args)


# ---- oracle frames (parent process) ------------------------------------------------------------------------------------
def code_frames(short, rate, m=M):
    """m distinct frames: a codeword (0 iterations), all-zero LLRs, saturated input, uniform random int8, a frame
    with every 97th LLR zeroed, a frame far below threshold (fails at 25 iterations), and make_llrs' spread around
    the code's threshold for the rest"""
    from test_gpu_parity import _SNR, make_llrs

    seed = 7000 + 100 * short + rate
    rng = np.random.default_rng(seed)
    n_spread = m - 6
    out = np.zeros((m, code_params(short, rate)["N"]), np.int8)
    out[6:] = make_llrs(short, rate, n_spread, seed)
    _, code = orclib.encode_frame(short, rate, rng)
    out[0] = np.where(code > 0, -9, 9)
    out[1] = 0
    out[2] = np.where(out[6 + n_spread // 2] < 0, -128, 127)
    out[3] = rng.integers(-128, 128, out.shape[1], dtype=np.int8)
    out[4] = out[6 + n_spread // 3]
    out[4, ::97] = 0
    _, code = orclib.encode_frame(short, rate, rng)
    out[5] = orclib.awgn_llr(code, _SNR[rate] + 0.4 * short - 1.5, rng)
    return out


def oracle_ldpc(short, rate, llr, max_trials):
    o = orclib.oracle()
    post = llr.copy()
    iters = np.array([o.orc_ldpc_decode(short, rate, post[i], max_trials) for i in range(len(llr))], np.int16)
    return post, iters


def oracle_stage(short, rate, post, iters):
    """BBFRAME bytes, BCH corrections and result flags from the 25-iteration posterior (what orc_decode_frame does
    after its LDPC decode, without decoding again)"""
    o = orclib.oracle()
    p = code_params(short, rate)
    K, kb = p["K"], p["kbch"] // 8
    bb = np.zeros((len(post), kb), np.uint8)
    corr = np.zeros(len(post), np.int16)
    flags = np.zeros(len(post), np.uint32)
    for i in range(len(post)):
        buf = np.zeros(K // 8, np.uint8)
        o.orc_repack(post[i], K, buf)
        corr[i] = o.orc_bch_decode(short, rate, buf)
        o.orc_descramble(short, rate, buf)
        bb[i] = buf[:kb]
        crc = o.orc_bbheader_crc8(np.ascontiguousarray(bb[i]))
        flags[i] = (iters[i] < 0) * 1 | (corr[i] < 0) * 2 | (crc != 0) * 4
    return bb, corr, flags


def key(short, rate, what):
    return f"{'s' if short else 'n'}{rate}_{what}"


# ---- worker (subprocess) -----------------------------------------------------------------------------------------------
class Compare:
    """mismatch counts per field over the positions of a tiled batch, and the first mismatch"""

    def __init__(self, content):
        self.content = content
        self.groups = [np.nonzero(content == c)[0] for c in range(int(content.max()) + 1)]
        self.counts = {}
        self.first = None

    def field(self, name, got, want):
        """got[p] must equal want[content[p]] at every position p"""
        bad = []
        for c, rows in enumerate(self.groups):
            g = got[rows].reshape(len(rows), -1)
            w = want[c].reshape(1, -1)
            bad.append(rows[(g != w).any(axis=1)])
        bad = np.sort(np.concatenate(bad))
        self.counts[name] = int(len(bad))
        if len(bad) and (self.first is None or bad[0] < self.first["position"]):
            p = int(bad[0])
            g, w = got[p].reshape(-1), want[self.content[p]].reshape(-1)
            i = int(np.nonzero(g != w)[0][0])
            self.first = dict(position=p, field=name, frame=int(self.content[p]), index=i, expected=int(w[i]), actual=int(g[i]))

    def positions(self, name, got):
        """got[p] == p (result tags)"""
        want = np.arange(len(got))
        bad = np.nonzero(got != want)[0]
        self.counts[name] = int(len(bad))
        if len(bad) and (self.first is None or bad[0] < self.first["position"]):
            p = int(bad[0])
            self.first = dict(position=p, field=name, expected=p, actual=int(got[p]))

    def report(self):
        return dict(positions=len(self.content), mismatches=self.counts, first=self.first)


def stage_fields(cmp, bb, res, want):
    cmp.field("bbframe", bb, want["bb"])
    cmp.field("ldpc_iters", res["ldpc_iters"], want["it25"])
    cmp.field("bch_corr", res["bch_corr"], want["corr"])
    cmp.field("flags", res["flags"], want["flags"])
    cmp.positions("tag", res["tag"])
    return cmp.report()


def kernels_of(prof, tmpdir):
    """kernels in launch order, with their launch shape, from the profiler's trace"""
    path = os.path.join(tmpdir, "trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
        ev = json.load(f)
    ev = ev.get("traceEvents", ev) if isinstance(ev, dict) else ev
    ks = sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e.get("ts", 0))
    return [dict(name=e["name"], grid=e.get("args", {}).get("grid"), block=e.get("args", {}).get("block")) for e in ks]


def main(npz_path, out_path):
    import torch
    from torch.profiler import ProfilerActivity, profile

    from fec import QPSK_MODCOD_OF_RATE, pkg

    t_start = time.time()
    data = np.load(npz_path)
    codes = [tuple(int(x) for x in c) for c in data["codes"]]
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = batch_size(sms)
    content = tile(n)
    dev = torch.device("cuda", 0)
    dec = pkg.DVBS2Decoder(devices=[0], max_batch=n, max_trials=25)
    dec255 = pkg.DVBS2Decoder(devices=[0], max_batch=255, max_trials=25)
    report = dict(env={k: v for k, v in os.environ.items() if k.startswith("DVBS2FEC_")}, sms=sms, n=n, codes={})
    cmp = lambda: Compare(content)  # noqa: E731
    with tempfile.TemporaryDirectory() as tmpdir:
        for short, rate in codes:
            t0 = time.time()
            want = {w: data[key(short, rate, w)] for w in ("llr", "post25", "it25", "post1", "it1", "post3", "it3", "bb", "corr", "flags")}
            frames = want["llr"]
            m = len(frames)
            for d in (dec, dec255):
                d.setDemodParams(QPSK_MODCOD_OF_RATE[rate], bool(short), False)
            batch = np.ascontiguousarray(frames[content])
            paths = {}
            # profiled: the M frames alone at max_trials 1 (non-streamed), then the whole batch in one streamed launch
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                small = frames.copy()
                it = dec.ldpc_decode(small, 1)
                bb, res = dec.decode_batch(batch)
                torch.cuda.synchronize()
            kernels = kernels_of(prof, tmpdir)
            own = Compare(np.arange(m))
            own.field("posterior", small, want["post1"])
            own.field("ldpc_iters", it, want["it1"])
            paths["ldpc_decode_max_trials_1"] = own.report()
            paths["decode_batch"] = stage_fields(cmp(), bb, res, want)
            small = frames.copy()
            it = dec.ldpc_decode(small, 3)
            own = Compare(np.arange(m))
            own.field("posterior", small, want["post3"])
            own.field("ldpc_iters", it, want["it3"])
            paths["ldpc_decode_max_trials_3"] = own.report()
            # 1: one non-streamed launch over the whole batch, posterior written in place
            work = batch.copy()
            it = dec.ldpc_decode(work, 25)
            c = cmp()
            c.field("posterior", work, want["post25"])
            c.field("ldpc_iters", it, want["it25"])
            paths["ldpc_decode"] = c.report()
            del work
            # 3: 255-frame chunks alternating over both slots, every full chunk ends in a half-empty pair
            bb, res = dec255.decode_batch(batch)
            paths["decode_batch_max_batch_255"] = stage_fields(cmp(), bb, res, want)
            # 4: torch device buffers
            d_llr = torch.from_numpy(batch).to(dev)
            d_bb = torch.empty((n, dec.kbch // 8), dtype=torch.uint8, device=dev)
            d_res = torch.empty((n, pkg.RESULT_DTYPE.itemsize), dtype=torch.uint8, device=dev)
            dec.decode_batch_device(d_llr.data_ptr(), n, d_bb.data_ptr(), d_res.data_ptr(), torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            res = d_res.cpu().numpy().view(pkg.RESULT_DTYPE).reshape(-1)
            paths["decode_batch_device"] = stage_fields(cmp(), d_bb.cpu().numpy(), res, want)
            del d_llr, d_bb, d_res
            report["codes"][f"{short},{rate}"] = dict(paths=paths, kernels=kernels, seconds=round(time.time() - t0, 2))
    dec.close()
    dec255.close()
    report["seconds"] = round(time.time() - t_start, 1)
    with open(out_path, "w") as f:
        json.dump(report, f)


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
