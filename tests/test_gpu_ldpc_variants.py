"""Every LDPC kernel variant against the CPU oracle, on all 21 codes, at batch sizes where every CTA of the
persistent grid decodes several frame pairs.  Needs a B200.

ldpc_prepare picks one kernel per code from a matrix of instantiations (one or two threads per row, first or second
generation, uniform or ragged, streamed or not, 2 or 3 CTAs per SM); three performance tables choose the cell, and
process-wide overrides flip them.  Each environment of ENVS runs in its own subprocess (the overrides are read once
per process): ldpc_variant_worker.py decodes a batch tiled from M oracle frames per code through four entry points
and compares every position with the oracle.  The profiler's kernel names prove which instantiation ran, and the
union over the matrix must contain every instantiation some code can select.

Also here: BCH on all 21 codes, with errors on the edges of the syndrome stage's per-lane byte chunks."""
import json
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import ldpc_variant_worker as W
import orclib
from fec import QPSK_MODCOD_OF_RATE, pkg
from orclib import ALL_CODES, code_params

pytestmark = pytest.mark.gpu

V2, LANES2, OCC3, CHAINS, MINLEV = ("DVBS2FEC_LDPC_V2", "DVBS2FEC_LDPC_LANES2", "DVBS2FEC_LDPC_OCC3", "DVBS2FEC_LDPC_CHAINS",
                                    "DVBS2FEC_CHAIN_MINLEV")
ENVS = {
    "default": {},
    "lanes2": {LANES2: "1"},
    "one-lane-occ2": {LANES2: "0", OCC3: "0"},
    "one-lane-occ3": {LANES2: "0", OCC3: "1"},
    "gen1": {V2: "0", CHAINS: "0", OCC3: "0"},
    "gen1-all-chains-occ3": {V2: "0", CHAINS: "1", MINLEV: "2", OCC3: "1"},   # every layer plan_chains accepts
    # the other two (chains, occupancy) pairs of the first-generation kernel, so that every instantiation runs
    "gen1-chains-occ2": {V2: "0", CHAINS: "1", OCC3: "0"},
    "gen1-occ3": {V2: "0", CHAINS: "0", OCC3: "1"},
}
PATHS = ("ldpc_decode", "ldpc_decode_max_trials_1", "ldpc_decode_max_trials_3", "decode_batch", "decode_batch_max_batch_255",
         "decode_batch_device")
WORKER = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ldpc_variant_worker.py")


def _code_job(code):
    short, rate = code
    llr = W.code_frames(short, rate)
    out = {"llr": llr}
    for mt in (25, 1, 3):
        out[f"post{mt}"], out[f"it{mt}"] = W.oracle_ldpc(short, rate, llr, mt)
    return out


@pytest.fixture(scope="module")
def oracle_npz(tmp_path_factory):
    """the M frames of every code and the oracle's answers: posterior and iterations at 25, 1 and 3 iterations,
    BBFRAME, BCH corrections and flags"""
    for short, rate in ALL_CODES:
        code_params(short, rate)          # the oracle builds its schedules lazily: once, before the threads
    orclib.oracle().orc_bch_decode(0, 3, np.zeros(4050, np.uint8))
    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:   # ctypes drops the GIL
        answers = dict(zip(ALL_CODES, ex.map(_code_job, ALL_CODES)))
    arrays = {"codes": np.array(ALL_CODES, np.int32)}
    for (short, rate), a in answers.items():
        a["bb"], a["corr"], a["flags"] = W.oracle_stage(short, rate, a["post25"], a["it25"])
        for k, v in a.items():
            arrays[W.key(short, rate, k)] = v
    path = tmp_path_factory.mktemp("ldpc_variants") / "oracle.npz"
    np.savez(path, **arrays)
    return path, {code: a["it25"] for code, a in answers.items()}


@pytest.fixture(scope="module")
def run_env(oracle_npz, tmp_path_factory):
    """env name -> the worker's report, one subprocess per environment, cached for the module"""
    reports = {}
    out_dir = tmp_path_factory.mktemp("ldpc_variant_reports")

    def run(name):
        if name not in reports:
            env = {k: v for k, v in os.environ.items() if not k.startswith("DVBS2FEC_")}
            env.update(ENVS[name])
            out = out_dir / f"{name}.json"
            flags = ["-s"] if sys.flags.no_user_site else []
            p = subprocess.run([sys.executable, *flags, WORKER, str(oracle_npz[0]), str(out)], env=env, timeout=900,
                               capture_output=True, text=True)
            assert p.returncode == 0, f"worker for {name} failed ({p.returncode}):\n{p.stdout[-3000:]}\n{p.stderr[-6000:]}"
            with open(out) as f:
                reports[name] = json.load(f)
        return reports[name]

    return run


@pytest.mark.parametrize("code", ALL_CODES, ids=lambda c: f"{'s' if c[0] else 'n'}{c[1]}")
def test_oracle_frames_cover_iteration_classes(oracle_npz, code):
    its = set(oracle_npz[1][code].tolist())
    assert 0 in its and -1 in its and len(its) >= 5, sorted(its)


def _ldpc_launches(kernels):
    return [(W.parse_kernel(k["name"]), k) for k in kernels if W.parse_kernel(k["name"])]


@pytest.mark.parametrize("env_name", list(ENVS))
def test_variant_bit_exact(run_env, env_name):
    rep = run_env(env_name)
    env = ENVS[env_name]
    sms, n = rep["sms"], rep["n"]
    assert n % 2 == 1 and n >= 8 * sms * 3
    assert sorted(rep["codes"]) == sorted(f"{s},{r}" for s, r in ALL_CODES)
    bad = []
    lines = [f"[{env_name}] {env or 'no overrides'}: {n} frames per batch, {sms} SMs, {rep['seconds']} s"]
    for ck, c in sorted(rep["codes"].items()):
        code = tuple(int(x) for x in ck.split(","))
        assert sorted(c["paths"]) == sorted(PATHS)
        for path, r in c["paths"].items():
            if any(r["mismatches"].values()):
                bad.append(f"code {code} {path}: {r['mismatches']}, first {r['first']}")
        launches = _ldpc_launches(c["kernels"])
        if not c["kernels"]:
            pytest.fail(f"the profiler returned no kernel records (code {code}, {env_name}): CUDA activity tracing is unavailable")
        # the profiled window runs the non-streamed ldpc_decode, then decode_batch's one streamed launch
        assert len(launches) == 2, (code, [k["name"] for k in c["kernels"]])
        (k1, _), (k2, big) = launches
        assert k1[3] is False and k2[3] is True, (code, k1, k2)         # STREAMED
        assert k1[:3] + k1[4:] == k2[:3] + k2[4:], (code, k1, k2)
        fam, cnt = k1[0], k1[1]
        two = W.has_two_lanes(code)
        want_cnt, want_u = W.selected_shape(code, fam == "ldpc_v2l_kernel")
        assert cnt == want_cnt and (k1[2] == want_u if fam == "ldpc_pair_kernel" else k1[2] != want_u), (code, k1)
        if env.get(LANES2) == "1":
            assert fam == ("ldpc_v2l_kernel" if two else "ldpc_v2_kernel"), (code, k1)
        if env.get(LANES2) == "0":
            assert fam != "ldpc_v2l_kernel", (code, k1)
        if env.get(V2) == "0":
            assert fam == "ldpc_pair_kernel", (code, k1)
            assert k1[4] == (env[CHAINS] == "1"), (code, k1)            # CHAINS
        if OCC3 in env and fam != "ldpc_v2l_kernel":
            assert k1[-1] == W.occupancy(cnt, env[OCC3] == "1"), (code, k1)
        # the streamed launch's grid: every CTA takes at least four pairs from the work counter
        grid = big["grid"][0] if big["grid"] else None
        assert grid is not None and 8 * grid <= n, (code, big)
        lines.append(f"  {code}: {k1[0]}<{', '.join(str(x) for x in k1[1:])}> grid {grid}x{big['block'][0]}, "
                     f"{sum(sum(r['mismatches'].values()) for r in c['paths'].values())} mismatches over "
                     f"{len(c['paths'])} paths, {c['seconds']} s")
    print("\n".join(lines))
    assert not bad, "\n".join(bad)


def test_every_reachable_instantiation_runs(run_env):
    launched = set()
    for name in ENVS:
        for c in run_env(name)["codes"].values():
            launched |= {k for k, _ in _ldpc_launches(c["kernels"])}
    reach = W.reachable_instantiations()
    missing = sorted(reach - launched, key=str)
    assert not missing, f"{len(missing)} reachable instantiations never ran: {missing[:20]}"
    assert launched <= reach, sorted(launched - reach, key=str)


# ---- BCH on all 21 codes ---------------------------------------------------------------------------------------------
def bch_error_sets(short, rate, rng):
    """bit positions to flip, one set per frame: random errors 0, 1, 2, t-1 .. t+2; the first and last bit of every
    lane's byte chunk of the syndrome stage (bch_decoder.cu: 32 chunks of ceil(nbch/256) bytes), t at a time and
    once t+1 of them; the last two parity bits; errors only in the last, short chunk"""
    p = code_params(short, rate)
    K, t = p["K"], p["t"]
    nbytes = K // 8
    chunk = -(-nbytes // 32)
    lanes = [(b, min(b + chunk, nbytes)) for b in range(0, nbytes, chunk)]
    edges = sorted({8 * b for b, _ in lanes} | {8 * e - 1 for _, e in lanes})
    sets = [rng.choice(K, ne, replace=False) for ne in (0, 1, 2, t - 1, t, t + 1, t + 2)]
    sets += [edges[i:i + t] for i in range(0, len(edges), t)]
    sets.append(edges[-t - 1:])
    sets.append([K - 2, K - 1])
    b, e = lanes[-1]
    sets.append(rng.choice(np.arange(8 * b, 8 * e), min(t, 8 * (e - b)), replace=False))
    return sets, lanes


@pytest.fixture(scope="module")
def bch_dec():
    d = pkg.DVBS2Decoder(max_batch=64, max_trials=25)
    yield d
    d.close()


@pytest.mark.parametrize("short,rate", ALL_CODES)
def test_bch_bit_exact_all_codes(bch_dec, short, rate):
    bch_dec.setDemodParams(QPSK_MODCOD_OF_RATE[rate], bool(short), False)
    o = orclib.oracle()
    p = code_params(short, rate)
    K, kbch, t = p["K"], p["kbch"], p["t"]
    rng = np.random.default_rng(300 + 20 * short + rate)
    sets, _ = bch_error_sets(short, rate, rng)
    frames = np.zeros((len(sets), K // 8), np.uint8)
    for i, where in enumerate(sets):
        frames[i, : kbch // 8] = rng.integers(0, 256, kbch // 8, dtype=np.uint8)
        assert o.orc_bch_encode(short, rate, frames[i]) == 0
        for e in where:
            frames[i, e >> 3] ^= 0x80 >> (e & 7)
    want = frames.copy()
    want_c = np.array([o.orc_bch_decode(short, rate, want[i]) for i in range(len(sets))], np.int16)
    for i, where in enumerate(sets):
        if len(where) <= t:
            assert want_c[i] == len(where), (i, len(where), want_c[i])
    got = frames.copy()
    got_c = bch_dec.bch_decode(got)
    assert np.array_equal(got_c, want_c), (got_c, want_c)
    assert np.array_equal(got, want)
