#!/usr/bin/env python3
"""Benchmark of the DVB-S2 decode stage (BASELINE.json metric: decoded information Gbit/s, QPSK 1/2 normal).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--esn0 DB] [--pool F] [--dump-outputs DIR]

One "step" = R passes of the hot path (LDPC + BCH + descramble, from int8 LLRs) over a pool of F synthetic
FECFRAMEs (defaults F = 16384, R = 5: 81920 frames per step, so that the driver's 20 steps time more than two
seconds of sustained decoding).  Per rank the pool is resident in HBM and larger than L2 (F*64800 B = 1.06 GB),
so consecutive launches never find their input in cache.  `value` is timed with CUDA events on the stream the
kernels run on; `e2e` goes through dvbs2fec_decode_batch with pinned HOST buffers (H2D + kernels + D2H).
After the timed region a sample of the last launch's results (the slowest frames and random ones) is checked
against the CPU oracle byte for byte: `parity_checked` / `parity_mismatches` (a mismatch makes the run fail).
Multi-GPU (torchrun, one rank per GPU): frames are independent, every rank decodes its own pool, no
data-path collective; timing is barrier-bracketed and the max over ranks is used.  With N > 1 rank 0 then
also drives ONE handle configured with all N devices (the in-process dispatcher the SDR++ plugin would use,
reference batch seam module_dvbs2_demod.cpp:343-367) through decode_batch and submit/collect while the other
ranks idle, checks its output bytes against the single-device result and reports `dispatcher`.

`--dump-outputs DIR` writes, after the timed steps, what rank 0's last timed launch returned, as float32 / float64
.npy files of at most DUMP_BYTES in all: the BBFRAME bytes of a fixed, seeded sample of DUMP_FRAMES frames
(bbframe_bytes.npy, rows in the order of frame_index.npy) and the result records (tag.npy, ldpc_iters.npy,
bch_corr.npy, flags.npy) of every frame, or of a seeded sample of DUMP_RECORDS frames when the pool is larger
(record_index.npy). The inputs are generated from fixed seeds, so two builds run with the same arguments can be
compared output for output.

`--impl reference` times the reference's own CPU code (oracle/_ref, compiled from /root/reference
unmodified; else the oracle port) on the host cores with the same pool generator and metric.
"""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODCOD, SHORT, RATE_ENUM = 4, False, 3  # QPSK 1/2 normal
MAX_TRIALS = 25
LLR_SCALE = 4.0  # "L4" generator of SURVEY.md 8d: rint(4 * true channel LLR), clamped to +-127
HBM_BYTES_PER_FRAME = 64800 + 32208 // 8 + 16  # algorithmic: LLRs in, BBFRAME + result record out
DUMP_FRAMES = 2048  # BBFRAMEs written by --dump-outputs: 2048 x 4026 bytes as float32 = 33 MB
DUMP_RECORDS = 1 << 19  # result records written by --dump-outputs: 32 bytes each with their index = 16.8 MB
DUMP_BYTES = 64 << 20


def sorted_sample(n, k, seed):
    """all of range(n) when it has at most k entries, else k of them drawn without replacement, ascending"""
    return np.arange(n) if n <= k else np.sort(np.random.default_rng(seed).choice(n, k, replace=False))


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f).get("hbm_gbs"), "measured"
    except Exception:
        return 6650.0, "fallback"


def newest_profile(pattern):
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", pattern)))
    for f in reversed(files):
        try:
            return json.load(open(f)), os.path.basename(f)
        except Exception:
            pass
    return None, None


def onchip_roofline(edge_updates_per_s, sm_mhz, sms):
    """Fractions of the MEASURED on-chip peaks (profiles/r*_onchip_peaks.json: ALU-pipe issue rate and shared-memory
    wavefront rate per SM, tools/micro/pipes.cu) that the live edge-update rate of this run amounts to, using the
    ALU-pipe instructions and shared-memory wavefronts per edge update of the newest committed ncu capture of the
    LDPC kernel (profiles/r*_ldpc_v2_kernel.json, tools/ncu_summary.py).  SURVEY.md 8(d) formulas."""
    cap, cap_name = newest_profile("r*_ldpc_v2_kernel.json")
    peaks, peaks_name = newest_profile("r*_onchip_peaks.json")
    if not cap or not peaks or "alu_warp_instr_per_edge_update" not in cap or not sm_mhz:
        return None
    alu_peak = peaks["issue"]["VIADDMNMX.S16x2.RELU"]                       # warp instructions / clk / SM, ALU pipe
    smem_peak = peaks["shared_memory"]["LDS.128"]["bytes_per_clk_per_sm"] / 128.0   # wavefronts / clk / SM
    clk = sm_mhz * 1e6
    alu_rate = edge_updates_per_s * cap["alu_warp_instr_per_edge_update"]
    smem_rate = edge_updates_per_s * cap["smem_wavefronts_per_edge_update"]
    return {"alu_frac": alu_rate / (alu_peak * sms * clk), "smem_frac": smem_rate / (smem_peak * sms * clk),
            "alu_peak_warp_instr_per_clk_per_sm": alu_peak, "smem_peak_wavefronts_per_clk_per_sm": smem_peak,
            "alu_warp_instr_per_edge_update": cap["alu_warp_instr_per_edge_update"],
            "smem_wavefronts_per_edge_update": cap["smem_wavefronts_per_edge_update"],
            "sm_clock_mhz": sm_mhz, "sms": sms, "peaks_from": peaks_name, "instruction_counts_from": cap_name,
            "ncu_of_that_capture": {k: cap.get(k) for k in ("alu_pipe_pct", "issue_slots_busy_pct", "fma_pipe_pct",
                                                            "lsu_pipe_pct", "dram_throughput_pct", "l2_hit_rate_pct")}}


def ncu_traffic_per_frame():
    cap, name = newest_profile("r*_ldpc_v2_kernel.json")
    if cap and "dram_traffic_bytes_per_frame" in cap:
        return cap["dram_traffic_bytes_per_frame"], name
    return None


def make_codewords(pkg, n, seed):
    rng = np.random.default_rng(seed)
    info = pkg.modcod_info(MODCOD, SHORT)
    out = np.zeros((n, info["nldpc"]), np.uint8)
    for i in range(n):
        out[i] = pkg.encode_fecframe(MODCOD, SHORT, rng.integers(0, 256, info["kbch"] // 8, dtype=np.uint8))
    return out


def llr_params(esn0_db):
    a = 1.0 / np.sqrt(2.0)
    sigma2 = 1.0 / (2.0 * 10 ** (esn0_db / 10.0))
    return a, sigma2


def make_pool_numpy(code_bits, nframes, esn0_db, seed):
    rng = np.random.default_rng(seed)
    a, sigma2 = llr_params(esn0_db)
    out = np.zeros((nframes, code_bits.shape[1]), np.int8)
    for i in range(nframes):
        y = (1.0 - 2.0 * code_bits[i % len(code_bits)].astype(np.float32)) * a
        y = y + rng.normal(0.0, np.sqrt(sigma2), y.shape).astype(np.float32)
        out[i] = np.clip(np.rint(LLR_SCALE * 2.0 * a * y / sigma2), -127, 127).astype(np.int8)
    return out


def make_pool_torch(torch, code_bits, nframes, esn0_db, seed, device):
    a, sigma2 = llr_params(esn0_db)
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    cw = torch.from_numpy(code_bits).to(device)
    pool = torch.empty((nframes, cw.shape[1]), dtype=torch.int8, device=device)
    step = 256
    for f0 in range(0, nframes, step):
        m = min(step, nframes - f0)
        idx = (torch.arange(f0, f0 + m, device=device) % cw.shape[0])
        y = (1.0 - 2.0 * cw[idx].float()) * a
        y += torch.randn(y.shape, generator=g, device=device) * float(np.sqrt(sigma2))
        pool[f0:f0 + m] = torch.clamp(torch.round(LLR_SCALE * 2.0 * a * y / sigma2), -127, 127).to(torch.int8)
    return pool


class ClockSampler:
    """nvidia-smi in loop mode (one process, 50 ms period) while the timed regions run."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def start(self):
        time.sleep(0.15)   # let the first samples arrive before the timed region

    def stop(self):
        if not self.proc:
            return
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            out = ""
        for ln in out.splitlines():
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) >= 6:
                self.rows.append(parts)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


# ------------------------------------------------------------------ CPU reference arm
# Nothing below imports the product library: codewords for this arm come from the oracle's own encoder.
_cpu_state = {}


def _cpu_worker_init(kind):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import orclib
    _cpu_state["orclib"] = orclib
    _cpu_state["kind"] = kind
    _cpu_state["lib"] = orclib.ref() if kind == "reference" else orclib.oracle()


def _cpu_decode(llr, mode):
    """llr: (n, 64800) int8 -> (frames done, decoded-ok count).
    mode 'simd16'   : the vendored library used as designed -- one frame per SSE4.1 lane, blocks = 16
                      (LDPCDecoder::operator(), layered_decoder.hh:121-133) + per-frame BBFrameBCH::decode + descrambler;
    mode 'lane0'    : one BBFrameLDPC::decode call per frame (bbframe_ldpc.cpp:123-139: lane 0 only), what a correct
                      per-frame use of the reference's own wrapper costs;
    mode 'shipped'  : the module's pattern (module_dvbs2_demod.cpp:345-367, SURVEY note N1): ONE decode call per 16
                      frames, which decodes only the first; all 16 then go through repack + BCH + descramble;
    mode 'port'     : the scalar oracle restatement (when the reference could not be compiled)."""
    orclib, lib = _cpu_state["orclib"], _cpu_state["lib"]
    n = llr.shape[0]
    ok = 0
    if mode == "port":
        bb = np.zeros(32208 // 8, np.uint8)
        for k in range(n):
            it, co = C.c_int(), C.c_int()
            lib.orc_decode_frame(0, RATE_ENUM, llr[k].copy(), MAX_TRIALS, bb, C.byref(it), C.byref(co))
            ok += co.value >= 0
        return n, ok
    lanes = 16
    for f0 in range(0, n, lanes):
        blk = np.ascontiguousarray(llr[f0:f0 + lanes])
        if blk.shape[0] < lanes:
            blk = np.concatenate([blk, np.repeat(blk[-1:], lanes - blk.shape[0], 0)])
        if mode == "simd16":
            lib.ref_ldpc_decode_simd(0, RATE_ENUM, blk.reshape(-1), MAX_TRIALS)
        elif mode == "lane0":
            for k in range(lanes):
                lib.ref_ldpc_decode(0, RATE_ENUM, blk[k], MAX_TRIALS)
        else:  # shipped
            lib.ref_ldpc_decode(0, RATE_ENUM, blk[0], MAX_TRIALS)
        for k in range(min(lanes, n - f0)):
            packed = np.packbits((blk[k, :32400] < 0).astype(np.uint8))
            c = lib.ref_bch_decode(0, RATE_ENUM, packed)
            lib.ref_descramble(0, RATE_ENUM, packed)
            ok += c >= 0
    return n, ok


def _cpu_worker(job):
    llr, mode = job
    return _cpu_decode(llr, mode)


def cpu_model():
    try:
        out = subprocess.run(["lscpu"], capture_output=True, text=True).stdout
        d = dict((ln.split(":", 1)[0].strip(), ln.split(":", 1)[1].strip()) for ln in out.splitlines() if ":" in ln)
        return {"model": d.get("Model name"), "logical_cpus": int(d.get("CPU(s)", 0)), "threads_per_core": int(d.get("Thread(s) per core", 1)),
                "sockets": int(d.get("Socket(s)", 1)), "hypervisor": d.get("Hypervisor vendor"),
                "compiler_flags": "g++ -O3 -std=c++17 -msse4.1 (the reference's own, CMakeLists.txt:56)"}
    except Exception:
        return {}


def cpu_baseline(pool_host, budget_s, procs, mode=None):
    """Bounded sample of the same workload on the host cores.  Returns dict for the JSON line."""
    import multiprocessing as mp
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import orclib
    kind = "reference" if orclib.have_ref() else "port"
    mode = mode or ("simd16" if kind == "reference" else "port")
    per_job = 16
    ctx = mp.get_context("fork")
    with ctx.Pool(procs, initializer=_cpu_worker_init, initargs=(kind,)) as pool:
        # calibrate on one job per process, then size the sample to the budget
        jobs = [(pool_host[(i * per_job) % len(pool_host):][:per_job], mode) for i in range(procs)]
        t0 = time.perf_counter()
        pool.map(_cpu_worker, jobs)
        dt = time.perf_counter() - t0
        rounds = max(1, min(64, int(budget_s / max(dt, 1e-3))))
        jobs = [(pool_host[(i * per_job) % (len(pool_host) - per_job + 1):][:per_job], mode) for i in range(procs * rounds)]
        t0 = time.perf_counter()
        res = pool.map(_cpu_worker, jobs)
        dt = time.perf_counter() - t0
    frames = sum(r[0] for r in res)
    what = {"simd16": "LDPC 16 frames per SSE4.1 call (blocks=16) + per-frame BCH + descramble",
            "lane0": "one BBFrameLDPC::decode (lane 0) per frame + BCH + descramble",
            "shipped": "module pattern: one LDPC call per 16 frames (15 of 16 NOT decoded, SURVEY N1) + BCH + descramble",
            "port": "scalar oracle port"}[mode]
    return {"value": frames * 32208 / dt / 1e9, "unit": "Gbit/s", "cores": procs, "kind": kind, "mode": mode,
            "frames_per_s": frames / dt, "seconds": dt, "decoded_ok": int(sum(r[1] for r in res)), "frames": frames,
            "sample": "%d frames of the QPSK 1/2 pool, %d processes, %s" % (frames, procs, what)}


def oracle_codewords(n, seed):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import orclib
    rng = np.random.default_rng(seed)
    return np.stack([orclib.encode_frame(0, RATE_ENUM, rng)[1] for _ in range(n)])


def parity_sample(pkg, llr_rows, bb_rows, res_rows):
    """The CPU oracle (test infrastructure, outside every timed region) on the given frames: LDPC iteration count,
    BCH correction count and BBFRAME bytes must equal what the GPU produced.  Returns the number of mismatches."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import orclib
    o = orclib.oracle()
    bad = 0
    want = np.zeros(bb_rows.shape[1], np.uint8)
    for k in range(llr_rows.shape[0]):
        it, co = C.c_int(), C.c_int()
        o.orc_decode_frame(0, RATE_ENUM, np.ascontiguousarray(llr_rows[k]).copy(), MAX_TRIALS, want, C.byref(it), C.byref(co))
        if it.value != int(res_rows["ldpc_iters"][k]) or co.value != int(res_rows["bch_corr"][k]) or not np.array_equal(want, bb_rows[k]):
            bad += 1
    return bad


# ------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--esn0", type=float, default=2.2)
    ap.add_argument("--pool", type=int, default=16384, help="distinct frames resident per GPU = frames per launch")
    ap.add_argument("--repeat", type=int, default=5, help="launches over the pool per step")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--parity-frames", type=int, default=64)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed launch's outputs as .npy files into DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the CUDA path; --impl reference has no device outputs")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    kbch, N, links = 32208, 64800, 226799
    workload = ("DVB-S2 QPSK 1/2 normal FECFRAME (64800) LDPC+BCH decode, synthetic AWGN int8 LLRs "
                "(rint(4*LLR)) at Es/N0 %.1f dB, %d max iterations" % (args.esn0, MAX_TRIALS))
    frames_per_step = args.pool * args.repeat
    config = {"workload": workload, "frames_per_step_per_gpu": frames_per_step, "frames_per_launch": args.pool,
              "launches_per_step": args.repeat, "esn0_db": args.esn0, "llr_generator": "L4", "max_iters": MAX_TRIALS,
              "cache": "pool of %d frames = %.0f MB per GPU > 126 MB L2" % (args.pool, args.pool * N / 1e6),
              "parallelism": "frames sharded by GPU, no collective"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        codes = oracle_codewords(32, 1)
        procs = os.cpu_count() or 1
        pool_host = make_pool_numpy(codes, 16 * min(procs, 64), args.esn0, 2)
        t_all, frames_all = 0.0, 0
        last = None
        for s in range(args.warmup + args.steps):
            last = cpu_baseline(pool_host, max(2.0, args.cpu_seconds / 2), procs)
            if s >= args.warmup:
                t_all += last["seconds"]
                frames_all += last["frames"]
        v = frames_all * kbch / t_all / 1e9
        config = dict(config, frames_per_step_per_gpu=last["frames"], frames_per_launch=None, launches_per_step=None,
                      cache="n/a (host)", parallelism="%d host processes, 16 frames per SSE4.1 call" % procs)
        line = {"impl": "reference", "metric": "decoded_info_gbit_s", "value": v, "unit": "Gbit/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_all / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int8", "data": "synthetic",
                "config": config, "frames_per_s": frames_all / t_all,
                "cpu_baseline": {"value": v, "unit": "Gbit/s", "cores": last["cores"], "kind": last["kind"], "sample": last["sample"],
                                 "host": cpu_model()},
                "e2e": {"value": v, "unit": "Gbit/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the decode stage has no CPU path")
    pkg = importlib.import_module("sdrpp-dvbs-demodulator_b200")
    info = pkg.modcod_info(MODCOD, SHORT)
    assert (info["kbch"], info["nldpc"], info["links_total"]) == (kbch, N, links)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    gloo = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        gloo = dist.new_group(backend="gloo")   # host-side waits that leave the GPUs alone (dispatcher leg)

    dec = pkg.DVBS2Decoder(devices=[local_rank], max_batch=args.pool, max_trials=MAX_TRIALS)
    dec.setDemodParams(MODCOD, SHORT, False, MAX_TRIALS)
    codes = make_codewords(pkg, 64, 1 + rank)
    pool = make_pool_torch(torch, codes, args.pool, args.esn0, 100 + rank, dev)
    d_bb = torch.empty((args.pool, kbch // 8), dtype=torch.uint8, device=dev)
    d_res = torch.empty((args.pool, 16), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()

    def step():
        for _ in range(args.repeat):
            dec.decode_batch_device(pool.data_ptr(), args.pool, d_bb.data_ptr(), d_res.data_ptr(), stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        step()
    barrier()
    launches_per_step = dec.last_launch_count() * args.repeat
    sampler = ClockSampler(local_rank)
    sampler.start()
    dec.set_profiling(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    demap_ms, ldpc_ms, bch_ms, nspans = dec.kernel_times()
    dec.set_profiling(False)
    res = d_res.cpu().numpy().view(pkg.RESULT_DTYPE).reshape(-1)
    iters = res["ldpc_iters"].astype(np.int32)
    mean_it = float(np.where(iters < 0, MAX_TRIALS, iters).mean())
    fer = float((res["bch_corr"] < 0).mean())
    dump = None
    if rank == 0 and args.dump_outputs:   # taken now: the parity and latency legs below reuse d_bb
        frame_index = sorted_sample(args.pool, DUMP_FRAMES, 0)
        record_index = sorted_sample(args.pool, DUMP_RECORDS, 1)
        rec = res[record_index]
        dump = {"frame_index": frame_index.astype(np.float64),
                "bbframe_bytes": d_bb[torch.from_numpy(frame_index).to(dev)].cpu().numpy().astype(np.float32),
                "record_index": record_index.astype(np.float64),
                "tag": rec["tag"].astype(np.float64), "ldpc_iters": rec["ldpc_iters"].astype(np.float32),
                "bch_corr": rec["bch_corr"].astype(np.float32), "flags": rec["flags"].astype(np.float64)}
        assert sum(a.nbytes for a in dump.values()) <= DUMP_BYTES

    # ---- parity of what was just timed (outside the timed region): the slowest frames of the last launch and
    #      random ones, GPU result vs CPU oracle
    parity_n = parity_bad = 0
    if rank == 0 and args.parity_frames > 0:
        n_slow = min(args.parity_frames // 4, args.pool)
        order = np.argsort(np.where(iters < 0, MAX_TRIALS + 1, iters))
        pick = set(order[-n_slow:].tolist())
        rng = np.random.default_rng(5)
        while len(pick) < min(args.parity_frames, args.pool):
            pick.add(int(rng.integers(0, args.pool)))
        idx = torch.tensor(sorted(pick), device=dev)
        llr_rows = pool[idx].cpu().numpy()
        bb_rows = d_bb[idx].cpu().numpy()
        parity_n = len(pick)
        parity_bad = parity_sample(pkg, llr_rows, bb_rows, res[sorted(pick)])

    # ---- e2e: public host API, pinned host buffers, copies inside the timed region
    e2e_frames = args.pool
    L = pkg.lib()
    h_in = L.dvbs2fec_alloc_pinned(e2e_frames * N)
    h_bb = L.dvbs2fec_alloc_pinned(e2e_frames * (kbch // 8))
    h_res = L.dvbs2fec_alloc_pinned(e2e_frames * 16)
    host_copy = pool.cpu().numpy()
    C.memmove(h_in, host_copy.ctypes.data, args.pool * N)
    # two chunks per call, one per pipeline slot (tools/e2e_sweep2.py: 8192-frame chunks give 21.2 Gbit/s, 4096 19.5, 1024 14.8:
    # a chunk is one kernel launch, and the fewer frame pairs a launch has per CTA the more its last wave costs)
    dec_e = pkg.DVBS2Decoder(devices=[local_rank], max_batch=max(256, min(8192, args.pool // 2)), max_trials=MAX_TRIALS)
    dec_e.setDemodParams(MODCOD, SHORT, False, MAX_TRIALS)
    for _ in range(2):
        dec_e.decode_batch_raw(h_in, e2e_frames, h_bb, h_res)
    barrier()
    t0 = time.perf_counter()
    e2e_steps = args.steps
    for _ in range(e2e_steps):
        dec_e.decode_batch_raw(h_in, e2e_frames, h_bb, h_res)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    sampler.stop()
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    # ---- what the host side can deliver at all: the same input bytes from page-locked memory, copies only, every rank at
    #      once (under torchrun the ranks share the host's memory controllers and PCIe root complexes)
    pin = torch.from_numpy(host_copy).pin_memory()
    pool.copy_(pin, non_blocking=True)
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    for _ in range(4):
        pool.copy_(pin, non_blocking=True)
    torch.cuda.synchronize()
    h2d_s = (time.perf_counter() - t0) / 4
    del pin
    bb_single = np.ctypeslib.as_array(C.cast(h_bb, C.POINTER(C.c_uint8)), shape=(e2e_frames, kbch // 8)).copy()
    res_single = np.ctypeslib.as_array(C.cast(h_res, C.POINTER(C.c_uint8)), shape=(e2e_frames, 16)).copy()

    # ---- per-frame latency vs batch size (device-resident, one call, median of 5)
    latency = {}
    for b in (2, 16, 128, 1024, 4096, args.pool):
        if b > args.pool or str(b) in latency:
            continue
        ts = []
        for _ in range(5):
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(stream)
            dec.decode_batch_device(pool.data_ptr(), b, d_bb.data_ptr(), d_res.data_ptr(), stream.cuda_stream)
            a1.record(stream)
            torch.cuda.synchronize()
            ts.append(a0.elapsed_time(a1))
        latency[str(b)] = round(sorted(ts)[2], 4)

    # ---- reduce over ranks
    dispatch = importlib.import_module("sdrpp-dvbs-demodulator_b200.dispatch")
    ms_max, e2e_ms_max, ldpc_ms_max, h2d_ms_max = dispatch.reduce_max([ms, e2e_s * 1e3, ldpc_ms, h2d_s * 1e3], device=dev)
    single_e2e_fps = e2e_frames * e2e_steps / e2e_s

    # ---- in-process dispatcher over all N GPUs (rank 0 only, the other ranks wait on the host)
    dispatcher = None
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier(group=gloo)
        if rank == 0:
            dispatcher = dispatcher_leg(pkg, L, world, h_in, e2e_frames, N, kbch, bb_single, res_single, single_e2e_fps)
        dist.barrier(group=gloo)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    frames_total = frames_per_step * args.steps * world
    value = frames_total * kbch / (ms_max * 1e-3) / 1e9
    e2e_value = e2e_frames * e2e_steps * world * kbch / (e2e_ms_max * 1e-3) / 1e9
    peak, peak_src = load_peaks()
    ldpc_launches = args.steps * args.repeat
    ldpc_avg_ms = ldpc_ms_max / max(1, ldpc_launches)
    achieved = args.pool * HBM_BYTES_PER_FRAME / (ldpc_avg_ms * 1e-3) / 1e9
    edge_rate = args.pool / (ldpc_avg_ms * 1e-3) * links * mean_it
    clocks = sampler.summary()
    tr = ncu_traffic_per_frame()
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    line = {
        "metric": "decoded_info_gbit_s", "value": value, "unit": "Gbit/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int8", "data": "synthetic", "config": config,
        "frames_per_s": frames_total / (ms_max * 1e-3), "mean_ldpc_iters": mean_it, "fer": fer,
        "timed_region_s": ms_max * 1e-3,
        "gpu_launches": launches_per_step * args.steps,
        "parity_checked": parity_n, "parity_mismatches": parity_bad,
        "kernel_ms_per_step": {"ldpc_v2_kernel": ldpc_ms / args.steps, "bch_kernel": bch_ms / args.steps},
        "e2e": {"value": e2e_value, "unit": "Gbit/s", "h2d_bytes_per_step": e2e_frames * N,
                "d2h_bytes_per_step": e2e_frames * (kbch // 8 + 16), "frames_per_step": e2e_frames, "steps": e2e_steps,
                "api": "dvbs2fec_decode_batch (pinned host buffers)",
                "host_ceiling": {"what": "the same input bytes copied host->device and nothing else, all ranks at once, max over ranks",
                                 "h2d_gb_s_per_gpu": args.pool * N / (h2d_ms_max * 1e-3) / 1e9,
                                 "h2d_gb_s_total": world * args.pool * N / (h2d_ms_max * 1e-3) / 1e9,
                                 "gbit_s_if_decoding_were_free": world * args.pool * kbch / (h2d_ms_max * 1e-3) / 1e9}},
        "roofline": {"kernel": "ldpc_v2_kernel", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": (tr[0] * args.pool / 1e9) if tr else None,
                     "traffic_unit": "GB per launch (ncu dram__bytes_read+write, %s)" % (tr[1] if tr else "n/a"), "peak_source": peak_src,
                     "algorithmic_bytes_per_frame": HBM_BYTES_PER_FRAME, "frames_per_launch": args.pool,
                     "edge_updates_per_s": edge_rate,
                     "note": "HBM is not the binding roof of this kernel (SURVEY 8d); the binding ones are on chip, see onchip",
                     "onchip": onchip_roofline(edge_rate, clocks.get("sm_mhz"), sms)},
        "latency_ms_per_batch": latency,
        "clocks": clocks,
    }
    if dispatcher is not None:
        line["dispatcher"] = dispatcher
    if not args.no_cpu and world == 1:   # the CPU reference is timed beside the N=1 run only
        procs = os.cpu_count() or 1
        pool_host = make_pool_numpy(codes, 16 * min(procs, 64), args.esn0, 2)
        cb = cpu_baseline(pool_host, args.cpu_seconds, procs)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        line["cpu_baseline"]["host"] = cpu_model()
        if cb["kind"] == "reference":   # SURVEY 8(d): the other ways of driving the reference, short samples
            variants = {}
            for name, mode, pr in (("simd16_1_thread", "simd16", 1), ("lane0_per_frame_1_thread", "lane0", 1),
                                   ("lane0_per_frame_all_cores", "lane0", procs), ("as_shipped_1_thread", "shipped", 1)):
                v = cpu_baseline(pool_host, 2.0, pr, mode)
                variants[name] = {"gbit_s": v["value"], "frames_per_s": v["frames_per_s"], "cores": pr, "decoded_ok": v["decoded_ok"],
                                  "frames": v["frames"], "sample": v["sample"]}
            line["cpu_baseline"]["variants"] = variants
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 1 if parity_bad else 0


def dispatcher_leg(pkg, L, ndev, h_in, nframes, N, kbch, bb_single, res_single, single_fps):
    """One handle, all devices: dvbs2fec_decode_batch on the same pinned input the single-device run decoded, and a
    stretch of the frame queue (submit_llr / collect).  Output bytes must equal the single-device result."""
    kb = kbch // 8
    # every device gets as many frames per call as the single-device run had (up to four times the pool: page-locked memory)
    rep = min(ndev, 4)
    nbig = nframes * rep
    h_big = L.dvbs2fec_alloc_pinned(nbig * N)
    for r in range(rep):
        C.memmove(h_big + r * nframes * N, h_in, nframes * N)
    dec = pkg.DVBS2Decoder(devices=list(range(ndev)), max_batch=max(256, min(8192, nbig // (2 * ndev))), max_trials=MAX_TRIALS)
    dec.setDemodParams(MODCOD, SHORT, False, MAX_TRIALS)
    h_bb = L.dvbs2fec_alloc_pinned(nbig * kb)
    h_res = L.dvbs2fec_alloc_pinned(nbig * 16)
    for _ in range(2):
        dec.decode_batch_raw(h_big, nbig, h_bb, h_res)
    reps = 4
    t0 = time.perf_counter()
    for _ in range(reps):
        dec.decode_batch_raw(h_big, nbig, h_bb, h_res)
    dt = time.perf_counter() - t0
    bb = np.ctypeslib.as_array(C.cast(h_bb, C.POINTER(C.c_uint8)), shape=(nbig, kb))
    rs = np.ctypeslib.as_array(C.cast(h_res, C.POINTER(C.c_uint8)), shape=(nbig, 16))
    equal = all(bool(np.array_equal(bb[r * nframes:(r + 1) * nframes], bb_single)) and
                bool(np.array_equal(rs[r * nframes:(r + 1) * nframes, 8:], res_single[:, 8:])) for r in range(rep))   # (tags differ by design)
    nframes_call = nbig
    fps = nframes_call * reps / dt
    # frame queue: in-order delivery over all devices
    nq = min(2048, nframes)
    src = np.ctypeslib.as_array(C.cast(h_in, C.POINTER(C.c_int8)), shape=(nframes, N))
    got_bb, got = [], 0
    t0 = time.perf_counter()
    for k in range(nq):
        while True:
            try:
                dec.submit_llr(src[k], k)
                break
            except pkg.DVBS2FecError as e:
                if e.code != pkg.EAGAIN:
                    raise
                b, r = dec.collect(4096, 1000)
                got_bb.append(b)
                got += len(b)
    dec.flush()
    while got < nq:
        b, r = dec.collect(4096, 100000)
        got_bb.append(b)
        got += len(b)
    qdt = time.perf_counter() - t0
    qbb = np.concatenate(got_bb) if got_bb else np.zeros((0, kb), np.uint8)
    q_equal = bool(np.array_equal(qbb[:nq], bb_single[:nq]))
    dec.close()
    L.dvbs2fec_free_pinned(h_bb)
    L.dvbs2fec_free_pinned(h_res)
    L.dvbs2fec_free_pinned(h_big)
    return {"devices": ndev, "frames_per_call": nframes_call, "api": "one handle, cfg.devices[0..N-1], dvbs2fec_decode_batch from pinned host memory",
            "frames_per_s": fps, "gbit_s": fps * kbch / 1e9, "single_device_e2e_frames_per_s": single_fps,
            "efficiency": fps / (ndev * single_fps), "bytes_equal_single_device": equal,
            "queue_frames_checked": nq, "queue_bytes_equal": q_equal, "queue_python_submit_frames_per_s": nq / qdt}


if __name__ == "__main__":
    sys.exit(main())
