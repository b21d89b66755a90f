#!/usr/bin/env python3
"""Fixed cost per frame pair of the LDPC kernel (GPU): QPSK 1/2 normal at five Es/N0 points, timed through
decode_batch_device on the bench generator, then a straight-line fit

    ldpc ms/step = a + b * mean_iters

over the points.  `a` is what a step pays besides the passes proper (loading a pair, the first screens and full
tests, the read-out, the per-launch drain); `b` is the cost of one more pass over the step's frames.  The residual
at 2.2 dB (the bench point) is the cost of the iteration spread inside a pair and a launch.  It also prints the
time of one launch of 4096 and of 16 384 frames: their difference leaves the fixed part of a launch.

    python tools/ldpc_fixed_cost.py [--pool 16384] [--repeat 5] [--steps 4] [--warmup 2] [--out FILE]
    python tools/ldpc_fixed_cost.py --stub      # the fit on made-up points, no device needed

One JSON object on stdout (and in --out), with the GPU's name, power limit and SM clock read in the same run."""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ESN0 = (10.0, 3.1, 2.2, 1.5, 0.4)
BENCH_POINT = 2.2


def fit(points):
    """least-squares line ldpc_ms = a + b * iters over the points; residual of the bench point"""
    x = np.array([p["mean_iters"] for p in points], np.float64)
    y = np.array([p["ldpc_ms_per_step"] for p in points], np.float64)
    b, a = np.polyfit(x, y, 1)
    out = {"a_ms": round(float(a), 3), "b_ms_per_iter": round(float(b), 4)}
    for p in points:
        if abs(p["esn0_db"] - BENCH_POINT) < 1e-9:
            line = a + b * p["mean_iters"]
            out["residual_ms_at_2.2dB"] = round(p["ldpc_ms_per_step"] - line, 3)
            out["fixed_share_at_2.2dB"] = round(float(a) / p["ldpc_ms_per_step"], 4)
    return out


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, plim, sm, smax = [s.strip() for s in r.stdout.strip().splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": plim, "sm_clock": sm, "sm_clock_max": smax}
    except Exception as e:   # the numbers stand without it, but say so
        return {"gpu": "unknown (%s)" % type(e).__name__}


def measure(args):
    import torch
    bench = importlib.import_module("bench")
    pkg = importlib.import_module("sdrpp-dvbs-demodulator_b200")
    if not torch.cuda.is_available():
        raise SystemExit("ldpc_fixed_cost.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    info = pkg.modcod_info(bench.MODCOD, bench.SHORT)
    dec = pkg.DVBS2Decoder(devices=[0], max_batch=args.pool, max_trials=bench.MAX_TRIALS)
    dec.setDemodParams(bench.MODCOD, bench.SHORT, False, bench.MAX_TRIALS)
    codes = bench.make_codewords(pkg, 64, 1)
    d_bb = torch.empty((args.pool, info["kbch"] // 8), dtype=torch.uint8, device=dev)
    d_res = torch.empty((args.pool, 16), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()

    def launch(pool, n):
        dec.decode_batch_device(pool.data_ptr(), n, d_bb.data_ptr(), d_res.data_ptr(), stream.cuda_stream)

    points, latency = [], {}
    for esn0 in ESN0:
        pool = bench.make_pool_torch(torch, codes, args.pool, esn0, 100, dev)   # the bench's pool at this Es/N0
        for _ in range(args.warmup * args.repeat):
            launch(pool, args.pool)
        torch.cuda.synchronize()
        dec.set_profiling(True)
        dec.kernel_times()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps * args.repeat):
            launch(pool, args.pool)
        e1.record(stream)
        torch.cuda.synchronize()
        _, ldpc_ms, _, _ = dec.kernel_times()
        dec.set_profiling(False)
        res = d_res.cpu().numpy().view(pkg.RESULT_DTYPE).reshape(-1)
        it = res["ldpc_iters"].astype(np.int32)
        points.append({"esn0_db": esn0, "mean_iters": round(float(np.where(it < 0, bench.MAX_TRIALS, it).mean()), 4),
                       "step_ms": round(e0.elapsed_time(e1) / args.steps, 3), "ldpc_ms_per_step": round(ldpc_ms / args.steps, 3)})
        print(json.dumps(points[-1]), file=sys.stderr, flush=True)
        if abs(esn0 - BENCH_POINT) < 1e-9:   # one launch of n frames, median of 7, at the bench point
            for n in (4096, args.pool):
                ts = []
                for _ in range(7):
                    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a0.record(stream)
                    launch(pool, n)
                    a1.record(stream)
                    torch.cuda.synchronize()
                    ts.append(a0.elapsed_time(a1))
                latency[str(n)] = round(sorted(ts)[3], 4)
        del pool
    dec.close()
    return points, latency


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--pool", type=int, default=16384, help="frames per launch")
    ap.add_argument("--repeat", type=int, default=5, help="launches per step")
    ap.add_argument("--steps", type=int, default=4, help="timed steps per Es/N0 point")
    ap.add_argument("--warmup", type=int, default=2, help="untimed steps per Es/N0 point")
    ap.add_argument("--out", help="also write the JSON here")
    ap.add_argument("--stub", action="store_true", help="fit made-up points (no device): checks the script")
    args = ap.parse_args()
    if args.stub:
        iters = {10.0: 1.01, 3.1: 6.2, 2.2: 7.4, 1.5: 12.0, 0.4: 25.0}
        points = [{"esn0_db": e, "mean_iters": it, "step_ms": 0.0, "ldpc_ms_per_step": 19.5 + 11.17 * it + (13.6 if e == 2.2 else 0.0)}
                  for e, it in iters.items()]
        latency, gpu = {"4096": 0.0, str(args.pool): 0.0}, {"gpu": "stub"}
    else:
        gpu = gpu_info()
        points, latency = measure(args)
    out = {"what": "LDPC ms/step = a + b * mean_iters, QPSK 1/2 normal, bench generator",
           "frames_per_step": args.pool * args.repeat, "steps": args.steps, **gpu,
           "fit": fit(points), "points": points, "latency_ms_per_launch": latency}
    if len(latency) == 2 and args.pool > 4096:
        t4, tp = latency["4096"], latency[str(args.pool)]
        out["launch_fixed_ms"] = round(t4 - (tp - t4) * 4096 / (args.pool - 4096), 4)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
