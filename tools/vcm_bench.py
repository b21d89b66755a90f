#!/usr/bin/env python3
"""VCM / ACM batches against the per-configuration path (GPU), all on device buffers, CUDA events on one stream.

(a) CCM through the VCM call: the bench pool (QPSK 1/2 normal, 16 384 frames, Es/N0 2.2 dB, 1.06 GB > L2) through
    `decode_batch_device` and through `dvbs2fec_decode_vcm_device` with all-equal descriptors, alternated.  The VCM call
    takes its path without reordering here, so the two should cost the same.
(b) An ACM mix from symbols: QPSK 1/2 N, 8PSK 3/5 N, 16APSK 3/4 N and QPSK 1/2 S in round robin, plus 2 % DUMMY
    PLFRAMEs, 16 384 frames (2.6 GB of symbols) through `decode_plframes_vcm_device` at max_batch 16 384, against the
    sum of four `decode_plframes_device` calls (one configured handle each) over the same frames.  Kernel times of
    both from `dvbs2fec_kernel_times` in a separate pass.

    python tools/vcm_bench.py [--frames 16384] [--repeat 7] [--warmup 2] [--out FILE]

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

MIX = ((4, 0, 0, 2.0), (12, 0, 0, 6.5), (19, 0, 0, 11.2), (4, 1, 0, 2.5))   # modcod, short, pilots, Es/N0 dB
DUMMY_EVERY = 50


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, plim, sm, smax = [s.strip() for s in r.stdout.strip().splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": plim, "sm_clock": sm, "sm_clock_max": smax}
    except Exception as e:   # the numbers stand without it, but say so
        return {"gpu": "unknown (%s)" % type(e).__name__}


def timed(torch, stream, fn, warmup, repeat):
    """median ms of fn() over repeat runs, each bracketed by events on stream, after warmup runs"""
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(repeat):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), ts


def kernel_times(dec, fn):
    import torch
    torch.cuda.synchronize()
    dec.set_profiling(True)
    dec.kernel_times()
    fn()
    t = dec.kernel_times()
    dec.set_profiling(False)
    return {"demap_ms": round(t[0], 3), "ldpc_ms": round(t[1], 3), "bch_ms": round(t[2], 3), "launches": t[3]}


def ccm_through_vcm(torch, pkg, bench, args, stream):
    dev = torch.device("cuda", 0)
    n = args.frames
    info = pkg.modcod_info(bench.MODCOD, bench.SHORT)
    codes = bench.make_codewords(pkg, 64, 1)
    pool = bench.make_pool_torch(torch, codes, n, 2.2, 100, dev)
    dec = pkg.DVBS2Decoder(devices=[0], max_batch=n, max_trials=bench.MAX_TRIALS)
    dec.setDemodParams(bench.MODCOD, bench.SHORT, False, bench.MAX_TRIALS)
    desc = np.tile(np.array([[bench.MODCOD, int(bench.SHORT), 0, 0]], np.int32), (n, 1))
    bb = [torch.empty(n * (info["kbch"] // 8), dtype=torch.uint8, device=dev) for _ in range(2)]
    res = [torch.empty((n, 16), dtype=torch.uint8, device=dev) for _ in range(2)]

    def ccm():
        dec.decode_batch_device(pool.data_ptr(), n, bb[0].data_ptr(), res[0].data_ptr(), stream.cuda_stream)

    def vcm():
        dec.decode_vcm_device(desc, pool.data_ptr(), bb[1].data_ptr(), res[1].data_ptr(), stream.cuda_stream)

    t = {"ccm": [], "vcm": []}
    for f in (ccm, vcm):
        timed(torch, stream, f, args.warmup, 1)
    for _ in range(args.repeat):   # alternated, so that drift on the shared host hits both alike
        t["ccm"].append(timed(torch, stream, ccm, 0, 1)[0])
        t["vcm"].append(timed(torch, stream, vcm, 0, 1)[0])
    same = torch.equal(bb[0], bb[1]) and torch.equal(res[0], res[1])
    out = {"frames": n, "decode_batch_device_ms": round(float(np.median(t["ccm"])), 3),
           "decode_vcm_device_ms": round(float(np.median(t["vcm"])), 3), "runs_ms": {k: [round(x, 3) for x in v] for k, v in t.items()},
           "outputs_equal": bool(same), "vcm_launches": None}
    out["ratio"] = round(out["decode_vcm_device_ms"] / out["decode_batch_device_ms"], 4)
    vcm()
    torch.cuda.synchronize()
    out["vcm_launches"] = dec.last_launch_count()
    dec.close()
    return out


def acm_mix(torch, pkg, args, stream):
    dev = torch.device("cuda", 0)
    n = args.frames
    rng = np.random.default_rng(4)
    kinds = []
    k = 0
    for i in range(n):
        if i % DUMMY_EVERY == DUMMY_EVERY - 1:
            kinds.append(-1)
        else:
            kinds.append(k % len(MIX))
            k += 1
    kinds = np.array(kinds)
    desc = np.array([(0, 0, 0, 0) if c < 0 else MIX[c][:3] + (0,) for c in kinds], np.int32)
    sym_off, _, bb_off = pkg.vcm_layout(desc)
    packed = torch.full((2 * int(sym_off[-1]),), float("nan"), dtype=torch.float32, device=dev)
    per_cfg, decs = [], []
    for c, (modcod, short, pilots, esn0) in enumerate(MIX):
        info = pkg.modcod_info(modcod, short, pilots)
        kb = info["kbch"] // 8
        tx = np.stack([pkg.modulate(modcod, short, pilots, pkg.encode_fecframe(modcod, short, rng.integers(0, 256, kb, dtype=np.uint8)))
                       for _ in range(16)])
        es = float(np.mean(np.abs(tx[tx != 0]) ** 2))
        sigma = float(np.sqrt(es / (2 * 10 ** (esn0 / 10))))
        idx = np.flatnonzero(kinds == c)
        g = torch.Generator(device=dev)
        g.manual_seed(100 + c)
        clean = torch.from_numpy(tx.view(np.float32)).to(dev)
        frames = clean[torch.arange(len(idx), device=dev) % 16]
        frames += torch.randn(frames.shape, generator=g, device=dev) * sigma
        for j, i in enumerate(idx):
            packed[2 * sym_off[i]:2 * sym_off[i + 1]] = frames[j]
        d = pkg.DVBS2Decoder(devices=[0], max_batch=n, max_trials=25)
        d.setDemodParams(modcod, bool(short), bool(pilots), 25)
        bb = torch.empty(len(idx) * kb, dtype=torch.uint8, device=dev)
        res = torch.empty((len(idx), 16), dtype=torch.uint8, device=dev)
        per_cfg.append((frames, bb, res, idx, kb))
        decs.append(d)
    vdec = pkg.DVBS2Decoder(devices=[0], max_batch=n, max_trials=25)
    v_bb = torch.empty(int(bb_off[-1]), dtype=torch.uint8, device=dev)
    v_res = torch.empty((n, 16), dtype=torch.uint8, device=dev)

    def ccm():
        for d, (frames, bb, res, idx, _) in zip(decs, per_cfg):
            d.decode_plframes_device(frames.data_ptr(), len(idx), bb.data_ptr(), res.data_ptr(), stream.cuda_stream)

    def vcm():
        vdec.decode_plframes_vcm_device(desc, packed.data_ptr(), v_bb.data_ptr(), v_res.data_ptr(), stream.cuda_stream)

    t = {"ccm_sum": [], "vcm": []}
    for f in (ccm, vcm):
        timed(torch, stream, f, args.warmup, 1)
    for _ in range(args.repeat):
        t["ccm_sum"].append(timed(torch, stream, ccm, 0, 1)[0])
        t["vcm"].append(timed(torch, stream, vcm, 0, 1)[0])
    torch.cuda.synchronize()
    # same results frame for frame
    vres = v_res.cpu().numpy().view(np.uint8).reshape(n, 16)
    vbb = v_bb.cpu().numpy()
    same = True
    for frames, bb, res, idx, kb in per_cfg:
        r = res.cpu().numpy()
        same &= bool(np.array_equal(vres[idx, 8:], r[:, 8:]))
        b = bb.cpu().numpy().reshape(len(idx), kb)
        same &= all(np.array_equal(vbb[bb_off[i]:bb_off[i + 1]], b[j]) for j, i in enumerate(idx[:: max(1, len(idx) // 64)]))
    kt_v = kernel_times(vdec, vcm)
    kt_c = [kernel_times(d, lambda d=d, p=p: d.decode_plframes_device(p[0].data_ptr(), len(p[3]), p[1].data_ptr(), p[2].data_ptr(),
                                                                        stream.cuda_stream)) for d, p in zip(decs, per_cfg)]
    vcm()
    torch.cuda.synchronize()
    out = {"frames": n, "mix": [list(m) for m in MIX], "dummy_every": DUMMY_EVERY, "symbol_bytes": int(sym_off[-1]) * 8,
           "ccm_sum_ms": round(float(np.median(t["ccm_sum"])), 3), "vcm_ms": round(float(np.median(t["vcm"])), 3),
           "runs_ms": {k: [round(x, 3) for x in v] for k, v in t.items()}, "outputs_equal": same,
           "vcm_launches": vdec.last_launch_count(), "vcm_kernel_times": kt_v,
           "ccm_kernel_times": {"demap_ms": round(sum(k["demap_ms"] for k in kt_c), 3), "ldpc_ms": round(sum(k["ldpc_ms"] for k in kt_c), 3),
                                "bch_ms": round(sum(k["bch_ms"] for k in kt_c), 3), "launches": sum(k["launches"] for k in kt_c)}}
    out["ratio"] = round(out["vcm_ms"] / out["ccm_sum_ms"], 4)
    for d in decs + [vdec]:
        d.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--frames", type=int, default=16384)
    ap.add_argument("--repeat", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("vcm_bench.py needs a CUDA device")
    bench = importlib.import_module("bench")
    pkg = importlib.import_module("sdrpp-dvbs-demodulator_b200")
    stream = torch.cuda.current_stream()
    out = dict(gpu_info())
    out["a_ccm_through_vcm"] = ccm_through_vcm(torch, pkg, bench, args, stream)
    print(json.dumps(out["a_ccm_through_vcm"]), file=sys.stderr, flush=True)
    out["b_acm_mix"] = acm_mix(torch, pkg, args, stream)
    out.update({k + "_after": v for k, v in gpu_info().items() if k != "gpu"})
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
