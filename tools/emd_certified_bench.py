"""Certified EMD on one GPU: time of a whole psd_emd_certified call, of each epsilon-scaling phase, of the certificate alone,
and the gap it proves, next to emdModule at the evaluation (eps 0.005, 50 iterations), training (0.05, 3000) and MSN-test
(0.002, 10000) settings on the same clouds.

    python tools/emd_certified_bench.py --out profiles/emd_certified_b200.json

Seeded U[0,1)^3 clouds, B = 32, n = 1024 and 2048, eps_end 1e-3 / 1e-4 / 1e-5 (eps_start 0.05, scale 4).  Times are CUDA
events around work on one stream, the median of --reps runs after one warm-up run.  The working set (under 2 MB) lives in
L2 after the first pass, as it does in an evaluation loop.  A phase that finds every point assigned still pays its launch,
the state load and the write-back: "empty_phase_ms" measures that fixed cost of one phase."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

EPS_START, SCALE, MAX_ITERS = 0.05, 4.0, 20000


def phase_eps(eps_end):
    e, end = float(np.float32(EPS_START)), float(np.float32(eps_end))
    out = []
    while e > end:
        out.append(float(np.float32(e)))
        e /= SCALE
    return out + [float(np.float32(end))]


def gpu_info(torch):
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.SubprocessError):
        info["nvidia_smi"] = None
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON here as well as to stdout")
    ap.add_argument("--b", type=int, default=32)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()

    import torch
    import psd_b200
    if not torch.cuda.is_available():
        raise SystemExit("emd_certified_bench.py measures on a CUDA device; none is visible")
    pkg = psd_b200.load()
    L = pkg._lib
    lib = L.lib
    dev = torch.device("cuda:0")
    vp = L.ptr
    stream = torch.cuda.current_stream(dev)
    sp = ctypes.c_void_p(stream.cuda_stream)

    def timed(fn, reps):
        fn()   # warm-up
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        return float(np.median(ts)), float(np.min(ts))

    b = args.b
    rng = np.random.default_rng(2024)
    result = {"gpu": gpu_info(torch), "b": b, "eps_start": EPS_START, "scale": SCALE, "max_iters_per_phase": MAX_ITERS,
              "reps": args.reps, "clouds": "uniform U[0,1)^3, numpy default_rng(2024)", "certified": [], "emdModule": []}
    for n in (1024, 2048):
        x = torch.from_numpy(rng.random((b, n, 3), dtype=np.float32)).to(dev)
        y = torch.from_numpy(rng.random((b, n, 3), dtype=np.float32)).to(dev)
        dist, price = torch.empty(b, n, device=dev), torch.empty(b, n, device=dev)
        ass = torch.empty(b, n, device=dev, dtype=torch.int32)
        bounds, status = torch.empty(b, 2, device=dev, dtype=torch.float64), torch.empty(b, device=dev, dtype=torch.int32)
        mid_1e5 = None
        for eps_end in (1e-3, 1e-4, 1e-5):
            def call():
                rc = lib.psd_emd_certified(vp(x), vp(y), b, n, EPS_START, eps_end, SCALE, MAX_ITERS, vp(dist), vp(ass), vp(price),
                                           vp(bounds), vp(status), sp)
                assert rc == 1, L.last_error()
            whole_med, whole_min = timed(call, args.reps)
            bd, st = bounds.cpu().numpy(), status.cpu().numpy()
            gap = bd[:, 1] - bd[:, 0]
            if eps_end == 1e-5:
                mid_1e5 = bd.mean(1)

            def cert():
                assert lib.psd_emd_dual_bound(vp(x), vp(y), b, n, vp(ass), vp(price), vp(bounds), vp(status), sp) == 1
            cert_med, _ = timed(cert, max(args.reps, 10))

            # the same phases one by one (psd_emd_forward_cluster with the automatic cluster size = what a phase launches)
            sched = phase_eps(eps_end)
            per_phase = [[] for _ in sched]
            for _ in range(args.reps):
                price.zero_()
                for i, e in enumerate(sched):
                    ass.fill_(-1)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    assert lib.psd_emd_forward_cluster(vp(x), vp(y), b, n, vp(dist), vp(ass), vp(price), None, e, MAX_ITERS, 0, sp) == 1
                    e1.record(stream)
                    e1.synchronize()
                    per_phase[i].append(e0.elapsed_time(e1))

            # fixed cost of a phase: the last phase again on its own complete assignment (no bidder in iteration 0)
            def empty_phase():
                assert lib.psd_emd_forward_cluster(vp(x), vp(y), b, n, vp(dist), vp(ass), vp(price), None, sched[-1], MAX_ITERS, 0, sp) == 1
            empty_med, _ = timed(empty_phase, max(args.reps, 10))
            result["certified"].append({
                "n": n, "eps_end": eps_end, "phases": len(sched), "phase_eps": sched,
                "whole_call_ms_median": whole_med, "whole_call_ms_min": whole_min,
                "phase_ms_median": [float(np.median(t)) for t in per_phase],
                "certificate_ms_median": cert_med, "empty_phase_ms_median": empty_med,
                "clouds_with_matching": int((st == 1).sum()),
                "gap_per_point_mean": float(gap.mean()), "gap_per_point_max": float(gap.max()),
                "lower_mean": float(bd[:, 0].mean()), "upper_mean": float(bd[:, 1].mean()),
            })
            print(json.dumps(result["certified"][-1]), flush=True)
        m = pkg.emdModule()
        for name, eps, iters in (("evaluation", 0.005, 50), ("training", 0.05, 3000), ("msn_test", 0.002, 10000)):
            out = {}

            def run():
                out["d"], out["a"] = m(x, y, eps, iters)
            med, mn = timed(run, args.reps)
            a = out["a"].cpu().numpy()
            perms = sum(int(np.array_equal(np.sort(r), np.arange(n))) for r in a)
            val = torch.sqrt(out["d"].double()).mean(1).cpu().numpy()
            result["emdModule"].append({
                "n": n, "setting": name, "eps": eps, "iters": iters, "ms_median": med, "ms_min": mn,
                "clouds_with_matching": perms,
                # deviation of the returned per-point EMD from the certified value (midpoint of the eps_end = 1e-5 bounds)
                "rel_dev_from_certified_mean": float(((val - mid_1e5) / mid_1e5).mean()),
                "rel_dev_from_certified_min": float(((val - mid_1e5) / mid_1e5).min()),
                "rel_dev_from_certified_max": float(((val - mid_1e5) / mid_1e5).max()),
            })
            print(json.dumps(result["emdModule"][-1]), flush=True)
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
