"""Ragged Sinkhorn batches on one GPU: one psd_sinkhorn_divergence_weighted launch with per-pair lengths, next to a per-sample
loop of psd_sinkhorn_divergence and to one launch over clouds padded to the largest size with zero-weight points.

    python tools/sinkhorn_ragged_bench.py --out profiles/sinkhorn_ragged_b200.json

B = 32 seeded U[0,1)^3 scans with sizes drawn uniformly from [128, 2048] against 1024-point predictions, blur / scaling
0.05 / 0.5, forward with both gradients.  Each time is the median of --reps CUDA-event timings on one stream after one warm-up
run; the loop's time includes its 32 launches from the host, as a training loop would pay them.  The padded variant pads each
scan with copies of its first point at weight 0 (the diameter is unchanged) and gives the others weight 1 / length.  The
imbalance rows time the largest pair alone and all 32 pairs at the largest size: one launch lasts at least as long as its
largest pair.  The working set (a few MB) lives in L2 after the first pass, as it does in a training loop."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def smi(fields):
    try:
        q = subprocess.run(["nvidia-smi", f"--query-gpu={fields}", "--format=csv,noheader,nounits"], capture_output=True,
                           text=True, timeout=30)
        return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON here as well as to stdout")
    ap.add_argument("--b", type=int, default=32)
    ap.add_argument("--n", type=int, default=1024, help="prediction size")
    ap.add_argument("--lo", type=int, default=128)
    ap.add_argument("--hi", type=int, default=2048)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--seeds", type=int, default=3, help="draws of the scan sizes")
    args = ap.parse_args()

    import torch
    import psd_b200
    if not torch.cuda.is_available():
        raise SystemExit("sinkhorn_ragged_bench.py measures on a CUDA device; none is visible")
    pkg = psd_b200.load()
    lib = pkg._lib.lib
    vp = pkg._lib.ptr
    dev = torch.device("cuda:0")
    stream = torch.cuda.current_stream(dev)
    sp = ctypes.c_void_p(stream.cuda_stream)
    blur, scaling = 0.05, 0.5

    def timed(fn, reps):
        fn()
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        return float(np.median(ts))

    b, n = args.b, args.n
    result = {"gpu": {"name": torch.cuda.get_device_name(0),
                      "name_power_limit_W_max_sm_clock_MHz": smi("name,power.limit,clocks.max.sm")},
              "b": b, "n_prediction": n, "scan_sizes": [args.lo, args.hi], "blur": blur, "scaling": scaling,
              "reps": args.reps, "clouds": "uniform U[0,1)^3, numpy default_rng(seed)", "runs": []}
    for seed in range(args.seeds):
        rng = np.random.default_rng(seed)
        lens = rng.integers(args.lo, args.hi + 1, b).astype(np.int32)
        M = int(lens.max())
        x = torch.from_numpy(rng.random((b, n, 3), dtype=np.float32)).to(dev)
        scans = [rng.random((k, 3), dtype=np.float32) for k in lens]
        yr = np.zeros((b, M, 3), np.float32)
        yp = np.zeros((b, M, 3), np.float32)
        wp = np.zeros((b, M), np.float32)
        for c, s in enumerate(scans):
            yr[c, :len(s)] = s
            yp[c, :len(s)], yp[c, len(s):] = s, s[0]
            wp[c, :len(s)] = np.float32(1) / np.float32(len(s))
        yr, yp, wp = (torch.from_numpy(v).to(dev) for v in (yr, yp, wp))
        yl = torch.from_numpy(lens).to(dev)
        ys = [torch.from_numpy(s).to(dev)[None] for s in scans]
        loss, gx, gy = torch.empty(b, device=dev), torch.empty(b, n, 3, device=dev), torch.empty(b, M, 3, device=dev)
        l1 = torch.empty(b, device=dev)
        g1x = [torch.empty(1, n, 3, device=dev) for _ in range(b)]
        g1y = [torch.empty(1, int(k), 3, device=dev) for k in lens]
        lp = torch.empty(b, device=dev)

        def ragged():
            assert lib.psd_sinkhorn_divergence_weighted(vp(x), vp(yr), b, n, M, None, vp(yl), None, None, blur, scaling, vp(loss),
                                                        vp(gx), vp(gy), None, None, sp) == 1

        def loop():
            for c in range(b):
                assert lib.psd_sinkhorn_divergence(vp(x[c:c + 1]), vp(ys[c]), 1, n, int(lens[c]), blur, scaling, vp(l1[c:c + 1]),
                                                   vp(g1x[c]), vp(g1y[c]), None, None, sp) == 1

        def padded():
            assert lib.psd_sinkhorn_divergence_weighted(vp(x), vp(yp), b, n, M, None, None, None, vp(wp), blur, scaling, vp(lp),
                                                        vp(gx), vp(gy), None, None, sp) == 1

        big = int(np.argmax(lens))
        xb, ybig = x[big:big + 1].contiguous(), ys[big]
        lb_ = torch.empty(1, device=dev)
        gbx, gby = torch.empty(1, n, 3, device=dev), torch.empty(1, M, 3, device=dev)

        def largest_alone():
            assert lib.psd_sinkhorn_divergence(vp(xb), vp(ybig), 1, n, M, blur, scaling, vp(lb_), vp(gbx), vp(gby), None, None,
                                               sp) == 1
        yfull = torch.from_numpy(np.random.default_rng(100 + seed).random((b, M, 3), dtype=np.float32)).to(dev)

        def all_at_max():
            assert lib.psd_sinkhorn_divergence(vp(x), vp(yfull), b, n, M, blur, scaling, vp(loss), vp(gx), vp(gy), None, None,
                                               sp) == 1
        row = {"seed": seed, "scan_sizes": lens.tolist(), "max_size": M, "mean_size": float(lens.mean())}
        # alternate the three variants so that drift in the clock or in neighbours' load hits each alike
        for _ in range(2):
            row["ragged_one_launch_ms"] = timed(ragged, args.reps)
            row["per_sample_loop_ms"] = timed(loop, args.reps)
            row["zero_weight_padding_ms"] = timed(padded, args.reps)
        row["largest_pair_alone_ms"] = timed(largest_alone, args.reps)
        row["all_pairs_at_max_size_ms"] = timed(all_at_max, args.reps)
        ragged(); loop(); padded()
        torch.cuda.synchronize()
        S_ragged = loss.clone()
        row["loop_vs_ragged_bits_equal"] = bool(torch.equal(S_ragged.view(torch.int32), l1.view(torch.int32)))
        row["padded_vs_ragged_max_rel_diff"] = float(((lp - S_ragged).abs() / S_ragged.abs()).max())
        row["speedup_vs_loop"] = row["per_sample_loop_ms"] / row["ragged_one_launch_ms"]
        row["sm_clock_MHz_after"] = smi("clocks.sm")
        result["runs"].append(row)
        print(json.dumps(row), flush=True)
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
