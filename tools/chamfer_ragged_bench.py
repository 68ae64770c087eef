"""Ragged Chamfer batches on one GPU: one psd_chamfer_forward_ragged launch with per-pair lengths, next to a per-sample loop of
standalone calls, to a uniform launch over clouds padded with a far-away sentinel, and to the uniform batch at the largest size.

    python tools/chamfer_ragged_bench.py --out profiles/chamfer_ragged_b200.json

The workload is that of tools/sinkhorn_ragged_bench.py, so that the two can be compared: B = 32 seeded U[0,1)^3 scans with sizes
drawn uniformly from [128, 2048] against 1024-point predictions, three draws.  Every row times the forward with both gradients:
the forward zero-fills the gradient buffers and the backward accumulates into them (psd_chamfer_forward_zero / _ragged, then
psd_chamfer_backward_ex / _ragged), with a random upstream gradient.  Each time is the median of --reps CUDA-event timings on one
stream after one warm-up run; the loop's time includes its 32 x 2 launches from the host, as a training loop would pay them.
The sentinel row pads every scan to the largest size with points at 1e6 (real rows keep their bits) and masks the upstream
gradient of the padding; its exact-scan fallback count is read from psd_chamfer_stats.  The working set (a few MB) lives in L2
after the first pass, as it does in a training loop."""
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
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--seeds", type=int, default=3, help="draws of the scan sizes")
    ap.add_argument("--sentinel", type=float, default=1e6)
    args = ap.parse_args()

    import torch
    import psd_b200
    if not torch.cuda.is_available():
        raise SystemExit("chamfer_ragged_bench.py measures on a CUDA device; none is visible")
    pkg = psd_b200.load()
    lib = pkg._lib.lib
    vp = pkg._lib.ptr
    dev = torch.device("cuda:0")
    stream = torch.cuda.current_stream(dev)
    sp = ctypes.c_void_p(stream.cuda_stream)

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

    def fallbacks(reset=1):
        out = np.zeros(2, np.int64)
        assert lib.psd_chamfer_stats(out.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)), reset) == 1
        return int(out[1])

    class Buffers:   # outputs and zero-filled gradients of one [b, n] x [b, m] call
        def __init__(self, b, n, m):
            self.d1, self.d2 = torch.empty(b, n, device=dev), torch.empty(b, m, device=dev)
            self.i1 = torch.empty(b, n, device=dev, dtype=torch.int32)
            self.i2 = torch.empty(b, m, device=dev, dtype=torch.int32)
            self.g = torch.empty(3 * b * (n + m), device=dev)
            self.g1, self.g2 = self.g[:3 * b * n], self.g[3 * b * n:]

    def uniform_step(x, y, gd1, gd2, o):
        b, n, m = x.shape[0], x.shape[1], y.shape[1]
        assert lib.psd_chamfer_forward_zero(vp(x), vp(y), b, n, m, 0, vp(o.d1), vp(o.d2), vp(o.i1), vp(o.i2), None, 0.0, None,
                                            vp(o.g), o.g.numel(), sp) == 1
        assert lib.psd_chamfer_backward_ex(vp(x), vp(y), vp(o.g1), vp(o.g2), vp(gd1), vp(gd2), vp(o.i1), vp(o.i2), b, n, m, 0,
                                           0, sp) == 1

    b, n = args.b, args.n
    result = {"gpu": {"name": torch.cuda.get_device_name(0),
                      "name_power_limit_W_max_sm_clock_MHz": smi("name,power.limit,clocks.max.sm")},
              "b": b, "n_prediction": n, "scan_sizes": [args.lo, args.hi], "reps": args.reps, "sentinel": args.sentinel,
              "timed": "forward (zero-filling the gradients) + backward to both clouds, median of CUDA-event timings",
              "clouds": "uniform U[0,1)^3, numpy default_rng(seed)", "runs": []}
    for seed in range(args.seeds):
        rng = np.random.default_rng(seed)
        lens = rng.integers(args.lo, args.hi + 1, b).astype(np.int32)
        M = int(lens.max())
        xh = rng.random((b, n, 3), dtype=np.float32)
        scans = [rng.random((k, 3), dtype=np.float32) for k in lens]
        yr = np.zeros((b, M, 3), np.float32)
        ys_np = np.full((b, M, 3), np.float32(args.sentinel), np.float32)
        for c, s in enumerate(scans):
            yr[c, :len(s)] = s
            ys_np[c, :len(s)] = s
        x = torch.from_numpy(xh).to(dev)
        yr_t, ysent = torch.from_numpy(yr).to(dev), torch.from_numpy(ys_np).to(dev)
        yl = torch.from_numpy(lens).to(dev)
        gd1 = torch.from_numpy(rng.random((b, n), dtype=np.float32)).to(dev)
        gd2 = torch.from_numpy(rng.random((b, M), dtype=np.float32)).to(dev)
        mask = (torch.arange(M, device=dev)[None, :] < yl[:, None]).float()
        gd2m = gd2 * mask
        ys = [torch.from_numpy(s).to(dev)[None] for s in scans]
        gd2s = [gd2[c:c + 1, :int(k)].contiguous() for c, k in enumerate(lens)]
        o_r, o_s, o_u = Buffers(b, n, M), Buffers(b, n, M), Buffers(b, n, M)
        o_l = [Buffers(1, n, int(k)) for k in lens]
        yfull = torch.from_numpy(np.random.default_rng(100 + seed).random((b, M, 3), dtype=np.float32)).to(dev)

        def ragged():
            assert lib.psd_chamfer_forward_ragged(vp(x), vp(yr_t), b, n, M, 0, None, vp(yl), vp(o_r.d1), vp(o_r.d2), vp(o_r.i1),
                                                  vp(o_r.i2), None, 0.0, None, vp(o_r.g), o_r.g.numel(), sp) == 1
            assert lib.psd_chamfer_backward_ragged(vp(x), vp(yr_t), vp(o_r.g1), vp(o_r.g2), vp(gd1), vp(gd2), vp(o_r.i1),
                                                   vp(o_r.i2), None, vp(yl), b, n, M, 0, sp) == 1

        def loop():
            for c in range(b):
                uniform_step(x[c:c + 1], ys[c], gd1[c:c + 1], gd2s[c], o_l[c])

        def sentinel():
            uniform_step(x, ysent, gd1, gd2m, o_s)

        def all_at_max():
            uniform_step(x, yfull, gd1, gd2, o_u)

        row = {"seed": seed, "scan_sizes": lens.tolist(), "max_size": M, "mean_size": float(lens.mean())}
        # alternate the variants so that drift in the clock or in neighbours' load hits each alike
        for _ in range(2):
            row["ragged_one_launch_ms"] = timed(ragged, args.reps)
            row["per_sample_loop_ms"] = timed(loop, args.reps)
            row["far_sentinel_padding_ms"] = timed(sentinel, args.reps)
            row["uniform_all_at_max_size_ms"] = timed(all_at_max, args.reps)
        torch.cuda.synchronize()
        fallbacks()
        ragged()
        torch.cuda.synchronize()
        row["ragged_fallback_queries"] = fallbacks()
        loop()
        torch.cuda.synchronize()
        row["per_sample_loop_fallback_queries"] = fallbacks()
        sentinel()
        torch.cuda.synchronize()
        row["far_sentinel_fallback_queries"] = fallbacks()
        all_at_max()
        torch.cuda.synchronize()
        row["uniform_all_at_max_size_fallback_queries"] = fallbacks()
        row["queries_per_launch"] = int(b * n + lens.sum())
        eq_loop = eq_sent = True
        gmax = 0.0
        for c, k in enumerate(lens):
            k = int(k)
            eq_loop &= torch.equal(o_r.d1[c].view(torch.int32), o_l[c].d1[0].view(torch.int32))
            eq_loop &= torch.equal(o_r.d2[c, :k].view(torch.int32), o_l[c].d2[0].view(torch.int32))
            eq_loop &= torch.equal(o_r.i2[c, :k], o_l[c].i2[0]) and torch.equal(o_r.i1[c], o_l[c].i1[0])
            eq_sent &= torch.equal(o_r.d1[c].view(torch.int32), o_s.d1[c].view(torch.int32))
            eq_sent &= torch.equal(o_r.d2[c, :k].view(torch.int32), o_s.d2[c, :k].view(torch.int32))
            g_r = o_r.g1.view(b, n, 3)[c]
            gmax = max(gmax, float(((g_r - o_l[c].g1.view(n, 3)).abs() / (o_l[c].g1.view(n, 3).abs() + 1e-6)).max()))
        row["ragged_vs_loop_bits_equal"] = bool(eq_loop)
        row["ragged_vs_sentinel_real_rows_bits_equal"] = bool(eq_sent)
        row["ragged_vs_loop_grad1_max_rel_diff"] = gmax
        row["speedup_vs_loop"] = row["per_sample_loop_ms"] / row["ragged_one_launch_ms"]
        row["speedup_vs_sentinel"] = row["far_sentinel_padding_ms"] / row["ragged_one_launch_ms"]
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
