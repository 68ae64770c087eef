"""Ragged ICP batches on one GPU: one psd_icp_batch_ragged launch next to a per-sample loop, and the ragged entry next to
psd_icp_batch at equal sizes.

    python tools/icp_ragged_bench.py --out profiles/icp_ragged_b200.json

Case "scans": B = 32 seeded scans of 512 to 4096 points (sizes drawn uniformly) as the moving sources against 1024-point
predictions, at the evaluation setting of testnet.py:57-64 (tolerance 1e-10, at most 1024 iterations).  Scan and prediction
of a sample are two noisy samplings of one random shape (16 Gaussian blobs), the scan turned by a small rotation and shifted.
One icp_ragged launch is timed against a loop of 32 single-sample icp_ragged calls on the unpadded scans, and each sample's
iteration count is recorded: a launch waits for its slowest sample, whose cost is iterations x na x nb point pairs per NN pass.
Case "equal": B = 32, n = m = 1024 (the same kind of data), icp_ragged with full lengths against icp_batch; the outputs are
compared bit for bit.  Each time is the median of --reps CUDA-event timings on one stream after --warmup untimed runs.  The
working set (under 1 MB) stays in shared memory and L2 whatever is done between runs."""
import argparse
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


def rot(axis, th):
    axis = np.asarray(axis, dtype=np.float64)
    axis /= np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * K @ K


def shape_pair(rng, k_scan, k_pred):
    """(scan [k_scan, 3], prediction [k_pred, 3]) float32: two samplings of 16 Gaussian blobs, the scan moved rigidly"""
    c = rng.random((16, 3))
    draw = lambda k: c[rng.integers(0, 16, size=k)] + 0.05 * rng.standard_normal((k, 3))
    scan, pred = draw(k_scan), draw(k_pred)
    R = rot(rng.standard_normal(3), 0.1 + 0.1 * rng.random())
    scan = (scan - 0.5) @ R.T + 0.5 + 0.03 * rng.standard_normal(3)
    return scan.astype(np.float32), pred.astype(np.float32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON here as well as to stdout")
    ap.add_argument("--b", type=int, default=32)
    ap.add_argument("--m", type=int, default=1024, help="prediction size")
    ap.add_argument("--lo", type=int, default=512)
    ap.add_argument("--hi", type=int, default=4096)
    ap.add_argument("--tolerance", type=float, default=1e-10)
    ap.add_argument("--max-iterations", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()

    import torch
    import psd_b200
    if not torch.cuda.is_available():
        raise SystemExit("icp_ragged_bench.py measures on a CUDA device; none is visible")
    pkg = psd_b200.load()
    dev = torch.device("cuda:0")
    kw = dict(tolerance=args.tolerance, max_iterations=args.max_iterations)

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(args.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        return {"median_ms": float(np.median(ts)), "min_ms": float(np.min(ts)), "max_ms": float(np.max(ts)), "reps": len(ts)}

    rng = np.random.default_rng(args.seed)
    result = {"gpu": {"name_power_limit_W_max_sm_clock_MHz": smi("name,power.limit,clocks.max.sm")},
              "torch": torch.__version__, "cuda": torch.version.cuda, "setting": vars(args)}

    # ---- case 1: scans of different sizes against fixed-size predictions
    sizes = [int(k) for k in rng.integers(args.lo, args.hi + 1, size=args.b)]
    pairs = [shape_pair(rng, k, args.m) for k in sizes]
    scans = [torch.from_numpy(s).to(dev) for s, _ in pairs]
    preds = torch.from_numpy(np.stack([p for _, p in pairs])).to(dev)
    gt, lengths = pkg.pack_clouds(scans)
    one = lambda: pkg.icp_ragged(gt, preds, lengths, **kw)
    loop = lambda: [pkg.icp_ragged(s[None], preds[i:i + 1], **kw) for i, s in enumerate(scans)]
    T, _, it = one()
    loop_out = loop()
    torch.cuda.synchronize()
    it = it.cpu().numpy()
    same = all(torch.equal(T[i].view(torch.int64), o[0][0].view(torch.int64)) and int(o[2][0]) == int(it[i])
               for i, o in enumerate(loop_out))
    cost = [int(it[i] + 1) * sizes[i] * args.m for i in range(args.b)]   # NN passes = iterations + 1 (the reference's i + 1)
    slow = int(np.argmax(cost))
    result["scans"] = {
        "sizes": sizes, "iterations": [int(x) for x in it], "nn_pair_tests": cost,
        "slowest_sample": {"index": slow, "na": sizes[slow], "nb": args.m, "iterations": int(it[slow])},
        "sum_over_max_nn_pair_tests": sum(cost) / max(cost),
        "one_launch": timed(one), "per_sample_loop": timed(loop), "loop_bits_equal_launch": bool(same)}
    print(json.dumps({"scans": {k: result["scans"][k] for k in ("one_launch", "per_sample_loop", "loop_bits_equal_launch")}}),
          flush=True)

    # ---- case 2: equal sizes, ragged entry against psd_icp_batch
    pairs = [shape_pair(rng, args.m, args.m) for _ in range(args.b)]
    A = torch.from_numpy(np.stack([s for s, _ in pairs])).to(dev)
    B = torch.from_numpy(np.stack([p for _, p in pairs])).to(dev)
    full = torch.full((args.b,), args.m, dtype=torch.int32, device=dev)
    rag = lambda: pkg.icp_ragged(A, B, full, full, **kw)
    uni = lambda: pkg.icp.icp_batch(A, B, None, args.max_iterations, args.tolerance)
    r, u = rag(), uni()
    torch.cuda.synchronize()
    eq = all(torch.equal(x.view(torch.int64) if x.dtype == torch.float64 else x, y.view(torch.int64) if y.dtype == torch.float64 else y)
             for x, y in zip(r, u))
    t_rag, t_uni, t_rag2, t_uni2 = timed(rag), timed(uni), timed(rag), timed(uni)   # alternated
    result["equal"] = {"n": args.m, "m": args.m, "iterations": [int(x) for x in u[2].cpu()], "icp_ragged": [t_rag, t_rag2],
                       "icp_batch": [t_uni, t_uni2], "bits_equal": bool(eq)}
    print(json.dumps({"equal": {k: result["equal"][k] for k in ("icp_ragged", "icp_batch", "bits_equal")}}), flush=True)
    result["gpu"]["after"] = smi("name,power.limit,clocks.max.sm")

    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
