"""Sinkhorn divergence on one GPU: psd_sinkhorn_divergence (forward only, and forward with both gradients) next to a plain-torch
fp32 restatement of the same steps (batched, and as the reference's per-sample loop), with emdModule and emd_certified for
context where they apply (n = m, a multiple of 1024).

    python tools/sinkhorn_bench.py --out profiles/sinkhorn_b200.json

Seeded U[0,1)^3 clouds, B = 32, n = m in {128, 256, 1024, 2048} and n = 1024 against m = 2048; blur / scaling 0.05 / 0.5 and
0.01 / 0.9.  Times are CUDA events around work on one stream, the median of --reps runs after one warm-up run per shape.  The
working set (at most a few MB for the kernel) lives in L2 after the first pass, as it does in a training loop.

Rates: a call evaluates B (n + m)^2 (len(eps_list) + 2) exponentials (four softmins per round over the init round, the loop and
the extrapolation).  The MUFU bound is that count over 16 ex2 per clock per SM x the SM count x the SM clock that nvidia-smi
reports right after the timed runs; "mufu_share" is that bound over the measured time."""
import argparse
import ctypes
import json
import math
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = ((128, 128), (256, 256), (1024, 1024), (2048, 2048), (1024, 2048))
SETTINGS = ((0.05, 0.5), (0.01, 0.9))


def smi(fields):
    try:
        q = subprocess.run(["nvidia-smi", f"--query-gpu={fields}", "--format=csv,noheader,nounits"], capture_output=True,
                           text=True, timeout=30)
        return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.SubprocessError):
        return None


def eps_list(D, blur, scaling):
    blur, scaling = float(np.float32(blur)), float(np.float32(scaling))
    return [D ** 2] + [float(np.exp(e)) for e in np.arange(2 * np.log(D), 2 * np.log(blur), 2 * np.log(scaling))] + [blur ** 2]


def torch_sinkhorn(torch, x, y, blur, scaling):
    """The kernel's steps in plain torch fp32 on [B, n, 3] / [B, m, 3] (every cloud with its own schedule, so B may be 1 for the
    per-sample loop); dense [B, n, m] cost matrices as geomloss's tensorized backend builds them.  Returns S [B]."""
    B, n, m = x.shape[0], x.shape[1], y.shape[1]
    pts = torch.cat([x, y], 1).detach()
    D = ((pts.amax(1).double() - pts.amin(1).double()) ** 2).sum(1).sqrt().tolist()
    E = [[float(np.float32(e)) for e in eps_list(d, blur, scaling)] for d in D]
    assert len({len(e) for e in E}) == 1, "the batched restatement needs one schedule length"
    E = torch.tensor(E, device=x.device, dtype=torch.float32).t()[:, :, None]          # [K, B, 1]
    la, lb = math.log(1.0 / n), math.log(1.0 / m)
    cost = lambda u, v: 0.5 * ((u[:, :, None, :] - v[:, None, :, :]) ** 2).sum(-1)
    C_xx, C_yy, C_xy, C_yx = cost(x, x.detach()), cost(y, y.detach()), cost(x, y.detach()), cost(y, x.detach())
    sm = lambda e, C, h: -e * torch.logsumexp(h[:, None, :] - C / e[:, :, None], dim=2)
    with torch.no_grad():
        e = E[0]
        za, zb = torch.full((B, n), la, device=x.device), torch.full((B, m), lb, device=x.device)
        g_ab, f_ba, f_aa, g_bb = sm(e, C_yx, za), sm(e, C_xy, zb), sm(e, C_xx, za), sm(e, C_yy, zb)
        for e in E:
            ft_ba, gt_ab = sm(e, C_xy, lb + g_ab / e), sm(e, C_yx, la + f_ba / e)
            ft_aa, gt_bb = sm(e, C_xx, la + f_aa / e), sm(e, C_yy, lb + g_bb / e)
            f_ba, g_ab, f_aa, g_bb = 0.5 * (f_ba + ft_ba), 0.5 * (g_ab + gt_ab), 0.5 * (f_aa + ft_aa), 0.5 * (g_bb + gt_bb)
    e = E[-1]
    f_ba, g_ab = sm(e, C_xy, (lb + g_ab / e).detach()), sm(e, C_yx, (la + f_ba / e).detach())
    f_aa, g_bb = sm(e, C_xx, (la + f_aa / e).detach()), sm(e, C_yy, (lb + g_bb / e).detach())
    return (f_ba - f_aa).mean(1) + (g_ab - g_bb).mean(1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON here as well as to stdout")
    ap.add_argument("--b", type=int, default=32)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()

    import torch
    import psd_b200
    if not torch.cuda.is_available():
        raise SystemExit("sinkhorn_bench.py measures on a CUDA device; none is visible")
    pkg = psd_b200.load()
    L = pkg._lib
    lib = L.lib
    dev = torch.device("cuda:0")
    vp = L.ptr
    stream = torch.cuda.current_stream(dev)
    sp = ctypes.c_void_p(stream.cuda_stream)
    num_sms = torch.cuda.get_device_properties(dev).multi_processor_count

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
        return float(np.median(ts))

    b = args.b
    rng = np.random.default_rng(2026)
    result = {"gpu": {"name": torch.cuda.get_device_name(0), "sms": num_sms,
                      "name_power_limit_W_max_sm_clock_MHz": smi("name,power.limit,clocks.max.sm")},
              "b": b, "reps": args.reps, "clouds": "uniform U[0,1)^3, numpy default_rng(2026)", "runs": []}
    for n, m in SHAPES:
        x = torch.from_numpy(rng.random((b, n, 3), dtype=np.float32)).to(dev)
        y = torch.from_numpy(rng.random((b, m, 3), dtype=np.float32)).to(dev)
        loss = torch.empty(b, device=dev)
        gx, gy = torch.empty(b, n, 3, device=dev), torch.empty(b, m, 3, device=dev)
        rounds = torch.empty(b, dtype=torch.int32, device=dev)
        for blur, scaling in SETTINGS:
            row = {"n": n, "m": m, "blur": blur, "scaling": scaling}

            def fwd():
                assert lib.psd_sinkhorn_divergence(vp(x), vp(y), b, n, m, blur, scaling, vp(loss), None, None, None, vp(rounds), sp) == 1

            def fwd_grad():
                assert lib.psd_sinkhorn_divergence(vp(x), vp(y), b, n, m, blur, scaling, vp(loss), vp(gx), vp(gy), None, vp(rounds),
                                                   sp) == 1
            row["kernel_fwd_ms"] = timed(fwd, args.reps)
            row["kernel_fwd_grad_ms"] = timed(fwd_grad, args.reps)
            K = rounds.cpu().numpy()
            row["rounds"] = sorted(set(int(k) for k in K))
            exps = float(sum((n + m) ** 2 * (int(k) + 2) for k in K))
            row["exponentials"] = exps
            clk = smi("clocks.sm")
            row["sm_clock_MHz_after"] = float(clk) if clk else None
            S_kernel = loss.clone()

            xr, yr = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
            out = {}

            def t_fwd():
                with torch.no_grad():
                    out["S"] = torch_sinkhorn(torch, x, y, blur, scaling)

            def t_fwd_grad():
                S = torch_sinkhorn(torch, xr, yr, blur, scaling)
                torch.autograd.grad(S.sum(), [xr, yr])

            def t_loop():
                for i in range(b):
                    torch_sinkhorn(torch, xr[i:i + 1], yr[i:i + 1], blur, scaling).sum().backward()
            row["torch_batched_fwd_ms"] = timed(t_fwd, args.reps)
            row["torch_batched_fwd_grad_ms"] = timed(t_fwd_grad, args.reps)
            row["torch_per_sample_loop_fwd_grad_ms"] = timed(t_loop, max(2, args.reps // 2))
            row["max_abs_diff_vs_torch_fp32"] = float((out["S"] - S_kernel).abs().max())
            if row["sm_clock_MHz_after"]:
                bound_ms = exps / (16.0 * num_sms * row["sm_clock_MHz_after"] * 1e6) * 1e3
                row["mufu_bound_ms"] = bound_ms
                row["mufu_share_fwd"] = bound_ms / row["kernel_fwd_ms"]
            row["pairs_per_s_fwd"] = exps / (row["kernel_fwd_ms"] * 1e-3)
            if n == m and n % 1024 == 0 and blur == 0.05:
                em = pkg.emdModule()
                row["emdModule_eval_ms"] = timed(lambda: em(x, y, 0.005, 50), args.reps)
                row["emd_certified_1e-4_ms"] = timed(lambda: pkg.emd_certified(x, y, eps_end=1e-4), args.reps)
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
