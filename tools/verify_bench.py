#!/usr/bin/env python3
"""Timings of ptau_msm_g2 and ptau_verify_powers; writes one JSON line to profiles/verify_bench.json (or --out).

  * MSM kernel time (CUDA events around the MSM launches, ptau_last_timing) of ptau_msm_g2 and, at the same sizes,
    ptau_kzg_commit; median of --reps calls.  Every call uploads its points and scalars before the timed kernels;
    there is no other L2 flush, so the 2^16 (13 MB of G2 points) case can be served from L2, the 2^22 one cannot.
  * Wall time of ptau_verify_powers on a 2^21 response and on a 2^21 fastkgz setup (host memory in, result out),
    next to ptau_preprocess (fused, fastkgz) on the same response; median of --reps calls.  One more call of each
    runs under torch.profiler (a run of its own) to split the kernel time by kernel family.
The device name and power limit are read by the same process, before the timings."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import numpy as np  # noqa: E402

import kzg_setup_powersoftau_b200 as kz  # noqa: E402
import ptau_oracle as o  # noqa: E402

R = o.R_ORDER


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    first = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    parts = [p.strip() for p in first.split(",")]
    return {"name": parts[0] if parts else "unknown", "power_limit": parts[1] if len(parts) > 1 else "unknown",
            "max_sm_clock": parts[2] if len(parts) > 2 else "unknown"}


def family(name: str) -> str:
    if "convert_kernel" in name:
        return "convert"
    if "msm_" in name:
        return "msm"
    if "ratio_coeff" in name:
        return "coefficients"
    if "pairing_product2" in name:
        return "pairing"
    return "other"


def profiled(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            k = family(ev.name)
            out[k] = out.get(k, 0.0) + ev.device_time_total / 1000.0
    return {k: round(v, 3) for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--log2", type=int, default=21)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "verify_bench.json"))
    args = ap.parse_args()
    dev = device_info()
    rec = {"device": dev, "reps": args.reps, "l2": "points and scalars uploaded before each timed MSM; no other flush"}
    rnd = np.random.default_rng(7)
    with kz.Context(1) as ctx:
        tau, alpha, beta = o.derive_scalars(0xBE7C)
        # ---- MSM: G2 next to G1
        nmax = 1 << 22
        g2 = ctx.convert(2, 1, ctx.generate(2, 1, 1, tau, 0, nmax), 4, 0).reshape(nmax, 200)
        g1 = ctx.convert(1, 1, ctx.generate(1, 1, 1, tau, 0, nmax), 4, 0).reshape(nmax, 104)
        sc_all = rnd.integers(0, 2**63, size=(nmax, 4), dtype=np.uint64)
        sc_all[:, 3] &= np.uint64(0x0FFFFFFFFFFFFFFF)  # < 2^252 < r
        sc_all = sc_all.view(np.uint8).reshape(nmax, 32)
        L = kz._ffi.lib()
        msm = {}
        for lg in (16, 18, 20, 22):
            n = 1 << lg
            sc = np.ascontiguousarray(sc_all[:n])
            row = {}
            for name, pts, fn in (("msm_g2", g2, L.ptau_msm_g2), ("kzg_commit_g1", g1, L.ptau_kzg_commit)):
                p = np.ascontiguousarray(pts[:n])
                out = np.zeros(200, dtype=np.uint8)
                ms = []
                for r in range(args.reps + 1):
                    assert fn(ctx._h, p.ctypes.data, sc.ctypes.data, n, out.ctypes.data) == 0
                    if r:
                        ms.append(ctx.timing()["kernel_ms"][0])
                med = statistics.median(ms)
                row[name] = {"kernel_ms": round(med, 3), "points_per_s": round(n / (med / 1000.0))}
            msm["2^%d" % lg] = row
        rec["msm"] = msm
        # ---- verify_powers on a 2^k response and fastkgz setup, preprocess on the same response
        n = 1 << args.log2
        g = lambda grp, s0, cnt: ctx.generate(grp, 2, s0, tau, 0, cnt)
        resp = np.concatenate([np.zeros(64, dtype=np.uint8), g(1, 1, 2 * n - 1), g(2, 1, n), g(1, alpha, n), g(1, beta, n),
                               g(2, beta, 1), np.zeros(o.PUBKEY_SIZE, dtype=np.uint8)])
        fast = ctx.preprocess(kz.VARIANT_FASTKGZ, resp, n)
        seed = b"\x5a" * 32
        calls = {
            "verify_response": lambda: ctx.verify_powers(kz.POWERS_RESPONSE, resp, n, seed=seed),
            "verify_fastkgz": lambda: ctx.verify_powers(kz.POWERS_FASTKGZ, fast, n, seed=seed),
            "preprocess_fastkgz": lambda: ctx.preprocess(kz.VARIANT_FASTKGZ, resp, n, out=fast),
        }
        walls = {}
        for name, fn in calls.items():
            ts = []
            for r in range(args.reps + 1):
                t0 = time.perf_counter()
                fn()
                if r:
                    ts.append((time.perf_counter() - t0) * 1000.0)
            walls[name] = {"wall_ms": round(statistics.median(ts), 1)}
        for name, fn in calls.items():
            walls[name]["kernel_ms_by_family"] = profiled(fn)
        rec["log2_powers"] = args.log2
        rec["calls"] = walls
    line = json.dumps(rec)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
