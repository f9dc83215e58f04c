"""Time a Powers-of-Tau contribution (ptau_contribute) and its check (ptau_verify_contribution) on the GPU.

Writes profiles/contribute_bench.json (or --out) with the device name and power limit read in the same run.
  - contribute host -> host, challenge and response in pinned memory, median of --reps after one warm-up, and the
    BLAKE2b of the challenge on the host apart; the conversion and contribution kernels apart from one call under
    torch.profiler, run after the timed calls;
  - the C oracle's scalar multiplication (oracle/cpu_ref.c, all threads) for scale;
  - G1 and G2 points per second of the whole call;
  - Fq products per point counted from the code (below) over the measured ptau_microbench kind-2 rate: the
    multiplication-bound floor of the contribution kernels;
  - verify_contribution wall time with and without the challenge.

Fq products per point (csrc/contribute.cuh; Fq2 product = 3 Fq products; the doubling is dbl-2009-l, 7 products; the
complete Jacobian addition 16; the batch inversion is amortised over 8 points and left out):
  G1: 128 doublings x 7 + 66 additions x 16 x 15/16 (digit non-zero) + table (1 doubling, 6 mixed additions x 11,
      8 endomorphism products) + affine/encode (~6) = ~1,970
  G2: (64 doublings x 7 + 68 additions x 16 x 15/16) x 3 + table (7 + 6 x 11 + 24 maps x 5) = ~4,760
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import kzg_setup_powersoftau_b200 as p  # noqa: E402
import ptau_oracle as o  # noqa: E402

FQ_PRODUCTS = {"g1": 128 * 7 + 66 * 16 * 15 / 16 + 7 + 6 * 11 + 8 + 6,
               "g2": (64 * 7 + 68 * 16 * 15 / 16) * 3 + 7 * 3 + 6 * 11 * 3 + 24 * 5 + 18}


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2", type=int, default=21)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "contribute_bench.json"))
    a = ap.parse_args()
    n = 1 << a.log2
    L = p._ffi.lib()
    ctx = p.Context(1)
    t0, a0, b0 = o.derive_scalars(21)
    chal = p.PinnedBuffer(L.ptau_challenge_size(n))
    resp = p.PinnedBuffer(L.ptau_response_size(n))
    cv = chal.array
    U = p.FMT_ZCASH_UNCOMPRESSED
    off = 64
    for g, s0, cnt in ((1, 1, 2 * n - 1), (2, 1, n), (1, a0, n), (1, b0, n), (2, b0, 1)):
        size = cnt * 96 * g
        ctx.generate(g, U, s0, t0, 0, cnt, out=cv[off:off + size])
        off += size
    rv = resp.array
    secrets = (3, 5, 7, 11, 13, 17)
    ctx.contribute(cv, n, secrets=secrets, out=rv)  # warm-up
    walls, gpus = [], []
    for _ in range(a.reps):
        t = time.perf_counter()
        ctx.contribute(cv, n, secrets=secrets, out=rv)
        walls.append((time.perf_counter() - t) * 1e3)
        tm = ctx.timing()
        gpus.append(tm["gpu_ms"][0])
    t = time.perf_counter()
    hashlib.blake2b(cv.data).digest()
    b2_ms = (time.perf_counter() - t) * 1e3
    vw = []
    for chal_arg in (cv, None):
        t = time.perf_counter()
        ctx.verify_contribution(chal_arg, rv, n)
        vw.append((time.perf_counter() - t) * 1e3)
    # conversion and contribution kernels apart: torch.profiler (CUPTI sees the library's kernels) over one call,
    # in a run of its own after the timed ones
    split = {}
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile

        torch.cuda.init()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ctx.contribute(cv, n, secrets=secrets, out=rv)
        for ev in prof.key_averages():
            for key in ("contribute_kernel", "convert_kernel"):
                if key in ev.key:
                    split[key] = split.get(key, 0.0) + ev.device_time_total / 1e3
    except Exception as e:  # the profiler is an extra; the timed numbers above stand without it
        split = {"not measured": repr(e)}
    # the C oracle's scalar multiplication (double-and-add over the full scalar, oracle/cpu_ref.c) on all threads
    import cpu_ref

    threads = os.cpu_count()
    cpu = {}
    for g, cnt in ((1, 4096), (2, 1024)):
        t = time.perf_counter()
        cpu_ref.generate(g, 2, 3, t0, 1, cnt, nthreads=threads)
        cpu["g%d_points_per_s" % g] = cnt / (time.perf_counter() - t)
    ms, ops = ctx.microbench(2, 2000)
    rate = ops / (ms * 1e-3)
    wall = statistics.median(walls)
    res = {
        "device": device_info(),
        "n_powers": n,
        "g1_points": 4 * n - 1, "g2_points": n + 1,
        "contribute_wall_ms_median": wall, "contribute_wall_ms": walls,
        "gpu_ms_median (per section: first enqueue -> last completion, summed)": statistics.median(gpus),
        "kernel_ms_by_kernel (torch.profiler, one call, device time summed per kernel name)": split,
        "c_oracle_cpu_scalar_mul (cpu_ref generate, %d threads)" % threads: cpu,
        "blake2b_challenge_ms (Python hashlib, one thread)": b2_ms,
        "points_per_s_whole_call": (5 * n) / (wall * 1e-3),
        "fq_products_per_point": FQ_PRODUCTS,
        "fq_mul_rate_per_s (microbench kind 2)": rate,
        "multiplication_floor_ms": ((4 * n - 1) * FQ_PRODUCTS["g1"] + (n + 1) * FQ_PRODUCTS["g2"]) / rate * 1e3,
        "verify_contribution_ms": {"with_challenge": vw[0], "without_challenge": vw[1]},
    }
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
