"""Coset openings of KZG10 on the GPU (ptau_kzg_open_cosets, ptau_kzg_check_cosets) with resident powers of a 2^21
setup:
    opens: n in {2^16, 2^18, 2^20, 2^21} coefficients, cosets of k = 2^e points for e in {0, 4, 8, 12}, m in {1, 16}
           cosets per call; wall time host to host and the library's CUDA-event kernel time (median of 5 runs after
           one warm-up); reference rows in the same run: open_many at the 2^e points of one coset (e <= 4), whose
           values must equal the coset opening's;
    checks: m in {1, 16, 256} items at e = 4 and e = 12 (a 2^16-coefficient polynomial);
    split:  in a separate torch.profiler pass, the kernel time of one coset opening at n = 2^21 by stage (quotient
           scan coset_quotient_*, NTT ntt_*, MSM) and of one check by stage.
Writes profiles/kzg_coset_bench.json (or the path given as the first argument) with the card's name and power limit
read in the same run."""
import json
import os
import random
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
REPS = 5


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return "unknown (%r)" % e


def timed(fn, ctx):
    fn()  # warm-up
    wall, kern = [], []
    for _ in range(REPS):
        t0 = time.perf_counter()
        fn()
        wall.append((time.perf_counter() - t0) * 1e3)
        kern.append(ctx.timing()["kernel_ms"][0])
    return {"wall_ms": statistics.median(wall), "kernel_ms": statistics.median(kern)}


def le_rows(vals):
    return np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in vals), dtype=np.uint8)


def split(prof, stages):
    import torch

    out = {s: 0.0 for s in stages}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
        for s, keys in stages.items():
            if any(key in ev.name for key in keys):
                out[s] += us
                break
    return {s + "_ms": v / 1e3 / REPS for s, v in out.items()}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "kzg_coset_bench.json")
    L = kz._ffi.lib()
    res = {"card": card(), "reps": REPS, "statistic": "median", "opens": [], "checks": [], "kernel_split": []}
    ctx = kz.Context(1)
    N = 1 << 21
    tau = o.derive_scalars(0x0C)[0]
    dev = kz.ResidentPoints(ctx, ctx.convert(1, 1, ctx.generate(1, 1, 1, tau, 0, N), 4, 0).reshape(N, 104))
    rng = np.random.default_rng(7)
    rnd = random.Random(7)

    def open_call(raw, n, e, hb, m, proofs, vals):
        return lambda: L.ptau_kzg_open_cosets(ctx._h, dev._h, raw.ctypes.data, n, e, hb.ctypes.data, m,
                                              proofs.ctypes.data, vals.ctypes.data)

    for lg in (16, 18, 20, 21):
        n = 1 << lg
        raw = np.ascontiguousarray(rng.integers(0, 256, size=(n, 32), dtype=np.uint8))
        raw[:, 31] &= 0x3F
        for e in (0, 4, 8, 12):
            k = 1 << e
            for m in (1, 16):
                hs = [rnd.randrange(1, R) for _ in range(m)]
                hb = le_rows(hs)
                proofs = np.zeros((m, 104), dtype=np.uint8)
                vals = np.zeros(m * k * 32, dtype=np.uint8)
                call = open_call(raw, n, e, hb, m, proofs, vals)
                t = timed(lambda: call() == 0 or sys.exit("open_cosets failed"), ctx)
                row = {"n": n, "e": e, "m": m, "open_cosets": t, "launches": ctx.timing()["kernel_launches"]}
                if e <= 4 and m == 1:  # the same 2^e points by open_many, one MSM per point
                    zb = le_rows(kz.coset_points(e, hs[0]))
                    op = np.zeros((k, 104), dtype=np.uint8)
                    ov = np.zeros(k * 32, dtype=np.uint8)
                    ref = lambda: L.ptau_kzg_open(ctx._h, dev._h, None, raw.ctypes.data, n, None, 0,  # noqa: E731
                                                  zb.ctypes.data, k, op.ctypes.data, ov.ctypes.data, None)
                    row["open_many_same_points"] = timed(lambda: ref() == 0 or sys.exit("open_many failed"), ctx)
                    row["values_equal"] = ov.tobytes() == vals.tobytes()
                    assert row["values_equal"], (n, e)
                res["opens"].append(row)
                print(json.dumps(row), flush=True)
    # checks on a 2^16-coefficient polynomial
    n = 1 << 16
    raw = np.ascontiguousarray(rng.integers(0, 256, size=(n, 32), dtype=np.uint8))
    raw[:, 31] &= 0x3F
    comm = dev.msm(raw)
    for e in (4, 12):
        k = 1 << e
        g2 = ctx.convert(2, 1, ctx.generate(2, 1, 1, tau, 0, 1), 4, 0).reshape(200)
        tk = ctx.convert(2, 1, ctx.generate(2, 1, 1, tau, k, 1), 4, 0).reshape(200)
        for m in (1, 16, 256):
            hs = [rnd.randrange(1, R) for _ in range(m)]
            hb = le_rows(hs)
            proofs = np.zeros((m, 104), dtype=np.uint8)
            vals = np.zeros(m * k * 32, dtype=np.uint8)
            assert open_call(raw, n, e, hb, m, proofs, vals)() == 0
            comms = np.ascontiguousarray(np.tile(comm, (m, 1)))
            ok = np.zeros(1, dtype=np.uint8)
            seed = bytes(32)

            def chk():
                rc = L.ptau_kzg_check_cosets(ctx._h, dev._h, g2.ctypes.data, tk.ctypes.data, e, comms.ctypes.data,
                                             hb.ctypes.data, vals.ctypes.data, proofs.ctypes.data, m, seed,
                                             ok.ctypes.data)
                assert rc == 0 and ok[0] == 1, (rc, ok[0])

            row = {"e": e, "m": m, "check_cosets": timed(chk, ctx)}
            res["checks"].append(row)
            print(json.dumps(row), flush=True)
    # per-stage kernel time from a torch.profiler pass of its own
    try:
        from torch.profiler import ProfilerActivity, profile
        import torch

        n = N
        raw = np.ascontiguousarray(rng.integers(0, 256, size=(n, 32), dtype=np.uint8))
        raw[:, 31] &= 0x3F
        for e in (0, 4, 12):
            k = 1 << e
            hb = le_rows([12345])
            proofs = np.zeros((1, 104), dtype=np.uint8)
            vals = np.zeros(k * 32, dtype=np.uint8)
            call = open_call(raw, n, e, hb, 1, proofs, vals)
            call()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(REPS):
                    assert call() == 0
                torch.cuda.synchronize()
            row = {"what": "open_cosets", "n": n, "e": e, "m": 1,
                   **split(prof, {"scan": ["coset_quotient"], "ntt": ["ntt_"], "msm": ["msm"]})}
            res["kernel_split"].append(row)
            print(json.dumps(row), flush=True)
    except Exception as e:  # noqa: BLE001
        res["kernel_split_error"] = repr(e)
    ctx.close()
    os.makedirs(os.path.dirname(out_path), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", out_path)


if __name__ == "__main__":
    main()
