"""KZG10::open on the GPU (ptau_kzg_open) against the previous path, with resident powers of a 2^21 setup:
    new: ptau_kzg_open (quotient scan on the device, straight into the MSM's scalars; k points per call)
    old: ptau_kzg_quotient (host recurrence) + ptau_kzg_commit_resident with u8 scalars, once per point
for n in {2^16, 2^18, 2^20, 2^21} coefficients and k in {1, 16} points: wall time host to host and the library's
CUDA-event kernel time (median of 5 runs after one warm-up), every output compared with the old path's.  Then
KZG10.open with Python ints before (host quotient + resident MSM) and after (open_many), and, in a separate
torch.profiler pass, the per-kernel split of one open into the quotient kernels (kzg_quotient_*) and the MSM.
Writes profiles/kzg_open_bench.json (or the path given as the first argument) with the card's name and power
limit read in the same run."""
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
        k_ms = fn()
        wall.append((time.perf_counter() - t0) * 1e3)
        kern.append(k_ms if k_ms is not None else ctx.timing()["kernel_ms"][0])
    return {"wall_ms": statistics.median(wall), "kernel_ms": statistics.median(kern)}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "kzg_open_bench.json")
    L = kz._ffi.lib()
    res = {"card": card(), "reps": REPS, "statistic": "median", "runs": [], "python_ints": [], "kernel_split": []}
    ctx = kz.Context(1)
    N = 1 << 21
    tau = o.derive_scalars(0x0B)[0]
    pts = ctx.convert(1, 1, ctx.generate(1, 1, 1, tau, 0, N), 4, 0).reshape(N, 104)
    dev = kz.ResidentPoints(ctx, pts)
    powers = kz.Powers(powers_of_g=dev, powers_of_gamma_g=dev)
    rng = np.random.default_rng(7)
    rnd = random.Random(7)
    for lg in (16, 18, 20, 21):
        n = 1 << lg
        raw = np.ascontiguousarray(rng.integers(0, 256, size=(n, 32), dtype=np.uint8))
        raw[:, 31] &= 0x3F
        for k in (1, 16):
            zs = [rnd.randrange(R) for _ in range(k)]
            zb = np.frombuffer(b"".join(z.to_bytes(32, "little") for z in zs), dtype=np.uint8)
            proofs = np.zeros((k, 104), dtype=np.uint8)
            vals = np.zeros(k * 32, dtype=np.uint8)

            def new():
                rc = L.ptau_kzg_open(ctx._h, dev._h, None, raw.ctypes.data, n, None, 0, zb.ctypes.data, k,
                                     proofs.ctypes.data, vals.ctypes.data, None)
                assert rc == 0, rc
                return None

            q = np.zeros((n - 1) * 32, dtype=np.uint8)
            v = np.zeros(32, dtype=np.uint8)
            old_proofs = np.zeros((k, 104), dtype=np.uint8)
            old_vals = np.zeros(k * 32, dtype=np.uint8)

            def old():
                kms = 0.0
                for j in range(k):
                    assert L.ptau_kzg_quotient(raw.ctypes.data, n, zb[32 * j:].ctypes.data, q.ctypes.data, v.ctypes.data) == 0
                    assert L.ptau_kzg_commit_resident(ctx._h, dev._h, q.ctypes.data, n - 1, old_proofs[j].ctypes.data) == 0
                    kms += ctx.timing()["kernel_ms"][0]
                    old_vals[32 * j:32 * j + 32] = v
                return kms

            t_new = timed(new, ctx)
            launches = ctx.timing()["kernel_launches"]
            t_old = timed(old, ctx)
            same = proofs.tobytes() == old_proofs.tobytes() and vals.tobytes() == old_vals.tobytes()
            res["runs"].append({"n": n, "k": k, "new": t_new, "old": t_old, "new_launches": launches,
                                "speedup_wall": t_old["wall_ms"] / t_new["wall_ms"], "outputs_equal": same})
            print(json.dumps(res["runs"][-1]), flush=True)
            assert same, (n, k)
        # KZG10.open with Python ints, before (host quotient + resident MSM) and after (open_many)
        ints = [int.from_bytes(raw[i].tobytes(), "little") for i in range(n)]
        z = rnd.randrange(R)

        def before():
            value, qq = kz.KZG10._quotient(ints, z)
            return value, kz.KZG10._msm(ctx, [(dev, qq)])

        def after():
            value, proof, _ = kz.KZG10.open(powers, ints, z, ctx=ctx)
            return value, proof

        walls = {}
        outs = {}
        for name, fn in (("before", before), ("after", after)):
            fn()
            ts = []
            for _ in range(REPS):
                t0 = time.perf_counter()
                outs[name] = fn()
                ts.append((time.perf_counter() - t0) * 1e3)
            walls[name] = statistics.median(ts)
        same = outs["before"][0] == outs["after"][0] and outs["before"][1].tobytes() == outs["after"][1].tobytes()
        res["python_ints"].append({"n": n, "before_wall_ms": walls["before"], "after_wall_ms": walls["after"],
                                   "outputs_equal": same})
        print(json.dumps(res["python_ints"][-1]), flush=True)
        assert same, n
    # per-kernel split of one open (k = 1) from a torch.profiler pass of its own
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile

        for lg in (16, 21):
            n = 1 << lg
            raw = np.ascontiguousarray(rng.integers(0, 256, size=(n, 32), dtype=np.uint8))
            raw[:, 31] &= 0x3F
            zb = np.frombuffer((12345).to_bytes(32, "little"), dtype=np.uint8)
            pr = np.zeros(104, dtype=np.uint8)
            vl = np.zeros(32, dtype=np.uint8)
            call = lambda: L.ptau_kzg_open(ctx._h, dev._h, None, raw.ctypes.data, n, None, 0, zb.ctypes.data, 1,  # noqa: E731
                                           pr.ctypes.data, vl.ctypes.data, None)
            call()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(REPS):
                    assert call() == 0
                torch.cuda.synchronize()
            quot, msm, names = 0.0, 0.0, {}
            for ev in prof.events():
                if ev.device_type != torch.autograd.DeviceType.CUDA:
                    continue
                us = ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
                if "kzg_quotient" in ev.name:
                    quot += us
                    names[ev.name] = names.get(ev.name, 0.0) + us
                elif "msm" in ev.name:
                    msm += us
            res["kernel_split"].append({"n": n, "k": 1, "quotient_kernels_ms": quot / 1e3 / REPS,
                                        "msm_kernels_ms": msm / 1e3 / REPS,
                                        "quotient_by_kernel_ms": {k2: v2 / 1e3 / REPS for k2, v2 in names.items()}})
            print(json.dumps(res["kernel_split"][-1]), flush=True)
    except Exception as e:  # noqa: BLE001
        res["kernel_split_error"] = repr(e)
    ctx.close()
    os.makedirs(os.path.dirname(out_path), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", out_path)


if __name__ == "__main__":
    main()
