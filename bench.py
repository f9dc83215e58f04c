#!/usr/bin/env python3
"""bench.py -- headline benchmark of the Powers-of-Tau -> arkworks path on B200.

Metric (BASELINE.json): G1/G2 points/sec, parse + decompress + on-curve + subgroup check +
arkworks re-encode.  Workload = BASELINE configs[2]: 2^21 compressed G1 tau-powers +
2^21 compressed G2 tau-powers (known tau) -> Fq / Fq2 sqrt decompression -> canonical +
on-curve + subgroup check -> ark little-endian records
(/root/reference/src/bin/preprocess-kgz.rs:105-110 then :140-153).  Under torchrun the SAME
workload is sharded by contiguous index ranges over the ranks (strong scaling, no data-path
collective): rank k owns [k N / G, (k+1) N / G) of each section.

One "step" = one pass of the hot path over the rank's share of both sections (two launches):
  value : inputs already in HBM, kernels only, CUDA events on the launch stream, L2 flushed
          between timed iterations, max over ranks
  e2e   : two ptau_convert() calls on pinned HOST buffers (H2D + kernel + D2H inside the timer)
`config5` (same JSON line, every N): BASELINE configs[4], the 2^26-power setup sharded by index
range over the ranks, device-resident and host -> host.  `extra` (N=1): the other kernels of
the path, the drop-in binary on files, the loaders, the KZG10 consumer calls.

`--impl reference` times the CPU restatement of the reference's algorithms (oracle/cpu_ref.c,
kind "port": the Rust reference cannot be built here) on a bounded sample of the same
workload (Algorithm-9 Fq2 sqrt, multiplication by r) with all host threads.

`--dump-outputs DIR` writes what the last timed headline step returned (see dump_outputs) as
DIR/<name>.npy, so that two builds run with the same arguments can be compared output for output.
"""
import argparse
import csv
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LOG2_POINTS = 21
IMAD_PER_FQMUL = 588  # SURVEY.md 8d: 12x32-bit CIOS, lo+hi counted separately
# SURVEY.md 8d algorithmic Fq multiplications per point
FQMUL = {"g1_unc": 1030, "g2_unc": 1180, "g1_comp": 1500, "g2_comp": 2120}
HBM_PEAK_FALLBACK_GBPS = 6552.0  # the value MEASURED_PEAKS.json held on this pool's B200s when this was written


def hbm_peak():
    """(GB/s, source): the driver-written copy bandwidth of MEASURED_PEAKS.json when the file travelled with the repo,
    else the value it held on this pool (the profiling recipe's fallback), saying which."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            v = float(json.load(f)["hbm_gbs"])
        if v > 0:
            return v, "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        pass
    return HBM_PEAK_FALLBACK_GBPS, "fallback: MEASURED_PEAKS.json absent, its last known value on this pool"


HBM_PEAK_GBPS, HBM_PEAK_SOURCE = hbm_peak()
METRIC = "G1+G2 points/sec parse+decompress+subgroup-check+ark re-encode (2^21 compressed G1 + 2^21 compressed G2 per step)"
TAU = 0x1234567890ABCDEF1234567890ABCDEF
# the ncu capture the `traffic` / pipe-busy figures of the roofline object are read from (tools/ncu_summary.py output)
NCU_SUMMARY = os.path.join("profiles", "r02_ncu_full_all_kernels.csv")
KERNEL_G1C, KERNEL_G2C = "convert_kernel<1, 2, 3, 1>", "convert_kernel<2, 2, 3, 1>"
# --dump-outputs: points per group it writes, 2^15 x (96 + 192) bytes as float32 = 38 MB, and the seed of their indices
DUMP_POINTS = 1 << 15
DUMP_SEED = 0xB200


def dump_outputs(out_dir, n, d_out1, d_out2, status):
    """Write the headline step's results as the caller receives them: the ark uncompressed G1 and G2 records
    (96 / 192 bytes each, one row per point, bytes as float32) of a fixed seeded sample of DUMP_POINTS point indices
    (every index when n is smaller), the sorted indices themselves, and the status word (-1: every point passed)."""
    import numpy as np
    import torch

    if n <= DUMP_POINTS:
        idx = np.arange(n)
    else:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_POINTS, replace=False))
    sel = torch.from_numpy(idx).to(d_out1.device)
    arrays = {"index": idx.astype(np.float64),
              "g1_ark_uncompressed": d_out1.view(n, 96).index_select(0, sel).cpu().numpy().astype(np.float32),
              "g2_ark_uncompressed": d_out2.view(n, 192).index_select(0, sel).cpu().numpy().astype(np.float32),
              "status": np.array([status.item()], dtype=np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_config(log2_points, world):
    """`config` of the JSON line: identical for the GPU arm and the reference arm."""
    n = 1 << log2_points
    return {
        "workload": "BASELINE configs[2]: 2^%d compressed G1 + 2^%d compressed G2 tau powers -> Fq/Fq2 sqrt "
                    "decompression + canonical + on-curve + subgroup check + ark LE re-encode" % (log2_points, log2_points),
        "g1_points": n, "g2_points": n, "checks": "strict", "input": "zcash compressed, [tau^i]G, known tau",
        "sharding": "contiguous index range of each section per rank (%d rank%s), no collective" % (world, "" if world == 1 else "s"),
        "l2": "GPU arm: flushed (256 MB fill) between timed iterations",
    }


def sample_clocks(stop, out):
    q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    dev = os.environ.get("LOCAL_RANK", "0")
    while not stop.is_set():
        try:
            r = subprocess.run(["nvidia-smi", "-i", dev, "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                               capture_output=True, text=True, timeout=5)
            f = [x.strip() for x in r.stdout.strip().split(",")]
            if len(f) >= 7:
                out.append(f)
        except Exception:
            pass
        stop.wait(0.1)


def summarize_clocks(samples):
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
    sm = sorted(int(float(s[0])) for s in samples)
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    reasons = [n for i, n in enumerate(names) if any(s[3 + i].lower().startswith("active") for s in samples)]
    return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(samples[0][1])), "reasons": reasons,
            "samples": len(samples), "power_w_max": max(float(s[2]) for s in samples)}


def ncu_summary_metrics(kernel):
    """Per-launch figures of `kernel` from the committed ncu --set full summary (None when the file is absent)."""
    path = os.path.join(ROOT, NCU_SUMMARY)
    if not os.path.exists(path):
        return None
    rows = list(csv.reader(open(path)))
    cols = [i for i, name in enumerate(rows[0]) if name.startswith("void " + kernel[:20]) and kernel in name]
    if not cols:
        return None
    import math

    def column(c):
        return {r[0]: r[c] for r in rows[1:] if len(r) > c}

    def num(m, name):
        try:
            v = float(m[name])
            return v if math.isfinite(v) else None
        except Exception:
            return None
    # the last capture of the kernel whose counters are complete (ncu leaves "-nan" in a column when a replay pass failed)
    usable = [c for c in cols if num(column(c), "dram__bytes_read.sum") is not None
              and num(column(c), "sm__pipe_fmaheavy_cycles_active.avg.pct_of_peak_sustained_elapsed") is not None]
    if not usable:
        return None
    m = column(usable[-1])

    def f(name):
        return num(m, name)
    grid, block = f("launch__grid_size"), f("launch__block_size")
    rd, wr = f("dram__bytes_read.sum"), f("dram__bytes_write.sum")
    units = {r[0]: r[1] for r in rows[1:]}
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    if rd is not None:
        rd *= scale.get(units.get("dram__bytes_read.sum", "byte"), 1.0)
    if wr is not None:
        wr *= scale.get(units.get("dram__bytes_write.sum", "byte"), 1.0)
    return {"points": grid * block if grid and block else None, "dram_bytes": (rd + wr) if rd is not None and wr is not None else None,
            "fmaheavy_pct": f("sm__pipe_fmaheavy_cycles_active.avg.pct_of_peak_sustained_elapsed"),
            "kernel_ms_in_capture": f("gpu__time_duration.sum"),
            "registers": f("launch__registers_per_thread"),
            "local_ld_sectors": f("l1tex__t_sectors_pipe_lsu_mem_local_op_ld.sum"),
            "local_st_sectors": f("l1tex__t_sectors_pipe_lsu_mem_local_op_st.sum")}


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle (C restatement of the reference's algorithms) on host cores
# ---------------------------------------------------------------------------------------------
def cpu_config3(n_sample, threads, fast_predicates=False, inputs=None):
    """n_sample compressed G1 + n_sample compressed G2 points through the reference's two stages:
    Accumulator::deserialize(Compressed, No) + serialize(No) (preprocess-kgz.rs:105-124: sqrt decompression, Fq2 by
    Algorithm 9) and read_g1/read_g2 (src/lib.rs:41-80: byte reversal + ark deserialize_uncompressed = multiplication
    by r) + serialize_uncompressed.  fast_predicates=True: same C code with the GPU's predicates (GLV / psi checks,
    norm-method Fq2 sqrt) -- separates the algorithmic from the hardware speed-up.
    -> (points/s, seconds, inputs)"""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import cpu_ref

    if inputs is None:
        inputs = {g: cpu_ref.generate(g, 2, 1, TAU, 0, n_sample, threads) for g in (1, 2)}
    fp = 16 if fast_predicates else 0
    t0 = time.perf_counter()
    for g in (1, 2):
        zu, st = cpu_ref.convert(g, 2, inputs[g], 1, fp, threads)
        assert not any(st)
        _, st = cpu_ref.convert(g, 1, zu, 3, 4 | fp, threads)
        assert not any(st)
    dt = time.perf_counter() - t0
    return 2 * n_sample / dt, dt, inputs


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    # size the per-step sample to ~3 s on this host
    rate, _, _ = cpu_config3(1 << 9, threads)
    n_sample = 1 << 9
    while 2 * (2 * n_sample) / rate <= 4.0 and n_sample < (1 << args.log2_points):
        n_sample *= 2
    _, _, inputs = cpu_config3(n_sample, threads)  # untimed: builds the inputs, warms the caches
    for _ in range(max(args.warmup - 1, 0)):
        cpu_config3(1 << 9, threads)
    t_total = 0.0
    for _ in range(args.steps):
        _, dt, _ = cpu_config3(n_sample, threads, inputs=inputs)
        t_total += dt
    value = 2 * n_sample * args.steps / t_total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "points/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64 (6x64-bit Montgomery)",
        "data": "synthetic", "config": workload_config(args.log2_points, args.gpus),
        "cpu_baseline": {"value": value, "unit": "points/s", "cores": threads, "kind": "port",
                         "sample": "first %d compressed G1 + first %d compressed G2 points of the workload per step: "
                                   "Fq sqrt / Algorithm-9 Fq2 sqrt decompression, then read_g1/read_g2 with the "
                                   "r-multiplication subgroup check (ark-ec 0.2 semantics), %d threads"
                                   % (n_sample, n_sample, threads)},
        "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------
# BASELINE configs[4]: the 2^K-power setup sharded over the ranks
# ---------------------------------------------------------------------------------------------
def run_config5(log2_powers, with_e2e, kz, sharding, torch, dist, ctx, rank, world, dev):
    """A 2^K-power synthetic setup (known tau) sharded by contiguous index ranges over the ranks.  Per rank: for each
    section of the kgz pipeline, its index range is generated on the GPU slab by slab (compressed zcash encoding,
    [s*tau^i]G) and pushed through the fused compressed -> strict checks -> ark kernel.  `value`: only the convert
    kernels are timed (CUDA events); `e2e`: every slab pinned host -> ptau_convert -> pinned host (wall clock).
    Strong scaling: the total work is fixed.  Returns the result object (all ranks take part in the reductions)."""
    n = 1 << log2_powers
    alpha, beta = 0x0FEDCBA987654321, 0x13579BDF02468ACE
    secs = [("tau_g1", kz.G1, 1, 2 * n - 1), ("tau_g2", kz.G2, 1, n), ("alpha_g1", kz.G1, alpha, n),
            ("beta_g1", kz.G1, beta, n)]
    slab = 1 << 22
    d_in = torch.empty(slab * 96, dtype=torch.uint8, device=dev)
    d_out = torch.empty(slab * 192, dtype=torch.uint8, device=dev)
    status = torch.full((1,), -1, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream()
    ZC, AU = kz.FMT_ZCASH_COMPRESSED, kz.FMT_ARK_UNCOMPRESSED
    h_in = h_out = None
    if with_e2e:
        h_in, h_out = kz.PinnedBuffer(slab * 96), kz.PinnedBuffer(slab * 192)
        h_in_t, h_out_t = torch.from_numpy(h_in.array), torch.from_numpy(h_out.array)
    e2e_s, h2d, d2h, e2e_launches, checked = 0.0, 0, 0, 0, set()
    for g in (kz.G1, kz.G2):  # warm-up (also builds the generator tables)
        ctx.generate_device(g, ZC, 1, TAU, 0, 4096, d_in.data_ptr(), stream=stream.cuda_stream)
        for _ in range(3):
            ctx.convert_device(g, ZC, d_in.data_ptr(), AU, d_out.data_ptr(), 4096, kz.CHECKS_STRICT, status.data_ptr(),
                               stream=stream.cuda_stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks, stop = [], threading.Event()
    th = threading.Thread(target=sample_clocks, args=(stop, clocks), daemon=True)
    th.start()
    t_wall = time.perf_counter()
    ms = {"G1": 0.0, "G2": 0.0}
    pts = {"G1": 0, "G2": 0}
    launches = 0
    for name, g, s0, cnt in secs:
        lo, hi = sharding.shard_range(cnt, rank, world)
        for a in range(lo, hi, slab):
            c = min(slab, hi - a)
            ctx.generate_device(g, ZC, s0, TAU, a, c, d_in.data_ptr(), stream=stream.cuda_stream)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            ctx.convert_device(g, ZC, d_in.data_ptr(), AU, d_out.data_ptr(), c, kz.CHECKS_STRICT, status.data_ptr(),
                               base_index=a, stream=stream.cuda_stream)
            e1.record(stream)
            e1.synchronize()
            key = "G1" if g == kz.G1 else "G2"
            ms[key] += e0.elapsed_time(e1)
            pts[key] += c
            launches += 1
            if h_in is not None:
                ri, ro = (48, 96) if g == kz.G1 else (96, 192)
                h_in_t[:c * ri].copy_(d_in[:c * ri])  # untimed: stands for the file read
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ctx.convert(g, ZC, h_in.array[:c * ri], AU, kz.CHECKS_STRICT, out=h_out.array[:c * ro])
                e2e_s += time.perf_counter() - t0
                e2e_launches += ctx.timing()["kernel_launches"]
                h2d += c * ri
                d2h += c * ro
                if name not in checked:  # byte-compare the first slab of every section with the device-resident pass
                    checked.add(name)
                    assert torch.equal(h_out_t[:c * ro], d_out[:c * ro].cpu()), "e2e output differs (%s)" % name
    torch.cuda.synchronize()
    wall = time.perf_counter() - t_wall
    stop.set()
    th.join()
    assert int(status.item()) == -1, "synthetic setup failed validation"
    if world > 1:
        dist.barrier()
    t_max = sharding.reduce_max_ms(ms["G1"] + ms["G2"])
    g1_ms, g2_ms = sharding.reduce_max_ms(ms["G1"]), sharding.reduce_max_ms(ms["G2"])
    tot_g1, tot_g2 = int(sharding.reduce_sum(pts["G1"])), int(sharding.reduce_sum(pts["G2"]))
    wall_max = sharding.reduce_max_ms(wall * 1e3)
    e2e = None
    if h_in is not None:
        e2e_ms = sharding.reduce_max_ms(e2e_s * 1e3)
        e2e = {"value": (tot_g1 + tot_g2) / (e2e_ms / 1e3), "unit": "points/s",
               "h2d_bytes_per_step": int(sharding.reduce_sum(h2d)), "d2h_bytes_per_step": int(sharding.reduce_sum(d2h)),
               "ms_per_step": e2e_ms, "note": "pinned host slabs of 2^22 points -> ptau_convert -> pinned host, max over ranks"}
        launches += e2e_launches
        h_in.free()
        h_out.free()
    return {
        "metric": "G1+G2 points/sec, compressed parse + sqrt decompress + subgroup check + ark re-encode "
                  "(2^%d-power setup, index-range sharded)" % log2_powers,
        "value": (tot_g1 + tot_g2) / (t_max / 1e3), "unit": "points/s", "n_gpus": world, "steps": 1, "warmup": 3,
        "ms_per_step": t_max, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u32 limbs (12x32-bit Montgomery, IMAD.WIDE carry chains)", "data": "synthetic",
        "config": {"workload": "BASELINE configs[4]: 2^%d powers, sections tau_g1 (2N-1), tau_g2 (N), alpha_g1 (N), "
                               "beta_g1 (N), compressed input generated on the GPU per slab" % log2_powers,
                   "g1_points": tot_g1, "g2_points": tot_g2, "g1_points_per_s": tot_g1 / (g1_ms / 1e3),
                   "g2_points_per_s": tot_g2 / (g2_ms / 1e3), "kernel_ms_g1_max_rank": g1_ms,
                   "kernel_ms_g2_max_rank": g2_ms, "wall_s_incl_generation": wall_max / 1e3,
                   "l2": "inputs larger than L2 (slabs of 2^22 points, 200-400 MB)"},
        "e2e": e2e, "gpu_launches": launches, "clocks": summarize_clocks(clocks),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log2-points", type=int, default=LOG2_POINTS, help="points per section of the headline workload")
    ap.add_argument("--no-extra", action="store_true", help="skip the non-headline legs (extra, config5, cpu_baseline)")
    ap.add_argument("--no-legs", action="store_true", help="skip only the N=1 `extra` legs and the CPU baseline (keeps config5)")
    ap.add_argument("--workload", default="config3", choices=["config3", "config5"],
                    help="config3 = headline (BASELINE configs[2], config5 reported inside the same line); config5 = only "
                         "the 2^K-power setup, printed as its own line")
    ap.add_argument("--log2-powers", type=int, default=26, help="powers of the config5 setup (0: skip it)")
    ap.add_argument("--no-e2e", action="store_true", help="config5: skip the host -> host leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed headline step to DIR/<name>.npy (one process only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "config3" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs writes the headline (config3) outputs of --impl b200 in a single process")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    import kzg_setup_powersoftau_b200 as kz
    from kzg_setup_powersoftau_b200 import sharding

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    N = 1 << args.log2_points
    lo, hi = sharding.shard_range(N, rank, world)
    n_loc = hi - lo
    # host pipeline chunk: 2^18 points at full size; for a small per-rank share keep ~8 chunks of whole waves
    wave = 148 * 2 * 128
    chunk = (1 << 18) if n_loc >= (1 << 20) else max(2 * wave, -(-(n_loc // 8) // wave) * wave)
    ctx = kz.Context(device_ids=[local], chunk_points=chunk)
    if args.workload == "config5":
        line = run_config5(args.log2_powers, not args.no_e2e, kz, sharding, torch, dist, ctx, rank, world, dev)
        if rank == 0:
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return 0
    ZU, ZC, AU, ML = kz.FMT_ZCASH_UNCOMPRESSED, kz.FMT_ZCASH_COMPRESSED, kz.FMT_ARK_UNCOMPRESSED, kz.FMT_ARK_MONT_LIMBS
    STRICT = kz.CHECKS_STRICT

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- synthetic input, generated on the GPU ([tau^i]G, i in this rank's range of each section) ----
    d_in1 = torch.empty(n_loc * 48, dtype=torch.uint8, device=dev)
    d_in2 = torch.empty(n_loc * 96, dtype=torch.uint8, device=dev)
    d_out1 = torch.empty(n_loc * 96, dtype=torch.uint8, device=dev)
    d_out2 = torch.empty(n_loc * 192, dtype=torch.uint8, device=dev)
    ctx.generate_device(kz.G1, ZC, 1, TAU, lo, n_loc, d_in1.data_ptr())
    ctx.generate_device(kz.G2, ZC, 1, TAU, lo, n_loc, d_in2.data_ptr())
    status = torch.full((1,), -1, dtype=torch.int64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    stream = torch.cuda.current_stream()

    def launch(group, in_fmt, din, out_fmt, dout, n, checks, first):
        ctx.convert_device(group, in_fmt, din.data_ptr(), out_fmt, dout.data_ptr(), n, checks, status.data_ptr(),
                           base_index=first, stream=stream.cuda_stream)

    def headline_step():
        launch(kz.G1, ZC, d_in1, AU, d_out1, n_loc, STRICT, lo)
        launch(kz.G2, ZC, d_in2, AU, d_out2, n_loc, STRICT, lo)

    clocks, stop = [], threading.Event()
    th = threading.Thread(target=sample_clocks, args=(stop, clocks), daemon=True)
    for _ in range(args.warmup):
        headline_step()
    barrier()
    th.start()
    ms_step = ms_g1 = ms_g2 = 0.0
    for _ in range(args.steps):
        flush.fill_(1)  # evict L2 between timed iterations (outside the timed events)
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record(stream)
        launch(kz.G1, ZC, d_in1, AU, d_out1, n_loc, STRICT, lo)
        e1.record(stream)
        launch(kz.G2, ZC, d_in2, AU, d_out2, n_loc, STRICT, lo)
        e2.record(stream)
        e2.synchronize()
        ms_step += e0.elapsed_time(e2)
        ms_g1 += e0.elapsed_time(e1)
        ms_g2 += e1.elapsed_time(e2)
    barrier()
    stop.set()
    th.join()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, n_loc, d_out1, d_out2, status)
    assert int(status.item()) == -1, "synthetic input failed validation"
    ms = sharding.reduce_max_ms(ms_step)
    ms_g1_max, ms_g2_max = sharding.reduce_max_ms(ms_g1), sharding.reduce_max_ms(ms_g2)
    value = 2 * N * args.steps / (ms / 1e3)
    launches = 2 * args.steps

    # ---- e2e: host buffers through the public C-ABI call ----
    h_in1, h_in2 = kz.PinnedBuffer(n_loc * 48), kz.PinnedBuffer(n_loc * 96)
    h_out1, h_out2 = kz.PinnedBuffer(n_loc * 96), kz.PinnedBuffer(n_loc * 192)
    torch.cuda.synchronize()
    torch.from_numpy(h_in1.array).copy_(d_in1.cpu())
    torch.from_numpy(h_in2.array).copy_(d_in2.cpu())

    def e2e_step():
        ctx.convert(kz.G1, ZC, h_in1, AU, STRICT, out=h_out1)
        k = ctx.timing()["kernel_launches"]
        ctx.convert(kz.G2, ZC, h_in2, AU, STRICT, out=h_out2)
        return k + ctx.timing()["kernel_launches"]

    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    e2e_launches = 0
    for _ in range(args.steps):
        e2e_launches += e2e_step()
    torch.cuda.synchronize()
    e2e_ms = sharding.reduce_max_ms((time.perf_counter() - t0) * 1e3)
    barrier()
    e2e_value = 2 * N * args.steps / (e2e_ms / 1e3)
    assert torch.equal(torch.from_numpy(h_out1.array), d_out1.cpu()), "e2e G1 output differs from device-resident output"
    assert torch.equal(torch.from_numpy(h_out2.array), d_out2.cpu()), "e2e G2 output differs from device-resident output"
    for b in (h_in1, h_in2, h_out1, h_out2):
        b.free()

    cfg = workload_config(args.log2_points, world)
    line = {
        "metric": METRIC, "value": value, "unit": "points/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u32 limbs (12x32-bit Montgomery, IMAD.WIDE carry chains)", "data": "synthetic",
        "config": cfg,
        "per_group": {"g1_points_per_s": N * args.steps / (ms_g1_max / 1e3), "g2_points_per_s": N * args.steps / (ms_g2_max / 1e3),
                      "g1_ms_per_step_max_rank": ms_g1_max / args.steps, "g2_ms_per_step_max_rank": ms_g2_max / args.steps,
                      "points_per_rank_per_section": n_loc, "host_pipeline_chunk_points": chunk},
        "e2e": {"value": e2e_value, "unit": "points/s", "h2d_bytes_per_step": int(sharding.reduce_sum(n_loc * (48 + 96))),
                "d2h_bytes_per_step": int(sharding.reduce_sum(n_loc * (96 + 192))), "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": launches + e2e_launches,
    }

    # ---- BASELINE configs[4] in the same run (all ranks) ----
    c5 = None
    if not args.no_extra and args.log2_powers > 0:
        del d_in1, d_in2, d_out1, d_out2
        c5 = run_config5(args.log2_powers, not args.no_e2e, kz, sharding, torch, dist, ctx, rank, world, dev)

    if rank == 0:
        line["clocks"] = summarize_clocks(clocks)
        if c5 is not None:
            line["config5"] = c5
        # ---- roofline: measured IMAD peak (microbenchmark, same process) ----
        mb = {}
        for kind, name in ((0, "imad32"), (1, "imad_wide"), (2, "fq_mul")):
            t, ops = ctx.microbench(kind, 4000)
            mb[name] = ops / (t / 1e3)

        def roofline(key, kernel, n_points, kernel_ms_total, rec_bytes):
            kernel_s = (kernel_ms_total / args.steps) / 1e3
            achieved = n_points * FQMUL[key] * IMAD_PER_FQMUL / kernel_s
            prof = ncu_summary_metrics(kernel)
            r = {"bound": "imad", "kernel": kernel, "achieved": achieved / 1e12, "peak": mb["imad32"] / 1e12,
                 "unit": "TIMAD/s", "frac": achieved / mb["imad32"], "traffic": None,
                 "avg_launch_ms": kernel_s * 1e3, "points_per_launch": n_points,
                 "note": "integer-multiply bound (the north_star's IMAD roofline; neither hbm nor tensor): achieved = %d "
                         "Fq-mul/point x 588 IMAD (SURVEY 8d, a squaring counted as a multiplication) x points / CUDA-event "
                         "launch time; peak = 32-bit IMAD microbenchmark measured in this run (148 SM x 64/clk). HBM traffic "
                         "is %d B/point = %.2f GB/s, <0.1%% of %.0f GB/s" % (
                             FQMUL[key], rec_bytes, rec_bytes * n_points / kernel_s / 1e9, HBM_PEAK_GBPS),
                 "measured_imad_wide_per_s": mb["imad_wide"], "measured_fq_mul_per_s": mb["fq_mul"]}
            if prof and prof.get("dram_bytes") and prof.get("points"):
                # dram__bytes_read.sum + dram__bytes_write.sum of this kernel, scaled from the captured launch to this one
                r["traffic"] = prof["dram_bytes"] * n_points / prof["points"]
                # honest utilisation of the multiplier pipe (a squaring issues fewer slots than the multiplication it is
                # counted as in `frac`): ncu's pipe-busy figure of the committed capture of this kernel
                r["frac_pipe_busy_ncu"] = prof["fmaheavy_pct"] / 100.0 if prof.get("fmaheavy_pct") else None
                r["ncu"] = {"source": NCU_SUMMARY, "points_in_capture": prof["points"],
                            "fma_heavy_pipe_busy_pct": prof["fmaheavy_pct"], "registers": prof["registers"],
                            "local_ld_sectors": prof["local_ld_sectors"], "local_st_sectors": prof["local_st_sectors"],
                            "kernel_ms_in_capture": prof["kernel_ms_in_capture"],
                            "kernel_ms_now_same_points": kernel_s * 1e3 * prof["points"] / n_points,
                            "note": "the capture predates the last kernel change of round 2 (G2 doubling with C = Y^4 "
                                    "unreduced, squaring runs of the sqrt chain in place): the launches are shorter now at "
                                    "the same pipe utilisation (profiles/r02c_ncu_full_g2_partial.csv: 83.4 % for the G2 "
                                    "uncompressed kernel after the change, 83.7 % before)"}
            return r

        line["roofline"] = roofline("g2_comp", KERNEL_G2C, n_loc, ms_g2, 96 + 192)  # dominant kernel of the step
        line["roofline_g1"] = roofline("g1_comp", KERNEL_G1C, n_loc, ms_g1, 48 + 96)
        # ---- other kernels of the path (not the headline) ----
        extra = {}
        # the other kernels of the path, the whole-job legs and the CPU baseline are reported at N=1 only: under
        # torchrun the other ranks would sit in the closing barrier while rank 0 runs them
        if not args.no_extra and not args.no_legs and world == 1:
            def timed_leg(group, in_fmt, out_fmt, checks, din, dout, n, steps, warmup):
                for _ in range(warmup):
                    launch(group, in_fmt, din, out_fmt, dout, n, checks, 0)
                torch.cuda.synchronize()
                total = 0.0
                for _ in range(steps):
                    flush.fill_(1)
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(stream)
                    launch(group, in_fmt, din, out_fmt, dout, n, checks, 0)
                    b.record(stream)
                    b.synchronize()
                    total += a.elapsed_time(b)
                return total

            def leg(name, group, in_fmt, out_fmt, checks, n, key):
                ri = kz._ffi.lib().ptau_record_size(group, in_fmt)
                ro = kz._ffi.lib().ptau_record_size(group, out_fmt)
                gen_fmt = ZU if in_fmt == AU else in_fmt
                din = torch.empty(n * ri, dtype=torch.uint8, device=dev)
                dout = torch.empty(n * ro, dtype=torch.uint8, device=dev)
                ctx.generate_device(group, gen_fmt, 1, TAU, 0, n, din.data_ptr())
                if in_fmt == AU:
                    tmp = torch.empty_like(din)
                    ctx.convert_device(group, ZU, din.data_ptr(), AU, tmp.data_ptr(), n, 0, status.data_ptr())
                    torch.cuda.synchronize()
                    din = tmp
                t = timed_leg(group, in_fmt, out_fmt, checks, din, dout, n, 5, 3) / 5
                r = {"points": n, "ms": t, "points_per_s": n / (t / 1e3), "GBps": n * (ri + ro) / (t / 1e3) / 1e9}
                if key:
                    r["imad_frac"] = n * FQMUL[key] * IMAD_PER_FQMUL / (t / 1e3) / mb["imad32"]
                extra[name] = r
                del din, dout

            leg("g1_uncompressed_strict(configs[1])", kz.G1, ZU, AU, STRICT, 1 << 20, "g1_unc")
            leg("g2_uncompressed_strict", kz.G2, ZU, AU, STRICT, 1 << 20, "g2_unc")
            leg("g1_decompress_only", kz.G1, ZC, ZU, 0, 1 << 21, None)
            leg("g2_decompress_only", kz.G2, ZC, ZU, 0, 1 << 21, None)
            leg("g1_load_unchecked(config4)", kz.G1, AU, ML, 0, 1 << 22, None)
            leg("g1_load_validated(config4)", kz.G1, AU, ML, STRICT, 1 << 22, None)
            leg("g1_reencode_only(hbm)", kz.G1, ZU, AU, 0, 1 << 23, None)
            assert int(status.item()) == -1
            # whole preprocess-kgz job at the ceremony's real size (2^21 powers, 604 MB response), host to host
            try:
                k = 21
                n21 = 1 << k
                L = kz._ffi.lib()
                resp = kz.PinnedBuffer(L.ptau_response_size(n21))
                setup = kz.PinnedBuffer(L.ptau_setup_size(kz.VARIANT_KGZ, n21))
                off = 64
                for g, s0, cnt in ((kz.G1, 1, 2 * n21 - 1), (kz.G2, 1, n21), (kz.G1, 7, n21), (kz.G1, 11, n21), (kz.G2, 11, 1)):
                    ln = cnt * L.ptau_record_size(g, ZC)
                    ctx.generate(g, ZC, s0, TAU, 0, cnt, out=resp.array[off:off + ln])
                    off += ln
                ctx.preprocess(kz.VARIANT_KGZ, resp, n21, STRICT, out=setup)  # warm
                t0 = time.perf_counter()
                ctx.preprocess(kz.VARIANT_KGZ, resp, n21, STRICT, out=setup)
                dt = time.perf_counter() - t0
                npts = (2 * n21 - 1) + n21 + n21
                extra["preprocess_kgz_2^21_fused(host->host)"] = {
                    "points": npts, "ms": dt * 1e3, "points_per_s": npts / dt,
                    "note": "ptau_preprocess on pinned host buffers: 4.2M+2.1M compressed G1, 2.1M compressed G2, all checks"}
                # the drop-in binary on files, as a user of the reference would run it (wall clock, process start included)
                try:
                    import hashlib
                    import shutil
                    import tempfile

                    tmpd = tempfile.mkdtemp(prefix="ptau_bench_")
                    resp.array.tofile(os.path.join(tmpd, "powersoftau"))
                    exe = os.path.join(ROOT, "kzg_setup_powersoftau_b200", "bin", "preprocess-kgz")
                    hexd = hashlib.blake2b(memoryview(resp.array), digest_size=64).hexdigest()
                    runs = {}
                    for tag, flags in (("like_reference(blake2b+uncompressed_file)", ["--expect-digest", hexd]),
                                       ("no_digest_no_intermediate", ["--skip-digest", "--no-uncompressed"])):
                        walls, rcs = [], []
                        for _ in range(5):
                            for f in ("powersoftau_uncompressed", "kzg_setup"):
                                if os.path.exists(os.path.join(tmpd, f)):
                                    os.remove(os.path.join(tmpd, f))
                            t0 = time.perf_counter()
                            r = subprocess.run([exe, "--dir", tmpd, "--log2-powers", str(k)] + flags,
                                               capture_output=True, text=True)
                            walls.append(time.perf_counter() - t0)
                            rcs.append(r.returncode)
                        runs[tag] = {"wall_s_min": min(walls), "wall_s_median": statistics.median(walls), "wall_s_all": walls,
                                     "rc": max(rcs)}
                    same = open(os.path.join(tmpd, "kzg_setup"), "rb").read() == setup.array.tobytes()
                    loads, loads_v = [], []
                    for _ in range(5):
                        t0 = time.perf_counter()
                        kz.load_kzg_setup(os.path.join(tmpd, "kzg_setup"), ctx=ctx)
                        loads.append(time.perf_counter() - t0)
                    for _ in range(3):
                        t0 = time.perf_counter()
                        kz.load_kzg_setup(os.path.join(tmpd, "kzg_setup"), ctx=ctx, checks=STRICT)
                        loads_v.append(time.perf_counter() - t0)
                    extra["cli_preprocess_kgz_2^21(file->file)"] = {
                        "runs": runs, "output_equals_host_path": same, "load_kzg_setup_s_min": min(loads),
                        "load_kzg_setup_s_median": statistics.median(loads), "load_kzg_setup_validated_s_min": min(loads_v),
                        "tmpdir_fs": tmpd,
                        "note": "604 MB response file -> kzg_setup (604 MB), 8.4 M points, all checks; wall clock of the binary, "
                                "5 runs each"}
                    shutil.rmtree(tmpd, ignore_errors=True)
                except Exception as e:
                    extra["cli_preprocess_kgz_2^21(file->file)"] = {"error": repr(e)}
                resp.free()
                setup.free()
            except Exception as e:  # pinned allocation of 1.2 GB may be refused on small hosts
                extra["preprocess_kgz_2^21_fused(host->host)"] = {"error": repr(e)}
            # SURVEY 8f-4 first step: KZG10 commit (MSM) over 2^20 powers, host -> host
            pw = None
            try:
                import numpy as np

                nc = 1 << 20
                pw = ctx.convert(kz.G1, ZU, ctx.generate(kz.G1, ZU, 1, TAU, 0, nc), ML, 0)
                sc = np.random.default_rng(1).integers(0, 256, size=nc * 32, dtype=np.uint8)
                sc.reshape(nc, 32)[:, 31] &= 0x3F  # < 2^254 < r
                outp = np.zeros(104, dtype=np.uint8)
                L = kz._ffi.lib()
                for _ in range(2):
                    rcc = L.ptau_kzg_commit(ctx._h, pw.ctypes.data, sc.ctypes.data, nc, outp.ctypes.data)
                assert rcc == 0
                kms = ctx.timing()["kernel_ms"][0]
                walls = []
                for _ in range(5):
                    t0 = time.perf_counter()
                    L.ptau_kzg_commit(ctx._h, pw.ctypes.data, sc.ctypes.data, nc, outp.ctypes.data)
                    walls.append(time.perf_counter() - t0)
                extra["kzg10_commit_2^20(msm)"] = {"points": nc, "kernel_ms": kms, "points_per_s_kernels": nc / (kms / 1e3),
                                                   "wall_ms_min_host_powers": 1e3 * min(walls),
                                                   "launches": ctx.timing()["kernel_launches"],
                                                   "note": "bucket method, signed windows, counting sort by atomics"}
                try:
                    res = kz.ResidentPoints(ctx, pw.reshape(nc, 104))
                    walls = []
                    for _ in range(6):
                        t0 = time.perf_counter()
                        rcc = L.ptau_kzg_commit_resident(ctx._h, res._h, sc.ctypes.data, nc, outp.ctypes.data)
                        walls.append(time.perf_counter() - t0)
                        assert rcc == 0
                    walls = walls[1:]
                    extra["kzg10_commit_2^20(msm)"]["wall_ms_min_resident_powers"] = 1e3 * min(walls)
                except Exception as e:
                    extra["kzg10_commit_2^20(msm)"]["resident_error"] = repr(e)
            except Exception as e:
                extra["kzg10_commit_2^20(msm)"] = {"error": repr(e)}
            # SURVEY 8f-4: KZG10::check (two Miller loops + one final exponentiation per opening)
            try:
                import numpy as np

                nk = 148 * 256
                pwk = pw.reshape(-1, 104)[:32]
                g2p = ctx.convert(kz.G2, ZU, ctx.generate(kz.G2, ZU, 1, TAU, 0, 2), ML, 0).reshape(2, 200)
                vk = kz.VerifierKey(g=pwk[0], gamma_g=pwk[5], h=g2p[0], beta_h=g2p[1])
                pws = kz.Powers(powers_of_g=pwk, powers_of_gamma_g=pwk[:1])
                poly = [int(x) for x in np.random.default_rng(2).integers(1, 1 << 62, size=16)]
                comm = kz.KZG10.commit(pws, poly, ctx=ctx)
                val, prf, _ = kz.KZG10.open(pws, poly, 12345, ctx=ctx)
                for _ in range(2):
                    okv = kz.KZG10.check_many(vk, np.tile(comm, (nk, 1)), [12345] * nk, [val] * nk, np.tile(prf, (nk, 1)), ctx=ctx)
                assert okv.all()
                kms = ctx.timing()["kernel_ms"][0]
                extra["kzg10_check_37888(pairings, kernel only)"] = {
                    "openings": nk, "ms": kms, "openings_per_s": nk / (kms / 1e3),
                    "note": "per opening: [v]g and [z]h scalar multiplications, two Miller loops, one final exponentiation"}
            except Exception as e:
                extra["kzg10_check_37888(pairings, kernel only)"] = {"error": repr(e)}
            hb = extra["g1_reencode_only(hbm)"]
            line["roofline_hbm"] = {"bound": "hbm", "kernel": "convert_kernel<1, 1, 3, 0> zcash->ark re-encode only (no checks)",
                                    "achieved": hb["GBps"], "peak": HBM_PEAK_GBPS, "unit": "GB/s",
                                    "frac": hb["GBps"] / HBM_PEAK_GBPS, "traffic": None, "peak_source": HBM_PEAK_SOURCE}
        line["extra"] = extra
        # ---- CPU baseline: the reference's algorithms on this box's host cores (rank 0, N=1 only) ----
        threads = os.cpu_count() or 1
        try:
            if world > 1:
                raise RuntimeError("cpu_baseline is measured at N=1 only")
            if args.no_extra or args.no_legs:
                raise RuntimeError("--no-extra / --no-legs")
            rate1, _, _ = cpu_config3(1 << 8, 1)
            n_s = 1 << 12  # probe (large enough to keep every thread busy), then size the sample to 10-20 s of host work
            rate, dt, _ = cpu_config3(n_s, threads)
            while n_s < N and 2 * (2 * n_s) / rate <= 20.0:
                n_s *= 2
            rate, dt, inputs = cpu_config3(n_s, threads)
            line["cpu_baseline"] = {
                "value": rate, "unit": "points/s", "cores": threads, "kind": "port",
                "sample": "first %d compressed G1 + first %d compressed G2 points of the workload, C restatement of the "
                          "reference's algorithms (6x64 Montgomery, Algorithm-9 Fq2 sqrt, r-multiplication subgroup check), "
                          "%d threads, %.1f s" % (n_s, n_s, threads, dt),
                "single_core_value": rate1,
                "same_code_with_gpu_predicates_value": cpu_config3(n_s, threads, True, inputs)[0],
            }
        except Exception as e:  # the oracle is optional for the product, never for correctness claims
            line["cpu_baseline"] = {"value": None, "unit": "points/s", "cores": threads, "kind": "port",
                                    "sample": "not measured in this run: %s" % (e,)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
