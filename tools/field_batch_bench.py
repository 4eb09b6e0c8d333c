"""Field images of a batch of solutions on one GPU: field_at_position_batch against a loop of
Solution.field_at_position, and the multi-set SCB_BS_Z pair sum in isolation.

End to end: a solve_batch vortex scan of the 20k-vertex C2 square (configs.c2_square), B = 16, 64, 256 entries with
one vortex each, evaluated on a 256 x 256 grid at z = 1 um over the film (B = 64 also on a 1000 x 1000 grid).
Device-synchronised wall time, median of --reps after one warm-up call of each shape; the host staging part of the
batch call (checks, target scaling, current densities into pinned memory, applied field) is timed on its own; the
largest difference between batch and loop in the same run.

Kernel rows: scb_biot_savart(SCB_BS_Z) with 8 ... 128 sets on 65k and 1M targets x the film's sources, CUDA events,
median of --reps: one call with all sets, the same sets as 8-set calls, and as one-set calls (the per-solution
path).  The L2 is not overwritten between launches: the operands (< 50 MB) stay L2-resident either way and the
pair sum is bound by fp64 arithmetic, not by memory.  The GPU name and power limit are read in the same run.
Prints one JSON object and writes it to --out.

    python tools/field_batch_bench.py --out field_batch.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    import torch

    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except OSError as e:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def time_call(fn, reps):
    import torch

    fn()  # warm-up of this shape
    torch.cuda.synchronize()
    ts, out = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), ts, out


def grid(k, z):
    x, y = np.meshgrid(np.linspace(-5.5, 5.5, k), np.linspace(-5.5, 5.5, k))
    return np.column_stack([x.ravel(), y.ravel()]), z


def end_to_end(sc, model, B, k, reps):
    from superscreen_b200 import solution

    rng = np.random.default_rng(B)
    vortices = [[sc.Vortex(x=float(x), y=float(y), film="film")] for x, y in rng.uniform(-4.5, 4.5, (B, 2))]
    sols = [s[-1] for s in sc.solve_batch(model=model, applied_fields=[None] * B, vortices=vortices, last_only=True)]
    positions, z = grid(k, 1.0)
    t_batch, ts_batch, out = time_call(
        lambda: sc.field_at_position_batch(sols, positions, zs=z, with_units=False), reps)
    t_stage, ts_stage, _ = time_call(lambda: solution._stage_field_batch(sols, positions, z, "linear", None), reps)
    t_loop, ts_loop, ref = time_call(
        lambda: np.stack([s.field_at_position(positions, zs=z, with_units=False) for s in sols]), reps)
    row = dict(B=B, grid=f"{k}x{k}", targets=k * k, batch_s=t_batch, batch_host_staging_s=t_stage, loop_s=t_loop,
               speedup=t_loop / t_batch, batch_reps_s=ts_batch, batch_host_staging_reps_s=ts_stage,
               loop_reps_s=ts_loop, bit_identical=bool(np.array_equal(out, ref)),
               max_abs_diff=float(np.abs(out - ref).max()), max_abs_field=float(np.abs(ref).max()),
               entries_differ=bool(not np.array_equal(ref[0], ref[-1])))
    print(json.dumps(row), flush=True)
    return row


def kernel_rows(sc, device, sets, targets, reps):
    import torch

    from superscreen_b200 import _lib

    L = _lib.lib()
    mesh = device.meshes["film"]
    n = len(mesh.sites)
    z0 = device.layers[device.films["film"].layer].z0
    src = torch.as_tensor(np.column_stack([mesh.sites, np.full(n, z0)]) * 1e-6).cuda().contiguous()
    area = torch.as_tensor(np.asarray(mesh.vertex_areas) * 1e-12).cuda()
    rng = np.random.default_rng(0)
    rows = []
    for m in targets:
        k = int(round(np.sqrt(m)))
        xy, _ = grid(k, 1.0)
        tgt = torch.as_tensor(np.column_stack([xy, np.ones(len(xy))]) * 1e-6).cuda().contiguous()
        mm = len(xy)
        for nsets in sets:
            J = torch.as_tensor(rng.standard_normal((nsets, n, 2))).cuda()
            out = torch.empty((nsets, mm), dtype=torch.float64, device="cuda")

            def launch(per_call):
                for s0 in range(0, nsets, per_call):
                    c = min(per_call, nsets - s0)
                    _lib.check(L.scb_biot_savart(1, mm, _lib.ptr(tgt), n, _lib.ptr(src), _lib.ptr(area),
                                                 _lib.ptr(J[s0:s0 + c]), 0.0, 1e-7, c, _lib.ptr(out[s0:s0 + c]),
                                                 _lib.stream_ptr()))

            row = dict(targets=mm, sources=n, sets=nsets)
            results = {}
            for label, per_call in (("one_call", nsets), ("8_set_calls", 8), ("1_set_calls", 1)):
                launch(per_call)  # warm-up
                torch.cuda.synchronize()
                ts = []
                for _ in range(reps):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    launch(per_call)
                    e1.record()
                    e1.synchronize()
                    ts.append(e0.elapsed_time(e1) * 1e-3)
                t = float(np.median(ts))
                results[label] = out.clone()
                row[f"{label}_s"] = t
                row[f"{label}_pair_sets_per_s"] = mm * n * nsets / t
            row["one_call_vs_1_set_calls_speedup"] = row["1_set_calls_s"] / row["one_call_s"]
            row["one_call_vs_8_set_calls_speedup"] = row["8_set_calls_s"] / row["one_call_s"]
            row["bit_identical_across_variants"] = bool(torch.equal(results["one_call"], results["8_set_calls"])
                                                        and torch.equal(results["one_call"], results["1_set_calls"]))
            rows.append(row)
            print(json.dumps(row), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--batches", type=int, nargs="+", default=[16, 64, 256])
    ap.add_argument("--large-grid-batch", type=int, default=64)
    ap.add_argument("--sets", type=int, nargs="+", default=[8, 16, 32, 64, 128])
    ap.add_argument("--targets", type=int, nargs="+", default=[65536, 1000000])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import superscreen_b200 as sc
    from superscreen_b200 import configs

    device = configs.c2_square()
    model = sc.factorize_model(device=device, current_units="uA")
    scans = [end_to_end(sc, model, B, 256, args.reps) for B in args.batches]
    if args.large_grid_batch:
        scans.append(end_to_end(sc, model, args.large_grid_batch, 1000, args.reps))
    result = dict(gpu=gpu_info(), vertices=len(device.meshes["film"].sites), reps=args.reps,
                  timing="end to end: device-synchronised wall time, median of --reps after one warm-up call of each "
                         "shape; kernel rows: CUDA events, median of --reps after one warm-up launch sequence",
                  l2_overwritten_between_launches=False,
                  scans=scans, kernel=kernel_rows(sc, device, args.sets, args.targets, args.reps))
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
