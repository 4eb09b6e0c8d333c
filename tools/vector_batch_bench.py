"""Vector field and vector potential images of a batch of solutions on one GPU: screening_field_at_position_batch
(vector=True) and vector_potential_at_position_batch against loops of the per-solution methods, and the multi-set
SCB_BS_VECTOR / SCB_BS_VECTOR_POTENTIAL pair sums in isolation.

End to end: a solve_batch vortex scan of the 20k-vertex C2 square (configs.c2_square), B = 16, 64, 256 entries with
one vortex each, evaluated on a 256 x 256 grid at z = 1 um over the film (B = 64 also on a 1000 x 1000 grid).
Device-synchronised wall time, median of --reps after one warm-up call of each shape; whether every batch row has the
bits of its loop row, checked in the same run.

Kernel rows: scb_biot_savart(SCB_BS_VECTOR, SCB_BS_VECTOR_POTENTIAL) with 8 ... 128 sets on 65k and 1M targets x the
film's sources, CUDA events, median of --reps after one warm-up launch sequence: one call with all sets (8-set
passes), the same sets as 4-set calls (4-set passes) and as one-set calls (the per-solution path).  The L2 is not
overwritten between launches: the operands (< 50 MB) stay L2-resident either way and the pair sum is bound by fp64
arithmetic, not by memory.  The GPU name and power limit are read in the same run.  Prints one JSON object and writes
it to --out.

    python tools/vector_batch_bench.py --out profiles/r09_vector_batch.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from field_batch_bench import gpu_info, grid, time_call  # noqa: E402

KINDS = {"vector": 2, "vector_potential": 3}


def end_to_end(sc, model, B, k, reps):
    rng = np.random.default_rng(B)
    vortices = [[sc.Vortex(x=float(x), y=float(y), film="film")] for x, y in rng.uniform(-4.5, 4.5, (B, 2))]
    sols = [s[-1] for s in sc.solve_batch(model=model, applied_fields=[None] * B, vortices=vortices, last_only=True)]
    positions, z = grid(k, 1.0)
    calls = {
        "vector": (lambda: sc.screening_field_at_position_batch(sols, positions, zs=z, vector=True, with_units=False),
                   lambda: np.stack([s.screening_field_at_position(positions, zs=z, vector=True, with_units=False)
                                     for s in sols])),
        "vector_potential": (lambda: sc.vector_potential_at_position_batch(sols, positions, zs=z, with_units=False),
                             lambda: np.stack([s.vector_potential_at_position(positions, zs=z, with_units=False)
                                               for s in sols])),
    }
    rows = []
    for kind, (batch, loop) in calls.items():
        t_batch, ts_batch, out = time_call(batch, reps)
        t_loop, ts_loop, ref = time_call(loop, reps)
        row = dict(kind=kind, B=B, grid=f"{k}x{k}", targets=k * k, batch_s=t_batch, loop_s=t_loop,
                   speedup=t_loop / t_batch, batch_reps_s=ts_batch, loop_reps_s=ts_loop,
                   bit_identical=bool(np.array_equal(out, ref)), max_abs_diff=float(np.abs(out - ref).max()),
                   max_abs_value=float(np.abs(ref).max()), entries_differ=bool(not np.array_equal(ref[0], ref[-1])))
        print(json.dumps(row), flush=True)
        rows.append(row)
        del out, ref
    return rows


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
    for kind, code in KINDS.items():
        nc = 3 if code == 2 else 2
        for m in targets:
            k = int(round(np.sqrt(m)))
            xy, _ = grid(k, 1.0)
            tgt = torch.as_tensor(np.column_stack([xy, np.ones(len(xy))]) * 1e-6).cuda().contiguous()
            mm = len(xy)
            for nsets in sets:
                J = torch.as_tensor(rng.standard_normal((nsets, n, 2))).cuda()
                out = torch.empty((nsets, mm, nc), dtype=torch.float64, device="cuda")

                def launch(per_call):
                    for s0 in range(0, nsets, per_call):
                        c = min(per_call, nsets - s0)
                        _lib.check(L.scb_biot_savart(code, mm, _lib.ptr(tgt), n, _lib.ptr(src), _lib.ptr(area),
                                                     _lib.ptr(J[s0:s0 + c]), 0.0, 1e-7, c, _lib.ptr(out[s0:s0 + c]),
                                                     _lib.stream_ptr()))

                row = dict(kind=kind, targets=mm, sources=n, sets=nsets)
                results = {}
                for label, per_call in (("one_call", nsets), ("4_set_calls", 4), ("1_set_calls", 1)):
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
                row["one_call_vs_4_set_calls_speedup"] = row["4_set_calls_s"] / row["one_call_s"]
                row["bit_identical_across_variants"] = bool(torch.equal(results["one_call"], results["4_set_calls"])
                                                            and torch.equal(results["one_call"], results["1_set_calls"]))
                rows.append(row)
                print(json.dumps(row), flush=True)
                del J, out, results
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
    scans = [row for B in args.batches for row in end_to_end(sc, model, B, 256, args.reps)]
    if args.large_grid_batch:
        scans += end_to_end(sc, model, args.large_grid_batch, 1000, args.reps)
    result = dict(gpu=gpu_info(), vertices=len(device.meshes["film"].sites), reps=args.reps,
                  timing="end to end: device-synchronised wall time, median of --reps after one warm-up call of each "
                         "shape; kernel rows: CUDA events, median of --reps after one warm-up launch sequence",
                  l2_overwritten_between_launches=False,
                  all_batch_rows_bit_identical_to_loop_rows=all(r["bit_identical"] for r in scans),
                  scans=scans, kernel=kernel_rows(sc, device, args.sets, args.targets, args.reps))
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
