"""Vortex-position scans on one GPU: solve_batch(vortices=...) against serial set_vortices + solve calls.

Two workloads:
  c2: the 20k-vertex C2 square (configs.c2_square), one vortex per entry anywhere in the film;
  c3: the C3 susceptometer (configs.c3_susceptometer), iterations=5, 1 mA in the field coil, one vortex per
      entry in the pickup-loop film "pl".
For every scan size B (default 16, 64, 256): one solve_batch call with B entries against B serial calls
``model.set_vortices([v_b]); solve(model=model)`` on the same factorization.  Device-synchronised wall time,
median of --reps after one warm-up call of each shape; the largest rel-L2 between batch and serial results
(stream, self field) of the same run.

With --parent-root DIR (a checkout of an earlier version of the package with its library built), the serial
scan also runs with that version's code, in a child process, on the same seeded meshes and positions; its
results are compared with this version's serial results.  The GPU name and power limit are read in the same
run.  Prints one JSON object and writes it to --out.

    python tools/vortex_batch_bench.py --out vortex_batch.json [--parent-root DIR]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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


def workload(sc, case):
    """-> (device, factorize_model kwargs, vortex film, iterations, position sampler)"""
    from superscreen_b200 import configs

    if case == "c2":
        device = configs.c2_square()

        def sample(rng, B):
            return rng.uniform(-4.5, 4.5, (B, 2))

        return device, {}, "film", 0, sample
    device, _ = configs.c3_susceptometer()

    def sample(rng, B):  # the pickup loop: r 0.5 - 1
        r, th = rng.uniform(0.6, 0.9, B), rng.uniform(0.0, 2 * np.pi, B)
        return np.column_stack([r * np.cos(th), r * np.sin(th)])

    return device, {"circulating_currents": {"fc_center": "1 mA"}}, "pl", 5, sample


def scan_vortices(sc, case, film, sample, B):
    xy = sample(np.random.default_rng(1000 * (case == "c3") + B), B)
    return [sc.Vortex(x=float(x), y=float(y), film=film) for x, y in xy]


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


def rel_l2(a, b):
    nb = np.linalg.norm(b)
    return float(np.linalg.norm(a - b) / (nb if nb > 0 else 1.0))


def serial_scan(sc, model, vortices, iterations):
    out = []
    for v in vortices:
        model.set_vortices([v])
        out.append(sc.solve(model=model, iterations=iterations)[-1])
    model.set_vortices([])
    return out


def stacked(sols, film, attr):
    return np.stack([getattr(s.film_solutions[film], attr) for s in sols])


def serial_only(args):
    """Child-process mode: the serial scans with the package found at --root; outputs to --dump."""
    import superscreen_b200 as sc

    device, kw, film, iterations, sample = workload(sc, args.case)
    model = sc.factorize_model(device=device, current_units="uA", **kw)
    rows, dump = [], {}
    for B in args.batches:
        vortices = scan_vortices(sc, args.case, film, sample, B)
        t, ts, sols = time_call(lambda: serial_scan(sc, model, vortices, iterations), args.reps)
        rows.append(dict(B=B, serial_s=t, serial_reps_s=ts))
        dump[f"stream_{B}"] = stacked(sols, film, "stream")
        dump[f"self_field_{B}"] = stacked(sols, film, "self_field")
    np.savez(args.dump, **dump)
    print(json.dumps(rows))


def case_section(sc, case, batches, reps, parent_root):
    device, kw, film, iterations, sample = workload(sc, case)
    model = sc.factorize_model(device=device, current_units="uA", **kw)
    rows = []
    parent = None
    if parent_root:
        with tempfile.TemporaryDirectory() as tmp:
            dump = os.path.join(tmp, "parent.npz")
            cmd = [sys.executable, os.path.abspath(__file__), "--serial-only", "--root", parent_root, "--case", case,
                   "--reps", str(reps), "--dump", dump, "--batches", *map(str, batches)]
            p = subprocess.run(cmd, capture_output=True, text=True)
            if p.returncode != 0:
                raise SystemExit(f"parent serial scan failed:\n{p.stdout}\n{p.stderr}")
            parent = dict(rows={r["B"]: r for r in json.loads(p.stdout.strip().splitlines()[-1])},
                          data=dict(np.load(dump)))
    for B in batches:
        vortices = scan_vortices(sc, case, film, sample, B)
        t_batch, ts_batch, rb = time_call(
            lambda: sc.solve_batch(model=model, applied_fields=[None] * B, vortices=[[v] for v in vortices],
                                   iterations=iterations, last_only=True), reps)
        t_serial, ts_serial, rs = time_call(lambda: serial_scan(sc, model, vortices, iterations), reps)
        b_stream, b_self = stacked([r[-1] for r in rb], film, "stream"), stacked([r[-1] for r in rb], film, "self_field")
        s_stream, s_self = stacked(rs, film, "stream"), stacked(rs, film, "self_field")
        norms = np.linalg.norm(b_stream, axis=1)
        row = dict(B=B, solve_batch_s=t_batch, serial_s=t_serial, speedup_vs_serial=t_serial / t_batch,
                   solve_batch_reps_s=ts_batch, serial_reps_s=ts_serial,
                   # what is compared: B entries of n values each, their norms, and whether entries differ
                   compared_values_per_entry=int(b_stream.shape[1]),
                   stream_norm_min_max=[float(norms.min()), float(norms.max())],
                   entries_differ=bool(not np.array_equal(b_stream[0], b_stream[-1])),
                   max_rel_l2_batch_vs_serial=max(max(rel_l2(b_stream[b], s_stream[b]), rel_l2(b_self[b], s_self[b]))
                                                  for b in range(B)),
                   max_abs_diff_stream_batch_vs_serial=float(np.abs(b_stream - s_stream).max()))
        if parent is not None:
            pr = parent["rows"][B]
            p_stream, p_self = parent["data"][f"stream_{B}"], parent["data"][f"self_field_{B}"]
            row.update(parent_serial_s=pr["serial_s"], parent_serial_reps_s=pr["serial_reps_s"],
                       speedup_serial_vs_parent_serial=pr["serial_s"] / t_serial,
                       speedup_batch_vs_parent_serial=pr["serial_s"] / t_batch,
                       max_rel_l2_serial_vs_parent_serial=max(
                           max(rel_l2(s_stream[b], p_stream[b]), rel_l2(s_self[b], p_self[b])) for b in range(B)),
                       max_abs_diff_stream_serial_vs_parent_serial=float(np.abs(s_stream - p_stream).max()))
        rows.append(row)
        print(json.dumps(row), flush=True)
    sizes = {name: len(device.meshes[name].sites) for name in device.films}
    return dict(vertices=sizes, vortex_film=film, iterations=iterations, scans=rows)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--batches", type=int, nargs="+", default=[16, 64, 256])
    ap.add_argument("--cases", nargs="+", default=["c2", "c3"], choices=["c2", "c3"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--parent-root", default=None)
    ap.add_argument("--out", default=None)
    # (child-process mode, see serial_only)
    ap.add_argument("--serial-only", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--root", default=ROOT, help=argparse.SUPPRESS)
    ap.add_argument("--case", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--dump", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.root))
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    if args.serial_only:
        return serial_only(args)
    import superscreen_b200 as sc

    result = dict(gpu=gpu_info(), timing="device-synchronised wall time per scan, median of --reps after one "
                                        "warm-up call of each shape; parent serial scans run in a child process "
                                        "before this version's scans of the same workload",
                  reps=args.reps)
    for case in args.cases:
        result[case] = case_section(sc, case, args.batches, args.reps,
                                    os.path.abspath(args.parent_root) if args.parent_root else None)
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
