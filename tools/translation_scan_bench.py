"""Scanning-SQUID position scans on one GPU: solve_batch(translations=...) against one solve per position.

Workload: the IBM "small" susceptometer (configs.ibm_susceptometer, 5 films of ~4k vertices on layers W2, W1,
BE) over a 20k-vertex sample square on its own layer 0.5 um below, iterations=5, 1 mA in ``fc_center``;
M = pickup-loop fluxoid / field-coil current.

  kernel: scb_film_coupling_translated in pair.sets/s against the one-set scb_film_coupling pair rate, for the
          sample film and for the field-coil film as targets (the packed sources of all films), CUDA events
          over a window of >= 1 s after warm-up calls;
  scan:   for B = 16, 64, 256 positions of the SQUID layers (an in-plane raster): one solve_batch call plus
          the pickup fluxoid of every entry (the lazy builds of the moved devices timed separately),
          against a loop of factorize + solve on the moved device over the first --loop positions.
          Device-synchronised wall time.  The largest |dM| between batch and loop for every position timed
          both ways.

The GPU name and power limit are read in the same run.  Prints one JSON object and writes it to --out.

    python tools/translation_scan_bench.py [--out profiles/r08_translation_scan.json]
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
SQUID_LAYERS = ("W2", "W1", "BE")


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


def scan_device(sc, n_squid, n_sample, h=0.5):
    from superscreen_b200 import configs
    from superscreen_b200.geometry import box
    from superscreen_b200.synthetic import make_mesh

    squid, rings, meshes = configs.ibm_susceptometer("small", n_squid, attach_meshes=False)
    sample = sc.Polygon("sample", layer="sample", points=box(10.0, 10.0, points=4, center=(0.5, -1.0)))
    device = sc.Device("scan", layers=list(squid.layers.values()) + [sc.Layer("sample", Lambda=0.08, z0=-h)],
                       films=list(squid.films.values()) + [sample], holes=list(squid.holes.values()),
                       length_units="um")
    meshes = dict(meshes, sample=make_mesh(box(10.8, 10.8, points=4, center=(0.5, -1.0)), target_vertices=n_sample,
                                           embedded=[sample.points[:-1]], seed=11))
    device.set_meshes(meshes)
    return device, rings["pl_center"]


def sync():
    import torch

    torch.cuda.synchronize()


def rate(fn, pairs, min_window=1.0):
    """pairs / s of fn() over a window of >= min_window s (CUDA events), after 3 warm-up calls."""
    import torch

    for _ in range(3):
        fn()
    sync()
    reps = 1
    while True:
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for _ in range(reps):
            fn()
        stop.record()
        stop.synchronize()
        dt = start.elapsed_time(stop) * 1e-3
        if dt >= min_window:
            return {"pairs_per_s": pairs * reps / dt, "calls": reps, "window_s": dt}
        reps = max(reps * 2, int(reps * 1.2 * min_window / max(dt, 1e-6)))


def kernel_rates(sc, device, nsets_list):
    import torch

    from superscreen_b200 import _lib
    from superscreen_b200.parallel import Comm, FilmLayout, film_owners
    from superscreen_b200.solver.solve import _packed_sources

    L = _lib.lib()
    model = sc.factorize_model(device=device, current_units="uA")
    names = list(device.films)
    layout = FilmLayout(names, {f: len(device.meshes[f].sites) for f in names}, film_owners(names, Comm()), 1)
    z0s = {f: float(device.layers[device.films[f].layer].z0) for f in names}
    dev = torch.device("cuda:0")
    src, area, film = _packed_sources(model, layout, z0s, dev)
    rng = np.random.default_rng(0)
    out = {}
    for dst in ("sample", "fc"):
        d = device.meshes[dst]._data
        lo, hi = layout.rows(dst)
        pairs = d.n * (layout.total - (hi - lo))
        row = {"targets": d.n, "sources": layout.total - (hi - lo)}
        J1 = torch.as_tensor(rng.standard_normal((layout.total, 1, 2))).to(dev)
        o1 = torch.empty(d.n, dtype=torch.float64, device=dev)

        def one():
            _lib.check(L.scb_film_coupling(d.n, _lib.ptr(d.sites), z0s[dst], layout.total, _lib.ptr(src),
                                           _lib.ptr(area), _lib.ptr(J1), lo, hi, 1.0, 1, _lib.ptr(o1),
                                           _lib.stream_ptr()))

        row["one_set_coupling"] = rate(one, pairs)
        for nsets in nsets_list:
            J = torch.as_tensor(rng.standard_normal((layout.total, nsets, 2))).to(dev)
            S = torch.as_tensor(rng.uniform(-1.0, 1.0, (nsets, len(names), 3))).to(dev)
            o = torch.empty((d.n, nsets), dtype=torch.float64, device=dev)

            def translated():
                _lib.check(L.scb_film_coupling_translated(
                    d.n, _lib.ptr(d.sites), z0s[dst], layout.total, _lib.ptr(src), _lib.ptr(area), _lib.ptr(J),
                    lo, hi, 1.0, nsets, names.index(dst), _lib.ptr(film), len(names), _lib.ptr(S), _lib.ptr(o),
                    _lib.stream_ptr()))

            r = rate(translated, pairs * nsets)
            r["vs_one_set"] = r["pairs_per_s"] / row["one_set_coupling"]["pairs_per_s"]
            row[f"translated_nsets_{nsets}"] = r
        out[dst] = row
        print(dst, json.dumps(row), flush=True)
    return out


def M_of(solution, ring, dxy):
    return sum(solution.hole_fluxoid("pl_center", points=ring + np.asarray(dxy), with_units=False)) / 1e-3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_translation_scan.json"))
    ap.add_argument("--squid-vertices", type=int, default=4000)
    ap.add_argument("--sample-vertices", type=int, default=20000)
    ap.add_argument("--batches", default="16,64,256")
    ap.add_argument("--loop", type=int, default=4, help="positions solved one by one")
    ap.add_argument("--nsets", default="1,2,16,64")
    args = ap.parse_args()
    sys.path.insert(0, ROOT)
    import torch

    import superscreen_b200 as sc
    from superscreen_b200.solver.solve import _translated_device

    torch.cuda.set_device(0)
    result = {"gpu": gpu_info(), "workload": {"squid": "configs.ibm_susceptometer('small')",
                                              "squid_vertices_per_film": args.squid_vertices,
                                              "sample_vertices": args.sample_vertices, "sample_gap_um": 0.5,
                                              "iterations": 5, "fc_center_current": "1 mA"}}
    device, ring = scan_device(sc, args.squid_vertices, args.sample_vertices)
    result["workload"]["vertices"] = {f: len(m.sites) for f, m in device.meshes.items()}
    result["kernel"] = kernel_rates(sc, device, [int(b) for b in args.nsets.split(",")])

    Bs = [int(b) for b in args.batches.split(",")]
    side = int(np.ceil(np.sqrt(max(Bs))))
    xs = np.linspace(-2.0, 2.0, side)
    raster = [(float(x), float(y)) for y in np.linspace(-1.5, 1.5, side) for x in xs]
    rng = np.random.default_rng(1)
    raster = [raster[k] for k in rng.permutation(len(raster))]  # every prefix spans the raster
    moves = [{layer: (x, y, 0.0) for layer in SQUID_LAYERS} for x, y in raster]

    # one position at a time: factorize + solve on the moved device (the first --loop positions)
    loop_M, loop_s = [], []
    for b in range(args.loop + 1):  # (the first call warms up)
        sync()
        t0 = time.perf_counter()
        moved = _translated_device(device, moves[b])
        sol = sc.solve(moved, circulating_currents={"fc_center": "1 mA"}, current_units="uA", iterations=5)[-1]
        M = M_of(sol, ring, raster[b])
        sync()
        if b > 0 or args.loop == 0:
            loop_s.append(time.perf_counter() - t0)
        loop_M.append(M)
    loop_M = loop_M[:args.loop] if args.loop else []
    result["loop"] = {"positions": args.loop, "per_position_s": float(np.median(loop_s)) if loop_s else None,
                      "per_position_all_s": loop_s}
    print("loop", json.dumps(result["loop"]), flush=True)

    sync()
    t0 = time.perf_counter()
    model = sc.factorize_model(device=device, current_units="uA", circulating_currents={"fc_center": "1 mA"})
    model.finish_checks()
    sync()
    result["factorize_s"] = time.perf_counter() - t0
    scans = {}
    for warm in (True, False):
        for B in Bs:
            sync()
            t0 = time.perf_counter()
            sols = sc.solve_batch(model=model, applied_fields=[None] * B, translations=moves[:B], iterations=5,
                                  last_only=True)
            sync()
            t_solve = time.perf_counter() - t0
            t0 = time.perf_counter()
            for s in sols:
                s[-1].device  # noqa: B018  (the lazy build of the moved device)
            t_build = time.perf_counter() - t0
            t0 = time.perf_counter()
            Ms = [M_of(s[-1], ring, raster[b]) for b, s in enumerate(sols)]
            sync()
            t_flux = time.perf_counter() - t0
            if warm:
                continue
            n_cmp = min(B, len(loop_M))
            dM = [abs(Ms[b] - loop_M[b]) for b in range(n_cmp)]
            row = {"solve_batch_s": t_solve, "device_builds_s": t_build, "fluxoids_s": t_flux,
                   "per_position_s": (t_solve + t_build + t_flux) / B,
                   "loop_per_position_s": result["loop"]["per_position_s"],
                   "speedup_vs_loop_per_position": (result["loop"]["per_position_s"] * B / (t_solve + t_build + t_flux)
                                                    if loop_s else None),
                   "compared_positions": n_cmp, "max_abs_dM_Phi0_per_A": max(dM) if dM else None,
                   "max_rel_dM": max(d / abs(loop_M[b]) for b, d in enumerate(dM)) if dM else None,
                   "M_range_Phi0_per_A": [min(Ms), max(Ms)]}
            scans[str(B)] = row
            print("B", B, json.dumps(row), flush=True)
    result["scan"] = scans
    result["loop_M_Phi0_per_A"] = loop_M
    text = json.dumps(result, indent=1)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
