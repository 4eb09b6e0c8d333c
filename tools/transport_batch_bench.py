"""Batched transport-terminal solves and the within-film field kernel on one GPU.

A 20k-vertex bar with one hole and source / drain terminals (meshed by Device.make_mesh):
  1. solve_batch with B distinct terminal currents against B serial solve calls sharing one
     factorization (device-synchronised wall time, median of --reps after one warm-up call each),
     with the rel-L2 between the two results;
  2. scb_biot_savart_within_film (its DMMA kernel for every full pass of 64 sets; fewer sets take the
     CUDA-core passes) against the same sum in 8-set CUDA-core passes (scb_film_coupling with every
     source in the target plane), CUDA events per launch, L2 overwritten before every launch, median;
     pairs * sets / s;
  3. the GPU name and power limit, read in the same run.
Prints one JSON object and writes it to --out.

    python tools/transport_batch_bench.py --out transport_batch.json
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


def bar_device(sc, target_vertices):
    from superscreen_b200.geometry import box, circle

    terminals = {"bar": [sc.Polygon("source", points=box(0.2, 2.0, points=4, center=(-4.0, 0.0))),
                         sc.Polygon("drain", points=box(0.2, 2.0, points=4, center=(4.0, 0.0)))]}
    device = sc.Device("bar", layers=[sc.Layer("layer", Lambda=0.4, z0=0.0)],
                       films=[sc.Polygon("bar", layer="layer", points=box(8.0, 3.0, points=400))],
                       holes=[sc.Polygon("hole", layer="layer", points=circle(0.6, 48, center=(0.5, 0.2)))],
                       terminals=terminals)
    device.make_mesh(min_points=target_vertices, seed=3)
    return device


def rel_l2(a, b):
    nb = np.linalg.norm(b)
    return float(np.linalg.norm(a - b) / (nb if nb > 0 else 1.0))


def time_call(fn, reps):
    import torch

    fn()  # warm-up
    torch.cuda.synchronize()
    ts = []
    out = None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), out


def solve_section(sc, device, batches, reps):
    model = sc.factorize_model(device=device, current_units="uA")
    info = model.film_info["bar"]
    rng = np.random.default_rng(0)
    rows = []
    for B in batches:
        currents = [float(x) for x in rng.uniform(-50.0, 50.0, B)]
        term = [{"bar": {"source": I, "drain": -I}} for I in currents]
        field = sc.ConstantField(0.05)

        def batched():
            return sc.solve_batch(model=model, applied_fields=[field] * B, terminal_currents=term)

        def serial():
            # B solve calls against the one factorization (the model's terminal currents set per call)
            out = []
            for tc in term:
                info.terminal_currents = tc["bar"]
                out.append(sc.solve(model=model, applied_field=field))
            info.terminal_currents = None
            return out

        t_batch, rb = time_call(batched, reps)
        t_serial, rs = time_call(serial, reps)
        err = max(max(rel_l2(rb[b][0].film_solutions["bar"].stream, rs[b][0].film_solutions["bar"].stream),
                      rel_l2(rb[b][0].film_solutions["bar"].self_field, rs[b][0].film_solutions["bar"].self_field))
                  for b in range(B))
        rows.append(dict(B=B, solve_batch_s=t_batch, serial_solves_s=t_serial, speedup=t_serial / t_batch,
                         max_rel_l2_stream_self_field=err))
        print(json.dumps(rows[-1]), flush=True)
    return rows


def kernel_section(device, sets, launches):
    import torch

    from superscreen_b200 import _lib

    L = _lib.lib()
    d = device.meshes["bar"]._data
    m, n = d.n, d.m
    rng = np.random.default_rng(1)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    src3 = torch.zeros(n, 3, dtype=torch.float64, device="cuda")
    src3[:, :2] = d.t["centroids"]
    pf = 1.0 / (4.0 * np.pi)
    rows = []
    for ns in sets:
        J = torch.as_tensor(rng.standard_normal((n, ns, 2))).cuda()
        out_mma = torch.empty(m, ns, dtype=torch.float64, device="cuda")
        out_cc = torch.empty(m, ns, dtype=torch.float64, device="cuda")

        def dmma():
            _lib.check(L.scb_biot_savart_within_film(m, _lib.ptr(d.sites), n, _lib.ptr(d.t["centroids"]),
                                                     _lib.ptr(d.t["triangle_areas"]), _lib.ptr(J), pf, ns,
                                                     _lib.ptr(out_mma), _lib.stream_ptr()))

        def cuda_core():
            _lib.check(L.scb_film_coupling(m, _lib.ptr(d.sites), 0.0, n, _lib.ptr(src3),
                                           _lib.ptr(d.t["triangle_areas"]), _lib.ptr(J), 0, 0, pf, ns,
                                           _lib.ptr(out_cc), _lib.stream_ptr()))

        def timed(fn):
            fn()
            ts = []
            for _ in range(launches):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                b.synchronize()
                ts.append(a.elapsed_time(b) * 1e-3)
            return float(np.median(ts))

        # alternate the two so that both see the same conditions
        t_mma, t_cc = [], []
        for _ in range(3):
            t_mma.append(timed(dmma))
            t_cc.append(timed(cuda_core))
        t_mma, t_cc = float(np.median(t_mma)), float(np.median(t_cc))
        work = float(m) * n * ns
        rows.append(dict(nsets=ns, targets=m, sources=n, dmma_s=t_mma, nb_coupling_8set_passes_s=t_cc,
                         speedup=t_cc / t_mma, dmma_pair_sets_per_s=work / t_mma,
                         nb_coupling_pair_sets_per_s=work / t_cc,
                         rel_l2_dmma_vs_cuda_core=rel_l2(out_mma.cpu().numpy(), out_cc.cpu().numpy())))
        print(json.dumps(rows[-1]), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--vertices", type=int, default=20000)
    ap.add_argument("--batches", type=int, nargs="+", default=[1, 8, 16, 64])
    ap.add_argument("--sets", type=int, nargs="+", default=[64, 128])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--launches", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import superscreen_b200 as sc

    device = bar_device(sc, args.vertices)
    result = dict(gpu=gpu_info(), vertices=len(device.meshes["bar"].sites),
                  triangles=len(device.meshes["bar"].elements))
    result["within_film_kernel"] = kernel_section(device, args.sets, args.launches)
    result["solve_batch_vs_serial"] = solve_section(sc, device, args.batches, args.reps)
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
