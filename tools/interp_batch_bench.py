"""Current-density and field images of a batch of solutions on one GPU: interp_current_density_batch /
interp_field_batch and their stages, against the per-solution host methods where those finish in reasonable time.

C2 square (configs.c2_square, 20k vertices, mesh = film = [-5, 5]^2): a solve_batch vortex scan with B = 1, 16, 64,
256 entries (one vortex each), images on 256 x 256 and 1000 x 1000 grids over [-6, 6]^2 (points outside the mesh
included).  Per (B, grid): the stages on the device with CUDA events (grid build, location, film mask, interpolation
of the B current densities, device-to-host copy of the (B, m, 2) result into pinned memory, with the copy's bytes
per second) and the whole interp_current_density_batch / interp_field_batch call as device-synchronised wall time;
median of --reps after one warm-up of each shape.  The L2 is not overwritten between launches (the 1000^2 results
exceed it; the 256^2 ones and the mesh do not).

IBM susceptometer (configs.ibm_susceptometer, host meshes): the stages on the mesh of the field-coil film, whose
film polygon is a union of rings (the mask kernel runs once per ring), 1000 x 1000 grid over the mesh.

Host rows: the per-solution Solution.interp_current_density on a 256 x 256 grid inside the mesh and on a 40 x 40 grid
over [-6, 6]^2 (outside points go through the host's exhaustive search), measured once per entry for --host-entries
entries; B times that is labelled extrapolated.  Batch rows are compared with the host rows in the same run.
The GPU name and power limit are read in the same run.  Prints one JSON object and writes it to --out.

    python tools/interp_batch_bench.py --out interp_batch.json
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


def grid(k, half=6.0):
    x, y = np.meshgrid(np.linspace(-half, half, k), np.linspace(-half, half, k))
    return np.column_stack([x.ravel(), y.ravel()])


def wall(fn, reps):
    import torch

    fn()
    torch.cuda.synchronize()
    ts, out = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), out


def events(fn, reps):
    import torch

    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e-3)
    return float(np.median(ts))


def stages(sc, sites, elements, polygon, values, positions, reps):
    """Device times of the stages of one batch call over all positions at once (values: (B, n, ncomp))."""
    import torch

    from superscreen_b200 import interp

    B, n, ncomp = values.shape
    m = len(positions)
    interp._TRI_GRIDS.clear()
    t_grid = events(lambda: (interp._TRI_GRIDS.clear(), interp.tri_grid(sites, elements)), reps)
    g = interp.tri_grid(sites, elements)
    xy = torch.as_tensor(positions).cuda()
    tri = torch.empty(m, dtype=torch.int64, device="cuda")
    bary = torch.empty((m, 3), dtype=torch.float64, device="cuda")
    inside = torch.empty(m, dtype=torch.uint8, device="cuda")
    vals = torch.as_tensor(values).cuda()
    out = torch.empty((B, m, ncomp), dtype=torch.float64, device="cuda")
    host = torch.empty((B, m, ncomp), dtype=torch.float64, pin_memory=True)
    rings = interp.upload_rings(polygon, torch.device("cuda"))
    t_loc = events(lambda: interp.locate(g, xy, tri, bary), reps)
    t_mask = events(lambda: interp.polygon_mask(rings, xy, inside), reps)
    t_int = events(lambda: interp.interpolate(g, tri, bary, vals, out, inside), reps)
    t_copy = events(lambda: host.copy_(out, non_blocking=True), reps)
    return dict(grid_cells=g.ncx * g.ncy, grid_entries=int(g.cell_tris.numel()), triangles=len(elements),
                polygon_rings=len(rings), polygon_vertices=sum(int(r.shape[0]) for _, r in rings),
                points_inside_mesh=int((tri >= 0).sum().item()), grid_build_s=t_grid, locate_s=t_loc, mask_s=t_mask,
                interpolate_s=t_int, d2h_copy_s=t_copy, d2h_bytes=B * m * ncomp * 8,
                d2h_bytes_per_s=B * m * ncomp * 8 / t_copy)


def c2_rows(sc, model, device, B, k, reps):
    rng = np.random.default_rng(B)
    vortices = [[sc.Vortex(x=float(x), y=float(y), film="film")] for x, y in rng.uniform(-4.5, 4.5, (B, 2))]
    sols = [s[-1] for s in sc.solve_batch(model=model, applied_fields=[None] * B, vortices=vortices, last_only=True)]
    positions = grid(k)
    mesh = device.meshes["film"]
    J = np.stack([s.film_solutions["film"].current_density for s in sols])
    row = dict(B=B, grid=f"{k}x{k} over [-6, 6]^2", targets=k * k)
    row.update(stages(sc, mesh.sites, mesh.elements, device.films["film"], J, positions, reps))
    row["interp_current_density_batch_s"], outJ = wall(
        lambda: sc.interp_current_density_batch(sols, positions, film="film"), reps)
    row["interp_field_batch_s"], _ = wall(lambda: sc.interp_field_batch(sols, positions, film="film"), reps)
    row["entries_differ"] = bool(not np.array_equal(outJ[0], outJ[-1]))
    print(json.dumps(row), flush=True)
    return row, sols


def host_rows(sc, sols, entries):
    """The per-solution host call, measured; the batch result of the same entries compared with it."""
    rows = []
    for label, positions in (("256x256 inside the mesh", grid(256, 4.99)), ("40x40 over [-6, 6]^2", grid(40))):
        ts, maxdiff, equal = [], 0.0, True
        batch = sc.interp_current_density_batch(sols[:entries], positions, film="film")
        for b in range(entries):
            t0 = time.perf_counter()
            ref = sols[b].interp_current_density(positions, film="film")
            ts.append(time.perf_counter() - t0)
            equal &= bool(np.array_equal(batch[b], ref))
            maxdiff = max(maxdiff, float(np.abs(batch[b] - ref).max()))
        t = float(np.median(ts))
        row = dict(grid=label, targets=len(positions), host_call_s_measured=t, host_call_s_each=ts,
                   host_calls_measured=entries,
                   batch_rows_bit_equal_to_host=equal, batch_max_abs_diff_to_host=maxdiff,
                   max_abs_J=float(np.abs(batch).max()),
                   host_loop_s_extrapolated={str(B): B * t for B in (1, 16, 64, 256)})
        print(json.dumps(row), flush=True)
        rows.append(row)
    return rows


def ibm_rows(sc, reps, k):
    from superscreen_b200 import configs

    device, _, meshes = configs.ibm_susceptometer(attach_meshes=False)
    rows = []
    for film in ("fc", "pl"):
        sites, elements = meshes[film]
        lo, hi = sites.min(axis=0), sites.max(axis=0)
        x, y = np.meshgrid(np.linspace(lo[0], hi[0], k), np.linspace(lo[1], hi[1], k))
        positions = np.column_stack([x.ravel(), y.ravel()])
        values = np.random.default_rng(0).standard_normal((64, len(sites), 2))
        row = dict(film=film, B=64, grid=f"{k}x{k} over the mesh", targets=k * k, vertices=len(sites),
                   polygon=type(device.films[film]).__name__)
        row.update(stages(sc, sites, elements, device.films[film], values, positions, reps))
        t0 = time.perf_counter()
        device.films[film].contains_points(positions)
        row["host_contains_points_s_measured"] = time.perf_counter() - t0
        print(json.dumps(row), flush=True)
        rows.append(row)
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--batches", type=int, nargs="+", default=[1, 16, 64, 256])
    ap.add_argument("--grids", type=int, nargs="+", default=[256, 1000])
    ap.add_argument("--host-entries", type=int, default=2)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import superscreen_b200 as sc
    from superscreen_b200 import configs

    info = gpu_info()
    device = configs.c2_square()
    model = sc.factorize_model(device=device, current_units="uA")
    scans, sols = [], None
    for B in args.batches:
        for k in args.grids:
            row, sols = c2_rows(sc, model, device, B, k, args.reps)
            scans.append(row)
    result = dict(gpu=info, vertices=len(device.meshes["film"].sites), reps=args.reps,
                  timing="stages: CUDA events over all targets at once; *_batch_s: device-synchronised wall time of "
                         "the public call (host staging, pinned allocations and chunked copies included); median of "
                         "--reps after one warm-up of each shape",
                  l2_overwritten_between_launches=False, c2_square=scans,
                  host=host_rows(sc, sols, args.host_entries), ibm_susceptometer=ibm_rows(sc, args.reps, 1000))
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
