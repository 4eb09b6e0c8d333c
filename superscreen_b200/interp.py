"""Point location, linear interpolation and polygon masks on the device (csrc/interp.cu, include/scb.h).

The device stage of ``interp_current_density_batch`` / ``interp_field_batch``: a uniform cell grid over a mesh's
triangles (built once per mesh and cached), the containing triangle and barycentric weights of every query point,
the interpolated values of many value sets at once, and the even-odd film mask.  The host functions they stand in
for, ``solution.linear_tri_interpolate`` / ``_locate`` and ``geometry.points_in_polygon``, stay the reference.
"""
from __future__ import annotations

import math
from typing import Any, Dict, List, NamedTuple

import numpy as np

from . import _lib


class TriGrid(NamedTuple):
    """Cell grid over the triangles of one mesh, on one device."""

    x0: float
    y0: float
    x1: float            # x0 + ncx * cell: points beyond the grid are outside
    y1: float
    cell: float
    ncx: int
    ncy: int
    sites: Any           # (n, 2) float64, device
    elements: Any        # (ntri, 3) int64, device
    start: Any           # (ncx * ncy + 1,) int32, device: cell c holds cell_tris[start[c]:start[c + 1]]
    cell_tris: Any       # int32, device


_TRI_GRIDS: Dict[tuple, Any] = {}


def grid_layout(sites: np.ndarray, ntri: int):
    """(x0, y0, cell, ncx, ncy) of the default grid of a mesh: its bounding box widened by 1e-6 of its extent,
    square cells, about two triangles' area per cell."""
    lo, hi = sites.min(axis=0), sites.max(axis=0)
    ext = float(max(hi[0] - lo[0], hi[1] - lo[1]))
    margin = 1e-6 * ext if ext > 0 else 1.0
    w, h = float(hi[0] - lo[0]) + 2 * margin, float(hi[1] - lo[1]) + 2 * margin
    cell = math.sqrt(2.0 * w * h / max(ntri, 1))
    ncx, ncy = max(1, math.ceil(w / cell)), max(1, math.ceil(h / cell))
    while ncx * ncy >= 1 << 26:
        cell *= 2.0
        ncx, ncy = max(1, math.ceil(w / cell)), max(1, math.ceil(h / cell))
    return float(lo[0]) - margin, float(lo[1]) - margin, cell, ncx, ncy


def tri_grid(sites: np.ndarray, elements: np.ndarray, layout=None) -> TriGrid:
    """The triangle grid of the mesh (sites, elements) on the current device, built on the first call and cached
    per (sites, elements) array pair (a replaced mesh array is a new key).  ``layout`` = (x0, y0, cell, ncx, ncy)
    overrides ``grid_layout``."""
    import torch

    L = _lib.lib()
    dev = torch.device(f"cuda:{torch.cuda.current_device()}")
    layout = tuple(layout) if layout is not None else None
    key = (id(sites), id(elements), str(dev), layout)
    hit = _TRI_GRIDS.get(key)
    if hit is not None and hit[0] is sites and hit[1] is elements:
        return hit[2]
    ntri = len(elements)
    x0, y0, cell, ncx, ncy = layout if layout is not None else grid_layout(np.asarray(sites), ntri)
    ncx, ncy = int(ncx), int(ncy)
    with torch.cuda.device(dev):
        s_d = torch.as_tensor(np.ascontiguousarray(sites, dtype=np.float64)).to(dev)
        e_d = torch.as_tensor(np.ascontiguousarray(elements, dtype=np.int64)).to(dev)
        ncells = ncx * ncy
        ws = torch.empty(int(L.scb_tri_grid_workspace_elems(ntri, ncells)), dtype=torch.int32, device=dev)
        _lib.check(L.scb_tri_grid_count(ntri, _lib.ptr(s_d), _lib.ptr(e_d), x0, y0, cell, ncx, ncy, _lib.ptr(ws),
                                        _lib.stream_ptr()))
        entries = int(ws[4 * ntri + ncells].item())  # (the one synchronisation of a grid build)
        cell_tris = torch.empty(max(entries, 1), dtype=torch.int32, device=dev)
        _lib.check(L.scb_tri_grid_fill(ntri, ncx, ncy, _lib.ptr(ws), _lib.ptr(cell_tris), _lib.stream_ptr()))
        start = ws[4 * ntri:4 * ntri + ncells + 1]
    grid = TriGrid(float(x0), float(y0), float(x0) + ncx * float(cell), float(y0) + ncy * float(cell), float(cell),
                   ncx, ncy, s_d, e_d, start, cell_tris)
    if len(_TRI_GRIDS) > 16:
        _TRI_GRIDS.clear()
    _TRI_GRIDS[key] = (sites, elements, grid)
    return grid


def locate(grid: TriGrid, xy, tri, bary) -> None:
    """tri (int64 [q]) and bary (float64 [q, 3]) of the device points xy [q, 2] (scb_tri_locate)."""
    L = _lib.lib()
    _lib.check(L.scb_tri_locate(int(xy.shape[0]), _lib.ptr(xy), _lib.ptr(grid.sites), _lib.ptr(grid.elements),
                                grid.x0, grid.y0, grid.x1, grid.y1, grid.cell, grid.ncx, grid.ncy,
                                _lib.ptr(grid.start), _lib.ptr(grid.cell_tris), _lib.ptr(tri), _lib.ptr(bary),
                                _lib.stream_ptr()))


def interpolate(grid: TriGrid, tri, bary, values, out, mask=None, scale: float = 1.0) -> None:
    """out [nsets, q, ncomp] <- the value sets values [nsets, n, ncomp] at the located points (scb_tri_interpolate);
    zero outside the mesh, where ``mask`` (uint8 [q]) is 0 and where a component is not finite."""
    L = _lib.lib()
    nsets, n, ncomp = (int(d) for d in values.shape)
    _lib.check(L.scb_tri_interpolate(int(tri.shape[0]), _lib.ptr(tri), _lib.ptr(bary), _lib.ptr(grid.elements), nsets,
                                     ncomp, n, _lib.ptr(values), _lib.ptr(mask), float(scale), _lib.ptr(out),
                                     _lib.stream_ptr()))


def polygon_rings(polygon) -> tuple:
    """(add rings, cut rings) of a film polygon, open and in the order ``contains_points`` tests them (the vertex
    order decides the rounding of every crossing)."""
    from .device import CompositePolygon

    def open_ring(ring):
        ring = np.asarray(ring, dtype=float)
        if len(ring) > 1 and np.array_equal(ring[0], ring[-1]):  # (as points_in_polygon drops the closing vertex)
            ring = ring[:-1]
        return np.ascontiguousarray(ring)

    if isinstance(polygon, CompositePolygon):
        return [open_ring(r) for r in polygon._add], [open_ring(r) for r in polygon._sub]
    return [open_ring(polygon.points)], []


def upload_rings(polygon, dev) -> List[tuple]:
    """[(op, device ring)] of ``polygon_mask``: the first ring sets the mask, further add rings OR, cut rings
    AND-NOT."""
    import torch

    add, sub = polygon_rings(polygon)
    rings = [(0 if k == 0 else 1, r) for k, r in enumerate(add)] + [(2, r) for r in sub]
    return [(op, torch.as_tensor(r).to(dev)) for op, r in rings]


def polygon_mask(rings: List[tuple], xy, inside) -> None:
    """inside (uint8 [q]) <- the film mask of the device points xy [q, 2] (scb_points_in_polygon per ring)."""
    L = _lib.lib()
    for op, ring in rings:
        _lib.check(L.scb_points_in_polygon(int(xy.shape[0]), _lib.ptr(xy), int(ring.shape[0]), _lib.ptr(ring), op,
                                           _lib.ptr(inside), _lib.stream_ptr()))


def points_in_polygon(polygon, points: np.ndarray) -> np.ndarray:
    """``polygon.contains_points(points)`` on the device (a ``Polygon`` or ``CompositePolygon``)."""
    import torch

    dev = torch.device(f"cuda:{torch.cuda.current_device()}")
    xy = torch.as_tensor(np.ascontiguousarray(np.atleast_2d(points), dtype=np.float64)).to(dev)
    inside = torch.empty(int(xy.shape[0]), dtype=torch.uint8, device=dev)
    polygon_mask(upload_rings(polygon, dev), xy, inside)
    return inside.cpu().numpy().astype(bool)
