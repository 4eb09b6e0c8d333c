"""Solution containers and post-processing (reference superscreen/solution.py).

The O(m*n) field evaluations (``field_at_position``, ``screening_field_at_position``,
``vector_potential_at_position``; reference solution.py:611-934 and sources/current.py:13-196)
run as tiled fp64 pair sums on the device (``scb_biot_savart``); fluxoids and interpolation are
O(n + polygon points) host work (reference solution.py:278-319,484-609).
"""
from __future__ import annotations

import datetime as dt
import logging
from dataclasses import dataclass
from typing import Any, Callable, Dict, List, NamedTuple, Optional, Sequence, Tuple, Union

import numpy as np

from . import _lib
from . import units as _u
from .device import Device, Polygon
from .geometry import points_in_polygon

try:  # the reference's Biot-Savart uses scipy.constants.mu_0 (SURVEY.md Q7)
    from scipy.constants import mu_0 as _MU0_BIOT_SAVART
except Exception:  # pragma: no cover
    _MU0_BIOT_SAVART = _u.MU_0

logger = logging.getLogger("solution")


class Fluxoid(NamedTuple):
    """flux part + supercurrent part (reference solution.py:39-59)."""

    flux_part: Union[float, _u.Quantity]
    supercurrent_part: Union[float, _u.Quantity]


@dataclass
class Vortex:
    """reference solution.py:62-92"""

    x: float
    y: float
    film: str
    nPhi0: float = 1


class FilmSolution:
    """Raw solution data for a single film (reference solution.py:95-130)."""

    def __init__(self, stream, current_density, applied_field, self_field, field_from_other_films=None):
        self.stream = np.asarray(stream)
        self.current_density = np.asarray(current_density)
        self.applied_field = np.asarray(applied_field)
        self.self_field = np.asarray(self_field)
        if field_from_other_films is not None:
            field_from_other_films = np.asarray(field_from_other_films)
        self.field_from_other_films = field_from_other_films
        self._total_field: Optional[np.ndarray] = None

    @property
    def total_field(self) -> np.ndarray:
        if self._total_field is None:
            self._total_field = self.applied_field + self.self_field
            if self.field_from_other_films is not None:
                self._total_field = self._total_field + self.field_from_other_films
        return self._total_field

    def to_hdf5(self, h5group) -> None:
        """reference solution.py:132-143"""
        from . import io as _io

        _io.film_solution_to_hdf5(self, h5group)

    @staticmethod
    def from_hdf5(h5group) -> "FilmSolution":
        """reference solution.py:145-164"""
        from . import io as _io

        return _io.film_solution_from_hdf5(h5group)

    def is_close(self, other: "FilmSolution", rtol: float = 1e-4, atol: float = 1e-7) -> bool:
        """reference solution.py:166-185"""
        kw = dict(rtol=rtol, atol=atol)
        return bool(np.allclose(self.stream, other.stream, **kw)
                    and np.allclose(self.applied_field, other.applied_field, **kw)
                    and np.allclose(self.self_field, other.self_field, **kw)
                    and np.allclose(self.total_field, other.total_field, **kw))

    def __eq__(self, other) -> bool:
        """reference solution.py:187-199 (tolerance-based, like the reference)"""
        if other is self:
            return True
        if not isinstance(other, FilmSolution):
            return False
        if (self.field_from_other_films is None) != (other.field_from_other_films is None):
            return False
        if self.field_from_other_films is not None and not np.allclose(self.field_from_other_films,
                                                                       other.field_from_other_films):
            return False
        return self.is_close(other)

    __hash__ = None


_LOCATORS: Dict[int, Any] = {}


def _triangle_locator(sites: np.ndarray, elements: np.ndarray):
    """KD-tree over triangle centroids, cached per elements array."""
    from scipy.spatial import cKDTree

    key = (id(elements), id(sites))
    hit = _LOCATORS.get(key)
    if hit is None or hit[0] is not elements or hit[1] is not sites:
        hit = (elements, sites, cKDTree(sites[elements].mean(axis=1)))
        if len(_LOCATORS) > 64:
            _LOCATORS.clear()
        _LOCATORS[key] = hit
    return hit[2]


def _barycentric(p: np.ndarray, xy: np.ndarray):
    """Barycentric coordinates of points xy (q, 2) in triangles p (q, k, 3, 2) -> (q, k, 3)."""
    a, b, c = p[..., 0, :], p[..., 1, :], p[..., 2, :]
    det = (b[..., 1] - c[..., 1]) * (a[..., 0] - c[..., 0]) + (c[..., 0] - b[..., 0]) * (a[..., 1] - c[..., 1])
    dx = xy[:, None, 0] - c[..., 0]
    dy = xy[:, None, 1] - c[..., 1]
    l1 = ((b[..., 1] - c[..., 1]) * dx + (c[..., 0] - b[..., 0]) * dy) / det
    l2 = ((c[..., 1] - a[..., 1]) * dx + (a[..., 0] - c[..., 0]) * dy) / det
    return np.stack([l1, l2, 1.0 - l1 - l2], axis=-1)


_LOCATIONS: Dict[tuple, Any] = {}


def _locate(sites: np.ndarray, elements: np.ndarray, xy: np.ndarray, candidates: int):
    """(inside mask, containing triangle, barycentric weights) of the query points; memoised per
    (mesh, query points): fluxoid polygons are evaluated for many solutions on the same mesh."""
    key = (id(elements), id(sites), xy.shape, xy.tobytes() if xy.size <= 4096 else None)
    if key[3] is not None:
        hit = _LOCATIONS.get(key)
        if hit is not None and hit[0] is elements and hit[1] is sites:
            return hit[2]
    k = min(candidates, len(elements))
    _, cand = _triangle_locator(sites, elements).query(xy, k=k)
    cand = cand.reshape(len(xy), k)
    lam = _barycentric(sites[elements[cand]], xy)          # (q, k, 3)
    mn = lam.min(axis=2)
    best = np.argmax(mn, axis=1)
    r = np.arange(len(xy))
    ok = mn[r, best] >= -1e-12
    tri = cand[r, best]
    w = lam[r, best]
    # unresolved points: exhaustive search (outside the mesh, or very anisotropic neighbourhoods)
    for q in np.where(~ok)[0]:
        lam_all = _barycentric(sites[elements][None, :, :, :], xy[q:q + 1])[0]
        mn_all = lam_all.min(axis=1)
        t = int(np.argmax(mn_all))
        if mn_all[t] >= -1e-12:
            ok[q], tri[q], w[q] = True, t, lam_all[t]
    if key[3] is not None:
        if len(_LOCATIONS) > 256:
            _LOCATIONS.clear()
        _LOCATIONS[key] = (elements, sites, (ok, tri, w))
    return ok, tri, w


def linear_tri_interpolate(sites: np.ndarray, elements: np.ndarray, values: np.ndarray, xy: np.ndarray,
                           candidates: int = 16) -> np.ndarray:
    """Piecewise-linear interpolation on a triangulation; NaN outside the mesh.  Stands in for
    ``matplotlib.tri.LinearTriInterpolator`` (reference solution.py:272-276,310-312).  The containing
    triangle is searched among the triangles with the nearest centroids (all triangles as a
    fallback for points that are not resolved that way)."""
    xy = np.atleast_2d(np.asarray(xy, dtype=float))
    values = np.asarray(values, dtype=float)
    out = np.full((len(xy),) + values.shape[1:], np.nan)
    if len(xy) == 0:
        return out
    ok, tri, w = _locate(sites, elements, xy, candidates)
    v = values[elements[tri]]                                # (q, 3, ...)
    res = np.einsum("qk,qk...->q...", w, v)
    out[ok] = res[ok]
    return out


def _normalize_positions(positions, zs, dtype):
    """Shared argument handling of the *_at_position methods (reference solution.py:660-676)."""
    positions = np.atleast_2d(positions)
    if positions.shape[1] == 3:
        if zs is not None:
            raise ValueError("If positions has shape (m, 3) then zs cannot be specified.")
        zs = positions[:, 2]
        positions = positions[:, :2]
    else:
        zs = np.squeeze(zs)
        if zs.ndim == 0:
            zs = zs.item() * np.ones(positions.shape[0], dtype=dtype)
    if not isinstance(zs, np.ndarray):
        raise ValueError(f"Expected zs to be an ndarray, but got {type(zs)}.")
    # (views where possible: a million-point grid is not copied just to be split into columns)
    return np.asarray(positions, dtype=np.float64), np.asarray(zs, dtype=np.float64)


# targets per pipelined chunk of a field evaluation: one full wave of the pair-sum kernel (148 SMs x 6 resident
# CTAs x 512 targets); smaller launches would split their sources and pay a reduction pass
_EVAL_CHUNK = 148 * 6 * 512


def biot_savart_2d(x, y, z, *, positions, current_densities, z0: float = 0, areas=None, length_units: str = "um",
                   current_units: str = "uA", vector: bool = True, device_tensors: Optional[dict] = None):
    """Field (tesla) of a current sheet at ``(x, y, z)`` (reference sources/current.py:113-196).
    ``areas`` is required (the Delaunay fallback of the reference, current.py:186-189, is host-side
    meshing and out of scope).  ``device_tensors``: optional dict that keeps the uploaded source arrays
    (SI units) between calls on the same current sheet -- ``Solution.field_at_position`` evaluates many
    target sets against one solution."""
    import torch

    L = _lib.lib()
    if areas is None:
        raise ValueError("areas (vertex areas of the current sheet) must be given.")
    to_meter = _u.conversion_factor(length_units, "m")
    to_amp_per_meter = _u.conversion_factor(f"({current_units}) / ({length_units})", "A / m")
    x, y, z = np.atleast_1d(x, y, z)
    dev = torch.device(f"cuda:{torch.cuda.current_device()}")
    m = len(x)
    with torch.cuda.device(dev):
        src_key = ("sources", str(dev))
        src = None if device_tensors is None else device_tensors.get(src_key)
        if src is None:
            positions, current_densities = np.atleast_2d(positions, current_densities)
            J = np.ascontiguousarray(current_densities * to_amp_per_meter, dtype=np.float64)
            pos = positions * to_meter
            zz = z0 * np.ones(len(pos)) * to_meter
            ar = np.ascontiguousarray(np.asarray(areas) * to_meter**2, dtype=np.float64)
            pos3 = np.ascontiguousarray(np.concatenate([pos, zz[:, None]], axis=1), dtype=np.float64)
            src = tuple(torch.as_tensor(a).to(dev) for a in (pos3, ar, J))
            if device_tensors is not None:
                device_tensors[src_key] = src
        pos_d, ar_d, J_d = src
        n = int(pos_d.shape[0])
        if m == 0:
            return np.empty((0, 3) if vector else (0,), dtype=np.float64)
        # Targets go through PINNED staging in chunks: the host scales chunk k + 1 into its staging block
        # (column by column: no (3, m) temporary) while the GPU evaluates chunk k, and every chunk's result
        # is copied back behind its kernel -- one synchronisation at the end, the host preparation and the
        # transfers of a million-point grid disappear behind the pair sums.
        chunk = m if m <= _EVAL_CHUNK else _EVAL_CHUNK
        ev_pin = torch.empty((m, 3), dtype=torch.float64, pin_memory=True)
        out_pin = torch.empty((m, 3) if vector else (m,), dtype=torch.float64, pin_memory=True)
        ev = ev_pin.numpy()
        zb = np.broadcast_to(z, (m,))  # (a length-1 z broadcasts)
        stream = torch.cuda.current_stream(dev)
        keep = []  # device blocks stay referenced until the final synchronisation (stream-ordered use)
        for lo in range(0, m, chunk):
            hi = min(m, lo + chunk)
            np.multiply(x[lo:hi], to_meter, out=ev[lo:hi, 0])
            np.multiply(y[lo:hi], to_meter, out=ev[lo:hi, 1])
            np.multiply(zb[lo:hi], to_meter, out=ev[lo:hi, 2])
            ev_d = ev_pin[lo:hi].to(dev, non_blocking=True)
            out_d = torch.empty((hi - lo, 3) if vector else (hi - lo,), dtype=torch.float64, device=dev)
            _lib.check(L.scb_biot_savart(2 if vector else 1, hi - lo, _lib.ptr(ev_d), n, _lib.ptr(pos_d), _lib.ptr(ar_d),
                                         _lib.ptr(J_d), 0.0, _MU0_BIOT_SAVART / (4 * np.pi), 1, _lib.ptr(out_d),
                                         _lib.stream_ptr()))
            out_pin[lo:hi].copy_(out_d, non_blocking=True)
            keep.append((ev_d, out_d))
        stream.synchronize()
        return out_pin.numpy()


class _FluxoidGeometry(NamedTuple):
    """Everything of ``polygon_fluxoid`` that depends only on (mesh, film, polygon)."""

    ix: np.ndarray            # mesh vertices inside the polygon
    w_ix: np.ndarray          # their vertex areas
    tri_vertices: np.ndarray  # (q, 3) vertices of the triangle containing every polygon point
    bary: np.ndarray          # (q, 3) barycentric weights
    valid: np.ndarray         # (q,) polygon point lies in the film and in the mesh
    dl: np.ndarray            # (q - 1, 2) polygon edge vectors
    Lambda_poly: np.ndarray   # (q,) Lambda at the polygon points
    # the supercurrent integral as ONE linear functional of the mesh values of J:
    # trapezoid_q(Lambda_q * sum_c J_poly[q, c] dl[q, c]) = sum_m J_coef[m] . J[J_idx[m]]
    J_idx: np.ndarray         # (3 (q - 1),) mesh vertices (corners of the triangles under the polygon points)
    J_coef: np.ndarray        # (3 (q - 1), 2) trapezoid weight * Lambda * barycentric weight * edge vector


_FLUXOID_GEOMETRY: Dict[tuple, Any] = {}


def _fluxoid_geometry(device: Device, film: str, mesh, polygon_coords) -> _FluxoidGeometry:
    """The fluxoid of the same polygon is evaluated for many solutions on the same mesh (every
    column / iterate of a mutual-inductance matrix): index sets and interpolation weights are
    memoised per (mesh, film polygon, fluxoid polygon)."""
    film_poly = device.films[film]
    Lambda = device.layers[film_poly.layer].Lambda
    raw = polygon_coords.points if isinstance(polygon_coords, Polygon) else np.asarray(polygon_coords, dtype=float)
    key = (id(mesh), raw.tobytes(), film_poly.points.tobytes(), None if callable(Lambda) else float(Lambda))
    hit = _FLUXOID_GEOMETRY.get(key)
    if hit is not None and hit[0] is mesh and (not callable(Lambda) or hit[1] is Lambda):
        return hit[2]
    polygon = polygon_coords if isinstance(polygon_coords, Polygon) else Polygon(points=polygon_coords)
    points = polygon.points  # closed and counter-clockwise (reference device/polygon.py:67-77)
    if not film_poly.contains_points(points).all():
        raise ValueError(f"The polygon is not contained within the film ({film!r}).")
    ix = np.where(polygon.contains_points(mesh.sites))[0]
    ok, tri, w = _locate(mesh.sites, mesh.elements, points, 16)
    valid = ok & film_poly.contains_points(points)
    if callable(Lambda):
        Lambda_poly = np.asarray(Lambda(points[:, 0], points[:, 1]), dtype=float) * np.ones(len(points))
    else:
        Lambda_poly = float(Lambda) * np.ones(len(points))
    dl = np.diff(points, axis=0)
    tri_vertices = mesh.elements[tri]
    nq = len(points) - 1  # samples of the trapezoid rule (reference solution.py:556-557 drops the last point)
    trap = np.ones(nq)
    if nq >= 2:
        trap[0] = trap[-1] = 0.5
    else:
        trap[:] = 0.0  # (np.trapezoid of a single sample is 0)
    per_point = trap * Lambda_poly[:-1] * valid[:-1]                                   # (nq,)
    J_coef = (per_point[:, None, None] * w[:-1, :, None] * dl[:, None, :]).reshape(-1, 2)  # (3 nq, 2)
    J_coef = np.where(np.isfinite(J_coef), J_coef, 0.0)  # (barycentric weights of points outside the mesh)
    J_idx = np.where(valid[:-1, None], tri_vertices[:-1], 0).reshape(-1)
    geo = _FluxoidGeometry(ix=ix, w_ix=mesh.vertex_areas[ix], tri_vertices=tri_vertices, bary=w,
                           valid=valid, dl=dl, Lambda_poly=Lambda_poly, J_idx=J_idx, J_coef=J_coef)
    if len(_FLUXOID_GEOMETRY) > 256:
        _FLUXOID_GEOMETRY.clear()
    _FLUXOID_GEOMETRY[key] = (mesh, Lambda, geo)
    return geo


class Solution:
    """reference solution.py:201-260 (container) + post-processing methods."""

    def __init__(self, *, device: Device, film_solutions: Dict[str, FilmSolution], applied_field_func: Callable,
                 field_units: str, current_units: str, circulating_currents: Optional[Dict[str, float]] = None,
                 terminal_currents: Optional[Dict[str, float]] = None, vortices=None,
                 solver: str = "superscreen_b200.solve", _device_is_copy: bool = False,
                 _device_builder: Optional[Callable[[], Device]] = None):
        # (the solver hands one private copy of the device to all the solutions of a call; a translated
        # entry of solve_batch gets a builder instead, shared by the entries with the same translation, that
        # makes the translated device on first access)
        self._device_builder = _device_builder
        if _device_builder is None:
            self.device = device if _device_is_copy else device.copy(with_mesh=True, copy_mesh=False)
        else:
            self._device = None
        self.film_solutions = film_solutions
        self.applied_field_func = applied_field_func
        self.circulating_currents = circulating_currents or {}
        self.terminal_currents = terminal_currents or {}
        self.vortices = vortices or []
        self._field_units = field_units
        self._current_units = current_units
        self._solver = solver
        self._time_created = dt.datetime.now()

    @property
    def device(self) -> Device:
        if self._device is None:
            self._device = self._device_builder()
        return self._device

    @device.setter
    def device(self, device: Device) -> None:
        self._device = device

    @property
    def version_info(self) -> Dict[str, str]:
        if getattr(self, "_version_info", None) is None:
            from . import io as _io

            self._version_info = _io.version_info()
        return self._version_info

    def to_hdf5(self, path_or_group, device_path: Optional[str] = None, compress: bool = True) -> None:
        """reference solution.py:936-978"""
        from . import io as _io

        _io.solution_to_hdf5(self, path_or_group, device_path=device_path, compress=compress)

    @staticmethod
    def from_hdf5(path_or_group) -> "Solution":
        """reference solution.py:980-1029"""
        from . import io as _io

        return _io.solution_from_hdf5(path_or_group)

    @staticmethod
    def save_solutions(solutions, path_or_group, compress: bool = True) -> None:
        """reference solution.py:1031-1063"""
        from . import io as _io

        _io.save_solutions(solutions, path_or_group, compress=compress)

    @staticmethod
    def load_solutions(path_or_group):
        """reference solution.py:1065-1087"""
        from . import io as _io

        return _io.load_solutions(path_or_group)

    def _source_cache(self, film: str) -> dict:
        """Device copies of a film's current sheet (sites, areas, J in SI units) for repeated field
        evaluations; dropped when the film's current density array is replaced."""
        cache = self.__dict__.setdefault("_bs_sources", {})
        J = self.film_solutions[film].current_density
        entry = cache.get(film)
        if entry is None or entry.get("J_ref") is not J:
            entry = cache[film] = {"J_ref": J}
        return entry

    field_units = property(lambda self: self._field_units)
    current_units = property(lambda self: self._current_units)
    solver = property(lambda self: self._solver)
    time_created = property(lambda self: self._time_created)

    # ---------------------------------------------------------------- interpolation
    def interp_field(self, positions, *, film: str, dataset: str = "total_field", method: str = "linear",
                     units: Optional[str] = None, with_units: bool = False):
        """reference solution.py:357-420 (linear only)."""
        from .solver.utils import convert_field

        valid = ("total_field", "applied_field", "self_field", "field_from_other_films")
        if dataset not in valid:
            raise ValueError(f"Unexpected dataset: {dataset}.")
        if method != "linear":
            raise NotImplementedError("Only linear interpolation is available.")
        positions = np.atleast_2d(positions)
        mesh = self.device.meshes[film]
        values = getattr(self.film_solutions[film], dataset)
        if values is None:
            return np.zeros(len(positions))
        out = linear_tri_interpolate(mesh.sites, mesh.elements, values, positions)
        out[~np.isfinite(out)] = 0
        if units is None or units == self.field_units:
            return _u.Quantity(out, self.field_units) if with_units else out
        return convert_field(out, units, old_units=self.field_units, with_units=with_units)

    def interp_current_density(self, positions, *, film: str, method: str = "linear", units: Optional[str] = None,
                               with_units: bool = False):
        """reference solution.py:278-319"""
        if method != "linear":
            raise NotImplementedError("Only linear interpolation is available.")
        device = self.device
        default_units = f"({self.current_units}) / ({device.length_units})"
        positions = np.atleast_2d(positions)
        mesh = device.meshes[film]
        J = linear_tri_interpolate(mesh.sites, mesh.elements, self.film_solutions[film].current_density, positions)
        in_film = device.films[film].contains_points(positions)
        J[~in_film] = 0
        J[~np.isfinite(J).all(axis=1)] = 0
        if units is not None and units != default_units:
            J = J * _u.conversion_factor(default_units, units)
        if with_units:
            return _u.Quantity(J, units or default_units)
        return J

    def current_through_path(self, path_coords: np.ndarray, *, film: str, interp_method: str = "linear",
                             units: Optional[str] = None, with_units: bool = True):
        """reference solution.py:321-355"""
        from .geometry import path_vectors

        units = units or self.current_units
        path_coords = np.asarray(path_coords, dtype=float)
        edge_lengths, unit_normals = path_vectors(path_coords)
        edge_centers = (path_coords[:-1] + path_coords[1:]) / 2
        J = self.interp_current_density(edge_centers, film=film, method=interp_method)
        total = np.sum(np.sum(J * unit_normals, axis=1) * edge_lengths)
        total = total * _u.conversion_factor(self.current_units, units)
        return _u.Quantity(total, units) if with_units else total

    def equals(self, other, require_same_timestamp: bool = False) -> bool:
        """reference solution.py:1089-1126 (solutions carry no creation time here, so
        ``require_same_timestamp`` has no effect; devices are compared by name and polygon data)."""
        if other is self:
            return True
        if not isinstance(other, Solution):
            return False

        def same_device(a, b):
            if a.name != b.name or list(a.films) != list(b.films) or list(a.holes) != list(b.holes):
                return False
            for pa, pb in zip(list(a.films.values()) + list(a.holes.values()),
                              list(b.films.values()) + list(b.holes.values())):
                if pa.layer != pb.layer or not np.array_equal(pa.points, pb.points):
                    return False
            return True

        if not (same_device(self.device, other.device) and self.field_units == other.field_units
                and self.current_units == other.current_units
                and self.circulating_currents == other.circulating_currents
                and self.terminal_currents == other.terminal_currents
                and self.applied_field_func == other.applied_field_func
                and list(self.vortices) == list(other.vortices)):
            return False
        return self.film_solutions == other.film_solutions

    # ---------------------------------------------------------------- fluxoid
    def polygon_flux(self, name: str, units: Optional[str] = None, with_units: bool = True):
        """Flux ``sum(mu_0 H_z w)`` through the polygon ``name`` of the device (a film, a hole or an abstract
        region), over the vertex areas of the film mesh that contains it (reference solution.py:430-482)."""
        from .solver.utils import convert_field

        device = self.device
        polygons = {p.name: p for p in device.get_polygons(include_terminals=False)}
        if name not in polygons:
            raise ValueError(f"Unknown polygon: {name!r}.")
        new_units = units or f"({self.field_units}) * ({device.length_units}) ** 2"
        polygon = polygons[name]
        if name in device.films:
            film_name = name
        else:
            film_name = None
            for film in device.films.values():
                film_name = film.name  # (the reference falls through to the last film if none contains it)
                if film.layer == polygon.layer and film.contains_points(polygon.points).all():
                    break
        mesh = device.meshes[film_name]
        ix = polygon.contains_points(mesh.sites, index=True)
        field_mT = convert_field(self.film_solutions[film_name].total_field[ix], "mT", old_units=self.field_units,
                                 with_units=False)
        flux = float(np.dot(field_mT, mesh.vertex_areas[ix]))
        flux = flux * _flux_conversion(f"mT * ({device.length_units}) ** 2", str(new_units))
        return _u.Quantity(flux, str(new_units)) if with_units else flux

    def polygon_fluxoid(self, polygon_coords, *, film: str, interp_method: str = "linear",
                        units: Optional[str] = "Phi_0", with_units: bool = True) -> Fluxoid:
        """reference solution.py:484-563"""
        device = self.device
        if interp_method != "linear":
            raise NotImplementedError("Only linear interpolation is available.")
        if units is None:
            units = f"({self.field_units}) * ({device.length_units}) ** 2"
        mesh = device.meshes[film]
        geo = _fluxoid_geometry(device, film, mesh, polygon_coords)
        fs = self.film_solutions[film]
        # flux part: total field (applied + self + other films, in that order) over the enclosed vertex areas
        if fs._total_field is not None:
            field_ix = fs._total_field[geo.ix]
        else:  # (no (n,) temporaries for a solution whose total field has not been asked for)
            field_ix = fs.applied_field[geo.ix] + fs.self_field[geo.ix]
            if fs.field_from_other_films is not None:
                field_ix = field_ix + fs.field_from_other_films[geo.ix]
        flux = float(np.dot(field_ix, geo.w_ix))
        conv = self.__dict__.get("_fluxoid_conversions", {}).get(units)
        if conv is None:
            flux_units = f"({self.field_units}) * ({device.length_units}) ** 2"
            J_units = f"({self.current_units}) / ({device.length_units})"
            conv = (_flux_conversion(flux_units, units),
                    _u.MU_0 * _u.conversion_factor(f"({J_units}) * ({device.length_units}) ** 2", "A * m")
                    * _u.conversion_factor("Wb", units))
            self.__dict__.setdefault("_fluxoid_conversions", {})[units] = conv
        flux_part = flux * conv[0]
        # supercurrent part: J at the polygon vertices (linear interpolation on the mesh, zero outside the film /
        # mesh: interp_current_density, reference solution.py:278-319), Lambda J . dl, trapezoid rule -- one
        # cached linear functional of the mesh values of J
        J_corner = fs.current_density[geo.J_idx]
        if np.isfinite(J_corner).all():
            int_J = float(np.einsum("mc,mc->", geo.J_coef, J_corner))
        else:  # the reference zeroes polygon points whose interpolated J is not finite
            J_poly = np.einsum("qk,qkc->qc", geo.bary, fs.current_density[geo.tri_vertices])
            J_poly[~geo.valid] = 0
            J_poly[~np.isfinite(J_poly).all(axis=1)] = 0
            int_J = np.trapezoid(geo.Lambda_poly[:-1] * np.sum(J_poly[:-1] * geo.dl, axis=1))
        # mu_0 * [J_units * length^2] -> units
        supercurrent_part = int_J * conv[1]
        if with_units:
            return Fluxoid(_u.Quantity(flux_part, units), _u.Quantity(supercurrent_part, units))
        return Fluxoid(flux_part, supercurrent_part)

    def hole_fluxoid(self, hole_name: str, points: Optional[np.ndarray] = None, interp_method: str = "linear",
                     units: Optional[str] = "Phi_0", with_units: bool = True) -> Fluxoid:
        """reference solution.py:565-609 (an explicit polygon is required)."""
        if points is None:
            from .fluxoid import make_fluxoid_polygons

            points = make_fluxoid_polygons(self.device, holes=hole_name)[hole_name]
        device = self.device
        hole = device.holes[hole_name]
        if not points_in_polygon(points, hole.points).all():
            raise ValueError(f"Hole {hole.name} is not completely enclosed by the given polygon.")
        film_name = None
        for film_name, holes in device.holes_by_film().items():
            if hole.name in [h.name for h in holes]:
                break
        return self.polygon_fluxoid(points, film=film_name, interp_method=interp_method, units=units,
                                    with_units=with_units)

    # ---------------------------------------------------------------- fields in space
    def screening_field_at_position(self, positions, *, zs=None, vector: bool = False, interp_method: str = "linear",
                                    units: Optional[str] = None, with_units: bool = True, return_sum: bool = True):
        """reference solution.py:611-723"""
        from .solver.utils import convert_field

        device = self.device
        dtype = np.float64  # the reference allocates float32 here after Device.copy (SURVEY.md Q5)
        units = units or self.field_units
        positions, zs = _normalize_positions(positions, zs, dtype)
        fields = {}
        for name, film in device.films.items():
            layer = device.layers[film.layer]
            mesh = device.meshes[name]
            shape = (len(positions), 3) if vector else (len(positions),)
            field_from_film = np.zeros(shape, dtype=dtype)
            in_film = np.zeros(len(positions), dtype=bool)
            if np.all(zs == layer.z0):
                in_film[film.contains_points(positions)] = True
                fin = self.interp_field(positions[in_film], film=name, dataset="self_field", method=interp_method,
                                        units="tesla", with_units=False)
                if vector:
                    zeros = np.zeros_like(fin)
                    fin = np.array([zeros, zeros, fin]).T
                field_from_film[in_film] = fin
            out = ~in_film
            if out.all():  # (the usual case of an evaluation plane above the device: no masked copies)
                field_from_film = biot_savart_2d(
                    positions[:, 0], positions[:, 1], zs, positions=mesh.sites, areas=mesh.vertex_areas,
                    current_densities=self.film_solutions[name].current_density, z0=layer.z0,
                    length_units=device.length_units, current_units=self.current_units, vector=vector,
                    device_tensors=self._source_cache(name))
            elif out.any():
                field_from_film[out] = biot_savart_2d(
                    positions[out, 0], positions[out, 1], zs[out], positions=mesh.sites, areas=mesh.vertex_areas,
                    current_densities=self.film_solutions[name].current_density, z0=layer.z0,
                    length_units=device.length_units, current_units=self.current_units, vector=vector,
                    device_tensors=self._source_cache(name))
            fields[name] = _convert_owned(field_from_film, units, "tesla", with_units)
        if return_sum:
            return _sum_owned(fields, with_units)
        return fields

    def field_at_position(self, positions, *, zs=None, interp_method: str = "linear", units: Optional[str] = None,
                          with_units: bool = True, return_sum: bool = True):
        """reference solution.py:725-831"""
        from .solver.utils import convert_field

        device = self.device
        dtype = np.float64
        units = units or self.field_units
        positions, zs = _normalize_positions(positions, zs, dtype)
        fields = self.screening_field_at_position(positions, zs=zs, vector=False, interp_method=interp_method,
                                                  units=self.field_units, with_units=False, return_sum=False)
        films_by_layer = device.polygons_by_layer("film")
        Hz_applied = np.zeros(len(positions), dtype=dtype)
        in_film = np.zeros(len(positions), dtype=bool)
        for name, layer in device.layers.items():
            if np.all(zs == layer.z0):
                for film in films_by_layer[name]:
                    ix = film.contains_points(positions)
                    in_film[ix] = True
                    Hz_applied[ix] = self.interp_field(positions[ix], film=film.name, dataset="applied_field",
                                                       method=interp_method, units=self.field_units)
                    Hz_applied[ix] += self.interp_field(positions[ix], film=film.name,
                                                        dataset="field_from_other_films", method=interp_method,
                                                        units=self.field_units)
                break
        mask = ~in_film
        if mask.all():
            Hz_applied = np.asarray(np.squeeze(
                self.applied_field_func(positions[:, 0], positions[:, 1], zs[:, np.newaxis])), dtype=dtype)
            Hz_applied = np.broadcast_to(Hz_applied, (len(positions),)) if Hz_applied.ndim == 0 else Hz_applied
        elif mask.any():
            Hz_applied[mask] = np.squeeze(
                self.applied_field_func(positions[mask, 0], positions[mask, 1], zs[mask, np.newaxis]))
        fields["applied_field"] = np.atleast_1d(Hz_applied).squeeze()
        for key, f in fields.items():  # (the applied field may be an array of the user's own function)
            fields[key] = _convert_owned(f, units, self.field_units, with_units, owned=key != "applied_field")
        if return_sum:
            return _sum_owned(fields, with_units, not_owned=("applied_field",))
        return fields

    def vector_potential_at_position(self, positions, *, zs=None, units: Optional[str] = None,
                                     with_units: bool = True, return_sum: bool = True):
        """reference solution.py:833-934; the (m x n x 2) temporary of the reference becomes a tiled
        pair sum on the device."""
        import torch

        L = _lib.lib()
        device = self.device
        dtype = np.float64
        units = units or f"({self.field_units}) * ({device.length_units})"
        positions, zs = _normalize_positions(positions, zs, dtype)
        dev = torch.device(f"cuda:{torch.cuda.current_device()}")
        tgt = torch.as_tensor(np.ascontiguousarray(np.column_stack([positions, zs]))).to(dev)
        # result in [current_units] * mu_0/4pi -> convert (A * mu_0 = T m) to the requested units
        scale = _u.MU_0 / (4 * np.pi) * _u.conversion_factor(self.current_units, "A") * _u.conversion_factor("T * m", units)
        out = {}
        for name, film in device.films.items():
            layer = device.layers[film.layer]
            dz = zs - layer.z0
            if np.all(dz == 0) and film.contains_points(positions).all():
                raise ValueError(f"Cannot evaluate vector potential inside the film ({name!r}).")
            d = device.meshes[name]._data
            n = d.n
            with torch.cuda.device(dev):
                src3 = torch.cat([d.sites.to(dev), torch.full((n, 1), float(layer.z0), dtype=torch.float64, device=dev)], 1).contiguous()
                J = torch.as_tensor(np.ascontiguousarray(self.film_solutions[name].current_density, dtype=np.float64)).to(dev)
                A2 = torch.empty(len(positions), 2, dtype=torch.float64, device=dev)
                areas_d = d.t["vertex_areas"].to(dev)
                _lib.check(L.scb_biot_savart(3, len(positions), _lib.ptr(tgt), n, _lib.ptr(src3),
                                             _lib.ptr(areas_d), _lib.ptr(J), 0.0, scale, 1,
                                             _lib.ptr(A2), _lib.stream_ptr()))
                Axy = A2.cpu().numpy()
            A = np.concatenate([Axy, np.zeros_like(Axy[:, :1])], axis=1)
            out[name] = _u.Quantity(A, units) if with_units else A
        if return_sum:
            return sum(out.values())
        return out


class _FilmBatch(NamedTuple):
    """One film's share of a staged batch evaluation."""

    name: str
    src: np.ndarray                # (n, 3) vertices and layer height (meters; length units for the vector potential)
    areas: np.ndarray              # (n,) vertex areas (square meters; squared length units)
    J: Any                         # pinned (B, n, 2) current densities (A / m; current / length units)
    out_idx: Optional[np.ndarray]  # positions evaluated by the pair sum (None: all of them)
    in_idx: Optional[np.ndarray]   # positions inside the film, in its plane
    in_field: Optional[np.ndarray]  # (B, len(in_idx)) interpolated self field (Bz) there, tesla


class _FieldBatchStage(NamedTuple):
    """Host side of the batch evaluators: checked inputs and staged arrays, no device work."""

    B: int
    m: int
    targets: Any                   # pinned (m, 3) evaluation points (meters; length units for the vector potential)
    films: List[_FilmBatch]
    kind: int                      # scb_biot_savart kind: 1 Bz, 2 (Bx, By, Bz), 3 vector potential
    prefactor: float
    chunked: bool                  # targets in _EVAL_CHUNK launches (biot_savart_2d) or all in one launch
    factors: Tuple[float, ...]     # unit factors applied to every film's result in turn (tesla -> ... -> units)
    units: str
    applied: Optional[np.ndarray]  # field_at_position: (k, m) distinct applied-field rows, in units
    applied_row: Optional[np.ndarray]  # (B,) row of ``applied`` of every entry


# B * points * components of one film's device result: bounds that buffer to 512 MiB by evaluating the entries in
# groups (a group of sets changes no bit of a pair sum, a chunk of targets would)
_BATCH_RESULT_ELEMS = 1 << 26


def _interp_batch(mesh, rows: Sequence[Optional[np.ndarray]], xy: np.ndarray) -> np.ndarray:
    """``interp_field`` of B datasets on one mesh at the same points (the triangles are located once): (B, q),
    zero outside the mesh and where the value is not finite."""
    out = np.zeros((len(rows), len(xy)))
    if len(xy) == 0:
        return out
    ok, tri, w = _locate(mesh.sites, mesh.elements, xy, 16)
    for b, values in enumerate(rows):  # (a missing dataset, such as field_from_other_films of one film, is zero)
        if values is not None:
            out[b] = np.einsum("qk,qk->q", w, np.asarray(values, dtype=float)[mesh.elements[tri]])
    out[:, ~ok] = 0
    out[~np.isfinite(out)] = 0
    return out


def _stage_field_batch(solutions, positions, zs, interp_method: str, units: Optional[str], what: str = "field",
                       vector: bool = False) -> _FieldBatchStage:
    """``what``: "field" (field_at_position), "screening" (screening_field_at_position, Bz or with ``vector`` the
    vector field) or "vector_potential" (vector_potential_at_position).  The operands are those of the per-solution
    methods: meters and A / m for the fields (biot_savart_2d), length and current units for the vector potential."""
    import torch

    solutions = list(solutions)
    for b, sol in enumerate(solutions):
        if not isinstance(sol, Solution):
            raise TypeError(f"solutions[{b}] is a {type(sol).__name__}, not a Solution.")
    positions, zs = _normalize_positions(positions, zs, np.float64)
    B, m = len(solutions), len(positions)
    kind = 3 if what == "vector_potential" else (2 if vector else 1)
    if B == 0:
        return _FieldBatchStage(0, m, None, [], kind, 1.0, True, (), units, None, None)
    first = solutions[0]
    device = first.device
    film_names = list(device.films)
    for b, sol in enumerate(solutions):
        d = sol.device
        if list(d.films) != film_names:
            raise ValueError(f"solutions[{b}] has the films {list(d.films)}, solutions[0] has {film_names}.")
        if d.length_units != device.length_units:
            raise ValueError(f"solutions[{b}] has length_units {d.length_units!r}, solutions[0] has "
                             f"{device.length_units!r}.")
        if sol.field_units != first.field_units or sol.current_units != first.current_units:
            raise ValueError(f"solutions[{b}] has units ({sol.field_units!r}, {sol.current_units!r}), solutions[0] "
                             f"has ({first.field_units!r}, {first.current_units!r}).")
        for name in film_names:
            if name not in sol.film_solutions:
                raise ValueError(f"solutions[{b}] holds no solution of film {name!r} (a solve_batch(gather=False) "
                                 f"result holds only the films of its rank).")
            mesh, mesh0 = d.meshes[name], device.meshes[name]
            if mesh is not mesh0 and not (np.array_equal(mesh.sites, mesh0.sites)
                                          and np.array_equal(mesh.elements, mesh0.elements)):
                raise ValueError(f"solutions[{b}] has another mesh of film {name!r} than solutions[0].")
            z0, z0_first = d.layers[d.films[name].layer].z0, device.layers[device.films[name].layer].z0
            if z0 != z0_first:
                raise ValueError(f"solutions[{b}] has film {name!r} at z0 = {z0}, solutions[0] at z0 = {z0_first}.")
    field_units, current_units, length_units = first.field_units, first.current_units, device.length_units
    if what == "vector_potential":
        for name, film in device.films.items():  # (as vector_potential_at_position raises it)
            if np.all(zs - device.layers[film.layer].z0 == 0) and film.contains_points(positions).all():
                raise ValueError(f"Cannot evaluate vector potential inside the film ({name!r}).")
        in_plane = [False] * len(film_names)
        units = units or f"({field_units}) * ({length_units})"
        to_meter = to_amp_per_meter = 1.0  # (multiplying by one is exact: the operands of the per-solution call)
        prefactor = (_u.MU_0 / (4 * np.pi) * _u.conversion_factor(current_units, "A")
                     * _u.conversion_factor("T * m", units))
        factors: Tuple[float, ...] = ()
    else:
        in_plane = [np.all(zs == device.layers[film.layer].z0) for film in device.films.values()]
        if interp_method != "linear" and any(in_plane):  # (as interp_field raises it)
            raise NotImplementedError("Only linear interpolation is available.")
        units = units or field_units
        to_meter = _u.conversion_factor(length_units, "m")
        to_amp_per_meter = _u.conversion_factor(f"({current_units}) / ({length_units})", "A / m")
        prefactor = _MU0_BIOT_SAVART / (4 * np.pi)
        # field_at_position converts the screening fields to field_units, then everything to units
        factors = ((_field_factor("tesla", field_units), _field_factor(field_units, units)) if what == "field"
                   else (_field_factor("tesla", units),))
    # (the same host arithmetic as biot_savart_2d, so the device sees the same operands)
    targets = torch.empty((m, 3), dtype=torch.float64, pin_memory=True)
    ev = targets.numpy()
    np.multiply(positions[:, 0], to_meter, out=ev[:, 0])
    np.multiply(positions[:, 1], to_meter, out=ev[:, 1])
    np.multiply(np.broadcast_to(zs, (m,)), to_meter, out=ev[:, 2])
    films = []
    for (name, film), plane in zip(device.films.items(), in_plane):
        mesh = device.meshes[name]
        z0 = device.layers[film.layer].z0
        out_idx = in_idx = in_field = None
        if plane:
            in_film = film.contains_points(positions)
            in_idx, out_idx = np.flatnonzero(in_film), np.flatnonzero(~in_film)
            in_field = _interp_batch(mesh, [s.film_solutions[name].self_field for s in solutions], positions[in_idx])
            if field_units != "tesla":
                from .solver.utils import convert_field

                in_field = convert_field(in_field, "tesla", old_units=field_units, with_units=False)
            if len(out_idx) == m:
                out_idx = in_idx = in_field = None
        n = len(mesh.sites)
        src = np.ascontiguousarray(np.concatenate([mesh.sites * to_meter, (z0 * np.ones(n) * to_meter)[:, None]],
                                                  axis=1), dtype=np.float64)
        areas = np.ascontiguousarray(np.asarray(mesh.vertex_areas) * to_meter**2, dtype=np.float64)
        J = torch.empty((B, n, 2), dtype=torch.float64, pin_memory=True)
        Jh = J.numpy()
        for b, sol in enumerate(solutions):
            Jh[b] = np.atleast_2d(sol.film_solutions[name].current_density) * to_amp_per_meter
        films.append(_FilmBatch(name, src, areas, J, out_idx, in_idx, in_field))
    if what != "field":
        return _FieldBatchStage(B, m, targets, films, kind, prefactor, what != "vector_potential", factors, units,
                                None, None)

    # applied field (field_at_position): interpolated from the solutions at in-plane points inside a film, the
    # applied-field function elsewhere -- evaluated once per distinct function object
    in_film = np.zeros(m, dtype=bool)
    per_entry = None
    films_by_layer = device.polygons_by_layer("film")
    for lname, layer in device.layers.items():
        if np.all(zs == layer.z0):
            per_entry = np.zeros((B, m))
            for film in films_by_layer[lname]:
                ix = film.contains_points(positions)
                in_film[ix] = True
                mesh, xy = device.meshes[film.name], positions[ix]
                fss = [s.film_solutions[film.name] for s in solutions]
                per_entry[:, ix] = (_interp_batch(mesh, [fs.applied_field for fs in fss], xy)
                                    + _interp_batch(mesh, [fs.field_from_other_films for fs in fss], xy))
            break
    mask = ~in_film
    func_row: Dict[int, int] = {}
    rows = []
    applied_row = np.empty(B, dtype=np.int64)
    for b, sol in enumerate(solutions):
        func = sol.applied_field_func
        k = func_row.get(id(func))
        if k is None and mask.any():
            value = np.squeeze(func(positions[mask, 0], positions[mask, 1], zs[mask, np.newaxis]))
            rows.append(np.broadcast_to(np.asarray(value, dtype=np.float64), (int(mask.sum()),)))
        if k is None:
            k = func_row[id(func)] = len(func_row)
        applied_row[b] = k
    if per_entry is None:
        applied = np.stack(rows) if rows else np.zeros((len(func_row), m))
    else:
        if mask.any():
            for b in range(B):
                per_entry[b, mask] = rows[applied_row[b]]
        applied, applied_row = per_entry, np.arange(B)
    to_units = factors[1]
    if to_units != 1.0:
        applied = applied * to_units
    return _FieldBatchStage(B, m, targets, films, kind, prefactor, True, factors, units, applied, applied_row)


def _evaluate_field_batch(stage: _FieldBatchStage, return_sum: bool):
    """Device side of the batch evaluators: for every group of entries, one multi-set pair sum per film (and chunk
    of targets), the unit factors and the sum over films on the device, one copy of every group's result to the
    host.  Returns (B, m) arrays (Bz) or (B, m, 3) arrays (vector field, vector potential with a zero z column)."""
    import torch

    L = _lib.lib()
    B, m = stage.B, stage.m
    tail = () if stage.kind == 1 else (3,)
    ncomp = 3 if stage.kind == 2 else (2 if stage.kind == 3 else 1)  # components the pair sum writes
    group = max(1, min(B, _BATCH_RESULT_ELEMS // max(m * (1 if stage.kind == 1 else 3), 1)))
    dev = torch.device(f"cuda:{torch.cuda.current_device()}")
    with torch.cuda.device(dev):
        targets = stage.targets.to(dev, non_blocking=True)
        per_film = []  # (sources, areas, targets of the pair sum, their indices or None) of every film
        for f in stage.films:
            src, areas = (torch.as_tensor(a).to(dev, non_blocking=True) for a in (f.src, f.areas))
            out_idx = None if f.out_idx is None else torch.as_tensor(f.out_idx).to(dev)
            per_film.append((src, areas, targets if out_idx is None else targets.index_select(0, out_idx), out_idx))
        applied = None
        if return_sum and stage.applied is not None:
            applied = torch.as_tensor(stage.applied).to(dev)
            applied_row = torch.as_tensor(stage.applied_row).to(dev)
        keys = ["total"] if return_sum else [f.name for f in stage.films]
        host = {key: torch.empty((B, m) + tail, dtype=torch.float64, pin_memory=True) for key in keys}
        for g0 in range(0, B, group):
            g1 = min(B, g0 + group)
            G = g1 - g0
            total, fields = None, {}
            for f, (src, areas, tgt, out_idx) in zip(stage.films, per_film):
                J = f.J[g0:g1].to(dev, non_blocking=True)
                field = torch.empty((G, m) + tail, dtype=torch.float64, device=dev)
                if stage.kind == 3:
                    field[..., 2] = 0.0
                if f.in_idx is not None:
                    in_idx = torch.as_tensor(f.in_idx).to(dev)
                    in_field = torch.as_tensor(f.in_field[g0:g1]).to(dev)
                    if stage.kind == 1:
                        field[:, in_idx] = in_field
                    else:  # (the in-plane self field has a z component only)
                        block = torch.zeros((G, len(f.in_idx), 3), dtype=torch.float64, device=dev)
                        block[..., 2] = in_field
                        field[:, in_idx] = block
                # the chunks of biot_savart_2d: the source split of the pair sum, hence every bit of it, depends on
                # the number of targets of a launch (vector_potential_at_position: all targets in one launch)
                mf = int(tgt.shape[0])
                chunk = mf if (mf <= _EVAL_CHUNK or not stage.chunked) else _EVAL_CHUNK
                for lo in range(0, mf, max(chunk, 1)):
                    hi = min(mf, lo + chunk)
                    direct = out_idx is None and hi - lo == m and stage.kind != 3
                    out = field if direct else torch.empty((G, hi - lo) + (() if ncomp == 1 else (ncomp,)),
                                                           dtype=torch.float64, device=dev)
                    _lib.check(L.scb_biot_savart(stage.kind, hi - lo, _lib.ptr(tgt[lo:hi]), int(src.shape[0]),
                                                 _lib.ptr(src), _lib.ptr(areas), _lib.ptr(J), 0.0, stage.prefactor,
                                                 G, _lib.ptr(out), _lib.stream_ptr()))
                    if direct:
                        continue
                    rows = slice(lo, hi) if out_idx is None else out_idx[lo:hi]
                    if stage.kind == 3:
                        field[:, rows, :2] = out
                    else:
                        field[:, rows] = out
                # unit factors, then films in device order: the operations of the per-solution methods
                for factor in stage.factors:
                    if factor != 1.0:
                        field.mul_(factor)
                if not return_sum:
                    fields[f.name] = field
                elif total is None:
                    total = field
                else:
                    total.add_(field)
            if return_sum:
                if applied is not None:
                    rows_g = applied.index_select(0, applied_row[g0:g1])
                    if total is None:
                        total = rows_g
                    else:
                        total.add_(rows_g)
                elif total is None:
                    total = torch.zeros((G, m) + tail, dtype=torch.float64, device=dev)
                fields = {"total": total}
            for key, t in fields.items():
                host[key][g0:g1].copy_(t, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
    if return_sum:
        return host["total"].numpy()
    out = {key: t.numpy() for key, t in host.items()}
    if stage.applied is not None:
        out["applied_field"] = stage.applied[stage.applied_row]
    return out


def _batch_result(stage: _FieldBatchStage, return_sum: bool, with_units: bool, tail: tuple = ()):
    value = _evaluate_field_batch(stage, return_sum) if stage.B else (np.empty((0, stage.m) + tail) if return_sum
                                                                      else {})
    if not with_units or (stage.B == 0 and stage.units is None):
        return value
    if return_sum:
        return _u.Quantity(value, stage.units)
    return {key: _u.Quantity(v, stage.units) for key, v in value.items()}


def field_at_position_batch(solutions: Sequence["Solution"], positions, *, zs=None, interp_method: str = "linear",
                            units: Optional[str] = None, with_units: bool = True, return_sum: bool = True):
    """``Solution.field_at_position`` of B solutions of one device (e.g. the entries of a ``solve_batch``) at the
    same positions, in one pass: row ``b`` is ``solutions[b].field_at_position(positions, zs=zs,
    interp_method=interp_method, units=units, with_units=False, return_sum=return_sum)``.

    Returns a ``(B, m)`` array (a ``Quantity`` with ``with_units``), or with ``return_sum=False`` a dict of
    ``(B, m)`` arrays, one per film and ``"applied_field"``.  Every film's field at the points off its plane is one
    pair sum over all B current densities (one r^-3 per pair serves the B entries), and its bits are those of the
    per-solution call.  The solutions must share the films, their meshes and heights, the length units, the field
    units and the current units; each must hold every film.  Applied-field functions are evaluated once per
    distinct function object."""
    stage = _stage_field_batch(solutions, positions, zs, interp_method, units)
    return _batch_result(stage, return_sum, with_units)


def screening_field_at_position_batch(solutions: Sequence["Solution"], positions, *, zs=None, vector: bool = False,
                                      interp_method: str = "linear", units: Optional[str] = None,
                                      with_units: bool = True, return_sum: bool = True):
    """``Solution.screening_field_at_position`` of B solutions of one device at the same positions, in one pass:
    row ``b`` is ``solutions[b].screening_field_at_position(positions, zs=zs, vector=vector,
    interp_method=interp_method, units=units, with_units=False, return_sum=return_sum)``.

    Returns a ``(B, m)`` array, ``(B, m, 3)`` with ``vector=True`` (a ``Quantity`` with ``with_units``), or with
    ``return_sum=False`` a dict of such arrays, one per film.  Every film's field at the points off its plane is one
    pair sum over all B current densities (one r^-3 per pair serves up to 8 entries), with the bits of the
    per-solution call; at in-plane points inside a film the film's self field is interpolated, as there.  The
    solutions must meet the conditions of ``field_at_position_batch``."""
    stage = _stage_field_batch(solutions, positions, zs, interp_method, units, what="screening", vector=vector)
    return _batch_result(stage, return_sum, with_units, (3,) if vector else ())


def vector_potential_at_position_batch(solutions: Sequence["Solution"], positions, *, zs=None,
                                       units: Optional[str] = None, with_units: bool = True, return_sum: bool = True):
    """``Solution.vector_potential_at_position`` of B solutions of one device at the same positions, in one pass: a
    ``(B, m, 3)`` array (zero z column) whose row ``b`` is ``solutions[b].vector_potential_at_position(positions,
    zs=zs, units=units, with_units=False, return_sum=return_sum)``, bit for bit (a ``Quantity`` with
    ``with_units``), or with ``return_sum=False`` a dict of such arrays, one per film.  One pair sum per film serves
    all B current densities (one r^-1 per pair for up to 8 entries).  Raises the ``ValueError`` of the per-solution
    method when every position lies inside a film in its plane, before any device work.  The solutions must meet
    the conditions of ``field_at_position_batch``."""
    stage = _stage_field_batch(solutions, positions, zs, "linear", units, what="vector_potential")
    return _batch_result(stage, return_sum, with_units, (3,))


# interpolated values per chunk of targets (B * points * components): bounds the device output buffer to 512 MiB
_INTERP_CHUNK_ELEMS = 1 << 26


def _stage_interp_batch(solutions, positions, film: str, method: str):
    """Host checks of the interpolation batches: (solutions, positions (m, 2)); raises before any device work."""
    solutions = list(solutions)
    for b, sol in enumerate(solutions):
        if not isinstance(sol, Solution):
            raise TypeError(f"solutions[{b}] is a {type(sol).__name__}, not a Solution.")
    if method != "linear":
        raise NotImplementedError("Only linear interpolation is available.")
    positions = np.ascontiguousarray(np.atleast_2d(np.asarray(positions, dtype=np.float64))[:, :2])
    if not solutions:
        return solutions, positions
    first = solutions[0]
    for b, sol in enumerate(solutions):
        d = sol.device
        if film not in d.films:
            raise ValueError(f"solutions[{b}] has no film {film!r} (films: {list(d.films)}).")
        if film not in sol.film_solutions:
            raise ValueError(f"solutions[{b}] holds no solution of film {film!r} (a solve_batch(gather=False) "
                             f"result holds only the films of its rank).")
        mesh, mesh0 = d.meshes[film], first.device.meshes[film]
        if mesh is not mesh0 and not (np.array_equal(mesh.sites, mesh0.sites)
                                      and np.array_equal(mesh.elements, mesh0.elements)):
            raise ValueError(f"solutions[{b}] has another mesh of film {film!r} than solutions[0].")
        if (sol.field_units, sol.current_units, d.length_units) != (first.field_units, first.current_units,
                                                                    first.device.length_units):
            raise ValueError(f"solutions[{b}] has units ({sol.field_units!r}, {sol.current_units!r}, "
                             f"{d.length_units!r}), solutions[0] has ({first.field_units!r}, "
                             f"{first.current_units!r}, {first.device.length_units!r}).")
    return solutions, positions


def _interp_batch_device(mesh, rows: Sequence[Optional[np.ndarray]], ncomp: int, positions: np.ndarray, polygon,
                         scale: float) -> np.ndarray:
    """Device side of the interpolation batches: (B, m, ncomp) values of the B value sets ``rows`` (None: zeros)
    at ``positions``.  The targets run in chunks of ``_INTERP_CHUNK_ELEMS // (B ncomp)`` points: each chunk is
    located and masked once for all B sets; the device holds the mesh, its grid, the B value sets, the positions
    and one chunk of results; every chunk is copied back behind its kernels, one synchronisation at the end."""
    import torch

    from . import interp

    B, m = len(rows), len(positions)
    n = len(mesh.sites)
    dev = torch.device(f"cuda:{torch.cuda.current_device()}")
    with torch.cuda.device(dev):
        grid = interp.tri_grid(mesh.sites, mesh.elements)
        vals = torch.empty((B, n, ncomp), dtype=torch.float64, pin_memory=True)
        vh = vals.numpy()
        for b, v in enumerate(rows):
            if v is None:
                vh[b] = 0.0
            else:
                vh[b] = np.asarray(v, dtype=np.float64).reshape(n, ncomp)
        pos_pin = torch.empty((m, 2), dtype=torch.float64, pin_memory=True)
        pos_pin.numpy()[:] = positions
        vals_d = vals.to(dev, non_blocking=True)
        xy_d = pos_pin.to(dev, non_blocking=True)
        rings = interp.upload_rings(polygon, dev) if polygon is not None else None
        host = torch.empty((B, m, ncomp), dtype=torch.float64, pin_memory=True)
        chunk = max(1, min(m, _INTERP_CHUNK_ELEMS // max(B * ncomp, 1)))
        # one set of chunk buffers: every use is ordered on this stream behind the copy of the previous chunk
        tri = torch.empty(chunk, dtype=torch.int64, device=dev)
        bary = torch.empty((chunk, 3), dtype=torch.float64, device=dev)
        inside = torch.empty(chunk, dtype=torch.uint8, device=dev) if rings is not None else None
        out = torch.empty((B, chunk, ncomp), dtype=torch.float64, device=dev)
        for lo in range(0, m, chunk):
            hi = min(m, lo + chunk)
            c = hi - lo
            xy = xy_d[lo:hi]
            interp.locate(grid, xy, tri[:c], bary[:c])
            if rings is not None:
                interp.polygon_mask(rings, xy, inside[:c])
            o = out if c == chunk else torch.empty((B, c, ncomp), dtype=torch.float64, device=dev)
            interp.interpolate(grid, tri[:c], bary[:c], vals_d, o, None if inside is None else inside[:c], scale)
            if c == m:
                host.copy_(o, non_blocking=True)
            else:
                for b in range(B):
                    host[b, lo:hi].copy_(o[b], non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
    return host.numpy()


def interp_current_density_batch(solutions: Sequence["Solution"], positions, *, film: str, method: str = "linear",
                                 units: Optional[str] = None, with_units: bool = False):
    """``Solution.interp_current_density`` of B solutions of one device at the same positions, on the GPU: a
    ``(B, m, 2)`` array whose row ``b`` is ``solutions[b].interp_current_density(positions, film=film,
    method=method, units=units, with_units=False)`` (a ``Quantity`` with ``with_units``).

    The positions are located in the film's mesh once for all entries (the triangle with the largest smallest
    barycentric coordinate, scb_tri_locate) and masked by the film polygon once; where the host and the device
    choose the same triangle the values carry the host's bits.  The solutions must share the film's mesh and
    their units, and each must hold the film.  Only ``method="linear"`` is available."""
    solutions, positions = _stage_interp_batch(solutions, positions, film, method)
    m = len(positions)
    if not solutions:
        J = np.zeros((0, m, 2))
        return _u.Quantity(J, units) if with_units and units is not None else J
    first = solutions[0]
    device = first.device
    default_units = f"({first.current_units}) / ({device.length_units})"
    scale = 1.0
    if units is not None and units != default_units:
        scale = _u.conversion_factor(default_units, units)
    J = np.zeros((len(solutions), m, 2))
    if m:
        J = _interp_batch_device(device.meshes[film], [s.film_solutions[film].current_density for s in solutions], 2,
                                 positions, device.films[film], scale)
    return _u.Quantity(J, units or default_units) if with_units else J


def interp_field_batch(solutions: Sequence["Solution"], positions, *, film: str, dataset: str = "total_field",
                       method: str = "linear", units: Optional[str] = None, with_units: bool = False):
    """``Solution.interp_field`` of B solutions of one device at the same positions, on the GPU: a ``(B, m)`` array
    whose row ``b`` is ``solutions[b].interp_field(positions, film=film, dataset=dataset, method=method,
    units=units, with_units=False)`` (a ``Quantity`` with ``with_units``).  A dataset that is None (e.g.
    ``field_from_other_films`` of a single film) gives a zero row; ``total_field`` interpolates the host array of
    ``FilmSolution.total_field``.  Located once for all entries, as ``interp_current_density_batch``."""
    valid = ("total_field", "applied_field", "self_field", "field_from_other_films")
    if dataset not in valid:
        raise ValueError(f"Unexpected dataset: {dataset}.")
    solutions, positions = _stage_interp_batch(solutions, positions, film, method)
    m = len(positions)
    if not solutions:
        out = np.zeros((0, m))
        return _u.Quantity(out, units) if with_units and units is not None else out
    field_units = solutions[0].field_units
    convert = units is not None and units != field_units
    rows = [getattr(s.film_solutions[film], dataset) for s in solutions]
    out = np.zeros((len(solutions), m))
    if m and any(r is not None for r in rows):
        mesh = solutions[0].device.meshes[film]
        scale = _field_factor(field_units, units) if convert else 1.0
        out = _interp_batch_device(mesh, rows, 1, positions, None, scale)[:, :, 0]
    if with_units:
        return _u.Quantity(out, units if convert else field_units)
    return out


_FIELD_FACTORS: Dict[tuple, float] = {}


def _field_factor(old_units: str, new_units: str) -> float:
    """The ``convert_field`` factor from ``old_units`` to ``new_units``, looked up once per unit pair."""
    from .solver.utils import convert_field

    key = (str(old_units), str(new_units))
    factor = _FIELD_FACTORS.get(key)
    if factor is None:
        factor = _FIELD_FACTORS[key] = float(convert_field(1.0, new_units, old_units=old_units, with_units=False))
    return factor


def _convert_owned(value, new_units: str, old_units: str, with_units: bool, owned: bool = True):
    """``convert_field`` for an array this module has just produced itself (a million-point field evaluation
    makes half a dozen such passes): the factor is looked up once per unit pair, a factor of one costs nothing
    and the scaling is done in place."""
    factor = _field_factor(old_units, new_units)
    if factor != 1.0:
        if owned and isinstance(value, np.ndarray) and value.flags.writeable and value.dtype == np.float64:
            np.multiply(value, factor, out=value)
        else:
            value = value * factor
    return _u.Quantity(value, new_units) if with_units else value


def _sum_owned(fields: Dict[str, Any], with_units: bool, not_owned: Sequence[str] = ()):
    """Sum of the per-source fields (reference: ``sum(fields.values())``), accumulated in place in the first
    array (which this module produced itself; entries named in ``not_owned`` are never written to)."""
    if with_units:
        return sum(fields.values())
    total = None
    for key, f in fields.items():
        if total is None:
            own = key not in not_owned and isinstance(f, np.ndarray) and f.flags.writeable and f.dtype == np.float64
            total = f if own else np.array(f, dtype=np.float64)
        elif np.shape(f) == total.shape or np.ndim(f) == 0:
            np.add(total, f, out=total)
        else:
            total = total + f
    return 0 if total is None else total


def _flux_conversion(old: str, new: str) -> float:
    """Flux units may be given as B*area (e.g. mT*um**2) or H*area; only B*area <-> Wb-like is needed."""
    return _u.conversion_factor(old, new)
