"""Thin Device / Layer / Polygon model: exactly the attributes the solve hot path reads
(reference solver/solve.py:391-409, solver/utils.py:241-304; the full shapely/matplotlib
geometry subsystem of superscreen/device/*.py is out of scope, SURVEY.md section 2a).
"""
from __future__ import annotations

import logging
import numbers
from typing import Callable, Dict, List, Optional, Sequence, Tuple, Union

import numpy as np

from . import units as _u
from .geometry import close_curve, orient_ccw, points_in_polygon
from .mesh import Mesh

logger = logging.getLogger("device")


class Layer:
    """reference device/layer.py: name, Lambda or (london_lambda, thickness), z0."""

    def __init__(self, name: str, Lambda=None, london_lambda=None, thickness=None, z0: float = 0):
        self.name = name
        self.thickness = thickness
        self.london_lambda = london_lambda
        self.z0 = z0
        if Lambda is None:
            if london_lambda is None or thickness is None:
                raise ValueError("Either Lambda or both london_lambda and thickness must be given.")
            self._Lambda = None
        else:
            if london_lambda is not None or thickness is not None:
                raise ValueError("Either Lambda or both london_lambda and thickness must be given (not both).")
            self._Lambda = Lambda

    @property
    def Lambda(self):
        if self._Lambda is not None:
            return self._Lambda
        if callable(self.london_lambda):
            ll, d = self.london_lambda, self.thickness
            return lambda x, y: ll(x, y) ** 2 / d
        return self.london_lambda**2 / self.thickness

    @Lambda.setter
    def Lambda(self, value):
        self._Lambda = value
        self.london_lambda = None
        self.thickness = None

    def to_hdf5(self, h5group) -> None:
        """reference device/layer.py: attributes name, z0, thickness, london_lambda | Lambda"""
        from . import io as _io

        _io.layer_to_hdf5(self, h5group)

    @staticmethod
    def from_hdf5(h5group) -> "Layer":
        from . import io as _io

        return _io.layer_from_hdf5(h5group)

    def copy(self) -> "Layer":
        if self._Lambda is not None:
            return Layer(self.name, Lambda=self._Lambda, z0=self.z0)
        return Layer(self.name, london_lambda=self.london_lambda, thickness=self.thickness, z0=self.z0)


class Polygon:
    """A simply connected polygon in a layer (reference device/polygon.py:28-162).  Points are
    stored closed and counter-clockwise, as the reference does (polygon.py:67-77)."""

    def __init__(self, name: Optional[str] = None, *, layer: Optional[str] = None, points):
        self.name = name
        self.layer = layer
        if isinstance(points, Polygon):
            points = points.points
        pts = np.asarray(points, dtype=float)
        if pts.ndim != 2 or pts.shape[-1] != 2:
            raise ValueError(f"Expected shape (n, 2), but got {pts.shape}.")
        self._points = close_curve(orient_ccw(pts))

    @property
    def points(self) -> np.ndarray:
        return self._points

    @property
    def is_valid(self) -> bool:
        return len(self._points) >= 4

    @property
    def extents(self) -> Tuple[float, float]:
        return tuple(np.ptp(self._points, axis=0))

    @property
    def area(self) -> float:
        """Area enclosed by the polygon (shoelace formula; reference device/polygon.py:93-96)."""
        from .geometry import signed_area

        return float(abs(signed_area(self._points)))

    def set_name(self, name: Optional[str]) -> "Polygon":
        self.name = name
        return self

    def set_layer(self, layer: Optional[str]) -> "Polygon":
        self.layer = layer
        return self

    def _origin(self, origin) -> np.ndarray:
        if isinstance(origin, str):
            if origin == "center":  # centre of the bounding box
                return 0.5 * (self._points.min(axis=0) + self._points.max(axis=0))
            if origin == "centroid":  # centre of mass of the enclosed area
                p = self._points
                cross = p[:-1, 0] * p[1:, 1] - p[1:, 0] * p[:-1, 1]
                return ((p[:-1] + p[1:]) * cross[:, None]).sum(axis=0) / (3.0 * cross.sum())
            raise ValueError(f"Unknown origin: {origin!r}.")
        return np.asarray(origin, dtype=float)

    def _mapped(self, points: np.ndarray, inplace: bool) -> "Polygon":
        polygon = self if inplace else self.copy()
        polygon._points = close_curve(orient_ccw(points))
        return polygon

    def translate(self, dx: float = 0.0, dy: float = 0.0, inplace: bool = False) -> "Polygon":
        """reference device/polygon.py:251-270"""
        return self._mapped(self._points + np.array([dx, dy], dtype=float), inplace)

    def rotate(self, degrees: float, origin=(0.0, 0.0), inplace: bool = False) -> "Polygon":
        """Counter-clockwise rotation about ``origin`` (reference device/polygon.py:226-249)."""
        c, s_ = np.cos(np.radians(degrees)), np.sin(np.radians(degrees))
        o = self._origin(origin)
        return self._mapped((self._points - o) @ np.array([[c, s_], [-s_, c]]) + o, inplace)

    def scale(self, xfact: float = 1.0, yfact: float = 1.0, origin=(0.0, 0.0), inplace: bool = False) -> "Polygon":
        """reference device/polygon.py:272-300 (negative factors mirror the polygon)"""
        o = self._origin(origin)
        return self._mapped((self._points - o) * np.array([xfact, yfact], dtype=float) + o, inplace)

    def union(self, *others, name: Optional[str] = None) -> "Polygon":
        """Union with other polygons / coordinate arrays (reference device/polygon.py:302-340) as a
        ``CompositePolygon`` (membership tests only, no outline)."""
        return CompositePolygon(name or self.name, layer=self.layer, add=[self._points] + _rings_of(others))

    def difference(self, *others, symmetric: bool = False, name: Optional[str] = None) -> "Polygon":
        """This polygon minus others (reference device/polygon.py:378-435), as a ``CompositePolygon``."""
        if symmetric:
            raise NotImplementedError("The symmetric difference needs polygon clipping (shapely); not available.")
        return CompositePolygon(name or self.name, layer=self.layer, add=[self._points], sub=_rings_of(others))

    def on_boundary(self, points, radius: float = 1e-3, index: bool = False):
        """Whether ``points`` lie within ``radius`` of the polygon boundary (reference device/polygon.py:164-190,
        there via matplotlib's path with a positive / negative radius; here by the distance to the nearest edge)."""
        pts = np.atleast_2d(np.asarray(points, dtype=float))
        boundary = np.zeros(len(pts), dtype=bool)
        for ring in self.rings:
            a, b = ring[:-1], ring[1:]
            ab = b - a
            len2 = np.maximum(np.einsum("ij,ij->i", ab, ab), 1e-300)
            for s0 in range(0, len(pts), 4096):  # (bounds the points x edges temporaries)
                q = pts[s0:s0 + 4096]
                t = np.clip(np.einsum("qej,ej->qe", q[:, None, :] - a[None, :, :], ab) / len2, 0.0, 1.0)
                d = np.linalg.norm(q[:, None, :] - (a[None, :, :] + t[:, :, None] * ab[None, :, :]), axis=2)
                boundary[s0:s0 + 4096] |= d.min(axis=1) <= abs(radius)
        if index:
            return np.where(boundary)[0]
        return boundary

    @property
    def rings(self) -> List[np.ndarray]:
        """The closed ring(s) that make up the polygon."""
        return [self._points]

    _mask_cache: Dict[tuple, np.ndarray] = {}

    def contains_points(self, points, index: bool = False, radius: float = 0):
        pts = np.atleast_2d(points)
        if len(pts) >= 16:
            # the same (polygon, points) query is repeated for every fluxoid / film-info evaluation;
            # memoise on the full content (a digest of the float64 bytes for large point sets)
            raw = np.ascontiguousarray(pts, dtype=float)
            if len(pts) >= 1024:
                import hashlib

                key = (self._points.tobytes(), pts.shape, hashlib.blake2b(raw.data, digest_size=16).digest())
            else:
                key = (self._points.tobytes(), pts.shape, raw.tobytes())
            mask = Polygon._mask_cache.get(key)
            if mask is None:
                if len(Polygon._mask_cache) > 1024:
                    Polygon._mask_cache.clear()
                mask = points_in_polygon(self._points, pts)
                mask.setflags(write=False)
                Polygon._mask_cache[key] = mask
        else:
            mask = points_in_polygon(self._points, pts)
        if index:
            return np.where(mask)[0]
        return mask

    def make_mesh(self, min_points: Optional[int] = None, max_edge_length: Optional[float] = None,
                  convex_hull: bool = False, smooth: int = 0, build_operators: bool = False, **meshpy_kwargs):
        """Creates a :class:`Mesh` for the polygon on the GPU (reference device/polygon.py:192-224)."""
        from . import meshgen
        from .mesh import Mesh as _Mesh

        points, triangles = meshgen.generate_mesh(self.points, min_points=min_points, max_edge_length=max_edge_length,
                                                  convex_hull=convex_hull, **meshpy_kwargs)
        mesh = _Mesh.from_triangulation(points, triangles, build_operators=build_operators and not smooth)
        return mesh.smooth(smooth, build_operators=build_operators) if smooth else mesh

    def to_hdf5(self, h5group) -> None:
        """reference device/polygon.py: attributes name, layer and the dataset ``points``"""
        from . import io as _io

        _io.polygon_to_hdf5(self, h5group)

    @staticmethod
    def from_hdf5(h5group) -> "Polygon":
        from . import io as _io

        return _io.polygon_from_hdf5(h5group)

    def resample(self, num_points: Optional[int] = None) -> "Polygon":
        """A copy whose vertices are uniformly distributed in arc length along the boundary (reference
        device/polygon.py:483-506: shapely ``segmentize`` + ``interpolate(linspace(0, 1, num_points), normalized=True)``,
        i.e. piecewise-linear interpolation of the closed boundary).  ``num_points=None``: as many as now; a false
        ``num_points`` returns an unaltered copy."""
        if num_points is None:
            num_points = len(self.points)
        if not num_points:
            return self.copy()
        pts = self.points
        closed = pts if np.allclose(pts[0], pts[-1]) else np.concatenate([pts, pts[:1]])
        arc = np.concatenate([[0.0], np.cumsum(np.linalg.norm(np.diff(closed, axis=0), axis=1))])
        t = np.linspace(0.0, 1.0, int(num_points)) * arc[-1]
        new = np.stack([np.interp(t, arc, closed[:, k]) for k in range(2)], axis=1)
        return Polygon(self.name, layer=self.layer, points=new)

    def copy(self) -> "Polygon":
        # the stored points are already closed and counter-clockwise: skip the constructor's normalisation
        new = object.__new__(Polygon)
        new.name, new.layer, new._points = self.name, self.layer, self._points.copy()
        return new

    def __repr__(self):
        return f"Polygon(name={self.name!r}, layer={self.layer!r}, points=<{len(self._points)} x 2>)"


class CompositePolygon(Polygon):
    """Union / difference of simple polygons, as far as the solve path needs it: membership tests.

    Stands in for the shapely-backed ``Polygon.union`` / ``Polygon.difference`` of the reference
    (device/polygon.py:302-435).  The resulting outline is never computed: a point is inside when it is
    inside any of the ``add`` rings and inside none of the ``sub`` rings, which is all that
    ``make_film_info`` (index sets), ``holes_by_film`` and the fluxoid checks ask of a film or hole.
    ``points`` is the concatenation of the closed ``add`` rings (a point cloud that covers the outline,
    NOT one ordered ring); ``rings`` gives the individual closed rings, e.g. for meshing."""

    def __init__(self, name: Optional[str] = None, *, layer: Optional[str] = None, add, sub=()):
        self.name = name
        self.layer = layer
        self._add = [close_curve(orient_ccw(np.asarray(r, dtype=float))) for r in add]
        self._sub = [close_curve(orient_ccw(np.asarray(r, dtype=float))) for r in sub]
        if not self._add:
            raise ValueError("A composite polygon needs at least one ring.")
        self._points = np.concatenate(self._add, axis=0)

    @property
    def rings(self) -> List[np.ndarray]:
        return list(self._add)

    @property
    def cut_rings(self) -> List[np.ndarray]:
        return list(self._sub)

    @property
    def area(self) -> float:
        raise NotImplementedError("The area of a composite polygon is not available (no outline is computed).")

    def _mapped(self, points, inplace):
        raise NotImplementedError("Affine maps of composite polygons are not supported; transform the parts.")

    def translate(self, dx: float = 0.0, dy: float = 0.0, inplace: bool = False) -> "CompositePolygon":
        """Every ring moved by ``(dx, dy)``, as ``Polygon.translate`` moves its points (so that
        ``Device.translate`` and the translated entries of ``solve_batch`` can move a composite film or hole)."""
        shift = np.array([dx, dy], dtype=float)
        polygon = self if inplace else self.copy()
        polygon._add = [close_curve(orient_ccw(r + shift)) for r in self._add]
        polygon._sub = [close_curve(orient_ccw(r + shift)) for r in self._sub]
        polygon._points = np.concatenate(polygon._add, axis=0)
        return polygon

    def contains_points(self, points, index: bool = False, radius: float = 0):
        pts = np.atleast_2d(points)
        mask = np.zeros(len(pts), dtype=bool)
        for ring in self._add:
            mask |= Polygon.contains_points(_ring_polygon(ring), pts)
        for ring in self._sub:
            mask &= ~Polygon.contains_points(_ring_polygon(ring), pts)
        return np.where(mask)[0] if index else mask

    def union(self, *others, name: Optional[str] = None) -> "CompositePolygon":
        return CompositePolygon(name or self.name, layer=self.layer, add=self._add + _rings_of(others), sub=self._sub)

    def difference(self, *others, symmetric: bool = False, name: Optional[str] = None) -> "CompositePolygon":
        if symmetric:
            raise NotImplementedError("The symmetric difference needs polygon clipping (shapely); not available.")
        return CompositePolygon(name or self.name, layer=self.layer, add=self._add, sub=self._sub + _rings_of(others))

    def copy(self) -> "CompositePolygon":
        return CompositePolygon(self.name, layer=self.layer, add=[r.copy() for r in self._add],
                                sub=[r.copy() for r in self._sub])

    def __repr__(self):
        return (f"CompositePolygon(name={self.name!r}, layer={self.layer!r}, "
                f"rings={len(self._add)}, cut_rings={len(self._sub)})")


def _ring_polygon(ring: np.ndarray) -> Polygon:
    """A plain Polygon over an already closed, counter-clockwise ring (no re-normalisation)."""
    new = object.__new__(Polygon)
    new.name, new.layer, new._points = None, None, ring
    return new


def _rings_of(items) -> List[np.ndarray]:
    rings = []
    for it in items:
        if isinstance(it, CompositePolygon):
            if it.cut_rings:
                raise NotImplementedError("Cannot combine with a composite polygon that has cut-outs.")
            rings.extend(it.rings)
        elif isinstance(it, Polygon):
            rings.append(it.points)
        else:
            rings.append(np.asarray(it, dtype=float))
    return rings


def _as_dict(items):
    if items is None:
        return {}
    if isinstance(items, dict):
        items = list(items.values())
    return {it.name: it for it in items}


class Device:
    """reference device/device.py:40-127 (constructor), :157-240 (layer/film queries, copy)."""

    def __init__(self, name: str, *, layers, films, holes=None, terminals=None, abstract_regions=None,
                 length_units: str = "um", solve_dtype="float64"):
        self.name = name
        self.layers: Dict[str, Layer] = _as_dict(layers)
        self.films: Dict[str, Polygon] = _as_dict(films)
        self.holes: Dict[str, Polygon] = _as_dict(holes)
        self.terminals: Dict[str, List[Polygon]] = terminals or {}
        if not set(self.terminals).issubset(self.films):
            raise ValueError(f"terminals.keys() must be a subset of films.keys() ({list(self.films)!r}).")
        for film_name, film_terminals in self.terminals.items():
            for terminal in film_terminals:
                terminal.layer = self.films[film_name].layer
        self.abstract_regions: Dict[str, Polygon] = _as_dict(abstract_regions)
        for polygons, label in [(self.films.values(), "film"), (self.holes.values(), "hole")]:
            for polygon in polygons:
                if not polygon.is_valid:
                    raise ValueError(f"The following {label} is not valid: {polygon}.")
                if polygon.layer not in self.layers:
                    raise ValueError(
                        f"The following {label} is assigned to a layer that doesn not "
                        f"exist in the device: {polygon}."
                    )
        self._length_units = length_units
        self.solve_dtype = solve_dtype
        self.meshes: Optional[Dict[str, Mesh]] = None

    ureg = _u  # the module plays the role of the reference's pint registry

    @property
    def length_units(self) -> str:
        return self._length_units

    @property
    def solve_dtype(self) -> np.dtype:
        return self._solve_dtype

    @solve_dtype.setter
    def solve_dtype(self, dtype) -> None:
        try:
            _ = np.finfo(dtype)
        except ValueError as e:
            raise ValueError(f"Invalid float dtype: {dtype}") from e
        if np.dtype(dtype) != np.float64:
            logger.info("superscreen_b200 computes in float64; solve_dtype only sets output dtype.")
        self._solve_dtype = np.dtype(dtype)

    def polygons_by_layer(self, polygon_type: Optional[str] = None) -> Dict[str, List[Polygon]]:
        polygon_type = (polygon_type or "all").lower()
        if polygon_type == "film":
            polys = list(self.films.values())
        elif polygon_type == "hole":
            polys = list(self.holes.values())
        elif polygon_type == "abstract":
            polys = list(self.abstract_regions.values())
        elif polygon_type == "all":
            polys = list(self.films.values()) + list(self.holes.values()) + list(self.abstract_regions.values())
        else:
            raise ValueError(f"Invalid polygon type ({polygon_type}).")
        out = {name: [] for name in self.layers}
        for p in polys:
            out[p.layer].append(p)
        return out

    def get_polygons(self, include_terminals: bool = True, polygon_type: Optional[str] = None) -> List[Polygon]:
        """All polygons of the device (reference ``get_polygons(include_terminals=True)``), or, as an extension,
        those of one kind (``polygon_type`` = film / hole / abstract / terminal; a string passed positionally is
        taken as the kind)."""
        if isinstance(include_terminals, str):
            include_terminals, polygon_type = True, include_terminals
        kinds = {"film": list(self.films.values()), "hole": list(self.holes.values()),
                 "abstract": list(self.abstract_regions.values()),
                 "terminal": [t for ts in self.terminals.values() for t in ts]}
        if polygon_type is not None:
            polygon_type = polygon_type.lower()
            if polygon_type not in kinds:
                raise ValueError(f"Invalid polygon type: {polygon_type!r}.")
            return kinds[polygon_type]
        out = kinds["film"] + kinds["hole"] + kinds["abstract"]
        return out + kinds["terminal"] if include_terminals else out

    def poly_points(self, films: bool = True, holes: bool = True, abstract: bool = True) -> np.ndarray:
        """Unique vertices of the selected polygons (reference device/device.py:221-240)."""
        polys = (list(self.films.values()) if films else []) + (list(self.holes.values()) if holes else []) \
            + (list(self.abstract_regions.values()) if abstract else [])
        pts = np.concatenate([p.points for p in polys]) if polys else np.zeros((0, 2))
        _, ix = np.unique(pts, axis=0, return_index=True)
        return pts[np.sort(ix)]

    def mesh_stats_dict(self) -> Dict[str, Dict[str, Union[int, float]]]:
        """Per-film mesh statistics (reference device/device.py:487-497)."""
        if not self.meshes:
            raise ValueError("The device does not have a mesh.")
        return {name: mesh.stats() for name, mesh in self.meshes.items()}

    def holes_by_film(self) -> Dict[str, List[Polygon]]:
        # memoised on the geometry (F x H point-in-polygon tests; asked for several times per solve)
        key = (tuple((f.name, f.layer, f.points.tobytes()) for f in self.films.values()),
               tuple((h.name, h.layer, h.points.tobytes()) for h in self.holes.values()))
        hit = self.__dict__.get("_holes_by_film_cache")
        if hit is not None and hit[0] == key:
            return {film: [self.holes[h] for h in names] for film, names in hit[1].items()}
        by_layer = self.polygons_by_layer("hole")
        out = {}
        for film in self.films.values():
            out[film.name] = [h for h in by_layer[film.layer] if film.contains_points(h.points).all()]
        self.__dict__["_holes_by_film_cache"] = (key, {film: [h.name for h in hs] for film, hs in out.items()})
        return out

    def copy(self, with_mesh: bool = True, copy_mesh: bool = False) -> "Device":
        d = Device(
            self.name,
            layers=[l.copy() for l in self.layers.values()],
            films=[f.copy() for f in self.films.values()],
            holes=[h.copy() for h in self.holes.values()],
            terminals={k: [t.copy() for t in v] for k, v in self.terminals.items()},
            abstract_regions=[r.copy() for r in self.abstract_regions.values()],
            length_units=self.length_units,
            solve_dtype=self.solve_dtype,  # the reference drops this (SURVEY.md Q5); we keep fp64
        )
        if with_mesh and self.meshes is not None:
            d.meshes = self.meshes
        return d

    # ------------------------------------------------------------ rigid transformations of the whole device
    def _warn_if_mesh_exist(self, method: str) -> None:
        if self.meshes:
            logger.warning(
                f"Calling device.{method} on a device whose mesh already exists returns a new device with no mesh. "
                f"Call new_device.make_mesh() to generate the mesh for the new device.")

    @staticmethod
    def _check_origin(origin) -> None:
        import numbers

        if not (isinstance(origin, tuple) and len(origin) == 2 and all(isinstance(v, numbers.Real) for v in origin)):
            raise TypeError("Origin must be a tuple of floats (x, y).")

    def scale(self, xfact: float = 1, yfact: float = 1, origin: Tuple[float, float] = (0, 0)) -> "Device":
        """reference device/device.py:266-292: a copy (without mesh) scaled about ``origin``; negative factors mirror."""
        self._check_origin(origin)
        self._warn_if_mesh_exist("scale()")
        device = self.copy(with_mesh=False)
        for polygon in device.get_polygons():
            polygon.scale(xfact=xfact, yfact=yfact, origin=origin, inplace=True)
        return device

    def rotate(self, degrees: float, origin: Tuple[float, float] = (0, 0)) -> "Device":
        """reference device/device.py:294-315: a copy (without mesh) rotated counter-clockwise about ``origin``."""
        self._check_origin(origin)
        self._warn_if_mesh_exist("rotate()")
        device = self.copy(with_mesh=False)
        for polygon in device.get_polygons():
            polygon.rotate(degrees, origin=origin, inplace=True)
        return device

    def mirror_layers(self, about_z: float = 0.0) -> "Device":
        """reference device/device.py:317-332: a copy (without mesh) with every layer mirrored about ``z = about_z``."""
        self._warn_if_mesh_exist("mirror_layers()")
        device = self.copy(with_mesh=False)
        for layer in device.layers.values():
            layer.z0 = about_z - layer.z0
        return device

    def translate(self, dx: float = 0, dy: float = 0, dz: float = 0, inplace: bool = False) -> "Device":
        """reference device/device.py:334-365.  Polygons (and meshes) move by ``(dx, dy)``, layers by ``dz``.  The
        reference shifts ``mesh.sites`` in place; here a device-resident mesh is rebuilt from the shifted sites
        (its operators are translation invariant, its coordinates are not)."""
        device = self if inplace else self.copy(with_mesh=True, copy_mesh=True)
        for polygon in device.get_polygons():
            polygon.translate(dx, dy, inplace=True)
        if device.meshes and (dx or dy):
            shift = np.array([[dx, dy]], dtype=float)
            device.set_meshes({name: (np.asarray(mesh.sites) + shift, np.asarray(mesh.elements))
                               for name, mesh in device.meshes.items()})
        if dz:
            for layer in device.layers.values():
                layer.z0 += dz
        return device

    def translation(self, dx: float, dy: float, dz: float = 0):
        """Context manager: the device is translated inside the block and moved back afterwards
        (reference device/device.py:367-381)."""
        from contextlib import contextmanager

        @contextmanager
        def moved():
            try:
                self.translate(dx, dy, dz=dz, inplace=True)
                yield
            finally:
                self.translate(-dx, -dy, dz=-dz, inplace=True)

        return moved()

    def to_hdf5(self, path_or_group, save_mesh: bool = True, compress: bool = True) -> None:
        """reference device/device.py:936-977"""
        from . import io as _io

        _io.device_to_hdf5(self, path_or_group, save_mesh=save_mesh, compress=compress)

    @staticmethod
    def from_hdf5(path_or_group) -> "Device":
        """reference device/device.py:979-1016"""
        from . import io as _io

        return _io.device_from_hdf5(path_or_group)

    # ---- meshes are inputs (mesh generation is out of scope, SURVEY.md section 2a) ----
    def set_meshes(self, meshes: Dict[str, Union[Mesh, Tuple[np.ndarray, np.ndarray]]]) -> None:
        """Attach one triangulation per film: ``{film: Mesh | (sites, elements)}``."""
        out = {}
        for name in self.films:
            if name not in meshes:
                raise ValueError(f"No mesh given for film {name!r}.")
            m = meshes[name]
            out[name] = m if isinstance(m, Mesh) else Mesh.from_triangulation(*m)
        self.meshes = out

    def make_mesh(self, buffer_factor: Union[float, Dict[str, float], None] = 0.05,
                  buffer: Union[float, Dict[str, float], None] = None, join_style: str = "mitre",
                  min_points: Union[int, Dict[str, int], None] = None,
                  max_edge_length: Union[float, Dict[str, float], None] = None, preserve_boundary: bool = False,
                  smooth: Union[int, Dict[str, int]] = 0, *, target_vertices: Union[int, Dict[str, int], None] = None,
                  seed: int = 0, **meshpy_kwargs) -> None:
        """Generates the triangular mesh of every film (reference device/device.py:383-471; same
        arguments).  Runs on the GPU (``meshgen.generate_mesh``: point cloud + Delaunay triangulation on
        the device, refined until ``min_points`` / ``max_edge_length`` hold).  As in the reference, the
        mesh of a film covers the film polygon plus a buffer region (``buffer`` in length units, or
        ``buffer_factor`` times the largest film dimension) unless the film has terminals or the buffer is
        0; the polygons of the holes / abstract regions inside the film become mesh vertices.  The buffered
        boundary is the convex hull of the film offset outward with mitre joins (the reference buffers the
        polygon itself with shapely, rounded joins -- the vacuum region differs, the film does not).
        ``smooth``: Laplacian-smoothing sweeps on the device (device/device.py:463-467 -> Mesh.smooth).

        ``target_vertices=...`` selects the host-side synthetic generator of the benchmark
        configurations instead (``synthetic.make_mesh``: scipy Delaunay, convex outlines only; runs
        without a GPU)."""
        if target_vertices is not None:
            return self._make_mesh_synthetic(target_vertices, buffer_factor if buffer_factor is not None else 0.0,
                                             seed, smooth if not isinstance(smooth, dict) else 0)
        from . import meshgen

        films = self.films

        def per_film(v):
            return v if isinstance(v, dict) else {name: v for name in films}

        buffer_factor, buffer, min_points = per_film(buffer_factor), per_film(buffer), per_film(min_points)
        max_edge_length, smooth = per_film(max_edge_length), per_film(smooth)
        holes_by_layer = self.polygons_by_layer("hole")
        abs_by_layer = self.polygons_by_layer("abstract")
        meshes = {}
        for k, (name, film) in enumerate(films.items()):
            film_terminals = self.terminals.get(name)
            film_ring = film.points[:-1]
            coords, embedded = [film_ring], []
            for poly in holes_by_layer.get(film.layer, []) + abs_by_layer.get(film.layer, []):
                if film.contains_points(poly.points).all():
                    coords.append(poly.points[:-1])
                    embedded.append(poly.points[:-1])
            if film_terminals or buffer.get(name) == 0 or (buffer_factor.get(name) is None and buffer.get(name) is None) \
                    or (buffer.get(name) is None and buffer_factor.get(name) == 0):
                boundary = film_ring
            else:
                size = buffer[name] if buffer.get(name) is not None else buffer_factor[name] * max(film.extents)
                hull = meshgen.convex_hull_ring(film_ring)
                boundary = meshgen.offset_convex_ring(hull, float(size))
                # (reference: Polygon(points=buffered).resample(len(film.points)))
                per = np.linalg.norm(np.roll(boundary, -1, axis=0) - boundary, axis=1).sum()
                boundary = meshgen._resample_ring(boundary, per / max(len(film_ring), 8))
                coords.append(boundary)
                embedded.append(film_ring)
            points, triangles = meshgen.generate_mesh(
                meshgen.ensure_unique(np.concatenate(coords, axis=0)), min_points=min_points.get(name),
                max_edge_length=max_edge_length.get(name), boundary=boundary, convex_hull=False,
                preserve_boundary=preserve_boundary or bool(film_terminals), seed=seed + k, embedded=embedded,
                **meshpy_kwargs)
            mesh = Mesh.from_triangulation(points, triangles, build_operators=not smooth.get(name))
            meshes[name] = mesh.smooth(smooth[name]) if smooth.get(name) else mesh
        self.meshes = meshes

    def _make_mesh_synthetic(self, target_vertices: Union[int, Dict[str, int]], buffer_factor: float, seed: int,
                             smooth: int) -> None:
        """Host-side generator of the benchmark / parity configurations: meshes the (scaled) convex outline
        of each film with ``synthetic.make_mesh`` (jittered lattice + scipy Delaunay)."""
        from .synthetic import make_mesh

        holes_by_film = self.holes_by_film()
        meshes = {}
        for k, (name, film) in enumerate(self.films.items()):
            nv = target_vertices[name] if isinstance(target_vertices, dict) else target_vertices
            pts = film.points[:-1]
            embedded = [h.points[:-1] for h in holes_by_film[name]]
            if buffer_factor:
                c = pts.mean(axis=0)
                outline = c + (pts - c) * (1.0 + 2 * buffer_factor)
                embedded = [pts] + embedded
            else:
                outline = pts
            meshes[name] = make_mesh(outline, target_vertices=nv, embedded=embedded, seed=seed + k)
        self.set_meshes(meshes)
        if smooth:
            self.meshes = {name: mesh.smooth(smooth) for name, mesh in self.meshes.items()}

    def boundary_vertices(self, film: str) -> np.ndarray:
        """Boundary vertex indices of a film's mesh ordered counter-clockwise (reference
        device/device.py:473-485 -> device/utils.py:205-227)."""
        from .mesh import boundary_vertices_ccw

        if not self.meshes:
            raise ValueError("The device does not have a mesh.")
        return boundary_vertices_ccw(self.meshes[film].elements)

    def mutual_inductance_matrix(self, hole_polygon_mapping: Optional[Dict[str, np.ndarray]] = None,
                                 units: str = "pH", all_iterations: bool = False, progress_bar: bool = False,
                                 comm=None, **solve_kwargs):
        """reference device/device.py:538-648.  Without ``hole_polygon_mapping`` the polygons come from
        ``fluxoid.make_fluxoid_polygons`` as in the reference (device.py:592-595; the holes are grown by half
        the distance to the nearest other polygon -- by scaling about the centroid here, by a shapely buffer
        there: identical for circular holes, pass explicit polygons for parity runs).  ``progress_bar`` is accepted
        for compatibility (there is no per-hole loop to show progress of).  The reference solves once
        per driven hole against one factorization; here all columns are one batched solve
        (``solve_batch``).  As in the reference, ``iterations`` is forwarded to the solver only if
        given explicitly (SURVEY.md Q8).  Films with transport terminals are solved as the reference solves
        them, with zero terminal currents: their boundary stays out of the linear system and their self
        field is the Biot-Savart sum over their triangles."""
        from .solver import factorize_model, solve_batch

        from . import _lib

        if hole_polygon_mapping is None:
            from .fluxoid import make_fluxoid_polygons

            hole_polygon_mapping = make_fluxoid_polygons(self)
        holes = self.holes
        hole_names = list(holes)
        with _lib.nvtx_range("scb.mim.validate"):
            # (the containment test of a given (polygon, hole) pair is remembered: the matrix is usually
            #  evaluated many times for one device -- parameter sweeps, the iterates of a fluxoid solve)
            checked = self.__dict__.setdefault("_mim_checked", {})
            for hole_name, polygon in hole_polygon_mapping.items():
                if hole_name not in holes:
                    raise ValueError(f"Hole '{hole_name}' does not exist in the device.")
                key = (hole_name, np.asarray(polygon, dtype=float).tobytes(), holes[hole_name].points.tobytes())
                ok = checked.get(key)
                if ok is None:
                    if len(checked) > 256:
                        checked.clear()
                    ok = checked[key] = bool(points_in_polygon(polygon, holes[hole_name].points).all())
                if not ok:
                    raise ValueError(f"Hole '{hole_name}' is not completely contained within the given polygon.")
        n_holes = len(hole_polygon_mapping)
        iterations = solve_kwargs.get("iterations", 1)
        I_circ_A = _u.to_quantity("1 mA", "A").to("A").magnitude
        if all_iterations:
            n_iter = 1 if len(self.layers) == 1 else iterations + 1
            sl = slice(None)
        else:
            n_iter = 1
            sl = slice(-1, None)
        M = np.zeros((n_iter, n_holes, n_holes))
        films_by_hole = {h.name: film for film, hs in self.holes_by_film().items() for h in hs}
        with _lib.nvtx_range("scb.mim.factorize_model"):
            model = factorize_model(device=self, current_units="mA", comm=comm, _defer_checks=True)
        # Multi-rank: every rank keeps only its own films' solutions (no replication of the results),
        # evaluates the fluxoid rows of the holes in those films, and the small matrix is summed over
        # the ranks -- M[i, j] only needs film(i)'s solution for the driven hole j.
        sharded = comm is not None and comm.world > 1
        with _lib.nvtx_range("scb.mim.solve_batch"):
            batch = solve_batch(
                model=model, applied_fields=[solve_kwargs.get("applied_field")] * len(hole_names),
                circulating_currents=[{name: 1.0} for name in hole_names],
                field_units=solve_kwargs.get("field_units", "mT"), iterations=solve_kwargs.get("iterations", 0),
                check_inversion=solve_kwargs.get("check_inversion", False), last_only=not all_iterations,
                gather=not sharded)
        to_units = _u.conversion_factor("H", units)
        with _lib.nvtx_range("scb.mim.fluxoids"):
            for j, hole_name in enumerate(hole_names):
                for nn, solution in enumerate(batch[j][sl]):
                    for i, name in enumerate(hole_names):
                        if films_by_hole[name] not in solution.film_solutions:
                            continue  # another rank's film
                        fluxoid = solution.polygon_fluxoid(hole_polygon_mapping[name], film=films_by_hole[name],
                                                           units="Phi_0", with_units=False)
                        M[nn, i, j] = sum(fluxoid) * _u.PHI_0 / I_circ_A * to_units
        if sharded:
            import torch

            dev = torch.device(f"cuda:{torch.cuda.current_device()}") if torch.cuda.is_available() \
                else torch.device("cpu")
            parts = torch.zeros((comm.world,) + M.shape, dtype=torch.float64, device=dev)
            comm.all_gather_into(parts.view(comm.world, -1), torch.as_tensor(M).to(dev).reshape(1, -1))
            M = parts.sum(dim=0).cpu().numpy()  # every entry is non-zero on exactly one rank
        result = [m for m in M]
        if not all_iterations:
            result = result[0]
        return result
