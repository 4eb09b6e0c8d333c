"""solve / factorize_model / FactorizedModel (reference solver/solve.py) on the B200.

Same signatures, return types and error behaviour as the reference; the arithmetic runs in
libsc_b200 (include/scb.h).  All per-film state stays on the device across the film-to-film
iterations (reference solve.py:491-547); only the O(n) result vectors of each ``Solution`` are
copied back to the host.
"""
from __future__ import annotations

import copy
import itertools
import logging
import numbers
import os
from dataclasses import dataclass, field
from typing import Callable, Dict, List, Optional, Sequence, Tuple, Union

import numpy as np

from .. import _lib
from .. import units as _u
from ..device import Device
from ..mesh import Mesh
from ..solution import FilmSolution, Solution, Vortex
from ..sources import ConstantField
from .solve_film import (  # noqa: F401  (TerminalSystems, solve_film: names the reference module exposes)
    LinearSystem, TerminalSystems, factorize_linear_systems, hole_boundary_state, make_vortex_state, solve_film,
    solve_film_device, terminal_transport_state)
from .utils import (FilmInfo, currents_to_floats, field_conversion_factor, get_holes_and_vortices_by_film,
                    make_film_info)

logger = logging.getLogger("solve")


def _torch():
    import torch

    return torch


def biot_savart_film_to_film(*, film1_sites, film1_z0: float, film1_areas, film1_J, film2_sites,
                             film2_z0: float) -> np.ndarray:
    """reference solver/solve.py:28-73 (host arrays in/out; the pair sum runs on the device)."""
    torch = _torch()
    _lib.lib()
    dev = torch.device(f"cuda:{torch.cuda.current_device()}")
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).to(dev)
    out = film_to_film_device(t(film1_sites), float(film1_z0), t(film1_areas), t(film1_J), t(film2_sites),
                              float(film2_z0))
    return out.cpu().numpy()


def film_to_film_device(src_sites, src_z0: float, src_areas, src_J, tgt_sites, tgt_z0: float):
    """Field of the source film's sheet current at the target sites, solver units.  ``src_J`` is
    ``(n, 2)`` -> ``(m,)`` or a batch ``(B, n, 2)`` -> ``(B, m)``."""
    torch = _torch()
    L = _lib.lib()
    m, n = int(tgt_sites.shape[0]), int(src_sites.shape[0])
    nsets = int(src_J.shape[0]) if src_J.dim() == 3 else 1
    with torch.cuda.device(tgt_sites.device):
        J = src_J.contiguous()
        out = torch.empty((nsets, m) if src_J.dim() == 3 else (m,), dtype=torch.float64, device=tgt_sites.device)
        _lib.check(L.scb_biot_savart(0, m, _lib.ptr(tgt_sites), n, _lib.ptr(src_sites), _lib.ptr(src_areas),
                                     _lib.ptr(J), float(tgt_z0) - float(src_z0),
                                     1.0 / (4.0 * np.pi), nsets, _lib.ptr(out), _lib.stream_ptr()))
    return out


@dataclass
class FactorizedModel:
    """reference solver/solve.py:76-220"""

    device: Device
    film_info: Dict[str, FilmInfo]
    film_systems: Dict[str, LinearSystem]
    hole_systems: Dict[str, Dict[str, LinearSystem]]
    terminal_systems: Dict[str, object]
    terminal_currents: Dict[str, Dict[str, float]]
    circulating_currents: Dict[str, float]
    vortices: Union[Sequence[Vortex], Dict[str, Sequence[Vortex]]]
    current_units: str
    comm: object = None  # parallel.Comm: film -> owner rank (None = single process)
    # read-backs of the factorization flags that have not happened yet (factorize_model(_defer_checks=True))
    _deferred_checks: list = field(default_factory=list, repr=False, compare=False)

    def finish_checks(self) -> None:
        """Reads back the singularity flags of factorizations that were enqueued without waiting for them
        (raises ``LinAlgError`` exactly as ``factorize_model`` would have); a no-op otherwise."""
        while self._deferred_checks:
            self._deferred_checks.pop(0)()

    def set_circulating_currents(self, circulating_currents: Dict[str, float]) -> None:
        diff = set(circulating_currents) - set(self.device.holes)
        if diff:
            raise KeyError(f"circulating_currents contains keys not in self.device.holes: {list(diff)!r}")
        self.circulating_currents = circulating_currents.copy()
        holes_by_film = self.device.holes_by_film()
        for film_name, film_info in self.film_info.items():
            holes = [hole.name for hole in holes_by_film[film_name]]
            film_info.circulating_currents = {}
            for hole, current in self.circulating_currents.items():
                if hole in holes:
                    film_info.circulating_currents[hole] = current

    def set_vortices(self, vortices: Sequence[Vortex]) -> None:
        for film in self.film_info.values():
            film.vortices = []
        for vortex in vortices:
            self.film_info[vortex.film].vortices.append(vortex)
        self.vortices = {}
        for name, film in self.film_info.items():
            film.vortices = tuple(film.vortices)
            self.vortices[name] = film.vortices

    def copy(self) -> "FactorizedModel":
        return copy.copy(self)

    def to_hdf5(self, h5group) -> None:
        """reference solver/solve.py:102-132 (same groups, datasets and attributes; ``superscreen_b200.io``)"""
        from .. import io as _io

        self.finish_checks()
        _io.model_to_hdf5(self, h5group)

    @staticmethod
    def from_hdf5(h5group, comm=None) -> "FactorizedModel":
        """reference solver/solve.py:134-180; operators and factors are rebuilt on the GPU from the stored
        triangulations."""
        from .. import io as _io

        return _io.model_from_hdf5(h5group, comm=comm)


def factorize_model(*, device: Device, current_units: str, terminal_currents=None, circulating_currents=None,
                    vortices: Optional[Sequence[Vortex]] = None, comm=None,
                    _defer_checks: bool = False) -> FactorizedModel:
    """reference solver/solve.py:223-287.  With a multi-rank ``comm`` (``parallel.DistComm``) each
    rank assembles and factorizes only the films it owns (one film factorization per GPU).
    ``_defer_checks`` (internal: callers that solve right away) returns while the GPU is still factoring;
    the zero-pivot flags are then read by ``FactorizedModel.finish_checks()`` / at the end of the solve."""
    ureg = device.ureg
    circulating_currents = currents_to_floats(circulating_currents or {}, ureg, current_units)
    terminal_currents = {
        film_name: currents_to_floats(currents, ureg, current_units)
        for film_name, currents in (terminal_currents or {}).items()
    }
    for film_name, currents in terminal_currents.items():
        if sum(currents.values()):
            raise ValueError(f"Terminal currents in film {film_name!r} are not conserved.")
    vortices = vortices or []
    if not device.meshes:
        raise ValueError("The device does not have a mesh. Call device.make_mesh() to generate it.")
    with _lib.nvtx_range("scb.make_film_info"):
        film_info = make_film_info(device=device, vortices=vortices, circulating_currents=circulating_currents,
                                   terminal_currents=terminal_currents)
    from ..parallel import Comm, film_owners

    comm = comm or Comm()
    owners = film_owners(list(device.films), comm)
    owned = {f for f, r in owners.items() if r == comm.rank}
    deferred = [] if (_defer_checks and os.environ.get("SCB_DEFER_CHECKS", "1") != "0") else None
    with _lib.nvtx_range("scb.factorize_linear_systems"):
        film_systems, hole_systems, terminal_systems = factorize_linear_systems(device, film_info, owned=owned,
                                                                                deferred=deferred)
    return FactorizedModel(device, film_info, film_systems, hole_systems, terminal_systems, terminal_currents,
                           circulating_currents, vortices, current_units, comm, deferred or [])


_UPLOAD_STREAMS: dict = {}


def _upload(host_array, dev):
    """Host array -> device tensor through a dedicated copy stream.  A pageable host-to-device copy is
    ordered behind everything already queued on its stream and blocks the host until it has run; issued on
    the compute stream right after ``factorize_model(_defer_checks=True)`` it would make the host wait for
    the whole factorization.  On the (otherwise idle) copy stream it completes at once; the compute stream
    then waits for it with an event."""
    import torch

    if dev.type != "cuda" or os.environ.get("SCB_UPLOAD_STREAM", "1") == "0":
        return torch.as_tensor(host_array).to(dev)
    st = _UPLOAD_STREAMS.get(dev)
    if st is None:
        st = _UPLOAD_STREAMS[dev] = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(st):
        t = torch.as_tensor(host_array).to(dev)
    cur = torch.cuda.current_stream(dev)
    cur.wait_stream(st)
    t.record_stream(cur)
    return t


def _to_host(t) -> np.ndarray:
    """Device tensor -> host numpy array.  Large arrays are copied into a pinned tensor of torch's
    caching host allocator (a pageable cudaMemcpy runs at a fraction of the PCIe/C2C rate) and
    handed out as a view of it: no second host copy; the block returns to the cache when the last
    view dies."""
    import torch

    t = t.contiguous()
    if t.numel() < (1 << 15):
        return t.cpu().numpy()
    stage = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    stage.copy_(t, non_blocking=True)
    torch.cuda.current_stream(t.device).synchronize()
    return stage.numpy()


def _solutions_from_host(device, host, film_names, host_fields, field_conversion, kwargs_list, batched,
                         device_builders=None):
    """HostResults (parallel.ResultPacker) -> [[Solution per batch entry] per stored iterate]
    (reference solve_film.py:566-573: fields are handed out in ``field_units``).  The arrays of the
    FilmSolutions are views of the one downloaded buffer; the applied field never left the host.
    ``device_builders`` (batched only): per entry ``None`` (the shared copy of ``device``) or the builder of
    its translated device."""
    applied = {name: host_fields[name] / field_conversion for name in film_names}
    shared = device.copy(with_mesh=True, copy_mesh=False)  # one copy shared by the solutions of this call
    out = []
    for it in host.iterates:
        row = []
        for b, kwargs in enumerate(kwargs_list):
            film_solutions = {}
            for name in film_names:
                g, J, self_field, other = host.film(it, b, name)
                film_solutions[name] = FilmSolution(
                    stream=g, current_density=J, applied_field=applied[name][b] if batched else applied[name],
                    self_field=self_field, field_from_other_films=other)
            row.append(Solution(device=shared, film_solutions=film_solutions, _device_is_copy=True,
                                _device_builder=None if device_builders is None else device_builders[b], **kwargs))
        out.append(row)
    return out


def _evaluate_applied_field(applied_field, device, film_info, meshes, field_conversion, films=None, moves=None):
    """reference solver/solve.py:422-436 -> {film: host float64 (n,) in solver units}.  ``moves``
    ({layer: (dx, dy, dz)}): the field at the vertices of those layers' films moved as ``Device.translate``
    moves them (``sites + (dx, dy)``, ``z0 + dz``)."""
    out = {}
    for film, mesh in meshes.items():
        if films is not None and film not in films:
            continue
        layer = device.layers[film_info[film].layer]
        sites, z0 = mesh.sites, layer.z0
        if moves and film_info[film].layer in moves:
            dx, dy, dz = moves[film_info[film].layer]
            sites = np.asarray(sites) + np.array([[dx, dy]], dtype=float) if (dx or dy) else sites
            z0 = z0 + dz
        z0 = z0 * np.ones(len(sites))
        Hz_applied = np.squeeze(applied_field(sites[:, 0], sites[:, 1], z0) * field_conversion)
        Hz_applied = np.asarray(Hz_applied, dtype=np.float64)
        if Hz_applied.ndim != 1:
            raise ValueError(
                "Expected applied_field to return a 1D vector,"
                f" got a {Hz_applied.shape[1]}D vector."
            )
        out[film] = np.ascontiguousarray(Hz_applied)
    return out


def _packed_sources(model: "FactorizedModel", layout, z0s, dev):
    """Static part of the film-to-film coupling: vertices (x, y, z0), vertex areas and the film index
    (position in ``layout.films``, int32) of ALL films in the packed layout of ``parallel.FilmLayout``
    (padding rows: far away, zero area, film -1).  Built once per model and device."""
    torch = _torch()
    cache = model.__dict__.setdefault("_packed_cache", {})
    key = (str(dev), tuple(layout.films), layout.world)
    hit = cache.get(key)
    if hit is None:
        src = torch.full((layout.total, 3), 1e30, dtype=torch.float64, device=dev)
        area = torch.zeros(layout.total, dtype=torch.float64, device=dev)
        film = torch.full((layout.total,), -1, dtype=torch.int32, device=dev)
        for k, name in enumerate(layout.films):
            d = model.device.meshes[name]._data
            lo, hi = layout.rows(name)
            src[lo:hi, :2] = d.sites.to(dev)
            src[lo:hi, 2] = z0s[name]
            area[lo:hi] = d.t["vertex_areas"].to(dev)
            film[lo:hi] = k
        hit = cache[key] = (src, area, film)
    return hit


def _run(model: "FactorizedModel", applied_fields, circ_by_film, vortex_flux, iterations, check_inversion,
         field_conversion: float, batch: Optional[int] = None, last_only: bool = False, gather: bool = True,
         terminal_currents: Optional[List[Dict[str, Dict[str, float]]]] = None,
         vortices: Optional[List[Dict[str, List[Vortex]]]] = None, shifts: Optional[np.ndarray] = None):
    """Runs the solve + film-to-film iterations on the device for single or batched right-hand
    sides.  ``terminal_currents`` (batched only): one ``{film: {terminal: current}}`` dict per entry
    (default: the model's for every entry).  ``vortices`` (batched only): one ``{film: [Vortex]}`` dict per
    entry (default: the model's vortices for every entry).  ``shifts`` (batched only): ``(B, films, 3)``, the
    rigid shift of every film per entry, films in device order; the film-to-film coupling then runs on the moved
    geometry (``scb_film_coupling_translated``).  Everything stays on the device until the
    end: every owned film's result of every stored iterate is packed into one buffer (``parallel.ResultPacker``), replicated over the ranks by one
    all-gather if ``gather`` and downloaded once.  Returns ``parallel.HostResults``."""
    torch = _torch()
    import contextlib

    from ..parallel import Comm, FilmLayout, ResultPacker, film_owners, run_film_iterations

    L = _lib.lib()
    device = model.device
    comm = model.comm or Comm()
    film_names = list(device.films)
    owners = film_owners(film_names, comm)
    meshes = device.meshes
    film_info = model.film_info
    z0s = {name: float(device.layers[film_info[name].layer].z0) for name in film_names}
    dev = next((t.device for t in applied_fields.values()), torch.device(f"cuda:{torch.cuda.current_device()}"))
    layout = FilmLayout(film_names, {f: len(meshes[f].sites) for f in film_names}, owners, comm.world)
    multi = len(film_names) >= 2 and iterations >= 1
    n_solutions = iterations + 1 if multi else 1
    iterates = [n_solutions - 1] if last_only else list(range(n_solutions))

    hole_states = {}  # hole boundary values + their effective field: constant over the iterations
    transport_states = {}  # terminal films: transport stream + its boundary field, constant likewise
    vortex_states = {}     # per film: the located vortices of every column, constant likewise
    n_solves = {}     # per film: number of the iterate being solved (the driver solves every film once per iterate)

    def solve_fn(name, other):
        with _lib.nvtx_range(f"scb.solve_film[{name}]"):
            return _solve_fn(name, other)

    def _solve_fn(name, other):
        it = n_solves.get(name, 0)
        n_solves[name] = it + 1
        circ = None if circ_by_film is None else circ_by_film[name]
        if name not in hole_states:
            info = film_info[name]
            hole_states[name] = hole_boundary_state(
                info, model.hole_systems[name], info.circulating_currents if circ is None else circ,
                applied_fields[name]) if model.hole_systems[name] else (None, None)
        terminal_systems = model.terminal_systems.get(name)
        if terminal_systems is not None and name not in transport_states:
            info = film_info[name]
            if terminal_currents is not None:
                currents = [tc.get(name, {}) for tc in terminal_currents]
            else:
                currents = info.terminal_currents or {}
                if batch is not None:
                    currents = [currents] * batch
            transport_states[name] = terminal_transport_state(device, info, terminal_systems, currents)
        if name not in vortex_states:
            if vortices is not None:
                columns = [v.get(name, ()) for v in vortices]
            else:
                columns = [film_info[name].vortices] * (1 if batch is None else batch)
            vortex_states[name] = make_vortex_state(film_info[name], model.film_systems[name], columns)
        return solve_film_device(
            film_info=film_info[name], film_system=model.film_systems[name],
            hole_systems=model.hole_systems[name], applied_field=applied_fields[name], vortex_flux=vortex_flux,
            field_from_other_films=other, check_inversion=check_inversion, circulating_currents=circ,
            terminal_systems=terminal_systems, device=device, hole_state=hole_states[name],
            transport_state=transport_states.get(name), vortex_state=vortex_states[name],
            want_self_field=it in iterates)  # (the self field of an iterate that is not stored is never used)

    inv4pi = 1.0 / (4.0 * np.pi)
    shift_table = None
    if shifts is not None and multi:
        shift_table = _upload(np.ascontiguousarray(shifts, dtype=np.float64), dev)

    def coupling_fn(dst, J_all):
        with _lib.nvtx_range(f"scb.film_coupling[{dst}]"):
            return _coupling_fn(dst, J_all)

    def _coupling_fn(dst, J_all):
        # sum over every other film of biot_savart_film_to_film (reference solve.py:495-515): one launch
        src, area, src_film = _packed_sources(model, layout, z0s, dev)
        d = meshes[dst]._data
        lo, hi = layout.rows(dst)
        with torch.cuda.device(dev):
            out = torch.empty((d.n, batch) if batch is not None else (d.n,), dtype=torch.float64, device=dev)
            if shift_table is None:
                _lib.check(L.scb_film_coupling(d.n, _lib.ptr(d.sites), z0s[dst], layout.total, _lib.ptr(src),
                                               _lib.ptr(area), _lib.ptr(J_all), lo, hi, inv4pi,
                                               batch if batch is not None else 1, _lib.ptr(out), _lib.stream_ptr()))
            else:
                _lib.check(L.scb_film_coupling_translated(
                    d.n, _lib.ptr(d.sites), z0s[dst], layout.total, _lib.ptr(src), _lib.ptr(area), _lib.ptr(J_all),
                    lo, hi, inv4pi, batch, layout.films.index(dst), _lib.ptr(src_film), len(layout.films),
                    _lib.ptr(shift_table), _lib.ptr(out), _lib.stream_ptr()))
        return out

    # the films of one Jacobi step are independent and each is latency-bound (getrs sweeps, small
    # N-body launches): one side stream per owned film, joined after every step
    mine = layout.by_rank[comm.rank]
    side = {}
    n_side = int(os.environ.get("SCB_FILM_STREAMS", "8"))
    if len(mine) > 1 and n_side > 0:
        pool = _lib.film_streams(dev, min(len(mine), n_side))
        side = {f: pool[k % len(pool)] for k, f in enumerate(mine)}

    @contextlib.contextmanager
    def film_scope(name):
        st = side.get(name)
        if st is None:
            yield
            return
        st.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(st):
            yield

    def join():
        main = torch.cuda.current_stream(dev)
        for st in set(side.values()):
            main.wait_stream(st)

    with torch.cuda.device(dev):
        if multi:
            _packed_sources(model, layout, z0s, dev)  # (on the main stream, before the side streams start)
        packer = ResultPacker(layout, comm, iterates, batch, torch.empty(0, dtype=torch.float64, device=dev))
        j_like = torch.empty((0, batch, 2) if batch is not None else (0, 2), dtype=torch.float64, device=dev)
        with _lib.nvtx_range("scb.film_iterations"):
            run_film_iterations(layout, comm, solve_fn, coupling_fn, iterations, film_scope=film_scope, join=join,
                                on_result=packer.put, j_like=j_like)
        packer.scale_fields(1.0 / field_conversion)
        model.finish_checks()  # (factorizations enqueued without waiting: their zero-pivot flags, now)
        with _lib.nvtx_range("scb.results_to_host"):
            return packer.to_host(gather, to_numpy=_to_host)


def _check_model_args(device, model, terminal_currents, circulating_currents, vortices, current_units):
    """Argument validation shared by solve / solve_batch (reference solver/solve.py:357-389)."""
    if model is None:
        if device is None:
            raise ValueError("Either a model or a device must be provided.")
        logger.info("Factorizing model.")
        model = factorize_model(device=device, current_units=current_units, terminal_currents=terminal_currents,
                                circulating_currents=circulating_currents, vortices=vortices, _defer_checks=True)
    else:
        if (device is not None or terminal_currents is not None or circulating_currents is not None
                or vortices is not None):
            raise ValueError(
                "If model argument is provided, device, terminal_currents,"
                " circulating_currents, and vortices must be None."
            )
    if not isinstance(model, FactorizedModel):
        raise TypeError(f"model must be an instance of FactorizedModel (got {type(model)}).")
    if not model.device.meshes:
        raise ValueError("The device does not have a mesh. Call device.make_mesh() to generate it.")
    return model


def solve(device: Optional[Device] = None, *, model: Optional[FactorizedModel] = None,
          applied_field: Optional[Callable] = None, terminal_currents=None, circulating_currents=None,
          vortices: Optional[Sequence[Vortex]] = None, field_units: str = "mT", current_units: str = "uA",
          check_inversion: bool = False, iterations: int = 0, return_solutions: bool = True,
          save_path: Optional[os.PathLike] = None, log_level: Optional[int] = None, progress_bar: bool = True,
          _solver: str = "superscreen_b200.solve") -> List[Solution]:
    """reference solver/solve.py:290-549"""
    torch = _torch()
    if log_level is not None:
        logging.basicConfig(level=log_level)
    model = _check_model_args(device, model, terminal_currents, circulating_currents, vortices, current_units)
    device = model.device
    current_units = model.current_units
    length_units = device.length_units
    applied_field = applied_field or ConstantField(0)
    field_conversion = field_conversion_factor(field_units, current_units, length_units=length_units).magnitude
    host_fields = _evaluate_applied_field(applied_field, device, model.film_info, device.meshes, field_conversion)
    owned = _owned_films(model)
    applied_fields = {f: _upload(h, device.meshes[f]._data.device) for f, h in host_fields.items() if f in owned}
    # Phi_0 / mu_0 in [current_units * length_units]  (reference solve.py:441)
    vortex_flux = _u.PHI_0 / _u.MU_0 * _u.conversion_factor("A * m", f"({current_units}) * ({length_units})")
    solution_kwargs = dict(applied_field_func=applied_field, field_units=field_units, current_units=current_units,
                           circulating_currents=model.circulating_currents,
                           terminal_currents=model.terminal_currents, vortices=model.vortices, solver=_solver)
    host = _run(model, applied_fields, None, vortex_flux, iterations, check_inversion, field_conversion)
    if not return_solutions:
        return None
    film_names = list(device.films)
    per_iter = _solutions_from_host(device, host, film_names, host_fields, field_conversion, [solution_kwargs],
                                    batched=False)
    solutions = [row[0] for row in per_iter]
    if save_path is not None:
        # reference solve.py:475-480,541-543: the device once in the root group, solution i in group str(i)
        # with a soft link to it (an HDF5 file path needs h5py; an open group works without)
        from .. import io as _io

        _io.save_solutions(solutions, save_path)
    return solutions


def _batch_terminal_currents(model: FactorizedModel, terminal_currents, B: int):
    """Validates and converts the per-entry terminal currents of ``solve_batch`` exactly as
    ``factorize_model`` + ``solve`` would (before any device work): floats or unit strings in
    ``model.current_units``, known films and terminals, conserved per film, and -- as the stream
    function needs it -- every terminal of a film that carries a current."""
    device = model.device
    if len(terminal_currents) != B:
        raise ValueError("applied_fields and terminal_currents must have the same length.")
    out = []
    for entry in terminal_currents:
        entry = entry or {}
        converted = {}
        for film_name, currents in entry.items():
            if film_name not in device.terminals:
                raise KeyError(f"terminal_currents contains a film without terminals: {film_name!r}")
            names = [t.name for t in device.terminals[film_name]]
            diff = set(currents) - set(names)
            if diff:
                raise KeyError(f"terminal_currents[{film_name!r}] contains unknown terminals: {sorted(diff)!r}")
            currents = currents_to_floats(currents, device.ureg, model.current_units)
            if sum(currents.values()):
                raise ValueError(f"Terminal currents in film {film_name!r} are not conserved.")
            if any(currents.values()):
                missing = [name for name in names if name not in currents]
                if missing:
                    raise KeyError(missing[0])
            converted[film_name] = currents
        out.append(converted)
    return out


def _batch_vortices(device: Device, vortices, B: int) -> List[Dict[str, List[Vortex]]]:
    """Validates the per-entry vortices of ``solve_batch`` with the reference's rules
    (``get_holes_and_vortices_by_film``: every item a ``Vortex``, in a film of the device, inside that
    film and not inside one of its holes) before any device work, naming the offending entry.  Returns
    one ``{film: [Vortex]}`` dict per entry (every film of the device a key)."""
    if len(vortices) != B:
        raise ValueError(f"applied_fields and vortices must have the same length (got {B} and {len(vortices)}).")
    out = []
    for b, entry in enumerate(vortices):
        if isinstance(entry, Vortex):
            raise TypeError(f"vortices[{b}]: expected a sequence of Vortex, but got a single {entry!r}.")
        entry = [] if entry is None else list(entry)
        for vortex in entry:
            if isinstance(vortex, Vortex) and vortex.film not in device.films:
                raise KeyError(f"vortices[{b}]: {vortex!r} is in a film the device does not have: {vortex.film!r}")
        try:
            _, by_film = get_holes_and_vortices_by_film(device, entry)
        except (TypeError, ValueError) as exc:
            raise type(exc)(f"vortices[{b}]: {exc}") from exc
        out.append(by_film)
    return out


def _batch_translations(device: Device, translations, B: int,
                        vortices: Sequence[Sequence[Vortex]]) -> Optional[List[Dict[str, Tuple[float, float, float]]]]:
    """Validates the per-entry layer translations of ``solve_batch`` before any device work, naming the
    offending entry.  ``vortices``: the vortices of every entry.  Returns one ``{layer: (dx, dy, dz)}`` dict per
    entry holding the layers it moves (a zero shift moves nothing), or ``None`` when no entry moves anything."""
    if len(translations) != B:
        raise ValueError(f"applied_fields and translations must have the same length "
                         f"(got {B} and {len(translations)}).")
    out = []
    for b, entry in enumerate(translations):
        entry = {} if entry is None else entry
        if not isinstance(entry, dict):
            raise TypeError(f"translations[{b}]: expected None or a dict {{layer: (dx, dy) | (dx, dy, dz)}}, "
                            f"but got {entry!r}.")
        moves = {}
        for layer, value in entry.items():
            if layer not in device.layers:
                raise KeyError(f"translations[{b}]: the device has no layer {layer!r}.")
            shift = tuple(value) if isinstance(value, (tuple, list, np.ndarray)) else ()
            if not (len(shift) in (2, 3) and all(isinstance(v, numbers.Real) and np.isfinite(v) for v in shift)):
                raise ValueError(f"translations[{b}]: the shift of layer {layer!r} must be 2 or 3 finite reals "
                                 f"(dx, dy[, dz]), but got {value!r}.")
            shift = tuple(float(v) for v in shift) + (0.0,) * (3 - len(shift))
            if any(shift):
                moves[layer] = shift
        for layer in moves:
            if callable(device.layers[layer].Lambda):
                raise ValueError(f"translations[{b}]: layer {layer!r} has a position-dependent Lambda, so moving it "
                                 "would change its factorization.")
        for vortex in vortices[b]:
            layer = device.films[vortex.film].layer
            if layer in moves:
                raise ValueError(f"translations[{b}]: {vortex!r} is in layer {layer!r}, which the entry moves; "
                                 "vortices in moved layers are not supported.")
        out.append(moves)
    return out if any(out) else None


def _translated_device(device: Device, moves: Dict[str, Tuple[float, float, float]]) -> Device:
    """A copy of ``device`` with the layers in ``moves`` (``{layer: (dx, dy, dz)}``) moved as
    ``Device.translate`` moves a whole device: every polygon of those layers (films, holes, terminals,
    abstract regions) by ``(dx, dy)``, the meshes of their films rebuilt from ``sites + (dx, dy)``, ``z0`` by
    ``dz``.  The meshes of the other films are shared with ``device``."""
    out = device.copy(with_mesh=False)
    for polygon in out.get_polygons():
        if polygon.layer in moves:
            polygon.translate(*moves[polygon.layer][:2], inplace=True)
    meshes = dict(device.meshes)
    for name, film in device.films.items():
        dx, dy, _ = moves.get(film.layer, (0.0, 0.0, 0.0))
        if dx or dy:
            mesh = device.meshes[name]
            meshes[name] = Mesh.from_triangulation(np.asarray(mesh.sites) + np.array([[dx, dy]], dtype=float),
                                                   np.asarray(mesh.elements))
    out.meshes = meshes
    for layer, (_, _, dz) in moves.items():
        if dz:
            out.layers[layer].z0 += dz
    return out


def _device_builders(device: Device, moves: List[Dict[str, Tuple[float, float, float]]]):
    """Per entry ``None`` (nothing moves) or a function that builds the entry's translated device on first
    call; entries with the same translation share the function and so the device."""
    by_key = {}
    out = []
    for entry in moves:
        if not entry:
            out.append(None)
            continue
        key = tuple(sorted(entry.items()))
        if key not in by_key:
            built = []

            def build(entry=entry, built=built):
                if not built:
                    built.append(_translated_device(device, entry))
                return built[0]

            by_key[key] = build
        out.append(by_key[key])
    return out


def solve_batch(*, model: FactorizedModel, applied_fields: Sequence[Optional[Callable]],
                circulating_currents: Optional[Sequence[Dict[str, float]]] = None,
                terminal_currents: Optional[Sequence[Dict[str, Dict[str, Union[float, str]]]]] = None,
                vortices: Optional[Sequence[Sequence[Vortex]]] = None,
                translations: Optional[Sequence[Optional[Dict[str, Sequence[float]]]]] = None,
                field_units: str = "mT",
                iterations: int = 0, check_inversion: bool = False, last_only: bool = False,
                gather: bool = True, _solver: str = "superscreen_b200.solve_batch") -> List[List[Solution]]:
    """Solves B models that share one factorization in a single batched pass (multi-RHS getrs,
    multi-RHS matrix-free operator, one film-to-film exchange per iteration for the whole batch).

    This is an extension with no counterpart in the reference, which would call ``solve`` B times
    (e.g. once per driven hole in ``Device.mutual_inductance_matrix``, device/device.py:610-639, or
    once per applied field in a sweep).  ``out[b]`` equals
    ``solve(model=model_b, applied_field=applied_fields[b], iterations=iterations)`` where
    ``model_b`` is ``model`` factorized with ``circulating_currents[b]`` (floats in ``model.current_units``),
    ``terminal_currents[b]`` and ``vortices[b]``.  ``terminal_currents`` has one
    ``{film: {terminal: current}}`` dict per entry (floats in ``model.current_units`` or unit strings; default: ``model.terminal_currents`` for
    every entry); an entry replaces the model's terminal currents completely: films it does not name
    carry no transport current.  The transport stream of every entry is computed once per call, with
    one column per entry in every device operation.  ``vortices`` has one sequence of ``Vortex`` per
    entry (default: ``model.vortices`` for every entry); likewise an entry replaces the model's vortices
    completely, and an empty sequence (or ``None``) means no vortices.  The vortices are checked as ``factorize_model``
    checks them (``TypeError`` for an item that is not a ``Vortex``, ``KeyError`` for an unknown film,
    ``ValueError`` for a vortex outside its film or inside a hole, naming the entry) before any device
    work.  Each vortex enters its own entry's right-hand side as a sparse correction, so a scan over
    vortex positions costs one batched solve, not one solve per position.

    ``translations`` has one ``None`` or ``{layer: (dx, dy) | (dx, dy, dz)}`` dict per entry (in
    ``device.length_units``): every film, hole, terminal and abstract region of a listed layer moves rigidly
    by ``(dx, dy)`` and the layer by ``dz``; other layers stay put.  ``model_b`` is then the factorization of
    the device with those layers moved as ``Device.translate`` moves them.  Only the applied field (evaluated
    at the moved vertices) and the film-to-film coupling depend on where a film sits, so a scan over the
    positions of a layer stack (a scanning SQUID over a sample) costs one batched solve against one
    factorization per film.  A layer with a position-dependent Lambda, or that holds a vortex of the entry,
    cannot move (``ValueError``, naming the entry); so do unknown layers (``KeyError``) and shifts that are
    not 2 or 3 finite reals (``ValueError``).  Films with terminals may move.  ``Solution.device`` of an
    entry that moves something is the moved device, built on first access and shared by the entries with
    the same translation, so ``hole_fluxoid``, ``polygon_fluxoid`` and ``field_at_position`` work on it
    unchanged (an explicit fluxoid contour must be moved with its layer by the caller).  When no entry moves
    anything the call is the one without ``translations``.  Multi-rank models replicate the small shift
    table; that path is untested, as it is for vortices.  With
    ``last_only`` only the final iterate is brought to the host (``out[b]`` has one element).
    With a multi-rank model, ``gather=False`` skips the replication of the results: every rank's
    solutions then hold only the films it owns (enough for per-film post-processing such as the
    fluxoid rows of ``Device.mutual_inductance_matrix``).
    """
    torch = _torch()
    model = _check_model_args(None, model, None, None, None, None)
    device = model.device
    B = len(applied_fields)
    if B == 0:
        return []
    if circulating_currents is None:
        circulating_currents = [model.circulating_currents] * B
    if len(circulating_currents) != B:
        raise ValueError("applied_fields and circulating_currents must have the same length.")
    for cc in circulating_currents:
        diff = set(cc) - set(device.holes)
        if diff:
            raise KeyError(f"circulating_currents contains keys not in self.device.holes: {list(diff)!r}")
    if terminal_currents is not None:
        terminal_currents = _batch_terminal_currents(model, terminal_currents, B)
    vortices_by_film = None
    if vortices is not None:
        vortices_by_film = _batch_vortices(device, vortices, B)
        vortices = [[] if entry is None else list(entry) for entry in vortices]
    moves = None
    if translations is not None:
        if vortices is not None:
            entry_vortices = vortices
        else:
            entry_vortices = [list(itertools.chain.from_iterable(model.vortices.values()))
                              if isinstance(model.vortices, dict) else list(model.vortices)] * B
        moves = _batch_translations(device, translations, B, entry_vortices)
    current_units = model.current_units
    length_units = device.length_units
    field_conversion = field_conversion_factor(field_units, current_units, length_units=length_units).magnitude
    zero_field = ConstantField(0)
    funcs = [f or zero_field for f in applied_fields]
    owned = _owned_films(model)
    film_names = [f for f in device.films if gather or f in owned]
    with _lib.nvtx_range("scb.solve_batch.fields"):
        # (a field function that appears several times in the batch is evaluated once per film and
        # translation of the film's layer)
        evaluated = {}
        per_b = []
        for b, f in enumerate(funcs):
            entry_moves = {} if moves is None else moves[b]
            fields = {}
            for name in film_names:
                layer = model.film_info[name].layer
                key = (id(f), name, entry_moves.get(layer))
                hit = evaluated.get(key)
                if hit is None:
                    hit = evaluated[key] = _evaluate_applied_field(f, device, model.film_info, device.meshes,
                                                                   field_conversion, films=[name],
                                                                   moves=entry_moves)[name]
                fields[name] = hit
            per_b.append(fields)
        host_fields = {name: np.stack([h[name] for h in per_b], axis=0) for name in film_names}  # (B, n) per film
        dev_fields = {}
        circ_by_film = {}
        # the circulating currents of all holes of all owned films: ONE table, one upload per device
        hole_rows, tables = {}, {}
        for name in film_names:
            if name in owned:
                dev = device.meshes[name]._data.device
                for hole in model.film_info[name].hole_indices:
                    hole_rows.setdefault(dev, []).append((name, hole))
        for dev, rows in hole_rows.items():
            tables[dev] = _upload(np.array([[float(cc.get(hole, 0.0)) for cc in circulating_currents]
                                            for _, hole in rows], dtype=np.float64), dev)
        for name in film_names:
            if name not in owned:
                continue
            dev = device.meshes[name]._data.device
            # rows are contiguous on the host (fast stack + one H2D copy); the (n, nrhs) layout is made on the device
            if not host_fields[name].any():
                dev_fields[name] = torch.zeros(host_fields[name].shape[::-1], dtype=torch.float64, device=dev)
            else:
                dev_fields[name] = _upload(host_fields[name], dev).t().contiguous()
            circ_by_film[name] = {hole: tables[dev][k] for k, (film, hole) in enumerate(hole_rows.get(dev, []))
                                  if film == name}
    vortex_flux = _u.PHI_0 / _u.MU_0 * _u.conversion_factor("A * m", f"({current_units}) * ({length_units})")
    shifts = None
    if moves is not None:
        shifts = np.array([[entry.get(film.layer, (0.0, 0.0, 0.0)) for film in device.films.values()]
                           for entry in moves], dtype=np.float64)  # (B, films, 3)
    host = _run(model, dev_fields, circ_by_film, vortex_flux, iterations, check_inversion, field_conversion,
                batch=B, last_only=last_only, gather=gather, terminal_currents=terminal_currents,
                vortices=vortices_by_film, shifts=shifts)
    kwargs_list = [dict(applied_field_func=funcs[b], field_units=field_units, current_units=current_units,
                        circulating_currents=dict(circulating_currents[b]),
                        terminal_currents=model.terminal_currents if terminal_currents is None
                        else terminal_currents[b], vortices=model.vortices if vortices is None else vortices[b],
                        solver=_solver)
                   for b in range(B)]
    with _lib.nvtx_range("scb.solve_batch.solutions"):
        per_iter_solutions = _solutions_from_host(device, host, film_names, host_fields, field_conversion,
                                                  kwargs_list, batched=True,
                                                  device_builders=None if moves is None
                                                  else _device_builders(device, moves))
    return [[it[b] for it in per_iter_solutions] for b in range(B)]


def _owned_films(model: FactorizedModel):
    """Names of the films whose systems this rank holds (all of them in a single process)."""
    from ..parallel import Comm, film_owners

    comm = model.comm or Comm()
    owners = film_owners(list(model.device.films), comm)
    return {f for f, r in owners.items() if r == comm.rank}
