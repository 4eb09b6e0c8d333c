"""Per-film linear systems on the B200 (reference solver/solve_film.py).

``factorize_linear_systems`` assembles ``-A`` for every film straight into its LU workspace
(``scb_system_assemble``: fused Q / Laplacian / grad-Lambda terms, one HBM write) and factors it
in place (``scb_getrf_nopiv``).  The hole slabs of ``_build_system_1d`` are never formed: their
only use, ``A_hole @ g[hole]`` (solve_film.py:498-503), is evaluated matrix-free by
``scb_apply_operator``.  ``solve_film`` runs getrs, the CSR gradients and the matrix-free
self-field ``Q @ (w*g)`` on the device and downloads only O(n) vectors.
"""
from __future__ import annotations

import contextlib
import logging
import os
from dataclasses import dataclass, field
from typing import Dict, Optional, Tuple, Union

import numpy as np

from .. import _lib
from ..device import Device
from ..geometry import close_curve, path_vectors  # noqa: F401  (names the reference module exposes)
from ..solution import FilmSolution
from .utils import FilmInfo, stream_from_terminal_current  # noqa: F401

logger = logging.getLogger("solve")

LU_BLOCK = 128


def _torch():
    import torch

    return torch


@dataclass
class LinearSystem:
    """reference solver/solve_film.py:18-35.  ``indices`` is a host int64 array; the factorization
    lives on the device (``lu``: padded row-major LU of ``-A`` without pivoting, ``dinv``: inverses
    of its diagonal blocks).  ``A`` and ``lu_piv`` are lazy host views for API compatibility."""

    indices: np.ndarray
    film_info: FilmInfo = field(repr=False, default=None)
    grad_Lambda_term: Union[float, object] = 0.0  # device CSR data on the operator pattern, or 0
    n_pad: int = 0
    lu: object = field(repr=False, default=None)      # torch (n_pad, n_pad) f64
    dinv: object = field(repr=False, default=None)    # torch f64
    indices_dev: object = field(repr=False, default=None)
    margin: object = field(repr=False, default=None)  # torch (n_int,) row-dominance lower bound
    refine: bool = False  # not provably dominant -> iterative refinement in every solve
    # symmetric mode: the factors are those of S = D (-A) D^-1, D = diag(sym_scale) = sqrt(w[indices])
    sym_scale: object = field(repr=False, default=None)
    pos: object = field(repr=False, default=None)  # torch int32 (n,): mesh vertex -> row of this system, -1 outside
    # pivoted factorization (scb_getrf_piv): P (-A) = L U.  piv: LAPACK-style interchanges (int32, n_pad),
    # perm: int64 (n_int,) with row r of P(-A) = row perm[r] of -A, rhs_indices_dev = indices_dev[perm]
    piv: object = field(repr=False, default=None)
    perm: object = field(repr=False, default=None)
    rhs_indices_dev: object = field(repr=False, default=None)

    @property
    def A(self) -> np.ndarray:
        """Dense A, re-assembled on demand: (n_int, n_int) for a factored system (the LU overwrote
        the workspace), or the (n, len(indices)) column slab of ``_build_system_1d`` (reference
        solve_film.py:285-293) for the hole / boundary systems, which are otherwise applied
        matrix-free."""
        torch = _torch()
        if self.n_pad == 0:
            d = self.film_info.mesh._data
            k = len(self.indices)
            with torch.cuda.device(d.device):
                E = torch.zeros(d.n, k, dtype=torch.float64, device=d.device)
                E[self.indices_dev, torch.arange(k, device=d.device)] = 1.0
                return apply_operator(self.film_info, E, src_idx=self.indices_dev).cpu().numpy()
        M = assemble_negA(self.film_info, self.indices_dev, len(self.indices), self.n_pad,
                          self.grad_Lambda_term if not isinstance(self.grad_Lambda_term, float) else None)[0]
        # (always the plain, unsymmetrised -A)
        n = len(self.indices)
        return (-M[:n, :n]).cpu().numpy()

    def to_hdf5(self, h5group) -> None:
        """reference solver/solve_film.py:37-51"""
        from .. import io as _io

        _io.linear_system_to_hdf5(self, h5group)

    @property
    def lu_piv(self) -> Tuple[np.ndarray, np.ndarray]:
        """(lu, piv) of ``-A`` in scipy.linalg.lu_factor layout; piv is the identity unless the system
        was factored with partial pivoting (``scb_getrf_piv``).
        In symmetric mode the stored factors belong to S = D (-A) D^-1; since
        -A = (D^-1 L D)(D^-1 U D) with D^-1 L D still unit lower triangular, they are rescaled
        element-wise on the way out."""
        n = len(self.indices)
        lu = self.lu[:n, :n]
        if self.sym_scale is not None:
            lu = lu * (self.sym_scale[None, :] / self.sym_scale[:, None])
        if self.piv is not None:  # partial pivoting: the interchanges, exactly scipy's `piv`
            return lu.cpu().numpy(), self.piv[:n].cpu().numpy().astype(np.int32)
        return lu.cpu().numpy(), np.arange(n, dtype=np.int32)


@dataclass
class TerminalSystems:
    """reference solver/solve_film.py:80-100: the systems needed for the transport-current stream
    function.  ``boundary`` / ``holes`` carry indices only (their slabs are applied matrix-free);
    ``film_without_boundary`` is the LU of the film interior INCLUDING holes;
    ``film_without_boundary_or_holes`` is the film's main system (interior minus holes)."""

    film: str
    boundary: LinearSystem
    holes: Dict[str, LinearSystem]
    film_without_boundary: LinearSystem
    film_without_boundary_or_holes: Optional[LinearSystem] = None


def assemble_negA(info: FilmInfo, ix_dev, n_int: int, n_pad: int, T=None, out=None, want_margin=False,
                  sym_scale_full=None, pos=None, margin=None):
    """-A restricted to ``ix`` in a padded workspace (reference solve_film.py:296-305), or, with
    ``sym_scale_full`` = sqrt(w) per mesh vertex, its diagonally similar symmetric form."""
    torch = _torch()
    L = _lib.lib()
    d = info.mesh._data
    with torch.cuda.device(d.device):
        M = out if out is not None else torch.empty(n_pad, n_pad, dtype=torch.float64, device=d.device)
        if pos is None:
            pos = torch.empty(d.n, dtype=torch.int32, device=d.device)
        if margin is None and want_margin:
            margin = torch.empty(n_int, dtype=torch.float64, device=d.device)
        _lib.check(L.scb_system_assemble(
            d.n, _lib.ptr(d.sites), _lib.ptr(d.t["vertex_areas"]), _lib.ptr(d.qdw), _lib.ptr(d.t["C"]),
            _lib.ptr(info.dev["Lambda"]), _lib.ptr(d.t["op_indptr"]), _lib.ptr(d.t["op_indices"]),
            _lib.ptr(d.t["laplacian"]), _lib.ptr(T), n_int, _lib.ptr(ix_dev), _lib.ptr(pos), n_pad,
            _lib.ptr(M), _lib.ptr(margin), _lib.ptr(sym_scale_full), _lib.stream_ptr()))
    return M, margin


def factorize_linear_systems(device: Device, film_info_dict: Dict[str, FilmInfo], owned=None, deferred=None):
    """reference solver/solve_film.py:151-282 (films without terminals).  ``owned`` restricts the
    (expensive) assembly + LU to the films this rank owns (multi-GPU film sharding).

    ``deferred``: an optional list.  The singularity flags of the factorizations are normally read back
    (one blocking download) before this function returns.  If a list is given and no system needs its
    dominance margin for a decision (symmetric or pivoted factorizations), the read-back is appended to it
    as a callable instead and the function returns while the GPU is still factoring: the caller enqueues
    the solves behind it and calls the check before it trusts the results (``FactorizedModel.finish_checks``)."""
    torch = _torch()
    L = _lib.lib()
    film_systems: Dict[str, LinearSystem] = {}
    hole_systems: Dict[str, Dict[str, LinearSystem]] = {}
    terminal_systems: Dict[str, object] = {}
    pending = []  # (film, system, info flag tensor, side stream): read back once at the end
    n_owned = sum(1 for f in film_info_dict if owned is None or f in owned)
    n_side = int(os.environ.get("SCB_FILM_STREAMS", "8"))
    side_streams = []  # several systems: factor them concurrently (small LUs are latency-bound)
    if n_side > 0 and (n_owned > 1 or any(f in device.terminals for f in film_info_dict)):
        dev0 = next(iter(film_info_dict.values())).mesh._data.device
        side_streams = _lib.film_streams(dev0, min(n_side, max(n_owned, 2)))
    for film_name, info in film_info_dict.items():
        if owned is not None and film_name not in owned:
            hole_systems[film_name] = {}
            continue
        d = info.mesh._data
        with torch.cuda.device(d.device):
            T = None
            if info.lambda_info.inhomogeneous:
                T = torch.empty_like(d.t["laplacian"])
                _lib.check(L.scb_grad_lambda_term(
                    d.n, _lib.ptr(d.t["op_indptr"]), _lib.ptr(d.t["op_indices"]), _lib.ptr(d.t["gradient_x"]),
                    _lib.ptr(d.t["gradient_y"]), _lib.ptr(info.dev["Lambda"]), _lib.ptr(T), _lib.stream_ptr()))
            info.dev["T"] = T
            # For a constant Lambda, -A is diagonally similar (D = W^1/2) to a symmetric matrix:
            # factor that one with the symmetric LU at half the flops (DESIGN.md section 4.3).
            Lam = info.lambda_info.Lambda
            # index sets uploaded once per (device, film, mesh): `geo` lives in the device-level geometry
            # cache of make_film_info, so repeated factorizations of one device (one model per
            # mutual-inductance call, Lambda sweeps) re-use the device copies
            geo = info.dev.get("_geo")
            if geo is None:
                geo = {}

            def cached(key, make):
                hit = geo.get(key)
                if hit is None:
                    hit = geo[key] = make()
                return hit

            sym_full = None
            if use_symmetric() and T is None and (info.dev.get("Lambda_constant")
                                                  or float(Lam.max()) == float(Lam.min())):
                sym_full = cached(("sqrt_w", str(d.device)), lambda: torch.sqrt(d.t["vertex_areas"]))
            hole_systems[film_name] = {}
            for hole_name, indices in info.hole_indices.items():
                hole_systems[film_name][hole_name] = LinearSystem(
                    indices=indices, film_info=info, grad_Lambda_term=T if T is not None else 0.0,
                    indices_dev=cached(("hole_ix", hole_name, str(d.device)),
                                       lambda: torch.as_tensor(indices).to(d.device)))
            def factor(indices, tag):
                indices = np.ascontiguousarray(indices, dtype=np.int64)
                n_int = len(indices)
                if n_int == 0:
                    raise ValueError(f"Film {film_name!r} has no interior mesh vertices.")
                n_pad = -(-n_int // LU_BLOCK) * LU_BLOCK
                # every buffer is allocated on the caller's stream; the kernels may run on a side stream
                ix_dev = cached(("ix", tag, str(d.device)), lambda: torch.as_tensor(indices).to(d.device))
                M = torch.empty(n_pad, n_pad, dtype=torch.float64, device=d.device)
                pos = torch.empty(d.n, dtype=torch.int32, device=d.device)
                margin = torch.empty(n_int, dtype=torch.float64, device=d.device)
                dinv = torch.empty(int(L.scb_getrf_dinv_bytes(n_pad)) // 8, dtype=torch.float64, device=d.device)
                lu_info = torch.zeros(1, dtype=torch.int32, device=d.device)
                sym_scale = None if sym_full is None else cached(
                    ("sym_scale", tag, str(d.device)), lambda: sym_full[ix_dev].contiguous())
                side = side_streams[len(pending) % len(side_streams)] if side_streams else None
                if side is not None:
                    side.wait_stream(torch.cuda.current_stream(d.device))
                piv = perm = rhs_ix = None
                with (torch.cuda.stream(side) if side is not None else contextlib.nullcontext()), \
                        _lib.nvtx_range(f"scb.assemble+getrf[{film_name}, n={n_int}]"):
                    assemble_negA(info, ix_dev, n_int, n_pad, T, out=M, want_margin=True, sym_scale_full=sym_full,
                                  pos=pos, margin=margin)
                    # Pivoting (SCB_PIVOT=auto): the symmetrised constant-Lambda system is definite and
                    # needs none; a general system gets LAPACK-style partial pivoting when its rows are
                    # not provably diagonally dominant (sign-indefinite grad-Lambda term, SURVEY.md Q11)
                    use_piv = False
                    if sym_full is None:
                        mode = pivot_mode()
                        use_piv = mode == "1" or (mode == "auto" and float(margin.min().item()) <= 0.0)
                    if use_piv:
                        piv = torch.empty(n_pad, dtype=torch.int32, device=d.device)
                        perm32 = torch.empty(n_pad, dtype=torch.int32, device=d.device)
                        _lib.check(L.scb_getrf_piv(n_pad, _lib.ptr(M), _lib.ptr(dinv), _lib.ptr(piv), _lib.ptr(perm32),
                                                   _lib.ptr(lu_info), _lib.stream_ptr()))
                        perm = perm32[:n_int].to(torch.int64)
                        rhs_ix = ix_dev[perm]
                    else:
                        getrf = L.scb_getrf_sym_nopiv if sym_full is not None else L.scb_getrf_nopiv
                        _lib.check(getrf(n_pad, _lib.ptr(M), _lib.ptr(dinv), _lib.ptr(lu_info), _lib.stream_ptr()))
                system = LinearSystem(indices=indices, film_info=info, grad_Lambda_term=T if T is not None else 0.0,
                                      n_pad=n_pad, lu=M, dinv=dinv, indices_dev=ix_dev, margin=margin,
                                      sym_scale=sym_scale, pos=pos, piv=piv, perm=perm, rhs_indices_dev=rhs_ix)
                # `pos`, `sym_full` and `T` are only read by kernels queued on the side stream: keep them
                # referenced until the side streams have been joined (the caching allocator would
                # otherwise hand their blocks to the next film's allocations on the caller's stream
                # while the assembly is still pending)
                pending.append((film_name, system, lu_info, side, (pos, sym_full, T)))
                return system

            interior = info.interior_indices
            interior_no_holes = interior
            if info.hole_indices:
                interior_no_holes = cached("interior_no_holes", lambda: np.setdiff1d(
                    interior, np.concatenate(list(info.hole_indices.values()))))
            # (for terminal films the boundary vertices are already excluded from `interior`,
            #  reference solve_film.py:273-274)
            film_systems[film_name] = factor(interior_no_holes, "no_holes")
            if film_name in device.terminals:
                # reference solve_film.py:220-263.  The reference factors the system without holes
                # twice (as the film system and as film_without_boundary_or_holes); once here.
                boundary = np.ascontiguousarray(info.boundary_indices, dtype=np.int64)
                with_holes = factor(interior, "interior") if info.hole_indices else film_systems[film_name]
                terminal_systems[film_name] = TerminalSystems(
                    film=film_name,
                    boundary=LinearSystem(indices=boundary, film_info=info,
                                          grad_Lambda_term=T if T is not None else 0.0,
                                          indices_dev=cached(("boundary_ix", str(d.device)),
                                                             lambda: torch.as_tensor(boundary).to(d.device))),
                    holes=hole_systems[film_name],
                    film_without_boundary=with_holes,
                    film_without_boundary_or_holes=film_systems[film_name] if info.hole_indices else None,
                )
    # independent systems were factored on side streams: join them, then one synchronising read per
    # system (singularity flag + dominance margin)
    for side in {id(p[3]): p[3] for p in pending if p[3] is not None}.values():
        with torch.cuda.device(side.device):
            torch.cuda.current_stream(side.device).wait_stream(side)
    # The dominance margin decides something only for a general, unpivoted system (SCB_PIVOT=0).  The
    # symmetrised constant-Lambda system is definite -- elimination without pivoting is stable on it whether
    # or not its rows are dominant (DESIGN.md section 4.3) -- and a pivoted system is safe by construction.
    needs_margin = [system.sym_scale is None and system.piv is None for _, system, _, _, _ in pending]

    def finish_checks():
        # one download for the flags (and margins) of all systems instead of two blocking reads per system
        if not pending:
            return
        by_dev = {}
        for k, p in enumerate(pending):
            by_dev.setdefault(p[2].device, []).append(k)
        flags_host = [0] * len(pending)
        margins_host = [None] * len(pending)
        for dev_k, ks in by_dev.items():
            km = [k for k in ks if needs_margin[k]]
            with torch.cuda.device(dev_k):
                packed = torch.stack([pending[k][2][0].to(torch.float64) for k in ks]
                                     + [pending[k][1].margin.min() for k in km]).cpu().numpy()
            for j, k in enumerate(ks):
                flags_host[k] = int(packed[j])
            for j, k in enumerate(km):
                margins_host[k] = float(packed[len(ks) + j])
        for k, (film_name, system, lu_info, _, _keepalive) in enumerate(pending):
            flag = flags_host[k]
            mm = margins_host[k]
            if flag != 0:
                raise np.linalg.LinAlgError(
                    f"Film {film_name!r}: zero or non-finite pivot at row {flag - 1} of the LU factorization."
                )
            if system.piv is not None:
                logger.info(f"Film {film_name!r}: factored with partial pivoting.")
            elif mm is not None and mm <= 0:
                # SURVEY.md Q11: dominance can fail for non-Delaunay (smoothed) meshes or strongly
                # inhomogeneous Lambda.  The unpivoted factors are then used as a preconditioner:
                # every solve is iteratively refined against the matrix-free operator and the
                # final residual is checked (see solve_film_device).
                system.refine = True
                logger.info(
                    f"Film {film_name!r}: system matrix is not provably row-diagonally dominant "
                    f"(margin lower bound {mm:.3e}); solves will use iterative refinement."
                )

    if deferred is not None and not any(needs_margin):
        deferred.append(finish_checks)
    else:
        finish_checks()
    return film_systems, hole_systems, terminal_systems


def pivot_mode() -> str:
    """SCB_PIVOT: 'auto' (default: partial pivoting for general systems whose rows are not provably
    diagonally dominant), '1' (every general system), '0' (never: unpivoted LU + iterative refinement)."""
    mode = os.environ.get("SCB_PIVOT", "auto").lower()
    return mode if mode in ("auto", "0", "1") else "auto"


def use_symmetric() -> bool:
    """Symmetric factorization for constant-Lambda films (default on; SCB_SYMMETRIC=0 disables)."""
    return os.environ.get("SCB_SYMMETRIC", "1") != "0"


def apply_operator(info: FilmInfo, v, src_idx=None, with_sparse: bool = True, out=None, accumulate: bool = False):
    """out[n, nrhs] (+)= A_full[:, src] @ v[src]  (matrix-free; v must vanish outside src)."""
    torch = _torch()
    L = _lib.lib()
    d = info.mesh._data
    v2 = v if v.dim() == 2 else v[:, None]
    v2 = v2.contiguous()
    nrhs = v2.shape[1]
    with torch.cuda.device(d.device):
        if out is None:
            out = torch.empty(d.n, nrhs, dtype=torch.float64, device=d.device)
            accumulate = False
        _lib.check(L.scb_apply_operator(
            d.n, _lib.ptr(d.sites), _lib.ptr(d.t["vertex_areas"]), _lib.ptr(d.qdw),
            _lib.ptr(info.dev["Lambda"]) if with_sparse else None, _lib.ptr(d.t["op_indptr"]),
            _lib.ptr(d.t["op_indices"]), _lib.ptr(d.t["laplacian"]),
            _lib.ptr(info.dev.get("T")) if with_sparse else None,
            0 if src_idx is None else int(src_idx.numel()), _lib.ptr(src_idx), nrhs, _lib.ptr(v2), _lib.ptr(out),
            1 if accumulate else 0, _lib.stream_ptr()))
    return out if v.dim() == 2 else out[:, 0]


def lu_solve(system: LinearSystem, h):
    """x with (-A) x = h for h of shape (n_int,) or (n_int, nrhs) (device tensors)."""
    torch = _torch()
    L = _lib.lib()
    n_int = len(system.indices)
    h2 = h if h.dim() == 2 else h[:, None]
    nrhs = h2.shape[1]
    with torch.cuda.device(system.lu.device):
        B = torch.zeros(system.n_pad, nrhs, dtype=torch.float64, device=system.lu.device)
        if system.perm is not None:  # P (-A) x = P h
            h2 = h2[system.perm]
        # symmetric mode: (-A) x = h  <=>  S (D x) = D h
        B[:n_int] = h2 if system.sym_scale is None else h2 * system.sym_scale[:, None]
        _lib.check(L.scb_getrs_nopiv(system.n_pad, _lib.ptr(system.lu), _lib.ptr(system.dinv), nrhs, _lib.ptr(B),
                                     _lib.stream_ptr()))
    x = B[:n_int]
    if system.sym_scale is not None:
        x = x / system.sym_scale[:, None]
    return x if h.dim() == 2 else x[:, 0]


def spmv(d, key: str, x, alpha: float = 1.0):
    """alpha * (operator @ x) for a vertex operator ('gradient_x' ...) or a triangle gradient."""
    torch = _torch()
    L = _lib.lib()
    x2 = (x if x.dim() == 2 else x[:, None]).contiguous()
    nrhs = x2.shape[1]
    if key in ("gtri_x", "gtri_y"):
        nrows, indptr, indices = d.m, d.gtri_indptr, d.t["gtri_indices"]
    else:
        nrows, indptr, indices = d.n, d.t["op_indptr"], d.t["op_indices"]
    with torch.cuda.device(d.device):
        y = torch.empty(nrows, nrhs, dtype=torch.float64, device=d.device)
        _lib.check(L.scb_spmv(nrows, _lib.ptr(indptr), _lib.ptr(indices), _lib.ptr(d.t[key]), nrhs, _lib.ptr(x2),
                              float(alpha), 0.0, _lib.ptr(y), _lib.stream_ptr()))
    return y if x.dim() == 2 else y[:, 0]


def hole_boundary_state(film_info: FilmInfo, hole_systems: Dict[str, LinearSystem], circ, like):
    """Hole boundary conditions (reference solve_film.py:493-503): ``g0[hole] = I_circ`` and the
    effective field ``Ha_eff = -sum_k A[:, hole_k] @ g0[hole_k]`` (matrix-free).  Depends only on the
    circulating currents, not on the applied field: evaluated once per solve call and shared by all
    film-to-film iterations.  ``like`` gives the shape ``(n,)`` / ``(n, B)``.  Returns ``(g0, Ha_eff)``
    or ``(None, None)`` when no hole carries a current."""
    torch = _torch()
    batched = like.dim() == 2
    g0 = None
    for name, s in hole_systems.items():
        cur = circ.get(name, 0)
        if torch.is_tensor(cur):
            if g0 is None:
                g0 = torch.zeros_like(like)
            g0[s.indices_dev] += cur.to(like.dtype)[None, :] if batched else cur.to(like.dtype)
        elif cur:
            if g0 is None:
                g0 = torch.zeros_like(like)
            g0[s.indices_dev] += float(cur)
    if g0 is None:
        return None, None
    src = torch.cat([s.indices_dev for s in hole_systems.values()])
    return g0, -apply_operator(film_info, g0, src_idx=src)


@dataclass
class VortexState:
    """The vortices of one film for every column of a solve, located once per solve call and reused by
    every film-to-film iteration.  Column ``c`` holds vortices ``col_ptr[c] .. col_ptr[c+1]`` (CSR);
    ``j_sub`` is each vortex's nearest system row (j_film), ``j_all`` its nearest mesh vertex (j_device)
    and ``row`` the row of the triangular-solve workspace it enters (``invperm[j_sub]`` for a pivoted
    system).  All device tensors are views of one upload, or outputs of ``scb_locate_vortices``."""

    nrhs: int
    nv: int = 0
    col_ptr: object = field(repr=False, default=None)  # torch int64 (nrhs + 1,)
    nphi0: object = field(repr=False, default=None)    # torch f64 (nv,)
    j_sub: object = field(repr=False, default=None)    # torch int64 (nv,)
    j_all: object = field(repr=False, default=None)    # torch int64 (nv,)
    row: object = field(repr=False, default=None)      # torch int64 (nv,)


def make_vortex_state(film_info: FilmInfo, film_system: LinearSystem, columns) -> VortexState:
    """``columns``: one sequence of ``Vortex`` per column of the solve (all in this film).  The table goes
    to the device in one copy; the nearest vertices are found there (``scb_locate_vortices``), so the solve
    needs no host synchronisation.  No device work when no column has a vortex."""
    counts = [len(c) for c in columns]
    nv = sum(counts)
    if nv == 0:
        return VortexState(nrhs=len(columns))
    torch = _torch()
    L = _lib.lib()
    d = film_info.mesh._data
    vortices = [v for c in columns for v in c]
    col_ptr = np.zeros(len(columns) + 1, dtype=np.int64)
    np.cumsum(counts, out=col_ptr[1:])
    xy = np.array([(float(v.x), float(v.y)) for v in vortices], dtype=np.float64)
    nphi0 = np.array([float(v.nPhi0) for v in vortices], dtype=np.float64)
    # one host buffer (the float64 parts stored bit for bit as int64), one asynchronous copy from pinned
    # memory: the caller's stream may still be factoring, and the host does not wait for it
    host = torch.from_numpy(np.concatenate([col_ptr, xy.ravel().view(np.int64), nphi0.view(np.int64)]))
    with torch.cuda.device(d.device):
        buf = host.pin_memory().to(d.device, non_blocking=True)
        nc = len(col_ptr)
        col_ptr_d = buf[:nc]
        xy_d = buf[nc:nc + 2 * nv].view(torch.float64)
        nphi0_d = buf[nc + 2 * nv:].view(torch.float64)
        j = torch.empty(2, nv, dtype=torch.int64, device=d.device)
        _lib.check(L.scb_locate_vortices(nv, _lib.ptr(xy_d), d.n, _lib.ptr(d.sites), len(film_system.indices),
                                         _lib.ptr(film_system.indices_dev), _lib.ptr(j[0]), _lib.ptr(j[1]),
                                         _lib.stream_ptr()))
        row = j[0]
        if film_system.perm is not None:  # B[r] = h[perm[r]]: the vortex at system row j enters row invperm[j]
            invperm = torch.empty_like(film_system.perm)
            invperm[film_system.perm] = torch.arange(len(film_system.perm), dtype=torch.int64, device=d.device)
            row = invperm[row]
    return VortexState(nrhs=len(columns), nv=nv, col_ptr=col_ptr_d, nphi0=nphi0_d, j_sub=j[0], j_all=j[1], row=row)


def apply_vortex_rhs(state: VortexState, film_info: FilmInfo, B, vortex_flux: float, scale=None,
                     workspace: bool = True) -> None:
    """Subtracts the vortex terms from the right-hand sides in place (``scb_vortex_rhs``): from the
    triangular-solve workspace ``B`` (``workspace``: rows permuted and scaled as the factors need them), or
    from ``h`` of ``(-A) x = h`` in system-row order (``lu_solve`` permutes and scales it)."""
    L = _lib.lib()
    d = film_info.mesh._data
    assert B.is_contiguous() and (B.shape[1] if B.dim() == 2 else 1) == state.nrhs
    _lib.check(L.scb_vortex_rhs(state.nrhs, _lib.ptr(state.col_ptr), _lib.ptr(state.row if workspace else state.j_sub),
                                _lib.ptr(state.j_all), _lib.ptr(state.nphi0), _lib.ptr(d.t["vertex_areas"]),
                                float(vortex_flux), _lib.ptr(scale if workspace else None), _lib.ptr(B),
                                _lib.stream_ptr()))


def solve_film_device(*, film_info: FilmInfo, film_system: LinearSystem, hole_systems: Dict[str, LinearSystem],
                      applied_field, vortex_flux: float, field_from_other_films=None,
                      check_inversion: bool = False, circulating_currents=None, terminal_systems=None,
                      device: Optional[Device] = None, hole_state=None, want_self_field: bool = True,
                      terminal_currents=None, transport_state=None, vortex_state=None):
    """Device-side body of ``solve_film`` (reference solve_film.py:483-565): all arguments and
    results are device tensors in solver units.  ``want_self_field=False`` skips the screening mat-vec
    ``Q @ (w g)`` (an output only: the next Jacobi step needs ``J``, not the self field) and returns
    ``None`` in its place.

    ``applied_field`` is ``(n,)`` or, for a batch of B right-hand sides sharing the factorization,
    ``(n, B)``; ``circulating_currents`` (default: ``film_info.circulating_currents``) maps hole
    names to a float or to a ``(B,)`` tensor.  ``hole_state`` = ``hole_boundary_state(...)`` if the
    caller has it already.  For a film with transport terminals, ``terminal_currents`` (default:
    ``film_info.terminal_currents``) is one ``{terminal: current}`` dict, or a sequence of B of them for a
    batch, and ``transport_state`` = ``terminal_transport_state(...)`` if the caller has it already.
    ``vortex_state`` = ``make_vortex_state(...)`` gives every column its own vortices (default: the film's
    vortices in every column); the vortex term is a correction to the right-hand side of each column
    (include/scb.h, scb_vortex_rhs), so it costs no solve of its own.  Returns ``(g, J, self_field)`` with
    shapes ``(n,), (n, 2), (n,)`` or ``(n, B), (n, B, 2), (n, B)``.
    """
    torch = _torch()
    L = _lib.lib()
    info = film_info
    d = info.mesh._data
    circ = info.circulating_currents if circulating_currents is None else circulating_currents
    batched = applied_field.dim() == 2
    nrhs = applied_field.shape[1] if batched else 1
    transport = terminal_systems is not None
    with torch.cuda.device(d.device):
        if vortex_state is None:
            vortex_state = make_vortex_state(info, film_system, [info.vortices] * nrhs)
        vortices = vortex_state.nv > 0
        if hole_state is None:
            hole_state = hole_boundary_state(info, hole_systems, circ, applied_field) if hole_systems \
                else (None, None)
        g0, Ha_eff = hole_state
        if not (transport or film_system.refine or check_inversion):
            # the common case in four fused steps: right-hand side, triangular solves, stream function,
            # current density (one kernel each instead of ~20 gather / scatter / elementwise launches)
            n_int, n_pad = len(film_system.indices), film_system.n_pad
            if film_system.pos is None:  # (a system that was not built by factorize_linear_systems)
                pos = torch.full((d.n,), -1, dtype=torch.int32, device=d.device)
                pos[film_system.indices_dev] = torch.arange(n_int, dtype=torch.int32, device=d.device)
                film_system.pos = pos
            B = torch.empty((n_pad, nrhs), dtype=torch.float64, device=d.device)
            applied_c = applied_field.contiguous()
            other_c = None if field_from_other_films is None else field_from_other_films.contiguous()
            s = _lib.stream_ptr()
            rhs_ix = film_system.indices_dev if film_system.rhs_indices_dev is None else film_system.rhs_indices_dev
            g = torch.empty_like(applied_c)
            if not vortices:
                # right-hand side, triangular solves, stream function and current density in ONE foreign call
                J = torch.empty((d.n, nrhs, 2) if batched else (d.n, 2), dtype=torch.float64, device=d.device)
                _lib.check(L.scb_solve_step(
                    d.n, n_int, n_pad, nrhs, _lib.ptr(rhs_ix), _lib.ptr(applied_c), _lib.ptr(other_c),
                    _lib.ptr(Ha_eff), _lib.ptr(film_system.sym_scale), _lib.ptr(film_system.lu),
                    _lib.ptr(film_system.dinv), _lib.ptr(B), _lib.ptr(film_system.pos), _lib.ptr(g0), _lib.ptr(g),
                    _lib.ptr(d.t["op_indptr"]), _lib.ptr(d.t["op_indices"]), _lib.ptr(d.t["gradient_x"]),
                    _lib.ptr(d.t["gradient_y"]), _lib.ptr(J), s))
                if not want_self_field:
                    return g, J, None
                return g, J, apply_operator(info, g, src_idx=None, with_sparse=False)
            _lib.check(L.scb_solve_rhs(n_int, n_pad, _lib.ptr(rhs_ix), nrhs, _lib.ptr(applied_c),
                                       _lib.ptr(other_c), _lib.ptr(Ha_eff), _lib.ptr(film_system.sym_scale),
                                       _lib.ptr(B), s))
            apply_vortex_rhs(vortex_state, info, B, vortex_flux, scale=film_system.sym_scale)
            _lib.check(L.scb_getrs_nopiv(n_pad, _lib.ptr(film_system.lu), _lib.ptr(film_system.dinv), nrhs,
                                         _lib.ptr(B), s))
            _lib.check(L.scb_solve_stream(d.n, nrhs, _lib.ptr(film_system.pos), _lib.ptr(B),
                                          _lib.ptr(film_system.sym_scale), _lib.ptr(g0), _lib.ptr(g), s))
        else:
            Hz = applied_field if field_from_other_films is None else applied_field + field_from_other_films
            g = torch.zeros_like(Hz) if g0 is None else g0.clone()
            if transport:
                # reference solve_film.py:505-524
                if transport_state is None:
                    if terminal_currents is None:
                        terminal_currents = info.terminal_currents or {}
                    if batched and isinstance(terminal_currents, dict):
                        terminal_currents = [terminal_currents] * nrhs
                    transport_state = terminal_transport_state(device, info, terminal_systems, terminal_currents)
                g_transport, Ha_transport = transport_state
                if g_transport is not None:  # (None: no entry carries a terminal current)
                    g = g + g_transport
                    Ha_eff = Ha_transport if Ha_eff is None else Ha_eff + Ha_transport
            ix = film_system.indices_dev
            h = Hz[ix] if Ha_eff is None else Hz[ix] - Ha_eff[ix]
            if vortices:  # (the refinement and check_inversion residuals then see the true right-hand side)
                apply_vortex_rhs(vortex_state, info, h, vortex_flux, workspace=False)
            gf = lu_solve(film_system, h)
            if film_system.refine or check_inversion:
                # residual of (-A) gf = h through the matrix-free operator (reference check_inversion,
                # solve_film.py:533-540); refinement steps when the LU is only a preconditioner
                def residual(x):
                    full = torch.zeros_like(Hz)
                    full[ix] = x
                    return h + apply_operator(info, full, src_idx=ix)[ix]

                r = residual(gf)
                scale = h.abs().max().clamp_min(1e-300)
                if film_system.refine:
                    for _ in range(5):
                        if float((r.abs().max() / scale).item()) <= 1e-13:
                            break
                        gf = gf + lu_solve(film_system, r)
                        r = residual(gf)
                err = float((r.abs().max() / scale).item())
                if film_system.refine and not err <= 1e-10:  # (NaN counts as not converged)
                    # the factors were only a preconditioner (system not provably dominant) and the
                    # refinement did not converge: never hand back an unconverged stream function
                    raise np.linalg.LinAlgError(
                        f"Film {info.name!r}: iterative refinement against the unpivoted LU stalled at a relative "
                        f"residual of {err:.3e} (> 1e-10); factorize with pivoting (SCB_PIVOT=1)."
                    )
                if err > 1e-8:
                    logger.warning(
                        f"Unable to solve for stream function in {info.name!r}), "
                        f"maximum error {r.abs().max().item():.3e} (relative {err:.3e})."
                    )
            g[ix] += gf
        # J = curl(g z) = [dg/dy, -dg/dx]: (n, 2), or (n, B, 2) for a batch (source-major, the layout
        # of the film-to-film exchange)
        g = g.contiguous()
        J = torch.empty((d.n, nrhs, 2) if batched else (d.n, 2), dtype=torch.float64, device=d.device)
        _lib.check(L.scb_current_density(d.n, _lib.ptr(d.t["op_indptr"]), _lib.ptr(d.t["op_indices"]),
                                         _lib.ptr(d.t["gradient_x"]), _lib.ptr(d.t["gradient_y"]), nrhs, _lib.ptr(g),
                                         _lib.ptr(J), _lib.stream_ptr()))
        if not want_self_field:
            self_field = None
        elif transport:
            # _biot_savart_within_film on per-triangle current densities (solve_film.py:557-562):
            # J_tri [m, nsets, 2] source-major
            J_tri = torch.stack([spmv(d, "gtri_y", g), spmv(d, "gtri_x", g, alpha=-1.0)], dim=-1).contiguous()
            self_field = torch.empty(g.shape, dtype=torch.float64, device=d.device)
            _lib.check(L.scb_biot_savart_within_film(
                d.n, _lib.ptr(d.sites), d.m, _lib.ptr(d.t["centroids"]), _lib.ptr(d.t["triangle_areas"]),
                _lib.ptr(J_tri), 1.0 / (4.0 * np.pi), nrhs, _lib.ptr(self_field), _lib.stream_ptr()))
        else:
            # Q @ (w * g), matrix-free
            self_field = apply_operator(info, g, src_idx=None, with_sparse=False)
    return g, J, self_field


def _terminal_boundary_values(device: Device, film_info: FilmInfo, terminal_systems: TerminalSystems,
                              columns) -> Optional[np.ndarray]:
    """Host part of reference solver/solve_film.py:308-335 for every ``{terminal: current}`` dict in
    ``columns``: the stream function on the (counter-clockwise) boundary, shifted by
    ``- max(g) + ptp(g) / 2`` per column.  Returns ``(n_boundary + 1, B)``: the boundary values and, in
    the last row, the value the shift gives every other vertex; a column without current is all zero.
    ``None`` when no column carries a current."""
    from .utils import stream_from_terminal_current

    if not any(any(c.values()) for c in columns):
        return None
    points = film_info.mesh.sites
    boundary_indices = terminal_systems.boundary.indices
    nb = len(boundary_indices)
    out = np.zeros((nb + 1, len(columns)))
    # per terminal: its boundary positions (ascending) -- the same for every column
    ix_by_terminal = {t.name: np.sort(t.contains_points(points[boundary_indices], index=True))
                      for t in device.terminals[film_info.name]}
    for k, terminal_currents in enumerate(columns):
        if not any(terminal_currents.values()):
            continue
        g = np.zeros(nb + 1)  # (boundary positions; the last entry stands for every other vertex)
        for name, ix_boundary in ix_by_terminal.items():
            current = terminal_currents[name]
            stream = stream_from_terminal_current(points[boundary_indices[ix_boundary]], -current)
            g[ix_boundary[:-1]] += stream
            g[ix_boundary[-1]:nb] += stream[-1]
        out[:, k] = g - np.max(g) + np.ptp(g) / 2
    return out


def solve_for_terminal_current_stream(device: Device, film_info: FilmInfo, terminal_systems: TerminalSystems,
                                      terminal_currents):
    """reference solver/solve_film.py:308-390 for one ``{terminal: current}`` dict -> ``(n,)``, or for a
    sequence of B of them -> ``(n, B)``.  The boundary values are a few hundred numbers per column and
    are set on the host exactly as the reference does (one upload for the whole batch); the slab products
    ``A_boundary @ g`` and ``A_hole @ g``, the hole averages and the two solves run on the device with
    one column per entry.  Returns the device tensor."""
    torch = _torch()
    batched = not isinstance(terminal_currents, dict)
    columns = list(terminal_currents) if batched else [terminal_currents]
    d = film_info.mesh._data
    values = _terminal_boundary_values(device, film_info, terminal_systems, columns)
    with torch.cuda.device(d.device):
        if values is None:
            g_dev = torch.zeros(d.n, len(columns), dtype=torch.float64, device=d.device)
            return g_dev if batched else g_dev[:, 0]
        values = torch.as_tensor(values).to(d.device)
        b_dev = terminal_systems.boundary.indices_dev
        nb = int(b_dev.numel())
        g_dev = values[nb:].expand(d.n, -1).clone()
        g_dev[b_dev] = values[:nb]
        # only the boundary entries enter A_boundary @ g[boundary] (the constant shift above also
        # moved the interior entries, which the solve below overwrites)
        v = torch.zeros_like(g_dev)
        v[b_dev] = values[:nb]
        Ha_eff = -apply_operator(film_info, v, src_idx=b_dev)
        # 2. interior ignoring the holes
        sys_all = terminal_systems.film_without_boundary
        g_dev[sys_all.indices_dev] = lu_solve(sys_all, -Ha_eff[sys_all.indices_dev])
        if len(terminal_systems.holes):
            # 3. holes at the weighted average of step 2, then the interior without holes
            w = d.t["vertex_areas"]
            for system in terminal_systems.holes.values():
                ixh = system.indices_dev
                v[ixh] = ((g_dev[ixh] * w[ixh, None]).sum(dim=0) / w[ixh].sum())[None, :]
                g_dev[ixh] = v[ixh]
            src = torch.cat([b_dev] + [s.indices_dev for s in terminal_systems.holes.values()])
            Ha_eff = -apply_operator(film_info, v, src_idx=src)
            sys_nh = terminal_systems.film_without_boundary_or_holes
            g_dev[sys_nh.indices_dev] = lu_solve(sys_nh, -Ha_eff[sys_nh.indices_dev])
    return g_dev if batched else g_dev[:, 0]


def _boundary_geometry(film_info: FilmInfo, terminal_systems: TerminalSystems):
    """Edge centres, lengths and unit normals of the closed boundary curve (reference
    solve_film.py:510-518); cached with the film's other index-set derived arrays."""
    torch = _torch()
    d = film_info.mesh._data
    geo = film_info.dev.get("_geo")
    key = ("boundary_edges", str(d.device))
    hit = None if geo is None else geo.get(key)
    if hit is None:
        b = terminal_systems.boundary.indices_dev
        boundary_sites = d.sites[b]
        centers = (0.5 * (boundary_sites + torch.roll(boundary_sites, -1, dims=0))).contiguous()
        dr = torch.roll(boundary_sites, -1, dims=0) - boundary_sites  # edges of the closed curve
        lengths = torch.linalg.norm(dr, dim=1)
        normals = (torch.stack([dr[:, 1], -dr[:, 0]], dim=1) / lengths[:, None]).contiguous()
        hit = (centers, lengths, normals)
        if geo is not None:
            geo[key] = hit
    return hit


def terminal_transport_state(device: Device, film_info: FilmInfo, terminal_systems: TerminalSystems,
                             terminal_currents):
    """Transport part of a terminal film's solve (reference solve_film.py:505-524): the stream function
    of the terminal currents and the effective field of its boundary values.  Depends neither on the
    applied field nor on the film-to-film iterate: evaluated once per solve call.  ``terminal_currents``
    is one ``{terminal: current}`` dict (results ``(n,)``) or a sequence of B of them (``(n, B)``).
    Returns ``(g_transport, Ha_transport)``, or ``(None, None)`` when no entry carries a current."""
    torch = _torch()
    L = _lib.lib()
    batched = not isinstance(terminal_currents, dict)
    columns = list(terminal_currents) if batched else [terminal_currents]
    if not any(any(c.values()) for c in columns):
        return None, None
    d = film_info.mesh._data
    with torch.cuda.device(d.device):
        g_transport = solve_for_terminal_current_stream(device, film_info, terminal_systems, columns)
        b = terminal_systems.boundary.indices_dev
        centers, lengths, normals = _boundary_geometry(film_info, terminal_systems)
        boundary_stream = g_transport[b]
        boundary_stream = 0.5 * (boundary_stream + torch.roll(boundary_stream, -1, dims=0))
        Ha_transport = torch.empty(d.n, len(columns), dtype=torch.float64, device=d.device)
        # _get_boundary_effective_field (solve_film.py:393-412): kind 4, strengths = stream * length [nb, B]
        _lib.check(L.scb_biot_savart(
            4, d.n, _lib.ptr(d.sites), int(b.numel()), _lib.ptr(centers),
            _lib.ptr((boundary_stream * lengths[:, None]).contiguous()), _lib.ptr(normals), 0.0,
            1.0 / (4.0 * np.pi), len(columns), _lib.ptr(Ha_transport), _lib.stream_ptr()))
    if not batched:
        return g_transport[:, 0], Ha_transport[:, 0]
    return g_transport, Ha_transport


def solve_film(*, device: Device, applied_field: np.ndarray, film_info: FilmInfo, film_system: LinearSystem,
               hole_systems: Dict[str, LinearSystem], field_conversion: float, vortex_flux: float,
               terminal_systems=None, field_from_other_films: Optional[np.ndarray] = None,
               check_inversion: bool = False) -> FilmSolution:
    """reference solver/solve_film.py:440-574 (host arrays in, FilmSolution out)."""
    torch = _torch()
    dev = film_info.mesh._data.device
    H = torch.as_tensor(np.ascontiguousarray(applied_field, dtype=np.float64)).to(dev)
    other = None
    if field_from_other_films is not None:
        other = torch.as_tensor(np.ascontiguousarray(field_from_other_films, dtype=np.float64)).to(dev)
    g, J, self_field = solve_film_device(
        film_info=film_info, film_system=film_system, hole_systems=hole_systems, applied_field=H,
        vortex_flux=vortex_flux, field_from_other_films=other, check_inversion=check_inversion,
        terminal_systems=terminal_systems, device=device)
    if field_from_other_films is not None:
        field_from_other_films = np.asarray(field_from_other_films) / field_conversion
    return FilmSolution(
        stream=g.cpu().numpy(),
        current_density=J.cpu().numpy(),
        applied_field=np.asarray(applied_field) / field_conversion,
        self_field=(self_field / field_conversion).cpu().numpy(),
        field_from_other_films=field_from_other_films,
    )
