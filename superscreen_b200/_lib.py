"""ctypes binding of libsc_b200.so (include/scb.h).

The shared library is the product: if it is missing, cannot be loaded, or no CUDA device is
present, every compute entry point raises -- there is no CPU fallback.  PyTorch is used only to
own device buffers and streams; raw device pointers cross the C ABI.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_int, c_int32, c_int64, c_uint8, c_uint64, c_void_p
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SCB_LIB_PATH") or os.path.join(_HERE, "libsc_b200.so")

_lib = None


class SCBError(RuntimeError):
    pass


class MeshOut(Structure):
    """Mirror of ``struct scb_mesh_out`` (include/scb.h)."""

    _fields_ = [
        (name, c_void_p)
        for name in (
            "triangle_areas", "vertex_areas", "centroids", "C",
            "adj_indptr", "adj_indices", "edges", "edge_is_boundary", "boundary_indices",
            "star_indptr", "star_heads", "star_tris",
            "edge_centers", "edge_directions", "edge_lengths",
            "op_indptr", "op_indices", "laplacian", "gradient_x", "gradient_y",
            "gtri_indices", "gtri_x", "gtri_y",
        )
    ]


EXPORTS = {
    # name: (restype, argtypes)
    "scb_version": (c_int, []),
    "scb_last_error": (c_char_p, []),
    "scb_launch_count": (c_int64, []),
    "scb_mesh_workspace_elems": (c_int64, [c_int64, c_int64]),
    "scb_mesh_analyze": (c_int, [c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "scb_mesh_build": (c_int, [c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_int, POINTER(MeshOut), c_void_p]),
    "scb_mesh_smooth": (c_int, [c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "scb_c_vector": (c_int, [c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "scb_kernel_diagonal": (c_int, [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "scb_grad_lambda_term": (c_int, [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "scb_system_assemble": (c_int, [c_int64] + [c_void_p] * 9 + [c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "scb_apply_operator": (c_int, [c_int64] + [c_void_p] * 8 + [c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_void_p]),
    "scb_getrf_dinv_bytes": (c_int64, [c_int64]),
    "scb_getrf_nopiv": (c_int, [c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "scb_getrf_sym_nopiv": (c_int, [c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "scb_getrf_piv": (c_int, [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "scb_getrs_nopiv": (c_int, [c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "scb_spmv": (c_int, [c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_double, c_double, c_void_p, c_void_p]),
    "scb_solve_rhs": (c_int, [c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "scb_solve_stream": (c_int, [c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "scb_current_density": (c_int, [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "scb_solve_step": (c_int, [c_int64, c_int64, c_int64, c_int64] + [c_void_p] * 17),
    "scb_locate_vortices": (c_int, [c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "scb_vortex_rhs": (c_int, [c_int64] + [c_void_p] * 5 + [c_double, c_void_p, c_void_p, c_void_p]),
    "scb_biot_savart": (c_int, [c_int, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_double, c_double, c_int64, c_void_p, c_void_p]),
    "scb_film_coupling": (c_int, [c_int64, c_void_p, c_double, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                  c_double, c_int64, c_void_p, c_void_p]),
    "scb_film_coupling_translated": (c_int, [c_int64, c_void_p, c_double, c_int64, c_void_p, c_void_p, c_void_p, c_int64,
                                             c_int64, c_double, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p,
                                             c_void_p]),
    "scb_biot_savart_within_film": (c_int, [c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_double, c_int64,
                                            c_void_p, c_void_p]),
    "scb_diag_issue_rate": (c_int, [c_int, c_int64, c_void_p, POINTER(c_double), c_void_p]),
    "scb_diag_scratch_elems": (c_int64, []),
    "scb_cdist": (c_int, [c_int, c_int, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "scb_points_in_rings": (c_int, [c_int64, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "scb_lattice_points": (c_int, [c_int64, c_int64, c_double, c_double, c_double, c_double, c_uint64, c_int, c_void_p,
                                   c_void_p, c_int64, c_void_p, c_double, c_void_p, c_void_p, c_void_p]),
    "scb_delaunay": (c_int, [c_int64, c_void_p, c_double, c_double, c_double, c_int32, c_int32, c_int64, c_void_p,
                             c_void_p, c_void_p]),
    "scb_tri_grid_workspace_elems": (c_int64, [c_int64, c_int64]),
    "scb_tri_grid_count": (c_int, [c_int64, c_void_p, c_void_p, c_double, c_double, c_double, c_int32, c_int32, c_void_p,
                                   c_void_p]),
    "scb_tri_grid_fill": (c_int, [c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "scb_tri_locate": (c_int, [c_int64, c_void_p, c_void_p, c_void_p, c_double, c_double, c_double, c_double, c_double,
                               c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "scb_tri_interpolate": (c_int, [c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int64, c_void_p, c_void_p,
                                    c_double, c_void_p, c_void_p]),
    "scb_points_in_polygon": (c_int, [c_int64, c_void_p, c_int64, c_void_p, c_int, c_void_p, c_void_p]),
}


def load_library(path: Optional[str] = None) -> ctypes.CDLL:
    """Loads libsc_b200.so and declares every prototype of include/scb.h.  Does not need a GPU."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if path is None and not os.environ.get("SCB_LIB_PATH"):
        # the library is built in-tree (python -m superscreen_b200._build).  (Re)build it when it is
        # missing or stale with respect to csrc/ + include/scb.h (content hash, file-locked so that
        # torchrun ranks do not race); a stale library that cannot be rebuilt is an error, never loaded.
        from . import _build

        if _build.needs_build():
            try:
                _build.build()
            except Exception as exc:  # noqa: BLE001
                raise SCBError(
                    f"{p} is missing or older than its sources and building it failed ({exc}). Run "
                    "`python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc). "
                    "superscreen_b200 has no CPU fallback."
                ) from exc
    if not os.path.exists(p):
        raise SCBError(
            f"{p} not found: the CUDA library has not been built. Run "
            "`python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc). "
            "superscreen_b200 has no CPU fallback."
        )
    lib = ctypes.CDLL(p)
    for name, (restype, argtypes) in EXPORTS.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    from ._build import ABI_VERSION

    if lib.scb_version() != ABI_VERSION:
        raise SCBError(f"{p}: ABI version {lib.scb_version()} != expected {ABI_VERSION} (stale library?)")
    if path is None:
        _lib = lib
    return lib


def lib() -> ctypes.CDLL:
    """The loaded library, after checking that a CUDA device is usable (fails loudly otherwise)."""
    import torch

    if not torch.cuda.is_available():
        raise SCBError(
            "superscreen_b200 needs a CUDA device (B200, sm_100a); no CPU fallback exists."
        )
    return load_library()


def check(rc: int) -> None:
    if rc != 0:
        msg = load_library().scb_last_error()
        raise SCBError(f"libsc_b200 error {rc}: {msg.decode() if msg else ''}")


def ptr(t) -> Optional[int]:
    """Device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "tensor must be a contiguous CUDA tensor"
    return t.data_ptr()


def stream_ptr() -> int:
    """Raw handle of torch's current stream on the current device (called before every launch: the direct
    binding, not ``torch.cuda.current_stream()``, which resolves and wraps the stream in Python objects)."""
    import torch

    try:
        return torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice())
    except AttributeError:  # (private binding moved: fall back to the public API)
        return torch.cuda.current_stream().cuda_stream


_FILM_STREAMS: dict = {}


def film_streams(dev, n: int):
    """``n`` side streams of device ``dev`` for independent films (factorizations, the solves of one Jacobi
    step).  One persistent set per device: a stream's first launch costs milliseconds of driver set-up, and
    ``torch.cuda.Stream()`` per call walks through torch's whole pool of 32 before it re-uses one."""
    import torch

    pool = _FILM_STREAMS.setdefault(str(dev), [])
    while len(pool) < n:
        pool.append(torch.cuda.Stream(device=dev))
    return pool[:n]


def launch_count() -> int:
    return int(load_library().scb_launch_count())


_NVTX = os.environ.get("SCB_NVTX", "0") not in ("", "0")
# SCB_HOST_TIMING=1: host wall time per range name (no device synchronisation: enqueue cost, not kernel time)
_HOST_TIMING = os.environ.get("SCB_HOST_TIMING", "0") not in ("", "0")
host_times: dict = {}


def host_timing_report(reset: bool = True) -> str:
    """Table of the accumulated host times of the ``nvtx_range`` sections (``SCB_HOST_TIMING=1``)."""
    lines = [f"{name:<44s} {n:6d} x {1e3 * t / max(n, 1):9.3f} ms = {1e3 * t:9.3f} ms"
             for name, (n, t) in sorted(host_times.items(), key=lambda kv: -kv[1][1])]
    if reset:
        host_times.clear()
    return "\n".join(lines)


class nvtx_range:
    """NVTX range around a stage of the path (``SCB_NVTX=1``; a no-op otherwise): mesh operators,
    film info, per-film assembly + factorization, every Jacobi step, result download."""

    def __init__(self, name: str):
        self.name = name

    def __enter__(self):
        if _NVTX:
            import torch

            torch.cuda.nvtx.range_push(self.name)
        if _HOST_TIMING:
            import time

            self._t0 = time.perf_counter()
        return self

    def __exit__(self, *exc):
        if _HOST_TIMING:
            import time

            key = self.name.split("[")[0]
            n, t = host_times.get(key, (0, 0.0))
            host_times[key] = (n + 1, t + time.perf_counter() - self._t0)
        if _NVTX:
            import torch

            torch.cuda.nvtx.range_pop()
        return False
