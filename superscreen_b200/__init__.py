"""superscreen_b200: a B200-native (sm_100a) implementation of SuperScreen's solve hot path.

Public names mirror ``superscreen/__init__.py:1-20`` for the path in scope (SURVEY.md section 8):
``solve``, ``factorize_model``, ``FactorizedModel``, ``Solution``, ``FilmSolution``, ``Fluxoid``,
``Vortex``, ``Device``, ``Layer``, ``Polygon``, ``Mesh``, ``fem``, ``distance``, ``sources``.
All arithmetic runs in ``libsc_b200.so`` (include/scb.h); there is no CPU fallback.
"""
from . import distance, fem, geometry, interp, io, meshgen, parallel, sources, units
from .device import Device, Layer, Polygon
from .fluxoid import find_fluxoid_solution, make_fluxoid_polygons
from .mesh import Mesh, MeshOperators
from .meshgen import generate_mesh
from .solution import (FilmSolution, Fluxoid, Solution, Vortex, field_at_position_batch, interp_current_density_batch,
                       interp_field_batch, screening_field_at_position_batch, vector_potential_at_position_batch)
from .solver import (
    FactorizedModel,
    FilmInfo,
    LambdaInfo,
    LinearSystem,
    convert_field,
    factorize_model,
    field_conversion_factor,
    solve,
    solve_batch,
)
from .sources import (CompositeParameter, Constant, ConstantField, DipoleField, MonopoleField, Parameter,
                      PearlVortexField, VortexField)

__version__ = "0.1.0"


def version_dict():
    """Versions of the package and of what it runs on (reference about.py ``version_dict``)."""
    return io.version_info()


def version_table(version_info=None, verbose: bool = False) -> str:
    """The same as an HTML table (reference about.py ``version_table``; returned as a string -- IPython is not a
    dependency here)."""
    info = version_info if version_info is not None else version_dict()
    rows = "".join(f"<tr><td>{k}</td><td>{v}</td></tr>" for k, v in info.items())
    return f"<table><tr><th>Software</th><th>Version</th></tr>{rows}</table>"
