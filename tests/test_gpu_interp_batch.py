"""Point location, polygon masks and interpolation on the device (csrc/interp.cu): scb_tri_locate against a brute-force
numpy restatement of its contract, scb_points_in_polygon against geometry.points_in_polygon, scb_tri_interpolate
against np.einsum, and interp_current_density_batch / interp_field_batch against the per-solution host methods row
by row; chunking, caching and host-side validation."""
import copy
import types

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sc():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import superscreen_b200 as sc

    return sc


def _dev(a, dtype=np.float64):
    import torch

    return torch.as_tensor(np.ascontiguousarray(a, dtype=dtype)).cuda()


# ---------------------------------------------------------------------------------------------
# meshes and points
# ---------------------------------------------------------------------------------------------
def _lattice_mesh(nx, ny, sx=1.0, sy=1.0, jitter=0.0, seed=0):
    """Structured triangulation of an nx x ny lattice (optionally jittered inside)."""
    x, y = np.meshgrid(np.arange(nx + 1) * sx, np.arange(ny + 1) * sy)
    sites = np.stack([x.ravel(), y.ravel()], axis=1).astype(float)
    if jitter:
        rng = np.random.default_rng(seed)
        inner = (x.ravel() > 0) & (x.ravel() < nx * sx) & (y.ravel() > 0) & (y.ravel() < ny * sy)
        sites[inner] += rng.uniform(-jitter, jitter, (int(inner.sum()), 2)) * [sx, sy]
    v = lambda i, j: j * (nx + 1) + i
    el = []
    for j in range(ny):
        for i in range(nx):
            el.append([v(i, j), v(i + 1, j), v(i + 1, j + 1)])
            el.append([v(i, j), v(i + 1, j + 1), v(i, j + 1)])
    return sites, np.array(el, dtype=np.int64)


def _edges(elements):
    e = np.sort(np.concatenate([elements[:, [0, 1]], elements[:, [1, 2]], elements[:, [2, 0]]]), axis=1)
    uniq, counts = np.unique(e, axis=0, return_counts=True)
    return uniq[counts == 2], uniq[counts == 1]  # interior, boundary


def _probe_points(sites, elements, rng, n_random=400, n_edges=150):
    interior, boundary = _edges(elements)
    lo, hi = sites.min(axis=0), sites.max(axis=0)
    ext = hi - lo
    pts = [rng.uniform(lo - 0.1 * ext, hi + 0.1 * ext, (n_random, 2)), sites]
    for edges in (interior, boundary):
        e = edges[rng.choice(len(edges), min(n_edges, len(edges)), replace=False)]
        a, b = sites[e[:, 0]], sites[e[:, 1]]
        mid = 0.5 * (a + b)
        d = b - a
        normal = np.stack([-d[:, 1], d[:, 0]], axis=1)  # (length of the edge)
        pts.append(mid)
        for rel in (1e-13, 1e-11):
            pts += [mid + rel * normal, mid - rel * normal]
    pts.append(np.array([[lo[0] - 10 * ext[0], lo[1]], [hi[0] + 1e3 * ext[0], hi[1] + 5 * ext[1]],
                         [np.nan, lo[1]], [lo[0], np.nan], [np.inf, 0.0], [np.nan, np.nan]]))
    return np.concatenate(pts)


def _reference_locate(sites, elements, xy, grid):
    """The contract of scb_tri_locate over ALL triangles (chunks of triangles, numpy)."""
    from superscreen_b200.solution import _barycentric

    q = len(xy)
    best = np.full(q, -np.inf)
    best_t = np.full(q, -1, dtype=np.int64)
    best_l = np.zeros((q, 3))
    P = sites[elements]
    step = max(1, 2_000_000 // max(q, 1))
    r = np.arange(q)
    with np.errstate(all="ignore"):
        for lo in range(0, len(elements), step):
            lam = _barycentric(P[None, lo:lo + step], xy)  # (q, k, 3)
            mn = np.where(np.isfinite(lam).all(axis=2), lam.min(axis=2), -np.inf)
            j = np.argmax(mn, axis=1)  # (first maximum: the lowest index in the chunk)
            v = mn[r, j]
            upd = v > best  # (strict: an earlier chunk keeps a tie)
            best[upd], best_t[upd], best_l[upd] = v[upd], lo + j[upd], lam[r, j][upd]
    ingrid = (xy[:, 0] >= grid.x0) & (xy[:, 0] <= grid.x1) & (xy[:, 1] >= grid.y0) & (xy[:, 1] <= grid.y1)
    inside = ingrid & (best >= -1e-12)
    return np.where(inside, best_t, -1), np.where(inside[:, None], best_l, 0.0)


def _device_locate(sc, sites, elements, xy, layout=None):
    import torch

    grid = sc.interp.tri_grid(sites, elements, layout)
    xy_d = _dev(xy)
    tri = torch.empty(len(xy), dtype=torch.int64, device="cuda")
    bary = torch.empty((len(xy), 3), dtype=torch.float64, device="cuda")
    sc.interp.locate(grid, xy_d, tri, bary)
    return grid, tri.cpu().numpy(), bary.cpu().numpy()


def _check_locate(sc, sites, elements, seed, layout=None):
    rng = np.random.default_rng(seed)
    xy = _probe_points(sites, elements, rng)
    grid, tri, bary = _device_locate(sc, sites, elements, xy, layout)
    ref_tri, ref_bary = _reference_locate(sites, elements, xy, grid)
    bad = np.flatnonzero(tri != ref_tri)
    assert len(bad) == 0, (len(bad), xy[bad[:5]], tri[bad[:5]], ref_tri[bad[:5]])
    assert np.array_equal(bary, ref_bary)
    assert (tri >= 0).any() and (tri < 0).any()
    return grid


def test_locate_ring_golden_mesh(sc, golden):
    g = golden("ring")
    _check_locate(sc, g["in_sites"], g["in_elements"], 0)


def test_locate_c2_square(sc):
    from superscreen_b200.synthetic import square_mesh

    sites, elements = square_mesh(10.0, 20164, seed=0)
    _check_locate(sc, sites, elements, 1)


def test_locate_sliver_mesh(sc):
    sites, elements = _lattice_mesh(60, 4, sx=1.0, sy=1e-4, jitter=0.2, seed=3)  # aspect ratio up to ~10^4
    _check_locate(sc, sites, elements, 2)


def test_locate_grid_through_vertices_and_one_cell(sc):
    sites, elements = _lattice_mesh(8, 8)
    # cell boundaries at every lattice line: vertices and edges lie on cell boundaries
    grid = _check_locate(sc, sites, elements, 4, layout=(0.0, 0.0, 1.0, 8, 8))
    assert grid.ncx == 8 and grid.x1 == 8.0
    _check_locate(sc, sites, elements, 5, layout=(-1.0, -1.0, 10.0, 1, 1))  # one cell
    _check_locate(sc, *_lattice_mesh(8, 8, jitter=0.3, seed=1), 6, layout=(0.0, 0.0, 2.0, 4, 4))


# ---------------------------------------------------------------------------------------------
# polygon masks
# ---------------------------------------------------------------------------------------------
def _polygon_probe(poly, rng, lo, hi):
    ring = poly if len(poly) < 2 or not np.array_equal(poly[0], poly[-1]) else poly[:-1]
    nxt = np.roll(ring, -1, axis=0)
    t = rng.uniform(0, 1, (len(ring), 1))
    on_edges = ring + t * (nxt - ring)
    horizontal = ring[np.isclose(ring[:, 1], nxt[:, 1])]
    level = [np.stack([np.linspace(lo[0], hi[0], 17), np.full(17, y)], axis=1) for y in horizontal[:8, 1]]
    return np.concatenate([ring, 0.5 * (ring + nxt), on_edges, rng.uniform(lo, hi, (3000, 2))] + level)


def test_points_in_polygon_equals_host(sc):
    from superscreen_b200.geometry import box, circle, points_in_polygon

    rng = np.random.default_rng(7)
    for poly in (box(4.0, 3.0, points=40), circle(2.0, 400), box(1.0, points=4)):
        P = sc.Polygon("p", layer="l", points=poly)
        lo, hi = P.points.min(axis=0) - 0.5, P.points.max(axis=0) + 0.5
        xy = _polygon_probe(P.points, rng, lo, hi)
        ref = points_in_polygon(P.points, xy)
        assert ref.any() and not ref.all()
        assert np.array_equal(sc.interp.points_in_polygon(P, xy), ref)
        assert np.array_equal(sc.interp.points_in_polygon(P, xy), P.contains_points(xy))


def test_points_in_composite_polygons_equal_host(sc):
    from superscreen_b200 import configs
    from superscreen_b200.device import CompositePolygon

    device, _, meshes = configs.ibm_susceptometer(attach_meshes=False)
    rng = np.random.default_rng(8)
    n_composite = 0
    for name, film in device.films.items():
        n_composite += isinstance(film, CompositePolygon)
        sites = meshes[name][0]
        rings = film.rings + (film.cut_rings if isinstance(film, CompositePolygon) else [])
        xy = np.concatenate([sites] + [_polygon_probe(r, rng, sites.min(axis=0), sites.max(axis=0)) for r in rings])
        ref = film.contains_points(xy)
        assert np.array_equal(sc.interp.points_in_polygon(film, xy), ref), name
    assert n_composite >= 2


# ---------------------------------------------------------------------------------------------
# interpolation kernel
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nsets", [1, 2, 7, 8, 9, 63, 64, 65, 130])
@pytest.mark.parametrize("ncomp", [1, 2])
def test_interpolate_kernel_against_einsum(sc, golden, nsets, ncomp):
    import torch

    g = golden("ring")
    sites, elements = g["in_sites"], g["in_elements"]
    rng = np.random.default_rng(nsets * 10 + ncomp)
    xy = _probe_points(sites, elements, rng, n_random=500, n_edges=50)
    grid, tri, bary = _device_locate(sc, sites, elements, xy)
    n, q = len(sites), len(xy)
    values = rng.standard_normal((nsets, n, ncomp)) * 10.0 ** rng.integers(-6, 6, (nsets, n, ncomp))
    bad = rng.random((nsets, n, ncomp)) < 0.01
    values[bad] = rng.choice([np.nan, np.inf, -np.inf], int(bad.sum()))
    values[:, :5] = -0.0
    mask = (rng.random(q) < 0.9).astype(np.uint8)
    for m_, scale in ((None, 1.0), (mask, 1e-3)):
        out = torch.full((nsets, q, ncomp), 7.0, dtype=torch.float64, device="cuda")
        sc.interp.interpolate(grid, _dev(tri, np.int64), _dev(bary), _dev(values), out,
                              None if m_ is None else _dev(m_, np.uint8), scale)
        out = out.cpu().numpy()
        ok = tri >= 0
        for s in range(nsets):
            v = values[s][:, 0] if ncomp == 1 else values[s]
            with np.errstate(all="ignore"):
                ref = np.einsum("qk,qk...->q...", bary, v[elements[np.where(ok, tri, 0)]]).reshape(q, ncomp)
            ref[~ok] = 0
            if m_ is not None:
                ref[m_ == 0] = 0
            ref[~np.isfinite(ref).all(axis=1)] = 0
            if scale != 1.0:
                ref = ref * scale
            assert np.array_equal(out[s], ref), (s, np.nanmax(np.abs(out[s] - ref)))
            assert not np.signbit(out[s][ref == 0]).any()


# ---------------------------------------------------------------------------------------------
# batches against the per-solution host methods
# ---------------------------------------------------------------------------------------------
def _ring_device(sc, g):
    device = sc.Device("ring", layers=[sc.Layer("layer", Lambda=5.0, z0=float(g["in_z0"]))],
                       films=[sc.Polygon("ring", layer="layer", points=g["in_film_polygon"])],
                       holes=[sc.Polygon("hole", layer="layer", points=g["in_hole_polygon"])])
    device.set_meshes({"ring": (g["in_sites"], g["in_elements"])})
    return device


def _two_rings_device(sc, g):
    layers = [sc.Layer("lo", Lambda=float(g["in_lower_Lambda"][0]), z0=float(g["in_lower_z0"])),
              sc.Layer("up", Lambda=float(g["in_upper_Lambda"][0]), z0=float(g["in_upper_z0"]))]
    films = [sc.Polygon("lower", layer="lo", points=g["in_lower_film_polygon"]),
             sc.Polygon("upper", layer="up", points=g["in_upper_film_polygon"])]
    holes = [sc.Polygon("lower_hole", layer="lo", points=g["in_lower_hole_polygon"]),
             sc.Polygon("upper_hole", layer="up", points=g["in_upper_hole_polygon"])]
    device = sc.Device("two", layers=layers, films=films, holes=holes)
    device.set_meshes({k: (g[f"in_{k}_sites"], g[f"in_{k}_elements"]) for k in ("lower", "upper")})
    return device


_BATCHES = {}


def _ring_batch(sc, g, B, seed=0):
    """B solve_batch entries on the ring: fields, circulating currents and 0-2 vortices."""
    key = ("ring", B, seed)
    if key in _BATCHES:
        return _BATCHES[key]
    model = sc.factorize_model(device=_ring_device(sc, g), current_units="uA")
    rng = np.random.default_rng(seed)
    fields = [None if b % 4 == 0 else sc.ConstantField(float(rng.uniform(-0.5, 0.5))) for b in range(B)]
    circ = [{"hole": float(rng.uniform(-20, 20))} if b % 3 == 1 else {} for b in range(B)]
    vortices = []
    for b in range(B):
        entry = []
        for _ in range(b % 3):
            rad, th = rng.uniform(2.3, 3.7), rng.uniform(0, 2 * np.pi)
            entry.append(sc.Vortex(x=float(rad * np.cos(th)), y=float(rad * np.sin(th)), film="ring"))
        vortices.append(entry)
    batch = sc.solve_batch(model=model, applied_fields=fields, circulating_currents=circ, vortices=vortices)
    _BATCHES[key] = [sols[-1] for sols in batch]
    return _BATCHES[key]


def _two_film_batch(sc, g, B=5):
    model = sc.factorize_model(device=_two_rings_device(sc, g), current_units="uA")
    batch = sc.solve_batch(model=model, applied_fields=[sc.ConstantField(0.1 * (b + 1)) for b in range(B)],
                           circulating_currents=[{"lower_hole": 10.0 * b} for b in range(B)], iterations=2)
    return [s[-1] for s in batch]


def _grid(half, k):
    # (shifted off the origin and the axes; covers the mesh and points outside it)
    x, y = np.meshgrid(np.linspace(-half, half, k) + 0.0123, np.linspace(-half, half, k) - 0.0071)
    return np.stack([x.ravel(), y.ravel()], axis=1)


def _near_boundary(sites, elements, xy, tol):
    _, boundary = _edges(elements)
    a, b = sites[boundary[:, 0]], sites[boundary[:, 1]]
    near = np.zeros(len(xy), dtype=bool)
    for k in range(len(xy)):
        d = b - a
        t = np.clip(np.einsum("ec,ec->e", xy[k] - a, d) / np.einsum("ec,ec->e", d, d), 0, 1)
        near[k] = np.min(np.linalg.norm(a + t[:, None] * d - xy[k], axis=1)) <= tol
    return near


def _assert_batch_rows(sc, batch, ref_rows, mesh, positions, film_mask=None):
    """Bits where the host's _locate and the device choose the same triangle (or both find none), 1e-13 max|row|
    elsewhere; the inside / outside decision may differ only within 1e-9 of the mesh boundary."""
    from superscreen_b200.solution import _locate

    ok, tri_h, _ = _locate(mesh.sites, mesh.elements, np.atleast_2d(positions).astype(float), 16)
    _, tri_d, _ = _device_locate(sc, mesh.sites, mesh.elements, positions)
    ok_d = tri_d >= 0
    differ = ok != ok_d
    if differ.any():
        assert _near_boundary(mesh.sites, mesh.elements, positions[differ], 1e-9).all()
    same = (~ok & ~ok_d) | (ok & ok_d & (tri_h == tri_d))
    assert same.mean() > 0.9
    assert len(batch) == len(ref_rows)
    for b, ref in enumerate(ref_rows):
        row = batch[b]
        assert row.shape == ref.shape, (row.shape, ref.shape)
        assert np.array_equal(row[same], ref[same]), (b, np.abs(row[same] - ref[same]).max())
        scale = np.abs(ref).max()
        assert np.abs(row[~same] - ref[~same]).max(initial=0) <= 1e-13 * scale, b


DATASETS = ("total_field", "applied_field", "self_field", "field_from_other_films")


@pytest.mark.parametrize("B", [1, 7, 64, 130])
def test_batch_rows_equal_per_solution_rows(sc, golden, B):
    sols = _ring_batch(sc, golden("ring"), B, seed=B)
    positions = _grid(5.0, 41)  # the mesh disk has radius 4.4: a quarter of the points lie outside it
    mesh = sols[0].device.meshes["ring"]
    J = sc.interp_current_density_batch(sols, positions, film="ring")
    assert J.shape == (B, len(positions), 2)
    _assert_batch_rows(sc, J, [s.interp_current_density(positions, film="ring") for s in sols], mesh, positions)
    for dataset in DATASETS:
        F = sc.interp_field_batch(sols, positions, film="ring", dataset=dataset)
        assert F.shape == (B, len(positions)), dataset
        _assert_batch_rows(sc, F, [s.interp_field(positions, film="ring", dataset=dataset) for s in sols], mesh,
                           positions)
    assert not sc.interp_field_batch(sols, positions, film="ring", dataset="field_from_other_films").any()


def test_batch_units(sc, golden):
    sols = _ring_batch(sc, golden("ring"), 7, seed=7)
    positions = _grid(5.0, 29)
    mesh = sols[0].device.meshes["ring"]
    for units in ("A / m", "mA / um", "(uA) / (um)", None):
        J = sc.interp_current_density_batch(sols, positions, film="ring", units=units, with_units=True)
        ref = [s.interp_current_density(positions, film="ring", units=units, with_units=True) for s in sols]
        assert str(J.units) == str(ref[0].units), units
        _assert_batch_rows(sc, J.magnitude, [r.magnitude for r in ref], mesh, positions)
        plain = sc.interp_current_density_batch(sols, positions, film="ring", units=units)
        assert isinstance(plain, np.ndarray) and np.array_equal(plain, J.magnitude)
    for units in ("uT", "A / m", "mT", None):
        for dataset in ("total_field", "self_field"):
            F = sc.interp_field_batch(sols, positions, film="ring", dataset=dataset, units=units, with_units=True)
            ref = [s.interp_field(positions, film="ring", dataset=dataset, units=units, with_units=True)
                   for s in sols]
            assert str(F.units) == str(ref[0].units), units
            _assert_batch_rows(sc, F.magnitude, [r.magnitude for r in ref], mesh, positions)


def test_two_film_device(sc, golden):
    sols = _two_film_batch(sc, golden("two_rings"))
    positions = _grid(6.0, 37)
    for film in ("lower", "upper"):
        mesh = sols[0].device.meshes[film]
        J = sc.interp_current_density_batch(sols, positions, film=film, units="A/m")
        _assert_batch_rows(sc, J, [s.interp_current_density(positions, film=film, units="A/m") for s in sols], mesh,
                           positions)
        for dataset in DATASETS:
            F = sc.interp_field_batch(sols, positions, film=film, dataset=dataset, units="uT")
            ref = [s.interp_field(positions, film=film, dataset=dataset, units="uT") for s in sols]
            _assert_batch_rows(sc, F, ref, mesh, positions)
        assert sc.interp_field_batch(sols, positions, film=film, dataset="field_from_other_films").any()


def test_chunk_boundaries(sc, golden, monkeypatch):
    from superscreen_b200 import solution

    sols = _ring_batch(sc, golden("ring"), 7, seed=7)
    positions = _grid(5.0, 23)
    J = sc.interp_current_density_batch(sols, positions, film="ring")
    F = sc.interp_field_batch(sols, positions, film="ring")
    monkeypatch.setattr(solution, "_INTERP_CHUNK_ELEMS", 97)  # 6 points per chunk of J, 13 of a field
    assert np.array_equal(sc.interp_current_density_batch(sols, positions, film="ring"), J)
    assert np.array_equal(sc.interp_field_batch(sols, positions, film="ring"), F)
    monkeypatch.setattr(solution, "_INTERP_CHUNK_ELEMS", 1)  # one point per chunk
    assert np.array_equal(sc.interp_field_batch(sols, positions[:50], film="ring"), F[:, :50])


def test_determinism_and_caches(sc, golden):
    sols = _ring_batch(sc, golden("ring"), 7, seed=7)
    positions = _grid(5.0, 31)
    J = sc.interp_current_density_batch(sols, positions, film="ring")
    assert np.array_equal(J, sc.interp_current_density_batch(sols, positions, film="ring"))
    # a replaced current-density array
    s = copy.copy(sols[2])
    fs = copy.copy(s.film_solutions["ring"])
    fs.current_density = 3.0 * fs.current_density
    s.film_solutions = {"ring": fs}
    mesh = sols[0].device.meshes["ring"]
    J2 = sc.interp_current_density_batch([sols[0], s], positions, film="ring")
    assert np.array_equal(J2[0], J[0])
    _assert_batch_rows(sc, J2, [sols[0].interp_current_density(positions, film="ring"),
                                s.interp_current_density(positions, film="ring")], mesh, positions)
    assert not np.array_equal(J2[1], J[2])
    # a replaced mesh (the same triangles, the vertices moved): a new grid, the host's result
    moved = types.SimpleNamespace(sites=mesh.sites * 1.1, elements=mesh.elements.copy())
    t = copy.copy(sols[1])
    t.device = t.device.copy()
    t.device.meshes = {"ring": moved}
    J3 = sc.interp_current_density_batch([t], positions, film="ring")
    _assert_batch_rows(sc, J3, [t.interp_current_density(positions, film="ring")], moved, positions)
    assert not np.array_equal(J3[0], J[1])


def test_empty_inputs(sc, golden):
    sols = _ring_batch(sc, golden("ring"), 7, seed=7)
    assert sc.interp_current_density_batch([], _grid(1.0, 4), film="ring").shape == (0, 16, 2)
    assert sc.interp_field_batch([], _grid(1.0, 4), film="ring").shape == (0, 16)
    assert sc.interp_current_density_batch(sols, np.zeros((0, 2)), film="ring").shape == (7, 0, 2)
    assert sc.interp_field_batch(sols, np.zeros((0, 2)), film="ring").shape == (7, 0)


# ---------------------------------------------------------------------------------------------
# validation
# ---------------------------------------------------------------------------------------------
def test_bad_batches_raise_before_any_device_work(sc, golden):
    from superscreen_b200 import _lib

    sols = _ring_batch(sc, golden("ring"), 7, seed=7)[:3]
    two = _two_film_batch(sc, golden("two_rings"), 2)

    def variant(**attrs):
        s = copy.copy(sols[1])
        s.device = s.device.copy()
        for key, value in attrs.items():
            if key == "mesh":
                s.device.meshes = dict(s.device.meshes)
                s.device.meshes["ring"] = value
            elif key == "length_units":
                s.device._length_units = value
            else:
                setattr(s, key, value)
        return s

    mesh = sols[0].device.meshes["ring"]
    cases = [
        ([sols[0], "nope"], {}, TypeError, r"solutions\[1\]"),
        ([sols[0], sols[1], two[0]], {}, ValueError, r"solutions\[2\].*'ring'"),
        ([sols[0], variant(film_solutions={})], {}, ValueError, r"solutions\[1\].*gather=False"),
        ([sols[0], variant(mesh=types.SimpleNamespace(sites=mesh.sites + 1e-3, elements=mesh.elements))], {},
         ValueError, r"solutions\[1\].*mesh"),
        ([sols[0], sols[2], variant(_field_units="uT")], {}, ValueError, r"solutions\[2\].*units"),
        ([sols[0], variant(_current_units="mA")], {}, ValueError, r"solutions\[1\].*units"),
        ([sols[0], variant(length_units="nm")], {}, ValueError, r"solutions\[1\].*units"),
        (sols, {"method": "cubic"}, NotImplementedError, "linear"),
    ]
    positions = _grid(5.0, 9)
    for batch, kw, exc, match in cases:
        for fn in (sc.interp_current_density_batch, sc.interp_field_batch):
            before = _lib.launch_count()
            with pytest.raises(exc, match=match):
                fn(batch, positions, film="ring", **kw)
            assert _lib.launch_count() == before, (fn.__name__, match)
    before = _lib.launch_count()
    with pytest.raises(ValueError, match="Unexpected dataset: bogus"):
        sc.interp_field_batch(sols, positions, film="ring", dataset="bogus")
    with pytest.raises(ValueError, match=r"solutions\[0\].*'nofilm'"):
        sc.interp_current_density_batch(sols, positions, film="nofilm")
    assert _lib.launch_count() == before
    with pytest.raises(NotImplementedError):
        sols[0].interp_current_density(positions, film="ring", method="cubic")
