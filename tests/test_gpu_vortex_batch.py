"""Per-entry vortices in batched solves: solve_batch(vortices=...) against the live-reference golden, the
CPU oracle and serial solves; batch semantics (linearity, permutation, defaults); the fluxoid of a trapped
vortex; host-side validation; the vortex kernels (scb_locate_vortices, scb_vortex_rhs) in isolation; the
HDF5 round trip of a batched solution with vortices."""
import numpy as np
import pytest

from conftest import rel_l2

TOL_SOLUTION = 1e-8
TOL_BATCH = 1e-12


@pytest.fixture(scope="module")
def sc():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import superscreen_b200 as sc

    return sc


def _ring_device(sc, g, with_mesh=True):
    """The 670-vertex ring of tests/golden/ring.npz: film r = 4, hole r = 2, Lambda = 5."""
    device = sc.Device("ring", layers=[sc.Layer("layer", Lambda=5.0, z0=float(g["in_z0"]))],
                       films=[sc.Polygon("ring", layer="layer", points=g["in_film_polygon"])],
                       holes=[sc.Polygon("hole", layer="layer", points=g["in_hole_polygon"])])
    if with_mesh:
        device.set_meshes({"ring": (g["in_sites"], g["in_elements"])})
    return device


def _square_device(sc, g):
    """The inhomogeneous-Lambda square of tests/golden/square_inhomogeneous.npz (general LU)."""
    from scipy.interpolate import NearestNDInterpolator

    from superscreen_b200.geometry import box

    lam = NearestNDInterpolator(g["in_sites"], g["in_Lambda"])  # exact at the mesh sites
    device = sc.Device("sq", layers=[sc.Layer("layer", Lambda=lambda x, y: lam(x, y), z0=0.0)],
                       films=[sc.Polygon("sq", layer="layer", points=box(6.0, points=4))])
    device.set_meshes({"sq": (g["in_sites"], g["in_elements"])})
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


def _bar_device(sc, g):
    """The 746-vertex bar of tests/golden/transport.npz: one hole, source and drain terminals."""
    terminals = {"bar": [sc.Polygon("source", points=g["in_source_polygon"]),
                         sc.Polygon("drain", points=g["in_drain_polygon"])]}
    device = sc.Device("bar", layers=[sc.Layer("layer", Lambda=float(g["in_Lambda"][0]), z0=0.0)],
                       films=[sc.Polygon("bar", layer="layer", points=g["in_film_polygon"])],
                       holes=[sc.Polygon("hole", layer="layer", points=g["in_hole_polygon"])], terminals=terminals)
    device.set_meshes({"bar": (g["in_sites"], g["in_elements"])})
    return device


def _oracle_films(device, model, Lambda=None):
    """CPU oracle films (oracle/port.py) on the device's meshes and index sets, terminals included."""
    from oracle import port

    films = {}
    for name, film in device.films.items():
        mesh = device.meshes[name]
        info = model.film_info[name]
        lam = Lambda if Lambda is not None else np.full(len(mesh.sites), float(device.layers[film.layer].Lambda))
        of = port.OracleFilm(name=name, mesh=port.build_mesh(mesh.sites, mesh.elements),
                             z0=float(device.layers[film.layer].z0), Lambda=lam,
                             interior_indices=info.interior_indices, hole_indices=dict(info.hole_indices),
                             film_polygon=film.points)
        if name in device.terminals:
            boundary = np.asarray(info.boundary_indices)
            of.boundary_ordered = boundary
            of.terminals = {t.name: np.sort(t.contains_points(mesh.sites[boundary], index=True))
                            for t in device.terminals[name]}
        films[name] = port.factorize_film(of)
    return films


def _as_tuples(vortices):
    return [(v.x, v.y, v.nPhi0) for v in vortices]


def _errs(fs, ref):
    return dict(stream=rel_l2(fs.stream, ref.stream), J=rel_l2(fs.current_density, ref.current_density),
                self_field=rel_l2(fs.self_field, ref.self_field), total=rel_l2(fs.total_field, ref.total_field))


def _assert_same(fs, ref, tol, tag):
    errs = _errs(fs, ref)
    assert all(e <= tol for e in errs.values()), (tag, errs)


def _ring_vortices(sc, film, rng, k, r=(2.3, 3.7)):
    out = []
    for _ in range(k):
        rad, th = rng.uniform(*r), rng.uniform(0, 2 * np.pi)
        out.append(sc.Vortex(x=float(rad * np.cos(th)), y=float(rad * np.sin(th)), film=film,
                             nPhi0=float(rng.choice([1.0, -1.0, 2.0]))))
    return out


def _vortex_entries(sc, film, B, seed, sampler):
    """B entries with 0, 1, 2, 3 vortices in turn, nPhi0 in {1, -1, 2}; entry 6 (if present) holds two
    vortices at the same place."""
    rng = np.random.default_rng(seed)
    entries = [sampler(rng, b % 4) for b in range(B)]
    if B > 6:
        v = sampler(rng, 1)[0]
        entries[6] = [v, sc.Vortex(x=v.x, y=v.y, film=film, nPhi0=-1.0)]
    return entries


def _ring_sampler(sc):
    return lambda rng, k: _ring_vortices(sc, "ring", rng, k)


# ---------------------------------------------------------------------------------------------
# against the reference golden and the oracle
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_ring_golden_vortex_in_a_mixed_batch(sc, golden):
    g = golden("ring")
    device = _ring_device(sc, g)
    model = sc.factorize_model(device=device, current_units="uA")
    vx, vy, nphi = g["in_vortex"]
    vortex = sc.Vortex(x=float(vx), y=float(vy), film="ring", nPhi0=float(nphi))
    batch = sc.solve_batch(model=model, applied_fields=[sc.ConstantField(1.0), None, None, sc.ConstantField(0.3)],
                           circulating_currents=[{}, {"hole": 1000.0}, {}, {"hole": 5.0}],
                           vortices=[[], [], [vortex], [vortex, vortex]])
    for key, sols in zip(["field", "circ", "vortex"], batch):
        fs = sols[0].film_solutions["ring"]
        errs = dict(stream=rel_l2(fs.stream, g[f"out_{key}_stream"]), J=rel_l2(fs.current_density, g[f"out_{key}_J"]),
                    self_field=rel_l2(fs.self_field, g[f"out_{key}_self_field"]))
        if np.any(g[f"out_{key}_applied_field"]):
            errs["applied"] = rel_l2(fs.applied_field, g[f"out_{key}_applied_field"])
        assert all(e <= TOL_SOLUTION for e in errs.values()), (key, errs)
    # entry 3 (0.3 mT, 5 uA, the vortex twice) is linear in the three golden cases: 0.3 field + 5/1000 circ
    # + 2 vortex
    fs = batch[3][0].film_solutions["ring"]
    for attr, key in (("stream", "stream"), ("current_density", "J"), ("self_field", "self_field")):
        ref = 0.3 * g[f"out_field_{key}"] + 0.005 * g[f"out_circ_{key}"] + 2.0 * g[f"out_vortex_{key}"]
        assert rel_l2(getattr(fs, attr), ref) <= TOL_SOLUTION, (attr, rel_l2(getattr(fs, attr), ref))
    assert rel_l2(fs.applied_field, 0.3 * g["out_field_applied_field"]) <= TOL_SOLUTION
    assert batch[2][0].vortices == [vortex] and batch[0][0].vortices == []
    assert batch[3][0].vortices == [vortex, vortex]


def _against_oracle(sc, device, model, films, name, entries, H, check_inversion=False):
    from oracle import port

    conv = port.field_conversion_mT_to_uA_per_um()
    batch = sc.solve_batch(model=model, applied_fields=[sc.ConstantField(h) for h in H],
                           vortices=entries, check_inversion=check_inversion)
    n = len(device.meshes[name].sites)
    for b, entry in enumerate(entries):
        ref = port.solve_film(films[name], np.full(n, H[b] * conv), {}, conv, vortices=_as_tuples(entry))
        _assert_same(batch[b][0].film_solutions[name], ref, TOL_SOLUTION, (b, len(entry)))
        assert batch[b][0].vortices == entry


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["ring", "square_general_lu", "ring_pivoted", "ring_check_inversion"])
def test_vortex_batch_against_oracle(sc, golden, monkeypatch, case):
    if case == "ring_pivoted":
        monkeypatch.setenv("SCB_PIVOT", "1")
        monkeypatch.setenv("SCB_SYMMETRIC", "0")
    if case == "square_general_lu":
        g = golden("square_inhomogeneous")
        device, name, Lambda = _square_device(sc, g), "sq", g["in_Lambda"]

        def sampler(rng, k):
            return [sc.Vortex(x=float(rng.uniform(-2.6, 2.6)), y=float(rng.uniform(-2.6, 2.6)), film="sq",
                              nPhi0=float(rng.choice([1.0, -1.0, 2.0]))) for _ in range(k)]
    else:
        g = golden("ring")
        device, name, Lambda, sampler = _ring_device(sc, g), "ring", None, _ring_sampler(sc)
    model = sc.factorize_model(device=device, current_units="uA")
    system = model.film_systems[name]
    if case == "ring_pivoted":
        assert system.perm is not None and system.sym_scale is None
    elif case == "square_general_lu":
        assert system.sym_scale is None
    else:
        assert system.sym_scale is not None
    entries = _vortex_entries(sc, name, 10, seed=len(case), sampler=sampler)
    H = [0.0 if b % 3 == 0 else 0.1 * b for b in range(10)]
    _against_oracle(sc, device, model, _oracle_films(device, model, Lambda), name, entries, H,
                    check_inversion=case == "ring_check_inversion")


@pytest.mark.gpu
def test_two_films_iterations_against_oracle(sc, golden):
    from oracle import port

    g = golden("two_rings")
    device = _two_rings_device(sc, g)
    model = sc.factorize_model(device=device, current_units="uA")
    V = lambda x, y, film, n=1.0: sc.Vortex(x=x, y=y, film=film, nPhi0=n)  # noqa: E731
    entries = [[V(2.2, 0.3, "lower")], [V(1.8, 0.1, "upper", -1.0)],
               [V(-0.2, -2.1, "lower", 2.0), V(0.0, 1.3, "upper")], []]
    circ = [{}, {"lower_hole": 100.0}, {}, {"upper_hole": -50.0}]
    H = [0.0, 0.2, 0.05, 0.1]
    batch = sc.solve_batch(model=model, applied_fields=[sc.ConstantField(h) for h in H], circulating_currents=circ,
                           vortices=entries, iterations=3)
    films = list(_oracle_films(device, model).values())
    for b, entry in enumerate(entries):
        by_film = {f: _as_tuples([v for v in entry if v.film == f]) for f in device.films}
        osols = port.solve(films, lambda x, y, z, h=H[b]: h * np.ones_like(x), circulating_currents=circ[b],
                           vortices=by_film, iterations=3)
        assert len(batch[b]) == 4
        for it in range(4):
            for name in device.films:
                _assert_same(batch[b][it].film_solutions[name], osols[it][name], TOL_SOLUTION, (b, it, name))
        # and serial solves with the model's vortices
        model.set_vortices(entry)
        model.set_circulating_currents(circ[b])
        ref = sc.solve(model=model, applied_field=sc.ConstantField(H[b]), iterations=3)
        for it in range(4):
            for name in device.films:
                _assert_same(batch[b][it].film_solutions[name], ref[it].film_solutions[name], TOL_BATCH, (b, it))
    model.set_vortices([])
    model.set_circulating_currents({})


@pytest.mark.gpu
def test_transport_film_with_vortices_against_oracle(sc, golden):
    from oracle import port

    g = golden("transport")
    device = _bar_device(sc, g)
    model = sc.factorize_model(device=device, current_units="uA")
    V = lambda x, y, n=1.0: sc.Vortex(x=x, y=y, film="bar", nPhi0=n)  # noqa: E731
    entries = [[V(-2.5, 0.3)], [], [V(2.8, -0.7, -1.0), V(-1.0, -1.0, 2.0)], [V(-2.5, 0.3), V(-2.5, 0.3)]]
    currents = [10.0, 0.0, -25.0, 4.0]
    term = [{"bar": {"source": I, "drain": -I}} for I in currents]
    H = [0.0, 0.1, 0.05, 0.0]
    batch = sc.solve_batch(model=model, applied_fields=[sc.ConstantField(h) for h in H], terminal_currents=term,
                           vortices=entries)
    film = _oracle_films(device, model)["bar"]
    conv = port.field_conversion_mT_to_uA_per_um()
    n = len(device.meshes["bar"].sites)
    for b, entry in enumerate(entries):
        ref = port.solve_film(film, np.full(n, H[b] * conv), {}, conv, vortices=_as_tuples(entry),
                              terminal_currents=term[b]["bar"])
        _assert_same(batch[b][0].film_solutions["bar"], ref, TOL_SOLUTION, b)
        model_b = sc.factorize_model(device=device, current_units="uA", terminal_currents=term[b], vortices=entry)
        serial = sc.solve(model=model_b, applied_field=sc.ConstantField(H[b]))[0]
        _assert_same(batch[b][0].film_solutions["bar"], serial.film_solutions["bar"], TOL_BATCH, b)


# ---------------------------------------------------------------------------------------------
# batch semantics
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 7, 64, 130])
def test_batch_equals_serial(sc, golden, B):
    device = _ring_device(sc, golden("ring"))
    model = sc.factorize_model(device=device, current_units="uA")
    rng = np.random.default_rng(B)
    entries = _vortex_entries(sc, "ring", B, seed=B, sampler=_ring_sampler(sc))
    fields = [None if b % 5 == 0 else sc.ConstantField(float(rng.uniform(-0.5, 0.5))) for b in range(B)]
    circ = [{"hole": float(rng.uniform(-20, 20))} if b % 3 == 1 else {} for b in range(B)]
    batch = sc.solve_batch(model=model, applied_fields=fields, circulating_currents=circ, vortices=entries)
    assert len(batch) == B
    for b in range(B):
        model.set_vortices(entries[b])
        model.set_circulating_currents(circ[b])
        ref = sc.solve(model=model, applied_field=fields[b])[0]
        _assert_same(batch[b][0].film_solutions["ring"], ref.film_solutions["ring"], TOL_BATCH, (B, b))
    model.set_vortices([])
    model.set_circulating_currents({})


@pytest.mark.gpu
def test_linearity_defaults_and_permutation(sc, golden):
    g = golden("ring")
    device = _ring_device(sc, g)
    V = lambda x, y, n=1.0: sc.Vortex(x=x, y=y, film="ring", nPhi0=n)  # noqa: E731
    a, b = V(3.0, 0.2), V(-1.5, -2.6, 2.0)
    model = sc.factorize_model(device=device, current_units="uA")
    field = sc.ConstantField(0.2)
    out = sc.solve_batch(model=model, applied_fields=[field] * 4, circulating_currents=[{"hole": 3.0}] * 4,
                         vortices=[[a, b], [a], [b], []])
    s = [o[0].film_solutions["ring"] for o in out]
    for attr in ("stream", "current_density", "self_field"):
        lhs = getattr(s[0], attr)
        rhs = getattr(s[1], attr) + getattr(s[2], attr) - getattr(s[3], attr)
        assert rel_l2(lhs, rhs) <= TOL_BATCH, attr
    # vortices=None: the model's vortices for every entry, bit for bit what a call without the argument gives
    fields = [sc.ConstantField(0.1 * k) for k in range(5)]
    model.set_vortices([a])
    plain = sc.solve_batch(model=model, applied_fields=fields)
    none = sc.solve_batch(model=model, applied_fields=fields, vortices=None)
    for p, q in zip(plain, none):
        assert np.array_equal(p[0].film_solutions["ring"].stream, q[0].film_solutions["ring"].stream)
        assert np.array_equal(p[0].film_solutions["ring"].self_field, q[0].film_solutions["ring"].self_field)
        assert list(q[0].vortices["ring"]) == [a]
    # all-empty vortices on a model without vortices: bit for bit vortices=None
    model.set_vortices([])
    none = sc.solve_batch(model=model, applied_fields=fields)
    empty = sc.solve_batch(model=model, applied_fields=fields, vortices=[[] for _ in fields])
    for p, q in zip(none, empty):
        assert np.array_equal(p[0].film_solutions["ring"].stream, q[0].film_solutions["ring"].stream)
        assert np.array_equal(p[0].film_solutions["ring"].current_density, q[0].film_solutions["ring"].current_density)
    # permuting the entries permutes the results
    B = 23
    entries = _vortex_entries(sc, "ring", B, seed=3, sampler=_ring_sampler(sc))
    fields = [sc.ConstantField(0.01 * k) for k in range(B)]
    perm = np.random.default_rng(4).permutation(B)
    x = sc.solve_batch(model=model, applied_fields=fields, vortices=entries)
    y = sc.solve_batch(model=model, applied_fields=[fields[p] for p in perm], vortices=[entries[p] for p in perm])
    for k, p in enumerate(perm):
        _assert_same(y[k][0].film_solutions["ring"], x[p][0].film_solutions["ring"], 1e-13, (k, p))


# ---------------------------------------------------------------------------------------------
# physics: the fluxoid of a trapped vortex (reference test_solution.py:221-232 tolerance)
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("nphi0", [1.0, -1.0, 2.0])
def test_fluxoid_around_vortex(sc, golden, nphi0):
    from superscreen_b200.geometry import circle

    device = _ring_device(sc, golden("ring"))
    model = sc.factorize_model(device=device, current_units="uA")
    batch = sc.solve_batch(model=model, applied_fields=[None, None],
                           vortices=[[sc.Vortex(x=3.0, y=0.2, film="ring", nPhi0=nphi0)], []])
    sol = batch[0][0]
    inside = sum(sol.polygon_fluxoid(circle(0.6, 101, center=(3.0, 0.2)), film="ring", with_units=False))
    outside = sum(sol.polygon_fluxoid(circle(0.6, 101, center=(-3.0, 0.2)), film="ring", with_units=False))
    assert abs(inside - nphi0) <= 0.08 * abs(nphi0), inside
    assert abs(outside) <= 0.08, outside
    empty = sum(batch[1][0].polygon_fluxoid(circle(0.6, 101, center=(3.0, 0.2)), film="ring", with_units=False))
    assert abs(empty) <= 1e-6


# ---------------------------------------------------------------------------------------------
# validation
# ---------------------------------------------------------------------------------------------
def _validation_cases(sc):
    V = sc.Vortex
    return [
        ([[V(3.0, 0.2, "ring")]], ValueError, "same length"),                       # wrong length
        ([[], [(3.0, 0.2)]], TypeError, "vortices[1]"),                             # not a Vortex
        ([[], V(3.0, 0.2, "ring")], TypeError, "vortices[1]"),                      # a Vortex, not a sequence
        ([[V(3.0, 0.2, "nofilm")], []], KeyError, "vortices[0]"),                  # unknown film
        ([[], [V(3.0, 0.2, "ring"), V(5.0, 0.0, "ring")]], ValueError, "vortices[1]"),  # outside the film
        ([[V(0.5, 0.5, "ring")], []], ValueError, "vortices[0]"),                  # inside the hole
    ]


def test_batch_vortices_are_checked_on_the_host(golden):
    """The validation helper needs only a Device (no mesh, no GPU)."""
    import superscreen_b200 as sc
    from superscreen_b200.solver.solve import _batch_vortices

    device = _ring_device(sc, golden("ring"), with_mesh=False)
    a, b = sc.Vortex(3.0, 0.2, "ring"), sc.Vortex(-2.5, 1.0, "ring", nPhi0=-1.0)
    ok = _batch_vortices(device, [[a, b], [], None, (b,), np.array([a, b], dtype=object)], 5)
    assert ok == [{"ring": [a, b]}, {"ring": []}, {"ring": []}, {"ring": [b]}, {"ring": [a, b]}]
    for vortices, exc, text in _validation_cases(sc):
        with pytest.raises(exc, match=text.replace("[", r"\[").replace("]", r"\]")):
            _batch_vortices(device, vortices, 2)


@pytest.mark.gpu
def test_bad_vortices_raise_before_any_device_work(sc, golden):
    from superscreen_b200 import _lib

    device = _ring_device(sc, golden("ring"))
    model = sc.factorize_model(device=device, current_units="uA")
    model.finish_checks()
    for vortices, exc, _ in _validation_cases(sc):
        before = _lib.launch_count()
        with pytest.raises(exc):
            sc.solve_batch(model=model, applied_fields=[sc.ConstantField(0.1), None], vortices=vortices)
        assert _lib.launch_count() == before


# ---------------------------------------------------------------------------------------------
# kernels in isolation
# ---------------------------------------------------------------------------------------------
def _locate(lib, torch, xy, sites, sub):
    from superscreen_b200 import _lib

    xy_d, sites_d, sub_d = (torch.as_tensor(np.ascontiguousarray(a)).cuda() for a in (xy, sites, sub))
    j = torch.full((2, len(xy)), -7, dtype=torch.int64, device="cuda")
    _lib.check(lib.scb_locate_vortices(len(xy), _lib.ptr(xy_d), len(sites), _lib.ptr(sites_d), len(sub),
                                       _lib.ptr(sub_d), _lib.ptr(j[0]), _lib.ptr(j[1]), _lib.stream_ptr()))
    torch.cuda.synchronize()
    return j.cpu().numpy()


def _argmin_reference(xy, P):
    """np.argmin(np.linalg.norm(P - q, axis=1)) for every query q, in chunks."""
    out = np.empty(len(xy), dtype=np.int64)
    for s in range(0, len(xy), 32):
        out[s:s + 32] = np.argmin(np.linalg.norm(P[None, :, :] - xy[s:s + 32, None, :], axis=2), axis=1)
    return out


@pytest.mark.gpu
def test_locate_vortices_matches_numpy_argmin(sc):
    import torch

    from superscreen_b200 import _lib

    lib = _lib.lib()
    rng = np.random.default_rng(0)
    for n in (1, 2, 37, 1000, 20000, 60000):
        sites = rng.uniform(-5.0, 5.0, (n, 2))
        n_sub = max(1, n // 3) if n > 1 else 1
        sub = np.sort(rng.choice(n, n_sub, replace=False)).astype(np.int64) if n > 1 else np.zeros(1, np.int64)
        if n >= 1000:
            sub = rng.permutation(sub)  # (any order: the result is the position in `sub`)
        xy = rng.uniform(-6.0, 6.0, (10000, 2))
        xy[:50] *= 1e3  # far outside the mesh
        j = _locate(lib, torch, xy, sites, sub)
        assert np.array_equal(j[1], _argmin_reference(xy, sites)), n
        assert np.array_equal(j[0], _argmin_reference(xy, sites[sub])), n
        for q in range(0, 10000, 997):  # the chunked reference is the per-query numpy expression
            assert j[1, q] == np.argmin(np.linalg.norm(sites - xy[q], axis=1))
        again = _locate(lib, torch, xy, sites, sub)
        assert np.array_equal(j, again)
    # exact ties: integer grid (shuffled), queries at midpoints of neighbours and on duplicated vertices
    gx, gy = np.meshgrid(np.arange(40.0), np.arange(30.0))
    grid = np.column_stack([gx.ravel(), gy.ravel()])
    grid = np.concatenate([grid, grid[:100]])[rng.permutation(len(grid) + 100)]
    mid = np.column_stack([rng.integers(0, 39, 3000) + 0.5, rng.integers(0, 30, 3000).astype(float)])
    mid2 = np.column_stack([rng.integers(0, 39, 3000) + 0.5, rng.integers(0, 29, 3000) + 0.5])
    xy = np.concatenate([mid, mid2, grid[:500]])
    sub = rng.permutation(len(grid))[:900].astype(np.int64)
    j = _locate(lib, torch, xy, grid, sub)
    assert np.array_equal(j[1], _argmin_reference(xy, grid))
    assert np.array_equal(j[0], _argmin_reference(xy, grid[sub]))
    # two different squared distances with the same rounded norm: 1 and 1 + 2^-52 (sqrt rounds to 1), the
    # larger one at the lower index -- numpy picks it, a squared-distance comparison would not
    sites = np.array([[1.0, 2.0 ** -26], [1.0, 0.0], [5.0, 5.0]])
    j = _locate(lib, torch, np.zeros((1, 2)), sites, np.array([2, 1, 0], dtype=np.int64))
    assert np.linalg.norm(sites[0]) == np.linalg.norm(sites[1]) and np.sum(sites[0] ** 2) != np.sum(sites[1] ** 2)
    assert j[1, 0] == 0 == np.argmin(np.linalg.norm(sites - 0.0, axis=1))
    assert j[0, 0] == 1  # sub = [2, 1, 0]: positions 1 (vertex 1) and 2 (vertex 0) tie, the lower position wins
    # nv = 0: nothing to do, nothing written
    _lib.check(lib.scb_locate_vortices(0, None, 10, None, 5, None, None, None, _lib.stream_ptr()))


def _vortex_rhs_reference(B, col_ptr, row, j_all, nphi0, w, flux, scale):
    B = B.copy()
    for c in range(B.shape[1]):
        for v in range(col_ptr[c], col_ptr[c + 1]):
            t = flux * nphi0[v] / w[j_all[v]]
            if scale is not None:
                t = t * scale[row[v]]
            B[row[v], c] = B[row[v], c] - t
    return B


@pytest.mark.gpu
def test_vortex_rhs_matches_numpy(sc):
    import torch

    from superscreen_b200 import _lib

    lib = _lib.lib()
    rng = np.random.default_rng(1)
    n, rows = 900, 700
    w = rng.uniform(0.01, 0.1, n)
    flux = 2.0678338484619295e-15 / (4e-7 * np.pi) * 1e12
    for nrhs in (1, 3, 64, 129, 300):
        counts = rng.integers(0, 4, nrhs)
        counts[::5] = 0  # empty columns
        col_ptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        nv = int(col_ptr[-1])
        j_sub = rng.integers(0, rows, nv).astype(np.int64)
        if nv > 3:
            j_sub[1] = j_sub[0]  # duplicate rows (same or neighbouring columns)
            j_sub[3] = j_sub[2]
        invperm = rng.permutation(rows).astype(np.int64)
        j_all = rng.integers(0, n, nv).astype(np.int64)
        nphi0 = rng.choice([1.0, -1.0, 2.0, 0.5], nv)
        B0 = rng.standard_normal((rows, nrhs))
        for row in (j_sub, invperm[j_sub]):
            for scale in (None, rng.uniform(0.1, 0.3, rows)):
                # (device copies held in variables: a temporary freed before the launch could be re-used)
                dev = [None if a is None else torch.as_tensor(np.ascontiguousarray(a)).cuda()
                       for a in (col_ptr, row, j_all, nphi0, w, scale)]
                outs = []
                for _ in range(2):
                    Bd = torch.as_tensor(B0.copy()).cuda()
                    _lib.check(lib.scb_vortex_rhs(nrhs, *(_lib.ptr(a) for a in dev[:5]), flux, _lib.ptr(dev[5]),
                                                  _lib.ptr(Bd), _lib.stream_ptr()))
                    torch.cuda.synchronize()
                    outs.append(Bd.cpu().numpy())
                ref = _vortex_rhs_reference(B0, col_ptr, row, j_all, nphi0, w, flux, scale)
                assert np.array_equal(outs[0], ref), (nrhs, scale is None)
                assert np.array_equal(outs[0], outs[1])


def test_vortex_entry_points_reject_bad_sizes_without_gpu():
    from superscreen_b200 import _lib

    lib = _lib.load_library()
    for args in [(-1, None, 1, None, 1), (1, None, 0, None, 1), (1, None, 1, None, 0), (1, None, -1, None, 1)]:
        rc = lib.scb_locate_vortices(*args, None, None, None, None)
        assert rc == -1 and b"sizes" in lib.scb_last_error()
    rc = lib.scb_vortex_rhs(-1, None, None, None, None, None, 1.0, None, None, None)
    assert rc == -1 and b"sizes" in lib.scb_last_error()
    assert lib.scb_vortex_rhs(0, None, None, None, None, None, 1.0, None, None, None) == 0


# ---------------------------------------------------------------------------------------------
# HDF5
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_batched_solution_with_vortices_round_trips(sc, golden):
    from superscreen_b200 import io as scio

    device = _ring_device(sc, golden("ring"))
    model = sc.factorize_model(device=device, current_units="uA")
    vortices = [sc.Vortex(3.0, 0.2, "ring"), sc.Vortex(-2.5, 1.0, "ring", nPhi0=-2.0)]
    sol = sc.solve_batch(model=model, applied_fields=[None, sc.ConstantField(0.1)],
                         vortices=[[], vortices])[1][0]
    g = scio.MemoryGroup()
    sol.to_hdf5(g)
    back = sc.Solution.from_hdf5(g)
    assert back.vortices == vortices and sol.vortices == vortices
    for attr in ("stream", "current_density", "applied_field", "self_field"):
        assert np.array_equal(getattr(back.film_solutions["ring"], attr), getattr(sol.film_solutions["ring"], attr))
