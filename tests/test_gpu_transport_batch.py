"""Films with transport terminals in batched solves: solve_batch(terminal_currents=...) against the
live-reference golden, against serial solves and against the CPU oracle; the mutual-inductance matrix and
the fluxoid solution of a device with terminals; the multi-set boundary field and the within-film field
kernels in isolation."""
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


def _bar_device(sc, g, with_mesh=True):
    """The 746-vertex bar of tests/golden/transport.npz: one hole, source and drain terminals."""
    terminals = {"bar": [sc.Polygon("source", points=g["in_source_polygon"]),
                         sc.Polygon("drain", points=g["in_drain_polygon"])]}
    device = sc.Device("bar", layers=[sc.Layer("layer", Lambda=float(g["in_Lambda"][0]), z0=0.0)],
                       films=[sc.Polygon("bar", layer="layer", points=g["in_film_polygon"])],
                       holes=[sc.Polygon("hole", layer="layer", points=g["in_hole_polygon"])], terminals=terminals)
    if with_mesh:
        device.set_meshes({"bar": (g["in_sites"], g["in_elements"])})
    return device


def _bar_ring_device(sc, g):
    """The bar (its outline resampled, so that the terminals cover boundary vertices of the generated
    mesh) plus a ring on a second layer, concentric with the bar's hole, both meshed by Device.make_mesh."""
    from superscreen_b200.geometry import box, circle

    device = _bar_device(sc, g, with_mesh=False)
    device = sc.Device(
        "bar_ring", layers=[device.layers["layer"], sc.Layer("upper", Lambda=0.5, z0=1.0)],
        films=[sc.Polygon("bar", layer="layer", points=box(8.0, 3.0, points=88)),
               sc.Polygon("ring", layer="upper", points=circle(1.2, 64, center=(0.5, 0.2)))],
        holes=[device.holes["hole"], sc.Polygon("ring_hole", layer="upper", points=circle(0.6, 48, center=(0.5, 0.2)))],
        terminals=device.terminals)
    device.make_mesh(min_points={"bar": 900, "ring": 700}, seed=5)
    return device


def _oracle_films(device, model):
    """CPU oracle films (oracle/port.py) on the device's meshes and index sets, terminals included."""
    from oracle import port

    films = []
    for name, film in device.films.items():
        mesh = device.meshes[name]
        info = model.film_info[name]
        om = port.build_mesh(mesh.sites, mesh.elements)
        of = port.OracleFilm(name=name, mesh=om, z0=float(device.layers[film.layer].z0),
                             Lambda=np.full(len(mesh.sites), float(device.layers[film.layer].Lambda)),
                             interior_indices=info.interior_indices, hole_indices=dict(info.hole_indices),
                             film_polygon=film.points)
        if name in device.terminals:
            boundary = np.asarray(info.boundary_indices)
            of.boundary_ordered = boundary
            of.terminals = {t.name: np.sort(t.contains_points(mesh.sites[boundary], index=True))
                            for t in device.terminals[name]}
        films.append(port.factorize_film(of))
    return films


def _oracle_solve(films, H, circulating_currents, terminal_currents, iterations):
    """port.solve (reference solver/solve.py:406-549) for a uniform applied field H (mT), with each
    terminal film driven by its terminal currents through port.solve_film."""
    from oracle import port

    conv = port.field_conversion_mT_to_uA_per_um()
    applied = {f.name: np.full(len(f.mesh.sites), H * conv) for f in films}

    def run(other):
        return {f.name: port.solve_film(f, applied[f.name], circulating_currents, conv,
                                        field_from_other_films=None if other is None else other[f.name],
                                        terminal_currents=terminal_currents.get(f.name))
                for f in films}

    sols = [run(None)]
    for _ in range(iterations):
        other = {f.name: np.zeros(len(f.mesh.sites)) for f in films}
        for src in films:
            for dst in films:
                if src is not dst:
                    other[dst.name] += port.biot_savart_film_to_film(
                        src.mesh.sites, float(src.z0), src.mesh.vertex_areas,
                        np.ascontiguousarray(sols[-1][src.name].current_density), dst.mesh.sites, float(dst.z0))
        sols.append(run(other))
    return sols


def _fluxoid_polygons(device):
    """Circles between each hole and its film's outer edge (the hole of the bar and of the ring are
    circles of radius 0.6 about (0.5, 0.2))."""
    from superscreen_b200.geometry import circle

    return {name: circle(0.9, 101, center=(0.5, 0.2)) for name in device.holes}


def _assert_same(a, b, tol, tag):
    errs = dict(stream=rel_l2(a.stream, b.stream), J=rel_l2(a.current_density, b.current_density),
                self_field=rel_l2(a.self_field, b.self_field), total=rel_l2(a.total_field, b.total_field))
    assert all(e <= tol for e in errs.values()), (tag, errs)


@pytest.mark.gpu
def test_golden_cases_as_one_batch(sc, golden):
    g = golden("transport")
    device = _bar_device(sc, g)
    model = sc.factorize_model(device=device, current_units="uA")
    keys = ["current", "mixed", "nocurrent"]
    terminal_currents = [{"bar": {"source": "10 uA", "drain": "-10 uA"}}, {"bar": {"source": 25.0, "drain": -25.0}},
                         {"bar": {"source": 0.0, "drain": 0.0}}]
    batch = sc.solve_batch(model=model, applied_fields=[None, sc.ConstantField(0.1), sc.ConstantField(0.1)],
                           circulating_currents=[{}, {"hole": 3.0}, {}], terminal_currents=terminal_currents)
    for key, sols in zip(keys, batch):
        fs = sols[0].film_solutions["bar"]
        errs = dict(stream=rel_l2(fs.stream, g[f"out_{key}_stream"]),
                    J=rel_l2(fs.current_density, g[f"out_{key}_J"]),
                    self_field=rel_l2(fs.self_field, g[f"out_{key}_self_field"]))
        if np.any(g[f"out_{key}_applied_field"]):
            errs["applied"] = rel_l2(fs.applied_field, g[f"out_{key}_applied_field"])
        assert all(e <= TOL_SOLUTION for e in errs.values()), (key, errs)
    assert batch[0][0].terminal_currents == {"bar": {"source": 10.0, "drain": -10.0}}
    assert batch[1][0].terminal_currents == {"bar": {"source": 25.0, "drain": -25.0}}


def _entries(sc, B, seed):
    rng = np.random.default_rng(seed)
    fields, circ, term = [], [], []
    for b in range(B):
        I = 0.0 if b % 7 == 3 else float(rng.uniform(-40.0, 40.0))  # (every seventh entry: no current)
        term.append({"bar": {"source": I, "drain": -I}})
        circ.append({"hole": float(rng.uniform(-5.0, 5.0))} if b % 3 == 1 else {})
        fields.append(None if b % 4 == 0 else sc.ConstantField(float(rng.uniform(-0.5, 0.5))))
    return fields, circ, term


def _batch_vs_serial(sc, device, B, seed, check_inversion=False):
    fields, circ, term = _entries(sc, B, seed)
    model = sc.factorize_model(device=device, current_units="uA")
    batch = sc.solve_batch(model=model, applied_fields=fields, circulating_currents=circ, terminal_currents=term,
                           check_inversion=check_inversion)
    assert len(batch) == B
    for b in range(B):
        model_b = sc.factorize_model(device=device, current_units="uA", terminal_currents=term[b],
                                     circulating_currents=circ[b])
        ref = sc.solve(model=model_b, applied_field=fields[b], check_inversion=check_inversion)[0]
        _assert_same(batch[b][0].film_solutions["bar"], ref.film_solutions["bar"], TOL_BATCH, (B, b))
        assert batch[b][0].terminal_currents == term[b]


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 5, 16, 37, 64, 130])
def test_batch_equals_serial(sc, golden, B):
    _batch_vs_serial(sc, _bar_device(sc, golden("transport")), B, seed=B)


@pytest.mark.gpu
def test_batch_equals_serial_inhomogeneous_pivoted(sc, golden, monkeypatch):
    """Callable, inhomogeneous Lambda: general (here: pivoted) LU of every transport system."""
    monkeypatch.setenv("SCB_PIVOT", "1")
    g = golden("transport")
    device = _bar_device(sc, g, with_mesh=False)
    device.layers["layer"].Lambda = lambda x, y: 0.4 + 0.05 * x * x + 0.1 * y
    device.set_meshes({"bar": (g["in_sites"], g["in_elements"])})
    model = sc.factorize_model(device=device, current_units="uA")
    assert model.film_systems["bar"].piv is not None
    assert model.terminal_systems["bar"].film_without_boundary.piv is not None
    _batch_vs_serial(sc, device, 21, seed=11)


@pytest.mark.gpu
def test_batch_equals_serial_check_inversion(sc, golden):
    _batch_vs_serial(sc, _bar_device(sc, golden("transport")), 19, seed=19, check_inversion=True)


@pytest.mark.gpu
def test_multi_film_iterations_against_serial_and_oracle(sc, golden):
    from oracle import port

    device = _bar_ring_device(sc, golden("transport"))
    fields, circ, term = [], [], []
    for b, I in enumerate([12.0, 0.0, -30.0, 7.5]):
        term.append({"bar": {"source": I, "drain": -I}})
        circ.append({"ring_hole": 4.0 * b, "hole": -1.0} if b % 2 else {"ring_hole": 2.0})
        fields.append(sc.ConstantField(0.05 * b))
    model = sc.factorize_model(device=device, current_units="uA")
    batch = sc.solve_batch(model=model, applied_fields=fields, circulating_currents=circ, terminal_currents=term,
                           iterations=2)
    last = sc.solve_batch(model=model, applied_fields=fields, circulating_currents=circ, terminal_currents=term,
                          iterations=2, last_only=True)
    films = None
    for b in range(len(fields)):
        model_b = sc.factorize_model(device=device, current_units="uA", terminal_currents=term[b],
                                     circulating_currents=circ[b])
        ref = sc.solve(model=model_b, applied_field=fields[b], iterations=2)
        assert len(batch[b]) == 3 and len(last[b]) == 1
        for it in range(3):
            for name in device.films:
                _assert_same(batch[b][it].film_solutions[name], ref[it].film_solutions[name], TOL_BATCH, (b, it, name))
        for name in device.films:
            _assert_same(last[b][0].film_solutions[name], batch[b][2].film_solutions[name], 0.0, (b, name))
        if films is None:
            films = _oracle_films(device, model)
        H = 0.05 * b
        osols = _oracle_solve(films, H, circ[b], term[b], iterations=2)
        for it in range(3):
            for name in device.films:
                fs, os_ = batch[b][it].film_solutions[name], osols[it][name]
                errs = [rel_l2(fs.stream, os_.stream), rel_l2(fs.current_density, os_.current_density),
                        rel_l2(fs.self_field, os_.self_field), rel_l2(fs.total_field, os_.total_field)]
                assert max(errs) <= TOL_SOLUTION, (b, it, name, errs)


@pytest.mark.gpu
def test_mutual_inductance_matrix_with_terminals(sc, golden):
    from oracle import port
    from superscreen_b200 import units as _u
    from superscreen_b200.geometry import close_curve, points_in_polygon

    device = _bar_ring_device(sc, golden("transport"))
    polygons = _fluxoid_polygons(device)
    holes = list(device.holes)
    film_of = {h.name: film for film, hs in device.holes_by_film().items() for h in hs}
    M = device.mutual_inductance_matrix(polygons, units="pH", iterations=2)
    assert M.shape == (2, 2)
    # column by column with serial solves (reference device/device.py:610-639)
    Ms = np.zeros((2, 2))
    Mo = np.zeros((2, 2))
    model = sc.factorize_model(device=device, current_units="mA")
    films = {f.name: f for f in _oracle_films(device, model)}
    in_poly = lambda poly, pts: points_in_polygon(poly, pts)
    conv_mA = 1e-3 / port.MU_0 * 1e-3  # mT -> mA/um
    for j, hole in enumerate(holes):
        model_j = sc.factorize_model(device=device, current_units="mA", circulating_currents={hole: 1.0})
        sol = sc.solve(model=model_j, iterations=2)[-1]
        osol = port.solve(list(films.values()), lambda x, y, z: 0.0 * x, circulating_currents={hole: 1.0},
                          iterations=2, field_conversion=conv_mA)[-1]
        for i, name in enumerate(holes):
            fl = sol.polygon_fluxoid(polygons[name], film=film_of[name], units="Phi_0", with_units=False)
            Ms[i, j] = sum(fl) * _u.PHI_0 / 1e-3 * 1e12
            flux, sup = port.polygon_fluxoid(films[film_of[name]], osol[film_of[name]], close_curve(polygons[name]),
                                             in_poly, current_to_A=1e-3)
            Mo[i, j] = (flux + sup) * port.PHI_0 / 1e-3 * 1e12
    assert np.abs(M - Ms).max() <= 1e-10 * np.abs(Ms).max(), (M, Ms)
    assert np.abs(M - Mo).max() <= 1e-8 * np.abs(Mo).max(), (M, Mo)
    assert abs(M[0, 1] - M[1, 0]) <= 0.05 * abs(M[0, 1])
    assert M[0, 0] > 0 and M[1, 1] > 0


@pytest.mark.gpu
def test_find_fluxoid_solution_with_bias_current(sc, golden):
    device = _bar_device(sc, golden("transport"))
    polygons = _fluxoid_polygons(device)
    model = sc.factorize_model(device=device, current_units="uA", terminal_currents={"bar": {"source": 20.0,
                                                                                             "drain": -20.0}})
    free = sc.solve(model=model)[-1]
    assert abs(sum(free.hole_fluxoid("hole", points=polygons["hole"], with_units=False))) > 1e-5
    sol = sc.find_fluxoid_solution(model, fluxoids={"hole": 0.0}, hole_polygon_mapping=polygons)
    assert sol.terminal_currents == {"bar": {"source": 20.0, "drain": -20.0}}
    assert abs(sum(sol.hole_fluxoid("hole", points=polygons["hole"], with_units=False))) <= 1e-6


@pytest.mark.gpu
def test_current_through_path_equals_terminal_current(sc, golden):
    device = _bar_device(sc, golden("transport"))
    model = sc.factorize_model(device=device, current_units="uA")
    currents = [5.0, -12.0, 30.0]
    batch = sc.solve_batch(model=model, applied_fields=[None] * 3,
                           terminal_currents=[{"bar": {"source": I, "drain": -I}} for I in currents])
    path = np.column_stack([np.full(401, -2.0), np.linspace(-1.4999, 1.4999, 401)])  # across the bar, left of the hole
    for I, sols in zip(currents, batch):
        through = sols[0].current_through_path(path, film="bar", units="uA", with_units=False)
        assert abs(abs(through) - abs(I)) <= 0.05 * abs(I), (I, through)


def test_solve_batch_terminal_current_arguments_are_checked_first(golden):
    """Rejected before any device work (no GPU needed): the checks run ahead of the solve."""
    import superscreen_b200 as sc
    from superscreen_b200.solver.solve import _batch_terminal_currents

    device = _bar_device(sc, golden("transport"), with_mesh=False)
    model = type("M", (), {"device": device, "current_units": "uA"})()
    ok = _batch_terminal_currents(model, [{"bar": {"source": "10 uA", "drain": -10.0}}, {}], 2)
    assert ok == [{"bar": {"source": 10.0, "drain": -10.0}}, {}]
    with pytest.raises(ValueError):
        _batch_terminal_currents(model, [{}], 2)
    with pytest.raises(ValueError):
        _batch_terminal_currents(model, [{"bar": {"source": 1.0, "drain": 0.0}}], 1)
    with pytest.raises(KeyError):
        _batch_terminal_currents(model, [{"nofilm": {"source": 1.0}}], 1)
    with pytest.raises(KeyError):
        _batch_terminal_currents(model, [{"bar": {"source": 1.0, "gate": -1.0}}], 1)


# ---------------------------------------------------------------------------------------------
# kernels in isolation
# ---------------------------------------------------------------------------------------------
NSETS = [1, 2, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65, 130]
TARGETS = [1, 63, 65, 746]
SOURCES = [1, 31, 33, 257, 1380]


def _within_film_reference(sites, centroids, areas, J):
    """port.biot_savart_within_film for every set of J [n, nsets, 2] at once (same formula)."""
    dx = sites[:, None, 0] - centroids[None, :, 0]
    dy = sites[:, None, 1] - centroids[None, :, 1]
    pref = areas * (dx * dx + dy * dy) ** (-1.5)
    return ((pref * dy) @ J[:, :, 0] - (pref * dx) @ J[:, :, 1]) / (4 * np.pi)


def _boundary_reference(sites, centers, lengths, normals, stream):
    """port.boundary_effective_field for every column of stream [n, nsets] at once (same formula)."""
    dr = sites[:, None, :] - centers[None, :, :]
    r3 = np.sum(dr * dr, axis=2) ** 1.5
    return (np.sum(dr * -normals[None, :, :], axis=2) / r3 * lengths) @ stream / (4 * np.pi)


def _kernel_inputs(g, m, n, nsets, seed):
    rng = np.random.default_rng(seed)
    sites = g["in_sites"]
    tri = sites[g["in_elements"]]
    centroids = tri.mean(axis=1)
    areas = 0.5 * np.abs(np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0]))
    tgt = sites[rng.choice(len(sites), m, replace=False)]
    pick = rng.choice(len(centroids), n, replace=False)
    return tgt, centroids[pick], areas[pick], rng.standard_normal((n, nsets, 2))


def _within_film(lib, torch, tgt, src, area, J):
    from superscreen_b200 import _lib

    tgt, src, area, J3 = (torch.as_tensor(np.ascontiguousarray(a)).cuda() for a in (tgt, src, area, J))
    nsets = J.shape[1]
    out = torch.full((len(tgt), nsets), np.nan, dtype=torch.float64, device="cuda")
    _lib.check(lib.scb_biot_savart_within_film(len(tgt), _lib.ptr(tgt), len(src), _lib.ptr(src), _lib.ptr(area),
                                               _lib.ptr(J3), 1.0 / (4 * np.pi), nsets, _lib.ptr(out),
                                               _lib.stream_ptr()))
    torch.cuda.synchronize()
    return out


def _boundary(lib, torch, tgt, centers, normals, strength):
    from superscreen_b200 import _lib

    nsets = strength.shape[1]
    tgt, centers, normals, strength = (torch.as_tensor(np.ascontiguousarray(a)).cuda()
                                       for a in (tgt, centers, normals, strength))
    out = torch.full((len(tgt), nsets), np.nan, dtype=torch.float64, device="cuda")
    _lib.check(lib.scb_biot_savart(4, len(tgt), _lib.ptr(tgt), len(centers), _lib.ptr(centers), _lib.ptr(strength),
                                   _lib.ptr(normals), 0.0, 1.0 / (4 * np.pi), nsets, _lib.ptr(out),
                                   _lib.stream_ptr()))
    torch.cuda.synchronize()
    return out


def _cases():
    big = [(m, n) for m in TARGETS for n in SOURCES]
    return [(m, n, s) for s in NSETS for (m, n) in [(746, 1380), (63, 33), (1, 257)]] + \
        [(m, n, s) for (m, n) in big for s in (1, 17, 65)]


@pytest.mark.gpu
def test_within_film_kernel_against_oracle(sc, golden):
    import torch

    from oracle import port
    from superscreen_b200 import _lib

    lib = _lib.lib()
    g = golden("transport")
    tgt, src, area, J = _kernel_inputs(g, 746, 1380, 3, 0)
    ref = _within_film_reference(tgt, src, area, J)
    for s in range(3):  # the vectorised restatement is port.biot_savart_within_film
        assert rel_l2(ref[:, s], port.biot_savart_within_film(tgt, src, area, J[:, s])) <= 1e-13
    for (m, n, nsets) in _cases():
        tgt, src, area, J = _kernel_inputs(g, m, n, nsets, m * 7 + n * 3 + nsets)
        out = _within_film(lib, torch, tgt, src, area, J)
        again = _within_film(lib, torch, tgt, src, area, J)
        assert torch.equal(out, again), (m, n, nsets)
        out = out.cpu().numpy()
        ref = _within_film_reference(tgt, src, area, J)
        errs = [rel_l2(out[:, s], ref[:, s]) for s in range(nsets)]
        assert max(errs) <= 1e-12, (m, n, nsets, max(errs))
    # no sources: zeros; no targets: nothing written
    out = torch.full((5, 20), np.nan, dtype=torch.float64, device="cuda")
    _lib.check(lib.scb_biot_savart_within_film(5, _lib.ptr(out), 0, None, None, None, 1.0, 20, _lib.ptr(out),
                                               _lib.stream_ptr()))
    assert torch.count_nonzero(out).item() == 0
    _lib.check(lib.scb_biot_savart_within_film(0, None, 10, None, None, None, 1.0, 20, None, _lib.stream_ptr()))


@pytest.mark.gpu
def test_multi_set_boundary_field_against_oracle(sc, golden):
    import torch

    from oracle import port
    from superscreen_b200 import _lib

    lib = _lib.lib()
    g = golden("transport")
    rng = np.random.default_rng(1)
    sites = g["in_sites"]
    boundary = sites[g["in_boundary_ordered"]]
    for nsets in NSETS:
        for m in TARGETS:
            for n in (1, 31, 33, len(boundary)):
                centers = 0.5 * (boundary[:n] + np.roll(boundary, -1, axis=0)[:n])
                theta = rng.uniform(0, 2 * np.pi, n)
                normals = np.column_stack([np.cos(theta), np.sin(theta)])
                lengths = rng.uniform(0.05, 0.2, n)
                stream = rng.standard_normal((n, nsets))
                tgt = sites[rng.choice(len(sites), m, replace=False)]
                out = _boundary(lib, torch, tgt, centers, normals, stream * lengths[:, None])
                again = _boundary(lib, torch, tgt, centers, normals, stream * lengths[:, None])
                assert torch.equal(out, again)
                out = out.cpu().numpy()
                ref = _boundary_reference(tgt, centers, lengths, normals, stream)
                if nsets <= 2:
                    for s in range(nsets):
                        assert rel_l2(ref[:, s], port.boundary_effective_field(tgt, centers, lengths, normals,
                                                                               stream[:, s])) <= 1e-13
                errs = [rel_l2(out[:, s], ref[:, s]) for s in range(nsets)]
                assert max(errs) <= 1e-12, (m, n, nsets, max(errs))


def test_new_entry_points_reject_bad_sizes_without_gpu():
    from superscreen_b200 import _lib

    lib = _lib.load_library()
    for args in [(-1, None, 1, None, None, None, 1.0, 1), (1, None, -1, None, None, None, 1.0, 1),
                 (1, None, 1, None, None, None, 1.0, 0)]:
        rc = lib.scb_biot_savart_within_film(*args, None, None)
        assert rc == -1 and b"sizes" in lib.scb_last_error()
    rc = lib.scb_biot_savart(4, 10, None, 10, None, None, None, 0.0, 1.0, 0, None, None)  # nsets = 0
    assert rc == -1 and b"sizes" in lib.scb_last_error()
