"""screening_field_at_position_batch and vector_potential_at_position_batch: the multi-set SCB_BS_VECTOR and
SCB_BS_VECTOR_POTENTIAL pair sums against a float64 direct sum and against one-set calls; the batched vector field
and vector potential of solve_batch solutions against the per-solution methods row by row (bits where only pair sums
ran, tolerances where the in-plane interpolation ran); chunks of targets, groups of entries and host-side validation."""
import copy
import types

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MU0_4PI = 1e-7  # prefactor of the kernel tests
VECTOR, VECPOT = 2, 3  # scb_biot_savart kinds


@pytest.fixture(scope="module")
def sc():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import superscreen_b200 as sc

    return sc


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


def _ring_batch(sc, g, B, seed=0):
    """B solve_batch entries on the ring: fields, circulating currents and 0-2 vortices."""
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
    return [sols[-1] for sols in batch]


def _two_rings_batch(sc, g, B=5, iterations=2):
    model = sc.factorize_model(device=_two_rings_device(sc, g), current_units="uA")
    return sc.solve_batch(model=model, applied_fields=[sc.ConstantField(0.1 * (b + 1)) for b in range(B)],
                          circulating_currents=[{"lower_hole": 10.0 * b} for b in range(B)], iterations=iterations)


def _grid(half, k, z=None):
    # (shifted off the origin and the axes, where the meshes have vertices)
    x, y = np.meshgrid(np.linspace(-half, half, k) + 0.0123, np.linspace(-half, half, k) - 0.0071)
    xy = np.stack([x.ravel(), y.ravel()], axis=1)
    return xy if z is None else np.concatenate([xy, np.full((len(xy), 1), z)], axis=1)


def _screening_rows(sols, positions, **kw):
    return [s.screening_field_at_position(positions, with_units=False, **kw) for s in sols]


def _potential_rows(sols, positions, **kw):
    return [s.vector_potential_at_position(positions, with_units=False, **kw) for s in sols]


def _assert_rows(batch, ref, tol, tag):
    assert batch.shape == (len(ref),) + np.shape(ref[0]), (tag, batch.shape, np.shape(ref[0]))
    for b, r in enumerate(ref):
        if tol == 0:
            assert np.array_equal(batch[b], r, equal_nan=True), (tag, b, np.nanmax(np.abs(batch[b] - r)))
        else:  # (a target on a mesh vertex of a film's plane gives NaN in both)
            assert np.array_equal(np.isnan(batch[b]), np.isnan(r)), (tag, b)
            d = np.abs(batch[b] - r)
            assert np.nanmax(d) <= tol * np.nanmax(np.abs(r)), (tag, b, np.nanmax(d))


# ---------------------------------------------------------------------------------------------
# the multi-set SCB_BS_VECTOR and SCB_BS_VECTOR_POTENTIAL pair sums
# ---------------------------------------------------------------------------------------------
def _bs(kind, tgt, src, area, J):
    import torch

    from superscreen_b200 import _lib

    L = _lib.lib()
    d = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).cuda()
    tgt_d, src_d, area_d, J_d = d(tgt), d(src), d(area), d(J)
    nsets = J.shape[0]
    out = torch.full((nsets, len(tgt), 3 if kind == VECTOR else 2), 7.0, dtype=torch.float64, device="cuda")
    _lib.check(L.scb_biot_savart(kind, len(tgt), _lib.ptr(tgt_d), len(src), _lib.ptr(src_d), _lib.ptr(area_d),
                                 _lib.ptr(J_d), 0.0, MU0_4PI, nsets, _lib.ptr(out), _lib.stream_ptr()))
    return out.cpu().numpy()


def _bs_reference(kind, tgt, src, area, J):
    """(nsets, m, 3) field or (nsets, m, 2) vector potential as a float64 direct sum."""
    dx = tgt[:, None, 0] - src[None, :, 0]
    dy = tgt[:, None, 1] - src[None, :, 1]
    dz = tgt[:, None, 2] - src[None, :, 2]
    r2 = dx * dx + dy * dy + dz * dz
    aJx, aJy = (area[None, :] * J[:, :, 0]).T, (area[None, :] * J[:, :, 1]).T  # (n, nsets)
    if kind == VECPOT:
        k1 = r2 ** -0.5
        return MU0_4PI * np.stack([(k1 @ aJx).T, (k1 @ aJy).T], axis=-1)
    k3 = r2 ** -1.5
    bx = (k3 * dz) @ aJy
    by = -((k3 * dz) @ aJx)
    bz = (k3 * dy) @ aJx - (k3 * dx) @ aJy
    return MU0_4PI * np.stack([bx.T, by.T, bz.T], axis=-1)


def _points(rng, k, z):
    return np.concatenate([rng.uniform(-3, 3, (k, 2)), z + rng.uniform(-0.2, 0.2, (k, 1))], axis=1)


# every pass width and remainder, the tile edges of m and n (n < 512: one source range; n >= 512: split sources and
# the reduction pass), and 10^5 sources split over many CTAs
CASES = [(1, 255, 256), (2, 256, 257), (3, 257, 255), (4, 512, 512), (5, 511, 513), (7, 1, 1), (8, 1000, 3000),
         (9, 5, 100000), (17, 63, 1), (130, 1000, 3000)]


@pytest.mark.parametrize("kind", [VECTOR, VECPOT], ids=["vector", "vector_potential"])
@pytest.mark.parametrize("nsets,m,n", CASES)
def test_multi_set_kernel(sc, kind, nsets, m, n):
    rng = np.random.default_rng(nsets * 1000 + m + n + kind)
    tgt, src = _points(rng, m, 1.0), _points(rng, n, 0.0)
    area, J = rng.uniform(0.5, 1.5, n), rng.standard_normal((nsets, n, 2))
    out = _bs(kind, tgt, src, area, J)
    ref = _bs_reference(kind, tgt, src, area, J)
    assert np.abs(out - ref).max() <= 1e-12 * np.abs(ref).max()
    for s in range(nsets):  # every set carries the bits of a one-set call
        assert np.array_equal(out[s], _bs(kind, tgt, src, area, J[s:s + 1])[0]), s
    assert np.array_equal(out, _bs(kind, tgt, src, area, J))  # and the same bits again


@pytest.mark.parametrize("kind", [VECTOR, VECPOT], ids=["vector", "vector_potential"])
def test_multi_set_kernel_empty(sc, kind):
    rng = np.random.default_rng(3)
    c = 3 if kind == VECTOR else 2
    out = _bs(kind, _points(rng, 65, 1.0), np.zeros((0, 3)), np.zeros(0), np.zeros((9, 0, 2)))
    assert out.shape == (9, 65, c) and not out.any()
    out = _bs(kind, np.zeros((0, 3)), _points(rng, 20, 0.0), np.ones(20), np.ones((9, 20, 2)))
    assert out.shape == (9, 0, c)


# ---------------------------------------------------------------------------------------------
# the batches against the per-solution methods
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 3, 8, 13, 64, 130])
def test_batch_rows_equal_per_solution_calls(sc, golden, B):
    sols = _ring_batch(sc, golden("ring"), B, seed=B)
    positions = _grid(5.0, 23)
    out = sc.screening_field_at_position_batch(sols, positions, zs=1.5, vector=True, with_units=False)
    _assert_rows(out, _screening_rows(sols, positions, zs=1.5, vector=True), 0, ("vector", B))
    out = sc.vector_potential_at_position_batch(sols, positions, zs=1.5, with_units=False)
    _assert_rows(out, _potential_rows(sols, positions, zs=1.5), 0, ("potential", B))
    if B == 13:
        out = sc.screening_field_at_position_batch(sols, positions, zs=1.5, with_units=False)
        _assert_rows(out, _screening_rows(sols, positions, zs=1.5), 0, "Bz")
        for fn, kw, per in ((sc.screening_field_at_position_batch, dict(vector=True), "screening_field_at_position"),
                            (sc.vector_potential_at_position_batch, {}, "vector_potential_at_position")):
            parts = fn(sols, positions, zs=1.5, with_units=False, return_sum=False, **kw)
            ref = [getattr(s, per)(positions, zs=1.5, with_units=False, return_sum=False, **kw) for s in sols]
            assert list(parts) == list(ref[0]) == ["ring"]
            _assert_rows(parts["ring"], [r["ring"] for r in ref], 0, per)


def test_units_and_three_column_positions(sc, golden):
    sols = _ring_batch(sc, golden("ring"), 9)
    positions = _grid(5.0, 17, z=-0.75)
    out = sc.screening_field_at_position_batch(sols, positions, vector=True, units="uT")
    assert str(out.units) == str(sols[0].screening_field_at_position(positions, vector=True, units="uT").units)
    _assert_rows(out.magnitude, _screening_rows(sols, positions, vector=True, units="uT"), 0, "uT")
    parts = sc.screening_field_at_position_batch(sols, positions, vector=True, units="A/m", return_sum=False)
    ref = [s.screening_field_at_position(positions, vector=True, units="A/m", return_sum=False) for s in sols]
    assert str(parts["ring"].units) == str(ref[0]["ring"].units)
    _assert_rows(parts["ring"].magnitude, [r["ring"].magnitude for r in ref], 0, "A/m")
    for units in (None, "uT * um", "mT * mm"):
        out = sc.vector_potential_at_position_batch(sols, positions, units=units)
        ref = [s.vector_potential_at_position(positions, units=units) for s in sols]
        assert str(out.units) == str(ref[0].units), units
        _assert_rows(out.magnitude, [r.magnitude for r in ref], 0, units)
        assert not out.magnitude[..., 2].any()


def test_two_films_two_layers_and_iterates(sc, golden):
    B = 5
    batch = _two_rings_batch(sc, golden("two_rings"), B)
    positions = _grid(6.0, 19)
    for sols in ([s[-1] for s in batch], [batch[b][b % 3] for b in range(B)]):  # last iterates; mixed iterates
        for zs in (0.5, 2.0):
            out = sc.screening_field_at_position_batch(sols, positions, zs=zs, vector=True, with_units=False)
            _assert_rows(out, _screening_rows(sols, positions, zs=zs, vector=True), 0, ("vector", zs))
            out = sc.vector_potential_at_position_batch(sols, positions, zs=zs, with_units=False)
            _assert_rows(out, _potential_rows(sols, positions, zs=zs), 0, ("potential", zs))
        parts = sc.vector_potential_at_position_batch(sols, positions, zs=2.0, with_units=False, return_sum=False)
        ref = [s.vector_potential_at_position(positions, zs=2.0, with_units=False, return_sum=False) for s in sols]
        assert list(parts) == list(ref[0]) == ["lower", "upper"]
        for key in parts:
            _assert_rows(parts[key], [r[key] for r in ref], 0, key)


@pytest.mark.parametrize("case", ["ring", "two_rings"])
def test_evaluation_plane_at_a_layer(sc, golden, case):
    """The screening field: points inside a film in its plane are interpolated, the rest are pair sums.  The vector
    potential is a pair sum everywhere."""
    if case == "ring":
        sols, z = _ring_batch(sc, golden("ring"), 6), float(golden("ring")["in_z0"])
    else:
        g = golden("two_rings")
        model = sc.factorize_model(device=_two_rings_device(sc, g), current_units="uA")
        batch = sc.solve_batch(model=model, applied_fields=[sc.ConstantField(0.2), None, sc.ConstantField(-0.1)],
                               circulating_currents=[{}, {"upper_hole": 5.0}, {"lower_hole": 3.0}], iterations=2)
        sols, z = [s[-1] for s in batch], float(g["in_lower_z0"])
    positions = _grid(6.0, 31)
    for vector in (True, False):
        out = sc.screening_field_at_position_batch(sols, positions, zs=z, vector=vector, with_units=False)
        _assert_rows(out, _screening_rows(sols, positions, zs=z, vector=vector), 1e-14, (case, vector))
        parts = sc.screening_field_at_position_batch(sols, positions, zs=z, vector=vector, with_units=False,
                                                     return_sum=False)
        ref = [s.screening_field_at_position(positions, zs=z, vector=vector, with_units=False, return_sum=False)
               for s in sols]
        for key in parts:
            _assert_rows(parts[key], [r[key] for r in ref], 1e-14, (key, vector))
    out = sc.vector_potential_at_position_batch(sols, positions, zs=z, with_units=False)
    _assert_rows(out, _potential_rows(sols, positions, zs=z), 0, (case, "potential"))
    with pytest.raises(NotImplementedError):
        sc.screening_field_at_position_batch(sols, positions, zs=z, vector=True, interp_method="cubic")
    sc.screening_field_at_position_batch(sols, positions, zs=z + 0.25, vector=True, interp_method="cubic")


def test_vector_potential_inside_a_film_raises_before_any_device_work(sc, golden):
    from superscreen_b200 import _lib

    g = golden("ring")
    sols, z = _ring_batch(sc, g, 4), float(g["in_z0"])
    film = sols[0].device.films["ring"]
    rng = np.random.default_rng(5)
    cand = np.column_stack([rng.uniform(-4, 4, 4000), rng.uniform(-4, 4, 4000)])
    inside = cand[film.contains_points(cand)][:40]
    assert len(inside) == 40
    with pytest.raises(ValueError, match="inside the film") as per_solution:
        sols[0].vector_potential_at_position(inside, zs=z)
    before = _lib.launch_count()
    with pytest.raises(ValueError, match="inside the film") as batch:
        sc.vector_potential_at_position_batch(sols, inside, zs=z)
    assert _lib.launch_count() == before
    assert str(batch.value) == str(per_solution.value)
    # one point outside the film (or off the plane): the pair sum runs, as in the per-solution method
    mixed = np.concatenate([inside, [[40.0123, -0.0071]]])
    _assert_rows(sc.vector_potential_at_position_batch(sols, mixed, zs=z, with_units=False),
                 _potential_rows(sols, mixed, zs=z), 0, "mixed")
    _assert_rows(sc.vector_potential_at_position_batch(sols, inside, zs=z + 0.5, with_units=False),
                 _potential_rows(sols, inside, zs=z + 0.5), 0, "off plane")


def test_chunk_boundaries(sc, golden, monkeypatch):
    from superscreen_b200 import solution

    sols = _ring_batch(sc, golden("ring"), 11)
    monkeypatch.setattr(solution, "_EVAL_CHUNK", 97)
    positions = _grid(5.0, 25)  # 625 points: 6 full chunks and a partial one
    out = sc.screening_field_at_position_batch(sols, positions, zs=1.0, vector=True, with_units=False)
    _assert_rows(out, _screening_rows(sols, positions, zs=1.0, vector=True), 0, "off-plane")
    z = float(golden("ring")["in_z0"])  # in plane: the chunks run over the points outside the film
    out = sc.screening_field_at_position_batch(sols, positions, zs=z, vector=True, with_units=False)
    _assert_rows(out, _screening_rows(sols, positions, zs=z, vector=True), 1e-14, "in-plane")
    out = sc.vector_potential_at_position_batch(sols, positions, zs=1.0, with_units=False)  # (one launch)
    _assert_rows(out, _potential_rows(sols, positions, zs=1.0), 0, "potential")


def test_entries_in_several_device_groups(sc, golden, monkeypatch):
    """A device result smaller than the batch: the entries run in groups, with the same bits."""
    from superscreen_b200 import solution

    B = 11
    batch = _two_rings_batch(sc, golden("two_rings"), B, iterations=1)
    sols = [s[-1] for s in batch]
    positions = _grid(6.0, 21)
    monkeypatch.setattr(solution, "_BATCH_RESULT_ELEMS", 4 * len(positions) * 3)  # groups of 4, 4, 3 entries
    out = sc.screening_field_at_position_batch(sols, positions, zs=1.25, vector=True, with_units=False)
    _assert_rows(out, _screening_rows(sols, positions, zs=1.25, vector=True), 0, "vector")
    parts = sc.vector_potential_at_position_batch(sols, positions, zs=1.25, with_units=False, return_sum=False)
    for key in ("lower", "upper"):
        _assert_rows(parts[key], [s.vector_potential_at_position(positions, zs=1.25, with_units=False,
                                                                 return_sum=False)[key] for s in sols], 0, key)
    monkeypatch.setattr(solution, "_BATCH_RESULT_ELEMS", 3 * len(positions))  # Bz in groups of 3, 3, 3, 2 entries
    out = sc.field_at_position_batch(sols, positions, zs=1.25, with_units=False)
    _assert_rows(out, [s.field_at_position(positions, zs=1.25, with_units=False) for s in sols], 0, "Bz")
    parts = sc.field_at_position_batch(sols, positions, zs=1.25, with_units=False, return_sum=False)
    ref = [s.field_at_position(positions, zs=1.25, with_units=False, return_sum=False) for s in sols]
    for key in parts:
        _assert_rows(parts[key], [np.broadcast_to(r[key], parts[key][0].shape) for r in ref], 0, key)


def test_bz_column_agrees_with_the_scalar_kind(sc, golden):
    sols = _ring_batch(sc, golden("ring"), 8)
    positions = _grid(5.0, 19)
    vec = sc.screening_field_at_position_batch(sols, positions, zs=0.8, vector=True, with_units=False)
    bz = sc.screening_field_at_position_batch(sols, positions, zs=0.8, with_units=False)
    assert np.abs(vec[..., 2] - bz).max() <= 1e-13 * np.abs(bz).max()
    assert np.abs(vec[..., :2]).max() > 0


def test_empty_batch_and_positions(sc, golden):
    sols = _ring_batch(sc, golden("ring"), 3)
    assert sc.screening_field_at_position_batch([], _grid(1.0, 4), zs=1.0, vector=True).shape == (0, 16, 3)
    assert sc.screening_field_at_position_batch([], _grid(1.0, 4), zs=1.0).shape == (0, 16)
    assert sc.vector_potential_at_position_batch([], _grid(1.0, 4), zs=1.0).shape == (0, 16, 3)
    empty = np.zeros((0, 2))
    assert sc.screening_field_at_position_batch(sols, empty, zs=1.0, vector=True, with_units=False).shape == (3, 0, 3)
    # (no position lies outside the film: the per-solution method raises for every plane)
    with pytest.raises(ValueError, match="inside the film"):
        sols[0].vector_potential_at_position(empty, zs=1.0)
    with pytest.raises(ValueError, match="inside the film"):
        sc.vector_potential_at_position_batch(sols, empty, zs=1.0)


# ---------------------------------------------------------------------------------------------
# validation
# ---------------------------------------------------------------------------------------------
def _bad_batches(sc, golden):
    sols = _ring_batch(sc, golden("ring"), 3)
    two = _two_rings_device(sc, golden("two_rings"))
    other = sc.solve(device=two, applied_field=sc.ConstantField(0.1))[-1]

    def variant(**attrs):
        s = copy.copy(sols[1])
        s.device = s.device.copy()
        for key, value in attrs.items():
            if key == "mesh":
                s.device.meshes = dict(s.device.meshes)
                s.device.meshes["ring"] = value
            elif key == "z0":
                s.device.layers["layer"].z0 = value
            elif key == "length_units":
                s.device._length_units = value
            else:
                setattr(s, key, value)
        return s

    mesh = sols[0].device.meshes["ring"]
    return sols, [
        ([sols[0], "nope"], TypeError, r"solutions\[1\]"),
        ([sols[0], sols[1], other], ValueError, r"solutions\[2\]"),
        ([sols[0], variant(mesh=types.SimpleNamespace(sites=mesh.sites + 1e-3, elements=mesh.elements))],
         ValueError, r"solutions\[1\]"),
        ([sols[0], variant(z0=0.75)], ValueError, r"solutions\[1\]"),
        ([sols[0], variant(length_units="nm")], ValueError, r"solutions\[1\]"),
        ([sols[0], sols[2], variant(_field_units="uT")], ValueError, r"solutions\[2\]"),
        ([sols[0], variant(_current_units="mA")], ValueError, r"solutions\[1\]"),
        ([sols[0], variant(film_solutions={})], ValueError, r"solutions\[1\]"),
    ]


def test_bad_batches_raise_before_any_device_work(sc, golden):
    from superscreen_b200 import _lib

    sols, cases = _bad_batches(sc, golden)
    positions = _grid(5.0, 9)
    calls = [lambda batch: sc.screening_field_at_position_batch(batch, positions, zs=1.0, vector=True),
             lambda batch: sc.screening_field_at_position_batch(batch, positions, zs=1.0),
             lambda batch: sc.vector_potential_at_position_batch(batch, positions, zs=1.0)]
    for call in calls:
        for batch, exc, match in cases:
            before = _lib.launch_count()
            with pytest.raises(exc, match=match):
                call(batch)
            assert _lib.launch_count() == before, match
