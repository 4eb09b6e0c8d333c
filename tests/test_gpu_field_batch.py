"""field_at_position_batch: the multi-set SCB_BS_Z pair sum against a float64 direct sum and against one-set
calls; the batched field of solve_batch solutions against Solution.field_at_position row by row (bits where only
pair sums ran, tolerances where the in-plane interpolation ran); chunking, applied-field functions, iterates and
host-side validation."""
import copy
import types

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MU0_4PI = 1e-7  # prefactor of the kernel tests


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


def _grid(half, k, z=None):
    # (shifted off the origin and the axes, where the meshes have vertices)
    x, y = np.meshgrid(np.linspace(-half, half, k) + 0.0123, np.linspace(-half, half, k) - 0.0071)
    xy = np.stack([x.ravel(), y.ravel()], axis=1)
    return xy if z is None else np.concatenate([xy, np.full((len(xy), 1), z)], axis=1)


def _rows(sols, positions, **kw):
    return [s.field_at_position(positions, with_units=False, **kw) for s in sols]


def _assert_rows(batch, ref, tol, tag):
    assert batch.shape == (len(ref), len(ref[0]) if np.ndim(ref[0]) else 1), tag
    for b, r in enumerate(ref):
        r = np.broadcast_to(r, batch[b].shape)
        if tol == 0:
            assert np.array_equal(batch[b], r, equal_nan=True), (tag, b, np.nanmax(np.abs(batch[b] - r)))
        else:  # (a target on a mesh vertex of a film's plane gives NaN in both)
            assert np.array_equal(np.isnan(batch[b]), np.isnan(r)), (tag, b)
            d = np.abs(batch[b] - r)
            assert np.nanmax(d) <= tol * np.nanmax(np.abs(r)), (tag, b, np.nanmax(d))


# ---------------------------------------------------------------------------------------------
# the multi-set SCB_BS_Z pair sum
# ---------------------------------------------------------------------------------------------
def _bs_z(sc, tgt, src, area, J):
    import torch

    from superscreen_b200 import _lib

    L = _lib.lib()
    d = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).cuda()
    tgt_d, src_d, area_d, J_d = d(tgt), d(src), d(area), d(J)
    nsets = J.shape[0]
    out = torch.full((nsets, len(tgt)), 7.0, dtype=torch.float64, device="cuda")
    _lib.check(L.scb_biot_savart(1, len(tgt), _lib.ptr(tgt_d), len(src), _lib.ptr(src_d), _lib.ptr(area_d),
                                 _lib.ptr(J_d), 0.0, MU0_4PI, nsets, _lib.ptr(out), _lib.stream_ptr()))
    return out.cpu().numpy()


def _bs_z_reference(tgt, src, area, J):
    dx = tgt[:, None, 0] - src[None, :, 0]
    dy = tgt[:, None, 1] - src[None, :, 1]
    dz = tgt[:, None, 2] - src[None, :, 2]
    k3 = (dx * dx + dy * dy + dz * dz) ** -1.5
    aJ = area[None, :, None] * J                               # (nsets, n, 2)
    return MU0_4PI * ((k3 * dy) @ aJ[:, :, 0].T - (k3 * dx) @ aJ[:, :, 1].T).T


def _points(rng, k, z):
    return np.concatenate([rng.uniform(-3, 3, (k, 2)), z + rng.uniform(-0.2, 0.2, (k, 1))], axis=1)


# every nsets, m and n of the pass and tile edges; the last case splits 10^5 sources over many CTAs
@pytest.mark.parametrize("nsets,m,n", [(1, 1, 1), (2, 63, 15), (3, 64, 16), (7, 65, 17), (8, 1000, 3000),
                                       (9, 1, 3000), (17, 63, 1), (63, 64, 15), (64, 65, 16), (65, 1000, 17),
                                       (130, 1000, 3000), (9, 5, 100000)])
def test_multi_set_z_kernel(sc, nsets, m, n):
    rng = np.random.default_rng(nsets * 1000 + m + n)
    tgt, src = _points(rng, m, 1.0), _points(rng, n, 0.0)
    area, J = rng.uniform(0.5, 1.5, n), rng.standard_normal((nsets, n, 2))
    out = _bs_z(sc, tgt, src, area, J)
    ref = _bs_z_reference(tgt, src, area, J)
    assert np.abs(out - ref).max() <= 1e-12 * np.abs(ref).max()
    for s in range(nsets):  # every set carries the bits of a one-set call
        assert np.array_equal(out[s], _bs_z(sc, tgt, src, area, J[s:s + 1])[0]), s
    assert np.array_equal(out, _bs_z(sc, tgt, src, area, J))


def test_multi_set_z_kernel_empty(sc):
    rng = np.random.default_rng(3)
    tgt = _points(rng, 65, 1.0)
    out = _bs_z(sc, tgt, np.zeros((0, 3)), np.zeros(0), np.zeros((9, 0, 2)))
    assert out.shape == (9, 65) and not out.any()
    out = _bs_z(sc, np.zeros((0, 3)), _points(rng, 20, 0.0), np.ones(20), np.ones((9, 20, 2)))
    assert out.shape == (9, 0)


# ---------------------------------------------------------------------------------------------
# field_at_position_batch against field_at_position
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 3, 8, 13, 64, 130])
def test_batch_rows_equal_per_solution_calls(sc, golden, B):
    sols = _ring_batch(sc, golden("ring"), B, seed=B)
    positions = _grid(5.0, 23)
    out = sc.field_at_position_batch(sols, positions, zs=1.5, with_units=False)
    _assert_rows(out, _rows(sols, positions, zs=1.5), 0, B)
    if B == 13:
        parts = sc.field_at_position_batch(sols, positions, zs=1.5, with_units=False, return_sum=False)
        ref = [s.field_at_position(positions, zs=1.5, with_units=False, return_sum=False) for s in sols]
        assert list(parts) == list(ref[0]) == ["ring", "applied_field"]
        for key in parts:
            _assert_rows(parts[key], [r[key] for r in ref], 0, key)


def test_units_and_three_column_positions(sc, golden):
    sols = _ring_batch(sc, golden("ring"), 9)
    positions = _grid(5.0, 17, z=-0.75)
    out = sc.field_at_position_batch(sols, positions, units="uT")
    assert str(out.units) == str(sols[0].field_at_position(positions, units="uT").units)
    _assert_rows(out.magnitude, _rows(sols, positions, units="uT"), 0, "uT")
    parts = sc.field_at_position_batch(sols, positions, units="A/m", return_sum=False)
    for key, value in parts.items():
        ref = [s.field_at_position(positions, units="A/m", return_sum=False)[key] for s in sols]
        assert str(value.units) == str(ref[0].units)
        _assert_rows(value.magnitude, [np.asarray(getattr(r, "magnitude", r)) for r in ref], 0, key)


def test_two_films_two_layers_and_iterates(sc, golden):
    g = golden("two_rings")
    model = sc.factorize_model(device=_two_rings_device(sc, g), current_units="uA")
    B = 5
    batch = sc.solve_batch(model=model, applied_fields=[sc.ConstantField(0.1 * (b + 1)) for b in range(B)],
                           circulating_currents=[{"lower_hole": 10.0 * b} for b in range(B)], iterations=2)
    positions = _grid(6.0, 19)
    for sols in ([s[-1] for s in batch], [batch[b][b % 3] for b in range(B)]):  # last iterates; mixed iterates
        for zs in (0.5, 2.0):
            out = sc.field_at_position_batch(sols, positions, zs=zs, with_units=False)
            _assert_rows(out, _rows(sols, positions, zs=zs), 0, zs)


@pytest.mark.parametrize("case", ["ring", "two_rings"])
def test_evaluation_plane_at_a_layer(sc, golden, case):
    """Points inside a film in its plane are interpolated, the rest are pair sums."""
    if case == "ring":
        sols, z = _ring_batch(sc, golden("ring"), 6), float(golden("ring")["in_z0"])
    else:
        g = golden("two_rings")
        model = sc.factorize_model(device=_two_rings_device(sc, g), current_units="uA")
        batch = sc.solve_batch(model=model, applied_fields=[sc.ConstantField(0.2), None, sc.ConstantField(-0.1)],
                               circulating_currents=[{}, {"upper_hole": 5.0}, {"lower_hole": 3.0}], iterations=2)
        sols, z = [s[-1] for s in batch], float(g["in_lower_z0"])
    positions = _grid(6.0, 31)
    out = sc.field_at_position_batch(sols, positions, zs=z, with_units=False)
    _assert_rows(out, _rows(sols, positions, zs=z), 1e-14, case)
    parts = sc.field_at_position_batch(sols, positions, zs=z, with_units=False, return_sum=False)
    ref = [s.field_at_position(positions, zs=z, with_units=False, return_sum=False) for s in sols]
    for key in parts:
        _assert_rows(parts[key], [r[key] for r in ref], 1e-14, key)
    with pytest.raises(NotImplementedError):
        sols[0].field_at_position(positions, zs=z, interp_method="cubic")
    with pytest.raises(NotImplementedError):
        sc.field_at_position_batch(sols, positions, zs=z, interp_method="cubic")
    sc.field_at_position_batch(sols, positions, zs=z + 0.25, interp_method="cubic")  # (off-plane: no interpolation)


def test_chunk_boundaries(sc, golden, monkeypatch):
    from superscreen_b200 import solution

    sols = _ring_batch(sc, golden("ring"), 11)
    monkeypatch.setattr(solution, "_EVAL_CHUNK", 97)
    positions = _grid(5.0, 25)  # 625 points: 6 full chunks and a partial one
    out = sc.field_at_position_batch(sols, positions, zs=1.0, with_units=False)
    _assert_rows(out, _rows(sols, positions, zs=1.0), 0, "off-plane")
    z = float(golden("ring")["in_z0"])  # in plane: the chunks run over the points outside the film
    out = sc.field_at_position_batch(sols, positions, zs=z, with_units=False)
    _assert_rows(out, _rows(sols, positions, zs=z), 1e-14, "in-plane")


class _Counting:
    def __init__(self, sc, value):
        self.field, self.calls = sc.ConstantField(value), 0

    def __call__(self, x, y, z):
        self.calls += 1
        return self.field(x, y, z)


def test_applied_field_functions_evaluated_once_each(sc, golden):
    model = sc.factorize_model(device=_ring_device(sc, golden("ring")), current_units="uA")
    f, h = _Counting(sc, 0.3), _Counting(sc, -0.2)
    sols = [s[-1] for s in sc.solve_batch(model=model, applied_fields=[f, h, f, None, None, h, f])]
    f.calls = h.calls = 0
    positions = _grid(5.0, 15)
    out = sc.field_at_position_batch(sols, positions, zs=1.2, with_units=False)
    assert f.calls == 1 and h.calls == 1
    _assert_rows(out, _rows(sols, positions, zs=1.2), 0, "mixed functions")


def test_empty_batch_and_positions(sc, golden):
    sols = _ring_batch(sc, golden("ring"), 3)
    assert sc.field_at_position_batch([], _grid(1.0, 4), zs=1.0).shape == (0, 16)
    out = sc.field_at_position_batch(sols, np.zeros((0, 2)), zs=1.0, with_units=False)
    assert out.shape == (3, 0)


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
        ([sols[0], sols[2], variant(_field_units="uT")], ValueError, r"solutions\[2\]"),
        ([sols[0], variant(_current_units="mA")], ValueError, r"solutions\[1\]"),
        ([sols[0], variant(film_solutions={})], ValueError, r"solutions\[1\]"),
    ]


def test_bad_batches_raise_before_any_device_work(sc, golden):
    from superscreen_b200 import _lib

    sols, cases = _bad_batches(sc, golden)
    positions = _grid(5.0, 9)
    # an equal copy of the mesh arrays is accepted
    mesh = sols[0].device.meshes["ring"]
    same = copy.copy(sols[1])
    same.device = same.device.copy()
    same.device.meshes = {"ring": types.SimpleNamespace(sites=mesh.sites.copy(), elements=mesh.elements.copy(),
                                                        vertex_areas=mesh.vertex_areas)}
    _assert_rows(sc.field_at_position_batch([sols[0], same], positions, zs=1.0, with_units=False),
                 _rows(sols[:2], positions, zs=1.0), 0, "equal mesh")
    for batch, exc, match in cases:
        before = _lib.launch_count()
        with pytest.raises(exc, match=match):
            sc.field_at_position_batch(batch, positions, zs=1.0)
        assert _lib.launch_count() == before, match
