"""Per-entry layer translations in batched solves: the translated film-to-film coupling kernel
(scb_film_coupling_translated) bit for bit against one-set scb_film_coupling calls on moved inputs;
solve_batch(translations=...) against the CPU oracle and serial solves on devices moved in the test; a
scanning-SQUID touchdown and scan; batch semantics (unmoved batches, mixing, permutation, shared devices, HDF5);
host-side validation."""
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


def _moved_polygon(sc, polygon, shift):
    """``polygon`` moved by ``shift`` = (dx, dy), rebuilt here from its rings."""
    from superscreen_b200.device import CompositePolygon

    if isinstance(polygon, CompositePolygon):
        return CompositePolygon(polygon.name, layer=polygon.layer, add=[r + shift for r in polygon.rings],
                                sub=[r + shift for r in polygon.cut_rings])
    return sc.Polygon(polygon.name, layer=polygon.layer, points=polygon.points + shift)


def _moved_device(sc, device, moves):
    """The device with the layers in ``moves`` ({layer: (dx, dy, dz)}) moved, built from scratch: polygons
    from shifted points, meshes from ``sites + (dx, dy)``, layers at ``z0 + dz``."""
    def shift_of(layer):
        dx, dy, _ = moves.get(layer, (0.0, 0.0, 0.0))
        return np.array([dx, dy], dtype=float)

    layers = [sc.Layer(l.name, Lambda=l.Lambda, z0=l.z0 + moves.get(l.name, (0.0, 0.0, 0.0))[2])
              for l in device.layers.values()]
    films = [_moved_polygon(sc, f, shift_of(f.layer)) for f in device.films.values()]
    holes = [_moved_polygon(sc, h, shift_of(h.layer)) for h in device.holes.values()]
    out = sc.Device(device.name, layers=layers, films=films, holes=holes, length_units=device.length_units)
    out.set_meshes({name: (np.asarray(device.meshes[name].sites) + shift_of(f.layer),
                           np.asarray(device.meshes[name].elements)) for name, f in device.films.items()})
    return out


def _full(moves):
    return {k: tuple(float(x) for x in v) + (0.0,) * (3 - len(v)) for k, v in (moves or {}).items()}


def _errs(fs, ref):
    return dict(stream=rel_l2(fs.stream, ref.stream), J=rel_l2(fs.current_density, ref.current_density),
                self_field=rel_l2(fs.self_field, ref.self_field), total=rel_l2(fs.total_field, ref.total_field))


# ---------------------------------------------------------------------------------------------
# the kernel: every set bit-identical to a one-set scb_film_coupling call on moved inputs
# ---------------------------------------------------------------------------------------------
def _packed(rng, sizes, pad_after):
    """Random packed sources: films of ``sizes`` back to back, ``pad_after[k]`` padding rows after film k."""
    rows, film, spans = [], [], []
    o = 0
    for k, (n, pad) in enumerate(zip(sizes, pad_after)):
        xy = rng.uniform(-3.0, 3.0, size=(n, 2))
        rows.append(np.column_stack([xy, np.full(n, rng.uniform(-1.0, 1.0))]))
        film += [k] * n
        spans.append((o, o + n))
        o += n
        if pad:
            rows.append(np.full((pad, 3), 1e30))
            film += [-1] * pad
            o += pad
    src = np.concatenate(rows)
    film = np.array(film, dtype=np.int32)
    area = np.where(film >= 0, rng.uniform(0.01, 0.1, size=len(film)), 0.0)
    return src, area, film, spans


def _shift_table(rng, nsets, nfilms):
    kinds = [lambda: (0.0, 0.0, 0.0), lambda: tuple(-rng.uniform(0.1, 2.0, 3)),
             lambda: tuple(rng.choice([-1e3, 1e3], 3) * rng.uniform(0.5, 1.0, 3)),
             lambda: (0.0, 0.0, rng.uniform(-0.5, 0.5)), lambda: (rng.uniform(-2.0, 2.0), 0.0, 0.0),
             lambda: tuple(rng.uniform(-1.0, 1.0, 3))]
    return np.array([[kinds[rng.integers(len(kinds))]() for _ in range(nfilms)] for _ in range(nsets)])


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["skip_start_split", "skip_middle_split", "skip_end_unsplit", "large_m_unsplit"])
def test_translated_coupling_is_bit_identical_to_one_set_calls(sc, case):
    import torch

    from superscreen_b200 import _lib

    L = _lib.lib()
    rng = np.random.default_rng(["skip_start_split", "skip_middle_split", "skip_end_unsplit", "large_m_unsplit"].index(case))
    layouts = {  # (film sizes, padding after each film, target film, number of targets)
        "skip_start_split": ([700, 1, 333, 1200], [0, 0, 0, 7], 0, 500),
        "skip_middle_split": ([400, 1, 900, 250, 77], [0, 16, 0, 0, 3], 2, 2000),
        "skip_end_unsplit": ([120, 1, 200, 60], [5, 0, 0, 0], 3, 3000),
        "large_m_unsplit": ([300, 1, 250], [0, 0, 9], 1, 1 << 19),
    }
    sizes, pads, dst, m = layouts[case]
    src, area, film, spans = _packed(rng, sizes, pads)
    n, nfilms = len(src), len(sizes)
    lo, hi = spans[dst]
    tgt = rng.uniform(-3.5, 3.5, size=(m, 2))
    tgt_z = float(rng.uniform(-1.0, 1.0))
    S = _shift_table(rng, 17, nfilms)
    J = rng.standard_normal((n, 17, 2))
    pf = 1.0 / (4.0 * np.pi)
    dev = torch.device("cuda:0")
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    d_tgt, d_src, d_area, d_film = t(tgt), t(src), t(area), t(film)

    # references: set r as a one-set call on the moved targets / sources and J column r
    ref = []
    for r in range(17):
        # (the inputs are kept referenced until the call has run)
        m_tgt = t(tgt + S[r, dst, :2])
        m_src = t(src + np.where(film[:, None] >= 0, S[r][np.maximum(film, 0)], 0.0))
        J_r = t(J[:, r:r + 1])
        out = torch.empty(m, dtype=torch.float64, device=dev)
        _lib.check(L.scb_film_coupling(m, _lib.ptr(m_tgt), tgt_z + S[r, dst, 2], n, _lib.ptr(m_src),
                                       _lib.ptr(d_area), _lib.ptr(J_r), lo, hi, pf, 1, _lib.ptr(out),
                                       _lib.stream_ptr()))
        ref.append(out.cpu().numpy())
    for nsets in range(1, 18):
        out = torch.empty((m, nsets), dtype=torch.float64, device=dev)
        d_S, d_J = t(S[:nsets]), t(J[:, :nsets])
        _lib.check(L.scb_film_coupling_translated(m, _lib.ptr(d_tgt), tgt_z, n, _lib.ptr(d_src), _lib.ptr(d_area),
                                                  _lib.ptr(d_J), lo, hi, pf, nsets, dst, _lib.ptr(d_film), nfilms,
                                                  _lib.ptr(d_S), _lib.ptr(out), _lib.stream_ptr()))
        got = out.cpu().numpy()
        for r in range(nsets):
            assert np.array_equal(got[:, r], ref[r]), (case, nsets, r)
    assert all(np.abs(x).max() > 0 for x in ref)


def test_translated_coupling_rejects_bad_sizes_without_gpu():
    from superscreen_b200 import _lib

    lib = _lib.load_library()

    def call(m=1, n=4, lo=0, hi=1, nsets=1, dst=0, nfilms=2):
        return lib.scb_film_coupling_translated(m, None, 0.0, n, None, None, None, lo, hi, 1.0, nsets, dst, None,
                                                nfilms, None, None, None)

    for kwargs, word in [(dict(m=-1), b"sizes"), (dict(n=-1), b"sizes"), (dict(nsets=0), b"sizes"),
                         (dict(lo=2, hi=1), b"skip"), (dict(hi=5), b"skip"), (dict(dst=2), b"dst"),
                         (dict(dst=-1), b"dst"), (dict(nfilms=0, dst=0), b"dst")]:
        assert call(**kwargs) == -1 and word in lib.scb_last_error(), kwargs
    assert call(m=0) == 0


# ---------------------------------------------------------------------------------------------
# solve_batch(translations=...) against the CPU oracle and against serial solves
# ---------------------------------------------------------------------------------------------
_TWO_RING_MOVES = [{"up": (0.0, 0.0)}, {"up": (0.3, -0.2)}, {"up": (0.0, 0.0, 0.4)}, {"up": (-0.25, 0.15, -0.3)}]


def _two_ring_fields(sc):
    dipole = sc.DipoleField(dipole_positions=[(0.4, -0.3, 2.5)], dipole_moments=[(0.0, 0.0, 1e9)], component="z")
    return [sc.ConstantField(0.2), dipole, None, dipole]


@pytest.mark.gpu
def test_two_rings_translated_against_oracle(sc, golden):
    from oracle import port

    device = _two_rings_device(sc, golden("two_rings"))
    model = sc.factorize_model(device=device, current_units="uA")
    fields = _two_ring_fields(sc)
    circ = [{}, {"upper_hole": 100.0}, {"lower_hole": -60.0}, {"upper_hole": 30.0, "lower_hole": 20.0}]
    batch = sc.solve_batch(model=model, applied_fields=fields, circulating_currents=circ,
                           translations=_TWO_RING_MOVES, iterations=3)
    zero = sc.ConstantField(0.0)
    for b, moves in enumerate(_TWO_RING_MOVES):
        moved = _moved_device(sc, device, _full(moves))
        info = sc.solver.utils.make_film_info(device=moved, vortices=[], circulating_currents=circ[b],
                                              terminal_currents={})
        films = []
        for name, film in moved.films.items():
            mesh = moved.meshes[name]
            films.append(port.factorize_film(port.OracleFilm(
                name=name, mesh=port.build_mesh(mesh.sites, mesh.elements), z0=float(moved.layers[film.layer].z0),
                Lambda=np.full(len(mesh.sites), float(moved.layers[film.layer].Lambda)),
                interior_indices=info[name].interior_indices, hole_indices=dict(info[name].hole_indices))))
        osols = port.solve(films, fields[b] or zero, circulating_currents=circ[b], iterations=3)
        assert len(batch[b]) == 4
        for it in range(4):
            for name in device.films:
                errs = _errs(batch[b][it].film_solutions[name], osols[it][name])
                assert all(e <= TOL_SOLUTION for e in errs.values()), (b, it, name, errs)


@pytest.mark.gpu
def test_two_rings_translated_against_serial_solves(sc, golden):
    device = _two_rings_device(sc, golden("two_rings"))
    model = sc.factorize_model(device=device, current_units="uA")
    fields = _two_ring_fields(sc)
    circ = [{"upper_hole": 50.0}, {}, {"upper_hole": 100.0}, {"lower_hole": 40.0}]
    batch = sc.solve_batch(model=model, applied_fields=fields, circulating_currents=circ,
                           translations=_TWO_RING_MOVES, iterations=3)
    worst = 0.0
    for b, moves in enumerate(_TWO_RING_MOVES):
        ref = sc.solve(_moved_device(sc, device, _full(moves)), applied_field=fields[b], circulating_currents=circ[b],
                       current_units="uA", iterations=3)
        for it in range(4):
            for name in device.films:
                errs = _errs(batch[b][it].film_solutions[name], ref[it].film_solutions[name])
                worst = max(worst, *errs.values())
                assert all(e <= TOL_SOLUTION for e in errs.values()), (b, it, name, errs)
    print(f"\ntwo rings, batch against serial solves on moved devices: max rel. L2 {worst:.3e}")


# ---------------------------------------------------------------------------------------------
# scanning SQUID: the IBM susceptometer over a sample film
# ---------------------------------------------------------------------------------------------
def _squid_over_sample(sc, n_vertices=2000, h=0.5):
    from superscreen_b200 import configs
    from superscreen_b200.geometry import box
    from superscreen_b200.synthetic import make_mesh

    squid, rings, meshes = configs.ibm_susceptometer("small", n_vertices, attach_meshes=False)
    sample = sc.Polygon("sample", layer="sample", points=box(8.0, 8.0, points=4, center=(0.5, -1.0)))
    layers = list(squid.layers.values()) + [sc.Layer("sample", Lambda=0.08, z0=-h)]
    device = sc.Device("scan", layers=layers, films=list(squid.films.values()) + [sample],
                       holes=list(squid.holes.values()), length_units="um")
    meshes = dict(meshes, sample=make_mesh(box(8.6, 8.6, points=4, center=(0.5, -1.0)), target_vertices=n_vertices,
                                           embedded=[sample.points[:-1]], seed=11))
    device.set_meshes(meshes)
    squid.set_meshes({k: v for k, v in meshes.items() if k != "sample"})
    return device, squid, rings["pl_center"]


def _M(solution, ring, shift=(0.0, 0.0)):
    """Field-coil -> pickup-loop mutual inductance (Phi_0 / A) at 1 mA in the field coil."""
    return sum(solution.hole_fluxoid("pl_center", points=ring + np.asarray(shift[:2]), with_units=False)) / 1e-3


@pytest.mark.gpu
def test_scanning_squid_touchdown_and_scan(sc):
    device, squid, ring = _squid_over_sample(sc)
    squid_layers = ("W2", "W1", "BE")
    touchdown = [0.0, 0.25, 0.75, 2.0]
    scan = [-1.5, 0.6, 2.5]
    entries = [{layer: (0.0, 0.0, dz) for layer in squid_layers} for dz in touchdown] + \
              [{layer: (dx, 0.0) for layer in squid_layers} for dx in scan]
    model = sc.factorize_model(device=device, current_units="uA", circulating_currents={"fc_center": "1 mA"})
    batch = sc.solve_batch(model=model, applied_fields=[None] * len(entries), translations=entries, iterations=5,
                           last_only=True)
    M_batch = [_M(batch[b][-1], ring, _full(e)["W1"]) for b, e in enumerate(entries)]
    M_serial = []
    for e in entries:
        ref = sc.solve(_moved_device(sc, device, _full(e)), circulating_currents={"fc_center": "1 mA"},
                       current_units="uA", iterations=5)[-1]
        M_serial.append(_M(ref, ring, _full(e)["W1"]))
    dM = np.abs(np.array(M_batch) - np.array(M_serial)) / np.abs(np.array(M_serial))
    M_free = _M(sc.solve(squid, circulating_currents={"fc_center": "1 mA"}, current_units="uA", iterations=5)[-1],
                ring)
    print(f"\nIBM small over a sample: M_free {M_free:.4f}, touchdown {dict(zip(touchdown, M_batch[:4]))}, "
          f"scan {dict(zip(scan, M_batch[4:]))} Phi_0/A; rel. |dM| batch vs serial {dM.tolist()}")
    # The susceptometer's meshes have vertices on the film and hole outlines; whether such a vertex is inside
    # its polygon is decided by rounding, so a device moved in-plane classifies some of them differently and
    # its serial solve is another discretization (about 1 % in M).  The batch keeps the unmoved classification.
    # A layer moved in z keeps every vertex where it was: the serial solve is the same problem.
    assert dM[:len(touchdown)].max() <= TOL_SOLUTION, (M_batch, M_serial)
    assert dM[len(touchdown):].max() <= 3e-2, (M_batch, M_serial)
    # diamagnetic screening by the sample lowers M, less so the farther the SQUID is
    gaps = [abs(M - M_free) for M in M_batch[:4]]
    assert all(M < M_free for M in M_batch[:4]), (M_batch, M_free)
    assert all(a > b for a, b in zip(gaps, gaps[1:])), (gaps, M_free)


# ---------------------------------------------------------------------------------------------
# batch semantics
# ---------------------------------------------------------------------------------------------
def _same_solutions(a, b, tol):
    for sa, sb in zip(a, b):
        for name in sa.film_solutions:
            fa, fb = sa.film_solutions[name], sb.film_solutions[name]
            if tol == 0:
                assert all(np.array_equal(getattr(fa, k), getattr(fb, k))
                           for k in ("stream", "current_density", "applied_field", "self_field",
                                     "field_from_other_films")), name
            else:
                errs = _errs(fa, fb)
                assert all(e <= tol for e in errs.values()), (name, errs)


@pytest.mark.gpu
def test_unmoved_batches_are_bit_identical(sc, golden):
    device = _two_rings_device(sc, golden("two_rings"))
    model = sc.factorize_model(device=device, current_units="uA")
    fields = _two_ring_fields(sc)
    circ = [{"upper_hole": 10.0}] * 4
    base = sc.solve_batch(model=model, applied_fields=fields, circulating_currents=circ, iterations=2)
    for translations in ([None] * 4, [{}] * 4, [{"up": (0.0, 0.0, 0.0)}, None, {"lo": (0.0, -0.0)}, {}]):
        got = sc.solve_batch(model=model, applied_fields=fields, circulating_currents=circ, iterations=2,
                             translations=translations)
        for b in range(4):
            _same_solutions(got[b], base[b], 0)
            assert got[b][-1]._device_builder is None


@pytest.mark.gpu
def test_mixed_batch_matches_per_entry_batches_and_permutations(sc, golden):
    device = _two_rings_device(sc, golden("two_rings"))
    model = sc.factorize_model(device=device, current_units="uA")
    fields = _two_ring_fields(sc) + [sc.ConstantField(0.1)]
    moves = _TWO_RING_MOVES + [{"lo": (0.1, 0.2, -0.1), "up": (0.5, 0.0)}]
    circ = [{"upper_hole": 20.0 * (b + 1)} for b in range(5)]
    mixed = sc.solve_batch(model=model, applied_fields=fields, circulating_currents=circ, translations=moves,
                           iterations=3)
    for b in range(5):
        single = sc.solve_batch(model=model, applied_fields=[fields[b]], circulating_currents=[circ[b]],
                                translations=[moves[b]], iterations=3)[0]
        _same_solutions(mixed[b], single, TOL_BATCH)
    perm = [3, 0, 4, 2, 1]
    permuted = sc.solve_batch(model=model, applied_fields=[fields[p] for p in perm],
                              circulating_currents=[circ[p] for p in perm], translations=[moves[p] for p in perm],
                              iterations=3)
    for k, p in enumerate(perm):
        _same_solutions(permuted[k], mixed[p], TOL_BATCH)


@pytest.mark.gpu
def test_equal_translations_share_one_lazily_built_device(sc, golden):
    device = _two_rings_device(sc, golden("two_rings"))
    model = sc.factorize_model(device=device, current_units="uA")
    moves = [{"up": (0.3, -0.2, 0.1)}, None, {"up": (0.3, -0.2, 0.1)}, {"up": (0.0, 0.0, 0.5)}]
    out = sc.solve_batch(model=model, applied_fields=[sc.ConstantField(0.1)] * 4, translations=moves, iterations=1)
    assert all(s._device is None for s in (out[0][0], out[2][0], out[3][0]))  # nothing built yet
    assert out[0][0].device is out[2][0].device is out[2][1].device
    assert out[3][0].device is not out[0][0].device and out[1][0].device is not out[0][0].device
    for b in (0, 3):
        got, want = out[b][0].device, _moved_device(sc, device, _full(moves[b]))
        for name in device.films:
            assert np.array_equal(got.films[name].points, want.films[name].points)
            assert np.array_equal(got.meshes[name].sites, want.meshes[name].sites)
            assert np.array_equal(got.meshes[name].elements, want.meshes[name].elements)
        for name in device.holes:
            assert np.array_equal(got.holes[name].points, want.holes[name].points)
        for name in device.layers:
            assert got.layers[name].z0 == want.layers[name].z0
    assert out[1][0].device.layers["up"].z0 == device.layers["up"].z0


@pytest.mark.gpu
def test_translated_solution_round_trips(sc, golden):
    from superscreen_b200 import io as scio

    device = _two_rings_device(sc, golden("two_rings"))
    model = sc.factorize_model(device=device, current_units="uA")
    sol = sc.solve_batch(model=model, applied_fields=[None, sc.ConstantField(0.1)],
                         translations=[None, {"up": (0.4, 0.1, 0.2)}], iterations=2)[1][-1]
    g = scio.MemoryGroup()
    sol.to_hdf5(g)
    back = sc.Solution.from_hdf5(g)
    assert back.device.layers["up"].z0 == sol.device.layers["up"].z0 == device.layers["up"].z0 + 0.2
    assert np.array_equal(back.device.meshes["upper"].sites, sol.device.meshes["upper"].sites)
    for name in device.films:
        for attr in ("stream", "current_density", "applied_field", "self_field"):
            assert np.array_equal(getattr(back.film_solutions[name], attr), getattr(sol.film_solutions[name], attr))


# ---------------------------------------------------------------------------------------------
# host-side validation (no GPU)
# ---------------------------------------------------------------------------------------------
def _host_device(Lambda_up=1.0):
    import superscreen_b200 as sc
    from superscreen_b200.geometry import box

    layers = [sc.Layer("lo", Lambda=1.0, z0=0.0), sc.Layer("up", Lambda=Lambda_up, z0=1.0)]
    films = [sc.Polygon("a", layer="lo", points=box(4.0, points=4)), sc.Polygon("b", layer="up", points=box(4.0, points=4))]
    return sc.Device("host", layers=layers, films=films)


def test_batch_translations_are_checked_on_the_host():
    import superscreen_b200 as sc
    from superscreen_b200.solver.solve import _batch_translations

    device = _host_device()
    none = [[]] * 3
    assert _batch_translations(device, [None, {}, {"up": (0.0, 0.0, 0.0)}], 3, none) is None
    got = _batch_translations(device, [None, {"up": (1, 2)}, {"lo": np.array([0.0, 0.5, -1.0])}], 3, none)
    assert got == [{}, {"up": (1.0, 2.0, 0.0)}, {"lo": (0.0, 0.5, -1.0)}]
    cases = [
        ([None, None], ValueError, "same length"),
        ([None, None, "up"], TypeError, "translations[2]"),
        ([None, {"side": (1.0, 0.0)}, None], KeyError, "translations[1]"),
        ([{"up": (1.0,)}, None, None], ValueError, "translations[0]"),
        ([None, {"up": (1.0, 2.0, 3.0, 4.0)}, None], ValueError, "translations[1]"),
        ([None, None, {"up": (np.nan, 0.0)}], ValueError, "translations[2]"),
        ([None, None, {"up": (0.0, np.inf, 0.0)}], ValueError, "translations[2]"),
        ([None, None, {"up": ("1", 0.0)}], ValueError, "translations[2]"),
        ([None, None, {"up": 1.0}], ValueError, "translations[2]"),
    ]
    for translations, exc, text in cases:
        with pytest.raises(exc) as info:
            _batch_translations(device, translations, 3, none)
        assert text in str(info.value), (translations, str(info.value))
    # a position-dependent Lambda cannot move (it may stay put)
    varying = _host_device(Lambda_up=lambda x, y: 1.0 + 0.1 * x)
    assert _batch_translations(varying, [{"lo": (1.0, 0.0)}], 1, [[]]) == [{"lo": (1.0, 0.0, 0.0)}]
    with pytest.raises(ValueError, match=r"translations\[0\].*position-dependent"):
        _batch_translations(varying, [{"up": (0.0, 0.0, 0.5)}], 1, [[]])
    lam = sc.Layer("up", london_lambda=lambda x, y: 0.1 + 0.0 * x, thickness=0.1, z0=1.0)
    varying.layers["up"] = lam
    with pytest.raises(ValueError, match=r"translations\[1\].*position-dependent"):
        _batch_translations(varying, [None, {"up": (1.0, 0.0)}], 2, [[], []])
    # a vortex in a moved layer is rejected; one in a layer that stays put is not
    vortex = sc.Vortex(0.5, 0.5, "b")
    assert _batch_translations(device, [{"lo": (1.0, 0.0)}], 1, [[vortex]]) == [{"lo": (1.0, 0.0, 0.0)}]
    with pytest.raises(ValueError, match=r"translations\[1\].*vortices in moved layers"):
        _batch_translations(device, [None, {"up": (1.0, 0.0)}], 2, [[], [vortex]])


def test_composite_polygons_translate_ring_by_ring():
    import superscreen_b200 as sc
    from superscreen_b200.geometry import box, circle

    comp = sc.Polygon("c", layer="l", points=box(2.0, points=4)).union(circle(0.5, 16) + 3.0)
    comp = comp.difference(circle(0.2, 12))
    moved = comp.translate(1.5, -0.5)
    assert moved is not comp
    for a, b in zip(moved.rings + moved.cut_rings, comp.rings + comp.cut_rings):
        assert np.array_equal(a, b + np.array([1.5, -0.5]))
    assert moved.contains_points([[1.5, -0.5 + 0.5], [1.5, -0.5]]).tolist() == [True, False]
    assert comp.translate(1.0, 0.0, inplace=True) is comp
