"""GPU tests of the batched / multi-film paths: solve_batch == repeated solve, fluxoids and the
mutual-inductance matrix against the CPU oracle, sharded field evaluation."""
import numpy as np
import pytest

from conftest import rel_l2

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sc():
    import torch

    assert torch.cuda.is_available()
    import superscreen_b200 as sc

    return sc


def _two_ring_device(sc, g):
    layers = [sc.Layer("lo", Lambda=float(g["in_lower_Lambda"][0]), z0=float(g["in_lower_z0"])),
              sc.Layer("up", Lambda=float(g["in_upper_Lambda"][0]), z0=float(g["in_upper_z0"]))]
    films = [sc.Polygon("lower", layer="lo", points=g["in_lower_film_polygon"]),
             sc.Polygon("upper", layer="up", points=g["in_upper_film_polygon"])]
    holes = [sc.Polygon("lower_hole", layer="lo", points=g["in_lower_hole_polygon"]),
             sc.Polygon("upper_hole", layer="up", points=g["in_upper_hole_polygon"])]
    device = sc.Device("two", layers=layers, films=films, holes=holes)
    device.set_meshes({k: (g[f"in_{k}_sites"], g[f"in_{k}_elements"]) for k in ("lower", "upper")})
    return device


def _oracle_films(g):
    from oracle import port

    films = []
    for name in ("lower", "upper"):
        mesh = port.build_mesh(g[f"in_{name}_sites"], g[f"in_{name}_elements"])
        film = port.OracleFilm(name=name, mesh=mesh, z0=float(g[f"in_{name}_z0"]), Lambda=g[f"in_{name}_Lambda"],
                               interior_indices=g[f"in_{name}_interior_indices"],
                               hole_indices={f"{name}_hole": g[f"in_{name}_hole_indices"]},
                               film_polygon=g[f"in_{name}_film_polygon"])
        films.append(port.factorize_film(film))
    return films


def test_solve_batch_equals_repeated_solve(sc, golden):
    g = golden("two_rings")
    device = _two_ring_device(sc, g)
    model = sc.factorize_model(device=device, current_units="uA")
    fields = [sc.ConstantField(0.2), None, lambda x, y, z: 0.1 * x + 0.05 * y, sc.ConstantField(-1.0),
              sc.ConstantField(0.3)]
    currents = [{"lower_hole": 1000.0}, {"upper_hole": -250.0}, {}, {"lower_hole": 10.0, "upper_hole": 20.0}, {}]
    batch = sc.solve_batch(model=model, applied_fields=fields, circulating_currents=currents, iterations=2)
    assert len(batch) == len(fields) and all(len(b) == 3 for b in batch)
    for b, (f, cc) in enumerate(zip(fields, currents)):
        model.set_circulating_currents(cc)
        ref = sc.solve(model=model, applied_field=f, iterations=2)
        for it in range(3):
            for name in ("lower", "upper"):
                a, r = batch[b][it].film_solutions[name], ref[it].film_solutions[name]
                assert rel_l2(a.stream, r.stream) <= 1e-12
                assert rel_l2(a.current_density, r.current_density) <= 1e-12
                assert rel_l2(a.total_field, r.total_field) <= 1e-12
    # iteration 3 of the golden case (batch entry 0 is the golden configuration)
    sol = sc.solve_batch(model=model, applied_fields=[sc.ConstantField(0.2)],
                         circulating_currents=[{"lower_hole": 1000.0}], iterations=3)[0]
    for name in ("lower", "upper"):
        assert rel_l2(sol[3].film_solutions[name].stream, g[f"out_it3_{name}_stream"]) <= 1e-8


def test_fluxoid_and_mutual_inductance_against_oracle(sc, golden):
    from oracle import port
    from superscreen_b200.geometry import circle, close_curve, points_in_polygon

    g = golden("two_rings")
    device = _two_ring_device(sc, g)
    polygons = {"lower_hole": circle(2.2, 101), "upper_hole": circle(1.5, 101, center=(0.3, -0.2))}
    iterations = 3
    M = device.mutual_inductance_matrix(polygons, units="pH", iterations=iterations)
    # oracle: one solve per driven hole + restated fluxoid (solution.py:484-563)
    films = _oracle_films(g)
    by_name = {f.name: f for f in films}
    in_poly = lambda poly, pts: points_in_polygon(poly, pts)
    Mref = np.zeros((2, 2))
    holes = ["lower_hole", "upper_hole"]
    film_of = {"lower_hole": "lower", "upper_hole": "upper"}
    conv_mA = 1e-3 / port.MU_0 * 1e-3  # mT -> mA/um
    for j, hole in enumerate(holes):
        sols = port.solve(films, lambda x, y, z: 0.0 * x, circulating_currents={hole: 1.0}, iterations=iterations,
                          field_conversion=conv_mA)
        for i, name in enumerate(holes):
            film = by_name[film_of[name]]
            flux, sup = port.polygon_fluxoid(film, sols[-1][film.name], close_curve(polygons[name]), in_poly,
                                             current_to_A=1e-3)
            Mref[i, j] = (flux + sup) * port.PHI_0 / 1e-3 * 1e12  # pH
    assert np.abs(M - Mref).max() <= 1e-8 * np.abs(Mref).max(), (M, Mref)
    # physics sanity kept from the reference's tests (test_solve.py:224-260): M symmetric to 5 %
    assert abs(M[0, 1] - M[1, 0]) <= 0.05 * abs(M[0, 1])
    assert M[0, 0] > 0 and M[1, 1] > 0
    # hole_fluxoid through the public API equals the oracle's restatement
    model = sc.factorize_model(device=device, current_units="uA", circulating_currents={"lower_hole": "1 mA"})
    sol = sc.solve(model=model, applied_field=sc.ConstantField(0.2), iterations=2)[-1]
    fl = sol.hole_fluxoid("lower_hole", points=polygons["lower_hole"], with_units=False)
    osol = port.solve(films, lambda x, y, z: 0.2 * np.ones_like(x), circulating_currents={"lower_hole": 1000.0},
                      iterations=2)[-1]
    oflux, osup = port.polygon_fluxoid(by_name["lower"], osol["lower"], close_curve(polygons["lower_hole"]), in_poly)
    assert abs(fl.flux_part - oflux) <= 1e-8 * abs(oflux)
    assert abs(fl.supercurrent_part - osup) <= 1e-8 * abs(osup)


def test_field_at_position_sharded_single_rank(sc, golden):
    g = golden("two_rings")
    device = _two_ring_device(sc, g)
    sol = sc.solve(device, applied_field=sc.ConstantField(0.2), circulating_currents={"lower_hole": 1000.0},
                   iterations=1)[-1]
    rng = np.random.default_rng(3)
    pos = np.column_stack([rng.uniform(-4, 4, 500), rng.uniform(-4, 4, 500), rng.uniform(1.5, 3.0, 500)])
    full = sol.field_at_position(pos, units="mT", with_units=False)
    sharded = sc.parallel.field_at_position_sharded(sol, pos, units="mT")
    assert np.array_equal(full, sharded)
    vec = sol.screening_field_at_position(pos, vector=True, units="mT", with_units=False)
    z = sol.screening_field_at_position(pos, vector=False, units="mT", with_units=False)
    assert vec.shape == (500, 3) and rel_l2(vec[:, 2], z) <= 1e-12
    A = sol.vector_potential_at_position(pos, with_units=False)
    assert A.shape == (500, 3) and np.all(A[:, 2] == 0) and np.isfinite(A).all()
    # oracle check of the vector potential (solution.py:917-928): mu0/4pi sum_j w_j J_j / rho
    from oracle import port

    ref = np.zeros((500, 2))
    for name, z0 in (("lower", 0.0), ("upper", 1.0)):
        mesh = device.meshes[name]
        J = sol.film_solutions[name].current_density
        d = pos[:, None, :2] - mesh.sites[None, :, :]
        rho = np.sqrt((d ** 2).sum(-1) + (pos[:, 2:3] - z0) ** 2)
        ref += np.einsum("ijk,j->ik", J[None, :, :] / rho[:, :, None], mesh.vertex_areas)
    ref *= port.MU_0 / (4 * np.pi) * 1e-6 * 1e3 * 1e6  # uA -> A, T*m -> mT*um
    assert rel_l2(A[:, :2], ref) <= 1e-8


def test_find_fluxoid_solution(sc):
    """reference fluxoid.py:55-119 / test_solve.py:300-328: the circulating currents that realise a
    target fluxoid state; checked by recomputing the fluxoids of the returned solution."""
    from superscreen_b200 import configs

    device, polygons = configs.c1_ring(1200)
    model = sc.factorize_model(device=device, current_units="uA")
    for target in (0.0, 1.0):
        sol = sc.find_fluxoid_solution(model, fluxoids={"ring_hole": target}, hole_polygon_mapping=polygons,
                                       applied_field=sc.ConstantField(0.05))
        fl = sol.hole_fluxoid("ring_hole", points=polygons["ring_hole"], with_units=False)
        assert abs(sum(fl) - target) <= 1e-6, (target, sum(fl))
        assert "ring_hole" in sol.circulating_currents
    # the model's own circulating currents are restored afterwards
    assert model.circulating_currents == {}


@pytest.mark.parametrize("nrhs", [3, 9, 16, 21, 70])
def test_many_rhs_tensor_core_substitution(sc, nrhs):
    """2..8 right-hand sides take the flag-driven DMMA sweeps in one chain of 8 columns (getrs.cu:
    trsm_sweep_dmma_kernel<8>), more run chains of 16 columns (trsm_sweep_dmma_kernel<16>); both must agree with
    column-by-column solves, including column counts that are not a multiple of the 8- / 16-column
    chunks and a padded last block."""
    import torch

    from superscreen_b200.geometry import box
    from superscreen_b200.solver.solve_film import apply_operator, lu_solve
    from superscreen_b200.synthetic import square_mesh

    sites, elements = square_mesh(10.0, 1500, seed=3)
    device = sc.Device("sq", layers=[sc.Layer("layer", Lambda=0.1, z0=0.0)],
                       films=[sc.Polygon("film", layer="layer", points=box(10.0, points=4))])
    device.set_meshes({"film": (sites, elements)})
    model = sc.factorize_model(device=device, current_units="uA")
    system, info = model.film_systems["film"], model.film_info["film"]
    assert system.n_pad > len(system.indices)  # identity-padded last block
    gen = torch.Generator(device="cuda").manual_seed(1)
    h = torch.randn(len(system.indices), nrhs, dtype=torch.float64, device="cuda", generator=gen)
    x = lu_solve(system, h)
    ref = torch.stack([lu_solve(system, h[:, c].contiguous()) for c in range(nrhs)], dim=1)
    assert float((x - ref).norm() / ref.norm()) <= 1e-13
    # and it solves the system: (-A) x = h through the matrix-free operator
    ix = system.indices_dev
    g = torch.zeros(info.mesh._data.n, dtype=torch.float64, device="cuda")
    g[ix] = x[:, nrhs - 1]
    res = -apply_operator(info, g, src_idx=ix)[ix] - h[:, nrhs - 1]
    assert float(res.abs().max() / h[:, nrhs - 1].abs().max()) <= 1e-10
    # the matrix-free operator itself: nrhs >= 16 columns go through the tensor-core kernel GEMM
    # (nbody.cu: kernel_gemm_kernel), fewer through the CUDA-core N-body kernel
    V = torch.zeros(info.mesh._data.n, nrhs, dtype=torch.float64, device="cuda")
    V[ix] = x
    out = apply_operator(info, V, src_idx=ix)
    cols = torch.stack([apply_operator(info, V[:, c].contiguous(), src_idx=ix) for c in range(nrhs)], dim=1)
    assert float((out - cols).norm() / cols.norm()) <= 1e-13
    full = apply_operator(info, V)  # no gather list: every vertex is a source (V vanishes outside ix)
    assert float((full - cols).norm() / cols.norm()) <= 1e-13


def test_empty_evaluation_sets(sc, golden):
    """Edge cases of the field evaluation: no evaluation points and points that all lie in a film."""
    g = golden("two_rings")
    device = _two_ring_device(sc, g)
    sol = sc.solve(device, applied_field=sc.ConstantField(0.3), circulating_currents={"lower_hole": 500.0})[0]
    empty = sol.field_at_position(np.zeros((0, 3)), units="mT", with_units=False)
    assert np.asarray(empty).shape == (0,)
    from superscreen_b200.solution import biot_savart_2d

    mesh = device.meshes["lower"]
    out = biot_savart_2d(np.zeros(0), np.zeros(0), np.zeros(0), positions=mesh.sites,
                         current_densities=sol.film_solutions["lower"].current_density, z0=0.0,
                         areas=mesh.vertex_areas, vector=True)
    assert out.shape == (0, 3)
    one = sol.field_at_position(np.array([[0.1, 0.2, 3.0]]), units="mT", with_units=False)
    assert np.asarray(one).shape in ((), (1,)) and np.isfinite(one).all()
