"""GPU parity on the BASELINE.json configurations as named (VERDICT round 1, "parity gaps"): the Ohio-shaped preset through
ClearwaterRiverine.update() (configs[1]), the 64-scenario ensemble on it (configs[3]), the 1M-cell x 16 mesh against the
ORACLE's own matrix and right-hand sides (configs[2]), the device mass balance against the oracle's on the reference's plans
(tests/test_final_mass.py, postproc_util.py:21-166), and a run with the flow hint turned against the flow.
Tolerance: concentrations within rtol 1e-9 per step of the reference's spsolve path (BASELINE.json north_star)."""
import numpy as np
import pytest

from oracle import reference_step as ref
from tests.helpers import golden_mesh, load_golden
from tests.test_gpu_parity import RTOL, close

pytestmark = pytest.mark.gpu
D = 0.1


def _oracle_mesh(plan, Dc=D):
    adv, _, _, cdiff, dt = ref.derive_coefficients(plan.face_flow, plan.edge_velocity, plan.face_x, plan.face_y,
                                                   plan.f1, plan.f2, Dc, plan.time_seconds)
    return ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, plan.edge_velocity, plan.volume, dt, Dc)


def test_ohio_preset_through_update_matches_oracle_every_step():
    """configs[1]: the Ohio-River-shaped mesh (2943 cells, hourly steps, Courant 2.5), one constituent, 60 steps through the
    reference-facing update() -- the on-chip solver k_solve_tiny with four rows per thread."""
    from clearwater_riverine_b200 import ClearwaterRiverine, synthetic
    plan = synthetic.ohio_like(n_time=61, seed=2)
    assert plan.n_real == 2943
    inputs = synthetic.make_inputs(plan, 1, seed=2)
    model = ClearwaterRiverine.from_arrays(plan.f1, plan.f2, plan.face_x, plan.face_y, plan.time_seconds, plan.face_flow,
                                           plan.edge_velocity, plan.volume, D, {"ecoli": inputs[0]})
    assert model.backend.options.solver_path == 4          # k_solve_chip
    oracle = ref.OracleRiverine(_oracle_mesh(plan), {"ecoli": inputs[0]})
    con = oracle.constituent_dict["ecoli"]
    for t in range(60):
        model.update()
        oracle.update()
        close(model.mesh["ecoli"][t + 1], con.concentration[t + 1], RTOL, f"ohio step {t}")
        fin = ~np.isnan(con.total_mass_flux[t])
        scale = np.abs(con.total_mass_flux[t][fin]).max()
        assert np.abs(model.constituent_dict["ecoli"].total_mass_flux[t][fin] - con.total_mass_flux[t][fin]).max() <= 1e-9 * scale
    assert max(s[2] for s in model.solver_info) == 0
    model.finalize()


def test_ensemble_of_64_scenarios_matches_oracle_on_sampled_scenarios():
    """configs[3]: 64 boundary-condition scenarios (BC series scaled per scenario) batched as 64 columns on the Ohio-shaped
    mesh; eight of them are replayed by the oracle."""
    from clearwater_riverine_b200 import TransportBackend, ensemble, synthetic
    T = 16
    plan = synthetic.ohio_like(n_time=T, seed=2)
    n = plan.n_real
    scales = np.exp(np.random.default_rng(100).normal(0.0, 0.5, size=64))
    base = synthetic.make_inputs(plan, 1, seed=2)[0]
    inputs = ensemble.scenario_inputs(base, n, scales)
    mesh = _oracle_mesh(plan)
    be = TransportBackend(plan.f1, plan.f2, plan.n_face, T, 64, D)
    be.set_hydro(0, mesh.adv, mesh.cdiff, mesh.vel, mesh.vol, mesh.dt)
    for k in range(64):
        be.set_inputs(k, inputs[k])
    info = be.run(0, T - 1)
    assert info.status == 0
    sampled = [0, 7, 13, 21, 34, 42, 55, 63]
    oracle = ref.OracleRiverine(mesh, {f"s{k}": inputs[k] for k in sampled})
    for _ in range(T - 1):
        oracle.update()
    for k in sampled:
        for t in (1, 8, T - 1):
            close(be.get_state(k, t), oracle.constituent_dict[f"s{k}"].concentration[t], RTOL, f"scenario {k} t {t}")
    be.close()


def test_1m_x16_against_the_oracles_own_matrix_and_right_hand_sides():
    """configs[2] at full size.  The oracle's numpy assembly of A and of every b takes seconds at 1M cells (its SuperLU
    solve would take ~50 s per column): (1) the GPU's LHS and RHS equal the oracle's; (2) the TRUE residual of every GPU
    column, formed with the ORACLE's A and b, is below 1e-12 ||b||; (3) one column equals an independent CPU solve of the
    oracle's system (scipy BiCGSTAB + Jacobi to 1e-13) within rtol 1e-9."""
    import bench
    plan, K = bench.workload_plan("1m16", 3, seed=2)
    assert plan.n_real == 1_000_000 and K == 16
    check_against_the_oracles_system(plan, K)


def check_against_the_oracles_system(plan, K, **want_options):
    """Two steps of plan (3 time slices, K constituents) at default options with the flow hint and raw hydrodynamics, as
    bench.py runs them, checked after the second step against the oracle's own A and b (see the test above).
    want_options: options the backend must have resolved to (the path the caller wrote its case for)."""
    import scipy.sparse as sp
    import scipy.sparse.linalg as spla
    from clearwater_riverine_b200 import TransportBackend, synthetic
    T = plan.n_time
    inputs = synthetic.make_inputs(plan, K, seed=2)
    mesh = _oracle_mesh(plan)
    be = TransportBackend(plan.f1, plan.f2, plan.n_face, T, K, D, flow_hint=plan.face_flow.mean(axis=0))
    for key, val in want_options.items():
        assert getattr(be.options, key) == val, (key, getattr(be.options, key), val)
    be.set_geometry(plan.face_x, plan.face_y)
    be.set_hydro_raw(0, plan.face_flow, plan.edge_velocity, plan.volume, mesh.dt)
    for k in range(K):
        be.set_inputs(k, inputs[k])
    assert be.step(0).status == 0
    c1 = be.get_state_all(1)                         # (K, n): the state the second step starts from
    info = be.step(1)
    assert info.status == 0 and info.max_relres <= 1e-13
    x = be.get_state_all(2)
    lhs = ref.LHS(mesh); lhs.update_values(mesh, 1)
    A = lhs.to_csr(); A.sum_duplicates(); A.sort_indices()
    Ag = be.get_lhs()
    assert np.array_equal(A.indptr, Ag.indptr) and np.array_equal(A.indices, Ag.indices)
    assert np.abs(A.data - Ag.data).max() <= 1e-14 * np.abs(A.data).max()
    worst = 0.0
    for k in range(K):
        rhs = ref.RHS(mesh, inputs[k]); rhs.update_values(c1[k].copy(), mesh, 1)
        b = np.asarray(rhs.vals, dtype=np.float64)
        bg = be.get_rhs(k)
        assert np.abs(b - bg).max() <= 1e-14 * np.abs(b).max(), k
        worst = max(worst, float(np.linalg.norm(A @ x[k] - b) / np.linalg.norm(b)))
    assert worst <= 1e-12, worst
    k = 5
    rhs = ref.RHS(mesh, inputs[k]); rhs.update_values(c1[k].copy(), mesh, 1)
    b = np.asarray(rhs.vals, dtype=np.float64)
    xs, status = spla.bicgstab(A, b, x0=c1[k].copy(), rtol=1e-13, atol=0.0, M=sp.diags(1.0 / A.diagonal()), maxiter=2000)
    assert status == 0
    assert np.abs(xs - x[k]).max() <= RTOL * np.abs(xs).max()
    be.close()


def test_1m_with_the_flow_hint_turned_against_the_flow():
    """Worst case of the static colouring: the hint says the water runs the other way, so the sweeps carry information
    upstream.  The solve must still converge to the same answer (more sweeps, no fallback needed: still an M-matrix)."""
    import bench
    from clearwater_riverine_b200 import TransportBackend, synthetic
    T = 3
    plan, _ = bench.workload_plan("1m16", T, seed=2)
    K = 4
    inputs = synthetic.make_inputs(plan, K, seed=2)
    dt = np.append(np.diff(plan.time_seconds), np.nan)
    outs, sweeps = {}, {}
    for name, sign in (("with", 1.0), ("against", -1.0)):
        be = TransportBackend(plan.f1, plan.f2, plan.n_face, T, K, D, flow_hint=sign * plan.face_flow.mean(axis=0))
        be.set_geometry(plan.face_x, plan.face_y)
        be.set_hydro_raw(0, plan.face_flow, plan.edge_velocity, plan.volume, dt)
        for k in range(K):
            be.set_inputs(k, inputs[k])
        for t in range(2):
            info = be.step(t)
            assert info.status == 0 and info.max_relres <= 1e-13, (name, t, info.status, info.max_relres)
        outs[name] = be.get_state_all(2)
        sweeps[name] = be.solver_stats()[0]
        be.close()
    assert np.abs(outs["with"] - outs["against"]).max() <= RTOL * np.abs(outs["with"]).max()
    assert sweeps["against"] > sweeps["with"], sweeps          # (the hint is what makes the sweeps cheap)


@pytest.mark.parametrize("case", ["p02_uniform100", "p01_uniform100", "p03_uniform100", "p01_random_two"])
def test_device_mass_balance_matches_the_oracles(case):
    """Next row N2 against postproc_util.py:21-166 as restated by the oracle, on the reference's own plans: Vol/Mass at start
    and end, per-boundary-line volume and mass (total / in / out), the closure error -- all from device reductions, no (T,E)
    flux history on the host.  Mass_end within 1e-9 relative (tests/test_final_mass.py:29-33, BASELINE.md)."""
    from clearwater_riverine_b200 import ClearwaterRiverine
    g = load_golden(case)
    if "override_steps" in g:
        pytest.skip("golden run with update_concentration overrides: covered by test_golden_free_running")
    names = [str(c) for c in g["constituents"]]
    mesh = golden_mesh(g)
    model = ClearwaterRiverine.from_arrays(g["f1"], g["f2"], g["face_x"], g["face_y"], g["time_seconds"], g["face_flow"],
                                           g["edge_velocity"], g["volume"], float(g["diffusion_coefficient"]),
                                           {c: g[f"input_{c}"] for c in names}, store_mass_flux=False, output="none")
    T = len(g["time_seconds"])
    for _ in range(T - 1):
        model.update()
    faces = {str(nm): np.array([f]) for nm, f in zip(g["bc_names"], g["bc_faces"])}
    for c in names:
        want = ref.mass_balance(mesh, g[f"conc_{c}"], g[f"totflux_{c}"], g["face_flow"], faces)
        mass_balance_close(model.mass_balance(c, faces), want, c)
    model.finalize()


def mass_balance_close(got, want, what):
    """ClearwaterRiverine.mass_balance() against ref.mass_balance: Mass_end within 1e-9 relative, the boundary sums within
    1e-9 of the largest boundary total."""
    assert abs(got["Mass_end"] - want["Mass_end"]) <= 1e-9 * abs(want["Mass_end"])
    assert abs(got["Mass_start"] - want["Mass_start"]) <= 1e-12 * abs(want["Mass_start"])
    assert abs(got["Vol_end"] - want["Vol_end"]) <= 1e-6 * abs(want["Vol_end"])          # (the oracle sums float32 volumes)
    scale_m = max(abs(want["bcTotalMassInAll"]), abs(want["bcTotalMassOutAll"]), 1e-300)
    scale_v = max(abs(want["bcTotalVolInAll"]), abs(want["bcTotalVolOutAll"]), 1e-300)
    for key, w in want.items():
        if key in ("Vol_start", "Vol_end", "Mass_start", "Mass_end", "error_vol", "vol_end_calc"):
            continue
        tol = 1e-9 * (scale_v if "vol" in key.lower() else scale_m)
        if key in ("mass_end_calc", "error_mass"):
            tol = 1e-9 * max(scale_m, abs(want["Mass_start"]))
        assert abs(got[key] - w) <= tol, (what, key, got[key], w)


class _Var:
    """The slice of an xarray DataArray attach() touches: `.values` backed by one array, `var[t]` a view of it."""
    def __init__(self, a):
        self.values = np.asarray(a)

    def __getitem__(self, i):
        return self.values[i]


class _Mesh(dict):
    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.attrs = {}

    nreal = property(lambda self: self.attrs["nreal"])
    diffusion_coefficient = property(lambda self: self.attrs["diffusion_coefficient"])


class _Con:
    pass


@pytest.mark.parametrize("case", ["p01_random_two", "p02_uniform100"])
def test_attach_swaps_update_on_a_reference_shaped_object(case):
    """attach(model) on an object with the reference's state layout (mesh[name].values, mesh.nreal, constituent_dict[...]
    .input_array / *_mass_flux, time_step): its update() -- overrides included -- must reproduce the golden run of the
    unmodified reference: concentrations (rtol 1e-9) and the three mass-flux arrays, in the object's own arrays."""
    from clearwater_riverine_b200 import attach
    from tests.helpers import golden_overrides
    g = load_golden(case)
    names = [str(c) for c in g["constituents"]]
    T, F = g["volume"].shape
    E = len(g["f1"])
    n = int(g["f1"].max()) + 1
    mesh = _Mesh({k: _Var(g[v]) for k, v in (("edges_face1", "f1"), ("edges_face2", "f2"), ("advection_coeff", "adv"),
                                            ("coeff_to_diffusion", "cdiff"), ("edge_velocity", "edge_velocity"),
                                            ("volume", "volume"), ("dt", "dt"))})
    mesh.attrs.update({"nreal": n - 1, "diffusion_coefficient": float(g["diffusion_coefficient"])})

    class Model:
        time_step = 0
        def update(self, update_concentration=None):
            raise AssertionError("the reference's own update() must have been replaced")
    model = Model()
    model.mesh = mesh
    model.constituent_dict = {}
    for c in names:
        con = _Con()
        con.input_array = g[f"input_{c}"].copy()
        con.advection_mass_flux, con.diffusion_mass_flux, con.total_mass_flux = np.zeros((T, E)), np.zeros((T, E)), np.zeros((T, E))
        model.constituent_dict[c] = con
        out = np.full((T, F), np.nan); out[0] = 0.0; out[0, :n] = con.input_array[0, :n]       # constituents.py:39-48, 94-98
        mesh[c] = _Var(out)
    stepper = attach(model)
    overrides = golden_overrides(g)
    steps = min(T - 1, 40)
    for t in range(steps):
        upd = {c: _Var(v) for c, v in overrides[t].items()} if t in overrides else None
        model.update(upd)
        assert model.time_step == t + 1
    for c in names:
        got, want = mesh[c].values, g[f"conc_{c}"]
        for t in range(steps + 1):
            close(got[t], want[t], RTOL, f"attach {c} row {t}")
        con = model.constituent_dict[c]
        for mine, theirs in ((con.advection_mass_flux, "advflux"), (con.diffusion_mass_flux, "diffflux"), (con.total_mass_flux, "totflux")):
            w = g[f"{theirs}_{c}"][:steps]
            fin = ~np.isnan(w)
            assert np.array_equal(np.isnan(mine[:steps]), ~fin)
            assert np.abs(mine[:steps][fin] - w[fin]).max() <= 1e-9 * max(np.abs(w[fin]).max(), 1e-300)
    stepper.detach()
    with pytest.raises(AssertionError):
        model.update()
