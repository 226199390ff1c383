"""First-order kinetics in the device step (cwr_set_kinetics): the spec compiler and the numpy restatement on the CPU,
the CUDA path against oracle.kinetics.KineticsRiverine on the GPU.  GPU tolerance as in test_gpu_parity: rtol 1e-9 per
step, mass fluxes within 1e-9 of their scale."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from oracle import reference_step as ref
from oracle.kinetics import KineticsRiverine, react
from tests.helpers import golden_mesh, golden_overrides, load_golden, same

ROOT = Path(__file__).resolve().parents[1]
RTOL = 1e-9
SPEC = {"BOD": {"decay_per_day": 0.23, "theta": 1.047, "yields": {"DO": -1.0}},
        "NH4": {"decay_per_day": 0.10, "theta": 1.083, "yields": {"NO3": 1.0, "DO": -4.57}}}


# ------------------------------------------------------------------------------------------------------------------
# CPU: spec compiler
# ------------------------------------------------------------------------------------------------------------------
def test_spec_compiles_to_the_abi_arrays():
    from clearwater_riverine_b200.kinetics import compile_kinetics
    names = ["DO", "NO3", "NH4", "BOD", "T"]
    kin = compile_kinetics(SPEC, names, "T")
    assert kin.decay_per_day.tolist() == [0.0, 0.0, 0.10, 0.23, 0.0]
    assert kin.theta.tolist() == [1.0, 1.0, 1.083, 1.047, 1.0]
    assert kin.yields[0, 3] == -1.0 and kin.yields[1, 2] == 1.0 and kin.yields[0, 2] == -4.57
    assert np.count_nonzero(kin.yields) == 3
    assert (kin.temperature_k, kin.temperature_c) == (4, 20.0)
    kin = compile_kinetics(SPEC, names, 12.5)
    assert (kin.temperature_k, kin.temperature_c) == (-1, 12.5)


@pytest.mark.parametrize("names", [["A", "B", "C", "D"], ["D", "C", "B", "A"], ["C", "A", "D", "B"]])
def test_a_chain_is_ordered_topologically_whatever_the_column_order(names):
    from clearwater_riverine_b200.kinetics import compile_kinetics
    spec = {"A": {"decay_per_day": 1.0, "yields": {"B": 1.0}}, "B": {"decay_per_day": 1.0, "yields": {"C": 0.5}},
            "C": {"decay_per_day": 1.0, "yields": {"D": 2.0}}}
    order = [names[k] for k in compile_kinetics(spec, names).order]
    assert order.index("A") < order.index("B") < order.index("C") < order.index("D")


INVALID = {
    "negative decay": ({"A": {"decay_per_day": -1.0}}, 20.0),
    "non-finite decay": ({"A": {"decay_per_day": float("inf")}}, 20.0),
    "zero theta": ({"A": {"decay_per_day": 1.0, "theta": 0.0}}, 20.0),
    "non-finite theta": ({"A": {"decay_per_day": 1.0, "theta": float("nan")}}, 20.0),
    "non-finite yield": ({"A": {"decay_per_day": 1.0, "yields": {"B": float("nan")}}}, 20.0),
    "self yield": ({"A": {"decay_per_day": 1.0, "yields": {"A": 0.5}}}, 20.0),
    "cycle": ({"A": {"decay_per_day": 1.0, "yields": {"B": 1.0}}, "B": {"decay_per_day": 1.0, "yields": {"A": 1.0}}}, 20.0),
    "temperature decays": ({"T": {"decay_per_day": 1.0}}, "T"),
    "temperature receives": ({"A": {"decay_per_day": 1.0, "yields": {"T": 1.0}}}, "T"),
    "unknown constituent": ({"X": {"decay_per_day": 1.0}}, 20.0),
    "unknown yield target": ({"A": {"decay_per_day": 1.0, "yields": {"X": 1.0}}}, 20.0),
    "unknown temperature": ({"A": {"decay_per_day": 1.0}}, "X"),
    "non-finite temperature": ({"A": {"decay_per_day": 1.0}}, float("nan")),
    "unknown key": ({"A": {"decay": 1.0}}, 20.0),
}


@pytest.mark.parametrize("case", sorted(INVALID))
def test_invalid_specs_are_rejected(case):
    from clearwater_riverine_b200.kinetics import compile_kinetics
    spec, temperature = INVALID[case]
    with pytest.raises(ValueError):
        compile_kinetics(spec, ["A", "B", "T"], temperature)


# ------------------------------------------------------------------------------------------------------------------
# CPU: the numpy restatement
# ------------------------------------------------------------------------------------------------------------------
def test_single_decay_is_exponential():
    rng = np.random.default_rng(0)
    c = 100.0 * rng.random((1, 50))
    for T, theta in ((20.0, 1.047), (27.5, 1.047), (8.0, 1.08)):
        got = react(c, 300.0, [2.5], [theta], None, T)
        want = c * np.exp(-2.5 * theta ** (T - 20.0) * 300.0 / 86400.0)
        assert np.abs(got - want).max() <= 1e-15 * np.abs(want).max()


def test_rate_is_unchanged_at_20_degrees_or_theta_1():
    c = np.full((1, 4), 3.0)
    want = c - c * -np.expm1(-(1.7 / 86400.0) * 60.0)
    assert same(react(c, 60.0, [1.7], [1.3], None, 20.0), want)
    assert same(react(c, 60.0, [1.7], [1.0], None, 31.0), want)


def test_a_to_b_chain_with_yield_one_conserves_mass():
    rng = np.random.default_rng(1)
    c = 10.0 * rng.random((2, 100))
    got = react(c, 3600.0, [5.0, 0.0], None, np.array([[0.0, 0.0], [1.0, 0.0]]), 15.0)
    assert np.abs((got[0] + got[1]) - (c[0] + c[1])).max() <= 1e-15 * np.abs(c[0] + c[1]).max()
    assert (got[0] < c[0]).all()


def test_permuting_the_columns_permutes_the_result():
    rng = np.random.default_rng(2)
    K = 5
    c = 50.0 * rng.random((K, 30)); c[4] = 10.0 + 20.0 * rng.random(30)
    decay = np.array([3.0, 1.0, 0.5, 2.0, 0.0]); theta = np.array([1.05, 1.02, 1.08, 1.01, 1.0])
    y = np.zeros((K, K)); y[1, 0] = 1.0; y[2, 1] = -0.5; y[3, 0] = 0.25
    base = react(c, 900.0, decay, theta, y, 4, True)
    perm = np.array([3, 4, 0, 2, 1])
    inv = np.argsort(perm)
    got = react(c[perm], 900.0, decay[perm], theta[perm], y[np.ix_(perm, perm)], int(inv[4]), True)
    assert np.abs(got - base[perm]).max() <= 1e-15 * np.abs(base).max()


def test_zero_rates_are_bitwise_the_oracle_with_overrides():
    g = load_golden("p01_random_two")
    mesh = golden_mesh(g)
    names = [str(c) for c in g["constituents"]]
    inputs = {c: g[f"input_{c}"] for c in names}
    overrides = golden_overrides(g)
    a = ref.OracleRiverine(mesh, inputs)
    b = KineticsRiverine(mesh, inputs, np.zeros(len(names)), np.full(len(names), 1.05), None, 12.0)
    for t in range(mesh.n_time - 1):
        a.update(overrides.get(t))
        b.update(overrides.get(t))
    for c in names:
        assert same(a.constituent_dict[c].concentration, b.constituent_dict[c].concentration)
        assert same(a.constituent_dict[c].total_mass_flux, b.constituent_dict[c].total_mass_flux)
    assert all((m == 0).all() for m in b.reaction_mass)


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def _parity():
    from tests import test_gpu_parity as tp
    return tp


def kinetic_backend(mesh, inputs, kin, **opt):
    be = _parity().make_backend(mesh, list(inputs), **opt)
    if kin is not None:
        be.set_kinetics(**kin)
    return be


def kinetic_oracle(mesh, inputs, kin):
    temperature = f"c{kin['temperature_k']}" if kin["temperature_k"] >= 0 else kin["temperature_c"]
    return KineticsRiverine(mesh, {f"c{k}": inputs[k] for k in range(len(inputs))}, kin["decay_per_day"], kin["theta"],
                            kin["yields"], temperature)


def mass_scale(mesh, inputs):
    n = mesh.n
    return np.array([abs((mesh.vol[0][:n] * a[0, :n]).sum()) for a in inputs])


def run_kinetic_parity(mesh, inputs, kin, steps, overrides=None, check_flux=True, **opt):
    tp = _parity()
    K = len(inputs)
    be = kinetic_backend(mesh, inputs, kin, **opt)
    oracle = kinetic_oracle(mesh, inputs, kin)
    for t in range(steps):
        upd = (overrides or {}).get(t)
        for name, v in (upd or {}).items():
            be.set_state(int(name[1:]), t, v)
        info = be.step(t)
        assert info.status == 0, (t, info.status, info.iterations, info.max_relres)
        oracle.update(upd)
        for k in range(K):
            con = oracle.constituent_dict[f"c{k}"]
            tp.close(be.get_state(k, t + 1), con.concentration[t + 1], RTOL, f"step {t} k {k}")
            tp.close(be.get_state(k, t), con.concentration[t], RTOL, f"history row {t} k {k}")
            if check_flux:
                tp.flux_close(be, k, t, mesh, con.concentration[t + 1], con.advection_mass_flux[t], con.diffusion_mass_flux[t],
                              con.total_mass_flux[t], f"step {t} k {k}")
    want = np.sum(oracle.reaction_mass, axis=0)
    got = np.array([be.reaction_mass(k) for k in range(K)])
    scale = np.maximum(np.abs(want), mass_scale(mesh, inputs))
    assert (np.abs(got - want) <= RTOL * scale).all(), (got, want)
    return be, oracle


def golden_kinetic_case():
    from clearwater_riverine_b200 import synthetic
    g = load_golden("p01_random_two")
    mesh = golden_mesh(g)
    names = [str(c) for c in g["constituents"]]
    a, b = g[f"input_{names[0]}"], g[f"input_{names[1]}"]
    inputs = np.stack([a, b, 0.5 * a + 0.25 * b, np.where(b != 0, b, 0.0)])      # the last one becomes the temperature
    inputs, kin = synthetic.make_kinetics(inputs, seed=3, decay_range=(2000.0, 20000.0))   # dt = 1 s here
    return g, mesh, inputs, kin


@pytest.mark.gpu
def test_golden_mesh_parity_with_overrides():
    g, mesh, inputs, kin = golden_kinetic_case()
    n = mesh.n
    overrides = {3: {"c1": 40.0 + np.arange(n, dtype=np.float64)}, 9: {"c0": np.full(n, 7.0), "c2": np.linspace(1, 2, n)}}
    be, _ = run_kinetic_parity(mesh, inputs, kin, 30, overrides)
    be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("solver", [1, 2])
@pytest.mark.parametrize("K", [1, 3, 16, 18, 19, 33])
def test_synthetic_meshes_on_the_large_path(K, solver):
    from clearwater_riverine_b200 import synthetic
    _, mesh, inputs = _parity().synthetic_case(40, 25, 8, K, seed=K + 50, dry_fraction=0.02)
    inputs, kin = synthetic.make_kinetics(inputs, seed=K)
    be, _ = run_kinetic_parity(mesh, inputs, kin, 7, solver_path=1, solver=solver)
    be.close()


@pytest.mark.gpu
def test_every_column_count_up_to_kmax():
    """k_react's tile is sized from K (shared memory within 48 KB for every K <= 128): one reacted step per K, on both
    paths, against the oracle."""
    from clearwater_riverine_b200 import synthetic
    plan, mesh, base = _parity().synthetic_case(12, 9, 3, 128, seed=91)
    for K in range(1, 129):
        inputs, kin = synthetic.make_kinetics(base[:K], seed=K)
        for solver_path in (1, 2):
            be, _ = run_kinetic_parity(mesh, inputs, kin, 1, check_flux=False, solver_path=solver_path)
            be.close()


@pytest.mark.gpu
def test_small_path_parity():
    from clearwater_riverine_b200 import synthetic
    _, mesh, inputs = _parity().synthetic_case(40, 25, 7, 5, seed=61, dry_fraction=0.02)
    inputs, kin = synthetic.make_kinetics(inputs, seed=5)
    be, _ = run_kinetic_parity(mesh, inputs, kin, 6, solver_path=2, precond_sweep=0)
    assert be.options.solver_path == 2
    be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 64])
def test_on_chip_path_on_the_ohio_shaped_mesh(K):
    """K = 1, and 64 scenarios of one constituent with 64 different decay rates (a rate sweep)."""
    from clearwater_riverine_b200 import synthetic
    plan = synthetic.ohio_like(7, seed=2)
    D = 0.1
    adv, _, _, cdiff, dt = ref.derive_coefficients(plan.face_flow, plan.edge_velocity, plan.face_x, plan.face_y, plan.f1, plan.f2,
                                                   D, plan.time_seconds)
    mesh = ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, plan.edge_velocity, plan.volume, dt, D)
    inputs = synthetic.make_inputs(plan, K, seed=7)
    kin = dict(decay_per_day=np.linspace(0.05, 3.0, K), theta=np.full(K, 1.047), yields=None, temperature_k=-1,
               temperature_c=17.0)
    be, _ = run_kinetic_parity(mesh, inputs, kin, 6, check_flux=K == 1)
    assert be.options.solver_path in (3, 4)
    be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("solver_path", [1, 2])
def test_zero_rates_are_bitwise_no_kinetics_with_one_more_launch(solver_path):
    from clearwater_riverine_b200 import synthetic
    _, mesh, inputs = _parity().synthetic_case(40, 25, 7, 4, seed=71, dry_fraction=0.02)
    inputs, kin = synthetic.make_kinetics(inputs, seed=9)
    kin0 = dict(kin, decay_per_day=np.zeros(4))
    plain = kinetic_backend(mesh, inputs, None, solver_path=solver_path)
    zero = kinetic_backend(mesh, inputs, kin0, solver_path=solver_path)
    toggled = kinetic_backend(mesh, inputs, kin, solver_path=solver_path)
    toggled.set_kinetics(None)
    for t in range(6):
        a, b, c = plain.step(t), zero.step(t), toggled.step(t)
        assert b.n_launches == a.n_launches + 1 and c.n_launches == a.n_launches
        assert same(plain.get_state_all(t + 1), zero.get_state_all(t + 1))
        assert same(plain.get_state_all(t + 1), toggled.get_state_all(t + 1))
        for k in range(4):
            assert all(same(x, y) for x, y in zip(plain.get_mass_flux(k, t), zero.get_mass_flux(k, t)))
    assert all(zero.reaction_mass(k) == 0.0 and plain.reaction_mass(k) == 0.0 for k in range(4))
    for be in (plain, zero, toggled):
        be.close()


@pytest.mark.gpu
def test_reaction_mass_is_not_doubled_by_the_defect_correction_fallback():
    """The setup of test_gpu_parity's fallback test: the sweeps diverge, the step forms its right-hand side again and
    solves with BiCGSTAB; the reaction mass of that step is counted once."""
    from clearwater_riverine_b200 import synthetic
    plan = synthetic.make_plan(60, 50, 6, seed=41, dry_fraction=0.02)
    vel = plan.edge_velocity.copy()
    vel[:, np.random.default_rng(1).random(plan.n_edge) < 0.05] *= -1
    D = 2.0
    adv, _, _, cdiff, dt = ref.derive_coefficients(plan.face_flow, vel, plan.face_x, plan.face_y, plan.f1, plan.f2, D, plan.time_seconds)
    mesh = ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, vel, plan.volume, dt, D)
    inputs = synthetic.make_inputs(plan, 3, seed=41)
    inputs, kin = synthetic.make_kinetics(inputs, seed=41)
    tp = _parity()
    be = kinetic_backend(mesh, inputs, kin, solver_path=1, solver=2)
    oracle = kinetic_oracle(mesh, inputs, kin)
    for t in range(3):
        assert be.step(t).status == 0
        oracle.update()
        for k in range(3):
            tp.close(be.get_state(k, t + 1), oracle.constituent_dict[f"c{k}"].concentration[t + 1], 1e-8, f"fallback k{k} t{t}")
        want = np.sum(oracle.reaction_mass, axis=0)
        for k in range(3):
            assert abs(be.reaction_mass(k) - want[k]) <= RTOL * max(abs(want[k]), mass_scale(mesh, inputs)[k]), (t, k)
    assert be.solver_stats()[1] >= 1, "the sweeps diverge on this matrix: the solver should have fallen back"
    be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("solver_path", [1, 2])
def test_run_is_bitwise_step_by_step_and_repeatable(solver_path):
    from clearwater_riverine_b200 import synthetic
    _, mesh, inputs = _parity().synthetic_case(30, 20, 10, 5, seed=81, dry_fraction=0.02)
    inputs, kin = synthetic.make_kinetics(inputs, seed=81)
    outs = []
    for mode in ("step", "run", "run"):
        be = kinetic_backend(mesh, inputs, kin, solver_path=solver_path)
        if mode == "step":
            for t in range(9):
                assert be.step(t).status == 0
        else:
            assert be.run(0, 9).status == 0
        outs.append((np.stack([be.get_state_all(t) for t in range(1, 10)]), [be.reaction_mass(k) for k in range(5)]))
        be.close()
    for states, masses in outs[1:]:
        assert same(states, outs[0][0]) and masses == outs[0][1]
    oracle = kinetic_oracle(mesh, inputs, kin)
    for _ in range(9):
        oracle.update()
    for k in range(5):
        _parity().close(outs[1][0][-1][k], oracle.constituent_dict[f"c{k}"].concentration[9][:mesh.n], RTOL, f"run k{k}")


@pytest.mark.gpu
def test_update_concentration_then_kinetics_and_the_mass_balance():
    """The coupling loop through ClearwaterRiverine: override -> reaction -> transport against the oracle given the same
    override; mass_balance() gains reaction_mass (and closes with it) only while kinetics is set."""
    from clearwater_riverine_b200 import ClearwaterRiverine, synthetic
    tp = _parity()
    plan, mesh, inputs = tp.synthetic_case(20, 14, 8, 3, seed=4)
    inputs, kin = synthetic.make_kinetics(inputs, seed=4)
    names = ["A", "B", "C"]
    spec = {names[k]: {"decay_per_day": float(kin["decay_per_day"][k]), "theta": float(kin["theta"][k]),
                       "yields": {names[j]: float(kin["yields"][j, k]) for j in range(3) if kin["yields"][j, k] != 0}}
            for k in range(3)}
    arrays = (plan.f1, plan.f2, plan.face_x, plan.face_y, plan.time_seconds, plan.face_flow, plan.edge_velocity, plan.volume, 0.1)
    model = ClearwaterRiverine.from_arrays(*arrays, dict(zip(names, inputs)), kinetics=spec, temperature=kin["temperature_c"])
    plain = ClearwaterRiverine.from_arrays(*arrays, dict(zip(names, inputs)))
    oracle = KineticsRiverine(mesh, dict(zip(names, inputs)), kin["decay_per_day"], kin["theta"], kin["yields"], kin["temperature_c"])
    n = mesh.n
    rng = np.random.default_rng(1)
    for t in range(7):
        upd = {"B": 50.0 + rng.random(n)} if t in (2, 4) else None
        model.update(upd)
        plain.update(upd)
        oracle.update(upd)
        for name in names:
            tp.close(model.mesh[name][t + 1], oracle.constituent_dict[name].concentration[t + 1], RTOL, f"{name} {t}")
            tp.close(model.mesh[name][t], oracle.constituent_dict[name].concentration[t], RTOL, f"{name} history {t}")
    faces = {nm: plan.boundary_faces[nm] for nm in ("upstream", "downstream")}
    for k, name in enumerate(names):
        got = model.mass_balance(name, faces)
        con = oracle.constituent_dict[name]
        want = ref.mass_balance(mesh, con.concentration, con.total_mass_flux, plan.face_flow, faces)   # 7 steps = the whole run
        reaction = float(np.sum(oracle.reaction_mass, axis=0)[k])
        want_error = want["mass_end_calc"] + reaction - want["Mass_end"]
        assert "reaction_mass" in got
        assert abs(got["reaction_mass"] - reaction) <= RTOL * abs(want["Mass_start"])
        assert abs(got["error_mass"] - want_error) <= RTOL * abs(want["Mass_start"]), (name, got["error_mass"], want_error)
        assert "reaction_mass" not in plain.mass_balance(name, faces)
    model.set_kinetics(None)
    assert "reaction_mass" not in model.mass_balance("A", faces)
    model.finalize(); plain.finalize()


@pytest.mark.gpu
def test_yaml_config_with_kinetics_blocks_is_bitwise_from_arrays(tmp_path):
    yaml = pytest.importorskip("yaml")
    import pandas as pd
    from clearwater_riverine_b200 import ClearwaterRiverine
    from clearwater_riverine_b200.io import ras
    from tests.ras_fixture import write_plan
    g = load_golden("p01_random_two")
    hdf = tmp_path / "plan.hdf"
    times = write_plan(hdf, g)
    plan = ras.read_ras_plan(hdf)
    n = plan.nreal + 1
    lines = sorted({str(x) for x in g["bc_names"]})
    cons = {}
    for name, ic, bc in (("NH4", 3.0, 5.0), ("NO3", 1.0, 2.0), ("T", 18.0, 21.0)):
        icf, bcf = tmp_path / f"{name}_ic.csv", tmp_path / f"{name}_bc.csv"
        pd.DataFrame({"Cell_Index": np.arange(n), "Concentration": ic + 0.01 * np.arange(n)}).to_csv(icf, index=False)
        pd.DataFrame({"Datetime": np.repeat([times[0], times[-1]], len(lines)), "RAS2D_TS_Name": lines * 2,
                      "Concentration": bc}).to_csv(bcf, index=False)
        cons[name] = {"initial_conditions": str(icf), "boundary_conditions": str(bcf), "units": "mg/L"}
    spec = {"NH4": {"decay_per_day": 900.0, "theta": 1.083, "yields": {"NO3": 1.0}}, "NO3": {"decay_per_day": 300.0}}
    cfg = {"diffusion_coefficient": 0.1, "flow_field_filepath": str(hdf), "temperature": "T",
           "constituents": {name: dict(c, **({"kinetics": spec[name]} if name in spec else {})) for name, c in cons.items()}}
    cfg_path = tmp_path / "model.yml"
    cfg_path.write_text(yaml.safe_dump(cfg))
    a = ClearwaterRiverine(config_filepath=str(cfg_path))
    inputs = {name: ras.build_input_array(len(plan.time), len(plan.face_x), plan.time, plan.f2, plan.boundary_data,
                                          c["initial_conditions"], c["boundary_conditions"]) for name, c in cons.items()}
    b = ClearwaterRiverine.from_arrays(plan.f1, plan.f2, plan.face_x, plan.face_y, plan.time_seconds, plan.face_flow,
                                       plan.edge_velocity, plan.volume, 0.1, inputs)
    b.set_kinetics(spec, temperature="T")
    for _ in range(12):
        a.update(); b.update()
    for name in cons:
        assert same(a.mesh[name][:13], b.mesh[name][:13]), name
        assert a.backend.reaction_mass(a._index[name]) == b.backend.reaction_mass(b._index[name])
    assert a.backend.reaction_mass(0) < 0.0
    a.finalize(); b.finalize()


@pytest.mark.gpu
def test_invalid_kinetics_straight_to_the_abi_return_einval():
    import ctypes as C
    from clearwater_riverine_b200.backend import CWR_EINVAL
    _, mesh, inputs = _parity().synthetic_case(12, 9, 4, 3, seed=2)
    be = _parity().make_backend(mesh, list(inputs))
    lib = be._lib
    ok_d, ok_th, ok_y = np.array([1.0, 1.0, 0.0]), np.ones(3), np.zeros((3, 3))
    nan = float("nan")

    def call(d, th=None, y=None, tk=-1, tc=20.0):
        p = lambda a: None if a is None else np.ascontiguousarray(a, np.float64).ctypes.data_as(C.POINTER(C.c_double))
        arrs = [None if a is None else np.ascontiguousarray(a, np.float64) for a in (d, th, y)]
        return lib.cwr_set_kinetics(be._h, *[p(a) for a in arrs], tk, tc)

    assert call(ok_d, ok_th, ok_y, 2) == 0
    cyc = ok_y.copy(); cyc[1, 0] = 1.0; cyc[0, 1] = 1.0
    selfy = ok_y.copy(); selfy[0, 0] = 0.5
    nany = ok_y.copy(); nany[1, 0] = nan
    to_t = ok_y.copy(); to_t[2, 0] = 1.0
    bad = [
        ([-1.0, 1.0, 0.0], None, None, -1, 20.0), ([nan, 1.0, 0.0], None, None, -1, 20.0), ([np.inf, 1.0, 0.0], None, None, -1, 20.0),
        (ok_d, [0.0, 1.0, 1.0], None, -1, 20.0), (ok_d, [-1.0, 1.0, 1.0], None, -1, 20.0), (ok_d, [np.inf, 1.0, 1.0], None, -1, 20.0),
        (ok_d, None, nany, -1, 20.0), (ok_d, None, selfy, -1, 20.0), (ok_d, None, cyc, -1, 20.0),
        ([1.0, 1.0, 1.0], None, None, 2, 20.0), (ok_d, None, to_t, 2, 20.0),
        (ok_d, None, None, 3, 20.0), (ok_d, None, None, -2, 20.0), (ok_d, None, None, -1, nan),
    ]
    for args in bad:
        assert call(*args) == CWR_EINVAL, args
        with pytest.raises(ValueError):
            be.set_kinetics(*args)
    be.close()


def _gpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_domain_decomposition_with_kinetics():
    if _gpus() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29531", str(ROOT / "tools" / "dd_check.py"), "--side", "150", "--K", "4", "--steps", "5", "--kinetics"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=850, cwd=ROOT)
    lines = [json.loads(ln) for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert out.returncode == 0, (out.stdout[-3000:], out.stderr[-3000:])
    assert len(lines) >= 4 and all(ln["ok"] for ln in lines), lines
    for ln in lines:
        assert ln["max_rel_diff_vs_oracle"] < 1e-9 and ln["max_rel_diff_vs_single_gpu"] < 1e-9
        assert ln["reaction_mass_rel_diff"] < 1e-9
