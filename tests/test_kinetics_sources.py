"""Zero-order sources and relaxation toward an equilibrium in the device step (cwr_set_kinetics_sources): the spec
compiler, the oxygen saturation and the numpy restatement (oracle.kinetics_sources) on the CPU, the CUDA path against
the restatement on the GPU.  GPU tolerance as in test_kinetics: rtol 1e-9 per step."""
import ctypes as C
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from oracle import kinetics as first_order
from oracle import reference_step as ref
from oracle.kinetics_sources import KineticsRiverine, o2sat, react
from tests.helpers import same

ROOT = Path(__file__).resolve().parents[1]
RTOL = 1e-9
SPEC = {"BOD": {"decay_per_day": 0.35, "theta": 1.047, "yields": {"DO": -1.0}},
        "DO": {"source_per_day": -1.5, "source_theta": 1.065, "exchange_per_day": 0.7, "exchange_theta": 1.024,
               "equilibrium": "oxygen_saturation"},
        "T": {"source_per_day": 0.2, "exchange_per_day": 0.3, "equilibrium": 18.0}}
# Streeter-Phelps closed box (every quantity of the analytic sag): decay, reaeration, initial BOD
KD, KA, L0 = 0.35, 0.7, 20.0


def sag(t_seconds, L0, kd=KD, ka=KA):
    """DO of the Streeter-Phelps sag from DO0 = O2sat(20 deg C): O2sat - kd L0 / (ka - kd) (e^(-kd t) - e^(-ka t))."""
    d = np.asarray(t_seconds, np.float64) / 86400.0
    return o2sat(20.0) - kd * np.asarray(L0) / (ka - kd) * (np.exp(-kd * d) - np.exp(-ka * d))


# ------------------------------------------------------------------------------------------------------------------
# CPU: spec compiler and the oxygen saturation
# ------------------------------------------------------------------------------------------------------------------
def test_spec_compiles_the_new_keys_to_the_abi_arrays():
    from clearwater_riverine_b200.kinetics import compile_kinetics
    names = ["DO", "BOD", "T", "X"]
    kin = compile_kinetics(SPEC, names, "T")
    assert kin.source_per_day.tolist() == [-1.5, 0.0, 0.2, 0.0]
    assert kin.source_theta.tolist() == [1.065, 1.0, 1.0, 1.0]
    assert kin.exchange_per_day.tolist() == [0.7, 0.0, 0.3, 0.0]
    assert kin.exchange_theta.tolist() == [1.024, 1.0, 1.0, 1.0]
    assert kin.equilibrium.tolist() == [0.0, 0.0, 18.0, 0.0]
    assert kin.equilibrium_kind.tolist() == [1, 0, 0, 0] and kin.equilibrium_kind.dtype == np.int32
    assert kin.decay_per_day.tolist() == [0.0, 0.35, 0.0, 0.0] and kin.yields[0, 1] == -1.0
    assert kin.has_sources
    args = kin.sources_arguments()
    assert sorted(args) == ["equilibrium", "equilibrium_kind", "exchange_per_day", "exchange_theta", "source_per_day",
                            "source_theta"]
    plain = compile_kinetics({"BOD": SPEC["BOD"]}, names, 12.0)
    assert not plain.has_sources and (plain.source_theta == 1).all() and (plain.equilibrium_kind == 0).all()


def test_kinetics_built_without_the_new_fields_has_no_sources():
    from clearwater_riverine_b200.kinetics import Kinetics
    kin = Kinetics(np.zeros(2), np.ones(2), np.zeros((2, 2)), -1, 20.0, (0, 1))
    assert not kin.has_sources and kin.source_per_day is None


INVALID = {
    "oxygen saturation on the temperature constituent": ({"T": {"exchange_per_day": 1.0, "equilibrium": "oxygen_saturation"}}, "T"),
    "exchange without equilibrium": ({"A": {"exchange_per_day": 1.0}}, 20.0),
    "unknown equilibrium name": ({"A": {"exchange_per_day": 1.0, "equilibrium": "saturation"}}, 20.0),
    "non-finite equilibrium": ({"A": {"exchange_per_day": 1.0, "equilibrium": float("inf")}}, 20.0),
    "non-finite source": ({"A": {"source_per_day": float("nan")}}, 20.0),
    "negative exchange": ({"A": {"exchange_per_day": -0.1, "equilibrium": 1.0}}, 20.0),
    "non-finite exchange": ({"A": {"exchange_per_day": float("inf"), "equilibrium": 1.0}}, 20.0),
    "zero source theta": ({"A": {"source_per_day": 1.0, "source_theta": 0.0}}, 20.0),
    "negative exchange theta": ({"A": {"exchange_per_day": 1.0, "exchange_theta": -1.02, "equilibrium": 1.0}}, 20.0),
    "non-finite source theta": ({"A": {"source_per_day": 1.0, "source_theta": float("inf")}}, 20.0),
    "unknown key": ({"A": {"source": 1.0}}, 20.0),
}


@pytest.mark.parametrize("case", sorted(INVALID))
def test_invalid_source_specs_are_rejected_naming_the_constituent(case):
    from clearwater_riverine_b200.kinetics import compile_kinetics
    spec, temperature = INVALID[case]
    with pytest.raises(ValueError, match="'A'|'T'"):
        compile_kinetics(spec, ["A", "B", "T"], temperature)


def test_validate_rejects_a_kind_other_than_0_or_1():
    from clearwater_riverine_b200.kinetics import validate
    with pytest.raises(ValueError, match="kind"):
        validate(np.zeros(2), np.ones(2), np.zeros((2, 2)), -1, 20.0, ("A", "B"), exchange_per_day=np.ones(2),
                 equilibrium=np.zeros(2), equilibrium_kind=np.array([0, 2]))


def test_oxygen_saturation_matches_the_table():
    from clearwater_riverine_b200.kinetics import oxygen_saturation
    T = np.array([0.0, 10.0, 20.0, 30.0, 40.0])
    table = np.array([14.621, 11.288, 9.092, 7.559, 6.413])
    assert np.abs(oxygen_saturation(T) - table).max() <= 1e-3
    assert np.abs(oxygen_saturation(T) - o2sat(T)).max() <= 1e-10 * table.max()     # Horner form against the written one
    assert abs(float(oxygen_saturation(20.0)) - 9.092) <= 1e-3


# ------------------------------------------------------------------------------------------------------------------
# CPU: the numpy restatement
# ------------------------------------------------------------------------------------------------------------------
def test_exchange_alone_is_exact_after_many_steps():
    rng = np.random.default_rng(0)
    c0 = 20.0 * rng.random((1, 40))
    ceq, ka, dt, steps = 8.5, 2.0, 600.0, 500
    c = c0
    for _ in range(steps):
        c = react(c, dt, [0.0], exchange_per_day=[ka], equilibrium=[ceq])
    want = ceq + (c0 - ceq) * np.exp(-ka / 86400.0 * dt * steps)
    assert np.abs(c - want).max() <= 1e-12 * 20.0


def test_source_alone_is_linear_in_time():
    c0 = np.array([[3.0, -1.0, 50.0]])
    c = c0
    for _ in range(100):
        c = react(c, 60.0, [0.0], source_per_day=[-4.0])
    assert np.abs(c - (c0 - 4.0 * 100 * 60.0 / 86400.0)).max() <= 1e-13 * 50.0


def test_theta_corrects_the_rates():
    c0 = np.array([[2.0, 7.0], [0.0, 0.0]])
    T, dt = 27.0, 900.0
    got = react(c0, dt, [0.0, 0.0], source_per_day=[0.0, 3.0], source_theta=[1.0, 1.08], exchange_per_day=[1.5, 0.0],
                exchange_theta=[1.024, 1.0], equilibrium=[4.0, 0.0], temperature=T)
    r = 1.5 * 1.024 ** (T - 20.0) / 86400.0
    assert np.abs(got[0] - (4.0 + (c0[0] - 4.0) * np.exp(-r * dt))).max() <= 1e-14
    assert np.abs(got[1] - 3.0 * 1.08 ** (T - 20.0) * dt / 86400.0).max() <= 1e-15
    # at 20 deg C theta does nothing
    a = react(c0, dt, [0.0, 0.0], source_per_day=[0.0, 3.0], source_theta=[1.0, 1.08], temperature=20.0)
    b = react(c0, dt, [0.0, 0.0], source_per_day=[0.0, 3.0], temperature=20.0)
    assert same(a, b)


def test_oxygen_saturation_follows_the_temperature_constituent_before_the_reactions():
    """DO relaxes toward O2sat of the cell's temperature as it was before the step, although the temperature itself
    relaxes toward 25 deg C in the same step."""
    c0 = np.array([[5.0, 6.0], [10.0, 30.0]])        # DO, T
    dt = 3600.0
    got = react(c0, dt, [0.0, 0.0], exchange_per_day=[3.0, 2.0], equilibrium=[0.0, 25.0], equilibrium_kind=[1, 0],
                temperature=1, temperature_is_index=True)
    r = 3.0 / 86400.0
    assert np.abs(got[0] - (o2sat(c0[1]) + (c0[0] - o2sat(c0[1])) * np.exp(-r * dt))).max() <= 1e-13
    assert np.abs(got[1] - (25.0 + (c0[1] - 25.0) * np.exp(-2.0 / 86400.0 * dt))).max() <= 1e-13


def test_all_zero_sources_are_bitwise_react_without_them():
    rng = np.random.default_rng(2)
    K = 4
    c = 50.0 * rng.random((K, 30)); c[3] = 10.0 + 20.0 * rng.random(30)
    decay = np.array([3.0, 1.0, 0.5, 0.0]); theta = np.array([1.05, 1.02, 1.08, 1.0])
    y = np.zeros((K, K)); y[1, 0] = 1.0; y[2, 1] = -0.5
    base = first_order.react(c, 900.0, decay, theta, y, 3, True)
    zero = react(c, 900.0, decay, theta, y, 3, True, source_per_day=np.zeros(K), source_theta=np.full(K, 1.1),
                 exchange_per_day=np.zeros(K), exchange_theta=np.full(K, 1.1), equilibrium=np.full(K, np.nan),
                 equilibrium_kind=np.ones(K, int))
    assert same(base, zero) and same(base, react(c, 900.0, decay, theta, y, 3, True))


def streeter_phelps_box(dt, days=10.0, L0=L0):
    """BOD and DO of one closed box, stepped with the restatement: the DO on the last day."""
    steps = int(round(days * 86400.0 / dt))
    c = np.array([[L0], [float(o2sat(20.0))]])
    y = np.array([[0.0, 0.0], [-1.0, 0.0]])
    for _ in range(steps):
        c = react(c, dt, [KD, 0.0], None, y, 20.0, exchange_per_day=[0.0, KA], equilibrium=[0.0, 0.0],
                  equilibrium_kind=[0, 1])
    return c[1, 0], steps * dt


def test_closed_box_streeter_phelps_converges_at_first_order():
    do900, t = streeter_phelps_box(900.0)
    err900 = abs(do900 - sag(t, L0))
    do450, _ = streeter_phelps_box(450.0)
    err450 = abs(do450 - sag(t, L0))
    assert err900 <= 3e-3, err900
    assert 1.9 <= err900 / err450 <= 2.1, (err900, err450)


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def _tk():
    from tests import test_kinetics as tk
    return tk


def source_backend(mesh, inputs, kin, src, **opt):
    be = _tk().kinetic_backend(mesh, inputs, kin, **opt)
    if src is not None:
        be.set_kinetics_sources(**src)
    return be


def source_oracle(mesh, inputs, kin, src):
    temperature = f"c{kin['temperature_k']}" if kin["temperature_k"] >= 0 else kin["temperature_c"]
    return KineticsRiverine(mesh, {f"c{k}": inputs[k] for k in range(len(inputs))}, kin["decay_per_day"], kin["theta"],
                            kin["yields"], temperature, **(src or {}))


def run_source_parity(mesh, inputs, kin, src, steps, overrides=None, check_flux=True, **opt):
    tp, tk = _tk()._parity(), _tk()
    K = len(inputs)
    be = source_backend(mesh, inputs, kin, src, **opt)
    oracle = source_oracle(mesh, inputs, kin, src)
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
    scale = np.maximum(np.abs(want), tk.mass_scale(mesh, inputs))
    assert (np.abs(got - want) <= RTOL * scale).all(), (got, want)
    return be, oracle


def synthetic_network(nx, ny, T, K, seed, **kw):
    from clearwater_riverine_b200 import synthetic
    _, mesh, inputs = _tk()._parity().synthetic_case(nx, ny, T, K, seed=seed, **kw)
    inputs, kin = synthetic.make_kinetics(inputs, seed=seed)
    return mesh, inputs, kin, synthetic.make_kinetics_sources(kin, seed=seed)


@pytest.mark.gpu
def test_golden_mesh_parity_with_overrides():
    from clearwater_riverine_b200 import synthetic
    g, mesh, inputs, kin = _tk().golden_kinetic_case()
    src = synthetic.make_kinetics_sources(kin, seed=3, rate_range=(2000.0, 20000.0))   # dt = 1 s here
    n = mesh.n
    overrides = {3: {"c1": 40.0 + np.arange(n, dtype=np.float64)}, 9: {"c0": np.full(n, 7.0), "c3": np.linspace(15, 25, n)}}
    be, _ = run_source_parity(mesh, inputs, kin, src, 30, overrides)
    be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("solver", [1, 2])
@pytest.mark.parametrize("K", [1, 3, 16, 18, 19, 33])
def test_synthetic_meshes_on_the_large_path(K, solver):
    mesh, inputs, kin, src = synthetic_network(40, 25, 8, K, seed=K + 50, dry_fraction=0.02)
    be, _ = run_source_parity(mesh, inputs, kin, src, 7, solver_path=1, solver=solver)
    be.close()


@pytest.mark.gpu
def test_every_column_count_up_to_kmax():
    """With source columns at a constant temperature (K < 4) k_react takes shared memory beyond its 48 KB tile: one
    step per K on both paths, against the restatement."""
    from clearwater_riverine_b200 import synthetic
    _, mesh, base = _tk()._parity().synthetic_case(12, 9, 3, 128, seed=91)
    for K in range(1, 129):
        inputs, kin = synthetic.make_kinetics(base[:K], seed=K)
        src = synthetic.make_kinetics_sources(kin, seed=K)
        for solver_path in (1, 2):
            be, _ = run_source_parity(mesh, inputs, kin, src, 1, check_flux=False, solver_path=solver_path)
            be.close()


@pytest.mark.gpu
def test_constant_temperature_with_every_column_a_source():
    """The largest constant-temperature coefficient table: K = 128 columns, every one with a source and an exchange."""
    from clearwater_riverine_b200 import synthetic
    _, mesh, inputs = _tk()._parity().synthetic_case(12, 9, 3, 128, seed=92)
    inputs, kin = synthetic.make_kinetics(inputs, seed=92)
    kin = dict(kin, temperature_k=-1, temperature_c=14.0)
    rng = np.random.default_rng(5)
    src = dict(source_per_day=100.0 * (rng.random(128) - 0.5), exchange_per_day=20.0 + 100.0 * rng.random(128),
               exchange_theta=np.full(128, 1.024), equilibrium=40.0 * rng.random(128),
               equilibrium_kind=(np.arange(128) % 3 == 0).astype(np.int32))
    for solver_path in (1, 2):
        be, _ = run_source_parity(mesh, inputs, kin, src, 2, check_flux=False, solver_path=solver_path)
        be.close()


@pytest.mark.gpu
def test_small_path_parity():
    mesh, inputs, kin, src = synthetic_network(40, 25, 7, 5, seed=61, dry_fraction=0.02)
    be, _ = run_source_parity(mesh, inputs, kin, src, 6, solver_path=2, precond_sweep=0)
    assert be.options.solver_path == 2
    be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 64])
def test_on_chip_path_on_the_ohio_shaped_mesh(K):
    """K = 1 (reaeration of one DO column), and 64 scenarios of one constituent with 64 different exchange rates."""
    from clearwater_riverine_b200 import synthetic
    plan = synthetic.ohio_like(7, seed=2)
    D = 0.1
    adv, _, _, cdiff, dt = ref.derive_coefficients(plan.face_flow, plan.edge_velocity, plan.face_x, plan.face_y, plan.f1, plan.f2,
                                                   D, plan.time_seconds)
    mesh = ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, plan.edge_velocity, plan.volume, dt, D)
    inputs = synthetic.make_inputs(plan, K, seed=7, ic_range=(0.0, 15.0))
    kin = dict(decay_per_day=np.full(K, 0.35), theta=np.full(K, 1.047), yields=None, temperature_k=-1, temperature_c=17.0)
    src = dict(source_per_day=np.full(K, -1.5), source_theta=np.full(K, 1.065), exchange_per_day=np.linspace(0.1, 6.0, K),
               exchange_theta=np.full(K, 1.024), equilibrium=np.zeros(K), equilibrium_kind=np.ones(K, np.int32))
    be, _ = run_source_parity(mesh, inputs, kin, src, 6, check_flux=K == 1)
    assert be.options.solver_path in (3, 4)
    be.close()


def closed_boxes(temperature_constituent: bool, dt=900.0, days=10.0):
    """Zero face flow, D = 0 and a constant volume: every cell is a closed box.  Constituents BOD (L0 from 5 to 35 per
    cell) and DO (from O2sat(20)), and with temperature_constituent a third one held at 20 deg C."""
    from clearwater_riverine_b200 import synthetic
    steps = int(round(days * 86400.0 / dt))
    plan = synthetic.make_plan(8, 6, steps + 1, dt=dt, seed=13)
    flow, vel = np.zeros_like(plan.face_flow), np.zeros_like(plan.edge_velocity)
    vol = np.repeat(plan.volume[:1], plan.n_time, axis=0)
    adv, _, _, cdiff, dts = ref.derive_coefficients(flow, vel, plan.face_x, plan.face_y, plan.f1, plan.f2, 0.0, plan.time_seconds)
    mesh = ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, vel, vol, dts, 0.0)
    n = plan.n_real
    K = 3 if temperature_constituent else 2
    inputs = np.zeros((K, plan.n_time, plan.n_face))
    L0s = np.linspace(5.0, 35.0, n)
    inputs[0, 0, :n] = L0s
    inputs[1, 0, :n] = float(o2sat(20.0))
    if temperature_constituent:
        inputs[2, 0, :n] = 20.0
    y = np.zeros((K, K)); y[1, 0] = -1.0
    kin = dict(decay_per_day=np.array([KD] + [0.0] * (K - 1)), theta=np.full(K, 1.047), yields=y,
               temperature_k=2 if temperature_constituent else -1, temperature_c=20.0)
    src = dict(exchange_per_day=np.array([0.0, KA] + [0.0] * (K - 2)), exchange_theta=np.full(K, 1.024),
               equilibrium=np.zeros(K), equilibrium_kind=np.array([0, 1] + [0] * (K - 2), np.int32))
    return plan, mesh, inputs, kin, src, L0s, steps


@pytest.mark.gpu
@pytest.mark.parametrize("temperature_constituent", [False, True])
def test_closed_box_streeter_phelps_on_the_device(temperature_constituent):
    plan, mesh, inputs, kin, src, L0s, steps = closed_boxes(temperature_constituent)
    n = plan.n_real
    be = source_backend(mesh, inputs, kin, src)
    assert be.run(0, steps).status == 0
    got_bod, got_do = be.get_state(0, steps)[:n], be.get_state(1, steps)[:n]
    oracle = source_oracle(mesh, inputs, kin, src)
    for _ in range(steps):
        oracle.update()
    tp = _tk()._parity()
    tp.close(got_bod, oracle.constituent_dict["c0"].concentration[steps][:n], RTOL, "BOD")
    tp.close(got_do, oracle.constituent_dict["c1"].concentration[steps][:n], RTOL, "DO")
    t = steps * 900.0
    assert np.abs(got_bod - L0s * np.exp(-KD * t / 86400.0)).max() <= 1e-9 * L0s.max()
    err = np.abs(got_do - sag(t, L0s))
    assert (err <= 3e-3 * L0s / L0).all(), err.max()      # the splitting error of the 900 s step, linear in L0
    be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("temperature_k", [-1, 3])
@pytest.mark.parametrize("solver_path", [1, 2])
def test_zero_sources_are_bitwise_kinetics_without_them(solver_path, temperature_k):
    """All-zero source and exchange rates: the same bits and the same launches as no sources; cwr_set_kinetics after
    cwr_set_kinetics_sources: the same bits as a run that never set sources."""
    mesh, inputs, kin, src = synthetic_network(40, 25, 7, 4, seed=71, dry_fraction=0.02)
    kin = dict(kin, temperature_k=temperature_k)
    zero_src = dict(src, source_per_day=np.zeros(4), exchange_per_day=np.zeros(4))
    plain = source_backend(mesh, inputs, kin, None, solver_path=solver_path)
    zero = source_backend(mesh, inputs, kin, zero_src, solver_path=solver_path)
    cleared = source_backend(mesh, inputs, kin, src, solver_path=solver_path)
    cleared.set_kinetics(**kin)
    for t in range(6):
        a, b, c = plain.step(t), zero.step(t), cleared.step(t)
        assert b.n_launches == a.n_launches and c.n_launches == a.n_launches
        assert same(plain.get_state_all(t + 1), zero.get_state_all(t + 1))
        assert same(plain.get_state_all(t + 1), cleared.get_state_all(t + 1))
        for k in range(4):
            assert all(same(x, y) for x, y in zip(plain.get_mass_flux(k, t), zero.get_mass_flux(k, t)))
    assert all(zero.reaction_mass(k) == plain.reaction_mass(k) == cleared.reaction_mass(k) for k in range(4))
    for be in (plain, zero, cleared):
        be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("solver_path", [1, 2])
def test_run_is_bitwise_step_by_step_and_repeatable(solver_path):
    mesh, inputs, kin, src = synthetic_network(30, 20, 10, 5, seed=81, dry_fraction=0.02)
    outs = []
    for mode in ("step", "run", "run"):
        be = source_backend(mesh, inputs, kin, src, solver_path=solver_path)
        if mode == "step":
            for t in range(9):
                assert be.step(t).status == 0
        else:
            assert be.run(0, 9).status == 0
        outs.append((np.stack([be.get_state_all(t) for t in range(1, 10)]), [be.reaction_mass(k) for k in range(5)]))
        be.close()
    for states, masses in outs[1:]:
        assert same(states, outs[0][0]) and masses == outs[0][1]
    oracle = source_oracle(mesh, inputs, kin, src)
    for _ in range(9):
        oracle.update()
    for k in range(5):
        _tk()._parity().close(outs[1][0][-1][k], oracle.constituent_dict[f"c{k}"].concentration[9][:mesh.n], RTOL, f"run k{k}")


@pytest.mark.gpu
def test_reaction_mass_counts_the_sources_once_under_the_defect_correction_fallback():
    """test_kinetics's fallback setup with sources: the sweeps diverge, the step forms its right-hand side again and
    solves with BiCGSTAB; the source and exchange mass of that step is counted once."""
    from clearwater_riverine_b200 import synthetic
    plan = synthetic.make_plan(60, 50, 6, seed=41, dry_fraction=0.02)
    vel = plan.edge_velocity.copy()
    vel[:, np.random.default_rng(1).random(plan.n_edge) < 0.05] *= -1
    D = 2.0
    adv, _, _, cdiff, dt = ref.derive_coefficients(plan.face_flow, vel, plan.face_x, plan.face_y, plan.f1, plan.f2, D, plan.time_seconds)
    mesh = ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, vel, plan.volume, dt, D)
    inputs = synthetic.make_inputs(plan, 3, seed=41)
    inputs, kin = synthetic.make_kinetics(inputs, seed=41)
    kin = dict(kin, decay_per_day=np.zeros(3))           # the reaction mass is the sources' and the exchange's alone
    src = synthetic.make_kinetics_sources(kin, seed=41)
    tp, tk = _tk()._parity(), _tk()
    be = source_backend(mesh, inputs, kin, src, solver_path=1, solver=2)
    oracle = source_oracle(mesh, inputs, kin, src)
    for t in range(3):
        assert be.step(t).status == 0
        oracle.update()
        for k in range(3):
            tp.close(be.get_state(k, t + 1), oracle.constituent_dict[f"c{k}"].concentration[t + 1], 1e-8, f"fallback k{k} t{t}")
        want = np.sum(oracle.reaction_mass, axis=0)
        assert (want != 0).all()
        for k in range(3):
            assert abs(be.reaction_mass(k) - want[k]) <= RTOL * max(abs(want[k]), tk.mass_scale(mesh, inputs)[k]), (t, k)
    assert be.solver_stats()[1] >= 1, "the sweeps diverge on this matrix: the solver should have fallen back"
    be.close()


@pytest.mark.gpu
def test_mass_balance_closes_with_sources():
    """ClearwaterRiverine with a BOD-DO-SOD-temperature spec against the restatement: the concentrations, and
    mass_balance() closing with the reaction mass that now includes the sources and the exchange."""
    from clearwater_riverine_b200 import ClearwaterRiverine
    from clearwater_riverine_b200.kinetics import compile_kinetics
    tp = _tk()._parity()
    plan, mesh, inputs = tp.synthetic_case(20, 14, 8, 3, seed=4)
    names = ["BOD", "DO", "T"]
    inputs[2] = np.where(inputs[2] != 0, 10.0 + 0.2 * inputs[2], 0.0)
    spec = {"BOD": {"decay_per_day": 150.0, "theta": 1.047, "yields": {"DO": -1.0}},
            "DO": {"source_per_day": -400.0, "source_theta": 1.065, "exchange_per_day": 300.0, "exchange_theta": 1.024,
                   "equilibrium": "oxygen_saturation"},
            "T": {"source_per_day": 20.0, "exchange_per_day": 100.0, "equilibrium": 18.0}}
    arrays = (plan.f1, plan.f2, plan.face_x, plan.face_y, plan.time_seconds, plan.face_flow, plan.edge_velocity, plan.volume, 0.1)
    model = ClearwaterRiverine.from_arrays(*arrays, dict(zip(names, inputs)), kinetics=spec, temperature="T")
    kin = compile_kinetics(spec, names, "T")
    oracle = KineticsRiverine(mesh, dict(zip(names, inputs)), kin.decay_per_day, kin.theta, kin.yields, "T",
                              **kin.sources_arguments())
    for t in range(7):
        model.update()
        oracle.update()
        for name in names:
            tp.close(model.mesh[name][t + 1], oracle.constituent_dict[name].concentration[t + 1], RTOL, f"{name} {t}")
    faces = {nm: plan.boundary_faces[nm] for nm in ("upstream", "downstream")}
    for k, name in enumerate(names):
        got = model.mass_balance(name, faces)
        con = oracle.constituent_dict[name]
        want = ref.mass_balance(mesh, con.concentration, con.total_mass_flux, plan.face_flow, faces)
        reaction = float(np.sum(oracle.reaction_mass, axis=0)[k])
        assert reaction != 0.0
        assert abs(got["reaction_mass"] - reaction) <= RTOL * abs(want["Mass_start"])
        assert abs(got["error_mass"] - (want["mass_end_calc"] + reaction - want["Mass_end"])) <= RTOL * abs(want["Mass_start"])
    model.finalize()


@pytest.mark.gpu
def test_yaml_config_with_source_keys_is_bitwise_from_arrays(tmp_path):
    yaml = pytest.importorskip("yaml")
    import pandas as pd
    from clearwater_riverine_b200 import ClearwaterRiverine
    from clearwater_riverine_b200.io import ras
    from tests.helpers import load_golden
    from tests.ras_fixture import write_plan
    g = load_golden("p01_random_two")
    hdf = tmp_path / "plan.hdf"
    times = write_plan(hdf, g)
    plan = ras.read_ras_plan(hdf)
    n = plan.nreal + 1
    lines = sorted({str(x) for x in g["bc_names"]})
    cons = {}
    for name, ic, bc in (("BOD", 8.0, 5.0), ("DO", 7.0, 8.0), ("T", 18.0, 21.0)):
        icf, bcf = tmp_path / f"{name}_ic.csv", tmp_path / f"{name}_bc.csv"
        pd.DataFrame({"Cell_Index": np.arange(n), "Concentration": ic + 0.01 * np.arange(n)}).to_csv(icf, index=False)
        pd.DataFrame({"Datetime": np.repeat([times[0], times[-1]], len(lines)), "RAS2D_TS_Name": lines * 2,
                      "Concentration": bc}).to_csv(bcf, index=False)
        cons[name] = {"initial_conditions": str(icf), "boundary_conditions": str(bcf), "units": "mg/L"}
    spec = {"BOD": {"decay_per_day": 900.0, "theta": 1.047, "yields": {"DO": -1.0}},
            "DO": {"source_per_day": -2000.0, "source_theta": 1.065, "exchange_per_day": 1500.0, "exchange_theta": 1.024,
                   "equilibrium": "oxygen_saturation"},
            "T": {"exchange_per_day": 500.0, "equilibrium": 25.0}}
    cfg = {"diffusion_coefficient": 0.1, "flow_field_filepath": str(hdf), "temperature": "T",
           "constituents": {name: dict(c, kinetics=spec[name]) for name, c in cons.items()}}
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
    assert a.kinetics.has_sources and a.backend.reaction_mass(a._index["T"]) != 0.0
    a.finalize(); b.finalize()


@pytest.mark.gpu
def test_invalid_sources_straight_to_the_abi_return_einval():
    from clearwater_riverine_b200.backend import CWR_EINVAL
    _, mesh, inputs = _tk()._parity().synthetic_case(12, 9, 4, 3, seed=2)
    be = _tk()._parity().make_backend(mesh, list(inputs))
    lib = be._lib
    nan, inf = float("nan"), float("inf")

    def call(s=None, sth=None, e=None, eth=None, eq=None, kind=None):
        arrs = [None if a is None else np.ascontiguousarray(a, np.float64) for a in (s, sth, e, eth, eq)]
        kd = None if kind is None else np.ascontiguousarray(kind, np.int32)
        p = [None if a is None else a.ctypes.data_as(C.POINTER(C.c_double)) for a in arrs]
        return lib.cwr_set_kinetics_sources(be._h, *p, None if kd is None else kd.ctypes.data_as(C.POINTER(C.c_int32)))

    ok = dict(s=[1.0, -1.0, 0.0], e=[0.5, 0.0, 0.2], eq=[3.0, nan, 20.0], kind=[1, 0, 0])
    assert call(**ok) == CWR_EINVAL                           # kinetics not set
    be.set_kinetics(np.zeros(3), None, None, 2)               # all-zero decay, temperature constituent 2
    assert call(**ok) == 0 and call() == 0 and call(s=[0.0, 0.0, 1.0]) == 0
    bad = [
        dict(ok, s=[nan, 0.0, 0.0]), dict(ok, s=[inf, 0.0, 0.0]),
        dict(ok, sth=[0.0, 1.0, 1.0]), dict(ok, sth=[nan, 1.0, 1.0]), dict(ok, eth=[1.0, -1.0, 1.0]), dict(ok, eth=[1.0, inf, 1.0]),
        dict(ok, e=[-0.5, 0.0, 0.2]), dict(ok, e=[nan, 0.0, 0.2]), dict(ok, e=[inf, 0.0, 0.2]),
        dict(ok, kind=[2, 0, 0]), dict(ok, kind=[-1, 0, 0]),
        dict(ok, eq=None), dict(ok, eq=[3.0, 0.0, nan]), dict(ok, eq=[3.0, 0.0, inf]),
        dict(ok, kind=[1, 0, 1]), dict(s=[0.0, 0.0, 1.0], kind=[0, 0, 1]),
    ]
    for args in bad:
        assert call(**args) == CWR_EINVAL, args
        with pytest.raises(ValueError):
            be.set_kinetics_sources(*[args.get(x) for x in ("s", "sth", "e", "eth", "eq", "kind")])
    be.set_kinetics(None)
    assert call(**ok) == CWR_EINVAL                           # kinetics switched off again
    be.close()


def _gpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_domain_decomposition_with_sources():
    if _gpus() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", str(ROOT / "tools" / "dd_check.py"), "--side", "150", "--K", "4", "--steps", "5", "--kinetics"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=850, cwd=ROOT)
    lines = [json.loads(ln) for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert out.returncode == 0, (out.stdout[-3000:], out.stderr[-3000:])
    runs = [ln for ln in lines if ln.get("sources")]
    assert len(runs) >= 2 and all(ln["ok"] for ln in lines), lines
    for ln in runs:
        assert ln["max_rel_diff_vs_oracle"] < 1e-9 and ln["max_rel_diff_vs_single_gpu"] < 1e-9
        assert ln["reaction_mass_rel_diff"] < 1e-9
