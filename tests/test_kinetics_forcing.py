"""Time-varying forcing of the device kinetics (cwr_set_kinetics_forcing): series of one value per model time index that
replace the constant temperature or an equilibrium, or scale a decay, source or exchange rate.  The spec compiler, the
config-file series and the numpy oracle (oracle.kinetics_forcing) on the CPU, with a closed-box diurnal DO case against
scipy's solve_ivp; the CUDA path against the oracle on the GPU (rtol 1e-9 per step, as test_kinetics)."""
import ctypes as C
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from oracle import reference_step as ref
from oracle.kinetics_forcing import KineticsRiverine, forcing_terms
from oracle.kinetics_depth import depth_terms
from oracle.kinetics_limits import limit_terms
from oracle.kinetics_sources import o2sat
from tests.helpers import same

ROOT = Path(__file__).resolve().parents[1]
RTOL = 1e-9
NAMES = ["DO", "BOD", "T"]


def _spec(T):
    t = np.arange(T, dtype=np.float64)
    return {"BOD": {"decay_per_day": 0.3, "theta": 1.047, "yields": {"DO": -1.0}, "decay_scale": 0.5 + 0.5 * np.cos(t) ** 2},
            "DO": {"source_per_day": 4.0, "source_scale": np.maximum(np.sin(t), 0.0), "exchange_per_day": 1.2,
                   "exchange_scale": 1.0 + 0.3 * np.sin(t), "equilibrium": "oxygen_saturation"},
            "T": {"exchange_per_day": 0.5, "equilibrium": 18.0 + np.sin(t)}}


# ------------------------------------------------------------------------------------------------------------------
# CPU: spec compiler, validation, config-file series
# ------------------------------------------------------------------------------------------------------------------
def test_spec_compiles_the_series():
    from clearwater_riverine_b200.kinetics import compile_kinetics
    T = 7
    spec = _spec(T)
    kin = compile_kinetics(spec, NAMES, np.linspace(15.0, 21.0, T), n_time=T)
    assert kin.has_forcing and kin.temperature_k == -1 and kin.temperature_c == 15.0
    # ordered by (target, column): temperature, equilibrium of T, decay of BOD, source of DO, exchange of DO
    assert kin.forcing_target.tolist() == [0, 1, 2, 3, 4] and kin.forcing_column.tolist() == [-1, 2, 1, 0, 0]
    assert kin.forcing_target.dtype == np.int32 and kin.forcing_column.dtype == np.int32
    args = kin.forcing_arguments()
    assert args["values"].shape == (5, T) and args["values"].dtype == np.float64
    assert same(args["values"][0], np.linspace(15.0, 21.0, T)) and same(args["values"][1], spec["T"]["equilibrium"])
    assert same(args["values"][3], spec["DO"]["source_scale"])
    assert kin.equilibrium[2] == spec["T"]["equilibrium"][0] and kin.equilibrium_kind[2] == 0
    assert kin.source_per_day[0] == 4.0 and kin.decay_per_day[1] == 0.3
    by_name = compile_kinetics(spec, NAMES, "T", n_time=T)
    assert by_name.forcing_target.tolist() == [1, 2, 3, 4] and by_name.temperature_k == 2
    plain = compile_kinetics({"BOD": {"decay_per_day": 0.3}}, NAMES, 20.0)
    assert not plain.has_forcing and plain.forcing_arguments()["target"] is None


def test_n_time_defaults_to_the_series_length_and_lengths_must_agree():
    from clearwater_riverine_b200.kinetics import compile_kinetics
    kin = compile_kinetics({"BOD": {"decay_per_day": 0.3, "decay_scale": np.ones(4)}}, NAMES, np.full(4, 20.0))
    assert kin.forcing_values.shape == (2, 4)
    with pytest.raises(ValueError, match="temperature.*5 values"):              # the first series sets n_time
        compile_kinetics({"BOD": {"decay_per_day": 0.3, "decay_scale": np.ones(5)}}, NAMES, np.full(4, 20.0))
    with pytest.raises(ValueError, match="'BOD'.*6 values"):
        compile_kinetics({"BOD": {"decay_per_day": 0.3, "decay_scale": np.ones(5)}}, NAMES, 20.0, n_time=6)
    with pytest.raises(ValueError, match="'BOD'.*series"):
        compile_kinetics({"BOD": {"decay_per_day": 0.3, "decay_scale": 0.5}}, NAMES, 20.0, n_time=6)
    with pytest.raises(ValueError, match="'BOD'.*datetimes"):
        compile_kinetics({"BOD": {"decay_per_day": 0.3, "decay_scale": {"csv": "x.csv"}}}, NAMES, 20.0, n_time=6)


def test_kinetics_built_without_the_new_fields_has_no_forcing():
    from clearwater_riverine_b200.kinetics import Kinetics
    kin = Kinetics(np.zeros(2), np.ones(2), np.zeros((2, 2)), -1, 20.0, (0, 1))
    assert not kin.has_forcing and kin.forcing_arguments()["values"] is None


SPEC_REJECTIONS = {
    "'BOD'.*>= 0; time index 3": {"BOD": {"decay_per_day": 0.3, "decay_scale": [1.0, 1.0, 1.0, -0.5, 1.0]}},
    "'DO'.*finite; time index 2": {"DO": {"source_per_day": 1.0, "source_scale": [1.0, 1.0, np.nan, 1.0, 1.0]}},
    "'DO'.*its source rate is 0": {"DO": {"source_scale": np.ones(5)}},
    "'DO'.*its exchange rate is 0": {"DO": {"source_per_day": 1.0, "exchange_scale": np.ones(5)}},
    "'BOD'.*its decay rate is 0": {"BOD": {"decay_scale": np.ones(5)}},
    "'T'.*no exchange": {"T": {"equilibrium": np.full(5, 18.0)}},
    "'T'.*finite; time index 4": {"T": {"exchange_per_day": 1.0, "equilibrium": [18.0, 18.0, 18.0, 18.0, np.inf]}},
}


@pytest.mark.parametrize("match", sorted(SPEC_REJECTIONS))
def test_invalid_series_are_rejected_naming_the_constituent_and_time_index(match):
    from clearwater_riverine_b200.kinetics import compile_kinetics
    with pytest.raises(ValueError, match=match):
        compile_kinetics(SPEC_REJECTIONS[match], NAMES, 20.0, n_time=5)


def test_a_temperature_series_rejects_bad_values_naming_the_time_index():
    from clearwater_riverine_b200.kinetics import compile_kinetics
    with pytest.raises(ValueError, match="temperature series.*finite; time index 1"):
        compile_kinetics({}, NAMES, [20.0, np.nan, 20.0], n_time=3)


def test_validate_rejects_every_abi_condition():
    from clearwater_riverine_b200.kinetics import validate
    T = 4
    d, th, y = np.array([0.5, 0.0, 0.0]), np.ones(3), np.zeros((3, 3))
    srcs = dict(source_per_day=np.array([0.0, 2.0, 0.0]), exchange_per_day=np.array([0.0, 1.0, 3.0]),
                equilibrium=np.array([0.0, 0.0, 9.0]), equilibrium_kind=np.array([0, 1, 0], np.int32))
    names = ("A", "B", "C")

    def forcing(*rows, values=None):
        tg = np.array([r[0] for r in rows], np.int32)
        col = np.array([r[1] for r in rows], np.int32)
        v = np.ones((len(rows), T)) if values is None else np.asarray(values, np.float64)
        return dict(forcing_target=tg, forcing_column=col, forcing_values=v, n_time=T)

    ok = forcing((0, -1), (1, 2), (2, 0), (3, 1), (4, 1), (4, 2))
    validate(d, th, y, -1, 20.0, names, **srcs, **ok)
    bad = {"unknown target": forcing((5, 0)), "takes column -1": forcing((0, 0)), "out of range": forcing((2, 3)),
           "out of range ": forcing((1, -1)), "given twice": forcing((2, 0), (2, 0)),
           "'A'.*finite; time index 2": forcing((2, 0), values=[[1.0, 1.0, np.nan, 1.0]]),
           "'B'.*>= 0; time index 0": forcing((3, 1), values=[[-1.0, 1.0, 1.0, 1.0]]),
           "'B'.*its decay rate is 0": forcing((2, 1)), "'A'.*its source rate is 0": forcing((3, 0)),
           "'A'.*its exchange rate is 0": forcing((4, 0)), "'A'.*no exchange": forcing((1, 0)),
           "'B'.*oxygen_saturation": forcing((1, 1)), "4 values": dict(forcing((2, 0)), n_time=5),
           "time index 3": forcing((0, -1), values=[[20.0, 20.0, 20.0, np.inf]])}
    for what, args in bad.items():
        with pytest.raises(ValueError, match=what.strip()):
            validate(d, th, y, -1, 20.0, names, **srcs, **args)
    with pytest.raises(ValueError, match="'C' is the temperature constituent"):
        validate(d, th, y, 2, 20.0, names, **dict(srcs, equilibrium_kind=np.zeros(3, np.int32)), **forcing((0, -1)))
    # an equilibrium series may be negative (the non-negativity guarantee then does not cover that column)
    validate(d, th, y, -1, 20.0, names, **srcs, **forcing((1, 2), values=[[-1.0, 0.0, 1.0, 2.0]]))


def test_csv_series_are_put_onto_the_model_times_as_the_boundary_conditions_are(tmp_path):
    """A series in a CSV file with hourly Datetime / Value rows, one of them empty, on a model of 20-minute times starting
    half an hour after the first row: the last row at or before each model time (a backward merge_asof), the model times
    of the empty row filled linearly over the model index, against a hand-interpolated series; and the same is what
    build_input_array gives a boundary condition."""
    import pandas as pd
    from clearwater_riverine_b200.io import ras
    from clearwater_riverine_b200.kinetics import compile_kinetics, read_csv_series
    stamps = pd.date_range("2024-06-01 00:00", periods=8, freq="h")
    values = np.array([10.0, 12.0, 15.0, np.nan, 18.0, 16.0, 13.0, 11.0])
    f = tmp_path / "light.csv"
    pd.DataFrame({"Datetime": stamps, "Value": values}).to_csv(f, index=False)
    time = pd.date_range("2024-06-01 00:30", periods=16, freq="20min").to_numpy()
    hours = (time - stamps[0].to_datetime64()) / np.timedelta64(1, "h")
    asof = values[np.minimum(np.floor(hours).astype(int), 7)]
    idx = np.arange(len(time))
    want = np.where(np.isnan(asof), np.interp(idx, idx[~np.isnan(asof)], asof[~np.isnan(asof)]), asof)
    assert np.isnan(asof).sum() == 3
    got = ras.read_series_csv(f, time)
    assert np.allclose(got, want, rtol=0, atol=1e-12), (got, want)
    spec = {"DO": {"source_per_day": 2.0, "source_scale": {"csv": str(f)}}, "BOD": {"decay_per_day": 0.2}}
    spec2, temp = read_csv_series(spec, {"csv": str(f)}, time)
    assert same(spec2["DO"]["source_scale"], got) and same(temp, got) and spec2["BOD"] == spec["BOD"]
    kin = compile_kinetics(spec2, NAMES, temp, n_time=len(time))
    assert kin.forcing_target.tolist() == [0, 3] and same(kin.forcing_values[1], got)
    bc = pd.DataFrame({"Datetime": stamps, "RAS2D_TS_Name": "up", "Concentration": values})
    ic = pd.DataFrame({"Cell_Index": [0], "Concentration": [1.0]})
    bd = pd.DataFrame({"Name": ["up"], "Face Index": [0]})
    inp = ras.build_input_array(len(time), 3, time, np.array([2]), bd, ic, bc)
    assert same(inp[:, 2], got)
    with pytest.raises(ValueError, match="csv: path"):
        read_csv_series({"DO": {"source_scale": {"file": "x"}}}, 20.0, time)


# ------------------------------------------------------------------------------------------------------------------
# CPU: the oracle
# ------------------------------------------------------------------------------------------------------------------
def _small_network(K=6, T=6, seed=3, constant=False):
    from clearwater_riverine_b200 import synthetic
    from tests.test_kinetics_depth import synthetic_network
    plan, mesh, inputs, kin, src, lim, dep = synthetic_network(12, 9, T, K, seed=seed, dry_fraction=0.05)
    if constant:
        kin = dict(kin, temperature_k=-1, temperature_c=17.0)
    frc = synthetic.make_kinetics_forcing(kin, src, plan.time_seconds, seed=seed, period=5 * 30.0)
    return plan, mesh, inputs, kin, src, lim, dep, frc


def forcing_oracle(mesh, inputs, kin, src, lim, dep, frc):
    temperature = f"c{kin['temperature_k']}" if kin["temperature_k"] >= 0 else kin["temperature_c"]
    return KineticsRiverine(mesh, {f"c{k}": inputs[k] for k in range(len(inputs))}, kin["decay_per_day"], kin["theta"],
                            kin["yields"], temperature, **(src or {}), **limit_terms(**(lim or {})),
                            **depth_terms(**(dep or {})), **forcing_terms(**(frc or {})))


def identity_forcing(kin, src, T):
    """Every target at its identity: scales of 1, the constant temperature and the constant equilibria as series."""
    K = len(kin["decay_per_day"])
    rows = []
    if kin["temperature_k"] < 0:
        rows.append((0, -1, np.full(T, float(kin["temperature_c"]))))
    for k in range(K):
        if src["exchange_per_day"][k] > 0 and src["equilibrium_kind"][k] == 0:
            rows.append((1, k, np.full(T, float(src["equilibrium"][k]))))
        if kin["decay_per_day"][k] > 0:
            rows.append((2, k, np.ones(T)))
        if src["source_per_day"][k] != 0:
            rows.append((3, k, np.ones(T)))
        if src["exchange_per_day"][k] > 0:
            rows.append((4, k, np.ones(T)))
    return dict(target=np.array([r[0] for r in rows], np.int32), column=np.array([r[1] for r in rows], np.int32),
                values=np.stack([r[2] for r in rows]))


@pytest.mark.parametrize("constant", [False, True])
def test_identity_series_are_bitwise_the_unforced_oracle(constant):
    _, mesh, inputs, kin, src, lim, dep, frc = _small_network(constant=constant)
    ident = identity_forcing(kin, src, mesh.n_time)
    assert len(ident["target"]) >= 8
    runs = [forcing_oracle(mesh, inputs, kin, src, lim, dep, f) for f in (None, ident, frc)]
    for _ in range(5):
        for o in runs:
            o.update()
    for k in range(len(inputs)):
        a, b, c = (o.constituent_dict[f"c{k}"].concentration[5] for o in runs)
        assert same(a, b), k
    assert same(np.array(runs[0].reaction_mass), np.array(runs[1].reaction_mass))
    assert not same(np.array(runs[0].reaction_mass), np.array(runs[2].reaction_mass))
    assert same(runs[2].decay, kin["decay_per_day"])                      # the constants are restored after each step


def test_each_target_substitutes_into_the_parameters_of_its_step():
    """Step t of the forced oracle is the unforced oracle's step with the substituted constants."""
    from oracle.kinetics_depth import KineticsRiverine as Unforced
    _, mesh, inputs, kin, src, lim, dep, frc = _small_network(constant=True, T=4)
    forced = forcing_oracle(mesh, inputs, kin, src, lim, dep, frc)
    for t in range(3):
        d, s = np.array(kin["decay_per_day"], float), {k: np.array(v, float) if k != "equilibrium_kind" else v
                                                       for k, v in src.items()}
        temp = kin["temperature_c"]
        for g, k, v in zip(frc["target"], frc["column"], frc["values"]):
            if g == 0:
                temp = v[t]
            elif g == 1:
                s["equilibrium"][k] = v[t]
            elif g == 2:
                d[k] *= v[t]
            elif g == 3:
                s["source_per_day"][k] *= v[t]
            else:
                s["exchange_per_day"][k] *= v[t]
        one = Unforced(mesh, {f"c{k}": inputs[k] for k in range(len(inputs))}, d, kin["theta"], kin["yields"], temp, **s,
                       **limit_terms(**lim), **depth_terms(**dep))
        for k in range(len(inputs)):
            one.constituent_dict[f"c{k}"].concentration[t] = forced.constituent_dict[f"c{k}"].concentration[t].copy()
        one.time_step = t
        one.update()
        forced.update()
        for k in range(len(inputs)):
            assert same(one.constituent_dict[f"c{k}"].concentration[t + 1], forced.constituent_dict[f"c{k}"].concentration[t + 1])


# the closed-box diurnal DO case: BOD decays with yield -1 to DO (oxygen demand); DO has photosynthesis Pmax L(t) as its
# source and reaeration toward O2sat(T(t)), with hourly light and temperature
KD, PMAX, KA = 0.35, 9.0, 1.1
THETA_D, THETA_A = 1.047, 1.024


def hourly_forcing(hours):
    h = np.arange(hours, dtype=np.float64)
    light = np.maximum(np.sin(2.0 * np.pi * (h - 6.0) / 24.0), 0.0)        # sunrise at 6, noon at 12
    temp = 20.0 + 4.0 * np.sin(2.0 * np.pi * (h - 9.0) / 24.0)             # warmest at 15
    return light, temp


def closed_box_mesh(T, dt, n_cells_side=2):
    from clearwater_riverine_b200 import synthetic
    plan = synthetic.make_plan(n_cells_side + 1, n_cells_side, T, dt=dt, seed=13)
    flow, vel = np.zeros_like(plan.face_flow), np.zeros_like(plan.edge_velocity)
    vol = np.repeat(plan.volume[:1], plan.n_time, axis=0)
    adv, _, _, cdiff, dts = ref.derive_coefficients(flow, vel, plan.face_x, plan.face_y, plan.f1, plan.f2, 0.0, plan.time_seconds)
    return plan, ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, vel, vol, dts, 0.0)


def diurnal_box(dt, hours, L0, DO0):
    """The model's closed box at step dt (a divisor of an hour) through oracle.kinetics_forcing: step t takes the hour
    that contains its start."""
    T = int(round(hours * 3600.0 / dt)) + 1
    plan, mesh = closed_box_mesh(T, dt)
    n = plan.n_real
    light, temp = hourly_forcing(hours + 1)
    hour_of = np.minimum((np.arange(T) * dt // 3600.0).astype(int), hours)
    inputs = np.zeros((2, T, plan.n_face))
    inputs[0, 0, :n], inputs[1, 0, :n] = L0, DO0
    y = np.array([[0.0, 0.0], [-1.0, 0.0]])
    oracle = KineticsRiverine(mesh, {"BOD": inputs[0], "DO": inputs[1]}, np.array([KD, 0.0]), np.array([THETA_D, 1.0]), y,
                              20.0, source_per_day=np.array([0.0, PMAX]), exchange_per_day=np.array([0.0, KA]),
                              exchange_theta=np.array([1.0, THETA_A]), equilibrium=np.zeros(2),
                              equilibrium_kind=np.array([0, 1], np.int32),
                              **forcing_terms(np.array([0, 3], np.int32), np.array([-1, 1], np.int32),
                                              np.stack([temp[hour_of], light[hour_of]])))
    for _ in range(T - 1):
        oracle.update()
    return oracle.constituent_dict["BOD"].concentration[T - 1][:n], oracle.constituent_dict["DO"].concentration[T - 1][:n]


def diurnal_ivp(hours, L0, DO0):
    from scipy.integrate import solve_ivp
    light, temp = hourly_forcing(hours)
    y = np.array([L0, DO0], np.float64)
    for h in range(hours):
        T, L = temp[h], light[h]
        kd = KD * THETA_D ** (T - 20.0) / 86400.0
        ka = KA * THETA_A ** (T - 20.0) / 86400.0
        sat = float(o2sat(T))

        def rhs(_, c):
            return [-kd * c[0], -kd * c[0] + PMAX * L / 86400.0 + ka * (sat - c[1])]
        y = solve_ivp(rhs, (0.0, 3600.0), y, method="DOP853", rtol=1e-12, atol=1e-12).y[:, -1]
    return y


def test_closed_box_diurnal_do_converges_at_first_order_to_solve_ivp():
    """Two days of the piecewise-constant hourly forcing: the error at the end halves with dt (the operator splitting of
    the chain and the exchange is first order), from 1 h down to 7.5 min."""
    hours, L0, DO0 = 48, 12.0, 7.0
    want = diurnal_ivp(hours, L0, DO0)
    errs = []
    for dt in (3600.0, 1800.0, 900.0, 450.0):
        bod, do = diurnal_box(dt, hours, L0, DO0)
        assert np.ptp(bod) == 0.0 and np.ptp(do) == 0.0
        assert abs(bod[0] - want[0]) <= 1e-9 * L0          # the decay alone is exact per step
        errs.append(abs(do[0] - want[1]))
    ratios = [errs[i + 1] / errs[i] for i in range(len(errs) - 1)]
    assert errs[0] > 1e-4, errs
    assert all(0.4 < r < 0.6 for r in ratios), (errs, ratios)


def test_synthetic_forcing_is_seeded_and_valid():
    from clearwater_riverine_b200 import synthetic
    from clearwater_riverine_b200.kinetics import validate
    _, mesh, inputs, kin, src, lim, dep, frc = _small_network(constant=True)
    again = _small_network(constant=True)[-1]
    assert all(same(frc[k], again[k]) for k in frc)
    assert set(frc["target"].tolist()) == {0, 1, 2, 3, 4}
    validate(kin["decay_per_day"], kin["theta"], kin["yields"], -1, 17.0, **src, forcing_target=frc["target"],
             forcing_column=frc["column"], forcing_values=frc["values"], n_time=mesh.n_time)
    light = synthetic.diurnal_light(np.arange(0, 86400.0, 600.0))
    assert light.min() == 0.0 and light.max() > 0.99 and (light == 0).mean() > 0.45


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def _tk():
    from tests import test_kinetics as tk
    return tk


def forced_backend(mesh, inputs, kin, src, lim, dep, frc, **opt):
    from tests.test_kinetics_depth import depth_backend
    be = depth_backend(mesh, inputs, kin, src, lim, dep, **opt)
    if frc is not None:
        be.set_kinetics_forcing(**frc)
    return be


def run_forced_parity(mesh, inputs, kin, src, lim, dep, frc, steps, check_flux=True, **opt):
    tp, tk = _tk()._parity(), _tk()
    K = len(inputs)
    be = forced_backend(mesh, inputs, kin, src, lim, dep, frc, **opt)
    oracle = forcing_oracle(mesh, inputs, kin, src, lim, dep, frc)
    for t in range(steps):
        info = be.step(t)
        assert info.status == 0, (t, info.status, info.iterations, info.max_relres)
        oracle.update()
        for k in range(K):
            con = oracle.constituent_dict[f"c{k}"]
            tp.close(be.get_state(k, t + 1), con.concentration[t + 1], RTOL, f"step {t} k {k}")
            if check_flux:
                tp.flux_close(be, k, t, mesh, con.concentration[t + 1], con.advection_mass_flux[t], con.diffusion_mass_flux[t],
                              con.total_mass_flux[t], f"step {t} k {k}")
    want = np.sum(oracle.reaction_mass, axis=0)
    got = np.array([be.reaction_mass(k) for k in range(K)])
    scale = np.maximum(np.abs(want), tk.mass_scale(mesh, inputs))
    assert (np.abs(got - want) <= RTOL * scale).all(), (got, want)
    return be, oracle


def forced_network(nx, ny, T, K, seed, constant=False, limits_too=True, depth_too=True, **kw):
    from clearwater_riverine_b200 import synthetic
    from tests.test_kinetics_depth import synthetic_network
    plan, mesh, inputs, kin, src, lim, dep = synthetic_network(nx, ny, T, K, seed, limits_too=limits_too, **kw)
    if constant:
        kin = dict(kin, temperature_k=-1, temperature_c=19.0)
    frc = synthetic.make_kinetics_forcing(kin, src, plan.time_seconds, seed=seed, period=5 * float(mesh.dt[0]))
    return plan, mesh, inputs, kin, src, lim, dep if depth_too else None, frc


@pytest.mark.gpu
@pytest.mark.parametrize("constant", [False, True])
@pytest.mark.parametrize("solver", [1, 2])
@pytest.mark.parametrize("K", [3, 6, 17])
def test_large_path_parity(K, solver, constant):
    _, mesh, inputs, kin, src, lim, dep, frc = forced_network(40, 25, 8, K, seed=K + 300, constant=constant,
                                                              dry_fraction=0.02)
    be, _ = run_forced_parity(mesh, inputs, kin, src, lim, dep, frc, 7, solver_path=1, solver=solver)
    be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("constant", [False, True])
@pytest.mark.parametrize("what", ["alone", "limits", "depth"])
def test_every_instantiation(what, constant):
    """Forcing with the chain and sources alone, with Monod factors, and with factors and depth flags."""
    _, mesh, inputs, kin, src, lim, dep, frc = forced_network(40, 25, 7, 6, seed=311, constant=constant,
                                                              limits_too=what != "alone", depth_too=what == "depth",
                                                              dry_fraction=0.02)
    be, _ = run_forced_parity(mesh, inputs, kin, src, lim if what != "alone" else None, dep, frc, 6, solver_path=1)
    be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("constant", [False, True])
def test_small_path_parity(constant):
    _, mesh, inputs, kin, src, lim, dep, frc = forced_network(40, 25, 7, 5, seed=321, constant=constant, dry_fraction=0.02)
    be, _ = run_forced_parity(mesh, inputs, kin, src, lim, dep, frc, 6, solver_path=2, precond_sweep=0)
    assert be.options.solver_path == 2
    be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 64])
def test_on_chip_path_on_the_ohio_shaped_mesh(K):
    """DO with a light-scaled source, wind-scaled reaeration toward O2sat(T(t)), a temperature series and, for K = 64,
    solar die-off."""
    from clearwater_riverine_b200 import synthetic
    plan = synthetic.ohio_like(7, seed=2)
    D = 0.1
    adv, _, _, cdiff, dt = ref.derive_coefficients(plan.face_flow, plan.edge_velocity, plan.face_x, plan.face_y, plan.f1, plan.f2,
                                                   D, plan.time_seconds)
    mesh = ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, plan.edge_velocity, plan.volume, dt, D)
    inputs = synthetic.make_inputs(plan, K, seed=7, ic_range=(0.0, 15.0))
    kin = dict(decay_per_day=np.full(K, 2.0), theta=np.full(K, 1.047), yields=None, temperature_k=-1, temperature_c=17.0)
    src = dict(source_per_day=np.full(K, 900.0), source_theta=np.full(K, 1.065), exchange_per_day=np.linspace(0.6, 36.0, K),
               exchange_theta=np.full(K, 1.024), equilibrium=np.zeros(K), equilibrium_kind=np.ones(K, np.int32))
    frc = synthetic.make_kinetics_forcing(kin, src, plan.time_seconds, seed=K, period=4 * float(dt[0]))
    assert set(frc["target"].tolist()) == ({0, 2, 3, 4} if K > 2 else {0, 3, 4})
    be, _ = run_forced_parity(mesh, inputs, kin, src, None, None, frc, 6, check_flux=K == 1)
    assert be.options.solver_path in (3, 4)
    be.close()


@pytest.mark.gpu
def test_every_column_count_up_to_kmax():
    from clearwater_riverine_b200 import synthetic
    from tests.test_kinetics_depth import varied_area
    plan, mesh, base = _tk()._parity().synthetic_case(12, 9, 3, 128, seed=391)
    area = varied_area(plan, 391)
    for K in range(1, 129):
        inputs, kin = synthetic.make_kinetics(base[:K], seed=K)
        src = synthetic.make_kinetics_sources(kin, seed=K)
        lim = synthetic.make_kinetics_limits(kin, src, seed=K) if K % 2 else None
        dep = None
        if K % 3 == 0:
            kin, src, flags = synthetic.make_kinetics_depth(kin, src, seed=K)
            dep = dict(cell_area=area, min_depth=0.05, **flags)
        if K % 4 == 1:
            kin = dict(kin, temperature_k=-1)
        frc = synthetic.make_kinetics_forcing(kin, src, plan.time_seconds, seed=K, period=3 * float(mesh.dt[0]))
        be, _ = run_forced_parity(mesh, inputs, kin, src, lim, dep, frc, 1, check_flux=False, solver_path=1 + K % 2)
        be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("temperature_k", [-1, 3])
@pytest.mark.parametrize("solver_path", [1, 2])
def test_identity_forcing_is_bitwise_no_forcing(solver_path, temperature_k):
    """All-ones scales and series equal to their constants; forcing cleared by a call with n = 0; by a new
    set_kinetics_sources; by a new set_kinetics: the same bits, launches and reaction mass as the run that never set
    forcing.  A run with limits and depth set after the forcing keeps it."""
    _, mesh, inputs, kin, src, lim, dep, frc = forced_network(40, 25, 7, 4, seed=371, dry_fraction=0.02)
    kin = dict(kin, temperature_k=temperature_k)
    ident = identity_forcing(kin, src, mesh.n_time)
    plain = forced_backend(mesh, inputs, kin, src, lim, dep, None, solver_path=solver_path)
    cases = [forced_backend(mesh, inputs, kin, src, lim, dep, ident, solver_path=solver_path)]
    for how in ("off", "sources", "kinetics"):
        be = forced_backend(mesh, inputs, kin, src, lim, dep, frc, solver_path=solver_path)
        if how == "off":
            be.set_kinetics_forcing(None)
        elif how == "sources":
            be.set_kinetics_sources(**src)
            be.set_kinetics_limits(**lim)
            be.set_kinetics_depth(**dep)
        else:
            be.set_kinetics(**kin)
            be.set_kinetics_sources(**src)
            be.set_kinetics_limits(**lim)
            be.set_kinetics_depth(**dep)
        cases.append(be)
    forced = forced_backend(mesh, inputs, kin, src, None, None, frc, solver_path=solver_path)
    forced.set_kinetics_limits(**lim)
    forced.set_kinetics_depth(**dep)
    forced_ref = forced_backend(mesh, inputs, kin, src, lim, dep, frc, solver_path=solver_path)
    for t in range(6):
        a = plain.step(t)
        forced.step(t)
        forced_ref.step(t)
        for be in cases:
            assert be.step(t).n_launches == a.n_launches
            assert same(plain.get_state_all(t + 1), be.get_state_all(t + 1)), t
            for k in range(4):
                assert all(same(x, y) for x, y in zip(plain.get_mass_flux(k, t), be.get_mass_flux(k, t)))
    assert not same(plain.get_state_all(6), forced.get_state_all(6))      # the forcing does act on this network
    assert same(forced.get_state_all(6), forced_ref.get_state_all(6))     # limits and depth after it keep it
    for be in cases:
        assert all(be.reaction_mass(k) == plain.reaction_mass(k) for k in range(4))
    for be in [plain, forced, forced_ref] + cases:
        be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("solver_path", [1, 2])
def test_run_is_bitwise_step_by_step_and_repeatable(solver_path):
    """cwr_run batches the steps (on the small path their step parameters go up at once): each must read its own row."""
    _, mesh, inputs, kin, src, lim, dep, frc = forced_network(30, 20, 10, 5, seed=381, constant=True, dry_fraction=0.02)
    outs = []
    for mode in ("step", "run", "run"):
        be = forced_backend(mesh, inputs, kin, src, lim, dep, frc, solver_path=solver_path)
        if mode == "step":
            for t in range(9):
                assert be.step(t).status == 0
        else:
            assert be.run(0, 9).status == 0
        outs.append((np.stack([be.get_state_all(t) for t in range(1, 10)]), [be.reaction_mass(k) for k in range(5)]))
        be.close()
    for states, masses in outs[1:]:
        assert same(states, outs[0][0]) and masses == outs[0][1]
    oracle = forcing_oracle(mesh, inputs, kin, src, lim, dep, frc)
    for _ in range(9):
        oracle.update()
    for k in range(5):
        _tk()._parity().close(outs[1][0][-1][k], oracle.constituent_dict[f"c{k}"].concentration[9][:mesh.n], RTOL, f"run k{k}")


def _model(plan, inputs_by_name, spec, temperature, **opt):
    from clearwater_riverine_b200 import ClearwaterRiverine
    arrays = (plan.f1, plan.f2, plan.face_x, plan.face_y, plan.time_seconds, plan.face_flow, plan.edge_velocity, plan.volume, 0.1)
    return ClearwaterRiverine.from_arrays(*arrays, inputs_by_name, kinetics=spec, temperature=temperature, **opt)


@pytest.mark.gpu
def test_model_run_and_stream_hydro_are_bitwise_update_by_update():
    """run() (cwr_run) and update() with the hydrodynamics streamed slice by slice give the bits of update() by update()."""
    tp = _tk()._parity()
    plan, mesh, inputs = tp.synthetic_case(20, 14, 9, 3, seed=5, dry_fraction=0.02)
    T = plan.n_time
    named = dict(zip(NAMES, inputs))
    named["T"] = np.where(named["T"] != 0, 18.0 + 0.05 * named["T"], 0.0)
    spec = _spec(T)
    models = []
    try:
        for opt in ({}, {}, dict(stream_hydro=True)):
            models.append(_model(plan, named, spec, np.linspace(14.0, 24.0, T), **opt))
        for _ in range(T - 1):
            models[0].update()
            models[2].update()
        models[1].run()
        assert models[0].kinetics.has_forcing
        for name in NAMES:
            for m in models[1:]:
                assert same(models[0].mesh[name], m.mesh[name]), name
    finally:
        for m in models:
            m.finalize()


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_several_tiles_per_cta():
    """One forced step pair on the large path at a size where every CTA of the resident grid takes two or more tiles,
    with every target: b, the reaction mass and the solve checked as test_kinetics_scale does, against the oracle's
    reacted step with step t's values substituted into the parameters."""
    from tests.test_kinetics_scale import _side, oracle_network, react_tile_rows, reacted_step, resident_cta_bound
    K, n = 3, 610_001
    tiles = -(-n // react_tile_rows(K))
    assert tiles >= 2 * resident_cta_bound()
    plan, mesh, inputs, kin, src, lim, dep, frc = forced_network(_side(n), _side(n), 3, K, seed=401, constant=True,
                                                                 n_exact=n, dry_fraction=0.02)
    assert mesh.n == n and set(frc["target"].tolist()) >= {0, 3, 4}
    be = forced_backend(mesh, inputs, kin, src, lim, dep, frc, solver_path=1)
    lhs = ref.LHS(mesh)
    before = np.zeros(K)
    for t in range(2):
        k2, s2 = dict(kin, decay_per_day=np.array(kin["decay_per_day"], float)), {k: np.array(v) for k, v in src.items()}
        s2 = {k: (v.astype(float) if k != "equilibrium_kind" else v) for k, v in s2.items()}
        for g, k, v in zip(frc["target"], frc["column"], frc["values"]):
            if g == 0:
                k2["temperature_c"] = v[t]
            elif g == 1:
                s2["equilibrium"][k] = v[t]
            elif g == 2:
                k2["decay_per_day"][k] *= v[t]
            elif g == 3:
                s2["source_per_day"][k] *= v[t]
            else:
                s2["exchange_per_day"][k] *= v[t]
        net = oracle_network(k2, s2, lim, dep)
        c_t = be.get_state_all(t)
        assert be.step(t).status == 0
        b, b0, mass, mass_abs = reacted_step(mesh, inputs, c_t, t, **net)
        row = np.maximum(np.abs(b).max(axis=0), np.abs(b0).max(axis=0))
        for k in range(K):
            bad = np.nonzero(np.abs(be.get_rhs(k) - b[k]) > 1e-12 * row)[0]
            assert bad.size == 0, f"step {t} k {k}: b differs in {bad.size} rows"
        after = np.array([be.reaction_mass(k) for k in range(K)])
        assert (np.abs((after - before) - mass) <= 1e-11 * mass_abs).all(), (t, after - before, mass)
        before = after
        lhs.update_values(mesh, t)
        A = lhs.to_csr()
        x = be.get_state_all(t + 1)
        for k in range(K):
            assert np.linalg.norm(A @ x[k] - b[k]) / np.linalg.norm(b[k]) <= 1e-12, (t, k)
    be.close()


@pytest.mark.gpu
def test_reaction_mass_under_the_defect_correction_fallback():
    from clearwater_riverine_b200 import synthetic
    from tests.test_kinetics_depth import varied_area
    plan = synthetic.make_plan(60, 50, 6, seed=41, dry_fraction=0.02)
    vel = plan.edge_velocity.copy()
    vel[:, np.random.default_rng(1).random(plan.n_edge) < 0.05] *= -1
    D = 2.0
    adv, _, _, cdiff, dt = ref.derive_coefficients(plan.face_flow, vel, plan.face_x, plan.face_y, plan.f1, plan.f2, D, plan.time_seconds)
    mesh = ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, vel, plan.volume, dt, D)
    inputs, kin = synthetic.make_kinetics(synthetic.make_inputs(plan, 3, seed=41), seed=41)
    src = synthetic.make_kinetics_sources(kin, seed=41)
    lim = synthetic.make_kinetics_limits(kin, src, seed=41)
    kin, src, flags = synthetic.make_kinetics_depth(kin, src, seed=41)
    dep = dict(cell_area=varied_area(plan, 41), min_depth=0.05, **flags)
    frc = synthetic.make_kinetics_forcing(kin, src, plan.time_seconds, seed=41, period=4 * float(dt[0]))
    tp, tk = _tk()._parity(), _tk()
    be = forced_backend(mesh, inputs, kin, src, lim, dep, frc, solver_path=1, solver=2)
    oracle = forcing_oracle(mesh, inputs, kin, src, lim, dep, frc)
    for t in range(3):
        assert be.step(t).status == 0
        oracle.update()
        for k in range(3):
            tp.close(be.get_state(k, t + 1), oracle.constituent_dict[f"c{k}"].concentration[t + 1], 1e-8, f"fallback k{k} t{t}")
        want = np.sum(oracle.reaction_mass, axis=0)
        for k in range(3):
            assert abs(be.reaction_mass(k) - want[k]) <= RTOL * max(abs(want[k]), tk.mass_scale(mesh, inputs)[k]), (t, k)
    assert be.solver_stats()[1] >= 1, "the sweeps diverge on this matrix: the solver should have fallen back"
    be.close()


@pytest.mark.gpu
def test_mass_balance_closes_with_forcing():
    tp = _tk()._parity()
    plan, mesh, inputs = tp.synthetic_case(20, 14, 8, 3, seed=4, dry_fraction=0.02)
    T = plan.n_time
    named = dict(zip(NAMES, inputs))
    named["T"] = np.where(named["T"] != 0, 10.0 + 0.2 * named["T"], 0.0)
    spec = {name: {k: (v * 300.0 if k.endswith("_per_day") else v) for k, v in block.items()} for name, block in _spec(T).items()}
    model = _model(plan, named, spec, "T")
    try:
        _mass_balance_closes(model, plan, mesh, named)
    finally:
        model.finalize()


def _mass_balance_closes(model, plan, mesh, named):
    tp = _tk()._parity()
    kin = model.kinetics
    assert kin.has_forcing
    oracle = KineticsRiverine(mesh, named, kin.decay_per_day, kin.theta, kin.yields, "T", **kin.sources_arguments(),
                              **forcing_terms(**kin.forcing_arguments()))
    for t in range(7):
        model.update()
        oracle.update()
        for name in NAMES:
            tp.close(model.mesh[name][t + 1], oracle.constituent_dict[name].concentration[t + 1], RTOL, f"{name} {t}")
    faces = {nm: plan.boundary_faces[nm] for nm in ("upstream", "downstream")}
    for k, name in enumerate(NAMES):
        got = model.mass_balance(name, faces)
        con = oracle.constituent_dict[name]
        want = ref.mass_balance(mesh, con.concentration, con.total_mass_flux, plan.face_flow, faces)
        reaction = float(np.sum(oracle.reaction_mass, axis=0)[k])
        assert reaction != 0.0
        assert abs(got["reaction_mass"] - reaction) <= RTOL * abs(want["Mass_start"])
        assert abs(got["error_mass"] - (want["mass_end_calc"] + reaction - want["Mass_end"])) <= RTOL * abs(want["Mass_start"])


@pytest.mark.gpu
def test_diurnal_do_stays_non_negative_with_its_minimum_at_night():
    """Closed boxes over four days of 15-minute steps: a heavy BOD load (40..120 mg/L) oxidised at a rate limited by DO,
    photosynthesis scaled by the light (>= 0), reaeration toward O2sat(T(t)).  Through ClearwaterRiverine.run(): DO >= 0
    everywhere, and on the last day the lowest DO falls at night and the highest in the afternoon."""
    days, dt = 4, 900.0
    T = int(days * 86400 / dt) + 1
    plan, mesh = closed_box_mesh(T, dt, n_cells_side=4)
    n = plan.n_real
    t = plan.time_seconds
    from clearwater_riverine_b200.synthetic import diurnal_light
    light = diurnal_light(t, phase=6 * 3600.0)                       # sunrise at 06:00
    temp = 20.0 + 4.0 * np.sin(2.0 * np.pi * (t / 86400.0 - 9.0 / 24.0))
    inputs = {"DO": np.zeros((T, plan.n_face)), "BOD": np.zeros((T, plan.n_face))}
    inputs["DO"][0, :n] = 6.0
    inputs["BOD"][0, :n] = np.linspace(40.0, 120.0, n)
    spec = {"BOD": {"decay_per_day": 0.6, "theta": 1.047, "yields": {"DO": -1.0}, "limited_by": {"DO": 0.5}},
            "DO": {"source_per_day": 14.0, "source_scale": light, "exchange_per_day": 0.8, "exchange_theta": 1.024,
                   "equilibrium": "oxygen_saturation"}}
    from clearwater_riverine_b200 import ClearwaterRiverine
    model = ClearwaterRiverine.from_arrays(plan.f1, plan.f2, plan.face_x, plan.face_y, t, np.zeros_like(plan.face_flow),
                                           np.zeros_like(plan.edge_velocity), np.repeat(plan.volume[:1], T, axis=0), 0.0,
                                           inputs, kinetics=spec, temperature=temp)
    try:
        model.run()
        do = model.mesh["DO"][:, :n].copy()
    finally:
        model.finalize()
    assert np.isfinite(do).all() and do.min() >= -1e-12 * float(o2sat(16.0)), do.min()
    last = slice(T - 1 - int(86400 / dt), T - 1)
    mean = do[last].mean(axis=1)
    hour = (t[last] % 86400.0) / 3600.0
    assert hour[int(np.argmin(mean))] < 8.0 or hour[int(np.argmin(mean))] > 20.0, hour[int(np.argmin(mean))]
    assert 12.0 <= hour[int(np.argmax(mean))] <= 19.0, hour[int(np.argmax(mean))]
    assert do.min() < 1.0                                            # the demand does drive it down to near zero


@pytest.mark.gpu
def test_yaml_config_with_csv_series_is_bitwise_from_arrays(tmp_path):
    yaml = pytest.importorskip("yaml")
    import pandas as pd
    from clearwater_riverine_b200 import ClearwaterRiverine
    from clearwater_riverine_b200.io import ras
    from tests.helpers import load_golden
    from tests.test_kinetics_depth import write_plan_with_area
    g = dict(load_golden("p01_random_two"))
    hdf = tmp_path / "plan.hdf"
    times = write_plan_with_area(hdf, g)
    plan = ras.read_ras_plan(hdf)
    n = plan.nreal + 1
    lines = sorted({str(x) for x in g["bc_names"]})
    cons = {}
    for name, ic, bc in (("DO", 0.5, 8.0), ("BOD", 8.0, 5.0)):
        icf, bcf = tmp_path / f"{name}_ic.csv", tmp_path / f"{name}_bc.csv"
        pd.DataFrame({"Cell_Index": np.arange(n), "Concentration": ic + 0.01 * np.arange(n)}).to_csv(icf, index=False)
        pd.DataFrame({"Datetime": np.repeat([times[0], times[-1]], len(lines)), "RAS2D_TS_Name": lines * 2,
                      "Concentration": bc}).to_csv(bcf, index=False)
        cons[name] = {"initial_conditions": str(icf), "boundary_conditions": str(bcf), "units": "mg/L"}
    stamps = pd.date_range(pd.Timestamp(times[0]) - pd.Timedelta(minutes=1), pd.Timestamp(times[-1]), periods=9)
    light, temp = tmp_path / "light.csv", tmp_path / "temperature.csv"
    pd.DataFrame({"Datetime": stamps, "Value": np.linspace(0.0, 1.0, 9) ** 2}).to_csv(light, index=False)
    pd.DataFrame({"Datetime": stamps, "Value": np.linspace(14.0, 22.0, 9)}).to_csv(temp, index=False)
    spec = {"BOD": {"decay_per_day": 40.0, "yields": {"DO": -1.0}, "limited_by": {"DO": 0.5}},
            "DO": {"source_per_day": 300.0, "source_scale": {"csv": str(light)}, "exchange_per_day": 50.0,
                   "equilibrium": "oxygen_saturation"}}
    cfg = {"diffusion_coefficient": 0.1, "flow_field_filepath": str(hdf), "temperature": {"csv": str(temp)},
           "constituents": {name: dict(c, kinetics=spec.get(name)) for name, c in cons.items()}}
    cfg_path = tmp_path / "model.yml"
    cfg_path.write_text(yaml.safe_dump(cfg))
    inputs = {name: ras.build_input_array(len(plan.time), len(plan.face_x), plan.time, plan.f2, plan.boundary_data,
                                          c["initial_conditions"], c["boundary_conditions"]) for name, c in cons.items()}
    a = ClearwaterRiverine(config_filepath=str(cfg_path))
    b = ClearwaterRiverine.from_arrays(plan.f1, plan.f2, plan.face_x, plan.face_y, plan.time_seconds, plan.face_flow,
                                       plan.edge_velocity, plan.volume, 0.1, inputs)
    try:
        _yaml_matches(a, b, cons, plan, spec, light, temp)
    finally:
        a.finalize(); b.finalize()


def _yaml_matches(a, b, cons, plan, spec, light, temp):
    from clearwater_riverine_b200.io import ras
    arrays = dict(spec, DO=dict(spec["DO"], source_scale=ras.read_series_csv(light, plan.time)))
    b.set_kinetics(arrays, temperature=ras.read_series_csv(temp, plan.time))
    steps = min(12, len(plan.time) - 1)
    for _ in range(steps):
        a.update(); b.update()
    for name in cons:
        assert same(a.mesh[name][:steps + 1], b.mesh[name][:steps + 1]), name
        assert a.backend.reaction_mass(a._index[name]) == b.backend.reaction_mass(b._index[name])
    assert a.kinetics.has_forcing and a.kinetics.forcing_target.tolist() == [0, 3]


@pytest.mark.gpu
def test_invalid_forcing_straight_to_the_abi_returns_einval():
    from clearwater_riverine_b200.backend import CWR_EINVAL
    plan, mesh, inputs = _tk()._parity().synthetic_case(12, 9, 4, 3, seed=2)
    be = _tk()._parity().make_backend(mesh, list(inputs))
    lib, T = be._lib, mesh.n_time

    def call(rows, values=None, n=None, n_time=T):
        tg = np.array([r[0] for r in rows] or [0], np.int32)
        col = np.array([r[1] for r in rows] or [0], np.int32)
        v = np.ascontiguousarray(np.ones((max(1, len(rows)), n_time)) if values is None else values, np.float64)
        return lib.cwr_set_kinetics_forcing(be._h, len(rows) if n is None else n, n_time,
                                            tg.ctypes.data_as(C.POINTER(C.c_int32)), col.ctypes.data_as(C.POINTER(C.c_int32)),
                                            v.ctypes.data_as(C.POINTER(C.c_double)))

    ok = [(0, -1), (1, 2), (2, 0), (3, 1), (4, 1), (4, 2)]
    assert call(ok) == CWR_EINVAL                                         # kinetics not set
    be.set_kinetics(np.array([1.0, 0.0, 0.0]), None, None, -1, 20.0)
    be.set_kinetics_sources(np.array([0.0, -1.0, 0.0]), None, np.array([0.0, 2.0, 3.0]), None, np.array([0.0, 0.0, 5.0]),
                            np.array([0, 1, 0], np.int32))
    assert call(ok) == 0 and call([], n=0) == 0 and call([(1, 2)], values=-np.ones((1, T))) == 0
    nan = np.ones((1, T)); nan[0, T - 1] = np.nan
    bad = [dict(rows=ok, n=-1), dict(rows=ok, n_time=T + 1), dict(rows=[(5, 0)]), dict(rows=[(-1, 0)]),
           dict(rows=[(0, 0)]), dict(rows=[(2, 3)]), dict(rows=[(2, -1)]), dict(rows=[(2, 0), (2, 0)]),
           dict(rows=[(2, 0)], values=nan), dict(rows=[(3, 1)], values=-np.ones((1, T))), dict(rows=[(2, 1)]),
           dict(rows=[(3, 0)]), dict(rows=[(4, 0)]), dict(rows=[(1, 0)]), dict(rows=[(1, 1)])]
    for args in bad:
        assert call(**args) == CWR_EINVAL, args
    be.set_kinetics(np.array([1.0, 0.0, 0.0]), None, None, 2, 20.0)
    assert call([(0, -1)]) == CWR_EINVAL                                  # a temperature constituent is set
    be.set_kinetics(None)
    assert call([(2, 0)]) == CWR_EINVAL                                   # kinetics switched off again
    with pytest.raises(ValueError, match="given twice"):
        be.set_kinetics(np.array([1.0, 0.0, 0.0]), None, None, -1, 20.0)
        be.set_kinetics_forcing([2, 2], [0, 0], np.ones((2, T)))
    be.close()


def _gpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_domain_decomposition_with_forcing():
    if _gpus() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", str(ROOT / "tools" / "dd_check.py"), "--side", "150", "--K", "4", "--steps", "5", "--kinetics"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=850, cwd=ROOT)
    lines = [json.loads(ln) for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert out.returncode == 0, (out.stdout[-3000:], out.stderr[-3000:])
    runs = [ln for ln in lines if ln.get("forcing")]
    assert len(runs) >= 3 and all(ln["ok"] for ln in lines), lines
    for ln in runs:
        assert ln["max_rel_diff_vs_oracle"] < 1e-9 and ln["max_rel_diff_vs_single_gpu"] < 1e-9
        assert ln["reaction_mass_rel_diff"] < 1e-9
