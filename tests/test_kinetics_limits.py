"""Monod limitation and inhibition of the device kinetics (cwr_set_kinetics_limits): the spec compiler and the numpy
restatement (oracle.kinetics_limits) on the CPU, the CUDA path against the restatement on the GPU.  GPU tolerance as in
test_kinetics: rtol 1e-9 per step."""
import ctypes as C
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
from scipy.integrate import solve_ivp

from oracle import kinetics_sources as sources
from oracle import reference_step as ref
from oracle.kinetics_limits import KineticsRiverine, limit_terms, react
from oracle.kinetics_sources import o2sat
from tests.helpers import same

ROOT = Path(__file__).resolve().parents[1]
RTOL = 1e-9
# the DO parameters of test_kinetics_sources.SPEC: BOD oxidation limited by DO, sediment oxygen demand limited by DO
KD, KA, SOD = 0.35, 0.7, -1.5
K_BOD, K_SOD = 0.5, 1.0
SPEC = {"BOD": {"decay_per_day": 0.35, "theta": 1.047, "yields": {"DO": -1.0}, "limited_by": {"DO": 0.5}},
        "NH4": {"decay_per_day": 0.1, "theta": 1.083, "yields": {"NO3": 1.0, "DO": -4.57}, "limited_by": {"DO": 0.7}},
        "NO3": {"decay_per_day": 0.1, "theta": 1.045, "inhibited_by": {"DO": 0.6}},
        "DO": {"source_per_day": -1.5, "source_theta": 1.065, "exchange_per_day": 0.7, "exchange_theta": 1.024,
               "equilibrium": "oxygen_saturation", "source_limited_by": {"DO": 1.0}},
        "T": {"source_per_day": 0.2, "exchange_per_day": 0.3, "equilibrium": 18.0, "source_inhibited_by": {"BOD": 4.0}}}
NAMES = ["DO", "BOD", "NH4", "NO3", "T"]


# ------------------------------------------------------------------------------------------------------------------
# CPU: spec compiler
# ------------------------------------------------------------------------------------------------------------------
def test_spec_compiles_the_factors_in_order():
    from clearwater_riverine_b200.kinetics import compile_kinetics
    spec = {"BOD": {"decay_per_day": 0.35, "yields": {"DO": -1.0, "X": -0.5}, "inhibited_by": {"NO3": 3.0, "T": 9.0},
                    "limited_by": {"X": 0.2, "DO": 0.5}},
            "DO": {"source_per_day": -1.5, "source_inhibited_by": {"X": 2.0}, "source_limited_by": {"DO": 1.0, "BOD": 7.0}}}
    kin = compile_kinetics(spec, ["DO", "BOD", "NO3", "T", "X"], 20.0)
    assert kin.has_limits
    args = kin.limits_arguments()
    assert sorted(args) == ["column", "factor_column", "factor_kind", "half_saturation", "process"]
    rows = list(zip(*(args[k].tolist() for k in ("process", "column", "factor_column", "factor_kind", "half_saturation"))))
    # per block: the limitations (decay, then source) first, then the inhibitions, each mapping in its order
    assert rows == [(0, 1, 4, 0, 0.2), (0, 1, 0, 0, 0.5), (0, 1, 2, 1, 3.0), (0, 1, 3, 1, 9.0),
                    (1, 0, 0, 0, 1.0), (1, 0, 1, 0, 7.0), (1, 0, 4, 1, 2.0)]
    assert all(args[k].dtype == np.int32 for k in ("process", "column", "factor_column", "factor_kind"))
    assert args["half_saturation"].dtype == np.float64
    plain = compile_kinetics({"BOD": {"decay_per_day": 0.35}}, ["DO", "BOD"], 20.0)
    assert not plain.has_limits and plain.limit_process is None


def test_kinetics_built_without_the_new_fields_has_no_limits():
    from clearwater_riverine_b200.kinetics import Kinetics
    kin = Kinetics(np.zeros(2), np.ones(2), np.zeros((2, 2)), -1, 20.0, (0, 1))
    assert not kin.has_limits and kin.limits_arguments()["process"] is None


INVALID = {
    "half-saturation zero": {"A": {"decay_per_day": 1.0, "limited_by": {"B": 0.0}}},
    "half-saturation negative": {"A": {"decay_per_day": 1.0, "inhibited_by": {"B": -1.0}}},
    "half-saturation infinite": {"A": {"decay_per_day": 1.0, "limited_by": {"B": float("inf")}}},
    "half-saturation nan": {"A": {"source_per_day": 1.0, "source_inhibited_by": {"B": float("nan")}}},
    "decay factor without decay": {"A": {"limited_by": {"B": 1.0}}},
    "source factor without source": {"A": {"exchange_per_day": 1.0, "equilibrium": 2.0, "source_limited_by": {"B": 1.0}}},
    "decay limited by itself": {"A": {"decay_per_day": 1.0, "limited_by": {"A": 1.0}}},
    "decay inhibited by itself": {"A": {"decay_per_day": 1.0, "inhibited_by": {"A": 1.0}}},
    "source inhibited by itself": {"A": {"source_per_day": -1.0, "source_inhibited_by": {"A": 1.0}}},
    "positive source limited by itself": {"A": {"source_per_day": 1.0, "source_limited_by": {"A": 1.0}}},
    "unknown factor constituent": {"A": {"decay_per_day": 1.0, "limited_by": {"Z": 1.0}}},
    "factor not a mapping": {"A": {"decay_per_day": 1.0, "limited_by": ["B"]}},
}


@pytest.mark.parametrize("case", sorted(INVALID))
def test_invalid_limit_specs_are_rejected_naming_the_constituent(case):
    from clearwater_riverine_b200.kinetics import compile_kinetics
    with pytest.raises(ValueError, match="'A'"):
        compile_kinetics(INVALID[case], ["A", "B", "T"], 20.0)


def test_validate_rejects_every_abi_condition():
    from clearwater_riverine_b200.kinetics import validate
    d, th, y = np.array([1.0, 0.0, 0.0]), np.ones(3), np.zeros((3, 3))
    s = np.array([0.0, -1.0, 2.0])
    ok = dict(limit_process=[0, 1], limit_column=[0, 1], limit_factor_column=[1, 1], limit_kind=[0, 0],
              limit_half_saturation=[1.0, 1.0])
    validate(d, th, y, -1, 20.0, ("A", "B", "C"), source_per_day=s, **ok)
    bad = {"process": dict(ok, limit_process=[2, 1]), "kind": dict(ok, limit_kind=[0, -1]),
           "range": dict(ok, limit_factor_column=[3, 1]), "column": dict(ok, limit_column=[-1, 1]),
           "given twice": dict(limit_process=[0, 0], limit_column=[0, 0], limit_factor_column=[1, 1], limit_kind=[1, 1],
                               limit_half_saturation=[1.0, 2.0]),
           "'C'": dict(limit_process=[1], limit_column=[2], limit_factor_column=[2], limit_kind=[0], limit_half_saturation=[1.0])}
    for what, args in bad.items():
        with pytest.raises(ValueError, match=what):
            validate(d, th, y, -1, 20.0, ("A", "B", "C"), source_per_day=s, **args)


# ------------------------------------------------------------------------------------------------------------------
# CPU: the numpy restatement
# ------------------------------------------------------------------------------------------------------------------
def network(seed=2, n=40):
    """A BOD-NH4-NO3-DO-T network of SPEC on n cells (columns in NAMES order) and its compiled arrays."""
    from clearwater_riverine_b200.kinetics import compile_kinetics
    rng = np.random.default_rng(seed)
    kin = compile_kinetics(SPEC, NAMES, "T")
    c = np.stack([10.0 * rng.random(n), 30.0 * rng.random(n), 5.0 * rng.random(n), 5.0 * rng.random(n),
                  10.0 + 20.0 * rng.random(n)])
    return c, kin


def react_kin(c, dt, kin, limits=True):
    lim = kin.limits_arguments() if limits else {}
    return react(c, dt, kin.decay_per_day, kin.theta, kin.yields, kin.temperature_k, True, **kin.sources_arguments(),
                 **limit_terms(**lim))


def test_without_factors_it_is_bitwise_the_sources_restatement():
    c, kin = network()
    want = sources.react(c, 900.0, kin.decay_per_day, kin.theta, kin.yields, 4, True, **kin.sources_arguments())
    assert same(react_kin(c, 900.0, kin, limits=False), want)
    assert same(react(c, 900.0, kin.decay_per_day, kin.theta, kin.yields, 4, True, **kin.sources_arguments(),
                      **limit_terms([], [], [], [], [])), want)


def test_an_inhibition_on_a_zero_column_is_bitwise_the_unlimited_network():
    """K / (K + 0) = 1.0 exactly, so M = 1.0 and every process with such a factor is the unlimited one, bit for bit."""
    c, kin = network()
    c = np.vstack([c, np.zeros(c.shape[1])])                  # column 5: zero everywhere
    K = 6
    pad = lambda a, v=0.0: np.append(a, v)
    y = np.zeros((K, K)); y[:5, :5] = kin.yields
    src = {k: (None if v is None else pad(v, 1.0 if "theta" in k else 0)) for k, v in kin.sources_arguments().items()}
    args = (np.append(kin.decay_per_day, 0.0), np.append(kin.theta, 1.0), y, 4, True)
    lim = limit_terms([0, 0, 0, 1, 1], [1, 2, 3, 0, 4], [5] * 5, [1] * 5, [0.5, 1.0, 3.0, 2.0, 7.0])
    assert same(react(c, 900.0, *args, **src, **lim), sources.react(c, 900.0, *args, **src))


def test_a_limited_decay_with_the_factor_held_fixed_is_the_exponential_of_r_m():
    c0 = np.array([[20.0, 5.0, 0.3], [3.0, 0.5, 12.0]])       # BOD, DO (DO takes no part but as the factor)
    dt, steps, Kh = 600.0, 10, 0.8
    c = c0
    for _ in range(steps):
        c = react(c, dt, [2.0, 0.0], theta=[1.05, 1.0], temperature=27.0, **limit_terms([0], [0], [1], [0], [Kh]))
    r = 2.0 * 1.05 ** 7.0 / 86400.0
    M = c0[1] / (Kh + c0[1])
    assert np.abs(c[0] - c0[0] * np.exp(-r * M * dt * steps)).max() <= 1e-14 * c0[0].max()
    inh = react(c0, dt, [2.0, 0.0], **limit_terms([0], [0], [1], [1], [Kh]))
    assert np.abs(inh[0] - c0[0] * np.exp(-2.0 / 86400.0 * Kh / (Kh + c0[1]) * dt)).max() <= 1e-14 * c0[0].max()


def test_negative_factor_constituents_count_as_zero():
    c0 = np.array([[20.0, 20.0], [-3.0, 0.0]])
    lim = react(c0, 900.0, [2.0, 0.0], **limit_terms([0], [0], [1], [0], [0.8]))
    assert same(lim[0], c0[0])                                 # c+ = 0: no decay
    inh = react(c0, 900.0, [2.0, 0.0], **limit_terms([0], [0], [1], [1], [0.8]))
    assert same(inh[0, 0], inh[0, 1])


def box_terms(L0, do0=None):
    c = np.array([[L0], [float(o2sat(20.0)) if do0 is None else do0]])
    y = np.array([[0.0, 0.0], [-1.0, 0.0]])
    kw = dict(source_per_day=[0.0, SOD], exchange_per_day=[0.0, KA], equilibrium=[0.0, 0.0], equilibrium_kind=[0, 1])
    lim = limit_terms([0, 1], [0, 1], [1, 1], [0, 0], [K_BOD, K_SOD])
    return c, y, kw, lim


def closed_box(dt, L0, limited=True, days=10.0):
    """BOD and DO of one closed box (BOD oxidation limited by DO, SOD limited by DO): the last state and the lowest DO."""
    c, y, kw, lim = box_terms(L0)
    lowest = c[1, 0]
    for _ in range(int(round(days * 86400.0 / dt))):
        c = react(c, dt, [KD, 0.0], None, y, 20.0, **kw, **(lim if limited else {}))
        lowest = min(lowest, c[1, 0])
    return c, lowest


def test_the_cap_takes_do_exactly_to_zero():
    """L0 = 200 and dt = 1 day: the BOD oxidation of one step would take far more oxygen than there is; the cap leaves
    exactly 0 after the chain, never less."""
    c, y, kw, lim = box_terms(200.0)
    for _ in range(10):
        chain = react(c, 86400.0, [KD, 0.0], None, y, 20.0, **lim)
        assert chain[1, 0] == 0.0 and chain[0, 0] < c[0, 0]
        c = react(c, 86400.0, [KD, 0.0], None, y, 20.0, **kw, **lim)
        assert c[1, 0] > 0.0


@pytest.mark.parametrize("dt", [900.0, 6 * 3600.0, 86400.0])
def test_guaranteed_constituents_stay_non_negative(dt):
    """DO (consumed only by limited processes, self-limited sink, equilibrium O2sat >= 0) and BOD over 10 days, L0 from
    0 to 500 mg/L, DO from 0."""
    L0s = np.linspace(0.0, 500.0, 26)
    c, y, kw, lim = box_terms(0.0)
    c = np.vstack([L0s, np.zeros_like(L0s)])
    for _ in range(int(round(10 * 86400.0 / dt))):
        c = react(c, dt, [KD, 0.0], None, y, 20.0, **kw, **lim)
        assert (c >= 0.0).all(), c.min()


def test_the_cap_is_exact_for_a_yield_other_than_minus_one():
    """Nitrification (yield -4.57 on DO) limited by DO, loaded so that the cap binds in every cell: DO after the chain is
    >= 0 exactly, to the last bit.  The nearest-rounded quotient would leave some cells one rounding below 0."""
    from oracle.kinetics_limits import div_down
    rng = np.random.default_rng(11)
    n = 20000
    c = np.stack([1e3 + 1e4 * rng.random(n), 10.0 ** rng.uniform(-6, 1, n)])      # NH4 heavy, DO from 1e-6 to 10
    y = np.array([[0.0, 0.0], [-4.57, 0.0]])
    lim = limit_terms([0], [0], [1], [0], [0.7])
    for dt in (900.0, 86400.0):
        chain = react(c, dt, [50.0, 0.0], None, y, 20.0, **lim)
        assert (chain[1] >= 0.0).all(), chain[1].min()
        assert (chain[1] <= 1e-15 * c[1]).mean() > 0.9                 # the cap binds: DO drained to (nearly) 0
    nearest = c[1] + (-4.57) * (c[1] / 4.57)
    assert (nearest < 0.0).any()
    assert (c[1] + (-4.57) * div_down(c[1], 4.57) >= 0.0).all()


def test_closed_box_stays_oxic_where_the_unlimited_contract_goes_negative():
    _, parent = closed_box(900.0, 60.0, limited=False)
    _, limited = closed_box(900.0, 60.0)
    assert parent < -7.0, parent
    assert limited >= 0.25, limited


def test_closed_box_converges_at_first_order_to_the_ode():
    def rhs(t, u):
        L, D = u
        dp = max(D, 0.0)
        ox = KD / 86400.0 * L * dp / (K_BOD + dp)
        return [-ox, -ox + SOD / 86400.0 * dp / (K_SOD + dp) + KA / 86400.0 * (float(o2sat(20.0)) - D)]
    c900, _ = closed_box(900.0, 60.0)
    c450, _ = closed_box(450.0, 60.0)
    sol = solve_ivp(rhs, (0.0, 10 * 86400.0), [60.0, float(o2sat(20.0))], method="Radau", rtol=1e-12, atol=1e-14)
    e900, e450 = abs(c900[1, 0] - sol.y[1, -1]), abs(c450[1, 0] - sol.y[1, -1])
    assert e900 <= 0.05, e900
    assert 1.9 <= e900 / e450 <= 2.1, (e900, e450)


def test_synthetic_limits_bind_the_cap_in_some_cells():
    """make_kinetics_limits over make_kinetics's large default rates: the cap drains a consumed constituent to zero in
    a non-zero share of cells (the unlimited chain never drains one in a step)."""
    from clearwater_riverine_b200 import synthetic
    plan = synthetic.make_plan(40, 25, 3, seed=7)
    n = plan.n_real
    inputs, kin = synthetic.make_kinetics(synthetic.make_inputs(plan, 16, seed=7), seed=7)
    src = synthetic.make_kinetics_sources(kin, seed=7)
    lim = synthetic.make_kinetics_limits(kin, src, seed=7)
    c = inputs[:, 0, :n]
    dt = float(np.diff(plan.time_seconds)[0])
    chain = react(c, dt, kin["decay_per_day"], kin["theta"], kin["yields"], kin["temperature_k"], True, **limit_terms(**lim))
    capped = [j for p, j, kd in zip(lim["process"], lim["factor_column"], lim["factor_kind"]) if p == 0 and kd == 0]
    assert capped and set(lim["factor_kind"].tolist()) == {0, 1} and 1 in lim["process"]
    share = np.mean([(np.abs(chain[j]) <= 1e-12 * np.abs(c[j]).max()) & (c[j] > 0) for j in capped])
    assert share > 0.0, share


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def _tk():
    from tests import test_kinetics as tk
    return tk


def _ts():
    from tests import test_kinetics_sources as ts
    return ts


def limit_backend(mesh, inputs, kin, src, lim, **opt):
    be = _ts().source_backend(mesh, inputs, kin, src, **opt)
    if lim is not None:
        be.set_kinetics_limits(**lim)
    return be


def limit_oracle(mesh, inputs, kin, src, lim):
    temperature = f"c{kin['temperature_k']}" if kin["temperature_k"] >= 0 else kin["temperature_c"]
    return KineticsRiverine(mesh, {f"c{k}": inputs[k] for k in range(len(inputs))}, kin["decay_per_day"], kin["theta"],
                            kin["yields"], temperature, **(src or {}), **limit_terms(**(lim or {})))


def run_limit_parity(mesh, inputs, kin, src, lim, steps, overrides=None, check_flux=True, **opt):
    tp, tk = _tk()._parity(), _tk()
    K = len(inputs)
    be = limit_backend(mesh, inputs, kin, src, lim, **opt)
    oracle = limit_oracle(mesh, inputs, kin, src, lim)
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
            if check_flux:
                tp.flux_close(be, k, t, mesh, con.concentration[t + 1], con.advection_mass_flux[t], con.diffusion_mass_flux[t],
                              con.total_mass_flux[t], f"step {t} k {k}")
    want = np.sum(oracle.reaction_mass, axis=0)
    got = np.array([be.reaction_mass(k) for k in range(K)])
    scale = np.maximum(np.abs(want), tk.mass_scale(mesh, inputs))
    assert (np.abs(got - want) <= RTOL * scale).all(), (got, want)
    return be, oracle


def with_factors(kin, src, seed):
    """make_kinetics_limits; a single column's positive source is made a sink so that it has a factor."""
    from clearwater_riverine_b200 import synthetic
    if len(kin["decay_per_day"]) == 1:
        src = dict(src, source_per_day=-np.abs(src["source_per_day"]))
    lim = synthetic.make_kinetics_limits(kin, src, seed=seed)
    assert len(lim["process"]) > 0
    return src, lim


def synthetic_network(nx, ny, T, K, seed, **kw):
    mesh, inputs, kin, src = _ts().synthetic_network(nx, ny, T, K, seed, **kw)
    src, lim = with_factors(kin, src, seed)
    return mesh, inputs, kin, src, lim


@pytest.mark.gpu
def test_golden_mesh_parity_with_overrides():
    from clearwater_riverine_b200 import synthetic
    g, mesh, inputs, kin = _tk().golden_kinetic_case()
    src = synthetic.make_kinetics_sources(kin, seed=3, rate_range=(2000.0, 20000.0))   # dt = 1 s here
    src, lim = with_factors(kin, src, 3)
    n = mesh.n
    overrides = {3: {"c1": 40.0 + np.arange(n, dtype=np.float64)}, 9: {"c0": np.full(n, 7.0), "c3": np.linspace(15, 25, n)}}
    be, _ = run_limit_parity(mesh, inputs, kin, src, lim, 30, overrides)
    be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("solver", [1, 2])
@pytest.mark.parametrize("K", [1, 3, 16, 18, 19, 33])
def test_synthetic_meshes_on_the_large_path(K, solver):
    mesh, inputs, kin, src, lim = synthetic_network(40, 25, 8, K, seed=K + 50, dry_fraction=0.02)
    be, _ = run_limit_parity(mesh, inputs, kin, src, lim, 7, solver_path=1, solver=solver)
    be.close()


@pytest.mark.gpu
def test_every_column_count_up_to_kmax():
    from clearwater_riverine_b200 import synthetic
    _, mesh, base = _tk()._parity().synthetic_case(12, 9, 3, 128, seed=91)
    for K in range(1, 129):
        inputs, kin = synthetic.make_kinetics(base[:K], seed=K)
        src, lim = with_factors(kin, synthetic.make_kinetics_sources(kin, seed=K), K)
        for solver_path in (1, 2):
            be, _ = run_limit_parity(mesh, inputs, kin, src, lim, 1, check_flux=False, solver_path=solver_path)
            be.close()


@pytest.mark.gpu
def test_small_path_parity():
    mesh, inputs, kin, src, lim = synthetic_network(40, 25, 7, 5, seed=61, dry_fraction=0.02)
    be, _ = run_limit_parity(mesh, inputs, kin, src, lim, 6, solver_path=2, precond_sweep=0)
    assert be.options.solver_path == 2
    be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 64])
def test_on_chip_path_on_the_ohio_shaped_mesh(K):
    """K = 1: one DO column with a self-limited sediment oxygen demand; K = 64: 64 scenarios of it with 64 half-saturations."""
    from clearwater_riverine_b200 import synthetic
    plan = synthetic.ohio_like(7, seed=2)
    D = 0.1
    adv, _, _, cdiff, dt = ref.derive_coefficients(plan.face_flow, plan.edge_velocity, plan.face_x, plan.face_y, plan.f1, plan.f2,
                                                   D, plan.time_seconds)
    mesh = ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, plan.edge_velocity, plan.volume, dt, D)
    inputs = synthetic.make_inputs(plan, K, seed=7, ic_range=(0.0, 15.0))
    kin = dict(decay_per_day=np.full(K, 0.35), theta=np.full(K, 1.047), yields=None, temperature_k=-1, temperature_c=17.0)
    src = dict(source_per_day=np.full(K, -150.0), source_theta=np.full(K, 1.065), exchange_per_day=np.linspace(0.1, 6.0, K),
               exchange_theta=np.full(K, 1.024), equilibrium=np.zeros(K), equilibrium_kind=np.ones(K, np.int32))
    ks = np.arange(K, dtype=np.int32)
    lim = dict(process=np.ones(K, np.int32), column=ks, factor_column=ks, factor_kind=np.zeros(K, np.int32),
               half_saturation=np.linspace(0.2, 5.0, K))
    be, _ = run_limit_parity(mesh, inputs, kin, src, lim, 6, check_flux=K == 1)
    assert be.options.solver_path in (3, 4)
    be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("temperature_k", [-1, 15])
def test_both_temperature_modes(temperature_k):
    """K = 16 with the temperature constituent and the same network at a constant temperature (the factored processes
    evaluated per row there, the others from the per-CTA coefficients)."""
    mesh, inputs, kin, src, lim = synthetic_network(40, 25, 6, 16, seed=66, dry_fraction=0.02)
    kin = dict(kin, temperature_k=temperature_k, temperature_c=21.0)
    be, _ = run_limit_parity(mesh, inputs, kin, src, lim, 5, solver_path=1)
    be.close()


@pytest.mark.gpu
def test_constant_temperature_with_every_column_limited():
    """K = 128 at a constant temperature, every column a limited decay and a self-limited sink."""
    _, mesh, inputs = _tk()._parity().synthetic_case(12, 9, 3, 128, seed=92)
    rng = np.random.default_rng(6)
    K = 128
    y = np.zeros((K, K))
    for k in range(K - 1):
        y[k + 1, k] = -0.6
    kin = dict(decay_per_day=20.0 + 180.0 * rng.random(K), theta=np.full(K, 1.04), yields=y, temperature_k=-1, temperature_c=14.0)
    src = dict(source_per_day=-(20.0 + 2000.0 * rng.random(K)), exchange_per_day=20.0 + 100.0 * rng.random(K),
               exchange_theta=np.full(K, 1.024), equilibrium=40.0 * rng.random(K),
               equilibrium_kind=(np.arange(K) % 3 == 0).astype(np.int32))
    ks = np.arange(K - 1, dtype=np.int32)
    lim = dict(process=np.concatenate([np.zeros(K - 1, np.int32), np.ones(K, np.int32)]),
               column=np.concatenate([ks, np.arange(K, dtype=np.int32)]),
               factor_column=np.concatenate([ks + 1, np.arange(K, dtype=np.int32)]), factor_kind=np.zeros(2 * K - 1, np.int32),
               half_saturation=0.1 + rng.random(2 * K - 1))
    for solver_path in (1, 2):
        be, _ = run_limit_parity(mesh, inputs, kin, src, lim, 2, check_flux=False, solver_path=solver_path)
        be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("temperature_k", [-1, 3])
@pytest.mark.parametrize("solver_path", [1, 2])
def test_no_factors_are_bitwise_sources_only(solver_path, temperature_k):
    """n = 0; limits cleared by set_kinetics_limits(None); by a new set_kinetics_sources; by a new set_kinetics (and the
    sources set again): the same bits, launches and reaction mass as sources-only kinetics."""
    mesh, inputs, kin, src, lim = synthetic_network(40, 25, 7, 4, seed=71, dry_fraction=0.02)
    kin = dict(kin, temperature_k=temperature_k)
    empty = {k: v[:0] for k, v in lim.items()}
    plain = limit_backend(mesh, inputs, kin, src, None, solver_path=solver_path)
    cases = [limit_backend(mesh, inputs, kin, src, empty, solver_path=solver_path)]
    for how in ("off", "sources", "kinetics"):
        be = limit_backend(mesh, inputs, kin, src, lim, solver_path=solver_path)
        if how == "off":
            be.set_kinetics_limits(None)
        elif how == "sources":
            be.set_kinetics_sources(**src)
        else:
            be.set_kinetics(**kin)
            be.set_kinetics_sources(**src)
        cases.append(be)
    limited = limit_backend(mesh, inputs, kin, src, lim, solver_path=solver_path)
    for t in range(6):
        a = plain.step(t)
        limited.step(t)
        for be in cases:
            assert be.step(t).n_launches == a.n_launches
            assert same(plain.get_state_all(t + 1), be.get_state_all(t + 1))
            for k in range(4):
                assert all(same(x, y) for x, y in zip(plain.get_mass_flux(k, t), be.get_mass_flux(k, t)))
    assert not same(plain.get_state_all(6), limited.get_state_all(6))     # the factors do act on this network
    for be in cases:
        assert all(be.reaction_mass(k) == plain.reaction_mass(k) for k in range(4))
    for be in [plain, limited] + cases:
        be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("solver_path", [1, 2])
def test_run_is_bitwise_step_by_step_and_repeatable(solver_path):
    mesh, inputs, kin, src, lim = synthetic_network(30, 20, 10, 5, seed=81, dry_fraction=0.02)
    outs = []
    for mode in ("step", "run", "run"):
        be = limit_backend(mesh, inputs, kin, src, lim, solver_path=solver_path)
        if mode == "step":
            for t in range(9):
                assert be.step(t).status == 0
        else:
            assert be.run(0, 9).status == 0
        outs.append((np.stack([be.get_state_all(t) for t in range(1, 10)]), [be.reaction_mass(k) for k in range(5)]))
        be.close()
    for states, masses in outs[1:]:
        assert same(states, outs[0][0]) and masses == outs[0][1]
    oracle = limit_oracle(mesh, inputs, kin, src, lim)
    for _ in range(9):
        oracle.update()
    for k in range(5):
        _tk()._parity().close(outs[1][0][-1][k], oracle.constituent_dict[f"c{k}"].concentration[9][:mesh.n], RTOL, f"run k{k}")


@pytest.mark.gpu
def test_reaction_mass_counts_the_limited_processes_once_under_the_defect_correction_fallback():
    from clearwater_riverine_b200 import synthetic
    plan = synthetic.make_plan(60, 50, 6, seed=41, dry_fraction=0.02)
    vel = plan.edge_velocity.copy()
    vel[:, np.random.default_rng(1).random(plan.n_edge) < 0.05] *= -1
    D = 2.0
    adv, _, _, cdiff, dt = ref.derive_coefficients(plan.face_flow, vel, plan.face_x, plan.face_y, plan.f1, plan.f2, D, plan.time_seconds)
    mesh = ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, vel, plan.volume, dt, D)
    inputs = synthetic.make_inputs(plan, 3, seed=41)
    inputs, kin = synthetic.make_kinetics(inputs, seed=41)
    src, lim = with_factors(kin, synthetic.make_kinetics_sources(kin, seed=41), 41)
    tp, tk = _tk()._parity(), _tk()
    be = limit_backend(mesh, inputs, kin, src, lim, solver_path=1, solver=2)
    oracle = limit_oracle(mesh, inputs, kin, src, lim)
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


def _scaled_spec(f):
    """SPEC with every rate multiplied by f (the synthetic meshes step in 30 s)."""
    out = {}
    for name, block in SPEC.items():
        b = dict(block)
        for key in ("decay_per_day", "source_per_day", "exchange_per_day"):
            if key in b:
                b[key] = b[key] * f
        out[name] = b
    return out


@pytest.mark.gpu
def test_mass_balance_closes_with_limits():
    from clearwater_riverine_b200 import ClearwaterRiverine
    from clearwater_riverine_b200.kinetics import compile_kinetics
    tp = _tk()._parity()
    plan, mesh, inputs = tp.synthetic_case(20, 14, 8, 5, seed=4)
    inputs[4] = np.where(inputs[4] != 0, 10.0 + 0.2 * inputs[4], 0.0)
    inputs[0] = 0.1 * inputs[0]                                # little DO: the factors and the cap act
    spec = _scaled_spec(300.0)
    arrays = (plan.f1, plan.f2, plan.face_x, plan.face_y, plan.time_seconds, plan.face_flow, plan.edge_velocity, plan.volume, 0.1)
    model = ClearwaterRiverine.from_arrays(*arrays, dict(zip(NAMES, inputs)), kinetics=spec, temperature="T")
    assert model.kinetics.has_limits
    kin = compile_kinetics(spec, NAMES, "T")
    oracle = KineticsRiverine(mesh, dict(zip(NAMES, inputs)), kin.decay_per_day, kin.theta, kin.yields, "T",
                              **kin.sources_arguments(), **limit_terms(**kin.limits_arguments()))
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
    model.finalize()


@pytest.mark.gpu
def test_yaml_config_with_limit_keys_is_bitwise_from_arrays(tmp_path):
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
    for name, ic, bc in (("DO", 0.5, 8.0), ("BOD", 8.0, 5.0), ("NH4", 2.0, 1.0), ("NO3", 1.0, 0.5), ("T", 18.0, 21.0)):
        icf, bcf = tmp_path / f"{name}_ic.csv", tmp_path / f"{name}_bc.csv"
        pd.DataFrame({"Cell_Index": np.arange(n), "Concentration": ic + 0.01 * np.arange(n)}).to_csv(icf, index=False)
        pd.DataFrame({"Datetime": np.repeat([times[0], times[-1]], len(lines)), "RAS2D_TS_Name": lines * 2,
                      "Concentration": bc}).to_csv(bcf, index=False)
        cons[name] = {"initial_conditions": str(icf), "boundary_conditions": str(bcf), "units": "mg/L"}
    spec = _scaled_spec(2000.0)
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
    assert a.kinetics.has_limits
    a.finalize(); b.finalize()


@pytest.mark.gpu
def test_invalid_limits_straight_to_the_abi_return_einval():
    from clearwater_riverine_b200.backend import CWR_EINVAL
    _, mesh, inputs = _tk()._parity().synthetic_case(12, 9, 4, 3, seed=2)
    be = _tk()._parity().make_backend(mesh, list(inputs))
    lib = be._lib

    def call(n=None, p=None, k=None, j=None, kind=None, half=None):
        ints = [None if a is None else np.ascontiguousarray(a, np.int32) for a in (p, k, j, kind)]
        h = None if half is None else np.ascontiguousarray(half, np.float64)
        n = len(p) if n is None and p is not None else (n or 0)
        return lib.cwr_set_kinetics_limits(be._h, n, *[None if a is None else a.ctypes.data_as(C.POINTER(C.c_int32)) for a in ints],
                                           None if h is None else h.ctypes.data_as(C.POINTER(C.c_double)))

    # decay of 0 (consumes 1), source of 1 (a sink) and of 2 (> 0)
    ok = dict(p=[0, 1, 1, 0], k=[0, 1, 2, 0], j=[1, 1, 0, 2], kind=[0, 0, 1, 1], half=[0.5, 1.0, 2.0, 3.0])
    assert call(**ok) == CWR_EINVAL                           # kinetics not set
    y = np.zeros((3, 3)); y[1, 0] = -1.0
    be.set_kinetics(np.array([1.0, 0.0, 0.0]), None, y, -1, 20.0)
    be.set_kinetics_sources(np.array([0.0, -1.0, 2.0]))
    assert call(**ok) == 0 and call() == 0 and call(n=0, **{k: v for k, v in ok.items()}) == 0
    bad = [
        dict(ok, n=-1),
        dict(ok, p=[2, 1, 1, 0]), dict(ok, p=[-1, 1, 1, 0]), dict(ok, kind=[0, 0, 2, 1]), dict(ok, kind=[0, -1, 1, 1]),
        dict(ok, k=[3, 1, 2, 0]), dict(ok, k=[-1, 1, 2, 0]), dict(ok, j=[1, 1, 3, 2]), dict(ok, j=[1, -1, 0, 2]),
        dict(ok, half=[0.0, 1.0, 2.0, 3.0]), dict(ok, half=[0.5, -1.0, 2.0, 3.0]), dict(ok, half=[0.5, 1.0, np.nan, 3.0]),
        dict(ok, half=[0.5, 1.0, 2.0, np.inf]),
        dict(ok, p=[0, 1, 1, 0], k=[1, 1, 2, 0]),              # decay factor on a column that does not decay
        dict(ok, p=[1, 1, 1, 0], k=[0, 1, 2, 0]),              # source factor on a column without a source
        dict(ok, j=[0, 1, 0, 2]),                              # a decay limited by its own column
        dict(ok, kind=[0, 1, 1, 1]),                           # a sink inhibited by its own column
        dict(ok, j=[1, 1, 2, 2], kind=[0, 0, 0, 1]),           # a positive source limited by its own column
        dict(p=[0, 0], k=[0, 0], j=[1, 1], kind=[0, 0], half=[0.5, 0.7]),   # given twice
    ]
    for args in bad:
        assert call(**args) == CWR_EINVAL, args
        if args.get("n", 1) >= 0:
            with pytest.raises(ValueError):
                be.set_kinetics_limits(*[args.get(x) for x in ("p", "k", "j", "kind", "half")])
    be.set_kinetics(None)
    assert call(**ok) == CWR_EINVAL                           # kinetics switched off again
    be.close()


def heavy_boxes(dt=900.0, days=4.0, oxygen_yield=-1.0):
    """The closed boxes of test_kinetics_sources, heavily loaded: BOD from 40 to 400 mg/L, DO from O2sat(20); the decay
    takes -oxygen_yield of DO per unit (-4.57: nitrification)."""
    plan, mesh, inputs, kin, src, _, _ = _ts().closed_boxes(False, dt, days)
    n = plan.n_real
    L0s = np.linspace(40.0, 400.0, n)
    inputs[0, 0, :n] = L0s
    y = np.array(kin["yields"], np.float64)
    y[1, 0] = oxygen_yield
    kin = dict(kin, yields=y)
    src = dict(src, source_per_day=np.array([0.0, SOD]))
    lim = dict(process=np.array([0, 1], np.int32), column=np.array([0, 1], np.int32), factor_column=np.array([1, 1], np.int32),
               factor_kind=np.zeros(2, np.int32), half_saturation=np.array([K_BOD, K_SOD]))
    return plan, mesh, inputs, kin, src, lim, int(round(days * 86400.0 / dt))


@pytest.mark.gpu
@pytest.mark.parametrize("oxygen_yield", [-1.0, -4.57])
def test_do_stays_non_negative_on_a_heavily_loaded_mesh(oxygen_yield):
    """run() over 4 days at 900 s: the lowest DO over all steps and cells is >= -1e-12 O2sat (solver tolerance) with
    the factors, and clearly negative without them."""
    plan, mesh, inputs, kin, src, lim, steps = heavy_boxes(oxygen_yield=oxygen_yield)
    n = plan.n_real
    lowest = {}
    for limited in (True, False):
        be = limit_backend(mesh, inputs, kin, src, lim if limited else None)
        assert be.run(0, steps).status == 0
        lowest[limited] = min(float(be.get_state(1, t)[:n].min()) for t in range(steps + 1))
        if limited:
            oracle = limit_oracle(mesh, inputs, kin, src, lim)
            for _ in range(steps):
                oracle.update()
            _tk()._parity().close(be.get_state(1, steps)[:n], oracle.constituent_dict["c1"].concentration[steps][:n], 1e-8, "DO")
        be.close()
    assert lowest[True] >= -1e-12 * float(o2sat(20.0)), lowest
    assert lowest[False] < -1.0, lowest


def _gpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_domain_decomposition_with_limits():
    if _gpus() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29537", str(ROOT / "tools" / "dd_check.py"), "--side", "150", "--K", "4", "--steps", "5", "--kinetics"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=850, cwd=ROOT)
    lines = [json.loads(ln) for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert out.returncode == 0, (out.stdout[-3000:], out.stderr[-3000:])
    runs = [ln for ln in lines if ln.get("limits")]
    assert len(runs) >= 2 and all(ln["ok"] for ln in lines), lines
    for ln in runs:
        assert ln["max_rel_diff_vs_oracle"] < 1e-9 and ln["max_rel_diff_vs_single_gpu"] < 1e-9
        assert ln["reaction_mass_rel_diff"] < 1e-9
