"""Depth-scaled kinetics (cwr_set_kinetics_depth): settling velocities, areal sources and transfer velocities acting
through each cell's depth h = max(V[t] / A, min_depth).  The spec compiler and the numpy restatement
(oracle.kinetics_depth) on the CPU, the CUDA path against the restatement on the GPU (rtol 1e-9 per step, as
test_kinetics)."""
import ctypes as C
import json
import re
import shutil
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from oracle import kinetics_limits as limits
from oracle import reference_step as ref
from oracle.kinetics_depth import KineticsRiverine, depth, depth_terms, react
from oracle.kinetics_limits import limit_terms
from oracle.kinetics_sources import o2sat
from tests.helpers import same

ROOT = Path(__file__).resolve().parents[1]
RTOL = 1e-9
# a BOD-DO-T model given through the depth: settling BOD, areal SOD limited by DO, reaeration and heat exchange by
# transfer velocities (m/day on a plan in m)
SPEC = {"BOD": {"decay_per_day": 0.23, "theta": 1.047, "yields": {"DO": -1.0}, "limited_by": {"DO": 0.5}},
        "PBOD": {"settling_per_day": 0.4},
        "DO": {"areal_source_per_day": -1.5, "source_theta": 1.065, "source_limited_by": {"DO": 1.0},
               "transfer_per_day": 1.4, "exchange_theta": 1.024, "equilibrium": "oxygen_saturation"},
        "T": {"transfer_per_day": 0.6, "equilibrium": 18.0}}
NAMES = ["DO", "BOD", "PBOD", "T"]


# ------------------------------------------------------------------------------------------------------------------
# CPU: spec compiler and validation
# ------------------------------------------------------------------------------------------------------------------
def test_spec_compiles_the_depth_keys():
    from clearwater_riverine_b200.kinetics import DEFAULT_MIN_DEPTH, compile_kinetics
    area = np.full(6, 50.0)
    kin = compile_kinetics(SPEC, NAMES, "T", cell_area=area)
    assert kin.has_depth and kin.min_depth == DEFAULT_MIN_DEPTH
    assert kin.decay_per_depth.tolist() == [0, 0, 1, 0]
    assert kin.source_per_depth.tolist() == [1, 0, 0, 0]
    assert kin.exchange_per_depth.tolist() == [1, 0, 0, 1]
    assert all(kin.depth_arguments()[k].dtype == np.int32 for k in ("decay_per_depth", "source_per_depth", "exchange_per_depth"))
    assert kin.decay_per_day[2] == 0.4 and kin.source_per_day[0] == -1.5 and kin.exchange_per_day[3] == 0.6
    assert same(kin.depth_arguments()["cell_area"], area)
    plain = compile_kinetics({"BOD": {"decay_per_day": 0.35}}, ["DO", "BOD"], 20.0)
    assert not plain.has_depth and plain.decay_per_depth is None


def test_a_zero_per_depth_rate_sets_no_flag():
    from clearwater_riverine_b200.kinetics import compile_kinetics
    kin = compile_kinetics({"A": {"settling_per_day": 0.0}}, ["A"], 20.0)
    assert not kin.has_depth


def test_kinetics_built_without_the_new_fields_has_no_depth():
    from clearwater_riverine_b200.kinetics import Kinetics
    kin = Kinetics(np.zeros(2), np.ones(2), np.zeros((2, 2)), -1, 20.0, (0, 1))
    assert not kin.has_depth and kin.depth_arguments()["decay_per_depth"] is None


INVALID = {
    "settling and decay": {"A": {"settling_per_day": 1.0, "decay_per_day": 1.0}},
    "areal and volumetric source": {"A": {"areal_source_per_day": 1.0, "source_per_day": 1.0}},
    "transfer and exchange": {"A": {"transfer_per_day": 1.0, "exchange_per_day": 1.0, "equilibrium": 2.0}},
    "transfer without equilibrium": {"A": {"transfer_per_day": 1.0}},
    "negative settling": {"A": {"settling_per_day": -1.0}},
    "negative transfer": {"A": {"transfer_per_day": -1.0, "equilibrium": 2.0}},
}


@pytest.mark.parametrize("case", sorted(INVALID))
def test_invalid_depth_specs_are_rejected_naming_the_constituent(case):
    from clearwater_riverine_b200.kinetics import compile_kinetics
    with pytest.raises(ValueError, match="'A'"):
        compile_kinetics(INVALID[case], ["A", "B"], 20.0, cell_area=np.ones(3))


def test_a_depth_key_without_a_cell_area_is_an_error():
    from clearwater_riverine_b200.kinetics import compile_kinetics
    with pytest.raises(ValueError, match="'A'.*cell_area"):
        compile_kinetics({"A": {"settling_per_day": 1.0}}, ["A", "B"], 20.0)


def test_validate_rejects_every_abi_condition():
    from clearwater_riverine_b200.kinetics import validate
    d, th, y = np.array([1.0, 0.0, 0.0]), np.ones(3), np.zeros((3, 3))
    s, e = np.array([0.0, -1.0, 0.0]), np.array([0.0, 0.0, 2.0])
    area = np.array([1.0, 2.0, 3.0, 4.0])
    base = dict(source_per_day=s, exchange_per_day=e, equilibrium=np.zeros(3))
    ok = dict(decay_per_depth=[1, 0, 0], source_per_depth=[0, 1, 0], exchange_per_depth=[0, 0, 1], cell_area=area,
              min_depth=0.1)
    validate(d, th, y, -1, 20.0, ("A", "B", "C"), **base, **ok)
    validate(d, th, y, -1, 20.0, ("A", "B", "C"), **base, decay_per_depth=[0, 0, 0])     # all zero: off, no area needed
    bad = {"0 or 1": dict(ok, decay_per_depth=[2, 0, 0]), "'A'.*0 or 1": dict(ok, decay_per_depth=[-1, 0, 0]),
           "'B'.*rate is 0": dict(ok, decay_per_depth=[1, 1, 0]), "'A'.*rate is 0": dict(ok, source_per_depth=[1, 1, 0]),
           "'B'.*rate is 0 ": dict(ok, exchange_per_depth=[0, 1, 1]), "'A'.*cell_area": dict(ok, cell_area=None),
           "min_depth": dict(ok, min_depth=0.0), "min_depth ": dict(ok, min_depth=float("nan")),
           "areas": dict(ok, cell_area=np.array([1.0, 0.0, 3.0])), "areas ": dict(ok, cell_area=np.array([1.0, np.inf])),
           "areas  ": dict(ok, cell_area=np.array([-1.0]))}
    for what, args in bad.items():
        with pytest.raises(ValueError, match=what.strip()):
            validate(d, th, y, -1, 20.0, ("A", "B", "C"), **base, **args)


# ------------------------------------------------------------------------------------------------------------------
# CPU: the numpy restatement
# ------------------------------------------------------------------------------------------------------------------
def network(seed=2, n=40):
    """The synthetic 6-constituent network with sources, factors and depth flags on n cells, and depths h."""
    from clearwater_riverine_b200 import synthetic
    plan = synthetic.make_plan(10, 4, 2, seed=seed, dry_fraction=0.05)
    inputs, kin = synthetic.make_kinetics(synthetic.make_inputs(plan, 6, seed=seed), seed=seed)
    src = synthetic.make_kinetics_sources(kin, seed=seed)
    lim = synthetic.make_kinetics_limits(kin, src, seed=seed)
    kin, src, flags = synthetic.make_kinetics_depth(kin, src, seed=seed)
    n = plan.n_real
    h = depth(plan.volume[0, :n], plan.cell_area[:n], 0.05)
    return inputs[:, 0, :n], kin, src, lim, flags, h


def react_all(c, dt, kin, src, lim, flags, h):
    return react(c, dt, kin["decay_per_day"], kin["theta"], kin["yields"], kin["temperature_k"], True, **src,
                 **limit_terms(**lim), **flags, h=h)


def test_without_flags_it_is_bitwise_the_limits_restatement():
    c, kin, src, lim, flags, h = network()
    want = limits.react(c, 900.0, kin["decay_per_day"], kin["theta"], kin["yields"], kin["temperature_k"], True, **src,
                        **limit_terms(**lim))
    zero = {k: np.zeros_like(v) for k, v in flags.items()}
    assert same(react_all(c, 900.0, kin, src, lim, zero, h), want)
    assert same(react_all(c, 900.0, kin, src, lim, {}, None), want)
    assert not same(react_all(c, 900.0, kin, src, lim, flags, h), want)


def test_settling_in_a_closed_box_is_the_exponential_of_the_depth():
    """c0 exp(-v_s t / h) per step, at three depths (the per-step solution is exact: only rounding differs)."""
    h = np.array([0.5, 2.0, 7.5])
    c = np.array([[10.0, 10.0, 10.0]])
    vs, dt = 3.0, 3600.0
    c0 = c.copy()
    for step in range(1, 25):
        c = react(c, dt, [vs], decay_per_depth=[1], h=h)
        want = c0[0] * np.exp(-vs / 86400.0 / h * dt * step)
        assert np.abs(c[0] - want).max() <= 1e-13 * c0.max(), step


def test_areal_rates_at_a_uniform_depth_are_the_volumetric_ones():
    """make_kinetics_depth multiplies every flagged rate by H = 2: at depth H everywhere the flagged network is the
    volumetric one to rounding, and at another depth it is not."""
    c, kin, src, lim, flags, _ = network()
    H = 2.0
    per_h = lambda a, f: np.where(flags[f] == 1, a / H, a)
    vkin = dict(kin, decay_per_day=per_h(kin["decay_per_day"], "decay_per_depth"))
    vsrc = dict(src, source_per_day=per_h(src["source_per_day"], "source_per_depth"),
                exchange_per_day=per_h(src["exchange_per_day"], "exchange_per_depth"))
    want = react_all(c, 900.0, vkin, vsrc, lim, {}, None)
    got = react_all(c, 900.0, kin, src, lim, flags, np.full(c.shape[1], H))
    scale = np.abs(want).max(axis=1, keepdims=True)
    assert (np.abs(got - want) <= 1e-12 * scale).all()
    other = react_all(c, 900.0, kin, src, lim, flags, np.full(c.shape[1], 0.5))
    assert (np.abs(other - want) > 1e-6 * scale).any()


def test_the_depth_follows_the_volume_of_the_step():
    vol = np.array([[2.0, 10.0, 0.0], [4.0, 5.0, 0.0]], np.float32)
    area = np.array([1.0, 5.0, 3.0])
    assert same(depth(vol[0], area, 0.1), np.array([2.0, 2.0, 0.1]))
    assert same(depth(vol[1], area, 0.1), np.array([4.0, 1.0, 0.1]))


def test_dry_cells_take_min_depth_and_stay_finite():
    c, kin, src, lim, flags, _ = network()
    h = np.full(c.shape[1], 1e-3)
    out = react_all(c, 86400.0, kin, src, lim, flags, h)
    assert np.isfinite(out).all()
    h_dry = depth(np.zeros(c.shape[1], np.float32), np.full(c.shape[1], 100.0), 1e-3)
    assert same(h_dry, h)


@pytest.mark.parametrize("dt", [900.0, 86400.0])
def test_a_do_limited_areal_sod_keeps_do_non_negative_at_min_depth(dt):
    """DO from 0 to 12 mg/L, an areal SOD of 1.5 g/m2/day limited by DO itself, h = min_depth = 1 cm: a volumetric rate
    of 150 mg/L/day.  With a day's step DO stays >= 0; BOD oxidation limited by DO is capped by what is there."""
    n = 25
    c = np.vstack([np.linspace(0.0, 12.0, n), np.linspace(0.0, 300.0, n)])     # DO, BOD
    h = np.full(n, 0.01)
    y = np.array([[0.0, -1.0], [0.0, 0.0]])
    for _ in range(int(round(5 * 86400.0 / dt))):
        c = react(c, dt, [0.0, 0.5], None, y, 20.0, source_per_day=[-1.5, 0.0], exchange_per_day=[2.0, 0.0],
                  equilibrium=[0.0, 0.0], equilibrium_kind=[1, 0], **limit_terms([1, 0], [0, 1], [0, 0], [0, 0], [1.0, 0.5]),
                  source_per_depth=[1, 0], exchange_per_depth=[1, 0], h=h)
        assert (c >= 0.0).all(), c.min()
    assert c[0].max() < float(o2sat(20.0))


def write_plan_with_area(path, g: dict):
    """tests.ras_fixture.write_plan, with g["cell_area"] (when present) written as the 2D flow area's geometry dataset
    "Cells Surface Area", f32 as HEC-RAS stores it.  The fixture's tree is extended just before it is written."""
    from tests import ras_fixture
    if g.get("cell_area") is None:
        return ras_fixture.write_plan(path, g)
    real = ras_fixture._Writer.write

    def write(self, p, tree):
        areas = tree["Geometry"]["2D Flow Areas"]
        name = next(k for k in areas if k != "Attributes")
        areas[name]["Cells Surface Area"] = (np.asarray(g["cell_area"], "<f4"), None)
        return real(self, p, tree)

    ras_fixture._Writer.write = write
    try:
        return ras_fixture.write_plan(path, g)
    finally:
        ras_fixture._Writer.write = real


def test_the_reader_round_trips_the_cell_area(tmp_path):
    from clearwater_riverine_b200.io import ras
    from tests.helpers import load_golden
    g = dict(load_golden("p01_random_two"))
    write_plan_with_area(tmp_path / "plain.hdf", g)
    assert ras.read_ras_plan(tmp_path / "plain.hdf").cell_area is None
    F = len(g["face_x"])
    g["cell_area"] = np.linspace(10.0, 200.0, F).astype(np.float32)
    write_plan_with_area(tmp_path / "area.hdf", g)
    plan = ras.read_ras_plan(tmp_path / "area.hdf")
    assert plan.cell_area.dtype == np.float64 and same(plan.cell_area, g["cell_area"].astype(np.float64))


def test_synthetic_cell_area_leaves_every_other_array_as_it_was():
    from clearwater_riverine_b200 import synthetic
    plan = synthetic.make_plan(12, 9, 4, seed=5, dry_fraction=0.05)
    n = plan.n_real
    assert plan.cell_area.shape == (plan.n_face,) and (plan.cell_area > 0).all()
    wet = plan.volume[0, :n] > 0
    h = plan.volume[0, :n][wet] / plan.cell_area[:n][wet]
    assert np.abs(h - 2.0).max() < 0.5                    # the default depth of make_plan
    assert set(np.unique(plan.cell_area[:n])) == {50.0, 100.0}


def _ptxas(src: Path, out: Path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(nvcc).is_file():
        pytest.skip("nvcc not found")
    return subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas=-v", "-c",
                           "-o", str(out), str(src)], capture_output=True, text=True, timeout=600)


def test_every_k_react_instantiation_is_free_of_spills(tmp_path):
    """The three instantiations compile for sm_100a with no local memory; k_react<false> keeps 48 registers."""
    src = tmp_path / "k_react.cu"
    src.write_text(f'#include "{ROOT / "clearwater_riverine_b200" / "csrc" / "cwr_kernels.cuh"}"\n'
                   "using namespace cwr;\n"
                   "#define KR(a, b) template __global__ void cwr::k_react<a, b>(DeviceModel, const KinStep*, int, "
                   "const KinYield*, int, double, const KinSrc*, int, int, const KinFac*, const int*, double*, KinState*, "
                   "int, const double*, const int*, double);\n"
                   "KR(false, false)\nKR(true, false)\nKR(true, true)\n")
    res = _ptxas(src, tmp_path / "k_react.o")
    assert res.returncode == 0, res.stderr[-3000:]
    props = re.findall(r"Function properties for (_ZN3cwr7k_reactILb(\d)ELb(\d)\S*)\n\s*(\d+) bytes stack frame, (\d+) bytes "
                       r"spill stores, (\d+) bytes spill loads\n.*?Used (\d+) registers", res.stdout + res.stderr, re.S)
    got = {(a, b): (int(f), int(s), int(l), int(r)) for _, a, b, f, s, l, r in props}
    assert set(got) == {("0", "0"), ("1", "0"), ("1", "1")}, got
    assert all(v[:3] == (0, 0, 0) for v in got.values()), got
    assert got[("0", "0")][3] == 48, got


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def _tk():
    from tests import test_kinetics as tk
    return tk


def _ts():
    from tests import test_kinetics_sources as ts
    return ts


def depth_backend(mesh, inputs, kin, src, lim, dep, **opt):
    be = _ts().source_backend(mesh, inputs, kin, src, **opt)
    if lim is not None:
        be.set_kinetics_limits(**lim)
    if dep is not None:
        be.set_kinetics_depth(**dep)
    return be


def depth_oracle(mesh, inputs, kin, src, lim, dep):
    temperature = f"c{kin['temperature_k']}" if kin["temperature_k"] >= 0 else kin["temperature_c"]
    return KineticsRiverine(mesh, {f"c{k}": inputs[k] for k in range(len(inputs))}, kin["decay_per_day"], kin["theta"],
                            kin["yields"], temperature, **(src or {}), **limit_terms(**(lim or {})), **depth_terms(**(dep or {})))


def run_depth_parity(mesh, inputs, kin, src, lim, dep, steps, check_flux=True, **opt):
    tp, tk = _tk()._parity(), _tk()
    K = len(inputs)
    be = depth_backend(mesh, inputs, kin, src, lim, dep, **opt)
    oracle = depth_oracle(mesh, inputs, kin, src, lim, dep)
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


def varied_area(plan, seed):
    """The synthetic plan areas times a seeded factor in [0.25, 4]: depths that vary several-fold across the mesh."""
    rng = np.random.default_rng(seed + 5)
    return plan.cell_area * np.exp(rng.uniform(np.log(0.25), np.log(4.0), plan.n_face))


def synthetic_network(nx, ny, T, K, seed, limits_too=True, **kw):
    from clearwater_riverine_b200 import synthetic
    plan, mesh, inputs = _tk()._parity().synthetic_case(nx, ny, T, K, seed=seed, **kw)
    inputs, kin = synthetic.make_kinetics(inputs, seed=seed)
    src = synthetic.make_kinetics_sources(kin, seed=seed)
    if K == 1:
        src = dict(src, source_per_day=-np.abs(src["source_per_day"]))
    lim = synthetic.make_kinetics_limits(kin, src, seed=seed) if limits_too else None
    kin, src, flags = synthetic.make_kinetics_depth(kin, src, seed=seed)
    if not any(f.any() for f in flags.values()):
        flags["decay_per_depth"][0] = 1
    dep = dict(cell_area=varied_area(plan, seed), min_depth=0.05, **flags)
    return plan, mesh, inputs, kin, src, lim, dep


@pytest.mark.gpu
@pytest.mark.parametrize("solver", [1, 2])
@pytest.mark.parametrize("K", [1, 3, 16, 18, 33])
def test_synthetic_meshes_on_the_large_path(K, solver):
    _, mesh, inputs, kin, src, lim, dep = synthetic_network(40, 25, 8, K, seed=K + 150, dry_fraction=0.02)
    be, _ = run_depth_parity(mesh, inputs, kin, src, lim, dep, 7, solver_path=1, solver=solver)
    be.close()


@pytest.mark.gpu
def test_large_path_without_factors():
    _, mesh, inputs, kin, src, _, dep = synthetic_network(40, 25, 6, 6, seed=157, limits_too=False, dry_fraction=0.02)
    be, _ = run_depth_parity(mesh, inputs, kin, src, None, dep, 5, solver_path=1)
    be.close()


@pytest.mark.gpu
def test_small_path_parity():
    _, mesh, inputs, kin, src, lim, dep = synthetic_network(40, 25, 7, 5, seed=161, dry_fraction=0.02)
    be, _ = run_depth_parity(mesh, inputs, kin, src, lim, dep, 6, solver_path=2, precond_sweep=0)
    assert be.options.solver_path == 2
    be.close()


@pytest.mark.gpu
def test_every_column_count_up_to_kmax():
    from clearwater_riverine_b200 import synthetic
    plan, mesh, base = _tk()._parity().synthetic_case(12, 9, 3, 128, seed=191)
    area = varied_area(plan, 191)
    for K in range(1, 129):
        inputs, kin = synthetic.make_kinetics(base[:K], seed=K)
        src = synthetic.make_kinetics_sources(kin, seed=K)
        if K == 1:
            src = dict(src, source_per_day=-np.abs(src["source_per_day"]))
        lim = synthetic.make_kinetics_limits(kin, src, seed=K) if K % 2 else None
        kin, src, flags = synthetic.make_kinetics_depth(kin, src, seed=K)
        dep = dict(cell_area=area, min_depth=0.05, **flags)
        for solver_path in (1, 2):
            be, _ = run_depth_parity(mesh, inputs, kin, src, lim, dep, 1, check_flux=False, solver_path=solver_path)
            be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 64])
def test_on_chip_path_on_the_ohio_shaped_mesh(K):
    """K = 1: DO with an areal self-limited SOD and reaeration by a transfer velocity; K = 64: 64 scenarios of it."""
    from clearwater_riverine_b200 import synthetic
    plan = synthetic.ohio_like(7, seed=2)
    D = 0.1
    adv, _, _, cdiff, dt = ref.derive_coefficients(plan.face_flow, plan.edge_velocity, plan.face_x, plan.face_y, plan.f1, plan.f2,
                                                   D, plan.time_seconds)
    mesh = ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, plan.edge_velocity, plan.volume, dt, D)
    inputs = synthetic.make_inputs(plan, K, seed=7, ic_range=(0.0, 15.0))
    kin = dict(decay_per_day=np.full(K, 2.0), theta=np.full(K, 1.047), yields=None, temperature_k=-1, temperature_c=17.0)
    src = dict(source_per_day=np.full(K, -900.0), source_theta=np.full(K, 1.065), exchange_per_day=np.linspace(0.6, 36.0, K),
               exchange_theta=np.full(K, 1.024), equilibrium=np.zeros(K), equilibrium_kind=np.ones(K, np.int32))
    ks = np.arange(K, dtype=np.int32)
    lim = dict(process=np.ones(K, np.int32), column=ks, factor_column=ks, factor_kind=np.zeros(K, np.int32),
               half_saturation=np.linspace(0.2, 5.0, K))
    dep = dict(cell_area=varied_area(plan, 3), min_depth=0.05, decay_per_depth=(ks % 2).astype(np.int32),
               source_per_depth=np.ones(K, np.int32), exchange_per_depth=(ks % 3 != 1).astype(np.int32))
    be, _ = run_depth_parity(mesh, inputs, kin, src, lim, dep, 6, check_flux=K == 1)
    assert be.options.solver_path in (3, 4)
    be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("temperature_k", [-1, 15])
def test_both_temperature_modes(temperature_k):
    _, mesh, inputs, kin, src, lim, dep = synthetic_network(40, 25, 6, 16, seed=166, dry_fraction=0.02)
    kin = dict(kin, temperature_k=temperature_k, temperature_c=21.0)
    be, _ = run_depth_parity(mesh, inputs, kin, src, lim, dep, 5, solver_path=1)
    be.close()


@pytest.mark.gpu
@pytest.mark.parametrize("temperature_k", [-1, 3])
@pytest.mark.parametrize("solver_path", [1, 2])
def test_no_flags_are_bitwise_the_run_without_the_depth_call(solver_path, temperature_k):
    """An area with all flags 0; flags cleared by set_kinetics_depth with none; by a new set_kinetics_sources; by a new
    set_kinetics: the same bits, launches and reaction mass as the run that never made the depth call."""
    plan, mesh, inputs, kin, src, lim, dep = synthetic_network(40, 25, 7, 4, seed=171, dry_fraction=0.02)
    kin = dict(kin, temperature_k=temperature_k)
    zero = dict(dep, **{k: np.zeros(4, np.int32) for k in ("decay_per_depth", "source_per_depth", "exchange_per_depth")})
    plain = depth_backend(mesh, inputs, kin, src, lim, None, solver_path=solver_path)
    cases = [depth_backend(mesh, inputs, kin, src, lim, zero, solver_path=solver_path)]
    for how in ("off", "sources", "kinetics"):
        be = depth_backend(mesh, inputs, kin, src, lim, dep, solver_path=solver_path)
        if how == "off":
            be.set_kinetics_depth(None)
        elif how == "sources":
            be.set_kinetics_sources(**src)
            be.set_kinetics_limits(**lim)
        else:
            be.set_kinetics(**kin)
            be.set_kinetics_sources(**src)
            be.set_kinetics_limits(**lim)
        cases.append(be)
    flagged = depth_backend(mesh, inputs, kin, src, lim, dep, solver_path=solver_path)
    for t in range(6):
        a = plain.step(t)
        flagged.step(t)
        for be in cases:
            assert be.step(t).n_launches == a.n_launches
            assert same(plain.get_state_all(t + 1), be.get_state_all(t + 1))
            for k in range(4):
                assert all(same(x, y) for x, y in zip(plain.get_mass_flux(k, t), be.get_mass_flux(k, t)))
    assert not same(plain.get_state_all(6), flagged.get_state_all(6))     # the flags do act on this network
    for be in cases:
        assert all(be.reaction_mass(k) == plain.reaction_mass(k) for k in range(4))
    for be in [plain, flagged] + cases:
        be.close()


@pytest.mark.gpu
def test_limits_after_depth_keep_the_depth():
    """cwr_set_kinetics_limits and cwr_set_kinetics_depth do not clear each other: either order, the same bits."""
    _, mesh, inputs, kin, src, lim, dep = synthetic_network(30, 20, 5, 5, seed=175, dry_fraction=0.02)
    a = depth_backend(mesh, inputs, kin, src, lim, dep)
    b = depth_backend(mesh, inputs, kin, src, None, dep)
    b.set_kinetics_limits(**lim)
    for t in range(4):
        a.step(t); b.step(t)
    assert same(a.get_state_all(4), b.get_state_all(4))
    a.close(); b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("solver_path", [1, 2])
def test_run_is_bitwise_step_by_step_and_repeatable(solver_path):
    _, mesh, inputs, kin, src, lim, dep = synthetic_network(30, 20, 10, 5, seed=181, dry_fraction=0.02)
    outs = []
    for mode in ("step", "run", "run"):
        be = depth_backend(mesh, inputs, kin, src, lim, dep, solver_path=solver_path)
        if mode == "step":
            for t in range(9):
                assert be.step(t).status == 0
        else:
            assert be.run(0, 9).status == 0
        outs.append((np.stack([be.get_state_all(t) for t in range(1, 10)]), [be.reaction_mass(k) for k in range(5)]))
        be.close()
    for states, masses in outs[1:]:
        assert same(states, outs[0][0]) and masses == outs[0][1]
    oracle = depth_oracle(mesh, inputs, kin, src, lim, dep)
    for _ in range(9):
        oracle.update()
    for k in range(5):
        _tk()._parity().close(outs[1][0][-1][k], oracle.constituent_dict[f"c{k}"].concentration[9][:mesh.n], RTOL, f"run k{k}")


@pytest.mark.gpu
def test_reaction_mass_counts_the_depth_processes_once_under_the_defect_correction_fallback():
    from clearwater_riverine_b200 import synthetic
    plan = synthetic.make_plan(60, 50, 6, seed=41, dry_fraction=0.02)
    vel = plan.edge_velocity.copy()
    vel[:, np.random.default_rng(1).random(plan.n_edge) < 0.05] *= -1
    D = 2.0
    adv, _, _, cdiff, dt = ref.derive_coefficients(plan.face_flow, vel, plan.face_x, plan.face_y, plan.f1, plan.f2, D, plan.time_seconds)
    mesh = ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, vel, plan.volume, dt, D)
    inputs = synthetic.make_inputs(plan, 3, seed=41)
    inputs, kin = synthetic.make_kinetics(inputs, seed=41)
    src = synthetic.make_kinetics_sources(kin, seed=41)
    lim = synthetic.make_kinetics_limits(kin, src, seed=41)
    kin, src, flags = synthetic.make_kinetics_depth(kin, src, seed=41)
    dep = dict(cell_area=varied_area(plan, 41), min_depth=0.05, **flags)
    tp, tk = _tk()._parity(), _tk()
    be = depth_backend(mesh, inputs, kin, src, lim, dep, solver_path=1, solver=2)
    oracle = depth_oracle(mesh, inputs, kin, src, lim, dep)
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
    out = {}
    for name, block in SPEC.items():
        b = dict(block)
        for key in ("decay_per_day", "areal_source_per_day", "transfer_per_day", "settling_per_day"):
            if key in b:
                b[key] = b[key] * f
        out[name] = b
    return out


@pytest.mark.gpu
def test_mass_balance_closes_with_depth():
    from clearwater_riverine_b200 import ClearwaterRiverine
    from clearwater_riverine_b200.kinetics import compile_kinetics
    tp = _tk()._parity()
    plan, mesh, inputs = tp.synthetic_case(20, 14, 8, 4, seed=4, dry_fraction=0.02)
    inputs[3] = np.where(inputs[3] != 0, 10.0 + 0.2 * inputs[3], 0.0)
    inputs[0] = 0.1 * inputs[0]
    spec = _scaled_spec(300.0)
    area = varied_area(plan, 4)
    arrays = (plan.f1, plan.f2, plan.face_x, plan.face_y, plan.time_seconds, plan.face_flow, plan.edge_velocity, plan.volume, 0.1)
    model = ClearwaterRiverine.from_arrays(*arrays, dict(zip(NAMES, inputs)), kinetics=spec, temperature="T",
                                           cell_area=area, min_depth=0.05)
    assert model.kinetics.has_depth and model.kinetics.has_limits
    kin = compile_kinetics(spec, NAMES, "T", cell_area=area, min_depth=0.05)
    oracle = KineticsRiverine(mesh, dict(zip(NAMES, inputs)), kin.decay_per_day, kin.theta, kin.yields, "T",
                              **kin.sources_arguments(), **limit_terms(**kin.limits_arguments()),
                              **depth_terms(**kin.depth_arguments()))
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
def test_yaml_config_with_depth_keys_is_bitwise_from_arrays(tmp_path):
    yaml = pytest.importorskip("yaml")
    import pandas as pd
    from clearwater_riverine_b200 import ClearwaterRiverine
    from clearwater_riverine_b200.io import ras
    from tests.helpers import load_golden
    g = dict(load_golden("p01_random_two"))
    F = len(g["face_x"])
    g["cell_area"] = np.linspace(0.5, 3.0, F).astype(np.float32) * float(np.median(g["volume"][0]))
    hdf = tmp_path / "plan.hdf"
    times = write_plan_with_area(hdf, g)
    plan = ras.read_ras_plan(hdf)
    n = plan.nreal + 1
    lines = sorted({str(x) for x in g["bc_names"]})
    cons = {}
    for name, ic, bc in (("DO", 0.5, 8.0), ("BOD", 8.0, 5.0), ("PBOD", 2.0, 1.0), ("T", 18.0, 21.0)):
        icf, bcf = tmp_path / f"{name}_ic.csv", tmp_path / f"{name}_bc.csv"
        pd.DataFrame({"Cell_Index": np.arange(n), "Concentration": ic + 0.01 * np.arange(n)}).to_csv(icf, index=False)
        pd.DataFrame({"Datetime": np.repeat([times[0], times[-1]], len(lines)), "RAS2D_TS_Name": lines * 2,
                      "Concentration": bc}).to_csv(bcf, index=False)
        cons[name] = {"initial_conditions": str(icf), "boundary_conditions": str(bcf), "units": "mg/L"}
    spec = _scaled_spec(2000.0)
    cfg = {"diffusion_coefficient": 0.1, "flow_field_filepath": str(hdf), "temperature": "T", "min_depth": 0.2,
           "constituents": {name: dict(c, kinetics=spec[name]) for name, c in cons.items()}}
    cfg_path = tmp_path / "model.yml"
    cfg_path.write_text(yaml.safe_dump(cfg))
    a = ClearwaterRiverine(config_filepath=str(cfg_path))
    inputs = {name: ras.build_input_array(len(plan.time), len(plan.face_x), plan.time, plan.f2, plan.boundary_data,
                                          c["initial_conditions"], c["boundary_conditions"]) for name, c in cons.items()}
    b = ClearwaterRiverine.from_arrays(plan.f1, plan.f2, plan.face_x, plan.face_y, plan.time_seconds, plan.face_flow,
                                       plan.edge_velocity, plan.volume, 0.1, inputs, cell_area=plan.cell_area, min_depth=0.2)
    b.set_kinetics(spec, temperature="T")
    for _ in range(12):
        a.update(); b.update()
    for name in cons:
        assert same(a.mesh[name][:13], b.mesh[name][:13]), name
        assert a.backend.reaction_mass(a._index[name]) == b.backend.reaction_mass(b._index[name])
    assert a.kinetics.has_depth and a.min_depth == 0.2
    a.finalize(); b.finalize()


@pytest.mark.gpu
def test_invalid_depth_straight_to_the_abi_return_einval():
    from clearwater_riverine_b200.backend import CWR_EINVAL
    plan, mesh, inputs = _tk()._parity().synthetic_case(12, 9, 4, 3, seed=2)
    be = _tk()._parity().make_backend(mesh, list(inputs))
    lib = be._lib
    F = plan.n_face

    def call(area=None, min_depth=0.1, d=None, s=None, e=None):
        a = None if area is None else np.ascontiguousarray(area, np.float64)
        fl = [None if x is None else np.ascontiguousarray(x, np.int32) for x in (d, s, e)]
        return lib.cwr_set_kinetics_depth(be._h, None if a is None else a.ctypes.data_as(C.POINTER(C.c_double)), float(min_depth),
                                          *[None if x is None else x.ctypes.data_as(C.POINTER(C.c_int32)) for x in fl])

    ok = dict(area=plan.cell_area, d=[1, 0, 0], s=[0, 1, 0], e=[0, 0, 1])
    assert call(**ok) == CWR_EINVAL                           # kinetics not set
    be.set_kinetics(np.array([1.0, 0.0, 0.0]), None, None, -1, 20.0)
    be.set_kinetics_sources(np.array([0.0, -1.0, 0.0]), None, np.array([0.0, 0.0, 2.0]), None, np.array([0.0, 0.0, 5.0]))
    assert call(**ok) == 0 and call() == 0 and call(d=[0, 0, 0]) == 0 and call(min_depth=-1.0, d=[0, 0, 0]) == 0
    ghost_nan = plan.cell_area.copy()
    ghost_nan[plan.n_real:] = np.nan                          # ghost cells are not read
    assert call(**dict(ok, area=ghost_nan)) == 0
    bad_area = plan.cell_area.copy()
    bad_area[3] = 0.0
    bad = [dict(ok, d=[2, 0, 0]), dict(ok, s=[0, -1, 0]), dict(ok, d=[0, 1, 0]), dict(ok, s=[1, 1, 0]), dict(ok, e=[0, 1, 1]),
           dict(ok, area=None), dict(ok, area=bad_area), dict(ok, area=np.where(np.arange(F) == 5, np.inf, plan.cell_area)),
           dict(ok, min_depth=0.0), dict(ok, min_depth=np.nan), dict(ok, min_depth=np.inf)]
    for args in bad:
        assert call(**args) == CWR_EINVAL, args
    be.set_kinetics(None)
    assert call(**ok) == CWR_EINVAL                           # kinetics switched off again
    be.close()


@pytest.mark.gpu
def test_do_stays_non_negative_with_an_areal_sod_at_min_depth():
    """Closed boxes, one of them dry-shallow (h = min_depth = 1 cm), an areal SOD limited by DO and BOD oxidation limited
    by DO, dt = 1 day: the lowest DO is >= -1e-12 O2sat (solver tolerance)."""
    plan, mesh, inputs, kin, src, _, _ = _ts().closed_boxes(False, 86400.0, 5.0)
    n = plan.n_real
    area = plan.cell_area.copy()
    area[: n // 2] = plan.volume[0, : n // 2] / 0.005            # h = 0.5 cm -> min_depth
    src = dict(src, source_per_day=np.array([0.0, -1.5]))
    lim = dict(process=np.array([0, 1], np.int32), column=np.array([0, 1], np.int32), factor_column=np.array([1, 1], np.int32),
               factor_kind=np.zeros(2, np.int32), half_saturation=np.array([0.5, 1.0]))
    dep = dict(cell_area=area, min_depth=0.01, decay_per_depth=None, source_per_depth=np.array([0, 1], np.int32),
               exchange_per_depth=np.array([0, 1], np.int32))
    be = depth_backend(mesh, inputs, kin, src, lim, dep)
    assert be.run(0, 5).status == 0
    lowest = min(float(be.get_state(1, t)[:n].min()) for t in range(6))
    oracle = depth_oracle(mesh, inputs, kin, src, lim, dep)
    for _ in range(5):
        oracle.update()
    _tk()._parity().close(be.get_state(1, 5)[:n], oracle.constituent_dict["c1"].concentration[5][:n], 1e-8, "DO")
    be.close()
    assert lowest >= -1e-12 * float(o2sat(20.0)), lowest


def _gpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_domain_decomposition_with_depth():
    if _gpus() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29539", str(ROOT / "tools" / "dd_check.py"), "--side", "150", "--K", "4", "--steps", "5", "--kinetics"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=850, cwd=ROOT)
    lines = [json.loads(ln) for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert out.returncode == 0, (out.stdout[-3000:], out.stderr[-3000:])
    runs = [ln for ln in lines if ln.get("depth")]
    assert len(runs) >= 2 and all(ln["ok"] for ln in lines), lines
    for ln in runs:
        assert ln["max_rel_diff_vs_oracle"] < 1e-9 and ln["max_rel_diff_vs_single_gpu"] < 1e-9
        assert ln["reaction_mass_rel_diff"] < 1e-9
