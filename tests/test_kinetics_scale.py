"""k_react at the sizes it runs at.  Every other kinetics test runs on at most 3,000 cells, where each CTA of k_react
takes one tile: here every CTA of the resident grid takes two or more, so the tile loop, the column sums carried across
tiles, the reloads of the tile's volumes and diagonal and the grid-wide reaction-mass sum run at full grid, for every
instantiation, with state slots on odd and even doubles.  An spsolve per column is out of reach at these sizes, so each
reacted step is checked where the kinetics acts: the right-hand sides and the reaction mass against the oracle's from the
device's own c[t] (reacted_step, pinned bitwise to oracle.kinetics_depth.KineticsRiverine.update on the CPU), and the
solve by its true residual with the oracle's matrix."""
import re
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import reference_step as ref
from oracle.kinetics_depth import KineticsRiverine, depth, depth_terms, react
from oracle.kinetics_limits import limit_terms
from tests.helpers import same
from tests.test_kinetics import kinetic_backend, mass_scale
from tests.test_kinetics_depth import depth_backend, depth_oracle, synthetic_network
from tests.test_gpu_parity import RTOL, close

ROOT = Path(__file__).resolve().parents[1]
K_MAX, THREADS = 128, 256          # kMaxK, kThreads (cwr_kernels.cuh)


def react_tile_rows(K):
    """react_tile_rows(K) of cwr_kernels.cuh: the rows of k_react's tile, the largest multiple of 32 (at most 256) whose
    R x (K + 3) doubles fit in 48 KB beside st[kMaxK] (32-byte KinStep) + 64 bytes, fac[kMaxK] and red[kThreads]."""
    free = 48 * 1024 - (32 * K_MAX + 64) - (K_MAX + THREADS) * 8
    rows = free // ((K + 3) * 8)
    return THREADS if rows >= THREADS else rows // 32 * 32


def oracle_network(kin, src=None, lim=None, dep=None):
    """The keyword arguments of oracle.kinetics_depth.KineticsRiverine after (mesh, inputs), for the arguments of
    set_kinetics, set_kinetics_sources, set_kinetics_limits and set_kinetics_depth (None: that call not made), with the
    constituents named c0, c1, ..."""
    temperature = f"c{kin['temperature_k']}" if kin["temperature_k"] >= 0 else kin["temperature_c"]
    return dict(decay_per_day=kin["decay_per_day"], theta=kin["theta"], yields=kin["yields"], temperature=temperature,
                **(src or {}), **limit_terms(**(lim or {})), **depth_terms(**(dep or {})))


def reacted_step(mesh, inputs, c_t, t, decay_per_day, theta=None, yields=None, temperature=None, cell_area=None,
                 min_depth=0.01, **terms):
    """What oracle.kinetics_depth.KineticsRiverine.update does before its solve, from the given c[t] (K, >= n) rather
    than its own: the inputs of step t merged into the real cells, the depth of step t, react, the reaction mass
    sum vol (c~' - c~) per column and the right-hand sides from c~'.  The network: the keyword arguments of
    KineticsRiverine (oracle_network).
    Returns (b (K, n), b of the unreacted c~ to rounding (K, n), reaction mass (K,), sum |vol (c~' - c~)| (K,))."""
    n, K = mesh.n, len(inputs)
    names = [f"c{k}" for k in range(K)]
    merged = np.empty((K, n))
    for k in range(K):
        solver = np.zeros(mesh.n_face)
        solver[0:n] = c_t[k][0:n]
        nz = inputs[k][t].nonzero()
        solver[nz] = inputs[k][t][nz]
        merged[k] = solver[0:n]
    is_index = isinstance(temperature, str)
    temp = names.index(temperature) if is_index else temperature
    h = None if cell_area is None else depth(mesh.vol[t][0:n], np.asarray(cell_area, np.float64)[0:n], float(min_depth))
    reacted = react(merged, np.float64(mesh.dt[t]), decay_per_day, theta, yields, temp, is_index, **terms, h=h)
    vol = mesh.vol[t][0:n]
    mass = np.array([(vol * (reacted[k] - merged[k])).sum() for k in range(K)])
    mass_abs = np.array([np.abs(vol * (reacted[k] - merged[k])).sum() for k in range(K)])
    b, b0 = np.empty((K, n)), np.empty((K, n))
    for k in range(K):
        rhs = ref.RHS(mesh, np.asarray(inputs[k], np.float64))
        b[k] = rhs._calculate_rhs(mesh, t, reacted[k])
        b0[k] = b[k] + rhs._calculate_load(mesh, t, merged[k] - reacted[k])     # (the boundary terms are the same)
    return b, b0, mass, mass_abs


# ------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,temperature_k", [(6, None), (6, -1), (3, None)])
def test_reacted_step_is_bitwise_the_oracles_update(K, temperature_k):
    """The full network (chain, sources, factors, depth flags) on a small plan, with a temperature constituent and at
    constant temperatures: at every step, from the oracle's own c[t], reacted_step gives its b and reaction mass bit
    for bit."""
    _, mesh, inputs, kin, src, lim, dep = synthetic_network(12, 9, 6, K, seed=40 + K, dry_fraction=0.05)
    if temperature_k is not None:
        kin = dict(kin, temperature_k=temperature_k, temperature_c=17.5)
    net = oracle_network(kin, src, lim, dep)
    oracle = KineticsRiverine(mesh, {f"c{k}": inputs[k] for k in range(K)}, **net)
    for t in range(5):
        c_t = np.stack([oracle.constituent_dict[f"c{k}"].concentration[t] for k in range(K)])
        b, _, mass, _ = reacted_step(mesh, inputs, c_t, t, **net)
        oracle.update()
        assert same(mass, oracle.reaction_mass[t]), t
        for k in range(K):
            assert same(b[k], oracle.constituent_dict[f"c{k}"].b.vals), (t, k)
    assert any(m.any() for m in oracle.reaction_mass)


def test_tile_rows_mirror_the_header(tmp_path):
    """react_tile_rows above against the header's for K = 1..128: a host program that includes cwr_kernels.cuh."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(nvcc).is_file():
        pytest.skip("nvcc not found")
    src = tmp_path / "tile_rows.cu"
    src.write_text(f'#include "{ROOT / "clearwater_riverine_b200" / "csrc" / "cwr_kernels.cuh"}"\n'
                   "#include <cstdio>\n"
                   "int main() {\n"
                   "    std::printf(\"kMaxK %d kThreads %d\\n\", cwr::kMaxK, cwr::kThreads);\n"
                   "    for (int K = 1; K <= cwr::kMaxK; ++K) std::printf(\"%d %d\\n\", K, cwr::react_tile_rows(K));\n"
                   "}\n")
    exe = tmp_path / "tile_rows"
    res = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-o", str(exe), str(src)],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60, check=True).stdout
    assert re.match(r"kMaxK (\d+) kThreads (\d+)", out).groups() == (str(K_MAX), str(THREADS))
    got = {int(k): int(r) for k, r in re.findall(r"^(\d+) (\d+)$", out, re.M)}
    assert got == {K: react_tile_rows(K) for K in range(1, K_MAX + 1)}
    assert (got[1], got[16], got[17], got[18], got[33], got[100], got[128]) == (256, 256, 256, 224, 128, 32, 32)


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def resident_cta_bound():
    """An upper bound on the CTAs of 256 threads that can be resident at once: SMs x (threads per SM / 256)."""
    import torch
    p = torch.cuda.get_device_properties(0)
    return p.multi_processor_count * (p.max_threads_per_multi_processor // THREADS)


def check_steps(be, mesh, inputs, net, steps=2):
    """Take `steps` steps from t = 0; after each: b of every column per element against reacted_step's within 1e-12 of
    the row's largest |b| (every column, before and after the reaction), the step's reaction mass within 1e-11 of
    sum |vol (c~' - c~)|, and the true residual of the solve with the oracle's A within 1e-12 of ||b||."""
    K = len(inputs)
    lhs = ref.LHS(mesh)
    before = np.array([be.reaction_mass(k) for k in range(K)])
    for t in range(steps):
        c_t = be.get_state_all(t)
        info = be.step(t)
        assert info.status == 0, (t, info.status, info.iterations, info.max_relres)
        b, b0, mass, mass_abs = reacted_step(mesh, inputs, c_t, t, **net)
        row = np.maximum(np.abs(b).max(axis=0), np.abs(b0).max(axis=0))
        for k in range(K):
            bad = np.nonzero(np.abs(be.get_rhs(k) - b[k]) > 1e-12 * row)[0]
            assert bad.size == 0, f"step {t} k {k}: b differs in {bad.size} rows, first {bad[:8].tolist()}"
        after = np.array([be.reaction_mass(k) for k in range(K)])
        err = np.abs((after - before) - mass)
        assert (err <= 1e-11 * mass_abs).all(), (t, np.nonzero(err > 1e-11 * mass_abs)[0], err, mass_abs)
        before = after
        lhs.update_values(mesh, t)
        A = lhs.to_csr()
        x = be.get_state_all(t + 1)
        for k in range(K):
            res = np.linalg.norm(A @ x[k] - b[k]) / np.linalg.norm(b[k])
            assert res <= 1e-12, (t, k, res)


def _side(n):
    """nx = ny for make_plan with n_exact = n: about 10 % of the quads split, as in the synthetic plans elsewhere."""
    return int(round(np.sqrt(n / 1.1)))


# (what runs, K, n): n is the least round number above 2 x 1184 tiles of react_tile_rows(K) rows -- twice the resident
# CTAs of a B200 (148 SMs x 8) -- odd where it can be, so that the state slot of every other step starts on an odd double
CASES = [
    pytest.param("full", 1, 610_001, id="full-K1"),           # G = 256 column-sum groups
    pytest.param("full", 3, 610_001, id="full-K3"),           # 16-byte pairs straddle rows
    pytest.param("full", 33, 305_001, id="full-K33"),         # 128-row tile
    pytest.param("full", 100, 76_000, id="full-K100"),        # G K = 200 < 256: idle threads in the column sums
    pytest.param("full", 127, 76_001, id="full-K127"),        # largest odd K
    pytest.param("full", 128, 76_000, id="full-K128"),        # kMaxK
    pytest.param("kinetics", 5, 610_001, id="kinetics-K5"),   # k_react<false>, temperature constituent
    pytest.param("limits", 19, 531_001, id="limits-K19"),     # k_react<true>, 224-row tile
    pytest.param("constant", 17, 610_001, id="constant-K17"),  # k_react<false>, every source column from sco
    pytest.param("history0", 3, 610_001, id="full-K3-keep_history0"),  # slots t & 1
]


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("what,K,n", CASES)
def test_several_tiles_per_cta(what, K, n):
    """Two consecutive steps on the large path, the state slot of the second on the other parity when n K is odd, and
    the reaction-mass ticket reset between two launches of the full grid.  full: chain, sources, factors and depth
    flags over areas varied 16-fold (k_react<true, true>); kinetics: the chain alone; limits: with factors, no depth
    (k_react<true>); constant: the chain and the sources at a constant temperature."""
    R = react_tile_rows(K)
    tiles, bound = -(-n // R), resident_cta_bound()
    assert tiles >= 2 * bound, (tiles, bound)
    _, mesh, inputs, kin, src, lim, dep = synthetic_network(_side(n), _side(n), 3, K, seed=K + 200, n_exact=n,
                                                            dry_fraction=0.02, limits_too=what != "kinetics")
    assert mesh.n == n
    if what == "kinetics":
        be, net = kinetic_backend(mesh, inputs, kin, solver_path=1), oracle_network(kin)
    elif what == "limits":
        be, net = depth_backend(mesh, inputs, kin, src, lim, None, solver_path=1), oracle_network(kin, src, lim)
    elif what == "constant":
        kin = dict(kin, temperature_k=-1, temperature_c=14.0)
        be, net = depth_backend(mesh, inputs, kin, src, None, None, solver_path=1), oracle_network(kin, src)
    else:
        opt = dict(keep_history=0) if what == "history0" else {}
        be, net = depth_backend(mesh, inputs, kin, src, lim, dep, solver_path=1, **opt), oracle_network(kin, src, lim, dep)
    assert be.options.solver_path == 1
    print(f"{what} K={K} n={n}: R={R}, {tiles} tiles >= 2 x {bound} resident CTAs, n K {'odd' if n * K % 2 else 'even'}")
    check_steps(be, mesh, inputs, net)
    be.close()


def _bench_case(full, constant):
    """bench.py's 1M x 16 plan with tools/kinetics_bench.py's network: the chain of make_kinetics (temperature
    constituent, or a constant temperature), with full=True its sources, Monod factors and depth flags over the plan
    areas."""
    import bench
    from clearwater_riverine_b200 import synthetic
    plan, K = bench.workload_plan("1m16", 3, seed=0)
    assert plan.n_real == 1_000_000 and K == 16
    adv, _, _, cdiff, dt = ref.derive_coefficients(plan.face_flow, plan.edge_velocity, plan.face_x, plan.face_y, plan.f1,
                                                   plan.f2, 0.1, plan.time_seconds)
    mesh = ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, plan.edge_velocity, plan.volume, dt, 0.1)
    inputs, kin = synthetic.make_kinetics(synthetic.make_inputs(plan, K, seed=0), seed=0, decay_range=(0.05, 2.0))
    if not full:
        return mesh, inputs, kin, None, None, None
    src = synthetic.make_kinetics_sources(kin, seed=0, rate_range=(0.05, 2.0))
    lim = synthetic.make_kinetics_limits(kin, src, seed=0)
    kin, src, flags = synthetic.make_kinetics_depth(kin, src, seed=0)
    if constant:
        kin = dict(kin, temperature_k=-1, temperature_c=24.0)
    return mesh, inputs, kin, src, lim, dict(cell_area=plan.cell_area, min_depth=0.01, **flags)


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("full,constant", [(True, False), (True, True), (False, False)],
                         ids=["full", "full-constant-temperature", "kinetics"])
def test_the_benchmarked_network_at_1m_x16(full, constant):
    """The shapes profiles/r03-r06 time: two steps, checked as test_several_tiles_per_cta checks them."""
    mesh, inputs, kin, src, lim, dep = _bench_case(full, constant)
    tiles, bound = -(-mesh.n // react_tile_rows(16)), resident_cta_bound()
    assert tiles >= 2 * bound, (tiles, bound)
    be = depth_backend(mesh, inputs, kin, src, lim, dep) if full else kinetic_backend(mesh, inputs, kin)
    assert be.options.solver_path == 1
    check_steps(be, mesh, inputs, oracle_network(kin, src, lim, dep))
    be.close()


@pytest.mark.gpu
def test_areas_given_before_the_ordering_is_rebuilt():
    """set_kinetics_depth before set_flow_hint: the hint rebuilds the ordering after the areas are uploaded, so they
    must be permuted again.  Bitwise the model whose depth call comes after the hint, hydrodynamics and inputs over 5
    steps (states and reaction mass), and the oracle's after the 5."""
    from clearwater_riverine_b200 import TransportBackend
    plan, mesh, inputs, kin, src, lim, dep = synthetic_network(60, 40, 7, 5, seed=211, dry_fraction=0.02)
    hint = plan.face_flow.mean(axis=0)
    K = len(inputs)

    def backend(areas_first):
        be = TransportBackend(mesh.f1, mesh.f2, mesh.n_face, mesh.n_time, K, mesh.diffusion_coefficient, solver_path=1)

        def kinetics():
            be.set_kinetics(**kin)
            be.set_kinetics_sources(**src)
            be.set_kinetics_limits(**lim)
            be.set_kinetics_depth(**dep)

        if areas_first:
            kinetics()
            perm = be.permutation()
        be.set_flow_hint(hint)
        if areas_first:
            assert not same(perm, be.permutation()), "the hint should have reordered the cells"
        be.set_hydro(0, mesh.adv, mesh.cdiff, mesh.vel, mesh.vol, mesh.dt)
        for k in range(K):
            be.set_inputs(k, inputs[k])
        if not areas_first:
            kinetics()
        return be

    first, after = backend(True), backend(False)
    assert same(first.permutation(), after.permutation())
    for t in range(5):
        assert first.step(t).status == 0 and after.step(t).status == 0
        assert same(first.get_state_all(t + 1), after.get_state_all(t + 1)), t
    assert all(first.reaction_mass(k) == after.reaction_mass(k) for k in range(K))
    oracle = depth_oracle(mesh, inputs, kin, src, lim, dep)
    for _ in range(5):
        oracle.update()
    for k in range(K):
        close(first.get_state(k, 5), oracle.constituent_dict[f"c{k}"].concentration[5], RTOL, f"k {k}")
    want = np.sum(oracle.reaction_mass, axis=0)
    got = np.array([first.reaction_mass(k) for k in range(K)])
    assert (np.abs(got - want) <= RTOL * np.maximum(np.abs(want), mass_scale(mesh, inputs))).all(), (got, want)
    first.close(); after.close()
