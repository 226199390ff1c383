"""The transport solver on polygon meshes: cells with five to ten neighbours (ELL widths W = 8 and 12), as real HEC-RAS
meshes have, through every solver path.  Every kernel family has a separate branch for rows wider than four -- k_assemble's
wide rows and fp32 copy, the wide loops of k_spmm and k_sweep, relax_tail of k_precond_gs, k_gs_strip's W > 4 branch,
k_solve_tiny<RPT, false>, k_solve_small's ELL blocks, and the ELL -> CSR of cwr_get_lhs -- and the path selection changes
at W > 4 (no k_solve_chip, no k_gs_tma, a smaller k_solve_tiny).  The meshes are make_plan plans with groups of cells
merged (tests/polygon_mesh.py).  Every case asserts the path it was written for, so that a change of the selection rules
cannot move it off its kernel quietly.  Tolerance: concentrations within rtol 1e-9 per step of the oracle's spsolve."""
import functools

import numpy as np
import pytest

from clearwater_riverine_b200 import synthetic
from oracle import reference_step as ref
from tests.polygon_mesh import ell_width, merge_cells, polygon_plan, row_lengths
from tests.test_gpu_configs import D, check_against_the_oracles_system, mass_balance_close
from tests.test_gpu_configs import _oracle_mesh as oracle_mesh
from tests.test_gpu_parity import RTOL, SOLVER_VARIANTS, close, make_backend, run_against_oracle

pytestmark = pytest.mark.gpu


@functools.lru_cache(maxsize=None)
def merged(nx, ny, T, sizes, n_groups, seed):
    """make_plan(nx, ny) with n_groups groups of `sizes` merged, boundary cells included."""
    plan = merge_cells(synthetic.make_plan(nx, ny, T, seed=seed, dry_fraction=0.02), sizes, n_groups, seed=seed)
    return plan, oracle_mesh(plan)


def large_w8():
    plan, mesh = merged(120, 90, 6, (2, 3), 1300, 200)          # 11,880 -> 9,930 cells
    assert ell_width(plan) == 8
    return plan, mesh


def large_w12():
    plan, mesh = merged(120, 90, 6, (2, 4), 1000, 201)          # 11,880 -> 9,880 cells
    assert ell_width(plan) == 12
    return plan, mesh


def resolved_sync(K, opts):
    """The sweep kernel a request resolves to on a mesh with W > 4: k_gs_tma (4) needs W == 4, k_gs_strip (3) moves 16-byte
    packs of the sweep type."""
    sync = opts["precond_sync"]
    if sync == 4:
        sync = 3
    if sync >= 3 and (K * (4 if opts.get("precond_precision", 32) == 32 else 8)) % 16 != 0:
        sync = 2
    return sync


def check_large_path(plan, mesh, inputs, K, opts):
    """Assert the large-mesh path and the sweep kernel opts resolve to, then run 5 steps against the oracle."""
    be = make_backend(mesh, list(inputs), solver_path=1, **opts)
    assert be.options.solver_path == 1 and be.options.solver == opts["solver"]
    if opts.get("precond_sweep", 1) == 1:
        sync = resolved_sync(K, opts)
        assert be.options.precond_sync == sync, (be.options.precond_sync, sync)
        if K == 16 and opts["precond_sync"] == 4 and opts.get("precond_precision", 32) == 32:
            assert sync == 3, "no k_gs_tma at W != 4"
        assert be.solver_stats()[2] == (plan.n_real // 512 if sync >= 2 else 0)
    else:
        assert be.options.precond_sync == 0
    be.close()
    run_against_oracle(mesh, inputs, 5, solver_path=1, **opts)


@pytest.mark.parametrize("K", [1, 3, 16])
@pytest.mark.parametrize("opts", SOLVER_VARIANTS, ids=lambda o: "-".join(f"{k}{v}" for k, v in o.items()))
def test_large_path_every_sweep_kernel_w8(K, opts):
    """~10k cells, W = 8, boundary cells merged too: BiCGSTAB / defect correction, grid-barrier / neighbour-synchronised /
    pipelined Gauss-Seidel sweeps and Jacobi steps over rows of up to 8 neighbours."""
    plan, mesh = large_w8()
    inputs = synthetic.make_inputs(plan, K, seed=200 + K)
    check_large_path(plan, mesh, inputs, K, opts)


@pytest.mark.parametrize("K", [3, 16])
@pytest.mark.parametrize("opts", [dict(solver=1, precond_sync=1), dict(solver=2, precond_sync=3),
                                  dict(solver=2, precond_sweep=0, precond_steps=6)],
                         ids=["bicgstab-gridbarrier", "dc-strip", "jacobi"])
def test_large_path_w12(K, opts):
    """W = 12 (cells of ten neighbours: three ELL blocks): BiCGSTAB with grid-barrier sweeps, defect correction with
    k_gs_strip (K = 16; K = 3 has 12-byte packs and takes the neighbour-synchronised k_precond_gs), Jacobi steps."""
    plan, mesh = large_w12()
    inputs = synthetic.make_inputs(plan, K, seed=300 + K)
    check_large_path(plan, mesh, inputs, K, opts)


@pytest.mark.parametrize("K", [1, 2, 33, 128])
@pytest.mark.parametrize("opts", [dict(precond_sweep=0, precond_precision=64, precond_steps=4),
                                  dict(precond_sweep=0, precond_steps=8),
                                  dict(precond_sweep=1, precond_steps=3),
                                  dict(precond_sweep=1, precond_steps=2, precond_colors=7),
                                  dict(precond_sweep=1, precond_steps=4, precond_precision=64, precond_colors=32)])
def test_jacobi_steps_and_fp64_sweeps_every_lane_width(K, opts):
    """The options of test_preconditioner_variants on a merged 40 x 25 mesh (W = 8): k_sweep and k_spmm at every lanes-per-row
    instantiation over wide rows."""
    if K == 128 and opts.get("precond_precision") == 64 and opts["precond_sweep"] == 0:
        pytest.skip("covered by K = 33")
    plan, mesh = merged(40, 25, 6, (2, 3), 120, 100)
    assert ell_width(plan) == 8
    inputs = synthetic.make_inputs(plan, K, seed=100 + K)
    be = make_backend(mesh, list(inputs), solver_path=1, **opts)
    assert be.options.solver_path == 1 and be.options.precond_sweep == opts["precond_sweep"]
    if opts["precond_sweep"] == 1:
        assert be.options.precond_sync == resolved_sync(K, dict(opts, precond_sync=4))
    else:
        assert be.options.precond_sync == 0
    be.close()
    run_against_oracle(mesh, inputs, 5, solver_path=1, **opts)


@pytest.mark.parametrize("solver_path", [1, 2])
@pytest.mark.parametrize("W,sizes", [(8, (2, 3)), (12, (2, 4))])
def test_system_read_back_equals_the_oracles(W, sizes, solver_path):
    """get_lhs() (the k_assemble wide branch, the host ELL -> CSR) equals the oracle's LHS: same pattern, values within
    1e-14; get_rhs() within 1e-13 at t = 0; on both paths (2: k_solve_tiny on this size)."""
    plan, mesh = merged(40, 25, 4, sizes, 110, 400 + W)
    assert ell_width(plan) == W
    K = 3
    inputs = synthetic.make_inputs(plan, K, seed=7)
    be = make_backend(mesh, list(inputs), solver_path=solver_path)
    assert be.options.solver_path == (1 if solver_path == 1 else 3)
    oracle = ref.OracleRiverine(mesh, {f"c{k}": inputs[k] for k in range(K)})
    assert be.step(0).status == 0
    oracle.update()
    A = oracle.last_A.copy(); A.sum_duplicates(); A.sort_indices()
    got = be.get_lhs(); got.sort_indices()
    assert np.array_equal(got.indptr, A.indptr) and np.array_equal(got.indices, A.indices)
    assert np.diff(A.indptr).max() == row_lengths(plan).max() + 1          # the widest row and its diagonal
    close(got.data, A.data, 1e-14, f"LHS W={W}")
    for k in range(K):
        close(be.get_rhs(k), oracle.constituent_dict[f"c{k}"].b.vals, 1e-13, f"RHS W={W} k{k}")
    be.close()


# ---- the small path across its boundaries ----------------------------------------------------------------------------
def tiny_smem_bytes(n, W):
    """cwr_small.cuh: val (n*W f64) | z, u (n f64 each) | idx (n*W u16, padded to 16 bytes)."""
    return n * W * 8 + 2 * n * 8 + ((n * W * 2 + 15) & ~15)


def tiny_limit(W):
    """The largest mesh k_solve_tiny takes at ELL width W: its dynamic shared memory plus 4 KB of static shared memory within
    the device's opt-in shared memory per block (cudaDevAttrMaxSharedMemoryPerBlockOptin), and at most 8 rows per thread."""
    import torch
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    n = min(4096, (optin - 4096) // (W * 10 + 16) + 1)
    while tiny_smem_bytes(n, W) + 4096 > optin:
        n -= 1
    return n


@functools.lru_cache(maxsize=None)
def small_case(n, W, T=7, seed=0):
    plan = polygon_plan(n, T, seed=seed + n, sizes=(2, 3) if W == 8 else (2, 4))
    assert ell_width(plan) == W, (n, W, ell_width(plan))
    return plan, oracle_mesh(plan)


def small_path_run(n, W, want_path, K=3, **opt):
    plan, mesh = small_case(n, W)
    inputs = synthetic.make_inputs(plan, K, seed=n)
    be = make_backend(mesh, list(inputs), **opt)
    assert be.options.solver_path == want_path, (n, W, be.options.solver_path, want_path)
    be.close()
    run_against_oracle(mesh, inputs, 5, **opt)


@pytest.mark.parametrize("W,rpt", [(8, 1), (8, 2), (8, 4), (8, 6), (12, 1), (12, 2), (12, 4)])
def test_tiny_kernel_every_rows_per_thread(W, rpt):
    """k_solve_tiny<RPT, false> (column-major [W][n] values and indices, the generic row_dot) at every instantiation the
    shared memory allows: n ~ 480, 1,000, 2,000 rows and the largest n that fits (RPT 6 at W = 8; RPT 4 at W = 12).  No
    k_solve_chip at W != 4: solver_path 3, never 4."""
    limit = tiny_limit(W)
    n = {1: 480, 2: 1000, 4: min(2000, limit), 6: limit}[rpt]
    assert (rpt - 1) * 512 < n <= rpt * 512 or (rpt == 6 and 2048 < n <= 3072), (W, rpt, n, limit)
    small_path_run(n, W, 3)


@pytest.mark.parametrize("W", [8, 12])
def test_first_mesh_past_the_tiny_limit_takes_k_solve_small(W):
    small_path_run(tiny_limit(W) + 1, W, 2)


@pytest.mark.parametrize("n,want_path", [(20_000, 2), (32_768, 2), (32_769, 1)])
def test_small_and_large_path_sizes_w8(n, want_path):
    """k_solve_small's ELL blocks at n ~ 20,000 and at its largest default size; one more cell takes the large path."""
    small_path_run(n, 8, want_path)


def test_tiny_kernel_64_column_ensemble_w8():
    """64 columns (one CTA each) on the largest W = 8 mesh k_solve_tiny takes."""
    n = tiny_limit(8)
    plan, mesh = small_case(n, 8)
    inputs = synthetic.make_inputs(plan, 64, seed=64)
    be = make_backend(mesh, list(inputs))
    assert be.options.solver_path == 3
    be.close()
    run_against_oracle(mesh, inputs, 3)


def test_strip_kernels_with_every_cta_w8():
    """~150k cells at W = 8: one strip per resident CTA.  The grid-barrier kernel and the neighbour-synchronised ones agree
    within 1e-11 with equal sweep counts.  k_precond_gs (sync 2) and k_gs_strip (sync 3) sum a wide row in the same order --
    the first ELL block, then the further blocks entry by entry; where k_precond_gs adds w * 0 for a neighbour not visited
    yet, k_gs_strip skips it, which leaves the sum's bits alone -- so they are bitwise equal here too."""
    plan, mesh = merged(410, 380, 4, (2, 3), 14_000, 77)        # 171k -> 150k cells
    assert ell_width(plan) == 8
    inputs = synthetic.make_inputs(plan, 4, seed=77)
    outs, sweeps = [], []
    for sync in (1, 2, 3):
        be = make_backend(mesh, list(inputs), solver_path=1, solver=2, precond_sync=sync)
        assert be.options.precond_sync == sync
        for t in range(3):
            info = be.step(t)
            assert info.status == 0 and info.max_relres <= 1e-13 and info.sweeps > 0
        outs.append(be.get_state_all(3))
        sweeps.append(be.solver_stats()[0])
        if sync >= 2:
            assert be.solver_stats()[2] >= 148 and be.solver_stats()[1] == 0
        be.close()
    close(outs[1], outs[0], 1e-11, "neighbour-synchronised vs grid-barrier sweeps")
    assert np.array_equal(outs[2], outs[1]), "k_gs_strip and k_precond_gs sum wide rows in the same order"
    assert sweeps[0] == sweeps[1] == sweeps[2], sweeps
    oracle = ref.OracleRiverine(mesh, {f"c{k}": inputs[k] for k in range(2)})
    for _ in range(3):
        oracle.update()
    for k in range(2):
        close(outs[1][k], oracle.constituent_dict[f"c{k}"].concentration[3][:mesh.n], RTOL, f"150k cells W=8 k{k}")


def test_bench_size_w8_against_the_oracles_own_matrix_and_right_hand_sides():
    """bench.py's 1M x 16 plan merged to W = 8 (910k cells), default options (defect correction, k_gs_strip: no k_gs_tma at
    W != 4): the GPU's LHS and RHS equal the oracle's, the true residual of every column with the oracle's A and b is below
    1e-12 ||b||, and one column equals scipy's BiCGSTAB on the oracle's system within rtol 1e-9."""
    import bench
    base, K = bench.workload_plan("1m16", 3, seed=2)
    plan = merge_cells(base, (2, 3), 60_000, seed=2)
    assert plan.n_real == 910_000 and K == 16 and ell_width(plan) == 8
    check_against_the_oracles_system(plan, K, solver_path=1, solver=2, precond_sync=3)


def test_ohio_shaped_polygon_mesh_through_update():
    """What a user of a real plan runs: the Ohio-shaped preset merged pairwise to 2,600 cells (W = 8), two constituents,
    30 steps of ClearwaterRiverine.update() at default options -- per-step concentrations and mass fluxes against the
    oracle, and mass_balance() against the oracle's.  Past the tiny limit at W = 8, such a mesh gets k_solve_small."""
    from clearwater_riverine_b200 import ClearwaterRiverine
    T = 31
    plan = merge_cells(synthetic.ohio_like(n_time=T, seed=2), 2, 343, seed=2)
    n = plan.n_real
    assert n == 2600 and ell_width(plan) == 8
    inputs = synthetic.make_inputs(plan, 2, seed=2)
    names = ("ecoli", "tracer")
    model = ClearwaterRiverine.from_arrays(plan.f1, plan.f2, plan.face_x, plan.face_y, plan.time_seconds, plan.face_flow,
                                           plan.edge_velocity, plan.volume, D, dict(zip(names, inputs)))
    assert model.backend.options.solver_path == (3 if n <= tiny_limit(8) else 2)
    mesh = oracle_mesh(plan)
    oracle = ref.OracleRiverine(mesh, dict(zip(names, inputs)))
    for t in range(T - 1):
        model.update()
        oracle.update()
        for name in names:
            con = oracle.constituent_dict[name]
            close(model.mesh[name][t + 1], con.concentration[t + 1], RTOL, f"{name} step {t}")
            fin = ~np.isnan(con.total_mass_flux[t])
            scale = np.abs(con.total_mass_flux[t][fin]).max()
            got = model.constituent_dict[name].total_mass_flux[t]
            assert np.array_equal(np.isnan(got), ~fin)
            assert np.abs(got[fin] - con.total_mass_flux[t][fin]).max() <= RTOL * scale, (name, t)
    lines = {key: plan.boundary_faces[key] for key in ("upstream", "downstream")}      # the lines with boundary series
    for name in names:
        con = oracle.constituent_dict[name]
        want = ref.mass_balance(mesh, con.concentration, con.total_mass_flux, plan.face_flow, lines)
        mass_balance_close(model.mass_balance(name, lines), want, name)
    model.finalize()
