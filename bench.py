#!/usr/bin/env python
"""Benchmark of the per-timestep implicit advection-diffusion step (BASELINE.json metric:
cell-timesteps/sec, fp64; solver HBM GB/s vs peak).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload 1m16|ohio|ens64|16m] [--impl reference] [--dump-outputs DIR]

A "step" = one ClearwaterRiverine.update(): LHS assembly, RHS, solve, store, mass flux for all K
constituents on the workload's mesh.  One cell-timestep = one real cell advanced one step for one
constituent.  The headline line is BASELINE.json configs[2]: the synthetic 1M-cell mesh with 16
constituents (the "named size" the metric's HBM fraction is defined on).  N > 1 (torchrun, one rank per
GPU): every rank advances its own 16 constituents on a replica of the mesh -- weak scaling over
independent units, no data-path collective; NCCL only reduces the mass-balance scalars.

The same JSON line carries the other BASELINE configurations under "extra" (bounded, inside the same run):
  extra.ohio   configs[1]  Ohio-River-shaped mesh, 1 constituent             (N = 1 only)
  extra.ens64  configs[3]  64 boundary-condition scenarios sharded over the N ranks (strong scaling)
  extra.ens_weak           128 scenarios per rank on the same mesh (weak scaling: the ensemble grows with the GPUs)
  extra.dd16m  configs[4]  16M-cell mesh as ONE model cut into N strips with NVLink halo exchange
                           (strong scaling; N = 1 is the single-GPU point of the curve), plus a small-mesh
                           parity figure of the decomposed path against the single-GPU answer (N > 1)

--impl reference: the reference's own CPU path for the same metric and config -- the oracle restatement of
linalg.py + csr_matrix + spsolve + _mass_flux (the reference package cannot be imported here: no
xarray/h5py) on the 1M-cell mesh, ONE constituent (the reference solves constituents one after another:
its rate in cell-timesteps/s does not depend on K), min(steps, 3) timed steps of ~50 s each.

--dump-outputs DIR (GPU arm, one GPU): after the timed steps, what the last of them handed its caller -- the
concentrations and the three mass-flux arrays of every constituent, on the cells and edges where they are defined --
as DIR/<name>.npy (float64, see dump_outputs).  The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

DIFFUSION = 0.1
METRIC, UNIT = "cell_timesteps_per_sec", "cell-timesteps/s"
T_START = time.perf_counter()

WORKLOAD_NAMES = {
    "1m16": "synthetic 1M-cell unstructured mesh, 16 constituents batched (BASELINE configs[2])",
    "ohio": "Ohio-River-shaped synthetic mesh (2943 cells), 1 constituent (BASELINE configs[1])",
    "ens64": "64 boundary-condition scenarios on the Ohio-shaped mesh (BASELINE configs[3])",
    "ensw": "128 boundary-condition scenarios PER GPU on the Ohio-shaped mesh (the ensemble of configs[3] grown with the GPUs: weak scaling)",
    "16m": "synthetic 16M-cell mesh, 1 constituent (BASELINE configs[4])",
}


def workload_plan(name: str, n_time: int, seed: int, scale: float = 1.0):
    from clearwater_riverine_b200 import synthetic
    if name == "1m16":
        side = max(8, int(round(953 * scale)))
        n_exact = 1_000_000 if scale == 1.0 else None
        plan = synthetic.make_plan(side, side, n_time, dt=30.0, tri_fraction=0.1, dry_fraction=0.02, courant=1.5,
                                   n_exact=n_exact, seed=seed)
        return plan, 16
    if name == "ohio":
        return synthetic.ohio_like(n_time, seed=seed), 1
    if name == "ens64":
        return synthetic.ohio_like(n_time, seed=seed), 64
    if name == "ensw":
        return synthetic.ohio_like(n_time, seed=seed), 128
    if name == "16m":
        side = max(8, int(round(3814 * scale)))
        plan = synthetic.make_plan(side, side, n_time, dt=30.0, tri_fraction=0.1, dry_fraction=0.02, courant=1.5,
                                   n_exact=16_000_000 if scale == 1.0 else None, seed=seed)
        return plan, 1
    raise SystemExit(f"unknown workload {name}")


class ClockSampler:
    """SM clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe): NVML polled every
    10 ms from a thread (no process start-up latency, so even a 100 ms region is covered); `nvidia-smi -lms` as
    the fallback.  Samples are tagged inside / outside the timed window; the summary uses the ones inside."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.proc, self.lines = device, None, []
        self.samples = []            # (time, sm_mhz, reasons bitmask)
        self.t0 = self.t1 = None
        self._stop = threading.Event()
        self._thread = None
        self.max_mhz = None
        self.source = None

    def _poll_nvml(self, nv, h):
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        i, reasons = 0, 0
        while not self._stop.is_set():
            try:
                if i % 4 == 0:                       # the reasons query is the slow one
                    reasons = int(get_reasons(h))
                self.samples.append((time.perf_counter(), float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), reasons))
            except Exception:
                pass
            i += 1
            self._stop.wait(0.005)

    def start(self):
        """Begin sampling (call before the warm-up: the device is under load from then on)."""
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.device)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self._nv = nv
            self._thread = threading.Thread(target=self._poll_nvml, args=(nv, h), daemon=True)
            self._thread.start()
            self.source = "nvml, 10 ms"
            return
        except Exception:
            self._thread = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.device)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            self.source = "nvidia-smi -lms 50"
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def window_begin(self):
        self.t0 = time.perf_counter()

    def window_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        if self._thread is not None:
            time.sleep(0.03)
            self._stop.set()
            self._thread.join(timeout=1.0)
            nv = self._nv
            bits = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                    "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                    "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                    "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            inside = [s for s in self.samples if self.t0 is not None and self.t0 <= s[0] <= (self.t1 or 1e300)]
            used = inside if inside else self.samples        # all samples are under load (warm-up + timed steps)
            reasons = sorted(nm for nm, bit in bits.items() if any(s[2] & bit for s in used))
            return {"sm_mhz": float(np.median([s[1] for s in used])) if used else None, "sm_max_mhz": self.max_mhz,
                    "samples": len(used), "samples_in_timed_region": len(inside), "reasons": reasons, "source": self.source}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvml and nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        sm, mx, reasons, n_in = [], [], set(), 0
        for ts, ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            n_in += int(self.t0 is not None and self.t0 <= ts <= (self.t1 or 1e300))
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "samples_in_timed_region": n_in, "reasons": sorted(reasons), "source": self.source}


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.is_file():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
        except Exception:
            pass
    return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


DUMP_STATE_BYTES, DUMP_FLUX_BYTES = 32 << 20, 24 << 20     # 56 MiB in all: under 64 MB whatever K is


def dump_outputs(be, t: int, out_dir, f2, inputs) -> dict:
    """Step t's results as its caller receives them, written to out_dir as float64 .npy files:
      concentration                                  (K, cells)  c[t + 1] of the real cells
      advection / diffusion / total_mass_flux        (K, edges)  the three per-edge mass-flux arrays of step t
    The fluxes are kept on the edges where they are defined: between two real cells, and into ghost cells that hold a
    boundary value (inputs (K, T, F) nonzero at t + 1) for every constituent.  Into any other ghost cell the flux is
    NaN by definition, as in the reference (the ghost concentration is NaN).  The edges are chosen from the mesh and the
    inputs alone, so a NaN on a kept edge is a defect of the build, not dropped.  Cells and edges beyond what fits
    DUMP_STATE_BYTES / DUMP_FLUX_BYTES are sampled at fixed, seeded indices (sorted), so the same mesh and inputs
    always give the same sample.  Returns {name: shape}."""
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    rng = np.random.default_rng(12345)

    def sample(candidates, cap):
        return np.sort(rng.choice(candidates, cap, replace=False)) if len(candidates) > cap else candidates

    K = be.K
    cells = sample(np.arange(be.n_real), DUMP_STATE_BYTES // (8 * K))
    arrays = {"concentration": be.get_state_all(t + 1)[:, cells]}
    if be.options.mass_flux:
        f2 = np.asarray(f2)
        defined = f2 < be.n_real
        ghost = np.flatnonzero(~defined)
        defined[ghost] = (np.asarray(inputs)[:, t + 1, f2[ghost]] != 0).all(axis=0)
        edges = sample(np.flatnonzero(defined), DUMP_FLUX_BYTES // (3 * 8 * K))
        flux = [be.get_mass_flux(k, t) for k in range(K)]
        for i, name in enumerate(("advection_mass_flux", "diffusion_mass_flux", "total_mass_flux")):
            arrays[name] = np.stack([f[i][edges] for f in flux])
    for name, a in arrays.items():
        np.save(out_dir / f"{name}.npy", np.ascontiguousarray(a, dtype=np.float64))
    return {name: list(a.shape) for name, a in arrays.items()}


def pinned(a: np.ndarray) -> np.ndarray:
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()


# ------------------------------------------------------------------------------------------------------
# CPU legs: the reference's arithmetic (oracle port) -- the only places bench.py executes oracle/
# ------------------------------------------------------------------------------------------------------
def cpu_reference_rate(steps: int, warmup: int, seed: int, full_size: bool):
    """Oracle (reference arithmetic: numpy COO assembly + csr_matrix + spsolve + mass flux), ONE constituent, on the
    headline 1M-cell mesh (full_size) or on a 100k-cell sample of the same generator (the bounded cpu_baseline leg)."""
    from clearwater_riverine_b200 import synthetic
    from oracle import reference_step as ref
    T = steps + warmup + 1
    if full_size:
        plan, _ = workload_plan("1m16", T, seed=seed)
    else:
        plan = synthetic.make_plan(302, 302, T, dt=30.0, tri_fraction=0.1, dry_fraction=0.02, courant=1.5,
                                   n_exact=100_000, seed=seed)
    adv, _, _, cdiff, dt = ref.derive_coefficients(plan.face_flow, plan.edge_velocity, plan.face_x, plan.face_y,
                                                   plan.f1, plan.f2, DIFFUSION, plan.time_seconds)
    mesh = ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, plan.edge_velocity, plan.volume, dt, DIFFUSION)
    inputs = synthetic.make_inputs(plan, 1, seed=seed)
    model = ref.OracleRiverine(mesh, {"c0": inputs[0]})
    for _ in range(warmup):
        model.update()
    t0 = time.perf_counter()
    for _ in range(steps):
        model.update()
    dt_s = time.perf_counter() - t0
    rate = plan.n_real * steps / dt_s
    what = ("the headline mesh" if full_size else "a sample mesh from the same generator (same dt, Courant, dry fraction)")
    sample = (f"{steps} steps of {what}: {plan.n_real} cells, 1 constituent (the reference solves constituents one after "
              f"another: cell-timesteps/s does not depend on K); numpy assembly + scipy csr_matrix + spsolve (SuperLU) + mass flux, "
              f"single-threaded")
    return rate, dt_s / steps * 1e3, sample, plan.n_real


def cpu_bicgstab_rate(seed: int):
    """Like-for-like algorithmic CPU reference (BASELINE.md section 3): the oracle's assembled system of one step
    of the sample mesh solved with scipy's Jacobi-preconditioned BiCGSTAB to the same 1e-13 instead of SuperLU."""
    import scipy.sparse as sp
    import scipy.sparse.linalg as spla
    from clearwater_riverine_b200 import synthetic
    from oracle import reference_step as ref
    plan = synthetic.make_plan(302, 302, 4, dt=30.0, tri_fraction=0.1, dry_fraction=0.02, courant=1.5, n_exact=100_000, seed=seed)
    adv, _, _, cdiff, dt = ref.derive_coefficients(plan.face_flow, plan.edge_velocity, plan.face_x, plan.face_y,
                                                   plan.f1, plan.f2, DIFFUSION, plan.time_seconds)
    mesh = ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, plan.edge_velocity, plan.volume, dt, DIFFUSION)
    inputs = synthetic.make_inputs(plan, 1, seed=seed)
    n = plan.n_real
    lhs = ref.LHS(mesh); lhs.update_values(mesh, 1)
    A = lhs.to_csr(); A.sum_duplicates()
    rhs = ref.RHS(mesh, inputs[0])
    rhs.update_values(inputs[0][0][:n].copy(), mesh, 1)
    b = np.asarray(rhs.vals, dtype=np.float64)
    M = sp.diags(1.0 / A.diagonal())
    its = [0]
    t0 = time.perf_counter()
    x, info = spla.bicgstab(A, b, x0=inputs[0][0][:n].copy(), rtol=1e-13, atol=0.0, M=M, maxiter=2000,
                            callback=lambda xk: its.__setitem__(0, its[0] + 1))
    el = time.perf_counter() - t0
    return {"value": n / el, "unit": UNIT, "iterations": its[0], "converged": info == 0, "seconds_per_solve": el,
            "what": f"scipy bicgstab + Jacobi, rtol 1e-13, one solve of the {n}-cell sample system (solve only, 1 thread)"}


def run_reference(args, rank):
    """--impl reference: the reference's CPU path on the headline configuration (1M cells; K = 1 timed, the rate in
    cell-timesteps/s is per constituent-cell and does not depend on K)."""
    if rank != 0:
        return
    steps = max(1, min(args.steps, 3))
    warm = 1 if args.warmup > 0 else 0
    full = args.workload == "1m16" and args.scale == 1.0 and not args.sample_reference
    rate, ms, sample, n = cpu_reference_rate(steps, warm, seed=2, full_size=full)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD_NAMES["1m16"], "cells": n, "constituents_timed": 1,
                   "note": "reference CPU path (oracle port of linalg.py + csr_matrix + spsolve + _mass_flux; the Python package itself "
                           "needs xarray/h5py, absent here).  One constituent is timed: the reference loops over constituents "
                           "(transport.py:231) and refactorises A for each, so 16 constituents take 16x the time per step and the "
                           "rate in cell-timesteps/s is the same",
                   "ms_per_step_16_constituents_extrapolated": ms * 16},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample,
                         "host_cores_available": os.cpu_count()},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
# GPU legs
# ------------------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, rank, world, local):
        self.rank, self.world, self.local = rank, world, local

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()


def family_bytes(o, n, nnz, E, K, Wd, sweeps_per_launch):
    """Algorithmic bytes per launch of every kernel family (DESIGN.md section 3; each operand counted once)."""
    V = 8.0 * n * K                                     # one fp64 (n, K) vector
    sweeps = max(0, o.precond_steps - 1)
    sb = 4 if o.precond_precision == 32 else 8          # bytes per entry of the sweep type
    pt = sb if sweeps else 8                            # type of the preconditioned vectors the products gather
    S = float(pt) * n * K
    ell = 4.0 * n * Wd                                  # ELL column indices
    handed = o.solver == 2 and o.precond_sync >= 3     # the residual reaches the sweep kernel in the sweep type (M.us)
    fb = {
        "assemble": 2 * ell + 12.0 * nnz + 4.0 * n + 8.0 * n * Wd + (4.0 * n * Wd if sb == 4 and sweeps else 0) + 8.0 * n,
        "rhs": 3 * V + 12.0 * n,
        "spmm_v": ell + 8.0 * n * Wd + S + 2 * V,                      # p^ gathered, rhat read, v written
        "spmm_t": ell + 8.0 * n * Wd + S + 3 * V,                      # s^ gathered, rhat, s read, t written
        "update_s": 3 * V,
        "update_xrp": 8 * V + 2.0 * S,                                 # x r p t v read, x r p written, p^ s^ read
        "mass_flux": 8.0 * E + 12.0 * E + 2 * 8.0 * E * K + 3 * 8.0 * E * K,
    }
    if o.solver == 2:     # defect correction: r = b - A x (x, b read; r written [+ its copy in the sweep type])
        fb["spmm_init"] = ell + 8.0 * n * Wd + 3 * V + (S if handed else 0)
        fb["dc_update"] = ell + 8.0 * n * Wd + S + 4 * V + (S if handed else 0)     # z gathered; r, x read and written
    else:                 # BiCGSTAB: x, b read; r, rhat, p written
        fb["spmm_init"] = ell + 8.0 * n * Wd + 5 * V
    if o.precond_sweep == 1:
        # one launch = all sweeps of one application / cycle: per sweep indices + values, u, z gathered, z written;
        # the grid-barrier and the plain strip kernel also read u once as the solver's fp64 vector
        per_sweep = ell + sb * n * Wd + 3.0 * sb * n * K
        fb["precond"] = sweeps_per_launch * per_sweep + (0.0 if o.precond_sync >= 3 else 8.0 * n * K)
    else:                 # one launch = one Jacobi step
        fb["precond"] = ell + sb * n * Wd + 3.0 * sb * n * K
    return fb


KERNEL_NAMES = {
    "spmm_t": "k_spmm<AT> (t = A s^ fused with four dot products)", "spmm_v": "k_spmm<AV> (v = A p^ fused with (rhat, v))",
    "update_xrp": "k_update_xrp", "dc_update": "k_spmm<DC> (r -= A z, x += z fused with (r, r) and the plan of the next cycle)",
    "solve_small": "k_solve_chip / k_solve_tiny / k_solve_small (whole solve of a constituent in one CTA, on chip up to 4096 cells; k_solve_chip: fp32 sweeps inside the fp64 BiCGSTAB, branch-free colour step)"}


def precond_kernel_name(o):
    if o.precond_sweep != 1:
        return "k_sweep (one Jacobi step of the polynomial preconditioner)"
    return {1: "k_precond_gs<STRIP=false> (multicolour Gauss-Seidel sweeps of one cycle, persistent, a grid barrier per colour)",
            2: "k_precond_gs<STRIP=true> (multicolour Gauss-Seidel sweeps of one cycle, persistent, one strip per CTA, neighbour flags)",
            3: "k_gs_strip (multicolour Gauss-Seidel sweeps of one cycle, persistent, one strip per CTA, neighbour flags, "
               "software-pipelined cp.async gathers)",
            4: "k_gs_tma (multicolour Gauss-Seidel sweeps of one cycle, persistent, one strip per CTA, neighbour flags; index / "
               "value / right-hand-side streams by cp.async.bulk + mbarrier into a per-warp ring, predicated ld.global.cg "
               "gathers in registers; fp32 x 16 constituents)"}.get(o.precond_sync, "k_precond_gs")


def gpu_workload(name, ctx, args, steps, warmup, profile_steps, opts, *, dd=False, want_roofline=True, want_e2e=False,
                 want_clocks=True, dump_dir=None):
    """One workload on the GPU(s): device-timed rate, per-kernel-family times, mass-balance scalars; with dump_dir, the
    outputs of the last timed step (dump_outputs)."""
    import torch
    import torch.distributed as dist
    from clearwater_riverine_b200 import TransportBackend, ensemble, synthetic
    rank, world, local = ctx.rank, ctx.world, ctx.local
    W, K_steps, P = warmup, steps, profile_steps
    T = W + K_steps + P + 1
    t_setup = time.perf_counter()
    plan, K = workload_plan(name, T, seed=2, scale=args.scale)
    n, E, F = plan.n_real, plan.n_edge, plan.n_face
    n_units = K * world                      # weak scaling: every rank brings its own K constituents
    if dd:
        n_units = K                          # one model cut into strips: total work fixed (strong scaling)
    if name in ("ens64", "ensw"):            # ens64: 64 scenarios sharded over the ranks (total work fixed); ensw: 128 per rank
        n_units = 64 if name == "ens64" else 128 * world
        mine = ensemble.shard_units(n_units, world, rank)
        K = len(mine)
        scales = np.exp(np.random.default_rng(100).normal(0.0, 0.5, size=n_units))      # same table on every rank
        base = synthetic.make_inputs(plan, 1, seed=2)[0]
        inputs = np.stack(ensemble.scenario_inputs(base, n, scales[mine.start:mine.stop]))
    elif dd:                                 # every rank holds the same inputs, owns a strip of the rows
        mine = range(K)
        inputs = synthetic.make_inputs(plan, K, seed=2)
    else:                                    # independent constituents: own ICs / BC series per rank
        mine = range(rank * K, (rank + 1) * K)
        inputs = synthetic.make_inputs(plan, K, seed=2 + 1000 * rank)
    dt = np.append(np.diff(plan.time_seconds), np.nan)
    # the Gauss-Seidel colours (and the strips of a domain decomposition) follow the time-mean flow
    hint = plan.face_flow[:: max(1, T // 32)].mean(axis=0, dtype=np.float64).astype(np.float32)
    if dd:
        from clearwater_riverine_b200.domain import DomainDecomposedBackend, merge_owned
        be = DomainDecomposedBackend(plan.f1, plan.f2, F, T, K, DIFFUSION, rank, world, device=local, flow_hint=hint, **opts)
    else:
        be = TransportBackend(plan.f1, plan.f2, F, T, K, DIFFUSION, device=local, flow_hint=hint, **opts)
    be.set_geometry(plan.face_x, plan.face_y)
    chunk = max(1, (256 << 20) // (4 * E))
    for t0 in range(0, T, chunk):
        t1 = min(T, t0 + chunk)
        be.set_hydro_raw(t0, plan.face_flow[t0:t1], plan.edge_velocity[t0:t1], plan.volume[t0:t1], dt[t0:t1])
    dd_info = be.attach() if dd else None
    for k in range(K):
        be.set_inputs(k, inputs[k])
    stream = torch.cuda.ExternalStream(be.stream())
    t_setup = time.perf_counter() - t_setup

    sampler = ClockSampler(local) if want_clocks else None
    if sampler:
        sampler.start()
    for t in range(W):
        be.step(t)
    ctx.barrier()
    torch.cuda.synchronize()
    if sampler:
        sampler.window_begin()
    l0, i0 = be.counters()
    sw0 = be.solver_stats()[0]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    info = be.run(W, W + K_steps)            # cwr_run: K_steps updates, no host round trip on the small-mesh path
    worst_status, worst_relres = info.status, info.max_relres
    e1.record(stream)
    torch.cuda.synchronize()
    if sampler:
        sampler.window_end()
    ctx.barrier()
    clocks = sampler.stop() if sampler else None
    l1, i1 = be.counters()
    sw1, fallbacks, n_strips, max_nbr = be.solver_stats()
    ms_total = ensemble.max_over_ranks(e0.elapsed_time(e1), device="cuda") if world > 1 else e0.elapsed_time(e1)
    value = n * n_units * K_steps / (ms_total / 1e3)
    o = be.options
    out = {"workload": name, "value": value, "unit": UNIT, "ms_per_step": ms_total / K_steps, "steps": K_steps, "warmup": W,
           "gpu_launches": int(l1 - l0), "setup_seconds": t_setup,
           "solver": {"kind": "defect correction (Gauss-Seidel sweeps as the solver)" if o.solver == 2 and o.solver_path == 1
                              else ("BiCGSTAB" if o.solver_path == 1 else "BiCGSTAB, one CTA per constituent"),
                      "iterations_or_cycles_per_step": (i1 - i0) / K_steps, "sweeps_per_step": (sw1 - sw0) / K_steps,
                      "fallbacks_to_bicgstab": int(fallbacks), "worst_status": worst_status, "max_relres": worst_relres,
                      "strips": n_strips, "max_strip_neighbours": max_nbr},
           "clocks": clocks}
    if dump_dir is not None:     # before the profiled steps below overwrite the device's mass fluxes
        out["dumped_outputs"] = dump_outputs(be, W + K_steps - 1, dump_dir, plan.f2, inputs)

    # ---- per-kernel device time (CUDA events between launches on the handle's stream) -> roofline -------------
    roofline = None
    if want_roofline and P > 0:
        be.profile(1)
        sp0 = be.solver_stats()[0]
        for t in range(W + K_steps, W + K_steps + P):
            be.step(t)
        prof = be.profile(0)
        sweeps_prof = be.solver_stats()[0] - sp0
        nnz = 2 * int(np.count_nonzero(plan.f2 < n))
        internal = plan.f2 < n
        Wd = 4 * ((int(np.bincount(np.concatenate([plan.f1[internal], plan.f2[internal]]), minlength=n).max()) + 3) // 4)
        nn, nz, EE = n, nnz, E
        if dd:      # a rank's kernels run over its strip: algorithmic bytes of the strip (rank 0's, the strips are equal)
            frac_own = dd_info.rows_owned / n
            nn, nz, EE = int(dd_info.rows_owned), int(nnz * frac_own), int(E * frac_own)
        n_pre = prof.get("precond", (0.0, 0))[1]
        spl = sweeps_prof / n_pre if (n_pre and o.solver == 2 and o.precond_sweep == 1) else max(0, o.precond_steps - 1)
        fam_bytes = family_bytes(o, nn, nz, EE, K, Wd, spl)
        peak, peak_src = measured_peak()
        total_ms = sum(v[0] for v in prof.values())
        kernels = {}
        for fam, (ms, cnt) in prof.items():
            if not cnt:
                continue
            per = ms / cnt
            entry = {"ms_per_launch": per, "launches_per_step": cnt / P, "ms_per_step": ms / P,
                     "share_of_step": ms / total_ms if total_ms else None}
            if fam in fam_bytes and per > 0:
                gbs = fam_bytes[fam] / (per * 1e-3) / 1e9
                entry.update({"algorithmic_bytes_per_launch": fam_bytes[fam], "achieved_gbs": gbs, "frac": gbs / peak})
            else:   # the one-CTA-per-constituent solve of small meshes works out of shared memory / L2: no HBM roofline
                entry.update({"algorithmic_bytes_per_launch": None, "achieved_gbs": None, "frac": None})
            kernels[fam] = entry
        if kernels:
            dom = max(kernels, key=lambda f: kernels[f]["ms_per_step"])
            names = dict(KERNEL_NAMES, precond=precond_kernel_name(o))
            traffic, traffic_src = None, None
            tp = ROOT / "profiles" / "dominant_kernel_traffic.json"
            if tp.is_file() and dom == "precond" and name == "1m16" and args.scale == 1.0:
                try:
                    tj = json.loads(tp.read_text())
                    ent = tj.get("kernels", {}).get(f"sync{o.precond_sync}")
                    if ent and tj.get("workload") == name and o.precond_colors == ent.get("colours"):
                        traffic = ent["dram_bytes_fixed"] + ent["dram_bytes_per_sweep"] * spl
                        traffic_src = ent.get("source")
                except Exception:
                    pass
            d = kernels[dom]
            roofline = {"bound": "hbm" if d["frac"] is not None else "latency (shared-memory / L2 resident: HBM roofline not applicable)",
                        "kernel": names.get(dom, dom), "family": dom, "achieved": d["achieved_gbs"], "peak": peak,
                        "unit": "GB/s", "frac": d["frac"], "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": d["algorithmic_bytes_per_launch"], "ms_per_launch": d["ms_per_launch"],
                        "sweeps_per_launch": spl if dom == "precond" else None,
                        "share_of_step": d["share_of_step"], "kernels": kernels}
    out["roofline"] = roofline

    # ---- mass-balance scalars: the only collective (NCCL all-reduce over the ranks' units) ------------------------
    t_end = W + K_steps
    local_rows = {}
    for k, unit in enumerate(mine):
        m = be.mass_totals(k, 0, t_end)
        _, f_in, f_out = be.flux_sums(k)
        local_rows[unit] = (m.mass_start, m.mass_end, float(np.nansum(f_in)), float(np.nansum(f_out)))
    if dd:      # every rank holds PARTIAL sums over its strip of the same units: add them up (NCCL all-reduce)
        part = np.array([local_rows[u] for u in range(n_units)])
        mass_table = merge_owned(part, np.ones(part.shape[1], bool), axis=1)
    else:
        mass_table = ensemble.reduce_mass_balance(local_rows, n_units, device="cuda")
    out["mass_balance"] = {"units": n_units, "mass_start_all_units": float(mass_table[:, 0].sum()),
                           "mass_end_all_units": float(mass_table[:, 1].sum()),
                           "boundary_mass_in_all_units": float(mass_table[:, 2].sum()),
                           "boundary_mass_out_all_units": float(mass_table[:, 3].sum()),
                           "reduced_with": "nccl all_reduce" if world > 1 else "single rank"}
    out["config"] = {
        "workload": WORKLOAD_NAMES[name] + (": domain-decomposed over the GPUs" if dd else (", single GPU" if name == "16m" else "")),
        "cells": n, "edges": E, "nnz_offdiag": 2 * int(np.count_nonzero(plan.f2 < n)), "constituents_per_gpu": K, "dt_s": float(dt[0]),
        "diffusion_coefficient": DIFFUSION, "rtol": o.rtol, "solver": o.solver, "solver_path": o.solver_path,
        "precond_steps": o.precond_steps, "precond_sweep": o.precond_sweep, "precond_sync": o.precond_sync,
        "precond_precision": o.precond_precision, "precond_colors": o.precond_colors,
        "l2": "per-step working set (vectors x n x K x 8 B + matrix) >> 126 MB L2; no flush needed"
              if n * K * 56 > 4 * 126e6 else "working set is L2-resident: launch/latency bound, HBM fraction not meaningful",
        "sharding": ("domain decomposition: rows cut into strips of the RCM band, halo rows stored into the peers over NVLink "
                     "from inside the sweep kernel, dot products all-reduced through peer inboxes (no NCCL on the data path)"
                     if dd else "independent constituents/scenarios per rank, mesh replicated, no data-path collective"),
        "domain_decomposition": None if not dd else {"rows_owned_rank0": dd_info.rows_owned, "halo_rows_sent_rank0": dd_info.rows_sent,
                                                       "neighbour_mask_rank0": dd_info.neighbour_mask},
        "units_per_rank": ensemble.ensemble_plan(n_units, world)}
    be.close()

    # ---- end to end through the reference-facing API with host buffers -------------------------------------------
    if want_e2e:
        out["e2e_legs"] = e2e_legs(plan, inputs, K, n_units, ctx, args, opts, W, K_steps)
    return out


def e2e_legs(plan, inputs, K, n_units, ctx, args, opts, W, K_steps):
    """ClearwaterRiverine.update() with HOST buffers: slice t+1 of flow / velocity / volume uploaded from pinned host
    arrays every step, results copied into the host arrays of the model every step.  Three legs:
      contract  -- what the reference's update() leaves on the host: c[t+1] AND the three (T,E) mass-flux arrays of every
                   constituent (transport.py:252-273), output='pipelined' (copies overlap the next update)
      lean      -- c[t+1] only; the mass flux is computed on the device every step and reduced there (N2), not copied
      lean_eager-- the same with output='eager' (every update() returns with the row in place)"""
    import torch
    import torch.distributed as dist
    from clearwater_riverine_b200 import ClearwaterRiverine
    n, E, F = plan.n_real, plan.n_edge, plan.n_face
    legs = {}
    base = {"h2d_bytes_per_step": 4 * E + 4 * E + 4 * F + 8}
    for leg, store_flux, output, n_steps in (("lean", False, "pipelined", K_steps), ("lean_eager", False, "eager", K_steps),
                                             ("contract", True, "pipelined", min(K_steps, 8))):
        Tl = W + n_steps + 1
        model = ClearwaterRiverine.from_arrays(
            plan.f1, plan.f2, plan.face_x, plan.face_y, plan.time_seconds[:Tl], pinned(plan.face_flow[:Tl]),
            pinned(plan.edge_velocity[:Tl]), pinned(plan.volume[:Tl]), DIFFUSION, {f"c{k}": inputs[k][:Tl] for k in range(K)},
            device=ctx.local, stream_hydro=True, store_mass_flux=store_flux, keep_history=0, output=output, **opts)
        for _ in range(W):
            model.update()
        model.sync()
        ctx.barrier()
        torch.cuda.synchronize()
        t_0 = time.perf_counter()
        for _ in range(n_steps):
            model.update()                      # H2D: slice t+1 of flow/velocity/volume; D2H: the step's results
        model.sync()
        torch.cuda.synchronize()
        el = torch.tensor([time.perf_counter() - t_0], device="cuda", dtype=torch.float64)
        if ctx.world > 1:
            dist.all_reduce(el, op=dist.ReduceOp.MAX)
        sec = float(el.item())
        legs[leg] = dict(base, value=n * n_units * n_steps / sec, unit=UNIT, ms_per_step=sec / n_steps * 1e3, steps=n_steps,
                         d2h_bytes_per_step=8 * n * K + (3 * 8 * E * K if store_flux else 0), output=output,
                         store_mass_flux=store_flux)
        model.finalize()
        del model
    return legs


def dd_small_parity(ctx, opts):
    """Domain-decomposed path against the single-GPU answer on a small mesh (N > 1): max scaled difference of the merged
    concentrations after a few steps, and the iteration counts of both."""
    import torch
    from clearwater_riverine_b200 import TransportBackend, synthetic
    from clearwater_riverine_b200.domain import DomainDecomposedBackend
    plan = synthetic.make_plan(260, 240, 6, seed=9, dry_fraction=0.02)
    K, T = 2, 6
    inputs = synthetic.make_inputs(plan, K, seed=9)
    dt = np.append(np.diff(plan.time_seconds), np.nan)
    hint = plan.face_flow.mean(axis=0, dtype=np.float64).astype(np.float32)

    def run(be):
        be.set_geometry(plan.face_x, plan.face_y)
        be.set_hydro_raw(0, plan.face_flow, plan.edge_velocity, plan.volume, dt)
        if isinstance(be, DomainDecomposedBackend):
            be.attach()
        for k in range(K):
            be.set_inputs(k, inputs[k])
        its = [be.step(t).iterations for t in range(T - 1)]
        if isinstance(be, DomainDecomposedBackend):
            return be.gather_state_all(T - 1), its           # collective: every rank's strip merged
        return be.get_state_all(T - 1), its

    dd = DomainDecomposedBackend(plan.f1, plan.f2, plan.n_face, T, K, DIFFUSION, ctx.rank, ctx.world, device=ctx.local, flow_hint=hint,
                                 solver_path=1, **opts)
    merged, its_dd = run(dd)
    dd.close()
    res = None
    if ctx.rank == 0:
        one = TransportBackend(plan.f1, plan.f2, plan.n_face, T, K, DIFFUSION, device=ctx.local, flow_hint=hint, solver_path=1, **opts)
        want, its_one = run(one)
        one.close()
        res = {"cells": plan.n_real, "constituents": K, "steps": T - 1,
               "max_scaled_difference_vs_single_gpu": float(np.abs(merged - want).max() / np.abs(want).max()),
               "cycles_per_step_dd": its_dd, "cycles_per_step_single_gpu": its_one}
    ctx.barrier()
    torch.cuda.synchronize()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline workload (its rate, ms_per_step and --dump-outputs); two legs time fewer "
                         "and report their own count: --impl reference min(steps, 3) (a SuperLU step of the 1M-cell mesh "
                         "takes ~50 s) and the e2e contract leg min(steps, 8) (it keeps the (T, E) mass-flux history of all "
                         "16 constituents in page-locked host memory, ~0.8 GB per step)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="1m16", choices=["1m16", "ohio", "ens64", "ensw", "16m"])
    ap.add_argument("--scale", type=float, default=1.0, help="mesh side scale (debugging only; 1.0 = the named size)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="only the headline workload (no extra.ohio / ens64 / dd16m)")
    ap.add_argument("--sample-reference", action="store_true", help="--impl reference on the 100k-cell sample instead of the 1M mesh")
    ap.add_argument("--extras-budget", type=float, default=420.0, help="seconds of wall clock after which no further extra is started")
    ap.add_argument("--profile-steps", type=int, default=2)
    ap.add_argument("--opt", action="append", default=[], metavar="KEY=VALUE",
                    help="cwr_options override, e.g. --opt precond_steps=8 --opt rtol=1e-12")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (GPU arm, one GPU)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "b200" or world > 1):
        ap.error("--dump-outputs applies to the GPU arm on one GPU")
    args.warmup = max(3, args.warmup) if args.impl == "b200" else args.warmup

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    from clearwater_riverine_b200.backend import bind_to_gpu_numa
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    numa_cpus = bind_to_gpu_numa(local)          # host arrays of this rank are first-touched next to its GPU
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = Ctx(rank, world, local)
    opts = {}
    for kv in args.opt:
        key, val = kv.split("=", 1)
        opts[key] = float(val) if key == "rtol" else int(val)

    dd_main = args.workload == "16m" and world > 1
    head = gpu_workload(args.workload, ctx, args, args.steps, args.warmup, args.profile_steps, opts, dd=dd_main,
                        want_e2e=not args.no_e2e and not dd_main, dump_dir=args.dump_outputs)

    # ---- the other BASELINE configurations, bounded ------------------------------------------------------------
    extra = {}
    if not args.no_extras and args.workload == "1m16" and args.scale == 1.0:
        def within_budget():
            ok = torch.tensor([1.0 if time.perf_counter() - T_START < args.extras_budget else 0.0], device="cuda")
            if world > 1:
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)       # every rank takes the same decision
            return bool(ok.item() > 0)

        def leg(fn):
            try:
                return fn()
            except Exception as exc:            # an extra must never cost the headline line
                return {"error": repr(exc)}

        if world == 1 and within_budget():
            extra["ohio"] = leg(lambda: slim(gpu_workload("ohio", ctx, args, 200, 3, 2, opts, want_e2e=False, want_clocks=False)))
        if within_budget():
            extra["ens64"] = leg(lambda: slim(gpu_workload("ens64", ctx, args, 200, 3, 2, opts, want_e2e=False, want_clocks=False)))
        if within_budget():
            extra["ens_weak"] = leg(lambda: slim(gpu_workload("ensw", ctx, args, 200, 3, 2, opts, want_e2e=False, want_clocks=False)))
        if world > 1 and within_budget():
            extra["dd_small_parity"] = leg(lambda: dd_small_parity(ctx, opts))
        if within_budget():
            extra["dd16m"] = leg(lambda: slim(gpu_workload("16m", ctx, args, 5, 3, 1, opts, dd=world > 1, want_e2e=False, want_clocks=False)))
        else:
            extra["dd16m"] = {"skipped": "extras budget used up"}

    if rank == 0:
        cpu = None
        if not args.no_cpu:
            rate, cms, sample, _ = cpu_reference_rate(4, 1, seed=2, full_size=False)
            cpu = {"value": rate, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample,
                   "ms_per_step": cms, "host_cores_available": os.cpu_count()}
            try:
                cpu["bicgstab_jacobi_solve_only"] = cpu_bicgstab_rate(seed=2)
            except Exception as exc:        # the like-for-like extra must never cost the headline line
                cpu["bicgstab_jacobi_solve_only"] = {"error": repr(exc)}
        legs = head.pop("e2e_legs", None)
        e2e = None
        if legs:
            c = legs["contract"]
            e2e = {"value": c["value"], "unit": UNIT, "h2d_bytes_per_step": c["h2d_bytes_per_step"],
                   "d2h_bytes_per_step": c["d2h_bytes_per_step"], "ms_per_step": c["ms_per_step"], "steps": c["steps"],
                   "api": "ClearwaterRiverine.update(), output='pipelined', store_mass_flux=True: slice t+1 of flow / velocity / volume "
                          "uploaded from pinned host arrays each step; c[t+1] AND the three (T,E) mass-flux arrays of every constituent "
                          "copied into the model's host arrays each step (what the reference's update() fills, transport.py:252-273); "
                          "PCIe-bound: see d2h_bytes_per_step",
                   "lean": dict(legs["lean"], api="the same without the mass-flux history on the host (store_mass_flux=False): the flux is "
                                                  "still computed on the device every step and reduced there (cwr_get_flux_sums)"),
                   "lean_eager": legs["lean_eager"]}
        line = {
            "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": head["steps"], "warmup": head["warmup"],
            "ms_per_step": head["ms_per_step"], "higher_is_better": True,
            "scaling": "strong" if args.workload == "ens64" or dd_main else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": dict(head["config"], host_numa_binding=numa_cpus is not None),
            "clocks": head["clocks"], "e2e": e2e, "gpu_launches": head["gpu_launches"],
            "roofline": head["roofline"], "cpu_baseline": cpu, "solver": head["solver"], "mass_balance": head["mass_balance"],
            "extra": extra or None,
            "wall_seconds": time.perf_counter() - T_START,
        }
        if "dumped_outputs" in head:
            line["dumped_outputs"] = {"dir": str(args.dump_outputs), "arrays": head["dumped_outputs"]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def slim(res):
    """An extra's record: rate, solver statistics and per-family times without the bulky bits."""
    r = res.get("roofline") or {}
    fam = {f: {"ms_per_launch": v["ms_per_launch"], "launches_per_step": v["launches_per_step"], "ms_per_step": v["ms_per_step"],
               "frac": v["frac"]} for f, v in (r.get("kernels") or {}).items()}
    return {"value": res["value"], "unit": UNIT, "ms_per_step": res["ms_per_step"], "steps": res["steps"],
            "scaling": "strong" if res["workload"] in ("ens64", "16m") else ("weak" if res["workload"] == "ensw" else "n/a"), "solver": res["solver"],
            "dominant_kernel": {"kernel": r.get("kernel"), "frac": r.get("frac"), "ms_per_launch": r.get("ms_per_launch"),
                                "share_of_step": r.get("share_of_step")},
            "families": fam, "config": {k: res["config"][k] for k in ("workload", "cells", "constituents_per_gpu", "precond_colors",
                                                                      "precond_sync", "solver", "solver_path", "domain_decomposition")},
            "mass_balance": res["mass_balance"], "gpu_launches": res["gpu_launches"], "setup_seconds": res["setup_seconds"]}


if __name__ == "__main__":
    main()
