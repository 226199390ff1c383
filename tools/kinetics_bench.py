#!/usr/bin/env python
"""What first-order kinetics on the device costs and what it saves (cwr_set_kinetics, k_react).

  python tools/kinetics_bench.py [--reps 20] [--out profiles/kinetics_bench.json]

1M x 16 (bench.py's 1m16 plan; a 16-constituent network with the last constituent as the temperature,
synthetic.make_kinetics): the step time with kinetics off and on, measured alternately on the same handle (the same step
t is taken again and again, so both see the same system) with CUDA events; k_react's time as the delta of the
CWR_FAM_RHS profile family (k_rhs + k_boundary_rhs + k_react), also with the same network at a constant temperature
(no per-row exp); its bytes 3V + 12n (read c~, vol, D; write c~' and b)
over that time against a device-to-device copy's rate.  Ohio-shaped mesh, K = 1 and 64 scenarios with 64 decay rates:
the time kinetics adds per step in cwr_run.  The coupled loop both ways at both sizes: the same reactions on the host
(every constituent copied down, reacted in numpy, pushed back through the update_concentration override) against the
device kinetics.  With sources (cwr_set_kinetics_sources), 1M x 16: the same network with the zero-order sources and
exchange of synthetic.make_kinetics_sources (sediment-oxygen-demand-like sinks, reaeration toward oxygen saturation, an
equilibrium temperature), with the temperature constituent and at a constant temperature, each against the same network
without its sources, alternately on the same handle: the step time and k_react's time (the CWR_FAM_RHS delta).
With Monod factors (cwr_set_kinetics_limits), 1M x 16: the network with its sources and the factors of
synthetic.make_kinetics_limits against the same network without the factors, alternately on the same handle, with the
temperature constituent and at a constant temperature (--limits-only: this leg alone).
With depth-scaled processes (cwr_set_kinetics_depth), 1M x 16: the network with its sources and the flags of
synthetic.make_kinetics_depth over the plan areas against the same network without the flags, alternately on the same
handle, with the temperature constituent and at a constant temperature (--depth-only: this leg alone).
With time-varying forcing (cwr_set_kinetics_forcing), 1M x 16: the network with its sources and the diurnal series of
synthetic.make_kinetics_forcing (light-scaled sources and die-off, wind-scaled exchange, moving equilibria and, at a
constant temperature, a temperature series) against the same network unforced, alternately on the same handle, with the
temperature constituent and at a constant temperature (--forcing-only: this leg alone).
--parent-root DIR: the kinetics-only, the sources-only and the sources-with-factors network timed in this tree's build
and in DIR's (another checkout with its library built), one process per measurement, alternating, --parent-rounds times each; every process also reports the spread of
its own repetitions.
Prints one JSON object and writes it to --out.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
if "--regression-child" in sys.argv:          # the package and its library from the tree named by --root
    sys.path.insert(0, sys.argv[sys.argv.index("--root") + 1])


def gpu_name_and_power():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else None
    except Exception:
        return None


def copy_rate_gbs(torch):
    """Device-to-device copy of 4 GiB (larger than L2): bytes read + written over the time, best of 5."""
    a = torch.empty(1 << 29, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    best = float("inf")
    for _ in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); b.copy_(a); e1.record(); e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    return 2 * 8 * (1 << 29) / (best * 1e-3) / 1e9


def build(plan, inputs, torch, **opt):
    from clearwater_riverine_b200 import TransportBackend
    K = inputs.shape[0]
    be = TransportBackend(plan.f1, plan.f2, plan.n_face, plan.n_time, K, 0.1, **opt)
    be.set_geometry(plan.face_x, plan.face_y)
    be.set_hydro_raw(0, plan.face_flow, plan.edge_velocity, plan.volume, np.append(np.diff(plan.time_seconds), np.nan))
    for k in range(K):
        be.set_inputs(k, inputs[k])
    return be


def timed(torch, be, fn, n):
    """ms per call of fn over n calls, CUDA events on the handle's stream."""
    s = torch.cuda.ExternalStream(be.stream())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    for _ in range(n):
        fn()
    e1.record(s)
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def alternate(torch, be, kin, fn, reps, n):
    """fn timed with kinetics off and on, alternately, reps times each: medians (ms)."""
    off, on = [], []
    for _ in range(reps):
        be.set_kinetics(None)
        off.append(timed(torch, be, fn, n))
        be.set_kinetics(**kin)
        on.append(timed(torch, be, fn, n))
    return float(np.median(off)), float(np.median(on))


def alternate_sources(torch, be, kin, src, step, reps):
    """The network without and with its sources, alternately, reps times each: medians of the step time (ms, CUDA events)
    and of the CWR_FAM_RHS family time (ms per step, in separate profiled steps)."""
    out = {"step_ms": ([], []), "rhs_family_ms": ([], [])}
    for _ in range(reps):
        for i, with_src in enumerate((False, True)):
            be.set_kinetics(**kin)
            if with_src:
                be.set_kinetics_sources(**src)
            step()
            out["step_ms"][i].append(timed(torch, be, step, 5))
            be.profile(1)
            for _ in range(5):
                step()
            out["rhs_family_ms"][i].append(be.profile(-1)["rhs"][0] / 5)
            be.profile(0)
    return {f"{key}_{name}": float(np.median(v[i])) for key, v in out.items() for i, name in enumerate(("without", "with"))}


def alternate_limits(torch, be, kin, src, lim, step, reps):
    """The network with its sources, without and with its Monod factors, alternately, reps times each: medians of the step
    time (ms, CUDA events) and of the CWR_FAM_RHS family time (ms per step, in separate profiled steps)."""
    out = {"step_ms": ([], []), "rhs_family_ms": ([], [])}
    for _ in range(reps):
        for i, with_lim in enumerate((False, True)):
            be.set_kinetics(**kin)
            be.set_kinetics_sources(**src)
            if with_lim:
                be.set_kinetics_limits(**lim)
            step()
            out["step_ms"][i].append(timed(torch, be, step, 5))
            be.profile(1)
            for _ in range(5):
                step()
            out["rhs_family_ms"][i].append(be.profile(-1)["rhs"][0] / 5)
            be.profile(0)
    return {f"{key}_{name}": float(np.median(v[i])) for key, v in out.items() for i, name in enumerate(("without", "with"))}


def limits_leg(torch, res, reps, scale):
    """1M x 16 with sources: without and with Monod factors, with the temperature constituent and at a constant one."""
    import bench
    from clearwater_riverine_b200 import synthetic
    plan, K = bench.workload_plan("1m16", 14, seed=0, scale=scale)
    inputs, kin = synthetic.make_kinetics(synthetic.make_inputs(plan, K, seed=0), seed=0, decay_range=(0.05, 2.0))
    src = synthetic.make_kinetics_sources(kin, seed=0, rate_range=(0.05, 2.0))
    lim = synthetic.make_kinetics_limits(kin, src, seed=0)
    be = build(plan, inputs, torch)
    for t in range(3):
        be.step(t)
    step = lambda: be.step(3)
    be.profile(1)
    for _ in range(10):
        step()
    fam_off = be.profile(-1)["rhs"][0] / 10
    be.profile(0)
    kin_const = dict(kin, temperature_k=-1, temperature_c=24.0)
    for key, k in (("1m16_limits", kin), ("1m16_limits_constant_temperature", kin_const)):
        r = alternate_limits(torch, be, k, src, lim, step, reps)
        r["k_react_ms_without_limits"] = r["rhs_family_ms_without"] - fam_off
        r["k_react_ms_with_limits"] = r["rhs_family_ms_with"] - fam_off
        r["k_react_added_ms"] = r["rhs_family_ms_with"] - r["rhs_family_ms_without"]
        r["step_added_ms"] = r["step_ms_with"] - r["step_ms_without"]
        r["factors"] = int(len(lim["process"]))
        r["limited_processes"] = int(len({(int(p), int(c)) for p, c in zip(lim["process"], lim["column"])}))
        res[key] = r
    be.close()


def alternate_depth(torch, be, kin, src, flags, dep, step, reps):
    """The network with its sources, without and with its depth flags (kin, src: the unflagged rates; flags: the flagged
    ones and the set_kinetics_depth arguments), alternately, reps times each: medians of the step time (ms, CUDA events)
    and of the CWR_FAM_RHS family time (ms per step, in separate profiled steps)."""
    out = {"step_ms": ([], []), "rhs_family_ms": ([], [])}
    for _ in range(reps):
        for i, with_depth in enumerate((False, True)):
            k, s = (flags[0], flags[1]) if with_depth else (kin, src)
            be.set_kinetics(**k)
            be.set_kinetics_sources(**s)
            if with_depth:
                be.set_kinetics_depth(**dep)
            step()
            out["step_ms"][i].append(timed(torch, be, step, 5))
            be.profile(1)
            for _ in range(5):
                step()
            out["rhs_family_ms"][i].append(be.profile(-1)["rhs"][0] / 5)
            be.profile(0)
    return {f"{key}_{name}": float(np.median(v[i])) for key, v in out.items() for i, name in enumerate(("without", "with"))}


def depth_leg(torch, res, reps, scale):
    """1M x 16 with sources: without and with depth flags, with the temperature constituent and at a constant one."""
    import bench
    from clearwater_riverine_b200 import synthetic
    plan, K = bench.workload_plan("1m16", 14, seed=0, scale=scale)
    inputs, kin = synthetic.make_kinetics(synthetic.make_inputs(plan, K, seed=0), seed=0, decay_range=(0.05, 2.0))
    src = synthetic.make_kinetics_sources(kin, seed=0, rate_range=(0.05, 2.0))
    kin_d, src_d, flags = synthetic.make_kinetics_depth(kin, src, seed=0)
    dep = dict(cell_area=plan.cell_area, min_depth=0.01, **flags)
    be = build(plan, inputs, torch)
    for t in range(3):
        be.step(t)
    step = lambda: be.step(3)
    be.profile(1)
    for _ in range(10):
        step()
    fam_off = be.profile(-1)["rhs"][0] / 10
    be.profile(0)
    for key, const in (("1m16_depth", False), ("1m16_depth_constant_temperature", True)):
        c = (lambda k: dict(k, temperature_k=-1, temperature_c=24.0)) if const else (lambda k: k)
        r = alternate_depth(torch, be, c(kin), src, (c(kin_d), src_d), dep, step, reps)
        r["k_react_ms_without_depth"] = r["rhs_family_ms_without"] - fam_off
        r["k_react_ms_with_depth"] = r["rhs_family_ms_with"] - fam_off
        r["k_react_added_ms"] = r["rhs_family_ms_with"] - r["rhs_family_ms_without"]
        r["step_added_ms"] = r["step_ms_with"] - r["step_ms_without"]
        r["flagged_processes"] = {k: int(np.sum(v)) for k, v in flags.items()}
        res[key] = r
    be.close()


def alternate_forcing(torch, be, kin, src, frc, step, reps):
    """The network with its sources, unforced and forced, alternately, reps times each: medians and ranges of the step
    time (ms, CUDA events) and of the CWR_FAM_RHS family time (ms per step, in separate profiled steps)."""
    out = {"step_ms": ([], []), "rhs_family_ms": ([], [])}
    for _ in range(reps):
        for i, forced in enumerate((False, True)):
            be.set_kinetics(**kin)
            be.set_kinetics_sources(**src)
            if forced:
                be.set_kinetics_forcing(**frc)
            step()
            out["step_ms"][i].append(timed(torch, be, step, 5))
            be.profile(1)
            for _ in range(5):
                step()
            out["rhs_family_ms"][i].append(be.profile(-1)["rhs"][0] / 5)
            be.profile(0)
    res = {}
    for key, v in out.items():
        for i, name in enumerate(("unforced", "forced")):
            res[f"{key}_{name}"] = float(np.median(v[i]))
            res[f"{key}_{name}_range"] = [float(min(v[i])), float(max(v[i]))]
    return res


def forcing_leg(torch, res, reps, scale):
    """1M x 16 with sources: unforced and forced, with the temperature constituent and at a constant one."""
    import bench
    from clearwater_riverine_b200 import synthetic
    plan, K = bench.workload_plan("1m16", 14, seed=0, scale=scale)
    inputs, kin = synthetic.make_kinetics(synthetic.make_inputs(plan, K, seed=0), seed=0, decay_range=(0.05, 2.0))
    src = synthetic.make_kinetics_sources(kin, seed=0, rate_range=(0.05, 2.0))
    be = build(plan, inputs, torch)
    for t in range(3):
        be.step(t)
    step = lambda: be.step(3)
    be.profile(1)
    for _ in range(10):
        step()
    fam_off = be.profile(-1)["rhs"][0] / 10
    be.profile(0)
    kin_const = dict(kin, temperature_k=-1, temperature_c=24.0)
    for key, k in (("1m16_forcing", kin), ("1m16_forcing_constant_temperature", kin_const)):
        frc = synthetic.make_kinetics_forcing(k, src, plan.time_seconds, seed=0)
        r = alternate_forcing(torch, be, k, src, frc, step, reps)
        r["k_react_ms_unforced"] = r["rhs_family_ms_unforced"] - fam_off
        r["k_react_ms_forced"] = r["rhs_family_ms_forced"] - fam_off
        r["k_react_added_ms"] = r["rhs_family_ms_forced"] - r["rhs_family_ms_unforced"]
        r["step_added_ms"] = r["step_ms_forced"] - r["step_ms_unforced"]
        r["series_per_target"] = {name: int(np.sum(frc["target"] == g)) for g, name in
                                  enumerate(("temperature", "equilibrium", "decay_scale", "source_scale", "exchange_scale"))}
        res[key] = r
    be.close()


def regression_child(reps, scale):
    """One process of --parent-root: kinetics off, the kinetics-only, the sources-only and the sources-with-factors 1M x 16
    network (temperature constituent) on one handle; medians and spreads (min, max) of the step time and of k_react's time (CWR_FAM_RHS
    delta).  Uses only calls both builds have."""
    import os
    import torch
    import bench
    from clearwater_riverine_b200 import synthetic
    from clearwater_riverine_b200.backend import library_path
    plan, K = bench.workload_plan("1m16", 14, seed=0, scale=scale)
    inputs, kin = synthetic.make_kinetics(synthetic.make_inputs(plan, K, seed=0), seed=0, decay_range=(0.05, 2.0))
    src = synthetic.make_kinetics_sources(kin, seed=0, rate_range=(0.05, 2.0))
    lim = synthetic.make_kinetics_limits(kin, src, seed=0)
    be = build(plan, inputs, torch)
    for t in range(3):
        be.step(t)
    step = lambda: be.step(3)
    modes = {"off": None, "kinetics": (kin, None, None), "sources": (kin, src, None), "limits": (kin, src, lim)}
    samples = {m: {"step_ms": [], "rhs_family_ms": []} for m in modes}
    for _ in range(reps):
        for m, v in modes.items():
            if v is None:
                be.set_kinetics(None)
            else:
                be.set_kinetics(**v[0])
                if v[1] is not None:
                    be.set_kinetics_sources(**v[1])
                if v[2] is not None:
                    be.set_kinetics_limits(**v[2])
            step()
            samples[m]["step_ms"].append(timed(torch, be, step, 5))
            be.profile(1)
            for _ in range(5):
                step()
            samples[m]["rhs_family_ms"].append(be.profile(-1)["rhs"][0] / 5)
            be.profile(0)
    be.close()
    lib = Path(os.environ.get("CWR_B200_LIB", library_path())).resolve()   # what load_library actually loaded
    out = {"library": str(lib.relative_to(Path.cwd().resolve())) if lib.is_relative_to(Path.cwd().resolve()) else str(lib)}
    off = np.array(samples["off"]["rhs_family_ms"])
    for m in ("kinetics", "sources", "limits"):
        st, fam = np.array(samples[m]["step_ms"]), np.array(samples[m]["rhs_family_ms"])
        react = fam - np.median(off)
        out[m] = {"step_ms": float(np.median(st)), "step_ms_min": float(st.min()), "step_ms_max": float(st.max()),
                  "k_react_ms": float(np.median(react)), "k_react_ms_min": float(react.min()),
                  "k_react_ms_max": float(react.max())}
    print(json.dumps(out))


def parent_comparison(parent_root: str, rounds: int, reps: int, scale: float) -> dict:
    """regression_child in this tree and in parent_root, alternately (one process each), `rounds` times each."""
    import os
    runs = {"this": [], "parent": []}
    for _ in range(rounds):
        for name, root in (("parent", parent_root), ("this", str(ROOT))):
            env = dict(os.environ, CWR_B200_LIB=str(Path(root) / "clearwater_riverine_b200" / "libcwr_b200.so"))
            out = subprocess.run([sys.executable, str(Path(__file__).resolve()), "--regression-child", "--root", root,
                                  "--reps", str(reps), "--scale", str(scale)], capture_output=True, text=True, env=env,
                                 timeout=1800)
            if out.returncode != 0:
                raise SystemExit(f"regression child failed ({name}):\n{out.stderr[-3000:]}")
            runs[name].append(json.loads(out.stdout.strip().splitlines()[-1]))
    res = {"rounds": rounds, "reps_per_round": reps, "runs": runs}
    for m in ("kinetics", "sources", "limits"):
        for key in ("step_ms", "k_react_ms"):
            a = [r[m][key] for r in runs["this"]]
            b = [r[m][key] for r in runs["parent"]]
            res[f"{m}_{key}_this_median"], res[f"{m}_{key}_parent_median"] = float(np.median(a)), float(np.median(b))
            res[f"{m}_{key}_this_range"], res[f"{m}_{key}_parent_range"] = [min(a), max(a)], [min(b), max(b)]
    return res


def host_loop(be, kin, t0, steps, dt):
    """The coupled loop with the reactions on the host: c[t] down, numpy reactions, override up, step.  s per step."""
    from oracle.kinetics import react
    be.set_kinetics(None)
    t_start = time.perf_counter()
    for t in range(t0, t0 + steps):
        c = be.get_state_all(t)
        temp = kin["temperature_k"] if kin["temperature_k"] >= 0 else kin["temperature_c"]
        c = react(c, dt, kin["decay_per_day"], kin["theta"], kin["yields"], temp, kin["temperature_k"] >= 0)
        be.set_state_all(t, c)
        be.step(t)
    be.get_state_all(t0 + steps)
    return (time.perf_counter() - t_start) / steps


def device_loop(torch, be, kin, t0, steps):
    be.set_kinetics(**kin)
    t_start = time.perf_counter()
    be.run(t0, t0 + steps)
    be.get_state_all(t0 + steps)
    return (time.perf_counter() - t_start) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--scale", type=float, default=1.0, help="1m16 mesh side scale (1.0 = 1M cells)")
    ap.add_argument("--out", default=None)
    ap.add_argument("--limits-only", action="store_true", help="only the Monod-factor leg (and --parent-root)")
    ap.add_argument("--depth-only", action="store_true", help="only the depth leg (and --parent-root)")
    ap.add_argument("--forcing-only", action="store_true", help="only the forcing leg (and --parent-root)")
    ap.add_argument("--parent-root", default=None,
                    help="another checkout with its library built: the no-factor networks timed in both builds, alternately")
    ap.add_argument("--parent-rounds", type=int, default=3)
    ap.add_argument("--regression-child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--root", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.regression_child:
        regression_child(args.reps, args.scale)
        return
    import torch
    import bench
    from clearwater_riverine_b200 import synthetic
    if not torch.cuda.is_available():
        raise SystemExit("kinetics_bench needs a CUDA device")
    res = {"gpu": gpu_name_and_power()}
    if args.limits_only or args.depth_only or args.forcing_only:
        leg = limits_leg if args.limits_only else depth_leg if args.depth_only else forcing_leg
        leg(torch, res, args.reps, args.scale)
        if args.parent_root:
            res["no_factor_paths_vs_parent"] = parent_comparison(args.parent_root, args.parent_rounds, max(3, args.reps // 3),
                                                                 args.scale)
        return emit(res, args.out)
    res["d2d_copy_gbs"] = copy_rate_gbs(torch)

    # --- 1M x 16 ------------------------------------------------------------------------------------------------
    T = 14
    plan, K = bench.workload_plan("1m16", T, seed=0, scale=args.scale)
    inputs, kin = synthetic.make_kinetics(synthetic.make_inputs(plan, K, seed=0), seed=0, decay_range=(0.05, 2.0))
    be = build(plan, inputs, torch)
    n = be.n_real
    for t in range(3):
        be.step(t)
    t = 3
    step = lambda: be.step(t)
    be.set_kinetics(**kin)
    for _ in range(3):
        step()
    off, on = alternate(torch, be, kin, step, args.reps, 5)
    fam = {}
    # "const": the same network at a constant temperature -- the per-row exp of theta^(T - 20) is gone (one factor per
    # constituent per CTA), what is left is the tile's load / chain / store
    kin_const = dict(kin, temperature_k=-1, temperature_c=24.0)
    for mode in ("off", "on", "const"):
        be.set_kinetics(None) if mode == "off" else be.set_kinetics(**(kin if mode == "on" else kin_const))
        step()
        be.profile(1)
        for _ in range(10):
            step()
        fam[mode] = be.profile(-1)["rhs"][0] / 10
        be.profile(0)
    react_ms = fam["on"] - fam["off"]
    react_const_ms = fam["const"] - fam["off"]
    nbytes = 3 * 8 * n * K + 12 * n
    res["1m16"] = {"cells": n, "K": K, "step_ms_off": off, "step_ms_on": on, "added_ms": on - off,
                   "added_fraction": (on - off) / off, "rhs_family_ms_off": fam["off"], "rhs_family_ms_on": fam["on"],
                   "k_react_ms": react_ms, "k_react_bytes": nbytes, "k_react_gbs": nbytes / (react_ms * 1e-3) / 1e9,
                   "k_react_of_copy_rate": nbytes / (react_ms * 1e-3) / 1e9 / res["d2d_copy_gbs"],
                   "k_react_ms_constant_temperature": react_const_ms,
                   "k_react_of_copy_rate_constant_temperature": nbytes / (react_const_ms * 1e-3) / 1e9 / res["d2d_copy_gbs"]}
    # the same network with its sources, and at a constant temperature (s, r ceq and phi once per CTA)
    src = synthetic.make_kinetics_sources(kin, seed=0, rate_range=(0.05, 2.0))
    for key, k in (("1m16_sources", kin), ("1m16_sources_constant_temperature", kin_const)):
        r = alternate_sources(torch, be, k, src, step, args.reps)
        r["k_react_added_ms"] = r["rhs_family_ms_with"] - r["rhs_family_ms_without"]
        r["step_added_ms"] = r["step_ms_with"] - r["step_ms_without"]
        r["k_react_ms_without_sources"] = r["rhs_family_ms_without"] - fam["off"]
        r["k_react_ms_with_sources"] = r["rhs_family_ms_with"] - fam["off"]
        r["source_columns"] = int(np.count_nonzero((src["source_per_day"] != 0) | (src["exchange_per_day"] != 0)))
        res[key] = r
    steps = 8
    res["1m16"]["coupled_host_ms_per_step"] = 1e3 * host_loop(be, kin, 4, steps, 30.0)
    res["1m16"]["coupled_device_ms_per_step"] = 1e3 * device_loop(torch, be, kin, 4, steps)
    be.close()
    del inputs, plan

    # --- Ohio-shaped mesh ---------------------------------------------------------------------------------------
    T = 202
    plan = synthetic.ohio_like(T, seed=2)
    for K in (1, 64):
        inputs = synthetic.make_inputs(plan, K, seed=2)
        kin = dict(decay_per_day=np.linspace(0.05, 3.0, K), theta=np.full(K, 1.047), yields=None, temperature_k=-1,
                   temperature_c=17.0)
        be = build(plan, inputs, torch)
        be.set_kinetics(**kin)
        be.run(0, 200)
        off, on = alternate(torch, be, kin, lambda: be.run(0, 200), max(3, args.reps // 3), 1)
        key = "ohio" if K == 1 else "ohio_ens64"
        res[key] = {"cells": be.n_real, "K": K, "solver_path": be.options.solver_path, "step_ms_off": off / 200,
                    "step_ms_on": on / 200, "added_us_per_step": 1e3 * (on - off) / 200}
        res[key]["coupled_host_ms_per_step"] = 1e3 * host_loop(be, kin, 0, 100, 3600.0)
        res[key]["coupled_device_ms_per_step"] = 1e3 * device_loop(torch, be, kin, 0, 100)
        be.close()
    limits_leg(torch, res, args.reps, args.scale)
    depth_leg(torch, res, args.reps, args.scale)
    forcing_leg(torch, res, args.reps, args.scale)
    if args.parent_root:
        res["no_factor_paths_vs_parent"] = parent_comparison(args.parent_root, args.parent_rounds, max(3, args.reps // 3),
                                                             args.scale)
    emit(res, args.out)


def emit(res: dict, out) -> None:
    print(json.dumps(res))
    if out:
        Path(out).parent.mkdir(parents=True, exist_ok=True)
        Path(out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
