#!/usr/bin/env python
"""Parity of the domain-decomposed path (one process per GPU, NVLink peer memory) -- run under torchrun:

  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 \
      tools/dd_check.py [--side 160] [--K 3] [--steps 6] [--kinetics]

Every rank builds the same synthetic mesh, owns one strip of it and steps; the merged concentrations are
compared with (a) the oracle (reference arithmetic incl. SuperLU, on rank 0; rtol 1e-9 per step as in
tests/test_gpu_parity.py) and (b) a single-GPU run of the same library on rank 0's GPU.  Mass totals and
boundary flux sums are checked as sums of the per-rank partial values.  --kinetics: the same with a first-order
network (synthetic.make_kinetics) reacted on the device, in every other case with sources and exchange as well
(synthetic.make_kinetics_sources), in every fourth with Monod factors (synthetic.make_kinetics_limits) and, in the cases
with sources 1 and 3 mod 4, with depth-scaled processes over the plan areas (synthetic.make_kinetics_depth) and, in every
case with sources, with time-varying forcing (synthetic.make_kinetics_forcing), the oracle being
oracle.kinetics_forcing.KineticsRiverine, and the ranks' reaction masses summed against the single-GPU ones.  Prints one JSON line per case on
rank 0; exit code 0 only if every check passed on every rank.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--side", type=int, default=160)
    ap.add_argument("--K", type=int, default=3)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--no-oracle", action="store_true")
    ap.add_argument("--kinetics", action="store_true",
                    help="react a first-order network on the device in every step, with sources and exchange in every other case "
                         "and Monod factors in every fourth")
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    from clearwater_riverine_b200 import TransportBackend, synthetic
    from clearwater_riverine_b200.domain import DomainDecomposedBackend, merge_owned
    from oracle import reference_step as ref
    from oracle.kinetics_depth import depth_terms
    from oracle.kinetics_forcing import KineticsRiverine, forcing_terms
    from oracle.kinetics_limits import limit_terms

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    D = 0.1
    ok_all = True
    cases = [dict(), dict(dd_halo_per_colour=1), dict(precond_sweep=0, precond_steps=4),
             dict(precond_precision=64, precond_steps=3, precond_colors=9), dict(solver=1), dict(precond_sync=2),
             dict(solver=1, precond_sync=1), dict(solver=1, precond_sweep=0, precond_steps=5)]
    for ci, opts in enumerate(cases):
        K, T = args.K, args.steps + 1
        plan = synthetic.make_plan(args.side, args.side * 3 // 4, T, dt=30.0, tri_fraction=0.1, dry_fraction=0.02,
                                   courant=1.5, seed=40 + ci)
        n = plan.n_real
        adv, _, _, cdiff, dt = ref.derive_coefficients(plan.face_flow, plan.edge_velocity, plan.face_x, plan.face_y,
                                                       plan.f1, plan.f2, D, plan.time_seconds)
        inputs = synthetic.make_inputs(plan, K, seed=40 + ci)
        kin = src = lim = dep = frc = None
        if args.kinetics:
            inputs, kin = synthetic.make_kinetics(inputs, seed=40 + ci)
            if ci % 2:
                src = synthetic.make_kinetics_sources(kin, seed=40 + ci)
            if ci % 4 == 3:
                lim = synthetic.make_kinetics_limits(kin, src, seed=40 + ci)
            if ci % 2 and ci < 4:
                kin, src, flags = synthetic.make_kinetics_depth(kin, src, seed=40 + ci)
                dep = dict(cell_area=plan.cell_area, min_depth=0.05, **flags)
            if ci % 2:
                frc = synthetic.make_kinetics_forcing(kin, src, plan.time_seconds, seed=40 + ci, period=6 * 30.0)
        be = DomainDecomposedBackend(plan.f1, plan.f2, plan.n_face, T, K, D, rank, world, device=local, **opts)
        be.set_hydro(0, adv, cdiff, plan.edge_velocity, plan.volume, dt)
        info = be.attach()
        for k in range(K):
            be.set_inputs(k, inputs[k])
        if kin is not None:
            be.set_kinetics(**kin)
        if src is not None:
            be.set_kinetics_sources(**src)
        if lim is not None:
            be.set_kinetics_limits(**lim)
        if dep is not None:
            be.set_kinetics_depth(**dep)
        if frc is not None:
            be.set_kinetics_forcing(**frc)
        single = oracle = None
        if rank == 0:
            single = TransportBackend(plan.f1, plan.f2, plan.n_face, T, K, D, device=local, solver_path=1,
                                      **{k: v for k, v in opts.items() if not k.startswith("dd_")})
            single.set_hydro(0, adv, cdiff, plan.edge_velocity, plan.volume, dt)
            for k in range(K):
                single.set_inputs(k, inputs[k])
            if kin is not None:
                single.set_kinetics(**kin)
            if src is not None:
                single.set_kinetics_sources(**src)
            if lim is not None:
                single.set_kinetics_limits(**lim)
            if dep is not None:
                single.set_kinetics_depth(**dep)
            if frc is not None:
                single.set_kinetics_forcing(**frc)
            if not args.no_oracle:
                mesh = ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, plan.edge_velocity, plan.volume, dt, D)
                named = {f"c{k}": inputs[k] for k in range(K)}
                if kin is None:
                    oracle = ref.OracleRiverine(mesh, named)
                else:
                    temperature = f"c{kin['temperature_k']}" if kin["temperature_k"] >= 0 else kin["temperature_c"]
                    oracle = KineticsRiverine(mesh, named, kin["decay_per_day"], kin["theta"], kin["yields"], temperature,
                                              **(src or {}), **limit_terms(**(lim or {})), **depth_terms(**(dep or {})),
                                              **forcing_terms(**(frc or {})))
        worst_oracle = worst_single = 0.0
        iters = []
        status = 0
        for t in range(args.steps):
            dist.barrier()                                           # rank 0 also runs the single-GPU and oracle steps
            si = be.step(t)
            status = status or si.status
            iters.append(si.iterations)
            merged = be.gather_state_all(t + 1)                      # collective
            if rank == 0:
                s1 = single.step(t)
                ref1 = single.get_state_all(t + 1)
                worst_single = max(worst_single, float(np.abs(merged - ref1).max() / np.abs(ref1).max()))
                if oracle is not None:
                    oracle.update()
                    want = np.stack([oracle.constituent_dict[f"c{k}"].concentration[t + 1][:n] for k in range(K)])
                    worst_oracle = max(worst_oracle, float(np.abs(merged - want).max() / np.abs(want).max()))
        # partial sums over the owned part -> totals
        m_dd = be.gather_mass_totals(0, 0, args.steps)
        fsum = np.nansum(np.stack(be.flux_sums(0)), axis=1)
        fsum = merge_owned(fsum, np.ones(3, bool))
        rmass = np.array([be.gather_reaction_mass(k) for k in range(K)]) if kin is not None else None   # collective
        ok = status == 0
        line = None
        if rank == 0:
            m1 = single.mass_totals(0, 0, args.steps)
            f1 = np.nansum(np.stack(single.flux_sums(0)), axis=1)
            mass_err = abs(m_dd[3] - m1.mass_end) / abs(m1.mass_end)
            flux_err = float(np.abs(fsum - f1).max() / max(1e-300, np.abs(f1).max()))
            ok = ok and worst_single < 1e-9 and (oracle is None or worst_oracle < 1e-9) and mass_err < 1e-9 and flux_err < 1e-9
            rmass_err = None
            if kin is not None:
                r1 = np.array([single.reaction_mass(k) for k in range(K)])
                rmass_err = float(np.abs(rmass - r1).max() / max(1e-300, np.abs(r1).max()))
                ok = ok and rmass_err < 1e-9
            line = {"case": opts, "world": world, "cells": n, "K": K, "steps": args.steps, "rows_owned_rank0": info.rows_owned,
                    "rows_sent_rank0": info.rows_sent, "colors": info.n_colors, "levels": info.n_levels,
                    "iterations_per_step": iters, "single_gpu_iterations_last_step": s1.iterations,
                    "max_rel_diff_vs_single_gpu": worst_single, "max_rel_diff_vs_oracle": worst_oracle if oracle is not None else None,
                    "mass_end_rel_diff": mass_err, "boundary_flux_sums_rel_diff": flux_err, "ok": bool(ok)}
            if kin is not None:
                line["reaction_mass_rel_diff"] = rmass_err
                line["sources"] = src is not None
                line["limits"] = lim is not None
                line["depth"] = dep is not None
                line["forcing"] = frc is not None
            single.close()
        flag = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok_all = ok_all and bool(flag.item())
        if rank == 0:
            print(json.dumps(line), flush=True)
        be.close()
        dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok_all else 1)


if __name__ == "__main__":
    main()
