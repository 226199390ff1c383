"""bench.py's reference arm runs on the host cores only (oracle = reference arithmetic incl. SuperLU) and must
print the benchmark's JSON line; checked here on CPU with --sample-reference (the 100k-cell sample: the arm's default,
the 1M-cell headline mesh, takes ~50 s per SuperLU solve).  The GPU arm: its --dump-outputs files on the small
Ohio-shaped workload (GPU test), and its refusal to run without a device."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]


@pytest.mark.timeout(300)
def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--sample-reference"],
                         capture_output=True, text=True, timeout=280, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "cell_timesteps_per_sec" and line["unit"] == "cell-timesteps/s"
    assert line["higher_is_better"] is True and line["n_gpus"] == 1 and line["steps"] == 1
    assert line["value"] > 0 and line["ms_per_step"] > 0
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == 1 and cb["value"] == line["value"] and "sample" in cb
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_gpu_arm_dumps_the_outputs_of_its_last_timed_step(tmp_path):
    """--dump-outputs: finite float64 arrays, the same on a second run, equal to the oracle's concentrations and mass
    fluxes after exactly --warmup + --steps steps of the same seeded workload."""
    import bench
    from clearwater_riverine_b200 import synthetic
    from oracle import reference_step as ref
    warmup, steps, profile_steps = 3, 4, 2

    def run(out_dir):
        out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "ohio", "--steps", str(steps), "--warmup", str(warmup),
                              "--profile-steps", str(profile_steps), "--no-e2e", "--no-cpu", "--dump-outputs", str(out_dir)],
                             capture_output=True, text=True, timeout=400, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        return json.loads(out.stdout.strip().splitlines()[-1])

    line = run(tmp_path / "a")
    run(tmp_path / "b")
    assert line["steps"] == steps
    names = ["advection_mass_flux", "concentration", "diffusion_mass_flux", "total_mass_flux"]
    assert sorted(p.stem for p in (tmp_path / "a").iterdir()) == names
    got = {nm: np.load(tmp_path / "a" / f"{nm}.npy") for nm in names}
    for nm in names:
        b = np.load(tmp_path / "b" / f"{nm}.npy")
        assert got[nm].dtype == np.float64 and np.isfinite(got[nm]).all(), nm
        np.testing.assert_allclose(got[nm], b, rtol=1e-12, atol=0)

    # the oracle on the same plan and inputs (bench.py's constituent 0 of rank 0), stepped to the last timed step
    plan, _ = bench.workload_plan("ohio", warmup + steps + profile_steps + 1, seed=2)
    adv, _, _, cdiff, dt = ref.derive_coefficients(plan.face_flow, plan.edge_velocity, plan.face_x, plan.face_y, plan.f1, plan.f2,
                                                   bench.DIFFUSION, plan.time_seconds)
    mesh = ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, plan.edge_velocity, plan.volume, dt, bench.DIFFUSION)
    oracle = ref.OracleRiverine(mesh, {"c0": synthetic.make_inputs(plan, 1, seed=2)[0]})
    for _ in range(warmup + steps):
        oracle.update()
    con, t = oracle.constituent_dict["c0"], warmup + steps - 1
    want = {"concentration": con.concentration[t + 1][: plan.n_real], "advection_mass_flux": con.advection_mass_flux[t],
            "diffusion_mass_flux": con.diffusion_mass_flux[t], "total_mass_flux": con.total_mass_flux[t]}
    defined = np.isfinite(con.total_mass_flux[t])     # NaN into ghost cells without a boundary value: not dumped
    assert line["dumped_outputs"]["arrays"] == {nm: [1, plan.n_real if nm == "concentration" else int(defined.sum())] for nm in names}
    for nm in names:
        w = want[nm] if nm == "concentration" else want[nm][defined]
        assert np.abs(got[nm][0] - w).max() <= 1e-9 * np.abs(w).max(), nm


def test_gpu_arm_refuses_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "1"], capture_output=True, text=True,
                         timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)
