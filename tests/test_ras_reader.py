"""This repo's h5py-free HEC-RAS reader (io/hdf5_mini.py, io/ras.py) and its vectorised IC / BC ingestion, against
what the UNMODIFIED reference read (the raw arrays and input arrays stored in tests/golden by tools/make_golden.py).
The plan files and IC / BC tables are rebuilt from those stored arrays (tests/ras_fixture.py): a HEC-RAS-layout HDF5
file with the mesh, hydrodynamics and boundary lines, and the reference test cases' uniform conditions (100 in every
real cell and on every boundary line)."""
import numpy as np
import pandas as pd
import pytest

from tests.helpers import load_golden
from tests.ras_fixture import write_plan

CASES = {   # golden case -> datetime_range the reference read it with
    "p02_uniform100": None,
    "p01_uniform100": (0, 300),
    "p03_uniform100": (0, 400),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_reader_and_ingestion_match_what_the_reference_read(case, tmp_path):
    from clearwater_riverine_b200.io import ras
    dtr = CASES[case]
    g = load_golden(case)
    hdf = tmp_path / "plan.hdf"
    times = write_plan(hdf, g, extra_times=0 if dtr is None else 5)
    plan = ras.read_ras_plan(hdf, dtr)
    assert np.array_equal(plan.f1, g["f1"]) and np.array_equal(plan.f2, g["f2"])
    assert np.array_equal(plan.face_x, g["face_x"]) and np.array_equal(plan.face_y, g["face_y"])
    assert np.array_equal(plan.time_seconds, g["time_seconds"])
    for mine, ref in ((plan.face_flow, g["face_flow"]), (plan.edge_velocity, g["edge_velocity"]), (plan.volume, g["volume"])):
        assert mine.dtype == np.float32 and np.array_equal(mine, ref)
    assert plan.nreal + 1 == int(g["f1"].max()) + 1
    # boundary lines: exactly the faces the reference attached its BC series to (the "Flow per Face" fix-up)
    bf = plan.boundary_faces()
    want = {}
    for name, face in zip(g["bc_names"], g["bc_faces"]):
        want.setdefault(str(name), set()).add(int(face))
    assert {k: set(int(x) for x in v) for k, v in bf.items()} == want
    # IC / BC ingestion -> the (T,F) input_array of the constituent, bit for bit
    cname = str(g["constituents"][0])
    n = plan.nreal + 1
    ic, bc = tmp_path / "ic.csv", tmp_path / "bc.csv"
    pd.DataFrame({"Cell_Index": np.arange(n), "Concentration": 100.0}).to_csv(ic, index=False)
    pd.DataFrame({"Datetime": np.repeat([times[0], times[-1]], len(want)), "RAS2D_TS_Name": sorted(want) * 2,
                  "Concentration": 100.0}).to_csv(bc, index=False)
    inp = ras.build_input_array(len(plan.time), len(plan.face_x), plan.time, plan.f2, plan.boundary_data, ic, bc)
    assert np.array_equal(inp, g[f"input_{cname}"], equal_nan=True)


def test_missing_file_raises_like_the_reference(tmp_path):
    from clearwater_riverine_b200.io import ras
    with pytest.raises(FileNotFoundError):        # reference io/inputs.py:39-44
        ras.read_ras_plan(tmp_path / "does_not_exist.hdf")
