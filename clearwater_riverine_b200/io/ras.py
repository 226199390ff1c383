"""HEC-RAS 2D plan reader and IC/BC ingestion for the transport step (host side, runs once).

Mirrors what the reference pulls out of the HDF file
(reference: src/clearwater_riverine/io/hdf.py:39-69 paths, 255-286 hydrodynamics,
356-436 boundary tables and the "Flow per Face" fix-up) and how it turns the
IC / BC CSV files into the per-constituent `input_array`
(reference: src/clearwater_riverine/constituents.py:78-98 and 100-164), but
returns plain numpy arrays instead of an xarray Dataset and needs neither h5py
nor xarray (see hdf5_mini.py).
"""
from __future__ import annotations

from dataclasses import dataclass
from pathlib import Path
from typing import Dict, Optional, Tuple

import numpy as np
import pandas as pd

from . import hdf5_mini

_TS = "Results/Unsteady/Output/Output Blocks/Base Output/Unsteady Time Series"


@dataclass
class RasPlan:
    area_name: str
    f1: np.ndarray              # (E,) int32  edges_face1
    f2: np.ndarray              # (E,) int32  edges_face2
    face_x: np.ndarray          # (F,) float64 cell-centre x
    face_y: np.ndarray          # (F,) float64 cell-centre y
    time: np.ndarray            # (T,) datetime64[ns]
    edge_velocity: np.ndarray   # (T,E) float32  "Face Velocity"
    face_flow: np.ndarray       # (T,E) float32  "Face Flow"
    volume: np.ndarray          # (T,F) float32  "Cell Volume"
    boundary_data: pd.DataFrame  # columns: BC Line ID, Face Index, Name, ...
    cell_area: Optional[np.ndarray] = None   # (F,) float64 "Cells Surface Area" (cell plan area), None when absent

    @property
    def nreal(self) -> int:     # reference io/hdf.py:268-269
        return int(self.f1.max())

    @property
    def time_seconds(self) -> np.ndarray:
        return (self.time - self.time[0]) / np.timedelta64(1, "s")

    def boundary_faces(self) -> Dict[str, np.ndarray]:
        return {name: g["Face Index"].to_numpy(dtype=np.int64)
                for name, g in self.boundary_data.groupby("Name", sort=False)}


def read_ras_plan(file_path: str | Path, datetime_range: Optional[Tuple[int, int]] = None) -> RasPlan:
    """Read the arrays the transport step needs from a HEC-RAS 2D output file."""
    file_path = Path(file_path)
    if not file_path.is_file():
        raise FileNotFoundError(str(file_path))   # reference io/inputs.py:39-44
    f = hdf5_mini.File(str(file_path))
    area = f["Geometry/2D Flow Areas/Attributes"].read()[0][0].decode("utf-8").strip()   # hdf.py:142-144
    geom = f[f"Geometry/2D Flow Areas/{area}"]
    fc = geom["Faces Cell Indexes"].read()
    centres = geom["Cells Center Coordinate"].read()
    cell_area = None
    if "Cells Surface Area" in geom:                   # the plan area of every cell (kinetics given per unit depth)
        a = np.asarray(geom["Cells Surface Area"].read(), dtype=np.float64).reshape(-1)
        F, n = len(centres), int(fc[:, 0].max()) + 1
        if len(a) == n:                                # real cells only: the ghost cells' areas are never read
            a = np.concatenate([a, np.zeros(F - n)])
        if len(a) != F:
            raise ValueError(f"{file_path}: 'Cells Surface Area' has {len(a)} entries for {F} cells")
        cell_area = np.ascontiguousarray(a)
    stamps = f[f"{_TS}/Time Date Stamp"].read()
    time = pd.to_datetime(pd.Series(stamps).str.decode("utf8").str.strip(), format="%d%b%Y %H:%M:%S")
    sl = slice(None)
    if datetime_range is not None:                     # hdf.py:158-162 (int form)
        sl = slice(int(datetime_range[0]), int(datetime_range[1]) + 1)
    res = f[f"{_TS}/2D Flow Areas/{area}"]
    vel = res["Face Velocity"].read()[sl]
    flow = res["Face Flow"].read()[sl]
    vol = res["Cell Volume"].read()[sl]

    # boundary tables (hdf.py:356-436)
    ext = pd.DataFrame(f["Geometry/Boundary Condition Lines/External Faces"].read())
    att_raw = f["Geometry/Boundary Condition Lines/Attributes"].read()
    att = pd.DataFrame({k: (np.char.decode(att_raw[k], "utf-8") if att_raw[k].dtype.kind == "S" else att_raw[k])
                        for k in att_raw.dtype.names})
    att["Name"] = att["Name"].str.strip()
    att["BC Line ID"] = att.index
    bd = pd.merge(ext, att, on="BC Line ID", how="left")
    bcs = f[f"{_TS}/Boundary Conditions"]
    keep = []
    for name in bd["Name"].unique():
        faces_fix = np.atleast_1d(bcs[f"{name} - Flow per Face"].attrs["Faces"])
        keep.append(bd[(bd["Name"] == name) & (bd["Face Index"].isin(faces_fix))])
    bd = pd.concat(keep).drop(columns=["Station Start", "Station End"]).drop_duplicates()

    return RasPlan(
        area_name=area,
        f1=np.ascontiguousarray(fc[:, 0], dtype=np.int32),
        f2=np.ascontiguousarray(fc[:, 1], dtype=np.int32),
        face_x=np.ascontiguousarray(centres[:, 0], dtype=np.float64),
        face_y=np.ascontiguousarray(centres[:, 1], dtype=np.float64),
        time=time.to_numpy()[sl],
        edge_velocity=np.ascontiguousarray(vel, dtype=np.float32),
        face_flow=np.ascontiguousarray(flow, dtype=np.float32),
        volume=np.ascontiguousarray(vol, dtype=np.float32),
        boundary_data=bd.reset_index(drop=True),
        cell_area=cell_area,
    )


def build_input_array(
    n_time: int,
    n_face: int,
    time: np.ndarray,
    f2: np.ndarray,
    boundary_data: pd.DataFrame,
    initial_conditions: str | Path | pd.DataFrame,
    boundary_conditions: str | Path | pd.DataFrame,
) -> np.ndarray:
    """(T,F) float64 `input_array`: IC in row 0, BC series in ghost-cell columns.

    Semantics of reference constituents.py:78-98 (IC) and 100-164 (BC): per BC
    line a backward `merge_asof` of the CSV onto model times followed by linear
    interpolation, then every face of the line -> its ghost cell `edges_face2[face]`.
    Vectorised over lines (one merge per line, one scatter for all faces).
    """
    inp = np.zeros((n_time, n_face))
    ic = initial_conditions if isinstance(initial_conditions, pd.DataFrame) else pd.read_csv(initial_conditions)
    inp[0, ic["Cell_Index"].astype(int).to_numpy()] = ic["Concentration"].to_numpy()
    bc = boundary_conditions if isinstance(boundary_conditions, pd.DataFrame) \
        else pd.read_csv(boundary_conditions, parse_dates=["Datetime"])
    model = pd.DataFrame({"Datetime": pd.DatetimeIndex(time), "Time Index": np.arange(n_time)})
    f2 = np.asarray(f2)
    for name, group in bc.groupby("RAS2D_TS_Name"):
        merged = pd.merge_asof(model, group.sort_values("Datetime"), on="Datetime")
        conc = merged["Concentration"].interpolate(method="linear").to_numpy()
        faces = boundary_data.loc[boundary_data["Name"] == name, "Face Index"].to_numpy(dtype=np.int64)
        if len(faces):
            inp[:, f2[faces]] = conc[:, None]
    return inp
