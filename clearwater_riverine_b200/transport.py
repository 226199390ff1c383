"""Host-side mirror of the reference's stepping interface, backed by the CUDA library.

Same names, argument meaning and per-step behaviour as the reference's
`ClearwaterRiverine` (reference: src/clearwater_riverine/transport.py:68-276) and
`Constituent` (constituents.py:17-76) for the hot path -- `update()` advances every
constituent one timestep -- so code written against the reference's loop

    for _ in range(n): model.update(update_concentration)

runs unchanged.  The mesh container is a plain dict of numpy arrays under the reference's
variable names (variables.py) instead of an xarray Dataset; xarray is not a dependency.
All arithmetic happens on the GPU through `TransportBackend` (no CPU fallback).
"""
from __future__ import annotations

import warnings
from pathlib import Path
from typing import Any, Dict, Optional, Tuple

import numpy as np

from .backend import CWR_OK, STATUS_NAMES, SolverWarning, TransportBackend, pin_host_array, unpin_host_array

# reference variables.py names
ADVECTION_COEFFICIENT = "advection_coeff"
COEFFICIENT_TO_DIFFUSION_TERM = "coeff_to_diffusion"
EDGES_FACE1 = "edges_face1"
EDGES_FACE2 = "edges_face2"
EDGE_VELOCITY = "edge_velocity"
VOLUME = "volume"
CHANGE_IN_TIME = "dt"
FLOW_ACROSS_FACE = "face_flow"
NUMBER_OF_REAL_CELLS = "nreal"


class ModelMesh(dict):
    """dict of numpy arrays + `.attrs`; `mesh.nreal`, `mesh.diffusion_coefficient` work as in the reference."""

    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.attrs: Dict[str, Any] = {}

    def __getattr__(self, item):
        if item.startswith("__"):
            raise AttributeError(item)
        if item in self:
            return self[item]
        attrs = self.__dict__.get("attrs", {})
        if item in attrs:
            return attrs[item]
        raise AttributeError(item)


class Constituent:
    """Array contract of reference constituents.py:19-76."""

    def __init__(self, name: str, mesh: ModelMesh, input_array: np.ndarray, units: str = "Unknown",
                 store_mass_flux: bool = True):
        T, F, E = len(mesh["time"]), mesh.attrs["n_face"], len(mesh[EDGES_FACE1])
        self.name = name
        self.units = units
        self.input_array = np.ascontiguousarray(input_array, dtype=np.float64)
        if self.input_array.shape != (T, F):
            raise ValueError(f"input_array for {name!r}: expected {(T, F)}, got {self.input_array.shape}")
        if store_mass_flux:
            self.advection_mass_flux = np.zeros((T, E))
            self.diffusion_mass_flux = np.zeros((T, E))
            self.total_mass_flux = np.zeros((T, E))
        else:
            self.advection_mass_flux = self.diffusion_mass_flux = self.total_mass_flux = None
        n = mesh.attrs[NUMBER_OF_REAL_CELLS] + 1
        out = np.full((T, F), np.nan)                    # constituents.py:39-48
        out[0] = 0.0
        out[0, :n] = self.input_array[0, :n]             # constituents.py:94-98 (IC row; BCs are merged later)
        mesh[name] = out


class ClearwaterRiverine:
    """Drop-in for the reference class on the stepping path.

    Construct either like the reference (HEC-RAS file + constituent CSVs, or a YAML config),
    or from arrays with `ClearwaterRiverine.from_arrays(...)`.
    """

    def __init__(
        self,
        flow_field_file_path: Optional[str | Path] = None,
        diffusion_coefficient_input: Optional[float] = None,
        constituent_dict: Optional[Dict[str, Dict[str, Any]]] = None,
        config_filepath: Optional[str] = None,
        verbose: Optional[bool] = False,
        datetime_range: Optional[Tuple[int, int]] = None,
        mesh_file_path: Optional[str | Path] = None,
        kinetics: Optional[Dict[str, Dict[str, Any]]] = None,
        temperature: Optional[str | float] = None,
        cell_area: Optional[np.ndarray] = None,
        min_depth: Optional[float] = None,
        **backend_options,
    ) -> None:
        from .io import ras
        if mesh_file_path:
            raise NotImplementedError("loading saved zarr/netCDF meshes is outside the transport-step scope")
        if config_filepath:                                        # reference io/config.py:33-47
            import yaml
            with open(config_filepath) as fh:
                cfg = yaml.safe_load(fh)
            for key in ("diffusion_coefficient", "flow_field_filepath", "constituents"):
                if key not in cfg:
                    raise ValueError(f"Missing required key in model config: {key}")
            if diffusion_coefficient_input is None:
                diffusion_coefficient_input = cfg["diffusion_coefficient"]
            if not flow_field_file_path:
                flow_field_file_path = cfg["flow_field_filepath"]
            constituent_dict = cfg["constituents"]
            if kinetics is None:                                   # optional `kinetics:` block per constituent
                kinetics = {name: c["kinetics"] for name, c in constituent_dict.items()
                            if isinstance(c, dict) and c.get("kinetics") is not None} or None
            if temperature is None:
                temperature = cfg.get("temperature")
            if min_depth is None:
                min_depth = cfg.get("min_depth")
        if not flow_field_file_path or not isinstance(constituent_dict, dict):
            raise TypeError("Missing a `config_filepath` or a `constituent_dict` and `flow_field_file_path` to run the model.")
        plan = ras.read_ras_plan(flow_field_file_path, datetime_range)
        if verbose:
            print("Populating Model Mesh...")
        inputs, units = {}, {}
        for name, cfg_c in constituent_dict.items():
            inputs[name] = ras.build_input_array(len(plan.time), len(plan.face_x), plan.time, plan.f2, plan.boundary_data,
                                                 cfg_c["initial_conditions"], cfg_c["boundary_conditions"])
            units[name] = cfg_c.get("units", "Unknown")
        self._setup(plan.f1, plan.f2, plan.face_x, plan.face_y, plan.time_seconds, plan.face_flow, plan.edge_velocity,
                    plan.volume, float(diffusion_coefficient_input), inputs, units, time=plan.time,
                    backend_options=backend_options, kinetics=kinetics, temperature=temperature,
                    cell_area=plan.cell_area if cell_area is None else cell_area, min_depth=min_depth)
        self.boundary_data = plan.boundary_data
        self.mesh.attrs["boundary_data"] = plan.boundary_data

    @classmethod
    def from_arrays(cls, f1, f2, face_x, face_y, time_seconds, face_flow, edge_velocity, volume,
                    diffusion_coefficient: float, inputs: Dict[str, np.ndarray], units: Optional[Dict[str, str]] = None,
                    kinetics: Optional[Dict[str, Dict[str, Any]]] = None, temperature: Optional[str | float] = None,
                    cell_area: Optional[np.ndarray] = None, min_depth: Optional[float] = None,
                    **backend_options) -> "ClearwaterRiverine":
        """cell_area (F,): the plan area of every cell, which kinetics given per unit depth need; min_depth: the floor of
        the depth V / cell_area (default kinetics.DEFAULT_MIN_DEPTH), both in the mesh's length unit."""
        self = cls.__new__(cls)
        self._setup(f1, f2, face_x, face_y, time_seconds, face_flow, edge_velocity, volume, float(diffusion_coefficient),
                    inputs, units or {}, time=None, backend_options=backend_options, kinetics=kinetics, temperature=temperature,
                    cell_area=cell_area, min_depth=min_depth)
        self.boundary_data = None
        return self

    # ------------------------------------------------------------------------------------------
    def _setup(self, f1, f2, face_x, face_y, time_seconds, face_flow, edge_velocity, volume, D, inputs, units, time,
               backend_options, kinetics=None, temperature=None, cell_area=None, min_depth=None):
        store_mass_flux = backend_options.pop("store_mass_flux", True)
        # 'eager': update() returns with the results in the host arrays; 'pipelined': the copies overlap the next
        # update() (sync() before reading); 'none': results stay on the device (read them through self.backend)
        self.output = backend_options.pop("output", "eager")
        if self.output not in ("eager", "pipelined", "none"):
            raise ValueError("output must be 'eager', 'pipelined' or 'none'")
        device = backend_options.pop("device", 0)
        T, F = volume.shape
        mesh = ModelMesh()
        mesh.attrs.update({"diffusion_coefficient": D, NUMBER_OF_REAL_CELLS: int(np.max(f1)), "n_face": F})
        mesh[EDGES_FACE1] = np.ascontiguousarray(f1, dtype=np.int32)
        mesh[EDGES_FACE2] = np.ascontiguousarray(f2, dtype=np.int32)
        mesh["face_x"], mesh["face_y"] = np.asarray(face_x, np.float64), np.asarray(face_y, np.float64)
        mesh["time"] = np.asarray(time_seconds, np.float64) if time is None else np.asarray(time)
        mesh[FLOW_ACROSS_FACE] = np.ascontiguousarray(face_flow, np.float32)
        mesh[EDGE_VELOCITY] = np.ascontiguousarray(edge_velocity, np.float32)
        mesh[VOLUME] = np.ascontiguousarray(volume, np.float32)
        tsec = np.asarray(time_seconds, np.float64)
        mesh[CHANGE_IN_TIME] = np.append(np.diff(tsec), np.nan)    # utilities.py:537-541
        self.mesh = mesh
        self.time_step = 0
        self.constituents = list(inputs.keys())
        self.constituent_dict = {name: Constituent(name, mesh, arr, units.get(name, "Unknown"), store_mass_flux)
                                 for name, arr in inputs.items()}
        # stream_hydro: keep only a few time slices on the device and upload slice t+1 inside update()
        # (meshes whose T x E arrays exceed device memory; also what bench.py's end-to-end leg times)
        self.stream_hydro = bool(backend_options.pop("stream_hydro", False))
        if self.stream_hydro:
            backend_options.setdefault("hydro_capacity", 4)       # t, t+1 in use; t+2, t+3 on their way
        q = mesh[FLOW_ACROSS_FACE]      # Gauss-Seidel colours follow the time-mean flow
        hint = np.nanmean(q[:: max(1, T // 32)], axis=0, dtype=np.float64).astype(np.float32)
        self.backend = TransportBackend(mesh[EDGES_FACE1], mesh[EDGES_FACE2], F, T, len(inputs), D, device=device,
                                        flow_hint=hint, **backend_options)
        # derived coefficients (utilities.py:513-541) are computed on the device from the raw arrays
        self.backend.set_geometry(mesh["face_x"], mesh["face_y"])
        self._resident = set()
        if self.stream_hydro:
            self._upload_slice(0)
        else:
            chunk = max(1, min(T, (64 << 20) // max(1, 4 * len(f1))))
            for t0 in range(0, T, chunk):
                t1 = min(T, t0 + chunk)
                self.backend.set_hydro_raw(t0, mesh[FLOW_ACROSS_FACE][t0:t1], mesh[EDGE_VELOCITY][t0:t1],
                                           mesh[VOLUME][t0:t1], mesh[CHANGE_IN_TIME][t0:t1])
        for k, name in enumerate(self.constituents):
            self.backend.set_inputs(k, self.constituent_dict[name].input_array)
        self._index = {name: k for k, name in enumerate(self.constituents)}
        from .kinetics import DEFAULT_MIN_DEPTH
        self.cell_area = None if cell_area is None else np.array(cell_area, np.float64).reshape(F)
        self.min_depth = DEFAULT_MIN_DEPTH if min_depth is None else float(min_depth)
        self.kinetics = None
        if kinetics is not None:
            self.set_kinetics(kinetics, 20.0 if temperature is None else temperature)
        # update() copies c[t+1] of every constituent straight into row t+1 of its output array; page-locking
        # those arrays lets the copies run at the full PCIe rate with no intermediate host buffer
        outputs = [self.mesh[name] for name in self.constituents]
        if store_mass_flux:
            for name in self.constituents:
                c = self.constituent_dict[name]
                outputs += [c.advection_mass_flux, c.diffusion_mass_flux, c.total_mass_flux]
        self._pinned = [a for a in outputs if pin_host_array(a)]
        self._row_cache = None
        self._mass_start: Dict[int, Tuple[float, float]] = {}
        self._store_flux = bool(store_mass_flux)
        self.solver_info = []

    def _upload_slice(self, t: int, overlap: bool = False):
        if t in self._resident or t >= len(self.mesh["time"]):
            return
        m = self.mesh
        send = self.backend.prefetch_hydro_raw if overlap else self.backend.set_hydro_raw
        send(t, m[FLOW_ACROSS_FACE][t:t + 1], m[EDGE_VELOCITY][t:t + 1], m[VOLUME][t:t + 1], m[CHANGE_IN_TIME][t:t + 1])
        cap = self.backend.options.hydro_capacity
        self._resident = {s for s in self._resident if s % cap != t % cap} | {t}

    # ------------------------------------------------------------------------------------------
    def update(self, update_concentration: Optional[Dict[str, np.ndarray]] = None):
        """Update a single timestep (reference transport.py:201-276)."""
        t = self.time_step
        n = self.mesh.attrs[NUMBER_OF_REAL_CELLS] + 1
        if isinstance(update_concentration, dict):
            if self.output == "pipelined":
                self.backend.fetch_wait()                    # row t of the host arrays may still be arriving
            for name, values in update_concentration.items():
                if name not in self.constituent_dict:        # transport.py:223-229
                    print(f"WARNING: {name} is not being used in the model.")
                    print("Please review the constituent names in the update dictionary")
                    continue
                values = np.asarray(getattr(values, "values", values), dtype=np.float64)[0:n]
                self.mesh[name][t][0:n] = values             # transport.py:233-236: history at t is overwritten too
                self.backend.set_state(self._index[name], t, values)
        if self.stream_hydro:
            self._upload_slice(t)
            self._upload_slice(t + 1)
        if t == 0 and not self._mass_start and self.backend.options.mass_flux:
            for k in range(len(self.constituents)):           # sum(V c) at the start (postproc_util.py:36-47)
                m0 = self.backend.mass_totals(k, 0, 0)
                self._mass_start[k] = (m0.vol_start, m0.mass_start)
        info = self.backend.step(t)
        self.solver_info.append((info.iterations, info.max_relres, info.status))
        if info.status != CWR_OK:
            warnings.warn(f"step {t}: {STATUS_NAMES.get(info.status, info.status)} "
                          f"({info.iterations} iterations, relres {info.max_relres:.3e})", SolverWarning)
        if self.stream_hydro:       # slices t+2, t+3 go up while c[t+1] comes down (full duplex); the next update() only
            self._upload_slice(t + 2, overlap=True)            # waits for t+2, which then has had a whole step to arrive
            if self.backend.options.hydro_capacity >= 4:
                self._upload_slice(t + 3, overlap=True)
        if self.output in ("eager", "pipelined"):
            self._fetch(t + 1)
        self.time_step += 1                                   # transport.py:276

    def _fetch(self, t1: int):
        """c[t1] of every constituent and the mass fluxes of step t1 - 1 (transport.py:252-273) gathered on the device
        and copied straight into row t1 / t1 - 1 of the constituents' (T,F) / (T,E) arrays.  output='eager' (default)
        waits for the copies, as the reference's update() leaves everything in place; output='pipelined' lets them
        overlap the next update() (two steps' worth can be in flight) -- call sync() before reading the arrays.
        Ghost cells get their BC value where one is set and stay NaN elsewhere (transport.py:258-264)."""
        n = self.mesh.attrs[NUMBER_OF_REAL_CELLS] + 1
        if self._row_cache is None:       # per constituent: its (T,F) array, ghost-column BC values (NaN where unset)
            self._row_cache = []
            for name in self.constituents:
                bc = self.constituent_dict[name].input_array[:, n:]
                self._row_cache.append((self.mesh[name], np.where(bc != 0, bc, np.nan)))
        flux = self._store_flux and bool(self.backend.options.mass_flux)
        cons = [self.constituent_dict[name] for name in self.constituents]
        self.backend.fetch_async(
            t1, [out[t1] for out, _ in self._row_cache],
            [c.advection_mass_flux[t1 - 1] for c in cons] if flux else None,
            [c.diffusion_mass_flux[t1 - 1] for c in cons] if flux else None,
            [c.total_mass_flux[t1 - 1] for c in cons] if flux else None)
        for out, ghost in self._row_cache:
            out[t1, n:] = ghost[t1]                             # (columns the device copy does not touch)
        if self.output == "eager":
            self.backend.fetch_wait()

    def set_kinetics(self, spec: Optional[Dict[str, Dict[str, Any]]], temperature: str | float = 20.0):
        """Kinetics applied on the device in every later step, after the update_concentration override and before
        transport: first-order decay and yields, then zero-order sources and relaxation toward an equilibrium such as
        reaeration toward oxygen saturation, each optionally scaled by Monod limitation and inhibition factors such as
        oxygen limitation of BOD oxidation, and processes given per unit depth such as settling, areal sediment oxygen
        demand or a surface transfer velocity, which act through each cell's depth V / cell_area (kinetics.py: spec format;
        temperature is a constituent name or a constant in deg C).  None switches kinetics off.  History rows are not
        rewritten: the reaction of step t shows in row t + 1."""
        from .kinetics import compile_kinetics
        if spec is None:
            self.backend.set_kinetics(None)
            self.kinetics = None
            return
        kin = compile_kinetics(spec, self.constituents, temperature, cell_area=self.cell_area, min_depth=self.min_depth,
                               n_real=self.mesh.attrs[NUMBER_OF_REAL_CELLS] + 1)
        self.backend.set_kinetics(kin.decay_per_day, kin.theta, kin.yields, kin.temperature_k, kin.temperature_c)
        if kin.has_sources:
            self.backend.set_kinetics_sources(**kin.sources_arguments())
        if kin.has_limits:
            self.backend.set_kinetics_limits(**kin.limits_arguments())
        if kin.has_depth:
            self.backend.set_kinetics_depth(**kin.depth_arguments())
        self.kinetics = kin

    def sync(self):
        """Wait for the output copies of the updates issued so far (output='pipelined')."""
        self.backend.fetch_wait()

    def mass_balance(self, constituent_name: str, boundary_faces: Optional[Dict[str, np.ndarray]] = None) -> Dict[str, float]:
        """Whole-domain mass balance over the steps taken so far, from device reductions (next row N2): the quantities
        of the reference's `_mass_bal_global` (postproc_util.py:21-166) under the same names -- Vol/Mass at the start and
        now, per boundary line the water volume and constituent mass that crossed it (total, in <= 0, out >= 0), the
        totals over all lines and the closure errors.  Nothing of it needs the (T,E) flux history on the host: the
        per-face running sums are kept by the mass-flux kernel.  While kinetics is set, `reaction_mass` (what decay,
        yields, sources and exchange formed) is reported and counted in mass_end_calc.  boundary_faces: {line name:
        face (edge) ids}; default: the lines of the HEC-RAS plan the model was built from."""
        if boundary_faces is None:
            bd = getattr(self, "boundary_data", None)
            if bd is None:
                raise ValueError("boundary_faces is required for a model built from arrays")
            boundary_faces = {str(nm): np.asarray(grp["Face Index"], dtype=np.int64) for nm, grp in
                              sorted(bd.groupby("Name"), key=lambda kv: float(np.mean(kv[1]["BC Line ID"])))}
        k = self._index[constituent_name]
        self.backend.fetch_wait()
        now = self.time_step
        m = self.backend.mass_totals(k, now, now)
        start = self._mass_start.get(k)
        if start is None:                                     # no step taken yet
            start = (m.vol_start, m.mass_start)
        out = {"Vol_start": start[0], "Mass_start": start[1], "Vol_end": m.vol_end, "Mass_end": m.mass_end}
        f_tot, f_in, f_out = self.backend.flux_sums(k)
        v_tot, v_in, v_out = self.backend.volume_sums()
        tv_in = tv_out = tm_in = tm_out = tv = tm = 0.0
        for name, faces in boundary_faces.items():
            faces = np.asarray(faces, dtype=np.int64)
            out[f"{name}_vol"], out[f"{name}_mass"] = float(v_tot[faces].sum()), float(f_tot[faces].sum())
            out[f"{name}_in_vol"], out[f"{name}_out_vol"] = float(v_in[faces].sum()), float(v_out[faces].sum())
            out[f"{name}_in_mass"], out[f"{name}_out_mass"] = float(f_in[faces].sum()), float(f_out[faces].sum())
            tv += out[f"{name}_vol"]; tm += out[f"{name}_mass"]
            tv_in += out[f"{name}_in_vol"]; tv_out += out[f"{name}_out_vol"]
            tm_in += out[f"{name}_in_mass"]; tm_out += out[f"{name}_out_mass"]
        out["bcTotalVolInOutAll"], out["bcTotalVolInAll"], out["bcTotalVolOutAll"] = tv, tv_in, tv_out
        out["bcTotalMassInOutAll"], out["bcTotalMassInAll"], out["bcTotalMassOutAll"] = tm, tm_in, tm_out
        out["vol_end_calc"] = out["Vol_start"] - tv_in - tv_out
        out["mass_end_calc"] = out["Mass_start"] - tm_in - tm_out
        if self.kinetics is not None:                         # mass the reactions, sources and exchange formed (< 0: lost)
            out["reaction_mass"] = self.backend.reaction_mass(k)
            out["mass_end_calc"] += out["reaction_mass"]
        out["error_vol"] = out["vol_end_calc"] - out["Vol_end"]
        out["error_mass"] = out["mass_end_calc"] - out["Mass_end"]
        out["prct_error_vol"] = out["error_vol"] / tv_in * 100 if tv_in else float("nan")
        out["prct_error_mass"] = out["error_mass"] / tm_in * 100 if tm_in else float("nan")
        return out

    def run(self, n_steps: Optional[int] = None):
        """`n_steps` updates back to back on the device, then one bulk copy of the concentrations
        (mass-flux history is only recorded by `update()`, which reads it back every step)."""
        T = len(self.mesh["time"])
        t0 = self.time_step
        t1 = T - 1 if n_steps is None else min(T - 1, t0 + n_steps)
        self.backend.fetch_wait()
        info = self.backend.run(t0, t1)
        self.time_step = t1
        if self.output == "eager" and self.backend.options.keep_history:
            for t in range(t0 + 1, t1 + 1):
                for name, k in self._index.items():
                    self.backend.get_state(k, t, self.mesh[name][t])
        return info

    def finalize(self, save: Optional[bool] = False, output_filepath: Optional[str] = None):
        """Reference transport.py:385-395: with save=True the mesh (every variable, the concentrations included) is written
        to `output_filepath` (.nc NetCDF-3 classic or .npz; io/outputs.py) and the boundary table next to it."""
        self.backend.fetch_wait()
        if save:
            from .io.outputs import save_mesh
            if not output_filepath:
                raise ValueError("finalize(save=True) needs output_filepath")
            save_mesh(self.mesh, output_filepath)
            bd = getattr(self, "boundary_data", None)
            if bd is not None:
                p = Path(output_filepath)
                bd.to_csv(f"{p.parent}/{p.stem}_boundary_data.csv")
        for a in getattr(self, "_pinned", []):
            unpin_host_array(a)
        self._pinned = []
        self.backend.close()
