"""CPU ORACLE of the device kinetics with depth-scaled processes (cwr_set_kinetics_depth, include/cwr.h) -- test
infrastructure only.

`react` and `KineticsRiverine` take the arguments of oracle.kinetics_limits's and, optionally, the depth flags
(decay_per_depth, source_per_depth, exchange_per_depth; (K,) 0/1 each) with the cell depth.  Without a flag set they are
oracle.kinetics_limits's, so their results are bitwise the same.  With flags, the whole step is restated here: the
step of oracle.kinetics_limits, every flagged rate (its theta^(T - 20) included) multiplied by g = 1 / h, the rounded
reciprocal of the cell's depth h = max(V[t] / A, min_depth).
"""
from __future__ import annotations

from typing import Dict, Optional, Union

import numpy as np
from scipy.sparse.linalg import spsolve

from . import kinetics as first_order
from . import kinetics_limits as limits
from . import kinetics_sources as sources
from .reference_step import HydroMesh, mass_flux

DEPTH_KEYS = ("decay_per_depth", "source_per_depth", "exchange_per_depth")


def depth(vol_t: np.ndarray, cell_area: np.ndarray, min_depth: float) -> np.ndarray:
    """h = max(V / A, min_depth) per real cell: V the f32 volume of the step widened to f64, A the plan area (f64)."""
    return np.fmax(np.asarray(vol_t, np.float32).astype(np.float64) / np.asarray(cell_area, np.float64), min_depth)


def _flags(a, K):
    return np.zeros(K, bool) if a is None else np.asarray(a).reshape(-1) != 0


def react(c: np.ndarray, dt: float, decay_per_day, theta=None, yields=None,
          temperature: Union[int, float, None] = None, temperature_is_index: bool = False,
          source_per_day=None, source_theta=None, exchange_per_day=None, exchange_theta=None, equilibrium=None,
          equilibrium_kind=None, limit_process=None, limit_column=None, limit_factor_column=None, limit_kind=None,
          limit_half_saturation=None, decay_per_depth=None, source_per_depth=None, exchange_per_depth=None,
          h=None) -> np.ndarray:
    """oracle.kinetics_limits.react with depth-scaled processes; h: the depth of every cell (the trailing axis of c), or
    a scalar.  A flagged rate is the unflagged one times g = 1.0 / h:
        decay of k:     r = decay_k theta_k^(T - 20) / 86400 * g
        source of k:    s = source_k source_theta_k^(T - 20) / 86400 * g
        exchange of k:  r = exchange_k exchange_theta_k^(T - 20) / 86400 * g
    and enters the step exactly as there (the factors, the cap, the self-limited sink, the exact solutions)."""
    lims = dict(limit_process=limit_process, limit_column=limit_column, limit_factor_column=limit_factor_column,
                limit_kind=limit_kind, limit_half_saturation=limit_half_saturation)
    srcs = dict(source_per_day=source_per_day, source_theta=source_theta, exchange_per_day=exchange_per_day,
                exchange_theta=exchange_theta, equilibrium=equilibrium, equilibrium_kind=equilibrium_kind)
    c0 = np.asarray(c, np.float64)
    K = c0.shape[0]
    fd, fs, fe = (_flags(a, K) for a in (decay_per_depth, source_per_depth, exchange_per_depth))
    if not (fd.any() or fs.any() or fe.any()):
        return limits.react(c, dt, decay_per_day, theta, yields, temperature, temperature_is_index, **srcs, **lims)
    g = 1.0 / np.asarray(h, np.float64)
    groups = {} if limit_process is None else limits._grouped(*lims.values())
    out = np.array(c0, dtype=np.float64, copy=True)
    decay = np.asarray(decay_per_day, np.float64)
    theta = np.ones(K) if theta is None else np.asarray(theta, np.float64)
    yields = np.zeros((K, K)) if yields is None else np.asarray(yields, np.float64)
    if temperature_is_index:
        T = c0[int(temperature)].copy()
    else:
        T = 20.0 if temperature is None else float(temperature)
    # the first-order chain
    for k in first_order.topological_order(yields):
        if decay[k] == 0.0:
            continue
        r = decay[k] * np.exp((T - 20.0) * np.log(theta[k])) / 86400.0
        if fd[k]:
            r = r * g
        M = 1.0
        for j, kd, hs in groups.get((0, k), ()):
            M = M * limits.factor(kd, hs, out[j])
        loss = out[k] * (-np.expm1(-(r * M) * dt))
        for j, kd, hs in groups.get((0, k), ()):
            if kd == 0 and yields[j, k] < 0.0:
                loss = np.fmin(loss, limits.div_down(np.fmax(out[j], 0.0), -yields[j, k]))
        out[k] -= loss
        for j in np.nonzero(yields[:, k])[0]:
            out[j] += yields[j, k] * loss
    if source_per_day is None and exchange_per_day is None:
        return out
    # the source columns
    src = np.zeros(K) if source_per_day is None else np.asarray(source_per_day, np.float64)
    exch = np.zeros(K) if exchange_per_day is None else np.asarray(exchange_per_day, np.float64)
    sth = np.ones(K) if source_theta is None else np.asarray(source_theta, np.float64)
    eth = np.ones(K) if exchange_theta is None else np.asarray(exchange_theta, np.float64)
    kind = np.zeros(K, int) if equilibrium_kind is None else np.asarray(equilibrium_kind)
    for k in range(K):
        if src[k] == 0.0 and exch[k] == 0.0:
            continue
        s = src[k] * np.exp((T - 20.0) * np.log(sth[k])) / 86400.0
        r = exch[k] * np.exp((T - 20.0) * np.log(eth[k])) / 86400.0
        if fs[k]:
            s = s * g
        if fe[k]:
            r = r * g
        if exch[k] == 0.0:
            ceq = 0.0
        else:
            ceq = sources.o2sat(T) if kind[k] == 1 else float(equilibrium[k])
        M, self_half = 1.0, None
        for j, kd, hs in groups.get((1, k), ()):
            if j == k:
                self_half = hs
            else:
                M = M * limits.factor(kd, hs, out[j])
        rr = r if self_half is None else r + (-s * M) / (self_half + np.fmax(out[k], 0.0))
        with np.errstate(invalid="ignore", divide="ignore"):
            phi = np.where(rr > 0.0, -np.expm1(-rr * dt) / rr, dt)
        if self_half is None:
            out[k] += (s * M + r * (ceq - out[k])) * phi
        else:
            out[k] += (r * ceq - rr * out[k]) * phi
    return out


class KineticsRiverine(limits.KineticsRiverine):
    """oracle.kinetics_limits.KineticsRiverine with the depth-scaled processes of `react` (keyword arguments
    decay_per_depth, source_per_depth, exchange_per_depth, besides the source and limit ones) over the plan areas
    cell_area (F,) with the floor min_depth; reaction_mass[t][k] includes them.  update() is the parent's, line for
    line, with this module's react and the depth of step t."""

    def __init__(self, mesh: HydroMesh, inputs: Dict[str, np.ndarray], decay_per_day, theta=None, yields=None,
                 temperature: Union[str, float, None] = None, cell_area=None, min_depth: float = 0.01, **terms):
        super().__init__(mesh, inputs, decay_per_day, theta, yields, temperature,
                         **{k: v for k, v in terms.items() if k not in DEPTH_KEYS})
        self.depth_flags = {k: v for k, v in terms.items() if k in DEPTH_KEYS}
        self.cell_area = None if cell_area is None else np.asarray(cell_area, np.float64)
        self.min_depth = float(min_depth)

    def update(self, update_concentration: Optional[Dict[str, np.ndarray]] = None):
        mesh, t, n = self.mesh, self.time_step, self.mesh.n
        self.lhs.update_values(mesh, t)
        A = self.lhs.to_csr()
        self.last_A = A
        merged = np.empty((len(self.names), n))
        for k, name in enumerate(self.names):
            c = self.constituent_dict[name]
            if isinstance(update_concentration, dict) and name in update_concentration:
                c.concentration[t][0:n] = np.asarray(update_concentration[name])[0:n]
                x = np.asarray(update_concentration[name])[0:n]
            else:
                x = c.concentration[t][0:n]
            solver = np.zeros(mesh.n_face)                   # linalg.py:193-201
            solver[0:n] = x
            nz = c.input_array[t].nonzero()
            solver[nz] = c.input_array[t][nz]
            merged[k] = solver[0:n]
        is_index = isinstance(self.temperature, str)
        temp = self.names.index(self.temperature) if is_index else self.temperature
        h = None if self.cell_area is None else depth(mesh.vol[t][0:n], self.cell_area[0:n], self.min_depth)
        reacted = react(merged, np.float64(mesh.dt[t]), self.decay, self.theta, self.yields, temp, is_index,
                        **self.sources, **self.limits, **self.depth_flags, h=h)
        vol = mesh.vol[t][0:n]
        self.reaction_mass.append(np.array([(vol * (reacted[k] - merged[k])).sum() for k in range(len(self.names))]))
        for k, name in enumerate(self.names):
            c = self.constituent_dict[name]
            c.b.vals[:] = c.b._calculate_rhs(mesh, t, reacted[k])
            x = spsolve(A, c.b.vals)
            c.concentration[t + 1][0:n] = x
            nz = np.nonzero(c.input_array[t + 1])[0]
            c.concentration[t + 1][nz] = c.input_array[t + 1][nz]
            mass_flux(mesh, c.concentration, c.advection_mass_flux, c.diffusion_mass_flux, c.total_mass_flux, t)
        self.time_step += 1


def depth_terms(cell_area=None, min_depth: float = 0.01, decay_per_depth=None, source_per_depth=None,
                exchange_per_depth=None) -> dict:
    """The keyword arguments of `KineticsRiverine` from those of TransportBackend.set_kinetics_depth."""
    return dict(cell_area=cell_area, min_depth=min_depth, decay_per_depth=decay_per_depth,
                source_per_depth=source_per_depth, exchange_per_depth=exchange_per_depth)
