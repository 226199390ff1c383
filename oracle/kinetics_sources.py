"""CPU ORACLE of the device kinetics with zero-order sources and exchange (cwr_set_kinetics_sources, include/cwr.h) --
test infrastructure only.

`react` and `KineticsRiverine` take the arguments of oracle.kinetics's and, optionally, the source and exchange arrays.
Without them they are oracle.kinetics's, so their results are bitwise the same.  With them, the first-order chain of
oracle.kinetics.react runs first, then every column with a source or exchange term, in ascending k, takes the exact
solution of dc/dt = s + r (ceq - c) over dt, with the temperature of the cell before any of the step's reactions.
"""
from __future__ import annotations

from typing import Dict, Optional, Union

import numpy as np
from scipy.sparse.linalg import spsolve

from . import kinetics as first_order
from .reference_step import HydroMesh, mass_flux


def o2sat(T):
    """APHA / Benson-Krause dissolved-oxygen saturation (mg/L) of fresh water at 1 atm, written as the contract states it."""
    Ta = np.asarray(T, np.float64) + 273.15
    return np.exp(-139.34411 + 1.575701e5 / Ta - 6.642308e7 / Ta ** 2 + 1.243800e10 / Ta ** 3 - 8.621949e11 / Ta ** 4)


def react(c: np.ndarray, dt: float, decay_per_day, theta=None, yields=None,
          temperature: Union[int, float, None] = None, temperature_is_index: bool = False,
          source_per_day=None, source_theta=None, exchange_per_day=None, exchange_theta=None, equilibrium=None,
          equilibrium_kind=None) -> np.ndarray:
    """oracle.kinetics.react, then for k ascending with source_k != 0 or exchange_k != 0:
            s = source_k source_theta_k^(T - 20) / 86400;  r = exchange_k exchange_theta_k^(T - 20) / 86400
            ceq = equilibrium_k (kind 0) | o2sat(T) (kind 1);  phi = -expm1(-r dt) / r, or dt when r == 0
            c_k += (s + r (ceq - c_k)) phi
    with T as the chain takes it (the value before the step's reactions).  A column without either term is skipped, and
    the equilibrium of a column without exchange is not read (the library lists neither)."""
    c0 = np.asarray(c, np.float64)
    out = first_order.react(c0, dt, decay_per_day, theta, yields, temperature, temperature_is_index)
    if source_per_day is None and exchange_per_day is None:
        return out
    K = out.shape[0]
    if temperature_is_index:
        T = c0[int(temperature)].copy()
    else:
        T = 20.0 if temperature is None else float(temperature)
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
        if exch[k] == 0.0:
            ceq = 0.0
        else:
            ceq = o2sat(T) if kind[k] == 1 else float(equilibrium[k])
        with np.errstate(invalid="ignore", divide="ignore"):
            phi = np.where(r > 0.0, -np.expm1(-r * dt) / r, dt)
        out[k] += (s + r * (ceq - out[k])) * phi
    return out


class KineticsRiverine(first_order.KineticsRiverine):
    """oracle.kinetics.KineticsRiverine with the sources and exchange of `react` (keyword arguments source_per_day, ...,
    equilibrium_kind); reaction_mass[t][k] includes them.  update() is the parent's, line for line, with this module's
    react in place of oracle.kinetics.react."""

    def __init__(self, mesh: HydroMesh, inputs: Dict[str, np.ndarray], decay_per_day, theta=None, yields=None,
                 temperature: Union[str, float, None] = None, **sources):
        super().__init__(mesh, inputs, decay_per_day, theta, yields, temperature)
        self.sources = sources

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
        reacted = react(merged, np.float64(mesh.dt[t]), self.decay, self.theta, self.yields, temp, is_index, **self.sources)
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
