"""CPU ORACLE of the device kinetics (cwr_set_kinetics, include/cwr.h) -- test infrastructure only.

A numpy restatement of the contract, kept apart from the product (clearwater_riverine_b200/kinetics.py only compiles
specs): step t forms every constituent's c~ (c[t] or the override, with the non-zero real-cell entries of input_array[t]
merged in, linalg.py:193-201), reacts all of them together, then builds each RHS from the reacted c~' with the
reference's RHS._calculate_rhs and solves with spsolve as OracleRiverine does.  History row t is not rewritten.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence, Union

import numpy as np
from scipy.sparse.linalg import spsolve

from .reference_step import HydroMesh, OracleRiverine, mass_flux


def topological_order(yields: np.ndarray) -> Sequence[int]:
    """k before j whenever yields[j, k] != 0; the smallest ready index first.  ValueError on a cycle."""
    y = np.asarray(yields) != 0
    K = y.shape[0]
    indeg = y.sum(axis=1).astype(int)
    done = np.zeros(K, bool)
    order = []
    for _ in range(K):
        ready = np.nonzero(~done & (indeg == 0))[0]
        if len(ready) == 0:
            raise ValueError("the yield graph has a cycle")
        k = int(ready[0])
        done[k] = True
        order.append(k)
        indeg -= y[:, k]
    return order


def react(c: np.ndarray, dt: float, decay_per_day, theta=None, yields=None,
          temperature: Union[int, float, None] = None, temperature_is_index: bool = False) -> np.ndarray:
    """c: (K, n) merged concentrations of one step; returns the reacted copy.
        T = temperature (deg C, default 20), or c[temperature] when temperature_is_index
        for k in topological order:  r = decay_k theta_k^(T - 20) / 86400  (theta^x as exp(x log theta))
                                     loss = c_k (-expm1(-r dt));  c_k -= loss;  c_j += yields[j, k] loss
    A constituent with decay 0 forms no loss and is skipped (so that a non-finite value is not spread through 0 * c)."""
    c = np.array(c, dtype=np.float64, copy=True)
    K = c.shape[0]
    decay = np.asarray(decay_per_day, np.float64)
    theta = np.ones(K) if theta is None else np.asarray(theta, np.float64)
    yields = np.zeros((K, K)) if yields is None else np.asarray(yields, np.float64)
    if temperature_is_index:
        T = c[int(temperature)].copy()
    else:
        T = 20.0 if temperature is None else float(temperature)
    for k in topological_order(yields):
        if decay[k] == 0.0:
            continue
        r = decay[k] * np.exp((T - 20.0) * np.log(theta[k])) / 86400.0
        loss = c[k] * (-np.expm1(-r * dt))
        c[k] -= loss
        for j in np.nonzero(yields[:, k])[0]:
            c[j] += yields[j, k] * loss
    return c


class KineticsRiverine(OracleRiverine):
    """OracleRiverine with the reactions applied to the merged c~ of every step.  reaction_mass[t][k] is
    sum_i V[t]_i (c~'_ik - c~_ik) of step t."""

    def __init__(self, mesh: HydroMesh, inputs: Dict[str, np.ndarray], decay_per_day, theta=None, yields=None,
                 temperature: Union[str, float, None] = None):
        super().__init__(mesh, inputs)
        self.names = list(inputs)
        self.decay, self.theta, self.yields = decay_per_day, theta, yields
        self.temperature = temperature
        self.reaction_mass = []

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
        reacted = react(merged, np.float64(mesh.dt[t]), self.decay, self.theta, self.yields, temp, is_index)
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
