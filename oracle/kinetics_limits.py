"""CPU ORACLE of the device kinetics with Monod limitation and inhibition (cwr_set_kinetics_limits, include/cwr.h) --
test infrastructure only.

`react` and `KineticsRiverine` take the arguments of oracle.kinetics_sources's and, optionally, the limit arrays
(process, column, factor column, kind, half-saturation; (n,) each).  Without them they are oracle.kinetics_sources's, so
their results are bitwise the same.  With them, the whole step is restated here: the first-order chain in topological
order, then the source columns in ascending k, every process that carries factors scaled by their product M (a factor
reads its constituent as the cell holds it when the process is applied), the decay capped by what it consumes of a
constituent that limits it, and a self-limited sink solved as a first-order sink.  A process without factors is computed
with the expressions of oracle.kinetics / oracle.kinetics_sources.
"""
from __future__ import annotations

from typing import Dict, Optional, Union

import numpy as np
from scipy.sparse.linalg import spsolve

from . import kinetics as first_order
from . import kinetics_sources as sources
from .reference_step import HydroMesh, mass_flux

LIMIT_KEYS = ("limit_process", "limit_column", "limit_factor_column", "limit_kind", "limit_half_saturation")


def factor(kind: int, half: float, c_j: np.ndarray) -> np.ndarray:
    """Limitation (kind 0) c+ / (K + c+), inhibition (kind 1) K / (K + c+), c+ = max(c, 0) (fmax: NaN counts as 0)."""
    cp = np.fmax(c_j, 0.0)
    return (half if kind else cp) / (half + cp)


def div_down(a, b):
    """a / b rounded toward -inf (a >= 0 finite, b > 0), as the device's __ddiv_rd: the nearest quotient q, stepped down
    once when q * b > a exactly (Dekker's error-free product decides it)."""
    a = np.asarray(a, np.float64)
    q = a / b
    p = q * b
    split = lambda x: (x * 134217729.0 - (x * 134217729.0 - x), x - (x * 134217729.0 - (x * 134217729.0 - x)))
    qh, ql = split(q)
    bh, bl = split(np.float64(b))
    err = ((qh * bh - p) + qh * bl + ql * bh) + ql * bl          # q * b - p, exactly
    over = (p > a) | ((p == a) & (err > 0.0))
    return np.where(over, np.nextafter(q, -np.inf), q)


def _grouped(limit_process, limit_column, limit_factor_column, limit_kind, limit_half_saturation):
    """{(process, column): [(factor column, kind, half-saturation), ...] in the order given}."""
    out: Dict[tuple, list] = {}
    for pr, k, j, kd, h in zip(limit_process, limit_column, limit_factor_column, limit_kind, limit_half_saturation):
        out.setdefault((int(pr), int(k)), []).append((int(j), int(kd), float(h)))
    return out


def react(c: np.ndarray, dt: float, decay_per_day, theta=None, yields=None,
          temperature: Union[int, float, None] = None, temperature_is_index: bool = False,
          source_per_day=None, source_theta=None, exchange_per_day=None, exchange_theta=None, equilibrium=None,
          equilibrium_kind=None, limit_process=None, limit_column=None, limit_factor_column=None, limit_kind=None,
          limit_half_saturation=None) -> np.ndarray:
    """oracle.kinetics_sources.react with Monod factors.  For every process with factors, M = prod f from 1.0:
        decay of k:   r = decay_k theta_k^(T - 20) / 86400;  loss = c_k (-expm1(-(r M) dt));
                      loss = min(loss, c+_j / -yields[j, k]) for every limitation on a j with yields[j, k] < 0, the
                      quotient rounded toward -inf (div_down), so that c_j + yields[j, k] loss >= 0 exactly;
                      c_k -= loss;  c_j += yields[j, k] loss
        source of k:  s M in place of s;  with a limitation on k itself (a sink): a = -s M' / (K + c+_k) (M' the other
                      factors), c_k += (r ceq - (r + a) c_k) phi(r + a)."""
    srcs = dict(source_per_day=source_per_day, source_theta=source_theta, exchange_per_day=exchange_per_day,
                exchange_theta=exchange_theta, equilibrium=equilibrium, equilibrium_kind=equilibrium_kind)
    if limit_process is None or len(limit_process) == 0:
        return sources.react(c, dt, decay_per_day, theta, yields, temperature, temperature_is_index, **srcs)
    groups = _grouped(limit_process, limit_column, limit_factor_column, limit_kind, limit_half_saturation)
    c0 = np.asarray(c, np.float64)
    out = np.array(c0, dtype=np.float64, copy=True)
    K = out.shape[0]
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
        fs = groups.get((0, k))
        if fs is None:
            loss = out[k] * (-np.expm1(-r * dt))
        else:
            M = 1.0
            for j, kd, h in fs:
                M = M * factor(kd, h, out[j])
            loss = out[k] * (-np.expm1(-(r * M) * dt))
            for j, kd, h in fs:
                if kd == 0 and yields[j, k] < 0.0:
                    loss = np.fmin(loss, div_down(np.fmax(out[j], 0.0), -yields[j, k]))
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
        if exch[k] == 0.0:
            ceq = 0.0
        else:
            ceq = sources.o2sat(T) if kind[k] == 1 else float(equilibrium[k])
        fs = groups.get((1, k))
        if fs is None:
            with np.errstate(invalid="ignore", divide="ignore"):
                phi = np.where(r > 0.0, -np.expm1(-r * dt) / r, dt)
            out[k] += (s + r * (ceq - out[k])) * phi
            continue
        M, self_half = 1.0, None
        for j, kd, h in fs:
            if j == k:
                self_half = h
            else:
                M = M * factor(kd, h, out[j])
        if self_half is None:
            with np.errstate(invalid="ignore", divide="ignore"):
                phi = np.where(r > 0.0, -np.expm1(-r * dt) / r, dt)
            out[k] += (s * M + r * (ceq - out[k])) * phi
        else:
            rr = r + (-s * M) / (self_half + np.fmax(out[k], 0.0))
            with np.errstate(invalid="ignore", divide="ignore"):
                phi = np.where(rr > 0.0, -np.expm1(-rr * dt) / rr, dt)
            out[k] += (r * ceq - rr * out[k]) * phi
    return out


class KineticsRiverine(sources.KineticsRiverine):
    """oracle.kinetics_sources.KineticsRiverine with the Monod factors of `react` (keyword arguments limit_process, ...,
    limit_half_saturation, besides the source ones); reaction_mass[t][k] includes them.  update() is the parent's, line
    for line, with this module's react in place of oracle.kinetics_sources.react."""

    def __init__(self, mesh: HydroMesh, inputs: Dict[str, np.ndarray], decay_per_day, theta=None, yields=None,
                 temperature: Union[str, float, None] = None, **terms):
        super().__init__(mesh, inputs, decay_per_day, theta, yields, temperature,
                         **{k: v for k, v in terms.items() if k not in LIMIT_KEYS})
        self.limits = {k: v for k, v in terms.items() if k in LIMIT_KEYS}

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
        reacted = react(merged, np.float64(mesh.dt[t]), self.decay, self.theta, self.yields, temp, is_index,
                        **self.sources, **self.limits)
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


def limit_terms(process=None, column=None, factor_column=None, factor_kind=None, half_saturation=None) -> dict:
    """The keyword arguments of `react` / `KineticsRiverine` from those of TransportBackend.set_kinetics_limits."""
    return dict(zip(LIMIT_KEYS, (process, column, factor_column, factor_kind, half_saturation)))
