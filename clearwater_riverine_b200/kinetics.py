"""Kinetics by constituent name -> the arrays of `cwr_set_kinetics`, `cwr_set_kinetics_sources` and
`cwr_set_kinetics_limits` (include/cwr.h), validated.

    {"BOD": {"decay_per_day": 0.23, "theta": 1.047, "yields": {"DO": -1.0}},
     "NH4": {"decay_per_day": 0.10, "theta": 1.083, "yields": {"NO3": 1.0, "DO": -4.57}},
     "DO":  {"source_per_day": -1.5, "source_theta": 1.065,                       # sediment oxygen demand
             "exchange_per_day": 0.7, "exchange_theta": 1.024, "equilibrium": "oxygen_saturation"},
     "T":   {"exchange_per_day": 0.3, "equilibrium": 18.0}}                       # equilibrium temperature

Monod factors, each a {constituent: half_saturation} mapping, scale a constituent's decay (`limited_by`, `inhibited_by`)
or its source (`source_limited_by`, `source_inhibited_by`) by c+/(K + c+) or K/(K + c+), c+ = max(c, 0):

    {"BOD": {"decay_per_day": 0.23, "yields": {"DO": -1.0}, "limited_by": {"DO": 0.5}},
     "NO3": {"decay_per_day": 0.1, "inhibited_by": {"DO": 0.6}},                  # denitrification
     "DO":  {"source_per_day": -1.5, "source_limited_by": {"DO": 1.0}}}           # self-limited sediment oxygen demand

Every step, each real cell is reacted before the load term is formed: for the decaying constituents k in topological
order of the yield graph, loss = c_k (1 - exp(-decay_k theta_k^(T - 20) dt / 86400)) leaves k and yield * loss is added
to every constituent k yields.  Then every constituent with a zero-order source s (per day) or an exchange rate r
(1/day) toward an equilibrium ceq follows dc/dt = s + r (ceq - c), solved exactly over the step, with s and r corrected
by their own theta^(T - 20); ceq is a constant or the oxygen saturation at T (`oxygen_saturation`).  The temperature T
(deg C) is a constant or another constituent's value in the cell before the step's reactions.
A decay limited by a constituent it consumes (a negative yield) never takes more of it than the cell holds, and a sink
limited by its own constituent is solved as a first-order sink, so such a constituent cannot be driven below zero.
The library checks the same conditions; checking them here names the constituents in the error.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Mapping, Optional, Sequence, Tuple, Union

import numpy as np

_KEYS = {"decay_per_day", "theta", "yields", "source_per_day", "source_theta", "exchange_per_day", "exchange_theta",
         "equilibrium", "limited_by", "inhibited_by", "source_limited_by", "source_inhibited_by"}
OXYGEN_SATURATION = "oxygen_saturation"
# spec key -> (process: 0 decay, 1 source; kind: 0 limitation, 1 inhibition), in the order a block's factors compile
_FACTOR_KEYS = {"limited_by": (0, 0), "source_limited_by": (1, 0), "inhibited_by": (0, 1), "source_inhibited_by": (1, 1)}


def oxygen_saturation(T):
    """Dissolved-oxygen saturation (mg/L) of fresh water at 1 atm, T in deg C: the APHA / Benson-Krause formula
    ln O2sat = -139.34411 + 1.575701e5/Ta - 6.642308e7/Ta^2 + 1.243800e10/Ta^3 - 8.621949e11/Ta^4, Ta = T + 273.15,
    evaluated as the device evaluates it, with no clamp."""
    x = 1.0 / (np.asarray(T, np.float64) + 273.15)
    return np.exp(-139.34411 + x * (1.575701e5 + x * (-6.642308e7 + x * (1.243800e10 + x * -8.621949e11))))


@dataclass(frozen=True)
class Kinetics:
    decay_per_day: np.ndarray     # (K,) 1/day
    theta: np.ndarray             # (K,) Arrhenius factor per deg C
    yields: np.ndarray            # (K, K) yields[j, k] = mass of j formed per mass of k decayed
    temperature_k: int            # temperature constituent, or -1
    temperature_c: float          # the constant temperature when temperature_k == -1
    order: Tuple[int, ...]        # topological order of the yield graph (the order the reactions are applied in)
    source_per_day: Optional[np.ndarray] = None     # (K,) zero-order source, concentration units per day (< 0: a sink)
    source_theta: Optional[np.ndarray] = None       # (K,)
    exchange_per_day: Optional[np.ndarray] = None   # (K,) 1/day, relaxation toward the equilibrium
    exchange_theta: Optional[np.ndarray] = None     # (K,)
    equilibrium: Optional[np.ndarray] = None        # (K,) the constant target of kind 0
    equilibrium_kind: Optional[np.ndarray] = None   # (K,) int32: 0 = constant, 1 = oxygen saturation at T
    # Monod factors, (n,) each: the process (int32 0 = decay, 1 = source) of `limit_column` scaled by a factor of
    # `limit_kind` (int32 0 = limitation, 1 = inhibition) on `limit_factor_column` with `limit_half_saturation`
    limit_process: Optional[np.ndarray] = None
    limit_column: Optional[np.ndarray] = None
    limit_factor_column: Optional[np.ndarray] = None
    limit_kind: Optional[np.ndarray] = None
    limit_half_saturation: Optional[np.ndarray] = None

    @property
    def has_sources(self) -> bool:
        """Whether any constituent has a source or an exchange term (otherwise cwr_set_kinetics_sources is not needed)."""
        return any(a is not None and (a != 0).any() for a in (self.source_per_day, self.exchange_per_day))

    def sources_arguments(self) -> dict:
        """The arguments of TransportBackend.set_kinetics_sources."""
        return dict(source_per_day=self.source_per_day, source_theta=self.source_theta, exchange_per_day=self.exchange_per_day,
                    exchange_theta=self.exchange_theta, equilibrium=self.equilibrium, equilibrium_kind=self.equilibrium_kind)

    @property
    def has_limits(self) -> bool:
        """Whether any process carries a Monod factor (otherwise cwr_set_kinetics_limits is not needed)."""
        return self.limit_process is not None and len(self.limit_process) > 0

    def limits_arguments(self) -> dict:
        """The arguments of TransportBackend.set_kinetics_limits."""
        return dict(process=self.limit_process, column=self.limit_column, factor_column=self.limit_factor_column,
                    factor_kind=self.limit_kind, half_saturation=self.limit_half_saturation)


def topological_order(yields: np.ndarray) -> Tuple[int, ...]:
    """Order of the constituents in which every one comes after all those it receives a yield from (edges k -> j where
    yields[j, k] != 0); among the ready ones the smallest index first, as the library orders them.  ValueError on a cycle."""
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
    return tuple(order)


def validate(decay_per_day, theta, yields, temperature_k: int, temperature_c: float, names: Sequence[str] = (), *,
             source_per_day=None, source_theta=None, exchange_per_day=None, exchange_theta=None, equilibrium=None,
             equilibrium_kind=None, limit_process=None, limit_column=None, limit_factor_column=None, limit_kind=None,
             limit_half_saturation=None) -> None:
    """The conditions cwr_set_kinetics, cwr_set_kinetics_sources and cwr_set_kinetics_limits reject with CWR_EINVAL, as
    ValueError.  The source arrays follow the ABI: None = none / all 1 / all 0 as there; the limit arrays are (n,) or
    None = no limits."""
    d, th, y = np.asarray(decay_per_day, np.float64), np.asarray(theta, np.float64), np.asarray(yields, np.float64)
    K = d.shape[0]
    nm = (lambda k: repr(names[k])) if len(names) == K else (lambda k: f"#{k}")
    for k in range(K):
        if not math.isfinite(d[k]) or d[k] < 0:
            raise ValueError(f"decay_per_day of {nm(k)} must be finite and >= 0, got {d[k]}")
        if not math.isfinite(th[k]) or th[k] <= 0:
            raise ValueError(f"theta of {nm(k)} must be finite and > 0, got {th[k]}")
    if not np.isfinite(y).all():
        raise ValueError("yields must be finite")
    for k in range(K):
        if y[k, k] != 0:
            raise ValueError(f"{nm(k)} cannot yield itself")
    if not -1 <= temperature_k < K:
        raise ValueError(f"temperature constituent index {temperature_k} out of range")
    if temperature_k < 0 and not math.isfinite(temperature_c):
        raise ValueError(f"temperature must be finite, got {temperature_c}")
    if temperature_k >= 0:
        if d[temperature_k] != 0:
            raise ValueError(f"the temperature constituent {nm(temperature_k)} cannot decay")
        if (y[temperature_k] != 0).any():
            raise ValueError(f"the temperature constituent {nm(temperature_k)} cannot receive a yield")
    topological_order(y)
    _validate_limits(d, y, source_per_day, nm, limit_process, limit_column, limit_factor_column, limit_kind,
                     limit_half_saturation)
    if source_per_day is None and exchange_per_day is None:
        return
    if exchange_per_day is not None and equilibrium is None:
        raise ValueError("an exchange rate needs an equilibrium")
    col = lambda a, fill: np.full(K, fill, np.float64) if a is None else np.asarray(a, np.float64)
    s, sth, e, eth = col(source_per_day, 0.0), col(source_theta, 1.0), col(exchange_per_day, 0.0), col(exchange_theta, 1.0)
    eq = col(equilibrium, 0.0)
    kind = np.zeros(K, np.int64) if equilibrium_kind is None else np.asarray(equilibrium_kind)
    for k in range(K):
        if not math.isfinite(s[k]):
            raise ValueError(f"source_per_day of {nm(k)} must be finite, got {s[k]}")
        for what, v in (("source_theta", sth[k]), ("exchange_theta", eth[k])):
            if not math.isfinite(v) or v <= 0:
                raise ValueError(f"{what} of {nm(k)} must be finite and > 0, got {v}")
        if not math.isfinite(e[k]) or e[k] < 0:
            raise ValueError(f"exchange_per_day of {nm(k)} must be finite and >= 0, got {e[k]}")
        if kind[k] not in (0, 1):
            raise ValueError(f"equilibrium kind of {nm(k)} must be 0 (constant) or 1 ({OXYGEN_SATURATION}), got {kind[k]}")
        if kind[k] == 0 and e[k] > 0 and not math.isfinite(eq[k]):
            raise ValueError(f"equilibrium of {nm(k)} must be finite, got {eq[k]}")
        if kind[k] == 1 and k == temperature_k:
            raise ValueError(f"the temperature constituent {nm(k)} cannot relax toward {OXYGEN_SATURATION}")


def _validate_limits(d, y, source_per_day, nm, process, column, factor_column, kind, half) -> None:
    if process is None:
        return
    arrs = [np.asarray(a).reshape(-1) for a in (process, column, factor_column, kind)]
    h = np.asarray(half, np.float64).reshape(-1)
    if any(len(a) != len(h) for a in arrs):
        raise ValueError("the limit arrays must have the same length")
    K = d.shape[0]
    s = np.zeros(K) if source_per_day is None else np.asarray(source_per_day, np.float64)
    seen = set()
    for pr, k, j, kd, hs in zip(*arrs, h):
        pr, k, j, kd = int(pr), int(k), int(j), int(kd)
        if pr not in (0, 1):
            raise ValueError(f"a limit's process must be 0 (decay) or 1 (source), got {pr}")
        if kd not in (0, 1):
            raise ValueError(f"a limit's kind must be 0 (limitation) or 1 (inhibition), got {kd}")
        if not (0 <= k < K and 0 <= j < K):
            raise ValueError(f"a limit's column index out of range: {k}, {j}")
        what = ("decay", "source")[pr] + " of " + nm(k)
        by = ("limitation", "inhibition")[kd] + " by " + nm(j)
        if not math.isfinite(hs) or hs <= 0:
            raise ValueError(f"{by} of the {what}: the half-saturation must be finite and > 0, got {hs}")
        if pr == 0 and d[k] == 0:
            raise ValueError(f"{by}: {nm(k)} does not decay")
        if pr == 1 and s[k] == 0:
            raise ValueError(f"{by}: {nm(k)} has no source")
        if pr == 0 and j == k:
            raise ValueError(f"the decay of {nm(k)} cannot be limited or inhibited by {nm(k)} itself")
        if pr == 1 and j == k and (kd != 0 or s[k] >= 0):
            raise ValueError(f"the source of {nm(k)} can only be limited by {nm(k)} itself when it is a sink (< 0); "
                             f"got {by} with source {s[k]}")
        if (pr, k, j, kd) in seen:
            raise ValueError(f"{by} of the {what} given twice")
        seen.add((pr, k, j, kd))


def compile_kinetics(spec: Mapping[str, Mapping], constituents: Sequence[str],
                     temperature: Union[str, float] = 20.0) -> Kinetics:
    """spec: {constituent: {"decay_per_day": float, "theta": float (default 1), "yields": {constituent: float},
    "source_per_day": float, "source_theta": float (default 1), "exchange_per_day": float, "exchange_theta": float
    (default 1), "equilibrium": float or "oxygen_saturation" (required when exchange_per_day > 0), "limited_by",
    "inhibited_by", "source_limited_by", "source_inhibited_by": {constituent: half_saturation}}};
    temperature: a constituent name, or a constant in deg C.  The factors compile per block in spec order of the blocks:
    the limitations (decay, then source) first, then the inhibitions (decay, then source), each mapping in its order."""
    names = list(constituents)
    index = {n: k for k, n in enumerate(names)}
    K = len(names)
    decay, theta, yields = np.zeros(K), np.ones(K), np.zeros((K, K))
    source, source_theta, exchange, exchange_theta = np.zeros(K), np.ones(K), np.zeros(K), np.ones(K)
    equilibrium, kind = np.zeros(K), np.zeros(K, np.int32)
    factors = []                     # (process, column, factor column, kind, half-saturation)
    for name, block in spec.items():
        if name not in index:
            raise ValueError(f"kinetics given for {name!r}, which is not a constituent of the model")
        if not isinstance(block, Mapping):
            raise ValueError(f"kinetics of {name!r}: expected a mapping, got {type(block).__name__}")
        unknown = set(block) - _KEYS
        if unknown:
            raise ValueError(f"kinetics of {name!r}: unknown keys {sorted(unknown)} (expected {sorted(_KEYS)})")
        k = index[name]
        decay[k] = float(block.get("decay_per_day", 0.0))
        theta[k] = float(block.get("theta", 1.0))
        for target, y in (block.get("yields") or {}).items():
            if target not in index:
                raise ValueError(f"kinetics of {name!r}: yield to {target!r}, which is not a constituent of the model")
            yields[index[target], k] = float(y)
        source[k] = float(block.get("source_per_day", 0.0))
        source_theta[k] = float(block.get("source_theta", 1.0))
        exchange[k] = float(block.get("exchange_per_day", 0.0))
        exchange_theta[k] = float(block.get("exchange_theta", 1.0))
        eq = block.get("equilibrium")
        if isinstance(eq, str):
            if eq != OXYGEN_SATURATION:
                raise ValueError(f"kinetics of {name!r}: equilibrium must be a number or {OXYGEN_SATURATION!r}, got {eq!r}")
            kind[k] = 1
        elif eq is not None:
            equilibrium[k] = float(eq)
        elif exchange[k] > 0:
            raise ValueError(f"kinetics of {name!r}: exchange_per_day > 0 needs an equilibrium")
        for key, (process, fkind) in _FACTOR_KEYS.items():
            entries = block.get(key) or {}
            if not isinstance(entries, Mapping):
                raise ValueError(f"kinetics of {name!r}: {key} must map constituents to half-saturations")
            for target, half in entries.items():
                if target not in index:
                    raise ValueError(f"kinetics of {name!r}: {key} {target!r}, which is not a constituent of the model")
                factors.append((process, k, index[target], fkind, float(half)))
    if isinstance(temperature, str):
        if temperature not in index:
            raise ValueError(f"temperature constituent {temperature!r} is not a constituent of the model")
        temperature_k, temperature_c = index[temperature], 20.0
    else:
        temperature_k, temperature_c = -1, float(temperature)
    lim = [None] * 5
    if factors:
        cols = list(zip(*factors))
        lim = [np.array(cols[i], np.int32) for i in range(4)] + [np.array(cols[4], np.float64)]
    validate(decay, theta, yields, temperature_k, temperature_c, names, source_per_day=source, source_theta=source_theta,
             exchange_per_day=exchange, exchange_theta=exchange_theta, equilibrium=equilibrium, equilibrium_kind=kind,
             limit_process=lim[0], limit_column=lim[1], limit_factor_column=lim[2], limit_kind=lim[3],
             limit_half_saturation=lim[4])
    return Kinetics(decay, theta, yields, temperature_k, temperature_c, topological_order(yields), source, source_theta,
                    exchange, exchange_theta, equilibrium, kind, *lim)
