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
Processes that act through the water depth -- settling, fluxes through the bed such as sediment oxygen demand, transfer
through the surface -- are given per unit depth, each in place of its volumetric key, and need the model's cell plan areas:

    {"PBOD": {"settling_per_day": 0.3},                                          # v_s, length/day: r = v_s / h
     "DO":   {"areal_source_per_day": -1.5, "source_limited_by": {"DO": 1.0},    # SOD, g/m2/day on an SI plan: s = SOD / h
              "transfer_per_day": 2.0, "equilibrium": "oxygen_saturation"}}      # K_L, length/day: r = K_L / h

with h = max(V / A, min_depth) the depth of each cell at each step, in the mesh's length unit (volume unit / area unit).
The library checks the same conditions; checking them here names the constituents in the error.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Mapping, Optional, Sequence, Tuple, Union

import numpy as np

_KEYS = {"decay_per_day", "theta", "yields", "source_per_day", "source_theta", "exchange_per_day", "exchange_theta",
         "equilibrium", "limited_by", "inhibited_by", "source_limited_by", "source_inhibited_by", "settling_per_day",
         "areal_source_per_day", "transfer_per_day"}
OXYGEN_SATURATION = "oxygen_saturation"
# per-depth spec key -> the volumetric key it replaces (the rate of the same process, divided by the depth)
_DEPTH_KEYS = {"settling_per_day": "decay_per_day", "areal_source_per_day": "source_per_day",
               "transfer_per_day": "exchange_per_day"}
# the floor of the depth h = max(V / A, min_depth), in mesh length units (1 cm on an SI plan): keeps the rates of dry and
# nearly dry cells finite
DEFAULT_MIN_DEPTH = 0.01
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
    # depth-scaled processes, (K,) int32 0/1 each or None: 1 divides the decay / source / exchange rate of column k by the
    # cell's depth h = max(V[t] / cell_area, min_depth); cell_area (F,) the plan areas, min_depth in mesh length units
    decay_per_depth: Optional[np.ndarray] = None
    source_per_depth: Optional[np.ndarray] = None
    exchange_per_depth: Optional[np.ndarray] = None
    cell_area: Optional[np.ndarray] = None
    min_depth: float = DEFAULT_MIN_DEPTH

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

    @property
    def has_depth(self) -> bool:
        """Whether any process is given per unit depth (otherwise cwr_set_kinetics_depth is not needed)."""
        return any(a is not None and (np.asarray(a) != 0).any()
                   for a in (self.decay_per_depth, self.source_per_depth, self.exchange_per_depth))

    def depth_arguments(self) -> dict:
        """The arguments of TransportBackend.set_kinetics_depth."""
        return dict(cell_area=self.cell_area, min_depth=self.min_depth, decay_per_depth=self.decay_per_depth,
                    source_per_depth=self.source_per_depth, exchange_per_depth=self.exchange_per_depth)


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
             limit_half_saturation=None, decay_per_depth=None, source_per_depth=None, exchange_per_depth=None,
             cell_area=None, min_depth: float = DEFAULT_MIN_DEPTH) -> None:
    """The conditions cwr_set_kinetics, cwr_set_kinetics_sources, cwr_set_kinetics_limits and cwr_set_kinetics_depth
    reject with CWR_EINVAL, as ValueError.  The source arrays follow the ABI: None = none / all 1 / all 0 as there; the
    limit arrays are (n,) or None = no limits; the depth flags (K,) or None = none; cell_area: the plan areas of the real
    cells (the ones the library reads), or None."""
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
    _validate_depth(d, source_per_day, exchange_per_day, nm, decay_per_depth, source_per_depth, exchange_per_depth,
                    cell_area, min_depth)
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


def _validate_depth(d, source_per_day, exchange_per_day, nm, decay_per_depth, source_per_depth, exchange_per_depth,
                    cell_area, min_depth) -> None:
    K = d.shape[0]
    rates = {"decay": d, "source": source_per_day, "exchange": exchange_per_day}
    per_depth = {"decay": decay_per_depth, "source": source_per_depth, "exchange": exchange_per_depth}
    flagged = []
    for what, flags in per_depth.items():
        if flags is None:
            continue
        f = np.asarray(flags).reshape(-1)
        if f.shape[0] != K:
            raise ValueError(f"{what}_per_depth: expected {K} flags, got {f.shape[0]}")
        for k in range(K):
            if f[k] not in (0, 1):
                raise ValueError(f"{what}_per_depth of {nm(k)} must be 0 or 1, got {f[k]}")
            if f[k] == 1:
                flagged.append((what, k))
    if not flagged:
        return
    for what, k in flagged:
        r = rates[what]
        if r is None or np.asarray(r, np.float64)[k] == 0:
            raise ValueError(f"the {what} of {nm(k)} is given per depth, but its rate is 0")
    if cell_area is None:
        what, k = flagged[0]
        raise ValueError(f"the {what} of {nm(k)} is given per depth, which needs the cell plan areas (cell_area)")
    if not (math.isfinite(min_depth) and min_depth > 0):
        raise ValueError(f"min_depth must be finite and > 0, got {min_depth}")
    a = np.asarray(cell_area, np.float64)
    bad = ~(np.isfinite(a) & (a > 0))
    if bad.any():
        i = int(np.argmax(bad))
        raise ValueError(f"cell areas must be finite and > 0 (processes of {nm(flagged[0][1])} are per depth); "
                         f"cell {i} has {a[i]}")


def compile_kinetics(spec: Mapping[str, Mapping], constituents: Sequence[str],
                     temperature: Union[str, float] = 20.0, *, cell_area=None, min_depth: float = DEFAULT_MIN_DEPTH,
                     n_real: Optional[int] = None) -> Kinetics:
    """spec: {constituent: {"decay_per_day": float, "theta": float (default 1), "yields": {constituent: float},
    "source_per_day": float, "source_theta": float (default 1), "exchange_per_day": float, "exchange_theta": float
    (default 1), "equilibrium": float or "oxygen_saturation" (required when exchange_per_day > 0), "limited_by",
    "inhibited_by", "source_limited_by", "source_inhibited_by": {constituent: half_saturation}, "settling_per_day",
    "areal_source_per_day", "transfer_per_day": the per-depth forms of decay_per_day, source_per_day and
    exchange_per_day, each in place of its counterpart}};
    temperature: a constituent name, or a constant in deg C; cell_area (F,) the plan areas, needed by the per-depth keys,
    of which the first n_real (default all) are the real cells; min_depth the floor of the depth.  The factors compile per block in spec order of the blocks:
    the limitations (decay, then source) first, then the inhibitions (decay, then source), each mapping in its order."""
    names = list(constituents)
    index = {n: k for k, n in enumerate(names)}
    K = len(names)
    decay, theta, yields = np.zeros(K), np.ones(K), np.zeros((K, K))
    source, source_theta, exchange, exchange_theta = np.zeros(K), np.ones(K), np.zeros(K), np.ones(K)
    equilibrium, kind = np.zeros(K), np.zeros(K, np.int32)
    factors = []                     # (process, column, factor column, kind, half-saturation)
    per_depth = {key: np.zeros(K, np.int32) for key in _DEPTH_KEYS}
    for name, block in spec.items():
        if name not in index:
            raise ValueError(f"kinetics given for {name!r}, which is not a constituent of the model")
        if not isinstance(block, Mapping):
            raise ValueError(f"kinetics of {name!r}: expected a mapping, got {type(block).__name__}")
        unknown = set(block) - _KEYS
        if unknown:
            raise ValueError(f"kinetics of {name!r}: unknown keys {sorted(unknown)} (expected {sorted(_KEYS)})")
        k = index[name]
        block = dict(block)
        for key, volumetric in _DEPTH_KEYS.items():
            if key in block:
                if volumetric in block:
                    raise ValueError(f"kinetics of {name!r}: {key} replaces {volumetric}; give one of them")
                block[volumetric] = block[key]
                per_depth[key][k] = float(block[key]) != 0.0
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
            key = "transfer_per_day" if per_depth["transfer_per_day"][k] else "exchange_per_day"
            raise ValueError(f"kinetics of {name!r}: {key} > 0 needs an equilibrium")
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
    depth = [per_depth[key] if per_depth[key].any() else None for key in _DEPTH_KEYS]
    area = None
    if cell_area is not None and any(f is not None for f in depth):
        area = np.ascontiguousarray(cell_area, np.float64)
    validate(decay, theta, yields, temperature_k, temperature_c, names, source_per_day=source, source_theta=source_theta,
             exchange_per_day=exchange, exchange_theta=exchange_theta, equilibrium=equilibrium, equilibrium_kind=kind,
             limit_process=lim[0], limit_column=lim[1], limit_factor_column=lim[2], limit_kind=lim[3],
             limit_half_saturation=lim[4], decay_per_depth=depth[0], source_per_depth=depth[1],
             exchange_per_depth=depth[2], cell_area=None if area is None else area[:n_real], min_depth=float(min_depth))
    return Kinetics(decay, theta, yields, temperature_k, temperature_c, topological_order(yields), source, source_theta,
                    exchange, exchange_theta, equilibrium, kind, *lim, *depth, area, float(min_depth))
