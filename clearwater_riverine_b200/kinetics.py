"""First-order kinetics by constituent name -> the arrays of `cwr_set_kinetics` (include/cwr.h), validated.

    {"BOD": {"decay_per_day": 0.23, "theta": 1.047, "yields": {"DO": -1.0}},
     "NH4": {"decay_per_day": 0.10, "theta": 1.083, "yields": {"NO3": 1.0, "DO": -4.57}}}

Every step, each real cell is reacted before the load term is formed: for the decaying constituents k in topological
order of the yield graph, loss = c_k (1 - exp(-decay_k theta_k^(T - 20) dt / 86400)) leaves k and yield * loss is added
to every constituent k yields.  The temperature T (deg C) is a constant or another constituent's value in the cell.
The library checks the same conditions; checking them here names the constituents in the error.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Mapping, Sequence, Tuple, Union

import numpy as np

_KEYS = {"decay_per_day", "theta", "yields"}


@dataclass(frozen=True)
class Kinetics:
    decay_per_day: np.ndarray     # (K,) 1/day
    theta: np.ndarray             # (K,) Arrhenius factor per deg C
    yields: np.ndarray            # (K, K) yields[j, k] = mass of j formed per mass of k decayed
    temperature_k: int            # temperature constituent, or -1
    temperature_c: float          # the constant temperature when temperature_k == -1
    order: Tuple[int, ...]        # topological order of the yield graph (the order the reactions are applied in)


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


def validate(decay_per_day, theta, yields, temperature_k: int, temperature_c: float, names: Sequence[str] = ()) -> None:
    """The conditions cwr_set_kinetics rejects with CWR_EINVAL, as ValueError."""
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


def compile_kinetics(spec: Mapping[str, Mapping], constituents: Sequence[str],
                     temperature: Union[str, float] = 20.0) -> Kinetics:
    """spec: {constituent: {"decay_per_day": float, "theta": float (default 1), "yields": {constituent: float}}};
    temperature: a constituent name, or a constant in deg C."""
    names = list(constituents)
    index = {n: k for k, n in enumerate(names)}
    K = len(names)
    decay, theta, yields = np.zeros(K), np.ones(K), np.zeros((K, K))
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
    if isinstance(temperature, str):
        if temperature not in index:
            raise ValueError(f"temperature constituent {temperature!r} is not a constituent of the model")
        temperature_k, temperature_c = index[temperature], 20.0
    else:
        temperature_k, temperature_c = -1, float(temperature)
    validate(decay, theta, yields, temperature_k, temperature_c, names)
    return Kinetics(decay, theta, yields, temperature_k, temperature_c, topological_order(yields))
