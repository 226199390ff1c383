"""CPU ORACLE of the device kinetics with time-varying forcing (cwr_set_kinetics_forcing, include/cwr.h) -- test
infrastructure only.

`KineticsRiverine` takes the arguments of oracle.kinetics_depth's and, optionally, the forcing (forcing_target,
forcing_column: (n,) each; forcing_values: (n, n_time)).  Its update() puts step t's entries of the series into the
parameters -- the temperature, decay f, source f, exchange f, the equilibrium -- and runs oracle.kinetics_depth's
update() with them, so the formulas are not restated here.  Without forcing it is oracle.kinetics_depth's, bit for bit.
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np

from . import kinetics_depth as depth
from .reference_step import HydroMesh

FORCING_KEYS = ("forcing_target", "forcing_column", "forcing_values")
TEMPERATURE, EQUILIBRIUM, DECAY_SCALE, SOURCE_SCALE, EXCHANGE_SCALE = range(5)


class KineticsRiverine(depth.KineticsRiverine):
    """oracle.kinetics_depth.KineticsRiverine with series that replace the constant temperature (target 0, column -1)
    or the constant equilibrium of a column (1), or scale its decay (2), source (3) or exchange rate (4); step t uses
    entry t, the scale multiplying the per-day rate before anything else acts on it."""

    def __init__(self, mesh: HydroMesh, inputs: Dict[str, np.ndarray], decay_per_day, theta=None, yields=None,
                 temperature=None, forcing_target=None, forcing_column=None, forcing_values=None, **terms):
        super().__init__(mesh, inputs, decay_per_day, theta, yields, temperature, **terms)
        n = 0 if forcing_target is None else len(forcing_target)
        self.forcing = [] if n == 0 else list(zip(np.asarray(forcing_target).tolist(), np.asarray(forcing_column).tolist(),
                                                  np.asarray(forcing_values, np.float64)))

    def update(self, update_concentration: Optional[Dict[str, np.ndarray]] = None):
        if not self.forcing:
            return super().update(update_concentration)
        t = self.time_step
        K = len(self.names)
        constants = (self.decay, self.temperature, self.sources)
        decay = np.array(self.decay, np.float64, copy=True)
        sources = dict(self.sources)
        for key in ("source_per_day", "exchange_per_day", "equilibrium"):
            if sources.get(key) is not None:
                sources[key] = np.array(sources[key], np.float64, copy=True)
        temperature = self.temperature
        for target, k, values in self.forcing:
            f = values[t]
            if target == TEMPERATURE:
                temperature = float(f)
            elif target == EQUILIBRIUM:
                sources["equilibrium"][k] = f
            elif target == DECAY_SCALE:
                decay[k] = decay[k] * f
            elif target == SOURCE_SCALE:
                sources["source_per_day"][k] = sources["source_per_day"][k] * f
            elif target == EXCHANGE_SCALE:
                sources["exchange_per_day"][k] = sources["exchange_per_day"][k] * f
            else:
                raise ValueError(f"unknown forcing target {target} (of {K} columns)")
        self.decay, self.temperature, self.sources = decay, temperature, sources
        try:
            super().update(update_concentration)
        finally:
            self.decay, self.temperature, self.sources = constants


def forcing_terms(target=None, column=None, values=None) -> dict:
    """The keyword arguments of `KineticsRiverine` from those of TransportBackend.set_kinetics_forcing."""
    return dict(zip(FORCING_KEYS, (target, column, values)))
