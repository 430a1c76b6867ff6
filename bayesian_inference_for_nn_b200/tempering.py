"""Parallel-tempering ladders for HMC (pyb_hmc_set_temperatures, include/pyesian_b200.h).

A ladder is a list of R inverse temperatures 1 = beta_0 > beta_1 > ... > beta_{R-1} > 0.  Every posterior chain becomes
a replica group of R chains, one per rung, laid out group-major: engine chain g R + r is rung r of group g.  Only rung 0
samples the posterior; the hotter rungs explore flatter versions of it and hand their states down through replica
swaps.  The checks here run before any engine exists, so a bad ladder fails on any machine.
"""
from __future__ import annotations

import math

MAX_RUNGS = 64


def validate_ladder(betas):
    """-> the ladder as a list of floats, or None when tempering is off (``betas`` None, empty or of length 1).
    Raises ValueError unless it starts at 1.0, decreases strictly, stays finite and > 0 and has at most 64 rungs."""
    if betas is None:
        return None
    try:
        b = [float(v) for v in betas]
    except TypeError:
        raise ValueError("inverse_temperatures must be a list of numbers") from None
    if len(b) == 0:
        return None
    if b[0] != 1.0:
        raise ValueError("the first inverse temperature must be 1.0, got %r" % b[0])
    if len(b) == 1:
        return None
    if len(b) > MAX_RUNGS:
        raise ValueError("a ladder has at most %d rungs, got %d" % (MAX_RUNGS, len(b)))
    for r in range(1, len(b)):
        if not (math.isfinite(b[r]) and 0.0 < b[r] < b[r - 1]):
            raise ValueError("inverse temperatures must decrease strictly and stay > 0: %r" % (b,))
    return b


def geometric_ladder(R: int, beta_min: float):
    """R inverse temperatures from 1 down to ``beta_min`` in equal ratios (a common first ladder to tune from)."""
    if R < 2 or not 0.0 < beta_min < 1.0:
        raise ValueError("need R >= 2 and 0 < beta_min < 1")
    return [beta_min ** (r / (R - 1)) for r in range(R)]
