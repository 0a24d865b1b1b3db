"""Asynchronous successive halving (ASHA) over the members of an ensemble run: the early-stopping rule of the
reference's hyper-parameter search (ray_hyperparam.py runs ``tune.run`` with an ASHA scheduler on the score that
jsrl_w_iql.py:589,592 reports).

The rule is that of Ray Tune's ``AsyncHyperBandScheduler`` with one bracket, written down here so that it can be
pinned by tests; Ray itself is not used and exact parity with it is not claimed.  Time is a member's number of reports
so far (Ray's ``training_iteration``).  The rungs sit at ``grace_period * reduction_factor**k`` for k = 0 .. n - 1,
n = floor(log(max_t / grace_period) / log(reduction_factor)) + 1.  A report at time t is compared at the highest rung
that t has reached and the member has not reported at yet: the member stops when its score is below the
(1 - 1 / reduction_factor) quantile of the scores recorded there so far (NaN scores ignored), and its score is recorded
there either way.  The first members to reach a rung therefore always continue.  Every report at t >= max_t stops.
"""
from __future__ import annotations

import math
import warnings
from typing import Dict, List, Optional, Tuple

import numpy as np

CONTINUE, STOP = "continue", "stop"


class ASHAScheduler:
    def __init__(self, max_t: int = 100, grace_period: int = 1, reduction_factor: float = 4, mode: str = "max"):
        if mode not in ("max", "min"):
            raise ValueError(f"mode must be 'max' or 'min', got {mode!r}")
        if grace_period < 1 or max_t < grace_period:
            raise ValueError(f"need 1 <= grace_period <= max_t, got grace_period={grace_period}, max_t={max_t}")
        if reduction_factor <= 1:
            raise ValueError(f"reduction_factor must be > 1, got {reduction_factor}")
        self.max_t, self.grace_period, self.rf, self.mode = max_t, grace_period, reduction_factor, mode
        n = int(math.floor(math.log(max_t / grace_period) / math.log(reduction_factor))) + 1
        # (milestone, {member: recorded score}), highest milestone first
        self.rungs: List[Tuple[float, Dict[int, float]]] = [(grace_period * reduction_factor ** k, {}) for k in reversed(range(n))]
        self.stopped: Dict[int, Tuple[int, Optional[int]]] = {}  # member -> (t, total_it) of the report that stopped it

    @property
    def milestones(self) -> List[float]:
        return [ms for ms, _ in self.rungs]

    def on_result(self, member: int, t: int, score: float, total_it: Optional[int] = None) -> str:
        """Report ``score`` of ``member`` at its ``t``-th report; returns "continue" or "stop"."""
        action = CONTINUE
        if t >= self.max_t:
            action = STOP
        else:
            s = float(score) if self.mode == "max" else -float(score)
            for milestone, recorded in self.rungs:
                if t < milestone or member in recorded:
                    continue
                if recorded:
                    with warnings.catch_warnings():  # every recorded score NaN: the cutoff is NaN and nobody stops
                        warnings.simplefilter("ignore", RuntimeWarning)
                        cutoff = np.nanpercentile(np.asarray(list(recorded.values()), dtype=np.float64), (1 - 1 / self.rf) * 100)
                    if s < cutoff:
                        action = STOP
                recorded[member] = s
                break
        if action == STOP:
            self.stopped[member] = (int(t), None if total_it is None else int(total_it))
        return action
