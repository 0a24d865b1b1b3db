#!/usr/bin/env python
"""GPU timeline of ONE update step as it runs inside the host-step CUDA graph (real overlap, PDL, side branches):
earliest CTA start and latest CTA end of every launch, from %globaltimer stamps (IQL_STEP_TRACE).
    python tools/step_trace.py [workload] [iterations]"""
import ctypes as C
import os
import sys

os.environ.setdefault("IQL_B200_DEBUG", "1")
os.environ.setdefault("IQL_STEP_TRACE", "1")
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
from jsrl_corl_b200 import IQLEnsemble, ReplayBuffer, _lib
from jsrl_corl_b200.synthetic import synthetic_dataset

SLOTS = ["refresh", "gather", "fused_fwd", "policy_head", "loss", "last_bwd", "lb_reduce", "hidden_wgrad", "hidden_dgrad", "first_wgrad",
         "adam_polyak", "advance", "bwd_chain"]


def main():
    name = sys.argv[1] if len(sys.argv) > 1 else "hopper_single"
    iters = int(sys.argv[2]) if len(sys.argv) > 2 else 200
    w = bench.WORKLOADS[name]
    S = w["members"]
    ens = IQLEnsemble(S, w["S"], w["A"], w["H"], w["L"], w["B"], deterministic=w["det"], actor_dropout=w["dropout"],
                      math_mode="tf32", device="cuda", max_steps_per_call=8, seeds=list(range(S)))
    n_rows = 200_000
    rb = ReplayBuffer(w["S"], w["A"], n_rows, "cuda")
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):
        rb.load_d4rl_dataset(synthetic_dataset(n_rows, w["S"], w["A"], 0, antmaze_rewards=w["antmaze"]))
    ens.bind_replay(rb)
    eng, L = ens.engine, _lib.lib()
    rng = np.random.RandomState(0)
    for _ in range(20):
        idx = rng.randint(0, n_rows, size=(S, w["B"]))
        eng.host_step(host_indices=idx.ctypes.data)
    buf = np.zeros(2 * len(SLOTS), dtype=np.uint64)
    acc = np.zeros((len(SLOTS), 2))
    cnt = np.zeros(len(SLOTS))
    span = 0.0
    for _ in range(iters):
        assert L.iql_debug_step_trace(eng._h, 1, None, 0, eng.stream.cuda_stream) == 0
        idx = rng.randint(0, n_rows, size=(S, w["B"]))
        eng.host_step(host_indices=idx.ctypes.data)
        n = L.iql_debug_step_trace(eng._h, 0, buf.ctypes.data_as(C.c_void_p), buf.size, None)
        assert n == buf.size, n
        t = buf.reshape(-1, 2).astype(np.float64)
        used = t[:, 1] > 0
        t0 = t[used, 0].min()
        span += (t[used, 1].max() - t0) / 1e3
        acc[used] += (t[used] - t0) / 1e3
        cnt += used
    print(f"{name}: {S} member(s), one K = 1 step inside the host-step graph, mean of {iters} steps; us from the first CTA start")
    print(f"{'launch':<14} {'start':>8} {'end':>8} {'duration':>9}")
    order = sorted([i for i in range(len(SLOTS)) if cnt[i]], key=lambda i: acc[i, 0] / cnt[i])
    for i in order:
        a, b = acc[i] / cnt[i]
        print(f"{SLOTS[i]:<14} {a:8.2f} {b:8.2f} {b - a:9.2f}")
    print(f"first start -> last end: {span / iters:.2f} us")


if __name__ == "__main__":
    main()
