#!/usr/bin/env python
"""What drawing each member's numpy index stream on the device (IQL_SAMPLE_MT19937) saves over the host draw that
ensemble_train_loop makes with its per-member RandomState objects, on the same indices:

1. offline K-step calls, 64 halfcheetah members, K = 256: the host draw (S x K randint calls) + mode="indices" call +
   loss read-back, against mode="numpy" and mode="philox" (a different stream) with the same read-back; plus the
   sampler's own time (the handle-free form of the same device code, CUDA events);
2. the online loop body (act, ring insert, logged update) at S = 1 / 8 / 64 with per-member randint draws, against the
   device stream;
3. ensemble_train_loop end to end on a toy env at 8 and 64 members, device_index_streams off and on.

Variants alternate within each repetition; medians are reported.  The card's name and power limit are read in the run.

    python tools/index_stream_rate.py [--out profiles/r08_index_streams.json] [--quick]
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from jsrl_corl_b200 import IQLEnsemble, ReplayBuffer, _lib
from jsrl_corl_b200.synthetic import synthetic_dataset

B = 256
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from ensemble_online_rate import ToyEnv, gpu_info  # noqa: E402


def offline(S, K, reps, rows=1_000_000):
    ens = IQLEnsemble(S, 17, 6, 256, 2, B, seeds=list(range(S)), max_steps_per_call=K)
    rb = ReplayBuffer(17, 6, rows, "cuda")
    rb.load_d4rl_dataset(synthetic_dataset(rows, 17, 6, 0))
    ens.bind_replay(rb)
    rngs = [np.random.RandomState(m) for m in range(S)]
    high = rb._high()

    def host():
        idx = np.zeros((S, K, B), dtype=np.int64)
        for m in range(S):
            for k in range(K):
                idx[m, k] = rngs[m].randint(0, high, size=B)
        return ens.train_steps(K, mode="indices", indices=torch.from_numpy(idx)).cpu()

    def device():
        return ens.train_steps(K, mode="numpy").cpu()

    def philox():
        return ens.train_steps(K, mode="philox").cpu()

    ens.set_index_streams([np.random.RandomState(m) for m in range(S)])
    variants = {"host_draw_indices": host, "device_numpy": device, "philox": philox}
    for f in variants.values():  # warm-up: graphs captured, modules loaded
        f()
    times = {k: [] for k in variants}
    for _ in range(reps):
        for name, f in variants.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            f()
            times[name].append(time.perf_counter() - t0)
    res = {"members": S, "K": K, "replay_rows": rows, "timer": "host perf_counter per call, losses read back"}
    for name, ts in times.items():
        med = float(np.median(ts))
        res[name] = {"call_ms": round(med * 1e3, 2), "member_steps_per_s": round(S * K / med)}
    # the sampler alone: the same device code through the handle-free entry point, S streams x K * B draws
    states = torch.from_numpy(np.stack([np.concatenate([r.get_state()[1], [r.get_state()[2], 0]]).astype(np.uint32)
                                        for r in rngs]).view(np.int32)).cuda()
    out = torch.empty(S, K * B, dtype=torch.int64, device="cuda")
    hi, cnt = np.full(S, high, np.int64), np.full(S, K * B, np.int64)
    L, st = _lib.lib(), torch.cuda.current_stream()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for _ in range(3):
        L.iql_mt19937_randint(states.data_ptr(), S, hi.ctypes.data, cnt.ctypes.data, out.data_ptr(), K * B, st.cuda_stream)
    n = 20
    ev[0].record()
    for _ in range(n):
        L.iql_mt19937_randint(states.data_ptr(), S, hi.ctypes.data, cnt.ctypes.data, out.data_ptr(), K * B, st.cuda_stream)
    ev[1].record()
    torch.cuda.synchronize()
    res["sampler_launch_us"] = round(ev[0].elapsed_time(ev[1]) / n * 1e3, 1)
    res["sampler_note"] = f"{S} streams x {K * B} draws at high {high}, CUDA events over {n} launches"
    return res


def online(S, n, warm, ring=10_000):
    """The online body as ensemble_train_loop runs it: act, insert, then per-member randint + logged update (host) or
    the logged update on the device streams; two identical learners, one per variant, alternating iterations."""
    rng = np.random.RandomState(1)
    obs = rng.randn(n + warm + 1, S, 17).astype(np.float32)
    src = np.where(np.arange(S) % 2 == 0, 2, 3).astype(np.int8)
    out, std = np.zeros((S, 6), np.float32), np.zeros((S, 6), np.float32)
    rew, done = np.ones(S, np.float32), np.zeros(S, np.float32)
    arms = {}
    for name in ("host_draw", "device_stream"):
        learner = IQLEnsemble(S, 17, 6, 256, 2, B, seeds=list(range(S)), max_steps_per_call=1)
        guide = IQLEnsemble(S, 17, 6, 256, 2, B, seeds=list(range(100, 100 + S)), max_steps_per_call=1)
        learner.set_guide(guide)
        rings = [ReplayBuffer(17, 6, ring, "cuda") for _ in range(S)]
        learner.bind_replay(rings)
        for i in range(B):
            learner.add_transitions(obs[i % (n + warm)], out, rew, obs[i % (n + warm) + 1], done)
        rngs = [np.random.RandomState(m) for m in range(S)]
        learner.set_index_streams(rngs)
        arms[name] = (learner, guide, rings, rngs, np.zeros((S, B), np.int64), [])

    def iteration(name, i):
        learner, _, rings, rngs, idx, ts = arms[name]
        t0 = time.perf_counter()
        learner.act(obs[i], src, 1.0, out=out, std=std)
        learner.add_transitions(obs[i], out, rew, obs[i + 1], done)
        if name == "host_draw":
            for m in range(S):
                idx[m] = rngs[m].randint(0, rings[m]._high(), size=B)
            learner.train_step_logged(idx)
        else:
            learner.train_step_logged(numpy_streams=True)
        ts.append(time.perf_counter() - t0)

    for i in range(n + warm):
        for name in arms:
            iteration(name, i)
    torch.cuda.synchronize()
    res = {"members": S}
    for name, arm in arms.items():
        med = float(np.median(arm[5][warm:]))
        res[name] = {"iteration_us": round(med * 1e6, 1), "member_env_steps_per_s": round(S / med)}
    # the two arms drew the same indices: the same weights
    res["same_params"] = bool(torch.equal(arms["host_draw"][0].engine.params, arms["device_stream"][0].engine.params))
    return res


def loop(S, off, on, eval_freq, n_episodes, device_streams):
    import contextlib
    import io

    from jsrl_corl_b200.jsrl_utils import JsrlTrainConfig
    from jsrl_corl_b200.jsrl_w_iql import ensemble_train_loop

    cfgs = [JsrlTrainConfig(device="cuda", env="Toy-v0", seed=m, eval_freq=eval_freq, n_episodes=n_episodes, offline_iterations=off,
                            online_iterations=on, batch_size=B, n_curriculum_stages=3, rolling_mean_n=1, tolerance=0.1 + 0.01 * m)
            for m in range(S)]
    rb = ReplayBuffer(3, 2, 20_000, "cuda")
    with contextlib.redirect_stdout(io.StringIO()):
        rb.load_d4rl_dataset(synthetic_dataset(20_000, 3, 2, 0))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        learner, _, _ = ensemble_train_loop(cfgs, [ToyEnv(m) for m in range(S)], [ToyEnv(1000 + m) for m in range(S)], rb, 3, 2, 1.0,
                                            ToyEnv.T, device_index_streams=device_streams)
        torch.cuda.synchronize()
    return time.perf_counter() - t0, learner.engine.params.clone()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="short windows (a functional run, not a measurement)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("index_stream_rate.py measures on the GPU; no CUDA device found")
    res = {"card": gpu_info(), "batch_size": B}
    res["offline_calls"] = offline(64, 256, 3 if args.quick else 9)
    print(json.dumps(res["offline_calls"]), flush=True)
    n, warm = (40, 10) if args.quick else (1000, 100)
    res["online_body"] = [online(S, n, warm) for S in (1, 8, 64)]
    print(json.dumps(res["online_body"]), flush=True)
    off, on, ev = (300, 300, 300) if args.quick else (500, 3000, 1000)
    res["ensemble_train_loop"] = []
    for S in (8, 64):
        walls = {False: [], True: []}
        params = {}
        for _ in range(1 if args.quick else 2):
            for dev in (False, True):
                w, params[dev] = loop(S, off, on, ev, 2, dev)
                walls[dev].append(w)
        row = {"members": S, "offline_iterations": off, "online_iterations": on, "eval_freq": ev, "n_episodes": 2,
               "host_draw_wall_s": round(float(np.median(walls[False])), 2),
               "device_stream_wall_s": round(float(np.median(walls[True])), 2),
               "same_params": bool(torch.equal(params[False], params[True]))}
        res["ensemble_train_loop"].append(row)
        print(json.dumps(row), flush=True)
    res["card_after"] = gpu_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))
