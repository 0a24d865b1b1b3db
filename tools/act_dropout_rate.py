#!/usr/bin/env python
"""What actor dropout costs in the batched act kernel, and what the online phase of a dropout ensemble costs.

1. The act call alone (IQLEnsemble.act, synchronised before every call, so no update is in flight): every member on
   the Gaussian distribution code 2 versus the training-mode dropout code 5 at p = 0.1; median of N calls after W
   warm-up calls, pen 45/24 2x256 and antmaze 29/8 3x256, S = 1 / 8 / 64.
2. The online body (act with code 5 + ring insert + logged update, no env) of the pen shape at S = 1 / 8 / 64, the
   protocol of tools/ensemble_online_rate.py, against the single-learner body whose training-mode dropout act runs
   through stock torch (GaussianPolicy.act with the actor in train mode): S sequential loops cost S times that.
3. ensemble_train_loop(..., philox_act_dropout=True) end to end on the toy env with actor_dropout = 0.1.

    python tools/act_dropout_rate.py [--out profiles/r07_act_dropout.json] [--quick]
"""
import argparse
import contextlib
import io
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import jsrl_corl_b200 as J
from jsrl_corl_b200 import IQLEnsemble, ReplayBuffer
from jsrl_corl_b200 import _lib
from jsrl_corl_b200.synthetic import synthetic_dataset

B, P = 256, 0.1
SHAPES = {"pen_gauss_2x256": (45, 24, 2), "antmaze_gauss_3x256": (29, 8, 3)}


def act_alone(S, Sd, A, L, n, warm):
    ens = IQLEnsemble(S, Sd, A, 256, L, B, actor_dropout=P, seeds=list(range(S)), max_steps_per_call=1)
    obs = np.random.RandomState(1).randn(S, Sd).astype(np.float32)
    out, std = np.zeros((S, A), np.float32), np.zeros((S, A), np.float32)
    row = {"members": S}
    for name, code in (("dist_code2", _lib.ACT_LEARNER_DIST), ("dist_dropout_code5", _lib.ACT_LEARNER_DIST_DROPOUT)):
        src = np.full(S, code, np.int8)
        ts = []
        for i in range(n + warm):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ens.act(obs, src, 1.0, out=out, std=std)
            if i >= warm:
                ts.append(time.perf_counter() - t0)
        row[name + "_median_us"] = round(float(np.median(ts)) * 1e6, 1)
    row["dropout_extra_us"] = round(row["dist_dropout_code5_median_us"] - row["dist_code2_median_us"], 1)
    return row


def body(S, Sd, A, L, n, warm, ring=10_000):
    learner = IQLEnsemble(S, Sd, A, 256, L, B, actor_dropout=P, seeds=list(range(S)), max_steps_per_call=1)
    rings = [ReplayBuffer(Sd, A, ring, "cuda") for _ in range(S)]
    learner.bind_replay(rings)
    rng = np.random.RandomState(1)
    obs = rng.randn(n + warm + 1, S, Sd).astype(np.float32)
    src = np.full(S, _lib.ACT_LEARNER_DIST_DROPOUT, np.int8)
    out, std = np.zeros((S, A), np.float32), np.zeros((S, A), np.float32)
    rew, done = np.ones(S, np.float32), np.zeros(S, np.float32)
    for i in range(B):  # the rings hold a batch before the first update
        learner.add_transitions(obs[i % (n + warm)], out, rew, obs[i % (n + warm) + 1], done)
    parts, t_all = np.zeros(3), 0.0
    for i in range(n + warm):
        t0 = time.perf_counter()
        learner.act(obs[i], src, 1.0, out=out, std=std)
        t1 = time.perf_counter()
        learner.add_transitions(obs[i], out, rew, obs[i + 1], done)
        t2 = time.perf_counter()
        learner.train_step_logged((rng.random_sample((S, B)) * rings[0]._size).astype(np.int64))
        t3 = time.perf_counter()
        if i >= warm:
            parts += (t1 - t0, t2 - t1, t3 - t2)
            t_all += t3 - t0
    torch.cuda.synchronize()
    us = parts / n * 1e6
    it = t_all / n * 1e6
    return {"members": S, "act_us": round(us[0], 1), "insert_us": round(us[1], 1), "step_us": round(us[2], 1),
            "iteration_us": round(it, 1), "member_env_steps_per_s": round(S * 1e6 / it)}


def single_body(Sd, A, L, n, warm):
    """tools/online_step_rate.py's body with a dropout actor acting in training mode (stock torch: GaussianPolicy.act
    has no engine kernel for active dropout)."""
    torch.manual_seed(0)
    q, v = J.TwinQ(Sd, A, 256, L), J.ValueFunction(Sd, 256, L)
    actor = J.GaussianPolicy(Sd, A, 1.0, 256, L, dropout=P)
    tr = J.ImplicitQLearning(1.0, actor, torch.optim.Adam(actor.parameters(), lr=3e-4), q, torch.optim.Adam(q.parameters(), lr=3e-4),
                             v, torch.optim.Adam(v.parameters(), lr=3e-4), device="cuda")
    rb = J.ReplayBuffer(Sd, A, 200_000, "cuda")
    with contextlib.redirect_stdout(io.StringIO()):
        rb.load_d4rl_dataset(synthetic_dataset(100_000, Sd, A, 0))
    actor.train()
    obs = np.random.RandomState(1).randn(n + warm + 1, Sd).astype(np.float32)
    np.random.seed(0)
    parts, t_all = np.zeros(4), 0.0
    for i in range(n + warm):
        t0 = time.perf_counter()
        a = actor.act(obs[i], "cuda")
        t1 = time.perf_counter()
        rb.add_transition(obs[i], a, 1.0, obs[i + 1], False)
        t2 = time.perf_counter()
        batch = rb.sample(B)
        t3 = time.perf_counter()
        tr.train(batch)
        t4 = time.perf_counter()
        if i >= warm:
            parts += (t1 - t0, t2 - t1, t3 - t2, t4 - t3)
            t_all += t4 - t0
    us = parts / n * 1e6
    return {"act_us": round(us[0], 1), "add_transition_us": round(us[1], 1), "sample_us": round(us[2], 1),
            "train_us": round(us[3], 1), "iteration_us": round(t_all / n * 1e6, 1)}


def loop(S, off, on, eval_freq, n_episodes):
    from ensemble_online_rate import ToyEnv  # noqa: E402  (tools/ is on sys.path as the script's directory)
    from jsrl_corl_b200.jsrl_utils import JsrlTrainConfig
    from jsrl_corl_b200.jsrl_w_iql import ensemble_train_loop

    cfgs = [JsrlTrainConfig(device="cuda", env="Toy-v0", seed=m, eval_freq=eval_freq, n_episodes=n_episodes, offline_iterations=off,
                            online_iterations=on, batch_size=B, n_curriculum_stages=3, rolling_mean_n=1, tolerance=0.1 + 0.01 * m,
                            actor_dropout=P)
            for m in range(S)]
    rb = ReplayBuffer(3, 2, 20_000, "cuda")
    with contextlib.redirect_stdout(io.StringIO()):
        rb.load_d4rl_dataset(synthetic_dataset(20_000, 3, 2, 0))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        learner, _, _ = ensemble_train_loop(cfgs, [ToyEnv(m) for m in range(S)], [ToyEnv(1000 + m) for m in range(S)], rb, 3, 2,
                                            1.0, ToyEnv.T, philox_act_dropout=True)
        torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    return {"members": S, "actor_dropout": P, "offline_iterations": off, "online_iterations": on, "eval_freq": eval_freq,
            "n_episodes": n_episodes, "wall_s": round(wall, 2), "member_online_env_steps": S * on,
            "learner_dropout_acts": int(learner.engine.act_steps.sum()), "member_updates_per_s": round(S * (off + on - B) / wall)}


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="short windows (a functional run, not a measurement)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("act_dropout_rate.py measures on the GPU; no CUDA device found")
    from ensemble_online_rate import gpu_info  # noqa: E402

    n, warm = (50, 10) if args.quick else (2000, 200)
    res = {"card": gpu_info(), "actor_dropout": P, "batch_size": B, "calls": n, "warmup_calls": warm,
           "timer": "host perf_counter; act_alone: median per call after a device synchronise; bodies: mean per iteration",
           "act_alone": {}, "online_body": {}}
    for name, (Sd, A, L) in SHAPES.items():
        res["act_alone"][name] = [act_alone(S, Sd, A, L, n, warm) for S in (1, 8, 64)]
        print(name, json.dumps(res["act_alone"][name]), flush=True)
    Sd, A, L = SHAPES["pen_gauss_2x256"]
    single = single_body(Sd, A, L, n, warm)
    rows = [body(S, Sd, A, L, n, warm) for S in (1, 8, 64)]
    for r in rows:
        r["speedup_vs_sequential_single_loops"] = round(r["members"] * single["iteration_us"] / r["iteration_us"], 2)
    res["online_body"]["pen_gauss_2x256"] = {"single_learner_body_torch_dropout_act": single, "ensemble_body_code5": rows}
    print(json.dumps(res["online_body"]), flush=True)
    res["ensemble_train_loop"] = [loop(S, 300 if args.quick else 500, 300 if args.quick else 3000, 300 if args.quick else 1000, 2)
                                  for S in (8, 64)]
    print(json.dumps(res["ensemble_train_loop"]), flush=True)
    res["card_after"] = gpu_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))
