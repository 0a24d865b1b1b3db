#!/usr/bin/env python
"""us per iteration of the ENSEMBLE online loop body as the host sees it, without the env: one act launch for every
member (IQLEnsemble.act: half the members on their Gaussian learner's distribution, half on their guide), one ring
insert launch (add_transitions) and one logged update (train_step_logged) on host-drawn indices.  Observations are
synthetic, as in tools/online_step_rate.py, whose single-learner body is measured in the same run: S sequential
single-learner loops cost S times that.  Then ensemble_train_loop end to end on a vectorised toy env, evaluations
included.

    python tools/ensemble_online_rate.py [--out profiles/r04_ensemble_online.json] [--quick]
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from jsrl_corl_b200 import IQLEnsemble, ReplayBuffer
from jsrl_corl_b200.synthetic import synthetic_dataset

B = 256


def body(S, Sd, A, L, n, warm, ring=10_000):
    learner = IQLEnsemble(S, Sd, A, 256, L, B, seeds=list(range(S)), max_steps_per_call=1)
    guide = IQLEnsemble(S, Sd, A, 256, L, B, seeds=list(range(100, 100 + S)), max_steps_per_call=1)
    learner.set_guide(guide)
    rings = [ReplayBuffer(Sd, A, ring, "cuda") for _ in range(S)]
    learner.bind_replay(rings)
    rng = np.random.RandomState(1)
    obs = rng.randn(n + warm + 1, S, Sd).astype(np.float32)
    src = np.where(np.arange(S) % 2 == 0, 2, 3).astype(np.int8)  # learner distribution / guide
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
        high = rings[0]._size
        learner.train_step_logged((rng.random_sample((S, B)) * high).astype(np.int64))
        t3 = time.perf_counter()
        if i >= warm:
            parts += (t1 - t0, t2 - t1, t3 - t2)
            t_all += t3 - t0
    torch.cuda.synchronize()
    us = parts / n * 1e6
    it = t_all / n * 1e6
    return {"members": S, "act_us": round(us[0], 1), "insert_us": round(us[1], 1), "step_us": round(us[2], 1),
            "iteration_us": round(it, 1), "member_env_steps_per_s": round(S * 1e6 / it)}


class ToyEnv:
    """gym-style 4-tuple env: 3-dim state (x, y, t/T), 2-dim action, reward = -|pos|, T = 100 steps."""
    T = 100

    def __init__(self, seed):
        self.rng = np.random.RandomState(seed)
        self.spec = type("Spec", (), {"id": "Toy-v0"})()

    def seed(self, s):
        self.rng = np.random.RandomState(s)

    def reset(self):
        self.pos, self.t = self.rng.uniform(-1, 1, 2), 0
        return np.array([self.pos[0], self.pos[1], 0.0], np.float32)

    def step(self, a):
        self.pos = np.clip(self.pos + 0.1 * np.asarray(a, np.float64)[:2], -2, 2)
        self.t += 1
        return np.array([self.pos[0], self.pos[1], self.t / self.T], np.float32), float(-np.linalg.norm(self.pos)), self.t >= self.T, {}


def loop(S, off, on, eval_freq, n_episodes):
    from jsrl_corl_b200.jsrl_utils import JsrlTrainConfig
    from jsrl_corl_b200.jsrl_w_iql import ensemble_train_loop

    cfgs = [JsrlTrainConfig(device="cuda", env="Toy-v0", seed=m, eval_freq=eval_freq, n_episodes=n_episodes, offline_iterations=off,
                            online_iterations=on, batch_size=B, n_curriculum_stages=3, rolling_mean_n=1, tolerance=0.1 + 0.01 * m)
            for m in range(S)]
    data = synthetic_dataset(20_000, 3, 2, 0)
    rb = ReplayBuffer(3, 2, 20_000, "cuda")
    with contextlib.redirect_stdout(io.StringIO()):
        rb.load_d4rl_dataset(data)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ensemble_train_loop(cfgs, [ToyEnv(m) for m in range(S)], [ToyEnv(1000 + m) for m in range(S)], rb, 3, 2, 1.0, ToyEnv.T)
        torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    eval_steps = S * ((off + on) // eval_freq) * n_episodes * ToyEnv.T + S * n_episodes * ToyEnv.T  # + guide-only probe
    return {"members": S, "offline_iterations": off, "online_iterations": on, "eval_freq": eval_freq, "n_episodes": n_episodes,
            "wall_s": round(wall, 2), "member_online_env_steps": S * on, "member_eval_env_steps": eval_steps,
            "member_updates_per_s": round(S * (off + on - B) / wall)}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as exc:  # the measurement still stands; the card is then named by torch only
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unknown ({exc})"}


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="short windows (a functional run, not a measurement)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ensemble_online_rate.py measures on the GPU; no CUDA device found")
    n, warm = (50, 10) if args.quick else (2000, 200)
    from online_step_rate import run as single_run  # noqa: E402  (tools/ is on sys.path as the script's directory)

    res = {"card": gpu_info(), "batch_size": B, "online_ring_rows": 10_000, "timer": "host perf_counter per iteration",
           "shapes": {}}
    for name, (Sd, A, L) in {"halfcheetah_gauss_2x256": (17, 6, 2), "antmaze_gauss_3x256": (29, 8, 3)}.items():
        single = single_run(Sd, A, L, False, n=n, warm=warm)
        rows = [body(S, Sd, A, L, n, warm) for S in (1, 8, 64)]
        for r in rows:
            r["speedup_vs_sequential_single_loops"] = round(r["members"] * single["iteration_us"] / r["iteration_us"], 2)
        res["shapes"][name] = {"single_learner_body": single, "ensemble_body": rows}
        print(name, json.dumps(res["shapes"][name]), flush=True)
    res["ensemble_train_loop"] = [loop(S, 500 if not args.quick else 300, 3000 if not args.quick else 300, 1000 if not args.quick else 300, 2)
                                  for S in (8, 64)]
    print(json.dumps(res["ensemble_train_loop"]), flush=True)
    res["card_after"] = gpu_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))
