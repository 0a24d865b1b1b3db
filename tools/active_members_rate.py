"""Cost of retired members (iql_set_active_members) on the GPU.

1. Member-steps/s of a 64-member halfcheetah-shaped engine (TF32, Philox sampling, K = 50 per call) with 64, 32, 16,
   8, 4 and 1 members active, each against a fresh engine of that many members; the two alternate, median / min / max
   over the rounds.
2. Host time of one set_active call at 64 members (tensor maps re-encoded).
3. An ASHA search end to end: 64 members, reduction factor 4, the offline phase on a toy env with one evaluation per
   rung step, with and without the scheduler: wall time and member-steps spent.

    python tools/active_members_rate.py [--rounds 5] [--out profiles/r06_active_members.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

from jsrl_corl_b200 import IQLEnsemble, ReplayBuffer  # noqa: E402
from jsrl_corl_b200.asha import ASHAScheduler  # noqa: E402
from jsrl_corl_b200.synthetic import synthetic_dataset  # noqa: E402

S_DIM, A_DIM, H, B, K = 17, 6, 256, 256, 50


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def stats(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs)), "n": len(xs)}


def timed_calls(ens, calls):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(calls):
        ens.train_steps(K)
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def engine_rates(rounds, calls):
    rb = ReplayBuffer(S_DIM, A_DIM, 200_000, "cuda")
    rb.load_d4rl_dataset(synthetic_dataset(200_000, S_DIM, A_DIM, 0))
    counts = [64, 32, 16, 8, 4, 1]
    big = IQLEnsemble(64, S_DIM, A_DIM, H, 2, B, max_steps_per_call=K)
    big.bind_replay(rb)
    fresh = {}
    for n in counts:
        fresh[n] = IQLEnsemble(n, S_DIM, A_DIM, H, 2, B, max_steps_per_call=K)
        fresh[n].bind_replay(rb)
        timed_calls(fresh[n], 1)  # graph capture, module load
    res = {n: {"retired": [], "fresh": []} for n in counts}
    paths = {}
    for r in range(rounds):
        for n in counts:
            big.engine.set_active(range(n))
            timed_calls(big, 1)  # the set change dropped the graphs: capture outside the timed window
            paths[n] = {"retired": dict(big.engine.paths), "fresh": dict(fresh[n].engine.paths)}
            order = ("retired", "fresh") if r % 2 == 0 else ("fresh", "retired")
            for which in order:
                dt = timed_calls(big if which == "retired" else fresh[n], calls)
                res[n][which].append(n * K * calls / dt)
    out = []
    for n in counts:
        ret, fr = stats(res[n]["retired"]), stats(res[n]["fresh"])
        out.append({"active": n, "member_steps_per_s_retired": ret, "member_steps_per_s_fresh": fr,
                    "retired_over_fresh": ret["median"] / fr["median"], "paths": paths[n]})
        print(json.dumps(out[-1]), flush=True)
    # 2. host time of set_active at 64 members
    host = {"to_32": [], "to_64": []}
    for _ in range(20):
        for key, n in (("to_32", 32), ("to_64", 64)):
            t0 = time.perf_counter()
            big.engine.set_active(range(n))
            host[key].append((time.perf_counter() - t0) * 1e3)
    set_active_ms = {k: stats(v) for k, v in host.items()}
    print(json.dumps({"set_active_host_ms": set_active_ms}), flush=True)
    return out, set_active_ms


class ToyEnv:
    """3-dim state, 2-dim action, reward -|pos|, 20 steps."""
    T = 20

    def __init__(self, seed=0):
        self.rng = np.random.RandomState(seed)
        self.spec = type("Spec", (), {"id": "Point-v0"})()

    def seed(self, s):
        self.rng = np.random.RandomState(s)

    def reset(self):
        self.pos = self.rng.uniform(-1, 1, 2)
        self.t = 0
        return np.array([self.pos[0], self.pos[1], 0.0], dtype=np.float32)

    def step(self, action):
        self.pos = np.clip(self.pos + 0.1 * np.asarray(action, dtype=np.float64).reshape(-1)[:2], -2, 2)
        self.t += 1
        return np.array([self.pos[0], self.pos[1], self.t / self.T], dtype=np.float32), float(-np.linalg.norm(self.pos)), \
            self.t >= self.T, {}


def asha_search(S, evals, eval_freq, rf):
    from jsrl_corl_b200.jsrl_utils import JsrlTrainConfig
    from jsrl_corl_b200.jsrl_w_iql import ensemble_train_loop

    rng = np.random.RandomState(1)
    n = 20_000
    data = {"observations": rng.uniform(-1, 1, (n, 3)).astype(np.float32), "actions": rng.uniform(-1, 1, (n, 2)).astype(np.float32),
            "rewards": rng.uniform(-1, 0, n).astype(np.float32), "next_observations": rng.uniform(-1, 1, (n, 3)).astype(np.float32),
            "terminals": np.zeros(n, bool)}
    rbs = []  # new_online_buffer=False (every offline step trains) asks for one buffer per member
    for _ in range(S):
        rbs.append(ReplayBuffer(3, 2, n, "cuda"))
        rbs[-1].load_d4rl_dataset(data)
    out = {}
    for label, sched in (("no_scheduler", None), ("asha", ASHAScheduler(max_t=evals, grace_period=1, reduction_factor=rf))):
        cfgs = [JsrlTrainConfig(device="cuda", env="Point-v0", seed=m, eval_freq=eval_freq, n_episodes=1,
                                offline_iterations=evals * eval_freq, online_iterations=0, batch_size=B,
                                new_online_buffer=False, beta=0.5 + 0.25 * (m % 16), iql_tau=0.6 + 0.005 * m)
                for m in range(S)]
        steps = [0] * S

        def log(m, d, step):
            if "offline_iter" in d:
                steps[m] += 1
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ensemble_train_loop(cfgs, [ToyEnv(m) for m in range(S)], [ToyEnv(1000 + m) for m in range(S)], rbs, 3, 2, 1.0,
                            ToyEnv.T, log=log, scheduler=sched)
        torch.cuda.synchronize()
        out[label] = {"wall_s": time.perf_counter() - t0, "member_steps": int(sum(steps)),
                      "stopped": None if sched is None else len(sched.stopped)}
        print(json.dumps({label: out[label]}), flush=True)
    # rung arithmetic: S / rf^k members reach rung k; a member that stops at rung k has run milestone_k reports
    ms = [rf ** k for k in range(int(np.floor(np.log(evals) / np.log(rf))) + 1)]
    reach = [S // rf ** k for k in range(len(ms))]
    units = sum(reach[k] * (ms[k] - (ms[k - 1] if k else 0)) for k in range(len(ms))) + reach[-1] * (evals - ms[-1])
    out["rung_arithmetic_member_evals"] = {"predicted": units, "without_scheduler": S * evals,
                                           "predicted_ratio": S * evals / units}
    out["measured_ratio_member_steps"] = out["no_scheduler"]["member_steps"] / out["asha"]["member_steps"]
    out["measured_ratio_wall"] = out["no_scheduler"]["wall_s"] / out["asha"]["wall_s"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--calls", type=int, default=4, help="timed K-step calls per configuration and round")
    ap.add_argument("--evals", type=int, default=64)
    ap.add_argument("--eval-freq", type=int, default=20)
    ap.add_argument("--out", default="profiles/r06_active_members.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a GPU")
    res = {"gpu": gpu_info(), "shape": "halfcheetah 17/6, 2x256, batch 256, tf32, philox", "K": K}
    res["engine"], res["set_active_host_ms"] = engine_rates(args.rounds, args.calls)
    res["asha_search"] = asha_search(64, args.evals, args.eval_freq, 4)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "asha": res["asha_search"]}))


if __name__ == "__main__":
    main()
