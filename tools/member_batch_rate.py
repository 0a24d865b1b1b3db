#!/usr/bin/env python
"""Member-steps/s of a 64-member halfcheetah-shaped ensemble (obs 17, act 6, 2 x 256, TF32, Philox sampling, K steps
per graph launch) when its members train with different batch sizes:

  (a) uniform: every member at B = 256;
  (b) padded: one engine at B = 256, member batch sizes cycling {64, 128, 256} (iql_set_batch_sizes);
  (c) split: the same sweep as three engines, one per batch size, run one after another;
  (d) padded at B = 512 with sizes cycling {128, 256, 512}, and (e) its split counterpart;
  plus uniform B = 512 for reference.

Each engine's kernel path (tensor cores or the FP32 kernels, chained backward) is reported beside its number: a batch
of 64 is outside the tcgen05 kernels (batch % 128 != 0), so the split run's 64-row engine takes the FP32 path, while the
padded engine keeps every member on tcgen05.  Configurations are timed in alternation, `--rounds` times; the median is
reported.

    python tools/member_batch_rate.py [--out profiles/r05_member_batch.json] [--quick]
"""
import argparse
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

S_DIM, A_DIM, H, L, MEMBERS, N_ROWS = 17, 6, 256, 2, 64, 200_000


def cycle(values, n):
    return [values[m % len(values)] for m in range(n)]


class Run:
    """One engine of n members at engine batch B (member sizes `sizes`, None = all B), timed over `calls` x K steps."""

    def __init__(self, rb, n, B, sizes, K):
        self.ens = IQLEnsemble(n, S_DIM, A_DIM, H, L, B, seeds=list(range(n)), max_steps_per_call=K, batch_sizes=sizes)
        self.ens.bind_replay(rb)
        self.n, self.B, self.K = n, B, K
        self.ens.train_steps(K)  # capture + warm-up
        self.ens.train_steps(K)
        torch.cuda.synchronize()

    def seconds(self, calls):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(calls):
            self.ens.train_steps(self.K)
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    def path(self):
        p = self.ens.engine.paths
        return {"batch": self.B, "members": self.n, "tensor_cores": p["tensor_cores"],
                "chained_backward_grads": p["chained_backward_grads"]}


def split(rb, sizes, K):
    """One engine per distinct size, holding the members of that size."""
    return [Run(rb, sizes.count(b), b, None, K) for b in sorted(set(sizes))]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as exc:  # the measurement itself does not depend on it
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unknown ({exc})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=50, help="steps per call (K)")
    ap.add_argument("--calls", type=int, default=20, help="calls per timed window")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--quick", action="store_true")
    a = ap.parse_args()
    if a.quick:
        a.steps, a.calls, a.rounds = 10, 4, 2
    if not torch.cuda.is_available():
        raise SystemExit("member_batch_rate.py measures on a CUDA device; none is available")
    torch.manual_seed(0)
    rb = ReplayBuffer(S_DIM, A_DIM, N_ROWS, "cuda")
    rb.load_d4rl_dataset(synthetic_dataset(N_ROWS, S_DIM, A_DIM, 0))
    K = a.steps
    mix256, mix512 = cycle((64, 128, 256), MEMBERS), cycle((128, 256, 512), MEMBERS)
    configs = {
        "a_uniform_256": [Run(rb, MEMBERS, 256, None, K)],
        "b_padded_256": [Run(rb, MEMBERS, 256, mix256, K)],
        "c_split_64_128_256": split(rb, mix256, K),
        "uniform_512": [Run(rb, MEMBERS, 512, None, K)],
        "d_padded_512": [Run(rb, MEMBERS, 512, mix512, K)],
        "e_split_128_256_512": split(rb, mix512, K),
    }
    samples = {k: [] for k in configs}
    for _ in range(a.rounds):
        for name, runs in configs.items():
            sec = sum(r.seconds(a.calls) for r in runs)  # split: the engines one after another
            samples[name].append(MEMBERS * K * a.calls / sec)
    out = dict(gpu_info(), shape="halfcheetah 17/6, 2 x 256, tf32, Philox sampling", members=MEMBERS, steps_per_call=K,
               calls=a.calls, rounds=a.rounds, results={})
    for name, runs in configs.items():
        v = np.array(samples[name])
        out["results"][name] = {"member_steps_per_s": round(float(np.median(v))), "min": round(float(v.min())),
                                "max": round(float(v.max())), "engines": [r.path() for r in runs]}
    r = {k: v["member_steps_per_s"] for k, v in out["results"].items()}
    out["winner_b_vs_c"] = "padded" if r["b_padded_256"] > r["c_split_64_128_256"] else "split"
    out["winner_d_vs_e"] = "padded" if r["d_padded_512"] > r["e_split_128_256_512"] else "split"
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
