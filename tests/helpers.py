"""Shared helpers for the parity tests (golden fixtures, oracle construction)."""
import hashlib
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


class Golden:
    def __init__(self, name):
        self.z = np.load(os.path.join(GOLDEN, name + ".npz"))
        self.meta = dict(zip([str(k) for k in self.z["meta_keys"]], [float(v) for v in self.z["meta_vals"]]))
        for k in ("S", "A", "H", "L", "det", "B", "steps", "n_rows", "seed", "idx_seed", "antmaze", "max_steps"):
            self.meta[k] = int(self.meta[k])
        self.losses = self.z["losses"]

    def tree(self, prefix):
        """{"qf": {...}, "vf": {...}, "actor": {...}[, "q_target"]} of arrays stored under prefix/."""
        out = {}
        for key in self.z.files:
            if key.startswith(prefix + "/"):
                parts = key[len(prefix) + 1:].split("/", 1)
                if len(parts) == 2 and parts[0] in ("qf", "vf", "actor", "q_target"):
                    out.setdefault(parts[0], {})[parts[1]] = self.z[key]
        return out

    def opt(self, prefix):
        """{"qf": {param: (exp_avg, exp_avg_sq)}} stored under prefix/opt/."""
        out = {}
        pre = prefix + "/opt/"
        for key in self.z.files:
            if key.startswith(pre) and key.endswith("/exp_avg"):
                grp, rest = key[len(pre):].split("/", 1)
                name = rest[: -len("/exp_avg")]
                out.setdefault(grp, {})[name] = (self.z[key], self.z[key[: -len("exp_avg")] + "exp_avg_sq"])
        return out

    def indices(self):
        """[steps, B] int64 -- stored, or regenerated from numpy's legacy MT19937 stream and checksum-verified."""
        m = self.meta
        if "indices" in self.z.files:
            idx = self.z["indices"].astype(np.int64)
        else:
            rs = np.random.RandomState(m["idx_seed"])
            idx = np.stack([rs.randint(0, m["n_rows"], size=m["B"]) for _ in range(m["steps"])]).astype(np.int64)
        assert hashlib.sha256(idx.tobytes()).hexdigest() == str(self.z["indices_sha256"])
        return idx

    def dropout_masks(self):
        m = self.meta
        bits = np.unpackbits(self.z["dropout_masks"])[: m["steps"] * m["L"] * m["B"] * m["H"]]
        return bits.reshape(m["steps"], m["L"], m["B"], m["H"]).astype(np.uint8)

    def dataset(self):
        from oracle.iql_numpy import synthetic_dataset

        m = self.meta
        return synthetic_dataset(m["n_rows"], m["S"], m["A"], 0, antmaze_rewards=bool(m["antmaze"]))

    def init_tree(self):
        """Initial weights: stored, or regenerated from torch.manual_seed and checksum-verified."""
        if "init_sha256" not in self.z.files:
            return self.tree("init")
        from jsrl_corl_b200.ensemble import reference_init

        m = self.meta
        q, v, actor = reference_init(m["seed"], m["S"], m["A"], m["H"], m["L"], bool(m["det"]), self.meta["dropout"])
        tree = {g: {k: t.detach().numpy().copy() for k, t in mod.state_dict().items()}
                for g, mod in (("qf", q), ("vf", v), ("actor", actor))}
        h = hashlib.sha256()
        flat = {f"init/{g}/{k}": a for g, d in tree.items() for k, a in d.items()}
        for k in sorted(flat):
            h.update(flat[k].tobytes())
        assert h.hexdigest() == str(self.z["init_sha256"]), "regenerated init weights differ from the reference's"
        return tree

    def oracle_config(self):
        from oracle.iql_numpy import OracleConfig

        m = self.meta
        return OracleConfig(m["S"], m["A"], m["H"], m["L"], bool(m["det"]), m["dropout"], m["iql_tau"], m["beta"],
                            m["discount"], m["tau"], m["lr"], m["lr"], m["lr"], m["max_steps"])


def oracle_from_state(cfg, tree, moments=None, steps=None, sched_epoch=0, total_it=0, actor_lr=None, dtype=np.float32):
    """A NumpyIQL that continues a learner from a given state rather than from its initial one.

    tree: {"qf", "vf", "actor"[, "q_target"]} weights; moments: {grp: {name: (exp_avg, exp_avg_sq)}}; steps: Adam step
    counts {"qf", "vf", "actor"}; sched_epoch: CosineAnnealingLR.last_epoch.  The current actor lr is the closed form of
    the schedule at that epoch unless `actor_lr` is given (e.g. the value a reference run stored)."""
    from oracle.iql_numpy import NumpyIQL, cosine_closed_form_lr

    orc = NumpyIQL(cfg, tree, dtype)
    steps = steps or {}
    for grp, o in (("qf", orc.q_opt), ("vf", orc.v_opt), ("actor", orc.a_opt)):
        o.step_count = int(steps.get(grp, 0))
        for name, (m, v) in (moments or {}).get(grp, {}).items():
            o.exp_avg[name][...] = m
            o.exp_avg_sq[name][...] = v
    orc.sched_epoch = int(sched_epoch)
    if actor_lr is not None:
        orc.a_opt.lr = float(actor_lr)
    elif cfg.max_steps is not None:
        orc.a_opt.lr = cosine_closed_form_lr(cfg.actor_lr, orc.sched_epoch, cfg.max_steps, cfg.lr_eta_min)
    orc.total_it = int(total_it)
    return orc


def batch_from(data, idx):
    return [data["observations"][idx], data["actions"][idx], data["rewards"][idx][:, None],
            data["next_observations"][idx], data["terminals"][idx].astype(np.float32)[:, None]]


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def tree_max_rel(tree_a, tree_b, groups=("qf", "vf", "actor")):
    worst, where = 0.0, None
    for g in groups:
        for k, b in tree_b[g].items():
            if np.linalg.norm(b) == 0:
                continue
            e = rel_err(tree_a[g][k], b)
            if e > worst:
                worst, where = e, f"{g}/{k}"
    return worst, where


def network_errors_vs_floor(g, state, step_prefix):
    """For each network: (relative error of the concatenated parameter vector vs the
    reference's fp32 weights, the reference's own fp32-vs-fp64 divergence of that vector)."""
    final = g.tree(step_prefix)
    out = {}
    for grp in ("qf", "vf", "actor"):
        num = den = floor = 0.0
        for k, ref in final[grp].items():
            ref = ref.astype(np.float64)
            num += float(np.sum((np.asarray(state[grp][k], dtype=np.float64) - ref) ** 2))
            den += float(np.sum(ref ** 2))
            floor += (float(g.z[f"noise/{grp}/{k}"]) ** 2) * float(np.sum(ref ** 2))
        out[grp] = (np.sqrt(num / den), np.sqrt(floor / den))
    return out


class LateSnapshot(Golden):
    """tests/golden/*_late_<at>.npz (oracle/gen_golden.py::late_snapshot): the full reference state after `at` steps,
    the batch indices / losses of step at + 1 and every 16th element of the post-step weights and target."""

    def __init__(self, name):
        super().__init__(name)
        self.at = self.meta["steps"] - 1
        self.pre = f"step{self.at}"
        self.next_indices = self.z["next_indices"].astype(np.int64)
        self.next_losses = self.losses[-1].astype(np.float64)

    def post_sampled(self):
        """{"qf"/"vf"/"actor"/"q_target": {name: values[::16]}} after step at + 1."""
        out, pre = {}, f"step{self.at + 1}/"
        for key in self.z.files:
            if key.startswith(pre) and key.endswith("@16"):
                grp, name = key[len(pre):-3].split("/", 1)
                out.setdefault(grp, {})[name] = self.z[key]
        return out

    def load_into_oracle(self, dtype=np.float32):
        return oracle_from_state(self.oracle_config(), self.tree(self.pre), self.opt(self.pre),
                                 {"qf": self.at, "vf": self.at, "actor": self.at}, int(self.z[f"{self.pre}/sched_epoch"]),
                                 self.at, actor_lr=float(self.z[f"{self.pre}/actor_lr"]), dtype=dtype)
