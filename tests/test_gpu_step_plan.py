"""The update step's launch sequence, pinned per shape: what `profile_step` reports (labels, flops, bytes), how many
launches each entry point makes, and the launch DAG of a two-step call (kernel nodes and their edges).

The expected values in golden/step_plan.json were recorded on a B200 (148 SMs: the grids of the persistent kernels follow
the SM count).  A change to how the step is assembled on the host must leave all three as they are; a change that means
to alter the step re-records them knowingly.

The shapes cover every branch of the step's assembly: the six bench.py workloads, the three step paths, FP32 math,
TF32 outside the tcgen05 shapes, the row-split output-layer backward and the K-split input-layer weight gradient, the
action widths at the output-layer kernel boundaries, the generic input layer, a depth past the fused forward, an engine
with a subset of its members active, and the chained backward with keep_grads."""
import json
import os
import re
import tempfile
from collections import namedtuple

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "step_plan.json")
N_ROWS = 3000

Shape = namedtuple("Shape", "id S A H L B det members dropout math step_path active keep_grads",
                   defaults=(256, 2, 256, False, 8, 0.0, "tf32", "auto", None, False))

SHAPES = [
    # bench.py workloads
    Shape("halfcheetah_ens64", 17, 6, members=64),
    Shape("hopper_ens64", 11, 3, det=True, members=64),
    Shape("hopper_single", 11, 3, det=True, members=1),
    Shape("antmaze_jsrl", 29, 8, L=3, members=1),
    Shape("pen_sweep256", 45, 24, members=256, dropout=0.1),
    Shape("stress_4x1024", 11, 3, H=1024, L=4, B=4096, det=True, members=1),
    # step paths at 8 members, 2x256
    Shape("path_phases", 17, 6, step_path="phases"),
    Shape("path_chain", 17, 6, step_path="chain"),
    Shape("path_chain_grads", 17, 6, step_path="chain_grads"),
    Shape("fp32_math", 17, 6, members=2, math="fp32"),
    Shape("tf32_b200", 17, 6, B=200, members=2),
    Shape("row_split_b4096", 11, 3, B=4096, det=True, members=1),
    Shape("k_split_b2048", 17, 6, B=2048, members=4),
    Shape("a9", 11, 9, members=2),
    Shape("a24", 11, 24, members=2),
    Shape("a33", 11, 33, members=2),
    Shape("a65_det", 11, 65, det=True, members=2),
    Shape("k0_73", 67, 6, members=2),
    Shape("l5", 11, 3, L=5, members=2),
    Shape("active_3_of_12", 17, 6, members=12, active=(1, 5, 10)),
    Shape("chain_keep_grads", 17, 6, step_path="chain", keep_grads=True),
]


def _ensemble(sh):
    from jsrl_corl_b200 import IQLEnsemble, ReplayBuffer
    from oracle.iql_numpy import synthetic_dataset

    rb = ReplayBuffer(sh.S, sh.A, N_ROWS, "cuda")
    rb.load_d4rl_dataset(synthetic_dataset(N_ROWS, sh.S, sh.A, 4))
    ens = IQLEnsemble(sh.members, sh.S, sh.A, sh.H, sh.L, sh.B, deterministic=sh.det, actor_dropout=sh.dropout,
                      math_mode=sh.math, seeds=list(range(sh.members)), max_steps_per_call=4, step_path=sh.step_path,
                      init=False)
    ens.bind_replay(rb)
    if sh.active is not None:
        ens.engine.set_active(sh.active)
    if sh.keep_grads:
        ens.engine.keep_grads(True)
    return ens, rb


def _indices(sh, k):
    return torch.from_numpy(np.random.RandomState(k).randint(0, N_ROWS, size=(sh.members, k, sh.B)).astype(np.int64))


def launch_counts(ens, sh):
    """last_launch_count after an eager K = 1 call, K = 3 graph calls (philox, indices) and a host step."""
    eng = ens.engine
    out = {}
    eng.train_steps(1)
    out["eager_k1"] = eng.last_launch_count()
    eng.train_steps(3)
    out["graph_k3_philox"] = eng.last_launch_count()
    eng.train_steps(3, mode="indices", indices=_indices(sh, 3))
    out["graph_k3_indices"] = eng.last_launch_count()
    idx = np.ascontiguousarray(_indices(sh, 1).numpy()[:, 0])
    eng.host_step(host_indices=idx.ctypes.data)
    out["host_step"] = eng.last_launch_count()
    torch.cuda.synchronize()
    return out


_NODE = re.compile(r'"graph_\d+_node_(\d+)"\[[^\]]*?label="\{(\w+)(.*?)\}"\];', re.S)
_LAUNCH = re.compile(r"\|\s*(\w+)\\<\\<\\<(.*?)\\>\\>\\>")
_EDGE = re.compile(r'"graph_\d+_node_(\d+)" -> "graph_\d+_node_(\d+)"\s*\[headlabel=(\d+)\]')


def parse_dot(text):
    """The nodes of a cudaGraphDebugDotPrint dump by node id -- a kernel node as its function name (anonymous-namespace
    hashes removed) and its <<<grid, block, dynamic shared memory>>>, any other node as its type -- and the edges as
    (from, to, dependency port).  Handles, addresses and kernel arguments are dropped."""
    nodes = {}
    for m in _NODE.finditer(text):
        if m.group(2) == "KERNEL":
            k = _LAUNCH.search(m.group(3))
            name = re.sub(r"_GLOBAL__N__[0-9a-f]{8}_(\d+_\w+?_cu)_[0-9a-f]{8}", r"_GLOBAL__N__\1", k.group(1))
            nodes[int(m.group(1))] = [name, k.group(2).replace("\\", "")]
        else:
            nodes[int(m.group(1))] = [m.group(2)]
    edges = sorted([int(a), int(b), int(port)] for a, b, port in _EDGE.findall(text))
    return {"nodes": [nodes[i] for i in sorted(nodes)], "edges": edges}


def capture_two_steps(sh, dot_path):
    """train_steps(2) of an engine built with IQL_B200_GRAPHS=0, captured into a torch CUDA graph after one warm-up call;
    writes the graph's debug dump to dot_path."""
    old = os.environ.get("IQL_B200_GRAPHS")
    os.environ["IQL_B200_GRAPHS"] = "0"
    try:
        ens, rb = _ensemble(sh)
    finally:
        if old is None:
            del os.environ["IQL_B200_GRAPHS"]
        else:
            os.environ["IQL_B200_GRAPHS"] = old
    eng = ens.engine
    out = torch.empty(sh.members, 2, 3, dtype=torch.float32, device=eng.device)
    eng.train_steps(2, out=out)  # uploads every table, scalar and attribute before the capture
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph(keep_graph=True)  # the dump needs the captured graph
    g.enable_debug_mode()
    with torch.cuda.graph(g, stream=eng.stream):
        eng.train_steps(2, out=out)
    g.debug_dump(dot_path)
    torch.cuda.synchronize()
    del g, ens, rb


def observe(sh, dot_path):
    ens, rb = _ensemble(sh)
    prof = [[p["label"], p["flops"], p["bytes"]] for p in ens.engine.profile_step(reps=1)]
    counts = launch_counts(ens, sh)
    del ens, rb
    capture_two_steps(sh, dot_path)
    with open(dot_path) as f:
        dag = parse_dot(f.read())
    return {"profile": prof, "launches": counts, "dag": dag}


@pytest.fixture(scope="module")
def golden():
    with open(GOLDEN) as f:
        return json.load(f)


@pytest.mark.parametrize("sh", SHAPES, ids=lambda s: s.id)
def test_step_plan_is_pinned(sh, golden):
    exp = golden[sh.id]
    with tempfile.TemporaryDirectory() as tmp:
        got = observe(sh, os.path.join(tmp, "step.dot"))
    assert [p[0] for p in got["profile"]] == [p[0] for p in exp["profile"]]
    for (label, fl, by), (_, efl, eby) in zip(got["profile"], exp["profile"]):
        assert fl == pytest.approx(efl, rel=1e-12, abs=0.0), label
        assert by == pytest.approx(eby, rel=1e-12, abs=0.0), label
    assert got["launches"] == exp["launches"]
    assert len(got["dag"]["nodes"]) > 0
    assert got["dag"]["nodes"] == exp["dag"]["nodes"]
    assert got["dag"]["edges"] == exp["dag"]["edges"]
