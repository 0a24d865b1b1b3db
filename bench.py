#!/usr/bin/env python
"""Headline benchmark: IQL gradient steps/sec, summed over ensemble members.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

One bench *step* = one fused engine call that runs ``inner`` IQL updates
(replay sample + V/Q/actor update + Polyak + LR schedule) for every one of the
S ensemble members resident on the GPU, i.e. ``S * inner`` gradient steps.
Default workload = BASELINE.json configs[2]: halfcheetah-medium-replay shape
(obs 17, act 6, 2x256 MLPs, Gaussian actor, batch 256), 64-member ensemble on a
1M-transition synthetic buffer, one B200.  Multi-GPU (torchrun) keeps S members
per GPU (weak scaling); members never exchange data -- the only collective is
the NCCL all-gather of the per-step loss scalars.

`--impl reference` times the UNMODIFIED reference classes (offline/iql.py, staged under
oracle/_ref by __graft_entry__.build()) on the host cores -- one member, all threads and one
thread, 1M-row buffer, a bounded number of steps -- and the same code with device="cuda"
(`torch_eager_b200`: what a user of the reference gets on this GPU today).

`--dump-outputs DIR` writes what the last timed step computed, as float32 .npy files: ``losses.npy`` (the [S, inner, 3]
losses the engine call returns), ``params.npy`` and ``target.npy`` (the parameter and Q-target arenas of all S members
after that call).  An array above 4 Mi elements is replaced by a fixed, seeded sample of 4 Mi of its flattened elements,
so a dump stays under 64 MB.  Inputs depend only on the arguments, so two builds run with the same arguments can be
compared file by file.  Multi-GPU runs dump rank 0's members.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: dict(S, A, H, L, B, det, dropout, members, beta, iql_tau, tau, antmaze)
    "halfcheetah_ens64": dict(S=17, A=6, H=256, L=2, B=256, det=False, dropout=0.0, members=64, beta=3.0, iql_tau=0.7,
                              tau=0.005, antmaze=False, desc="BASELINE configs[2]: halfcheetah-medium-replay shape, 64-seed ensemble"),
    "hopper_ens64": dict(S=11, A=3, H=256, L=2, B=256, det=True, dropout=0.0, members=64, beta=3.0, iql_tau=0.7,
                         tau=0.001, antmaze=False, desc="north_star target: hopper-medium shape, 64-seed ensemble"),
    "hopper_single": dict(S=11, A=3, H=256, L=2, B=256, det=True, dropout=0.0, members=1, beta=3.0, iql_tau=0.7,
                          tau=0.001, antmaze=False, desc="BASELINE configs[0]: hopper-medium shape, single seed"),
    "antmaze_jsrl": dict(S=29, A=8, H=256, L=3, B=256, det=False, dropout=0.0, members=1, beta=10.0, iql_tau=0.9,
                         tau=0.005, antmaze=True, desc="BASELINE configs[1]: antmaze-umaze shape, 3x256, single learner"),
    "pen_sweep256": dict(S=45, A=24, H=256, L=2, B=256, det=False, dropout=0.1, members=256, beta=3.0, iql_tau=0.8,
                         tau=0.005, antmaze=False, scaling="strong",
                         desc="BASELINE configs[3]: pen-human shape, dropout actor, 256-member sweep SPLIT over the GPUs"),
    "stress_4x1024": dict(S=11, A=3, H=1024, L=4, B=4096, det=True, dropout=0.0, members=1, beta=3.0, iql_tau=0.7,
                          tau=0.005, antmaze=False, desc="BASELINE configs[4]: batch 4096, 4x1024 MLPs, hopper shape"),
}
N_ROWS = 1_000_000


def flops_per_step(w):
    """GEMM FLOPs of one member-step (BASELINE.md section 4)."""
    S, A, H, L, B = w["S"], w["A"], w["H"], w["L"], w["B"]

    def fwd(i, o):
        return 2 * (i * H + (L - 1) * H * H + H * o)

    def bwd(i, o):
        return 2 * fwd(i, o) - 2 * i * H

    v, q, pi = (S, 1), (S + A, 1), (S, A)
    return B * (2 * fwd(*v) + 4 * fwd(*q) + fwd(*pi) + bwd(*v) + 2 * bwd(*q) + bwd(*pi))


def gather_bytes_per_step(w):
    return w["B"] * (2 * w["S"] + w["A"] + 2) * 4


DUMP_MAX_ELEMS = 1 << 22  # per array: three float32 arrays stay under 64 MB


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy in float32; one above DUMP_MAX_ELEMS becomes a seeded sample of its
    flattened elements (the same positions on every run with the same shape)."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float32)
        if a.size > DUMP_MAX_ELEMS:
            pick = np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))
            a = a.reshape(-1)[pick]
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _run_nvml(self):
        # in-process NVML: a sample every 25 ms (an nvidia-smi process per sample gave 3-7 samples in a 2 s region)
        import pynvml as N

        N.nvmlInit()
        h = N.nvmlDeviceGetHandleByIndex(self.index)
        mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
        get_reasons = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = [(0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap")]
        while not self._stop.is_set():
            r = int(get_reasons(h))
            self.rows.append([str(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)), str(mx), "0"] +
                             ["Active" if r & b else "Not Active" for b, _ in bits])
            self._stop.wait(0.025)

    def _run(self):
        try:
            self._run_nvml()
            return
        except Exception:
            pass
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


TF32_NOMINAL_TFLOPS = 1125.0  # B200 dense TF32 = half of the 2.25 PFLOP/s bf16 figure


def pinned_tf32_peak(torch, device):
    """The TF32 denominator is PINNED: profiles/tf32_peak.json (one measurement of cuBLAS TF32 8192^3 on this pool's
    B200, committed with its method and clocks).  Only when that file is absent is it measured live."""
    path = os.path.join(ROOT, "profiles", "tf32_peak.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        # burst figure (the higher, conservative denominator): the step's tcgen05 kernels run in short bursts between
        # HBM-bound launches, not under the sustained power cap of a 4 s GEMM loop (sustained is reported beside it)
        return float(d["tf32_tflops_burst"]), "pinned: profiles/tf32_peak.json burst (" + d.get("how", "") + ")"
    return measure_tf32_peak(torch, device), "cuBLAS TF32 8192^3 measured live (profiles/tf32_peak.json missing)"


def tf32_sustained():
    path = os.path.join(ROOT, "profiles", "tf32_peak.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get("tf32_tflops_sustained")
    return None


def measure_tf32_peak(torch, device):
    """cuBLAS TF32 8192^3 GEMM, sustained for ~1.5 s, same method as MEASURED_PEAKS.json uses for bf16
    (the file has no TF32 entry).  Library call used as a yardstick only."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device=device)
        b = torch.randn(n, n, device=device)
        for _ in range(3):
            a @ b
        torch.cuda.synchronize(device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 40
        e0.record()
        for _ in range(reps):
            a @ b
        e1.record()
        torch.cuda.synchronize(device)
        return 2.0 * n ** 3 * reps / (e0.elapsed_time(e1) * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


# ---------------------------------------------------------------------------
# Reference arm: the UNMODIFIED reference classes (algorithms/offline/iql.py, staged under oracle/_ref by
# __graft_entry__.build()) on the host cores -- and, as "what users get today", on the GPU in stock eager mode.
# Falls back to the numpy port of the oracle (kind "port") only when the staged files are missing.
# ---------------------------------------------------------------------------
def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def build_reference_trainer(w, device, n_rows, seed=0):
    """ReplayBuffer + ImplicitQLearning of the unmodified reference (offline/iql.py:125-184, 397-537) on `device`,
    built the way offline/iql.py:564-621 builds them (class-default Adam, TwinQ -> V -> policy order)."""
    import contextlib
    import io

    import torch

    from jsrl_corl_b200.synthetic import synthetic_dataset
    from oracle.ref_loader import load_reference_iql

    ref = load_reference_iql("offline")
    data = synthetic_dataset(n_rows, w["S"], w["A"], 0, antmaze_rewards=w["antmaze"])
    rb = ref.ReplayBuffer(w["S"], w["A"], n_rows, device)
    with contextlib.redirect_stdout(io.StringIO()):
        rb.load_d4rl_dataset(data)
    torch.manual_seed(seed)
    q = ref.TwinQ(w["S"], w["A"], hidden_dim=w["H"], n_hidden=w["L"]).to(device)
    v = ref.ValueFunction(w["S"], hidden_dim=w["H"], n_hidden=w["L"]).to(device)
    pol = ref.DeterministicPolicy if w["det"] else ref.GaussianPolicy
    actor = pol(w["S"], w["A"], 1.0, hidden_dim=w["H"], n_hidden=w["L"],
                dropout=w["dropout"] if w["dropout"] > 0 else None).to(device)
    trainer = ref.ImplicitQLearning(
        max_action=1.0, actor=actor, actor_optimizer=torch.optim.Adam(actor.parameters(), lr=3e-4),
        q_network=q, q_optimizer=torch.optim.Adam(q.parameters(), lr=3e-4), v_network=v,
        v_optimizer=torch.optim.Adam(v.parameters(), lr=3e-4), iql_tau=w["iql_tau"], beta=w["beta"],
        max_steps=1_000_000, discount=0.99, tau=w["tau"], device=device)
    return rb, trainer


def time_reference_loop(rb, trainer, B, device, steps, warmup, sync=None):
    """The reference's hot loop, verbatim (offline/iql.py:631-635): sample -> .to(device) -> train."""
    def one():
        batch = rb.sample(B)
        batch = [b.to(device) for b in batch]
        return trainer.train(batch)

    for _ in range(warmup):
        one()
    if sync:
        sync()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    if sync:
        sync()
    dt = time.perf_counter() - t0
    return steps / dt, dt


def reference_available():
    try:
        from oracle.ref_loader import reference_available as ra
        return ra()
    except Exception:
        return False


def cpu_reference_measurements(w, steps_all, steps_one, warmup, n_rows=N_ROWS):
    """steps/s of ONE member through the unmodified reference on the host: all cores, then one thread."""
    import torch

    cores = os.cpu_count() or 1
    rb, trainer = build_reference_trainer(w, "cpu", n_rows)
    prev = torch.get_num_threads()
    torch.set_num_threads(cores)  # torchrun pins OMP_NUM_THREADS=1 in the workers' environment; undo that for this arm
    sps_all, dt_all = time_reference_loop(rb, trainer, w["B"], "cpu", steps_all, warmup)
    used = torch.get_num_threads()
    torch.set_num_threads(1)
    sps_one, dt_one = time_reference_loop(rb, trainer, w["B"], "cpu", steps_one, min(warmup, 5))
    torch.set_num_threads(prev)
    return {"all": sps_all, "dt_all": dt_all, "one": sps_one, "dt_one": dt_one, "cores": used, "nproc": cores}


def torch_eager_b200(w, steps=300, warmup=30, n_rows=N_ROWS):
    """The unmodified reference with device="cuda": what a user of the reference gets on this B200 today."""
    import torch

    if not torch.cuda.is_available() or not reference_available():
        return None
    dev = "cuda"
    rb, trainer = build_reference_trainer(w, dev, n_rows)
    sps, dt = time_reference_loop(rb, trainer, w["B"], dev, steps, warmup, sync=torch.cuda.synchronize)
    del rb, trainer
    torch.cuda.empty_cache()
    return {"value": sps, "unit": "steps/s", "members": 1, "steps": steps,
            "what": "unmodified reference offline/iql.py classes, device='cuda', stock eager torch, sample()+train() loop"}


def cpu_port_steps_per_sec(w, steps, warmup, n_rows=200_000):
    """Fallback when the staged reference files are absent: the numpy port under oracle/ (kind "port")."""
    import numpy as np

    from jsrl_corl_b200.ensemble import reference_init
    from oracle.iql_numpy import NumpyIQL, OracleConfig, synthetic_dataset

    cores = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=cores)
        cores = max([p.get("num_threads", 1) for p in threadpool_info()] + [1])
    except Exception:
        pass
    data = synthetic_dataset(n_rows, w["S"], w["A"], 0, antmaze_rewards=w["antmaze"])
    q, v, actor = reference_init(0, w["S"], w["A"], w["H"], w["L"], w["det"], w["dropout"])
    init = {g: {k: t.detach().numpy().copy() for k, t in mod.state_dict().items()} for g, mod in (("qf", q), ("vf", v), ("actor", actor))}
    orc = NumpyIQL(OracleConfig(w["S"], w["A"], w["H"], w["L"], w["det"], w["dropout"], w["iql_tau"], w["beta"], 0.99,
                                w["tau"]), init, np.float32)
    rng = np.random.RandomState(0)
    keep = 1.0 - w["dropout"]

    def one():
        idx = np.random.randint(0, n_rows, size=w["B"])  # the reference's sampler (iql.py:172)
        batch = [data["observations"][idx], data["actions"][idx], data["rewards"][idx][:, None],
                 data["next_observations"][idx], data["terminals"][idx].astype(np.float32)[:, None]]
        masks = (rng.uniform(size=(w["L"], w["B"], w["H"])) < keep) if w["dropout"] > 0 else None
        orc.train(batch, dropout_masks=masks)

    for _ in range(warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = time.perf_counter() - t0
    return steps / dt, dt, cores


def cpu_baseline_block(w, cpu_steps):
    """The `cpu_baseline` object of the JSON line (rank 0, N = 1): a bounded sample of the workload's member-step."""
    if reference_available():
        big = w["H"] > 256 or w["B"] > 256
        m = (cpu_reference_measurements(w, 12, 3, 2) if big else
             cpu_reference_measurements(w, max(20, cpu_steps), max(10, cpu_steps // 4), 20))
        return {"value": m["all"], "unit": "steps/s", "cores": m["cores"], "kind": "reference",
                "one_thread": m["one"], "nproc": m["nproc"], "cpu_model": cpu_model(),
                "one_member_per_core_derived": m["one"] * m["nproc"],
                "sample": f"unmodified reference offline/iql.py (staged oracle/_ref), ONE member, {N_ROWS}-row buffer, sample()+train(): "
                          f"{m['dt_all']:.1f} s on {m['cores']} threads, {m['dt_one']:.1f} s on 1 thread"}
    sps, dt, cores = cpu_port_steps_per_sec(w, cpu_steps, 5)
    return {"value": sps, "unit": "steps/s", "cores": cores, "kind": "port",
            "sample": f"{cpu_steps} sample+train steps of ONE member, numpy port of the reference update (staged reference "
                      f"files missing), {dt:.1f} s"}


def run_reference_arm(args, w, rank):
    if rank != 0:
        return
    big = w["H"] > 256 or w["B"] > 256
    inner = args.inner if args.inner else (2 if big else 100)  # reference steps per bench step (bounded sample)
    steps_total = max(1, args.steps) * inner
    warm = max(3, args.warmup) * (1 if big else 5)
    if reference_available():
        m = cpu_reference_measurements(w, steps_total, max(10, steps_total // 4), warm)
        sps, dt, cores, kind = m["all"], m["dt_all"], m["cores"], "reference"
        extra = {"one_thread": m["one"], "nproc": m["nproc"], "cpu_model": cpu_model(),
                 "one_member_per_core_derived": m["one"] * m["nproc"]}
        sample = (f"{steps_total} sample()+train() steps of ONE member through the unmodified reference offline/iql.py "
                  f"(staged oracle/_ref), {N_ROWS}-row buffer, {dt:.1f} s on {cores} threads; 1 thread: {m['one']:.1f} steps/s")
        eager = None
        if not args.no_eager:
            try:
                eager = torch_eager_b200(w, steps=30 if big else 300, warmup=5 if big else 30)
            except Exception as ex:  # the CPU arm must not fail because the GPU leg did
                eager = {"error": repr(ex)[:200]}
    else:
        sps, dt, cores = cpu_port_steps_per_sec(w, steps_total, warm)
        kind, extra, eager = "port", {}, None
        sample = f"{steps_total} sample+train steps of ONE member (numpy port: staged reference files missing), 200k-row buffer, {dt:.1f} s"
    line = {
        "impl": "reference", "metric": "iql_gradient_steps_per_sec_summed_over_seeds", "value": sps, "unit": "steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / max(1, args.steps) * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "desc": w["desc"], "members": 1, "inner_steps_per_bench_step": inner,
                   "batch": w["B"], "hidden": f'{w["L"]}x{w["H"]}', "obs": w["S"], "act": w["A"], "buffer_rows": N_ROWS,
                   "same_shape_and_buffer_as_ours": kind == "reference",
                   "note": "the reference trains ONE member per process (ray_trainer.py:20-24); our arm sums 64+ members"},
        "cpu_baseline": dict({"value": sps, "unit": "steps/s", "cores": cores, "kind": kind, "sample": sample}, **extra),
        "torch_eager_b200": eager,
        "e2e": {"value": sps, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------
def run_ours(args, w, rank, world, local_rank, collect=None):
    import numpy as np
    import torch

    from jsrl_corl_b200 import IQLEnsemble, ReplayBuffer
    from jsrl_corl_b200.synthetic import synthetic_dataset

    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    scaling = w.get("scaling", "weak")
    if scaling == "strong":  # a fixed member count split over the ranks (pen sweep: 256 -> 128 / 64 / 32 per GPU)
        if w["members"] % world:
            raise SystemExit(f"{w['members']} members do not split over {world} GPUs")
        S_local = w["members"] // world
    else:
        S_local = w["members"]
    # one bench step = `inner` updates per member in ONE engine call; sized so that the default 20 timed steps last >= 2 s
    inner = args.inner if args.inner else ((320 if w["members"] >= 32 else 1000) if w["H"] <= 256 and w["B"] <= 256 else 100)
    first_member = rank * S_local  # weak scaling: every GPU trains its own block of members
    seeds = list(range(first_member, first_member + S_local))
    hp = [dict(beta=w["beta"], iql_tau=w["iql_tau"], tau=w["tau"], cosine_t_max=1_000_000) for _ in seeds]
    ens = IQLEnsemble(S_local, w["S"], w["A"], w["H"], w["L"], w["B"], deterministic=w["det"], actor_dropout=w["dropout"],
                      math_mode=args.math, device=device, max_steps_per_call=inner, seeds=seeds, hparams=hp,
                      init=not args.fast_init)
    if args.fast_init:  # same distribution family, one draw for all members (bench-only shortcut)
        ens.init_member(0, seeds[0])
        ens.engine.params[1:] = ens.engine.params[0]
        ens.engine.target[1:] = ens.engine.target[0]
    data = synthetic_dataset(N_ROWS, w["S"], w["A"], 0, antmaze_rewards=w["antmaze"])
    rb = ReplayBuffer(w["S"], w["A"], N_ROWS, device)
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):  # the reference-compatible "Dataset size" print must not reach stdout
        rb.load_d4rl_dataset(data)
    ens.bind_replay(rb)
    eng = ens.engine
    losses = torch.empty(S_local, inner, 3, dtype=torch.float32, device=device)
    gathered = torch.empty(world, S_local, inner, 3, dtype=torch.float32, device=device) if world > 1 else None

    def step():
        eng.train_steps(inner, out=losses)
        if world > 1:
            dist.all_gather_into_tensor(gathered, losses)  # the only collective: log scalars

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    for _ in range(max(3, args.warmup)):
        step()
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    with ClockSampler(local_rank) as clk:
        sync_all()
        e0.record()
        for _ in range(args.steps):
            step()
            launches += eng.last_launch_count()
        e1.record()
        sync_all()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    final = losses.cpu().numpy()
    assert np.isfinite(final).all(), "non-finite losses in the timed region"
    if args.dump_outputs and rank == 0:  # before the e2e leg below trains the same engine further
        dump_outputs(args.dump_outputs, {"losses": final, "params": eng.params.cpu(), "target": eng.target.cpu()})
    total_steps = world * S_local * inner * args.steps
    value = total_steps / (ms * 1e-3)

    # ---- e2e: the same work through the public API with HOST inputs -------------
    # every bench step DRAWS that step's sample indices on the host inside the timed loop (the reference draws them per
    # step with numpy, iql.py:172), copies them from pinned host memory into the engine's staging buffer, runs the K
    # fused steps and reads the loss scalars back.  The draw for call i+1 overlaps the GPU work of call i.
    rs = np.random.RandomState(rank)
    idx_host = [torch.empty(S_local, inner, w["B"], dtype=torch.int64).pin_memory() for _ in range(2)]
    idx_host[0].numpy()[...] = rs.randint(0, N_ROWS, size=(S_local, inner, w["B"]))
    loss_host = torch.empty(S_local, inner, 3, dtype=torch.float32).pin_memory()
    state = {"i": 0}

    def e2e_step():
        cur = state["i"] & 1
        state["i"] += 1
        out = eng.train_steps(inner, mode="indices", indices=idx_host[cur], out=losses)
        loss_host.copy_(out, non_blocking=True)
        idx_host[cur ^ 1].numpy()[...] = rs.randint(0, N_ROWS, size=(S_local, inner, w["B"]))  # next call's indices
        torch.cuda.current_stream(device).synchronize()  # the caller consumes the log dict every call

    for _ in range(3):
        e2e_step()
    sync_all()
    e2e_steps = args.steps
    e0.record()
    for _ in range(e2e_steps):
        e2e_step()
    e1.record()
    sync_all()
    ms_e2e = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_e2e], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = float(t.item())
    e2e_value = world * S_local * inner * e2e_steps / (ms_e2e * 1e-3)

    # ---- drop-in loop (S = 1): the reference's own hot loop, verbatim, on the facade classes ----------------
    dropin = None
    if rank == 0 and world == 1 and not args.no_dropin:
        dropin = dropin_loop_rate(w, device, rb)

    # per-kernel CUDA-event timing of the step (events on the engine's launch stream), after the timed region
    kernels = eng.profile_step(reps=5) if rank == 0 else []

    if rank == 0:
        peaks, peak_src = measured_peaks()
        tf32_peak, tf32_src = pinned_tf32_peak(torch, device) if args.math == "tf32" else (148 * 128 * 2 * 1.965e9 / 1e12, "fp32 FMA nominal")
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        fl = flops_per_step(w)
        achieved_tflops = (S_local * inner * args.steps * fl) / (ms * 1e-3) / 1e12  # per GPU, whole step
        traffic_path = os.path.join(ROOT, "profiles", "traffic.json")
        traffic = json.load(open(traffic_path)) if os.path.exists(traffic_path) else {}
        table = []
        for kq in kernels:
            t = kq["ms"] * 1e-3
            tf, gb = kq["flops"] / t / 1e12, kq["bytes"] / t / 1e9
            bound = "tensor" if kq["flops"] / (tf32_peak * 1e12) > kq["bytes"] / (hbm_peak * 1e9) else "hbm"
            table.append({"kernel": kq["label"], "us": round(kq["ms"] * 1e3, 2), "bound": bound, "tflops": round(tf, 2),
                          "gbs": round(gb, 1), "frac": round(tf / tf32_peak if bound == "tensor" else gb / hbm_peak, 4)})
        step_us = sum(r["us"] for r in table)
        dom = max(table, key=lambda r: r["us"]) if table else None
        roof = None
        if dom is not None:
            dk = next(kq for kq in kernels if kq["label"] == dom["kernel"])
            roof = {"bound": dom["bound"], "achieved": dom["tflops"] if dom["bound"] == "tensor" else dom["gbs"],
                    "peak": tf32_peak if dom["bound"] == "tensor" else hbm_peak,
                    "unit": "TFLOP/s" if dom["bound"] == "tensor" else "GB/s", "frac": dom["frac"],
                    "traffic": traffic.get(dom["kernel"]),
                    "kernel": dom["kernel"], "kernel_us": dom["us"], "kernel_share_of_step": round(dom["us"] / step_us, 3),
                    "algorithmic_bytes_per_launch": dk["bytes"], "algorithmic_flops_per_launch": dk["flops"],
                    "peak_source": (f"HBM {peak_src} (MEASURED_PEAKS.json)" if dom["bound"] == "hbm" else
                                    tf32_src),
                    "how": "CUDA events on the engine's launch stream around every kernel of the step, 5 reps, "
                           "after the timed region (iql_profile_step)"}
        step_view = {"step_us_sum_of_kernels": round(step_us, 1),
                     "whole_step_tflops": round(achieved_tflops, 2), "tf32_peak_tflops": round(tf32_peak, 1),
                     "tf32_peak_source": tf32_src, "tf32_nominal_tflops": TF32_NOMINAL_TFLOPS,
                     "whole_step_frac_of_nominal_tf32": round(achieved_tflops / TF32_NOMINAL_TFLOPS, 4),
                     "tf32_sustained_tflops": tf32_sustained(),
                     "whole_step_frac_of_tensor_peak": round(achieved_tflops / tf32_peak, 4),
                     "whole_step_hbm_gbs": round(sum(kq["bytes"] for kq in kernels) / (step_us * 1e-6) / 1e9, 1) if step_us else None,
                     "hbm_peak_gbs": hbm_peak, "bf16_peak_tflops": peaks.get("bf16_tflops"), "peak_source": peak_src}
        cpu = None
        if not args.no_cpu_baseline and world == 1:  # rank 0 at N = 1 only
            cpu = cpu_baseline_block(w, args.cpu_steps)
        eager = None
        if world == 1 and not args.no_eager:
            try:
                eager = torch_eager_b200(w, steps=30 if (w["H"] > 256 or w["B"] > 256) else 300, warmup=5 if w["H"] > 256 else 30)
            except Exception as ex:
                eager = {"error": repr(ex)[:200]}
        line = {
            "metric": "iql_gradient_steps_per_sec_summed_over_seeds", "value": value, "unit": "steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "tf32" if args.math == "tf32" else "f32", "data": "synthetic",
            "config": {"workload": args.workload, "desc": w["desc"], "members_per_gpu": S_local, "members_total": world * S_local,
                       "inner_steps_per_bench_step": inner, "batch": w["B"], "hidden": f'{w["L"]}x{w["H"]}', "obs": w["S"],
                       "act": w["A"], "buffer_rows": N_ROWS, "sampler": "philox in-kernel",
                       "l2_policy": "inputs larger than L2: per-step working set (params+Adam+activations of all members) "
                                    f"= {(eng.params.numel() * 4 * 4 + eng.workspace.numel()) / 1e6:.0f} MB plus random rows of a "
                                    f"{rb.rows.numel() * 4 / 1e6:.0f} MB buffer",
                       "math_mode": args.math, "parallelism": f"members sharded x{world}, no update-path collective"},
            "e2e": {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": idx_host[0].numel() * 8,
                    "d2h_bytes_per_step": loss_host.numel() * 4,
                    "note": "int64 sample indices drawn on the host INSIDE the timed loop (numpy), copied from pinned memory, "
                            "loss scalars read back, one sync per bench step"},
            "e2e_dropin": dropin,
            "torch_eager_b200": eager,
            "gpu_launches": launches,
            "roofline": roof,
            "step_roofline": step_view,
            "kernels": table,
            "hbm": {"gather_bytes_per_member_step": gather_bytes_per_step(w)},
            "cpu_baseline": cpu,
            "clocks": clk.summary(),
            "flop_per_member_step": fl,
            "last_losses_member0": [float(x) for x in final[0, -1]],
        }
        if collect is not None:
            collect.append(line)
        else:
            print(json.dumps(line), flush=True)
    del ens, eng, rb
    torch.cuda.empty_cache()
    if world > 1:
        dist.destroy_process_group()


def dropin_loop_rate(w, device, rb, steps=3000, warmup=300):
    """`batch = rb.sample(B); trainer.train(batch)` (offline/iql.py:631-635) on the drop-in classes, one learner."""
    import numpy as np
    import torch

    from jsrl_corl_b200 import iql as facade

    torch.manual_seed(0)
    np.random.seed(0)
    q = facade.TwinQ(w["S"], w["A"], w["H"], w["L"])
    v = facade.ValueFunction(w["S"], w["H"], w["L"])
    pol = facade.DeterministicPolicy if w["det"] else facade.GaussianPolicy
    actor = pol(w["S"], w["A"], 1.0, w["H"], w["L"], dropout=w["dropout"])
    trainer = facade.ImplicitQLearning(1.0, actor, torch.optim.Adam(actor.parameters(), lr=3e-4), q,
                                       torch.optim.Adam(q.parameters(), lr=3e-4), v, torch.optim.Adam(v.parameters(), lr=3e-4),
                                       iql_tau=w["iql_tau"], beta=w["beta"], max_steps=1_000_000, discount=0.99, tau=w["tau"],
                                       device=str(device))
    if w["H"] > 256 or w["B"] > 256:
        steps, warmup = 200, 20
    for _ in range(warmup):
        trainer.train(rb.sample(w["B"]))
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    for _ in range(steps):
        log = trainer.train(rb.sample(w["B"]))
    torch.cuda.synchronize(device)
    dt = time.perf_counter() - t0
    assert all(np.isfinite(x) for x in log.values())
    out = {"value": steps / dt, "unit": "steps/s", "members": 1, "steps": steps,
           "what": "ReplayBuffer.sample() + ImplicitQLearning.train(batch) per step through the drop-in classes "
                   "(numpy index stream, host-visible log dict every step), wall clock"}
    # the ONLINE loop body as the host sees it (jsrl_w_iql.py:445-548 without the env): act -> add_transition -> sample -> train
    if not actor.net.has_dropout_modules or w["dropout"] in (None, 0.0):
        actor.eval()
        n_on = max(100, steps // 3)
        obs = np.random.RandomState(1).randn(n_on + 1, w["S"]).astype(np.float32)
        size0, ptr0 = rb._size, rb._pointer
        row_keep = rb._rows[0:1].clone()  # the shared bench buffer is full: every insert rewrites row 0, restored below
        t0 = time.perf_counter()
        for i in range(n_on):
            a = actor.act(obs[i], str(device))
            rb._pointer = 0
            rb.add_transition(obs[i], a, 1.0, obs[i + 1], False)
            rb._size = size0
            log = trainer.train(rb.sample(w["B"]))
        torch.cuda.synchronize(device)
        dt_on = time.perf_counter() - t0
        rb._rows[0:1].copy_(row_keep)
        rb._size, rb._pointer = size0, ptr0
        out["online_loop"] = {"value": n_on / dt_on, "unit": "iterations/s", "us_per_iteration": dt_on / n_on * 1e6, "iterations": n_on,
                              "what": "actor.act(obs) + add_transition + sample(B) + train(batch) per iteration (no env), wall clock"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="halfcheetah_ens64", choices=sorted(WORKLOADS))
    ap.add_argument("--math", default="tf32", choices=["tf32", "fp32"])
    ap.add_argument("--inner", type=int, default=0, help="updates per engine call (0 = workload default)")
    ap.add_argument("--members", type=int, default=0, help="override members per GPU")
    ap.add_argument("--cpu-steps", type=int, default=1500)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager", action="store_true", help="skip the stock-torch-on-GPU leg (torch_eager_b200)")
    ap.add_argument("--no-dropin", action="store_true", help="skip the S=1 drop-in loop leg (e2e_dropin)")
    ap.add_argument("--fast-init", action="store_true")
    ap.add_argument("--all-configs", action="store_true",
                    help="N = 1: run every BASELINE.json workload back to back and print ONE line with the table")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's losses, parameters and Q targets to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.all_configs):
        ap.error("--dump-outputs needs --impl ours and a single workload")
    w = dict(WORKLOADS[args.workload])
    if args.members:
        w["members"] = args.members
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, w, rank)
        return
    if args.all_configs:
        if world != 1:
            raise SystemExit("--all-configs is a single-GPU summary")
        rows = []
        for name in ("hopper_single", "antmaze_jsrl", "halfcheetah_ens64", "hopper_ens64", "pen_sweep256", "stress_4x1024"):
            args.workload = name
            args.inner = 0
            got = []
            run_ours(args, dict(WORKLOADS[name]), 0, 1, local_rank, collect=got)
            ln = got[0]
            rows.append({"workload": name, "desc": ln["config"]["desc"], "members": ln["config"]["members_total"],
                         "steps_per_s": round(ln["value"], 1), "e2e_steps_per_s": round(ln["e2e"]["value"], 1),
                         "e2e_dropin_steps_per_s": (round(ln["e2e_dropin"]["value"], 1) if ln.get("e2e_dropin") else None),
                         "torch_eager_b200_steps_per_s": (round(ln["torch_eager_b200"]["value"], 1) if ln.get("torch_eager_b200") and "value" in ln["torch_eager_b200"] else None),
                         "cpu_reference_steps_per_s": (round(ln["cpu_baseline"]["value"], 1) if ln.get("cpu_baseline") else None),
                         "whole_step_tflops": ln["step_roofline"]["whole_step_tflops"],
                         "frac_of_tf32_peak": ln["step_roofline"]["whole_step_frac_of_tensor_peak"],
                         "hbm_gbs": ln["step_roofline"]["whole_step_hbm_gbs"],
                         "dominant_kernel": ln["roofline"]["kernel"] if ln.get("roofline") else None,
                         "dominant_frac": ln["roofline"]["frac"] if ln.get("roofline") else None,
                         "launches_per_step": round(ln["gpu_launches"] / (ln["steps"] * ln["config"]["inner_steps_per_bench_step"]), 2),
                         "clocks": ln["clocks"]})
        print(json.dumps({"all_configs": rows, "n_gpus": 1, "tf32_peak_tflops": got[0]["step_roofline"]["tf32_peak_tflops"],
                          "hbm_peak_gbs": got[0]["step_roofline"]["hbm_peak_gbs"]}), flush=True)
        return
    if world == 1 and args.gpus > 1:
        print(json.dumps({"error": f"--gpus {args.gpus} must be launched with torch.distributed.run (one rank per GPU)"}))
        sys.exit(2)
    run_ours(args, w, rank, world, local_rank)


if __name__ == "__main__":
    main()
