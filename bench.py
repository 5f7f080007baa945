#!/usr/bin/env python
"""bench.py -- plan-loop Hz / rollout-steps per second of the MPPI rollout hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config c2|c3|c4|c5] [--scaling strong|weak]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is ONE MPPI plan of a BASELINE configuration: shift U -> K1 sample/clamp -> K2 articulated rollout -> Objective cost ->
K3 fused cost/softmax/weighted sum -> [exchange of the shard partials] -> K4 update.

  --config   c2 (default) = the headline, panda 7-DoF reach K = 10 000, T = 30 (BASELINE C2*); c3 = boxer_push K = 4 000, T = 20;
             c4 = heijn_push K = 16 000, T = 25 (BASELINE: 4 GPUs); c5 = panda_pick K = 65 536, T = 30 (BASELINE: 8 GPUs)
  --scaling  strong (default; BASELINE.md section 4: the configuration's K is the GLOBAL sample count, sharded over the N ranks) or
             weak (every GPU owns the configuration's K).  With N > 1 the strong run also reports a short weak run under "weak".

Printed JSON (rank 0, one line):
  value         rollout-steps/s (= K_total * T * plans/s), inputs resident in HBM, CUDA events per plan, max over ranks
  e2e           the same metric through MPPIisaacPlanner.compute_action_tensor(dof_bytes, root_bytes) with host buffers; every other
                call carries a NEW root-state message (moving goal), the others only a new joint state
  roofline      K3 (fused cost-softmax-weighted-sum) achieved HBM GB/s vs the measured peak (MEASURED_PEAKS.json)
  cpu_baseline  the CPU restatement of the reference pipeline (oracle/) on this box's host cores (N = 1 only), with its parallel efficiency
  correctness   N > 1: max |action| difference across ranks and between the peer-memory exchange and the NCCL all-gather
--dump-outputs DIR writes what the last timed plan returned to its caller as DIR/<name>.npy (rank 0, see dump_outputs); the inputs are
seeded, so two builds run with the same arguments can be compared output for output.
--impl reference times that CPU restatement as the reference arm (the reference's own engines, IsaacGym/PhysX and mppi_torch, are
closed / un-vendored and cannot run here: BASELINE.md section 2).
"""
import argparse
import copy
import json
import os
import sys
import threading
import time

sys.dont_write_bytecode = True         # the tree may be read-only; bench.py leaves nothing in it
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "rollout_steps_per_sec"
UNIT = "rollout-steps/s"

PANDA_Q = [0.0, -0.94, 0.0, -2.8, 0.0, 1.8675, 0.0]
CONFIGS = {
    "c2": dict(cfg="config_panda_b200", K=10000, T=30, baseline_gpus=1, q=None,
               workload="panda 7-DoF reach (BASELINE C2*): K=10000, T=30, dt=0.05, substeps=2, Gaussian sampling, cost O1 (PandaReachObjective)"),
    "c3": dict(cfg="config_boxer_push_b200", K=4000, T=20, baseline_gpus=1, q=[0.0, 2.5, 0.0],
               workload="boxer_push non-prehensile contact (BASELINE C3): K=4000, T=20, dt=0.05, substeps=2, cost O2 (PushObjective)"),
    "c4": dict(cfg="config_heijn_push_b200", K=16000, T=25, baseline_gpus=4, q=[0.0, 0.0, 0.0],
               workload="heijn_push omni base + obstacles (BASELINE C4): K=16000, T=25, dt=0.1, substeps=1, cost O2 (PushObjective)"),
    "c5": dict(cfg="config_panda_pick_b200", K=65536, T=30, baseline_gpus=8, q=PANDA_Q + [0.02, 0.02],
               workload="panda_pick 7-DoF + grasp contacts (BASELINE C5): K=65536, T=30, dt=0.05, substeps=2, cost O3 (PandaPickObjective)"),
}
# kept for the tools/ scripts that import bench
K_PER_GPU = CONFIGS["c2"]["K"]
T_HORIZON = CONFIGS["c2"]["T"]


def make_objective(name, device="cuda", fused=True, cpu_threads=1):
    from mppi_isaac_b200.objectives import PandaPickObjective, PandaReachObjective, PushObjective
    if name == "c2":
        if device == "cpu":
            from oracle.backend import OraclePandaReachObjective
            return OraclePandaReachObjective(nthreads=cpu_threads)
        return PandaReachObjective(fused=fused)
    if name == "c3":
        return PushObjective(robot="boxer", link="ee_link")
    if name == "c4":
        return PushObjective()
    return PandaPickObjective()


def load_cfg(name, k_total, device):
    from mppi_isaac_b200.utils.config_store import load_isaacgym_config
    c = CONFIGS[name]
    cfg = copy.deepcopy(load_isaacgym_config(c["cfg"]))
    cfg.mppi.num_samples, cfg.mppi.horizon, cfg.mppi.device = int(k_total), int(c["T"]), device
    return cfg


def panda_cfg(K, device):
    return load_cfg("c2", K, device)


def base_config(name, world, scaling):
    """The `config` object of the JSON line: identical keys and values in both arms (b200 / reference)."""
    c = CONFIGS[name]
    k_total = c["K"] * (world if scaling == "weak" else 1)
    return {"workload": c["workload"], "name": name, "K_total": k_total, "T": c["T"], "scaling": scaling,
            "parallelism": f"sample-shard x{world}"}


def synthetic_state(seed=1234 + 2):
    """SURVEY 8(d) C2: q0 ~ U(lower+0.1, upper-0.1), qd0 = 0, goal ~ U([0.3,0.7]x[-0.4,0.4]x[0.2,0.7])."""
    g = np.random.default_rng(seed)
    lo = np.array([-2.8973, -1.7628, -2.8973, -3.0718, -2.8973, -0.0175, -2.8973]) + 0.1
    hi = np.array([2.8973, 1.7628, 2.8973, -0.0698, 2.8973, 3.7525, 2.8973]) - 0.1
    q0 = g.uniform(lo, hi)
    goal = g.uniform([0.3, -0.4, 0.2], [0.7, 0.4, 0.7])
    return q0, goal


def init_world(planner, name):
    """Synthetic initial world of a configuration (host-side setters; the planner then holds it on its device)."""
    c = CONFIGS[name]
    if name == "c2":
        q0, goal = synthetic_state()
        planner.sim.set_actor_position_by_name(goal, "goal")
        planner.sim.reset_robot_state(q0, np.zeros(7))
    else:
        planner.sim.reset_robot_state(c["q"], [0.0] * len(c["q"]))


def world_messages(planner, rng=None, dq=0.0, goal_shift=None, base_shift=None):
    """(dof_bytes, root_bytes, n_bytes): the world -> planner message of the reference (torch.save bytes of the (1, 2*ndof) DOF row and
    the (1, A, 13) root states, transport.py:5-14), built from the planner's current world with an optional perturbation."""
    from mppi_isaac_b200.utils.transport import torch_to_bytes
    sim = planner.sim
    nd, nv = sim.scene.ndof, sim.scene.virtual_dofs
    st = sim._state0.detach().cpu().numpy().copy()
    q, qd = st[nv:nd].copy(), st[nd + nv:2 * nd].copy()
    if rng is not None and dq:
        q = q + rng.uniform(-dq, dq, q.shape).astype(np.float32)
        qd = qd + rng.uniform(-2 * dq, 2 * dq, qd.shape).astype(np.float32)
    dof = torch.from_numpy(np.stack([q, qd], 1).reshape(1, -1).astype(np.float32))
    root = sim._root0.detach().cpu().clone().unsqueeze(0)
    if goal_shift is not None:
        root[0, sim._get_actor_index_by_name("goal"), 0:3] += torch.as_tensor(goal_shift, dtype=torch.float32)
    if base_shift is not None:
        root[0, sim.scene.robot_actor, 0:3] += torch.as_tensor(base_shift, dtype=torch.float32)
    return torch_to_bytes(dof), torch_to_bytes(root), dof.numel() * 4 + root.numel() * 4


def world_bytes(planner, q, qd, goal):
    """panda reach message from explicit (q, qd, goal) -- used by tools/."""
    from mppi_isaac_b200.utils.transport import torch_to_bytes
    dof = torch.tensor([[v for a, b in zip(q, qd) for v in (a, b)]], dtype=torch.float32)
    root = torch.from_numpy(planner.sim.scene.root_state0.copy()).unsqueeze(0)
    root[0, planner.sim._get_actor_index_by_name("goal"), 0:3] = torch.tensor(goal, dtype=torch.float32)
    return torch_to_bytes(dof), torch_to_bytes(root), dof.numel() * 4 + root.numel() * 4


class Clocks:
    """SM clock and throttle reasons DURING the timed region, sampled IN PROCESS through NVML (what nvidia-smi reads) by a background
    thread on rank 0 only (every 2 ms; the NVML call releases the GIL).  Not from the timing loop itself: with the exchange fused into
    the kernels every rank waits for the slowest one, and 8 ranks calling into the driver's NVML lock between plans produced
    millisecond stragglers (profiles/r2_multigpu.md).  No nvidia-smi subprocess either (round-1 review)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap", 0x80: "hw_power_brake"}

    def __init__(self, cuda_index, enabled=True, period_s=0.002):
        self.ok, self.sm, self.mask, self.h, self.period = False, [], 0, None, period_s
        self._stop, self._thread = threading.Event(), None
        if not enabled:
            self.err = "not sampled on this rank"
            return
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(cuda_index).uuid)
                try:
                    self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
                except TypeError:
                    self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES")
                phys = int(vis.split(",")[cuda_index]) if vis and vis.split(",")[cuda_index].isdigit() else cuda_index
                self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as e:  # noqa: BLE001
            self.err = f"{type(e).__name__}: {e}"

    def sample(self):
        nv = self.nv
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
        try:
            get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            self.mask |= int(get(self.h))
        except Exception:  # noqa: BLE001
            pass

    def start(self):
        if not self.ok:
            return

        def loop():
            while not self._stop.is_set():
                try:
                    self.sample()
                except Exception:  # noqa: BLE001
                    return
                self._stop.wait(self.period)
        self._thread = threading.Thread(target=loop, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=2)

    def summary(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"NVML unavailable ({getattr(self, 'err', '?')})"]}
        busy = sorted(self.sm)
        return {"sm_mhz": busy[len(busy) // 2] if busy else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(n for bit, n in self.REASONS.items() if self.mask & bit), "samples": len(self.sm),
                "how": f"NVML in process, background thread on rank 0, one sample per {int(self.period * 1e3)} ms while the timed plans run"}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# --------------------------------------------------------------------------------------------------
# CPU restatement arm (cpu_baseline and --impl reference)
# --------------------------------------------------------------------------------------------------
def cpu_plan_rate(name, k_sample, steps, warmup, threads):
    """Seconds per plan of the oracle pipeline (sample -> rollout -> Objective -> reduce -> finalize) on `threads` host threads:
    persistent worker pool inside the oracle, the Objective of c2 evaluated by the oracle's threaded cost function, torch intra-op
    threads = `threads` for the torch-op Objectives of the contact configurations."""
    from mppi_isaac_b200 import MPPIisaacPlanner
    from oracle.backend import OracleBackend
    torch.set_num_threads(max(1, min(threads, 32)))
    planner = MPPIisaacPlanner(load_cfg(name, k_sample, "cpu"), make_objective(name, "cpu", cpu_threads=threads), backend=OracleBackend(nthreads=threads))
    init_world(planner, name)
    for _ in range(warmup):
        planner.mppi.command()
    t0 = time.perf_counter()
    for _ in range(steps):
        planner.mppi.command()
    return (time.perf_counter() - t0) / max(steps, 1)


def pick_cpu_sample(name, threads, budget_s, k_max):
    """Largest K (<= the configuration's K, multiple of 4) whose single plan fits `budget_s` on this host, from a small probe."""
    k_probe = max(64, min(512, 8 * threads // 4 * 4))
    probe = cpu_plan_rate(name, k_probe, 2, 1, threads)
    k = int(min(k_max, max(k_probe, budget_s / (probe / k_probe))))
    return max(64, (k // 4) * 4)


def host_cores():
    """Host threads this process may run on (the affinity mask, not the machine's CPU count)."""
    try:
        return len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        return os.cpu_count() or 1


def best_thread_count(name):
    """Thread count that gives the highest plan rate on THIS host: shared boxes report 128 logical CPUs of which far fewer are
    available (tools/cpu_scaling.py on the GPU box: linear to 16 threads, best at 32, slower beyond) -- an all-CPUs run would
    understate the CPU arm.  Probed on a small K with the candidates {all, 1/2, 1/4, 1/8 of the affinity mask, 32, 16}."""
    cores = host_cores()
    cands = sorted({c for c in (cores, cores // 2, cores // 4, cores // 8, 32, 16) if 1 <= c <= cores}, reverse=True)
    k_probe = 2048
    rates = {}
    for c in cands:
        rates[c] = k_probe / cpu_plan_rate(name, k_probe, 2, 1, c)
    best = max(rates, key=rates.get)
    return best, {str(c): round(r * CONFIGS[name]["T"]) for c, r in rates.items()}


def cpu_baseline(name, n_plans=5, budget_s=2.0, threads=None):
    probe = None
    if threads is None:
        threads, probe = best_thread_count(name)
    T = CONFIGS[name]["T"]
    k_s = pick_cpu_sample(name, threads, budget_s, CONFIGS[name]["K"])
    dt = cpu_plan_rate(name, k_s, n_plans, 1, threads)
    k1 = max(64, min(256, k_s))
    dt1 = cpu_plan_rate(name, k1, 3, 1, 1)
    v, v1 = k_s * T / dt, k1 * T / dt1
    return {"value": v, "unit": UNIT, "cores": threads, "host_cpus": host_cores(), "kind": "port",
            "sample": f"{n_plans} plans of K={k_s} of the K={CONFIGS[name]['K']} workload, CPU restatement (oracle/) on {threads} threads "
                      f"(persistent pool; the thread count with the highest rate on this host)",
            "thread_probe_rollout_steps_per_s": probe,
            "plan_hz_at_config_K_est": 1.0 / (dt * CONFIGS[name]["K"] / k_s),
            "parallel_efficiency": v / (threads * v1),
            "one_thread": {"value": v1, "unit": UNIT, "sample": f"3 plans of K={k1} on 1 thread",
                           "plan_hz_at_config_K_est": 1.0 / (dt1 * CONFIGS[name]["K"] / k1)}}, dt, k_s


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    from oracle import oracle as orc
    orc.build()
    name = args.config
    T = CONFIGS[name]["T"]
    threads, probe = best_thread_count(name)
    k_s = pick_cpu_sample(name, threads, 2.0, CONFIGS[name]["K"])
    dt = cpu_plan_rate(name, k_s, args.steps, args.warmup, threads)
    value = k_s * T / dt
    k1 = max(64, min(256, k_s))
    dt1 = cpu_plan_rate(name, k1, 2, 1, 1)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt * 1e3, "plan_hz_at_sample": 1.0 / dt, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": base_config(name, world, args.scaling),
        "note": "CPU restatement of the reference pipeline (oracle/), not IsaacGym/PhysX: those cannot run here (BASELINE.md section 2)",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "host_cpus": host_cores(), "kind": "port",
                         "sample": f"{args.steps} plans of K={k_s} of the K={CONFIGS[name]['K']} workload on {threads} threads (rate is per rollout-step, K-independent)",
                         "thread_probe_rollout_steps_per_s": probe, "parallel_efficiency": value / (threads * (k1 * T / dt1))},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def graph_time_us(fn, reps, replays=3):
    """Device time of `fn` (us per call): `reps` back-to-back calls captured in ONE CUDA graph, so that the
    measurement is free of Python/ctypes launch overhead; CUDA events on the replaying stream, best of `replays`."""
    fn(); torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay(); torch.cuda.synchronize()
    best = float("inf")
    for _ in range(replays):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); g.replay(); b.record(); torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b) * 1e3 / reps)
    return best


def time_kernels(planner, reps=20):
    """Per-kernel device time (us) of one plan (graph-captured back-to-back launches, warm L2)."""
    m, be, sim = planner.mppi, planner.mppi.backend, planner.sim
    from mppi_isaac_b200.model.blob import MODE_SIMPLE
    x = m.noise if be.params.mode == MODE_SIMPLE else m.actions

    def t(fn):
        return graph_time_us(fn, reps)

    out = {"sample_us": t(lambda: m._sample()),
           "rollout_us": t(lambda: sim.rollout_all(m.actions)),
           "cost_objective_us": t(lambda: m._cost_batched())}      # the Objective as benchmarked
    obj = planner.objective
    if getattr(obj, "fused", False):
        obj.fused = False
        out["cost_objective_torch_ops_us"] = t(lambda: m._cost_batched())   # same Objective written with ~28 torch launches
        obj.fused = True
    cost = m._cost_batched()
    out["reduce_us_warm_l2"] = t(lambda: be.reduce(cost, x, m.U, m.partial))
    u_tmp = m.U.clone()
    out["finalize_us"] = t(lambda: be.finalize(m.partial.view(1, -1), 1, u_tmp, m._action, m.stats))
    if m.world == 1:        # what a single-GPU plan actually launches: K3 with K4 done by its last CTA
        out["reduce_finalize_fused_us_warm_l2"] = t(lambda: be.reduce_finalize(cost, x, u_tmp, m.partial, m._action, m.stats))
    return out


def k3_roofline(planner, peak_gbs, K_list):
    """K3 alone, inputs rotated over > L2 worth of distinct buffers so every launch reads HBM (cold L2)."""
    from mppi_isaac_b200.backend import CudaBackend
    from mppi_isaac_b200.model.blob import MppibParams
    dev = planner.sim.device
    T, nu = planner.mppi.T, planner.mppi.nu
    res = []
    for K in K_list:
        p = MppibParams.from_buffer_copy(bytes(planner.mppi.backend.params))
        p.K = K
        be = CudaBackend(dev)
        be.create(planner.sim.scene.model, p)
        bytes_alg = 4 * K * T * (nu + 1) + 4 * (T * nu + 2)
        nbuf = min(64, max(2, int(np.ceil(300e6 / bytes_alg))))            # > 2x the 126 MB L2
        xs = [torch.randn((T, nu, K), device=dev) * 0.3 for _ in range(nbuf)]
        cs = [torch.rand((T, K), device=dev) * 10 for _ in range(nbuf)]
        U = torch.zeros((T, nu), device=dev)
        partial = torch.zeros(2 + T * nu, device=dev)

        def sweep():
            for i in range(nbuf):
                be.reduce(cs[i], xs[i], U, partial)
        us = graph_time_us(sweep, 2) / nbuf
        gbs = bytes_alg / (us * 1e-6) / 1e9
        res.append({"K": K, "bytes": bytes_alg, "us": us, "GBps": gbs, "frac": gbs / peak_gbs, "l2": f"cold: {nbuf} rotating input sets ({nbuf * bytes_alg / 1e6:.0f} MB)"})
        del xs, cs
        be.destroy()
    return res


def timed_plans(planner, steps, warmup, flush, barrier, clocks=None):
    """`steps` plans, each bracketed by CUDA events on the launching stream, L2 flushed before every one; returns per-plan ms."""
    for _ in range(max(warmup, 3)):
        planner.mppi.command()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    import gc
    gc.collect()
    gc.disable()                     # a collection pause on one rank stalls every rank (they wait for its shard row)
    if clocks is not None:
        clocks.start()
    barrier()
    try:
        for i in range(steps):
            flush.zero_()
            starts[i].record()
            planner.mppi.command()
            ends[i].record()
        barrier()
    finally:
        gc.enable()
        if clocks is not None:
            clocks.stop()
    return [s.elapsed_time(e) for s, e in zip(starts, ends)]


def dump_outputs(planner, out_dir, n_samples=4096):
    """float32 .npy files of what the last plan handed its caller: `action` (the first action, command()'s return value),
    `mean_action` (the updated control sequence U, (T, nu)) and `perturbed_action_sample` (the sampled control sequences of a fixed
    seeded subset of at most `n_samples` of the K samples, in ascending sample order, (n, T, nu)) -- under 6 MB at every configuration."""
    m = planner.mppi
    torch.cuda.synchronize()
    idx = np.sort(np.random.default_rng(0).choice(m.K, min(m.K, n_samples), replace=False))
    outs = {"action": m._action, "mean_action": m.mean_action,
            "perturbed_action_sample": m.perturbed_action[torch.as_tensor(idx, device=m.actions.device)]}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outs.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().to(torch.float32).cpu().numpy())


def run_gpu_arm(args, rank, world, local_rank):
    import torch.distributed as dist
    import __graft_entry__
    __graft_entry__.build()
    from mppi_isaac_b200 import MPPIisaacPlanner
    from mppi_isaac_b200.utils.transport import bytes_to_torch

    name = args.config
    C = CONFIGS[name]
    T = C["T"]
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
    k_total = C["K"] * (world if args.scaling == "weak" else 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    planner = MPPIisaacPlanner(load_cfg(name, k_total, dev), make_objective(name), use_cuda_graph=True)
    init_world(planner, name)
    nu = planner.mppi.nu
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # > 126 MB L2
    clocks = Clocks(local_rank, enabled=(rank == 0 and os.environ.get("BENCH_NO_CLOCKS", "0") in ("", "0")))

    # ---- device-resident timing ------------------------------------------------------------------------------------
    per_step_ms = timed_plans(planner, args.steps, args.warmup, flush, barrier, clocks)
    if args.dump_outputs and rank == 0:
        dump_outputs(planner, args.dump_outputs)
    graph_on = planner.mppi._graph is not None
    total_s = reduce_max(sum(per_step_ms)) * 1e-3
    value = k_total * T * args.steps / total_s
    p50_ms = reduce_max(float(np.percentile(per_step_ms, 50)))

    # ---- end to end through the plugin API with host buffers ----------------------------------------------------------
    # the caller's side of the wire (building / pickling the world state) is prepared outside the timed region, in the reference's own
    # torch.save byte format (transport.py:5-14).  Odd steps carry a NEW root message (the goal has moved: parse + upload of the root
    # states), even steps only a new joint state.
    rng = np.random.default_rng(99)
    has_goal = "goal" in [a.name for a in planner.sim.env_cfg]
    msgs, h2d = [], 0
    for i in range(args.steps):
        gs = rng.uniform(-0.02, 0.02, 3) if (has_goal and i % 2 == 1) else None
        d, r, nbytes = world_messages(planner, rng, dq=0.02, goal_shift=gs)
        msgs.append((d, r)); h2d = nbytes
    d0, r0, _ = world_messages(planner)

    def e2e_loop(inputs):
        for _ in range(3):
            bytes_to_torch(planner.compute_action_tensor(d0, r0))
        barrier()
        outs = []
        t0 = time.perf_counter()
        for d, r in inputs:
            outs.append(planner.compute_action_tensor(d, r))     # bytes in -> H2D -> plan -> D2H -> bytes out
        torch.cuda.synchronize()
        dt = reduce_max(time.perf_counter() - t0)
        assert all(bytes_to_torch(o).shape == (nu,) for o in outs)
        return dt
    e2e_s = e2e_loop(msgs)
    e2e_static_s = e2e_loop([(m[0], r0) for m in msgs])                                      # joint state only
    e2e_moving_s = e2e_loop([(m[0], world_messages(planner, goal_shift=rng.uniform(-0.02, 0.02, 3))[1]) for m in msgs]) if has_goal else None
    e2e = {"value": k_total * T * args.steps / e2e_s, "unit": UNIT, "plan_hz": args.steps / e2e_s, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": nu * 4, "api": "MPPIisaacPlanner.compute_action_tensor(dof_bytes, root_bytes) -> bytes",
           "inputs": "new joint state every call; every other call also a new root-state message (moved goal)",
           "plan_hz_joint_state_only": args.steps / e2e_static_s,
           "plan_hz_new_root_message_every_call": (args.steps / e2e_moving_s) if e2e_moving_s else None}
    # the reference's in-process entry point: compute_action(q, qdot) with host lists in, host tensor out (fixed-base robots)
    if planner.sim.scene.virtual_dofs == 0:
        nd = planner.sim.scene.ndof
        st = planner.sim._state0.detach().cpu().numpy()
        qs = [list(st[:nd] + rng.uniform(-0.02, 0.02, nd)) for _ in range(args.steps)]
        qds = [list(rng.uniform(-0.05, 0.05, nd)) for _ in range(args.steps)]
        for _ in range(3):
            planner.compute_action(qs[0], qds[0])
        barrier()
        t0 = time.perf_counter()
        for i in range(args.steps):
            planner.compute_action(qs[i], qds[i])
        torch.cuda.synchronize()
        e2e["compute_action_plan_hz"] = args.steps / reduce_max(time.perf_counter() - t0)
    # a moved robot base changes a kernel constant: the captured graph is dropped and re-captured inside the call
    if world == 1 and planner.sim.scene.virtual_dofs == 0:
        db, rb, _ = world_messages(planner, base_shift=[0.01, 0.0, 0.0])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        planner.compute_action_tensor(db, rb)
        torch.cuda.synchronize()
        e2e["ms_first_call_after_base_move_graph_recapture"] = (time.perf_counter() - t0) * 1e3
        planner.compute_action_tensor(d0, r0)

    # ---- multi-GPU correctness keys -----------------------------------------------------------------------------------
    correctness = None
    if world > 1:
        def one_plan(pl):
            pl.sim.reset_to_initial_poses()      # the e2e loops above left their last message (a shifted goal) in the timed planner's world
            init_world(pl, name)
            pl.mppi.U.zero_(); pl.mppi.plan_ctr.zero_()
            pl.mppi.command()
            torch.cuda.synchronize()
            return pl.mppi._action.detach().clone(), pl.mppi.U.detach().clone()
        a_peer, u_peer = one_plan(planner)
        gathered = [torch.zeros_like(a_peer) for _ in range(world)]
        dist.all_gather(gathered, a_peer)
        across = max(float((g - gathered[0]).abs().max()) for g in gathered)
        os.environ["MPPIB_EXCHANGE"] = "nccl"
        p_nccl = MPPIisaacPlanner(load_cfg(name, k_total, dev), make_objective(name), use_cuda_graph=True)
        os.environ["MPPIB_EXCHANGE"] = "peer"
        a_nccl, u_nccl = one_plan(p_nccl)
        correctness = {"action_max_abs_diff_across_ranks": reduce_max(across),
                       "peer_vs_nccl_max_abs_diff": reduce_max(max(float((a_peer - a_nccl).abs().max()), float((u_peer - u_nccl).abs().max()))),
                       "peer_exchange_active": bool(planner.mppi._peer_exchange), "nccl_planner_used_peer": bool(p_nccl.mppi._peer_exchange)}
        p_nccl.mppi.invalidate_graph(); p_nccl.mppi.close_peers()
        del p_nccl

    # ---- weak-scaling companion of a strong-scaling run ----------------------------------------------------------------
    weak = None
    if world > 1 and args.scaling == "strong":
        planner.mppi.invalidate_graph()
        pw = MPPIisaacPlanner(load_cfg(name, C["K"] * world, dev), make_objective(name), use_cuda_graph=True)
        init_world(pw, name)
        ms = timed_plans(pw, args.steps, args.warmup, flush, barrier)
        tw = reduce_max(sum(ms)) * 1e-3
        weak = {"K_total": C["K"] * world, "value": C["K"] * world * T * args.steps / tw, "unit": UNIT, "ms_per_step": tw * 1e3 / args.steps,
                "ms_per_step_p50": reduce_max(float(np.percentile(ms, 50)))}
        pw.mppi.invalidate_graph(); pw.mppi.close_peers()
        del pw

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        fused_obj = bool(getattr(planner.objective, "fused", False))
        n_obj = 1 if fused_obj else None
        launches_per_plan = (4 + (n_obj or 0) if world == 1 else 5 + (n_obj or 0))   # shift, sample, rollout, [fused cost], reduce(+finalize at 1 GPU) [, finalize]
        cfg_line = base_config(name, world, args.scaling)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": total_s * 1e3 / args.steps, "ms_per_step_p50": p50_ms, "plan_hz": args.steps / total_s, "plan_hz_p50": 1e3 / p50_ms,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg_line,
            "gpu_config": {"K_per_gpu": planner.sim.num_envs, "baseline_gpus": C["baseline_gpus"],
                           "exchange": "none" if world == 1 else ("peer-memory stores fused into K3 (NVLink), flags acquired by K4" if planner.mppi._peer_exchange else "NCCL all-gather"),
                           "cuda_graph": graph_on, "l2": "flushed (256 MiB write) before every timed plan",
                           "k2_mapping": planner.mppi.backend.rollout_mapping(),
                           "ms_per_step_p10_p50_p90_max": [float(np.percentile(per_step_ms, p)) for p in (10, 50, 90, 100)],
                           "slowest_steps": sorted(range(len(per_step_ms)), key=lambda i: -per_step_ms[i])[:3]},
            "e2e": e2e,
            "gpu_launches": (launches_per_plan * args.steps) if n_obj else None,
            "clocks": clocks.summary(),
        }
        if not n_obj:
            line["gpu_launches"] = 4 * args.steps if world == 1 else 5 * args.steps
            line["gpu_launches_note"] = "own kernels only (shift, sample, rollout, reduce[, finalize]); this configuration's Objective runs as torch ops"
        if correctness:
            line["correctness"] = correctness
        if weak:
            line["weak"] = weak
        if world == 1:
            if fused_obj:
                # transparency: the same plan with the Objective written as plain torch ops (~28 element-wise launches instead of the
                # one fused ops.pose_cost launch) -- what an unmodified user Objective costs, device-timed and end to end
                planner.objective.fused = False
                planner.mppi.invalidate_graph()
                ms = timed_plans(planner, min(args.steps, 30), 3, flush, barrier)
                t_e2e = e2e_loop(msgs)
                line["objective_as_torch_ops"] = {"ms_per_step": float(np.mean(ms)), "plan_hz": 1e3 / float(np.mean(ms)),
                                                  "value": k_total * T / (float(np.mean(ms)) * 1e-3), "unit": UNIT,
                                                  "e2e_plan_hz": args.steps / t_e2e, "e2e_value": k_total * T * args.steps / t_e2e}
                planner.objective.fused = True
                planner.mppi.invalidate_graph()
                planner.mppi.command()
            kt = time_kernels(planner)
            ks = sorted({planner.sim.num_envs, 65536, 262144})
            roof = k3_roofline(planner, peak, ks)
            head = next(r for r in roof if r["K"] == planner.sim.num_envs)
            traffic = {(10000, 30, 7): 9666560}.get((head["K"], T, nu))
            line["roofline"] = {"kernel": "K3 reduce_kernel (fused cost accumulate + softmax + weighted control sum)", "bound": "hbm",
                                "achieved": head["GBps"], "peak": peak, "unit": "GB/s", "frac": head["frac"], "traffic": traffic,
                                "traffic_source": "ncu --set full dram__bytes_read.sum + write of one K3 launch at this K (profiles/r2_ncu_summaries.txt): 1.007 x algorithmic; 1.0003 x at K = 262 144" if traffic else None,
                                "peak_source": peak_src, "bytes_per_launch": head["bytes"], "us_per_launch": head["us"], "K": head["K"],
                                "note": "the named K is launch/latency bound (9.6 MB = 1.5 us of HBM time at C2*); the sweep shows the asymptote",
                                "sweep": roof}
            line["kernels_us"] = kt
            line["cpu_baseline"], _, _ = cpu_baseline(name)
        print(json.dumps(line), flush=True)
    if world > 1:
        shutdown_distributed(planner)


def shutdown_distributed(planner):
    """Tear NCCL down without hanging: a live CUDA graph that holds NCCL kernels blocks destroy_process_group(), so the
    captured plan is released first; a watchdog force-exits if the teardown still does not return."""
    import gc
    import torch.distributed as dist
    planner.mppi.invalidate_graph()
    planner.mppi.close_peers()          # collective: unmap the peer-memory exchange windows before the group goes away
    del planner
    gc.collect()
    torch.cuda.synchronize()
    dist.barrier()
    sys.stdout.flush()
    timer = threading.Timer(20.0, lambda: os._exit(0))
    timer.daemon = True
    timer.start()
    dist.destroy_process_group()
    timer.cancel()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the last timed plan's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm: the reference arm picks its sample count from the host's speed")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback; use --impl reference for the CPU arm)")
    run_gpu_arm(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
