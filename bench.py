#!/usr/bin/env python
"""Benchmark of the MultiAgentEnv.step hot path (BASELINE.json metric: batched env-steps/s
incl. power flow).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (config.workload = "C1"): the reference's IEEE-13 coordinated-buildings scenario
(3 x building+PV+storage on load 675c, load factor 1.2, shared voltage penalty;
examples/marl/openai/train.py:165-188) batched to 4096 envs per GPU.  One "step" = one
pgw_step over the batch: fused component kernel + batched power flow.  Actions are
synthetic U(-1, 1) float64, pre-generated and resident in HBM for `value`; `e2e` goes
through the host-buffer call (pinned host actions in, obs/reward/done out, every step).

Timing: W >= 3 untimed steps, then K steps each bracketed by CUDA events on the launch
stream with a write of a 256 MiB buffer (> 126 MB L2) between steps, i.e. every timed step
starts with a cold L2; value = envs x K / sum of step times, max over ranks.  N > 1 runs one
process per GPU (torchrun), envs sharded with no data-path collective (weak scaling:
4096 envs per GPU); the only collective is the all-reduce of the 8-entry statistics vector
at the end of the timed region.

--impl reference times the reference's CPU implementation of the same path: the oracle
port (the reference's own Python classes are not on the GPU box, and its power flow,
OpenDSS, is not installable) on all host cores via multiprocessing.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ENVS_PER_GPU = 4096          # BASELINE.json configs[1]; --envs overrides (size sweeps)
PF_KERNEL = "tc2"            # tcgen05 split-FP16 solver; --pf-kernel fp64 / tc select the others
WORKLOAD = "c1"              # --workload c2 = component-only EV+PV+storage (BASELINE configs[2])
GRAPHS = None                # --graphs 0/1 overrides PGW_OPT_GRAPHS (experiments)
METRIC, UNIT = "env_steps_per_s", "env-steps/s"
LOAD_FACTOR = 1.2
# algorithmic bytes per env-step of the component kernel, SURVEY.md section 8(d)
SURVEY_BYTES = {"c1": 3 * (264 + 28 + 40) + 1, "c2": (16 * 100 + 72 + 8 * 4) + 28 + 40 + 1,
                # C3: 40 PV + 30 storage + 10 EV(25) + 20 x (building + PV + storage)
                "c3": 40 * 28 + 30 * 40 + 10 * (16 * 25 + 72 + 8) + 20 * (264 + 28 + 40) + 1,
                # HS house: 4 actions in, 12 obs + P + reward (+ep_ret, rew_copy) out, meta state
                # 5 rows r/w, storage 2 rows r/w, vehicle energy + cost + mask r/w
                "hs": 4 * 8 + 12 * 8 + 5 * 8 + 5 * 16 + 2 * 16 + 2 * 16 + 8 + 1}


_PF_NAMES = {"fp64": "fp64-simt", "tc": "tcgen05 split-tf32", "tc2": "tcgen05 split-fp16, Z-bus in smem"}


def _dtype_label(has_pf):
    """The arithmetic the step computes in (not a precision claim)."""
    if not has_pf or PF_KERNEL == "fp64":
        return "f64"
    if PF_KERNEL == "tc2":
        return "f64 components; power flow: split-fp16 operands / fp32 accumulate (tcgen05) + f64 polish sweeps"
    return "f64 components; power flow: split-tf32 operands / fp32 accumulate (tcgen05)"


def _config(n_gpus, workload=None, envs=None):
    WORKLOAD = workload or globals()["WORKLOAD"]
    ENVS_PER_GPU = envs or globals()["ENVS_PER_GPU"]
    if WORKLOAD == "c2":
        return {"workload": "C2: component-only EV station (100 vehicles) + PV + storage, "
                            f"{ENVS_PER_GPU} envs per GPU, no power flow",
                "envs_per_gpu": ENVS_PER_GPU, "agents_per_env": 3,
                "global_envs": ENVS_PER_GPU * n_gpus, "parallelism": f"env-sharded x{n_gpus}",
                "l2": "flushed between timed steps (256 MiB write)"}
    if WORKLOAD == "hs":
        return {"workload": "HS: Home-Steward house (PV -> storage -> EV charger -> devices, blended "
                            f"energy cost), {ENVS_PER_GPU} houses per GPU, no power flow",
                "envs_per_gpu": ENVS_PER_GPU, "agents_per_env": 1,
                "global_envs": ENVS_PER_GPU * n_gpus, "parallelism": f"env-sharded x{n_gpus}",
                "l2": "flushed between timed steps (256 MiB write)"}
    if WORKLOAD == "c3":
        return {"workload": "C3: 123-bus-class synthetic feeder (251 nodes, 85 load branches), 100 "
                            f"heterogeneous DER agents, {ENVS_PER_GPU} envs per GPU",
                "envs_per_gpu": ENVS_PER_GPU, "agents_per_env": 100,
                "global_envs": ENVS_PER_GPU * n_gpus, "parallelism": f"env-sharded x{n_gpus}",
                "l2": "flushed between timed steps (256 MiB write)", "pf_kernel": _PF_NAMES[PF_KERNEL]}
    return {"workload": "C1: IEEE-13 coordinated buildings (3 x building+PV+storage @675c), "
                        f"{ENVS_PER_GPU} envs per GPU",
            "envs_per_gpu": ENVS_PER_GPU, "agents_per_env": 3, "global_envs": ENVS_PER_GPU * n_gpus,
            "feeder": "IEEE-13 (38 nodes, 14 load branches)", "load_factor": LOAD_FACTOR,
            "parallelism": f"env-sharded x{n_gpus}", "l2": "flushed between timed steps "
            "(256 MiB write)",
            "pf_kernel": _PF_NAMES[PF_KERNEL]}


def _make_env(ns, workload=None, **kw):
    """The benchmark scenario (powergridworld_b200/scenarios/bench.py) against a plugin
    namespace: None = the product, the oracle namespace for the CPU arm."""
    from powergridworld_b200.scenarios import bench as SB
    wl = workload or WORKLOAD
    if ns is None:
        return SB.make_env(wl, **kw)
    # ---- CPU arm (oracle classes; the one place outside tests/ and smoke() that runs oracle/)
    if wl == "c2":
        from oracle.multiagent import PowerFlowSolver

        class NoPF(PowerFlowSolver):
            def __init__(self, **k):
                pass

            def calculate_power_flow(self, *a, **k):
                pass

            def get_bus_voltages(self):
                return {}

            def get_bus_voltage_by_name(self, n):
                return 1.0
        return SB.c2_env(ns, NoPF, **kw)
    if wl == "hs":
        from oracle.namespace import ORACLE_HS_NS as OHS
        from powergridworld_b200.scenarios import catalog_hs as SH
        return _OracleHouse(OHS.HSMultiComponentEnv(**SH.shipped(OHS)))
    return SB.make_env(wl, ns, **kw)


class _OracleHouse:
    """The HS oracle house behind the MultiAgentEnv-shaped surface the CPU worker drives."""

    def __init__(self, house):
        self.house = house
        self.agents = [house]
        self.action_space = {"house": house.action_space}

    def reset(self):
        return {"house": self.house.reset(init_storage=8.1)}

    def step(self, action):
        ob, rew, done, _ = self.house.step(action["house"])
        return {"house": ob}, {"house": rew}, {"__all__": done}, {}


# --------------------------------------------------------------------------- CPU arm
def _cpu_worker(args):
    """One independent CPU env stepped for `budget` seconds (episodes restart as needed); returns
    (steps done, seconds spent stepping) -- building the env is not part of the measurement.
    kind "port": the oracle's restatement of the reference classes; kind "reference": the
    UNMODIFIED reference classes (baseline/_ref or $PGW_REFERENCE_ROOT through oracle/ref_harness.py)
    with the power-flow port plugged into pf_config["cls"] (gridworld/multiagent_env.py:80)."""
    seed, budget, kind = args
    import contextlib

    import numpy as np

    from oracle.flatten import action_layout, unflatten_action
    quiet = contextlib.nullcontext
    if kind == "reference":
        from oracle.powerflow import OracleOpenDSSSolver
        from oracle.ref_harness import quiet_stdout as quiet, reference_namespace
        from powergridworld_b200.scenarios import catalog as S
        ns = reference_namespace()
        with quiet():
            env = ns.CoordinatedMultiBuildingControlEnv(
                **S.buildings_scenario(ns, OracleOpenDSSSolver, LOAD_FACTOR))
    else:
        from oracle.namespace import ORACLE_NS as NS
        env = _make_env(NS)
    rng = np.random.default_rng(seed)
    np.random.seed(seed)
    layout = action_layout(env)
    dim = sum(len(lo) for _, _, lo, _, _ in layout)
    with quiet():
        env.reset()
        for _ in range(3):                             # warm caches / lazy imports
            env.step(unflatten_action(env, rng.uniform(-1, 1, size=dim)))
        t0 = time.perf_counter()
        done = 0
        while time.perf_counter() - t0 < budget:
            _, _, dn, _ = env.step(unflatten_action(env, rng.uniform(-1, 1, size=dim)))
            done += 1
            if dn["__all__"]:
                env.reset()
        return done, time.perf_counter() - t0


def _reference_classes_available():
    if WORKLOAD != "c1":
        return False
    try:
        from oracle.ref_harness import reference_available
        return reference_available()
    except Exception:
        return False


def cpu_throughput(total_seconds_target=15.0, kind="port"):
    """CPU implementation of the path on all host cores: one independent env per core
    (multiprocessing), all stepping concurrently for the time budget; value = steps done by all
    of them / the longest stepping time."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    tasks = [(i + 1, float(total_seconds_target), kind) for i in range(cores)]
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(cores) as pool:
        res = pool.map(_cpu_worker, tasks, chunksize=1)
    wall = time.perf_counter() - t0
    total = sum(n for n, _ in res)
    busy = max(t for _, t in res)
    what = "oracle envs (port of the reference classes + power-flow port)" if kind == "port" else \
        "envs of the UNMODIFIED reference classes (power-flow port plugged into pf_config['cls'])"
    return {"value": total / busy, "unit": UNIT, "cores": cores,
            "kind": "port" if kind == "port" else "reference-classes+pf-port",
            "sample": f"{cores} independent {what}, one per core (multiprocessing.Pool({cores})), stepping "
                      f"concurrently for {busy:.1f} s: {total} env-steps, {1e3 * busy * cores / max(total, 1):.2f} "
                      f"ms/step per core ({wall:.1f} s wall with the env construction)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.perf_counter()
    budget = max(10.0, min(60.0, 0.1 * args.steps))
    port = cpu_throughput(total_seconds_target=budget, kind="port")
    real = cpu_throughput(total_seconds_target=budget, kind="reference") if _reference_classes_available() else None
    cb = real or port
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 / cb["value"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": _config(args.gpus), "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "port": port,
            "note": ("the reference's own MultiAgentEnv / component classes (unmodified, installed in "
                     "baseline/_ref) with the complex128 power-flow port plugged into pf_config['cls']; "
                     "`port` = the oracle's restatement of those classes, ~10x faster per core"
                     if real else
                     "oracle port of the reference classes + complex128 power-flow restatement (no "
                     "reference tree on this box)") +
                    "; the reference's OpenDSS engine is not installable (no network)",
            "wall_s": time.perf_counter() - t0}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- GPU arm
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.max_mhz = None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
                time.sleep(0.002)
        except Exception as exc:                      # NVML missing: report that, not a guess
            self.reasons.add(f"nvml_unavailable:{type(exc).__name__}")

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as fh:
            return json.load(fh), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def _ncu_capture(workload, E):
    """dram bytes per launch (read + write) and tensor-pipe activity per kernel, PARSED from the
    committed `ncu --set full` export of this workload (profiles/r2_ncu_full_raw_<workload>_<E>.csv,
    `ncu -i ... --page raw --csv`); {} when no capture of this size is committed."""
    import csv
    import glob
    paths = sorted(glob.glob(os.path.join(ROOT, "profiles", f"r2*_ncu_full_raw_{workload}_{E}.csv")))
    if not paths:
        return {}
    path = paths[-1]
    with open(path, newline="") as fh:
        rows = list(csv.reader(fh))
    hdr, units, body = rows[0], rows[1], rows[2:]
    col = {n: i for i, n in enumerate(hdr)}
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}

    def val(r, name):
        if name not in col or r[col[name]] == "":
            return None
        return float(r[col[name]].replace(",", "")) * scale.get(units[col[name]], 1.0)
    out = {}
    for r in body:
        k = r[col["Kernel Name"]]
        for key in ("step_fused_kernel", "component_kernel", "pf_tc2_kernel", "pf_fixed_point_kernel"):
            if key in k:
                rd, wr = val(r, "dram__bytes_read.sum"), val(r, "dram__bytes_write.sum")
                tp = val(r, "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active")
                d = out.setdefault(key, {"traffic": [], "tensor_pct": [], "us": []})
                if rd is not None and wr is not None:
                    d["traffic"].append(rd + wr)
                if tp is not None:
                    d["tensor_pct"].append(tp)
                t = val(r, "gpu__time_duration.sum")
                if t is not None:
                    d["us"].append(t * {"us": 1.0, "ns": 1e-3, "ms": 1e3}.get(units[col["gpu__time_duration.sum"]], 1.0))
    mean = lambda v: sum(v) / len(v) if v else None
    res = {k: {"traffic": mean(d["traffic"]), "tensor_pct": mean(d["tensor_pct"]), "us_under_ncu": mean(d["us"]),
               "launches_captured": len(d["traffic"])} for k, d in out.items()}
    res["_source"] = os.path.relpath(path, ROOT) + " (ncu --set full --clock-control none, parsed at run time)"
    return res


DUMP_MAX_BYTES = 64 * 10 ** 6


def _dump_outputs(out_dir, batches):
    """--dump-outputs: what the timed path handed its caller at the last timed step -- each batch's
    observations [obs_dim, E], rewards [agents, E] (float64) and done flags [E] (float32) -- as
    out_dir/<prefix>obs.npy, <prefix>reward.npy, <prefix>done.npy.  ``batches`` maps a file-name
    prefix to an env.  Above DUMP_MAX_BYTES in all, every batch keeps the same share of its env
    columns, drawn by a fixed seed; their indices go to <prefix>env_index.npy (float64)."""
    import numpy as np
    per_env = {p: 8 * env.obs_dim + 8 * len(env.agents) + 4 for p, env in batches.items()}
    total = sum(per_env[p] * env.num_envs for p, env in batches.items())
    budget = DUMP_MAX_BYTES - 4096                   # room for the .npy headers
    share = 1.0 if total <= budget else \
        budget / sum((per_env[p] + 8) * env.num_envs for p, env in batches.items())
    os.makedirs(out_dir, exist_ok=True)
    for prefix, env in batches.items():
        arrays = {"obs": env.obs.cpu().numpy(), "reward": env.rew.cpu().numpy(),
                  "done": env.done.cpu().numpy().astype(np.float32)}
        if share < 1.0:
            keep = max(1, int(env.num_envs * share))
            cols = np.sort(np.random.default_rng(0).choice(env.num_envs, size=keep, replace=False))
            arrays = {k: v[..., cols] for k, v in arrays.items()}
            arrays["env_index"] = cols.astype(np.float64)
        for name, arr in arrays.items():
            np.save(os.path.join(out_dir, f"{prefix}{name}.npy"), np.ascontiguousarray(arr))


def _bind_to_gpu_numa(index):
    """Run this rank (and first-touch its pinned buffers) on the CPUs next to its GPU."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(index)
        words = nv.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * i + b for i, wd in enumerate(words) for b in range(64) if (wd >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def _component_bytes(env, workload, E, W, K):
    """Algorithmic bytes per launch of the component work: SURVEY.md 8(d)'s per-env figure x envs; for
    the EV station the bytes of the vehicles actually parked in the timed events."""
    survey = SURVEY_BYTES[workload] * E
    alg = survey
    if workload == "c2":
        ev = [c for c in env._b.comps if c.type == 3][0]
        rows = env._itab[W + 1:W + 1 + K]
        n_win = float(rows[:, ev.itab_off].mean())
        n_left = float(rows[:, ev.itab_off + 1].mean())
        alg = (16.0 * n_win + 8.0 * n_left + 32.0 + 72.0 + 28.0 + 40.0 + 1.0) * E
    return alg, survey


def measure(workload, E, K, W, dev, world=1, rank=0, headline=False, pdl=1, dump_dir=None):
    """One workload on this rank's GPU: K device-timed steps with a cold L2 before each, the
    per-kernel durations of the same loop, and the rooflines they give.  With ``dump_dir``, rank 0
    writes the outputs of the last timed step there (_dump_outputs)."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from powergridworld_b200 import _native as N

    env = _make_env(None, workload=workload, num_envs=E, device=dev)
    has_pf = env.pf_solver is not None
    if PF_KERNEL != "fp64" and has_pf:
        env.set_option(N.OPT_PF_KERNEL, {"tc": 1, "tc2": 2}[PF_KERNEL])
    if not pdl:
        env.set_option(N.OPT_PDL, 0)
    if GRAPHS is not None:
        env.set_option(N.OPT_GRAPHS, GRAPHS)
    A = len(env.agents)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    # a fresh action tensor every step, as a policy loop hands them in: eight buffers in rotation;
    # the handle replays ONE step graph and re-points its kernel nodes at each of them
    pool_n = 8
    act_pool = [torch.rand((env.act_dim, E), generator=gen, device=dev, dtype=torch.float64) * 2.0 - 1.0
                for _ in range(pool_n)]
    rng = np.random.default_rng(rank)
    soc = torch.as_tensor(30.0 + 5.0 * rng.uniform(-1, 1, size=(env.num_storage, E))).to(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def one_step(i):
        if env._needs_reset:
            env.reset_batch(soc)
        env.step_batch(act_pool[i % pool_n])

    def begin_pass():
        """Every pass starts from a fresh episode + W untimed steps, so that all passes see
        the same events (the EV station's work depends on the time of day)."""
        env.reset_batch(soc)
        for i in range(W):
            one_step(i)
        barrier()

    env.reset_batch(soc)
    for i in range(3):
        one_step(i)
    begin_pass()

    # ---- timed region: K steps, device-timed one by one, cold L2 before each
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    launches0 = env.launch_count
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    wall0 = time.perf_counter()
    for i in range(K):
        flush.zero_()
        starts[i].record()
        one_step(W + i)
        ends[i].record()
    launches = env.launch_count - launches0
    stats = env.all_reduce_stats()                    # the only collective: after the timed steps
    barrier()
    wall = time.perf_counter() - wall0
    step_ms = [s.elapsed_time(e) for s, e in zip(starts, ends)]
    total_ms = float(sum(step_ms))
    if dump_dir is not None and rank == 0:            # before the passes below overwrite them
        _dump_outputs(dump_dir, {"": env})
    iters_mean = float(env.get_field(7).abs().double().mean()) if has_pf else 0.0
    if world > 1:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    value = E * world * K / (total_ms * 1e-3)

    # ---- per-kernel durations for the roofline: same loop (cold L2 before each step), plain
    #      launches with CUDA events between the kernels on the launch stream
    begin_pass()
    env.set_kernel_timing(True)
    for i in range(K):
        flush.zero_()
        one_step(W + i)
    t_a_ms, t_pf_ms, n_timed = env.kernel_timing()
    env.set_kernel_timing(False)
    sampler.stop_flag = True
    fused = bool(has_pf and launches == K)            # one kernel does the whole step
    k_a_ms, pf_ms = t_a_ms / max(n_timed, 1), t_pf_ms / max(n_timed, 1)

    out = {"env": env, "E": E, "A": A, "value": value, "ms_per_step": total_ms / K, "launches": int(launches),
           "stats": stats, "wall": wall, "clocks": sampler.summary(), "has_pf": has_pf, "fused": fused,
           "barrier": barrier, "one_step": one_step, "begin_pass": begin_pass, "soc": soc}
    if rank != 0:
        return out

    peaks, peak_src = _peaks()
    hbm = peaks["hbm_gbs"]
    ncu = _ncu_capture(workload, E)
    comp_bytes, survey_bytes = _component_bytes(env, workload, E, W, K)
    f = env.pf_solver.feeder if has_pf else None
    flops = (8.0 * f.nb * f.nb * iters_mean + 8.0 * f.nn * f.nb) * E if has_pf else 0.0
    pf_peak = peaks.get("bf16_tflops", 1590.0) * (0.5 if PF_KERNEL == "tc" else 1.0)
    pf_peak_src = ("measured bf16 (= fp16 dense), " if PF_KERNEL != "tc" else "0.5 x measured bf16 (tf32 dense), ") + peak_src
    hook = 1 if getattr(env, "_penalty", None) is not None else 0

    def roof(kernel, alg_bytes, ms, extra=None):
        gbs = alg_bytes / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
        cap = ncu.get(kernel, {})
        r = {"kernel": kernel, "bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm,
             "traffic": cap.get("traffic"), "traffic_source": ncu.get("_source") if cap else None,
             "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": ms}
        if extra:
            r.update(extra)
        return r

    def tensor_part(kernel, ms):
        tfs = flops / (ms * 1e-3) / 1e12 if ms > 0 else 0.0
        return {"algorithmic_flops_per_launch": flops, "mean_iterations": iters_mean,
                "tensor": {"achieved_tflops": tfs, "peak_tflops": pf_peak, "frac": tfs / pf_peak,
                           "peak_source": pf_peak_src,
                           "pipe_active_pct_ncu": ncu.get(kernel, {}).get("tensor_pct")}}

    rooflines = {}
    if fused:
        # whole step in one kernel: the components' bytes + the power flow's state and results;
        # the agents' power, the rewards before the penalty and the second read of the episode
        # returns never leave the chip
        pf_bytes = (16.0 * f.nb * 2 + 8.0 * f.nn + 16.0 + 8.0 * A + 4.0 + 8.0) * E
        rooflines["step_fused_kernel"] = roof("step_fused_kernel", comp_bytes + pf_bytes, k_a_ms,
                                              tensor_part("step_fused_kernel", k_a_ms))
        dominant = rooflines["step_fused_kernel"]
        share = {"step_fused_kernel": 1.0}
    else:
        rooflines["component_kernel"] = roof("component_kernel", comp_bytes, k_a_ms,
                                             {"survey_bytes_per_launch": survey_bytes})
        dominant = rooflines["component_kernel"]
        share = {"components": k_a_ms / max(k_a_ms + pf_ms, 1e-12), "powerflow": pf_ms / max(k_a_ms + pf_ms, 1e-12)}
        if has_pf:
            # per env: agents' power in, warm-start branch voltages in and out, node magnitudes,
            # min/max, bus voltages, iterations, and -- with the penalty hook -- rewards in/out
            pf_bytes = (8.0 * A + 16.0 * f.nb * 2 + 16.0 * A * hook + 8.0 * f.nn + 16.0 + 8.0 * A + 4.0) * E
            kname = {"tc": "pf_tc_kernel", "tc2": "pf_tc2_kernel"}.get(PF_KERNEL, "pf_fixed_point_kernel")
            rooflines[kname] = roof(kname, pf_bytes, pf_ms, tensor_part(kname, pf_ms))
            rooflines[kname]["arithmetic_intensity_flop_per_byte"] = flops / pf_bytes
            rooflines[kname]["ridge_flop_per_byte"] = pf_peak * 1e12 / (hbm * 1e9)
            if pf_ms > k_a_ms:
                dominant = rooflines[kname]
    out.update({"rooflines": rooflines, "dominant": dominant, "kernel_share": share})
    return out


def measure_rotating(workload, E, K, W, dev, first_env):
    """K steps back to back over R independent batches of E envs in rotation (R x per-batch state and
    buffers > 1.5 x L2, so every step finds its own state cold), timed with ONE event pair."""
    import numpy as np
    import torch

    from powergridworld_b200 import _native as N

    l2 = torch.cuda.get_device_properties(dev).L2_cache_size
    per_env = (first_env._b.sd_rows + first_env.act_dim + first_env.obs_dim + 4 * len(first_env.agents)
               + (first_env.pf_solver.feeder.nn + 2 * 16 + 4 if first_env.pf_solver else 0)) * 8
    R = int(np.ceil(1.5 * l2 / (per_env * E)))
    envs, acts = [], []
    rng = np.random.default_rng(5)
    gen = torch.Generator(device=dev)
    gen.manual_seed(99)
    for r in range(R):
        e = _make_env(None, workload=workload, num_envs=E, device=dev)
        if PF_KERNEL != "fp64" and e.pf_solver is not None:
            e.set_option(N.OPT_PF_KERNEL, {"tc": 1, "tc2": 2}[PF_KERNEL])
        if GRAPHS is not None:
            e.set_option(N.OPT_GRAPHS, GRAPHS)
        e.reset_batch(torch.as_tensor(30.0 + 5.0 * rng.uniform(-1, 1, size=(e.num_storage, E))).to(dev))
        envs.append(e)
        # two action buffers per batch in turn: the node parameters are rewritten every step (as for a
        # policy's fresh tensor) and carry the event index
        acts.append([torch.rand((e.act_dim, E), generator=gen, device=dev, dtype=torch.float64) * 2.0 - 1.0
                     for _ in range(2)])
    for i in range(max(W, 3) * R):
        envs[i % R].step_batch(acts[i % R][(i // R) % 2])
    torch.cuda.synchronize(dev)
    steps = min(K, (envs[0].episode_length - max(W, 3) - 1)) * 1
    steps = max(R, steps // R * R)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t0 = time.perf_counter()
    for i in range(steps):
        envs[i % R].step_batch(acts[i % R][(i // R) % 2])
    host_us = (time.perf_counter() - t0) * 1e6 / steps
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    out = {"value": E / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps, "batches": R,
           "envs_per_batch": E, "state_bytes_all_batches": int(per_env * E * R), "l2_bytes": int(l2),
           "host_submit_us_per_step": host_us,
           "l2": "cold by construction: the batches' state exceeds the L2 1.5x, each batch is stepped once per "
                 "rotation; no flush kernel and no per-step event pair inside the timed window"}
    for e in envs:
        e.close()
    return out


def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    K, W = args.steps, max(args.warmup, 3)

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_throughput()                   # before CUDA is initialised (fork)
        if _reference_classes_available():
            cpu_base["reference_classes"] = cpu_throughput(total_seconds_target=8.0, kind="reference")

    numa_cpus = _bind_to_gpu_numa(local)
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        _init_nccl(dev)
    E = ENVS_PER_GPU
    stream = torch.cuda.Stream(dev)                   # a non-default stream: pgw_step replays its graph
    torch.cuda.set_stream(stream)
    m = measure(WORKLOAD, E, K, W, dev, world, rank, headline=True, pdl=args.pdl,
                dump_dir=args.dump_outputs)
    env, A, has_pf = m["env"], m["A"], m["has_pf"]
    barrier, one_step, begin_pass, soc = m["barrier"], m["one_step"], m["begin_pass"], m["soc"]

    # ---- same loop with a warm L2 (reported next to the headline, not instead of it)
    begin_pass()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    t_sub0 = time.perf_counter()
    for i in range(K):
        one_step(W + i)
    host_submit_us = (time.perf_counter() - t_sub0) * 1e6 / K
    ev1.record()
    barrier()
    warm_ms = ev0.elapsed_time(ev1) / K

    # ---- back to back with a cold L2 by construction: R independent batches of E envs stepped in turn,
    #      their state larger than the L2 (the timing rules' other option: "inputs larger than L2"), one
    #      event pair around the K launches -- no flush kernel and no per-step event pair inside the window
    rotating = None
    if rank == 0 and world == 1 and WORKLOAD == "c1" and not args.no_extra:
        rotating = measure_rotating(WORKLOAD, E, K, W, dev, env)

    # ---- end to end: host buffers in, host buffers out, every step (the public host-buffer call;
    #      page-locked buffers are read and written in place by the step's kernels over PCIe)
    host_act = [torch.rand((env.act_dim, E), dtype=torch.float64).mul_(2).sub_(1).pin_memory()
                for _ in range(4)]
    env.reset_host(soc.cpu().numpy())
    for i in range(3):
        env.step_host(host_act[i % 4])
    barrier()
    ke = min(K, 100)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t_host0 = time.perf_counter()
    for i in range(ke):
        if env._needs_reset:
            env.reset_host(soc.cpu().numpy())
        obs, rew, done = env.step_host(host_act[i % 4])
    e1.record()
    torch.cuda.synchronize(dev)
    e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - t_host0) * 1e3)
    if world > 1:
        t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_value = E * world * ke / (e2e_ms * 1e-3)
    h2d = env.act_dim * E * 8
    d2h = env.obs_dim * E * 8 + A * E * 8 + E

    # ---- the other single-GPU configurations of BASELINE.json, a few steps each (rank 0, N = 1)
    extra = {}
    if rank == 0 and world == 1 and WORKLOAD == "c1" and not args.no_extra:
        env.close()
        del m["env"]
        for name, wl, e_n in (("c1x64", "c1", 262144), ("c2", "c2", 65536), ("c3", "c3", 16384),
                                 ("hs", "hs", 262144)):
            try:
                x = measure(wl, e_n, 20, 5, dev)
                extra[name] = {"workload": _config(1, wl, e_n)["workload"], "envs": e_n, "value": x["value"],
                               "unit": UNIT, "ms_per_step": x["ms_per_step"], "steps": 20, "warmup": 5,
                               "gpu_launches": x["launches"], "roofline": x["dominant"],
                               "rooflines": x["rooflines"], "kernel_share": x["kernel_share"]}
                x["env"].close()
            except Exception as exc:                  # a leg that fails must not take the headline down
                extra[name] = {"error": f"{type(exc).__name__}: {exc}"}

        # C4 (the scenario mix: three handles on three streams) in a process of its own
        try:
            import subprocess
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--workload", "c4", "--steps", "20",
                                "--warmup", "5", "--pf-kernel", PF_KERNEL], capture_output=True, text=True,
                               timeout=300)
            c4 = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
            extra["c4"] = {k: c4[k] for k in ("config", "value", "unit", "ms_per_step", "steps", "warmup",
                                             "gpu_launches", "roofline", "e2e", "agent_steps_per_s")}
            extra["c4"]["envs"] = c4["config"]["envs_per_gpu"]
        except Exception as exc:
            extra["c4"] = {"error": f"{type(exc).__name__}: {exc}"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": m["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": _dtype_label(has_pf), "data": "synthetic",
            "config": _config(world),
            "agent_steps_per_s": m["value"] * A,
            "clocks": m["clocks"],
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / ke, "steps": ke,
                    "path": "pgw_step_host on page-locked buffers: the kernels read the actions and write "
                            "observations / rewards / done flags in host memory (zero-copy over PCIe)"},
            "gpu_launches": m["launches"],
            # `roofline` = the kernel with the largest share of the step; all of them under `rooflines`
            "roofline": m["dominant"],
            "rooflines": m["rooflines"],
            "kernel_share": m["kernel_share"],
            "step_kernels": list(m["rooflines"].keys()),
            "collective_in_timed_region": False,
            "scaling_note": "value times each step on the device (CUDA events, max over ranks): the env shards "
                            "never exchange data, the statistics all-reduce runs after the timed steps; e2e "
                            "(host buffers, wall clock, max over ranks) is the figure that sees the host",
            "warm_l2": {"ms_per_step": warm_ms, "value": E * world / (warm_ms * 1e-3),
                        "host_submit_us_per_step": host_submit_us,
                        "note": "K launches back to back on one batch, one event pair; a step cannot be "
                                "shorter than the host needs to submit it"},
            "stats": [float(x) for x in m["stats"].cpu()],
            "wall_s_timed_region": m["wall"],
            "parity": {"voltages_pu": 1e-6, "rewards": "rtol 1e-5, atol 2e-5 (float64 polish of the tcgen05 solve)",
                       "components": "bit-identical to the two-kernel path; <= 6e-14 relative to the oracle",
                       "tests": "tests/test_gpu_parity.py, tests/test_gpu_api.py"},
            "numa_cpus_bound": numa_cpus,
        }
        if rotating is not None:
            line["back_to_back_cold"] = rotating
        if extra:
            line["extra"] = {"workloads": extra}
        if cpu_base is not None:
            line["cpu_baseline"] = cpu_base
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------- C4: scenario mix
C4_MIX = (("c1", 65536), ("c3", 16384), ("c2", 49152))   # 131 072 envs per GPU, 1 048 576 on 8


def _init_nccl(dev):
    """init_process_group with eager communicator creation.  NCCL announces its version on the
    process's stdout when NCCL_DEBUG is set (the GPU boxes set it): stdout carries the one JSON
    line of the contract and nothing else, so file descriptor 1 points at stderr meanwhile."""
    import torch
    import torch.distributed as dist
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier()
        torch.cuda.synchronize(dev)
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)


def run_mix(args):
    """BASELINE configs[4]: heterogeneous scenario mix, ~1 M env instances over 8 GPUs.  Every GPU
    holds three env batches (IEEE-13 buildings, 123-bus DER feeder, component-only EV station),
    each with its own device handle and stream; one "step" advances all of them once, the
    batches overlapping on the GPU.  The only collective is the statistics all-reduce."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from powergridworld_b200 import _native as N

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    K, W = args.steps, max(args.warmup, 3)
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        _init_nccl(dev)
    scale = args.envs / 131072.0 if args.envs else 1.0
    parts = []
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    rng = np.random.default_rng(rank)
    for wl, n in C4_MIX:
        E = max(128, int(n * scale) // 128 * 128)
        env = _make_env(None, workload=wl, num_envs=E, device=dev)
        if env.pf_solver is not None and PF_KERNEL != "fp64":
            env.set_option(N.OPT_PF_KERNEL, {"tc": 1, "tc2": 2}[PF_KERNEL])
        stream = torch.cuda.Stream(dev)
        acts = torch.rand((4, env.act_dim, E), generator=gen, device=dev, dtype=torch.float64) * 2 - 1
        soc = torch.as_tensor(30.0 + 5.0 * rng.uniform(-1, 1, size=(env.num_storage, E))).to(dev)
        parts.append({"wl": wl, "E": E, "env": env, "stream": stream, "acts": acts, "soc": soc,
                      "done": torch.cuda.Event()})
    total_envs = sum(pt["E"] for pt in parts)
    agent_steps = sum(pt["E"] * len(pt["env"].agents) for pt in parts)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    main_stream = torch.cuda.current_stream(dev)

    def step_all(i, fence=None):
        for pt in parts:
            with torch.cuda.stream(pt["stream"]):
                if fence is not None:
                    pt["stream"].wait_event(fence)
                if pt["env"]._needs_reset:
                    pt["env"].reset_batch(pt["soc"])
                pt["env"].step_batch(pt["acts"][i % 4])
                pt["done"].record(pt["stream"])
        for pt in parts:
            main_stream.wait_event(pt["done"])

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for pt in parts:
        with torch.cuda.stream(pt["stream"]):
            pt["env"].reset_batch(pt["soc"])
    for i in range(max(W, 6)):                        # captures the step graphs (untimed)
        step_all(i)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = sum(pt["env"].launch_count for pt in parts)
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    for i in range(K):
        flush.zero_()
        starts[i].record(main_stream)
        step_all(W + i, fence=starts[i])
        ends[i].record(main_stream)
    barrier()
    if args.dump_outputs is not None and rank == 0:
        _dump_outputs(args.dump_outputs, {f"{pt['wl']}_": pt["env"] for pt in parts})
    launches = sum(pt["env"].launch_count for pt in parts) - launches0
    sampler.stop_flag = True
    total_ms = float(sum(s_.elapsed_time(e_) for s_, e_ in zip(starts, ends)))
    stats = None
    for pt in parts:                                   # the only collective of the path
        with torch.cuda.stream(pt["stream"]):
            st = pt["env"].all_reduce_stats()
        torch.cuda.synchronize(dev)
        stats = st.clone() if stats is None else torch.cat([stats[:6] + st[:6], torch.minimum(
            stats[6:7], st[6:7]), torch.maximum(stats[7:8], st[7:8])])
    if world > 1:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    value = total_envs * world * K / (total_ms * 1e-3)

    # end to end: host buffers in and out for every batch, every step
    host_act = [pt["acts"][0].cpu().pin_memory() for pt in parts]
    for pt in parts:
        with torch.cuda.stream(pt["stream"]):
            pt["env"].reset_host(pt["soc"].cpu().numpy())
    barrier()
    ke = min(K, 20)
    t0 = time.perf_counter()
    for i in range(ke):
        for pt, ha in zip(parts, host_act):
            with torch.cuda.stream(pt["stream"]):
                if pt["env"]._needs_reset:
                    pt["env"].reset_host(pt["soc"].cpu().numpy())
                pt["env"].step_host(ha)
    torch.cuda.synchronize(dev)
    e2e_ms = (time.perf_counter() - t0) * 1e3
    if world > 1:
        t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    h2d = sum(pt["env"].act_dim * pt["E"] * 8 for pt in parts)
    d2h = sum((pt["env"].obs_dim + len(pt["env"].agents)) * pt["E"] * 8 + pt["E"] for pt in parts)
    if rank == 0:
        peaks, peak_src = _peaks()
        alg = float(sum(SURVEY_BYTES[pt["wl"]] * pt["E"] for pt in parts))
        step_ms = total_ms / K
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "C4: scenario mix per GPU = " + " + ".join(
                f"{pt['E']} x {pt['wl'].upper()}" for pt in parts) + ", one device handle and stream "
                "per scenario", "envs_per_gpu": total_envs, "global_envs": total_envs * world,
                "parallelism": f"env-sharded x{world}", "pf_kernel": _PF_NAMES[PF_KERNEL],
                "l2": "flushed between timed steps (256 MiB write)"},
            "agent_steps_per_s": agent_steps * world * K / (total_ms * 1e-3),
            "clocks": sampler.summary(),
            "e2e": {"value": total_envs * world * ke / (e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / ke, "steps": ke},
            "gpu_launches": int(launches),
            "roofline": {"kernel": "component_kernel (all three batches; whole step as the "
                         "denominator, power flow included)", "bound": "hbm",
                         "achieved": alg / (step_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"],
                         "unit": "GB/s", "frac": alg / (step_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                         "traffic": None, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg},
            "stats": [float(x) for x in stats.cpu()],
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    global ENVS_PER_GPU, PF_KERNEL, WORKLOAD, GRAPHS
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the C1x64 / C2 / C3 legs after the headline")
    ap.add_argument("--pdl", type=int, default=1, choices=[0, 1],
                    help="power flow as a programmatic dependent launch of the component kernel "
                         "(library default 1; applies to feeders whose solver CTA leaves room on the SM)")
    ap.add_argument("--graphs", type=int, default=None, choices=[0, 1],
                    help="PGW_OPT_GRAPHS override (library default: the fused step kernel is launched directly, "
                         "the two-kernel step replays one captured graph)")
    ap.add_argument("--envs", type=int, default=None,
                    help="envs per GPU (default: 4096 for C1, 65536 for C2, 16384 for C3)")
    ap.add_argument("--pf-kernel", default=PF_KERNEL, choices=["fp64", "tc", "tc2"])
    ap.add_argument("--workload", default="c1", choices=["c1", "c2", "c3", "c4", "hs"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the observations, rewards and done flags of the last timed step as "
                         "DIR/*.npy (rank 0's envs; a seeded sample of env columns above 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    if args.envs is None and args.workload != "c4":
        args.envs = {"c1": 4096, "c2": 65536, "c3": 16384, "hs": 262144}[args.workload]
    ENVS_PER_GPU, PF_KERNEL, WORKLOAD, GRAPHS = args.envs, args.pf_kernel, args.workload, args.graphs
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "c4":
        run_mix(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
