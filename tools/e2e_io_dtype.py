"""GPU measurement: float64 against float32 actions / observations (``io_dtype``) on the end-to-end
host-buffer step and on the device step, in one process so that both forms run on the same card in
the same session.  One JSON line per case goes to profiles/r4_e2e_io_dtype.jsonl (``--out``).

Cases
  * C1 at 4096 envs, zero-copy ``step_host`` (page-locked buffers read / written in place by the
    fused kernel): float64 and float32 alternated ``--rounds`` times, wall microseconds per call
    (the call synchronises), env-steps/s, and the GPU time of the call from CUDA events around it.
  * the split of that step (as tools/e2e_probe2.py): actions on the device and results in host
    memory, and the reverse, through the raw C calls, for both forms.
  * the same alternation on the device path (``step_batch``).
  * the host path of C2 (65 536 envs), C3 (4096) and HS (65 536).
  * the stagger of the zero-copy fused step for 128-byte float32 action rows
    (PGW_STAGGER_CYCLES_PER_ROW sweep), float32 and float64.
  * the kernel names torch.profiler records for the float32 env (proof that the IO32 instantiations
    ran).
Every line carries the card's name, power limit and SM clock (nvidia-smi, read in the same run),
the warm-up steps and whether the L2 was flushed before each timed step (it is not: the step's
device working set at C1 is a few MB, and its host buffers cross PCIe on every call anyway)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from powergridworld_b200 import _native as N                                   # noqa: E402
from powergridworld_b200.scenarios import bench as SB                          # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    dev = torch.cuda.current_device()
    vals = [v.strip() for v in out[dev].split(",")] if len(out) > dev else []
    return dict(zip(q.split(","), vals))


def emit(fh, rec, args):
    rec = dict(rec, session=args.session, gpu=gpu_info(), warmup_steps=args.warmup,
               l2_flushed_before_each_step=False)
    line = json.dumps(rec)
    print(line, flush=True)
    fh.write(line + "\n")
    fh.flush()


def make(workload, E, io_dtype):
    if workload == "c1":
        return SB.c1_env(num_envs=E, pf_kernel="tc2", io_dtype=io_dtype)
    if workload == "c3":
        return SB.c3_env(num_envs=E, pf_kernel="tc2", io_dtype=io_dtype)
    return SB.make_env(workload, num_envs=E, io_dtype=io_dtype)


def soc_of(env):
    return np.full((env.num_storage, env.num_envs), 30.0) if env.num_storage else None


def pinned_actions(env, n=4):
    dt = torch.float32 if env.io_dtype == "float32" else torch.float64
    return [(torch.rand((env.act_dim, env.num_envs), dtype=torch.float64) * 2 - 1).to(dt).pin_memory()
            for _ in range(n)]


def time_host(env, acts, warm, steps):
    """Wall us per step_host call, median GPU us of the call (events around it)."""
    env.reset_host(soc_of(env))
    for i in range(warm):
        env.step_host(acts[i % len(acts)])
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    t0 = time.perf_counter()
    for i in range(steps):
        ev[i][0].record()
        env.step_host(acts[i % len(acts)])
        ev[i][1].record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / steps * 1e6
    gpu = np.array([a.elapsed_time(b) * 1e3 for a, b in ev])
    return wall, float(np.median(gpu))


def time_device(env, acts, warm, steps):
    env.reset_batch(soc_of(env))
    dev = [a.cuda() for a in acts]
    for i in range(warm):
        env.step_batch(dev[i % len(dev)])
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    t0 = time.perf_counter()
    for i in range(steps):
        ev[i][0].record()
        env.step_batch(dev[i % len(dev)])
        ev[i][1].record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / steps * 1e6
    gpu = np.array([a.elapsed_time(b) * 1e3 for a, b in ev])
    return wall, float(np.median(gpu))


def time_split(env, acts, warm, steps):
    """GPU us of the raw step with (actions on the device, outputs in host memory) and the reverse."""
    f32 = env.io_dtype == "float32"
    step = env._lib.pgw_step_f32 if f32 else env._lib.pgw_step
    pin = env._pinned()
    a_dev = acts[0].cuda()
    s = torch.cuda.current_stream().cuda_stream
    out = {}
    for label, ap, op, rp, dp in (
            ("actions device, outputs host", a_dev.data_ptr(), pin["obs"].data_ptr(), pin["rew"].data_ptr(),
             pin["done"].data_ptr()),
            ("actions host, outputs device", acts[0].data_ptr(), env.obs.data_ptr(), env.rew.data_ptr(),
             env.done.data_ptr()),
            ("actions device, outputs device", a_dev.data_ptr(), env.obs.data_ptr(), env.rew.data_ptr(),
             env.done.data_ptr())):
        env.reset_batch(soc_of(env))
        for _ in range(warm):
            N.check(step(env._h, ap, op, rp, dp, s))
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for i in range(steps):
            ev[i][0].record()
            N.check(step(env._h, ap, op, rp, dp, s))
            ev[i][1].record()
        torch.cuda.synchronize()
        out[label] = float(np.median([a.elapsed_time(b) * 1e3 for a, b in ev]))
    env._needs_reset = True
    return out


def bytes_per_step(env):
    el = 4 if env.io_dtype == "float32" else 8
    E = env.num_envs
    return {"actions": env.act_dim * E * el, "obs": env.obs_dim * E * el, "rew": len(env.agents) * E * 8,
            "done": E}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_e2e_io_dtype.jsonl"))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--stagger", default="0,2,3,5,8,10,15,20")
    ap.add_argument("--session", type=int, default=0, help="label of this run, recorded in every line")
    ap.add_argument("--append", action="store_true", help="append to --out (several runs in one file)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs the GPU"
    st = torch.cuda.Stream()
    torch.cuda.set_stream(st)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a" if args.append else "w") as fh:
        # ---- C1, 4096 envs: zero-copy host step and device step, float64 / float32 alternated
        envs = {dt: make("c1", 4096, dt) for dt in ("float64", "float32")}
        acts = {dt: pinned_actions(e) for dt, e in envs.items()}
        steps = min(args.steps, envs["float64"].episode_length - args.warmup - 1)
        for path, timer in (("host zero-copy", time_host), ("device", time_device)):
            for r in range(args.rounds):
                for dt, env in envs.items():
                    wall, gpu = timer(env, acts[dt], args.warmup, steps)
                    emit(fh, {"case": f"c1 {path}", "workload": "c1", "envs": 4096, "io_dtype": dt, "round": r,
                              "timed_steps": steps, "wall_us_per_step": wall, "gpu_us_per_step_median": gpu,
                              "env_steps_per_s": 4096 / wall * 1e6, "bytes_per_step": bytes_per_step(env)}, args)
        for r in range(args.rounds):
            for dt, env in envs.items():
                emit(fh, {"case": "c1 split", "workload": "c1", "envs": 4096, "io_dtype": dt, "round": r,
                          "timed_steps": steps, "gpu_us_median": time_split(env, acts[dt], args.warmup, steps)},
                     args)
        # ---- stagger of the zero-copy fused step per action row
        for dt, env in envs.items():
            for v in [int(x) for x in args.stagger.split(",")]:
                os.environ["PGW_STAGGER_CYCLES_PER_ROW"] = str(v)
                env.set_option(N.OPT_GRAPHS, 1)           # drops the captured graphs: re-captured with v
                res = [time_host(env, acts[dt], args.warmup, steps) for _ in range(args.rounds)]
                emit(fh, {"case": "c1 stagger sweep", "workload": "c1", "envs": 4096, "io_dtype": dt,
                          "stagger_cycles_per_row": v, "timed_steps": steps,
                          "wall_us_per_step": [w for w, _ in res], "gpu_us_per_step_median": [g for _, g in res]},
                     args)
            os.environ.pop("PGW_STAGGER_CYCLES_PER_ROW", None)
            env.set_option(N.OPT_GRAPHS, 1)
        # ---- kernel names of the float32 env (device step and host step)
        from torch.profiler import ProfilerActivity, profile
        e32 = envs["float32"]
        e32.reset_batch(soc_of(e32))
        a = acts["float32"][0].cuda()
        e32.set_option(N.OPT_GRAPHS, 0)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            e32.step_batch(a)
            torch.cuda.synchronize()
        e32.set_option(N.OPT_GRAPHS, 1)
        names = sorted({ev.name for ev in prof.events() if "pgw::" in ev.name})
        emit(fh, {"case": "kernel names", "workload": "c1", "io_dtype": "float32", "kernels": names}, args)
        for env in envs.values():
            env.close()
        # ---- host path of C2, C3 and HS
        for wl, E in (("c2", 65536), ("c3", 4096), ("hs", 65536)):
            envs = {dt: make(wl, E, dt) for dt in ("float64", "float32")}
            acts = {dt: pinned_actions(e) for dt, e in envs.items()}
            steps = min(args.steps, envs["float64"].episode_length - args.warmup - 1)
            for r in range(args.rounds):
                for dt, env in envs.items():
                    wall, gpu = time_host(env, acts[dt], args.warmup, steps)
                    emit(fh, {"case": f"{wl} host zero-copy", "workload": wl, "envs": E, "io_dtype": dt,
                              "round": r, "timed_steps": steps, "wall_us_per_step": wall,
                              "gpu_us_per_step_median": gpu, "env_steps_per_s": E / wall * 1e6,
                              "bytes_per_step": bytes_per_step(env)}, args)
            e32 = envs["float32"]
            e32.reset_host(soc_of(e32))
            e32.set_option(N.OPT_GRAPHS, 0)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                e32.step_host(acts["float32"][0])
            names = sorted({ev.name for ev in prof.events() if "pgw::" in ev.name})
            emit(fh, {"case": "kernel names", "workload": wl, "io_dtype": "float32", "kernels": names}, args)
            for env in envs.values():
                env.close()


if __name__ == "__main__":
    main()
