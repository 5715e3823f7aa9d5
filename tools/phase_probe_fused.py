#!/usr/bin/env python
"""Phase breakdown of step_fused_kernel from SM-clock stamps (instrumented build, see phase_probe.py).
    gpurun -- python tools/phase_probe_fused.py [envs]"""
import ctypes as C
import os
import subprocess
import sys

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from powergridworld_b200 import _native as N  # noqa: E402

SECOND = os.environ.get("PGW_PROBE_SECOND", "0") == "1"      # stamps of each CTA's second tile (build with
#                                                               -DPGW_STAMP_SECOND_TILE, run with PGW_FUSED_GRID=64)
# PGW_B200_LIB: another instrumented build (e.g. a parent commit's, for an A/B of the phases)
N.LIB_PATH = os.environ.get("PGW_B200_LIB") or os.path.join(
    ROOT, "tools", "_build", "libpgw_b200_phases2.so" if SECOND else "libpgw_b200_phases.so")
from powergridworld_b200.scenarios import bench as SB  # noqa: E402

PHASES = ["clock read + barrier init + TMA issue", "wait tables / component blob",
          "wait event row", "component steps (this thread's)", "barrier after the components",
          "agent sums + nominal power + first currents + barrier", "fixed-point loop",
          "float32 pre-sweep + float64 polish", "expansion + node magnitudes + barrier",
          "penalty, rewards, bus voltages"]


def main():
    E = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
    polish = int(os.environ.get("PGW_POLISH", "-1"))
    env = SB.c1_env(num_envs=E, pf_kernel="tc2")
    env.set_option(N.OPT_FUSED, 2)
    if polish >= 0:
        env.set_option(N.OPT_PF_POLISH, polish)
    lib = env._lib
    lib.pgw_debug_phases.restype = C.c_int
    lib.pgw_debug_phases.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    mhz = float(subprocess.run(["nvidia-smi", "--query-gpu=clocks.max.sm", "--format=csv,noheader,nounits"],
                               capture_output=True, text=True).stdout.split()[0])
    ctas = min((E + 31) // 32, int(os.environ.get("PGW_FUSED_GRID", "148")))
    rng = np.random.default_rng(0)
    soc = rng.uniform(10, 45, size=(env.num_storage, E))
    acts = torch.as_tensor(rng.uniform(-1, 1, size=(env.act_dim, E))).cuda()
    # PGW_PROBE_ROTATE=1: two action buffers in turn, i.e. the node parameters are rewritten every
    # step and carry the event index (the kernel skips its clock read), as in bench.py's loop
    rotate = os.environ.get("PGW_PROBE_ROTATE", "0") == "1"
    acts2 = acts.clone()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    st = torch.cuda.Stream()
    torch.cuda.set_stream(st)
    for cold in (True, False):
        env.reset_batch(soc)
        acc, ev = [], []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for t in range(60):
            if cold:
                flush.fill_(t & 0xFF)
            e0.record()
            env.step_batch(acts2 if (rotate and t % 2) else acts)
            e1.record()
            if t >= 20:
                buf = np.zeros((ctas, 16), dtype=np.int64)
                N.check(lib.pgw_debug_phases(env._h, buf.ctypes.data_as(C.c_void_p), ctas))
                acc.append(buf)
                ev.append(e0.elapsed_time(e1) * 1e3)
        a = np.stack(acc).astype(np.float64)
        d = np.diff(a[:, :, :11], axis=2) / mhz
        span = (a[:, :, 13].max(axis=1) - a[:, :, 12].min(axis=1)) / 1e3
        print(f"--- fused C1 E={E} ctas={ctas} {'event index from the host' if rotate else 'device clock'}, {'cold' if cold else 'warm'} L2, SM {mhz:.0f} MHz, iterations "
              f"{a[:, :, 11].mean():.2f}; first entry -> last exit {span.mean():.2f} us; step by CUDA events "
              f"{np.mean(ev):.2f} us")
        for k, name in enumerate(PHASES):
            if SECOND and k < 3:
                continue
            print(f"  {name:64s} mean {d[:, :, k].mean():6.2f} us   max-CTA mean {d[:, :, k].max(axis=1).mean():6.2f} us")
        tot = (a[:, :, 10] - a[:, :, 3]) / mhz if SECOND else (a[:, :, 14] - a[:, :, 0]) / mhz
        print(f"  {'entry -> exit':64s} mean {tot.mean():6.2f} us   max-CTA mean {tot.max(axis=1).mean():6.2f} us")


if __name__ == "__main__":
    main()
