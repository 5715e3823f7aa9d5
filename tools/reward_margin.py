#!/usr/bin/env python
"""How close the benchmarked solver's rewards come to the parity bound over whole episodes: fused step
kernel (float32 fixed point + float64 polish) against the FP64 SIMT solver, 4096 envs x 2 full episodes of
random actions; prints the worst |error| / (2e-5 + 1e-5 |reward|) (must stay below 1) and the worst
absolute error."""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from powergridworld_b200 import _native as N                                   # noqa: E402
from powergridworld_b200.scenarios import bench as SB                          # noqa: E402

E = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
st = torch.cuda.Stream()
torch.cuda.set_stream(st)
a = SB.c1_env(num_envs=E, pf_kernel="tc2")          # fused kernel (automatic at this size)
b = SB.c1_env(num_envs=E, pf_kernel="fp64")
if os.environ.get("PGW_TOL_NANO"):                   # convergence threshold of the fixed-point loop, 1e-9 p.u. units
    a.set_option(N.OPT_PF_TC_TOL_NANO, int(os.environ["PGW_TOL_NANO"]))
gen = torch.Generator(device="cuda")
gen.manual_seed(7)
worst_ratio, worst_abs, worst_v = 0.0, 0.0, 0.0
for ep in range(2):
    soc = torch.rand((a.num_storage, E), generator=gen, device="cuda", dtype=torch.float64) * 40 + 5
    a.reset_batch(soc), b.reset_batch(soc)
    for t in range(a.episode_length):
        act = torch.rand((a.act_dim, E), generator=gen, device="cuda", dtype=torch.float64) * 2.2 - 1.1
        _, ra, _, _ = a.step_batch(act)
        _, rb, _, _ = b.step_batch(act)
        err = (ra - rb).abs()
        worst_ratio = max(worst_ratio, float((err / (2e-5 + 1e-5 * rb.abs())).max()))
        worst_abs = max(worst_abs, float(err.max()))
        if t % 40 == 0:
            worst_v = max(worst_v, float((a.get_field(N.FIELD_VOLTAGES) - b.get_field(N.FIELD_VOLTAGES)).abs().max()))
iters = float(a.get_field(N.FIELD_PF_ITERS).abs().double().mean())
print(json.dumps({"tol_nano": os.environ.get("PGW_TOL_NANO", "default"), "mean_iterations_last_step": iters, "envs": E, "episodes": 2, "steps": 2 * a.episode_length, "launches_per_step": a.launch_count / (2 * a.episode_length + 2),
                  "worst_error_over_bound": worst_ratio, "worst_abs_reward_error": worst_abs,
                  "worst_voltage_error_pu": worst_v}))
