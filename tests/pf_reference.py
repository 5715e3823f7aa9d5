"""Float64 reference of the power flow of one env step, and the feeder variants that the
power-flow kernel tests run on: IEEE-13 variants for the fused step, truncations and an extension
of the packaged 123-bus-class feeder for the tc2 and FP64 kernels.

``solve64`` is the Z-bus fixed point u <- u0 - Zbb i(u) over a batch of envs with the load
characteristic of the device tables (models 1 and 2 clamp |u|^2 to their band, model 5 draws a
current of constant magnitude), iterated to max |d u| < 1e-13.  ``step_powers`` rebuilds the
branch powers that one step of a product env solves for from the env's event table and the
agents' real power, as the device does."""
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SHIPPED = "ieee_13_dss/IEEE13Nodeckt.dss"
LOADSHAPE = "ieee_13_dss/annual_hourly_load_profile.csv"

# variants of the published IEEE-13 feeder (golden/ieee13_original.dss): (loads dropped, loads
# renamed).  o16: 16 branches, models {1, 2, 5}, and the three-phase delta load 671 under a
# single-phase name, so that an agent on it feeds three delta legs and its bus node 671.1 is not a
# wye-load node; o15: an odd branch count with model 5; o14z: models {1, 2} only.
VARIANTS = {
    "o16": (("670a",), {"671": "671a"}),
    "o15": (("670a", "670b"), {}),
    "o14z": (("670a", "692", "611"), {}),
}
FEEDERS = ("shipped",) + tuple(VARIANTS)


def feeder_file(fid, directory):
    """Path of feeder ``fid``: the shipped IEEE13Nodeckt.dss, or a variant written to ``directory``."""
    if fid == "shipped":
        return SHIPPED
    drop, rename = VARIANTS[fid]
    out = []
    with open(os.path.join(GOLD, "ieee13_original.dss")) as fh:
        for line in fh:
            words = line.split()
            if len(words) > 1 and words[0] == "New" and words[1].startswith("Load."):
                name = words[1][5:]
                if name in drop:
                    continue
                if name in rename:
                    line = line.replace(f"Load.{name} ", f"Load.{rename[name]} ", 1)
            out.append(line)
    path = os.path.join(str(directory), f"ieee13_{fid}.dss")
    with open(path, "w") as fh:
        fh.writelines(out)
    return path


SYNTHETIC123 = os.path.join(os.path.dirname(os.path.dirname(GOLD)), "powergridworld_b200", "data",
                            "feeders", "synthetic123.dss")
# loads copied (same bus, same kW / kvar) under a new name and a new model for the x100 variant:
# 100 load branches, beyond tc2's 88 -> pf_fixed_point_kernel<32, 4, false> (nbp = 128)
EXTRA_LOADS = (("37a", 1), ("58a", 2), ("56b", 5), ("18a", 1), ("33b", 2), ("111c", 5), ("4a", 1),
               ("34a", 2), ("101a", 5), ("32b", 1), ("72a", 2), ("42a", 5), ("30b", 1), ("118a", 2),
               ("117b", 5))


def synthetic_feeder(directory, n_loads=85, extra=False):
    """The packaged 123-bus-class feeder (85 single-phase wye loads) with only its first
    ``n_loads`` loads, or (``extra``) with the loads of EXTRA_LOADS added as ``x<i>m<model>``."""
    out, seen = [], 0
    with open(SYNTHETIC123) as fh:
        for line in fh:
            if line.startswith("New Load."):
                seen += 1
                if seen > n_loads:
                    continue
                name = line.split()[1][5:]
                for i, (src, model) in enumerate(EXTRA_LOADS if extra else ()):
                    if src == name:
                        out.append(line.replace(f"Load.{name} ", f"Load.x{i}m{model} ", 1)
                                   .replace("Model=1", f"Model={model}"))
            out.append(line)
    path = os.path.join(str(directory), f"synthetic_{'x100' if extra else n_loads}.dss")
    with open(path, "w") as fh:
        fh.writelines(out)
    return path


def synthetic_config(ns, path, load_factor=0.9, hook_agents=0):
    """Scenario on a synthetic123-class feeder.  ``hook_agents`` = 0: storage and PV agents spread
    so that every rule of the branch powers and bus voltages is used -- three on the model-1 load
    37a (summed in agent order; the third bus voltage goes past the two per-branch slots), two on
    58a, one each on the model-5 load 5b and the model-2 load 20c (power ignored, bus voltage read),
    one on the bus 10a that carries no load, one on 7b (a load of the full feeder only) and one on
    4a.  ``hook_agents`` = n: n storage agents, all on 37a (the shared-penalty bus)."""
    import pandas as pd
    store = lambda kw: {"max_power": kw, "storage_range": (3., 80.)}
    if hook_agents:
        agents = [{"name": f"s{i}", "bus": "37a", "cls": ns.EnergyStorageEnv, "config": store(10. + i)}
                  for i in range(hook_agents)]
    else:
        pv = lambda scale: {"profile_csv": "pv_profile.csv", "scaling_factor": scale}
        roster = [("37a", ns.EnergyStorageEnv, store(60.)), ("37a", ns.PVEnv, pv(150.)),
                  ("37a", ns.EnergyStorageEnv, store(25.)), ("58a", ns.EnergyStorageEnv, store(40.)),
                  ("58a", ns.EnergyStorageEnv, store(15.)), ("5b", ns.EnergyStorageEnv, store(30.)),
                  ("20c", ns.EnergyStorageEnv, store(30.)), ("10a", ns.EnergyStorageEnv, store(20.)),
                  ("7b", ns.EnergyStorageEnv, store(35.)), ("4a", ns.PVEnv, pv(80.))]
        agents = [{"name": f"a{i}", "bus": bus, "cls": cls, "config": cfg}
                  for i, (bus, cls, cfg) in enumerate(roster)]
    return {"common_config": {"start_time": "08-12-2021 00:00:00", "end_time": "08-13-2021 00:00:00",
                              "control_timedelta": pd.Timedelta(300, "s")},
            "pf_config": {"cls": ns.OpenDSSSolver,
                          "config": {"feeder_file": path, "loadshape_file": LOADSHAPE,
                                     "system_load_rescale_factor": load_factor}},
            "agents": agents}


def band(f):
    """clamp band of |u|^2 and the load characteristic per branch: k = 1 / clamp (models 1, 2),
    1 / sqrt(clamp) with an open band (model 5)."""
    m = np.asarray(f.branch_model)
    lo = np.where(m == 2, 1.0, f.branch_vmin ** 2)
    hi = np.where(m == 2, 1.0, f.branch_vmax ** 2)
    lo = np.where(m == 5, 1e-30, lo)
    hi = np.where(m == 5, 3e38, hi)
    return lo, hi, m == 5


def solve64(f, s, tol=1e-13, max_iter=500):
    """Fixed point for complex branch powers ``s`` [nb, E] (MVA, p.u. of the feeder's base):
    branch voltages u [nb, E], branch currents i [nb, E], node magnitudes |w - Znb i| [nn, E]."""
    s = np.asarray(s, dtype=np.complex128).reshape(f.nb, -1)
    lo, hi, m5 = (x[:, None] for x in band(f))
    u0 = f.u0[:, None]

    def current(u):
        c = np.clip(np.abs(u) ** 2, lo, hi)
        return np.conj(s) * u / np.where(m5, np.sqrt(c), c)

    u = np.repeat(u0, s.shape[1], axis=1)
    for _ in range(max_iter):
        un = u0 - f.zbb @ current(u)
        d = np.abs(un - u).max()
        u = un
        if d < tol:
            break
    else:
        raise AssertionError(f"float64 reference did not converge: max |d u| = {d:.1e}")
    i = current(u)
    return u, i, np.abs(f.w[:, None] - f.znb @ i)


def step_powers(env, t, agent_p):
    """Branch powers [nb, E] of step ``t`` (0-based) of a product env: the event table's base
    loads (row t + 1; row 0 is the reset) plus, per load, the real power of the agents on it
    (``agent_p`` = FIELD_AGENT_P [A, E]) summed in agent order."""
    f = env.pf_solver.feeder
    nl, E = f.nl, agent_p.shape[1]
    row = env._dtab[t + 1]
    ctl = np.zeros((nl, E))
    for a, rec in enumerate(env._agent_recs):
        if rec.load_slot >= 0:
            ctl[rec.load_slot] += agent_p[a]
    kw = row[2:2 + nl, None] + ctl
    kvar = np.broadcast_to(row[2 + nl:2 + 2 * nl, None], kw.shape)
    return (kw + 1j * kvar)[f.branch_load] * f.branch_share[:, None] * 1e-3
