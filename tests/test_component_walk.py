"""component_kernel on CTAs that walk several env blocks.

pgw_create splits a budget of CTAs over the agents by a cost estimate (PGW_CTA_BUDGET overrides the
budget).  Agent a gets n[a] CTAs, and CTA j of that agent walks the 64-env blocks j, j + n, j + 2n, ...
of [e_lo, e_hi).  Every workload of the benchmark walks, so each case here forces or reaches a walk
and checks:
- the CTA table against a Python mirror of the allocation, and the kernel template that ran;
- budget invariance: budget 1 (one CTA per agent walks every block), an uneven middle budget and the
  default budget give identical bits in every output and state field of every env;
- sampled envs (env 0, the first and last env of a block some CTA reaches after its first one, the
  last env of the partial block) against the float64 oracle;
- the staged host path in chunks (e_lo > 0) and float32 I/O under a walk, against the device path.
"""
import ctypes as C
import json
import math
import os
import re
import subprocess
import sys
import warnings

import numpy as np
import pandas as pd
import pytest

from powergridworld_b200 import _native as N
from powergridworld_b200.scenarios import bench as SB
from tests import scenarios as S
from tests import scenarios_hs as SH
from tests.flatten import flat_obs, unflatten_action
from tests.oracle_hs_ns import ORACLE_HS_NS as OHS
from tests.oracle_ns import ORACLE_NS as ONS, storage_socs_to_dict
from tests.product_ns import PRODUCT_NS as PNS

pytestmark = pytest.mark.gpu

F, T_ = "false", "true"
STATE_FIELDS = (N.FIELD_STATE_D, N.FIELD_STATE_I, N.FIELD_AGENT_P, N.FIELD_EP_RETURN)
PF_FIELDS = (N.FIELD_VBUS, N.FIELD_VOLTAGES, N.FIELD_PF_STATE)


def _torch():
    import torch
    return torch


# ------------------------------------------------------------------ the CTA table
def walk_plan(env, budget=None):
    """CTAs per agent: a mirror of build_comp_tables' water-filling allocation (tables.cpp)."""
    comps, ipar, agents = env._b.comps, env._b.ipar, list(env._agent_recs)
    A, blocks = len(agents), (env.num_envs + 63) // 64
    if budget is None:
        budget = 148 * 10 if A == 1 else 148 * 16
    w = []
    for ag in agents:
        x = 0.5
        for c in comps[ag.comp_begin:ag.comp_end]:
            if c.type in (N.EV, N.HS_EV):
                x += 1.0 + 0.04 * ipar[c.ipar_off]
            else:
                x += {N.BUILDING: 2.0, N.STORAGE: 0.8, N.HS_BEGIN: 1.0, N.HS_STORAGE: 1.0,
                      N.HS_DEVICES: 1.0}.get(c.type, 0.5)
        w.append(x)
    n, capped = [0] * A, [False] * A
    left, wleft, again = float(budget), sum(w), True
    while again:
        again = False
        for a in range(A):
            if not capped[a] and left * w[a] / wleft >= blocks:
                capped[a], n[a], again = True, blocks, True
                left -= blocks
                wleft -= w[a]
    for a in range(A):
        if not capped[a]:
            n[a] = max(1, min(blocks, math.ceil(left * w[a] / wleft)))
    return n


def _blocks_of(j, n, blocks):
    return len(range(j, blocks, n))


def _num_ctas(env):
    lib = env._lib
    lib.pgw_debug_num_comp_ctas.restype = C.c_int
    lib.pgw_debug_num_comp_ctas.argtypes = [C.c_void_p]
    return int(lib.pgw_debug_num_comp_ctas(env._h))


def _sample_envs(E, n):
    """env 0, the first and last env of the second block of the longest walk (block j + n of
    CTA j = 0), the last env of the last (possibly partial) block."""
    blocks = (E + 63) // 64
    out = {0, E - 1}
    walking = [na for na in n if na < blocks]
    if walking:                                  # CTA 0 of the agent with the fewest CTAs walks block na second
        na = min(walking)
        out |= {64 * na, min(E, 64 * na + 64) - 1}
    return out


def _component_kernels(env, act):
    """(kernel, template arguments) of the kernels of one step, from torch.profiler."""
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile
    env.set_option(N.OPT_GRAPHS, 0)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        env.step_batch(act)
        torch.cuda.synchronize()
    env.set_option(N.OPT_GRAPHS, 1)
    found = set()
    for ev in prof.events():
        m = re.search(r"(component_kernel|step_fused_kernel)<([^>]*)>", ev.name)
        if m:
            found.add((m.group(1),) + tuple(x.strip() for x in m.group(2).split(",")))
    return found


# ------------------------------------------------------------------ scenarios and their oracles
class NoPF:
    """Feeder-less oracle runs: the reference's MultiAgentEnv needs a solver object."""
    def __init__(self, **kw):
        pass

    def calculate_power_flow(self, *a, **k):
        pass

    def get_bus_voltages(self):
        return {}

    def get_bus_voltage_by_name(self, n):
        return 1.0


def _dt900(ns):
    return ns.MultiAgentEnv(**S.time_base_scenario(ns, ns.OpenDSSSolver, "dt900_max50"))


def _c1(ns):
    return ns.CoordinatedMultiBuildingControlEnv(**S.buildings_scenario(ns, ns.OpenDSSSolver, 1.2))


def _c3(ns):
    return ns.MultiAgentEnv(**S.der123_scenario(ns, ns.OpenDSSSolver))


def _building_subset(ns):
    """A stand-alone building with a non-default observation set: the table-driven path."""
    return {"common_config": {"start_time": "08-12-2020 00:00:00", "end_time": "08-13-2020 00:00:00",
                              "control_timedelta": pd.Timedelta(300, "s")},
            "agents": [{"name": "b", "bus": None, "cls": ns.FiveZoneROMThermalEnergyEnv,
                        "config": {"obs_config": {"zone_temp": (16., 40.), "outdoor_temp": (0., 56.),
                                                  "p_consumed": (0., 150.), "comfort_upper": (25., 30.)}}}]}


STATION = dict(num_vehicles=37, minutes_per_step=5, max_charge_rate_kw=7., peak_threshold=40.,
               vehicle_multiplier=2., rescale_spaces=True, randomize=True)
STATION_COMMON = {"start_time": "08-12-2020 00:00:00", "end_time": "08-13-2020 00:00:00",
                  "control_timedelta": pd.Timedelta(300, "s")}


def _house(step_meta):
    from tests.test_hs_tables_emu import house_batch
    return lambda **kw: house_batch("shipped", step_meta=step_meta, **kw)


# name: (product maker, E, middle budget, episodes (steps of each), options, component template,
#        oracle kind, tolerances (obs atol, reward rtol, reward atol, voltage atol))
MAE_TOL = (1e-7, 1e-5, 2e-5, 1e-7)
CASES = {
    # tc2 with the penalty hook: the power flow finishes the rewards; the fast building path
    "c1_tc2": (lambda **k: SB.c1_env(pf_kernel="tc2", **k), 1000, 8, (24,), ((N.OPT_FUSED, 0),),
               (F, F, F), ("mae", _c1), (2e-5, 1e-5, 2e-5, 5e-7)),
    # no hook: owns_reward and ep_ret; an EV charging set; max_episode_steps = 50 ends the episode
    # after 49 steps (done = 1 at the last), then a second reset
    "heterogeneous_dt900_max50": (lambda **k: PNS.MultiAgentEnv(
        **S.time_base_scenario(PNS, PNS.OpenDSSSolver, "dt900_max50"), **k), 1000, 8, (49, 6), (),
        (F, F, F), ("mae", _dt900), MAE_TOL),
    # no feeder: the component kernel advances the clock
    "c2": (SB.c2_env, 1000, 8, (40,), (), (F, F, F),
           ("mae", lambda ns: ns.MultiAgentEnv(**S.ev_pv_storage_scenario(ns, NoPF))), (1e-10, 1e-9, 1e-12, 0)),
    "building_obs_subset": (lambda **k: PNS.MultiAgentEnv(pf_config=None, **_building_subset(PNS), **k),
                            1000, 3, (30,), (), (F, F, F),
                            ("mae", lambda ns: ns.MultiAgentEnv(pf_config={"cls": NoPF, "config": {}},
                                                                **_building_subset(ns))), MAE_TOL),
    "ev_per_env_rosters": (lambda **k: PNS.MultiAgentEnv(
        common_config=STATION_COMMON, pf_config=None,
        agents=[{"name": "ev", "bus": None, "cls": PNS.EVChargingEnv, "config": STATION}], **k),
        1000, 3, (40,), (), (F, F, T_), ("station", None), (1e-9, 1e-9, 1e-12, 0)),
    "hs_house": (_house(False), 1000, 3, (30,), (), (T_, F, F), ("hs", None), (1e-12, 1e-12, 1e-13, 0)),
    "hs_house_telemetry": (_house(True), 1000, 3, (30,), (), (T_, T_, F), ("hs", None),
                           (1e-12, 1e-12, 1e-13, 0)),
    # 100 agents: walks at the default budget
    "c3_100_agents": (SB.c3_env, 3000, 500, (6,), (), (F, F, F), ("mae", _c3), (1e-9, 1e-9, 1e-10, 1e-8)),
    # the walk a user gets without any knob (790 CTAs per agent over 938 blocks), pdl_trigger 2
    "c1_60000_default": (lambda **k: SB.c1_env(pf_kernel="tc2", **k), 60000, None, (8,), ((N.OPT_FUSED, 0),),
                         (F, F, F), ("mae", _c1), (2e-5, 1e-5, 2e-5, 5e-7)),
}


def _make(monkeypatch, make, E, budget, options=(), **kw):
    """The env under CTA budget `budget` (None: the library default), with its CTA table checked."""
    if budget is None:
        monkeypatch.delenv("PGW_CTA_BUDGET", raising=False)
    else:
        monkeypatch.setenv("PGW_CTA_BUDGET", str(budget))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        env = make(num_envs=E, **kw)
    monkeypatch.delenv("PGW_CTA_BUDGET", raising=False)
    for opt, val in options:
        env.set_option(opt, val)
    n = walk_plan(env, budget)
    assert _num_ctas(env) == sum(n), (budget, n)
    return env, n


def _fields(env):
    fs = STATE_FIELDS + (PF_FIELDS if env.pf_solver is not None else ())
    return {f: env.get_field(f).clone() for f in fs}


def _bits(env, SI, e):
    """Charging sets of the top-level EV agents of env e, as Python ints."""
    out = []
    for ag in env.agents:
        if hasattr(ag, "num_vehicles"):
            off, words = ag._slot["si"]
            out.append(sum(int(np.uint32(SI[off + w, e])) << (32 * w) for w in range(words)))
    return out


def _run_budgets(monkeypatch, name, budgets):
    """Every budget's env in lock step on the same inputs: bit-identical outputs and fields.
    Returns the sampled columns of the first env (for the oracle) and the sample."""
    torch = _torch()
    make, E, mid, episodes, options, *_ = CASES[name]
    envs, plans = [], []
    for b in budgets:
        env, n = _make(monkeypatch, make, E, b, options)
        envs.append(env)
        plans.append(n)
    blocks = (E + 63) // 64
    for b, n in zip(budgets, plans):
        print(f"{name}: budget {b}: CTAs per agent {n}, blocks per CTA "
              f"{sorted({_blocks_of(j, na, blocks) for na in n for j in range(na)}, reverse=True)}")
    sample = sorted(set().union(*(_sample_envs(E, n) for n in plans)))
    ref = envs[0]
    rng = np.random.default_rng(list(CASES).index(name))
    gen = torch.Generator(device="cuda").manual_seed(7)
    lo, hi = (-1.2, 1.2)
    rec = []
    for ep, T in enumerate(episodes):
        soc = rng.uniform(5, 45, size=(ref.num_storage, E)) if ref.num_storage else None
        if name.startswith("hs"):                      # inside the shipped battery's [0.5, 14] kWh
            soc = rng.uniform(1, 13.5, size=(1, E))
        obs0 = []
        for env in envs:
            np.random.seed(100 + ep)                   # per-env rosters: the same draws for every budget
            obs0.append(env.reset_batch(soc).clone())
        for o in obs0[1:]:
            assert torch.equal(o, obs0[0]), f"{name} ep {ep}: reset observations"
        cur = {"soc": soc, "obs0": obs0[0][:, sample].cpu().numpy(), "steps": []}
        for t in range(T):
            act = (torch.rand((ref.act_dim, E), generator=gen, device="cuda", dtype=torch.float64)
                   * (hi - lo) + lo).contiguous()
            outs = []
            for env in envs:
                env.step_batch(act)
                outs.append((env.obs.clone(), env.rew.clone(), env.done.clone()))
            for k, o in enumerate(outs[1:], 1):
                for x, y, what in zip(o, outs[0], ("obs", "rew", "done")):
                    assert torch.equal(x, y), f"{name} ep {ep} t={t}: {what} of budget {budgets[k]}"
            if t in (0, T // 2, T - 1):
                f0 = _fields(ref)
                for k, env in enumerate(envs[1:], 1):
                    fk = _fields(env)
                    for f in f0:
                        assert torch.equal(fk[f], f0[f]), f"{name} ep {ep} t={t}: field {f} of budget {budgets[k]}"
            step = {"act": act[:, sample].cpu().numpy(), "obs": outs[0][0][:, sample].cpu().numpy(),
                    "rew": outs[0][1][:, sample].cpu().numpy(), "done": outs[0][2][sample].cpu().numpy()}
            if ref.pf_solver is not None:
                step["v"] = ref.get_field(N.FIELD_VOLTAGES)[:, sample].cpu().numpy()
            si = ref.get_field(N.FIELD_STATE_I)
            step["bits"] = [_bits(ref, si[:, sample].cpu().numpy(), k) for k in range(len(sample))]
            cur["steps"].append(step)
        rec.append(cur)
    info = {"node_names": ref.pf_solver.feeder.node_names if ref.pf_solver is not None else None,
            "plans": plans}
    for env in envs:
        env.close()
    return rec, sample, info


def _replay_oracle(name, rec, sample, info):
    """The sampled envs against the float64 oracle; returns the worst errors (obs, rew, v)."""
    _, E, _, _, _, _, (kind, ora), (o_tol, r_rtol, r_atol, v_tol) = CASES[name]
    worst = np.zeros(3)
    refs = {}
    for k, e in enumerate(sample):
        for ep, cur in enumerate(rec):
            if kind == "mae":
                if e not in refs:
                    with warnings.catch_warnings():
                        warnings.simplefilter("ignore")
                        refs[e] = ora(ONS)
                ref = refs[e]
                soc = cur["soc"]
                o0 = flat_obs(ref, ref.reset(init_storage=None if soc is None else
                                             storage_socs_to_dict(ref, soc[:, e])))
            elif kind == "hs":
                ref = refs.setdefault(e, OHS.HSMultiComponentEnv(**SH.shipped(OHS)))
                flat = lambda ob, h=ref: np.concatenate([np.asarray(ob[c.name], dtype=np.float64).ravel()
                                                          for c in h.envs])
                o0 = flat(ref.reset(init_storage=cur["soc"][0, e]))
            else:                                      # env e's roster is the (e + 1)-th draw
                ref = refs.setdefault(e, ONS.EVChargingEnv(**STATION))
                n_all = len(PNS.EVChargingEnv(**STATION)._roster_energy)
                np.random.seed(100 + ep)
                for _ in range(e):
                    np.random.choice(n_all, size=STATION["num_vehicles"], replace=False)
                o0 = ref.reset()[0]
            np.testing.assert_allclose(cur["obs0"][:, k], o0, rtol=0, atol=o_tol, err_msg=f"{name} env {e} reset")
            worst[0] = max(worst[0], np.abs(cur["obs0"][:, k] - o0).max())
            for t, st in enumerate(cur["steps"]):
                a = st["act"][:, k]
                if kind == "mae":
                    o, r, dn, _ = ref.step(unflatten_action(ref, a))
                    o, r, d = flat_obs(ref, o), np.array([r[x.name] for x in ref.agents]), dn["__all__"]
                elif kind == "hs":
                    o, r, d, _ = ref.step({c.name: a[i:i + 1] for i, c in enumerate(ref.envs)})
                    o, r = flat(o), np.array([r])
                else:
                    o, r = ref.step(a)[:2]
                    r, d = np.array([r]), False          # 40 of 288 steps: the episode runs on
                msg = f"{name} env {e} episode {ep} t={t}"
                np.testing.assert_allclose(st["obs"][:, k], o, rtol=0, atol=o_tol, err_msg=msg)
                np.testing.assert_allclose(st["rew"][:, k], r, rtol=r_rtol, atol=r_atol, err_msg=msg)
                assert bool(st["done"][k]) == bool(d), msg
                worst[0] = max(worst[0], np.abs(st["obs"][:, k] - o).max())
                worst[1] = max(worst[1], (np.abs(st["rew"][:, k] - r) / (r_atol + r_rtol * np.abs(r))).max())
                if "v" in st:
                    v = [ref.voltages[x] for x in info["node_names"]]
                    np.testing.assert_allclose(st["v"][:, k], v, rtol=0, atol=v_tol, err_msg=msg)
                    worst[2] = max(worst[2], np.abs(st["v"][:, k] - v).max())
                if kind == "mae":                        # the charging set, bit for bit
                    want = [sum(1 << int(i) for i in ag.charging_vehicles)
                            for ag in ref.agents if hasattr(ag, "charging_vehicles")]
                    assert st["bits"][k] == want, msg
    print(f"{name}: oracle on envs {sample}: worst obs error {worst[0]:.2e} (bound {o_tol:.0e}), "
          f"reward error {worst[1]:.3f} of its bound, voltage error {worst[2]:.2e} (bound {v_tol:.0e})")
    return worst


F32_CASES = ("c1_tc2", "hs_house")


def _probe_main():
    """Child process of the `kernels` fixture: one profiled step of every case, under its middle
    budget (float64) and under budget 1 (float32); prints {case/dtype: [kernel, template args]}."""
    torch = _torch()
    out = {}
    for name, dt, budget in ([(k, "float64", CASES[k][2]) for k in CASES] +
                             [(k, "float32", 1) for k in F32_CASES]):
        make, E, _, _, options, *_ = CASES[name]
        if budget is None:
            os.environ.pop("PGW_CTA_BUDGET", None)
        else:
            os.environ["PGW_CTA_BUDGET"] = str(budget)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            env = make(num_envs=E, io_dtype=dt)
        for opt, val in options:
            env.set_option(opt, val)
        env.reset_batch()
        act = torch.zeros((env.act_dim, E), dtype=getattr(torch, dt), device="cuda")
        out[f"{name}/{dt}"] = sorted(_component_kernels(env, act))
        env.close()
    print(json.dumps(out))


@pytest.fixture(scope="module")
def kernels():
    """The kernels each case launches, read in one child process: torch.profiler stops recording
    kernels after about a dozen sessions in one process (torch 2.11), and the rest of the suite
    already opens that many."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", "from tests.test_component_walk import _probe_main; _probe_main()"],
                       cwd=root, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    return {k: {tuple(x) for x in v} for k, v in json.loads(r.stdout.strip().splitlines()[-1]).items()}


@pytest.mark.parametrize("name", list(CASES))
def test_walk_matches_oracle_and_is_budget_invariant(monkeypatch, kernels, name):
    _, E, mid, _, _, want, *_ = CASES[name]
    assert kernels[f"{name}/float64"] == {("component_kernel",) + want + (F,)}, kernels[f"{name}/float64"]
    if E > 10000:                                      # budget 1 walks 938 blocks: one CTA per agent
        budgets = (1, None)
    else:
        budgets = (1, mid, None)
    rec, sample, info = _run_budgets(monkeypatch, name, budgets)
    if E > 10000:
        assert sum(info["plans"][-1]) > 148 * 4          # pdl_trigger 2: released at the end of each CTA
    _replay_oracle(name, rec, sample, info)


def test_worked_walks():
    """The allocation on the numbers the documentation quotes."""
    class Fake:
        pass

    def fake(weights_types, E):
        f = Fake()
        f.num_envs = E
        comps, recs, ipar = [], [], [0]
        for types in weights_types:
            b = len(comps)
            for t, nv in types:
                c = N.Component()
                c.type, c.ipar_off = t, len(ipar)
                ipar.append(nv)
                comps.append(c)
            recs.append(N.Agent(b, len(comps), 0, 0))
        f._b = Fake()
        f._b.comps, f._b.ipar = comps, ipar
        f._agent_recs = recs
        return f

    bldg = [(N.BUILDING, 0), (N.PV, 0), (N.STORAGE, 0)]
    c1 = fake([bldg] * 3, 1000)
    assert walk_plan(c1, 1) == [1, 1, 1]
    assert walk_plan(c1, 8) == [3, 3, 3]
    assert [_blocks_of(j, 3, 16) for j in range(3)] == [6, 5, 5]
    het = fake([bldg, [(N.PV, 0)], [(N.EV, 25)]], 1000)
    assert walk_plan(het, 8) == [5, 2, 3]
    big = fake([bldg] * 3, 60000)
    assert walk_plan(big) == [790, 790, 790] and 3 * 790 > 148 * 4
    assert sum(_blocks_of(j, 790, 938) == 2 for j in range(790)) == 148


# ------------------------------------------------------------------ staged host path in chunks
def _staged(env, soc, acts):
    env.set_option(N.OPT_HOST_ZERO_COPY, 0)
    env.set_option(N.OPT_HOST_CHUNKS, 4)
    out = [np.array(env.reset_host(soc))]
    for a in acts:
        out.append(tuple(np.array(x) for x in env.step_host(a)))
    return out


def _device(env, soc, acts):
    torch = _torch()
    out = [env.reset_batch(soc).cpu().numpy()]
    for a in acts:
        o, r, d, _ = env.step_batch(torch.from_numpy(a).cuda())
        out.append((o.cpu().numpy(), r.cpu().numpy(), d.cpu().numpy()))
    return out


@pytest.mark.parametrize("scenario", ["c1_tc2", "c2"])
@pytest.mark.parametrize("E", [1000, 600])
def test_staged_host_chunks_under_a_walk(monkeypatch, scenario, E):
    """OPT_HOST_CHUNKS = 4 on the staged path: chunks of whole 128-env tiles, so every chunk after the
    first starts at e_lo > 0.  1000 envs: 256 + 256 + 256 + 232 (a partial block); 600 envs:
    256 + 256 + 88 and an empty fourth chunk.  Under budget 1 and the default budget, in float64
    and float32, the results must equal the device path bit for bit."""
    make, _, _, _, options, *_ = CASES[scenario]
    T = 8
    rng = np.random.default_rng(E)
    for dt in ("float64", "float32"):
        kw = {"io_dtype": dt}
        dev, _ = _make(monkeypatch, make, E, None, options, **kw)
        soc = rng.uniform(10, 40, size=(dev.num_storage, E))
        acts = [rng.uniform(-1.2, 1.2, size=(dev.act_dim, E)).astype(dt) for _ in range(T)]
        want = _device(dev, soc, acts)
        dev.close()
        for budget in (1, None):
            env, n = _make(monkeypatch, make, E, budget, options, **kw)
            got = _staged(env, soc, acts)
            np.testing.assert_array_equal(got[0], want[0], err_msg=f"{dt} budget {budget} reset")
            for t in range(T):
                for k, what in enumerate(("obs", "rew", "done")):
                    np.testing.assert_array_equal(got[t + 1][k], want[t + 1][k],
                                                  err_msg=f"{dt} budget {budget} t={t} {what}")
            env.close()


# ------------------------------------------------------------------ float32 I/O on a walk
@pytest.mark.parametrize("name", F32_CASES)
def test_float32_io_under_budget_one(monkeypatch, kernels, name):
    from tests.test_gpu_io_f32 import _run_episode
    make, E, _, _, options, want, *_ = CASES[name]
    assert kernels[f"{name}/float32"] == {("component_kernel",) + want + (T_,)}, kernels[f"{name}/float32"]
    e64, n = _make(monkeypatch, make, E, 1, options)
    e32, _ = _make(monkeypatch, make, E, 1, options, io_dtype="float32")
    assert n == [1] * len(n)
    _run_episode(e64, e32, seed=5, steps=30)
    e64.close()
    e32.close()
