"""GPU tier: the CUDA path, called through the C ABI, against (a) golden traces recorded
from the unmodified reference, (b) the CPU oracle on seeded random batches, and (c) at
BASELINE.json's full sizes through size-independent properties.

Tolerances (BASELINE.json north_star): voltages 1e-4 p.u., component states 1e-6
relative, rewards 1e-5 relative, integer EV state bit-exact.  What is asserted is
tighter wherever float64 allows; see tests/test_host_tables_emu.py for why rewards that
multiply a voltage by 1e4 carry an absolute floor."""
import os

import numpy as np
import pytest

from tests import pf_reference as R
from tests import scenarios as S
from tests.flatten import flat_obs, unflatten_action
from tests.oracle_ns import ORACLE_NS as ONS, storage_socs_to_dict
from tests.product_ns import PRODUCT_NS as PNS

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
OBS_ATOL, REW_RTOL, REW_ATOL, V_ATOL = 1e-7, 1e-5, 2e-5, 1e-7

CASES = {
    "c0_buildings": lambda ns, **k: ns.CoordinatedMultiBuildingControlEnv(
        **S.buildings_scenario(ns, ns.OpenDSSSolver, 1.2), **k),
    "heterogeneous": lambda ns, **k: ns.MultiAgentEnv(
        **S.heterogeneous_scenario(ns, ns.OpenDSSSolver, 0.65), **k),
    "heterogeneous_max250": lambda ns, **k: ns.MultiAgentEnv(
        **S.heterogeneous_scenario(ns, ns.OpenDSSSolver, 0.6, max_episode_steps=250), **k),
    "test_heterogeneous": lambda ns, **k: ns.MultiAgentEnv(
        **S.test_heterogeneous_scenario(ns, ns.OpenDSSSolver), **k),
}


def _torch():
    import torch
    return torch


TIMEBASE = {"timebase_" + v: (lambda v: lambda ns, **k: ns.MultiAgentEnv(
    **S.time_base_scenario(ns, ns.OpenDSSSolver, v), **k))(v) for v in S.TIME_BASE_VARIANTS}


@pytest.mark.parametrize("name", list(TIMEBASE))
def test_other_time_bases_replay_reference_trace(name):
    """The heterogeneous scenario on other clocks (10-minute, 1-minute and 15-minute control
    intervals, day windows that do not start at midnight, max_episode_steps): batch of 5 replicas
    through the batched API, every column against the trace recorded from the reference."""
    torch = _torch()
    g = np.load(os.path.join(GOLD, name + ".npz"))
    E = 5
    env = TIMEBASE[name](PNS, num_envs=E)
    T = g["actions"].shape[0]
    assert env.episode_length == T
    obs0 = env.reset_batch(np.repeat(g["init_soc"].reshape(-1, 1), E, axis=1)).cpu().numpy()
    np.testing.assert_allclose(obs0, np.repeat(g["obs0"][:, None], E, 1), rtol=0, atol=OBS_ATOL)
    for t in range(T):
        a = torch.as_tensor(np.repeat(g["actions"][t][:, None], E, 1)).cuda()
        obs, rew, done, all_done = env.step_batch(a)
        np.testing.assert_allclose(obs.cpu().numpy(), np.repeat(g["obs"][t][:, None], E, 1),
                                   rtol=0, atol=OBS_ATOL, err_msg=f"t={t}")
        np.testing.assert_allclose(rew.cpu().numpy(), np.repeat(g["rew"][t][:, None], E, 1),
                                   rtol=REW_RTOL, atol=REW_ATOL)
        assert bool(done.cpu().numpy().all()) == bool(g["done"][t])
    assert all_done


@pytest.mark.parametrize("name", list(CASES))
def test_dict_api_replays_reference_trace(name):
    """num_envs == 1 through the reference's dict API."""
    g = np.load(os.path.join(GOLD, name + ".npz"))
    env = CASES[name](PNS)
    names = [str(n) for n in g["node_names"]]
    obs0 = env.reset(init_storage=g["init_soc"])
    np.testing.assert_allclose(flat_obs(env, obs0), g["obs0"], rtol=0, atol=OBS_ATOL)
    v = env.voltages
    np.testing.assert_allclose([v[k] for k in names], g["volt"][0], rtol=0, atol=V_ATOL)
    T = g["actions"].shape[0]
    for t in range(T):
        ob, rew, dn, _ = env.step(unflatten_action(env, g["actions"][t]))
        np.testing.assert_allclose(flat_obs(env, ob), g["obs"][t], rtol=0, atol=OBS_ATOL,
                                   err_msg=f"obs t={t}")
        np.testing.assert_allclose([rew[a.name] for a in env.agents], g["rew"][t],
                                   rtol=REW_RTOL, atol=REW_ATOL, err_msg=f"rew t={t}")
        np.testing.assert_allclose([a.real_power for a in env.agents], g["agent_p"][t],
                                   rtol=1e-12, atol=1e-12)
        assert dn["__all__"] == bool(g["done"][t])
        if t % 40 == 0 or t == T - 1:
            v = env.voltages
            np.testing.assert_allclose([v[k] for k in names], g["volt"][t + 1], rtol=0, atol=V_ATOL)
    with pytest.raises(RuntimeError):
        env.step(unflatten_action(env, g["actions"][0]))     # episode over: reset required


@pytest.mark.parametrize("name,E", [("c0_buildings", 33), ("heterogeneous", 130)])
def test_batch_replicas_replay_reference_trace(name, E):
    """Ragged batch sizes (not multiples of 16 / 32 / 128): every env gets the golden
    actions, so every column must reproduce the golden trace."""
    torch = _torch()
    g = np.load(os.path.join(GOLD, name + ".npz"))
    env = CASES[name](PNS, num_envs=E)
    soc = np.repeat(g["init_soc"].reshape(-1, 1), E, axis=1)
    obs0 = env.reset_batch(soc).cpu().numpy()
    np.testing.assert_allclose(obs0, np.repeat(g["obs0"][:, None], E, 1), rtol=0, atol=OBS_ATOL)
    T = g["actions"].shape[0]
    for t in range(T):
        a = torch.as_tensor(np.repeat(g["actions"][t][:, None], E, 1)).cuda()
        obs, rew, done, all_done = env.step_batch(a)
        if t % 15 == 0 or t == T - 1:
            np.testing.assert_allclose(obs.cpu().numpy(), np.repeat(g["obs"][t][:, None], E, 1),
                                       rtol=0, atol=OBS_ATOL, err_msg=f"t={t}")
            np.testing.assert_allclose(rew.cpu().numpy(), np.repeat(g["rew"][t][:, None], E, 1),
                                       rtol=REW_RTOL, atol=REW_ATOL)
            assert bool(done.cpu().numpy().all()) == bool(g["done"][t])
            assert bool(done.cpu().numpy().any()) == bool(g["done"][t])
    assert all_done


@pytest.mark.parametrize("name", ["c0_buildings", "heterogeneous", "test_heterogeneous"])
def test_random_batch_matches_oracle(name):
    """Different actions and initial SOC per env, checked env by env against the oracle."""
    torch = _torch()
    E, T = 6, 60
    env = CASES[name](PNS, num_envs=E)
    rng = np.random.default_rng(42)
    soc = rng.uniform(5, 45, size=(env.num_storage, E))
    acts = rng.uniform(-1.1, 1.1, size=(T, env.act_dim, E))
    if name == "test_heterogeneous":          # raw (unscaled) action spaces there
        acts = np.abs(acts)
    obs0 = env.reset_batch(soc).cpu().numpy().copy()
    O, R, V, SI = [], [], [], []
    for t in range(T):
        o, r, _, _ = env.step_batch(torch.as_tensor(acts[t]).cuda())
        O.append(o.cpu().numpy().copy())
        R.append(r.cpu().numpy().copy())
        V.append(env.get_field(3).cpu().numpy())
        SI.append(env.get_field(1).cpu().numpy())
    node_names = env.pf_solver.feeder.node_names
    for e in range(E):
        ref = CASES[name](ONS)
        o0 = ref.reset(init_storage=storage_socs_to_dict(ref, soc[:, e]))
        np.testing.assert_allclose(obs0[:, e], flat_obs(ref, o0), rtol=0, atol=OBS_ATOL)
        for t in range(T):
            o, r, _, _ = ref.step(unflatten_action(ref, acts[t][:, e]))
            np.testing.assert_allclose(O[t][:, e], flat_obs(ref, o), rtol=0, atol=OBS_ATOL,
                                       err_msg=f"env {e} t={t}")
            np.testing.assert_allclose(R[t][:, e], [r[a.name] for a in ref.agents],
                                       rtol=REW_RTOL, atol=REW_ATOL, err_msg=f"env {e} t={t}")
            np.testing.assert_allclose(V[t][:, e], [ref.voltages[n] for n in node_names],
                                       rtol=0, atol=V_ATOL)
            # integer EV state: the charging set, bit for bit
            for ag_o, ag_p in zip(ref.agents, env.agents):
                if hasattr(ag_o, "charging_vehicles"):
                    off, words = ag_p._slot["si"]
                    bits = 0
                    for w in range(words):
                        bits |= int(np.uint32(SI[t][off + w, e])) << (32 * w)
                    want = 0
                    for i in ag_o.charging_vehicles:
                        want |= 1 << int(i)
                    assert bits == want, f"EV charging set env {e} t={t}"


def test_component_only_env_matches_oracle():
    """BASELINE C2 composition (EV 100 vehicles + PV + storage, no feeder)."""
    torch = _torch()
    E, T = 5, 286
    env = PNS.MultiAgentEnv(**S.ev_pv_storage_scenario(PNS), num_envs=E)
    assert env.episode_length == 286
    rng = np.random.default_rng(3)
    soc = rng.uniform(5, 45, size=(env.num_storage, E))
    acts = rng.uniform(-1.0, 1.0, size=(T, env.act_dim, E))
    obs0 = env.reset_batch(soc).cpu().numpy().copy()
    O, R, SD = [], [], []
    for t in range(T):
        o, r, d, all_done = env.step_batch(torch.as_tensor(acts[t]).cuda())
        O.append(o.cpu().numpy().copy())
        R.append(r.cpu().numpy().copy())
    energy = env.get_field(0).cpu().numpy()
    assert all_done

    from oracle.multiagent import PowerFlowSolver

    class NoPF(PowerFlowSolver):
        def __init__(self, **kw):
            pass

        def calculate_power_flow(self, *a, **k):
            pass

        def get_bus_voltages(self):
            return {}

        def get_bus_voltage_by_name(self, n):
            return 1.0

    for e in range(E):
        ref = ONS.MultiAgentEnv(**S.ev_pv_storage_scenario(ONS, NoPF))
        o0 = ref.reset(init_storage=storage_socs_to_dict(ref, soc[:, e]))
        np.testing.assert_allclose(obs0[:, e], flat_obs(ref, o0), rtol=1e-12, atol=1e-12)
        for t in range(T):
            o, r, dn, _ = ref.step(unflatten_action(ref, acts[t][:, e]))
            np.testing.assert_allclose(O[t][:, e], flat_obs(ref, o), rtol=1e-10, atol=1e-10)
            np.testing.assert_allclose(R[t][:, e], [r[a.name] for a in ref.agents],
                                       rtol=1e-9, atol=1e-12)
        assert dn["__all__"]
        ev = ref.agents[0]
        off, n = env.agents[0]._slot["sd"]
        np.testing.assert_allclose(energy[off:off + n, e], ev.energy, rtol=1e-12, atol=1e-12)


def test_full_size_c1_properties():
    """4096 IEEE-13 envs (BASELINE C1): replicas given identical inputs stay bit-identical,
    SOC stays inside its range, voltages stay physical, every solve converges, and the
    on-device statistics agree with torch reductions."""
    torch = _torch()
    E, T = 4096, 25
    env = CASES["c0_buildings"](PNS, num_envs=E)
    rng = np.random.default_rng(0)
    half = E // 2
    soc_h = rng.uniform(5, 45, size=(env.num_storage, half))
    soc = np.concatenate([soc_h, soc_h], axis=1)
    env.reset_batch(soc)
    for t in range(T):
        a_h = rng.uniform(-1, 1, size=(env.act_dim, half))
        a = torch.as_tensor(np.concatenate([a_h, a_h], axis=1)).cuda()
        obs, rew, done, _ = env.step_batch(a)
    assert torch.equal(obs[:, :half], obs[:, half:])
    assert torch.equal(rew[:, :half], rew[:, half:])
    sd = env.get_field(0)
    for ag in env.agents:
        st = ag.env_dict["storage"]
        row = sd[st._slot["sd"][0]]
        assert float(row.min()) >= st.storage_range[0] and float(row.max()) <= st.storage_range[1]
    vmag = env.get_field(3)
    assert 0.85 < float(vmag.min()) and float(vmag.max()) < 1.06
    iters = env.get_field(7)
    assert int(iters.min()) > 0, "a power flow did not converge"
    s = env.stats().cpu().numpy()
    assert s[0] == E * T
    np.testing.assert_allclose(s[1], float(rew.sum()), rtol=1e-9)
    np.testing.assert_allclose(s[2], float(env.get_field(8).sum()), rtol=1e-9)
    assert s[4] == 0
    np.testing.assert_allclose(s[5], float(iters.sum()))
    np.testing.assert_allclose(s[6], float(env.get_field(4).min()))
    np.testing.assert_allclose(s[7], float(env.get_field(5).max()))


def test_host_buffer_path_equals_device_path():
    torch = _torch()
    E, T = 257, 10
    a_env = CASES["c0_buildings"](PNS, num_envs=E)
    b_env = CASES["c0_buildings"](PNS, num_envs=E)
    rng = np.random.default_rng(5)
    soc = rng.uniform(5, 45, size=(a_env.num_storage, E))
    o_a = a_env.reset_batch(soc).cpu().numpy()
    o_b = b_env.reset_host(soc)
    np.testing.assert_array_equal(o_a, o_b)
    for t in range(T):
        act = rng.uniform(-1, 1, size=(a_env.act_dim, E))
        oa, ra, da, _ = a_env.step_batch(torch.as_tensor(act).cuda())
        ob, rb, db = b_env.step_host(act)
        np.testing.assert_array_equal(oa.cpu().numpy(), ob)
        np.testing.assert_array_equal(ra.cpu().numpy(), rb)
        np.testing.assert_array_equal(da.cpu().numpy(), db)


def test_standalone_solver_like_reference_test_opendss():
    """tests/distribution_system/test_opendss.py:7-16 of the reference + a value check."""
    cfg = dict(S.IEEE13, system_load_rescale_factor=0.7)
    s = PNS.OpenDSSSolver(**cfg)
    s.calculate_power_flow(current_time="01-01-2021 05:00:00")
    v = s.get_bus_voltages()
    o = ONS.OpenDSSSolver(**cfg)
    o.calculate_power_flow(current_time="01-01-2021 05:00:00")
    vo = o.get_bus_voltages()
    assert set(v) == set(vo) and len(v) == 38
    np.testing.assert_allclose([v[k] for k in vo], list(vo.values()), rtol=0, atol=V_ATOL)
    s.calculate_power_flow(current_time="01-01-2021 05:00:00",
                           p_controllable_consumed={"675c": 800.0, "634a": -50.0},
                           q_controllable_consumed={"675c": 0.0, "634a": 10.0})
    o.calculate_power_flow(current_time="01-01-2021 05:00:00",
                           p_controllable_consumed={"675c": 800.0, "634a": -50.0},
                           q_controllable_consumed={"675c": 0.0, "634a": 10.0})
    vo = o.get_bus_voltages()
    v = s.get_bus_voltages()
    np.testing.assert_allclose([v[k] for k in vo], list(vo.values()), rtol=0, atol=V_ATOL)
    assert s.get_bus_voltage_by_name("675c") == v["675.3"]
    assert s.get_bus_voltage_by_name("671") == [v["671.1"], v["671.2"], v["671.3"]]


def test_original_ieee13_feeder_on_gpu_matches_published_profile():
    """All three load models, delta and wye, capacitors and regulator taps through the CUDA
    solver: published IEEE 13-node voltages within 2e-3 p.u. (see test_oracle_powerflow)."""
    import json
    s = PNS.OpenDSSSolver(os.path.join(GOLD, "ieee13_original.dss"),
                          "ieee_13_dss/annual_hourly_load_profile.csv", 1.0)
    s.annual_hourly_load_profile = np.ones(8760)          # nominal loads
    s.calculate_power_flow(current_time="01-01-2021 00:00:00")
    v = s.get_bus_voltages()
    pub = json.load(open(os.path.join(GOLD, "ieee13_published_voltages.json")))
    for bus, vals in pub.items():
        if bus.startswith("_"):
            continue
        for ph, want in enumerate(vals, 1):
            if want is not None:
                assert abs(v[f"{bus}.{ph}"] - want) < 2e-3, (bus, ph)


def test_abi_error_paths():
    env = CASES["c0_buildings"](PNS, num_envs=4)
    torch = _torch()
    with pytest.raises(RuntimeError):
        env.step_batch(torch.zeros((env.act_dim, 4), dtype=torch.float64, device="cuda"))
    env.reset_batch()
    with pytest.raises(ValueError):
        env.step_batch(torch.zeros((env.act_dim, 5), dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        env.step_batch(torch.zeros((env.act_dim, 4), dtype=torch.float32, device="cuda"))
    from powergridworld_b200 import _native as N
    out = torch.empty(3, dtype=torch.float64, device="cuda")
    import ctypes as C
    rc = env._lib.pgw_get(env._h, N.FIELD_VMIN, C.c_void_p(out.data_ptr()), 24, None)
    assert rc == -1 and b"size mismatch" in env._lib.pgw_last_error()


@pytest.mark.parametrize("kernel", [1, 2])
@pytest.mark.parametrize("name,E", [("c0_buildings", 300), ("heterogeneous", 128)])
def test_tensor_core_power_flow_matches_fp64_kernel(name, E, kernel):
    """tcgen05 fixed point (split-TF32 operands, FP32 accumulate/epilogue) vs the FP64 SIMT
    kernel on the same batch: node voltages within 1e-6 p.u. -- two orders inside the 1e-4 p.u.
    tolerance of the reference's own solver -- and rewards within 1e-5 relative (+ the
    1e4 x voltage floor of the violation penalty)."""
    torch = _torch()
    from powergridworld_b200 import _native as N
    T = 40
    a_env = CASES[name](PNS, num_envs=E)
    b_env = CASES[name](PNS, num_envs=E)
    b_env.set_option(N.OPT_PF_KERNEL, kernel)
    rng = np.random.default_rng(11)
    soc = rng.uniform(5, 45, size=(a_env.num_storage, E))
    oa = a_env.reset_batch(soc).cpu().numpy()
    ob = b_env.reset_batch(soc).cpu().numpy()
    np.testing.assert_allclose(ob, oa, rtol=0, atol=2e-5)
    np.testing.assert_allclose(b_env.get_field(3).cpu().numpy(), a_env.get_field(3).cpu().numpy(),
                               rtol=0, atol=1e-6)
    for t in range(T):
        act = torch.as_tensor(rng.uniform(-1, 1, size=(a_env.act_dim, E))).cuda()
        oa, ra, _, _ = a_env.step_batch(act)
        ob, rb, _, _ = b_env.step_batch(act)
        np.testing.assert_allclose(b_env.get_field(3).cpu().numpy(),
                                   a_env.get_field(3).cpu().numpy(), rtol=0, atol=1e-6,
                                   err_msg=f"voltages t={t}")
        np.testing.assert_allclose(ob.cpu().numpy(), oa.cpu().numpy(), rtol=0, atol=2e-5)
        # kernel 2 = what bench.py runs: its float64 polish holds the rewards to the float64
        # solver's bound; kernel 1 (split-TF32, no polish) keeps the 1e4 x voltage floor
        np.testing.assert_allclose(rb.cpu().numpy(), ra.cpu().numpy(), rtol=1e-5,
                                   atol=2e-5 if kernel == 2 else 1e-2, err_msg=f"rewards t={t}")
    it = b_env.get_field(7)
    assert int(it.min()) > 0, "tensor-core solve did not converge"
    assert float(it.double().mean()) < 25


@pytest.mark.parametrize("kernel", [1, 2])
def test_tensor_core_golden_trace_within_north_star_tolerances(kernel):
    """Reference golden trace through the tcgen05 solvers: voltages 1e-4 p.u., observations
    1e-6 (x10 for the scaled voltage entries), rewards 1e-5 relative."""
    from powergridworld_b200 import _native as N
    g = np.load(os.path.join(GOLD, "c0_buildings.npz"))
    env = CASES["c0_buildings"](PNS)
    env.set_option(N.OPT_PF_KERNEL, kernel)
    names = [str(n) for n in g["node_names"]]
    obs0 = env.reset(init_storage=g["init_soc"])
    np.testing.assert_allclose(flat_obs(env, obs0), g["obs0"], rtol=0, atol=1e-5)
    for t in range(g["actions"].shape[0]):
        ob, rew, dn, _ = env.step(unflatten_action(env, g["actions"][t]))
        np.testing.assert_allclose(flat_obs(env, ob), g["obs"][t], rtol=0, atol=1e-5)
        np.testing.assert_allclose([rew[a.name] for a in env.agents], g["rew"][t],
                                   rtol=1e-5, atol=2e-5 if kernel == 2 else 1e-2)
        if t % 50 == 0:
            v = env.voltages
            np.testing.assert_allclose([v[k] for k in names], g["volt"][t + 1], rtol=0, atol=1e-4)
            np.testing.assert_allclose([v[k] for k in names], g["volt"][t + 1], rtol=0, atol=2e-6)


def test_der123_scenario_matches_oracle():
    """BASELINE C3 composition on the authored 123-bus-class feeder (251 nodes, 85 load
    branches -> the 3-rows-per-lane FP64 kernel, feeder tables read through L1/L2; load models
    1, 2 and 5; 100 heterogeneous agents)."""
    import warnings
    torch = _torch()
    E, T = 3, 12
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        env = PNS.MultiAgentEnv(**S.der123_scenario(PNS, PNS.OpenDSSSolver), num_envs=E)
    rng = np.random.default_rng(5)
    soc = rng.uniform(10, 50, size=(env.num_storage, E))
    acts = rng.uniform(-1, 1, size=(T, env.act_dim, E))
    obs0 = env.reset_batch(soc).cpu().numpy().copy()
    O, R, V = [], [], []
    for t in range(T):
        o, r, _, _ = env.step_batch(torch.as_tensor(acts[t]).cuda())
        O.append(o.cpu().numpy().copy())
        R.append(r.cpu().numpy().copy())
        V.append(env.get_field(3).cpu().numpy())
    assert int(env.get_field(7).min()) > 0
    names = env.pf_solver.feeder.node_names
    for e in range(E):
        ref = ONS.MultiAgentEnv(**S.der123_scenario(ONS, ONS.OpenDSSSolver))
        o0 = ref.reset(init_storage=storage_socs_to_dict(ref, soc[:, e]))
        np.testing.assert_allclose(obs0[:, e], flat_obs(ref, o0), rtol=0, atol=1e-9)
        for t in range(T):
            o, r, _, _ = ref.step(unflatten_action(ref, acts[t][:, e]))
            np.testing.assert_allclose(O[t][:, e], flat_obs(ref, o), rtol=0, atol=1e-9)
            np.testing.assert_allclose(R[t][:, e], [r[a.name] for a in ref.agents], rtol=1e-9, atol=1e-10)
            np.testing.assert_allclose(V[t][:, e], [ref.voltages[n] for n in names], rtol=0, atol=1e-8)


def test_der123_fp16_tensor_core_power_flow_matches_fp64_kernel():
    """C3 composition (85 load branches, 251 nodes, load models 1/2/5, 100 agents) through the
    split-FP16 tcgen05 solver with the Z-bus resident in shared memory vs the FP64 SIMT kernel on
    the same batch: 300 envs = two full tiles of 128 + a ragged one.  Voltages within 1e-6 p.u.
    (two orders inside the reference solver's 1e-4), rewards 1e-5 relative."""
    import warnings
    torch = _torch()
    from powergridworld_b200 import _native as N
    E, T = 300, 16
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        a_env = PNS.MultiAgentEnv(**S.der123_scenario(PNS, PNS.OpenDSSSolver), num_envs=E)
        b_env = PNS.MultiAgentEnv(**S.der123_scenario(PNS, PNS.OpenDSSSolver), num_envs=E)
    b_env.set_option(N.OPT_PF_KERNEL, 2)
    rng = np.random.default_rng(23)
    soc = rng.uniform(10, 50, size=(a_env.num_storage, E))
    oa = a_env.reset_batch(soc).cpu().numpy()
    ob = b_env.reset_batch(soc).cpu().numpy()
    va, vb = a_env.get_field(3).cpu().numpy(), b_env.get_field(3).cpu().numpy()
    np.testing.assert_allclose(vb, va, rtol=0, atol=1e-6, err_msg="reset voltages")
    np.testing.assert_allclose(ob, oa, rtol=0, atol=2e-5)
    for t in range(T):
        act = torch.as_tensor(rng.uniform(-1, 1, size=(a_env.act_dim, E))).cuda()
        oa, ra, _, _ = a_env.step_batch(act)
        ob, rb, _, _ = b_env.step_batch(act)
        va, vb = a_env.get_field(3).cpu().numpy(), b_env.get_field(3).cpu().numpy()
        np.testing.assert_allclose(vb, va, rtol=0, atol=1e-6, err_msg=f"voltages t={t}")
        np.testing.assert_allclose(b_env.get_field(4).cpu().numpy(), va.min(axis=0), rtol=0, atol=1e-6)
        np.testing.assert_allclose(b_env.get_field(5).cpu().numpy(), va.max(axis=0), rtol=0, atol=1e-6)
        np.testing.assert_allclose(b_env.get_field(6).cpu().numpy(), a_env.get_field(6).cpu().numpy(),
                                   rtol=0, atol=1e-6)
        np.testing.assert_allclose(ob.cpu().numpy(), oa.cpu().numpy(), rtol=0, atol=2e-5)
        np.testing.assert_allclose(rb.cpu().numpy(), ra.cpu().numpy(), rtol=1e-5, atol=1e-4)
    # warm-start state agrees as well (branch voltages, complex)
    ua, ub = a_env.get_field(9).cpu().numpy(), b_env.get_field(9).cpu().numpy()
    nb = a_env.pf_solver.feeder.nb
    np.testing.assert_allclose(ub.reshape(-1, E, 2)[:nb], ua.reshape(-1, E, 2)[:nb], rtol=0, atol=2e-6)
    it = b_env.get_field(7)
    assert int(it.min()) > 0, "tensor-core solve did not converge"
    assert float(it.double().mean()) < 25


# ------------------------------------------------------------------ Home-Steward house (SURVEY 8f-2)
def _hs_batch(name, num_envs):
    from powergridworld_b200.base_hs import house_agent_config
    from tests import scenarios_hs as SH
    from tests.product_hs_ns import PRODUCT_HS_NS as HNS
    cfg = SH.VARIANTS[name](HNS)
    return PNS.MultiAgentEnv(
        common_config={"start_time": cfg["start_time"], "end_time": "01-01-2031 00:00:00",
                       "control_timedelta": cfg["control_timedelta"]},
        pf_config=None, num_envs=num_envs,
        agents=[{"name": "house", "bus": None, "cls": HNS.HSMultiComponentEnv,
                 "config": house_agent_config(cfg)}])


@pytest.mark.parametrize("name", ["shipped", "two_vehicles", "raw_spaces"])
def test_hs_house_golden_trace_on_gpu(name):
    """The reference's HSMultiComponentEnv trace (recorded from the unmodified reference) through
    the CUDA path, one house per env, every env fed the golden actions: observations 1e-12,
    rewards 1e-12 relative, done flags and the house's real power."""
    torch = _torch()
    g = np.load(os.path.join(GOLD, f"hs_{name}.npz"))
    E = 5
    env = _hs_batch(name, E)
    assert env.episode_length == 288
    obs0 = env.reset_batch(np.repeat(g["init_soc"].reshape(1, 1), E, axis=1)).cpu().numpy()
    for e in range(E):
        np.testing.assert_allclose(obs0[:, e], g["obs0"], rtol=0, atol=1e-13)
    for t in range(g["actions"].shape[0]):
        act = torch.as_tensor(np.repeat(g["actions"][t].reshape(4, 1), E, axis=1)).cuda()
        o, r, d, alld = env.step_batch(act)
        o, r = o.cpu().numpy(), r.cpu().numpy()
        for e in (0, E - 1):
            np.testing.assert_allclose(o[:, e], g["obs"][t], rtol=0, atol=1e-12, err_msg=f"t={t}")
            np.testing.assert_allclose(r[0, e], g["rew"][t], rtol=1e-12, atol=1e-13, err_msg=f"t={t}")
        assert bool(d[0]) == bool(g["done"][t])
        np.testing.assert_allclose(env.get_field(2).cpu().numpy()[0], g["real_power"][t],
                                   rtol=1e-14, atol=0)


@pytest.mark.parametrize("case", [0, 3, 5])
def test_hs_random_houses_two_episodes_on_gpu(case):
    """tests/golden/hs_random_configs.npz (six random houses x two consecutive episodes recorded
    from the unmodified reference): the house through the reference's own per-object API
    (house.reset() draws the SOC from the same RNG stream; house.step(dict))."""
    import json
    from tests import scenarios_hs as SH
    from tests.product_hs_ns import PRODUCT_HS_NS as HNS
    g = np.load(os.path.join(GOLD, "hs_random_configs.npz"))
    m = json.loads(str(g["meta"]))[case]
    house = HNS.HSMultiComponentEnv(**SH.parametrised(HNS, m["hp"]))
    names = [e.name for e in house.envs]
    flat = lambda obs: np.concatenate([np.asarray(obs[n], dtype=np.float64).ravel() for n in names])
    for ep in range(2):
        key = f"{case}_{ep}"
        np.random.seed(m["seed"] + ep)
        obs0 = house.reset()
        np.testing.assert_allclose(flat(obs0), g["obs0_" + key], rtol=0, atol=1e-13, err_msg=key)
        A = g["act_" + key]
        for t in range(A.shape[0]):
            ob, rew, done, _ = house.step({n: A[t][k:k + 1] for k, n in enumerate(names)})
            np.testing.assert_allclose(flat(ob), g["obs_" + key][t], rtol=0, atol=1e-12, err_msg=f"{key} t={t}")
            np.testing.assert_allclose(rew, g["rew_" + key][t], rtol=1e-12, atol=1e-13, err_msg=f"{key} t={t}")
        assert done


def test_hs_house_batch_matches_oracle_per_env():
    """Different actions and initial storage per env against the HS oracle, two episodes back to
    back (the storage cost and the meta state survive the reset, as in the reference)."""
    torch = _torch()
    from tests import scenarios_hs as SH
    from tests.oracle_hs_ns import ORACLE_HS_NS as OHS
    E, T = 6, 60
    env = _hs_batch("two_vehicles", E)
    rng = np.random.default_rng(17)
    refs = [OHS.HSMultiComponentEnv(**SH.two_vehicles(OHS)) for _ in range(E)]
    flat = lambda h, ob: np.concatenate([np.asarray(ob[c.name], dtype=np.float64).ravel() for c in h.envs])
    for episode in range(2):
        soc = rng.uniform(3, 19, size=(1, E))
        obs0 = env.reset_batch(soc).cpu().numpy()
        for e in range(E):
            np.testing.assert_allclose(obs0[:, e], flat(refs[e], refs[e].reset(init_storage=soc[0, e])),
                                       rtol=0, atol=1e-12)
        for t in range(T):
            acts = rng.uniform(-1.2, 1.2, size=(4, E))
            o, r, _, _ = env.step_batch(torch.as_tensor(acts).cuda())
            o, r = o.cpu().numpy(), r.cpu().numpy()
            for e in range(E):
                ob, rw, _, _ = refs[e].step({c.name: acts[k:k + 1, e] for k, c in enumerate(refs[e].envs)})
                np.testing.assert_allclose(o[:, e], flat(refs[e], ob), rtol=0, atol=1e-12)
                np.testing.assert_allclose(r[0, e], rw, rtol=1e-12, atol=1e-13)


def test_hs_house_object_protocol():
    """HSMultiComponentEnv(**make_env_config()) stepped on its own like the reference object:
    reset() -> obs dict, step(action dict) -> (obs, reward, done, meta_state)."""
    from powergridworld_b200.base_hs import HSMultiComponentEnv
    from powergridworld_b200.scenarios.heterogeneous_hs import make_env_config
    g = np.load(os.path.join(GOLD, "hs_shipped.npz"))
    house = HSMultiComponentEnv(**make_env_config())
    obs = house.reset(init_storage=float(g["init_soc"][0]))
    assert set(obs) == {"pv", "storage", "ev-charging", "other-devices"}
    names = [e.name for e in house.envs]
    for t in range(5):
        a = g["actions"][t]
        obs, rew, done, meta = house.step({n: a[k:k + 1] for k, n in enumerate(names)})
        got = np.concatenate([np.asarray(obs[n]).ravel() for n in names])
        np.testing.assert_allclose(got, g["obs"][t], rtol=0, atol=1e-12)
        np.testing.assert_allclose(rew, g["rew"][t], rtol=1e-12, atol=1e-13)
        assert not done
        # golden meta order: grid_cost, es_cost, grid_power, pv_power, es_power, pv_cost
        np.testing.assert_allclose(
            [meta[k] for k in ("grid_cost", "es_cost", "grid_power", "pv_power", "es_power", "pv_cost")],
            g["meta"][t], rtol=1e-14, atol=0)
        # the per-device telemetry records of base_hs.py:158-164
        assert [r["device_id"] for r in meta["step_meta"]] == names
        for k, rec in enumerate(meta["step_meta"]):
            vals = [rec["cost"], rec["reward"], rec["action"][0], rec["solar_power_consumed"],
                    rec["es_power_consumed"], rec["grid_power_consumed"]]
            vals += [float(v) for v in rec["device_custom_info"].values()]
            want = g["telemetry"][t, k]
            np.testing.assert_allclose(vals, want[:len(vals)], rtol=1e-12, atol=1e-13)
            assert np.isnan(want[len(vals):]).all()


# ------------------------------------------------------------------ tc2 tile widths / stand-alone solve
# about twice the worst error measured on a B200 (1000 W): 1.39e-7 / 1.43e-7 / 1.28e-7 p.u.
STANDALONE_TOL = {24: 2.8e-7, 50: 2.9e-7, 85: 2.6e-7}


@pytest.mark.parametrize("n_loads", [24, 50, 85])
def test_tc2_every_tile_width_standalone_and_in_env(tmp_path, n_loads):
    """24 / 50 / 85 load branches -> the NCH = 4 / 8 / 11 instantiations of pf_tc2_kernel, through
    the stand-alone solve (pgw_pf_solve, its own instantiation) and inside a stepping env, against
    the FP64 kernel: voltages within 1e-6 p.u.; the stand-alone solve also against the float64
    reference."""
    torch = _torch()
    from powergridworld_b200 import _native as N
    path = R.synthetic_feeder(tmp_path, n_loads)
    shape = "ieee_13_dss/annual_hourly_load_profile.csv"
    a, b = PNS.OpenDSSSolver(path, shape, 0.9), PNS.OpenDSSSolver(path, shape, 0.9)
    assert a.feeder.nb == n_loads
    for s_, k in ((a, 0), (b, 2)):
        s_.calculate_power_flow(current_time="08-12-2021 12:00:00")
        s_._host_env.set_option(N.OPT_PF_KERNEL, k)
    names = a.feeder.load_names
    ctrl = {names[0]: 150.0, names[3]: -80.0, names[n_loads - 1]: 40.0}
    for s_ in (a, b):
        s_.calculate_power_flow(current_time="08-12-2021 12:00:00", p_controllable_consumed=ctrl,
                                q_controllable_consumed={names[0]: 20.0})
    va, vb = a.get_bus_voltages(), b.get_bus_voltages()
    np.testing.assert_allclose([vb[k] for k in va], list(va.values()), rtol=0, atol=1e-6)
    assert min(va.values()) < 0.999                      # the loads did move the profile
    # the stand-alone tc2 build (pf_tc2_kernel<NCH, *, true>) against the float64 reference of
    # the solve's load table (ctrl reaches the model-1 loads only)
    f = b.feeder
    kw, kvar = b.base_load_at("08-12-2021 12:00:00")
    for n in b.load_bus_name:
        kw[f.load_index(n)] += ctrl.get(n, 0.0)
        kvar[f.load_index(n)] += {names[0]: 20.0}.get(n, 0.0)
    _, _, v64 = R.solve64(f, (kw + 1j * kvar)[f.branch_load] * f.branch_share * 1e-3)
    err = np.abs([vb[n] for n in f.node_names] - v64[:, 0]).max()
    print(f"stand-alone tc2, {n_loads} loads: max error {err:.2e} against the float64 reference")
    assert err < STANDALONE_TOL[n_loads]

    import pandas as pd
    def env(kernel):
        agents = [{"name": f"s{i}", "bus": names[(7 * i) % n_loads], "cls": PNS.EnergyStorageEnv,
                   "config": {"max_power": 40. + 10 * i, "storage_range": (3., 80.)}}
                  for i in range(6)]
        e = PNS.MultiAgentEnv(
            common_config={"start_time": "08-12-2021 00:00:00", "end_time": "08-13-2021 00:00:00",
                           "control_timedelta": pd.Timedelta(300, "s")},
            pf_config={"cls": PNS.OpenDSSSolver, "config": {
                "feeder_file": path, "loadshape_file": shape, "system_load_rescale_factor": 0.9}},
            agents=agents, num_envs=200)
        e.set_option(N.OPT_PF_KERNEL, kernel)
        return e
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ea, eb = env(0), env(2)
    rng = np.random.default_rng(n_loads)
    soc = rng.uniform(10, 70, size=(6, 200))
    ea.reset_batch(soc); eb.reset_batch(soc)
    for t in range(6):
        act = torch.as_tensor(rng.uniform(-1, 1, size=(ea.act_dim, 200))).cuda()
        ea.step_batch(act); eb.step_batch(act)
        np.testing.assert_allclose(eb.get_field(3).cpu().numpy(), ea.get_field(3).cpu().numpy(),
                                   rtol=0, atol=1e-6, err_msg=f"t={t}")
    assert int(eb.get_field(7).min()) > 0


def test_tc2_is_bitwise_deterministic():
    """The wave-pipelined tensor-core solve has no data race: two handles fed the same inputs
    (one replaying CUDA graphs, one with plain launches) produce bit-identical voltages,
    observations, rewards and iteration counts on the 123-bus-class feeder."""
    import warnings
    torch = _torch()
    from powergridworld_b200 import _native as N
    E, T = 300, 10
    envs = []
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for graphs in (1, 0):
            e = PNS.MultiAgentEnv(**S.der123_scenario(PNS, PNS.OpenDSSSolver), num_envs=E)
            e.set_option(N.OPT_PF_KERNEL, 2)
            e.set_option(N.OPT_GRAPHS, graphs)
            envs.append(e)
    rng = np.random.default_rng(3)
    soc = rng.uniform(10, 50, size=(envs[0].num_storage, E))
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        o = [e.reset_batch(soc).clone() for e in envs]
        assert torch.equal(o[0], o[1])
        for t in range(T):
            act = torch.as_tensor(rng.uniform(-1, 1, size=(envs[0].act_dim, E))).cuda()
            res = [e.step_batch(act) for e in envs]
            assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1]), t
            for f in (3, 4, 5, 6, 7, 9):
                assert torch.equal(envs[0].get_field(f), envs[1].get_field(f)), (t, f)
    stream.synchronize()


@pytest.mark.parametrize("kernel", [0, 1, 2])
def test_power_flow_non_convergence_is_data(kernel):
    """SURVEY 8b: non-convergence is data, not an error.  With the iteration budget cut to 2 every
    solver reports -2 iterations per env and pgw_stats counts the envs; with the default budget
    the same batch converges (positive counts)."""
    torch = _torch()
    from powergridworld_b200 import _native as N
    E = 200
    rng = np.random.default_rng(2)
    for budget, ok in ((2, False), (None, True)):
        env = PNS.CoordinatedMultiBuildingControlEnv(
            **S.buildings_scenario(PNS, PNS.OpenDSSSolver, 1.2), num_envs=E, pf_max_iter=budget)
        env.set_option(N.OPT_PF_KERNEL, kernel)
        env.reset_batch(rng.uniform(10, 40, size=(env.num_storage, E)))
        env.step_batch(torch.as_tensor(rng.uniform(-1, 1, size=(env.act_dim, E))).cuda())
        it = env.get_field(7).cpu().numpy()
        st = env.stats().cpu().numpy()
        if ok:
            assert (it > 0).all() and st[4] == 0
        else:
            assert (it == -2).all() and st[4] == E
        v = env.get_field(3).cpu().numpy()
        assert np.isfinite(v).all() and v.min() > 0.8 and v.max() < 1.1


@pytest.mark.parametrize("kernel,E", [(0, 260), (2, 260), (2, 13000)])
def test_runtime_options_do_not_change_results(kernel, E):
    """PGW_OPT_WARM_START = 0 (every solve from the no-load voltages) gives the same voltages as
    the default within the solver's own tolerance and needs more iterations; PGW_OPT_PDL = 0
    (no programmatic dependent launch of the power flow; default on: released after the clock
    read at 260 envs, at the end of the component CTAs at 13 000) changes nothing at all."""
    torch = _torch()
    from powergridworld_b200 import _native as N
    T = 5
    rng = np.random.default_rng(8)
    soc = rng.uniform(10, 40, size=(3, E))
    acts = [torch.as_tensor(rng.uniform(-1, 1, size=(24, E))).cuda() for _ in range(T)]
    out = {}
    for label, opts in (("default", {}), ("cold", {N.OPT_WARM_START: 0}), ("pdl", {N.OPT_PDL: 0})):
        env = PNS.CoordinatedMultiBuildingControlEnv(
            **S.buildings_scenario(PNS, PNS.OpenDSSSolver, 1.2), num_envs=E)
        env.set_option(N.OPT_PF_KERNEL, kernel)
        for k, v in opts.items():
            env.set_option(k, v)
        stream = torch.cuda.Stream()
        with torch.cuda.stream(stream):
            env.reset_batch(soc)
            for a in acts:
                env.step_batch(a)
            out[label] = (env.get_field(3).cpu().numpy(), env.get_field(7).cpu().numpy(),
                          env.rew.cpu().numpy().copy())
        stream.synchronize()
    tol = 2e-9 if kernel == 0 else 3e-7
    for label in ("cold", "pdl"):
        np.testing.assert_allclose(out[label][0], out["default"][0], rtol=0, atol=tol, err_msg=label)
        np.testing.assert_allclose(out[label][2], out["default"][2], rtol=1e-6, atol=1e4 * tol)
    for k in range(3):                               # same arithmetic, another launch order
        np.testing.assert_array_equal(out["pdl"][k], out["default"][k])
    assert out["cold"][1].mean() > out["default"][1].mean()


def test_full_size_c3_shard_invariance_with_tc2():
    """BASELINE C3 at its full size (16 384 envs, 100 agents, tc2 solver): an env's trajectory does
    not depend on the batch it sits in -- the first 384 envs of the big batch agree with a 384-env
    batch fed the same inputs, bit for bit: the shard is three whole tiles of the big batch, and a
    tile's arithmetic depends only on its own envs; every solve converges."""
    import warnings
    torch = _torch()
    from powergridworld_b200 import _native as N
    E, S_, T = 16384, 384, 6
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        big = PNS.MultiAgentEnv(**S.der123_scenario(PNS, PNS.OpenDSSSolver), num_envs=E, pf_kernel="tc2")
        small = PNS.MultiAgentEnv(**S.der123_scenario(PNS, PNS.OpenDSSSolver), num_envs=S_, pf_kernel="tc2")
    gen = torch.Generator(device="cuda")
    gen.manual_seed(4)
    soc = 10 + 40 * torch.rand((big.num_storage, E), generator=gen, device="cuda", dtype=torch.float64)
    ob, os_ = big.reset_batch(soc), small.reset_batch(soc[:, :S_].contiguous())
    assert torch.equal(ob[:, :S_], os_)
    for t in range(T):
        act = 2 * torch.rand((big.act_dim, E), generator=gen, device="cuda", dtype=torch.float64) - 1
        ob, rb, _, _ = big.step_batch(act)
        os_, rs, _, _ = small.step_batch(act[:, :S_].contiguous())
        for f in (0, 3, 4, 5, 6, 7, 8, 9):           # state, voltages, min / max, bus, iterations, u
            whole = big.get_field(f)
            assert torch.equal(whole[:S_] if whole.dim() == 1 else whole[:, :S_], small.get_field(f)), (t, f)
        assert torch.equal(ob[:, :S_], os_) and torch.equal(rb[:, :S_], rs), t
    it = big.get_field(7)
    assert int(it.min()) > 0 and int(it.max()) < 20
    st = big.stats().cpu().numpy()
    assert st[0] == E * T and st[4] == 0


def test_full_size_c2_and_house_replicas_and_integer_state():
    """BASELINE C2 (65 536 envs, EV station of 100 vehicles + PV + storage) and 65 536 Home-Steward
    houses: replicas fed identical inputs stay bit-identical; the charging-set bitmask agrees with
    the num_active_vehicles observation; energies never go negative."""
    torch = _torch()
    E, T = 65536, 12
    half = E // 2
    gen = torch.Generator(device="cuda")
    gen.manual_seed(9)
    env = PNS.MultiAgentEnv(**S.ev_pv_storage_scenario(PNS), num_envs=E)
    soc_h = 10 + 30 * torch.rand((env.num_storage, half), generator=gen, device="cuda", dtype=torch.float64)
    env.reset_batch(torch.cat([soc_h, soc_h], dim=1))
    for t in range(T):
        a_h = 2 * torch.rand((env.act_dim, half), generator=gen, device="cuda", dtype=torch.float64) - 1
        obs, rew, _, _ = env.step_batch(torch.cat([a_h, a_h], dim=1))
    assert torch.equal(obs[:, :half], obs[:, half:]) and torch.equal(rew[:, :half], rew[:, half:])
    ev = [a for a in env.agents if hasattr(a, "num_vehicles")][0]
    o_off, _ = ev._slot["obs"]
    s_off, n = ev._slot["sd"]
    m_off, words = ev._slot["si"]
    energy = env.get_field(0)[s_off:s_off + n]
    assert float(energy.min()) >= 0.0
    mask = env.get_field(1)[m_off:m_off + words].to(torch.int64) & 0xFFFFFFFF
    pop = sum(((mask >> b) & 1) for b in range(32)).sum(dim=0)
    raw_active = (obs[o_off + 1] + 1) / 2 * ev._observation_space.high[1] if ev.rescale_spaces else obs[o_off + 1]
    torch.testing.assert_close(raw_active, pop.double() * ev.vehicle_multiplier, rtol=0, atol=1e-9)

    house = _hs_batch("two_vehicles", E)
    soc_h = 3 + 16 * torch.rand((1, half), generator=gen, device="cuda", dtype=torch.float64)
    house.reset_batch(torch.cat([soc_h, soc_h], dim=1))
    for t in range(T):
        a_h = 2.4 * torch.rand((4, half), generator=gen, device="cuda", dtype=torch.float64) - 1.2
        obs, rew, _, _ = house.step_batch(torch.cat([a_h, a_h], dim=1))
    assert torch.equal(obs[:, :half], obs[:, half:]) and torch.equal(rew[:, :half], rew[:, half:])
    assert bool(torch.isfinite(rew).all())


def test_randomized_rosters_replay_reference_trace_on_gpu():
    """EVChargingEnv(randomize=True) (ev_charging_env.py:154-157), dict API, two episodes: every
    reset draws new rosters on the host (same RNG stream as the reference), pushes them with
    pgw_update_tables and the cached step graphs keep running on the new tables."""
    from tests.test_oracle_golden import _replay_randomized

    def step(env, a):
        ob, rew, dn, _ = env.step(unflatten_action(env, a))
        return flat_obs(env, ob), np.array([rew[x.name] for x in env.agents]), dn["__all__"]

    _replay_randomized(
        lambda: PNS.MultiAgentEnv(**S.randomized_ev_scenario(PNS, PNS.OpenDSSSolver)),
        lambda env: flat_obs(env, env.reset()), step, exact=False)


def test_randomized_station_standalone_and_batched_vs_oracle():
    """Per-object protocol and a ragged batch: every env of the batch draws its OWN roster at
    reset (one np.random.choice per env instance, env 0 first -- ev_charging_env.py:154-157 is per
    instance), every env replays the oracle station that drew the same roster; the host-buffer
    entry points go through the same draws."""
    torch = _torch()
    cfg = dict(num_vehicles=37, minutes_per_step=5, max_charge_rate_kw=7., peak_threshold=40.,
               vehicle_multiplier=2., rescale_spaces=True, randomize=True)
    rng = np.random.default_rng(5)
    # (a) station on its own, three resets
    dev, ora = PNS.EVChargingEnv(**cfg), ONS.EVChargingEnv(**cfg)
    for ep in range(3):
        np.random.seed(9 + ep)
        od, _ = dev.reset()
        np.random.seed(9 + ep)
        oo, _ = ora.reset()
        np.testing.assert_allclose(od, oo, rtol=0, atol=1e-12)
        for t in range(120):
            a = rng.uniform(-1.1, 1.1, size=1)
            rd, ro = dev.step(a), ora.step(a)
            np.testing.assert_allclose(rd[0], ro[0], rtol=0, atol=1e-9, err_msg=f"ep={ep} t={t}")
            np.testing.assert_allclose(rd[1], ro[1], rtol=1e-9, atol=1e-12)
    # (b) batch of 70 envs, device and host entry points
    E = 70
    common = {"start_time": "08-12-2020 00:00:00", "end_time": "08-13-2020 00:00:00",
              "control_timedelta": __import__("pandas").Timedelta(300, "s")}
    env = PNS.MultiAgentEnv(common_config=common, pf_config=None, num_envs=E, agents=[
        {"name": "ev", "bus": None, "cls": PNS.EVChargingEnv, "config": cfg}])
    for ep, host in enumerate([False, True, False]):
        np.random.seed(30 + ep)
        obs0 = env.reset_host() if host else env.reset_batch().cpu().numpy()
        refs = [ONS.EVChargingEnv(**cfg) for _ in range(3)]
        n_all = len(dev._roster_energy)
        for r, e in zip(refs, [0, 33, 69]):          # env e's draw is the (e + 1)-th of the stream
            np.random.seed(30 + ep)
            for _ in range(e):
                np.random.choice(n_all, size=cfg["num_vehicles"], replace=False)
            o, _ = r.reset()
            np.testing.assert_allclose(obs0[:, e], o, rtol=0, atol=1e-12)
        station = env.agents[0]
        assert station._rows.shape == (E, cfg["num_vehicles"]) and len({tuple(x) for x in station._rows}) == E
        acts = rng.uniform(-1.1, 1.1, size=(100, 1, E))
        for t in range(100):
            if host:
                obs, rew, _ = env.step_host(acts[t])
            else:
                o_, r_, _, _ = env.step_batch(torch.as_tensor(acts[t]).cuda())
                obs, rew = o_.cpu().numpy(), r_.cpu().numpy()
            for k, e in enumerate([0, 33, 69]):
                ro = refs[k].step(acts[t][:, e])
                np.testing.assert_allclose(obs[:, e], ro[0], rtol=0, atol=1e-9,
                                           err_msg=f"ep={ep} t={t} env={e}")
                np.testing.assert_allclose(rew[0, e], ro[1], rtol=1e-9, atol=1e-12)
