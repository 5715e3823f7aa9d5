"""GPU tier, round 2: the fused step kernel, the patched step graph, the zero-copy host step, the
step metas against reference-recorded ones, the checkpointed reset count."""
import os

import numpy as np
import pytest

from oracle.flatten import flat_obs, unflatten_action
from powergridworld_b200 import _native as N
from powergridworld_b200.scenarios import bench as SB
from powergridworld_b200.scenarios import catalog as S
from powergridworld_b200.scenarios.namespace import PRODUCT_NS as PNS

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _torch():
    import torch
    return torch


def _flatten_meta(meta, prefix=""):
    out = {}
    for k, v in meta.items():
        path = f"{prefix}{k}"
        if isinstance(v, dict):
            out.update(_flatten_meta(v, path + "/"))
        else:
            a = np.asarray(v, dtype=np.float64).reshape(-1)
            if a.size == 1 and not isinstance(v, np.ndarray):
                out[path] = float(a[0])
            else:
                for i, x in enumerate(a):
                    out[f"{path}/{i}"] = float(x)
    return out


@pytest.mark.parametrize("name", ["c0_buildings", "heterogeneous"])
def test_step_meta_matches_the_reference(name):
    """The 4th return value of step(): every stock component's meta as the UNMODIFIED reference
    returned it (tests/golden/make_golden_meta.py), keys and values."""
    g = np.load(os.path.join(GOLD, f"meta_{name}.npz"))
    if name == "c0_buildings":
        env = PNS.CoordinatedMultiBuildingControlEnv(**S.buildings_scenario(PNS, PNS.OpenDSSSolver, 1.2))
    else:
        env = PNS.MultiAgentEnv(**S.heterogeneous_scenario(PNS, PNS.OpenDSSSolver, 0.65))
    env.reset(init_storage=g["init_soc"])
    keys = [str(k) for k in g["keys"]]
    for t in range(g["actions"].shape[0]):
        _, _, _, meta = env.step(unflatten_action(env, g["actions"][t]))
        meta = {k: v for k, v in meta.items() if k != "voltage_violation"}   # train.py's meta_transform
        flat = _flatten_meta(meta)
        assert list(flat.keys()) == keys, (t, [k for k in keys if k not in flat], [k for k in flat if k not in keys])
        got, want = np.array([flat[k] for k in keys]), g["meta"][t]
        fin = np.isfinite(want)
        assert (np.isfinite(got) == fin).all()
        np.testing.assert_allclose(got[fin], want[fin], rtol=1e-9, atol=1e-7, err_msg=f"step {t}")


def test_meta_batch_shapes_and_values():
    torch = _torch()
    E = 64
    env = SB.c1_env(num_envs=E)
    rng = np.random.default_rng(0)
    soc = rng.uniform(10, 40, size=(env.num_storage, E))
    env.reset_batch(soc)
    lag = env._grid_snapshot(batch=True)
    env.step_batch(torch.as_tensor(rng.uniform(-1, 1, size=(env.act_dim, E))).cuda())
    m = env.meta_batch(lag)
    assert set(m) == {"building-0", "building-1", "building-2"}
    b = m["building-1"]
    assert b["storage"]["state_of_charge"].shape == (1, E)
    assert b["building"]["zone_temp_3"].shape == (E,) and b["building"]["p_consumed"].shape == (E,)
    sd = env.get_field(N.FIELD_STATE_D)
    stor = env.agents[1].envs[2]
    assert torch.equal(b["storage"]["state_of_charge"][0], sd[stor._slot["sd"][0]])
    assert float(b["pv"]["real_power"]) <= 0.0


@pytest.mark.parametrize("E", [33, 300, 4096])
def test_fused_step_kernel_matches_two_kernel_path(E):
    """Same batch through the fused kernel and through component_kernel + pf_tc2_kernel: the
    component side (observations, state, agent power, done) bit for bit, rewards and voltages
    within the float64 solver's bounds.  E = 33: odd stride (actions not staged by TMA) and a
    partial tile; 300: partial tile; 4096: the benchmark batch."""
    torch = _torch()
    T = 12
    rng = np.random.default_rng(E)
    envs = []
    for fused in (0, 2):
        env = SB.c1_env(num_envs=E, pf_kernel="tc2")
        env.set_option(N.OPT_FUSED, fused)
        envs.append(env)
    ref = SB.c1_env(num_envs=E, pf_tol=1e-13, pf_max_iter=200)       # FP64 SIMT solver
    soc = rng.uniform(5, 45, size=(ref.num_storage, E))
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        o0 = [e.reset_batch(soc).clone() for e in envs + [ref]]
        assert torch.equal(o0[0], o0[1])
        for t in range(T):
            act = torch.as_tensor(rng.uniform(-1.1, 1.1, size=(ref.act_dim, E))).cuda()
            res = [tuple(x.clone() for x in e.step_batch(act)[:3]) for e in envs + [ref]]
            (oa, ra, da), (ob, rb, db), (oc, rc, _) = res
            assert torch.equal(oa, ob) and torch.equal(da, db), f"observations / done, step {t}"
            np.testing.assert_allclose(rb.cpu().numpy(), rc.cpu().numpy(), rtol=1e-5, atol=2e-5,
                                       err_msg=f"rewards vs the FP64 solver, step {t}")
            np.testing.assert_allclose(ra.cpu().numpy(), rc.cpu().numpy(), rtol=1e-5, atol=2e-5)
            v = [e.get_field(N.FIELD_VOLTAGES).cpu().numpy() for e in envs + [ref]]
            np.testing.assert_allclose(v[1], v[2], rtol=0, atol=1e-6)
        for f in (N.FIELD_STATE_D, N.FIELD_AGENT_P):
            assert torch.equal(envs[0].get_field(f), envs[1].get_field(f))
        np.testing.assert_allclose(envs[1].get_field(N.FIELD_EP_RETURN).cpu().numpy(),
                                   ref.get_field(N.FIELD_EP_RETURN).cpu().numpy(), rtol=1e-5, atol=1e-3)
        it = envs[1].get_field(N.FIELD_PF_ITERS)
        assert int(it.min()) > 0, "the fused solve did not converge"
    st.synchronize()
    assert envs[0].launch_count > envs[1].launch_count


def test_fused_kernel_serves_the_heterogeneous_scenario_and_refuses_others():
    """EV station + grid-aware PV + composite on IEEE-13 (no penalty hook, lagged grid variables in
    the observations): fused = two-kernel bit for bit on the component side; a scenario that is
    not eligible (123-bus class feeder) refuses PGW_OPT_FUSED = 2."""
    torch = _torch()
    E, T = 96, 20
    rng = np.random.default_rng(4)
    envs = []
    for fused in (0, 2):
        env = PNS.MultiAgentEnv(**S.heterogeneous_scenario(PNS, PNS.OpenDSSSolver, 0.65), num_envs=E,
                                pf_kernel="tc2")
        env.set_option(N.OPT_FUSED, fused)
        envs.append(env)
    soc = rng.uniform(10, 200, size=(envs[0].num_storage, E))
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        for e in envs:
            e.reset_batch(soc)
        for t in range(T):
            act = torch.as_tensor(rng.uniform(-1, 1, size=(envs[0].act_dim, E))).cuda()
            (oa, ra, _, _), (ob, rb, _, _) = [e.step_batch(act) for e in envs]
            # the lagged voltages enter the observations: float32-level differences of the two
            # solvers' epilogues show up one step later, scaled by the observation ranges
            np.testing.assert_allclose(oa.cpu().numpy(), ob.cpu().numpy(), rtol=0, atol=2e-5, err_msg=f"t={t}")
            np.testing.assert_allclose(ra.cpu().numpy(), rb.cpu().numpy(), rtol=1e-5, atol=1e-3)
        assert torch.equal(envs[0].get_field(N.FIELD_STATE_I), envs[1].get_field(N.FIELD_STATE_I))
    st.synchronize()
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        big = SB.c3_env(num_envs=8, pf_kernel="tc2")
    with pytest.raises(N.NativeError):
        big.set_option(N.OPT_FUSED, 2)


@pytest.mark.parametrize("fused", [0, 1])
def test_one_step_graph_serves_fresh_action_tensors(fused):
    """A policy loop hands in a newly allocated action tensor every step: the handle captures ONE
    graph and re-points its kernel nodes (pgw_graph_captures stays 1), results equal a run that
    reuses one buffer, bit for bit."""
    import time
    torch = _torch()
    E, T = 512, 280
    rng = np.random.default_rng(2)
    a_env, b_env = (SB.c1_env(num_envs=E, pf_kernel="tc2") for _ in range(2))
    for e in (a_env, b_env):
        e.set_option(N.OPT_FUSED, fused)
    soc = rng.uniform(10, 40, size=(a_env.num_storage, E))
    acts = rng.uniform(-1, 1, size=(T, a_env.act_dim, E))
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        a_env.reset_batch(soc), b_env.reset_batch(soc)
        reuse = torch.empty((a_env.act_dim, E), dtype=torch.float64, device="cuda")
        keep, host_s = [], 0.0
        for t in range(T):
            fresh = torch.as_tensor(acts[t]).cuda()           # a new allocation every step
            keep.append(fresh)                                # (kept alive: no pointer is recycled)
            reuse.copy_(fresh)
            t0 = time.perf_counter()
            oa, ra, _, _ = a_env.step_batch(fresh)
            host_s += time.perf_counter() - t0
            ob, rb, _, _ = b_env.step_batch(reuse)
            if t % 40 == 0 or t == T - 1:
                assert torch.equal(oa, ob) and torch.equal(ra, rb), t
        assert a_env._lib.pgw_graph_captures(a_env._h) == 1
        assert b_env._lib.pgw_graph_captures(b_env._h) == 1
    st.synchronize()
    print(f"host time per step_batch with a fresh tensor: {1e6 * host_s / T:.1f} us")
    assert 1e6 * host_s / T < 60.0


@pytest.mark.parametrize("E", [2048 + 96, 7000])
@pytest.mark.parametrize("fused", [0, 1])
def test_host_step_zero_copy_staged_and_chunked_agree(fused, E):
    """pgw_step_host on page-locked buffers read / written in place, the same call staged through
    device buffers (one chunk and four pipelined chunks), a chain of zero-copy chunks, pageable
    buffers (always staged) and the device-buffer path: identical results, bit for bit.  E = 7000:
    219 tiles of the fused kernel, so that CTAs of the one-chunk calls run two tiles."""
    torch = _torch()
    T = 10
    rng = np.random.default_rng(9)
    soc = rng.uniform(10, 40, size=(3, E))
    acts = rng.uniform(-1, 1, size=(T, 24, E))
    outs = {}
    for label, zc, chunks, pinned in (("zero-copy", 1, 0, True), ("zero-copy chain", 1, 4, True),
                                      ("staged", 0, 1, True), ("staged x4", 0, 4, True),
                                      ("pageable", 1, 0, False), ("device", None, None, None)):
        env = SB.c1_env(num_envs=E, pf_kernel="tc2")
        env.set_option(N.OPT_FUSED, fused)
        res = []
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            if label == "device":
                env.reset_batch(soc)
                for t in range(T):
                    o, r, d, _ = env.step_batch(torch.as_tensor(acts[t]).cuda())
                    res.append((o.cpu().numpy().copy(), r.cpu().numpy().copy(), d.cpu().numpy().copy()))
            else:
                env.set_option(N.OPT_HOST_ZERO_COPY, zc)
                env.set_option(N.OPT_HOST_CHUNKS, chunks)
                env.reset_host(soc)
                for t in range(T):
                    a = torch.as_tensor(acts[t].copy())
                    if pinned:
                        a = a.pin_memory()
                        o, r, d = env.step_host(a)
                    else:                                     # raw C call on pageable NumPy buffers
                        o = np.empty((env.obs_dim, E)); r = np.empty((3, E)); d = np.empty(E, dtype=np.uint8)
                        an = np.ascontiguousarray(acts[t])
                        N.check(env._lib.pgw_step_host(env._h, an.ctypes.data, o.ctypes.data, r.ctypes.data,
                                                       d.ctypes.data, torch.cuda.current_stream().cuda_stream))
                        env.episode_step += 1
                    res.append((np.array(o), np.array(r), np.array(d)))
        st.synchronize()
        outs[label] = res
        env.close()
    for label, res in outs.items():
        for t in range(T):
            for k in range(3):
                np.testing.assert_array_equal(res[t][k], outs["device"][t][k], err_msg=f"{label} step {t} out {k}")


def test_checkpoint_carries_the_reset_count_of_a_house():
    """ADVICE round 1: a Home-Steward handle restored from a checkpoint must not treat its next
    reset as the first one (the house meta state and the storage cost survive resets)."""
    torch = _torch()
    E = 16
    rng = np.random.default_rng(3)
    a = SB.hs_env(num_envs=E)
    soc = rng.uniform(6, 9, size=(a.num_storage, E))
    acts = [torch.as_tensor(rng.uniform(-1, 1, size=(a.act_dim, E))).cuda() for _ in range(12)]
    a.reset_batch(soc)
    for x in acts[:6]:
        a.step_batch(x)
    ck = a.state_dict()
    assert ck["resets"] == 1
    b = SB.hs_env(num_envs=E)
    b.load_state_dict(ck)
    for env in (a, b):
        env.reset_batch(soc)                                  # second reset of the run
        for x in acts[6:]:
            env.step_batch(x)
    assert torch.equal(a.obs, b.obs) and torch.equal(a.rew, b.rew)
    assert torch.equal(a.get_field(N.FIELD_STATE_D), b.get_field(N.FIELD_STATE_D))
    fresh = SB.hs_env(num_envs=E)
    ck0 = fresh.state_dict()                                  # before any reset
    assert ck0["episode_step"] is None
    other = SB.hs_env(num_envs=E)
    other.load_state_dict(ck0)
    assert other._needs_reset


def test_standalone_solve_on_an_owned_solver_is_refused():
    env = SB.c1_env(num_envs=2)
    with pytest.raises(RuntimeError):
        env.pf_solver.calculate_power_flow(current_time="08-12-2021 00:00:00")
    solo = PNS.OpenDSSSolver(feeder_file="ieee_13_dss/IEEE13Nodeckt.dss",
                             loadshape_file="ieee_13_dss/annual_hourly_load_profile.csv",
                             system_load_rescale_factor=0.7)
    solo.calculate_power_flow(current_time="08-12-2021 00:00:00")
    v = solo.get_bus_voltages()
    assert len(v) == 38 and 0.9 < min(v.values()) < max(v.values()) < 1.1


def test_rllib_style_adapter_speaks_the_gymnasium_multi_agent_protocol():
    """examples/marl/rllib/heterogeneous/train.py:12-17 hands RLlib `MultiAgentEnv(**config)`; the
    adapter is the same env behind reset -> (obs, infos) / step -> 5-tuple."""
    from powergridworld_b200.adapters import RLlibMultiAgentEnv
    cfg = S.heterogeneous_scenario(PNS, PNS.OpenDSSSolver, 0.65)
    ad = RLlibMultiAgentEnv(dict(cfg, max_episode_steps=6))
    ref = PNS.MultiAgentEnv(**dict(cfg, max_episode_steps=6))
    np.random.seed(3)
    obs, infos = ad.reset(seed=3)
    np.random.seed(3)
    want = ref.reset()
    assert set(obs) == set(ad.possible_agents) == set(infos) == set(ref.agent_names)
    np.testing.assert_array_equal(flat_obs(ad.env, obs), flat_obs(ref, want))
    rng = np.random.default_rng(0)
    for t in range(ad.max_episode_steps):
        flat = rng.uniform(-1, 1, size=ref.act_dim)
        o, r, term, trunc, info = ad.step(unflatten_action(ad.env, flat))
        o2, r2, d2, m2 = ref.step(unflatten_action(ref, flat))
        np.testing.assert_array_equal(flat_obs(ad.env, o), flat_obs(ref, o2))
        assert r == r2 and term == d2 and not any(trunc.values())
        assert set(info) <= set(ref.agent_names) | {"__common__"}
        assert info["pv"]["real_power"] == m2["pv"]["real_power"]
    assert term["__all__"]


def test_batched_joint_vector_env_autoresets_and_matches_step_host():
    from powergridworld_b200.adapters import BatchedJointVectorEnv
    E = 96
    cfg = dict(S.buildings_scenario(PNS, PNS.OpenDSSSolver, 1.2), max_episode_steps=5,
               env_cls=PNS.CoordinatedMultiBuildingControlEnv, pf_kernel="tc2")
    vec = BatchedJointVectorEnv(cfg, num_envs=E)
    ref = PNS.CoordinatedMultiBuildingControlEnv(
        **{k: v for k, v in cfg.items() if k != "env_cls"}, num_envs=E)
    soc = np.random.default_rng(1).uniform(10, 40, size=(ref.num_storage, E))
    obs, _ = vec.reset(options={"init_storage": soc})
    want = ref.reset_host(soc)
    assert obs.shape == (E, ref.obs_dim) == vec.observation_space.shape
    np.testing.assert_array_equal(obs, want.T)
    rng = np.random.default_rng(2)
    steps = vec.env.episode_length
    for t in range(steps):
        a = rng.uniform(-1, 1, size=(E, ref.act_dim))
        o, r, term, trunc, info = vec.step(a)
        o2, r2, d2 = ref.step_host(np.ascontiguousarray(a.T))
        np.testing.assert_array_equal(info["agent_rewards"], r2)
        np.testing.assert_array_equal(r, r2.sum(axis=0))
        last = t == steps - 1
        assert term.all() == last and not trunc.any()
        np.testing.assert_array_equal(info["final_observation"] if last else o, o2.T)
    assert vec.episodes == 1 and o.shape == (E, ref.obs_dim)   # o is the next episode's first observation
    sl = vec.agent_obs_slices["building-1"]
    assert sl.stop - sl.start == sum(s.shape[0] for s in ref.observation_space["building-1"].values())


def test_rllib_base_env_adapter_steps_a_batch_like_independent_envs():
    """RLlib's BaseEnv protocol over a batch: poll / send_actions / try_reset with {env_id: {agent:
    ...}} dicts; every env id replays a single env driven through the dict API with the same SOC and
    actions (the heterogeneous scenario: composite, PV and EV-station agents)."""
    from powergridworld_b200.adapters import RLlibBatchedBaseEnv
    E, T = 5, 6
    cfg = dict(S.heterogeneous_scenario(PNS, PNS.OpenDSSSolver, 0.65), max_episode_steps=T + 1)
    be = RLlibBatchedBaseEnv(cfg, num_envs=E)
    singles = [PNS.MultiAgentEnv(**cfg) for _ in range(E)]
    rng = np.random.default_rng(4)
    soc = rng.uniform(10, 40, size=(be.env.num_storage, E))
    obs, infos = be.try_reset(options={"init_storage": soc})
    assert sorted(obs) == list(range(E))
    for i, s in enumerate(singles):
        want = s.reset(init_storage=soc[:, i])
        np.testing.assert_array_equal(flat_obs(be.env, obs[i]), flat_obs(s, want))
    for t in range(be.env.episode_length):
        flat = rng.uniform(-1, 1, size=(E, be.env.act_dim))
        be.send_actions({i: unflatten_action(be.env, flat[i]) for i in range(E)})
        obs, rew, term, trunc, infos, _ = be.poll()
        for i, s in enumerate(singles):
            o, r, d, _ = s.step(unflatten_action(s, flat[i]))
            np.testing.assert_allclose(flat_obs(be.env, obs[i]), flat_obs(s, o), rtol=0, atol=1e-12)
            assert rew[i].keys() == r.keys()
            np.testing.assert_allclose([rew[i][k] for k in r], list(r.values()), rtol=1e-12, atol=1e-12)
            assert term[i]["__all__"] == d["__all__"] and not trunc[i]["__all__"]
    assert term[0]["__all__"]
    first, _ = be.try_reset(0)
    rest, _ = be.try_reset(3)
    assert list(first) == [0] and list(rest) == [3]
    be.stop()


def test_event_index_and_device_clock_modes_interleave():
    """The fused step reads its event row through the host-supplied index when the graph's node
    parameters are rewritten for new caller buffers, and through the device clock when the same buffers
    come again: any interleaving of the two gives the trajectory of a run on one buffer.  At 300 envs
    and at 7000, where CTAs run two tiles, of which only the first waits for the event row."""
    torch = _torch()
    T = 14
    for E in (300, 7000):
        rng = np.random.default_rng(12)
        soc = rng.uniform(10, 40, size=(3, E))
        acts = rng.uniform(-1, 1, size=(T, 24, E))
        a_env, b_env = (SB.c1_env(num_envs=E, pf_kernel="tc2") for _ in range(2))
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            a_env.reset_batch(soc), b_env.reset_batch(soc)
            bufs = [torch.empty((24, E), dtype=torch.float64, device="cuda") for _ in range(3)]
            pattern = [0, 1, 1, 1, 0, 0, 2, 1, 1, 2, 2, 2, 0, 1]          # which buffer each step uses
            one = torch.empty((24, E), dtype=torch.float64, device="cuda")
            for t in range(T):
                x = torch.as_tensor(acts[t]).cuda()
                bufs[pattern[t]].copy_(x)
                one.copy_(x)
                oa, ra, _, _ = a_env.step_batch(bufs[pattern[t]])
                ob, rb, _, _ = b_env.step_batch(one)
                assert torch.equal(oa, ob) and torch.equal(ra, rb), (E, t)
            assert a_env._lib.pgw_graph_captures(a_env._h) == 1
            assert a_env.episode_step == b_env.episode_step == T
            assert torch.equal(a_env.get_field(N.FIELD_EP_RETURN), b_env.get_field(N.FIELD_EP_RETURN)), E
        st.synchronize()
