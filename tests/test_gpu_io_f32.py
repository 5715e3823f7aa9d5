"""Float32 actions and observations (``MultiAgentEnv(io_dtype="float32")``, the ``pgw_*_f32`` entry
points) on the GPU.  The kernels compute in float64 either way, so a float32 env driven with actions
``a32`` must reproduce a float64 env driven with ``a32.double()``: observations equal the float64
ones rounded to nearest float32, bit for bit, and rewards, done flags, state, voltages, episode
returns and power-flow state are identical.  Every kernel variant the scenarios reach is covered,
and the kernel names torch.profiler records prove that the float32 instantiation ran."""
import gc
import re
import warnings

import numpy as np
import pytest

from powergridworld_b200 import _native as N
from powergridworld_b200.scenarios import bench as SB
from powergridworld_b200.scenarios import catalog
from powergridworld_b200.scenarios.namespace import PRODUCT_NS as PNS

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    return torch


FIELDS = (N.FIELD_STATE_D, N.FIELD_STATE_I, N.FIELD_VOLTAGES, N.FIELD_EP_RETURN, N.FIELD_PF_STATE,
          N.FIELD_VBUS, N.FIELD_VMIN, N.FIELD_VMAX, N.FIELD_AGENT_P)


def _fields(env):
    torch = _torch()
    out = {}
    for f in FIELDS:
        if env.pf_solver is None and f in (N.FIELD_VOLTAGES, N.FIELD_PF_STATE, N.FIELD_VBUS,
                                           N.FIELD_VMIN, N.FIELD_VMAX):
            continue
        out[f] = env.get_field(f)
    torch.cuda.synchronize()
    return out


def _assert_fields_equal(f32, f64, what):
    torch = _torch()
    for k in f64:
        assert torch.equal(f32[k], f64[k]), f"{what}: field {k} differs"


def _io32_kernels(env, act):
    """(kernel, template arguments) of the component / fused kernels one step launches."""
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile
    env.set_option(N.OPT_GRAPHS, 0)
    # free the cyclic garbage of earlier tests (envs, profiler traces) before the session: in a long test
    # process torch.profiler has recorded none or only some of a session's kernels without this
    gc.collect()
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


def _twins(make, E, options=(), seed=0):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        e64 = make(num_envs=E)
        e32 = make(num_envs=E, io_dtype="float32")
    for opt, val in options:
        e64.set_option(opt, val)
        e32.set_option(opt, val)
    return e64, e32


def _reset_both(e64, e32, seed):
    torch = _torch()
    rng = np.random.default_rng(seed)
    soc = rng.uniform(10, 40, size=(e64.num_storage, e64.num_envs)) if e64.num_storage else None
    np.random.seed(seed)                               # randomised rosters: the same draws on both
    o64 = e64.reset_batch(soc).clone()
    np.random.seed(seed)
    o32 = e32.reset_batch(soc)
    assert o32.dtype == torch.float32 and torch.equal(o32, o64.float()), "reset observations"


def _run_episode(e64, e32, seed, steps=None, want=None):
    """Both envs over an episode (or `steps` steps) with float32 actions in [-1.2, 1.2];
    `want`: the template arguments the float32 env's kernels must show."""
    torch = _torch()
    _reset_both(e64, e32, seed)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    T = e64.episode_length if steps is None else steps
    shape = (e64.act_dim, e64.num_envs)
    for t in range(T):
        a32 = (torch.rand(shape, generator=gen, device="cuda", dtype=torch.float32) * 2.4 - 1.2).contiguous()
        if t == 1 and want is not None:                 # this step runs under the profiler
            got = _io32_kernels(e32, a32)
            assert want in got, f"float32 kernel {want} not among {got}"
            assert all(k[-1] == "true" for k in got), got
        else:
            e32.step_batch(a32)
        e64.step_batch(a32.double())
        assert e32.obs.dtype == torch.float32
        assert torch.equal(e32.obs, e64.obs.float()), f"obs t={t}"
        assert torch.equal(e32.rew, e64.rew), f"rew t={t}"
        assert torch.equal(e32.done, e64.done), f"done t={t}"
        if t in (0, T // 2):
            _assert_fields_equal(_fields(e32), _fields(e64), f"t={t}")
    _assert_fields_equal(_fields(e32), _fields(e64), "end of episode")


def _building_obs_subset(num_envs=1, **kw):
    """A stand-alone building with a non-default observation set: the table-driven path."""
    import pandas as pd
    return PNS.MultiAgentEnv(
        common_config={"start_time": "08-12-2020 00:00:00", "end_time": "08-13-2020 00:00:00",
                       "control_timedelta": pd.Timedelta(300, "s")},
        pf_config=None, num_envs=num_envs,
        agents=[{"name": "b", "bus": None, "cls": PNS.FiveZoneROMThermalEnergyEnv,
                 "config": {"obs_config": {"zone_temp": (16., 40.), "outdoor_temp": (0., 56.),
                                           "p_consumed": (0., 150.), "comfort_upper": (25., 30.)}}}],
        **kw)


def _house(step_meta):
    from tests.test_hs_tables_emu import house_batch
    return lambda **kw: house_batch("shipped", step_meta=step_meta, **kw)


def _c1(**kw):
    return SB.c1_env(pf_kernel="tc2", **kw)


F, T_ = "false", "true"
KERNEL_CASES = {
    # C1 on the fused kernel: actions staged in shared memory by 128-byte TMA rows
    "c1_fused_4096": (_c1, 4096, (), ("step_fused_kernel", F, T_)),
    # 4094 envs: E % 4 != 0, so float32 tiles read their actions from global memory (float64 stages them)
    "c1_fused_4094": (_c1, 4094, (), ("step_fused_kernel", F, T_)),
    # ~14 000 envs, PGW_OPT_FUSED = 2: CTAs run several tiles
    "c1_fused_multi_tile": (_c1, 14000, ((N.OPT_FUSED, 2),), ("step_fused_kernel", F, T_)),
    "c1_component_kernel_tc2": (_c1, 4096, ((N.OPT_FUSED, 0),), ("component_kernel", F, F, F, T_)),
    "c1_fp64_power_flow": (lambda **k: SB.c1_env(pf_kernel="fp64", **k), 1024, (),
                           ("component_kernel", F, F, F, T_)),
    # C2 = EV(100) + PV + storage without a feeder: the component-only path
    "c2_component_only": (SB.c2_env, 4096, (), ("component_kernel", F, F, F, T_)),
    "ev_per_env_rosters": (lambda **k: PNS.MultiAgentEnv(
        **catalog.randomized_ev_scenario(PNS, PNS.OpenDSSSolver), **k), 256, (),
        ("component_kernel", F, F, T_, T_)),
    "c3_123_bus": (lambda **k: SB.c3_env(pf_kernel="auto", **k), 1024, (),
                   ("component_kernel", F, F, F, T_)),
    "hs_house": (_house(False), 512, (), ("component_kernel", T_, F, F, T_)),
    "hs_house_telemetry": (_house(True), 512, (), ("component_kernel", T_, T_, F, T_)),
    "building_obs_subset": (_building_obs_subset, 512, (), ("component_kernel", F, F, F, T_)),
}


@pytest.mark.parametrize("name", list(KERNEL_CASES))
def test_float32_io_equals_float64_rounded(name):
    make, E, options, want = KERNEL_CASES[name]
    e64, e32 = _twins(make, E, options)
    _run_episode(e64, e32, seed=11, want=want)
    e64.close()
    e32.close()


def _host_run(env, soc, acts, setup):
    """reset_host / step_host of a float32 env in one of three setups; host copies of the results."""
    torch = _torch()
    E = env.num_envs
    out = []
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        if setup == "pinned":
            env.set_option(N.OPT_HOST_ZERO_COPY, 1)
            out.append(np.array(env.reset_host(soc)))
            for a in acts:
                o, r, d = env.step_host(torch.from_numpy(a).pin_memory())
                out.append((np.array(o), np.array(r), np.array(d)))
        else:
            env.set_option(N.OPT_HOST_ZERO_COPY, 0 if setup == "staged x4" else 1)
            env.set_option(N.OPT_HOST_CHUNKS, 4 if setup == "staged x4" else 0)
            s = torch.cuda.current_stream().cuda_stream
            o = np.empty((env.obs_dim, E), np.float32)
            sp = np.ascontiguousarray(soc)
            N.check(env._lib.pgw_reset_host_f32(env._h, sp.ctypes.data, o.ctypes.data, s))
            env.episode_step, env._needs_reset = 0, False
            out.append(o.copy())
            for a in acts:                                 # pageable NumPy buffers: the staged path
                o = np.empty((env.obs_dim, E), np.float32)
                r = np.empty((len(env.agents), E))
                d = np.empty(E, np.uint8)
                N.check(env._lib.pgw_step_host_f32(env._h, a.ctypes.data, o.ctypes.data, r.ctypes.data,
                                                   d.ctypes.data, s))
                env.episode_step += 1
                out.append((o, r, d))
    st.synchronize()
    return out


def test_host_paths_equal_the_device_path():
    torch = _torch()
    E, T = 4096, 12
    rng = np.random.default_rng(5)
    soc = rng.uniform(10, 40, size=(3, E))
    acts = [rng.uniform(-1.2, 1.2, size=(24, E)).astype(np.float32) for _ in range(T)]
    dev = _c1(num_envs=E, io_dtype="float32")
    want = [dev.reset_batch(soc).cpu().numpy()]
    for a in acts:
        o, r, d, _ = dev.step_batch(torch.from_numpy(a).cuda())
        want.append((o.cpu().numpy(), r.cpu().numpy(), d.cpu().numpy()))
    dev.close()
    for setup in ("pinned", "pageable", "staged x4"):
        env = _c1(num_envs=E, io_dtype="float32")
        got = _host_run(env, soc, acts, setup)
        assert got[0].dtype == np.float32
        np.testing.assert_array_equal(got[0], want[0], err_msg=f"{setup} reset")
        for t in range(T):
            assert got[t + 1][0].dtype == np.float32
            for k in range(3):
                np.testing.assert_array_equal(got[t + 1][k], want[t + 1][k], err_msg=f"{setup} t={t} out {k}")
        env.close()


def test_graphs_one_per_io_form():
    torch = _torch()
    E, T = 1024, 8
    st = torch.cuda.Stream()
    rng = np.random.default_rng(6)
    soc = rng.uniform(10, 40, size=(3, E))
    acts = [torch.from_numpy(rng.uniform(-1.2, 1.2, size=(24, E)).astype(np.float32)) for _ in range(T)]
    with torch.cuda.stream(st):
        # a fresh float32 action tensor every step: one capture, its nodes re-pointed
        env = _c1(num_envs=E, io_dtype="float32")
        env.reset_batch(soc)
        for a in acts:
            env.step_batch(a.cuda())
        st.synchronize()
        assert int(env._lib.pgw_graph_captures(env._h)) == 1
        env.close()
        # one handle alternating float64 and float32 steps: two captures, and the trajectory of a
        # float64 handle driven with the same (widened) actions
        one, ref = _c1(num_envs=E), _c1(num_envs=E)
        one.reset_batch(soc)
        ref.reset_batch(soc)
        o32 = torch.empty((one.obs_dim, E), dtype=torch.float32, device="cuda")
        s = torch.cuda.current_stream().cuda_stream
        for t, a in enumerate(acts):
            a64 = a.double().cuda()
            if t % 2:
                a32 = a.cuda()
                N.check(one._lib.pgw_step_f32(one._h, a32.data_ptr(), o32.data_ptr(), one.rew.data_ptr(),
                                              one.done.data_ptr(), s))
                one.episode_step += 1
            else:
                one.step_batch(a64)
            ref.step_batch(a64)
            if t % 2:
                assert torch.equal(o32, ref.obs.float()), t
            else:
                assert torch.equal(one.obs, ref.obs), t
            assert torch.equal(one.rew, ref.rew), t
        st.synchronize()
        assert int(one._lib.pgw_graph_captures(one._h)) == 2
        _assert_fields_equal(_fields(one), _fields(ref), "alternating handle")


def test_checkpoint_round_trip_and_dtype_mismatch():
    torch = _torch()
    E, k, T = 512, 5, 10
    gen = torch.Generator(device="cuda").manual_seed(3)
    acts = [(torch.rand((24, E), generator=gen, device="cuda") * 2.4 - 1.2).contiguous() for _ in range(T)]
    soc = np.random.default_rng(4).uniform(10, 40, size=(3, E))
    a = _c1(num_envs=E, io_dtype="float32")
    a.reset_batch(soc)
    for t in range(k):
        a.step_batch(acts[t])
    ckpt = a.state_dict()
    assert ckpt["obs"].dtype == torch.float32
    rest = []
    for t in range(k, T):
        o, r, _, _ = a.step_batch(acts[t])
        rest.append((o.clone(), r.clone()))
    b = _c1(num_envs=E, io_dtype="float32")
    b.load_state_dict(ckpt)
    assert torch.equal(b.obs, ckpt["obs"])
    for t in range(k, T):
        o, r, _, _ = b.step_batch(acts[t])
        assert torch.equal(o, rest[t - k][0]) and torch.equal(r, rest[t - k][1]), t
    c64 = _c1(num_envs=E)
    with pytest.raises(ValueError, match="io_dtype"):
        c64.load_state_dict(ckpt)
    c64.reset_batch(soc)
    with pytest.raises(ValueError, match="io_dtype"):
        b.load_state_dict(c64.state_dict())
    for e in (a, b, c64):
        e.close()


def test_meta_batch_under_float32():
    torch = _torch()
    E = 256
    e64, e32 = _twins(SB.c2_env, E)
    _reset_both(e64, e32, 8)
    gen = torch.Generator(device="cuda").manual_seed(8)
    for t in range(20):
        a = (torch.rand((e64.act_dim, E), generator=gen, device="cuda") * 2.4 - 1.2).contiguous()
        e32.step_batch(a)
        e64.step_batch(a.double())
    m64, m32 = e64.meta_batch(), e32.meta_batch()
    # exact oracle: the metas the float64 env's state gives when its observation rows are rounded to
    # float32 (the float32 env's rows equal those bit for bit, checked above)
    from powergridworld_b200.multiagent_env import _MetaCtx
    sd = e64.get_field(N.FIELD_STATE_D)
    want = {a.name: a._meta(_MetaCtx(e64, i, sd, e64.obs.float(), e64.episode_step, None, True))
            for i, a in enumerate(e64.agents)}
    ev_obs_keys = set(e64.agents[0]._obs_labels)
    checked = {"f32": 0, "f64": 0}

    def walk(w, x32, x64, path):
        if isinstance(w, dict):
            assert set(w) == set(x32) == set(x64), path
            for k in w:
                walk(w[k], x32[k], x64[k], path + (k,))
        elif isinstance(w, torch.Tensor):
            assert x32.dtype == w.dtype and torch.equal(x32, w), path
            if x32.dtype == torch.float32:
                # only the station's entries built from the delivered observation rows are float32
                assert path[0] == "ev" and path[-1] in ev_obs_keys | {"peak_reward"}, path
                checked["f32"] += 1
            else:
                assert torch.equal(x32, x64), path
                checked["f64"] += 1
        else:
            assert x32 == w == x64 or all(np.isnan(v) for v in (x32, w, x64)), path

    walk(want, m32, m64, ())
    assert checked["f32"] > 0 and checked["f64"] > 0, checked
    e64.close()
    e32.close()


def test_batched_joint_vector_env_float32_episode():
    from powergridworld_b200.adapters import BatchedJointVectorEnv
    E = 256
    cfg = dict(catalog.buildings_scenario(PNS, PNS.OpenDSSSolver, 1.2), max_episode_steps=12,
               env_cls=PNS.CoordinatedMultiBuildingControlEnv, pf_kernel="tc2")
    vec = BatchedJointVectorEnv(cfg, num_envs=E, io_dtype="float32")
    assert vec.single_action_space.dtype == np.float32 and vec.observation_space.dtype == np.float32
    ref = PNS.CoordinatedMultiBuildingControlEnv(**{k: v for k, v in cfg.items() if k != "env_cls"},
                                                 num_envs=E, io_dtype="float32")
    soc = np.random.default_rng(1).uniform(10, 40, size=(ref.num_storage, E))
    obs, _ = vec.reset(options={"init_storage": soc})
    assert obs.dtype == np.float32
    np.testing.assert_array_equal(obs, ref.reset_host(soc).T)
    rng = np.random.default_rng(2)
    steps = vec.env.episode_length
    for t in range(steps):
        a = rng.uniform(-1.2, 1.2, size=(E, ref.act_dim)).astype(np.float32)
        o, r, term, trunc, info = vec.step(a)
        o2, r2, d2 = ref.step_host(np.ascontiguousarray(a.T))
        np.testing.assert_array_equal(info["agent_rewards"], r2)
        np.testing.assert_array_equal(info["final_observation"] if t == steps - 1 else o, o2.T)
    assert vec.episodes == 1
    vec.close()
    ref.close()


def test_rllib_base_env_float32_steps_like_step_host():
    from powergridworld_b200.adapters import RLlibBatchedBaseEnv
    E = 64
    cfg = dict(catalog.buildings_scenario(PNS, PNS.OpenDSSSolver, 1.2), max_episode_steps=6,
               env_cls=PNS.CoordinatedMultiBuildingControlEnv, pf_kernel="tc2")
    base = RLlibBatchedBaseEnv(cfg, num_envs=E, io_dtype="float32")
    ref = PNS.CoordinatedMultiBuildingControlEnv(**{k: v for k, v in cfg.items() if k != "env_cls"},
                                                 num_envs=E, io_dtype="float32")
    np.random.seed(5)
    obs, *_ = base.poll()
    np.random.seed(5)
    o_ref = ref.reset_host()
    rng = np.random.default_rng(4)
    for t in range(base.env.episode_length):
        flat = rng.uniform(-1.2, 1.2, size=(ref.act_dim, E)).astype(np.float32)
        actions = {}
        for i in range(E):
            actions[i] = {}
            for agent, comp, a0, n in base._act_items:
                v = flat[a0:a0 + n, i]
                if comp is None:
                    actions[i][agent] = v
                else:
                    actions[i].setdefault(agent, {})[comp] = v
        base.send_actions(actions)
        obs, rew, term, trunc, infos, _ = base.poll()
        o_ref, r_ref, d_ref = ref.step_host(flat)
        for i in (0, E // 2, E - 1):
            for agent, comp, o0, n in base._obs_items:
                got = obs[i][agent] if comp is None else obs[i][agent][comp]
                assert got.dtype == np.float32
                np.testing.assert_array_equal(got, o_ref[o0:o0 + n, i])
            for k, a in enumerate(ref.agent_names):
                assert rew[i][a] == float(r_ref[k, i])
    assert term[0]["__all__"]
    base.stop()
    ref.close()


def test_misaligned_float32_actions_fall_back_to_global_reads():
    """A contiguous float32 action view that starts 4 bytes past a 16-byte boundary: the fused kernel
    must not stage its tiles with bulk copies (misaligned source), and the results must not change."""
    torch = _torch()
    E, T = 4096, 6
    e_a, e_b = _c1(num_envs=E, io_dtype="float32"), _c1(num_envs=E, io_dtype="float32")
    soc = np.random.default_rng(12).uniform(10, 40, size=(3, E))
    e_a.reset_batch(soc)
    e_b.reset_batch(soc)
    gen = torch.Generator(device="cuda").manual_seed(12)
    buf = torch.empty(24 * E + 4, dtype=torch.float32, device="cuda")
    for t in range(T):
        a = (torch.rand((24, E), generator=gen, device="cuda") * 2.4 - 1.2).contiguous()
        view = buf[1:1 + 24 * E].view(24, E)
        view.copy_(a)
        assert view.is_contiguous() and view.data_ptr() % 16 == 4
        e_a.step_batch(a)
        e_b.step_batch(view)
        assert torch.equal(e_a.obs, e_b.obs) and torch.equal(e_a.rew, e_b.rew), t
    e_a.close()
    e_b.close()


def test_errors():
    torch = _torch()
    E = 64
    env = _c1(num_envs=E, io_dtype="float32")
    env.reset_batch(np.full((3, E), 20.0))
    with pytest.raises(ValueError, match="float32"):
        env.step_batch(torch.zeros((24, E), dtype=torch.float64, device="cuda"))
    env.close()
    one = _c1(num_envs=1, io_dtype="float32")
    for call in (lambda: one.reset(), lambda: one.get_obs(), lambda: one.step({})):
        with pytest.raises(RuntimeError, match="float64"):
            call()
    one.close()
