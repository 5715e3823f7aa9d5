"""GPU tier: the tc2 tensor-core power flow (csrc/powerflow_tc2.cu) and the FP64 SIMT kernel
(csrc/powerflow.cu) against a float64 reference of the same power flow (tests/pf_reference.py):
every tc2 tile width and FP64 row count on the 123-bus-class feeders, blocks of the FP64 kernel
that loop over several env groups, CTAs of tc2 that run several tiles (bit for bit against
batches whose CTAs run one), and the reward-hook epilogue with four thread groups."""
import gc
import re
import warnings

import numpy as np
import pytest

from powergridworld_b200 import _native as N
from powergridworld_b200.scenarios import bench as SB
from tests import pf_reference as R
from tests.product_ns import PRODUCT_NS as PNS
from tests.test_fused_step_reference import SHARD_FIELDS, _check_voltages, _config as _ieee13_config

pytestmark = pytest.mark.gpu

TILE = 128                                  # envs per tc2 tile
# Bounds against the float64 reference, about twice the worst errors measured on a B200 (1000 W)
# over the tests of this file: (node magnitudes incl. min / max / bus voltages, branch voltages u).
# tc2 stops at max |d u| < 1e-7 and has no FP64 polish above 16 branches; per tile width NCH:
TOL_TC2 = {4: (5e-7, 2.5e-7),               # measured 2.53e-7, 1.18e-7
           8: (4.5e-7, 2e-7),               # 2.27e-7, 9.67e-8
           11: (6e-7, 3.8e-7)}              # 2.95e-7, 1.88e-7 (C3, later tiles)
# The FP64 kernel stops at max |d u| < 1e-9; per padded row count nbp:
TOL_FP64 = {16: (2.3e-10, 2.3e-10),         # 1.12e-10, 1.13e-10 (C1, 9600 envs)
            32: (6.1e-11, 6.2e-11),         # 3.04e-11, 3.10e-11
            64: (7.4e-11, 8.5e-11),         # 3.67e-11, 4.24e-11
            96: (1.13e-10, 1.2e-10),        # 5.65e-11, 5.99e-11
            128: (9e-11, 1.37e-10)}         # 4.51e-11, 6.81e-11
# IEEE-13 through the two-kernel tc2 path, with the hook (FP64 polish): (nodes, the penalty node's
# float64 row, u); measured 2.46e-7, 3.17e-9, 4.82e-8 (C1) and 2.34e-7, 5.59e-9, 8.20e-8 (o16)
TOL_C1 = {"shipped": (5e-7, 6.5e-9, 1e-7), "o16": (5e-7, 1.2e-8, 1.7e-7)}
TOL_IEEE13 = (4.5e-7, None, 2e-7)           # no hook: 2.25e-7, 9.46e-8


def _torch():
    import torch
    return torch


@pytest.fixture(scope="module")
def feeders(tmp_path_factory):
    d = tmp_path_factory.mktemp("feeders")
    out = {n: R.synthetic_feeder(d, n) for n in (24, 50, 85)}
    out["x100"] = R.synthetic_feeder(d, extra=True)
    out["o16"] = R.feeder_file("o16", d)
    return out


def _env(cfg, hook=False, **kw):
    cls = PNS.CoordinatedMultiBuildingControlEnv if hook else PNS.MultiAgentEnv
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")       # agents on loads whose power the reference ignores
        return cls(**cfg, **kw)


def _nch(env):
    w = (env.pf_solver.feeder.nb + 7) // 8
    return next((c for c in (2, 4, 8, 11) if c >= w), None)


def _instantiations(torch, envs, act):
    """Template arguments of the power-flow kernels that one step of each env launches, from the
    kernel names torch.profiler records (plain launches: PGW_OPT_GRAPHS = 0 for the step)."""
    from torch.profiler import ProfilerActivity, profile
    for e in envs:
        e.set_option(N.OPT_GRAPHS, 0)
    # free the cyclic garbage of earlier tests (envs, profiler traces) before the session: in a long test
    # process torch.profiler has recorded none or only some of a session's kernels without this
    gc.collect()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for e, a in zip(envs, act):
            e.step_batch(a)
        torch.cuda.synchronize()
    for e in envs:
        e.set_option(N.OPT_GRAPHS, 1)
    found = set()
    for ev in prof.events():
        m = re.search(r"(pf_tc2_kernel|pf_fixed_point_kernel)<([^>]*)>", ev.name)
        if m:
            found.add((m.group(1),) + tuple(x.strip() for x in m.group(2).split(",")))
    return found


def _tc2(nch, m5, occ, polish=False):
    return ("pf_tc2_kernel", str(nch), str(m5).lower(), "false", str(occ), str(polish).lower())


def _fp64(nbp):
    return ("pf_fixed_point_kernel",) + {16: ("16", "1", "true"), 32: ("32", "1", "false"),
                                         64: ("32", "2", "false"), 96: ("32", "3", "false"),
                                         128: ("32", "4", "false")}[nbp]


# ------------------------------------------------------------------ (a) accuracy on 123-bus feeders
@pytest.mark.parametrize("fid", [24, 50, 85, "x100"])
def test_123_bus_feeders_match_float64_reference(feeders, fid):
    """300 envs (a ragged third tile), 8 steps, through tc2 (NCH = 4 streamed Znb chunks, 8 with an
    all-padding chunk, 11; none for x100) and through the FP64 kernel (nbp = 32 / 64 / 96 / 128),
    against the float64 reference: node magnitudes, min / max, bus voltages (three agents on one
    node, agents on a bus without a load and on model-2/5 loads), branch voltages."""
    torch = _torch()
    E, T = 300, 8
    cfg = lambda: R.synthetic_config(PNS, feeders[fid])
    fp64 = _env(cfg(), num_envs=E)
    envs = {"fp64": fp64}
    if fid == "x100":                           # beyond tc2: refused, and "auto" is the FP64 kernel
        with pytest.raises(N.NativeError, match="88 load"):
            _env(cfg(), num_envs=E, pf_kernel="tc2")
        envs["auto"] = _env(cfg(), num_envs=E, pf_kernel="auto")
    else:
        envs["tc2"] = _env(cfg(), num_envs=E, pf_kernel="tc2")
    f = fp64.pf_solver.feeder
    nch, nbp = _nch(fp64), fp64._nbp()
    rng = np.random.default_rng(sum(map(ord, str(fid))))
    soc = rng.uniform(5, 75, size=(fp64.num_storage, E))
    worst = {k: np.zeros(3) for k in envs}
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        for e in envs.values():
            e.reset_batch(soc)
        for t in range(T):
            act = torch.as_tensor(rng.uniform(-1.1, 1.1, size=(fp64.act_dim, E))).cuda()
            if t == 0:
                got = _instantiations(torch, list(envs.values()), [act] * len(envs))
                want = {_fp64(nbp)} | ({_tc2(nch, True, 2 if nch <= 4 else 1)} if "tc2" in envs else set())
                assert got == want, got
            else:
                for e in envs.values():
                    e.step_batch(act)
            p = fp64.get_field(N.FIELD_AGENT_P)
            for e in envs.values():
                assert torch.equal(e.get_field(N.FIELD_AGENT_P), p), f"agent powers, step {t}"
            u, _, v = R.solve64(f, R.step_powers(fp64, t, p.cpu().numpy()))
            for k, e in envs.items():
                tol = TOL_TC2[nch] if k == "tc2" else TOL_FP64[nbp]
                worst[k] = np.maximum(worst[k], _check_voltages(e, u, v, None, (tol[0], None, tol[1]), t, k))
            if "auto" in envs:
                for fld in SHARD_FIELDS:
                    assert torch.equal(envs["auto"].get_field(fld), fp64.get_field(fld)), f"auto, field {fld}"
    st.synchronize()
    for k, w in worst.items():
        print(f"synthetic {fid} (nb {f.nb}) {k}: max error nodes {w[0]:.2e}, u {w[2]:.2e}")


@pytest.mark.parametrize("case,E", [("c1", 9600), ("t85", 4900)])
def test_fp64_blocks_over_several_env_groups_match_float64_reference(feeders, case, E):
    """The FP64 kernel's grid is capped at 592 blocks: above 9472 envs at 16 threads per env
    (IEEE-13, Zbb rows in registers) and 4736 at 32 (85 branches, nbp = 96) blocks loop over a
    second env group.  The reference checks the first groups and the last ones, which ran as a
    block's second group."""
    torch = _torch()
    T = 6
    env = SB.c1_env(num_envs=E) if case == "c1" else _env(R.synthetic_config(PNS, feeders[85]), num_envs=E)
    f = env.pf_solver.feeder
    epb = 16 if f.nb <= 16 else 8
    assert (E + epb - 1) // epb > 592
    cols = np.r_[0:64, 592 * epb - 64:E]
    rng = np.random.default_rng(E)
    soc = rng.uniform(5, 45, size=(env.num_storage, E))
    worst, tol = np.zeros(3), TOL_FP64[env._nbp()]
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        env.reset_batch(soc)
        for t in range(T):
            act = torch.as_tensor(rng.uniform(-1.1, 1.1, size=(env.act_dim, E))).cuda()
            if t == 0:
                assert _instantiations(torch, [env], [act]) == {_fp64(env._nbp())}
            else:
                env.step_batch(act)
            p = env.get_field(N.FIELD_AGENT_P).cpu().numpy()[:, cols]
            u, _, v = R.solve64(f, R.step_powers(env, t, p))
            worst = np.maximum(worst, _check_voltages(env, u, v, None, (tol[0], None, tol[1]),
                                                      t, case, cols))
    st.synchronize()
    print(f"{case} FP64 at {E} envs: max error nodes {worst[0]:.2e}, u {worst[2]:.2e}")


# ------------------------------------------------------------------ (b) CTAs that run several tiles
SHARD_CASES = [("c1", 262144), ("c1", 75001), ("o16", 40000), ("ieee13", 100000), ("t24", 40000),
               ("t50", 40000), ("c3", 45000)]


@pytest.mark.parametrize("case,E", SHARD_CASES)
def test_tc2_multi_tile_ctas_equal_single_tile_shards(feeders, case, E):
    """A batch whose tc2 CTAs run several tiles equals, bit for bit, the same envs run as shards
    whose CTAs run one tile each (a tile's arithmetic depends only on its 128 envs, the tables and
    the event row), and its later tiles match the float64 reference.  Reaches: the FP64-polish
    build <2, *, false, 2, true> (c1: bench.py's C1 x 64; o16: the recomputed penalty row), the
    dense IEEE-13 build <2, *, false, 4> against the regular one of the shards, the streamed Znb
    chunks of <4, ..> (24 loads), <8, ..> (50 loads, up to three tiles per CTA) and <11, ..> (C3)."""
    torch = _torch()
    T = 4

    def make(n):
        if case == "c1":
            e = SB.c1_env(num_envs=n, pf_kernel="tc2")
        elif case == "o16":
            e = _env(_ieee13_config(PNS, feeders["o16"], "o16", True), True, num_envs=n, pf_kernel="tc2")
        elif case == "ieee13":
            e = _env(_ieee13_config(PNS, R.SHIPPED, "shipped", False), num_envs=n, pf_kernel="tc2")
        elif case == "c3":
            e = SB.c3_env(num_envs=n, pf_kernel="tc2")
        else:
            e = _env(R.synthetic_config(PNS, feeders[int(case[1:])]), num_envs=n, pf_kernel="tc2")
        e.set_option(N.OPT_FUSED, 0)           # the two-kernel path: component kernel + pf_tc2_kernel
        return e

    big = make(E)
    f = big.pf_solver.feeder
    nch, hook = _nch(big), case in ("c1", "o16")
    m5 = bool((np.asarray(f.branch_model) == 5).any())
    per_sm = 2 if nch <= 4 else 1
    tiles, shard = (E + TILE - 1) // TILE, 148 * per_sm * TILE
    dense = case == "ieee13"
    grid = min(tiles, 148 * (4 if dense else per_sm))
    assert tiles > grid, "every CTA runs one tile"
    bounds = list(range(0, E, shard)) + [E]
    parts = list(zip(bounds[:-1], bounds[1:]))
    shards = [make(b - a) for a, b in parts]
    row = big.pf_solver.node_for_bus_name(big.agent_name_bus_map[big.agent_names[0]]) if hook else None
    if hook:
        tol = TOL_C1["o16" if case == "o16" else "shipped"]
    elif nch == 2:
        tol = TOL_IEEE13
    else:
        tol = (TOL_TC2[nch][0], None, TOL_TC2[nch][1])
    cols = np.arange(grid * TILE, E)           # tiles that ran as a CTA's second or later tile
    rng = np.random.default_rng(E)
    soc = rng.uniform(5, 45, size=(big.num_storage, E))
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        ob = big.reset_batch(soc)
        for (a, b), s in zip(parts, shards):
            assert torch.equal(ob[:, a:b], s.reset_batch(np.ascontiguousarray(soc[:, a:b])))
        for t in range(T):
            act = torch.as_tensor(rng.uniform(-1.1, 1.1, size=(big.act_dim, E))).cuda()
            sact = [act[:, a:b].contiguous() for a, b in parts]
            counts = [e.launch_count for e in [big] + shards]
            if t == 0:
                got = _instantiations(torch, [big], [act])
                assert got == {_tc2(nch, m5, 4 if dense else per_sm, hook)}, got
                got = _instantiations(torch, shards, sact)
                assert got == {_tc2(nch, m5, per_sm, hook)}, got
            else:
                for e, x in zip([big] + shards, [act] + sact):
                    e.step_batch(x)
            assert [e.launch_count for e in [big] + shards] == [c + 2 for c in counts], \
                "a step did not run as the component kernel + the power-flow kernel"
            for (a, b), s in zip(parts, shards):
                msg = f"envs [{a}, {b}), step {t}"
                assert torch.equal(big.obs[:, a:b], s.obs), f"observations, {msg}"
                assert torch.equal(big.rew[:, a:b], s.rew), f"rewards, {msg}"
                assert torch.equal(big.done[a:b], s.done), f"done, {msg}"
            for fld in SHARD_FIELDS:
                whole = big.get_field(fld)
                for (a, b), s in zip(parts, shards):
                    part = whole[a:b] if whole.dim() == 1 else whole[:, a:b]
                    assert torch.equal(part, s.get_field(fld)), f"field {fld}, envs [{a}, {b}), step {t}"
        p = big.get_field(N.FIELD_AGENT_P).cpu().numpy()[:, cols]
        u, _, v = R.solve64(f, R.step_powers(big, T - 1, p))
        w = _check_voltages(big, u, v, row, tol, T - 1, f"{case}, later tiles", cols)
    st.synchronize()
    print(f"{case} at {E} envs ({tiles} tiles on {grid} CTAs), tiles >= {grid}: "
          f"max error nodes {w[0]:.2e}, float64 row {w[1]:.2e}, u {w[2]:.2e}")


# ------------------------------------------------------------------ (c) reward hook, four groups
def test_tc2_reward_hook_with_four_groups(feeders):
    """20 agents on one load of the 85-branch feeder (NCH = 11: G = 4 groups of 128 threads, the
    hook's agent loop runs twice; 18 of the agents' bus voltages come from the tail list when there
    is no hook): the hook changes no voltage, subtracts max(0, lo - v, v - hi) * 1e4 / A from every
    agent's reward (v = the device's magnitude at the penalty node), accumulates the episode
    return and writes the bus voltages; voltages match the float64 reference."""
    torch = _torch()
    E, T, A = 300, 8, 20
    cfg = lambda: R.synthetic_config(PNS, feeders[85], load_factor=2.0, hook_agents=A)
    hook, plain = _env(cfg(), True, num_envs=E, pf_kernel="tc2"), _env(cfg(), num_envs=E, pf_kernel="tc2")
    f = hook.pf_solver.feeder
    assert _nch(hook) == 11
    node = hook.pf_solver.node_for_bus_name("37a")
    lo, hi, unit = hook._penalty
    rng = np.random.default_rng(20)
    soc = rng.uniform(5, 75, size=(A, E))
    ret = torch.zeros((A, E), dtype=torch.float64, device="cuda")
    active, worst = 0, np.zeros(3)
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        hook.reset_batch(soc)
        plain.reset_batch(soc)
        for t in range(T):
            act = torch.as_tensor(rng.uniform(-1.1, 1.1, size=(A, E))).cuda()
            rh, rp = hook.step_batch(act)[1].clone(), plain.step_batch(act)[1].clone()
            for fld in (N.FIELD_VOLTAGES, N.FIELD_VMIN, N.FIELD_VMAX, N.FIELD_PF_STATE, N.FIELD_PF_ITERS,
                        N.FIELD_AGENT_P, N.FIELD_VBUS):
                assert torch.equal(hook.get_field(fld), plain.get_field(fld)), f"field {fld}, step {t}"
            vol = hook.get_field(N.FIELD_VOLTAGES)
            assert torch.equal(hook.get_field(N.FIELD_VBUS), vol[node].expand(A, E)), f"bus voltages, step {t}"
            v = vol[node]
            pen = torch.clamp(torch.maximum(lo - v, v - hi), min=0.0) * unit / A
            active += int((pen > 0).sum())
            torch.testing.assert_close(rp - rh, pen.expand(A, E), rtol=0,
                                       atol=4 * np.finfo(np.float64).eps * float(rp.abs().max() + pen.max()))
            ret += rh
            assert torch.equal(hook.get_field(N.FIELD_EP_RETURN), ret), f"episode return, step {t}"
            p = hook.get_field(N.FIELD_AGENT_P).cpu().numpy()
            u, _, vr = R.solve64(f, R.step_powers(hook, t, p))
            worst = np.maximum(worst, _check_voltages(hook, u, vr, None, (TOL_TC2[11][0], None, TOL_TC2[11][1]),
                                                      t, "hook"))
    st.synchronize()
    print(f"hook G=4: penalty active in {active} agent-steps; max error nodes {worst[0]:.2e}, u {worst[2]:.2e}")
    assert 0 < active < A * E * T, "the penalty was never (or always) active"
