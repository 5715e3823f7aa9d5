"""GPU tier: the fused step kernel's fixed point runs on mma.sync in two m-tiles of 16 envs per
32-env tile, and each m-tile leaves the loop when its own envs have converged.  So an env's
results may depend on the 15 envs of its m-tile and on nothing else: here the halves of the tiles
need different iteration counts (one half's actions swing from one bound to the other every step,
the other's hold still), and the same envs stepped with the halves paired differently, and in the
other m-tile, must give the same bits.  The last tile is ragged: its second m-tile has no env."""
import gc
import re

import numpy as np
import pytest
import torch

from powergridworld_b200 import _native as N
from powergridworld_b200.scenarios import bench as SB

pytestmark = pytest.mark.gpu

FIELDS = (N.FIELD_VOLTAGES, N.FIELD_PF_STATE, N.FIELD_PF_ITERS, N.FIELD_EP_RETURN, N.FIELD_VMIN,
          N.FIELD_VMAX, N.FIELD_VBUS)


def _fused_kernels(env, act):
    from torch.profiler import ProfilerActivity, profile
    # free the cyclic garbage of earlier tests (envs, profiler traces) before the session: in a long test
    # process torch.profiler has recorded none or only some of a session's kernels without this
    gc.collect()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        env.step_batch(act)
        torch.cuda.synchronize()
    found = set()
    for ev in prof.events():
        m = re.search(r"step_fused_kernel<([^>]*)>", ev.name)
        if m:
            found.add(tuple(x.strip() for x in m.group(1).split(",")))
    return found


def test_m_tiles_leave_the_loop_on_their_own():
    halves = 40                                        # 20 full tiles, then a tile of 10 envs
    E, T = 16 * halves + 10, 8
    # B holds the halves of A rotated by one: every full half gets a new partner and the other m-tile
    perm = np.concatenate([np.arange(16 * ((h + 1) % halves), 16 * ((h + 1) % halves) + 16)
                           for h in range(halves)] + [np.arange(16 * halves, E)])
    a, b = SB.c1_env(num_envs=E, pf_kernel="tc2"), SB.c1_env(num_envs=E, pf_kernel="tc2")
    for env in (a, b):
        env.set_option(N.OPT_FUSED, 2)
        env.set_option(N.OPT_GRAPHS, 0)
    rng = np.random.default_rng(13)
    soc = rng.uniform(5, 45, size=(a.num_storage, E))
    calm = rng.uniform(-0.2, 0.2, size=(a.act_dim, E))
    swing = (np.arange(E) // 16) % 2 == 1              # the second m-tile of every tile
    differ = 0
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        oa = a.reset_batch(soc)
        ob = b.reset_batch(np.ascontiguousarray(soc[:, perm]))
        assert torch.equal(oa[:, perm], ob)
        for t in range(T):
            act = np.where(swing[None, :], 1.1 if t % 2 else -1.1, calm)
            ta = torch.as_tensor(act).cuda()
            tb = torch.as_tensor(np.ascontiguousarray(act[:, perm])).cuda()
            if t == 2:
                names = _fused_kernels(a, ta) | _fused_kernels(b, tb)
                assert names == {("false", "false")}, names
                oa, ra, da = a.obs, a.rew, a.done
                ob, rb, db = b.obs, b.rew, b.done
            else:
                oa, ra, da, _ = a.step_batch(ta)
                ob, rb, db, _ = b.step_batch(tb)
            msg = f"step {t}"
            assert torch.equal(oa[:, perm], ob), f"observations, {msg}"
            assert torch.equal(ra[:, perm], rb), f"rewards, {msg}"
            assert torch.equal(da[perm], db), f"done, {msg}"
            for fld in FIELDS:
                fa, fb = a.get_field(fld), b.get_field(fld)
                assert torch.equal(fa[perm] if fa.dim() == 1 else fa[:, perm], fb), f"field {fld}, {msg}"
            it = a.get_field(N.FIELD_PF_ITERS).abs().cpu().numpy()
            assert it.min() > 0, f"a power flow did not converge, {msg}"
            per_half = it[:16 * halves].reshape(halves // 2, 2, 16).max(axis=2)
            differ += int((per_half[:, 0] != per_half[:, 1]).sum())
    st.synchronize()
    assert differ > 0, "the halves of every tile needed the same iterations: the test misses its case"
