"""CPU tier of the float32 I/O option (``MultiAgentEnv(io_dtype="float32")``): argument checks,
the adapters' spaces, and the host build of the component arithmetic with float32 actions and
observations (tests/io_f32_host.cpp, ``AgentIOT<float, float>``) against the float64 host build
(tests/emu) on golden scenarios.  The arithmetic is float64 either way, so driven with the same
float32 actions the two builds must agree bit for bit: observations after rounding to float32,
state and rewards exactly.  The GPU tier is tests/test_gpu_io_f32.py."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from powergridworld_b200 import adapters
from tests import scenarios as S
from tests.emu.harness import EmulatedEnv
from tests.product_ns import PRODUCT_NS as NS
from tests.test_hs_tables_emu import house_batch

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")


def _heterogeneous(**k):
    return NS.MultiAgentEnv(**S.heterogeneous_scenario(NS, NS.OpenDSSSolver, 0.65), **k)


def _buildings(**k):
    return NS.CoordinatedMultiBuildingControlEnv(**S.buildings_scenario(NS, NS.OpenDSSSolver, 1.2), **k)


def test_io_dtype_is_recorded_and_validated():
    assert _heterogeneous(_dry_run=True).io_dtype == "float64"
    assert _heterogeneous(_dry_run=True, io_dtype="float32").io_dtype == "float32"
    for bad in ("float16", "fp32", np.float32, None):
        with pytest.raises(ValueError, match="io_dtype"):
            _heterogeneous(_dry_run=True, io_dtype=bad)


def test_float32_entry_points_are_declared_exported_and_bound():
    import re
    from powergridworld_b200 import _native as N
    root = os.path.dirname(HERE)
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(root, "include", "pgw.h")).read(), flags=re.S)
    declared = set(re.findall(r"\b(pgw_\w+_f32)\s*\(", text))
    assert declared == set(N.SYMBOLS_F32) == {"pgw_reset_f32", "pgw_step_f32", "pgw_reset_host_f32",
                                              "pgw_step_host_f32"}
    assert not declared & set(N.SYMBOLS)
    lib = N.lib()
    for name, (_, args) in N.SYMBOLS_F32.items():
        assert getattr(lib, name).argtypes == args
    # same arity as the float64 forms they mirror
    for name in N.SYMBOLS_F32:
        assert len(N.SYMBOLS_F32[name][1]) == len(N.SYMBOLS[name[:-4]][1])


class _NoDeviceEnv:
    """What the adapters read from an env, without opening a device handle."""

    def __new__(cls, io_dtype, **kw):
        return _heterogeneous(_dry_run=True, io_dtype=io_dtype)


@pytest.mark.parametrize("io_dtype", ["float64", "float32"])
def test_adapter_spaces_have_the_io_dtype(io_dtype):
    want = np.dtype(io_dtype)
    vec = adapters.BatchedJointVectorEnv({"env_cls": _NoDeviceEnv}, num_envs=3, io_dtype=io_dtype)
    for sp in (vec.single_observation_space, vec.single_action_space, vec.observation_space,
               vec.action_space):
        assert np.dtype(sp.dtype) == want
    assert vec.action_space.shape == (3, vec.env.act_dim)
    base = adapters.RLlibBatchedBaseEnv({"env_cls": _NoDeviceEnv}, num_envs=3, io_dtype=io_dtype)

    def boxes(sp):
        if isinstance(sp, dict) or hasattr(sp, "spaces") and isinstance(sp.spaces, dict):
            for v in (sp.spaces if hasattr(sp, "spaces") else sp).values():
                yield from boxes(v)
        else:
            yield sp

    found = list(boxes(base.observation_space)) + list(boxes(base.action_space))
    assert found and all(np.dtype(b.dtype) == want for b in found)


def _build_f32_host(tmp):
    src = os.path.join(HERE, "io_f32_host.cpp")
    so = os.path.join(tmp, "libpgw_io_f32.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC",
                           "-x", "c++", "-o", so, src])
    return C.CDLL(so)


def _f32_twin(env, lib):
    """An EmulatedEnv whose library and observation buffer are the float32 build's."""
    emu = EmulatedEnv(env)
    emu.lib = lib
    emu.obs = np.zeros((env.obs_dim, emu.E), dtype=np.float32)
    return emu


def _step(emu, actions):
    """EmulatedEnv.step without its float64 conversion of the actions."""
    event = emu.t + 1
    emu.lib.emu_step(C.byref(emu._args(event, actions=np.ascontiguousarray(actions))))
    emu._powerflow(event, controllable=True)
    pen = emu.env._penalty
    if pen is not None:
        node = emu.env.pf_solver.node_for_bus_name(str(list(set(emu.env.agent_name_bus_map.values()))[0]))
        v = emu.vmag[node]
        emu.rew -= (np.maximum(0.0, np.maximum(pen[0] - v, v - pen[1])) * pen[2]) / emu.A
    emu.t += 1


CASES = {
    "heterogeneous": (lambda: _heterogeneous(_dry_run=True), "heterogeneous"),
    "c0_buildings": (lambda: _buildings(_dry_run=True), "c0_buildings"),
    "hs_shipped": (lambda: house_batch("shipped", _dry_run=True), "hs_shipped"),
}


@pytest.mark.parametrize("name", list(CASES))
def test_float32_host_build_equals_float64_rounded(name):
    make, gold = CASES[name]
    g = np.load(os.path.join(GOLD, gold + ".npz"))
    env = make()
    with tempfile.TemporaryDirectory() as tmp:
        lib32 = _build_f32_host(tmp)
        e64, e32 = EmulatedEnv(env), _f32_twin(env, lib32)
        soc = np.asarray(g["init_soc"], dtype=np.float64).reshape(-1, 1)
        e64.reset(soc)
        e32.reset(soc)
        assert e32.obs.dtype == np.float32
        np.testing.assert_array_equal(e32.obs, e64.obs.astype(np.float32))
        rng = np.random.default_rng(3)
        T = min(g["actions"].shape[0], 96)
        for t in range(T):
            a32 = rng.uniform(-1.2, 1.2, size=(env.act_dim, 1)).astype(np.float32)
            _step(e64, a32.astype(np.float64))
            _step(e32, a32)
            # bit for bit: the float32 build's observations are the float64 ones rounded to nearest
            assert np.array_equal(e32.obs, e64.obs.astype(np.float32)), f"obs t={t}"
            assert np.array_equal(e32.sd, e64.sd) and np.array_equal(e32.si, e64.si), f"state t={t}"
            assert np.array_equal(e32.rew, e64.rew) and np.array_equal(e32.agent_p, e64.agent_p), t
        # the rounding is visible: float32 observations are not the float64 values
        assert not np.array_equal(e32.obs.astype(np.float64), e64.obs)
