"""CPU tier: pgw_create validates a spec BEFORE it touches CUDA -- every scenario of the catalog
passes the validation (the call then stops at the missing device), a spec that is off by a row
is rejected as PGW_ERR_INVALID (ADVICE round 1: out-of-range rows must not reach the kernels)."""
import ctypes as C

import numpy as np
import pytest
import torch

from powergridworld_b200 import _native as N
from powergridworld_b200.scenarios import bench as SB

INVALID = -1


def _create(env, mutate=None):
    spec, keep = env._build_spec()
    if mutate:
        mutate(spec)
    h = C.c_void_p()
    rc = N.lib().pgw_create(C.byref(spec), C.byref(h))
    if rc == 0:
        N.lib().pgw_destroy(h)
    return rc, N.lib().pgw_last_error().decode()


@pytest.mark.parametrize("make", [SB.c1_env, SB.c2_env, SB.c3_env, SB.hs_env])
def test_catalog_scenarios_pass_validation(make):
    rc, msg = _create(make(num_envs=4, _dry_run=True))
    assert rc != INVALID, msg
    if not torch.cuda.is_available():
        assert rc == -2 and "cudaGetDevice" in msg      # validated, then no device


def _bump(field, comp_type, delta):
    def mutate(spec):
        for i in range(spec.num_components):
            if spec.components[i].type == comp_type:
                setattr(spec.components[i], field, getattr(spec.components[i], field) + delta)
                return
        raise AssertionError("component kind not in the scenario")
    return mutate


@pytest.mark.parametrize("field,ctype,delta,what", [
    ("act_off", N.BUILDING, 10 ** 6, "action rows"),
    ("act_off", N.BUILDING, 19, "action rows"),          # 6 rows no longer fit behind the offset
    ("sd_off", N.STORAGE, 10 ** 6, "state rows"),
    ("sd_off", N.BUILDING, -1000, "state rows"),
    ("dtab_off", N.BUILDING, 10 ** 6, "event-row"),
    ("obs_dim", N.STORAGE, -1, "observation rows"),
])
def test_off_by_rows_is_rejected(field, ctype, delta, what):
    rc, msg = _create(SB.c1_env(num_envs=4, _dry_run=True), _bump(field, ctype, delta))
    assert rc == INVALID and (what in msg or "out of range" in msg), (rc, msg)


def test_ev_station_tables_are_checked():
    rc, msg = _create(SB.c2_env(num_envs=4, _dry_run=True), _bump("itab_off", N.EV, 10 ** 6))
    assert rc == INVALID and "event-row" in msg
    rc, msg = _create(SB.c2_env(num_envs=4, _dry_run=True), _bump("si_off", N.EV, 1))
    assert rc == INVALID and "state rows" in msg


def test_per_env_rosters_validate_their_inputs(tmp_path):
    """EVChargingEnv(randomize=True) in a batch: window words hold whole minutes in [0, 65535) and a
    station holds at most 256 vehicles; anything else is refused loudly on the host."""
    import pandas as pd
    from powergridworld_b200.agents.vehicles.ev_charging_env import EVChargingEnv, _popcount
    assert [_popcount(np.int32(v)) for v in (0, 1, -1, 0x40000001)] == [0.0, 1.0, 32.0, 2.0]
    st = EVChargingEnv(num_vehicles=5, randomize=True, name="ev")
    st._num_envs = 3
    np.random.seed(0)
    st._draw_roster()
    assert st._rows.shape == (3, 5)
    words, energy = st._per_env_rows()
    assert words.shape == (5, 3) and words.dtype == np.uint32 and energy.shape == (5, 3)
    start, end = words >> 16, words & 0xFFFF
    np.testing.assert_array_equal(start.T, np.floor(st._roster_start[st._rows]))
    np.testing.assert_array_equal(end.T, np.floor(st._roster_end[st._rows]))
    np.testing.assert_array_equal(energy.T, st._roster_energy[st._rows])
    # the reference rounds parking times down to the step (ev_charging_env.py:75-76): only a fractional
    # step leaves fractional minutes
    csv = tmp_path / "vehicles.csv"
    pd.DataFrame({"start_time_min": [12.7, 20.0, 30.0], "end_time_park_min": [102.9, 200.0, 300.0],
                  "energy_required_kwh": [5.0, 6.0, 7.0]}).to_csv(csv)
    frac = EVChargingEnv(num_vehicles=3, randomize=True, name="ev", vehicle_csv=str(csv), minutes_per_step=2.5)
    frac._num_envs = 2
    frac._draw_roster()
    with pytest.raises(NotImplementedError, match="whole minutes"):
        frac._per_env_rows()
    big = EVChargingEnv(num_vehicles=300, randomize=True, name="ev")
    big._num_envs = 2
    from powergridworld_b200.multiagent_env import SpecBuilder
    with pytest.raises(NotImplementedError, match="256"):
        big._emit(SpecBuilder(0), 0, True)


def _feeder(field, value):
    def mutate(spec):
        setattr(spec.feeder.contents, field, value)
    return mutate


def _branch_load(value):
    def mutate(spec):
        f = spec.feeder.contents
        C.cast(f.branch_load, C.POINTER(C.c_int32 * f.nb)).contents[3] = value
    return mutate


def _short_event_row(spec):
    spec.feeder.contents.nl = spec.dtab_stride // 2     # base loads: 2 + 2 nl doubles of the row


def _staging(spec):
    spec.itab_stride = 40 * 1024                        # event row alone: 160 kB of int32
    for i in range(spec.num_components):
        spec.components[i].itab_off = 0


@pytest.mark.parametrize("make,mutate,msg", [
    (SB.c1_env, _feeder("nb", 129), "feeder dimensions out of range (1..128 load branches)"),
    (SB.c1_env, _branch_load(10 ** 6), "branch load index out of range"),
    (SB.c1_env, _branch_load(-1), "branch load index out of range"),
    (SB.c1_env, _feeder("penalty_node", 10 ** 6), "penalty node out of range"),
    (SB.c1_env, _short_event_row, "event row too short for the feeder base loads"),
    (SB.c1_env, _staging, "scenario tables exceed the shared-memory staging budget"),
], ids=["nb", "branch-load-high", "branch-load-low", "penalty-node", "dtab-stride", "staging"])
def test_feeder_and_staging_checks_come_before_the_device(make, mutate, msg):
    """The checks of the feeder tables and of the shared-memory staging budget run on the host
    before any CUDA call: a malformed spec is PGW_ERR_INVALID with or without a device."""
    env = make(num_envs=4, _dry_run=True)
    rc, got = _create(env, mutate)
    assert (rc, got) == (INVALID, msg)
