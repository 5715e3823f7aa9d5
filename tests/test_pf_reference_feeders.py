"""CPU tier: the float64 power-flow reference (tests/pf_reference.py) on the 123-bus-class feeders
that the tc2 / FP64 kernel tests run on -- truncations to 24 / 50 / 85 loads and the x100
extension -- against the oracle's Y-matrix solve (oracle/powerflow.py), with a roster that puts
several agents on one load, agents on model-2/5 loads and on buses without a load."""
import warnings

import numpy as np
import pytest

from oracle.powerflow import compile_feeder, solve_snapshot
from tests import pf_reference as R
from tests.product_ns import PRODUCT_NS as PNS

# feeder -> (load branches, FP64 rows per env nbp, tc2 tile width NCH or None)
FEEDERS = {24: (24, 32, 4), 50: (50, 64, 8), 85: (85, 96, 11), "x100": (100, 128, None)}


@pytest.fixture(scope="module")
def paths(tmp_path_factory):
    d = tmp_path_factory.mktemp("feeders")
    return {k: R.synthetic_feeder(d, extra=True) if k == "x100" else R.synthetic_feeder(d, k)
            for k in FEEDERS}


def _env(path, E):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")       # agents on loads whose power the reference ignores
        return PNS.MultiAgentEnv(**R.synthetic_config(PNS, path), num_envs=E, _dry_run=True)


@pytest.mark.parametrize("fid", list(FEEDERS))
def test_synthetic_feeder_compiles_to_the_intended_kernel_shapes(paths, fid):
    """nb and the FP64 kernel's padded row count nbp; tc2 takes up to 88 load branches (11 chunks
    of 8), so x100 (nbp = 128, pf_fixed_point_kernel<32, 4, false>) is FP64 only."""
    nb, nbp, nch = FEEDERS[fid]
    env = _env(paths[fid], 1)
    f = env.pf_solver.feeder
    assert (f.nb, f.nl, env._nbp()) == (nb, nb, nbp)
    assert ((f.nb + 7) // 8 <= 11) == (nch is not None)
    if nch is not None:
        assert min(w for w in (2, 4, 8, 11) if w >= (f.nb + 7) // 8) == nch
    assert set(np.asarray(f.branch_model).tolist()) == {1, 2, 5}
    if fid == "x100":
        assert sum(n.startswith("x") for n in f.load_names) == len(R.EXTRA_LOADS)


@pytest.mark.parametrize("fid", list(FEEDERS))
def test_step_powers_and_solve64_match_the_oracle(paths, fid):
    """step_powers against a statement of the rule by load name (agents' real power summed onto
    the model-1 load they name; any other bus adds nothing), then solve64 against the oracle's
    Y-matrix solve of the same loads for two envs: node magnitudes within 1e-8 p.u."""
    E = 2
    env = _env(paths[fid], E)
    f = env.pf_solver.feeder
    rng = np.random.default_rng(7)
    A = len(env.agents)
    p = rng.uniform(-60, 60, size=(A, E))
    t = 100                                    # 08:20, a row of the loadshape past the first
    s = R.step_powers(env, t, p)
    row = env._dtab[t + 1]
    kw = {n: np.full(E, row[2 + k]) for k, n in enumerate(f.load_names)}
    kvar = {n: np.full(E, row[2 + f.nl + k]) for k, n in enumerate(f.load_names)}
    for a, ag in enumerate(env.agents):
        bus = env.agent_name_bus_map[ag.name]
        if bus in kw and f.load_model[f.load_names.index(bus)] == 1:
            kw[bus] = kw[bus] + p[a]
    assert env.agent_name_bus_map["a2"] == "37a" and any(
        env._agent_recs[a].load_slot < 0 for a in range(A))
    want = np.array([(kw[f.load_names[l]] + 1j * kvar[f.load_names[l]]) * f.branch_share[k] * 1e-3
                     for k, l in enumerate(f.branch_load)])
    np.testing.assert_allclose(s, want, rtol=1e-15, atol=0)

    _, _, v = R.solve64(f, s)
    ckt = compile_feeder(paths[fid])
    names = [ld["name"] for ld in ckt.loads]
    idx = [ckt.node_names.index(n) for n in f.node_names]
    for e in range(E):
        vo = solve_snapshot(ckt, [kw[n][e] for n in names], [kvar[n][e] for n in names], tol=1e-12)
        np.testing.assert_allclose(v[:, e], (np.abs(vo) / ckt.vbase)[idx], rtol=0, atol=1e-8,
                                   err_msg=f"env {e}")
    assert v.min() < 0.99                      # the loads did move the profile
