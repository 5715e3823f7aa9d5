"""CPU tier of the table construction (powergridworld_b200/csrc/tables.cpp): the host build of the
module, driven with the specs of dry-run envs, against direct statements of each layout -- the CTA
list against walk_plan, the FP64 blob against the feeder arrays, the FP16 operand images and the
fused kernel's mma.sync fragments against the split models of test_fp16_split_model.py /
test_mma_fixed_point_model.py, and the agent / branch maps."""
import ctypes as C
import os
import subprocess
import warnings

import numpy as np
import pytest

from powergridworld_b200 import _native as N
from powergridworld_b200.scenarios import bench as SB
from tests import pf_reference as R
from tests.product_ns import PRODUCT_NS as PNS
from tests.test_component_walk import walk_plan
from tests.test_fused_step_reference import _config as ieee13_config
from tests.test_mma_fixed_point_model import _interleaved, _scale_for, _split16

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "powergridworld_b200", "csrc")


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("host_tables") / "libhost_tables.so")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")      # cuda_fp16.h and the vector types
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", f"-I{cuda}/include", "-o", so,
                           os.path.join(CSRC, "tables.cpp"), os.path.join(HERE, "host_tables_shim.cpp")])
    lib = C.CDLL(so)
    lib.ht_build.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.ht_error.restype = C.c_char_p
    lib.ht_table.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
    lib.ht_table.restype = C.c_long
    lib.ht_value.argtypes = [C.c_char_p]
    lib.ht_value.restype = C.c_double
    return lib


def _quiet(make):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")         # agents on loads whose power the reference ignores
        return make()


@pytest.fixture(scope="module")
def feeders(tmp_path_factory):
    d = tmp_path_factory.mktemp("feeders")
    out = {f"s{n}": R.synthetic_feeder(d, n) for n in (24, 50, 85)}
    out["x100"] = R.synthetic_feeder(d, extra=True)
    out.update({fid: R.feeder_file(fid, d) for fid in R.VARIANTS})
    return out


SCENARIOS = {
    "c1": lambda fd: SB.c1_env(num_envs=300, _dry_run=True),
    "c2": lambda fd: SB.c2_env(num_envs=300, _dry_run=True),
    "c3": lambda fd: SB.c3_env(num_envs=300, _dry_run=True),
    "hs": lambda fd: SB.hs_env(num_envs=300, _dry_run=True),
    **{fid: (lambda fd, fid=fid: _quiet(lambda: PNS.MultiAgentEnv(
        **ieee13_config(PNS, fd[fid], fid, False), num_envs=64, _dry_run=True))) for fid in R.VARIANTS},
    "o16_hook": lambda fd: _quiet(lambda: PNS.CoordinatedMultiBuildingControlEnv(
        **ieee13_config(PNS, fd["o16"], "o16", True), num_envs=64, _dry_run=True)),
    **{fid: (lambda fd, fid=fid: _quiet(lambda: PNS.MultiAgentEnv(
        **R.synthetic_config(PNS, fd[fid]), num_envs=64, _dry_run=True))) for fid in ("s24", "s50", "s85", "x100")},
}


FEEDER_CASES = [n for n in SCENARIOS if n not in ("c2", "hs")]      # C2 and HS run without a feeder


def _tc2_nch(nb):
    return next((c for c in (2, 4, 8, 11) if c >= (nb + 7) // 8), 0)


class Tables:
    def __init__(self, lib, env, budget=148 * 16):
        self.env = env
        self.spec, self._keep = env._build_spec()
        f = self.spec.feeder.contents if self.spec.feeder else None
        rc = lib.ht_build(C.addressof(self.spec), budget, _tc2_nch(f.nb) if f else 0)
        assert rc == 0, lib.ht_error().decode()
        self.lib, self.f = lib, f

    def table(self, name):
        p = C.c_void_p()
        n = self.lib.ht_table(name.encode(), C.byref(p))
        return np.frombuffer(C.string_at(p, n), dtype=np.uint8) if n else np.zeros(0, np.uint8)

    def __getitem__(self, name):
        v = self.lib.ht_value(name.encode())
        assert not np.isnan(v), name
        return int(v) if float(v).is_integer() and "scale" not in name else v

    def feeder(self, name, n, dtype=np.float64):
        return np.ctypeslib.as_array(getattr(self.f, name), shape=(n,)).astype(dtype)

    def cplx(self, name, *shape):
        a = self.feeder(name, 2 * int(np.prod(shape)))
        return (a[0::2] + 1j * a[1::2]).reshape(shape)

    def agents(self):
        s = self.spec
        return np.array([(s.agents[a].load_slot, s.agents[a].bus_node) for a in range(s.num_agents)]).reshape(-1, 2)


def _at(blob, off, dtype, n):
    return np.frombuffer(blob[off:off + np.dtype(dtype).itemsize * n].tobytes(), dtype=dtype)


def _weights(env):
    w = []
    for ag in env._agent_recs:
        x = 0.5
        for c in env._b.comps[ag.comp_begin:ag.comp_end]:
            x += (1.0 + 0.04 * env._b.ipar[c.ipar_off]) if c.type in (N.EV, N.HS_EV) else \
                {N.BUILDING: 2.0, N.STORAGE: 0.8, N.HS_BEGIN: 1.0, N.HS_STORAGE: 1.0, N.HS_DEVICES: 1.0}.get(c.type, 0.5)
        w.append(x)
    return w


@pytest.mark.parametrize("budget", [1, 7, 1480, 2368])
@pytest.mark.parametrize("name", ["c1", "c2", "c3", "hs"])
def test_cta_list_follows_the_walk_plan(lib, feeders, name, budget):
    env = SCENARIOS[name](feeders)
    t = Tables(lib, env, budget)
    work = _at(t.table("work"), 0, np.int32, t["c.num_ctas"] * 12).reshape(-1, 12)
    assert t["c.tickets"] == len(work)
    n = walk_plan(env, budget)
    agents = [a for i, a in enumerate(work[:, 0]) if i == 0 or work[i - 1, 0] != a]
    assert sorted(agents) == list(range(len(n)))                   # each agent's CTAs in one run
    w = _weights(env)
    assert agents == sorted(range(len(n)), key=lambda a: -w[a])    # heaviest first, stable
    s = t.spec
    dstart = sorted([s.components[c].dpar_off for c in range(s.num_components)] + [s.dpar_len])
    istart = sorted([s.components[c].ipar_off for c in range(s.num_components)] + [s.ipar_len])
    for a in agents:
        rows = work[work[:, 0] == a]
        assert len(rows) == n[a] and list(rows[:, 1]) == list(range(n[a])) and set(rows[:, 2]) == {n[a]}
        c_lo, c_n, d_lo, d_n, i_lo, i_n = rows[0, 4:10]
        assert (c_lo, c_lo + c_n) == (s.agents[a].comp_begin, s.agents[a].comp_end)
        assert d_lo % 2 == d_n % 2 == i_lo % 4 == i_n % 4 == 0
        for c in range(c_lo, c_lo + c_n):
            k = s.components[c]
            if k.dpar_off < s.dpar_len:
                end = next(x for x in dstart if x > k.dpar_off)
                assert d_lo <= k.dpar_off and end <= d_lo + d_n
            if k.ipar_off < s.ipar_len:
                end = next(x for x in istart if x > k.ipar_off)
                assert i_lo <= k.ipar_off and end <= i_lo + i_n
    assert t["c.max_cn"] == work[:, 5].max() and t["c.max_dn"] == work[:, 7].max()
    blob = t.table("comp")
    assert t["c.blob_bytes"] == len(blob) and len(blob) % 16 == 0
    np.testing.assert_array_equal(_at(blob, t["c.off_dpar"], np.float64, s.dpar_len), env._b.dpar)


@pytest.mark.parametrize("name", FEEDER_CASES)
def test_fp64_blob_decodes_to_the_feeder(lib, feeders, name):
    t = Tables(lib, SCENARIOS[name](feeders))
    nb, nn, nbp, nnp, A = t["f.nb"], t["f.nn"], t["f.nbp"], t["f.nnp"], t.spec.num_agents
    assert nbp == (16 if nb <= 16 else -(-nb // 32) * 32) and nnp == nn + nn % 2
    blob = t.table("pf")
    assert t["f.blob_bytes"] == len(blob) and t["f.stage_blob"] == (len(blob) <= 96 * 1024)
    c128 = lambda off, n: (lambda a: a[0::2] + 1j * a[1::2])(_at(blob, off, np.float64, 2 * n))
    zbbT = c128(0, nb * nbp).reshape(nb, nbp)
    np.testing.assert_array_equal(zbbT[:, :nb], t.cplx("zbb", nb, nb).T)
    assert not zbbT[:, nb:].any()
    u0 = c128(t["f.off_u0"], nbp)
    np.testing.assert_array_equal(u0[:nb], t.cplx("u0", nb))
    assert (u0[nb:] == 1).all()
    znbT = c128(t["f.off_znbT"], nb * nnp).reshape(nb, nnp)
    np.testing.assert_array_equal(znbT[:, :nn], t.cplx("znb", nn, nb).T)
    np.testing.assert_array_equal(c128(t["f.off_w"], nnp)[:nn], t.cplx("w", nn))
    pad = lambda a, v: np.concatenate([a, np.full(nbp - nb, v, a.dtype)])
    for off, field, fill, dt in (("f.off_share", "branch_share", 0.0, np.float64),
                                 ("f.off_vmin", "vminpu", 0.95, np.float64), ("f.off_vmax", "vmaxpu", 1.05, np.float64),
                                 ("f.off_bload", "branch_load", 0, np.int32), ("f.off_bmodel", "branch_model", 1, np.int32)):
        np.testing.assert_array_equal(_at(blob, t[off], dt, nbp), pad(t.feeder(field, nb, dt), fill))
    np.testing.assert_array_equal(_at(blob, t["f.off_slot"], np.int32, A), t.agents()[:, 0])
    np.testing.assert_array_equal(_at(blob, t["f.off_node"], np.int32, A), t.agents()[:, 1])


def _wye_nodes(t):
    """Node -> branch of every wye load (row n of Znb = c row k of Zbb, w[n] = c u0[k]), first match."""
    zbb, znb, u0, w = t.cplx("zbb", t["f.nb"], t["f.nb"]), t.cplx("znb", t["f.nn"], t["f.nb"]), t.cplx("u0", t["f.nb"]), \
        t.cplx("w", t["f.nn"])
    dnode, taken = {}, set()
    for n in range(t["f.nn"]):
        for k in range(t["f.nb"]):
            den = u0[k].real ** 2 + u0[k].imag ** 2
            if k in taken or den <= 0 or not (c := (w[n] * np.conj(u0[k])).real / den) > 0:
                continue
            err = max(abs(w[n] - c * u0[k]), np.abs(znb[n] - c * zbb[k]).max())
            if err <= 1e-10 * max(abs(w[n]), np.abs(znb[n]).max()):
                dnode[k] = n
                taken.add(k)
                break
    return dnode


def _image(blob, off, N):
    """An N x N FP16 UMMA image (K-major, no swizzle) as the matrix it holds."""
    r, k = np.meshgrid(np.arange(N), np.arange(N), indexing="ij")
    idx = (r // 8) * (N // 8) * 128 + (k // 8) * 128 + (r % 8) * 16 + (k % 8) * 2
    return _at(blob, off, np.float16, N * N)[idx // 2].astype(np.float64)


@pytest.mark.parametrize("name", [n for n in FEEDER_CASES if n != "x100"])   # x100: beyond tc2
def test_tc2_images_and_maps(lib, feeders, name):
    t = Tables(lib, SCENARIOS[name](feeders))
    nb, nn, A = t["f.nb"], t["f.nn"], t.spec.num_agents
    nch = t["t.nch"]
    N, NBP = 16 * nch, 8 * nch
    blob = t.table("tc2")
    zbb, znb = t.cplx("zbb", nb, nb), t.cplx("znb", nn, nb)
    dnode = _wye_nodes(t)
    if name in ("c1", "c3"):
        assert len(dnode) == {"c1": 11, "c3": 85}[name]
    xnode = [n for n in range(nn) if n not in dnode.values()]
    assert t["t.nx"] == len(xnode) and t["t.ncc"] == -(-len(xnode) // NBP)
    sb1, sb2 = _scale_for(zbb.view(np.float64)), _scale_for(znb.view(np.float64))
    assert t["t.descale1"] == np.float32(1 / (sb1 * 2048)) and t["t.descale2"] == np.float32(1 / (sb2 * 2048))
    pos = lambda item, im: 16 * (item // 8) + item % 8 + 8 * im
    part = t["t.part_bytes"]

    def check(off, z):                         # rows: the items of z, columns: the branch currents
        want_hi, want_lo = _split16(np.block([[-z.real, z.imag], [-z.imag, -z.real]]) * (sb1 if z is zbb else sb2))
        rows = [pos(i, 0) for i in range(len(z))] + [pos(i, 1) for i in range(len(z))]
        cols = [pos(k, 0) for k in range(nb)] + [pos(k, 1) for k in range(nb)]
        for img, want in ((_image(blob, off, N), want_hi), (_image(blob, off + part, N), want_lo)):
            np.testing.assert_array_equal(img[np.ix_(rows, cols)], want)
            assert np.count_nonzero(img) == np.count_nonzero(want)
    check(0, zbb)
    for cc in range(t["t.ncc"]):
        check(t["t.off_zn"] + cc * 2 * part, znb[xnode[cc * NBP:(cc + 1) * NBP]])
    tab = lambda key, n: _at(blob, t["t.off_tab"] + t[key], np.int32, n)
    slot, node = t.agents()[:, 0], t.agents()[:, 1]
    nl = t["f.nl"]
    lptr = np.concatenate([[0], np.cumsum(np.bincount(slot[slot >= 0], minlength=nl))])
    np.testing.assert_array_equal(tab("t.t_lptr", nl + 1), lptr)
    np.testing.assert_array_equal(tab("t.t_lidx", A)[:lptr[-1]], np.argsort(np.where(slot >= 0, slot, nl), kind="stable")[:lptr[-1]])
    bl = t.feeder("branch_load", nb, np.int32)
    on = [np.flatnonzero(slot == bl[k]) for k in range(nb)]
    np.testing.assert_array_equal(tab("t.t_bagent", nb), [-1 if len(a) == 0 else (a[0] if len(a) == 1 else -2) for a in on])
    np.testing.assert_array_equal(tab("t.t_dnode", NBP), [dnode.get(k, -1) for k in range(NBP)])
    branch_of = {n: k for k, n in dnode.items()}
    vag, vtail = -np.ones((NBP, 2), np.int32), []
    for a in range(A):
        k = branch_of.get(node[a], -1)
        free = np.flatnonzero(vag[k] < 0) if k >= 0 else []
        if len(free):
            vag[k, free[0]] = a
        else:
            vtail.append(a)
    np.testing.assert_array_equal(tab("t.t_vag", 2 * NBP).reshape(NBP, 2), vag)
    assert t["t.ntail"] == len(vtail)
    np.testing.assert_array_equal(tab("t.t_vtail", len(vtail)), vtail)
    assert t["t.polish_ok"] == (nch == 2)
    if not t["t.polish_ok"]:
        assert t["t.ftab_bytes"] == 0
        return
    punit, pen = t["f.punit"], t["f.penalty_node"]
    ftab = lambda key, dt, n: _at(blob, t["t.off_ftab"] + t[key], dt, n)
    np.testing.assert_array_equal(ftab("t.f_aslot", np.int32, A), [branch_of.get(n, -1) for n in node])
    assert t["t.pen_slot"] == (branch_of.get(pen, -1) if punit else -1)
    rows = {branch_of[n] for n in node if n in branch_of} | ({branch_of[pen]} if punit and pen in branch_of else set())
    tc2p = t.table("tc2p")
    rows_off = 16 * 16 * (16 + 8) + 16 * 16 + 4 * 16 * 8 + 16 * 4     # Tc2Polish.rows: behind zT .. model
    assert int(_at(tc2p, rows_off, np.uint32, 1)[0]) == sum(1 << k for k in rows)
    assert t["t.polish_row"] == (pen if punit and pen not in branch_of else -1)
    np.testing.assert_array_equal(ftab("t.f_kp", np.uint8, len(tc2p)), tc2p)
    # fused f_xz: [n-tile][lane][k-step][hi b0, hi b1, lo b0, lo b1] of the interleaved operators
    frags = ftab("t.f_xz", np.float16, (4 + 4 * t["t.ncc"]) * 32 * 16).astype(np.float64).reshape(-1, 32, 2, 2, 2, 2)
    j, lane, st, hl, reg, ii = np.indices(frags.shape)
    g, tq = lane >> 2, lane & 3
    r, q = 4 * j + g // 2, 8 * st + tq + 4 * reg
    for lo_tile, z, sb in [(0, zbb, sb1)] + [(4 + 4 * cc, znb[xnode[16 * cc:16 * cc + 16]], sb2)
                                             for cc in range(t["t.ncc"])]:
        m = np.zeros((32, 32))
        m[:2 * len(z), :2 * nb] = _interleaved(z) * sb
        hi, lo = _split16(m)
        sel = (j >= lo_tile) & (j < lo_tile + 4)
        rr, qq = 2 * (r[sel] - 4 * lo_tile) + (g[sel] & 1), 2 * q[sel] + ii[sel]
        np.testing.assert_array_equal(frags[sel], np.where(hl[sel] == 0, hi[rr, qq], lo[rr, qq]))
