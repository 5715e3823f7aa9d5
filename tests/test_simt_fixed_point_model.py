"""CPU model of the float32 power flow of the fused step kernel (csrc/step_fused.cu): the fixed
point u <- u0 - Zbb i(u) with one branch per thread, currents scaled by xscale, the drop as two
FFMA chains against Zbb^T / xscale, per-env convergence on max |d drop| with frozen currents,
the float32 pre-sweep of the polish, and the expansion v = w - Znb i against Znb^T / xscale.
Checks the accuracy claims of DESIGN.md 4.3d against a float64 solve, on the shipped IEEE-13 feeder
and on the variants of the published one in tests/pf_reference.py (model-2/5 loads, 14, 15 and 16
load branches)."""
import numpy as np
import pytest

from powergridworld_b200.distribution_system.feeder import compile_feeder
from tests.pf_reference import FEEDERS, band, feeder_file, solve64

XS = 2048.0
F32 = np.float32


def _fma(a, b, c):
    """float32 fmaf: the float64 product of two float32 values is exact."""
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(F32)


@pytest.fixture(scope="module", params=FEEDERS)
def feeder(request, tmp_path_factory):
    return compile_feeder(feeder_file(request.param, tmp_path_factory.mktemp("feeder")))


def _powers(f, load_scale):
    return (f.load_kw + 1j * f.load_kvar)[f.branch_load] * load_scale


def _solve64(f, load_scale):
    """float64 fixed point: branch voltages and currents (p.u.)."""
    u, i, _ = solve64(f, _powers(f, load_scale) * f.branch_share * 1e-3)
    return u[:, 0], i[:, 0]


def _current32(f, d_re, d_im, sr, si):
    """t2_current32 on every branch: scaled currents of the drop (d_re, d_im) in float32."""
    lo, hi, m5 = band(f)
    ur = (f.u0.real.astype(F32) + d_re).astype(F32)
    ui = (f.u0.imag.astype(F32) + d_im).astype(F32)
    m2 = _fma(ur, ur, (ui * ui).astype(F32))
    cl = np.minimum(np.maximum(m2, lo.astype(F32)), hi.astype(F32))
    kf = np.where(m5, (1.0 / np.sqrt(cl.astype(np.float64))), 1.0 / cl.astype(np.float64)).astype(F32)
    tr, ti = (ur * kf).astype(F32), (ui * kf).astype(F32)
    x = _fma(sr, tr, (si * ti).astype(F32))
    y = _fma(sr, ti, (-(si * tr)).astype(F32))
    return x, y


def _zdot(acc_re, acc_im, z, x, y):
    """acc - sum_k z[:, k] (x_k + j y_k) as the kernel's zdot: two chains of t2_cmac_sub32
    (even / odd k), summed at the end; z = Z / xscale in float32, rows = outputs."""
    zr, zi = z.real.astype(F32), z.imag.astype(F32)
    a = [[acc_re.astype(F32), acc_im.astype(F32)],
         [np.zeros_like(acc_re, dtype=F32), np.zeros_like(acc_im, dtype=F32)]]
    for k in range(z.shape[1]):
        ch = a[k & 1]
        ch[0] = _fma(-zr[:, k], np.full(len(zr), x[k], F32), ch[0])
        ch[0] = _fma(zi[:, k], np.full(len(zr), y[k], F32), ch[0])
        ch[1] = _fma(-zr[:, k], np.full(len(zr), y[k], F32), ch[1])
        ch[1] = _fma(-zi[:, k], np.full(len(zr), x[k], F32), ch[1])
    return (a[0][0] + a[1][0]).astype(F32), (a[0][1] + a[1][1]).astype(F32)


def _simt_solve(f, load_scale, tol, max_iter=60):
    """The kernel's power flow for one env: fixed point, pre-sweep, expansion."""
    p = _powers(f, load_scale)
    sh = (f.branch_share * 1e-3).astype(F32) * F32(XS)
    sr, si = (p.real.astype(F32) * sh).astype(F32), (p.imag.astype(F32) * sh).astype(F32)
    z32 = f.zbb / XS
    dr = np.zeros(f.nb, F32)
    di = np.zeros(f.nb, F32)
    x, y = _current32(f, dr, di, sr, si)
    it = 0
    while True:
        it += 1
        nr, ni = _zdot(np.zeros(f.nb, F32), np.zeros(f.nb, F32), z32, x, y)
        dd = max(np.abs(nr - dr).max(), np.abs(ni - di).max())
        x, y = _current32(f, nr, ni, sr, si)
        dr, di = nr, ni
        if dd < tol or it >= max_iter:
            break
    u_loop = f.u0 + (dr.astype(np.float64) + 1j * di.astype(np.float64))
    # the polish's float32 pre-sweep: the iteration once more, from the last drop
    xp, yp = _current32(f, dr, di, sr, si)
    pr, pi = _zdot(np.zeros(f.nb, F32), np.zeros(f.nb, F32), z32, xp, yp)
    u_pre = f.u0 + (pr.astype(np.float64) + 1j * pi.astype(np.float64))
    # expansion from the loop's final currents
    dvr, dvi = _zdot(np.zeros(f.nn, F32), np.zeros(f.nn, F32), f.znb / XS, x, y)
    vr, vi = (f.w.real.astype(F32) + dvr).astype(F32), (f.w.imag.astype(F32) + dvi).astype(F32)
    m2 = _fma(vr, vr, (vi * vi).astype(F32))
    vmag = np.sqrt(m2.astype(np.float64)).astype(F32).astype(np.float64)
    return it, u_loop, u_pre, vmag


@pytest.mark.parametrize("tol", [1e-6, 1e-7])
@pytest.mark.parametrize("load_scale", [0.3, 1.0, 1.6])
def test_float32_fixed_point_reaches_the_float64_solution(feeder, tol, load_scale):
    f = feeder
    u_ref, _ = _solve64(f, load_scale)
    it, u_loop, u_pre, _ = _simt_solve(f, load_scale, tol)
    assert it < 60, "the float32 fixed point did not converge"
    err_loop = np.abs(u_loop - u_ref).max()
    err_pre = np.abs(u_pre - u_ref).max()
    assert err_loop < 3e-7, f"fixed point {err_loop:.2e} p.u. after {it} iterations"
    assert err_pre < 1e-7, f"pre-sweep {err_pre:.2e} p.u."


@pytest.mark.parametrize("load_scale", [0.3, 1.0, 1.6])
def test_expansion_node_magnitudes_within_1e6(feeder, load_scale):
    f = feeder
    _, i_ref = _solve64(f, load_scale)
    v_ref = np.abs(f.w - f.znb @ i_ref)
    _, _, _, vmag = _simt_solve(f, load_scale, 1e-6)
    err = np.abs(vmag - v_ref).max()
    assert err < 1e-6, f"node magnitudes {err:.2e} p.u."
