"""CPU model of the power flow of the fused step kernel (csrc/step_fused.cu) on mma.sync: the
fixed point u <- u0 - Zbb i(u), its float32 pre-sweep and the expansion v = w - Znb i as row
products of split-FP16 operands, in the arrangement the kernel uses -- currents x xscale split into
FP16 hi / lo, the realified Zbb x sb1 and Znb x sb2 split the same way, (Re, Im) interleaved per
branch along K and per output along N, hi.hi + hi.lo + lo.hi accumulated in FP32 -- with per-env
convergence on max |d drop| and frozen currents.  Checked against the float64 solve on the shipped
IEEE-13 feeder and the variants of tests/pf_reference.py (model-2/5 loads, 14, 15, 16 branches)."""
import numpy as np
import pytest

from powergridworld_b200.distribution_system.feeder import compile_feeder
from tests.pf_reference import FEEDERS, band, feeder_file, solve64

XS = 2048.0
F32 = np.float32


@pytest.fixture(scope="module", params=FEEDERS)
def feeder(request, tmp_path_factory):
    return compile_feeder(feeder_file(request.param, tmp_path_factory.mktemp("feeder")))


def _scale_for(m):
    """tables.cpp scale_for: the power of two that takes the largest entry into [8192, 16384)."""
    return 2.0 ** np.floor(np.log2(16384.0 / np.abs(m).max()))


def _interleaved(z):
    """The realified operator with (Re, Im) interleaved: M[2r + io, 2q + ii], rows = outputs."""
    m = np.zeros((2 * z.shape[0], 2 * z.shape[1]))
    m[0::2, 0::2], m[0::2, 1::2] = -z.real, z.imag
    m[1::2, 0::2], m[1::2, 1::2] = -z.imag, -z.real
    return m


def _split16(a):
    """images(): hi = fp16(a), lo = fp16(a - hi), both as float64 values."""
    hi = a.astype(F32).astype(np.float16)
    lo = (a - hi.astype(np.float64)).astype(F32).astype(np.float16)
    return hi.astype(np.float64), lo.astype(np.float64)


def _product(xh, xl, bh, bl):
    """Three products of FP16 operands with FP32 accumulation, the small terms first."""
    acc = (xl @ bh.T).astype(F32)
    acc = (acc + (xh @ bl.T).astype(F32)).astype(F32)
    return (acc + (xh @ bh.T).astype(F32)).astype(F32)


def _current(f, dn, ds1, sr, si):
    """t2_current on every branch of every env: scaled currents, interleaved (Re, Im), from the
    scaled drops dn [envs, 2 nb]."""
    lo, hi, m5 = band(f)
    ur = (dn[:, 0::2].astype(np.float64) * ds1 + f.u0.real.astype(F32)).astype(F32)
    ui = (dn[:, 1::2].astype(np.float64) * ds1 + f.u0.imag.astype(F32)).astype(F32)
    m2 = (ur.astype(np.float64) * ur + (ui * ui).astype(F32)).astype(F32)
    cl = np.minimum(np.maximum(m2, lo.astype(F32)), hi.astype(F32)).astype(np.float64)
    kf = np.where(m5, 1.0 / np.sqrt(cl), 1.0 / cl).astype(F32)
    tr, ti = (ur * kf).astype(F32), (ui * kf).astype(F32)
    x = np.empty_like(dn)
    x[:, 0::2] = (sr.astype(np.float64) * tr + (si * ti).astype(F32)).astype(F32)
    x[:, 1::2] = (sr.astype(np.float64) * ti - (si * tr).astype(F32)).astype(F32)
    return x


def _mma_solve(f, load_scales, tol, max_iter=60):
    """The kernel's power flow for a batch of envs (one load scale each)."""
    p = (f.load_kw + 1j * f.load_kvar)[f.branch_load][None, :] * np.asarray(load_scales)[:, None]
    sh = (f.branch_share * 1e-3).astype(F32) * F32(XS)
    sr, si = (p.real.astype(F32) * sh).astype(F32), (p.imag.astype(F32) * sh).astype(F32)
    sb1, sb2 = _scale_for(np.abs(np.stack([f.zbb.real, f.zbb.imag]))), \
        _scale_for(np.abs(np.stack([f.znb.real, f.znb.imag])))
    ds1, ds2 = 1.0 / (sb1 * XS), 1.0 / (sb2 * XS)
    bh, bl = _split16(_interleaved(f.zbb) * sb1)
    tol_s = F32(tol) / F32(ds1)
    n_env = len(load_scales)
    dp = np.zeros((n_env, 2 * f.nb), F32)
    x = _current(f, dp, ds1, sr, si)
    conv = np.zeros(n_env, bool)
    iters = np.zeros(n_env, int)
    it = 0
    while not conv.all():
        it += 1
        xh, xl = _split16(x.astype(np.float64))
        dn = _product(xh, xl, bh, bl)                  # drop / descale1
        dd = np.abs(dn - dp).max(axis=1)
        xn = _current(f, dn, ds1, sr, si)
        x = np.where(conv[:, None], x, xn)             # converged envs keep their currents
        dp = dn
        live = ~conv
        iters[live] = it
        conv = conv | (dd < tol_s) | (it >= max_iter)
    u_loop = f.u0 + (dp[:, 0::2] + 1j * dp[:, 1::2]).astype(np.complex128) * ds1
    # pre-sweep: once more from the last drop (the kernel's correctly rounded reciprocals)
    xh, xl = _split16(_current(f, dp, ds1, sr, si).astype(np.float64))
    pr = _product(xh, xl, bh, bl)
    u_pre = f.u0 + (pr[:, 0::2] + 1j * pr[:, 1::2]).astype(np.complex128) * ds1
    # expansion from the loop's final currents: - Znb i summed from zero, w added once
    nh, nl = _split16(_interleaved(f.znb) * sb2)
    xh, xl = _split16(x.astype(np.float64))
    dv = (_product(xh, xl, nh, nl) * F32(ds2)).astype(F32)
    vr = (f.w.real.astype(F32) + dv[:, 0::2]).astype(F32)
    vi = (f.w.imag.astype(F32) + dv[:, 1::2]).astype(F32)
    m2 = (vr.astype(np.float64) * vr + (vi * vi).astype(F32)).astype(F32)
    return iters, u_loop, u_pre, np.sqrt(m2.astype(np.float64))


def test_interleaved_images_reorder_the_realified_operators(feeder):
    """The interleaved B images are a permutation of the block-realified Zbb / Znb of the tc2
    kernel: output (r, Re/Im) and input (q, Re/Im) at 2r + io, 2q + ii instead of io n + r."""
    for z in (feeder.zbb, feeder.znb):
        block = np.block([[-z.real, z.imag], [-z.imag, -z.real]])
        rows, cols = z.shape
        po = np.array([io * rows + r for r in range(rows) for io in (0, 1)])
        pi = np.array([ii * cols + q for q in range(cols) for ii in (0, 1)])
        np.testing.assert_array_equal(_interleaved(z), block[np.ix_(po, pi)])
        assert sorted(po) == list(range(2 * rows)) and sorted(pi) == list(range(2 * cols))


@pytest.mark.parametrize("tol", [1e-6, 1e-7])
def test_split_fp16_fixed_point_reaches_the_float64_solution(feeder, tol):
    f = feeder
    scales = np.array([0.3, 1.0, 1.6])
    iters, u_loop, u_pre, vmag = _mma_solve(f, scales, tol)
    assert iters.max() < 60, "the fixed point did not converge"
    for k, ls in enumerate(scales):
        u_ref, i_ref, v_ref = solve64(f, ((f.load_kw + 1j * f.load_kvar)[f.branch_load] * ls
                                          * f.branch_share * 1e-3)[:, None])
        err_loop = np.abs(u_loop[k] - u_ref[:, 0]).max()
        err_pre = np.abs(u_pre[k] - u_ref[:, 0]).max()
        err_v = np.abs(vmag[k] - v_ref[:, 0]).max()
        assert err_loop < 3e-7, f"fixed point {err_loop:.2e} p.u. after {iters[k]} iterations"
        assert err_pre < 1e-7, f"pre-sweep {err_pre:.2e} p.u."
        assert err_v < 5e-7, f"node magnitudes {err_v:.2e} p.u."


def test_the_correction_products_carry_the_accuracy(feeder):
    """hi.hi alone is off by orders of magnitude more than the three-product sum."""
    f = feeder
    sb1 = _scale_for(np.abs(np.stack([f.zbb.real, f.zbb.imag])))
    u, i, _ = solve64(f, ((f.load_kw + 1j * f.load_kvar)[f.branch_load] * f.branch_share * 1e-3)[:, None])
    x = np.empty((1, 2 * f.nb))
    x[0, 0::2], x[0, 1::2] = i[:, 0].real * XS, i[:, 0].imag * XS
    bh, bl = _split16(_interleaved(f.zbb) * sb1)
    xh, xl = _split16(x.astype(F32).astype(np.float64))
    exact = x.astype(F32).astype(np.float64) @ _interleaved(f.zbb).T * sb1
    three = np.abs(_product(xh, xl, bh, bl) - exact).max()
    single = np.abs(xh @ bh.T - exact).max()
    assert single > 10 * three
