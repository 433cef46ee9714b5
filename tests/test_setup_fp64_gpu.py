"""The set-up, per-pixel and atom kernels, run once each through the C ABI test hook (fdes_b200_sweep_test, ops
SCATTER_TABLE .. RECORDS) and compared with the float64 models of setup_models.py and with the oracle's float32
restatements, always with rectangular pixels (d1 / d2 = 2.1, as qsctilt64) so that a swapped kx / ky or x / y axis
shows; one d1 == d2 case pins the shipped configuration.  The end-to-end tests at the bottom run modes 0, 1 and 2
with rectangular pixels and a rectangular image inside the square sample against orc.build_measurements.

Setting FDES_SETUP_ERRORS=<file.json> records the errors of a run per table and size (the bounds below were set
from such a run).
"""
import json
import os

import numpy as np
import pytest

import setup_models as mdl
from conftest import TOL_INTENSITY, TOL_WAVE, rel_l2

pytestmark = pytest.mark.gpu

SIZES = [64, 128, 256, 512, 1024, 2048, 4096, 320, 800, 1000, 96, 250, 600, 1022, 143]   # test_sweeps_fp64_gpu.py
TABLE_SIZES = SIZES + [8, 9, 8192]
PIXEL_SIZES = SIZES + [8, 9]
BIG = 8192                           # per-pixel kernels: one flag / dn pair / table mode there (67 M pixels)
D1, D2 = 2.1e-11, 1.0e-11            # rectangular pixels
LAM = 2.507934e-12
EPS = mdl.EPS32

# Bounds, in units of float32 eps, about three times the largest error over all sizes measured on an NVIDIA B200
# (1000 W power limit, 1965 MHz); the run of this file there took 2.3 min.  Also measured there:
# no entry of the 2/3 mask differs from the exact integer test at any size (at 4096 and 8192 the sums near the edge
# are still below 2^24), no aperture point depends on how nu1^2 + nu2^2 is fused, one Anscombe count flips.
# "x32": against the oracle's float32 restatement.  name: (largest measured, at size) -> bound
MEASURED = {
    "scatter": (4.8, 4096), "scatter32": (6.0, 4096),
    "prop": (1.5, 600), "prop32": (1.2, 1000),
    "lens": (3.3, 1000), "lens32": (4.0, 8192),
    "detector": (2.3, 8192), "detector32": (2.5, 8192),
    "tilt": (1.7, 8192), "tilt32": (1.3, 8192),
    "tukey": (1.1, 143), "tukey32": (0.33, 1000),
    "area": (1.8, 2048), "area32": (1.5, 4096),
}
BOUND = {
    "scatter": 15, "scatter32": 18,      # relative error
    "prop": 5, "prop32": 4,              # |err| / (|ref| (1 + |phase|))
    "lens": 10, "lens32": 11,            # |err| / (scale (1 + the magnitude of chi's terms))
    "detector": 7, "detector32": 8,      # relative error / (1 + exponent)
    "tilt": 5, "tilt32": 4,              # |err| / (|psi| (1 + the magnitude of the phase's terms))
    "tukey": 4, "tukey32": 1,            # |err| / (|psi| (1 + N / dn1 + N / dn2))
    "area": 6, "area32": 5,              # |err| / (1 + |psi|)
}
# the jitter's normals differ from the oracle's float32 Box-Muller by at most 1.2e-6 (1 + |x|) (the device's logf and
# __sincosf); bound 4e-6
_ERRORS = {}


@pytest.fixture(scope="module", autouse=True)
def _record_errors():
    yield
    path = os.environ.get("FDES_SETUP_ERRORS")
    if path:
        with open(path, "w") as f:
            json.dump(_ERRORS, f, indent=1, sort_keys=True)


def check(name, n, err):
    """err: per-entry error in units of float32 eps."""
    e = float(np.max(err)) if np.size(err) else 0.0
    d = _ERRORS.setdefault(name, {})
    d[str(n)] = max(e, d.get(str(n), 0.0))
    assert np.isfinite(e) and e <= BOUND[name], f"{name} {n}: {e:.2f} eps"


def run(fb, op, n, bufs, iargs=(), fargs=()):
    cp = [np.ascontiguousarray(b).copy() for b in bufs]
    fb.sweep_test(op, n, 1, cp, iargs, fargs)
    return cp


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint32), np.ascontiguousarray(b).view(np.uint32))


def crand(rng, shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)


# ---------------------------------------------------------------------------------------------------
# quarter tables
# ---------------------------------------------------------------------------------------------------
def scatter(fb, n, Z, d1, d2, sigma=7288400.5):
    q = n // 2 + 1
    return run(fb, fb.SCATTER_TABLE, n, [np.full(q * q, np.nan, np.float32)], [Z], [d1, d2, sigma])[0]


@pytest.mark.parametrize("n", TABLE_SIZES)
def test_scattering_table(n, fb):
    zs = list(range(1, 104)) + [0, 104, 200] if n in (8, 9, 64, 143) else [1, 6, 14, 79, 103, 0]
    for Z in zs:
        got = scatter(fb, n, Z, D1, D2).astype(np.float64)
        ref = mdl.scatter_q64(Z, n, D1, D2, 7288400.5)
        check("scatter", n, np.abs(got - ref) / np.abs(ref) / EPS)
        r32 = mdl.scatter_q32(Z, n, D1, D2, 7288400.5).astype(np.float64)
        check("scatter32", n, np.abs(got - r32) / np.abs(r32) / EPS)
    # the fallback row: f = 3 for every q
    np.testing.assert_array_equal(scatter(fb, n, 0, D1, D2), scatter(fb, n, 200, D1, D2))
    # the quarter table is what the sweeps read through quarter_to_full: entry (ky, kx) of the full grid
    import sweep_model as sm
    full = sm.quarter_to_full(scatter(fb, n, 79, D1, D2), n)
    ref = mdl.scatter_q64(79, n, D1, D2, 7288400.5).reshape(n // 2 + 1, n // 2 + 1)
    kx, ky = n // 2, 1                                     # Nyquist column (even n), kx != ky
    assert abs(full[ky, kx] - ref[kx, ky]) <= BOUND["scatter"] * EPS * ref[kx, ky]
    assert abs(full[0, 0] - ref[0, 0]) <= BOUND["scatter"] * EPS * ref[0, 0]


def test_scattering_table_square_pixels(fb):
    n = 256
    got = scatter(fb, n, 14, 2.5e-11, 2.5e-11).astype(np.float64)
    ref = mdl.scatter_q64(14, n, 2.5e-11, 2.5e-11, 7288400.5)
    check("scatter", n, np.abs(got - ref) / ref / EPS)
    g = got.reshape(n // 2 + 1, -1)
    np.testing.assert_array_equal(g, g.T)                  # d1 == d2: symmetric under kx <-> ky


def prop(fb, n, d1, d2, d3=2e-10, lam=LAM):
    q = n // 2 + 1
    return run(fb, fb.PROP_TABLE, n, [np.full(q * q, np.nan, np.complex64)], [], [d1, d2, d3, lam])[0]


@pytest.mark.parametrize("n", TABLE_SIZES)
def test_propagator_table(n, fb):
    got = prop(fb, n, D1, D2)
    keep = mdl.prop_mask_q(n)
    # the 2/3 mask: exactly zeroHighFreq's float32 test (at 4096 and 8192 (float)(i1^2 + i2^2) rounds)
    np.testing.assert_array_equal(got != 0, keep)
    exact = mdl.prop_mask_exact_q(n)
    _ERRORS.setdefault("prop mask entries differing from the integer test", {})[str(n)] = int((keep != exact).sum())
    import sweep_model as sm
    np.testing.assert_array_equal(sm.quarter_to_full(got, n) != 0, sm.keep_mask(n))
    ref, ph = mdl.prop_q64(n, D1, D2, 2e-10, LAM)
    err = np.abs(got[keep].astype(np.complex128) * n * n - ref[keep] * n * n) / (1 + np.abs(ph[keep])) / EPS
    check("prop", n, err)
    r32 = mdl.prop_q32(n, D1, D2, 2e-10, LAM)
    check("prop32", n, np.abs(got[keep] - r32[keep]).astype(np.float64) * n * n / (1 + np.abs(ph[keep])) / EPS)


def test_propagator_table_square_pixels(fb):
    n = 256
    g = prop(fb, n, 2.5e-11, 2.5e-11).reshape(n // 2 + 1, -1)
    assert same_bits(g, np.ascontiguousarray(g.T))


# ---------------------------------------------------------------------------------------------------
# lens table
# ---------------------------------------------------------------------------------------------------
AB0 = [-6.1e-8, 2e-9, 3e-8, 4e-8, 2e-5, 5e-7, 6e-7, 7e-6, 8e-6, 9e-6, 1e-3, 2e-3, 3e-3, 4e-3]
AB1 = [0.0, 0.3, -0.7, 1.1, 0.0, 0.5, -1.3, 0.9, 2.1, -0.4, 0.0, 1.7, -2.5, 0.6]


def lens_objap(n):
    """An aperture radius that equals |nu| of a grid point near 3/8 of the band (in float32): that point and every
    point at the same |nu| are cut, neighbours within a few ulp are not."""
    nu = mdl.lens_nu32_candidates(n, D1, D2, LAM)[0]
    i = max(1, (3 * n) // 16)
    return float(nu[0, i])


def lens(fb, n, mode, transposed, objap, scale=0.75, defocus=-2e-8, spread=3e-9):
    f = [np.float32(v) for v in AB0 + AB1] + [defocus, spread, LAM, D1, D2, objap, scale]
    return run(fb, fb.LENS_TABLE, n, [np.full(n * n, np.nan, np.complex64)], [mode, transposed], f)[0].reshape(n, n)


@pytest.mark.parametrize("n,mode", [(n, m) for n in PIXEL_SIZES for m in (0, 2)] + [(BIG, 0)])
def test_lens_table(n, mode, fb, orc):
    objap = lens_objap(n)
    got = lens(fb, n, mode, 0, objap)
    assert same_bits(lens(fb, n, mode, 1, objap), np.ascontiguousarray(got.T))
    # aperture: exactly the float32 test nu < ObjAp, wherever the rounding of |nu| does not depend on how the
    # compiler fuses nu1^2 + nu2^2
    cands = [c < np.float32(objap) for c in mdl.lens_nu32_candidates(n, D1, D2, LAM)]
    sure = (cands[0] == cands[1]) & (cands[0] == cands[2])
    ap = got != 0
    np.testing.assert_array_equal(ap[sure], cands[0][sure])
    _ERRORS.setdefault("lens aperture points with a fusion-dependent test", {})[str(n)] = int((~sure).sum())
    assert (~ap).any() and ap.any()
    ref, chi = mdl.lens64(n, AB0, AB1, -2e-8, 3e-9, LAM, D1, D2, objap, 0.75, mode)
    check("lens", n, np.abs(got[ap] - ref[ap]) / (0.75 * (1 + chi[ap])) / EPS)
    p = mdl.params(n, D1, D2, lam=np.float32(LAM), ObjAp=np.float32(objap), defocspread=np.float32(3e-9), mode=mode,
                   pi=np.float32(mdl.PI32))
    p.ab0 = dict(zip(orc.ABERRATION_KEYS, map(np.float32, AB0)))
    p.ab1 = dict(zip(orc.ABERRATION_KEYS, map(np.float32, AB1)))
    p.defoci = np.array([-2e-8], np.float32)
    ctf32, _ = orc.lens_function(p, 0)
    check("lens32", n, np.abs(got[ap] - 0.75 * ctf32[ap].astype(np.complex128)) / (0.75 * (1 + chi[ap])) / EPS)


# ---------------------------------------------------------------------------------------------------
# detector table
# ---------------------------------------------------------------------------------------------------
MTF4 = (0.58, 0.42, 2.7, 15.5)


@pytest.mark.parametrize("n", PIXEL_SIZES + [BIG])
def test_detector_table(n, fb):
    scale = 1.0 / (n * n)
    for mode in ((0, 1) if n < BIG else (0,)):
        # exponents of the incoherence envelope about 9 at the Nyquist frequency of the finer axis
        ill = 3 / (np.pi * 5e-8 * LAM / (2 * D2)) if mode == 0 else 6 * LAM / (np.pi * n * D1)
        for use_inc in ((0, 1) if n < BIG else (1,)):
            for use_mtf in ((0, 1) if n < BIG else (1,)):
                fa = [*MTF4, ill, -5e-8, LAM, D1, D2, scale]
                got = run(fb, fb.DETECTOR_TABLE, n, [np.full(n * n, np.nan, np.float32)], [mode, use_inc, use_mtf],
                          fa)[0].reshape(n, n).astype(np.float64)
                ref, arg = mdl.detector64(n, MTF4, ill, -5e-8, LAM, D1, D2, scale, mode, use_inc, use_mtf)
                check("detector", n, np.abs(got - ref) / np.abs(ref) / (1 + arg) / EPS)
                r32 = mdl.detector32(n, MTF4, ill, -5e-8, LAM, D1, D2, scale, mode, use_inc, use_mtf)
                check("detector32", n, np.abs(got - r32) / np.abs(r32) / (1 + arg) / EPS)
                if not use_inc and not use_mtf:
                    assert np.all(got == np.float32(scale))


# ---------------------------------------------------------------------------------------------------
# tilt / Tukey / area mask
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", PIXEL_SIZES + [BIG])
def test_tilt_beam(n, fb):
    rng = np.random.default_rng(n)
    psi = crand(rng, (n, n))
    tbx, tby = 1.3e-3, -0.4e-3                             # asymmetric: tb_x pairs with d2 and the row index
    for flag in ((1, -1) if n < BIG else (-1,)):
        got = run(fb, fb.TILT_BEAM, n, [psi], [flag], [D1, D2, LAM, tbx, tby])[0]
        ph, mag = mdl.tilt_phase64(n, D1, D2, LAM, tbx, tby, flag)
        ref = psi * np.exp(1j * ph)
        scale = np.abs(psi) * (1 + mag)
        check("tilt", n, np.abs(got - ref) / scale / EPS)
        r32 = mdl.tilt32(psi, n, D1, D2, LAM, tbx, tby, flag)
        check("tilt32", n, np.abs(got - r32.astype(np.complex128)) / scale / EPS)


def dn_pairs(n):
    if n == BIG:
        return [(3, n // 5)]                               # the steepest taper: the largest N / dn
    return [(0, n // 2), (n // 2, 0), (min(3, n // 2), max(1, n // 5)), (max(1, n // 7), min(n // 2, 2 * n // 5))]


@pytest.mark.parametrize("n", PIXEL_SIZES + [BIG])
def test_tukey_and_area_mask(n, fb):
    rng = np.random.default_rng(n + 1)
    psi = crand(rng, (n, n))
    for dn1, dn2 in dn_pairs(n):
        got = run(fb, fb.TUKEY, n, [psi], [dn1, dn2])[0]
        ref = psi * mdl.tukey64(n, dn1, dn2)
        ts = mdl.tukey_err_scale(n, dn1, dn2)
        check("tukey", n, np.abs(got - ref) / np.abs(psi) / ts / EPS)
        check("tukey32", n, np.abs(got - mdl.tukey32(psi, n, dn1, dn2)) / np.abs(psi) / ts / EPS)
        got = run(fb, fb.AREA_MASK, n, [psi], [dn1, dn2])[0]
        w = mdl.area64(n, dn1, dn2)
        ref = (1 - w) + psi * w
        check("area", n, np.abs(got - ref) / (1 + np.abs(psi)) / EPS)
        check("area32", n, np.abs(got - mdl.area_blend32(psi, n, dn1, dn2)) / (1 + np.abs(psi)) / EPS)


@pytest.mark.parametrize("n", PIXEL_SIZES)
def test_plane_wave_and_zero_outband(n, fb):
    batch = 3
    want = np.zeros((batch, n, n), np.complex64)
    want[:, :, 0] = 1
    for nb in (batch, batch - 1):                          # images past the batch stay untouched
        got = [np.full((batch, n, n), np.nan, np.complex64)]
        fb.sweep_test(fb.PLANE_WAVE, n, nb, got)
        assert same_bits(got[0][:nb], want[:nb]) and np.isnan(got[0][nb:]).all()
    rng = np.random.default_rng(n + 2)
    psi = crand(rng, (batch, n, n))
    for lo, hi in ((n // 3, n - n // 3), (0, n), (1, 1), (n - 1, n)):
        cp = [psi.copy()]
        fb.sweep_test(fb.ZERO_OUTBAND, n, batch, cp, [lo, hi])
        want = psi.copy()
        want[:, :, lo:hi] = 0
        assert same_bits(cp[0], want), (lo, hi)


@pytest.mark.parametrize("n", [1, 5, 143 * 143, 5_000_011])          # past the grid-stride cap of 148 * 8 CTAs
def test_absorptive_factor_and_scale(n, fb):
    rng = np.random.default_rng(n)
    v = crand(rng, n)
    imp = np.float32(0.0837)
    got = run(fb, fb.ABSORPTIVE, n, [v], [], [imp])[0]
    assert same_bits(got.real, v.real) and same_bits(got.imag, (v.real * imp).astype(np.float32))
    s = np.float32(1.0 / 143)
    got = run(fb, fb.SCALE_CPX, n, [v], [], [s])[0]
    assert same_bits(got.real, (v.real * s).astype(np.float32)) and same_bits(got.imag, (v.imag * s).astype(np.float32))


# ---------------------------------------------------------------------------------------------------
# reductions
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 143 * 143, 1_000_003, 8192 * 8192])
def test_norm2(n, fb):
    rng = np.random.default_rng(n)
    p = crand(rng, n)
    outs = [run(fb, fb.NORM2, n, [p, np.zeros(2, np.float32)])[1] for _ in range(2)]
    assert same_bits(outs[0], outs[1])
    got = float(outs[0].view(np.float64)[0])
    ref = float(np.sum(p.real.astype(np.float64) ** 2) + np.sum(p.imag.astype(np.float64) ** 2))
    assert abs(got - ref) <= 1e-13 * ref, (got, ref)


@pytest.mark.parametrize("n,nsrc", [(n, s) for n in (1, 3, 4, 5, 143 * 143, 2 * 143 * 143) for s in (1, 2, 15)]
                         + [(4096 * 4096, s) for s in (1, 2, 3)])
def test_peer_sum(n, nsrc, fb):
    rng = np.random.default_rng(n + nsrc)
    bufs = [rng.standard_normal(n).astype(np.float32) * np.float32(10.0 ** (r % 5)) for r in range(nsrc + 1)]
    got = run(fb, fb.PEER_SUM, n, bufs, [nsrc])
    want = bufs[0].copy()
    for b in bufs[1:]:
        want = (want + b).astype(np.float32)                # in order, float32
    assert same_bits(got[0], want)
    for a, b in zip(got[1:], bufs[1:]):
        assert same_bits(a, b)                              # sources untouched


# ---------------------------------------------------------------------------------------------------
# random numbers
# ---------------------------------------------------------------------------------------------------
def jitter(fb, xyz, dwf, pairs):
    nat = len(dwf)
    total = sum(c for b, c in pairs if b >= 0)
    out = np.full((total, nat, 3), np.nan, np.float32)
    return run(fb, fb.JITTER, nat, [xyz, dwf, out], [v for pr in pairs for v in pr])[2]


@pytest.fixture(scope="module")
def xorwow_draws(orc):
    """The oracle's XORWOW normals of 3 * 70 streams, 90 draws each ([draw][stream])."""
    nat = 70
    x = orc.Xorwow(1, 3 * nat)
    return nat, np.stack([x.normal() for _ in range(90)])


@pytest.mark.parametrize("burn,nconf", [(0, 1), (1, 1), (3, 2), (0, 40), (7, 40)])
def test_jitter_draws(burn, nconf, fb, xorwow_draws):
    """xyz = 0 and dwf = 1: configuration c holds 0.112539540f * (normal number burn + c) of every stream."""
    nat, draws = xorwow_draws
    xyz = np.zeros((nat, 3), np.float32)
    dwf = np.ones(nat, np.float32)
    got = jitter(fb, xyz, dwf, [(burn, nconf)]).reshape(nconf, -1).astype(np.float64)
    want = draws[burn:burn + nconf].astype(np.float64) * float(np.float32(0.112539540))
    # the device's logf / __sincosf against float32 libm: a few 1e-6 of the normal
    err = np.abs(got - want) / (np.float32(0.112539540) * (1 + np.abs(draws[burn:burn + nconf])))
    _ERRORS.setdefault("jitter normal abs error", {})[f"{burn},{nconf}"] = float(err.max())
    _ERRORS.setdefault("jitter draws bitwise equal (%)", {})[f"{burn},{nconf}"] = float(
        100 * np.mean(got == (want.astype(np.float32)).astype(np.float64)))
    assert err.max() <= 4e-6


def test_jitter_batch_equals_single_calls_and_restart(fb, orc):
    """One call of 40 configurations is bitwise 40 calls of one; a restart (the engine's rng re-init when a
    configuration before the stream position is asked for) followed by a burn gives the same draws again; the
    draws of the reference for tests/data/phonon64.cnf come out bit for bit."""
    from conftest import DATA, golden
    p, Z, xyz, dwf, occ = orc.read_cnf(str(DATA / "phonon64.cnf"))
    xyz = np.ascontiguousarray(xyz, np.float32)
    dwf = np.ascontiguousarray(dwf, np.float32)
    one = jitter(fb, xyz, dwf, [(0, 40)])
    many = jitter(fb, xyz, dwf, [(0, 1)] * 40)
    assert same_bits(one, many)
    again = jitter(fb, xyz, dwf, [(0, 3), (-1, 0), (5, 2), (0, 4)])
    assert same_bits(again[:3], one[:3])
    assert same_bits(again[3:], one[5:11])
    g, _ = golden("phonon64")
    assert same_bits(one[:p.frPh], g["xyz_cfg"][:p.frPh])


def test_anscombe_noise(fb, orc):
    n = 4096
    dose = np.float32(37.0)
    rng = np.random.default_rng(5)
    thr = np.float32(1e-2)
    fi = np.concatenate([
        np.nextafter(thr, np.float32(0)) * np.ones(8, np.float32), np.full(8, thr, np.float32),
        np.nextafter(thr, np.float32(1)) + np.arange(8, dtype=np.float32) * np.float32(1e-9),
        rng.uniform(0.01, 0.5, 1000).astype(np.float32),       # many round to 0
        rng.uniform(0.5, 50, 1000).astype(np.float32),
        rng.uniform(1e3, 1e6, 1000).astype(np.float32),
        np.zeros(24, np.float32), -rng.uniform(0, 1, 24).astype(np.float32)])
    fi = np.concatenate([fi, rng.uniform(0, 2e-2, n - len(fi)).astype(np.float32)])
    f1 = (fi / dose).astype(np.float32) + 1j * rng.standard_normal(n).astype(np.float32)
    f1 = f1.astype(np.complex64)
    f2 = np.roll(f1, 7)                                       # other pixels lit in the second call
    g1, g2 = run(fb, fb.ANSCOMBE, n, [f1, f2], [1 + 3], [dose])
    x = orc.Xorwow(1 + 3, n)
    d1, d2 = x.normal(), x.normal()
    lit1 = (f1.real * dose).astype(np.float32) > thr
    lit2 = (f2.real * dose).astype(np.float32) > thr
    flips = 0
    for f, g, lit, nrm in ((f1, g1, lit1, d1), (f2, g2, lit2, np.where(lit1, d2, d1))):
        assert same_bits(g.imag, f.imag)
        assert same_bits(g.real[~lit], f.real[~lit])           # dark pixels untouched
        fil = (f.real[lit] * dose).astype(np.float32)
        want, arg, v = mdl.anscombe32(fil, nrm[lit], dose)
        got = g.real[lit]
        diff = got != want
        # a rounding flip is one count: only where the rounded value sits within the propagated error of x.5
        dn = 4e-6 * (1 + np.abs(nrm[lit]))
        slack = 4 * np.spacing(np.abs(arg)) + 0.5 * np.abs(v) * dn * np.sqrt(1 - np.exp(-fil / 0.777134))
        near = np.abs(np.abs(arg - np.trunc(arg)) - 0.5) <= slack
        assert np.all(near[diff]), np.flatnonzero(diff & ~near)[:5]
        # the counts differ by exactly one
        np.testing.assert_array_equal(np.abs(np.rint(got[diff] * np.float64(dose)) - np.rint(want[diff] * np.float64(dose))), 1)
        flips += int(diff.sum())
        assert np.any(want == 0) and np.any(want > 1e3)
    _ERRORS.setdefault("anscombe rounding flips", {})["4096"] = flips


# ---------------------------------------------------------------------------------------------------
# deposit records
# ---------------------------------------------------------------------------------------------------
RD1 = 2.0 ** -35                                          # power of two: x1 = x / d1 + m/2 - 1/2 exact, .5 ties
RD2 = float(np.float32(2.1 * RD1))
RD3 = 2e-10


def atoms_for(n, m3, nat, nconf, seed, reject_conf=None):
    """[nconf][nat][3] coordinates: random inside the box, plus atoms on x1 = 1 and m - 2 (rejected), on the
    first and last slice, and on .5 ties of x1."""
    rng = np.random.default_rng(seed)
    xyz = np.empty((nconf, nat, 3), np.float32)
    for c in range(nconf):
        x1 = rng.uniform(-0.5, n + 0.5, nat)
        x2 = rng.uniform(-0.5, n + 0.5, nat)
        x3 = rng.uniform(-1.0, m3, nat)
        k = min(nat // 8, 64)
        x2[:2 * k] = rng.uniform(2.0, n - 3.0, 2 * k)       # the edge cases of x1 and i3 inside in y
        x3[:k] = rng.uniform(0.0, m3 - 1.0, k)
        x1[k:2 * k] = rng.uniform(2.0, n - 3.0, k)
        x1[:k] = np.tile([1.0, n - 2.0, 1.5, n - 2.5, np.floor(n / 3) + 0.5, 2.5, n / 2 + 0.5, 1.0 + 2 ** -20],
                         k // 8 + 1)[:k]
        x3[k:2 * k] = np.tile([0.0, m3 - 1.0, -0.5, m3 - 0.5 - 1e-3], k // 4 + 1)[:k]
        xyz[c, :, 0] = ((x1 - n / 2 + 0.5) * RD1).astype(np.float32)
        xyz[c, :, 1] = ((x2 - n / 2 + 0.5) * RD2).astype(np.float32)
        xyz[c, :, 2] = ((x3 - m3 / 2 + 0.5) * RD3).astype(np.float32)
        if c == reject_conf:
            xyz[c, :, 2] = 1e-6                            # every atom above the slab
    return xyz


@pytest.mark.parametrize("n,m3,nz,nat,nconf", [
    (8, 2, 2, 40, 3),            # 5-bit keys: one digit pass (rounded up to two)
    (64, 4, 3, 1500, 40),        # 10 bits: two passes; 6000 records per configuration: two sort blocks
    (143, 5, 2, 5000, 3),        # generic size (no row masks), 11 bits
    (1024, 40, 3, 3000, 3),      # 17 bits: three passes (rounded up to four)
    (512, 8, 4, 20000, 1),       # 15 bits, 80000 records: twenty sort blocks
    (4096, 1100, 4, 2000, 1),    # 25 bits: four passes
])
def test_records(n, m3, nz, nat, nconf, fb):
    rng = np.random.default_rng(n + nconf)
    xyz = atoms_for(n, m3, nat, nconf, n * 7 + nconf, reject_conf=1 if nconf > 1 else None)
    zidx = rng.integers(0, nz, nat).astype(np.int32)
    occ = rng.uniform(0.2, 1.0, nat).astype(np.float32)
    nkeys = m3 * nz * n
    e = fb.sweep_geom(n)["line_points"]
    rp_stride = nkeys + 1 + ((nkeys // n) * (n // e) if e else 0)
    nrec = 4 * nat
    bufs = [xyz, zidx, occ, np.zeros(nconf * nrec, np.int32), np.zeros(nconf * nrec, np.int32),
            np.zeros(nconf * nrec, np.float32), np.full(nconf * rp_stride, -7, np.int32)]
    _, _, _, keys, cols, w, rp = run(fb, fb.RECORDS, n, bufs, [m3, nz, nconf], [RD1, RD2, RD3])
    keys = keys.view(np.uint32).reshape(nconf, nrec)
    cols, w, rp = cols.reshape(nconf, nrec), w.reshape(nconf, nrec), rp.reshape(nconf, rp_stride)
    seen_tie = seen_edge = False
    for c in range(nconf):
        k, cc, ww, rowptr, (i1, i2, i3, ok) = mdl.records_model(xyz[c], zidx, occ, n, m3, nz, RD1, RD2, RD3)
        np.testing.assert_array_equal(keys[c], k, err_msg=f"keys of configuration {c}")
        np.testing.assert_array_equal(cols[c], cc, err_msg=f"columns of configuration {c}")
        assert same_bits(w[c], ww), f"weights of configuration {c}"
        np.testing.assert_array_equal(rp[c, :nkeys + 1], rowptr, err_msg=f"row pointers of configuration {c}")
        if e:
            np.testing.assert_array_equal(rp[c, nkeys + 1:].view(np.uint32), mdl.row_masks(rowptr, nkeys, n, e))
        if c == 1 and nconf > 1:
            assert not ok.any() and rowptr[-1] == 0          # the configuration without any accepted atom
        else:
            assert ok.any() and not ok.all()
            seen_tie |= bool(np.any(ok & (i1 * 2 == np.floor(n / 3) * 2 + 2)))
            seen_edge |= bool(np.any(ok & (i3 == 0)) and np.any(ok & (i3 == m3 - 1)))
    assert seen_tie and seen_edge


# ---------------------------------------------------------------------------------------------------
# end to end: rectangular pixels, a rectangular image in the square sample
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("m", [512, 143])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_rectangular_pixels_end_to_end(m, mode, fb, orc, tmp_path):
    from fdes_b200 import specimens
    d1, d2 = 0.21e-10, 0.1e-10
    n1, n2 = (m * 3) // 4, m // 2
    n1 -= (m - n1) % 2
    n2 += (m - n2) % 2
    dn1, dn2 = (m - n1) // 2, (m - n2) // 2
    rng = np.random.default_rng(m + mode)
    nat = 60
    atoms = np.zeros((nat, 6), np.float64)
    atoms[:, 0] = rng.choice([79, 14, 8], nat)
    atoms[:, 1] = rng.uniform(-0.3, 0.3, nat) * m * d1
    atoms[:, 2] = rng.uniform(-0.3, 0.3, nat) * m * d2
    atoms[:, 3] = rng.uniform(-2e-10, 2e-10, nat)
    atoms[:, 4] = 0.005e-20
    atoms[:, 5] = 1.0
    cnf = specimens.write_cnf(tmp_path / "rect.cnf", image_size=n1, border_size=dn1, image_size_y=n2,
                              border_size_y=dn2, slices=3, pixel_size=d1, pixel_size_y=d2, slice_thickness=2e-10,
                              atoms=atoms, voltage=200e3, mode=mode, objective_aperture=20e-3,
                              focus_spread=4e-9, illumination_angle=0.5e-3, mtf=(0.6, 0.4, 2.0, 10.0),
                              aberrations={"C1": (-3e-8, 0.0), "A1": (2e-9, 0.4), "C3": (1e-4, 0.0)},
                              beam_tilts=[(1.5e-3, -0.6e-3)], defoci=[-1e-8])
    p, Z, xyz, dwf, occ = orc.read_cnf(str(cnf))
    assert (p.m1, p.m2, p.n1, p.n2, p.dn1, p.dn2) == (m, m, n1, n2, dn1, dn2) and p.d1 != p.d2
    ref = orc.build_measurements(p, Z, xyz, dwf, occ)
    with fb.Simulation(cnf, want_exitwave=True) as sim:
        img, ew = sim.simulate()
    assert img.shape == (1, n2, n1)
    assert rel_l2(ew, ref.exitwave) < TOL_WAVE
    assert rel_l2(img, ref.image) < TOL_INTENSITY
    # without an exit wave to keep, imaging at a pipelined size applies the CTF inside the last slice's column
    # transform (the transposed lens table): the production imaging path
    assert fb.sweep_geom(m)["pipelined"] == (m == 512)
    with fb.Simulation(cnf) as sim:
        img2, _ = sim.simulate()
    assert rel_l2(img2, ref.image) < TOL_INTENSITY
