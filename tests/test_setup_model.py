"""CPU: the float64 models of setup_models.py (the references of test_setup_fp64_gpu.py) against the oracle's
float32 restatements of the same kernels, to float32 rounding, with rectangular pixels -- so that an error in a
model shows without a GPU."""
import numpy as np
import pytest

import setup_models as mdl

D1, D2, LAM = 2.1e-11, 1.0e-11, 2.507934e-12
EPS = mdl.EPS32


@pytest.mark.parametrize("n", [8, 9, 64, 143])
def test_quarter_table_models(n):
    for Z in (1, 6, 79, 103, 0, 200):
        ref = mdl.scatter_q64(Z, n, D1, D2, 7288400.5)
        r32 = mdl.scatter_q32(Z, n, D1, D2, 7288400.5)
        assert np.max(np.abs(r32 - ref) / ref) < 16 * EPS, Z
    ref, ph = mdl.prop_q64(n, D1, D2, 2e-10, LAM)
    r32 = mdl.prop_q32(n, D1, D2, 2e-10, LAM)
    keep = mdl.prop_mask_q(n)
    np.testing.assert_array_equal(r32 != 0, keep)
    assert np.max(np.abs(r32[keep] - ref[keep]) * n * n / (1 + np.abs(ph[keep]))) < 16 * EPS
    # a swapped d1 / d2 is far outside that bound
    sw, _ = mdl.prop_q64(n, D2, D1, 2e-10, LAM)
    assert n < 9 or np.max(np.abs(sw[keep] - ref[keep]) * n * n) > 1e-3


def test_propagator_mask_float_semantics():
    for n in (64, 143, 4096, 8192):
        diff = int((mdl.prop_mask_q(n) != mdl.prop_mask_exact_q(n)).sum())
        assert diff == 0 or n >= 4096


@pytest.mark.parametrize("n", [9, 64, 143])
@pytest.mark.parametrize("mode", [0, 2])
def test_lens_model(n, mode, orc):
    ab0 = [-6.1e-8, 2e-9, 3e-8, 4e-8, 2e-5, 5e-7, 6e-7, 7e-6, 8e-6, 9e-6, 1e-3, 2e-3, 3e-3, 4e-3]
    ab1 = [0.0, 0.3, -0.7, 1.1, 0.0, 0.5, -1.3, 0.9, 2.1, -0.4, 0.0, 1.7, -2.5, 0.6]
    ref, chi = mdl.lens64(n, ab0, ab1, -2e-8, 3e-9, LAM, D1, D2, 1.0, 1.0, mode)
    p = mdl.params(n, D1, D2, lam=np.float32(LAM), ObjAp=np.float32(1.0), defocspread=np.float32(3e-9), mode=mode,
                   pi=np.float32(mdl.PI32))
    p.ab0 = dict(zip(orc.ABERRATION_KEYS, map(np.float32, ab0)))
    p.ab1 = dict(zip(orc.ABERRATION_KEYS, map(np.float32, ab1)))
    p.defoci = np.array([-2e-8], np.float32)
    ctf, ap = orc.lens_function(p, 0)
    assert ap.all()
    assert np.max(np.abs(ctf - ref) / (1 + chi)) < 16 * EPS


@pytest.mark.parametrize("n", [9, 64, 143])
def test_detector_model(n):
    for mode in (0, 1):
        ill = 3 / (np.pi * 5e-8 * LAM / (2 * D2)) if mode == 0 else 6 * LAM / (np.pi * n * D1)
        for inc in (0, 1):
            for mt in (0, 1):
                ref, arg = mdl.detector64(n, (0.58, 0.42, 2.7, 15.5), ill, -5e-8, LAM, D1, D2, 0.5, mode, inc, mt)
                r32 = mdl.detector32(n, (0.58, 0.42, 2.7, 15.5), ill, -5e-8, LAM, D1, D2, 0.5, mode, inc, mt)
                assert np.max(np.abs(r32 - ref) / ref / (1 + arg)) < 16 * EPS
                if inc:
                    assert arg.max() > 1                # the envelope is not flat


@pytest.mark.parametrize("n", [8, 9, 64, 143])
def test_real_space_models(n):
    rng = np.random.default_rng(n)
    psi = (rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))).astype(np.complex64)
    for flag in (1, -1):
        ph, mag = mdl.tilt_phase64(n, D1, D2, LAM, 1.3e-3, -0.4e-3, flag)
        r32 = mdl.tilt32(psi, n, D1, D2, LAM, 1.3e-3, -0.4e-3, flag)
        assert np.max(np.abs(r32 - psi * np.exp(1j * ph)) / np.abs(psi) / (1 + mag)) < 16 * EPS
    for dn1, dn2 in [(0, n // 2), (n // 2, 0), (3, 1), (1, 3)]:
        w = mdl.tukey64(n, dn1, dn2)
        assert np.max(np.abs(mdl.tukey32(psi, n, dn1, dn2) - psi * w) / np.abs(psi)
                      / mdl.tukey_err_scale(n, dn1, dn2)) < 4 * EPS
        w = mdl.area64(n, dn1, dn2)
        assert np.max(np.abs(mdl.area_blend32(psi, n, dn1, dn2) - ((1 - w) + psi * w)) / (1 + np.abs(psi))) < 4 * EPS


def test_xorwow_normals_against_box_muller(orc):
    """The oracle's curand_normal restatement against the float64 Box-Muller of its own raw words."""
    x = orc.Xorwow(1, 300)
    y = orc.Xorwow(1, 300)
    for _ in range(3):
        a, b = x.normal(), x.normal()
        u, v = y.next_u32(), y.next_u32()
        s, c = mdl.box_muller64(u, v)
        assert np.max(np.abs(a - s) / (1 + np.abs(s))) < 4e-6
        assert np.max(np.abs(b - c) / (1 + np.abs(c))) < 4e-6


def test_records_model(orc):
    n, m3, nz, nat = 64, 3, 2, 400
    rng = np.random.default_rng(1)
    xyz = np.stack([rng.uniform(-0.55, 0.55, nat) * n * 2.0 ** -35, rng.uniform(-0.55, 0.55, nat) * n * 2.1 * 2.0 ** -35,
                    rng.uniform(-2.5, 2.5, nat) * 2e-10], 1).astype(np.float32)
    zidx = (np.arange(nat) % nz).astype(np.int32)
    occ = np.ones(nat, np.float32)
    k, c, w, rp, (i1, i2, i3, ok) = mdl.records_model(xyz, zidx, occ, n, m3, nz, 2.0 ** -35, 2.1 * 2.0 ** -35, 2e-10)
    assert np.all(np.diff(k.astype(np.int64)) >= 0) and ok.any() and not ok.all()
    assert rp[-1] == 4 * ok.sum()
    # the weights of an atom sum to its occupancy; the density of each slice / species is the oracle's
    np.testing.assert_allclose(w.sum(), ok.sum(), rtol=1e-5)
    p = mdl.params(n, 2.0 ** -35, 2.1 * 2.0 ** -35, d3=np.float32(2e-10), m3=m3)
    for s in range(m3):
        for z in range(nz):
            dens = np.zeros(n * n, np.float64)
            lo, hi = rp[(s * nz + z) * n], rp[(s * nz + z + 1) * n]
            np.add.at(dens, ((k[lo:hi] - (s * nz + z) * n) * n + c[lo:hi]).astype(np.int64), w[lo:hi])
            ref = orc.square_atoms(zidx, z, xyz, occ, 0.0, s, p).real.reshape(-1)
            np.testing.assert_allclose(dens, ref, atol=1e-6)
    masks = mdl.row_masks(rp, m3 * nz * n, n, 8)
    assert masks.shape == (m3 * nz * 8,)
