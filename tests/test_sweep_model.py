"""CPU checks of oracle/sweep_model.py, the float64 models the per-sweep GPU tests (test_sweeps_fp64_gpu.py,
test_formation_fp64_gpu.py) compare the kernels with: composed S1..S6 they must reproduce the reference's phase
grating and forward propagation (fdes_oracle, float32) to float32 rounding -- which pins the models' conventions (domains,
normalisations, table layouts, pair packing) to the reference's semantics."""
import numpy as np
import pytest

from conftest import DATA, rel_l2

import sweep_model as sm

SIZES = [64, 128, 256, 512, 1024, 2048, 4096, 320, 800, 1000, 96, 250, 600, 1022, 143]


def deposit_records(orc, p, Z, xyz, occ):
    """The product's deposit records of one configuration (launch_bin_atoms: 4 per accepted atom, key
    (slice * nZ + species) * N + row), sorted by key, and the row pointers over all keys."""
    Zlist = orc.list_of_elements(np.asarray(Z))
    zidx = np.array([Zlist.index(z) for z in Z])
    i1, i2, i3, r1, r2, ok = orc.bin_atoms(xyz, p)
    ok = ok & (i3 >= 0) & (i3 < p.m3)
    g1, g2 = np.where(r1 < 0, -1, 1), np.where(r2 < 0, -1, 1)
    a1, a2 = np.abs(r1), np.abs(r2)
    oc = np.asarray(occ, np.float32)
    one = np.float32(1)
    w = [(one - a1) * (one - a2) * oc, (one - a1) * a2 * oc, a1 * a2 * oc, a1 * (one - a2) * oc]
    rows = [i2, i2 + g2, i2 + g2, i2]
    cols = [i1, i1, i1 + g1, i1 + g1]
    n, nz = p.m1, len(Zlist)
    keys = np.concatenate([((i3 * nz + zidx) * n + r)[ok] for r in rows])
    order = np.argsort(keys, kind="stable")
    c = np.concatenate([cc[ok] for cc in cols])[order].astype(np.int32)
    ww = np.concatenate([x[ok] for x in w])[order].astype(np.float32)
    rowptr = np.searchsorted(keys[order], np.arange(p.m3 * nz * n + 1)).astype(np.int32)
    return Zlist, rowptr, c, ww


def test_model_slice_pair_matches_reference(orc):
    """S1..S6 of the model for the first slice pair of tem64 (3 species, imPot set) and a plane wave against
    fdes_oracle.phase_grating + forward_propagation."""
    p, Z, xyz, dwf, occ = orc.read_cnf(str(DATA / "tem64.cnf"))
    p = p.copy()
    orc.set_sub_slices(p, orc.sub_slice_ratio(p.d3, p.subSlTh))
    p.imPot = np.float32(0.05)          # the absorptive factor takes part in the comparison
    n = p.m1
    assert p.m3 >= 2
    Zlist, rowptr, cols, w = deposit_records(orc, p, Z, xyz, occ)
    nz = len(Zlist)
    Gq = np.stack([sm.full_to_quarter(orc.scattering_factor(z, p), n) for z in Zlist])
    Pq = sm.full_to_quarter(orc.fresnel_propagator(p), n)
    # the quarter tables hold the whole tables (the reference's float32 tables are symmetric to rounding)
    np.testing.assert_allclose(sm.quarter_to_full(Gq[0], n), orc.scattering_factor(Zlist[0], p), rtol=1e-6)
    np.testing.assert_array_equal(sm.quarter_to_full(Pq, n), orc.fresnel_propagator(p))

    A, written = sm.s1_density_rows(rowptr[None], cols[None], w[None], n, nz, 1, 0, 1)
    assert written.any() and not written.all()
    B = sm.s2_potential_cols(A, Gq, rowptr[None], n, nz, 1, 0, 1)
    D, V = sm.s3_transmit_rows(B, 2, p.imPot)
    D = sm.s4_bandlimit_cols(D, 2, 1)
    band = np.ones(n, bool)
    Psi = sm.plane_wave_rowspace(n)
    psi_ref = np.ones((n, n), np.complex64)
    for s in range(2):
        Psi = sm.s5_multiply_rows(Psi, D[s:s + 1], 0, band, False)
        Psi = sm.s6_propagate_cols(Psi, Pq, band)
        V_ref = orc.phase_grating(s, np.asarray(Z), Zlist, xyz, occ, p.imPot, p)
        # the pair packing: slice s in the real part, slice s + 1 in the imaginary part of one potential
        Vs = V[0].real if s == 0 else V[0].imag
        assert rel_l2(Vs * (1 + 1j * float(p.imPot)), V_ref) < 1e-6
        psi_ref = orc.forward_propagation(psi_ref, V_ref, p)
        # psi = IFFT_row(Psi) in the (kx, y) convention Psi = FFT_row(psi) / N
        e = rel_l2(sm.ifft_rows(Psi[0]), psi_ref)
        assert e < 3e-6, (s, e)


def test_model_odd_pairing_and_absent_species(orc):
    """(cfg_stride, cfg_off2) = (2, 1): image b packs configuration 2b (real) and 2b + 1 (imaginary); a species
    with no records adds nothing to S2."""
    rng = np.random.default_rng(5)
    n, nz, nsl, nconf = 32, 2, 1, 4
    rowptr = np.zeros((nconf, nsl * nz * n + 1), np.int32)
    cols = np.zeros((nconf, 40), np.int32)
    w = np.zeros((nconf, 40), np.float32)
    for c in range(nconf):
        rows = np.sort(rng.integers(0, n, 40))          # species 0 only
        rowptr[c] = np.searchsorted(rows, np.arange(nsl * nz * n + 1))
        cols[c] = rng.integers(0, n, 40)
        w[c] = rng.random(40)
    A, _ = sm.s1_density_rows(rowptr, cols, w, n, nz, 2, 0, 0, 2, 1)
    for b in range(2):
        d = sm.ifft_rows(A[b, 0]) / n
        np.testing.assert_allclose(d.real, sm.density(rowptr, cols, w, n, nz, 0, 0, 2 * b), atol=1e-12)
        np.testing.assert_allclose(d.imag, sm.density(rowptr, cols, w, n, nz, 0, 0, 2 * b + 1), atol=1e-12)
        assert not A[b, 1].any()
    Gq = rng.random((nz, (n // 2 + 1) ** 2))
    B = sm.s2_potential_cols(A, Gq, rowptr, n, nz, 2, 0, 0, 2, 1)
    ref = sm.ifft_cols(sm.fft_cols(A[:, 0]) * sm.quarter_to_full(Gq[0], n))
    np.testing.assert_allclose(B, ref, atol=1e-9 * np.abs(ref).max())


@pytest.mark.parametrize("n", SIZES)
def test_library_geometry_matches_model(fb, n):
    """The band columns the library's sweeps run with (make_sweep_geom) are those of the model: kb from the float32
    test of zeroHighFreq, bounds rounded outwards to multiples of 32; every column on the generic sweeps."""
    g = fb.sweep_geom(n)
    assert (g["lo_end"], g["hi_start"]) == sm.band_limits(n, g["line_points"] > 0)
    band = sm.band_columns(n, g["lo_end"], g["hi_start"])
    # every column the 2/3 limit keeps anywhere is a band column
    assert band[sm.keep_mask(n).any(axis=0)].all()
    assert g["pipelined"] == (n in (512, 1024, 2048, 4096))


@pytest.mark.parametrize("n", [64, 143])
def test_probe_model_whole_pixel_shift_is_roll(n):
    """A probe shifted by whole pixels (sx = p / N) is the unshifted probe rolled by p pixels: psi = IFFT_row(Psi)
    in the (kx, y) convention Psi = FFT_row(psi) / N, and the shift moves the probe towards +x, +y."""
    rng = np.random.default_rng(11)
    psi0 = rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))
    PSI0 = sm.fft_cols(sm.fft_rows(psi0) / n)
    band = np.ones(n, bool)
    p1, p2 = 5, -(n // 3)
    Psi = sm.probe_cols(PSI0, [[0.0, 0.0], [p1 / n, p2 / n]], band)
    np.testing.assert_allclose(sm.ifft_rows(Psi[0]), psi0, atol=1e-12)
    np.testing.assert_allclose(sm.ifft_rows(Psi[1]), np.roll(psi0, (p2, p1), axis=(0, 1)), atol=1e-12)


def test_detector_model_everything_is_parseval():
    """A ring covering every |k| sums N * sum |Psi|^2 over the band columns (Parseval along the columns)."""
    rng = np.random.default_rng(12)
    n = 128
    Psi = rng.standard_normal((2, n, n)) + 1j * rng.standard_normal((2, n, n))
    band = sm.band_columns(n, 32, 96)
    out0 = np.array([[1.0, 2.0], [3.0, 4.0]])
    res = sm.detector_cols(Psi, band, [0.0, 0.0], [np.inf, 0.0], 1.0, 1.0, 0.5, out0)
    parseval = n * (np.abs(Psi[..., band]) ** 2).sum(axis=(-2, -1))
    np.testing.assert_allclose(res[:, 0], out0[:, 0] + 0.5 * parseval, rtol=1e-12)
    np.testing.assert_array_equal(res[:, 1], out0[:, 1])          # in2 == out2: empty


@pytest.mark.parametrize("n", [143, 144])
def test_rows_model_store_shift_is_fftshift(n):
    rng = np.random.default_rng(13)
    x = rng.standard_normal((2, n, n)) + 1j * rng.standard_normal((2, n, n))
    got = sm.rows_fft(x, -1, sm.ROW_STORE_SHIFT, 0.5)
    np.testing.assert_allclose(got, 0.5 * np.fft.fftshift(np.fft.fft(x, axis=-1), axes=(-2, -1)), rtol=1e-12, atol=1e-9)
