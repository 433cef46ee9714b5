"""4D-STEM without a GPU: a float64 model of the 4D detector sweep against the reference's
diffraction pattern, and the window rules of fdes_b200_stem_4d_side (host only)."""
import types

import numpy as np
import pytest

import sweep_model as sm


def detector4d_model(Psi, band, Q, b, weight, out0):
    """float64 model of launch_detector4d_cols: out[b] = out0[b] + weight * (|FFT_col(Psi_b)|^2 over the band columns, 0
    in the others, fftshifted as fdes_oracle.fftshift2 -- out[(i + N/2) mod N] = in[i] --, cropped to [o, o + Q)^2 with
    o = (N - Q) / 2 and summed over b x b bins): [batch][Q/b][Q/b]."""
    Psi = np.asarray(Psi)
    n = Psi.shape[-1]
    inten = np.abs(sm.fft_cols(np.where(band, Psi, 0))) ** 2
    o, s = (n - Q) // 2, Q // b
    win = np.roll(inten, (n // 2, n // 2), axis=(-2, -1))[..., o:o + Q, o:o + Q]
    binned = win.reshape(*win.shape[:-2], s, b, s, b).sum(axis=(-3, -1))
    return np.array(out0, np.float64) + float(weight) * binned


def _crop_bin(img, q, b):
    n = img.shape[-1]
    o, s = (n - q) // 2, q // b
    w = img[..., o:o + q, o:o + q].astype(np.float64)
    return w.reshape(*w.shape[:-2], s, b, s, b).sum(axis=(-3, -1))


@pytest.mark.parametrize("n", [16, 17, 30, 45])
@pytest.mark.parametrize("b", [1, 2, 3])
@pytest.mark.parametrize("full", [True, False])
def test_model_is_the_cropped_binned_diffraction_pattern(orc, fb, n, b, full):
    """detector4d_model of Psi = FFT_row(psi) / N is diffractionPattern (|FFT2 psi|^2 / N^2 in the fftshift frame),
    cropped to the centred window and binned."""
    if full:
        q = n - n % b if (n - n % b - n) % 2 == 0 else n - n % b - b
        if q < 1 or (n - q) % 2:
            pytest.skip("no full-size window of this parity and bin")
    else:
        try:
            q = fb.stem_4d_side(n, 0, b) * b
        except fb.FdesError:
            assert n % 2 == 1 and b % 2 == 0
            pytest.skip("no admissible default window")
    rng = np.random.default_rng(100 * n + b)
    psi = (rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))).astype(np.complex64)
    p = types.SimpleNamespace(doBeamTilt=False, mode=2, m1=n, m2=n)
    want = _crop_bin(orc.diffraction_pattern(psi, p, 0), q, b)
    Psi = sm.fft_rows(psi) / n
    out0 = rng.random((1, q // b, q // b))
    got = detector4d_model(Psi[None], np.ones(n, bool), q, b, 0.5, out0)
    np.testing.assert_allclose(got[0], out0[0] + 0.5 * want, rtol=2e-5, atol=2e-6 * np.abs(want).max())


@pytest.mark.parametrize("n", [8, 9, 64, 143, 320, 512, 600, 1000, 1022, 4096, 8192])
def test_default_window_holds_the_band_limit(orc, fb, n):
    p = types.SimpleNamespace(m1=n, m2=n)
    keep = orc.band_mask(p)
    for b in (1, 2, 3, 4):
        try:
            q = fb.stem_4d_side(n, 0, b) * b
        except fb.FdesError as e:
            assert n % 2 == 1 and b % 2 == 0, (n, b, str(e))
            assert "parity" in str(e)
            continue
        assert (n - q) % 2 == 0 and q % b == 0 and 1 <= q <= n
        # every kept frequency lands inside the window of the fftshifted grid
        o = (n - q) // 2
        shifted = np.roll(keep, (n // 2, n // 2), axis=(0, 1))
        assert shifted[o:o + q, o:o + q].sum() == keep.sum(), (n, b, q)
        # and it is the smallest such window: two pixels less loses a kept frequency (or breaks the bin)
        if q - 2 * b >= 1 or q - 2 >= 1:
            smaller = [s for s in range(q - 2, 0, -2) if s % b == 0][:1]
            for s in smaller:
                o2 = (n - s) // 2
                assert shifted[o2:o2 + s, o2:o2 + s].sum() < keep.sum(), (n, b, s)


def test_frequency_of_window_pixels(fb):
    """window pixel q holds frequency q - Q//2: the zero frequency sits at [Q//2][Q//2]"""
    for n in (8, 9, 64, 143):
        for q in range(n % 2 or 2, n + 1, 2):
            o = (n - q) // 2
            idx = np.roll(np.arange(n), n // 2)[o:o + q]         # unshifted index at window pixel
            freq = np.where(idx > n // 2, idx - n, idx)
            assert freq[q // 2] == 0
            if n % 2 or q < n:
                np.testing.assert_array_equal(freq, np.arange(q) - q // 2)


@pytest.mark.parametrize("n, window, b, why", [
    (9, 0, 2, "parity"),          # odd grid, even bin: no odd window is a multiple of 2
    (8, 0, 5, "parity"),          # the band limit needs 6 of the 8 pixels; no even multiple of 5 up to 8
    (512, 511, 1, "parity"),
    (511, 300, 1, "parity"),
    (512, 300, 7, "multiple"),
    (512, 514, 1, "larger"),
    (512, -2, 1, ">= 0"),
    (512, 0, 0, "bin"),
])
def test_inadmissible_windows_are_refused(fb, n, window, b, why):
    with pytest.raises(fb.FdesError, match=why):
        fb.stem_4d_side(n, window, b)


def test_side_of_admissible_windows(fb):
    assert fb.stem_4d_side(512) == 342
    assert fb.stem_4d_side(512, 0, 2) == 171
    assert fb.stem_4d_side(512, 512, 4) == 128
    assert fb.stem_4d_side(143, 143, 11) == 13
    assert fb.stem_4d_side(9, 1, 1) == 1


def test_sweep_op_value(fb):
    assert fb.SWEEP_DETECTOR4D == 13
