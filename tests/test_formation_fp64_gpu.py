"""The launchers of the image formation and of the STEM scan, run once through the C ABI test hook
(fdes_b200_sweep_test) and compared with the float64 models of oracle/sweep_model.py at the fifteen grid sizes of
test_sweeps_fp64_gpu.py: the ten register-resident sizes and five of the generic sweeps (odd 143 included).

* rows (launch_rows_fft): both directions with every epilogue (store, accumulation onto non-zero outputs, intensity
  accumulation, fftshift store, real crop), band-limited input (NaN outside the band) and output (exact zeros
  there), real input, the in-place store, crop windows on and next to the row boundaries of a CTA;
* columns (launch_cols_fft): the plain transform in both directions and the real-table filter (MTF, spatial
  incoherence) with a random non-symmetric table, out of place and in place;
* the probe sweep (launch_probe_cols): shifts 0, +-0.5, 0.4999, -0.4567, 1.37 and random ones, one per batch slot;
* the detector sweep (launch_detector_cols): box lengths whose reciprocals are exact powers of two, so that every
  pixel's |k|^2 is exact in float32 and ring bounds can sit on attainable values; eight overlapping rings, an empty
  one, k = 0 alone, everything (Parseval), the band edge, an anisotropic grid, and a grid with inexact |k|^2.

Checks: (a) per line (row of a row sweep, column of a column sweep) ||err||_2 <= TAU * rms(ref) * sqrt(L) and a
global rel-L2 bound; (b) NaN in everything a launcher must not read, sentinels in everything it must not write (an
extra image or row past the output), exact zeros where it must write them; (c) image b of a batch is bitwise the
image run alone; (d) two launches agree bitwise.

Setting FDES_FORMATION_ERRORS=<file.json> records the errors of a run per op and size (the bounds below were set
from such a run).
"""
import json
import os

import numpy as np
import pytest

import sweep_model as sm

pytestmark = pytest.mark.gpu

FAST = [64, 128, 256, 512, 1024, 2048, 4096, 320, 800, 1000]
GENERIC = [96, 250, 600, 1022, 143]
SIZES = FAST + GENERIC
PIPELINED = [512, 1024, 2048, 4096]
B_ODD = 3
SENT = np.complex64(complex(1234.5, -777.25))
SENT_F = np.float32(-4321.75)

# Bounds of the per-line metric ||err_line|| / (rms(ref) sqrt(L)) and of the global rel-L2 per op, about three times
# the largest value over all fifteen sizes measured on an NVIDIA B200 (1000 W power limit); the run of this file
# there took 3.8 min.  op: (measured line, at size; measured global, at size) -> bounds in TAU / GLOB
MEASURED = {
    "rows": (2.2e-7, 143, 1.4e-7, 143),
    "cols": (2.3e-7, 143, 1.9e-7, 4096),
    "probe": (2.5e-7, 96, 1.9e-7, 1000),     # before the phase was reduced per product: 1.6e-5 (64) .. 5.7e-4 (4096)
}
TAU = {"rows": 7e-7, "cols": 7e-7, "probe": 8e-7}
GLOB = {"rows": 4.5e-7, "cols": 6e-7, "probe": 6e-7}
DET_TAU = 3.5e-6        # |out - ref| / (|out0| + weight * ring sum); measured 1.2e-6 (4096)
_ERRORS = {}            # this run's errors (FDES_FORMATION_ERRORS)


@pytest.fixture(scope="module", autouse=True)
def _record_errors():
    yield
    path = os.environ.get("FDES_FORMATION_ERRORS")
    if path:
        with open(path, "w") as f:
            json.dump(_ERRORS, f, indent=1, sort_keys=True)


def record(op, n, **vals):
    d = _ERRORS.setdefault(op, {}).setdefault(str(n), {})
    for k, v in vals.items():
        d[k] = max(float(v), d.get(k, 0.0))


@pytest.fixture(scope="module")
def fbm():
    import fdes_b200
    return fdes_b200


_GEOM = {}


def geom(fb, n):
    if n not in _GEOM:
        _GEOM[n] = fb.sweep_geom(n)
    return _GEOM[n]


def band_of(fb, n):
    g = geom(fb, n)
    return sm.band_columns(n, g["lo_end"], g["hi_start"])


def row_cta_rows(fb, n):
    """Rows per CTA of the row sweeps: RowCfg<N>::RPB of sweep_kernels.cuh, one row on the generic sweeps."""
    e = geom(fb, n)["line_points"]
    if e == 0:
        return 1
    t = n // e
    return 4 if t & (t - 1) else max(128 // t, 1)


def crand(rng, shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)


def check_lines(op, n, out, ref, cols=None, rows_axis=True):
    """(a): per-line and global error of out against ref over the columns `cols` (all if None); lines are rows
    (rows_axis) or columns."""
    out = np.asarray(out)
    ref = np.asarray(ref)
    if cols is not None:
        out, ref = out[..., cols], ref[..., cols]
    assert not np.isnan(out).any(), f"{op} {n}: NaN in the output"
    err = out.astype(np.complex128) - ref
    rms = np.sqrt(np.mean(np.abs(ref) ** 2))
    if rows_axis:
        per, L = np.linalg.norm(err, axis=-1), err.shape[-1]
    else:
        per, L = np.linalg.norm(err, axis=-2), err.shape[-2]
    line = float(per.max() / (rms * np.sqrt(L)))
    glob = float(np.linalg.norm(err) / np.linalg.norm(ref))
    record(op, n, line=line, glob=glob)
    assert line <= TAU[op], f"{op} {n}: per-line error {line:.3e}"
    assert glob <= GLOB[op], f"{op} {n}: global rel-L2 {glob:.3e}"


def run(fb, op, n, batch, bufs, iargs=(), fargs=()):
    """Launch on copies; returns the buffers after the launch."""
    cp = [np.ascontiguousarray(b).copy() for b in bufs]
    fb.sweep_test(op, n, batch, cp, iargs, fargs)
    return cp


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint32), np.ascontiguousarray(b).view(np.uint32))


NONE = np.zeros(0, np.complex64)      # a buffer the launch does not use


# ---------------------------------------------------------------------------------------------------
# rows
# ---------------------------------------------------------------------------------------------------
# name: (dir, epilogue, options); options: real (in_is_real), band_in (NaN outside the band), band_out, in_place
ROW_CASES = {
    "store_fwd": (-1, sm.ROW_STORE, ()),
    "store_inv": (1, sm.ROW_STORE, ()),
    "accum_fwd": (-1, sm.ROW_ACCUM, ()),
    "accum_inv": (1, sm.ROW_ACCUM, ()),
    "intens_fwd": (-1, sm.ROW_INTENS_ACCUM, ()),
    "intens_inv": (1, sm.ROW_INTENS_ACCUM, ()),
    "shift_fwd": (-1, sm.ROW_STORE_SHIFT, ()),
    "shift_inv": (1, sm.ROW_STORE_SHIFT, ()),
    "crop_fwd": (-1, sm.ROW_CROP_REAL, ()),
    "crop_inv": (1, sm.ROW_CROP_REAL, ()),
    "band_in": (1, sm.ROW_STORE, ("band_in",)),
    "band_out": (-1, sm.ROW_STORE, ("band_out",)),
    "real_in": (-1, sm.ROW_STORE, ("real",)),
    "in_place_band_out": (-1, sm.ROW_STORE, ("in_place", "band_out")),
    "in_place_fwd": (-1, sm.ROW_STORE, ("in_place",)),
    "in_place_inv": (1, sm.ROW_STORE, ("in_place",)),
}
ROW_SCALE = np.float32(0.6180339)


def crop_windows(fb, n):
    """(dn1, dn2, n1, n2): dn1 != dn2 and n1 != n2 on the row boundaries of a CTA; one row either side of them; a
    1-pixel border; the last CTA's rows."""
    r = row_cta_rows(fb, n)
    return [(3, r, n - 7, 2 * r), (n // 4 + 1, r - 1 if r > 1 else 1, n // 2, r + 2), (1, 1, n - 2, n - 2),
            (0, n - r, n, r)]


def rows_launch(fb, n, batch, x, out0, dir, epi, opts, crop=(0, 0, 0, 0)):
    ia = [dir, epi, int("real" in opts), int("band_in" in opts), int("band_out" in opts), *crop,
          int("in_place" in opts)]
    if "in_place" in opts:
        return run(fb, fb.SWEEP_ROWS_FFT, n, batch, [x, NONE], ia, [ROW_SCALE])[0]
    return run(fb, fb.SWEEP_ROWS_FFT, n, batch, [x, out0], ia, [ROW_SCALE])[1]


def rows_inputs(rng, n, epi, opts, band, crop):
    """Input and output buffers of a row case: the output holds one image (crop: row) of sentinels past the
    batch; accumulating epilogues start from non-zero outputs."""
    if "real" in opts:
        x = rng.standard_normal((B_ODD, n, n)).astype(np.float32)
    else:
        x = crand(rng, (B_ODD, n, n))
    if "band_in" in opts:
        x[..., ~band] = np.nan
    if epi == sm.ROW_ACCUM:
        out0 = np.concatenate([crand(rng, (B_ODD, n, n)) * np.float32(np.sqrt(n)), np.full((1, n, n), SENT)])
    elif epi == sm.ROW_INTENS_ACCUM:
        out0 = np.concatenate([(rng.random((B_ODD, n, n)) * n).astype(np.float32), np.full((1, n, n), SENT_F)])
    elif epi == sm.ROW_CROP_REAL:
        out0 = np.full(B_ODD * crop[2] * crop[3] + crop[2], SENT_F)
    else:
        out0 = np.full((B_ODD + 1, n, n), SENT, np.complex64)
    return x, out0


def check_rows_case(fb, n, dir, epi, opts, crop, seed):
    rng = np.random.default_rng(seed)
    band = band_of(fb, n)
    x, out0 = rows_inputs(rng, n, epi, opts, band, crop)
    out = rows_launch(fb, n, B_ODD, x, out0, dir, epi, opts, crop)
    ref = sm.rows_fft(x, dir, epi, float(ROW_SCALE), out0[:B_ODD] if epi in (sm.ROW_ACCUM, sm.ROW_INTENS_ACCUM) else None,
                      band if "band_in" in opts else None, band if "band_out" in opts else None, crop)
    if epi == sm.ROW_CROP_REAL:
        win = B_ODD * crop[2] * crop[3]
        assert (out[win:] == SENT_F).all(), "crop written past its window"
        got = out[:win].reshape(B_ODD, crop[3], crop[2])
    elif "in_place" in opts:
        got = out
    else:
        assert (out[B_ODD] == out0[B_ODD]).all(), "written past the batch"
        got = out[:B_ODD]
    check_lines("rows", n, got, ref)
    if "band_out" in opts:
        assert (got[..., ~band] == 0).all()
    # (c) the last image alone
    b = B_ODD - 1
    if epi == sm.ROW_CROP_REAL:
        one = rows_launch(fb, n, 1, x[b:b + 1], out0[:crop[2] * crop[3]], dir, epi, opts, crop)
    else:
        one = rows_launch(fb, n, 1, x[b:b + 1], out0[b:b + 1], dir, epi, opts, crop)
    assert same_bits(one.reshape(got[b].shape), got[b])
    # (d)
    assert same_bits(rows_launch(fb, n, B_ODD, x, out0, dir, epi, opts, crop), out)


@pytest.mark.parametrize("case", list(ROW_CASES))
@pytest.mark.parametrize("n", SIZES)
def test_rows_fft(fbm, n, case):
    dir, epi, opts = ROW_CASES[case]
    crop = crop_windows(fbm, n)[0] if epi == sm.ROW_CROP_REAL else (0, 0, 0, 0)
    check_rows_case(fbm, n, dir, epi, opts, crop, 10000 + n + 37 * list(ROW_CASES).index(case))


@pytest.mark.parametrize("window", [1, 2, 3])
@pytest.mark.parametrize("n", SIZES)
def test_rows_crop_windows(fbm, n, window):
    """The final crop of the detector tail (an inverse transform) for the other windows of crop_windows."""
    check_rows_case(fbm, n, 1, sm.ROW_CROP_REAL, (), crop_windows(fbm, n)[window], 11000 + n + window)


def test_rows_refuses_bad_arguments(fbm):
    n = 128
    x = np.zeros((1, n, n), np.complex64)
    with pytest.raises(Exception, match="crop window outside the grid"):
        rows_launch(fbm, n, 1, x, np.zeros(n * n, np.float32), 1, sm.ROW_CROP_REAL, (), (1, 0, n, 1))
    with pytest.raises(Exception, match="in place only"):
        rows_launch(fbm, n, 1, x, NONE, 1, sm.ROW_ACCUM, ("in_place",))


# ---------------------------------------------------------------------------------------------------
# columns
# ---------------------------------------------------------------------------------------------------
COL_CASES = {      # name: (ColOp, dir, in place)
    "plain_fwd": (0, -1, False),
    "plain_inv": (0, 1, False),
    "plain_fwd_in_place": (0, -1, True),
    "plain_inv_in_place": (0, 1, True),
    "real_table": (2, -1, False),
    "real_table_in_place": (2, -1, True),
}


@pytest.mark.parametrize("case", list(COL_CASES))
@pytest.mark.parametrize("n", SIZES)
def test_cols_fft(fbm, n, case):
    op, dir, in_place = COL_CASES[case]
    rng = np.random.default_rng(12000 + n + 10 * list(COL_CASES).index(case))
    x = crand(rng, (B_ODD, n, n))
    # a random table [ky][kx]: far from symmetric, so a transposed read is an O(1) error
    tab = rng.random((n, n)).astype(np.float32) + np.float32(0.25) if op == fbm.COL_MUL_REAL_INV else np.zeros(0, np.float32)
    scale = np.float32(0.75 / n)
    out0 = np.full((B_ODD + 1, n, n), SENT, np.complex64)
    ia = [op, dir, int(in_place)]

    def launch(batch, xx, oo):
        bufs = run(fbm, fbm.SWEEP_COLS_FFT, n, batch, [xx, NONE if in_place else oo, tab], ia, [scale])
        return bufs[0] if in_place else bufs[1]

    out = launch(B_ODD, x, out0)
    if op == fbm.COL_MUL_REAL_INV:
        ref = sm.cols_mul_real_inv(x, tab, float(scale))
    else:
        ref = sm.cols_plain(x, dir, float(scale))
    if not in_place:
        assert (out[B_ODD] == SENT).all(), "written past the batch"
        out = out[:B_ODD]
    check_lines("cols", n, out, ref, rows_axis=False)
    b = B_ODD - 1
    assert same_bits(launch(1, x[b:b + 1], out0[b:b + 1]).reshape(n, n), out[b])
    again = launch(B_ODD, x, out0)
    assert same_bits(again if in_place else again[:B_ODD], out)


# ---------------------------------------------------------------------------------------------------
# probe
# ---------------------------------------------------------------------------------------------------
def probe_shifts(name):
    if name == "edges":
        s = [(0.0, 0.0), (0.5, -0.5), (-0.5, 0.4999)]
    elif name == "large":
        s = [(0.4999, -0.4567), (1.37, -1.37), (-0.4567, 1.37)]
    else:
        s = np.random.default_rng(13000).uniform(-0.5, 0.5, (B_ODD, 2))
    return np.asarray(s, np.float32)


@pytest.mark.parametrize("shifts", ["edges", "large", "random"])
@pytest.mark.parametrize("n", SIZES)
def test_probe_cols(fbm, n, shifts):
    """Psi_b = (1/N) IFFT_col[PSI0 exp(-2 pi i (iw(kx) sx + iw(ky) sy))] on the band columns; the Nyquist row (and
    column where it is a band column) take part; columns outside the band keep their sentinel."""
    rng = np.random.default_rng(14000 + n)
    band = band_of(fbm, n)
    PSI0 = crand(rng, (1, n, n))
    PSI0[..., ~band] = np.nan                   # not read
    sh = probe_shifts(shifts)
    Psi0 = np.full((B_ODD + 1, n, n), SENT, np.complex64)
    out = run(fbm, fbm.SWEEP_PROBE, n, B_ODD, [Psi0, PSI0, sh])[0]
    ref = sm.probe_cols(PSI0[0], sh, band)
    assert (out[B_ODD] == SENT).all(), "written past the batch"
    assert (out[:B_ODD][..., ~band] == SENT).all(), "columns outside the band written"
    check_lines("probe", n, out[:B_ODD], ref, cols=band, rows_axis=False)
    b = B_ODD - 1
    one = run(fbm, fbm.SWEEP_PROBE, n, 1, [Psi0[:1], PSI0, sh[b:b + 1]])[0]
    assert same_bits(one[0], out[b])
    assert same_bits(run(fbm, fbm.SWEEP_PROBE, n, B_ODD, [Psi0, PSI0, sh])[0], out)


# ---------------------------------------------------------------------------------------------------
# detector
# ---------------------------------------------------------------------------------------------------
J = 3


def exact_box(n, j):
    """A float32 pixel size d near 2^j / N with fl32(1 / fl32(N d)) == 2^-j."""
    d0 = np.float32(2.0 ** j / n)
    cands, up, down = [d0], d0, d0
    for _ in range(16):
        up, down = np.nextafter(up, np.float32(np.inf)), np.nextafter(down, np.float32(0))
        cands += [up, down]
    for d in cands:
        if sm.inv_length(n, d) == np.float32(2.0 ** -j):
            return d
    raise AssertionError(f"no float32 d near 2^{j}/{n} with an exact reciprocal box length")


def band_edge(fb, n):
    """Largest |iw(kx)| of a band column."""
    g = geom(fb, n)
    return max(g["lo_end"] - 1, n - g["hi_start"]) if g["lo_end"] < g["hi_start"] else n // 2


def ring_values(ksq, band):
    return np.unique(ksq[:, band])


def exact_rings(fb, n, aniso):
    """Eight rings [in2, out2) of exact |k|^2 values in units of 4^-J (isotropic: i1^2 + i2^2) or 4^-(J+1) (d2 = 2 d1:
    4 i1^2 + i2^2), most bounds on attainable values."""
    a = 4 if aniso else 1                   # weight of i1^2
    e = band_edge(fb, n)
    q = n // 4
    rings = [
        (0, 1),                             # k = 0 alone
        (1, a + 1),                         # the nearest pixels: 1 attainable, a + 1 = (1, 1) excluded
        (25, 25 + a * 25),                  # (0, 5) .. (5, 5) excluded
        (a * 25, a * 25),                   # empty
        (0, 4 * n * n),                     # everything
        (a * e * e, a * e * e + q * q),     # through the band-edge columns: (e, 0) included, (e, q) excluded
        (q * q, a * q * q + q * q),         # a wide ring overlapping the edge ring
        (1, 26),                            # overlapping the first ones
    ]
    return rings


def det_check(fb, n, Psi, band, in2, out2, d1, d2, seed, exact_bounds=()):
    rng = np.random.default_rng(seed)
    ndet = len(in2)
    weight = np.float32(0.37)
    out0 = np.concatenate([(rng.random(B_ODD * ndet) + 0.5).astype(np.float32), np.full(8, SENT_F)])
    fa = [d1, d2, weight, *in2, *out2]
    out = run(fb, fb.SWEEP_DETECTOR, n, B_ODD, [Psi, out0], [ndet], fa)[1]
    assert (out[B_ODD * ndet:] == SENT_F).all(), "written past the batch"
    il1, il2 = sm.inv_length(n, d1), sm.inv_length(n, d2)
    ksq = sm.detector_ksq(n, il1, il2)
    vals = ring_values(ksq, band)
    for v in exact_bounds:              # bounds on attainable |k|^2: a < / <= slip changes the ring
        assert np.isin(np.float64(v), vals), (n, v)
    base = out0[:B_ODD * ndet].reshape(B_ODD, ndet).astype(np.float64)
    ref = sm.detector_cols(Psi[:B_ODD], band, in2, out2, il1, il2, weight, base)
    got = out[:B_ODD * ndet].reshape(B_ODD, ndet)
    assert not np.isnan(got).any(), f"{n}: NaN in the detector output (a tile not summed, or a NaN column read)"
    err = np.abs(got - ref) / (np.abs(base) + np.abs(ref - base))
    record("detector", n, rel=err.max())
    assert err.max() <= DET_TAU, f"{n}: detector error {err.max():.3e}"
    empty = np.asarray(in2) == np.asarray(out2)
    assert same_bits(got[:, empty], out0[:B_ODD * ndet].reshape(B_ODD, ndet)[:, empty])
    b = B_ODD - 1
    one = run(fb, fb.SWEEP_DETECTOR, n, 1, [Psi[b:b + 1], out0[b * ndet:(b + 1) * ndet]], [ndet], fa)[1]
    assert same_bits(one, got[b])
    assert same_bits(run(fb, fb.SWEEP_DETECTOR, n, B_ODD, [Psi, out0], [ndet], fa)[1], out)
    return ref, base


def detector_psi(rng, n, band):
    Psi = crand(rng, (B_ODD, n, n))
    Psi[:, :, 0] += np.float32(1.0)         # a strong k = 0 term: the ring holding only k = 0 is not small
    Psi[..., ~band] = np.nan                # not read
    return Psi


@pytest.mark.parametrize("aniso", [False, True])
@pytest.mark.parametrize("n", SIZES)
def test_detector_cols_exact_rings(fbm, n, aniso):
    rng = np.random.default_rng(15000 + n + aniso)
    band = band_of(fbm, n)
    Psi = detector_psi(rng, n, band)
    d1 = exact_box(n, J)
    d2 = np.float32(2 * d1) if aniso else d1
    assert sm.inv_length(n, d2) == np.float32(2.0 ** -(J + 1 if aniso else J))
    unit = 4.0 ** -(J + 1 if aniso else J)
    rings = exact_rings(fbm, n, aniso)
    # i1^2 + i2^2 < 2^24 (4 i1^2 + i2^2 with d2 = 2 d1) on the band: every |k|^2 is exact in float32
    iw = sm.signed_index(n)
    assert (4 if aniso else 1) * int((iw[band] ** 2).max()) + (n // 2) ** 2 < 2 ** 24
    in2 = [np.float32(a * unit) for a, _ in rings]
    out2 = [np.float32(b * unit) for _, b in rings]
    exact = [in2[1], out2[1], in2[2], out2[2], in2[5], out2[5]]
    ref, base = det_check(fbm, n, Psi, band, in2, out2, d1, d2, 15500 + n, exact)
    # the ring covering everything holds Parseval's sum N sum |Psi|^2 over the band columns
    pars = n * (np.abs(Psi[:, :, band].astype(np.complex128)) ** 2).sum(axis=(-2, -1))
    np.testing.assert_allclose(ref[:, 4], base[:, 4] + float(np.float32(0.37)) * pars, rtol=1e-9)


@pytest.mark.parametrize("n", SIZES)
def test_detector_cols_inexact(fbm, n):
    """Pixel sizes without an exact reciprocal: |k|^2 rounds in float32, so the ring bounds sit in gaps of the
    attainable values at least 1e-6 relative wide."""
    rng = np.random.default_rng(16000 + n)
    band = band_of(fbm, n)
    Psi = detector_psi(rng, n, band)
    d1, d2 = np.float32(0.0123 * 1024 / n), np.float32(0.0157 * 1024 / n)
    ksq = sm.detector_ksq(n, sm.inv_length(n, d1), sm.inv_length(n, d2))
    vals = ring_values(ksq, band)

    def gap_bound(target):
        """the middle of the widest gap between attainable values in [0.9, 1.1] * target"""
        i0, i1 = np.searchsorted(vals, [0.9 * target, 1.1 * target])
        i = i0 + int(np.argmax(np.diff(vals[i0 - 1:i1 + 1])))
        lo, hi = vals[i - 1], vals[i]
        b = np.float32(0.5 * (lo + hi))
        assert (b - lo) > 1e-6 * b and (hi - b) > 1e-6 * b, (n, target, lo, hi)
        return b

    k1 = float(sm.inv_length(n, d1))
    targets = [0.5, 4.5, 30.5, 100.5]          # in units of k1^2: small radii, where the gaps are wide
    bounds = [gap_bound(t * k1 * k1) for t in targets]
    in2 = [np.float32(0), bounds[0], bounds[1], bounds[0], np.float32(0)]
    out2 = [bounds[0], bounds[2], bounds[3], bounds[3], np.float32(4 * float(vals[-1]))]
    det_check(fbm, n, Psi, band, in2, out2, d1, d2, 16500 + n)


def test_detector_refuses_bad_ring_count(fbm):
    n = 128
    Psi = np.zeros((1, n, n), np.complex64)
    for ndet in (0, 9):
        with pytest.raises(Exception, match="detectors"):
            run(fbm, fbm.SWEEP_DETECTOR, n, 1, [Psi, np.zeros(16, np.float32)], [ndet], [1.0] * 21)
