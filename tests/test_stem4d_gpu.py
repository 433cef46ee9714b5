"""4D-STEM on the GPU: the 4D detector sweep (launch_detector4d_cols) through the C ABI test hook against a float64
model (detector4d_model below) at the fifteen grid sizes of test_sweeps_fp64_gpu.py, and the whole scan
(Simulation.stem_scan_4d) against the oracle's per-probe restatement of the reference, against the annular scan, across
pass sizes, sessions and GPUs, and from the command line.

Setting FDES_STEM4D_ERRORS=<file.json> records the errors of the per-sweep tests per size (the bounds below were set
from such a run).
"""
import json
import os
import subprocess

import numpy as np
import pytest

import sweep_model as sm
from conftest import DATA, ROOT, TOL_INTENSITY

pytestmark = pytest.mark.gpu

FAST = [64, 128, 256, 512, 1024, 2048, 4096, 320, 800, 1000]
GENERIC = [96, 250, 600, 1022, 143]
SIZES = FAST + GENERIC
B_ODD = 3
SENT_F = np.float32(-4321.75)


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


# Error of the sweep against the model: max |out - ref| / max |ref - out0| and the rel-L2 of out - ref against
# ref - out0, about three times the largest values over the fifteen sizes measured on an NVIDIA B200 (1000 W power
# limit): (measured peak, at size; measured global, at size)
MEASURED = (4.7e-7, 4096, 3.1e-7, 4096)       # both on the small window with bin 4
PEAK_TOL = 1.5e-6
GLOB_TOL = 1e-6
_ERRORS = {}


@pytest.fixture(scope="module", autouse=True)
def _record_errors():
    yield
    path = os.environ.get("FDES_STEM4D_ERRORS")
    if path:
        with open(path, "w") as f:
            json.dump(_ERRORS, f, indent=1, sort_keys=True)


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint32), np.ascontiguousarray(b).view(np.uint32))


def run(fb, n, batch, Psi, out0, q, b, weight):
    bufs = [np.ascontiguousarray(Psi).copy(), np.ascontiguousarray(out0).copy()]
    fb.sweep_test(fb.SWEEP_DETECTOR4D, n, batch, bufs, [q, b], [weight])
    return bufs[1]


def windows(fb, n, b):
    """default, full (the largest admissible) and small windows for bin b; those that do not exist are left out"""
    out = {}
    try:
        out["default"] = fb.stem_4d_side(n, 0, b) * b
    except fb.FdesError:
        pass
    full = [q for q in range(n, 0, -2) if q % b == 0]
    if full:
        out["full"] = full[0]
    small = [q for q in range(n % 2 or 2, n + 1, 2) if q % b == 0 and q >= 3 * b]
    if small:
        out["small"] = small[0]
    return out


@pytest.mark.parametrize("b", [1, 4])
@pytest.mark.parametrize("n", SIZES)
def test_detector4d_cols(fb, n, b):
    g = fb.sweep_geom(n)
    band = sm.band_columns(n, g["lo_end"], g["hi_start"])
    rng = np.random.default_rng(21000 + n + b)
    Psi = (rng.standard_normal((B_ODD, n, n)) + 1j * rng.standard_normal((B_ODD, n, n))).astype(np.complex64)
    Psi[:, :, 0] += np.float32(1.0)
    Psi[..., ~band] = np.nan                    # never read
    weight = np.float32(0.37)
    wins = windows(fb, n, b)
    if not wins:
        pytest.skip("no admissible window")
    for name, q in wins.items():
        s = q // b
        level = float(n) * b * b                # mean of a bin of |FFT_col(Psi)|^2
        out0 = np.concatenate([(rng.random(B_ODD * s * s) * level).astype(np.float32), np.full(8, SENT_F)])
        got_all = run(fb, n, B_ODD, Psi, out0, q, b, weight)
        assert (got_all[B_ODD * s * s:] == SENT_F).all(), f"{n} {name}: written past the batch"
        got = got_all[:B_ODD * s * s].reshape(B_ODD, s, s)
        assert not np.isnan(got).any(), f"{n} {name}: NaN (a band pixel not written, or a column outside the band read)"
        base = out0[:B_ODD * s * s].reshape(B_ODD, s, s)
        ref = detector4d_model(Psi, band, q, b, weight, base.astype(np.float64))
        add = ref - base
        peak = float(np.abs(got - ref).max() / np.abs(add).max())
        glob = float(np.linalg.norm(got - ref) / np.linalg.norm(add))
        d = _ERRORS.setdefault(str(n), {})
        d[f"{name} b{b}"] = {"peak": peak, "glob": glob}
        assert peak <= PEAK_TOL and glob <= GLOB_TOL, (n, name, b, peak, glob)
        if b == 1:
            # window columns outside the band: nothing added, out0 kept bit for bit
            o = (n - q) // 2
            idx = np.roll(np.arange(n), n // 2)[o:o + q]
            assert same_bits(got[:, :, ~band[idx]], base[:, :, ~band[idx]])
        # image b of the batch is the image run alone; a second launch gives the same bits
        k = B_ODD - 1
        one = run(fb, n, 1, Psi[k:k + 1], base[k].ravel(), q, b, weight)
        assert same_bits(one, got[k].ravel()), (n, name)
        assert same_bits(run(fb, n, B_ODD, Psi, out0, q, b, weight), got_all), (n, name)


def test_detector4d_refuses_bad_windows(fb):
    Psi = np.zeros((1, 64, 64), np.complex64)
    out = np.zeros(64 * 64, np.float32)
    for q, b in ((0, 1), (63, 1), (66, 1), (62, 4), (64, 0)):
        with pytest.raises(fb.FdesError):
            fb.sweep_test(fb.SWEEP_DETECTOR4D, 64, 1, [Psi, out], [q, b], [1.0])


# ---------------------------------------------------------------------------------------------
# the whole scan
# ---------------------------------------------------------------------------------------------
def _oracle_4d(orc, p, Z, xyz_list, occ, pos, q, b):
    """The reference algorithm per probe (mode 2, atoms translated by -r_p, whole-pixel positions), its diffraction
    pattern fftshifted, cropped to the centred window and binned, averaged over the configurations."""
    ps = p.copy()
    orc.set_sub_slices(ps, orc.sub_slice_ratio(ps.d3, ps.subSlTh))
    mask = orc.band_mask(ps)
    P = orc.fresnel_propagator(ps, mask)
    Zl = orc.list_of_elements(Z)
    n = ps.m1
    o, s = (n - q) // 2, q // b
    out = np.zeros((len(pos), s, s), np.float64)
    for xyz in xyz_list:
        for i, (px, py) in enumerate(pos):
            shifted = xyz.copy()
            shifted[:, 0] -= np.float32(px)
            shifted[:, 1] -= np.float32(py)
            psi = orc.incoming_wave(ps, 0, mask)
            bins = orc.bin_atoms(shifted, ps)
            for sl in range(ps.m3):
                V = orc.phase_grating(sl, Z, Zl, shifted, occ, ps.imPot, ps, bins)
                psi = orc.forward_propagation(psi, V, ps, P, mask)
            I = orc.diffraction_pattern(psi, ps, 0, mask).astype(np.float64)[o:o + q, o:o + q]
            out[i] += I.reshape(s, b, s, b).sum(axis=(1, 3)) / len(xyz_list)
    return out


def _specimen_128(fb, tmp_path, frozen):
    from fdes_b200 import specimens
    N, d = 128, 0.25e-10
    atoms = specimens.random_slab(40, N * d * 0.55, 4 * 2e-10, seed=11, species=(79, 14, 8))
    cnf = tmp_path / "stem.cnf"
    specimens.write_cnf(cnf, image_size=N, border_size=0, slices=4, pixel_size=d, slice_thickness=2e-10, atoms=atoms,
                        voltage=200e3, mode=2, objective_aperture=12e-3, frozen_phonons=frozen,
                        aberrations={"C1": (-2e-8, 0.0), "C3": (2e-4, 0.0)})
    return cnf, atoms, d


def _configs(orc, cnf, frozen):
    p, Z, xyz, dwf, occ = orc.read_cnf(str(cnf))
    if frozen:
        x = orc.Xorwow(1, 3 * len(Z))
        return p, Z, [orc.atom_jitter(xyz, dwf, x) for _ in range(frozen)], occ
    return p, Z, [xyz], occ


DET = np.array([[0, 10], [10, 25], [25, 45]], np.float32)


@pytest.mark.parametrize("frozen", [0, 2])
def test_stem_scan_4d_against_oracle(frozen, fb, orc, tmp_path):
    cnf, atoms, d = _specimen_128(fb, tmp_path, frozen)
    pos = np.array([[0, 0], [3, -5], [-7, 2], [12, 9]], np.float32) * np.float32(d)
    p, Z, xyz_list, occ = _configs(orc, cnf, frozen)
    with fb.Simulation(cnf, batch=3) as sim:
        for b in (1, 2):
            got, sig, ms = sim.stem_scan_4d(pos, bin=b)
            q = fb.stem_4d_side(128, 0, b) * b
            want = _oracle_4d(orc, p, Z, xyz_list, occ, pos, q, b)
            assert got.shape == want.shape and sig is None and ms > 0
            np.testing.assert_allclose(got, want, rtol=TOL_INTENSITY, atol=1e-4 * want.max())


@pytest.mark.parametrize("N", [320, 800, 1000, 600])
def test_stem_scan_4d_non_power_of_two_grids(N, fb, orc, tmp_path):
    from fdes_b200 import specimens
    d = 0.25e-10
    atoms = specimens.random_slab(30, N * d * 0.5, 2 * 2e-10, seed=N, species=(79, 14))
    cnf = specimens.write_cnf(tmp_path / "stem.cnf", image_size=N, border_size=0, slices=2, pixel_size=d,
                              slice_thickness=2e-10, atoms=atoms, voltage=200e3, mode=2, objective_aperture=10e-3)
    pos = np.array([[0, 0], [5, -3]], np.float32) * np.float32(d)
    with fb.Simulation(cnf, batch=2) as sim:
        got, _, _ = sim.stem_scan_4d(pos)
    p, Z, xyz, dwf, occ = orc.read_cnf(str(cnf))
    want = _oracle_4d(orc, p, Z, [xyz], occ, pos, fb.stem_4d_side(N), 1)
    np.testing.assert_allclose(got, want, rtol=TOL_INTENSITY, atol=1e-4 * want.max())


def _ring_masks(n, d, lam, det):
    """ring membership [ndet][ky][kx] of the fftshifted full grid, |k|^2 in float32 as the detector sweep forms it"""
    iw = np.roll(sm.signed_index(n), n // 2).astype(np.float32)
    il = np.float32(1) / (np.float32(n) * np.float32(d))
    k1 = (iw * il).astype(np.float32)
    ksq = (k1[None, :] * k1[None, :] + k1[:, None] * k1[:, None]).astype(np.float32)
    out = []
    for a, b in det:
        lo = (np.sin(np.float32(a * 1e-3)) / np.float32(lam)) ** 2
        hi = (np.sin(np.float32(b * 1e-3)) / np.float32(lam)) ** 2
        out.append((ksq >= np.float32(lo)) & (ksq < np.float32(hi)))
    return out


@pytest.mark.parametrize("frozen", [0, 2])
def test_annular_signals_and_ring_sums(frozen, fb, tmp_path):
    cnf, atoms, d = _specimen_128(fb, tmp_path, frozen)
    pos = np.array([[0, 0], [3, -5], [-7, 2], [12, 9], [1, 1]], np.float32) * np.float32(d)
    with fb.Simulation(cnf, batch=2) as sim:
        ref, _ = sim.stem_scan(pos, DET)
        pat, sig, _ = sim.stem_scan_4d(pos, window=128, bin=1, detectors_mrad=DET)
        lam, d1 = sim.lam, sim.d1
    assert same_bits(sig, ref), "annular signals differ from stem_scan"
    for r, m in enumerate(_ring_masks(128, d1, lam, DET)):
        np.testing.assert_allclose(pat[:, m].astype(np.float64).sum(axis=1), ref[:, r], rtol=1e-5, atol=1e-6 * ref.max())
    # empty specimen, default window: the whole pattern is n1 * n2
    a0 = np.ascontiguousarray(atoms, np.float32)
    a0[:, 3] = 1e-6
    with fb.Simulation(cnf, atoms6=a0) as sim:
        pat, _, _ = sim.stem_scan_4d(pos[:2])
    np.testing.assert_allclose(pat.astype(np.float64).sum(axis=(1, 2)), 128 * 128, rtol=1e-5)


def test_passes_batches_and_sessions_are_bit_identical(fb, tmp_path):
    cnf, atoms, d = _specimen_128(fb, tmp_path, 2)
    rng = np.random.default_rng(3)
    pos = (rng.integers(-10, 10, (7, 2)) * d).astype(np.float32)
    with fb.Simulation(cnf, batch=3) as sim:
        whole, sig, _ = sim.stem_scan_4d(pos, bin=2, detectors_mrad=DET)
        again, sig2, _ = sim.stem_scan_4d(pos, bin=2, detectors_mrad=DET)
        mm = np.memmap(tmp_path / "scan.f32", np.float32, "w+", shape=whole.shape)
        ret, _, _ = sim.stem_scan_4d(pos, bin=2, out=mm)
        assert ret is mm
        mm.flush()
        part, psig, _ = sim.stem_scan_4d(pos[2:5], bin=2, detectors_mrad=DET)
    with fb.Simulation(cnf, batch=2) as sim:
        passes, sig3, _ = sim.stem_scan_4d(pos, bin=2, detectors_mrad=DET, probes_per_pass=3)
    assert same_bits(again, whole) and same_bits(sig2, sig)
    assert same_bits(np.fromfile(tmp_path / "scan.f32", np.float32).reshape(whole.shape), whole)
    assert same_bits(part, whole[2:5]) and same_bits(psig, sig[2:5])
    assert same_bits(passes, whole) and same_bits(sig3, sig)
    with fb.Simulation(cnf) as sim:
        with pytest.raises(fb.FdesError, match="out must be"):
            sim.stem_scan_4d(pos, out=np.zeros((7, 3, 3), np.float32))
        with pytest.raises(fb.FdesError, match="parity"):
            sim.stem_scan_4d(pos, window=127)


def _gpu_pairs():
    import torch
    return [[0, 0]] + ([[0, 1]] if torch.cuda.device_count() >= 2 else [])


def test_multi_gpu_replicas_and_config_shards(fb, tmp_path):
    pos = (np.stack(np.meshgrid(np.arange(3), np.arange(4), indexing="ij"), -1).reshape(-1, 2) - 1.0).astype(np.float32) * 2e-11
    det = np.array([[0.0, 30.0], [30.0, 300.0]], np.float32)
    cnf = str(DATA / "cbed64.cnf")                 # no phonons: probes dealt out (replicas)
    with fb.Simulation(cnf, batch=4) as sim:
        ref, rsig, _ = sim.stem_scan_4d(pos, detectors_mrad=det, probes_per_pass=5)
    fcnf, _, _ = _specimen_128(fb, tmp_path, 2)    # two configurations: sharded over the devices
    fpos = pos[:5] * np.float32(5)
    with fb.Simulation(fcnf, batch=2) as sim:
        fref, fsig, _ = sim.stem_scan_4d(fpos, detectors_mrad=DET)
    for gpus in _gpu_pairs():
        with fb.Simulation(cnf, batch=4, gpus=gpus) as sim:
            assert sim.num_gpus == 2
            got, sig, ms = sim.stem_scan_4d(pos, detectors_mrad=det, probes_per_pass=5)
        assert ms > 0 and same_bits(got, ref) and same_bits(sig, rsig), gpus
        with fb.Simulation(fcnf, batch=2, gpus=gpus) as sim:
            assert sim.num_gpus == 2
            got, sig, _ = sim.stem_scan_4d(fpos, detectors_mrad=DET, probes_per_pass=2)
        np.testing.assert_allclose(got, fref, rtol=2e-6, atol=1e-7 * fref.max())
        np.testing.assert_allclose(sig, fsig, rtol=2e-6, atol=0)


def test_cli_stem_4d(fb, tmp_path):
    for f in ("stem128.qsc", "sto.cfg"):
        (tmp_path / f).write_text((DATA / f).read_text())
    exe = ROOT / "fdes_b200" / "bin" / "FDES"
    base = [str(exe), "--input_name", "stem128.qsc", "--stem_scan"]
    r = subprocess.run(base + ["--image_name", "plain.bin"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-500:]
    r = subprocess.run(base + ["--image_name", "with4d.bin", "--stem_4d", "scan4d.bin", "--stem_4d_bin", "2"], cwd=tmp_path,
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-500:]
    assert (tmp_path / "plain.bin").read_bytes() == (tmp_path / "with4d.bin").read_bytes()
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        xy, det = fb.qsc_scan(tmp_path / "stem128.qsc")
        with fb.Simulation(tmp_path / "stem128.qsc", batch=37) as sim:
            want, _, _ = sim.stem_scan_4d(xy.reshape(-1, 2), bin=2)
            side = fb.stem_4d_side(sim.m1, 0, 2)
    finally:
        os.chdir(cwd)
    raw = np.fromfile(tmp_path / "scan4d.bin", np.float32)
    assert raw.size == xy.shape[0] * xy.shape[1] * side * side
    assert same_bits(raw.reshape(xy.shape[0], xy.shape[1], side, side), want.reshape(xy.shape[0], xy.shape[1], side, side))
    r = subprocess.run(base + ["--stem_4d", "x.bin", "--stem_4d_bin", "0"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode != 0 and "bin" in r.stderr
