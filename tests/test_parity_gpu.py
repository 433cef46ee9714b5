"""GPU (B200): the CUDA library, called through its C ABI, against
  * the golden vectors recorded from the unmodified reference (tests/golden/),
  * the numpy oracle on the same inputs (small cases and the full-size 1024^2 configuration),
  * the reference itself run live on this box when oracle/_ref/ref_harness travelled with the repo,
  * size-independent properties at BASELINE.json's full sizes.
Bit-exact for integer work (bin indices, sort, phonon displacements); exit waves rel-L2 <= 1e-5
and intensities <= 1e-4 (north_star tolerances)."""
import ctypes
import os
import pathlib
import subprocess

import numpy as np
import pytest

from conftest import CASES, DATA, ROOT, TOL_INTENSITY, TOL_WAVE, golden, live_reference_missing, rel_l2

pytestmark = pytest.mark.gpu
HARNESS = ROOT / "oracle" / "_ref" / "ref_harness"


# ---------------------------------------------------------------------------------------------
# building blocks
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [64, 128, 256, 512, 1024, 2048, 4096, 320, 800, 1000,
                               8, 30, 96, 250, 600, 686, 1022, 1536, 2500])     # second line: generic run-time-N sweeps
def test_fft2d_against_numpy(n, fb):
    rng = np.random.default_rng(n)
    a = (rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))).astype(np.complex64)
    ref = np.fft.fft2(a.astype(np.complex128))
    got = fb.fft2d(a, -1)
    assert rel_l2(got, ref) < 2e-6
    back = fb.fft2d(got, +1) / (n * n)
    assert rel_l2(back, a) < 2e-6
    # linearity and a delta -> constant (exact)
    d = np.zeros((n, n), np.complex64)
    d[0, 0] = 1
    assert np.array_equal(fb.fft2d(d, -1), np.ones((n, n), np.complex64))


@pytest.mark.parametrize("n,nkeys", [(0, 10), (1, 1), (257, 3), (4096, 4096), (100_000, 70_000), (46208, 11 * 1024)])
def test_sort_records_is_stable_and_exact(n, nkeys, fb):
    rng = np.random.default_rng(n + nkeys)
    keys = rng.integers(0, nkeys + 1, n, dtype=np.uint32)      # key == nkeys marks rejected records
    cols = rng.integers(0, 1 << 20, n, dtype=np.int32)
    w = rng.standard_normal(n).astype(np.float32)
    k, c, ww, rp = fb.sort_records(keys, cols, w, nkeys)
    order = np.argsort(keys, kind="stable")
    np.testing.assert_array_equal(k, keys[order])
    np.testing.assert_array_equal(c, cols[order])
    np.testing.assert_array_equal(ww, w[order])
    np.testing.assert_array_equal(rp, np.searchsorted(keys[order], np.arange(nkeys + 1), side="left"))


@pytest.mark.parametrize("case", CASES)
def test_bins_jitter_and_potential(case, fb, orc):
    g, meta = golden(case)
    p, Z, xyz, dwf, occ = orc.read_cnf(str(DATA / f"{case}.cnf"))
    with fb.Simulation(DATA / f"{case}.cnf") as sim:
        ps = p.copy()
        orc.set_sub_slices(ps, orc.sub_slice_ratio(ps.d3, ps.subSlTh))
        assert (sim.m1, sim.m3, sim.nAt) == (ps.m1, ps.m3, len(Z))
        assert np.float32(sim.lam) == ps.lam and np.float32(sim.sigma) == ps.sigma
        # frozen-phonon displacements: same XORWOW streams as the reference -> bit-exact
        for j in range(max(1, p.frPh)):
            np.testing.assert_array_equal(sim.jitter_next(0), g["xyz_cfg"][j])
        xyz0 = g["xyz_cfg"][0]
        # integer bin tuples: bit-exact against the oracle's restatement of squareAtoms_d
        bins = sim.bin_atoms(xyz0)
        i1, i2, i3, _, _, ok = orc.bin_atoms(xyz0, ps)
        ok = ok & (i3 >= 0) & (i3 < ps.m3)
        np.testing.assert_array_equal(bins[:, 0] >= 0, ok)
        np.testing.assert_array_equal(bins[ok, 0], i1[ok])
        np.testing.assert_array_equal(bins[ok, 1], i2[ok])
        np.testing.assert_array_equal(bins[ok, 2], i3[ok])
        Zl = orc.list_of_elements(Z)
        np.testing.assert_array_equal(bins[:, 3], [Zl.index(z) for z in Z])
        for s in range(g["V"].shape[0]):
            V = sim.phase_grating(xyz0, s)
            if np.linalg.norm(g["V"][s]) > 0:
                assert rel_l2(V, g["V"][s]) < TOL_WAVE, s
            else:
                assert not V.any()
        psi = sim.exit_wave(xyz0, 0)
        assert rel_l2(psi, g["psi_exit"][0]) < TOL_WAVE


@pytest.mark.parametrize("case", CASES)
def test_full_run_against_reference_golden_and_oracle(case, fb, oracle_runs):
    g, meta = golden(case)
    with fb.Simulation(DATA / f"{case}.cnf", want_exitwave=True) as sim:
        img, ew = sim.simulate()
        assert sim.counters()["launches"] > 0
    assert rel_l2(ew, g["exitwave"]) < TOL_WAVE
    assert rel_l2(img, g["image"]) < TOL_INTENSITY
    res, _ = oracle_runs(case)
    assert rel_l2(ew, res.exitwave) < TOL_WAVE
    assert rel_l2(img, res.image) < TOL_INTENSITY


def test_runs_are_bit_reproducible(fb):
    """Sorted, segmented deposition instead of float atomics: two runs agree bit for bit (the
    reference does not, src/crystalMaker.cu:100-119)."""
    out = []
    for _ in range(2):
        with fb.Simulation(DATA / "phonon64.cnf", want_exitwave=True) as sim:
            out.append(sim.simulate())
    np.testing.assert_array_equal(out[0][0], out[1][0])
    np.testing.assert_array_equal(out[0][1], out[1][1])


@pytest.mark.parametrize("batch", [1, 2, 3])
def test_batching_does_not_change_results(batch, fb):
    with fb.Simulation(DATA / "phonon64.cnf", want_exitwave=True, batch=1) as a:
        ia, ea = a.simulate()
    with fb.Simulation(DATA / "phonon64.cnf", want_exitwave=True, batch=batch) as b:
        ib, eb = b.simulate()
    np.testing.assert_array_equal(ia, ib)
    np.testing.assert_array_equal(ea, eb)


@pytest.mark.parametrize("n", [128, 1024, 600])
def test_odd_slice_count_pairs_last_slices_of_two_configurations(n, fb, orc, tmp_path):
    """With an odd number of slices and an even batch the last slices of configurations 2j and 2j + 1 share one
    complex transform through S1 / S2 / S3 (real and imaginary part), instead of running as half-empty pairs:
    same result as batch 1 up to rounding, and parity with the oracle (3 species, absorptive, 5 slices,
    4 frozen-phonon configurations; 1024: TMA-pipelined sweeps, 600: generic sweeps)."""
    from fdes_b200 import specimens
    d = 0.2e-10
    atoms = specimens.random_slab(200, n * d, 5 * 2e-10, seed=n, species=(79, 14, 8))
    cnf = specimens.write_cnf(tmp_path / "odd.cnf", image_size=n // 2, border_size=n // 4, slices=5, pixel_size=d,
                              slice_thickness=2e-10, atoms=atoms, voltage=120e3, absorptive=0.03, frozen_phonons=4)
    out = {}
    for batch in (1, 2, 4):
        with fb.Simulation(cnf, want_exitwave=True, batch=batch) as sim:
            assert sim.m3 == 5
            out[batch] = sim.simulate()
    for batch in (2, 4):
        assert rel_l2(out[batch][1], out[1][1]) < 1e-6 and rel_l2(out[batch][0], out[1][0]) < 1e-6
    p, Z, xyz, dwf, occ = orc.read_cnf(str(cnf))
    res = orc.build_measurements(p, Z, xyz, dwf, occ)
    assert rel_l2(out[4][1], res.exitwave) < TOL_WAVE
    assert rel_l2(out[4][0], res.image) < TOL_INTENSITY


def test_rank_shards_sum_to_the_whole(fb, tmp_path):
    """rank/world sharding of the phonon configurations incl. the RNG positioning: for every
    measurement k the partial sums of (rank 0, rank 1) of 2 add up to the single-rank result (the
    XORWOW streams are consumed in the reference's global (k, j) order on every rank)."""
    import torch
    from fdes_b200 import specimens
    cnf = tmp_path / "ph2.cnf"
    atoms = specimens.random_slab(30, 64 * 0.25e-10 * 0.8, 4 * 2e-10, seed=3, species=(38, 22, 8))
    specimens.write_cnf(cnf, image_size=32, border_size=16, slices=4, pixel_size=0.25e-10, slice_thickness=2e-10,
                        atoms=atoms, frozen_phonons=3, image_size_z=2, defoci=[2e-9, -5e-9],
                        aberrations={"C3": (1e-3, 0.0)}, objective_aperture=0.02)
    with fb.Simulation(cnf, want_exitwave=True) as whole:
        ref = []
        for k in range(2):
            whole.run_k(k)
            ref.append(whole.finish_k(k))
    n = 64 * 64
    accI = torch.zeros(n, dtype=torch.float32, device="cuda")
    accE = torch.zeros(2 * n, dtype=torch.float32, device="cuda")
    parts = [fb.Simulation(cnf, want_exitwave=True, rank=r, world=2) for r in range(2)]
    try:
        for k in range(2):
            sumI = torch.zeros_like(accI)
            sumE = torch.zeros_like(accE)
            for part in parts:
                part.set_accumulators(accI.data_ptr(), accE.data_ptr())
                part.run_k(k)
                torch.cuda.synchronize()
                sumI += accI
                sumE += accE
            accI.copy_(sumI)
            accE.copy_(sumE)
            torch.cuda.synchronize()
            img_s, ew_s = parts[1].finish_k(k)
            assert rel_l2(ew_s, ref[k][1]) < 1e-6, k
            assert rel_l2(img_s, ref[k][0]) < 1e-6, k
    finally:
        for part in parts:
            part.close()


# ---------------------------------------------------------------------------------------------
# the drop-in boundary
# ---------------------------------------------------------------------------------------------
def test_FDES_drop_in_call(fb, orc, tmp_path, monkeypatch):
    """The exported FDES() with the argument meaning of src/FDESExport.cu:59-178: atoms from the
    caller's array (occupancy truncated to int, src/paramStructure.cu:323), image into the caller's
    buffer and into image_name as raw float32 [n3][n2][n1]."""
    monkeypatch.chdir(tmp_path)
    cnf = DATA / "tilt64.cnf"
    p, Z, xyz, dwf, occ = orc.read_cnf(str(cnf))
    atoms6 = np.column_stack([Z.astype(np.float32), xyz, dwf, occ]).astype(np.float32)
    dst = np.zeros((p.n3, p.n2, p.n1), np.float32)
    fb.cuda_FDES(0, 2, str(cnf), str(tmp_path / "M.bin"), str(tmp_path / "r.emd"), atoms6, len(atoms6), dst)
    res = orc.build_measurements(p, Z, xyz, dwf, np.trunc(occ).astype(np.float32))
    assert rel_l2(dst, res.image) < TOL_INTENSITY
    on_disk = np.fromfile(tmp_path / "M.bin", np.float32).reshape(dst.shape)
    np.testing.assert_array_equal(on_disk, dst)
    import h5min          # results file = EMD/HDF5 with the exit wave stored [m1][m2][n3][2] (src/rwHdf5.cu:248-267)
    ew = np.ascontiguousarray(h5min.File(tmp_path / "r.emd").root["data/exit_wave/data"].data.transpose(2, 1, 0, 3)).view(np.complex64)[..., 0]
    assert rel_l2(ew, res.exitwave) < TOL_WAVE
    assert (tmp_path / "dataFDES_used.cnf").exists()     # side-effect file of getParams (:629-631)


def test_cli_binary(orc, tmp_path, oracle_runs):
    exe = ROOT / "fdes_b200" / "bin" / "FDES"
    r = subprocess.run([str(exe), "--input_name", str(DATA / "sub128.cnf"), "--image_name", "out.bin",
                        "--print_level", "2"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-500:]
    res, _ = oracle_runs("sub128")
    img = np.fromfile(tmp_path / "out.bin", np.float32).reshape(res.image.shape)
    assert rel_l2(img, res.image) < TOL_INTENSITY
    import h5min
    f = h5min.File(tmp_path / "results.emd")
    ew = np.ascontiguousarray(f.root["data/exit_wave/data"].data.transpose(2, 1, 0, 3)).view(np.complex64)[..., 0]
    np.testing.assert_array_equal(f.root["data/images/data"].data.transpose(2, 1, 0), img)
    assert (tmp_path / "config.emd").exists()      # side-effect file of the CLI for .cnf / .qsc inputs (src/FDES.cu:229-232)
    assert rel_l2(ew, res.exitwave) < TOL_WAVE


def test_unsupported_inputs_fail_loudly(fb, tmp_path):
    from fdes_b200 import specimens
    cnf = specimens.write_cnf(tmp_path / "rect.cnf", image_size=40, border_size=12, slices=2, pixel_size=0.25e-10,
                              slice_thickness=2e-10, atoms=specimens.au_cuboctahedron(1))
    text = open(cnf).read().replace("image_size_y: 40", "image_size_y: 48")
    open(cnf, "w").write(text)
    with pytest.raises(fb.FdesError, match="non-square"):
        fb.Simulation(cnf)
    specimens.write_cnf(tmp_path / "tiny.cnf", image_size=3, border_size=1, slices=2, pixel_size=0.25e-10,
                        slice_thickness=2e-10, atoms=specimens.au_cuboctahedron(1))
    with pytest.raises(fb.FdesError, match="between 8 and 8192"):
        fb.Simulation(tmp_path / "tiny.cnf")
    with pytest.raises(fb.FdesError, match="cannot read"):
        fb.Simulation(tmp_path / "missing.cnf")


# ---------------------------------------------------------------------------------------------
# full size (BASELINE.json configs[1]: Si[001] 11k atoms, 1024^2, 2 A slices)
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def si1024(tmp_path_factory, fb):
    from fdes_b200 import specimens
    d = tmp_path_factory.mktemp("si1024")
    cnf = d / "si001_1024.cnf"
    specimens.config_si001_1024(cnf)
    with fb.Simulation(cnf, want_exitwave=True) as sim:
        img, ew = sim.simulate()
    return cnf, img, ew


def test_si1024_against_oracle(si1024, orc):
    cnf, img, ew = si1024
    p, Z, xyz, dwf, occ = orc.read_cnf(str(cnf))
    res = orc.build_measurements(p, Z, xyz, dwf, occ)
    assert rel_l2(ew, res.exitwave) < TOL_WAVE
    assert rel_l2(img, res.image) < TOL_INTENSITY


def test_si1024_against_live_reference(si1024, tmp_path):
    """Without the reference build (oracle/_ref/ref_harness) the comparison is test_si1024_against_oracle's."""
    cnf, img, ew = si1024
    if live_reference_missing(HARNESS):
        return
    out = tmp_path / "ref"
    subprocess.run([str(HARNESS), "run", str(cnf), str(out), "2"], check=True, capture_output=True)
    rimg = np.fromfile(out / "image.f32", np.float32).reshape(img.shape)
    rew = np.fromfile(out / "exitwave.f32", np.float32).view(np.complex64).reshape(ew.shape)
    assert rel_l2(ew, rew) < TOL_WAVE
    assert rel_l2(img, rimg) < TOL_INTENSITY


def test_si1024_properties(si1024, fb, orc, tmp_path):
    cnf, img, ew = si1024
    # elastic scattering without absorption only loses intensity through the 2/3 band limit
    n = ew.shape[-1] * ew.shape[-2]
    total = float(np.sum(np.abs(ew.astype(np.complex128)) ** 2)) / n
    assert 0.9 < total <= 1.0 + 1e-5
    # the specimen is mirror-symmetric in x <-> y about the grid centre up to the (fixed) structure
    # origin; a cheap invariant that needs no such assumption: the image is finite and positive
    assert np.isfinite(img).all() and img.min() > 0
    # empty specimen (all atoms outside the slab): the plane wave passes unchanged
    p, Z, xyz, dwf, occ = orc.read_cnf(str(cnf))
    atoms6 = np.column_stack([Z.astype(np.float32), xyz, dwf, occ]).astype(np.float32)
    atoms6[:, 3] = 1e-6
    with fb.Simulation(cnf, atoms6=atoms6, want_exitwave=True) as sim:
        img0, ew0 = sim.simulate()
    assert np.allclose(ew0, 1.0, atol=1e-5)
    assert np.allclose(img0, 1.0, atol=1e-4)


# ---------------------------------------------------------------------------------------------
# the other grid sizes of BASELINE.json: 2048^2 (Au cuboctahedron), 4096^2 (random slab, 3 species),
# 512^2 CBED probe (the per-probe unit of the STEM configuration)
# ---------------------------------------------------------------------------------------------
def _oracle_vs_library(cnf, fb, orc, atoms6=None):
    p, Z, xyz, dwf, occ = orc.read_cnf(str(cnf))
    if atoms6 is not None:
        Z, xyz, dwf, occ = atoms6[:, 0].astype(np.int32), atoms6[:, 1:4].copy(), atoms6[:, 4].copy(), atoms6[:, 5].copy()
    with fb.Simulation(cnf, atoms6=atoms6, want_exitwave=True) as sim:
        img, ew = sim.simulate()
    res = orc.build_measurements(p, Z, xyz, dwf, occ)
    assert rel_l2(ew, res.exitwave) < TOL_WAVE
    assert rel_l2(img, res.image) < TOL_INTENSITY
    return img, ew


@pytest.mark.parametrize("slices,mode", [(1, 0), (2, 0), (5, 0), (4, 1)])
def test_first_and_last_slice_shortcuts_match_the_plain_sweeps(fb, tmp_path, monkeypatch, slices, mode):
    """Plane wave: the first slice runs without S5 (S6 reads N * FFT_row(t) from the transmission stack); imaging
    mode without an exit wave to keep: the CTF rides on the last slice's S6.  Same images as the six plain sweeps
    per slice + the separate CTF sweep (FDES_B200_NO_FIRST_SLICE_SHORTCUT=1), 1024^2 = pipelined column sweeps;
    one slice = first and last at once."""
    from fdes_b200 import specimens
    d = 0.2e-10
    atoms = specimens.random_slab(300, 1024 * d, slices * 2e-10, seed=7 + slices, species=(79, 14))
    cnf = specimens.write_cnf(tmp_path / "fl.cnf", image_size=512, border_size=256, slices=slices, pixel_size=d,
                              slice_thickness=2e-10, atoms=atoms, voltage=120e3, absorptive=0.03, frozen_phonons=4, mode=mode,
                              objective_aperture=0.015, aberrations={"C1": (-2e-8, 0.0), "C3": (3e-4, 0.0)})
    out = {}
    for off in ("0", "1"):
        monkeypatch.setenv("FDES_B200_NO_FIRST_SLICE_SHORTCUT", off)
        with fb.Simulation(cnf, want_exitwave=False) as sim:       # no exit wave kept: the fused CTF path
            out[off, False] = sim.simulate()[0]
        with fb.Simulation(cnf, want_exitwave=True) as sim:        # exit wave kept: separate CTF sweep
            out[off, True] = sim.simulate()
    ref_img, ref_ew = out["1", True]
    assert np.isfinite(ref_img).all() and ref_img.mean() > 0.1
    assert rel_l2(out["0", True][1], ref_ew) < 2e-6
    for key in (("0", False), ("1", False)):
        assert rel_l2(out[key], ref_img) < 2e-6
    assert rel_l2(out["0", True][0], ref_img) < 2e-6


@pytest.mark.parametrize("n,dn,mode", [(41, 20, 0), (75, 0, 2), (101, 13, 1)])
def test_odd_grid_sizes_against_oracle(fb, orc, tmp_path, n, dn, mode):
    """Odd sample sizes (81, 75, 127 = prime): the run-time-N sweeps against the numpy oracle (the live
    reference covers odd sizes in test_random_grid_sizes_against_live_reference)."""
    from fdes_b200 import specimens
    m = n + 2 * dn
    d = 0.25e-10
    atoms = specimens.random_slab(60, m * d, 4 * 2e-10, seed=n, species=(79, 14))
    cnf = specimens.write_cnf(tmp_path / f"odd{m}.cnf", image_size=n, border_size=dn, slices=4, pixel_size=d,
                              slice_thickness=2e-10, atoms=atoms, voltage=200e3, mode=mode, absorptive=0.03,
                              objective_aperture=0.015, frozen_phonons=2 if mode == 0 else 0,
                              aberrations={"C1": (-1e-8, 0.0), "C3": (2e-4, 0.0)})
    img, ew = _oracle_vs_library(cnf, fb, orc)
    assert ew.shape[-1] == m


def test_au_2048_against_oracle(fb, orc, tmp_path):
    from fdes_b200 import specimens
    cnf = tmp_path / "au.cnf"
    specimens.config_au_2048(cnf, frozen_phonons=0)
    _oracle_vs_library(cnf, fb, orc)


def test_random_4096_against_oracle(fb, orc, tmp_path):
    from fdes_b200 import specimens
    cnf = tmp_path / "slab.cnf"
    atoms = specimens.random_slab(3000, 4096 * 0.1e-10, 5 * 2e-10)
    specimens.write_cnf(cnf, image_size=2048, border_size=1024, slices=5, pixel_size=0.1e-10, slice_thickness=2e-10,
                        atoms=atoms, voltage=200e3, absorptive=0.05)
    _oracle_vs_library(cnf, fb, orc)


@pytest.mark.parametrize("n,border,mode", [(320, 80, 0), (800, 200, 0), (1000, 170, 0), (320, 0, 2), (800, 100, 1),
                                           (600, 100, 0), (384, 64, 0), (250, 25, 2), (686, 43, 1), (146, 13, 0)])
def test_mixed_radix_grids_against_oracle(n, border, mode, fb, orc, tmp_path):
    """The 2^a 5^b grids of the reference's shipped examples (Au 320^2, SrTiO3 800^2, Si 1000^2:
    radix-5 passes, lines of 16 / 40 / 50 threads) and sizes without a register-resident instantiation,
    which run on the generic run-time-N sweeps (generic_sweeps.cu): 600 = 2^3 3 5^2, 384 = 2^7 3,
    250 = 2 5^3, 686 = 2 7^3, 146 = 2 * 73 (a radix-73 pass)."""
    from fdes_b200 import specimens
    cnf = tmp_path / f"g{n}.cnf"
    d = 0.2e-10
    atoms = specimens.random_slab(150, n * d, 5 * 2e-10, seed=n, species=(79, 14, 8))
    specimens.write_cnf(cnf, image_size=n - 2 * border, border_size=border, slices=5, pixel_size=d, slice_thickness=2e-10,
                        atoms=atoms, voltage=120e3, mode=mode, absorptive=0.03, objective_aperture=0.015,
                        frozen_phonons=2 if mode == 0 else 0, mtf=(0.58, 0.42, 2.7, 15.5),
                        aberrations={"C1": (-3e-8, 0.0), "C3": (5e-4, 0.0), "A1": (1e-9, 0.4)})
    _oracle_vs_library(cnf, fb, orc)


def test_srtio3_512_probe_against_oracle(fb, orc, tmp_path):
    """mode 2 (CBED probe at the grid centre): the per-probe unit of the STEM configuration."""
    from fdes_b200 import specimens
    cnf = tmp_path / "sto.cnf"
    atoms = specimens.srtio3_slab(4, 4, 8)
    specimens.write_cnf(cnf, image_size=512, border_size=0, slices=16, pixel_size=19.525e-10 / 512,
                        slice_thickness=1.9525e-10, atoms=atoms, voltage=200e3, mode=2, objective_aperture=20e-3)
    _oracle_vs_library(cnf, fb, orc)


# ---------------------------------------------------------------------------------------------
# STEM scan (extension): a scan position is the reference's mode-2 probe shifted periodically.  Oracle
# (SURVEY.md section 8c): the reference algorithm in mode 2 with every atom translated by -r_p, the
# detector an annular sum over the diffraction intensity before the detector tail.  Positions are
# whole pixels so that the bilinear deposition of the translated atoms is the same deposition.
# ---------------------------------------------------------------------------------------------
def _oracle_stem(orc, p, Z, xyz_list, occ, pos, det_mrad):
    ps = p.copy()
    orc.set_sub_slices(ps, orc.sub_slice_ratio(ps.d3, ps.subSlTh))
    mask = orc.band_mask(ps)
    P = orc.fresnel_propagator(ps, mask)
    Zl = orc.list_of_elements(Z)
    N = ps.m1
    kx = (orc.ow(N).astype(np.float32) / np.float32(N * ps.d1))[None, :]
    ky = (orc.ow(N).astype(np.float32) / np.float32(N * ps.d2))[:, None]
    ksq = (kx * kx + ky * ky).astype(np.float32)
    rings = [((np.sin(np.float32(a * 1e-3)) / ps.lam) ** 2, (np.sin(np.float32(b * 1e-3)) / ps.lam) ** 2) for a, b in det_mrad]
    out = np.zeros((len(pos), len(det_mrad)), np.float64)
    for xyz in xyz_list:
        for i, (px, py) in enumerate(pos):
            shifted = xyz.copy()
            shifted[:, 0] -= np.float32(px)
            shifted[:, 1] -= np.float32(py)
            psi = orc.incoming_wave(ps, 0, mask)
            bins = orc.bin_atoms(shifted, ps)
            for s in range(ps.m3):
                V = orc.phase_grating(s, Z, Zl, shifted, occ, ps.imPot, ps, bins)
                psi = orc.forward_propagation(psi, V, ps, P, mask)
            I = orc.diffraction_pattern(psi, ps, 0, mask).astype(np.float64)
            for d, (lo, hi) in enumerate(rings):
                out[i, d] += I[(ksq >= lo) & (ksq < hi)].sum() / len(xyz_list)
    return out


@pytest.mark.parametrize("frozen", [0, 2])
def test_stem_scan_against_oracle(frozen, fb, orc, tmp_path):
    from fdes_b200 import specimens
    N, d = 128, 0.25e-10
    rng = np.random.default_rng(7)
    atoms = specimens.random_slab(40, N * d * 0.55, 4 * 2e-10, seed=11, species=(79, 14, 8))   # central region only
    cnf = tmp_path / "stem.cnf"
    specimens.write_cnf(cnf, image_size=N, border_size=0, slices=4, pixel_size=d, slice_thickness=2e-10, atoms=atoms,
                        voltage=200e3, mode=2, objective_aperture=12e-3, frozen_phonons=frozen,
                        aberrations={"C1": (-2e-8, 0.0), "C3": (2e-4, 0.0)})
    pos_px = np.array([[0, 0], [3, -5], [-7, 2], [12, 9]], np.float32)
    pos = pos_px * np.float32(d)
    det = np.array([[0, 10], [10, 25], [25, 45]], np.float32)
    with fb.Simulation(cnf, batch=3) as sim:
        got, ms = sim.stem_scan(pos, det)
    p, Z, xyz, dwf, occ = orc.read_cnf(str(cnf))
    if frozen:
        x = orc.Xorwow(1, 3 * len(Z))
        xyz_list = [orc.atom_jitter(xyz, dwf, x) for _ in range(frozen)]
    else:
        xyz_list = [xyz]
    want = _oracle_stem(orc, p, Z, xyz_list, occ, pos, det)
    assert got.shape == want.shape and ms > 0
    assert np.all(want[:, 0] > 1.0)                       # the bright-field disc carries signal
    np.testing.assert_allclose(got, want, rtol=TOL_INTENSITY, atol=1e-4 * want.max())
    # empty specimen: the whole pattern integrates to n1*n2 (probe normalisation, src/multisliceSimulation.cu:578-580)
    a0 = np.ascontiguousarray(atoms, np.float32)
    a0[:, 3] = 1e-6
    with fb.Simulation(cnf, atoms6=a0) as sim:
        tot, _ = sim.stem_scan(pos[:2], np.array([[0, 1000]], np.float32))
    np.testing.assert_allclose(tot, N * N, rtol=1e-5)


@pytest.mark.parametrize("N", [320, 800, 1000, 600])
def test_stem_detector_sums_at_non_power_of_two_grids(N, fb, orc, tmp_path):
    """The detector reduction runs with 160 / 320 / 200 threads per CTA at 320 / 800 / 1000 (and on the generic
    sweeps at 600): every thread's partial sum must reach the result.  Empty specimen: a detector that covers the
    whole pattern collects n1 * n2 (probe normalisation, src/multisliceSimulation.cu:578-580); with atoms: parity
    with the oracle's per-probe restatement for two positions and three rings."""
    from fdes_b200 import specimens
    d = 0.25e-10
    atoms = specimens.random_slab(30, N * d * 0.5, 2 * 2e-10, seed=N, species=(79, 14))
    cnf = specimens.write_cnf(tmp_path / "stem.cnf", image_size=N, border_size=0, slices=2, pixel_size=d,
                              slice_thickness=2e-10, atoms=atoms, voltage=200e3, mode=2, objective_aperture=10e-3)
    pos = np.array([[0, 0], [5, -3]], np.float32) * np.float32(d)
    det = np.array([[0, 8], [8, 30], [30, 120]], np.float32)
    with fb.Simulation(cnf, batch=2) as sim:
        got, _ = sim.stem_scan(pos, det)
    p, Z, xyz, dwf, occ = orc.read_cnf(str(cnf))
    want = _oracle_stem(orc, p, Z, [xyz], occ, pos, det)
    np.testing.assert_allclose(got, want, rtol=TOL_INTENSITY, atol=1e-4 * want.max())
    a0 = np.ascontiguousarray(atoms, np.float32)
    a0[:, 3] = 1e-6                                    # all atoms outside the slab
    with fb.Simulation(cnf, atoms6=a0, batch=2) as sim:
        tot, _ = sim.stem_scan(pos, np.array([[0, 1000]], np.float32))
    np.testing.assert_allclose(tot, N * N, rtol=1e-5)


def test_stem_scan_needs_probe_mode(fb):
    with fb.Simulation(DATA / "tem64.cnf") as sim:
        with pytest.raises(fb.FdesError, match="mode 2"):
            sim.stem_scan(np.zeros((1, 2), np.float32), np.array([[0, 10]], np.float32))
