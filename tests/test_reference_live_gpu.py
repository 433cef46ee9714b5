"""Parity of the BASELINE.json shapes against the UNMODIFIED reference run on the same box
(oracle/_ref/ref_harness: the reference's own objects driven through getParams -> buildMeasurements,
see oracle/ref_harness.cu), at sizes the numpy oracle would need minutes for:

  * configs[2]  Au cuboctahedron, 2048^2, frozen phonons (same XORWOW streams in both programs)
  * configs[4]  random slab, 4096^2, 3 species, 50 slices, absorptive potential
  * configs[3]  SrTiO3 512^2 x 40 slices, STEM probes off the grid centre: the reference has no scan,
                so a probe at r_p is its mode-2 run with every atom translated by -r_p (SURVEY.md 8c),
                detector sums taken from its intensity BEFORE addNoiseAndMtf (I_d of `ref_harness trace`)
  * configs[0]  SrTiO3 800^2 from .qsc, 400 sub-slices: three-way distances with a float64 evaluation
                of the same model (oracle.exit_wave_fp64) and two runs of the reference

Bounds are north_star's: exit waves rel-L2 <= 1e-5, detector intensities <= 1e-4.  Where the reference
build is absent, each test compares the library on the same input with the numpy oracle instead (the
independent float32 restatement of the reference that tests/test_oracle_golden.py pins to the
reference's recorded outputs), under the same bounds, and a warning says that the live comparison did
not run.
"""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, TOL_INTENSITY, TOL_WAVE, live_reference_missing, rel_l2

pytestmark = pytest.mark.gpu
HARNESS = ROOT / "oracle" / "_ref" / "ref_harness"
# rel-L2 of the reference's exit wave to the float64 evaluation at BASELINE configs[0] (400 sub-slices, plane
# wave), measured in the live comparison of test_srtio3_800_400_subslices_error_budget (DESIGN.md)
REF_FP64_SRTIO3_400 = 1.8e-5


def _against_oracle(orc, cnf, img, ew):
    p, Z, xyz, dwf, occ = orc.read_cnf(str(cnf))
    res = orc.build_measurements(p, Z, xyz, dwf, occ)
    d_ew, d_img = rel_l2(ew, res.exitwave), rel_l2(img, res.image)
    print(f"{cnf.name} against the oracle: exit wave {d_ew:.3e}, image {d_img:.3e}")
    assert d_ew < TOL_WAVE and d_img < TOL_INTENSITY


def _ref_run(cnf, out, shape_img, shape_ew):
    subprocess.run([str(HARNESS), "run", str(cnf), str(out), "2"], check=True, capture_output=True, timeout=1500)
    rimg = np.fromfile(out / "image.f32", np.float32).reshape(shape_img)
    rew = np.fromfile(out / "exitwave.f32", np.float32).view(np.complex64).reshape(shape_ew)
    return rimg, rew


def test_au_2048_frozen_phonons_against_live_reference(fb, orc, tmp_path):
    from fdes_b200 import specimens
    cnf = tmp_path / "au.cnf"
    specimens.config_au_2048(cnf, frozen_phonons=3)
    with fb.Simulation(cnf, want_exitwave=True) as sim:
        assert (sim.m1, sim.configs) == (2048, 3)
        img, ew = sim.simulate()
    if live_reference_missing(HARNESS):
        return _against_oracle(orc, cnf, img, ew)
    rimg, rew = _ref_run(cnf, tmp_path / "ref", img.shape, ew.shape)
    d_ew, d_img = rel_l2(ew, rew), rel_l2(img, rimg)
    print(f"au_2048 x 3 phonon configurations: exit wave {d_ew:.3e}, image {d_img:.3e}")
    assert d_ew < TOL_WAVE and d_img < TOL_INTENSITY


def test_slab_4096_three_species_50_slices_against_live_reference(fb, orc, tmp_path):
    from fdes_b200 import specimens
    cnf = tmp_path / "slab.cnf"
    atoms = specimens.random_slab(10_000, 4096 * 0.1e-10, 50 * 2e-10)
    specimens.write_cnf(cnf, image_size=2048, border_size=1024, slices=50, pixel_size=0.1e-10, slice_thickness=2e-10,
                        atoms=atoms, voltage=200e3, absorptive=0.05, mtf=(0.58, 0.42, 2.7, 15.5))
    with fb.Simulation(cnf, want_exitwave=True) as sim:
        assert (sim.m1, sim.m3, sim.nZ) == (4096, 50, 3)
        img, ew = sim.simulate()
    if live_reference_missing(HARNESS):
        return _against_oracle(orc, cnf, img, ew)
    rimg, rew = _ref_run(cnf, tmp_path / "ref", img.shape, ew.shape)
    d_ew, d_img = rel_l2(ew, rew), rel_l2(img, rimg)
    print(f"slab_4096, 3 species x 50 slices: exit wave {d_ew:.3e}, image {d_img:.3e}")
    assert d_ew < TOL_WAVE and d_img < TOL_INTENSITY


def test_stem_512_offcentre_probes_against_live_reference(fb, orc, tmp_path):
    from fdes_b200 import specimens
    N, d = 512, 19.525e-10 / 512
    atoms = specimens.srtio3_slab(4, 4, 20)
    kw = dict(image_size=N, border_size=0, slices=40, pixel_size=d, slice_thickness=1.9525e-10, voltage=200e3, mode=2,
              objective_aperture=20e-3)
    cnf = specimens.write_cnf(tmp_path / "stem.cnf", atoms=atoms, **kw)
    # whole-pixel positions inside the central unit cell (the translated atoms then deposit identically)
    pos_px = np.array([[0, 0], [17, -9], [-23, 31], [40, 12], [-5, -44]], np.float32)
    pos = pos_px * np.float32(d)
    det = np.array([[70.0, 200.0], [11.0, 22.0], [0.0, 20.0]], np.float32)       # HAADF, ABF, BF
    with fb.Simulation(cnf, batch=4) as sim:
        assert (sim.m1, sim.m3) == (512, 40)
        got, ms = sim.stem_scan(pos, det)
    if live_reference_missing(HARNESS):
        from test_parity_gpu import _oracle_stem     # the reference algorithm per probe: translated atoms, mode 2
        p, Z, xyz, dwf, occ = orc.read_cnf(str(cnf))
        want = _oracle_stem(orc, p, Z, [xyz], occ, pos, det)
        print("STEM 512^2 x 40 slices, ours / oracle per probe and detector:\n", got / want)
        assert np.all(want[:, 2] > 1.0)
        np.testing.assert_allclose(got, want, rtol=TOL_INTENSITY, atol=1e-4 * want.max())
        return
    p = orc.read_cnf(str(cnf))[0]
    lam = np.float32(p.lam)
    kx = (orc.ow(N).astype(np.float32) / np.float32(N * np.float32(d)))[None, :]
    ky = (orc.ow(N).astype(np.float32) / np.float32(N * np.float32(d)))[:, None]
    ksq = (kx * kx + ky * ky).astype(np.float32)
    rings = [((np.sin(np.float32(a * 1e-3)) / lam) ** 2, (np.sin(np.float32(b * 1e-3)) / lam) ** 2) for a, b in det]
    want = np.zeros_like(got, dtype=np.float64)
    for i, (px, py) in enumerate(pos):
        shifted = atoms.copy()
        # float32 subtraction as the library's probe shift sees it: atoms are float32 in both programs
        shifted[:, 1] = (atoms[:, 1].astype(np.float32) - np.float32(px)).astype(np.float64)
        shifted[:, 2] = (atoms[:, 2].astype(np.float32) - np.float32(py)).astype(np.float64)
        c = specimens.write_cnf(tmp_path / f"probe{i}.cnf", atoms=shifted, **kw)
        out = tmp_path / f"ref{i}"
        subprocess.run([str(HARNESS), "trace", str(c), str(out), "0"], check=True, capture_output=True, timeout=600)
        I = np.fromfile(out / "I_d.c64", np.float32).reshape(N, N, 2)[..., 0].astype(np.float64)
        for k, (lo, hi) in enumerate(rings):
            want[i, k] = I[(ksq >= lo) & (ksq < hi)].sum()
    print("STEM 512^2 x 40 slices, ours / reference per probe and detector:\n", got / want)
    assert np.all(want[:, 2] > 1.0)
    np.testing.assert_allclose(got, want, rtol=TOL_INTENSITY, atol=1e-4 * want.max())


def test_srtio3_800_400_subslices_error_budget(fb, orc, qorc, tmp_path):
    """BASELINE configs[0] at its full depth (400 sub-slices = 1600 chained float32 transforms in both
    programs).  Whose rounding is it?  Distances to the float64 evaluation of the same model:
    the library must be within 1e-5 of the reference, or at least as close to the exact result as
    the reference itself is (x 1.25 for run-to-run scatter of the reference's float atomics).  Without the
    reference build: at least as close to the float64 evaluation as the reference was when measured live
    (REF_FP64_SRTIO3_400), and the image against the oracle's."""
    from fdes_b200 import specimens
    qsc = specimens.config_srtio3_qsc_800(tmp_path, ncell_z=20)
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        with fb.Simulation(qsc, want_exitwave=True) as sim:
            assert (sim.m1, sim.m3, sim.nZ) == (800, 400, 3)
            img, ew = sim.simulate()
        p, Z, xyz, dwf, occ = qorc.read_qsc(str(qsc))
    finally:
        os.chdir(cwd)
    truth = orc.exit_wave_fp64(p, Z, xyz, occ).reshape(ew.shape)
    if live_reference_missing(HARNESS):
        res = orc.build_measurements(p, Z, xyz, dwf, occ)
        d = {"ours-fp64": rel_l2(ew, truth), "image ours-oracle": rel_l2(img, res.image)}
        print("srtio3_800, 400 sub-slices: " + ", ".join(f"{k} {v:.3e}" for k, v in d.items()))
        assert d["ours-fp64"] <= 1.25 * REF_FP64_SRTIO3_400, d
        assert d["ours-fp64"] < 3 * TOL_WAVE
        assert d["image ours-oracle"] < TOL_INTENSITY
        return
    rimg1, rew1 = _ref_run(qsc, tmp_path / "ref1", img.shape, ew.shape)
    rimg2, rew2 = _ref_run(qsc, tmp_path / "ref2", img.shape, ew.shape)
    d = {"ours-ref": rel_l2(ew, rew1), "ours-fp64": rel_l2(ew, truth), "ref-fp64": rel_l2(rew1, truth),
         "ref-ref": rel_l2(rew1, rew2), "image ours-ref": rel_l2(img, rimg1)}
    print("srtio3_800, 400 sub-slices: " + ", ".join(f"{k} {v:.3e}" for k, v in d.items()))
    (tmp_path / "budget.txt").write_text(repr(d))
    assert d["ours-ref"] < TOL_WAVE or d["ours-fp64"] <= 1.25 * d["ref-fp64"], d
    assert d["ours-fp64"] < 3 * TOL_WAVE
    assert d["image ours-ref"] < TOL_INTENSITY


@pytest.mark.parametrize("seed", [1, 2, 3, 4, 5, 6, 7])
def test_random_grid_sizes_against_live_reference(seed, fb, orc, tmp_path):
    """Any sample size the reference accepts (seeds 5 .. 7: odd sizes) (m = n + 2 dn, src/paramStructure.cu:650-651): random
    image / border sizes, random mode, 3 species, against the unmodified reference run on the same input.
    Sizes without a register-resident instantiation take the generic run-time-N sweeps."""
    from fdes_b200 import specimens
    rng = np.random.default_rng(1000 + seed)
    n = 2 * int(rng.integers(32, 500)) + (1 if seed >= 5 else 0)
    dn = int(rng.integers(0, 200))
    m = n + 2 * dn
    mode = int(rng.integers(0, 3))
    d = 0.2e-10
    atoms = specimens.random_slab(120, m * d, 6 * 2e-10, seed=seed, species=(79, 14, 8))
    cnf = specimens.write_cnf(tmp_path / f"g{m}.cnf", image_size=n, border_size=dn, slices=6, pixel_size=d,
                              slice_thickness=2e-10, atoms=atoms, voltage=150e3, mode=mode, absorptive=0.04,
                              objective_aperture=0.012, frozen_phonons=2 if mode == 0 else 0, mtf=(0.58, 0.42, 2.7, 15.5),
                              aberrations={"C1": (-2e-8, 0.0), "C3": (3e-4, 0.0)})
    with fb.Simulation(cnf, want_exitwave=True) as sim:
        assert sim.m1 == m
        img, ew = sim.simulate()
    if live_reference_missing(HARNESS):
        return _against_oracle(orc, cnf, img, ew)
    rimg, rew = _ref_run(cnf, tmp_path / "ref", img.shape, ew.shape)
    d_ew, d_img = rel_l2(ew, rew), rel_l2(img, rimg)
    print(f"grid {m} = {n} + 2 x {dn}, mode {mode}: exit wave {d_ew:.3e}, image {d_img:.3e}")
    assert d_ew < TOL_WAVE and d_img < TOL_INTENSITY
