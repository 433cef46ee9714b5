"""The reference's shipped example inputs, run as shipped (and with the Poisson noise switched off),
against golden vectors the UNMODIFIED reference produced for the same files on a B200
(tools/make_shipped_golden.py -> tests/golden/shipped/*.npz; cases: tests/shipped_cases.py):

  bin/test.qsc                CBED (cal_mode 2), pixel_dose 10, SrTiO3 9x9x20 cells, 800^2, 400 sub-slices
  bin/dataFDES.cnf            Au-309 particle, 320^2, 25 tilts, 132 sub-slices, pixel_dose 100
  ExampleSpecimens/Au_*_cnf   same particle at 50 kV;  ExampleSpecimens/Au_*_emd: its EMD/HDF5 twin
  ExampleSpecimens/Si_001_11k 1000^2, 205 slices of 0.1 A
  ExampleSpecimens/SrTiO3_qsc the QSTEM parameter file of the SrTiO3 example

Exit waves rel-L2 <= 1e-5, images <= 1e-4 (north_star).  With the Poisson noise on, both programs draw from
the same XORWOW streams (curand_init(1 + n3, pixel, 0), src/crystalMaker.cu:295) and round to whole
electron counts (:50-70): a pixel whose noisy value sits within float32 rounding of a half-integer can
land one count apart, so those images are held to <= 5e-4 (1e-3 for the deep probe cases) and to
identical mean counts.

The two .qsc inputs send a focused probe through 400 sub-slices (1600 chained float32 transforms).  There
the reference itself sits 5.5e-5 .. 6.3e-5 (exit wave) and 5e-5 .. 6e-5 (total intensity) away from a
float64 evaluation of the same model started from the same float32 probe (oracle.exit_wave_fp64, stored
in the goldens as ew_crop_fp64 / ew_power_fp64 when they were generated), so no float32 program can be
within 1e-5 of it and be right.  For these cases the bound on the exit wave is: at least as close to the
float64 result as the reference is (measured: 3.5e-5 .. 4.3e-5 against the reference's 5.5e-5 .. 6.3e-5)."""
import os

import numpy as np
import pytest

import shipped_cases as sc
from conftest import GOLDEN, TOL_INTENSITY, TOL_WAVE, rel_l2

pytestmark = pytest.mark.gpu


def _golden(case):
    f = GOLDEN / "shipped" / f"{case}.npz"
    if not f.exists():
        pytest.fail(f"{f} missing (tools/make_shipped_golden.py)")
    return sc.load_golden(f.parent, case)


def _run(fb, path, workdir):
    cwd = os.getcwd()
    os.chdir(workdir)
    try:
        with fb.Simulation(path, want_exitwave=True) as sim:
            img, ew = sim.simulate()
    finally:
        os.chdir(cwd)
    return img, ew


def _compare(case, img, ew, noisy):
    g = _golden(case)
    assert tuple(g["shape"]) == (img.shape[0], img.shape[1], img.shape[2], ew.shape[1], ew.shape[2])
    r = sc.reduce(img, ew)
    d_ew = rel_l2(r["ew_crop"], g["ew_crop"])
    d_pw = float(np.max(np.abs(r["ew_power"] / g["ew_power"] - 1)))
    d_img = rel_l2(r["image_keep"], g["image_keep"])
    d_norm = float(np.max(np.abs(r["image_norm"] / g["image_norm"] - 1)))
    d_mean = float(np.max(np.abs(r["image_mean"] / g["image_mean"] - 1)))
    print(f"{case}: exit-wave crop {d_ew:.2e}, |psi|^2 sums {d_pw:.2e}, images {d_img:.2e}, image norms {d_norm:.2e}, means {d_mean:.2e}")
    deep = case in sc.DEEP_PROBE_CASES
    if deep:
        t_ours, t_ref = rel_l2(r["ew_crop"], g["ew_crop_fp64"]), rel_l2(g["ew_crop"], g["ew_crop_fp64"])
        p_ours = float(np.max(np.abs(r["ew_power"] / g["ew_power_fp64"] - 1)))
        p_ref = float(np.max(np.abs(g["ew_power"] / g["ew_power_fp64"] - 1)))
        print(f"   distance to the float64 evaluation: exit-wave crop ours {t_ours:.2e} / reference {t_ref:.2e}, "
              f"|psi|^2 sum ours {p_ours:.2e} / reference {p_ref:.2e}")
        # exit wave: no farther from the float64 result than the reference; total intensity: both float32
        # programs end 5e-5 .. 8e-5 above it after 400 sub-slices (measured; systematic float32 rounding of
        # the per-slice factors) -- held to the 1e-4 of north_star's intensities
        assert t_ours <= t_ref
        assert p_ours < TOL_INTENSITY and p_ref < TOL_INTENSITY and d_pw < TOL_INTENSITY
        assert d_ew < 1e-4
    else:
        assert d_ew < TOL_WAVE and d_pw < TOL_WAVE
    assert d_img < ((1e-3 if deep else 5e-4) if noisy else TOL_INTENSITY)
    assert d_norm < TOL_INTENSITY and d_mean < TOL_INTENSITY


@pytest.mark.parametrize("case", sorted(sc.CASES))
def test_shipped_input_against_reference_golden(case, fb, tmp_path):
    inp = sc.stage(case, tmp_path)
    img, ew = _run(fb, inp, tmp_path)
    noisy = sc.CASES[case][1] is None and case != "si_001_11k"
    _compare(case, img, ew, noisy)


def test_shipped_emd_input_matches_its_cnf_twin(fb, tmp_path):
    """ExampleSpecimens/Au_cubeoctahedron_emd/Auparticle.emd (written by libhdf5 for the reference) read by
    the library's own HDF5 parser: same parameters and atoms as the .cnf twin (SURVEY 8c), so the golden
    of that file applies."""
    emd = sc.au_particle_emd(tmp_path)
    img, ew = _run(fb, emd, tmp_path)
    _compare("au_particle_cnf", img, ew, noisy=True)
