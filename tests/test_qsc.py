"""QSTEM .qsc / .cfg input (SURVEY section 8f item 4; BASELINE configs[0] is a .qsc input).

CPU: the oracle's restatement of readQsc (oracle/qsc_oracle.py) against the `ParamsUsedQsc.txt`
files the unmodified reference wrote for tests/data/*.qsc (tests/golden/*.ParamsUsedQsc.txt,
tools/make_golden.py), and the product's C++ reader (fdes_b200/csrc/qsc.cpp, through the C ABI)
bit-for-bit against the oracle.  GPU: the full run from a .qsc against the reference's exit wave /
image and against the oracle."""
import os
import re

import numpy as np
import pytest

from conftest import DATA, GOLDEN, TOL_INTENSITY, TOL_WAVE, golden, rel_l2

QSC_CASES = sorted(p.stem for p in DATA.glob("qsc*.qsc"))
AB = ["C1", "A1", "A2", "B2", "C3", "A3", "S3", "A4", "B4", "D4", "C5", "A5", "R5", "S5"]


@pytest.fixture(scope="module")
def qorc(orc):
    import qsc_oracle
    return qsc_oracle


def parse_used(text):
    """key -> list of numbers, plus the atom table, of a file written by writeConfig
    (src/paramStructure.cu:360-487)."""
    keys, atoms = {}, []
    in_atoms = False
    for line in text.splitlines():
        line = line.split("#")[0].strip()
        if not line:
            continue
        if line.startswith("Number of atoms:"):
            keys["nAt"] = [float(line.split(":")[1])]
            in_atoms = True
            continue
        toks = line.split()
        if in_atoms:
            if toks[0] == "atom:":
                toks = toks[1:]
            atoms.append([float(t) for t in toks[:6]])
        elif toks[0].endswith(":"):
            keys.setdefault(toks[0][:-1], []).append([float(t) for t in toks[1:] if re.match(r"^[-+0-9.]", t)])
    return keys, np.array(atoms, np.float64).reshape(-1, 6)


def close(a, b, rel=2e-7):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.all(np.abs(a - b) <= rel * np.maximum(np.abs(b), 1e-300) + 0.0)


def used_from_params(p, Z, xyz, dwf, occ):
    k = dict(voltage=p.E0, lam=p.lam, sigma=p.sigma, gamma=p.gamma, focus_spread=p.defocspread,
             illumination_angle=p.illangle, mtf_a=p.mtfa, mtf_b=p.mtfb, mtf_c=p.mtfc, mtf_d=p.mtfd,
             objective_aperture=p.ObjAp, mode=p.mode, sample_size_x=p.m1, sample_size_y=p.m2, sample_size_z=p.m3,
             pixel_size_x=p.d1, pixel_size_y=p.d2, pixel_size_z=p.d3, border_size_x=p.dn1, border_size_y=p.dn2,
             image_size_x=p.n1, image_size_y=p.n2, image_size_z=p.n3, specimen_tilt_offset_x=p.tilt_off[0],
             specimen_tilt_offset_y=p.tilt_off[1], specimen_tilt_offset_z=p.tilt_off[2], frozen_phonons=p.frPh,
             pixel_dose=p.pD, subpixel_size_z=p.subSlTh, absorptive_potential_factor=p.imPot)
    return k


@pytest.mark.parametrize("case", QSC_CASES)
def test_oracle_qsc_reader_matches_reference(case, qorc):
    """Pins the oracle: what the reference's readQsc understood (its ParamsUsedQsc.txt, printed with
    %14.8g) against the restatement."""
    f = GOLDEN / f"{case}.ParamsUsedQsc.txt"
    if not f.exists():
        pytest.fail(f"{f} missing (tools/make_golden.py on a GPU box)")
    keys, atoms = parse_used(f.read_text(errors="replace"))
    cwd = os.getcwd()
    os.chdir(DATA)
    try:
        p, Z, xyz, dwf, occ = qorc.read_qsc(str(DATA / f"{case}.qsc"))
    finally:
        os.chdir(cwd)
    mine = used_from_params(p, Z, xyz, dwf, occ)
    mine["lambda"] = mine.pop("lam")
    for k, v in mine.items():
        ref = keys[k][0][0]
        if isinstance(v, (int, np.integer)):
            assert int(ref) == int(v), k
        else:
            assert close(v, ref), (k, v, ref)
    for name in AB:
        ref = keys[name][0]
        assert close(p.ab0[name], ref[0]), name
        if len(ref) > 1:
            assert close(p.ab1[name], ref[1]), name
    assert close(p.tiltbeam[:2], keys["beam_tilt"][0])
    assert close(p.tiltspec[:2], keys["specimen_tilt"][0])
    assert int(keys["nAt"][0]) == len(Z) == len(atoms)
    np.testing.assert_array_equal(atoms[:, 0].astype(np.int32), Z)        # species and ORDER bit-exact
    assert np.max(np.abs(atoms[:, 1:4] - xyz)) <= 2e-7 * np.max(np.abs(xyz))
    assert close(atoms[:, 4], dwf) and close(atoms[:, 5], occ)


@pytest.mark.parametrize("case", QSC_CASES)
def test_cpp_qsc_reader_matches_oracle_bitwise(case, fb, orc, qorc, tmp_path):
    cwd = os.getcwd()
    os.chdir(DATA)
    try:
        r = fb.parse_cnf(DATA / f"{case}.qsc")
        p, Z, xyz, dwf, occ = qorc.read_qsc(str(DATA / f"{case}.qsc"))
        lib = fb.load_library()
        used = tmp_path / "used.txt"
        assert lib.fdes_b200_write_used_cnf(str(DATA / f"{case}.qsc").encode(), str(used).encode()) == 0
    finally:
        os.chdir(cwd)
    keys, atoms = parse_used(used.read_text())
    orc.set_sub_slices(p, orc.sub_slice_ratio(p.d3, p.subSlTh))
    for k, v in dict(n1=p.n1, n2=p.n2, n3=p.n3, m1=p.m1, m2=p.m2, m3=p.m3, nAt=len(Z), frPh=p.frPh, mode=p.mode,
                     nZ=len(orc.list_of_elements(Z))).items():
        assert r[k] == v, k
    for k, v in dict(lam=p.lam, sigma=p.sigma, gamma=p.gamma, d1=p.d1, d2=p.d2, d3=p.d3, E0=p.E0, imPot=p.imPot).items():
        assert np.float32(r[k]) == np.float32(v), k       # bit-exact float32
    np.testing.assert_array_equal(r["atoms"][:, 0].astype(np.int32), Z)
    np.testing.assert_array_equal(r["atoms"][:, 1:4], xyz)
    np.testing.assert_array_equal(r["atoms"][:, 4], dwf)
    np.testing.assert_array_equal(r["atoms"][:, 5], occ)
    np.testing.assert_array_equal(r["tiltbeam"].ravel(), p.tiltbeam[:2])
    # the rest of params_t through the written side-effect file (%14.8g)
    for name in AB:
        assert close(p.ab0[name], keys[name][0][0]) and close(p.ab1[name], keys[name][0][1]), name
    for k in ("focus_spread", "illumination_angle", "mtf_a", "mtf_b", "mtf_c", "mtf_d", "objective_aperture",
              "pixel_dose", "specimen_tilt_offset_x", "specimen_tilt_offset_y", "specimen_tilt_offset_z"):
        v = used_from_params(p, Z, xyz, dwf, occ)[k]
        assert close(v, keys[k][0][0]), k
    assert len(atoms) == len(Z)


@pytest.mark.parametrize("seed", range(8))
def test_cpp_qsc_reader_matches_oracle_on_random_cells(seed, fb, qorc, tmp_path, monkeypatch):
    """Random triclinic cells, atom lists, replications, tilts, offsets and key orders: the C++ reader and the
    (reference-pinned) oracle agree bit for bit on every parameter and atom."""
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.integers(1, 7))
    H = np.diag(rng.uniform(2.5, 6.0, 3)) + np.tril(rng.uniform(-1.0, 1.0, (3, 3)), -1) * (seed % 2)
    vel = seed % 3 == 0
    lines = [f"Number of particles = {n}", f"A = {rng.choice([1.0, 0.9, 1.25])} Angstrom"]
    lines += [f"H0({a + 1},{b + 1}) = {H[a, b]:.5f} A" for a in range(3) for b in range(3)]
    ncols = int(rng.integers(0, 3))                                  # extra columns: DWF, occupancy
    lines += ([] if vel else [".NO_VELOCITY."]) + [f"entry_count = {3 + ncols}"]
    species = [("12.011", "C"), ("28.086", "Si"), ("196.97", "Au"), ("15.999", "O"), ("55.845", "Fe")]
    for i in range(n):
        if i == 0 or rng.random() < 0.5:
            m, el = species[int(rng.integers(len(species)))]
            lines += [m + (" # mass" if rng.random() < 0.3 else ""), el]
        xyz = rng.uniform(0, 1, 3).round(4) + i * 1e-3                # distinct sites
        cols = [f"{v:.4f}" for v in xyz] + (["0", "0", "0"] if vel else [])
        cols += [f"{rng.uniform(0.2, 0.9):.4f}", "1.0"][:ncols]
        lines.append((" " if rng.random() < 0.3 else "") + "  ".join(cols))
    (tmp_path / "cell.cfg").write_text("\n".join(lines) + "\n")
    ncell = rng.integers(1, 4, 3)
    keys = {
        "mode": "mode: TEM", "file": "filename: " + rng.choice(["cell.cfg", '"cell"', "cell"]),
        "nc": f"NCELLX: {ncell[0]}\nNCELLY: {ncell[1]}\nNCELLZ: {ncell[2]}",
        "v0": f"v0: {rng.choice([80.0, 120.0, 300.0])}", "nx": "nx: 32" + ("\nny: 32" if seed % 2 else ""),
        "res": "" if seed % 4 == 0 else "resolutionX: 0.31\nresolutionY: 0.29",
        "sl": rng.choice(["slice-thickness: 2.1\nslices: 5", "slices: 6", "slice-thickness: 1.7"]),
        "tilt": f"Crystal tilt X: {rng.uniform(-0.05, 0.05):.4f}\nCrystal tilt Y: {rng.uniform(-2, 2):.3f} deg\n"
                f"Crystal tilt Z: {rng.uniform(-0.2, 0.2):.4f}" if seed % 2 else "",
        "beam": f"Beam tilt X: {rng.uniform(-0.1, 0.1):.4f} deg\nBeam tilt Y: {rng.uniform(-2e-3, 2e-3):.5f}",
        "off": f"xOffset: {rng.uniform(-1, 1):.3f}\nyOffset: {rng.uniform(-1, 1):.3f}" if seed % 3 else "",
        "lens": f"Cs: {rng.uniform(0.01, 1.5):.3f}\nalpha: {rng.uniform(5, 20):.2f}\n"
                f"defocus: {rng.choice(['Scherzer', 'opt', f'{rng.uniform(-60, 60):.2f}'])}\n"
                f"astigmatism: {rng.uniform(0, 3):.2f}\nastigmatism angle: {rng.uniform(0, 90):.1f}",
        "fdes": f"cal_mode: {int(rng.integers(0, 3))}\nobjective_aperture: {rng.uniform(5e-3, 3e-2):.4g}\n"
                f"frozen_phonons: {int(rng.integers(0, 3))}\nabsorptive_potential_factor: {rng.uniform(0, 0.2):.3f}\n"
                f"focus_spread: {rng.uniform(0, 5e-9):.3g}\nmtf_a: 0.6\nmtf_b: 0.4\nmtf_c: 2.5\npixel_dose: 0",
    }
    order = [k for k in keys if k != "mode"]
    rng.shuffle(order)                                               # readparam wraps: any order of UNIQUE keys works,
    order = ["mode"] + order                                         # but "mode:" must precede "cal_mode:" (strstr)
    (tmp_path / "r.qsc").write_text("\n".join(keys[k] for k in order if keys[k]) + "\n")
    monkeypatch.chdir(tmp_path)
    r = fb.parse_cnf(tmp_path / "r.qsc")
    p, Z, xyz, dwf, occ = qorc.read_qsc(str(tmp_path / "r.qsc"))
    used = tmp_path / "used.txt"
    assert fb.load_library().fdes_b200_write_used_cnf(str(tmp_path / "r.qsc").encode(), str(used).encode()) == 0
    keysu, atoms = parse_used(used.read_text())
    assert (r["n1"], r["n2"], r["m1"], r["nAt"], r["frPh"], r["mode"]) == (p.n1, p.n2, p.m1, len(Z), p.frPh, p.mode)
    sub = p.copy()
    import fdes_oracle as orc
    orc.set_sub_slices(sub, orc.sub_slice_ratio(sub.d3, sub.subSlTh))
    assert (r["m3"], np.float32(r["d3"])) == (sub.m3, np.float32(sub.d3))
    for k, v in dict(lam=p.lam, sigma=p.sigma, d1=p.d1, d2=p.d2, E0=p.E0, imPot=p.imPot).items():
        assert np.float32(r[k]) == np.float32(v), k
    np.testing.assert_array_equal(r["atoms"][:, 0].astype(np.int32), Z)
    np.testing.assert_array_equal(r["atoms"][:, 1:4], xyz)
    np.testing.assert_array_equal(r["atoms"][:, 4], dwf)
    np.testing.assert_array_equal(r["tiltbeam"].ravel(), p.tiltbeam[:2])
    for name in AB:
        assert close(p.ab0[name], keysu[name][0][0]) and close(p.ab1[name], keysu[name][0][1]), name
    for k in ("illumination_angle", "objective_aperture", "specimen_tilt_offset_x", "specimen_tilt_offset_y",
              "specimen_tilt_offset_z", "subpixel_size_z", "focus_spread", "mtf_c"):
        assert close(used_from_params(p, Z, xyz, dwf, occ)[k], keysu[k][0][0]), k


def test_qsc_reader_refuses_what_it_cannot_reproduce(fb, tmp_path):
    lib = fb.load_library()
    base = (DATA / "qsc64.qsc").read_text()
    (tmp_path / "sto.cfg").write_text((DATA / "sto.cfg").read_text())
    bad = {
        "cbed": base.replace("mode: TEM", "mode: CBED"),   # ("STEM" contains "TEM" and passes, src/rwQsc.cu:35)
        "tds": base.replace("tds: no", "tds: yes"),
        "cube": base.replace("tds: no", "tds: no\nCube: 10 10 10"),
        "cssr": base.replace("filename: sto.cfg", "filename: sto.cssr"),
        "nocfg": base.replace("filename: sto.cfg", "filename: missing.cfg"),
    }
    for name, text in bad.items():
        f = tmp_path / f"{name}.qsc"
        f.write_text(text)
        assert lib.fdes_b200_parse_cnf(str(f).encode(), None, None, None, None, 0) == -1, name
        assert lib.fdes_b200_last_error()
    # partial occupancy in the unit cell: the reference draws a lottery with ran1 -> refused
    (tmp_path / "sto.cfg").write_text((DATA / "sto.cfg").read_text().replace("0 0 0 0.6214 1.0", "0 0 0 0.6214 0.5"))
    f = tmp_path / "occ.qsc"
    f.write_text(base)
    assert lib.fdes_b200_parse_cnf(str(f).encode(), None, None, None, None, 0) == -1
    assert b"occupanc" in lib.fdes_b200_last_error()


@pytest.mark.gpu
@pytest.mark.parametrize("case", QSC_CASES)
def test_qsc_full_run_against_reference_golden_and_oracle(case, fb, orc, qorc):
    g, meta = golden(case)
    cwd = os.getcwd()
    os.chdir(DATA)
    try:
        p, Z, xyz, dwf, occ = qorc.read_qsc(str(DATA / f"{case}.qsc"))
        with fb.Simulation(DATA / f"{case}.qsc", want_exitwave=True) as sim:
            img, ew = sim.simulate()
            assert sim.counters()["launches"] > 0
    finally:
        os.chdir(cwd)
    assert (p.m1, p.m2) == (int(meta["m1"]), int(meta["m2"])) and len(Z) == int(meta["nAt"])
    assert rel_l2(ew, g["exitwave"]) < TOL_WAVE
    assert rel_l2(img, g["image"]) < TOL_INTENSITY
    res = orc.build_measurements(p, Z, xyz, dwf, occ)
    assert rel_l2(ew, res.exitwave) < TOL_WAVE
    assert rel_l2(img, res.image) < TOL_INTENSITY


@pytest.mark.gpu
@pytest.mark.parametrize("ncell_z,tol_wave", [(5, TOL_WAVE)])
def test_srtio3_800_qsc_against_live_reference(ncell_z, tol_wave, fb, orc, qorc, tmp_path):
    """BASELINE configs[0]: SrTiO3 9x9xN cells from a .qsc + .cfg, 800^2 grid (2^5 * 5^2 lines), plane
    wave -- our exit wave and image against the unmodified reference run here, N = 5 (100 sub-slices),
    held to the north-star bound of 1e-5.  The full depth (N = 20, 400 sub-slices) is examined in
    tests/test_reference_live_gpu.py::test_srtio3_800_400_subslices_error_budget against a float64
    evaluation of the model.  Without the reference build: the comparison with the oracle."""
    import subprocess
    from conftest import ROOT, live_reference_missing
    from fdes_b200 import specimens
    harness = ROOT / "oracle" / "_ref" / "ref_harness"
    qsc = specimens.config_srtio3_qsc_800(tmp_path, ncell_z=ncell_z)
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        with fb.Simulation(qsc, want_exitwave=True) as sim:
            assert (sim.m1, sim.m3, sim.nAt, sim.nZ) == (800, 20 * ncell_z, 405 * ncell_z, 3)
            img, ew = sim.simulate()
        p, Z, xyz, dwf, occ = qorc.read_qsc(str(qsc))
    finally:
        os.chdir(cwd)
    res = orc.build_measurements(p, Z, xyz, dwf, occ) if ncell_z == 5 else None
    if res is not None:
        print(f"srtio3_800 N={ncell_z}: ours-vs-oracle {rel_l2(ew, res.exitwave):.3e}, image {rel_l2(img, res.image):.3e}")
        assert rel_l2(ew, res.exitwave) < tol_wave
        assert rel_l2(img, res.image) < TOL_INTENSITY
    if live_reference_missing(harness):
        return
    out = tmp_path / "ref"
    subprocess.run([str(harness), "run", str(qsc), str(out), "2"], check=True, capture_output=True)
    rimg = np.fromfile(out / "image.f32", np.float32).reshape(img.shape)
    rew = np.fromfile(out / "exitwave.f32", np.float32).view(np.complex64).reshape(ew.shape)
    d_ref = rel_l2(ew, rew)
    print(f"srtio3_800 N={ncell_z}: ours-vs-reference exit wave {d_ref:.3e}, image {rel_l2(img, rimg):.3e}")
    if res is not None:
        print(f"   reference-vs-oracle {rel_l2(rew, res.exitwave):.3e}")
    assert d_ref < tol_wave
    assert rel_l2(img, rimg) < TOL_INTENSITY


@pytest.mark.gpu
def test_fdes_export_accepts_qsc(fb, tmp_path):
    """FDES() with a .qsc: parameters from the file, atoms from the caller (atomsFromExternal,
    src/FDESExport.cu:73), side-effect file ParamsUsedQsc.txt (src/rwQsc.cu:1084)."""
    for f in ("qsc64.qsc", "sto.cfg"):
        (tmp_path / f).write_text((DATA / f).read_text())
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        r = fb.parse_cnf(tmp_path / "qsc64.qsc")
        atoms6 = np.ascontiguousarray(r["atoms"], np.float32)
        dst = np.zeros((r["n3"], r["n2"], r["n1"]), np.float32)
        fb.cuda_FDES(0, 0, str(tmp_path / "qsc64.qsc"), str(tmp_path / "M.bin"), str(tmp_path / "r.emd"), atoms6,
                     len(atoms6), dst)
        with fb.Simulation(tmp_path / "qsc64.qsc") as sim:
            img, _ = sim.simulate()
    finally:
        os.chdir(cwd)
    assert (tmp_path / "ParamsUsedQsc.txt").exists()
    np.testing.assert_array_equal(dst, img)


# ---------------------------------------------------------------------------------------------
# `mode: STEM` parameter files: scan raster + detectors (keys readQsc parses, src/rwQsc.cu:444-466,
# 698-735, and FDES never uses) feeding the batched STEM scan
# ---------------------------------------------------------------------------------------------
def test_stem_qsc_scan_keys_cpp_matches_oracle(fb, qorc, monkeypatch):
    monkeypatch.chdir(DATA)
    xy, det = fb.qsc_scan(DATA / "stem128.qsc")
    oxy, odet = qorc.read_qsc_scan(str(DATA / "stem128.qsc"))
    assert xy.shape == (4, 3, 2) and det.shape == (3, 2)
    np.testing.assert_array_equal(xy, oxy)            # bit-exact float32
    np.testing.assert_array_equal(det, odet)
    np.testing.assert_array_equal(det, np.array([[70, 200], [11, 22], [0, 10]], np.float32))
    # QSTEM raster: start + i (stop - start) / pixels in the super-cell frame, minus the centring shift
    p, Z, xyz, dwf, occ, shift = qorc.read_qsc(str(DATA / "stem128.qsc"), return_shift=True)
    step = (5.8575 - 1.9525) / 4 * 1e-10
    np.testing.assert_allclose(xy[:, 0, 0], 1.9525e-10 + step * np.arange(4) - shift[0], rtol=0, atol=5e-17)
    np.testing.assert_allclose(xy[0, :, 1], 1.9525e-10 + (4.88125 - 1.9525) / 3 * 1e-10 * np.arange(3) - shift[1], rtol=0, atol=5e-17)
    r = fb.parse_cnf(DATA / "stem128.qsc")
    assert (r["mode"], r["m1"], r["nAt"]) == (2, 128, 40)     # "STEM" contains "TEM" (src/rwQsc.cu:35); cal_mode 2
    lib = fb.load_library()
    assert lib.fdes_b200_qsc_scan(str(DATA / "qsc64.qsc").encode(), None, None, 0, None, 0) == -1   # no scan keys
    assert b"scan_x_start" in lib.fdes_b200_last_error()


@pytest.mark.gpu
def test_stem_scan_from_qsc_against_oracle(fb, orc, qorc, monkeypatch):
    """The whole path from a QSTEM STEM file: reader -> raster/detectors -> batched probe scan, against
    the oracle's per-probe restatement (reference mode-2 run with the atoms translated by -r_p)."""
    from test_parity_gpu import _oracle_stem
    monkeypatch.chdir(DATA)
    qsc = DATA / "stem128.qsc"
    xy, det = fb.qsc_scan(qsc)
    with fb.Simulation(qsc, batch=5) as sim:
        got, ms = sim.stem_scan(xy.reshape(-1, 2), det)
    p, Z, xyz, dwf, occ = qorc.read_qsc(str(qsc))
    want = _oracle_stem(orc, p, Z, [xyz], occ, xy.reshape(-1, 2), det)
    assert got.shape == want.shape == (12, 3) and ms > 0
    np.testing.assert_allclose(got, want, rtol=TOL_INTENSITY, atol=1e-4 * want.max())
    assert np.ptp(want[:, 0]) > 1e-3 * want[:, 0].mean()        # the HAADF signal really varies over the raster


@pytest.mark.gpu
def test_cli_stem_scan_from_qsc(fb, tmp_path):
    """FDES --stem_scan (extension): the STEM .qsc drives the batched probe scan from the command line;
    image_name holds float32 [detector][x][y]."""
    import subprocess
    from conftest import ROOT
    for f in ("stem128.qsc", "sto.cfg"):
        (tmp_path / f).write_text((DATA / f).read_text())
    exe = ROOT / "fdes_b200" / "bin" / "FDES"
    r = subprocess.run([str(exe), "--input_name", "stem128.qsc", "--stem_scan", "--image_name", "stem.bin"], cwd=tmp_path,
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-500:]
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        xy, det = fb.qsc_scan(tmp_path / "stem128.qsc")
        with fb.Simulation(tmp_path / "stem128.qsc", batch=32) as sim:
            want, _ = sim.stem_scan(xy.reshape(-1, 2), det)
    finally:
        os.chdir(cwd)
    got = np.fromfile(tmp_path / "stem.bin", np.float32).reshape(len(det), xy.shape[0], xy.shape[1])
    np.testing.assert_array_equal(got, want.reshape(xy.shape[0], xy.shape[1], len(det)).transpose(2, 0, 1))
    r = subprocess.run([str(exe), "--input_name", str(DATA / "qsc64.qsc"), "--stem_scan"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode != 0 and "scan_x_start" in r.stderr
