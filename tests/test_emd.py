"""EMD / HDF5 input and output (SURVEY section 8f item 1) without libhdf5.

The anchor is a file libhdf5 itself wrote: the reference's shipped
ExampleSpecimens/Au_cubeoctahedron_emd/Auparticle.emd.  tests/h5min.py (independent pure-Python
reader) parses it; tools/make_emd_fixture.py recorded its structure and the raw bytes of
representative header messages in tests/golden/emd_structure.json.  The product's writer
(fdes_b200/csrc/emd.cpp) must produce files that (a) h5min parses, (b) have the same groups,
datasets, dtypes and attributes in the same order, (c) carry byte-identical header messages for
identical content, (d) hold the arrays in the reference's transposed layouts, and (e) read back
through the product's own reader (the .emd input path).  The product's reader is also run on the
real file (shipped_cases.au_particle_emd: its exact bytes, stored compressed under
tests/golden/shipped_inputs/) and compared with its .cnf twin."""
import json

import numpy as np
import pytest

import h5min
import shipped_cases as sc
from conftest import DATA, GOLDEN, ROOT

REAL_CNF = sc.SHIPPED / "ExampleSpecimens" / "Au_cubeoctahedron_cnf" / "dataFDES_Auparticle.cnf"
FIX = json.loads((GOLDEN / "emd_structure.json").read_text())


def message_hex(f, node, mtype):
    p, s = [(p, s) for t, p, s in node.messages if t == mtype][0]
    return f.b[p - 8:p + s].hex()


def attr_hex(f, node, name):
    for t, p, s in node.messages:
        if t == 0x0C and f._attribute(p)[0] == name:
            return f.b[p - 8:p + s].hex()
    raise KeyError(name)


@pytest.fixture(scope="module")
def au_emd(fb, tmp_path_factory):
    """Results file for an input with the real file's header content: 50 kV, 320^2 sample, 309 atoms."""
    from fdes_b200 import specimens
    d = tmp_path_factory.mktemp("emd")
    cnf = d / "au.cnf"
    specimens.write_cnf(cnf, image_size=160, border_size=80, slices=12, pixel_size=0.25e-10, slice_thickness=2.1e-10,
                        atoms=specimens.au_cuboctahedron(), voltage=50e3, comment="Au cuboctahedron 309 atoms")
    r = fb.parse_cnf(cnf)
    assert r["nAt"] == 309 and r["m1"] == 320
    rng = np.random.default_rng(7)
    img = rng.random((r["n3"], r["n2"], r["n1"]), np.float32)
    ew = (rng.random((r["n3"], r["m2"], r["m1"]), np.float32) + 1j * rng.random((r["n3"], r["m2"], r["m1"]), np.float32)).astype(np.complex64)
    pot = (rng.random((3, r["m2"], r["m1"]), np.float32) * (1 + 0.1j)).astype(np.complex64)
    out = d / "results.emd"
    fb.write_emd(cnf, out, img, pot, ew)
    return cnf, out, r, img, pot, ew


def test_writer_output_parses_and_matches_libhdf5_structure(au_emd):
    cnf, out, r, img, pot, ew = au_emd
    f = h5min.File(out)                      # superblock, headers, B-trees, heaps, symbol nodes all consistent
    sb = FIX["superblock"]
    assert (f.sb_version, f.leaf_k, f.internal_k, f.size_offsets, f.size_lengths, f.base) == (
        sb["version"], sb["leaf_k"], sb["internal_k"], sb["size_offsets"], sb["size_lengths"], sb["base"])
    ours = {path: node for path, node in f.root.walk()}
    for path, ref in FIX["paths"].items():          # everything libhdf5 wrote for the reference is there
        assert path in ours, path
        node = ours[path]
        assert ("dataset" if node.data is not None else "group") == ref["kind"], path
        assert list(node.attrs) == ref["attrs"], path                     # same attributes, same order
        if ref["kind"] == "dataset":
            assert str(node.data.dtype) == ref["dtype"] and node.data.ndim == ref["rank"], path
        for k, v in node.attrs.items():
            kind = type(v).__name__ if not hasattr(v, "dtype") else str(v.dtype) + str(list(v.shape))
            assert kind == ref["attr_types"][k], (path, k)
    extra = sorted(set(ours) - set(FIX["paths"]))
    assert extra == sorted(f"/data/{g}{s}" for g in ("exit_wave", "potential_slices")
                           for s in ("", "/data", "/dim1", "/dim2", "/dim3", "/dim4"))


def test_header_messages_are_byte_identical_to_libhdf5(au_emd):
    cnf, out, *_ = au_emd
    f = h5min.File(out)
    m = FIX["messages"]
    zs, xs = f.root["sample/atomic_numbers"], f.root["sample/x_coordinates"]
    assert message_hex(f, zs, 1) == m["int32_dataset"]["dataspace_309"]
    assert message_hex(f, zs, 3) == m["int32_dataset"]["datatype"]
    assert message_hex(f, zs, 5) == m["int32_dataset"]["fill"]
    assert message_hex(f, xs, 3) == m["float32_dataset"]["datatype"]
    assert message_hex(f, xs, 5) == m["float32_dataset"]["fill"]
    assert attr_hex(f, xs, "units") == m["float32_dataset"]["attr_units"]
    assert attr_hex(f, f.root["microscope"], "voltage") == m["attr_float32_voltage_50000"]
    assert attr_hex(f, f.root["imaging"], "sample_size_x") == m["attr_int32_sample_size_x_320"]
    assert attr_hex(f, f.root["data/images"], "emd_group_type") == m["attr_uint8_emd_group_type_1"]
    assert attr_hex(f, f.root["microscope"], "voltage_units") == m["attr_string_voltage_units"]


def test_arrays_are_stored_in_the_reference_layouts(au_emd):
    """/data/images/data [n1][n2][n3] (src/rwHdf5.cu:413-427), exit wave [m1][m2][n3][2] (:248-267),
    potential [m1][m2][m3][2] (:78-96); axes i - (m-1)/2 and the index for dim3 of images / exit wave."""
    cnf, out, r, img, pot, ew = au_emd
    f = h5min.File(out)
    np.testing.assert_array_equal(f.root["data/images/data"].data, img.transpose(2, 1, 0))
    np.testing.assert_array_equal(f.root["data/exit_wave/data"].data, ew.view(np.float32).reshape(*ew.shape, 2).transpose(2, 1, 0, 3))
    np.testing.assert_array_equal(f.root["data/potential_slices/data"].data, pot.view(np.float32).reshape(*pot.shape, 2).transpose(2, 1, 0, 3))
    np.testing.assert_array_equal(f.root["data/images/dim1"].data, (np.arange(r["n1"]) - (r["n1"] - 1) / 2.0).astype(np.float32))
    np.testing.assert_array_equal(f.root["data/exit_wave/dim2"].data, (np.arange(r["m2"]) - (r["m2"] - 1) / 2.0).astype(np.float32))
    np.testing.assert_array_equal(f.root["data/images/dim3"].data, np.arange(r["n3"], dtype=np.float32))
    np.testing.assert_array_equal(f.root["data/potential_slices/dim3"].data, (np.arange(3) - 1.0).astype(np.float32))
    assert list(f.root["data/exit_wave/dim4"].data) == [b"real", b"imag"]
    assert f.root["data/exit_wave/dim4"].attrs == {"name": "complex", "units": "[]"}
    assert f.root.attrs["version"][0] == np.float32(0.1)
    np.testing.assert_array_equal(f.root["sample/atomic_numbers"].data, r["atoms"][:, 0].astype(np.int32))
    np.testing.assert_array_equal(f.root["sample/y_coordinates"].data, r["atoms"][:, 2])
    assert f.root["sample/debeye_waller_factors"].attrs["units"] == "[m^2]"
    assert f.root["comments"].attrs["comment"].startswith("Au cuboctahedron 309 atoms")


@pytest.mark.parametrize("case", ["tilt64", "cbedtilt64", "noise64", "sub128", "qsctilt64.qsc"])
def test_emd_round_trip_through_the_product_reader(case, fb, tmp_path, monkeypatch):
    """write_emd(params of X) read back as an .emd input gives X's parameters and atoms bit for bit
    (readHdf5 + consitentParams, src/rwHdf5.cu:1946-2571)."""
    monkeypatch.chdir(DATA)
    src = DATA / (case if "." in case else f"{case}.cnf")
    a = fb.parse_cnf(src)
    fb.write_emd(src, tmp_path / "config.emd")
    b = fb.parse_cnf(tmp_path / "config.emd")
    assert set(a) == set(b)
    for k in a:
        if isinstance(a[k], np.ndarray):
            np.testing.assert_array_equal(a[k], b[k], err_msg=k)
        else:
            assert a[k] == b[k], k
    lib = fb.load_library()
    ua, ub = tmp_path / "a.txt", tmp_path / "b.txt"
    assert lib.fdes_b200_write_used_cnf(str(src).encode(), str(ua).encode()) == 0
    assert lib.fdes_b200_write_used_cnf(str(tmp_path / "config.emd").encode(), str(ub).encode()) == 0
    strip = lambda t: [l for l in t.splitlines() if not l.startswith(("comment", "sample_name", "material"))]
    assert strip(ua.read_text()) == strip(ub.read_text())       # every field of params_t that writeConfig prints


def test_reader_rejects_what_is_not_an_emd(fb, tmp_path):
    lib = fb.load_library()
    bad = tmp_path / "bad.emd"
    bad.write_bytes(b"not hdf5" * 40)
    assert lib.fdes_b200_parse_cnf(str(bad).encode(), None, None, None, None, 0) == -1
    assert b"not an HDF5 file" in lib.fdes_b200_last_error()
    fb.write_emd(DATA / "tem64.cnf", tmp_path / "ok.emd")
    raw = bytearray((tmp_path / "ok.emd").read_bytes())
    cut = tmp_path / "cut.emd"
    cut.write_bytes(raw[: len(raw) // 3])
    assert lib.fdes_b200_parse_cnf(str(cut).encode(), None, None, None, None, 0) == -1


def test_h5min_and_product_reader_on_the_real_libhdf5_file(fb, tmp_path):
    """The file libhdf5 wrote: h5min's structure equals the committed fixture, and the product's
    reader returns what the .cnf twin of the same specimen holds (SURVEY section 8c: same parameters)."""
    real = sc.au_particle_emd(tmp_path)
    f = h5min.File(real)
    assert {p: n for p, n in ((p, list(n.attrs)) for p, n in f.root.walk())} == {p: v["attrs"] for p, v in FIX["paths"].items()}
    e = fb.parse_cnf(real)
    c = fb.parse_cnf(REAL_CNF)
    for k in ("n1", "n2", "n3", "m1", "m2", "m3", "nZ", "frPh", "mode", "lam", "sigma", "gamma", "d1", "d2", "d3", "E0", "imPot"):
        assert e[k] == c[k], k
    np.testing.assert_array_equal(e["tiltspec"], c["tiltspec"])
    np.testing.assert_array_equal(e["defoci"], c["defoci"])
    assert e["nAt"] == 309 and c["nAt"] in (309, 310)       # the .cnf ends with a newline: last atom read twice
    np.testing.assert_array_equal(e["atoms"], c["atoms"][:309])


@pytest.mark.gpu
def test_fdes_writes_the_results_emd_and_reads_it_back_as_input(fb, orc, tmp_path, monkeypatch):
    """FDES() at print level 2: emd_save_name is a real EMD with images, potential slices and exit
    waves; the file is then used as the INPUT of a second run, which reproduces the first image."""
    from conftest import TOL_INTENSITY, TOL_WAVE, rel_l2
    monkeypatch.chdir(tmp_path)
    cnf = DATA / "tilt64.cnf"
    p, Z, xyz, dwf, occ = orc.read_cnf(str(cnf))
    atoms6 = np.column_stack([Z.astype(np.float32), xyz, dwf, occ]).astype(np.float32)
    dst = np.zeros((p.n3, p.n2, p.n1), np.float32)
    fb.cuda_FDES(0, 2, str(cnf), str(tmp_path / "M.bin"), str(tmp_path / "r.emd"), atoms6, len(atoms6), dst)
    f = h5min.File(tmp_path / "r.emd")
    np.testing.assert_array_equal(f.root["data/images/data"].data.transpose(2, 1, 0), dst)
    ew = np.ascontiguousarray(f.root["data/exit_wave/data"].data.transpose(2, 1, 0, 3)).view(np.complex64)[..., 0]
    res = orc.build_measurements(p, Z, xyz, dwf, np.trunc(occ).astype(np.float32))
    assert rel_l2(ew, res.exitwave) < TOL_WAVE
    assert f.root["data/potential_slices/data"].data.shape == (p.m1, p.m2, p.m3, 2)
    assert h5min.File(tmp_path / "config.emd").root["imaging"].attrs["image_size_z"][0] == p.n3   # src/FDESExport.cu:141
    dst2 = np.zeros_like(dst)
    fb.cuda_FDES(0, 0, str(tmp_path / "r.emd"), str(tmp_path / "M2.bin"), str(tmp_path / "r2.emd"), atoms6, len(atoms6), dst2)
    np.testing.assert_array_equal(dst2, dst)
    assert (tmp_path / "ParamsUsedEmd.txt").exists()


def test_array_layouts_with_several_measurements(fb, tmp_path):
    """n3 = 2 (tilt64): the k index is the FASTEST spatial index of the stored arrays
    (f_xyz[i * n3 * n2 + j * n3 + k], src/rwHdf5.cu:413-419) -- a layout a single image cannot tell apart."""
    r = fb.parse_cnf(DATA / "tilt64.cnf")
    assert r["n3"] == 2
    rng = np.random.default_rng(3)
    img = rng.random((2, r["n2"], r["n1"]), np.float32)
    ew = (rng.random((2, r["m2"], r["m1"])) + 1j * rng.random((2, r["m2"], r["m1"]))).astype(np.complex64)
    fb.write_emd(DATA / "tilt64.cnf", tmp_path / "r.emd", img, None, ew)
    f = h5min.File(tmp_path / "r.emd")
    d = f.root["data/images/data"].data
    assert d.shape == (r["n1"], r["n2"], 2)
    for k in range(2):
        np.testing.assert_array_equal(d[:, :, k], img[k].T)
        np.testing.assert_array_equal(f.root["data/exit_wave/data"].data[:, :, k, 0], ew[k].real.T)
        np.testing.assert_array_equal(f.root["data/exit_wave/data"].data[:, :, k, 1], ew[k].imag.T)
    assert "potential_slices" not in f.root["data"].children
    np.testing.assert_array_equal(f.root["imaging/specimen_tilt_x"].data, r["tiltspec"][:, 0])
    np.testing.assert_array_equal(f.root["imaging/defoci"].data, r["defoci"])


def test_reader_survives_corrupted_files(fb, tmp_path):
    """The .emd input path is reachable from FDES() and the CLI: truncated or corrupted HDF5 bytes
    (undefined addresses 0xFF..FF, broken B-tree / heap offsets, unterminated names) must end in an error
    code or in parsed values, never in an out-of-bounds read."""
    lib = fb.load_library()
    src = sc.au_particle_emd(tmp_path).read_bytes()
    rng = np.random.default_rng(0)
    rejected = 0
    for i in range(120):
        b = bytearray(src[: (len(src) if i % 2 else int(rng.integers(100, 6000)))])
        for _ in range(int(rng.integers(1, 8))):
            j = int(rng.integers(0, min(len(b), 6000)))
            b[j] = int(rng.integers(0, 256)) if rng.random() < 0.5 else 0xFF
        f = tmp_path / "c.emd"
        f.write_bytes(bytes(b))
        rc = lib.fdes_b200_parse_cnf(str(f).encode(), None, None, None, None, 0)
        rejected += rc < 0
    assert rejected > 20
