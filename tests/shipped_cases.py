"""The reference's shipped example inputs, run AS SHIPPED (tests/data/shipped/ holds unmodified copies of
/root/reference/bin and /root/reference/ExampleSpecimens: they are input data, not code) plus one
variant each with `pixel_dose: 0` (deterministic detector tail).  Shared by tools/make_shipped_golden.py
(runs the unmodified reference on a GPU box -> tests/golden/shipped/*.npz) and tests/test_shipped_inputs.py.

Golden content per case (reductions keep the repository small): the image of the measurements K_KEEP,
mean and L2 norm of every image, a central crop of the coherent exit wave of the same measurements and
the sum of |psi|^2 of every exit wave.  <case>.npz holds the per-image statistics,
<case>.k<i>.<array>.<j>.npz the rows of chunk j of an array of the i-th kept measurement.

The shipped EMD file (Au_cubeoctahedron_emd/Auparticle.emd, 2.6 MB, almost all of it unused HDF5 space)
is stored xz-compressed as tests/golden/shipped_inputs/Auparticle.emd.xz; au_particle_emd() gives its exact
bytes back."""
import lzma
import pathlib
import re
import shutil

import numpy as np

SHIPPED = pathlib.Path(__file__).resolve().parent / "data" / "shipped"

# name -> (file relative to SHIPPED, pixel dose override or None = as shipped)
CASES = {
    "bin_test_qsc": ("bin/test.qsc", None),                       # CBED (cal_mode 2), pixel_dose 10: test.qsc:80,87
    "bin_test_qsc_dose0": ("bin/test.qsc", 0.0),
    "bin_dataFDES": ("bin/dataFDES.cnf", None),                   # Au-309, 320^2, 25 tilts, dose 100
    "bin_dataFDES_dose0": ("bin/dataFDES.cnf", 0.0),
    "au_particle_cnf": ("ExampleSpecimens/Au_cubeoctahedron_cnf/dataFDES_Auparticle.cnf", None),
    "au_particle_cnf_dose0": ("ExampleSpecimens/Au_cubeoctahedron_cnf/dataFDES_Auparticle.cnf", 0.0),
    "si_001_11k": ("ExampleSpecimens/Si_001_11k_cnf/dataFDES_11k.cnf", None),   # 1000^2, 205 slices, dose 0 as shipped
    "srtio3_qsc": ("ExampleSpecimens/SrTiO3_qsc/SrTiO3.qsc", None),
    "srtio3_qsc_dose0": ("ExampleSpecimens/SrTiO3_qsc/SrTiO3.qsc", 0.0),
}
CROP = 96          # half-width of the central exit-wave crop
PER_K = ("image_keep", "ew_crop", "ew_crop_fp64")     # arrays stored per kept measurement, in row chunks
CHUNK = 800_000    # bytes of a stored chunk: every golden file stays under 1 MB
# focused probe through 400 sub-slices: the goldens also carry a float64 evaluation of the model
DEEP_PROBE_CASES = ("bin_test_qsc", "bin_test_qsc_dose0", "srtio3_qsc", "srtio3_qsc_dose0")


def stage(case: str, workdir: pathlib.Path) -> pathlib.Path:
    """Copy the input (and the .cfg a .qsc names) into workdir, apply the dose override, return the path."""
    rel, dose = CASES[case]
    src = SHIPPED / rel
    workdir.mkdir(parents=True, exist_ok=True)
    for f in src.parent.iterdir():
        if f.suffix == ".cfg":
            shutil.copy(f, workdir / f.name)
    dst = workdir / src.name
    raw = src.read_bytes()
    if dose is not None:
        raw, n = re.subn(rb"(?m)^(pixel_dose:\s*)[-+0-9.eE]+", lambda m: m.group(1) + repr(float(dose)).encode(), raw)
        assert n == 1, f"{src}: pixel_dose line not found"
    dst.write_bytes(raw)
    return dst


def k_keep(n3: int):
    return sorted({0, n3 // 2, n3 - 1})


def reduce(image: np.ndarray, exitwave: np.ndarray) -> dict:
    """image [n3][n2][n1] float32, exitwave [n3][m2][m1] complex64 -> the golden reductions."""
    n3 = image.shape[0]
    ks = k_keep(n3)
    m2, m1 = exitwave.shape[1:]
    c2, c1 = m2 // 2, m1 // 2
    h = min(CROP, c1, c2)
    return {
        "k_keep": np.array(ks, np.int32),
        "image_keep": np.ascontiguousarray(image[ks]),
        "image_mean": image.reshape(n3, -1).mean(axis=1, dtype=np.float64),
        "image_norm": np.sqrt((image.reshape(n3, -1).astype(np.float64) ** 2).sum(axis=1)),
        "ew_crop": np.ascontiguousarray(exitwave[ks][:, c2 - h:c2 + h, c1 - h:c1 + h]),
        "ew_power": (np.abs(exitwave.reshape(n3, -1).astype(np.complex128)) ** 2).sum(axis=1),
        "shape": np.array([n3, image.shape[1], image.shape[2], m2, m1], np.int32),
    }


def au_particle_emd(workdir: pathlib.Path) -> pathlib.Path:
    """The reference's shipped ExampleSpecimens/Au_cubeoctahedron_emd/Auparticle.emd, unpacked into workdir."""
    src = SHIPPED.parent.parent / "golden" / "shipped_inputs" / "Auparticle.emd.xz"
    workdir.mkdir(parents=True, exist_ok=True)
    dst = workdir / "Auparticle.emd"
    dst.write_bytes(lzma.decompress(src.read_bytes()))
    return dst


def save_golden(directory: pathlib.Path, case: str, g: dict) -> None:
    np.savez_compressed(directory / f"{case}.npz", **{k: v for k, v in g.items() if k not in PER_K})
    for key in PER_K:
        for i, a in enumerate(g.get(key, [])):
            for j, part in enumerate(np.array_split(a, -(-a.nbytes // CHUNK), axis=0)):
                np.savez_compressed(directory / f"{case}.k{i}.{key}.{j}.npz", a=part)


def load_golden(directory: pathlib.Path, case: str) -> dict:
    g = dict(np.load(directory / f"{case}.npz"))
    for key in PER_K:
        per_k = []
        for i in range(len(g["k_keep"])):
            parts = sorted(directory.glob(f"{case}.k{i}.{key}.*.npz"), key=lambda f: int(f.stem.rsplit(".", 1)[1]))
            if parts:
                per_k.append(np.concatenate([np.load(f)["a"] for f in parts]))
        if per_k:
            g[key] = np.stack(per_k)
    return g
