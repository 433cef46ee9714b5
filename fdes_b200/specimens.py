"""Synthetic specimens and .cnf writers for the benchmark / parity configurations of BASELINE.json.

The reference ships its example specimens as data files (ExampleSpecimens/, bin/); they are not
copied here.  The same structures are regenerated from their crystallography instead, in the
`.cnf` key syntax the reference reader accepts (src/paramStructure.cu:42-302):

  si001_slab        diamond-cubic Si, [001] zone axis, 19 x 19 x 4 cells = 11 552 atoms
                    (the shape of ExampleSpecimens/Si_001_11k_cnf)               -> config 2
  au_cuboctahedron  fcc Au cuboctahedron with 4 shells = 309 atoms
                    (the shape of ExampleSpecimens/Au_cubeoctahedron_*)          -> config 3
  srtio3_slab       cubic perovskite SrTiO3 (basis and Debye-Waller factors as in
                    bin/SrTiO3.cfg), nx x ny x nz cells                          -> configs 1, 4
  random_slab       uniformly random atoms, Z cycling {8, 22, 38}                -> config 5
"""
from __future__ import annotations

import pathlib
from typing import Dict, Iterable, Optional, Sequence, Tuple

import numpy as np

_ABERRATIONS = ["C1", "A1", "A2", "B2", "C3", "A3", "S3", "A4", "B4", "D4", "C5", "A5", "R5", "S5"]
_ROUND = {"C1", "C3", "C5"}


def _centre(xyz: np.ndarray) -> np.ndarray:
    return xyz - 0.5 * (xyz.min(axis=0) + xyz.max(axis=0))


def si001_slab(nx: int = 19, ny: int = 19, nz: int = 4, a: float = 5.43071e-10, dwf: float = 5.3837e-21):
    """[nAt, 6] = Z x y z DWF occ (metres), centred on the origin."""
    basis = np.array([[0, 0, 0], [0, .5, .5], [.5, 0, .5], [.5, .5, 0],
                      [.25, .25, .25], [.25, .75, .75], [.75, .25, .75], [.75, .75, .25]])
    cells = np.stack(np.meshgrid(np.arange(nx), np.arange(ny), np.arange(nz), indexing="ij"), -1).reshape(-1, 3)
    xyz = _centre((cells[:, None, :] + basis[None, :, :]).reshape(-1, 3) * a)
    out = np.zeros((len(xyz), 6), np.float64)
    out[:, 0], out[:, 1:4], out[:, 4], out[:, 5] = 14, xyz, dwf, 1.0
    return out


def au_cuboctahedron(shells: int = 4, a: float = 4.0782e-10, dwf: float = 6e-21):
    r = np.arange(-2 * shells, 2 * shells + 1)
    g = np.stack(np.meshgrid(r, r, r, indexing="ij"), -1).reshape(-1, 3)
    keep = (g.sum(1) % 2 == 0) & (np.abs(g).max(1) <= shells) & (np.abs(g).sum(1) <= 2 * shells)
    xyz = g[keep] * (a / 2)
    out = np.zeros((len(xyz), 6), np.float64)
    out[:, 0], out[:, 1:4], out[:, 4], out[:, 5] = 79, xyz, dwf, 1.0
    return out


def srtio3_slab(nx: int, ny: int, nz: int, a: float = 3.905e-10):
    """Sr (0,0,0), Ti (.5,.5,.5), O (.5,.5,0) (.5,0,.5) (0,.5,.5); DWF[m^2] = B[A^2] * 1e-20."""
    basis = [(38, (0, 0, 0), 0.6214e-20), (22, (.5, .5, .5), 0.4390e-20), (8, (.5, .5, 0), 0.7323e-20),
             (8, (.5, 0, .5), 0.7323e-20), (8, (0, .5, .5), 0.7323e-20)]
    cells = np.stack(np.meshgrid(np.arange(nx), np.arange(ny), np.arange(nz), indexing="ij"), -1).reshape(-1, 3)
    rows = []
    for Z, f, dw in basis:
        xyz = (cells + np.array(f)) * a
        rows.append(np.column_stack([np.full(len(xyz), Z), xyz, np.full(len(xyz), dw), np.ones(len(xyz))]))
    out = np.concatenate(rows).astype(np.float64)
    # interleave species like a unit-cell-major file would
    order = np.argsort(np.tile(np.arange(len(cells)), len(basis)), kind="stable")
    out = out[order]
    out[:, 1:4] = _centre(out[:, 1:4])
    return out


def random_slab(n_atoms: int, fov_xy: float, thickness: float, seed: int = 12345, species=(8, 22, 38),
                dwf: float = 5e-21):
    rng = np.random.default_rng(seed)
    out = np.zeros((n_atoms, 6), np.float64)
    out[:, 0] = np.array(species)[np.arange(n_atoms) % len(species)]
    out[:, 1] = rng.uniform(-0.45 * fov_xy, 0.45 * fov_xy, n_atoms)
    out[:, 2] = rng.uniform(-0.45 * fov_xy, 0.45 * fov_xy, n_atoms)
    out[:, 3] = rng.uniform(-0.5 * thickness, 0.5 * thickness, n_atoms)
    out[:, 4], out[:, 5] = dwf, 1.0
    return out


def write_cnf(path, *, image_size: int, border_size: int, slices: int, pixel_size: float, slice_thickness: float,
              atoms: Optional[np.ndarray] = None, voltage: float = 200e3, mode: int = 0, frozen_phonons: int = 0,
              sub_slice_thickness: Optional[float] = None, image_size_z: int = 1, absorptive: float = 0.0,
              objective_aperture: float = 1.57, focus_spread: float = 0.0, illumination_angle: float = 0.0,
              mtf: Sequence[float] = (1.0, 0.0, 0.0, 0.0), aberrations: Optional[Dict[str, Tuple[float, float]]] = None,
              specimen_tilts: Optional[Iterable[Tuple[float, float]]] = None,
              beam_tilts: Optional[Iterable[Tuple[float, float]]] = None, defoci: Optional[Iterable[float]] = None,
              tilt_offset: Sequence[float] = (0.0, 0.0, 0.0), comment: str = "fdes_b200 synthetic specimen",
              pixel_size_y: Optional[float] = None, image_size_y: Optional[int] = None,
              border_size_y: Optional[int] = None) -> pathlib.Path:
    """Write a parameter file (atoms optional: FDES() takes them as an array).  The file does not
    end with a newline: the reference reader would read the last atom twice otherwise.  The y sizes default to the
    x ones; the sample stays square (image_size + 2 border_size == image_size_y + 2 border_size_y)."""
    py = pixel_size if pixel_size_y is None else pixel_size_y
    ny = image_size if image_size_y is None else image_size_y
    by = border_size if border_size_y is None else border_size_y
    ab = {k: (0.0, 0.0) for k in _ABERRATIONS}
    ab.update(aberrations or {})
    m = image_size + 2 * border_size
    if ny + 2 * by != m:
        raise ValueError(f"image_size_y + 2 border_size_y = {ny + 2 * by} != {m}: the sample must be square")
    L = [f"comment: {comment}", f"voltage: {voltage:.9g}", f"focus_spread: {focus_spread:.9g}",
         f"illumination_angle: {illumination_angle:.9g}", f"mtf_a: {mtf[0]:.9g}", f"mtf_b: {mtf[1]:.9g}",
         f"mtf_c: {mtf[2]:.9g}", f"mtf_d: {mtf[3]:.9g}", f"objective_aperture: {objective_aperture:.9g}"]
    for k in _ABERRATIONS:
        L.append(f"{k}: {ab[k][0]:.9g}" if k in _ROUND else f"{k}: {ab[k][0]:.9g} {ab[k][1]:.9g}")
    sub = slice_thickness if sub_slice_thickness is None else sub_slice_thickness
    L += [f"mode: {mode}", f"sample_size_x: {m}", f"sample_size_y: {m}", f"sample_size_z: {slices}",
          f"pixel_size_x: {pixel_size:.9g}", f"pixel_size_y: {py:.9g}", f"pixel_size_z: {slice_thickness:.9g}",
          f"border_size_x: {border_size}", f"border_size_y: {by}", f"image_size_x: {image_size}",
          f"image_size_y: {ny}", f"image_size_z: {image_size_z}",
          f"specimen_tilt_offset_x: {tilt_offset[0]:.9g}", f"specimen_tilt_offset_y: {tilt_offset[1]:.9g}",
          f"specimen_tilt_offset_z: {tilt_offset[2]:.9g}", f"frozen_phonons: {frozen_phonons}", "pixel_dose: 0.0",
          f"subpixel_size_z: {sub:.9g}", "sample_name: synthetic", "material: synthetic",
          f"absorptive_potential_factor: {absorptive:.9g}"]
    for a, b in (specimen_tilts or [(0.0, 0.0)] * image_size_z):
        L.append(f"specimen_tilt: {a:.9g} {b:.9g}")
    for a, b in (beam_tilts or [(0.0, 0.0)] * image_size_z):
        L.append(f"beam_tilt: {a:.9g} {b:.9g}")
    for a in (defoci or [0.0] * image_size_z):
        L.append(f"defoci: {a:.9g}")
    if atoms is not None:
        for Z, x, y, z, dw, oc in np.asarray(atoms, np.float64):
            L.append(f"atom: {int(Z)} {x:.9g} {y:.9g} {z:.9g} {dw:.9g} {oc:.9g}")
    path = pathlib.Path(path)
    path.write_text("\n".join(L))
    return path


# ---- the named configurations of BASELINE.json (SURVEY.md section 8d) -------------------------
def config_si001_1024(path, frozen_phonons: int = 0, with_atoms: bool = True):
    """Config 2: Si[001] 11 552 atoms, 100 kV, 1024^2 grid (512 + 2*256), 0.1 A pixels, 11 x 2 A slices."""
    atoms = si001_slab()
    write_cnf(path, image_size=512, border_size=256, slices=11, pixel_size=0.01e-9, slice_thickness=2e-10,
              atoms=atoms if with_atoms else None, voltage=100e3, frozen_phonons=frozen_phonons,
              mtf=(0.58, 0.42, 2.7, 15.5), comment="Si [001] 11k atoms, 1024^2, 2 A slices")
    return atoms


def config_au_2048(path, frozen_phonons: int = 32, sub_slices: bool = False, with_atoms: bool = True):
    """Config 3: Au cuboctahedron 309 atoms, 50 kV, 2048^2 grid (1024 + 2*512), 0.25 A pixels,
    12 x 2.1 A slices (x 11 sub-slices of ~0.19 A when sub_slices is set, as in the shipped file)."""
    atoms = au_cuboctahedron()
    write_cnf(path, image_size=1024, border_size=512, slices=12, pixel_size=0.25e-10, slice_thickness=2.1e-10,
              sub_slice_thickness=0.2e-10 if sub_slices else 2.1e-10, atoms=atoms if with_atoms else None,
              voltage=50e3, frozen_phonons=frozen_phonons, comment="Au cuboctahedron 309 atoms, 2048^2")
    return atoms


def config_random_4096(path, n_atoms: int = 100_000, slices: int = 500, frozen_phonons: int = 64,
                       with_atoms: bool = True):
    """Config 5: 100k random atoms, 4096^2 grid (2048 + 2*1024), 0.1 A pixels, 500 x 2 A slices."""
    atoms = random_slab(n_atoms, 4096 * 0.1e-10, slices * 2e-10)
    write_cnf(path, image_size=2048, border_size=1024, slices=slices, pixel_size=0.1e-10, slice_thickness=2e-10,
              atoms=atoms if with_atoms else None, voltage=200e3, frozen_phonons=frozen_phonons,
              comment="synthetic random slab, 4096^2")
    return atoms


def config_random_4096_short(path, frozen_phonons: int = 2, with_atoms: bool = True):
    """Config 5 geometry with 20 of its 500 slices (4000 of its 100 000 atoms: same areal density per slice)."""
    return config_random_4096(path, n_atoms=4000, slices=20, frozen_phonons=frozen_phonons, with_atoms=with_atoms)


def config_srtio3_800(path, frozen_phonons: int = 0, with_atoms: bool = True):
    """Config 1 in .cnf form: SrTiO3 9 x 9 x 20 cells (8100 atoms, 3 species), 200 kV, 800^2 grid (400 + 2*200) at
    0.087862 A, 40 slices of 1.9525 A run as 400 sub-slices of 0.19525 A, absorptive factor 0.1 -- the geometry
    of config_srtio3_qsc_800 (the .qsc form, which the parity tests run against the reference)."""
    atoms = srtio3_slab(9, 9, 20)
    write_cnf(path, image_size=400, border_size=200, slices=40, pixel_size=0.087862e-10, slice_thickness=1.9525e-10,
              sub_slice_thickness=0.19525e-10, atoms=atoms if with_atoms else None, voltage=200e3, absorptive=0.1,
              objective_aperture=20e-3, frozen_phonons=frozen_phonons,
              comment="SrTiO3 9x9x20 cells, 800^2, 400 sub-slices")
    return atoms


def config_srtio3_stem_512(path, frozen_phonons: int = 0, with_atoms: bool = True):
    """Config 4: SrTiO3 4 x 4 x 20 cells centred in a 5-cell-wide 512^2 box (d = 19.525 A / 512),
    40 x 1.9525 A slices, 200 kV, 20 mrad probe (mode 2), no aberrations."""
    atoms = srtio3_slab(4, 4, 20)
    write_cnf(path, image_size=512, border_size=0, slices=40, pixel_size=19.525e-10 / 512, slice_thickness=1.9525e-10,
              atoms=atoms if with_atoms else None, voltage=200e3, mode=2, objective_aperture=20e-3,
              frozen_phonons=frozen_phonons, comment="SrTiO3 4x4x20 cells, 512^2, STEM probe")
    return atoms


SRTIO3_CFG = """Number of particles = 5
A = 1.0 Angstrom (basic length-scale)
H0(1,1) = 3.905 A
H0(1,2) = 0 A
H0(1,3) = 0 A
H0(2,1) = 0 A
H0(2,2) = 3.905 A
H0(2,3) = 0 A
H0(3,1) = 0 A
H0(3,2) = 0 A
H0(3,3) = 3.905 A
.NO_VELOCITY.
entry_count = 5
87.62
Sr
0 0 0 0.6214 1.0
47.867
Ti
0.5 0.5 0.5 0.4390 1.0
15.999
O
0 0.5 0.5 0.7323 1.0
0.5 0 0.5 0.7323 1.0
0.5 0.5 0 0.7323 1.0
"""


def config_srtio3_qsc_800(directory, cal_mode: int = 0, pixel_dose: float = 0.0, frozen_phonons: int = 0,
                          ncell_z: int = 20):
    """Config 1 (BASELINE configs[0]): the SrTiO3 plane-wave case of the reference's bin/test.qsc +
    bin/SrTiO3.cfg as a QSTEM parameter file: 9 x 9 x 20 cells (8100 atoms, 3 species), 200 kV,
    nx = 400 -> 800^2 grid at 0.087862 A, 40 slices of 1.9525 A -> 400 sub-slices of 0.19525 A.
    Writes <directory>/SrTiO3.cfg and <directory>/srtio3_800.qsc (SURVEY 8d overrides: cal_mode 0,
    pixel_dose 0) and returns the .qsc path.  ncell_z < 20 gives a thinner crystal (2 slices per cell)."""
    import pathlib
    d = pathlib.Path(directory)
    d.mkdir(parents=True, exist_ok=True)
    (d / "SrTiO3.cfg").write_text(SRTIO3_CFG)
    qsc = d / "srtio3_800.qsc"
    qsc.write_text(f"""% SrTiO3 [001] plane-wave exit wave, QSTEM syntax (generated by fdes_b200.specimens)
mode: TEM
filename: SrTiO3.cfg
resolutionX:  0.087862
resolutionY:  0.087862
NCELLX: 9
NCELLY: 9
NCELLZ: {ncell_z}
v0: 200.0
tds: no
slice-thickness: 1.9525
slices: {2 * ncell_z}
center slices: no
nx: 400
ny: 400
Cs: 0.05
C5: 0.0
alpha: 15.0
defocus: 13.7
astigmatism: 0.0
astigmatism angle: 0.0
cal_mode:  {cal_mode}
focus_spread:  1e-9
mtf_a:  1
mtf_b:  0
mtf_c:  0
pixel_dose:  {pixel_dose}
objective_aperture:  20e-3
absorptive_potential_factor:  0.1
frozen_phonons: {frozen_phonons}
""")
    return qsc


def stem_raster(n_side: int, cell: float = 3.905e-10):
    """n_side x n_side probe positions on a uniform raster over the central unit cell [m]."""
    g = (np.arange(n_side) + 0.5) / n_side * cell - 0.5 * cell
    xx, yy = np.meshgrid(g, g, indexing="xy")
    return np.column_stack([xx.ravel(), yy.ravel()]).astype(np.float32)
