"""fdes_b200 -- B200-native forward multislice behind the FDES interface.

Host-side Python mirror of the reference's Python entry point (Python/pyFDES.py:33-41,
``cuda_FDES``) plus a thin ctypes binding of the session API in ``include/fdes_b200.h``.
All compute happens in ``fdes_b200/lib/libfdes_b200.so`` (hand-written sm_100a kernels);
there is no CPU or PyTorch fallback -- importing works anywhere, computing needs a B200
and the built library, and fails loudly otherwise.
"""
from __future__ import annotations

import ctypes
import os
import pathlib
from typing import Optional

import numpy as np

_PKG = pathlib.Path(__file__).resolve().parent
LIB_PATH = pathlib.Path(os.environ.get("FDES_B200_LIB", _PKG / "lib" / "libfdes_b200.so"))
_lib = None


class FdesError(RuntimeError):
    pass


def load_library() -> ctypes.CDLL:
    """Load libfdes_b200.so (built in-tree by ``__graft_entry__.build()`` / ``make``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise FdesError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(there is no fallback implementation)")
    lib = ctypes.CDLL(str(LIB_PATH), mode=ctypes.RTLD_GLOBAL)
    c_f = ctypes.POINTER(ctypes.c_float)
    c_i = ctypes.POINTER(ctypes.c_int)
    vp = ctypes.c_void_p
    lib.fdes_b200_last_error.restype = ctypes.c_char_p
    lib.fdes_b200_version.restype = ctypes.c_int
    lib.fdes_b200_release_cache.restype = None
    lib.fdes_b200_open_cnf.restype = vp
    lib.fdes_b200_open_cnf.argtypes = [ctypes.c_char_p, c_f, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                       ctypes.c_int, ctypes.c_int, ctypes.c_int]
    lib.fdes_b200_open_multi.restype = vp
    lib.fdes_b200_open_multi.argtypes = [ctypes.c_char_p, c_f, ctypes.c_int, c_i, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    lib.fdes_b200_num_gpus.argtypes = [vp]
    lib.fdes_b200_parse_gpu_list.argtypes = [ctypes.c_char_p, ctypes.c_int, c_i, ctypes.c_int]
    lib.fdes_b200_parse_cnf.argtypes = [ctypes.c_char_p, c_i, c_f, c_f, c_f, ctypes.c_int]
    lib.fdes_b200_write_used_cnf.argtypes = [ctypes.c_char_p, ctypes.c_char_p]
    lib.fdes_b200_write_emd.argtypes = [ctypes.c_char_p, ctypes.c_char_p, c_f, c_f, ctypes.c_int, c_f]
    lib.fdes_b200_qsc_scan.argtypes = [ctypes.c_char_p, c_i, c_f, ctypes.c_int, c_f, ctypes.c_int]
    lib.fdes_b200_close.argtypes = [vp]
    lib.fdes_b200_close.restype = None
    lib.fdes_b200_get_dims.argtypes = [vp, c_i]
    lib.fdes_b200_get_scalars.argtypes = [vp, c_f]
    lib.fdes_b200_set_accumulators.argtypes = [vp, vp, vp]
    lib.fdes_b200_run_k.argtypes = [vp, ctypes.c_int]
    lib.fdes_b200_finish_k.argtypes = [vp, ctypes.c_int, c_f, c_f]
    lib.fdes_b200_simulate.argtypes = [vp, c_f, c_f]
    lib.fdes_b200_potential_slices_count.argtypes = [vp]
    lib.fdes_b200_potential.argtypes = [vp, c_f]
    lib.fdes_b200_jitter_next.argtypes = [vp, ctypes.c_int, c_f]
    lib.fdes_b200_bin_atoms.argtypes = [vp, c_f, c_i]
    lib.fdes_b200_phase_grating.argtypes = [vp, c_f, ctypes.c_int, c_f]
    lib.fdes_b200_exit_wave.argtypes = [vp, c_f, ctypes.c_int, c_f]
    lib.fdes_b200_bench_configs.argtypes = [vp, ctypes.c_int, ctypes.c_int]
    lib.fdes_b200_bench_configs.restype = ctypes.c_double
    lib.fdes_b200_stem_scan.argtypes = [vp, ctypes.c_int, ctypes.c_int, c_f, ctypes.c_int, c_f, c_f]
    lib.fdes_b200_stem_scan.restype = ctypes.c_double
    lib.fdes_b200_stem_scan_4d.argtypes = [vp, ctypes.c_int, ctypes.c_int, c_f, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_f,
                                           ctypes.c_int, c_f, c_f]
    lib.fdes_b200_stem_scan_4d.restype = ctypes.c_double
    lib.fdes_b200_stem_4d_side.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int]
    lib.fdes_b200_time_sweeps.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_f]
    lib.fdes_b200_get_counters.argtypes = [vp, ctypes.POINTER(ctypes.c_longlong), ctypes.c_int]
    lib.fdes_b200_fft2d.argtypes = [c_f, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    lib.fdes_b200_sort_records.argtypes = [ctypes.POINTER(ctypes.c_uint), c_i, c_f, ctypes.c_int, ctypes.c_int,
                                           c_i, ctypes.c_int]
    lib.fdes_b200_sweep_test.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, c_i, ctypes.c_int, c_f, ctypes.c_int,
                                         ctypes.POINTER(c_f), ctypes.POINTER(ctypes.c_longlong), ctypes.c_int,
                                         ctypes.c_int, ctypes.c_int, c_i]
    lib.FDES.restype = None
    lib.FDES.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, c_f,
                         ctypes.c_int, c_f]
    _lib = lib
    return lib


def declared_symbols():
    """Names of every function include/fdes_b200.h declares (the drop-in boundary)."""
    import re
    text = (_PKG.parent / "include" / "fdes_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(FDES|fdes_b200_\w+)\s*\(", text)))


def _fp(a: np.ndarray):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


def _ip(a: np.ndarray):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_int))


def cuda_FDES(gpu_Index, print_Level, input_name, image_name, emd_save_name, pointerAtomsArray, numAtoms,
              pointerImagesArray):
    """Same call as ``cuda_FDES`` in the reference's Python/pyFDES.py:33-41; the two array
    arguments may be ctypes float pointers (as there) or float32 numpy arrays."""
    lib = load_library()
    if isinstance(pointerAtomsArray, np.ndarray):
        pointerAtomsArray = _fp(np.ascontiguousarray(pointerAtomsArray, np.float32))
    if isinstance(pointerImagesArray, np.ndarray):
        assert pointerImagesArray.dtype == np.float32 and pointerImagesArray.flags.c_contiguous
        pointerImagesArray = _fp(pointerImagesArray)
    enc = lambda s: s if isinstance(s, bytes) else str(s).encode()
    return lib.FDES(int(gpu_Index), int(print_Level), enc(input_name), enc(image_name), enc(emd_save_name),
                    pointerAtomsArray, int(numAtoms), pointerImagesArray)


def parse_cnf(cnf_path):
    """Host-only view of what the engine would run for a .cnf (no GPU needed): dict of dims,
    scalars, per-measurement tilts/defoci and the atom table [nAt, 6]."""
    lib = load_library()
    d = np.zeros(10, np.int32)
    s = np.zeros(8, np.float32)
    n = lib.fdes_b200_parse_cnf(str(cnf_path).encode(), _ip(d), _fp(s), None, None, 0)
    if n < 0:
        raise FdesError(lib.fdes_b200_last_error().decode())
    per_k = np.zeros((int(d[2]), 5), np.float32)
    atoms = np.zeros((n, 6), np.float32)
    lib.fdes_b200_parse_cnf(str(cnf_path).encode(), _ip(d), _fp(s), _fp(per_k), _fp(atoms), n)
    keys_d = ["n1", "n2", "n3", "m1", "m2", "m3", "nAt", "nZ", "frPh", "mode"]
    keys_s = ["lam", "sigma", "gamma", "d1", "d2", "d3", "E0", "imPot"]
    out = {k: int(v) for k, v in zip(keys_d, d)}
    out.update({k: np.float32(v) for k, v in zip(keys_s, s)})
    out["tiltspec"], out["tiltbeam"], out["defoci"] = per_k[:, 0:2].copy(), per_k[:, 2:4].copy(), per_k[:, 4].copy()
    out["atoms"] = atoms
    return out


def qsc_scan(qsc_path):
    """Host-only: (positions [nx, ny, 2] in metres, detectors [ndet, 2] in mrad) of a `mode: STEM` .qsc,
    ready for Simulation.stem_scan(positions.reshape(-1, 2), detectors)."""
    lib = load_library()
    nxy = np.zeros(2, np.int32)
    nd = lib.fdes_b200_qsc_scan(str(qsc_path).encode(), _ip(nxy), None, 0, None, 0)
    if nd < 0:
        raise FdesError(lib.fdes_b200_last_error().decode())
    xy = np.zeros((int(nxy[0]), int(nxy[1]), 2), np.float32)
    det = np.zeros((nd, 2), np.float32)
    lib.fdes_b200_qsc_scan(str(qsc_path).encode(), _ip(nxy), _fp(xy), xy.shape[0] * xy.shape[1], _fp(det), nd)
    return xy, det


def write_emd(input_path, emd_path, image=None, potential=None, exitwave=None):
    """Host-only: EMD (HDF5) file with the reference's layout from a parameter file and arrays
    (image [n3,n2,n1] float32, potential [m3,m2,m1] complex64, exitwave [n3,m2,m1] complex64)."""
    lib = load_library()
    keep = []

    def ptr(a, dt):
        if a is None:
            return None
        a = np.ascontiguousarray(a, dt)
        keep.append(a)
        return a.view(np.float32).ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    nslices = 0 if potential is None else int(np.asarray(potential).shape[0])
    rc = lib.fdes_b200_write_emd(str(input_path).encode(), str(emd_path).encode(), ptr(image, np.float32),
                                 ptr(potential, np.complex64), nslices, ptr(exitwave, np.complex64))
    if rc != 0:
        raise FdesError(lib.fdes_b200_last_error().decode())


def stem_4d_side(n: int, window: int = 0, bin: int = 1) -> int:
    """Host-only: side of the 4D-STEM patterns (Q / bin) on an n x n grid; window 0 is the smallest centred window
    that holds the band limit.  Raises FdesError with the reason when window / bin are not admissible."""
    lib = load_library()
    side = lib.fdes_b200_stem_4d_side(int(n), int(window), int(bin))
    if side < 0:
        raise FdesError(lib.fdes_b200_last_error().decode())
    return side


def parse_gpu_list(spec, first: int = 0):
    """Device ordinals of an FDES_B200_GPUS / --gpus value ("4" or "0,2,5")."""
    lib = load_library()
    enc = None if spec is None else str(spec).encode()
    n = lib.fdes_b200_parse_gpu_list(enc, first, None, 0)
    out = np.zeros(max(n, 1), np.int32)
    lib.fdes_b200_parse_gpu_list(enc, first, _ip(out), len(out))
    return [int(v) for v in out[:n]]


class Simulation:
    """One simulation (session API of include/fdes_b200.h) on one GPU, or -- ``gpus=[...]`` -- sharded
    over several GPUs of this process (fdes_b200_open_multi: frozen-phonon configurations, tilt series
    or STEM probes dealt out, partial sums reduced onto the first device)."""

    def __init__(self, cnf_path, atoms6: Optional[np.ndarray] = None, gpu_index: int = 0, batch: int = 0,
                 rank: int = 0, world: int = 1, want_exitwave: bool = False, gpus=None):
        self._lib = load_library()
        self._h = None
        a_ptr, n_at = None, 0
        if atoms6 is not None:
            self._atoms6 = np.ascontiguousarray(atoms6, np.float32).reshape(-1, 6)
            a_ptr, n_at = _fp(self._atoms6), self._atoms6.shape[0]
        if gpus is not None:
            g = np.ascontiguousarray(list(gpus), np.int32)
            h = self._lib.fdes_b200_open_multi(str(cnf_path).encode(), a_ptr, n_at, _ip(g), len(g), batch,
                                               1 if want_exitwave else 0)
        else:
            h = self._lib.fdes_b200_open_cnf(str(cnf_path).encode(), a_ptr, n_at, gpu_index, batch, rank, world,
                                             1 if want_exitwave else 0)
        if not h:
            raise FdesError(self._lib.fdes_b200_last_error().decode())
        self._h = h
        d = np.zeros(10, np.int32)
        self._ck(self._lib.fdes_b200_get_dims(h, _ip(d)))
        (self.n1, self.n2, self.n3, self.m1, self.m2, self.m3, self.nAt, self.nZ, self.configs, self.batch) = map(int, d)
        s = np.zeros(8, np.float32)
        self._ck(self._lib.fdes_b200_get_scalars(h, _fp(s)))
        self.lam, self.sigma, self.gamma, self.d1, self.d2, self.d3, self.E0, self.imPot = map(float, s)
        self.want_exitwave = want_exitwave
        self.gpu_index = int(gpus[0]) if gpus is not None else int(gpu_index)
        self.num_gpus = int(self._lib.fdes_b200_num_gpus(h))

    def _ck(self, rc):
        if rc != 0:
            raise FdesError(self._lib.fdes_b200_last_error().decode())

    def close(self):
        if self._h:
            self._lib.fdes_b200_close(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- reference-facing -------------------------------------------------------------------
    def simulate(self):
        """All measurements on this GPU: (image [n3,n2,n1] float32, exitwave [n3,m2,m1] complex64|None)."""
        img = np.zeros((self.n3, self.n2, self.n1), np.float32)
        ew = np.zeros((self.n3, self.m2, self.m1), np.complex64) if self.want_exitwave else None
        self._ck(self._lib.fdes_b200_simulate(self._h, _fp(img), _fp(ew.view(np.float32)) if ew is not None else None))
        return img, ew

    def set_accumulators(self, intensity_dev_ptr: int, exitwave_dev_ptr: int = 0):
        """Install device accumulators (raw pointers, e.g. torch tensor .data_ptr())."""
        self._ck(self._lib.fdes_b200_set_accumulators(self._h, ctypes.c_void_p(intensity_dev_ptr or None),
                                                      ctypes.c_void_p(exitwave_dev_ptr or None)))

    def run_k(self, k: int):
        self._ck(self._lib.fdes_b200_run_k(self._h, k))

    def finish_k(self, k: int):
        img = np.zeros((self.n2, self.n1), np.float32)
        ew = np.zeros((self.m2, self.m1), np.complex64) if self.want_exitwave else None
        self._ck(self._lib.fdes_b200_finish_k(self._h, k, _fp(img),
                                              _fp(ew.view(np.float32)) if ew is not None else None))
        return img, ew

    def potential(self):
        n = self._lib.fdes_b200_potential_slices_count(self._h)
        out = np.zeros((n, self.m2, self.m1), np.complex64)
        self._ck(self._lib.fdes_b200_potential(self._h, _fp(out.view(np.float32))))
        return out

    # ---- building blocks ----------------------------------------------------------------------
    def jitter_next(self, k: int = 0):
        xyz = np.zeros((self.nAt, 3), np.float32)
        self._ck(self._lib.fdes_b200_jitter_next(self._h, k, _fp(xyz)))
        return xyz

    def bin_atoms(self, xyz: np.ndarray):
        xyz = np.ascontiguousarray(xyz, np.float32)
        bins = np.zeros((self.nAt, 4), np.int32)
        self._ck(self._lib.fdes_b200_bin_atoms(self._h, _fp(xyz), _ip(bins)))
        return bins

    def phase_grating(self, xyz: np.ndarray, s: int):
        xyz = np.ascontiguousarray(xyz, np.float32)
        V = np.zeros((self.m2, self.m1), np.complex64)
        self._ck(self._lib.fdes_b200_phase_grating(self._h, _fp(xyz), s, _fp(V.view(np.float32))))
        return V

    def exit_wave(self, xyz: np.ndarray, k: int = 0):
        xyz = np.ascontiguousarray(xyz, np.float32)
        psi = np.zeros((self.m2, self.m1), np.complex64)
        self._ck(self._lib.fdes_b200_exit_wave(self._h, _fp(xyz), k, _fp(psi.view(np.float32))))
        return psi

    def bench_configs(self, k: int, configs: int) -> float:
        ms = self._lib.fdes_b200_bench_configs(self._h, k, configs)
        if ms < 0:
            raise FdesError(self._lib.fdes_b200_last_error().decode())
        return float(ms)

    def counters(self, reset: bool = False):
        c = (ctypes.c_longlong * 4)()
        self._ck(self._lib.fdes_b200_get_counters(self._h, c, 1 if reset else 0))
        return {"slices": int(c[0]), "launches": int(c[1]), "band_columns": int(c[2])}

    def stem_scan(self, positions: np.ndarray, detectors_mrad: np.ndarray, k: int = 0):
        """STEM scan (mode 2 .cnf): positions [n, 2] in metres relative to the grid centre,
        detectors_mrad [ndet, 2] = (inner, outer).  Returns (signals [n, ndet], device ms)."""
        pos = np.ascontiguousarray(positions, np.float32).reshape(-1, 2)
        det = np.ascontiguousarray(detectors_mrad, np.float32).reshape(-1, 2)
        out = np.zeros((pos.shape[0], det.shape[0]), np.float32)
        ms = self._lib.fdes_b200_stem_scan(self._h, k, pos.shape[0], _fp(pos), det.shape[0], _fp(det), _fp(out))
        if ms < 0:
            raise FdesError(self._lib.fdes_b200_last_error().decode())
        return out, float(ms)

    def stem_scan_4d(self, positions: np.ndarray, window: int = 0, bin: int = 1, detectors_mrad=None, k: int = 0,
                     probes_per_pass: int = 0, out: Optional[np.ndarray] = None):
        """4D-STEM scan (mode 2 .cnf): the diffraction pattern of every probe, fftshifted, cropped to the centred
        window of side `window` (0: the smallest that holds the band limit) and binned bin x bin
        (fdes_b200_stem_scan_4d).  positions [n, 2] as for stem_scan; detectors_mrad [ndet, 2] (optional) adds the
        annular signals of the same pass, bitwise those of stem_scan.  out: a caller-owned float32 C-contiguous
        array [n, side, side] (e.g. an np.memmap, so that a scan larger than the RAM streams to disk).
        Returns (patterns [n, side, side], signals [n, ndet] or None, device ms)."""
        pos = np.ascontiguousarray(positions, np.float32).reshape(-1, 2)
        side = stem_4d_side(self.m1, window, bin)
        shape = (pos.shape[0], side, side)
        if out is None:
            out = np.zeros(shape, np.float32)
        elif out.dtype != np.float32 or not out.flags.c_contiguous or out.shape != shape or not out.flags.writeable:
            raise FdesError(f"out must be a writeable C-contiguous float32 array of shape {shape}")
        det = None if detectors_mrad is None else np.ascontiguousarray(detectors_mrad, np.float32).reshape(-1, 2)
        ndet = 0 if det is None else det.shape[0]
        sig = np.zeros((pos.shape[0], ndet), np.float32) if ndet else None
        ms = self._lib.fdes_b200_stem_scan_4d(self._h, k, pos.shape[0], _fp(pos), window, bin, ndet,
                                              _fp(det) if ndet else None, probes_per_pass, _fp(out),
                                              _fp(sig) if ndet else None)
        if ms < 0:
            raise FdesError(self._lib.fdes_b200_last_error().decode())
        return out, sig, float(ms)

    def time_sweeps(self, k: int = 0, batch: int = 0, reps: int = 20):
        """Average launch duration [ms] of the six per-slice sweeps S1..S6."""
        ms = np.zeros(6, np.float32)
        self._ck(self._lib.fdes_b200_time_sweeps(self._h, k, batch or self.batch, reps, _fp(ms)))
        return ms


def fft2d(a: np.ndarray, direction: int = -1, gpu_index: int = 0) -> np.ndarray:
    """2-D complex64 FFT with the library's sweeps (unnormalised; -1 forward, +1 inverse)."""
    lib = load_library()
    out = np.ascontiguousarray(a, np.complex64).copy()
    n = out.shape[0]
    assert out.shape == (n, n)
    if lib.fdes_b200_fft2d(_fp(out.view(np.float32)), n, direction, gpu_index) != 0:
        raise FdesError(lib.fdes_b200_last_error().decode())
    return out


# operations of fdes_b200_sweep_test (include/fdes_b200.h)
SWEEP_GEOM, SWEEP_DENSITY, SWEEP_POTENTIAL, SWEEP_TRANSMIT, SWEEP_BANDLIMIT, SWEEP_MULTIPLY, SWEEP_PROPAGATE, \
    SWEEP_PROPAGATE_FROM, SWEEP_COLS_FFT, SWEEP_ROWS_FFT_SUM, SWEEP_ROWS_FFT, SWEEP_PROBE, SWEEP_DETECTOR = range(13)
SWEEP_DETECTOR4D = 13
# the set-up, per-pixel and atom kernels through the same hook
SCATTER_TABLE, PROP_TABLE, LENS_TABLE, DETECTOR_TABLE, TILT_BEAM, TUKEY, AREA_MASK, NORM2, PEER_SUM, JITTER, ANSCOMBE, \
    RECORDS, PLANE_WAVE, ZERO_OUTBAND, ABSORPTIVE, SCALE_CPX = range(14, 30)
# ColOp and RowEpilogue values (fdes_b200/csrc/kernels.cuh)
COL_PLAIN, COL_MUL_CPX_INV, COL_MUL_REAL_INV, COL_DP_ACCUM = range(4)
ROW_STORE, ROW_ACCUM, ROW_INTENS_ACCUM, ROW_STORE_SHIFT, ROW_CROP_REAL = range(5)


def sweep_test(op: int, n: int, batch: int, bufs, iargs=(), fargs=(), gpu_index: int = 0, pipe_ctas: int = 0) -> int:
    """One sweep launcher run once on host arrays (fdes_b200_sweep_test).  `bufs` are C-contiguous
    complex64 / float32 / int32 arrays, uploaded, and overwritten in place with what the device holds
    after the sweep.  pipe_ctas: CTAs of a pipelined column sweep (0: one per SM as in the engine, c >= 1:
    min(c, tiles)).  Returns the grid of the pipelined launch (0: the op launched none)."""
    lib = load_library()
    for b in bufs:
        assert b.flags.c_contiguous and b.dtype in (np.complex64, np.float32, np.int32), b.dtype
    ia = np.ascontiguousarray(list(iargs) or [0], np.int32)
    fa = np.ascontiguousarray(list(fargs) or [0.0], np.float32)
    ptrs = (ctypes.POINTER(ctypes.c_float) * max(len(bufs), 1))(
        *[b.ctypes.data_as(ctypes.POINTER(ctypes.c_float)) for b in bufs])
    sizes = (ctypes.c_longlong * max(len(bufs), 1))(*[b.nbytes // 4 for b in bufs])
    grid = np.zeros(1, np.int32)
    rc = lib.fdes_b200_sweep_test(op, n, batch, _ip(ia), len(iargs), _fp(fa), len(fargs), ptrs, sizes, len(bufs),
                                  gpu_index, pipe_ctas, _ip(grid))
    if rc != 0:
        raise FdesError(lib.fdes_b200_last_error().decode())
    return int(grid[0])


def sweep_geom(n: int) -> dict:
    """The geometry the sweeps of an n x n grid run with (host only): band columns [0, lo_end) and
    [hi_start, n), points per thread of a line (0: generic sweeps), pipelined column sweeps."""
    out = np.zeros(5, np.int32)
    sweep_test(SWEEP_GEOM, n, 1, [out])
    return dict(zip(["n", "lo_end", "hi_start", "line_points", "pipelined"], map(int, out)))


def sort_records(keys: np.ndarray, cols: np.ndarray, w: np.ndarray, nkeys: int, gpu_index: int = 0):
    lib = load_library()
    k = np.ascontiguousarray(keys, np.uint32).copy()
    c = np.ascontiguousarray(cols, np.int32).copy()
    ww = np.ascontiguousarray(w, np.float32).copy()
    rp = np.zeros(nkeys + 1, np.int32)
    rc = lib.fdes_b200_sort_records(k.ctypes.data_as(ctypes.POINTER(ctypes.c_uint)), _ip(c), _fp(ww), len(k), nkeys,
                                    _ip(rp), gpu_index)
    if rc != 0:
        raise FdesError(lib.fdes_b200_last_error().decode())
    return k, c, ww, rp
