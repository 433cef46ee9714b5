"""Inputs, launch helper and error bounds of the per-sweep GPU tests (test_sweeps_fp64_gpu.py,
test_col_pipeline_gpu.py): every sweep runs once through the C ABI test hook fdes_b200_sweep_test and is
compared with the float64 models of oracle/sweep_model.py.

Conventions: NaN wherever a sweep must not read (rows of A without deposit records, columns outside the band,
image slots a stride skips); the sentinel SENT wherever it must not write."""
import numpy as np

import sweep_model as sm

PIPELINED = [512, 1024, 2048, 4096]         # column sweeps on the TMA pipeline (persistent CTAs)
SENT = np.complex64(complex(1234.5, -777.25))

# Bounds of the per-line metric ||err_line|| / (rms(ref) sqrt(L)) and of the global rel-L2 per op, about three times
# the largest value over all fifteen sizes of test_sweeps_fp64_gpu.py measured on an NVIDIA B200 (1000 W power
# limit); the run of that file there took 5.3 min.  op: (measured line, at size; measured global, at size) -> bounds
# in TAU / GLOB
MEASURED = {
    "S1": (2.7e-6, 2048, 1.7e-7, 1022),         # lines with few deposits carry a small share of rms(ref)
    "S2": (2.3e-7, 143, 1.8e-7, 4096),
    "S3": (9.3e-7, 143, 6.3e-7, 143),
    "S4": (2.9e-7, 143, 1.8e-7, 4096),
    "S5": (3.0e-7, 143, 2.4e-7, 2048),
    "S6": (2.5e-7, 143, 1.9e-7, 4096),
    "S6 from": (2.2e-7, 1024, 1.9e-7, 4096),
    "CTF": (2.3e-7, 143, 1.9e-7, 4096),
    "DP accum": (3.2e-8, 96, 2.7e-8, 320),
    "rows sum": (1.6e-7, 143, 1.1e-7, 4096),
}
TAU = {"S1": 8e-6, "S2": 7e-7, "S3": 3e-6, "S4": 9e-7, "S5": 9e-7, "S6": 8e-7, "S6 from": 7e-7, "CTF": 7e-7,
       "DP accum": 1e-7, "rows sum": 5e-7}
GLOB = {"S1": 5e-7, "S2": 5e-7, "S3": 2e-6, "S4": 5e-7, "S5": 7e-7, "S6": 6e-7, "S6 from": 6e-7, "CTF": 6e-7,
        "DP accum": 8e-8, "rows sum": 3.5e-7}
ERRORS = {}         # this run's errors per op and size (FDES_SWEEP_ERRORS in test_sweeps_fp64_gpu.py)


def record(op, n, **vals):
    d = ERRORS.setdefault(op, {}).setdefault(str(n), {})
    for k, v in vals.items():
        d[k] = max(float(v), d.get(k, 0.0))


_GEOM = {}


def geom(fb, n):
    if n not in _GEOM:
        _GEOM[n] = fb.sweep_geom(n)
    return _GEOM[n]


def band_of(fb, n):
    g = geom(fb, n)
    return sm.band_columns(n, g["lo_end"], g["hi_start"])


def crand(rng, shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)


def check_lines(op, n, out, ref, cols=None, rows_axis=True, line_mask=None):
    """Per-line and global error of out against ref over the columns `cols` (all if None); lines are rows
    (rows_axis) or columns.  line_mask [..., N] restricts the lines compared (rows of S1)."""
    out = np.asarray(out)
    ref = np.asarray(ref)
    if cols is not None:
        out, ref = out[..., cols], ref[..., cols]
    assert not np.isnan(out).any(), f"{op} {n}: NaN in the output"
    err = out.astype(np.complex128) - ref
    if line_mask is not None:
        err, refm = err[line_mask], ref[line_mask]
    else:
        refm = ref
    rms = np.sqrt(np.mean(np.abs(refm) ** 2))
    if rows_axis:
        per, L = np.linalg.norm(err, axis=-1), err.shape[-1]
    else:
        per, L = np.linalg.norm(err, axis=-2), err.shape[-2]
    line = float(per.max() / (rms * np.sqrt(L)))
    glob = float(np.linalg.norm(err) / np.linalg.norm(refm))
    record(op, n, line=line, glob=glob)
    assert line <= TAU[op], f"{op} {n}: per-line error {line:.3e}"
    assert glob <= GLOB[op], f"{op} {n}: global rel-L2 {glob:.3e}"


def run(fb, op, n, batch, bufs, iargs=(), fargs=()):
    """Launch on copies; returns the buffers after the sweep."""
    cp = [np.ascontiguousarray(b).copy() for b in bufs]
    fb.sweep_test(op, n, batch, cp, iargs, fargs)
    return cp


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint32), np.ascontiguousarray(b).view(np.uint32))


def nz_of(n):
    return 2 if n >= 4096 else 4


# ---------------------------------------------------------------------------------------------------
# deposit records (S1 / S2)
# ---------------------------------------------------------------------------------------------------
NSL = 3
NCONF = 6
# species present per slice (configuration 1 has no deposit at all).  The pair (0, 1): species 0 in both, 1 only
# in the second slice, 2 in neither, 3 only in the first.  Slice 2 alone or paired with itself: species 0 (and 3),
# 1 and 2 absent -- so with the two species of 4096 both edges remain: 1 only in the second slice of the pair,
# 1 absent from slice 2.
PRESENT = {0: {0, 3}, 1: {0, 1}, 2: {0, 3}}


def make_records(n, nz, seed, nconf=NCONF, empty=(1,)):
    """Sorted deposit records of `nconf` configurations (those in `empty` without any deposit): row pointers
    [nconf][NSL * nz * n + 1], columns and weights [nconf][rec_stride]."""
    rng = np.random.default_rng(seed)
    special = sorted({r for r in (0, 1, 3, 4, 7, 8, 31, 32, 63, 64, n // 2 - 1, n // 2, n - 2, n - 1) if 0 <= r < n})
    per = []
    for c in range(nconf):
        keys, cols, ws = [], [], []
        if c not in empty:
            for s in range(NSL):
                for z in range(nz):
                    if z not in PRESENT[s]:
                        continue
                    rows = set(special) | set(rng.choice(n, max(n // 16, 1), replace=False).tolist())
                    for r in sorted(rows):
                        k = int(rng.integers(1, 4))
                        keys += [(s * nz + z) * n + r] * k
                        cols += rng.integers(0, n, k).tolist()
                        ws += (rng.random(k) + 0.1).tolist()
                    keys += [(s * nz + z) * n + n // 2] * 40          # many records on one pixel
                    cols += [min(5, n - 1)] * 40
                    ws += rng.random(40).tolist()
        per.append((np.array(keys, np.int64), np.array(cols, np.int32), np.array(ws, np.float32)))
    rec_stride = max(len(k) for k, _, _ in per)
    nkeys = NSL * nz * n
    rowptr = np.zeros((nconf, nkeys + 1), np.int32)
    cols = np.zeros((nconf, rec_stride), np.int32)
    w = np.zeros((nconf, rec_stride), np.float32)
    for c, (k, cc, ww) in enumerate(per):
        o = np.argsort(k, kind="stable")
        rowptr[c] = np.searchsorted(k[o], np.arange(nkeys + 1))
        cols[c, :len(k)] = cc[o]
        w[c, :len(k)] = ww[o]
    return rowptr, cols, w


_RECORDS = {}


def records(n):
    if n not in _RECORDS:
        _RECORDS[n] = make_records(n, nz_of(n), 1000 + n)
    return _RECORDS[n]


def confs_of(b, cs, off):
    return [b * cs] if off == 0 else [b * cs, b * cs + off]


FROM_VARIANTS = {          # (src_img_stride, times_n, lens): first slice of a pair / of the odd pairing, the CTF
    "pair_first": (2, True, False),
    "odd_first": (1, True, False),
    "ctf_last": (1, False, True),
    "single_slice": (2, True, True),
}


def stack_with_nan(rng, n, images, entries, band):
    W = np.full((images, n, n), np.nan + 1j * np.nan, np.complex64)
    for e in entries:
        W[e] = crand(rng, (n, n))
        W[e][:, ~band] = np.nan
    return W


def random_pq(rng, n):
    Q = n // 2 + 1
    return crand(rng, Q * Q) / np.float32(n)
