"""The pipelined column sweeps (col_pipe.cuh: S2, S4, S6, S6 from another stack, the CTF sweep at 512, 1024, 2048
and 4096) in steady state.  They run as persistent CTAs that walk tiles t, t + grid, ...; what can go wrong there
(mbarrier phases, reuse of the landing and staging buffers while a copy is in flight, the prefetch of the next
tile, S2 skipping absent species and empty images across tile boundaries) shows only from a CTA's second tile on.

(a) Every op at every pipelined size on 5 images runs under the reference schedule (one CTA per tile: nothing is
    reused) and then under grids of 1, 2, 3 and 7 CTAs, tiles - 1 (one CTA takes two tiles), the engine's default
    (one CTA per SM) and 149 CTAs (a second wave).  Every buffer -- outputs, sentinel and NaN regions, the source
    stacks -- must be bitwise the reference schedule's; the reference schedule and grid 1 are also compared with
    the float64 models of oracle/sweep_model.py on the first and last image.  The grid that ran is asserted for
    every schedule (fdes_b200_sweep_test reports it).
(b) The batches the engine launches (40 images at 512 and 1024, 20 at 2048, 10 at 4096) at the default grid,
    bitwise against the reference schedule, and the first, middle and last image against the float64 model.
(c) Whole simulations at the pipelined sizes (frozen phonons, an even slice count, a defocus series, three
    automatic batches with a partial last one) are bitwise the same for batch 1, 7 and automatic and from one
    session to the next, with and without the exit wave kept; two engines on one device repeat themselves.

Setting FDES_PIPE_SCHEDULES=<file.json> records the grids each case ran with.  The run of this file on an NVIDIA
B200 (148 SMs, 1000 W power limit) took 6.1 min, a third of it in the 4096² cases.
"""
import hashlib
import json
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import sweep_model as sm
from conftest import rel_l2
from sweep_cases import (FROM_VARIANTS, NSL, PIPELINED, SENT, band_of, check_lines, confs_of, crand, geom, make_records,
                         nz_of, random_pq, stack_with_nan)

pytestmark = pytest.mark.gpu

BATCH = 5                                       # (a): an odd batch
ENGINE_BATCH = {512: 40, 1024: 40, 2048: 20, 4096: 10}
S2_PAIRINGS = {"pair": (0, 1, 1, 0), "single": (2, -1, 1, 0), "configs": (2, 2, 2, 1)}  # slice slice2 cfg_stride off2
S2_NCONF = 10                                   # (2, 1) pairing of 5 images: configurations 0 .. 9
S2_EMPTY = (0, 2, 3)                            # configurations without any deposit: at the start and in the middle
_SCHEDULES = {}


@pytest.fixture(scope="module", autouse=True)
def _record_schedules():
    yield
    path = os.environ.get("FDES_PIPE_SCHEDULES")
    if path:
        with open(path, "w") as f:
            json.dump(_SCHEDULES, f, indent=1, sort_keys=True)


@pytest.fixture(scope="module")
def fbm():
    import fdes_b200
    return fdes_b200


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def digests(a):
    """One digest per image (leading axis) of a stack, one for the whole of a table."""
    a = np.ascontiguousarray(a)
    parts = [a[i] for i in range(a.shape[0])] if a.ndim >= 3 else [a]
    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        return list(ex.map(lambda p: hashlib.sha1(memoryview(p).cast("B")).digest(), parts))


# ---------------------------------------------------------------------------------------------------
# cases: buffers of fdes_b200_sweep_test, the indices it writes, tile count, per-image model check
# ---------------------------------------------------------------------------------------------------
class Case:
    def __init__(self, name, op, n, batch, bufs, written, ntiles, check, ia=(), fa=()):
        self.name, self.op, self.n, self.batch = name, op, n, batch
        self.bufs, self.written, self.ntiles, self.ia, self.fa = bufs, written, ntiles, list(ia), list(fa)
        self.check = check          # check(b, bufs after the sweep): image b against the float64 model + regions


def tile_width(n):
    return 8192 // n                            # PipeCfg<N>::CW


def band_tiles(fb, n):
    g = geom(fb, n)
    cols = n if g["lo_end"] >= g["hi_start"] else g["lo_end"] + n - g["hi_start"]
    return cols // tile_width(n)


def cached(f):
    memo = {}
    return lambda b: memo[b] if b in memo else memo.setdefault(b, f(b))


_RECORDS = {}


def s2_case(fb, n, batch, pairing, seed):
    slice_, slice2, cs, off = S2_PAIRINGS[pairing]
    nz = nz_of(n)
    nconf = max(S2_NCONF, (batch - 1) * cs + off + 1)
    if (n, nconf) not in _RECORDS:
        _RECORDS[n, nconf] = make_records(n, nz, 1000 + n, nconf, S2_EMPTY)[0]
    rowptr = _RECORDS[n, nconf]
    rng = np.random.default_rng(seed)
    Q = n // 2 + 1
    Gq = rng.random((nz, Q * Q)).astype(np.float32)
    A = np.empty((batch, nz, n, n), np.complex64)
    for b in range(batch):
        ca, cb = b * cs, b * cs + off
        for z in range(nz):
            A[b, z] = crand(rng, (n, n))
            keep = sm.deposit_rows(rowptr, n, nz, z, slice_, ca)
            if slice2 >= 0:
                keep |= sm.deposit_rows(rowptr, n, nz, z, slice2, cb)
            A[b, z][~keep] = np.nan             # rows S1 did not write: never read
    B0 = np.full((batch, n, n), SENT, np.complex64)

    @cached
    def model(b):
        cf = confs_of(b, cs, off)
        return sm.s2_potential_cols(A[b:b + 1], Gq, rowptr[cf], n, nz, 1, slice_, slice2, cs, off)[0]

    def check(b, out):
        ref = model(b)
        if not ref.any():                       # no species present in the image: exact zeros
            assert (out[0][b] == 0).all(), f"S2 {pairing} {n}: image {b} holds no deposit and must be zero"
        else:
            check_lines("S2", n, out[0][b][None], ref[None], rows_axis=False)

    ia = [slice_, slice2, nz, NSL, cs, off, nconf]
    return Case(f"S2 {pairing}", fb.SWEEP_POTENTIAL, n, batch, [B0, A, Gq, rowptr], {0}, (n // tile_width(n)) * batch,
                check, ia)


def s4_case(fb, n, batch, npair, seed):
    rng = np.random.default_rng(seed)
    band = band_of(fb, n)
    images = batch if npair == 0 else 2 * batch
    entries = sm.stack_entries(batch, npair)
    W = stack_with_nan(rng, n, images, entries, band)

    def mine(b):
        return [b] if npair == 0 else [2 * b + p for p in range(npair)]

    @cached
    def model(b):
        return np.stack([sm.s4_bandlimit_cols(np.where(band, W[e], 0)[None], 0, 1)[0] for e in mine(b)])

    def check(b, out):
        got = out[0][mine(b)]
        check_lines("S4", n, got, model(b), cols=band, rows_axis=False)
        assert np.isnan(got[..., ~band]).all()                      # outside the band: not read, not written
        if npair:
            skipped = [2 * b + p for p in range(npair, 2)]
            assert np.isnan(out[0][skipped]).all()                  # slots the pairing skips

    ntiles = band_tiles(fb, n) * (batch if npair == 0 else batch * npair)
    return Case(f"S4 npair {npair}", fb.SWEEP_BANDLIMIT, n, batch, [W], {0}, ntiles, check, [npair])


def s6_case(fb, n, batch, seed):
    rng = np.random.default_rng(seed)
    band = band_of(fb, n)
    Psi = stack_with_nan(rng, n, batch, range(batch), band)
    Pq = random_pq(rng, n)

    @cached
    def model(b):
        return sm.s6_propagate_cols(Psi[b:b + 1], Pq, band)[0]

    def check(b, out):
        check_lines("S6", n, out[0][b][None], model(b)[None], cols=band, rows_axis=False)
        assert np.isnan(out[0][b][..., ~band]).all()

    return Case("S6", fb.SWEEP_PROPAGATE, n, batch, [Psi, Pq], {0}, band_tiles(fb, n) * batch, check)


def s6_from_case(fb, n, batch, variant, seed):
    stride, times_n, use_lens = FROM_VARIANTS[variant]
    rng = np.random.default_rng(seed)
    band = band_of(fb, n)
    images = (batch - 1) * stride + 1
    src = stack_with_nan(rng, n, images, range(0, images, stride), band)
    Pq = random_pq(rng, n)
    lens = crand(rng, (n, n)) if use_lens else np.zeros(0, np.complex64)
    out0 = np.full((batch, n, n), SENT, np.complex64)

    @cached
    def model(b):
        return sm.s6_propagate_cols_from(src[b * stride:b * stride + 1], 1, 1, Pq, band, times_n,
                                         lens if use_lens else None)[0]

    def check(b, out):
        check_lines("S6 from", n, out[0][b][None], model(b)[None], cols=band, rows_axis=False)
        assert (out[0][b][..., ~band] == SENT).all()

    return Case(f"S6 from {variant}", fb.SWEEP_PROPAGATE_FROM, n, batch, [out0, src, Pq, lens], {0},
                band_tiles(fb, n) * batch, check, [stride, images, int(times_n)])


def ctf_case(fb, n, batch, seed):
    rng = np.random.default_rng(seed)
    band = band_of(fb, n)
    x = stack_with_nan(rng, n, batch, range(batch), band)      # the pipelined sweep must not read outside the band
    tab = crand(rng, (n, n))
    scale = np.float32(1.0 / n)
    out0 = np.full((batch, n, n), SENT, np.complex64)

    @cached
    def model(b):
        return sm.cols_mul_cpx_inv(np.where(band, x[b:b + 1], 0), tab, float(scale), band)[0]

    def check(b, out):
        check_lines("CTF", n, out[1][b][None], model(b)[None], cols=band, rows_axis=False)
        assert (out[1][b][..., ~band] == SENT).all()

    return Case("CTF", fb.SWEEP_COLS_FFT, n, batch, [x, out0, tab], {1}, band_tiles(fb, n) * batch, check,
                [fb.COL_MUL_CPX_INV, -1], [scale])


def make_case(fb, n, batch, kind, seed):
    op, _, arg = kind.partition(":")
    if op == "S2":
        return s2_case(fb, n, batch, arg, seed)
    if op == "S4":
        return s4_case(fb, n, batch, int(arg), seed)
    if op == "S6":
        return s6_case(fb, n, batch, seed)
    if op == "S6from":
        return s6_from_case(fb, n, batch, arg, seed)
    return ctf_case(fb, n, batch, seed)


KINDS = ([f"S2:{p}" for p in S2_PAIRINGS] + [f"S4:{k}" for k in (0, 1, 2)] + ["S6"] +
         [f"S6from:{v}" for v in FROM_VARIANTS] + ["CTF"])


# ---------------------------------------------------------------------------------------------------
# schedules
# ---------------------------------------------------------------------------------------------------
def launch(fb, case, ctas, in_digests):
    """One launch with pipe_ctas = ctas on fresh copies of the written buffers; the read-only buffers go in as
    they are and must come back unchanged.  Returns (buffers after the sweep, grid that ran)."""
    cur = [b.copy() if i in case.written else b for i, b in enumerate(case.bufs)]
    grid = fb.sweep_test(case.op, case.n, case.batch, cur, case.ia, case.fa, pipe_ctas=ctas)
    for i, d in in_digests.items():
        changed = [k for k, (x, y) in enumerate(zip(digests(cur[i]), d)) if x != y]
        assert not changed, f"{case.name} {case.n}, {ctas} CTAs: read-only buffer {i} changed (images {changed})"
    return cur, grid


def run_schedules(fb, case, schedules, expected, model_images, model_grids=()):
    """The reference schedule (one CTA per tile), then each of `schedules` (pipe_ctas values); every written buffer
    bitwise against the reference schedule's, per image.  The images `model_images` of the reference schedule
    (and of the schedules in model_grids) are checked against the float64 model.  Returns {pipe_ctas: grid}."""
    in_digests = {i: digests(b) for i, b in enumerate(case.bufs) if i not in case.written}
    ref, grid = launch(fb, case, case.ntiles, in_digests)
    assert grid == case.ntiles, f"{case.name} {case.n}: reference schedule ran {grid} CTAs for {case.ntiles} tiles"
    for b in model_images:
        case.check(b, ref)
    ref_digests = {i: digests(ref[i]) for i in case.written}
    del ref
    grids = {}
    for c in schedules:
        cur, grid = launch(fb, case, c, in_digests)
        grids[c] = grid
        assert grid == expected(c), f"{case.name} {case.n}: pipe_ctas {c} ran {grid} CTAs, expected {expected(c)}"
        for i, d in ref_digests.items():
            diff = [k for k, (x, y) in enumerate(zip(digests(cur[i]), d)) if x != y]
            assert not diff, (f"{case.name} {case.n}: {grid} CTAs over {case.ntiles} tiles differ from one CTA per "
                              f"tile in buffer {i}, images {diff}")
        if c in model_grids:
            for b in model_images:
                case.check(b, cur)
    _SCHEDULES.setdefault(case.name, {})[f"{case.n} x{case.batch}"] = {"tiles": case.ntiles, "grids": grids}
    return grids


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", PIPELINED)
def test_tile_schedules_are_bit_identical(fbm, sms, n, kind):
    """(a): grids 1, 2, 3, 7, tiles - 1, the default and 149 against one CTA per tile, 5 images."""
    case = make_case(fbm, n, BATCH, kind, 11000 + n + KINDS.index(kind))
    T = case.ntiles
    schedules = [1, 2, 3, 7, T - 1, 0, 149]
    grids = run_schedules(fbm, case, schedules, lambda c: min(c if c > 0 else sms, T), [0, BATCH - 1],
                          model_grids=(1,))
    # the schedules reached the steady state: a CTA with every tile, shares that do not divide the tiles, and at
    # least 3 tiles on one CTA
    assert grids[1] == 1
    assert any(T % g for g in grids.values())
    assert max(-(-T // g) for g in grids.values()) >= 3


@pytest.mark.parametrize("kind", ["S2:pair", "S4:2", "S6", "S6from:ctf_last", "CTF"])
@pytest.mark.parametrize("n", PIPELINED)
def test_engine_batches_match_one_cta_per_tile(fbm, sms, n, kind):
    """(b): the batch the engine launches at this size, at the default grid (one CTA per SM), against one CTA per
    tile.  (The S4 pair stack at 4096 holds 10 images for 5 configurations, to keep the host memory of the test to
    a few GB.)"""
    batch = ENGINE_BATCH[n]
    if kind == "S4:2" and n == 4096:
        batch = 5
    case = make_case(fbm, n, batch, kind, 12000 + n)
    run_schedules(fbm, case, [0], lambda c: min(sms, case.ntiles), [0, batch // 2, batch - 1])


# ---------------------------------------------------------------------------------------------------
# (c) whole simulations
# ---------------------------------------------------------------------------------------------------
ENGINE_CONFIGS = {512: 85, 1024: 85, 2048: 45, 4096: 25}       # automatic batch 40 / 40 / 20 / 10: 3 batches


def engine_cnf(n, tmp_path):
    from fdes_b200 import specimens
    d = 0.2e-10 if n <= 1024 else 0.1e-10
    atoms = specimens.random_slab(40, n * d, 2 * 2e-10, seed=n, species=(79, 14))
    return specimens.write_cnf(tmp_path / f"det{n}.cnf", image_size=n // 2, border_size=n // 4, slices=2,
                               pixel_size=d, slice_thickness=2e-10, atoms=atoms, voltage=200e3, absorptive=0.03,
                               frozen_phonons=ENGINE_CONFIGS[n], image_size_z=2, defoci=[0.0, -5e-9],
                               objective_aperture=0.02, aberrations={"C3": (1e-3, 0.0)})


def same(a, b):
    return a is None and b is None or np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32))


@pytest.mark.parametrize("n", PIPELINED)
def test_simulations_are_bit_identical_across_batches_and_sessions(fbm, n, tmp_path):
    """Batch 1, 7 and automatic (twice, separate sessions), with the exit wave kept and without (the CTF fused into
    the last S6): bitwise the same within each setting.  An even slice count: with an odd one the last slices of
    configurations 2j and 2j + 1 share a transform, which changes the rounding (bounded elsewhere)."""
    cnf = engine_cnf(n, tmp_path)
    for keep_ew in (True, False):
        out = {}
        for key, batch in (("1", 1), ("7", 7), ("auto", 0), ("auto again", 0)):
            with fbm.Simulation(cnf, want_exitwave=keep_ew, batch=batch) as sim:
                assert sim.m1 == n and sim.m3 == 2 and sim.n3 == 2
                if batch == 0:
                    assert sim.batch == ENGINE_BATCH[n] and sim.configs % sim.batch and sim.configs > 2 * sim.batch
                out[key] = sim.simulate()
        img, ew = out["auto"]
        assert np.isfinite(img).all() and img.mean() > 0.1
        for key in ("1", "7", "auto again"):
            assert same(out[key][0], img), f"{n}, exit wave kept {keep_ew}: images of batch {key} differ"
            assert same(out[key][1], ew), f"{n}, exit wave kept {keep_ew}: exit waves of batch {key} differ"


def test_two_engines_on_one_device_repeat_themselves_at_1024(fbm, tmp_path):
    cnf = engine_cnf(1024, tmp_path)
    with fbm.Simulation(cnf, want_exitwave=True) as sim:
        img, ew = sim.simulate()
    with fbm.Simulation(cnf, want_exitwave=True, gpus=[0, 0]) as sim:
        assert sim.num_gpus == 2
        img2, ew2 = sim.simulate()
        img3, ew3 = sim.simulate()
    assert same(img2, img3) and same(ew2, ew3)
    assert rel_l2(ew2, ew) < 1e-6 and rel_l2(img2, img) < 1e-6
