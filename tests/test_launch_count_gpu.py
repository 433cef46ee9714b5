"""The reported launch count (counters()["launches"], fdes_b200_get_counters, bench.py gpu_launches) against the
kernels the GPU actually ran: torch.profiler with CUDA activities records every kernel, those replayed from CUDA
graphs included, and each step below -- opening the session first, so the constructor is covered -- must show
exactly as many kernels of the library (names containing "fdes::") as the session counted, and no other kernel.
"""
import re

import numpy as np
import pytest
import torch
from torch.autograd import DeviceType
from torch.profiler import ProfilerActivity, profile

from fdes_b200 import specimens

pytestmark = pytest.mark.gpu


def profiled(step):
    """Runs step() under the profiler; returns (its result, names of the kernels the GPU ran)"""
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = step()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA]
    return out, [n for n in names if not n.startswith(("Memcpy", "Memset"))]


def check_launches(fb, cnf, steps, **session):
    """Opens a session on cnf and runs steps [(label, f(sim))] in turn, each in a profiler of its own"""
    sim, kernels = profiled(lambda: fb.Simulation(cnf, **session))
    try:
        for label, step in [("open", None)] + steps:
            if step is not None:
                _, kernels = profiled(lambda: step(sim))
            counted = sim.counters(reset=True)["launches"]
            others = sorted({k for k in kernels if "fdes::" not in k})
            assert not others, f"{label}: kernels outside the library: {others}"
            assert counted == len(kernels), f"{label}: {counted} launches counted, {len(kernels)} kernels ran"
            assert counted > 0, label
    finally:
        sim.close()


def slab_cnf(path, n, border, slices, seed, **kw):
    d = 0.25e-10
    m = n + 2 * border
    atoms = specimens.random_slab(60, m * d * 0.8, slices * 2e-10, seed=seed, species=(79, 14, 8))
    return specimens.write_cnf(path, image_size=n, border_size=border, slices=slices, pixel_size=d, slice_thickness=2e-10,
                               atoms=atoms, **kw)


def with_dose(cnf, dose):
    text, n = re.subn(r"(?m)^pixel_dose: .*$", f"pixel_dose: {dose}", cnf.read_text())
    assert n == 1
    cnf.write_text(text)
    return cnf


def test_graph_path_with_phonons_odd_slices_and_exit_wave(fb, tmp_path):
    """128^2, 6 configurations in batches of 4 and 2 (one graph per record set), 5 slices (the odd last slices of two
    configurations share a transform), exit wave kept, pixel dose > 0: the first run_k runs the sweeps plainly, the
    second captures and launches the graphs, the third replays them"""
    cnf = with_dose(slab_cnf(tmp_path / "g.cnf", 64, 32, 5, seed=1, frozen_phonons=6), 500.0)
    xyz = np.zeros((60, 3), np.float32)
    steps = [(f"run_k #{i}", lambda s: s.run_k(0)) for i in range(3)]
    steps += [("finish_k", lambda s: s.finish_k(0)),
              ("simulate", lambda s: s.simulate()),
              ("bench_configs", lambda s: s.bench_configs(0, 6)),
              ("bench_configs again", lambda s: s.bench_configs(0, 6)),
              ("potential", lambda s: s.potential()),
              ("phase_grating", lambda s: s.phase_grating(xyz, 2)),
              ("exit_wave", lambda s: s.exit_wave(xyz)),
              ("time_sweeps", lambda s: s.time_sweeps(0, 2, 3))]
    check_launches(fb, cnf, steps, batch=4, want_exitwave=True)


def test_pipelined_imaging_without_exit_wave(fb, tmp_path):
    """512^2, 10 configurations in one batch: plain launches, the first slice without S5, the CTF on the last S6"""
    cnf = slab_cnf(tmp_path / "p.cnf", 256, 128, 4, seed=2, frozen_phonons=10)
    steps = [("run_k", lambda s: s.run_k(0)), ("finish_k", lambda s: s.finish_k(0)),
             ("bench_configs", lambda s: s.bench_configs(0, 10)), ("bench_configs again", lambda s: s.bench_configs(0, 10))]
    check_launches(fb, cnf, steps)


def test_generic_odd_size_cbed_with_beam_tilt(fb, tmp_path):
    """143^2 (generic sweeps), CBED with beam tilt: the incident probe and the diffraction-pattern tail of mode 2"""
    cnf = slab_cnf(tmp_path / "c.cnf", 99, 22, 3, seed=3, mode=2, objective_aperture=15e-3, beam_tilts=[(2e-3, -1e-3)])
    steps = [("run_k", lambda s: s.run_k(0)), ("finish_k", lambda s: s.finish_k(0)),
             ("bench_configs", lambda s: s.bench_configs(0, 1))]
    check_launches(fb, cnf, steps)


def test_stem_scans_with_detectors(fb, tmp_path):
    """stem_scan and stem_scan_4d with annular detectors, two configurations, the 4D scan in three passes"""
    cnf = slab_cnf(tmp_path / "s.cnf", 128, 0, 3, seed=4, mode=2, objective_aperture=12e-3, frozen_phonons=2)
    pos = np.array([[0.0, 0.0], [1e-10, 0.0], [0.0, 2e-10], [-1e-10, 1e-10], [2e-10, -2e-10]], np.float32)
    det = np.array([[0.0, 10.0], [20.0, 60.0]], np.float32)
    steps = [("stem_scan", lambda s: s.stem_scan(pos, det)),
             ("stem_scan_4d", lambda s: s.stem_scan_4d(pos, window=0, bin=2, detectors_mrad=det, probes_per_pass=2)),
             ("stem_scan_4d without detectors", lambda s: s.stem_scan_4d(pos, bin=1))]
    check_launches(fb, cnf, steps, batch=2)
