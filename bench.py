#!/usr/bin/env python3
"""Benchmark of the FDES forward-multislice hot path (BASELINE.json metric: multislice
Mpixel*slices/s) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload si001_1024] [--impl reference]
                    [--dump-outputs DIR]

--steps K sets the timed steps of `value` and `e2e`; the `stem` and `job` legs time one call each
whatever K is.  --warmup W runs max(W, 3) untimed steps before `value` with --impl ours.

A *step* is one pass of the hot path over one batch of synthetic input: `configs_per_step`
frozen-phonon configurations of the workload specimen per GPU (400 for the default workload, so that
the 20 timed steps of the driver last about two seconds), each a complete multislice run (atom
jitter -> binning/sort -> per slice: projected potential, band-limited transmission, Fresnel
propagation -> detector accumulation).  Frozen-phonon configurations are independent, so N GPUs
process N x configs_per_step configurations per step with no data-path collective (weak scaling).
With N > 1 the line also carries `job`: BASELINE configs[2] (Au 2048^2, 32 configurations) and
configs[3] (256 x 256 STEM probes) each run as ONE job sharded over the N ranks, with the all-reduce
of the partial intensities / the all-gather of the detector signals inside the timed region (strong
scaling; at N = 1 the same jobs give the single-GPU reference time).

  value  whole-job Mpx*slices/s with the specimen resident in HBM, CUDA-event time of the steps,
         max over ranks.
  e2e    same metric through the drop-in C-ABI call FDES() (include/fdes_b200.h; reference
         src/FDESExport.cu:59-178): parameter file + host atom array in, host image out; session
         set-up, host->device and device->host copies and the side-effect files are inside the
         timed region (wall clock).
  roofline      the six sweeps of one slice (one launch each over the batch): algorithmic bytes
                (SURVEY 8d: 16 nZ + 80 B per pixel and slice) / the sum of their live CUDA-event launch
                times, against the measured HBM peak and the nominal 8 TB/s of north_star; the
                per-sweep table and the whole-step figure (value x bytes) are reported next to it.
  --dump-outputs DIR  (rank 0) what the timed calls returned in their last step, as DIR/<name>.npy:
                image (finish_k of the last step's configurations: the phonon-averaged image [n2, n1]),
                e2e_image (FDES() [1, n2, n1]), stem_signals and the job outputs when those legs run.  The
                inputs are generated from fixed seeds, so two builds run with the same arguments can be
                compared output for output.
  cpu_baseline  the numpy/pocketfft restatement (oracle/fdes_oracle.py) on this box's host cores,
                bounded sample, rank 0 at N=1 only.  Reported baseline, not a target.

`--impl reference` times the UNMODIFIED reference (oracle/_ref/ref_harness, built from
/root/reference by oracle/Makefile: cuFFT + cuBLAS + its own kernels) on the same workload.  FDES
has no CPU implementation -- its own implementation of this path is that single-GPU CUDA program
-- so the reference arm runs on GPU 0 of the box (rank 0 only), whole-call wall time of the
reference's exported flow (ref_harness e2e), which is what `e2e` of this arm is compared with.
Its `config` is the one of our arm; a step of it is a bounded sample of that workload (16 of the 400
configurations per call: the reference needs about 0.1 s per configuration, and 16 per call keep
its fixed per-call cost below 5 % of the call).
"""
import argparse
import json
import os
import pathlib
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "multislice_Mpixel_slices_per_s"
UNIT = "Mpx*slices/s"

WORKLOADS = {
    # name: (builder, description, species count)
    "srtio3_800": ("config_srtio3_800", "SrTiO3 9x9x20 cells 8100 atoms / 3 species, 800^2 grid, 40 x 1.9525 A slices in 400 "
                                        "sub-slices, 200 kV (BASELINE configs[0] geometry in .cnf form)"),
    "si001_1024": ("config_si001_1024", "Si[001] 11552 atoms, 1024^2 grid, 11 x 2 A slices, 100 kV (BASELINE configs[1])"),
    "au_2048": ("config_au_2048", "Au cuboctahedron 309 atoms, 2048^2 grid, 12 x 2.1 A slices, 50 kV (BASELINE configs[2])"),
    "slab_4096": ("config_random_4096_short", "random slab 4000 atoms / 3 species, 4096^2 grid, 20 x 2 A slices, 200 kV "
                                             "(BASELINE configs[4] geometry, 20 of its 500 slices, same areal density)"),
    "slab_4096_full": ("config_random_4096", "random slab 100000 atoms / 3 species, 4096^2 grid, 500 x 2 A slices, 200 kV "
                                            "(BASELINE configs[4] at its named size)"),
}
DEFAULT_CONFIGS_PER_STEP = {"srtio3_800": 20, "si001_1024": 400, "au_2048": 80, "slab_4096": 20, "slab_4096_full": 2}
REF_SAMPLE_CONFIGS = {"srtio3_800": 1, "si001_1024": 16, "au_2048": 4, "slab_4096": 1, "slab_4096_full": 1}


def peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        return float(json.loads(f.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.stop, self.th = gpu_index, [], threading.Event(), None

    def _loop(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.gpu)], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    self.rows.append([c.strip() for c in line.split(",")])
            except Exception:
                pass
            self.stop.wait(0.1)

    def __enter__(self):
        self.th = threading.Thread(target=self._loop, daemon=True)
        self.th.start()
        return self

    def __exit__(self, *exc):
        self.stop.set()
        self.th.join(timeout=10)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[1]) for r in self.rows)
        reasons = set()
        for r in self.rows:
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                              ("sw_power_cap", 8)):
                if r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][2]), "reasons": sorted(reasons),
                "samples": len(self.rows), "power_w_max": max(float(r[3]) for r in self.rows)}


def algorithmic_bytes_per_px(nZ):
    """SURVEY.md section 8(d) / DESIGN.md: bytes per pixel and slice of each sweep."""
    return {"S1_density_rows": 8 * nZ, "S2_potential_cols": 8 * nZ + 8, "S3_transmit_rows": 16,
            "S4_bandlimit_cols": 16, "S5_multiply_rows": 24, "S6_propagate_cols": 16}


def workload_config(a, cps, world):
    """`config` of the JSON line: identical in our arm and in the reference arm."""
    return {"workload": a.workload, "description": WORKLOADS[a.workload][1],
            "configs_per_step_per_gpu": cps, "parallelism": f"phonon-configs x{world}",
            "l2": "no explicit flush: every sweep streams a batched working set of several hundred MiB of wave / "
                  "potential grids (126 MB L2) and every step draws new atom positions"}


def run_ours(a):
    import torch
    import torch.distributed as dist
    import fdes_b200 as fb
    from fdes_b200 import specimens

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (fdes_b200 has no CPU path)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cps = a.configs_per_step or DEFAULT_CONFIGS_PER_STEP[a.workload]
    tmp = pathlib.Path(tempfile.mkdtemp(prefix=f"fdes_bench_r{rank}_"))
    cnf = tmp / f"{a.workload}.cnf"
    atoms = getattr(specimens, WORKLOADS[a.workload][0])(cnf, frozen_phonons=cps)
    atoms6 = np.ascontiguousarray(atoms, np.float32)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sim = fb.Simulation(cnf, atoms6=atoms6, gpu_index=local, batch=a.batch)
    px = sim.m1 * sim.m2
    slices_per_step = sim.m3 * cps
    for _ in range(a.warmup):
        sim.bench_configs(0, cps)
    sim.counters(reset=True)
    outputs = {}
    with ClockSampler(local) as clk:
        time.sleep(0.3)            # let the sampler take its first reading before the timed region
        barrier()
        t_wall = time.perf_counter()
        dev_ms = 0.0
        for _ in range(a.steps):
            dev_ms += sim.bench_configs(0, cps)
        barrier()
        t_wall = (time.perf_counter() - t_wall) * 1e3
    cnt = sim.counters()
    if a.dump_outputs:
        outputs["image"] = sim.finish_k(0)[0]       # detector tail of the intensity the last step accumulated
    t = torch.tensor([dev_ms, t_wall], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, t_wall = float(t[0]), float(t[1])
    value = world * px * slices_per_step * a.steps / (dev_ms * 1e-3) / 1e6

    # live per-sweep kernel times (CUDA events on the engine's stream) -> roofline of a slice
    sweep_ms = sim.time_sweeps(0, 0, 20)
    nZ, batch = sim.nZ, sim.batch
    grid, slices = [sim.m1, sim.m2], sim.m3
    sim.close()

    # end to end: the drop-in FDES() call, host buffers in and out
    # caller-side buffers of the drop-in call in pinned host memory (torch only allocates them: plumbing)
    atoms6_pin = torch.empty(atoms6.shape, dtype=torch.float32, pin_memory=True)
    atoms6_pin.numpy()[...] = atoms6
    atoms6 = atoms6_pin.numpy()
    img_pin = torch.zeros((1, sim.n2, sim.n1), dtype=torch.float32, pin_memory=True)
    img = img_pin.numpy()
    cwd = os.getcwd()
    os.chdir(tmp)
    devnull = os.open(os.devnull, os.O_WRONLY)
    saved_err = os.dup(2)
    os.dup2(devnull, 2)     # FDES() prints its banner / progress to stderr like the reference
    try:
        for _ in range(max(1, min(a.warmup, 3))):
            fb.cuda_FDES(local, 0, str(cnf), str(tmp / "Measurements.bin"), str(tmp / "results.emd"), atoms6,
                         len(atoms6), img)
        barrier()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            fb.cuda_FDES(local, 0, str(cnf), str(tmp / "Measurements.bin"), str(tmp / "results.emd"), atoms6,
                         len(atoms6), img)
        barrier()
        e2e_ms = (time.perf_counter() - t0) * 1e3
    finally:
        os.dup2(saved_err, 2)
        os.close(devnull)
        os.chdir(cwd)
    t = torch.tensor([e2e_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t[0])
    e2e_value = world * px * slices_per_step * a.steps / (e2e_ms * 1e-3) / 1e6
    assert np.isfinite(img).all() and img.mean() > 0.1, "FDES() returned an implausible image"
    if a.dump_outputs:
        outputs["e2e_image"] = img.copy()

    stem = None if a.no_stem else run_stem(a, fb, specimens, tmp, local, world, barrier, dist, torch, outputs)
    job = None if a.no_job else run_jobs(a, fb, specimens, tmp, local, rank, world, barrier, dist, torch, outputs)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = peaks()
    traffic, traffic_src = None, None
    tf = ROOT / "profiles" / "dram_traffic.json"     # per-launch dram bytes of the six sweeps from a committed ncu capture
    if tf.exists() and a.workload == "si001_1024":
        tj = json.loads(tf.read_text())
        traffic_src = tj.get("source", "profiles/dram_traffic.json")
        per = tj.get("per_launch_bytes", tj)
        if all(n in per for n in algorithmic_bytes_per_px(nZ)):
            # S1..S4 launches cover a slice PAIR: per slice, half of them
            traffic = int(sum(per[n] * (0.5 if n[:2] in ("S1", "S2", "S3", "S4") else 1.0) for n in algorithmic_bytes_per_px(nZ))
                          * batch / tj.get("batch", batch))
    ab = algorithmic_bytes_per_px(nZ)
    names = list(ab)
    slice_bytes = sum(ab.values()) * px * batch
    slice_ms = float(np.sum(sweep_ms))
    slice_gbs = slice_bytes / (slice_ms * 1e-3) / 1e9
    step_gbs = value * 1e6 / world * sum(ab.values()) / 1e9      # per GPU: whole step incl. atom preparation, image formation
    cfg = workload_config(a, cps, world)
    line = {
        "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": round(dev_ms / a.steps, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "complex64 (f32)", "data": "synthetic",
        "config": cfg,
        "shape": {"grid": grid, "slices": slices, "atoms": int(len(atoms6)), "species": nZ, "batch": batch,
                  "batched_working_set_MiB": round((4 + nZ) * batch * px * 8 / 2**20)},
        "wall_ms_per_step": round(t_wall / a.steps, 4),
        "e2e": {"value": round(e2e_value, 3), "unit": UNIT, "h2d_bytes_per_step": int(24 * len(atoms6)),
                "d2h_bytes_per_step": int(img.nbytes), "ms_per_step": round(e2e_ms / a.steps, 4),
                "call": "FDES() drop-in C-ABI: .cnf + host atom array -> host image; session set-up, copies and "
                        "side-effect files inside the timed region (pinned caller buffers)"},
        "gpu_launches": cnt["launches"],
        "clocks": clk.summary(),
        "roofline": {"bound": "hbm", "kernel": "S1..S6: the six sweeps of one slice, one launch each over the batch",
                     "achieved": round(slice_gbs, 1), "peak": peak, "unit": "GB/s", "frac": round(slice_gbs / peak, 4),
                     "frac_of_8TBps": round(slice_gbs / 8000.0, 4),
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": int(slice_bytes), "algorithmic_bytes_per_px_slice": sum(ab.values()),
                     "launch_ms": round(slice_ms, 5),
                     "whole_step": {"achieved": round(step_gbs, 1), "frac": round(step_gbs / peak, 4),
                                    "frac_of_8TBps": round(step_gbs / 8000.0, 4),
                                    "note": "value x algorithmic bytes per pixel and slice, per GPU: atom preparation, wave "
                                            "copies and image formation included; the first slice of a plane wave runs "
                                            "without S5 (psi = 1) and moves 24 B/px less than this model counts"}},
        "sweeps": {n: {"ms": round(float(m), 5), "alg_GBps": round(ab[n] * px * batch / (float(m) * 1e-3) / 1e9, 1),
                       "frac": round(ab[n] * px * batch / (float(m) * 1e-3) / 1e9 / peak, 4)}
                   for n, m in zip(names, sweep_ms)},
    }
    if stem is not None:
        line["stem"] = stem
    if job is not None:
        line["job"] = job
    if world == 1 and not a.no_cpu:
        line["cpu_baseline"] = cpu_baseline(cnf, a.cpu_seconds)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, outputs)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_stem(a, fb, specimens, tmp, local, world, barrier, dist, torch, outputs):
    """Second metric of BASELINE.json: STEM probes/s on configs[3] (SrTiO3, 512^2 probe grid, 40 slices,
    HAADF + ABF detectors).  Every rank scans its own `probes_per_gpu` positions of the raster (weak
    scaling: 8 x 8192 = the 256 x 256 scan); the transmission stack is built once per call, inside the
    timed region.  value = device time of the scan (CUDA events), e2e = wall time of the call with host
    positions in and host detector signals out."""
    cnf = tmp / "stem_512.cnf"
    atoms = specimens.config_srtio3_stem_512(cnf)
    pos = specimens.stem_raster(256)
    rank = int(os.environ.get("RANK", "0"))
    n = a.stem_probes
    mine = pos[(rank * n) % len(pos):][:n]
    det = np.array([[70.0, 200.0], [11.0, 22.0]], np.float32)      # HAADF, ABF [mrad]
    with fb.Simulation(cnf, atoms6=np.ascontiguousarray(atoms, np.float32), gpu_index=local, batch=a.stem_batch) as sim:
        sim.stem_scan(mine[:256], det)        # warm-up
        barrier()
        t0 = time.perf_counter()
        sig, dev_ms = sim.stem_scan(mine, det)
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        m1, m3, batch = sim.m1, sim.m3, sim.batch
    t = torch.tensor([dev_ms, wall_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, wall_ms = float(t[0]), float(t[1])
    peak, _ = peaks()
    alg = 40.0 * m1 * m1 * m3 * n * world / (dev_ms * 1e-3) / 1e9      # A_prop = 40 B/px/slice (SURVEY 8d)
    assert np.isfinite(sig).all() and sig[:, 0].min() > 0
    outputs["stem_signals"] = sig
    return {"metric": "stem_probes_per_s", "value": round(world * n / (dev_ms * 1e-3), 1), "unit": "probes/s",
            "e2e": {"value": round(world * n / (wall_ms * 1e-3), 1), "unit": "probes/s",
                    "h2d_bytes_per_step": int(mine.nbytes), "d2h_bytes_per_step": int(sig.nbytes)},
            "config": {"workload": "srtio3_stem_512", "grid": [m1, m1], "slices": m3, "atoms": int(len(atoms)),
                       "probes_per_gpu": n, "batch": batch, "detectors_mrad": det.tolist()},
            "roofline": {"bound": "hbm", "kernel": "S5+S6 per probe slice", "achieved": round(alg / world, 1), "peak": peak,
                         "unit": "GB/s per GPU", "frac": round(alg / world / peak, 4), "frac_of_8TBps": round(alg / world / 8000.0, 4),
                         "algorithmic_bytes_per_px_slice": 40},
            "haadf_mean": float(sig[:, 0].mean()), "abf_mean": float(sig[:, 1].mean())}


def run_jobs(a, fb, specimens, tmp, local, rank, world, barrier, dist, torch, outputs):
    """Strong scaling: ONE job sharded over the `world` ranks, collective inside the timed region.
      au_2048_x32   BASELINE configs[2]: Au cuboctahedron 2048^2, 32 frozen-phonon configurations; the ranks
                    run 32/world configurations each, all-reduce (NCCL) of the partial intensity, detector tail.
      stem_256x256  BASELINE configs[3]: 65 536 probe positions on the SrTiO3 512^2 x 40-slice specimen; the ranks scan
                    contiguous ranges of the raster, all-gather of the detector signals.
    Wall clock between barriers (session set-up included), max over ranks."""
    from fdes_b200.distributed import simulate_sharded, stem_scan_sharded
    out = {}
    cnf = tmp / "job_au_2048.cnf"
    atoms = np.ascontiguousarray(specimens.config_au_2048(cnf, frozen_phonons=32), np.float32)
    open_sim = lambda r, w: fb.Simulation(cnf, atoms6=atoms, gpu_index=local, rank=r, world=w)
    simulate_sharded(open_sim)                      # warm-up (function attributes, memory pool, NCCL channels)
    tm = {}
    barrier()
    t0 = time.perf_counter()
    img, _ = simulate_sharded(open_sim, timings=tm)
    barrier()
    ms = (time.perf_counter() - t0) * 1e3
    t = torch.tensor([ms, tm.get("collective_ms", 0.0)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, coll = float(t[0]), float(t[1])
    assert np.isfinite(img).all() and img.mean() > 0.1
    outputs["job_au_2048_x32_image"] = img
    out["au_2048_x32"] = {"configs": 32, "grid": [2048, 2048], "slices": 12, "ms": round(ms, 3),
                          "value": round(2048 * 2048 * 12 * 32 / (ms * 1e-3) / 1e6, 1), "unit": UNIT,
                          "collective": "all_reduce(SUM) of the partial intensity, 2048^2 float32",
                          "collective_ms": round(coll, 3), "collective_share": round(coll / ms, 4)}
    if not a.no_stem:
        cnf = tmp / "job_stem_512.cnf"
        atoms = np.ascontiguousarray(specimens.config_srtio3_stem_512(cnf), np.float32)
        pos = specimens.stem_raster(256)[: a.job_probes]
        det = np.array([[70.0, 200.0], [11.0, 22.0]], np.float32)
        open_sim = lambda r, w: fb.Simulation(cnf, atoms6=atoms, gpu_index=local, batch=a.stem_batch)
        barrier()
        t0 = time.perf_counter()
        sig = stem_scan_sharded(open_sim, pos, det)
        barrier()
        ms = (time.perf_counter() - t0) * 1e3
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0])
        assert sig.shape == (len(pos), 2) and np.isfinite(sig).all()
        outputs["job_stem_256x256_signals"] = sig
        out["stem_256x256"] = {"probes": int(len(pos)), "grid": [512, 512], "slices": 40, "ms": round(ms, 3),
                               "value": round(len(pos) / (ms * 1e-3), 1), "unit": "probes/s",
                               "collective": "all_gather of the detector signals [probes][2] float32"}
    out["scaling"] = "strong"
    return out


def dump_outputs(directory, outputs):
    """--dump-outputs: one float32 / float64 .npy per array, 64 MB in all at most."""
    d = pathlib.Path(directory)
    d.mkdir(parents=True, exist_ok=True)
    arrays = {name: np.ascontiguousarray(v) for name, v in outputs.items()}
    assert all(v.dtype in (np.float32, np.float64) for v in arrays.values())
    assert sum(v.nbytes for v in arrays.values()) <= 64 << 20, {n: v.nbytes for n, v in arrays.items()}
    for name, v in arrays.items():
        np.save(d / f"{name}.npy", v)


def cpu_baseline(cnf, budget_s):
    """numpy/pocketfft restatement of the same workload on the host cores: whole configurations
    (binning + all slices) repeated until ~budget_s seconds have passed."""
    sys.path.insert(0, str(ROOT / "oracle"))
    import fdes_oracle as orc
    p, Z, xyz, dwf, occ = orc.read_cnf(str(cnf))
    p.frPh = 0   # one configuration per repetition, equilibrium coordinates (same arithmetic per slice)
    t0 = time.perf_counter()
    n = 0
    res = None
    while True:
        res = orc.build_measurements(p, Z, xyz, dwf, occ)
        n += 1
        if time.perf_counter() - t0 > budget_s or n >= 50:
            break
    dt = time.perf_counter() - t0
    ps = res.params
    return {"value": round(ps.m1 * ps.m2 * ps.m3 * n / dt / 1e6, 3), "unit": UNIT, "cores": orc._WORKERS,
            "kind": "port", "sample": f"{n} configuration(s) x {ps.m3} slices at {ps.m1}x{ps.m2} in {dt:.1f} s "
                                      "(numpy float32 + scipy.fft/pocketfft, incl. image formation)"}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    harness = ROOT / "oracle" / "_ref" / "ref_harness"
    if not harness.exists():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/ref_harness not built (needs /root/reference + make -C oracle)"}))
        return
    from fdes_b200 import specimens
    # Bounded sample of our arm's workload: the reference needs 0.1 - 1 s per configuration, so a
    # step of this arm is `ref_configs` configurations of the step our arm runs (the metric is per
    # pixel*slice; 16 per call keep the reference's fixed per-call cost below 5 %), and the run stops
    # after --ref-seconds even if fewer than --steps steps are done (the line reports the steps timed).
    cps = a.ref_configs or REF_SAMPLE_CONFIGS[a.workload]
    our_cps = a.configs_per_step or DEFAULT_CONFIGS_PER_STEP[a.workload]
    tmp = pathlib.Path(tempfile.mkdtemp(prefix="fdes_bench_ref_"))
    cnf = tmp / f"{a.workload}.cnf"
    atoms = getattr(specimens, WORKLOADS[a.workload][0])(cnf, frozen_phonons=cps)
    env = dict(os.environ, TMPDIR=str(tmp), CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0])
    with ClockSampler(0) as clk:
        r = subprocess.run([str(harness), "e2e", str(cnf), str(a.steps), str(a.warmup), str(a.ref_seconds)], env=env,
                           capture_output=True, text=True, timeout=3000)
    js = [l for l in r.stdout.splitlines() if l.startswith('{"ref_e2e"')]
    if r.returncode != 0 or not js:
        print(json.dumps({"impl": "reference", "unavailable": f"ref_harness failed rc={r.returncode}: {r.stderr[-300:]}"}))
        return
    j = json.loads(js[-1])
    # slice-loop only (device resident), for context
    r2 = subprocess.run([str(harness), "time", str(cnf), "2", "1"], env=env, capture_output=True, text=True, timeout=3000)
    j2 = [json.loads(l) for l in r2.stdout.splitlines() if l.startswith('{"ref_time"')]
    value = j["mpx_slices_per_s"]
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world,
        "steps": j["reps"], "steps_requested": a.steps, "warmup": a.warmup, "ms_per_step": round(j["ms_per_call"], 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "complex64 (f32)", "data": "synthetic",
        "config": workload_config(a, our_cps, world),
        "shape": {"grid": [j["m1"], j["m2"]], "slices": j["slices"], "atoms": int(len(atoms))},
        "note": "unmodified reference (cuFFT/cuBLAS build for sm_100) on ONE B200: FDES has no CPU or multi-GPU path; "
                "whole-call wall time of its exported flow (getParams -> readAtomsFromArray -> buildMeasurements -> "
                "image copy)",
        "cpu_baseline": {"value": round(value, 3), "unit": UNIT, "cores": 1, "kind": "reference",
                         "sample": f"{j['reps']} call(s), each {cps} of the {our_cps} configurations of a step x {j['slices']} slices "
                                   f"(bounded to {a.ref_seconds:.0f} s); 1 host thread driving 1 B200 (the reference's only "
                                   "implementation is CUDA)"},
        "e2e": {"value": round(value, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "clocks": clk.summary(),
        "slice_loop_only": j2[-1] if j2 else None,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="si001_1024", choices=sorted(WORKLOADS))
    ap.add_argument("--configs-per-step", type=int, default=0)
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--ref-configs", type=int, default=0)
    ap.add_argument("--no-job", action="store_true")
    ap.add_argument("--job-probes", type=int, default=65536)
    ap.add_argument("--ref-seconds", type=float, default=120.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-stem", action="store_true")
    ap.add_argument("--stem-probes", type=int, default=8192)
    ap.add_argument("--stem-batch", type=int, default=37)   # 24 column tiles x 37 probes = 6.0 waves of 148 SMs
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed calls returned in their last step to DIR/<name>.npy")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    a.warmup = max(a.warmup, 3) if a.impl == "ours" else a.warmup
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
