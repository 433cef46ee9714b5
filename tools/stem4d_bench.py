"""4D-STEM throughput against the annular scan on BASELINE configs[3]: SrTiO3, 512^2 grid, 40 slices, the first 8192
positions of the 256 x 256 raster, batch 37, the HAADF and ABF rings of bench.py.  After a warm-up, stem_scan and
stem_scan_4d (default window, bins 1 and 4) alternate three times.  Reports device-loop probes/s (CUDA events around
the slice loop), wall-clock probes/s (host clock around the whole call, the device-to-host copy of the passes
included) and the bytes of patterns written, with the card name and power limit.

    python tools/stem4d_bench.py [--out result.json]
"""
import argparse
import json
import pathlib
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parent.parent))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--probes", type=int, default=8192)
    ap.add_argument("--repeats", type=int, default=3)
    a = ap.parse_args()
    import fdes_b200 as fb
    from fdes_b200 import specimens
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip().splitlines()
    det = np.array([[70.0, 200.0], [11.0, 22.0]], np.float32)      # HAADF, ABF [mrad] (bench.py)
    with tempfile.TemporaryDirectory() as tmp:
        cnf = pathlib.Path(tmp) / "stem_512.cnf"
        atoms = np.ascontiguousarray(specimens.config_srtio3_stem_512(cnf), np.float32)
        pos = specimens.stem_raster(256)[:a.probes]
        with fb.Simulation(cnf, atoms6=atoms, batch=37) as sim:
            outs = {b: np.ones((len(pos), fb.stem_4d_side(sim.m1, 0, b), fb.stem_4d_side(sim.m1, 0, b)), np.float32)
                    for b in (1, 4)}                                 # touched once: no page faults in the timed calls
            runs = {"annular": lambda: sim.stem_scan(pos, det)[1],
                    "4d_bin1": lambda: sim.stem_scan_4d(pos, bin=1, detectors_mrad=det, out=outs[1])[2],
                    "4d_bin4": lambda: sim.stem_scan_4d(pos, bin=4, detectors_mrad=det, out=outs[4])[2]}
            sim.stem_scan(pos[:256], det)
            sim.stem_scan_4d(pos[:256], bin=1, detectors_mrad=det, out=outs[1][:256])
            sim.stem_scan_4d(pos[:256], bin=4, detectors_mrad=det, out=outs[4][:256])
            res = {k: {"device_ms": [], "wall_ms": []} for k in runs}
            for _ in range(a.repeats):
                for k, f in runs.items():
                    t0 = time.perf_counter()
                    ms = f()
                    res[k]["wall_ms"].append((time.perf_counter() - t0) * 1e3)
                    res[k]["device_ms"].append(ms)
    line = {"workload": "srtio3_stem_512", "probes": len(pos), "batch": 37, "detectors_mrad": det.tolist(), "gpu": card}
    for k, r in res.items():
        dev, wall = min(r["device_ms"]), min(r["wall_ms"])
        line[k] = {"device_probes_per_s": round(len(pos) / (dev * 1e-3), 1), "wall_probes_per_s": round(len(pos) / (wall * 1e-3), 1),
                   "device_ms": [round(v, 2) for v in r["device_ms"]], "wall_ms": [round(v, 2) for v in r["wall_ms"]]}
        if k != "annular":
            b = int(k[-1])
            line[k]["bytes_written"] = int(outs[b].nbytes)
            line[k]["device_vs_annular"] = round(dev / min(res["annular"]["device_ms"]), 3)
            line[k]["wall_vs_annular"] = round(wall / min(res["annular"]["wall_ms"]), 3)
    print(json.dumps(line))
    if a.out:
        pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        pathlib.Path(a.out).write_text(json.dumps(line, indent=1) + "\n")


if __name__ == "__main__":
    main()
