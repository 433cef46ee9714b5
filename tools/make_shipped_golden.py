#!/usr/bin/env python3
"""TEST INFRASTRUCTURE -- golden vectors of the reference's SHIPPED example inputs, run as shipped:

    gpurun -- 'python tools/make_shipped_golden.py --out gpurun_out/golden_shipped'
    cp gpurun_out/golden_shipped/*.npz tests/golden/shipped/

Runs the UNMODIFIED reference (oracle/_ref/ref_harness run <input> <dir> 2: stock getParams / readQsc
-> buildMeasurements, print level 2) on every case of tests/shipped_cases.py and stores the reductions
defined there (selected images, per-image statistics, exit-wave crops)."""
import argparse
import pathlib
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tests"))
import shipped_cases as sc  # noqa: E402

HARNESS = ROOT / "oracle" / "_ref" / "ref_harness"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "tests" / "golden" / "shipped"))
    ap.add_argument("cases", nargs="*")
    a = ap.parse_args()
    out = pathlib.Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    for case in (a.cases or sc.CASES):
        with tempfile.TemporaryDirectory() as td:
            td = pathlib.Path(td)
            inp = sc.stage(case, td)
            t0 = time.time()
            subprocess.run([str(HARNESS), "run", str(inp), str(td / "run"), "2"], check=True, cwd=td,
                           stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            meta = dict((l.split()[0], float(l.split()[1])) for l in open(td / "run" / "meta.txt"))
            n1, n2, n3, m1, m2 = (int(meta[k]) for k in ("n1", "n2", "n3", "m1", "m2"))
            img = np.fromfile(td / "run" / "image.f32", np.float32).reshape(n3, n2, n1)
            ew = np.fromfile(td / "run" / "exitwave.f32", np.float32).view(np.complex64).reshape(n3, m2, m1)
            g = sc.reduce(img, ew)
            if case in sc.DEEP_PROBE_CASES:
                # float64 evaluation of the same model from the float32 probe: the yardstick for 400 chained
                # sub-slices of a focused probe, where float32 programs differ by several 1e-5 from each other
                sys.path.insert(0, str(ROOT / "oracle"))
                import fdes_oracle as orc
                import qsc_oracle as qorc
                import os
                cwd = os.getcwd()
                os.chdir(td)
                try:
                    p, Z, xyz, dwf, occ = qorc.read_qsc(str(inp))
                finally:
                    os.chdir(cwd)
                ps = p.copy()
                orc.set_sub_slices(ps, orc.sub_slice_ratio(ps.d3, ps.subSlTh))
                psi0 = orc.incoming_wave(ps, 0, orc.band_mask(ps))
                truth = orc.exit_wave_fp64(p, Z, xyz, occ, psi0=psi0).astype(np.complex64)[None]
                r64 = sc.reduce(img, truth)
                g["ew_crop_fp64"], g["ew_power_fp64"] = r64["ew_crop"], r64["ew_power"]
            g["meta_keys"] = np.array(sorted(meta))
            g["meta_vals"] = np.array([meta[k] for k in sorted(meta)], np.float64)
            sc.save_golden(out, case, g)
            print(f"golden {case}: {m1}x{m2}, m3={int(meta.get('m3', 0))}, n3={n3}, mode={int(meta.get('mode', -1))}, "
                  f"reference took {time.time() - t0:.1f} s", flush=True)


if __name__ == "__main__":
    main()
