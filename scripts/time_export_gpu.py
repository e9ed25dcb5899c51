"""Cost of exporting resident fields as NanoVDB grids on the device (Simulation.export_grid) on bench.py's workload (config 4, after one
frame), in one process:

  * by CUDA events on the launch stream, the export of density and of the velocity, whole-domain (tolerance < 0) and pruned at a few
    tolerances (mean over --reps calls; an export returns when its grid is complete, so this is the whole call: kernels, the one
    readback of the counts and the header copy), with the kept leaves and GB/s against the copy rate;
  * by wall clock, the download of each grid to host memory;
  * by wall clock, what the export replaces: the field's download (Simulation.scalar / velocity) plus the host writer io.grid_from_sidecar.

    python scripts/time_export_gpu.py [--reps 20] [--out profiles/r3d_time_export.txt]

Algorithmic bytes of an export: the field read once (4 B per voxel and component of the listed leaves) and the grid written; pruned
exports read the field once more to classify it. The copy rate is MEASURED_PEAKS.json hbm_gbs when present, as in bench.py; the card's
name and power limit are read in the same run.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import hnanosolver_b200 as H  # noqa: E402
from bench import ITERATIONS, PARAMS6, build_workload, hbm_peak  # noqa: E402
from hnanosolver_b200 import io as hio  # noqa: E402
from time_fused_combustion_gpu import card  # noqa: E402
from time_sourcing_gpu import events_ms  # noqa: E402


def wall_ms(fn, reps: int) -> float:
    fn()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    return (time.perf_counter() - t0) / reps * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3d_time_export.txt"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    peak, peak_from = hbm_peak()
    w, names, fields, kind = build_workload("c4", 0, 1)
    assert kind == "full"
    grid = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    sim = H.Simulation(grid, len(fields))
    sim.set_combustion(True, names.index("fuel"), names.index("waste"), names.index("temperature"), names.index("flame"),
                       H.CombustionParams(*PARAMS6))
    sim.upload(w.velocity, fields)
    sim.step(ITERATIONS, w.dt)
    sim.sync()
    N = w.num_voxels
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    out = {"card": card(), "peak_gbs": peak, "peak_from": peak_from, "voxels": N, "leaves": w.num_leaves, "exports": [], "host_path": []}
    say(f"card: {out['card']}; copy rate {peak:.0f} GB/s ({peak_from}); config 4 after one frame: {w.num_leaves} leaves, {N} voxels")
    vg = H.ValueGrid()
    for target, key, comps in ((names.index("density"), "density", 1), ("velocity", "velocity", 3)):
        for tol in (-1.0, 0.0, 1e-3, 1e-1):
            ms = events_ms(lambda: sim.export_grid(target, key, tol, vg), args.reps)
            read = 4 * comps * N * (2 if tol >= 0 else 1)
            nbytes = read + vg.nbytes
            dl = wall_ms(vg.download, 3)
            row = dict(target=key, tolerance=tol, kept_leaves=vg.num_leaves, grid_bytes=vg.nbytes, ms=ms, gbs=nbytes / ms / 1e6,
                       frac_of_copy=nbytes / ms / 1e6 / peak, download_ms=dl)
            out["exports"].append(row)
            say(f"export {key:8s} tolerance {tol:7.3g}: {vg.num_leaves:7d} of {w.num_leaves} leaves, {vg.nbytes / 1e6:8.1f} MB in {ms:.4f} ms "
                f"-> {row['gbs']:.0f} GB/s = {row['frac_of_copy']:.3f} of the copy rate; download {dl:.2f} ms")
        field = (lambda: sim.velocity()) if comps == 3 else (lambda: sim.scalar(target))
        t_dl = wall_ms(field, 3)
        v = field()
        t_build = wall_ms(lambda: hio.grid_from_sidecar(w.origins, v, w.voxel_size, key), 3)
        out["host_path"].append(dict(target=key, download_ms=t_dl, host_writer_ms=t_build))
        say(f"host path {key:8s}: field download {t_dl:.2f} ms + io.grid_from_sidecar {t_build:.2f} ms = {t_dl + t_build:.2f} ms")
    say(json.dumps(out))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
