"""Cost of sourcing on resident state (Simulation.add_source, compSum on the device) on bench.py's workload (config 4, I = 40), in one
process, by CUDA events on the launch stream:

  * one add_source into a scalar and into the velocity, for an emitter covering 1 % and 100 % of the leaves (mean over --reps calls);
  * what it replaces: one scalar field's upload from pinned host memory (sourcing on the host also downloads it first);
  * the frame with density, temperature, fuel and the velocity sourced (1 % emitter) against the frame without, alternating over
    --rounds rounds of --frames frames from the same inputs.

    python scripts/time_sourcing_gpu.py [--reps 50] [--rounds 5] [--frames 10]

Algorithmic bytes of an add: 8 B per voxel and component (the field read and written) plus 4 B per voxel and component of the source
leaves inside the domain; reported as GB/s and as a fraction of the measured copy rate (MEASURED_PEAKS.json hbm_gbs when present, as in
bench.py), with the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import hnanosolver_b200 as H  # noqa: E402
from bench import ITERATIONS, PARAMS6, build_workload, hbm_peak  # noqa: E402
from hnanosolver_b200 import io as hio  # noqa: E402
from hnanosolver_b200 import synth  # noqa: E402
from time_fused_combustion_gpu import card  # noqa: E402


def events_ms(fn, reps: int) -> float:
    """mean ms per call of fn over reps calls, CUDA events on the current stream"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--frames", type=int, default=10)
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
    N = w.num_voxels
    out = {"card": card(), "peak_gbs": peak, "peak_from": peak_from, "voxels": N, "leaves": w.num_leaves, "adds": []}
    print(f"card: {out['card']}; copy rate {peak:.0f} GB/s ({peak_from})", flush=True)
    speed = 0.05 * float(np.abs(w.velocity).max())
    emitters = {}
    for frac in (0.01, 1.0):
        so, values = synth.emitter(w.origins, fraction=frac, speed=speed)
        emitters[frac] = {k: H.Source(hio.grid_from_sidecar(so, v, w.voxel_size, k)) for k, v in values.items()}
        del values
        for target, key, comps in ((names.index("density"), "density", 1), ("velocity", "velocity", 3)):
            src = emitters[frac][key]
            inside = src.num_leaves - src.leaves_outside(grid)
            ms = events_ms(lambda: sim.add_source(target, src), args.reps)
            nbytes = 8 * comps * N + 4 * comps * 512 * inside
            row = dict(emitter=frac, target=key, source_leaves_inside=inside, ms=ms, gb=nbytes / 1e9, gbs=nbytes / ms / 1e6,
                       frac_of_copy=nbytes / ms / 1e6 / peak)
            out["adds"].append(row)
            print(f"add_source {key:8s} emitter {frac:5.0%} ({inside} leaves inside): {ms:.4f} ms, {row['gb']:.3f} GB -> "
                  f"{row['gbs']:.0f} GB/s = {row['frac_of_copy']:.3f} of the copy rate", flush=True)
        if frac == 1.0:
            del emitters[frac]
    pinned = torch.from_numpy(fields[0]).pin_memory().numpy()
    up = events_ms(lambda: sim.upload(scalars=[pinned]), 5)
    out["scalar_upload_ms"] = up
    print(f"one scalar field ({4 * N / 1e6:.0f} MB) uploaded from pinned memory: {up:.3f} ms ({4 * N / up / 1e6:.1f} GB/s)", flush=True)

    em = emitters[0.01]
    feeds = [(names.index("density"), em["density"]), (names.index("temperature"), em["temperature"]), (names.index("fuel"), em["fuel"]),
             ("velocity", em["velocity"])]

    def arm(sourced: bool) -> float:
        sim.upload(w.velocity, fields)
        torch.cuda.synchronize()

        def frames():
            for _ in range(args.frames):
                if sourced:
                    for t, s in feeds:
                        sim.add_source(t, s)
                sim.step(ITERATIONS, w.dt)
        return events_ms(frames, 1) / args.frames

    rows = {False: [], True: []}
    for r in range(args.rounds):
        for sourced in ((False, True) if r % 2 == 0 else (True, False)):
            rows[sourced].append(arm(sourced))
            print(f"round {r} {'sourced' if sourced else 'plain  '}: {rows[sourced][-1]:.4f} ms per frame", flush=True)
    for sourced, label in ((False, "plain"), (True, "sourced")):
        a = np.array(rows[sourced])
        out[f"frame_{label}_ms"] = {"median": float(np.median(a)), "min": float(a.min()), "max": float(a.max())}
    d = out["frame_sourced_ms"]["median"] - out["frame_plain_ms"]["median"]
    out["frame_cost_of_sourcing_ms"] = d
    print(f"frame: plain {out['frame_plain_ms']['median']:.4f} ms, with 3 scalars + velocity sourced {out['frame_sourced_ms']['median']:.4f} ms "
          f"({d:+.4f} ms)", flush=True)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
