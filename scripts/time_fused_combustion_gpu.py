"""A/B of the frame's combustion stage on bench.py's workload (config 4, I = 40), in one process: HNS_FUSED_COMBUSTION=0 (combustion
as a pass of its own) and =1 (its field update inside advect_vector, the expansion term in the divergence pass, the buoyancy force in
the gradient pass) alternate over --rounds rounds of Simulation.time_frames(--frames, 40, dt), every round from the same inputs.

    python scripts/time_fused_combustion_gpu.py [--rounds 7] [--frames 20] [--kernels]

Prints per round and arm the frame time and the pressure-solve time per frame (CUDA events on the launch stream), then per arm the
median, min and max, the launches per frame, the card and its power limit and the SM clock while the arm ran (nvidia-smi).
--kernels: instead, per arm the device time per frame of every kernel over --frames frames under torch.profiler (a run of its own:
the profiler slows the host, the frame times above are taken without it).
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import hnanosolver_b200 as H  # noqa: E402
from bench import ITERATIONS, PARAMS6, ClockSampler, build_workload  # noqa: E402
from hnanosolver_b200 import _lib  # noqa: E402


def card() -> dict:
    q = "name,power.limit,clocks.max.sm"
    try:
        row = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
        return dict(zip(q.split(","), [x.strip() for x in row.split(",")]))
    except Exception as e:
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--kernels", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    lib = _lib.lib()
    w, names, fields, kind = build_workload("c4", 0, 1)
    assert kind == "full"
    grid = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    sim = H.Simulation(grid, len(fields))
    sim.set_combustion(True, names.index("fuel"), names.index("waste"), names.index("temperature"), names.index("flame"),
                       H.CombustionParams(*PARAMS6))
    print(f"card: {card()}", flush=True)
    print(f"workload: {w.name}, {w.num_leaves} leaves, {w.num_voxels} voxels, S={len(fields)}, I={ITERATIONS}", flush=True)

    def run(arm: str, frames: int):
        os.environ["HNS_FUSED_COMBUSTION"] = arm
        sim.upload(w.velocity, fields)                          # every round from the same inputs (outside the timed frames)
        torch.cuda.synchronize()
        lib.hns_launch_count_reset()
        packed0 = lib.hns_packed_advection_launches()
        ms, pr = sim.time_frames(frames, ITERATIONS, w.dt)
        return ms / frames, pr / frames, lib.hns_launch_count() / frames, (lib.hns_packed_advection_launches() - packed0) / frames

    for arm in ("0", "1"):
        run(arm, 3)                                             # warm-up of both arms (modules, attributes, scratch allocations)
    if args.kernels:
        import tempfile

        from torch.profiler import ProfilerActivity, profile

        for arm in ("0", "1"):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                run(arm, args.frames)
                torch.cuda.synchronize()
            with tempfile.TemporaryDirectory() as tmp:          # the trace goes to a temporary directory, never into the tree
                prof.export_chrome_trace(os.path.join(tmp, "trace.json"))
                trace = json.load(open(os.path.join(tmp, "trace.json")))
            per = {}
            for e in trace.get("traceEvents", []):
                if e.get("cat") == "kernel":
                    name = e["name"].replace("(anonymous namespace)::", "").replace("void ", "").split("(")[0]
                    t = per.setdefault(name, [0, 0.0])
                    t[0] += 1
                    t[1] += float(e.get("dur", 0.0)) / 1e3
            print(f"HNS_FUSED_COMBUSTION={arm}: device ms per frame by kernel over {args.frames} frames", flush=True)
            for k, (n, ms) in sorted(per.items(), key=lambda kv: -kv[1][1]):
                print(f"  {k[:60]:60s} {n / args.frames:5.1f} launches {ms / args.frames:8.4f} ms", flush=True)
            print(f"  {'total':60s} {'':14s} {sum(v[1] for v in per.values()) / args.frames:8.4f} ms", flush=True)
        return
    res = {"0": [], "1": []}
    clocks = {"0": [], "1": []}
    for r in range(args.rounds):
        for arm in (("0", "1") if r % 2 == 0 else ("1", "0")):
            sampler = ClockSampler(0)
            sampler.start()
            time.sleep(0.3)
            t0 = time.time()
            row = run(arm, args.frames)
            t1 = time.time()
            clocks[arm].append(sampler.stop(t0, t1).get("sm_mhz"))
            res[arm].append(row)
            print(f"round {r} HNS_FUSED_COMBUSTION={arm}: {row[0]:.4f} ms/frame, pressure {row[1]:.4f} ms/frame, "
                  f"{row[2]:.0f} launches/frame, {row[3]:.0f} packed advection launches/frame, SM {clocks[arm][-1]} MHz", flush=True)
    summary = {}
    for arm, label in (("0", "split"), ("1", "fused")):
        ms = np.array([x[0] for x in res[arm]])
        pr = np.array([x[1] for x in res[arm]])
        sm = [c for c in clocks[arm] if c is not None]
        summary[label] = {"ms_per_frame_median": float(np.median(ms)), "ms_min": float(ms.min()), "ms_max": float(ms.max()),
                          "spread_ms": float(ms.max() - ms.min()), "ms_pressure_median": float(np.median(pr)),
                          "ms_pressure_spread": float(pr.max() - pr.min()), "launches_per_frame": res[arm][0][2],
                          "packed_advection_launches_per_frame": res[arm][0][3], "sm_mhz_median": float(np.median(sm)) if sm else None}
        s = summary[label]
        print(f"{label:5s} (HNS_FUSED_COMBUSTION={arm}): median {s['ms_per_frame_median']:.4f} ms/frame, min {s['ms_min']:.4f}, "
              f"max {s['ms_max']:.4f} (spread {s['spread_ms']:.4f}); ms_pressure median {s['ms_pressure_median']:.4f} "
              f"(spread {s['ms_pressure_spread']:.4f}); SM {s['sm_mhz_median']} MHz", flush=True)
    d = summary["split"]["ms_per_frame_median"] - summary["fused"]["ms_per_frame_median"]
    print(f"fused - split: {-d:+.4f} ms/frame ({-d / summary['split']['ms_per_frame_median'] * 100:+.2f} %)", flush=True)
    print(json.dumps({"card": card(), "rounds": args.rounds, "frames": args.frames, "voxels": w.num_voxels, **summary,
                      "saved_ms_per_frame": d}), flush=True)


if __name__ == "__main__":
    main()
