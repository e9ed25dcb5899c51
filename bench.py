#!/usr/bin/env python
"""bench.py -- one advect+project frame of the HNanoSolver hot path on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4] [--impl reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0). A "step" is one full frame over one synthetic sparse smoke domain:
  metric  : active voxel-updates/s  (N_voxels / frame time), BASELINE.json's metric
  value   : device-resident frame (inputs in HBM when the timed region starts), CUDA events on the launch stream
  e2e     : the same frame through the drop-in launcher calls (CreateIndexGrid + Compute_Sim) on pinned HOST buffers,
            host<->device copies inside the timed region
  roofline: the dominant kernel (fused red+black pressure sweep): algorithmic bytes per launch / measured launch time
  cpu_baseline: the CPU oracle port on the box's host cores, bounded sample
--impl reference runs the UNMODIFIED reference (its own src/Cuda kernels compiled for sm_100a, oracle/_ref) through its own
launchers CreateIndexGrid + Compute_Sim on the same workload (the reference has no CPU implementation of this path: its
implementation IS CUDA; see DESIGN.md section 6).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ITERATIONS = 40
PARAMS6 = [0.5, 2.0, 1.5, 0.1, 0.0, 1.0]  # expansionRate, temperatureRelease, buoyancyStrength, ambientTemp, vorticityScale (off), factorScale
FULL_FRAME_FIELDS = ["density", "fuel", "waste", "temperature", "flame"]


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ----------------------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0: float, t1: float) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1 + 0.1] or [r for _, r in self.rows[-3:]]
        sm, reasons, mx = [], set(), None
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------
# workload
# ----------------------------------------------------------------------------------------------------------------
def build_workload(name: str, rank: int, world: int, scaling: str = "weak"):
    """Returns (workload, field_names, fields, frame_kind). N > 1: weak scaling, the bounding box grows with N
    (512^3 -> 1024x512x512 -> 1024x1024x512 -> 1024^3) and each rank generates and owns one contiguous leaf range."""
    from hnanosolver_b200 import synth

    if world > 1:
        from hnanosolver_b200 import dist

        return dist.build_sharded_workload(name, rank, world, scaling)
    w = synth.WORKLOADS[name](with_coords=False)
    if name in ("c4", "c5"):
        fields = dict(density=w.scalars[0], **synth.combustion_fields(w))
        return w, list(fields), list(fields.values()), "full"
    return w, list(w.scalar_names), list(w.scalars), "north_star"


def hbm_peak():
    """(GB/s, where it came from): the driver-measured copy bandwidth when present, else the profiling guide's fallback"""
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        return float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def algorithmic_bytes_per_voxel(S: int, I: int, full: bool) -> int:
    b = 80 + 16 * I + 8 * S                      # BASELINE.md section 3
    if full:
        b += 40 + 12                             # combustion_oxygen (4 R + 4 W + div RW) + temperature_buoyancy (T R, v.y RW)
    return b


# ----------------------------------------------------------------------------------------------------------------
# multigrid frame (BASELINE.json config 3; reported beside the red-black frame on config 4)
# ----------------------------------------------------------------------------------------------------------------
MG_NU, MG_OMEGA = (2, 2), 1.15


def multigrid_setup(H, sim, grid, w, args, N):
    """Builds the hierarchy and finds how many V-cycles the first frame's divergence needs for a relative residual of 1e-4 (the timed
    frames then run that fixed count: no host round trip inside a frame)."""
    t = time.perf_counter()
    mg = H.Multigrid(grid)
    build_ms = (time.perf_counter() - t) * 1e3
    sim.advect_velocity(w.dt)
    sim.divergence(True)
    if args.mg_cycles > 0:
        cycles, _ = sim.pressure_solve_mg(mg, args.mg_cycles, 0.0, MG_NU[0], MG_NU[1], MG_OMEGA)
    elif args.workload == "c3" or args.solver == "mg":
        cycles, _ = sim.pressure_solve_mg(mg, 30, 1e-4, MG_NU[0], MG_NU[1], MG_OMEGA)
    else:
        cycles, _ = sim.pressure_solve_mg(mg, 2, 0.0, MG_NU[0], MG_NU[1], MG_OMEGA)   # config 4 side line: two cycles
    rel = sim.relative_residual()
    cells = [mg.level_cells(k) for k in range(mg.num_levels)]
    return mg, {"cycles": int(cycles), "nu": list(MG_NU), "omega_smooth": MG_OMEGA, "levels": mg.num_levels, "cells_per_level": cells,
                "leaves_per_level": [mg.level_leaves(k) for k in range(mg.num_levels)], "relative_residual_at_cycles": rel,
                "hierarchy_build_ms": build_ms, "fine_half_sweeps_per_solve": 2 * sum(MG_NU) * int(cycles)}


def mg_frame_bytes_per_voxel(S: int, full: bool, info: dict) -> float:
    """SURVEY.md 8d: a scheme with fewer sweeps is scored with its own sweep count per level, coarse levels weighted by their cell
    counts. Per V-cycle and level: (nu1+nu2) iterations x 16 B/cell (+4 for the diagonal on coarse levels); residual 8 (+4) B/cell read
    + 0.5 written to the parent; prolongation 8 (+4) B/cell + 0.5 read; the parent's p and rhs zeroed (1 B per cell of this level)."""
    cells = info["cells_per_level"]
    n0 = float(cells[0])
    per_cycle = 0.0
    for k, c in enumerate(cells):
        coarse = 4.0 if k else 0.0
        b = sum(info["nu"]) * (16.0 + coarse)
        if k + 1 < len(cells):
            b += (8.0 + coarse + 0.5) + (8.0 + coarse + 0.5) + 1.0
        per_cycle += b * c / n0
    return 80 + 8 * S + (52 if full else 0) + 4 + per_cycle * info["cycles"]      # + 4: p zeroed once per solve


def stage_breakdown(H, sim, w, S: int, full: bool, peak: float, reps: int = 5) -> dict:
    """Every stage of the frame on its own (CUDA events on the launch stream, median of `reps`), with its algorithmic bytes per voxel
    (SURVEY.md 8d / BASELINE.md section 3) and the fraction of the measured HBM copy rate that makes."""
    import torch

    omega = H.launchers.omega_compute(w.voxel_size)
    stages = [("advect_vector", 24, lambda: sim.advect_velocity(w.dt)), ("divergence", 16, lambda: sim.divergence(True))]
    if full:
        stages.append(("combustion+buoyancy", 52, lambda: sim.combustion_buoyancy(w.dt)))
    stages += [(f"pressure_solve({ITERATIONS})", 16 * ITERATIONS, lambda: sim.pressure_solve(ITERATIONS, omega)),
               ("subtract_gradient", 28, lambda: sim.subtract_gradient(True)), (f"advect_scalars({S})", 12 + 8 * S, lambda: sim.advect_scalars(w.dt, 0))]
    acc = {k: [] for k, _, _ in stages}
    from hnanosolver_b200 import _lib
    packed0 = _lib.lib().hns_packed_advection_launches()
    for r in range(reps + 1):
        for k, _, fn in stages:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            if r:
                acc[k].append(e0.elapsed_time(e1))
    out = {}
    measured = kernel_traffic()
    # which advection kernels ran: the third generation (packed float4 groups written by the gradient / combustion passes, advect.cu)
    # or the second (brick fields); with the packed layout the gradient and combustion passes move more bytes than the algorithm needs
    packed = int(_lib.lib().hns_packed_advection_launches() - packed0) > 0
    gen = "4" if packed else "2"
    layout = {"advect_vector": 28, "combustion+buoyancy": 64, "subtract_gradient": 48} if packed and full and S == 5 else {}
    for k, b, _ in stages:
        ms = float(np.median(acc[k]))
        gbs = b * w.num_voxels / (ms * 1e-3) / 1e9
        out[k] = {"ms": ms, "algorithmic_bytes_per_voxel": b, "algorithmic_GBps": gbs, "frac_of_peak": gbs / peak}
        if k in layout:       # bytes this layout actually moves (second copy of the velocity / combustion fields as packed groups)
            out[k]["layout_bytes_per_voxel"] = layout[k]
            out[k]["layout_frac_of_peak"] = layout[k] * w.num_voxels / (ms * 1e-3) / 1e9 / peak
        key = {"advect_vector": f"k_advect_vector{gen}", f"advect_scalars({S})": f"k_advect_scalars{gen}(S={S})"}.get(k)
        if key:
            out[k]["kernel"] = key
        if key in measured:   # dram bytes of the ncu capture of this kernel (profiles/kernel_traffic.json), scaled to this voxel count
            out[k]["traffic"] = measured[key]["dram_bytes_per_voxel"] * w.num_voxels
    return out


def kernel_traffic() -> dict:
    """dram__bytes_read + dram__bytes_write per voxel of the committed `ncu --set full` captures (profiles/kernel_traffic.json names them);
    measured on the config-4 workload with this round's kernels, never inside a timed run"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "kernel_traffic.json")))
    except Exception:
        return {}


def workload_label(name: str, w, kind: str, S: int) -> str:
    """config.workload of both arms (ours and --impl reference): one function, so that the two lines name the workload identically"""
    return (f"{name}: {w.name}, {w.num_leaves} leaves = {w.num_voxels} active voxels, frame={kind}, I={ITERATIONS} red-black iterations, "
            f"S={S} scalar fields, dt=1/24, voxel size 0.1, CFL<=2.5")


def frame_quality(sim) -> dict:
    """of the frame the state just ran: relative Poisson residual of its pressure and ||div(u_new)||_2 (rms), both reduced on the device"""
    a, b = sim.residual_sums()
    d = sim.divergence_sum_squares(of_advected=False)
    return {"relative_residual": float(np.sqrt(a / b)) if b > 0 else 0.0, "div_rms_before": float(np.sqrt(b / max(sim.n, 1))),
            "div_rms_after": float(np.sqrt(d / max(sim.n, 1)))}


DUMP_VOXELS = 1 << 20     # 8 B of index + 4 B per float of velocity and scalars each: 40 MB with config 4's five scalar fields


def dump_outputs(directory: str, sim, names) -> None:
    """--dump-outputs: what the last timed frame hands back, the velocity (N, 3) and each scalar field (N), as float32 .npy files, at
    DUMP_VOXELS voxels drawn with a fixed seed (all of them on smaller domains); voxel_index.npy (float64) says which voxels."""
    os.makedirs(directory, exist_ok=True)
    n = sim.n
    idx = np.arange(n) if n <= DUMP_VOXELS else np.sort(np.random.default_rng(0).choice(n, DUMP_VOXELS, replace=False))
    np.save(os.path.join(directory, "voxel_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(directory, "velocity.npy"), sim.velocity()[idx])
    for i, name in enumerate(names):
        np.save(os.path.join(directory, f"{name}.npy"), sim.scalar(i)[idx])


# ----------------------------------------------------------------------------------------------------------------
# CPU baseline (oracle port) on a bounded sample
# ----------------------------------------------------------------------------------------------------------------
def cpu_baseline(w, names, fields, full: bool, sample_leaves: int = 12288, budget_s: float = 20.0) -> dict:
    from hnanosolver_b200 import synth
    from oracle import oracle as O

    L = min(sample_leaves, w.num_leaves)
    n = L * 512
    coords = synth.dense_coords(w.origins[:L])
    ix = O.OracleIndex(coords)
    vel = w.velocity[:n]
    fl = {k: a[:n] for k, a in zip(names, fields)}
    frames, t_used = 0, 0.0
    while frames < 1 or (t_used < budget_s / 2 and frames < 3):
        t = time.perf_counter()
        if full:
            ix.compute_sim(vel, fl, ITERATIONS, w.dt, w.voxel_size, PARAMS6)
        else:
            ix.frame(vel, list(fl.values()), ITERATIONS, w.dt, w.voxel_size)
        t_used += time.perf_counter() - t
        frames += 1
    return {"value": n * frames / t_used, "unit": "voxel-updates/s", "cores": O.num_threads(), "kind": "port",
            "sample": f"first {L} of {w.num_leaves} leaves ({n} voxels) of the same workload, {frames} full frame(s) at I={ITERATIONS}, "
                      f"oracle/hns_oracle.c with OpenMP"}


# ----------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c4", choices=["c1", "c2", "c3", "c4", "c5"])
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--forward-only", action="store_true", help="no back-to-front black sweeps (disables the L2 reuse between launches)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="multi-GPU c4: weak = 512^3 of sparse smoke per GPU (the box grows), strong = BASELINE.json config 4 as stated, the 512^3 box "
                         "split over the GPUs. c5 (1024^3 narrow band, ~2e8 voxels) is always a fixed total")
    ap.add_argument("--solver", default=None, choices=["rbgs", "mg"],
                    help="pressure solve of the timed frame: the reference's I red-black SOR iterations (default; bit-exact with the reference) or "
                         "multigrid V-cycles to a relative Poisson residual of 1e-4 (default for --workload c3, BASELINE.json config 3)")
    ap.add_argument("--mg-cycles", type=int, default=0, help="fixed number of V(2,2) cycles instead of solving to 1e-4")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the velocity and scalar fields of the last timed frame (a seeded sample of voxels) to DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)

    import torch

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: hnanosolver_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if args.dump_outputs and (args.impl == "reference" or world > 1):
        raise SystemExit("--dump-outputs: single-GPU runs of this implementation only")
    if args.impl == "reference":  # rank 0 alone times the reference; the other ranks leave without joining a process group
        return reference_arm(args, rank, world)
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import hnanosolver_b200 as H
    from hnanosolver_b200 import _lib, synth

    _lib.lib().hns_set_device(local_rank)
    t0 = time.time()
    w, names, fields, kind = build_workload(args.workload, rank, world, args.scaling)
    full = kind == "full"
    S = len(fields)
    log(f"[rank {rank}] workload {w.name}: {w.num_leaves} leaves, {w.num_voxels} voxels, S={S}, frame={kind}, generated in {time.time()-t0:.1f}s")
    flags = H.Simulation.FLAG_FORWARD_ONLY if args.forward_only else 0

    if world > 1:
        from hnanosolver_b200 import dist as hdist

        sampler = ClockSampler(local_rank) if rank == 0 else None
        if sampler:
            sampler.start()
        res = hdist.run_sharded_bench(w, names, fields, full, args, ITERATIONS, PARAMS6, rank, world, local_rank)
        if rank == 0:
            t_lo, t_hi = res.pop("_timed_wall")
            res["clocks"] = sampler.stop(t_lo, t_hi)
            # roofline of the dominant kernel on the slowest rank: one pressure half-sweep moves 8 B per OWNED voxel of that rank
            # (interior + boundary sweep together), timed with CUDA events around the pressure phase of one extra frame
            peak, peak_src = hbm_peak()
            pressure_ms, owned_voxels = res.pop("_pressure")
            sweep_ms = pressure_ms / (2 * ITERATIONS)
            achieved = 8 * owned_voxels / (sweep_ms * 1e-3) / 1e9
            res["roofline"] = {"bound": "hbm", "kernel": "k_rbgs_split (interior sweep + fused boundary sweep/ghost push of one colour, per rank)",
                               "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                               "traffic": (kernel_traffic()["k_rbgs_split"]["dram_bytes_per_voxel"] * owned_voxels) if "k_rbgs_split" in kernel_traffic() else None,
                               "algorithmic_bytes_per_launch": 8 * owned_voxels, "avg_launch_ms": sweep_ms, "launches_timed": 2 * ITERATIONS,
                               "peak_source": peak_src, "note": "max over ranks of the pressure phase incl. the pipelined ghost exchange"}
            print(json.dumps(res), flush=True)
        return

    # ---- device-resident frame -------------------------------------------------------------------------------
    grid = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    sim = H.Simulation(grid, S)
    sim.upload(w.velocity, fields)
    if full:
        sim.set_combustion(True, names.index("fuel"), names.index("waste"), names.index("temperature"), names.index("flame"),
                           H.CombustionParams(*PARAMS6))
    solver = args.solver or ("mg" if args.workload == "c3" else "rbgs")
    N = w.num_voxels
    mg = mg_info = None
    if solver == "mg" or args.workload == "c4":
        mg, mg_info = multigrid_setup(H, sim, grid, w, args, N)
    if solver == "mg":
        sim.set_pressure_solver(mg, mg_info["cycles"], MG_NU[0], MG_NU[1], MG_OMEGA)
    sim.time_frames(args.warmup, ITERATIONS, w.dt, flags)          # W untimed warm-up frames
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    _lib.lib().hns_launch_count_reset()
    packed0 = _lib.lib().hns_packed_advection_launches()
    torch.cuda.synchronize()
    tc0 = time.time()
    ms_total, ms_pressure = sim.time_frames(args.steps, ITERATIONS, w.dt, flags)   # K timed frames, CUDA events on the launch stream
    torch.cuda.synchronize()
    tc1 = time.time()
    launches = int(_lib.lib().hns_launch_count())
    packed_launches = int(_lib.lib().hns_packed_advection_launches() - packed0)
    clocks = sampler.stop(tc0, tc1)
    if args.dump_outputs:       # every timed frame starts from the same inputs: the state now holds the last one's result
        dump_outputs(args.dump_outputs, sim, names)
    ms_step = ms_total / args.steps
    value = N / (ms_step * 1e-3)
    solve_quality = frame_quality(sim)          # relative Poisson residual + ||div u_new|| of the frame just timed

    # ---- roofline of the dominant kernel -------------------------------------------------------------------------
    peak, peak_src = hbm_peak()
    if solver == "rbgs":
        n_sweeps = ITERATIONS * args.steps * 2
        sweep_ms = ms_pressure / n_sweeps
    else:
        # the same kernel dominates the multigrid frame: time 2 x 20 fine-level half-sweeps on their own (CUDA events, same stream)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sim.pressure_solve(3, H.launchers.omega_compute(w.voxel_size), flags)
        torch.cuda.synchronize()
        e0.record()
        sim.pressure_solve(20, H.launchers.omega_compute(w.voxel_size), flags)
        e1.record()
        torch.cuda.synchronize()
        n_sweeps, sweep_ms = 40, e0.elapsed_time(e1) / 40
    bytes_per_launch = 8 * N                                           # one colour: read other-colour p, read+write this colour's p, read its div
    achieved = bytes_per_launch / (sweep_ms * 1e-3) / 1e9
    # dram__bytes_read + dram__bytes_write of the kernel per launch from the committed `ncu --set full` capture of THIS kernel on the
    # config-4 workload (profiles/kernel_traffic.json says which capture), scaled by the voxel count; never measured inside a timed run
    kt = kernel_traffic().get("k_rbgs_split")
    traffic = kt["dram_bytes_per_voxel"] * N if kt else None
    roofline = {"bound": "hbm", "kernel": "k_rbgs_split (one red or black half-sweep on colour-split bricks)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "algorithmic_bytes_per_launch": bytes_per_launch, "avg_launch_ms": sweep_ms, "launches_timed": n_sweeps,
                "peak_source": peak_src,
                "share_of_frame": (ms_pressure / ms_total) if solver == "rbgs" else (sweep_ms * mg_info["fine_half_sweeps_per_solve"] / ms_step),
                "frame_algorithmic_GBps": (algorithmic_bytes_per_voxel(S, ITERATIONS, full) if solver == "rbgs" else
                                           mg_frame_bytes_per_voxel(S, full, mg_info)) * N / (ms_step * 1e-3) / 1e9}

    stages = stage_breakdown(H, sim, w, S, full, peak)

    # ---- the other solver beside it (config 4): the same frame with the pressure stage swapped -----------------------
    other = None
    if args.workload == "c4" and solver == "rbgs":
        sim.set_pressure_solver(mg, mg_info["cycles"], MG_NU[0], MG_NU[1], MG_OMEGA)
        sim.time_frames(args.warmup, ITERATIONS, w.dt, flags)
        ms2, pr2 = sim.time_frames(args.steps, ITERATIONS, w.dt, flags)
        other = dict(mg_info, ms_per_step=ms2 / args.steps, ms_pressure=pr2 / args.steps, value=N / (ms2 / args.steps * 1e-3), **frame_quality(sim),
                     frame_algorithmic_GBps=mg_frame_bytes_per_voxel(S, full, mg_info) * N / (ms2 / args.steps * 1e-3) / 1e9,
                     note="same frame, pressure stage = V-cycles instead of the reference's I red-black iterations: not the reference's "
                          "arithmetic, converges further (compare relative_residual with the headline frame's)")
        # ... and with ONE cycle: the relative Poisson residual of the reference's 40 iterations (solve_quality.relative_residual of the
        # headline frame) is reached or beaten by a single V(2,2) cycle, in a quarter of the time
        sim.set_pressure_solver(mg, 1, MG_NU[0], MG_NU[1], MG_OMEGA)
        sim.time_frames(args.warmup, ITERATIONS, w.dt, flags)
        ms1, pr1 = sim.time_frames(args.steps, ITERATIONS, w.dt, flags)
        other["one_cycle"] = dict(cycles=1, ms_per_step=ms1 / args.steps, ms_pressure=pr1 / args.steps, value=N / (ms1 / args.steps * 1e-3),
                                  **frame_quality(sim))
        sim.set_pressure_solver(None)
    del mg

    # ---- end to end through the drop-in launchers on pinned host buffers -------------------------------------------
    del sim
    data = H.GridIndexedData()
    data.setAllocationType(H.AllocationType.CudaPinned)
    data.allocateCoords(N)
    for a in range(0, w.num_leaves, 8192):
        b = min(w.num_leaves, a + 8192)
        data.pCoords()[a * 512:b * 512] = synth.dense_coords(w.origins[a:b])
    data.addValueBlock(H.VEC3F, "vel")
    data.pValues(H.VEC3F, "vel")[:] = w.velocity
    e2e_names = list(names)
    for nm, a in zip(names, fields):
        data.addValueBlock(H.FLOAT, nm)
        data.pValues(H.FLOAT, nm)[:] = a
    if not full:  # Compute_Sim needs the four combustion blocks (HNanoSolver.cu:193); add them so the same call can be made
        extra = synth.combustion_fields(w)
        for nm, a in extra.items():
            if nm not in e2e_names:
                data.addValueBlock(H.FLOAT, nm)
                data.pValues(H.FLOAT, nm)[:] = a
                e2e_names.append(nm)
    params = H.CombustionParams(*PARAMS6)

    t_grid = [0.0]

    def cook():
        t = time.perf_counter()
        g = H.CreateIndexGrid(data, w.voxel_size)                      # per cook, like SOP_HNanoSolverVerb::cook (SOP_HNanoSolver.cpp:231)
        t_grid[0] += time.perf_counter() - t                           # synchronous: host build, upload, neighbour-table kernel
        H.Compute_Sim(data, g, ITERATIONS, w.dt, w.voxel_size, params, False)
        g.reset()

    for _ in range(2):
        cook()
    torch.cuda.synchronize()
    t_grid[0] = 0.0
    te = time.perf_counter()
    for _ in range(args.e2e_steps):
        cook()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - te) * 1e3 / args.e2e_steps
    Se = len(e2e_names)
    e2e = {"value": N / (e2e_ms * 1e-3), "unit": "voxel-updates/s", "ms_per_step": e2e_ms, "steps": args.e2e_steps,
           "create_index_grid_ms": t_grid[0] * 1e3 / args.e2e_steps,
           "h2d_bytes_per_step": int(N * (12 + 4 * Se) + grid.nanovdb_buffer().size + w.num_leaves * 16),
           "d2h_bytes_per_step": int(N * (12 + 4 * Se)),
           "call": "CreateIndexGrid + Compute_Sim on a pinned GridIndexedData (velocity + %d float blocks), in place, synchronous" % Se}

    out = {"metric": "active voxel-updates/s per advect+project frame", "value": value, "unit": "voxel-updates/s", "n_gpus": 1,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": workload_label(args.workload, w, kind, S),
                      "l2": "inputs larger than L2 (per-field %.0f MB, frame working set %.1f GB); no flush" % (4 * N / 1e6, (9 + 2 * S) * 4 * N / 1e9),
                      "pressure": ("red/black half-sweeps on colour-split bricks, " + ("forward only" if args.forward_only else "alternating direction"))
                      if solver == "rbgs" else
                      f"multigrid: {mg_info['cycles']} V({MG_NU[0]},{MG_NU[1]}) cycles, omega {MG_OMEGA}, {mg_info['levels']} levels, "
                      f"solved to a relative Poisson residual of {mg_info['relative_residual_at_cycles']:.2e} (target 1e-4)"},
           "pressure_solver": solver, "solve_quality": solve_quality,
           "roofline": roofline, "stages": stages, "e2e": e2e, "gpu_launches": launches,
           "packed_advection_launches": packed_launches,   # of gpu_launches: advect_vector4 / advect_scalars4 (advect.cu, third generation)
           "clocks": clocks}
    if solver == "mg":
        out["multigrid"] = mg_info
    if other is not None:
        out["multigrid_frame"] = other
    if not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(w, names, fields, full)
    print(json.dumps(out), flush=True)


def reference_arm(args, rank, world):
    """The unmodified reference through its own launchers on the same workload (rank 0 only)."""
    if rank != 0:
        return
    import torch

    from hnanosolver_b200 import synth
    from oracle import oracle as O

    w, names, fields, kind = build_workload(args.workload, 0, 1)
    full = kind == "full"
    N = w.num_voxels
    line = {"impl": "reference", "metric": "active voxel-updates/s per advect+project frame", "unit": "voxel-updates/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": workload_label(args.workload, w, kind, len(fields))}}   # the same string as our arm's: same workload
    if O.ref_gpu_available():
        rd = O.RefData(synth.dense_coords(w.origins), 2)  # AllocationType::CudaPinned
        rd.add_vec3("vel", w.velocity)
        fl = dict(zip(names, fields))
        if not full:
            for k, v in synth.combustion_fields(w).items():
                fl.setdefault(k, v)
        for k, v in fl.items():
            rd.add_float(k, v)
        for _ in range(args.warmup):
            O.ref_cook_frame(rd, ITERATIONS, w.dt, w.voxel_size, PARAMS6)
        torch.cuda.synchronize()
        t = time.perf_counter()
        for _ in range(args.steps):
            O.ref_cook_frame(rd, ITERATIONS, w.dt, w.voxel_size, PARAMS6)
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t) * 1e3 / args.steps
        Se = len(fl)
        line.update(value=N / (ms * 1e-3), ms_per_step=ms,
                    reference_kind="the reference's own CUDA kernels and launchers (src/Cuda/*.cu compiled unmodified for sm_100a), "
                                   "CreateIndexGrid + Compute_Sim on a CudaPinned GridIndexedData, as SOP_HNanoSolverVerb::cook calls them",
                    e2e={"value": N / (ms * 1e-3), "unit": "voxel-updates/s", "h2d_bytes_per_step": int(N * (12 + 24 + 4 * Se)),
                         "d2h_bytes_per_step": int(N * (12 + 4 * Se)),
                         "note": "the reference API is host-buffer-in / host-buffer-out by construction, so value == e2e"})
    else:
        line.update(value=None, ms_per_step=None, reference_kind="oracle/_ref/libhns_ref.so not present; CPU port only")
    if not args.no_cpu_baseline:
        cb = cpu_baseline(w, names, fields, full)
        line["cpu_baseline"] = cb
        if line.get("value") is None:
            line["value"], line["ms_per_step"] = cb["value"], N / cb["value"] * 1e3
            line["e2e"] = {"value": cb["value"], "unit": "voxel-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
