"""Sharded multigrid against the sharded red-black solve on config 4 (BASELINE.json: the 512^3 sparse smoke box) split over the ranks.

    torchrun --nproc-per-node N scripts/time_sharded_multigrid_gpu.py [--frames 10] [--out sharded_mg.json]

Three pressure solvers in the same sharded frame (ShardedSimulation.frame_timed, CUDA events between the phases): red-black with
I = 40, 1 x V(2,2), 2 x V(2,2). For each: median frame and pressure-phase time over --frames timed frames (slowest rank), the level-1
gather bytes per cycle of each rank, and the global relative residual sqrt(sum (div - L p)^2 / sum div^2) of the last frame (per-rank
residual sums added with torch.distributed). With one rank the same solvers also run through Simulation.time_frames on the whole grid:
the difference is the overhead of the sharded path. One GPU per rank (NCCL process group); the card name and power limit are read in
the same run."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from hnanosolver_b200 import _lib  # noqa: E402
from hnanosolver_b200 import dist as hdist  # noqa: E402
from hnanosolver_b200 import launchers as H  # noqa: E402

ARMS = [("red-black I=40", None), ("1 x V(2,2)", 1), ("2 x V(2,2)", 2)]


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q.stdout.strip().splitlines())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(lr)
    _lib.lib().hns_set_device(lr)
    dev = torch.device("cuda", lr)
    dist.init_process_group("nccl", device_id=dev)
    w, names, fields, _ = hdist.build_sharded_workload("c4", rank, world, "strong")
    plan = w.meta["plan"]
    go = hdist.global_sparse_origins(w.meta["box"])
    P = H.CombustionParams(0.5, 2.0, 1.5, 0.1, 0.0, 1.0)
    sh = hdist.ShardedSimulation(plan, w.origins, w.voxel_size, len(fields), dev)
    sh.set_combustion(names, P)
    result = dict(world=world, card=card() if rank == 0 else None, global_leaves=int(go.shape[0]), frames=a.frames,
                  multi_gpu_measured=world > 1, arms=[])
    for label, cycles in ARMS:
        sh.set_pressure_solver(None if cycles is None else go, cycles=cycles or 2)
        sh.upload(w.velocity, fields)
        dist.barrier()
        for _ in range(a.warmup):
            sh.frame(40, w.dt)
        torch.cuda.synchronize()
        g0 = sh.mg_gathers
        frame_ms, pressure_ms = [], []
        for _ in range(a.frames):
            ph = sh.frame_timed(40, w.dt)
            frame_ms.append(sum(v for k, v in ph.items() if k in hdist.ShardedSimulation.PHASES))
            pressure_ms.append(ph["pressure"])
        sh.check_errors()
        g1 = sh.mg_gathers
        sums = torch.tensor(sh.sim.residual_sums(), dtype=torch.float64, device=dev)
        dist.all_reduce(sums)
        t = torch.tensor([float(np.median(frame_ms)), float(np.median(pressure_ms))], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        per_cycle = (g1[1] - g0[1]) // max(1, g1[0] - g0[0]) if cycles else 0
        pc = torch.tensor([float(per_cycle)], device=dev)
        allpc = [torch.zeros_like(pc) for _ in range(world)]
        dist.all_gather(allpc, pc)
        arm = dict(solver=label, frame_ms=float(t[0]), pressure_ms=float(t[1]), gather_bytes_per_cycle_per_rank=[int(x.item()) for x in allpc],
                   rel_residual=float(np.sqrt(sums[0].item() / sums[1].item())) if sums[1].item() > 0 else 0.0)
        if world == 1:
            # the same solver through the single-GPU frame over the whole grid
            g = H.create_index_grid_from_origins(go, w.voxel_size)
            sim = H.Simulation(g, len(fields))
            sim.set_combustion(True, 1, 2, 3, 4, P)
            mg = H.Multigrid(g) if cycles else None
            sim.set_pressure_solver(mg, cycles or 2)
            sim.upload(w.velocity, fields)
            sim.time_frames(a.warmup, 40, w.dt)
            tot, pr = sim.time_frames(a.frames, 40, w.dt)
            arm.update(single_gpu_frame_ms=tot / a.frames, single_gpu_pressure_ms=pr / a.frames,
                       single_gpu_rel_residual=sim.relative_residual())
            del sim, mg, g
        result["arms"].append(arm)
        if rank == 0:
            print(json.dumps(arm), flush=True)
    sh.close()
    dist.destroy_process_group()
    if rank == 0:
        print("RESULT", json.dumps(result), flush=True)
        if a.out:
            os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
            with open(a.out, "w") as f:
                json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
