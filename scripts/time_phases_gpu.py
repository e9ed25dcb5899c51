"""Per-stage device time of the resident frame on one GPU (CUDA events on the launch stream, no profiler).
Usage: time_phases_gpu.py [workload=c4] [repeats=10] [vorticity_scale,factor_scale]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import hnanosolver_b200 as H
from hnanosolver_b200 import synth

name = sys.argv[1] if len(sys.argv) > 1 else "c4"
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
vs, vf = (float(x) for x in (sys.argv[3] if len(sys.argv) > 3 else "0,1").split(","))
w = synth.WORKLOADS[name](with_coords=False)
fields = dict(density=w.scalars[0], **synth.combustion_fields(w))
names = list(fields)
g = H.create_index_grid_from_origins(w.origins, w.voxel_size)
sim = H.Simulation(g, len(fields))
sim.upload(w.velocity, list(fields.values()))
sim.set_combustion(True, names.index("fuel"), names.index("waste"), names.index("temperature"), names.index("flame"),
                   H.CombustionParams(0.5, 2.0, 1.5, 0.1, vs, vf))
from hnanosolver_b200 import launchers as HL
omega = HL.omega_compute(w.voxel_size)
st = torch.cuda.current_stream().cuda_stream
stages = [("advect_vector", lambda: sim.advect_velocity(w.dt, st)),
          ("vorticity", lambda: sim.vorticity_confinement(w.dt, vs, vf, st)),
          ("divergence", lambda: sim.divergence(True, st)),
          ("combustion+buoyancy", lambda: sim.combustion_buoyancy(w.dt, st)),
          ("pressure_solve(40)", lambda: sim.pressure_solve(40, omega, 0, st)),
          ("pressure_solve(40) forward only", lambda: sim.pressure_solve(40, omega, 2, st)),
          ("pressure_solve(40) again", lambda: sim.pressure_solve(40, omega, 0, st)),
          ("subtract_gradient", lambda: sim.subtract_gradient(True, st)),
          ("advect_scalars(5)", lambda: sim.advect_scalars(w.dt, 0, st))]
acc = {k: [] for k, _ in stages}
for r in range(reps + 2):
    for k, fn in stages:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        if r >= 2:
            acc[k].append(e0.elapsed_time(e1))
tot = 0.0
for k, v in acc.items():
    m = float(np.median(v)); tot += m
    print(f"{k:36s} {m:8.3f} ms  (min {min(v):.3f})")
print(f"{'sum':22s} {tot:8.3f} ms   {w.num_voxels / tot / 1e6:.1f} M voxel-updates/ms-frame -> {w.num_voxels / (tot * 1e-3) / 1e9:.2f} G/s")
