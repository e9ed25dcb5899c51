"""Headless driver: what the Houdini SOP does around the hot path, without Houdini (reference src/SOP/HNanoSolver/SOP_HNanoSolver.cpp:
build the sidecar, CreateIndexGrid once per topology, then one Compute_Sim per frame), on a 128^3-bounded smoke plume.

    python examples/headless_driver.py [frames=8] [out_dir] [--redomain]

Two ways to run a frame are shown side by side and must agree bit for bit:
  * the drop-in launchers on HOST buffers (CreateIndexGrid + Compute_Sim), every frame crossing PCIe like the reference does, and
  * the resident state (Simulation.step), which keeps the fields in HBM between frames.
An emitter at the plume's base (density, temperature and fuel sources and an upward velocity source, as NanoVDB grids) is added in
front of every frame, as the SOP does with compSum (SOP_HNanoSolver.cpp:159-181): on the host blocks with io.comp_sum, on the
resident state with Simulation.add_source. The domain stays fixed: the emitter's leaves outside it are dropped.
With --redomain the domain follows the fluid, as the SOP's does: before every frame both paths rebuild it from the velocity's active
voxels (|v| > 0.6), dilated by one voxel, united with the emitter's leaves and the collider's (SOP_HNanoSolver.cpp:188-199). The
host-buffer path rebuilds its sidecar (io.union_topology, build_domain, io.build_sidecar with the SDF block rebuilt from the collider
grid, CreateIndexGrid); the resident path calls Simulation.redomain, then add_source, then step. The leaf count is printed per frame.
With an output directory the last frame is written as a NanoVDB file + sidecar blocks (hnanosolver_b200.io) and read back, and every
field is written as a float / Vec3f .nvdb grid twice: by the host writer from the host buffers, and exported from the resident state on
the device (Simulation.export_grid), which must give the same bytes; a pruned export (tolerance 0) is written next to it.
"""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import hnanosolver_b200 as H
from hnanosolver_b200 import io as hio
from hnanosolver_b200 import synth

redomain = "--redomain" in sys.argv
argv = [a for a in sys.argv[1:] if a != "--redomain"]
frames = int(argv[0]) if len(argv) > 0 else 8
out_dir = argv[1] if len(argv) > 1 else None
tolerance, padding = 0.6, 1  # --redomain
iterations = 40
w = synth.smoke_plume(128, 2)
fields = dict(density=w.scalars[0], **synth.combustion_fields(w))
# a sphere collider in the plume's way (third SOP input), 0.05 per voxel so the 0.1-wide boundary band is two voxels thick
c = w.coords.astype(np.float32)
fields["collision_sdf"] = (0.05 * (np.sqrt(((c - np.array([64.0, 72.0, 64.0], np.float32)) ** 2).sum(1)) - 10.0)).astype(np.float32)
params = H.CombustionParams(0.5, 2.0, 1.5, 0.1, 1.0, 0.5)  # expansion, temperature gain, buoyancy, ambient, vorticity 1, factor_scale 0.5 (SOP defaults)
names = list(fields)

# ---- drop-in launchers on host buffers ----
data = H.GridIndexedData()
data.setAllocationType(H.AllocationType.CudaPinned)
data.allocateCoords(w.num_voxels)
data.pCoords()[:] = w.coords
data.addValueBlock(H.VEC3F, "vel")
data.pValues(H.VEC3F, "vel")[:] = w.velocity
for k, v in fields.items():
    data.addValueBlock(H.FLOAT, k)
    data.pValues(H.FLOAT, k)[:] = v
grid = H.CreateIndexGrid(data, w.voxel_size)

# ---- resident state ----
sim = H.Simulation(grid, len(fields))
sim.upload(w.velocity, list(fields.values()))
sim.set_combustion(True, names.index("fuel"), names.index("waste"), names.index("temperature"), names.index("flame"), params)
sim.set_collision(names.index("collision_sdf"))

# ---- emitter: 2 % of the leaves at the plume's base and four leaves outside the domain ----
src_origins, src_values = synth.emitter(w.origins, fraction=0.02, speed=0.2 * float(np.abs(w.velocity).max()))
emitter = {k: hio.grid_from_sidecar(src_origins, v, w.voxel_size, k) for k, v in src_values.items()}
host_sources = [("vel" if k == "velocity" else k, buf) for k, buf in emitter.items()]
device_sources = [("velocity" if k == "velocity" else names.index(k), H.Source(buf)) for k, buf in emitter.items()]
print(f"emitter: {len(src_origins)} leaves, {device_sources[0][1].leaves_outside(grid)} of them outside the domain "
      f"({'pulling the domain there' if redomain else 'dropped'})")
# --redomain: the collider as a grid over the first domain, so every later domain keeps its leaves and the SDF block can be rebuilt
sdf_grid = hio.grid_from_sidecar(w.origins, fields["collision_sdf"], w.voxel_size, "collision_sdf")
origins = w.origins

t_host = t_dev = 0.0
for f in range(frames):
    if not redomain:
        data.pValues(H.FLOAT, "collision_sdf")[:] = fields["collision_sdf"]   # the launcher hands the SDF block back zeroed, like the reference
    t0 = time.perf_counter()
    if redomain:
        vel = data.pValues(H.VEC3F, "vel")
        active = ~(np.abs(vel.reshape(-1, 512, 3)) <= np.float32(tolerance)).all(2)
        masks = np.packbits(active, axis=1, bitorder="little").view("<u8").astype(np.uint64)   # word x, bit y*8+z
        keep = active.any(1)
        topo = hio.union_topology((origins[keep], masks[keep]), *[hio.leaf_topology(buf) for _, buf in host_sources])
        new_origins = H.build_domain(topo[0], topo[1], padding, w.origins)
        grids = [("vel", hio.grid_from_sidecar(origins, vel, w.voxel_size, "vel"), False)]
        grids += [(k, hio.grid_from_sidecar(origins, data.pValues(H.FLOAT, k), w.voxel_size, k), False) for k in names if k != "collision_sdf"]
        grids.append(("collision_sdf", sdf_grid, True))
        origins = new_origins
        data = hio.build_sidecar(origins, grids)
        grid = H.CreateIndexGrid(data, w.voxel_size)
    hio.comp_sum(origins, data, host_sources)
    H.Compute_Sim(data, grid, iterations, w.dt, w.voxel_size, params, True)
    t1 = time.perf_counter()
    if redomain:
        sim = sim.redomain(tolerance, padding, [src for _, src in device_sources], w.origins)
    for target, src in device_sources:
        sim.add_source(target, src)
    sim.step(iterations, w.dt)
    sim.sync()
    t2 = time.perf_counter()
    t_host += t1 - t0
    t_dev += t2 - t1
    vel = data.pValues(H.VEC3F, "vel")
    same = np.array_equal(sim.velocity(), vel) and all(np.array_equal(sim.scalar(i), data.pValues(H.FLOAT, k)) for i, k in enumerate(names) if k != "collision_sdf")
    print(f"frame {f + 1}: {len(origins)} leaves  max|u| {np.abs(vel).max():8.4f}  mean density {data.pValues(H.FLOAT, 'density').mean():.6f}  "
          f"max temperature {data.pValues(H.FLOAT, 'temperature').max():.4f}  host-buffer path == resident path: {same}", flush=True)
    assert same
print(f"{len(origins)} leaves, {512 * len(origins)} voxels, {iterations} pressure iterations: {t_host / frames * 1e3:.2f} ms per frame through the "
      f"launchers on host buffers (sourcing on the host included), {t_dev / frames * 1e3:.2f} ms per frame on resident state")

if out_dir:
    hio.save_cache(out_dir, grid.nanovdb_buffer(), data)
    origins, h, back = hio.load_cache(out_dir)
    g2 = H.create_index_grid_from_origins(origins, h)
    assert np.array_equal(g2.nanovdb_buffer()[672:], grid.nanovdb_buffer()[672:]) and np.array_equal(back.pValues(H.VEC3F, "vel"), vel)
    print(f"wrote and re-read {out_dir}/grid.nvdb ({os.path.getsize(os.path.join(out_dir, 'grid.nvdb'))} bytes) + {back.numValueBlocks()} sidecar blocks")
    # the cache frame as the SOP writes it (writeIndexGrid per field): from the host buffers, and exported from the resident state on
    # the device, whole-domain (the same bytes) and pruned at tolerance 0 (leaves that hold only zeros left out). The collision SDF is
    # an input, not a result: the launcher hands its block back zeroed, the resident state keeps it.
    paths = hio.write_index_grids(os.path.join(out_dir, "grids"), origins, data, w.voxel_size)
    pruned_dir = os.path.join(out_dir, "grids_pruned")
    os.makedirs(pruned_dir, exist_ok=True)
    vg = H.ValueGrid()
    for path in paths:
        name = os.path.basename(path)[:-len(".nvdb")]
        if name == "collision_sdf":
            continue
        target = "velocity" if name == "vel" else names.index(name)
        assert np.array_equal(sim.export_grid(target, name, -1.0, vg).download(), hio.read_nvdb(path)), name
        pruned = os.path.join(pruned_dir, f"{name}.nvdb")
        hio.write_nvdb(pruned, sim.export_grid(target, name, 0.0, vg).download())
        print(f"{name:12s} whole domain {os.path.getsize(path):10d} bytes (host writer == device export), pruned at 0: "
              f"{os.path.getsize(pruned):10d} bytes, {vg.num_leaves} of {len(origins)} leaves")
