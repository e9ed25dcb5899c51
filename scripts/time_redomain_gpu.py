"""Cost of re-domaining a resident simulation on the device (Simulation.redomain) on bench.py's workload (config 4, after a few frames),
in one process:

  * by wall clock around calls that end in a device synchronise: the domain build (hns_state_domain_build: classify, candidates, sort,
    one readback), the index grid build (hns_domain_create_grid), the state allocation plus remap (hns_state_create_remapped), and the
    whole Simulation.redomain;
  * by CUDA events, the remap kernel alone: the stream is held by a device-side sleep while the host allocates, so the events bracket
    only the kernel (and an already satisfied wait on the allocation's memsets);
  * by wall clock, the host round trip the device path replaces: download every field, io.grid_from_sidecar + build_domain +
    io.sidecar_from_grid per field, upload into a new state.

    python scripts/time_redomain_gpu.py [--frames 3] [--tolerance 1e-3] [--padding 2] [--reps 5] [--out profiles/r3e_time_redomain.txt]

Algorithmic bytes of the remap: every new voxel's 3 + S floats written once, and read once where the old grid has its leaf; the copy
rate is MEASURED_PEAKS.json hbm_gbs when present, as in bench.py. The card's name and power limit are read in the same run.
"""
import argparse
import ctypes as C
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
from hnanosolver_b200 import _lib  # noqa: E402
from hnanosolver_b200 import io as hio  # noqa: E402
from hnanosolver_b200.launchers import _stream  # noqa: E402
from time_fused_combustion_gpu import card  # noqa: E402


def wall_ms(fn, reps: int):
    """(mean ms per call, last result); every call ends in a device synchronise"""
    out = None
    t = 0.0
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        t += time.perf_counter() - t0
    return t / reps * 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=3)
    ap.add_argument("--tolerance", type=float, default=1e-3)
    ap.add_argument("--padding", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3e_time_redomain.txt"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    L = _lib.lib()
    peak, peak_from = hbm_peak()
    w, names, fields, kind = build_workload("c4", 0, 1)
    assert kind == "full"
    grid = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    sim = H.Simulation(grid, len(fields))
    sim.set_combustion(True, names.index("fuel"), names.index("waste"), names.index("temperature"), names.index("flame"),
                       H.CombustionParams(*PARAMS6))
    sim.upload(w.velocity, fields)
    for _ in range(args.frames):
        sim.step(ITERATIONS, w.dt)
    sim.sync()
    S = len(fields)
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    tol, pad = args.tolerance, args.padding
    out = {"card": card(), "peak_gbs": peak, "peak_from": peak_from, "old_leaves": w.num_leaves, "scalars": S, "tolerance": tol, "padding": pad,
           "frames_before": args.frames}
    say(f"card: {out['card']}; copy rate {peak:.0f} GB/s ({peak_from}); config 4 after {args.frames} frames: {w.num_leaves} leaves, "
        f"{S} scalars; tolerance {tol:g}, padding {pad}")
    none = (C.c_void_p * 1)()

    def domain_build():
        d = C.c_void_p()
        _lib.check(L.hns_state_domain_build(sim._h, tol, pad, 0, none, None, 0, C.byref(d)))
        return d

    ms_dom, d = wall_ms(domain_build, args.reps)
    n_new = int(L.hns_domain_num_leaves(d))
    new_origins = np.empty((n_new, 3), np.int32)
    _lib.check(L.hns_domain_origins(d, new_origins.ctypes.data_as(_lib.c_i32p)))

    def grid_build():
        g = C.c_void_p()
        _lib.check(L.hns_domain_create_grid(d, w.voxel_size, C.byref(g)))
        return H.IndexGridHandle(g.value)

    ms_grid, new_grid = wall_ms(grid_build, args.reps)
    L.hns_domain_destroy(d)

    def remap(stream=None):
        h = C.c_void_p()
        _lib.check(L.hns_state_create_remapped(sim._h, new_grid._h, _stream(stream), C.byref(h)))
        return h

    def alloc_remap():
        L.hns_state_destroy(remap())

    ms_alloc_remap, _ = wall_ms(alloc_remap, args.reps)
    # the kernel alone: the stream sleeps on the device while the host allocates and zeroes the new state
    st = torch.cuda.Stream()
    kernel_ms = []
    for _ in range(args.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        with torch.cuda.stream(st):
            torch.cuda._sleep(1_000_000_000)
            e0.record(st)
            h = remap(st)
            e1.record(st)
        torch.cuda.synchronize()
        kernel_ms.append(e0.elapsed_time(e1))
        L.hns_state_destroy(h)
    ms_kernel = float(np.median(kernel_ms))
    old_keys = {tuple(x) for x in w.origins.tolist()}
    found = sum(tuple(x) in old_keys for x in new_origins.tolist())
    nbytes = (3 + S) * 4 * 512 * (n_new + found)
    ms_redomain, new_sim = wall_ms(lambda: sim.redomain(tol, pad), args.reps)
    assert new_sim.grid.num_leaves == n_new
    out.update(new_leaves=n_new, carried_leaves=found, domain_build_ms=ms_dom, grid_build_ms=ms_grid, alloc_remap_ms=ms_alloc_remap,
               redomain_ms=ms_redomain, remap_kernel_ms=ms_kernel, remap_kernel_ms_all=kernel_ms, remap_bytes=nbytes,
               remap_gbs=nbytes / ms_kernel / 1e6, remap_frac_of_copy=nbytes / ms_kernel / 1e6 / peak)
    say(f"new domain: {n_new} leaves, {found} of them carried over from the old grid")
    say(f"domain build {ms_dom:.3f} ms, grid build {ms_grid:.3f} ms, state allocation + remap {ms_alloc_remap:.3f} ms, whole redomain "
        f"{ms_redomain:.3f} ms (wall clock, mean of {args.reps})")
    say(f"remap kernel: {nbytes / 1e9:.3f} GB in {ms_kernel:.4f} ms (CUDA events, median of {args.reps}) -> {out['remap_gbs']:.0f} GB/s = "
        f"{out['remap_frac_of_copy']:.3f} of the copy rate")
    del new_sim

    # the host round trip it replaces
    t0 = time.perf_counter()
    vel = sim.velocity()
    sc = [sim.scalar(i) for i in range(S)]
    t1 = time.perf_counter()
    active = ~(np.abs(vel.reshape(-1, 512, 3)) <= np.float32(tol)).all(2)
    masks = np.packbits(active, axis=1, bitorder="little").view("<u8").astype(np.uint64)
    keep = active.any(1)
    host_origins = H.build_domain(w.origins[keep], masks[keep], pad)
    new_vel = hio.sidecar_from_grid(hio.grid_from_sidecar(w.origins, vel, w.voxel_size, "vel"), host_origins, 0)
    new_sc = [hio.sidecar_from_grid(hio.grid_from_sidecar(w.origins, s, w.voxel_size, "f"), host_origins, 0) for s in sc]
    t2 = time.perf_counter()
    host = H.Simulation(H.create_index_grid_from_origins(host_origins, w.voxel_size), S)
    host.upload(new_vel, new_sc)
    host.sync()
    t3 = time.perf_counter()
    assert np.array_equal(host_origins, new_origins)
    out.update(host_download_ms=(t1 - t0) * 1e3, host_rebuild_ms=(t2 - t1) * 1e3, host_upload_ms=(t3 - t2) * 1e3, host_total_ms=(t3 - t0) * 1e3,
               host_bytes_each_way=(3 + S) * 4 * w.num_voxels)
    say(f"host round trip: download {out['host_download_ms']:.1f} ms + topology / build_domain / sidecar rebuild {out['host_rebuild_ms']:.1f} ms "
        f"+ grid and state creation and upload {out['host_upload_ms']:.1f} ms = {out['host_total_ms']:.1f} ms")
    say(json.dumps(out))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
