"""Generates tests/golden/*.npz by running the UNMODIFIED reference (oracle/_ref/libhns_ref.so: the reference's own
src/Cuda/*.cu compiled for sm_100a) on small seeded inputs. Needs a GPU and the reference build under oracle/_ref/:

    python tests/golden/make_golden.py

The fixtures pin (a) the oracle (CPU tests, tests/test_oracle_golden.py) and (b) the CUDA path (tests/test_gpu_*.py)
to outputs of the reference itself.
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from hnanosolver_b200 import synth  # noqa: E402
from oracle import oracle as O  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
PARAMS = np.array([0.5, 2.0, 1.5, 0.1, 0.0, 1.0], np.float32)  # expansion, temp release, buoyancy, ambient, vorticity (off), factor


def case_inputs(name):
    if name == "soup":      # many missing neighbours, negative coordinates, three root tiles
        w = synth.random_leaves(28, 4, 7, offset=(-24, 4096 - 16, -16), cfl=1.8, S=2)
    elif name == "sphere":  # 32^3 smoke sphere (config-1 shape at half size)
        w = synth.smoke_sphere(32, 1)
    else:
        raise KeyError(name)
    rng = np.random.default_rng(123)
    n = w.num_voxels
    comb = dict(fuel=(rng.random(n) * (rng.random(n) < 0.4)).astype(np.float32), waste=(0.3 * rng.random(n)).astype(np.float32),
                temperature=rng.random(n).astype(np.float32), flame=(0.2 * rng.random(n)).astype(np.float32))
    for a in comb.values():
        a[0] = 0.0
    return w, comb


def collision_sdf(w):
    """a sphere collider in the middle of the active region; 0.05 per voxel, so that the reference's 0.1-wide boundary band
    (Kernel.cu:99, 438, 814) is two voxels thick and holds plenty of voxels; sidecar element 0 stays 0"""
    c = w.coords.astype(np.float32)
    centre = np.round(c.mean(0))
    r = np.sqrt(((c - centre) ** 2).sum(1))
    sdf = (0.05 * (r - 6.0)).astype(np.float32)
    sdf[0] = 0.0
    return sdf


def case_arrays(name):
    """Every array the reference is given in case `name`, under the name the fixture uses for it. The fixture stores only their
    digests: the tests regenerate them here (integer hashing and IEEE arithmetic, the same bits on every machine)."""
    w, comb = case_inputs(name)
    rng = np.random.default_rng(5)
    q = np.concatenate([w.coords[::5], w.coords[::9] + rng.integers(-9, 10, size=w.coords[::9].shape).astype(np.int32)])
    out = dict(origins=w.origins, coords=w.coords, velocity=w.velocity, query_ijk=q, collision_sdf=collision_sdf(w))
    for i, s in enumerate(w.scalars):
        out[f"scalar{i}"] = s
    for k, v in comb.items():
        out[f"comb_{k}"] = v
    return out


def digest(a) -> str:
    """SHA-256 of an array's dtype, shape and values; -0.0 counts as +0.0, as it does for `==`"""
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = a + a.dtype.type(0)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


# stored as they are: parameters, and what compresses to a few kilobytes (the index grid and its lookups)
KEEP = ("voxel_size", "dt", "iterations", "params", "scalar_names", "vorticity_cases", "nanovdb", "query_values")
SAMPLE = 32             # voxels whose output values are stored, for a readable failure message


def compact(name, out: dict) -> dict:
    """What the fixture stores of a case's full record `out`: KEEP as it is, the SHA-256 of every input (case_arrays) and of every
    output, and each output's values at SAMPLE seeded voxels. A test compares an output value for value on the sample and bit for bit
    (through the digest) on the whole array; the full record of both cases would take 10 MB."""
    inputs = case_arrays(name)
    n = len(inputs["coords"])
    idx = np.sort(np.random.default_rng(2024).choice(n, SAMPLE, replace=False))
    z = {"sample_index": idx}
    for k, v in out.items():
        if k in KEEP:
            z[k] = v
            continue
        if k in inputs:
            assert digest(v) == digest(inputs[k]), k
        else:
            z[k + ".sample"] = np.asarray(v)[idx]
        z[k + ".sha256"] = np.array(digest(v))
    return z


def make(name, iterations):
    w, comb = case_inputs(name)
    out = dict(case_arrays(name), voxel_size=np.float32(w.voxel_size), dt=np.float32(w.dt), iterations=np.int32(iterations), params=PARAMS,
               scalar_names=np.array(w.scalar_names))

    def data(vec=True, floats=()):
        d = O.RefData(w.coords)
        if vec:
            d.add_vec3("vel", w.velocity)
        for nm, a in floats:
            d.add_float(nm, a)
        return d

    # index grid
    d = data(floats=list(zip(w.scalar_names, w.scalars)))
    g = O.RefGrid(d, w.voxel_size)
    out["nanovdb"] = g.buffer()
    out["query_values"] = g.get_values(out["query_ijk"])
    # kernels, stage by stage (north-star frame)
    f = O.RefFrame(d, g, w.scalar_names)
    f.run(iterations, w.dt, w.voxel_size, 1)
    r = f.download()
    out.update(frame_adv=r["adv"], frame_div=r["div"], frame_p=r["p"], frame_vel=r["vel"])
    for i, s in enumerate(r["scalars"]):
        out[f"frame_scalar{i}"] = s
    # vorticityConfinement, the reference kernel launched out of place on the input velocity
    vc = [(1.0, 1.0), (0.7, 2.9), (1.3, -1.0)]
    out["vorticity_cases"] = np.array(vc, np.float32)
    for i, (sc, fs) in enumerate(vc):
        out[f"vorticity_{i}"] = f.vorticity(w.dt, w.voxel_size, sc, fs)
    # the hasCollision path, kernel by kernel (inputs of stages 2 and 3 are frame_adv / frame_p and frame_vel above)
    sdf = out["collision_sdf"]
    out["coll_enforce"] = f.collision_stage(0, sdf, w.dt, w.voxel_size)
    out["coll_advect_vector"] = f.collision_stage(1, sdf, w.dt, w.voxel_size)
    out["coll_gradient"] = f.collision_stage(2, sdf, w.dt, w.voxel_size)
    for i, sc in enumerate(f.collision_stage(3, sdf, w.dt, w.voxel_size)):
        out[f"coll_scalar{i}"] = sc
    # stand-alone launchers
    d = data(floats=list(zip(w.scalar_names, w.scalars)))
    O.ref_advect_index_grid(d, w.dt, w.voxel_size)
    for i, nm in enumerate(w.scalar_names):
        out[f"advect_index_grid_{i}"] = d.blocks[nm].copy()
    d = data()
    O.ref_advect_index_grid_velocity(d, w.dt, w.voxel_size)
    out["advect_index_grid_velocity"] = d.blocks["vel"].copy()
    d = data()
    O.ref_project_non_divergent(d, iterations, w.voxel_size)
    out["project_non_divergent"] = d.blocks["vel"].copy()
    d = data(floats=[("divergence", np.zeros(w.num_voxels, np.float32))])
    O.ref_divergence(d, w.voxel_size)
    out["divergence"] = d.blocks["divergence"].copy()
    # the all-in-one node: density + the four combustion fields, vorticity off
    fl = [("density", w.scalars[0])] + list(comb.items())
    d = data(floats=fl)
    g2 = O.RefGrid(d, w.voxel_size)
    O.ref_compute_sim(d, g2, iterations, w.dt, w.voxel_size, PARAMS, False)
    out["compute_sim_vel"] = d.blocks["vel"].copy()
    for nm, _ in fl:
        out[f"compute_sim_{nm}"] = d.blocks[nm].copy()
    # the same with the SOP's default vorticity parameters (scale 1, factor_scale 0.5: the offset truncates to 0, the in-place pass
    # then adds exactly zero)
    pv = PARAMS.copy()
    pv[4], pv[5] = 1.0, 0.5
    d = data(floats=fl)
    g3 = O.RefGrid(d, w.voxel_size)
    O.ref_compute_sim(d, g3, iterations, w.dt, w.voxel_size, pv, False)
    out["compute_sim_sopdefault_vel"] = d.blocks["vel"].copy()
    # the all-in-one node with a collision_sdf block and hasCollision = true
    d = data(floats=fl + [("collision_sdf", sdf)])
    g4 = O.RefGrid(d, w.voxel_size)
    O.ref_compute_sim(d, g4, iterations, w.dt, w.voxel_size, PARAMS, True)
    out["compute_sim_coll_vel"] = d.blocks["vel"].copy()
    for nm, _ in fl:
        out[f"compute_sim_coll_{nm}"] = d.blocks[nm].copy()
    out["compute_sim_coll_sdf_out"] = d.blocks["collision_sdf"].copy()  # what the reference hands back in the collision_sdf block
    np.savez_compressed(os.path.join(HERE, f"ref_{name}.npz"), **compact(name, out))
    print(name, "leaves", w.num_leaves, "voxels", w.num_voxels, "->", f"ref_{name}.npz")


if __name__ == "__main__":
    make("soup", 6)
    make("sphere", 12)
