"""Sources on resident state (hns_source_*, hns_state_add_source_*; Simulation.add_source): openvdb::tools::compSum of NanoVDB float and
Vec3f grids into the fields, as SOP_HNanoSolverVerb::cook does every cook (reference SOP_HNanoSolver.cpp:159-181). The contract is
io.comp_sum on the host, bit for bit: every voxel of the domain gets value + s, s = +0.0 where the source has no leaf (which turns a
-0.0 into +0.0), source leaves outside the fixed domain are dropped."""
import numpy as np
import pytest

import hnanosolver_b200 as H
from hnanosolver_b200 import _lib, synth
from hnanosolver_b200 import io as hio

PARAMS6 = [0.5, 2.0, 1.5, 0.1, 0.0, 1.0]
TINY = np.float32(np.ldexp(1.0, -140))  # a subnormal


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _float_grid(origins, seed=0):
    o = np.ascontiguousarray(origins, np.int32)
    v = np.random.default_rng(seed).random(len(o) * 512).astype(np.float32)
    return hio.grid_from_sidecar(o, v, 0.1, "src")


def _code(buf):
    with pytest.raises(_lib.HnsError) as e:
        H.Source(buf)
    return e.value.code


# ---- host validation: refused before any CUDA call (on a machine without a GPU a valid buffer fails with HNS_ERR_CUDA instead) ----
def test_source_refuses_malformed_buffers_before_touching_cuda():
    o = synth.random_leaves(6, 3, 1, with_coords=False).origins
    buf = _float_grid(o)
    assert _code(buf[: buf.size // 2]) == -1                                  # truncated
    past = buf.copy()
    past[672 + 32:672 + 36] = np.frombuffer(np.uint32(10 ** 6).tobytes(), np.uint8)   # TreeData::nodeCount[0]: the leaf table reaches past the end
    assert _code(past) == -1
    assert "leaf nodes lie outside" in _lib.lib().hns_last_error().decode()
    dup = buf.copy()
    leaf0 = 672 + int(np.frombuffer(buf[672:680].tobytes(), np.uint64)[0])    # TreeData::nodeOffset[0]
    dup[leaf0 + 2144:leaf0 + 2144 + 12] = buf[leaf0:leaf0 + 12]               # leaf 1 gets leaf 0's bboxMin
    assert _code(dup) == -1
    assert "have the origin" in _lib.lib().hns_last_error().decode()
    index = buf.copy()
    index[636:640] = np.frombuffer(np.uint32(hio.GRID_TYPE_ONINDEX).tobytes(), np.uint8)
    assert _code(index) == -5                                                 # HNS_ERR_UNSUPPORTED
    double = buf.copy()
    double[636:640] = np.frombuffer(np.uint32(2).tobytes(), np.uint8)         # GridType::Double
    assert _code(double) == -5


# ---- GPU ---------------------------------------------------------------------------------------------------------------------------
def _domain():
    """leaves in two root tiles, one of them at negative coordinates"""
    a = synth.random_leaves(40, 5, 3, with_coords=False).origins
    b = synth.random_leaves(20, 4, 4, offset=(-4096 - 64, -32, -8), with_coords=False).origins
    o = np.concatenate([a, b])
    return np.ascontiguousarray(o[synth.nanovdb_order(o)])


def _special(n, rng, comps=1):
    """random values with planted -0.0, +0.0 and subnormals of both signs"""
    v = (rng.random((n, comps)) - 0.5).astype(np.float32)
    flat = v.reshape(-1)
    k = flat.size
    flat[rng.integers(0, k, k // 8)] = np.float32(-0.0)
    flat[rng.integers(0, k, k // 16)] = np.float32(0.0)
    flat[rng.integers(0, k, k // 16)] = TINY * rng.integers(1, 5, k // 16).astype(np.float32)
    flat[rng.integers(0, k, k // 16)] = -TINY
    return v if comps == 3 else v.reshape(-1)


def _source(domain, rng, comps):
    """half the domain's leaves, plus leaves outside it in both root tiles: (origins, values, NanoVDB buffer)"""
    inside = domain[rng.permutation(len(domain))[: len(domain) // 2]]
    outside = np.array([[4096 + 8, 0, 0], [-4096 - 64 - 800, -32, -8], [-8, -8, -8]], np.int32)
    o = np.concatenate([inside, outside])
    o = np.ascontiguousarray(o[synth.nanovdb_order(o)])
    v = _special(len(o) * 512, rng, comps)
    return o, v, hio.grid_from_sidecar(o, v, 0.25, "src")


def _comp_sum(domain, field, buf, comps):
    data = H.GridIndexedData()
    data.allocateCoords(len(domain) * 512)
    kind = H.VEC3F if comps == 3 else H.FLOAT
    data.addValueBlock(kind, "f")
    data.pValues(kind, "f")[:] = field
    hio.comp_sum(domain, data, [("f", buf)])
    return data.pValues(kind, "f").copy()


@pytest.mark.gpu
def test_add_source_is_comp_sum_bit_for_bit():
    rng = np.random.default_rng(5)
    domain = _domain()
    n = len(domain) * 512
    grid = H.create_index_grid_from_origins(domain, 0.1)
    vel, s0, s1 = _special(n, rng, 3), _special(n, rng), _special(n, rng)
    sim = H.Simulation(grid, 2)
    sim.upload(vel, [s0, s1])
    so, _, fbuf = _source(domain, rng, 1)
    vo, _, vbuf = _source(domain, rng, 3)
    fsrc, vsrc = H.Source(fbuf), H.Source(vbuf)
    assert (fsrc.components, vsrc.components) == (1, 3) and fsrc.num_leaves == len(so)
    known = {tuple(x) for x in domain.tolist()}
    assert fsrc.leaves_outside(grid) == sum(tuple(x) not in known for x in so.tolist()) == 3
    assert vsrc.leaves_outside(grid) == 3
    sim.add_source(1, fsrc)
    sim.add_source("velocity", vsrc)
    sim.sync()
    assert np.array_equal(_bits(sim.scalar(1)), _bits(_comp_sum(domain, s1, fbuf, 1)))
    assert np.array_equal(_bits(sim.velocity()), _bits(_comp_sum(domain, vel, vbuf, 3)))
    assert np.array_equal(_bits(sim.scalar(0)), _bits(s0))                    # the other field is untouched
    assert (np.signbit(s1) & (s1 == 0)).any() and ((s1 != 0) & (np.abs(s1) < np.finfo(np.float32).tiny)).any()


@pytest.mark.gpu
def test_empty_source_turns_minus_zero_into_plus_zero_and_nothing_else():
    rng = np.random.default_rng(6)
    domain = _domain()
    n = len(domain) * 512
    sim = H.Simulation(H.create_index_grid_from_origins(domain, 0.1), 1)
    vel, s0 = _special(n, rng, 3), _special(n, rng)
    sim.upload(vel, [s0])
    none = np.zeros((0, 3), np.int32)
    fsrc = H.Source(hio.grid_from_sidecar(none, np.zeros(0, np.float32), 0.1, "empty"))
    vsrc = H.Source(hio.grid_from_sidecar(none, np.zeros((0, 3), np.float32), 0.1, "empty"))
    assert fsrc.num_leaves == vsrc.num_leaves == 0 and fsrc.leaves_outside(sim.grid) == 0
    _lib.lib().hns_launch_count_reset()
    sim.add_source(0, fsrc)
    sim.add_source("velocity", vsrc)
    sim.sync()
    assert _lib.lib().hns_launch_count() == 2
    for got, was in ((sim.scalar(0), s0), (sim.velocity(), vel)):
        want = np.where(was == 0, np.float32(0.0), was)                     # -0.0 -> +0.0, every other value (subnormals too) kept
        assert np.array_equal(_bits(got), _bits(want))
        assert (np.signbit(was) & (was == 0)).any() and (_bits(got) != _bits(was)).sum() == (np.signbit(was) & (was == 0)).sum()


def _plume():
    w = synth.smoke_plume(64, 2, with_coords=False)
    fields = dict(density=w.scalars[0], **synth.combustion_fields(w))
    so, values = synth.emitter(w.origins, fraction=0.1, speed=0.1 * float(np.abs(w.velocity).max()))
    bufs = {k: hio.grid_from_sidecar(so, v, w.voxel_size, k) for k, v in values.items()}
    return w, fields, bufs


def _resident_frames(w, fields, bufs, targets, combustion, collision, frames, by_upload):
    """`frames` frames of Simulation.step with the sources `targets` added in front of each, on the device (add_source) or by
    download -> io.comp_sum -> upload (by_upload). -> (every field after the last frame, packed advection launches)"""
    names = list(fields) + (["collision_sdf"] if collision else [])
    arrays = list(fields.values())
    if collision:
        c = synth.dense_coords(w.origins).astype(np.float32)
        arrays.append((0.05 * (np.sqrt(((c - np.float32(32.0)) ** 2).sum(1)) - 8.0)).astype(np.float32))
    grid = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    sim = H.Simulation(grid, len(names))
    sim.upload(w.velocity, arrays)
    if combustion:
        sim.set_combustion(True, 1, 2, 3, 4, H.CombustionParams(*PARAMS6))
    if collision:
        sim.set_collision(len(names) - 1)
    srcs = {k: H.Source(bufs[k]) for k in targets}
    lib = _lib.lib()
    packed0 = lib.hns_packed_advection_launches()
    for _ in range(frames):
        if by_upload:
            data = H.GridIndexedData()
            data.allocateCoords(w.num_voxels)
            data.addValueBlock(H.VEC3F, "velocity")
            data.pValues(H.VEC3F, "velocity")[:] = sim.velocity()
            for i, k in enumerate(names):
                data.addValueBlock(H.FLOAT, k)
                data.pValues(H.FLOAT, k)[:] = sim.scalar(i)
            hio.comp_sum(w.origins, data, [(k, bufs[k]) for k in targets])
            sim.upload(data.pValues(H.VEC3F, "velocity"), [data.pValues(H.FLOAT, k) for k in names])
        else:
            for k, src in srcs.items():
                sim.add_source("velocity" if k == "velocity" else names.index(k), src)
        sim.step(12, w.dt)
    sim.sync()
    packed = lib.hns_packed_advection_launches() - packed0
    out = dict(velocity=sim.velocity(), pressure=sim.aux(H.Simulation.AUX_PRESSURE))
    out.update({k: sim.scalar(i) for i, k in enumerate(names)})
    return out, packed


@pytest.mark.gpu
@pytest.mark.parametrize("combustion,packed,collision", [(True, True, False), (True, False, False), (False, True, False), (False, False, False),
                                                         (True, True, True)])
def test_sourced_frames_equal_sourcing_on_the_host(combustion, packed, collision):
    w, fields, bufs = _plume()
    frames = 3
    previous = _lib.lib().hns_set_packed_advection(int(packed))
    try:
        _, packed_plain = _resident_frames(w, fields, bufs, [], combustion, collision, frames, False)
        for targets in (["density", "temperature", "fuel"], ["density", "temperature", "fuel", "velocity"]):
            got, packed_got = _resident_frames(w, fields, bufs, targets, combustion, collision, frames, False)
            want, _ = _resident_frames(w, fields, bufs, targets, combustion, collision, frames, True)
            for k in want:
                assert np.array_equal(_bits(got[k]), _bits(want[k])), (targets, k)
            if "velocity" not in targets:
                assert packed_got == packed_plain      # group 0's velocity lanes stay current: advect_vector keeps the third generation
            elif packed and not collision:
                assert packed_got == packed_plain - (frames - 1)   # a sourced velocity: advect_vector takes the second generation
        if packed and not collision and combustion:
            assert packed_plain == 2 * frames - 1      # the first frame's advect_vector finds no group yet (the upload)
        if not packed or collision:
            assert packed_plain == 0
    finally:
        _lib.lib().hns_set_packed_advection(previous)


@pytest.mark.gpu
def test_compute_sim_with_comp_sum_equals_resident_add_source():
    """the headless driver's loop on a small box: combustion, vorticity confinement and the collision path"""
    w, fields, bufs = _plume()
    c = synth.dense_coords(w.origins).astype(np.float32)
    fields["collision_sdf"] = (0.05 * (np.sqrt(((c - np.array([32.0, 36.0, 32.0], np.float32)) ** 2).sum(1)) - 6.0)).astype(np.float32)
    params = H.CombustionParams(0.5, 2.0, 1.5, 0.1, 1.0, 2.0)
    names = list(fields)
    data = H.GridIndexedData()
    data.allocateCoords(w.num_voxels)
    data.pCoords()[:] = synth.dense_coords(w.origins)
    data.addValueBlock(H.VEC3F, "vel")
    data.pValues(H.VEC3F, "vel")[:] = w.velocity
    for k, v in fields.items():
        data.addValueBlock(H.FLOAT, k)
        data.pValues(H.FLOAT, k)[:] = v
    grid = H.CreateIndexGrid(data, w.voxel_size)
    sim = H.Simulation(grid, len(fields))
    sim.upload(w.velocity, list(fields.values()))
    sim.set_combustion(True, names.index("fuel"), names.index("waste"), names.index("temperature"), names.index("flame"), params)
    sim.set_collision(names.index("collision_sdf"))
    srcs = {k: H.Source(b) for k, b in bufs.items()}
    assert srcs["density"].leaves_outside(grid) == 4
    host_sources = [("vel" if k == "velocity" else k, b) for k, b in bufs.items()]
    for _ in range(3):
        data.pValues(H.FLOAT, "collision_sdf")[:] = fields["collision_sdf"]
        hio.comp_sum(w.origins, data, host_sources)
        H.Compute_Sim(data, grid, 12, w.dt, w.voxel_size, params, True)
        for k, src in srcs.items():
            sim.add_source("velocity" if k == "velocity" else names.index(k), src)
        sim.step(12, w.dt)
        sim.sync()
        assert np.array_equal(_bits(sim.velocity()), _bits(data.pValues(H.VEC3F, "vel")))
        for i, k in enumerate(names):
            if k != "collision_sdf":
                assert np.array_equal(_bits(sim.scalar(i)), _bits(data.pValues(H.FLOAT, k))), k


@pytest.mark.gpu
def test_add_source_refusals():
    w, fields, bufs = _plume()
    grid = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    sim = H.Simulation(grid, 2)
    fsrc, vsrc = H.Source(bufs["density"]), H.Source(bufs["velocity"])
    for target, src in (("velocity", fsrc), (0, vsrc), (-1, fsrc), (2, fsrc)):
        with pytest.raises(_lib.HnsInvalidArgument):
            sim.add_source(target, src)
    with pytest.raises(ValueError):
        sim.add_source("density", fsrc)
    import torch

    if torch.cuda.device_count() < 2:
        return
    lib = _lib.lib()
    lib.hns_set_device(1)
    try:
        other = H.Source(bufs["density"])
    finally:
        lib.hns_set_device(0)
    with pytest.raises(_lib.HnsInvalidArgument):
        sim.add_source(0, other)
    with pytest.raises(_lib.HnsInvalidArgument):
        other.leaves_outside(grid)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_sourcing_is_bitwise_the_single_gpu_sourcing(world):
    from test_sharded_gpu import _gpus, _run

    modes = [dict(source=True), dict(source=True, collision=True, vorticity=[0.8, 2.0]), dict(source=True, combustion=False, frames=3)]
    reports = _run(world, modes, _gpus() < world)
    assert all(r["sources"] == 4 for r in reports)
