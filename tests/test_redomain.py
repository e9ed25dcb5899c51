"""Re-domaining a resident state (hns_state_domain_build, hns_state_create_remapped; Simulation.redomain): the SOP's domain step
(reference SOP_HNanoSolver.cpp:188-199) and the sidecar rebuild over the new domain (GridBuilder.hpp:87-166), on the device.

The contract is a composition of host functions that are tested elsewhere, restated here (`restate_*`):
  leaves = oracle.domain_leaves(io.union_topology(velocity topology at the tolerance, io.leaf_topology(source)...), padding, collider)
  field  = io.sidecar_from_grid(whole-domain export of the field, new leaves, fill 0; 0x01 for the collision SDF)
The velocity topology is io.leaf_topology of the Vec3f grid io.grid_from_sidecar writes over the leaves with an active voxel
(!(|v| <= tolerance) in any component, NaN active), with those masks; tolerance < 0: every leaf, every voxel. Results are compared as
float32 bits, so -0.0 != +0.0."""
import ctypes as C

import numpy as np
import pytest

import hnanosolver_b200 as H
from hnanosolver_b200 import _lib, synth
from hnanosolver_b200 import io as hio

PARAMS = [0.5, 2.0, 1.5, 0.1, 1.0, 2.0]  # combustion with vorticity confinement
H_VOX = 0.1


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


# ---- the host restatement ----------------------------------------------------------------------------------------------------------
def velocity_topology(origins, velocity, tolerance, voxel_size=H_VOX):
    """(origins, masks) of the velocity grid as export_grid("velocity", tolerance) writes it, read back with io.leaf_topology"""
    o = np.ascontiguousarray(np.asarray(origins, np.int32).reshape(-1, 3))
    v = np.asarray(velocity, np.float32).reshape(-1, 512, 3)
    if tolerance < 0:
        return o, np.full((len(o), 8), np.uint64(0xFFFFFFFFFFFFFFFF))
    with np.errstate(invalid="ignore"):
        active = ~(np.abs(v) <= np.float32(tolerance)).all(2)                  # NaN is active
    masks = np.packbits(active, axis=1, bitorder="little").view("<u8").astype(np.uint64)   # voxel n = x<<6|y<<3|z: bit n & 63 of word n >> 6
    keep = active.any(1)
    grid = hio.grid_from_sidecar(o[keep], v[keep].reshape(-1, 3), voxel_size, "vel", masks[keep])
    return hio.leaf_topology(grid)


def restate_leaves(O, origins, velocity, tolerance, padding, source_bufs=(), sdf_origins=None):
    topo = hio.union_topology(velocity_topology(origins, velocity, tolerance), *[hio.leaf_topology(b) for b in source_bufs])
    return O.domain_leaves(topo[0], topo[1], padding, sdf_origins)


def restate_field(old_origins, values, new_origins, fill=0, voxel_size=H_VOX):
    return hio.sidecar_from_grid(hio.grid_from_sidecar(old_origins, values, voxel_size, "f"), new_origins, fill)


# ---- CPU -----------------------------------------------------------------------------------------------------------------------------
def test_refusals_before_any_cuda_call():
    L = _lib.lib()
    d = C.c_void_p()
    cases = [((None, float("nan"), 0, 0, None, None, 0), "NaN"), ((None, 0.0, -1, 0, None, None, 0), "padding"),
             ((None, 0.0, 65, 0, None, None, 0), "padding"), ((None, 0.0, 0, 0, None, None, 0), "null")]
    for args, msg in cases:
        assert L.hns_state_domain_build(*args, C.byref(d)) == -1, args
        assert msg in L.hns_last_error().decode(), (args, L.hns_last_error())
        assert not d.value
    assert L.hns_state_domain_build(None, 0.0, 0, 0, None, None, 0, None) == -1
    assert L.hns_state_create_remapped(None, None, None, C.byref(d)) == -1 and "null" in L.hns_last_error().decode()


def _leaf(values_at):
    """one leaf's 512 voxels x 3 components, zero except {voxel offset x<<6|y<<3|z: value}"""
    v = np.zeros((512, 3), np.float32)
    for n, x in values_at.items():
        v[n, 1] = x
    return v


def test_restatement_known_answers(oracle_mod):
    O = oracle_mod
    o = np.array([[0, 0, 0], [16, 0, 0]], np.int32)
    vel = np.concatenate([_leaf({}), _leaf({3 << 6 | 3 << 3 | 3: 2.0})])    # leaf 0 all zero, leaf 1 one voxel in its middle
    # a leaf dropped by the tolerance contributes nothing, not even itself; tolerance < 0 keeps every leaf with every voxel
    assert restate_leaves(O, o, vel, 0.0, 0).tolist() == [[16, 0, 0]]
    assert restate_leaves(O, o, vel, 0.0, 3).tolist() == [[16, 0, 0]]      # voxel 3 +- 3 stays inside its leaf
    assert len(restate_leaves(O, o, vel, 0.0, 4)) == 8                      # 3 - 4 reaches the leaves below it, 3 + 4 does not
    assert restate_leaves(O, o, vel, 2.0, 1).shape == (0, 3)                # |2| <= 2: nothing is left
    assert restate_leaves(O, o, vel, -1.0, 0).tolist() == o.tolist()
    assert len(restate_leaves(O, o, vel, -1.0, 1)) == 27 + 27 - 9            # every voxel active: two 3x3x3 blocks sharing a face layer
    nan = np.concatenate([_leaf({}), _leaf({5: np.nan})])
    assert restate_leaves(O, o, nan, np.inf, 0).tolist() == [[16, 0, 0]]    # NaN is active at any tolerance
    # a face voxel with padding 1 reaches exactly the leaf across that face
    face = _leaf({7 << 6 | 3 << 3 | 3: -1.0})
    assert restate_leaves(O, o[:1], face, 0.0, 1).tolist() == [[0, 0, 0], [8, 0, 0]]
    # a source leaf outside the domain adds itself and what it reaches: its corner voxel (0, 0, 0) reaches the 7 leaves below it
    src = hio.grid_from_sidecar(np.array([[64, 0, 0]], np.int32), np.zeros(512, np.float32), H_VOX, "s",
                                np.array([[1, 0, 0, 0, 0, 0, 0, 0]], np.uint64))
    got = restate_leaves(O, o[:1], face, 0.0, 1, [src])
    want = {(0, 0, 0), (8, 0, 0)} | {(64 + 8 * a, 8 * b, 8 * c) for a in (-1, 0) for b in (-1, 0) for c in (-1, 0)}
    assert {tuple(x) for x in got.tolist()} == want and len(got) == len(want)
    assert np.array_equal(synth.nanovdb_order(got), np.arange(len(got)))
    # an empty source leaf is still a node; the collider's leaves are nodes
    empty = hio.grid_from_sidecar(np.array([[-64, 0, 0]], np.int32), np.zeros(512, np.float32), H_VOX, "s", np.zeros((1, 8), np.uint64))
    got = restate_leaves(O, o, vel, 2.0, 8, [empty], np.array([[0, 64, 0]], np.int32))     # the velocity contributes nothing
    assert got.tolist() == [[-64, 0, 0], [0, 64, 0]]
    # fields: carried over bit for bit where the old grid has the leaf, fill bytes elsewhere
    s = np.full(2 * 512, np.float32(-0.0))
    s[512:] = np.float32(np.ldexp(1.0, -140))
    new = np.array([[0, 0, 0], [8, 0, 0], [16, 0, 0]], np.int32)
    got = restate_field(o, s, new, 1)
    assert np.array_equal(_bits(got[:512]), _bits(s[:512])) and np.array_equal(_bits(got[1024:]), _bits(s[512:]))
    assert (_bits(got[512:1024]) == 0x01010101).all()
    assert (_bits(restate_field(o, vel, new, 0)[512:1024]) == 0).all()


# ---- GPU -----------------------------------------------------------------------------------------------------------------------------
def _domain():
    """leaves in two root tiles, one of them at negative coordinates, in NanoVDB order"""
    a = synth.random_leaves(40, 5, 3, with_coords=False).origins
    b = synth.random_leaves(20, 4, 4, offset=(-4096 - 64, -32, -8), with_coords=False).origins
    o = np.concatenate([a, b])
    return np.ascontiguousarray(o[synth.nanovdb_order(o)])


def _fields(domain, rng, S=3):
    """a sparse velocity (a third of the leaves zero, the rest zero but for a few voxels, small values among them, -0.0 and subnormals)
    with a NaN-only leaf, and S scalars with -0.0 and subnormals"""
    n = len(domain)
    vel = np.zeros((n, 512, 3), np.float32)
    live = rng.permutation(n)[: 2 * n // 3]
    for l in live:
        k = rng.integers(1, 6)
        vel[l, rng.integers(0, 512, k), rng.integers(0, 3, k)] = (rng.random(k) - 0.5).astype(np.float32) * np.float32(10.0) ** -rng.integers(0, 5, k)
    vel[live[0], :, 0] = np.float32(-0.0)
    vel[live[1], :7, 2] = np.float32(np.ldexp(1.0, -140))
    dead = np.setdiff1d(np.arange(n), live)
    vel[dead[0], 100:103, 1] = np.nan                                       # a leaf whose only non-zero values are NaN
    sc = [(rng.random(n * 512) - 0.5).astype(np.float32) for _ in range(S)]
    for s in sc:
        s[rng.integers(0, s.size, s.size // 8)] = np.float32(-0.0)
        s[rng.integers(0, s.size, s.size // 16)] = np.float32(np.ldexp(1.0, -140))
    return vel.reshape(-1, 3), sc


def _sources(domain, rng):
    """a float and a Vec3f source with partial masks: some domain leaves and some leaves outside it (one below every domain leaf)"""
    out = []
    for comps, far in ((1, [[-8200, -8, -8], [4096 + 8, 0, 0]]), (3, [[-4096 - 64 - 800, -32, -8], [200, 200, 200]])):
        inside = domain[rng.permutation(len(domain))[:5]]
        o = np.concatenate([inside, np.array(far, np.int32)])
        o = np.ascontiguousarray(o[synth.nanovdb_order(o)])
        v = (rng.random((len(o) * 512, comps)) - 0.5).astype(np.float32).reshape((-1, 3) if comps == 3 else -1)
        masks = np.zeros((len(o), 8), np.uint64)
        masks[:, rng.integers(0, 8)] = np.uint64(1) << np.uint64(rng.integers(0, 64))
        masks[0, 0] = np.uint64(1)                                          # voxel (0, 0, 0): reaches the lower neighbours
        out.append(hio.grid_from_sidecar(o, v, H_VOX, "src", masks))
    return out


def _state(domain, vel, sc, collision=None, combustion=False):
    sim = H.Simulation(H.create_index_grid_from_origins(domain, H_VOX), len(sc))
    sim.upload(vel, sc)
    if combustion:
        sim.set_combustion(True, 0, 1, 2, 3, H.CombustionParams(*PARAMS))
    if collision is not None:
        sim.set_collision(collision)
    return sim


def _origins(sim):
    o, _ = hio.leaf_topology(sim.export_grid(0, "o").download())
    return o


LEAF_CASES = [dict(tol=-1.0, pad=0, src=False, sdf=False), dict(tol=0.0, pad=0, src=False, sdf=False),
              dict(tol=0.0, pad=1, src=True, sdf=True), dict(tol=1e-3, pad=4, src=True, sdf=False),
              dict(tol=1e-3, pad=8, src=False, sdf=True), dict(tol=np.inf, pad=13, src=True, sdf=True),
              dict(tol=np.inf, pad=0, src=False, sdf=False), dict(tol=0.0, pad=64, src=True, sdf=False),
              dict(tol=-1.0, pad=13, src=True, sdf=True)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", LEAF_CASES)
def test_leaf_lists_equal_the_restatement(oracle_mod, case):
    rng = np.random.default_rng(7)
    domain = _domain()
    vel, sc = _fields(domain, rng)
    sim = _state(domain, vel, sc)
    bufs = _sources(domain, rng) if case["src"] else []
    sdf = domain[::9] if case["sdf"] else None
    want = restate_leaves(oracle_mod, domain, vel, case["tol"], case["pad"], bufs, sdf)
    new = sim.redomain(case["tol"], case["pad"], [H.Source(b) for b in bufs], sdf)
    assert np.array_equal(_origins(new), want)
    assert new.grid.num_leaves == len(want) and new.n == 512 * len(want)
    if case["tol"] == np.inf and not case["src"] and not case["sdf"]:
        assert len(want) == 1                                               # the NaN-only leaf and nothing else


@pytest.mark.gpu
def test_empty_and_collider_only_results(oracle_mod):
    domain = _domain()
    vel = np.zeros((len(domain) * 512, 3), np.float32)
    sim = _state(domain, vel, [np.ones(len(domain) * 512, np.float32)], collision=0)
    empty = sim.redomain(0.0, 8)
    assert empty.grid.num_leaves == 0 and empty.n == 0
    empty.step(4, 0.1)                                                       # a state without leaves takes a frame
    sdf = np.array([[-8200, 0, 0], domain[5]], np.int32)                   # NanoVDB order: the negative root tile first
    only = sim.redomain(0.0, 8, (), sdf)
    assert np.array_equal(_origins(only), restate_leaves(oracle_mod, domain, vel, 0.0, 8, (), sdf)) and only.grid.num_leaves == 2
    assert (_bits(only.scalar(0))[:512] == 0x01010101).all()                          # not in the old domain: the SDF fill
    assert (_bits(only.scalar(0))[512:] == _bits(np.ones(512, np.float32))).all()    # in the old domain: carried over


@pytest.mark.gpu
@pytest.mark.parametrize("tol,pad", [(0.0, 1), (-1.0, 4), (1e-3, 13)])
def test_fields_equal_the_restatement(oracle_mod, tol, pad):
    rng = np.random.default_rng(11)
    domain = _domain()
    vel, sc = _fields(domain, rng, S=4)
    sim = _state(domain, vel, sc, collision=2)
    bufs = _sources(domain, rng)
    new = sim.redomain(tol, pad, [H.Source(b) for b in bufs], domain[::7])
    no = _origins(new)
    assert np.array_equal(no, restate_leaves(oracle_mod, domain, vel, tol, pad, bufs, domain[::7]))
    assert not (domain == no[0]).all(1).any()                               # the new leaf 0 ("element 0" of advect_scalars) is new
    old = {tuple(x) for x in domain.tolist()}
    assert any(tuple(x) not in old for x in no.tolist()) and any(tuple(x) in old for x in no.tolist())
    whole = lambda t: sim.export_grid(t, "f", -1.0).download()               # noqa: E731
    assert np.array_equal(_bits(new.velocity()), _bits(hio.sidecar_from_grid(whole("velocity"), no, 0)))
    for i in range(4):
        want = hio.sidecar_from_grid(whole(i), no, 1 if i == 2 else 0)
        assert np.array_equal(_bits(new.scalar(i)), _bits(want)), i
        assert np.array_equal(_bits(want), _bits(restate_field(domain, sc[i], no, 1 if i == 2 else 0)))
    assert (_bits(new.scalar(2))[:512] == 0x01010101).all() and (_bits(new.scalar(1))[:512] == 0).all()
    # the pressure, divergence and advected velocity start as a new state's: zero
    for which in (H.Simulation.AUX_DIVERGENCE, H.Simulation.AUX_PRESSURE, H.Simulation.AUX_ADVECTED):
        assert (_bits(new.aux(which)) == 0).all()


def _frames(sim, n, stream=None):
    for _ in range(n):
        sim.step(8, 0.05, stream=stream)
    sim.sync(stream)
    out = dict(velocity=sim.velocity(), pressure=sim.aux(H.Simulation.AUX_PRESSURE))
    out.update({i: sim.scalar(i) for i in range(sim.n_scalars)})
    return out


def _plume_state(w, collision=True):
    c = synth.dense_coords(w.origins).astype(np.float32)
    sdf = (0.05 * (np.sqrt(((c - np.array([32.0, 30.0, 32.0], np.float32)) ** 2).sum(1)) - 6.0)).astype(np.float32)
    fields = [w.scalars[0], *synth.combustion_fields(w).values()]            # density, fuel, waste, temperature, flame
    fields = [fields[1], fields[2], fields[3], fields[4], fields[0], sdf]    # fuel, waste, temperature, flame, density, sdf
    return fields


@pytest.mark.gpu
@pytest.mark.parametrize("packed", [True, False])
def test_noop_redomain_keeps_every_bit(packed):
    w = synth.smoke_plume(64, 2, with_coords=False)
    fields = _plume_state(w)
    previous = _lib.lib().hns_set_packed_advection(int(packed))
    try:
        a = _state(w.origins, w.velocity, fields, collision=5, combustion=True)
        b = _state(w.origins, w.velocity, fields, collision=5, combustion=True)
        assert _lib.lib().hns_state_vorticity_active(a._h) == 1
        r = a.redomain(-1.0, 0)
        assert np.array_equal(_origins(r), w.origins)
        lib = _lib.lib()
        p0 = lib.hns_packed_advection_launches()
        want = _frames(b, 3)
        p1 = lib.hns_packed_advection_launches()
        got = _frames(r, 3)
        assert lib.hns_packed_advection_launches() - p1 == p1 - p0
        assert lib.hns_state_vorticity_active(r._h) == 1 and lib.hns_state_collision_active(r._h) == 1
        for k in want:
            assert np.array_equal(_bits(got[k]), _bits(want[k])), k
    finally:
        _lib.lib().hns_set_packed_advection(previous)


@pytest.mark.gpu
@pytest.mark.parametrize("packed,collision", [(True, False), (False, False), (True, True)])
def test_frames_after_a_change_equal_a_fresh_upload(oracle_mod, packed, collision):
    w = synth.smoke_plume(64, 2, with_coords=False)
    fields = _plume_state(w)
    so, values = synth.emitter(w.origins, fraction=0.1, speed=0.5)
    bufs = [hio.grid_from_sidecar(so, values["density"], w.voxel_size, "density"), hio.grid_from_sidecar(so, values["velocity"], w.voxel_size, "v")]
    previous = _lib.lib().hns_set_packed_advection(int(packed))
    try:
        sdf = 5 if collision else None
        sim = _state(w.origins, w.velocity, fields, collision=sdf, combustion=True)
        mg = H.Multigrid(sim.grid)
        sim.set_pressure_solver(mg, 2)
        _frames(sim, 1)
        vel, sc = sim.velocity(), [sim.scalar(i) for i in range(6)]
        new = sim.redomain(0.6, 1, [H.Source(b) for b in bufs], w.origins[::11])
        no = restate_leaves(oracle_mod, w.origins, vel, 0.6, 1, bufs, w.origins[::11])
        assert np.array_equal(_origins(new), no)
        old = {tuple(x) for x in w.origins.tolist()}
        new_set = {tuple(x) for x in no.tolist()}
        assert new_set - old                                                # the emitter's leaves outside the domain pull it there
        fresh = _state(no, restate_field(w.origins, vel, no), [restate_field(w.origins, s, no, 1 if i == sdf else 0) for i, s in enumerate(sc)],
                       collision=sdf, combustion=True)
        lib = _lib.lib()
        p0 = lib.hns_packed_advection_launches()
        want = _frames(fresh, 3)                                            # red-black: the multigrid solver is not carried over
        p1 = lib.hns_packed_advection_launches()
        got = _frames(new, 3)
        assert lib.hns_packed_advection_launches() - p1 == p1 - p0
        if packed and not collision:
            assert p1 - p0 > 0                                              # the packed kernels ran (they do not run with collision)
        for k in want:
            assert np.array_equal(_bits(got[k]), _bits(want[k])), k
    finally:
        _lib.lib().hns_set_packed_advection(previous)


@pytest.mark.gpu
def test_cook_loop_equals_the_host_loop(oracle_mod):
    """smoke_plume with an emitter and a sphere collider: restated domain -> build_sidecar -> comp_sum -> CreateIndexGrid -> Compute_Sim,
    the SDF block rebuilt from the collider every frame, against redomain -> add_source -> step"""
    O = oracle_mod
    w = synth.smoke_plume(64, 2, with_coords=False)
    h, iters, tol, pad = w.voxel_size, 12, 0.6, 1
    params = H.CombustionParams(*PARAMS)
    fields = dict(zip(["fuel", "waste", "temperature", "flame", "density", "collision_sdf"], _plume_state(w)))
    names = list(fields)
    inside = np.abs(fields["collision_sdf"].reshape(-1, 512)).min(1) < 0.3
    collider = np.ascontiguousarray(w.origins[inside])
    sdf_grid = hio.grid_from_sidecar(collider, fields["collision_sdf"].reshape(-1, 512)[inside].reshape(-1), h, "collision_sdf")
    so, values = synth.emitter(w.origins, fraction=0.1, speed=0.5)
    emitter = {k: hio.grid_from_sidecar(so, v, h, k) for k, v in values.items()}
    host_sources = [("vel" if k == "velocity" else k, b) for k, b in emitter.items()]
    sources = [H.Source(b) for b in emitter.values()]

    grids = [("vel", hio.grid_from_sidecar(w.origins, w.velocity, h, "vel"), False)]
    grids += [(k, hio.grid_from_sidecar(w.origins, v, h, k), False) for k, v in fields.items() if k != "collision_sdf"]
    grids += [("collision_sdf", sdf_grid, True)]
    origins = w.origins
    data = hio.build_sidecar(origins, grids)
    sim = H.Simulation(H.create_index_grid_from_origins(origins, h), len(names))
    sim.upload(data.pValues(H.VEC3F, "vel"), [data.pValues(H.FLOAT, k) for k in names])
    sim.set_combustion(True, 0, 1, 2, 3, params)
    sim.set_collision(5)
    counts, grew, shed = [len(origins)], False, False
    for _ in range(4):
        vel = data.pValues(H.VEC3F, "vel")
        topo = hio.union_topology(velocity_topology(origins, vel, tol, h), *[hio.leaf_topology(b) for b in emitter.values()])
        domain = O.domain_leaves(topo[0], topo[1], pad, collider)
        grids = [("vel", hio.grid_from_sidecar(origins, vel, h, "vel"), False)]
        grids += [(k, hio.grid_from_sidecar(origins, data.pValues(H.FLOAT, k), h, k), False) for k in names if k != "collision_sdf"]
        grids += [("collision_sdf", sdf_grid, True)]
        old, new = {tuple(x) for x in origins.tolist()}, {tuple(x) for x in domain.tolist()}
        grew, shed = grew or bool(new - old), shed or bool(old - new)
        origins = domain
        data = hio.build_sidecar(origins, grids)
        hio.comp_sum(origins, data, host_sources)
        grid = H.CreateIndexGrid(data, h)
        H.Compute_Sim(data, grid, iters, w.dt, h, params, True)

        sim = sim.redomain(tol, pad, sources, collider)
        for k, src in zip(emitter, sources):
            sim.add_source("velocity" if k == "velocity" else names.index(k), src)
        sim.step(iters, w.dt)
        sim.sync()
        counts.append(len(origins))
        assert np.array_equal(_origins(sim), origins)
        assert np.array_equal(_bits(sim.velocity()), _bits(data.pValues(H.VEC3F, "vel")))
        for i, k in enumerate(names[:-1]):
            assert np.array_equal(_bits(sim.scalar(i)), _bits(data.pValues(H.FLOAT, k))), (len(counts), k)
    assert grew and shed, counts


@pytest.mark.gpu
def test_source_state_is_unchanged():
    rng = np.random.default_rng(3)
    domain = _domain()
    vel, sc = _fields(domain, rng, S=5)
    vel = np.where(np.isnan(vel), np.float32(0.0), vel)
    a = _state(domain, vel, sc, collision=4, combustion=True)
    b = _state(domain, vel, sc, collision=4, combustion=True)
    before = [a.velocity()] + [a.scalar(i) for i in range(5)]
    stream = __import__("torch").cuda.Stream()
    a.redomain(0.0, 2, [H.Source(x) for x in _sources(domain, rng)], domain[:3], stream=stream)
    a.redomain(-1.0, 9)
    after = [a.velocity()] + [a.scalar(i) for i in range(5)]
    for x, y in zip(before, after):
        assert np.array_equal(_bits(x), _bits(y))
    got, want = _frames(a, 2), _frames(b, 2)
    for k in want:
        assert np.array_equal(_bits(got[k]), _bits(want[k])), k


@pytest.mark.gpu
def test_refusals_on_the_gpu():
    L = _lib.lib()
    domain = _domain()
    rng = np.random.default_rng(1)
    vel, sc = _fields(domain, rng, S=1)
    sim = _state(domain, vel, sc)
    d = C.c_void_p()

    def build(srcs=None, n_src=0, sdf=None):
        so = None if sdf is None else np.ascontiguousarray(sdf, np.int32)
        return L.hns_state_domain_build(sim._h, 0.0, 1, n_src, srcs, so.ctypes.data_as(_lib.c_i32p) if so is not None else None,
                                        0 if so is None else len(so), C.byref(d))

    assert build((C.c_void_p * 1)(None), 1) == -1 and "null source" in L.hns_last_error().decode()
    assert build(None, 1) == -1
    assert build(sdf=[[3, 0, 0]]) == -4
    assert build(sdf=[[1 << 23, 0, 0]]) == -5
    assert build(sdf=[[-(1 << 23) + 64, 0, 0]]) == -5
    far = H.Source(hio.grid_from_sidecar(np.array([[(1 << 23) - 64, 0, 0]], np.int32), np.zeros(512, np.float32), H_VOX, "s"))
    with pytest.raises(_lib.HnsError) as e:
        sim.redomain(0.0, 1, [far])
    assert e.value.code == -5
    edge = _state(np.array([[1 << 23, 0, 0]], np.int32), np.ones((512, 3), np.float32), [np.zeros(512, np.float32)])
    with pytest.raises(_lib.HnsError) as e:
        edge.redomain(-1.0, 0)
    assert e.value.code == -5
    with pytest.raises(_lib.HnsInvalidArgument):
        sim.redomain(float("nan"), 1)
    with pytest.raises(_lib.HnsInvalidArgument):
        sim.redomain(0.0, 65)
    # a sharded state: a one-rank plan installs a work list
    owned = np.ascontiguousarray(np.arange(len(domain)), np.int32)
    h = C.c_void_p()
    _lib.check(L.hns_dist_create(None, 0, 1, C.byref(h)))
    try:
        _lib.check(L.hns_dist_set_plan(h, sim._h, 0, None, None, None, None, None, len(owned), owned.ctypes.data_as(_lib.c_i32p)))
        with pytest.raises(_lib.HnsError) as e:
            sim.redomain(0.0, 1)
        assert e.value.code == -5 and "sharded" in e.value.message
        other = H.create_index_grid_from_origins(domain, H_VOX)
        assert L.hns_state_create_remapped(sim._h, other._h, None, C.byref(d)) == -5
    finally:
        L.hns_dist_destroy(h)
    import torch

    if torch.cuda.device_count() < 2:
        return
    L.hns_set_device(1)
    try:
        src1 = H.Source(hio.grid_from_sidecar(domain[:1], np.zeros(512, np.float32), H_VOX, "s"))
        grid1 = H.create_index_grid_from_origins(domain, H_VOX)
    finally:
        L.hns_set_device(0)
    plain = _state(domain, vel, sc)
    with pytest.raises(_lib.HnsInvalidArgument):
        plain.redomain(0.0, 1, [src1])
    assert L.hns_state_create_remapped(plain._h, grid1._h, None, C.byref(d)) == -1
