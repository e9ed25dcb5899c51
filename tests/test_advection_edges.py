"""The paths the benchmark times and the edges of the third-generation advection kernels (advect.cu), against the reference and the
CPU oracle, bit for bit:

* the timed frame (Simulation.time_frames: group 0 packed in front of every frame, so advect_vector runs the packed kernel, with the
  combustion update fused into it) on config 4, against what the reference computed for the same inputs;
* traces whose floors land on both sides of every bound of the staged region (footprint4: leaf-local -3..9 in x and y, -4..10 in z),
  exact integers and one ulp beyond them included, in leaves that hold hot and cold voxels at once;
* persistent CTAs that walk two to four work items (the metadata ring, the double buffer and the early issue of the next item);
* the fused combustion update with vorticity confinement on, every scalar count the state accepts, and advect_scalar semantics (inactive
  corners read 0) on the packed group.

Every test also checks which kernels ran (hns_packed_advection_launches, hns_launch_count): a silent fall-back to the second generation
would prove nothing here.
"""
import contextlib
import functools
import os

import numpy as np
import pytest

import hnanosolver_b200 as H
from helpers import RECORDED, Reference, assert_close, combustion_fields
from hnanosolver_b200 import _lib, synth
from hnanosolver_b200.grid_data import FLOAT, VEC3F, GridIndexedData
from oracle import oracle as O

pytestmark = pytest.mark.gpu
PARAMS6 = [0.5, 2.0, 1.5, 0.1, 0.0, 1.0]  # expansionRate, temperatureRelease, buoyancyStrength, ambientTemp, vorticity off
COMBUSTION = ["fuel", "waste", "temperature", "flame"]


@pytest.fixture(scope="module", autouse=True)
def _save_recording():
    yield
    if RECORDED.recording:
        RECORDED.save()


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def assert_same_bits(got, want, what):
    """equal bit for bit, signed zeros included"""
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    assert got.shape == want.shape, what
    assert_close(got, want, what)
    assert np.array_equal(_bits(got), _bits(want)), f"{what}: equal values but not equal bits (signed zeros)"


@contextlib.contextmanager
def schedule(packed: bool, fused: bool = True):
    """the packed advection kernels on or off (hns_set_packed_advection) and the fused combustion update on or off
    (HNS_FUSED_COMBUSTION, read at every frame); both restored afterwards"""
    lib = _lib.lib()
    prev = lib.hns_set_packed_advection(int(packed))
    before = os.environ.get("HNS_FUSED_COMBUSTION")
    os.environ["HNS_FUSED_COMBUSTION"] = "1" if fused else "0"
    try:
        yield
    finally:
        lib.hns_set_packed_advection(prev)
        if before is None:
            del os.environ["HNS_FUSED_COMBUSTION"]
        else:
            os.environ["HNS_FUSED_COMBUSTION"] = before


@contextlib.contextmanager
def counting():
    """{"launches": kernel launches, "packed": third-generation advection launches} of the block, filled in when it ends"""
    lib = _lib.lib()
    out = {}
    lib.hns_launch_count_reset()
    packed0 = lib.hns_packed_advection_launches()
    yield out
    out["launches"] = int(lib.hns_launch_count())
    out["packed"] = int(lib.hns_packed_advection_launches() - packed0)


def frame_launches(iterations, packed_in_front=False, combustion=None):
    """kernel launches of one frame on resident fields: [group 0 packed in front (time_frames)] + advect_vector (hot + flagged leaves) +
    divergence + iterations x (red, black) + the combustion stage's own kernels ("fused": none, "one_pass": the pass that also packs
    group 1, "two_passes": combustion and buoyancy) + gradient + advect_scalars (hot + flagged leaves)"""
    return int(packed_in_front) + 2 + 1 + 2 * iterations + {None: 0, "fused": 0, "one_pass": 1, "two_passes": 2}[combustion] + 1 + 2


def _simulation(origins, voxel_size, velocity, fields, combustion, params=PARAMS6):
    sim = H.Simulation(H.create_index_grid_from_origins(origins, voxel_size), len(fields))
    sim.upload(velocity, list(fields.values()))
    if combustion:
        names = list(fields)
        sim.set_combustion(True, *[names.index(k) for k in COMBUSTION], H.CombustionParams(*params))
    return sim


def _outputs(sim, names):
    out = dict(vel=sim.velocity(), adv=sim.aux(H.Simulation.AUX_ADVECTED), div=sim.aux(H.Simulation.AUX_DIVERGENCE),
               p=sim.aux(H.Simulation.AUX_PRESSURE))
    out.update({k: sim.scalar(i) for i, k in enumerate(names)})
    return out


# ------------------------------------------------------------------------------------------------------------------
# A. the timed frame on config 4 against the reference
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def c4():
    w = synth.WORKLOADS["c4"](with_coords=False)
    return w, dict(density=w.scalars[0], **synth.combustion_fields(w))


@pytest.fixture(scope="module")
def c4_cook_reference(c4):
    """what the reference's CreateIndexGrid + Compute_Sim computed on config 4 with density and the four combustion fields, I = 40"""
    w, fields = c4
    coords = synth.dense_coords(w.origins)

    def live():
        rd = O.RefData(coords)
        rd.add_vec3("vel", w.velocity)
        for k, v in fields.items():
            rd.add_float(k, v)
        O.ref_cook_frame(rd, 40, w.dt, w.voxel_size, np.asarray(PARAMS6, np.float32))
        return {k: v.copy() for k, v in rd.blocks.items()}

    return Reference(f"cook/{w.name}", live, [coords, w.velocity, *fields.values()])


@pytest.mark.parametrize("which", ["fused", "split", "second_generation"])
def test_timed_frame_with_combustion_matches_reference_on_config4(c4, c4_cook_reference, which):
    """bench.py's frame as bench.py times it: every one of the two frames starts from the inputs, group 0 packed in front"""
    w, fields = c4
    sim = _simulation(w.origins, w.voxel_size, w.velocity, fields, True)
    packed = which != "second_generation"
    with schedule(packed, fused=which == "fused"), counting() as n:
        sim.time_frames(2, 40, w.dt)
        sim.sync()
    assert n["packed"] == (2 * 2 if packed else 0)  # advect_vector and advect_scalars on the packed groups in both frames
    assert n["launches"] == 2 * frame_launches(40, packed, {"fused": "fused", "split": "one_pass", "second_generation": "two_passes"}[which])
    c4_cook_reference.check(sim.velocity(), "vel", f"{which}: velocity")
    for i, k in enumerate(fields):
        c4_cook_reference.check(sim.scalar(i), k, f"{which}: {k}")
    sim.close()


def test_timed_north_star_frame_matches_reference_on_config4(c4):
    w, _ = c4

    def live():
        rd = O.RefData(synth.dense_coords(w.origins))
        rd.add_vec3("vel", w.velocity)
        for n, a in zip(w.scalar_names, w.scalars):
            rd.add_float(n, a)
        rf = O.RefFrame(rd, O.RefGrid(rd, w.voxel_size), w.scalar_names)
        rf.run(40, w.dt, w.voxel_size, 1)
        want = rf.download()
        return dict(want, **{f"scalar{i}": s for i, s in enumerate(want.pop("scalars"))})

    ref = Reference(f"frame/{w.name}", live, [w.origins, w.velocity, *w.scalars])
    sim = _simulation(w.origins, w.voxel_size, w.velocity, dict(zip(w.scalar_names, w.scalars)), False)
    with schedule(True), counting() as n:
        sim.time_frames(2, 40, w.dt)
        sim.sync()
    assert n["packed"] == 2          # advect_vector only: two scalars have no producer for their second group
    assert n["launches"] == 2 * frame_launches(40, True)
    got = _outputs(sim, [f"scalar{i}" for i in range(len(w.scalars))])
    for k in ("adv", "div", "p", "vel", "scalar0", "scalar1"):
        ref.check(got[k], k, k)
    sim.close()


# ------------------------------------------------------------------------------------------------------------------
# B. the edges of the staged region
# ------------------------------------------------------------------------------------------------------------------
# footprint4 / footprint: the floor of a trace, relative to the leaf origin, must lie in [-3, 9] (x, y) and [-4, 10] (z)
LO = np.array([-3, -3, -4])
HI = np.array([9, 9, 10])
EDGE_H = EDGE_DT = 0.5  # sdt = dt / h = 1: the back-trace is p - u and the forward trace b + u(b), each rounded once


def _edge_origins():
    """a dense 3x3x3 block, scattered leaves with missing neighbours (an isolated pair among them), and leaves at negative
    coordinates on both sides of the root-tile boundary y = 4096"""
    dense = [(8 * i, 8 * j, 8 * k) for i in range(3) for j in range(3) for k in range(3)]
    scattered = [(48, 0, 0), (56, 0, 0), (40, 40, 40), (0, 48, 24), (64, 16, 8), (32, 64, 56), (72, 72, 0), (24, 0, 48)]
    tiles = [(x, y, z) for x in (-16, -8) for y in (4080, 4088, 4096) for z in (-16, -8)] + [(-40, 4104, -32), (-64, 4072, 8)]
    o = np.array(dense + scattered + tiles, np.int32)
    return np.ascontiguousarray(o[synth.nanovdb_order(o)])


def _edge_displacement(kind, o, axis):
    """one component of a leaf's constant displacement (voxels per step) for a displacement kind; `o` = the leaf origin's component"""
    lo, hi = int(LO[axis]), int(HI[axis])
    if kind == "lo_exact":    # voxel 0 traces to exactly o + lo: the lowest floor the region accepts
        return np.float32(-lo)
    if kind == "hi_exact":    # voxel 7 traces to exactly o + hi + 1: the first floor past the region
        return np.float32(-(hi + 1 - 7))
    if kind in ("lo_ulp", "hi_ulp"):  # one ulp below o + lo (outside) / below o + hi + 1 (inside), where that u is a float
        p0, edge = (o, o + lo) if kind == "lo_ulp" else (o + 7, o + hi + 1)
        return np.float32(np.float64(p0) - np.float64(np.nextafter(np.float32(edge), np.float32(-np.inf))))
    return np.float32(kind)


# per-axis displacement kinds: the exact and one-ulp traces, both sides of each bound, small values, a tiny one, and far ones (tree walk)
EDGE_KINDS = ["lo_exact", "hi_exact", "lo_ulp", "hi_ulp", 0.0, 0.5, -0.75, 1.25, -1.5, 2.5, -2.5, 3.5, -3.5, 4.5, -4.5, 2.0 ** -20, 12.0, -5.25]


@functools.lru_cache(maxsize=None)
def edge_case():
    origins = _edge_origins()
    L = len(origins)
    coords = synth.dense_coords(origins)
    disp = np.empty((L, 3), np.float32)
    for l in range(L):
        kinds = [EDGE_KINDS[(7 * l + 5 * a + (l // len(EDGE_KINDS))) % len(EDGE_KINDS)] for a in range(3)]
        if l < 12:   # the exact and one-ulp traces once more per axis, the other two axes well inside the region
            kinds = [0.5, 0.5, 0.5]
            kinds[l % 3] = EDGE_KINDS[l // 3]
        for a in range(3):
            disp[l, a] = _edge_displacement(kinds[a], int(origins[l, a]), a)
    velocity = np.repeat(disp, 512, axis=0)   # sdt = 1: velocity = displacement
    rng = np.random.default_rng(11)
    n = L * 512
    density = rng.random(n).astype(np.float32)
    density[0] = 100.0                         # advect_scalars' inactive corners read element 0: make it stand out
    comb = combustion_fields(n, seed=5)
    for k, v in zip(COMBUSTION, (0.75, 0.125, 0.875, 0.0625)):
        comb[k][0] = v
    return origins, coords, velocity, density, comb


def classify(origins, coords, velocity):
    """host copy of footprint4 for both traces of advect_vector: (b, f, floors of b and f relative to the leaf origin)"""
    o = np.repeat(origins.astype(np.int64), 512, axis=0)
    b = coords.astype(np.float32) - velocity                            # fmaf(-1, u, p)
    ub = O.OracleIndex(coords).trilinear_v(velocity.reshape(-1), b)      # the velocity at b, the reference's sampler
    f = b + ub                                                           # fmaf(1, u(b), b)
    return b, f, np.floor(b).astype(np.int64) - o, np.floor(f).astype(np.int64) - o


def _inside(fl):
    return ((fl >= LO) & (fl <= HI)).all(1)


def test_edge_inputs_reach_both_sides_of_every_bound():
    """the inputs of the edge tests do what they are built for (classified on the host, no kernel involved)"""
    origins, coords, velocity, _, _ = edge_case()
    b, f, bl, fl = classify(origins, coords, velocity)
    o = np.repeat(origins.astype(np.int64), 512, axis=0)
    hot_b = _inside(bl)
    hot = hot_b & _inside(fl)
    for a in range(3):
        others = [c for c in range(3) if c != a]
        for trace, fl_, gate in (("back", bl, np.ones_like(hot_b)), ("forward", fl, hot_b)):
            ok = gate & ((fl_[:, others] >= LO[others]) & (fl_[:, others] <= HI[others])).all(1)   # this axis alone decides
            for floor in (LO[a] - 1, LO[a], HI[a], HI[a] + 1):
                assert (ok & (fl_[:, a] == floor)).any(), f"{trace} trace: no floor {floor} on axis {'xyz'[a]}"
        ok = ((bl[:, others] >= LO[others]) & (bl[:, others] <= HI[others])).all(1)
        for edge in (LO[a], HI[a] + 1):
            exact = (o[:, a] + edge).astype(np.float32)
            below = np.nextafter(exact, np.float32(-np.inf))
            assert (ok & (b[:, a] == exact)).any(), f"back trace: none exactly at {edge} on axis {'xyz'[a]}"
            assert (ok & (b[:, a] == below)).any(), f"back trace: none one ulp below {edge} on axis {'xyz'[a]}"
    per_leaf = hot.reshape(-1, 512)
    mixed = per_leaf.any(1) & ~per_leaf.all(1)
    assert mixed.sum() >= len(origins) // 2, f"only {mixed.sum()} of {len(origins)} leaves hold hot and cold voxels"
    assert per_leaf.all(1).any() and (~per_leaf).all(1).any()     # and some leaves are all hot, some all cold


@pytest.mark.parametrize("which", ["second_generation", "packed", "fused"])
def test_staged_region_edges_match_oracle(which):
    """one frame through time_frames on the edge inputs: every output against the oracle (with combustion for `fused`, whose cold
    exits are the only place the combustion outputs of those voxels are written)"""
    origins, coords, velocity, density, comb = edge_case()
    ix = O.OracleIndex(coords)
    I = 3
    packed = which != "second_generation"
    fields = dict(density=density, **comb) if which == "fused" else dict(density=density)
    sim = _simulation(origins, EDGE_H, velocity, fields, which == "fused")
    with schedule(packed), counting() as n:
        sim.time_frames(1, I, EDGE_DT)
        sim.sync()
    assert n["packed"] == (2 if packed else 0)    # advect_vector, and advect_scalars on group 0 (S = 1) or groups 0 and 1
    assert n["launches"] == frame_launches(I, packed, "fused" if which == "fused" else None)
    got = _outputs(sim, list(fields))
    sim.close()
    if which == "fused":
        want_vel, want = ix.compute_sim(velocity, fields, I, EDGE_DT, EDGE_H, np.asarray(PARAMS6, np.float32))
        assert_same_bits(got["vel"], want_vel, "velocity")
        for k in fields:
            assert_same_bits(got[k], want[k], k)
        return
    assert_same_bits(got["adv"], ix.advect_vector(velocity, EDGE_DT, EDGE_H), "advect_vector")
    want = ix.frame(velocity, [density], I, EDGE_DT, EDGE_H)
    for k in ("adv", "div", "p", "vel"):
        assert_same_bits(got[k], want[k], k)
    assert_same_bits(got["density"], want["scalars"][0], "density")


# ------------------------------------------------------------------------------------------------------------------
# C. persistent CTAs that walk several leaves, over consecutive frames
# ------------------------------------------------------------------------------------------------------------------
def _sms():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


@functools.lru_cache(maxsize=None)
def walk_case(n_leaves):
    """a random soup at CFL 2.5, 5 % of the leaves displaced far beyond the staged region"""
    extent = int(np.ceil((3 * n_leaves) ** (1 / 3)))
    w = synth.random_leaves(n_leaves, extent, 21, cfl=2.5, S=1)
    assert w.num_leaves == n_leaves
    far = np.random.default_rng(3).choice(n_leaves, max(1, n_leaves // 20), replace=False)
    v = w.velocity.reshape(-1, 512, 3)
    v[far] *= np.float32(3.5)
    return w, dict(density=w.scalars[0], **combustion_fields(w.num_voxels, seed=9))


@functools.lru_cache(maxsize=None)
def walk_oracle(n_leaves, combustion, iterations, frames=3):
    w, fields = walk_case(n_leaves)
    ix = O.OracleIndex(w.coords)
    vel = w.velocity
    if not combustion:
        sc = [fields["density"]]
        for _ in range(frames):
            r = ix.frame(vel, sc, iterations, w.dt, w.voxel_size)
            vel, sc = r["vel"], r["scalars"]
        return dict(vel=vel, density=sc[0])
    for _ in range(frames):
        vel, fields = ix.compute_sim(vel, fields, iterations, w.dt, w.voxel_size, np.asarray(PARAMS6, np.float32))
    return dict(vel=vel, **fields)


@pytest.mark.parametrize("which", ["fused", "split", "density_only", "second_generation"])
@pytest.mark.parametrize("size", ["2sm+1", "6.5sm+3"])
def test_multi_item_ctas_over_consecutive_frames_match_oracle(size, which):
    """L = 2 SMs + 1 and 6 SMs + SMs / 2 + 3 leaves: the 2 SMs CTAs of the advection kernels walk two to four leaves each, with an
    uneven tail. Three step() frames: the first finds no group 0 (second-generation advect_vector), the next two run the packed
    advect_vector, fused with the combustion update unless `split`."""
    sms = _sms()
    L = 2 * sms + 1 if size == "2sm+1" else 6 * sms + sms // 2 + 3
    assert L > 2 * sms
    w, fields = walk_case(L)
    combustion = which != "density_only"
    if not combustion:
        fields = dict(density=fields["density"])
    I = 6
    sim = _simulation(w.origins, w.voxel_size, w.velocity, fields, combustion)
    packed = which != "second_generation"
    with schedule(packed, fused=which == "fused"), counting() as n:
        for _ in range(3):
            sim.step(I, w.dt)
        sim.sync()
    assert n["packed"] == (1 + 2 + 2 if packed else 0)
    comb = {"fused": ["one_pass", "fused", "fused"], "split": ["one_pass"] * 3, "density_only": [None] * 3, "second_generation": ["two_passes"] * 3}
    assert n["launches"] == sum(frame_launches(I, False, c) for c in comb[which])
    want = walk_oracle(L, combustion, I)
    assert_same_bits(sim.velocity(), want["vel"], "velocity")
    for i, k in enumerate(fields):
        assert_same_bits(sim.scalar(i), want[k], k)
    sim.close()


# ------------------------------------------------------------------------------------------------------------------
# D. the fused combustion update with vorticity confinement
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scale,factor_scale", [(0.8, 1.0), (1.3, 2.9)])
def test_fused_combustion_with_vorticity_matches_oracle(scale, factor_scale):
    w = synth.random_leaves(60, 5, 13, cfl=1.8, S=1)
    fields = dict(density=w.scalars[0], **combustion_fields(w.num_voxels, seed=17))
    params = list(PARAMS6)
    params[4], params[5] = scale, factor_scale
    vel, want = w.velocity, fields
    ix = O.OracleIndex(w.coords)
    for _ in range(3):
        vel, want = ix.compute_sim(vel, want, 5, w.dt, w.voxel_size, np.asarray(params, np.float32))
    counts = {}
    for fused in (True, False):
        sim = _simulation(w.origins, w.voxel_size, w.velocity, fields, True, params)
        with schedule(True, fused), counting() as n:
            for _ in range(3):
                sim.step(5, w.dt)
            sim.sync()
        counts[fused] = n
        assert_same_bits(sim.velocity(), vel, f"fused={fused}: velocity")
        for i, k in enumerate(fields):
            assert_same_bits(sim.scalar(i), want[k], f"fused={fused}: {k}")
        sim.close()
    assert counts[True]["packed"] == counts[False]["packed"] == 1 + 2 + 2
    assert counts[False]["launches"] - counts[True]["launches"] == 2   # frames 2 and 3 ran without a combustion pass of their own


# ------------------------------------------------------------------------------------------------------------------
# E. every scalar count the state accepts
# ------------------------------------------------------------------------------------------------------------------
def _scalar_case(S):
    w = synth.random_leaves(28, 4, 7, offset=(-24, 4096 - 16, -16), cfl=1.8, S=S)
    for k, s in enumerate(w.scalars):
        s[0] = 50.0 + k       # a distinct element 0 per field (advect_scalars' inactive corners)
    return w


@pytest.mark.parametrize("S", range(1, 17))
def test_resident_frame_with_every_scalar_count_matches_oracle(S):
    """the second generation stages the scalars four at a time: S = 4, 8, 12, 16 end on a stage of three, S >= 6 takes three or more
    stages per leaf"""
    w = _scalar_case(S)
    I = 4
    sim = _simulation(w.origins, w.voxel_size, w.velocity, dict(zip(w.scalar_names, w.scalars)), False)
    with schedule(True), counting() as n:
        sim.step(I, w.dt)
        sim.sync()
    assert n["packed"] == (1 if S == 1 else 0)     # only one scalar finds all its groups packed (group 0, by the gradient pass)
    assert n["launches"] == frame_launches(I)
    want = O.OracleIndex(w.coords).frame(w.velocity, w.scalars, I, w.dt, w.voxel_size)
    got = _outputs(sim, [])
    for k in ("adv", "div", "p", "vel"):
        assert_same_bits(got[k], want[k], k)
    for i in range(S):
        assert_same_bits(sim.scalar(i), want["scalars"][i], f"scalar {i} of {S}")
    sim.close()


@pytest.mark.parametrize("others", range(1, 13))
def test_compute_sim_with_every_scalar_count_matches_oracle(others):
    w = _scalar_case(others)
    fields = dict(combustion_fields(w.num_voxels, seed=31 + others))
    for k, s in enumerate(w.scalars):
        fields[f"s{k}"] = s
    d = GridIndexedData.from_arrays(w.coords, w.velocity, "vel", **fields)
    g = H.CreateIndexGrid(d, w.voxel_size)
    with counting() as n:
        H.Compute_Sim(d, g, 5, w.dt, w.voxel_size, H.CombustionParams(*PARAMS6), False)
    assert n["packed"] == (1 if others == 1 else 0)   # density + the four combustion fields: advect_scalars on groups 0 and 1
    want_vel, want = O.OracleIndex(w.coords).compute_sim(w.velocity, fields, 5, w.dt, w.voxel_size, np.asarray(PARAMS6, np.float32))
    assert_same_bits(d.pValues(VEC3F, "vel"), want_vel, "Compute_Sim velocity")
    for k in fields:
        assert_same_bits(d.pValues(FLOAT, k), want[k], f"Compute_Sim {k} ({4 + others} fields)")


def test_more_than_16_scalars_are_refused():
    w = _scalar_case(13)
    g = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    with pytest.raises(H.HnsError, match=r"n_scalars must be in \[0, 16\]"):
        H.Simulation(g, 17)
    fields = dict(combustion_fields(w.num_voxels), **{f"s{k}": s for k, s in enumerate(w.scalars)})
    assert len(fields) == 17
    d = GridIndexedData.from_arrays(w.coords, w.velocity, "vel", **fields)
    with pytest.raises(H.HnsError, match="more than 16 float blocks"):
        H.Compute_Sim(d, H.CreateIndexGrid(d, w.voxel_size), 5, w.dt, w.voxel_size, H.CombustionParams(*PARAMS6), False)


# ------------------------------------------------------------------------------------------------------------------
# F. advect_scalar semantics on the packed group
# ------------------------------------------------------------------------------------------------------------------
def test_advect_scalar_semantics_on_the_packed_group_match_oracle():
    """subtract_gradient(True) packs group 0 with the one scalar; advect_scalars(dt, 1) then runs k_advect_scalars4<1> (inactive
    corners read 0, not element 0), and its flagged leaves the cold kernel"""
    w, fields = walk_case(90)
    s0 = fields["density"].copy()
    s0[0] = 100.0
    sim = H.Simulation(H.create_index_grid_from_origins(w.origins, w.voxel_size), 1)
    sim.upload(w.velocity, [s0])
    with schedule(True), counting() as n:
        sim.advect_velocity(w.dt)
        sim.divergence(True)
        sim.pressure_solve(4, H.launchers.omega_compute(w.voxel_size))
        sim.subtract_gradient(True)
        sim.sync()
    assert n["packed"] == 0       # the uploaded velocity has no group 0
    projected = sim.velocity()
    with schedule(True), counting() as n:
        sim.advect_scalars(w.dt, 1)
        sim.sync()
    assert n["packed"] == 1 and n["launches"] == 2
    ix = O.OracleIndex(w.coords)
    want = ix.advect_scalar(projected, s0, w.dt, w.voxel_size)
    assert_same_bits(sim.scalar(0), want, "advect_scalar on group 0")
    assert not np.array_equal(want, ix.advect_scalars(projected, [s0], w.dt, w.voxel_size)[0])   # the two semantics differ here
    sim.close()
