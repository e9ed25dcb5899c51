"""GPU parity tests: the CUDA path, called through the C ABI (hnanosolver_b200.launchers -> ctypes -> libhns_b200.so), against
(1) the CPU oracle, (2) the committed golden fixtures, (3) the unmodified reference kernels / launchers: live on the same GPU when
their build (oracle/_ref/libhns_ref.so) is present, else what they computed on the same inputs (tests/golden/ref_recorded.npz), and
(4) size-independent properties at full size.

Bar (north star): index topology bit-exact; fields within 1e-5 relative (helpers.REL_TOL) of the reference kernels.
"""
import os

import numpy as np
import pytest

import hnanosolver_b200 as H
from helpers import GOLDEN, RECORDED, Golden, Reference, assert_close, combustion_fields, nanovdb_compare_mask, rel_err
from hnanosolver_b200 import synth
from hnanosolver_b200.grid_data import FLOAT, VEC3F, GridIndexedData
from oracle import oracle as O

pytestmark = pytest.mark.gpu
PARAMS6 = np.array([0.5, 2.0, 1.5, 0.1, 0.0, 1.0], np.float32)


@pytest.fixture(scope="module", autouse=True)
def _save_recording():
    yield
    if RECORDED.recording:
        RECORDED.save()


def _copies(rd):
    return {k: v.copy() for k, v in rd.blocks.items()}


def _masked_nanovdb(buf):
    """voxelsToGrid's buffer with the bytes it leaves uninitialised zeroed (helpers.nanovdb_compare_mask)"""
    T = int(np.frombuffer(buf[672 + 40:672 + 44].tobytes(), np.uint32)[0])
    return np.where(nanovdb_compare_mask(buf.size, T), buf, 0).astype(np.uint8)


def small_cases():
    return {
        "soup_negative_multitile": synth.random_leaves(28, 4, 7, offset=(-24, 4096 - 16, -16), cfl=1.8, S=2),
        "soup_dense": synth.random_leaves(60, 4, 9, cfl=1.2, S=3),
        "single_leaf": synth.random_leaves(1, 1, 1, S=1),
        "sphere32": synth.smoke_sphere(32, 1),
    }


@pytest.fixture(scope="module", params=list(small_cases()))
def case(request):
    return small_cases()[request.param]


def run_product_frame(w, iterations, flags=0):
    g = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    sim = H.Simulation(g, len(w.scalars))
    sim.upload(w.velocity, w.scalars)
    sim.step(iterations, w.dt, flags)
    sim.sync()
    return dict(vel=sim.velocity(), div=sim.aux(0), p=sim.aux(1), adv=sim.aux(2), scalars=[sim.scalar(i) for i in range(len(w.scalars))])


# ------------------------------------------------------------------------------------------------------------------
# topology
# ------------------------------------------------------------------------------------------------------------------
def test_index_grid_matches_oracle_bit_exact(case):
    w = case
    data = GridIndexedData.from_arrays(w.coords)
    g = H.CreateIndexGrid(data, w.voxel_size, validate=True)
    ix = O.OracleIndex(w.coords)
    assert g.num_leaves == ix.num_leaves == w.num_leaves
    assert np.array_equal(g.nanovdb_buffer(), ix.nanovdb_buffer(w.voxel_size))
    rng = np.random.default_rng(0)
    q = np.concatenate([w.coords, w.coords[::3] + rng.integers(-17, 18, size=w.coords[::3].shape).astype(np.int32),
                        rng.integers(-9000, 9000, size=(2000, 3)).astype(np.int32)])
    assert np.array_equal(g.get_values(q), ix.get_values(q))
    assert np.array_equal(g.get_values(w.coords), np.arange(1, w.num_voxels + 1, dtype=np.uint64))


def test_index_grid_matches_reference_voxelsToGrid(case):
    w = case
    g = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    rng = np.random.default_rng(1)
    q = np.concatenate([w.coords[::2], w.coords[::3] + rng.integers(-12, 13, size=w.coords[::3].shape).astype(np.int32)])

    def live():
        rg = O.RefGrid(O.RefData(w.coords), w.voxel_size)
        return dict(nanovdb=_masked_nanovdb(rg.buffer()), values=rg.get_values(q))

    ref = Reference(f"index_grid/{w.name}", live, [w.coords, q])
    ref.check(_masked_nanovdb(g.nanovdb_buffer()), "nanovdb", "NanoVDB buffer vs voxelsToGrid")
    ref.check(g.get_values(q), "values", "getValue")


def test_neighbor_table(case):
    w = case
    g = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    nbr = g.neighbors()
    lut = {tuple(o): i for i, o in enumerate(w.origins.tolist())}
    for l, o in enumerate(w.origins.tolist()):
        for dx in (-1, 0, 1):
            for dy in (-1, 0, 1):
                for dz in (-1, 0, 1):
                    want = lut.get((o[0] + 8 * dx, o[1] + 8 * dy, o[2] + 8 * dz), -1)
                    assert nbr[l, (dx + 1) * 9 + (dy + 1) * 3 + dz + 1] == want


def test_topology_errors():
    w = synth.random_leaves(10, 3, 2)
    with pytest.raises(H.HnsError, match="NanoVDB order"):
        H.create_index_grid_from_origins(w.origins[::-1].copy(), 0.1)
    with pytest.raises(H.HnsError, match="multiple of 8"):
        H.create_index_grid_from_origins(w.origins + 1, 0.1)
    with pytest.raises(ValueError, match="voxelSize"):
        H.create_index_grid_from_origins(w.origins, 0.0)
    bad = GridIndexedData.from_arrays(w.coords[:-1])
    with pytest.raises(H.HnsError, match="multiple of 512"):
        H.CreateIndexGrid(bad, 0.1)
    c = w.coords.copy()
    c[700] += 1
    with pytest.raises(H.HnsError, match="not a dense leaf"):
        H.CreateIndexGrid(GridIndexedData.from_arrays(c), 0.1, validate=True)
    empty = H.create_index_grid_from_origins(np.zeros((0, 3), np.int32), 0.1)
    assert empty.num_leaves == 0 and empty.nanovdb_buffer().size == 672 + 64 + 96


# ------------------------------------------------------------------------------------------------------------------
# kernels, stage by stage
# ------------------------------------------------------------------------------------------------------------------
def test_frame_stages_match_oracle(case):
    w = case
    I = 6
    ix = O.OracleIndex(w.coords)
    want = ix.frame(w.velocity, w.scalars, I, w.dt, w.voxel_size)
    got = run_product_frame(w, I)
    for k in ("adv", "div", "p", "vel"):
        assert_close(got[k], want[k], k)
    for i in range(len(w.scalars)):
        assert_close(got["scalars"][i], want["scalars"][i], f"scalar {i}")


def test_sweep_direction_does_not_change_the_bits(case):
    """Black half-sweeps walk the leaves back to front for L2 reuse; a half-sweep has no intra-colour dependencies, so the
    traversal order must not change a single bit."""
    a = run_product_frame(case, 7, flags=0)
    b = run_product_frame(case, 7, flags=H.Simulation.FLAG_FORWARD_ONLY)
    for k in ("p", "vel"):
        assert np.array_equal(a[k], b[k]), k


def _ref_frame(w, iterations):
    """the reference's north-star frame on its own kernels: adv, div, p, vel, scalar{i} and the divergence norm of vel"""
    rd = O.RefData(w.coords)
    rd.add_vec3("vel", w.velocity)
    for n, a in zip(w.scalar_names, w.scalars):
        rd.add_float(n, a)
    rg = O.RefGrid(rd, w.voxel_size)
    rf = O.RefFrame(rd, rg, w.scalar_names)
    rf.run(iterations, w.dt, w.voxel_size, 1)
    want = rf.download()
    want.update({f"scalar{i}": s for i, s in enumerate(want.pop("scalars"))}, div_norm=_div_norm(w, want["vel"]))
    return want


def _div_norm(w, vel):
    return np.array([np.sqrt(np.mean(O.OracleIndex(w.coords).divergence(vel, w.voxel_size).astype(np.float64) ** 2))])


def test_frame_stages_match_reference_kernels(case):
    w = case
    I = 9
    got = run_product_frame(w, I)
    ref = Reference(f"frame/{w.name}", lambda: _ref_frame(w, I), [w.coords, w.velocity, *w.scalars])
    for k in ("adv", "div", "p", "vel"):
        ref.check(got[k], k, k)
    for i in range(len(w.scalars)):
        ref.check(got["scalars"][i], f"scalar{i}", f"scalar {i}")
    # divergence L2 norm of the projected velocity agrees with the reference's (BASELINE.md parity gate)
    ref.check(_div_norm(w, got["vel"]), "div_norm", "||div u|| of the projected velocity")


def test_far_samples_take_the_tree_walk_path():
    """CFL ~ 20: back-traced points land several leaves away, outside the 3x3x3 neighbour table."""
    w = synth.random_leaves(50, 5, 4, cfl=20.0, S=1)
    ix = O.OracleIndex(w.coords)
    g = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    sim = H.Simulation(g, 1)
    sim.upload(w.velocity, w.scalars)
    sim.advect_velocity(w.dt)
    sim.advect_scalars(w.dt, 0)
    sim.sync()
    assert_close(sim.aux(2), ix.advect_vector(w.velocity, w.dt, w.voxel_size), "advect_vector, CFL 20")
    assert_close(sim.scalar(0), ix.advect_scalars(w.velocity, w.scalars, w.dt, w.voxel_size)[0], "advect_scalars, CFL 20")
    sim.upload(w.velocity, w.scalars)
    sim.advect_scalars(w.dt, 1)
    sim.sync()
    assert_close(sim.scalar(0), ix.advect_scalar(w.velocity, w.scalars[0], w.dt, w.voxel_size), "advect_scalar, CFL 20")


def test_inactive_corner_semantics_differ_between_the_two_scalar_kernels():
    """advect_scalars reads array element 0 for inactive corners (Kernel.cu:192), advect_scalar reads 0 (Stencils.hpp:83)."""
    w = synth.random_leaves(6, 3, 5, cfl=1.5, S=1)
    w.scalars[0][0] = 100.0  # make element 0 stand out
    ix = O.OracleIndex(w.coords)
    g = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    outs = []
    for sem in (0, 1):
        sim = H.Simulation(g, 1)
        sim.upload(w.velocity, w.scalars)
        sim.advect_scalars(w.dt, sem)
        sim.sync()
        outs.append(sim.scalar(0))
    assert_close(outs[0], ix.advect_scalars(w.velocity, w.scalars, w.dt, w.voxel_size)[0], "advect_scalars semantics")
    assert_close(outs[1], ix.advect_scalar(w.velocity, w.scalars[0], w.dt, w.voxel_size), "advect_scalar semantics")
    assert not np.array_equal(outs[0], outs[1])


# ------------------------------------------------------------------------------------------------------------------
# the drop-in launchers on host sidecars
# ------------------------------------------------------------------------------------------------------------------
def _sidecar(w, floats):
    return GridIndexedData.from_arrays(w.coords, w.velocity, "vel", **floats)


def test_launchers_match_oracle(case):
    w = case
    ix = O.OracleIndex(w.coords)
    h, dt = w.voxel_size, w.dt
    d = _sidecar(w, dict(zip(w.scalar_names, w.scalars)))
    H.AdvectIndexGrid(d, dt, h)
    for n, s in zip(w.scalar_names, w.scalars):
        assert_close(d.pValues(FLOAT, n), ix.advect_scalar(w.velocity, s, dt, h), f"AdvectIndexGrid {n}")
    d = _sidecar(w, {})
    H.AdvectIndexGridVelocity(d, dt, h)
    assert_close(d.pValues(VEC3F, "vel"), ix.advect_vector(w.velocity, dt, h), "AdvectIndexGridVelocity")
    d = _sidecar(w, dict(divergence=np.zeros(w.num_voxels, np.float32)))
    H.Divergence(d, h)
    assert_close(d.pValues(FLOAT, "divergence"), ix.divergence(w.velocity, h), "Divergence")
    d = _sidecar(w, {})
    H.ProjectNonDivergent(d, 5, h)
    assert_close(d.pValues(VEC3F, "vel"), ix.project_non_divergent(w.velocity, 5, h)[0], "ProjectNonDivergent")


def test_compute_sim_matches_oracle(case):
    w = case
    ix = O.OracleIndex(w.coords)
    fields = dict(density=w.scalars[0], **combustion_fields(w.num_voxels))
    want_vel, want = ix.compute_sim(w.velocity, fields, 5, w.dt, w.voxel_size, PARAMS6)
    d = _sidecar(w, fields)
    g = H.CreateIndexGrid(d, w.voxel_size)
    H.Compute_Sim(d, g, 5, w.dt, w.voxel_size, H.CombustionParams(*PARAMS6.tolist()), False)
    assert_close(d.pValues(VEC3F, "vel"), want_vel, "Compute_Sim velocity")
    for k, v in want.items():
        assert_close(d.pValues(FLOAT, k), v, f"Compute_Sim {k}")


@pytest.mark.parametrize("order", [["density", "fuel", "waste", "temperature", "flame"], ["flame", "temperature", "density", "waste", "fuel"]])
def test_compute_sim_equals_the_resident_frame_bitwise(case, order):
    """Compute_Sim feeds the frame while its inputs are still crossing PCIe: the term combustion adds to the divergence goes in as soon
    as fuel and waste have landed, the buoyancy force is applied from fuel, waste and temperature after the solve, the field updates
    follow behind the gradient pass (api.cu::frame, FrameDeps). The resident frame runs the reference's step order on fields that are
    all there. Independent steps in another order: every bit must agree, whatever the order of the float blocks."""
    w = case
    comb = combustion_fields(w.num_voxels)
    fields = {k: (w.scalars[0] if k == "density" else comb[k]) for k in order}
    d = _sidecar(w, {k: v.copy() for k, v in fields.items()})
    g = H.CreateIndexGrid(d, w.voxel_size)
    H.Compute_Sim(d, g, 7, w.dt, w.voxel_size, H.CombustionParams(*PARAMS6.tolist()), False)
    grid = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    sim = H.Simulation(grid, len(order))
    sim.upload(w.velocity, [fields[k] for k in order])
    sim.set_combustion(True, order.index("fuel"), order.index("waste"), order.index("temperature"), order.index("flame"),
                       H.CombustionParams(*PARAMS6.tolist()))
    sim.step(7, w.dt)
    sim.sync()
    assert np.array_equal(d.pValues(VEC3F, "vel").reshape(-1, 3), sim.velocity().reshape(-1, 3))
    for i, k in enumerate(order):
        assert np.array_equal(d.pValues(FLOAT, k), sim.scalar(i)), k


def _ref_compute_sim(w, fields, iterations, params, has_collision=False):
    """the reference's CreateIndexGrid + Compute_Sim on a copy of the sidecar: every block afterwards"""
    rd = O.RefData(w.coords)
    rd.add_vec3("vel", w.velocity)
    for k, v in fields.items():
        rd.add_float(k, v)
    rg = O.RefGrid(rd, w.voxel_size)
    O.ref_compute_sim(rd, rg, iterations, w.dt, w.voxel_size, params, has_collision)
    return _copies(rd)


def test_compute_sim_matches_reference_compute_sim(case):
    w = case
    fields = dict(density=w.scalars[0], **combustion_fields(w.num_voxels))
    d = _sidecar(w, fields)
    g = H.CreateIndexGrid(d, w.voxel_size)
    H.Compute_Sim(d, g, 8, w.dt, w.voxel_size, H.CombustionParams(*PARAMS6.tolist()), False)
    ref = Reference(f"compute_sim/{w.name}", lambda: _ref_compute_sim(w, fields, 8, PARAMS6), [w.coords, w.velocity, *fields.values()])
    ref.check(d.pValues(VEC3F, "vel"), "vel", "Compute_Sim velocity")
    for k in fields:
        ref.check(d.pValues(FLOAT, k), k, f"Compute_Sim {k}")


# ------------------------------------------------------------------------------------------------------------------
# vorticity confinement (SURVEY.md 8f rank 1): out-of-place evaluation of the reference kernel
# ------------------------------------------------------------------------------------------------------------------
VORTICITY_CASES = [(1.0, 1.0), (0.7, 2.9), (1.3, -1.0), (1.0, 7.0), (0.5, 8.0), (1.0, 9.5)]  # (scale, factorScale); 9.5 -> offset 9: far path


def _product_vorticity(w, scale, factor_scale):
    g = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    sim = H.Simulation(g, len(w.scalars))
    sim.upload(w.velocity, w.scalars)
    sim.advect_velocity(0.0)          # dt = 0: the advected velocity is the input velocity (BFECC of a zero displacement is exact)
    before = sim.aux(H.Simulation.AUX_ADVECTED)
    sim.vorticity_confinement(w.dt, scale, factor_scale)
    sim.sync()
    return before, sim.aux(H.Simulation.AUX_ADVECTED)


@pytest.mark.parametrize("scale,factor_scale", VORTICITY_CASES)
def test_vorticity_confinement_matches_oracle(case, scale, factor_scale):
    w = case
    before, got = _product_vorticity(w, scale, factor_scale)
    assert np.array_equal(before, w.velocity)
    want = O.OracleIndex(w.coords).vorticity_confinement(w.velocity, w.dt, w.voxel_size, scale, factor_scale)
    assert np.array_equal(got, want), f"max |diff| {np.abs(got - want).max()}"
    assert not np.array_equal(got, w.velocity) or w.num_leaves == 1


@pytest.mark.parametrize("scale,factor_scale", VORTICITY_CASES[:4])
def test_vorticity_confinement_matches_reference_kernel_out_of_place(case, scale, factor_scale):
    """The reference kernel itself, given separate input and output buffers (Compute() passes the same buffer twice and races)."""
    w = case

    def live():
        rd = O.RefData(w.coords)
        rd.add_vec3("vel", w.velocity)
        for n, a in zip(w.scalar_names, w.scalars):
            rd.add_float(n, a)
        rg = O.RefGrid(rd, w.voxel_size)
        return dict(vel=O.RefFrame(rd, rg, w.scalar_names).vorticity(w.dt, w.voxel_size, scale, factor_scale))

    _, got = _product_vorticity(w, scale, factor_scale)
    ref = Reference(f"vorticity/{w.name}/{scale}/{factor_scale}", live, [w.coords, w.velocity, *w.scalars])
    ref.check(got, "vel", "vorticityConfinement")


def test_vorticity_identity_cases(case):
    """scale 0, or a factorScale below 1 (the SOP default 0.5 truncates to a zero offset): the force is exactly zero"""
    w = case
    for scale, fs in ((0.0, 3.0), (1.0, 0.5), (2.0, -0.9)):
        _, got = _product_vorticity(w, scale, fs)
        assert np.array_equal(got, w.velocity)
        want = O.OracleIndex(w.coords).vorticity_confinement(w.velocity, w.dt, w.voxel_size, scale, fs)
        assert np.array_equal(want, w.velocity)


def test_compute_sim_with_vorticity_matches_oracle(case):
    w = case
    params = PARAMS6.copy()
    params[4], params[5] = 0.8, 1.0
    ix = O.OracleIndex(w.coords)
    fields = dict(density=w.scalars[0], **combustion_fields(w.num_voxels))
    want_vel, want = ix.compute_sim(w.velocity, fields, 5, w.dt, w.voxel_size, params)
    off_vel, _ = ix.compute_sim(w.velocity, fields, 5, w.dt, w.voxel_size, PARAMS6)
    d = _sidecar(w, fields)
    g = H.CreateIndexGrid(d, w.voxel_size)
    H.Compute_Sim(d, g, 5, w.dt, w.voxel_size, H.CombustionParams(*params.tolist()), False)
    assert_close(d.pValues(VEC3F, "vel"), want_vel, "Compute_Sim velocity (vorticity on)")
    for k, v in want.items():
        assert_close(d.pValues(FLOAT, k), v, f"Compute_Sim {k} (vorticity on)")
    if w.num_leaves > 1:
        assert not np.array_equal(want_vel, off_vel)


def test_compute_sim_default_sop_vorticity_parameters_match_reference(case):
    """SOP defaults: vorticity 1, factor_scale 0.5 (SOP_HNanoSolver.cpp:73-86). The offset truncates to 0, the in-place race of the
    reference is then harmless, and both sides must agree."""
    w = case
    params = PARAMS6.copy()
    params[4], params[5] = 1.0, 0.5
    fields = dict(density=w.scalars[0], **combustion_fields(w.num_voxels))
    d = _sidecar(w, fields)
    g = H.CreateIndexGrid(d, w.voxel_size)
    H.Compute_Sim(d, g, 6, w.dt, w.voxel_size, H.CombustionParams(*params.tolist()), False)
    ref = Reference(f"compute_sim_sop_default/{w.name}", lambda: _ref_compute_sim(w, fields, 6, params), [w.coords, w.velocity, *fields.values()])
    ref.check(d.pValues(VEC3F, "vel"), "vel", "Compute_Sim velocity")
    for k in fields:
        ref.check(d.pValues(FLOAT, k), k, f"Compute_Sim {k}")


# ------------------------------------------------------------------------------------------------------------------
# SDF collision path (SURVEY.md 8f rank 2)
# ------------------------------------------------------------------------------------------------------------------
def _collision_sdf(w):
    c = w.coords.astype(np.float32)
    centre = np.round(c.mean(0))
    sdf = (0.05 * (np.sqrt(((c - centre) ** 2).sum(1)) - 6.0)).astype(np.float32)
    sdf[0] = 0.0
    return sdf


def _collision_sim(w, sdf):
    g = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    sim = H.Simulation(g, len(w.scalars) + 1)
    sim.upload(w.velocity, list(w.scalars) + [sdf])
    sim.set_collision(len(w.scalars))
    return sim


def test_collision_kernels_match_oracle(case):
    w = case
    sdf = _collision_sdf(w)
    ix = O.OracleIndex(w.coords)
    sim = _collision_sim(w, sdf)
    sim.enforce_collision()
    sim.sync()
    v1 = ix.collision_boundary(w.velocity, sdf, w.voxel_size, ix.SITE_ENFORCE)
    assert np.array_equal(sim.velocity(), v1), "enforceCollisionBoundaries"
    sim.advect_velocity(w.dt)
    sim.sync()
    adv = ix.advect_vector_sdf(v1, sdf, w.dt, w.voxel_size)
    assert np.array_equal(sim.aux(H.Simulation.AUX_ADVECTED), adv), "advect_vector(hasCollision)"
    sim.divergence(True)
    sim.pressure_solve(4, H.launchers.omega_compute(w.voxel_size))
    sim.subtract_gradient(True)
    sim.sync()
    div = ix.divergence(adv, w.voxel_size)
    p = ix.rbgs(div, np.zeros(w.num_voxels, np.float32), w.voxel_size, 4, O.omega_compute(w.voxel_size))
    proj = ix.collision_boundary(ix.subtract_gradient(adv, p, w.voxel_size), sdf, w.voxel_size, ix.SITE_GRADIENT)
    assert np.array_equal(sim.velocity(), proj), "subtractPressureGradient(hasCollision)"
    sim.advect_scalars(w.dt, 0)
    sim.sync()
    want = ix.advect_scalars_sdf(proj, w.scalars, sdf, w.dt, w.voxel_size)
    for i in range(len(w.scalars)):
        assert np.array_equal(sim.scalar(i), want[i]), f"advect_scalars(hasCollision)[{i}]"
    assert np.array_equal(sim.scalar(len(w.scalars)), sdf), "the SDF itself is not advected"


def _compute_sim_collision(w, has_collision, iterations=5):
    fields = dict(density=w.scalars[0], **combustion_fields(w.num_voxels), collision_sdf=_collision_sdf(w))
    d = _sidecar(w, fields)
    g = H.CreateIndexGrid(d, w.voxel_size)
    H.Compute_Sim(d, g, iterations, w.dt, w.voxel_size, H.CombustionParams(*PARAMS6.tolist()), has_collision)
    return fields, d


def test_compute_sim_with_collision_matches_oracle(case):
    w = case
    fields, d = _compute_sim_collision(w, True)
    ix = O.OracleIndex(w.coords)
    want_vel, want = ix.compute_sim(w.velocity, fields, 5, w.dt, w.voxel_size, PARAMS6, has_collision=True)
    assert_close(d.pValues(VEC3F, "vel"), want_vel, "Compute_Sim(hasCollision) velocity")
    for k, v in want.items():
        assert_close(d.pValues(FLOAT, k), v, f"Compute_Sim(hasCollision) {k}")
    assert not d.pValues(FLOAT, "collision_sdf").any()
    # hasCollision = false with the block present: carried, zeroed, no other effect
    fields0, d0 = _compute_sim_collision(w, False)
    want_vel0, _ = ix.compute_sim(w.velocity, {k: v for k, v in fields0.items() if k != "collision_sdf"}, 5, w.dt, w.voxel_size, PARAMS6)
    assert_close(d0.pValues(VEC3F, "vel"), want_vel0, "Compute_Sim velocity, collision_sdf present but hasCollision false")
    assert not d0.pValues(FLOAT, "collision_sdf").any()


def test_compute_sim_with_collision_matches_reference(case):
    w = case
    fields, d = _compute_sim_collision(w, True, iterations=7)
    ref = Reference(f"compute_sim_collision/{w.name}", lambda: _ref_compute_sim(w, fields, 7, PARAMS6, True),
                    [w.coords, w.velocity, *fields.values()])
    ref.check(d.pValues(VEC3F, "vel"), "vel", "Compute_Sim(hasCollision) velocity")
    for k in fields:
        if k != "collision_sdf":
            ref.check(d.pValues(FLOAT, k), k, f"Compute_Sim(hasCollision) {k}")


@pytest.mark.parametrize("name", ["soup", "sphere"])
def test_collision_against_golden_reference_outputs(name):
    path = os.path.join(GOLDEN, f"ref_{name}.npz")
    if not os.path.exists(path):
        pytest.skip("no golden fixture")
    z = Golden(name)
    if "collision_sdf" not in z:
        pytest.skip("fixture predates the collision vectors")
    origins, h, dt, I = z["origins"], float(z["voxel_size"]), float(z["dt"]), int(z["iterations"])
    S = len(z["scalar_names"])
    g = H.create_index_grid_from_origins(origins, h)
    sim = H.Simulation(g, S + 1)
    sim.upload(z["velocity"], [z[f"scalar{i}"] for i in range(S)] + [z["collision_sdf"]])
    sim.set_collision(S)
    sim.enforce_collision()
    sim.sync()
    z.check(sim.velocity(), "coll_enforce", "enforceCollisionBoundaries")
    sim.upload(z["velocity"], [z[f"scalar{i}"] for i in range(S)] + [z["collision_sdf"]])
    sim.advect_velocity(dt)
    sim.sync()
    z.check(sim.aux(H.Simulation.AUX_ADVECTED), "coll_advect_vector", "advect_vector(hasCollision)")
    # all-in-one node
    fields = dict(density=z["scalar0"], fuel=z["comb_fuel"], waste=z["comb_waste"], temperature=z["comb_temperature"], flame=z["comb_flame"],
                  collision_sdf=z["collision_sdf"])
    d = H.GridIndexedData()
    d.allocateCoords(len(z["coords"]))
    d.pCoords()[:] = z["coords"]
    d.addValueBlock(VEC3F, "vel")
    d.pValues(VEC3F, "vel")[:] = z["velocity"]
    for k, v in fields.items():
        d.addValueBlock(FLOAT, k)
        d.pValues(FLOAT, k)[:] = v
    gh = H.CreateIndexGrid(d, h)
    H.Compute_Sim(d, gh, I, dt, h, H.CombustionParams(*z["params"].tolist()), True)
    z.check(d.pValues(VEC3F, "vel"), "compute_sim_coll_vel", "Compute_Sim(hasCollision) velocity")
    for k in fields:
        if k != "collision_sdf":
            z.check(d.pValues(FLOAT, k), f"compute_sim_coll_{k}", k)


def test_standalone_launchers_match_reference_launchers(case):
    w = case
    h, dt = w.voxel_size, w.dt

    def live():
        rd = O.RefData(w.coords)
        rd.add_vec3("vel", w.velocity)
        for n, s in zip(w.scalar_names, w.scalars):
            rd.add_float(n, s)
        O.ref_advect_index_grid(rd, dt, h)
        out = {"advect_" + n: rd.blocks[n].copy() for n in w.scalar_names}
        rd = O.RefData(w.coords)
        rd.add_vec3("vel", w.velocity)
        O.ref_project_non_divergent(rd, 10, h)
        return dict(out, project=rd.blocks["vel"].copy())

    ref = Reference(f"launchers/{w.name}", live, [w.coords, w.velocity, *w.scalars])
    d = _sidecar(w, dict(zip(w.scalar_names, w.scalars)))
    H.AdvectIndexGrid(d, dt, h)
    for n in w.scalar_names:
        ref.check(d.pValues(FLOAT, n), "advect_" + n, f"AdvectIndexGrid {n}")
    d = _sidecar(w, {})
    H.ProjectNonDivergent(d, 10, h)
    ref.check(d.pValues(VEC3F, "vel"), "project", "ProjectNonDivergent")


def test_compute_sim_errors():
    w = synth.random_leaves(4, 2, 1, S=1)
    d = _sidecar(w, dict(density=w.scalars[0]))
    g = H.CreateIndexGrid(d, w.voxel_size)
    p = H.CombustionParams()
    with pytest.raises(RuntimeError, match="Missing required input field for combustion: fuel"):
        H.Compute_Sim(d, g, 4, w.dt, w.voxel_size, p, False)
    two = _sidecar(w, dict(density=w.scalars[0]))
    two.addValueBlock(VEC3F, "vel2")
    with pytest.raises(RuntimeError, match="exactly one Vec3f block"):
        H.Compute_Sim(two, g, 4, w.dt, w.voxel_size, p, False)
    nof = _sidecar(w, {})
    with pytest.raises(RuntimeError, match="No float blocks"):
        H.Compute_Sim(nof, g, 4, w.dt, w.voxel_size, p, False)
    empty = GridIndexedData()
    H.Compute_Sim(empty, g, 4, w.dt, w.voxel_size, p, False)  # totalVoxels == 0 -> silent return (HNanoSolver.cu:26-28)


# ------------------------------------------------------------------------------------------------------------------
# golden fixtures (outputs of the reference itself, committed)
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["soup", "sphere"])
def test_against_golden_reference_outputs(name):
    path = os.path.join(GOLDEN, f"ref_{name}.npz")
    if not os.path.exists(path):
        pytest.skip("fixture not committed")
    z = Golden(name)
    h, dt, I = float(z["voxel_size"]), float(z["dt"]), int(z["iterations"])
    g = H.create_index_grid_from_origins(z["origins"], h)
    ref = z["nanovdb"]
    T = int(np.frombuffer(ref[672 + 40:672 + 44].tobytes(), np.uint32)[0])
    assert not ((g.nanovdb_buffer() != ref) & nanovdb_compare_mask(ref.size, T)).any()
    assert np.array_equal(g.get_values(z["query_ijk"]), z["query_values"])
    S = len(z["scalar_names"])
    sim = H.Simulation(g, S)
    sim.upload(z["velocity"], [z[f"scalar{i}"] for i in range(S)])
    sim.step(I, dt)
    sim.sync()
    z.check(sim.aux(2), "frame_adv", "advect_vector")
    z.check(sim.aux(0), "frame_div", "divergence")
    z.check(sim.aux(1), "frame_p", "pressure")
    z.check(sim.velocity(), "frame_vel", "projected velocity")
    for i in range(S):
        z.check(sim.scalar(i), f"frame_scalar{i}", f"scalar {i}")
    fields = dict(density=z["scalar0"], fuel=z["comb_fuel"], waste=z["comb_waste"], temperature=z["comb_temperature"], flame=z["comb_flame"])
    d = GridIndexedData.from_arrays(z["coords"], z["velocity"], "vel", **fields)
    H.Compute_Sim(d, H.CreateIndexGrid(d, h), I, dt, h, H.CombustionParams(*z["params"].tolist()), False)
    z.check(d.pValues(VEC3F, "vel"), "compute_sim_vel", "Compute_Sim velocity")
    for k in fields:
        z.check(d.pValues(FLOAT, k), f"compute_sim_{k}", f"Compute_Sim {k}")


# ------------------------------------------------------------------------------------------------------------------
# full-size checks (BASELINE.json configs 2 and 4)
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def c4():
    return synth.sparse_smoke(512, 0.30, 4, with_coords=False)


def test_config2_full_frame_matches_oracle():
    w = synth.smoke_plume(128, 2)
    ix = O.OracleIndex(w.coords)
    want = ix.frame(w.velocity, w.scalars, 40, w.dt, w.voxel_size)
    got = run_product_frame(w, 40)
    for k in ("adv", "div", "p", "vel"):
        assert_close(got[k], want[k], k)
    for i in range(2):
        assert_close(got["scalars"][i], want["scalars"][i], f"scalar {i}")


def test_config4_full_frame_matches_reference_kernels(c4):
    w = c4

    def live():
        rd = O.RefData(synth.dense_coords(w.origins))
        rd.add_vec3("vel", w.velocity)
        for n, a in zip(w.scalar_names, w.scalars):
            rd.add_float(n, a)
        rg = O.RefGrid(rd, w.voxel_size)
        rf = O.RefFrame(rd, rg, w.scalar_names)
        rf.run(40, w.dt, w.voxel_size, 1)
        want = rf.download()
        return dict(want, **{f"scalar{i}": s for i, s in enumerate(want.pop("scalars"))})

    got = run_product_frame(w, 40)
    ref = Reference(f"frame/{w.name}", live, [w.origins, w.velocity, *w.scalars])
    for k in ("adv", "div", "p", "vel"):
        ref.check(got[k], k, k)
    for i in range(2):
        ref.check(got["scalars"][i], f"scalar{i}", f"scalar {i}")


def test_config4_all_in_one_frame_matches_reference_compute_sim(c4):
    """What bench.py times: the FULL HNanoSolver frame (combustion + buoyancy, S = 5 float blocks, I = 40) on the 512^3 sparse smoke,
    through the launcher pair CreateIndexGrid + Compute_Sim, against the unmodified reference's own CreateIndexGrid + Compute_Sim on
    the same GPU."""
    w = c4
    fields = dict(density=w.scalars[0], **synth.combustion_fields(w))
    coords = synth.dense_coords(w.origins)

    def live():
        rd = O.RefData(coords)
        rd.add_vec3("vel", w.velocity)
        for k, v in fields.items():
            rd.add_float(k, v)
        O.ref_cook_frame(rd, 40, w.dt, w.voxel_size, PARAMS6)
        return _copies(rd)

    ref = Reference(f"cook/{w.name}", live, [coords, w.velocity, *fields.values()])
    d = GridIndexedData.from_arrays(coords, w.velocity.copy(), "vel", **{k: v.copy() for k, v in fields.items()})
    g = H.CreateIndexGrid(d, w.voxel_size)
    H.Compute_Sim(d, g, 40, w.dt, w.voxel_size, H.CombustionParams(*PARAMS6.tolist()), False)
    ref.check(d.pValues(VEC3F, "vel"), "vel", "Compute_Sim velocity")
    for k in fields:
        ref.check(d.pValues(FLOAT, k), k, f"Compute_Sim {k}")


def test_config1_reference_host_path_case():
    """BASELINE.json config 1 at its stated size: 64^3 smoke sphere, one density advection (the stand-alone advect_scalar semantics of
    AdvectIndexGrid) + one divergence, against the oracle and -- when present -- the reference's own launchers."""
    w = synth.WORKLOADS["c1"]()
    assert w.origins.max() + 8 <= 64 + 16
    ix = O.OracleIndex(w.coords)
    d = GridIndexedData.from_arrays(w.coords, w.velocity.copy(), "vel", density=w.scalars[0].copy(), divergence=np.zeros(w.num_voxels, np.float32))
    H.Divergence(d, w.voxel_size)
    assert_close(d.pValues(FLOAT, "divergence"), ix.divergence(w.velocity, w.voxel_size), "divergence")
    d2 = GridIndexedData.from_arrays(w.coords, w.velocity.copy(), "vel", density=w.scalars[0].copy())
    H.AdvectIndexGrid(d2, w.dt, w.voxel_size)
    assert_close(d2.pValues(FLOAT, "density"), ix.advect_scalar(w.velocity, w.scalars[0], w.dt, w.voxel_size), "advect_scalar")
    if O.ref_gpu_available():
        rd = O.RefData(w.coords)
        rd.add_vec3("vel", w.velocity)
        rd.add_float("density", w.scalars[0])
        O.ref_advect_index_grid(rd, w.dt, w.voxel_size)
        assert_close(d2.pValues(FLOAT, "density"), rd.blocks["density"], "AdvectIndexGrid vs the reference launcher")
        rd = O.RefData(w.coords)
        rd.add_vec3("vel", w.velocity)
        rd.add_float("divergence", np.zeros(w.num_voxels, np.float32))
        O.ref_divergence(rd, w.voxel_size)
        assert_close(d.pValues(FLOAT, "divergence"), rd.blocks["divergence"], "Divergence vs the reference launcher")


def test_config4_size_independent_properties(c4):
    w = c4
    g = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    sim = H.Simulation(g, 2)
    # (1) alternating and forward-only sweep orders give the same bits at full size
    sim.upload(w.velocity, w.scalars)
    sim.step(10, w.dt, 0)
    sim.sync()
    p_f, v_f = sim.aux(1), sim.velocity()
    sim.upload(w.velocity, w.scalars)
    sim.step(10, w.dt, H.Simulation.FLAG_FORWARD_ONLY)
    sim.sync()
    assert np.array_equal(p_f, sim.aux(1)) and np.array_equal(v_f, sim.velocity())
    # (2) linearity of the pressure solve and projection in the velocity: scaling by 2 is exact in binary floating point
    sim.upload(w.velocity, w.scalars)
    sim.divergence(of_advected=False)
    sim.pressure_solve(5, 1.5)
    sim.sync()
    p1 = sim.aux(1)
    sim.upload(2 * w.velocity, w.scalars)
    sim.divergence(of_advected=False)
    sim.pressure_solve(5, 1.5)
    sim.sync()
    assert np.array_equal(sim.aux(1), 2 * p1)
    # (3) zero velocity: BFECC advection is the identity (back-trace lands on the voxel, weights (1,0,..,0))
    sim.upload(np.zeros_like(w.velocity), w.scalars)
    sim.advect_scalars(w.dt, 0)
    sim.sync()
    assert np.array_equal(sim.scalar(0), w.scalars[0]) and np.array_equal(sim.scalar(1), w.scalars[1])
    # (4) a constant velocity field has zero divergence wherever all six neighbours exist; host round trip is lossless
    const = np.tile(np.array([0.3, -1.1, 0.7], np.float32), (w.num_voxels, 1))
    sim.upload(const, w.scalars)
    assert np.array_equal(sim.velocity(), const)
    sim.divergence(of_advected=False)
    sim.sync()
    div = sim.aux(0).reshape(-1, 8, 8, 8)
    assert np.abs(div[:, 1:7, 1:7, 1:7]).max() == 0.0


def _three_frames(w, fields, comb, packed, iterations=6):
    """three consecutive resident frames; returns every field and how many third-generation advection launches they took"""
    from hnanosolver_b200 import _lib

    lib = _lib.lib()
    names = list(fields)
    g = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    sim = H.Simulation(g, len(names))
    sim.upload(w.velocity, list(fields.values()))
    if comb:
        sim.set_combustion(True, names.index("fuel"), names.index("waste"), names.index("temperature"), names.index("flame"),
                           H.CombustionParams(*PARAMS6.tolist()))
    prev = lib.hns_set_packed_advection(int(packed))
    try:
        before = lib.hns_packed_advection_launches()
        for _ in range(3):
            sim.step(iterations, w.dt)
        sim.sync()
        used = lib.hns_packed_advection_launches() - before
    finally:
        lib.hns_set_packed_advection(prev)
    out = dict(vel=sim.velocity(), div=sim.aux(0), p=sim.aux(1), adv=sim.aux(2))
    out.update({k: sim.scalar(i) for i, k in enumerate(names)})
    return out, used


@pytest.mark.parametrize("layout", ["density_first", "density_last", "density_only", "two_scalars"])
def test_packed_advection_is_bit_identical_over_consecutive_frames(layout):
    """The third-generation advection kernels stage from float4 groups that the gradient and combustion passes write (advect.cu): same
    bits as the second generation on the brick fields, frame after frame, and the packed kernels really are the ones that ran --
    advect_scalars in every frame, advect_vector from the second frame on (the first one finds no group yet). `two_scalars` has no
    producer for its second group and must stay on the second generation."""
    w = synth.random_leaves(60, 4, 9, cfl=1.2, S=2)
    comb = combustion_fields(w.num_voxels)
    fields, with_comb, expect = {
        "density_first": (dict(density=w.scalars[0], **comb), True, 5),
        "density_last": (dict(**comb, density=w.scalars[0]), True, 5),
        "density_only": (dict(density=w.scalars[0]), False, 5),
        "two_scalars": (dict(density=w.scalars[0], temperature=w.scalars[1]), False, 2),   # advect_vector only, frames 2 and 3
    }[layout]
    got, used = _three_frames(w, fields, with_comb, True)
    want, used_off = _three_frames(w, fields, with_comb, False)
    assert used == expect and used_off == 0
    for k in want:
        assert np.array_equal(got[k], want[k]), k


def test_packed_advection_far_samples_still_take_the_tree_walk_path():
    """a CFL far beyond the staged region: the packed kernels flag the leaves and the generic pass redoes them, as before"""
    w = synth.random_leaves(40, 3, 5, cfl=9.0, S=1)
    fields = dict(density=w.scalars[0])
    got, used = _three_frames(w, fields, False, True, iterations=3)
    want, _ = _three_frames(w, fields, False, False, iterations=3)
    assert used == 5
    for k in want:
        assert np.array_equal(got[k], want[k]), k


def test_every_launch_is_counted():
    from hnanosolver_b200 import _lib

    w = synth.random_leaves(8, 3, 0, S=2)
    g = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    sim = H.Simulation(g, 2)
    sim.upload(w.velocity, w.scalars)
    _lib.lib().hns_launch_count_reset()
    sim.step(10, w.dt)
    sim.sync()
    # advect_vector (+ its pass over flagged leaves), divergence, 10 x (red, black), gradient, advect_scalars (+ flagged leaves)
    assert _lib.lib().hns_launch_count() == 2 + 1 + 2 * 10 + 1 + 2


# ------------------------------------------------------------------------------------------------------------------
# the drop-in: the reference's own seven symbols (compat/libhns_compat.so) driven by the same C++ caller code as the reference
# ------------------------------------------------------------------------------------------------------------------
needs_compat = pytest.mark.skipif(not (O.compat_driver_available() and O.ref_gpu_available()), reason="compat driver / reference build not present")


def _drive(which, w, fields, iterations):
    """CreateIndexGrid + Compute_Sim + the four stand-alone launchers through the reference's C++ signatures."""
    out = {}
    with O.reference_library(which):
        d = O.RefData(w.coords)
        d.add_vec3("vel", w.velocity)
        for k, v in fields.items():
            d.add_float(k, v)
        g = O.RefGrid(d, w.voxel_size)
        out["nanovdb"] = g.buffer()
        O.ref_compute_sim(d, g, iterations, w.dt, w.voxel_size, PARAMS6, False)
        out["sim_vel"] = d.blocks["vel"].copy()
        for k in fields:
            out["sim_" + k] = d.blocks[k].copy()
        # the same node with the SOP's default vorticity parameters and a collision SDF (third SOP input, hasCollision = true)
        d = O.RefData(w.coords)
        d.add_vec3("vel", w.velocity)
        for k, v in fields.items():
            d.add_float(k, v)
        d.add_float("collision_sdf", _collision_sdf(w))
        params = PARAMS6.copy()
        params[4], params[5] = 1.0, 0.5
        O.ref_compute_sim(d, g, iterations, w.dt, w.voxel_size, params, True)
        out["coll_vel"] = d.blocks["vel"].copy()
        for k in fields:
            out["coll_" + k] = d.blocks[k].copy()
        d = O.RefData(w.coords)
        d.add_vec3("vel", w.velocity)
        for n, s in zip(w.scalar_names, w.scalars):
            d.add_float(n, s)
        O.ref_advect_index_grid(d, w.dt, w.voxel_size)
        for n in w.scalar_names:
            out["adv_" + n] = d.blocks[n].copy()
        d = O.RefData(w.coords)
        d.add_vec3("vel", w.velocity)
        O.ref_advect_index_grid_velocity(d, w.dt, w.voxel_size)
        out["advvel"] = d.blocks["vel"].copy()
        d = O.RefData(w.coords)
        d.add_vec3("vel", w.velocity)
        O.ref_project_non_divergent(d, iterations, w.voxel_size)
        out["proj"] = d.blocks["vel"].copy()
        d = O.RefData(w.coords)
        d.add_vec3("vel", w.velocity)
        d.add_float("divergence", np.zeros(w.num_voxels, np.float32))
        O.ref_divergence(d, w.voxel_size)
        out["div"] = d.blocks["divergence"].copy()
    return out


@needs_compat
def test_compat_library_is_a_drop_in_for_the_reference_launchers(case):
    w = case
    fields = dict(density=w.scalars[0], **combustion_fields(w.num_voxels))
    ref = _drive("reference", w, fields, 7)
    mine = _drive("compat", w, fields, 7)
    T = int(np.frombuffer(ref["nanovdb"][672 + 40:672 + 44].tobytes(), np.uint32)[0])
    assert ref["nanovdb"].size == mine["nanovdb"].size
    assert not ((ref["nanovdb"] != mine["nanovdb"]) & nanovdb_compare_mask(ref["nanovdb"].size, T)).any()
    for k in ref:
        if k != "nanovdb":
            assert_close(mine[k], ref[k], k)


@needs_compat
def test_compat_library_throws_the_reference_exception_types():
    w = synth.random_leaves(4, 2, 1, S=1)
    with O.reference_library("compat"):
        d = O.RefData(w.coords)
        d.add_vec3("vel", w.velocity)
        d.add_float("density", w.scalars[0])
        g = O.RefGrid(d, w.voxel_size)
        with pytest.raises(RuntimeError, match="Missing required input field for combustion"):
            O.ref_compute_sim(d, g, 4, w.dt, w.voxel_size, PARAMS6, False)
        with pytest.raises(RuntimeError, match="voxelSize must be positive"):
            O.ref_compute_sim(d, g, 4, w.dt, 0.0, PARAMS6, False)
        # a sidecar whose 512-blocks are not dense bricks in offset order is refused by the drop-in CreateIndexGrid (C++ exception through
        # the reference's own signature), not simulated wrongly; the reference itself accepts it silently
        c = w.coords.copy()
        c[512 + 64] += np.array([1, 0, 0], np.int32)
        bad = O.RefData(c)
        bad.add_vec3("vel", w.velocity)
        with pytest.raises(RuntimeError, match="not a dense leaf"):
            O.RefGrid(bad, w.voxel_size)


def test_two_devices_in_one_process():
    """hns_set_device: function attributes (the >48 KB dynamic shared memory opt-in of the advection kernels) and the SM count belong
    to a device, not to the process."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from hnanosolver_b200 import _lib

    w = synth.smoke_sphere(32, 1)
    want = None
    try:
        for dev in (0, 1, 0):
            _lib.check(_lib.lib().hns_set_device(dev))
            got = run_product_frame(w, 4)
            if want is None:
                want = got
            for k in ("adv", "p", "vel"):
                assert np.array_equal(got[k], want[k]), (dev, k)
    finally:
        _lib.lib().hns_set_device(0)

