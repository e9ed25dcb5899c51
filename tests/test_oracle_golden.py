"""The oracle against outputs of the reference itself (fixtures made by tests/golden/make_golden.py on a B200 from
oracle/_ref/libhns_ref.so = the unmodified reference kernels and launchers). Runs without a GPU."""
import os

import numpy as np
import pytest

from helpers import GOLDEN, Golden, nanovdb_compare_mask
from oracle import oracle as O

CASES = [c for c in ("soup", "sphere") if os.path.exists(os.path.join(GOLDEN, f"ref_{c}.npz"))]
pytestmark = pytest.mark.skipif(not CASES, reason="no golden fixtures committed yet")


@pytest.fixture(scope="module", params=CASES)
def gold(request):
    return Golden(request.param)


def _scalars(g):
    return [g[f"scalar{i}"] for i in range(len(g["scalar_names"]))]


def test_index_grid_bit_exact(gold):
    ix = O.OracleIndex(gold["coords"])
    assert np.array_equal(ix.get_values(gold["query_ijk"]), gold["query_values"])
    buf = ix.nanovdb_buffer(float(gold["voxel_size"]))
    ref = gold["nanovdb"]
    assert buf.size == ref.size
    T = int(np.frombuffer(ref[672 + 40:672 + 44].tobytes(), np.uint32)[0])
    m = nanovdb_compare_mask(ref.size, T)
    bad = np.nonzero((buf != ref) & m)[0]
    assert bad.size == 0, f"oracle NanoVDB buffer differs from voxelsToGrid at bytes {bad[:16]}"


def test_frame_stages(gold):
    ix = O.OracleIndex(gold["coords"])
    h, dt, I = float(gold["voxel_size"]), float(gold["dt"]), int(gold["iterations"])
    r = ix.frame(gold["velocity"], _scalars(gold), I, dt, h)
    gold.check(r["adv"], "frame_adv", "advect_vector")
    gold.check(r["div"], "frame_div", "divergence")
    gold.check(r["p"], "frame_p", "pressure after RBGS")
    gold.check(r["vel"], "frame_vel", "projected velocity")
    for i, s in enumerate(r["scalars"]):
        gold.check(s, f"frame_scalar{i}", f"advect_scalars[{i}]")


def test_standalone_launchers(gold):
    ix = O.OracleIndex(gold["coords"])
    h, dt, I = float(gold["voxel_size"]), float(gold["dt"]), int(gold["iterations"])
    for i, s in enumerate(_scalars(gold)):
        gold.check(ix.advect_scalar(gold["velocity"], s, dt, h), f"advect_index_grid_{i}", f"AdvectIndexGrid[{i}]")
    gold.check(ix.advect_vector(gold["velocity"], dt, h), "advect_index_grid_velocity", "AdvectIndexGridVelocity")
    gold.check(ix.divergence(gold["velocity"], h), "divergence", "Divergence")
    vel, _, _ = ix.project_non_divergent(gold["velocity"], I, h)
    gold.check(vel, "project_non_divergent", "ProjectNonDivergent")


def test_compute_sim(gold):
    ix = O.OracleIndex(gold["coords"])
    h, dt, I = float(gold["voxel_size"]), float(gold["dt"]), int(gold["iterations"])
    fields = dict(density=gold["scalar0"], fuel=gold["comb_fuel"], waste=gold["comb_waste"], temperature=gold["comb_temperature"],
                  flame=gold["comb_flame"])
    vel, out = ix.compute_sim(gold["velocity"], fields, I, dt, h, gold["params"])
    gold.check(vel, "compute_sim_vel", "Compute_Sim velocity")
    for k, v in out.items():
        gold.check(v, f"compute_sim_{k}", f"Compute_Sim {k}")


def test_vorticity_confinement(gold):
    """oracle vs the reference's vorticityConfinement kernel launched out of place (tests/golden/make_golden.py)"""
    if "vorticity_cases" not in gold:
        pytest.skip("fixture predates the vorticity vectors")
    ix = O.OracleIndex(gold["coords"])
    h, dt = float(gold["voxel_size"]), float(gold["dt"])
    for i, (scale, fs) in enumerate(gold["vorticity_cases"]):
        got = ix.vorticity_confinement(gold["velocity"], dt, h, float(scale), float(fs))
        gold.check(got, f"vorticity_{i}", f"vorticityConfinement scale={scale} factorScale={fs}")
        assert not np.array_equal(got, gold["velocity"])


def test_compute_sim_sop_default_vorticity_is_identity(gold):
    if "compute_sim_sopdefault_vel" not in gold:
        pytest.skip("fixture predates the vorticity vectors")
    assert gold.sha256("compute_sim_sopdefault_vel") == gold.sha256("compute_sim_vel")
    ix = O.OracleIndex(gold["coords"])
    h, dt, I = float(gold["voxel_size"]), float(gold["dt"]), int(gold["iterations"])
    fields = dict(density=gold["scalar0"], fuel=gold["comb_fuel"], waste=gold["comb_waste"], temperature=gold["comb_temperature"],
                  flame=gold["comb_flame"])
    p = gold["params"].copy()
    p[4], p[5] = 1.0, 0.5
    vel, _ = ix.compute_sim(gold["velocity"], fields, I, dt, h, p)
    gold.check(vel, "compute_sim_sopdefault_vel", "Compute_Sim velocity, SOP default vorticity parameters")


# ------------------------------------------------------------------------------------------------------------------
# the hasCollision path (SURVEY.md 8f-2): reference kernels launched one by one with a sphere-collider SDF
# ------------------------------------------------------------------------------------------------------------------
def _needs_collision(gold):
    if "collision_sdf" not in gold:
        pytest.skip("fixture predates the collision vectors")


def test_collision_kernels(gold):
    _needs_collision(gold)
    ix = O.OracleIndex(gold["coords"])
    h, dt, I = float(gold["voxel_size"]), float(gold["dt"]), int(gold["iterations"])
    sdf = gold["collision_sdf"]
    assert (sdf < 0).sum() > 100 and ((sdf >= 0) & (sdf < 0.1)).sum() > 100      # the fixture exercises both branches
    got = ix.collision_boundary(gold["velocity"], sdf, h, ix.SITE_ENFORCE)
    gold.check(got, "coll_enforce", "enforceCollisionBoundaries")
    assert not np.array_equal(got, gold["velocity"])
    got = ix.advect_vector_sdf(gold["velocity"], sdf, dt, h)
    gold.check(got, "coll_advect_vector", "advect_vector(hasCollision)")
    # the tail of subtractPressureGradient acts on the kernel's own result = the collision-free projected velocity (the reference's
    # frame_vel, rebuilt by the oracle's frame and checked against it)
    frame_vel = ix.frame(gold["velocity"], _scalars(gold), I, dt, h)["vel"]
    gold.check(frame_vel, "frame_vel", "projected velocity")
    got = ix.collision_boundary(frame_vel, sdf, h, ix.SITE_GRADIENT)
    gold.check(got, "coll_gradient", "subtractPressureGradient(hasCollision)")
    outs = ix.advect_scalars_sdf(frame_vel, _scalars(gold), sdf, dt, h)
    for i, o in enumerate(outs):
        gold.check(o, f"coll_scalar{i}", f"advect_scalars(hasCollision)[{i}]")
        assert not gold.matches(o, f"frame_scalar{i}")


def test_compute_sim_with_collision(gold):
    _needs_collision(gold)
    ix = O.OracleIndex(gold["coords"])
    h, dt, I = float(gold["voxel_size"]), float(gold["dt"]), int(gold["iterations"])
    fields = dict(density=gold["scalar0"], fuel=gold["comb_fuel"], waste=gold["comb_waste"], temperature=gold["comb_temperature"],
                  flame=gold["comb_flame"], collision_sdf=gold["collision_sdf"])
    vel, out = ix.compute_sim(gold["velocity"], fields, I, dt, h, gold["params"], has_collision=True)
    gold.check(vel, "compute_sim_coll_vel", "Compute_Sim(hasCollision) velocity")
    for k, v in out.items():
        if k == "collision_sdf":
            gold.check(v, "compute_sim_coll_sdf_out", k)          # zeros: the reference's never-written output buffer
        else:
            gold.check(v, f"compute_sim_coll_{k}", k)
    # without hasCollision the SDF block is carried (and zeroed) but changes nothing else
    vel0, out0 = ix.compute_sim(gold["velocity"], fields, I, dt, h, gold["params"], has_collision=False)
    gold.check(vel0, "compute_sim_vel", "Compute_Sim velocity, collision_sdf present but hasCollision false")
    assert not np.array_equal(vel0, vel)
