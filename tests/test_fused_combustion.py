"""The frame's combustion stage without a pass of its own (api.cu, fused_combustion): the field update rides in the packed advect_vector
kernel, the expansion term in the divergence pass, the buoyancy force in the gradient pass. HNS_FUSED_COMBUSTION=0 restores the
separate pass. Both schedules must give the same bits in every output, signed zeros included."""
import os

import numpy as np
import pytest

import hnanosolver_b200 as H
from hnanosolver_b200 import _lib, synth

pytestmark = pytest.mark.gpu
PARAMS6 = [0.5, 2.0, 1.5, 0.1, 0.0, 1.0]  # expansionRate, temperatureRelease, buoyancyStrength, ambientTemp, vorticity off
FIELDS = ["density", "fuel", "waste", "temperature", "flame"]
AMBIENT = np.float32(PARAMS6[3])


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _frames(origins, voxel_size, dt, velocity, fields, fused, frames=2, iterations=40):
    """`frames` resident frames through Simulation.time_frames (each from the same inputs, with group 0 packed in front as a running
    simulation finds it) under HNS_FUSED_COMBUSTION=fused: every output of the last frame, and the launches and packed advection
    launches the frames took"""
    lib = _lib.lib()
    sim = H.Simulation(H.create_index_grid_from_origins(origins, voxel_size), len(FIELDS))
    sim.upload(velocity, [fields[k] for k in FIELDS])
    sim.set_combustion(True, 1, 2, 3, 4, H.CombustionParams(*PARAMS6))
    before = os.environ.get("HNS_FUSED_COMBUSTION")
    os.environ["HNS_FUSED_COMBUSTION"] = "1" if fused else "0"
    try:
        lib.hns_launch_count_reset()
        packed0 = lib.hns_packed_advection_launches()
        sim.time_frames(frames, iterations, dt)
        sim.sync()
        counts = (lib.hns_launch_count(), lib.hns_packed_advection_launches() - packed0)
    finally:
        if before is None:
            del os.environ["HNS_FUSED_COMBUSTION"]
        else:
            os.environ["HNS_FUSED_COMBUSTION"] = before
    out = dict(vel=sim.velocity(), adv=sim.aux(H.Simulation.AUX_ADVECTED), div=sim.aux(H.Simulation.AUX_DIVERGENCE),
               p=sim.aux(H.Simulation.AUX_PRESSURE))
    out.update({k: sim.scalar(i) for i, k in enumerate(FIELDS)})
    sim.close()
    return out, counts


def _assert_same_bits(origins, voxel_size, dt, velocity, fields, frames=2):
    want, (launches_split, packed_split) = _frames(origins, voxel_size, dt, velocity, fields, False, frames)
    got, (launches_fused, packed_fused) = _frames(origins, voxel_size, dt, velocity, fields, True, frames)
    assert packed_split == packed_fused == 2 * frames        # advect_vector and advect_scalars on the packed groups in every frame
    assert launches_split - launches_fused == frames         # the combustion pass is gone from every frame
    for k in want:
        assert np.array_equal(_bits(got[k]), _bits(want[k])), k


def test_fused_combustion_is_bit_identical_on_config4():
    """bench.py's frame: config 4, the 512^3 sparse smoke with density and the four combustion fields, I = 40"""
    w = synth.WORKLOADS["c4"](with_coords=False)
    fields = dict(density=w.scalars[0], **synth.combustion_fields(w))
    _assert_same_bits(w.origins, w.voxel_size, w.dt, w.velocity, fields)


def test_fused_combustion_is_bit_identical_on_every_branch():
    """Inputs that take every branch of the combustion and buoyancy terms: no oxygen (fuel + waste > 1), fuel below 0.001, a
    temperature at or below ambient, and divergences of exactly -0.0 both where there is no oxygen (left as they are) and where there is
    (fma(burn, expansion, -0.0) turns them into +0.0 or more). The -0.0 divergences come from velocities of a few subnormal steps with
    1 / voxel size = 0.25: the last product of the divergence rounds -1 and -2 steps to -0.0."""
    w = synth.random_leaves(60, 4, 9, cfl=1.2, S=1)
    n, h = w.num_voxels, 4.0
    rng = np.random.default_rng(7)
    velocity = rng.integers(-3, 4, (n, 3)).astype(np.float32) * np.float32(np.ldexp(1.0, -149))
    fuel = rng.choice(np.array([0.0, 0.0005, 0.3, 0.6, 0.9], np.float32), n)
    waste = (0.6 * rng.random(n)).astype(np.float32)
    temperature = (0.3 * rng.random(n)).astype(np.float32)
    temperature[::7] = AMBIENT
    fields = dict(density=rng.random(n).astype(np.float32), fuel=fuel, waste=waste, temperature=temperature,
                  flame=(0.2 * rng.random(n)).astype(np.float32))

    f = np.where(fuel < np.float32(0.001), np.float32(0), fuel)
    no_oxygen = (np.float32(1) - f - waste) < 0
    sim = H.Simulation(H.create_index_grid_from_origins(w.origins, h), 0)
    sim.upload(velocity)
    sim.advect_velocity(w.dt)
    sim.divergence(of_advected=True)
    sim.sync()
    div = sim.aux(H.Simulation.AUX_DIVERGENCE)          # before the expansion term
    sim.close()
    minus_zero = (div == 0) & np.signbit(div)
    assert (minus_zero & no_oxygen).any() and (minus_zero & ~no_oxygen).any()
    assert (fuel == np.float32(0.0005)).any() and no_oxygen.any() and (~no_oxygen).any()
    assert ((temperature <= AMBIENT) & ((f == 0) | no_oxygen)).any()   # temperatures combustion leaves at or below ambient
    _assert_same_bits(w.origins, h, w.dt, velocity, fields, frames=3)
