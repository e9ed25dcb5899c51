"""Sampler semantics: the reference's own known answers (Tests/IndexGrid.cpp) + the oracle against the reference's
__hostdev__ samplers running on the CPU over a real NanoVDB host grid."""
import numpy as np
import pytest

from oracle import oracle as O

needs_refhost = pytest.mark.skipif(not O.ref_host_available(), reason="needs oracle/_ref/libref_host.so, built only from the original project's sources (oracle/Makefile REF)")


def _line(axis, n=15):
    c = np.zeros((n, 3), np.int32)
    c[:, axis] = np.arange(n)
    return c


def test_trilinear_known_answers():
    # Tests/IndexGrid.cpp:157-224: density(i,0,0) = i -> f(0.5,0,0) = 0.5, f(1.25,0,0) = 1.25, inactive (1,1,0) -> 0
    pts = _line(0)
    ix = O.OracleIndex(pts)
    data = ix.get_values(pts).astype(np.float32) * 0
    data[ix.get_values(pts).astype(np.int64) - 1] = np.arange(15, dtype=np.float32)
    got = ix.trilinear_f(data, [[0.5, 0, 0], [1.25, 0, 0], [5.0, 0, 0]])
    assert got.tolist() == [0.5, 1.25, 5.0]
    assert ix.nearest_f(data, [[1, 1, 0]])[0] == 0.0
    # Tests/IndexGrid.cpp:226-282: nearest (i,0,0) -> i ; Vec3f at (0,i,0) -> (i,i,i)
    assert ix.nearest_f(data, pts).tolist() == list(range(15))
    pv = _line(1)
    iv = O.OracleIndex(pv)
    vdata = np.zeros((15, 3), np.float32)
    vdata[iv.get_values(pv).astype(np.int64) - 1] = np.arange(15, dtype=np.float32)[:, None]
    assert iv.trilinear_v(vdata, [[0, 5.0, 0]])[0].tolist() == [5.0, 5.0, 5.0]
    # Tests/IndexGrid.cpp:84-155: values scaled x2 -> sample(5.5) == 11
    assert ix.trilinear_f(data * 2, [[5.5, 0, 0]])[0] == 11.0
    assert iv.trilinear_v(vdata * 2, [[0, 5.5, 0]])[0][0] == 11.0


def test_floor_rounds_down_for_negative_positions():
    # Floor() uses __float2int_rd (Stencils.hpp:25-43): -0.25 -> cell -1, fraction 0.75
    pts = np.array([[-1, 0, 0], [0, 0, 0]], np.int32)
    ix = O.OracleIndex(pts)
    data = np.zeros(2, np.float32)
    data[ix.get_values(pts).astype(np.int64) - 1] = [10.0, 20.0]
    assert ix.trilinear_f(data, [[-0.25, 0, 0]])[0] == np.float32(10.0) + np.float32(0.75) * np.float32(10.0)


@needs_refhost
def test_samplers_match_reference_host_code():
    rng = np.random.default_rng(11)
    pts = np.unique(rng.integers(-12, 30, size=(6000, 3)).astype(np.int32), axis=0)
    ix, rh = O.OracleIndex(pts), O.RefHostGrid(pts)
    n = ix.num_active
    f = rng.standard_normal(n).astype(np.float32)
    v = rng.standard_normal((n, 3)).astype(np.float32)
    q = pts[:400] + rng.integers(-1, 2, size=(400, 3)).astype(np.int32)
    assert np.array_equal(ix.nearest_f(f, q), rh.nearest_f(f, q))          # integer lookups + loads: bit exact
    xyz = (pts[:400] + rng.uniform(-1.5, 1.5, size=(400, 3))).astype(np.float32)
    # The oracle follows the DEVICE arithmetic (fused a + w*(b-a), see hns_oracle.c header); the host build of the
    # reference samplers is unfused, so agreement is to rounding, not bitwise: tolerance 4 ulp of the data range.
    tol = 4 * np.finfo(np.float32).eps * 4.0
    assert np.abs(ix.trilinear_f(f, xyz) - rh.trilinear_f(f, xyz)).max() <= tol
    assert np.abs(ix.trilinear_v(v, xyz) - rh.trilinear_v(v, xyz)).max() <= tol


# ------------------------------------------------------------------------------------------------------------------
# vorticity confinement (Kernel.cu:969-1025), out-of-place restatement: properties that hold by construction
# ------------------------------------------------------------------------------------------------------------------
class _Block:
    """all leaves of an m x m x m block, sidecar (leaf-major, x<<6|y<<3|z) order, with a smooth + noisy velocity"""

    def __init__(self, m=3, seed=3):
        a = np.arange(m, dtype=np.int32) * 8
        origins = np.stack(np.meshgrid(a, a, a, indexing="ij"), -1).reshape(-1, 3)  # x-major == NanoVDB order inside one lower node
        o = np.arange(8, dtype=np.int32)
        off = np.stack(np.meshgrid(o, o, o, indexing="ij"), -1).reshape(-1, 3)
        self.coords = (origins[:, None, :] + off[None, :, :]).reshape(-1, 3).astype(np.int32)
        rng = np.random.default_rng(seed)
        c = self.coords.astype(np.float32)
        self.velocity = (np.stack([np.sin(0.3 * c[:, 1]), np.cos(0.2 * c[:, 2]), np.sin(0.25 * c[:, 0] + 0.1 * c[:, 1])], 1)
                         + 0.2 * rng.standard_normal((len(c), 3))).astype(np.float32)
        self.dt, self.voxel_size = 1.0 / 24.0, 0.1


def _dense_block(m=3):
    return _Block(m)


def test_vorticity_identity_when_scale_or_offset_is_zero():
    w = _dense_block()
    ix = O.OracleIndex(w.coords)
    for scale, fs in ((0.0, 2.0), (1.0, 0.5), (3.0, -0.99), (1.0, 0.0)):
        assert np.array_equal(ix.vorticity_confinement(w.velocity, w.dt, w.voxel_size, scale, fs), w.velocity)


def test_vorticity_of_a_rigid_rotation_is_uniform_so_the_force_vanishes_inside():
    # u = k * (-y, x, 0): curl = (0, 0, 2k) everywhere away from the domain boundary -> |curl| constant -> grad 0 -> no force
    w = _dense_block(3)
    c = w.coords.astype(np.float32)
    vel = np.stack([-(c[:, 1] - 12.0), c[:, 0] - 12.0, np.zeros(len(c), np.float32)], 1).astype(np.float32) * np.float32(0.25)
    ix = O.OracleIndex(w.coords)
    out = ix.vorticity_confinement(vel, w.dt, w.voxel_size, 1.0, 1.0)
    lo, hi = w.coords.min(0), w.coords.max(0)
    inside = np.all((w.coords >= lo + 2) & (w.coords <= hi - 2), axis=1)  # stencil radius 1 + offset 1
    assert inside.sum() > 1000
    assert np.array_equal(out[inside], vel[inside])
    assert not np.array_equal(out[~inside], vel[~inside])  # at the boundary inactive samples (0) create a gradient


def test_vorticity_offset_is_truncated_toward_zero_and_odd_in_sign():
    w = _dense_block(2)
    ix = O.OracleIndex(w.coords)
    a = ix.vorticity_confinement(w.velocity, w.dt, w.voxel_size, 1.0, 2.0)
    b = ix.vorticity_confinement(w.velocity, w.dt, w.voxel_size, 1.0, 2.9)
    assert np.array_equal(a, b)                      # (int)2.9 == 2
    m = ix.vorticity_confinement(w.velocity, w.dt, w.voxel_size, 1.0, -2.0)
    # a negative offset swaps the +/- samples: the gradient, hence the force, changes sign exactly
    assert np.array_equal((a - w.velocity != 0), (m - w.velocity != 0))
    f_pos, f_neg = a.astype(np.float64) - w.velocity, m.astype(np.float64) - w.velocity
    assert np.allclose(f_pos, -f_neg, rtol=1e-4, atol=1e-7)
