"""The multigrid pressure solve (csrc/multigrid.cu) on every shape of hierarchy and with every solver option.

Three layers, so that a mismatch can be told apart from a modelling error both sides share:
- the device V-cycle equals its CPU restatement (oracle.OracleMultigrid) bit for bit, on hierarchies chosen so that together they
  reach every branch of v_cycle / mg_coarse_cycle, and with each option: CUDA graph on and off, the graph cache, rel_tol, the
  coarsest level's iteration count, the frame;
- the restatement's pieces (restriction, prolongation, coarse diagonal, residual) equal their plain definitions, in fp64;
- the converged solve is compared with an fp64 solution of the 7-point Poisson equation, which depends on neither implementation.

When a bitwise check fails, localise it with max_levels=2, one cycle and V(1,0) or V(0,1) (a single restriction, coarsest solve and
prolongation), then max_levels=3 and so on up the levels."""
import numpy as np
import pytest

from hnanosolver_b200 import synth


def _workload(name, origins, seed=5):
    """dense leaves at `origins`, a rough velocity (hash noise, up to 1.5 voxels per step) and one scalar"""
    o = np.asarray(origins, np.int32).reshape(-1, 3)
    o = np.ascontiguousarray(o[synth.nanovdb_order(o)])
    c = synth.dense_coords(o)
    d = np.stack([3.0 * (synth.hash_noise(seed, c, ch) - 0.5) for ch in range(3)], -1)
    vel = (d * np.float32(synth.VOXEL_SIZE / synth.DT)).astype(np.float32)
    return synth.Workload(name, o, c, vel, [synth.hash_noise(seed, c, 10)], ["density"])


def _grid_origins(xs, ys, zs):
    return np.stack(np.meshgrid(xs, ys, zs, indexing="ij"), -1).reshape(-1, 3)


def _block4_isolated_first():
    # a 4x4x4-leaf block, plus one leaf in the root tile x < -4096 (which sorts first): the last level keeps the block's single cell
    # group in leaf 1 and an empty parent of the lone leaf in leaf 0
    return _workload("block4_isolated_first", np.concatenate([_grid_origins(*[np.arange(0, 32, 8)] * 3), [[-4160, -8, 0]]]))


SOUP = dict(n_leaves=60, extent=7, seed=11, offset=(-24, -8, -40))   # tests/test_multigrid.py's soup
# name -> (workload, max_levels)
CASES = {
    "one": (lambda: _workload("one", [[0, 0, 0]]), 16),
    "block2": (lambda: _workload("block2", _grid_origins(*[[0, 8]] * 3)), 16),
    "block4_isolated_first": (_block4_isolated_first, 16),
    "scattered": (lambda: _workload("scattered", _grid_origins(np.arange(0, 160, 16), np.arange(0, 96, 16), np.arange(0, 96, 16))), 16),
    "slab": (lambda: _workload("slab", _grid_origins(np.arange(-64, 64, 8), np.arange(-64, 64, 8), [0])), 16),
    "soup_capped": (lambda: synth.random_leaves(**SOUP), 2),
    "c2_capped": (lambda: synth.WORKLOADS["c2"](), 3),
    "sphere40": (lambda: synth.smoke_sphere(40, 2), 16),
    "soup": (lambda: synth.random_leaves(**SOUP), 16),
    "c2": (lambda: synth.WORKLOADS["c2"](), 16),
}
# name -> (cells per level, non-empty leaves on the last level, index of the last non-empty leaf there, how the build ended)
BRANCHES = {
    "one": ([512], 1, 0, "one leaf"),                                          # n == 1: plain red-black sweeps
    "block2": ([4096, 512], 1, 0, "one leaf"),                                 # one-CTA coarsest solve on leaf 0
    "block4_isolated_first": ([33280, 4160, 520, 65, 8], 1, 1, "one leaf"),    # one-CTA coarsest solve at an offset
    "scattered": ([184320, 23040, 2880, 360], 12, 11, "no cells"),             # masked smoothing on many leaves
    "slab": ([131072, 16384, 2048, 256], 4, 3, "no cells"),
    "soup_capped": ([30720, 3840], 38, 37, "max_levels"),
    "c2_capped": ([685056, 85632, 10704], 44, 43, "max_levels"),
    "sphere40": ([64000, 8000, 1000, 125], 1, 0, "one leaf"),
    "soup": ([30720, 3840, 480, 60], 8, 7, "no cells"),
    "c2": ([685056, 85632, 10704, 1338, 123], 1, 0, "one leaf"),
}

_built = {}


def _case(name):
    """(workload, max_levels), built once per session"""
    if name not in _built:
        make, max_levels = CASES[name]
        _built[name] = (make(), max_levels)
    return _built[name]


def _leaf_sets(origins, max_levels=16):
    """hns_mg_create's hierarchy restated: per level the leaf origins (NanoVDB order) and which of their cells lie inside the domain.
    A coarse level holds the parents of ALL leaves of the level below, empty ones included; a cell is inside iff its 8 children are.
    Returns (levels, non-empty leaf ids of the last level, how the build ended)."""
    max_levels = max_levels if max_levels > 0 else 16
    org = np.asarray(origins, np.int64).reshape(-1, 3)
    inside = np.ones((org.shape[0], 8, 8, 8), bool)
    levels = [(org, inside)]
    while True:
        non_empty = np.flatnonzero(inside.reshape(org.shape[0], -1).any(1))
        if non_empty.size <= 1:
            end = "one leaf"
            break
        if len(levels) >= max_levels:
            end = "max_levels"
            break
        porg, inv = np.unique((org >> 4) * 8, axis=0, return_inverse=True)
        order = synth.nanovdb_order(porg)
        rank = np.empty_like(order)
        rank[order] = np.arange(order.size)
        porg, parent = porg[order], rank[inv.reshape(-1)]
        covered = inside.reshape(-1, 4, 2, 4, 2, 4, 2).all(axis=(2, 4, 6))
        pin = np.zeros((porg.shape[0], 8, 8, 8), bool)
        octant = ((org >> 3) & 1) * 4
        for l in range(org.shape[0]):
            x, y, z = octant[l]
            pin[parent[l], x:x + 4, y:y + 4, z:z + 4] |= covered[l]
        if not pin.any():
            end = "no cells"
            break
        org, inside = porg, pin
        levels.append((org, inside))
    return levels, non_empty, end


def _div_of_advected(O, w):
    ix = O.OracleIndex(w.coords)
    return ix.divergence(ix.advect_vector(w.velocity, w.dt, w.voxel_size), w.voxel_size)


def _oracle_mg(O, name, **kw):
    w, max_levels = _case(name)
    return O.OracleMultigrid(w.coords, w.voxel_size, max_levels=max_levels, **kw)


def _bits_differ(got, want, what):
    """'' when got and want are the same float32 bits, else a short description of where they differ"""
    g, e = np.asarray(got, np.float32).view(np.uint32), np.asarray(want, np.float32).view(np.uint32)
    bad = np.flatnonzero(g != e)
    if bad.size == 0:
        return ""
    d = np.abs(np.asarray(got, np.float64) - want).max() / max(np.abs(np.asarray(want, np.float64)).max(), 1e-30)
    return f"{what}: {bad.size} of {g.size} values differ (first at {bad[0]}), max relative difference {d:.2e}"


# ---- CPU: each case reaches its branch ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CASES))
def test_case_reaches_its_branch(oracle_mod, name):
    w, max_levels = _case(name)
    levels, non_empty, end = _leaf_sets(w.origins, max_levels)
    cells, n_last, last_leaf, how = BRANCHES[name]
    assert [int(inside.sum()) for _, inside in levels] == cells
    assert (non_empty.size, int(non_empty[-1]), end) == (n_last, last_leaf, how)
    omg = _oracle_mg(oracle_mod, name)
    assert [ix.n for ix, _ in omg.levels] == cells                            # the restatement builds the oracle's hierarchy
    # the oracle's own choice of coarsest solver: one-leaf SOR (coarsest_omega) iff the last level has one non-empty leaf
    assert (np.unique(omg.levels[-1][0].coords >> 3, axis=0).shape[0] == 1) == (n_last == 1)


def test_restated_leaf_sets_keep_empty_parents():
    # the lone leaf's 8^3 cells shrink to one cell on level 3 and to none on level 4, where its parent leaf is kept, empty, and sorts
    # first (root tile x < 0)
    levels, non_empty, _ = _leaf_sets(_block4_isolated_first().origins)
    assert [o.shape[0] for o, _ in levels] == [65, 9, 2, 2, 2]
    assert [int(inside[0].sum()) for _, inside in levels[1:]] == [64, 8, 1, 0]
    assert levels[-1][0].tolist() == [[-264, -8, 0], [0, 0, 0]]
    assert non_empty.tolist() == [1]


# ---- CPU: the oracle's pieces against their definitions ---------------------------------------------------------------------------
def _finder(coords):
    """index of each queried coordinate in `coords`, -1 where absent"""
    def key(c):
        c = np.asarray(c, np.int64) + (1 << 20)
        return (c[..., 0] << 42) | (c[..., 1] << 21) | c[..., 2]
    keys = key(coords)
    order = np.argsort(keys)
    sk = keys[order]

    def find(q):
        k = key(q)
        pos = np.minimum(np.searchsorted(sk, k), sk.size - 1)
        return np.where(sk[pos] == k, order[pos], -1)
    return find


def _gather(values, find, q):
    """values at coordinates q (float64), 0 where q is not a cell"""
    i = find(q)
    return np.where(i >= 0, np.asarray(values, np.float64)[np.maximum(i, 0)], 0.0)


_FACES = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1]], np.int64)
_EPS = float(np.finfo(np.float32).eps)


@pytest.mark.parametrize("name", ["block4_isolated_first", "slab"])
def test_oracle_pieces_match_their_definitions(oracle_mod, name):
    import ctypes as C

    O = oracle_mod
    L = O.lib()
    f32p, i32p = C.POINTER(C.c_float), C.POINTER(C.c_int32)
    omg = _oracle_mg(O, name)
    rng = np.random.default_rng(7)
    for k, (ix, dx) in enumerate(omg.levels):
        c = ix.coords.astype(np.int64)
        find = _finder(ix.coords)
        # diagonal: 6 + (faces outside) * (1/theta_k - 1), theta_k = 1/2 + 2^-(k+1), two float32 roundings
        if k:
            extra = np.float32(1.0 / (0.5 + 2.0 ** -(k + 1)) - 1.0)
            diag = np.empty(ix.n, np.float32)
            L.ora_mg_diag(ix._h, ix.coords.ctypes.data_as(i32p), ix.n, extra, diag.ctypes.data_as(f32p))
            outside = sum((find(c + f) < 0).astype(np.int32) for f in _FACES)
            assert np.array_equal(diag.view(np.uint32), (np.float32(6.0) + outside.astype(np.float32) * extra).astype(np.float32).view(np.uint32))
            assert np.array_equal(diag, omg.diag[k])
        # residual: rhs - (sum of the 6 neighbours - diag p) / dx^2, p = 0 outside, within fp32 rounding
        p = rng.standard_normal(ix.n).astype(np.float32)
        rhs = (rng.standard_normal(ix.n) / float(dx) ** 2).astype(np.float32)
        r = omg.residual(k, p, rhs)
        nb = np.stack([_gather(p, find, c + f) for f in _FACES])
        dg = np.float64(6.0) if k == 0 else omg.diag[k].astype(np.float64)
        want = rhs - (nb.sum(0) - dg * p) / np.float64(dx) ** 2
        scale = np.abs(rhs) + (np.abs(nb).sum(0) + dg * np.abs(p)) / np.float64(dx) ** 2
        assert np.all(np.abs(r - want) <= 8 * _EPS * scale)
        if k + 1 == len(omg.levels):
            continue
        # restriction of a residual on nine tenths of this level's cells onto all their parents: the mean of the 8 children, a
        # missing child counting 0
        keep = rng.random(ix.n) < 0.9
        sub, rs = O.OracleIndex(ix.coords[keep]), np.ascontiguousarray(r[keep])
        parents = np.unique(sub.coords >> 1, axis=0).astype(np.int32)
        out = np.empty(parents.shape[0], np.float32)
        L.ora_mg_restrict(sub._h, rs.ctypes.data_as(f32p), parents.ctypes.data_as(i32p), parents.shape[0], out.ctypes.data_as(f32p))
        kids = np.stack([_gather(rs, _finder(sub.coords), 2 * parents.astype(np.int64) + np.array([a, b, e]))
                         for a in (0, 1) for b in (0, 1) for e in (0, 1)])
        assert np.all(np.abs(out - kids.mean(0)) <= 4 * _EPS * np.abs(kids).sum(0) / 8)
        assert np.any(np.all(kids != 0, axis=0)) and np.any(np.any(kids == 0, axis=0))
        # prolongation: p += the tensor product of (3/4 own parent, 1/4 the parent on the child's side) per axis, missing parents 0
        ixc = omg.levels[k + 1][0]
        e = rng.standard_normal(ixc.n).astype(np.float32)
        p0 = np.zeros(ix.n, np.float32)
        L.ora_mg_prolong_add(ixc._h, e.ctypes.data_as(f32p), ix.coords.ctypes.data_as(i32p), ix.n, p0.ctypes.data_as(f32p))
        findc = _finder(ixc.coords)
        own, side = c >> 1, np.where(c & 1, 1, -1)
        want = np.zeros(ix.n)
        bound = np.zeros(ix.n)
        for m in range(8):
            sel = np.array([(m >> 2) & 1, (m >> 1) & 1, m & 1])
            wgt = np.prod(np.where(sel == 1, 0.25, 0.75))
            v = wgt * _gather(e, findc, own + sel * side)
            want += v
            bound += np.abs(v)
        assert np.all(np.abs(p0 - want) <= 8 * _EPS * bound)
        assert np.any(np.abs(want) < bound * (1 - 1e-6))                       # not every fine cell sees 8 parents of one sign


# ---- CPU: the restatement's converged solve against an fp64 Poisson solution --------------------------------------------------------
# max |p - p64| / max |p64|, V(2,2) cycles with omega 1.15, measured on the CPU restatement (the device solve is the same bits);
# gates at about 4x. To rel_tol = 1e-5 the algebraic error dominates: sphere40 5.2e-6 after 4 cycles, soup 2.2e-5 after 3,
# block4_isolated_first 4.5e-5 after 3. After 8 cycles only fp32 rounding is left (cycles 5 to 12 stay at a floor): at most 6.4e-7,
# 2.7e-7 and 2.8e-7.
P64_GATE = {"sphere40": (2e-5, 2.5e-6), "soup": (9e-5, 1.1e-6), "block4_isolated_first": (1.8e-4, 1.1e-6)}
_p64 = {}


def _poisson64(O, name):
    """(div, fp64 solution of (sum of the 6 neighbours - 6 p) / dx^2 = div with p = 0 outside, the fp64 operator)"""
    if name not in _p64:
        import scipy.sparse as sp
        import scipy.sparse.linalg as spla

        w, _ = _case(name)
        div = _div_of_advected(O, w)
        c = w.coords.astype(np.int64)
        find = _finder(w.coords)
        n = c.shape[0]
        rows, cols = [], []
        for f in _FACES:
            j = find(c + f)
            rows.append(np.flatnonzero(j >= 0))
            cols.append(j[j >= 0])
        rows, cols = np.concatenate(rows), np.concatenate(cols)
        dx2 = float(np.float32(w.voxel_size)) ** 2
        A = (sp.csr_matrix((np.ones(rows.size), (rows, cols)), shape=(n, n)) - 6.0 * sp.identity(n, format="csr")) / dx2
        p64, info = spla.cg(-A, -div.astype(np.float64), rtol=1e-13, maxiter=20000)
        assert info == 0
        _p64[name] = (div, p64, A)
    return _p64[name]


def _against_p64(A, div, p64, p):
    """(fp64 relative residual of p, max |p - p64| / max |p64|)"""
    b = div.astype(np.float64)
    return (np.linalg.norm(b - A @ p.astype(np.float64)) / np.linalg.norm(b),
            np.abs(p.astype(np.float64) - p64).max() / np.abs(p64).max())


@pytest.mark.parametrize("name", list(P64_GATE))
def test_oracle_solve_matches_the_fp64_poisson_solution(oracle_mod, name):
    div, p64, A = _poisson64(oracle_mod, name)
    assert np.linalg.norm(div - A @ p64) <= 1e-12 * np.linalg.norm(div)
    omg = _oracle_mg(oracle_mod, name)
    p, cycles, rel = omg.solve(div, 20, 2, 2, 1.15, rel_tol=1e-5)
    rel64, err = _against_p64(A, div, p64, p)
    assert cycles <= 4 and rel64 <= 1e-5 and abs(rel64 - rel) <= 1e-6 * rel and err <= P64_GATE[name][0], (cycles, rel64, err)
    p, _, _ = omg.solve(div, 8, 2, 2, 1.15)
    assert _against_p64(A, div, p64, p)[1] <= P64_GATE[name][1]


# ---- GPU ----------------------------------------------------------------------------------------------------------------------------
def _gpu(name, velocity=None):
    """(workload, grid, Simulation with the advected divergence computed)"""
    import hnanosolver_b200 as H

    w, _ = _case(name)
    grid = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    sim = _sim(grid, w, velocity)
    return w, grid, sim


def _sim(grid, w, velocity=None):
    import hnanosolver_b200 as H

    sim = H.Simulation(grid, 0)
    sim.upload(w.velocity if velocity is None else velocity)
    sim.advect_velocity(w.dt)
    sim.divergence(True)
    return sim


def _multigrid(grid, name):
    import hnanosolver_b200 as H

    return H.Multigrid(grid, _case(name)[1])


def _oracle_cycles(omg, div, cycles, nu_pre, nu_post, omega):
    """the oracle's pressure after each of `cycles` V-cycles from p = 0, and the fp64 relative residual after each"""
    p = np.zeros_like(div)
    out, rel = [], []
    for _ in range(cycles):
        omg.v_cycle(p, div, nu_pre, nu_post, np.float32(omega))
        out.append(p.copy())
        a, b = omg.residual_sums(p, div)
        rel.append(float(np.sqrt(a / b)))
    return out, rel


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_device_hierarchy_matches_the_restatement(oracle_mod, name):
    w, grid, _ = _gpu(name)
    mg = _multigrid(grid, name)
    levels, _, _ = _leaf_sets(w.origins, _case(name)[1])
    omg = _oracle_mg(oracle_mod, name)
    assert mg.num_levels == len(omg.levels) == len(levels)
    assert [mg.level_cells(k) for k in range(mg.num_levels)] == [ix.n for ix, _ in omg.levels]
    assert [mg.level_leaves(k) for k in range(mg.num_levels)] == [o.shape[0] for o, _ in levels]


NUS = [(2, 2), (1, 0), (0, 1), (3, 1)]
SETTINGS = [(nu, om) for nu in NUS for om in (1.0, 1.15)]
FEW_SETTINGS = [((2, 2), 1.15), ((1, 0), 1.0)]   # on c2 / c2_capped, the largest cases


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_v_cycles_match_the_cpu_restatement_bit_for_bit(oracle_mod, monkeypatch, name):
    import hnanosolver_b200 as H

    O = oracle_mod
    w, grid, sim = _gpu(name)
    div = _div_of_advected(O, w)
    assert np.array_equal(sim.aux(0), div)
    mg = _multigrid(grid, name)
    omg = _oracle_mg(O, name)
    fails = []
    for (nu_pre, nu_post), omega in (FEW_SETTINGS if name.startswith("c2") else SETTINGS):
        want, _ = _oracle_cycles(omg, div, 3, nu_pre, nu_post, omega)
        for cycles in (1, 3):
            assert sim.pressure_solve_mg(mg, cycles, 0.0, nu_pre, nu_post, omega) == (cycles, -1.0)
            fails.append(_bits_differ(sim.aux(1), want[cycles - 1], f"{cycles} x V({nu_pre},{nu_post}) omega {omega}"))
    # the same solve with every launch issued directly (no CUDA graph)
    monkeypatch.setenv("HNS_MG_GRAPH", "0")
    direct = H.Multigrid(grid, _case(name)[1])
    sim.pressure_solve_mg(direct, 3, 0.0, 3, 1, 1.15)
    fails.append(_bits_differ(sim.aux(1), _oracle_cycles(omg, div, 3, 3, 1, 1.15)[0][2], "graph off, 3 x V(3,1) omega 1.15"))
    fails = [f for f in fails if f]
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["block4_isolated_first", "soup_capped"])
def test_graph_cache_follows_state_parameters_and_coarsest_iterations(oracle_mod, name):
    O = oracle_mod
    w, grid, a = _gpu(name)
    b = _sim(grid, w, velocity=np.ascontiguousarray(w.velocity[::-1] * np.float32(0.5)))   # another state, another right-hand side
    ix = O.OracleIndex(w.coords)
    rhs = {id(a): _div_of_advected(O, w), id(b): ix.divergence(ix.advect_vector(w.velocity[::-1] * np.float32(0.5), w.dt, w.voxel_size),
                                                                   w.voxel_size)}
    assert np.array_equal(b.aux(0), rhs[id(b)])
    mg = _multigrid(grid, name)
    oracles = {ci: _oracle_mg(O, name, coarsest_iterations=ci) for ci in (8, 32)}
    got = {}
    # (state, nu_pre, nu_post, omega, coarsest iterations): every solve changes one key of the cached graph
    seq = [(a, 2, 2, 1.15, 32), (a, 2, 2, 1.15, 8), (b, 2, 2, 1.15, 8), (b, 1, 0, 1.15, 8), (b, 1, 0, 1.0, 8), (a, 1, 0, 1.0, 8),
           (a, 1, 0, 1.0, 32), (b, 1, 0, 1.0, 32), (b, 0, 1, 1.0, 32), (b, 0, 1, 1.0, 8), (a, 2, 2, 1.15, 8)]
    for s, nu_pre, nu_post, omega, ci in seq:
        mg.set_coarsest_iterations(ci)
        s.pressure_solve_mg(mg, 2, 0.0, nu_pre, nu_post, omega)
        p = s.aux(1)
        want, _, _ = oracles[ci].solve(rhs[id(s)], 2, nu_pre, nu_post, omega)
        assert not _bits_differ(p, want, ""), _bits_differ(p, want, f"state {'ab'[s is b]}, V({nu_pre},{nu_post}) omega {omega}, coarsest {ci}")
        got[(s is b, nu_pre, nu_post, omega, ci)] = p
    # the coarsest iteration count reaches the kernel: 8 and 32 iterations give different pressures
    assert not np.array_equal(got[(False, 2, 2, 1.15, 32)], got[(False, 2, 2, 1.15, 8)])
    assert not np.array_equal(got[(False, 1, 0, 1.0, 8)], got[(False, 1, 0, 1.0, 32)])
    with pytest.raises(Exception):
        mg.set_coarsest_iterations(0)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sphere40", "soup", "block4_isolated_first"])
def test_rel_tol_stops_where_the_restatement_does(oracle_mod, name):
    O = oracle_mod
    w, grid, sim = _gpu(name)
    div = _div_of_advected(O, w)
    mg = _multigrid(grid, name)
    want, rel = _oracle_cycles(_oracle_mg(O, name), div, 5, 2, 2, 1.15)
    # a tolerance between two consecutive residuals (their geometric mean: far from both, so the device's atomically summed norm
    # cannot land on the other side) stops after the second of them
    tried = 0
    for i in range(3):
        if rel[i] < 2 * rel[i + 1]:
            continue
        tried += 1
        cycles, got_rel = sim.pressure_solve_mg(mg, 20, float(np.sqrt(rel[i] * rel[i + 1])), 2, 2, 1.15)
        assert cycles == i + 2
        assert not _bits_differ(sim.aux(1), want[i + 1], ""), _bits_differ(sim.aux(1), want[i + 1], f"rel_tol stop after {i + 2} cycles")
        assert abs(got_rel - rel[i + 1]) <= 1e-6 * rel[i + 1]
    assert tried >= 2
    # a tolerance never reached: exactly max_cycles, and the norm after the last one still the fp64 residual although the solve sits
    # at its fp32 floor (where a residual taken in fp32 comes out percents too small)
    cycles, got_rel = sim.pressure_solve_mg(mg, 5, 1e-12, 2, 2, 1.15)
    assert cycles == 5 and abs(got_rel - rel[4]) <= 1e-6 * rel[4], (got_rel, rel[4])
    assert not _bits_differ(sim.aux(1), want[4], "")
    assert abs(sim.relative_residual() - rel[4]) <= 1e-6 * rel[4]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["block4_isolated_first", "soup_capped"])
def test_frame_with_the_multigrid_solver_is_a_frame(name):
    import hnanosolver_b200 as H

    w, _ = _case(name)
    grid = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    a, b = H.Simulation(grid, len(w.scalars)), H.Simulation(grid, len(w.scalars))
    mg = _multigrid(grid, name)
    for s in (a, b):
        s.upload(w.velocity, w.scalars)
    a.set_pressure_solver(mg, 2, 3, 1, 1.0)
    a.step(40, w.dt)
    b.advect_velocity(w.dt)
    b.divergence(True)
    b.pressure_solve_mg(mg, 2, 0.0, 3, 1, 1.0)
    b.subtract_gradient(True)
    b.advect_scalars(w.dt, 0)
    a.sync(), b.sync()
    assert np.array_equal(a.velocity(), b.velocity()) and np.array_equal(a.aux(1), b.aux(1))
    assert all(np.array_equal(a.scalar(i), b.scalar(i)) for i in range(len(w.scalars)))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(P64_GATE))
def test_device_solve_matches_the_fp64_poisson_solution(oracle_mod, name):
    div, p64, A = _poisson64(oracle_mod, name)
    _, grid, sim = _gpu(name)
    assert np.array_equal(sim.aux(0), div)
    mg = _multigrid(grid, name)
    # four cycles or fewer to 1e-5 (the V-cycle's contraction, which a wrong coarse level would spoil), a residual that scipy confirms
    cycles, rel = sim.pressure_solve_mg(mg, 20, 1e-5, 2, 2, 1.15)
    rel64, err = _against_p64(A, div, p64, sim.aux(1))
    assert cycles <= 4 and rel <= 1e-5 and rel64 <= 1e-5 and err <= P64_GATE[name][0], (cycles, rel, rel64, err)
    assert abs(rel64 - sim.relative_residual()) <= 1e-6 * rel64
    # converged: the fp64 solution up to fp32 rounding (a wrong sign, dx scaling or boundary condition would be off by far more)
    sim.pressure_solve_mg(mg, 8, 0.0, 2, 2, 1.15)
    assert _against_p64(A, div, p64, sim.aux(1))[1] <= P64_GATE[name][1]
