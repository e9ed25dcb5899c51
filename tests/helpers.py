"""Shared helpers of the parity tests."""
import importlib.util
import os

import numpy as np
import pytest

from oracle import oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
_spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLDEN, "make_golden.py"))
make_golden = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(make_golden)

# Tolerance of the north star: advected / projected fields within 1e-5 relative of the reference kernels.
# "Relative" is measured against the field's max magnitude (a voxel-wise relative error is meaningless at zero crossings).
REL_TOL = 1e-5


def rel_err(a, b) -> float:
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(1e-30, np.abs(b).max()))


def assert_close(a, b, what, tol=REL_TOL, exact=True):
    """The north star's tolerance (1e-5 of the field's magnitude) is the contract; what the product actually delivers -- and what
    DESIGN.md claims -- is equality float for float with the oracle and with the reference's own kernels, so that is asserted too
    (`exact`; +0.0 == -0.0). A one-ulp regression in a kernel rewrite fails here, not three orders of magnitude later."""
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, what
    e = rel_err(a, b)
    assert e <= tol, f"{what}: relative error {e:.3e} > {tol:.1e}"
    if exact:
        bad = a != b
        if bad.any():
            ulp = np.abs(a.astype(np.float32).view(np.int32).astype(np.int64) - b.astype(np.float32).view(np.int32).astype(np.int64))[bad]
            raise AssertionError(f"{what}: {int(bad.sum())} of {a.size} values differ bitwise (max {int(ulp.max())} ulp, relative error {e:.3e})")


# Byte ranges of the NanoVDB buffer that voxelsToGrid leaves uninitialised (SURVEY.md Appendix C): grid name bytes 1..255,
# RootData tail padding, root-tile tail (state padding + value). Everything else must be bit-identical.
def nanovdb_compare_mask(nbytes: int, num_tiles: int) -> np.ndarray:
    m = np.ones(nbytes, bool)
    m[41:296] = False                       # GridData::mGridName[1..255]
    root = 672 + 64
    m[root + 28:root + 32] = False          # padding after mTableSize
    m[root + 72:root + 96] = False          # RootData tail padding
    for t in range(num_tiles):
        tile = root + 96 + 32 * t
        m[tile + 20:tile + 32] = False      # padding after state + the untouched tile value
    return m


class Golden:
    """One fixture of tests/golden (make_golden.compact): the reference's inputs, regenerated and checked against their digests, and
    its outputs, each held as values at a sample of voxels plus the SHA-256 of the whole array."""

    def __init__(self, name: str):
        z = np.load(os.path.join(GOLDEN, f"ref_{name}.npz"))
        self._z = {k: z[k] for k in z.files}
        self._arrays = {k: v for k, v in self._z.items() if "." not in k}
        for k, v in make_golden.case_arrays(name).items():
            assert make_golden.digest(v) == self.sha256(k), f"regenerated input {k} is not the one the reference was given"
            self._arrays[k] = v

    def __contains__(self, key: str) -> bool:
        return key in self._arrays or key + ".sha256" in self._z

    def __getitem__(self, key: str) -> np.ndarray:
        """a parameter, the index grid or an input; outputs are only compared, through check / matches"""
        return self._arrays[key]

    def sha256(self, key: str) -> str:
        return str(self._z[key + ".sha256"])

    def matches(self, a, key: str) -> bool:
        """`a` equals output `key` value for value (+0.0 == -0.0)"""
        return make_golden.digest(a) == self.sha256(key)

    def check(self, a, key: str, what: str):
        """assert_close of `a` and output `key` on the stored sample of voxels, then bitwise equality of the whole array"""
        a = np.asarray(a)
        assert_close(a[self._z["sample_index"]], self._z[key + ".sample"], what)
        assert self.matches(a, key), f"{what}: equal on the sample of {self._z['sample_index'].size} voxels but not everywhere (SHA-256 differs)"


class Recording:
    """Outputs of the reference's own kernels and launchers by key (tests/golden/ref_recorded.npz), each held as its values at a seeded
    sample of rows plus the SHA-256 of the whole array, and per key the digest of the inputs they were computed from.

    With HNS_RECORD_REFERENCE=1 and the reference build present (oracle/_ref), `record` stores the reference's own output and `save`
    merges what a run recorded into the file. The file as committed was recorded on a B200 from this project's CUDA path at a state
    whose kernels, input generator and test inputs equal those of commit a7bb57e, where every one of these comparisons had passed bit
    for bit against the live reference (profiles/r2f_gpu_tests_final.log). Its vorticity outputs for the two cases the golden fixtures
    share (random28 = soup, sphere32 = sphere) agree bit for bit with those fixtures, which come from the reference itself."""

    SAMPLE = 32

    def __init__(self, path: str):
        self.path = path
        self.recording = os.environ.get("HNS_RECORD_REFERENCE") == "1"
        self._z = {}
        if os.path.exists(path):
            z = np.load(path)
            self._z = {k: z[k] for k in z.files}

    @classmethod
    def _rows(cls, n: int) -> np.ndarray:
        return np.sort(np.random.default_rng(7).choice(n, min(n, cls.SAMPLE), replace=False))

    @staticmethod
    def _inputs_digest(arrays) -> str:
        return make_golden.digest(np.array([make_golden.digest(a) for a in arrays]))

    def record_inputs(self, key: str, arrays):
        self._z[key + "/inputs.sha256"] = np.array(self._inputs_digest(arrays))

    def record(self, want, key: str):
        want = np.asarray(want)
        self._z[key + ".sample"], self._z[key + ".sha256"] = want[self._rows(len(want))], np.array(make_golden.digest(want))

    def check_inputs(self, key: str, arrays):
        """the recorded outputs under `key` apply only to the inputs they were computed from"""
        assert key + "/inputs.sha256" in self._z, f"no recorded reference outputs for {key}"
        assert self._inputs_digest(arrays) == str(self._z[key + "/inputs.sha256"]), \
            f"{key}: the inputs differ from those the recorded reference outputs were computed from (input generator or numpy changed)"

    def check(self, a, key: str, what: str):
        a = np.asarray(a)
        idx = self._rows(len(a))
        assert key + ".sha256" in self._z, f"{what}: no recorded reference output {key}"
        assert_close(a[idx], self._z[key + ".sample"], what)
        assert make_golden.digest(a) == str(self._z[key + ".sha256"]), \
            f"{what}: equal on the sample of {idx.size} rows but not everywhere (SHA-256 differs)"

    def save(self):
        np.savez_compressed(self.path, **self._z)


RECORDED = Recording(os.path.join(GOLDEN, "ref_recorded.npz"))


class Reference:
    """The reference's outputs under `key` (test, case, parameters) for `inputs`: `live()` runs its own kernels and launchers when their
    build is present (and, with HNS_RECORD_REFERENCE=1, records what they return); otherwise the recording of what they computed from
    the same inputs stands in (Recording). A module that builds one saves RECORDED when it is done recording."""

    def __init__(self, key: str, live, inputs):
        self.key, self.want = key, None
        if O.ref_gpu_available():
            self.want = live()
            if RECORDED.recording:
                RECORDED.record_inputs(key, inputs)
        elif RECORDED.recording:
            pytest.fail("recording the reference's outputs needs its build (oracle/_ref/libhns_ref.so)")
        else:
            RECORDED.check_inputs(key, inputs)

    def check(self, got, name: str, what: str):
        if self.want is None:
            RECORDED.check(got, f"{self.key}/{name}", what)
            return
        assert_close(got, self.want[name], what)
        if RECORDED.recording:
            RECORDED.record(self.want[name], f"{self.key}/{name}")


def cube(n, off=(0, 0, 0)) -> np.ndarray:
    """origins of the n[0] x n[1] x n[2] block of leaves whose first leaf lies at `off`"""
    ax = [np.arange(k) * 8 + o for k, o in zip(n, off)]
    return np.stack(np.meshgrid(*ax, indexing="ij"), -1).reshape(-1, 3).astype(np.int32)


def _nanovdb_sorted(o) -> np.ndarray:
    from hnanosolver_b200 import synth

    o = np.asarray(o, np.int32).reshape(-1, 3)
    return np.ascontiguousarray(o[synth.nanovdb_order(o)])


def _three_blobs():
    return _nanovdb_sorted(np.concatenate([cube((4, 4, 4), off) for off in ((0, 0, 0), (512, 0, 0), (0, 512, 0))]))


def _diagonal():
    i = np.arange(12)
    steps = np.stack([8 * i] * 3, 1)
    side = np.array([[8 * k + 8, 8 * k, 8 * k] for k in (0, 3, 6, 9)])
    return _nanovdb_sorted(np.concatenate([steps, side]))


def _multitile_negative():
    from hnanosolver_b200 import synth

    soup = synth.random_leaves(60, 5, 3, offset=(-24, 4080, -16), with_coords=False).origins
    return _nanovdb_sorted(np.concatenate([soup, cube((3, 2, 2), (-4112, -8, -8))]))


# Partitions of the sharded frame (hnanosolver_b200/dist.py make_plan, csrc/dist.cu) chosen so that together they reach every branch
# of its plan and ghost-exchange protocol. name -> (global leaf origins in NanoVDB order, worlds, what each world reaches). The reach
# is restated by partition_reach below and pinned by tests/test_sharded_partitions.py, so a change of make_plan that stops reaching
# a branch fails there instead of silently testing less. Reach keys:
#   pipelined  ranks without boundary leaves (they run pipelined_sweeps beside peers that run the fused pressure pipeline)
#   no_interior  ranks without interior leaves (every owned leaf goes through the boundary / push path)
#   no_push  ranks with a send list whose every entry has push mask 0 (an empty push CSR, yet they signal every flag)
#   send_only / recv_only  (rank, peer) pairs where the rank only sends to / only receives from the peer
#   push_kinds  the push mask kinds of all send-list entries: "none", "xy" (x / y faces only), "z" (a z face)
#   all_to_all  every rank has every other rank as a peer
#   root_tiles / negative  root tiles (4096^3) the domain spans / whether it has negative coordinates
#   leaf0_alone  global leaf 0 is the only leaf of its root tile
PARTITIONS = {
    "three_blobs": (_three_blobs, {
        # rank 0 runs the fused pipeline and its only boundary leaf (leaf 0, held by every rank) touches nobody across a face; ranks 1
        # and 2 only receive leaf 0 and run pipelined_sweeps
        3: dict(pipelined=[1, 2], no_interior=[], no_push=[0], send_only=[(0, 1), (0, 2)], recv_only=[(1, 0), (2, 0)],
                push_kinds={"none"}, all_to_all=False),
        2: dict(pipelined=[], no_interior=[], no_push=[], send_only=[], recv_only=[], push_kinds={"none", "xy"}, all_to_all=True),
    }),
    "block8": (lambda: cube((2, 2, 2)), {
        2: dict(pipelined=[], no_interior=[0, 1], no_push=[], send_only=[], recv_only=[], push_kinds={"xy"}, all_to_all=True),
        3: dict(pipelined=[], no_interior=[0, 1, 2], no_push=[], send_only=[], recv_only=[], push_kinds={"none", "xy", "z"}, all_to_all=True),
        4: dict(pipelined=[], no_interior=[0, 1, 2, 3], no_push=[], send_only=[], recv_only=[], push_kinds={"none", "xy"}, all_to_all=True),
    }),
    "diagonal": (_diagonal, {
        # edge and corner contacts only: at 2 ranks no send-list leaf is pushed
        2: dict(pipelined=[], no_interior=[], no_push=[0, 1], send_only=[], recv_only=[], push_kinds={"none"}, all_to_all=True),
        3: dict(pipelined=[], no_interior=[], no_push=[2], send_only=[(0, 2)], recv_only=[(2, 0)], push_kinds={"none", "xy"}, all_to_all=True),
    }),
    "multitile_negative": (_multitile_negative, {
        3: dict(pipelined=[], no_interior=[], no_push=[], send_only=[], recv_only=[], push_kinds={"none", "xy"}, all_to_all=True),
        4: dict(pipelined=[], no_interior=[], no_push=[], send_only=[], recv_only=[], push_kinds={"none", "xy", "z"}, all_to_all=True),
    }),
    "isolated_leaf0": (lambda: _nanovdb_sorted(np.concatenate([[[-4096, -4096, -4096]], cube((6, 4, 4))])), {
        2: dict(pipelined=[], no_interior=[], no_push=[], send_only=[], recv_only=[], push_kinds={"none", "xy", "z"}, all_to_all=True),
        4: dict(pipelined=[], no_interior=[1, 2], no_push=[], send_only=[(0, 2), (0, 3)], recv_only=[(2, 0), (3, 0)],
                push_kinds={"none", "xy", "z"}, all_to_all=False),
    }),
    "too_few": (lambda: np.array([[0, 0, 0], [8, 0, 0]], np.int32), {3: None}),   # fewer leaves than ranks: make_plan refuses
}
# properties of the whole domain: (leaves, root tiles, negative coordinates, leaf 0 alone in its root tile)
PARTITION_DOMAINS = {
    "three_blobs": (192, 1, False, False),
    "block8": (8, 1, False, False),
    "diagonal": (16, 1, False, False),
    "multitile_negative": (72, 14, True, False),
    "isolated_leaf0": (97, 2, True, True),
    "too_few": (2, 1, False, False),
}


def partition_origins(name: str) -> np.ndarray:
    return PARTITIONS[name][0]()


def partition_domain(origins):
    """(leaves, root tiles, negative coordinates, leaf 0 alone in its root tile)"""
    o = np.asarray(origins, np.int64)
    tiles = o >> 12
    return (int(o.shape[0]), int(np.unique(tiles, axis=0).shape[0]), bool((o < 0).any()),
            bool(o.shape[0] > 0 and int((tiles == tiles[0]).all(1).sum()) == 1))


_FACES = ((-8, 0, 0), (8, 0, 0), (0, -8, 0), (0, 8, 0), (0, 0, -8), (0, 0, 8))   # hns_dist_ipc_finish's face bits 0..5


def rank_reach(origins, plans):
    """Per rank, restated from hns_dist_set_plan (owned = boundary, which some send list names, + interior) and hns_dist_ipc_finish
    (push mask of a send-list entry: the faces of the leaf whose neighbour the peer owns; kind "z" if a z face is among them, "xy" if
    only x / y faces, "none" if it touches the peer only across edges and corners). Returns a list of dicts: boundary, interior,
    send_only, recv_only (peer ranks), kinds ({peer: [kind per send-list entry]})."""
    o = np.asarray(origins, np.int64)
    lut = {tuple(v): i for i, v in enumerate(o.tolist())}
    world = len(plans)
    owner = np.empty(o.shape[0], np.int64)
    for p in plans:
        owner[p.local_ids[p.owned_local]] = p.rank
    out = []
    for p in plans:
        owned = p.local_ids[p.owned_local]
        sent = set()
        kinds = {}
        for q, ids in p.send.items():
            g = p.local_ids[ids]
            sent.update(g.tolist())
            ks = []
            for leaf in g.tolist():
                mask = 0
                for f, d in enumerate(_FACES):
                    nb = lut.get((o[leaf][0] + d[0], o[leaf][1] + d[1], o[leaf][2] + d[2]))
                    if nb is not None and owner[nb] == q:
                        mask |= 1 << f
                ks.append("none" if not mask else "z" if mask & 0x30 else "xy")
            kinds[q] = ks
        snd = {q for q, v in p.send.items() if len(v)}
        rcv = {q for q, v in p.recv.items() if len(v)}
        out.append(dict(boundary=sum(1 for l in owned.tolist() if l in sent), interior=sum(1 for l in owned.tolist() if l not in sent),
                        send_only=sorted(snd - rcv), recv_only=sorted(rcv - snd), kinds=kinds, peers=sorted(snd | rcv)))
        assert world == p.world
    return out


def partition_reach(origins, plans) -> dict:
    """what a partition reaches, in the keys of PARTITIONS' rows"""
    rr = rank_reach(origins, plans)
    world = len(plans)
    return dict(pipelined=[r for r, x in enumerate(rr) if x["boundary"] == 0],
                no_interior=[r for r, x in enumerate(rr) if x["interior"] == 0],
                no_push=[r for r, x in enumerate(rr) if x["kinds"] and all(k == "none" for ks in x["kinds"].values() for k in ks)],
                send_only=[(r, q) for r, x in enumerate(rr) for q in x["send_only"]],
                recv_only=[(r, q) for r, x in enumerate(rr) for q in x["recv_only"]],
                push_kinds={k for x in rr for ks in x["kinds"].values() for k in ks},
                all_to_all=all(x["peers"] == [q for q in range(world) if q != r] for r, x in enumerate(rr)))


def combustion_fields(n, seed=123):
    """fuel / waste / temperature / flame of the small cases: fuel in about 40 % of the voxels, element 0 zero"""
    rng = np.random.default_rng(seed)
    f = dict(fuel=(rng.random(n) * (rng.random(n) < 0.4)).astype(np.float32), waste=(0.3 * rng.random(n)).astype(np.float32),
             temperature=rng.random(n).astype(np.float32), flame=(0.2 * rng.random(n)).astype(np.float32))
    for a in f.values():
        a[0] = 0.0
    return f
