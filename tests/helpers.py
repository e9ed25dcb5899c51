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


def combustion_fields(n, seed=123):
    """fuel / waste / temperature / flame of the small cases: fuel in about 40 % of the voxels, element 0 zero"""
    rng = np.random.default_rng(seed)
    f = dict(fuel=(rng.random(n) * (rng.random(n) < 0.4)).astype(np.float32), waste=(0.3 * rng.random(n)).astype(np.float32),
             temperature=rng.random(n).astype(np.float32), flame=(0.2 * rng.random(n)).astype(np.float32))
    for a in f.values():
        a[0] = 0.0
    return f
