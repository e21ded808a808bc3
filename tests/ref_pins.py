"""Stored outputs of the reference's own code, for the tests that pin the oracle, the host mirror of FrontierFinder and
the fused map to it without needing the reference on the machine that runs them.

tools/make_ref_pins.py runs every case a test module lists in its REF_PINS table ({name: (function, [argument tuples])})
against oracle/_ref/libfuel_ref.so (the reference's sdf_map.cpp, raycast.cpp, bspline_optimizer.cpp,
frontier_finder.cpp and perception_utils.cpp compiled unmodified, see oracle/Makefile) and writes what each returns to
tests/golden/ref_pins.npz.  An array of at most FULL_BYTES is stored whole; a larger one as its shape, the SHA-256 of
its canonical bytes and a fixed sample of its elements, so every comparison stays exact over the whole array while the
file stays small.  Canonical form: integers as int64, floats as float64 with one NaN and no negative zero (the tests
compare with ==, under which -0.0 == 0.0, and treat NaN as equal to NaN).

File layout (one row per stored array, rows sorted by key): keys (bytes), kind (bit 0: float, bit 1: digest),
shape (padded with -1), start (offset of the row's values in `floats` or `ints`: the whole array, or the sample),
sha256 (zero for arrays stored whole)."""
import hashlib
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_pins.npz")
FULL_BYTES = 256
N_SAMPLE = 8
MAX_NDIM = 4

_data = None


def canonical(a):
    a = np.asarray(a)
    if a.dtype == bool:
        a = a.astype(np.uint8)
    if a.dtype.kind == "f":
        a = a.astype(np.float64)
        a = np.where(np.isnan(a), np.nan, a + 0.0)
    elif a.dtype.kind in "iu":
        a = a.astype(np.int64)
    else:
        raise TypeError("no canonical form for dtype %s" % a.dtype)
    return np.ascontiguousarray(a)


def digest(a):
    return np.frombuffer(hashlib.sha256(a.tobytes()).digest(), np.uint8)


def sample_index(size):
    return np.sort(np.random.default_rng(size).choice(size, min(N_SAMPLE, size), replace=False))


def _same(a, b):
    eq = a == b
    if a.dtype.kind == "f" and b.dtype.kind == "f":
        eq |= np.isnan(a) & np.isnan(b)
    return eq


def case_prefix(module, name, table, args):
    """args must be one of the argument tuples table[name] lists"""
    return "%s/%s/%d" % (module, name, table[name][1].index(tuple(args)))


def pack(prefix, outputs):
    """{name: array-like} -> {key: canonical array} of one case"""
    return {prefix + "/" + k: canonical(v) for k, v in outputs.items()}


def save(arrays, path=PATH):
    keys = sorted(arrays)
    kind = np.zeros(len(keys), np.int8)
    shape = np.full((len(keys), MAX_NDIM), -1, np.int64)
    start = np.zeros(len(keys), np.int64)
    sha = np.zeros((len(keys), 32), np.uint8)
    vals = {"f": [], "i": []}
    size = {"f": 0, "i": 0}
    for j, k in enumerate(keys):
        a = arrays[k]
        t = "f" if a.dtype.kind == "f" else "i"
        shape[j, :a.ndim] = a.shape
        v = a.reshape(-1)
        if a.nbytes > FULL_BYTES:
            kind[j] = 2
            sha[j] = digest(a)
            v = v[sample_index(v.size)]
        kind[j] |= t == "f"
        start[j] = size[t]
        vals[t].append(v)
        size[t] += v.size
    np.savez_compressed(path, keys=np.array([k.encode() for k in keys]), kind=kind, shape=shape, start=start, sha256=sha,
                        floats=np.concatenate(vals["f"] or [np.zeros(0)]),
                        ints=np.concatenate(vals["i"] or [np.zeros(0, np.int64)]))


def _load(path=PATH):
    with np.load(path) as z:
        f = {k: z[k] for k in z.files}
    out = {}
    for j, k in enumerate(f["keys"]):
        shape = tuple(int(s) for s in f["shape"][j] if s >= 0)
        size = int(np.prod(shape, dtype=np.int64))
        whole = not f["kind"][j] & 2
        n = size if whole else len(sample_index(size))
        pool = f["floats"] if f["kind"][j] & 1 else f["ints"]
        v = pool[f["start"][j]:f["start"][j] + n]
        out[k.decode()] = (shape, v.reshape(shape) if whole else v, None if whole else f["sha256"][j])
    return out


class Pinned:
    """The stored outputs of one case.  check(key, got) asserts that `got` equals what the reference returned."""

    def __init__(self, data, prefix):
        self.data, self.prefix = data, prefix

    def check(self, key, got, what=""):
        k = self.prefix + "/" + key
        assert k in self.data, "no stored reference output %s (tools/make_ref_pins.py)" % k
        shape, want, sha = self.data[k]
        a = canonical(got)
        label = "%s%s" % (key, (" (%s)" % what) if what else "")
        assert a.shape == shape, "%s: shape %s, the reference's %s" % (label, a.shape, shape)
        assert a.dtype == want.dtype, "%s: %s values, the reference's are %s" % (label, a.dtype, want.dtype)
        if sha is None:
            nbad = int((~_same(a, want)).sum())
            assert nbad == 0, "%s: %d of %d elements differ from the reference's" % (label, nbad, a.size)
            return
        nbad = int((~_same(a.reshape(-1)[sample_index(a.size)], want)).sum())
        assert nbad == 0, "%s: %d of %d sampled elements differ from the reference's" % (label, nbad, len(want))
        assert np.array_equal(digest(a), sha), "%s differs from the reference's (SHA-256 of the whole array)" % label


def load(module, name, table, args=()):
    global _data
    if _data is None:
        _data = _load()
    return Pinned(_data, case_prefix(module, name, table, args))
