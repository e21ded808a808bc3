"""Every launch form of the ESDF tile transform (esdf_tile.cu) against the oracle of SDFMap::updateESDF3d, voxel for
voxel, to the exact squared voxel distance (tests.helpers.assert_esdf_exact).

The transform picks its kernels from the box: the z-pack is vectorised or scalar, each tile pass (K1: the y lines of
the zy tiles, K2: the x lines) runs 32- or 64-sample bands in a CTA of 256, 512 or 1024 threads or a 2-CTA cluster,
and the hand-over is cut into chunks of Wc z words.  `forms` restates that choice; `test_cases_cover_every_form`
(CPU) checks that the cases below reach every (pass, form) pair in every site mode, and every GPU case checks the
launch count, which shows the intended chunking ran.  FUELGPU_ESDF_BAND / FUELGPU_ESDF_CLUSTER are read once per
process, so those forms run in child processes."""
import os
import subprocess
import sys

import numpy as np
import pytest

from fuel_b200 import workloads as W
from tests.helpers import ESDF_EXACT_STATS, assert_esdf_exact, make_sdf_map, orc_grid

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RES = 0.1

# mode -> (optimistic, signed); the site modes of the z sweep it runs (esdf.cu esdf_update_impl: 0 optimistic,
# 1 unknown counts as a site, 2 the negative field of signed mode)
MODES = {"opt": (True, False), "nonopt": (False, False), "signed": (True, True)}
SITE_MODES = {"opt": (0,), "nonopt": (1,), "signed": (0, 2)}


# ---- the form choice, restated ------------------------------------------------------------------------------------
def zpack_form(n, lo, hi):
    """launch_zpack (esdf_tile.cu:194-208): 16-byte loads when the box's z range is whole words on a 16-byte
    boundary (one GPU: chunk_stride = 0)"""
    nzb = hi[2] - lo[2] + 1
    base0 = (lo[0] * n[1] + lo[1]) * n[2] + lo[2]
    return "vec" if nzb % 32 == 0 and n[2] % 16 == 0 and base0 % 16 == 0 else "scalar"


def tile_form(length, band=32, cluster=True):
    """launch_tile (esdf_tile.cu:687-748) for a pass over lines of `length` samples -> (band width, threads per CTA,
    2-CTA cluster).  One GPU: K2's piece_rows is 1 << 20, a multiple of 64, so both passes choose alike."""
    logm = 6 if length > 128 and band == 64 else 5
    nb = -(-length // (1 << logm))
    if logm == 5 and nb > 16 and cluster:
        return (32, 512, True)
    if logm == 5:
        return (32, 256 if nb <= 8 else 512 if nb <= 16 else 1024, False)
    return (64, 256 if nb <= 8 else 512, False)


def chunking(n, lo, hi):
    """(Wc, chunks): esdf_tile_scratch_sizes (esdf_tile.cu:756-767) sizes the two P buffers from the map,
    esdf_tile_transform (:793-801) cuts the box's NW z words into chunks of Wc"""
    def wc_of(nx, ny, nw, cap=None):
        per_word = nx * ny * 128
        w = nw
        if per_word * nw > 48 << 20:
            w = max(1, (32 << 20) // per_word)
        if cap is not None and per_word * w > cap:
            w = cap // per_word
        return w, per_word * w
    _, p_bytes = wc_of(n[0], n[1], -(-n[2] // 32))
    ext = [hi[i] - lo[i] + 1 for i in range(3)]
    nw = -(-ext[2] // 32)
    wc, _ = wc_of(ext[0], ext[1], nw, p_bytes)
    return wc, -(-nw // wc)


def forms(n, lo, hi, band=32, cluster=True):
    ext = [hi[i] - lo[i] + 1 for i in range(3)]
    return dict(zpack=zpack_form(n, lo, hi), zy=tile_form(ext[1], band, cluster), x=tile_form(ext[0], band, cluster),
                chunks=chunking(n, lo, hi))


def launches(n, lo, hi, mode):
    """zpack + (zy, x) per chunk; signed mode runs two transforms and the merge"""
    t = 1 + 2 * chunking(n, lo, hi)[1]
    return 2 * t + 1 if MODES[mode][1] else t


# ---- the cases ----------------------------------------------------------------------------------------------------
TILE_N = [1, 31, 32, 33, 255, 256, 257, 300, 481, 511, 512, 513, 1023, 1024]
ZPACK_NZ = [32, 64, 96, 160, 224]
CHUNK_MAPS = [((256, 256, 320), None), ((256, 256, 256), None), ((256, 256, 576), None),
              ((256, 256, 320), ((0, 0, 17), (255, 255, 318)))]
ENV = {"cluster0": dict(FUELGPU_ESDF_CLUSTER="0"), "band64": dict(FUELGPU_ESDF_BAND="64")}
ENV_N = {"cluster0": [513, 545, 700, 1023, 1024], "band64": [129, 200, 256, 300, 511, 512, 513, 1023, 1024]}


def line_shape(axis, n, z):
    return (n, 7, z) if axis == "x" else (7, n, z)


def full_box(shape):
    return (0, 0, 0), tuple(s - 1 for s in shape)


def zpack_boxes(nz):
    """full box; a box at z = 16 with whole words (vectorised); z from 3 and a box of partial words (scalar)"""
    out = [("full", (0, 0, 0), (8, 11, nz - 1))]
    if nz >= 64:
        out.append(("lo16", (1, 2, 16), (7, 10, 16 + 32 * ((nz - 16) // 32) - 1)))
    out.append(("lo3", (1, 2, 3), (7, 10, nz - 1)))
    out.append(("part", (0, 1, 0), (8, 11, nz - 6)))
    return out


def all_cases():
    """(group, id, shape, lo, hi, mode, env) of every case below"""
    cases = []
    for axis in "xy":
        for n in TILE_N:
            for z in (64, 40):
                for mode in MODES:
                    s = line_shape(axis, n, z)
                    cases.append(("tile", "%s%d-z%d-%s" % (axis, n, z, mode), s) + full_box(s) + (mode, None))
    for nz in ZPACK_NZ:
        for name, lo, hi in zpack_boxes(nz):
            for mode in MODES:
                cases.append(("zpack", "nz%d-%s-%s" % (nz, name, mode), (9, 12, nz), lo, hi, mode, None))
    for s, box in CHUNK_MAPS:
        lo, hi = box or full_box(s)
        for mode in ("opt", "signed"):
            cases.append(("chunk", "%dx%dx%d-z%d-%s" % (s + (lo[2], mode)), s, lo, hi, mode, None))
    for env, ns in ENV_N.items():
        for axis in "xy":
            for n in ns:
                for mode in MODES:
                    s = line_shape(axis, n, 64)
                    cases.append(("env", "%s-%s%d-%s" % (env, axis, n, mode), s) + full_box(s) + (mode, env))
    return cases


def test_cases_cover_every_form():
    """every (pass, form) pair of the launchers runs in every site mode; the chunk cases reach Wc > 1 with a partial
    last chunk and three or more chunks"""
    want = {("zpack", f) for f in ("vec", "scalar")}
    for band, cluster in ((32, True), (32, False), (64, True)):
        for n in range(1, 1025):
            want |= {(p, tile_form(n, band, cluster)) for p in ("zy", "x")}
    assert len(want) == 2 + 2 * 6
    seen = {}
    chunkings = set()
    for group, cid, shape, lo, hi, mode, env in all_cases():
        e = ENV.get(env, {})
        f = forms(shape, lo, hi, band=int(e.get("FUELGPU_ESDF_BAND", 32)),
                  cluster=e.get("FUELGPU_ESDF_CLUSTER", "1") != "0")
        for key in (("zpack", f["zpack"]), ("zy", f["zy"]), ("x", f["x"])):
            seen.setdefault(key, set()).update(SITE_MODES[mode])
        chunkings.add((f["chunks"], MODES[mode][1]))
    assert set(seen) == want
    for key, modes in seen.items():
        assert modes == {0, 1, 2}, (key, modes)
    # (Wc, chunks): 4, 4, 2 / 4, 4 / 4, 4, 4, 4, 2 words, in both unsigned and signed mode
    for ch in ((4, 3), (4, 2), (4, 5)):
        assert (ch, False) in chunkings and (ch, True) in chunkings
    assert forms((256, 256, 320), (0, 0, 17), (255, 255, 318))["zpack"] == "scalar"


# ---- scenes -------------------------------------------------------------------------------------------------------
def line_scene(shape, axis, dense, seed):
    """dense: 30 % sites and 20 % unknown voxels at random.  sparse: a few sites in the first third of the line axis
    only (the rest of the line, and whole planes across it, have none: long distances, +inf rows in the partial) and
    an unknown slab across 40-60 % of the line axis"""
    rng = np.random.default_rng(seed)
    ax = 0 if axis == "x" else 1
    if dense:
        inflate = (rng.random(shape) < 0.3).astype(np.int8)
        unknown = rng.random(shape) < 0.2
    else:
        inflate = np.zeros(shape, dtype=np.int8)
        lim = max(1, shape[ax] // 3)
        for _ in range(3):
            p = [rng.integers(0, s) for s in shape]
            p[ax] = rng.integers(0, lim)
            inflate[tuple(p)] = 1
        unknown = np.zeros(shape, dtype=bool)
        sl = [slice(None)] * 3
        sl[ax] = slice(int(0.4 * shape[ax]), max(int(0.6 * shape[ax]), int(0.4 * shape[ax]) + 1))
        unknown[tuple(sl)] = True
    tri = np.full(shape, W.FREE, dtype=np.uint8)
    tri[unknown] = W.UNKNOWN
    tri[(inflate == 1) & ~unknown] = W.OCCUPIED
    return inflate, tri


def block_scene(shape, seed, p_site=0.0005, blocks=12):
    """sparse random sites, inflated blocks (the negative field has depth) and unknown blobs"""
    rng = np.random.default_rng(seed)
    inflate = (rng.random(shape) < p_site).astype(np.int8)
    for _ in range(blocks):
        c = [rng.integers(0, s) for s in shape]
        e = [rng.integers(2, max(3, s // 8)) for s in shape]
        inflate[c[0]:c[0] + e[0], c[1]:c[1] + e[1], c[2]:c[2] + e[2]] = 1
    tri = np.full(shape, W.FREE, dtype=np.uint8)
    tri[rng.random(shape) < 0.2] = W.UNKNOWN
    tri[inflate == 1] = W.OCCUPIED
    return inflate, tri


def run_case(fuel, orc, g, m, inflate, tri, lo, hi, mode, threads=8):
    """one update of box [lo, hi] in `mode` on map m (already holding inflate/tri); returns the device field after it"""
    before = m.download().copy()
    m.optimistic_, m.signed_dist_ = MODES[mode]
    m.local_bound_min_, m.local_bound_max_ = np.array(lo, np.int32), np.array(hi, np.int32)
    c0 = m.launch_count()
    m.updateESDF3d()
    assert m.launch_count() - c0 == launches(g.n, lo, hi, mode)
    got = m.download().copy()
    check_case(orc, g, inflate, tri, lo, hi, mode, got, before, threads)
    return got


def check_case(orc, g, inflate, tri, lo, hi, mode, got, before, threads=8):
    opt, signed = MODES[mode]
    ref = orc.update_esdf3d(orc_grid(orc, g), inflate, tri, lo, hi, opt, signed, dist=before.astype(np.float64),
                            threads=threads)
    assert_esdf_exact(got, ref, g.res, box=(lo, hi), signed=signed)
    outside = np.ones(g.n, dtype=bool)
    outside[lo[0]:hi[0] + 1, lo[1]:hi[1] + 1, lo[2]:hi[2] + 1] = False
    assert np.array_equal(got[outside], before[outside])  # bit for bit


@pytest.fixture(scope="module", autouse=True)
def exact_report():
    ESDF_EXACT_STATS.update(max_dev=0.0, voxels=0)
    yield
    print("\n[esdf forms] largest |(got/res)^2 - N_ref| = %.4f over %d voxel comparisons"
          % (ESDF_EXACT_STATS["max_dev"], ESDF_EXACT_STATS["voxels"]))


# ---- tile lengths -------------------------------------------------------------------------------------------------
def case_params(group):
    """the GPU tests run the very cases test_cases_cover_every_form checks"""
    return [pytest.param(*c[2:], id=c[1]) for c in all_cases() if c[0] == group]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,lo,hi,mode,env", case_params("tile"))
def test_tile_lengths(fuel, orc, shape, lo, hi, mode, env):
    """lines of n samples along x (K2) or y (K1): every band count, partial last bands, every CTA form; z = 64 takes
    the vectorised z-pack, z = 40 the scalar one"""
    axis, n, z = ("x", shape[0], shape[2]) if shape[1] == 7 else ("y", shape[1], shape[2])
    g = W.Grid(shape, (0.0, 0.0, 0.0), RES)
    m = fuel.SDFMap(shape, RES, (0.0, 0.0, 0.0), optimistic=True)
    try:
        for dense in (True, False):
            inflate, tri = line_scene(shape, axis, dense, seed=n * 7 + z + (0 if dense else 1))
            m.occupancy_buffer_inflate_[...] = inflate
            m.setOccupancyBuffer(tristate=tri)
            m.upload()
            run_case(fuel, orc, g, m, inflate, tri, lo, hi, mode)
    finally:
        m.close()


# ---- the z-pack ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("nz", ZPACK_NZ)
def test_zpack_boxes(fuel, orc, nz, mode):
    """NW = 1, 2, 3, 5, 7 words per line (3, 5, 7: lane groups with idle lanes); boxes that keep the 16-byte loads and
    boxes that do not, on one map in turn (voxels outside each box keep their value)"""
    shape = (9, 12, nz)
    g = W.Grid(shape, (0.0, 0.0, 0.0), RES)
    inflate, tri = block_scene(shape, seed=nz, p_site=0.01, blocks=4)
    m = make_sdf_map(fuel, g, inflate, tri)
    try:
        kinds = []
        for name, lo, hi in zpack_boxes(nz):
            kinds.append(zpack_form(shape, lo, hi))
            run_case(fuel, orc, g, m, inflate, tri, lo, hi, mode)
        assert "vec" in kinds and "scalar" in kinds
    finally:
        m.close()


# ---- chunked hand-over --------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("shape,lo,hi,mode,env", case_params("chunk"))
def test_chunked_handover(fuel, orc, shape, lo, hi, mode, env):
    """Wc = 4 words per chunk: 4+4+2 (partial last chunk), 4+4, 4+4+4+4+2 (five chunks over the two streams), and a
    box z in [17, 318] (scalar z-pack, output offset, padding lane of the last word)"""
    g = W.Grid(shape, (0.0, 0.0, 0.0), RES)
    inflate, tri = block_scene(shape, seed=shape[2] + lo[2])
    m = make_sdf_map(fuel, g, inflate, tri)
    try:
        run_case(fuel, orc, g, m, inflate, tri, lo, hi, mode, threads=16)
    finally:
        m.close()


# ---- forms selected by the environment ----------------------------------------------------------------------------
_CHILD = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import fuel_b200
inp = np.load(sys.argv[2])
out = {}
for key in sorted({k.split("|")[0] for k in inp.files}):
    infl, tri = inp[key + "|inflate"], inp[key + "|tri"]
    m = fuel_b200.SDFMap(infl.shape, float(sys.argv[4]), (0.0, 0.0, 0.0))
    m.occupancy_buffer_inflate_[...] = infl
    m.setOccupancyBuffer(tristate=tri)
    m.upload()
    for mode, (opt, signed) in (("opt", (True, False)), ("nonopt", (False, False)), ("signed", (True, True))):
        m.optimistic_, m.signed_dist_ = opt, signed
        c0 = m.launch_count()
        m.updateESDF3d()
        out["%s|%s|launches" % (key, mode)] = np.array(m.launch_count() - c0)
        out["%s|%s" % (key, mode)] = m.download().copy()
    m.close()
np.savez(sys.argv[3], **out)
"""


@pytest.fixture(scope="module")
def env_runs(fuel, tmp_path_factory):
    """the device fields of every env case, each setting computed in one child process"""
    runs = {}
    for env, ns in ENV_N.items():
        d = tmp_path_factory.mktemp(env)
        scenes, inp = {}, {}
        for axis in "xy":
            for n in ns:
                for dense in (True, False):
                    key = "%s%d-%s" % (axis, n, "dense" if dense else "sparse")
                    shape = line_shape(axis, n, 64)
                    scenes[key] = line_scene(shape, axis, dense, seed=3 * n + (0 if dense else 1))
                    inp[key + "|inflate"], inp[key + "|tri"] = scenes[key]
        np.savez(d / "in.npz", **inp)
        subprocess.run([sys.executable, "-c", _CHILD, ROOT, str(d / "in.npz"), str(d / "out.npz"), repr(RES)],
                       env=dict(os.environ, **ENV[env]), check=True, timeout=900)
        runs[env] = (scenes, np.load(d / "out.npz"))
    return runs


@pytest.mark.gpu
@pytest.mark.parametrize("shape,lo,hi,mode,env", case_params("env"))
def test_env_forms(orc, env_runs, shape, lo, hi, mode, env):
    """FUELGPU_ESDF_CLUSTER=0: lines of 513..1024 samples in one 1024-thread CTA; FUELGPU_ESDF_BAND=64: 64-sample
    bands in 256- and 512-thread CTAs"""
    scenes, res = env_runs[env]
    axis, n = ("x", shape[0]) if shape[1] == 7 else ("y", shape[1])
    g = W.Grid(shape, (0.0, 0.0, 0.0), RES)
    e = ENV[env]
    f = forms(shape, lo, hi, band=int(e.get("FUELGPU_ESDF_BAND", 32)), cluster=e.get("FUELGPU_ESDF_CLUSTER", "1") != "0")
    assert f["x" if axis == "x" else "zy"] != tile_form(n)  # the environment changes this pass's form
    for dense in ("dense", "sparse"):
        key = "%s%d-%s" % (axis, n, dense)
        inflate, tri = scenes[key]
        assert int(res["%s|%s|launches" % (key, mode)]) == launches(shape, lo, hi, mode)
        got = res["%s|%s" % (key, mode)]
        check_case(orc, g, inflate, tri, lo, hi, mode, got, np.zeros(shape, np.float32))  # full box: no outside


# ---- state across updates -----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_state_across_updates(fuel, orc):
    """one map: whole box, shrinking boxes, an occupancy change, then optimistic -> non-optimistic -> signed (the first
    signed update allocates dist_neg) -> signed on another box -> optimistic.  Inside each box the field equals the
    oracle's chained update; outside it is bit-identical to the previous download."""
    shape = (300, 140, 96)
    g = W.Grid(shape, (0.0, 0.0, 0.0), RES)
    inflate, tri = block_scene(shape, seed=77, p_site=0.001)
    m = make_sdf_map(fuel, g, inflate, tri, optimistic=True)
    A = ((5, 3, 16), (290, 130, 79))   # vectorised z-pack
    B = ((20, 10, 3), (200, 100, 70))  # scalar
    full = full_box(shape)
    try:
        run_case(fuel, orc, g, m, inflate, tri, *full, "opt")
        run_case(fuel, orc, g, m, inflate, tri, *A, "opt")
        run_case(fuel, orc, g, m, inflate, tri, *B, "opt")
        inflate[60:70, 40:50, 20:40] = 1
        tri[60:70, 40:50, 20:40] = W.OCCUPIED
        inflate[100:180, 20:90, 30:60] = 0
        tri[100:180, 20:90, 30:60] = W.FREE
        m.occupancy_buffer_inflate_[...] = inflate
        m.setOccupancyBuffer(tristate=tri)
        m.upload()
        run_case(fuel, orc, g, m, inflate, tri, *B, "opt")
        run_case(fuel, orc, g, m, inflate, tri, *B, "nonopt")
        run_case(fuel, orc, g, m, inflate, tri, *A, "signed")
        run_case(fuel, orc, g, m, inflate, tri, *B, "signed")
        run_case(fuel, orc, g, m, inflate, tri, *full, "opt")
    finally:
        m.close()
