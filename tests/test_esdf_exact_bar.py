"""What the exact ESDF bar (tests.helpers.assert_esdf_exact) catches that the 1e-4 relative bar does not: an oracle
field rounded to fp32 the way the device stores it passes; the same field with the squared voxel distance N moved by
+-1 at a few voxels with N ~ 10^4 and ~ 10^6 fails the exact bar and still passes the relative one."""
import numpy as np
import pytest

from fuel_b200 import workloads as W
from tests.helpers import assert_esdf_exact, assert_esdf_rel, orc_grid

RES = 0.1
N_MAP = (1024, 3, 4)


def device_rounding(n_sq, res):
    """fl32(res32 * sqrt(N)) as envelope_tile_kernel stores it (numpy's sqrt is correctly rounded, sqrt.approx is
    within a few units of 2^-24 of it)"""
    r32 = np.float32(res)
    return (r32 * np.sqrt(np.asarray(n_sq, dtype=np.float32))).astype(np.float32)


@pytest.fixture(scope="module")
def field(orc):
    """unsigned (optimistic) and signed oracle fields of a 1024-voxel line map whose first 20 x planes are inflated:
    N runs from 0 to about 1004^2 and the negative field reaches N = 400"""
    g = W.Grid(N_MAP, (0.0, 0.0, 0.0), RES)
    inflate = np.zeros(N_MAP, dtype=np.int8)
    inflate[:20] = 1
    tri = np.where(inflate == 1, W.OCCUPIED, W.FREE).astype(np.uint8)
    og = orc_grid(orc, g)
    hi = np.array(N_MAP) - 1
    return {s: orc.update_esdf3d(og, inflate, tri, [0, 0, 0], hi, True, s) for s in (False, True)}


def rounded(ref, signed):
    """the fp32 field the device would produce for this reference (signed: dist = fl32(res32 - neg32) where neg > 0)"""
    out = np.empty(ref.shape, dtype=np.float32)
    fin = np.abs(ref) <= 1e150
    out[~fin] = np.where(ref[~fin] > 0, np.inf, -np.inf)
    r = ref[fin]
    neg = signed & (r <= 0)
    n_sq = np.rint(np.where(neg, RES - r, r) ** 2 / RES ** 2)
    d = device_rounding(n_sq, RES)
    out[fin] = np.where(neg, np.float32(RES) - d, d)
    return out


def perturb(got, ref, signed, targets, delta):
    """move N by `delta` at the voxel whose N is closest to each target"""
    bad = got.copy()
    r = np.where(signed & (ref <= 0), RES - ref, ref)
    n_sq = np.rint((r / RES) ** 2)
    hit = []
    for t in targets:
        i = np.unravel_index(int(np.argmin(np.abs(n_sq - t))), ref.shape)
        d = device_rounding(n_sq[i] + delta, RES)
        bad[i] = np.float32(RES) - d if signed and ref[i] <= 0 else d
        hit.append(int(n_sq[i]))
    return bad, hit


@pytest.mark.parametrize("signed", [False, True])
def test_device_rounding_passes(field, signed):
    ref = field[signed]
    got = rounded(ref, signed)
    worst = assert_esdf_exact(got, ref, RES, signed=signed)
    assert 0.0 < worst < 0.3
    assert_esdf_rel(got, ref)


@pytest.mark.parametrize("signed", [False, True])
@pytest.mark.parametrize("delta", [-1, 1])
@pytest.mark.parametrize("target", [1e4, 1e6])
def test_off_by_one_is_caught(field, signed, delta, target):
    ref = field[signed]
    bad, hit = perturb(rounded(ref, signed), ref, signed, [target], delta)
    assert abs(hit[0] - target) < 0.05 * target
    with pytest.raises(AssertionError, match="squared voxel distance differs at 1 of"):
        assert_esdf_exact(bad, ref, RES, signed=signed)
    assert_esdf_rel(bad, ref)  # the gap the exact bar closes


def test_negative_field_off_by_one_is_caught(field):
    """the signed field's negative side (inflated block, N of a few hundred) through the res - d recovery"""
    ref = field[True]
    assert ref.min() < -0.5
    got = rounded(ref, True)
    i = np.unravel_index(int(np.argmin(ref)), ref.shape)
    n_sq = int(np.rint(((RES - ref[i]) / RES) ** 2))
    bad = got.copy()
    bad[i] = np.float32(RES) - device_rounding(n_sq + 1, RES)
    with pytest.raises(AssertionError, match="squared voxel distance differs"):
        assert_esdf_exact(bad, ref, RES, signed=True)


def test_sentinel_and_range(field):
    ref = field[False].copy()
    got = rounded(ref, False)
    got[5, 0, 0] = np.inf  # +inf where the reference is finite
    with pytest.raises(AssertionError, match="sentinel"):
        assert_esdf_exact(got, ref, RES)
    # above N = 2^20 the relative bar applies: N + 1 passes there, 1e-3 relative does not
    ref2 = np.full((2, 1, 1), RES * np.sqrt(1100.0 ** 2))
    ok = device_rounding([1100 ** 2 + 1] * 2, RES).reshape(2, 1, 1)
    assert_esdf_exact(ok, ref2, RES)
    off = (ok * np.float32(1.001)).astype(np.float32)
    with pytest.raises(AssertionError, match="beyond N = 2"):
        assert_esdf_exact(off, ref2, RES)
