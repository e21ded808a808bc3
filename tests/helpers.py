"""Shared builders for the parity tests (inputs only)."""
import numpy as np

from fuel_b200 import workloads as W


def random_scene(n, seed, p_site=0.02, p_unknown=0.3, blobs=6):
    """Small random occupancy: sparse inflate bits + blobby known region."""
    rng = np.random.default_rng(seed)
    inflate = (rng.random(n) < p_site).astype(np.int8)
    tri = np.full(n, W.FREE, dtype=np.uint8)
    # unknown blobs
    ax = [np.arange(k) for k in n]
    X, Y, Z = np.meshgrid(*ax, indexing="ij")
    unk = np.zeros(n, dtype=bool)
    for _ in range(blobs):
        c = rng.uniform(0, 1, 3) * np.array(n)
        r = rng.uniform(0.15, 0.45) * min(n)
        unk |= ((X - c[0]) ** 2 + (Y - c[1]) ** 2 + (Z - c[2]) ** 2) < r * r
    if p_unknown > 0:
        tri[unk] = W.UNKNOWN
    tri[(inflate == 1) & (tri == W.FREE)] = W.OCCUPIED
    return inflate, tri


def make_sdf_map(fuel, g, inflate, tri, optimistic=False, signed=False):
    m = fuel.SDFMap(g.n, g.res, g.origin, g.box_min, g.box_max, optimistic=optimistic, signed_dist=signed)
    m.occupancy_buffer_inflate_[...] = inflate
    m.setOccupancyBuffer(tristate=tri)
    m.upload()
    return m


def sdf_map_geometry(params):
    """map_voxel_num_, map_origin_ and map_size_ as the reference's SDFMap::initMap derives them from its
    sdf_map/* parameters (sdf_map.cpp:33-37): the map is centred in x, y and starts at ground_height in z"""
    size = np.array([params["map_size_" + a] for a in "xyz"])
    n = tuple(int(np.ceil(s / params["resolution"])) for s in size)
    return n, np.array([-size[0] / 2.0, -size[1] / 2.0, params["ground_height"]]), size


def viewpoint_rows(visib, yaw, pos):
    """the viewpoints of one cluster as sorted rows (-visib, yaw, x, y, z): the reference sorts them by visib_num_
    with std::sort, whose order among ties is unspecified, so they are compared as multisets"""
    rows = np.column_stack([-np.asarray(visib, np.float64), yaw, np.reshape(pos, (-1, 3))])
    return rows[np.lexsort(rows.T[::-1])]


def orc_grid(orc, g):
    return orc.make_grid(g.n, g.res, g.origin, g.box_min, g.box_max)


def rel_err(a, b, floor=0.0):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.abs(a - b) / np.maximum(np.abs(b), floor if floor > 0 else np.finfo(np.float64).tiny)
