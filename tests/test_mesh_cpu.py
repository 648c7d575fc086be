"""CPU checks of the o3dtsdf mesh exporter: the marching-cubes tables, the numpy oracle (oracle/mesh_ref.py) on analytic
input, the cluster filter, the PLY writer and the argument errors of the C entry points."""
import ctypes as C
import math
import os

import numpy as np
import pytest

from dn_splatter_b200 import mc_tables as M
from oracle import mesh_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------------- tables
def test_every_triangle_edge_is_in_the_case_edge_mask():
    assert len(M.TRI_TABLE) == 256
    for case, tri in enumerate(M.TRI_TABLE):
        crossed = {e for e, (a, b) in enumerate(M.EDGE_CORNERS) if ((case >> a) & 1) != ((case >> b) & 1)}
        assert len(tri) % 3 == 0
        assert set(tri) == crossed, case


def test_generated_header_matches_the_python_tables():
    import importlib.util

    spec = importlib.util.spec_from_file_location("gen_mc_tables", os.path.join(ROOT, "scripts", "gen_mc_tables.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    with open(os.path.join(ROOT, "dn_splatter_b200", "csrc", "mc_tables.cuh")) as f:
        assert f.read() == gen.render()


def _edge_counts(tris):
    t = tris.astype(np.int64)
    directed = np.concatenate([t[:, [0, 1]], t[:, [1, 2]], t[:, [2, 0]]])
    return directed


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_random_fields_give_a_closed_consistently_oriented_surface(seed):
    n = 24
    rng = np.random.default_rng(seed)
    units = np.array([(x, y, z) for x in range(2) for y in range(2) for z in range(2)], np.int64)
    data = np.zeros((8, 5, R.RES ** 3), np.float32)
    for i, u in enumerate(units):
        g = np.arange(R.RES)
        gx, gy, gz = np.meshgrid(g + u[0] * R.RES, g + u[1] * R.RES, g + u[2] * R.RES, indexing="ij")
        inside = (gx < n) & (gy < n) & (gz < n)
        blk = np.zeros((5, R.RES, R.RES, R.RES), np.float32)  # [c, x, y, z]
        blk[0] = rng.uniform(-1, 1, size=gx.shape).astype(np.float32)
        blk[1] = inside
        data[i] = blk.transpose(0, 3, 2, 1).reshape(5, -1)
    v, c, t, keys = R.extract(units, data, 0.1)
    assert len(t) > 1000
    directed = _edge_counts(t)
    # an edge of the open surface lies in one of the grid's outer faces: both ends on the same border plane
    gl, ax = keys[:, :3], keys[:, 3]
    on = np.zeros((len(keys), 6), bool)
    for a in range(3):
        on[:, 2 * a] = (gl[:, a] == 0) & (ax != a)
        on[:, 2 * a + 1] = (gl[:, a] == n - 1) & (ax != a)
    border = (on[directed[:, 0]] & on[directed[:, 1]]).any(1)
    inner = directed[~border]
    assert len(inner) > 0.9 * len(directed)
    fwd = {}
    for a, b in inner.tolist():
        fwd[(a, b)] = fwd.get((a, b), 0) + 1
    for (a, b), k in fwd.items():
        assert k == 1, "an interior edge is used twice in the same direction"
        assert fwd.get((b, a), 0) == 1, "an interior edge is not used in the opposite direction"
    assert (np.isfinite(v).all()) and len(c) == len(v)


# ---------------------------------------------------------------------- analytic sphere through the oracle
def sphere_views(n_az=8, elevations=(-40.0, 0.0, 40.0), W=128, H=96, radius=1.0, dist=3.0, rgb=(0.3, 0.6, 0.9)):
    """Ray-sphere z-depth maps (0 where the ray misses) and a constant colour, from cameras looking at the origin."""
    from dn_splatter_b200.synthetic import look_at_c2w
    import torch

    fx = fy = 0.9 * W
    cx, cy = W / 2.0, H / 2.0
    views = []
    for el in elevations:
        for i in range(n_az):
            az = 2 * math.pi * (i + 0.5 * (el > 0)) / n_az
            e = math.radians(el)
            pos = torch.tensor([dist * math.cos(e) * math.cos(az), dist * math.cos(e) * math.sin(az), dist * math.sin(e)])
            c2w = look_at_c2w(pos, torch.zeros(3), torch.tensor([0.0, 0.0, 1.0])).numpy().astype(np.float32)
            views.append((sphere_depth(c2w, fx, fy, cx, cy, W, H, radius), np.broadcast_to(np.array(rgb, np.float32), (H, W, 3)),
                          fx, fy, cx, cy, c2w))
    return views


def sphere_depth(c2w, fx, fy, cx, cy, W, H, radius):
    R_cv = c2w[:3, :3].astype(np.float64) @ np.diag([1.0, -1.0, -1.0])
    o = c2w[:3, 3].astype(np.float64)
    v, u = np.mgrid[0:H, 0:W]
    d = np.stack([(u + 0.5 - cx) / fx, (v + 0.5 - cy) / fy, np.ones_like(u, dtype=np.float64)], -1) @ R_cv.T
    a = (d * d).sum(-1)
    b = 2 * (d @ o)
    c = o @ o - radius * radius
    disc = b * b - 4 * a * c
    t = (-b - np.sqrt(np.maximum(disc, 0))) / (2 * a)
    return np.where(disc > 0, t, 0.0).astype(np.float32)


@pytest.fixture(scope="module")
def sphere_mesh():
    views = [(*vw, None) for vw in sphere_views()]
    return R.fuse(views, voxel_size=0.02, sdf_trunc=0.06)


def test_sphere_fuses_into_one_closed_cluster(sphere_mesh):
    v, c, t, vol = sphere_mesh
    labels, sizes = R.triangle_clusters(t)
    assert len(sizes) == 1
    e = np.sort(np.concatenate([t[:, [0, 1]], t[:, [1, 2]], t[:, [2, 0]]]), axis=1)
    uniq, cnt = np.unique(e, axis=0, return_counts=True)
    assert (cnt == 2).all(), "every edge of the sphere is shared by exactly two triangles"
    assert len(v) - len(uniq) + len(t) == 2, "Euler characteristic"


def test_sphere_geometry_and_colour(sphere_mesh):
    v, c, t, vol = sphere_mesh
    r = np.linalg.norm(v.astype(np.float64), axis=1)
    assert np.abs(r - 1.0).max() <= 0.02
    a, b, cc = (v[t[:, i]].astype(np.float64) for i in range(3))
    vol6 = np.einsum("ij,ij->i", a, np.cross(b, cc)).sum() / 6.0
    assert abs(abs(vol6) / (4.0 / 3.0 * math.pi) - 1.0) < 0.02
    want = np.floor(np.array([0.3, 0.6, 0.9], np.float32) * np.float32(255)) / 255.0
    assert np.abs(c - want).max() <= 1.0 / 255.0


def test_degenerate_triangles_do_not_occur(sphere_mesh):
    v, c, t, vol = sphere_mesh
    assert ((t[:, 0] != t[:, 1]) & (t[:, 1] != t[:, 2]) & (t[:, 2] != t[:, 0])).all()


# ---------------------------------------------------------------------- cluster filter
def _strip(n_tris, base):
    """A strip of n_tris triangles sharing edges, vertex ids from base."""
    return np.array([(base + i, base + i + 1, base + i + 2) for i in range(n_tris)], np.int32)


def test_components_touching_at_one_vertex_are_two_clusters():
    t = np.array([[0, 1, 2], [2, 3, 4]], np.int32)
    labels, sizes = R.triangle_clusters(t)
    assert len(sizes) == 2 and labels[0] != labels[1]


def test_threshold_with_more_than_50_clusters():
    sizes = list(range(1, 121))  # 120 clusters of 1..120 triangles: the 50th largest has 71
    tris, base = [], 0
    for s in sizes:
        tris.append(_strip(s, base))
        base += s + 2
    t = np.concatenate(tris)
    v = np.zeros((base, 3), np.float32)
    assert R.cluster_threshold(np.array(sizes)) == 71
    v2, c2, t2 = R.filter_small_clusters(v, v, t)
    assert len(t2) == sum(s for s in sizes if s >= 71)
    assert len(v2) == sum(s + 2 for s in sizes if s >= 71)
    assert R.cluster_threshold(np.array(sizes) // 3) == 50


def test_threshold_with_fewer_than_50_clusters():
    t = np.concatenate([_strip(60, 0), _strip(49, 62), _strip(50, 113)])
    v = np.arange(165 * 3, dtype=np.float32).reshape(-1, 3)
    v2, c2, t2 = R.filter_small_clusters(v, v, t)
    assert len(t2) == 110
    assert np.array_equal(v2[t2], v[np.concatenate([_strip(60, 0), _strip(50, 113)])])


# ---------------------------------------------------------------------- PLY
def test_ply_round_trip(tmp_path):
    from dn_splatter_b200.export_mesh import TriangleMesh, read_ply, write_ply

    rng = np.random.default_rng(0)
    v = rng.normal(size=(50, 3)).astype(np.float32)
    col = rng.uniform(size=(50, 3)).astype(np.float32)
    t = rng.integers(0, 50, size=(70, 3)).astype(np.int32)
    p = tmp_path / "m.ply"
    write_ply(str(p), TriangleMesh(v, col, t))
    v2, c2, t2 = read_ply(str(p))
    assert np.array_equal(v2, v) and np.array_equal(t2, t)
    assert np.array_equal(c2, np.round(np.clip(col, 0, 1) * 255).astype(np.uint8))
    assert open(p, "rb").read().startswith(b"ply\nformat binary_little_endian 1.0\n")


# ---------------------------------------------------------------------- C entry points
@pytest.fixture(scope="module")
def lib():
    from dn_splatter_b200 import _lib as L

    if not os.path.exists(L.LIB_PATH):
        from dn_splatter_b200.build import build

        build()
    return L.load()


def test_tsdf_entry_points_reject_bad_arguments(lib):
    from dn_splatter_b200 import _lib as L

    vol = L.DnrTsdfVolume()
    view = L.DnrTsdfView()
    assert lib.dnr_tsdf_reset(None, None) == -1
    assert lib.dnr_tsdf_allocate(None, C.byref(view), None) == -1
    assert lib.dnr_tsdf_allocate(C.byref(vol), C.byref(view), None) == -1  # no buffers
    assert lib.dnr_tsdf_integrate(C.byref(vol), None, None) == -1
    assert lib.dnr_tsdf_extract_workspace_bytes(-1) < 0
    assert lib.dnr_tsdf_extract_count(None, 0, None, 0, None) == -1
    assert lib.dnr_tsdf_extract_emit(None, 0, None, 0, None, None, None, None) == -1
    assert lib.dnr_mesh_cluster_workspace_bytes(-1, 3) < 0
    assert lib.dnr_mesh_cluster_count(None, 5, 3, 50, 50, None, 0, None) == -1
    assert lib.dnr_mesh_cluster_emit(None, None, None, 5, 3, None, 0, None, None, None, None) == -1
    # sizes are checked before any pointer is touched on the device
    buf = C.create_string_buffer(64)
    bad = L.DnrTsdfVolume()
    for f in ("hash_keys", "hash_vals", "hash_stamp", "voxels", "touched", "counters"):
        setattr(bad, f, C.cast(buf, C.c_void_p))
    bad.voxel_size, bad.sdf_trunc, bad.depth_trunc, bad.capacity, bad.hash_size = 0.01, 0.03, 20.0, 16, 24  # not 2^k
    assert lib.dnr_tsdf_reset(C.byref(bad), None) == -2
    bad.hash_size, bad.voxel_size = 32, 0.0
    assert lib.dnr_tsdf_reset(C.byref(bad), None) == -2
