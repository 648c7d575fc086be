"""numpy restatement of the o3dtsdf mesh exporter (reference dn_splatter/export_mesh.py:931-1047): Open3D's legacy
ScalableTSDFVolume (integrate + extract_triangle_mesh) and the cluster filter that follows it.  Slow, for small volumes;
imported by the tests and scripts/mesh_bench.py only.

Floating-point order is spelled out so the CUDA kernels (csrc/tsdf.cu, built with -fmad=false) can be compared bit for
bit: allocation in fp64, integration in fp32 with the camera point walked along z as Open3D's column loop does,
extraction positions / colours in fp64.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import numpy as np

from dn_splatter_b200.mc_tables import EDGE_CORNERS, EDGE_OWNER, EDGE_TABLE, TRI_TABLE, CORNERS

RES = 16                 # voxels per volume-unit side (Open3D's default volume_unit_resolution)
STRIDE = 4               # depth_sampling_stride of the allocation point cloud
F32 = np.float32


def camera_matrices(c2w: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """(pose [4,4] f64, extrinsic [4,4] f32) from a nerfstudio [3,4] camera_to_world, as export_mesh.py:972-1017 and
    Open3D build them: OpenGL -> OpenCV flip in fp32, extrinsic = inv(c2w) in fp32, pose = inv(extrinsic) in fp64."""
    m = np.eye(4, dtype=F32)
    m[:3, :4] = np.asarray(c2w, dtype=F32).reshape(3, 4)
    m = m @ np.diag(np.array([1, -1, -1, 1], dtype=F32))
    ext = np.linalg.inv(m).astype(F32)
    return np.linalg.inv(ext.astype(np.float64)), ext


class Volume:
    """Sparse TSDF volume: unit coordinates -> [5, 4096] fp32 (tsdf, weight, r, g, b; voxel index x + 16 y + 256 z)."""

    def __init__(self, voxel_size: float = 0.01, sdf_trunc: float = 0.03, depth_trunc: float = 20.0):
        self.voxel, self.trunc, self.depth_trunc = float(voxel_size), float(sdf_trunc), float(depth_trunc)
        self.unit_len = self.voxel * RES
        self.units: Dict[Tuple[int, int, int], np.ndarray] = {}
        self.touched_log = []  # per view: [n,3] int64 touched unit coordinates (sorted)

    # ------------------------------------------------------------------ per view
    def prepare(self, depth, rgb, mask=None):
        d = np.array(depth, dtype=F32).reshape(np.shape(depth)[0], np.shape(depth)[1]).copy()
        d[d > F32(self.depth_trunc)] = 0.0
        if mask is not None:
            d[~np.asarray(mask, dtype=bool).reshape(d.shape)] = 0.0
        c = np.clip(np.asarray(rgb, dtype=F32) * F32(255), 0, 255).astype(np.uint8)
        return d, c

    def touched_units(self, depth: np.ndarray, fx, fy, cx, cy, pose: np.ndarray) -> np.ndarray:
        H, W = depth.shape
        v, u = np.mgrid[0:H:STRIDE, 0:W:STRIDE]
        z = depth[v, u].astype(np.float64)
        keep = z > 0
        u, v, z = u[keep].astype(np.float64), v[keep].astype(np.float64), z[keep]
        x = (u - float(cx)) * z / float(fx)
        y = (v - float(cy)) * z / float(fy)
        p = np.stack([((pose[i, 0] * x + pose[i, 1] * y) + pose[i, 2] * z) + pose[i, 3] for i in range(3)], -1)
        lo = np.floor((p - self.trunc) / self.unit_len).astype(np.int64)
        hi = np.floor((p + self.trunc) / self.unit_len).astype(np.int64)
        span = int((hi - lo).max()) + 1 if len(p) else 0
        out = []
        for dx in range(span):
            for dy in range(span):
                for dz in range(span):
                    c = lo + np.array([dx, dy, dz])
                    ok = (c <= hi).all(-1)
                    out.append(c[ok])
        if not out:
            return np.zeros((0, 3), np.int64)
        return np.unique(np.concatenate(out), axis=0)

    def integrate(self, depth, rgb, fx, fy, cx, cy, c2w, mask=None) -> None:
        d, c8 = self.prepare(depth, rgb, mask)
        pose, ext = camera_matrices(c2w)
        touched = self.touched_units(d, fx, fy, cx, cy, pose)
        self.touched_log.append(touched)
        for key in map(tuple, touched.tolist()):
            if key not in self.units:
                self.units[key] = np.zeros((5, RES ** 3), F32)
        if len(touched):
            data = np.stack([self.units[k] for k in map(tuple, touched.tolist())])
            self._integrate_units(data, touched, d, c8, fx, fy, cx, cy, ext)
            for i, k in enumerate(map(tuple, touched.tolist())):
                self.units[k] = data[i]

    def _integrate_units(self, data, units, depth, c8, fx, fy, cx, cy, ext) -> None:
        H, W = depth.shape
        fx, fy, cx, cy = F32(fx), F32(fy), F32(cx), F32(cy)
        vox = F32(self.voxel)
        half = vox * F32(0.5)
        trunc = F32(self.trunc)
        trunc_inv = F32(1.0) / trunc
        safe_w, safe_h = F32(W) - F32(0.0001), F32(H) - F32(0.0001)
        xx = (np.arange(W, dtype=F32) - cx) * (F32(1.0) / fx)
        yy = (np.arange(H, dtype=F32) - cy) * (F32(1.0) / fy)
        mult = np.sqrt(xx[None, :] * xx[None, :] + yy[:, None] * yy[:, None] + F32(1.0))
        origin = units.astype(np.float64) * self.unit_len                         # [K,3]
        ij = np.arange(RES, dtype=F32)
        lx = (half + vox * ij).astype(np.float64)                                 # fp32 offset, then + fp64 origin
        px = (lx[None, None, :] + origin[:, 0, None, None]).astype(F32)           # [K,1,16]  (y, x)
        py = (lx[None, :, None] + origin[:, 1, None, None]).astype(F32)           # [K,16,1]
        pz = (np.float64(half) + origin[:, 2]).astype(F32)[:, None, None]         # [K,1,1]
        px, py, pz = np.broadcast_arrays(px, py, pz)
        pc = [((ext[i, 0] * px + ext[i, 1] * py) + ext[i, 2] * pz) + ext[i, 3] for i in range(3)]
        step = [ext[i, 2] * vox for i in range(3)]
        K = len(units)
        for z in range(RES):
            sl = slice(z * RES * RES, (z + 1) * RES * RES)
            tsdf, w = data[:, 0, sl].reshape(K, RES, RES), data[:, 1, sl].reshape(K, RES, RES)
            cz = pc[2]
            with np.errstate(divide="ignore", invalid="ignore"):
                uf = (pc[0] * fx) / cz + cx + F32(0.5)
                vf = (pc[1] * fy) / cz + cy + F32(0.5)
            ok = (cz > 0) & (uf >= F32(0.0001)) & (uf < safe_w) & (vf >= F32(0.0001)) & (vf < safe_h)
            u = np.where(ok, uf, 0).astype(np.int64)
            v = np.where(ok, vf, 0).astype(np.int64)
            d = depth[v, u]
            ok &= d > 0
            sdf = (d - cz) * mult[v, u]
            ok &= sdf > -trunc
            t = np.minimum(F32(1.0), sdf * trunc_inv)
            wn = w + F32(1.0)
            new_t = (tsdf * w + t) / wn
            col = c8[v, u].astype(F32)                                            # [K,16,16,3]
            for ch in range(3):
                cch = data[:, 2 + ch, sl].reshape(K, RES, RES)
                newc = (cch * w + col[..., ch]) / wn
                data[:, 2 + ch, sl] = np.where(ok, newc, cch).reshape(K, -1)
            data[:, 0, sl] = np.where(ok, new_t, tsdf).reshape(K, -1)
            data[:, 1, sl] = np.where(ok, wn, w).reshape(K, -1)
            pc = [pc[i] + step[i] for i in range(3)]

    # ------------------------------------------------------------------ extraction
    def sorted_units(self) -> Tuple[np.ndarray, np.ndarray]:
        """(unit coordinates [K,3] in lexicographic (x, y, z) order, data [K,5,4096])."""
        keys = sorted(self.units)
        if not keys:
            return np.zeros((0, 3), np.int64), np.zeros((0, 5, RES ** 3), F32)
        return np.array(keys, np.int64), np.stack([self.units[k] for k in keys])

    def extract_triangle_mesh(self):
        return extract(*self.sorted_units(), self.voxel)


def extract(units: np.ndarray, data: np.ndarray, voxel: float):
    """Marching cubes over a sparse volume (Open3D ScalableTSDFVolume::ExtractTriangleMesh), in a fixed order: units in
    lexicographic order, then voxel index x + 16 y + 256 z, then axis.  Returns (vertices [V,3] f32, colours [V,3] f32,
    triangles [T,3] i32, vertex keys [V,4] = global voxel x, y, z and axis)."""
    empty = (np.zeros((0, 3), F32), np.zeros((0, 3), F32), np.zeros((0, 3), np.int32), np.zeros((0, 4), np.int64))
    if len(units) == 0:
        return empty
    lo = units.min(0)
    dims = (units.max(0) - lo + 1) * RES
    grid = np.zeros((5, dims[0] + 1, dims[1] + 1, dims[2] + 1), F32)             # one voxel of zero-weight padding
    rank = np.full(tuple(units.max(0) - lo + 1), -1, np.int64)
    for r, (uc, blk) in enumerate(zip(units, data)):
        o = (uc - lo) * RES
        grid[:, o[0]:o[0] + RES, o[1]:o[1] + RES, o[2]:o[2] + RES] = blk.reshape(5, RES, RES, RES).transpose(0, 3, 2, 1)
        rank[tuple(uc - lo)] = r
    tsdf, w = grid[0], grid[1]
    NX, NY, NZ = dims
    f = np.stack([tsdf[c[0]:c[0] + NX, c[1]:c[1] + NY, c[2]:c[2] + NZ] for c in CORNERS])
    ws = np.stack([w[c[0]:c[0] + NX, c[1]:c[1] + NY, c[2]:c[2] + NZ] for c in CORNERS])
    case = np.zeros((NX, NY, NZ), np.int64)
    for i in range(8):
        case |= (f[i] < 0).astype(np.int64) << i
    valid = (ws > 0).all(0) & (case != 0) & (case != 255)
    ci = np.argwhere(valid)                                                      # [M,3] dense cell coords
    cases = case[valid]

    def order_key(g):  # dense voxel coords -> (rank, local index) order key
        r = rank[g[:, 0] // RES, g[:, 1] // RES, g[:, 2] // RES]
        loc = g % RES
        return r * RES ** 3 + loc[:, 0] + RES * loc[:, 1] + RES * RES * loc[:, 2]

    ck = order_key(ci)
    perm = np.argsort(ck, kind="stable")
    ci, cases, ck = ci[perm], cases[perm], ck[perm]
    em = np.array(EDGE_TABLE, np.int64)[cases]
    owners = []
    for e in range(12):
        sel = (em >> e) & 1 == 1
        ox, oy, oz, ax = EDGE_OWNER[e]
        g = ci[sel] + np.array([ox, oy, oz])
        owners.append(order_key(g) * 3 + ax)
    vkey = np.unique(np.concatenate(owners)) if owners else np.zeros(0, np.int64)
    # per-cell edge -> vertex id
    edge_vid = np.full((len(ci), 12), -1, np.int64)
    for e in range(12):
        ox, oy, oz, ax = EDGE_OWNER[e]
        k = order_key(ci + np.array([ox, oy, oz])) * 3 + ax
        sel = (em >> e) & 1 == 1
        edge_vid[sel, e] = np.searchsorted(vkey, k[sel])
    tris = []
    for j, c in enumerate(cases.tolist()):
        t = TRI_TABLE[c]
        for i in range(0, len(t), 3):
            tris.append((edge_vid[j, t[i]], edge_vid[j, t[i + 2]], edge_vid[j, t[i + 1]]))
    tris = np.array(tris, np.int32).reshape(-1, 3)
    # vertices: decode keys back to dense coords
    ax = vkey % 3
    rk, loc = np.divmod(vkey // 3, RES ** 3)
    lx, ly, lz = loc % RES, (loc // RES) % RES, loc // (RES * RES)
    gl = units[rk] * RES + np.stack([lx, ly, lz], -1)                            # global voxel index
    dn = gl - lo * RES
    step = np.eye(3, dtype=np.int64)[ax]
    dn1 = dn + step
    f0 = np.abs(tsdf[dn[:, 0], dn[:, 1], dn[:, 2]].astype(np.float64))
    f1 = np.abs(tsdf[dn1[:, 0], dn1[:, 1], dn1[:, 2]].astype(np.float64))
    pos = 0.5 * voxel + voxel * gl.astype(np.float64)
    pos[np.arange(len(ax)), ax] += f0 * voxel / (f0 + f1)
    c0 = grid[2:5, dn[:, 0], dn[:, 1], dn[:, 2]].T.astype(np.float64)
    c1 = grid[2:5, dn1[:, 0], dn1[:, 1], dn1[:, 2]].T.astype(np.float64)
    col = (c0 * f1[:, None] + c1 * f0[:, None]) / (f0 + f1)[:, None] / 255.0
    return pos.astype(F32), col.astype(F32), tris, np.concatenate([gl, ax[:, None]], 1)


# ---------------------------------------------------------------------- cluster filter
def triangle_clusters(tris: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """Open3D cluster_connected_triangles: triangles sharing an edge are connected.  (labels [T], sizes [n])."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components

    T = len(tris)
    if T == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    t = tris.astype(np.int64)
    a = np.concatenate([t[:, 0], t[:, 1], t[:, 2]])
    b = np.concatenate([t[:, 1], t[:, 2], t[:, 0]])
    key = np.minimum(a, b) << 32 | np.maximum(a, b)
    tid = np.tile(np.arange(T), 3)
    o = np.lexsort((tid, key))
    key, tid = key[o], tid[o]
    same = key[1:] == key[:-1]
    g = coo_matrix((np.ones(int(same.sum())), (tid[1:][same], tid[:-1][same])), shape=(T, T))
    n, labels = connected_components(g, directed=False)
    return labels, np.bincount(labels, minlength=n)


def cluster_threshold(sizes: np.ndarray, keep_largest: int = 50, min_triangles: int = 50) -> int:
    """max(size of the keep_largest-th largest cluster, min_triangles); min_triangles when there are fewer clusters
    (the reference's np.sort(...)[-50] raises there)."""
    s = np.sort(sizes)[::-1]
    kth = int(s[keep_largest - 1]) if len(s) >= keep_largest else 0
    return max(kth, int(min_triangles))


def filter_small_clusters(vertices, colors, tris, keep_largest: int = 50, min_triangles: int = 50):
    """remove_triangles_by_mask(cluster size < threshold) + remove_unreferenced_vertices (order kept)."""
    labels, sizes = triangle_clusters(tris)
    thr = cluster_threshold(sizes, keep_largest, min_triangles)
    kept = tris[sizes[labels] >= thr] if len(tris) else tris
    used = np.zeros(len(vertices), bool)
    used[kept.reshape(-1)] = True
    remap = np.cumsum(used) - 1
    return vertices[used], colors[used], remap[kept].astype(np.int32).reshape(-1, 3)


def fuse(views, voxel_size=0.01, sdf_trunc=0.03, depth_trunc=20.0, keep_largest=50, min_triangles=50):
    """Full o3dtsdf pipeline over [(depth [H,W], rgb [H,W,3], fx, fy, cx, cy, c2w [3,4], mask or None)]."""
    vol = Volume(voxel_size, sdf_trunc, depth_trunc)
    for depth, rgb, fx, fy, cx, cy, c2w, mask in views:
        vol.integrate(depth, rgb, fx, fy, cx, cy, c2w, mask)
    v, c, t, _ = vol.extract_triangle_mesh()
    return (*filter_small_clusters(v, c, t, keep_largest, min_triangles), vol)
