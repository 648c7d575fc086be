"""The `gs-mesh o3dtsdf` exporter (reference dn_splatter/export_mesh.py:931-1047) on the device.

Every training view is rendered by the render service straight into its static device maps, fused into a sparse TSDF
volume (Open3D's legacy ScalableTSDFVolume semantics: 16^3-voxel units allocated from the stride-4 depth point cloud,
per-view integration of the touched units), meshed by marching cubes, and cleaned by the exporter's cluster filter.
The kernels are csrc/tsdf.cu behind include/dnr.h; oracle/mesh_ref.py states the same contract in numpy.  No CPU path.

    mesh = o3d_tsdf_fusion(model, cameras, output_dir="out")     # writes out/Open3dTSDFfusion_mesh.ply
"""
from __future__ import annotations

import ctypes as C
import math
import os
from dataclasses import dataclass
from typing import Optional, Sequence, Tuple

import numpy as np
import torch
from torch import Tensor

from . import _lib as L
from .rasterize import DnrCapacityError

UNIT_VOXELS = 16 ** 3
CHECK_LAG = 2  # views between an integration and the read of its pool counters


@dataclass
class TriangleMesh:
    vertices: Tensor        # [V,3] f32
    vertex_colors: Tensor   # [V,3] f32 in [0,1]
    triangles: Tensor       # [T,3] i32


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _need_cuda(*ts: Tensor) -> None:
    for t in ts:
        if t is not None and t.device.type != "cuda":
            raise L.DnrError("dn_splatter_b200.export_mesh needs CUDA tensors (no CPU path)")


def camera_matrices(c2w) -> Tuple[np.ndarray, np.ndarray]:
    """(pose [4,4] f64, extrinsic [4,4] f32) from a nerfstudio [3,4] camera_to_world, as export_mesh.py:972-1017 and
    Open3D build them: OpenGL -> OpenCV flip in fp32, extrinsic = inv(c2w) in fp32, pose = inv(extrinsic) in fp64."""
    m = np.eye(4, dtype=np.float32)
    m[:3, :4] = np.asarray(c2w, dtype=np.float32).reshape(3, 4)
    m = m @ np.diag(np.array([1, -1, -1, 1], dtype=np.float32))
    ext = np.linalg.inv(m).astype(np.float32)
    return np.linalg.inv(ext.astype(np.float64)), ext


def _camera_params(camera):
    c2w = camera.camera_to_worlds.detach().reshape(-1, 3, 4)[0].cpu().numpy()
    vals = [float(torch.as_tensor(getattr(camera, k)).flatten()[0]) for k in ("fx", "fy", "cx", "cy")]
    return (*vals, c2w)


class TSDFVolume:
    """Sparse TSDF volume on the device.  `integrate` enqueues on the current stream without synchronising; a pool that
    runs out of units is reported (`needed_units`), never silently truncated: `extract_triangle_mesh` raises
    DnrCapacityError on an overflowed volume."""

    def __init__(self, voxel_size: float = 0.01, sdf_trunc: float = 0.03, depth_trunc: float = 20.0, device=None,
                 capacity: int = 4096):
        self.voxel_size, self.sdf_trunc, self.depth_trunc = float(voxel_size), float(sdf_trunc), float(depth_trunc)
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.type != "cuda":
            raise L.DnrError("TSDFVolume lives on a CUDA device (no CPU path)")
        self._snap = [torch.zeros(4, dtype=torch.int32).pin_memory() for _ in range(CHECK_LAG + 1)]
        self._snap_ev = [None] * (CHECK_LAG + 1)
        self.regrows = 0  # pool regrowths of o3d_tsdf_fusion
        self.reset(capacity)

    def reset(self, capacity: Optional[int] = None) -> None:
        """Empties the volume (and resizes the pool to `capacity` units)."""
        if capacity is not None:
            self.capacity = max(1, int(capacity))
            self.hash_size = 1 << max(4, math.ceil(math.log2(2 * self.capacity)))
            dev = self.device
            self.hash_keys = torch.empty(self.hash_size, dtype=torch.int64, device=dev)
            self.hash_vals = torch.empty(self.hash_size, dtype=torch.int32, device=dev)
            self.hash_stamp = torch.empty(self.hash_size, dtype=torch.int32, device=dev)
            self.touched = torch.empty(self.hash_size, dtype=torch.int32, device=dev)
            self.voxels = torch.empty((self.capacity, 5, UNIT_VOXELS), dtype=torch.float32, device=dev)
            self.counters = torch.empty(4, dtype=torch.int32, device=dev)
            s = L.DnrTsdfVolume()
            s.voxel_size, s.sdf_trunc, s.depth_trunc = self.voxel_size, self.sdf_trunc, self.depth_trunc
            s.capacity, s.hash_size = self.capacity, self.hash_size
            for f in ("hash_keys", "hash_vals", "hash_stamp", "voxels", "touched", "counters"):
                setattr(s, f, getattr(self, f).data_ptr())
            self._s = s
        self.n_views = 0
        self._snap_ev = [None] * (CHECK_LAG + 1)
        L.check(L.load().dnr_tsdf_reset(C.byref(self._s), _stream()), "dnr_tsdf_reset")

    def integrate(self, depth: Tensor, rgb: Tensor, camera, mask: Optional[Tensor] = None) -> None:
        """Fuses one view: depth [H,W(,1)] f32, rgb [H,W,3] f32 in [0,1], mask [H,W(,1)] bool (False = no depth)."""
        _need_cuda(depth, rgb, mask)
        H, W = int(depth.shape[0]), int(depth.shape[1])
        if depth.dtype != torch.float32 or rgb.dtype != torch.float32 or tuple(rgb.shape) != (H, W, 3) or depth.numel() != H * W:
            raise L.DnrError(f"integrate: depth [H,W(,1)] and rgb [H,W,3] float32 expected, got {tuple(depth.shape)} "
                             f"{depth.dtype}, {tuple(rgb.shape)} {rgb.dtype}")
        depth, rgb = depth.contiguous(), rgb.contiguous()
        m = None
        if mask is not None:
            if mask.numel() != H * W:
                raise L.DnrError(f"integrate: mask of {mask.numel()} entries for a {H}x{W} view")
            m = mask.reshape(H, W).to(torch.uint8).contiguous()
        fx, fy, cx, cy, c2w = _camera_params(camera)
        pose, ext = camera_matrices(c2w)
        v = L.DnrTsdfView()
        v.width, v.height, v.stamp = W, H, self.n_views
        v.fx, v.fy, v.cx, v.cy = fx, fy, cx, cy
        for i in range(16):
            v.extrinsic[i] = float(ext.flat[i])
            v.pose[i] = float(pose.flat[i])
        v.depth, v.rgb, v.mask = depth.data_ptr(), rgb.data_ptr(), None if m is None else m.data_ptr()
        lib = L.load()
        L.check(lib.dnr_tsdf_allocate(C.byref(self._s), C.byref(v), _stream()), "dnr_tsdf_allocate")
        L.check(lib.dnr_tsdf_integrate(C.byref(self._s), C.byref(v), _stream()), "dnr_tsdf_integrate")
        k = self.n_views % len(self._snap)
        if self._snap_ev[k] is not None:
            self._snap_ev[k].synchronize()  # that snapshot is CHECK_LAG + 1 views old: its copy has long landed
        self._snap[k].copy_(self.counters, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self._snap_ev[k] = ev
        self.n_views += 1

    def _needed(self, c) -> int:
        n_alloc, _, hash_full, out_of_range = (int(x) for x in c.tolist())
        if out_of_range:
            raise L.DnrError(f"{out_of_range} depth points map to volume units beyond +-2^20 per axis")
        if n_alloc > self.capacity or hash_full:
            return max(n_alloc, self.capacity + 1)
        return 0

    def needed_units(self, lag: int = CHECK_LAG) -> int:
        """Units the pool needs (0 while it is large enough) as of the view integrated `lag` views ago; lag=0 waits for
        the latest view."""
        if self.n_views == 0:
            return 0
        i = self.n_views - 1 - min(lag, self.n_views - 1)
        if lag >= len(self._snap) or (self.n_views - 1 - i) >= len(self._snap):
            raise ValueError(f"lag must be < {len(self._snap)}")
        k = i % len(self._snap)
        self._snap_ev[k].synchronize()
        return self._needed(self._snap[k])

    @property
    def n_units(self) -> int:
        return int(self.counters[0])

    def units(self) -> Tuple[Tensor, Tensor]:
        """(unit coordinates [K,3] int64 in lexicographic order, data [K,5,4096] f32) of the allocated units."""
        keys = self.hash_keys
        ok = (keys != -1) & (self.hash_vals >= 0)
        k, slot = keys[ok], self.hash_vals[ok].long()
        order = torch.argsort(k)
        k, slot = k[order], slot[order]
        bias, m = 1 << 20, (1 << 21) - 1
        coords = torch.stack([((k >> 42) & m) - bias, ((k >> 21) & m) - bias, (k & m) - bias], -1)
        return coords, self.voxels[slot]

    def extract_triangle_mesh(self) -> TriangleMesh:
        """Marching cubes over the allocated units (ScalableTSDFVolume::ExtractTriangleMesh), in a deterministic order."""
        need = self._needed(self.counters.cpu())
        if need:
            raise DnrCapacityError(f"the TSDF pool holds {self.capacity} units, the fused views needed {need}")
        lib = L.load()
        n = self.n_units
        nbytes = lib.dnr_tsdf_extract_workspace_bytes(n)
        if nbytes < 0:
            raise L.DnrError(f"dnr_tsdf_extract_workspace_bytes({n}) failed")
        ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        L.check(lib.dnr_tsdf_extract_count(C.byref(self._s), n, ws.data_ptr(), nbytes, _stream()), "dnr_tsdf_extract_count")
        nv, nt = (int(x) for x in ws[:16].view(torch.int64).cpu())
        verts = torch.empty((nv, 3), dtype=torch.float32, device=self.device)
        cols = torch.empty((nv, 3), dtype=torch.float32, device=self.device)
        tris = torch.empty((nt, 3), dtype=torch.int32, device=self.device)
        L.check(lib.dnr_tsdf_extract_emit(C.byref(self._s), n, ws.data_ptr(), nbytes, verts.data_ptr(), cols.data_ptr(),
                                          tris.data_ptr(), _stream()), "dnr_tsdf_extract_emit")
        return TriangleMesh(verts, cols, tris)


def filter_small_clusters(mesh: TriangleMesh, keep_largest: int = 50, min_triangles: int = 50) -> TriangleMesh:
    """export_mesh.py:1021-1039: remove the triangles of clusters (connected through shared edges) smaller than
    max(size of the keep_largest-th largest cluster, min_triangles), then the unreferenced vertices; order is kept.
    With fewer than keep_largest clusters the threshold is min_triangles (the reference raises there)."""
    _need_cuda(mesh.vertices, mesh.vertex_colors, mesh.triangles)
    tris = mesh.triangles.to(torch.int32).contiguous()
    verts, cols = mesh.vertices.float().contiguous(), mesh.vertex_colors.float().contiguous()
    T, V = tris.shape[0], verts.shape[0]
    lib = L.load()
    nbytes = lib.dnr_mesh_cluster_workspace_bytes(T, V)
    if nbytes < 0:
        raise L.DnrError(f"dnr_mesh_cluster_workspace_bytes({T}, {V}) failed")
    ws = torch.empty(nbytes, dtype=torch.uint8, device=verts.device)
    L.check(lib.dnr_mesh_cluster_count(tris.data_ptr(), T, V, int(keep_largest), int(min_triangles), ws.data_ptr(), nbytes,
                                       _stream()), "dnr_mesh_cluster_count")
    nv, nt = (int(x) for x in ws[:16].view(torch.int64).cpu())
    out = TriangleMesh(torch.empty((nv, 3), dtype=torch.float32, device=verts.device),
                       torch.empty((nv, 3), dtype=torch.float32, device=verts.device),
                       torch.empty((nt, 3), dtype=torch.int32, device=verts.device))
    L.check(lib.dnr_mesh_cluster_emit(tris.data_ptr(), verts.data_ptr(), cols.data_ptr(), T, V, ws.data_ptr(), nbytes,
                                      out.triangles.data_ptr(), out.vertices.data_ptr(), out.vertex_colors.data_ptr(),
                                      _stream()), "dnr_mesh_cluster_emit")
    return out


def _np(x) -> np.ndarray:
    return x.detach().cpu().numpy() if isinstance(x, Tensor) else np.asarray(x)


def write_ply(path: str, mesh: TriangleMesh) -> None:
    """Binary little-endian PLY: float x y z, uchar red green blue (round(colour * 255)), int face lists."""
    v = np.ascontiguousarray(_np(mesh.vertices), dtype="<f4").reshape(-1, 3)
    c = np.round(np.clip(_np(mesh.vertex_colors).astype(np.float64), 0.0, 1.0) * 255.0).astype(np.uint8).reshape(-1, 3)
    t = np.ascontiguousarray(_np(mesh.triangles), dtype="<i4").reshape(-1, 3)
    vrec = np.empty(len(v), dtype=[("xyz", "<f4", 3), ("rgb", "u1", 3)])
    vrec["xyz"], vrec["rgb"] = v, c
    frec = np.empty(len(t), dtype=[("n", "u1"), ("idx", "<i4", 3)])
    frec["n"], frec["idx"] = 3, t
    header = ("ply\nformat binary_little_endian 1.0\n"
              f"element vertex {len(v)}\nproperty float x\nproperty float y\nproperty float z\n"
              "property uchar red\nproperty uchar green\nproperty uchar blue\n"
              f"element face {len(t)}\nproperty list uchar int vertex_indices\nend_header\n")
    with open(path, "wb") as f:
        f.write(header.encode("ascii"))
        f.write(vrec.tobytes())
        f.write(frec.tobytes())


def read_ply(path: str) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Reads what write_ply writes: (vertices [V,3] f32, colours [V,3] uint8, triangles [T,3] i32)."""
    with open(path, "rb") as f:
        data = f.read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    head = data[:end].decode("ascii").split("\n")
    nv = int(next(l for l in head if l.startswith("element vertex")).split()[-1])
    nt = int(next(l for l in head if l.startswith("element face")).split()[-1])
    vrec = np.frombuffer(data, dtype=[("xyz", "<f4", 3), ("rgb", "u1", 3)], count=nv, offset=end)
    frec = np.frombuffer(data, dtype=[("n", "u1"), ("idx", "<i4", 3)], count=nt, offset=end + vrec.nbytes)
    if nt and not (frec["n"] == 3).all():
        raise ValueError(f"{path}: only triangle faces are supported")
    return vrec["xyz"].copy(), vrec["rgb"].copy(), frec["idx"].copy()


def _camera_list(cameras) -> list:
    if isinstance(cameras, (list, tuple)):
        return list(cameras)
    return [cameras[i] for i in range(int(cameras.shape[0]))]


def o3d_tsdf_fusion(model, cameras, masks: Optional[Sequence[Optional[Tensor]]] = None, voxel_size: float = 0.01,
                    sdf_truc: float = 0.03, depth_trunc: float = 20.0, output_dir: Optional[str] = None,
                    capacity: int = 4096, return_volume: bool = False):
    """Open3DTSDFFusion.main (export_mesh.py:931-1047) over `cameras` (field names and defaults kept, `sdf_truc`
    included): render every view on the device, fuse its depth and colour, extract, filter small clusters, and with
    `output_dir` write Open3dTSDFfusion_mesh.ply.  `capacity` is the initial unit pool: when it overflows it grows to
    1.5x what was needed and the views are fused again from the first (the volume's `regrows` counts that).  Returns the
    mesh, or (mesh, volume) with return_volume=True."""
    from .render_service import ViewRenderer

    if model.device.type != "cuda":
        raise L.DnrError("o3d_tsdf_fusion runs on a CUDA model (no CPU path)")
    cams = _camera_list(cameras)
    if masks is not None and len(masks) != len(cams):
        raise ValueError(f"{len(masks)} masks for {len(cams)} cameras")
    vol = TSDFVolume(voxel_size, sdf_truc, depth_trunc, device=model.device, capacity=capacity)
    renderer = ViewRenderer(model, keys=("rgb", "depth"), to_host=False)
    while True:
        need = 0
        for idx, maps in renderer.render(cams):
            mask = None if masks is None or masks[idx] is None else masks[idx].to(model.device, non_blocking=True)
            vol.integrate(maps["depth"], maps["rgb"], cams[idx], mask)
            need = vol.needed_units()
            if need:
                break
        if not need:
            need = vol.needed_units(lag=0)
        if not need:
            break
        vol.regrows += 1
        vol.reset(math.ceil(1.5 * need))
    mesh = filter_small_clusters(vol.extract_triangle_mesh())
    if output_dir is not None:
        os.makedirs(output_dir, exist_ok=True)
        write_ply(os.path.join(output_dir, "Open3dTSDFfusion_mesh.ply"), mesh)
    return (mesh, vol) if return_volume else mesh
