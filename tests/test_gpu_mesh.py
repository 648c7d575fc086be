"""The o3dtsdf kernels (csrc/tsdf.cu through dn_splatter_b200.export_mesh) against the numpy oracle (oracle/mesh_ref.py):
integration, extraction and the cluster filter on the same inputs, the whole exporter end to end, masks, and the
regrowth of an overflowing unit pool."""
import numpy as np
import pytest
import torch

from oracle import mesh_ref as R

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")]

VOXEL, TRUNC = 0.1, 0.3  # the synthetic scene fills a 10 m cube


def _cam(c2w, fx, fy, cx, cy, W, H):
    from dn_splatter_b200.cameras import Cameras

    return Cameras(torch.as_tensor(np.asarray(c2w))[None].cuda(), fx, fy, cx, cy, W, H)


@pytest.fixture(scope="module")
def scene():
    from dn_splatter_b200.dn_model import DNSplatterModelConfig
    from dn_splatter_b200.synthetic import make_scene, ring_cameras

    m = DNSplatterModelConfig(random_init=True, num_random=16, background_color="black", ssim_lambda=0.0).setup(device="cuda")
    m.load_gaussians(make_scene(3000, seed=5))
    m.step = 30000
    cams = [_cam(c["c2w"].numpy(), c["fx"], c["fy"], c["cx"], c["cy"], c["width"], c["height"]) for c in ring_cameras(12, 160, 120)]
    return m, cams


def _host_maps(model, cams):
    from dn_splatter_b200.render_service import ViewRenderer

    out = []
    for idx, maps in ViewRenderer(model, keys=("rgb", "depth"), graph=False, to_host=True).render(cams):
        out.append((maps["depth"].numpy()[..., 0].copy(), maps["rgb"].numpy().copy()))
    return out


def _views(maps, cams, masks=None):
    res = []
    for i, ((d, rgb), c) in enumerate(zip(maps, cams)):
        fx, fy, cx, cy = (float(getattr(c, k).flatten()[0]) for k in ("fx", "fy", "cx", "cy"))
        res.append((d, rgb, fx, fy, cx, cy, c.camera_to_worlds[0].cpu().numpy(), None if masks is None else masks[i]))
    return res


def _fuse_gpu(views, voxel, trunc, capacity=4096):
    from dn_splatter_b200.export_mesh import TSDFVolume

    vol = TSDFVolume(voxel, trunc, device="cuda", capacity=capacity)
    for d, rgb, fx, fy, cx, cy, c2w, mask in views:
        H, W = d.shape
        vol.integrate(torch.from_numpy(d).cuda(), torch.from_numpy(np.ascontiguousarray(rgb)).cuda(),
                      _cam(c2w, fx, fy, cx, cy, W, H), None if mask is None else torch.from_numpy(mask).cuda())
    assert vol.needed_units(lag=0) == 0
    return vol


def _compare_volumes(vol, ref):
    units, data = (t.cpu().numpy() for t in vol.units())
    ru, rd = ref.sorted_units()
    assert np.array_equal(units, ru), "allocated unit sets differ"
    w, rw = data[:, 1], rd[:, 1]
    same_w = w == rw
    assert same_w.mean() >= 0.999, f"weights agree on {same_w.mean():.5f} of the voxels"
    ok = same_w & (w > 0)
    assert np.abs(data[:, 0][ok] - rd[:, 0][ok]).max() <= 1e-5
    for ch in range(3):
        assert np.abs(data[:, 2 + ch][ok] - rd[:, 2 + ch][ok]).max() <= 1e-3
    return units, data


def _sphere_views():
    from tests.test_mesh_cpu import sphere_views

    return [(*v, None) for v in sphere_views(n_az=6, elevations=(-30.0, 30.0))]


@pytest.mark.parametrize("source", ["sphere", "scene"])
def test_integration_and_extraction_match_the_oracle(source, scene):
    if source == "sphere":
        views, voxel, trunc = _sphere_views(), 0.02, 0.06
    else:
        model, cams = scene
        views, voxel, trunc = _views(_host_maps(model, cams), cams), VOXEL, TRUNC
    ref = R.Volume(voxel, trunc)
    for v in views:
        ref.integrate(*v)
    vol = _fuse_gpu(views, voxel, trunc)
    units, data = _compare_volumes(vol, ref)
    # extraction of the GPU volume on both sides
    mesh = vol.extract_triangle_mesh()
    rv, rc, rt, _ = R.extract(units, data, voxel)
    assert mesh.vertices.shape[0] == len(rv) and mesh.triangles.shape[0] == len(rt) and len(rt) > 100
    assert np.abs(mesh.vertices.cpu().numpy() - rv).max() <= 1e-5
    assert np.abs(mesh.vertex_colors.cpu().numpy() - rc).max() <= 1e-6
    assert np.array_equal(mesh.triangles.cpu().numpy(), rt)
    # the cluster filter on the GPU mesh
    from dn_splatter_b200.export_mesh import filter_small_clusters

    for keep, mn in ((50, 50), (3, 4), (1000, 1)):
        f = filter_small_clusters(mesh, keep, mn)
        fv, fc, ft = R.filter_small_clusters(mesh.vertices.cpu().numpy(), mesh.vertex_colors.cpu().numpy(),
                                             mesh.triangles.cpu().numpy(), keep, mn)
        assert np.array_equal(f.vertices.cpu().numpy(), fv) and np.array_equal(f.vertex_colors.cpu().numpy(), fc)
        assert np.array_equal(f.triangles.cpu().numpy(), ft)


def test_end_to_end_matches_oracle_and_writes_identical_files(scene, tmp_path):
    from dn_splatter_b200.export_mesh import o3d_tsdf_fusion

    model, cams = scene
    mesh = o3d_tsdf_fusion(model, cams, voxel_size=VOXEL, sdf_truc=TRUNC, output_dir=str(tmp_path / "a"))
    o3d_tsdf_fusion(model, cams, voxel_size=VOXEL, sdf_truc=TRUNC, output_dir=str(tmp_path / "b"))
    a = (tmp_path / "a" / "Open3dTSDFfusion_mesh.ply").read_bytes()
    assert a == (tmp_path / "b" / "Open3dTSDFfusion_mesh.ply").read_bytes()
    rv, rc, rt, _ = R.fuse(_views(_host_maps(model, cams), cams), VOXEL, TRUNC)
    assert len(rt) > 100
    assert mesh.triangles.shape[0] == len(rt) and np.array_equal(mesh.triangles.cpu().numpy(), rt)
    assert np.abs(mesh.vertices.cpu().numpy() - rv).max() <= 1e-5
    assert np.abs(mesh.vertex_colors.cpu().numpy() - rc).max() <= 1e-5


def test_masks_zero_the_masked_depth(scene):
    from dn_splatter_b200.export_mesh import o3d_tsdf_fusion

    model, cams = scene
    masks = []
    for i in range(len(cams)):
        m = np.ones((120, 160), bool)
        m[:, : 40 + 5 * i] = False
        masks.append(m)
    mesh, vol = o3d_tsdf_fusion(model, cams, masks=[torch.from_numpy(m) for m in masks], voxel_size=VOXEL, sdf_truc=TRUNC,
                                return_volume=True)
    ref = R.Volume(VOXEL, TRUNC)
    maps = _host_maps(model, cams)
    for v in _views(maps, cams, masks):
        ref.integrate(*v)
    _compare_volumes(vol, ref)
    unmasked = R.Volume(VOXEL, TRUNC)
    for v in _views(maps, cams):
        unmasked.integrate(*v)
    assert len(ref.units) < len(unmasked.units)


def test_small_pool_regrows_to_the_same_mesh(scene):
    from dn_splatter_b200.export_mesh import o3d_tsdf_fusion

    model, cams = scene
    big, vb = o3d_tsdf_fusion(model, cams, voxel_size=VOXEL, sdf_truc=TRUNC, capacity=100000, return_volume=True)
    small, vs = o3d_tsdf_fusion(model, cams, voxel_size=VOXEL, sdf_truc=TRUNC, capacity=4, return_volume=True)
    assert vb.regrows == 0 and vs.regrows > 0
    for a, b in ((big.vertices, small.vertices), (big.vertex_colors, small.vertex_colors), (big.triangles, small.triangles)):
        assert torch.equal(a, b)


def test_extract_refuses_an_overflowed_volume():
    from dn_splatter_b200.export_mesh import TSDFVolume
    from dn_splatter_b200.rasterize import DnrCapacityError

    views = _sphere_views()[:2]
    d, rgb, fx, fy, cx, cy, c2w, _ = views[0]
    vol = TSDFVolume(0.02, 0.06, device="cuda", capacity=2)
    vol.integrate(torch.from_numpy(d).cuda(), torch.from_numpy(np.ascontiguousarray(rgb)).cuda(), _cam(c2w, fx, fy, cx, cy, *d.shape[::-1]))
    assert vol.needed_units(lag=0) > 2
    with pytest.raises(DnrCapacityError):
        vol.extract_triangle_mesh()


def test_cpu_tensors_are_refused():
    from dn_splatter_b200 import _lib as L
    from dn_splatter_b200.export_mesh import TSDFVolume, TriangleMesh, filter_small_clusters

    vol = TSDFVolume(device="cuda")
    with pytest.raises(L.DnrError):
        vol.integrate(torch.zeros(4, 4), torch.zeros(4, 4, 3), None)
    with pytest.raises(L.DnrError):
        filter_small_clusters(TriangleMesh(torch.zeros(3, 3), torch.zeros(3, 3), torch.zeros(1, 3, dtype=torch.int32)))
