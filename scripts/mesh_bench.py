"""o3dtsdf mesh export timing on the device (not bench.py): render + TSDF allocate + integrate per view, then extraction
and the cluster filter, on the C2 workload (1M Gaussians, 200 ring views at 1920x1080), voxel 0.02 m / truncation
0.06 m (the exporter defaults' 3:1 ratio).  The synthetic scene is random Gaussians filling a 10 m cube rather than a
surface, so the band of touched units is thick: the allocated units and their bytes are reported beside the timings.
Prints one JSON line.

    python scripts/mesh_bench.py [--gaussians N] [--views V] [--width W --height H] [--voxel 0.02 --trunc 0.06]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU


def card():
    import torch

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True)
    return {"gpu": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gaussians", type=int, default=1_000_000)
    ap.add_argument("--views", type=int, default=200)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--voxel", type=float, default=0.02)
    ap.add_argument("--trunc", type=float, default=0.06)
    ap.add_argument("--capacity", type=int, default=1 << 17)
    args = ap.parse_args()

    import torch

    from dn_splatter_b200 import _lib as L
    from dn_splatter_b200.cameras import Cameras
    from dn_splatter_b200.dn_model import DNSplatterModelConfig
    from dn_splatter_b200.export_mesh import TSDFVolume, filter_small_clusters
    from dn_splatter_b200.render_service import ViewRenderer
    from dn_splatter_b200.synthetic import make_scene, ring_cameras

    if not torch.cuda.is_available():
        raise SystemExit("mesh_bench.py needs a CUDA device")
    model = DNSplatterModelConfig(random_init=True, num_random=16, background_color="black", ssim_lambda=0.0).setup(device="cuda")
    model.load_gaussians(make_scene(args.gaussians, seed=0))
    model.step = 30000
    cams = [Cameras(c["c2w"][None].cuda(), c["fx"], c["fy"], c["cx"], c["cy"], c["width"], c["height"])
            for c in ring_cameras(args.views, args.width, args.height)]
    renderer = ViewRenderer(model, keys=("rgb", "depth"), to_host=False)
    for _ in renderer.render(cams[:3]):  # capture the graphs, warm up
        pass
    torch.cuda.synchronize()

    # render alone
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in renderer.render(cams):
        pass
    e1.record()
    torch.cuda.synchronize()
    render_ms = e0.elapsed_time(e1)

    # fused: allocate and integrate bracketed by events
    lib = L.load()
    spans = {"dnr_tsdf_allocate": [], "dnr_tsdf_integrate": []}
    for name in spans:
        fn = getattr(lib, name)

        def timed(*a, _fn=fn, _name=name):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            rc = _fn(*a)
            e.record()
            spans[_name].append((s, e))
            return rc

        lib.__dict__[name] = timed
    vol = TSDFVolume(args.voxel, args.trunc, device="cuda", capacity=args.capacity)
    warm = TSDFVolume(args.voxel, args.trunc, device="cuda", capacity=args.capacity)  # first-launch costs off the clock
    for idx, maps in renderer.render(cams[:1]):
        warm.integrate(maps["depth"], maps["rgb"], cams[idx])
    del warm
    for v in spans.values():
        v.clear()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e0.record()
    for idx, maps in renderer.render(cams):
        vol.integrate(maps["depth"], maps["rgb"], cams[idx])
    e1.record()
    torch.cuda.synchronize()
    fuse_ms = e0.elapsed_time(e1)
    need = vol.needed_units(lag=0)
    if need:
        raise SystemExit(f"--capacity {args.capacity} is too small: the views need {need} units")
    alloc_ms = sum(s.elapsed_time(e) for s, e in spans["dnr_tsdf_allocate"])
    integ_ms = sum(s.elapsed_time(e) for s, e in spans["dnr_tsdf_integrate"])
    e0.record()
    mesh = vol.extract_triangle_mesh()
    e1.record()
    torch.cuda.synchronize()
    extract_ms = e0.elapsed_time(e1)
    e0.record()
    clean = filter_small_clusters(mesh)
    e1.record()
    torch.cuda.synchronize()
    filter_ms = e0.elapsed_time(e1)
    wall_s = time.perf_counter() - t0
    n_units = vol.n_units
    updates = float(vol.voxels[:n_units, 1].double().sum()) if n_units else 0.0  # each update adds 1 to a weight
    out = {
        "workload": {"gaussians": args.gaussians, "views": args.views, "width": args.width, "height": args.height,
                     "voxel_size": args.voxel, "sdf_truc": args.trunc},
        "card": card(),
        "ms_per_view": {"render": render_ms / args.views, "allocate": alloc_ms / args.views, "integrate": integ_ms / args.views,
                        "fused_loop": fuse_ms / args.views},
        "ms": {"render_all": render_ms, "fuse_all": fuse_ms, "extract": extract_ms, "filter": filter_ms,
               "total": fuse_ms + extract_ms + filter_ms},
        "wall_s_fuse_extract_filter": wall_s,
        "units_allocated": n_units, "unit_bytes": n_units * 5 * 4096 * 4,
        "voxel_updates": updates,
        "vertices": int(mesh.vertices.shape[0]), "triangles": int(mesh.triangles.shape[0]),
        "vertices_filtered": int(clean.vertices.shape[0]), "triangles_filtered": int(clean.triangles.shape[0]),
        "integrate_bytes_per_s": 40.0 * updates / (integ_ms * 1e-3) if integ_ms > 0 else None,
        "integrate_share_of_hbm_peak": 40.0 * updates / (integ_ms * 1e-3) / HBM_BYTES_PER_S if integ_ms > 0 else None,
    }
    print(json.dumps(out))


if __name__ == "__main__":
    main()
