#!/usr/bin/env python
"""bench.py — rendered Mpix/s (forward+backward, RGB + depth + normal) of the dn-splatter hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py ... --dump-outputs DIR                         # + the last timed step's results as DIR/*.npy
    python bench.py --impl reference ...                           # the reference's CPU path (oracle port)
    torchrun --nproc-per-node N ... bench.py --gpus N ...          # one rank per GPU, per-camera sharding

A step = one training iteration of the reference on one batch: every rank renders ONE 1080p view of the 1M-Gaussian
synthetic scene through the public API (DNSplatterModel.get_outputs -> get_loss_dict -> backward -> optimizer step):
project -> bin/sort (supertile lists) -> composite RGB+depth+normal -> depth fill + surface normal -> photometric loss
(0.8 L1 + 0.2 (1-SSIM), the reference's default ssim_lambda) + DNRegularization (EdgeAwareLogL1 depth, L1+TV normal,
min-scale) -> raster backward (loss gradients evaluated in its prologue) -> projection backward (straight into the flat
gradient bucket) -> [N>1: one NCCL all-reduce of the bucket] -> Adam step of the six parameter groups (one launch).
`value` is measured with the supervision maps resident in HBM; `e2e` pulls each step's maps from pinned host
memory (H2D inside the timed region) and reads the loss back (D2H).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "rendered Mpix/s (fwd+bwd, RGB+depth+normal)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n-gauss", type=int, default=1_000_000)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--views", type=int, default=200)
    ap.add_argument("--gt-sets", type=int, default=16, help="distinct supervision-map sets cycled over the views")
    ap.add_argument("--no-normals", action="store_true", help="BASELINE config C2 literal: RGB+depth only")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--cpu-crop", default="512x288")
    ap.add_argument("--sync", action="store_true", help="read the intersection count back every view (host sync)")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of the CUDA-graph captured step")
    ap.add_argument("--no-graph-multi", action="store_true", help="multi-rank runs: launch eagerly instead of replaying the "
                                                                   "captured step (the all-reduce stays outside the graph)")
    ap.add_argument("--no-ssim", action="store_true", help="ssim_lambda = 0 (round-1 step: L1 only)")
    ap.add_argument("--no-optimizer", action="store_true", help="leave the Adam step out of the step (round-1 step)")
    ap.add_argument("--list-shift", type=int, default=2, help="intersection lists per (16 << s)-pixel supertile")
    ap.add_argument("--variant", type=int, default=0, help="raster kernel tuning knob (A/B timing)")
    ap.add_argument("--no-fused-loss-bwd", action="store_true", help="loss gradients as images from separate kernels (A/B)")
    ap.add_argument("--nccl-allreduce", action="store_true", help="multi-rank: dense NCCL all-reduce of the bucket + Adam instead "
                                                                  "of the peer-memory reduction fused into the Adam pass")
    ap.add_argument("--epochs", type=int, default=0, help="extra measurement after the --steps timed steps: median ms/view "
                                                          "over this many passes over ALL views (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step produced (loss, per-parameter gradients, "
                         "parameters after the Adam step; a fixed seeded sample of the Gaussians) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_BYTES = 64_000_000  # the whole --dump-outputs set stays below this


def dump_outputs(out_dir, model, bucket, loss):
    """Writes the results of the last training step as float32 .npy files: `loss`, and for every optimised parameter
    `<name>` (its value after the optimizer step) and `grad_<name>` (this rank's gradient of the step).  Both are
    restricted to the same rows: all Gaussians if they fit in DUMP_BYTES, else a sorted sample drawn with a fixed seed,
    so the rows depend only on the Gaussian count."""
    import numpy as np

    params = {n: model.gauss_params[n].detach() for n in bucket.names}
    n = next(iter(params.values())).shape[0]
    row_bytes = 2 * 4 * sum(p[0].numel() for p in params.values())
    rows = min(n, (DUMP_BYTES - 65536) // row_bytes)  # 64 KB for the loss and the .npy headers
    idx = torch.arange(n) if rows == n else torch.randperm(n, generator=torch.Generator().manual_seed(0))[:rows].sort().values
    idx = idx.to(params[bucket.names[0]].device)
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss.detach().float().reshape(1)}
    for name, p in params.items():
        arrays[name] = p.index_select(0, idx)
        arrays[f"grad_{name}"] = bucket.views[name].index_select(0, idx)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.float().cpu().numpy())
    return rows


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clocks / throttle reasons every 200 ms while the timed region runs, in-process through NVML
    (nvidia_ml_py).  A resident `nvidia-smi -lms` poller was measured to stall kernel launches on these hosts
    (the sampled run was 3-6x slower than the unsampled e2e run), so it is only the fallback."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self.thread, self.how = None, None

    def _loop_nvml(self, nv, h):
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.2)

    def start(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            h = nv.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.how = "nvml"
            self.thread = threading.Thread(target=self._loop_nvml, args=(nv, h), daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.how = "nvidia-smi (single shots before/after)"
            self._smi_once()

    def _smi_once(self):
        try:
            out = subprocess.run(["nvidia-smi", f"--id={self.index}", "--query-gpu=clocks.sm,clocks.max.sm,"
                                  "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                                  "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap",
                                  "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
            f = [x.strip() for x in out.strip().split(",")]
            self.samples.append(float(f[0]))
            self.max_mhz = float(f[1])
            for nm, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[2:6]):
                if v.lower().startswith("active"):
                    self.reasons.add(nm)
        except Exception:  # noqa: BLE001
            pass

    def stop(self):
        self._stop.set()
        if self.thread is not None:
            self.thread.join(timeout=2)
        else:
            self._smi_once()
        sm = sorted(self.samples)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(sm), "how": self.how}


# ------------------------------------------------------------------------------------------------ workload
def build_workload(args, device, normals: bool):
    from dn_splatter_b200.cameras import Cameras
    from dn_splatter_b200.dn_model import DNSplatterModelConfig
    from dn_splatter_b200.losses import DepthLossType
    from dn_splatter_b200.synthetic import make_scene, ring_cameras

    cfg = DNSplatterModelConfig(
        random_init=True, num_random=16, use_depth_loss=True, depth_lambda=0.2, depth_loss_type=DepthLossType.EdgeAwareLogL1,
        predict_normals=normals, use_normal_loss=normals, normal_supervision="mono",
        ssim_lambda=0.0 if args.no_ssim else 0.2, background_color="black", sync_free=not args.sync,
        list_shift=args.list_shift, fuse_loss_backward=not args.no_fused_loss_bwd,
    )
    model = cfg.setup(device=device)
    model.load_gaussians(make_scene(args.n_gauss, seed=0))
    model.background_color = torch.tensor([0.1490, 0.1647, 0.2157])
    model.step = 30000  # full SH degree (sh_degree_interval schedule done)
    model.train()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    peer = world > 1 and not args.nccl_allreduce and not args.no_optimizer
    try:
        bucket = model.enable_flat_grads(peer=peer)
    except Exception as exc:  # noqa: BLE001 — no symmetric memory on this box: keep the NCCL path and say so
        print(f"[bench] peer-memory bucket unavailable ({type(exc).__name__}: {exc}); using NCCL all-reduce", file=sys.stderr)
        bucket = model.enable_flat_grads(peer=False)
    model.__dict__["_raster_variant"] = args.variant
    cams = [Cameras(c["c2w"][None], c["fx"], c["fy"], c["cx"], c["cy"], c["width"], c["height"],
                    metadata={"cam_idx": i}) for i, c in enumerate(ring_cameras(args.views, args.width, args.height))]
    return model, bucket, cams


def make_gt_sets(model, cams, args, normals: bool, n_sets: int):
    """Synthetic supervision (SURVEY §8d): gt rgb = U[0,1) as uint8, gt depth = the scene's own depth rendered
    from a perturbed copy (dense, > 0.1), gt normal = normal_from_depth_image(gt depth) in [0,1]."""
    from dn_splatter_b200.utils.normal_utils import normal_from_depth_image

    g = torch.Generator().manual_seed(1)
    H, W = args.height, args.width
    sets = []
    saved = model.gauss_params["means"].data
    model.gauss_params["means"].data = saved + 0.01 * torch.randn(saved.shape, generator=g).to(saved.device)
    with torch.no_grad():
        for s in range(n_sets):
            cam = cams[(s * max(1, len(cams) // n_sets)) % len(cams)]
            out = model.get_outputs(cam)
            depth = out["depth"].clone()
            depth = torch.where(depth > 0.1, depth, torch.full_like(depth, 5.0))
            batch = {"image": (torch.rand(H, W, 3, generator=g) * 255).to(torch.uint8), "mono_depth": depth.cpu()}
            if normals:
                n = normal_from_depth_image(depth, float(cam.fx[0, 0]), float(cam.fy[0, 0]), float(cam.cx[0, 0]),
                                            float(cam.cy[0, 0]), (W, H), torch.eye(4, device=depth.device), depth.device)
                n01 = (1 + torch.cat([n[..., :1], -n[..., 1:]], dim=-1)) / 2
                batch["normal"] = (n01 * 255).round().to(torch.uint8).cpu()  # mono normals ship as 8-bit maps (as PNGs do)
            sets.append(batch)
    model.gauss_params["means"].data = saved
    return sets


def run_step(model, bucket, cam, batch, reduce=True, optimizer=None):
    bucket.zero_()
    outputs = model.get_outputs(cam)
    loss_dict = model.get_loss_dict(outputs, dict(batch))
    loss = loss_dict["main_loss"] + loss_dict["scale_reg"]
    loss.backward()
    if reduce and optimizer is not None and hasattr(bucket, "peer_flat"):
        optimizer.step_reduce(bucket)
        return loss
    if reduce:
        bucket.all_reduce()
    if optimizer is not None:
        optimizer.step()
    return loss


# ------------------------------------------------------------------------------------------------ CPU baseline
def cpu_reference_sample(args, normals: bool, crop: str, steps: int = 1, warmup: int = 0):
    """The reference's pure-PyTorch CPU path (oracle/: gsplat-1.0.0 restatement + dn-splatter glue + the
    reference's regularisers), forward+backward(+SSIM, +Adam), on a centred crop of the SAME scene's views: `warmup`
    untimed then `steps` timed iterations, iteration s on view (37 s) mod views like the CUDA arm.  Returns the
    cpu_baseline object (value = crop Mpix / mean seconds per timed step) and the mean seconds per step."""
    from dn_splatter_b200.synthetic import BACKGROUND, make_scene, ring_cameras
    from oracle import dn_ref

    # torch's intra-op pool thrashes on the per-tile tensors beyond ~16 threads (measured: 128 threads are 100x slower
    # than 8 on this path), so the port uses at most 16 of the host's cores and reports that number.
    cores = min(os.cpu_count() or 1, 16)
    torch.set_num_threads(cores)
    cw, ch = (int(x) for x in crop.split("x"))
    cw, ch = min(cw, args.width), min(ch, args.height)
    params = {k: v.requires_grad_(True) for k, v in make_scene(args.n_gauss, seed=0).items()}
    cams = ring_cameras(args.views, args.width, args.height)
    g = torch.Generator().manual_seed(1)
    gt_img = torch.rand(ch, cw, 3, generator=g).clamp(min=10 / 255.0)
    opt = None
    if not args.no_optimizer:  # the reference's per-group Adam (dn_config.py:29-68), stepped inside the sample like ours
        from dn_splatter_b200.dn_config import optimizer_groups

        groups = optimizer_groups()
        opt = [torch.optim.Adam([p], lr=groups[k]["lr"], eps=groups[k]["eps"]) for k, p in params.items() if k in groups]
    times = []
    for s in range(warmup + steps):
        cam = cams[(VIEW_STRIDE * s) % len(cams)]
        cx, cy = cam["cx"] - (args.width - cw) / 2, cam["cy"] - (args.height - ch) / 2
        for p in params.values():
            p.grad = None
        t0 = time.perf_counter()
        out = dn_ref.get_outputs(params, cam["c2w"], cam["fx"], cam["fy"], cx, cy, cw, ch, torch.tensor(BACKGROUND),
                                 predict_normals=normals)
        gt_depth = (out["depth"].detach() + 0.05).clamp(min=0.2)
        gt_normal = out["surface_normal"].detach()
        reg = dn_ref.dn_regularization(out["depth"], gt_depth, out["normal"], gt_normal, params["scales"], gt_img,
                                       depth_lambda=0.2, use_normal_loss=normals)
        l1 = (out["rgb"] - gt_img).abs().mean()
        if args.no_ssim:
            photo = l1
        else:  # torchmetrics SSIM restated in torch (the reference's default ssim_lambda = 0.2, dn_model.py:180,624-628)
            from dn_splatter_b200.dn_model import ssim

            photo = 0.8 * l1 + 0.2 * (1 - ssim(gt_img.permute(2, 0, 1)[None], out["rgb"].permute(2, 0, 1)[None]))
        loss = photo + reg
        loss.backward()
        if opt is not None:
            for o in opt:
                o.step()
        if s >= warmup:
            times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    sample = (f"{steps} view(s) (+{warmup} warm-up), centred {cw}x{ch} crop of the {args.width}x{args.height} frame, "
              f"N={args.n_gauss}, fwd+bwd{'' if args.no_ssim else '+SSIM'}{'' if args.no_optimizer else '+Adam(dense, all N)'}, "
              f"{dt:.1f} s per view")
    return {"value": cw * ch / 1e6 / dt, "unit": "Mpix/s", "cores": cores, "kind": "port",
            "sample": sample + "; oracle/ = CPU port of gsplat-1.0.0 + the reference's own loss code (gsplat is CUDA-only "
                               "and absent)"}, dt


def reference_crop(args) -> str:
    """The bounded sample of the reference arm: one view costs ~7-8 s on 16 cores at 512x288, so K + W iterations stay
    within a few minutes by shrinking the window when many are asked for."""
    n = args.steps + args.warmup
    if args.cpu_crop != "512x288" or n <= 30:
        return args.cpu_crop
    return "384x216" if n <= 60 else "256x144"


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    normals = not args.no_normals
    crop = reference_crop(args)
    last, dt = cpu_reference_sample(args, normals, crop, steps=args.steps, warmup=args.warmup)
    v = last["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "Mpix/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, normals, 1, sample=f"each step = ONE view cropped to the centred {crop} window of the "
                                                              f"{args.width}x{args.height} frame (the full frame takes minutes per view on "
                                                              f"the host); Mpix/s counts the crop's pixels only"),
        "cpu_baseline": last,
        "e2e": {"value": v, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, normals, world, sample=None):
    ssim = not args.no_ssim
    opt = not args.no_optimizer
    cfg = {
        "workload": f"BASELINE configs[1]: {args.n_gauss} Gaussians, {args.views} synthetic ring views {args.width}x{args.height}, "
                    f"{'RGB+depth+normal' if normals else 'RGB+depth'} render fwd+bwd, 1 view per GPU per step",
        "n_gauss": args.n_gauss, "width": args.width, "height": args.height, "views": args.views, "sh_degree": 3,
        "normals": normals,
        "losses": ("0.8 L1 + 0.2 (1-SSIM) rgb (the reference's default ssim_lambda)" if ssim else "L1 rgb")
                  + " + DNRegularization(EdgeAwareLogL1 depth (1+0.2), L1+TV normal, min-scale)",
        "optimizer": "Adam over the six parameter groups with the reference's learning rates, inside the step" if opt else "not in the step",
        "parallelism": (f"per-camera sharding x{world}, " + ("dense NCCL all-reduce of the gradient bucket, then Adam"
                        if (args.nccl_allreduce or args.no_optimizer) else "gradient rows gathered over NVLink peer memory inside the Adam pass"))
                       if world > 1 else "single GPU",
        "l2_policy": "inputs larger than L2 (236 MB parameters + 236 MB gradients + 472 MB Adam moments per step; a different "
                     "view and supervision set every step)",
        "gt_sets": args.gt_sets, "view_order": "step s renders view (37 s) mod views of the rank's shard (the ring is sampled evenly)",
    }
    if sample is not None:
        cfg["sample"] = sample
    return cfg


VIEW_STRIDE = 37  # coprime with 200: K consecutive steps sample the camera ring evenly


def view_of(step: int, my_views):
    return my_views[(step * VIEW_STRIDE) % len(my_views)]


# ------------------------------------------------------------------------------------------------ main (ours)
def main():
    args = parse()
    if args.impl == "reference":
        reference_arm(args)
        return
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (impl=ours) needs a GPU: there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    torch.cuda.set_stream(torch.cuda.Stream(device=device))  # never the legacy default stream (CUDA-graph friendly)
    if world > 1:
        import datetime

        dist.init_process_group("nccl", device_id=device, timeout=datetime.timedelta(seconds=180))
    normals = not args.no_normals
    import dn_splatter_b200.rasterize as R
    from dn_splatter_b200.optim import FusedAdam

    model, bucket, cams = build_workload(args, device, normals)
    optimizer = None if args.no_optimizer else FusedAdam.for_model(model)
    stats_dev = torch.zeros(4, dtype=torch.int64, device=device)
    my_views = list(range(rank, len(cams), world)) or [0]
    host_sets = make_gt_sets(model, cams, args, normals, args.gt_sets)
    dev_sets = [{k: v.to(device) for k, v in b.items()} for b in host_sets]
    pin_sets = [{k: v.pin_memory() for k, v in b.items()} for b in host_sets]
    h2d_bytes = sum(v.numel() * v.element_size() for v in host_sets[0].values())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n_steps, step_fn):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in range(n_steps):
            step_fn(s)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    graphed = None

    peer_reduce = hasattr(bucket, "peer_flat")

    def finish_step():
        """What follows the (captured) forward + backward: gradient reduction and the Adam step — one fused pass over
        NVLink peer memory (dnr_adam_step_reduce), or NCCL all-reduce then Adam."""
        if peer_reduce:
            optimizer.step_reduce(bucket)
            return
        bucket.all_reduce()
        if optimizer is not None:
            optimizer.step()

    last = {}  # the loss of the latest resident step (for --dump-outputs); detached, so no autograd graph outlives its step

    def resident_step(s):
        cam = cams[view_of(s, my_views)]
        if graphed is None:
            last["loss"] = run_step(model, bucket, cam, dev_sets[s % len(dev_sets)], optimizer=optimizer).detach()
        else:  # supervision maps: device-resident set -> the graph's static buffers (D2D), then ONE graph launch
            for k, v in dev_sets[s % len(dev_sets)].items():
                graphed.batches[0][k].copy_(v, non_blocking=True)
            last["loss"] = graphed(cam, 0)
            finish_step()

    losses = []
    copy_stream = torch.cuda.Stream(device=device)
    loss_host = torch.zeros(64, dtype=torch.float32).pin_memory()
    NBUF = 3  # device staging buffers (allocated once: no allocator traffic, no cross-stream frees in the timed region)
    stage = [{k: torch.empty_like(v, device=device) for k, v in pin_sets[0].items()} for _ in range(NBUF)]

    def use_graph_buffers():
        nonlocal NBUF, stage
        NBUF, stage = len(graphed.batches), graphed.batches  # H2D straight into the graph's static buffers

    ready = [torch.cuda.Event() for _ in range(NBUF)]     # H2D of the slot finished (recorded on the copy stream)
    consumed = [torch.cuda.Event() for _ in range(NBUF)]  # compute that read the slot finished (compute stream)
    state = {"prefetched": -1, "pending": []}

    def prefetch(s):
        """H2D of step s's supervision maps on the copy stream (overlaps the previous step's compute)."""
        slot = s % NBUF
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])  # the step that last used this slot has finished reading it
            for k, v in pin_sets[s % len(pin_sets)].items():
                stage[slot][k].copy_(v, non_blocking=True)
            ready[slot].record(copy_stream)
        state["prefetched"] = s

    def e2e_step(s):
        if state["prefetched"] < s:
            prefetch(s)
        slot = s % NBUF
        cur = torch.cuda.current_stream()
        cur.wait_event(ready[slot])
        prefetch(s + 1)
        cam = cams[view_of(s, my_views)]
        if graphed is None:
            loss = run_step(model, bucket, cam, stage[slot], optimizer=optimizer)
        else:
            loss = graphed(cam, slot)
            finish_step()
        consumed[slot].record(cur)
        ls = s % 64
        loss_host[ls:ls + 1].copy_(loss.detach().reshape(1), non_blocking=True)  # D2H read of the step's result
        rev = torch.cuda.Event()
        rev.record()
        state["pending"].append((ls, rev))
        while len(state["pending"]) > 2:  # consume results at most 2 steps late
            sl, e = state["pending"].pop(0)
            e.synchronize()
            losses.append(float(loss_host[sl]))

    def e2e_flush():
        for sl, e in state["pending"]:
            e.synchronize()
            losses.append(float(loss_host[sl]))
        state["pending"] = []
        state["prefetched"] = -1

    # untimed setup: visit every view of this rank once (camera caches, intersection-capacity statistics) — a training
    # run revisits each view thousands of times; then the warm-up steps, then the timed device-resident run
    with torch.no_grad():
        for v in my_views:
            model.get_outputs(cams[v])
    for s in range(max(3, args.warmup)):
        resident_step(s)
    launches_per_step, graph_error = None, None
    if not args.no_graph and (world == 1 or not args.no_graph_multi):
        from dn_splatter_b200 import _lib as _L0
        from dn_splatter_b200.graph_step import GraphedTrainStep

        l0 = dict(_L0.LAUNCHES)
        try:
            graphed = GraphedTrainStep(model, bucket, cams[my_views[0]], dev_sets[0], n_slots=3, warmup=2)
        except Exception as exc:  # noqa: BLE001 — keep measuring with eager launches rather than losing the run
            graphed, graph_error = None, f"{type(exc).__name__}: {exc}"[:300]
            torch.cuda.synchronize()
        if graphed is not None:
            n_eager = 2 + 3  # warm-up calls + one capture per slot
            launches_per_step = {k: (_L0.LAUNCHES[k] - l0[k]) // n_eager for k in l0}
            use_graph_buffers()
        for s in range(3):
            resident_step(s)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    from dn_splatter_b200 import _lib as _L

    launches0 = dict(_L.LAUNCHES)
    ms = timed(args.steps, resident_step)
    launches = {k: _L.LAUNCHES[k] - launches0[k] for k in launches0}
    if launches_per_step is not None:  # graph replays re-issue the launches recorded at capture (+ the eager Adam step)
        launches = {k: v * args.steps + launches[k] for k, v in launches_per_step.items()}
    clocks = sampler.stop() if rank == 0 else None
    dumped_rows = None
    if args.dump_outputs and rank == 0:  # before anything else runs a step: the e2e / epoch passes below train further
        dumped_rows = dump_outputs(args.dump_outputs, model, bucket, last["loss"])
    pix = args.width * args.height
    value = world * args.steps * pix / 1e6 / (ms / 1e3)

    e2e = None
    if not args.skip_e2e:
        for s in range(3):
            e2e_step(s)
        e2e_flush()

        def e2e_run(s):
            e2e_step(s)
            if s == args.steps - 1:
                e2e_flush()

        ms_e = timed(args.steps, e2e_run)
        e2e = {"value": world * args.steps * pix / 1e6 / (ms_e / 1e3), "unit": "Mpix/s", "h2d_bytes_per_step": h2d_bytes,
               "d2h_bytes_per_step": 4, "ms_per_step": ms_e / args.steps}

    # --epochs E (SURVEY §8d asks for >= 5): median over E passes over the whole view set; the K timed steps above stay
    # the headline
    epochs = None
    if args.epochs > 0:
        per_epoch = []
        n_v = len(my_views)
        for ep in range(args.epochs):
            per_epoch.append(timed(n_v, lambda s, ep=ep: resident_step(ep * n_v + s)) / n_v)
        per_epoch.sort()
        med = per_epoch[len(per_epoch) // 2]
        epochs = {"epochs": args.epochs, "views_per_epoch_per_rank": n_v, "median_ms_per_step": med,
                  "min_ms_per_step": per_epoch[0], "max_ms_per_step": per_epoch[-1], "median_value": world * pix / 1e6 / (med / 1e3),
                  "unit": "Mpix/s"}
    if graphed is not None:
        graphed.check_capacity(wait=True)  # raises if any replayed view was truncated

    # per-stage device times (CUDA events on the launching stream) for the roofline of the dominant kernel
    stages, roof = {}, None
    graph_info = ({"capacity": graphed.capacity, "slots": len(graphed.graphs), "max_count": graphed.max_count} if graphed is not None
                  else ({"error": graph_error, "fallback": "eager launches"} if graph_error else None))
    graphed = None  # the instrumented pass below runs eagerly
    if rank == 0:
        R.STAGE_EVENTS = []
        model.__dict__["_raster_stats"] = stats_dev
        n_prof = min(args.steps, 10)
        for s in range(n_prof):  # rank 0 only: no collective in here
            run_step(model, bucket, cams[view_of(s, my_views)], dev_sets[s % len(dev_sets)], reduce=False, optimizer=optimizer)
        torch.cuda.synchronize()
        model.__dict__["_raster_stats"] = None
        for name, a, b in R.STAGE_EVENTS:
            stages[name] = stages.get(name, 0.0) + a.elapsed_time(b) / n_prof
        R.STAGE_EVENTS = None
        walked_f, kept_f, walked_b, kept_b = (x / n_prof for x in stats_dev.tolist())
        info = model.raster_out.info
        I = int(info["n_isects_dev"])
        H, W = args.height, args.width
        i_eff = int(kept_b)  # (tile, Gaussian) pairs the backward composites: kept by the tile filter up to the deepest last id
        cn = 1 if normals else 0
        P = H * W
        from json import load as _jl

        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = float(_jl(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
        G = 48 + 12 * cn
        alg = {
            "raster_bwd": (28 + 12 * cn) * P + (20 + 12 * cn) * P + (4 + 44 + 12 * cn) * i_eff + G * i_eff,
            "raster_fwd": (4 + 44 + 12 * cn) * int(kept_f) + (28 + 12 * cn) * P,
            "bin_sort": 44 * I,
            "project_fwd": (44 + 32 + 12 * 16 + 12 + 12 * cn) * args.n_gauss,
            "project_bwd": (G + 44 + 44 + 12 * 16) * args.n_gauss,
        }
        dom = max((k for k in stages if k in alg), key=lambda k: stages[k])
        ach = alg[dom] / (stages[dom] / 1e3) / 1e9
        traffic = None  # dram__bytes_read.sum + dram__bytes_write.sum of that kernel from the committed ncu --set full capture
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            t = _jl(open(tpath))
            key = f"{dom}:{args.n_gauss}:{args.width}x{args.height}:{'n' if normals else 'c'}"
            traffic = t.get(key, {}).get("dram_bytes_per_launch")
        roof = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg[dom],
                "n_isects": I, "n_isects_composited": i_eff, "ms_per_launch": stages[dom],
                "list_entries_walked_fwd": int(walked_f), "kept_by_tile_filter_fwd": int(kept_f),
                "list_entries_walked_bwd": int(walked_b), "list_tile_px": info["list_tile"]}

    cpu = None
    if rank == 0 and not args.skip_cpu_baseline and world == 1:
        cpu, _ = cpu_reference_sample(args, normals, args.cpu_crop, steps=2)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "Mpix/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args, normals, world), "clocks": clocks, "e2e": e2e,
            "gpu_launches": launches["handwritten"],
            "gpu_launches_note": f"hand-written dnr kernels counted at the C-ABI calls of the timed region; the same calls ran "
                                 f"{launches['cub']} cub radix-sort/scan passes (compiled into libdnr_b200.so)",
            "roofline": roof, "stages_ms": stages, "epochs": epochs, "cpu_baseline": cpu, "last_loss": losses[-1] if losses else None,
            "cuda_graph": graph_info, "isect_capacity_report": {str(k): v for k, v in R.capacity_report().items()},
        }
        if dumped_rows is not None:
            line["dump_outputs"] = {"dir": args.dump_outputs, "step": args.steps - 1, "gaussian_rows": dumped_rows}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
