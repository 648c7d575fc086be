"""ctypes binding of libdnr_b200.so (include/dnr.h).  There is NO fallback: if the library is missing
or a call fails, this module raises."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libdnr_b200.so")

FLAG_ACTIVATED, FLAG_ANTIALIASED, FLAG_NORMALS, FLAG_ACCUMULATE, FLAG_EXACT_LISTS = 1, 2, 4, 8, 16
FLAG_HOST_CAMERA = 32
FLAG_COMPACT_BWD = 64
FLAG_TOUCHED_BWD = 128
LOSS_FUSED_BWD, LOSS_IMG_U8, LOSS_NORMAL_U8, LOSS_EDGE_FROM_IMAGE = 1, 2, 4, 8
REC_FLOATS, REC_FLOATS_N, GRAD_FLOATS = 12, 16, 16
DEPTH_LOSS_TYPES = {None: 0, "EdgeAwareLogL1": 1, "LogL1": 2, "L1": 3, "MSE": 4}

_f, _i, _p = C.c_float, C.c_int32, C.c_void_p


class DnrArgs(C.Structure):
    """Field-for-field mirror of `struct DnrArgs` in include/dnr.h (tests/test_abi.py checks the order)."""

    _fields_ = [
        ("n_gauss", _i), ("width", _i), ("height", _i), ("tile_size", _i), ("sh_degree", _i), ("sh_bases", _i),
        ("flags", C.c_uint32), ("list_shift", _i),
        ("near_plane", _f), ("far_plane", _f), ("eps2d", _f), ("radius_clip", _f),
        ("background", _f * 3), ("reserved1", _f),
        ("n_isects", C.c_int64),
        ("viewmat", _p), ("K", _p), ("c2w", _p),
        ("means", _p), ("quats", _p), ("scales", _p), ("opacities", _p), ("sh_dc", _p), ("sh_rest", _p),
        ("radii", _p), ("means2d", _p), ("depths", _p), ("conics", _p), ("opac_act", _p), ("compensations", _p),
        ("colors", _p), ("normals_world", _p), ("tiles_per_gauss", _p), ("depth_keys", _p), ("records", _p), ("cull_lim", _p),
        ("ws_scan", _p), ("ws_sort", _p), ("flatten_ids", _p), ("tile_offsets", _p), ("n_isects_dev", _p),
        ("out_rgb", _p), ("out_depth", _p), ("out_alpha", _p), ("out_normal", _p), ("out_surface_normal", _p),
        ("last_ids", _p), ("normal_norm", _p), ("clamp_mask", _p), ("depth_max", _p),
        ("v_rgb", _p), ("v_depth", _p), ("v_normal", _p), ("v_alpha", _p), ("grad_records", _p),
        ("v_means", _p), ("v_quats", _p), ("v_scales", _p), ("v_opacities", _p), ("v_sh_dc", _p), ("v_sh_rest", _p),
        ("v_means2d", _p), ("v_means2d_abs", _p),
        ("gt_depth", _p), ("gt_normal", _p), ("gt_rgb", _p), ("loss_partials", _p), ("v_loss", _p),
        ("depth_lambda", _f), ("depth_tolerance", _f), ("depth_loss_type", _i), ("use_normal_loss", _i),
        ("host_cam", _f * 32),
        ("depth_order", _p),
        ("loss_flags", C.c_uint32), ("variant", _i), ("gt_image", _p), ("v_l1", _p), ("touched", _p), ("stats", _p),
    ]


class DnrAdamSeg(C.Structure):
    """Mirror of struct DnrAdamSeg (include/dnr.h)."""

    _fields_ = [("p", _p), ("g", _p), ("m", _p), ("v", _p), ("n", C.c_int64), ("lr", C.c_double), ("eps", C.c_double),
                ("bc1", C.c_double), ("bc2_sqrt", C.c_double), ("dense", C.c_int64)]


PEER_MAX = 8


class DnrPeerReduce(C.Structure):
    """Mirror of struct DnrPeerReduce (include/dnr.h)."""

    _fields_ = [("world", _i), ("rank", _i), ("n_gauss", _i), ("reserved", _i), ("peer_flat", _p * PEER_MAX),
                ("peer_touched", _p * PEER_MAX), ("mask", _p)]


class DnrKnnGrid(C.Structure):
    """Mirror of struct DnrKnnGrid (include/dnr.h)."""

    _fields_ = [("lo", _f * 3), ("cell", _f), ("inv_cell", _f), ("dims", C.c_int32 * 3)]


class DnrTsdfVolume(C.Structure):
    """Mirror of struct DnrTsdfVolume (include/dnr.h)."""

    _fields_ = [("voxel_size", C.c_double), ("sdf_trunc", C.c_double), ("depth_trunc", _f), ("capacity", _i),
                ("hash_size", _i), ("reserved", _i), ("hash_keys", _p), ("hash_vals", _p), ("hash_stamp", _p),
                ("voxels", _p), ("touched", _p), ("counters", _p)]


class DnrTsdfView(C.Structure):
    """Mirror of struct DnrTsdfView (include/dnr.h)."""

    _fields_ = [("width", _i), ("height", _i), ("stamp", _i), ("reserved", _i), ("fx", _f), ("fy", _f), ("cx", _f), ("cy", _f),
                ("extrinsic", _f * 16), ("pose", C.c_double * 16), ("depth", _p), ("rgb", _p), ("mask", _p)]


POINTER_FIELDS = {n for n, t in DnrArgs._fields_ if t is _p}

_lib: Optional[C.CDLL] = None

# hand-written kernels launched per C-ABI call (cub's radix-sort / scan passes are counted separately)
KERNELS_PER_CALL = {
    "dnr_project_fwd": (1, 0), "dnr_bin_scan": (2, 8), "dnr_bin_sort": (3, 4), "dnr_raster_fwd": (1, 0),
    "dnr_finalize_fwd": (1, 0), "dnr_normal_from_depth": (1, 0), "dnr_raster_bwd": (1, 0), "dnr_project_bwd": (1, 0),
    "dnr_loss_fwd": (2, 0), "dnr_loss_bwd": (1, 0), "dnr_scale_loss_fwd": (1, 0), "dnr_scale_loss_bwd": (1, 0),
    "dnr_l1_fwd": (1, 0), "dnr_l1_bwd": (1, 0), "dnr_u8_to_f32": (1, 0),
    "dnr_ssim_fwd": (1, 0), "dnr_ssim_bwd": (1, 0), "dnr_ssim_fwd_ex": (1, 0), "dnr_ssim_bwd_ex": (1, 0), "dnr_photometric_fwd": (2, 0), "dnr_photometric_bwd": (1, 0), "dnr_adam_step": (1, 0), "dnr_adam_step_reduce": (2, 0),
    "dnr_knn_build": (2, 1), "dnr_knn_query": (1, 0), "dnr_density": (1, 0), "dnr_ray_densities": (1, 0),
    "dnr_tsdf_allocate": (1, 0), "dnr_tsdf_integrate": (1, 0), "dnr_tsdf_extract_count": (5, 3), "dnr_tsdf_extract_emit": (1, 0),
    "dnr_mesh_cluster_count": (8, 4), "dnr_mesh_cluster_emit": (1, 0),
}
LAUNCHES = {"handwritten": 0, "cub": 0}


class _Counting:
    """Thin proxy over the CDLL that counts kernel launches per call (bench.py's gpu_launches)."""

    def __init__(self, lib):
        self._lib = lib

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        k = KERNELS_PER_CALL.get(name)
        if k is None:
            return fn

        debug = os.environ.get("DNR_DEBUG_CAPTURE") == "1"

        def call(*args):
            LAUNCHES["handwritten"] += k[0]
            LAUNCHES["cub"] += k[1]
            rc = fn(*args)
            if debug:  # name the C-ABI call that invalidates an ongoing stream capture
                import torch

                try:  # raises cudaErrorStreamCaptureInvalidated once the capture is broken
                    torch.cuda.is_current_stream_capturing()
                except Exception as exc:  # noqa: BLE001
                    raise DnrError(f"stream capture invalidated by {name} (rc {rc}): {exc}") from exc
            return rc

        self.__dict__[name] = call
        return call


class DnrError(RuntimeError):
    pass


def load():
    """Loads the shared library, failing loudly when it has not been built (python -m dn_splatter_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DnrError(
            f"{LIB_PATH} is missing: build it with `python -m dn_splatter_b200.build` "
            "(nvcc, sm_100a). dn_splatter_b200 has no CPU or PyTorch fallback."
        )
    lib = C.CDLL(LIB_PATH)
    A = C.POINTER(DnrArgs)
    lib.dnr_version.restype = C.c_int
    lib.dnr_error_string.restype = C.c_char_p
    lib.dnr_error_string.argtypes = [C.c_int]
    for name in ("dnr_project_fwd", "dnr_bin_sort", "dnr_raster_fwd", "dnr_finalize_fwd", "dnr_normal_from_depth",
                 "dnr_raster_bwd", "dnr_project_bwd", "dnr_loss_fwd"):
        fn = getattr(lib, name)
        fn.restype = C.c_int
        fn.argtypes = [A, C.c_void_p]
    lib.dnr_bin_scan.restype = C.c_int
    lib.dnr_bin_scan.argtypes = [A, C.c_void_p, C.POINTER(C.c_int64)]
    lib.dnr_loss_bwd.restype = C.c_int
    lib.dnr_loss_bwd.argtypes = [A, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dnr_scale_loss_fwd.restype = C.c_int
    lib.dnr_scale_loss_fwd.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
    lib.dnr_scale_loss_bwd.restype = C.c_int
    lib.dnr_scale_loss_bwd.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dnr_l1_fwd.restype = C.c_int
    lib.dnr_l1_fwd.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]
    lib.dnr_l1_bwd.restype = C.c_int
    lib.dnr_l1_bwd.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dnr_u8_to_f32.restype = C.c_int
    lib.dnr_u8_to_f32.argtypes = [C.c_void_p, C.c_int64, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
    lib.dnr_ssim_fwd.restype = C.c_int
    lib.dnr_ssim_fwd.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dnr_ssim_fwd_ex.restype = C.c_int
    lib.dnr_ssim_fwd_ex.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_void_p]
    lib.dnr_ssim_bwd_ex.restype = C.c_int
    lib.dnr_ssim_bwd_ex.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p]
    lib.dnr_photometric_fwd.restype = C.c_int
    lib.dnr_photometric_fwd.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_void_p,
                                        C.c_void_p, C.c_void_p]
    lib.dnr_photometric_bwd.restype = C.c_int
    lib.dnr_photometric_bwd.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dnr_adam_step.restype = C.c_int
    lib.dnr_adam_step.argtypes = [C.c_void_p, C.c_int32, C.c_double, C.c_double, C.c_void_p]
    lib.dnr_adam_step_reduce.restype = C.c_int
    lib.dnr_adam_step_reduce.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_double, C.c_double, C.c_void_p, C.c_void_p]
    lib.dnr_knn_workspace_bytes.restype = C.c_int64
    lib.dnr_knn_workspace_bytes.argtypes = [C.c_int32, C.c_void_p]
    lib.dnr_knn_build.restype = C.c_int
    lib.dnr_knn_build.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    lib.dnr_knn_query.restype = C.c_int
    lib.dnr_knn_query.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                  C.c_void_p, C.c_void_p]
    lib.dnr_density.restype = C.c_int
    lib.dnr_density.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_int32, C.c_float, C.c_void_p, C.c_void_p]
    lib.dnr_ray_densities.restype = C.c_int
    lib.dnr_ray_densities.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dnr_ssim_bwd.restype = C.c_int
    lib.dnr_ssim_bwd.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p]
    lib.dnr_depth_order_ptr.restype = C.c_void_p
    lib.dnr_depth_order_ptr.argtypes = [C.c_void_p, C.c_int32]
    lib.dnr_bin_scan_workspace_bytes.restype = C.c_size_t
    lib.dnr_bin_scan_workspace_bytes.argtypes = [C.c_int32]
    lib.dnr_bin_sort_workspace_bytes.restype = C.c_size_t
    lib.dnr_bin_sort_workspace_bytes.argtypes = [C.c_int32, C.c_int64, C.c_int32]
    V, W = C.POINTER(DnrTsdfVolume), C.POINTER(DnrTsdfView)
    lib.dnr_tsdf_reset.restype = C.c_int
    lib.dnr_tsdf_reset.argtypes = [V, C.c_void_p]
    for name in ("dnr_tsdf_allocate", "dnr_tsdf_integrate"):
        getattr(lib, name).restype = C.c_int
        getattr(lib, name).argtypes = [V, W, C.c_void_p]
    lib.dnr_tsdf_extract_workspace_bytes.restype = C.c_int64
    lib.dnr_tsdf_extract_workspace_bytes.argtypes = [C.c_int32]
    lib.dnr_tsdf_extract_count.restype = C.c_int
    lib.dnr_tsdf_extract_count.argtypes = [V, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]
    lib.dnr_tsdf_extract_emit.restype = C.c_int
    lib.dnr_tsdf_extract_emit.argtypes = [V, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dnr_mesh_cluster_workspace_bytes.restype = C.c_int64
    lib.dnr_mesh_cluster_workspace_bytes.argtypes = [C.c_int32, C.c_int32]
    lib.dnr_mesh_cluster_count.restype = C.c_int
    lib.dnr_mesh_cluster_count.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]
    lib.dnr_mesh_cluster_emit.restype = C.c_int
    lib.dnr_mesh_cluster_emit.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int64,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    _lib = _Counting(lib)
    return _lib


EXPORTS = (
    "dnr_version", "dnr_error_string", "dnr_project_fwd", "dnr_bin_scan_workspace_bytes", "dnr_bin_scan",
    "dnr_bin_sort_workspace_bytes", "dnr_bin_sort", "dnr_depth_order_ptr", "dnr_raster_fwd", "dnr_finalize_fwd", "dnr_normal_from_depth",
    "dnr_raster_bwd", "dnr_project_bwd", "dnr_loss_fwd", "dnr_loss_bwd", "dnr_scale_loss_fwd", "dnr_scale_loss_bwd",
    "dnr_l1_fwd", "dnr_l1_bwd", "dnr_u8_to_f32", "dnr_ssim_fwd", "dnr_ssim_bwd", "dnr_ssim_fwd_ex", "dnr_ssim_bwd_ex", "dnr_photometric_fwd", "dnr_photometric_bwd", "dnr_adam_step", "dnr_adam_step_reduce", "dnr_knn_workspace_bytes", "dnr_knn_build", "dnr_knn_query",
    "dnr_density", "dnr_ray_densities", "dnr_tsdf_reset", "dnr_tsdf_allocate", "dnr_tsdf_integrate",
    "dnr_tsdf_extract_workspace_bytes", "dnr_tsdf_extract_count", "dnr_tsdf_extract_emit", "dnr_mesh_cluster_workspace_bytes",
    "dnr_mesh_cluster_count", "dnr_mesh_cluster_emit",
)


def check(code: int, what: str) -> None:
    if code != 0:
        msg = load().dnr_error_string(code).decode()
        raise DnrError(f"{what} failed with code {code}: {msg}")
