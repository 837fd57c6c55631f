"""ctypes binding of the C ABI declared in include/dgvcc_b200.h.

There is no CPU fallback anywhere in this package: if the shared library is missing it is
(re)built with nvcc, and if that fails -- or there is no CUDA device when a kernel is called --
the call raises.
"""
import ctypes
import os
import threading
from ctypes import POINTER, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p

from . import build as _build

_lock = threading.Lock()
_lib = None


class BLLayout(ctypes.Structure):
    """Mirror of struct dgvcc_bl_layout."""
    _fields_ = [(n, c_int64) for n in
                ("amax", "rz", "pbg", "ebg", "counts", "wsel", "residual", "loss_img", "ticket", "cpart", "zpart",
                 "minpart", "gpart", "total", "dens", "gfinal", "flags", "err", "push_ticket", "goff", "gsorted", "cshare", "ztick", "gtick", "queue")] + \
               [("tiles", c_int32), ("rows_per_thread", c_int32), ("cols_per_thread", c_int32), ("share_rows", c_int32)]


class BLPacked(ctypes.Structure):
    """Mirror of struct dgvcc_bl_packed."""
    _fields_ = [(n, c_int64) for n in
                ("total_points", "total_rows", "total_chunks", "multi_chunk", "meta_bytes", "off_points", "off_targets",
                 "total_bytes")]


BL_OPT_MIN_CELL, BL_OPT_BAND_TILE = 0, 1  # dgvcc_bl_set_option
BL_PHASES = 8  # DGVCC_BL_PHASES
BL_PH_DENS, BL_PH_MIN, BL_PH_Z, BL_PH_CNT, BL_PH_LOSS, BL_PH_GPART, BL_PH_GRAD, BL_PH_OUT = range(BL_PHASES)


class BLShard(ctypes.Structure):
    """Mirror of struct dgvcc_bl_shard."""
    _fields_ = [(n, c_int32) for n in ("rank", "world", "chunk_lo", "chunk_hi", "pt_lo", "pt_hi", "img_lo", "img_hi", "row_lo", "row_hi")] + \
               [("push_first", c_int32 * (BL_PHASES + 1)), ("wait_mask", ctypes.c_uint32 * BL_PHASES),
                ("signal_mask", ctypes.c_uint32 * BL_PHASES), ("epoch", ctypes.c_uint32), ("fuse_waits", c_int32),
                ("band_lo", c_int32), ("band_hi", c_int32)]


class DmapPlan(ctypes.Structure):
    """Mirror of struct dgvcc_dmap_plan."""
    _fields_ = [(n, c_int64) for n in
                ("total_heads", "total_pixels", "fine_tiles", "coarse_tasks", "knn_tasks", "knn_query_blocks", "knn_max_slices",
                 "off_stamps", "off_boxes", "off_wtab", "off_fmask", "off_tmpl", "off_desc", "off_ccount", "off_ctotal", "off_clist", "splat_workspace_bytes",
                 "off_knn_d2", "off_knn_idx", "off_knn_pts32", "off_knn_max", "knn_workspace_bytes", "max_side")]


DMAP_META_COLS = 12  # DGVCC_DMAP_META_COLS
DTYPE_F16, DTYPE_BF16 = 1, 2  # DGVCC_DTYPE_F16, DGVCC_DTYPE_BF16
DEN_META_COLS = 8    # DGVCC_DEN_META_COLS

# name -> (restype, argtypes); every symbol include/dgvcc_b200.h declares must appear here
SIGNATURES = {
    "dgvcc_abi_version": (c_int, []),
    "dgvcc_bounds_checked": (c_int, []),
    "dgvcc_bl_workspace_layout": (c_int, [c_int64, c_int, c_int, c_int, c_int, POINTER(BLLayout)]),
    "dgvcc_bl_set_option": (c_int, [c_int, c_int]),
    "dgvcc_bl_pack_host": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_size_t, POINTER(BLPacked)]),
    "dgvcc_bl_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int64,
                                 c_int, c_int, c_float, c_float, c_float, c_int, c_int, c_float, c_void_p, c_size_t,
                                 c_void_p, c_void_p]),
    "dgvcc_bl_forward_profiled": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                          c_int64, c_int, c_int, c_float, c_float, c_float, c_int, c_int, c_float,
                                          c_void_p, c_size_t, c_void_p, c_void_p, POINTER(c_void_p)]),
    "dgvcc_bl_backward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_int, c_int, c_float, c_float,
                                  c_int, c_int, c_float, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p]),
    "dgvcc_bl_posterior": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_int, c_int, c_float,
                                   c_float, c_float, c_int, c_void_p, c_size_t, c_void_p, c_void_p]),
    "dgvcc_bl_bayloss_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int64,
                                         c_float, c_void_p, c_size_t, c_void_p, c_void_p]),
    "dgvcc_bl_bayloss_backward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_float, c_void_p,
                                          c_void_p, c_size_t, c_void_p, c_void_p]),
    "dgvcc_bl_shard_workspace_layout": (c_int, [c_int64, c_int, c_int, c_int, c_int, c_int, POINTER(BLLayout)]),
    "dgvcc_bl_shard_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int64,
                                       c_int, c_int, c_float, c_float, c_float, c_int, c_int, c_float, POINTER(BLShard),
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p, c_int, c_void_p,
                                       POINTER(c_void_p)]),
    "dgvcc_bl_shard_backward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_int, c_float, c_float, c_int,
                                        c_int, c_float, c_void_p, POINTER(BLShard), c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_size_t, c_void_p, c_void_p, c_void_p, POINTER(c_void_p)]),
    "dgvcc_bl_shard_preload": (c_int, []),
    "dgvcc_bl_band_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_int,
                                      c_float, c_float, c_float, c_int, c_int, c_float, POINTER(BLShard), c_void_p, c_void_p,
                                      c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, POINTER(c_void_p)]),
    "dgvcc_bl_band_backward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_int, c_float, c_float, c_int,
                                       c_int, c_float, c_void_p, POINTER(BLShard), c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_size_t, c_void_p, c_void_p, POINTER(c_void_p)]),
    "dgvcc_peer_alloc": (c_int, [c_size_t, POINTER(c_void_p)]),
    "dgvcc_peer_free": (c_int, [c_void_p]),
    "dgvcc_peer_export": (c_int, [c_void_p, c_void_p]),
    "dgvcc_peer_open": (c_int, [c_void_p, POINTER(c_void_p)]),
    "dgvcc_peer_close": (c_int, [c_void_p]),
    "dgvcc_dmap_knn_workspace_bytes": (c_size_t, [c_int]),
    "dgvcc_dmap_knn_sigma": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dgvcc_dmap_batch_plan": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, POINTER(DmapPlan)]),
    "dgvcc_dmap_knn_sigma_batch": (c_int, [c_void_p, c_int, c_void_p, POINTER(DmapPlan), c_void_p, c_void_p, c_void_p,
                                           c_void_p, c_size_t, c_void_p]),
    "dgvcc_dmap_splat_batch": (c_int, [c_void_p, c_void_p, c_double, c_double, c_int, c_void_p, POINTER(DmapPlan),
                                       c_void_p, c_size_t, c_void_p, c_void_p]),
    "dgvcc_isw_instnorm_forward": (c_int, [c_void_p, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dgvcc_isw_instnorm_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "dgvcc_isw_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "dgvcc_isw_covariance": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p,
                                     c_void_p]),
    "dgvcc_isw_covariance_backward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_size_t,
                                              c_void_p, c_void_p]),
    "dgvcc_isw_loss_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                                       c_size_t, c_void_p, c_void_p]),
    "dgvcc_isw_loss_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                        c_int, c_void_p, c_size_t, c_void_p, c_void_p]),
    "dgvcc_isw_instnorm_forward_h": (c_int, [c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p,
                                             c_void_p]),
    "dgvcc_isw_instnorm_backward_h": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                                              c_void_p]),
    "dgvcc_isw_covariance_h": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p,
                                       c_void_p]),
    "dgvcc_isw_covariance_backward_h": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_size_t,
                                                c_void_p, c_void_p]),
    "dgvcc_isw_loss_backward_h": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                          c_int, c_void_p, c_size_t, c_void_p, c_void_p]),
    "dgvcc_isw_sx_tc": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "dgvcc_isw_covstat_var": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "dgvcc_isw_topk_mask": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dgvcc_lw_standardize_forward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p,
                                             c_void_p]),
    "dgvcc_lw_standardize_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                                              c_void_p]),
    "dgvcc_isw_gram": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p, c_void_p]),
    "dgvcc_lw_loss_forward": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p, c_void_p]),
    "dgvcc_lw_loss_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_size_t,
                                       c_void_p, c_void_p]),
    "dgvcc_ortho_loss_forward": (c_int, [c_void_p, c_int, c_int, c_void_p, c_size_t, c_void_p, c_void_p]),
    "dgvcc_ortho_loss_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_size_t,
                                          c_void_p, c_void_p, c_void_p]),
    "dgvcc_isw_gram_h": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p, c_void_p]),
    "dgvcc_ortho_loss_backward_h": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_size_t,
                                            c_void_p, c_void_p, c_void_p]),
    "dgvcc_lw_standardize_stats_h": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p,
                                             c_void_p]),
    "dgvcc_lw_gram_h": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_size_t,
                                c_void_p, c_void_p]),
    "dgvcc_lw_loss_backward_h": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                         c_int, c_void_p, c_size_t, c_void_p, c_void_p]),
    "dgvcc_lw_standardize_backward_h": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                                c_int, c_int, c_void_p, c_void_p]),
    "dgvcc_isw_gram_tc_partials": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "dgvcc_bay_knn_mean": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "dgvcc_bay_crop_targets": (c_int, [c_void_p, c_void_p, c_int, c_int, c_double, c_double, c_double, c_double, c_void_p,
                                       c_void_p, c_void_p, c_void_p]),
    "dgvcc_den_train_targets": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "dgvcc_sw_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "dgvcc_sw_instance_stats": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t,
                                        c_void_p]),
    "dgvcc_sw_batch_mean": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "dgvcc_sw_batch_cov": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "dgvcc_sw_update_running": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_double, c_double, c_void_p]),
    "dgvcc_sw_whiten_forward": (c_int, [c_void_p] * 9 + [c_int] * 6 + [c_float, c_void_p, c_void_p, c_void_p, c_size_t,
                                                                       c_void_p]),
    "dgvcc_sw_backward_stats": (c_int, [c_void_p] * 9 + [c_int] * 6 + [c_float] + [c_void_p] * 6 + [c_void_p, c_size_t,
                                                                                                  c_void_p]),
    "dgvcc_sw_backward_apply": (c_int, [c_void_p] * 9 + [c_double] + [c_int] * 5 + [c_void_p, c_void_p, c_size_t,
                                                                                   c_void_p]),
    "dgvcc_probe_ex2": (c_int, [c_void_p, c_int, POINTER(c_int64), c_void_p]),
    "dgvcc_probe_ffma": (c_int, [c_void_p, c_int, POINTER(c_int64), c_void_p]),
    "dgvcc_probe_ex2_fma": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "dgvcc_probe_tf32": (c_int, [c_void_p, c_int, POINTER(c_int64), c_void_p]),
}


def lib():
    """The loaded shared library (built on first use if stale or missing).  With DGVCC_BOUNDS_CHECK=1 in the
    environment it is the checked variant (libdgvcc_b200_chk.so: device-side index checks, see build.py)."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                path = _build.build(force=bool(os.environ.get("DGVCC_REBUILD")))  # returns at once unless stale
                handle = ctypes.CDLL(path)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(handle, name)  # AttributeError here = header / library mismatch
                    fn.restype = res
                    fn.argtypes = args
                _lib = handle
    return _lib


ERR_UNSUPPORTED = -3  # DGVCC_ERR_UNSUPPORTED: a shape or alignment the kernel does not tile
_ERRORS = {-1: "invalid argument", -2: "workspace too small", ERR_UNSUPPORTED: "unsupported configuration"}


_half_codes = None


def half_code(dtype):
    """DTYPE_F16 / DTYPE_BF16 for torch.float16 / torch.bfloat16, None for any other dtype."""
    global _half_codes
    if _half_codes is None:
        import torch
        _half_codes = {torch.float16: DTYPE_F16, torch.bfloat16: DTYPE_BF16}
    return _half_codes.get(dtype)


def use_tensor_cores():
    """DGVCC_ISW_TENSOR_CORES (default 1), read on every call: 0 runs the ISW-family GEMMs on their exact fp32
    CUDA-core kernels and sends fp16 / bf16 inputs down the upcast route."""
    return int(os.environ.get("DGVCC_ISW_TENSOR_CORES", "1"))


def check(rc, what):
    if rc != 0:
        msg = _ERRORS.get(rc, f"cudaError_t {rc}")
        raise RuntimeError(f"{what} failed: {msg}")


def require_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError(f"{what}: dgvcc_b200 runs on CUDA tensors only (got device {t.device}); "
                           "there is no CPU path")


def ptr(t):
    return c_void_p(t.data_ptr()) if t is not None else c_void_p(0)


def stream_ptr(device):
    """cudaStream_t of torch's current stream on ``device`` (raw handle; ~20x cheaper than building a Stream object)."""
    import torch
    idx = device.index if isinstance(device, torch.device) else torch.device(device).index
    if idx is None:
        idx = torch.cuda.current_device()
    return c_void_p(torch._C._cuda_getCurrentRawStream(idx))
