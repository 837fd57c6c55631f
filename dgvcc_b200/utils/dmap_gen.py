"""Drop-in for the reference's ``utils/dmap_gen.py`` (density-map generation) on B200.

Same functions and call signatures as the reference (utils/dmap_gen.py:14, 53, 83):

    gaussian_filter_density(img, points)        -> np.ndarray [H, W] float32   (k=3 kNN-adaptive sigma)
    gaussian_filter_density_fixed(img, points)  -> np.ndarray [H, W] float32   (sigma 4, 15x15 stamps)
    run(img_fn)                                 <name>.jpg + <name>.npy -> <name>_dmap.npy
    python -m dgvcc_b200.utils.dmap_gen --path <root>

and, beyond the reference (whose unit of work is one image in a Pool(8) worker, dmap_gen.py:116-117):

    gaussian_filter_density_batch(shapes, points_list, fixed=False) -> list of [H, W] float32 maps
    run_many(img_fns, batch=32)                 run() for a list of files, `batch` images per launch set

``img`` is only inspected for ``.shape[0:2]``; ``points`` is [N,2] (col,row), float32 or float64.
Host numpy in / host numpy out like the reference; the work runs in csrc/dmap_kernels.cu.
CUDA is initialised lazily on first call, so the functions are safe to import before a fork.
"""
import argparse
import ctypes
import os
from glob import glob

import numpy as np
import torch

from .. import _native

ADAPTIVE_TRUNCATE = 4.0      # scipy.ndimage.gaussian_filter default, dmap_gen.py:49
FIXED_SIGMA = 4.0            # dmap_gen.py:78
FIXED_TRUNCATE = 7 / 4       # dmap_gen.py:79: truncate=7/sigma


def _device(device):
    if not torch.cuda.is_available():
        raise RuntimeError("dgvcc_b200.utils.dmap_gen needs a CUDA device; there is no CPU path")
    return torch.device(device if device is not None else "cuda")


def _pinned(shape, dtype):
    """Page-locked host tensor from torch's caching host allocator: after the first call of a given size this is a
    free-list pop (no cudaHostAlloc, which costs milliseconds), and a block is only handed out again once every
    copy that used it has completed.  Results returned to the caller are numpy views of such tensors -- the view keeps
    the block alive, dropping it returns the block to the cache -- so no staging copy follows the device-to-host copy."""
    return torch.empty(shape, dtype=dtype, pin_memory=True)


def _to_device(array, dev):
    """Host numpy array -> device tensor through a pinned staging block, asynchronous on the current stream."""
    host = _pinned(array.shape, torch.from_numpy(array[:0] if array.ndim else array).dtype)
    host.numpy()[...] = array
    return host.to(dev, non_blocking=True)


def _as_points(points):
    pts = np.ascontiguousarray(np.asarray(points), dtype=np.float64)  # KDTree(points.copy()) works in float64
    if pts.ndim != 2 or pts.shape[1] != 2:
        raise ValueError(f"points must be [N,2], got {pts.shape}")
    return pts


def _require_finite(pts):
    """The adaptive reference builds KDTree(points) before anything else, and KDTree raises ValueError on NaN / inf.
    The kernels would turn such a head into pixel 0 ((int)NaN) and a NaN sigma into the identity filter."""
    if not np.isfinite(pts).all():
        bad = int(np.argmin(np.isfinite(pts).all(axis=1)))
        raise ValueError(f"points must be finite, head {bad} is {tuple(pts[bad])}")


def _check_points(points, height, width, adaptive):
    pts = _as_points(points)
    if adaptive:
        _require_finite(pts)
    # the reference's per-head loop (dmap_gen.py:41-42): `int(y) < height and int(x) < width` (int() of NaN raises
    # ValueError, of +-inf OverflowError; x is not converted when y is already out of range), then pt2d[int(y), int(x)]
    # (numpy raises IndexError below -size).  The first head that raises decides, in index order.
    fin = np.isfinite(pts)
    ty, tx = np.trunc(pts[:, 1]), np.trunc(pts[:, 0])
    with np.errstate(invalid="ignore"):
        y_bad = ~fin[:, 1]
        x_bad = ~y_bad & (ty < height) & ~fin[:, 0]
        neg = fin.all(axis=1) & (ty < height) & (tx < width) & ((ty < -height) | (tx < -width))
    fails = y_bad | x_bad | neg
    if fails.any():
        i = int(np.argmax(fails))
        if neg[i]:
            raise IndexError(f"head {i} {tuple(pts[i])}: index out of bounds for the image (negative beyond its size)")
        v = pts[i, 1] if y_bad[i] else pts[i, 0]
        if np.isnan(v):
            raise ValueError(f"head {i} {tuple(pts[i])}: cannot convert float NaN to integer")
        raise OverflowError(f"head {i} {tuple(pts[i])}: cannot convert float infinity to integer")
    return pts


def knn_sigma(points, device=None):
    """(distances [N,4] f64, locations [N,4] i64, sigma [N] f64) of dmap_gen.py:34-36,45-48, as host arrays."""
    pts = np.ascontiguousarray(np.asarray(points), dtype=np.float64)
    _require_finite(pts)
    dev = _device(device)
    n = len(pts)
    if n == 0:
        return np.zeros((0, 4)), np.zeros((0, 4), dtype=np.int64), np.zeros((0,))
    d_pts = _to_device(pts, dev)
    idx = torch.empty((n, 4), dtype=torch.int32, device=dev)
    dist = torch.empty((n, 4), dtype=torch.float64, device=dev)
    sigma = torch.empty((n,), dtype=torch.float64, device=dev)
    kws_bytes = _native.lib().dgvcc_dmap_knn_workspace_bytes(n)
    kws = torch.empty((kws_bytes,), dtype=torch.uint8, device=dev)
    _native.check(_native.lib().dgvcc_dmap_knn_sigma(_native.ptr(d_pts), n, _native.ptr(idx), _native.ptr(dist),
                                                     _native.ptr(sigma), _native.ptr(kws), kws_bytes,
                                                     _native.stream_ptr(dev)), "dgvcc_dmap_knn_sigma")
    return dist.cpu().numpy(), idx.cpu().numpy().astype(np.int64), sigma.cpu().numpy()


class _Plan:
    """Host plan of one batched launch set (include/dgvcc_b200.h: dgvcc_dmap_batch_plan)."""

    def __init__(self, shapes, counts):
        lib = _native.lib()
        b = len(shapes)
        heights = np.ascontiguousarray([int(s[0]) for s in shapes], dtype=np.int32)
        widths = np.ascontiguousarray([int(s[1]) for s in shapes], dtype=np.int32)
        cnts = np.ascontiguousarray(counts, dtype=np.int32)
        self.meta = np.zeros((b + 1, _native.DMAP_META_COLS), dtype=np.int64)
        self.plan = _native.DmapPlan()
        _native.check(lib.dgvcc_dmap_batch_plan(b, heights.ctypes.data, widths.ctypes.data, cnts.ctypes.data,
                                                self.meta.ctypes.data, ctypes.byref(self.plan)),
                      "dgvcc_dmap_batch_plan")
        self.n_images = b
        self.out_off = self.meta[:, 4]
        self.pt_off = self.meta[:, 0]


def _density_batch_device(shapes, pts_list, adaptive, dev):
    """(packed device tensor [sum H*W] f32, per-image offsets into it) for a list of images; ``pts_list`` holds
    host float64 [N,2] arrays.  Images are launched in order of falling head count -- the crowded ones, whose
    tiles take longest, start first -- so the packed layout follows that order, not the caller's."""
    lib = _native.lib()
    counts = np.array([len(p) for p in pts_list], dtype=np.int64)
    order = np.argsort(-counts, kind="stable")
    plan = _Plan([shapes[i] for i in order], counts[order])
    pl = plan.plan
    stream = _native.stream_ptr(dev)
    meta = _to_device(plan.meta, dev)
    out = torch.empty((pl.total_pixels,), dtype=torch.float32, device=dev)
    ws = torch.empty((pl.splat_workspace_bytes,), dtype=torch.uint8, device=dev)
    d_pts = sigma = None
    if pl.total_heads:
        host_pts = _pinned((int(pl.total_heads), 2), torch.float64)
        np.concatenate([pts_list[i] for i in order if counts[i]], axis=0, out=host_pts.numpy())
        d_pts = host_pts.to(dev, non_blocking=True)
        if adaptive:
            sigma = torch.empty((pl.total_heads,), dtype=torch.float64, device=dev)
            kws = torch.empty((pl.knn_workspace_bytes,), dtype=torch.uint8, device=dev)
            _native.check(lib.dgvcc_dmap_knn_sigma_batch(_native.ptr(d_pts), plan.n_images, _native.ptr(meta),
                                                         ctypes.byref(pl), None, None, _native.ptr(sigma),
                                                         _native.ptr(kws), pl.knn_workspace_bytes, stream),
                          "dgvcc_dmap_knn_sigma_batch")
    _native.check(lib.dgvcc_dmap_splat_batch(
        _native.ptr(d_pts), _native.ptr(sigma), FIXED_SIGMA, ADAPTIVE_TRUNCATE if adaptive else FIXED_TRUNCATE,
        plan.n_images, _native.ptr(meta), ctypes.byref(pl), _native.ptr(ws), pl.splat_workspace_bytes,
        _native.ptr(out), stream), "dgvcc_dmap_splat_batch")
    offsets = np.empty(len(shapes), dtype=np.int64)
    offsets[order] = plan.out_off[:-1]
    return out, offsets


def _density_device(height, width, pts, adaptive, dev):
    """Device tensor [H,W] f32 for one image; ``pts`` is a host float64 [N,2] array."""
    out, _ = _density_batch_device([(height, width)], [pts], adaptive, dev)
    return out.view(height, width)


def _density(img, points, adaptive, device=None):
    height, width = int(img.shape[0]), int(img.shape[1])
    if len(points) == 0:  # dmap_gen.py:28-29
        return np.zeros((height, width), dtype=np.float32)
    pts = _check_points(points, height, width, adaptive)
    dev = _device(device)
    host = _pinned((height, width), torch.float32)
    host.copy_(_density_device(height, width, pts, adaptive, dev), non_blocking=True)
    torch.cuda.current_stream(dev).synchronize()
    return host.numpy()


def gaussian_filter_density(img, points, device=None):
    """Geometry-adaptive density map (reference: utils/dmap_gen.py:14-51)."""
    return _density(img, points, True, device)


def gaussian_filter_density_fixed(img, points, device=None):
    """Fixed-sigma density map, what ``run`` uses (reference: utils/dmap_gen.py:53-81)."""
    return _density(img, points, False, device)


def gaussian_filter_density_batch(shapes, points_list, fixed=False, device=None):
    """A list of images through ONE set of launches (kNN, prepare, two culling passes, splat), one packed
    device-to-host copy and one synchronisation; returns a list of [H,W] float32 arrays (views of one buffer)."""
    shapes = [(int(h), int(w)) for h, w in shapes]
    if not shapes:
        return []
    # every image is checked (in the caller's order, like one reference call per image) before anything is launched
    pts = [_check_points(p, h, w, not fixed) if len(p) else np.zeros((0, 2)) for (h, w), p in zip(shapes, points_list)]
    dev = _device(device)
    out, offsets = _density_batch_device(shapes, pts, not fixed, dev)
    host = _pinned(out.shape, torch.float32)
    host.copy_(out, non_blocking=True)
    torch.cuda.current_stream(dev).synchronize()
    flat = host.numpy()
    return [flat[o:o + h * w].reshape(h, w) for o, (h, w) in zip(offsets, shapes)]


def _image_shape(img_fn):
    from PIL import Image
    with Image.open(img_fn) as im:
        w, h = im.size
    return np.empty((h, w, 0))


def _paths(img_fn):
    img_ext = os.path.splitext(img_fn)[1]
    basename = os.path.basename(img_fn).replace(img_ext, '')
    gt_fn = img_fn.replace(img_ext, '.npy')
    return gt_fn, gt_fn.replace(basename, basename + '_dmap')


def run(img_fn):
    """File protocol of dmap_gen.py:83-95: <name>.<ext> + <name>.npy -> <name>_dmap.npy, skipped when present."""
    gt_fn, dmap_fn = _paths(img_fn)

    if os.path.exists(dmap_fn):
        return

    img = _image_shape(img_fn)  # the reference decodes the image only for its shape
    gt = np.load(gt_fn)
    dmap = gaussian_filter_density_fixed(img, gt)
    np.save(dmap_fn, dmap)


def run_many(img_fns, batch=32):
    """``run`` for a list of images, ``batch`` at a time through the batched launch set (what replaces the
    reference's ``Pool(8)``, dmap_gen.py:116-117)."""
    todo = [fn for fn in img_fns if not os.path.exists(_paths(fn)[1])]
    for k in range(0, len(todo), batch):
        chunk = todo[k:k + batch]
        shapes = [_image_shape(fn).shape[:2] for fn in chunk]
        gts = [np.load(_paths(fn)[0]) for fn in chunk]
        gts = [g if len(g) else np.zeros((0, 2)) for g in gts]
        for fn, dmap in zip(chunk, gaussian_filter_density_batch(shapes, gts, fixed=True)):
            np.save(_paths(fn)[1], dmap)


if __name__ == '__main__':
    parser = argparse.ArgumentParser()
    parser.add_argument('--path', type=str)
    args = parser.parse_args()

    path = args.path
    if not os.path.exists(path):
        raise Exception("Path does not exist")

    img_fns = []
    for phase in ['test']:
        img_fns += glob(os.path.join(path, phase, '*.jpg'))
    img_fns = [fn for fn in img_fns if 'aug' not in fn]

    # the reference fans out over Pool(8); batched launches on one GPU stream are faster and need no fork
    run_many(img_fns)
