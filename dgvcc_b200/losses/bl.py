"""Drop-in for the reference's ``losses/bl.py`` (Bayesian loss) on B200.

Same classes, constructor keywords and call signatures as the reference
(losses/bl.py:5-91), so ``get_loss('bl', params)`` (main.py:51-53) and the
trainers' ``loss.__class__.__name__ == 'BL'`` dispatch (dgtrainer.py:59) work
unchanged:

    BL(sigma, c_size, stride, background_ratio, use_background, device)
        .forward(points, st_sizes, target_list, pre_density) -> 0-dim loss

``BL.forward`` runs the fused CUDA path (csrc/bl_kernels.cu) that never builds
the [points x pixels] posterior; ``Post_Prob`` / ``Bay_Loss`` keep their own
reference signatures for callers that want the materialised posteriors.

Extensions that do not change reference behaviour:
  * rectangular grids: the grid is taken from ``pre_density.shape[-2:]``
    (the reference is square-only because x and y share ``cood``, bl.py:14-16);
  * image sharding: ``BL.global_batch`` (default: the local batch) is the
    divisor of bl.py:79, so a rank holding B_local of B_global images returns
    its partial loss and ``dgvcc_b200.sharding`` all-reduces it.
"""
import os
from math import ceil

import numpy as np
import torch
from torch.nn import Module

from .. import _native


def _as_point_list(points):
    """bl.py:21-22 accepts a list/tuple of [N_i,2] tensors; empty ones may be any shape with 0 elements."""
    out = []
    for p in points:
        if p.numel() == 0:
            p = p.reshape(0, 2)
        if p.dim() != 2 or p.shape[1] != 2:
            raise ValueError(f"points must be [N,2] tensors, got {tuple(p.shape)}")
        out.append(p)
    return out


_CHUNK_POINTS = int(os.environ.get("DGVCC_BL_CHUNK", "512"))  # read once, at import (512: measured, scripts/bl_tune_1gpu.py)


def chunk_points():
    """Points per chunk: big images are cut into near-equal slices of at most this many points."""
    return _CHUNK_POINTS


def build_meta(counts, rows, chunk, tail_split=0):
    """The int32 table of include/dgvcc_b200.h: pt_off, row_off, keep, icb, chunks[C][4].

    ``tail_split`` > 1 (sharded sweeps, where a rank has only a round or two of warp tasks): the last quarter of every
    image's chunks is cut into ``tail_split`` pieces each -- with the longest-first queue the sweep then ends on tasks a
    fraction as long, for a few more partial arrays."""
    counts = np.asarray(counts, dtype=np.int64)
    rows = np.asarray(rows, dtype=np.int64)
    b = len(counts)
    n_chunks = np.maximum(1, -(-counts // chunk))
    if tail_split and tail_split > 1:
        img_l, start_l, cnt_l = [], [], []
        for i in range(b):
            n, nc = int(counts[i]), int(n_chunks[i])
            edges = [n * k // nc for k in range(nc + 1)]
            n_tail = nc // 4 if nc >= 4 else 0
            for k in range(nc):
                a, e = edges[k], edges[k + 1]
                parts = tail_split if k >= nc - n_tail and e - a >= 32 * tail_split else 1
                for q in range(parts):
                    s0, s1 = a + (e - a) * q // parts, a + (e - a) * (q + 1) // parts
                    img_l.append(i); start_l.append(s0); cnt_l.append(s1 - s0)
        img = np.asarray(img_l, dtype=np.int64)
        start, cnt = np.asarray(start_l, dtype=np.int64), np.asarray(cnt_l, dtype=np.int64)
        n_chunks = np.bincount(img, minlength=b).astype(np.int64)
        stop = start + cnt
    else:
        img = start = stop = None
    total_chunks = int(n_chunks.sum())
    meta = np.zeros(4 * b + 3 + 4 * total_chunks, dtype=np.int32)
    meta[1:b + 1] = np.cumsum(counts)
    meta[b + 2:2 * b + 2] = np.cumsum(rows)
    # bl.py:76: num = ceil(0.9 * (len(res) - 1)), the same double arithmetic as Python's
    meta[2 * b + 2:3 * b + 2] = np.ceil(0.9 * (rows - 1).astype(np.float64))
    ends = np.cumsum(n_chunks)
    meta[3 * b + 3:4 * b + 3] = ends
    table = meta[4 * b + 3:].reshape(total_chunks, 4)
    if img is None:
        img = np.repeat(np.arange(b), n_chunks)
        k = np.arange(total_chunks) - (ends - n_chunks)[img]      # chunk index inside its image
        start = counts[img] * k // n_chunks[img]                   # near-equal slices
        stop = counts[img] * (k + 1) // n_chunks[img]
    table[:, 0], table[:, 1], table[:, 2] = img, start, stop - start
    # schedule: longest chunks first -- the sweeps hand the launch slots out through a work queue, so this is a
    # longest-processing-time schedule (the tail of a sweep is made of the shortest tasks)
    table[:, 3] = np.argsort(-(stop - start), kind="stable")
    return meta, total_chunks, int(n_chunks.max() > 1)


class _Staging:
    """A small ring of pinned host buffers per device: one packed H2D copy per step, no per-call
    cudaHostAlloc.  A buffer is re-used only after the copy that read it has completed (event)."""
    RING = 4

    def __init__(self):
        self.bufs = [None] * self.RING
        self.events = [None] * self.RING
        self.next = 0

    def take(self, nbytes):
        i = self.next
        self.next = (i + 1) % self.RING
        if self.events[i] is not None:
            self.events[i].synchronize()
        if self.bufs[i] is None or self.bufs[i].numel() < nbytes:
            size = max(nbytes + nbytes // 4, 1 << 20)
            if self.bufs[i] is None and not any(b is not None for b in self.bufs):
                # first use: pin the whole ring now (cudaHostAlloc takes milliseconds, and longer when several
                # processes pin at once), not one slot per step over the first RING steps
                self.bufs = [torch.empty((size,), dtype=torch.uint8).pin_memory() for _ in range(self.RING)]
            else:
                self.bufs[i] = torch.empty((size,), dtype=torch.uint8).pin_memory()
        return i, self.bufs[i]

    def sent(self, i, device):
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(device))
        self.events[i] = ev


_staging = {}


def _host_f32(t):
    """Zero-copy numpy view of a host tensor when it already is fp32, else a converted copy."""
    if t.dtype != torch.float32 or t.requires_grad:
        t = t.detach().to(torch.float32)
    return t.numpy()


def _align16(n):
    return (n + 15) // 16 * 16


def _pack_into(view, meta, points, targets, total_points):
    """The host buffer of a packed batch, ``[int32 table | align16 | points | align16 | targets]`` (what
    dgvcc_bl_pack_host writes).  Returns (o_pts, o_tgt, total bytes) for ``meta`` and ``total_points``; with a uint8
    array ``view`` of at least that size it also writes table, points and, unless ``targets`` is None, targets."""
    n = max(total_points, 1)
    o_pts = _align16(meta.nbytes)
    o_tgt = o_pts + _align16(8 * n)
    if view is not None:
        view[:meta.nbytes].view(np.int32)[:] = meta
        if total_points:
            np.concatenate([_host_f32(p.cpu()).reshape(-1, 2) for p in points if p.numel()], axis=0,
                           out=view[o_pts:o_pts + 8 * total_points].view(np.float32).reshape(-1, 2))
            if targets is not None:
                np.concatenate([_host_f32(t.cpu()).reshape(-1) for t in targets if t.numel()],
                               out=view[o_tgt:o_tgt + 4 * total_points].view(np.float32))
    return o_pts, o_tgt, o_tgt + _align16(4 * n)


class PackedBatch:
    """A ragged batch already packed on the host (table + points + targets in ONE buffer), built by
    ``pack_batch`` -- e.g. inside a DataLoader ``collate_fn`` in place of bay_dataset.py:13-19's tuples -- so that
    the training step only has to upload it.  Pass it to ``BL.forward`` as ``points`` (``target_list=None``).
    ``pin_memory()`` is what ``DataLoader(pin_memory=True)`` calls on custom batch types."""

    def __init__(self, buf, meta_bytes, o_pts, o_tgt, total, counts, rows, total_chunks, multi_chunk, use_bg):
        self.buf, self.meta_bytes, self.o_pts, self.o_tgt, self.total = buf, meta_bytes, o_pts, o_tgt, total
        self.counts, self.rows, self.total_chunks, self.multi_chunk, self.use_bg = counts, rows, total_chunks, multi_chunk, use_bg

    def pin_memory(self):
        self.buf = self.buf.pin_memory()
        return self

    def __len__(self):
        return len(self.counts)


def pack_batch(points, targets, use_background=True, chunk=None):
    """Host-side CSR packing of lists of [N_i,2] points and [N_i] targets (CPU tensors) into a ``PackedBatch``."""
    points = _as_point_list(points)
    if len(points) == 0:
        raise ValueError("empty batch")
    counts = np.asarray([int(p.shape[0]) for p in points], dtype=np.int64)
    rows = np.where(counts == 0, 1, counts + (1 if use_background else 0))
    targets = [t.reshape(-1) for t in targets]
    for t, n in zip(targets, counts):
        if t.shape[0] != n:
            raise ValueError(f"target length {t.shape[0]} does not match its {n} points")
    meta, total_chunks, multi_chunk = build_meta(counts, rows, chunk or chunk_points())
    total_points = int(counts.sum())
    o_pts, o_tgt, total = _pack_into(None, meta, points, targets, total_points)
    buf = torch.zeros((total,), dtype=torch.uint8)
    _pack_into(buf.numpy(), meta, points, targets, total_points)
    return PackedBatch(buf, meta.nbytes, o_pts, o_tgt, total, counts, rows, total_chunks, multi_chunk, bool(use_background))


def _plain_f32(tensors):
    return all(t.dtype == torch.float32 and t.is_contiguous() and not t.requires_grad for t in tensors)


def pack_host_native(points, targets, use_bg, chunk, dst_ptr, dst_bytes, args=None):
    """dgvcc_bl_pack_host on lists of contiguous fp32 CPU tensors; ``dst_ptr=None`` only sizes the buffer.
    Returns (BLPacked info, the ctypes argument arrays for a second call)."""
    import ctypes
    if args is None:
        b = len(points)
        args = ((ctypes.c_void_p * b)(*[p.data_ptr() for p in points]),
                (ctypes.c_void_p * b)(*[t.data_ptr() for t in targets]) if targets is not None else None,
                (ctypes.c_int32 * b)(*[p.shape[0] for p in points]), b)
    info = _native.BLPacked()
    _native.check(_native.lib().dgvcc_bl_pack_host(args[0], args[1], args[2], args[3], int(bool(use_bg)), int(chunk),
                                                   dst_ptr, dst_bytes, ctypes.byref(info)), "dgvcc_bl_pack_host")
    return info, args


class _Packed:
    """CSR packing of one ragged batch + the small int32 table the kernels read (include/dgvcc_b200.h).

    Host lists (e.g. straight from the DataLoader) are packed on the host -- table, points and targets in
    one pinned buffer -- and uploaded with a single asynchronous copy; device lists are concatenated on
    the device like bl.py:21-22.
    """

    def __init__(self, points, use_bg, device, targets=None):
        if isinstance(points, PackedBatch):
            self._from_packed_batch(points, use_bg, device)
            return
        if device.type == "cuda" and self._init_from_host_lists(points, targets, use_bg, device):
            return
        points = _as_point_list(points)
        self.batch = len(points)
        if self.batch == 0:
            raise ValueError("empty batch")
        counts = np.asarray([int(p.shape[0]) for p in points], dtype=np.int64)
        rows = np.where(counts == 0, 1, counts + (1 if use_bg else 0))
        self.counts = counts
        self.rows = rows
        self.total_points = int(counts.sum())
        self.total_rows = int(rows.sum())
        b = self.batch
        self.targets = None
        if targets is not None:
            targets = [t.reshape(-1) for t in targets]
            for t, n in zip(targets, counts):
                if t.shape[0] != n:
                    raise ValueError(f"target length {t.shape[0]} does not match its {n} points")
        self.on_host = device.type == "cuda" and all(p.device.type == "cpu" for p in points) and \
            (targets is None or all(t.device.type == "cpu" for t in targets))
        n_pts = max(self.total_points, 1)
        self.pt_off = np.concatenate(([0], np.cumsum(counts))).astype(np.int32)
        self.row_off = np.concatenate(([0], np.cumsum(rows))).astype(np.int32)
        meta, self.total_chunks, self.multi_chunk = build_meta(counts, rows, chunk_points())
        if self.on_host:
            o_pts, o_tgt, total = _pack_into(None, meta, points, targets, self.total_points)
            ring = _staging.setdefault(device, _Staging())
            slot, host = ring.take(total)
            _pack_into(host.numpy(), meta, points, targets, self.total_points)
            dev_buf = host[:total].to(device, non_blocking=True)
            ring.sent(slot, device)
            self.meta = dev_buf[:meta.nbytes].view(torch.int32)
            self.pts = dev_buf[o_pts:o_pts + 8 * n_pts].view(torch.float32).view(-1, 2)
            if targets is not None:
                self.targets = dev_buf[o_tgt:o_tgt + 4 * n_pts].view(torch.float32)
        else:
            host = torch.from_numpy(meta)
            if device.type == "cuda":
                host = host.pin_memory()
            self.meta = host.to(device, non_blocking=True)
            if self.total_points == 0:
                self.pts = torch.zeros((1, 2), dtype=torch.float32, device=device)  # never read
            else:
                self.pts = torch.cat([p.to(device=device, dtype=torch.float32) for p in points], dim=0).contiguous()
            if targets is not None:
                if self.total_points == 0:
                    self.targets = torch.zeros((1,), dtype=torch.float32, device=device)
                else:
                    self.targets = torch.cat([t.to(device=device, dtype=torch.float32) for t in targets]).contiguous()


    def _init_from_host_lists(self, points, targets, use_bg, device):
        """Fast path for what a DataLoader delivers: lists of contiguous fp32 CPU tensors.  One pass over the lists
        collects pointers and sizes; table + points + targets are then written into the pinned staging buffer by
        one native call (csrc/bl_pack_host.cu) and uploaded with ONE asynchronous copy.  Returns False (nothing
        done) when a tensor does not qualify; the general path then validates and converts."""
        import ctypes
        b = len(points)
        if b == 0 or (targets is not None and len(targets) != b):
            return False
        pp, cn = (ctypes.c_void_p * b)(), (ctypes.c_int32 * b)()
        tp = (ctypes.c_void_p * b)() if targets is not None else None
        f32 = torch.float32
        for i in range(b):
            p = points[i]
            if p.dtype is not f32 or p.is_cuda or p.requires_grad or not p.is_contiguous():
                return False
            if p.dim() == 2 and p.shape[1] == 2:
                n = p.shape[0]
            elif p.numel() == 0:
                n = 0
            else:
                return False  # the general path raises the shape error
            cn[i] = n
            pp[i] = p.data_ptr()
            if tp is not None:
                t = targets[i]
                if t.dtype is not f32 or t.is_cuda or t.requires_grad or not t.is_contiguous() or t.numel() != n:
                    return False
                tp[i] = t.data_ptr()
        args = (pp, tp, cn, b)
        info, _ = pack_host_native(None, None, use_bg, chunk_points(), None, 0, args)
        ring = _staging.setdefault(device, _Staging())
        slot, host = ring.take(info.total_bytes)
        pack_host_native(None, None, use_bg, chunk_points(), host.data_ptr(), host.numel(), args)
        dev_buf = host[:info.total_bytes].to(device, non_blocking=True)
        ring.sent(slot, device)
        n_pts = max(int(info.total_points), 1)
        self.batch, self.on_host = b, True
        self._counts_c = cn
        self._use_bg = bool(use_bg)
        self.total_points, self.total_rows = int(info.total_points), int(info.total_rows)
        self.total_chunks, self.multi_chunk = int(info.total_chunks), int(info.multi_chunk)
        self.meta = dev_buf[:info.meta_bytes].view(torch.int32)
        self.pts = dev_buf[info.off_points:info.off_points + 8 * n_pts].view(torch.float32).view(-1, 2)
        self.targets = dev_buf[info.off_targets:info.off_targets + 4 * n_pts].view(torch.float32) if tp is not None else None
        return True

    def __getattr__(self, name):
        # per-image bookkeeping of the fast path, built only when somebody asks (Post_Prob, tests)
        if name in ("counts", "rows", "pt_off", "row_off") and "_counts_c" in self.__dict__:
            counts = np.asarray(list(self._counts_c), dtype=np.int64)
            rows = np.where(counts == 0, 1, counts + (1 if self._use_bg else 0))
            self.counts, self.rows = counts, rows
            self.pt_off = np.concatenate(([0], np.cumsum(counts))).astype(np.int32)
            self.row_off = np.concatenate(([0], np.cumsum(rows))).astype(np.int32)
            return self.__dict__[name]
        raise AttributeError(name)

    def _from_packed_batch(self, pb, use_bg, device):
        if pb.use_bg != bool(use_bg):
            raise ValueError("PackedBatch was packed for a different use_background setting")
        self.batch = len(pb.counts)
        self.counts, self.rows = pb.counts, pb.rows
        self.total_points, self.total_rows = int(pb.counts.sum()), int(pb.rows.sum())
        self.total_chunks, self.multi_chunk = pb.total_chunks, pb.multi_chunk
        b = self.batch
        meta = pb.buf[:pb.meta_bytes].numpy().view(np.int32)
        self.pt_off, self.row_off = meta[:b + 1].copy(), meta[b + 1:2 * b + 2].copy()
        self.on_host = True
        dev_buf = pb.buf.to(device, non_blocking=True)  # one copy; asynchronous when the batch is pinned
        n_pts = max(self.total_points, 1)
        self.meta = dev_buf[:pb.meta_bytes].view(torch.int32)
        self.pts = dev_buf[pb.o_pts:pb.o_pts + 8 * n_pts].view(torch.float32).view(-1, 2)
        self.targets = dev_buf[pb.o_tgt:pb.o_tgt + 4 * n_pts].view(torch.float32)


def _pack_targets(target_list, packed, device):
    """Targets of a batch whose points are already packed (bench / tests helper)."""
    if packed.total_points == 0:
        return torch.zeros((1,), dtype=torch.float32, device=device)
    parts = [t.reshape(-1) for t in target_list]
    for t, n in zip(parts, packed.counts):
        if t.shape[0] != n:
            raise ValueError(f"target length {t.shape[0]} does not match its {n} points")
    return torch.cat([t.to(device=device, dtype=torch.float32) for t in parts], dim=0).contiguous()


def _layout(total_rows, total_chunks, batch, hp, wp):
    lay = _native.BLLayout()
    _native.check(_native.lib().dgvcc_bl_workspace_layout(total_rows, total_chunks, batch, hp, wp, lay),
                  "dgvcc_bl_workspace_layout")
    return lay


def _workspace(lay, device):
    """Caller-owned scratch of one forward/backward pair.  ``torch.empty`` is a free-list pop of the caching
    allocator after the first step (no cudaMalloc, no launch); nothing in it needs initialising -- the kernels
    clear their own arrival counter.  It is NOT shared between calls: autograd may hold several graphs at once."""
    return torch.empty((lay.total,), dtype=torch.uint8, device=device)


def _region(ws, offset, n, dtype=torch.float32):
    return ws[offset:offset + 4 * n].view(dtype)


class _FusedBL(torch.autograd.Function):
    """dgvcc_bl_forward / dgvcc_bl_backward; only the density receives gradient (bl.py:73-79)."""

    @staticmethod
    def forward(ctx, density, packed, targets, st_sizes, stride, sigma, bg_ratio, use_bg, inv_batch, keep, cull):
        _native.require_cuda(density, "BL.forward")
        b, hp, wp = density.shape[0], density.shape[-2], density.shape[-1]
        dens = density.detach().reshape(b, hp, wp).to(torch.float32).contiguous()
        dev = dens.device
        lay = _layout(packed.total_rows, packed.total_chunks, b, hp, wp)
        ws = _workspace(lay, dev)
        loss = torch.empty((1,), dtype=torch.float32, device=dev)
        rc = _native.lib().dgvcc_bl_forward(
            _native.ptr(packed.pts), _native.ptr(targets), _native.ptr(packed.meta), _native.ptr(st_sizes),
            _native.ptr(dens), b, hp, wp, packed.total_rows, packed.total_chunks, packed.multi_chunk, stride, sigma,
            bg_ratio, int(use_bg), int(cull), inv_batch,
            _native.ptr(ws), lay.total, _native.ptr(loss), _native.stream_ptr(dev))
        _native.check(rc, "dgvcc_bl_forward")
        ctx.packed, ctx.ws, ctx.lay = packed, ws, lay
        ctx.geom = (b, hp, wp, stride, sigma, int(use_bg), inv_batch, int(cull))
        ctx.dens_shape, ctx.dens_dtype = density.shape, density.dtype
        if keep is not None:  # debugging / tests: expose the workspace regions
            keep["workspace"], keep["layout"], keep["packed"] = ws, lay, packed
        return loss.reshape(())

    @staticmethod
    def backward(ctx, grad_loss):
        b, hp, wp, stride, sigma, use_bg, inv_batch, cull = ctx.geom
        packed, ws, lay = ctx.packed, ctx.ws, ctx.lay
        dev = ws.device
        g = grad_loss.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
        grad = torch.empty((b, hp, wp), dtype=torch.float32, device=dev)
        rc = _native.lib().dgvcc_bl_backward(
            _native.ptr(packed.pts), _native.ptr(packed.meta), b, hp, wp, packed.total_rows, packed.total_chunks,
            packed.multi_chunk, stride, sigma, use_bg, cull, inv_batch, _native.ptr(g), _native.ptr(ws), lay.total,
            _native.ptr(grad), _native.stream_ptr(dev))
        _native.check(rc, "dgvcc_bl_backward")
        return (grad.reshape(ctx.dens_shape).to(ctx.dens_dtype),) + (None,) * 10


class Post_Prob(Module):
    """Posterior label probabilities, materialised (reference: losses/bl.py:5-52)."""

    def __init__(self, sigma, c_size, stride, background_ratio, use_background, device):
        super(Post_Prob, self).__init__()
        assert c_size % stride == 0

        self.sigma = sigma
        self.bg_ratio = background_ratio
        self.device = device
        self.c_size = c_size
        self.stride = stride
        # kept for attribute compatibility (bl.py:14-16); the kernels rebuild the same values on the fly
        self.cood = (torch.arange(0, c_size, step=stride, dtype=torch.float32, device=device) + stride / 2).unsqueeze(0)
        self.use_bg = use_background

    def forward(self, points, st_sizes, grid=None):
        """List of [N_i(+1), H'*W'] posteriors, ``None`` for images without points (bl.py:36-51).

        ``grid=(rows, cols)`` selects a rectangular grid; the default is the reference's square
        ``c_size // stride`` grid.
        """
        hp, wp = grid if grid is not None else (self.c_size // self.stride,) * 2
        dev = st_sizes.device
        _native.require_cuda(st_sizes, "Post_Prob.forward")
        packed = _Packed(points, self.use_bg, dev)
        if packed.total_points == 0:
            return [None for _ in range(packed.batch)]
        st = st_sizes.to(torch.float32).contiguous()
        lay = _layout(packed.total_rows, packed.total_chunks, packed.batch, hp, wp)
        ws = _workspace(lay, dev)
        prob = torch.empty((packed.total_rows, hp * wp), dtype=torch.float32, device=dev)
        rc = _native.lib().dgvcc_bl_posterior(
            _native.ptr(packed.pts), _native.ptr(packed.meta), _native.ptr(st), packed.batch, hp, wp,
            packed.total_rows, packed.total_chunks, packed.multi_chunk, float(self.stride), float(self.sigma), float(self.bg_ratio), int(self.use_bg),
            _native.ptr(ws), lay.total, _native.ptr(prob), _native.stream_ptr(dev))
        _native.check(rc, "dgvcc_bl_posterior")
        out = []
        for i in range(packed.batch):
            if packed.counts[i] == 0:
                out.append(None)
            else:
                out.append(prob[packed.row_off[i]:packed.row_off[i + 1]])
        return out


class _BayLossOnProb(torch.autograd.Function):
    @staticmethod
    def forward(ctx, density, prob, targets, meta, total_rows, inv_batch):
        b, hp, wp = density.shape[0], density.shape[-2], density.shape[-1]
        dens = density.detach().reshape(b, hp, wp).to(torch.float32).contiguous()
        dev = dens.device
        lay = _layout(total_rows, b, b, hp, wp)
        ws = _workspace(lay, dev)
        loss = torch.empty((1,), dtype=torch.float32, device=dev)
        rc = _native.lib().dgvcc_bl_bayloss_forward(
            _native.ptr(prob), _native.ptr(targets), _native.ptr(meta), _native.ptr(dens), b, hp, wp, total_rows,
            inv_batch, _native.ptr(ws), lay.total, _native.ptr(loss), _native.stream_ptr(dev))
        _native.check(rc, "dgvcc_bl_bayloss_forward")
        ctx.saved = (prob, meta, ws, lay, b, hp, wp, total_rows, inv_batch, density.shape, density.dtype)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, grad_loss):
        prob, meta, ws, lay, b, hp, wp, total_rows, inv_batch, shape, dtype = ctx.saved
        dev = ws.device
        g = grad_loss.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
        grad = torch.empty((b, hp, wp), dtype=torch.float32, device=dev)
        rc = _native.lib().dgvcc_bl_bayloss_backward(
            _native.ptr(prob), _native.ptr(meta), b, hp, wp, total_rows, inv_batch, _native.ptr(g), _native.ptr(ws),
            lay.total, _native.ptr(grad), _native.stream_ptr(dev))
        _native.check(rc, "dgvcc_bl_bayloss_backward")
        return (grad.reshape(shape).to(dtype),) + (None,) * 5


class Bay_Loss(Module):
    """Trimmed-L1 count loss on given posteriors (reference: losses/bl.py:54-80)."""

    def __init__(self, use_background, device):
        super(Bay_Loss, self).__init__()
        self.device = device
        self.use_bg = use_background

    def forward(self, prob_list, target_list, pre_density):
        _native.require_cuda(pre_density, "Bay_Loss.forward")
        dev = pre_density.device
        b = len(prob_list)
        m = pre_density.shape[-2] * pre_density.shape[-1]
        probs, tgts, rows, counts = [], [], [], []
        for idx, prob in enumerate(prob_list):
            if prob is None or prob.shape[0] == 0:  # bl.py:63-65: count = sum of density, target 0
                probs.append(torch.ones((1, m), dtype=torch.float32, device=dev))
                rows.append(1)
                counts.append(0)
            else:
                n = prob.shape[0] - 1 if self.use_bg else prob.shape[0]
                probs.append(prob.detach().to(device=dev, dtype=torch.float32).reshape(prob.shape[0], m))
                tgts.append(target_list[idx].reshape(-1)[:n].to(device=dev, dtype=torch.float32))
                rows.append(prob.shape[0])
                counts.append(n)
        meta, _, _ = build_meta(np.asarray(counts, dtype=np.int64), np.asarray(rows, dtype=np.int64), 1 << 30)
        meta_dev = torch.from_numpy(meta).pin_memory().to(dev, non_blocking=True)
        prob_all = torch.cat(probs, dim=0).contiguous()
        targets = torch.cat(tgts).contiguous() if tgts else torch.zeros((1,), dtype=torch.float32, device=dev)
        return _BayLossOnProb.apply(pre_density, prob_all, targets, meta_dev, int(sum(rows)), 1.0 / b)


class BL(Module):
    """Bayesian loss, fused (reference: losses/bl.py:82-91)."""

    def __init__(self, sigma, c_size, stride, background_ratio, use_background, device):
        super(BL, self).__init__()
        self.post_prob = Post_Prob(sigma, c_size, stride, background_ratio, use_background, device)
        self.bay_loss = Bay_Loss(use_background, device)
        self.global_batch = None  # set by dgvcc_b200.sharding when images are partitioned across ranks
        # Skip (point, pixel-tile) pairs whose exponentials are provably exact zeros.  The results are bit-identical
        # to the dense evaluation (tests/test_bl_gpu.py) and 3-4x faster on crowded images, so it is the product
        # default; ``exact_cull = False`` (or DGVCC_BL_EXACT_CULL=0) selects the dense sweep that bench.py grades.
        self.exact_cull = bool(int(os.environ.get("DGVCC_BL_EXACT_CULL", "1")))

    def forward(self, points, st_sizes, target_list, pre_density, _keep=None):
        pp = self.post_prob
        dev = pre_density.device
        _native.require_cuda(pre_density, "BL.forward")
        if len(points) != pre_density.shape[0]:
            raise ValueError(f"{len(points)} point sets for a batch of {pre_density.shape[0]} density maps")
        if isinstance(points, PackedBatch) and target_list is not None:
            raise ValueError("a PackedBatch already carries its targets; pass target_list=None")
        packed = _Packed(points, pp.use_bg, dev, targets=target_list)
        targets = packed.targets
        st = st_sizes.to(device=dev, dtype=torch.float32).contiguous()
        inv_batch = 1.0 / float(self.global_batch or packed.batch)
        return _FusedBL.apply(pre_density, packed, targets, st, float(pp.stride), float(pp.sigma),
                              float(pp.bg_ratio), bool(pp.use_bg), inv_batch, _keep, self.exact_cull)
