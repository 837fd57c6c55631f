"""Drop-in for the reference's ``models/ISW/instance_whitening.py`` on B200.

Same names and signatures as the reference (instance_whitening.py:5, 19, 30), imported by name in
``models/ISW/__init__.py:12``, ``deepv3.py:33`` and ``Resnet.py:41``:

    InstanceWhitening(dim).forward(x)                       -> (x_norm, x_norm)
    get_covariance_matrix(f_map, eye=None)                  -> (f_cor [B,C,C], B)
    instance_whitening_loss(f_map, eye, mask_matrix, margin, num_remove_cov) -> 0-dim loss

The Gram X X^T is the only dense contraction of the path: csrc/isw_gram_tc.cu runs it on the
tcgen05 tensor cores (3xTF32 split, fp32 accumulation in TMEM) where the shape tiles, otherwise
the exact-fp32 CUDA-core kernel of csrc/isw_kernels.cu.  ``margin`` / ``num_remove_cov`` may be
Python numbers or 0-dim tensors, as in the reference (cov_settings.py:47,73).

fp16 / bf16 feature maps (``torch.autocast`` training) run natively: the kernels read and write the half tensors, and
autograd keeps the half map (plus the per-plane mean / invstd of the instance norm) instead of fp32 copies.  The
results are those of the fp32 path on the upcast map, bit for bit: y and the gradients come back in the input dtype,
``f_cor`` and the loss are fp32.  Shapes the half tensor-core kernels do not tile (HW % 8 != 0, C < 32, C % 4 != 0,
a misaligned view) and ``DGVCC_ISW_TENSOR_CORES=0`` take the upcast route; the forward's choice holds for its backward.
"""
import os

import weakref

import torch
import torch.nn as nn

from ... import _native


def _use_tc():
    return int(os.environ.get("DGVCC_ISW_TENSOR_CORES", "1"))


def _f32c(t, dev=None):
    """``t`` as a detached contiguous fp32 tensor (on ``dev``); no copy, and one call only, when it already is one."""
    if t.dtype is torch.float32 and t.is_contiguous() and (dev is None or t.device == dev):
        return t.detach()
    return t.detach().to(device=dev if dev is not None else t.device, dtype=torch.float32).contiguous()


_HALF = {torch.float16: _native.DTYPE_F16, torch.bfloat16: _native.DTYPE_BF16}


def _half3d(f_map):
    """(dtype code, contiguous half [B,C,HW] view) when ``f_map`` is fp16 / bf16 and the tensor cores are on, else
    (None, None): the caller then takes the fp32 route of ``_as3d``."""
    dt = _HALF.get(f_map.dtype)
    if dt is None or not _use_tc():
        return None, None
    _native.require_cuda(f_map, "instance_whitening")
    b, c, h, w = f_map.shape
    return dt, f_map.detach().contiguous().view(b, c, h * w)


def _as3d(f_map):
    _native.require_cuda(f_map, "instance_whitening")
    b, c, h, w = f_map.shape
    return _f32c(f_map).view(b, c, h * w), b, c, h * w


_UNSUPPORTED = -3  # DGVCC_ERR_UNSUPPORTED

_ws_bytes = {}


def _workspace(b, c, hw, dev):
    n = _ws_bytes.get((b, c, hw))
    if n is None:
        n = _ws_bytes[(b, c, hw)] = _native.lib().dgvcc_isw_workspace_bytes(b, c, hw)
    return torch.empty((n,), dtype=torch.uint8, device=dev), n


_scalars = {}  # (device, value) -> 1-element device tensor for Python-number margins / counts (read-only)


def _scalar(v, dev):
    if torch.is_tensor(v):
        return _f32c(v, dev).reshape(1)
    key = (dev, float(v))
    t = _scalars.get(key)
    if t is None:
        if len(_scalars) > 256:
            _scalars.clear()
        t = _scalars[key] = torch.full((1,), float(v), dtype=torch.float32, device=dev)
    return t


class _InstanceNorm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, eps):
        _native.require_cuda(x, "InstanceWhitening")
        b, c, h, w = x.shape
        ctx.half = _HALF.get(x.dtype)
        if ctx.half is not None:  # y = RN(fp32 y) in the input dtype; the backward recomputes fp32 y from x
            xc = x.detach().contiguous()
            y = torch.empty_like(xc)
            mean = torch.empty((b * c,), dtype=torch.float32, device=x.device)
            invstd = torch.empty_like(mean)
            _native.check(_native.lib().dgvcc_isw_instnorm_forward_h(
                _native.ptr(xc), ctx.half, b * c, h * w, eps, _native.ptr(y), _native.ptr(mean), _native.ptr(invstd),
                _native.stream_ptr(x.device)), "dgvcc_isw_instnorm_forward_h")
            ctx.save_for_backward(xc, mean, invstd)
            return y
        xc = _f32c(x)
        y = torch.empty_like(xc)
        mean = torch.empty((b * c,), dtype=torch.float32, device=x.device)
        invstd = torch.empty_like(mean)
        _native.check(_native.lib().dgvcc_isw_instnorm_forward(
            _native.ptr(xc), b * c, h * w, eps, _native.ptr(y), _native.ptr(mean), _native.ptr(invstd),
            _native.stream_ptr(x.device)), "dgvcc_isw_instnorm_forward")
        ctx.save_for_backward(y, invstd)
        ctx.in_dtype = x.dtype
        return y.to(x.dtype)

    @staticmethod
    def backward(ctx, dy):
        if ctx.half is not None:
            xc, mean, invstd = ctx.saved_tensors
            b, c, h, w = xc.shape
            g = dy.contiguous()
            dx = torch.empty_like(xc)
            _native.check(_native.lib().dgvcc_isw_instnorm_backward_h(
                _native.ptr(g), _native.ptr(xc), _native.ptr(mean), _native.ptr(invstd), ctx.half, b * c, h * w,
                _native.ptr(dx), _native.stream_ptr(xc.device)), "dgvcc_isw_instnorm_backward_h")
            return dx, None
        y, invstd = ctx.saved_tensors
        b, c, h, w = y.shape
        g = _f32c(dy)
        dx = torch.empty_like(y)
        _native.check(_native.lib().dgvcc_isw_instnorm_backward(
            _native.ptr(g), _native.ptr(y), _native.ptr(invstd), b * c, h * w, _native.ptr(dx),
            _native.stream_ptr(y.device)), "dgvcc_isw_instnorm_backward")
        return dx.to(ctx.in_dtype), None


class InstanceWhitening(nn.Module):

    def __init__(self, dim):
        super(InstanceWhitening, self).__init__()
        self.dim = dim
        self.eps = 1e-5  # nn.InstanceNorm2d(dim, affine=False) default, instance_whitening.py:9

    def forward(self, x):
        x = _InstanceNorm.apply(x, self.eps)
        w = x
        return x, w


class _Covariance(torch.autograd.Function):
    @staticmethod
    def forward(ctx, f_map, eye):
        ctx.half, x = _half3d(f_map)
        if ctx.half is not None:
            b, c, hw = x.shape
            dev = x.device
            ws, n = _workspace(b, c, hw, dev)
            f_cor = torch.empty((b, c, c), dtype=torch.float32, device=dev)
            rc = _native.lib().dgvcc_isw_covariance_h(_native.ptr(x), ctx.half, _native.ptr(_f32c(eye, dev)), b, c, hw,
                                                      _native.ptr(ws), n, _native.ptr(f_cor), _native.stream_ptr(dev))
            if rc == _UNSUPPORTED:
                ctx.half = None
            else:
                _native.check(rc, "dgvcc_isw_covariance_h")
                ctx.save_for_backward(x)
                ctx.meta = (f_map.shape, f_map.dtype)
                return f_cor
        x, b, c, hw = _as3d(f_map)
        dev = x.device
        ws, n = _workspace(b, c, hw, dev)
        f_cor = torch.empty((b, c, c), dtype=torch.float32, device=dev)
        eye32 = _f32c(eye, dev)
        _native.check(_native.lib().dgvcc_isw_covariance(
            _native.ptr(x), _native.ptr(eye32), b, c, hw, _use_tc(), _native.ptr(ws), n, _native.ptr(f_cor),
            _native.stream_ptr(dev)), "dgvcc_isw_covariance")
        ctx.save_for_backward(x)
        ctx.meta = (f_map.shape, f_map.dtype)
        return f_cor

    @staticmethod
    def backward(ctx, d_fcor):
        (x,) = ctx.saved_tensors
        b, c, hw = x.shape
        dev = x.device
        ws, n = _workspace(b, c, hw, dev)
        g = _f32c(d_fcor)
        dx = torch.empty_like(x)
        if ctx.half is not None:
            _native.check(_native.lib().dgvcc_isw_covariance_backward_h(
                _native.ptr(x), ctx.half, _native.ptr(g), b, c, hw, _native.ptr(ws), n, _native.ptr(dx),
                _native.stream_ptr(dev)), "dgvcc_isw_covariance_backward_h")
            return dx.view(ctx.meta[0]), None
        _native.check(_native.lib().dgvcc_isw_covariance_backward(
            _native.ptr(x), _native.ptr(g), b, c, hw, _use_tc(), _native.ptr(ws), n, _native.ptr(dx),
            _native.stream_ptr(dev)), "dgvcc_isw_covariance_backward")
        shape, dtype = ctx.meta
        return dx.view(shape).to(dtype), None


_binary_masks = {}  # id(mask tensor) -> (version, bool); dropped when the tensor dies


def _mask_is_binary(mask):
    """True when every entry is 0 or 1: one device read-back per mask tensor (they live for an epoch,
    cov_settings.py:52-73), cached until the tensor is modified in place or freed."""
    key = id(mask)
    hit = _binary_masks.get(key)
    if hit is None or hit[0] != mask._version:
        if hit is None:
            weakref.finalize(mask, _binary_masks.pop, key, None)
        hit = _binary_masks[key] = (mask._version, bool(((mask == 0) | (mask == 1)).all()))
    return hit[1]


class _WhiteningLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, f_map, eye, mask_matrix, margin, num_remove_cov):
        ctx.half, x = _half3d(f_map)
        if ctx.half is None:
            x, b, c, hw = _as3d(f_map)
        else:
            b, c, hw = x.shape
        dev = x.device
        lib = _native.lib()
        ws, n = _workspace(b, c, hw, dev)
        f_cor = torch.empty((b, c, c), dtype=torch.float32, device=dev)
        eye32 = _f32c(eye, dev)
        mask = _f32c(mask_matrix, dev)
        if mask.shape != (c, c):
            raise ValueError(f"mask_matrix must be [{c},{c}], got {tuple(mask.shape)}")
        mg, nr = _scalar(margin, dev), _scalar(num_remove_cov, dev)
        stream = _native.stream_ptr(dev)
        if ctx.half is not None:
            rc = lib.dgvcc_isw_covariance_h(_native.ptr(x), ctx.half, _native.ptr(eye32), b, c, hw, _native.ptr(ws), n,
                                            _native.ptr(f_cor), stream)
            if rc == _UNSUPPORTED:  # a shape the half tensor-core kernels do not tile: upcast, as for every other dtype
                ctx.half = None
                x = _as3d(f_map)[0]
            else:
                _native.check(rc, "dgvcc_isw_covariance_h")
        if ctx.half is None:
            _native.check(lib.dgvcc_isw_covariance(_native.ptr(x), _native.ptr(eye32), b, c, hw, _use_tc(), _native.ptr(ws),
                                                   n, _native.ptr(f_cor), stream), "dgvcc_isw_covariance")
        loss = torch.empty((1,), dtype=torch.float32, device=dev)
        _native.check(lib.dgvcc_isw_loss_forward(_native.ptr(f_cor), _native.ptr(mask), _native.ptr(mg), _native.ptr(nr),
                                                 b, c, hw, _native.ptr(ws), n, _native.ptr(loss), stream),
                      "dgvcc_isw_loss_forward")
        ctx.save_for_backward(x, f_cor, mask, nr, ws)
        ctx.meta = (f_map.shape, f_map.dtype, n, _mask_is_binary(mask_matrix))
        return loss.reshape(())

    @staticmethod
    def backward(ctx, grad_loss):
        x, f_cor, mask, nr, ws = ctx.saved_tensors
        shape, dtype, n, binary = ctx.meta
        b, c, hw = x.shape
        dev = x.device
        g = _f32c(grad_loss, dev).reshape(1)
        dx = torch.empty_like(x)
        if ctx.half is not None:
            _native.check(_native.lib().dgvcc_isw_loss_backward_h(
                _native.ptr(x), ctx.half, _native.ptr(f_cor), _native.ptr(mask), _native.ptr(nr), _native.ptr(g), b, c, hw,
                int(binary), _native.ptr(ws), n, _native.ptr(dx), _native.stream_ptr(dev)), "dgvcc_isw_loss_backward_h")
            return dx.view(shape), None, None, None, None
        _native.check(_native.lib().dgvcc_isw_loss_backward(
            _native.ptr(x), _native.ptr(f_cor), _native.ptr(mask), _native.ptr(nr), _native.ptr(g), b, c, hw, _use_tc(),
            int(binary), _native.ptr(ws), n, _native.ptr(dx), _native.stream_ptr(dev)), "dgvcc_isw_loss_backward")
        return dx.view(shape).to(dtype), None, None, None, None


def instance_whitening_loss(f_map, eye, mask_matrix, margin, num_remove_cov):
    return _WhiteningLoss.apply(f_map, eye, mask_matrix, margin, num_remove_cov)


def get_covariance_matrix(f_map, eye=None):
    B, C, H, W = f_map.shape  # i-th feature size (B X C X H X W)
    if eye is None:
        eye = torch.eye(C, device=f_map.device)
    return _Covariance.apply(f_map, eye), B


def variance_of_covariance(f_map, eye, reverse_eye):
    """The statistic of ``cal_covstat`` (models/ISW/__init__.py:93-104): ``torch.var(f_cor * reverse_eye, dim=0)``
    with ``f_cor`` the covariance of the (image, augmented image) pair; feed it to
    ``CovMatrix_ISW.set_variance_of_covariance``.  No gradient (the reference calls it under ``no_grad``)."""
    with torch.no_grad():
        f_cor, b = get_covariance_matrix(f_map, eye=eye)
        c = f_cor.shape[-1]
        rev = reverse_eye.detach().to(device=f_cor.device, dtype=torch.float32).contiguous()
        out = torch.empty((c, c), dtype=torch.float32, device=f_cor.device)
        _native.check(_native.lib().dgvcc_isw_covstat_var(_native.ptr(f_cor), _native.ptr(rev), b, c, _native.ptr(out),
                                                          _native.stream_ptr(f_cor.device)), "dgvcc_isw_covstat_var")
    return out
