"""Drop-in for the reference's ``losses/lw.py`` (instance-whitening Gram loss) on B200.

    lw_loss(x, mask=None) -> 0-dim loss          (reference: losses/lw.py:5-18; imported in trainers/dgtrainer.py:24)

x [N, C, H, W], mask [N, 1, H, W] or None.  Per-(n, c) standardisation with the unbiased variance, optional spatial
mask, Gram on the tensor cores (csrc/isw_gram_tc.cu, the kernel of the ISW path), sum of the squared strictly-upper
entries; the backward is the ISW path's dX = S X GEMM followed by the standardisation backward.

fp16 / bf16 input (``torch.autocast``) runs natively and the standardised map is never materialised: one kernel writes
the per-plane mean / sd / invstd, the Gram's and dY = S Y's converter warps standardise (and mask) the half map as they
load it, and the standardisation backward recomputes it from x.  Loss and gradient are those of the fp32 route on
``x.float()`` bit for bit (the gradient rounded to the input dtype).  Autograd keeps the half x, the per-plane statistics,
the Gram and the workspace.  Shapes the half tensor-core kernels do not tile (HW % 8 != 0, C < 32, C % 4 != 0, a
misaligned view) and ``DGVCC_ISW_TENSOR_CORES=0`` take the upcast route; the forward's choice holds for its backward.
"""
import torch

from .. import _native


def _forward_half(ctx, x, m, dt):
    """The native route for a half x; False (nothing kept) when the shape is not one the half kernels tile."""
    n, c, h, w = x.shape
    hw = h * w
    dev = x.device
    lib = _native.lib()
    stream = _native.stream_ptr(dev)
    xh = x.detach().contiguous().view(n, c, hw)
    stats = torch.empty((3, n * c), dtype=torch.float32, device=dev)
    mean, sd, invstd = stats[0], stats[1], stats[2]
    _native.check(lib.dgvcc_lw_standardize_stats_h(_native.ptr(xh), dt, n, c, hw, 1e-5, _native.ptr(mean), _native.ptr(sd),
                                                   _native.ptr(invstd), stream), "dgvcc_lw_standardize_stats_h")
    nbytes = lib.dgvcc_isw_workspace_bytes(n, c, hw)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    gram = torch.empty((n, c, c), dtype=torch.float32, device=dev)
    rc = lib.dgvcc_lw_gram_h(_native.ptr(xh), dt, _native.ptr(mean), _native.ptr(sd), _native.ptr(m), n, c, hw,
                             _native.ptr(ws), nbytes, _native.ptr(gram), stream)
    if rc == _native.ERR_UNSUPPORTED:
        return None
    _native.check(rc, "dgvcc_lw_gram_h")
    loss = torch.empty((1,), dtype=torch.float32, device=dev)
    _native.check(lib.dgvcc_lw_loss_forward(_native.ptr(gram), n, c, hw, _native.ptr(ws), nbytes, _native.ptr(loss), stream),
                  "dgvcc_lw_loss_forward")
    ctx.save_for_backward(xh, stats, gram, ws)
    ctx.mask = m
    ctx.meta = (x.shape, x.dtype, nbytes)
    ctx.half = dt
    return loss.reshape(())


def _backward_half(ctx, grad_loss):
    xh, stats, gram, ws = ctx.saved_tensors
    shape, dtype, nbytes = ctx.meta
    n, c, hw = xh.shape
    dev = xh.device
    lib = _native.lib()
    stream = _native.stream_ptr(dev)
    mean, sd, invstd = stats[0], stats[1], stats[2]
    g = grad_loss.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
    dy = torch.empty((n, c, hw), dtype=torch.float32, device=dev)
    _native.check(lib.dgvcc_lw_loss_backward_h(_native.ptr(xh), ctx.half, _native.ptr(mean), _native.ptr(sd),
                                               _native.ptr(ctx.mask), _native.ptr(gram), _native.ptr(g), n, c, hw,
                                               _native.ptr(ws), nbytes, _native.ptr(dy), stream), "dgvcc_lw_loss_backward_h")
    dx = torch.empty_like(xh)
    _native.check(lib.dgvcc_lw_standardize_backward_h(_native.ptr(dy), _native.ptr(xh), ctx.half, _native.ptr(mean),
                                                      _native.ptr(sd), _native.ptr(invstd), _native.ptr(ctx.mask), n, c,
                                                      hw, _native.ptr(dx), stream), "dgvcc_lw_standardize_backward_h")
    return dx.view(shape), None


class _LwLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, mask):
        _native.require_cuda(x, "lw_loss")
        n, c, h, w = x.shape
        hw = h * w
        dev = x.device
        lib = _native.lib()
        stream = _native.stream_ptr(dev)
        m = None
        if mask is not None:
            m = mask.detach().to(device=dev, dtype=torch.float32).reshape(n, hw).contiguous()
        ctx.half = None
        dt = _native.half_code(x.dtype)
        if dt is not None and _native.use_tensor_cores():
            loss = _forward_half(ctx, x, m, dt)
            if loss is not None:
                return loss
        xc = x.detach().to(torch.float32).contiguous()
        yhat = torch.empty((n, c, hw), dtype=torch.float32, device=dev)
        ym = torch.empty_like(yhat) if m is not None else None
        invstd = torch.empty((n * c,), dtype=torch.float32, device=dev)
        _native.check(lib.dgvcc_lw_standardize_forward(_native.ptr(xc), _native.ptr(m), n, c, hw, 1e-5, _native.ptr(yhat),
                                                       _native.ptr(ym), _native.ptr(invstd), stream),
                      "dgvcc_lw_standardize_forward")
        y = ym if m is not None else yhat
        nbytes = lib.dgvcc_isw_workspace_bytes(n, c, hw)
        ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        gram = torch.empty((n, c, c), dtype=torch.float32, device=dev)
        _native.check(lib.dgvcc_isw_gram(_native.ptr(y), n, c, hw, _native.use_tensor_cores(), _native.ptr(ws), nbytes,
                                         _native.ptr(gram), stream), "dgvcc_isw_gram")
        loss = torch.empty((1,), dtype=torch.float32, device=dev)
        _native.check(lib.dgvcc_lw_loss_forward(_native.ptr(gram), n, c, hw, _native.ptr(ws), nbytes, _native.ptr(loss),
                                                stream), "dgvcc_lw_loss_forward")
        ctx.save_for_backward(yhat, y, invstd, gram, ws)
        ctx.mask = m
        ctx.meta = (x.shape, x.dtype, nbytes)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, grad_loss):
        if ctx.half is not None:
            return _backward_half(ctx, grad_loss)
        yhat, y, invstd, gram, ws = ctx.saved_tensors
        shape, dtype, nbytes = ctx.meta
        n, c, hw = yhat.shape
        dev = yhat.device
        lib = _native.lib()
        stream = _native.stream_ptr(dev)
        g = grad_loss.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
        dy = torch.empty_like(yhat)
        _native.check(lib.dgvcc_lw_loss_backward(_native.ptr(y), _native.ptr(gram), _native.ptr(g), n, c, hw,
                                                 _native.use_tensor_cores(), _native.ptr(ws), nbytes, _native.ptr(dy),
                                                 stream),
                      "dgvcc_lw_loss_backward")
        dx = torch.empty_like(yhat)
        _native.check(lib.dgvcc_lw_standardize_backward(_native.ptr(dy), _native.ptr(yhat), _native.ptr(invstd),
                                                        _native.ptr(ctx.mask), n, c, hw, _native.ptr(dx), stream),
                      "dgvcc_lw_standardize_backward")
        return dx.view(shape).to(dtype), None


def lw_loss(x, mask=None):
    # Instance Whitening Loss
    # x: (N, C, H, W)
    # mask: (N, 1, H, W)
    # return: scalar
    return _LwLoss.apply(x, mask)
