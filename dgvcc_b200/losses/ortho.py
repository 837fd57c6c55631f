"""Drop-in for the reference's ``losses/ortho.py`` (orthogonality loss between two feature banks) on B200.

    ortho_loss(x, y) -> 0-dim loss               (reference: losses/ortho.py:5-11; imported in trainers/dgtrainer.py:23)

x, y [C, P].  ``x y^T`` is the off-diagonal block of the Gram of the stacked operand ``[x; y]``, so the forward is
the ISW path's tensor-core Gram kernel; the two gradients are two dX = S X GEMMs of the same path.

fp16 / bf16 inputs (``torch.autocast``, both of one dtype) run natively: ``[x; y]`` is stacked in the input dtype, the
Gram and the two dX GEMMs read it directly, and autograd keeps the half stack.  Loss and gradients are those of the fp32
route on the upcast inputs bit for bit (gradients rounded to the input dtype).  Shapes the half tensor-core kernels do
not tile (P % 8 != 0, C < 32, C % 4 != 0) and ``DGVCC_ISW_TENSOR_CORES=0`` take the upcast route; the forward's choice
holds for its backward.
"""
import torch

from .. import _native


class _OrthoLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, y):
        _native.require_cuda(x, "ortho_loss")
        _native.require_cuda(y, "ortho_loss")
        if x.dim() != 2 or x.shape != y.shape:
            raise ValueError(f"ortho_loss expects two [C, P] tensors, got {tuple(x.shape)} and {tuple(y.shape)}")
        c, p = x.shape
        dev = x.device
        lib = _native.lib()
        stream = _native.stream_ptr(dev)
        nbytes = lib.dgvcc_isw_workspace_bytes(1, 2 * c, p)
        ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        gram = torch.empty((2 * c, 2 * c), dtype=torch.float32, device=dev)
        # the Gram tiles [x; y] (2C rows); the two dX GEMMs need C >= 32 and C % 4 == 0 themselves
        ctx.half = None
        if x.dtype == y.dtype and c >= 32 and c % 4 == 0 and _native.use_tensor_cores():
            ctx.half = _native.half_code(x.dtype)
        if ctx.half is not None:
            z = torch.cat([x.detach(), y.detach()], dim=0).contiguous()  # [2C, P] in the input dtype
            rc = lib.dgvcc_isw_gram_h(_native.ptr(z), ctx.half, 1, 2 * c, p, _native.ptr(ws), nbytes, _native.ptr(gram),
                                      stream)
            if rc == _native.ERR_UNSUPPORTED:
                ctx.half = None
            else:
                _native.check(rc, "dgvcc_isw_gram_h")
        if ctx.half is None:
            z = torch.cat([x.detach().to(torch.float32), y.detach().to(torch.float32)], dim=0).contiguous()  # [2C, P]
            _native.check(lib.dgvcc_isw_gram(_native.ptr(z), 1, 2 * c, p, _native.use_tensor_cores(), _native.ptr(ws),
                                             nbytes, _native.ptr(gram), stream), "dgvcc_isw_gram")
        loss = torch.empty((1,), dtype=torch.float32, device=dev)
        _native.check(lib.dgvcc_ortho_loss_forward(_native.ptr(gram), c, p, _native.ptr(ws), nbytes, _native.ptr(loss), stream),
                      "dgvcc_ortho_loss_forward")
        ctx.save_for_backward(z, gram, ws)
        ctx.meta = (c, p, nbytes, x.dtype, y.dtype)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, grad_loss):
        z, gram, ws = ctx.saved_tensors
        c, p, nbytes, xdt, ydt = ctx.meta
        dev = z.device
        g = grad_loss.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
        if ctx.half is not None:
            gx = torch.empty((c, p), dtype=z.dtype, device=dev)
            gy = torch.empty_like(gx)
            _native.check(_native.lib().dgvcc_ortho_loss_backward_h(
                _native.ptr(z[:c]), _native.ptr(z[c:]), ctx.half, _native.ptr(gram), _native.ptr(g), c, p, _native.ptr(ws),
                nbytes, _native.ptr(gx), _native.ptr(gy), _native.stream_ptr(dev)), "dgvcc_ortho_loss_backward_h")
            return gx, gy
        gx = torch.empty((c, p), dtype=torch.float32, device=dev)
        gy = torch.empty((c, p), dtype=torch.float32, device=dev)
        _native.check(_native.lib().dgvcc_ortho_loss_backward(
            _native.ptr(z[:c]), _native.ptr(z[c:]), _native.ptr(gram), _native.ptr(g), c, p, _native.use_tensor_cores(),
            _native.ptr(ws), nbytes, _native.ptr(gx), _native.ptr(gy), _native.stream_ptr(dev)),
            "dgvcc_ortho_loss_backward")
        return gx.to(xdt), gy.to(ydt)


def ortho_loss(x, y):
    # x: (C, P)
    # y: (C, P)
    # return: scalar
    return _OrthoLoss.apply(x, y)
