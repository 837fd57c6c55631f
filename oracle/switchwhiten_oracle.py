"""CPU oracle for switchable whitening -- TEST INFRASTRUCTURE, not product code.

Restates /root/reference/models/ISW/switchwhiten.py:84-183 (``SwitchWhiten2d.forward``) and
/root/reference/models/ISW/sync_switchwhiten.py:9-56,135-223 (``SyncMeanCov`` / ``SyncSwitchWhiten2d.forward``;
byte-identical copies live under models/SW/ops/) -- SURVEY.md section 8f, rank 4.  Two restatements:

* ``forward``: the reference's op sequence in torch (any dtype), gradients by autograd, the batch statistics through a
  custom Function with SyncMeanCov's hand-written backward when a process group is given.  Pinned by
  tests/golden/sw_cases.npz, produced by the unmodified files loaded by path (tests/golden/make_golden.py: make_sw).
* ``decomposed``: the same mathematics in the order the CUDA kernels evaluate it (one-pass moments shifted by a
  sample mean of each plane, batch covariance from the per-sample ones, closed-form adjoint of the Newton iteration,
  the two affine passes), numpy fp64, no autograd.  tests/test_oracle_sw.py checks it against ``forward``; it is the
  specification the kernels in dgvcc_b200/csrc/sw_kernels.cu are compared with.
"""
import numpy as np
import torch


# ----------------------------------------------------------------------------------------------------------------
# 1. the reference's op sequence
# ----------------------------------------------------------------------------------------------------------------

class _SyncMeanCov(torch.autograd.Function):
    """sync_switchwhiten.py:9-56 with ``all_reduce`` / ``world_size`` passed in (no global process-group lookups)."""

    @staticmethod
    def forward(ctx, in_data, running_mean, running_cov, momentum, training, all_reduce, world_size):
        g, c, nhw = in_data.size()
        ctx.nhw, ctx.training, ctx.all_reduce, ctx.world_size = nhw, training, all_reduce, world_size
        if training:
            mean_bn = in_data.mean(-1, keepdim=True)
            all_reduce(mean_bn)
            mean_bn /= world_size
            in_data_bn = in_data - mean_bn
            cov_bn = torch.bmm(in_data_bn, in_data_bn.transpose(1, 2)).div(nhw)
            all_reduce(cov_bn)
            cov_bn /= world_size
            running_mean.mul_(momentum)
            running_mean.add_((1 - momentum) * mean_bn.data)
            running_cov.mul_(momentum)
            running_cov.add_((1 - momentum) * cov_bn.data)
        else:
            mean_bn, cov_bn = running_mean.clone(), running_cov.clone()
        ctx.save_for_backward(in_data.data, mean_bn.data)
        return mean_bn, cov_bn

    @staticmethod
    def backward(ctx, grad_mean_out, grad_cov_out):
        in_data, mean_bn = ctx.saved_tensors
        grad_mean_out, grad_cov_out = grad_mean_out.clone(), grad_cov_out.clone()
        world_size = 1
        if ctx.training:
            ctx.all_reduce(grad_mean_out)
            ctx.all_reduce(grad_cov_out)
            world_size = ctx.world_size
        grad_cov_out = (grad_cov_out + grad_cov_out.transpose(1, 2)) / 2
        grad_cov_in = 2 * torch.bmm(grad_cov_out, (in_data - mean_bn)) / (ctx.nhw * world_size)
        grad_mean_in = grad_mean_out / ctx.nhw / world_size
        return grad_mean_in + grad_cov_in, None, None, None, None, None, None


def forward(x, sw_mean_weight, sw_var_weight, weight, bias, running_mean, running_cov, *, num_pergroup=16, sw_type=2,
            T=5, eps=1e-5, momentum=0.99, training=True, all_reduce=None, world_size=1):
    """y = SwitchWhiten2d(x).  ``sw_var_weight=None`` is tie_weight; ``weight=None`` is affine=False; the running
    buffers are updated in place when training (switchwhiten.py:101-104).  With ``all_reduce`` the batch statistics
    follow SyncMeanCov; without it they are the plain autograd graph of switchwhiten.py:94-99."""
    n, ch, h, w = x.shape
    c, g = num_pergroup, ch // num_pergroup
    in_data_t = x.transpose(0, 1).contiguous().view(g, c, -1)
    if all_reduce is not None:
        mean_bn, cov_bn = _SyncMeanCov.apply(in_data_t, running_mean, running_cov, momentum, training, all_reduce,
                                             world_size)
    elif training:
        mean_bn = in_data_t.mean(-1, keepdim=True)
        in_data_bn = in_data_t - mean_bn
        cov_bn = torch.bmm(in_data_bn, in_data_bn.transpose(1, 2)).div(h * w * n)
        running_mean.mul_(momentum)
        running_mean.add_((1 - momentum) * mean_bn.data)
        running_cov.mul_(momentum)
        running_cov.add_((1 - momentum) * cov_bn.data)
    else:
        mean_bn, cov_bn = running_mean, running_cov
    mean_bn = mean_bn.view(1, g, c, 1).expand(n, g, c, 1).contiguous().view(n * g, c, 1)
    cov_bn = cov_bn.view(1, g, c, c).expand(n, g, c, c).contiguous().view(n * g, c, c)
    in_data = x.reshape(n * g, c, -1)
    eye = torch.eye(c, dtype=x.dtype).view(1, c, c).expand(n * g, c, c)
    mean_in = in_data.mean(-1, keepdim=True)
    x_in = in_data - mean_in
    cov_in = torch.bmm(x_in, x_in.transpose(1, 2)).div(h * w)
    if sw_type in (3, 5):
        flat = x.reshape(n, -1)
        mean_ln = flat.mean(-1, keepdim=True).view(n, 1, 1, 1).expand(n, g, 1, 1).contiguous().view(n * g, 1, 1)
        var_ln = flat.var(-1, keepdim=True).view(n, 1, 1, 1).expand(n, g, 1, 1).contiguous().view(n * g, 1, 1) * eye
    if sw_type == 5:
        var_bn = torch.diag_embed(torch.diagonal(cov_bn, dim1=-2, dim2=-1))
        var_in = torch.diag_embed(torch.diagonal(cov_in, dim1=-2, dim2=-1))
    mean_weight = torch.softmax(sw_mean_weight, 0)
    var_weight = mean_weight if sw_var_weight is None else torch.softmax(sw_var_weight, 0)
    if sw_type == 2:
        mean = mean_weight[0] * mean_bn + mean_weight[1] * mean_in
        cov = var_weight[0] * cov_bn + var_weight[1] * cov_in + eps * eye
    elif sw_type == 3:
        mean = mean_weight[0] * mean_bn + mean_weight[1] * mean_in + mean_weight[2] * mean_ln
        cov = var_weight[0] * cov_bn + var_weight[1] * cov_in + var_weight[2] * var_ln + eps * eye
    else:  # 5: note the covariance reuses weights 0 and 1 for the diagonal-only terms (switchwhiten.py:160-163)
        mean = (mean_weight[0] + mean_weight[2]) * mean_bn + (mean_weight[1] + mean_weight[3]) * mean_in + \
            mean_weight[4] * mean_ln
        cov = var_weight[0] * cov_bn + var_weight[1] * cov_in + var_weight[0] * var_bn + var_weight[1] * var_in + \
            var_weight[4] * var_ln + eps * eye
    p = torch.eye(c, dtype=x.dtype).expand(n * g, c, c)
    r_tr = (cov * p).sum((1, 2), keepdim=True).reciprocal()
    cov_n = cov * r_tr
    for _ in range(T):
        p = torch.baddbmm(p, torch.matrix_power(p, 3), cov_n, beta=1.5, alpha=-0.5)
    wm = p * r_tr.sqrt()
    x_hat = torch.bmm(wm, in_data - mean).view(n, ch, h, w)
    if weight is not None:
        x_hat = x_hat * weight.view(1, ch, 1, 1) + bias.view(1, ch, 1, 1)
    return x_hat


def forward_backward(x, gy, sw_mean_weight, sw_var_weight, weight, bias, running_mean, running_cov, **kw):
    """Returns (y, dict of gradients); inputs are cloned, the running buffers passed in are updated in place."""
    leaves = {"x": x, "sw_mean_weight": sw_mean_weight, "sw_var_weight": sw_var_weight, "weight": weight, "bias": bias}
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in leaves.items() if v is not None}
    y = forward(leaves["x"], leaves["sw_mean_weight"], leaves.get("sw_var_weight"), leaves.get("weight"),
                leaves.get("bias"), running_mean, running_cov, **kw)
    y.backward(gy)
    return y.detach(), {k: v.grad for k, v in leaves.items()}


# ----------------------------------------------------------------------------------------------------------------
# 2. the kernels' evaluation order (numpy fp64)
# ----------------------------------------------------------------------------------------------------------------

def _mix(sw_type, mw, vw):
    """(a_bn, a_in, a_ln), (b_bn, b_in, b_ln), (d_bn, d_in): mean, covariance and diagonal-only coefficients."""
    if sw_type == 2:
        return (mw[0], mw[1], 0.0), (vw[0], vw[1], 0.0), (0.0, 0.0)
    if sw_type == 3:
        return (mw[0], mw[1], mw[2]), (vw[0], vw[1], vw[2]), (0.0, 0.0)
    return (mw[0] + mw[2], mw[1] + mw[3], mw[4]), (vw[0], vw[1], vw[4]), (vw[0], vw[1])


def _softmax(v):
    e = np.exp(v - v.max())
    return e / e.sum()


def newton_forward(cov, T):
    """switchwhiten.py:166-175 for one c x c matrix; returns wm and what the adjoint needs."""
    c = cov.shape[0]
    r = 1.0 / np.trace(cov)
    cov_n = cov * r
    ps = [np.eye(c)]
    for _ in range(T):
        p = ps[-1]
        ps.append(1.5 * p - 0.5 * (p @ p @ p) @ cov_n)
    return ps[-1] * np.sqrt(r), (ps, r, cov_n)


def newton_backward(g_wm, cov, saved):
    """d loss / d cov given d loss / d wm."""
    ps, r, cov_n = saved
    c = cov.shape[0]
    g_p = g_wm * np.sqrt(r)
    g_r = (g_wm * ps[-1]).sum() * 0.5 / np.sqrt(r)
    g_covn = np.zeros((c, c))
    for k in range(len(ps) - 2, -1, -1):
        p = ps[k]
        p2 = p @ p
        g_covn += -0.5 * (p2 @ p).T @ g_p
        g_p3 = -0.5 * g_p @ cov_n.T
        g_p = 1.5 * g_p + g_p3 @ p2.T + p.T @ g_p3 @ p.T + p2.T @ g_p3
    g_cov = g_covn * r
    g_r += (g_covn * cov).sum()
    return g_cov + (-g_r * r * r) * np.eye(c)


def sample_shift(xg):
    """The per-channel centre of the forward moments pass: the mean of up to 128 pixels of the plane (16 runs of 8
    consecutive pixels starting at (c hw) // 16, or every pixel when hw <= 128), rounded to fp32.  The kernel sums the sample in
    fp32 and may land an ulp away; any centre gives the same statistics up to rounding, so only the choice of pixels is
    specification."""
    hw = xg.shape[-1]
    idx = ((np.arange(16)[:, None] * hw) // 16 + np.arange(8)).ravel() if hw > 128 else np.arange(hw)
    return xg[..., idx].mean(-1).astype(np.float32).astype(np.float64)


def decomposed(x, gy, sw_mean_weight, sw_var_weight, weight, bias, running_mean, running_cov, *, num_pergroup=16,
               sw_type=2, T=5, eps=1e-5, training=True, all_reduce=None, world_size=1, stages=None):
    """Forward and backward in the kernels' order.  ``all_reduce(array)`` sums a numpy array over ranks in place (the
    four exchanges of SyncMeanCov); ``running_*`` are only read (eval mode).  Returns (y, grads, (mean_bn, cov_bn)).
    A dict passed as ``stages`` receives the intermediates the C entry points return: mean_in [n, g, c],
    cov_in [n, g, c, c], a_fwd [n, g, c, c], g_mean_bn [g, c] and g_cov_bn [g, c, c] (before any exchange)."""
    x = np.asarray(x, np.float64)
    gy = np.asarray(gy, np.float64)
    n, ch, h, w = x.shape
    c, g, hw = num_pergroup, ch // num_pergroup, h * w
    xg = x.reshape(n, g, c, hw)
    gyg = gy.reshape(n, g, c, hw)
    reduce_ = all_reduce if all_reduce is not None else (lambda a: a)

    # --- moments pass: one read of x, shifted by a sample mean of each channel -----------------------------------
    shift = sample_shift(xg)[..., None]
    s1 = (xg - shift).sum(-1)
    s2 = np.einsum("ngip,ngjp->ngij", xg - shift, xg - shift)
    delta = s1 / hw
    mean_in = shift[..., 0] + delta                                   # [n, g, c]
    cov_in = s2 / hw - delta[..., :, None] * delta[..., None, :]      # [n, g, c, c]

    # --- batch statistics from the per-sample ones ---------------------------------------------------------------
    if training:
        mean_bn = mean_in.mean(0)
        reduce_(mean_bn)
        mean_bn = mean_bn / world_size
        d = mean_in - mean_bn
        cov_bn = (cov_in + d[..., :, None] * d[..., None, :]).mean(0)
        reduce_(cov_bn)
        cov_bn = cov_bn / world_size
    else:
        mean_bn = np.asarray(running_mean, np.float64).reshape(g, c)
        cov_bn = np.asarray(running_cov, np.float64).reshape(g, c, c)

    # --- layer statistics from the per-sample ones ---------------------------------------------------------------
    mean_ln = mean_in.reshape(n, -1).mean(1)
    diag_in = np.einsum("ngii->ngi", cov_in)
    ln_scale = hw / (ch * hw - 1.0)
    var_ln = ln_scale * (diag_in + (mean_in - mean_ln[:, None, None]) ** 2).reshape(n, -1).sum(1)

    mw = _softmax(np.asarray(sw_mean_weight, np.float64))
    vw = mw if sw_var_weight is None else _softmax(np.asarray(sw_var_weight, np.float64))
    (a_bn, a_in, a_ln), (b_bn, b_in, b_ln), (d_bn, d_in) = _mix(sw_type, mw, vw)
    eye = np.eye(c)
    wgt = np.ones(ch) if weight is None else np.asarray(weight, np.float64)
    bia = np.zeros(ch) if bias is None else np.asarray(bias, np.float64)
    wgt_g, bia_g = wgt.reshape(g, c), bia.reshape(g, c)

    mean = a_bn * mean_bn[None] + a_in * mean_in + a_ln * mean_ln[:, None, None]
    cov = np.empty_like(cov_in)
    wm = np.empty_like(cov_in)
    saved = {}
    for i in range(n):
        for k in range(g):
            cov[i, k] = b_bn * cov_bn[k] + b_in * cov_in[i, k] + d_bn * np.diag(np.diag(cov_bn[k])) + \
                d_in * np.diag(np.diag(cov_in[i, k])) + (b_ln * var_ln[i] + eps) * eye
            wm[i, k], saved[i, k] = newton_forward(cov[i, k], T)

    # --- forward affine pass: y = A x + cst, A = diag(weight) wm, cst = bias - A mean -----------------------------
    a_fwd = wgt_g[None, :, :, None] * wm
    cst_fwd = bia_g[None] - np.einsum("ngij,ngj->ngi", a_fwd, mean)
    y = np.einsum("ngij,ngjp->ngip", a_fwd, xg) + cst_fwd[..., None]

    # --- backward moments pass: one read of x and gy -------------------------------------------------------------
    s_gy = gyg.sum(-1)                                                           # [n, g, c]
    k_raw = np.einsum("ngip,ngjp->ngij", gyg, xg - mean_in[..., None])          # centred on mean_in

    # --- small per-(n, g) adjoints -------------------------------------------------------------------------------
    k_c = k_raw + s_gy[..., :, None] * (mean_in - mean)[..., None, :]           # sum_p gy_i (x_j - mean_j)
    g_bias = s_gy.sum(0).reshape(-1)
    g_weight = np.einsum("ngij,ngij->gi", wm, k_c).reshape(-1)
    g_wm = wgt_g[None, :, :, None] * k_c
    g_mean = -np.einsum("ngij,ngi->ngj", wm, wgt_g[None] * s_gy)
    g_cov = np.empty_like(cov)
    for i in range(n):
        for k in range(g):
            g_cov[i, k] = newton_backward(g_wm[i, k], cov[i, k], saved[i, k])
    tr_g = np.einsum("ngii->ng", g_cov)
    diag_g = np.einsum("ngii->ngi", g_cov)

    # --- cross-(n, g) reductions ---------------------------------------------------------------------------------
    g_cov_in = b_in * g_cov + d_in * diag_g[..., None] * eye
    g_cov_bn = (b_bn * g_cov + d_bn * diag_g[..., None] * eye).sum(0)
    g_var_ln = b_ln * tr_g.sum(1)
    g_mean_ln = a_ln * g_mean.reshape(n, -1).sum(1)
    g_mean_in = a_in * g_mean + (g_mean_ln / ch)[:, None, None] + \
        (g_var_ln * ln_scale)[:, None, None] * 2.0 * (mean_in - mean_ln[:, None, None])
    g_cov_in = g_cov_in + (g_var_ln * ln_scale)[:, None, None, None] * eye
    g_mean_bn = a_bn * g_mean.sum(0)

    dot_cov_bn = np.einsum("ngij,gij->", g_cov, cov_bn)
    dot_cov_in = np.einsum("ngij,ngij->", g_cov, cov_in)
    dot_diag_bn = np.einsum("ngi,gi->", diag_g, np.einsum("gii->gi", cov_bn))
    dot_diag_in = (diag_g * diag_in).sum()
    dot_ln = (tr_g.sum(1) * var_ln).sum()
    dot_mean_bn = (g_mean * mean_bn[None]).sum()
    dot_mean_in = (g_mean * mean_in).sum()
    dot_mean_ln = (g_mean.reshape(n, -1).sum(1) * mean_ln).sum()
    if sw_type == 2:
        gm, gv = np.array([dot_mean_bn, dot_mean_in]), np.array([dot_cov_bn, dot_cov_in])
    elif sw_type == 3:
        gm = np.array([dot_mean_bn, dot_mean_in, dot_mean_ln])
        gv = np.array([dot_cov_bn, dot_cov_in, dot_ln])
    else:
        gm = np.array([dot_mean_bn, dot_mean_in, dot_mean_bn, dot_mean_in, dot_mean_ln])
        gv = np.array([dot_cov_bn + dot_diag_bn, dot_cov_in + dot_diag_in, 0.0, 0.0, dot_ln])
    if sw_var_weight is None:
        gm, gv = gm + gv, None
    g_mw = mw * (gm - (mw * gm).sum())
    g_vw = None if gv is None else vw * (gv - (vw * gv).sum())

    if stages is not None:
        stages.update(mean_in=mean_in, cov_in=cov_in, a_fwd=a_fwd, g_mean_bn=g_mean_bn.copy(), g_cov_bn=g_cov_bn.copy())
    if training:
        reduce_(g_mean_bn)
        reduce_(g_cov_bn)
        s_bn = (g_cov_bn + np.swapaxes(g_cov_bn, -1, -2)) / (n * hw * world_size)
        m_bn = g_mean_bn / (n * hw * world_size)
    elif all_reduce is not None:
        # SyncMeanCov.backward does not look at ``training`` for the data gradient (sync_switchwhiten.py:48-55): in
        # eval mode the synchronised layer still back-propagates through the running statistics as if they were
        # this rank's batch statistics (no exchange, world_size 1).  The plain layer's running buffers get nothing.
        s_bn = (g_cov_bn + np.swapaxes(g_cov_bn, -1, -2)) / (n * hw)
        m_bn = g_mean_bn / (n * hw)
    else:
        s_bn, m_bn = np.zeros((g, c, c)), np.zeros((g, c))

    # --- backward affine pass: gx = M1 gy + M2 x + cst -----------------------------------------------------------
    s_in = (g_cov_in + np.swapaxes(g_cov_in, -1, -2)) / hw
    m1 = np.swapaxes(a_fwd, -1, -2)
    m2 = s_in + s_bn[None]
    cst = g_mean_in / hw + m_bn[None] - np.einsum("ngij,ngj->ngi", s_in, mean_in) - \
        np.einsum("gij,gj->gi", s_bn, mean_bn)[None]
    gx = np.einsum("ngij,ngjp->ngip", m1, gyg) + np.einsum("ngij,ngjp->ngip", m2, xg) + cst[..., None]

    grads = {"x": gx.reshape(x.shape), "sw_mean_weight": g_mw, "sw_var_weight": g_vw,
             "weight": None if weight is None else g_weight, "bias": None if bias is None else g_bias}
    return y.reshape(x.shape), grads, (mean_bn, cov_bn)
