"""CPU oracle for the Bayesian loss -- TEST INFRASTRUCTURE, not product code.

Restates /root/reference/losses/bl.py on the CPU with torch-CPU ops in the
reference's own rounding order, extended in two per-pixel-exact ways the
reference cannot do itself (SURVEY.md section 8c):

* rectangular grids: the reference shares one ``cood`` vector between x and y
  (bl.py:14-16), i.e. it is square-only.  Every operation in ``Post_Prob`` is
  independent per pixel, so using two coordinate vectors gives exactly the
  slice ``prob.view(N+1, c/s, c/s)[:, :H', :W']`` of the square reference.
* one image at a time / pixel chunks: the loss is a mean of per-image terms
  (bl.py:62-79), so images never need the batch concat of bl.py:21-32.

Parity pin: ``tests/golden/bl_*.npz`` were produced by the UNMODIFIED reference
module (``tests/golden/make_golden.py``); ``tests/test_oracle_bl.py`` checks
this file against them.
"""
from math import ceil

import torch


def grid_coords(n_cells, stride, dtype=torch.float32):
    """Pixel-centre coordinates, image pixels.  bl.py:14-16."""
    return (torch.arange(0, n_cells * stride, step=stride, dtype=dtype) + stride / 2).unsqueeze(0)


def axis_sqdist(p, cood):
    """[N,1] x [1,G] -> [N,G]: -2*p*c + p*p + c*c, rounded step by step.  bl.py:27-28."""
    return -2 * torch.matmul(p, cood) + p * p + cood * cood


def sq_distances(points, hp, wp, stride, dtype=torch.float32):
    """dis[n, r*W'+c] = ydis[n,r] + xdis[n,c]  (row index = y).  bl.py:25-32."""
    pts = points.to(dtype)
    x = pts[:, 0:1]
    y = pts[:, 1:2]
    x_dis = axis_sqdist(x, grid_coords(wp, stride, dtype))
    y_dis = axis_sqdist(y, grid_coords(hp, stride, dtype))
    dis = y_dis.unsqueeze(2) + x_dis.unsqueeze(1)
    return dis.reshape(dis.size(0), -1)


def ieee_sqrt(t):
    """Correctly rounded square root: torch.sqrt on CUDA, where the reference trains, and the kernels' __fsqrt_rn.
    torch's CPU sqrt of a long fp32 tensor (the MKL vector path) is one ulp off in about 0.7 % of the elements -- the
    fixtures under tests/golden hold those roots -- and one ulp of the root moves a pixel's background argument
    (bl.py:41) by up to ~10 ulp.  The fp64 root rounded once to fp32 is the IEEE fp32 root."""
    if t.dtype == torch.float32:
        return torch.sqrt(t.double()).to(torch.float32)
    return torch.sqrt(t)


def posterior_from_dis(dis, st_size, sigma, bg_ratio, use_bg, sqrt=torch.sqrt):
    """Softmax over points (+ background row appended last).  bl.py:38-44.  ``sqrt``: ``ieee_sqrt`` for the roots of
    the reference's CUDA run (the default, torch's CPU sqrt, reproduces its CPU run and the fixtures)."""
    if use_bg:
        min_dis = torch.clamp(torch.min(dis, dim=0, keepdim=True)[0], min=0.0)
        d = st_size * bg_ratio
        bg_dis = (d - sqrt(min_dis)) ** 2
        dis = torch.cat([dis, bg_dis], 0)
    dis = -dis / (2.0 * sigma ** 2)
    return torch.softmax(dis, dim=0)


def posterior(points, st_size, hp, wp, stride, sigma, bg_ratio=1.0, use_bg=True,
              dtype=torch.float32, sqrt=torch.sqrt):
    """Posterior matrix of ONE image, [N(+1), H'*W'], or None when it has no points."""
    if len(points) == 0:
        return None
    st = torch.as_tensor(st_size, dtype=dtype)
    return posterior_from_dis(sq_distances(points, hp, wp, stride, dtype), st, sigma, bg_ratio, use_bg, sqrt)


def trimmed_l1(residual):
    """Sum of the ceil(0.9*(L-1)) smallest of residual[:-1] plus residual[-1].  bl.py:75-78."""
    num = ceil(0.9 * (len(residual) - 1))
    return torch.sum(torch.topk(residual[:-1], num, largest=False)[0]) + residual[-1]


def image_target(targets, n_rows, use_bg, dtype=torch.float32):
    """Per-row targets: the image's targets, then 0 for the background row.  bl.py:67-72."""
    if use_bg:
        t = torch.zeros((n_rows,), dtype=dtype)
        t[:-1] = targets.to(dtype)
        return t
    return targets.to(dtype)


def bl_forward_backward(points, st_sizes, targets, density, stride, sigma,
                        bg_ratio=1.0, use_bg=True, dtype=torch.float32, sqrt=torch.sqrt):
    """Materialising oracle: loss, d loss / d density, per-image expected counts.

    ``density`` is [B,1,H',W'].  Uses autograd exactly like the reference
    (only ``density`` receives gradient, bl.py:73-79).
    """
    B, _, hp, wp = density.shape
    dens = density.detach().to(dtype).clone().requires_grad_(True)
    loss = 0
    counts = []
    for i in range(B):
        prob = posterior(points[i], st_sizes[i], hp, wp, stride, sigma, bg_ratio, use_bg, dtype, sqrt)
        if prob is None:
            pre_count = torch.sum(dens[i]).reshape(1)
            target = torch.zeros((1,), dtype=dtype)
        else:
            target = image_target(targets[i], len(prob), use_bg, dtype)
            pre_count = torch.sum(dens[i].view((1, -1)) * prob, dim=1)
        counts.append(pre_count.detach().clone())
        loss = loss + trimmed_l1(torch.abs(target - pre_count))
    loss = loss / B
    loss.backward()
    return loss.detach(), dens.grad.detach(), counts


def bl_forward_backward_chunked(points, st_sizes, targets, density, stride, sigma,
                                bg_ratio=1.0, use_bg=True, dtype=torch.float32,
                                chunk_rows=16, sqrt=torch.sqrt):
    """Same numbers without holding [N+1, M]: row bands of the grid, explicit gradient.

    Per-pixel independence of the posterior makes band-wise evaluation exact;
    only the summation order of the counts over pixels differs from the
    materialising path (fp32 re-association, ~1e-7 relative).
    Gradient: dL/dD[m] = (1/B) * sum_{n kept} sign(c_n - t_n) * p[n,m]   (bl.py:73-79).
    """
    B, _, hp, wp = density.shape
    dens = density.detach().to(dtype)
    grad = torch.zeros_like(dens)
    loss = torch.zeros((), dtype=dtype)
    counts = []
    for i in range(B):
        pts = points[i]
        if len(pts) == 0:
            s = torch.sum(dens[i])
            counts.append(s.reshape(1).clone())
            loss = loss + torch.abs(s)
            grad[i] = torch.sign(s) / B
            continue
        st = torch.as_tensor(st_sizes[i], dtype=dtype)
        p = pts.to(dtype)
        x_dis = axis_sqdist(p[:, 0:1], grid_coords(wp, stride, dtype))
        y_dis = axis_sqdist(p[:, 1:2], grid_coords(hp, stride, dtype))
        n_rows = len(pts) + (1 if use_bg else 0)
        c = torch.zeros((n_rows,), dtype=dtype)

        def band_prob(r0, r1):
            dis = (y_dis[:, r0:r1].unsqueeze(2) + x_dis.unsqueeze(1)).reshape(len(pts), -1)
            return posterior_from_dis(dis, st, sigma, bg_ratio, use_bg, sqrt)

        for r0 in range(0, hp, chunk_rows):
            r1 = min(hp, r0 + chunk_rows)
            prob = band_prob(r0, r1)
            c += torch.sum(dens[i, 0, r0:r1].reshape(1, -1) * prob, dim=1)
        counts.append(c.clone())
        target = image_target(targets[i], n_rows, use_bg, dtype)
        res = torch.abs(target - c)
        num = ceil(0.9 * (n_rows - 1))
        kept = torch.topk(res[:-1], num, largest=False)
        loss = loss + torch.sum(kept[0]) + res[-1]
        w = torch.zeros((n_rows,), dtype=dtype)
        sgn = torch.sign(c - target)
        w[kept[1]] = sgn[kept[1]]
        w[-1] = sgn[-1]
        w = w / B
        for r0 in range(0, hp, chunk_rows):
            r1 = min(hp, r0 + chunk_rows)
            prob = band_prob(r0, r1)
            grad[i, 0, r0:r1] = torch.sum(w.unsqueeze(1) * prob, dim=0).reshape(r1 - r0, wp)
    return loss / B, grad, counts
