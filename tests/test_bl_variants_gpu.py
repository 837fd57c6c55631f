"""Every instantiation of the Bayesian-loss kernels against the CPU oracle.

bl_z, bl_counts, bl_grad and the posterior kernel are templates over the pixel tile of a thread (8x2, 8x1, 4x1 or 2x1
pixels; the host picks one from the number of warp tasks) and over POW2 (a power-of-two 2*sigma^2 scales exactly, any
other takes the Markstein-corrected division).  Here every (tile, POW2, culling) combination runs on a ragged grid --
190 x 250 cells: 190 is no multiple of 4 or 8, 250 none of 32 or 64, so every tile has a partial last row band and
column block -- and each case asserts the tile it was built to reach.

Besides the usual rtol 1e-5 gates, the per-pixel softmax max (workspace region ``amax``) is compared EXACTLY with an
fp32 restatement of bl.py:38-43 (DESIGN section 3: the softmax arguments are the reference's fp32 sequence bit for bit).
It depends only on the distance expansion, the minimum over the points, an IEEE square root and one division, so a
1-ulp error or a minimum taken from the wrong point shows up there even where it hides under rtol 1e-5.
"""
import functools
import math

import numpy as np
import pytest
import torch

from dgvcc_b200 import synthetic
from oracle import bl_oracle
from helpers import assert_close
from test_bl_gpu import RTOL, _region, check_against, run_cuda
from test_bl_sharded_gpu import _band_table_on_one_gpu, run_banded, run_sharded, single_gpu_with_table

pytestmark = pytest.mark.gpu

HP, WP = 190, 250
CHUNK = 64
TILES = ["8x2", "8x1", "4x1", "2x1"]
# Point counts per tile.  With 64-point chunks the number of chunks alone selects the tile on this grid (pick_variant:
# the first tile with at least 148 * 16 warp tasks; one chunk is 96 tasks of 8x2, 192 of 8x1, 384 of 4x1): 26, 17, 9
# and 6 chunks.  An image with one chunk and an image without points ride along.  At most ~7e7 (point, pixel) pairs.
TILE_COUNTS = {"8x2": [1530, 7, 0], "8x1": [900, 7, 0], "4x1": [440, 7, 0], "2x1": [200, 7, 0]}
SIGMAS = [(8.0, 1.0),    # 2 sigma^2 = 128: the power-of-two path
          (7.3, 0.15),   # 2 sigma^2 = 106.58 is no fp32 number: the general division, background ring far inside
          (1.5, 1.0)]    # 2 sigma^2 = 4.5: almost every exponential underflows, culling skips almost every point


def _pow2(sigma):
    """The kernels' POW2 template argument: is fl32(2 sigma^2) a power of two (make_scale, is_pow2)?"""
    return math.frexp(float(np.float32(2.0 * sigma ** 2)))[0] == 0.5


def _tile_of(layout):
    return f"{layout.rows_per_thread}x{layout.cols_per_thread}"


def _case_id(tile, sigma, bg_ratio, use_bg, stride):
    return f"{tile}-sigma{sigma:g}-{'pow2' if _pow2(sigma) else 'general'}-{'bg' if use_bg else 'nobg'}-stride{stride}"


@functools.lru_cache(maxsize=None)
def _tile_batch(tile, stride):
    pts, tgt, dens, st = synthetic.bl_batch(70 + TILES.index(tile), TILE_COUNTS[tile], WP * stride, HP * stride, stride)
    return ([torch.from_numpy(p) for p in pts], torch.from_numpy(st), [torch.from_numpy(t) for t in tgt],
            torch.from_numpy(dens))


def _band_dis(points, hp, wp, stride, band=16):
    """bl_oracle.sq_distances, one band of grid rows at a time: (r0, r1, dis [N, (r1 - r0) * wp])."""
    p = points.to(torch.float32)
    x_dis = bl_oracle.axis_sqdist(p[:, 0:1], bl_oracle.grid_coords(wp, stride))
    y_dis = bl_oracle.axis_sqdist(p[:, 1:2], bl_oracle.grid_coords(hp, stride))
    for r0 in range(0, hp, band):
        r1 = min(hp, r0 + band)
        yield r0, r1, (y_dis[:, r0:r1].unsqueeze(2) + x_dis.unsqueeze(1)).reshape(len(p), -1)


def softmax_max(points, st_size, hp, wp, stride, sigma, bg_ratio, use_bg):
    """[hp, wp]: the largest softmax argument of every pixel, bl.py:38-43 in fp32 up to the softmax (the squared
    distances, the background row from the clamped minimum, -dis / (2 sigma^2)), then the max over the rows.
    0 for an image without points (its only row is the sum of the density; the kernels store 0).  The root is the
    IEEE one of the reference's CUDA run (bl_oracle.ieee_sqrt)."""
    amax = torch.zeros((hp, wp), dtype=torch.float32)
    if len(points) == 0:
        return amax
    st = torch.as_tensor(st_size, dtype=torch.float32)
    for r0, r1, dis in _band_dis(points, hp, wp, stride):
        if use_bg:
            min_dis = torch.clamp(torch.min(dis, dim=0, keepdim=True)[0], min=0.0)
            dis = torch.cat([dis, (st * bg_ratio - bl_oracle.ieee_sqrt(min_dis)) ** 2], 0)
        amax[r0:r1] = torch.max(-dis / (2.0 * sigma ** 2), dim=0)[0].reshape(r1 - r0, wp)
    return amax


def assert_amax_exact(got, ref, what):
    # values, not bits: a distance of exactly 0 gives -0 in the reference and +0 from the general-sigma division
    bad = got != ref
    if bad.any():
        idx = tuple(torch.nonzero(bad)[0].tolist())
        g, r = float(got[idx]), float(ref[idx])
        ulps = abs(int(np.float32(g).view(np.int32)) - int(np.float32(r).view(np.int32)))
        raise AssertionError(f"{what}: softmax max differs in {int(bad.sum())}/{bad.numel()} pixels; first at {idx}: "
                             f"got {g!r} ref {r!r} ({ulps} ulp)")


def _amax(keep, dens):
    b, _, hp, wp = dens.shape
    return _region(keep, "amax", b * hp * wp).view(b, hp, wp).cpu()


def check_amax(keep, points, st, dens, stride, sigma, bg_ratio, use_bg, what=""):
    got = _amax(keep, dens)
    for i, p in enumerate(points):
        ref = softmax_max(p, st[i], dens.shape[2], dens.shape[3], stride, sigma, bg_ratio, use_bg)
        assert_amax_exact(got[i], ref, f"{what} image {i} ({len(p)} points)")
    return got


# ------------------------------------------------------------------------------ tile x sigma x culling, one GPU
MATRIX = ([(tile, s, b, True, 8) for tile in TILES for s, b in SIGMAS] +
          [(tile, 7.3, 0.15, False, 8) for tile in TILES] +        # no background row
          [("8x2", 8.0, 1.0, True, 16), ("8x2", 7.3, 0.15, True, 4)])  # other strides: other cell centres


@functools.lru_cache(maxsize=None)
def _matrix_oracle(tile, sigma, bg_ratio, use_bg, stride):
    pts, st, tgt, dens = _tile_batch(tile, stride)
    loss, grad, counts = bl_oracle.bl_forward_backward_chunked(pts, st, tgt, dens, stride, sigma, bg_ratio, use_bg,
                                                               chunk_rows=16, sqrt=bl_oracle.ieee_sqrt)
    return loss, grad, dict(enumerate(counts))


@pytest.mark.parametrize("cull", [False, True], ids=["dense", "culled"])
@pytest.mark.parametrize("tile,sigma,bg_ratio,use_bg,stride", MATRIX, ids=[_case_id(*c) for c in MATRIX])
def test_every_tile_and_sigma_path_against_oracle(tile, sigma, bg_ratio, use_bg, stride, cull, monkeypatch):
    monkeypatch.setattr("dgvcc_b200.losses.bl._CHUNK_POINTS", CHUNK)
    pts, st, tgt, dens = _tile_batch(tile, stride)
    keep = {}
    got = run_cuda(pts, st, tgt, dens, stride, sigma, bg_ratio, use_bg, exact_cull=cull, keep=keep)
    assert _tile_of(keep["layout"]) == tile, "the batch no longer selects the tile this case was built for"
    check_against(*got, *_matrix_oracle(tile, sigma, bg_ratio, use_bg, stride))
    amax = check_amax(keep, pts, st, dens, stride, sigma, bg_ratio, use_bg, "amax")
    if cull:   # culling skips exact zeros only: not a bit may change
        keep_d = {}
        dense = run_cuda(pts, st, tgt, dens, stride, sigma, bg_ratio, use_bg, exact_cull=False, keep=keep_d)
        assert torch.equal(got[0], dense[0]), "loss"
        assert torch.equal(got[1], dense[1]), f"gradient differs in {int((got[1] != dense[1]).sum())} pixels"
        assert all(torch.equal(a, b) for a, b in zip(got[2], dense[2])), "expected counts"
        assert torch.equal(amax, _amax(keep_d, dens)), "softmax max"


# ------------------------------------------------------------------------------ posteriors per tile and POW2
def _posterior_reference(points, st_size, hp, wp, stride, sigma, bg_ratio, use_bg, rows):
    """Rows ``rows`` and the column sums of bl_oracle.posterior, one band of grid rows at a time."""
    st = torch.as_tensor(st_size, dtype=torch.float32)
    sel = torch.empty((len(rows), hp * wp), dtype=torch.float32)
    colsum = torch.empty((hp * wp,), dtype=torch.float32)
    for r0, r1, dis in _band_dis(points, hp, wp, stride):
        prob = bl_oracle.posterior_from_dis(dis, st, sigma, bg_ratio, use_bg, sqrt=bl_oracle.ieee_sqrt)
        sel[:, r0 * wp:r1 * wp] = prob[rows]
        colsum[r0 * wp:r1 * wp] = prob.sum(0)
    return sel, colsum


@pytest.mark.parametrize("tile,sigma,bg_ratio", [(t, s, b) for t in TILES for s, b in SIGMAS],
                         ids=[f"{t}-sigma{s:g}-{'pow2' if _pow2(s) else 'general'}" for t in TILES for s, _ in SIGMAS])
def test_posteriors_of_every_tile_against_oracle(tile, sigma, bg_ratio, monkeypatch):
    from dgvcc_b200.losses.bl import Post_Prob, _layout, build_meta
    monkeypatch.setattr("dgvcc_b200.losses.bl._CHUNK_POINTS", CHUNK)
    pts, st, _, _ = _tile_batch(tile, 8)
    counts = np.asarray([len(p) for p in pts])
    rows = np.where(counts == 0, 1, counts + 1)
    _, total_chunks, _ = build_meta(counts, rows, CHUNK)
    assert _tile_of(_layout(int(rows.sum()), total_chunks, len(pts), HP, WP)) == tile   # what dgvcc_bl_posterior plans
    dev = torch.device("cuda:0")
    probs = Post_Prob(sigma, max(HP, WP) * 8, 8, bg_ratio, True, dev)([p.to(dev) for p in pts], st.to(dev), grid=(HP, WP))
    for i, p in enumerate(probs):
        n = len(pts[i])
        if n == 0:
            assert p is None
            continue
        sel = sorted({0, 1, n // 2, n - 1, n})   # first, second, middle and last point, background
        ref_rows, ref_colsum = _posterior_reference(pts[i], st[i], HP, WP, 8, sigma, bg_ratio, True, sel)
        assert_close(p[sel].cpu(), ref_rows, RTOL, 1e-30, f"posterior rows {sel} image {i}")
        assert_close(p.sum(0).cpu(), ref_colsum, RTOL, 0, f"posterior column sums image {i}")


# ------------------------------------------------------------------------------ minima and the point grid
@pytest.fixture
def min_cell():
    """Sets DGVCC_BL_OPT_MIN_CELL (process-global, read when a plan is made); the default 64 comes back afterwards."""
    from dgvcc_b200 import _native

    def set_cell(value):
        _native.check(_native.lib().dgvcc_bl_set_option(_native.BL_OPT_MIN_CELL, int(value)), "dgvcc_bl_set_option")
    try:
        yield set_cell
    finally:
        set_cell(64)


def _min_cell_case(name):
    if name == "config3":   # 16 images, 192 x 256 grid: the workload bench.py times
        w, h = synthetic.CONFIG_SHAPES[3]
        pts, tgt, dens, st = synthetic.bl_batch(3, synthetic.config_counts(3), w, h, 8)
        sigma, bg_ratio = 8.0, 1.0
    else:                   # one 2048 x 2048 px image: cells of 8 or 16 px are more than GRID_MAX_CELLS, the cell grows
        pts, tgt, dens, st = synthetic.bl_batch(77, [4000], 2048, 2048, 8)
        sigma, bg_ratio = 7.3, 0.15
    return ([torch.from_numpy(p) for p in pts], torch.from_numpy(st), [torch.from_numpy(t) for t in tgt],
            torch.from_numpy(dens), 8, sigma, bg_ratio, True)


@pytest.mark.parametrize("cell", [8, 16, 256, 4096])
@pytest.mark.parametrize("case", ["config3", "image2048"])
def test_minima_do_not_depend_on_the_point_grid(case, cell, min_cell):
    """A minimum is exact in any order of the points, so the cell size of the grid the minima walk cannot change a bit
    of loss, gradient or softmax max (4096 px: one cell holds every point)."""
    args = _min_cell_case(case)

    def run(cull):
        keep = {}
        loss, grad, counts = run_cuda(*args, exact_cull=cull, keep=keep)
        return loss, grad, _amax(keep, args[3])

    for cull in (False, True):
        min_cell(64)
        ref = run(cull)
        min_cell(cell)
        got = run(cull)
        assert torch.equal(got[0], ref[0]), f"loss with {cell} px cells"
        assert torch.equal(got[1], ref[1]), f"gradient with {cell} px cells: {int((got[1] != ref[1]).sum())} pixels"
        assert torch.equal(got[2], ref[2]), f"softmax max with {cell} px cells: {int((got[2] != ref[2]).sum())} pixels"


# ------------------------------------------------------------------------------ heads far outside the grid
def _far_batch():
    """45 x 61 grid (360 x 488 px, extent e = 488 px).  Images whose heads all sit 1, 4, 10 and 100 extents outside,
    on every side; one whose heads sit about 1e5 px away; an ordinary crowd; an image without points."""
    hp, wp, stride = 45, 61, 8
    h, w = hp * stride, wp * stride
    e = max(h, w)
    rng = np.random.default_rng(4242)
    pts = []
    for k in (1, 4, 10, 100):
        m = 6   # heads per side
        d = k * e * (1.0 + rng.uniform(0.0, 0.05, size=(4, m)))
        xs, ys = rng.uniform(0, w, size=(2, m)), rng.uniform(0, h, size=(2, m))
        pts.append(np.concatenate([np.stack([-d[0], ys[0]], 1), np.stack([w + d[1], ys[1]], 1),
                                   np.stack([xs[0], -d[2]], 1), np.stack([xs[1], h + d[3]], 1)]))
    ang = rng.uniform(0, 2 * np.pi, size=24)
    r = 1e5 * (1.0 + rng.uniform(0.0, 0.01, size=24))
    pts.append(np.stack([w / 2 + r * np.cos(ang), h / 2 + r * np.sin(ang)], 1))
    pts.append(synthetic.crowd_points(rng, 300, w, h))
    pts.append(np.zeros((0, 2)))
    pts = [torch.from_numpy(np.asarray(p, dtype=np.float32)) for p in pts]
    tgt = [torch.from_numpy(rng.uniform(0.3, 1.0, size=len(p)).astype(np.float32)) for p in pts]
    dens = torch.from_numpy((np.abs(rng.normal(size=(len(pts), 1, hp, wp))) * 0.01).astype(np.float32))
    st = torch.full((len(pts),), float(min(h, w)))
    return pts, st, tgt, dens, stride


@pytest.mark.parametrize("use_bg", [True, False], ids=["bg", "nobg"])
@pytest.mark.parametrize("sigma,bg_ratio", [(8.0, 1.0), (7.3, 0.15)], ids=["pow2", "general"])
def test_heads_far_outside_the_grid(sigma, bg_ratio, use_bg, monkeypatch):
    monkeypatch.setattr("dgvcc_b200.losses.bl._CHUNK_POINTS", 8)   # several chunks per image
    pts, st, tgt, dens, stride = _far_batch()
    ref = bl_oracle.bl_forward_backward(pts, st, tgt, dens, stride, sigma, bg_ratio, use_bg, sqrt=bl_oracle.ieee_sqrt)
    results = []
    for cull in (False, True):
        keep = {}
        got = run_cuda(pts, st, tgt, dens, stride, sigma, bg_ratio, use_bg, exact_cull=cull, keep=keep)
        for name, t in (("loss", got[0]), ("gradient", got[1]), ("counts", torch.cat(got[2]))):
            assert torch.isfinite(t).all(), f"{name} not finite (exact_cull={cull})"
        check_against(*got, ref[0], ref[1], dict(enumerate(ref[2])))
        amax = check_amax(keep, pts, st, dens, stride, sigma, bg_ratio, use_bg, f"amax (exact_cull={cull})")
        assert torch.isfinite(amax).all()
        results.append(got + (amax,))
    dense, culled = results
    assert torch.equal(dense[0], culled[0]) and torch.equal(dense[1], culled[1]) and torch.equal(dense[3], culled[3])


# ------------------------------------------------------------------------------ sharded splits, general sigma
SHARD_COUNTS = [600, 7, 0, 250]
SHARD_SIGMA, SHARD_BG = 7.3, 0.15


@pytest.fixture
def band_tile():
    """Forces the pixel tile of the sharded layouts (DGVCC_BL_OPT_BAND_TILE: rows * 10 + cols), 0 (by task count)
    afterwards.  The option is process-global and read by the C layout; the plans cached on the Python side hold the
    layout of the tile that was in force when they were made, so both caches are emptied with every change."""
    from dgvcc_b200 import _native
    from dgvcc_b200.losses import bl_banded, bl_sharded

    def set_tile(value):
        _native.check(_native.lib().dgvcc_bl_set_option(_native.BL_OPT_BAND_TILE, int(value)), "dgvcc_bl_set_option")
        bl_sharded._plan_cache.clear()
        bl_banded._plan_cache.clear()
    try:
        yield set_tile
    finally:
        set_tile(0)


@functools.lru_cache(maxsize=None)
def _shard_batch():
    pts, tgt, dens, st = synthetic.bl_batch(79, SHARD_COUNTS, WP * 8, HP * 8, 8)
    pts, tgt = [torch.from_numpy(p) for p in pts], [torch.from_numpy(t) for t in tgt]
    st, dens = torch.from_numpy(st), torch.from_numpy(dens)
    oracle = bl_oracle.bl_forward_backward_chunked(pts, st, tgt, dens, 8, SHARD_SIGMA, SHARD_BG, True, chunk_rows=16,
                                                    sqrt=bl_oracle.ieee_sqrt)
    return pts, tgt, st, dens, oracle


@pytest.mark.parametrize("tile", TILES)
@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("split", ["chunks", "bands"])
def test_sharded_splits_with_general_sigma_on_every_tile(split, world, tile, band_tile, monkeypatch):
    """Point chunks: loss and gradient bit-identical to one GPU running the same chunk table.  Row bands: the same loss
    bits on every rank, gradient bit-identical to one GPU.  Both within rtol 1e-5 of the oracle.

    One GPU picks its own tile (the option only applies to the sharded layouts), and the expected counts are summed over
    pixels per CTA of pixel tiles, so the loss bits of the point-chunk split equal one GPU's only where both run the
    same tile; elsewhere every rank still returns the same bits, within 1e-6 of one GPU.  The gradient is per pixel and
    does not depend on the tile."""
    from dgvcc_b200.losses.bl import _layout
    monkeypatch.setattr("dgvcc_b200.losses.bl._CHUNK_POINTS", CHUNK)
    band_tile(int(tile.replace("x", "")))
    pts, tgt, st, dens, (o_loss, o_grad, _) = _shard_batch()
    owners = [(3 * i + 1) % world for i in range(len(pts))]
    args = (pts, tgt, st, dens, 8, SHARD_SIGMA, SHARD_BG, True)
    for cull in (False, True):
        if split == "chunks":
            losses, grad, plan = run_sharded(world, *args, cull, owners, steps=2, defer=cull)
            ref_loss, ref_grad = single_gpu_with_table(plan, *args, cull)
            assert all(torch.equal(l, losses[0]) for l in losses), [float(l) for l in losses]
            if _tile_of(_layout(plan.total_rows, plan.total_chunks, plan.batch, HP, WP)) == tile:
                assert torch.equal(losses[0], ref_loss), f"loss {float(losses[0])!r} vs {float(ref_loss)!r} on one GPU"
            assert_close(losses[0], ref_loss, 1e-6, 0, "sharded loss vs one GPU")
        else:
            losses, grad, plan = run_banded(world, *args, cull, owners, steps=2, chunk=CHUNK)
            assert all(torch.equal(l, losses[0]) for l in losses), [float(l) for l in losses]
            ref_loss, ref_grad = _band_table_on_one_gpu(plan, *args, cull)
            assert_close(losses[0], ref_loss, 1e-6, 0, "banded loss vs one GPU")
        assert _tile_of(plan.layout) == tile
        assert torch.equal(grad, ref_grad), f"gradient differs in {int((grad != ref_grad).sum())} pixels"
        assert_close(losses[0], o_loss, RTOL, 0, f"{split} loss vs oracle")
        assert_close(grad, o_grad, RTOL, 2e-7 * float(o_grad.abs().max()), f"{split} gradient vs oracle")
