"""The FMA-pipe exponential of the Bayesian-loss sweeps (ex2_fma, csrc/common.cuh).

The sweeps take the exponentials of the pixels on global grid rows 6, 7 (mod 8) in odd 32-column blocks from a
polynomial on the FMA pipe instead of MUFU.EX2.  That is only invisible to the loss if ex2_fma is at least as accurate
as ex2.approx.ftz.f32, returns +0 for exactly the arguments MUFU flushes (exact_cull skips points by that zero set) and
propagates NaN and infinities the same way -- checked here over every fp32 argument the loss can produce -- and if the
rule picks the same pixels whatever the pixel tile, so that Z, the counts and the gradient see the same bits for a pair
on every layout.
"""
import math

import numpy as np
import pytest
import torch

from dgvcc_b200 import synthetic
from test_bl_gpu import _region, run_cuda

pytestmark = pytest.mark.gpu

CHUNK = 1 << 26


def _ex2_both(t):
    """(MUFU.EX2, ex2_fma) of a float32 CUDA tensor."""
    from dgvcc_b200 import _native
    mufu, fma = torch.empty_like(t), torch.empty_like(t)
    _native.check(_native.lib().dgvcc_probe_ex2_fma(_native.ptr(t), t.numel(), _native.ptr(mufu), _native.ptr(fma),
                                                    _native.stream_ptr(t.device)), "dgvcc_probe_ex2_fma")
    return mufu, fma


def _bits(x):
    return int(np.float32(x).view(np.int32))


def test_ex2_fma_on_every_fp32_argument_against_mufu_and_fp64():
    """Every fp32 t in [-130, 2^-8] (the loss's exponents are <= 2^-8): the largest relative error against fp64 exp2
    over t >= -126 is no larger than MUFU's, the zero sets are identical (+0 exactly for t < -126), and each lane of
    the packed evaluation gives the same bits whatever its neighbour."""
    dev = torch.device("cuda:0")
    worst = {"mufu": 0.0, "fma": 0.0}
    # int32 views: -0 .. -130 are the bit patterns 0x80000000 .. 0xC3020000, +0 .. 2^-8 are 0 .. 0x3B800000
    for lo, hi in ((-(1 << 31), _bits(-130.0)), (0, _bits(2.0 ** -8))):
        for a in range(lo, hi + 1, CHUNK):
            t = torch.arange(a, min(a + CHUNK, hi + 1), dtype=torch.int32, device=dev).view(torch.float32)
            mufu, fma = _ex2_both(t)
            zero_m, zero_f = mufu == 0, fma == 0
            assert torch.equal(zero_m, zero_f), f"zero sets differ at t = {t[zero_m != zero_f][:4].tolist()}"
            assert torch.equal(zero_f, t < -126), "ex2_fma is +0 exactly below -126"
            assert bool((fma[zero_f].view(torch.int32) == 0).all()), "zeros are +0"
            normal = t >= -126
            ref = torch.exp2(t[normal].double())
            for name, v in (("mufu", mufu), ("fma", fma)):
                worst[name] = max(worst[name], float(((v[normal].double() - ref).abs() / ref).max()))
            _, shifted = _ex2_both(t[1:].contiguous())   # every value now shares its pair with the other neighbour
            assert torch.equal(shifted.view(torch.int32), fma[1:].view(torch.int32)), "lanes are independent"
    print(f"max relative error over t in [-126, 2^-8]: MUFU.EX2 {worst['mufu']:.3e}, ex2_fma {worst['fma']:.3e}")
    assert worst["fma"] <= worst["mufu"], worst
    assert worst["fma"] < 1e-7, worst


def test_ex2_fma_special_values():
    dev = torch.device("cuda:0")
    t = torch.tensor([math.nan, -math.nan, math.inf, -math.inf, -0.0, 0.0, -126.0, -126.5, -127.0, -1e30, -1.0, 5.0],
                     dtype=torch.float32, device=dev)
    mufu, fma = _ex2_both(t)
    mufu, fma = mufu.cpu(), fma.cpu()
    assert torch.isnan(fma[:2]).all() and torch.isnan(mufu[:2]).all()
    assert torch.equal(fma[2:].view(torch.int32), mufu[2:].view(torch.int32)), (fma[2:].tolist(), mufu[2:].tolist())
    assert fma[2] == math.inf and fma[3].view(torch.int32) == 0 and fma[4] == 1.0 and fma[5] == 1.0
    assert fma[6] == 2.0 ** -126 and fma[7] == 0 and fma[8] == 0 and fma[10] == 0.5 and fma[11] == 32.0


# One GPU picks the pixel tile from the number of warp tasks: on a 190 x 250 grid with 64-point chunks, 26, 17, 9 and 6
# chunks select 8x2, 8x1, 4x1 and 2x1.  Image 0 (4 chunks) and the first two single-chunk images are the same in every
# batch; the further single-chunk images only move the tile.
HP, WP, STRIDE = 190, 250, 8
TILE_CHUNKS = {"8x2": 26, "8x1": 17, "4x1": 9, "2x1": 6}


@pytest.mark.parametrize("sigma,bg_ratio", [(8.0, 1.0), (7.3, 0.15)], ids=["pow2", "general"])
def test_denominators_are_bit_identical_on_every_pixel_tile(sigma, bg_ratio, monkeypatch):
    """1/Z (workspace region rz) of the images every batch shares, on all four pixel tiles, bit for bit: Z sums the
    exponentials of a multi-chunk image in chunk order, so a tile-dependent choice of MUFU or ex2_fma would show here."""
    monkeypatch.setattr("dgvcc_b200.losses.bl._CHUNK_POINTS", 64)
    n_img = max(TILE_CHUNKS.values()) - 3
    pts, tgt, dens, st = synthetic.bl_batch(91, [200] + [7] * (n_img - 1), WP * STRIDE, HP * STRIDE, STRIDE)
    pts, tgt = [torch.from_numpy(p) for p in pts], [torch.from_numpy(t) for t in tgt]
    dens, st = torch.from_numpy(dens), torch.from_numpy(st)
    shared = min(TILE_CHUNKS.values()) - 3
    rz = {}
    for tile, chunks in TILE_CHUNKS.items():
        b = chunks - 3   # image 0 has four chunks
        keep = {}
        run_cuda(pts[:b], st[:b], tgt[:b], dens[:b], STRIDE, sigma, bg_ratio, True, keep=keep)
        lay = keep["layout"]
        assert f"{lay.rows_per_thread}x{lay.cols_per_thread}" == tile, "the batch no longer selects this tile"
        rz[tile] = _region(keep, "rz", b * HP * WP).view(b, HP, WP)[:shared].cpu()
    assert bool(torch.isfinite(rz["8x2"]).all())
    for tile in TILE_CHUNKS:
        diff = rz[tile].view(torch.int32) != rz["8x2"].view(torch.int32)
        assert not diff.any(), f"{tile}: 1/Z differs from 8x2 in {int(diff.sum())} pixels, rows {diff.nonzero()[:4, 1].tolist()}"
