"""Every dispatch arm of the auxiliary Gram losses (lw_loss, ortho_loss) against an fp64 evaluation of the oracle.

Both losses run the kernels of the ISW path: the tensor-core Gram (csrc/isw_gram_tc.cu; the SIMT Gram where it refuses
the shape), the general 3xTF32 dX = S X GEMM (csrc/isw_sx_tc.cu; the SIMT GEMM where it refuses), and their own
standardisation, S-matrix and triu-square kernels (csrc/isw_kernels.cu).  Each shape below names the arm it was built to
reach -- pair mode (C <= 64: two samples per CTA), C % 4 != 0 in the Gram epilogue, split-K with a one-block last split,
16 / 17 / 32 / 33+ k blocks per CTA (the edges of the TMEM segment drain), partial last k block and n tile of S X -- and
proves that it took it:

* Gram: the split plan restated from gram_plan_tc (isw_kernels.cu) is handed to dgvcc_isw_gram_tc_partials; the
  partials summed in split order must be BIT-identical to what dgvcc_isw_gram returns.  The SIMT Gram gives other bits,
  so this also shows the launcher did not fall back.  Shapes meant for the SIMT Gram must be refused (-3).
* dX = S X: the loss backward must be bit-identical to dgvcc_isw_sx_tc applied to the S matrix built by torch in the
  kernel's arithmetic; shapes meant for the SIMT GEMM must be refused and give the same bits with the tensor cores on
  or off.

Gates against the oracle evaluated in float64: loss rtol 1e-5, gradients rtol 1e-4 + 2e-6 max|ref| (the gate of
test_aux_gpu.py).  The fp32 torch-CPU evaluation of the same oracle is recorded beside the kernels as an (accuracy)
margin: it stays well inside these gates, so a kernel outside them is wrong, not merely unlucky.
"""
import functools
import warnings

import pytest
import torch

from dgvcc_b200 import _native
from dgvcc_b200.losses.lw import lw_loss
from dgvcc_b200.losses.ortho import ortho_loss
from oracle import aux_losses_oracle as ao
from helpers import assert_close, record_margin

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
UNSUPPORTED = -3            # DGVCC_ERR_UNSUPPORTED
LOSS_RTOL = 1e-5
GRAD_RTOL, GRAD_ATOL = 1e-4, 2e-6
KINDS = ["normal", "correlated"]


def cdiv(a, b):
    return -(-a // b)


def gram_plan_tc(batch, c, hw):
    """gram_plan_tc (isw_kernels.cu) restated: (pair, splits, k_per_split)."""
    pair = c <= 64
    t1 = 1 if pair else cdiv(c, 128)
    units = (cdiv(batch, 2) if pair else batch) * t1 * (t1 + 1) // 2
    s = 0 if units > 148 else 148 // units
    s = max(1, min(s, cdiv(hw, 256)))
    kps = cdiv(cdiv(hw, s), 32) * 32
    return pair, cdiv(hw, kps), kps


def plan_summary(batch, c, hw):
    """(pair, splits, k blocks of the first and the last split, TMEM segments of the first and the last split)."""
    pair, splits, kps = gram_plan_tc(batch, c, hw)
    kb = (cdiv(min(kps, hw), 32), cdiv(hw - (splits - 1) * kps, 32))
    return pair, splits, kb, tuple(cdiv(k, 16) for k in kb)


# (shape, Gram arm, S X on the tensor cores).  Gram arm: plan_summary of the tensor-core plan, or None for the SIMT Gram.
LW_CASES = [
    ((3, 50, 32, 32), (True, 4, (8, 8), (1, 1)), False),           # pair, C % 4 != 0 in the epilogue and in S X
    ((2, 130, 64, 96), (False, 24, (8, 8), (1, 1)), False),        # 3 tiles, partial second tile, C % 4 != 0
    ((7, 36, 38, 54), (True, 9, (8, 1), (1, 1)), True),            # odd batch, last split of 1 k block; S X k and n tails
    ((1, 64, 128, 128), (True, 64, (8, 8), (1, 1)), True),         # batch 1: the second sample of the pair is all TMA fill
    ((149, 64, 32, 32), (True, 1, (32, 32), (2, 2)), True),        # odd batch, 2 full segments
    ((150, 64, 17, 32), (True, 1, (17, 17), (2, 2)), True),        # last segment of one k block
    ((8, 512, 16, 32), (False, 1, (16, 16), (1, 1)), True),        # exactly one segment
    ((8, 512, 17, 32), (False, 1, (17, 17), (2, 2)), True),
    ((8, 512, 32, 32), (False, 1, (32, 32), (2, 2)), True),
    ((8, 512, 20, 53), (False, 1, (34, 34), (3, 3)), True),        # 1060 = 33 * 32 + 4: partial last k block
    ((16, 256, 64, 64), (False, 3, (43, 42), (3, 3)), True),
    ((8, 64, 160, 160), (True, 37, (22, 8), (2, 1)), True),        # config-5 shape
    ((3, 100, 28, 23), (False, 3, (7, 7), (1, 1)), True),          # S X: 644 = 5 * 128 + 4, C = 100 = 3 * 32 + 4
    ((2, 24, 20, 20), None, False),                                # C < 32
    ((1, 48, 7, 9), None, False),                                  # HW % 4 != 0
]
# ortho_loss(x, y) with x, y [C, P]: the Gram of the stacked [x; y] has 2C rows
ORTHO_CASES = [
    ((16, 64), (True, 1, (2, 2), (1, 1)), False),                  # 2C = 32, C < 32 for S X
    ((20, 1000), (True, 4, (8, 8), (1, 1)), False),
    ((33, 96), (False, 1, (3, 3), (1, 1)), False),                 # 2C = 66: C % 4 != 0 outside pair mode
    ((36, 132), (False, 1, (5, 5), (1, 1)), True),                 # S X: partial k block and n tile
    ((200, 8192), (False, 14, (19, 9), (2, 1)), True),
    ((768, 544), (False, 1, (17, 17), (2, 2)), True),              # 78 tiles
    ((768, 1024), (False, 1, (32, 32), (2, 2)), True),
    ((100, 333), None, False),                                     # P % 4 != 0
    ((8, 100), None, False),                                       # 2C < 32
]


def _lw_id(case):
    return "x".join(map(str, case[0][:2])) + f"x{case[0][2] * case[0][3]}"


def _ortho_id(case):
    return "x".join(map(str, case[0]))


# ------------------------------------------------------------------------------------------------------- inputs
def _seed(shape, kind):
    return 1000 + 7 * sum(i * v for i, v in enumerate(shape, 1)) + KINDS.index(kind)


@functools.lru_cache(maxsize=None)
def lw_inputs(shape, kind):
    """i.i.d. normal without a mask, or correlated channels with per-channel offsets and a binary 50 % mask."""
    g = torch.Generator().manual_seed(_seed(shape, kind))
    n, c, h, w = shape
    x = torch.randn(shape, generator=g)
    if kind == "normal":
        return x, None
    x = x + 0.4 * x.roll(1, 1) + 0.8 * torch.randn(1, c, 1, 1, generator=g)
    return x, (torch.rand(n, 1, h, w, generator=g) < 0.5).float()


@functools.lru_cache(maxsize=None)
def ortho_inputs(shape, kind):
    """y = 0.5 x + noise, so the entries of x y^T do not all cancel."""
    g = torch.Generator().manual_seed(_seed(shape, kind))
    c, p = shape
    x = torch.randn(shape, generator=g)
    if kind == "correlated":
        x = x + 0.4 * x.roll(1, 0) + 0.8 * torch.randn(c, 1, generator=g)
    return x, 0.5 * x + torch.randn(shape, generator=g)


def _oracle(fn, leaves, upstream=1.0, extra=()):
    """{dtype: (loss, [gradients of upstream * loss for each leaf])} of fn at float64 and float32 (torch CPU)."""
    out = {}
    for dt in (torch.float64, torch.float32):
        # copies: .to(float32) of a float32 input is the input itself, and the cached inputs must stay gradient-free
        # (a CUDA copy of a tensor that requires grad is no leaf, so its .grad would stay None)
        ls = [t.to(dt, copy=True).requires_grad_(True) for t in leaves]
        loss = fn(*ls, *(None if t is None else t.to(dt) for t in extra))
        (upstream * loss).backward()
        out[dt] = (loss.detach(), [t.grad for t in ls])
    return out


@functools.lru_cache(maxsize=None)
def lw_reference(shape, kind):
    x, mask = lw_inputs(shape, kind)
    return _oracle(ao.lw_loss, [x], extra=[mask])


@functools.lru_cache(maxsize=None)
def ortho_reference(shape, kind):
    return _oracle(ao.ortho_loss, list(ortho_inputs(shape, kind)))


def check_against_fp64(what, loss, grads, ref):
    """Gate the kernels' loss and gradients against the fp64 evaluation; record where they and the fp32 reference sit."""
    l64, g64 = ref[torch.float64]
    l32, g32 = ref[torch.float32]
    loss = loss.detach().cpu().double().reshape(())
    assert_close(loss, l64, LOSS_RTOL, 0, f"{what}: loss")
    for i, (got, want) in enumerate(zip(grads, g64)):
        assert_close(got.detach().cpu(), want, GRAD_RTOL, GRAD_ATOL * float(want.abs().max()), f"{what}: gradient {i}")
    gate_l = LOSS_RTOL * l64.abs().reshape(1)
    for who, l, gs in (("CUDA", loss, [g.detach().cpu() for g in grads]), ("reference fp32", l32, g32)):
        record_margin(f"{who}: loss (accuracy)", (l.double() - l64).abs().reshape(1), gate_l, LOSS_RTOL, 0)
        for got, want in zip(gs, g64):
            atol = GRAD_ATOL * float(want.abs().max())
            record_margin(f"{who}: gradient / aux gate (accuracy)", (got.double() - want).abs(),
                          atol + GRAD_RTOL * want.abs(), GRAD_RTOL, atol)


# ---------------------------------------------------------------------------------------------- the C ABI directly
def _lib():
    return _native.lib()


def _stream():
    return _native.stream_ptr(DEV)


def standardize(x, mask):
    """The Gram input lw_loss builds: yhat, or yhat * mask."""
    n, c, h, w = x.shape
    hw = h * w
    m = None if mask is None else mask.reshape(n, hw).contiguous()
    yhat = torch.empty((n, c, hw), device=DEV)
    ym = torch.empty_like(yhat) if m is not None else None
    invstd = torch.empty((n * c,), device=DEV)
    _native.check(_lib().dgvcc_lw_standardize_forward(_native.ptr(x.contiguous()), _native.ptr(m), n, c, hw, 1e-5,
                                                      _native.ptr(yhat), _native.ptr(ym), _native.ptr(invstd), _stream()),
                  "dgvcc_lw_standardize_forward")
    return ym if m is not None else yhat


def gram(y, tc):
    """dgvcc_isw_gram of y [B, C, HW]: (gram [B, C, C], workspace, its size)."""
    b, c, hw = y.shape
    nbytes = _lib().dgvcc_isw_workspace_bytes(b, c, hw)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=DEV)
    out = torch.empty((b, c, c), device=DEV)
    _native.check(_lib().dgvcc_isw_gram(_native.ptr(y), b, c, hw, tc, _native.ptr(ws), nbytes, _native.ptr(out), _stream()),
                  "dgvcc_isw_gram")
    return out, ws, nbytes


def check_gram_dispatch(y, arm, what):
    """The restated plan is the expected one, and the tensor-core partials taken with it are summed, in split order, to
    exactly what dgvcc_isw_gram returns.  arm None: the tensor-core Gram must refuse the shape."""
    b, c, hw = y.shape
    pair, splits, kps = gram_plan_tc(b, c, hw)
    tile = 64 if pair else 128
    t1 = 1 if pair else cdiv(c, 128)
    n_tiles = t1 * (t1 + 1) // 2
    part = torch.full((b, splits, n_tiles, tile, tile), float("nan"), device=DEV)
    rc = _lib().dgvcc_isw_gram_tc_partials(_native.ptr(y), b, c, hw, splits, kps, _native.ptr(part), _stream())
    if arm is None:
        assert rc == UNSUPPORTED, f"{what}: the tensor-core Gram took a shape meant for the SIMT Gram (rc {rc})"
        return
    assert plan_summary(b, c, hw) == arm, f"{what}: plan {plan_summary(b, c, hw)}, expected {arm}"
    assert rc == 0, f"{what}: the tensor-core Gram refused its plan (rc {rc})"
    acc = part[:, 0]
    for s in range(1, splits):
        acc = acc + part[:, s]
    full = torch.full((b, c, c), float("nan"), device=DEV)
    t = 0
    for ti in range(t1):
        for tj in range(ti, t1):
            r0, r1, c0, c1 = ti * tile, min(c, ti * tile + tile), tj * tile, min(c, tj * tile + tile)
            full[:, r0:r1, c0:c1] = acc[:, t, :r1 - r0, :c1 - c0]
            t += 1
    want, _, _ = gram(y, 1)
    iu = torch.triu_indices(c, c, device=DEV)
    bad = full[:, iu[0], iu[1]] != want[:, iu[0], iu[1]]
    assert not bool(bad.any()), (f"{what}: {int(bad.sum())} of {bad.numel()} upper entries of dgvcc_isw_gram differ from "
                                 f"the tensor-core partials of plan (pair {pair}, {splits} splits, {kps} k per split)")


def sx_tc(s, x):
    """dgvcc_isw_sx_tc(S, X) -> (rc, dX)."""
    b, c, hw = x.shape
    dx = torch.full((b, c, hw), float("nan"), device=DEV)
    rc = _lib().dgvcc_isw_sx_tc(_native.ptr(s), _native.ptr(x), b, c, hw, _native.ptr(dx), _stream())
    return rc, dx


def assert_same_bits(a, b, what):
    assert a.shape == b.shape, f"{what}: shapes {tuple(a.shape)} and {tuple(b.shape)}"
    same = (a.view(torch.int32) == b.view(torch.int32))
    assert bool(same.all()), f"{what}: {int((~same).sum())} of {same.numel()} elements differ"


# --------------------------------------------------------------------------------------- every arm, every kind
@pytest.mark.parametrize("tc", [1, 0])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("case", LW_CASES, ids=_lw_id)
def test_lw_loss_against_fp64(case, kind, tc, monkeypatch):
    monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", str(tc))
    shape = case[0]
    x, mask = lw_inputs(shape, kind)
    xd = x.to(DEV).requires_grad_(True)
    loss = lw_loss(xd, None if mask is None else mask.to(DEV))
    loss.backward()
    check_against_fp64(f"lw {shape} {kind} tc={tc}", loss, [xd.grad], lw_reference(shape, kind))


@pytest.mark.parametrize("tc", [1, 0])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("case", ORTHO_CASES, ids=_ortho_id)
def test_ortho_loss_against_fp64(case, kind, tc, monkeypatch):
    monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", str(tc))
    shape = case[0]
    x, y = ortho_inputs(shape, kind)
    xd, yd = x.to(DEV).requires_grad_(True), y.to(DEV).requires_grad_(True)
    loss = ortho_loss(xd, yd)
    loss.backward()
    check_against_fp64(f"ortho {shape} {kind} tc={tc}", loss, [xd.grad, yd.grad], ortho_reference(shape, kind))


@pytest.mark.parametrize("case", LW_CASES, ids=_lw_id)
def test_lw_takes_the_arm_it_was_built_for(case):
    shape, arm, sx_on_tc = case
    n, c, h, w = shape
    hw = h * w
    x, mask = lw_inputs(shape, "correlated")
    y = standardize(x.to(DEV), mask.to(DEV))
    what = f"lw {shape}"
    check_gram_dispatch(y, arm, what)
    g, ws, nbytes = gram(y, 1)
    up = torch.tensor([0.37], device=DEV)

    def backward(tc):
        dy = torch.empty_like(y)
        _native.check(_lib().dgvcc_lw_loss_backward(_native.ptr(y), _native.ptr(g), _native.ptr(up), n, c, hw, tc,
                                                    _native.ptr(ws), nbytes, _native.ptr(dy), _stream()),
                      "dgvcc_lw_loss_backward")
        return dy

    dy = backward(1)
    t = torch.triu(g, 1)
    s = ((2.0 * up) * (t + t.transpose(1, 2))).contiguous()   # lw_grad_s_kernel: (2.f * g) * upper entry
    rc, want = sx_tc(s, y)
    if sx_on_tc:
        assert rc == 0, f"{what}: dgvcc_isw_sx_tc refused the shape (rc {rc})"
        assert_same_bits(dy, want, f"{what}: dgvcc_lw_loss_backward vs dgvcc_isw_sx_tc")
    else:
        assert rc == UNSUPPORTED, f"{what}: dgvcc_isw_sx_tc took a shape meant for the SIMT GEMM (rc {rc})"
        assert_same_bits(dy, backward(0), f"{what}: backward with the tensor cores on vs off")


@pytest.mark.parametrize("case", ORTHO_CASES, ids=_ortho_id)
def test_ortho_takes_the_arm_it_was_built_for(case):
    (c, p), arm, sx_on_tc = case
    x, y = ortho_inputs((c, p), "correlated")
    z = torch.cat([x, y]).to(DEV).contiguous()
    what = f"ortho {(c, p)}"
    check_gram_dispatch(z.view(1, 2 * c, p), arm, what)
    g, ws, nbytes = gram(z.view(1, 2 * c, p), 1)
    g = g[0]
    up = torch.tensor([0.37], device=DEV)

    def backward(tc):
        gx, gy = torch.empty((c, p), device=DEV), torch.empty((c, p), device=DEV)
        _native.check(_lib().dgvcc_ortho_loss_backward(_native.ptr(z[:c]), _native.ptr(z[c:]), _native.ptr(g),
                                                       _native.ptr(up), c, p, tc, _native.ptr(ws), nbytes, _native.ptr(gx),
                                                       _native.ptr(gy), _stream()), "dgvcc_ortho_loss_backward")
        return gx, gy

    gx, gy = backward(1)
    cf = torch.tensor(float(c), device=DEV)
    k = (2.0 * up) / (cf * cf)                                 # ortho_grad_s_kernel, float32
    sx = (k * torch.triu(g[:c, c:], 1)).contiguous()
    sy = sx.t().contiguous()
    rc_x, want_x = sx_tc(sx.view(1, c, c), z[c:].view(1, c, p))
    rc_y, want_y = sx_tc(sy.view(1, c, c), z[:c].view(1, c, p))
    if sx_on_tc:
        assert rc_x == 0 and rc_y == 0, f"{what}: dgvcc_isw_sx_tc refused the shape (rc {rc_x}, {rc_y})"
        assert_same_bits(gx, want_x[0], f"{what}: grad x vs dgvcc_isw_sx_tc(Sx, y)")
        assert_same_bits(gy, want_y[0], f"{what}: grad y vs dgvcc_isw_sx_tc(Sx^T, x)")
    else:
        assert rc_x == UNSUPPORTED and rc_y == UNSUPPORTED, \
            f"{what}: dgvcc_isw_sx_tc took a shape meant for the SIMT GEMM (rc {rc_x}, {rc_y})"
        gx0, gy0 = backward(0)
        assert_same_bits(gx, gx0, f"{what}: grad x with the tensor cores on vs off")
        assert_same_bits(gy, gy0, f"{what}: grad y with the tensor cores on vs off")


# ------------------------------------------------------------------------------------------ exact properties
@pytest.mark.parametrize("tc", [1, 0])
@pytest.mark.parametrize("shape,changed", [((7, 36, 38, 54), (3, 6, 1)),     # pair mode: middle, last (alone), odd
                                           ((5, 130, 28, 23), (2, 4, 1))])   # 3 tiles, 3 splits
def test_lw_samples_stay_independent(shape, changed, tc, monkeypatch):
    """Changing one sample must not move a bit of any other sample's Gram or gradient: the split plan depends only on
    the shape, so a leak between the two samples of a pair CTA, or between tiles, would show here."""
    monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", str(tc))
    gen = torch.Generator().manual_seed(sum(shape))
    x = torch.randn(shape, generator=gen)

    def run(xc):
        xd = xc.to(DEV).requires_grad_(True)
        lw_loss(xd).backward()
        g, _, _ = gram(standardize(xd.detach(), None), tc)
        return g, xd.grad

    g0, d0 = run(x)
    for k in changed:
        x2 = x.clone()
        x2[k] = 2.0 * torch.randn(shape[1:], generator=gen) + 0.3
        g1, d1 = run(x2)
        others = [j for j in range(shape[0]) if j != k]
        assert_same_bits(g1[others], g0[others], f"{shape} tc={tc}: Gram of the other samples after changing sample {k}")
        assert_same_bits(d1[others], d0[others], f"{shape} tc={tc}: x.grad of the other samples after changing sample {k}")
        assert not torch.equal(g1[k], g0[k])


@pytest.mark.parametrize("tc", [1, 0])
@pytest.mark.parametrize("shape", [(33, 96), (200, 1000), (768, 544)])
def test_stacked_ortho_gram_is_exactly_symmetric(shape, tc):
    c, p = shape
    x, y = ortho_inputs(shape, "normal")
    g, _, _ = gram(torch.cat([x, y]).to(DEV).view(1, 2 * c, p), tc)
    assert_same_bits(g[0], g[0].t().contiguous(), f"stacked Gram {2 * c}x{2 * c} tc={tc} against its transpose")


@pytest.mark.parametrize("tc", [1, 0])
def test_two_runs_give_the_same_bits(tc, monkeypatch):
    monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", str(tc))
    x, mask = lw_inputs((16, 256, 64, 64), "correlated")
    xo, yo = ortho_inputs((200, 8192), "correlated")
    runs = []
    for _ in range(2):
        xd = x.to(DEV).requires_grad_(True)
        l1 = lw_loss(xd, mask.to(DEV))
        l1.backward()
        ad, bd = xo.to(DEV).requires_grad_(True), yo.to(DEV).requires_grad_(True)
        l2 = ortho_loss(ad, bd)
        l2.backward()
        runs.append([l1.detach().reshape(1), xd.grad, l2.detach().reshape(1), ad.grad, bd.grad])
    for name, a, b in zip(["lw loss", "lw grad", "ortho loss", "ortho grad x", "ortho grad y"], *runs):
        assert_same_bits(a, b, f"tc={tc}: {name} of two runs")


@pytest.mark.parametrize("tc", [1, 0])
def test_one_channel_gives_exactly_zero(tc, monkeypatch):
    """C = 1: no strictly-upper entries, so the loss and every gradient are exactly 0."""
    monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", str(tc))
    gen = torch.Generator().manual_seed(3)
    xd = torch.randn((2, 1, 8, 8), generator=gen).to(DEV).requires_grad_(True)
    loss = lw_loss(xd)
    loss.backward()
    assert float(loss) == 0.0 and bool((xd.grad == 0).all())
    ad = torch.randn((1, 64), generator=gen).to(DEV).requires_grad_(True)
    bd = torch.randn((1, 64), generator=gen).to(DEV).requires_grad_(True)
    loss = ortho_loss(ad, bd)
    loss.backward()
    assert float(loss) == 0.0 and bool((ad.grad == 0).all()) and bool((bd.grad == 0).all())


@pytest.mark.parametrize("tc", [1, 0])
def test_one_pixel_gives_nan_like_the_reference(tc, monkeypatch):
    """HW = 1: the unbiased variance is 0 / 0."""
    monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", str(tc))
    x = torch.randn((2, 40, 1, 1), generator=torch.Generator().manual_seed(4))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")   # torch.var warns about zero degrees of freedom
        ref = ao.lw_loss(x.double())
    assert torch.isnan(ref)
    assert torch.isnan(lw_loss(x.to(DEV)).cpu())


# ------------------------------------------------------------------------------------- input edges against fp64
def _lw_case(what, x, mask, tc, upstream=1.0):
    xd = x.to(DEV).requires_grad_(True)
    loss = lw_loss(xd, None if mask is None else mask.to(DEV))
    (upstream * loss).backward()
    check_against_fp64(f"{what} tc={tc}", loss, [xd.grad], _oracle(ao.lw_loss, [x], upstream, [mask]))


@pytest.mark.parametrize("tc", [1, 0])
@pytest.mark.parametrize("shape", [(4, 64, 32, 32), (2, 132, 32, 32)])
def test_lw_low_variance_and_constant_channels(shape, tc, monkeypatch):
    """Every fourth channel scaled by 1e-3 (var ~ 1e-6: the 1e-5 inside sqrt(var + eps) matters) and one exactly
    constant channel: HW is a power of two, so its mean is exact, yhat is 0 and the backward divides by sqrt(1e-5)."""
    monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", str(tc))
    x = torch.randn(shape, generator=torch.Generator().manual_seed(sum(shape)))
    x[:, ::4] *= 1e-3
    x[:, 1] = 0.75
    _lw_case(f"lw low variance {shape}", x, None, tc)


@pytest.mark.parametrize("tc", [1, 0])
@pytest.mark.parametrize("shape", [(3, 48, 24, 24), (3, 132, 16, 16)])
def test_lw_fractional_empty_and_single_pixel_masks(shape, tc, monkeypatch):
    monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", str(tc))
    gen = torch.Generator().manual_seed(sum(shape) + 1)
    n, c, h, w = shape
    x = torch.randn(shape, generator=gen)
    mask = torch.zeros((n, 1, h, w))
    mask[0] = torch.rand((1, h, w), generator=gen)   # fractional
    mask[2, 0, h // 3, w // 2] = 0.6                  # one pixel; image 1 has an all-zero mask
    _lw_case(f"lw masks {shape}", x, mask, tc)


@pytest.mark.parametrize("tc", [1, 0])
def test_upstream_gradient_other_than_one(tc, monkeypatch):
    monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", str(tc))
    x, mask = lw_inputs((7, 36, 38, 54), "correlated")
    _lw_case("lw upstream -0.37", x, mask, tc, upstream=-0.37)
    a, b = ortho_inputs((36, 132), "correlated")
    ad, bd = a.to(DEV).requires_grad_(True), b.to(DEV).requires_grad_(True)
    loss = ortho_loss(ad, bd)
    (-0.37 * loss).backward()
    check_against_fp64(f"ortho upstream -0.37 tc={tc}", loss, [ad.grad, bd.grad], _oracle(ao.ortho_loss, [a, b], -0.37))


@pytest.mark.parametrize("tc", [1, 0])
@pytest.mark.parametrize("shape", [(36, 132), (200, 1000)])
def test_ortho_of_a_tensor_with_itself(shape, tc, monkeypatch):
    """ortho_loss(x, x): autograd adds the two gradients."""
    monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", str(tc))
    x, _ = ortho_inputs(shape, "correlated")
    xd = x.to(DEV).requires_grad_(True)
    loss = ortho_loss(xd, xd)
    loss.backward()
    ref = _oracle(lambda a: ao.ortho_loss(a, a), [x])
    check_against_fp64(f"ortho(x, x) {shape} tc={tc}", loss, [xd.grad], ref)


@pytest.mark.parametrize("tc", [1, 0])
def test_non_contiguous_inputs_give_the_bits_of_their_contiguous_copy(tc, monkeypatch):
    monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", str(tc))
    gen = torch.Generator().manual_seed(6)
    base = torch.randn((4, 64, 40, 24), generator=gen).to(DEV).requires_grad_(True)
    view = base.transpose(2, 3)                        # [4, 64, 24, 40], not contiguous
    copy = view.detach().contiguous().requires_grad_(True)
    l_view, l_copy = lw_loss(view), lw_loss(copy)
    l_view.backward()
    l_copy.backward()
    assert_same_bits(l_view.detach().reshape(1), l_copy.detach().reshape(1), f"tc={tc}: lw loss")
    assert_same_bits(base.grad.transpose(2, 3).contiguous(), copy.grad, f"tc={tc}: lw grad")

    bx = torch.randn((132, 36), generator=gen).to(DEV).requires_grad_(True)
    by = torch.randn((132, 36), generator=gen).to(DEV).requires_grad_(True)
    cx = bx.detach().t().contiguous().requires_grad_(True)
    cy = by.detach().t().contiguous().requires_grad_(True)
    l_view, l_copy = ortho_loss(bx.t(), by.t()), ortho_loss(cx, cy)
    l_view.backward()
    l_copy.backward()
    assert_same_bits(l_view.detach().reshape(1), l_copy.detach().reshape(1), f"tc={tc}: ortho loss")
    assert_same_bits(bx.grad.t().contiguous(), cx.grad, f"tc={tc}: ortho grad x")
    assert_same_bits(by.grad.t().contiguous(), cy.grad, f"tc={tc}: ortho grad y")
