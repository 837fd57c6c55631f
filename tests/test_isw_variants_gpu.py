"""Every ISW-specific kernel arm against an fp64 evaluation: instance norm, loss slicing, clamp gate, backward arms, and the
native fp16 / bf16 route.

The Gram and dX = S X GEMMs are proven bit for bit at every split plan in test_aux_variants_gpu.py; this file covers
the kernels of csrc/isw_kernels.cu around them.  Each case names the arm it was built to reach, restates the host
predicate that picks that arm, asserts the predicate says what the case id says, and -- where the arm shows through
the C ABI -- proves the kernels took it:

* instance norm: a plane is cached in shared memory while hw * sizeof(T) <= 200 KB, with the opt-in above 46 KB (the
  kernel's static shared memory shares the default 48 KB); past 200 KB it is read from HBM twice.  Shapes sit at and on either side of both edges, in fp32, fp16 and bf16.
* loss forward: max(1, min(32, C*C / 4096)) slices per sample, a float4 path when C*C % 4 == 0 and both pointers are
  16-byte aligned, a scalar path otherwise, and a finishing loop over the samples that strides by 256.  The per-slice
  partials sit in the workspace (layout restated from `carve`): the test hands the kernel a NaN-filled workspace and
  checks that exactly the planned slices were written, that each matches an fp64 sum of its element range, and that
  the slices added in slice order in fp32, minus the margin, give off[b] bit for bit.
* clamp: some samples of one batch clamped and others not; a sample exactly on the boundary (margin = the kernel's own
  off[b]) keeps its gradient, as torch's clamp passes the gradient at the boundary.
* loss backward: the factored EXACT GEMM (0/1 mask), the general GEMM (fractional mask), and the SIMT GEMM
  (DGVCC_ISW_TENSOR_CORES=0, C % 4 != 0, HW % 4 != 0, a misaligned map); covariance backward on the general GEMM and on
  SIMT.  The general arms are bit-identical to dgvcc_isw_sx_tc applied to S built by torch in the kernel's arithmetic.
* half route: the TILED shapes and config-5 layers of test_isw_half_gpu.py against fp64, stage by stage.

Gates (those of test_isw_gpu.py and test_aux_variants_gpu.py): loss rtol 1e-5; f_cor rtol 1e-5 + 5e-7 max|ref|;
instance norm rtol 1e-5 + 1e-6; gradients rtol 1e-4 + 2e-6 max|ref| (max per plane for the instance norm).  Where a
half value is written the gate adds half an ulp of the dtype.  torch's own fp32 evaluation of each quantity is recorded
beside the kernels as an (accuracy) margin, so the session summary shows the gates are not loose.
"""
import functools

import pytest
import torch
import torch.nn.functional as F

from dgvcc_b200 import _native
from dgvcc_b200.models.ISW import InstanceWhitening, get_covariance_matrix, instance_whitening_loss
from oracle import isw_oracle
from helpers import record_margin

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
UNSUPPORTED = -3            # DGVCC_ERR_UNSUPPORTED
LOSS_RTOL = 1e-5
COV_RTOL, COV_ATOL = 1e-5, 5e-7
NORM_RTOL, NORM_ATOL = 1e-5, 1e-6
GRAD_RTOL, GRAD_ATOL = 1e-4, 2e-6
EPS = 1e-5                  # nn.InstanceNorm2d default
UPSTREAM = -0.37            # an upstream gradient other than 1


def cdiv(a, b):
    return -(-a // b)


def align_up(n, a):
    return cdiv(n, a) * a


# ------------------------------------------------------------------------------------ host predicates restated
SMEM_NO_OPT_IN, SMEM_CAP = 48 * 1024 - 2048, 200 * 1024


def norm_arm(hw, itemsize):
    """instnorm_forward (isw_kernels.cu): which arm a plane of hw elements takes (the opt-in leaves 2 KB of the default
    48 KB to the kernel's static shared memory)."""
    nbytes = hw * itemsize
    if nbytes > SMEM_CAP:
        return "uncached"
    return "cached-optin" if nbytes > SMEM_NO_OPT_IN else "cached"


LOSS_CHUNKS = 32


def loss_slices(c):
    """dgvcc_isw_loss_forward: slices (CTAs) per sample."""
    return max(1, min(LOSS_CHUNKS, c * c // 4096))


def loss_vector(c, f_cor, mask):
    """isw_loss_kernel: the float4 path, else the scalar one."""
    return (c * c) % 4 == 0 and ((f_cor.data_ptr() | mask.data_ptr()) & 15) == 0


def sx_tc_tiles(c, hw, *tensors):
    """sx_tc_tiles and tma_aligned (isw_tc.cuh): dX = S X on the tensor cores."""
    return hw % 4 == 0 and c % 4 == 0 and c >= 32 and all(t.data_ptr() % 16 == 0 for t in tensors)


def half_tc_tiles(c, hw, *tensors):
    """half_tc_tiles and tma_aligned (isw_tc.cuh): the native fp16 / bf16 route."""
    return hw % 8 == 0 and c % 4 == 0 and c >= 32 and all(t.data_ptr() % 16 == 0 for t in tensors)


def mask_is_binary(mask):
    return bool(((mask == 0) | (mask == 1)).all())


def gram_plan_simt(b, c, hw):
    t1 = cdiv(c, 64)
    n = t1 * (t1 + 1) // 2
    s = 1 if b * n >= 296 else cdiv(296, b * n)
    s = max(1, min(s, cdiv(hw, 256)))
    kps = cdiv(cdiv(hw, s), 32) * 32
    return cdiv(hw, kps), n, 64


def gram_plan_tc(b, c, hw):
    pair = c <= 64
    t1 = 1 if pair else cdiv(c, 128)
    n = t1 * (t1 + 1) // 2
    units = (cdiv(b, 2) if pair else b) * n
    s = 0 if units > 148 else 148 // units
    s = max(1, min(s, cdiv(hw, 256)))
    kps = cdiv(cdiv(hw, s), 32) * 32
    return cdiv(hw, kps), n, 64 if pair else 128


def workspace_layout(b, c, hw):
    """carve (isw_kernels.cu): (byte offset of off[B], total bytes).  off[B] is followed by the [B][32] slice partials."""
    part = max(b * s * n * t * t for s, n, t in (gram_plan_simt(b, c, hw), gram_plan_tc(b, c, hw)))
    off = align_up(part * 4, 256)
    total = off + align_up(b * (2 + LOSS_CHUNKS) * 4, 256) + 256 + align_up(b * c * c * 4, 256)
    return off, total


# ---------------------------------------------------------------------------------------------------- checking
def half_ulp(v, dtype):
    """Half an ulp of dtype at |v| (subnormal spacing below the normal range)."""
    fi = torch.finfo(dtype)
    mant = {torch.float16: 10, torch.bfloat16: 7}[dtype]
    _, e = torch.frexp(v.abs().clamp_min(fi.smallest_normal))
    return torch.ldexp(torch.ones_like(v), e - 1 - mant) * 0.5


def check(what, got, ref, rtol, atol, ref32=None, dtype=None):
    """|got - ref| <= atol + rtol |ref| (+ half an ulp of dtype at |ref| + that gate), ref in fp64; atol may be a tensor
    broadcast against ref.  ref32: torch's own fp32 evaluation, recorded (not asserted) against the same gate."""
    got = got.detach().double().reshape(ref.shape)
    tol = atol + rtol * ref.abs()
    if dtype is not None:
        tol = tol + half_ulp(ref.abs() + tol, dtype)
    err = (got - ref).abs()
    base = float(atol.max()) if torch.is_tensor(atol) else float(atol)
    record_margin(what, err.cpu(), tol.cpu(), rtol, base)
    if ref32 is not None:
        record_margin(f"reference fp32: {what} (accuracy)", (ref32.detach().double().reshape(ref.shape) - ref).abs().cpu(),
                      tol.cpu(), rtol, base)
        record_margin(f"CUDA: {what} (accuracy)", err.cpu(), tol.cpu(), rtol, base)
    bad = ~(err <= tol)
    if bool(bad.any()):
        idx = tuple(torch.nonzero(bad)[0].tolist())
        raise AssertionError(f"{what}: {int(bad.sum())}/{bad.numel()} out of tolerance; worst err/tol "
                             f"{float((err / tol).max()):.3g}; first at {idx}: got {float(got[idx]):.9g} "
                             f"ref {float(ref[idx]):.9g}")
    if ref32 is not None:
        print(f"{what}: worst err/gate {float((err / tol).max()):.3g}, torch fp32 "
              f"{float(((ref32.detach().double().reshape(ref.shape) - ref).abs() / tol).max()):.3g}")


def assert_same_bits(a, b, what):
    assert a.shape == b.shape and a.dtype == b.dtype, f"{what}: {a.shape} {a.dtype} vs {b.shape} {b.dtype}"
    same = a.contiguous().view(torch.int32 if a.element_size() == 4 else torch.int16) == \
        b.contiguous().view(torch.int32 if b.element_size() == 4 else torch.int16)
    assert bool(same.all()), f"{what}: {int((~same).sum())} of {same.numel()} elements differ"


def lib():
    return _native.lib()


def stream():
    return _native.stream_ptr(DEV)


P = _native.ptr


# ========================================================================================= 1. instance norm
# (arm, dtype, (B, C, H, W)); C = 6 special channels, see norm_input
NORM_CASES = [
    ("cached", torch.float32, (2, 6, 92, 128)),              # 11 776 fp32 = 46 KB: the largest plane without the opt-in
    ("cached-optin", torch.float32, (2, 6, 128, 96)),        # 12 288 = 48 KB exactly: needs the opt-in (static smem)
    ("cached-optin", torch.float32, (2, 6, 116, 106)),       # 12 296
    ("cached-optin", torch.float32, (2, 6, 160, 320)),       # 51 200 = 200 KB exactly: the largest cached plane
    ("uncached", torch.float32, (2, 6, 160, 321)),           # 51 360: past 200 KB
    ("uncached", torch.float32, (2, 6, 256, 256)),           # 65 536: a 512-px crop's first layer
    ("cached", torch.float16, (2, 6, 92, 256)),              # 23 552 half = 46 KB
    ("cached-optin", torch.float16, (2, 6, 128, 192)),       # 24 576 = 48 KB exactly
    ("cached-optin", torch.float16, (2, 6, 116, 212)),       # 24 592
    ("cached-optin", torch.float16, (2, 6, 320, 320)),       # 102 400 = 200 KB: a 640-px crop's first layer
    ("uncached", torch.float16, (2, 6, 320, 328)),           # 104 960
    ("cached", torch.bfloat16, (2, 6, 92, 256)),
    ("cached-optin", torch.bfloat16, (2, 6, 128, 192)),
    ("cached-optin", torch.bfloat16, (2, 6, 320, 320)),
    ("uncached", torch.bfloat16, (2, 6, 320, 328)),
]
CONST = 0.75    # a dyadic constant: the plane's fp32 sums and its mean are exact, so y is exactly 0


def _dt(dtype):
    return {torch.float32: "f32", torch.float16: "f16", torch.bfloat16: "bf16"}[dtype]


def _norm_id(case):
    arm, dtype, (b, c, h, w) = case
    return f"{arm}-{_dt(dtype)}-hw{h * w}"


def norm_input(shape, dtype, seed):
    """Channels: N(0,1); std 1e-3, 3.16e-3 and 1e-2 (variance 1e-6 .. 1e-4, where eps = 1e-5 matters); the constant
    CONST; mean 1e3 with std 1.  Returned in dtype on the device, with an upstream gradient N(0,1) in dtype."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(shape, generator=g)
    x[:, 1] *= 1e-3
    x[:, 2] *= 10 ** -2.5
    x[:, 3] *= 1e-2
    x[:, 4] = CONST
    x[:, 5] += 1e3
    dy = torch.randn(shape, generator=g)
    return x.to(dtype).to(DEV), dy.to(dtype).to(DEV)


@pytest.mark.parametrize("case", NORM_CASES, ids=_norm_id)
def test_instance_norm_against_fp64(case):
    arm, dtype, shape = case
    b, c, h, w = shape
    hw = h * w
    assert norm_arm(hw, torch.tensor([], dtype=dtype).element_size()) == arm
    x, dy = norm_input(shape, dtype, seed=hw + c)

    xk = x.clone().requires_grad_(True)
    y, _ = InstanceWhitening(c)(xk)
    y.backward(dy)
    assert y.dtype == dtype and xk.grad.dtype == dtype

    x64 = x.double().requires_grad_(True)
    y64 = F.instance_norm(x64, eps=EPS)
    y64.backward(dy.double())
    x32 = x.float().requires_grad_(True)          # torch's own fp32 instance norm, the accuracy yardstick
    y32 = F.instance_norm(x32, eps=EPS)
    y32.backward(dy.float())

    # the constant plane: exact mean, y exactly 0
    assert bool((y[:, 4] == 0).all()), f"{arm}: constant plane gives y != 0"
    half = dtype if dtype is not torch.float32 else None
    # A plane's fp32 mean carries ~ulp(|mean|) of rounding (torch's own fp32 norm as well), which shifts the whole plane
    # of y by that times invstd: the mean-1e3 plane gets 4 * 2^-24 |mean| invstd on top of the absolute floor.
    x64d = x64.detach()
    mean = x64d.mean((2, 3), keepdim=True)
    invstd = 1.0 / torch.sqrt(x64d.var((2, 3), unbiased=False, keepdim=True) + EPS)
    atol_y = NORM_ATOL + 4 * 2.0 ** -24 * mean.abs() * invstd
    check(f"{arm} {_dt(dtype)} y", y, y64.detach(), NORM_RTOL, atol_y, y32, half)
    g64 = x64.grad
    atol_g = GRAD_ATOL * g64.abs().amax((2, 3), keepdim=True)
    check(f"{arm} {_dt(dtype)} dx", xk.grad, g64, GRAD_RTOL, atol_g, x32.grad, half)


# ========================================================================================= 2. loss forward slicing
def correlated_map(shape, seed, strength=0.7, scales=None):
    """x_c = z_c + r_b s_c common with random signs s_c: every covariance entry sits near +-r^2 / (1 + r^2), far from 0,
    so no masked entry has a sign the fp32 evaluation could get wrong."""
    g = torch.Generator().manual_seed(seed)
    b, c, h, w = shape
    z = torch.randn(shape, generator=g)
    common = torch.randn(b, 1, h, w, generator=g)
    s = torch.where(torch.rand(1, c, 1, 1, generator=g) < 0.5, -1.0, 1.0)
    r = torch.full((b, 1, 1, 1), strength) if scales is None else torch.tensor(scales).view(b, 1, 1, 1)
    return z + r * s * common


def binary_mask(c, seed):
    return isw_oracle.upper_mask(c, 0.5, seed)


def fractional_mask(c, seed):
    g = torch.Generator().manual_seed(seed + 1)
    return binary_mask(c, seed) * (0.25 + 0.75 * torch.rand(c, c, generator=g))


def loss_forward_abi(f_cor, mask, margin, nr, hw):
    """dgvcc_isw_loss_forward with a NaN-filled workspace of the test's own: (loss, off[B], slice partials [B][32])."""
    b, c, _ = f_cor.shape
    n = lib().dgvcc_isw_workspace_bytes(b, c, hw)
    off_at, total = workspace_layout(b, c, hw)
    assert n == total, f"workspace layout restated wrongly: {total} bytes, the library says {n}"
    ws = torch.full((n // 4,), float("nan"), device=DEV)
    loss = torch.full((1,), float("nan"), device=DEV)
    _native.check(lib().dgvcc_isw_loss_forward(P(f_cor), P(mask), P(margin), P(nr), b, c, hw, P(ws), n, P(loss),
                                               stream()), "dgvcc_isw_loss_forward")
    torch.cuda.synchronize()
    o = off_at // 4
    return loss, ws[o:o + b].clone(), ws[o + b:o + b + b * LOSS_CHUNKS].view(b, LOSS_CHUNKS).clone()


def check_slices(what, f_cor, mask, margin, off, part):
    """Exactly the planned slices were written; each matches an fp64 sum of its element range; off[b] is their fp32
    sum in slice order minus the margin, bit for bit."""
    b, c, _ = f_cor.shape
    k = loss_slices(c)
    assert bool(torch.isfinite(part[:, :k]).all()), f"{what}: a planned slice partial was not written"
    assert bool(torch.isnan(part[:, k:]).all()), f"{what}: a slice beyond the planned {k} was written"
    acc = part[:, 0].clone()
    for j in range(1, k):
        acc = acc + part[:, j]
    assert_same_bits(off, acc - margin, f"{what}: off[b] vs the fp32 sum of its slices in slice order minus the margin")
    cc = c * c
    per = cdiv(cdiv(cc, k), 4) * 4
    flat = (f_cor.double() * mask.double()).abs().reshape(b, cc)
    ref = torch.stack([flat[:, j * per:min(cc, (j + 1) * per)].sum(1) for j in range(k)], 1)
    check(f"{what}: slice partials", part[:, :k], ref, LOSS_RTOL, 0)


# (arm, (B, C, H, W)): arm = slices per sample, vector or scalar path
LOSS_CASES = [
    ("1slice-scalar", (3, 33, 16, 16)),      # C*C = 1089, odd
    ("1slice-vector", (3, 64, 16, 16)),
    ("4slices-vector", (2, 128, 16, 16)),
    ("9slices-vector", (2, 200, 16, 16)),
    ("15slices-scalar", (2, 255, 16, 16)),   # 65 025, odd
    ("31slices-vector", (2, 362, 16, 16)),
    ("32slices-scalar", (2, 363, 16, 16)),   # 131 769, odd
    ("32slices-vector", (2, 512, 16, 16)),
    ("1slice-vector-B300", (300, 40, 8, 8)),  # the finishing loop's second pass (samples 256..299)
]


@pytest.mark.parametrize("case", LOSS_CASES, ids=[c[0] + "-c" + str(c[1][1]) for c in LOSS_CASES])
def test_loss_forward_slicing_against_fp64(case):
    arm, shape = case
    b, c, h, w = shape
    hw = h * w
    x = correlated_map(shape, seed=7 * c + b)
    mask = binary_mask(c, seed=c).to(DEV)
    xd = x.to(DEV)
    eye = torch.eye(c, device=DEV)
    f_cor, _ = get_covariance_matrix(xd, eye)
    want = f"{loss_slices(c)}slice" + ("s" if loss_slices(c) > 1 else "") + \
        ("-vector" if loss_vector(c, f_cor, mask) else "-scalar")
    assert arm.startswith(want), f"{arm}: the host predicates say {want}"

    zero, nr = torch.zeros(1, device=DEV), mask.sum().reshape(1)
    loss, off, part = loss_forward_abi(f_cor, mask, zero, nr, hw)
    check_slices(arm, f_cor, mask, zero, off, part)
    off64 = (f_cor.double() * mask.double()).abs().sum((1, 2))
    check(f"{arm}: off[b]", off, off64, LOSS_RTOL, 0)

    # the module end to end against the oracle on fp64 inputs
    loss_m = instance_whitening_loss(xd, eye, mask, 0, nr.reshape(()))
    ref64 = isw_oracle.whitening_loss(xd.double(), eye.double(), mask.double(), 0, nr.double().reshape(()))
    ref32 = isw_oracle.whitening_loss(xd, eye, mask, 0, nr.reshape(()))
    assert_same_bits(loss_m.reshape(1), loss, f"{arm}: module loss vs dgvcc_isw_loss_forward on its f_cor")
    check(f"{arm}: loss", loss_m, ref64, LOSS_RTOL, 0, ref32)


@pytest.mark.parametrize("c", [64, 128, 362])
def test_misaligned_mask_takes_the_scalar_path_with_the_same_bits(c):
    """A mask view 4 bytes past a 16-byte boundary takes the scalar path.  The two paths add in different orders, so on
    data whose every partial sum is exact in fp32 (entries k / 256 with |k| <= 16, a 0/1 mask) both must give that one
    exact value: the same bits, slice for slice, and the fp64 sum itself."""
    b, hw = 3, 256
    g = torch.Generator().manual_seed(c)
    f_cor = (torch.randint(-16, 17, (b, c, c), generator=g).double() / 256).float().to(DEV)
    mask = binary_mask(c, seed=c + 1).to(DEV)
    buf = torch.zeros(c * c + 1, device=DEV)
    buf[1:] = mask.reshape(-1)
    mis = buf[1:].view(c, c)
    assert loss_vector(c, f_cor, mask) and not loss_vector(c, f_cor, mis)
    zero, nr = torch.zeros(1, device=DEV), mask.sum().reshape(1)
    l_a, off_a, part_a = loss_forward_abi(f_cor, mask, zero, nr, hw)
    l_m, off_m, part_m = loss_forward_abi(f_cor, mis, zero, nr, hw)
    check_slices(f"c{c} misaligned", f_cor, mis, zero, off_m, part_m)
    k = loss_slices(c)
    assert_same_bits(part_m[:, :k], part_a[:, :k], f"c{c}: slice partials, scalar vs vector path")
    assert_same_bits(off_m, off_a, f"c{c}: off, scalar vs vector path")
    assert_same_bits(l_m, l_a, f"c{c}: loss, scalar vs vector path")
    exact = (f_cor.double() * mask.double()).abs().sum((1, 2))
    assert torch.equal(off_m.double(), exact), f"c{c}: off is not the exact sum"


@pytest.mark.parametrize("tc", [1, 0])
def test_misaligned_mask_through_the_module(tc, monkeypatch):
    """Random data through the module: the misaligned mask's loss sits within the gate of fp64, and its gradient (the
    gradient kernel reads the mask element-wise, whatever its alignment) has the bits of the aligned mask's."""
    monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", str(tc))
    shape = (3, 128, 16, 16)
    c = shape[1]
    xd = correlated_map(shape, seed=31).to(DEV)
    mask = binary_mask(c, seed=32).to(DEV)
    buf = torch.zeros(c * c + 1, device=DEV)
    buf[1:] = mask.reshape(-1)
    mis = buf[1:].view(c, c)
    eye = torch.eye(c, device=DEV)
    grads, losses = [], []
    for m in (mask, mis):
        xk = xd.clone().requires_grad_(True)
        loss = instance_whitening_loss(xk, eye, m, 0, m.sum())
        (UPSTREAM * loss).backward()
        grads.append(xk.grad)
        losses.append(loss.detach())
    ref64 = isw_oracle.whitening_loss(xd.double(), eye.double(), mask.double(), 0, mask.sum().double())
    for what, l in zip(("aligned", "misaligned"), losses):
        check(f"tc={tc} {what} mask: loss", l, ref64, LOSS_RTOL, 0)
    assert_same_bits(grads[1], grads[0], f"tc={tc}: gradient with the misaligned mask vs the aligned one")


# ========================================================================================= 3. clamp and margin
def oracle_grad(x, eye, mask, margin, nr, upstream=UPSTREAM, dtype=torch.float64):
    xr = x.detach().to(dtype).requires_grad_(True)
    loss = isw_oracle.whitening_loss(xr, eye.to(dtype), mask.to(dtype), margin, nr)
    (upstream * loss).backward()
    return loss.detach(), xr.grad


def ambiguous_rows(f_cor64, mask):
    """[B, C] rows holding a masked covariance entry below the fp32 evaluation error (its sign is not well defined)."""
    amb = (f_cor64.abs() < 2 * COV_ATOL * f_cor64.abs().amax()) & (mask.double() > 0)
    rows = torch.zeros(f_cor64.shape[:2], dtype=torch.bool, device=f_cor64.device)
    for b_i, i, j in amb.nonzero().tolist():
        rows[b_i, i] = rows[b_i, j] = True
    return rows


def check_grad(what, got, ref64, ref32, f_cor64, mask):
    """The gradient gate, with the rows of sign-ambiguous masked entries checked for magnitude only (count printed)."""
    rows = ambiguous_rows(f_cor64, mask)
    keep = ~rows[:, :, None, None].expand_as(ref64)
    amax = float(ref64.abs().max())
    got = got.detach().double()
    check(what, torch.where(keep, got, ref64), ref64, GRAD_RTOL, GRAD_ATOL * amax, torch.where(keep, ref32.double(), ref64))
    if bool((~keep).any()):
        assert float((got - ref64)[~keep].abs().max()) <= 4 * amax
    print(f"{what}: {int(rows.sum())} channel rows with a sign-ambiguous masked covariance entry")


@pytest.mark.parametrize("arm,tc,fractional", [("exact", 1, False), ("general", 1, True), ("simt", 0, False)])
def test_clamp_splits_one_batch(arm, tc, fractional, monkeypatch):
    """A margin between the samples' masked sums: the samples below it are clamped (loss term 0, gradient exactly 0),
    the others follow fp64."""
    monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", str(tc))
    shape = (6, 64, 16, 16)
    c = shape[1]
    x = correlated_map(shape, seed=41, scales=[0.2, 1.2, 0.4, 1.0, 0.6, 0.8])
    mask = (fractional_mask if fractional else binary_mask)(c, seed=42)
    eye = torch.eye(c)
    f64, _ = isw_oracle.covariance(x.double(), eye.double())
    off0 = (f64 * mask.double()).abs().sum((1, 2))
    srt = off0.sort().values
    margin = float((srt[2] + srt[3]) / 2)
    assert float((off0 - margin).abs().min()) > 1e-2 * margin, "the margin must sit far from every sample's sum"
    clamped = off0 < margin
    assert int(clamped.sum()) == 3
    nr = float(mask.sum())

    xd = x.to(DEV).requires_grad_(True)
    loss = instance_whitening_loss(xd, eye.to(DEV), mask.to(DEV), margin, nr)
    (UPSTREAM * loss).backward()
    l64, g64 = oracle_grad(x, eye, mask, margin, nr)
    l32, g32 = oracle_grad(x, eye, mask, margin, nr, dtype=torch.float32)
    check(f"{arm}: loss", loss, l64, LOSS_RTOL, 0, l32)
    got = xd.grad.cpu()
    assert bool((got[clamped] == 0).all()), f"{arm}: a clamped sample has a nonzero gradient"
    assert bool((got[~clamped] != 0).any())
    check_grad(f"{arm}: gradient", got, g64, g32, f64, mask)


def test_sample_on_the_clamp_boundary_keeps_its_gradient():
    """margin = the kernel's own off[b] puts sample b at exactly 0: its loss term is 0, and the gate (off / n >= 0) stays
    open, as torch's clamp passes the gradient at the boundary -- its gradient is the margin-0 gradient bit for bit.
    margin and num_remove_cov as Python numbers, fp32 and fp64 0-dim tensors give the same bits."""
    shape = (5, 64, 16, 16)
    b, c, h, w = shape
    hw = h * w
    xd = correlated_map(shape, seed=51, scales=[0.3, 0.9, 0.5, 1.1, 0.7]).to(DEV)
    mask = binary_mask(c, seed=52).to(DEV)
    eye = torch.eye(c, device=DEV)
    nr = float(mask.sum())
    f_cor, _ = get_covariance_matrix(xd, eye)
    nr_t = torch.full((1,), nr, device=DEV)
    _, off, _ = loss_forward_abi(f_cor, mask, torch.zeros(1, device=DEV), nr_t, hw)
    bstar = int(off.argsort()[2])                         # the median sample: two below it, two above
    m = off[bstar].reshape(1)
    _, off_m, _ = loss_forward_abi(f_cor, mask, m, nr_t, hw)
    assert float(off_m[bstar]) == 0.0, "margin = off[b] must put sample b at exactly 0"
    below = off < m

    def run(margin, num):
        xk = xd.clone().requires_grad_(True)
        loss = instance_whitening_loss(xk, eye, mask, margin, num)
        (UPSTREAM * loss).backward()
        return loss.detach(), xk.grad

    _, g0 = run(0.0, nr)
    mv = float(m)
    runs = [run(margin, num) for margin, num in
            ((mv, nr),
             (torch.tensor(mv, dtype=torch.float32, device=DEV), torch.tensor(nr, dtype=torch.float32, device=DEV)),
             (torch.tensor(mv, dtype=torch.float64, device=DEV), torch.tensor(nr, dtype=torch.float64, device=DEV)))]
    for i, (l, g) in enumerate(runs[1:], 1):
        assert_same_bits(l.reshape(1), runs[0][0].reshape(1), f"loss, scalar form {i} vs Python numbers")
        assert_same_bits(g, runs[0][1], f"gradient, scalar form {i} vs Python numbers")
    loss, g = runs[0]
    assert_same_bits(g[bstar], g0[bstar], "the boundary sample's gradient vs its margin-0 gradient")
    assert bool((g[below] == 0).all()) and bool((g[~below] != 0).any())
    l64, g64 = oracle_grad(xd, eye, mask, mv, nr)
    check("boundary: loss", loss, l64, LOSS_RTOL, 0)
    open_ = ~below
    open_[bstar] = False          # fp64 puts the boundary sample a hair to either side; checked bit for bit above
    _, g32 = oracle_grad(xd, eye, mask, mv, nr, dtype=torch.float32)
    f64, _ = isw_oracle.covariance(xd.double(), eye.double())
    check_grad("boundary: gradient of the open samples", g[open_], g64[open_], g32[open_], f64[open_], mask)


# ========================================================================================= 4. backward arms
def general_s(f_cor, mask, off, nr, grad, hw):
    """S of isw_loss_grad_kernel (general form) in the kernel's fp32 arithmetic, with 1-element CUDA tensors so that
    every division is a true division: scale = g * gate / (nr * B) / (hw - 1); S = scale * (T + T^T)."""
    b = f_cor.shape[0]
    v = f_cor * mask
    t = torch.where(v > 0, 1.0, torch.where(v < 0, -1.0, 0.0)) * mask      # sgn(-0) = +0, as in the kernel
    t = t + t.transpose(1, 2)
    one = torch.ones(1, device=DEV)
    gate = torch.where(off / nr >= 0, 1.0, 0.0)
    scale = grad * gate / (nr * (b * one)) / ((hw - 1) * one)
    return (scale.view(b, 1, 1) * t).contiguous()


def sx_tc(s, x):
    b, c, hw = x.shape
    dx = torch.full((b, c, hw), float("nan"), device=DEV)
    rc = lib().dgvcc_isw_sx_tc(P(s), P(x), b, c, hw, P(dx), stream())
    torch.cuda.synchronize()
    return rc, dx


def misaligned_copy(x):
    """The same values 4 bytes past a 16-byte boundary (a contiguous view at storage offset 1)."""
    buf = torch.empty(x.numel() + 1, device=DEV)
    buf[1:] = x.reshape(-1)
    v = buf[1:].view(x.shape)
    assert v.is_contiguous() and v.data_ptr() % 16 != 0
    return v


# (arm, (B, C, H, W), mask kind, DGVCC_ISW_TENSOR_CORES, misaligned map)
LOSS_BWD_CASES = [
    ("exact", (3, 64, 16, 16), "binary", 1, False),
    ("exact", (2, 200, 12, 20), "binary", 1, False),
    ("general", (3, 64, 16, 16), "fractional", 1, False),
    ("general", (2, 200, 12, 20), "fractional", 1, False),
    ("simt-tc-off", (3, 64, 16, 16), "binary", 0, False),
    ("simt-tc-off", (3, 64, 16, 16), "fractional", 0, False),
    ("simt-c%4", (3, 50, 16, 16), "binary", 1, False),
    ("simt-hw%4", (3, 64, 9, 15), "binary", 1, False),
    ("simt-misaligned", (3, 64, 16, 16), "binary", 1, True),
]


def _bwd_id(case):
    arm, (b, c, h, w), kind, tc, _ = case
    return f"{arm}-{kind}-c{c}-hw{h * w}"


@pytest.mark.parametrize("case", LOSS_BWD_CASES, ids=_bwd_id)
def test_loss_backward_arm_against_fp64(case, monkeypatch):
    arm, shape, kind, tc, misaligned = case
    monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", str(tc))
    b, c, h, w = shape
    hw = h * w
    x = correlated_map(shape, seed=hw + 3 * c)
    mask = (binary_mask if kind == "binary" else fractional_mask)(c, seed=c + 5)
    eye = torch.eye(c)
    xd = x.to(DEV)
    if misaligned:
        xd = misaligned_copy(xd)
    dx_probe = torch.empty_like(xd)
    tiles = sx_tc_tiles(c, hw, xd, dx_probe)
    expect = {"exact": tiles and tc and mask_is_binary(mask), "general": tiles and tc and not mask_is_binary(mask)}
    assert expect.get(arm, not (tiles and tc)), f"{arm}: the host predicates pick another arm"

    xk = xd.detach().clone() if not misaligned else misaligned_copy(xd)
    xk.requires_grad_(True)
    md, nr = mask.to(DEV), float(mask.sum())
    loss = instance_whitening_loss(xk, eye.to(DEV), md, 0, nr)
    (UPSTREAM * loss).backward()
    got = xk.grad

    l64, g64 = oracle_grad(x, eye, mask, 0, nr)
    l32, g32 = oracle_grad(x, eye, mask, 0, nr, dtype=torch.float32)
    f64, _ = isw_oracle.covariance(x.double(), eye.double())
    check(f"{arm}: loss", loss, l64, LOSS_RTOL, 0, l32)
    check_grad(f"{arm}: gradient", got.cpu(), g64, g32, f64, mask)

    x3 = xd.detach().reshape(b, c, hw)
    if arm == "general":
        f_cor, _ = get_covariance_matrix(xd, eye.to(DEV))
        nr_t = torch.full((1,), nr, device=DEV)
        _, off, _ = loss_forward_abi(f_cor, md, torch.zeros(1, device=DEV), nr_t, hw)
        s = general_s(f_cor, md, off, nr_t, torch.full((1,), UPSTREAM, device=DEV), hw)
        rc, want = sx_tc(s, x3.contiguous())
        assert rc == 0
        assert_same_bits(got.reshape(b, c, hw), want, f"{arm}: loss backward vs dgvcc_isw_sx_tc(S built by torch, X)")
    if tc:
        rc, _ = sx_tc(torch.zeros((b, c, c), device=DEV), x3)
        if arm.startswith("simt"):
            assert rc == UNSUPPORTED, f"{arm}: dgvcc_isw_sx_tc took a shape meant for the SIMT GEMM"
        else:
            assert rc == 0, f"{arm}: dgvcc_isw_sx_tc refused the shape, so the launcher fell back to the SIMT GEMM"
    if arm.startswith("simt"):
        # the SIMT arms give the bits of the aligned map with the tensor cores off
        monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", "0")
        xa = x.to(DEV).requires_grad_(True)
        (UPSTREAM * instance_whitening_loss(xa, eye.to(DEV), md, 0, nr)).backward()
        assert_same_bits(got, xa.grad, f"{arm}: gradient vs the aligned map with the tensor cores off")


# (arm, (B, C, H, W), DGVCC_ISW_TENSOR_CORES)
COV_BWD_CASES = [
    ("general", (3, 64, 16, 16), 1),
    ("general", (2, 200, 12, 20), 1),
    ("simt-tc-off", (3, 64, 16, 16), 0),
    ("simt-c%4", (3, 50, 16, 16), 1),
    ("simt-hw%4", (3, 64, 9, 15), 1),
]


@pytest.mark.parametrize("case", COV_BWD_CASES, ids=[f"{a}-c{s[1]}-hw{s[2] * s[3]}" for a, s, _ in COV_BWD_CASES])
def test_covariance_backward_arm_against_fp64(case, monkeypatch):
    arm, shape, tc = case
    monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", str(tc))
    b, c, h, w = shape
    hw = h * w
    x = correlated_map(shape, seed=hw + 5 * c)
    up = torch.randn((b, c, c), generator=torch.Generator().manual_seed(c))
    eye = torch.eye(c)
    xd = x.to(DEV)
    tiles = sx_tc_tiles(c, hw, xd, xd)
    assert (arm == "general") == bool(tiles and tc), f"{arm}: the host predicates pick another arm"
    xk = xd.clone().requires_grad_(True)
    f_cor, _ = get_covariance_matrix(xk, eye.to(DEV))
    (f_cor * up.to(DEV)).sum().backward()

    refs = {}
    for dt in (torch.float64, torch.float32):
        xr = x.to(dt).requires_grad_(True)
        fr, _ = isw_oracle.covariance(xr, eye.to(dt))
        (fr * up.to(dt)).sum().backward()
        refs[dt] = (fr.detach(), xr.grad)
    f64, g64 = refs[torch.float64]
    check(f"{arm}: f_cor", f_cor.cpu(), f64, COV_RTOL, COV_ATOL * float(f64.abs().max()), refs[torch.float32][0])
    check(f"{arm}: gradient", xk.grad.cpu(), g64, GRAD_RTOL, GRAD_ATOL * float(g64.abs().max()), refs[torch.float32][1])

    x3 = xd.reshape(b, c, hw)
    d = up.to(DEV)
    s = ((d + d.transpose(1, 2)) / torch.full_like(d, hw - 1)).contiguous()   # isw_cov_grad_kernel
    rc, want = sx_tc(s, x3)
    if arm == "general":
        assert rc == 0
        assert_same_bits(xk.grad.reshape(b, c, hw), want, f"{arm}: covariance backward vs dgvcc_isw_sx_tc(S, X)")
    else:
        if tc:
            assert rc == UNSUPPORTED, f"{arm}: dgvcc_isw_sx_tc took a shape meant for the SIMT GEMM"
        monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", "0")
        xa = xd.clone().requires_grad_(True)
        fa, _ = get_covariance_matrix(xa, eye.to(DEV))
        (fa * d).sum().backward()
        assert_same_bits(xk.grad, xa.grad, f"{arm}: gradient vs the tensor cores off")


# ========================================================================================= 5. half route vs fp64
HALF_SHAPES = [
    (7, 32, 24, 24), (5, 64, 16, 40), (4, 128, 16, 16), (3, 192, 16, 24), (2, 256, 32, 32), (2, 512, 16, 16),
    (3, 100, 24, 23), (8, 512, 16, 32), (8, 512, 17, 32), (8, 512, 32, 32), (8, 512, 34, 32), (8, 512, 28, 38),
    (8, 64, 160, 160), (8, 256, 80, 80), (8, 512, 40, 40),
]


@functools.lru_cache(maxsize=4)
def _half_input(shape, dtype):
    return correlated_map(shape, seed=sum(shape)).to(dtype).to(DEV)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["f16", "bf16"])
@pytest.mark.parametrize("shape", HALF_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_half_route_against_fp64(shape, dtype):
    """The native route restated in fp64 stage by stage, each stage fed the kernels' own half output of the one before:
    y = RN(instance_norm(x)); the loss and its gradient dL/dy on that y (0/1 and fractional masks); dx = RN(instance
    norm backward(dL/dy)); f_cor and its backward for a random upstream gradient.  The module's x.grad is the
    composition of the stages bit for bit."""
    b, c, h, w = shape
    hw = h * w
    x = _half_input(shape, dtype)
    assert half_tc_tiles(c, hw, x, torch.empty_like(x)), "a TILED shape the half route does not tile"
    dn = _dt(dtype)
    eye = torch.eye(c, device=DEV)

    # instance norm forward
    y, _ = InstanceWhitening(c)(x)
    y64 = F.instance_norm(x.double(), eps=EPS)
    check(f"{dn} y", y, y64, NORM_RTOL, NORM_ATOL, F.instance_norm(x.float(), eps=EPS), dtype)

    # loss and dL/dy on the half y, both masks
    y64r = y.double()
    f64, _ = isw_oracle.covariance(y64r, eye.double())
    for kind, make in (("binary", binary_mask), ("fractional", fractional_mask)):
        mask = make(c, seed=c + 11).to(DEV)
        nr = float(mask.sum())
        yk = y.detach().clone().requires_grad_(True)
        loss = instance_whitening_loss(yk, eye, mask, 0, nr)
        (UPSTREAM * loss).backward()
        assert yk.grad.dtype == dtype
        l64, g64 = oracle_grad(y64r, eye, mask, 0, nr)
        l32, g32 = oracle_grad(y64r, eye, mask, 0, nr, dtype=torch.float32)
        check(f"{dn} {kind}: loss", loss, l64, LOSS_RTOL, 0, l32)
        rows = ambiguous_rows(f64, mask)
        keep = ~rows[:, :, None, None].expand_as(g64)
        got = yk.grad.double()
        check(f"{dn} {kind}: dL/dy", torch.where(keep, got, g64), g64, GRAD_RTOL, GRAD_ATOL * float(g64.abs().max()),
              torch.where(keep, g32.double(), g64), dtype)
        print(f"{dn} {kind}: {int(rows.sum())} channel rows with a sign-ambiguous masked covariance entry")
        if kind == "binary":
            dy = yk.grad

    # instance norm backward fed the kernels' half dL/dy, and the module end to end
    xk = x.clone().requires_grad_(True)
    yk, _ = InstanceWhitening(c)(xk)
    yk.backward(dy)
    x64 = x.double().requires_grad_(True)
    F.instance_norm(x64, eps=EPS).backward(dy.double())
    x32 = x.float().requires_grad_(True)
    F.instance_norm(x32, eps=EPS).backward(dy.float())
    check(f"{dn} dx", xk.grad, x64.grad, GRAD_RTOL, GRAD_ATOL * x64.grad.abs().amax((2, 3), keepdim=True), x32.grad,
          dtype)
    mask = binary_mask(c, seed=c + 11).to(DEV)
    xm = x.clone().requires_grad_(True)
    (UPSTREAM * instance_whitening_loss(InstanceWhitening(c)(xm)[1], eye, mask, 0, float(mask.sum()))).backward()
    assert_same_bits(xm.grad, xk.grad, f"{dn}: module x.grad vs the composition of the stages")

    # covariance and its backward on the half map
    up = torch.randn((b, c, c), generator=torch.Generator().manual_seed(c)).to(DEV)
    xc = x.clone().requires_grad_(True)
    f_cor, _ = get_covariance_matrix(xc, eye)
    (f_cor * up).sum().backward()
    xr = x.double().requires_grad_(True)
    fr, _ = isw_oracle.covariance(xr, eye.double())
    (fr * up.double()).sum().backward()
    f32, _ = isw_oracle.covariance(x.float(), eye)
    check(f"{dn} f_cor", f_cor, fr.detach(), COV_RTOL, COV_ATOL * float(fr.abs().max()), f32)
    check(f"{dn} covariance dx", xc.grad, xr.grad, GRAD_RTOL, GRAD_ATOL * float(xr.grad.abs().max()), None, dtype)
