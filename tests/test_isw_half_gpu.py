"""fp16 / bf16 feature maps through the ISW path (InstanceWhitening, get_covariance_matrix, instance_whitening_loss).

The native half path must give exactly what the fp32 path gives on the upcast map -- torch.equal on y, f_cor, the loss
and the gradient into x.  "The fp32 path on the upcast map" is restated with explicit casts: x.float() into the fp32
modules, y rounded to the input dtype, then .float() into the loss; autograd's cast nodes round the gradients where
the upcast route of the modules does.  The reasons the bits agree are in DESIGN section 5 (half-precision input): a
finite half value is its own TF32 hi part and its lo part is 0, so every dropped MMA adds exact zeros.
"""
import gc

import pytest
import torch

from dgvcc_b200 import _native
from dgvcc_b200.models.ISW import InstanceWhitening, get_covariance_matrix, instance_whitening_loss

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
DTYPES = [torch.float16, torch.bfloat16]
CODE = {torch.float16: _native.DTYPE_F16, torch.bfloat16: _native.DTYPE_BF16}
UNSUPPORTED, ERR_ARG = -3, -1


def cdiv(a, b):
    return -(-a // b)


def gram_plan_tc(batch, c, hw):
    """gram_plan_tc (isw_kernels.cu) restated: k blocks on the first split's CTA."""
    pair = c <= 64
    t1 = 1 if pair else cdiv(c, 128)
    units = (cdiv(batch, 2) if pair else batch) * t1 * (t1 + 1) // 2
    s = 0 if units > 148 else 148 // units
    s = max(1, min(s, cdiv(hw, 256)))
    kps = cdiv(cdiv(hw, s), 32) * 32
    return cdiv(min(kps, hw), 32)


# shapes the half tensor-core kernels tile: (B, C, H, W)
TILED = [
    (7, 32, 24, 24),     # pair mode, odd batch
    (5, 64, 16, 40),     # pair mode, odd batch
    (4, 128, 16, 16),
    (3, 192, 16, 24),    # partial second row tile
    (2, 256, 32, 32),
    (2, 512, 16, 16),
    (3, 100, 24, 23),    # partial tile, last k block of 8 (552 = 17 * 32 + 8), partial n tile of S X
    (8, 512, 16, 32),    # 16 k blocks on one CTA: exactly one TMEM segment
    (8, 512, 17, 32),    # 17: a second segment of one k block
    (8, 512, 32, 32),    # 32: two full segments
    (8, 512, 34, 32),    # 34: three segments
    (8, 512, 28, 38),    # 34 with a partial last k block (1064 = 33 * 32 + 8)
]
CONFIG5 = [(8, 64, 160, 160), (8, 256, 80, 80), (8, 512, 40, 40)]
KBLOCKS = {(8, 512, 16, 32): 16, (8, 512, 17, 32): 17, (8, 512, 32, 32): 32, (8, 512, 34, 32): 34, (8, 512, 28, 38): 34}
# shapes they do not tile (the upcast route runs them)
UNTILED = [(2, 48, 12, 13), (4, 16, 16, 16), (3, 50, 16, 16)]   # HW % 8 == 4, C = 16, C % 4 != 0


def sid(shape):
    return "x".join(map(str, shape))


def make_input(shape, dtype, kind, seed=0):
    g = torch.Generator().manual_seed(seed)
    b, c, h, w = shape
    x = torch.randn(shape, generator=g)
    if kind == "wide":
        # magnitudes from subnormal to near the top of the range, one all-zero channel
        top = 6.0e4 if dtype is torch.float16 else 1.0e15
        e = torch.randint(0, 4, shape, generator=g)
        x = torch.where(e == 0, x * 1e-7, torch.where(e == 1, x.clamp(-1, 1) * top, torch.where(e == 2, x * 1e3, x)))
        x[:, c // 2] = 0
    return x.to(dtype).to(DEV)


def make_mask(c, fractional, seed=1):
    g = torch.Generator().manual_seed(seed)
    m = (torch.rand(c, c, generator=g) < 0.5).float()
    if fractional:
        m = m * torch.rand(c, c, generator=g)
    return m.triu(1).to(DEV)


def module_step(x, mask, restated):
    """InstanceWhitening + instance_whitening_loss, forward and backward: (y, loss, x.grad)."""
    c = x.shape[1]
    eye = torch.eye(c, device=DEV)
    x = x.detach().clone().requires_grad_(True)
    if restated:
        y32, _ = InstanceWhitening(c)(x.float())
        y = y32.to(x.dtype)
        loss = instance_whitening_loss(y.float(), eye, mask, 0, mask.sum())
    else:
        y, w = InstanceWhitening(c)(x)
        assert y is w and y.dtype is x.dtype
        loss = instance_whitening_loss(w, eye, mask, 0, mask.sum())
    loss.backward()
    return y.detach(), loss.detach(), x.grad


def covariance_step(x, restated):
    """get_covariance_matrix forward and backward (upstream gradient: a fixed random matrix): (f_cor, B, x.grad)."""
    c = x.shape[1]
    wgt = torch.randn(c, c, generator=torch.Generator().manual_seed(3)).to(DEV)
    x = x.detach().clone().requires_grad_(True)
    f_cor, b = get_covariance_matrix(x.float() if restated else x)
    (f_cor * wgt).sum().backward()
    return f_cor.detach(), b, x.grad


def loss_step(x, mask, restated):
    c = x.shape[1]
    x = x.detach().clone().requires_grad_(True)
    loss = instance_whitening_loss(x.float() if restated else x, torch.eye(c, device=DEV), mask, 0, mask.sum())
    loss.backward()
    return loss.detach(), x.grad


def assert_all_equal(got, ref):
    for i, (g, r) in enumerate(zip(got, ref)):
        if torch.is_tensor(r):
            assert g.dtype == r.dtype and g.shape == r.shape, i
            assert torch.equal(g, r), f"output {i}: max |diff| {(g.float() - r.float()).abs().max().item()}"
        else:
            assert g == r


def check_value_identity(x, fractional):
    mask = make_mask(x.shape[1], fractional)
    got = module_step(x, mask, False)
    assert got[0].dtype == x.dtype and got[1].dtype == torch.float32 and got[2].dtype == x.dtype
    assert_all_equal(got, module_step(x, mask, True))
    got = covariance_step(x, False)
    assert got[0].dtype == torch.float32 and got[2].dtype == x.dtype
    assert_all_equal(got, covariance_step(x, True))
    assert_all_equal(loss_step(x, mask, False), loss_step(x, mask, True))


def abi_codes(x, dtype_code=None, fractional=False):
    """Return codes of dgvcc_isw_covariance_h, dgvcc_isw_loss_backward_h and dgvcc_isw_covariance_backward_h on x
    ([B, C, HW] view, any alignment)."""
    lib = _native.lib()
    b, c, hw = x.shape
    code = CODE[x.dtype] if dtype_code is None else dtype_code
    n = lib.dgvcc_isw_workspace_bytes(b, c, hw)
    ws = torch.empty((n,), dtype=torch.uint8, device=DEV)
    f_cor = torch.zeros((b, c, c), device=DEV)
    eye, mask = torch.eye(c, device=DEV), make_mask(c, fractional)
    one, nr = torch.ones(1, device=DEV), mask.sum().reshape(1)
    dx = torch.empty((b, c, hw), dtype=x.dtype, device=DEV)
    st = _native.stream_ptr(DEV)
    p = _native.ptr
    rc_cov = lib.dgvcc_isw_covariance_h(p(x), code, p(eye), b, c, hw, p(ws), n, p(f_cor), st)
    if rc_cov == 0:
        loss = torch.empty(1, device=DEV)
        zero = torch.zeros(1, device=DEV)
        assert lib.dgvcc_isw_loss_forward(p(f_cor), p(mask), p(zero), p(nr), b, c, hw, p(ws), n, p(loss), st) == 0
    rc_loss = lib.dgvcc_isw_loss_backward_h(p(x), code, p(f_cor), p(mask), p(nr), p(one), b, c, hw, int(not fractional),
                                            p(ws), n, p(dx), st)
    rc_covb = lib.dgvcc_isw_covariance_backward_h(p(x), code, p(f_cor), b, c, hw, p(ws), n, p(dx), st)
    torch.cuda.synchronize()
    return rc_cov, rc_loss, rc_covb


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
@pytest.mark.parametrize("shape", TILED + CONFIG5, ids=sid)
def test_value_identity_on_tiled_shapes(shape, dtype):
    if shape in KBLOCKS:
        assert gram_plan_tc(shape[0], shape[1], shape[2] * shape[3]) == KBLOCKS[shape]
    x = make_input(shape, dtype, "normal")
    b, c, h, w = shape
    for fractional in (False, True):
        assert abi_codes(x.view(b, c, h * w), fractional=fractional) == (0, 0, 0)
    check_value_identity(x, fractional=False)
    check_value_identity(x, fractional=True)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
@pytest.mark.parametrize("shape", [(5, 64, 16, 40), (3, 192, 16, 24), (8, 512, 28, 38), (8, 64, 160, 160)], ids=sid)
def test_value_identity_on_wide_range_data(shape, dtype):
    x = make_input(shape, dtype, "wide")
    assert torch.isfinite(x).all()
    check_value_identity(x, fractional=False)
    check_value_identity(x, fractional=True)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
@pytest.mark.parametrize("shape", UNTILED, ids=sid)
def test_untiled_shapes_are_refused_and_match_through_the_upcast_route(shape, dtype):
    x = make_input(shape, dtype, "normal")
    b, c, h, w = shape
    assert abi_codes(x.view(b, c, h * w)) == (UNSUPPORTED,) * 3
    check_value_identity(x, fractional=False)
    check_value_identity(x, fractional=True)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
def test_misaligned_map_is_refused_and_matches_through_the_upcast_route(dtype):
    shape = (2, 64, 16, 16)
    n = 2 * 64 * 256
    buf = make_input((1, 1, 1, n + 1), dtype, "normal").view(-1)
    x = buf[1:].view(shape)                  # contiguous, 2 bytes past a 16-byte boundary
    assert x.is_contiguous() and x.data_ptr() % 16 != 0
    assert abi_codes(x.view(2, 64, 256)) == (UNSUPPORTED,) * 3
    mask = make_mask(64, False)
    assert_all_equal(covariance_step(x, False), covariance_step(x, True))
    assert_all_equal(loss_step(x, mask, False), loss_step(x, mask, True))


def test_bad_dtype_code_is_an_argument_error():
    x = make_input((2, 64, 16, 16), torch.float16, "normal")
    for code in (0, 3, -1):
        assert abi_codes(x.view(2, 64, 256), dtype_code=code) == (ERR_ARG,) * 3
    lib = _native.lib()
    mean = torch.empty(128, device=DEV)
    y = torch.empty_like(x)
    st, p = _native.stream_ptr(DEV), _native.ptr
    assert lib.dgvcc_isw_instnorm_forward_h(p(x), 3, 128, 256, 1e-5, p(y), p(mean), p(mean), st) == ERR_ARG
    assert lib.dgvcc_isw_instnorm_backward_h(p(x), p(x), p(mean), p(mean), 0, 128, 256, p(y), st) == ERR_ARG


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
def test_tensor_cores_off_takes_the_upcast_route(dtype, monkeypatch):
    monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", "0")
    x = make_input((3, 128, 16, 16), dtype, "normal")
    check_value_identity(x, fractional=False)


def held_after_forward(fn):
    gc.collect()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(DEV)
    out = fn()
    torch.cuda.synchronize()
    held = torch.cuda.memory_allocated(DEV) - base
    del out
    return held


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
def test_native_step_holds_less_memory_after_forward(dtype):
    shape = (8, 64, 160, 160)
    x = make_input(shape, dtype, "normal").requires_grad_(True)
    c = shape[1]
    mask, eye = make_mask(c, False), torch.eye(c, device=DEV)
    nr = mask.sum()
    iw = InstanceWhitening(c)

    def native():
        return instance_whitening_loss(iw(x)[1], eye, mask, 0, nr)

    def restated():
        return instance_whitening_loss(iw(x.float())[1].to(dtype).float(), eye, mask, 0, nr)

    for _ in range(2):   # warm the allocator and the cached workspace sizes
        held_after_forward(native), held_after_forward(restated)
    h_native, h_restated = held_after_forward(native), held_after_forward(restated)
    assert h_restated - h_native >= 5 * x.numel(), (h_native, h_restated)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
@pytest.mark.parametrize("shape", [(4, 64, 32, 32), (2, 256, 16, 16)], ids=sid)
def test_half_module_step_replays_as_a_cuda_graph(shape, dtype):
    b, c, h, w = shape
    xs = [make_input(shape, dtype, "normal", seed=s) for s in range(3)]
    mask = make_mask(c, False)
    eye, nrm = torch.eye(c, device=DEV), mask.sum()
    iw = InstanceWhitening(c)

    def step(x):
        _, wt = iw(x)
        loss = instance_whitening_loss(wt, eye, mask, 0, nrm)
        loss.backward()
        return loss

    eager = []
    for x in xs:
        xe = x.clone().requires_grad_(True)
        eager.append((step(xe).detach().clone(), xe.grad.clone()))
    static = xs[0].clone().requires_grad_(True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            static.grad = None
            step(static)
    torch.cuda.current_stream().wait_stream(side)
    static.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_loss = step(static)
    for x, (l_ref, g_ref) in zip(xs, eager):
        with torch.no_grad():
            static.copy_(x)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(static_loss.detach(), l_ref) and torch.equal(static.grad, g_ref)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
def test_channels_last_input_gives_the_bits_of_its_contiguous_copy(dtype):
    x = make_input((4, 128, 16, 24), dtype, "normal")
    xcl = x.to(memory_format=torch.channels_last)
    assert not xcl.is_contiguous()
    mask = make_mask(128, False)
    assert_all_equal(module_step(xcl, mask, False), module_step(x, mask, False))
    assert_all_equal(covariance_step(xcl, False), covariance_step(x, False))
    assert_all_equal(loss_step(xcl, mask, False), loss_step(x, mask, False))


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
def test_two_runs_give_the_same_bits(dtype):
    x = make_input((8, 256, 40, 40), dtype, "normal")
    for fractional in (False, True):
        mask = make_mask(256, fractional)
        assert_all_equal(module_step(x, mask, False), module_step(x, mask, False))


def same_with_nan(a, b):
    return a.dtype == b.dtype and torch.allclose(a.float(), b.float(), rtol=0, atol=0, equal_nan=True)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
def test_inf_pixel_behaves_like_the_upcast_route(dtype):
    """An inf pixel makes its sample's covariance row non-finite, so that sample's sum |f_cor * mask| is NaN (inf times a
    zero of the mask).  The fp32 loss clamp (max(NaN, 0) = 0, unchanged here) then drops the sample and closes its
    gradient gate, in the upcast route and the native route alike: the loss is the finite loss of the other samples, the
    other samples' gradients are untouched, and the affected sample's gradient is non-finite (0 * inf in dX = S X)."""
    x = make_input((2, 64, 16, 16), dtype, "normal")
    x[1, 5, 3, 7] = float("inf")
    mask = make_mask(64, False)
    for run in (lambda r: module_step(x, mask, r)[1:], lambda r: loss_step(x, mask, r)):
        (loss, grad), (loss_ref, grad_ref) = run(False), run(True)
        assert torch.equal(loss, loss_ref)
        assert torch.equal(grad[0], grad_ref[0]) and torch.isfinite(grad[0]).all()
        assert not torch.isfinite(grad[1]).all() and not torch.isfinite(grad_ref[1]).all()


def test_overflowing_bf16_map_gives_a_non_finite_loss():
    """A finite bf16 map whose Gram overflows fp32 gives an infinite f_cor and, with a mask without zeros, an infinite
    loss -- in both routes, bit for bit."""
    x = (torch.rand((2, 32, 8, 8), generator=torch.Generator().manual_seed(4)) + 1).mul(1e20).to(torch.bfloat16).to(DEV)
    mask = torch.ones(32, 32, device=DEV)
    (loss, grad), (loss_ref, grad_ref) = loss_step(x, mask, False), loss_step(x, mask, True)
    assert torch.isinf(loss) and torch.equal(loss, loss_ref) and same_with_nan(grad, grad_ref)
