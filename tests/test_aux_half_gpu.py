"""fp16 / bf16 inputs through lw_loss and ortho_loss.

The native half route must give exactly what the fp32 route gives on the upcast input: torch.equal on the loss and on
the gradient, which the upcast route rounds to the input dtype.  The native lw_loss never materialises the standardised
map: the Gram and dY = S Y standardise the half map as they load it (DESIGN section 5b, f4), so the kernel arms are also
checked one by one against the fp32 entry points on the materialised map.
"""
import pytest
import torch

from dgvcc_b200 import _native
from dgvcc_b200.losses.lw import lw_loss
from dgvcc_b200.losses.ortho import ortho_loss

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
DTYPES = [torch.float16, torch.bfloat16]
DT_IDS = ["f16", "bf16"]
CODE = {torch.float16: _native.DTYPE_F16, torch.bfloat16: _native.DTYPE_BF16}
UNSUPPORTED = -3
P = _native.ptr


def sid(shape):
    return "x".join(map(str, shape))


# (B, C, H, W) shapes the half tensor-core kernels tile
TILED = [
    (1, 32, 16, 16), (3, 32, 16, 16),    # pair mode, the second sample of the last pair missing
    (1, 48, 16, 16), (3, 48, 12, 16),    # pair mode, rows 48-63 of each half zero-filled
    (1, 64, 16, 16), (3, 64, 16, 24),
    (2, 96, 16, 24),                     # a partial 128-row tile
    (2, 192, 16, 24),                    # a partial second row tile: off-diagonal tiles
    (2, 128, 64, 64),                    # split-K over 16 CTAs
    (8, 512, 16, 32),                    # 16 k blocks on one CTA: exactly one TMEM segment (SEG_KB)
    (8, 512, 17, 32),                    # 17: a second segment of one k block
    (8, 512, 32, 32),                    # 32: two full segments
    (8, 512, 34, 32),                    # 34: three segments
    (2, 64, 8, 13),                      # HW = 104: a partial last k block of 8
    (3, 100, 24, 23),                    # C % 128 = 100, HW = 552 = 17 * 32 + 8
]
CONFIG5 = [(8, 64, 160, 160), (8, 256, 80, 80), (8, 512, 40, 40)]
MASKS = ["none", "binary", "soft"]


def make_x(shape, dtype, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(shape, generator=g) * 1.5 + 0.3).to(dtype).to(DEV)


def make_mask(shape, kind, seed=1):
    if kind == "none":
        return None
    b, _, h, w = shape
    g = torch.Generator().manual_seed(seed)
    m = torch.rand((b, 1, h, w), generator=g)
    return ((m < 0.6).float() if kind == "binary" else m).to(DEV)


def same(a, b):
    """torch.equal, with NaN equal to NaN."""
    return a.dtype == b.dtype and a.shape == b.shape and torch.allclose(a.float(), b.float(), rtol=0, atol=0, equal_nan=True)


def lw_cast_route(x, mask):
    xr = x.detach().float().requires_grad_(True)
    loss = lw_loss(xr, mask)
    loss.backward()
    return loss.detach(), xr.grad.to(x.dtype)


def lw_native(x, mask):
    xn = x.detach().requires_grad_(True)   # the same storage: a misaligned view stays misaligned
    loss = lw_loss(xn, mask)
    route = loss.grad_fn.half
    loss.backward()
    return loss.detach(), xn.grad, route


def check_lw(x, mask, expect_native=True):
    l_ref, g_ref = lw_cast_route(x, mask)
    l, g, route = lw_native(x, mask)
    assert route == (CODE[x.dtype] if expect_native else None)
    assert l.dtype == torch.float32 and g.dtype == x.dtype
    assert same(l, l_ref), (l.item(), l_ref.item())
    assert same(g, g_ref), (g.float() - g_ref.float()).abs().max().item()


@pytest.mark.parametrize("mask", MASKS)
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("shape", TILED, ids=sid)
def test_lw_native_matches_the_cast_route(shape, dtype, mask):
    check_lw(make_x(shape, dtype), make_mask(shape, mask))


@pytest.mark.parametrize("mask", ["none", "soft"])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("shape", CONFIG5, ids=sid)
def test_lw_native_matches_the_cast_route_on_config5_layers(shape, dtype, mask):
    check_lw(make_x(shape, dtype), make_mask(shape, mask))


def extreme_x(shape, dtype, inf_pixel):
    b, c, h, w = shape
    g = torch.Generator().manual_seed(3)
    x = torch.randn(shape, generator=g)
    top = 6.0e4 if dtype is torch.float16 else 1.0e30
    tiny = 1e-7 if dtype is torch.float16 else 1e-39           # subnormal in the type
    x[:, 0] = x[:, 0].clamp(-1, 1) * top                         # extremes of the range
    x[:, 1] = x[:, 1] * tiny                                     # subnormals
    x[:, 2] = 0.75                                               # constant channel: sd = sqrt(eps)
    x[:, 3] = 1e3 + x[:, 3]                                      # mean 1e3
    x = x.to(dtype)
    if inf_pixel:
        x[0, 5, 1, 2] = float("inf")
    return x.to(DEV)


@pytest.mark.parametrize("inf_pixel", [False, True], ids=["finite", "inf"])
@pytest.mark.parametrize("mask", MASKS)
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_lw_extreme_data_matches_the_cast_route(dtype, mask, inf_pixel):
    shape = (3, 64, 16, 24)
    check_lw(extreme_x(shape, dtype, inf_pixel), make_mask(shape, mask))
    shape = (2, 192, 16, 16)
    check_lw(extreme_x(shape, dtype, inf_pixel), make_mask(shape, mask))


# ------------------------------------------------------------------ the kernel arms on their own
def materialised(x, mask):
    """yhat, the Gram input y and invstd from the fp32 standardisation on the upcast map."""
    n, c, h, w = x.shape
    hw = h * w
    xf = x.float().contiguous()
    m = mask.reshape(n, hw).contiguous() if mask is not None else None
    yhat = torch.empty((n, c, hw), device=DEV)
    ym = torch.empty_like(yhat) if m is not None else None
    invstd = torch.empty((n * c,), device=DEV)
    lib = _native.lib()
    _native.check(lib.dgvcc_lw_standardize_forward(P(xf), P(m), n, c, hw, 1e-5, P(yhat), P(ym), P(invstd), None), "fwd")
    return yhat, (ym if m is not None else yhat), invstd, m


@pytest.mark.parametrize("mask", MASKS)
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("shape", [(3, 48, 12, 16), (2, 192, 16, 24), (2, 128, 64, 64), (2, 64, 8, 13)], ids=sid)
def test_kernel_arms_equal_the_fp32_entry_points_on_the_materialised_map(shape, dtype, mask):
    n, c, h, w = shape
    hw = h * w
    lib = _native.lib()
    x = make_x(shape, dtype)
    mk = make_mask(shape, mask)
    yhat, y, invstd_ref, m = materialised(x, mk)
    # statistics
    stats = torch.empty((3, n * c), device=DEV)
    mean, sd, invstd = stats
    assert lib.dgvcc_lw_standardize_stats_h(P(x), CODE[dtype], n, c, hw, 1e-5, P(mean), P(sd), P(invstd), None) == 0
    assert torch.equal(invstd, invstd_ref)
    assert torch.equal((x.float().reshape(n * c, hw) - mean[:, None]) / sd[:, None], yhat.reshape(n * c, hw))
    # Gram
    nbytes = lib.dgvcc_isw_workspace_bytes(n, c, hw)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=DEV)
    g_ref = torch.empty((n, c, c), device=DEV)
    g = torch.empty_like(g_ref)
    assert lib.dgvcc_isw_gram(P(y), n, c, hw, 1, P(ws), nbytes, P(g_ref), None) == 0
    assert lib.dgvcc_lw_gram_h(P(x), CODE[dtype], P(mean), P(sd), P(m), n, c, hw, P(ws), nbytes, P(g), None) == 0
    assert torch.equal(g, g_ref)
    # dY = S Y
    gl = torch.full((1,), 0.37, device=DEV)
    dy_ref = torch.empty((n, c, hw), device=DEV)
    dy = torch.empty_like(dy_ref)
    assert lib.dgvcc_lw_loss_backward(P(y), P(g_ref), P(gl), n, c, hw, 1, P(ws), nbytes, P(dy_ref), None) == 0
    assert lib.dgvcc_lw_loss_backward_h(P(x), CODE[dtype], P(mean), P(sd), P(m), P(g_ref), P(gl), n, c, hw, P(ws), nbytes,
                                        P(dy), None) == 0
    assert torch.equal(dy, dy_ref)
    # standardisation backward
    dx_ref = torch.empty((n, c, hw), device=DEV)
    dx = torch.empty((n, c, hw), dtype=dtype, device=DEV)
    assert lib.dgvcc_lw_standardize_backward(P(dy_ref), P(yhat), P(invstd_ref), P(m), n, c, hw, P(dx_ref), None) == 0
    assert lib.dgvcc_lw_standardize_backward_h(P(dy), P(x), CODE[dtype], P(mean), P(sd), P(invstd), P(m), n, c, hw, P(dx),
                                               None) == 0
    assert torch.equal(dx, dx_ref.to(dtype))


# ------------------------------------------------------------------ fallbacks
UNTILED = [(2, 48, 12, 13), (2, 16, 16, 16), (2, 50, 16, 16)]   # HW % 8 == 4, C < 32, C % 4 != 0


def h_return_codes(x, mask):
    n, c, h, w = x.shape
    hw = h * w
    lib = _native.lib()
    stats = torch.empty((3, n * c), device=DEV)
    nbytes = lib.dgvcc_isw_workspace_bytes(n, c, hw)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=DEV)
    gram = torch.zeros((n, c, c), device=DEV)
    dy = torch.empty((n, c, hw), device=DEV)
    gl = torch.ones((1,), device=DEV)
    m = mask.reshape(n, hw).contiguous() if mask is not None else None
    return (lib.dgvcc_lw_gram_h(P(x), CODE[x.dtype], P(stats[0]), P(stats[1]), P(m), n, c, hw, P(ws), nbytes, P(gram), None),
            lib.dgvcc_lw_loss_backward_h(P(x), CODE[x.dtype], P(stats[0]), P(stats[1]), P(m), P(gram), P(gl), n, c, hw,
                                         P(ws), nbytes, P(dy), None),
            lib.dgvcc_isw_gram_h(P(x), CODE[x.dtype], n, c, hw, P(ws), nbytes, P(gram), None))


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("shape", UNTILED, ids=sid)
def test_lw_untiled_shapes_are_refused_and_match_through_the_cast_route(shape, dtype):
    x = make_x(shape, dtype)
    mask = make_mask(shape, "soft")
    assert h_return_codes(x, mask) == (UNSUPPORTED,) * 3
    check_lw(x, mask, expect_native=False)
    check_lw(x, None, expect_native=False)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_lw_misaligned_view_is_refused_and_matches_through_the_cast_route(dtype):
    shape = (2, 64, 16, 16)
    flat = torch.empty(2 * 64 * 256 + 1, dtype=dtype, device=DEV)
    x = flat[1:].view(shape)
    x.copy_(make_x(shape, dtype))
    assert x.is_contiguous() and x.data_ptr() % 16 != 0
    assert h_return_codes(x, None) == (UNSUPPORTED,) * 3
    check_lw(x, make_mask(shape, "binary"), expect_native=False)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_tensor_cores_off_takes_the_cast_route(dtype, monkeypatch):
    monkeypatch.setenv("DGVCC_ISW_TENSOR_CORES", "0")
    shape = (3, 64, 16, 16)
    check_lw(make_x(shape, dtype), make_mask(shape, "soft"), expect_native=False)
    xs = make_x((64, 256), dtype), make_x((64, 256), dtype, seed=5)
    check_ortho(*xs, expect_native=False)


# ------------------------------------------------------------------ memory, graphs, determinism
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("shape", CONFIG5, ids=sid)
def test_lw_forward_holds_no_fp32_map(shape, dtype):
    n, c, h, w = shape
    x = make_x(shape, dtype).requires_grad_(True)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(DEV)
    loss = lw_loss(x, None)
    torch.cuda.synchronize()
    held = torch.cuda.memory_allocated(DEV) - base
    assert loss.grad_fn.half == CODE[dtype]
    ws = _native.lib().dgvcc_isw_workspace_bytes(n, c, h * w)
    # Gram + workspace + statistics + the loss; the caching allocator may hand out up to 1 MB more than asked for a
    # large block (it does not split off a remainder that small)
    bound = n * c * c * 4 + ws + 3 * n * c * 4 + 512 + 2 * (1 << 20)
    assert held <= bound, (held, bound)
    saved = loss.grad_fn.saved_tensors
    assert not any(t.dtype == torch.float32 and t.numel() >= n * c * h * w for t in saved)
    assert any(t.dtype == dtype and t.numel() == n * c * h * w for t in saved)   # the half x itself
    del loss, saved


@pytest.mark.parametrize("mask", ["none", "soft"])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_lw_step_replays_as_a_cuda_graph(dtype, mask):
    shape = (4, 256, 16, 24)
    xs = [make_x(shape, dtype, seed=s) for s in range(3)]
    mk = make_mask(shape, mask)

    def step(x):
        loss = lw_loss(x, mk)
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


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_two_runs_give_the_same_bits(dtype):
    shape = (8, 256, 24, 32)
    x, mk = make_x(shape, dtype), make_mask(shape, "soft")
    a, b = lw_native(x, mk), lw_native(x, mk)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    y, z = make_x((100, 1000), dtype), make_x((100, 1000), dtype, seed=9)
    a, b = ortho_native(y, z), ortho_native(y, z)
    assert all(torch.equal(u, v) for u, v in zip(a[:3], b[:3]))


# ------------------------------------------------------------------ ortho_loss
def ortho_cast_route(x, y):
    xr = x.detach().float().requires_grad_(True)
    yr = y.detach().float().requires_grad_(True)
    loss = ortho_loss(xr, yr)
    loss.backward()
    return loss.detach(), xr.grad.to(x.dtype), yr.grad.to(y.dtype)


def ortho_native(x, y):
    xn = x.detach().requires_grad_(True)
    yn = y.detach().requires_grad_(True)
    loss = ortho_loss(xn, yn)
    route = loss.grad_fn.half
    loss.backward()
    return loss.detach(), xn.grad, yn.grad, route


def check_ortho(x, y, expect_native=True):
    ref = ortho_cast_route(x, y)
    out = ortho_native(x, y)
    assert out[3] == (CODE[x.dtype] if expect_native else None)
    assert out[1].dtype == x.dtype and out[2].dtype == y.dtype
    for a, b in zip(out[:3], ref):
        assert same(a, b)


@pytest.mark.parametrize("p", [104, 1000, 2056])
@pytest.mark.parametrize("c", [32, 64, 100, 512])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_ortho_native_matches_the_cast_route(c, p, dtype):
    check_ortho(make_x((c, p), dtype), make_x((c, p), dtype, seed=4))


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("cp", [(64, 100), (16, 256), (50, 256)], ids=sid)
def test_ortho_untiled_shapes_are_refused_and_match_through_the_cast_route(cp, dtype):
    c, p = cp
    x, y = make_x(cp, dtype), make_x(cp, dtype, seed=4)
    lib = _native.lib()
    nbytes = lib.dgvcc_isw_workspace_bytes(1, 2 * c, p)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=DEV)
    z = torch.cat([x, y]).contiguous()
    gram = torch.zeros((2 * c, 2 * c), device=DEV)
    gx, gy = torch.empty_like(x), torch.empty_like(y)
    gl = torch.ones((1,), device=DEV)
    # the stacked Gram has 2C rows: only P % 8 != 0 refuses it; the two dX GEMMs refuse every one of these shapes
    assert lib.dgvcc_isw_gram_h(P(z), CODE[dtype], 1, 2 * c, p, P(ws), nbytes, P(gram), None) == (
        UNSUPPORTED if p % 8 else 0)
    assert lib.dgvcc_ortho_loss_backward_h(P(x), P(y), CODE[dtype], P(gram), P(gl), c, p, P(ws), nbytes, P(gx), P(gy),
                                           None) == UNSUPPORTED
    check_ortho(x, y, expect_native=False)


def test_ortho_mixed_dtypes_take_the_cast_route():
    x, y = make_x((64, 256), torch.float16), make_x((64, 256), torch.bfloat16, seed=4)
    xr, yr = x.float().requires_grad_(True), y.float().requires_grad_(True)
    l_ref = ortho_loss(xr, yr)
    l_ref.backward()
    xn, yn = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
    loss = ortho_loss(xn, yn)
    assert loss.grad_fn.half is None
    loss.backward()
    assert torch.equal(loss.detach(), l_ref.detach())
    assert torch.equal(xn.grad, xr.grad.half()) and torch.equal(yn.grad, yr.grad.bfloat16())


def test_bad_dtype_code_is_an_argument_error():
    lib = _native.lib()
    x = make_x((2, 64, 16, 16), torch.float16)
    st = torch.empty((3, 128), device=DEV)
    assert lib.dgvcc_lw_standardize_stats_h(P(x), 0, 2, 64, 256, 1e-5, P(st[0]), P(st[1]), P(st[2]), None) == -1
    assert lib.dgvcc_lw_standardize_stats_h(P(x), 3, 2, 64, 256, 1e-5, P(st[0]), P(st[1]), P(st[2]), None) == -1
