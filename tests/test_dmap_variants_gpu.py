"""Every arm of the density-map splat (csrc/dmap_kernels.cu) at its edges, against the closed form and against each other.

dgvcc_dmap_splat_batch picks one of three arms:

  A  per-head sigma (sigma != NULL): dmap_prepare_kernel -> dmap_splat_kernel with per-head weight tables;
  B  fixed sigma, general: dmap_fixed_template_kernel + dmap_prepare_fixed_kernel -> dmap_splat_kernel with the
     template's table (radius != 7, or an image side >= 65536);
  C  fixed sigma, radius int(truncate*sigma + 0.5) == 7 and every side < 65536: dmap_prepare_fast_kernel -> lists of
     packed (row << 16 | column) centres -> dmap_splat_fixed_kernel.

The cases drive the C ABI directly with caller-chosen sigmas (no kNN), so each one reaches the arm and edge it names:
narrow / wide stamps (radius < or >= TAB = 32), chunks with at most or more than GEN_MAX = 8 wide heads, the warp and the
serial normaliser (<= or > MAX_LEAVES = 256 pairwise leaves), the CHUNK = 2048 head chunks and 256 px coarse tiles of
the culling passes, skipped and wrapped heads.  Each case proves the arm it took: the host selection rule is restated
and asserted, and the splat workspace, filled with 0xFF before the launch, is read back -- arm C never writes the Stamp
array, A and B write every head's Stamp (pixel, radius and coef exact, normaliser within a few ulp of numpy's pairwise
sum), and only A writes per-head weight tables.

Gates: against oracle.dmap_oracle.density_closed_form, assert_map_close (rtol 1e-5 + 1e-7 max|ref|: GPU fp64 exp may
differ from numpy's in the last ulp), with the pixels that are not bit-identical printed.  Between device arms the maps
must be bit-identical: every arm adds fl32(f64(fl32(w[|dy|])) * w[|dx|]) per pixel in head order, from weights computed
by the same device functions.
"""
import ctypes
import functools

import numpy as np
import pytest
import torch

from dgvcc_b200 import _native, synthetic
from dgvcc_b200.utils import dmap_gen
from oracle import dmap_oracle
from helpers import assert_map_close, record_margin

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
PATTERN = 0xFF
TAB, GEN_MAX, MAX_LEAVES, CHUNK, COARSE, FINE, FAST_R = 32, 8, 256, 2048, 256, 32, 7
FIXED_SIGMA, FIXED_TRUNCATE = dmap_gen.FIXED_SIGMA, dmap_gen.FIXED_TRUNCATE
NORM_ULPS = 8
STAMP = np.dtype([("ix", "<i4"), ("iy", "<i4"), ("radius", "<i4"), ("pad_", "<i4"), ("coef", "<f8"), ("norm", "<f8")])
assert STAMP.itemsize == 32
EMPTY = np.zeros((0, 2))
WIDE_EMPTY = (1, 65536)  # an empty image that puts the batch's max_side at 65536: fixed sigma then takes arm B


# ------------------------------------------------------------------------------------------------ restated rules
def fast_arm(per_head_sigma, fixed_sigma, truncate, max_side):
    """The `fast` predicate of dgvcc_dmap_splat_batch."""
    return not per_head_sigma and int(truncate * fixed_sigma + 0.5) == FAST_R and 0 < max_side < 65536


@functools.lru_cache(maxsize=None)
def leaf_count(n):
    """enumerate_leaves (dmap_kernels.cu) restated: leaves of numpy's pairwise summation over n elements."""
    if n <= 128:
        return 1
    n2 = n // 2
    n2 -= n2 % 8
    return leaf_count(n2) + leaf_count(n - n2)


@functools.lru_cache(maxsize=None)
def stamp_shape(sigma, truncate):
    """(radius, coef, normaliser) of scipy's 1-D kernel: numpy's own phi.sum(); identity when sigma <= 1e-15."""
    if not sigma > 1e-15:
        return 0, 0.0, 1.0
    radius = int(truncate * sigma + 0.5)
    x = np.arange(-radius, radius + 1)
    phi = np.exp(-0.5 / (sigma * sigma) * x ** 2)
    return radius, -0.5 / (sigma * sigma), float(phi.sum())


def one_hot_pixel(x, y, h, w):
    """dmap_gen.py:41-42: (kept, column, row) after int() truncation and numpy's negative-index wrap."""
    ix, iy = int(x), int(y)
    keep = iy < h and ix < w
    iy, ix = iy + h if iy < 0 else iy, ix + w if ix < 0 else ix
    return keep and iy >= 0 and ix >= 0, ix, iy


# ------------------------------------------------------------------------------------------------ one launch set
class Splat:
    """One launch set of dgvcc_dmap_splat_batch over `shapes` in the caller's order, with the workspace and the output
    filled with 0xFF bytes first; keeps the maps and the workspace as host arrays."""

    def __init__(self, shapes, pts_list, sigmas=None, fixed_sigma=FIXED_SIGMA, truncate=FIXED_TRUNCATE):
        self.shapes = [tuple(s) for s in shapes]
        self.pts = [np.ascontiguousarray(p, dtype=np.float64).reshape(-1, 2) for p in pts_list]
        self.sigmas = None if sigmas is None else [np.asarray(s, dtype=np.float64) for s in sigmas]
        self.fixed_sigma, self.truncate = fixed_sigma, truncate
        self.plan = dmap_gen._Plan(self.shapes, [len(p) for p in self.pts])
        pl = self.plan.plan
        meta = torch.from_numpy(self.plan.meta).to(DEV)
        ws = torch.full((pl.splat_workspace_bytes,), PATTERN, dtype=torch.uint8, device=DEV)
        out = torch.full((pl.total_pixels * 4,), PATTERN, dtype=torch.uint8, device=DEV)  # NaN until written
        d_pts = sig = None
        if pl.total_heads:
            d_pts = torch.from_numpy(np.concatenate(self.pts)).to(DEV)
            if self.sigmas is not None:
                sig = torch.from_numpy(np.concatenate(self.sigmas)).to(DEV)
        _native.check(_native.lib().dgvcc_dmap_splat_batch(
            _native.ptr(d_pts), _native.ptr(sig), fixed_sigma, truncate, len(self.shapes), _native.ptr(meta),
            ctypes.byref(pl), _native.ptr(ws), pl.splat_workspace_bytes, _native.ptr(out), _native.stream_ptr(DEV)),
            "dgvcc_dmap_splat_batch")
        torch.cuda.synchronize()
        flat = out.cpu().numpy().view(np.float32)
        self.ws = ws.cpu().numpy()
        self.maps = [flat[o:o + h * w].reshape(h, w) for o, (h, w) in zip(self.plan.out_off[:-1], self.shapes)]

    def region(self, off, nbytes):
        return self.ws[int(off):int(off) + int(nbytes)]

    def occupancy(self, image):
        """Occupancy bits of the fine tiles of one image."""
        pl, meta = self.plan.plan, self.plan.meta
        words = self.region(pl.off_fmask, (pl.fine_tiles // 32 + 1) * 4).view(np.uint32)
        t = np.arange(meta[image, 5], meta[image + 1, 5])
        return (words[t >> 5] >> (t & 31).astype(np.uint32)) & 1

    def assert_arm(self, arm):
        """Prove that this launch took `arm`: the host rule restated, then what the launch left in the workspace."""
        pl = self.plan.plan
        assert fast_arm(self.sigmas is not None, self.fixed_sigma, self.truncate, pl.max_side) == (arm == "C")
        assert (self.sigmas is not None) == (arm == "A")
        n = int(pl.total_heads)
        raw = self.region(pl.off_stamps, n * STAMP.itemsize)
        wtab_raw = self.region(pl.off_wtab, n * TAB * 8)
        if arm == "C":
            assert (raw == PATTERN).all(), "arm C wrote Stamps: the launch did not take the fast arm"
            return
        if arm == "B":
            assert (wtab_raw == PATTERN).all(), "arm B wrote per-head weight tables"
        stamps, wtab = raw.view(STAMP), wtab_raw.view(np.float64).reshape(n, TAB)
        k = 0
        for img, ((h, w), pts) in enumerate(zip(self.shapes, self.pts)):
            for j, (x, y) in enumerate(pts):
                s = stamps[k]
                keep, ix, iy = one_hot_pixel(x, y, h, w)
                if not keep:
                    assert s["radius"] == -1, f"image {img} head {j} ({x}, {y}) is skipped, radius {s['radius']}"
                    k += 1
                    continue
                sd = float(self.sigmas[img][j]) if arm == "A" else self.fixed_sigma
                radius, coef, norm = stamp_shape(sd, self.truncate)
                what = f"image {img} head {j} sigma {sd!r}"
                assert (s["ix"], s["iy"]) == (ix, iy), what
                assert s["radius"] == radius and s["coef"] == coef, f"{what}: {s}"
                assert abs(s["norm"] - norm) <= NORM_ULPS * np.spacing(norm), f"{what}: norm {s['norm']!r} vs numpy {norm!r}"
                if arm == "A" and radius < TAB:  # the per-head table: w[|d|] = phi(d) / norm
                    ref = np.exp(coef * np.arange(radius + 1) ** 2) / s["norm"]
                    assert np.all(np.abs(wtab[k, :radius + 1] - ref) <= NORM_ULPS * np.spacing(ref)), what
                k += 1


def closed_form(shape, pts, sigmas, truncate):
    return dmap_oracle.density_closed_form(shape, np.asarray(pts, dtype=np.float64), sigmas=np.asarray(sigmas, dtype=np.float64),
                                           truncate=truncate)


def gate(got, shape, pts, sigmas, truncate, what):
    """Closed-form gate; returns the oracle map."""
    ref = closed_form(shape, pts, sigmas, truncate)
    diff = assert_map_close(got, ref, what)
    err = torch.from_numpy(np.abs(got.astype(np.float64) - ref))
    record_margin(what, err, torch.from_numpy(1e-5 * np.abs(ref) + 1e-7 * float(np.abs(ref).max(initial=0.0))), 1e-5, 1e-7)
    print(f"{what}: {diff} of {got.size} pixels not bit-identical to the closed form")
    return ref


def assert_head_order(got, ref, shape, pts, sigmas, truncate, what):
    """The case is order-sensitive (the fp32 sums change when the heads are reversed), and the device map follows the
    forward order: it equals the forward closed form on more of those pixels than the reversed one."""
    rev = closed_form(shape, pts[::-1], np.asarray(sigmas)[::-1], truncate)
    sensitive = ref != rev
    assert sensitive.sum() >= 10, f"{what}: head order barely changes the sums, the case cannot catch a reordering"
    fwd_hits, rev_hits = int((got[sensitive] == ref[sensitive]).sum()), int((got[sensitive] == rev[sensitive]).sum())
    print(f"{what}: {int(sensitive.sum())} order-sensitive pixels, device == forward on {fwd_hits}, == reversed on {rev_hits}")
    assert fwd_hits > rev_hits, f"{what}: the device map follows the reversed head order"


def three_way(shapes, pts_list, what):
    """Fixed sigma 4, truncate 7/4 through arms C, B (the batch plus an empty image of side 65536) and A (a sigma
    array of 4.0): bit-identical maps, each checked against the closed form once.  Returns the arm-C run."""
    c = Splat(shapes, pts_list)
    c.assert_arm("C")
    b = Splat(list(shapes) + [WIDE_EMPTY], list(pts_list) + [EMPTY])
    b.assert_arm("B")
    assert not b.maps[-1].any() and not b.occupancy(len(shapes)).any()
    a = Splat(shapes, pts_list, sigmas=[np.full(len(p), FIXED_SIGMA) for p in pts_list])
    a.assert_arm("A")
    for i, (shape, pts) in enumerate(zip(shapes, pts_list)):
        assert np.array_equal(c.maps[i], b.maps[i]), f"{what} image {i}: arms C and B differ"
        assert np.array_equal(c.maps[i], a.maps[i]), f"{what} image {i}: arms C and A differ"
        gate(c.maps[i], shape, pts, np.full(len(pts), FIXED_SIGMA), FIXED_TRUNCATE, f"{what} image {i} {shape}")
    return c


def in_tile(rng, n, x0, y0, size=FINE):
    return rng.uniform([x0, y0], [x0 + size, y0 + size], size=(n, 2))


# ------------------------------------------------------------------------------------ 1. three-way fixed identity
def edge_hugging_points():
    xs = [0.0, 0.5, 3.2, 6.9, 7.1, 450.3, 892.5, 893.0, 898.7, 899.99, -0.5, -1.0]
    ys = [0.0, 0.5, 4.0, 6.99, 350.2, 692.01, 693.0, 699.5, -0.3, -1.0]
    pts = np.array([(x, y) for x in xs for y in ys] + [(900.0, 5.0), (5.0, 700.0)])
    np.random.default_rng(11).shuffle(pts, axis=0)
    return (700, 900), pts


@pytest.mark.parametrize("crowd", ["dense", "sparse_edges"])
def test_fixed_sigma_three_arms_bit_identical(crowd):
    if crowd == "dense":
        shape = (2048, 2048)
        pts = synthetic.crowd_points(np.random.default_rng(5001), 25000, 2048, 2048, dtype=np.float64)
    else:
        shape, pts = edge_hugging_points()
    three_way([shape], [pts], crowd)


@pytest.mark.parametrize("width", [65535, 65536, 70000])
def test_fixed_public_api_past_the_16_bit_column(width):
    """Arm C packs a centre column into 16 bits: a side of 65536 or more must take arm B, also for heads in columns
    >= 65536."""
    cols = [3.0, width - 9.5, width - 7.0, width - 1.0, width - 0.5, 65529.5, 65534.5, 65535.0, 65535.9, 65536.0,
            65537.2, 69999.9, 70000.0]
    rows = [0.0, 0.7, -0.5, -1.0, 1.0]
    pts = np.array([(c, rows[i % len(rows)]) for i, c in enumerate(cols)])
    shape = (1, width)
    run = Splat([shape], [pts])
    run.assert_arm("C" if width < 65536 else "B")
    got = dmap_gen.gaussian_filter_density_fixed(np.empty(shape + (0,)), pts)
    assert np.array_equal(got, run.maps[0]), "public API and the C ABI differ"
    gate(got, shape, pts, np.full(len(pts), FIXED_SIGMA), FIXED_TRUNCATE, f"(1, {width})")
    if width > 65536:
        assert got[0, 65536:].any(), "heads past column 65535 left no trace"


# ------------------------------------------------------------------------------- 2. other fixed sigmas: arm B == A
@pytest.mark.parametrize("sigma,truncate,radius", [
    (2.0, 4.0, 8),      # narrow shared table
    (7.75, 4.0, 31),    # the widest narrow stamp
    (8.0, 4.0, 32),     # the narrowest wide stamp
    (10.0, 4.0, 40),    # wide: weights evaluated per tile, more than GEN_MAX wide heads per chunk
])
def test_fixed_sigma_arm_b_equals_arm_a(sigma, truncate, radius):
    assert stamp_shape(sigma, truncate)[0] == radius
    shape = (500, 700)
    pts = synthetic.crowd_points(np.random.default_rng(6000 + radius), 3000, 700, 500, dtype=np.float64)
    b = Splat([shape], [pts], fixed_sigma=sigma, truncate=truncate)
    b.assert_arm("B")
    a = Splat([shape], [pts], sigmas=[np.full(len(pts), sigma)], truncate=truncate)
    a.assert_arm("A")
    assert np.array_equal(a.maps[0], b.maps[0]), "arms A and B differ"
    gate(b.maps[0], shape, pts, np.full(len(pts), sigma), truncate, f"sigma {sigma} radius {radius}")


# ------------------------------------------------------------------------------------------ 3. narrow / wide edge
def test_narrow_wide_edge_in_one_tile():
    """Radii 30, 31 (narrow: per-head table) and 32, 33 (wide: weights per tile) mixed in one tile, stamps overlapping;
    7.874999 / 7.875 sit on either side of the radius 31 / 32 rounding."""
    rng = np.random.default_rng(7)
    sig_choices = np.array([7.5, 7.75, 7.874999, 7.875, 8.0, 8.25])
    assert [stamp_shape(s, 4.0)[0] for s in sig_choices] == [30, 31, 31, 32, 32, 33]
    shape = (160, 192)
    pts = in_tile(rng, 24, 64, 64)
    sigmas = rng.permutation(np.tile(sig_choices, 4))
    run = Splat([shape], [pts], sigmas=[sigmas], truncate=4.0)
    run.assert_arm("A")
    ref = gate(run.maps[0], shape, pts, sigmas, 4.0, "narrow/wide edge")
    assert_head_order(run.maps[0], ref, shape, pts, sigmas, 4.0, "narrow/wide edge")


# ---------------------------------------------------------------------------------------------- 4. GEN_MAX edge
@pytest.mark.parametrize("n_heads,n_wide", [(32, 0), (32, 1), (32, 8), (32, 9), (32, 31), (32, 32), (300, 75)])
def test_wide_heads_per_chunk(n_heads, n_wide):
    """n_heads on one fine tile, n_wide of them wide, spread over the index order between narrow ones: one staged group
    of 32 when a chunk holds <= GEN_MAX wide heads, groups of 8 above; 300 heads (> SPLAT_THREADS) are compacted in
    three passes."""
    rng = np.random.default_rng(100 * n_heads + n_wide)
    wide = np.zeros(n_heads, dtype=bool)
    wide[np.round(np.linspace(0, n_heads - 1, n_wide)).astype(int)] = True
    assert wide.sum() == n_wide
    sigmas = np.where(wide, rng.uniform(8.0, 12.0, n_heads), rng.uniform(1.0, 7.8, n_heads))
    assert all((stamp_shape(s, 4.0)[0] >= TAB) == wd for s, wd in zip(sigmas, wide))
    shape = (160, 192)
    pts = in_tile(rng, n_heads, 64, 64)
    run = Splat([shape], [pts], sigmas=[sigmas], truncate=4.0)
    run.assert_arm("A")
    what = f"{n_heads} heads, {n_wide} wide"
    ref = gate(run.maps[0], shape, pts, sigmas, 4.0, what)
    assert_head_order(run.maps[0], ref, shape, pts, sigmas, 4.0, what)


# ------------------------------------------------------------------------------------ 5. identity filter, radius 0
def test_identity_filter_and_radius_zero():
    """sigma <= 1e-15 copies the input (scipy); sigma 0.1 has radius 0 (a one-element kernel of weight 1); coincident
    heads add up exactly."""
    rng = np.random.default_rng(5)
    shape = (64, 80)
    sig_choices = np.array([0.0, 1e-16, 1e-15, 2e-15, 0.1, 0.12, 1.0, 3.0])
    pts = rng.uniform([0, 0], [80, 64], size=(40, 2))
    pts[10:14] = pts[3]
    sigmas = np.tile(sig_choices, 5)
    sigmas[[3, 10, 11, 12, 13]] = 0.0
    run = Splat([shape], [pts], sigmas=[sigmas], truncate=4.0)
    run.assert_arm("A")
    gate(run.maps[0], shape, pts, sigmas, 4.0, "identity / radius 0")
    iy, ix = int(pts[3, 1]), int(pts[3, 0])
    assert run.maps[0][iy, ix] >= 5.0
    for fixed in (0.0, 0.1):  # arm B: a radius-0 template, identity or not
        b = Splat([shape], [pts], fixed_sigma=fixed, truncate=4.0)
        b.assert_arm("B")
        a = Splat([shape], [pts], sigmas=[np.full(len(pts), fixed)], truncate=4.0)
        a.assert_arm("A")
        assert np.array_equal(a.maps[0], b.maps[0]), f"fixed sigma {fixed}: arms A and B differ"
        gate(b.maps[0], shape, pts, np.full(len(pts), fixed), 4.0, f"fixed sigma {fixed}")


def test_coincident_heads_adaptive_public_api():
    """Four coincident heads in a full-size crowd: their kNN sigma is 0, the identity filter."""
    shape = (768, 1024)
    pts = synthetic.crowd_points(np.random.default_rng(44), 1500, 1024, 768, dtype=np.float64)
    pts[4:7] = pts[0]
    sigmas = dmap_oracle.adaptive_sigmas(pts)
    assert np.array_equal(sigmas[[0, 4, 5, 6]], np.zeros(4))
    got = dmap_gen.gaussian_filter_density(np.empty(shape + (0,)), pts)
    gate(got, shape, pts, sigmas, 4.0, "coincident heads")
    assert got[int(pts[0, 1]), int(pts[0, 0])] >= 4.0


# ------------------------------------------------------------------------------------------------ 6. normaliser
R_256 = max(r for r in range(15000, 16000) if leaf_count(2 * r + 1) == MAX_LEAVES)
R_257 = min(r for r in range(15000, 16000) if leaf_count(2 * r + 1) == MAX_LEAVES + 1)


@pytest.mark.parametrize("radius", [R_256, R_257])
def test_normaliser_warp_and_serial(radius):
    """2r+1 elements in exactly 256 pairwise leaves (one warp sums them) and in 257 (lane 0 sums them serially);
    stamps far larger than the image."""
    assert R_257 == R_256 + 1
    sigma = radius / 4.0  # int(4 * sigma + 0.5) == radius
    assert stamp_shape(sigma, 4.0)[0] == radius
    shape = (40, 50)
    pts = np.array([[3.5, 2.0], [49.9, 39.9], [25.0, 20.0], [60.0, 3.0]])
    sigmas = np.full(len(pts), sigma)
    a = Splat([shape], [pts], sigmas=[sigmas], truncate=4.0)
    a.assert_arm("A")  # normaliser within NORM_ULPS of numpy's phi.sum()
    b = Splat([shape], [pts], fixed_sigma=sigma, truncate=4.0)
    b.assert_arm("B")
    assert np.array_equal(a.maps[0], b.maps[0]), "arms A and B differ"
    gate(a.maps[0], shape, pts, sigmas, 4.0, f"radius {radius} ({leaf_count(2 * radius + 1)} leaves)")


# -------------------------------------------------------------------------------------------------- 7. culling
def test_culling_chunks_and_coarse_tile_edges():
    """2047 / 2048 / 2049 / 4097 heads on one coarse tile (the CHUNK boundaries of the coarse passes), heads at
    x, y = 255, 256, 257 whose stamps span four coarse tiles, sides 255 / 256 / 257 and sides that are no multiple of 32;
    fixed sigma through all three arms, then per-head sigmas up to radius 48 through arm A."""
    rng = np.random.default_rng(2049)
    shapes = [(255, 257), (256, 300), (257, 255), (300, 290)]
    counts = [2047, 2048, 2049, 4097]
    edge = np.array([(x, y) for x in (250.5, 255.0, 255.5, 256.0, 257.0) for y in (252.0, 255.0, 256.0, 256.7, 257.0)])
    pts_list = []
    for (h, w), n in zip(shapes, counts):
        p = rng.uniform([0, 0], [min(w, COARSE), min(h, COARSE)], size=(n, 2))
        p[rng.choice(n, len(edge), replace=False)] = edge
        pts_list.append(p)
    three_way(shapes, pts_list, "culling")
    sigmas = [rng.uniform(0.5, 12.0, len(p)) for p in pts_list]
    a = Splat(shapes, pts_list, sigmas=sigmas, truncate=4.0)
    a.assert_arm("A")
    for i, (shape, p, s) in enumerate(zip(shapes, pts_list, sigmas)):
        gate(a.maps[i], shape, p, s, 4.0, f"culling, per-head sigma, image {i} {shape}")


# ---------------------------------------------------------------------------------------- 8. skipped and wrapped
def skip_wrap_batch():
    rng = np.random.default_rng(808)
    special = [(90.0, 5.0), (5.0, 70.0), (89.99, 69.99), (-0.5, 10.0), (10.0, -0.999), (-1.0, 20.0), (-90.0, 20.0),
               (-89.5, 30.0), (20.0, -70.0), (20.0, -1.5), (1e6, 3.0),
               (95.0, -100.0),   # x out of range: skipped, y below -height never indexes (the reference's `and`)
               (-100.0, 80.0)]   # y out of range: skipped before x is looked at
    wrap = rng.uniform([0, 0], [90, 70], size=(40 + len(special), 2))
    wrap[3::4][:len(special)] = special          # in the middle of the staged groups
    skipped = np.array([(65.0, 1.0), (70.2, 10.0), (3.0, 33.0), (3.0, 40.5), (1e9, 1e9), (-100.0, 33.0), (66.0, -50.0)])
    crowd = synthetic.crowd_points(rng, 200, 150, 120, dtype=np.float64)
    shapes = [(70, 90), (40, 50), (33, 65), (100, 64), (120, 150)]
    return shapes, [wrap, EMPTY, skipped, EMPTY, crowd]


def test_skipped_and_wrapped_heads_all_arms():
    shapes, pts_list = skip_wrap_batch()
    c = three_way(shapes, pts_list, "skip/wrap")
    assert not c.maps[2].any() and not c.occupancy(2).any(), "an image whose heads are all skipped"
    assert c.occupancy(4).any()
    sigmas = [dmap_oracle.adaptive_sigmas(p) if len(p) else np.zeros(0) for p in pts_list]
    a = Splat(shapes, pts_list, sigmas=sigmas, truncate=4.0)
    a.assert_arm("A")
    assert not a.maps[2].any() and not a.occupancy(2).any()
    for i, (shape, p, s) in enumerate(zip(shapes, pts_list, sigmas)):
        gate(a.maps[i], shape, p, s, 4.0, f"skip/wrap adaptive image {i} {shape}")


@pytest.mark.parametrize("fixed", [True, False])
def test_skipped_and_wrapped_heads_batch_api_caller_order(fixed):
    """The batch API launches images by falling head count and must return the maps in the caller's order."""
    shapes, pts_list = skip_wrap_batch()
    counts = [len(p) for p in pts_list]
    assert list(np.argsort(-np.array(counts), kind="stable")) != list(range(len(counts)))
    outs = dmap_gen.gaussian_filter_density_batch(shapes, pts_list, fixed=fixed)
    for i, (shape, p, o) in enumerate(zip(shapes, pts_list, outs)):
        assert o.shape == shape
        s = np.full(len(p), FIXED_SIGMA) if fixed else (dmap_oracle.adaptive_sigmas(p) if len(p) else np.zeros(0))
        gate(o, shape, p, s, FIXED_TRUNCATE if fixed else 4.0, f"batch API fixed={fixed} image {i} {shape}")
        fn = dmap_gen.gaussian_filter_density_fixed if fixed else dmap_gen.gaussian_filter_density
        assert np.array_equal(o, fn(np.empty(shape + (0,)), p)), f"image {i}: batched and single-image maps differ"
    assert not outs[2].any()


# ---------------------------------------------------------------------------------------------- 9. kNN slice plan
@pytest.mark.parametrize("counts,max_slices", [([100, 700, 2100, 1200], 64), ([76000] * 4, 1)])
def test_batched_knn_at_both_ends_of_the_slice_plan(counts, max_slices):
    plist = [np.random.default_rng(900 + i).uniform(0, 4000, size=(n, 2)) for i, n in enumerate(counts)]
    plan = dmap_gen._Plan([(2048, 2048)] * len(counts), counts)
    pl = plan.plan
    assert pl.knn_max_slices == max_slices
    meta = torch.from_numpy(plan.meta).to(DEV)
    d_pts = torch.from_numpy(np.concatenate(plist)).to(DEV)
    idx = torch.empty((pl.total_heads, 4), dtype=torch.int32, device=DEV)
    dist = torch.empty((pl.total_heads, 4), dtype=torch.float64, device=DEV)
    sigma = torch.empty((pl.total_heads,), dtype=torch.float64, device=DEV)
    kws = torch.empty((pl.knn_workspace_bytes,), dtype=torch.uint8, device=DEV)
    _native.check(_native.lib().dgvcc_dmap_knn_sigma_batch(
        _native.ptr(d_pts), len(counts), _native.ptr(meta), ctypes.byref(pl), _native.ptr(idx), _native.ptr(dist),
        _native.ptr(sigma), _native.ptr(kws), pl.knn_workspace_bytes, _native.stream_ptr(DEV)), "knn batch")
    idx, dist, sigma = idx.cpu().numpy(), dist.cpu().numpy(), sigma.cpu().numpy()
    for i, p in enumerate(plist):
        assert len(np.unique(p, axis=0)) == len(p)
        lo, hi = plan.pt_off[i], plan.pt_off[i + 1]
        rd, rl = dmap_oracle.knn4(p)
        assert np.array_equal(idx[lo:hi], rl) and np.array_equal(dist[lo:hi], rd), f"image {i} (n={len(p)})"
        assert np.array_equal(sigma[lo:hi], (rd[:, 1] + rd[:, 2] + rd[:, 3]) * 0.1)


# ---------------------------------------------------------------------------------------- non-finite heads
def reference_outcome(fn):
    try:
        fn()
    except (ValueError, OverflowError, IndexError) as e:
        return type(e)
    return None


def assert_raises_like_reference(expected, fn):
    with pytest.raises(Exception) as ei:
        fn()
    assert type(ei.value) is expected, f"raised {type(ei.value).__name__}: {ei.value}, the reference raises {expected.__name__}"


SHAPE = (20, 30)
BASE = np.array([[3.0, 4.0], [10.5, 7.25], [29.5, 19.5], [-0.5, 2.0], [15.0, 12.0], [6.0, 18.0]])


@pytest.mark.parametrize("fixed", [True, False])
@pytest.mark.parametrize("head", [0, 4])
@pytest.mark.parametrize("coord", [0, 1])
@pytest.mark.parametrize("value", [np.nan, np.inf, -np.inf])
def test_non_finite_heads_raise_like_the_reference(value, coord, head, fixed):
    pts = BASE.copy()
    pts[head, coord] = value
    expected = reference_outcome(lambda: dmap_oracle.density_reference_like(SHAPE, pts, fixed=fixed))
    assert expected is not None
    fn = dmap_gen.gaussian_filter_density_fixed if fixed else dmap_gen.gaussian_filter_density
    assert_raises_like_reference(expected, lambda: fn(np.empty(SHAPE + (0,)), pts))
    assert_raises_like_reference(expected, lambda: dmap_gen.gaussian_filter_density_batch(
        [(25, 25), SHAPE], [BASE, pts], fixed=fixed))


@pytest.mark.parametrize("fixed", [True, False])
@pytest.mark.parametrize("case", ["index_then_nan", "nan_then_index", "skipped_nan_x", "skipped_negative"])
def test_first_offending_head_decides(case, fixed):
    """The reference raises at the first head whose int() or one-hot write fails; the kNN of the adaptive path fails
    first on any non-finite head.  A head whose row is already out of range is skipped before its column is converted."""
    pts = BASE.copy()
    if case == "index_then_nan":
        pts[1] = (-50.0, 2.0)
        pts[3] = (np.nan, 1.0)
    elif case == "nan_then_index":
        pts[1] = (1.0, np.nan)
        pts[3] = (-50.0, 2.0)
    elif case == "skipped_nan_x":
        pts[2] = (np.nan, 25.0)
    else:
        pts[2] = (-50.0, 25.0)
        pts[4] = (40.0, -50.0)
    expected = reference_outcome(lambda: dmap_oracle.density_reference_like(SHAPE, pts, fixed=fixed))
    fn = dmap_gen.gaussian_filter_density_fixed if fixed else dmap_gen.gaussian_filter_density
    if expected is None:
        ref = dmap_oracle.density_reference_like(SHAPE, pts, fixed=fixed)
        assert_map_close(fn(np.empty(SHAPE + (0,)), pts), ref, case)
        assert_map_close(dmap_gen.gaussian_filter_density_batch([SHAPE], [pts], fixed=fixed)[0], ref, case)
    else:
        assert_raises_like_reference(expected, lambda: fn(np.empty(SHAPE + (0,)), pts))
        # images are checked in the caller's order: the first image's error wins
        assert_raises_like_reference(expected, lambda: dmap_gen.gaussian_filter_density_batch(
            [SHAPE, SHAPE], [pts, np.array([[np.nan, np.nan]] * 5)], fixed=fixed))


@pytest.mark.parametrize("value", [np.nan, np.inf, -np.inf])
def test_knn_sigma_rejects_non_finite_heads_like_kdtree(value):
    pts = BASE.copy()
    pts[2, 1] = value
    assert reference_outcome(lambda: dmap_oracle.knn4(pts)) is ValueError
    assert_raises_like_reference(ValueError, lambda: dmap_gen.knn_sigma(pts))
