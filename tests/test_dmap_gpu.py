"""Parity of the CUDA density-map generator (through the C ABI) with the reference fixtures and the oracle.

Gates (SURVEY.md section 8d): kNN neighbour indices and in-bounds bookkeeping bit-exact; sigma <= 1 ulp;
density maps rtol 1e-5 with atol 1e-7*max|ref| (fp64 exp on the GPU may differ from numpy's in the last
ulp; after the two fp32 roundings that is almost always invisible -- the tests also report how many
pixels are not bit-identical)."""
import os

import numpy as np
import pytest

from dgvcc_b200 import synthetic
from oracle import dmap_oracle
from helpers import GOLDEN, assert_map_close

pytestmark = pytest.mark.gpu

CASES = ["a40", "a4", "a3", "a1", "a0", "a25f32", "oob", "dup"]


@pytest.fixture(scope="module")
def fixtures():
    return np.load(os.path.join(GOLDEN, "dmap_cases.npz"))


@pytest.mark.parametrize("name", CASES)
def test_maps_match_reference_fixture(fixtures, name):
    from dgvcc_b200.utils import dmap_gen
    shape = tuple(int(v) for v in fixtures[f"{name}_shape"])
    pts = fixtures[f"{name}_points"]
    img = np.zeros(shape + (3,), dtype=np.uint8)
    diff_a = assert_map_close(dmap_gen.gaussian_filter_density(img, pts), fixtures[f"{name}_adaptive"], f"{name} adaptive")
    diff_f = assert_map_close(dmap_gen.gaussian_filter_density_fixed(img, pts), fixtures[f"{name}_fixed"], f"{name} fixed")
    print(f"{name}: pixels not bit-identical: adaptive {diff_a}, fixed {diff_f} of {shape[0] * shape[1]}")


@pytest.mark.parametrize("name", ["knn2000", "knn700f32"])
def test_knn_bit_exact(fixtures, name):
    from dgvcc_b200.utils import dmap_gen
    pts = fixtures[f"{name}_points"]
    dist, loc, sigma = dmap_gen.knn_sigma(pts)
    assert np.array_equal(loc, fixtures[f"{name}_loc"]), "neighbour indices"
    assert np.array_equal(dist, fixtures[f"{name}_dist"]), "neighbour distances"
    ref_sigma = (fixtures[f"{name}_dist"][:, 1] + fixtures[f"{name}_dist"][:, 2] + fixtures[f"{name}_dist"][:, 3]) * 0.1
    assert np.array_equal(sigma, ref_sigma)


def test_few_points_knn_convention():
    from dgvcc_b200.utils import dmap_gen
    pts = np.array([[3.0, 4.0], [10.0, 4.0]])
    dist, loc, sigma = dmap_gen.knn_sigma(pts)
    rd, rl = dmap_oracle.knn4(pts)
    assert np.array_equal(dist, rd) and np.array_equal(loc, rl) and np.array_equal(sigma, [15.0, 15.0])


@pytest.mark.parametrize("seed,n,h,w,dtype", [
    (1, 1500, 768, 1024, np.float64),     # ShanghaiTech-like
    (2, 6000, 1100, 1700, np.float32),    # sides that are no multiple of the tile
    (3, 8, 600, 900, np.float64),         # sparse: huge sigmas, stamps larger than the image
    (4, 25000, 2048, 2048, np.float64),   # JHU-shaped maximum of BASELINE config 4
])
def test_full_size_against_closed_form_oracle(seed, n, h, w, dtype):
    from dgvcc_b200.utils import dmap_gen
    rng = np.random.default_rng(4000 + seed)
    pts = synthetic.crowd_points(rng, n, w, h, dtype=dtype)
    img = np.empty((h, w, 0))
    dist, loc, sigma = dmap_gen.knn_sigma(pts)
    rd, rl = dmap_oracle.knn4(pts)
    assert len(np.unique(pts, axis=0)) == n, "synthetic heads must be distinct (tie order is implementation-defined)"
    assert np.array_equal(loc, rl) and np.array_equal(dist, rd)
    ref = dmap_oracle.density_closed_form((h, w), pts, sigmas=(rd[:, 1] + rd[:, 2] + rd[:, 3]) * 0.1)
    got = dmap_gen.gaussian_filter_density(img, pts)
    diff = assert_map_close(got, ref, "adaptive")
    ref_f = dmap_oracle.density_closed_form((h, w), pts, fixed=True)
    diff_f = assert_map_close(dmap_gen.gaussian_filter_density_fixed(img, pts), ref_f, "fixed")
    print(f"n={n} {h}x{w}: pixels not bit-identical: adaptive {diff}, fixed {diff_f} of {h * w}")
    # mass conservation away from the border: every in-bounds head contributes <= 1
    assert got.sum(dtype=np.float64) <= n * (1 + 1e-6)


def test_sparse_images_with_huge_sigma():
    """4..10 heads spread over a 2048 px image: sigma in the hundreds, kernel radius in the thousands
    (deep pairwise splits of the normaliser sum)."""
    from dgvcc_b200.utils import dmap_gen
    for n, seed in ((4, 1), (5, 2), (7, 3), (10, 4)):
        rng = np.random.default_rng(seed)
        h, w = 2048, 1900
        pts = rng.uniform([0, 0], [w - 1, h - 1], size=(n, 2))
        ref = dmap_oracle.density_closed_form((h, w), pts)
        got = dmap_gen.gaussian_filter_density(np.empty((h, w, 0)), pts)
        assert_map_close(got, ref, f"sparse n={n}")


def test_batch_api_and_file_protocol(tmp_path):
    from dgvcc_b200.utils import dmap_gen
    from PIL import Image
    rng = np.random.default_rng(9)
    shapes = [(120, 160), (90, 90), (64, 200)]
    plist = [synthetic.crowd_points(rng, n, s[1], s[0], dtype=np.float64) for n, s in zip((50, 0, 7), shapes)]
    outs = dmap_gen.gaussian_filter_density_batch(shapes, plist, fixed=True)
    for s, p, o in zip(shapes, plist, outs):
        assert_map_close(o, dmap_oracle.density_closed_form(s, p, fixed=True), "batch")
    # run(): <name>.jpg + <name>.npy -> <name>_dmap.npy, idempotent (dmap_gen.py:83-95)
    fn = tmp_path / "img_7.jpg"
    Image.fromarray(np.zeros((120, 160, 3), dtype=np.uint8)).save(fn)
    np.save(tmp_path / "img_7.npy", plist[0])
    dmap_gen.run(str(fn))
    saved = np.load(tmp_path / "img_7_dmap.npy")
    assert_map_close(saved, dmap_oracle.density_closed_form((120, 160), plist[0], fixed=True), "run()")
    mtime = os.path.getmtime(tmp_path / "img_7_dmap.npy")
    dmap_gen.run(str(fn))
    assert os.path.getmtime(tmp_path / "img_7_dmap.npy") == mtime
    # run_many(): what the CLI does for a directory -- batched, existing outputs skipped
    fns = [str(fn)]
    for k, (s, p) in enumerate(zip(shapes, plist)):
        f2 = tmp_path / f"img_b{k}.jpg"
        Image.fromarray(np.zeros(s + (3,), dtype=np.uint8)).save(f2)
        np.save(tmp_path / f"img_b{k}.npy", p)
        fns.append(str(f2))
    dmap_gen.run_many(fns, batch=2)
    assert os.path.getmtime(tmp_path / "img_7_dmap.npy") == mtime
    for k, (s, p) in enumerate(zip(shapes, plist)):
        saved = np.load(tmp_path / f"img_b{k}_dmap.npy")
        assert saved.shape == s and saved.dtype == np.float32
        assert_map_close(saved, dmap_oracle.density_closed_form(s, p, fixed=True), "run_many()")


def test_batched_launch_matches_oracle_on_a_ragged_list():
    """One launch set for a ragged list (empty image, < 4 heads, > CHUNK heads, sides that are no multiple of the
    fine / coarse tile): every map bit-identical to the closed-form oracle and to the single-image call."""
    from dgvcc_b200.utils import dmap_gen
    rng = np.random.default_rng(77)
    spec = [(300, 520, 0), (257, 513, 3), (700, 333, 2500), (64, 32, 1), (1030, 1290, 5000), (40, 700, 60), (512, 512, 4)]
    shapes = [(h, w) for h, w, _ in spec]
    plist = [synthetic.crowd_points(np.random.default_rng(100 + i), n, w, h, dtype=np.float64)
             for i, (h, w, n) in enumerate(spec)]
    for fixed in (False, True):
        outs = dmap_gen.gaussian_filter_density_batch(shapes, plist, fixed=fixed)
        assert len(outs) == len(spec)
        for (h, w), p, o in zip(shapes, plist, outs):
            assert o.shape == (h, w) and o.dtype == np.float32
            if len(p) == 0:
                assert not o.any()
                continue
            ref = dmap_oracle.density_closed_form((h, w), p, fixed=fixed)
            assert_map_close(o, ref, f"batch {h}x{w} n={len(p)} fixed={fixed}")
            fn = dmap_gen.gaussian_filter_density_fixed if fixed else dmap_gen.gaussian_filter_density
            assert np.array_equal(o, fn(np.empty((h, w, 0)), p)), "batched and single-image launches differ"


def test_config4_full_set_matches_oracle():
    """The FULL BASELINE config-4 set (64 JHU-shaped images, sides 512..2048, 0..25 000 heads, float64 and float32
    points) through the batched API, adaptive and fixed: kNN neighbours bit-exact against scipy's KDTree, every map
    against the closed-form oracle (bit-identical up to the few pixels assert_map_close allows)."""
    from dgvcc_b200.utils import dmap_gen
    images = synthetic.config4_images()
    shapes = [s for s, _ in images]
    plist = [p for _, p in images]
    assert len(images) == 64 and any(len(p) == 0 for p in plist) and max(len(p) for p in plist) > 15000
    sig = {}
    for i, p in enumerate(plist):
        if len(p) > 3:
            p64 = np.ascontiguousarray(p, dtype=np.float64)
            rd, rl = dmap_oracle.knn4(p64)
            if i % 8 == 0:  # the device kNN on its own for every eighth image (all of them feed the maps below)
                dist, loc, sigma = dmap_gen.knn_sigma(p64)
                assert np.array_equal(loc, rl) and np.array_equal(dist, rd), f"kNN image {i}"
            sig[i] = (rd[:, 1] + rd[:, 2] + rd[:, 3]) * 0.1
    for fixed in (False, True):
        outs = dmap_gen.gaussian_filter_density_batch(shapes, plist, fixed=fixed)
        bad = 0
        for i, ((h, w), p, o) in enumerate(zip(shapes, plist, outs)):
            assert o.shape == (h, w) and o.dtype == np.float32
            if len(p) == 0:
                assert not o.any()
                continue
            p64 = np.ascontiguousarray(p, dtype=np.float64)
            ref = dmap_oracle.density_closed_form((h, w), p64, fixed=fixed, sigmas=None if fixed else sig.get(i))
            bad += assert_map_close(o, ref, f"config 4 image {i} ({h}x{w}, {len(p)} heads, fixed={fixed})")
        print(f"config 4, fixed={fixed}: {bad} pixels of {sum(h * w for h, w in shapes)} not bit-identical")


def test_batched_knn_bit_exact():
    import ctypes
    import torch
    from dgvcc_b200 import _native
    from dgvcc_b200.utils import dmap_gen
    counts = [0, 1, 3, 4, 257, 2048, 2049, 5000]
    plist = [synthetic.crowd_points(np.random.default_rng(200 + i), n, 1500, 1100, dtype=np.float64) for i, n in enumerate(counts)]
    plan = dmap_gen._Plan([(1100, 1500)] * len(counts), counts)
    pl = plan.plan
    dev = torch.device("cuda")
    meta = torch.from_numpy(plan.meta).to(dev)
    d_pts = torch.from_numpy(np.concatenate([p for p in plist if len(p)])).to(dev)
    idx = torch.empty((pl.total_heads, 4), dtype=torch.int32, device=dev)
    dist = torch.empty((pl.total_heads, 4), dtype=torch.float64, device=dev)
    sigma = torch.empty((pl.total_heads,), dtype=torch.float64, device=dev)
    kws = torch.empty((pl.knn_workspace_bytes,), dtype=torch.uint8, device=dev)
    _native.check(_native.lib().dgvcc_dmap_knn_sigma_batch(
        _native.ptr(d_pts), len(counts), _native.ptr(meta), ctypes.byref(pl), _native.ptr(idx), _native.ptr(dist),
        _native.ptr(sigma), _native.ptr(kws), pl.knn_workspace_bytes, _native.stream_ptr(dev)), "knn batch")
    idx, dist, sigma = idx.cpu().numpy(), dist.cpu().numpy(), sigma.cpu().numpy()
    for i, p in enumerate(plist):
        if not len(p):
            continue
        lo, hi = plan.pt_off[i], plan.pt_off[i + 1]
        rd, rl = dmap_oracle.knn4(p)
        assert np.array_equal(idx[lo:hi], rl) and np.array_equal(dist[lo:hi], rd), f"image {i} (n={len(p)})"
        ref_sigma = (rd[:, 1] + rd[:, 2] + rd[:, 3]) * 0.1 if len(p) > 3 else np.full(len(p), 15.0)
        assert np.array_equal(sigma[lo:hi], ref_sigma)


def test_batched_knn_fp32_filter_stays_exact_far_from_the_origin():
    """The batched search skips candidates through an fp32 bound; crowds far from the origin (large |coordinates|,
    small separations: the worst case for fp32) and near-coincident heads must still give KDTree's answer bit for bit."""
    import ctypes
    import torch
    from dgvcc_b200 import _native
    from dgvcc_b200.utils import dmap_gen
    rng = np.random.default_rng(321)
    clouds = [
        1.0e6 + rng.uniform(0, 300, size=(3000, 2)),                       # far from the origin
        np.concatenate([rng.uniform(0, 2000, size=(2500, 2)),              # tight pairs: separations ~1e-4 px
                        rng.uniform(0, 2000, size=(2500, 2))]) ,
        rng.uniform(-5.0e4, 5.0e4, size=(2600, 2)),                        # both signs, wide range
        (rng.uniform(0, 1500, size=(4100, 2))).astype(np.float32).astype(np.float64),
    ]
    clouds[1][2500:] = clouds[1][:2500] + rng.uniform(1e-5, 1e-4, size=(2500, 2))
    counts = [len(c) for c in clouds]
    plan = dmap_gen._Plan([(2048, 2048)] * len(clouds), counts)
    pl = plan.plan
    dev = torch.device("cuda")
    meta = torch.from_numpy(plan.meta).to(dev)
    d_pts = torch.from_numpy(np.concatenate(clouds)).to(dev)
    idx = torch.empty((pl.total_heads, 4), dtype=torch.int32, device=dev)
    dist = torch.empty((pl.total_heads, 4), dtype=torch.float64, device=dev)
    sigma = torch.empty((pl.total_heads,), dtype=torch.float64, device=dev)
    kws = torch.empty((pl.knn_workspace_bytes,), dtype=torch.uint8, device=dev)
    _native.check(_native.lib().dgvcc_dmap_knn_sigma_batch(
        _native.ptr(d_pts), len(counts), _native.ptr(meta), ctypes.byref(pl), _native.ptr(idx), _native.ptr(dist),
        _native.ptr(sigma), _native.ptr(kws), pl.knn_workspace_bytes, _native.stream_ptr(dev)), "knn batch")
    idx, dist = idx.cpu().numpy(), dist.cpu().numpy()
    for i, c in enumerate(clouds):
        lo, hi = plan.pt_off[i], plan.pt_off[i + 1]
        rd, rl = dmap_oracle.knn4(c)
        assert np.array_equal(dist[lo:hi], rd), f"cloud {i}: distances"
        assert np.array_equal(idx[lo:hi], rl), f"cloud {i}: indices"


def test_negative_beyond_size_raises_like_numpy():
    from dgvcc_b200.utils import dmap_gen
    with pytest.raises(IndexError):
        dmap_gen.gaussian_filter_density_fixed(np.empty((20, 20, 0)), np.array([[-30.0, 2.0]]))
