"""CPU oracle for the density-map generator -- TEST INFRASTRUCTURE, not product code.

Restates /root/reference/utils/dmap_gen.py:14-81.  Two levels:

* ``density_reference_like``: the reference's own algorithm with the same third-party calls
  (scipy.spatial.KDTree.query k=4, scipy.ndimage.gaussian_filter of a one-hot image per point).
  O(N*H*W*r): only for small cases.
* ``density_closed_form``: the closed form of that one-hot filter (SURVEY.md section 8c):
  ``fl32(f64(fl32(w[dy])) * w[dx])`` with ``w`` = scipy's normalised fp64 1-D kernel of radius
  ``int(truncate*sigma + 0.5)``, stamps added in ascending point order in fp32.  Bit-identical to
  the level above (tests/test_oracle_dmap.py) and fast enough for full-size images.

Third-party arithmetic (KDTree, gaussian_filter) is unpinned by the reference (no requirements
file); the de-facto pin is scipy 1.18.1 of this image, and tests/golden/dmap_*.npz hold outputs of
the unmodified reference functions.
"""
import numpy as np
from scipy.ndimage import gaussian_filter
from scipy.spatial import KDTree


def knn4(points):
    """distances [N,4] f64 / locations [N,4] of dmap_gen.py:34-36 (column 0 is the point itself)."""
    tree = KDTree(np.array(points, copy=True), leafsize=2048)
    return tree.query(points, k=4)


def adaptive_sigmas(points):
    """sigma per point, dmap_gen.py:45-48: 0.1 * (d1 + d2 + d3) when there are more than 3 points, else 15.
    The tree is built for any number of points (dmap_gen.py:34-36), so NaN / inf heads raise ValueError here."""
    n = len(points)
    d, _ = knn4(points)
    if n > 3:
        return (d[:, 1] + d[:, 2] + d[:, 3]) * 0.1
    return np.full((n,), 15.0)


def in_bounds(points, shape):
    """dmap_gen.py:41: int() truncation toward zero, test against the image size only from above."""
    keep = np.zeros(len(points), dtype=bool)
    for i, pt in enumerate(points):
        keep[i] = int(pt[1]) < shape[0] and int(pt[0]) < shape[1]
    return keep


def density_reference_like(shape, points, fixed=False):
    density = np.zeros(shape, dtype=np.float32)
    if len(points) == 0:
        return density
    sig = None if fixed else adaptive_sigmas(points)
    for i, pt in enumerate(points):
        if not (int(pt[1]) < shape[0] and int(pt[0]) < shape[1]):
            continue
        onehot = np.zeros(shape, dtype=np.float32)
        onehot[int(pt[1]), int(pt[0])] = 1.0
        if fixed:
            density += gaussian_filter(onehot, 4, truncate=7 / 4, mode="constant")
        else:
            density += gaussian_filter(onehot, sig[i], mode="constant")
    return density


def kernel1d(sigma, truncate):
    """scipy.ndimage._filters._gaussian_kernel1d(sigma, 0, int(truncate*sigma+0.5)); identity when sigma <= 1e-15."""
    sd = float(sigma)
    if not sd > 1e-15:
        return np.ones(1), 0
    radius = int(truncate * sd + 0.5)
    sigma2 = sd * sd
    x = np.arange(-radius, radius + 1)
    phi = np.exp(-0.5 / sigma2 * x ** 2)
    return phi / phi.sum(), radius


def density_closed_form(shape, points, fixed=False, sigmas=None, truncate=None):
    """``truncate``: scipy's, 7/4 (fixed) or 4 (adaptive) by default."""
    h, w = shape
    density = np.zeros(shape, dtype=np.float32)
    if len(points) == 0:
        return density
    if sigmas is None:
        sigmas = np.full(len(points), 4.0) if fixed else adaptive_sigmas(points)
    if truncate is None:
        truncate = 7 / 4 if fixed else 4.0
    for i, pt in enumerate(points):
        iy, ix = int(pt[1]), int(pt[0])
        if not (iy < h and ix < w):
            continue
        if iy < 0:
            iy += h  # numpy negative indexing of the one-hot write
        if ix < 0:
            ix += w
        wk, r = kernel1d(sigmas[i], truncate)
        y0, y1 = max(0, iy - r), min(h, iy + r + 1)
        x0, x1 = max(0, ix - r), min(w, ix + r + 1)
        wy = wk[y0 - iy + r:y1 - iy + r].astype(np.float32).astype(np.float64)
        wx = wk[x0 - ix + r:x1 - ix + r]
        density[y0:y1, x0:x1] += (wy[:, None] * wx[None, :]).astype(np.float32)
    return density
