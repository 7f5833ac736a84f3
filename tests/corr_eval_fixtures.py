"""Seeded inputs of the CorrEval tests: PixelMask<float> rasters as (rows, cols, 2) float32 {value, valid} and
PixelMask<Vector2f> disparities as (rows, cols, 3) float32 {dx, dy, valid}."""
import numpy as np

METRICS = ("ncc", "stddev", "parabola_curvature", "cramer_rao")


def texture(rows, cols, seed, shift=(0.0, 0.0)):
    """A smooth random texture (a few sines) sampled at (x - shift_x, y - shift_y)."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:rows, 0:cols].astype(np.float64)
    xx, yy = xx - shift[0], yy - shift[1]
    img = np.zeros((rows, cols))
    for _ in range(5):
        fx, fy, ph = rng.uniform(0.15, 0.9), rng.uniform(0.15, 0.9), rng.uniform(0, 6.3)
        img += rng.uniform(0.3, 1.0) * np.sin(fx * xx + ph) * np.cos(fy * yy - ph)
    return img.astype(np.float32)


def masked(img, invalid_fraction=0.0, seed=0):
    """{value, valid} pairs; invalid pixels keep their value."""
    rng = np.random.default_rng(seed)
    out = np.stack([img, np.ones_like(img)], axis=-1).astype(np.float32)
    out[..., 1][rng.random(img.shape) < invalid_fraction] = 0.0
    return out


def smooth_disparity(rows, cols, seed, base=(2.3, -0.7), invalid_fraction=0.05):
    """A smooth fractional disparity around base with about invalid_fraction invalid pixels."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:rows, 0:cols].astype(np.float64)
    d = np.zeros((rows, cols, 3), np.float32)
    d[..., 0] = base[0] + 0.8 * np.sin(xx / 17.0 + 0.3) * np.cos(yy / 23.0) + 0.01 * xx
    d[..., 1] = base[1] + 0.6 * np.cos(xx / 19.0) * np.sin(yy / 13.0 + 0.7)
    d[..., 2] = (rng.random((rows, cols)) >= invalid_fraction).astype(np.float32)
    return d


def scene(rows, cols, seed, right_shape=None, invalid_fraction=0.05, base=(2.3, -0.7)):
    """A left / right pair related by about `base`, masks on both, and a smooth disparity."""
    rs = right_shape or (rows, cols)
    left = masked(texture(rows, cols, seed), invalid_fraction, seed + 1)
    right = masked(texture(rs[0], rs[1], seed, shift=base), invalid_fraction, seed + 2)
    return left, right, smooth_disparity(rows, cols, seed + 3, base, invalid_fraction)


def tiny_case(seed=41, bbox=(4, 6, 44, 36)):
    """Disparity components far below the ulp of the pixel positions, of both signs: the first sum
    double(left_pix) + double(d) loses them.  dy >= 0 everywhere except one valid sampled pixel on the bbox's first row
    with dy = -1e-20, which therefore holds the right crop's minimum; the sum rounds it to the integer row, not below."""
    left, right, disp = scene(48, 56, seed)
    rng = np.random.default_rng(seed)
    disp[..., 1] = np.abs(disp[..., 1])
    tiny = np.array([1e-20, 1e-13, 3e-9, 1e-30], np.float32)
    pick = rng.random(disp.shape[:2]) < 0.3
    for ch in (0, 1):
        vals = tiny[rng.integers(0, tiny.size, disp.shape[:2])] * (1 if ch else rng.choice([-1.0, 1.0], disp.shape[:2]))
        disp[..., ch] = np.where(pick, vals.astype(np.float32), disp[..., ch])
    x0, y0 = bbox[0], bbox[1]
    disp[y0, x0 + 2] = (-1e-20, -1e-20, 1.0)
    return left, right, disp, bbox
