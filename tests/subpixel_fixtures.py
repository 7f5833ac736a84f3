"""Inputs for the sub-pixel refinement tests (PyramidSubpixelView), shared by the CPU and GPU test modules."""
import numpy as np


def _bicubic_u8(img, xs, ys):
    """BicubicInterpolation over ZeroEdgeExtension (Image/Interpolation.h:138-185) sampled at (xs, ys), rounded and
    clamped to uint8 as channel_cast_round_and_clamp does."""
    src = np.pad(img.astype(np.float64), 2)
    x = np.floor(xs).astype(np.int64)
    y = np.floor(ys).astype(np.int64)
    nx, ny = xs - x, ys - y
    s = [((2 - nx) * nx - 1) * nx, (3 * nx - 5) * nx * nx + 2, ((4 - 3 * nx) * nx + 1) * nx, (nx - 1) * nx * nx]
    t = [((2 - ny) * ny - 1) * ny, (3 * ny - 5) * ny * ny + 2, ((4 - 3 * ny) * ny + 1) * ny, (ny - 1) * ny * ny]
    h, w = img.shape

    def at(xx, yy):
        ok = (xx >= -2) & (xx < w + 2) & (yy >= -2) & (yy < h + 2)
        return np.where(ok, src[np.clip(yy + 2, 0, h + 3), np.clip(xx + 2, 0, w + 3)], 0.0)

    res = 0.0
    for r in range(4):
        row = 0.0
        for c in range(4):
            row = row + s[c] * at(x - 1 + c, y - 1 + r)
        res = res + t[r] * row
    res = res * 0.25
    exact = (xs == x) & (ys == y)
    res = np.where(exact, at(x, y), res)
    return np.clip(np.floor(res + 0.5), 0, 255).astype(np.uint8)


def _rand48_uniform01(seed, n):
    """boost::rand48 gen(seed) (x0 = seed << 16 | 0x330E; x <- (0x5DEECE66D x + 0xB) mod 2^48; output x >> 17) through
    boost::uniform_01<double>: output / 2^31."""
    x = ((seed << 16) | 0x330E) & ((1 << 48) - 1)
    out = np.empty(n, np.float64)
    for k in range(n):
        x = (0x5DEECE66D * x + 0xB) & ((1 << 48) - 1)
        out[k] = (x >> 17) * (1.0 / 2147483648.0)
    return out


def kat_case(istretch, size=100):
    """TestSubPixel.cxx:47-65.  image1 = transform(channel_cast_rescale<uint8>(uniform_noise_view(rand48(10), 100, 100)),
    AffineTransform(3 I, 0), ZeroEdgeExtension, BicubicInterpolation): the interpolation view rasterises the edge-extended
    noise over the reverse-transformed bbox grown to integers and padded by the bicubic pixel buffer
    (Image/Interpolation.h:284-291, Math/Transform.h:176-186, Math/BBox.tcc:368-388) -- [-2, 36)^2, so the in-image
    36 x 36 pixels are drawn in raster order -- then samples it at the reverse-mapped positions (Math/Transform.h:333-338,
    inverse of Math/Matrix.h:2209-2216).  image2 squeezes image1 by `stretch` the same way.  Inputs are
    channel_cast_rescale<float> of both, the starting disparity int32(stretch * i + translation - i)."""
    stretch = np.float32(np.float32(istretch) / np.float32(100))
    drawn = 36
    u = _rand48_uniform01(10, drawn * drawn).reshape(drawn, drawn)
    noise = np.zeros((size, size), np.uint8)
    noise[:drawn, :drawn] = np.minimum(np.maximum(u, 0.0), 1.0) * 255.0     # channel_cast_rescale<uint8>: truncation
    yy, xx = np.mgrid[0:size, 0:size].astype(np.float64)
    third = 3.0 / 9.0
    image1 = _bicubic_u8(noise, third * xx, third * yy)
    half = size // 2
    translation = np.float32(np.float32(half) - np.float32(half) * stretch)
    inv = 1.0 / float(stretch)
    image2 = _bicubic_u8(image1, inv * (xx - float(translation)), yy)
    disp = np.zeros((size, size, 3), np.float32)
    i = np.arange(size, dtype=np.float32)
    disp[:, :, 0] = ((stretch * i + translation) - i).astype(np.int32)[None, :]
    disp[:, :, 2] = 1.0
    left = (image1.astype(np.float64) * (1.0 / 255.0)).astype(np.float32)
    right = (image2.astype(np.float64) * (1.0 / 255.0)).astype(np.float32)
    return left, right, disp, float(stretch), float(translation)


def check_error(disp, stretch, translation):
    """TestSubPixel.cxx:67-82, including its `+ disparity[1]` term: a float per pixel, summed in double with the
    column index outermost."""
    size = disp.shape[0]
    st, tr = np.float32(stretch), np.float32(translation)
    error = 0.0
    invalid = 0
    for i in range(size):
        expected = np.float32(np.float32(st * np.float32(i)) + tr) - np.float32(i)
        for j in range(size):
            d = disp[j, i]
            error += float(np.float32(d[1] + np.float32(abs(np.float32(d[0] - expected)))))
            invalid += int(d[2] == 0)
    return error / (float(size) * float(size)), invalid


def smooth_pair(h, w, shift=(1.3, -0.6), seed=3, scale=1.0):
    """A smooth random texture and a sub-pixel shifted copy, values in [0, scale]; an integer starting disparity with
    about 5 % invalid pixels."""
    rng = np.random.default_rng(seed)
    base = rng.random((h // 4 + 4, w // 4 + 4))
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64)

    def sample(x, y):
        x4, y4 = x / 4.0 + 1, y / 4.0 + 1
        x0, y0 = np.floor(x4).astype(int), np.floor(y4).astype(int)
        fx, fy = x4 - x0, y4 - y0
        x0 = np.clip(x0, 0, base.shape[1] - 2)
        y0 = np.clip(y0, 0, base.shape[0] - 2)
        return ((1 - fx) * (1 - fy) * base[y0, x0] + fx * (1 - fy) * base[y0, x0 + 1] + (1 - fx) * fy * base[y0 + 1, x0]
                + fx * fy * base[y0 + 1, x0 + 1])

    left = (sample(xx, yy) * scale).astype(np.float32)
    right = (sample(xx - shift[0], yy - shift[1]) * scale).astype(np.float32)
    disp = np.zeros((h, w, 3), np.float32)
    disp[:, :, 0] = np.round(shift[0])
    disp[:, :, 1] = np.round(shift[1])
    disp[:, :, 2] = (rng.random((h, w)) > 0.05).astype(np.float32)
    return left, right, disp


def chain_case(w=40, h=24):
    """An invalidation chain for a 3 x 3 kernel (at least 4 good pixels needed): row 10 is valid for x in [10, 30) and
    row 11 at every third pixel, so every row-10 pixel has 4 good pixels against the input validity.  (10, 10) has only
    3 and is invalidated; scanning in place, that leaves (11, 10) with 3, and so on along the row."""
    left, right, disp = smooth_pair(h, w, seed=11)
    disp[:, :, 2] = 0.0
    disp[10, 10:30, 2] = 1.0
    disp[11, 12:30:3, 2] = 1.0
    disp[11, 9, 2] = 1.0
    return left, right, disp
