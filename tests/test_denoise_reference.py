"""CPU tier: the f64 reference of the non-local-means film filter (tests/denoise_ref.py) keeps the properties drt_cuda.h states."""
import numpy as np
import pytest

import denoise_ref

N = 5
W_L = np.array([0.1, 0.3, 0.4, 0.15, 0.05])


def _film(width, height, seed, spp=16):
    """A noisy film: a smooth image with per-pixel noise, M2 of `spp` samples."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:height, 0:width]
    base = (1.0 + 0.5 * np.sin(xx / 3.0) * np.cos(yy / 4.0)).reshape(-1, 1) * np.linspace(0.5, 1.5, N)
    mean = (base * (1.0 + 0.1 * rng.standard_normal(base.shape))).astype(np.float32)
    m2 = (0.01 * base ** 2 * (spp - 1) * rng.uniform(0.5, 1.5, base.shape)).astype(np.float32)
    return mean, m2, np.full(width * height, spp, np.float32)


def test_constant_film_is_unchanged():
    w, h = 11, 9
    mean = np.tile(np.linspace(0.2, 1.0, N, dtype=np.float32), (w * h, 1))
    m2 = np.full((w * h, N), 0.3, np.float32)
    out = denoise_ref.denoise(mean, m2, np.full(w * h, 8, np.float32), W_L, w, h)
    assert np.allclose(out, mean, rtol=1e-12, atol=0)


def test_zero_variance_distinct_luminances_is_the_identity():
    w, h = 10, 7
    lum = np.random.default_rng(1).permutation(w * h).astype(np.float64) + 1.0
    mean = (lum[:, None] * np.ones(N)).astype(np.float32)
    out = denoise_ref.denoise(mean, np.zeros_like(mean), np.full(w * h, 4, np.float32), W_L, w, h, r=3, f=1)
    assert np.array_equal(out.astype(np.float32), mean)


def test_self_weight_is_one():
    """With r = 1 and neighbours far in luminance, every pixel keeps its own mean exactly (its own weight is 1, the others 0); with
    equal neighbours the weights are 1 (wt(p, p) = 1, and d2 <= 0 for patches of equal luminance)."""
    w, h = 6, 5
    mean, m2, filt = _film(w, h, 2)
    y, v, _ = denoise_ref.guide(mean, m2, filt, W_L)
    assert np.all(v > 0)
    # luminances far apart relative to the noise
    scale = (1.0 + 50.0 * np.random.default_rng(7).permutation(w * h))[:, None]
    far = (mean * scale).astype(np.float32)
    out = denoise_ref.denoise(far, m2, filt, W_L, w, h, r=1, f=0)
    assert np.allclose(out, far, rtol=1e-9)
    flat = np.tile(mean[:1], (w * h, 1))
    out = denoise_ref.denoise(flat, np.tile(m2[:1], (w * h, 1)), filt, W_L, w, h, r=1, f=0)
    assert np.allclose(out, flat, rtol=1e-12)


def test_unusable_pixels_pass_through():
    w, h = 9, 8
    mean, m2, filt = _film(w, h, 3)
    filt[5] = 1.0                      # n = 1
    mean[17, 2] = np.nan               # NaN mean
    m2[30, 0] = np.inf                 # infinite M2
    filt[40] = 0.0                     # empty
    mean[40] = 0.0
    out = denoise_ref.denoise(mean, m2, filt, W_L, w, h, r=2, f=1)
    for p in (5, 17, 30, 40):
        assert np.array_equal(out[p].astype(np.float32), mean[p], equal_nan=True), p
    others = np.setdiff1d(np.arange(w * h), [5, 17, 30, 40])
    assert np.isfinite(out[others]).all()
    assert not np.allclose(out[others], mean[others])     # the usable pixels are filtered


def test_unusable_neighbours_take_no_weight():
    """Changing the spectrum of an unusable pixel (n = 1) changes nothing else: it enters no sum."""
    w, h = 8, 6
    mean, m2, filt = _film(w, h, 4)
    filt[10] = 1.0
    a = denoise_ref.denoise(mean, m2, filt, W_L, w, h, r=2, f=1)
    mean2 = mean.copy()
    mean2[10] *= 7.0
    m2b = m2.copy()
    m2b[10] *= 3.0
    b = denoise_ref.denoise(mean2, m2b, filt, W_L, w, h, r=2, f=1)
    keep = np.arange(w * h) != 10
    assert np.array_equal(a[keep], b[keep])


def test_black_pixels_next_to_lit_ones_keep_their_edge():
    """Culled black pixels (all samples zero: Y = v = 0) beside noisy lit ones stay black, and the lit ones take no black."""
    w, h = 12, 8
    mean, m2, filt = _film(w, h, 5)
    black = (np.arange(w * h) % w) < 4
    mean[black] = 0.0
    m2[black] = 0.0
    out = denoise_ref.denoise(mean, m2, filt, W_L, w, h)
    assert np.array_equal(out[black], np.zeros_like(out[black]))
    lit = ~black
    assert (out[lit] @ W_L).min() > 0.5 * (mean[lit].astype(np.float64) @ W_L).min()


@pytest.mark.parametrize("r,f", [(1, 0), (2, 1), (4, 2)])
def test_border_clamps(r, f):
    """Patch cells outside the image take the nearest border pixel: the reference equals a direct loop over offsets and patch cells."""
    w, h = 7, 5
    mean, m2, filt = _film(w, h, 6)
    filt[3] = 1.0
    k = 0.45
    out = denoise_ref.denoise(mean, m2, filt, W_L, w, h, r=r, f=f, k=k)
    y, v, usable = denoise_ref.guide(mean, m2, filt, W_L)
    y, v, usable = y.reshape(h, w), v.reshape(h, w), usable.reshape(h, w)
    spec = mean.astype(np.float64).reshape(h, w, N)

    def at(a, yy, xx):
        return a[min(max(yy, 0), h - 1), min(max(xx, 0), w - 1)]

    for py in range(h):
        for px in range(w):
            if not usable[py, px]:
                continue
            num, den = np.zeros(N), 0.0
            for dy in range(-r, r + 1):
                for dx in range(-r, r + 1):
                    qy, qx = py + dy, px + dx
                    if not (0 <= qy < h and 0 <= qx < w and usable[qy, qx]):
                        continue
                    d = []
                    for oy in range(-f, f + 1):
                        for ox in range(-f, f + 1):
                            ya, va = at(y, py + oy, px + ox), at(v, py + oy, px + ox)
                            yb, vb = at(y, qy + oy, qx + ox), at(v, qy + oy, qx + ox)
                            d.append(((ya - yb) ** 2 - (va + min(va, vb))) / (1e-10 + k * k * (va + vb)))
                    wt = 1.0 if (dx, dy) == (0, 0) else np.exp(-max(0.0, float(np.mean(d))))
                    num += wt * spec[qy, qx]
                    den += wt
            assert np.allclose(out[py * w + px], num / den, rtol=1e-12, atol=0), (px, py)
