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


def test_negative_m2_counts_as_zero_variance():
    """v = (sum_l w_l sqrt(max(0, M2_l / (n (n - 1)))))^2: a negative M2 value adds nothing to v and makes no NaN."""
    w, h = 8, 6
    mean, m2, filt = _film(w, h, 8)
    m2[13, 2] = -1e-30
    m2[20, :] = -4.0
    y, v, usable = denoise_ref.guide(mean, m2, filt, W_L)
    zeroed = m2.copy()
    zeroed[13, 2] = 0.0
    zeroed[20, :] = 0.0
    y0, v0, _ = denoise_ref.guide(mean, zeroed, filt, W_L)
    assert usable.all() and np.array_equal(v, v0) and v[20] == 0.0
    out = denoise_ref.denoise(mean, m2, filt, W_L, w, h, r=2, f=1)
    assert np.isfinite(out).all()
    assert np.array_equal(out, denoise_ref.denoise(mean, zeroed, filt, W_L, w, h, r=2, f=1))


def test_guide_beyond_flt_max_is_unusable():
    """A pixel whose Y or v lies beyond FLT_MAX (decided in f64, from finite statistics) is copied bit for bit and weighs nothing."""
    w, h = 9, 7
    mean, m2, filt = _film(w, h, 9)
    w2 = 2.0 * W_L                                              # sum 2: a guide can pass FLT_MAX with finite statistics
    mean[10] = np.float32(3e38)                                 # |Y| = 3e38 x 2 > FLT_MAX
    m2[30], filt[30] = np.float32(3e38), 2.0                    # v = (2 sqrt(1.5e38))^2 > FLT_MAX
    mean[40] = np.float32(1e36)                                 # Y = 2e36: finite, usable
    y, v, usable = denoise_ref.guide(mean, m2, filt, w2)
    assert not usable[10] and not usable[30] and usable[40] and usable.sum() == w * h - 2
    out = denoise_ref.denoise(mean, m2, filt, w2, w, h, r=2, f=1)
    for p in (10, 30):
        assert np.array_equal(out[p].astype(np.float32), mean[p])
    assert np.isfinite(out).all()
    # as far as the other pixels are concerned the two are like n = 1 pixels
    f1 = filt.copy()
    f1[[10, 30]] = 1.0
    keep = usable.copy()
    assert np.array_equal(out[keep], denoise_ref.denoise(mean, m2, f1, w2, w, h, r=2, f=1)[keep])


def test_nan_distance_takes_no_weight():
    """A NaN patch distance gives weight 0, not the weight 1 that max(0, NaN) = 0 would give.  With k^2 = inf every distance of a
    zero-variance film is 0 / (1e-10 + inf x 0) = NaN, so every pixel keeps its own mean."""
    w, h = 6, 5
    mean, _, filt = _film(w, h, 11)
    out = denoise_ref.denoise(mean, np.zeros_like(mean), filt, W_L, w, h, r=2, f=1, k=1e200)
    assert np.array_equal(out, mean.astype(np.float64))


@pytest.mark.parametrize("seed", range(4))
def test_window_equals_whole_frame(seed):
    """denoise_window equals denoise on random windows of small films, corners included."""
    rng = np.random.default_rng(100 + seed)
    w, h = 23, 17
    mean, m2, filt = _film(w, h, 10 + seed)
    filt[rng.integers(0, w * h, 5)] = 1.0
    r, f = [(1, 0), (2, 1), (4, 3), (7, 2)][seed]
    full = denoise_ref.denoise(mean, m2, filt, W_L, w, h, r=r, f=f).reshape(h, w, N)
    wins = [(0, 0, 4, 3), (w - 5, 0, w, 6), (0, h - 2, 7, h), (w - 1, h - 1, w, h)]
    for _ in range(4):
        x0, y0 = rng.integers(0, w), rng.integers(0, h)
        wins.append((x0, y0, rng.integers(x0 + 1, w + 1), rng.integers(y0 + 1, h + 1)))
    for x0, y0, x1, y1 in wins:
        got = denoise_ref.denoise_window(mean, m2, filt, W_L, w, h, x0, y0, x1, y1, r=r, f=f)
        assert np.array_equal(got, full[y0:y1, x0:x1].reshape(-1, N)), (x0, y0, x1, y1)


# (width, height, N, seed, (r, f) pairs) of films of tests/test_gpu_denoise_edges.py: the 45 x 19 film of its radius sweep, the 41 x 13
# films of its wavelength layouts and the larger films of its shape sweep (smaller ones have too few neighbours to weigh)
def _edge_cases():
    import test_gpu_denoise_edges as edges
    cases = [(45, 19, 69, 19, [(1, 0), (1, 4), (4, 2), (7, 3), (15, 0), (15, 4)])]
    cases += [(41, 13, n, 500 + n, [(3, 1)] + ([(7, 3)] if n in (33, 97) else [])) for n in sorted(edges.GRID)]
    cases += [(w, h, 18, edges.shape_seed(w, h), [(1, 0), (7, 3)]) for w in (33, 100) for h in (9, 33)]
    return edges, cases


def _weights(n):
    import common
    import test_gpu_denoise_edges as edges
    grid = {} if n == 69 else dict(zip(("min_wl", "max_wl", "wl_interval"), edges.GRID[n]))
    cfg, tables, sc, camera = common.load("init_cornell", 8, 8, 1, 4, **grid)
    return denoise_ref.luminance_weights(tables, n)


@pytest.mark.parametrize("case", range(len(_edge_cases()[1])))
def test_edge_films_tell_slips_apart(case):
    """On each synthetic film of the GPU edge suite, every indexing slip of denoise_ref.SLIPS moves the reference output 10x past the
    GPU tolerance (1e-4 relative at the 99.9th percentile or 1e-3 at the maximum), and the weights are informative: the median share of
    a pixel's weight from its neighbours lies in [0.3, 0.95] (with a single-pixel patch, f = 0, only at r = 1: a one-cell patch of a
    smooth film matches most of a wide search window)."""
    edges, cases = _edge_cases()
    w, h, n, seed, pairs = cases[case]
    yw = _weights(n)
    f = edges.film(w, h, n, seed)
    for r, pf in pairs:
        ref = denoise_ref.denoise(f["mean"], f["m2"], f["filter"], yw, w, h, r=r, f=pf)
        floor = 1e-6 * np.abs(ref).max()
        for slip in denoise_ref.SLIPS:
            if slip == "zero_pad" and pf == 0:
                continue                    # a one-cell patch reads no cell outside the image
            alt = denoise_ref.denoise(f["mean"], f["m2"], f["filter"], yw, w, h, r=r, f=pf, slip=slip)
            rel = np.abs(alt - ref) / np.maximum(np.abs(ref), floor)
            assert np.quantile(rel, 0.999) >= 1e-3 or rel.max() >= 1e-2, (r, pf, slip, np.quantile(rel, 0.999), rel.max())
        if pf > 0 or r == 1:
            share = np.median(denoise_ref.neighbour_share(f["mean"], f["m2"], f["filter"], yw, w, h, r=r, f=pf))
            assert 0.3 <= share <= 0.95, (r, pf, share)
