"""f64 numpy reference of the non-local-means film filter of drt_cuda_film_denoise (include/drt_cuda.h states the filter)."""
import numpy as np
from numpy.lib.stride_tricks import sliding_window_view


def guide(mean, m2, filt, w):
    """(Y, v, usable) per pixel, f64, from planes mean[npix, N], m2[npix, N], filter[npix] and luminance weights w[N]."""
    mean = np.asarray(mean, np.float64)
    m2 = np.asarray(m2, np.float64)
    n = np.asarray(filt, np.float64)
    usable = (n >= 2) & np.isfinite(mean).all(axis=1) & np.isfinite(m2).all(axis=1)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        y = mean @ w
        v = (np.sqrt(m2 / (n * (n - 1))[:, None]) @ w) ** 2
    return np.where(usable, y, 0.0), np.where(usable, v, 0.0), usable


def denoise(mean, m2, filt, w, width, height, r=7, f=3, k=0.45):
    """The filtered mean plane [W*H, N] (f64) of a film; unusable pixels keep their mean."""
    mean = np.asarray(mean).reshape(width * height, -1)
    nwl = mean.shape[1]
    y, v, usable = guide(mean, np.asarray(m2).reshape(width * height, nwl), filt, np.asarray(w, np.float64))
    y, v, usable = y.reshape(height, width), v.reshape(height, width), usable.reshape(height, width)
    spec = np.where(usable.reshape(-1, 1), mean.astype(np.float64), 0.0).reshape(height, width, nwl)
    R = r + f
    yp, vp = np.pad(y, R, mode="edge"), np.pad(v, R, mode="edge")
    up = np.pad(usable, r, mode="constant", constant_values=False)
    sp = np.pad(spec, ((r, r), (r, r), (0, 0)))
    kk = float(k) * float(k)
    # a: cells of the image and its f halo (border replicated), b: the same cells shifted by (dx, dy)
    ya, va = yp[r:r + height + 2 * f, r:r + width + 2 * f], vp[r:r + height + 2 * f, r:r + width + 2 * f]
    num = np.zeros((height, width, nwl))
    den = np.zeros((height, width))
    for dy in range(-r, r + 1):
        for dx in range(-r, r + 1):
            yb = yp[r + dy:r + dy + height + 2 * f, r + dx:r + dx + width + 2 * f]
            vb = vp[r + dy:r + dy + height + 2 * f, r + dx:r + dx + width + 2 * f]
            with np.errstate(over="ignore", invalid="ignore"):
                d = ((ya - yb) ** 2 - (va + np.minimum(va, vb))) / (1e-10 + kk * (va + vb))
                d2 = sliding_window_view(d, (2 * f + 1, 2 * f + 1)).mean(axis=(2, 3))
                wt = np.exp(-np.maximum(0.0, d2))
            wt = np.where(up[r + dy:r + dy + height, r + dx:r + dx + width], wt, 0.0)
            if dx == 0 and dy == 0:
                wt = np.ones_like(wt)
            num += wt[:, :, None] * sp[r + dy:r + dy + height, r + dx:r + dx + width]
            den += wt
    with np.errstate(invalid="ignore", divide="ignore"):
        out = num / den[:, :, None]
    out = out.reshape(width * height, nwl)
    return np.where(usable.reshape(-1, 1), out, mean.astype(np.float64))


def luminance_weights(tables, n):
    """w_l = cmf_y * ref_white as the device holds them (f32, drt_fill_rgb_tables), widened to f64."""
    return (np.array(tables.cmf_y[:n]) * np.array(tables.ref_white[:n])).astype(np.float32).astype(np.float64)
