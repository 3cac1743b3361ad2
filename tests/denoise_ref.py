"""f64 numpy reference of the non-local-means film filter of drt_cuda_film_denoise (include/drt_cuda.h states the filter)."""
import numpy as np
from numpy.lib.stride_tricks import sliding_window_view

FLT_MAX = float(np.finfo(np.float32).max)

# indexing slips a kernel could make, for checking that a film tells them apart from the filter (denoise(..., slip=...))
SLIPS = ("column", "row", "patch", "zero_pad", "wavelength", "v_a")


def guide(mean, m2, filt, w):
    """(Y, v, usable) per pixel, f64, from planes mean[npix, N], m2[npix, N], filter[npix] and luminance weights w[N].
    A negative M2 counts as zero variance; a pixel whose Y or v lies beyond FLT_MAX (no finite f32 guide) is unusable."""
    mean = np.asarray(mean, np.float64)
    m2 = np.asarray(m2, np.float64)
    n = np.asarray(filt, np.float64)
    usable = (n >= 2) & np.isfinite(mean).all(axis=1) & np.isfinite(m2).all(axis=1)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        y = mean @ w
        v = (np.sqrt(np.maximum(0.0, m2 / (n * (n - 1))[:, None])) @ w) ** 2
        usable &= (np.abs(y) <= FLT_MAX) & (v <= FLT_MAX)
    return np.where(usable, y, 0.0), np.where(usable, v, 0.0), usable


def denoise(mean, m2, filt, w, width, height, r=7, f=3, k=0.45, slip=None):
    """The filtered mean plane [W*H, N] (f64) of a film; unusable pixels keep their mean.  `slip` (one of SLIPS) computes the
    filter with that indexing mistake instead."""
    return _nlm(mean, m2, filt, w, width, height, r, f, k, slip)[0]


def neighbour_share(mean, m2, filt, w, width, height, r=7, f=3, k=0.45):
    """Per usable pixel, the share of its weight sum that comes from pixels other than itself: 1 - 1 / sum_q wt(p, q)."""
    _, den, usable = _nlm(mean, m2, filt, w, width, height, r, f, k, None)
    return 1.0 - 1.0 / den.reshape(-1)[usable.reshape(-1)]


def _nlm(mean, m2, filt, w, width, height, r, f, k, slip):
    """(filtered mean [W*H, N], weight sums [H, W], usable [H, W])."""
    mean = np.asarray(mean).reshape(width * height, -1)
    nwl = mean.shape[1]
    y, v, usable = guide(mean, np.asarray(m2).reshape(width * height, nwl), filt, np.asarray(w, np.float64))
    y, v, usable = y.reshape(height, width), v.reshape(height, width), usable.reshape(height, width)
    spec = np.where(usable.reshape(-1, 1), mean.astype(np.float64), 0.0).reshape(height, width, nwl)
    if slip == "wavelength":                      # out_l takes the spectra of wavelength l + 1 (the last one of l)
        spec = np.concatenate([spec[:, :, 1:], spec[:, :, -1:]], axis=2)
    pf = f + 1 if slip == "patch" else f
    R = r + pf
    pad = dict(mode="constant") if slip == "zero_pad" else dict(mode="edge")
    yp, vp = np.pad(y, R, **pad), np.pad(v, R, **pad)
    # usable flags and spectra padded by r + 1: the column and row slips read one pixel past the search window
    up = np.pad(usable, r + 1, mode="constant", constant_values=False)
    sp = np.pad(spec, ((r + 1, r + 1), (r + 1, r + 1), (0, 0)))
    sx, sy = (1 if slip == "column" else 0), (1 if slip == "row" else 0)
    kk = float(k) * float(k)
    # a: cells of the image and its f halo (border replicated), b: the same cells shifted by (dx, dy)
    ya, va = yp[r:r + height + 2 * pf, r:r + width + 2 * pf], vp[r:r + height + 2 * pf, r:r + width + 2 * pf]
    num = np.zeros((height, width, nwl))
    den = np.zeros((height, width))
    for dy in range(-r, r + 1):
        for dx in range(-r, r + 1):
            yb = yp[r + dy:r + dy + height + 2 * pf, r + dx:r + dx + width + 2 * pf]
            vb = vp[r + dy:r + dy + height + 2 * pf, r + dx:r + dx + width + 2 * pf]
            with np.errstate(over="ignore", invalid="ignore"):
                d = ((ya - yb) ** 2 - (va + (va if slip == "v_a" else np.minimum(va, vb)))) / (1e-10 + kk * (va + vb))
                d2 = sliding_window_view(d, (2 * pf + 1, 2 * pf + 1)).mean(axis=(2, 3))
                wt = np.where(np.isnan(d2), 0.0, np.exp(-np.maximum(0.0, d2)))     # a NaN distance takes no weight
            qy, qx = r + 1 + dy, r + 1 + dx
            wt = np.where(up[qy:qy + height, qx:qx + width], wt, 0.0)
            if dx == 0 and dy == 0:
                wt = np.ones_like(wt)
            num += wt[:, :, None] * sp[qy + sy:qy + sy + height, qx + sx:qx + sx + width]
            den += wt
    with np.errstate(invalid="ignore", divide="ignore"):
        out = num / den[:, :, None]
    out = out.reshape(width * height, nwl)
    return np.where(usable.reshape(-1, 1), out, mean.astype(np.float64)), den, usable


def host_array(a):
    """A numpy view of a numpy array or a (device) torch tensor."""
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def denoise_window(mean, m2, filt, w, width, height, x0, y0, x1, y1, r=7, f=3, k=0.45):
    """denoise() of the pixels x0 <= x < x1, y0 <= y < y1 only, as [(y1 - y0) * (x1 - x0), N] (row-major): the reference runs on the
    window and a margin of r + f, clipped to the image.  Every pixel and patch cell the window's pixels read lies within r + f of them,
    so the result equals denoise() of the whole frame there.  The planes may be numpy arrays or torch tensors (device ones too); only
    the window and its margin are read."""
    R = r + f
    xa, ya, xb, yb = max(0, x0 - R), max(0, y0 - R), min(width, x1 + R), min(height, y1 + R)
    cw, ch = xb - xa, yb - ya
    sub = [host_array(p.reshape(height, width, -1)[ya:yb, xa:xb]).reshape(cw * ch, -1) for p in (mean, m2)]
    fs = host_array(filt.reshape(height, width)[ya:yb, xa:xb]).reshape(cw * ch)
    out = denoise(sub[0], sub[1], fs, w, cw, ch, r=r, f=f, k=k).reshape(ch, cw, -1)
    return out[y0 - ya:y1 - ya, x0 - xa:x1 - xa].reshape((y1 - y0) * (x1 - x0), -1)


def luminance_weights(tables, n):
    """w_l = cmf_y * ref_white as the device holds them (f32, drt_fill_rgb_tables), widened to f64."""
    return (np.array(tables.cmf_y[:n]) * np.array(tables.ref_white[:n])).astype(np.float32).astype(np.float64)
