"""CPU tier: numpy model of the compact-record replay and its film statistics (drt_render.cuh: replay_compact, BatchStats,
PixelFilm::add_batch), against the forward replay and the per-sample Welford update they replace.

Backward (Horner) replay: a path of bounces b with next-event spectra n_b and sampled-direction spectra s_b, ending on the light
(e = 1) or not (e = 0), has radiance E * r with r = n_0 + s_0 (n_1 + s_1 (... (n_last + s_last e))); the forward replay carries
u = throughput * E and adds u * n_b per bounce and u at the closing emitter.

Film in units of E: each half warp sums S = sum r and Q = sum (r - K)^2 about its first sample K over one batch, the batch's zero
samples join as r = 0, and the batch is folded into (count, sum, mean, M2) by one pairwise update scaled by E and E^2."""
import numpy as np
import pytest

N = 69


def forward(E, n, s, e):
    u = E.astype(np.float32).copy()
    dst = np.zeros_like(u)
    for nb, sb in zip(n, s):
        dst = (u * nb + dst).astype(np.float32)
        u = (u * sb).astype(np.float32)
    return dst + u * np.float32(e)


def backward(n, s, e):
    r = (n[-1] + s[-1] * np.float32(e)).astype(np.float32)
    for nb, sb in zip(n[-2::-1], s[-2::-1]):
        r = (nb + sb * r).astype(np.float32)
    return r


@pytest.mark.parametrize("seed", range(8))
def test_horner_matches_forward_replay(seed):
    rng = np.random.default_rng(seed)
    E = rng.uniform(0, 20, N).astype(np.float32)
    E[rng.integers(0, N, 5)] = 0          # wavelengths the light does not emit
    for _ in range(200):
        nb = int(rng.integers(1, 12))
        D, G = rng.uniform(0, 1, (2, nb, N)).astype(np.float32)
        wn = rng.uniform(0, 2, (nb, 2)) * (rng.uniform(size=(nb, 1)) < 0.7)   # the light is hidden at some bounces
        ws = rng.uniform(0, 3, (nb, 2))
        n = (wn[:, :1] * D + wn[:, 1:] * G).astype(np.float32)
        s = (ws[:, :1] * D + ws[:, 1:] * G).astype(np.float32)
        e = int(rng.integers(0, 2))
        ref = forward(E.astype(np.float64), n.astype(np.float64), s.astype(np.float64), e)
        got = E * backward(n, s, e)
        scale = max(np.abs(ref).max(), 1e-30)
        assert np.all(np.abs(got - ref) <= 1e-5 * np.maximum(np.abs(ref), 1e-6 * scale))
        assert np.allclose(forward(E, n, s, e), ref, rtol=1e-5, atol=1e-6 * scale)


class Film:
    """PixelFilm of one half warp (f32), with the kernel's per-sample Welford update (the general kernel, and this repository's
    compact-record kernels before per-batch statistics) and the per-batch fold."""

    def __init__(self):
        self.cnt, self.lit = np.float32(0), False
        self.sum, self.mean, self.m2 = (np.zeros(N, np.float32) for _ in range(3))

    def add(self, c):
        self.cnt += np.float32(1)
        self.lit = True
        inv = np.float32(1) / self.cnt
        self.sum = self.sum + c
        delta = c - self.mean
        self.mean = (self.mean + inv * delta).astype(np.float32)
        self.m2 = (self.m2 + delta * (c - self.mean)).astype(np.float32)

    def add_zeros(self, k):
        n0 = self.cnt
        self.cnt = np.float32(self.cnt + k)
        if not self.lit or k == 0:
            return
        w = np.float32(k) / self.cnt
        self.m2 = (self.m2 + self.mean * self.mean * (n0 * w)).astype(np.float32)
        self.mean = (self.mean - self.mean * w).astype(np.float32)

    def add_batch(self, nz, rs, E):
        if len(rs) == 0:
            return self.add_zeros(nz)
        K = rs[0]
        S = np.zeros(N, np.float32)
        Q = np.zeros(N, np.float32)
        for r in rs:
            S = S + r
            d = r - K
            Q = (Q + d * d).astype(np.float32)
        nb, n0 = np.float32(len(rs) + nz), self.cnt
        self.cnt = np.float32(self.cnt + nb)
        self.lit = True
        w = nb / self.cnt
        m = S * (np.float32(1) / nb)
        dk = m - K
        m2b = np.maximum(Q + np.float32(nz) * K * K - nb * dk * dk, 0).astype(np.float32)
        delta = E * m - self.mean
        self.sum = (self.sum + E * S).astype(np.float32)
        self.m2 = (self.m2 + E * E * m2b + delta * delta * (n0 * w)).astype(np.float32)
        self.mean = (self.mean + delta * w).astype(np.float32)

    def merge(self, o):
        n = self.cnt + o.cnt
        wb = o.cnt / n if n > 0 else np.float32(0)
        delta = o.mean - self.mean
        self.m2 = (self.m2 + o.m2 + delta * delta * self.cnt * wb).astype(np.float32)
        self.mean = (self.mean + delta * wb).astype(np.float32)
        self.sum = (self.sum + o.sum).astype(np.float32)
        self.cnt, self.lit = np.float32(n), self.lit or o.lit


def render(samples, E, batched):
    """One pixel's samples (r, or None for a path without bounce records) in batches of 32, two half warps, as the kernel walks
    them: the zeros of a batch first (half 0), then the replayed paths alternately to half 0 and half 1."""
    halves = [Film(), Film()]
    for b0 in range(0, len(samples), 32):
        batch = samples[b0:b0 + 32]
        nz = sum(r is None for r in batch)
        rep = [r for r in batch if r is not None]
        if batched:
            halves[0].add_batch(nz, rep[0::2], E)
            halves[1].add_batch(0, rep[1::2], E)
        else:
            halves[0].add_zeros(nz)
            for i, r in enumerate(rep):
                halves[i & 1].add((E * r).astype(np.float32))
    halves[0].merge(halves[1])
    return halves[0]


def _cases():
    rng = np.random.default_rng(3)
    E = rng.uniform(0.5, 30, N).astype(np.float32)
    E[::7] = 0                                                     # E with zero entries
    base = rng.uniform(0.2, 1, N).astype(np.float32)
    yield "large mean, tiny variance", E, [(1e3 * base * (1 + 1e-4 * rng.standard_normal(N))).astype(np.float32) for _ in range(1024)]
    yield "runs of zeros", E, [None if (i // 40) % 2 else rng.exponential(1, N).astype(np.float32) for i in range(1000)]
    yield "mostly zeros, one bright sample", E, [None] * 500 + [(50 * base).astype(np.float32)] + [None] * 523
    yield "replayed paths of zero radiance", E, [np.zeros(N, np.float32) if i % 3 else None for i in range(97)]
    yield "heavy tail, partial batch", E, [(rng.pareto(1.5, N) * base).astype(np.float32) for _ in range(97)]


@pytest.mark.parametrize("name,E,samples", list(_cases()), ids=lambda x: x if isinstance(x, str) else "")
def test_batched_shifted_sums_match_welford(name, E, samples):
    c = np.stack([np.zeros(N) if r is None else E.astype(np.float64) * r for r in samples])
    ref_sum, ref_mean = c.sum(0), c.mean(0)
    ref_m2 = ((c - ref_mean) ** 2).sum(0)
    new, old = render(samples, E, True), render(samples, E, False)
    assert new.cnt == old.cnt == len(samples)
    assert new.lit == old.lit == any(r is not None for r in samples)
    for f in (new, old):
        assert np.all(f.sum[E == 0] == 0) and np.all(f.mean[E == 0] == 0) and np.all(f.m2[E == 0] == 0)
    for got, ref, tol in ((new.sum, ref_sum, 1e-5), (new.mean, ref_mean, 1e-5), (new.m2, ref_m2, 1e-3)):
        floor = 1e-6 * max(np.abs(ref).max(), 1e-30)
        assert np.all(np.abs(got - ref) <= tol * np.maximum(np.abs(ref), floor)), name
    # the per-batch statistics are at least as close to the exact M2 as the per-sample update they replace
    floor = 1e-6 * max(ref_m2.max(), 1e-30)
    err_new = (np.abs(new.m2 - ref_m2) / np.maximum(ref_m2, floor)).max()
    err_old = (np.abs(old.m2 - ref_m2) / np.maximum(ref_m2, floor)).max()
    assert err_new <= max(2 * err_old, 1e-5), (err_new, err_old)


def test_unlit_pixel_stays_exactly_zero():
    f = Film()
    f.add_batch(32, [], np.ones(N, np.float32))
    f.add_batch(17, [], np.ones(N, np.float32))
    assert f.cnt == 49 and not f.lit and not f.mean.any() and not f.m2.any() and not f.sum.any()
