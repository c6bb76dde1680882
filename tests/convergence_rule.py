"""The convergence rule of progressive frames (rt_frame_set_convergence) restated in numpy: the checkpoint lattice, the
check, and per pixel the sample count n_p a frame stops it at, from per-pixel moments of any source of samples.

A pixel's samples are a pure function of (seed, pixel, sample index), so a frame under the rule holds, for every pixel p,
the sums and Q of sample indices [0, n_p): n_probe where the probe stopped it, the first checkpoint where its standard
error E was <= the tolerance, or samples_done where it is still being sampled."""
import numpy as np


def numpy_se(sums, sq):
    """E from {T_r, T_g, T_b, n} and Q: D = n Q - sum_c T_c^2 in int64, E = sqrt(D / (3 n^2 (n - 1))) in float64, +inf where
    n < 2 (the same operations, in the same order, as pixel_standard_error)."""
    sums = np.asarray(sums).astype(np.int64)
    n = sums[..., 3]
    t = sums[..., :3]
    d = n * np.asarray(sq).astype(np.int64) - (t[..., 0] * t[..., 0] + t[..., 1] * t[..., 1] + t[..., 2] * t[..., 2])
    nd = n.astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        e = np.sqrt(d.astype(np.float64) / (3.0 * nd * nd * (n - 1).astype(np.float64)))
    return np.where(n < 2, np.inf, e)


def checkpoints(min_samples, interval, upto):
    """The checkpoints c = min_samples + j interval with c <= upto."""
    return list(range(min_samples, upto + 1, interval)) if upto >= min_samples else []


def next_checkpoint(min_samples, interval, samples_done):
    """The first checkpoint above samples_done."""
    if samples_done < min_samples:
        return min_samples
    return min_samples + ((samples_done - min_samples) // interval + 1) * interval


def probe(moments, n, spp, adaptive):
    """renderPixel's probe (Scene.fs:172-188) over pixels 0 .. n-1: ([n, 4] int64 sums with the count, [n] int64 Q,
    n_probe, the flags of the pixels that go on).  `moments(idx, s0, s1)` gives ([len(idx), 3] sums, [len(idx)] Q) of
    sample indices [s0, s1) of the pixels idx."""
    every = np.arange(n)
    if not adaptive:
        return np.zeros((n, 4), np.int64), np.zeros(n, np.int64), 0, np.ones(n, bool)
    ft = min(5, spp // 2)
    n_probe = 2 * ft + 1
    a, qa = moments(every, 0, ft + 1)
    b, qb = moments(every, ft + 1, n_probe)
    s = a + b
    flagged = np.abs(s // n_probe - a // (ft + 1)).sum(1) != 0
    return np.concatenate([s, np.full((n, 1), n_probe, np.int64)], 1), qa + qb, n_probe, flagged


def converge(moments, sums, sq, flagged, samples_done, tolerance, min_samples, interval):
    """The frame after its probe (`sums`, `sq`, `flagged`, as probe() gives them) advanced under the rule to samples_done:
    (sums [n, 4], Q [n], the pixels still being sampled, the checks run).  A check at checkpoint c stops every pixel still
    being sampled whose E over [0, c) is <= tolerance; once no pixel is left, nothing more is traced or checked."""
    sums, sq, active = sums.copy(), sq.copy(), flagged.copy()
    checks = 0
    at = int(sums[flagged, 3].max()) if flagged.any() else 0
    at = min(at, samples_done)
    while active.any() and at < samples_done:
        end = min(next_checkpoint(min_samples, interval, at), samples_done)
        idx = np.flatnonzero(active)
        ds, dq = moments(idx, at, end)
        sums[idx, :3] += ds
        sums[idx, 3] = end
        sq[idx] += dq
        at = end
        if at >= min_samples and (at - min_samples) % interval == 0:
            active &= ~(numpy_se(sums, sq) <= tolerance)
            checks += 1
    return sums, sq, active, checks
