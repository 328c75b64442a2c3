"""fp64 numpy / scipy restatement of torchmetrics' SI-SDR and SDR.

* SI-SDR: `scale_invariant_signal_distortion_ratio(preds, target, zero_mean)`, which the reference's
  src/metrics/si_sdr.py wraps (ScaleInvariantSignalDistortionRatio, zero_mean=False by default):
  alpha = (<p,t> + eps) / (||t||^2 + eps), 10 log10((||alpha t||^2 + eps) / (||alpha t - p||^2 + eps)), eps = FLT_EPSILON.
* SDR: `signal_distortion_ratio(preds, target, filter_length, zero_mean, load_diag)` on its direct-solve path: fp64,
  optional mean removal, both signals divided by max(||x||, 1e-6), the autocorrelation of the target and its
  cross-correlation with the prediction for lags < filter_length by a zero-padded FFT, load_diag added to r[0], the
  symmetric Toeplitz system solved (here by `scipy.linalg.solve_toeplitz`), coh = b.x, 10 log10(coh / (1 - coh)).

torchmetrics is not a dependency of this project, so this file is written from torchmetrics' definitions and parity
with the library itself is unpinned, as for SI-SNR and STOI (DESIGN.md §0c, §8, §9).  A singular system (an all-zero
target without load_diag) raises here, as torchmetrics' dense solve does; the CUDA kernel returns NaN for it instead.
"""
import numpy as np
import scipy.linalg as sl

FLT_EPS = float(np.finfo(np.float32).eps)
NORM_FLOOR = 1e-6


def lag_sums_fft(t, p, L):
    """b[l] = sum_n t[n] p[n + l] for l < L, by torchmetrics' zero-padded rfft / irfft."""
    n = 1 << int(np.ceil(np.log2(len(t) + len(p) - 1)))
    tf = np.fft.rfft(t, n)
    return np.fft.irfft(np.conj(tf) * np.fft.rfft(p, n), n)[:L]


def lag_sums_direct(t, p, L):
    T = len(t)
    return np.array([t[:T - l] @ p[l:] for l in range(L)])


def si_sdr(p, t, zero_mean=False, eps=FLT_EPS):
    p = np.asarray(p, np.float64)
    t = np.asarray(t, np.float64)
    if zero_mean:
        p = p - p.mean()
        t = t - t.mean()
    alpha = (p @ t + eps) / (t @ t + eps)
    s = alpha * t
    e = s - p
    return 10 * np.log10((s @ s + eps) / (e @ e + eps))


def sdr(p, t, filter_length=512, zero_mean=False, load_diag=None, solve=None):
    """`solve(r, b)` defaults to scipy.linalg.solve_toeplitz (r the first column of the symmetric Toeplitz matrix)."""
    p = np.asarray(p, np.float64)
    t = np.asarray(t, np.float64)
    if zero_mean:
        p = p - p.mean()
        t = t - t.mean()
    t = t / max(np.linalg.norm(t), NORM_FLOOR)
    p = p / max(np.linalg.norm(p), NORM_FLOOR)
    r = lag_sums_fft(t, t, filter_length)
    b = lag_sums_fft(t, p, filter_length)
    if load_diag is not None:
        r[0] += load_diag
    x = (solve or sl.solve_toeplitz)(r, b)
    coh = b @ x
    return 10 * np.log10(coh / (1 - coh))


def pit_all(metric, s1p, s2p, s1, s2, mix=None, **kw):
    """rows (B,6) of [s1p.s1, s2p.s2, s1p.s2, s2p.s1, mix.s1, mix.s2] (NaN without mix) and summary (7):
    [mean (r0+r1)/2, mean (r2+r3)/2, max, max - mean (r4+r5)/2, mean r4, mean r5, B] (3..5 NaN without mix)."""
    B = s1p.shape[0]
    rows = np.full((B, 6), np.nan)
    for b in range(B):
        pairs = [(s1p, s1), (s2p, s2), (s1p, s2), (s2p, s1)]
        if mix is not None:
            pairs += [(mix, s1), (mix, s2)]
        for q, (p, t) in enumerate(pairs):
            rows[b, q] = metric(p[b], t[b], **kw)
    p1 = np.mean((rows[:, 0] + rows[:, 1]) / 2)
    p2 = np.mean((rows[:, 2] + rows[:, 3]) / 2)
    sep = max(p1, p2)
    m1, m2 = rows[:, 4].mean(), rows[:, 5].mean()
    return rows, np.array([p1, p2, sep, sep - (m1 + m2) / 2, m1, m2, B])
