"""fp64 numpy restatement of STOI and extended STOI (pystoi 0.4 `stoi(x, y, fs, extended)`).

x is the clean target, y the prediction: torchmetrics' ShortTimeObjectiveIntelligibility (which the reference's
src/metrics/stoi.py wraps) calls `stoi(target, preds, fs, extended)`.  pystoi is not a dependency of this project, so
this file is written from pystoi's algorithm; parity with pystoi itself is unpinned (DESIGN.md §0c, §8).

Differences from pystoi, on purpose:
* extended STOI: pystoi adds EPS-scale Gaussian noise before each row / column normalisation.  It is left out so the
  value is deterministic; each normalisation divides by (norm + EPS) instead, so a constant row (an all-zero
  prediction) normalises to zeros, where pystoi's noise would give a random unit vector of expected correlation 0;
* a signal shorter than one 256-sample frame after resampling raises ValueError (pystoi fails on an empty max).

Pipeline: resample to 10 kHz (`resample_oct`), drop frames of the clean signal more than 40 dB below its loudest
frame (`remove_silent_frames`, the same frames of both signals), 512-point STFT of 256-sample Hann frames at hop 128,
15 one-third octave bands from 150 Hz, correlations over 30-frame (384 ms) segments.
"""
import numpy as np
from scipy.signal import resample_poly

FS = 10000
N_FRAME = 256
HOP = 128
NFFT = 512
NUMBAND = 15
MINFREQ = 150
N = 30                     # frames per segment
BETA = -15.0               # lower SDR bound, dB
DYN_RANGE = 40.0           # dB
EPS = np.finfo(float).eps
SHORT_VALUE = 1e-5         # value when fewer than N STFT frames remain


def resample_filter(p, q):
    """pystoi `resample_oct`'s Kaiser-windowed sinc for a p/q resampler (p, q coprime): (h, L, beta), sum(h) = 1."""
    stopband = 1.0 / (2 * max(p, q))
    roll_off = stopband / 10
    rejection_db = 60.0
    L = int(np.ceil((rejection_db - 8) / (28.714 * roll_off)))
    t = np.arange(-L, L + 1)
    beta = 0.1102 * (rejection_db - 8.7)
    h = np.kaiser(2 * L + 1, beta) * 2 * p * stopband * np.sinc(2 * stopband * t)
    return h / np.sum(h), L, beta


def resample_ratio(fs):
    g = np.gcd(FS, fs)
    return FS // g, fs // g


def resample(x, fs):
    """x at fs -> 10 kHz, as pystoi does: scipy.signal.resample_poly with the `resample_filter` window."""
    x = np.asarray(x, np.float64)
    if fs == FS:
        return x
    p, q = resample_ratio(fs)
    h, _, _ = resample_filter(p, q)
    return resample_poly(x, p, q, window=h)


def resample_closed_form(x, fs):
    """The same as `resample`, written out: y[n] = p sum_m h[nq - mp + L] x[m] for n < ceil(T p / q)."""
    x = np.asarray(x, np.float64)
    p, q = resample_ratio(fs)
    h, L, _ = resample_filter(p, q)
    T = len(x)
    n_out = -(-T * p // q)
    y = np.zeros(n_out)
    for n in range(n_out):
        m_lo = max(0, -(-(n * q - L) // p))
        m_hi = min(T - 1, (n * q + L) // p)
        m = np.arange(m_lo, m_hi + 1)
        y[n] = p * np.dot(h[n * q - m * p + L], x[m])
    return y


def resampled_length(T, fs):
    p, q = resample_ratio(fs)
    return -(-T * p // q)


def hann():
    return np.hanning(N_FRAME + 2)[1:-1]


def thirdoct(fs=FS, nfft=NFFT, num_bands=NUMBAND, min_freq=MINFREQ):
    """One-third octave band matrix (num_bands, nfft/2 + 1) and its [lo, hi) bin edges (pystoi `thirdoct`)."""
    f = np.linspace(0, fs, nfft + 1)[:nfft // 2 + 1]
    k = np.arange(num_bands, dtype=float)
    lo = min_freq * 2.0 ** ((2 * k - 1) / 6)
    hi = min_freq * 2.0 ** ((2 * k + 1) / 6)
    obm = np.zeros((num_bands, len(f)))
    edges = []
    for i in range(num_bands):
        a = int(np.argmin((f - lo[i]) ** 2))
        b = int(np.argmin((f - hi[i]) ** 2))
        obm[i, a:b] = 1
        edges.append((a, b))
    return obm, edges


OBM, BAND_EDGES = thirdoct()


def frame_energies(x):
    """dB energy of every Hann-windowed 256-sample frame at hop 128 (frames start at 0 .. len - 256)."""
    w = hann()
    frames = np.array([w * x[i:i + N_FRAME] for i in range(0, len(x) - N_FRAME + 1, HOP)])
    return 20 * np.log10(np.linalg.norm(frames, axis=1) + EPS)


def _overlap_add(frames):
    out = np.zeros((len(frames) - 1) * HOP + N_FRAME)
    for i, f in enumerate(frames):
        out[i * HOP:i * HOP + N_FRAME] += f
    return out


def remove_silent_frames(x, y):
    """Keep the frames whose clean energy is above max - 40 dB (strict); overlap-add the kept windowed frames of x
    and y.  Returns (x_sil, y_sil, mask)."""
    w = hann()
    starts = range(0, len(x) - N_FRAME + 1, HOP)
    xf = np.array([w * x[i:i + N_FRAME] for i in starts])
    yf = np.array([w * y[i:i + N_FRAME] for i in starts])
    e = 20 * np.log10(np.linalg.norm(xf, axis=1) + EPS)
    mask = e > np.max(e) - DYN_RANGE
    return _overlap_add(xf[mask]), _overlap_add(yf[mask]), mask


def stft(x):
    """(frames, 257) rfft of Hann-windowed frames starting at range(0, len - 256, 128): no frame starts at len - 256."""
    w = hann()
    return np.array([np.fft.rfft(w * x[i:i + N_FRAME], n=NFFT) for i in range(0, len(x) - N_FRAME, HOP)]).reshape(
        -1, NFFT // 2 + 1)


def envelopes(x):
    """(15, frames) one-third octave band amplitudes sqrt(OBM |X|^2)."""
    X = stft(x).T
    return np.sqrt(OBM @ np.abs(X) ** 2)


def _segments(env):
    return np.array([env[:, m - N:m] for m in range(N, env.shape[1] + 1)])


def _normalise(a, axis):
    a = a - a.mean(axis=axis, keepdims=True)
    return a / (np.linalg.norm(a, axis=axis, keepdims=True) + EPS)


def stoi_from_envelopes(x_env, y_env, extended=False):
    if x_env.shape[1] < N:
        return SHORT_VALUE
    xs, ys = _segments(x_env), _segments(y_env)     # (J, 15, 30)
    J = xs.shape[0]
    if extended:
        xn = _normalise(_normalise(xs, 2), 1)
        yn = _normalise(_normalise(ys, 2), 1)
        return float(np.sum(xn * yn / N) / J)
    c = np.linalg.norm(xs, axis=2, keepdims=True) / (np.linalg.norm(ys, axis=2, keepdims=True) + EPS)
    yp = np.minimum(ys * c, xs * (1 + 10 ** (-BETA / 20)))
    yp = _normalise(yp, 2)
    xc = _normalise(xs, 2)
    return float(np.sum(yp * xc) / (J * NUMBAND))


def stoi(x, y, fs=16000, extended=False, return_kept=False):
    """STOI (or ESTOI) of prediction y against clean target x, both 1-D at fs.  With return_kept, also the number of
    frames kept by the silent-frame removal."""
    x = np.asarray(x, np.float64)
    y = np.asarray(y, np.float64)
    if x.shape != y.shape or x.ndim != 1:
        raise ValueError(f"x and y must be 1-D of one length, got {x.shape} and {y.shape}")
    x, y = resample(x, fs), resample(y, fs)
    if len(x) < N_FRAME:
        raise ValueError(f"signal of {len(x)} samples at 10 kHz is shorter than one {N_FRAME}-sample frame")
    xs, ys, mask = remove_silent_frames(x, y)
    d = stoi_from_envelopes(envelopes(xs), envelopes(ys), extended)
    return (d, int(mask.sum())) if return_kept else d


def stoi_all(s1_pred, s2_pred, s1, s2, fs=16000, extended=False):
    """Batch (B, T) arrays -> (rows (B,4) [s1p.s1, s2p.s2, s1p.s2, s2p.s1], kept (B,2) per target, summary (3,)):
    summary = [mean (row0 + row1)/2, mean (row2 + row3)/2, max of the two] (batch-level PIT)."""
    B = np.asarray(s1).shape[0]
    rows = np.zeros((B, 4))
    kept = np.zeros((B, 2), np.int64)
    for b in range(B):
        y1, y2, g1, g2 = (resample(np.asarray(a[b], np.float64), fs) for a in (s1_pred, s2_pred, s1, s2))
        if len(g1) < N_FRAME:
            raise ValueError(f"signal of {len(g1)} samples at 10 kHz is shorter than one {N_FRAME}-sample frame")
        env = {}
        for t, g in enumerate((g1, g2)):
            gs, p1s, mask = remove_silent_frames(g, y1)
            _, p2s, _ = remove_silent_frames(g, y2)
            env[t] = (envelopes(gs), envelopes(p1s), envelopes(p2s))
            kept[b, t] = int(mask.sum())
        for q, (t, k) in enumerate(((0, 1), (1, 2), (1, 1), (0, 2))):
            rows[b, q] = stoi_from_envelopes(env[t][0], env[t][k], extended)
    p1 = float(np.mean((rows[:, 0] + rows[:, 1]) / 2))
    p2 = float(np.mean((rows[:, 2] + rows[:, 3]) / 2))
    return rows, kept, np.array([p1, p2, max(p1, p2)])
