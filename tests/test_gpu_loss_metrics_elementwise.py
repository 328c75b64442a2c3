"""The loss and metric kernels (csrc/sisnr.cu, csrc/sdr.cu) element by element against fp64 references.

k_sisnr_moments reduces 16 raw fp64 moments per chunk of 8192 samples; k_sisnr_finalize centres them algebraically
(<p_c, g_c> = Spg - Sp Sg / T) into the SI-SNR metric rows, the loss rows and the PIT summary; k_sisdr_finalize does
the same for SI-SDR; k_sisnr_loss_backward is the only gradient the project computes; k_sdr_corr / k_sdr_solve are the
lag sums and the Levinson recursion of BSS-eval SDR.  A whole-tensor tolerance hides an error confined to one chunk, the
last CTA's tail, one lag chunk or one Levinson order; here every output element gets its own bound from an error model
written above its family, and every output written through ctypes is a view into a larger allocation whose guard cells
must keep their sentinel bit pattern.

References are fp64 numpy (oracle/vatss_oracle.py, oracle/sdr_oracle.py) computed from the exact fp32 samples the
kernels read, plus an fp64 torch autograd restatement of the reference loss for the gradient.  u = 2^-53 is the unit
roundoff of fp64.  Each family prints `WORST-RATIO <family>: <max |err| / bound>`."""
import ctypes
import math

import numpy as np
import pytest
import torch
from scipy.signal import lfilter

from oracle import sdr_oracle as D
from oracle import vatss_oracle as O

gpu = pytest.mark.gpu
needs_cuda = pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")

U = 2.0 ** -53            # unit roundoff of fp64
U32 = 2.0 ** -24          # unit roundoff of fp32
U_REF = float(np.finfo(np.longdouble).eps) / 2   # the moment reference sums in long double
EPS = float(np.finfo(np.float32).eps)
LN10 = math.log(10.0)
CHUNK = 8192              # SISNR_CHUNK
GUARD = 64                # sentinel cells before and after every output view
SENT64 = 0x7FF8DEAD5A5A5A5A   # NaN bit patterns: a cell the kernel should have written and did not fails every bound
SENT32 = 0x7FC05A5A
PAIRS = [(0, 2), (1, 3), (0, 3), (1, 2), (4, 2), (4, 3)]   # rows: (prediction, target) of [s1p, s2p, s1, s2, mix]


def DEV():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def lib():
    from speech_separation_b200 import _lib

    return _lib.load()


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _check(lib, rc, what):
    assert rc == 0, f"{what} failed (rc={rc}): {lib.vatss_last_error().decode('utf-8', 'replace')}"


def guarded(n, dtype=torch.float64):
    """(allocation, view): n cells between GUARD sentinel cells on each side; every cell starts as the sentinel."""
    buf = torch.empty(n + 2 * GUARD, dtype=dtype, device=DEV())
    if dtype == torch.float64:
        buf.view(torch.int64).fill_(SENT64)
    else:
        buf.view(torch.int32).fill_(SENT32)
    return buf, buf[GUARD:GUARD + n]


def assert_guard(buf, n, label):
    ib = buf.view(torch.int64 if buf.dtype == torch.float64 else torch.int32)
    sent = SENT64 if buf.dtype == torch.float64 else SENT32
    for name, part in (("before", ib[:GUARD]), ("after", ib[GUARD + n:])):
        bad = int((part != sent).sum())
        assert bad == 0, f"{label}: {bad} guard cells {name} the output overwritten"


def check_elements(got, want, bound, label, same_ok=True):
    """|got - want| <= bound element by element; equal values (infinities of one sign, or NaN in both when
    same_ok) pass.  Returns the worst |err| / bound over the finite comparisons."""
    got = np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    bound = np.broadcast_to(np.asarray(bound, np.float64), got.shape)
    with np.errstate(invalid="ignore"):
        err = np.abs(got - want)
        ok = err <= bound
        if same_ok:
            ok |= (got == want) | (np.isnan(got) & np.isnan(want))
    if not ok.all():
        idx = tuple(int(i) for i in np.argwhere(~ok)[0])
        raise AssertionError(f"{label}: {int((~ok).sum())} of {ok.size} elements out of bound; first at {idx}: got "
                             f"{got[idx]:.17g} want {want[idx]:.17g} err {err[idx]:.3e} bound {bound[idx]:.3e}")
    fin = np.isfinite(err) & (bound > 0)
    return float((err[fin] / bound[fin]).max()) if fin.any() else 0.0


def report(family, ratio, label=""):
    print(f"WORST-RATIO {family}: {ratio:.3e} {label}")


# ----------------------------------------------------------------------------------------------------------------------
# inputs
# ----------------------------------------------------------------------------------------------------------------------
def sisnr_batch(B, T, seed, snr=(-30.0, 100.0), offsets=(0.0, 1.0, 100.0), amps=(1e-4, 1e3)):
    """(5, B, T) float32 [s1p, s2p, s1, s2, mix]: per utterance a SI-SNR from a sweep over `snr` dB, a DC offset of
    offsets[b % 3] standard deviations on every signal and an amplitude from a log sweep over `amps`."""
    rng = np.random.default_rng(seed)
    out = np.zeros((5, B, T), np.float64)
    snrs = np.linspace(snr[0], snr[1], B) if B > 1 else np.array([0.5 * (snr[0] + snr[1])])
    amp = np.geomspace(amps[0], amps[1], B) if B > 1 else np.array([1.0])
    rng.shuffle(amp)
    for b in range(B):
        a, off = amp[b], offsets[b % len(offsets)]
        for k, t in ((0, 2), (1, 3)):
            x = rng.standard_normal(T)
            n = rng.standard_normal(T)
            n *= np.sqrt((x @ x) / max(n @ n, 1e-300) / 10 ** (snrs[(b + k) % B] / 10))
            out[t, b] = a * (x + off)
            out[k, b] = a * (0.7 * x + 0.7 * n + 1.3 * off)
    out[4] = out[2] + out[3]
    return out.astype(np.float32)


def _dev(*arrs):
    return [None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(DEV()) for a in arrs]


# ======================================================================================================================
# 1. Moments (k_sisnr_moments)
# ======================================================================================================================
# A CTA reduces one chunk of 8192 samples of one utterance.  The products of two fp32 samples are exact in fp64, so only
# the additions round: <= 32 serial adds per thread, a 5-level shuffle tree and 8 warp partials added in order, a depth
# of 45:   |m^ - m| <= 45 u sum|terms|   (+ the long-double reference's own rounding, 14 U_REF sum|terms|).
MOM_T = [1, 17, 255, 256, 257, 8191, 8192, 8193, 16385, 64000, 160000, 960000]


def _mom_batches(T):
    if T <= 8193:
        return [1, 3, 257, 300]
    if T <= 16385:
        return [1, 3, 257]
    return [1, 3] if T <= 160000 else [1]


def moment_terms(x5, has_mix, i):
    """(B, T) float64 terms of moment i, in the kernel's order (exact: products of two fp32 samples)."""
    a, c, x, y = (v.astype(np.float64) for v in x5[:4])
    z = x5[4].astype(np.float64) if has_mix else np.zeros_like(a)
    return [a, c, x, y, z, a * a, c * c, x * x, y * y, z * z, a * x, c * y, a * y, c * x, z * x, z * y][i]


def run_pit_sisnr(lib, x5, has_mix, B, T):
    """vatss_pit_sisnr into guarded outputs; returns numpy (rows, rows_loss, summary, scratch (B, chunks, 16))."""
    chunks = lib.vatss_sisnr_chunks(T)
    s1p, s2p, s1, s2, mix = _dev(*x5[:4], x5[4] if has_mix else None)
    outs = [guarded(n) for n in (B * 6, B * 4, 8, B * chunks * 16)]
    _check(lib, lib.vatss_pit_sisnr(_p(s1p), _p(s2p), _p(s1), _p(s2), _p(mix), B, T, *[_p(v) for _, v in outs], None),
           "vatss_pit_sisnr")
    torch.cuda.synchronize()
    for (buf, v), name in zip(outs, ("rows", "rows_loss", "summary", "scratch")):
        assert_guard(buf, v.numel(), f"pit_sisnr B={B} T={T} {name}")
    rows, rows_loss, summary, scratch = (v.cpu().numpy() for _, v in outs)
    return rows.reshape(B, 6), rows_loss.reshape(B, 4), summary, scratch.reshape(B, chunks, 16)


@gpu
@needs_cuda
@pytest.mark.parametrize("has_mix", [True, False], ids=["mix", "nomix"])
@pytest.mark.parametrize("T", MOM_T)
def test_moments_match_exact_chunk_sums(lib, T, has_mix):
    worst = 0.0
    for B in _mom_batches(T):
        x5 = sisnr_batch(B, T, seed=T * 7 + B)
        _, _, _, got = run_pit_sisnr(lib, x5, has_mix, B, T)
        chunks = got.shape[1]
        want, mag = np.zeros_like(got), np.zeros_like(got)
        for i in range(16):
            terms = np.pad(moment_terms(x5, has_mix, i), ((0, 0), (0, chunks * CHUNK - T))).reshape(B, chunks, CHUNK)
            want[:, :, i] = terms.astype(np.longdouble).sum(-1).astype(np.float64)
            mag[:, :, i] = np.abs(terms).sum(-1)
        bound = (45 * U + 14 * U_REF) * mag
        worst = max(worst, check_elements(got, want, bound, f"moments B={B} T={T} mix={has_mix}", same_ok=False))
        if not has_mix:
            assert (got[:, :, [4, 9, 14, 15]] == 0.0).all(), "the mixture moments must be exactly 0 without mix"
    report("moments", worst, f"(T={T} mix={has_mix})")


# ======================================================================================================================
# 2. SI-SNR metric and loss rows, PIT summary (k_sisnr_finalize); SI-SDR rows (k_sisdr_finalize)
# ======================================================================================================================
# Moment i of an utterance sums its chunk values in chunk order: |S^ - S| <= (45 + chunks) u M, M = sum|terms|.
# Centring dot = Spg - Sp Sg / T (and pp, gg alike) adds E_pg + |Sg|/T E_p + |Sp|/T E_g + 4 u (M_pg + |Sp Sg| / T).
# The value is f(dot, pp, gg): the torchmetrics form 10 log10((a^2 gg + eps) / (n + eps)), a = (dot + eps)/(gg + eps),
# n = a^2 gg - 2 a dot + pp clamped at 0, or the loss -20 log10(s / n), s = dot^2 / gg, n = pp - s.  The evaluation of
# n cancels (8 u (a^2 gg + 2|a dot| + pp), resp. 4 u (pp + s), added to E_pp).  The bound is twice the linear
# propagation sum_i max_+- |f(x +- E_i e_i) - f(x)| over the three centred inputs, evaluated in fp64 from the
# reference's own dot, pp, gg, plus 16 u |f|.  The magnification is kappa = raw square sum / centred residual: tight
# at low SNR, widening honestly with the SNR and the DC offset (where it reaches the dB scale the bound says so).
def _f_metric(dot, pp, gg):
    with np.errstate(divide="ignore", invalid="ignore"):
        alpha = (dot + EPS) / (gg + EPS)
        sig = alpha * alpha * gg
        noise = np.maximum(sig - 2.0 * alpha * dot + pp, 0.0)
        return 10.0 * np.log10((sig + EPS) / (noise + EPS))


def _f_loss(dot, pp, gg):
    with np.errstate(divide="ignore", invalid="ignore"):
        s = dot * dot / gg
        n = np.maximum(pp - s, 0.0)
        return -20.0 * np.log10(s / n)


def _propagate(f, x, e):
    """2 sum_i max_+- |f(x +- e_i) - f(x)| + 16 u |f(x)| over the three inputs x = (dot, pp, gg)."""
    f0 = f(*x)
    tot = np.zeros_like(f0)
    with np.errstate(invalid="ignore"):
        for i in range(3):
            worst = np.zeros_like(f0)
            for sgn in (1.0, -1.0):
                xi = list(x)
                xi[i] = x[i] + sgn * e[i]
                d = np.abs(f(*xi) - f0)
                worst = np.maximum(worst, np.where(np.isnan(d) & ~np.isnan(f0), np.inf, d))
            tot = tot + worst
    return 2.0 * tot + 16 * U * np.abs(f0)


def pair_model(P, G, T, chunks, centre=True):
    """Reference (dot, pp, gg) of each row (two-pass fp64 when centring, raw otherwise) and their kernel error bounds."""
    p, g = P.astype(np.float64), G.astype(np.float64)
    dep = (45 + chunks) * U
    Sp, Sg = p.sum(-1), g.sum(-1)
    Mp, Mg, Mpp, Mgg, Mpg = np.abs(p).sum(-1), np.abs(g).sum(-1), (p * p).sum(-1), (g * g).sum(-1), np.abs(p * g).sum(-1)
    if centre:
        pc, gc = p - p.mean(-1, keepdims=True), g - g.mean(-1, keepdims=True)
        dot, pp, gg = (pc * gc).sum(-1), (pc * pc).sum(-1), (gc * gc).sum(-1)
        ref = (math.log2(max(T, 2)) + 4) * U   # the pairwise two-pass reference's own rounding
        Edot = dep * (Mpg + np.abs(Sg) / T * Mp + np.abs(Sp) / T * Mg) + 4 * U * (Mpg + np.abs(Sp * Sg) / T) \
            + ref * np.abs(pc * gc).sum(-1)
        Epp = dep * (Mpp + 2 * np.abs(Sp) / T * Mp) + 4 * U * (Mpp + Sp * Sp / T) + ref * pp
        Egg = dep * (Mgg + 2 * np.abs(Sg) / T * Mg) + 4 * U * (Mgg + Sg * Sg / T) + ref * gg
    else:
        dot, pp, gg = (p * g).sum(-1), Mpp, Mgg
        ref = (math.log2(max(T, 2)) + 2) * U
        Edot, Epp, Egg = (dep + ref) * Mpg, (dep + ref) * Mpp, (dep + ref) * Mgg
    return (dot, pp, gg), (Edot, Epp, Egg)


def metric_bound(x, e):
    dot, pp, gg = x
    with np.errstate(divide="ignore", invalid="ignore"):
        alpha = np.where(gg + EPS > 0, (dot + EPS) / (gg + EPS), 0.0)
    e = (e[0], e[1] + 8 * U * (alpha * alpha * gg + 2 * np.abs(alpha * dot) + pp), e[2])
    return _propagate(_f_metric, x, e)


def loss_bound(x, e):
    dot, pp, gg = x
    with np.errstate(divide="ignore", invalid="ignore"):
        s = np.where(gg > 0, dot * dot / gg, 0.0)
    e = (e[0], e[1] + 4 * U * (pp + s), e[2])
    return _propagate(_f_loss, x, e)


def sisnr_references(x5, has_mix, T, chunks):
    """want / bound of the metric rows (B, 6) and the loss rows (B, 4)."""
    d = [a.astype(np.float64) for a in x5]
    B = x5.shape[1]
    m_want, m_bnd = np.zeros((B, 6)), np.zeros((B, 6))
    l_want, l_bnd = np.zeros((B, 4)), np.zeros((B, 4))
    for q, (ip, ig) in enumerate(PAIRS):
        if q >= 4 and not has_mix:
            continue
        x, e = pair_model(x5[ip], x5[ig], T, chunks)
        with np.errstate(divide="ignore", invalid="ignore"):
            m_want[:, q] = O.si_snr_metric_rows(d[ip], d[ig])
        m_bnd[:, q] = metric_bound(x, e)
        if q < 4:
            with np.errstate(divide="ignore", invalid="ignore"):
                l_want[:, q] = O.sisnr_loss_rows(d[ip], d[ig])
            l_bnd[:, q] = loss_bound(x, e)
    return m_want, m_bnd, l_want, l_bnd


def sisnr_summary_replay(rows, rows_loss, has_mix):
    """k_sisnr_finalize's summary recomputed from its own rows in its order, in IEEE fp64."""
    B = rows.shape[0]
    mm, ml = [0.0] * 6, [0.0] * 4
    for b in range(B):
        for q in range(6):
            mm[q] += float(rows[b, q])
        for q in range(4):
            ml[q] += float(rows_loss[b, q])
    mm = [v / B for v in mm]
    ml = [v / B for v in ml]
    l1, l2 = (ml[0] + ml[1]) * 0.5, (ml[2] + ml[3]) * 0.5
    s1, s2 = (mm[0] + mm[1]) * 0.5, (mm[2] + mm[3]) * 0.5
    sep = s1 if s1 > s2 else s2
    return np.array([l2 if l2 < l1 else l1, l1, l2, sep, sep - (mm[4] + mm[5]) * 0.5 if has_mix else 0.0,
                     mm[4], mm[5], float(B)])


def assert_bitwise(got, want, label):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    same = (got == want) | (np.isnan(got) & np.isnan(want))
    assert same.all(), f"{label}: entries {np.nonzero(~same)[0].tolist()} differ: got {got} want {want}"


def summary_oracle_bound(m_want, m_bnd, l_want, l_bnd, has_mix):
    """The summary of the oracle rows and its bound (means of the row bounds)."""
    l1, l2 = (l_want[:, 0] + l_want[:, 1]).mean() / 2, (l_want[:, 2] + l_want[:, 3]).mean() / 2
    s1, s2 = (m_want[:, 0] + m_want[:, 1]).mean() / 2, (m_want[:, 2] + m_want[:, 3]).mean() / 2
    bl1, bl2 = (l_bnd[:, 0] + l_bnd[:, 1]).mean() / 2, (l_bnd[:, 2] + l_bnd[:, 3]).mean() / 2
    bs1, bs2 = (m_bnd[:, 0] + m_bnd[:, 1]).mean() / 2, (m_bnd[:, 2] + m_bnd[:, 3]).mean() / 2
    m4, m5, b4, b5 = m_want[:, 4].mean(), m_want[:, 5].mean(), m_bnd[:, 4].mean(), m_bnd[:, 5].mean()
    sep = max(s1, s2)
    want = np.array([min(l1, l2), l1, l2, sep, sep - (m4 + m5) / 2 if has_mix else 0.0, m4, m5, m_want.shape[0]])
    bound = np.array([max(bl1, bl2), bl1, bl2, max(bs1, bs2), max(bs1, bs2) + (b4 + b5) / 2, b4, b5, 0.0])
    return want, bound + 1e-12 * np.abs(want)


SISNR_CASES = [  # (B, T, seed, label)
    (24, 16385, 1, "snr-sweep"),
    (9, 17, 2, "short"),
    (6, 8193, 3, "chunk+1"),
    (4, 64000, 4, "4s"),
    (300, 257, 5, "B300"),
]


@gpu
@needs_cuda
@pytest.mark.parametrize("has_mix", [True, False], ids=["mix", "nomix"])
@pytest.mark.parametrize("B,T,seed,label", SISNR_CASES, ids=[c[3] for c in SISNR_CASES])
def test_sisnr_rows_and_summary(lib, B, T, seed, label, has_mix):
    x5 = sisnr_batch(B, T, seed)
    if B > 2:   # swapped rows: a third of the batch has its predictions exchanged
        x5[[0, 1], ::3] = x5[[1, 0], ::3]
    rows, rows_loss, summary, _ = run_pit_sisnr(lib, x5, has_mix, B, T)
    chunks = lib.vatss_sisnr_chunks(T)
    m_want, m_bnd, l_want, l_bnd = sisnr_references(x5, has_mix, T, chunks)
    if not has_mix:
        assert (rows[:, 4:] == 0.0).all()
    r1 = check_elements(rows[:, :6 if has_mix else 4], m_want[:, :6 if has_mix else 4],
                        m_bnd[:, :6 if has_mix else 4], f"si-snr rows {label}")
    r2 = check_elements(rows_loss, l_want, l_bnd, f"loss rows {label}")
    assert_bitwise(summary, sisnr_summary_replay(rows, rows_loss, has_mix), f"summary replay {label}")
    sw, sb = summary_oracle_bound(m_want, m_bnd, l_want, l_bnd, has_mix)
    sel = [0, 1, 2, 3, 7] + ([4, 5, 6] if has_mix else [])
    r3 = check_elements(summary[sel], sw[sel], sb[sel], f"summary vs oracle {label}")
    report("si-snr rows", r1, label)
    report("loss rows", r2, label)
    report("summary", r3, label)


@gpu
@needs_cuda
def test_sisnr_silent_target_constant_prediction_and_tie(lib):
    B, T = 6, 4000
    x5 = sisnr_batch(B, T, seed=11, snr=(0.0, 30.0), offsets=(0.0, 1.0), amps=(0.1, 10.0))
    x5[2, 0] = 0.0                       # silent s1 in utterance 0: loss rows 0 and 3 NaN, metric rows finite
    x5[0, 1] = np.float32(0.37)          # constant s1p in utterance 1: the metric by its eps form, the loss 0/0
    x5[4] = x5[2] + x5[3]
    rows, rows_loss, summary, _ = run_pit_sisnr(lib, x5, True, B, T)
    m_want, m_bnd, l_want, l_bnd = sisnr_references(x5, True, T, 1)
    assert np.isnan(rows_loss[0, [0, 3]]).all() and np.isfinite(rows[0]).all()
    assert np.isfinite(rows[1]).all()
    r1 = check_elements(rows, m_want, m_bnd, "si-snr rows, silent target and constant prediction")
    keep = np.ones((B, 4), bool)
    keep[1, [0, 2]] = False              # the loss of a constant prediction is 0/0: not defined
    r2 = check_elements(rows_loss[keep], l_want[keep], l_bnd[keep], "loss rows, silent target")
    assert_bitwise(summary, sisnr_summary_replay(rows, rows_loss, True), "summary replay, silent target")
    # exact PIT tie with distinct permutations: utterance 1 is utterance 0 with its predictions exchanged, so the four
    # per-pair sums are equal bit for bit and l1 == l2; the kernel keeps permutation 1 (`l2 < l1` is false)
    t5 = sisnr_batch(1, 3000, seed=12, snr=(5.0, 15.0))
    x5 = np.concatenate([t5, t5], axis=1)
    x5[[0, 1], 1] = x5[[1, 0], 1]
    rows, rows_loss, summary, _ = run_pit_sisnr(lib, x5, True, 2, 3000)
    assert summary[1] == summary[2] and summary[0] == summary[1], f"no exact tie: {summary[:3]}"
    assert_bitwise(summary, sisnr_summary_replay(rows, rows_loss, True), "summary replay, tie")
    report("si-snr rows", r1, "(silent / constant)")
    report("loss rows", r2, "(silent target)")


@gpu
@needs_cuda
@pytest.mark.parametrize("zero_mean", [False, True], ids=["raw", "zero-mean"])
@pytest.mark.parametrize("B,T,seed,label", SISNR_CASES, ids=[c[3] for c in SISNR_CASES])
def test_sisdr_rows_match_oracle(lib, B, T, seed, label, zero_mean):
    x5 = sisnr_batch(B, T, seed + 100)
    if B > 2:
        x5[[0, 1], ::3] = x5[[1, 0], ::3]
    x5[2, 0] = 0.0 if B > 1 else x5[2, 0]   # a silent target: torchmetrics' eps form keeps the rows finite
    x5[4] = x5[2] + x5[3]
    chunks = lib.vatss_sisnr_chunks(T)
    s1p, s2p, s1, s2, mix = _dev(*x5)
    outs = [guarded(n) for n in (B * 6, 7, B * chunks * 16)]
    _check(lib, lib.vatss_pit_sisdr(_p(s1p), _p(s2p), _p(s1), _p(s2), _p(mix), B, T, int(zero_mean),
                                    *[_p(v) for _, v in outs], None), "vatss_pit_sisdr")
    torch.cuda.synchronize()
    for (buf, v), name in zip(outs, ("rows", "summary", "scratch")):
        assert_guard(buf, v.numel(), f"pit_sisdr {label} {name}")
    rows = outs[0][1].cpu().numpy().reshape(B, 6)
    summary = outs[1][1].cpu().numpy()
    d = x5.astype(np.float64)
    want, bnd = np.zeros((B, 6)), np.zeros((B, 6))
    for q, (ip, ig) in enumerate(PAIRS):
        want[:, q] = [D.si_sdr(d[ip, b], d[ig, b], zero_mean=zero_mean) for b in range(B)]
        bnd[:, q] = metric_bound(*pair_model(x5[ip], x5[ig], T, chunks, centre=zero_mean))
    ratio = check_elements(rows, want, bnd, f"si-sdr rows {label} zero_mean={zero_mean}")
    # the summary is pit_summary7 of the kernel's own rows, in its order
    p1 = p2 = m1 = m2 = 0.0
    for b in range(B):
        p1 += (rows[b, 0] + rows[b, 1]) * 0.5
        p2 += (rows[b, 2] + rows[b, 3]) * 0.5
        m1 += rows[b, 4]
        m2 += rows[b, 5]
    p1, p2, m1, m2 = p1 / B, p2 / B, m1 / B, m2 / B
    sep = p1 if p1 > p2 else p2
    assert_bitwise(summary, [p1, p2, sep, sep - (m1 + m2) * 0.5, m1, m2, B], f"si-sdr summary {label}")
    report("si-sdr rows", ratio, f"{label} zero_mean={zero_mean}")


# ======================================================================================================================
# 3. Loss gradient (k_sisnr_loss_backward)
# ======================================================================================================================
# g = up (gc / dot - e / n), up = grad_out (-40 / ln 10) / (2B), gc = g - mg, e = p - mp - a gc, a = dot / gg, with the
# means, dot, gg and n = pp - dot^2/gg from the moments (errors as in §2) and the per-sample terms in fp64:
#   E_a  = |a| (E_dot/|dot| + E_gg/gg) + 2u|a|,   E_n = E_pp + 2|a| E_dot + a^2 E_gg + 4u (pp + s)
#   E_gc = E_S_g / T + u |gc|,   E_e = E_S_p / T + |a| E_gc + |gc| E_a + 3u (|p| + |mp| + |a gc|)
#   E    = E_gc/|dot| + |gc| E_dot/dot^2 + E_e/n + |e| E_n/n^2 + 2u (|gc/dot| + |e/n|)
# Bound: 2 |up| E (the factor 2 covers the fp64 reference's own rounding) + 2^-24 |g| (the final fp32 rounding).
def grad_bound(P, G, T, chunks, up_abs):
    p, g = P.astype(np.float64), G.astype(np.float64)
    (dot, pp, gg), (Edot, Epp, Egg) = pair_model(P, G, T, chunks)
    dot, pp, gg, Edot, Epp, Egg = (v[:, None] for v in (dot, pp, gg, Edot, Epp, Egg))
    dep = (45 + chunks) * U
    mp, mg = p.mean(-1, keepdims=True), g.mean(-1, keepdims=True)
    Emp = dep * np.abs(p).sum(-1, keepdims=True) / T + U * np.abs(mp)
    Emg = dep * np.abs(g).sum(-1, keepdims=True) / T + U * np.abs(mg)
    a = dot / gg
    s = dot * dot / gg
    n = pp - s
    gc = g - mg
    e = p - mp - a * gc
    Ea = np.abs(a) * (Edot / np.abs(dot) + Egg / gg) + 2 * U * np.abs(a)
    En = Epp + 2 * np.abs(a) * Edot + a * a * Egg + 4 * U * (pp + s)
    Egc = Emg + U * np.abs(gc)
    Ee = Emp + np.abs(a) * Egc + np.abs(gc) * Ea + 3 * U * (np.abs(p) + np.abs(mp) + np.abs(a * gc))
    E = (Egc / np.abs(dot) + np.abs(gc) * Edot / dot ** 2 + Ee / n + np.abs(e) * En / n ** 2
         + 2 * U * (np.abs(gc / dot) + np.abs(e / n)))
    return 2 * up_abs * E


def torch_ref_loss(s1p, s2p, s1, s2):
    """fp64 restatement of BaseSSLoss.forward / SiSNRLoss.forward (ss_losses.py:10-26,100-114) for torch autograd."""
    def l(p, g):
        p = p - p.mean(-1, keepdim=True)
        g = g - g.mean(-1, keepdim=True)
        s = (g * p).sum(-1, keepdim=True) / (g * g).sum(-1, keepdim=True) * g
        e = p - s
        return (-20 * torch.log10((s * s).sum(-1) / (e * e).sum(-1))).mean()

    p1 = (l(s1p, s1) + l(s2p, s2)) / 2
    p2 = (l(s1p, s2) + l(s2p, s1)) / 2
    return p2 if p2 < p1 else p1


def torch_ref_grad(x4):
    s1p, s2p = (torch.from_numpy(x4[k].astype(np.float64)).requires_grad_(True) for k in (0, 1))
    s1, s2 = (torch.from_numpy(x4[k].astype(np.float64)) for k in (2, 3))
    torch_ref_loss(s1p, s2p, s1, s2).backward()
    return s1p.grad.numpy(), s2p.grad.numpy()


def run_backward(lib, x4, B, T, upstream):
    """forward then vatss_pit_sisnr_backward into guarded gradients; returns (g1, g2, summary) numpy."""
    chunks = lib.vatss_sisnr_chunks(T)
    s1p, s2p, s1, s2 = _dev(*x4)
    rows, rows_loss, summary, scratch = (torch.empty(n, dtype=torch.float64, device=DEV())
                                         for n in (B * 6, B * 4, 8, B * chunks * 16))
    _check(lib, lib.vatss_pit_sisnr(_p(s1p), _p(s2p), _p(s1), _p(s2), None, B, T, _p(rows), _p(rows_loss),
                                    _p(summary), _p(scratch), None), "vatss_pit_sisnr")
    out = []
    for up in upstream:
        go = torch.tensor([up], dtype=torch.float32, device=DEV())
        (b1, g1), (b2, g2) = guarded(B * T, torch.float32), guarded(B * T, torch.float32)
        _check(lib, lib.vatss_pit_sisnr_backward(_p(s1p), _p(s2p), _p(s1), _p(s2), B, T, _p(scratch), _p(summary),
                                                 _p(go), _p(g1), _p(g2), None), "vatss_pit_sisnr_backward")
        torch.cuda.synchronize()
        assert_guard(b1, B * T, f"backward B={B} T={T} g1")
        assert_guard(b2, B * T, f"backward B={B} T={T} g2")
        out.append((g1.cpu().numpy().reshape(B, T), g2.cpu().numpy().reshape(B, T)))
    return out, summary.cpu().numpy(), rows_loss.cpu().numpy().reshape(B, 4)


def check_grads(got, x4, up, T, chunks, label, oracle=None, autograd=None):
    """Each prediction's gradient against the oracle closed form and fp64 autograd; returns the worst ratio."""
    B = x4.shape[1]
    d = x4.astype(np.float64)
    oracle = oracle or O.pit_sisnr_loss_grad(*d)
    autograd = autograd or torch_ref_grad(x4)
    loss = lambda a, b: O.sisnr_loss_rows(a, b).mean()
    swap = (loss(d[0], d[3]) + loss(d[1], d[2])) / 2 < (loss(d[0], d[2]) + loss(d[1], d[3])) / 2
    tgt = (3, 2) if swap else (2, 3)
    up = float(np.float32(up))   # the kernel reads grad_out as fp32
    up_abs = abs(up) * 40.0 / LN10 / (2 * B)
    worst = 0.0
    for k in range(2):
        bnd = grad_bound(x4[k], x4[tgt[k]], T, chunks, up_abs)
        for name, ref in (("oracle", oracle[k]), ("autograd", autograd[k])):
            want = up * ref
            worst = max(worst, check_elements(got[k], want, bnd + U32 * np.abs(want),
                                              f"{label} g{k + 1} vs {name} (upstream {up})", same_ok=False))
    return worst


def check_near_exact_rule(outs, summary, rows_loss):
    """A prediction whose loss row in the chosen permutation is -inf gets a zero gradient; all gradients are finite."""
    swap = summary[2] < summary[1]
    for g1g2 in outs:
        for k, g in enumerate(g1g2):
            row = rows_loss[:, 2 + k if swap else k]
            assert np.isfinite(g).all(), "non-finite gradient"
            assert (g[np.isneginf(row)] == 0.0).all(), "a -inf loss row must get a zero gradient"


BWD_T = [2, 17, 2047, 2048, 2049, 8193, 64000, 160000]
UPSTREAM = [1.0, -0.37, 0.0, 1e4]


@gpu
@needs_cuda
@pytest.mark.parametrize("T", BWD_T)
def test_loss_gradient_matches_fp64(lib, T):
    worst = 0.0
    for B in ([1, 2, 33, 300] if T <= 8193 else [1, 2]):
        x5 = sisnr_batch(B, T, seed=T + B, snr=(-10.0, 40.0), offsets=(0.0, 1.0, 10.0), amps=(1e-2, 1e2))
        if (T + B) % 2:          # every other batch swapped whole: the PIT picks permutation 2
            x5[[0, 1]] = x5[[1, 0]]
        x4 = x5[:4]
        outs, summary, rows_loss = run_backward(lib, x4, B, T, UPSTREAM)
        if T == 2:
            # two centred samples are collinear: every estimate is exact, the residual power is rounding only
            check_near_exact_rule(outs, summary, rows_loss)
            continue
        oracle, autograd = O.pit_sisnr_loss_grad(*x4.astype(np.float64)), torch_ref_grad(x4)
        for up, got in zip(UPSTREAM, outs):
            worst = max(worst, check_grads(got, x4, up, T, lib.vatss_sisnr_chunks(T), f"grad B={B} T={T}",
                                           oracle, autograd))
    report("loss gradient", worst, f"(T={T})")


@gpu
@needs_cuda
def test_loss_gradient_at_an_exact_tie_follows_permutation_1(lib):
    t5 = sisnr_batch(1, 5000, seed=21, snr=(5.0, 15.0))
    x4 = np.concatenate([t5, t5], axis=1)[:4].copy()
    x4[[0, 1], 1] = x4[[1, 0], 1]
    (got,), summary, _ = run_backward(lib, x4, 2, 5000, [1.0])
    assert summary[1] == summary[2], "the batch is not an exact tie"
    d = x4.astype(np.float64)
    # the reference's `if loss_perm_2 < loss_perm_1` is false at a tie: permutation 1, s1p with s1
    oracle = tuple(O.pit_sisnr_loss_grad(d[0], d[1], d[2], d[3]))
    ratio = check_grads(got, x4, 1.0, 5000, 1, "tie", oracle, torch_ref_grad(x4))
    perm2 = O.pit_sisnr_loss_grad(d[0], d[1], d[3], d[2])
    assert np.abs(got[0] - perm2[0]).max() > 1e3 * np.abs(got[0]).max() * U32, "permutations indistinguishable"
    report("loss gradient", ratio, "(exact tie)")


def _v():
    import speech_separation_b200 as V

    return V


@gpu
@needs_cuda
def test_loss_gradient_through_autograd_entry_points(lib):
    V = _v()
    B, T = 3, 6001
    x5 = sisnr_batch(B, T, seed=31, snr=(0.0, 20.0), offsets=(0.0, 1.0), amps=(0.1, 10.0))
    x4 = x5[:4]
    d = x4.astype(np.float64)
    oracle = O.pit_sisnr_loss_grad(*d)
    up_abs = 40.0 / LN10 / (2 * B)
    bnd = [grad_bound(x4[k], x4[2 + k], T, 1, up_abs) + U32 * np.abs(oracle[k]) for k in range(2)]
    worst = 0.0
    # a (B, 1, T) input
    p1, p2, s1, s2 = _dev(*(x.reshape(B, 1, T) for x in x4))
    p1.requires_grad_(True)
    p2.requires_grad_(True)
    V.SiSNRWavLoss()(s1_pred=p1, s2_pred=p2, s1=s1, s2=s2)["loss"].backward()
    for k, p in enumerate((p1, p2)):
        assert p.grad.shape == (B, 1, T)
        worst = max(worst, check_elements(p.grad.reshape(B, T).cpu().numpy(), oracle[k], bnd[k], f"(B,1,T) g{k + 1}"))
    # only one prediction requires grad
    p1, p2, s1, s2 = _dev(*x4)
    p2.requires_grad_(True)
    V.SiSNRWavLoss()(s1_pred=p1, s2_pred=p2, s1=s1, s2=s2)["loss"].backward()
    assert p1.grad is None
    worst = max(worst, check_elements(p2.grad.cpu().numpy(), oracle[1], bnd[1], "one prediction requires grad"))
    # the same tensor as both predictions: autograd adds the two halves
    same = np.stack([x4[0], x4[0], x4[2], x4[3]])
    p, _, s1, s2 = _dev(*same)
    p.requires_grad_(True)
    V.SiSNRWavLoss()(s1_pred=p, s2_pred=p, s1=s1, s2=s2)["loss"].backward()
    o = O.pit_sisnr_loss_grad(*same.astype(np.float64))
    dd = same.astype(np.float64)
    lo = lambda a, b: O.sisnr_loss_rows(a, b).mean()
    swap = (lo(dd[0], dd[3]) + lo(dd[1], dd[2])) / 2 < (lo(dd[0], dd[2]) + lo(dd[1], dd[3])) / 2
    tg = (3, 2) if swap else (2, 3)
    b_same = sum(grad_bound(same[k], same[tg[k]], T, 1, up_abs) for k in range(2)) + U32 * np.abs(o[0] + o[1]) + \
        U32 * (np.abs(o[0]) + np.abs(o[1]))
    worst = max(worst, check_elements(p.grad.cpu().numpy(), o[0] + o[1], b_same, "same tensor as both predictions"))
    # a graph in front: p_k = w x_k + c; SI-SNR is offset-invariant, so dL/dc ~ 0
    xs = _dev(x4[0], x4[1])
    w = torch.tensor(0.7, device=DEV(), requires_grad=True)
    c = torch.tensor(0.3, device=DEV(), requires_grad=True)
    s1, s2 = _dev(x4[2], x4[3])
    V.SiSNRWavLoss()(s1_pred=w * xs[0] + c, s2_pred=w * xs[1] + c, s1=s1, s2=s2)["loss"].backward()
    pw = [np.float32(0.7) * x4[k] + np.float32(0.3) for k in range(2)]   # fp32, as the graph computes them
    og = O.pit_sisnr_loss_grad(pw[0].astype(np.float64), pw[1].astype(np.float64), d[2], d[3])
    xk = [x4[k].astype(np.float64) for k in range(2)]
    want_w = sum(float((og[k] * xk[k]).sum()) for k in range(2))
    n = 2 * B * T
    gb = [grad_bound(pw[k], x4[2 + k], T, 1, up_abs) + U32 * np.abs(og[k]) for k in range(2)]
    bw = sum(float((gb[k] * np.abs(xk[k])).sum()) for k in range(2)) + \
        2 * n * U32 * sum(float(np.abs(og[k] * xk[k]).sum()) for k in range(2))
    bc = sum(float(gb[k].sum()) for k in range(2)) + 2 * n * U32 * sum(float(np.abs(og[k]).sum()) for k in range(2))
    worst = max(worst, check_elements(float(w.grad), want_w, bw, "w.grad of p = w x + c"))
    assert abs(float(c.grad)) <= bc, f"c.grad {float(c.grad):.3e} above {bc:.3e}: the loss must be offset-invariant"
    report("loss gradient", worst, "(autograd entry points)")


@gpu
@needs_cuda
def test_single_pair_loss_is_differentiable(lib):
    V = _v()
    B, T = 4, 9000
    x5 = sisnr_batch(B, T, seed=41, snr=(-5.0, 30.0), offsets=(0.0, 1.0), amps=(0.1, 10.0))
    pred, gt = _dev(x5[0], x5[2])
    with torch.no_grad():
        plain = float(V.SiSNRLoss()(pred, gt))
    pred.requires_grad_(True)
    loss = V.SiSNRLoss()(pred, gt)
    np.testing.assert_allclose(float(loss.detach()), plain, rtol=4 * U32)
    loss.backward()
    pg = torch.from_numpy(x5[0].astype(np.float64)).requires_grad_(True)
    g64 = torch.from_numpy(x5[2].astype(np.float64))
    pc, gc = pg - pg.mean(-1, keepdim=True), g64 - g64.mean(-1, keepdim=True)
    s = (gc * pc).sum(-1, keepdim=True) / (gc * gc).sum(-1, keepdim=True) * gc
    (-20 * torch.log10((s * s).sum(-1) / ((pc - s) ** 2).sum(-1))).mean().backward()
    want = pg.grad.numpy()
    bnd = 2 * grad_bound(x5[0], x5[2], T, 1, 40.0 / LN10 / (2 * B)) + 2 * U32 * np.abs(want)
    report("loss gradient", check_elements(pred.grad.cpu().numpy(), want, bnd, "SiSNRLoss gradient"), "(SiSNRLoss)")


@gpu
@needs_cuda
def test_near_exact_estimates_follow_one_rule(lib):
    """p = a g + b in fp32: where the shared residual power is <= 0 the forward row is -inf and the backward writes a
    zero gradient for that prediction; elsewhere both are finite and the loss is far below any real estimate's."""
    B, T = 48, 4096
    rng = np.random.default_rng(51)
    g = (rng.standard_normal((B, T)) * np.geomspace(1e-3, 1e2, B)[:, None]).astype(np.float32)
    a = np.where(np.arange(B) % 4 == 0, 1.0, rng.uniform(-3, 3, B)).astype(np.float32)
    b = np.where(np.arange(B) % 4 == 0, 0.0, rng.choice([0.0, 1.0, 100.0], B) * g.std(-1)).astype(np.float32)
    p = (a[:, None] * g + b[:, None]).astype(np.float32)
    g2 = rng.standard_normal((B, T)).astype(np.float32)
    p2 = (g2 + 0.1 * rng.standard_normal((B, T))).astype(np.float32)
    x4 = np.stack([p, p2, g, g2])
    (got,), summary, rows_loss = run_backward(lib, x4, B, T, [1.0])
    assert summary[1] <= summary[2], "the near-exact pairs must be in permutation 1"
    ninf = np.isneginf(rows_loss[:, 0])
    assert (ninf | np.isfinite(rows_loss[:, 0])).all(), rows_loss[:, 0]
    with np.errstate(divide="ignore", invalid="ignore"):
        want = O.sisnr_loss_rows(p.astype(np.float64), g.astype(np.float64))
    check_elements(rows_loss[:, 0], want, loss_bound(*pair_model(p, g, T, 1)), "near-exact loss rows")
    check_near_exact_rule([got], summary, rows_loss)
    print(f"near-exact: {int(ninf.sum())} of {B} rows -inf (zero gradient), {int((~ninf).sum())} finite")
    # the same rule through autograd: SiSNRLoss of exact copies, per utterance
    V = _v()
    pred, gt = _dev(g[::4], g[::4])
    _, rows_loss, _ = V.pit_sisnr_all(pred, pred, gt, gt)
    pred.requires_grad_(True)
    V.SiSNRLoss()(pred, gt).backward()
    ninf = torch.isneginf(rows_loss[:, 0])
    assert torch.isfinite(pred.grad).all() and bool((pred.grad[ninf] == 0).all())


# ----------------------------------------------------------------------------------------------------------------------
# argument checks (no device work)
# ----------------------------------------------------------------------------------------------------------------------
def test_batch_limit_and_empty_batch_raise_before_device_work():
    from speech_separation_b200 import loss as L

    big = torch.zeros(65536, 1)
    with pytest.raises(ValueError, match="at most 65535"):
        L.pit_sisnr_all(big, big, big, big)
    with pytest.raises(ValueError, match="at most 65535"):
        L.SiSNRWavLoss()(s1_pred=big.clone().requires_grad_(True), s2_pred=big, s1=big, s2=big)
    with pytest.raises(ValueError, match="at most 65535"):
        L.SiSNRLoss()(big.clone().requires_grad_(True), big)
    three = torch.zeros(256, 256, 1)   # leading dims multiply past 65535
    with pytest.raises(ValueError, match="at most 65535"):
        L.pit_sisnr_all(three, three, three, three)
    empty = torch.zeros(2, 0)
    with pytest.raises(ValueError, match="empty batch"):
        L.SiSNRWavLoss()(s1_pred=empty.clone().requires_grad_(True), s2_pred=empty, s1=empty, s2=empty)
    with pytest.raises(ValueError, match="empty batch"):
        L.pit_sisnr_all(empty, empty, empty, empty)


def test_library_rejects_batches_above_grid_limit():
    from speech_separation_b200 import _lib

    lib = _lib.load()
    fake = ctypes.c_void_p(256)   # never dereferenced: the argument check returns first
    rc = lib.vatss_pit_sisnr(fake, fake, fake, fake, None, 65536, 1, fake, fake, fake, fake, None)
    assert rc != 0 and "at most 65535" in lib.vatss_last_error().decode()
    rc = lib.vatss_pit_sisnr_backward(fake, fake, fake, fake, 65536, 1, fake, fake, None, fake, fake, None)
    assert rc != 0 and "at most 65535" in lib.vatss_last_error().decode()


# ======================================================================================================================
# 4. SDR (k_sdr_corr, k_sdr_solve)
# ======================================================================================================================
# Geometry (DESIGN §9 "Memory", sdr_geometry in sdr.cu): tiles of 1024 samples, ranges of ceil(tiles / 128) tiles,
# 512-lag chunks; the workspace holds the moments, then (256-byte aligned) part[b, g, range, k, Lpad].
# Lag sums: a thread accumulates one lag over the range's samples by serial fp64 FMAs, so the depth is the range length
# R_k = tiles_per_range * 1024; the products of fp32 samples are exact (with zero_mean the staged samples fl(x - mean)
# are reproduced bit for bit from the kernel's own moments and the product rounds once).  The reference is an fp64
# torch matmul over the same R samples:   |part^ - part| <= (R_k + R + 1) u sum_n |t[n] p[n + l]|.
def sdr_geometry(B, T, L):
    ceil = lambda a, b: -(-a // b)
    chunks, lag_chunks = ceil(T, CHUNK), ceil(L, 512)
    tiles = ceil(T, 1024)
    tpp = ceil(tiles, 128)
    parts = ceil(tiles, tpp)
    align = lambda x: (x + 255) // 256 * 256
    off_part = align(B * chunks * 16 * 8)
    Lpad = lag_chunks * 512
    return dict(chunks=chunks, Lpad=Lpad, tpp=tpp, parts=parts, off_part=off_part,
                bytes=off_part + align(B * 2 * parts * 4 * Lpad * 8))


def test_sdr_workspace_geometry_matches_the_documented_layout():
    from speech_separation_b200 import _lib

    lib = _lib.load()
    for B, T, L in [(1, 2, 2), (3, 131072, 512), (2, 131073, 513), (1, 262145, 2048), (32, 64000, 512), (5, 9, 7)]:
        assert lib.vatss_sdr_workspace_bytes(B, T, L) == sdr_geometry(B, T, L)["bytes"], (B, T, L)


def run_sdr(lib, x5, has_mix, L, zero_mean, load_diag=None):
    """vatss_sdr with a caller-owned guarded workspace; returns (rows (B,6), summary, workspace bytes, geometry)."""
    B, T = x5.shape[1], x5.shape[2]
    geo = sdr_geometry(B, T, L)
    nbytes = lib.vatss_sdr_workspace_bytes(B, T, L)
    assert nbytes == geo["bytes"]
    nd = nbytes // 8
    (wb, ws), (rb, rows), (sb, summ) = guarded(nd), guarded(B * 6), guarded(7)
    s1p, s2p, s1, s2, mix = _dev(*x5[:4], x5[4] if has_mix else None)
    _check(lib, lib.vatss_sdr(_p(s1p), _p(s2p), _p(s1), _p(s2), _p(mix), B, T, L, int(zero_mean),
                              -1.0 if load_diag is None else float(load_diag), _p(rows), _p(summ), _p(ws),
                              ctypes.c_size_t(nbytes), None), "vatss_sdr")
    torch.cuda.synchronize()
    for buf, n, name in ((wb, nd, "workspace"), (rb, B * 6, "rows"), (sb, 7, "summary")):
        assert_guard(buf, n, f"sdr B={B} T={T} L={L} {name}")
    return rows.cpu().numpy().reshape(B, 6), summ.cpu().numpy(), ws, geo


def _kernel_mean(mom, b, i, T):
    v = 0.0
    for c in range(mom.shape[1]):
        v += float(mom[b, c, i])
    return v / T


SDR_LAG_CASES = ([(L, L, True, False) for L in (2, 7, 8, 9, 511, 512, 513, 1000, 1024, 1025, 1536, 2047, 2048)]
                 + [(L, L + 1, False, True) for L in (2, 9, 512, 513, 1025, 2048)]
                 + [(L, L + 1, True, True) for L in (8, 1000, 1536)]
                 + [(512, 131072, True, False), (1024, 131072, False, True), (2, 131073, False, False),
                    (513, 131073, True, True), (2048, 131073, False, True), (1025, 262145, True, False),
                    (7, 262145, False, True)])


@gpu
@needs_cuda
@pytest.mark.parametrize("L,T,has_mix,zero_mean", SDR_LAG_CASES,
                         ids=[f"L{c[0]}-T{c[1]}-{'mix' if c[2] else 'nomix'}-{'zm' if c[3] else 'raw'}"
                              for c in SDR_LAG_CASES])
def test_sdr_lag_sums_match_direct_sums(lib, L, T, has_mix, zero_mean):
    B = 2 if T < 100000 else 1
    x5 = speech_like(B, T, seed=L * 3 + T)
    x5 += np.float32(0.05) * (np.arange(5)[:, None, None] + 1).astype(np.float32)   # a DC offset on every signal
    x5[4] = x5[2] + x5[3]
    _, _, ws, geo = run_sdr(lib, x5, has_mix, L, zero_mean)
    parts, Lpad, tpp = geo["parts"], geo["Lpad"], geo["tpp"]
    mom = ws[:B * geo["chunks"] * 16].cpu().numpy().reshape(B, geo["chunks"], 16)
    part_all = ws.view(torch.uint8)[geo["off_part"]:geo["off_part"] + B * 2 * parts * 4 * Lpad * 8]
    part_all = part_all.view(torch.float64).reshape(B, 2, parts, 4, Lpad)
    nk = 4 if has_mix else 3
    if not has_mix:   # the mixture's partials are never written
        assert (part_all[:, :, :, 3].contiguous().view(torch.int64) == SENT64).all()
    got_all = part_all[:, :, :, :nk].cpu().numpy()
    worst = 0.0
    for b in range(B):
        for g in range(2):
            src = [2 + g, 0, 1, 4][:nk]          # partner k: the target, s1p, s2p, mix
            mi = [2 + g, 0, 1, 4]
            xs = []
            for k, s in enumerate(src):
                v = torch.from_numpy(x5[s, b].astype(np.float64))
                if zero_mean:
                    v = v - _kernel_mean(mom, b, mi[k], T)
                xs.append(v)
            t = xs[0].to(DEV())
            P = torch.nn.functional.pad(torch.stack(xs), (0, Lpad + tpp * 1024)).to(DEV())
            want = torch.empty(parts, nk, Lpad, dtype=torch.float64, device=DEV())
            mag = torch.empty_like(want)
            Rmax = []
            for r in range(parts):
                n0, n1 = r * tpp * 1024, min((r + 1) * tpp * 1024, T)
                H = P[:, n0:n1 + Lpad - 1].unfold(1, Lpad, 1)            # (nk, R, Lpad): H[k, i, l] = p_k[n0 + i + l]
                tr = t[n0:n1]
                want[r] = torch.einsum("i,kil->kl", tr, H)
                mag[r] = torch.einsum("i,kil->kl", tr.abs(), H.abs())
                Rmax.append(n1 - n0)
            R = torch.tensor(Rmax, dtype=torch.float64, device=DEV())[:, None, None]
            bound = (tpp * 1024 + R + 1) * U * mag
            worst = max(worst, check_elements(got_all[b, g], want.cpu().numpy(), bound.cpu().numpy(),
                                              f"sdr lag sums L={L} T={T} b={b} target {g}", same_ok=False))
    report("sdr lag sums", worst, f"(L={L} T={T} ranges={parts} lag chunks={Lpad // 512})")


# Rows: the solve is compared in coherence coh = b.x, recovered from the row as r / (1 + r), r = 10^(dB / 10).  With
# the normalised Toeplitz matrix R (r[0] = 1 + load_diag) the lag sums perturb R and b by at most d u per entry (d the
# lag-sum depth plus the range count and the normalisation), so |d coh| <= 3 L kappa(R) d u to first order, and the
# Levinson recursion and scipy's solve_toeplitz each add O(L kappa u):   bound = 8 (L + d) kappa(R) u + 8 u.
def speech_like(B, T, seed, snrs=(-5, 20)):
    """(5, B, T) float32 [s1p, s2p, s1, s2, mix]: resonant AR(2) targets under a -30..0 dB envelope, predictions =
    target + white noise at snrs dB, mix = s1 + s2 (the coloured targets of tests/test_sdr.py)."""
    rng = np.random.default_rng(seed)
    out = np.zeros((5, B, T), np.float64)
    for b in range(B):
        for k, t in ((0, 2), (1, 3)):
            env = np.repeat(10 ** (rng.uniform(-30, 0, -(-T // 1600)) / 20), 1600)[:T]
            x = lfilter([1.0], [1.0, -1.3, 0.6], rng.standard_normal(T)) * env
            n = rng.standard_normal(T)
            n *= np.sqrt((x @ x) / (n @ n) / 10 ** (rng.uniform(*snrs) / 10))
            out[t, b], out[k, b] = x, x + n
    out[4] = out[2] + out[3]
    return out.astype(np.float32)


def _coherence(db):
    """coh from 10 log10(coh / (1 - coh)); +inf dB (a prediction equal to its target) is coh = 1."""
    with np.errstate(over="ignore"):
        return 1.0 / (1.0 + 10.0 ** (-np.asarray(db, np.float64) / 10.0))


def _toeplitz_kappa(t, L, zero_mean, load_diag):
    import scipy.linalg as sl

    t = t - t.mean() if zero_mean else t
    t = t / max(np.linalg.norm(t), D.NORM_FLOOR)
    r = D.lag_sums_direct(t, t, L) if L <= 64 else D.lag_sums_fft(t, t, L)
    if load_diag is not None:
        r[0] += load_diag
    return float(np.linalg.cond(sl.toeplitz(r)))


SDR_ROW_CASES = [(L, ld, kind) for L in (513, 1024, 2048) for ld in (None, 1e-3) for kind in ("speech", "ar2")]


@gpu
@needs_cuda
@pytest.mark.parametrize("L,load_diag,kind", SDR_ROW_CASES,
                         ids=[f"L{c[0]}-{'ld' if c[1] else 'nold'}-{c[2]}" for c in SDR_ROW_CASES])
def test_sdr_rows_match_solve_toeplitz(lib, L, load_diag, kind):
    B, T = 2, 20000
    x5 = speech_like(B, T, seed=L + (7 if load_diag else 0))
    if kind == "ar2":   # a strongly coloured target: AR(2) with poles at radius 0.99, so kappa(R) is large
        rng = np.random.default_rng(L)
        th = 0.3
        t = lfilter([1.0], [1.0, -2 * 0.99 * np.cos(th), 0.99 ** 2], rng.standard_normal((B, T)), axis=-1)
        x5[2] = t.astype(np.float32)
        x5[0] = (t + 0.05 * t.std() * rng.standard_normal((B, T))).astype(np.float32)
        x5[4] = x5[2] + x5[3]
    zero_mean = kind == "ar2"
    rows, summary, _, geo = run_sdr(lib, x5, True, L, zero_mean, load_diag)
    d = x5.astype(np.float64)
    depth = geo["tpp"] * 1024 + geo["parts"] + 64
    worst, kmax = 0.0, 0.0
    kap = {(b, g): _toeplitz_kappa(d[2 + g, b], L, zero_mean, load_diag) for b in range(B) for g in range(2)}
    for b in range(B):
        for q, (ip, ig) in enumerate(PAIRS):
            want = D.sdr(d[ip, b], d[ig, b], filter_length=L, zero_mean=zero_mean, load_diag=load_diag)
            rw, rg = _coherence(want), _coherence(rows[b, q])
            kappa = kap[(b, ig - 2)]
            kmax = max(kmax, kappa)
            bound = 8 * (L + depth) * kappa * U + 8 * U
            worst = max(worst, check_elements(rg, rw, bound,
                                              f"sdr coherence L={L} load_diag={load_diag} {kind} b={b} row {q}"))
    report("sdr rows", worst, f"(L={L} load_diag={load_diag} {kind}, max kappa {kmax:.2e})")


@gpu
@needs_cuda
def test_sdr_all_zero_target_at_2048_taps_gives_nan_only_for_its_rows(lib):
    B, T, L = 3, 8000, 2048
    x5 = speech_like(B, T, seed=61)
    x5[3, 1] = 0.0
    x5[4] = x5[2] + x5[3]
    x5[4, 1] += np.float32(0.5) * x5[1, 1]   # the mixture is not s1 itself (coh = 1, an infinite SDR)
    rows, _, _, _ = run_sdr(lib, x5, True, L, False)
    nan = np.isnan(rows)
    want = np.zeros_like(nan)
    want[1, [1, 2, 5]] = True            # the rows scored against s2 of utterance 1
    assert (nan == want).all(), nan
    d = x5.astype(np.float64)
    kap = {}
    for b, q in zip(*np.nonzero(~want)):
        ip, ig = PAIRS[q]
        w = D.sdr(d[ip, b], d[ig, b], filter_length=L)
        rw, rg = _coherence(w), _coherence(rows[b, q])
        kappa = kap.setdefault((b, ig), _toeplitz_kappa(d[ig, b], L, False, None))
        check_elements(rg, rw, 8 * (L + 1024 + 64) * kappa * U + 8 * U, f"sdr row {b},{q}")
