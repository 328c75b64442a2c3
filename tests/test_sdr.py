"""SI-SDR (`vatss_pit_sisdr`) and SDR with its distortion filter (`vatss_sdr`), with `sisdr_all`, `sdr_all`,
`SISDRMetric`, `SDRMetric` and `SDRiMetric`, against the fp64 restatement in oracle/sdr_oracle.py (DESIGN.md §9).
Parity with torchmetrics itself is not pinned: torchmetrics is not a dependency."""
import ctypes

import numpy as np
import pytest
import scipy.linalg as sl
import torch
from scipy.signal import lfilter

from oracle import sdr_oracle as D
from oracle import vatss_oracle as O

TOL_SISDR = 1e-6   # dB
TOL_SDR = 1e-4     # dB


# ---------------------------------------------------------------------------------------------
# speech-like test signals
# ---------------------------------------------------------------------------------------------
def _clean(rng, T):
    """A resonant AR(2) process (a formant near 1.6 kHz at 16 kHz) under a 0.1 s piecewise envelope of -30 .. 0 dB."""
    seg = 1600
    env = np.repeat(10 ** (rng.uniform(-30, 0, -(-T // seg)) / 20), seg)[:T]
    return lfilter([1.0], [1.0, -1.3, 0.6], rng.standard_normal(T)) * env


def speech_batch(B, T, seed, snrs=(-5, 20)):
    """(s1_pred, s2_pred, s1, s2, mix) float32 (B, T): coloured targets, predictions = target + white noise at SNRs
    between snrs[0] and snrs[1] dB, mix = s1 + s2."""
    rng = np.random.default_rng(seed)
    out = np.zeros((5, B, T), np.float32)
    for b in range(B):
        for k, t in ((0, 2), (1, 3)):
            x = _clean(rng, T)
            n = rng.standard_normal(T)
            n *= np.sqrt((x @ x) / (n @ n) / 10 ** (rng.uniform(*snrs) / 10))
            out[t, b] = x
            out[k, b] = x + n
    out[4] = out[2] + out[3]
    return out


def _f64(a):
    return np.asarray(a, np.float32).astype(np.float64)


# ---------------------------------------------------------------------------------------------
# CPU: the oracle on its own
# ---------------------------------------------------------------------------------------------
def test_fft_lag_sums_equal_direct_lag_sums():
    _, _, s1, _, mix = speech_batch(1, 6000, seed=1).astype(np.float64)
    for L in (1, 64, 512):
        for t, p in ((s1[0], s1[0]), (s1[0], mix[0])):
            a, b = D.lag_sums_fft(t, p, L), D.lag_sums_direct(t, p, L)
            assert np.max(np.abs(a - b)) <= 1e-12 * np.abs(b).max()


def test_solve_toeplitz_equals_dense_solve():
    s1p, _, s1, _, _ = speech_batch(2, 16000, seed=2).astype(np.float64)
    for b in range(2):
        t, p = s1[b] / np.linalg.norm(s1[b]), s1p[b] / np.linalg.norm(s1p[b])
        for L in (64, 512):
            r, rhs = D.lag_sums_direct(t, t, L), D.lag_sums_direct(t, p, L)
            x1, x2 = sl.solve_toeplitz(r, rhs), np.linalg.solve(sl.toeplitz(r), rhs)
            assert np.max(np.abs(x1 - x2)) <= 1e-10 * np.abs(x2).max()
            assert abs(D.sdr(s1p[b], s1[b], L) - D.sdr(s1p[b], s1[b], L, solve=lambda r, y: np.linalg.solve(
                sl.toeplitz(r), y))) < 1e-10


def test_sisdr_equals_sisnr_on_zero_mean_signals():
    s1p, s2p, s1, s2, _ = speech_batch(4, 8000, seed=3).astype(np.float64)
    for p, t in ((s1p, s1), (s2p, s2), (s1p, s2)):
        p = p - p.mean(-1, keepdims=True)
        t = t - t.mean(-1, keepdims=True)
        ref = O.si_snr_metric_rows(p, t)
        got = np.array([D.si_sdr(p[b], t[b]) for b in range(4)])
        assert np.max(np.abs(got - ref)) < 1e-9
        assert np.max(np.abs(got - [D.si_sdr(p[b] + 0.3, t[b] - 0.1, zero_mean=True) for b in range(4)])) < 1e-9


def test_sdr_invariant_to_prediction_gain():
    s1p, _, s1, _, _ = speech_batch(1, 16000, seed=4).astype(np.float64)
    for L, zm, ld in ((512, False, None), (64, True, 1e-3), (1, False, None)):
        ref = D.sdr(s1p[0], s1[0], L, zm, ld)
        for g in (1e-3, 0.5, 7.0):
            assert abs(D.sdr(g * s1p[0], s1[0], L, zm, ld) - ref) < 1e-9


def test_short_fir_distortion_is_forgiven_by_sdr_only():
    """A prediction equal to the target through a random 16-tap FIR, plus -60 dB noise: the 512-tap distortion filter
    absorbs the FIR (SDR >= 40 dB) where the single scale of SI-SDR cannot (< 20 dB)."""
    T = 64000
    for seed in range(3):
        rng = np.random.default_rng(10 + seed)
        t = _clean(rng, T)
        h = rng.standard_normal(16) * np.exp(-np.arange(16) / 4)
        p = np.convolve(t, h)[:T]
        p = p + 1e-3 * np.linalg.norm(p) / np.sqrt(T) * rng.standard_normal(T)
        assert D.sdr(p, t) >= 40.0
        assert D.si_sdr(p, t) < 20.0


def test_one_tap_sdr_is_sisdr_without_eps():
    s1p, s2p, s1, _, _ = speech_batch(3, 16000, seed=5).astype(np.float64)
    for p, t in ((s1p, s1), (s2p, s1)):
        for b in range(3):
            assert abs(D.sdr(p[b], t[b], 1) - D.si_sdr(p[b], t[b], eps=0.0)) < 1e-12


def test_workspace_bytes_errors():
    from speech_separation_b200 import _lib

    lib = _lib.load()

    def err(B, T, L):
        assert lib.vatss_sdr_workspace_bytes(B, T, L) == 0
        return lib.vatss_last_error().decode()

    assert "empty batch" in err(0, 64000, 512)
    assert "empty batch" in err(2, 0, 512)
    assert "empty batch" in err(2, -5, 512)
    assert "at least 1" in err(2, 64000, 0)
    assert "longer than the signals" in err(2, 511, 512)
    assert "above 2048" in err(2, 64000, 2049)
    assert "at most 65535" in err(65536, 1000, 16)
    assert lib.vatss_sdr_workspace_bytes(2, 512, 512) > 0
    assert lib.vatss_sdr_workspace_bytes(1, 1, 1) > 0
    ten_min = lib.vatss_sdr_workspace_bytes(4, 600 * 16000, 512)
    assert 0 < ten_min < 2 ** 26
    rc = lib.vatss_sdr(None, None, None, None, None, 1, 64000, 512, 0, -1.0, None, None, None, ctypes.c_size_t(0), None)
    assert rc != 0 and "NULL" in lib.vatss_last_error().decode()
    rc = lib.vatss_pit_sisdr(None, None, None, None, None, 1, 64000, 0, None, None, None, None)
    assert rc != 0 and "NULL" in lib.vatss_last_error().decode()


def test_python_argument_errors_before_device_work():
    """CPU tensors: a ValueError (not the 'CUDA tensor' error) shows the arguments are checked first."""
    from speech_separation_b200 import SDRiMetric, SDRMetric, SISDRMetric, sdr_all, sisdr_all

    a = torch.zeros(2, 4000)
    for fn in (sdr_all, sisdr_all):
        with pytest.raises(RuntimeError, match="CUDA tensor"):
            fn(a, a, a, a)
        with pytest.raises(ValueError, match="expected"):
            fn(a, a, a, torch.zeros(2, 3999))
        with pytest.raises(ValueError, match="expected"):
            fn(a, a, a, a, mix=torch.zeros(3, 4000))
        with pytest.raises(ValueError, match=r"\(B, T\)"):
            fn(a[0], a[0], a[0], a[0])
        with pytest.raises(ValueError, match="empty"):
            fn(a[:0], a[:0], a[:0], a[:0])
    for L in (0, -3, 4001, 2049, 64.0, True, "512"):
        with pytest.raises(ValueError, match="filter_length"):
            sdr_all(a, a, a, a, filter_length=L)
    for ld in (-1e-3, float("nan"), float("inf"), "1"):
        with pytest.raises(ValueError, match="load_diag"):
            sdr_all(a, a, a, a, load_diag=ld)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        sdr_all(a, a, a, a, filter_length=2048, load_diag=0)
    with pytest.raises(ValueError, match="longer than the signals"):
        SDRMetric(filter_length=5000)(s1_pred=a, s2_pred=a, s1=a, s2=a)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        SDRiMetric()(s1_pred=a, s2_pred=a, s1=a, s2=a, mix=a)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        SISDRMetric()(s1_pred=a, s2_pred=a, s1=a, s2=a)


# ---------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def V():
    assert torch.cuda.is_available(), "run with -m gpu on a CUDA box"
    import speech_separation_b200 as V

    return V


def _gpu(arrs):
    return [torch.from_numpy(np.ascontiguousarray(a)).to(dev()) for a in arrs]


def _check(got, want, tol, what):
    """Equal NaN pattern (the mixture rows without a mixture), and |delta| <= tol everywhere else."""
    for g, w in zip((t.cpu().numpy() for t in got), want):
        assert np.array_equal(np.isnan(g), np.isnan(w)), (what, g, w)
        err = np.abs(np.nan_to_num(g) - np.nan_to_num(w))
        assert err.max() <= tol, (what, err.max(), np.unravel_index(err.argmax(), err.shape))


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,L,zero_mean,load_diag", [
    (32, 64000, 512, False, None),
    (32, 64000, 512, True, None),
    (3, 63999, 512, False, 1e-3),
    (3, 16001, 64, True, None),
    (1, 512, 512, False, None),
    (3, 512, 64, True, 1e-2),
    (1, 63999, 1, False, None),
    (32, 16001, 1, True, 0.1),
    (3, 64000, 64, False, 1e-5),
    (1, 16001, 512, True, 1e-3),
])
def test_against_oracle(V, B, T, L, zero_mean, load_diag):
    batch = speech_batch(B, T, seed=B * 7 + T + L)
    gb = _gpu(batch)
    x = [_f64(a) for a in batch]
    for mix in (True, False):
        m = x[4] if mix else None
        got = V.sisdr_all(*gb[:4], mix=gb[4] if mix else None, zero_mean=zero_mean)
        _check(got, D.pit_all(D.si_sdr, *x[:4], m, zero_mean=zero_mean), TOL_SISDR, "sisdr")
        got = V.sdr_all(*gb[:4], mix=gb[4] if mix else None, filter_length=L, zero_mean=zero_mean, load_diag=load_diag)
        want = D.pit_all(D.sdr, *x[:4], m, filter_length=L, zero_mean=zero_mean, load_diag=load_diag)
        _check(got, want, TOL_SDR, "sdr")
        if not mix:
            assert np.isnan(got[0][:, 4:].cpu().numpy()).all() and np.isnan(got[1][3:6].cpu().numpy()).all()


@pytest.mark.gpu
def test_all_zero_target_gives_nan_rows_only_for_it(V):
    batch = speech_batch(3, 16000, seed=70)
    zeroed = batch.copy()
    zeroed[2, 1] = 0.0          # utterance 1: s1 all zeros
    zeroed[4] = zeroed[2] + zeroed[3]
    rows, summ = V.sdr_all(*_gpu(zeroed))
    rows = rows.cpu().numpy()
    assert np.isnan(rows[1, [0, 3, 4]]).all()          # every pairing against the zero target
    assert np.isfinite(rows[1, [1, 2, 5]]).all()
    assert np.isfinite(np.delete(rows, 1, axis=0)).all()
    assert np.isnan(summ.cpu().numpy()[[0, 1, 2, 3, 4]]).all()
    for b in (0, 2):
        one = V.sdr_all(*(t[b:b + 1] for t in _gpu(zeroed)))[0]
        assert np.array_equal(one.cpu().numpy()[0], rows[b])


@pytest.mark.gpu
def test_reproducible_and_batch_independent(V):
    batch = _gpu(speech_batch(32, 64000, seed=30))
    for fn in (lambda *t: V.sisdr_all(*t[:4], mix=t[4]), lambda *t: V.sdr_all(*t[:4], mix=t[4]),
               lambda *t: V.sdr_all(*t[:4], mix=t[4], filter_length=64, zero_mean=True, load_diag=1e-3)):
        a = fn(*batch)
        b = fn(*batch)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
        for i in (0, 17, 31):
            one = fn(*(t[i:i + 1].clone() for t in batch))
            assert torch.equal(one[0][0], a[0][i])


@pytest.mark.gpu
def test_swapped_predictions_pick_the_other_permutation(V):
    s1p, s2p, s1, s2, mix = _gpu(speech_batch(4, 16000, seed=20, snrs=(5, 20)))
    for fn in (V.sisdr_all, V.sdr_all):
        rows, summ = fn(s1p, s2p, s1, s2, mix)
        rows_x, summ_x = fn(s2p, s1p, s1, s2, mix)
        assert summ[0] > summ[1] and summ_x[1] > summ_x[0]
        assert torch.equal(rows_x[:, :4], rows[:, [3, 2, 1, 0]])
        assert torch.equal(summ_x[[1, 0, 2, 3, 4, 5, 6]], summ)


@pytest.mark.gpu
def test_metric_classes_and_no_host_sync(V):
    s1p, s2p, s1, s2, mix = _gpu(speech_batch(4, 32000, seed=40))
    batch = dict(s1_pred=s1p, s2_pred=s2p, s1=s1, s2=s2, mix=mix)
    x = [t.cpu().double().numpy() for t in (s1p, s2p, s1, s2, mix)]
    _, r_sisdr = D.pit_all(D.si_sdr, *x)
    _, r_sdr = D.pit_all(D.sdr, *x, filter_length=256, load_diag=1e-4)
    cases = [(V.SISDRMetric(), r_sisdr[2], TOL_SISDR), (V.SDRMetric(filter_length=256, load_diag=1e-4), r_sdr[2], TOL_SDR),
             (V.SDRiMetric(filter_length=256, load_diag=1e-4), r_sdr[3], TOL_SDR)]
    for m, want, tol in cases:
        v = m(**batch)
        assert isinstance(v, float) and abs(v - want) <= tol
        per = m.per_utterance(**batch)
        assert per.dtype == torch.float64 and per.shape == (4,)
        m.device_value(**batch)
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            d = m.device_value(**batch)
        finally:
            torch.cuda.set_sync_debug_mode("default")
        assert d.is_cuda and d.dim() == 0 and d.dtype == torch.float32
        assert abs(float(d) - want) <= max(tol, 1e-6 * abs(want))
    rows, _ = V.sdr_all(s1p, s2p, s1, s2, mix, filter_length=256, load_diag=1e-4)
    sep = torch.maximum((rows[:, 0] + rows[:, 1]) / 2, (rows[:, 2] + rows[:, 3]) / 2)
    assert torch.equal(cases[1][0].per_utterance(**batch), sep)
    assert torch.equal(cases[2][0].per_utterance(**batch), sep - (rows[:, 4] + rows[:, 5]) / 2)
    assert V.SISDRMetric().name == "SISDRMetric" and V.SDRiMetric(name="SDRi").name == "SDRi"


@pytest.mark.gpu
def test_inferencer_tracks_sisdr_and_sdri(V):
    torch.manual_seed(42)
    kw = dict(num_features=128, video_emb_size=512, hidden_video=128, kernel_size_enc=7, hidden_dim=128, num_blocks=2,
              chunk_size=150, step_size=75, num_heads=4, dropout=0.1, bidir=True)
    net = V.DPTNAVWavEncDec(**kw).eval().to(dev())
    B, T = 2, 32000
    batches = []
    for i in range(3):
        _, _, s1, s2, mix = speech_batch(B, T, seed=50 + i)
        g = torch.Generator().manual_seed(60 + i)
        batches.append({"mix": torch.from_numpy(mix), "s1": torch.from_numpy(s1), "s2": torch.from_numpy(s2),
                        "s1_embedding": torch.randn(B, 512, T // 640, generator=g),
                        "s2_embedding": torch.randn(B, 512, T // 640, generator=g),
                        "audio_path": [f"/data/mix/utt_{i}_{b}.wav" for b in range(B)]})
    cfg = {"inferencer": {"device_tensors": ["mix", "s1", "s2", "s1_embedding", "s2_embedding"],
                          "from_pretrained": None}}
    mets = [V.SISNRiMetric(name="SISNRi"), V.SISDRMetric(name="SISDR"), V.SDRiMetric(name="SDRi")]
    inf = V.Inferencer(net, cfg, dev(), {"val": [dict(b) for b in batches]}, None, metrics={"inference": mets},
                       skip_model_load=True)
    logs = inf.run_inference()["val"]
    want = {"SISNRi": 0.0, "SISDR": 0.0, "SDRi": 0.0}
    with torch.no_grad():
        for b in batches:
            d = {k: (v.to(dev()) if torch.is_tensor(v) else v) for k, v in b.items()}
            d.update(net(**d))
            want["SISNRi"] += float(mets[0](**d)) / 3
            want["SISDR"] += mets[1](**d) / 3
            want["SDRi"] += mets[2](**d) / 3
    for k in want:
        assert logs[k] == pytest.approx(want[k], abs=1e-4), k


@pytest.mark.gpu
def test_long_recording_separated_then_scored(V):
    from oracle.gen_golden import PROD

    torch.manual_seed(42)
    lf = V.LongFormSeparator(V.DPTNWavEncDec(**dict(PROD["dptn_wav"], num_blocks=2)).eval().to(dev()))
    T = 60 * 16000
    _, _, s1, s2, mix = speech_batch(1, T, seed=60)
    with torch.no_grad():
        out = lf(mix=torch.from_numpy(mix).to(dev()))
    g = [out["s1_pred"], out["s2_pred"]] + _gpu([s1, s2, mix])
    x = [t.cpu().double().numpy() for t in g]
    _check(V.sisdr_all(*g[:4], mix=g[4]), D.pit_all(D.si_sdr, *x), TOL_SISDR, "sisdr 60 s")
    _check(V.sdr_all(*g[:4], mix=g[4]), D.pit_all(D.sdr, *x), TOL_SDR, "sdr 60 s")
