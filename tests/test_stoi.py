"""STOI / ESTOI (`vatss_stoi`, `stoi_all`, `STOIMetric`) against the fp64 restatement in oracle/stoi_oracle.py
(DESIGN.md §8).  Parity with pystoi itself is not pinned: pystoi is not a dependency."""
import ctypes

import numpy as np
import pytest
import torch
from scipy.signal import resample_poly

from oracle import stoi_oracle as S

TOL = 1e-5


# ---------------------------------------------------------------------------------------------
# speech-like test signals
# ---------------------------------------------------------------------------------------------
def _clean(rng, T, fs):
    """Noise under a random syllable-rate envelope (piecewise levels of 0.1 s between -30 and 0 dB), with leading,
    trailing and interior silences, some exact zeros and some at -60 dB."""
    seg = fs // 10
    n = -(-T // seg)
    lv = 10 ** (rng.uniform(-30, 0, n) / 20)
    for where in (0, n - 1, int(rng.integers(2, max(3, n - 2)))):
        lv[where] = 0.0 if rng.random() < 0.5 else 1e-3
    env = np.repeat(lv, seg)[:T]
    return env * rng.standard_normal(T)


def _clear_of_threshold(x, fs, margin=1e-3):
    """No frame energy within `margin` dB of the silent-frame threshold: a kept-frame mismatch is then a bug, not a
    tie between fp32 and fp64."""
    e = S.frame_energies(S.resample(x, fs))
    return np.min(np.abs(e - (e.max() - S.DYN_RANGE))) > margin


def speech_batch(B, T, fs, seed, snrs=(-5, 20)):
    """(s1_pred, s2_pred, s1, s2) float32 (B, T): targets from `_clean`, predictions = target + white noise at SNRs
    between snrs[0] and snrs[1] dB.  Utterances whose clean frames touch the threshold are redrawn."""
    rng = np.random.default_rng(seed)
    out = np.zeros((4, B, T), np.float32)
    for b in range(B):
        for t in (2, 3):
            while True:
                x = _clean(rng, T, fs).astype(np.float32)
                if _clear_of_threshold(x.astype(np.float64), fs):
                    break
            out[t, b] = x
        for k, t in ((0, 2), (1, 3)):
            x = out[t, b].astype(np.float64)
            snr = rng.uniform(*snrs)
            noise = rng.standard_normal(T)
            noise *= np.sqrt(np.mean(x ** 2) / np.mean(noise ** 2) / 10 ** (snr / 10))
            out[k, b] = (x + noise).astype(np.float32)
    return out


# ---------------------------------------------------------------------------------------------
# CPU: the oracle on its own
# ---------------------------------------------------------------------------------------------
def test_oracle_identity():
    s1p, _, s1, _ = speech_batch(1, 32000, 16000, seed=1).astype(np.float64)
    x, y = s1[0], s1p[0]
    assert abs(S.stoi(x, x) - 1.0) < 1e-12
    assert abs(S.stoi(x, x, extended=True) - 1.0) < 1e-12
    assert S.stoi(x, y) < 1.0


def test_oracle_scale_invariant():
    s1p, _, s1, _ = speech_batch(1, 32000, 16000, seed=2).astype(np.float64)
    x, y = s1[0], s1p[0]
    for ext in (False, True):
        ref = S.stoi(x, y, extended=ext)
        for a, b in ((3.0, 0.2), (0.01, 50.0)):
            assert abs(S.stoi(a * x, b * y, extended=ext) - ref) < 1e-9


def test_oracle_zero_prediction():
    _, _, s1, _ = speech_batch(1, 32000, 16000, seed=3).astype(np.float64)
    assert S.stoi(s1[0], np.zeros_like(s1[0])) == 0.0
    assert S.stoi(s1[0], np.zeros_like(s1[0]), extended=True) == 0.0


def test_oracle_falls_with_snr():
    T = 24000
    for ext in (False, True):
        means = []
        for snr in (-10, -5, 0, 5, 10, 20):
            vals = []
            for seed in range(4):
                rng = np.random.default_rng(100 + seed)
                x = _clean(rng, T, 16000)
                n = rng.standard_normal(T)
                n *= np.sqrt(np.mean(x ** 2) / np.mean(n ** 2) / 10 ** (snr / 10))
                vals.append(S.stoi(x, x + n, extended=ext))
            means.append(np.mean(vals))
        assert all(a < b for a, b in zip(means, means[1:])), means


def test_resample_filter_and_closed_form():
    h, L, beta = S.resample_filter(5, 8)
    assert len(h) == 581 and L == 290
    assert beta == pytest.approx(5.65326, abs=1e-12)
    assert abs(h.sum() - 1.0) < 1e-12
    rng = np.random.default_rng(0)
    for fs, T in ((16000, 3001), (8000, 1203), (22050, 2205)):
        x = rng.standard_normal(T)
        p, q = S.resample_ratio(fs)
        hh, _, _ = S.resample_filter(p, q)
        a = resample_poly(x, p, q, window=hh)
        b = S.resample_closed_form(x, fs)
        assert len(a) == len(b) == S.resampled_length(T, fs) == -(-T * p // q)
        assert np.max(np.abs(a - b)) < 1e-12
        assert np.array_equal(S.resample(x, fs), a)
    assert S.resample_ratio(16000) == (5, 8) and S.resample_ratio(8000) == (5, 4)


def test_band_table():
    assert S.BAND_EDGES == [(7, 9), (9, 11), (11, 14), (14, 17), (17, 22), (22, 27), (27, 34), (34, 43), (43, 55),
                            (55, 69), (69, 87), (87, 109), (109, 138), (138, 174), (174, 219)]
    assert S.OBM.shape == (15, 257) and S.OBM.sum() == 219 - 7


def _all_loud(K, seed=0):
    """A 10 kHz signal of exactly K frames, every one of them kept (white noise, flat level)."""
    return np.random.default_rng(seed).standard_normal(S.N_FRAME + (K - 1) * S.HOP)


def test_frame_count_quirks():
    x = _all_loud(40)
    xs, ys, mask = S.remove_silent_frames(x, x)
    assert mask.sum() == 40 and len(xs) == 39 * 128 + 256
    assert S.stft(xs).shape == (39, 257)        # K kept frames -> K - 1 STFT frames
    for K in (30, 31):
        x = _all_loud(K)
        y = x + 0.3 * np.random.default_rng(1).standard_normal(len(x))
        for ext in (False, True):
            v = S.stoi(x, y, fs=10000, extended=ext)
            assert (v == 1e-5) == (K == 30) and 0 < v < 1
    with pytest.raises(ValueError, match="shorter than one"):
        S.stoi(np.ones(255), np.ones(255), fs=10000)
    with pytest.raises(ValueError, match="shorter than one"):
        S.stoi(np.ones(408), np.ones(408), fs=16000)   # ceil(408 * 5 / 8) = 255; 409 samples give 256


def test_workspace_bytes_errors():
    from speech_separation_b200 import _lib

    lib = _lib.load()

    def err(B, T, fs):
        assert lib.vatss_stoi_workspace_bytes(B, T, fs) == 0
        return lib.vatss_last_error().decode()

    assert "empty batch" in err(0, 64000, 16000)
    assert "empty batch" in err(2, 0, 16000)
    assert "sample rate" in err(2, 64000, 0)
    assert "sample rate" in err(2, 64000, -16000)
    assert "shorter than one 256-sample frame" in err(2, 408, 16000)
    assert "shorter than one 256-sample frame" in err(2, 255, 10000)
    assert lib.vatss_stoi_workspace_bytes(2, 409, 16000) > 0
    assert lib.vatss_stoi_workspace_bytes(2, 256, 10000) > 0
    hour = lib.vatss_stoi_workspace_bytes(1, 3600 * 16000, 16000)
    assert 0 < hour < 2 ** 31                     # one hour at 16 kHz
    rc = lib.vatss_stoi(None, None, None, None, 1, 64000, 16000, 0, None, None, None, None, ctypes.c_size_t(0), None)
    assert rc != 0 and "NULL" in lib.vatss_last_error().decode()


def test_python_argument_errors_cpu():
    from speech_separation_b200 import STOIMetric, stoi_all

    a = torch.zeros(2, 64000)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        stoi_all(a, a, a, a)
    with pytest.raises(ValueError, match="expected"):
        stoi_all(a, a, a, torch.zeros(2, 63999))
    with pytest.raises(ValueError, match=r"\(B, T\)"):
        stoi_all(a[0], a[0], a[0], a[0])
    for fs in (0, -8000, 16000.5, True):
        with pytest.raises(ValueError, match="fs"):
            stoi_all(a, a, a, a, fs=fs)
    with pytest.raises(ValueError, match="shorter than one"):
        stoi_all(a[:, :408], a[:, :408], a[:, :408], a[:, :408])
    with pytest.raises(ValueError, match="empty"):
        stoi_all(a[:0], a[:0], a[:0], a[:0])
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        STOIMetric()(s1_pred=a, s2_pred=a, s1=a, s2=a)


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


def _check_against_oracle(V, batch, fs):
    for ext in (False, True):
        rows, kept, summary = V.stoi_all(*_gpu(batch), fs=fs, extended=ext)
        r_rows, r_kept, r_sum = S.stoi_all(*batch.astype(np.float64), fs=fs, extended=ext)
        assert np.array_equal(kept.cpu().numpy(), r_kept)
        err = np.abs(rows.cpu().numpy() - r_rows)
        assert err.max() <= TOL, (ext, err.max(), np.unravel_index(err.argmax(), err.shape))
        assert np.abs(summary.cpu().numpy() - r_sum).max() <= TOL


@pytest.mark.gpu
def test_cfg2_batch_against_oracle(V):
    """32 x 4 s at 16 kHz, SNR -5 .. 20 dB."""
    batch = speech_batch(32, 64000, 16000, seed=10)
    for t in (2, 3):
        assert all(_clear_of_threshold(x.astype(np.float64), 16000) for x in batch[t])
    _check_against_oracle(V, batch, 16000)


@pytest.mark.gpu
@pytest.mark.parametrize("fs,T", [(16000, 63999), (16000, 16001), (16000, 64037), (10000, 40000), (10000, 25037),
                                  (8000, 32000), (8000, 32037)])
def test_lengths_and_rates_against_oracle(V, fs, T):
    _check_against_oracle(V, speech_batch(4, T, fs, seed=T + fs), fs)


@pytest.mark.gpu
def test_swapped_predictions_pick_the_other_permutation(V):
    s1p, s2p, s1, s2 = _gpu(speech_batch(8, 32000, 16000, seed=20, snrs=(5, 20)))
    for ext in (False, True):
        rows, _, summ = V.stoi_all(s1p, s2p, s1, s2, extended=ext)
        rows_x, _, summ_x = V.stoi_all(s2p, s1p, s1, s2, extended=ext)
        assert summ[0] > summ[1] and summ_x[1] > summ_x[0]
        assert torch.equal(rows_x, rows[:, [3, 2, 1, 0]])
        assert torch.equal(summ_x[[1, 0, 2]], summ)


@pytest.mark.gpu
def test_boundaries(V):
    """29 / 30 STFT frames, an all-zero prediction, a target with one loud frame."""
    rng = np.random.default_rng(5)
    for K, short in ((30, True), (31, False)):
        T = S.N_FRAME + (K - 1) * S.HOP
        x = rng.standard_normal((2, T)).astype(np.float32)
        y = (x + 0.3 * rng.standard_normal((2, T))).astype(np.float32)
        batch = np.stack([y, y[::-1], x, x[::-1]])
        for ext in (False, True):
            rows, kept, _ = V.stoi_all(*_gpu(batch), fs=10000, extended=ext)
            assert (kept.cpu().numpy() == K).all()
            assert ((rows.cpu().numpy() == 1e-5).all()) == short
        _check_against_oracle(V, batch, 10000)
    s1p, s2p, s1, s2 = speech_batch(2, 32000, 16000, seed=6)
    zero = np.zeros_like(s1p)
    for ext in (False, True):
        rows, _, _ = V.stoi_all(*_gpu([zero, zero, s1, s2]), extended=ext)
        assert (rows.cpu().numpy() == 0.0).all()
    loud = (1e-4 * rng.standard_normal((2, 32000))).astype(np.float32)
    loud[:, 16000:16160] += rng.standard_normal((2, 160)).astype(np.float32)
    assert all(_clear_of_threshold(x.astype(np.float64), 16000) for x in loud)
    batch = np.stack([s1p, s2p, loud, loud.copy()])
    _check_against_oracle(V, batch, 16000)
    rows, kept, _ = V.stoi_all(*_gpu(batch))
    assert (rows.cpu().numpy() == 1e-5).all() and (kept.cpu().numpy() <= 4).all()


@pytest.mark.gpu
def test_reproducible_and_batch_independent(V):
    batch = _gpu(speech_batch(32, 64000, 16000, seed=30))
    for ext in (False, True):
        a = V.stoi_all(*batch, extended=ext)
        b = V.stoi_all(*batch, extended=ext)
        for u, v in zip(a, b):
            assert torch.equal(u, v)
        for i in (0, 17, 31):
            one = V.stoi_all(*(t[i:i + 1].clone() for t in batch), extended=ext)
            assert torch.equal(one[0][0], a[0][i]) and torch.equal(one[1][0], a[1][i])


@pytest.mark.gpu
def test_metric_values_and_no_host_sync(V):
    s1p, s2p, s1, s2 = _gpu(speech_batch(4, 32000, 16000, seed=40))
    batch = dict(s1_pred=s1p, s2_pred=s2p, s1=s1, s2=s2, mix=s1 + s2)
    for ext in (False, True):
        m = V.STOIMetric(extended=ext)
        _, _, ref = S.stoi_all(*(t.cpu().double().numpy() for t in (s1p, s2p, s1, s2)), extended=ext)
        assert abs(m(**batch) - ref[2]) <= TOL
        rows, _, _ = V.stoi_all(s1p, s2p, s1, s2, extended=ext)
        per = m.per_utterance(**batch)
        assert per.dtype == torch.float64 and per.shape == (4,)
        assert torch.equal(per, torch.maximum((rows[:, 0] + rows[:, 1]) / 2, (rows[:, 2] + rows[:, 3]) / 2))
        m.device_value(**batch)
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            v = m.device_value(**batch)
        finally:
            torch.cuda.set_sync_debug_mode("default")
        assert v.is_cuda and v.dim() == 0 and v.dtype == torch.float32
        assert abs(float(v) - ref[2]) <= TOL
    assert V.STOIMetric().name == "STOIMetric" and V.STOIMetric(name="ESTOI", extended=True).name == "ESTOI"


@pytest.mark.gpu
def test_inferencer_tracks_stoi(V, tmp_path):
    from torch.utils.data import DataLoader

    from oracle.gen_golden import PROD

    torch.manual_seed(42)
    net = V.DPTNWavEncDec(**dict(PROD["dptn_wav"], num_blocks=2)).eval().to(dev())
    T = 32000
    data = speech_batch(6, T, 16000, seed=50)

    class Utterances(torch.utils.data.Dataset):
        def __len__(self):
            return 6

        def __getitem__(self, i):
            s1, s2 = torch.from_numpy(data[2, i]), torch.from_numpy(data[3, i])
            return {"mix": s1 + s2, "s1": s1, "s2": s2, "audio_path": f"/data/mix/utt_{i}.wav"}

    loader = DataLoader(Utterances(), batch_size=3)
    cfg = {"inferencer": {"device_tensors": ["mix", "s1", "s2"]}}
    mets = [V.SISNRiMetric(name="SISNRi"), V.STOIMetric(name="STOI"), V.STOIMetric(name="ESTOI", extended=True)]
    inf = V.Inferencer(net, cfg, dev(), {"test": loader}, None, metrics={"inference": mets}, skip_model_load=True)
    logs = inf.run_inference()["test"]
    want = {"STOI": 0.0, "ESTOI": 0.0}
    with torch.no_grad():
        for b in loader:
            out = net(mix=b["mix"].to(dev()))
            args = [out["s1_pred"].cpu().double().numpy(), out["s2_pred"].cpu().double().numpy(),
                    b["s1"].double().numpy(), b["s2"].double().numpy()]
            want["STOI"] += S.stoi_all(*args)[2][2] / len(loader)
            want["ESTOI"] += S.stoi_all(*args, extended=True)[2][2] / len(loader)
    assert logs["STOI"] == pytest.approx(want["STOI"], abs=TOL)
    assert logs["ESTOI"] == pytest.approx(want["ESTOI"], abs=TOL)
    assert "SISNRi" in logs


@pytest.mark.gpu
def test_long_recording_separated_then_scored(V):
    from oracle.gen_golden import PROD

    torch.manual_seed(42)
    lf = V.LongFormSeparator(V.DPTNWavEncDec(**dict(PROD["dptn_wav"], num_blocks=2)).eval().to(dev()))
    T = 60 * 16000
    _, _, s1, s2 = speech_batch(1, T, 16000, seed=60)
    with torch.no_grad():
        out = lf(mix=torch.from_numpy(s1 + s2).to(dev()))
    for ext in (False, True):
        rows, kept, summ = V.stoi_all(out["s1_pred"], out["s2_pred"], *_gpu([s1, s2]), extended=ext)
        r_rows, r_kept, r_sum = S.stoi_all(out["s1_pred"].cpu().double().numpy(),
                                           out["s2_pred"].cpu().double().numpy(), s1.astype(np.float64),
                                           s2.astype(np.float64), extended=ext)
        assert np.array_equal(kept.cpu().numpy(), r_kept)
        assert np.abs(rows.cpu().numpy() - r_rows).max() <= TOL
        assert np.abs(summ.cpu().numpy() - r_sum).max() <= TOL
