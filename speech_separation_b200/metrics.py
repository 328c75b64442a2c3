"""SI-SNR / SI-SNRi metrics, drop-in for src/metrics/si_snr.py:6-12 and src/metrics/si_snri.py:7-30, STOI / ESTOI,
drop-in for src/metrics/stoi.py, SI-SDR, drop-in for src/metrics/si_sdr.py, and SDR / SDRi.

The reference wraps torchmetrics' ScaleInvariantSignalNoiseRatio, calls it 4 (+2) times and
`.item()`s each result; PIT is batch-level (`max` over the two permutations of the batch means,
src/metrics/base_metric.py:53-60).  Here one kernel pass produces all six per-utterance values
and the batch-level decisions (`vatss_pit_sisnr`).  STOI is computed on the device by `vatss_stoi` (DESIGN.md §8):
all four pairings of the batch and the same batch-level PIT, where the reference runs pystoi on the host per pair.
SI-SDR (`vatss_pit_sisdr`) and BSS-eval SDR with its distortion filter (`vatss_sdr`) follow torchmetrics' definitions
(DESIGN.md §9); all six pairings and the summary come from one call each.
"""
import ctypes
import math
import numbers

import torch

from . import _lib
from .loss import pit_sisnr_all


class SS2BaseMetric:
    def __init__(self, name=None, lower_better=False, *args, **kwargs):
        self.name = name if name is not None else type(self).__name__
        if lower_better:
            raise ValueError("the fused SI-SNR kernel implements higher-is-better PIT only")
        self.device = kwargs.get("device", None)

    def _summary(self, s1_pred, s2_pred, s1, s2, mix=None):
        if self.device is not None and self.device != "auto":
            dev = torch.device(self.device)
            s1_pred, s2_pred, s1, s2 = (t.to(dev) for t in (s1_pred, s2_pred, s1, s2))
            mix = mix.to(dev) if mix is not None else None
        return pit_sisnr_all(s1_pred, s2_pred, s1, s2, mix)

    def _shared_summary(self, shared, s1_pred, s2_pred, s1, s2, mix):
        """summary[8] of the batch; `shared` (inference._SharedSisnr) lets several metrics reuse one kernel pass."""
        if shared is not None and (self.device is None or self.device == "auto"):
            return shared.summary({"s1_pred": s1_pred, "s2_pred": s2_pred, "s1": s1, "s2": s2, "mix": mix})
        return self._summary(s1_pred, s2_pred, s1, s2, mix)[2]


class SISNRMetric(SS2BaseMetric):
    """__call__(**batch) -> float: batch-level PIT SI-SNR in dB."""

    def __call__(self, s1_pred, s2_pred, s1, s2, **batch):
        _, _, summary = self._summary(s1_pred, s2_pred, s1, s2)
        return float(summary[3].item())

    def device_value(self, s1_pred, s2_pred, s1, s2, mix=None, shared=None, **batch):
        """Same value as __call__, as a 0-d float32 device tensor (no host synchronisation)."""
        return self._shared_summary(shared, s1_pred, s2_pred, s1, s2, mix)[3].float()


class SISNRiMetric(SS2BaseMetric):
    """__call__(**batch) -> 0-d tensor: PIT SI-SNR minus the mean SI-SNR of the mixture."""

    def __call__(self, s1_pred, s2_pred, s1, s2, mix, **batch):
        _, _, summary = self._summary(s1_pred, s2_pred, s1, s2, mix)
        return summary[4].float()

    def device_value(self, s1_pred, s2_pred, s1, s2, mix, shared=None, **batch):
        return self._shared_summary(shared, s1_pred, s2_pred, s1, s2, mix)[4].float()

    def per_utterance(self, s1_pred, s2_pred, s1, s2, mix, **batch):
        """Per-utterance PIT SI-SNRi (B,) f64 - what src/utils/eval_si_snri.py:31-39 computes file by file."""
        rows, _, _ = self._summary(s1_pred, s2_pred, s1, s2, mix)
        sep = torch.maximum((rows[:, 0] + rows[:, 1]) / 2, (rows[:, 2] + rows[:, 3]) / 2)
        return sep - (rows[:, 4] + rows[:, 5]) / 2


def stoi_all(s1_pred, s2_pred, s1, s2, fs=16000, extended=False):
    """STOI (ESTOI with extended=True) of the four pairings of a batch, on the device (`vatss_stoi`).

    Inputs are (B, T) CUDA tensors at `fs` Hz.  Returns (rows (B,4) f64, kept (B,2) int32, summary (3,) f64):
    rows: per-utterance [s1p.s1, s2p.s2, s1p.s2, s2p.s1]; kept: frames of s1 and s2 that survive the silent-frame
    removal; summary: [mean (row0 + row1)/2, mean (row2 + row3)/2, max of the two] (batch-level PIT).
    Argument errors raise before any device work."""
    ts = {"s1_pred": s1_pred, "s2_pred": s2_pred, "s1": s1, "s2": s2}
    for name, t in ts.items():
        if not isinstance(t, torch.Tensor) or t.dim() != 2:
            raise ValueError(f"{name} must be a (B, T) tensor, got {getattr(t, 'shape', type(t))}")
        if t.shape != s1_pred.shape:
            raise ValueError(f"{name} has shape {tuple(t.shape)}, expected {tuple(s1_pred.shape)}")
    if isinstance(fs, bool) or not isinstance(fs, numbers.Integral) or fs <= 0:
        raise ValueError(f"fs must be a positive integer sample rate, got {fs!r}")
    B, T = s1_pred.shape
    if B == 0 or T == 0:
        raise ValueError(f"empty batch of shape {(B, T)}")
    lib = _lib.load()
    nbytes = lib.vatss_stoi_workspace_bytes(B, T, int(fs))
    if nbytes == 0:
        raise ValueError(lib.vatss_last_error().decode("utf-8", "replace"))
    for name, t in ts.items():
        _lib.require_cuda(t, name)
    s1_pred, s2_pred, s1, s2 = (_lib.f32c(t, n) for n, t in ts.items())
    dev = s1_pred.device
    rows = torch.empty((B, 4), dtype=torch.float64, device=dev)
    kept = torch.empty((B, 2), dtype=torch.int32, device=dev)
    summary = torch.empty(3, dtype=torch.float64, device=dev)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.vatss_stoi(s1_pred.data_ptr(), s2_pred.data_ptr(), s1.data_ptr(), s2.data_ptr(), B, T, int(fs),
                                  1 if extended else 0, rows.data_ptr(), kept.data_ptr(), summary.data_ptr(),
                                  ws.data_ptr(), ctypes.c_size_t(nbytes), _lib.stream_ptr()), "vatss_stoi")
    return rows, kept, summary


class STOIMetric(SS2BaseMetric):
    """__call__(**batch) -> float: batch-level PIT STOI (ESTOI with extended=True) of the predictions.

    Drop-in for src/metrics/stoi.py.  That class is not part of this repository, so the constructor
    `STOIMetric(name=None, fs=16000, extended=False, device=None)` is modelled on torchmetrics'
    ShortTimeObjectiveIntelligibility(fs, extended), which it wraps (INTEGRATION.md)."""

    def __init__(self, name=None, fs=16000, extended=False, device=None, *args, **kwargs):
        super().__init__(name=name, device=device)
        self.fs = fs
        self.extended = extended

    def _stoi(self, s1_pred, s2_pred, s1, s2):
        if self.device is not None and self.device != "auto":
            dev = torch.device(self.device)
            s1_pred, s2_pred, s1, s2 = (t.to(dev) for t in (s1_pred, s2_pred, s1, s2))
        return stoi_all(s1_pred, s2_pred, s1, s2, fs=self.fs, extended=self.extended)

    def __call__(self, s1_pred, s2_pred, s1, s2, **batch):
        return float(self._stoi(s1_pred, s2_pred, s1, s2)[2][2].item())

    def device_value(self, s1_pred, s2_pred, s1, s2, shared=None, **batch):
        """Same value as __call__, as a 0-d float32 device tensor (no host synchronisation)."""
        return self._stoi(s1_pred, s2_pred, s1, s2)[2][2].float()

    def per_utterance(self, s1_pred, s2_pred, s1, s2, **batch):
        """(B,) f64: per utterance, the better of the two permutations."""
        rows, _, _ = self._stoi(s1_pred, s2_pred, s1, s2)
        return torch.maximum((rows[:, 0] + rows[:, 1]) / 2, (rows[:, 2] + rows[:, 3]) / 2)


def _pit_inputs(s1_pred, s2_pred, s1, s2, mix):
    """Validates the (B, T) inputs before any device work; returns them as float32 contiguous CUDA tensors."""
    ts = {"s1_pred": s1_pred, "s2_pred": s2_pred, "s1": s1, "s2": s2}
    if mix is not None:
        ts["mix"] = mix
    for name, t in ts.items():
        if not isinstance(t, torch.Tensor) or t.dim() != 2:
            raise ValueError(f"{name} must be a (B, T) tensor, got {getattr(t, 'shape', type(t))}")
        if t.shape != s1_pred.shape:
            raise ValueError(f"{name} has shape {tuple(t.shape)}, expected {tuple(s1_pred.shape)}")
    B, T = s1_pred.shape
    if B == 0 or T == 0:
        raise ValueError(f"empty batch of shape {(B, T)}")
    return ts


def _ptrs(ts):
    return [ts[n].data_ptr() for n in ("s1_pred", "s2_pred", "s1", "s2")] + \
        [ts["mix"].data_ptr() if "mix" in ts else None]


def sisdr_all(s1_pred, s2_pred, s1, s2, mix=None, zero_mean=False):
    """SI-SDR (torchmetrics' form, eps = FLT_EPSILON) of the six pairings of a batch, on the device (`vatss_pit_sisdr`).

    Inputs are (B, T) CUDA tensors; mix may be None.  Returns (rows (B,6) f64, summary (7,) f64): rows per utterance
    [s1p.s1, s2p.s2, s1p.s2, s2p.s1, mix.s1, mix.s2] in dB (the last two NaN without mix); summary [mean (row0 +
    row1)/2, mean (row2 + row3)/2, max of the two (batch-level PIT), SI-SDRi = max - mean (row4 + row5)/2, mean row4,
    mean row5, B] (3..5 NaN without mix).  Argument errors raise before any device work."""
    ts = _pit_inputs(s1_pred, s2_pred, s1, s2, mix)
    B, T = s1_pred.shape
    if B > 65535:
        raise ValueError(f"batch of {B} utterances: at most 65535")
    lib = _lib.load()
    for name, t in ts.items():
        _lib.require_cuda(t, name)
    ts = {n: _lib.f32c(t, n) for n, t in ts.items()}
    dev = ts["s1_pred"].device
    rows = torch.empty((B, 6), dtype=torch.float64, device=dev)
    summary = torch.empty(7, dtype=torch.float64, device=dev)
    scratch = torch.empty(B * lib.vatss_sisnr_chunks(T) * 16, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.vatss_pit_sisdr(*_ptrs(ts), B, T, 1 if zero_mean else 0, rows.data_ptr(), summary.data_ptr(),
                                       scratch.data_ptr(), _lib.stream_ptr()), "vatss_pit_sisdr")
    return rows, summary


def sdr_all(s1_pred, s2_pred, s1, s2, mix=None, filter_length=512, zero_mean=False, load_diag=None):
    """BSS-eval SDR with a `filter_length`-tap distortion filter (torchmetrics' signal_distortion_ratio, direct solve)
    of the six pairings of a batch, on the device (`vatss_sdr`).  Rows and summary as for `sisdr_all` (summary[3] is
    SDRi).  A target whose Toeplitz system is singular (all zeros without load_diag) gets NaN rows.
    Argument errors raise before any device work."""
    ts = _pit_inputs(s1_pred, s2_pred, s1, s2, mix)
    if isinstance(filter_length, bool) or not isinstance(filter_length, numbers.Integral):
        raise ValueError(f"filter_length must be an integer, got {filter_length!r}")
    if load_diag is not None and (isinstance(load_diag, bool) or not isinstance(load_diag, numbers.Real)
                                  or not math.isfinite(load_diag) or load_diag < 0):
        raise ValueError(f"load_diag must be None or a finite number >= 0, got {load_diag!r}")
    B, T = s1_pred.shape
    lib = _lib.load()
    nbytes = lib.vatss_sdr_workspace_bytes(B, T, int(filter_length))
    if nbytes == 0:
        raise ValueError(lib.vatss_last_error().decode("utf-8", "replace"))
    for name, t in ts.items():
        _lib.require_cuda(t, name)
    ts = {n: _lib.f32c(t, n) for n, t in ts.items()}
    dev = ts["s1_pred"].device
    rows = torch.empty((B, 6), dtype=torch.float64, device=dev)
    summary = torch.empty(7, dtype=torch.float64, device=dev)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.vatss_sdr(*_ptrs(ts), B, T, int(filter_length), 1 if zero_mean else 0,
                                 -1.0 if load_diag is None else float(load_diag), rows.data_ptr(), summary.data_ptr(),
                                 ws.data_ptr(), ctypes.c_size_t(nbytes), _lib.stream_ptr()), "vatss_sdr")
    return rows, summary


class _PitRowsMetric(SS2BaseMetric):
    """Shared face of the SI-SDR / SDR classes: `_all(s1_pred, s2_pred, s1, s2, mix)` -> (rows (B,6), summary (7))."""

    _with_mix = False   # the i-variants score the mixture too and report summary[3]

    def _rows(self, s1_pred, s2_pred, s1, s2, mix):
        if self.device is not None and self.device != "auto":
            dev = torch.device(self.device)
            s1_pred, s2_pred, s1, s2 = (t.to(dev) for t in (s1_pred, s2_pred, s1, s2))
            mix = mix.to(dev) if mix is not None else None
        return self._all(s1_pred, s2_pred, s1, s2, mix if self._with_mix else None)

    def _value(self, s1_pred, s2_pred, s1, s2, mix):
        return self._rows(s1_pred, s2_pred, s1, s2, mix)[1][3 if self._with_mix else 2]

    def __call__(self, s1_pred, s2_pred, s1, s2, mix=None, **batch):
        return float(self._value(s1_pred, s2_pred, s1, s2, mix).item())

    def device_value(self, s1_pred, s2_pred, s1, s2, mix=None, shared=None, **batch):
        """Same value as __call__, as a 0-d float32 device tensor (no host synchronisation)."""
        return self._value(s1_pred, s2_pred, s1, s2, mix).float()

    def per_utterance(self, s1_pred, s2_pred, s1, s2, mix=None, **batch):
        """(B,) f64: per utterance, the better of the two permutations (minus the mixture's mean for the i-variants)."""
        rows, _ = self._rows(s1_pred, s2_pred, s1, s2, mix)
        sep = torch.maximum((rows[:, 0] + rows[:, 1]) / 2, (rows[:, 2] + rows[:, 3]) / 2)
        return sep - (rows[:, 4] + rows[:, 5]) / 2 if self._with_mix else sep


class SISDRMetric(_PitRowsMetric):
    """__call__(**batch) -> float: batch-level PIT SI-SDR in dB.  Drop-in for src/metrics/si_sdr.py (torchmetrics'
    ScaleInvariantSignalDistortionRatio behind SS2BaseMetric's PIT); zero_mean=False as in torchmetrics."""

    def __init__(self, name=None, zero_mean=False, device=None, *args, **kwargs):
        super().__init__(name=name, device=device)
        self.zero_mean = zero_mean

    def _all(self, s1_pred, s2_pred, s1, s2, mix):
        return sisdr_all(s1_pred, s2_pred, s1, s2, mix, zero_mean=self.zero_mean)


class SDRMetric(_PitRowsMetric):
    """__call__(**batch) -> float: batch-level PIT SDR in dB, modelled on torchmetrics'
    SignalDistortionRatio(filter_length, zero_mean, load_diag) (direct solve; no conjugate-gradient path)."""

    def __init__(self, name=None, filter_length=512, zero_mean=False, load_diag=None, device=None, *args, **kwargs):
        super().__init__(name=name, device=device)
        self.filter_length = filter_length
        self.zero_mean = zero_mean
        self.load_diag = load_diag

    def _all(self, s1_pred, s2_pred, s1, s2, mix):
        return sdr_all(s1_pred, s2_pred, s1, s2, mix, filter_length=self.filter_length, zero_mean=self.zero_mean,
                       load_diag=self.load_diag)


class SDRiMetric(SDRMetric):
    """__call__(**batch) -> float: PIT SDR minus the mean SDR of the mixture against s1 and s2 (as SISNRiMetric)."""

    _with_mix = True

    def __call__(self, s1_pred, s2_pred, s1, s2, mix, **batch):
        return super().__call__(s1_pred, s2_pred, s1, s2, mix)

    def device_value(self, s1_pred, s2_pred, s1, s2, mix, shared=None, **batch):
        return super().device_value(s1_pred, s2_pred, s1, s2, mix)

    def per_utterance(self, s1_pred, s2_pred, s1, s2, mix, **batch):
        return super().per_utterance(s1_pred, s2_pred, s1, s2, mix)
