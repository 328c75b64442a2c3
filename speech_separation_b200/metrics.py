"""SI-SNR / SI-SNRi metrics, drop-in for src/metrics/si_snr.py:6-12 and src/metrics/si_snri.py:7-30, and STOI / ESTOI,
drop-in for src/metrics/stoi.py.

The reference wraps torchmetrics' ScaleInvariantSignalNoiseRatio, calls it 4 (+2) times and
`.item()`s each result; PIT is batch-level (`max` over the two permutations of the batch means,
src/metrics/base_metric.py:53-60).  Here one kernel pass produces all six per-utterance values
and the batch-level decisions (`vatss_pit_sisnr`).  STOI is computed on the device by `vatss_stoi` (DESIGN.md §8):
all four pairings of the batch and the same batch-level PIT, where the reference runs pystoi on the host per pair.
"""
import ctypes
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
