"""PIT SI-SNR loss, drop-in for src/loss/ss_losses.py (SiSNRLoss :96-114, SiSNRWavLoss :117-130).

Semantics kept from the reference: zero-mean SI-SNR without eps, value = -20*log10(power ratio)
(= -2 x SI-SNR dB), mean over the batch, and ONE permutation chosen for the whole batch
(BaseSSLoss.forward :10-26).  All of it is evaluated by `vatss_pit_sisnr` on the device in a single
pass over the waveforms; the returned 0-d tensor stays on the device, so unlike the reference's
Python `if loss_perm_2 < loss_perm_1` there is no host synchronisation.

The loss is differentiable with respect to the predictions: when `s1_pred` / `s2_pred` require grad, `SiSNRWavLoss`
returns a tensor whose `.backward()` (src/trainer/trainer.py:46) runs `vatss_pit_sisnr_backward` - one more pass over the
four waveforms, reusing the forward's moments and its batch-level permutation.  (The separation models themselves are
forward-only; this is the first piece of SURVEY.md §8f rank 2.)  `SiSNRLoss` is differentiable the same way.

The moments are raw fp64 sums, centred algebraically, so for a near-exact estimate the residual power pp - dot^2/gg can
round to zero or below.  The forward then reports -inf for that pair (the loss has no finite minimum there) and the
backward returns a zero gradient for that prediction: -inf offers no descent direction.  A silent target gives NaN in
both.
"""
import math

import torch
from torch import nn

from . import _lib


MAX_B = 65535   # utterances per call: the kernels put the batch in grid.y


def _batch_dims(shape):
    """(B, T) of a (..., T) batch; raises ValueError for an empty or too large batch, before any device work."""
    T = shape[-1] if len(shape) else 0
    B = math.prod(shape[:-1]) if T > 0 else 0
    if B == 0 or T == 0:
        raise ValueError("empty batch")
    if B > MAX_B:
        raise ValueError(f"batch of {B} utterances: at most {MAX_B}")
    return B, T


def pit_sisnr_all(s1_pred, s2_pred, s1, s2, mix=None):
    """Runs the fused kernel.  Returns (rows (B,6) f64, rows_loss (B,4) f64, summary (8,) f64) on device.

    rows: per-utterance SI-SNR dB of [s1p.s1, s2p.s2, s1p.s2, s2p.s1, mix.s1, mix.s2];
    rows_loss: per-utterance reference-loss values of the first four pairs;
    summary: [loss, loss_perm1, loss_perm2, SI-SNR(PIT), SI-SNRi, mean SI-SNR(mix,s1), mean SI-SNR(mix,s2), B].
    """
    shape = s1_pred.shape
    for name, t in (("s2_pred", s2_pred), ("s1", s1), ("s2", s2), ("mix", mix)):
        if t is not None and t.shape != shape:
            raise ValueError(f"{name} has shape {tuple(t.shape)}, expected {tuple(shape)}")
    B, T = _batch_dims(shape)
    s1_pred = _lib.f32c(s1_pred, "s1_pred")
    s2_pred = _lib.f32c(s2_pred, "s2_pred")
    s1 = _lib.f32c(s1, "s1")
    s2 = _lib.f32c(s2, "s2")
    if mix is not None:
        mix = _lib.f32c(mix, "mix")
    lib = _lib.load()
    dev = s1_pred.device
    chunks = lib.vatss_sisnr_chunks(T)
    rows = torch.empty((B, 6), dtype=torch.float64, device=dev)
    rows_loss = torch.empty((B, 4), dtype=torch.float64, device=dev)
    summary = torch.empty(8, dtype=torch.float64, device=dev)
    scratch = torch.empty(B * chunks * 16, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.vatss_pit_sisnr(s1_pred.data_ptr(), s2_pred.data_ptr(), s1.data_ptr(), s2.data_ptr(),
                                       mix.data_ptr() if mix is not None else None, B, T, rows.data_ptr(),
                                       rows_loss.data_ptr(), summary.data_ptr(), scratch.data_ptr(),
                                       _lib.stream_ptr()), "vatss_pit_sisnr")
    return rows, rows_loss, summary


class _PitSisnrLoss(torch.autograd.Function):
    """summary[0] of `vatss_pit_sisnr` with the analytic gradient of `vatss_pit_sisnr_backward`."""

    @staticmethod
    def forward(ctx, s1_pred, s2_pred, s1, s2):
        B, T = _batch_dims(s1_pred.shape)
        s1_pred, s2_pred, s1, s2 = (_lib.f32c(t.detach(), n) for t, n in
                                    ((s1_pred, "s1_pred"), (s2_pred, "s2_pred"), (s1, "s1"), (s2, "s2")))
        lib = _lib.load()
        dev = s1_pred.device
        chunks = lib.vatss_sisnr_chunks(T)
        rows = torch.empty((B, 6), dtype=torch.float64, device=dev)
        rows_loss = torch.empty((B, 4), dtype=torch.float64, device=dev)
        summary = torch.empty(8, dtype=torch.float64, device=dev)
        scratch = torch.empty(B * chunks * 16, dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.vatss_pit_sisnr(s1_pred.data_ptr(), s2_pred.data_ptr(), s1.data_ptr(), s2.data_ptr(), None, B,
                                           T, rows.data_ptr(), rows_loss.data_ptr(), summary.data_ptr(),
                                           scratch.data_ptr(), _lib.stream_ptr()), "vatss_pit_sisnr")
        ctx.save_for_backward(s1_pred, s2_pred, s1, s2, scratch, summary)
        ctx.dims = (B, T)
        return summary[0].float()

    @staticmethod
    def backward(ctx, grad_out):
        s1_pred, s2_pred, s1, s2, scratch, summary = ctx.saved_tensors
        B, T = ctx.dims
        g1, g2 = torch.empty_like(s1_pred), torch.empty_like(s2_pred)
        go = grad_out.detach().float().contiguous()
        with torch.cuda.device(s1_pred.device):
            _lib.check(_lib.load().vatss_pit_sisnr_backward(s1_pred.data_ptr(), s2_pred.data_ptr(), s1.data_ptr(),
                                                            s2.data_ptr(), B, T, scratch.data_ptr(), summary.data_ptr(),
                                                            go.data_ptr(), g1.data_ptr(), g2.data_ptr(),
                                                            _lib.stream_ptr()), "vatss_pit_sisnr_backward")
        return g1, g2, None, None


class SiSNRLoss(nn.Module):
    """Single-pair loss: mean_b[-20 log10(||a g||^2 / ||p - a g||^2)] (ss_losses.py:100-114).

    Differentiable with respect to `pred`: the pair is passed as both PIT pairs, whose moments are then bitwise equal, so
    the kernel keeps permutation 1 and the value is the single-pair mean; the two 1/(2B) gradient halves add up to 1/B."""

    def forward(self, pred, gt, **batch):
        if torch.is_grad_enabled() and pred.requires_grad:
            if gt.shape != pred.shape:
                raise ValueError(f"gt has shape {tuple(gt.shape)}, expected {tuple(pred.shape)}")
            return _PitSisnrLoss.apply(pred, pred, gt, gt)
        _, rows_loss, _ = pit_sisnr_all(pred, pred, gt, gt)
        return rows_loss[:, 0].mean().float()


class SiSNRWavLoss(nn.Module):
    """forward(s1_pred, s2_pred, s1, s2, **batch) -> {"loss": 0-d tensor} (ss_losses.py:122-130)."""

    def forward(self, s1_pred, s2_pred, s1, s2, **batch):
        if torch.is_grad_enabled() and (s1_pred.requires_grad or s2_pred.requires_grad):
            for name, t in (("s2_pred", s2_pred), ("s1", s1), ("s2", s2)):
                if t.shape != s1_pred.shape:
                    raise ValueError(f"{name} has shape {tuple(t.shape)}, expected {tuple(s1_pred.shape)}")
            return {"loss": _PitSisnrLoss.apply(s1_pred, s2_pred, s1, s2)}
        _, _, summary = pit_sisnr_all(s1_pred, s2_pred, s1, s2)
        return {"loss": summary[0].float()}
