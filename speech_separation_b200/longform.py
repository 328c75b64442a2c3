"""Separation of recordings of any length: overlapping windows, on-device speaker alignment, crossfade stitching.

No reference counterpart: the reference trains on fixed 2 s clips and separates one clip per forward.  A single
forward over a long recording needs a workspace that grows with its length and an inter-chunk pass that grows with
its square, and the models have only ever seen short inputs.  `LongFormSeparator` instead cuts each recording into
windows of `window` samples every `hop` samples, separates the windows as fixed-shape batches, orders the speakers of
every window like its predecessor's by the normalised correlation over their overlap (the models are trained with a
scale-invariant loss, so the gain may differ between windows) and crossfades the overlaps.  Cutting, alignment and
stitching are CUDA kernels of libvatss_b200.so (`vatss_window_cut`, `vatss_window_stitch`); nothing reads back to the
host on the way.  Geometry and rules: DESIGN.md §7.
"""
import torch
from torch import nn

from . import _lib
from .model import _DualPathEncDec


def micro_batches(total, max_batch):
    """Split `total` windows into near-equal consecutive micro-batches of at most `max_batch`: [(first, count), ...],
    larger ones first, so a call switches the model's cached workspace between at most two shapes once."""
    if max_batch < 1:
        raise ValueError(f"max_batch must be >= 1, got {max_batch}")
    nb = -(-total // max_batch)
    base, extra = divmod(total, nb)
    out, first = [], 0
    for b in range(nb):
        count = base + (b < extra)
        out.append((first, count))
        first += count
    return out


class LongFormSeparator(nn.Module):
    """Wraps a separator (`DPTNAVWavEncDec`, `DPTNWavEncDec`, `DPTNEncDec`, `DPRNNEncDec`) so that its forward takes
    recordings of any length: same call, same {"s1_pred", "s2_pred"} of shape (R, T), usable as the model of
    `Inferencer`.  `state_dict` / `load_state_dict` are the wrapped model's (reference checkpoint keys).

    window, hop: samples, window / 2 <= hop < window; the overlap window - hop is crossfaded.
    max_batch: most windows per forward (the model's workspace is sized for it).
    samples_per_video_frame: audio samples per embedding frame of the audio-visual model (16 kHz / 25 fps = 640);
    window and hop must be multiples of it there, and the embeddings must have Tv frames with |Tv spf - T| < spf.

    A recording no longer than one window goes through the wrapped model unchanged.  All recordings of one call have
    the same length.  Output speaker order follows the first window of each recording.
    """

    def __init__(self, model, window=64000, hop=48000, max_batch=32, samples_per_video_frame=640):
        super().__init__()
        if not isinstance(model, _DualPathEncDec):
            raise TypeError(f"LongFormSeparator wraps a speech_separation_b200 separator, got {type(model).__name__}")
        W, H, spf = int(window), int(hop), int(samples_per_video_frame)
        if not (2 * H >= W and H < W and H > 0):
            raise ValueError(f"hop {H} must satisfy window/2 <= hop < window (window={W})")
        if max_batch < 1:
            raise ValueError(f"max_batch must be >= 1, got {max_batch}")
        d = model._desc
        if W < d.K or (W - d.K) // (d.K // 2) + 1 < d.C:
            raise ValueError(f"a window of {W} samples is shorter than one chunk of the model "
                             f"({d.C} frames of kernel {d.K})")
        self.av = model.KIND == "dptn_av"
        if self.av and (spf < 1 or W % spf or H % spf):
            raise ValueError(f"window {W} and hop {H} must be multiples of samples_per_video_frame {spf}")
        self.model = model
        self.window, self.hop, self.max_batch, self.samples_per_video_frame = W, H, int(max_batch), spf

    # the wrapped model's parameters under its own (reference) key names
    def state_dict(self, *args, **kwargs):
        return self.model.state_dict(*args, **kwargs)

    def load_state_dict(self, state_dict, strict=True, assign=False):
        return self.model.load_state_dict(state_dict, strict=strict, assign=assign)

    def _inputs(self, mix, e1, e2):
        """Every argument error is raised before any device work."""
        _lib.require_cuda(mix, "mix")
        if mix.dim() != 2:
            raise ValueError(f"mix must be (recordings, time), got {tuple(mix.shape)}")
        R, T = mix.shape
        if not self.av:
            return _lib.f32c(mix, "mix"), None, None
        if e1 is None or e2 is None:
            raise ValueError("the audio-visual model needs s1_embedding and s2_embedding")
        _lib.require_cuda(e1, "s1_embedding")
        _lib.require_cuda(e2, "s2_embedding")
        E = self.model._desc.E
        if e1.shape != e2.shape or e1.dim() != 3 or tuple(e1.shape[:2]) != (R, E):
            raise ValueError(f"embeddings must both be ({R}, {E}, frames); got {tuple(e1.shape)} and "
                             f"{tuple(e2.shape)}")
        spf = self.samples_per_video_frame
        if abs(e1.shape[2] * spf - T) >= spf:
            raise ValueError(f"{e1.shape[2]} video frames do not match {T} samples at {spf} samples per frame")
        return _lib.f32c(mix, "mix"), _lib.f32c(e1, "s1_embedding"), _lib.f32c(e2, "s2_embedding")

    def forward(self, mix, s1_embedding=None, s2_embedding=None, return_alignment=False, **batch):
        """mix (R, T) -> {"s1_pred", "s2_pred"} (R, T).  return_alignment=True adds "swaps" (R, n-1) uint8, 1 where
        window j+1's speakers were swapped relative to window j, and "corr" (R, n-1, 8) float64, the overlap sums
        [a1.b1, a1.b2, a2.b1, a2.b2, a1.a1, a2.a2, b1.b1, b2.b2] the decision was taken on (both empty when T <= W)."""
        mix, e1, e2 = self._inputs(mix, s1_embedding, s2_embedding)
        R, T = mix.shape
        W, H = self.window, self.hop
        if T <= W:
            out = self.model(mix, e1, e2) if self.av else self.model(mix)
            if return_alignment:
                out["swaps"] = torch.empty(R, 0, dtype=torch.uint8, device=mix.device)
                out["corr"] = torch.empty(R, 0, 8, dtype=torch.float64, device=mix.device)
            return out
        lib = _lib.load()
        n = lib.vatss_longform_windows(T, W, H)
        _lib.check(min(n, 0), "vatss_longform_windows")
        dev = mix.device
        batches = micro_batches(R * n, self.max_batch)
        Bmax = batches[0][1]
        Tv = e1.shape[2] if self.av else 0
        E, spf = self.model._desc.E, self.samples_per_video_frame
        with torch.cuda.device(dev):
            y1 = torch.empty(R * n, W, dtype=torch.float32, device=dev)
            y2 = torch.empty_like(y1)
            xb = torch.empty(Bmax, W, dtype=torch.float32, device=dev)
            eb1 = eb2 = None
            if self.av:
                eb1 = torch.empty(Bmax, E, W // spf, dtype=torch.float32, device=dev)
                eb2 = torch.empty_like(eb1)
            for first, count in batches:
                _lib.check(lib.vatss_window_cut(mix.data_ptr(), e1.data_ptr() if self.av else None,
                                                e2.data_ptr() if self.av else None, R, T, Tv, E, W, H, spf, first,
                                                count, xb.data_ptr(), eb1.data_ptr() if self.av else None,
                                                eb2.data_ptr() if self.av else None, _lib.stream_ptr()),
                           "vatss_window_cut")
                self.model._run_into(xb[:count], eb1[:count] if self.av else None, eb2[:count] if self.av else None,
                                     y1[first:first + count], y2[first:first + count])
            s1 = torch.empty(R, T, dtype=torch.float32, device=dev)
            s2 = torch.empty_like(s1)
            swaps = corr = None
            if return_alignment:
                swaps = torch.empty(R, n - 1, dtype=torch.uint8, device=dev)
                corr = torch.empty(R, n - 1, 8, dtype=torch.float64, device=dev)
            nbytes = int(lib.vatss_window_stitch_scratch_bytes(R, n))
            scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            _lib.check(lib.vatss_window_stitch(y1.data_ptr(), y2.data_ptr(), R, T, W, H, s1.data_ptr(), s2.data_ptr(),
                                               swaps.data_ptr() if swaps is not None else None,
                                               corr.data_ptr() if corr is not None else None,
                                               scratch.data_ptr(), nbytes, _lib.stream_ptr()), "vatss_window_stitch")
        out = {"s1_pred": s1, "s2_pred": s2}
        if return_alignment:
            out["swaps"], out["corr"] = swaps, corr
        return out
