"""Drop-in nn.Modules for the reference's dual-path separators, executed by libvatss_b200.so.

Host-side mirror of the reference interface (same class names, constructor arguments,
`forward` signatures, return dicts and `state_dict` keys):

    DPTNAVWavEncDec   <- src/model/dptn_wav.py:129-207
    DPTNWavEncDec     <- src/model/dptn_wav.py:64-126
    DPTNEncDec        <- src/model/dptn.py:146-208
    DPRNNEncDec       <- src/model/dprnn.py:230-289
    SplitToFolds      <- src/model/dprnn.py:116-136
    OverlapAdd        <- src/model/dprnn.py:139-163

The torch.nn sub-modules created here are parameter containers only: they give the
state_dict its reference key names/shapes (so reference checkpoints load with
`load_state_dict`) and, because they are created in the reference's order, reproduce the
reference's default initialisation under the same `torch.manual_seed`.  None of their
`forward`s is ever called: the whole forward pass is one call into the C ABI
(`vatss_forward`, include/vatss.h).  There is no CPU path and no autograd: the backward pass
is out of scope (SURVEY.md §8f), tensors come back detached.  Attention dropout (active only
in the reference's train() mode) is not applied.
"""
import ctypes
import warnings

import torch
from torch import nn

from . import _lib


# --------------------------------------------------------------------------------------
# parameter containers (state_dict layout of the reference)
# --------------------------------------------------------------------------------------
class _TransformerParams(nn.Module):
    """Parameters of TransformerDPRNN (src/model/dptn.py:14-34)."""

    def __init__(self, num_features, hidden_dim, num_heads, dropout, bidir=True):
        super().__init__()
        self.mha = nn.MultiheadAttention(embed_dim=num_features, num_heads=num_heads, dropout=dropout,
                                         batch_first=True)
        self.ln1 = nn.LayerNorm(num_features)
        self.rnn = nn.LSTM(input_size=num_features, hidden_size=hidden_dim, bidirectional=bidir, batch_first=True)
        self.ffn = nn.Sequential(nn.ReLU(), nn.Linear(hidden_dim * (bidir + 1), num_features))
        self.ln2 = nn.LayerNorm(num_features)


class _ChunkRNNParams(nn.Module):
    """Parameters of IntraChunkRNN / InterChunkRNN (src/model/dprnn.py:12-22,55-63)."""

    def __init__(self, num_features, hidden_dim, bidir=True):
        super().__init__()
        self.rnn = nn.LSTM(input_size=num_features, hidden_size=hidden_dim, batch_first=True, bidirectional=bidir)
        self.fc = nn.Linear(hidden_dim * (bidir + 1), num_features)
        self.norm1d = nn.LayerNorm(num_features)


class _BlockParams(nn.Module):
    def __init__(self, intra, inter):
        super().__init__()
        self.intra_chunk_block = intra
        self.inter_chunk_block = inter


class _SeparatorParams(nn.Module):
    """The sub-module the reference calls `dprnn` (DPTNWav / DPTN / DPRNN)."""

    def __init__(self, kind, num_features, hidden_dim, num_blocks, num_heads, dropout, bidir):
        super().__init__()
        self.model = nn.Sequential()
        for _ in range(num_blocks):
            if kind == "dprnn":
                blk = _BlockParams(_ChunkRNNParams(num_features, hidden_dim, True),
                                   _ChunkRNNParams(num_features, hidden_dim, bidir))
            else:
                blk = _BlockParams(_TransformerParams(num_features, hidden_dim, num_heads, dropout, True),
                                   _TransformerParams(num_features, hidden_dim, num_heads, dropout, bidir))
            self.model.append(blk)
        self.speakers_separation = nn.Sequential(nn.PReLU(), nn.Conv2d(num_features, 2 * num_features, 1))
        if kind == "dptn_mask":
            self.output_gate = nn.Sequential(nn.Conv1d(num_features, num_features, 1), nn.Sigmoid())
            self.output = nn.Sequential(nn.Conv1d(num_features, num_features, 1), nn.Tanh())
            self.postprocessing = nn.Sequential(nn.ReLU())
        else:
            self.postprocessing = nn.Sequential(nn.Conv1d(num_features, num_features, 1))


# --------------------------------------------------------------------------------------
# the executable module
# --------------------------------------------------------------------------------------
class _DualPathEncDec(nn.Module):
    KIND = None

    def _build(self, num_features, kernel_size_enc, hidden_dim, num_blocks, chunk_size, step_size, num_heads,
               dropout, bidir, video_emb_size=0, hidden_video=0):
        kind = self.KIND
        self.encoder = nn.Conv1d(1, num_features, kernel_size=kernel_size_enc, stride=kernel_size_enc // 2,
                                 bias=False)
        if kind == "dptn_av":
            if hidden_video != num_features:
                raise ValueError("hidden_video must equal num_features (the fusion adds them element-wise)")
            self.visual_compression = nn.Linear(video_emb_size, hidden_video // 2)
            self.gate = nn.Parameter(torch.randn([1]), requires_grad=True)
            self.video_ln = nn.LayerNorm(hidden_video)
        self.dprnn = _SeparatorParams(kind, num_features, hidden_dim, num_blocks, num_heads, dropout, bidir)
        self.decoder = nn.ConvTranspose1d(num_features, 1, kernel_size=kernel_size_enc,
                                          stride=kernel_size_enc // 2, bias=False)
        self._desc = _lib.ModelDesc(kind=_lib.KIND[kind], N=num_features, K=kernel_size_enc, H=hidden_dim,
                                    num_blocks=num_blocks, C=chunk_size, P=step_size, heads=num_heads,
                                    bidir=int(bool(bidir)), E=video_emb_size, engine=_lib.ENGINE["auto"],
                                    reserved=0)
        self._bidir = bool(bidir)
        self._cache_key = None
        self._ptr_table = None
        self._packed = None
        self._workspaces = {}
        self._keepalive = None

    # -- engine selection (shape specialisation inside the same CUDA library) ---------------
    def set_engine(self, name):
        """'auto' (default), 'generic' (fp32 SIMT kernels) or 'tensor' (tcgen05 kernels)."""
        self._desc.engine = _lib.ENGINE[name]
        self._cache_key = None
        self._workspaces = {}
        return self

    # -- parameter table ---------------------------------------------------------------------
    def _param_names(self):
        kind = self.KIND
        names = []
        for g in _lib.P_GLOBAL:
            if g == "HEAD_W":
                g = "dprnn.output.0.weight" if kind == "dptn_mask" else "dprnn.postprocessing.0.weight"
            elif g == "HEAD_B":
                g = "dprnn.output.0.bias" if kind == "dptn_mask" else "dprnn.postprocessing.0.bias"
            names.append(g)
        sub = _lib.S_DPRNN if kind == "dprnn" else _lib.S_DPTN
        for b in range(self._desc.num_blocks):
            for path in ("intra_chunk_block", "inter_chunk_block"):
                for s in sub:
                    names.append(None if s is None else f"dprnn.model.{b}.{path}.{s}")
        return names

    def _prepare(self, device):
        lib = _lib.load()
        named = dict(self.named_parameters())
        key = tuple((p.data_ptr(), p._version) for p in named.values()) + (str(device), self._desc.engine)
        if key == self._cache_key:
            return lib
        names = self._param_names()
        table = (ctypes.c_void_p * len(names))()
        keep = []
        for i, n in enumerate(names):
            p = named.get(n) if n is not None else None
            if p is None:
                table[i] = None
                continue
            if not p.is_cuda or p.device != device:
                raise RuntimeError(f"parameter {n} is on {p.device}, input on {device}: move the module with "
                                   ".to(device); speech_separation_b200 has no CPU path")
            t = p.detach()
            if t.dtype != torch.float32 or not t.is_contiguous():
                t = t.float().contiguous()
            keep.append(t)
            table[i] = t.data_ptr()
        why = lib.vatss_engine_fallback_reason(ctypes.byref(self._desc))
        if why is not None and not getattr(self, "_warned_fallback", False):
            self._warned_fallback = True
            warnings.warn(f"{type(self).__name__}: the tcgen05 tensor engine does not cover this model ({why.decode()}); "
                          "running on the fp32 SIMT engine, which is roughly 20x slower", RuntimeWarning, stacklevel=3)
        nbytes = lib.vatss_packed_weight_bytes(ctypes.byref(self._desc))
        packed = torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)
        _lib.check(lib.vatss_pack_weights(ctypes.byref(self._desc), table, len(names), packed.data_ptr(),
                                          packed.numel(), _lib.stream_ptr()), "vatss_pack_weights")
        self._ptr_table, self._packed, self._keepalive, self._cache_key = table, packed, keep, key
        return lib

    def _workspace(self, lib, B, T, Tv, device):
        k = (B, T, Tv, str(device))
        ws = self._workspaces.get(k)
        if ws is None:
            nbytes = int(lib.vatss_workspace_bytes(ctypes.byref(self._desc), B, T, Tv))
            if nbytes == 0:
                _lib.check(-1, "vatss_workspace_bytes")
            self._workspaces.clear()  # one live workspace per module
            ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
            self._workspaces[k] = ws
        return ws

    def _run(self, mix, e1, e2):
        mix = _lib.f32c(mix, "mix")
        return self._run_into(mix, e1, e2, torch.empty_like(mix), torch.empty_like(mix))

    def _run_into(self, mix, e1, e2, s1, s2):
        """The forward with caller-provided outputs: s1, s2 contiguous float32 (B, T) on mix's device."""
        mix = _lib.f32c(mix, "mix")
        if mix.dim() != 2:
            raise ValueError(f"mix must be (batch, time), got {tuple(mix.shape)}")
        for t, name in ((s1, "s1"), (s2, "s2")):
            if t.shape != mix.shape or t.dtype != torch.float32 or not t.is_contiguous() or t.device != mix.device:
                raise ValueError(f"{name} output must be contiguous float32 {tuple(mix.shape)} on {mix.device}")
        B, T = mix.shape
        Tv = 0
        if self.KIND == "dptn_av":
            e1 = _lib.f32c(e1, "s1_embedding")
            e2 = _lib.f32c(e2, "s2_embedding")
            if e1.shape != e2.shape or e1.dim() != 3 or e1.shape[0] != B or e1.shape[1] != self._desc.E:
                raise ValueError(f"embeddings must both be (batch, {self._desc.E}, frames); got "
                                 f"{tuple(e1.shape)} and {tuple(e2.shape)}")
            Tv = e1.shape[2]
        with torch.cuda.device(mix.device):
            lib = self._prepare(mix.device)
            ws = self._workspace(lib, B, T, Tv, mix.device)
            rc = lib.vatss_forward(ctypes.byref(self._desc), self._ptr_table, len(self._ptr_table),
                                   self._packed.data_ptr(), mix.data_ptr(),
                                   e1.data_ptr() if e1 is not None else None,
                                   e2.data_ptr() if e2 is not None else None, B, T, Tv, s1.data_ptr(),
                                   s2.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr())
            _lib.check(rc, "vatss_forward")
        return {"s1_pred": s1, "s2_pred": s2}

    def __str__(self):
        all_parameters = sum(p.numel() for p in self.parameters())
        trainable = sum(p.numel() for p in self.parameters() if p.requires_grad)
        return f"{super().__str__()}\nAll parameters: {all_parameters}\nTrainable parameters: {trainable}"


class DPTNAVWavEncDec(_DualPathEncDec):
    KIND = "dptn_av"

    def __init__(self, num_features=64, video_emb_size=1024, hidden_video=128, kernel_size_enc=2, hidden_dim=32,
                 num_blocks=6, chunk_size=10, step_size=5, num_heads=4, dropout=0.1, bidir=True):
        super().__init__()
        self._build(num_features, kernel_size_enc, hidden_dim, num_blocks, chunk_size, step_size, num_heads,
                    dropout, bidir, video_emb_size, hidden_video)

    def forward(self, mix, s1_embedding, s2_embedding, **batch):
        return self._run(mix, s1_embedding, s2_embedding)


class DPTNWavEncDec(_DualPathEncDec):
    KIND = "dptn_wav"

    def __init__(self, num_features=64, kernel_size_enc=2, hidden_dim=32, num_blocks=6, chunk_size=10,
                 step_size=5, num_heads=4, dropout=0.1, bidir=True):
        super().__init__()
        self._build(num_features, kernel_size_enc, hidden_dim, num_blocks, chunk_size, step_size, num_heads,
                    dropout, bidir)

    def forward(self, mix, **batch):
        return self._run(mix, None, None)


class DPTNEncDec(_DualPathEncDec):
    KIND = "dptn_mask"

    def __init__(self, num_features=64, kernel_size_enc=2, hidden_dim=32, num_blocks=6, chunk_size=10,
                 step_size=5, num_heads=4, dropout=0.1, bidir=True):
        super().__init__()
        self._build(num_features, kernel_size_enc, hidden_dim, num_blocks, chunk_size, step_size, num_heads,
                    dropout, bidir)

    def forward(self, mix, **batch):
        return self._run(mix, None, None)


class DPRNNEncDec(_DualPathEncDec):
    KIND = "dprnn"

    def __init__(self, num_features=64, kernel_size_enc=2, hidden_dim=32, num_blocks=6, chunk_size=10,
                 step_size=5, bidir=True):
        super().__init__()
        self._build(num_features, kernel_size_enc, hidden_dim, num_blocks, chunk_size, step_size, 1, 0.0, bidir)

    def forward(self, mix, **batch):
        return self._run(mix, None, None)


# --------------------------------------------------------------------------------------
# stand-alone segmentation primitives (reference layout, bit-exact)
# --------------------------------------------------------------------------------------
class SplitToFolds(nn.Module):
    """(B,N,ts) -> (B,N,S,chunk) with S=(ts-chunk)//step+1; exact copy, no padding."""

    def __init__(self, chunk_size, step_size):
        super().__init__()
        self.chunk_size, self.step_size = chunk_size, step_size

    def forward(self, data):
        x = _lib.f32c(data, "data")
        B, N, L = x.shape
        C, P = self.chunk_size, self.step_size
        if L < C:
            raise RuntimeError(f"SplitToFolds: length {L} shorter than one chunk ({C})")
        S = (L - C) // P + 1
        out = torch.empty((B, N, S, C), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().vatss_segment(x.data_ptr(), B, N, L, C, P, out.data_ptr(), _lib.stream_ptr()),
                       "vatss_segment")
        return out


class OverlapAdd(nn.Module):
    """(B,N,S,chunk) -> (B,N,(S-1)*step+chunk); plain sum of overlapping entries."""

    def __init__(self, chunk_size, step_size):
        super().__init__()
        self.chunk_size, self.step_size = chunk_size, step_size

    def forward(self, data):
        y = _lib.f32c(data, "data")
        B, N, S, C = y.shape
        P = self.step_size
        out = torch.empty((B, N, (S - 1) * P + C), dtype=torch.float32, device=y.device)
        with torch.cuda.device(y.device):
            _lib.check(_lib.load().vatss_overlap_add(y.data_ptr(), B, N, S, C, P, out.data_ptr(),
                                                     _lib.stream_ptr()), "vatss_overlap_add")
        return out
