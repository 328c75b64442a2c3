"""CPU oracle for the VAT-SS dual-path separation hot path (TEST INFRASTRUCTURE ONLY).

This file is a numpy restatement of the algorithm the reference implements with stock
torch.nn ops.  It exists to CHECK the CUDA path; it is never imported by the product
package (`speech_separation_b200/`).  Only `tests/`, `__graft_entry__.smoke()` and
`bench.py`'s cpu_baseline / `--impl reference` legs may import it.

Parity pinning: the reference ships no tests or golden vectors (SURVEY.md §4).  This
oracle is pinned against outputs of the reference's own modules, imported unmodified
from /root/reference with `oracle/ref_import.py` and run on CPU by
`oracle/gen_golden.py`; the resulting fixtures are committed under `tests/golden/` and
`tests/test_oracle_golden.py` re-checks the oracle against them on every run.
The one boundary that stays "parity unpinned" is the torchmetrics SI-SNR used by
`src/metrics/si_snr.py` / `si_snri.py`: torchmetrics is not installed here and not
vendored by the reference, so `si_snr_metric_rows` restates its published algorithm
(zero_mean=True SI-SDR with eps) and is cross-checked against the reference's own
`SiSNRLoss` (= -2 x SI-SNR dB), which IS importable.

Every function cites the reference lines it follows (paths relative to /root/reference).
All arithmetic is done in the dtype of `P` (float64 by default) so the oracle doubles as
the error yardstick for the fp32 reference itself.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np

LN_EPS = 1e-5  # torch.nn.LayerNorm default (src/model/dptn.py:22,34)


# --------------------------------------------------------------------------------------
# configuration
# --------------------------------------------------------------------------------------
@dataclass(frozen=True)
class PathConfig:
    """Hyper-parameters of one dual-path model (src/configs/model/*.yaml)."""

    kind: str  # "dptn_av" | "dptn_wav" | "dptn_mask" | "dprnn"
    num_features: int = 128
    kernel_size_enc: int = 7
    hidden_dim: int = 128
    num_blocks: int = 6
    chunk_size: int = 150
    step_size: int = 75
    num_heads: int = 4
    bidir: bool = True
    video_emb_size: int = 512

    @property
    def stride(self) -> int:
        return self.kernel_size_enc // 2

    def frames(self, T: int) -> int:
        """L of nn.Conv1d(1,N,K,stride=K//2) (src/model/dptn_wav.py:153)."""
        return (T - self.kernel_size_enc) // self.stride + 1

    def chunks(self, L: int) -> int:
        """S of F.unfold without padding (src/model/dprnn.py:131-135)."""
        return (L - self.chunk_size) // self.step_size + 1


def to_numpy_state(state_dict, dtype=np.float64):
    """torch state_dict (or dict of arrays) -> dict of numpy arrays of `dtype`."""
    out = {}
    for k, v in state_dict.items():
        if hasattr(v, "detach"):
            v = v.detach().cpu().numpy()
        out[k] = np.asarray(v, dtype=dtype)
    return out


# --------------------------------------------------------------------------------------
# primitives
# --------------------------------------------------------------------------------------
def layer_norm(x, w, b):
    """nn.LayerNorm over the last axis, biased variance, eps=1e-5 (dptn.py:22,34,47,51)."""
    mu = x.mean(axis=-1, keepdims=True)
    var = ((x - mu) ** 2).mean(axis=-1, keepdims=True)
    return (x - mu) / np.sqrt(var + LN_EPS) * w + b


def sigmoid(x):
    return 1.0 / (1.0 + np.exp(-x))


def encode(mix, w_enc, stride):
    """E1: nn.Conv1d(1,N,K,stride,bias=False) (dptn_wav.py:153,180).

    mix (B,T), w_enc (N,1,K) -> token-major (B,L,N): enc[b,l,n] = sum_k W[n,0,k] mix[b, st*l+k].
    """
    B, T = mix.shape
    N, _, K = w_enc.shape
    L = (T - K) // stride + 1
    idx = stride * np.arange(L)[:, None] + np.arange(K)[None, :]  # (L,K)
    frames = mix[:, idx]  # (B,L,K)
    return frames @ w_enc[:, 0, :].T  # (B,L,N)


def interp_linear_index(L, Tv, dtype=np.float64):
    """F.interpolate(mode='linear', align_corners=False) source indices (dptn_wav.py:181-183).

    ATen upsample_linear1d: scale = Tv/L, src = max(0, scale*(l+0.5)-0.5), i0=floor(src),
    i1 = min(i0+1, Tv-1), lam = src - i0.
    The arithmetic of src is done in `dtype` so that a float32 oracle reproduces ATen's
    float32 index maths exactly.
    """
    dt = np.dtype(dtype).type
    scale = dt(Tv) / dt(L)
    l = np.arange(L).astype(dtype)
    src = scale * (l + dt(0.5)) - dt(0.5)
    src = np.maximum(src, dt(0.0))
    i0 = np.floor(src).astype(np.int64)
    i0 = np.minimum(i0, Tv - 1)
    i1 = np.minimum(i0 + 1, Tv - 1)
    lam = src - i0.astype(dtype)
    return i0, i1, lam


def av_fuse(enc, emb1, emb2, P, index=None):
    """F1: tanh-gated lip-embedding fusion (dptn_wav.py:173-184).

    enc (B,L,N) token-major; emb* (B,E,Tv).  compress -> concat -> interpolate -> LN -> gate.
    index: the interpolation's (i0, i1, lam), default interp_linear_index(L, Tv, enc.dtype); tests pass the float32
    source indices of a float32 implementation to compare everything else in enc.dtype.
    """
    Wv, bv = P["visual_compression.weight"], P["visual_compression.bias"]
    v1 = np.einsum("bet,je->btj", emb1, Wv) + bv
    v2 = np.einsum("bet,je->btj", emb2, Wv) + bv
    v = np.concatenate([v1, v2], axis=-1)  # (B,Tv,N)
    L = enc.shape[1]
    Tv = v.shape[1]
    i0, i1, lam = interp_linear_index(L, Tv, dtype=enc.dtype) if index is None else index
    vi = (1.0 - lam)[None, :, None] * v[:, i0, :] + lam[None, :, None] * v[:, i1, :]
    g = np.tanh(P["gate"][0])
    return enc + g * layer_norm(vi, P["video_ln.weight"], P["video_ln.bias"])


def segment_channel_major(x, C, Pstep):
    """S1 in the reference's own layout: SplitToFolds.forward (dprnn.py:122-136).

    x (B,N,L) -> (B,N,S,C) with seg[b,n,s,k] = x[b,n,P*s+k]; no padding, tail dropped.
    """
    B, N, L = x.shape
    S = (L - C) // Pstep + 1
    idx = Pstep * np.arange(S)[:, None] + np.arange(C)[None, :]
    return np.ascontiguousarray(x[:, :, idx])


def overlap_add_channel_major(y, Pstep):
    """S3 in the reference's own layout: OverlapAdd.forward (dprnn.py:145-163).

    y (B,N,S,C) -> (B,N,(S-1)P+C), plain sum of overlapping entries (no normalisation).
    Chunks are accumulated in increasing s, matching col2im's loop order; with <=2 addends
    per output the order cannot change the float result.
    """
    B, N, S, C = y.shape
    out = np.zeros((B, N, (S - 1) * Pstep + C), dtype=y.dtype)
    for s in range(S):
        out[:, :, Pstep * s : Pstep * s + C] += y[:, :, s, :]
    return out


def centre_pad_last(x, target):
    """The 'dirty hack' centred zero pad (dptn_wav.py:51-55 and :189-192)."""
    d = target - x.shape[-1]
    left = d // 2
    right = d - left
    pad = [(0, 0)] * (x.ndim - 1) + [(left, right)]
    return np.pad(x, pad)


def mha_self(z, P, pre, heads):
    """nn.MultiheadAttention(batch_first=True) self-attention, eval mode (dptn.py:16-21,46).

    z (G,len,N).  Packed in_proj rows [0,N)=Q, [N,2N)=K, [2N,3N)=V; head h owns features
    [h*hd,(h+1)*hd); softmax(QK^T/sqrt(hd)) V; concat; out_proj.
    """
    G, Ls, N = z.shape
    hd = N // heads
    qkv = z @ P[pre + "mha.in_proj_weight"].T + P[pre + "mha.in_proj_bias"]
    q, k, v = qkv[..., :N], qkv[..., N : 2 * N], qkv[..., 2 * N :]
    q = q.reshape(G, Ls, heads, hd).transpose(0, 2, 1, 3)
    k = k.reshape(G, Ls, heads, hd).transpose(0, 2, 1, 3)
    v = v.reshape(G, Ls, heads, hd).transpose(0, 2, 1, 3)
    o = np.empty_like(q)
    step = max(1, (1 << 24) // (heads * Ls * Ls))  # sequences per pass: score matrices of <= 128 MB in fp64
    for g0 in range(0, G, step):
        sl = slice(g0, g0 + step)
        s = (q[sl] @ k[sl].transpose(0, 1, 3, 2)) / math.sqrt(hd)
        s = s - s.max(axis=-1, keepdims=True)
        p = np.exp(s)
        p = p / p.sum(axis=-1, keepdims=True)
        o[sl] = p @ v[sl]
    o = o.transpose(0, 2, 1, 3).reshape(G, Ls, N)
    return o @ P[pre + "mha.out_proj.weight"].T + P[pre + "mha.out_proj.bias"]


def lstm_direction(x, Wih, Whh, bih, bhh, reverse):
    """One direction of nn.LSTM(batch_first=True), h0=c0=0 (dptn.py:23-29,49; dprnn.py:18,60).

    Gate order i,f,g,o along 4H.  x (G,len,N) -> (G,len,H).
    """
    G, Ls, _ = x.shape
    H = Whh.shape[1]
    pre = x @ Wih.T + (bih + bhh)
    h = np.zeros((G, H), dtype=x.dtype)
    c = np.zeros((G, H), dtype=x.dtype)
    out = np.empty((G, Ls, H), dtype=x.dtype)
    order = range(Ls - 1, -1, -1) if reverse else range(Ls)
    WhhT = Whh.T
    for t in order:
        g = pre[:, t, :] + h @ WhhT
        i_g = sigmoid(g[:, :H])
        f_g = sigmoid(g[:, H : 2 * H])
        g_g = np.tanh(g[:, 2 * H : 3 * H])
        o_g = sigmoid(g[:, 3 * H :])
        c = f_g * c + i_g * g_g
        h = o_g * np.tanh(c)
        out[:, t, :] = h
    return out


def lstm(x, P, pre, bidir):
    f = lstm_direction(
        x, P[pre + "rnn.weight_ih_l0"], P[pre + "rnn.weight_hh_l0"],
        P[pre + "rnn.bias_ih_l0"], P[pre + "rnn.bias_hh_l0"], reverse=False,
    )
    if not bidir:
        return f
    r = lstm_direction(
        x, P[pre + "rnn.weight_ih_l0_reverse"], P[pre + "rnn.weight_hh_l0_reverse"],
        P[pre + "rnn.bias_ih_l0_reverse"], P[pre + "rnn.bias_hh_l0_reverse"], reverse=True,
    )
    return np.concatenate([f, r], axis=-1)


def improved_transformer(z, P, pre, heads, bidir, taps=None):
    """B2: TransformerDPRNN.forward (dptn.py:36-52).

    x1 = LN1(MHA(z)+z); out = LN2(Linear(ReLU(LSTM(x1))) + x1).
    """
    a = mha_self(z, P, pre, heads)
    x1 = layer_norm(a + z, P[pre + "ln1.weight"], P[pre + "ln1.bias"])
    r = lstm(x1, P, pre, bidir)
    y = np.maximum(r, 0.0) @ P[pre + "ffn.1.weight"].T + P[pre + "ffn.1.bias"]
    out = layer_norm(y + x1, P[pre + "ln2.weight"], P[pre + "ln2.bias"])
    if taps is not None:
        taps[pre + "attn"] = a
        taps[pre + "x1"] = x1
        taps[pre + "rnn"] = r
        taps[pre + "out"] = out
    return out


def dprnn_subblock(z, P, pre, bidir):
    """R1: IntraChunkRNN / InterChunkRNN core (dprnn.py:37-45,78-87): LN(Linear(LSTM(z))) + z."""
    r = lstm(z, P, pre, bidir)
    y = r @ P[pre + "fc.weight"].T + P[pre + "fc.bias"]
    return layer_norm(y, P[pre + "norm1d.weight"], P[pre + "norm1d.bias"]) + z


def dual_path_blocks(x, P, cfg: PathConfig, taps=None):
    """B1: the stack of DPTNBlock / DPRNNBlock (dptn.py:62-79, dprnn.py:103-113).

    x token-major (B,S,C,N).  intra sequences = (b,s) over k; inter sequences = (b,k) over s.
    The intra path is always bidirectional (dptn.py:59, dprnn.py:18); inter follows cfg.bidir.
    """
    B, S, C, N = x.shape
    for blk in range(cfg.num_blocks):
        pi = f"dprnn.model.{blk}.intra_chunk_block."
        pe = f"dprnn.model.{blk}.inter_chunk_block."
        z = x.reshape(B * S, C, N)
        if cfg.kind == "dprnn":
            z = dprnn_subblock(z, P, pi, True)
        else:
            z = improved_transformer(z, P, pi, cfg.num_heads, True, taps)
        x = z.reshape(B, S, C, N)
        z = x.transpose(0, 2, 1, 3).reshape(B * C, S, N)
        if cfg.kind == "dprnn":
            z = dprnn_subblock(z, P, pe, cfg.bidir)
        else:
            z = improved_transformer(z, P, pe, cfg.num_heads, cfg.bidir, taps)
        x = z.reshape(B, C, S, N).transpose(0, 2, 1, 3)
        if taps is not None:
            taps[f"block{blk}"] = x.copy()
    return x


def separator_tail(x, enc, P, cfg: PathConfig, taps=None, round_ola=None):
    """T1+S3: PReLU -> 1x1 Conv2d(N->2N) -> overlap-add -> centred pad -> speaker split -> head.

    dptn_wav.py:47-59 (dptn.py:129-141 for the masking variant, dprnn.py:213-225).
    x (B,S,C,N) token-major, enc (B,L,N).  Returns the two decoder inputs u_j (B,L,N).
    round_ola: optional map applied to the overlap-added tensor (tests: the fp16 rounding an engine stores it with).
    """
    B, S, C, N = x.shape
    L = enc.shape[1]
    a = P["dprnn.speakers_separation.0.weight"][0]
    p = np.where(x >= 0, x, a * x)
    Wspk = P["dprnn.speakers_separation.1.weight"].reshape(2 * N, N)
    y = p @ Wspk.T + P["dprnn.speakers_separation.1.bias"]  # (B,S,C,2N)
    Pstep = cfg.step_size
    ola = np.zeros((B, (S - 1) * Pstep + C, 2 * N), dtype=x.dtype)
    for s in range(S):
        ola[:, Pstep * s : Pstep * s + C, :] += y[:, s, :, :]
    d = L - ola.shape[1]
    ola = np.pad(ola, [(0, 0), (d // 2, d - d // 2), (0, 0)])
    if round_ola is not None:
        ola = round_ola(ola)
    if taps is not None:
        taps["ola"] = ola
    outs = []
    for j in range(2):
        o = ola[:, :, j * N : (j + 1) * N]
        if cfg.kind == "dptn_mask":
            # dptn.py:103-115,141: ReLU(tanh(conv(o)) * sigmoid(conv_gate(o))), decoder on m*enc (:189)
            t = np.tanh(o @ P["dprnn.output.0.weight"][:, :, 0].T + P["dprnn.output.0.bias"])
            g = sigmoid(o @ P["dprnn.output_gate.0.weight"][:, :, 0].T + P["dprnn.output_gate.0.bias"])
            outs.append(np.maximum(t * g, 0.0) * enc)
        else:
            h = o @ P["dprnn.postprocessing.0.weight"][:, :, 0].T + P["dprnn.postprocessing.0.bias"]
            outs.append(h + enc)
    return outs


def decode(u, w_dec, stride, T):
    """D1: nn.ConvTranspose1d(N,1,K,stride,bias=False) + centred pad (dptn_wav.py:187-193).

    u (B,L,N) -> (B,T): w[b, st*l+k] += sum_n Wd[n,0,k] u[b,l,n].
    """
    B, L, N = u.shape
    K = w_dec.shape[-1]
    fr = u @ w_dec[:, 0, :]  # (B,L,K)
    out = np.zeros((B, (L - 1) * stride + K), dtype=u.dtype)
    for k in range(K):
        out[:, k : k + stride * L : stride] += fr[:, :, k]
    return centre_pad_last(out, T)


def segment_token_major(enc, C, Pstep):
    """S1 on token-major data: x[b,s,k,:] = enc[b,P*s+k,:]."""
    B, L, N = enc.shape
    S = (L - C) // Pstep + 1
    idx = Pstep * np.arange(S)[:, None] + np.arange(C)[None, :]
    return enc[:, idx, :]


def forward(P, cfg: PathConfig, mix, emb1=None, emb2=None, taps=None):
    """Whole forward: DPTNAVWavEncDec / DPTNWavEncDec / DPTNEncDec / DPRNNEncDec.

    dptn_wav.py:171-194, :101-113; dptn.py:183-195; dprnn.py:263-276.
    Returns (s1_pred, s2_pred), each (B,T).
    """
    dtype = P["encoder.weight"].dtype
    mix = np.asarray(mix, dtype=dtype)
    T = mix.shape[1]
    enc = encode(mix, P["encoder.weight"], cfg.stride)
    if cfg.kind == "dptn_av":
        enc = av_fuse(enc, np.asarray(emb1, dtype=dtype), np.asarray(emb2, dtype=dtype), P)
    if taps is not None:
        taps["encoded"] = enc
    x = segment_token_major(enc, cfg.chunk_size, cfg.step_size)
    x = dual_path_blocks(x, P, cfg, taps)
    us = separator_tail(x, enc, P, cfg, taps)
    return tuple(decode(u, P["decoder.weight"], cfg.stride, T) for u in us)


# --------------------------------------------------------------------------------------
# loss and metrics
# --------------------------------------------------------------------------------------
def sisnr_loss_rows(pred, gt):
    """L1 per row, before the batch mean: SiSNRLoss.forward (ss_losses.py:100-114).

    -20*log10(||a g||^2 / ||p - a g||^2) with zero-mean p,g and a=<g,p>/||g||^2, no eps.
    """
    p = pred - pred.mean(axis=-1, keepdims=True)
    g = gt - gt.mean(axis=-1, keepdims=True)
    alpha = (g * p).sum(-1, keepdims=True) / (g * g).sum(-1, keepdims=True)
    s = alpha * g
    e = p - s
    return -20.0 * np.log10((s * s).sum(-1) / (e * e).sum(-1))


def pit_sisnr_loss(s1p, s2p, s1, s2):
    """L2: BaseSSLoss.forward with SiSNRLoss (ss_losses.py:10-26,117-130): batch-level PIT."""
    l = lambda a, b: sisnr_loss_rows(a, b).mean()
    p1 = (l(s1p, s1) + l(s2p, s2)) / 2
    p2 = (l(s1p, s2) + l(s2p, s1)) / 2
    return p2 if p2 < p1 else p1


def pit_sisnr_loss_grad(s1p, s2p, s1, s2):
    """Gradient of `pit_sisnr_loss` with respect to (s1p, s2p): what `batch["loss"].backward()` (src/trainer/trainer.py:46)
    deposits on the predictions through BaseSSLoss.forward / SiSNRLoss.forward (ss_losses.py:10-26,100-114).

    With zero-mean p_c, g_c, a = <g_c,p_c>/||g_c||^2, e = p_c - a g_c:
        d/dp [-20 log10(||a g_c||^2 / ||e||^2)] = -(40/ln 10) (g_c/<g_c,p_c> - e/||e||^2)
    (g_c and e sum to zero, so the centring Jacobian is the identity); batch mean and the two terms of a permutation give
    the factor 1/(2B); the permutation is the one the forward chose for the whole batch."""
    l = lambda a, b: sisnr_loss_rows(a, b).mean()
    swap = (l(s1p, s2) + l(s2p, s1)) / 2 < (l(s1p, s1) + l(s2p, s2)) / 2
    t1, t2 = (s2, s1) if swap else (s1, s2)
    B = s1p.shape[0]

    def one(pred, gt):
        p = pred - pred.mean(axis=-1, keepdims=True)
        g = gt - gt.mean(axis=-1, keepdims=True)
        dot = (g * p).sum(-1, keepdims=True)
        e = p - dot / (g * g).sum(-1, keepdims=True) * g
        return -(40.0 / np.log(10.0)) / (2.0 * B) * (g / dot - e / (e * e).sum(-1, keepdims=True))

    return one(s1p, t1), one(s2p, t2)


def si_snr_metric_rows(pred, target, eps=None):
    """torchmetrics scale_invariant_signal_noise_ratio per row (restated; see header).

    zero-mean both; a=(<p,t>+eps)/(||t||^2+eps); 10*log10((||a t||^2+eps)/(||a t - p||^2+eps)).
    Call sites: src/metrics/base_metric.py:53-56, si_snri.py:25-26.
    """
    if eps is None:
        eps = np.finfo(np.float32).eps
    p = pred - pred.mean(axis=-1, keepdims=True)
    t = target - target.mean(axis=-1, keepdims=True)
    alpha = ((p * t).sum(-1, keepdims=True) + eps) / ((t * t).sum(-1, keepdims=True) + eps)
    ts = alpha * t
    noise = ts - p
    val = ((ts * ts).sum(-1) + eps) / ((noise * noise).sum(-1) + eps)
    return 10.0 * np.log10(val)


def pit_si_snr(s1p, s2p, s1, s2):
    """L3: SS2BaseMetric.forward (base_metric.py:41-60): batch-mean metric, batch-level max."""
    m = lambda a, b: float(si_snr_metric_rows(a, b).mean())
    return max((m(s1p, s1) + m(s2p, s2)) / 2, (m(s1p, s2) + m(s2p, s1)) / 2)


def pit_si_snri(s1p, s2p, s1, s2, mix):
    """SISNRiMetric.__call__ (si_snri.py:12-30)."""
    m = lambda a, b: float(si_snr_metric_rows(a, b).mean())
    return pit_si_snr(s1p, s2p, s1, s2) - (m(mix, s1) + m(mix, s2)) / 2
