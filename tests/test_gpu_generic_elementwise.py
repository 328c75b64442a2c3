"""The GENERIC engine's fp32 SIMT kernels (csrc/generic_block.cu) element by element against fp64 references, and its
whole forward against the fp64 oracle at the configurations that run on it.

engine="auto" falls back to this engine for every shape the tensor engine refuses (hidden_dim != 128, num_features
outside {64, 128}, DPRNN with N != 64, head dims outside {16, 32}), so its kernels must hold for every dimension they
accept: any sequence length, any head dim up to 64, H up to 128.  A waveform rel-L2 hides an error confined to one
head, the last key or one LSTM direction; here every output element gets its own bound from an error model of the
kernel, and every output is a view into a larger allocation whose guard rows and unused pitched columns must keep
their sentinel bit pattern.

References are computed in float64 with torch on the device, from the exact fp32 operands the kernels read, and never
go through the library.  u = 2^-24 is the unit roundoff of fp32."""
import ctypes
import math
import warnings

import numpy as np
import pytest
import torch

from oracle import vatss_oracle as O

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")]

DEV = torch.device("cuda:0")
U = 2.0 ** -24            # unit roundoff of fp32
TINY = 2.0 ** -126        # smallest normal fp32: covers underflow of a product
GUARD_ROWS = 8            # whole sentinel rows before and after every output view
SENT_BITS = 0x7FC05A5A    # a NaN bit pattern: an element the kernel should have written and did not fails every bound


@pytest.fixture(scope="module")
def lib():
    from speech_separation_b200 import _lib

    return _lib.load()


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _err(lib):
    return lib.vatss_last_error().decode("utf-8", "replace")


def _check(lib, rc, what):
    assert rc == 0, f"{what} failed (rc={rc}): {_err(lib)}"


def guarded(rows, cols, ld=None, col0=0):
    """(allocation, view): a (rows, cols) fp32 view with row pitch ld starting at column col0 inside an allocation with
    GUARD_ROWS sentinel rows before and after it; every element starts as the sentinel."""
    ld = ld or cols
    buf = torch.empty(rows + 2 * GUARD_ROWS, ld, dtype=torch.float32, device=DEV)
    buf.view(torch.int32).fill_(SENT_BITS)
    return buf, buf[GUARD_ROWS:GUARD_ROWS + rows, col0:col0 + cols]


def assert_guard(buf, rows, cols, label, col0=0):
    """Everything of the allocation outside the (rows, cols) view at column col0 still holds the sentinel."""
    outside = torch.ones(buf.shape, dtype=torch.bool, device=DEV)
    outside[GUARD_ROWS:GUARD_ROWS + rows, col0:col0 + cols] = False
    bad = (buf.view(torch.int32) != SENT_BITS) & outside
    n = int(bad.sum())
    if n:
        r, c = [int(v) for v in bad.nonzero()[0]]
        raise AssertionError(f"{label}: {n} elements written outside the output, first at allocation row {r} "
                             f"(output row {r - GUARD_ROWS}), column {c}")


def check_elements(got, want, bound, label):
    """|got - want| <= bound element by element (NaN fails); returns the worst |err| / bound."""
    got = got.double()
    err = (got - want).abs()
    ok = err <= bound
    if not bool(ok.all()):
        idx = tuple(int(t) for t in (~ok).nonzero()[0])
        raise AssertionError(f"{label}: {int((~ok).sum())} of {ok.numel()} elements out of bound; first at {idx}: "
                             f"got {float(got[idx]):.8g} want {float(want[idx]):.8g} err {float(err[idx]):.3e} "
                             f"bound {float(bound[idx]):.3e}")
    return float((err / bound).max())


def report(family, ratio, label=""):
    print(f"WORST-RATIO {family}: {ratio:.3f} {label}")


# ======================================================================================================================
# A. GEMM (k_gemm_simt)
# ======================================================================================================================
# C = act(A) W^T + bias + bias2 + R, fp32 FMA accumulation in k order from 0, then the three adds, each rounded:
#   |c^ - c| <= (K + 3) u (sum_k |act(a_k) w_nk| + |bias| + |bias2| + |r|) + 2^-126
# (K + 3 roundings of partial sums each at most that large; PReLU's fp32 product slope * a adds one more relative
# rounding to the A terms, so K + 4 there; 2^-126 covers an underflowing product).
GEMM_M = [1, 63, 65, 4097]
GEMM_NK = [(4, 4), (24, 12), (48, 24), (96, 96), (384, 256), (512, 256), (512, 4), (4, 256)]
GEMM_ACT = [(0, None), (1, None), (2, -0.3), (2, 1.7)]


def _gemm_case(lib, M, NOUT, K, act, slope, full, seed):
    g = torch.Generator().manual_seed(seed)
    # A is the second half of a (M, 2K) row-major buffer: the tail's `ola + j N` with lda = 2N
    a_buf = torch.randn(M, 2 * K, generator=g).to(DEV)
    A = a_buf[:, K:]
    W = (torch.randn(NOUT, K, generator=g) / K ** 0.5).to(DEV)
    bias = torch.randn(NOUT, generator=g).to(DEV) if full else None
    bias2 = torch.randn(NOUT, generator=g).to(DEV) if full else None
    ldr = NOUT + 3
    r_buf = torch.randn(M, ldr, generator=g).to(DEV)
    R = r_buf[:, :NOUT] if full else None
    prelu = torch.tensor([slope if slope is not None else 0.0], device=DEV)
    # output at column offset NOUT of a (M, 2 NOUT) pitched buffer: the LSTM input projection's `pre + dir 4H`
    buf, out = guarded(M, NOUT, ld=2 * NOUT, col0=NOUT)
    rc = lib.vatss_generic_gemm(_p(A), 2 * K, _p(W), _p(bias), _p(bias2), _p(R), ldr if full else 0, _p(out),
                                2 * NOUT, M, NOUT, K, act, _p(prelu) if act == 2 else None, None)
    _check(lib, rc, "vatss_generic_gemm")
    torch.cuda.synchronize()
    label = f"gemm M={M} NOUT={NOUT} K={K} act={act} slope={slope} {'bias+bias2+R' if full else 'bare'}"
    assert_guard(buf, M, NOUT, label, col0=NOUT)
    a = A.double()
    if act == 1:
        a = a.clamp_min(0.0)
    elif act == 2:
        a = torch.where(a >= 0, a, slope * a)     # the fp32 slope value, exact in fp64
    want = a @ W.double().t()
    mag = a.abs() @ W.double().abs().t()
    extra = torch.zeros_like(want)
    if full:
        add = bias.double() + bias2.double() + R.double()
        want = want + add
        extra = bias.double().abs() + bias2.double().abs() + R.double().abs()
    nround = K + 3 + (1 if act == 2 else 0)
    bound = nround * U * (mag + extra) + TINY
    return check_elements(out, want, bound, label)


@pytest.mark.parametrize("act,slope", GEMM_ACT, ids=["none", "relu", "prelu-0.3", "prelu1.7"])
@pytest.mark.parametrize("NOUT,K", GEMM_NK, ids=[f"{n}x{k}" for n, k in GEMM_NK])
def test_gemm_matches_fp64(lib, NOUT, K, act, slope):
    worst = 0.0
    for M in GEMM_M:
        for full in (True, False):
            worst = max(worst, _gemm_case(lib, M, NOUT, K, act, slope, full, seed=M + NOUT + K + act))
    report(f"gemm act={act}", worst, f"(NOUT={NOUT} K={K})")


# ======================================================================================================================
# B. LayerNorm (k_layernorm: one warp per row, NI = ceil(N / 32) values per lane)
# ======================================================================================================================
# x = in + res (mode 0, one rounding u|x|), mu = warp tree sum (NI - 1 + 5 adds) / N, var = the same over d^2, rstd =
# rsqrtf(var + eps) (2 ulp), y = (x - mu) rstd w + b (3 roundings), mode 1 then y + res (1 rounding).  Per row:
#   d_mu  = (NI + 6) u sum|x| / N                        error of the mean (the inputs' rounding included)
#   r_sd  = (NI + 8) u / 2 + 2 u + 2^-22 + d_mu^2 / (2 (var + eps))   relative error of rstd (the sum of squares,
#           the eps add, rsqrtf, and the mean's error entering the variance to second order)
# Per element:
#   |y - y^| <= |w| rstd (d_mu + u |x_n|) + |(x_n - mu) rstd w| (r_sd + 3 u) + 2 u (|y_ln| + |y^|) + 2^-126
LN_N = [4, 12, 32, 36, 64, 96, 128, 256]
LN_ROWS = 203          # not a multiple of the 8 rows per CTA
N_STRESS = 12          # rows 0-3 constant, 4-7 mean 10^3 std 1, 8-11 variance ~ eps (res is zero on these rows)


def _ln_inputs(N, with_res, seed):
    g = torch.Generator().manual_seed(seed)
    x = 2.0 * torch.randn(LN_ROWS, N, generator=g, dtype=torch.float64) + 0.5
    for i, c in enumerate((3.0, -0.5, 0.1, 1e3)):
        x[i] = c
    x[4:8] = 1e3 + torch.randn(4, N, generator=g, dtype=torch.float64)
    x[8:12] = -0.25 + 3.2e-3 * torch.randn(4, N, generator=g, dtype=torch.float64)
    res = None
    if with_res:
        res = torch.randn(LN_ROWS, N, generator=g)
        res[:N_STRESS] = 0.0
        res = res.to(DEV)
    w = (1 + 0.2 * torch.randn(N, generator=g)).to(DEV)
    b = (0.1 * torch.randn(N, generator=g)).to(DEV)
    return x.float().to(DEV), res, w, b


def ln_reference(x_in, res, w, b, mode):
    """fp64 LayerNorm and the per-element bound of the model above."""
    N = x_in.shape[1]
    NI = (N + 31) // 32
    x = x_in.double() + (res.double() if (mode == 0 and res is not None) else 0.0)
    mu = x.mean(-1, keepdim=True)
    d = x - mu
    var = (d * d).mean(-1, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + 1e-5)
    y_ln = d * rstd * w.double() + b.double()
    y = y_ln + (res.double() if (mode == 1 and res is not None) else 0.0)
    d_mu = (NI + 6) * U * x.abs().sum(-1, keepdim=True) / N
    r_sd = (NI + 8) * U / 2 + 2 * U + 2.0 ** -22 + d_mu ** 2 / (2 * (var + 1e-5))
    aw = w.double().abs()
    bound = (aw * rstd * (d_mu + U * x.abs()) + (d * rstd * w.double()).abs() * (r_sd + 3 * U)
             + 2 * U * (y_ln.abs() + y.abs()) + TINY)
    return y, bound


@pytest.mark.parametrize("mode,with_res", [(0, True), (0, False), (1, True), (1, False)],
                         ids=["ln-of-sum", "ln", "ln-plus-res", "ln-no-res"])
@pytest.mark.parametrize("N", LN_N)
def test_layernorm_matches_fp64(lib, N, mode, with_res):
    x, res, w, b = _ln_inputs(N, with_res, seed=N + 2 * mode + int(with_res))
    worst = 0.0
    for rows in (LN_ROWS, 1, 7, 17):
        buf, out = guarded(rows, N)
        r = res[:rows] if res is not None else None
        rc = lib.vatss_generic_layernorm(_p(x), _p(r), _p(w), _p(b), _p(out), rows, N, mode, None)
        _check(lib, rc, "vatss_generic_layernorm")
        torch.cuda.synchronize()
        label = f"layernorm mode={mode} res={with_res} N={N} rows={rows}"
        assert_guard(buf, rows, N, label)
        want, bound = ln_reference(x[:rows], r, w, b, mode)
        worst = max(worst, check_elements(out, want, bound, label))
        if rows == LN_ROWS:
            # constant rows whose sums are exact: d = 0, so the output is b itself (res is zero on them)
            for i in (0, 1, 3):
                assert torch.equal(out[i], b), f"{label}: constant row {i} is not b"
    report(f"layernorm mode={mode}{' res' if with_res else ''}", worst, f"(N={N})")


def test_layernorm_rejects_n_above_256(lib):
    x = torch.randn(16, 260, device=DEV)
    w = torch.ones(260, device=DEV)
    buf, out = guarded(16, 260)
    rc = lib.vatss_generic_layernorm(_p(x), None, _p(w), _p(w), _p(out), 16, 260, 0, None)
    torch.cuda.synchronize()
    assert rc != 0 and "N=260" in _err(lib)
    assert_guard(buf, 0, 0, "layernorm N=260")


# ======================================================================================================================
# C. attention (k_attention_simt: one query per thread, K / V streamed through shared memory in key tiles)
# ======================================================================================================================
# The softmax error model of test_gpu_tc_elementwise.py with cP = 0 (P stays fp32) and u = 2^-24, per output element
# o of a row (p_j = softmax weights, m = sum_j p_j |v_j| >= |o^|):
#   |o - o^| <= u |o^| + (gamma + sigma) m + 2^-126
#   u |o^|     the final multiply by 1 / l.
#   gamma = (4 len + 16) u + 2^-20   fp32 accumulation of acc and of the row sum l (len roundings each), a rescale of
#              both per key at most (another len each; the rescale factor itself cancels in acc / l), the divide; 2^-20
#              covers expf (2 ulp, 2^-22 relative) on every p_j, in numerator and denominator (2 m per 2^-22).
#   sigma = 2 (hd + 6) u max_j sum_d |q_d k_jd| / sqrt(hd)   the fp32 score error: hd FMA roundings, rsqrtf (2 ulp)
#              and the q * scale rounding, the subtraction of the running maximum; ds moves p_j by ds relatively,
#              which moves o by at most 2 ds m.
ATT_HDS = [1, 2, 4, 8, 16, 32, 64, 3, 12, 20, 24, 48]
ATT_LENS = [1, 2, 127, 128, 129, 400, 401, 800, 801, 3198]
ATT_HEADS = 2


def _seqs(x, mode, B, S, C):
    """(B, S, C, F) -> (G, len, F): intra sequences (b, s) over c, inter sequences (b, c) over s."""
    return x.reshape(B * S, C, -1) if mode == 0 else x.permute(0, 2, 1, 3).reshape(B * C, S, -1)


def _unseqs(y, mode, B, S, C):
    return y.reshape(B, S, C, -1) if mode == 0 else y.reshape(B, C, S, -1).permute(0, 2, 1, 3)


def attention_inputs(kind, mode, B, S, C, N, heads, seed):
    """fp32 qkv (B, S, C, 3N), q unscaled as the in-projection leaves it (the kernel applies 1 / sqrt(hd)).
    random:  q x2 for a peakier softmax.
    leak:    (intra) the keys of every other sequence score ~20 above the others for every query, so a key of a
             neighbouring sequence that leaks across the len boundary dominates its row.
    growing: key scale grows along the sequence (logits up to ~30): the online rescale runs at almost every key.
    onehot:  one key per sequence scores ~30 above all others: near-one-hot rows.
    uniform: all keys equal: uniform rows, o = mean of v."""
    hd = N // heads
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, S, C, 3 * N, generator=g)
    L = C if mode == 0 else S
    kv_shape = (1, 1, L, 1) if mode == 0 else (1, L, 1, 1)
    d = torch.ones(N) / hd ** 0.5                        # per head a unit direction
    if kind == "random":
        x[..., :N] *= 2.0
    elif kind == "leak":
        assert mode == 0
        a = math.sqrt(20.0 * hd ** 0.5)
        x[..., :N] += a * d
        hot = (torch.arange(B * S) % 2 == 0).reshape(B, S, 1, 1).float()
        x[..., N:2 * N] += hot * a * d
    elif kind == "growing":
        x[..., :N] *= 2.0
        x[..., N:2 * N] *= torch.linspace(0.3, 6.0, L).reshape(kv_shape)
    elif kind == "onehot":
        a = math.sqrt(30.0 * hd ** 0.5)
        x[..., :N] = 0.3 * x[..., :N] + a * d
        pick = torch.zeros(L)
        pick[int(torch.randint(L, (1,), generator=g))] = 1.0
        x[..., N:2 * N] = 0.3 * x[..., N:2 * N] + pick.reshape(kv_shape) * a * d
    elif kind == "uniform":
        x[..., N:2 * N] = 0.5
    else:
        raise ValueError(kind)
    return x.to(DEV).contiguous()


def attention_reference(qkv, mode, B, S, C, N, heads):
    """fp64 o^ = softmax(q k^T / sqrt(hd)) v and the per-element bound of the model above, as (B, S, C, N)."""
    hd = N // heads
    seq = _seqs(qkv.double(), mode, B, S, C)
    G, L = seq.shape[0], seq.shape[1]
    q, k, v = (seq[..., i * N:(i + 1) * N].reshape(G, L, heads, hd).transpose(1, 2) for i in range(3))
    s = q @ k.transpose(-1, -2) / math.sqrt(hd)
    p = torch.softmax(s, dim=-1)
    del s
    o = p @ v
    m = p @ v.abs()
    del p
    smag = (q.abs() @ k.abs().transpose(-1, -2)).amax(-1, keepdim=True) / math.sqrt(hd)
    sigma = 2 * (hd + 6) * U * smag
    gamma = (4 * L + 16) * U + 2.0 ** -20
    bound = U * o.abs() + (gamma + sigma) * m + TINY
    back = lambda t: _unseqs(t.transpose(1, 2).reshape(G, L, N), mode, B, S, C)
    return back(o), back(bound)


def _attn_case(lib, kind, mode, B, S, C, N, heads, seed):
    qkv = attention_inputs(kind, mode, B, S, C, N, heads, seed)
    tokens = B * S * C
    buf, out = guarded(tokens, N)
    rc = lib.vatss_generic_attention(_p(qkv), _p(out), mode, B, S, C, N, heads, None)
    _check(lib, rc, "vatss_generic_attention")
    torch.cuda.synchronize()
    label = f"attention {kind} mode={mode} B={B} S={S} C={C} N={N} heads={heads}"
    assert_guard(buf, tokens, N, label)
    want, bound = attention_reference(qkv, mode, B, S, C, N, heads)
    return check_elements(out.reshape(B, S, C, N), want, bound, label)


def _att_shape(mode, L):
    return (1, 3, L) if mode == 0 else (1, L, 3)     # three sequences of length L


@pytest.mark.parametrize("mode", [0, 1], ids=["intra", "inter"])
@pytest.mark.parametrize("hd", ATT_HDS)
def test_attention_length_sweep(lib, hd, mode):
    """Every head dim at lengths around the query blocks (128) and the key tiles (4096 / HDMAX keys: 512, 256, 128,
    64), up to the default model's inter length 3198.  Intra inputs use the leak pattern."""
    worst, at = 0.0, None
    N = hd * ATT_HEADS
    for L in ATT_LENS:
        B, S, C = _att_shape(mode, L)
        r = _attn_case(lib, "leak" if mode == 0 else "random", mode, B, S, C, N, ATT_HEADS, seed=L + hd)
        if r > worst:
            worst, at = r, L
    report(f"attention hd={hd} {'intra' if mode == 0 else 'inter'} sweep", worst, f"(len {at})")


STRESS_SHAPES = [(0, 2, 3, 150), (0, 1, 2, 513), (1, 1, 283, 3), (1, 1, 801, 2)]


@pytest.mark.parametrize("kind", ["growing", "onehot", "uniform"])
@pytest.mark.parametrize("hd", [4, 12, 16, 24, 32, 64])
def test_attention_stress_inputs(lib, hd, kind):
    worst = 0.0
    for heads in (1, 4):
        for mode, B, S, C in STRESS_SHAPES:
            worst = max(worst, _attn_case(lib, kind, mode, B, S, C, hd * heads, heads, seed=S + C + hd + heads))
    report(f"attention hd={hd} {kind}", worst)


def test_attention_head_dim_above_64_is_an_error(lib):
    N, heads, B, S, C = 128, 1, 1, 2, 5
    qkv = torch.randn(B * S * C, 3 * N, device=DEV)
    buf, out = guarded(B * S * C, N)
    rc = lib.vatss_generic_attention(_p(qkv), _p(out), 0, B, S, C, N, heads, None)
    torch.cuda.synchronize()
    assert rc != 0 and "head dim 128" in _err(lib)
    assert_guard(buf, 0, 0, "attention hd 128")


# ======================================================================================================================
# D. LSTM recurrence (k_lstm_simt: 8 sequences of one direction per CTA, W_hh^T in shared memory)
# ======================================================================================================================
# The reference is an fp64 recurrence from the same fp32 `pre` (x W_ih^T + b_ih + b_hh) and the same W_hh: fp32
# values, or rounded to fp16 exactly where the launcher does (16 H^2 + 192 H > 204800 bytes of shared memory, i.e.
# H >= 108).  What remains is fp32 arithmetic: per step the gate pre-activations carry H FMA roundings of terms
# |w h| <= |w| (random signs: ~sqrt(H) u of their scale), sigmoid / tanh through expf / tanhf (2 ulp each), and the
# c / h updates (4 roundings).  The forget gate (< 1) contracts the error carried in c and the W_hh feedback of
# random-sign errors averages out, so the bound is a constant per element, independent of the length:
#   |h - h^| <= (16 + 2 sqrt(H)) u
# (an fp32 emulation of the kernel stays below 6 u for H <= 128 up to 710 steps; W_hh rounded to fp16 where the
# reference keeps fp32 gives ~850 u at H = 104).
LSTM_H = [4, 12, 32, 64, 100, 104, 108, 128]
LSTM_SHAPES = [
    # mode, B, S, C:  G = B S (intra) or B C (inter), G % 8 in {0, 1, 7}
    (0, 1, 8, 50), (0, 3, 3, 1), (0, 1, 7, 33), (1, 1, 710, 7), (1, 2, 130, 8), (1, 1, 1, 9), (1, 3, 41, 3),
]


def whh_is_fp16(H):
    """launch_lstm_simt: W_hh^T stays fp32 while 2 * 8 H + 8 * 4 H floats of state plus 4 H^2 fp32 weights fit in
    200 KB of shared memory."""
    return 16 * H * H + 192 * H > 200 * 1024


def _lstm_operands(H, ndir, B, S, C, seed):
    """pre (rows, ndir 4H) fp32 = x W_ih^T + 3 (b_ih + b_hh) (biases x3 so that the gates saturate), W_hh per
    direction fp32 (PyTorch initialisation)."""
    torch.manual_seed(seed)
    rnn = torch.nn.LSTM(64, H, batch_first=True, bidirectional=(ndir == 2)).double()
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B * S * C, 64, generator=g, dtype=torch.float64)
    sufs = ["", "_reverse"][:ndir]
    pre = torch.cat([x @ getattr(rnn, "weight_ih_l0" + s).detach().t()
                     + 3.0 * (getattr(rnn, "bias_ih_l0" + s) + getattr(rnn, "bias_hh_l0" + s)).detach()
                     for s in sufs], dim=1)
    whh = [getattr(rnn, "weight_hh_l0" + s).detach().float().to(DEV).contiguous() for s in sufs]
    return pre.float().to(DEV).contiguous(), whh


def lstm_reference(pre, whh, H, mode, B, S, C):
    """fp64 recurrence; returns h as (B, S, C, ndir H)."""
    ndir = len(whh)
    seq = _seqs(pre.double().reshape(B, S, C, -1), mode, B, S, C)       # (G, L, ndir 4H)
    G, L = seq.shape[0], seq.shape[1]
    outs = []
    for d in range(ndir):
        W = whh[d].half().double() if whh_is_fp16(H) else whh[d].double()
        h = torch.zeros(G, H, dtype=torch.float64, device=DEV)
        c = torch.zeros_like(h)
        y = torch.empty(G, L, H, dtype=torch.float64, device=DEV)
        for step in range(L):
            t = step if d == 0 else L - 1 - step
            a = seq[:, t, d * 4 * H:(d + 1) * 4 * H] + h @ W.t()
            i_, f_, g_, o_ = a.split(H, dim=1)
            c = torch.sigmoid(f_) * c + torch.sigmoid(i_) * torch.tanh(g_)
            h = torch.sigmoid(o_) * torch.tanh(c)
            y[:, t] = h
        outs.append(y)
    return _unseqs(torch.cat(outs, dim=-1), mode, B, S, C)


def check_lstm(out, ref, H, mode, B, S, C, bound, label):
    """Per element against the constant bound, then the worst error per step band (first / middle / last tenth of the
    direction's processing order, and its first step)."""
    got = out.reshape(B, S, C, -1)
    ratio = check_elements(got, ref, torch.full_like(ref, bound), label)
    e = _seqs((got.double() - ref).abs(), mode, B, S, C)              # (G, L, ndir H)
    L = e.shape[1]
    n = max(1, L // 10)
    bands = []
    for d in range(e.shape[2] // H):
        ed = e[..., d * H:(d + 1) * H].amax(dim=(0, 2))
        if d == 1:
            ed = ed.flip(0)
        mid = (L - n) // 2
        bands.append(f"dir{d} first {float(ed[:n].max()):.2e} mid {float(ed[mid:mid + n].max()):.2e} "
                     f"last {float(ed[-n:].max()):.2e} step0 {float(ed[0]):.2e}")
    print(f"{label}: " + "; ".join(bands))
    return ratio


@pytest.mark.parametrize("ndir", [1, 2])
@pytest.mark.parametrize("H", LSTM_H)
def test_lstm_matches_fp64_recurrence(lib, H, ndir):
    bound = (16 + 2 * math.sqrt(H)) * U
    worst = 0.0
    for mode, B, S, C in LSTM_SHAPES:
        pre, whh = _lstm_operands(H, ndir, B, S, C, seed=H + ndir + S + C)
        rows = B * S * C
        buf, out = guarded(rows, ndir * H)
        rc = lib.vatss_generic_lstm(_p(pre), _p(whh[0]), _p(whh[1]) if ndir == 2 else None, _p(out), mode, B, S, C,
                                    H, ndir, None)
        _check(lib, rc, "vatss_generic_lstm")
        torch.cuda.synchronize()
        label = (f"lstm H={H} ({'fp16' if whh_is_fp16(H) else 'fp32'} W_hh) ndir={ndir} mode={mode} "
                 f"B={B} S={S} C={C}")
        assert_guard(buf, rows, ndir * H, label)
        ref = lstm_reference(pre, whh, H, mode, B, S, C)
        worst = max(worst, check_lstm(out, ref, H, mode, B, S, C, bound, label))
    report(f"lstm H={H} ndir={ndir}", worst)


def test_lstm_whh_precision_boundary():
    """The rule the reference above applies: fp32 W_hh up to H = 104, fp16 from H = 108 (H is a multiple of 4)."""
    assert [H for H in range(4, 129, 4) if whh_is_fp16(H)] == list(range(108, 129, 4))


# ======================================================================================================================
# E. whole forward on the GENERIC engine against the fp64 oracle
# ======================================================================================================================
LN_NAMES = ("ln1.", "ln2.", "video_ln.", "norm1d.")
LARGE_BIAS = ("speakers_separation.1.bias", "postprocessing.0.bias", "output.0.bias", "output_gate.0.bias")


def make_net(kind, seed, **kw):
    """Random non-default weights as in test_gpu_tc_elementwise.py: dense ~ 0.6 / sqrt(fan-in), LayerNorm affine
    1 + 0.2 n / 0.1 n, split and head biases ~ N(0, 1)."""
    import speech_separation_b200 as V

    cls = {"dptn_av": V.DPTNAVWavEncDec, "dptn_wav": V.DPTNWavEncDec, "dptn_mask": V.DPTNEncDec,
           "dprnn": V.DPRNNEncDec}[kind]
    net = cls(**kw).eval()
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in net.named_parameters():
            r = torch.randn(p.shape, generator=g, dtype=torch.float64)
            if name.endswith(LARGE_BIAS):
                v = r
            elif any(s in name for s in LN_NAMES):
                v = 1 + 0.2 * r if name.endswith("weight") else 0.1 * r
            elif name == "gate":
                v = 0.5 + 0.5 * r.abs()
            elif name == "decoder.weight":
                v = 0.6 * r / math.sqrt(p.shape[0])
            elif p.dim() >= 2:
                v = 0.6 * r / math.sqrt(p[0].numel())
            else:
                v = 0.1 * r
            p.copy_(v)
    return net.to(DEV)


PROD = dict(num_features=128, kernel_size_enc=7, hidden_dim=128, num_blocks=1, chunk_size=150, step_size=75,
            num_heads=4)
SMALL = dict(kernel_size_enc=16, num_blocks=1, chunk_size=100, step_size=50)
FORWARD_CASES = [
    # id, kind, constructor arguments, engine, B, T
    ("dptn_wav-class-defaults-2-blocks", "dptn_wav", dict(num_blocks=2), "auto", 1, 16000),
    ("dprnn-N128", "dprnn", dict(SMALL, num_features=128, hidden_dim=128), "auto", 2, 16000),
    ("dptn_wav-N96-h4", "dptn_wav", dict(SMALL, num_features=96, hidden_dim=128, num_heads=4), "auto", 2, 16000),
    ("dptn_wav-N128-h2-8s", "dptn_wav", dict(PROD, num_heads=2), "auto", 1, 128000),
    ("dptn_av-production-generic-12.5s", "dptn_av", dict(PROD, video_emb_size=512, hidden_video=128), "generic", 1,
     200000),
    ("dptn_wav-H104", "dptn_wav", dict(SMALL, num_features=64, hidden_dim=104, num_heads=4), "auto", 2, 16000),
    ("dptn_wav-H108", "dptn_wav", dict(SMALL, num_features=64, hidden_dim=108, num_heads=4), "auto", 2, 16000),
    ("dptn_mask-unidir-inter", "dptn_mask", dict(SMALL, num_features=64, hidden_dim=64, num_heads=4, bidir=False),
     "auto", 2, 16000),
]


@pytest.mark.parametrize("kind,kw,engine,B,T", [c[1:] for c in FORWARD_CASES], ids=[c[0] for c in FORWARD_CASES])
def test_generic_forward_matches_oracle(lib, kind, kw, engine, B, T):
    net = make_net(kind, seed=B + T + kw.get("num_features", 64), **kw).set_engine(engine)
    g = torch.Generator().manual_seed(T)
    mix = torch.randn(B, T, generator=g)
    Tv = -(-T // 640)                                    # 25 video frames per second at 16 kHz
    e1 = torch.randn(B, 512, Tv, generator=g) if kind == "dptn_av" else None
    e2 = torch.randn(B, 512, Tv, generator=g) if kind == "dptn_av" else None
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always", RuntimeWarning)
        with torch.no_grad():
            if e1 is None:
                out = net(mix=mix.to(DEV))
            else:
                out = net(mix=mix.to(DEV), s1_embedding=e1.to(DEV), s2_embedding=e2.to(DEV))
        got = (out["s1_pred"].cpu().numpy(), out["s2_pred"].cpu().numpy())
    fallback = [w for w in caught if "fp32 SIMT engine" in str(w.message)]
    if engine == "auto":
        assert fallback, f"{kind} {kw}: engine='auto' ran the generic engine without its fallback warning"
    else:
        assert not fallback
    assert lib.vatss_packed_weight_bytes(ctypes.byref(net._desc)) == 0, "the model did not run on the generic engine"
    nk = dict(kw)
    nk.pop("hidden_video", None)
    defaults = dict(num_features=64, kernel_size_enc=2, hidden_dim=32, num_blocks=6, chunk_size=10, step_size=5,
                    num_heads=4, bidir=True, video_emb_size=512)
    defaults.update(nk)
    cfg = O.PathConfig(kind=kind, **defaults)
    ref = O.forward(O.to_numpy_state(net.state_dict(), np.float64), cfg, mix.double().numpy(),
                    None if e1 is None else e1.double().numpy(), None if e2 is None else e2.double().numpy())
    worst = 0.0
    for spk, (gw, rw) in enumerate(zip(got, ref)):
        assert np.isfinite(gw).all(), f"{kind} spk{spk}: non-finite output"
        for b in range(B):
            rel = float(np.linalg.norm(gw[b] - rw[b]) / np.linalg.norm(rw[b]))
            assert rel <= 2e-4, f"{kind} {kw} spk{spk} utt{b}: rel-L2 {rel:.3e} > 2e-4"
            worst = max(worst, rel)
    print(f"generic forward {kind} {kw} B={B} T={T}: worst rel-L2 {worst:.2e}")
