"""The tcgen05 attention, LSTM and GEMM kernels element by element against fp64 references, at every head layout the
tensor engine accepts.

test_gpu_tensor_kernels.py checks one global rel-L2 per launch, which an error confined to one head, one row, the last
key or the first reverse step hides under.  Here every output element gets its own bound from an error model of the
kernel, every output buffer is a view into a larger allocation whose guard rows (and unused pitched columns) must keep
their sentinel bit pattern, and the persistent kernels must give bit-identical results whatever the grid.

References are computed in float64 with torch on the device, from the same fp16-rounded operands the kernels read, and
never go through the library.  Every debug switch is reset in a `finally`."""
import contextlib
import ctypes
import math
import warnings

import numpy as np
import pytest
import torch

from oracle import vatss_oracle as O

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")]

DEV = torch.device("cuda:0")
U16 = 2.0 ** -11          # unit roundoff of fp16
LOG2E = 1.4426950408889634
GUARD_ROWS = 8            # whole sentinel rows before and after every output view (keeps 16-byte row alignment)
SENTINEL = {torch.float16: (torch.int16, 0x7E5A), torch.float32: (torch.int32, 0x7FC05A5A)}   # NaN bit patterns
LAYOUTS = [(128, 4), (128, 8), (64, 4), (64, 2)]   # (N, heads): head dim 32 / 16 with 2 / 1 groups of 64 features


@pytest.fixture(scope="module")
def lib():
    assert torch.cuda.is_available()
    from speech_separation_b200 import _lib

    return _lib.load()


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _check(rc, what):
    from speech_separation_b200 import _lib

    _lib.check(rc, what)


@contextlib.contextmanager
def debug_reset(lib):
    """Every debug switch back to its production default, however the block exits."""
    try:
        yield
    finally:
        lib.vatss_debug_attention_version(3)
        lib.vatss_debug_cta_limit(0)
        lib.vatss_debug_lstm_pingpong(1)
        lib.vatss_debug_lstm_groups(0)
        lib.vatss_debug_gemm_l2_order(-1)   # -1: re-read VATSS_GEMM_L2_ORDER (default on) at the next forward


def guarded(rows, cols, dtype, ld=None):
    """(allocation, view): a (rows, cols) view with row pitch ld inside an allocation with GUARD_ROWS sentinel rows
    before and after it; every element starts as the sentinel NaN pattern."""
    ld = ld or cols
    itype, pat = SENTINEL[dtype]
    buf = torch.empty(rows + 2 * GUARD_ROWS, ld, dtype=dtype, device=DEV)
    buf.view(itype).fill_(pat)
    return buf, buf[GUARD_ROWS:GUARD_ROWS + rows, :cols]


def assert_guard(buf, rows, cols, label):
    """Everything of the allocation outside the (rows, cols) view still holds the sentinel."""
    itype, pat = SENTINEL[buf.dtype]
    outside = torch.ones(buf.shape, dtype=torch.bool, device=DEV)
    outside[GUARD_ROWS:GUARD_ROWS + rows, :cols] = False
    bad = (buf.view(itype) != pat) & outside
    n = int(bad.sum())
    if n:
        r, c = [int(v) for v in bad.nonzero()[0]]
        raise AssertionError(f"{label}: {n} elements written outside the output, first at allocation row {r} "
                             f"(output row {r - GUARD_ROWS}), column {c}")


def report(family, ratio, label=""):
    print(f"WORST-RATIO {family}: {ratio:.3f} {label}")


# ======================================================================================================================
# A. attention
# ======================================================================================================================
# Error model, per output element o of row i (p_j = softmax weights, m = sum_j p_j |v_j|, |o^| <= m):
#   |o - o^| <= u |o^| + c u m + 2^-24
#   u |o^|        the rounding of the output to fp16.
#   c = cP + cP 2^-25 (sum_j |v_j| / l) / (u m) + (gamma + sigma) / u, computed per row:
#     cP          roundings of P to fp16 before the P V MMA.  The row sum l is accumulated from the fp32 values, so a
#                 relative rounding d_j of P_j moves the output by sum_j p_j d_j v_j, at most u m per rounding.
#                 v3 (tc_attn3.cu): 2 - P is rounded once by the cvt, and on the rescale path the P chunks already
#                 written are multiplied by 2^(old - new reference) in fp16 (__hmul2), a second rounding.
#                 v1 (tc_attention.cu): 1 - the row maximum is exact (resident S, or the two-pass stream), P is rounded
#                 once.  SIMT: 0 - P stays fp32.
#     cP 2^-25 sum_j |v_j| / l   P values below 2^-14 are fp16 subnormals with absolute (not relative) error 2^-25 per
#                 rounding; the kernels' row sums are >= the true l = sum_j 2^(s_j - max s) (their reference is at most
#                 the row maximum; the ragged tile's strip partials add up to l exactly).
#     gamma = (2 len + 16) 2^-24 + 2^-20   fp32 accumulation of the P V products and of the row sum (len terms each,
#                 up to one 2^-23 truncation per add in the tensor core), the rescales, the strip merge and the divide;
#                 2^-20 covers ex2.approx (relative error < 2^-22) in numerator and denominator.
#     sigma = 2 ln2 (hd + 2) 2^-23 max_j sum_d |q_d k_jd|   the fp32 score error (hd products, one truncation per add,
#                 plus the subtraction of the reference) moves every 2^(s_j - ref) by ln2 ds relatively, in the
#                 numerator and in the row sum.
#   2^-24         the output's own subnormal range.
ATT_CP = {"v3": 2.0, "v1": 1.0, "simt": 0.0}


def _attn_launch(lib, kernel, qkv, mode, B, S, C, N, heads):
    tokens = B * S * C
    buf, out = guarded(tokens, N, torch.float16)
    lib.vatss_debug_attention_version(1 if kernel == "v1" else 3)
    try:
        rc = lib.vatss_tc_attention(_p(qkv), _p(out), mode, B, S, C, N, heads, 1 if kernel == "simt" else 0, None)
    finally:
        lib.vatss_debug_attention_version(3)
    _check(rc, f"vatss_tc_attention {kernel}")
    torch.cuda.synchronize()
    assert_guard(buf, tokens, N, f"attention {kernel}")
    return out


def _seqs(x, mode, B, S, C):
    """(B, S, C, F) -> (G, len, F): intra sequences (b, s) over c, inter sequences (b, c) over s."""
    return x.reshape(B * S, C, -1) if mode == 0 else x.permute(0, 2, 1, 3).reshape(B * C, S, -1)


def _unseqs(y, mode, B, S, C):
    return y.reshape(B, S, C, -1) if mode == 0 else y.reshape(B, C, S, -1).permute(0, 2, 1, 3)


def attention_reference(qkv, mode, B, S, C, N, heads):
    """fp64: o^ = softmax_2(q k^T) v, the mass m and the per-row terms of the error model, all as (B, S, C, N)."""
    hd = N // heads
    seq = _seqs(qkv.double(), mode, B, S, C)
    G, L = seq.shape[0], seq.shape[1]
    q, k, v = (seq[..., i * N:(i + 1) * N].reshape(G, L, heads, hd).transpose(1, 2) for i in range(3))
    s = q @ k.transpose(-1, -2)
    p = torch.exp2(s - s.amax(-1, keepdim=True))
    l = p.sum(-1, keepdim=True)
    p = p / l
    o = p @ v
    m = p @ v.abs()
    smag = (q.abs() @ k.abs().transpose(-1, -2)).amax(-1, keepdim=True)     # max_j sum_d |q_d k_jd|
    sigma = 2 * math.log(2) * (hd + 2) * 2.0 ** -23 * smag
    gamma = (2 * L + 16) * 2.0 ** -24 + 2.0 ** -20
    sub = 2.0 ** -25 * v.abs().sum(-2, keepdim=True) / l                    # (G, h, L, hd)
    back = lambda t: _unseqs(t.expand(G, heads, L, hd).transpose(1, 2).reshape(G, L, N), mode, B, S, C)
    return back(o), back(m), back((gamma + sigma).expand(G, heads, L, 1)), back(sub)


def check_attention(out, ref, kernel, mode, B, S, C, N, label):
    """Per-element bound; returns the worst |err| / bound."""
    o_hat, m, gs, sub = ref
    cP = ATT_CP[kernel]
    got = out.reshape(B, S, C, N).double()
    bound = U16 * o_hat.abs() + cP * U16 * m + cP * sub + gs * m + 2.0 ** -24
    err = (got - o_hat).abs()
    ok = err <= bound                       # NaN (an element never written) fails
    if not bool(ok.all()):
        bad = (~ok).nonzero()
        b, s_, c, f = [int(t) for t in bad[0]]
        raise AssertionError(
            f"{label}: {bad.shape[0]} elements out of bound; first (b={b}, s={s_}, c={c}, feature {f}) got "
            f"{float(got[b, s_, c, f]):.6g} want "
            f"{float(o_hat[b, s_, c, f]):.6g} err {float(err[b, s_, c, f]):.3e} bound {float(bound[b, s_, c, f]):.3e}")
    return float((err / bound).max())


def attention_inputs(kind, mode, B, S, C, N, heads, seed):
    """fp16 qkv (B, S, C, 3N) on the device; q pre-scaled by log2(e)/sqrt(hd) as the in-projection leaves it.
    random:  q x2 for a peakier softmax.
    leak:    (intra) the keys of every other sequence ("hot": 0, 2, ...) score ~20 above the others for every query,
             so a key of a neighbouring sequence that leaks across the len boundary dominates its row.
    growing: key scale grows along the sequence (logits up to ~30): v3's rescale path.
    onehot:  one key per sequence scores ~30 above all others: near-one-hot rows.
    uniform: all keys equal: uniform rows, o = mean of v."""
    hd = N // heads
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, S, C, 3 * N, generator=g)
    x[..., :N] *= LOG2E / hd ** 0.5
    L = C if mode == 0 else S
    kv_shape = (1, 1, L, 1) if mode == 0 else (1, L, 1, 1)
    if kind == "random":
        x[..., :N] *= 2.0
    elif kind == "leak":
        assert mode == 0
        d = torch.ones(N) / hd ** 0.5                                # per head a unit direction
        a = math.sqrt(20.0)
        x[..., :N] += a * d
        hot = (torch.arange(B * S) % 2 == 0).reshape(B, S, 1, 1).float()
        x[..., N:2 * N] += hot * a * d
    elif kind == "growing":
        x[..., N:2 * N] *= torch.linspace(0.3, 6.0, L).reshape(kv_shape)
    elif kind == "onehot":
        d = torch.ones(N) / hd ** 0.5
        x[..., :N] = 0.3 * x[..., :N] + math.sqrt(30.0) * d
        pick = torch.zeros(L)
        pick[int(torch.randint(L, (1,), generator=g))] = 1.0
        x[..., N:2 * N] = 0.3 * x[..., N:2 * N] + pick.reshape(kv_shape) * math.sqrt(30.0) * d
    elif kind == "uniform":
        x[..., N:2 * N] = 0.5
    else:
        raise ValueError(kind)
    return x.half().to(DEV).contiguous()


def _attn_case(lib, kernel, kind, mode, B, S, C, N, heads, seed):
    qkv = attention_inputs(kind, mode, B, S, C, N, heads, seed)
    out = _attn_launch(lib, kernel, qkv, mode, B, S, C, N, heads)
    ref = attention_reference(qkv, mode, B, S, C, N, heads)
    label = f"attention {kernel} {kind} mode={mode} B={B} S={S} C={C} N={N} heads={heads}"
    return check_attention(out, ref, kernel, mode, B, S, C, N, label)


SWEEP_LENS = list(range(1, 201)) + [255, 256, 257, 258, 259, 260, 283, 287, 288, 289, 290, 383, 384, 385, 400, 577,
                                    710, 711]
# v1: resident S up to 3 kv blocks of 64 (len <= 192), resident K / V up to 5 (len <= 320), then streamed
SUBSET_LENS = [1, 2, 15, 16, 17, 31, 32, 33, 63, 64, 65, 96, 97, 127, 128, 129, 150, 160, 161, 191, 192, 193, 250, 283,
               320, 321, 400, 577, 710, 711]


def _sweep_shape(mode, L):
    return (1, 3, L) if mode == 0 else (1, L, 3)     # three sequences of length L


@pytest.mark.parametrize("mode", [0, 1], ids=["intra", "inter"])
@pytest.mark.parametrize("N,heads", LAYOUTS, ids=[f"N{n}-h{h}" for n, h in LAYOUTS])
@pytest.mark.parametrize("kernel", ["v3", "v1", "simt"])
def test_attention_length_sweep(lib, kernel, N, heads, mode):
    """v3 at every len 1-200 and the kv-block / query-tile boundaries above; v1 and SIMT on a subset that crosses
    their resident / streamed switches.  Intra inputs use the leak pattern (neighbouring sequences' keys ~20 hotter)."""
    lens = SWEEP_LENS if kernel == "v3" else SUBSET_LENS
    worst, at = 0.0, None
    with debug_reset(lib):
        for L in lens:
            B, S, C = _sweep_shape(mode, L)
            r = _attn_case(lib, kernel, "leak" if mode == 0 else "random", mode, B, S, C, N, heads, seed=L + N + heads)
            if r > worst:
                worst, at = r, L
    report(f"attention {kernel} N={N} heads={heads} {'intra' if mode == 0 else 'inter'} sweep", worst, f"(len {at})")


STRESS_SHAPES = [(0, 2, 3, 150), (0, 1, 2, 250), (1, 1, 283, 3), (1, 1, 710, 2)]


@pytest.mark.parametrize("kind", ["growing", "onehot", "uniform"])
@pytest.mark.parametrize("N,heads", LAYOUTS, ids=[f"N{n}-h{h}" for n, h in LAYOUTS])
@pytest.mark.parametrize("kernel", ["v3", "v1", "simt"])
def test_attention_stress_inputs(lib, kernel, N, heads, kind):
    worst = 0.0
    with debug_reset(lib):
        for mode, B, S, C in STRESS_SHAPES:
            worst = max(worst, _attn_case(lib, kernel, kind, mode, B, S, C, N, heads, seed=S + C + N + heads))
    report(f"attention {kernel} N={N} heads={heads} {kind}", worst)


SCHED_CASES = [
    # mode, B, S, C, N, heads: odd item counts (N = 64: one item per sequence) and a two-group layout
    (0, 1, 7, 150, 64, 2), (1, 1, 283, 5, 64, 4), (0, 1, 7, 129, 128, 8), (1, 1, 400, 3, 128, 4), (0, 3, 3, 33, 64, 4),
]


@pytest.mark.parametrize("kernel", ["v3", "v1"])
@pytest.mark.parametrize("mode,B,S,C,N,heads", SCHED_CASES)
def test_attention_schedule_independence(lib, kernel, mode, B, S, C, N, heads):
    """A persistent CTA walks items with its ring stage / phase carried across them: one, two or five CTAs must give
    the uncapped grid's output bit for bit."""
    qkv = attention_inputs("random", mode, B, S, C, N, heads, seed=S + C)
    with debug_reset(lib):
        want = _attn_launch(lib, kernel, qkv, mode, B, S, C, N, heads).clone()
        for cap in (1, 2, 5):
            lib.vatss_debug_cta_limit(cap)
            got = _attn_launch(lib, kernel, qkv, mode, B, S, C, N, heads)
            lib.vatss_debug_cta_limit(0)
            assert torch.equal(got.view(torch.int16), want.view(torch.int16)), f"{kernel} with {cap} CTAs"
    ref = attention_reference(qkv, mode, B, S, C, N, heads)
    check_attention(want, ref, kernel, mode, B, S, C, N, f"{kernel} schedule case")


# ======================================================================================================================
# B. LSTM
# ======================================================================================================================
# The reference is the kernel's own arithmetic in fp64: fp16 x and W (the plain kernel stores the i / f / o rows times
# 0.5, rounded to fp16 - restated exactly), fp32 b_ih + b_hh, h rounded to fp16 before it is fed back, output = that
# fp16 h (relu when act = 1).  What remains: fp32 accumulation, tanh.approx (relative error 2^-11: 2^-12 absolute on
# the 0.5 + 0.5 tanh(x / 2) sigmoids, 2^-11 on g and tanh(c)), and the fp16 rounding flips these cause.
# Per step the fresh error of h is <= 2^-12 (o) + 2^-11 (tanh c) + |o| dc with dc <= 2^-12 |c| + 2^-12 |g| + 2^-11 |i|
# + f dc_prev: with |c| <= ~2 that is ~4 2^-11 before rounding, plus one ulp (2^-11) when the two roundings of h land
# on different sides.  The forget gate (< 1) contracts the carried part and the W_hh feedback of random-sign errors
# averages out, so the bound is a constant, independent of the length: 8 u.
# PRECISE (hi/lo split, ex2 + rcp gates, ~1e-6): the fresh error is ~1e-6, and what is left is one rounding flip of
# the fp16 h (2^-11) and its small echo through W_hh: 2 u.
LSTM_BOUND = 8 * U16
LSTM_BOUND_PRECISE = 2 * U16
H = 128


def pick_inter_tile(C, B):
    """tc_lstm.cu pick_inter_tile: the (Kc chunk positions x Bc utterances) tile with the fewest tiles."""
    best, Kc, Bc = -1, 0, 0
    for k in range(1, min(128, C) + 1):
        b = min(128 // k, B)
        if b < 1:
            continue
        tiles = -(-C // k) * -(-B // b)
        if best < 0 or tiles < best or (tiles == best and k * b > Kc * Bc):
            best, Kc, Bc = tiles, k, b
    return Kc, Bc


def make_lstm(N, ndir, seed):
    """PyTorch-initialised weights (U(+-1/sqrt(H))), biases x3 so that a dropped bias is visible."""
    torch.manual_seed(seed)
    rnn = torch.nn.LSTM(N, H, batch_first=True, bidirectional=(ndir == 2))
    with torch.no_grad():
        for name, p in rnn.named_parameters():
            if name.startswith("bias"):
                p.mul_(3.0)
    sufs = ["", "_reverse"][:ndir]
    names = ["weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0"]
    return [[getattr(rnn, n + s).detach().to(DEV).float().contiguous() for n in names] for s in sufs]


def _run_lstm(lib, params, x16, xlo, mode, B, S, C, N, act, variant):
    ndir = len(params)
    keep = [t for d in params for t in d]
    table = (ctypes.c_void_p * 8)(*([t.data_ptr() for t in keep] + [None] * (8 - len(keep))))
    rows = B * S * C
    buf, out = guarded(rows, ndir * H, torch.float16)
    precise = xlo is not None
    wpack = torch.empty(ndir * 512 * ((2 * N if precise else N) + H), dtype=torch.float16, device=DEV)
    bpack = torch.empty(ndir * 512, dtype=torch.float32, device=DEV)
    pingpong, groups = variant
    lib.vatss_debug_lstm_pingpong(pingpong)
    lib.vatss_debug_lstm_groups(groups)
    try:
        rc = lib.vatss_tc_lstm(_p(x16), _p(xlo), table, _p(out), mode, B, S, C, N, ndir, act, _p(wpack), _p(bpack), None)
    finally:
        lib.vatss_debug_lstm_pingpong(1)
        lib.vatss_debug_lstm_groups(0)
    _check(rc, "vatss_tc_lstm")
    torch.cuda.synchronize()
    assert_guard(buf, rows, ndir * H, f"lstm variant {variant}")
    return out


def lstm_reference(params, x, mode, B, S, C, act, precise):
    """fp64 recurrence with the kernel's roundings; x: (B, S, C, N) fp64 (fp16 values, or fp32 for PRECISE)."""
    seq = _seqs(x, mode, B, S, C)                       # (G, L, N)
    G, L = seq.shape[0], seq.shape[1]
    outs = []
    gs = torch.ones(4 * H, dtype=torch.float64, device=DEV)
    if not precise:
        gs[:2 * H] = 0.5
        gs[3 * H:] = 0.5                                # i, f, o rows packed times 0.5 (gate order i, f, g, o)
    for d, (wih, whh, bih, bhh) in enumerate(params):
        if precise:
            Wih = wih.double()
            Whh = whh.half().double()
        else:
            Wih = (wih.double() * gs[:, None]).half().double() / gs[:, None]
            Whh = (whh.double() * gs[:, None]).half().double() / gs[:, None]
        b = (bih + bhh).double()                        # fp32 sum, then exact in fp64
        xw = seq @ Wih.t() + b                          # (G, L, 4H)
        h = torch.zeros(G, H, dtype=torch.float64, device=DEV)
        c = torch.zeros_like(h)
        y = torch.empty(G, L, H, dtype=torch.float64, device=DEV)
        for step in range(L):
            t = step if d == 0 else L - 1 - step
            a = xw[:, t] + h @ Whh.t()
            i_, f_, g_, o_ = a.split(H, dim=1)
            c = torch.sigmoid(f_) * c + torch.sigmoid(i_) * torch.tanh(g_)
            h = (torch.sigmoid(o_) * torch.tanh(c)).half().double()
            y[:, t] = h
        outs.append(y)
    y = torch.cat(outs, dim=-1)
    if act:
        y = torch.relu(y)
    return _unseqs(y, mode, B, S, C)                    # (B, S, C, ndir H)


def check_lstm(out, ref, mode, B, S, C, bound, label):
    got = out.reshape(B, S, C, -1).double()
    err = (got - ref).abs()
    ok = err <= bound
    if not bool(ok.all()):
        bad = (~ok).nonzero()
        b, s, c, f = [int(t) for t in bad[0]]
        raise AssertionError(f"{label}: {bad.shape[0]} elements over {bound:.2e}; first (b={b}, s={s}, c={c}, "
                             f"direction {f // H}, unit {f % H}) got {float(got[b, s, c, f]):.5f} "
                             f"want {float(ref[b, s, c, f]):.5f}")
    # worst error per step band (first / middle / last tenth of the direction's processing order)
    e = _seqs(err, mode, B, S, C)                       # (G, L, ndir H)
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
    return float(err.max()) / bound


LSTM_VARIANTS = [((1, 0), "half-tile auto"), ((1, 2), "half-tile 2 groups"), ((1, 3), "half-tile 3 groups"),
                 ((1, 4), "half-tile 4 groups"), ((0, 0), "one-tile")]

LSTM_INTRA = [
    # B, S (G = B S sequences), C, N, ndir, act:  G % 128 in {1, 63, 64, 65, 127}
    (1, 129, 150, 128, 2, 1), (1, 63, 250, 64, 2, 0), (2, 32, 150, 64, 2, 1), (1, 65, 250, 128, 2, 0),
    (1, 127, 150, 128, 1, 1),
]
LSTM_INTER = [
    # B, S, C, N, ndir, act
    (3, 1, 7, 128, 2, 1), (33, 2, 129, 64, 2, 0), (32, 53, 150, 128, 2, 1), (3, 283, 250, 64, 2, 0),
    (33, 710, 7, 128, 2, 1), (1, 53, 250, 128, 1, 0), (3, 283, 129, 128, 2, 0),
]


def _lstm_ids(cases, mode):
    ids = []
    for B, S, C, N, ndir, act in cases:
        if mode == 0:
            ids.append(f"G{B * S}-C{C}-N{N}-dir{ndir}-act{act}")
        else:
            kc, bc = pick_inter_tile(C, B)
            ids.append(f"B{B}-S{S}-C{C}-Kc{kc}-Bc{bc}-N{N}-dir{ndir}-act{act}")
    return ids


def _lstm_case(lib, mode, B, S, C, N, ndir, act, seed):
    params = make_lstm(N, ndir, seed)
    g = torch.Generator().manual_seed(seed)
    x16 = torch.randn(B, S, C, N, generator=g).half().to(DEV)
    ref = lstm_reference(params, x16.double(), mode, B, S, C, act, False)
    worst = {}
    with debug_reset(lib):
        for variant, name in LSTM_VARIANTS:
            out = _run_lstm(lib, params, x16, None, mode, B, S, C, N, act, variant)
            label = f"lstm {name} mode={mode} B={B} S={S} C={C} N={N} ndir={ndir} act={act}"
            worst[name] = check_lstm(out, ref, mode, B, S, C, LSTM_BOUND, label)
    for name, r in worst.items():
        report(f"lstm {name}", r, f"(mode={mode} B={B} S={S} C={C} N={N})")


@pytest.mark.parametrize("B,S,C,N,ndir,act", LSTM_INTRA, ids=_lstm_ids(LSTM_INTRA, 0))
def test_lstm_intra_matches_fp64_recurrence(lib, B, S, C, N, ndir, act):
    _lstm_case(lib, 0, B, S, C, N, ndir, act, seed=B * S + C + N)


@pytest.mark.parametrize("B,S,C,N,ndir,act", LSTM_INTER, ids=_lstm_ids(LSTM_INTER, 1))
def test_lstm_inter_matches_fp64_recurrence(lib, B, S, C, N, ndir, act):
    _lstm_case(lib, 1, B, S, C, N, ndir, act, seed=B + S + C + N)


@pytest.mark.parametrize("mode,B,S,C", [(0, 1, 65, 250), (0, 2, 64, 150), (1, 3, 283, 7), (1, 33, 53, 129)])
def test_lstm_hi_lo_split_matches_fp32_input_recurrence(lib, mode, B, S, C):
    """PRECISE (DPRNN, N = 64): fp32 x and W_ih through hi/lo fp16 splits; the reference keeps them fp32."""
    N, ndir = 64, 2
    params = make_lstm(N, ndir, seed=mode + S)
    g = torch.Generator().manual_seed(S + C)
    xf = (3.0 * torch.randn(B, S, C, N, generator=g)).to(DEV)
    hi = xf.half()
    lo = (xf - hi.float()).half()
    ref = lstm_reference(params, xf.double(), mode, B, S, C, 0, True)
    with debug_reset(lib):
        for variant, name in LSTM_VARIANTS:
            out = _run_lstm(lib, params, hi, lo, mode, B, S, C, N, 0, variant)
            r = check_lstm(out, ref, mode, B, S, C, LSTM_BOUND_PRECISE, f"lstm hi/lo {name} mode={mode} S={S} C={C}")
            report(f"lstm hi/lo {name}", r, f"(mode={mode} B={B} S={S} C={C})")


# ======================================================================================================================
# C. GEMM epilogues
# ======================================================================================================================
# fp16 outputs, per element: |o - o^| <= u |o^| + (K + 2) 2^-23 (|A| |W|^T + |bias|) + 2^-24 (output rounding;
# K fp32 accumulations with at most one 2^-23 truncation each; subnormals).  fp32 and LayerNorm rows: rel-L2 per row
# <= 1e-5 (~K 2^-24 worst case for K <= 256, times the LayerNorm's 1 / sigma gain on random rows).
GEMM_CASES = [
    # epi, NOUT, K, M:  M % 128 in {1, 127}
    (0, 384, 128, 129), (0, 192, 64, 1023), (1, 256, 128, 255), (1, 64, 64, 1153), (2, 128, 128, 641),
    (2, 64, 256, 383), (3, 128, 256, 897), (3, 64, 128, 129), ("ln16", 128, 128, 1407), ("ln16", 64, 64, 257),
]
EPI_NAME = {0: "fp16", 1: "fp32 + residual", 2: "LayerNorm(x + residual)", 3: "LayerNorm(x) + residual",
            "ln16": "LayerNorm(x + fp16 residual)"}


def _gemm_inputs(epi, NOUT, K, M):
    g = torch.Generator().manual_seed(M + NOUT + K)
    A = torch.randn(M, K, generator=g).half().to(DEV)
    W = (torch.randn(NOUT, K, generator=g) / K ** 0.5).half().to(DEV)
    bias = torch.randn(NOUT, generator=g).to(DEV)
    res = torch.randn(M, NOUT, generator=g).to(DEV)
    if epi == "ln16":
        res = res.half()
    lw = (1 + 0.2 * torch.randn(NOUT, generator=g)).to(DEV)
    lb = (0.1 * torch.randn(NOUT, generator=g)).to(DEV)
    return A, W, bias, res, lw, lb


def _run_gemm(lib, epi, NOUT, K, M, inputs, pitch):
    A, W, bias, res, lw, lb = inputs
    slope = torch.tensor([0.25], device=DEV)
    ld32, ld16 = (NOUT + 4, NOUT + 8) if pitch else (NOUT, NOUT)     # pitched rows stay 16-byte aligned
    b32, o32 = guarded(M, NOUT, torch.float32, ld32)
    b16, o16 = guarded(M, NOUT, torch.float16, ld16)
    p32 = None if epi == 0 else _p(o32)                 # each epilogue gets only the outputs it writes
    p16 = _p(o16) if epi in (0, 2, "ln16") else None
    if epi == "ln16":
        rc = lib.vatss_tc_gemm_ln16(_p(A), K, _p(W), _p(bias), _p(res), NOUT, _p(lw), _p(lb), p32, ld32, p16,
                                    ld16, 1, None, M, NOUT, K, None)
    else:
        act16 = 2 if epi == 2 else 0
        rc = lib.vatss_tc_gemm(epi, _p(A), K, _p(W), _p(bias), _p(res), NOUT, _p(lw), _p(lb), p32, ld32, p16,
                               ld16, act16, _p(slope), M, NOUT, K, None)
    _check(rc, f"gemm epi {epi}")
    torch.cuda.synchronize()
    return b32, o32, b16, o16


def _ln(x, w, b):
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + 1e-5) * w + b


def _rowwise_rel(got, want, label, tol=1e-5):
    e = (got.double() - want).norm(dim=1) / want.norm(dim=1)
    ok = e <= tol
    if not bool(ok.all()):
        r = int((~ok).nonzero()[0])
        raise AssertionError(f"{label}: {int((~ok).sum())} rows over rel-L2 {tol:.0e}; first row {r} of "
                             f"{want.shape[0]} ({float(e[r]):.3e})")
    return float(e.max()) / tol


@pytest.mark.parametrize("pitch", [False, True], ids=["dense", "pitched"])
@pytest.mark.parametrize("epi,NOUT,K,M", GEMM_CASES, ids=[f"epi{c[0]}-{c[1]}x{c[2]}-M{c[3]}" for c in GEMM_CASES])
def test_gemm_epilogue_rows(lib, epi, NOUT, K, M, pitch):
    inputs = _gemm_inputs(epi, NOUT, K, M)
    A, W, bias, res, lw, lb = inputs
    with debug_reset(lib):
        b32, o32, b16, o16 = _run_gemm(lib, epi, NOUT, K, M, inputs, pitch)
    label = f"gemm epi {epi} NOUT={NOUT} K={K} M={M}{' pitched' if pitch else ''}"
    base = A.double() @ W.double().t() + bias.double()
    mag = A.double().abs() @ W.double().abs().t() + bias.double().abs()
    if epi == 0:
        assert_guard(b16, M, NOUT, label + " out16")
        assert_guard(b32, 0, 0, label + " out32 (unused)")
        bound = U16 * base.abs() + (K + 2) * 2.0 ** -23 * mag + 2.0 ** -24
        err = (o16.double() - base).abs()
        ok = err <= bound
        if not bool(ok.all()):
            r, c = [int(t) for t in (~ok).nonzero()[0]]
            raise AssertionError(f"{label}: {int((~ok).sum())} elements out of bound; first row {r} col {c}")
        ratio = float((err / bound).max())
    else:
        assert_guard(b32, M, NOUT, label + " out32")
        if epi == 1:
            want = base + res.double()
        elif epi == 3:
            want = _ln(base, lw.double(), lb.double()) + res.double()
        else:
            want = _ln(base + res.double(), lw.double(), lb.double())
        ratio = _rowwise_rel(o32, want, label)
        if epi in (2, "ln16"):
            assert_guard(b16, M, NOUT, label + " out16")
            want16 = torch.where(want >= 0, want, 0.25 * want) if epi == 2 else torch.relu(want)
            # fp16 copy of the fp32 row: its rounding plus the fp32 row's own error (1e-5 of the row norm)
            bound = U16 * want16.abs() + 1e-5 * want.norm(dim=1, keepdim=True) + 2.0 ** -24
            assert bool(((o16.double() - want16).abs() <= bound).all()), label + " out16"
        else:
            assert_guard(b16, 0, 0, label + " out16 (unused)")
    report(f"gemm {EPI_NAME[epi]}", ratio, f"(NOUT={NOUT} K={K} M={M})")


@pytest.mark.parametrize("epi,NOUT,K,M", [(0, 384, 128, 1023), (1, 128, 128, 769), (2, 128, 256, 1153),
                                          (3, 64, 256, 639), ("ln16", 128, 128, 897)])
def test_gemm_schedule_independence(lib, epi, NOUT, K, M):
    """Grids capped at 1 and 3 CTAs (one CTA walks all row tiles, its accumulator slots and phases carried across
    them) must give the default grid's outputs bit for bit."""
    inputs = _gemm_inputs(epi, NOUT, K, M)
    with debug_reset(lib):
        _, w32, _, w16 = _run_gemm(lib, epi, NOUT, K, M, inputs, False)
        for cap in (1, 3):
            lib.vatss_debug_cta_limit(cap)
            _, g32, _, g16 = _run_gemm(lib, epi, NOUT, K, M, inputs, False)
            lib.vatss_debug_cta_limit(0)
            assert torch.equal(g32.view(torch.int32), w32.view(torch.int32)), f"fp32 output with {cap} CTAs"
            assert torch.equal(g16.view(torch.int16), w16.view(torch.int16)), f"fp16 output with {cap} CTAs"


# ======================================================================================================================
# D. whole forward at the head layouts the tests above add
# ======================================================================================================================
def _classes():
    import speech_separation_b200 as V

    return {"dptn_av": V.DPTNAVWavEncDec, "dptn_wav": V.DPTNWavEncDec, "dptn_mask": V.DPTNEncDec}


LARGE_BIAS = ("speakers_separation.1.bias", "postprocessing.0.bias", "output.0.bias", "output_gate.0.bias")


def make_net(kind, N, heads, K, C, P, bidir, seed):
    """Random weights as in test_gpu_tail_frontend.py: dense ~ 0.6 / sqrt(fan-in), LayerNorm affine 1 + 0.2 n /
    0.1 n, split and head biases ~ N(0, 1)."""
    kw = dict(num_features=N, kernel_size_enc=K, hidden_dim=128, num_blocks=1, chunk_size=C, step_size=P, bidir=bidir,
              num_heads=heads)
    if kind == "dptn_av":
        kw.update(video_emb_size=512, hidden_video=N)
    net = _classes()[kind](**kw).eval()
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in net.named_parameters():
            r = torch.randn(p.shape, generator=g, dtype=torch.float64)
            if name.endswith(LARGE_BIAS):
                v = r
            elif any(s in name for s in ("ln1.", "ln2.", "video_ln.")):
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


def check_waveforms(got, ref, tol, hop, label):
    """Per utterance and speaker: global rel-L2 <= tol and, for every hop-long window w, ||err_w|| <= 3 tol ||ref||
    sqrt(w / T) (test_gpu_tail_frontend.py's hop-wise check)."""
    worst = 0.0
    for spk, (g, r) in enumerate(zip(got, ref)):
        g = np.asarray(g, dtype=np.float64)
        r = np.asarray(r, dtype=np.float64)
        assert g.shape == r.shape and np.isfinite(g).all(), (label, spk)
        T = r.shape[1]
        for b in range(r.shape[0]):
            e, rn = g[b] - r[b], np.linalg.norm(r[b])
            rel = np.linalg.norm(e) / rn
            worst = max(worst, rel)
            assert rel <= tol, f"{label} spk{spk} utt{b}: rel-L2 {rel:.3e} > {tol:.0e}"
            for i0 in range(0, T, hop):
                w = min(hop, T - i0)
                bound = tol * rn * math.sqrt(w / T)
                ew = np.linalg.norm(e[i0:i0 + w])
                assert ew <= 3 * bound, f"{label} spk{spk} utt{b}: samples [{i0}, {i0 + w}) error {ew:.3e}"
    return worst


def _forward_case(kind, N, heads, bidir, engine, B=2, T=16000, Tv=25, K=16, C=100, P=50):
    net = make_net(kind, N, heads, K, C, P, bidir, seed=N + heads + int(bidir)).set_engine(engine)
    g = torch.Generator().manual_seed(heads + T)
    mix = torch.randn(B, T, generator=g)
    e1 = torch.randn(B, 512, Tv, generator=g) if kind == "dptn_av" else None
    e2 = torch.randn(B, 512, Tv, generator=g) if kind == "dptn_av" else None

    def run():
        with torch.no_grad():
            if e1 is None:
                out = net(mix=mix.to(DEV))
            else:
                out = net(mix=mix.to(DEV), s1_embedding=e1.to(DEV), s2_embedding=e2.to(DEV))
        return out["s1_pred"].cpu().numpy(), out["s2_pred"].cpu().numpy()

    cfg = O.PathConfig(kind=kind, num_features=N, kernel_size_enc=K, hidden_dim=128, num_blocks=1, chunk_size=C,
                       step_size=P, num_heads=heads, bidir=bidir, video_emb_size=512)
    ref = lambda: O.forward(O.to_numpy_state(net.state_dict(), np.float64), cfg, mix.double().numpy(),
                            None if e1 is None else e1.double().numpy(), None if e2 is None else e2.double().numpy())
    return net, run, ref, P * (K // 2)


FORWARD_LAYOUTS = [("dptn_av", 128, 8, True), ("dptn_av", 128, 8, False), ("dptn_wav", 64, 2, True),
                   ("dptn_mask", 64, 2, True)]


@pytest.mark.parametrize("engine", ["auto", "generic"])
@pytest.mark.parametrize("kind,N,heads,bidir", FORWARD_LAYOUTS,
                         ids=[f"{k}-N{n}-h{h}{'' if b else '-unidir'}" for k, n, h, b in FORWARD_LAYOUTS])
def test_forward_at_new_head_layouts(lib, kind, N, heads, bidir, engine):
    net, run, ref, hop = _forward_case(kind, N, heads, bidir, engine)
    with warnings.catch_warnings():
        warnings.simplefilter("error", RuntimeWarning)    # auto must not fall back
        got = run()
    if engine == "auto":
        assert lib.vatss_packed_weight_bytes(ctypes.byref(net._desc)) > 0, "auto did not select the tensor engine"
        # the forward does not depend on the persistent grids or on the GEMM's L2 order
        with debug_reset(lib):
            for cap, l2 in ((1, 1), (3, 0), (0, 0)):
                lib.vatss_debug_cta_limit(cap)
                lib.vatss_debug_gemm_l2_order(l2)
                again = run()
                assert all(np.array_equal(a, b) for a, b in zip(again, got)), f"cta cap {cap}, l2 order {l2}"
    label = f"{engine} {kind} N={N} heads={heads}{'' if bidir else ' unidir'}"
    err = check_waveforms(got, ref(), {"auto": 1e-3, "generic": 2e-4}[engine], hop, label)
    print(f"forward {label}: rel-L2 {err:.2e}")


@pytest.mark.parametrize("N,heads", [(128, 2), (64, 8)])
def test_forward_head_dims_off_the_tensor_engine_fall_back(lib, N, heads):
    net, run, ref, hop = _forward_case("dptn_wav", N, heads, True, "auto", T=8000)
    with pytest.warns(RuntimeWarning, match="head dim not in"):
        got = run()
    assert lib.vatss_packed_weight_bytes(ctypes.byref(net._desc)) == 0
    check_waveforms(got, ref(), 2e-4, hop, f"fallback N={N} heads={heads}")


@pytest.mark.parametrize("engine", ["auto", "generic"])
def test_forward_head_dim_128_is_an_error(lib, engine):
    """One head of 128 features: no kernel of either engine has head dim 128, so the forward must raise, naming it."""
    net, run, _, _ = _forward_case("dptn_wav", 128, 1, True, engine, T=8000)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        with pytest.raises(RuntimeError, match="head dim 128"):
            run()
