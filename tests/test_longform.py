"""Long recordings (`LongFormSeparator`, `vatss_window_cut`, `vatss_window_stitch`) against an fp64 numpy restatement
of the window geometry, the cut and the alignment + crossfade (`longform_windows`, `longform_cut`, `longform_stitch`
below; DESIGN.md §7).  No reference counterpart: the reference separates whole fixed-length clips."""
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle.gen_golden import PROD, TINY, make_inputs

KINDS = ["dptn_av", "dptn_wav", "dptn_mask", "dprnn"]
W, H = 16000, 12800     # 1 s windows, 0.2 s overlap (multiples of 640 samples): production models at test cost
O_ = W - H


def geometries(W, H, k=3):
    return [W - 1, W, W + 1, W + H, k * H + W, k * H + W + 1]


# ---------------------------------------------------------------------------------------------
# fp64 restatement (test infrastructure: the product package never uses it)
# ---------------------------------------------------------------------------------------------
def longform_windows(T, W, H):
    """Windows of [jH, jH + W) covering T samples: 1 if T <= W, else 1 + ceil((T - W) / H)."""
    if not (2 * H >= W and H < W):
        raise ValueError(f"hop {H} must satisfy W/2 <= hop < W (W={W})")
    return 1 if T <= W else 1 + -(-(T - W) // H)


def longform_cut(mix, W, H, emb1=None, emb2=None, spf=640):
    """mix (R,T) -> (R n, W), zero past T; emb (R,E,Tv) -> (R n, E, W/spf), frames past Tv repeat frame Tv-1."""
    mix = np.asarray(mix)
    R, T = mix.shape
    n = longform_windows(T, W, H)
    padded = np.zeros((R, (n - 1) * H + W), dtype=mix.dtype)
    padded[:, :T] = mix
    out = np.stack([padded[:, j * H:j * H + W] for j in range(n)], axis=1).reshape(R * n, W)
    if emb1 is None:
        return out
    Wv, Hv = W // spf, H // spf
    embs = []
    for e in (np.asarray(emb1), np.asarray(emb2)):
        Tv = e.shape[2]
        idx = np.minimum(np.arange(n)[:, None] * Hv + np.arange(Wv)[None, :], Tv - 1)   # (n, Wv)
        embs.append(e[:, :, idx].transpose(0, 2, 1, 3).reshape(R * n, e.shape[1], Wv))
    return out, embs[0], embs[1]


def longform_stitch(y1, y2, R, T, W, H):
    """Window outputs y1, y2 (R n, W) -> (s1, s2 (R,T), swaps (R, n-1) bool, sums (R, n-1, 8)).

    sums over the overlap of windows j (from offset H) and j+1 (from offset 0), all below T:
    [a1.b1, a1.b2, a2.b1, a2.b2, a1.a1, a2.a2, b1.b1, b2.b2]; swap when cos01 + cos10 > cos00 + cos11.
    Window j gives speaker s from row s ^ parity_j (prefix XOR of the swaps), so the output keeps window 0's order;
    overlaps are crossfaded with a = (i + 0.5) / O."""
    n = longform_windows(T, W, H)
    O = W - H
    y = np.stack([np.asarray(y1, np.float64), np.asarray(y2, np.float64)], 1).reshape(R, n, 2, W)
    sums = np.zeros((R, max(n - 1, 0), 8))
    for j in range(n - 1):
        a, b = y[:, j, :, H:], y[:, j + 1, :, :O]
        sums[:, j, :4] = np.einsum("rxi,ryi->rxy", a, b).reshape(R, 4)
        sums[:, j, 4:6] = (a * a).sum(-1)
        sums[:, j, 6:] = (b * b).sum(-1)

    def cos(c, ea, eb):
        ok = (ea > 0) & (eb > 0)
        return np.where(ok, c / np.sqrt(np.where(ok, ea * eb, 1.0)), 0.0)

    s = sums
    keep = cos(s[..., 0], s[..., 4], s[..., 6]) + cos(s[..., 3], s[..., 5], s[..., 7])
    swap = cos(s[..., 1], s[..., 4], s[..., 7]) + cos(s[..., 2], s[..., 5], s[..., 6])
    swaps = swap > keep
    parity = np.concatenate([np.zeros((R, 1), bool), np.logical_xor.accumulate(swaps, axis=1)], 1)
    aligned = np.where(parity[:, :, None, None], y[:, :, ::-1], y)       # (R, n, 2, W) in window 0's order
    out = np.zeros((R, 2, (n - 1) * H + W))
    alpha = (np.arange(O) + 0.5) / O
    for j in range(n):
        seg = aligned[:, j].copy()
        if j > 0:
            seg[..., :O] *= alpha
        if j < n - 1:
            seg[..., H:] *= 1.0 - alpha
        out[..., j * H:j * H + W] += seg
    return out[:, 0, :T], out[:, 1, :T], swaps, sums


# ---------------------------------------------------------------------------------------------
# CPU: the restatement itself
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("Wg,Hg", [(16000, 12000), (64000, 48000), (100, 50), (101, 99)])
def test_window_geometry(Wg, Hg):
    want = {Wg - 1: 1, Wg: 1, Wg + 1: 2, Wg + Hg: 2, 3 * Hg + Wg: 4, 3 * Hg + Wg + 1: 5}
    for T, n in want.items():
        assert longform_windows(T, Wg, Hg) == n
        # every sample in one or two windows, the last window reaches T, every overlap lies below T
        assert (n - 1) * Hg + Wg >= T
        if n > 1:
            assert (n - 2) * Hg + Wg < T
        cover = np.zeros(T, int)
        for j in range(n):
            cover[j * Hg:j * Hg + Wg] += 1
        assert cover.min() >= 1 and cover.max() <= 2
    for bad in (Wg // 2 - 1, Wg):
        with pytest.raises(ValueError):
            longform_windows(Wg + 5, Wg, bad)


def _planted(R, T, Wp, Hp, seed, noise_db=None):
    rng = np.random.default_rng(seed)
    s1, s2 = rng.standard_normal((R, T)), rng.standard_normal((R, T))
    y1, y2 = longform_cut(s1, Wp, Hp), longform_cut(s2, Wp, Hp)
    n = longform_windows(T, Wp, Hp)
    planted = rng.random((R, n)) < 0.5
    sw = planted.reshape(-1)
    y1[sw], y2[sw] = y2[sw].copy(), y1[sw].copy()
    if noise_db is not None:
        sigma = 10 ** (noise_db / 20)
        y1 = y1 + sigma * rng.standard_normal(y1.shape)
        y2 = y2 + sigma * rng.standard_normal(y2.shape)
    return s1, s2, y1, y2, planted


@pytest.mark.parametrize("T", [3 * 1200 + 1600, 3 * 1200 + 1601, 7777])
def test_oracle_recovers_planted_permutations(T):
    Wp, Hp, R = 1600, 1200, 3
    s1, s2, y1, y2, planted = _planted(R, T, Wp, Hp, seed=T)
    o1, o2, swaps, sums = longform_stitch(y1, y2, R, T, Wp, Hp)
    assert np.array_equal(swaps, planted[:, 1:] ^ planted[:, :-1])
    first = planted[:, :1]                       # the output keeps window 0's order
    assert np.abs(o1 - np.where(first, s2, s1)).max() < 1e-12
    assert np.abs(o2 - np.where(first, s1, s2)).max() < 1e-12
    assert sums.shape == (R, longform_windows(T, Wp, Hp) - 1, 8)
    # noise at -30 dB on every window: the decisions do not move
    _, _, y1n, y2n, planted_n = _planted(R, T, Wp, Hp, seed=T, noise_db=-30)
    assert np.array_equal(longform_stitch(y1n, y2n, R, T, Wp, Hp)[2], planted_n[:, 1:] ^ planted_n[:, :-1])


def test_oracle_cut_embeddings():
    R, E, Wp, Hp, spf = 2, 3, 1920, 1280, 640
    T = 4 * 1280 + 100
    Tv = -(-T // spf)
    rng = np.random.default_rng(0)
    mix, e = rng.standard_normal((R, T)), rng.standard_normal((R, E, Tv))
    x, c1, c2 = longform_cut(mix, Wp, Hp, e, -e, spf)
    n = longform_windows(T, Wp, Hp)
    assert x.shape == (R * n, Wp) and c1.shape == (R * n, E, Wp // spf)
    for r in range(R):
        for j in range(n):
            for f in range(Wp // spf):
                assert np.array_equal(c1[r * n + j, :, f], e[r, :, min(j * Hp // spf + f, Tv - 1)])
    assert np.array_equal(c2, -c1)


def test_argument_errors_cpu():
    import speech_separation_b200 as V

    net = V.DPTNWavEncDec(**PROD["dptn_wav"])
    for kw in (dict(window=16000, hop=7999), dict(window=16000, hop=16000), dict(max_batch=0),
               dict(window=400, hop=300)):           # (400 - 7) // 3 + 1 = 132 frames < one chunk of 150
        with pytest.raises(ValueError):
            V.LongFormSeparator(net, **kw)
    av = V.DPTNAVWavEncDec(**PROD["dptn_av"])
    for kw in (dict(window=16000, hop=12100), dict(window=16100, hop=12160), dict(samples_per_video_frame=0)):
        with pytest.raises(ValueError):
            V.LongFormSeparator(av, **kw)
    with pytest.raises(TypeError):
        V.LongFormSeparator(torch.nn.Linear(2, 2))
    lf = V.LongFormSeparator(net)
    with pytest.raises(RuntimeError, match="CUDA"):
        lf(torch.zeros(1, 200000))
    # the wrapper's state_dict is the model's, under the reference keys
    assert list(lf.state_dict()) == list(net.state_dict())


def test_micro_batches_are_near_equal():
    from speech_separation_b200.longform import micro_batches

    for total in (1, 5, 32, 33, 200, 1201):
        for mb in (1, 7, 32, 10 ** 6):
            b = micro_batches(total, mb)
            assert b[0][0] == 0 and sum(c for _, c in b) == total
            assert all(b[i][0] + b[i][1] == b[i + 1][0] for i in range(len(b) - 1))
            counts = [c for _, c in b]
            assert max(counts) <= mb and max(counts) - min(counts) <= 1 and counts == sorted(counts, reverse=True)


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


@pytest.fixture(scope="module")
def lib(V):
    from speech_separation_b200 import _lib

    return _lib.load()


def _cls(V, kind):
    return {"dptn_av": V.DPTNAVWavEncDec, "dptn_wav": V.DPTNWavEncDec, "dptn_mask": V.DPTNEncDec,
            "dprnn": V.DPRNNEncDec}[kind]


_NETS = {}


def prod_net(V, kind):
    if kind not in _NETS:
        torch.manual_seed(42)
        _NETS[kind] = _cls(V, kind)(**PROD[kind]).eval().to(dev())
    return _NETS[kind]


def inputs(kind, R, T, seed, E=512):
    """mix (R,T) and, for the AV model, embeddings with ceil(T / 640) frames, on the GPU."""
    mix, s1, s2, _, _ = make_inputs(R, T, seed=seed)
    if kind != "dptn_av":
        return mix.to(dev()), None, None
    g = torch.Generator().manual_seed(seed + 1)
    Tv = -(-T // 640)
    return mix.to(dev()), torch.randn(R, E, Tv, generator=g).to(dev()), torch.randn(R, E, Tv, generator=g).to(dev())


def stream():
    from speech_separation_b200 import _lib

    return _lib.stream_ptr()


@pytest.mark.gpu
@pytest.mark.parametrize("R", [1, 3])
def test_window_cut_bit_exact(V, lib, R):
    Wc, Hc, spf, E = 1920, 1280, 640, 24
    for T in geometries(Wc, Hc) + [4 * Hc + Wc - O_ // 8]:
        mix, e1, e2 = inputs("dptn_av", R, T, seed=T, E=E)
        n = longform_windows(T, Wc, Hc)
        want, w1, w2 = (torch.from_numpy(a) for a in longform_cut(mix.cpu().numpy(), Wc, Hc, e1.cpu().numpy(),
                                                                    e2.cpu().numpy(), spf))
        # the torch definition of the cut: pad, unfold; frames past Tv repeat the last one
        padded = torch.nn.functional.pad(mix.cpu(), (0, (n - 1) * Hc + Wc - T))
        assert torch.equal(want, padded.unfold(1, Wc, Hc).reshape(R * n, Wc))
        total = R * n
        for first, count in [(0, total), (total // 2, total - total // 2), (1, max(total - 2, 0)), (total - 1, 1)]:
            if count == 0:
                continue
            xo = torch.full((count, Wc), float("nan"), device=dev())
            o1 = torch.full((count, E, Wc // spf), float("nan"), device=dev())
            o2 = torch.full_like(o1, float("nan"))
            rc = lib.vatss_window_cut(mix.data_ptr(), e1.data_ptr(), e2.data_ptr(), R, T, e1.shape[2], E, Wc, Hc, spf,
                                      first, count, xo.data_ptr(), o1.data_ptr(), o2.data_ptr(), stream())
            assert rc == 0
            assert torch.equal(xo.cpu(), want[first:first + count])
            assert torch.equal(o1.cpu(), w1[first:first + count]) and torch.equal(o2.cpu(), w2[first:first + count])
            # audio only
            xa = torch.full((count, Wc), float("nan"), device=dev())
            assert lib.vatss_window_cut(mix.data_ptr(), None, None, R, T, 0, 0, Wc, Hc, 0, first, count, xa.data_ptr(),
                                        None, None, stream()) == 0
            assert torch.equal(xa.cpu(), want[first:first + count])
    assert lib.vatss_window_cut(mix.data_ptr(), None, None, R, T, 0, 0, Wc, Hc, 0, total, 1, xa.data_ptr(), None, None,
                                stream()) < 0
    assert lib.vatss_longform_windows(T, Wc, Wc // 2 - 1) < 0 and b"hop" in lib.vatss_last_error()


def _stitch(lib, y1, y2, R, T, Ws, Hs):
    n = longform_windows(T, Ws, Hs)
    s1 = torch.empty(R, T, device=dev())
    s2 = torch.empty_like(s1)
    sw = torch.empty(R, n - 1, dtype=torch.uint8, device=dev())
    corr = torch.empty(R, n - 1, 8, dtype=torch.float64, device=dev())
    nb = lib.vatss_window_stitch_scratch_bytes(R, n)
    scratch = torch.empty(nb, dtype=torch.uint8, device=dev())
    rc = lib.vatss_window_stitch(y1.data_ptr(), y2.data_ptr(), R, T, Ws, Hs, s1.data_ptr(), s2.data_ptr(),
                                 sw.data_ptr(), corr.data_ptr(), scratch.data_ptr(), nb, stream())
    assert rc == 0, lib.vatss_last_error()
    return s1, s2, sw, corr


def check_against_oracle(y1, y2, s1, s2, sw, corr, R, T, Ws, Hs):
    a1, a2 = y1.cpu().double().numpy(), y2.cpu().double().numpy()
    o1, o2, swaps, sums = longform_stitch(a1, a2, R, T, Ws, Hs)
    assert np.array_equal(sw.cpu().numpy().astype(bool), swaps)
    # the fp64 sums, to 1e-12 of the sum of the absolute products (the cross sums can cancel)
    n, Os = longform_windows(T, Ws, Hs), Ws - Hs
    ya = np.stack([np.abs(a1), np.abs(a2)], 1).reshape(R, n, 2, Ws)
    for j in range(n - 1):
        a, b = ya[:, j, :, Hs:], ya[:, j + 1, :, :Os]
        scale = np.concatenate([np.einsum("rxi,ryi->rxy", a, b).reshape(R, 4), (a * a).sum(-1), (b * b).sum(-1)], 1)
        assert (np.abs(corr.cpu().numpy()[:, j] - sums[:, j]) <= 1e-12 * scale + 1e-300).all()
    ymax = max(np.abs(a1).max(), np.abs(a2).max())
    g1, g2 = s1.cpu().double().numpy(), s2.cpu().double().numpy()
    assert np.abs(g1 - o1).max() <= 1e-6 * ymax and np.abs(g2 - o2).max() <= 1e-6 * ymax
    # per overlap region, so an error confined to one crossfade cannot hide in the aggregate
    for j in range(1, n):
        sl = slice(j * Hs, j * Hs + Os)
        for g, o in ((g1, o1), (g2, o2)):
            assert np.abs(g[:, sl] - o[:, sl]).max() <= 1e-6 * ymax, f"overlap {j}"
    return swaps


@pytest.mark.gpu
@pytest.mark.parametrize("R", [1, 3])
def test_window_stitch_against_oracle(V, lib, R):
    for T in geometries(W, H, k=5) + [40 * H + W + 7]:
        n = longform_windows(T, W, H)
        if n == 1:
            continue
        _, _, y1, y2, planted = _planted(R, T, W, H, seed=T + R, noise_db=-20)
        y1 = torch.from_numpy(y1).float().to(dev())
        y2 = torch.from_numpy(y2).float().to(dev())
        # a scale that differs per window: normalised correlation ignores it
        gain = torch.exp(torch.randn(R * n, 1, generator=torch.Generator().manual_seed(T))).to(dev())
        y1, y2 = (y1 * gain).contiguous(), (y2 * gain).contiguous()
        s1, s2, sw, corr = _stitch(lib, y1, y2, R, T, W, H)
        swaps = check_against_oracle(y1, y2, s1, s2, sw, corr, R, T, W, H)
        assert np.array_equal(swaps, planted[:, 1:] ^ planted[:, :-1])
        # bitwise reproducible
        t1, t2, tsw, tcorr = _stitch(lib, y1, y2, R, T, W, H)
        assert torch.equal(t1, s1) and torch.equal(t2, s2) and torch.equal(tsw, sw) and torch.equal(tcorr, corr)


def _call(lf, kind, mix, e1, e2, **kw):
    with torch.no_grad():
        if kind == "dptn_av":
            return lf(mix=mix, s1_embedding=e1, s2_embedding=e2, **kw)
        return lf(mix=mix, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_single_window_is_the_plain_forward(V, kind):
    net = prod_net(V, kind)
    lf = V.LongFormSeparator(net, window=W, hop=H)
    for T in (W - 1, W):
        mix, e1, e2 = inputs(kind, 2, T, seed=5)
        a = _call(lf, kind, mix, e1, e2)
        b = _call(net, kind, mix, e1, e2)
        assert torch.equal(a["s1_pred"], b["s1_pred"]) and torch.equal(a["s2_pred"], b["s2_pred"])


def plain_windows(net, kind, mix, e1, e2, Ws, Hs, max_batch, spf=640):
    """The wrapped model's forward on torch-cut windows, in the micro-batches LongFormSeparator uses."""
    from speech_separation_b200.longform import micro_batches

    R, T = mix.shape
    cut = longform_cut(mix.cpu().numpy(), Ws, Hs, *(() if e1 is None else (e1.cpu().numpy(), e2.cpu().numpy(), spf)))
    x, c1, c2 = (cut, None, None) if e1 is None else cut
    y1, y2 = [], []
    for first, count in micro_batches(x.shape[0], max_batch):
        sl = slice(first, first + count)
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a[sl])).to(dev())
        out = _call(net, kind, t(x), *((None, None) if e1 is None else (t(c1), t(c2))))
        y1.append(out["s1_pred"])
        y2.append(out["s2_pred"])
    return torch.cat(y1), torch.cat(y2)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("R", [1, 2])
def test_end_to_end_against_oracle(V, kind, R):
    net = prod_net(V, kind)
    lf = V.LongFormSeparator(net, window=W, hop=H, max_batch=7)
    for T in (W + 1, 3 * H + W - 5, 4 * H + W + 1):     # the last: a final window of O + 1 real samples
        mix, e1, e2 = inputs(kind, R, T, seed=T + R)
        out = _call(lf, kind, mix, e1, e2, return_alignment=True)
        y1, y2 = plain_windows(net, kind, mix, e1, e2, W, H, 7)
        check_against_oracle(y1, y2, out["s1_pred"], out["s2_pred"], out["swaps"], out["corr"], R, T, W, H)


@pytest.mark.gpu
def test_end_to_end_generic_engine_tiny(V):
    torch.manual_seed(0)
    net = V.DPTNAVWavEncDec(**TINY["dptn_av"]).eval().to(dev())
    net.set_engine("generic")
    Wt, Ht = 1920, 1280
    lf = V.LongFormSeparator(net, window=Wt, hop=Ht, max_batch=4)
    for R in (1, 2):
        T = 5 * Ht + Wt + 3
        mix, e1, e2 = inputs("dptn_av", R, T, seed=R, E=TINY["dptn_av"]["video_emb_size"])
        out = _call(lf, "dptn_av", mix, e1, e2, return_alignment=True)
        y1, y2 = plain_windows(net, "dptn_av", mix, e1, e2, Wt, Ht, 4)
        check_against_oracle(y1, y2, out["s1_pred"], out["s2_pred"], out["swaps"], out["corr"], R, T, Wt, Ht)


def decided(corr, eps=1e-6):
    """Pairs whose swap decision has a margin above eps: the only ones a 1e-5 change of the windows cannot flip."""
    s = corr.cpu().numpy()
    cos = lambda c, ea, eb: c / np.sqrt(ea * eb)
    margin = np.abs(cos(s[..., 1], s[..., 4], s[..., 7]) + cos(s[..., 2], s[..., 5], s[..., 6])
                    - cos(s[..., 0], s[..., 4], s[..., 6]) - cos(s[..., 3], s[..., 5], s[..., 7]))
    return margin > eps


def _rel_l2(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


@pytest.mark.gpu
def test_micro_batch_size_independence(V):
    kind = "dptn_av"
    net = prod_net(V, kind)
    R, T = 2, 9 * H + W + 100
    mix, e1, e2 = inputs(kind, R, T, seed=77)
    n = longform_windows(T, W, H)
    runs = {}
    for mb in (1, 7, R * n):
        lf = V.LongFormSeparator(net, window=W, hop=H, max_batch=mb)
        runs[mb] = _call(lf, kind, mix, e1, e2, return_alignment=True)
        again = _call(lf, kind, mix, e1, e2, return_alignment=True)
        for k in ("s1_pred", "s2_pred", "swaps", "corr"):
            assert torch.equal(again[k], runs[mb][k]), f"max_batch={mb}: repeated call differs in {k}"
    ref = runs[R * n]
    sure = decided(ref["corr"])
    for mb in (1, 7):
        assert np.array_equal(runs[mb]["swaps"].cpu().numpy()[sure], ref["swaps"].cpu().numpy()[sure])
        for k in ("s1_pred", "s2_pred"):
            assert _rel_l2(runs[mb][k], ref[k]) < 1e-5


@pytest.mark.gpu
def test_recordings_are_independent(V):
    kind = "dptn_wav"
    net = prod_net(V, kind)
    T = 6 * H + W + 321
    mix, _, _ = inputs(kind, 3, T, seed=8)
    n = longform_windows(T, W, H)
    lf = V.LongFormSeparator(net, window=W, hop=H, max_batch=3 * n)
    lf1 = V.LongFormSeparator(net, window=W, hop=H, max_batch=n)
    both = _call(lf, kind, mix, None, None, return_alignment=True)
    for r in range(3):
        one = _call(lf1, kind, mix[r:r + 1], None, None, return_alignment=True)
        sure = decided(one["corr"])
        assert np.array_equal(one["swaps"].cpu().numpy()[sure], both["swaps"][r:r + 1].cpu().numpy()[sure])
        for k in ("s1_pred", "s2_pred"):
            assert _rel_l2(one[k], both[k][r:r + 1]) < 1e-5


@pytest.mark.gpu
def test_no_host_sync(V):
    for kind in ("dptn_av", "dprnn"):
        lf = V.LongFormSeparator(prod_net(V, kind), window=W, hop=H, max_batch=6)   # micro-batches 6, 5, 5
        mix, e1, e2 = inputs(kind, 2, 7 * H + W + 9, seed=3)
        _call(lf, kind, mix, e1, e2)
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            out = _call(lf, kind, mix, e1, e2, return_alignment=True)
        finally:
            torch.cuda.set_sync_debug_mode("default")
        assert torch.isfinite(out["s1_pred"]).all()


@pytest.mark.gpu
def test_argument_errors_gpu(V):
    lf = V.LongFormSeparator(prod_net(V, "dptn_av"), window=W, hop=H)
    T = 3 * W
    mix, e1, e2 = inputs("dptn_av", 1, T, seed=1)
    with pytest.raises(ValueError, match="video frames"):
        lf(mix, e1[..., :-2], e2[..., :-2])
    with pytest.raises(ValueError):
        lf(mix, e1, None)
    with pytest.raises(ValueError):
        lf(mix[0], e1, e2)


@pytest.mark.gpu
def test_inferencer_with_long_recordings(V, tmp_path):
    from torch.utils.data import DataLoader

    torch.manual_seed(42)
    kw = dict(PROD["dptn_av"], num_blocks=2)
    net = V.DPTNAVWavEncDec(**kw).eval().to(dev())
    ckpt = tmp_path / "model_best.pth"
    torch.save({"state_dict": net.state_dict()}, ckpt)           # reference keys
    torch.manual_seed(7)
    lf = V.LongFormSeparator(V.DPTNAVWavEncDec(**kw).eval().to(dev()))   # other weights until the checkpoint loads
    T = 30 * 16000
    Tv = T // 640

    class Recordings(torch.utils.data.Dataset):
        def __len__(self):
            return 4

        def __getitem__(self, i):
            g = torch.Generator().manual_seed(100 + i)
            s1, s2 = 0.1 * torch.randn(T, generator=g), 0.1 * torch.randn(T, generator=g)
            return {"mix": s1 + s2, "s1": s1, "s2": s2, "s1_embedding": torch.randn(512, Tv, generator=g),
                    "s2_embedding": torch.randn(512, Tv, generator=g), "audio_path": f"/data/mix/rec_{i}.wav"}

    loader = DataLoader(Recordings(), batch_size=2)
    cfg = {"inferencer": {"device_tensors": ["mix", "s1", "s2", "s1_embedding", "s2_embedding"],
                          "from_pretrained": str(ckpt)}}
    mets = [V.SISNRiMetric(name="SISNRi")]
    inf = V.Inferencer(lf, cfg, dev(), {"test": loader}, tmp_path / "out", metrics={"inference": mets})
    logs = inf.run_inference()["test"]
    want = 0.0
    for b in loader:
        d = {k: (v.to(dev()) if torch.is_tensor(v) else v) for k, v in b.items()}
        d.update(_call(lf, "dptn_av", d["mix"], d["s1_embedding"], d["s2_embedding"]))
        want += float(mets[0](**d)) / len(loader)
        for i, p in enumerate(b["audio_path"]):
            rec = torch.load(tmp_path / "out" / "test" / f"{Path(p).stem}.pth")
            assert rec["s1_pred"].shape == (T,)
            assert torch.equal(rec["s1_pred"], d["s1_pred"][i].cpu())
            assert torch.equal(rec["s2_pred"], d["s2_pred"][i].cpu())
    assert logs["SISNRi"] == pytest.approx(want, abs=1e-4)
    # the checkpoint really replaced the wrapped model's weights
    d = {k: (v.to(dev()) if torch.is_tensor(v) else v) for k, v in next(iter(loader)).items()}
    a = _call(lf, "dptn_av", d["mix"], d["s1_embedding"], d["s2_embedding"])
    b = _call(V.LongFormSeparator(net), "dptn_av", d["mix"], d["s1_embedding"], d["s2_embedding"])
    assert torch.equal(a["s1_pred"], b["s1_pred"]) and torch.equal(a["s2_pred"], b["s2_pred"])
