"""The separator tail and the front end away from the reference's own configurations, against the fp64 oracle.

The production configurations all use chunk_size = 2 * step_size and kernel_size_enc in {2, 7}; the modules accept any
chunk geometry and kernel size, and engine="auto" runs the tensor engine for all of them.  These tests cover

  a. the tensor engine's tail on its own (vatss_tc_tail): the staged kernel (C = 2P), the gather kernel (any other
     non-masking geometry, up to 3 and 4 overlapping rows, no overlap, and the gap frames between chunks when
     step_size > chunk_size) and the unfused sequence (the masking head, or K outside {2, 7});
  b. the whole forward of both engines at those geometries, num_blocks = 0 and an unsupported kernel size;
  c. the encoder + AV fusion + segmentation (vatss_encoder) over widths, kernel sizes, lengths and video rates.

Every waveform comparison checks, per utterance and speaker, the global rel-L2 and a hop-wise bound (each window of one
hop, P * K/2 samples: ||err_w|| <= 3 tol ||ref|| sqrt(w / T)), so that an error confined to the centred pad, the first
or last hop or the gap frames cannot hide in the aggregate.  Weights are random (not the default initialisation), the
biases of the speaker split and of the heads are as large as the signal (a frame's split bias counts once per
overlapping chunk row), and the LayerNorm affine parameters are random too."""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import torch_port
from oracle import vatss_oracle as O

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


@pytest.fixture(scope="module")
def lib():
    assert torch.cuda.is_available()
    from speech_separation_b200 import _lib

    return _lib.load()


def _classes():
    import speech_separation_b200 as V

    return {"dptn_av": V.DPTNAVWavEncDec, "dptn_wav": V.DPTNWavEncDec, "dptn_mask": V.DPTNEncDec,
            "dprnn": V.DPRNNEncDec}


def _config(kind, N, K, C, P, num_blocks=1, bidir=True, E=512):
    kw = dict(num_features=N, kernel_size_enc=K, hidden_dim=128, num_blocks=num_blocks, chunk_size=C, step_size=P,
              bidir=bidir)
    if kind != "dprnn":
        kw.update(num_heads=4)
    if kind == "dptn_av":
        kw.update(video_emb_size=E, hidden_video=N)
    return kw


LARGE_BIAS = ("speakers_separation.1.bias", "postprocessing.0.bias", "output.0.bias", "output_gate.0.bias")


def make_net(kind, N, K, C, P, seed, num_blocks=1, bidir=True, E=512):
    """A module with random weights: dense weights ~ 0.6 / sqrt(fan-in), LayerNorm affine 1 + 0.2 n / 0.1 n, the
    split and head biases ~ N(0, 1) (the size of the signal they are added to)."""
    net = _classes()[kind](**_config(kind, N, K, C, P, num_blocks, bidir, E)).eval()
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in net.named_parameters():
            r = torch.randn(p.shape, generator=g, dtype=torch.float64)
            if name.endswith(LARGE_BIAS):
                v = r
            elif any(s in name for s in ("ln1.", "ln2.", "norm1d.", "video_ln.")):
                v = 1 + 0.2 * r if name.endswith("weight") else 0.1 * r
            elif name == "dprnn.speakers_separation.0.weight":
                v = 0.1 + 0.3 * r.abs()
            elif name == "gate":
                v = 0.5 + 0.5 * r.abs()
            elif name == "decoder.weight":
                v = 0.6 * r / math.sqrt(p.shape[0])
            elif p.dim() >= 2:
                v = 0.6 * r / math.sqrt(p[0].numel())
            else:
                v = 0.1 * r
            p.copy_(v)
    return net


def oracle_cfg(kind, N, K, C, P, num_blocks=1, bidir=True, E=512):
    return O.PathConfig(kind=kind, num_features=N, kernel_size_enc=K, hidden_dim=128, num_blocks=num_blocks,
                        chunk_size=C, step_size=P, num_heads=4, bidir=bidir, video_emb_size=E)


def check_waveforms(got, ref, tol, hop, label):
    """got, ref: sequences (speaker) of (B, T) arrays.  Global rel-L2 and the hop-wise bound, per utterance and speaker;
    returns the worst global error and the worst window ratio ||err_w|| / (tol ||ref|| sqrt(w / T))."""
    worst, worst_w = 0.0, 0.0
    for spk, (g, r) in enumerate(zip(got, ref)):
        g = np.asarray(g, dtype=np.float64)
        r = np.asarray(r, dtype=np.float64)
        assert g.shape == r.shape and np.isfinite(g).all(), (label, spk)
        T = r.shape[1]
        for b in range(r.shape[0]):
            e, rn = g[b] - r[b], np.linalg.norm(r[b])
            assert rn > 0
            rel = np.linalg.norm(e) / rn
            worst = max(worst, rel)
            assert rel <= tol, f"{label} spk{spk} utt{b}: rel-L2 {rel:.3e} > {tol:.0e}"
            for i0 in range(0, T, hop):
                w = min(hop, T - i0)
                ew = np.linalg.norm(e[i0:i0 + w])
                bound = tol * rn * math.sqrt(w / T)
                worst_w = max(worst_w, ew / bound)
                assert ew <= 3 * bound, (f"{label} spk{spk} utt{b}: samples [{i0}, {i0 + w}) error {ew:.3e} > "
                                         f"3 x {bound:.3e} (global rel-L2 {rel:.3e})")
    return worst, worst_w


def _lengths(C, P, K, shapes):
    """T for each (S, L - Lo): encoded length L = (S-1) P + C + (L - Lo); (T - K) % (K/2) = K/2 - 1."""
    st = K // 2
    out = []
    for S, r in shapes:
        L = (S - 1) * P + C + r
        T = (L - 1) * st + K + (st - 1)
        assert (T - K) // st + 1 == L and (L - C) // P + 1 == S
        out.append(T)
    return out


# ----------------------------------------------------------------------------------------------------------------------
# a. the tensor engine's tail on its own
# ----------------------------------------------------------------------------------------------------------------------
TAIL_CASES = [
    # kind, N, K, C, P, path
    ("dptn_wav", 64, 7, 150, 75, "staged + gather"),
    ("dptn_av", 128, 7, 150, 75, "staged + gather"),
    ("dprnn", 64, 2, 250, 125, "staged + gather"),
    ("dptn_av", 128, 2, 250, 125, "gather (staged ring over 200 KB)"),
    ("dptn_wav", 64, 7, 150, 50, "gather, 3 rows"),
    ("dptn_wav", 128, 7, 20, 7, "gather, 2-3 rows, C % P != 0"),
    ("dptn_wav", 64, 2, 64, 64, "gather, no overlap"),
    ("dptn_wav", 64, 7, 40, 60, "gather, gap frames"),
    ("dprnn", 64, 2, 30, 70, "gather, gap frames, P > 2C"),
    ("dptn_wav", 64, 4, 150, 75, "unfused"),
    ("dptn_av", 128, 16, 100, 50, "unfused"),
    ("dptn_mask", 64, 7, 150, 75, "unfused, masking"),
    ("dptn_mask", 128, 2, 40, 60, "unfused, masking, gap frames"),
]


def _unfused(kind, N, K):
    return kind == "dptn_mask" or K not in (2, 7) or N not in (64, 128)


def _run_tail(lib, net, x16, enc, T):
    from speech_separation_b200 import _lib

    B = x16.shape[0]
    net._prepare(DEV)
    d = net._desc
    ws = torch.empty(int(lib.vatss_workspace_bytes(ctypes.byref(d), B, T, 0)), dtype=torch.uint8, device=DEV)
    s1 = torch.full((B, T), float("nan"), device=DEV)
    s2 = torch.full((B, T), float("nan"), device=DEV)
    rc = lib.vatss_tc_tail(ctypes.byref(d), net._ptr_table, len(net._ptr_table), net._packed.data_ptr(),
                           x16.data_ptr(), enc.data_ptr(), B, T, s1.data_ptr(), s2.data_ptr(), ws.data_ptr(), ws.numel(),
                           _lib.stream_ptr())
    _lib.check(rc, "vatss_tc_tail")
    torch.cuda.synchronize()
    return s1.cpu().numpy(), s2.cpu().numpy()


def _tail_reference(net, cfg, x16, enc, T, unfused):
    """oracle.separator_tail + oracle.decode in fp64 on the fp16 input (PReLU slope 1: x16 is PReLU(x) already).  The
    unfused engine stores Wspk, the head / gate weights and the overlap-add in fp16: the reference rounds them too."""
    P = O.to_numpy_state(net.state_dict(), np.float64)
    P["dprnn.speakers_separation.0.weight"] = np.ones(1)
    r16 = lambda a: a.astype(np.float16).astype(np.float64)
    round_ola = None
    if unfused:
        for k in ("dprnn.speakers_separation.1.weight", "dprnn.postprocessing.0.weight", "dprnn.output.0.weight",
                  "dprnn.output_gate.0.weight"):
            if k in P:
                P[k] = r16(P[k])
        round_ola = r16
    us = O.separator_tail(x16.cpu().double().numpy(), enc.cpu().double().numpy(), P, cfg, round_ola=round_ola)
    return [O.decode(u, P["decoder.weight"], cfg.stride, T) for u in us]


def _tail_inputs(B, S, C, N, L, seed):
    g = torch.Generator().manual_seed(seed)
    x16 = torch.randn(B, S, C, N, generator=g).half().to(DEV)
    enc = torch.randn(B, L, N, generator=g).to(DEV)
    return x16, enc


@pytest.mark.parametrize("kind,N,K,C,P,path", TAIL_CASES, ids=[f"{c[0]}-N{c[1]}-K{c[2]}-C{c[3]}-P{c[4]}" for c in TAIL_CASES])
def test_tc_tail_matches_oracle(lib, kind, N, K, C, P, path):
    unfused = _unfused(kind, N, K)
    tol = 1e-4 if unfused else 1e-5
    net = make_net(kind, N, K, C, P, seed=N + K + C + P).to(DEV)
    cfg = oracle_cfg(kind, N, K, C, P)
    hop = P * (K // 2)
    # (S, L - Lo): one chunk; no centred pad; right-only pad; the largest pad
    shapes = [(1, P - 1), (7, 0), (12, 1), (5, P - 1)]
    try:
        for i, (T, B) in enumerate(zip(_lengths(C, P, K, shapes), (1, 3, 1, 3))):
            L = cfg.frames(T)
            S = cfg.chunks(L)
            x16, enc = _tail_inputs(B, S, C, N, L, seed=100 * i + N + K)
            ref = _tail_reference(net, cfg, x16, enc, T, unfused)
            got = _run_tail(lib, net, x16, enc, T)
            err, win = check_waveforms(got, ref, tol, hop, f"{kind} N={N} K={K} C={C} P={P} T={T} B={B}")
            print(f"tc_tail {path:34s} {kind} N={N} K={K} C={C} P={P} B={B} T={T} (S={S}, L-Lo={L - (S - 1) * P - C}):"
                  f" rel-L2 {err:.2e}, worst hop {win:.2f} x tol")
            if C == 2 * P:
                lib.vatss_debug_tail_staged(0)
                gather = _run_tail(lib, net, x16, enc, T)
                lib.vatss_debug_tail_staged(1)
                for a, b_ in zip(got, gather):
                    assert np.array_equal(a, b_), f"staged and gather tails differ at T={T} B={B}"
    finally:
        lib.vatss_debug_tail_staged(1)


def test_tc_tail_large_batch_wraps_the_staged_ring(lib):
    """24 utterances of 4 s at the reference's 150 / 75: 24 x 286 work units, the staged kernel's grid of one CTA per
    SM walks its two-stage ring many times."""
    kind, N, K, C, P, B, T = "dptn_wav", 64, 7, 150, 75, 24, 64000
    net = make_net(kind, N, K, C, P, seed=5).to(DEV)
    cfg = oracle_cfg(kind, N, K, C, P)
    L = cfg.frames(T)
    S = cfg.chunks(L)
    x16, enc = _tail_inputs(B, S, C, N, L, seed=6)
    ref = _tail_reference(net, cfg, x16, enc, T, False)
    try:
        got = _run_tail(lib, net, x16, enc, T)
        lib.vatss_debug_tail_staged(0)
        gather = _run_tail(lib, net, x16, enc, T)
    finally:
        lib.vatss_debug_tail_staged(1)
    err, win = check_waveforms(got, ref, 1e-5, P * (K // 2), "large batch")
    print(f"tc_tail large batch B={B} T={T} S={S}: rel-L2 {err:.2e}, worst hop {win:.2f} x tol")
    for a, b_ in zip(got, gather):
        assert np.array_equal(a, b_)


def test_tc_tail_rejects_a_model_off_the_tensor_engine(lib):
    from speech_separation_b200 import _lib

    net = make_net("dptn_wav", 64, 7, 150, 75, seed=1).to(DEV)
    net._prepare(DEV)
    d = _lib.ModelDesc.from_buffer_copy(net._desc)
    d.engine = _lib.ENGINE["generic"]
    rc = lib.vatss_tc_tail(ctypes.byref(d), net._ptr_table, len(net._ptr_table), net._packed.data_ptr(), None, None, 1,
                           16000, None, None, None, 0, None)
    assert rc != 0 and b"TENSOR engine" in lib.vatss_last_error()


# ----------------------------------------------------------------------------------------------------------------------
# b. the whole forward, both engines
# ----------------------------------------------------------------------------------------------------------------------
FORWARD_CASES = [
    # kind, N, K, C, P, bidir, B, T, Tv
    ("dptn_av", 128, 16, 100, 50, True, 2, 24011, 37),
    ("dptn_wav", 64, 4, 150, 50, True, 2, 16001, 0),
    ("dptn_mask", 64, 7, 64, 64, True, 2, 16000, 0),
    ("dptn_wav", 64, 7, 40, 60, True, 2, 16000, 0),       # gap frames
    ("dprnn", 64, 2, 30, 45, True, 2, 8000, 0),           # gap frames
    ("dprnn", 64, 2, 100, 30, True, 2, 8000, 0),          # 4 rows per frame
    ("dptn_av", 128, 7, 20, 7, False, 2, 8000, 13),
]
TOL = {"auto": 1e-3, "generic": 2e-4}


def _inputs(kind, B, T, Tv, E, seed):
    g = torch.Generator().manual_seed(seed)
    mix = torch.randn(B, T, generator=g)
    e1 = torch.randn(B, E, Tv, generator=g) if kind == "dptn_av" else None
    e2 = torch.randn(B, E, Tv, generator=g) if kind == "dptn_av" else None
    return mix, e1, e2


def _forward(net, mix, e1, e2):
    with torch.no_grad():
        if e1 is None:
            out = net(mix=mix.to(DEV))
        else:
            out = net(mix=mix.to(DEV), s1_embedding=e1.to(DEV), s2_embedding=e2.to(DEV))
    return out["s1_pred"].cpu().numpy(), out["s2_pred"].cpu().numpy()


@pytest.mark.parametrize("engine", ["auto", "generic"])
@pytest.mark.parametrize("kind,N,K,C,P,bidir,B,T,Tv", FORWARD_CASES,
                         ids=[f"{c[0]}-N{c[1]}-K{c[2]}-C{c[3]}-P{c[4]}{'' if c[5] else '-unidir'}" for c in FORWARD_CASES])
def test_forward_matches_oracle(kind, N, K, C, P, bidir, B, T, Tv, engine):
    net = make_net(kind, N, K, C, P, seed=N + K + C + P, bidir=bidir).to(DEV).set_engine(engine)
    cfg = oracle_cfg(kind, N, K, C, P, bidir=bidir)
    mix, e1, e2 = _inputs(kind, B, T, Tv, 512, seed=K + C)
    got = _forward(net, mix, e1, e2)
    Pd = O.to_numpy_state(net.state_dict(), np.float64)
    ref = O.forward(Pd, cfg, mix.double().numpy(), None if e1 is None else e1.double().numpy(),
                    None if e2 is None else e2.double().numpy())
    label = f"{engine} {kind} N={N} K={K} C={C} P={P}"
    err, win = check_waveforms(got, ref, TOL[engine], P * (K // 2), label)
    print(f"forward {label}: rel-L2 {err:.2e}, worst hop {win:.2f} x tol")
    if P > C:
        # the gap frames' semantics from the reference's own ops: F.unfold / F.fold on a float64 copy of the module
        net64 = _classes()[kind](**_config(kind, N, K, C, P, 1, bidir)).eval()
        net64.load_state_dict({k: v.cpu() for k, v in net.state_dict().items()})
        net64 = net64.double()
        tp = torch_port.forward(net64, mix.double(), None if e1 is None else e1.double(),
                                None if e2 is None else e2.double())
        tp = [tp["s1_pred"].numpy(), tp["s2_pred"].numpy()]
        for a, b_ in zip(tp, ref):
            assert np.linalg.norm(a - b_) <= 1e-9 * np.linalg.norm(b_)
        check_waveforms(got, tp, TOL[engine], P * (K // 2), label + " vs torch_port")


@pytest.mark.parametrize("kind", ["dptn_av", "dptn_wav", "dptn_mask", "dprnn"])
def test_forward_without_blocks_falls_back_to_generic(kind):
    """num_blocks = 0 (an empty nn.Sequential in the reference): the tensor engine has no block epilogue to take
    PReLU(x) from, so AUTO must fall back to the generic engine with the usual warning and still be exact."""
    N, K, C, P, B, T, Tv = 64, 7, 150, 75, 2, 8000, 9
    net = make_net(kind, N, K, C, P, seed=3, num_blocks=0).to(DEV)
    mix, e1, e2 = _inputs(kind, B, T, Tv, 512, seed=4)
    with pytest.warns(RuntimeWarning, match="no dual-path blocks"):
        got = _forward(net, mix, e1, e2)
    Pd = O.to_numpy_state(net.state_dict(), np.float64)
    ref = O.forward(Pd, oracle_cfg(kind, N, K, C, P, num_blocks=0), mix.double().numpy(),
                    None if e1 is None else e1.double().numpy(), None if e2 is None else e2.double().numpy())
    err, win = check_waveforms(got, ref, 1e-5, P * (K // 2), f"num_blocks=0 {kind}")
    print(f"forward num_blocks=0 {kind}: rel-L2 {err:.2e}, worst hop {win:.2f} x tol")


@pytest.mark.parametrize("engine", ["auto", "generic"])
def test_kernel_size_above_the_decoder_limit_is_rejected(engine):
    net = make_net("dptn_wav", 64, 18, 100, 50, seed=2).to(DEV).set_engine(engine)
    with pytest.raises(RuntimeError, match="kernel_size_enc 18 > 16"):
        _forward(net, torch.randn(1, 8000), None, None)


# ----------------------------------------------------------------------------------------------------------------------
# c. front end: encoder + AV fusion + token-major segmentation
# ----------------------------------------------------------------------------------------------------------------------
FRONT_CASES = [
    # kind, N, K, C, P, B, T, E, Tv   (Tv as an expression of T and L)
    ("dptn_wav", 16, 7, 20, 7, 1, 100, 0, None),              # scalar kernel, L = 32 < 64
    ("dptn_wav", 96, 2, 64, 64, 3, 5000, 0, None),            # scalar kernel, L = 4999
    ("dptn_wav", 256, 16, 100, 30, 1, 16000, 0, None),        # scalar kernel at its widest, 4 rows
    ("dptn_wav", 64, 4, 40, 60, 3, 3001, 0, None),            # vec<2>, gap frames
    ("dptn_wav", 128, 7, 150, 50, 1, 9000, 0, None),          # vec<4>, 3 rows
    ("dprnn", 64, 2, 30, 70, 3, 1000, 0, None),               # gap frames, P > 2C
    ("dptn_av", 16, 2, 20, 7, 1, 50, 24, "1"),               # N/2 = 8 outputs, E < 32, one video frame, L < 64
    ("dptn_av", 16, 7, 40, 60, 3, 4000, 1000, "2"),
    ("dptn_av", 64, 4, 150, 75, 3, 16000, 24, "25T"),
    ("dptn_av", 64, 7, 150, 50, 1, 7001, 512, "L-1"),
    ("dptn_av", 96, 16, 64, 64, 3, 3333, 1000, "L"),
    ("dptn_av", 96, 7, 30, 70, 1, 2222, 512, "2L+1"),
    ("dptn_av", 128, 2, 250, 125, 3, 16000, 1000, "25T"),
    ("dptn_av", 128, 7, 20, 7, 1, 1000, 24, "2L+1"),
    ("dptn_av", 128, 16, 100, 50, 3, 24011, 512, "L-1"),
    ("dptn_av", 256, 7, 150, 75, 1, 16000, 512, "25T"),
    ("dptn_av", 256, 4, 100, 30, 3, 2000, 24, "L"),
    ("dptn_av", 128, 4, 150, 75, 1, 16000, 512, "1"),
]


def _tv(spec, T, L):
    return {"1": 1, "2": 2, "25T": max(1, 25 * T // 16000), "L-1": L - 1, "L": L, "2L+1": 2 * L + 1}[spec]


def _fp32_source_index(L, Tv):
    """F.interpolate(linear, align_corners=False) source indices as float32 arithmetic computes them on the GPU, where
    scale * (l + 0.5) - 0.5 is one fused multiply-add (one rounding).  A source index of a few thousand carries an
    fp32 rounding of up to 1.2e-4 - as much as the interpolation weight itself moves - so the fp64 reference takes
    the float32 indices, and everything downstream of them is compared in fp64."""
    scale = np.float64(np.float32(Tv) / np.float32(L))
    src = (scale * (np.arange(L) + 0.5) - 0.5).astype(np.float32)   # exact in fp64, then the single fp32 rounding
    src = np.maximum(src, np.float32(0))
    i0 = np.minimum(np.floor(src).astype(np.int64), Tv - 1)
    i1 = np.minimum(i0 + 1, Tv - 1)
    return i0, i1, (src - i0.astype(np.float32)).astype(np.float64)


def _front_params(kind, N, K, E, seed):
    """Host table of the global parameter slots vatss_encoder reads (the rest NULL) and the fp64 oracle state."""
    from speech_separation_b200 import _lib

    g = torch.Generator().manual_seed(seed)
    p = {"encoder.weight": torch.randn(N, 1, K, generator=g) / math.sqrt(K)}
    if kind == "dptn_av":
        p["visual_compression.weight"] = torch.randn(N // 2, E, generator=g) / math.sqrt(E)
        p["visual_compression.bias"] = 0.5 * torch.randn(N // 2, generator=g)
        p["gate"] = torch.tensor([0.8])
        p["video_ln.weight"] = 1 + 0.2 * torch.randn(N, generator=g)
        p["video_ln.bias"] = 0.1 * torch.randn(N, generator=g)
    dev = {k: v.to(DEV).contiguous() for k, v in p.items()}
    table = (ctypes.c_void_p * len(_lib.P_GLOBAL))()
    for i, name in enumerate(_lib.P_GLOBAL):
        table[i] = dev[name].data_ptr() if name in dev else None
    return table, dev, {k: v.double().numpy() for k, v in p.items()}


@pytest.mark.parametrize("kind,N,K,C,P,B,T,E,tv", FRONT_CASES,
                         ids=[f"{c[0]}-N{c[1]}-K{c[2]}-C{c[3]}-P{c[4]}-B{c[5]}-T{c[6]}" + (f"-E{c[7]}-Tv{c[8]}" if c[8] else "")
                              for c in FRONT_CASES])
def test_encoder_matches_oracle(lib, kind, N, K, C, P, B, T, E, tv):
    from speech_separation_b200 import _lib

    cfg = oracle_cfg(kind, N, K, C, P, E=E or 512)
    L = cfg.frames(T)
    S = cfg.chunks(L)
    Tv = _tv(tv, T, L) if tv else 0
    d = _lib.ModelDesc(kind=_lib.KIND[kind], N=N, K=K, H=128, num_blocks=0, C=C, P=P, heads=4, bidir=1, E=E or 0,
                       engine=0)
    table, keep, Pd = _front_params(kind, N, K, E, seed=N + K + T)
    g = torch.Generator().manual_seed(T + Tv)
    mix = torch.randn(B, T, generator=g)
    e1 = torch.randn(B, E, Tv, generator=g) if Tv else None
    e2 = torch.randn(B, E, Tv, generator=g) if Tv else None
    md = mix.to(DEV)
    e1d = e1.to(DEV) if Tv else None
    e2d = e2.to(DEV) if Tv else None
    enc = torch.full((B, L, N), float("nan"), device=DEV)
    seg = torch.full((B, S, C, N), float("nan"), device=DEV)
    vis = torch.empty(max(B * Tv * N, 1), device=DEV)
    rc = lib.vatss_encoder(ctypes.byref(d), table, md.data_ptr(), e1d.data_ptr() if Tv else None,
                           e2d.data_ptr() if Tv else None, B, T, Tv, enc.data_ptr(), seg.data_ptr(), vis.data_ptr(),
                           _lib.stream_ptr())
    _lib.check(rc, "vatss_encoder")
    torch.cuda.synchronize()
    got = enc.cpu().double().numpy()
    ref = O.encode(mix.double().numpy(), Pd["encoder.weight"], cfg.stride)
    if Tv:
        ref = O.av_fuse(ref, e1.double().numpy(), e2.double().numpy(), Pd, index=_fp32_source_index(L, Tv))
    err = np.linalg.norm(got - ref) / np.linalg.norm(ref)
    mx = np.abs(got - ref).max() / np.abs(ref).max()
    print(f"encoder {kind} N={N} K={K} B={B} T={T} L={L} E={E} Tv={Tv}: rel-L2 {err:.2e}, max {mx:.2e} of max|ref|")
    assert err <= 1e-5 and mx <= 1e-5
    want = torch.from_numpy(O.segment_token_major(enc.cpu().numpy(), C, P))
    assert torch.equal(seg.cpu(), want), "segmentation is not an exact copy of the encoder output"


def test_encoder_rejects_more_than_256_features(lib):
    from speech_separation_b200 import _lib

    N, K, B, T = 260, 7, 1, 4000
    d = _lib.ModelDesc(kind=_lib.KIND["dptn_wav"], N=N, K=K, H=128, num_blocks=0, C=150, P=75, heads=4, bidir=1, E=0,
                       engine=0)
    table, keep, _ = _front_params("dptn_wav", N, K, 0, seed=0)
    L = (T - K) // (K // 2) + 1
    mix = torch.randn(B, T, device=DEV)
    enc = torch.empty(B, L, N, device=DEV)
    rc = lib.vatss_encoder(ctypes.byref(d), table, mix.data_ptr(), None, None, B, T, 0, enc.data_ptr(), None, None,
                           _lib.stream_ptr())
    assert rc != 0 and b"num_features 260 > 256" in lib.vatss_last_error()
