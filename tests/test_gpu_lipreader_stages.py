"""The lipreader kernels stage by stage against fp64 references: the front end, both max pools, every trunk convolution,
shortcut and residual block, and the average pool, on both engines.

test_lipreader.py checks one rel-L2 over the final (B, T, 512) features, which an error confined to the image border,
one tap, the ragged last 128-row tile of one convolution or the last frame of an utterance hides under: the features
are an average pool after 17 convolutions and a max pool.  Here `vatss_debug_lipreader_capture` copies every stage the
forward writes (same buffers, rotation and chunking as production) into guarded buffers, and each stage is checked per
element against an fp64 reference computed from the *captured input of that stage*, so errors do not compound and every
bound is an error model of one kernel.

References are computed in float64 with torch on the device (explicit im2col + matmul: no cuDNN algorithm choice) and
never go through the library.  Every debug switch is reset in a `finally`."""
import contextlib
import ctypes
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as Fn

from oracle import lipreader_oracle as LO

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")]

DEV = torch.device("cuda:0")
U32 = 2.0 ** -24          # unit roundoff of fp32
U16 = 2.0 ** -11          # unit roundoff of fp16
NSTAGES = 26
CHUNK = 1024              # frames per pass through the trunk (LIP_CHUNK)
GUARD_ROWS = 4            # whole sentinel frames before and after every capture / output view
SENTINEL = {torch.float16: (torch.int16, 0x7E5A), torch.float32: (torch.int32, 0x7FC05A5A)}   # NaN bit patterns
WS_TAIL = 1 << 16         # sentinel bytes after the workspace the library asked for
F32_TOL, TENSOR_TOL = 2e-5, 2e-3   # test_lipreader.py's whole-forward tolerances, here per frame
ACT = {"relu": 1, "prelu": 2, "swish": 3}

# ======================================================================================================================
# Error model.  A convolution stage computes, per output element,
#     y = act(z),   z = acc * s + h (+ r),   acc = sum_k x_k w_k
# with s, h the BatchNorm folded into a per-channel scale / shift, r the residual (block output only).  The reference
# y^ = act(z^) is fp64 from the kernel's own operands: the captured input (fp32, or fp16 under the tensor engine), the
# weights as the packing kernels round them (fp32, or fp16 RN), the captured residual, and s, h folded in fp64 from the
# fp32 BatchNorm tensors.  Then
#     |y - y^| <= L_act E_z + r_act |y^|            (fp32 output)
#     |y - y^| <= (1 + u16) (L_act E_z + r_act |y^|) + u16 |y^| + 2^-25     (fp16 output: RN, subnormal half-ulp)
#     E_z = |s| c_K M + 2^-22 (|acc^ s| + |mean s| + |h|) + u32 |acc^ s + h| (+ u32 |z^| with a residual)
#   M = sum_k |x_k| |w_k| (fp64), c_K the accumulation error:
#     fp32 engine: one FMA chain of K terms (k_lip_front3d: K = 245; k_lip_conv_f32: K = 9 Cin, or Cin for the 1x1
#                  shortcut), gamma_K = K u32 / (1 - K u32).
#     tensor engine: fp16 x fp16 products are exact in fp32; the tensor core adds them in fp32 with at most one 2^-23
#                  truncation per add, c_K = (K + 2) 2^-23 (K = 256 for the front-end GEMM, whose taps 245 - 255 are
#                  zero columns; 9 Cin or Cin in the trunk).
#   2^-22 (...)   k_lip_fold_bn folds in fp32: s = g / sqrtf(var + eps) is three roundings (< 2^-22 relative), and
#                 h = b - mean s inherits it through mean s plus its own two roundings.
#   u32 |...|     the fmaf of the epilogue, and the fp32 residual add.
#   L_act         Lipschitz constant of the activation: 1 for relu / prelu (slopes < 1) / none, 1.1 for swish
#                 (max of x sigmoid(x)' is 1.0998).
#   r_act         the activation's own arithmetic, relative to |y^|: relu 0; prelu u32 (v * slope); swish on the fp32
#                 engine 8 u32 (expf within 2 ulp, 1 + e, the IEEE divide, the product); swish on the tensor engine
#                 (|v| + 8) u32 with v = z^: __expf(-v) = ex2.approx(-v log2 e) - the product's rounding is a relative
#                 error |v| u32 of e, ex2.approx < 2^-22 - then 1 + e and __fdividef (rcp.approx + product).
# Max pools are exact (a max of stored values), so the check is bit for bit (values; the sign of a zero is not checked).
# Average pool: HW fp32 adds and one divide, (HW + 1) u32 mean |x| per (frame, channel).
# ======================================================================================================================
L_ACT = {"relu": 1.0, "prelu": 1.0, "swish": 1.1, None: 1.0}


def r_act(relu_type, engine, z):
    if relu_type is None or relu_type == "relu":
        return 0.0
    if relu_type == "prelu":
        return U32
    return 8 * U32 if engine == "f32" else (z.abs() + 8) * U32


@pytest.fixture(scope="module")
def lib():
    from speech_separation_b200 import _lib

    return _lib.load()


@contextlib.contextmanager
def debug_reset(lib):
    """Every lipreader debug switch back to its production default, however the block exits."""
    try:
        yield
    finally:
        lib.vatss_debug_lipreader_capture(None, 0)
        lib.vatss_debug_lipreader(0)
        lib.vatss_debug_lipreader_kernel(1)


def guarded(frames, per_frame, dtype):
    """(allocation, view): a (frames, per_frame) view with GUARD_ROWS sentinel frames before and after it."""
    itype, pat = SENTINEL[dtype]
    buf = torch.empty(frames + 2 * GUARD_ROWS, per_frame, dtype=dtype, device=DEV)
    buf.view(itype).fill_(pat)
    return buf, buf[GUARD_ROWS:GUARD_ROWS + frames]


def assert_guard(buf, frames, label, written=True):
    """The guard frames (and, for a stage that must never be written, the whole buffer) still hold the sentinel."""
    itype, pat = SENTINEL[buf.dtype]
    b = buf.view(itype) != pat
    if written:
        b[GUARD_ROWS:GUARD_ROWS + frames] = False
    n = int(b.sum())
    if n:
        r = int(b.nonzero()[0, 0])
        raise AssertionError(f"{label}: {n} values written outside the stage, first in allocation frame {r}")


def report(engine, stage, ratio, label):
    print(f"WORST-RATIO lipreader {engine} {stage}: {ratio:.3f} {label}")


# ---------------------------------------------------------------------------------------------------------- geometry
def out_dim(n, k, s, p):
    return (n + 2 * p - k) // s + 1


def geometry(Hc, Wc):
    """(H1, W1) of the front end, [(H_l, W_l)] of the four trunk layers (lipreader.cu lip_geometry)."""
    H1, W1 = out_dim(Hc, 7, 2, 3), out_dim(Wc, 7, 2, 3)
    hw = [(out_dim(H1, 3, 2, 1), out_dim(W1, 3, 2, 1))]
    for _ in range(3):
        hw.append((out_dim(hw[-1][0], 3, 2, 1), out_dim(hw[-1][1], 3, 2, 1)))
    return H1, W1, hw


def stage_shapes(Hc, Wc):
    """(H, W, C) per capture slot; None for the shortcut slot of a block without a shortcut convolution."""
    H1, W1, hw = geometry(Hc, Wc)
    shapes = [(H1, W1, 64), (hw[0][0], hw[0][1], 64)]
    for k in range(8):
        l = k // 2
        s = (hw[l][0], hw[l][1], 64 << l)
        shapes += [s, s if (l > 0 and k % 2 == 0) else None, s]
    return shapes


def block_names(k):
    l, b = k // 2 + 1, k % 2
    p = f"trunk.layer{l}.{b}"
    stride = 2 if (l > 1 and b == 0) else 1
    return p, stride


# --------------------------------------------------------------------------------------------------------------- cases
def conv_m(F, Hc, Wc):
    """Output rows M = F Ho Wo of every convolution family: front-end GEMM, layers 1-4 (the shortcuts share their
    layer's M).  The frames of one launch are those of one chunk; the cases below stay within one."""
    H1, W1, hw = geometry(Hc, Wc)
    return {"front": F * H1 * W1, **{f"layer{l + 1}": F * h * w for l, (h, w) in enumerate(hw)}}


def search_ragged(done):
    """Cheapest (F, Hc, Wc) - by F Hc Wc - whose M > 128 has M mod 128 = 1 or 127 for each family not yet in `done`,
    greedily preferring cases that cover several families."""
    want = {f for f in ("front", "layer1", "layer2", "layer3", "layer4")} - set(done)
    per_frame = {(Hc, Wc): conv_m(1, Hc, Wc) for Hc in range(8, 49) for Wc in range(8, 89)}
    picked = []
    while want:
        best = None
        for F in range(1, 33):
            for (Hc, Wc), ms in per_frame.items():
                hit = {f for f, m in ms.items() if F * m > 128 and F * m % 128 in (1, 127)} & want
                key = (-len(hit), F * Hc * Wc)
                if hit and (best is None or key < best[0]):
                    best = (key, (F, Hc, Wc), hit)
        picked.append(best[1])
        want -= best[2]
    return picked


def residues(F, Hc, Wc):
    return {f: m % 128 for f, m in conv_m(F, Hc, Wc).items()}


RELUS = ["swish", "prelu", "relu"]
# name: (relu, B, T, Hc, Wc, raw): raw = integer 96 x 96 frames through the crop + affine of extract_embeddings (the
# crop window of the 88 x 88 production case; other crops from the top-left corner), otherwise preprocessed N(0, 1) input
CASES = {
    "production": ("swish", 2, 7, 88, 88, True),
    "odd-70x58": ("prelu", 2, 2, 70, 58, False),
    "odd-33x87": ("relu", 1, 3, 33, 87, False),
    "odd-16x8": ("swish", 3, 4, 16, 8, False),
    "narrow-8x8-T1": ("prelu", 3, 1, 8, 8, False),
    "narrow-8x12-T2": ("relu", 2, 2, 8, 12, False),
    "narrow-12x8-T3": ("swish", 2, 3, 12, 8, True),
    "tall-416x88": ("prelu", 2, 3, 416, 88, False),
    "ragged-88x88-F55": ("relu", 1, 55, 88, 88, True),
    "ragged-88x88-F57": ("swish", 3, 19, 88, 88, True),
    "two-chunks-F1030": ("swish", 10, 103, 88, 88, True),
}
for _i, (_F, _Hc, _Wc) in enumerate(search_ragged({"layer2", "layer4"})):
    CASES[f"ragged-{_Hc}x{_Wc}-F{_F}"] = (RELUS[(_i + 1) % 3], 1, _F, _Hc, _Wc, False)
RAGGED = [n for n in CASES if n.startswith("ragged")]


def checked_frames(B, T):
    """Frames whose stages are checked: all of them, or for more than one chunk the frames within 3 of each seam and
    the whole last chunk."""
    F = B * T
    if F <= CHUNK:
        return torch.arange(F)
    last = (F - 1) // CHUNK * CHUNK
    sel = set(range(last, F))
    for s in range(CHUNK, F, CHUNK):
        sel |= set(range(max(0, s - 3), min(F, s + 4)))
    return torch.tensor(sorted(sel))


# ------------------------------------------------------------------------------------------------------ running it
class Net:
    """Packed weights (Lipreading._prepare) and the fp64 reference weights of one relu type, on the device."""

    def __init__(self, relu_type, seed):
        from speech_separation_b200 import Lipreading

        self.relu_type = relu_type
        sd = LO.make_state_dict(relu_type, seed)
        m = Lipreading(relu_type=relu_type, extract_feats=True)
        m.load_state_dict(sd, strict=True)
        self.module = m.to(DEV)
        self.module._prepare(DEV)
        self.sd = {k: v.to(DEV) for k, v in sd.items()}


def make_video(name, relu, B, T, Hc, Wc, raw):
    """(video (B, T, Hin, Win) fp32, crop (y0, x0), pre_scale, pre_shift, normalised input (B, T, Hc, Wc) fp64): the
    last is what the kernels see.  pre_scale / pre_shift reach the kernel as fp32, and v * s + t compiles to one FFMA
    in both front-end kernels, so for integer v <= 255 (exact product and sum in fp64) fp32(v s + t) reproduces it."""
    from speech_separation_b200.lipreader import PRE_MEAN, PRE_STD, center_crop_window

    seed = sum(map(ord, name))
    if raw:
        Hin, Win = max(96, Hc), max(96, Wc)
        video = torch.from_numpy(LO.make_frames(B, T, Hin, Win, seed=seed)).to(DEV)
        y0, x0 = center_crop_window(Hin, Win)[:2] if (Hc, Wc) == (88, 88) else (0, 0)
        s = float(np.float32(1.0 / (255.0 * PRE_STD)))
        t = float(np.float32(-PRE_MEAN / PRE_STD))
        vn = (video[:, :, y0:y0 + Hc, x0:x0 + Wc].double() * s + t).float().double()
        return video, (y0, x0), s, t, vn
    g = torch.Generator().manual_seed(seed)
    video = torch.randn(B, T, Hc, Wc, generator=g).to(DEV)
    return video, (0, 0), 1.0, 0.0, video.double()


def run_forward(lib, net, video, crop, s, t, Hc, Wc, engine, capture=True):
    """One vatss_lipreader_forward through the C ABI with every stage captured; checks the guards and the workspace
    tail.  Returns (features (F, 512) fp32, [stage views or None])."""
    B, T, Hin, Win = video.shape
    F = B * T
    dtype = torch.float32 if engine == "f32" else torch.float16
    ws_bytes = int(lib.vatss_lipreader_workspace_bytes(B, T, Hc, Wc))
    assert ws_bytes > 0
    ws = torch.empty(ws_bytes + WS_TAIL, dtype=torch.uint8, device=DEV)
    ws[ws_bytes:].fill_(0xA5)
    obuf, out = guarded(F, 512, torch.float32)
    bufs, views = [], []
    shapes = stage_shapes(Hc, Wc)
    for i, shp in enumerate(shapes):
        full = shp or shapes[i + 1]       # a slot that must stay unwritten gets the size the block would write
        b, v = guarded(F, full[0] * full[1] * full[2], dtype)
        bufs.append(b)
        views.append(v if shp is not None else None)
    table = (ctypes.c_void_p * NSTAGES)(*[b.data_ptr() + GUARD_ROWS * b.shape[1] * b.element_size() for b in bufs])
    m = net.module
    with debug_reset(lib):
        if capture:
            lib.vatss_debug_lipreader_capture(table, NSTAGES)
        rc = lib.vatss_lipreader_forward(m._packed.data_ptr(), m._packed.numel(), ACT[net.relu_type], video.data_ptr(),
                                         B, T, Hin, Win, crop[0], crop[1], Hc, Wc, s, t, out.data_ptr(), ws.data_ptr(),
                                         ws_bytes, 0 if engine == "f32" else 1, None)
        from speech_separation_b200 import _lib

        _lib.check(rc, "vatss_lipreader_forward")
        torch.cuda.synchronize()
    tail = ws[ws_bytes:]
    assert bool((tail == 0xA5).all()), f"workspace: {int((tail != 0xA5).sum())} bytes written past the size it asked for"
    assert_guard(obuf, F, "features")
    for i, (b, v) in enumerate(zip(bufs, views)):
        assert_guard(b, F, f"capture slot {i}", written=capture and v is not None)
    return out, views


# ---------------------------------------------------------------------------------------------------------- references
def bn_fold(sd, prefix):
    s = sd[prefix + ".weight"].double() / torch.sqrt(sd[prefix + ".running_var"].double() + LO.EPS)
    h = sd[prefix + ".bias"].double() - sd[prefix + ".running_mean"].double() * s
    return s, h, (sd[prefix + ".running_mean"].double() * s).abs()


def act64(z, relu_type, slope):
    if relu_type is None:
        return z
    if relu_type == "relu":
        return torch.relu(z)
    if relu_type == "prelu":
        return torch.where(z >= 0, z, z * slope.double())
    return z * torch.sigmoid(z)


def conv_ref(x, w, stride, pad):
    """x (n, H, W, C) fp64, w (O, C, k, k) fp64 -> (sum x w, sum |x| |w|), both (n, Ho, Wo, O)."""
    n, H, W, C = x.shape
    O, k = w.shape[0], w.shape[-1]
    Ho, Wo = out_dim(H, k, stride, pad), out_dim(W, k, stride, pad)
    cols = Fn.unfold(x.permute(0, 3, 1, 2), k, padding=pad, stride=stride)     # (n, C k k, Ho Wo), order (c, ky, kx)
    wm = w.reshape(O, -1)
    acc = (wm @ cols).transpose(1, 2).reshape(n, Ho, Wo, O)
    mag = (wm.abs() @ cols.abs()).transpose(1, 2).reshape(n, Ho, Wo, O)
    return acc, mag


def front_ref_inputs(vn, T, frames):
    """vn (B, T, Hc, Wc) fp64 -> (n, Hc + 6, Wc + 6, 5) padded 5-frame stacks of the given frames: the 3-D front end as
    a 2-D 7 x 7 stride-2 convolution over 5 channels (kt), zero padding per utterance in time and space."""
    vp = Fn.pad(vn, (3, 3, 3, 3, 2, 2))                                      # (B, T + 4, Hc + 6, Wc + 6)
    f = frames.to(DEV)
    st = vp[(f // T)[:, None], (f % T)[:, None] + torch.arange(5, device=DEV)]   # (n, 5, Hp, Wp)
    return st.permute(0, 2, 3, 1)


def stage_bound(z_hat, y_hat, acc, mag, s, h, ms, cK, relu, engine, res=None):
    ez = s.abs() * cK * mag + 2.0 ** -22 * ((acc * s).abs() + ms + h.abs()) + U32 * (acc * s + h).abs()
    if res is not None:
        ez = ez + U32 * z_hat.abs()
    b = L_ACT[relu] * ez + r_act(relu, engine, z_hat) * y_hat.abs()
    if engine == "f32":
        return b + 2.0 ** -126
    return (1 + U16) * b + U16 * y_hat.abs() + 2.0 ** -25


def c_acc(K, engine):
    return K * U32 / (1 - K * U32) if engine == "f32" else (K + 2) * 2.0 ** -23


def locate(idx, frames, shape, F, label):
    """A failing element's coordinates and where it sits: image border, ragged last 128-row tile, last chunk."""
    i, y, x, c = idx
    f = int(frames[i])
    H, W = shape[0], shape[1]
    f0 = f // CHUNK * CHUNK
    nf = min(CHUNK, F - f0)
    m, M = (f - f0) * H * W + y * W + x, nf * H * W
    where = []
    if y in (0, H - 1) or x in (0, W - 1):
        where.append("image border")
    if M % 128 and m >= M // 128 * 128:
        where.append(f"ragged last 128-row tile (M = {M})")
    if F > CHUNK and f >= (F - 1) // CHUNK * CHUNK:
        where.append("last chunk")
    return f"{label}: frame {f}, y {y}, x {x}, channel {c}" + (f" [{', '.join(where)}]" if where else "")


def check_elements(got, want, bound, frames, F, label):
    """Every element within its bound (a NaN - a value never written - fails); returns the worst |err| / bound."""
    err = (got.double() - want).abs()
    ok = err <= bound
    if not bool(ok.all()):
        bad = (~ok).nonzero()
        idx = [int(v) for v in bad[0]]
        at = locate(idx, frames, got.shape[1:], F, label)
        raise AssertionError(f"{bad.shape[0]} elements out of bound; first at {at}: got {float(got[tuple(idx)]):.7g} "
                             f"want {float(want[tuple(idx)]):.7g} err {float(err[tuple(idx)]):.3e} "
                             f"bound {float(bound[tuple(idx)]):.3e}")
    return float((err / bound).max())


def maxpool_ref(x):
    """MaxPool 3 x 3, stride 2, padding 1 as the max over the -inf-padded window: x (n, H, W, C) -> (n, Ho, Wo, C)."""
    xp = Fn.pad(x.permute(0, 3, 1, 2).double(), (1, 1, 1, 1), value=-math.inf)
    return xp.unfold(2, 3, 2).unfold(3, 3, 2).amax(dim=(-1, -2)).permute(0, 2, 3, 1)


def check_stages(net, engine, views, vn, B, T, Hc, Wc, frames, out, label):
    """Every stage from its captured input; returns {stage: worst ratio}."""
    relu, sd, F = net.relu_type, net.sd, B * T
    f32 = engine == "f32"
    rnd = (lambda t: t.double()) if f32 else (lambda t: t.half().double())   # weights as the packing kernels store them
    cap = lambda slot: views[slot][frames.to(DEV)].reshape(len(frames), *stage_shapes(Hc, Wc)[slot]).double()
    worst = {}

    def note(stage, r):
        worst[stage] = max(worst.get(stage, 0.0), r)

    # front end: Conv3d(1 -> 64, 5 x 7 x 7, stride 1 x 2 x 2, pad 2 x 3 x 3) + BN + act
    x = front_ref_inputs(vn, T, frames)
    if not f32:
        x = x.float().half().double()                                         # k_lip_im2col_front rounds to fp16 (RN)
    w = rnd(sd["frontend3D.0.weight"]).reshape(64, 5, 7, 7)
    acc, mag = conv_ref(x, w, 2, 0)
    s, h, ms = bn_fold(sd, "frontend3D.1")
    z = acc * s + h
    y = act64(z, relu, sd.get("frontend3D.2.weight"))
    bound = stage_bound(z, y, acc, mag, s, h, ms, c_acc(245 if f32 else 256, engine), relu, engine)
    note("front end", check_elements(cap(0), y, bound, frames, F, f"{label} front end"))
    # max pool: bit for bit against the max over the -inf-padded window of the captured pre-pool map
    pooled, want = cap(1), maxpool_ref(cap(0))
    if not bool((pooled == want).all()):
        idx = [int(v) for v in (pooled != want).nonzero()[0]]
        raise AssertionError(f"max pool differs at {locate(idx, frames, pooled.shape[1:], F, label)}: got "
                             f"{float(pooled[tuple(idx)])} want {float(want[tuple(idx)])}")
    note("max pool", 0.0)
    # trunk: conv1 -> act, shortcut, act(conv2 + residual), each from its captured inputs
    xin = 1
    for k in range(8):
        p, stride = block_names(k)
        c1, sc, yo = 2 + 3 * k, 3 + 3 * k, 4 + 3 * k
        xb = cap(xin)
        cin = xb.shape[-1]
        acc, mag = conv_ref(xb, rnd(sd[p + ".conv1.weight"]), stride, 1)
        s, h, ms = bn_fold(sd, p + ".bn1")
        z = acc * s + h
        y = act64(z, relu, sd.get(p + ".relu1.weight"))
        bound = stage_bound(z, y, acc, mag, s, h, ms, c_acc(9 * cin, engine), relu, engine)
        note("conv1", check_elements(cap(c1), y, bound, frames, F, f"{label} block {k} conv1"))
        if views[sc] is not None:
            acc, mag = conv_ref(xb, rnd(sd[p + ".downsample.0.weight"]), stride, 0)
            s, h, ms = bn_fold(sd, p + ".downsample.1")
            z = acc * s + h
            bound = stage_bound(z, z, acc, mag, s, h, ms, c_acc(cin, engine), None, engine)
            note("shortcut", check_elements(cap(sc), z, bound, frames, F, f"{label} block {k} shortcut"))
            res = cap(sc)
        else:
            res = xb
        t1 = cap(c1)
        acc, mag = conv_ref(t1, rnd(sd[p + ".conv2.weight"]), 1, 1)
        s, h, ms = bn_fold(sd, p + ".bn2")
        z = acc * s + h + res
        y = act64(z, relu, sd.get(p + ".relu2.weight"))
        bound = stage_bound(z, y, acc, mag, s, h, ms, c_acc(9 * t1.shape[-1], engine), relu, engine, res=res)
        note("block output", check_elements(cap(yo), y, bound, frames, F, f"{label} block {k} output"))
        xin = yo
    # average pool of the last block output: the forward's own output
    last = cap(25)
    hw = last.shape[1] * last.shape[2]
    want = last.mean(dim=(1, 2))
    bound = (hw + 1) * U32 * last.abs().mean(dim=(1, 2)) + 2.0 ** -126
    got = out[frames.to(DEV)].double()
    err = (got - want).abs()
    bad = ~(err <= bound)
    if bool(bad.any()):
        i, c = [int(v) for v in bad.nonzero()[0]]
        raise AssertionError(f"{label} average pool: frame {int(frames[i])} channel {c} err {float(err[i, c]):.3e} "
                             f"bound {float(bound[i, c]):.3e}")
    note("average pool", float((err / bound).max()))
    return worst


def whole_forward_per_frame(net, vn, B, T, out, engine, label):
    """Every frame's 512-vector within the whole-forward tolerance of the fp64 oracle (the tolerance of
    test_lipreader.py, per frame instead of over the batch)."""
    with torch.no_grad():
        ref = LO.forward(net.sd, vn[:, None], net.relu_type, dtype=torch.float64).reshape(B * T, 512)
    rel = (out.double() - ref).norm(dim=1) / ref.norm(dim=1)
    tol = F32_TOL if engine == "f32" else TENSOR_TOL
    if not bool((rel <= tol).all()):
        f = int((~(rel <= tol)).nonzero()[0])
        raise AssertionError(f"{label}: frame {f} (utterance {f // T}, t {f % T}) rel-L2 {float(rel[f]):.3e} > {tol:.0e}")
    return float(rel.max()) / tol


_NETS = {}


def get_net(relu_type):
    if relu_type not in _NETS:
        _NETS[relu_type] = Net(relu_type, seed={"swish": 31, "prelu": 32, "relu": 33}[relu_type])
    return _NETS[relu_type]


def residue_note(F, Hc, Wc):
    hits = {f: r for f, r in residues(F, Hc, Wc).items() if r in (1, 127)}
    return f"M mod 128 in {{1, 127}}: {hits}" if hits else ""


@pytest.mark.parametrize("engine", ["f32", "tensor"])
@pytest.mark.parametrize("name", list(CASES))
def test_lipreader_stages_match_fp64(lib, name, engine):
    relu, B, T, Hc, Wc, raw = CASES[name]
    net = get_net(relu)
    video, crop, s, t, vn = make_video(name, relu, B, T, Hc, Wc, raw)
    out, views = run_forward(lib, net, video, crop, s, t, Hc, Wc, engine)
    frames = checked_frames(B, T)
    label = f"{name} ({relu}, B={B} T={T} {Hc}x{Wc}) {engine}"
    if B * T <= CHUNK:
        print(f"{label}: {residue_note(B * T, Hc, Wc)}")
    worst = check_stages(net, engine, views, vn, B, T, Hc, Wc, frames, out, label)
    worst["forward per frame"] = whole_forward_per_frame(net, vn, B, T, out, engine, label)
    for stage, r in worst.items():
        report(engine, stage, r, f"({name})")


@pytest.mark.parametrize("name", ["production"] + RAGGED)
def test_tensor_kernel_variants_capture_bit_identical_stages(lib, name):
    """The persistent tcgen05 convolution (vatss_debug_lipreader_kernel(2)) and the two-CTA-per-SM variant for 64-channel
    layers (vatss_debug_lipreader(256)) against the default kernel: every captured stage bit for bit."""
    relu, B, T, Hc, Wc, raw = CASES[name]
    net = get_net(relu)
    video, crop, s, t, _ = make_video(name, relu, B, T, Hc, Wc, raw)
    out, views = run_forward(lib, net, video, crop, s, t, Hc, Wc, "tensor")
    want = [v.clone() if v is not None else None for v in views] + [out.clone()]
    for switch, value in (("vatss_debug_lipreader_kernel", 2), ("vatss_debug_lipreader", 256)):
        with debug_reset(lib):
            getattr(lib, switch)(value)
            o2, v2 = run_forward(lib, net, video, crop, s, t, Hc, Wc, "tensor")
            for i, (a, b) in enumerate(zip(want, v2 + [o2])):
                if a is None:
                    continue
                itype = torch.int16 if a.dtype == torch.float16 else torch.int32
                assert torch.equal(a.view(itype), b.view(itype)), f"{switch}({value}): capture slot {i} differs"


def test_capture_off_leaves_the_outputs_alone(lib):
    """With the capture table empty the forward is the production launch sequence: same features bit for bit, and no
    capture buffer written."""
    relu, B, T, Hc, Wc, raw = CASES["odd-16x8"]
    net = get_net(relu)
    video, crop, s, t, _ = make_video("odd-16x8", relu, B, T, Hc, Wc, raw)
    for engine in ("f32", "tensor"):
        on, _ = run_forward(lib, net, video, crop, s, t, Hc, Wc, engine)
        off, _ = run_forward(lib, net, video, crop, s, t, Hc, Wc, engine, capture=False)
        assert torch.equal(on.view(torch.int32), off.view(torch.int32)), engine
