"""Lipreader front end (SURVEY.md §8f rank 4): oracle pinned to the reference's `Lipreading`, host-side mirror on CPU,
and the CUDA path (through the C ABI) against the reference-generated goldens.

Goldens: tests/golden/lipreader_*.npz - outputs of the reference class itself (oracle/gen_lipreader_golden.py) on the
synthetic weights of oracle.lipreader_oracle.make_state_dict.  Tolerances: the fp32 engine is held to 2e-5 relative L2
(fp32 summation order only); the tcgen05 engine (fp16 activations through 17 convolutions, fp32 accumulation) to 2e-3 (measured 3e-4 - 5e-4) -
the reference states no tolerance for this path; the separation model layer-normalises what it receives.
"""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import lipreader_oracle as LO

CASES = [("swish", 2, 7), ("prelu", 1, 5), ("relu", 1, 5)]
F32_TOL = 2e-5
TENSOR_TOL = 2e-3


def rel_l2(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def load_case(golden_dir, relu_type, B, T):
    z = np.load(os.path.join(golden_dir, f"lipreader_{relu_type}_B{B}_T{T}.npz"))
    return z["frames"].astype(np.float32), z["features"], int(z["weight_seed"])


# ------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("relu_type,B,T", CASES)
def test_oracle_matches_reference_lipreading(golden_dir, relu_type, B, T):
    frames, feats, seed = load_case(golden_dir, relu_type, B, T)
    sd = LO.make_state_dict(relu_type, seed)
    x = torch.from_numpy(LO.preprocess(frames).astype(np.float32))[:, None]
    with torch.no_grad():
        y32 = LO.forward(sd, x, relu_type).numpy()
        y64 = LO.forward(sd, x, relu_type, dtype=torch.float64).numpy()
    assert y32.shape == feats.shape == (B, T, 512)
    assert rel_l2(y32, feats) < 1e-6      # same torch ops in the same order as the reference modules
    assert rel_l2(y64, feats) < 2e-6      # the reference ran in fp32


@pytest.mark.parametrize("relu_type,B,T", [("prelu", 1, 5), ("relu", 1, 5)])
def test_numpy_restatement_matches_reference_lipreading(golden_dir, relu_type, B, T):
    """The numpy-only fp64 restatement (sliding windows + einsum; none of torch's convolution, pooling or BatchNorm code)
    against the reference class's output."""
    frames, feats, seed = load_case(golden_dir, relu_type, B, T)
    sd = {k: v.numpy() for k, v in LO.make_state_dict(relu_type, seed).items()}
    y = LO.forward_numpy(sd, LO.preprocess(frames)[:, None], relu_type)
    assert y.shape == feats.shape
    assert rel_l2(y, feats) < 2e-6


def test_frames_generator_is_deterministic(golden_dir):
    frames, _, _ = load_case(golden_dir, "swish", 2, 7)
    assert np.array_equal(LO.make_frames(2, 7), frames)


def test_mirror_state_dict_and_constructor_contract():
    from speech_separation_b200 import Lipreading
    from speech_separation_b200.lipreader import _conv_param_names, center_crop_window

    for relu_type in ("swish", "prelu", "relu"):
        m = Lipreading(relu_type=relu_type, extract_feats=True)
        own = {k: tuple(v.shape) for k, v in m.state_dict().items() if not k.endswith("num_batches_tracked")}
        ref = dict(LO.state_dict_names(relu_type))
        assert own == ref
        assert list(own) == [k for k, _ in LO.state_dict_names(relu_type)]   # the reference's key order
        sd = LO.make_state_dict(relu_type)
        sd["tcn.tcn_output.weight"] = torch.zeros(500, 768)                  # a full checkpoint also has the head
        m.load_state_dict(sd, strict=False)
        names = _conv_param_names(relu_type)
        assert len(names) == 25 * 6
        assert {n for n in names if n} == set(ref)
        assert not m.training
        with pytest.raises(NotImplementedError):
            m.train()
    for kw in ({"extract_feats": False}, {"modality": "audio", "extract_feats": True},
               {"backbone_type": "shufflenet", "extract_feats": True}, {"use_boundary": True, "extract_feats": True}):
        with pytest.raises(NotImplementedError):
            Lipreading(**kw)
    assert center_crop_window(96, 96) == (4, 4, 88, 88)
    # conv init scale of the reference (model.py:281-293): std = sqrt(2 / (prod(kernel) * out_channels))
    torch.manual_seed(0)
    m = Lipreading(relu_type="swish", extract_feats=True)
    w = m.trunk.layer3[1].conv2.weight
    assert abs(float(w.detach().std()) - (2.0 / (9 * 256)) ** 0.5) < 2e-4
    assert float(m.frontend3D[1].weight.min()) == 1.0 and float(m.frontend3D[1].bias.abs().max()) == 0.0


def test_no_cpu_path():
    from speech_separation_b200 import Lipreading

    m = Lipreading(relu_type="swish", extract_feats=True)
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 1, 3, 88, 88), lengths=[3])


# ------------------------------------------------------------------------------------------- GPU
def _net(relu_type, seed, engine):
    from speech_separation_b200 import Lipreading

    m = Lipreading(relu_type=relu_type, extract_feats=True)
    m.load_state_dict(LO.make_state_dict(relu_type, seed), strict=True)
    return m.to("cuda:0").set_engine(engine)


@pytest.mark.gpu
@pytest.mark.parametrize("engine,tol", [("f32", F32_TOL), ("tensor", TENSOR_TOL)])
@pytest.mark.parametrize("relu_type,B,T", CASES)
def test_cuda_forward_matches_reference_golden(golden_dir, relu_type, B, T, engine, tol):
    frames, feats, seed = load_case(golden_dir, relu_type, B, T)
    net = _net(relu_type, seed, engine)
    x = torch.from_numpy(LO.preprocess(frames).astype(np.float32))[:, None].to("cuda:0")
    y = net(x, lengths=[T] * B).cpu().numpy()
    assert y.shape == feats.shape
    err = rel_l2(y, feats)
    print(f"lipreader {relu_type} {engine}: rel-L2 {err:.3e}")
    assert err < tol


@pytest.mark.gpu
@pytest.mark.parametrize("engine,tol", [("f32", F32_TOL), ("tensor", TENSOR_TOL)])
def test_cuda_embeddings_from_raw_frames(golden_dir, engine, tol):
    """make_embeddings.py:58-66: raw 96 x 96 crops -> (512, T); crop + normalisation folded into the first kernel."""
    from speech_separation_b200 import extract_embeddings

    frames, feats, seed = load_case(golden_dir, "swish", 2, 7)
    net = _net("swish", seed, engine)
    emb = extract_embeddings(net, torch.from_numpy(frames).to("cuda:0"))
    assert tuple(emb.shape) == (2, 512, 7)
    assert rel_l2(emb.transpose(1, 2).cpu().numpy(), feats) < tol
    one = extract_embeddings(net, torch.from_numpy(frames[1]).to("cuda:0"))     # a single (T, H, W) clip
    assert rel_l2(one[0].T.cpu().numpy(), feats[1]) < tol


@pytest.mark.gpu
def test_cuda_utterance_boundaries_and_frame_chunks():
    """Temporal zero padding at utterance boundaries against the CPU oracle, and more frames than one trunk pass holds
    (1024): the chunk seam falls inside an utterance, whose rows must not change (utterances are independent and a
    pixel's result does not depend on the tile it lands in - bit for bit on both engines)."""
    relu_type, B, T = "swish", 3, 40
    sd = LO.make_state_dict(relu_type, 11)
    frames = LO.make_frames(B, T, seed=3)
    x = torch.from_numpy(LO.preprocess(frames).astype(np.float32))[:, None]
    with torch.no_grad():
        ref = LO.forward(sd, x, relu_type).numpy()
    net = _net(relu_type, 11, "f32")
    y = net(x.to("cuda:0"), lengths=[T] * B).cpu().numpy()
    assert rel_l2(y, ref) < F32_TOL
    yt = net.set_engine("tensor")(x.to("cuda:0"), lengths=[T] * B).cpu().numpy()
    assert rel_l2(yt, ref) < TENSOR_TOL
    big = x.to("cuda:0").repeat(9, 1, 1, 1, 1)[:26]            # 26 x 40 = 1040 frames: seam at utterance 25, t = 24
    for engine, small in (("f32", y), ("tensor", yt)):
        net.set_engine(engine)
        yb = net(big, lengths=[T] * 26).cpu().numpy()
        for b in range(26):
            assert np.array_equal(yb[b], small[b % 3]), (engine, b)


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,H,W", [(1, 1, 88, 88), (2, 2, 70, 58), (1, 3, 33, 87), (3, 4, 16, 8), (2, 3, 8, 8),
                                     (1, 4, 12, 8), (2, 2, 8, 11)])
def test_cuda_odd_geometries_and_short_clips(B, T, H, W):
    """Shapes the production pipeline never produces but the reference class accepts: a single frame (all temporal taps
    but one fall into the zero padding), odd widths after every stride-2 stage (58 -> 29 -> 15 -> 8 -> 4 -> 2), ragged last
    row tiles, images smaller than a convolution tile, and crops of 8 - 12 pixels on a side, where layer 4 (1 x 1 x 512)
    is the largest trunk activation - against the CPU oracle, both engines."""
    relu_type = "prelu"
    sd = LO.make_state_dict(relu_type, 21)
    rng = np.random.Generator(np.random.PCG64(B * 1000 + T * 100 + H + W))
    x = torch.from_numpy(rng.normal(0.0, 1.0, (B, 1, T, H, W)).astype(np.float32))
    with torch.no_grad():
        ref = LO.forward(sd, x, relu_type).numpy()
    net = _net(relu_type, 21, "f32")
    y = net(x.to("cuda:0"), lengths=[T] * B).cpu().numpy()
    assert y.shape == ref.shape == (B, T, 512)
    assert rel_l2(y, ref) < F32_TOL
    yt = net.set_engine("tensor")(x.to("cuda:0"), lengths=[T] * B).cpu().numpy()
    assert rel_l2(yt, ref) < TENSOR_TOL


@pytest.mark.gpu
def test_cuda_rejects_unsupported_geometry():
    net = _net("swish", 2024, "tensor")
    with pytest.raises(ValueError):
        net(torch.zeros(1, 1, 2, 88, 120, device="cuda:0"), lengths=[2])     # wider than the front-end tile supports
    with pytest.raises(ValueError):
        net(torch.zeros(1, 2, 88, 88, device="cuda:0"), lengths=[2])         # not (B, 1, T, H, W)


@pytest.mark.gpu
def test_persistent_convolution_kernel_equals_one_tile_per_cta_kernel():
    """The persistent tcgen05 convolution (experiment, vatss_debug_lipreader_kernel(2)) against the default one-tile-per-CTA
    kernel: same K-slab order, same MMA shapes, same epilogue arithmetic - bit-identical features (270 frames: tiles in
    every role's second lap)."""
    from speech_separation_b200 import _lib

    net = _net("swish", 5, "tensor")
    x = torch.from_numpy(LO.preprocess(LO.make_frames(3, 90, seed=9)).astype(np.float32))[:, None].to("cuda:0")
    lib = _lib.load()
    try:
        lib.vatss_debug_lipreader_kernel(2)
        y2 = net(x, lengths=[90] * 3).cpu().numpy()
    finally:
        lib.vatss_debug_lipreader_kernel(1)
    y1 = net(x, lengths=[90] * 3).cpu().numpy()
    assert np.isfinite(y2).all() and np.array_equal(y1, y2)


@pytest.mark.gpu
def test_lipreader_feeds_the_separator(golden_dir):
    """profiler.py:17-22: video -> lipreader -> permute -> DPTN-AV; shapes and finiteness end to end on the device."""
    from speech_separation_b200 import DPTNAVWavEncDec, extract_embeddings

    net = _net("swish", 2024, "tensor")
    frames = torch.from_numpy(LO.make_frames(2, 25, seed=5)).to("cuda:0")
    emb = extract_embeddings(net, frames)                       # (2, 512, 25): one second of video per speaker
    torch.manual_seed(42)
    sep = DPTNAVWavEncDec(num_features=128, video_emb_size=512, hidden_video=128, kernel_size_enc=7, hidden_dim=128,
                          num_blocks=2, chunk_size=150, step_size=75).eval().to("cuda:0")
    mix = 0.1 * torch.randn(1, 16000, device="cuda:0")
    out = sep(mix=mix, s1_embedding=emb[0:1].contiguous(), s2_embedding=emb[1:2].contiguous())
    assert tuple(out["s1_pred"].shape) == (1, 16000)
    assert bool(torch.isfinite(out["s1_pred"]).all()) and bool(torch.isfinite(out["s2_pred"]).all())


def test_init_lipreader_reads_the_reference_config_and_checkpoint_format(tmp_path):
    """init_utils.py:168-207 + lipreading/utils.py:159-189: JSON config -> model; `checkpoint["model_state_dict"]` is loaded
    by key, the classification head's tensors are ignored."""
    import json

    from speech_separation_b200 import init_lipreader

    cfg = tmp_path / "lrw_resnet18_mstcn.json"   # the fields of src/lipreader/configs/lrw_resnet18_mstcn.json
    cfg.write_text(json.dumps({"backbone_type": "resnet", "relu_type": "swish", "tcn_dropout": 0.2, "tcn_dwpw": False,
                               "tcn_kernel_size": [3, 5, 7], "tcn_num_layers": 4, "tcn_width_mult": 1, "width_mult": 1.0}))
    sd = LO.make_state_dict("swish", 3)
    full = dict(sd)
    full["tcn.mb_ms_tcn.tcn0.cbcr0_0.conv.weight"] = torch.zeros(256, 512, 3)
    ckpt = tmp_path / "lipreader.pth"
    torch.save({"model_state_dict": full, "epoch_idx": 80}, ckpt)
    m = init_lipreader(str(cfg), str(ckpt))
    assert m.relu_type == "swish" and not m.training
    for k, v in sd.items():
        assert torch.equal(m.state_dict()[k], v), k
    assert "All parameters: 11182784" in str(m)      # model.py:196-207-style summary line
    m2 = init_lipreader(str(cfg))                     # no checkpoint: the reference's random initialisation
    assert float(m2.trunk.layer1[0].bn1.weight.min()) == 1.0


def test_make_embeddings_file_formats_and_batching(tmp_path, monkeypatch):
    """make_embeddings.py:52-73: `.npz` with `data` (T, H, W) in, `.npz` with `embedding` (512, T) out, same file names;
    clips of equal shape share a call.  Host logic only: the device call is replaced by a deterministic stand-in."""
    import speech_separation_b200.lipreader as L

    src, dst = tmp_path / "mouths", tmp_path / "embeddings"
    src.mkdir()
    rng = np.random.default_rng(0)
    shapes = {"a.npz": (5, 96, 96), "b.npz": (5, 96, 96), "c.npz": (7, 96, 96), "d.npz": (5, 96, 96)}
    for n, sh in shapes.items():
        np.savez_compressed(src / n, data=rng.integers(0, 256, sh).astype(np.uint8))
    calls = []

    def fake_extract(lipreader, frames):
        calls.append(tuple(frames.shape))
        assert frames.dtype == torch.float32
        return frames.mean(dim=(2, 3))[:, None, :].repeat(1, 512, 1)     # (B, 512, T)

    monkeypatch.setattr(L, "extract_embeddings", fake_extract)
    n = L.make_embeddings(object(), str(src), str(dst), device="cpu", max_clips_per_call=2)
    assert n == 4 and sorted(os.listdir(dst)) == sorted(shapes)
    assert sorted(calls) == [(1, 5, 96, 96), (1, 7, 96, 96), (2, 5, 96, 96)]
    for name, sh in shapes.items():
        e = np.load(dst / name)["embedding"]
        assert e.shape == (512, sh[0]) and e.dtype == np.float32
        np.testing.assert_allclose(e[0], np.load(src / name)["data"].astype(np.float32).mean(axis=(1, 2)), rtol=1e-6)
    with pytest.raises(NotADirectoryError):
        L.make_embeddings(object(), str(tmp_path / "missing"), str(dst))


@pytest.mark.gpu
def test_make_embeddings_end_to_end_on_the_device(golden_dir, tmp_path):
    """Mouth-crop `.npz` files -> `make_embeddings` -> embedding `.npz` files equal to the reference's features for the same
    clips (the golden clips, written one per file as make_embeddings.py expects them)."""
    from speech_separation_b200 import make_embeddings

    frames, feats, seed = load_case(golden_dir, "swish", 2, 7)
    src, dst = tmp_path / "mouths", tmp_path / "embeddings"
    src.mkdir()
    for b in range(2):
        np.savez_compressed(src / f"clip{b}.npz", data=frames[b].astype(np.uint8))
    net = _net("swish", seed, "tensor")
    assert make_embeddings(net, str(src), str(dst), device="cuda:0") == 2
    for b in range(2):
        e = np.load(dst / f"clip{b}.npz")["embedding"]
        assert e.shape == (512, 7)
        assert rel_l2(e.T, feats[b]) < TENSOR_TOL


def test_preprocessing_matches_reference_classes_when_available(golden_dir):
    """`center_crop_window` / `LO.preprocess` for square, non-square and odd frame sizes against the stored output of the
    Normalize / CenterCrop / Normalize pipeline (tests/golden/lipreader_preprocess.npz, oracle/gen_lipreader_golden.py),
    and, where a checkout of the reference is present, against the reference's own classes as well."""
    from oracle import ref_import
    from oracle.gen_lipreader_golden import PREPROCESS_SIZES
    from speech_separation_b200.lipreader import center_crop_window

    z = np.load(os.path.join(golden_dir, "lipreader_preprocess.npz"))
    assert [tuple(s) for s in z["sizes"]] == list(PREPROCESS_SIZES)
    pipeline = None
    if ref_import.available():
        from oracle.gen_lipreader_golden import load_reference, reference_pipeline

        pipeline = reference_pipeline(load_reference()[1])
    rng = np.random.default_rng(1)
    for i, (h, w) in enumerate(PREPROCESS_SIZES):
        frames = rng.integers(0, 256, (3, h, w)).astype(np.float32)
        assert np.array_equal(frames, z[f"c{i}.frames"])
        want = z[f"c{i}.want"]
        if pipeline is not None:
            np.testing.assert_allclose(pipeline(frames), want, rtol=1e-6, atol=1e-6)
        y0, x0, th, tw = center_crop_window(h, w)
        assert want.shape == (3, th, tw)
        got = (frames[:, y0:y0 + th, x0:x0 + tw] / 255.0 - 0.421) / 0.165
        np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-6)
        if (h, w) == (96, 96):
            np.testing.assert_array_equal(LO.preprocess(frames), want)
