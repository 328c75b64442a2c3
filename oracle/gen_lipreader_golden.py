"""Generate tests/golden/lipreader_*.npz from the reference's own `Lipreading` class (imported unmodified).

TEST INFRASTRUCTURE ONLY.  Run in the build container (needs /root/reference):
    python -m oracle.gen_lipreader_golden
For every relu_type the reference supports ("swish" is what src/lipreader/configs/lrw_resnet18_mstcn.json selects) the
script instantiates `Lipreading(..., extract_feats=True)` exactly as src/utils/init_utils.py:168-207 does, loads the
synthetic weights of oracle.lipreader_oracle.make_state_dict (strict=False: the classification head keeps its own
init and is not on the path), runs the reference preprocessing classes (Normalize, CenterCrop, Normalize -
dataloaders.py:24-27; `cv2`, which preprocess.py imports for an unrelated transform, is not installed and is stubbed
by an empty module) and the reference forward, and stores the raw frames (uint8) and the (B, T, 512) features.
`python -m oracle.gen_lipreader_golden preprocess` writes tests/golden/lipreader_preprocess.npz (write_preprocess_golden).
"""
import importlib
import json
import os
import sys
import types

import numpy as np
import torch

from . import lipreader_oracle as LO

REF_ROOT = os.environ.get("VATSS_REFERENCE_ROOT", "/root/reference")
OUT_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
# square, non-square and odd frame sizes: the crop offsets round half the excess
PREPROCESS_SIZES = ((96, 96), (88, 88), (97, 101), (120, 90), (89, 96))


def load_reference():
    sys.dont_write_bytecode = True
    if "src" not in sys.modules:
        src = types.ModuleType("src")
        src.__path__ = [os.path.join(REF_ROOT, "src")]
        sys.modules["src"] = src
    for name in ("src.lipreader", "src.lipreader.lipreading", "src.lipreader.lipreading.models"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.__path__ = [os.path.join(REF_ROOT, *name.split("."))]
            sys.modules[name] = m
    sys.modules.setdefault("cv2", types.ModuleType("cv2"))
    model = importlib.import_module("src.lipreader.lipreading.model")
    pre = importlib.import_module("src.lipreader.lipreading.preprocess")
    return model, pre


def build_reference(model_mod, relu_type):
    cfg = json.load(open(os.path.join(REF_ROOT, "src", "lipreader", "configs", "lrw_resnet18_mstcn.json")))
    tcn_options = {"num_layers": cfg.get("tcn_num_layers", 4), "kernel_size": cfg.get("tcn_kernel_size", [3]),
                   "dropout": cfg.get("tcn_dropout", 0.2), "dwpw": cfg.get("tcn_dwpw", False),
                   "width_mult": cfg.get("tcn_width_mult", 1)}
    return model_mod.Lipreading(modality="video", num_classes=cfg.get("num_classes", 500), tcn_options=tcn_options,
                                densetcn_options={}, backbone_type=cfg["backbone_type"], relu_type=relu_type,
                                width_mult=cfg["width_mult"], use_boundary=cfg.get("use_boundary", False),
                                extract_feats=True)


def main():
    model_mod, pre = load_reference()
    pipeline = reference_pipeline(pre)
    for relu_type, (B, T) in (("swish", (2, 7)), ("prelu", (1, 5)), ("relu", (1, 5))):
        torch.manual_seed(0)
        ref = build_reference(model_mod, relu_type).eval()
        sd = LO.make_state_dict(relu_type)
        missing, unexpected = ref.load_state_dict(sd, strict=False)
        assert not unexpected and all(k.startswith("tcn.") or k.endswith("num_batches_tracked") for k in missing), \
            (missing, unexpected)
        frames = LO.make_frames(B, T)
        feats = []
        with torch.no_grad():
            for b in range(B):   # make_embeddings.py:58-65, one clip at a time
                data = pipeline(frames[b])
                x = torch.FloatTensor(data)[None, None]
                feats.append(ref(x, lengths=[T]).squeeze(0).numpy())
        feats = np.stack(feats)
        path = os.path.join(OUT_DIR, f"lipreader_{relu_type}_B{B}_T{T}.npz")
        np.savez_compressed(path, frames=frames.astype(np.uint8), features=feats.astype(np.float32),
                            relu_type=np.array(relu_type), weight_seed=np.array(2024))
        print(path, feats.shape, float(np.abs(feats).mean()), os.path.getsize(path))


def reference_pipeline(pre):
    """dataloaders.py:24-27 built from the reference's own preprocessing classes."""
    return pre.Compose([pre.Normalize(0.0, 255.0), pre.CenterCrop((88, 88)), pre.Normalize(0.421, 0.165)])


def write_preprocess_golden():
    """tests/golden/lipreader_preprocess.npz: 3 frames per size of PREPROCESS_SIZES (default_rng(1)) and what
    Normalize(0, 255) -> CenterCrop(88, 88) -> Normalize(0.421, 0.165) makes of them.  Computed by the reference's classes
    where its checkout is present, otherwise by the restatement LO.preprocess; `source` records which."""
    if os.path.isfile(os.path.join(REF_ROOT, "src", "lipreader", "lipreading", "preprocess.py")):
        pipeline, source = reference_pipeline(load_reference()[1]), "reference preprocess.py classes"
    else:
        pipeline, source = LO.preprocess, "oracle.lipreader_oracle.preprocess (reference checkout not present)"
    rng = np.random.default_rng(1)
    out = {"sizes": np.array(PREPROCESS_SIZES, dtype=np.int64), "source": np.array(source)}
    for i, (h, w) in enumerate(PREPROCESS_SIZES):
        frames = rng.integers(0, 256, (3, h, w)).astype(np.float32)
        out[f"c{i}.frames"] = frames.astype(np.uint8)
        out[f"c{i}.want"] = np.asarray(pipeline(frames), dtype=np.float32)
    path = os.path.join(OUT_DIR, "lipreader_preprocess.npz")
    np.savez_compressed(path, **out)
    print(path, source, os.path.getsize(path))


if __name__ == "__main__":
    if sys.argv[1:] == ["preprocess"]:
        write_preprocess_golden()
    else:
        main()
