"""Device time of one forward of the production DPTN-AV model (bench.py's MODEL_KW, 6 blocks) on the GENERIC engine.

    python tools/generic_forward_time.py [--batch 32] [--seconds 4] [--iters 5]

Times `engine="generic"` forwards with CUDA events around each call (after one warm-up forward), and the attention
stage alone through the library's per-stage profile.  Select another build of the library with VATSS_LIB_OVERRIDE to
compare two versions in one process each.  Prints one JSON line, with the GPU's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--seconds", type=float, default=4.0)
    ap.add_argument("--iters", type=int, default=5)
    args = ap.parse_args()

    import torch

    import speech_separation_b200 as V
    from speech_separation_b200 import _lib

    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    kw = dict(num_features=128, video_emb_size=512, hidden_video=128, kernel_size_enc=7, hidden_dim=128, num_blocks=6,
              chunk_size=150, step_size=75, num_heads=4, dropout=0.1, bidir=True)
    torch.manual_seed(42)
    net = V.DPTNAVWavEncDec(**kw).eval().to(dev).set_engine("generic")
    B, T = args.batch, int(args.seconds * 16000)
    Tv = -(-T // 640)
    g = torch.Generator().manual_seed(0)
    mix = torch.randn(B, T, generator=g).to(dev)
    e1 = torch.randn(B, 512, Tv, generator=g).to(dev)
    e2 = torch.randn(B, 512, Tv, generator=g).to(dev)
    with torch.no_grad():
        out = net(mix=mix, s1_embedding=e1, s2_embedding=e2)
        torch.cuda.synchronize()
        ms = []
        for _ in range(args.iters):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            net(mix=mix, s1_embedding=e1, s2_embedding=e2)
            b.record()
            b.synchronize()
            ms.append(a.elapsed_time(b))
        with _lib.stage_profile() as prof:
            out = net(mix=mix, s1_embedding=e1, s2_embedding=e2)
        torch.cuda.synchronize()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    print(json.dumps({"lib": os.path.basename(_lib.LIB_PATH), "batch": B, "seconds": args.seconds,
                      "forward_ms": sorted(ms), "forward_ms_median": sorted(ms)[len(ms) // 2],
                      "attention_ms": prof.ms["attention"], "stage_ms": prof.ms,
                      "s1_checksum": float(out["s1_pred"].double().abs().sum()), "gpu": smi}))


if __name__ == "__main__":
    main()
