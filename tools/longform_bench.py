"""Long recordings through `LongFormSeparator`: DPTN-AV at the production shape (seeded random weights and inputs),
window 64000, hop 48000, max_batch 32, one recording per call.

Prints one JSON document (and writes it to --out): per recording length the time per call, recording-seconds and
windows per second, the window cut + stitch on their own (CUDA events, L2 overwritten before every repetition), and
for the lengths given with --one-shot the plain forward over the whole recording with its workspace.  The GPU name
and power limit are read in the same process.

    python tools/longform_bench.py --seconds 60 600 --one-shot 60 --out profiles/longform_bench.json
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import speech_separation_b200 as V  # noqa: E402
from speech_separation_b200 import _lib  # noqa: E402
from speech_separation_b200.longform import micro_batches  # noqa: E402

SR, SPF = 16000, 640
MODEL_KW = dict(num_features=128, video_emb_size=512, hidden_video=128, kernel_size_enc=7, hidden_dim=128,
                num_blocks=6, chunk_size=150, step_size=75, num_heads=4, dropout=0.1, bidir=True)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def timed(fn, reps, flush=None):
    """Mean device milliseconds of fn over reps (events around fn only; flush runs outside the events)."""
    total = 0.0
    for _ in range(reps):
        if flush is not None:
            flush()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        total += a.elapsed_time(b)
    return total / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=int, nargs="+", default=[60, 600])
    ap.add_argument("--one-shot", type=int, nargs="*", default=[60])
    ap.add_argument("--window", type=int, default=64000)
    ap.add_argument("--hop", type=int, default=48000)
    ap.add_argument("--max-batch", type=int, default=32)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "longform_bench needs a CUDA device"
    dev = torch.device("cuda:0")
    torch.manual_seed(42)
    net = V.DPTNAVWavEncDec(**MODEL_KW).eval().to(dev)
    lf = V.LongFormSeparator(net, window=a.window, hop=a.hop, max_batch=a.max_batch)
    lib = _lib.load()
    W, H = a.window, a.hop
    flush_buf = torch.empty(512 * 2 ** 20, dtype=torch.uint8, device=dev)   # 512 MB > 126 MB of L2
    flush = lambda: flush_buf.fill_(1)
    res = {"gpu": gpu_info(), "model": "dptn_av production shape, 6 blocks", "window": W, "hop": H,
           "max_batch": a.max_batch, "recordings_per_call": 1, "rows": []}
    for sec in a.seconds:
        T = sec * SR
        g = torch.Generator().manual_seed(sec)
        mix = (0.1 * torch.randn(1, T, generator=g) + 0.1 * torch.randn(1, T, generator=g)).to(dev)
        e1 = torch.randn(1, 512, T // SPF, generator=g).to(dev)
        e2 = torch.randn(1, 512, T // SPF, generator=g).to(dev)
        n = lib.vatss_longform_windows(T, W, H)
        with torch.no_grad():
            call = lambda: lf(mix, e1, e2)
            call(); call()
            reps = max(2, min(10, 600 // sec))
            ms = timed(call, reps)
            # cut + stitch alone, on the same buffers the call uses
            batches = micro_batches(n, a.max_batch)
            Bm, E, Wv = batches[0][1], 512, W // SPF
            xb = torch.empty(Bm, W, device=dev)
            eb1, eb2 = torch.empty(Bm, E, Wv, device=dev), torch.empty(Bm, E, Wv, device=dev)
            y1, y2 = 0.1 * torch.randn(n, W, device=dev), 0.1 * torch.randn(n, W, device=dev)
            s1, s2 = torch.empty(1, T, device=dev), torch.empty(1, T, device=dev)
            nb = int(lib.vatss_window_stitch_scratch_bytes(1, n))
            scratch = torch.empty(nb, dtype=torch.uint8, device=dev)
            st = _lib.stream_ptr()

            def cut():
                for first, count in batches:
                    _lib.check(lib.vatss_window_cut(mix.data_ptr(), e1.data_ptr(), e2.data_ptr(), 1, T, T // SPF, E,
                                                    W, H, SPF, first, count, xb.data_ptr(), eb1.data_ptr(),
                                                    eb2.data_ptr(), st), "vatss_window_cut")

            def stitch():
                _lib.check(lib.vatss_window_stitch(y1.data_ptr(), y2.data_ptr(), 1, T, W, H, s1.data_ptr(),
                                                   s2.data_ptr(), None, None, scratch.data_ptr(), nb, st),
                           "vatss_window_stitch")

            cut(); stitch()
            cut_ms = timed(cut, 50, flush)
            stitch_ms = timed(stitch, 50, flush)
        stitch_bytes = 4 * (2 * n * W + 2 * (n - 1) * (W - H) + 2 * T)   # reads of y (overlaps twice), writes of s
        row = {"seconds": sec, "T": T, "windows": n, "micro_batches": [c for _, c in batches],
               "ms_per_call": round(ms, 3), "recording_s_per_s": round(sec / (ms / 1e3), 1),
               "windows_per_s": round(n / (ms / 1e3), 1),
               "cut_ms": round(cut_ms, 4), "stitch_ms": round(stitch_ms, 4),
               "cut_stitch_share_of_call": round((cut_ms + stitch_ms) / ms, 5),
               "stitch_GB_per_s": round(stitch_bytes / (stitch_ms / 1e3) / 1e9, 1),
               "l2": "overwritten (512 MB fill) before every cut / stitch repetition; not before the whole calls",
               "window_outputs_bytes": 2 * n * W * 4,
               "model_workspace_bytes_largest_micro_batch":
                   int(lib.vatss_workspace_bytes(ctypes.byref(net._desc), Bm, W, Wv))}
        if sec in a.one_shot:
            with torch.no_grad():
                one = lambda: net(mix, e1, e2)
                one(); one()
                row["one_shot_ms"] = round(timed(one, reps), 3)
                row["one_shot_recording_s_per_s"] = round(sec / (row["one_shot_ms"] / 1e3), 1)
        row["one_shot_workspace_bytes"] = int(lib.vatss_workspace_bytes(ctypes.byref(net._desc), 1, T, T // SPF))
        res["rows"].append(row)
        print(json.dumps(row), flush=True)
        del y1, y2, xb, eb1, eb2, s1, s2, scratch
        torch.cuda.empty_cache()
    res["gpu_after"] = gpu_info()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
