"""SI-SDR and SDR / SDRi on the device (`SISDRMetric`, `SDRMetric`, `SDRiMetric` `.device_value`) and their cost
inside the evaluation loop.

Prints one JSON document (and writes it to --out):
* per shape (32 x 4 s, the cfg-2 batch, and 4 x 10 min at 16 kHz) and metric: CUDA-event time of `device_value`
  (mean over repetitions, after warm-up) and the per-kernel device times of one call from torch.profiler, run
  separately so that tracing does not slow the timed calls;
* the multiply-adds of the SDR lag sums (4 partners x T x filter_length per target) and the rate they imply;
* `Inferencer` audio-seconds per second over the same 32 x 4 s batches (DPTN-AV at the production shape, seeded
  weights, no files written) with [SISNRi] against [SISNRi, SISDR, SDRi], alternated;
* for context, the host time of oracle/sdr_oracle.py (fp64 numpy / scipy, FFT correlation and solve_toeplitz) for
  the six pairings of one 4 s utterance: not torchmetrics.
The GPU name and power limit are read in the same process.

    python tools/sdr_bench.py --out profiles/sdr_bench.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import speech_separation_b200 as V  # noqa: E402
from oracle import sdr_oracle as D  # noqa: E402

SR = 16000
L = 512
MODEL_KW = dict(num_features=128, video_emb_size=512, hidden_video=128, kernel_size_enc=7, hidden_dim=128,
                num_blocks=6, chunk_size=150, step_size=75, num_heads=4, dropout=0.1, bidir=True)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def signals(B, T, seed, dev):
    """Speech-like targets (noise under a 0.1 s piecewise envelope, -30 .. 0 dB) and predictions at 10 dB SNR."""
    g = torch.Generator().manual_seed(seed)
    lv = 10 ** (-1.5 * torch.rand(2, B, -(-T // 1600), generator=g))
    s = torch.randn(2, B, T, generator=g) * lv.repeat_interleave(1600, -1)[..., :T]
    p = s + 0.3 * s.std() * torch.randn(2, B, T, generator=g)
    return p[0].to(dev), p[1].to(dev), s[0].to(dev), s[1].to(dev)


def timed(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def kernel_times(fn):
    """Device milliseconds per kernel name of one call of fn (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type == torch.autograd.DeviceType.CUDA and ("k_sdr" in ev.key or "k_sis" in ev.key):
            name = ev.key.split("(")[0].split("::")[-1]
            out[name] = round(out.get(name, 0.0) + ev.device_time_total / 1e3, 4)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=8, help="32 x 4 s batches per Inferencer pass")
    ap.add_argument("--rounds", type=int, default=3, help="alternated Inferencer passes per metric list")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "sdr_bench needs a CUDA device"
    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info(), "filter_length": L, "shapes": []}

    for B, sec, reps in ((32, 4, 50), (4, 600, 5)):
        s1p, s2p, s1, s2 = signals(B, sec * SR, sec, dev)
        batch = dict(s1_pred=s1p, s2_pred=s2p, s1=s1, s2=s2, mix=s1 + s2)
        row = {"B": B, "seconds": sec}
        for name, m in (("sisdr", V.SISDRMetric()), ("sdr", V.SDRMetric(filter_length=L)),
                        ("sdri", V.SDRiMetric(filter_length=L))):
            m.device_value(**batch)
            torch.cuda.synchronize()
            ms = timed(lambda: m.device_value(**batch), reps)
            row[name] = {"device_value_ms": round(ms, 4), "audio_s_per_s": round(B * sec / (ms / 1e3), 1),
                         "kernels_ms": kernel_times(lambda: m.device_value(**batch))}
            if name != "sisdr":
                partners = 4 if name == "sdri" else 3
                fma = 2 * B * partners * sec * SR * L
                k = row[name]["kernels_ms"].get("k_sdr_corr")
                row[name]["corr_fp64_fma"] = fma
                row[name]["corr_fp64_tflops"] = round(2 * fma / (k / 1e3) / 1e12, 2) if k else None
        res["shapes"].append(row)
        print(json.dumps(row), flush=True)
        del s1p, s2p, s1, s2, batch
        torch.cuda.empty_cache()

    # evaluation loop: the same batches, [SISNRi] vs [SISNRi, SISDR, SDRi], alternated
    torch.manual_seed(42)
    net = V.DPTNAVWavEncDec(**MODEL_KW).eval().to(dev)
    B, T = 32, 4 * SR
    data = []
    for i in range(a.batches):
        s1p, s2p, s1, s2 = signals(B, T, 100 + i, dev)
        g = torch.Generator().manual_seed(200 + i)
        data.append({"mix": s1 + s2, "s1": s1, "s2": s2, "s1_embedding": torch.randn(B, 512, T // 640, generator=g).to(dev),
                     "s2_embedding": torch.randn(B, 512, T // 640, generator=g).to(dev)})
    lists = {"sisnri": lambda: [V.SISNRiMetric(name="SISNRi")],
             "sisnri_sisdr_sdri": lambda: [V.SISNRiMetric(name="SISNRi"), V.SISDRMetric(name="SISDR"),
                                           V.SDRiMetric(name="SDRi")]}
    loop = {k: [] for k in lists}
    for r in range(a.rounds + 1):
        for k, mk in lists.items():
            inf = V.Inferencer(net, {"inferencer": {}}, dev, {"test": [dict(d) for d in data]}, None,
                               metrics={"inference": mk()}, skip_model_load=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            inf.run_inference()   # ends in the tracker's device -> host read
            torch.cuda.synchronize()
            if r > 0:            # round 0 warms up
                loop[k].append(a.batches * B * T / SR / (time.perf_counter() - t0))
    res["inferencer"] = {"batches": a.batches, "batch": "32 x 4 s, DPTN-AV production shape",
                         "audio_s_per_s": {k: [round(v, 1) for v in vs] for k, vs in loop.items()},
                         "median_ratio_with_sdr": round(float(np.median(loop["sisnri_sisdr_sdri"]) /
                                                              np.median(loop["sisnri"])), 4)}
    print(json.dumps(res["inferencer"]), flush=True)

    # host context: the numpy / scipy restatement, six pairings of one 4 s utterance
    x = [t[0].cpu().double().numpy() for t in signals(1, 4 * SR, 7, "cpu")]
    x.append(x[2] + x[3])
    t0 = time.perf_counter()
    D.pit_all(D.sdr, *(v[None] for v in x), filter_length=L)
    res["cpu_oracle_ms_per_utterance_4s"] = {
        "ms": round((time.perf_counter() - t0) * 1e3, 2),
        "what": "oracle/sdr_oracle.py SDR of six pairings, fp64 numpy FFT + scipy solve_toeplitz (not torchmetrics)"}
    res["gpu_after"] = gpu_info()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
