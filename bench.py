#!/usr/bin/env python
"""Benchmark of the hot path: DPTN-AV separation forward (+ PIT SI-SNRi) in separated audio-seconds/s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|eager]
                    [--batch 32] [--seconds 4] [--engine auto|generic|tensor]
                    [--total-utterances 1024 --micro-batch 16]   (cfg-3: strong scaling of a fixed job over the ranks)
                    [--loss]                                     (cfg-5: forward + PIT SI-SNR loss, data-parallel mean)
                    [--dump-outputs DIR]                         (what the last timed step computed, as DIR/<name>.npy)

One "step" = one forward pass of DPTN-AV (src/configs/model/dptn_wav_av.yaml) over one batch of
synthetic 16 kHz mixtures + synthetic lip embeddings, followed by the PIT SI-SNRi reduction.
N=1 workload = BASELINE.json configs[1] (batch 32 x 4 s).  For N>1 (torchrun, one rank per GPU) every
rank processes its own batch of the same size (utterance sharding, weak scaling) and the ranks
all-reduce their SI-SNRi sums over NCCL each step - the path's only exchange.

Prints ONE JSON line (see the task contract): `value` = whole-job audio-s/s with inputs resident in
HBM; `e2e` = the same through the public nn.Module API from pinned host buffers (H2D + D2H inside
the timed region); `roofline` for the dominant stage; `cpu_baseline` = the torch-op CPU port of the
reference (oracle/torch_port.py) on the host cores for a bounded sample.
`--impl reference` times that CPU port as the reference arm.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR = 16000
CPU_SAMPLE_BATCH = 4     # BASELINE.md 3.1: the reference's CPU path is timed at a reduced batch of 4 utterances per step
MODEL_KW = dict(num_features=128, video_emb_size=512, hidden_video=128, kernel_size_enc=7, hidden_dim=128,
                num_blocks=6, chunk_size=150, step_size=75, num_heads=4, dropout=0.1, bidir=True)
# the other BASELINE.json configurations (src/configs/model/{dptn_wav,dptn,dprnn}.yaml)
OTHER_MODELS = {
    "dptn_wav": ("DPTNWavEncDec", dict(num_features=64, kernel_size_enc=7, hidden_dim=128, num_blocks=6, chunk_size=150,
                                       step_size=75, num_heads=4, dropout=0.1, bidir=True)),
    "dptn_mask": ("DPTNEncDec", dict(num_features=64, kernel_size_enc=7, hidden_dim=128, num_blocks=6, chunk_size=150,
                                     step_size=75, num_heads=4, dropout=0.1, bidir=True)),
    "dprnn": ("DPRNNEncDec", dict(num_features=64, kernel_size_enc=2, hidden_dim=128, num_blocks=6, chunk_size=250,
                                  step_size=125, bidir=True)),
}
METRIC = "dptn_av_separated_audio_seconds_per_second"
UNIT = "audio-s/s"
DUMP_LIMIT = 64 << 20    # bytes --dump-outputs writes at most, .npy headers included


def geometry(T):
    L = (T - 7) // 3 + 1
    S = (L - 150) // 75 + 1
    return L, S


def stage_flops(B, T, model="dptn_av"):
    """Algorithmic FLOPs (2MNK) per forward by stage (SURVEY.md §8a per-token figures)."""
    if model == "dprnn":
        L = (T - 2) // 1 + 1
        S = (L - 250) // 125 + 1
        tok = B * S * 250
        N, H = 64, 128
        return {"lstm_recurrent": 12 * tok * 2 * (N + H) * 8 * H, "ffn_ln2": 12 * tok * 2 * 2 * H * N,
                "tail": tok * 2 * N * 2 * N + 2 * B * L * (2 * N * N + 2 * N * 2), "frontend": B * L * 2 * N * 2,
                "qkv": 0, "attention": 0, "outproj_ln1": 0, "lstm_input": 0}
    L, S = geometry(T)
    tok = B * S * 150
    N, H = (128, 128) if model == "dptn_av" else (64, 128)
    per_sub = {
        "qkv": 2 * N * 3 * N,
        "outproj_ln1": 2 * N * N,
        "lstm_input": 2 * N * 8 * H,
        "lstm_recurrent": 2 * H * 8 * H,
        "ffn_ln2": 2 * 2 * H * N,
    }
    fl = {k: 12 * tok * v for k, v in per_sub.items()}
    fl["attention"] = 6 * tok * 4 * N * (150 + S)  # QK^T and PV, intra (len C) + inter (len S)
    fl["tail"] = tok * 2 * N * 2 * N + 2 * B * L * (2 * N * N + 2 * N * 7)
    fl["frontend"] = B * L * 2 * N * 7 + (2 * B * (T // 640) * 512 * N if model == "dptn_av" else 0)
    return fl


def stage_bytes(B, T, model="dptn_av", f16res=False):
    """Algorithmic HBM bytes per forward by stage (DESIGN.md 3: fp16 activations, block residual stream as an fp16 hi / lo pair)."""
    if model == "dprnn":
        return {}
    L, S = geometry(T)
    tok = B * S * 150
    N, H = (128, 128) if model == "dptn_av" else (64, 128)
    # block residual x: fp16 hi + fp16 lo pair (hi is the operand copy the projections read); the masking model keeps
    # fp32 + fp16 copies, the fp16-stream engine only hi
    lo = 0 if f16res else (4 * N if model == "dptn_mask" else 2 * N)   # bytes beyond the fp16 operand copy
    res_read = 2 * N if f16res else (4 * N if model == "dptn_mask" else 4 * N)   # what the out-projection reads of x
    per_sub = {
        "qkv": 2 * N + 2 * 3 * N,                                  # x16 in, qkv16 out
        "attention": 2 * 3 * N + 2 * N,                            # qkv16 in, att16 out
        "outproj_ln1": 2 * N + res_read + 2 * N,                   # att16 + residual x (hi + lo) in, y16 out
        "lstm_recurrent": 2 * 2 * N + 2 * 2 * H,                   # y16 read by both directions, ReLU(h) fp16 out
        "ffn_ln2": 2 * 2 * H + 2 * N + lo + 2 * N,                 # rnn16 + residual y16 in, x lo + x16 (hi) out
    }
    return {k: 12 * tok * v for k, v in per_sub.items()}


def ncu_traffic():
    """DRAM traffic per launch (dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture) of the
    headline workload's kernels, from profiles/ncu_traffic.json - a file written next to the capture it comes from,
    which names the commit and the kernel.  Not hard-coded here: a number from another kernel generation must not
    survive silently (VERDICT round 1).  Missing / unreadable file or stage -> None."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except (OSError, ValueError):
        return {}


def make_batch(B, T, seed):
    import torch

    g = torch.Generator().manual_seed(seed)
    s1 = 0.1 * torch.randn(B, T, generator=g)
    s2 = 0.1 * torch.randn(B, T, generator=g)
    Tv = 25 * T // SR
    e1 = torch.randn(B, 512, Tv, generator=g)
    e2 = torch.randn(B, 512, Tv, generator=g)
    return s1 + s2, s1, s2, e1, e2


def dump_outputs(arrays, out_dir):
    """Writes every tensor of `arrays` as out_dir/<name>.npy (float32, or float64 where the path computes in float64) so
    that two builds can be compared output for output.  Arrays of up to 1 MiB are written whole; above DUMP_LIMIT in all,
    each larger array is cut to the same fraction of its flattened elements, a fixed, seeded sample in ascending index
    order, identical from run to run."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    arrays = {k: a if a.dtype in (np.float32, np.float64) else a.astype(np.float32) for k, a in arrays.items()}
    large = {k for k, a in arrays.items() if a.nbytes > (1 << 20)}
    # 256 bytes bound one .npy header
    budget = DUMP_LIMIT - 256 * len(arrays) - sum(a.nbytes for k, a in arrays.items() if k not in large)
    total = sum(arrays[k].nbytes for k in large)
    for name, a in arrays.items():
        if name in large and total > budget:
            n = a.size * budget // total
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, n, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "200", "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons, power = [], [], set(), []
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); power.append(float(c[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        if sm:
            sm_sorted = sorted(sm)
            out.update(sm_mhz=sm_sorted[len(sm) // 2], sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm),
                       power_w_max=max(power))
        return out


def cpu_reference_arm(steps, warmup, B_sample, T, model="dptn_av"):
    """The reference's CPU path (torch-op port) on the host cores; returns (audio-s/s, ms/step, info)."""
    import torch

    import speech_separation_b200 as V
    from oracle import torch_port

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(42)
    if model == "dptn_av":
        net = V.DPTNAVWavEncDec(**MODEL_KW).eval()
    else:
        net = getattr(V, OTHER_MODELS[model][0])(**OTHER_MODELS[model][1]).eval()
    mix, s1, s2, e1, e2 = make_batch(B_sample, T, 1234)
    if model != "dptn_av":
        e1 = e2 = None
    for _ in range(warmup):
        torch_port.forward(net, mix, e1, e2)
    t0 = time.perf_counter()
    for _ in range(steps):
        torch_port.forward(net, mix, e1, e2)
    dt = (time.perf_counter() - t0) / max(steps, 1)
    val = B_sample * T / SR / dt
    info = {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{B_sample} utterance(s) x {T / SR:g} s of the same workload per step, fp32 torch ops "
                      f"(oracle/torch_port.py), {steps} step(s) after {warmup} warm-up"}
    return val, dt * 1e3, info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "eager"])
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--seconds", type=float, default=4.0)
    ap.add_argument("--engine", default="auto", choices=["auto", "generic", "tensor", "tensor-f16res"])
    ap.add_argument("--model", default="dptn_av", choices=["dptn_av"] + sorted(OTHER_MODELS),
                    help="dptn_av = the headline config; the others are the remaining BASELINE.json models")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--no-lipreader", action="store_true", help="skip the lipreader front-end side measurement")
    ap.add_argument("--total-utterances", type=int, default=0,
                    help="cfg-3: a fixed job of this many utterances, sharded over the ranks (strong scaling)")
    ap.add_argument("--micro-batch", type=int, default=32)
    ap.add_argument("--loss", action="store_true", help="cfg-5: every step also computes the PIT SI-SNR loss")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (separated waveforms, SI-SNR rows and summary, loss) as DIR/<name>.npy; "
                         "the inputs are seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    B, T = args.batch, int(round(args.seconds * SR))
    wname = {"dptn_av": "DPTN-AV (dptn_wav_av.yaml)", "dptn_wav": "DPTN audio-only (dptn_wav.yaml)",
             "dptn_mask": "DPTN masking (dptn.yaml)", "dprnn": "DPRNN (dprnn.yaml)"}[args.model]
    config = {"workload": f"{wname} inference, batch {B} x {args.seconds:g} s 16 kHz per GPU, "
                          + (f"synthetic lip embeddings (B,512,{25 * T // SR}), " if args.model == "dptn_av" else "")
                          + "random-init weights seed 42, + PIT SI-SNRi reduction",
              "batch_per_gpu": B, "seconds": args.seconds, "sharding": f"utterance x{max(world, args.gpus)}",
              "l2": "256 MiB buffer written between timed steps (L2 flush); per-step activations >> 126 MB L2",
              "reference_arm_sample": f"--impl reference and cpu_baseline time {CPU_SAMPLE_BATCH} utterance(s) x "
                                      f"{args.seconds:g} s of this workload per step on the host cores (BASELINE.md 3.1)"}
    if args.total_utterances:
        config["workload"] = (f"{wname} inference, {args.total_utterances} x {args.seconds:g} s 16 kHz sharded by utterance over "
                              f"the ranks, micro-batches of {args.micro_batch}, NCCL all-reduce of the SI-SNRi sums per step, "
                              "synthetic lip embeddings, random-init weights seed 42")
        config["total_utterances"] = args.total_utterances
        config["micro_batch"] = args.micro_batch
    if args.loss:
        config["workload"] += " + PIT SI-SNR loss (SiSNRWavLoss), data-parallel mean over the ranks"

    if args.impl == "reference":
        if rank != 0:
            return 0
        # bounded sample: CPU_SAMPLE_BATCH utterances per step keep K steps within minutes on the host cores
        val, ms, info = cpu_reference_arm(max(args.steps, 1), min(args.warmup, 1), CPU_SAMPLE_BATCH, T, args.model)
        print(json.dumps({"metric": METRIC.replace("dptn_av", args.model), "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                          "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                          "impl": "reference", "cpu_baseline": info, "gpu_launches": 0,
                          "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0

    if args.impl == "eager":
        # SURVEY.md 8(d): the same stock torch.nn modules on one B200 ("library Blackwell kernels": cuDNN LSTM, fused
        # MHA, cuBLAS) - a second reported baseline, not part of the driver contract.  fp32 with torch's default TF32 flags.
        if rank != 0:
            return 0
        import torch

        import speech_separation_b200 as V
        from oracle import torch_port
        dev = torch.device("cuda", local_rank)
        torch.manual_seed(42)
        net = (V.DPTNAVWavEncDec(**MODEL_KW) if args.model == "dptn_av"
               else getattr(V, OTHER_MODELS[args.model][0])(**OTHER_MODELS[args.model][1])).eval().to(dev)
        mix, s1, s2, e1, e2 = (t.to(dev) for t in make_batch(B, T, 1234))
        if args.model != "dptn_av":
            e1 = e2 = None
        for _ in range(max(args.warmup, 3)):
            torch_port.forward(net, mix, e1, e2)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.steps):
            torch_port.forward(net, mix, e1, e2)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / args.steps
        print(json.dumps({"metric": METRIC.replace("dptn_av", args.model), "value": B * T / SR / (ms * 1e-3), "unit": UNIT,
                          "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
                          "higher_is_better": True, "dtype": "f32 (TF32 defaults)", "data": "synthetic", "config": config,
                          "impl": "eager_torch_gpu", "peak_mem_gb": torch.cuda.max_memory_allocated() / 2**30}))
        return 0

    import torch
    import torch.distributed as dist

    import speech_separation_b200 as V
    from speech_separation_b200 import _lib
    from speech_separation_b200.sharding import all_reduce_sisnr_sums, separate_in_micro_batches, shard_range, sisnr_sums

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    torch.manual_seed(42)
    av = args.model == "dptn_av"
    if av:
        net = V.DPTNAVWavEncDec(**MODEL_KW)
    else:
        net = getattr(V, OTHER_MODELS[args.model][0])(**OTHER_MODELS[args.model][1])
    net = net.eval().to(dev).set_engine(args.engine)
    metric = V.SISNRiMetric()
    loss_fn = V.SiSNRWavLoss()
    sharded_job = args.total_utterances > 0
    if sharded_job:     # cfg-3: this rank's contiguous shard of the fixed job, streamed through one workspace
        lo, hi = shard_range(args.total_utterances, rank, world)
        B = hi - lo
    mix_h, s1_h, s2_h, e1_h, e2_h = (t.pin_memory() for t in make_batch(B, T, 1234 + rank))
    mix, s1, s2, e1, e2 = (t.to(dev) for t in (mix_h, s1_h, s2_h, e1_h, e2_h))
    out_h = [torch.empty(B, T).pin_memory() for _ in range(2)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def fwd(m, a, b):
        if sharded_job:
            return separate_in_micro_batches(net, m, a if av else None, b if av else None, micro_batch=args.micro_batch)
        return net(mix=m, s1_embedding=a, s2_embedding=b) if av else net(mix=m)

    def step_loss(out):
        """cfg-5: batch-level PIT SI-SNR loss of this rank's batch; data-parallel mean over the ranks (NCCL)."""
        loss = loss_fn(s1_pred=out["s1_pred"], s2_pred=out["s2_pred"], s1=s1, s2=s2)["loss"]
        if world > 1:
            loss = loss.clone()
            dist.all_reduce(loss)
            loss = loss / world
        return loss

    last = {}    # what the latest step computed, for --dump-outputs

    def step_resident():
        out = fwd(mix, e1, e2)
        rows, rows_loss, summary = V.pit_sisnr_all(out["s1_pred"], out["s2_pred"], s1, s2, mix)
        last.update(s1_pred=out["s1_pred"], s2_pred=out["s2_pred"], sisnr_rows=rows, sisnr_loss_rows=rows_loss,
                    sisnr_summary=summary)
        if args.loss:
            last["loss"] = step_loss(out)
        # N > 1: the NCCL all-reduce of the SI-SNR sums is issued every step, stream-ordered; the reduced vector stays on
        # the device (an evaluation loop reads it once per partition, not once per batch)
        if world > 1:
            last["sisnr_sums"] = all_reduce_sisnr_sums(sisnr_sums(rows, rows_loss))
            return last["sisnr_sums"]
        return rows

    # End-to-end step through the public nn.Module / metric API from PINNED HOST buffers.  Input copies are double
    # buffered the way an evaluation loop over a DataLoader runs (speech_separation_b200.Inferencer): while step k
    # computes, the inputs of step k + 1 travel host -> device on a second stream.  Every copy lies inside the timed
    # region (step k's interval contains the copy for step k + 1; K steps contain K input copies and K output copies).
    copy_stream = torch.cuda.Stream(dev)
    pending = []

    def issue_inputs():
        with torch.cuda.stream(copy_stream):
            ts = tuple(x.to(dev, non_blocking=True) for x in (mix_h, e1_h, e2_h))
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return ts, ev

    def step_e2e():
        if not pending:
            pending.append(issue_inputs())
        (m, a, b), ev = pending.pop()
        cur = torch.cuda.current_stream()
        cur.wait_event(ev)
        for t in (m, a, b):
            t.record_stream(cur)
        pending.append(issue_inputs())
        out = fwd(m, a, b)
        out_h[0].copy_(out["s1_pred"], non_blocking=True)
        out_h[1].copy_(out["s2_pred"], non_blocking=True)
        val = metric(s1_pred=out["s1_pred"], s2_pred=out["s2_pred"], s1=s1, s2=s2, mix=m)
        if args.loss:
            return float(step_loss(out))
        return float(val)  # device -> host read of the step's metric (synchronises)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """Per-step CUDA events on the current stream, L2 flush between steps (outside the events)."""
        evs = []
        barrier()
        wall0 = time.perf_counter()
        for _ in range(steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            evs.append((a, b))
        barrier()
        wall = time.perf_counter() - wall0
        total_ms = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), wall

    for _ in range(max(args.warmup, 3)):
        step_resident()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = lib.vatss_launch_count()
    total_ms, wall = timed(step_resident, args.steps)
    launches = lib.vatss_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else {}
    if args.dump_outputs and rank == 0:
        dump_outputs(last, args.dump_outputs)

    for _ in range(2):
        step_e2e()
    e2e_ms, _ = timed(step_e2e, args.steps)

    # per-stage device time (CUDA events recorded by the library on the launching stream)
    with _lib.stage_profile() as prof:
        for _ in range(2):
            step_resident()
        torch.cuda.synchronize()
    stage_ms = {k: v / 2 for k, v in prof.ms.items()}
    stage_launches = {k: v // 2 for k, v in prof.launches.items()}

    # parity signal carried with the number: SI-SNRi of this rank's batch
    with torch.no_grad():
        out = fwd(mix, e1, e2)
        snri = float(metric(s1_pred=out["s1_pred"], s2_pred=out["s2_pred"], s1=s1, s2=s2, mix=mix))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    n = max(world, 1)
    audio_s_per_step = (args.total_utterances if sharded_job else n * B) * T / SR
    ms_per_step = total_ms / args.steps
    value = audio_s_per_step / (ms_per_step / 1e3)
    e2e_value = audio_s_per_step / (e2e_ms / args.steps / 1e3)

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_bw = float(peaks.get("hbm_gbs", 6500.0))
    fl = stage_flops(B, T, args.model)
    by = stage_bytes(B, T, args.model, args.engine == "tensor-f16res")
    if stage_ms.get("lstm_input", 0.0) == 0.0:   # tensor engine: input and recurrent contractions are one kernel
        fl["lstm_recurrent"] = fl.get("lstm_recurrent", 0) + fl.pop("lstm_input", 0)
        fl["lstm_input"] = 0
    # per stage: achieved rate against both roofs (algorithmic work / CUDA-event time of the stage's launches);
    # the binding roof of a stage is the one it is closer to
    stages = {}
    for k, ms in stage_ms.items():
        if ms <= 0 or k in ("frontend", "tail", "sisnr", "lstm_input"):
            continue
        tf = fl.get(k, 0) / (ms / 1e3) / 1e12
        gb = by.get(k, 0) / (ms / 1e3) / 1e9
        stages[k] = {"ms": round(ms, 3), "launches": int(stage_launches.get(k, 0)), "tflops": round(tf, 1),
                     "tensor_frac": round(tf / peak_tf, 3), "gbs": round(gb, 1), "hbm_frac": round(gb / peak_bw, 3)}
    dom = max(stages, key=lambda k: stages[k]["ms"])
    d = stages[dom]
    dom_launches = max(d["launches"], 1)
    hbm_bound = d["hbm_frac"] >= d["tensor_frac"]
    headline = args.model == "dptn_av" and B == 32 and abs(args.seconds - 4.0) < 1e-9 and args.engine in ("auto", "tensor")
    roofline = {"bound": "hbm" if hbm_bound else "tensor", "kernel": dom,
                "achieved": d["gbs"] if hbm_bound else d["tflops"], "peak": peak_bw if hbm_bound else peak_tf,
                "unit": "GB/s" if hbm_bound else "TFLOP/s", "frac": d["hbm_frac"] if hbm_bound else d["tensor_frac"],
                "traffic": (ncu_traffic().get("kernels", {}).get(dom, {}).get("dram_bytes_per_launch") if headline else None),
                "traffic_source": (ncu_traffic().get("source") if headline else None),
                "algorithmic_bytes_per_launch": by.get(dom, 0) / dom_launches,
                "algorithmic_flops_per_launch": fl.get(dom, 0) / dom_launches,
                "peak_source": ("MEASURED_PEAKS.json hbm_gbs / bf16_tflops_sustained" if peaks
                                else "fallback 6.5 TB/s / 1.4 PFLOP/s sustained"),
                "launches_per_step": dom_launches, "ms_per_step": d["ms"],
                "note": "attention and the LSTM are bound by MUFU / synchronisation latency rather than by either roof "
                        "(DESIGN.md 3.2-3.4); the GEMM stages are HBM-bound",
                "whole_forward_frac": sum(fl.values()) / (sum(stage_ms[k] for k in fl) / 1e3) / 1e12 / peak_tf,
                "stages": stages,
                "stage_ms": {k: round(v, 3) for k, v in stage_ms.items()}}

    line = {"metric": METRIC.replace("dptn_av", args.model), "value": value, "unit": UNIT, "n_gpus": n, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if sharded_job else "weak", "vs_baseline": None,
            "dtype": "f32" if args.engine == "generic" or not _engine_is_tensor(lib, net) else "f16",
            "data": "synthetic", "config": config, "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT,
                    "h2d_bytes_per_step": int(mix_h.numel() + (e1_h.numel() + e2_h.numel() if av else 0)) * 4,
                    "d2h_bytes_per_step": int(2 * B * T) * 4 + 4,
                    "note": "bytes of rank 0; mixture + lip embeddings host->device and both separated waveforms + the "
                            "metric device->host every step; the ground-truth sources s1, s2 (metric inputs only) stay resident; "
                            "the input copy of step k+1 runs on a second stream while step k computes (double-buffered, inside the timed region)"},
            "gpu_launches": int(launches), "roofline": roofline, "si_snri_db": snri, "wall_s_timed": wall}
    if world == 1 and not args.no_eager_baseline and not sharded_job:
        # SURVEY.md 8(d): the reference's own torch.nn modules on this GPU (cuDNN LSTM, fused MHA, cuBLAS; fp32 with
        # torch's default TF32 flags) - the "existing Blackwell library kernels" bar, 3 steps after 2 warm-ups
        try:
            from oracle import torch_port
            ea, eb_ = (e1, e2) if av else (None, None)
            for _ in range(2):
                torch_port.forward(net, mix, ea, eb_)
            torch.cuda.synchronize()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(3):
                torch_port.forward(net, mix, ea, eb_)
            t1.record()
            torch.cuda.synchronize()
            ems = t0.elapsed_time(t1) / 3
            line["eager_gpu_baseline"] = {"value": B * T / SR / (ems * 1e-3), "unit": UNIT, "ms_per_step": ems,
                                          "what": "the same torch.nn modules (oracle/torch_port.py) in eager PyTorch on this GPU, "
                                                  "forward only, fp32 / TF32 defaults, 3 steps after 2 warm-ups"}
        except Exception as e:   # a baseline must never take the bench line down
            line["eager_gpu_baseline"] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
        torch.cuda.empty_cache()
    if world == 1 and av and not args.no_lipreader and not sharded_job:
        # SURVEY.md 8f rank 4: the lipreader front end that produces this batch's lip embeddings from raw mouth crops
        # (2 speakers x B clips x Tv frames of 96 x 96), timed beside the separation step; not part of `value`
        try:
            from speech_separation_b200 import Lipreading, extract_embeddings
            torch.manual_seed(7)
            lip = Lipreading(relu_type="swish", extract_feats=True).to(dev)
            Tv = 25 * T // SR
            video = (torch.rand(2 * B, Tv, 96, 96, device=dev) * 255).round()
            for _ in range(2):
                extract_embeddings(lip, video)
            torch.cuda.synchronize()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n0 = lib.vatss_launch_count()
            t0.record()
            for _ in range(3):
                emb = extract_embeddings(lip, video)
            t1.record()
            torch.cuda.synchronize()
            lms = t0.elapsed_time(t1) / 3
            frames = 2 * B * Tv
            line["lipreader_frontend"] = {
                "frames_per_s": frames / (lms * 1e-3), "ms_per_batch_video": lms, "frames": frames,
                "tflops": frames * 632317952 / (lms * 1e-3) / 1e12, "gpu_launches": int(lib.vatss_launch_count() - n0),
                "output": list(emb.shape), "engine": "tensor (tcgen05 trunk, fp16 activations)",
                "what": "Lipreading(video, resnet, swish, extract_feats=True) on raw 96 x 96 mouth crops of this batch "
                        "(crop + normalisation folded into the first kernel), 3 runs after 2 warm-ups; 632.3 MFLOP per frame"}
            del lip, video, emb
        except Exception as e:   # a side measurement must never take the bench line down
            line["lipreader_frontend"] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
        torch.cuda.empty_cache()
    if world == 1 and not args.no_cpu_baseline:
        _, _, info = cpu_reference_arm(2, 1, CPU_SAMPLE_BATCH, T, args.model)
        line["cpu_baseline"] = info
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def _engine_is_tensor(lib, net):
    import ctypes

    return lib.vatss_packed_weight_bytes(ctypes.byref(net._desc)) > 0


if __name__ == "__main__":
    sys.exit(main())
