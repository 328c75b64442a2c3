"""CPU-side tests: the C ABI library loads and exports every declared symbol, the host-side
mirror of the reference interface behaves, and the multi-rank reduction logic is right (gloo)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="session")
def lib():
    from speech_separation_b200 import _lib

    if not os.path.isfile(_lib.LIB_PATH):
        import __graft_entry__ as g

        g.build()
    return _lib.load()


def test_every_declared_symbol_is_exported(lib):
    hdr = open(os.path.join(ROOT, "include", "vatss.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(vatss_[a-z_0-9]+)\s*\(", hdr))
    assert len(names) >= 14
    from speech_separation_b200 import _lib

    for n in sorted(names):
        assert hasattr(lib, n), f"{n} declared in include/vatss.h but not exported"
        assert n in _lib.EXPORTS, f"{n} has no ctypes prototype"
    assert lib.vatss_abi_version() == 1


def test_geometry_matches_reference_index_maths(lib):
    from speech_separation_b200 import _lib
    from oracle.vatss_oracle import PathConfig

    for (K, C, P, T, L, S) in [(7, 150, 75, 64000, 21332, 283), (7, 150, 75, 160000, 53332, 710),
                               (2, 250, 125, 64000, 63999, 510), (7, 150, 75, 32000, 10665, 141)]:
        d = _lib.ModelDesc(kind=1, N=64, K=K, H=128, num_blocks=6, C=C, P=P, heads=4, bidir=1, E=0, engine=0)
        assert lib.vatss_frames(ctypes.byref(d), T) == L
        assert lib.vatss_chunks(ctypes.byref(d), L) == S
        cfg = PathConfig(kind="dptn_wav", kernel_size_enc=K, chunk_size=C, step_size=P)
        assert cfg.frames(T) == L and cfg.chunks(L) == S


def test_bad_arguments_report_errors(lib):
    from speech_separation_b200 import _lib

    d = _lib.ModelDesc(kind=9, N=64, K=7, H=128, num_blocks=6, C=150, P=75, heads=4, bidir=1, E=0, engine=0)
    assert lib.vatss_workspace_bytes(ctypes.byref(d), 1, 16000, 0) == 0
    assert b"unknown model kind" in lib.vatss_last_error()
    d.kind = 1
    assert lib.vatss_workspace_bytes(ctypes.byref(d), 1, 100, 0) == 0  # shorter than one chunk
    assert b"shorter than one chunk" in lib.vatss_last_error()
    assert lib.vatss_workspace_bytes(ctypes.byref(d), 4, 64000, 0) > 0
    assert lib.vatss_segment(None, 1, 1, 5, 10, 5, None, None) != 0
    # no dual-path blocks: AUTO falls back to the generic engine and says why
    assert lib.vatss_engine_fallback_reason(ctypes.byref(d)) is None
    d.num_blocks = 0
    assert b"no dual-path blocks" in lib.vatss_engine_fallback_reason(ctypes.byref(d))
    assert lib.vatss_packed_weight_bytes(ctypes.byref(d)) == 0


def test_state_dict_layout_and_init_match_reference_checksum(golden_dir):
    import speech_separation_b200 as V

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle.gen_golden import PROD, state_checksum

    for kind, cls in [("dptn_av", V.DPTNAVWavEncDec), ("dptn_wav", V.DPTNWavEncDec), ("dptn_mask", V.DPTNEncDec),
                      ("dprnn", V.DPRNNEncDec)]:
        torch.manual_seed(42)
        net = cls(**PROD[kind])
        z = np.load(os.path.join(golden_dir, f"prod_{kind}_B2_T16000.npz"))
        assert abs(state_checksum(net.state_dict()) - float(z["weight_checksum"])) < 1e-9
    n = sum(p.numel() for p in V.DPTNAVWavEncDec(**PROD["dptn_av"]).parameters())
    assert n == 4448194  # SURVEY.md §6
    assert "All parameters: 4448194" in str(V.DPTNAVWavEncDec(**PROD["dptn_av"]))


def test_tiny_reference_state_dict_loads(golden_dir):
    import speech_separation_b200 as V

    z = np.load(os.path.join(golden_dir, "tiny_dptn_av.npz"))
    kw = {k: v for k, v in zip(z["cfg_keys"], z["cfg_vals"])}
    net = V.DPTNAVWavEncDec(num_features=int(kw["num_features"]), video_emb_size=int(kw["video_emb_size"]),
                            hidden_video=int(kw["hidden_video"]), kernel_size_enc=int(kw["kernel_size_enc"]),
                            hidden_dim=int(kw["hidden_dim"]), num_blocks=int(kw["num_blocks"]),
                            chunk_size=int(kw["chunk_size"]), step_size=int(kw["step_size"]),
                            num_heads=int(kw["num_heads"]), bidir=bool(kw["bidir"]))
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}
    missing, unexpected = net.load_state_dict(sd, strict=True)
    assert not missing and not unexpected


def test_no_cpu_fallback():
    import speech_separation_b200 as V

    net = V.DPTNWavEncDec(num_features=8, kernel_size_enc=4, hidden_dim=8, num_blocks=1, chunk_size=12, step_size=6,
                          num_heads=2)
    with pytest.raises(RuntimeError, match="no CPU path"):
        net(mix=torch.zeros(1, 400))
    with pytest.raises(RuntimeError, match="no CPU path"):
        V.SiSNRWavLoss()(s1_pred=torch.zeros(1, 8), s2_pred=torch.zeros(1, 8), s1=torch.zeros(1, 8), s2=torch.zeros(1, 8))
    with pytest.raises(RuntimeError, match="no CPU path"):
        V.SplitToFolds(4, 2)(torch.zeros(1, 1, 8))


def test_product_package_never_imports_oracle():
    pkg = os.path.join(ROOT, "speech_separation_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert "oracle" not in src.replace("the CPU oracle", ""), f"{f} mentions the oracle"


def test_shard_range_partitions():
    from speech_separation_b200.sharding import shard_range

    for n in (0, 1, 7, 32, 1024, 1025):
        for w in (1, 2, 3, 4, 8):
            spans = [shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(w - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_range(4, 2, 2)


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist

    from oracle import vatss_oracle as O
    from speech_separation_b200.sharding import reduce_sisnr, shard_range, sisnr_sums

    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    g = np.random.default_rng(3)
    n, T = 10, 600
    s1, s2 = g.standard_normal((n, T)), g.standard_normal((n, T))
    s1p = s1 + 0.3 * g.standard_normal((n, T))
    s2p = s2 + 0.5 * g.standard_normal((n, T))
    s1p[3], s2p[3] = s2p[3].copy(), s1p[3].copy()  # one utterance with swapped speakers
    mix = s1 + s2
    pairs = [(s1p, s1), (s2p, s2), (s1p, s2), (s2p, s1), (mix, s1), (mix, s2)]
    rows = np.stack([O.si_snr_metric_rows(a, b) for a, b in pairs], axis=1)
    rows_loss = np.stack([O.sisnr_loss_rows(a, b) for a, b in pairs[:4]], axis=1)
    lo, hi = shard_range(n, rank, world)
    out = reduce_sisnr(sisnr_sums(torch.from_numpy(rows[lo:hi]), torch.from_numpy(rows_loss[lo:hi])))
    # the stream-ordered form (vector left on the device, read once): two steps accumulate to twice the sums, and the
    # metrics derived from them are those of the one-shot reduction
    from speech_separation_b200.sharding import all_reduce_sisnr_sums, metrics_from_sums
    red = all_reduce_sisnr_sums(sisnr_sums(torch.from_numpy(rows[lo:hi]), torch.from_numpy(rows_loss[lo:hi])))
    acc = red + all_reduce_sisnr_sums(sisnr_sums(torch.from_numpy(rows[lo:hi]), torch.from_numpy(rows_loss[lo:hi])))
    assert metrics_from_sums(red.tolist()) == out
    twice = metrics_from_sums(acc.tolist())
    assert twice["count"] == 2 * out["count"] and abs(twice["si_snri_batch_pit"] - out["si_snri_batch_pit"]) < 1e-12
    if rank == 0:
        q.put((out, O.pit_si_snri(s1p, s2p, s1, s2, mix), O.pit_sisnr_loss(s1p, s2p, s1, s2),
               float(np.mean(np.maximum((rows[:, 0] + rows[:, 1]) / 2, (rows[:, 2] + rows[:, 3]) / 2)
                             - (rows[:, 4] + rows[:, 5]) / 2))))
    dist.destroy_process_group()


def test_world_size_2_reduction_matches_single_process():
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out, snri, loss, utt = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert out["count"] == 10
    assert abs(out["si_snri_batch_pit"] - snri) < 1e-9
    assert abs(out["loss_batch_pit"] - loss) < 1e-9
    assert abs(out["si_snri_utt_pit"] - utt) < 1e-9
    assert out["si_snri_utt_pit"] > out["si_snri_batch_pit"]  # per-utterance PIT can only help


def test_header_is_plain_c_and_a_c_program_links_against_the_library(tmp_path):
    """The boundary is a C ABI: include/vatss.h must compile as C99 (no C++-isms, no torch types) and a C program must link
    against libvatss_b200.so and call the entry points that need no GPU."""
    import shutil
    import subprocess

    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    hdr = os.path.join(ROOT, "include", "vatss.h")
    subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-fsyntax-only", "-x", "c", hdr], check=True)
    src = tmp_path / "abi.c"
    src.write_text(
        '#include <stdio.h>\n#include "vatss.h"\n'
        "int main(void) {\n"
        "  vatss_model_desc d = {VATSS_KIND_DPTN_AV, 128, 7, 128, 6, 150, 75, 4, 1, 512, VATSS_ENGINE_AUTO, 0};\n"
        "  int L = vatss_frames(&d, 64000), S = vatss_chunks(&d, L);\n"
        '  printf("%d %d %d %d %zu\\n", vatss_abi_version(), L, S, vatss_sisnr_chunks(64000), vatss_lipreader_packed_bytes());\n'
        "  return (L == 21332 && S == 283 && vatss_abi_version() == VATSS_ABI_VERSION) ? 0 : 1;\n}\n")
    exe = tmp_path / "abi"
    libdir = os.path.join(ROOT, "speech_separation_b200")
    subprocess.run([gcc, "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                    os.path.join(libdir, "libvatss_b200.so"), f"-Wl,-rpath,{libdir}"], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    assert out[:4] == ["1", "21332", "283", "8"] and int(out[4]) > 0
