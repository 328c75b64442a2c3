"""ctypes binding of libvatss_b200.so (the C ABI declared in include/vatss.h).

There is deliberately no fallback: if the shared library is missing or a tensor is not on a
CUDA device the call raises.  Build the library with `python -c "import __graft_entry__ as g;
g.build()"` or `make -C speech_separation_b200/csrc`.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# VATSS_LIB_OVERRIDE: experiments only (tools/build_variant.sh) - another build of the same library
LIB_PATH = os.environ.get("VATSS_LIB_OVERRIDE") or os.path.join(_HERE, "libvatss_b200.so")

KIND = {"dptn_av": 0, "dptn_wav": 1, "dptn_mask": 2, "dprnn": 3}
ENGINE = {"auto": 0, "generic": 1, "tensor": 2, "tensor-f16res": 3}

P_GLOBAL = [
    "encoder.weight", "decoder.weight", "visual_compression.weight", "visual_compression.bias", "gate",
    "video_ln.weight", "video_ln.bias", "dprnn.speakers_separation.0.weight",
    "dprnn.speakers_separation.1.weight", "dprnn.speakers_separation.1.bias",
    "HEAD_W", "HEAD_B", "dprnn.output_gate.0.weight", "dprnn.output_gate.0.bias",
]
S_DPTN = [
    "mha.in_proj_weight", "mha.in_proj_bias", "mha.out_proj.weight", "mha.out_proj.bias", "ln1.weight", "ln1.bias",
    "rnn.weight_ih_l0", "rnn.weight_hh_l0", "rnn.bias_ih_l0", "rnn.bias_hh_l0",
    "rnn.weight_ih_l0_reverse", "rnn.weight_hh_l0_reverse", "rnn.bias_ih_l0_reverse", "rnn.bias_hh_l0_reverse",
    "ffn.1.weight", "ffn.1.bias", "ln2.weight", "ln2.bias",
]
S_DPRNN = [
    None, None, None, None, None, None,
    "rnn.weight_ih_l0", "rnn.weight_hh_l0", "rnn.bias_ih_l0", "rnn.bias_hh_l0",
    "rnn.weight_ih_l0_reverse", "rnn.weight_hh_l0_reverse", "rnn.bias_ih_l0_reverse", "rnn.bias_hh_l0_reverse",
    "fc.weight", "fc.bias", "norm1d.weight", "norm1d.bias",
]


class ModelDesc(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in
                ("kind", "N", "K", "H", "num_blocks", "C", "P", "heads", "bidir", "E", "engine", "reserved")]


EXPORTS = {
    # name: (restype, argtypes)
    "vatss_last_error": (ctypes.c_char_p, []),
    "vatss_abi_version": (ctypes.c_int, []),
    "vatss_frames": (ctypes.c_int, [ctypes.POINTER(ModelDesc), ctypes.c_int]),
    "vatss_chunks": (ctypes.c_int, [ctypes.POINTER(ModelDesc), ctypes.c_int]),
    "vatss_workspace_bytes": (ctypes.c_size_t, [ctypes.POINTER(ModelDesc), ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "vatss_packed_weight_bytes": (ctypes.c_size_t, [ctypes.POINTER(ModelDesc)]),
    "vatss_pack_weights": (ctypes.c_int, [ctypes.POINTER(ModelDesc), ctypes.POINTER(ctypes.c_void_p), ctypes.c_int,
                                          ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "vatss_forward": (ctypes.c_int, [ctypes.POINTER(ModelDesc), ctypes.POINTER(ctypes.c_void_p), ctypes.c_int,
                                     ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                     ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                     ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "vatss_segment": (ctypes.c_int, [ctypes.c_void_p] + [ctypes.c_int] * 5 + [ctypes.c_void_p, ctypes.c_void_p]),
    "vatss_overlap_add": (ctypes.c_int, [ctypes.c_void_p] + [ctypes.c_int] * 5 + [ctypes.c_void_p, ctypes.c_void_p]),
    "vatss_encoder": (ctypes.c_int, [ctypes.POINTER(ModelDesc), ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p,
                                     ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "vatss_decoder": (ctypes.c_int, [ctypes.POINTER(ModelDesc), ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                     ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "vatss_tc_gemm": (ctypes.c_int, [ctypes.c_int, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p, ctypes.c_void_p,
                                     ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p, ctypes.c_void_p,
                                     ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p, ctypes.c_longlong,
                                     ctypes.c_int, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_void_p]),
    "vatss_tc_gemm_ln16": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p, ctypes.c_void_p,
                                          ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p, ctypes.c_void_p,
                                          ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p, ctypes.c_longlong,
                                          ctypes.c_int, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_int,
                                          ctypes.c_void_p]),
    "vatss_tc_lstm": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p] +
                      [ctypes.c_int] * 7 + [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "vatss_tc_attention": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 7 + [ctypes.c_void_p]),
    "vatss_generic_gemm": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_longlong] + [ctypes.c_void_p] * 4 +
                           [ctypes.c_longlong, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_longlong, ctypes.c_int,
                            ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "vatss_generic_layernorm": (ctypes.c_int, [ctypes.c_void_p] * 5 + [ctypes.c_longlong, ctypes.c_int, ctypes.c_int,
                                                                       ctypes.c_void_p]),
    "vatss_generic_attention": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 6 +
                                [ctypes.c_void_p]),
    "vatss_generic_lstm": (ctypes.c_int, [ctypes.c_void_p] * 4 + [ctypes.c_int] * 6 + [ctypes.c_void_p]),
    "vatss_tc_tail": (ctypes.c_int,[ctypes.POINTER(ModelDesc), ctypes.POINTER(ctypes.c_void_p), ctypes.c_int,
                                     ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t,
                                     ctypes.c_void_p]),
    "vatss_launch_count": (ctypes.c_ulonglong, []),
    "vatss_engine_fallback_reason": (ctypes.c_char_p, [ctypes.POINTER(ModelDesc)]),
    "vatss_debug_lstm_trace": (None, [ctypes.c_void_p]),
    "vatss_debug_cta_limit": (None, [ctypes.c_int]),
    "vatss_debug_lstm_pingpong": (None, [ctypes.c_int]),
    "vatss_debug_lstm_groups": (None, [ctypes.c_int]),
    "vatss_debug_tail_staged": (None, [ctypes.c_int]),
    "vatss_debug_gemm_l2_order": (None, [ctypes.c_int]),
    "vatss_debug_attention_version": (None, [ctypes.c_int]),
    "vatss_profile_begin": (ctypes.c_int, []),
    "vatss_profile_end": (ctypes.c_int, [ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_int), ctypes.c_int]),
    "vatss_sisnr_chunks": (ctypes.c_int, [ctypes.c_int]),
    "vatss_pit_sisnr": (ctypes.c_int, [ctypes.c_void_p] * 5 + [ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 5),
    "vatss_pit_sisdr": (ctypes.c_int, [ctypes.c_void_p] * 5 + [ctypes.c_int] * 3 + [ctypes.c_void_p] * 4),
    "vatss_sdr_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int] * 3),
    "vatss_sdr": (ctypes.c_int, [ctypes.c_void_p] * 5 + [ctypes.c_int] * 4 + [ctypes.c_double] + [ctypes.c_void_p] * 3 +
                  [ctypes.c_size_t, ctypes.c_void_p]),
    "vatss_pit_sisnr_backward": (ctypes.c_int, [ctypes.c_void_p] * 4 + [ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 6),
    "vatss_longform_windows": (ctypes.c_int, [ctypes.c_int] * 3),
    "vatss_window_cut": (ctypes.c_int, [ctypes.c_void_p] * 3 + [ctypes.c_int] * 9 + [ctypes.c_void_p] * 4),
    "vatss_window_stitch_scratch_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int]),
    "vatss_window_stitch": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 4 +
                            [ctypes.c_void_p] * 5 + [ctypes.c_size_t, ctypes.c_void_p]),
    "vatss_stoi_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int] * 3),
    "vatss_stoi": (ctypes.c_int, [ctypes.c_void_p] * 4 + [ctypes.c_int] * 4 + [ctypes.c_void_p] * 4 +
                   [ctypes.c_size_t, ctypes.c_void_p]),
    "vatss_debug_lipreader": (None, [ctypes.c_int]),
    "vatss_debug_lipreader_kernel": (None, [ctypes.c_int]),
    "vatss_debug_lipreader_trace": (None, [ctypes.c_void_p]),
    "vatss_debug_lipreader_capture": (None, [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int]),
    "vatss_lipreader_packed_bytes": (ctypes.c_size_t, []),
    "vatss_lipreader_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int] * 4),
    "vatss_lipreader_pack_weights": (ctypes.c_int, [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int, ctypes.c_int,
                                                    ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "vatss_lipreader_forward": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p] +
                                [ctypes.c_int] * 8 + [ctypes.c_float, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p,
                                                      ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p]),
}

_lib = None


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: the CUDA library is not built and there is no CPU fallback. "
            "Run `python -c 'import __graft_entry__ as g; g.build()'` at the repo root.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    if lib.vatss_abi_version() != 1:
        raise RuntimeError("libvatss_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().vatss_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (rc={rc}): {msg}")


def require_cuda(t, name):
    import torch

    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: speech_separation_b200 has no CPU path")
    return t


def f32c(t, name):
    """float32, contiguous CUDA tensor (no copy when already so)."""
    import torch

    require_cuda(t, name)
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def stream_ptr():
    import torch

    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


STAGES = ["frontend", "qkv", "attention", "outproj_ln1", "lstm_input", "lstm_recurrent", "ffn_ln2", "tail", "sisnr"]


class stage_profile:
    """Context manager: per-stage device milliseconds / launch counts of the calls made inside."""

    def __enter__(self):
        check(load().vatss_profile_begin(), "vatss_profile_begin")
        self.ms, self.launches = {}, {}
        return self

    def __exit__(self, *exc):
        ms = (ctypes.c_float * len(STAGES))()
        n = (ctypes.c_int * len(STAGES))()
        check(load().vatss_profile_end(ms, n, len(STAGES)), "vatss_profile_end")
        self.ms = {k: float(ms[i]) for i, k in enumerate(STAGES)}
        self.launches = {k: int(n[i]) for i, k in enumerate(STAGES)}
        return False
