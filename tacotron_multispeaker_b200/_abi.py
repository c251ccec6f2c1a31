"""ctypes binding of ``libtaco_b200.so`` (C ABI in ``include/taco_b200.h``).

There is no fallback: if the shared object is missing or cannot be loaded the
import of the product path raises.  PyTorch is only used by the callers for
device memory and streams; nothing here touches torch.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtaco_b200.so")

TACO_OK = 0
TACO_ERR_INVALID = -1
TACO_ERR_CUDA = -2
TACO_ERR_MISSING_WEIGHT = -3
TACO_ERR_STATE = -4
TACO_ERR_OOB_ID = -5
TACO_ERR_UNSUPPORTED = -6

BN_MOVING, BN_BATCH = 0, 1
ACT_NONE, ACT_RELU, ACT_SIGMOID, ACT_TANH = 0, 1, 2, 3
CBHG_ENCODER, CBHG_POST = 0, 1
GEMM_BF16X3, GEMM_BF16 = 1, 2

# Every symbol include/taco_b200.h declares (tests check the library exports all of them).
SYMBOLS = [
    "taco_create", "taco_destroy", "taco_last_error", "taco_version",
    "taco_set_weight", "taco_finalize_weights", "taco_num_weights", "taco_weight_name",
    "taco_max_steps", "taco_forward", "taco_forward_host", "taco_forward_host_begin", "taco_forward_host_wait",
    "taco_forward_host_end",
    "taco_embed", "taco_check_ids", "taco_encoder", "taco_decode", "taco_cbhg", "taco_postnet",
    "taco_bigru", "taco_conv1d", "taco_maxpool_affine", "taco_bn_batch_stats",
    "taco_set_gemm_mode", "taco_launch_count", "taco_decoder_geometry", "taco_set_decoder_clusters", "taco_set_profiling", "taco_last_stage_ms", "taco_set_cuda_graphs",
    "taco_wav_length", "taco_griffin_lim", "taco_spectrogram_frames", "taco_spectrogram",
    "taco_resample_length", "taco_resample_positions", "taco_resample", "taco_durations",
    "taco_umma_plan", "taco_gemm_unit", "taco_highway4_unit", "taco_bigru_unit", "taco_decoder_plan",
]


class TacoHParams(C.Structure):
    _fields_ = [
        ("num_mels", C.c_int32), ("num_freq", C.c_int32), ("outputs_per_step", C.c_int32),
        ("max_iters", C.c_int32), ("embedding_text_channels", C.c_int32),
        ("embedding_id_channels", C.c_int32), ("num_symbols", C.c_int32), ("id_num", C.c_int32),
    ]


class TacoAudioParams(C.Structure):
    _fields_ = [
        ("sample_rate", C.c_int32), ("griffin_lim_iters", C.c_int32),
        ("frame_length_ms", C.c_double), ("frame_shift_ms", C.c_double), ("preemphasis", C.c_double),
        ("min_level_db", C.c_double), ("ref_level_db", C.c_double), ("power", C.c_double),
    ]


class TacoGemmDesc(C.Structure):
    """``taco_gemm_desc``: one dense / conv GEMM with its epilogue (pointers as integers)."""
    _fields_ = [
        ("x", C.c_void_p), ("x_bs", C.c_int64), ("ldx", C.c_int32),
        ("x_hi", C.c_void_p), ("x_lo", C.c_void_p),
        ("N", C.c_int32), ("T", C.c_int32), ("Cin", C.c_int32), ("taps", C.c_int32), ("bank", C.c_int32),
        ("Cout", C.c_int32),
        ("w_host", C.c_void_p), ("bias_host", C.c_void_p),
        ("scale_host", C.c_void_p), ("shift_host", C.c_void_p),
        ("res", C.c_void_p), ("res_bs", C.c_int64), ("ldres", C.c_int32),
        ("act", C.c_int32),
        ("out", C.c_void_p), ("out_bs", C.c_int64), ("ldo", C.c_int32), ("col_off", C.c_int32),
        ("out_hi", C.c_void_p), ("out_lo", C.c_void_p), ("out_cp", C.c_int32),
    ]


class TacoGemmPlan(C.Structure):
    """``taco_gemm_plan``: the launch shape of a tensor-core GEMM."""
    _fields_ = [(n, C.c_int32) for n in ("valid", "tiles", "ctas", "persistent", "long_k", "stages", "epi_warps",
                                         "acc_cols", "vec_epi", "variant", "smem_bytes")]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class TacoDecoderPlan(C.Structure):
    """``taco_decoder_plan_t``: how the default decoder runs a batch (clusters, residency of the attention operands)."""
    _fields_ = [(n, C.c_int32) for n in ("valid", "clusters", "s_max", "att_res", "ring_kb", "smem_bytes")]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class TacoError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("taco_b200 error %d: %s" % (code, msg))
        self.code = code


_lib = None


def load() -> C.CDLL:
    """Load the CUDA library; raise (never fall back) if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libtaco_b200.so is not built (%s). Run `python -m tacotron_multispeaker_b200.build` "
            "or __graft_entry__.build(); there is no CPU fallback for this path." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, ip, fp = C.c_void_p, C.c_void_p, C.c_void_p  # device pointers travel as integers
    i, i64 = C.c_int, C.c_int64
    H = C.c_void_p
    lib.taco_create.argtypes = [C.POINTER(TacoHParams), i, C.POINTER(H)]
    lib.taco_destroy.argtypes = [H]
    lib.taco_last_error.argtypes = [H]
    lib.taco_last_error.restype = C.c_char_p
    lib.taco_version.restype = C.c_char_p
    lib.taco_set_weight.argtypes = [H, C.c_char_p, C.c_void_p, C.POINTER(i64), i]
    lib.taco_finalize_weights.argtypes = [H]
    lib.taco_num_weights.argtypes = [H]
    lib.taco_weight_name.argtypes = [H, i]
    lib.taco_weight_name.restype = C.c_char_p
    lib.taco_max_steps.argtypes = [H, i, i]
    lib.taco_forward.argtypes = [H, ip, ip, ip, fp, i, i, i, i, i, fp, fp, fp, C.POINTER(C.c_int32), vp]
    lib.taco_forward_host.argtypes = [H, ip, ip, ip, fp, i, i, i, i, i, fp, fp, fp, C.POINTER(C.c_int32), vp]
    lib.taco_forward_host_begin.argtypes = [H, ip, ip, ip, fp, i, i, i, i, i, fp, fp, fp, vp]
    lib.taco_forward_host_wait.argtypes = [H, i]
    lib.taco_forward_host_end.argtypes = [H, C.POINTER(C.c_int32), vp]
    lib.taco_set_decoder_clusters.argtypes = [H, i]
    lib.taco_embed.argtypes = [H, ip, ip, i, i, fp, vp]
    lib.taco_check_ids.argtypes = [H, vp]
    lib.taco_encoder.argtypes = [H, ip, ip, ip, i, i, i, fp, vp]
    lib.taco_decode.argtypes = [H, fp, i, i, fp, i, i, fp, fp, C.POINTER(C.c_int32), vp]
    lib.taco_cbhg.argtypes = [H, i, fp, ip, i, i, i, i64, fp, vp]
    lib.taco_postnet.argtypes = [H, fp, i, i, i, i64, fp, i64, vp]
    lib.taco_bigru.argtypes = [H, i, fp, ip, i, i, fp, vp]
    lib.taco_conv1d.argtypes = [H, fp, i, i, i, fp, fp, i, i, i, fp, vp]
    lib.taco_maxpool_affine.argtypes = [H, fp, i, i, i, fp, fp, fp, vp]
    lib.taco_bn_batch_stats.argtypes = [H, fp, i, i, i, fp, fp, fp, fp, vp]
    lib.taco_set_gemm_mode.argtypes = [H, i]
    lib.taco_launch_count.argtypes = [H]
    lib.taco_launch_count.restype = i64
    lib.taco_decoder_geometry.argtypes = [H, i, C.POINTER(i), C.POINTER(i), C.POINTER(i)]
    lib.taco_set_profiling.argtypes = [H, i]
    lib.taco_set_cuda_graphs.argtypes = [H, i]
    lib.taco_last_stage_ms.argtypes = [H, C.POINTER(C.c_float)]
    lib.taco_wav_length.argtypes = [C.POINTER(TacoAudioParams), i]
    lib.taco_wav_length.restype = i64
    lib.taco_griffin_lim.argtypes = [H, C.POINTER(TacoAudioParams), fp, i, i, i64, fp, vp]
    lib.taco_spectrogram_frames.argtypes = [C.POINTER(TacoAudioParams), i64]
    lib.taco_spectrogram_frames.restype = i64
    lib.taco_spectrogram.argtypes = [H, C.POINTER(TacoAudioParams), fp, C.c_void_p, i, i64, i, fp, fp, vp]
    lib.taco_resample_length.argtypes = [i64, C.c_int32, C.c_int32]
    lib.taco_resample_length.restype = i64
    lib.taco_resample_positions.argtypes = [C.c_int32, C.c_int32, i64, i64, vp, vp, vp, vp, vp]
    lib.taco_resample.argtypes = [H, C.c_int32, C.c_int32, fp, C.c_void_p, i, i64, fp, i64, vp]
    lib.taco_durations.argtypes = [H, fp, i, i, i, C.c_void_p, C.c_void_p, ip, vp]
    lib.taco_umma_plan.argtypes = [C.POINTER(TacoGemmDesc), i, C.POINTER(TacoGemmPlan)]
    lib.taco_gemm_unit.argtypes = [H, C.POINTER(TacoGemmDesc), C.POINTER(TacoGemmPlan), vp]
    lib.taco_highway4_unit.argtypes = [H, fp, i64, i, vp, vp, vp, vp, fp, vp, vp, vp]
    lib.taco_bigru_unit.argtypes = [H, i, fp, ip, i, i, vp, vp, fp, vp]
    lib.taco_decoder_plan.argtypes = [i, i, i, C.POINTER(TacoDecoderPlan)]
    for name in SYMBOLS:
        getattr(lib, name)  # AttributeError here = header and library out of sync
    _lib = lib
    return lib


def umma_plan(desc: TacoGemmDesc, sms: int = 148) -> dict:
    """``taco_umma_plan``: how the tensor-core kernel would run ``desc`` on ``sms`` SMs (host only, no device)."""
    plan = TacoGemmPlan()
    load().taco_umma_plan(C.byref(desc), int(sms), C.byref(plan))
    return plan.as_dict()


def decoder_plan(N: int, T_in: int, max_clusters: int = 7) -> dict:
    """``taco_decoder_plan``: clusters, utterances per cluster and attention residency of the default decoder for a batch of
    ``N`` utterances of ``T_in`` positions, ``max_clusters`` co-resident (7 on a B200).  Host only, no device."""
    plan = TacoDecoderPlan()
    load().taco_decoder_plan(int(N), int(T_in), int(max_clusters), C.byref(plan))
    return plan.as_dict()


def check(lib, handle, rc: int) -> None:
    if rc != TACO_OK:
        msg = lib.taco_last_error(handle)
        raise TacoError(rc, msg.decode() if msg else "")
