"""ctypes binding of ``libseqpan_b200.so`` (include/seqpan_b200.h).

There is deliberately no fallback: if the library is missing or no sm_100 device is present, the
product path raises.  (The CPU oracle under ``oracle/`` is test infrastructure and is never imported here.)
"""
from __future__ import annotations

import ctypes as C
import os

# More hardware work queues than the default 8: the eval sweep uses compute lanes + a copy stream (+ the handles' side / capture
# streams); when two of them alias to one queue, kernels queue up behind a 1.5 ms host->device copy kernel.  Measured on B200:
# the same e2e sweep gives 93-158 k queries/s from run to run with 8 connections and a stable 157 k with 32.  Read by the driver
# when the CUDA context is created, so it has to be in the environment before the first CUDA call of the process.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SEQPAN_LIB") or os.path.join(PKG, "libseqpan_b200.so")   # SEQPAN_LIB: instrumented builds

ABI_VERSION = 2
VARIANT_SEQPAN, VARIANT_BASEFAST, VARIANT_MULTITEACHER, VARIANT_BACKBONE, VARIANT_STUDENT4 = 0, 1, 2, 3, 4
PREC_FP32, PREC_BF16, PREC_TF32 = 0, 1, 2
SAMPLE_ORIGINAL, SAMPLE_TRUNCATION, SAMPLE_SAMELEN = 0, 1, 2


class SeqpanShapes(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("abi_version", "max_batch", "vlen", "max_tlen", "max_clen", "vdim",
                                         "num_words", "num_chars", "precision", "pretrained_words", "variant")]


class SeqpanGemm(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("M", "N", "K", "a_rs", "a_cs", "b_rs", "b_cs", "c_rs", "c_cs",
                                         "a_b0", "a_b1", "b_b0", "b_b1", "c_b0", "c_b1")] + \
               [("batch0", C.c_int32), ("batch1", C.c_int32), ("alpha", C.c_float), ("beta", C.c_float), ("splitk", C.c_int32)]


class SeqpanEwise(C.Structure):
    _fields_ = [("op", C.c_int32), ("accumulate", C.c_int32), ("shape", C.c_int64 * 4), ("so", C.c_int64 * 4),
                ("sa", C.c_int64 * 4), ("sb", C.c_int64 * 4), ("sc", C.c_int64 * 4), ("alpha", C.c_float), ("beta", C.c_float)]


class SeqpanSoftmax(C.Structure):
    _fields_ = [("rows0", C.c_int64), ("rows1", C.c_int64), ("r0_stride", C.c_int64), ("r1_stride", C.c_int64),
                ("cols", C.c_int32), ("c_stride", C.c_int64)]


class SeqpanAdamW(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("lr", "beta1", "beta2", "eps", "weight_decay", "bias1", "bias2_sqrt", "max_grad_norm")]


EW = dict(COPY=0, AXPBY=1, MUL=2, RELU=3, RELU_BWD=4, SIGMOID=5, SIGMOID_BWD=6, MASK_LOGITS=7, FMA=8, LOG=9, EXP=10, DIV=11,
          SQRT=12, AFFINE=13, EQ=14, DIV_SAFE=15, DROPOUT=16)


class SeqpanError(RuntimeError):
    pass


_lib = None

# every symbol include/seqpan_b200.h declares: (restype, argtypes)
_vp, _i, _i64, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_size_t
SIGNATURES = {
    "seqpan_num_weights": (_i, []),
    "seqpan_weight_name": (C.c_char_p, [_i]),
    "seqpan_weight_numel": (_i64, [C.POINTER(SeqpanShapes), _i]),
    "seqpan_arena_bytes": (_sz, [C.POINTER(SeqpanShapes)]),
    "seqpan_workspace_bytes": (_sz, [C.POINTER(SeqpanShapes)]),
    "seqpan_create": (_i, [C.POINTER(SeqpanShapes), C.POINTER(_vp), _vp, _sz, _vp, C.POINTER(_vp)]),
    "seqpan_repack": (_i, [_vp, C.POINTER(_vp), _vp]),
    "seqpan_destroy": (None, [_vp]),
    "seqpan_forward": (_i, [_vp] + [_vp] * 6 + [_i, _i, _i] + [_vp] * 3 + [_vp, _sz, _vp]),
    "seqpan_forward_shared_video": (_i, [_vp] + [_vp] * 4 + [_i] + [_vp] * 3 + [_i, _i, _i] + [_vp] * 3 + [_vp, _sz, _vp]),
    "seqpan_encode_videos": (_i, [_vp, _vp, _i, _vp, _vp, _sz, _vp]),
    "seqpan_forward_encoded": (_i, [_vp] + [_vp] * 4 + [_i] + [_vp] * 3 + [_i, _i, _i] + [_vp] * 3 + [_vp, _sz, _vp]),
    "seqpan_span_decode": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "seqpan_iou_counters": (_i, [_vp, _vp, _i, _vp, _vp]),
    "seqpan_iou_counters_exact": (_i, [_vp, _vp, _i, _vp, _vp]),
    "seqpan_gumbel_noise": (_i, [C.c_uint64, C.c_uint32, _i, _i, _vp, _vp]),
    "seqpan_span_topk": (_i, [_vp, _vp, _vp, _i, _i, _i, C.c_float, _vp, _vp, _vp, _vp, _vp]),
    "seqpan_topk_counters": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "seqpan_h2d_ragged": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "seqpan_collate_clips": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "seqpan_collate_text": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "seqpan_debug_tap": (_i64, [_vp, C.c_char_p, _vp, _vp, _i64, _vp]),
    "seqpan_last_launch_count": (_i, [_vp]),
    "seqpan_op_linear_scratch_bytes": (_sz, [_i64, _i, _i]),
    "seqpan_op_linear": (_i, [_vp] * 5 + [_i64, _i, _i, _i, _i, _vp, _sz, _vp]),
    "seqpan_op_layernorm": (_i, [_vp, _vp, _vp, C.c_float, _vp, _i64, _vp]),
    "seqpan_t_gemm": (_i, [_vp, _vp, _vp, _vp, C.POINTER(SeqpanGemm), _vp]),
    "seqpan_t_gemm_bf16": (_i, [_vp, _vp, _vp, _vp, C.POINTER(SeqpanGemm), _vp]),
    "seqpan_t_ewise": (_i, [_vp, _vp, _vp, _vp, C.POINTER(SeqpanEwise), _vp]),
    "seqpan_t_softmax": (_i, [_vp, _vp, C.POINTER(SeqpanSoftmax), _vp]),
    "seqpan_t_softmax_bwd": (_i, [_vp, _vp, _vp, C.POINTER(SeqpanSoftmax), _vp]),
    "seqpan_t_layernorm_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_float, _i64, _vp]),
    "seqpan_t_dwconv": (_i, [_vp, _vp, _vp, _i64, _i, _i, _vp]),
    "seqpan_t_dwconv_bwd_w": (_i, [_vp, _vp, _vp, _i64, _i, _vp]),
    "seqpan_t_gather_rows": (_i, [_vp, _vp, _vp, _i64, _i, _i64, _vp]),
    "seqpan_t_scatter_add_rows": (_i, [_vp, _vp, _vp, _i64, _i, _i64, _vp]),
    "seqpan_t_maxpool": (_i, [_vp, _vp, _vp, _i64, _i, _i, _vp]),
    "seqpan_t_maxpool_bwd": (_i, [_vp, _vp, _vp, _i64, _i, _i, _vp]),
    "seqpan_t_sumsq": (_i, [_vp, _i64, _vp, _vp]),
    "seqpan_t_adamw": (_i, [_vp, _vp, _vp, _vp, _i64, C.POINTER(SeqpanAdamW), _vp, _vp, _vp]),
    "seqpan_t_gemm_det_scratch_bytes": (_sz, [C.POINTER(SeqpanGemm)]),
    "seqpan_t_gemm_det": (_i, [_vp, _vp, _vp, _vp, C.POINTER(SeqpanGemm), _vp, _sz, _vp]),
    "seqpan_t_gemm_bf16_det": (_i, [_vp, _vp, _vp, _vp, C.POINTER(SeqpanGemm), _vp, _sz, _vp]),
    "seqpan_t_layernorm_bwd_det_scratch_bytes": (_sz, [_i64]),
    "seqpan_t_layernorm_bwd_det": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_float, _i64, _vp, _sz, _vp]),
    "seqpan_t_dwconv_bwd_w_det_scratch_bytes": (_sz, [_i64]),
    "seqpan_t_dwconv_bwd_w_det": (_i, [_vp, _vp, _vp, _i64, _i, _vp, _sz, _vp]),
    "seqpan_t_scatter_add_rows_det": (_i, [_vp, _vp, _vp, _i64, _i, _i64, _vp]),
    "seqpan_t_sumsq_det_scratch_bytes": (_sz, [_i64]),
    "seqpan_t_sumsq_det": (_i, [_vp, _i64, _vp, _vp, _sz, _vp]),
    "seqpan_t_last_error": (C.c_char_p, []),
    "seqpan_last_error": (C.c_char_p, []),
    "seqpan_device_ok": (_i, []),
    "seqpan_set_debug": (_i, [_vp, _i]),
    "seqpan_set_profile": (_i, [_vp, _i]),
    "seqpan_set_side_stream": (_i, [_vp, _i]),
    "seqpan_profile_summary": (_i, [_vp, C.c_char_p, _sz]),
}


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SeqpanError(f"{LIB_PATH} is missing: build it with `python -m vmrframe_b200.build` "
                              "(there is no CPU or PyTorch fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


DIAG_LIB_PATH = os.path.join(PKG, "libseqpan_diag.so")
DIAG_SIGNATURES = {"seqpan_test_umma": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp])}   # include/seqpan_b200_diag.h
_diag = None


def diag_lib() -> C.CDLL:
    """The diagnostics library (tcgen05 descriptor probe): tests and profiles/ only, never the product path."""
    global _diag
    if _diag is None:
        if not os.path.exists(DIAG_LIB_PATH):
            raise SeqpanError(f"{DIAG_LIB_PATH} is missing: build it with `python -m vmrframe_b200.build`")
        L = C.CDLL(DIAG_LIB_PATH)
        for name, (res, args) in DIAG_SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _diag = L
    return _diag


def check(rc: int) -> int:
    if rc < 0:
        raise SeqpanError(f"seqpan_b200 error {rc}: {lib().seqpan_last_error().decode()}")
    return rc


def weight_names() -> list[str]:
    L = lib()
    return [L.seqpan_weight_name(i).decode() for i in range(L.seqpan_num_weights())]


def require_device() -> None:
    if not lib().seqpan_device_ok():
        raise SeqpanError("no sm_100 (B200) CUDA device visible: the SeqPAN hot path has no CPU fallback")
