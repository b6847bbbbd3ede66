"""vmrframe_b200: B200-native SeqPAN inference hot path behind the interface of VMRFrame's ``models/SeqPAN.py``.

The five names the reference's registry exports per model (``models/__init__.py:2,19``) are available here, so
``eval(configs.model.name)`` style dispatch (``main.py:21,87,99``) resolves against this package unchanged.
"""
from .seqpan import (BackBone, BaseFast, MultiTeacher, OneTeacher, infer_OneTeacher, SeqPAN, extract_index, extract_topk, infer_basic, infer_basic_device, infer_BaseFast,  # noqa: F401
                     infer_BackBone, infer_MultiTeacher, infer_SeqPAN, train_engine_BackBone, train_engine_BaseFast, train_engine_MultiTeacher,
                     infer_topk, train_engine_SeqPAN, VideoEncodings)
from .engine import (IouCounters, TopkCounters, append_ious, append_ious_topk, calculate_iou, calculate_iou_accuracy,  # noqa: F401
                     evaluate, draw_chunks, get_i345_mi, gumbel_noise, metrics_from_counters, metrics_topk_from_counters,
                     recall_at_k, shard_batches)

from . import data_utils  # noqa: F401  (device versions of utils/data_utils.py's clip resampling / padding, SURVEY.md section 8 f2)

__all__ = ["data_utils", "SeqPAN", "infer_SeqPAN", "train_engine_SeqPAN", "BaseFast", "infer_BaseFast", "train_engine_BaseFast", "MultiTeacher", "infer_MultiTeacher", "train_engine_MultiTeacher", "BackBone", "infer_BackBone", "train_engine_BackBone", "OneTeacher", "infer_OneTeacher", "extract_index", "infer_basic", "extract_topk", "infer_topk", "VideoEncodings", "evaluate",
           "append_ious", "get_i345_mi", "IouCounters", "TopkCounters", "append_ious_topk", "recall_at_k", "metrics_topk_from_counters", "shard_batches", "draw_chunks",
           "gumbel_noise"]
