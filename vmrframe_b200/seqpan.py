"""Drop-in ``SeqPAN`` module: the interface of the reference's ``models/SeqPAN.py`` over the B200 C-ABI library.

Mirrors (reference file:line):
  * ``SeqPAN(configs, word_vectors)``                       models/SeqPAN.py:11-47
  * ``forward(word_ids, char_ids, vfeat_in, vmask, tmask)``  models/SeqPAN.py:50-95 (positional, same order)
    returning the same 6-key dict (``slogits, elogits, vmask, match_score, label_embs, consume_time``)
  * ``state_dict()`` keys/shapes, including the reference's 20 dead tensors (SURVEY.md §0 #13), so a
    reference checkpoint loads with ``strict=True`` (``module.`` prefixes from DataParallel are stripped)
  * ``infer_SeqPAN(output, configs)``                        models/SeqPAN.py:185-192
  * ``extract_index(start_logits, end_logits)``              models/layers.py:549-557
  * ``train_engine_SeqPAN``                                  models/SeqPAN.py:171-182 (forward + the reference's losses)

PyTorch is plumbing here: ``nn.Conv1d`` / ``nn.LayerNorm`` / ``nn.Embedding`` / ``nn.MultiheadAttention`` objects are
used only as parameter containers (same names, shapes and default initialisation as the reference; their
``forward`` is never called), tensors provide device memory and the CUDA stream.  All arithmetic of the forward
and of the span decode runs in ``libseqpan_b200.so``; there is no CPU or eager fallback.
"""
from __future__ import annotations

import ctypes as C
import os
import time

import numpy as np
import torch
import torch.nn as nn

from . import _cabi

_PRECISIONS = {"fp32": _cabi.PREC_FP32, "bf16": _cabi.PREC_BF16, "tf32": _cabi.PREC_TF32}


class _Holder(nn.Module):
    """Parameter container; arithmetic lives in the CUDA library."""

    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError("container module: call SeqPAN.forward")


class _Conv1D(_Holder):  # models/layers.py:15-26
    def __init__(self, in_dim, out_dim):
        super().__init__()
        self.conv1d = nn.Conv1d(in_dim, out_dim, kernel_size=1, padding=0, stride=1, bias=True)


class _WordEmbedding(_Holder):  # models/layers.py:28-48
    def __init__(self, num_words, word_dim, word_vectors):
        super().__init__()
        self.is_pretrained = word_vectors is not None
        if self.is_pretrained:
            self.pad_vec = nn.Parameter(torch.zeros(1, word_dim), requires_grad=False)
            unk = torch.empty(1, word_dim)
            nn.init.xavier_uniform_(unk)
            self.unk_vec = nn.Parameter(unk, requires_grad=True)
            self.glove_vec = nn.Parameter(torch.tensor(np.asarray(word_vectors), dtype=torch.float32), requires_grad=False)
        else:
            self.word_emb = nn.Embedding(num_words, word_dim, padding_idx=0)


class _CharacterEmbedding(_Holder):  # models/layers.py:51-75
    def __init__(self, num_chars, char_dim):
        super().__init__()
        self.char_emb = nn.Embedding(num_chars, char_dim, padding_idx=0)
        self.char_convs = nn.ModuleList([
            nn.Sequential(nn.Conv2d(char_dim, ch, kernel_size=(1, k), stride=(1, 1), padding=0, bias=True), nn.ReLU())
            for k, ch in zip([1, 2, 3, 4], [10, 20, 30, 40])])


class _Embedding(_Holder):  # models/layers.py:78-93
    def __init__(self, num_words, num_chars, word_dim, char_dim, out_dim, word_vectors):
        super().__init__()
        self.word_emb = _WordEmbedding(num_words, word_dim, word_vectors)
        self.char_emb = _CharacterEmbedding(num_chars, char_dim)
        self.query_conv1d = _Conv1D(word_dim + char_dim, out_dim)
        self.q_layer_norm = nn.LayerNorm(out_dim, eps=1e-6)


class _VisualProjection(_Holder):  # models/layers.py:110-123
    def __init__(self, visual_dim, dim):
        super().__init__()
        self.video_conv1d = _Conv1D(visual_dim, dim)
        self.v_layer_norm = nn.LayerNorm(dim, eps=1e-6)


class _PositionalEmbedding(_Holder):  # models/layers.py:96-107
    def __init__(self, n, dim):
        super().__init__()
        self.position_embeddings = nn.Embedding(n, dim)


class _ConvBlock(_Holder):  # models/layers.py:126-148
    def __init__(self, dim, kernel_size=7, num_layers=4):
        super().__init__()
        self.depthwise_separable_conv = nn.ModuleList([
            nn.Sequential(nn.Conv1d(dim, dim, kernel_size, groups=dim, padding=kernel_size // 2, bias=False),
                          nn.Conv1d(dim, dim, 1, padding=0, bias=True), nn.ReLU()) for _ in range(num_layers)])
        self.layer_norms = nn.ModuleList([nn.LayerNorm(dim, eps=1e-6) for _ in range(num_layers)])


class _FeatureEncoder(_Holder):  # models/layers.py:388-399
    def __init__(self, dim, max_pos_len, num_layers=4):
        super().__init__()
        self.pos_embedding = _PositionalEmbedding(max_pos_len, dim)
        self.conv_block = _ConvBlock(dim, num_layers=num_layers)


class _BiLinear(_Holder):  # models/layers.py:246-263 (dense_2 is dead in the reference but is a state_dict key)
    def __init__(self, dim):
        super().__init__()
        self.dense_1 = _Conv1D(dim, dim)
        self.dense_2 = _Conv1D(dim, dim)
        self.bias_value = nn.Parameter(torch.zeros(dim))


class _DualMultiAttention(_Holder):  # models/layers.py:300-327
    def __init__(self, dim):
        super().__init__()
        for name in ("query", "f_key", "f_value", "t_key", "t_value", "s_dense", "x_dense", "s_gate", "x_gate",
                     "guided_dense"):
            setattr(self, name, _Conv1D(dim, dim))
        self.bilinear_1 = _BiLinear(dim)
        self.bilinear_2 = _BiLinear(dim)
        self.layer_norm1 = nn.LayerNorm(dim, eps=1e-6)   # dead in the reference forward
        self.layer_norm2 = nn.LayerNorm(dim, eps=1e-6)   # dead
        self.out_layer = _Conv1D(dim, dim)               # dead


class _DualAttentionBlock(_Holder):  # models/layers.py:266-279
    def __init__(self, dim):
        super().__init__()
        self.layer_norm_1 = nn.LayerNorm(dim, eps=1e-6)
        self.layer_norm_2 = nn.LayerNorm(dim, eps=1e-6)
        self.layer_norm_t = nn.LayerNorm(dim, eps=1e-6)
        self.dense_1 = _Conv1D(dim, dim)
        self.dense_2 = _Conv1D(dim, dim)
        self.dual_multihead_attention = _DualMultiAttention(dim)


class _CQAttention(_Holder):  # models/layers.py:402-415
    def __init__(self, dim):
        super().__init__()
        w4C, w4Q, w4mlu = torch.empty(dim, 1), torch.empty(dim, 1), torch.empty(1, 1, dim)
        nn.init.xavier_uniform_(w4C)
        nn.init.xavier_uniform_(w4Q)
        nn.init.xavier_uniform_(w4mlu)
        self.w4C, self.w4Q, self.w4mlu = nn.Parameter(w4C), nn.Parameter(w4Q), nn.Parameter(w4mlu)
        self.cqa_linear = _Conv1D(4 * dim, dim)


class _WeightedPool(_Holder):  # models/layers.py:440-445
    def __init__(self, dim):
        super().__init__()
        w = torch.empty(dim, 1)
        nn.init.xavier_uniform_(w)
        self.weight = nn.Parameter(w)


class _CQConcatenate(_Holder):  # models/layers.py:456-460
    def __init__(self, dim):
        super().__init__()
        self.weighted_pool = _WeightedPool(dim)
        self.conv1d = _Conv1D(2 * dim, dim)


class _TopSelfAttention2(_Holder):  # models/layers.py:567-570
    def __init__(self, dim, num_heads, droprate):
        super().__init__()
        self.selfattn = nn.MultiheadAttention(dim, num_heads, dropout=droprate)


class _FeatureEncoderPredict(_Holder):  # models/layers.py:613-624
    def __init__(self, dim, num_heads, max_pos_len, droprate):
        super().__init__()
        self.pos_embedding = _PositionalEmbedding(max_pos_len, dim)
        self.conv_block = _ConvBlock(dim)
        self.layer_norm_1 = nn.LayerNorm(dim)   # default eps 1e-5 (SURVEY.md §0 #15)
        self.layer_norm_2 = nn.LayerNorm(dim)
        self.top_self_attention = _TopSelfAttention2(dim, num_heads, droprate)
        self.dense = _Conv1D(dim, dim)


class _SeqPANPredictor(_Holder):  # models/layers.py:642-657
    def __init__(self, dim, vlen, droprate):
        super().__init__()
        self.feature_encoder = _FeatureEncoderPredict(dim, 4, vlen, droprate)
        self.start_layer_norm = nn.LayerNorm(dim, eps=1e-6)
        self.end_layer_norm = nn.LayerNorm(dim, eps=1e-6)
        self.start_hidden = _Conv1D(2 * dim, dim)
        self.end_hidden = _Conv1D(2 * dim, dim)
        self.start_dense = _Conv1D(dim, 1)
        self.end_dense = _Conv1D(dim, 1)


class VideoEncodings:
    """Encoded clips of :meth:`SeqPAN.encode_videos`: ``rows`` is the ``[U,vlen,128]`` fp32 CUDA tensor of VisualProjection +
    the video half of the shared FeatureEncoder (DESIGN.md section 12), owned by the caller.  ``precision``, ``variant`` and
    ``signature`` (the weights' ``(data_ptr, _version)`` signature when they were packed, with the count of explicit
    ``repack()`` calls) record what made them: a forward refuses encodings of another precision, another model variant or
    weights that changed since."""

    __slots__ = ("rows", "precision", "variant", "signature")

    def __init__(self, rows: torch.Tensor, precision: str, variant: int, signature):
        self.rows, self.precision, self.variant, self.signature = rows, precision, variant, signature

    def __len__(self):
        return self.rows.shape[0]

    @property
    def device(self):
        return self.rows.device


class SeqPAN(nn.Module):
    """B200-native SeqPAN.  Extra, optional knobs beyond the reference constructor:

    ``precision``   "bf16" (tcgen05 tensor cores, default), "tf32" (every projection on tcgen05 kind::tf32 from fp32 rows: the
                    arithmetic the reference itself gets on a GPU, where nn.Conv1d runs under cudnn.allow_tf32 = True) or
                    "fp32" (CUDA-core parity mode); may also come from
                    ``configs.model.precision`` or the ``SEQPAN_PRECISION`` environment variable.
    ``sync_timing`` True (default) keeps the reference's two ``torch.cuda.synchronize()`` calls around the forward so
                    ``consume_time`` means what ``main.py:102,127`` expects; False makes the call asynchronous
                    (``consume_time`` = 0.0), which pipelined evaluation uses.
    """

    _VARIANT = _cabi.VARIANT_SEQPAN   # which sibling model of the reference the library handle computes
    _ENC_LAYERS = 4                   # conv layers of the shared FeatureEncoder (models/SeqPAN.py:28)
    _OWN_TEXT_ENCODER = False         # BackBone: the text has its own FeatureEncoder (models/BackBone.py:24)
    _MATCH_HEAD = True                # BackBone: no match_conv1d / label_embs / Gumbel softmax (models/BackBone.py:59-63)

    def __init__(self, configs, word_vectors, precision: str | None = None, sync_timing: bool = True):
        super().__init__()
        self.configs = configs
        m = configs.model
        dim = m.dim
        if dim != 128 or m.num_heads != 4 or m.word_dim != 300 or m.char_dim != 100:
            raise ValueError("the B200 kernels are specialised for dim=128, num_heads=4, word_dim=300, char_dim=100 "
                             "(every SeqPAN config of the reference)")
        droprate = m.droprate
        # construction order == reference order, so torch.manual_seed(s) yields the reference's initial weights
        self.text_encoder = _Embedding(configs.num_words, configs.num_chars, m.word_dim, m.char_dim, dim, word_vectors)
        if self._OWN_TEXT_ENCODER:      # models/BackBone.py:24 (constructed before video_affine)
            self.tfeat_encoder = _FeatureEncoder(dim, m.vlen, 4)
        self.video_affine = _VisualProjection(m.vdim, dim)
        self.vfeat_encoder = _FeatureEncoder(dim, m.vlen, self._ENC_LAYERS)
        self.dual_attention_block_1 = _DualAttentionBlock(dim)
        self.dual_attention_block_2 = _DualAttentionBlock(dim)
        self.q2v_attn = _CQAttention(dim)
        self.v2q_attn = _CQAttention(dim)
        self.cq_cat = _CQConcatenate(dim)
        if self._MATCH_HEAD:
            self.match_conv1d = _Conv1D(dim, 4)
            self.label_embs = nn.Parameter(torch.nn.init.orthogonal_(torch.empty(dim, 4, dtype=torch.float32)))
        self.predictor = _SeqPANPredictor(dim, m.vlen, droprate)

        prec = precision or getattr(m, "precision", None) or os.environ.get("SEQPAN_PRECISION", "bf16")
        if prec not in _PRECISIONS:
            raise ValueError(f"precision must be one of {list(_PRECISIONS)}")
        self.precision = prec
        self.sync_timing = sync_timing
        self._handle = None
        self._limits = None          # (max_batch, max_tlen, max_clen) the handle was created for
        self._arena = self._workspace = None
        self._wsig = None
        self._wptrs = None
        self._ctxs = {}              # parked kernel contexts (see use_context)
        self._ctx_key = 0
        self._frozen = False
        self._debug = False
        self._repacks = 0            # explicit repack() calls: part of what VideoEncodings are checked against
        self._register_load_state_dict_pre_hook(self._strip_module_prefix)

    # ---- checkpoint compatibility ----------------------------------------------------------------------
    @staticmethod
    def _strip_module_prefix(state_dict, prefix, *args):
        # checkpoints saved from nn.DataParallel carry a "module." prefix (main.py:22-28)
        for k in list(state_dict.keys()):
            if k.startswith(prefix + "module."):
                state_dict[prefix + k[len(prefix) + 7:]] = state_dict.pop(k)

    # ---- handle management -----------------------------------------------------------------------------
    def freeze(self, frozen: bool = True):
        """Skip the per-call "did a parameter change?" check (weights are packed once)."""
        self._frozen = frozen
        return self

    def set_debug_taps(self, on: bool = True):
        self._debug = on
        if self._handle is not None:
            _cabi.check(_cabi.lib().seqpan_set_debug(self._handle, int(on)))

    def set_side_stream(self, on: bool = True):
        """Text branch of the forward on a side stream, concurrent with the video affine (default on).  Applies to every kernel
        context of the module; :func:`vmrframe_b200.evaluate` turns it off while it runs (its copy kernel owns the PCIe bus)."""
        self._side_stream = bool(on)
        handles = [self._handle] + [st[0] for st in self._ctxs.values()]
        for h in handles:
            if h is not None:
                _cabi.check(_cabi.lib().seqpan_set_side_stream(h, int(on)))
        return self

    def use_context(self, key=0):
        """Selects an independent kernel context (library handle + workspace).  One context per CUDA stream lets
        forwards of different batches overlap on the GPU (the engine's multi-stream sweep); the default context 0 is
        all a drop-in user ever sees."""
        if key == self._ctx_key:
            return self
        self._ctxs[self._ctx_key] = (self._handle, self._limits, self._arena, self._workspace, self._wsig, self._wptrs)
        (self._handle, self._limits, self._arena, self._workspace, self._wsig,
         self._wptrs) = self._ctxs.pop(key, (None, None, None, None, None, None))
        self._ctx_key = key
        return self

    def _weight_tensors(self):
        # resolved by walking attributes (not named_parameters()): nn.DataParallel replicas keep their broadcast copies as
        # plain tensor attributes with empty _parameters dicts (torch/nn/parallel/replicate.py)
        out = []
        for name in _cabi.weight_names():
            obj = self
            for part in name.split("."):
                if part.isdigit() and isinstance(obj, (nn.ModuleList, nn.Sequential)):
                    obj = obj[int(part)] if int(part) < len(obj) else None   # e.g. layers 2, 3 of BaseFast's 2-layer encoder
                else:
                    obj = getattr(obj, part, None)
                if obj is None:
                    break
            out.append(obj if isinstance(obj, torch.Tensor) else None)
        return out

    def _replicate_for_data_parallel(self):
        # main.py:22-24 wraps the model in nn.DataParallel when several GPUs are visible.  A replica must not share the
        # original's library handle / arena / workspace (its __del__ would destroy a handle the original still uses, and
        # the packed weights live on another device): it starts without kernel state and builds its own on first use.
        replica = super()._replicate_for_data_parallel()
        replica._handle = replica._limits = replica._arena = replica._workspace = None
        replica._wsig = replica._wptrs = None
        replica._ctxs = {}
        replica._ctx_key = 0
        replica._frozen = False
        return replica

    def repack(self):
        """Re-derives the packed weights (bf16 copies, folded products, host mirrors of the small vectors) from the current
        parameter values.  Needed only after edits the version counters cannot see -- ``p.data.copy_(...)`` /
        ``p.data.mul_(...)`` (EMA swaps) do not bump ``Tensor._version`` -- or while :meth:`freeze` is on; ordinary optimizer
        steps, ``load_state_dict`` and ``.to()`` are detected automatically.  Encodings of :meth:`encode_videos` made before
        the call are stale afterwards: the edits it exists for leave the weights' signature unchanged."""
        self._repacks += 1
        for key in [self._ctx_key] + list(self._ctxs):
            self.use_context(key)
            if self._handle is not None:
                self._wsig = None
                frozen, self._frozen = self._frozen, False
                try:
                    self._ensure_handle(self._arena.device, 1, 1, 4)
                finally:
                    self._frozen = frozen
        return self

    def _signature(self, tensors):
        return tuple((t.data_ptr(), t._version) if t is not None else None for t in tensors)

    def _release(self, all_contexts: bool = False):
        if self._handle is not None:
            _cabi.lib().seqpan_destroy(self._handle)
            self._handle = None
        if all_contexts:
            for st in self._ctxs.values():
                if st[0] is not None:
                    _cabi.lib().seqpan_destroy(st[0])
            self._ctxs = {}

    def __del__(self):
        try:
            self._release(all_contexts=True)
        except Exception:
            pass

    def _ensure_handle(self, device, B, T, Cc):
        L = _cabi.lib()
        m = self.configs.model
        lim = self._limits
        need_new = self._handle is None or B > lim[0] or T > lim[1] or Cc > lim[2] or self._arena.device != device
        tensors = None
        if need_new or not self._frozen:
            tensors = self._weight_tensors()
            for name, t in zip(_cabi.weight_names(), tensors):
                if t is not None and (t.device != device or t.dtype != torch.float32 or not t.is_contiguous()):
                    raise _cabi.SeqpanError(f"parameter {name} must be a contiguous float32 tensor on {device} "
                                            f"(call model.to(device))")
        if need_new:
            self._release()
            old = lim or (0, 0, 0)
            lim = (max(B, old[0]), min(m.vlen, _cabi_max_tlen(), max(T, old[1], 16)), min(64, max(Cc, old[2], 8)))
            if T > lim[1]:
                raise _cabi.SeqpanError(f"T={T} exceeds the supported text length {lim[1]} (<= vlen: the text shares "
                                        f"the video position table, models/SeqPAN.py:59-60)")
            pretrained = int(self.text_encoder.word_emb.is_pretrained)
            shp = _cabi.SeqpanShapes(_cabi.ABI_VERSION, lim[0], m.vlen, lim[1], lim[2], m.vdim, self.configs.num_words,
                                     self.configs.num_chars, _PRECISIONS[self.precision], pretrained, self._VARIANT)
            ab, wb = L.seqpan_arena_bytes(C.byref(shp)), L.seqpan_workspace_bytes(C.byref(shp))
            if ab == 0 or wb == 0:
                raise _cabi.SeqpanError(f"unsupported shapes: {L.seqpan_last_error().decode()}")
            self._check_numel(shp, tensors)
            self._arena = torch.empty(ab, dtype=torch.uint8, device=device)
            self._workspace = torch.empty(wb, dtype=torch.uint8, device=device)
            self._shapes = shp
            ptrs = (C.c_void_p * len(tensors))(*[t.data_ptr() if t is not None else None for t in tensors])
            h = C.c_void_p()
            stream = torch.cuda.current_stream(device).cuda_stream
            _cabi.check(L.seqpan_create(C.byref(shp), ptrs, self._arena.data_ptr(), ab, stream, C.byref(h)))
            self._handle, self._limits, self._wptrs = h, lim, tensors
            self._wsig = self._signature(tensors)
            if self._debug:
                _cabi.check(L.seqpan_set_debug(h, 1))
            if not getattr(self, "_side_stream", True):
                _cabi.check(L.seqpan_set_side_stream(h, 0))
        elif not self._frozen:
            sig = self._signature(tensors)
            if sig != self._wsig:  # parameters were updated in place or re-assigned: re-pack derived weights
                self._check_numel(self._shapes, tensors)
                ptrs = (C.c_void_p * len(tensors))(*[t.data_ptr() if t is not None else None for t in tensors])
                stream = torch.cuda.current_stream(device).cuda_stream
                _cabi.check(L.seqpan_repack(self._handle, ptrs, stream))
                self._wsig, self._wptrs = sig, tensors

    @staticmethod
    def _check_numel(shp, tensors):
        """Every weight the library will read must have exactly the element count its kernels index (a short GloVe table
        or a foreign checkpoint would otherwise be read out of bounds)."""
        L = _cabi.lib()
        for i, (name, t) in enumerate(zip(_cabi.weight_names(), tensors)):
            want = int(L.seqpan_weight_numel(C.byref(shp), i))
            if want > 0 and t is None:
                raise _cabi.SeqpanError(f"parameter {name} is missing")
            if want > 0 and t.numel() != want:
                raise _cabi.SeqpanError(f"parameter {name} has {t.numel()} elements, the configured shapes need {want} "
                                        f"(configs.num_words / num_chars / vlen / vdim must match the tensors)")

    def _check_inputs(self, word_ids, char_ids, vfeat_in, vmask, tmask, video_index, encoded=False):
        if not vfeat_in.is_cuda:
            raise _cabi.SeqpanError("inputs must be CUDA tensors (the reference moves them in train_engine_SeqPAN, "
                                    "models/SeqPAN.py:173); there is no CPU path")
        device = vfeat_in.device
        for name, t in (("word_ids", word_ids), ("char_ids", char_ids), ("vmask", vmask), ("tmask", tmask)):
            if t.device != device:
                raise _cabi.SeqpanError(f"{name} is on {t.device} but vfeat_in is on {device}: all five inputs must be on one CUDA device")
        if vmask.dim() != 2 or word_ids.dim() != 2 or char_ids.dim() != 3 or tmask.dim() != 2:
            raise _cabi.SeqpanError("expected word_ids [B,T], char_ids [B,T,C], vmask [B,L], tmask [B,T]")
        B, Lv = vmask.shape
        T, Cc = word_ids.shape[1], char_ids.shape[2]
        if word_ids.shape != (B, T) or char_ids.shape != (B, T, Cc) or tmask.shape != (B, T):
            raise _cabi.SeqpanError(f"batch / length mismatch: word_ids {tuple(word_ids.shape)}, char_ids {tuple(char_ids.shape)}, "
                                    f"tmask {tuple(tmask.shape)} against vmask {tuple(vmask.shape)}")
        U = B if video_index is None and not encoded else vfeat_in.shape[0]
        if encoded:   # vfeat_in = the rows of VideoEncodings: any number of clips, at least B without video_index
            if Lv != self.configs.model.vlen or vfeat_in.shape != (U, Lv, 128) or U < (B if video_index is None else 1):
                raise _cabi.SeqpanError(f"video_encodings.rows must be [U,{self.configs.model.vlen},128] with U >= 1 (U >= B={B} "
                                        f"without video_index), got {tuple(vfeat_in.shape)} with vmask {tuple(vmask.shape)}")
        elif Lv != self.configs.model.vlen or vfeat_in.shape != (U, Lv, self.configs.model.vdim) or not 1 <= U <= B:
            raise _cabi.SeqpanError(f"vfeat_in must be [B,{self.configs.model.vlen},{self.configs.model.vdim}] (or [U<=B,...] "
                                    f"with video_index), got {tuple(vfeat_in.shape)} with vmask {tuple(vmask.shape)}")
        if video_index is not None and video_index.shape != (B,):
            raise _cabi.SeqpanError(f"video_index must be [B={B}], got {tuple(video_index.shape)}")
        return device, B, Lv, T, Cc, U

    # ---- the hot path ----------------------------------------------------------------------------------
    def forward(self, word_ids, char_ids, vfeat_in, vmask, tmask, *, gumbel=None, video_index=None, video_encodings=None):
        """models/SeqPAN.py:50-95.  ``gumbel`` (keyword-only, optional) injects the ``[B,L,4]`` noise that
        ``F.gumbel_softmax`` would draw (parity tests against a CPU run); by default it is drawn on the device by
        the same torch call the reference makes, so a seeded reference on the same GPU sees the same noise.

        ``video_index`` (keyword-only, optional; SURVEY.md section 8 row f1): ``vfeat_in`` then holds every clip ONCE,
        ``[U,vlen,vdim]``, and ``video_index[b]`` names the clip of pair ``b``.  The query-independent video branch
        (VisualProjection + the video half of the shared encoder, models/SeqPAN.py:57,59) runs once per clip; the
        outputs equal the plain call on ``vfeat_in[video_index]``.

        ``video_encodings`` (keyword-only, optional; DESIGN.md section 12): clips stored by :meth:`encode_videos`, in place of
        ``vfeat_in`` (pass ``None`` for it).  ``video_index[b]`` names the clip of pair ``b`` among them (``None``: clip ``b``);
        only the query half of the forward runs, and the outputs are bit-identical to ``forward(vfeats, video_index=...)`` on the
        raw clips.  Eval mode only; encodings of another precision or model variant, or of weights that changed since they
        were made (optimizer step, ``load_state_dict``, :meth:`repack`; not checked under :meth:`freeze`), raise.

        In ``train()`` mode (no ``video_index``) the forward runs with dropout on the training kernels.  When grad mode is on
        and some parameter or ``vfeat_in`` requires grad, the outputs carry an autograd graph: ``loss.backward()`` of any torch
        loss on them fills ``p.grad`` (and ``vfeat_in.grad``) through the training kernels' backward, once per forward (no
        double backward, no ``retain_graph``).  ``eval()`` mode never records one."""
        if video_encodings is not None:
            self._check_encoded_call(video_encodings, vfeat_in, video_index)
        _cabi.require_device()
        if self.training:
            # training mode (dropout active, models/layers.py nn.Dropout sites): the primitive-by-primitive forward of
            # vmrframe_b200/train.py.  With grad mode on and a parameter (or vfeat_in) that requires grad, the outputs are
            # attached to the autograd graph through one node whose backward runs the tape's adjoints on the training
            # kernels, so any torch loss on them backpropagates; otherwise (no_grad, inference_mode, all frozen) no tape is
            # recorded.  Both routes compute bit-identical values.  train_engine_SeqPAN / TrainStep run forward, the
            # reference's losses and backward in one call instead.
            if self._VARIANT not in (_cabi.VARIANT_SEQPAN, _cabi.VARIANT_BASEFAST, _cabi.VARIANT_MULTITEACHER,
                                     _cabi.VARIANT_BACKBONE) or video_index is not None:
                raise NotImplementedError("the training forward exists for SeqPAN, BaseFast, MultiTeacher and BackBone (no video_index)")
            from . import train as _train
            device = self._check_inputs(word_ids, char_ids, vfeat_in, vmask, tmask, None)[0]
            if self.sync_timing:
                torch.cuda.synchronize()
            start = time.time()
            graph = torch.is_grad_enabled() and (vfeat_in.requires_grad or any(p.requires_grad for p in self.parameters()))
            fwd = _train.forward_differentiable if graph else _train.forward_only
            with torch.cuda.device(device):
                sl, el, ms = fwd(self, word_ids.to(torch.int64).contiguous(), char_ids.to(torch.int64).contiguous(),
                                 vfeat_in.contiguous(), vmask, tmask, gumbel)
            consume_time = 0.0
            if self.sync_timing:
                torch.cuda.synchronize()
                consume_time = time.time() - start
            if ms is None:      # BackBone: the reference's four keys (models/BackBone.py:70-75)
                return {"slogits": sl, "elogits": el, "vmask": vmask, "consume_time": consume_time}
            return {"slogits": sl, "elogits": el, "vmask": vmask, "match_score": ms, "label_embs": self.label_embs,
                    "consume_time": consume_time}
        enc = video_encodings
        device, B, Lv, T, Cc, U = self._check_inputs(word_ids, char_ids, vfeat_in if enc is None else enc.rows, vmask, tmask,
                                                     video_index, encoded=enc is not None)
        if video_index is not None:
            video_index = video_index.to(device=device, dtype=torch.int32).contiguous()
        word_ids = word_ids.to(torch.int64).contiguous()
        char_ids = char_ids.to(torch.int64).contiguous()
        vfeat = vfeat_in.to(torch.float32).contiguous() if enc is None else enc.rows
        vm = vmask.to(torch.float32).contiguous()
        tm = tmask.to(torch.float32).contiguous()
        if not self._MATCH_HEAD:      # BackBone: no Gumbel softmax, nothing drawn (the library ignores the pointer)
            gumbel = torch.empty(0, dtype=torch.float32, device=device)
        elif gumbel is None:
            # == F.gumbel_softmax's draw (torch/nn/functional.py): -empty_like(logits).exponential_().log()
            gumbel = -torch.empty(B, Lv, 4, dtype=torch.float32, device=device).exponential_().log()
        else:
            gumbel = gumbel.to(device=device, dtype=torch.float32).contiguous()
        with torch.cuda.device(device):
            self._ensure_handle(device, B, T, Cc)
            if enc is not None:
                self._check_encoding_weights(enc)
            slogits = torch.empty(B, Lv, dtype=torch.float32, device=device)
            elogits = torch.empty(B, Lv, dtype=torch.float32, device=device)
            match_score = torch.empty(B, Lv, 4, dtype=torch.float32, device=device)
            if self.sync_timing:
                torch.cuda.synchronize()
            start = time.time()
            stream = torch.cuda.current_stream(device).cuda_stream
            if enc is not None:
                _cabi.check(_cabi.lib().seqpan_forward_encoded(
                    self._handle, word_ids.data_ptr(), char_ids.data_ptr(), vfeat.data_ptr(),
                    video_index.data_ptr() if video_index is not None else None, U, vm.data_ptr(), tm.data_ptr(),
                    gumbel.data_ptr(), B, T, Cc, slogits.data_ptr(), elogits.data_ptr(), match_score.data_ptr(),
                    self._workspace.data_ptr(), self._workspace.numel(), stream))
            elif video_index is None:
                _cabi.check(_cabi.lib().seqpan_forward(
                    self._handle, word_ids.data_ptr(), char_ids.data_ptr(), vfeat.data_ptr(), vm.data_ptr(), tm.data_ptr(),
                    gumbel.data_ptr(), B, T, Cc, slogits.data_ptr(), elogits.data_ptr(), match_score.data_ptr(),
                    self._workspace.data_ptr(), self._workspace.numel(), stream))
            else:
                _cabi.check(_cabi.lib().seqpan_forward_shared_video(
                    self._handle, word_ids.data_ptr(), char_ids.data_ptr(), vfeat.data_ptr(), video_index.data_ptr(), U,
                    vm.data_ptr(), tm.data_ptr(), gumbel.data_ptr(), B, T, Cc, slogits.data_ptr(), elogits.data_ptr(),
                    match_score.data_ptr(), self._workspace.data_ptr(), self._workspace.numel(), stream))
            consume_time = 0.0
            if self.sync_timing:
                torch.cuda.synchronize()
                consume_time = time.time() - start
        if not self._MATCH_HEAD:     # models/BackBone.py:70-74: four keys
            return {"slogits": slogits, "elogits": elogits, "vmask": vmask, "consume_time": consume_time}
        return {"slogits": slogits, "elogits": elogits, "vmask": vmask, "match_score": match_score,
                "label_embs": self.label_embs, "consume_time": consume_time}

    def forward_into(self, word_ids, char_ids, vfeat, vmask, tmask, gumbel, slogits, elogits, match_score, video_index=None,
                     video_encodings=None):
        """The raw call behind :meth:`forward` for callers that own every buffer (the engine's static ring): all
        arguments are contiguous CUDA tensors of the C ABI's dtypes (int64 ids, float32 everything else; int32
        ``video_index`` with ``vfeat`` = the ``[U,L,V]`` unique clips) on one device; nothing is allocated, converted or
        checked here beyond what the library checks.  With ``video_encodings`` (see :meth:`forward`) ``vfeat`` is ignored
        and ``video_index`` indexes the encodings' rows (out-of-range indices are clamped by the library, not reported)."""
        device = (vfeat if video_encodings is None else video_encodings.rows).device
        B, T, Cc = word_ids.shape[0], word_ids.shape[1], char_ids.shape[2]
        with torch.cuda.device(device):
            self._ensure_handle(device, B, T, Cc)
            if video_encodings is not None:
                rows = video_encodings.rows
                _cabi.check(_cabi.lib().seqpan_forward_encoded(
                    self._handle, word_ids.data_ptr(), char_ids.data_ptr(), rows.data_ptr(),
                    video_index.data_ptr() if video_index is not None else None, rows.shape[0], vmask.data_ptr(),
                    tmask.data_ptr(), gumbel.data_ptr(), B, T, Cc, slogits.data_ptr(), elogits.data_ptr(),
                    match_score.data_ptr(), self._workspace.data_ptr(), self._workspace.numel(),
                    torch.cuda.current_stream(device).cuda_stream))
                return
            if video_index is not None:
                _cabi.check(_cabi.lib().seqpan_forward_shared_video(
                    self._handle, word_ids.data_ptr(), char_ids.data_ptr(), vfeat.data_ptr(), video_index.data_ptr(),
                    vfeat.shape[0], vmask.data_ptr(), tmask.data_ptr(), gumbel.data_ptr(), B, T, Cc, slogits.data_ptr(),
                    elogits.data_ptr(), match_score.data_ptr(), self._workspace.data_ptr(), self._workspace.numel(),
                    torch.cuda.current_stream(device).cuda_stream))
                return
            _cabi.check(_cabi.lib().seqpan_forward(
                self._handle, word_ids.data_ptr(), char_ids.data_ptr(), vfeat.data_ptr(), vmask.data_ptr(),
                tmask.data_ptr(), gumbel.data_ptr(), B, T, Cc, slogits.data_ptr(), elogits.data_ptr(),
                match_score.data_ptr(), self._workspace.data_ptr(), self._workspace.numel(),
                torch.cuda.current_stream(device).cuda_stream))

    # ---- stored video encodings (DESIGN.md section 12) ---------------------------------------------------------
    def encode_videos(self, vfeats, chunk: int = 256) -> VideoEncodings:
        """Runs the query-independent video branch -- VisualProjection + the video half of the shared FeatureEncoder
        (models/SeqPAN.py:57,59) -- once over ``vfeats`` ``[U,vlen,vdim]`` and returns its ``[U,vlen,128]`` fp32 rows as
        :class:`VideoEncodings` for ``forward(..., None, ..., video_encodings=, video_index=)`` and
        ``evaluate(video_encodings=)``: later queries of these clips move no video bytes and skip that branch.  ``vfeats`` is a
        CUDA tensor; the encodings land on its device.  At most ``chunk`` clips go through the library per call, which bounds
        the workspace (``chunk`` above the library's batch limit of 768 is lowered to it); a clip's encoding does not depend on
        the chunking.  Eval mode only: in ``train()``
        dropout acts on the video branch of every pair, so there is nothing to store."""
        if self.training:
            raise _cabi.SeqpanError("encode_videos needs eval(): in train() dropout acts on the video branch of every pair")
        m = self.configs.model
        if vfeats.dim() != 3 or tuple(vfeats.shape[1:]) != (m.vlen, m.vdim):
            raise _cabi.SeqpanError(f"vfeats must be [U,{m.vlen},{m.vdim}], got {tuple(vfeats.shape)}")
        if int(chunk) < 1:
            raise ValueError(f"chunk={chunk} must be >= 1")
        _cabi.require_device()
        if not vfeats.is_cuda:
            raise _cabi.SeqpanError("vfeats must be a CUDA tensor (there is no CPU path)")
        device, U = vfeats.device, vfeats.shape[0]
        n = max(1, min(int(chunk), U, _MAX_BATCH))
        rows = torch.empty(U, m.vlen, 128, dtype=torch.float32, device=device)
        with torch.cuda.device(device):
            self._ensure_handle(device, n, 1, 4)
            stream = torch.cuda.current_stream(device).cuda_stream
            for lo in range(0, U, n):
                vf = vfeats[lo:lo + n].to(torch.float32).contiguous()
                _cabi.check(_cabi.lib().seqpan_encode_videos(self._handle, vf.data_ptr(), vf.shape[0], rows[lo:lo + n].data_ptr(),
                                                             self._workspace.data_ptr(), self._workspace.numel(), stream))
        return VideoEncodings(rows, self.precision, self._VARIANT, self._packed_weights_key())

    def _check_encoded_call(self, enc, vfeat_in, video_index):
        """The checks of a forward on stored encodings that need neither the device nor the library handle."""
        if vfeat_in is not None:
            raise _cabi.SeqpanError("pass vfeat_in=None with video_encodings: the clips come from the encodings")
        if self.training:
            raise _cabi.SeqpanError("video_encodings need eval(): in train() dropout acts on the video branch of every pair")
        if not isinstance(enc, VideoEncodings):
            raise _cabi.SeqpanError(f"video_encodings must come from encode_videos, got {type(enc).__name__}")
        if enc.precision != self.precision or enc.variant != self._VARIANT:
            raise _cabi.SeqpanError(f"the encodings were made by a {enc.precision} model of variant {enc.variant}, this is a "
                                    f"{self.precision} model of variant {self._VARIANT}")
        rows, vlen = enc.rows, self.configs.model.vlen
        if rows.dim() != 3 or tuple(rows.shape[1:]) != (vlen, 128) or rows.dtype != torch.float32 or not rows.is_contiguous():
            raise _cabi.SeqpanError(f"video_encodings.rows must be a contiguous float32 [U,{vlen},128] tensor, got "
                                    f"{rows.dtype} {tuple(rows.shape)}")
        if video_index is not None and video_index.numel() > 0:
            lo, hi = int(video_index.min()), int(video_index.max())
            if lo < 0 or hi >= rows.shape[0]:
                raise _cabi.SeqpanError(f"video_index values [{lo},{hi}] outside [0,{rows.shape[0]}) of the encodings")

    def _packed_weights_key(self):
        """What the current kernel context packed: the weights' signature at packing time (under :meth:`freeze` it can lag the
        parameters) and the count of explicit :meth:`repack` calls (which follow edits the signature cannot see)."""
        return self._repacks, self._wsig

    def _check_encoding_weights(self, enc):
        """Encodings made with other weights are stale (the current kernel context's signature is fresh after _ensure_handle)."""
        if not self._frozen and enc.signature != self._packed_weights_key():
            raise _cabi.SeqpanError("the weights changed since these encodings were made (optimizer step, load_state_dict, "
                                    "repack): call encode_videos again")

    def set_profile(self, on: bool = True):
        """Per-launch CUDA-event timing inside the library (bench.py's per-kernel roofline)."""
        _cabi.check(_cabi.lib().seqpan_set_profile(self._handle, int(on)))

    def profile_summary(self) -> dict:
        """{kernel tag: (launch count, total ms)} since ``set_profile(True)``; synchronises the device."""
        buf = C.create_string_buffer(1 << 16)
        _cabi.check(_cabi.lib().seqpan_profile_summary(self._handle, buf, len(buf)))
        out = {}
        for line in buf.value.decode().splitlines():
            tag, n, ms = line.rsplit(" ", 2)
            out[tag] = (int(n), float(ms))
        return out

    def last_launch_count(self) -> int:
        return int(_cabi.lib().seqpan_last_launch_count(self._handle)) if self._handle is not None else 0

    def debug_tap(self, name: str) -> torch.Tensor:
        """Intermediate tensor of the last forward (needs ``set_debug_taps(True)`` before it)."""
        cap = self._limits[0] * self.configs.model.vlen * 128
        out = torch.empty(cap, dtype=torch.float32, device=self._workspace.device)
        stream = torch.cuda.current_stream(out.device).cuda_stream
        rows = _cabi.check(_cabi.lib().seqpan_debug_tap(self._handle, name.encode(), self._workspace.data_ptr(),
                                                        out.data_ptr(), cap, stream))
        return out[: rows * 128].view(rows, 128)

    @staticmethod
    def extract_index(start_logits, end_logits):
        return extract_index(start_logits, end_logits)


def _cabi_max_tlen() -> int:
    return 128  # SEQPAN_MAX_TLEN in include/seqpan_b200.h


_MAX_BATCH = 768   # largest SeqpanShapes.max_batch the library accepts (check_shapes in csrc/seqpan_api.cu)


def _decode(start_logits, end_logits, vmask, want_idx, want_fracs):
    _cabi.require_device()
    if not start_logits.is_cuda:
        raise _cabi.SeqpanError("span decode needs CUDA tensors (no CPU path)")
    s = start_logits.detach().to(torch.float32).contiguous()
    e = end_logits.detach().to(torch.float32).contiguous()
    B, L = s.shape
    dev = s.device
    vm = vmask.detach().to(device=dev, dtype=torch.float32).contiguous() if vmask is not None else None
    si = torch.empty(B, dtype=torch.int64, device=dev) if want_idx else None
    ei = torch.empty(B, dtype=torch.int64, device=dev) if want_idx else None
    fr = torch.empty(B, 2, dtype=torch.float32, device=dev) if want_fracs else None
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().seqpan_span_decode(
            s.data_ptr(), e.data_ptr(), vm.data_ptr() if vm is not None else None, B, L,
            si.data_ptr() if si is not None else None, ei.data_ptr() if ei is not None else None,
            fr.data_ptr() if fr is not None else None, torch.cuda.current_stream(dev).cuda_stream))
    return si, ei, fr


def extract_index(start_logits, end_logits):
    """``ConditionedPredictor.extract_index`` (models/layers.py:549-557): (start_index, end_index) LongTensors."""
    si, ei, _ = _decode(start_logits, end_logits, None, True, False)
    return si, ei


def infer_basic(start_logits, end_logits, vmask):
    """``utils/engine.py:28-44``: ``np.ndarray float32 (B,2)`` of start/end indices divided by ``vmask.sum(1)``."""
    _, _, fr = _decode(start_logits, end_logits, vmask, False, True)
    return fr.cpu().numpy()


def infer_basic_device(start_logits, end_logits, vmask):
    """Same as :func:`infer_basic` but leaves the ``[B,2]`` fractions on the device (no host sync)."""
    return _decode(start_logits, end_logits, vmask, False, True)[2]


def _topk(start_logits, end_logits, vmask, k, nms_thresh, want_fracs):
    _cabi.require_device()
    if not start_logits.is_cuda:
        raise _cabi.SeqpanError("top-k span retrieval needs CUDA tensors (no CPU path)")
    s = start_logits.detach().to(torch.float32).contiguous()
    e = end_logits.detach().to(torch.float32).contiguous()
    B, L = s.shape
    dev = s.device
    vm = vmask.detach().to(device=dev, dtype=torch.float32).contiguous() if vmask is not None else None
    k = int(k)
    si = torch.empty(B, max(k, 0), dtype=torch.int64, device=dev)
    ei = torch.empty_like(si)
    sc = torch.empty(B, max(k, 0), dtype=torch.float32, device=dev)
    fr = torch.empty(B, max(k, 0), 2, dtype=torch.float32, device=dev) if want_fracs else None
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().seqpan_span_topk(
            s.data_ptr(), e.data_ptr(), vm.data_ptr() if vm is not None else None, B, L, k, float(nms_thresh),
            si.data_ptr(), ei.data_ptr(), sc.data_ptr(), fr.data_ptr() if fr is not None else None,
            torch.cuda.current_stream(dev).cuda_stream))
    return si, ei, sc, fr


def extract_topk(start_logits, end_logits, vmask=None, k: int = 5, nms_thresh: float = 0.5):
    """The ``k`` best spans of every sample after greedy temporal NMS, as device tensors ``(start_idx, end_idx, scores)`` of
    shape ``[B,k]`` (int64, int64, fp32) in selection order.  Scores are ``sp[i] * ep[j]`` with ``infer_basic``'s
    probabilities (``mask_logits`` first when ``vmask`` is given); a candidate whose IoU with a kept span is at least
    ``nms_thresh`` is suppressed (``nms_thresh=1``: plain top-k).  Slots past the last surviving candidate hold ``-1, -1, 0``.
    At ``k=1`` the start equals :func:`extract_index`'s; the end too unless the best score is attained by several spans."""
    si, ei, sc, _ = _topk(start_logits, end_logits, vmask, k, nms_thresh, False)
    return si, ei, sc


def infer_topk(output, k: int = 5, nms_thresh: float = 0.5):
    """Top-k counterpart of ``infer_SeqPAN`` for the output dict of any of the five models: ``np.ndarray float32 (B,k,2)`` of
    span fractions (indices divided by ``vmask.sum(1)``) in selection order; empty slots are ``-1``."""
    return _topk(output["slogits"], output["elogits"], output["vmask"], k, nms_thresh, True)[3].cpu().numpy()


class BaseFast(SeqPAN):
    """Drop-in for the reference's ``models/BaseFast.py:10-97`` (SURVEY.md section 8 row f3): the same blocks as SeqPAN with a
    2-layer shared ``FeatureEncoder`` (``:27``) and without the two ``DualAttentionBlock`` passes (``:62-68`` are commented
    out; the blocks are still constructed, so they stay in the ``state_dict`` and a reference checkpoint loads with
    ``strict=True``).  Same constructor, ``forward`` signature and output dict as :class:`SeqPAN`."""
    _VARIANT = _cabi.VARIANT_BASEFAST
    _ENC_LAYERS = 2


class BackBone(SeqPAN):
    """Drop-in for the reference's ``models/BackBone.py:10-75``: SeqPAN without the match head (the ``CQConcatenate``
    output feeds the predictor directly, unmasked) and with a second ``FeatureEncoder`` (``tfeat_encoder``) for the text.
    Returns the reference's four keys (``slogits, elogits, vmask, consume_time``)."""
    _VARIANT = _cabi.VARIANT_BACKBONE
    _OWN_TEXT_ENCODER = True
    _MATCH_HEAD = False


class MultiTeacher(SeqPAN):
    """The student forward of the reference's ``models/MultiTeacher.py:12-91``: SeqPAN with a 2-layer shared
    ``FeatureEncoder`` (``:26``); the teachers only enter its training loss (dataset side)."""
    _VARIANT = _cabi.VARIANT_MULTITEACHER
    _ENC_LAYERS = 2


class _Student4(SeqPAN):
    """SeqPAN's blocks on a 4-layer shared encoder without the DualAttentionBlock passes: the student of OneTeacher."""
    _VARIANT = _cabi.VARIANT_STUDENT4


def _runner(cls, configs, modules, precision, sync_timing):
    """A ``SeqPAN``-family runner (library handle management + forward) over EXISTING parameter containers: ``modules`` maps the
    attribute names the weight table walks (``text_encoder``, ``vfeat_encoder``, ...) to modules / parameters owned by someone
    else.  Nothing is constructed (no RNG is consumed)."""
    r = cls.__new__(cls)
    nn.Module.__init__(r)
    r.configs = configs
    for k, v in modules.items():
        setattr(r, k, v)
    r.precision, r.sync_timing = precision, sync_timing
    r._handle = r._limits = r._arena = r._workspace = r._wsig = r._wptrs = None
    r._ctxs, r._ctx_key, r._frozen, r._debug, r._repacks = {}, 0, False, False, 0
    r.eval()
    return r


class OneTeacher(nn.Module):
    """Drop-in for the reference's ``models/OneTeacher.py:10-122`` (SURVEY.md section 8 row f3): a SeqPAN teacher (``*_t0``
    parameters) and a student without DualAttentionBlocks, both evaluated per call (teacher first: its Gumbel draw comes first,
    ``:77`` then ``:108``).  Same constructor and positional ``forward``; the 10-key output dict of ``:114-128``; the reference's
    ``state_dict`` keys and, because the containers are created in the reference's order, its seed-identical default init."""

    def __init__(self, configs, word_vectors, precision: str | None = None, sync_timing: bool = True):
        super().__init__()
        self.configs = configs
        m = configs.model
        dim, droprate = m.dim, m.droprate
        if dim != 128 or m.num_heads != 4 or m.word_dim != 300 or m.char_dim != 100:
            raise ValueError("the B200 kernels are specialised for dim=128, num_heads=4, word_dim=300, char_dim=100")
        # student (models/OneTeacher.py:18-31)
        self.text_encoder = _Embedding(configs.num_words, configs.num_chars, m.word_dim, m.char_dim, dim, word_vectors)
        self.video_affine = _VisualProjection(m.vdim, dim)
        self.feat_encoder = _FeatureEncoder(dim, m.vlen, 4)
        self.q2v_attn = _CQAttention(dim)
        self.v2q_attn = _CQAttention(dim)
        self.cq_cat = _CQConcatenate(dim)
        self.match_conv1d = _Conv1D(dim, 4)
        self.label_embs = nn.Parameter(torch.nn.init.orthogonal_(torch.empty(dim, 4, dtype=torch.float32)))
        self.predictor = _SeqPANPredictor(dim, m.vlen, droprate)
        # teacher 0 (:35-52)
        self.text_encoder_t0 = _Embedding(configs.num_words, configs.num_chars, m.word_dim, m.char_dim, dim, word_vectors)
        self.video_affine_t0 = _VisualProjection(m.vdim, dim)
        self.feat_encoder_t0 = _FeatureEncoder(dim, m.vlen, 4)
        self.dual_attention_block_1_t0 = _DualAttentionBlock(dim)
        self.dual_attention_block_2_t0 = _DualAttentionBlock(dim)
        self.q2v_attn_t0 = _CQAttention(dim)
        self.v2q_attn_t0 = _CQAttention(dim)
        self.cq_cat_t0 = _CQConcatenate(dim)
        self.match_conv1d_t0 = _Conv1D(dim, 4)
        self.label_embs_t0 = nn.Parameter(torch.nn.init.orthogonal_(torch.empty(dim, 4, dtype=torch.float32)))
        self.predictor_t0 = _SeqPANPredictor(dim, m.vlen, droprate)
        prec = precision or getattr(m, "precision", None) or os.environ.get("SEQPAN_PRECISION", "bf16")
        if prec not in _PRECISIONS:
            raise ValueError(f"precision must be one of {list(_PRECISIONS)}")
        self.precision, self.sync_timing = prec, sync_timing
        self._register_load_state_dict_pre_hook(SeqPAN._strip_module_prefix)
        # runners over the containers above; kept out of nn.Module's registry (they own no parameters of their own)
        student = _runner(_Student4, configs, dict(
            text_encoder=self.text_encoder, video_affine=self.video_affine, vfeat_encoder=self.feat_encoder, q2v_attn=self.q2v_attn,
            v2q_attn=self.v2q_attn, cq_cat=self.cq_cat, match_conv1d=self.match_conv1d, label_embs=self.label_embs,
            predictor=self.predictor), prec, False)
        teacher = _runner(SeqPAN, configs, dict(
            text_encoder=self.text_encoder_t0, video_affine=self.video_affine_t0, vfeat_encoder=self.feat_encoder_t0,
            dual_attention_block_1=self.dual_attention_block_1_t0, dual_attention_block_2=self.dual_attention_block_2_t0,
            q2v_attn=self.q2v_attn_t0, v2q_attn=self.v2q_attn_t0, cq_cat=self.cq_cat_t0, match_conv1d=self.match_conv1d_t0,
            label_embs=self.label_embs_t0, predictor=self.predictor_t0), prec, False)
        object.__setattr__(self, "_runners", (teacher, student))

    def forward(self, word_ids, char_ids, vfeat_in, vmask, tmask, *, gumbel=None, gumbel_t0=None, video_encodings=None):
        """models/OneTeacher.py:54-128.  ``gumbel_t0`` / ``gumbel`` inject the teacher's / student's noise (parity tests)."""
        if video_encodings is not None:
            raise NotImplementedError("OneTeacher has two video branches (teacher and student): no stored encodings")
        _cabi.require_device()
        if self.training:
            raise NotImplementedError("OneTeacher ships the inference forward; call model.eval()")
        teacher, student = self._runners
        if self.sync_timing:
            torch.cuda.synchronize()
        start = time.time()
        t = teacher(word_ids, char_ids, vfeat_in, vmask, tmask, gumbel=gumbel_t0)
        s = student(word_ids, char_ids, vfeat_in, vmask, tmask, gumbel=gumbel)
        consume_time = 0.0
        if self.sync_timing:
            torch.cuda.synchronize()
            consume_time = time.time() - start
        return {"slogits_t0": t["slogits"], "elogits_t0": t["elogits"], "match_score_t0": t["match_score"],
                "label_embs_t0": self.label_embs_t0, "slogits": s["slogits"], "elogits": s["elogits"],
                "match_score": s["match_score"], "label_embs": self.label_embs, "vmask": vmask, "consume_time": consume_time}


    def encode_videos(self, vfeats, chunk: int = 256):
        raise NotImplementedError("OneTeacher has two video branches (teacher and student); stored encodings exist for SeqPAN, "
                                  "BaseFast, MultiTeacher and BackBone")


def infer_OneTeacher(output, configs=None):
    """models/OneTeacher.py:169-173: the span decode of the STUDENT's logits."""
    return infer_basic(output["slogits"], output["elogits"], output["vmask"])


def infer_SeqPAN(output, configs=None):
    """models/SeqPAN.py:185-192."""
    return infer_basic(output["slogits"], output["elogits"], output["vmask"])


def train_engine_SeqPAN(model, data, configs, runtype=None):
    """models/SeqPAN.py:171-182: moves the batch to ``configs.device``, runs the forward and returns ``(loss, output)``.

    ``model.train()`` (main.py:82-97): forward with dropout, both losses (models/loss.py:24-54) AND the backward run on the
    training kernels (vmrframe_b200/train.py); the returned ``loss`` is attached to the parameters, so the reference's
    ``optimizer.zero_grad(); loss.backward(); clip_grad_norm_(...); optimizer.step()`` works unchanged.
    ``model.eval()`` (main.py:112-127): the fused inference forward; the loss is a value without a graph."""
    return _train_engine_on_tape(model, data, configs, "train", _LABELS, _reference_loss)


def infer_BaseFast(output, configs=None):
    """models/BaseFast.py:130-136."""
    return infer_basic(output["slogits"], output["elogits"], output["vmask"])


def train_engine_BaseFast(model, data, configs, runtype=None):
    """models/BaseFast.py:113-127: like ``train_engine_SeqPAN`` but the location loss sees ``sigmoid(logits)`` (``:119-120``).
    ``model.train()``: forward, losses and backward on the training kernels (``loss.backward()`` hands out the gradients);
    ``model.eval()``: fused inference forward, loss value only."""
    return _train_engine_on_tape(model, data, configs, "train", _LABELS,
                                 lambda output, data: _reference_loss(output, data, sigmoid_first=True))


_LABELS = ("label1ds", "NER_labels")      # what train_engine_SeqPAN / _BaseFast compute their losses from


def _reference_loss(output, data, sigmoid_first=False):
    """The loss value of ``train_engine_SeqPAN`` / ``_BaseFast`` on the inference outputs: ``engine.lossfun_loc`` (on
    ``sigmoid(logits)`` with ``sigmoid_first``) + ``lossfun_match`` in torch."""
    from .engine import lossfun_loc, lossfun_match
    s, e = output["slogits"], output["elogits"]
    if sigmoid_first:
        s, e = torch.sigmoid(s), torch.sigmoid(e)
    return lossfun_loc(s, e, data["label1ds"][:, 0, :], data["label1ds"][:, 1, :], data["vmasks"]) + lossfun_match(
        output["match_score"], output["label_embs"], data["NER_labels"], data["vmasks"])


def _train_engine_on_tape(model, data, configs, runtype, labels=(), eval_loss=None):
    """Common body of the train engines: moves the batch to ``configs.device``; ``model.train()`` -> forward, the model's loss
    terms and the backward on the training kernels (``loss.backward()`` hands out the gradients); ``model.eval()`` -> fused
    inference forward and the loss VALUE, ``eval_loss(output, data)`` or else from the same loss kernels as the tape.  A batch
    without one of the keys ``labels`` runs the module's forward in either mode and has no loss."""
    from . import train as _train
    data = {k: v.to(configs.device) for k, v in data.items()}
    runtype = "train" if runtype is None else runtype
    labelled = all(k in data for k in labels)
    if model.training and labelled:
        start = time.time()
        loss, output = _train.tape_loss(model, data, runtype=runtype)
        output["consume_time"] = time.time() - start
        return loss, output
    output = model(data["words_ids"], data["char_ids"], data["vfeats"], data["vmasks"], data["tmasks"])
    if not labelled:
        return None, output
    loss = eval_loss(output, data) if eval_loss is not None else _train.loss_from_outputs(model, output, data, runtype)
    return loss, output


def train_engine_MultiTeacher(model, data, configs, runtype=None):
    """models/MultiTeacher.py:165-195: location loss on ``sigmoid(logits)`` (the match loss is commented out there, ``:175``); for
    ``runtype == "train"`` plus, per teacher k in 0..2, ``mean(calculate_adapt_cof(label1d_tks, label1ds) *
    lossfun_softloc(..., configs.loss.tk_temperature)) * configs.loss.tk_cof`` on the teacher labels the collate adds
    (``label1d_t0s`` / ``_t1s`` / ``_t2s``, ``[B,2,L]``)."""
    return _train_engine_on_tape(model, data, configs, runtype)


def train_engine_BackBone(model, data, configs, runmode=None):
    """models/BackBone.py:94-107: the location loss only."""
    return _train_engine_on_tape(model, data, configs, runmode)


def infer_MultiTeacher(output, configs=None):
    """models/MultiTeacher.py (infer_MultiTeacher): the same span decode."""
    return infer_basic(output["slogits"], output["elogits"], output["vmask"])


def infer_BackBone(output, configs=None):
    """models/BackBone.py (infer_BackBone): the same span decode."""
    return infer_basic(output["slogits"], output["elogits"], output["vmask"])
