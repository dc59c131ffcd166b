"""Verbalizer with the reference's interface (trainer/verb.py:420-643, copy in demo/verb.py).

`ManualVerbalizer(tokenizer, classes, label_words, prefix, multi_token_handler, post_log_softmax)` keeps
the constructor, `register_calibrate_logits` and `process_logits(logits[B, V]) -> [B, C]` (project,
handle_multi_token, normalize, calibrate, log and aggregate of trainer/verb.py:524-643 in one kernel,
lrb_verbalizer_from_logits).  The fast path is

    score_hidden(hidden_last[B, H], lm_head_weight[V, H]) -> [B, C]

which never forms the [B, V] logits: the CUDA kernel multiplies only the label-word rows of the
lm_head (model/llm.py:113-114 projects all T positions onto all V tokens) and applies
project -> (softmax -> log) -> aggregate in the same launch.
"""
from __future__ import annotations

from typing import List, Mapping, Optional, Sequence, Union

import torch

from . import _lib


class ManualVerbalizer:
    def __init__(self, tokenizer, classes: Optional[Sequence] = None, num_classes: Optional[int] = None,
                 label_words: Optional[Union[Sequence, Mapping]] = None, prefix: Optional[str] = " ",
                 multi_token_handler: Optional[str] = "first", post_log_softmax: Optional[bool] = True):
        self.tokenizer = tokenizer
        if classes is not None and num_classes is not None:
            assert len(classes) == num_classes, "len(classes) != num_classes"
        self.classes = list(classes) if classes is not None else None
        self.num_classes = len(self.classes) if self.classes is not None else num_classes
        self.prefix = prefix
        self.multi_token_handler = multi_token_handler
        self.post_log_softmax = post_log_softmax
        self._label_words = None
        self._calibrate_logits = None
        if label_words is not None:
            self.label_words = label_words

    # ---- calibration (trainer/verb.py:202-208, 616-643) ---------------------------------------------
    def register_calibrate_logits(self, logits: Optional[torch.Tensor]) -> None:
        """Registers the [V] calibration logits (None removes them).  With `post_log_softmax` the label-word
        probabilities are then divided by the calibration vector's own label-word probabilities (+1e-15) and
        renormalised over all label words before the log -- `ManualVerbalizer.calibrate` -- inside the same kernel."""
        if logits is not None:
            if logits.dim() != 1:
                raise AssertionError("self._calibrate_logits are not 1-d tensor")       # trainer/verb.py:626-628
            logits = logits.detach().to(torch.float32).contiguous()
        self._calibrate_logits = logits
        if hasattr(self, "_dev_cache"):
            self._dev_cache = {k: v for k, v in self._dev_cache.items() if not (isinstance(k, tuple) and k[0] == "cal")}

    def _calib_ptr(self, dev, V: int):
        """Device pointer of the calibration logits (0 = none); they are only consulted in post_log_softmax mode."""
        if self._calibrate_logits is None or not self.post_log_softmax:
            return None
        if self._calibrate_logits.numel() != V:
            raise ValueError(f"calibration logits have {self._calibrate_logits.numel()} entries, the vocabulary {V}")
        key = ("cal", str(dev))
        if key not in self._dev_cache:
            self._dev_cache[key] = self._calibrate_logits.to(dev)
        return self._dev_cache[key]

    # ---- label words (trainer/verb.py:136-160 setter semantics, :463-522) -------------------------
    @property
    def label_words(self):
        return self._label_words

    @label_words.setter
    def label_words(self, label_words):
        if label_words is None:
            return
        if isinstance(label_words, Mapping):
            if self.classes is None:
                self.classes = list(label_words.keys())
                self.num_classes = len(self.classes)
            label_words = [label_words[c] for c in self.classes]
        label_words = list(label_words)
        if len(label_words) > 0 and isinstance(label_words[0], str):
            label_words = [[w] for w in label_words]
        with_prefix: List[List[str]] = []
        for words in label_words:
            row = []
            for w in words:
                row.append(w.split("<!>")[1] if w.startswith("<!>") else (self.prefix or "") + w)
            with_prefix.append(row)
        self._label_words = with_prefix
        self.generate_parameters()

    def generate_parameters(self) -> None:
        ids = [[self.tokenizer.encode(w, add_special_tokens=False) for w in words] for words in self._label_words]
        max_len = max(max(len(t) for t in per) for per in ids)
        max_words = max(len(per) for per in ids)
        C = len(ids)
        words_ids = torch.zeros(C, max_words, max_len, dtype=torch.int64)
        words_ids_mask = torch.zeros(C, max_words, max_len, dtype=torch.int64)
        for c, per in enumerate(ids):
            for w, toks in enumerate(per):
                words_ids[c, w, : len(toks)] = torch.tensor(toks, dtype=torch.int64)
                words_ids_mask[c, w, : len(toks)] = 1
        self.label_words_ids = words_ids                                   # [C, W, T]
        self.words_ids_mask = words_ids_mask                               # [C, W, T]
        self.label_words_mask = torch.clamp(words_ids_mask.sum(dim=-1), max=1)   # [C, W]
        self._dev_cache = {}

    def _check_token_ids(self, V: int) -> None:
        """The reference indexes `logits[:, label_words_ids]` (trainer/verb.py:539), which raises IndexError for a
        token id >= V; the kernels would read token 0 instead, for a negative id too.  Checked on the host copy of the
        ids, so no device synchronisation."""
        lo, hi = int(self.label_words_ids.min()), int(self.label_words_ids.max())
        if lo < 0 or hi >= V:
            raise IndexError(f"label word token ids span [{lo}, {hi}], outside the {V} rows of the logits / lm_head")

    # ---- fused fast path ---------------------------------------------------------------------------
    def _device_params(self, dev):
        key = str(dev)
        if key not in self._dev_cache:
            first = self.label_words_ids[:, :, 0].to(torch.int32).contiguous().to(dev)
            mask = self.label_words_mask.to(torch.uint8).contiguous().to(dev)
            self._dev_cache[key] = (first, mask)
        return self._dev_cache[key]

    @torch.no_grad()
    def score_hidden(self, hidden_last: torch.Tensor, lm_head_weight: torch.Tensor,
                     round_logits_to_bf16: bool = True) -> torch.Tensor:
        """[B, H] bf16 x label rows of [V, H] bf16 -> [B, C] fp32 label scores.

        round_logits_to_bf16 mirrors `lm_head(hidden).float()` of a bf16 model (model/llm.py:113-114),
        whose logits are bf16 values widened to fp32."""
        if self.multi_token_handler != "first":
            raise NotImplementedError("the fused kernel implements multi_token_handler='first' "
                                      "(the reference default, trainer/verb.py:441)")
        self._check_token_ids(lm_head_weight.shape[0])
        if not hidden_last.is_cuda:
            raise RuntimeError("score_hidden runs on the GPU only (no CPU fallback)")
        lib = _lib.load()
        dev = hidden_last.device
        h = hidden_last.to(torch.bfloat16).contiguous()
        w = lm_head_weight.to(torch.bfloat16).contiguous()
        ids, mask = self._device_params(dev)
        B, H = h.shape
        C, W = ids.shape
        out = torch.empty(B, C, dtype=torch.float32, device=dev)
        cal = self._calib_ptr(dev, w.shape[0])
        with _lib.on_device(h):
            _lib.check(lib.lrb_verbalizer_score(_lib.ptr(h), _lib.ptr(w), B, H, w.shape[0], _lib.ptr(ids),
                                                _lib.ptr(mask), C, W, 1 if self.post_log_softmax else 0,
                                                1 if round_logits_to_bf16 else 0,
                                                _lib.ptr(cal) if cal is not None else None, _lib.ptr(out),
                                                _lib.stream_handle()))
        return out

    # ---- the reference's entry point on precomputed logits (trainer/verb.py:524-614) ----------------
    _HANDLERS = {"first": 0, "max": 1, "mean": 2}

    def process_logits(self, logits: torch.Tensor) -> torch.Tensor:
        """trainer/verb.py:546-586.  CUDA logits run in lrb_verbalizer_from_logits (one kernel: gather the
        label-word logits, multi-token handler, project, normalize/log, aggregate); host tensors -- the
        reference's trainer hands over numpy logits (trainer/llm.py:65-68) -- are moved to the current CUDA
        device first when there is one."""
        if self.multi_token_handler not in self._HANDLERS:
            raise ValueError(f"multi_token_handler {self.multi_token_handler} not configured")
        self._check_token_ids(logits.shape[-1])
        if not logits.is_cuda and torch.cuda.is_available():
            return self.process_logits(logits.cuda()).to(logits.device)
        if logits.is_cuda:
            lib = _lib.load()
            dev = logits.device
            lg = logits.to(torch.float32)
            B, V = lg.shape
            # the kernel reads rows at a pitch >= V with unit inner stride: broadcast rows (stride 0) are copied
            if lg.stride(-1) != 1 or (B > 1 and lg.stride(0) < V):
                lg = lg.contiguous()
            ld = lg.stride(0) if B > 1 else V       # the pitch of a single row is never used
            ids, tmask, wmask = self._device_token_params(dev)
            C, W, T = ids.shape
            out = torch.empty(B, C, dtype=torch.float32, device=dev)
            cal = self._calib_ptr(dev, V)
            with _lib.on_device(lg):
                _lib.check(lib.lrb_verbalizer_from_logits(lg.data_ptr(), ld, B, V, _lib.ptr(ids),
                                                          _lib.ptr(tmask), _lib.ptr(wmask), C, W, T,
                                                          self._HANDLERS[self.multi_token_handler],
                                                          1 if self.post_log_softmax else 0,
                                                          _lib.ptr(cal) if cal is not None else None, _lib.ptr(out),
                                                          _lib.stream_handle()))
            return out
        raise RuntimeError("ManualVerbalizer.process_logits needs a CUDA device: project / normalize / aggregate "
                           "(trainer/verb.py:524-614) run in one kernel, there is no CPU path")

    def _device_token_params(self, dev):
        key = ("tok", str(dev))
        if key not in self._dev_cache:
            self._dev_cache[key] = (self.label_words_ids.to(torch.int32).contiguous().to(dev),
                                    self.words_ids_mask.to(torch.uint8).contiguous().to(dev),
                                    self.label_words_mask.to(torch.uint8).contiguous().to(dev))
        return self._dev_cache[key]
