"""Drop-in LRURec for B200 (reference: model/lru.py).

`LRURec(args)` has the reference's constructor, parameter names / dtypes (so
`load_state_dict(torch.load('best_acc_model.pth')['model_state_dict'])` works unchanged) and
`forward(x) -> FloatTensor[B, L, N+1]`.  All arithmetic runs in the sm_100a kernels behind the C ABI
(include/llamarec_b200.h); torch only owns device memory and streams.  The module's sub-modules are
parameter containers -- their own forward() is never called.

Fast entry points added on top of the reference interface:
    encode(x)                -> u[B, 64]      last-position state (what trainer/lru.py:33 slices out)
    retrieve(x, k, ...)      -> top-k ids/scores (+ label ranks and Recall/MRR/NDCG sums) without
                                materialising the B x (N+1) score matrix
"""
from __future__ import annotations

import functools
import math
import warnings
from typing import Dict, Optional, Sequence

import torch
import torch.nn as nn

from . import _lib
from .packing import pack_encoder_weights, unpack_encoder_grads

SMALL_CATALOGUE_ROWS = 1 << 17   # up to here 'auto' precision scores in exact fp32


def _on_model_device(fn):
    """Runs a method with the model's device current: the C-ABI launches go to the CURRENT device's stream, so a
    model on cuda:1 called from a process whose current device is cuda:0 would otherwise launch on the wrong GPU."""
    @functools.wraps(fn)
    def wrap(self, *args, **kwargs):
        w = self.embedding.token.weight
        if not w.is_cuda:
            raise RuntimeError("llamarec_b200 has no CPU path: move the model to a CUDA device (model.cuda())")
        with torch.cuda.device(w.device):
            return fn(self, *args, **kwargs)
    return wrap


class _TrainStep(torch.autograd.Function):
    """loss = CrossEntropyLoss(ignore_index)(model(x).view(-1, N+1), labels.view(-1)) with a backward: ONE call of
    lrb_train_step (lrb_train_step_dropout with dropout) computes the loss and the gradient of every parameter
    (forward activations never leave the library's workspace); backward() hands the stored gradients to autograd,
    scaled by the incoming gradient.
    `dropout` is (p_embed, p_attn, p_ffn, seed) or None.  Inputs after (model, x, labels, ignore_index, dropout) are
    the model's parameters in named_parameters() order."""

    @staticmethod
    def forward(ctx, model, x, labels, ignore_index, dropout, *params):
        loss, grads = model._train_step(x, labels, ignore_index, dropout)
        ctx.grads = grads
        return loss

    @staticmethod
    def backward(ctx, grad_out):
        out = tuple(None if g is None else g * grad_out for g in ctx.grads)
        return (None, None, None, None, None) + out


def _draw_seed(generator: Optional[torch.Generator]) -> int:
    """One 64-bit draw from a CPU generator (torch's default one if None): torch.manual_seed reproduces it."""
    v = torch.randint(-(1 << 63), (1 << 63) - 1, (), dtype=torch.int64, generator=generator)
    return int(v) & 0xFFFF_FFFF_FFFF_FFFF


class _Container(nn.Module):
    def forward(self, *a, **k):  # pragma: no cover - containers hold parameters only
        raise RuntimeError("parameter container: arithmetic lives in the CUDA kernels")


def _trunc_normal_(t: torch.Tensor, std=0.02, lo=-0.04, hi=0.04):
    # inverse-CDF truncated normal (the initialisation family of model/lru.py:16-36)
    a = (1.0 + math.erf((lo / std) / math.sqrt(2.0))) / 2.0
    b = (1.0 + math.erf((hi / std) / math.sqrt(2.0))) / 2.0
    with torch.no_grad():
        u = torch.empty_like(t, dtype=torch.float32).uniform_(2 * a - 1, 2 * b - 1)
        t.copy_(torch.erfinv(u) * (std * math.sqrt(2.0)))
    return t


class LRURec(nn.Module):
    def __init__(self, args):
        super().__init__()
        self.args = args
        d = int(getattr(args, "bert_hidden_units", 64))
        if d != 64:
            raise ValueError("llamarec_b200 kernels are specialised for bert_hidden_units == 64")
        n_blocks = int(getattr(args, "bert_num_blocks", 2) or 2)
        vocab = int(args.num_items) + 1
        self.num_items = int(args.num_items)
        # train-mode dropout rates of model/lru.py:47-52,93-97 (used by ce_loss(..., dropout=True) only)
        self.bert_dropout = float(getattr(args, "bert_dropout", 0.0) or 0.0)
        self.bert_attn_dropout = float(getattr(args, "bert_attn_dropout", 0.0) or 0.0)

        self.embedding = _Container()
        self.embedding.token = nn.Embedding(vocab, d)
        self.embedding.layer_norm = nn.LayerNorm(d)
        self.model = _Container()
        blocks = []
        for _ in range(n_blocks):
            blk = _Container()
            blk.lru_layer = _Container()
            u1, u2 = torch.rand(2 * d), torch.rand(2 * d)
            r_min, r_max = 0.8, 0.99
            nu_log = torch.log(-0.5 * torch.log(u1 * (r_max ** 2 - r_min ** 2) + r_min ** 2))
            theta_log = torch.log(u2 * (2 * math.pi))
            gamma_log = torch.log(torch.sqrt(1 - torch.exp(-torch.exp(nu_log)) ** 2))
            blk.lru_layer.params_log = nn.Parameter(torch.vstack((nu_log, theta_log, gamma_log)))
            with warnings.catch_warnings():   # torch warns that complex nn.Modules are experimental
                warnings.simplefilter("ignore")
                blk.lru_layer.in_proj = nn.Linear(d, 2 * d).to(torch.cfloat)
                blk.lru_layer.out_proj = nn.Linear(2 * d, d).to(torch.cfloat)
            blk.lru_layer.layer_norm = nn.LayerNorm(d)
            blk.feed_forward = _Container()
            blk.feed_forward.w_1 = nn.Linear(d, 4 * d)
            blk.feed_forward.w_2 = nn.Linear(4 * d, d)
            blk.feed_forward.layer_norm = nn.LayerNorm(d)
            blocks.append(blk)
        self.model.lru_blocks = nn.ModuleList(blocks)
        self.model.bias = nn.Parameter(torch.zeros(vocab))
        for name, p in self.named_parameters():
            if "layer_norm" in name or "params_log" in name:     # model/lru.py:21 -- model.bias IS initialised
                continue
            if torch.is_complex(p):
                with torch.no_grad():
                    re, im = torch.empty(p.shape), torch.empty(p.shape)
                    _trunc_normal_(re), _trunc_normal_(im)
                    p.copy_(torch.complex(re, im))
            else:
                _trunc_normal_(p.data)
        self._prepared_sig = None
        self._cache: Dict[str, torch.Tensor] = {}
        self._ws: Dict[tuple, torch.Tensor] = {}
        # optional list; when set, retrieve() appends (start, end) CUDA events around the scoring launch
        self.profile_events = None
        # row shard of the item table owned by this instance: [row_begin, row_end)
        self.row_begin, self.row_end = 0, vocab

    # ------------------------------------------------------------------ reference-compatible API
    @classmethod
    def from_reference(cls, ref_model) -> "LRURec":
        m = cls(ref_model.args)
        m.load_state_dict(ref_model.state_dict())
        return m

    @_on_model_device
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """model/lru.py:38-41 -- scores at every position, [B, L, N+1] fp32 (exact fp32 scoring).  Eval semantics in
        either mode: no dropout (only ce_loss(..., dropout=True) applies it)."""
        hidden = self.hidden_states(x)
        B, L, _ = hidden.shape
        rows = self.row_end - self.row_begin
        c = self._prepare()
        out = torch.empty(B, L, rows, dtype=torch.float32, device=hidden.device)
        lib = _lib.load()
        _lib.check(lib.lrb_score_dense(_lib.ptr(hidden), _lib.ptr(c["table_f32_shard"]), _lib.ptr(c["bias_pad"]),
                                       None, B * L, rows, 1, _lib.ptr(out), rows, _lib.stream_handle()))
        return out

    # ------------------------------------------------------------------ fast entry points
    def set_row_shard(self, row_begin: int, row_end: int) -> None:
        """Restrict scoring to item rows [row_begin, row_end) (row-sharded multi-GPU retrieval)."""
        self.row_begin, self.row_end = int(row_begin), int(row_end)
        self._prepared_sig = None

    @_on_model_device
    def hidden_states(self, x: torch.Tensor) -> torch.Tensor:
        """Encoder output at every position, [B, L, 64] (model/lru.py:73-83).  Eval semantics in either mode: no
        dropout."""
        return self._encode(x, all_positions=True)[0]

    @_on_model_device
    def encode(self, x: torch.Tensor, want_bf16: bool = False):
        """Last-position user state u[B, 64] fp32 (and optionally its bf16 copy)."""
        u, u16, _ = self._encode(x, all_positions=False, want_bf16=want_bf16)
        return (u, u16) if want_bf16 else u

    @_on_model_device
    @torch.no_grad()
    def retrieve(self, x: torch.Tensor, k: int = 20, exclude_history: bool = True,
                 labels: Optional[torch.Tensor] = None, ks: Optional[Sequence[int]] = None,
                 precision: str = "auto", u: Optional[torch.Tensor] = None,
                 u_bf16: Optional[torch.Tensor] = None, merge: bool = True,
                 packed_out: Optional[torch.Tensor] = None, seq: Optional[dict] = None,
                 scatter: Optional[dict] = None, packed_layout: str = "planes") -> Dict[str, torch.Tensor]:
        """encode -> catalogue score -> (history mask) -> top-k -> (metrics), all on device.  Eval semantics in either
        mode: no dropout.

        Replaces calculate_metrics / the per-user loop of generate_candidates (trainer/lru.py:30-42,
        61-88).  Returns ids/scores [B, k] sorted by (score desc, id asc); with `labels` also
        `label_rank` [B] (0-based, -1 = not in the top k) and `metric_sums` [len(ks), 3] holding the
        per-batch sums of Recall/MRR/NDCG@ks (divide by the user count of your choice: per batch for
        BaseTrainer.validate/test, num_users for generate_candidates -- SURVEY section 8a).
        With merge=False the per-split partial lists are returned instead (used by the sharded path).
        `seq` (optional) is a prepared descriptor holding `excl_sorted`/`excl_bloom`/`excl_stride` for the
        rows of `u`; with it `x` may be None -- the sharded path scores user states and exclusion lists
        that were encoded on other ranks.  `scatter` ({"dst_scores": [...], "dst_ids": [...], "users_per_dst": n,
        "out_stride": s} of raw device/peer addresses) makes the merge write every user's list straight into
        the buffer of the rank that owns the user (lrb_merge_metrics_scatter).
        """
        lib = _lib.load()
        c = self._prepare()
        dev = c["table_f32"].device
        rows = self.row_end - self.row_begin
        prec = self._precision(precision, rows)
        if x is None:
            if seq is None or (u is None and u_bf16 is None):
                raise ValueError("retrieve(x=None) needs the user states (u / u_bf16) and a prepared `seq`")
            B = (u if u is not None else u_bf16).shape[0]
        else:
            x = x.to(dev).contiguous()
            B = x.shape[0]
            if seq is None:
                seq = self._prepare_sequences(x, all_positions=False, want_excl=exclude_history)
        if u is None and u_bf16 is not None and prec == 0:
            pass                                    # bf16 states supplied by the caller
        elif u is None:
            u, u_bf16, _ = self._encode(x, all_positions=False, want_bf16=(prec == 0), seq=seq)
        elif prec == 0 and u_bf16 is None:
            u_bf16 = u.to(torch.bfloat16).contiguous()
        slots = _lib.c_int(0)
        _lib.check(lib.lrb_score_topk_slots(B, rows, prec, _lib.ctypes.byref(slots)))
        S = slots.value
        part_s = self._buf(("part_s", B, S, k), (B, S, k), torch.float32, dev)
        part_i = self._buf(("part_i", B, S, k), (B, S, k), torch.int32, dev)
        part_c = self._buf(("part_c", B, S), (B, S), torch.int32, dev)
        scratch = self._buf(("scratch", B), (lib.lrb_score_scratch_bytes(B),), torch.uint8, dev)
        if prec == 1:
            uu, table, bias_blk = u, c["table_f32_shard"], None
        else:
            uu, table, bias_blk = u_bf16, c["table_bf16"], c["bias_blk"]
        if self.profile_events is not None:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
        _lib.check(lib.lrb_score_topk(
            _lib.ptr(uu), _lib.ptr(table), _lib.ptr(c["bias_pad"]), _lib.ptr(bias_blk), B, rows, self.row_begin,
            _lib.ptr(seq["excl_sorted"]) if exclude_history else None,
            _lib.ptr(seq["excl_bloom"]) if exclude_history else None,
            seq["excl_stride"], k, prec, _lib.ptr(part_s), _lib.ptr(part_i), _lib.ptr(part_c), S,
            _lib.ptr(scratch), _lib.stream_handle()))
        if self.profile_events is not None:
            ev1.record()
            self.profile_events.append((ev0, ev1))
        if not merge:
            return {"part_scores": part_s, "part_ids": part_i, "part_cnt": part_c, "u": u}
        out = merge_lists(part_s, part_i, part_c, k_out=k, labels=labels, ks=ks, packed_out=packed_out,
                          scatter=scatter, packed_layout=packed_layout)
        out["u"] = u
        return out

    def ce_loss(self, x: torch.Tensor, labels: torch.Tensor, ignore_index: int = 0,
                return_row_loss: bool = False, dropout: bool = False,
                generator: Optional[torch.Generator] = None):
        """The train-step loss, `CrossEntropyLoss(ignore_index=0)(model(x).view(-1, N+1), labels.view(-1))`
        (trainer/lru.py:20-28), without the [B*L, N+1] logits.  With autograd enabled (and no per-row losses asked
        for) the result carries a backward: `loss.backward()` fills `.grad` of every parameter from ONE fused
        forward + backward pass (lrb_train_step), like trainer/base.py:107-111 does through torch's autograd.
        Under torch.no_grad() it is the forward value only (lrb_ce_loss_fwd).

        Dropout is active when `dropout and self.training` (like nn.Dropout): the reference's four train-mode sites
        (model/lru.py:57-60,160,174-175) at rates bert_dropout (embedding, PFFN) and bert_attn_dropout (after
        out_proj).  The masks are counter-based (include/llamarec_b200.h, lrb_train_step_dropout) and keyed by one
        64-bit draw per call from `generator`, a CPU torch.Generator (torch's default one if None), so
        torch.manual_seed reproduces a run; they are not torch's own dropout masks.  Active dropout needs the
        backward path: under torch.no_grad() or with return_row_loss it raises ValueError.  In eval mode, or with
        dropout=False, nothing changes."""
        rates = None
        if dropout and self.training:
            rates = (self.bert_dropout, self.bert_attn_dropout, self.bert_dropout)
            if not all(0.0 <= p < 1.0 for p in rates):     # False for NaN as well
                raise ValueError(f"dropout rates must satisfy 0 <= p < 1, got bert_dropout={self.bert_dropout}, "
                                 f"bert_attn_dropout={self.bert_attn_dropout}")
            if return_row_loss or not torch.is_grad_enabled():
                raise ValueError("dropout=True in training mode runs the fused train step: it has no per-row losses "
                                 "and no value-only path (call it with autograd enabled, or use model.eval())")
        return self._ce_loss(x, labels, ignore_index, return_row_loss, rates, generator)

    @_on_model_device
    def _ce_loss(self, x, labels, ignore_index, return_row_loss, rates, generator):
        if rates is not None:
            drop = (float(rates[0]), float(rates[1]), float(rates[2]), _draw_seed(generator))
            return _TrainStep.apply(self, x, labels, int(ignore_index), drop, *[p for _, p in self.named_parameters()])
        if torch.is_grad_enabled() and not return_row_loss and any(p.requires_grad for p in self.parameters()):
            return _TrainStep.apply(self, x, labels, int(ignore_index), None, *[p for _, p in self.named_parameters()])
        with torch.no_grad():
            return self._ce_loss_value(x, labels, ignore_index, return_row_loss)

    def _ce_loss_value(self, x, labels, ignore_index, return_row_loss):
        lib = _lib.load()
        if self.row_begin != 0 or self.row_end != self.num_items + 1:
            raise RuntimeError("ce_loss needs the whole item table on this device (no row shard)")
        hidden = self.hidden_states(x)                              # [B, L, 64]
        c = self._prepare()
        dev = hidden.device
        B, L, _ = hidden.shape
        M, rows = B * L, self.num_items + 1
        labels = labels.to(dev).reshape(-1).to(torch.int64).contiguous()
        if labels.numel() != M:
            raise ValueError(f"labels has {labels.numel()} entries, expected B*L = {M}")
        ws_bytes = lib.lrb_ce_workspace_bytes(M, rows)
        ws = self._buf(("ce_ws", M, rows), (ws_bytes,), torch.uint8, dev)
        row_loss = torch.empty(M, dtype=torch.float32, device=dev) if return_row_loss else None
        acc = torch.zeros(2, dtype=torch.float32, device=dev)
        _lib.check(lib.lrb_ce_loss_fwd(_lib.ptr(hidden), _lib.ptr(c["table_f32"]), _lib.ptr(c["bias_pad"]), M, rows,
                                       _lib.ptr(labels), int(ignore_index), _lib.ptr(row_loss), _lib.ptr(acc),
                                       _lib.ptr(ws), ws_bytes, _lib.stream_handle()))
        loss = acc[0] / acc[1]                                       # nan when every label is ignored, like torch
        return (loss, row_loss.view(B, L)) if return_row_loss else loss

    @torch.no_grad()
    def _train_step(self, x: torch.Tensor, labels: torch.Tensor, ignore_index: int = 0, dropout=None):
        """-> (loss, [gradient per parameter in named_parameters() order]) from one lrb_train_step call, or one
        lrb_train_step_dropout call when `dropout` = (p_embed, p_attn, p_ffn, seed) is given."""
        lib = _lib.load()
        if self.row_begin != 0 or self.row_end != self.num_items + 1:
            raise RuntimeError("the train step needs the whole item table on this device (no row shard)")
        c = self._prepare()
        dev = c["table_f32"].device
        x = x.to(dev).contiguous()
        if x.dtype not in (torch.int64, torch.int32):
            x = x.to(torch.int64)
        B, L = x.shape
        rows = self.num_items + 1
        labels = labels.to(dev).reshape(-1).to(torch.int64).contiguous()
        if labels.numel() != B * L:
            raise ValueError(f"labels has {labels.numel()} entries, expected B*L = {B * L}")
        n_blocks = c["n_blocks"]
        params_log = torch.stack([blk.lru_layer.params_log.detach().float() for blk in self.model.lru_blocks]).contiguous()
        bias = self.model.bias.detach().float().contiguous()
        ws_bytes = lib.lrb_train_workspace_bytes(B, L, n_blocks)
        ws = self._buf(("train_ws", B, L), (ws_bytes,), torch.uint8, dev)
        g_w = torch.empty(c["blob"].numel(), dtype=torch.float32, device=dev)
        g_table = torch.empty(rows, 64, dtype=torch.float32, device=dev)
        g_bias = torch.empty(rows, dtype=torch.float32, device=dev)
        acc = torch.empty(2, dtype=torch.float32, device=dev)
        step_args = (_lib.ptr(x), x.element_size(), _lib.ptr(labels), B, L, _lib.ptr(c["table_f32"]), rows,
                     _lib.ptr(bias), _lib.ptr(c["blob"]), _lib.ptr(params_log), n_blocks, int(ignore_index),
                     _lib.ptr(acc), _lib.ptr(g_w), _lib.ptr(g_table), _lib.ptr(g_bias), _lib.ptr(ws), ws_bytes,
                     _lib.stream_handle())
        if dropout is None:
            _lib.check(lib.lrb_train_step(*step_args))
        else:
            _lib.check(lib.lrb_train_step_dropout(*step_args, *dropout))
        loss = acc[0] / acc[1]
        named = unpack_encoder_grads(g_w, n_blocks)
        named["embedding.token.weight"] = g_table
        named["model.bias"] = g_bias
        grads = []
        for name, p in self.named_parameters():
            g = named.get(name)
            if g is None or not p.requires_grad:
                grads.append(None)
            else:
                grads.append(g.to(p.dtype).reshape(p.shape))
        return loss, grads

    # ------------------------------------------------------------------ internals
    @staticmethod
    def _precision(precision: str, rows: int) -> int:
        if precision == "auto":
            return 1 if rows <= SMALL_CATALOGUE_ROWS else 0
        if precision in ("fp32", "f32", 1):
            return 1
        if precision in ("bf16", 0):
            return 0
        raise ValueError(f"unknown precision {precision!r}")

    def _buf(self, key, shape, dtype, dev) -> torch.Tensor:
        t = self._ws.get(key)
        if t is None or t.device != dev:
            t = torch.empty(shape, dtype=dtype, device=dev)
            self._ws[key] = t
        return t

    def _signature(self):
        return tuple((p.data_ptr(), p._version, str(p.device)) for p in self.parameters()) + \
            (self.row_begin, self.row_end)

    def _prepare(self) -> Dict[str, torch.Tensor]:
        """(Re)builds the device-side layouts when parameters changed: packed encoder blob, fp32
        table, bf16 shard copy, padded bias and folded-bias block."""
        sig = self._signature()
        if sig == self._prepared_sig:
            return self._cache
        table = self.embedding.token.weight
        if not table.is_cuda:
            raise RuntimeError("llamarec_b200 has no CPU path: move the model to a CUDA device (model.cuda())")
        lib = _lib.load()
        dev = table.device
        sd = {k: v.detach() for k, v in self.state_dict().items()}
        blob = pack_encoder_weights(sd).to(dev)
        table_f32 = table.detach().to(torch.float32).contiguous()
        bias = self.model.bias.detach().to(torch.float32).contiguous()
        rows = self.row_end - self.row_begin
        rows_pad = (rows + 255) // 256 * 256
        table_bf16 = torch.empty(rows, 64, dtype=torch.bfloat16, device=dev)
        bias_pad = torch.empty(rows_pad, dtype=torch.float32, device=dev)
        has_bias = bool((bias[self.row_begin:self.row_end] != 0).any().item())
        bias_blk = torch.empty(lib.lrb_bias_blk_bytes(rows), dtype=torch.uint8, device=dev) if has_bias else None
        _lib.check(lib.lrb_prepare_table(_lib.ptr(table_f32), _lib.ptr(bias), self.row_begin, rows,
                                         _lib.ptr(table_bf16), _lib.ptr(bias_pad), _lib.ptr(bias_blk),
                                         _lib.stream_handle()))
        self._cache = {
            "blob": blob, "table_f32": table_f32, "table_bf16": table_bf16, "bias_pad": bias_pad,
            "bias_blk": bias_blk, "table_f32_shard": table_f32[self.row_begin:self.row_end],
            "n_blocks": len(self.model.lru_blocks),
        }
        self._prepared_sig = sig
        return self._cache

    def _prepare_sequences(self, x: torch.Tensor, all_positions: bool, want_excl: bool):
        lib = _lib.load()
        B, L = x.shape
        dev = x.device
        if x.dtype not in (torch.int64, torch.int32):     # both widths are consumed natively by the kernels
            x = x.to(torch.int64)
        stride = lib.lrb_excl_stride(L)
        tok_first = self._buf(("tok_first", B), (B,), torch.int32, dev)
        tok_offset = self._buf(("tok_offset", B), (B + 1,), torch.int32, dev)
        excl_sorted = self._buf(("excl_sorted", B, stride), (B, stride), torch.int32, dev) if want_excl else None
        excl_bloom = self._buf(("excl_bloom", B), (B, 4), torch.int32, dev) if want_excl else None
        _lib.check(lib.lrb_prepare_sequences(_lib.ptr(x), x.element_size(), B, L, 1 if all_positions else 0,
                                             _lib.ptr(tok_first),
                                             _lib.ptr(tok_offset), _lib.ptr(excl_sorted), _lib.ptr(excl_bloom),
                                             _lib.stream_handle()))
        return {"ids": x, "tok_first": tok_first, "tok_offset": tok_offset, "excl_sorted": excl_sorted,
                "excl_bloom": excl_bloom, "excl_stride": stride}

    @torch.no_grad()
    def _encode(self, x: torch.Tensor, all_positions: bool, want_bf16: bool = False, seq=None):
        lib = _lib.load()
        c = self._prepare()
        dev = c["table_f32"].device
        x = x.to(dev).contiguous()
        B, L = x.shape
        if seq is None:
            seq = self._prepare_sequences(x, all_positions=all_positions, want_excl=False)
        elif all_positions:
            raise ValueError("a prepared eval-mode sequence descriptor cannot be reused for all positions")
        ws_bytes = lib.lrb_encode_workspace_bytes(B, L, 1 if all_positions else 0)
        ws = self._buf(("enc_ws", B, L), (ws_bytes,), torch.uint8, dev)
        if all_positions:
            out = torch.empty(B, L, 64, dtype=torch.float32, device=dev)
            out16 = None
        else:
            out = torch.empty(B, 64, dtype=torch.float32, device=dev)
            out16 = torch.empty(B, 64, dtype=torch.bfloat16, device=dev) if want_bf16 else None
        _lib.check(lib.lrb_encode_fwd(_lib.ptr(seq["ids"]), seq["ids"].element_size(), B, L, _lib.ptr(c["table_f32"]),
                                      c["table_f32"].shape[0],
                                      _lib.ptr(c["blob"]), c["n_blocks"], 1 if all_positions else 0,
                                      _lib.ptr(seq["tok_first"]), _lib.ptr(seq["tok_offset"]), _lib.ptr(out),
                                      _lib.ptr(out16), _lib.ptr(ws), ws_bytes, _lib.stream_handle()))
        return out, out16, seq


def merge_lists(list_scores: torch.Tensor, list_ids: torch.Tensor, list_cnt: Optional[torch.Tensor], k_out: int,
                labels: Optional[torch.Tensor] = None, ks: Optional[Sequence[int]] = None,
                layout: str = "user_major", packed_out: Optional[torch.Tensor] = None,
                strides: Optional[tuple] = None, scatter: Optional[dict] = None,
                packed_layout: str = "planes") -> Dict[str, torch.Tensor]:
    """Fused k-way merge + metrics (lrb_merge_metrics).

    layout 'user_major': lists are [B, S, K] (output of lrb_score_topk);
    layout 'list_major': lists are [R, B, K] (all-gathered per-rank results).
    packed_out (optional int32 output buffer) is laid out as `packed_layout` says -- never guessed from its
    shape: 'planes' = [2, B, k_out] (all scores, then all ids: one all-gather payload), 'per_user' =
    [B, 2, k_out] (per user scores then ids: rows of an all-to-all payload split by user range).
    """
    with _lib.on_device(list_scores):
        return _merge_lists(list_scores, list_ids, list_cnt, k_out, labels, ks, layout, packed_out, strides, scatter,
                            packed_layout)


def _merge_lists(list_scores, list_ids, list_cnt, k_out, labels, ks, layout, packed_out, strides, scatter,
                 packed_layout):
    lib = _lib.load()
    dev = list_scores.device
    if layout == "user_major":
        B, S, K = list_scores.shape
        stride_list, stride_user = K, S * K
        cnt_sl, cnt_su = 1, S
    else:
        S, B, K = list_scores.shape
        stride_list, stride_user = B * K, K
        cnt_sl, cnt_su = B, 1
    if strides is not None:          # explicit element strides (views into a packed gather buffer)
        stride_list, stride_user = strides
    else:
        list_scores, list_ids = list_scores.contiguous(), list_ids.contiguous()
    if scatter is not None:
        # all-to-all fused into the merge: rows go to the owner rank's recv buffer (peer-mapped addresses)
        n_dst = len(scatter["dst_scores"])
        arr_s = (_lib.ctypes.c_void_p * n_dst)(*scatter["dst_scores"])
        arr_i = (_lib.ctypes.c_void_p * n_dst)(*scatter["dst_ids"])
        _lib.check(lib.lrb_merge_metrics_scatter(
            list_scores.data_ptr(), list_ids.data_ptr(),
            _lib.ptr(list_cnt.contiguous()) if list_cnt is not None else None, S, stride_list, stride_user, cnt_sl,
            cnt_su, K, B, k_out, arr_s, arr_i, n_dst, int(scatter["users_per_dst"]), int(scatter["out_stride"]),
            _lib.stream_handle()))
        return {}
    ks = list(ks) if ks is not None else []
    out_stride = 0
    if packed_out is not None and packed_layout not in ("planes", "per_user"):
        raise ValueError(f"unknown packed_layout {packed_layout!r}")
    if packed_out is not None and (packed_out.dtype != torch.int32 or not packed_out.is_contiguous()):
        raise ValueError("packed_out must be a contiguous int32 tensor")
    if packed_out is not None and packed_layout == "planes":
        # [2, B, k_out] int32: scores (bit pattern) then ids, one gather payload
        if tuple(packed_out.shape) != (2, B, k_out):
            raise ValueError(f"packed_out is {tuple(packed_out.shape)}, layout 'planes' needs {(2, B, k_out)}")
        top_s = packed_out[0].view(torch.float32)
        top_i = packed_out[1]
    elif packed_out is not None:
        # [B, 2, k_out] int32: per user scores then ids (rows of an all-to-all payload split by user range)
        if tuple(packed_out.shape) != (B, 2, k_out):
            raise ValueError(f"packed_out is {tuple(packed_out.shape)}, layout 'per_user' needs {(B, 2, k_out)}")
        top_s = packed_out.view(torch.float32)[:, 0]
        top_i = packed_out[:, 1]
        out_stride = 2 * k_out
    else:
        top_s = torch.empty(B, k_out, dtype=torch.float32, device=dev)
        top_i = torch.empty(B, k_out, dtype=torch.int32, device=dev)
    rank = torch.empty(B, dtype=torch.int32, device=dev) if labels is not None else None
    sums = torch.zeros(max(len(ks), 1) * 3, dtype=torch.float32, device=dev) if labels is not None else None
    if labels is not None:
        labels = labels.to(dev).reshape(-1).to(torch.int64).contiguous()
    ks_arr = (_lib.ctypes.c_int32 * max(len(ks), 1))(*ks) if ks else None
    _lib.check(lib.lrb_merge_metrics(
        list_scores.data_ptr(), list_ids.data_ptr(),
        _lib.ptr(list_cnt.contiguous()) if list_cnt is not None else None, S, stride_list, stride_user, cnt_sl,
        cnt_su, K, B, k_out, _lib.ptr(labels), ks_arr, len(ks), top_s.data_ptr(), top_i.data_ptr(), out_stride,
        _lib.ptr(rank), _lib.ptr(sums), _lib.stream_handle()))
    out = {"scores": top_s, "ids": top_i}
    if labels is not None:
        out["label_rank"] = rank
        out["metric_sums"] = sums[: 3 * len(ks)].reshape(len(ks), 3) if ks else sums[:0].reshape(0, 3)
    return out
