"""CPU oracle for the stage-1 hot path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A plain torch-CPU fp32 restatement of the reference's algorithm for LRURec encode -> catalogue
score -> history mask -> top-k.  Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline
legs may import this package; the product path (llamarec_b200/) never does and has no CPU
fallback.

Parity status: PINNED.  The reference has no tests or golden vectors of its own (SURVEY.md
section 4), so the pin is the reference code itself, executed in the build container by
oracle/make_golden.py; its outputs are committed under tests/golden/ and
tests/test_oracle_golden.py checks every function here against them.

Every function cites the reference lines it restates (paths relative to the reference tree).
State dicts use the reference's parameter names (SURVEY.md section 3.2).
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

LN_EPS = 1e-5  # nn.LayerNorm default used by every LayerNorm in model/lru.py


def _ln(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    return F.layer_norm(x, (x.shape[-1],), w, b, LN_EPS)


def complex_of(dtype: torch.dtype) -> torch.dtype:
    """The complex dtype whose parts are `dtype`: complex64 for float32 (the reference), complex128 for float64."""
    return torch.complex128 if dtype == torch.float64 else torch.complex64


def cast_state_dict(sd: Dict[str, torch.Tensor], dtype: Optional[torch.dtype]) -> Dict[str, torch.Tensor]:
    """Real tensors to `dtype`, complex ones to complex_of(dtype); None keeps `sd` as it is.  Differentiable."""
    if dtype is None:
        return sd
    return {k: v.to(complex_of(dtype) if v.is_complex() else dtype) for k, v in sd.items()}


def n_blocks_of(sd: Dict[str, torch.Tensor]) -> int:
    n = 0
    while f"model.lru_blocks.{n}.lru_layer.params_log" in sd:
        n += 1
    return n


def embed(ids: torch.Tensor, sd: Dict[str, torch.Tensor]) -> Tuple[torch.Tensor, torch.Tensor]:
    """model/lru.py:54-60 -- mask = ids > 0; LayerNorm(Embedding[ids]); dropout is identity in eval.

    Row 0 of the table is an ordinary trained row (no padding_idx)."""
    mask = ids > 0
    x = sd["embedding.token.weight"][ids]
    return _ln(x, sd["embedding.layer_norm.weight"], sd["embedding.layer_norm.bias"]), mask


def lru_constants(params_log: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """model/lru.py:151-152 -- lambda = exp(-exp(nu_log) + i exp(theta_log)), gamma = exp(gamma_log)."""
    nu, theta, gamma = torch.exp(params_log).split((1, 1, 1))
    lam = torch.exp(torch.complex(-nu, theta))
    return lam, gamma


def tree_scan(bu: torch.Tensor, lam: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
    """model/lru.py:135-147,155-159 -- the recursive-doubling scan.

    bu [B, Lp, H] complex with Lp a power of two, lam [1, H] of the same dtype, mask [B, Lp] bool.
    Level i works on aligned blocks of 2^i: every element j (0-based) of the second half receives
    lambda^(j+1) * (last element of the first half) * mask(last element of the first half).
    The power table doubles each level exactly as the reference builds it (table ++ table*last).
    """
    B, Lp, H = bu.shape
    levels = int(round(math.log2(Lp)))
    assert 1 << levels == Lp
    h = bu.clone()
    powers = lam.reshape(1, H)  # lambda^1
    for i in range(1, levels + 1):
        blk, half = 1 << i, 1 << (i - 1)
        if i > 1:
            powers = torch.cat((powers, powers * powers[-1]), 0)  # lambda^(1..half)
        hv = h.view(B, Lp // blk, blk, H)
        mv = mask.view(B, Lp // blk, blk)
        carry = hv[:, :, half - 1, :] * mv[:, :, half - 1].unsqueeze(-1)       # [B, nb, H]
        upd = hv[:, :, half:, :] + powers.view(1, 1, half, H) * carry.unsqueeze(2)
        h = torch.cat((hv[:, :, :half, :], upd), dim=2).reshape(B, Lp, H)
    return h


def lru_layer(x: torch.Tensor, mask: torch.Tensor, sd: Dict[str, torch.Tensor], blk: int) -> torch.Tensor:
    """model/lru.py:149-161 -- in_proj (complex) * gamma, tree scan, Re(out_proj) + residual, LayerNorm."""
    p = f"model.lru_blocks.{blk}.lru_layer."
    lam, gamma = lru_constants(sd[p + "params_log"])
    bu = F.linear(x.to(complex_of(x.dtype)), sd[p + "in_proj.weight"], sd[p + "in_proj.bias"]) * gamma
    h = tree_scan(bu, lam, mask)
    y = F.linear(h, sd[p + "out_proj.weight"], sd[p + "out_proj.bias"]).real + x
    return _ln(y, sd[p + "layer_norm.weight"], sd[p + "layer_norm.bias"])


def pffn(x: torch.Tensor, sd: Dict[str, torch.Tensor], blk: int) -> torch.Tensor:
    """model/lru.py:164-175 -- LayerNorm(W2 gelu_erf(W1 x + b1) + b2 + x)."""
    p = f"model.lru_blocks.{blk}.feed_forward."
    z = F.gelu(F.linear(x, sd[p + "w_1.weight"], sd[p + "w_1.bias"]))
    z = F.linear(z, sd[p + "w_2.weight"], sd[p + "w_2.bias"])
    return _ln(z + x, sd[p + "layer_norm.weight"], sd[p + "layer_norm.bias"])


def hidden_states(ids: torch.Tensor, sd: Dict[str, torch.Tensor],
                  dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    """model/lru.py:38-41,73-83 -- encoder output at every position, [B, L, 64] fp32.

    The sequence is left-padded with zero vectors / False mask to the next power of two before the
    blocks run and cut back afterwards.  `dtype` (e.g. torch.float64) runs the same arithmetic with
    `sd` cast to it (complex parts too); None computes in the dtypes of `sd`, the reference's fp32."""
    sd = cast_state_dict(sd, dtype)
    x, mask = embed(ids, sd)
    L = ids.shape[1]
    Lp = 1 << max(0, math.ceil(math.log2(L))) if L > 1 else 1
    Lp = max(Lp, 1)
    x = F.pad(x, (0, 0, Lp - L, 0))
    mask = F.pad(mask, (Lp - L, 0))
    for blk in range(n_blocks_of(sd)):
        x = lru_layer(x, mask, sd, blk)
        x = pffn(x, sd, blk)
    return x[:, Lp - L:, :]


def encode(ids: torch.Tensor, sd: Dict[str, torch.Tensor], dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    """User state = encoder output at the last position (trainer/lru.py:33 takes scores[:, -1])."""
    return hidden_states(ids, sd, dtype)[:, -1, :]


def forward_scores(ids: torch.Tensor, sd: Dict[str, torch.Tensor],
                   dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    """model/lru.py:85 -- scores at every position, [B, L, N+1] (tied embedding + bias)."""
    sd = cast_state_dict(sd, dtype)
    return torch.matmul(hidden_states(ids, sd), sd["embedding.token.weight"].t()) + sd["model.bias"]


def ce_loss(ids: torch.Tensor, labels: torch.Tensor, sd: Dict[str, torch.Tensor]) -> torch.Tensor:
    """trainer/lru.py:20-28 in eval mode: CrossEntropyLoss(ignore_index=0) on the logits at every position."""
    logits = forward_scores(ids, sd)
    return torch.nn.functional.cross_entropy(logits.view(-1, logits.size(-1)), labels.view(-1), ignore_index=0)


def last_scores(ids: torch.Tensor, sd: Dict[str, torch.Tensor]) -> torch.Tensor:
    """model(x)[:, -1, :] without materialising the other positions (bit-identical, SURVEY probe P4)."""
    return torch.matmul(encode(ids, sd), sd["embedding.token.weight"].t()) + sd["model.bias"]


def mask_history(scores: torch.Tensor, ids: torch.Tensor) -> torch.Tensor:
    """trainer/lru.py:36-38 -- every id of the input row (padding 0 included) gets -1e9."""
    out = scores.clone()
    out.scatter_(1, ids, -1e9)
    out[:, 0] = -1e9
    return out


def topk_sorted(scores: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """torch.topk of trainer/lru.py:82-84 with a *defined* tie rule: score desc, then id asc.

    (torch.topk / argsort tie order is implementation-defined, SURVEY probe P1.)"""
    n = scores.shape[1]
    order = torch.argsort(-scores.double() * 1.0, dim=1, stable=True)  # stable => lower id first on ties
    idx = order[:, : min(k, n)]
    return scores.gather(1, idx), idx


def retrieve(ids: torch.Tensor, sd: Dict[str, torch.Tensor], k: int, exclude_history: bool = True,
             u: Optional[torch.Tensor] = None, table: Optional[torch.Tensor] = None,
             bias: Optional[torch.Tensor] = None, chunk: int = 65536) -> Tuple[torch.Tensor, torch.Tensor]:
    """encode -> score -> (mask) -> top-k, chunked over item ranges so that large catalogues fit.

    `u`, `table`, `bias` override the fp32 operands (e.g. the bf16-rounded copies the tensor-core
    kernel consumes, SURVEY section 0 fact 5).  Scoring restates model/lru.py:85 per chunk with a
    running top-k; it is bit-identical to last_scores() + topk when one chunk covers the table."""
    if u is None:
        u = encode(ids, sd)
    if table is None:
        table = sd["embedding.token.weight"]
    if bias is None:
        bias = sd["model.bias"]
    B = u.shape[0]
    n_rows = table.shape[0]
    best_s = torch.empty(B, 0)
    best_i = torch.empty(B, 0, dtype=torch.int64)
    for lo in range(0, n_rows, chunk):
        hi = min(n_rows, lo + chunk)
        s = u.float() @ table[lo:hi].float().t() + bias[lo:hi]
        if exclude_history:
            inside = (ids >= lo) & (ids < hi)
            rows = torch.arange(B).unsqueeze(1).expand_as(ids)[inside]
            s[rows, ids[inside] - lo] = -1e9
            if lo == 0:
                s[:, 0] = -1e9
        cat_s = torch.cat((best_s, s), 1)
        cat_i = torch.cat((best_i, torch.arange(lo, hi).unsqueeze(0).expand(B, -1)), 1)
        # stable sort keeps earlier (lower) ids first among equal scores
        order = torch.argsort(-cat_s.double(), dim=1, stable=True)[:, :k]
        best_s, best_i = cat_s.gather(1, order), cat_i.gather(1, order)
    return best_s, best_i


def sequential_scan_reference(bu: torch.Tensor, lam: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
    """h_t = lambda * (mask_{t-1} h_{t-1}) + bu_t -- equals tree_scan for left-padded masks only
    (SURVEY probe P1); kept to document the equivalence the CUDA scan is tested for."""
    B, Lp, H = bu.shape
    h = torch.zeros_like(bu)
    prev = torch.zeros(B, H, dtype=bu.dtype)
    for t in range(Lp):
        gate = mask[:, t - 1].unsqueeze(-1) if t > 0 else torch.zeros(B, 1, dtype=torch.bool)
        prev = lam.reshape(1, H) * (prev * gate) + bu[:, t]
        h[:, t] = prev
    return h


def state_dict_to_numpy(sd: Dict[str, torch.Tensor]):
    return {k: v.detach().cpu().numpy() for k, v in sd.items()}


def state_dict_from_numpy(d) -> Dict[str, torch.Tensor]:
    return {k: torch.from_numpy(d[k]) for k in d.keys()}
