"""CPU oracle for the train step WITH dropout -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The reference applies dropout at four places in training (model/lru.py):

    site 0        LRUEmbedding.forward (:57-60)        layer_norm(embed_dropout(token(x)))     width 64,  bert_dropout
    site 1 + 3i   LRULayer.forward of block i (:160)   dropout(out_proj(h).real) + x           width 64,  bert_attn_dropout
    site 2 + 3i   PositionwiseFeedForward (:174)       dropout(gelu(w_1(x)))                   width 256, bert_dropout
    site 3 + 3i   PositionwiseFeedForward (:175)       layer_norm(dropout(w_2(x_)) + x)        width 64,  bert_dropout

torch's dropout RNG stream cannot be parity-matched, so the library draws counter-based masks instead
(include/llamarec_b200.h, lrb_train_step_dropout).  This module regenerates those masks bit for bit (a vectorised
numpy Philox4x32-10) and restates the reference's train-mode forward + CrossEntropyLoss(ignore_index) in
differentiable torch-CPU fp32 with the multipliers applied at the four sites; torch autograd of it gives the
gradients the fused train step is checked against.  With every multiplier 1 it is the reference's eval-mode
autograd (pinned by tests/golden/grad_case.npz).

Rows of the power-of-two padding the reference adds inside LRUModel.forward never reach the loss (the scan carry
is multiplied by mask 0 there); they get multiplier 1.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import numpy as np
import torch
import torch.nn.functional as F

from .lru_oracle import _ln, cast_state_dict, complex_of, lru_constants, n_blocks_of, tree_scan

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_MASK32 = np.uint64(0xFFFFFFFF)
_S32 = np.uint64(32)


def philox4x32_10(ctr: np.ndarray, key) -> np.ndarray:
    """Philox4x32-10 (Random123): ctr [..., 4] uint32, key (k0, k1) -> [..., 4] uint32.  The key is bumped by
    (W0, W1) before every round but the first."""
    c = np.asarray(ctr, dtype=np.uint32).astype(np.uint64)
    c0, c1, c2, c3 = c[..., 0], c[..., 1], c[..., 2], c[..., 3]
    k0, k1 = np.uint64(int(key[0]) & 0xFFFFFFFF), np.uint64(int(key[1]) & 0xFFFFFFFF)
    for r in range(10):
        if r:
            k0, k1 = (k0 + _W0) & _MASK32, (k1 + _W1) & _MASK32
        p0, p1 = _M0 * c0, _M1 * c2                       # < 2^64: exact in uint64
        c0, c1, c2, c3 = (p1 >> _S32) ^ c1 ^ k0, p1 & _MASK32, (p0 >> _S32) ^ c3 ^ k1, p0 & _MASK32
    return np.stack((c0, c1, c2, c3), axis=-1).astype(np.uint32)


def threshold(p: float) -> int:
    """floor(double(float(p)) * 2^32): an element is kept iff its Philox word is >= this."""
    return int(math.floor(float(np.float32(p)) * 4294967296.0))


def multipliers(seed: int, site: int, B: int, L: int, width: int, p: float) -> np.ndarray:
    """[B, L, width] float32 multipliers of one site: 1 / (1 - p) (fp32) where kept, 0 where dropped.
    Element (t, j), t = b*L + l, uses word j & 3 of Philox(counter = (t, j >> 2, site, 0), key = (seed lo, hi))."""
    seed = int(seed) & 0xFFFF_FFFF_FFFF_FFFF
    T, groups = B * L, (width + 3) // 4
    ctr = np.zeros((T, groups, 4), dtype=np.uint32)
    ctr[..., 0] = np.arange(T, dtype=np.uint32)[:, None]
    ctr[..., 1] = np.arange(groups, dtype=np.uint32)[None, :]
    ctr[..., 2] = site
    r = philox4x32_10(ctr, (seed & 0xFFFFFFFF, seed >> 32)).reshape(T, groups * 4)[:, :width]
    p32 = np.float32(p)
    scale = np.float32(1.0) / (np.float32(1.0) - p32)
    out = np.where(r >= np.uint64(threshold(p32)), scale, np.float32(0.0)).astype(np.float32)
    return out.reshape(B, L, width)


def site_multipliers(seed: int, B: int, L: int, n_blocks: int, p_embed: float, p_attn: float,
                     p_ffn: float) -> Dict[int, torch.Tensor]:
    """Multipliers of every site of an n_blocks model, {site: FloatTensor [B, L, width]}."""
    out = {0: torch.from_numpy(multipliers(seed, 0, B, L, 64, p_embed))}
    for i in range(n_blocks):
        out[1 + 3 * i] = torch.from_numpy(multipliers(seed, 1 + 3 * i, B, L, 64, p_attn))
        out[2 + 3 * i] = torch.from_numpy(multipliers(seed, 2 + 3 * i, B, L, 256, p_ffn))
        out[3 + 3 * i] = torch.from_numpy(multipliers(seed, 3 + 3 * i, B, L, 64, p_ffn))
    return out


def ce_loss_train(ids: torch.Tensor, labels: torch.Tensor, sd: Dict[str, torch.Tensor],
                  mults: Optional[Dict[int, torch.Tensor]] = None, ignore_index: int = 0,
                  dtype: Optional[torch.dtype] = None, reduction: str = "mean") -> torch.Tensor:
    """trainer/lru.py:20-28 in train mode: CrossEntropyLoss(ignore_index) on the logits at every position of the
    reference's forward (model/lru.py:38-41,57-60,73-86,149-161,164-175) with dropout multipliers `mults`
    ({site: [B, L, width]}, a missing site = multiplier 1).  Differentiable in every tensor of `sd`.
    `dtype` (e.g. torch.float64) computes with `sd` and the multipliers cast to it (complex parts too); None computes
    in the dtypes of `sd`.  `reduction` is cross_entropy's ('none': the row losses, 0 where ignored)."""
    mults = mults or {}
    sd = cast_state_dict(sd, dtype)
    B, L = ids.shape
    Lp = 1 << max(0, math.ceil(math.log2(L))) if L > 1 else 1

    def drop(v: torch.Tensor, site: int) -> torch.Tensor:
        m = mults.get(site)
        if m is None:
            return v
        m = m.to(v.dtype)
        if v.shape[1] != L:                                    # padded positions: multiplier 1
            m = torch.cat((torch.ones(B, v.shape[1] - L, m.shape[-1], dtype=v.dtype), m), 1)
        return v * m

    x = drop(sd["embedding.token.weight"][ids], 0)
    x = _ln(x, sd["embedding.layer_norm.weight"], sd["embedding.layer_norm.bias"])
    mask = F.pad(ids > 0, (Lp - L, 0))
    x = F.pad(x, (0, 0, Lp - L, 0))
    for i in range(n_blocks_of(sd)):
        p = f"model.lru_blocks.{i}.lru_layer."
        lam, gamma = lru_constants(sd[p + "params_log"])
        bu = F.linear(x.to(complex_of(x.dtype)), sd[p + "in_proj.weight"], sd[p + "in_proj.bias"]) * gamma
        h = tree_scan(bu, lam, mask)
        o = drop(F.linear(h, sd[p + "out_proj.weight"], sd[p + "out_proj.bias"]).real, 1 + 3 * i)
        x = _ln(o + x, sd[p + "layer_norm.weight"], sd[p + "layer_norm.bias"])
        q = f"model.lru_blocks.{i}.feed_forward."
        z = drop(F.gelu(F.linear(x, sd[q + "w_1.weight"], sd[q + "w_1.bias"])), 2 + 3 * i)
        z = drop(F.linear(z, sd[q + "w_2.weight"], sd[q + "w_2.bias"]), 3 + 3 * i)
        x = _ln(z + x, sd[q + "layer_norm.weight"], sd[q + "layer_norm.bias"])
    hidden = x[:, Lp - L:, :]
    logits = torch.matmul(hidden, sd["embedding.token.weight"].t()) + sd["model.bias"]
    return F.cross_entropy(logits.reshape(-1, logits.shape[-1]), labels.reshape(-1), ignore_index=ignore_index,
                           reduction=reduction)


def loss_and_grads(ids: torch.Tensor, labels: torch.Tensor, sd: Dict[str, torch.Tensor],
                   mults: Optional[Dict[int, torch.Tensor]] = None, ignore_index: int = 0,
                   dtype: Optional[torch.dtype] = None):
    """-> (loss, {parameter name: gradient as numpy}) of ce_loss_train by torch autograd.  With `dtype` the leaves
    are `sd` cast to it, so the gradients come out in that dtype (complex128 for the complex parameters of fp64)."""
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in cast_state_dict(sd, dtype).items()}
    loss = ce_loss_train(ids, labels, leaves, mults, ignore_index)
    loss.backward()
    return loss.item(), {k: v.grad.numpy() for k, v in leaves.items()}
