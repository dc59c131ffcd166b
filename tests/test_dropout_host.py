"""CPU: the dropout masks of the train step (numpy Philox restatement in oracle/dropout_oracle.py) and the train-mode
oracle, plus the argument checks of LRURec.ce_loss(..., dropout=True) that run before any device work."""
import math
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from conftest import GOLDEN, load_case
from llamarec_b200 import LRURec
from oracle import dropout_oracle as DO


def test_philox_known_answer_vectors():
    """Random123's known-answer vectors of Philox4x32-10."""
    cases = [
        ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
        ((0xFFFFFFFF,) * 4, (0xFFFFFFFF, 0xFFFFFFFF), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
        ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
         (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
    ]
    for ctr, key, want in cases:
        got = DO.philox4x32_10(np.array(ctr, dtype=np.uint32), key)
        assert tuple(int(v) for v in got) == want
    # vectorised over a batch of counters: each row equals the scalar call
    ctrs = np.array([c for c, _, _ in cases[:1]] * 3, dtype=np.uint32)
    assert (DO.philox4x32_10(ctrs, (0, 0)) == np.array(cases[0][2], dtype=np.uint32)).all()


B, L, W = 64, 64, 256          # 2^20 elements per mask


def _within_4_sigma(frac, q, n):
    return abs(frac - q) <= 4.0 * math.sqrt(q * (1.0 - q) / n)


@pytest.mark.parametrize("p", [0.1, 0.2, 0.5])
def test_keep_fraction_and_kept_value(p):
    m = DO.multipliers(0x0123456789ABCDEF, 2, B, L, W, p)
    assert m.shape == (B, L, W) and m.dtype == np.float32
    keep = m != 0
    assert _within_4_sigma(keep.mean(), 1.0 - p, keep.size), keep.mean()
    scale = np.float32(1.0) / (np.float32(1.0) - np.float32(p))
    assert (m[keep] == scale).all()


def test_rate_zero_keeps_everything():
    m = DO.multipliers(99, 0, 8, 50, 64, 0.0)
    assert (m == 1.0).all()
    assert DO.threshold(0.0) == 0


@pytest.mark.parametrize("p", [0.2, 0.5])
def test_masks_are_independent_across_sites_seeds_and_rows(p):
    """Two masks agree on an element with probability p^2 + (1-p)^2 if they are independent."""
    q = p * p + (1 - p) * (1 - p)
    a = DO.multipliers(7, 2, B, L, W, p) != 0
    for other in (DO.multipliers(7, 5, B, L, W, p) != 0,          # another site
                  DO.multipliers(8, 2, B, L, W, p) != 0,          # another seed (low word)
                  DO.multipliers(7 + (1 << 32), 2, B, L, W, p) != 0):   # another seed (high word)
        assert _within_4_sigma((a == other).mean(), q, a.size)
    flat = a.reshape(B * L, W)                                    # row t against row t + 1
    assert _within_4_sigma((flat[:-1] == flat[1:]).mean(), q, flat[:-1].size)
    feat = a.reshape(-1, 4)                                       # words of one Philox call against each other
    assert _within_4_sigma((feat[:, 0] == feat[:, 1]).mean(), q, feat.shape[0])


def test_oracle_without_dropout_reproduces_reference_autograd(golden_sd):
    """All multipliers 1: the train-mode restatement is the reference's eval-mode autograd (grad_case.npz, written by
    the reference itself) -- loss and all 30 gradients."""
    gcase = np.load(os.path.join(GOLDEN, "grad_case.npz"))
    for name in ("left_l20", "left_l50"):
        ids = torch.from_numpy(load_case(name)["ids"])
        labels = torch.from_numpy(gcase[f"{name}_labels"])
        ones = DO.site_multipliers(5, ids.shape[0], ids.shape[1], 2, 0.0, 0.0, 0.0)
        assert all(bool((m == 1).all()) for m in ones.values()) and len(ones) == 7
        loss, grads = DO.loss_and_grads(ids, labels, golden_sd, ones)
        assert abs(loss - float(gcase[f"{name}_loss"])) <= 1e-6
        assert len(grads) == 30
        for k, g in grads.items():
            want = gcase[f"{name}:{k}"]
            assert g.shape == want.shape and g.dtype == want.dtype, k
            np.testing.assert_allclose(g, want, rtol=1e-5, atol=1e-5 * float(np.abs(want).max()) + 1e-12, err_msg=k)


def test_oracle_dropout_changes_loss_and_zeroes_dropped_embedding_rows(golden_sd):
    ids = torch.from_numpy(load_case("left_l20")["ids"])
    labels = torch.from_numpy(np.load(os.path.join(GOLDEN, "grad_case.npz"))["left_l20_labels"])
    m = DO.site_multipliers(11, ids.shape[0], ids.shape[1], 2, 0.2, 0.3, 0.2)
    base = DO.ce_loss_train(ids, labels, golden_sd).item()
    assert DO.ce_loss_train(ids, labels, golden_sd, m).item() != base
    # the embedding site sits before the LayerNorm: with every row dropped the LayerNorm sees zeros (x_hat = 0), so its
    # weight gets no gradient while its bias still does
    only_embed = {0: torch.zeros(ids.shape[0], ids.shape[1], 64)}
    _, g0 = DO.loss_and_grads(ids, labels, golden_sd, only_embed)
    assert np.abs(g0["embedding.layer_norm.weight"]).max() == 0
    assert np.abs(g0["embedding.layer_norm.bias"]).max() > 0


def _args(p_embed=0.2, p_attn=0.3):
    return SimpleNamespace(num_items=50, bert_hidden_units=64, bert_num_blocks=2, bert_dropout=p_embed,
                           bert_attn_dropout=p_attn)


def test_rates_default_to_zero():
    m = LRURec(SimpleNamespace(num_items=50, bert_hidden_units=64, bert_num_blocks=2))
    assert m.bert_dropout == 0.0 and m.bert_attn_dropout == 0.0
    m = LRURec(_args())
    assert m.bert_dropout == pytest.approx(0.2) and m.bert_attn_dropout == pytest.approx(0.3)


def test_ce_loss_with_dropout_has_no_cpu_path():
    m = LRURec(_args()).train()
    ids = torch.tensor([[0, 3, 4, 5]])
    with pytest.raises(RuntimeError, match="no CPU path"):
        m.ce_loss(ids, ids, dropout=True)


@pytest.mark.parametrize("rates", [(1.0, 0.2), (0.2, 1.0), (-0.1, 0.2), (0.2, float("nan")), (1.5, 0.0)])
def test_ce_loss_rejects_rates_outside_unit_interval(rates):
    m = LRURec(_args(*rates)).train()
    ids = torch.tensor([[0, 3, 4, 5]])
    with pytest.raises(ValueError, match="0 <= p < 1"):
        m.ce_loss(ids, ids, dropout=True)
    m.eval()                                   # in eval mode dropout is off: the rates are not used
    with pytest.raises(RuntimeError, match="no CPU path"):
        m.ce_loss(ids, ids, dropout=True)


def test_ce_loss_dropout_needs_the_backward_path():
    m = LRURec(_args()).train()
    ids = torch.tensor([[0, 3, 4, 5]])
    with torch.no_grad(), pytest.raises(ValueError, match="no value-only path"):
        m.ce_loss(ids, ids, dropout=True)
    with pytest.raises(ValueError, match="no per-row losses"):
        m.ce_loss(ids, ids, dropout=True, return_row_loss=True)
