"""GPU (-m gpu): dropout in the fused train step (lrb_train_step_dropout / LRURec.ce_loss(..., dropout=True)) against
the train-mode oracle (oracle/dropout_oracle.py) under the same counter-based masks: mask bits, loss and all 30
gradients at the bar of the eval-mode gradient test (rtol 1e-3, atol 1e-3 of the largest entry)."""
import math
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from conftest import GOLDEN, load_case
from llamarec_b200 import LRURec, LRURetriever, _lib, synth
from llamarec_b200.model import _draw_seed
from oracle import dropout_oracle as DO

pytestmark = pytest.mark.gpu


def _args(n, p_embed, p_attn):
    return SimpleNamespace(num_items=n, bert_hidden_units=64, bert_num_blocks=2, bert_dropout=p_embed,
                           bert_attn_dropout=p_attn, metric_ks=[1, 5, 10, 20, 50], llm_negative_sample_size=19)


@pytest.fixture(scope="module")
def gcase():
    return np.load(os.path.join(GOLDEN, "grad_case.npz"))


def _model(golden_sd, p_embed=0.2, p_attn=0.3):
    m = LRURec(_args(400, p_embed, p_attn))
    m.load_state_dict(golden_sd)
    return m.cuda().train()


def _batch(gcase, name):
    return torch.from_numpy(load_case(name)["ids"]), torch.from_numpy(gcase[f"{name}_labels"])


def _grads(m):
    return {k: p.grad.detach().clone() for k, p in m.named_parameters()}


def _step(m, ids, labels, **kw):
    m.zero_grad(set_to_none=True)
    loss = m.ce_loss(ids.cuda(), labels.cuda(), **kw)
    loss.backward()
    return loss.item(), _grads(m)


def _device_keep(seed, site, T, width, p):
    keep = torch.empty(T, width, dtype=torch.uint8, device="cuda")
    _lib.check(_lib.load().lrb_dropout_mask(seed, site, T, width, p, keep.data_ptr(), _lib.stream_handle()))
    torch.cuda.synchronize()
    return keep.cpu().numpy().astype(bool)


@pytest.mark.parametrize("T", [203, 1000])
@pytest.mark.parametrize("seed", [0, 0x0123456789ABCDEF])
def test_mask_bits_match_restatement(T, seed):
    """Every site of a 2-block model, both widths, a T that is not a multiple of 4: bit-identical keep masks."""
    widths = {0: 64, 1: 64, 2: 256, 3: 64, 4: 64, 5: 256, 6: 64}
    for site, width in widths.items():
        for p in (0.1, 0.3, 0.5):
            want = DO.multipliers(seed, site, 1, T, width, p).reshape(T, width) != 0
            got = _device_keep(seed, site, T, width, p)
            assert np.array_equal(got, want), (site, width, p, int((got != want).sum()))
    assert _device_keep(seed, 2, T, 256, 0.0).all()
    # a width that is not a multiple of 4 writes exactly width bytes per row
    assert np.array_equal(_device_keep(seed, 3, T, 62, 0.3), DO.multipliers(seed, 3, 1, T, 62, 0.3).reshape(T, 62) != 0)


def _check_against_oracle(m, golden_sd, ids, labels, p_embed, p_attn, gen_seed):
    """One ce_loss(dropout=True) step with generator seeded gen_seed, against the oracle under the same multipliers."""
    seed = _draw_seed(torch.Generator().manual_seed(gen_seed))
    loss, got = _step(m, ids, labels, dropout=True, generator=torch.Generator().manual_seed(gen_seed))
    mults = DO.site_multipliers(seed, ids.shape[0], ids.shape[1], 2, p_embed, p_attn, p_embed)
    ref_loss, want = DO.loss_and_grads(ids, labels, golden_sd, mults)
    assert abs(loss - ref_loss) <= 1e-5 * max(1.0, abs(ref_loss)), (loss, ref_loss)
    assert len(got) == len(want) == 30
    for k, w in want.items():
        g = got[k].cpu().numpy()
        assert g.shape == w.shape and g.dtype == w.dtype, k
        np.testing.assert_allclose(g, w, rtol=1e-3, atol=1e-3 * float(np.abs(w).max()) + 1e-9, err_msg=k)
    return loss, ref_loss


@pytest.mark.parametrize("name", ["left_l20", "left_l50"])
def test_dropout_gradients_match_oracle_autograd(golden_sd, gcase, name):
    ids, labels = _batch(gcase, name)
    m = _model(golden_sd, 0.2, 0.3)
    loss, _ = _check_against_oracle(m, golden_sd, ids, labels, 0.2, 0.3, gen_seed=2024)
    assert abs(loss - float(gcase[f"{name}_loss"])) > 1e-4       # dropout did change the loss
    # the two rates are not interchangeable: the oracle with swapped rates gives another loss
    seed = _draw_seed(torch.Generator().manual_seed(2024))
    swapped = DO.ce_loss_train(ids, labels, golden_sd,
                               DO.site_multipliers(seed, ids.shape[0], ids.shape[1], 2, 0.3, 0.2, 0.3)).item()
    assert abs(swapped - loss) > 1e-4


def test_dropout_gradients_match_oracle_at_half(golden_sd, gcase):
    ids, labels = _batch(gcase, "left_l50")
    _check_against_oracle(_model(golden_sd, 0.5, 0.5), golden_sd, ids, labels, 0.5, 0.5, gen_seed=7)


def _assert_same(a, b, rtol=1e-6):
    (la, ga), (lb, gb) = a, b
    assert abs(la - lb) <= rtol * max(1.0, abs(lb)), (la, lb)
    for k in gb:
        scale = float(gb[k].abs().max())
        assert torch.allclose(ga[k], gb[k], rtol=rtol, atol=rtol * scale + 1e-12), k


@pytest.mark.parametrize("name", ["left_l20", "left_l50"])
def test_zero_rates_and_eval_mode_equal_the_plain_step(golden_sd, gcase, name):
    """Rates 0 through lrb_train_step_dropout, and dropout=True in eval mode, give today's lrb_train_step result
    (float atomics in the TN GEMMs and LayerNorm reductions: compared to 1e-6, not bitwise)."""
    ids, labels = _batch(gcase, name)
    m = _model(golden_sd, 0.2, 0.3)
    plain = _step(m, ids, labels)                                  # dropout=False: lrb_train_step
    assert abs(plain[0] - float(gcase[f"{name}_loss"])) <= 1e-5 * max(1.0, abs(plain[0]))
    m.eval()
    _assert_same(_step(m, ids, labels, dropout=True), plain)       # eval mode: dropout is off
    m.train()
    m.bert_dropout = m.bert_attn_dropout = 0.0
    _assert_same(_step(m, ids, labels, dropout=True), plain)       # the dropout entry point with every rate 0


def test_manual_seed_reproduces_and_steps_differ(golden_sd, gcase):
    ids, labels = _batch(gcase, "left_l50")
    m = _model(golden_sd)
    torch.manual_seed(31)
    a = _step(m, ids, labels, dropout=True)
    b = _step(m, ids, labels, dropout=True)                        # next draw of the default generator
    torch.manual_seed(31)
    a2 = _step(m, ids, labels, dropout=True)
    _assert_same(a2, a, rtol=1e-4)
    assert a[0] != b[0]


def test_accumulation_and_incoming_gradient_scale_with_dropout(golden_sd, gcase):
    ids, labels = _batch(gcase, "left_l20")
    m = _model(golden_sd)
    _, g1 = _step(m, ids, labels, dropout=True, generator=torch.Generator().manual_seed(5))
    m.zero_grad(set_to_none=True)
    (2.0 * m.ce_loss(ids.cuda(), labels.cuda(), dropout=True, generator=torch.Generator().manual_seed(5))).backward()
    for k, p in m.named_parameters():
        assert torch.allclose(p.grad, 2.0 * g1[k], rtol=1e-4, atol=1e-4 * float(g1[k].abs().max()) + 1e-12), k
    m.ce_loss(ids.cuda(), labels.cuda(), dropout=True, generator=torch.Generator().manual_seed(5)).backward()
    for k, p in m.named_parameters():                              # accumulates like autograd: 2 g + g
        assert torch.allclose(p.grad, 3.0 * g1[k], rtol=1e-4, atol=1e-4 * float(g1[k].abs().max()) + 1e-12), k


def test_retriever_calculate_loss_passes_the_flag(golden_sd, gcase):
    ids, labels = _batch(gcase, "left_l20")
    m = _model(golden_sd)
    tr = LRURetriever(_args(400, 0.2, 0.3), m)
    torch.manual_seed(3)
    a = tr.calculate_loss((ids.cuda(), labels.cuda()), dropout=True).item()
    torch.manual_seed(3)
    b = m.ce_loss(ids.cuda(), labels.cuda(), dropout=True).item()
    assert abs(a - b) <= 1e-6 * max(1.0, abs(b))
    plain = tr.calculate_loss((ids.cuda(), labels.cuda())).item()
    assert abs(plain - float(gcase["left_l20_loss"])) <= 1e-5 * max(1.0, abs(plain))


def test_dropout_without_backward_path_raises(golden_sd, gcase):
    ids, labels = _batch(gcase, "left_l20")
    m = _model(golden_sd)
    with torch.no_grad(), pytest.raises(ValueError):
        m.ce_loss(ids.cuda(), labels.cuda(), dropout=True)
    with pytest.raises(ValueError):
        m.ce_loss(ids.cuda(), labels.cuda(), dropout=True, return_row_loss=True)


def test_c_entry_point_rejects_bad_rates():
    lib = _lib.load()
    # ids, id_bytes, labels, B, L, table, rows, bias, weights, params_log, n_blocks, ignore_index, loss_sum, grad_weights,
    # grad_table, grad_bias, workspace, workspace_bytes, stream: the rates are checked before anything else
    n = [None, 8, None, 1, 1, None, 1, None, None, None, 2, 0, None, None, None, None, None, 0, None]
    for p in (1.0, float("nan"), -0.25):
        for rates in ((p, 0.0, 0.0), (0.0, p, 0.0), (0.0, 0.0, p)):
            rc = lib.lrb_train_step_dropout(*n, *rates, 1)
            assert rc == -1 and b"dropout rates" in lib.lrb_last_error(), (rates, rc)
    keep = torch.empty(4, 64, dtype=torch.uint8, device="cuda")
    for p in (1.0, float("nan")):
        assert lib.lrb_dropout_mask(1, 0, 4, 64, p, keep.data_ptr(), None) == -1


def test_adam_training_with_dropout_reduces_the_loss():
    cfg = synth.Config("dropout_smoke", 512, 300, 20, 64)
    ids, last = synth.make_sequences(cfg, seed=3)
    labels = torch.zeros_like(ids)
    labels[:, :-1] = ids[:, 1:]
    labels[:, -1] = last.view(-1)
    labels[ids == 0] = 0
    m = LRURec(_args(cfg.num_items, 0.2, 0.2))
    m.load_state_dict(synth.make_state_dict(cfg.num_items, seed=3))
    m = m.cuda().train()
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    x, y = ids[:64].cuda(), labels[:64].cuda()
    torch.manual_seed(0)
    losses = []
    for _ in range(50):
        opt.zero_grad(set_to_none=True)
        loss = m.ce_loss(x, y, dropout=True)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert all(math.isfinite(v) for v in losses)
    assert np.mean(losses[-5:]) < np.mean(losses[:5]), losses
