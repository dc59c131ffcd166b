"""CPU: the oracle run in float64 (complex128 for the recurrence) is the same restatement as the fp32 one that the
fixtures pin.  The fp64 results must agree with the reference's own fp32 outputs at the bar the fp32 oracle meets
(tests/test_oracle_golden.py), so the fp64 oracle can serve as the tighter reference of the GPU tests."""
import os

import numpy as np
import pytest
import torch

from conftest import CASES, GOLDEN, load_case
from oracle import dropout_oracle as DO
from oracle import lru_oracle as O
from oracle import verbalizer_oracle as VO

F64 = torch.float64


@pytest.mark.parametrize("name", CASES)
def test_fp64_hidden_and_scores_match_the_fixtures(golden_sd, name):
    c = load_case(name)
    ids = torch.from_numpy(c["ids"])
    hid = O.hidden_states(ids, golden_sd, F64)
    assert hid.dtype == F64
    np.testing.assert_allclose(hid.numpy(), c["hidden"], atol=2e-6, rtol=1e-5)
    np.testing.assert_allclose(O.encode(ids, golden_sd, F64).numpy(), c["hidden"][:, -1], atol=2e-6, rtol=1e-5)
    scores = O.forward_scores(ids, golden_sd, F64)
    assert scores.dtype == F64
    np.testing.assert_allclose(scores[:, -1].numpy(), c["last_scores"], atol=2e-6, rtol=1e-5)


@pytest.mark.parametrize("name", ["left_l20", "left_l50"])
def test_fp64_loss_and_grads_match_reference_autograd(golden_sd, name):
    """The reference's own fp32 autograd (grad_case.npz) against the fp64 oracle's: every parameter within 1e-4 of
    the tensor's largest entry."""
    g = np.load(os.path.join(GOLDEN, "grad_case.npz"))
    ids = torch.from_numpy(load_case(name)["ids"])
    labels = torch.from_numpy(g[f"{name}_labels"])
    loss, grads = DO.loss_and_grads(ids, labels, golden_sd, dtype=F64)
    assert abs(loss - float(g[f"{name}_loss"])) <= 1e-5 * abs(loss)
    assert len(grads) == 30
    for k, w64 in grads.items():
        want = g[f"{name}:{k}"]
        assert w64.dtype == (np.complex128 if np.iscomplexobj(want) else np.float64), k
        scale = float(np.abs(w64).max())
        np.testing.assert_allclose(w64, want, rtol=1e-4, atol=1e-4 * scale, err_msg=k)


def test_fp64_verbalizer_oracle_matches_the_fixtures():
    """process_logits on float64 inputs computes in float64 and reproduces the reference's own outputs
    (verbalizer_case.npz, verbalizer_handlers.npz) at the fp32 oracle's tolerances: every handler, both modes,
    multi-word classes and calibration.  The hidden-state outputs are compared on the bf16 logits the reference's
    lm_head produced, widened to float64."""
    from llamarec_b200 import ManualVerbalizer

    class Tok:
        def encode(self, word, add_special_tokens=False):
            return [17 + (ord(c) * 7) % 250 for c in word]
    d = np.load(os.path.join(GOLDEN, "verbalizer_case.npz"))
    h = np.load(os.path.join(GOLDEN, "verbalizer_handlers.npz"))
    logits = torch.from_numpy(d["logits"]).to(F64)
    ids, tm, wm = (torch.from_numpy(d[k]) for k in ("label_words_ids", "words_ids_mask", "label_words_mask"))
    lg = VO.lm_head_last(torch.from_numpy(d["hidden"]).to(torch.bfloat16),
                         torch.from_numpy(d["lm_head"]).to(torch.bfloat16)).to(F64)
    for pls in (0, 1):
        o = VO.process_logits(logits, ids, tm, wm, bool(pls))
        assert o.dtype == F64
        np.testing.assert_allclose(o.numpy(), d[f"out_pls{pls}"], atol=1e-6)
        np.testing.assert_allclose(VO.process_logits(lg, ids, tm, wm, bool(pls)).numpy(), d[f"hidden_out_pls{pls}"],
                                   atol=1e-5)
    ids2, tm2, wm2 = (torch.from_numpy(d[k]) for k in ("multi_label_words_ids", "multi_words_ids_mask",
                                                       "multi_label_words_mask"))
    np.testing.assert_allclose(VO.process_logits(logits, ids2, tm2, wm2, True).numpy(), d["multi_out"], atol=1e-6)
    lw = {i: ([chr(ord("A") + i), "xy" + chr(ord("a") + i)] if i % 4 else [chr(ord("A") + i) + "q"]) for i in range(16)}
    cal = torch.from_numpy(h["calibrate_logits"]).to(F64)
    for handler in ("first", "max", "mean"):
        v = ManualVerbalizer(Tok(), classes=list(range(16)), label_words=lw, prefix="", multi_token_handler=handler)
        for pls in (0, 1):
            o = VO.process_logits(logits, v.label_words_ids, v.words_ids_mask, v.label_words_mask, bool(pls), handler)
            assert o.dtype == F64
            np.testing.assert_allclose(o.numpy(), h[f"{handler}_pls{pls}"], atol=1e-6)
        if handler != "max":
            o = VO.process_logits(logits, v.label_words_ids, v.words_ids_mask, v.label_words_mask, True, handler,
                                  calibrate_logits=cal)
            assert o.dtype == F64
            np.testing.assert_allclose(o.numpy(), h[f"{handler}_calibrated"], atol=1e-5)


def test_default_dtype_is_the_fp32_restatement(golden_sd):
    """Without a dtype nothing changes: fp32 in, fp32 (complex64 inside) out, and the fp64 multipliers of a dropout
    site are applied in the computation's dtype."""
    ids = torch.from_numpy(load_case("left_l20")["ids"])
    assert O.hidden_states(ids, golden_sd).dtype == torch.float32
    labels = torch.zeros_like(ids)
    labels[:, :-1] = ids[:, 1:]
    mults = DO.site_multipliers(11, ids.shape[0], ids.shape[1], 2, 0.2, 0.3, 0.2)
    l32 = DO.ce_loss_train(ids, labels, golden_sd, mults)
    l64 = DO.ce_loss_train(ids, labels, golden_sd, mults, dtype=F64)
    assert l32.dtype == torch.float32 and l64.dtype == F64
    assert abs(l32.item() - l64.item()) <= 1e-5 * abs(l64.item())
    rows = DO.ce_loss_train(ids, labels, golden_sd, mults, dtype=F64, reduction="none")
    counted = labels.reshape(-1) != 0
    assert torch.allclose(rows[counted].mean(), l64) and bool((rows[~counted] == 0).all())
