"""GPU (-m gpu): the CUDA path, driven through the C ABI, against the CPU oracle on the same seeded inputs,
against the committed golden fixtures (reference outputs), and -- at BASELINE.json's full sizes -- through
size-independent properties.  Tolerances: scores 1e-3 relative (north_star); candidate ids identical except
for ties inside that tolerance; metrics to 4 decimals."""
import os
import pickle
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from conftest import CASES, GOLDEN, load_case, metrics_vector
from llamarec_b200 import LRURec, LRURetriever, ManualVerbalizer, absolute_recall_mrr_ndcg_for_ks, merge_lists, synth
from oracle import lru_oracle as O
from oracle import metrics_oracle as MO
from oracle import verbalizer_oracle as VO

pytestmark = pytest.mark.gpu
RTOL = 1e-3


def _args(n):
    return SimpleNamespace(num_items=n, bert_hidden_units=64, bert_num_blocks=2, bert_dropout=0.2,
                           bert_attn_dropout=0.2, metric_ks=[1, 5, 10, 20, 50], llm_negative_sample_size=19)


@pytest.fixture(scope="module")
def model(golden_sd):
    m = LRURec(_args(400))
    m.load_state_dict(golden_sd)
    return m.cuda().eval()


def assert_topk_equivalent(ids_a, s_a, ids_b, s_b, rtol=RTOL):
    """Lists equal, or differing only by swaps / boundary replacements among scores tied within rtol."""
    ids_a, s_a, ids_b, s_b = (np.asarray(t) for t in (ids_a, s_a, ids_b, s_b))
    n_diff_rows = 0
    for r in range(ids_a.shape[0]):
        if np.array_equal(ids_a[r], ids_b[r]):
            continue
        n_diff_rows += 1
        tol = rtol * max(1.0, float(np.abs(s_b[r]).max()))
        assert np.allclose(s_a[r], s_b[r], atol=tol), f"row {r}: scores differ beyond tolerance"
        pos_b = {int(i): p for p, i in enumerate(ids_b[r])}
        for p, i in enumerate(ids_a[r]):
            if ids_b[r][p] == i:
                continue
            if int(i) in pos_b:
                assert abs(s_a[r][p] - s_b[r][pos_b[int(i)]]) <= tol, f"row {r}: id {i} moved across non-tied scores"
            else:
                assert abs(s_a[r][p] - s_b[r][-1]) <= tol, f"row {r}: id {i} is not a boundary tie"
    return n_diff_rows


@pytest.mark.parametrize("name", CASES)
def test_hidden_states_match_reference(model, name):
    c = load_case(name)
    ids = torch.from_numpy(c["ids"]).cuda()
    hid = model.hidden_states(ids).cpu().numpy()
    np.testing.assert_allclose(hid, c["hidden"], atol=1e-4, rtol=1e-4)
    u = model.encode(ids).cpu().numpy()
    np.testing.assert_allclose(u, c["hidden"][:, -1, :], atol=1e-4, rtol=1e-4)


@pytest.mark.parametrize("name", ["left_l20", "holes_l37"])
def test_forward_scores_match_reference(model, golden_sd, name):
    c = load_case(name)
    ids = torch.from_numpy(c["ids"])
    out = model(ids.cuda()).cpu()
    assert out.shape == (ids.shape[0], ids.shape[1], 401)
    ref = O.forward_scores(ids, golden_sd)
    np.testing.assert_allclose(out.numpy(), ref.numpy(), atol=1e-4, rtol=RTOL)
    np.testing.assert_allclose(out[:, -1].numpy(), c["last_scores"], atol=1e-4, rtol=RTOL)


@pytest.mark.parametrize("name", CASES)
def test_retrieve_fp32_matches_reference_topk(model, name):
    c = load_case(name)
    ids = torch.from_numpy(c["ids"]).cuda()
    res = model.retrieve(ids, k=20, exclude_history=True, precision="fp32")
    assert_topk_equivalent(res["ids"].cpu().numpy(), res["scores"].cpu().numpy(), c["top_ids"], c["top_scores"])


@pytest.mark.parametrize("name", CASES)
def test_retrieve_bf16_matches_oracle_on_same_operands(model, golden_sd, name):
    c = load_case(name)
    ids_cpu = torch.from_numpy(c["ids"])
    u, u16 = model.encode(ids_cpu.cuda(), want_bf16=True)
    res = model.retrieve(ids_cpu.cuda(), k=20, exclude_history=True, precision="bf16")
    table16 = golden_sd["embedding.token.weight"].to(torch.bfloat16).float()
    ref_s, ref_i = O.retrieve(ids_cpu, golden_sd, 20, u=u16.float().cpu(), table=table16)
    assert_topk_equivalent(res["ids"].cpu().numpy(), res["scores"].cpu().numpy(), ref_i.numpy(), ref_s.numpy(), rtol=1e-5)
    # and against the fp32 reference scores within the north_star tolerance
    np.testing.assert_allclose(res["scores"].cpu().numpy()[:, 0], c["top_scores"][:, 0], atol=5e-3, rtol=1e-2)


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("exclude", [True, False])
def test_calculate_metrics_to_4_decimals(model, name, exclude):
    c = load_case(name)
    ks = c["ks"].tolist()
    tr = LRURetriever(_args(400), model)
    got = tr.calculate_metrics((torch.from_numpy(c["ids"]).cuda(), torch.from_numpy(c["labels"]).cuda().view(-1, 1)),
                               exclude_history=exclude)
    want = c["metrics_masked"] if exclude else c["metrics_raw"]
    np.testing.assert_allclose(metrics_vector(got, ks), want, atol=5e-5)
    assert list(got.keys())[0] == "Recall@50"     # reference key order: k descending


def test_metrics_function_on_dense_scores(model):
    c = load_case("left_l50")
    ks = c["ks"].tolist()
    scores = torch.from_numpy(c["last_scores"]).cuda()
    got = absolute_recall_mrr_ndcg_for_ks(scores, torch.from_numpy(c["labels"]).cuda(), ks)
    np.testing.assert_allclose(metrics_vector(got, ks), c["metrics_raw"], atol=5e-5)


def test_generate_candidates_matches_reference_pickle(model, tmp_path):
    with open(os.path.join(GOLDEN, "generate_candidates_ref.pkl"), "rb") as f:
        g = pickle.load(f)
    bs, ks, ref = g["batch"], g["ks"], g["ref"]
    mk = lambda ids, lab: [(torch.from_numpy(ids[i:i + bs]), torch.from_numpy(lab[i:i + bs]).unsqueeze(1))
                           for i in range(0, len(ids), bs)]
    args = _args(g["num_items"])
    args.num_users = g["num_users"]
    tr = LRURetriever(args, model, mk(g["ids_val"], g["lab_val"]), mk(g["ids_test"], g["lab_test"]))
    path = str(tmp_path / "retrieved.pkl")
    tr.generate_candidates(path)
    with open(path, "rb") as f:
        ours = pickle.load(f)
    assert set(ours.keys()) == set(ref.keys())
    for key in ("val_users", "test_users", "non_test_users", "test_labels"):
        assert ours[key] == ref[key], key
    # candidate lists: identical, or -- the fixture records the reference's scores of every test user --
    # differing only among items whose reference scores tie within the tolerance (torch.topk's tie order is
    # implementation-defined)
    ref_scores = g.get("test_scores")
    for key in ("val_candidates", "test_candidates", "test_probs"):
        assert len(ours[key]) == len(ref[key])
        n_diff = 0
        for idx, (a, b) in enumerate(zip(ours[key], ref[key])):
            assert len(a) == len(b) and len(set(a)) == len(a), (key, idx)
            if a == b:
                continue
            n_diff += 1
            assert sorted(a)[:-1] == sorted(b)[:-1] or sorted(a) == sorted(b) or len(set(a) ^ set(b)) <= 2, (key, idx, a, b)
            if ref_scores is not None and key == "test_probs":
                sc = ref_scores[idx]
                for pa, pb in zip(a, b):
                    if pa != pb:
                        assert abs(sc[pa] - sc[pb]) <= RTOL * max(1.0, abs(sc[pb])), (key, idx, pa, pb)
        assert n_diff <= 1, (key, n_diff, len(ref[key]))                 # at most one tie-swapped list
    for key in ("val_metrics", "test_metrics"):
        for k, v in ref[key].items():
            assert abs(ours[key][k] - v) < 5e-5, (key, k)
    for key in ("retrieval_metrics", "non_retrieval_metrics"):
        for k, v in ref["test_retrieval"][key].items():
            assert abs(ours["test_retrieval"][key][k] - v) < 5e-5, (key, k)
    assert ours["test_retrieval"]["retrieval_size"] == ref["test_retrieval"]["retrieval_size"]


def test_verbalizer_kernel_matches_reference():
    d = np.load(os.path.join(GOLDEN, "verbalizer_case.npz"))

    class Tok:
        def encode(self, word, add_special_tokens=False):
            return [17 + (ord(c) * 7) % 250 for c in word]
    hid = torch.from_numpy(d["hidden"]).to(torch.bfloat16).cuda()
    w = torch.from_numpy(d["lm_head"]).to(torch.bfloat16).cuda()
    for pls in (0, 1):
        v = ManualVerbalizer(Tok(), classes=list(range(20)), label_words={i: chr(ord("A") + i) for i in range(20)},
                             prefix="", post_log_softmax=bool(pls))
        assert np.array_equal(v.label_words_ids.numpy(), d["label_words_ids"])
        out = v.score_hidden(hid, w).cpu().numpy()
        # logits are bf16-rounded like the reference's; a different fp32 summation order may flip a rounding
        np.testing.assert_allclose(out, d[f"hidden_out_pls{pls}"], atol=4e-2, rtol=8e-3)
        close = np.isclose(out, d[f"hidden_out_pls{pls}"], atol=1e-4, rtol=1e-4).mean()
        assert close > 0.9
        exact = v.score_hidden(hid, w, round_logits_to_bf16=False).cpu()
        lg = torch.nn.functional.linear(hid.float().cpu(), w.float().cpu())
        ref = v.process_logits(lg)
        np.testing.assert_allclose(exact.numpy(), ref.numpy(), atol=2e-4, rtol=RTOL)
        # process_logits on precomputed logits (lrb_verbalizer_from_logits) reproduces the reference outputs
        np.testing.assert_allclose(v.process_logits(torch.from_numpy(d["logits"])).numpy(), d[f"out_pls{pls}"],
                                   atol=5e-6, rtol=2e-6)
    # multi-token label words, all three handlers, against the reference class (verbalizer_handlers.npz)
    h = np.load(os.path.join(GOLDEN, "verbalizer_handlers.npz"))
    lw = {i: ([chr(ord("A") + i), "xy" + chr(ord("a") + i)] if i % 4 else [chr(ord("A") + i) + "q"]) for i in range(16)}
    logits = torch.from_numpy(d["logits"]).cuda()
    for handler in ("first", "max", "mean"):
        for pls in (0, 1):
            v = ManualVerbalizer(Tok(), classes=list(range(16)), label_words=lw, prefix="",
                                 post_log_softmax=bool(pls), multi_token_handler=handler)
            got = v.process_logits(logits).cpu().numpy()
            np.testing.assert_allclose(got, h[f"{handler}_pls{pls}"], atol=5e-6, rtol=2e-6)
    # calibration (register_calibrate_logits -> ManualVerbalizer.calibrate, trainer/verb.py:202-208,616-643) against
    # the reference class, on precomputed logits (first / mean handlers) and through the hidden-state kernel
    cal = torch.from_numpy(h["calibrate_logits"])
    for handler in ("first", "mean"):
        vc = ManualVerbalizer(Tok(), classes=list(range(16)), label_words=lw, prefix="", post_log_softmax=True,
                              multi_token_handler=handler)
        vc.register_calibrate_logits(cal)
        np.testing.assert_allclose(vc.process_logits(logits).cpu().numpy(), h[f"{handler}_calibrated"], atol=2e-5, rtol=1e-5)
        vc.register_calibrate_logits(None)
        np.testing.assert_allclose(vc.process_logits(logits).cpu().numpy(), h[f"{handler}_pls1"], atol=5e-6, rtol=2e-6)
    vh = ManualVerbalizer(Tok(), classes=list(range(20)), label_words={i: chr(ord("A") + i) for i in range(20)},
                          prefix="", post_log_softmax=True)
    vh.register_calibrate_logits(cal)
    lg = torch.nn.functional.linear(hid.float().cpu(), w.float().cpu())
    want = VO.process_logits(lg, vh.label_words_ids, vh.words_ids_mask, vh.label_words_mask, True, "first",
                             calibrate_logits=cal)
    np.testing.assert_allclose(vh.score_hidden(hid, w, round_logits_to_bf16=False).cpu().numpy(), want.numpy(),
                               atol=2e-4, rtol=RTOL)
    with pytest.raises(AssertionError):
        vh.register_calibrate_logits(torch.zeros(2, 3))
    # a non-contiguous view of a wider logits matrix (row pitch > V)
    wide = torch.zeros(logits.shape[0], logits.shape[1] + 37, device="cuda")
    wide[:, :logits.shape[1]] = logits
    np.testing.assert_allclose(v.process_logits(wide[:, :logits.shape[1]]).cpu().numpy(), got, atol=1e-7)


@pytest.mark.parametrize("name", ["left_l20", "holes_l37", "left_l200"])
def test_train_step_loss_matches_reference_cross_entropy(model, golden_sd, name):
    """Fused log-sum-exp loss (no logits tensor) against the reference's LRUTrainer.calculate_loss
    (trainer/lru.py:20-28, fixture ce_case.npz); labels = the next item, 0 where the input is padding."""
    ce = np.load(os.path.join(GOLDEN, "ce_case.npz"))             # the reference's own loss on these inputs
    ids = torch.from_numpy(load_case(name)["ids"])
    labels = torch.from_numpy(ce[f"{name}_labels"])
    ref = float(ce[f"{name}_loss"])
    assert abs(O.ce_loss(ids, labels, golden_sd).item() - ref) < 1e-6
    loss, rows = model.ce_loss(ids.cuda(), labels.cuda(), return_row_loss=True)
    assert abs(loss.item() - ref) <= 1e-5 * max(1.0, abs(ref)), (loss.item(), ref)
    np.testing.assert_allclose(rows.cpu().numpy(), ce[f"{name}_row_loss"], atol=2e-5, rtol=1e-5)
    # the retriever-level mirror of LRUTrainer.calculate_loss (value only here: rows with zeros in the middle have no
    # backward -- the train step takes the left-padded batches the reference's dataloader produces)
    retr = LRURetriever(_args(400), model)
    with torch.no_grad():
        assert abs(retr.calculate_loss((ids.cuda(), labels.cuda())).item() - ref) <= 1e-5 * max(1.0, abs(ref))


@pytest.mark.parametrize("name", ["left_l50", "left_l20"])
def test_train_step_gradients_match_reference_autograd(golden_sd, name):
    """loss.backward() through the fused train step (lrb_train_step) against the gradients torch's autograd computes
    for the REFERENCE model on the same batch (fixture grad_case.npz, `python oracle/make_golden.py grad`):
    every parameter, rtol 1e-3 (atol = 1e-3 of the gradient's largest entry; fp32 summation order differs)."""
    gcase = np.load(os.path.join(GOLDEN, "grad_case.npz"))
    m = LRURec(_args(400))
    m.load_state_dict(golden_sd)
    m = m.cuda().train()                                     # dropout is the identity in the kernels either way
    ids = torch.from_numpy(load_case(name)["ids"]).cuda()
    labels = torch.from_numpy(gcase[f"{name}_labels"]).cuda()
    loss = m.ce_loss(ids, labels)
    assert loss.requires_grad
    ref_loss = float(gcase[f"{name}_loss"])
    assert abs(loss.item() - ref_loss) <= 1e-5 * max(1.0, abs(ref_loss)), (loss.item(), ref_loss)
    (2.0 * loss).backward()                                  # the incoming gradient scales every parameter gradient
    checked = 0
    for k, p in m.named_parameters():
        want = gcase[f"{name}:{k}"]
        assert p.grad is not None, k
        got = (p.grad / 2.0).detach().cpu().numpy()
        assert got.shape == want.shape and got.dtype == want.dtype, (k, got.shape, got.dtype, want.dtype)
        scale = float(np.abs(want).max())
        np.testing.assert_allclose(got, want, rtol=1e-3, atol=1e-3 * scale + 1e-9, err_msg=k)
        checked += 1
    assert checked == len(list(m.named_parameters())) == 30
    # gradients accumulate like autograd's: a second backward doubles them
    g0 = m.model.bias.grad.clone()
    m.ce_loss(ids, labels).backward()
    assert torch.allclose(m.model.bias.grad, g0 * 1.5, rtol=1e-5, atol=1e-9)
    # under no_grad the same entry point is the forward value only
    with torch.no_grad():
        v = m.ce_loss(ids, labels)
    assert not v.requires_grad and abs(v.item() - ref_loss) <= 1e-5 * max(1.0, abs(ref_loss))


def test_train_step_rejects_rows_that_are_not_left_padded(model):
    from llamarec_b200._lib import LrbError
    ids = torch.tensor([[0, 5, 0, 7, 9]], dtype=torch.int64).cuda()
    labels = torch.tensor([[0, 0, 0, 9, 3]], dtype=torch.int64).cuda()
    with pytest.raises(LrbError):
        model.ce_loss(ids, labels)


def test_train_step_loss_all_labels_ignored_is_nan(model):
    ids = torch.zeros(3, 20, dtype=torch.int64)
    ids[:, -1] = 5
    loss = model.ce_loss(ids.cuda(), torch.zeros_like(ids).cuda())
    assert torch.isnan(loss)                                   # torch's CrossEntropyLoss gives nan as well


def test_stage2_caller_matches_full_lm_head_chain():
    """score_candidates (transformer body -> last hidden state -> label-row kernel) against the reference chain
    lm_head at every position -> .float() -> [:, -1] -> process_logits (model/llm.py:113-131, trainer/llm.py:63-72)
    on a tiny random-init Llama; the metrics on the label scores match the metrics oracle."""
    transformers = pytest.importorskip("transformers")
    from llamarec_b200 import stage2

    class Tok:   # 'A'..'T' -> fixed ids, like the fake tokenizer of oracle/make_golden.py
        def encode(self, word, add_special_tokens=False):
            return [100 + ord(word[-1]) - ord("A")]

    cfg = transformers.LlamaConfig(vocab_size=1000, hidden_size=512, intermediate_size=1024, num_hidden_layers=2,
                                   num_attention_heads=4, num_key_value_heads=4, max_position_embeddings=128)
    torch.manual_seed(0)
    llm = transformers.LlamaForCausalLM(cfg).to(torch.bfloat16).cuda().eval()
    ids = torch.randint(5, 1000, (37, 23), device="cuda")
    labels = torch.randint(0, 20, (37,), device="cuda")
    for post in (False, True):
        vb = ManualVerbalizer(tokenizer=Tok(), prefix="", post_log_softmax=post, classes=list(range(20)),
                              label_words={i: chr(ord("A") + i) for i in range(20)})
        got = stage2.score_candidates(llm, vb, ids)
        with torch.no_grad():
            logits = llm(input_ids=ids).logits.float()[:, -1]
        ref = vb.process_logits(logits)
        # both sides round the 20 logits to bf16 (fp32 accumulation order may move one of them by one bf16 ulp)
        assert torch.allclose(got, ref, atol=2e-2, rtol=1e-2), (got - ref).abs().max()
        # bf16-rounded logits can tie exactly; argsort's tie order is implementation-defined, so de-tie first
        got = got - 1e-4 * torch.arange(20, device="cuda", dtype=torch.float32)
        m = stage2.rerank_metrics(got, labels, [1, 5, 10])
        m_ref = MO.recall_mrr_ndcg(got.cpu(), labels.cpu(), [1, 5, 10])
        for k, v in m_ref.items():
            assert abs(m[k] - v) < 5e-5, (k, m[k], v)


# ------------------------------------------------------------------------------------------------
# Larger shapes: oracle on the same seeded inputs (seconds on CPU) and size-independent properties
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def games_model():
    cfg = synth.CONFIGS["c3_games"]
    sd = synth.make_state_dict(cfg.num_items, seed=42, bias_std=0.01)
    m = LRURec(_args(cfg.num_items))
    m.load_state_dict(sd)
    return m.cuda().eval(), sd, cfg


def test_games_shaped_batch_2048_against_oracle(games_model):
    m, sd, cfg = games_model
    ids, labels = synth.make_sequences(cfg, num_users=2048, seed=42)
    res = m.retrieve(ids.cuda(), k=50, exclude_history=True, labels=labels.cuda(), ks=[1, 5, 10, 20, 50], precision="fp32")
    u_ref = O.encode(ids, sd)
    np.testing.assert_allclose(res["u"].cpu().numpy(), u_ref.numpy(), atol=2e-4, rtol=RTOL)
    ref_s, ref_i = O.retrieve(ids, sd, 50, u=u_ref)
    diff_rows = assert_topk_equivalent(res["ids"].cpu().numpy(), res["scores"].cpu().numpy(), ref_i.numpy(), ref_s.numpy())
    assert diff_rows <= 0.02 * 2048          # >= 98 % of the 2048 lists bit-identical in order
    # label ranks and metric sums agree with the oracle's ranking
    rank = res["label_rank"].cpu().numpy()
    pos = (ref_i == labels.view(-1, 1)).float()
    ref_rank = torch.where(pos.sum(1) > 0, pos.argmax(1), torch.full((2048,), -1)).numpy()
    assert (rank == ref_rank).mean() > 0.995
    # bf16 tensor-core path: same operands -> same lists
    u, u16 = m.encode(ids.cuda(), want_bf16=True)
    res16 = m.retrieve(ids.cuda(), k=20, exclude_history=True, precision="bf16")
    t16 = sd["embedding.token.weight"].to(torch.bfloat16).float()
    r16_s, r16_i = O.retrieve(ids, sd, 20, u=u16.float().cpu(), table=t16)
    assert_topk_equivalent(res16["ids"].cpu().numpy(), res16["scores"].cpu().numpy(), r16_i.numpy(), r16_s.numpy(), rtol=1e-5)


def test_virtual_rank_sharding_is_exact(games_model):
    """Shard -> local top-k -> concatenate -> merge on one device equals the unsharded result exactly, for k = 20 and
    k = 50 (the K <= 50 kernel and the default metric_ks)."""
    m, sd, cfg = games_model
    ids, _ = synth.make_sequences(cfg, num_users=300, seed=7)
    x = ids.cuda()
    for k in (20, 50):
        for prec in ("fp32", "bf16"):
            m.set_row_shard(0, cfg.num_items + 1)
            full = m.retrieve(x, k=k, precision=prec)
            u = full["u"]
            parts_s, parts_i = [], []
            R = 4
            per = (cfg.num_items + 1 + R - 1) // R
            for r in range(R):
                m.set_row_shard(r * per, min((r + 1) * per, cfg.num_items + 1))
                loc = m.retrieve(x, k=k, precision=prec, u=u)
                parts_s.append(loc["scores"].clone())
                parts_i.append(loc["ids"].clone())
            m.set_row_shard(0, cfg.num_items + 1)
            merged = merge_lists(torch.stack(parts_s), torch.stack(parts_i), None, k_out=k, layout="list_major")
            assert torch.equal(merged["ids"], full["ids"]) and torch.equal(merged["scores"], full["scores"]), (k, prec)


def test_batches_beyond_one_tile_per_sm_are_chunked(games_model):
    """More users than 128 x SMs (the all-gathered users of a data-parallel job): scored as consecutive launches
    over user chunks; every user's list equals what a small-batch call returns for the same user."""
    m, sd, cfg = games_model
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = 128 * sms + 128 + 37                                   # two chunks, the second one ragged
    ids, _ = synth.make_sequences(cfg, num_users=512, seed=11)
    ids = ids.repeat((B + 511) // 512, 1)[:B]
    ids[512:, -1] = torch.randint(1, cfg.num_items, (B - 512,), generator=torch.Generator().manual_seed(3))
    x = ids.cuda()
    u, u16 = m.encode(x, want_bf16=True)
    big = m.retrieve(x, k=20, precision="bf16", u=u, u_bf16=u16)
    big_i, big_s = big["ids"].clone(), big["scores"].clone()
    for lo in (0, 128 * sms - 64, B - 300):                   # first chunk, across the boundary, ragged tail
        hi = min(lo + 300, B)
        ref = m.retrieve(x[lo:hi], k=20, precision="bf16", u=u[lo:hi].contiguous(), u_bf16=u16[lo:hi].contiguous())
        assert torch.equal(ref["ids"], big_i[lo:hi]) and torch.equal(ref["scores"], big_s[lo:hi])


def test_data_parallel_exchange_records_on_one_device(games_model):
    """The data-parallel path scores users it never saw the ids of: user state + sorted exclusion list + filter
    (the all-gathered exchange record) must give the same lists as the ids themselves, and the [B, 2, k]
    row payload + merge_rows must equal the plain result."""
    from llamarec_b200.sharded import CudaBackend
    m, sd, cfg = games_model
    ids, labels = synth.make_sequences(cfg, num_users=640, seed=13)
    x = ids.cuda()
    ref = m.retrieve(x, k=20, precision="bf16", labels=labels.cuda(), ks=[1, 5, 10, 20])
    ref_i, ref_s, ref_sums = ref["ids"].clone(), ref["scores"].clone(), ref["metric_sums"].clone()
    R = 2
    backs = []
    for r in range(R):
        mm = LRURec(_args(cfg.num_items)); mm.load_state_dict(sd); mm = mm.cuda().eval()
        backs.append(CudaBackend(mm, r, R, precision="bf16"))
    st = backs[0].encode_states(x, True)
    rows = [b.local_topk_rows(st["state"], st["excl"], st["bloom"], st["excl_stride"], 20).clone() for b in backs]
    out = backs[0].merge_rows(torch.stack(rows), 20, labels.cuda(), [1, 5, 10, 20])
    assert torch.equal(out["ids"], ref_i) and torch.equal(out["scores"], ref_s)
    assert torch.allclose(out["metric_sums"], ref_sums, rtol=1e-5)


def test_peer_push_and_scatter_merge_with_local_destinations(games_model):
    """The exchange kernels with every "peer" mapped to local memory: lrb_peer_push copies each array into its
    slot of every destination; lrb_merge_metrics_scatter writes user b's list to row b % n of destination b / n
    and equals the plain merge."""
    from llamarec_b200 import _lib
    lib = _lib.load()
    m, sd, cfg = games_model
    dev = torch.device("cuda")
    g = torch.Generator(device="cuda").manual_seed(5)
    arrays = [torch.randn(96, 64, device=dev, generator=g).to(torch.bfloat16),
              torch.randint(0, 1 << 30, (96, 52), device=dev, generator=g, dtype=torch.int32),
              torch.randint(0, 1 << 30, (96, 4), device=dev, generator=g, dtype=torch.int32)]
    n_dst, slot = 3, 1
    dst = [[torch.zeros((4 * a.shape[0],) + tuple(a.shape[1:]), dtype=a.dtype, device=dev) for _ in range(n_dst)]
           for a in arrays]
    src = (_lib.ctypes.c_void_p * 3)(*[a.data_ptr() for a in arrays])
    nbytes = (_lib.ctypes.c_size_t * 3)(*[a.numel() * a.element_size() for a in arrays])
    ptrs = (_lib.ctypes.c_void_p * 9)(*[dst[a][d][slot * 96:].data_ptr() for a in range(3) for d in range(n_dst)])
    _lib.check(lib.lrb_peer_push(src, nbytes, 3, ptrs, n_dst, _lib.stream_handle()))
    for a in range(3):
        for d in range(n_dst):
            assert torch.equal(dst[a][d][slot * 96:(slot + 1) * 96], arrays[a])
            assert not dst[a][d][:slot * 96].any() and not dst[a][d][(slot + 1) * 96:].any()
    # scatter merge: 300 users, 2 destinations of 150 rows each, rows [2][k] interleaved
    ids, _ = synth.make_sequences(cfg, num_users=300, seed=21)
    part = m.retrieve(ids.cuda(), k=20, precision="bf16", merge=False)
    plain = merge_lists(part["part_scores"], part["part_ids"], part["part_cnt"], k_out=20)
    recv = [torch.full((150, 2, 20), -7, dtype=torch.int32, device=dev) for _ in range(2)]
    scatter = {"dst_scores": [r.data_ptr() for r in recv], "dst_ids": [r.data_ptr() + 20 * 4 for r in recv],
               "users_per_dst": 150, "out_stride": 40}
    merge_lists(part["part_scores"], part["part_ids"], part["part_cnt"], k_out=20, scatter=scatter)
    got = torch.cat(recv)
    assert torch.equal(got[:, 0].view(torch.float32), plain["scores"]) and torch.equal(got[:, 1], plain["ids"])


def test_scout_bound_ignores_pad_columns_of_the_ragged_last_tile():
    """Adversarial case for the union bound's scout pass (zero bias => no folded-bias block => TMA zero-fills the
    pad columns of the last item tile, which then score exactly 0.0).  Every real score is negative, the second
    half of the catalogue scores ten times lower than the first, and rows % 256 = 20 leaves both column halves
    of the last tile with more all-pad 16-item groups than the c = 5 entries a stream must publish: if pad
    columns counted as admissible items, the last stream would publish 0.0, the union bound would sit at the
    first stream's 5th best and ranks 11..20 of every list would be dropped.  9472 users = 37 pair tiles = two
    full streams, no shared stream (the chunk shape of every multi-GPU step)."""
    rows = 256 * 274 + 20                                    # 70,164 rows: 137 tiles per stream >= 128 => scout on
    n, B, K = rows - 1, 9472, 20
    g = torch.Generator().manual_seed(3)
    table = torch.rand(rows, 64, generator=g) * 0.01 + 0.01
    table[rows // 2:] *= 10.0
    m = LRURec(_args(n))
    with torch.no_grad():
        m.embedding.token.weight.copy_(table)
        m.model.bias.zero_()
    m = m.cuda().eval()
    u = -(torch.rand(B, 64, generator=g) + 0.5)
    ids = torch.zeros(B, 50, dtype=torch.int64)
    ids[:, -9:] = torch.randint(1, rows, (B, 9), generator=g)
    ids[::7, -9:] = torch.randint(rows - 16 * 256, rows, (B // 7 + 1, 9), generator=g)[: len(ids[::7])]   # E > 0
    u16 = u.to(torch.bfloat16)
    res = m.retrieve(ids.cuda(), k=K, exclude_history=True, precision="bf16", u=u.cuda(), u_bf16=u16.cuda())
    got_i, got_s = res["ids"].cpu(), res["scores"].cpu()
    assert (got_i >= 1).all() and (got_s < 0).all()          # 20 real items for every user, nothing dropped
    sel = torch.arange(0, B, 37)                             # 256 users spread over all 37 pair tiles
    t16 = table.to(torch.bfloat16).float()
    ref_s, ref_i = O.retrieve(ids[sel], {}, K, u=u16[sel].float(), table=t16, bias=torch.zeros(rows))
    assert_topk_equivalent(got_i[sel].numpy(), got_s[sel].numpy(), ref_i.numpy(), ref_s.numpy(), rtol=1e-5)


def test_full_size_10m_catalogue_properties():
    """BASELINE config 4 (10M items, batch 4096): properties that need no CPU pass over the table, plus an
    exact check of 4 users against a plain torch fp32 matmul over the same bf16 operands."""
    N, B, L, K = 10_000_000, 4096, 50, 20
    sd = synth.make_state_dict(1000, seed=42)
    table, bias = synth.make_table_bf16(N, seed=42, device="cuda")
    m = LRURec(_args(N)).cuda()
    small = {k: v for k, v in sd.items() if k not in ("embedding.token.weight", "model.bias")}
    m.load_state_dict(small, strict=False)
    with torch.no_grad():
        m.embedding.token.weight.copy_(table)
        m.model.bias.copy_(bias)
    del table
    ids, labels = synth.make_sequences_fast(B, N, L, seed=42)
    res = m.retrieve(ids.cuda(), k=K, exclude_history=True, labels=labels.cuda(), ks=[1, 5, 10, 20])
    s, i = res["scores"].cpu(), res["ids"].cpu().long()
    assert torch.all(s[:, 1:] <= s[:, :-1])                              # sorted
    assert torch.all(i >= 1) and torch.all(i <= N)                       # pad item 0 never returned
    assert all(len(set(r.tolist())) == K for r in i[:256])               # unique ids
    hist = ids[:, None, :] == i[:, :, None]
    assert not hist.any()                                                # history excluded
    # idempotence
    res2 = m.retrieve(ids.cuda(), k=K, exclude_history=True)
    assert torch.equal(res2["ids"].cpu().long(), i)
    # exact check of a few users
    u, u16 = m.encode(ids.cuda(), want_bf16=True)
    t16 = m._prepare()["table_bf16"]
    for b in (0, 17, 2048, 4095):
        sc = (t16.float() @ u16[b].float())                              # bias is zero in this config
        sc[ids[b].cuda()] = -1e9
        sc[0] = -1e9
        ts, ti = torch.topk(sc, K)
        assert_topk_equivalent(i[b:b + 1].numpy(), s[b:b + 1].numpy(), ti.cpu().numpy()[None], ts.cpu().numpy()[None], rtol=1e-5)


# ------------------------------------------------------------------------------------------------
# Edge cases the reference's call sites can produce
# ------------------------------------------------------------------------------------------------
def test_single_user_single_position_and_int32_ids(model, golden_sd):
    ids = torch.tensor([[7]], dtype=torch.int64)
    res = model.retrieve(ids.cuda(), k=5, precision="fp32")
    ref_s, ref_i = O.retrieve(ids, golden_sd, 5)
    assert_topk_equivalent(res["ids"].cpu().numpy(), res["scores"].cpu().numpy(), ref_i.numpy(), ref_s.numpy())
    # int32 ids are accepted (converted on device), empty history rows keep the last position
    ids2 = torch.zeros(3, 20, dtype=torch.int32)
    ids2[1, -3:] = torch.tensor([5, 9, 11], dtype=torch.int32)
    res2 = model.retrieve(ids2.cuda(), k=20, precision="fp32")
    ref_s2, ref_i2 = O.retrieve(ids2.long(), golden_sd, 20)
    assert_topk_equivalent(res2["ids"].cpu().numpy(), res2["scores"].cpu().numpy(), ref_i2.numpy(), ref_s2.numpy())


def test_k_larger_than_valid_items_and_no_exclusion():
    """Tiny catalogue: 30 items, histories cover most of it, k=20 > #valid items for some users."""
    n = 30
    sd = synth.make_state_dict(n, seed=5, bias_std=0.05)
    m = LRURec(_args(n))
    m.load_state_dict(sd)
    m = m.cuda().eval()
    rng = np.random.default_rng(0)
    ids = np.zeros((6, 25), dtype=np.int64)
    for b in range(6):
        hist = rng.permutation(np.arange(1, n + 1))[: 8 + 3 * b]
        ids[b, 25 - len(hist):] = hist
    x = torch.from_numpy(ids)
    for prec in ("fp32", "bf16"):
        res = m.retrieve(x.cuda(), k=20, exclude_history=True, precision=prec)
        got_i, got_s = res["ids"].cpu().numpy(), res["scores"].cpu().numpy()
        for b in range(6):
            valid = sorted(set(range(1, n + 1)) - set(ids[b].tolist()))
            k_valid = min(20, len(valid))
            assert set(got_i[b, :k_valid].tolist()) <= set(valid)
            assert len(set(got_i[b, :k_valid].tolist())) == k_valid          # every valid item at most once
            if k_valid < 20:                                                  # the rest is marked missing
                assert np.all(got_i[b, k_valid:] == -1) and np.all(np.isinf(got_s[b, k_valid:]))
    # exclude_history=False (BaseTrainer.validate): item 0 and history items compete (trainer/base.py:141)
    res = m.retrieve(x.cuda(), k=10, exclude_history=False, precision="fp32")
    ref_s, ref_i = O.retrieve(x, sd, 10, exclude_history=False)
    assert_topk_equivalent(res["ids"].cpu().numpy(), res["scores"].cpu().numpy(), ref_i.numpy(), ref_s.numpy())


def test_exact_fp32_selection_with_massive_ties_and_row_shards():
    """The exact-fp32 path of small catalogues (dense scores + one warp per user: history mask, radix select, rank
    sort) on a table whose rows repeat every 7 items and whose bias is zero: every score occurs ~n/7 times, so the
    K-th key is tied many times over and the list is decided by the tie rule alone -- (score desc, id asc), i.e. the
    lowest ids of each tied class, after the history mask.  Also as two row shards merged (virtual ranks), K = 50,
    and a catalogue whose row count is not a multiple of 4."""
    n = 1001                                                     # rows = 1002, not a multiple of 4
    sd = synth.make_state_dict(n, seed=3)
    tab = sd["embedding.token.weight"].clone()
    for r in range(n + 1):
        tab[r] = tab[r % 7]
    sd["embedding.token.weight"] = tab
    sd["model.bias"] = torch.zeros(n + 1)
    m = LRURec(_args(n))
    m.load_state_dict(sd)
    m = m.cuda().eval()
    cfg = synth.Config("ties", 64, n, 30, 64)
    ids, _ = synth.make_sequences(cfg, seed=9)
    for k in (20, 50):
        res = m.retrieve(ids.cuda(), k=k, exclude_history=True, precision="fp32")
        got_i, got_s = res["ids"].cpu().numpy(), res["scores"].cpu().numpy()
        raw = O.last_scores(ids, sd)                                          # [B, n+1] fp32 oracle scores
        canon = raw[:, torch.arange(n + 1) % 7]                               # one value per tied class (a CPU matmul may
        dense = O.mask_history(canon, ids).numpy()                            # round identical rows differently); history
        for b in range(ids.shape[0]):                                         # and item 0 at -1e9
            order = np.lexsort((np.arange(n + 1), -dense[b]))                 # score desc, id asc
            want = [int(i) for i in order[:k]]
            assert got_i[b].tolist() == want, (k, b, got_i[b][:8], want[:8])
            np.testing.assert_allclose(got_s[b], dense[b][want], rtol=1e-5, atol=1e-6)
    # the same through two row shards (row_offset != 0 in the second) merged like ranks would merge them
    full = m.retrieve(ids.cuda(), k=20, exclude_history=True, precision="fp32")
    parts_s, parts_i = [], []
    cut = 500
    for lo, hi in ((0, cut), (cut, n + 1)):
        m.set_row_shard(lo, hi)
        r = m.retrieve(ids.cuda(), k=20, exclude_history=True, precision="fp32")
        parts_s.append(r["scores"]); parts_i.append(r["ids"])
    m.set_row_shard(0, n + 1)
    merged = merge_lists(torch.stack(parts_s), torch.stack(parts_i), None, k_out=20, layout="list_major")
    assert torch.equal(merged["ids"], full["ids"]) and torch.equal(merged["scores"], full["scores"])


def test_demo_retriever_export_and_retrieve_candidates(tmp_path, model, golden_sd):
    """The demo's path (setup_demo.py:46-47, demo/inference.py:20-23,46-53): export the retriever, load it back on the
    GPU, `retrieve_candidates(model, history, top_k)` == topk of the oracle's last-position scores (no history mask)."""
    from llamarec_b200 import stage2
    path = str(tmp_path / "retriever.pth")
    stage2.export_retriever(model, path)
    loaded = stage2.load_retriever(path, device="cuda")
    rows = load_case("left_l20")["ids"]
    hist = next([int(v) for v in r if v > 0] for r in rows if (r > 0).sum() >= 3)   # (the fixture also has empty rows)
    with pytest.raises(ValueError):
        stage2.retrieve_candidates(loaded, [], top_k=5)
    got = stage2.retrieve_candidates(loaded, hist, top_k=20)
    x = torch.tensor(hist).unsqueeze(0)
    res = loaded.retrieve(x.cuda(), k=20, exclude_history=False)
    assert got == res["ids"][0].tolist()
    ref_s, ref_i = O.retrieve(x, golden_sd, 20, exclude_history=False)
    assert_topk_equivalent(res["ids"].cpu().numpy(), res["scores"].cpu().numpy(), ref_i.numpy(), ref_s.numpy())


def test_errors_are_loud():
    from llamarec_b200._lib import LrbError
    m = LRURec(_args(50)).cuda().eval()
    with pytest.raises(LrbError):
        m.retrieve(torch.ones(2, 300, dtype=torch.int64).cuda(), k=5)        # L > LRB_MAX_LEN
    with pytest.raises(LrbError):
        m.retrieve(torch.ones(2, 10, dtype=torch.int64).cuda(), k=64)        # K > LRB_MAX_K
    with pytest.raises(ValueError):
        LRURec(SimpleNamespace(num_items=10, bert_hidden_units=32, bert_num_blocks=2))
