"""Top-K lists longer than 50 (k in [51, 1024], DESIGN section 2.2).

The reference is lrb_score_dense (precision 0 for the bf16 path, 1 for the fp32 path) in user chunks, the history
(and id 0) set to -inf when excluding, then torch.sort(descending=True, stable=True): (score desc, id asc).  Lists
must equal it bit for bit in ids and scores, where fewer than k items are admissible padded with (-inf, -1);
label ranks must equal it exactly and metric sums to 1e-6 relative.
"""
from types import SimpleNamespace

import pytest
import torch

from llamarec_b200 import LRURec, LRURetriever, _lib, merge_lists
from llamarec_b200.model import wide_policy
from llamarec_b200.sharded import CudaBackend

pytestmark = pytest.mark.gpu


def _args(n_items, metric_ks=(1, 5, 10, 20, 50)):
    return SimpleNamespace(num_items=n_items, bert_hidden_units=64, bert_num_blocks=2, bert_dropout=0.0,
                           bert_attn_dropout=0.0, metric_ks=list(metric_ks), num_users=1)


_MODELS = {}


def _model(rows, bias, seed=0):
    key = (rows, bias, seed)
    if key not in _MODELS:
        _MODELS.clear()
        torch.cuda.empty_cache()
        torch.manual_seed(seed)
        with torch.device("cuda"):
            m = LRURec(_args(rows - 1))
        with torch.no_grad():
            if bias:
                m.model.bias.normal_(0.0, 0.01)
            else:
                m.model.bias.zero_()
        _MODELS[key] = m.eval()
    return _MODELS[key]


def _inputs(B, rows, seed, L=20):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randint(1, rows, (B, L), device="cuda", generator=g)
    labels = torch.randint(1, rows, (B,), device="cuda", generator=g)
    u = torch.randn(B, 64, device="cuda", generator=g) * 4.0
    return x, labels, u


def _dense(m, u, precision):
    c = m._prepare()
    rows = m.row_end - m.row_begin
    out = torch.empty(u.shape[0], rows, dtype=torch.float32, device="cuda")
    lib = _lib.load()
    if precision == 0:
        x, tab, blk = u.to(torch.bfloat16).contiguous(), c["table_bf16"], c["bias_blk"]
    else:
        x, tab, blk = u.contiguous(), c["table_f32_shard"], None
    _lib.check(lib.lrb_score_dense(_lib.ptr(x), _lib.ptr(tab), _lib.ptr(c["bias_pad"]), _lib.ptr(blk), u.shape[0],
                                   rows, precision, _lib.ptr(out), rows, _lib.stream_handle()))
    return out


def _reference(m, u, x, k, precision, exclude, users=None, chunk=64):
    """(scores [n, k], ids [n, k]) of the reference ranking for the rows `users`, (-inf, -1) past the admissible items."""
    users = torch.arange(u.shape[0], device="cuda") if users is None else users
    rs, ri = [], []
    for i0 in range(0, users.numel(), chunk):
        us = users[i0:i0 + chunk]
        s = _dense(m, u[us], precision)
        if exclude:
            lo = m.row_begin
            h = torch.cat([x[us], torch.zeros(us.numel(), 1, dtype=x.dtype, device="cuda")], 1) - lo
            ok = (h >= 0) & (h < s.shape[1])
            rr = torch.arange(us.numel(), device="cuda")[:, None].expand_as(h)
            s[rr[ok], h[ok]] = float("-inf")
        ss, si = torch.sort(s, dim=1, descending=True, stable=True)
        ss, si = ss[:, :k].contiguous(), si[:, :k].to(torch.int32) + m.row_begin
        si[~(ss > float("-inf"))] = -1
        rs.append(ss)
        ri.append(si)
    return torch.cat(rs), torch.cat(ri)


def _check_lists(res, ref_s, ref_i, users=None):
    s, i = res["scores"], res["ids"]
    if users is not None:
        s, i = s[users], i[users]
    assert torch.equal(i, ref_i), (i != ref_i).sum().item()
    assert torch.equal(s.view(torch.int32), ref_s.view(torch.int32))


def _ref_metrics(ref_i, labels, ks):
    hit = ref_i == labels[:, None].to(torch.int32)
    rank = torch.where(hit.any(1), hit.int().argmax(1), torch.full_like(labels, -1)).to(torch.int32)
    sums = torch.zeros(len(ks), 3, dtype=torch.float64)
    for j, kk in enumerate(ks):
        r = rank[(rank >= 0) & (rank < kk)].double().cpu()
        sums[j] = torch.tensor([r.numel(), (1.0 / (r + 1)).sum(), (1.0 / torch.log2(r + 2)).sum()])
    return rank, sums


# ---------------------------------------------------------------------------------------------- collect with scores
@pytest.mark.parametrize("M", [1, 300, 20_000])
@pytest.mark.parametrize("shard", [(0, 5000), (1234, 5000)])
@pytest.mark.parametrize("bias", [False, True])
def test_collect_scores_match_dense(M, shard, bias):
    rows = 5000
    m = _model(rows, bias)
    m.set_row_shard(*shard)
    try:
        lib = _lib.load()
        c = m._prepare()
        n = shard[1] - shard[0]
        g = torch.Generator(device="cuda").manual_seed(M)
        u = torch.randn(M, 64, device="cuda", generator=g)
        dense = _dense(m, u, 0)
        q = torch.randint(50, 600, (M,), device="cuda", generator=g)
        tau = torch.sort(dense, 1, descending=True).values.gather(1, q[:, None]).flatten().contiguous()
        cap = 400
        ids = torch.full((M, cap), -7, dtype=torch.int32, device="cuda")
        scs = torch.empty(M, cap, dtype=torch.float32, device="cuda")
        cnt = torch.empty(M, dtype=torch.int32, device="cuda")
        ub = u.to(torch.bfloat16).contiguous()
        _lib.check(lib.lrb_score_collect_scores(_lib.ptr(ub), _lib.ptr(c["table_bf16"]), _lib.ptr(c["bias_blk"]), M,
                                                n, shard[0], _lib.ptr(tau), cap, _lib.ptr(ids), _lib.ptr(scs),
                                                _lib.ptr(cnt), _lib.stream_handle()))
        want = dense >= tau[:, None]
        assert torch.equal(cnt, want.sum(1, dtype=torch.int32))
        if M > 1:
            assert (cnt > cap).any() and (cnt <= cap).any()
        stored = torch.clamp(cnt, max=cap)
        for b in range(0, M, max(1, M // 97)):
            k = int(stored[b])
            got = ids[b, :k].long() - shard[0]
            assert got.unique().numel() == k
            assert bool(want[b, got].all())
            assert torch.equal(scs[b, :k].view(torch.int32), dense[b, got].view(torch.int32))
            if int(cnt[b]) <= cap:
                assert torch.equal(got.sort().values, torch.nonzero(want[b]).flatten())
    finally:
        m.set_row_shard(0, rows)


# ---------------------------------------------------------------------------------------------- lattice threshold
@pytest.mark.parametrize("r", [1, 3, 61])
@pytest.mark.parametrize("mm", [1, 20, 50])
@pytest.mark.parametrize("bias", [False, True])
def test_lattice_threshold(r, mm, bias):
    rows, shard, B = 20_011, (1001, 20_011), 300      # ragged last sample tile for every r
    m = _model(rows, bias)
    m.set_row_shard(*shard)
    try:
        lib = _lib.load()
        c = m._prepare()
        n = shard[1] - shard[0]
        x, _, u = _inputs(B, rows, r * 100 + mm, L=200)
        x[:, :100] = shard[0] + r * torch.arange(100, device="cuda")          # history on the lattice
        seq = m._prepare_sequences(x, all_positions=False, want_excl=True)
        ub = u.to(torch.bfloat16).contiguous()
        tau = torch.empty(B, dtype=torch.float32, device="cuda")
        ws_bytes = lib.lrb_wide_sample_workspace_bytes(B, n, seq["excl_stride"], r, mm)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        _lib.check(lib.lrb_wide_sample_threshold(_lib.ptr(ub), _lib.ptr(c["table_bf16"]), _lib.ptr(c["bias_blk"]), B,
                                                 n, shard[0], _lib.ptr(seq["excl_sorted"]), seq["excl_stride"], r, mm,
                                                 _lib.ptr(tau), _lib.ptr(ws), ws_bytes, _lib.stream_handle()))
        dense = _dense(m, u, 0)
        h = torch.cat([x, torch.zeros(B, 1, dtype=x.dtype, device="cuda")], 1) - shard[0]
        ok = (h >= 0) & (h < n)
        rr = torch.arange(B, device="cuda")[:, None].expand_as(h)
        dense[rr[ok], h[ok]] = float("-inf")
        lat = torch.sort(dense[:, ::r], 1, descending=True).values[:, mm - 1]
        assert torch.equal(tau.view(torch.int32), lat.view(torch.int32))
    finally:
        m.set_row_shard(0, rows)


# ---------------------------------------------------------------------------------------------- bf16 wide lists
CASES = [(1, 1024, True), (129, 51, False), (129, 256, True), (4097, 100, True), (4097, 1024, False)]


@pytest.mark.parametrize("rows", [131_073, 600_000, 2_000_000])
@pytest.mark.parametrize("bias", [False, True])
@pytest.mark.parametrize("B,k,hist", CASES)
def test_bf16_wide_equals_reference(rows, bias, B, k, hist):
    m = _model(rows, bias)
    x, labels, u = _inputs(B, rows, rows + B + k, L=50)
    ks = [1, 10, 50, k]
    res = m.retrieve(x, k=k, precision="bf16", u=u, exclude_history=hist, labels=labels, ks=ks)
    users = None if B <= 129 else torch.arange(0, B, 64, device="cuda")
    ref_s, ref_i = _reference(m, u, x, k, 0, hist, users)
    _check_lists(res, ref_s, ref_i, users)
    rank, sums = _ref_metrics(ref_i, labels if users is None else labels[users], ks)
    got_rank = res["label_rank"] if users is None else res["label_rank"][users]
    assert torch.equal(got_rank, rank)
    if users is None:
        torch.testing.assert_close(res["metric_sums"].double().cpu(), sums, rtol=1e-6, atol=0)
    p = torch.bincount(res["topk_path"].long(), minlength=3).tolist()
    print(f"rows={rows} bias={bias} B={B} k={k} hist={hist}: paths {p}, collected mean "
          f"{res['topk_collected'].float().mean().item():.0f} max {res['topk_collected'].max().item()}")


@pytest.mark.parametrize("k", [100, 1024])
def test_bf16_wide_10m(k):
    rows, B = 10_000_000, 512
    m = _model(rows, True)
    x, labels, u = _inputs(B, rows, k, L=50)
    res = m.retrieve(x, k=k, precision="bf16", u=u)
    users = torch.arange(0, B, 16, device="cuda")
    ref_s, ref_i = _reference(m, u, x, k, 0, True, users, chunk=8)
    _check_lists(res, ref_s, ref_i, users)


# ---------------------------------------------------------------------------------------------- every branch
def _plant(m, rows_idx, vecs):
    with torch.no_grad():
        m.embedding.token.weight[rows_idx] = vecs
    m._prepared_sig = None


def test_every_branch_reached():
    rows, B, k = 40_000, 129, 100
    m = _model(rows, False, seed=5)
    x, _, u = _inputs(B, rows, 7, L=50)
    u[:] = u[0]                                  # one direction for every user: planted rows rank the same for all
    v = u[0] / u[0].norm()
    m_s, r, _ = wide_policy(k, 52)
    seen = set()
    try:
        # default: path 0
        res = m.retrieve(x, k=k, precision="bf16", u=u)
        seen |= set(res["topk_path"].tolist())
        ref_s, ref_i = _reference(m, u, x, k, 0, True)
        _check_lists(res, ref_s, ref_i)
        # lattice rows planted high: tau above the k-th best -> short -> dense rows (path 2)
        idx = r * torch.arange(1, m_s + 1, device="cuda")
        _plant(m, idx, v[None] * (5.0 + torch.arange(m_s, 0, -1, device="cuda")[:, None].float()))
        res = m.retrieve(x, k=k, precision="bf16", u=u)
        short = (res["topk_path"] == 2) & (res["topk_collected"] < k)      # the first collect found < k items
        assert int(short.sum()) >= B - 10, int(short.sum())                # (a history may hit a planted row)
        seen |= set(res["topk_path"].tolist())
        ref_s, ref_i = _reference(m, u, x, k, 0, True)
        _check_lists(res, ref_s, ref_i)
        # repeated rows on a fresh table: 1200 rows tie at the top, 60 of them on the lattice, so tau is the tied
        # score; more than topk_cap = 500 items reach it, the retry at the k-th best stored score (the same tied
        # score) overflows again -> dense rows (path 2)
        _MODELS.clear()
        m = _model(rows, False, seed=5)
        idx = torch.arange(1000, 1000 + 1200, device="cuda")
        _plant(m, idx, v[None].expand(1200, 64) * 4.0)
        res = m.retrieve(x, k=k, precision="bf16", u=u, topk_cap=500)
        assert bool((res["topk_path"] == 2).all())
        assert bool((res["topk_collected"] > 500).all())                   # the retry's count, past the cap
        ref_s, ref_i = _reference(m, u, x, k, 0, True)
        _check_lists(res, ref_s, ref_i)
        seen |= set(res["topk_path"].tolist())
    finally:
        _MODELS.clear()
    # a small cap: overflow, then the k-th best stored score is a tight enough threshold (path 1)
    m = _model(rows, True, seed=6)
    x, _, u = _inputs(B, rows, 8, L=50)
    res = m.retrieve(x, k=60, precision="bf16", u=u, topk_cap=200)
    ref_s, ref_i = _reference(m, u, x, 60, 0, True)
    _check_lists(res, ref_s, ref_i)
    seen |= set(res["topk_path"].tolist())
    print("paths with topk_cap=200:", torch.bincount(res["topk_path"].long(), minlength=3).tolist())
    assert seen == {0, 1, 2}, seen
    # a history covering most of a small catalogue: padded lists, k <= rows
    rows, k = 300, 100
    m = _model(rows, True, seed=7)
    g = torch.Generator(device="cuda").manual_seed(3)
    x = torch.stack([torch.randperm(rows - 1, device="cuda", generator=g)[:250] + 1 for _ in range(5)])
    u = torch.randn(5, 64, device="cuda", generator=g)
    res = m.retrieve(x, k=k, precision="bf16", u=u)
    assert bool((res["topk_path"] == 2).all())
    ref_s, ref_i = _reference(m, u, x, k, 0, True)
    _check_lists(res, ref_s, ref_i)
    assert bool((res["ids"][:, 49:] == -1).all()) and bool(torch.isneginf(res["scores"][:, 49:]).all())


# ---------------------------------------------------------------------------------------------- fp32 wide lists
@pytest.mark.parametrize("rows,B,ks_", [(1683, 300, (51, 100, 1000, 1024)), (11_001, 2048, (100, 1024)),
                                         (500_000, 129, (100,))])
def test_fp32_wide_equals_reference(rows, B, ks_):
    m = _model(rows, True)
    x, labels, u = _inputs(B, rows, rows, L=50)
    for k in ks_:
        res = m.retrieve(x, k=k, precision="fp32", u=u, labels=labels, ks=[1, 10, k])
        users = None if B <= 300 else torch.arange(0, B, 8, device="cuda")
        ref_s, ref_i = _reference(m, u, x, k, 1, True, users)
        _check_lists(res, ref_s, ref_i, users)
        rank, _ = _ref_metrics(ref_i, labels if users is None else labels[users], [k])
        assert torch.equal(res["label_rank"] if users is None else res["label_rank"][users], rank)
    k50 = m.retrieve(x, k=50, precision="fp32", u=u)
    k100 = m.retrieve(x, k=100, precision="fp32", u=u)
    assert torch.equal(k100["ids"][:, :50], k50["ids"])
    assert torch.equal(k100["scores"][:, :50].view(torch.int32), k50["scores"].view(torch.int32))


def test_bf16_prefix_against_streaming_list():
    """The k = 50 list comes from the CTA-pair streaming kernel, the k = 100 list from single-CTA scores: compared
    with a float64 tolerance, and the count of bit-identical lists printed."""
    rows, B = 600_000, 1024
    m = _model(rows, True)
    x, _, u = _inputs(B, rows, 11, L=50)
    a = m.retrieve(x, k=50, precision="bf16", u=u)
    b = m.retrieve(x, k=100, precision="bf16", u=u)
    s50, s100 = a["scores"].double(), b["scores"][:, :50].double()
    tol = 2.0 ** -8 * u.double().abs().sum(1, keepdim=True) * m._prepare()["exact_bound"][:64].double().max()
    assert bool(((s50 - s100).abs() <= tol).all())
    same = (a["ids"] == b["ids"][:, :50]).all(1) & (a["scores"] == b["scores"][:, :50]).all(1)
    print(f"bit-identical k=50 prefixes: {int(same.sum())} of {B}")


# ---------------------------------------------------------------------------------------------- other features
def test_packed_merge_labels_ubf16_and_shards():
    rows, B = 300_000, 257
    m = _model(rows, True)
    x, labels, u = _inputs(B, rows, 21, L=50)
    ks = [1, 5, 10, 50, 100, 200, 500, 1024]
    full = m.retrieve(x, k=1024, precision="bf16", u=u, labels=labels, ks=ks)
    ref_s, ref_i = _reference(m, u, x, 1024, 0, True)
    _check_lists(full, ref_s, ref_i)
    rank, sums = _ref_metrics(ref_i, labels, ks)
    assert torch.equal(full["label_rank"], rank)
    torch.testing.assert_close(full["metric_sums"].double().cpu(), sums, rtol=1e-6, atol=0)
    # packed_out, merge=False, u_bf16 only (with a prepared seq)
    buf = torch.empty(2, B, 1024, dtype=torch.int32, device="cuda")
    m.retrieve(x, k=1024, precision="bf16", u=u, packed_out=buf)
    assert torch.equal(buf[1], full["ids"]) and torch.equal(buf[0], full["scores"].view(torch.int32))
    parts = m.retrieve(x, k=1024, precision="bf16", u=u, merge=False)
    mg = merge_lists(parts["part_scores"], parts["part_ids"], parts["part_cnt"], k_out=1024)
    assert torch.equal(mg["ids"], full["ids"])
    seq = m._prepare_sequences(x, all_positions=False, want_excl=True)
    r16 = m.retrieve(None, k=1024, precision="bf16", u_bf16=u.to(torch.bfloat16).contiguous(), seq=seq)
    assert torch.equal(r16["ids"], full["ids"])
    # two row shards on one device, merged like ranks
    for k in (100, 1024):
        want = m.retrieve(x, k=k, precision="bf16", u=u)
        lists_s, lists_i = [], []
        for sh in ((0, 140_001), (140_001, rows)):
            m.set_row_shard(*sh)
            r = m.retrieve(x, k=k, precision="bf16", u=u)
            lists_s.append(r["scores"])
            lists_i.append(r["ids"])
        m.set_row_shard(0, rows)
        mg = merge_lists(torch.stack(lists_s), torch.stack(lists_i), None, k_out=k, layout="list_major")
        assert torch.equal(mg["ids"], want["ids"])
        assert torch.equal(mg["scores"].view(torch.int32), want["scores"].view(torch.int32))


def test_retriever_metric_ks_beyond_50():
    rows, B = 1683, 400
    ks = [1, 5, 10, 20, 50, 100, 200]
    torch.manual_seed(0)
    with torch.device("cuda"):
        m = LRURec(_args(rows - 1, ks)).eval()
    r = LRURetriever(_args(rows - 1, ks), m)
    x, labels, _ = _inputs(B, rows, 5, L=50)
    got = r.calculate_metrics((x, labels.view(-1, 1)))
    u = m.encode(x)
    _, ref_i = _reference(m, u, x, 200, 1, True)
    _, sums = _ref_metrics(ref_i, labels, ks)
    for j, kk in enumerate(ks):
        assert abs(got["Recall@%d" % kk] - sums[j, 0].item() / B) < 1e-4
        assert abs(got["NDCG@%d" % kk] - sums[j, 2].item() / B) < 1e-4


# ---------------------------------------------------------------------------------------------- refusals
def test_refusals():
    m = _model(2000, False)
    x, _, u = _inputs(4, 2000, 1)
    with pytest.raises(_lib.LrbError):
        m.retrieve(x, k=1025, precision="fp32", u=u)
    with pytest.raises(_lib.LrbError):
        m.retrieve(x, k=1025, precision="bf16", u=u)
    small = _model(80, False)
    xs, _, us = _inputs(4, 80, 1)
    with pytest.raises(_lib.LrbError):
        small.retrieve(xs, k=81, precision="bf16", u=us)
    with pytest.raises(_lib.LrbError):
        small.retrieve(xs, k=81, precision="fp32", u=us)
    big = _model(600_000, False)
    xb, _, ub = _inputs(4, 600_000, 1)
    for prec in ("fp32", "exact"):
        with pytest.raises(ValueError, match="dense \\+ select"):
            big.retrieve(xb, k=51, precision=prec, u=ub)
    be = CudaBackend(big, 0, 1, precision="bf16")
    with pytest.raises(ValueError):
        be.local_topk_packed(xb, ub, 51, True)


# ---------------------------------------------------------------------------------------------- against the CPU oracle
# The golden C1 model (ML-100k shaped: 943 users x 1682 items, L = 200) and its sequences, as in test_gpu_configs.py;
# here the results for k > 50 are compared with the oracle's restatement of the reference model, not with a kernel.
@pytest.fixture(scope="module")
def c1():
    import os
    import pickle

    import numpy as np
    from conftest import GOLDEN
    from llamarec_b200 import synth

    with open(os.path.join(GOLDEN, "c1_ml100k_ref.pkl"), "rb") as f:
        ref = pickle.load(f)
    d = np.load(os.path.join(GOLDEN, "c1_ml100k_weights.npz"))
    sd = {k: torch.from_numpy(d[k]) for k in d.files}
    cfg = synth.CONFIGS["c1_ml100k"]
    splits = {}
    for name in ("val", "test"):
        ids, labels = synth.make_sequences(cfg, seed=42, split=name)
        assert int(ids.sum().item()) == ref[f"{name}_ids_sha"], "synthetic sequences differ from the fixture's"
        splits[name] = (ids, labels)
    _MODELS.clear()
    m = LRURec(_c1_args(cfg, ref["ks"]))
    m.load_state_dict(sd)
    return m.cuda().eval(), sd, ref, splits, cfg


def _c1_args(cfg, ks, neg=19):
    return SimpleNamespace(num_items=cfg.num_items, bert_hidden_units=64, bert_num_blocks=2, bert_dropout=0.2,
                           bert_attn_dropout=0.2, metric_ks=list(ks), llm_negative_sample_size=neg,
                           num_users=cfg.num_users)


def test_c1_golden_k200_against_oracle(c1):
    import numpy as np
    from oracle import lru_oracle as O
    from test_gpu_parity import assert_topk_equivalent

    m, sd, ref, splits, cfg = c1
    ids, _ = splits["test"]
    ref_s, ref_i = O.retrieve(ids, sd, 200)
    res = m.retrieve(ids.cuda(), k=200)                          # 'auto' on 1683 rows: fp32 dense + select
    got_i = res["ids"].cpu().numpy().astype(np.int64)
    got_s = res["scores"].cpu().numpy()
    np.testing.assert_allclose(got_s, ref_s.numpy(), atol=1e-5, rtol=1e-4)
    n_diff = assert_topk_equivalent(got_i, got_s, ref_i.numpy(), ref_s.numpy(), rtol=2e-6)
    assert n_diff <= len(got_i) // 100, n_diff
    ex = m.retrieve(ids.cuda(), k=200, precision="exact")       # "exact" is the same path at this size
    assert torch.equal(ex["ids"], res["ids"]) and torch.equal(ex["scores"], res["scores"])
    print(f"C1 k=200: {len(got_i) - n_diff} of {len(got_i)} lists identical to the oracle's")


def test_c1_generate_candidates_100_against_oracle(c1):
    """llm_negative_sample_size = 99: candidate lists of 100; metric_ks up to 200, so the ranked ids of the test
    users (200 per user) also go through the subset metrics."""
    import numpy as np
    from llamarec_b200 import DeviceEvalSet
    from oracle import lru_oracle as O
    from oracle import metrics_oracle as MO
    from test_gpu_parity import assert_topk_equivalent

    m, sd, ref, splits, cfg = c1
    ks = sorted(set(list(ref["ks"]) + [100, 200]))
    args = _c1_args(cfg, ks, neg=99)
    bs = ref["batch"]
    loaders = {name: DeviceEvalSet.from_tensors(ids, labels, batch_size=bs, device="cuda")
               for name, (ids, labels) in splits.items()}
    ours = LRURetriever(args, m, loaders["val"], loaders["test"]).generate_candidates()
    cpu = {name: [(ids[i:i + bs], labels[i:i + bs]) for i in range(0, ids.shape[0], bs)]
           for name, (ids, labels) in splits.items()}
    want = MO.generate_candidates(lambda s: O.last_scores(s, sd), cpu["val"], cpu["test"], args, ks)
    scores = {name: O.mask_history(O.last_scores(ids, sd), ids).numpy() for name, (ids, _) in splits.items()}
    for key in ("val_users", "test_users", "non_test_users", "test_labels"):
        assert ours[key] == want[key], key
    for key, split, users in (("val_candidates", "val", ours["val_users"]),
                              ("test_candidates", "test", ours["test_users"]),
                              ("test_probs", "test", list(range(1, cfg.num_users + 1)))):
        a, b = np.array(ours[key], dtype=np.int64), np.array(want[key], dtype=np.int64)
        assert a.shape == b.shape == (len(users), 100 if key != "test_probs" else 200), (key, a.shape, b.shape)
        sc = scores[split][np.array(users) - 1]
        s_a, s_b = np.take_along_axis(sc, a, 1), np.take_along_axis(sc, b, 1)
        n_diff = assert_topk_equivalent(a, s_a, b, s_b, rtol=2e-6)
        assert n_diff <= max(1, len(a) // 100), (key, n_diff)
    for key in ("val_metrics", "test_metrics"):
        for k, v in want[key].items():
            assert abs(ours[key][k] - v) < 5e-5, (key, k, ours[key][k], v)
    for key in ("retrieval_metrics", "non_retrieval_metrics"):
        for k, v in want["test_retrieval"][key].items():
            assert abs(ours["test_retrieval"][key][k] - v) < 5e-5, (key, k)
    assert ours["test_retrieval"]["retrieval_size"] == want["test_retrieval"]["retrieval_size"]


def test_c1_stage2_retrieve_candidates_beyond_50(c1):
    import numpy as np
    from llamarec_b200 import stage2
    from oracle import lru_oracle as O
    from test_gpu_parity import assert_topk_equivalent

    m, sd, ref, splits, cfg = c1
    ids, _ = splits["test"]
    for row in (0, 17, 500, 942):
        query = [int(t) for t in ids[row] if int(t) != 0]
        got = stage2.retrieve_candidates(m, query, top_k=128)
        seqs = torch.tensor(query, dtype=torch.int64)[None]
        ref_s, ref_i = O.retrieve(seqs, sd, 128, exclude_history=False)
        sc = O.last_scores(seqs, sd)[0].numpy()
        a = np.array([got], dtype=np.int64)
        assert a.shape == (1, 128)
        assert_topk_equivalent(a, sc[a], ref_i.numpy(), ref_s.numpy(), rtol=2e-6)
