"""precision="exact": the fp32 ranking from bf16 tensor-core candidates (DESIGN section 2.1).

* The bound: on the hardware, |bf16-operand score - fp32 score| <= eps_u for every item (lrb_score_dense precision
  0 against precision 1 on the same operands).
* The collect mode of the tensor-core kernel (lrb_score_collect) collects exactly {j : bf16 score >= tau_u}.
* retrieve(precision="exact") equals retrieve(precision="fp32") bit for bit in ids, scores and label ranks, on the
  fp32 dense + select path's range (131 073 rows), the fp32 streaming path's (600 000, 2 M), with and without the
  history mask and bias.  metric_sums are sums over users that lrb_merge_metrics adds with float atomics in block
  order, so two fp32 calls may differ in their last bits; they are compared to 1e-6 (label ranks, which fully
  determine them, bit for bit).
* exact_path reaches every branch: certified, collected, fp32 path.
"""
from types import SimpleNamespace

import pytest
import torch

from llamarec_b200 import LRURec, LRURetriever, _lib, merge_lists
from llamarec_b200.sharded import CudaBackend

pytestmark = pytest.mark.gpu

RHO = 2.0 ** -7 + 2.0 ** -12       # exact.cu
RHO_B = 2.0 ** -12


def _args(n_items):
    return SimpleNamespace(num_items=n_items, bert_hidden_units=64, bert_num_blocks=2, bert_dropout=0.0,
                           bert_attn_dropout=0.0, metric_ks=[1, 5, 10, 20, 50], num_users=1)


_MODELS = {}


def _model(rows, bias, seed=0):
    """Random-init LRURec (trunc-normal table) with `rows` rows, bias 0 or N(0, 0.01)."""
    key = (rows, bias, seed)
    if key not in _MODELS:
        _MODELS.clear()
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


def _seqs(B, rows, seed, L=20):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randint(1, rows, (B, L), device="cuda", generator=g)
    labels = torch.randint(1, rows, (B,), device="cuda", generator=g)
    return x, labels


def _eps64(u, bound):
    """eps_u in float64 (the kernel evaluates it rounding upwards, so its value is at least this)."""
    c = bound[:64].double()
    return RHO * (u.double().abs() * c).sum(1) + RHO_B * float(bound[64])


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


def _same(a, b, labels=None):
    assert torch.equal(a["ids"], b["ids"])
    assert torch.equal(a["scores"].view(torch.int32), b["scores"].view(torch.int32))
    if labels is not None:
        assert torch.equal(a["label_rank"], b["label_rank"])
        torch.testing.assert_close(a["metric_sums"], b["metric_sums"], rtol=1e-6, atol=0)


# ---------------------------------------------------------------------------------------------- the bound
@pytest.mark.parametrize("rows,shard,bias,B", [
    (5000, (0, 5000), False, 300),            # ragged last tile, no bias block
    (5000, (777, 5000), True, 300),           # row_offset != 0, bias block
    (131_100, (0, 131_100), True, 129),
    (600_000, (123_457, 600_000), False, 1),
])
def test_bound_holds_for_every_item(rows, shard, bias, B):
    m = _model(rows, bias)
    m.set_row_shard(*shard)
    try:
        g = torch.Generator(device="cuda").manual_seed(rows + B)
        u = torch.randn(B, 64, device="cuda", generator=g)
        u[0, 3] = 40.0                                                      # one large coordinate
        # values just above a bf16 rounding midpoint: they round up by almost half an ulp
        u[-1] = torch.where(torch.arange(64, device="cuda") % 2 == 0, 1.0 + 2.0 ** -8 + 2.0 ** -22, -0.75)
        s16 = _dense(m, u, 0).double()
        s32 = _dense(m, u, 1).double()
        eps = _eps64(u, m._prepare()["exact_bound"])
        ratio = ((s16 - s32).abs() / eps[:, None]).max().item()
        assert ratio <= 1.0, ratio
        print(f"rows={rows} shard={shard} bias={bias}: max |bf16 - fp32| / eps = {ratio:.3f}")
    finally:
        m.set_row_shard(0, rows)


# ---------------------------------------------------------------------------------------------- collect mode
@pytest.mark.parametrize("M", [1, 300, 20_000])      # one user tile; several; more tiles than SMs (shared streams)
@pytest.mark.parametrize("shard", [(0, 5000), (1234, 5000)])
def test_collect_matches_dense_threshold(M, shard):
    rows = 5000
    m = _model(rows, True)
    m.set_row_shard(*shard)
    try:
        lib = _lib.load()
        c = m._prepare()
        n = shard[1] - shard[0]
        g = torch.Generator(device="cuda").manual_seed(M)
        u = torch.randn(M, 64, device="cuda", generator=g)
        dense = _dense(m, u, 0)
        tau = dense.topk(min(40, n), dim=1).values[:, -1].contiguous()
        tau[::7] = float("inf")                                 # collects nothing
        over = 1 if M > 1 else 0
        tau[over] = -1e30                                       # every item: counts far past the cap
        cap = 256
        ids = torch.full((M, cap), -7, dtype=torch.int32, device="cuda")
        cnt = torch.empty(M, dtype=torch.int32, device="cuda")
        ub = u.to(torch.bfloat16).contiguous()
        _lib.check(lib.lrb_score_collect(_lib.ptr(ub), _lib.ptr(c["table_bf16"]), _lib.ptr(c["bias_blk"]), M, n,
                                         shard[0], _lib.ptr(tau), cap, _lib.ptr(ids), _lib.ptr(cnt),
                                         _lib.stream_handle()))
        want = dense >= tau[:, None]
        assert torch.equal(cnt.long(), want.sum(1))
        assert int(cnt[over]) == n and (M == 1 or n > cap)
        ids_h, cnt_h, want_h = ids.cpu(), cnt.cpu(), want.cpu()
        for b in range(M):
            k = int(cnt_h[b])
            got = ids_h[b, :min(k, cap)].long() - shard[0]
            assert (ids_h[b, min(k, cap):] == -7).all()
            if k <= cap:
                ref = torch.nonzero(want_h[b]).flatten()
                assert torch.equal(got.sort().values, ref), b
            else:
                assert got.unique().numel() == cap and bool(want_h[b][got].all())
    finally:
        m.set_row_shard(0, rows)


# ---------------------------------------------------------------------------------------------- exactness
@pytest.mark.parametrize("rows", [131_073, 600_000, 2_000_000])
@pytest.mark.parametrize("bias", [False, True])
def test_exact_equals_fp32(rows, bias):
    m = _model(rows, bias)
    seen = torch.zeros(3, dtype=torch.int64)
    for B in (1, 100, 4097):
        x, labels = _seqs(B, rows, seed=B + rows)
        for k in (1, 20, 50):
            ks = [kk for kk in (1, 5, 10, 20, 50) if kk <= k]
            for excl in (True, False):
                ex = m.retrieve(x, k=k, exclude_history=excl, labels=labels, ks=ks, precision="exact")
                ref = m.retrieve(x, k=k, exclude_history=excl, labels=labels, ks=ks, precision="fp32")
                _same(ex, ref, labels)
                assert ex["exact_path"].dtype == torch.int8 and ex["exact_path"].shape == (B,)
                seen += torch.bincount(ex["exact_path"].long().cpu(), minlength=3)
    print(f"rows={rows} bias={bias}: certified / collected / fp32 = {seen.tolist()}")
    if rows > 131_072:
        assert seen[0] > 0 and seen[1] > 0           # random weights: K = 20 certifies, K = 50 never can


def test_exact_packed_and_unmerged():
    rows = 600_000
    m = _model(rows, True)
    x, labels = _seqs(300, rows, seed=5)
    for layout, shape in (("planes", (2, 300, 20)), ("per_user", (300, 2, 20))):
        p_ex = torch.empty(shape, dtype=torch.int32, device="cuda")
        p_32 = torch.empty(shape, dtype=torch.int32, device="cuda")
        m.retrieve(x, k=20, packed_out=p_ex, packed_layout=layout, precision="exact")
        m.retrieve(x, k=20, packed_out=p_32, packed_layout=layout, precision="fp32")
        assert torch.equal(p_ex, p_32)
    part = m.retrieve(x, k=20, merge=False, precision="exact")
    assert part["part_scores"].shape == (300, 1, 20) and part["part_cnt"].shape == (300, 1)
    _same(merge_lists(part["part_scores"], part["part_ids"], part["part_cnt"], k_out=20),
          m.retrieve(x, k=20, precision="fp32"))


# ---------------------------------------------------------------------------------------------- every branch
def _planted(rows, kind, seed=3):
    """kind 'near_dup': 300 rows that are the same large positive vector up to ~1e-6 relative noise (every user with
    a positive state ranks them first, with gaps far below eps).  kind 'repeat': the table repeats 64 rows, so every
    score ties about rows / 64 times."""
    torch.manual_seed(seed)
    with torch.device("cuda"):
        m = LRURec(_args(rows - 1))
    g = torch.Generator(device="cuda").manual_seed(seed)
    w = m.embedding.token.weight
    with torch.no_grad():
        m.model.bias.zero_()
        if kind == "near_dup":
            base = torch.rand(64, device="cuda", generator=g) + 1.0
            w[1000:1300] = base * (1 + 1e-6 * torch.randn(300, 64, device="cuda", generator=g))
        else:
            v = torch.randn(64, 64, device="cuda", generator=g) * 0.05
            w.copy_(v[torch.arange(rows, device="cuda") % 64])
    return m.eval()


def test_near_duplicates_defeat_the_certificate():
    rows = 200_000
    m = _planted(rows, "near_dup")
    g = torch.Generator(device="cuda").manual_seed(1)
    u = torch.rand(130, 64, device="cuda", generator=g) + 0.1
    x = torch.randint(1, rows, (130, 20), device="cuda", generator=g)
    seq = m._prepare_sequences(x, all_positions=False, want_excl=True)
    for k in (1, 20):
        ex = m.retrieve(None, k=k, u=u, seq=seq, precision="exact")
        _same(ex, m.retrieve(None, k=k, u=u, seq=seq, precision="fp32"))
        assert (ex["exact_path"] == 1).all()
        assert (ex["exact_collected"] >= 300 - 20).all()
        # a cap below the collected count sends every user to the fp32 path
        small = m.retrieve(None, k=k, u=u, seq=seq, precision="exact", exact_cap=16)
        _same(small, ex)
        assert (small["exact_path"] == 2).all()


def test_repeated_rows_tie_order():
    rows = 140_000
    m = _planted(rows, "repeat")
    x, labels = _seqs(257, rows, seed=9)
    for excl in (True, False):
        ex = m.retrieve(x, k=50, exclude_history=excl, labels=labels, ks=[10, 50], precision="exact",
                        exact_cap=1 << 15)
        _same(ex, m.retrieve(x, k=50, exclude_history=excl, labels=labels, ks=[10, 50], precision="fp32"), labels)
        assert (ex["exact_path"] == 1).all()
        assert (ex["ids"][:, :-1] < ex["ids"][:, 1:]).any()        # ties resolved by ascending id


def test_nonfinite_goes_to_fp32():
    rows = 140_000
    m = _planted(rows, "repeat")
    x, _ = _seqs(64, rows, seed=11)
    u = m.encode(x)
    u[5, 0] = float("inf")
    seq = m._prepare_sequences(x, all_positions=False, want_excl=True)
    ex = m.retrieve(None, k=20, u=u, seq=seq, precision="exact")
    assert int(ex["exact_path"][5]) == 2
    ref = m.retrieve(None, k=20, u=u, seq=seq, precision="fp32")
    assert torch.equal(ex["ids"], ref["ids"])


# ---------------------------------------------------------------------------------------------- shards, retriever
def test_row_shards_merge_to_the_unsharded_result():
    rows = 600_000
    m = _model(rows, True)
    x, _ = _seqs(513, rows, seed=21)
    full = m.retrieve(x, k=20, precision="exact")
    _same(full, m.retrieve(x, k=20, precision="fp32"))
    lists_s, lists_i = [], []
    try:
        for lo, hi in ((0, 300_000), (300_000, rows)):
            m.set_row_shard(lo, hi)
            r = m.retrieve(x, k=20, precision="exact")
            assert (r["exact_path"] == 0).any()
            lists_s.append(r["scores"])
            lists_i.append(r["ids"])
    finally:
        m.set_row_shard(0, rows)
    merged = merge_lists(torch.stack(lists_s), torch.stack(lists_i), None, k_out=20, layout="list_major")
    _same(merged, full)


def test_retriever_precision_passthrough():
    rows = 600_000
    m = _model(rows, True)
    x, labels = _seqs(1000, rows, seed=31)
    args = _args(rows - 1)
    r_ex = LRURetriever(args, m, precision="exact").calculate_metrics((x, labels))
    r_32 = LRURetriever(args, m, precision="fp32").calculate_metrics((x, labels))
    assert list(r_ex) == list(r_32)
    for key in r_32:
        assert r_ex[key] == pytest.approx(r_32[key], rel=1e-6, abs=0), key


def test_refusals():
    rows = 200_000
    m = _model(rows, False)
    with pytest.raises(ValueError):
        CudaBackend(m, 0, 1, precision="exact")
    x, _ = _seqs(4, rows, seed=1)
    with pytest.raises(_lib.LrbError):
        m.retrieve(x, k=64, precision="exact")
