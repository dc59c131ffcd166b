"""Top-K retrieval on every dispatch branch of lrb_score_topk, against a float64 reference.

lrb_score_topk picks one of about a dozen kernel configurations from (B, rows, K, precision): CTA pairs or single CTAs,
the number of full streams per user and whether a shared stream exists, the union bound's c and the scout pass, the
K <= 20 / 32 / 50 kernel variants (the longer lists keep no shared-memory copy of the exclusion list), user chunks of
one launch each, the merge's register or global-memory path, and on the exact-fp32 side the dense + select path (in
user blocks) or the streaming kernel.  Each case below names the branch it targets and asserts it through a Python
restatement of the host-side decomposition (score.cu); the CPU test pins that restatement to lrb_score_topk_slots.

Reference: plain torch float64 GEMMs (cuBLAS DGEMM) over the exact operands the kernel consumed -- the bf16 user
states and table upcast, or the fp32 ones -- plus the fp32 bias; -inf at every history id and at item 0 (global ids);
top K by (score desc, id asc).  Comparator, per user b, with tol_b = 128 * 2^-24 * max_n(sum_k |u_bk e_nk| + |bias_n|)
(twice the sequential fp32 bound for 64 products and the 16-wide folded-bias block; tensor-core accumulation rounding
is not documented as IEEE):
  * every returned id is in the shard's range, unique and admissible (not in the history, not 0 when excluded);
  * the list is sorted by (score desc, id asc) under the kernel's own scores;
  * |s_kernel - s64(id)| <= tol_b for every returned id;
  * every admissible id whose s64 exceeds the reference's K-th by more than 2 tol_b is returned, and no returned id
    lies more than 2 tol_b below it (any other difference is a swap inside the tie band);
  * (-inf, -1) entries appear exactly when fewer than K admissible items exist.

Inputs are seeded and built on the device.  Two regimes: "zero" (bias identically zero: no folded-bias block, pad
columns of the last tile score 0 while every real score is negative) and "bias" (a bias that dominates the dot
product, so an error in its hi/mid/lo bf16 split shows).  "Hot" items -- every user's highest scorers -- are planted
in the scouted tail of every full-stream segment and in the ragged last tile; every third user has a long history
holding them (with duplicates), so the exclusion list, the scout's count of excluded ids and the history mask all
decide the lists."""
import math
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from llamarec_b200 import LRURec, LRURetriever, _lib, merge_lists
from oracle import metrics_oracle as MO

# ------------------------------------------------------------------------------------------------
# Restatement of the host-side dispatch of lrb_score_topk (score.cu, score_topk_tc.cuh)
# ------------------------------------------------------------------------------------------------
BM, BN = 128, 256              # users per CTA tile, items per tile
SLOT_PARTS = 2                 # LRB_EW20 / 4: partial-list slots per stream
PARTS = 2                      # epilogue_warps_for(K) / 4 (8 epilogue warps for every K)
MAX_C_SMALL, MAX_C_LARGE = 6, 12
RESTART_TILES = 150.0          # LRB_RESTART_TILES
EX_CAP = 56                    # ints per row of the shared-memory exclusion copy
RING_BYTES_PER_SM = 512 * 24 * 80   # epilogue threads x RING_GROUPS x RING_REC_BYTES
MERGE_REG_ENTRIES = 32 * 32    # lrb_merge_metrics keeps up to 32 entries per lane in registers
F32_ROWS, F32_IT = 128, 64
SMS_WITHOUT_DEVICE = 148


def users_per_launch(B, sms):
    units = sms // 2 if sms >= 2 else 1
    cap = max(units, 1) * 2 * BM
    return min(B, cap)


def cta_group_for(B, sms):
    if os.environ.get("LRB_SCORE_CTA_GROUP", "") == "1":
        return 1
    return 2 if (B > BM and sms >= 2) else 1


def decompose(B, rows, units, bm):
    m_tiles = -(-B // bm)
    n_tiles = -(-rows // BN)
    G = max(1, min(m_tiles * n_tiles, units))
    s_full = G // m_tiles
    rem = G - s_full * m_tiles
    if s_full == 0:
        rem, y_tiles, full_tiles = G, n_tiles, 0
    elif rem == 0:
        y_tiles, full_tiles = 0, n_tiles
    else:
        R0 = RESTART_TILES
        if R0 > n_tiles / (8.0 * s_full):
            R0 = n_tiles / (8.0 * s_full)
        m_over_rem = m_tiles / rem
        y = (n_tiles / s_full + R0 * (0.5 - m_over_rem)) / (1.0 / s_full + m_over_rem)
        y_tiles = min(int(math.floor(max(y, 0.0) + 0.5)), n_tiles)
        if y_tiles <= 0:
            y_tiles, rem = 0, 0
        full_tiles = n_tiles - y_tiles
    slots = SLOT_PARTS * (s_full + (2 if rem > 0 else 0))
    return dict(m_tiles=m_tiles, n_tiles=n_tiles, s_full=s_full, rem=rem, y_tiles=y_tiles, full_tiles=full_tiles,
                slots=slots)


def bf16_plan(B, rows, K, sms, L=None):
    """One dict per chunk launch: decomposition, c / c_share, scout tiles and the kernel variant (KMAX, CMAX)."""
    cap = users_per_launch(B, sms)
    chunks = []
    for c0 in range(0, B, cap):
        Bc = min(cap, B - c0)
        cg = cta_group_for(Bc, sms)
        d = decompose(Bc, rows, sms // cg, BM * cg)
        c = -(-K // (PARTS * d["s_full"])) if d["s_full"] > 0 else 99
        c_max = MAX_C_LARGE if (cg == 2 and K <= 20) else MAX_C_SMALL
        c_share = c if c <= c_max else 0
        seg = d["full_tiles"] // d["s_full"] if d["s_full"] > 0 else 0
        scout = (32 if seg >= 512 else 16) if (c_share > 0 and seg >= 128) else 0
        kmax = 20 if K <= 20 else (32 if K <= 32 else 50)
        cmax = MAX_C_LARGE if (cg == 2 and K <= 20 and c_share > MAX_C_SMALL) else MAX_C_SMALL
        d.update(c0=c0, B=Bc, cg=cg, c=c, c_share=c_share, scout=scout, kmax=kmax, cmax=cmax)
        if L is not None:
            stride = ((L + 1) + 3) & ~3
            d["excl_in_smem"] = kmax <= 20 and stride <= EX_CAP
        chunks.append(d)
    return chunks


def bf16_slots(B, rows, sms):
    return max(ch["slots"] for ch in bf16_plan(B, rows, 1, sms))


def f32_select_users(rows, sms):
    ld = (rows + 3) // 4 * 4
    return (2 * sms * RING_BYTES_PER_SM) // (ld * 4) // F32_ROWS * F32_ROWS


def f32_splits(B, rows, sms, ctas_per_sm=2):
    m_tiles = -(-B // F32_ROWS)
    chunks = -(-rows // F32_IT)
    want = (ctas_per_sm * sms + m_tiles - 1) // m_tiles
    max_splits = max(1, (chunks + 3) // 4)
    return max(1, min(want, max_splits, 1024))


def lib_slots(B, rows, precision):
    lib = _lib.load()
    s = _lib.c_int(0)
    _lib.check(lib.lrb_score_topk_slots(B, rows, precision, _lib.ctypes.byref(s)))
    return s.value


def _library_sms():
    # what the library uses: the current device's SM count, 148 without a device
    return torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else SMS_WITHOUT_DEVICE


def test_dispatch_restatement_matches_the_library():
    """The restated decomposition gives lrb_score_topk_slots' slot counts on a grid of shapes; the fp32 select path
    (one sorted list per user) applies exactly where the restatement says."""
    sms = _library_sms()
    Bs = [1, 2, 37, 100, 128, 129, 200, 255, 256, 257, 300, 1000, 2048, 4096, 9472, 9473, 18944, 18945, 19244, 40000]
    rows_list = [46, 256, 401, 11001, 70164, 200003, 300001, 500000, 570000, 600001, 1250001, 3000001, 10000001]
    for B in Bs:
        for rows in rows_list:
            assert lib_slots(B, rows, 0) == bf16_slots(B, rows, sms), (B, rows)
            sel = f32_select_users(rows, sms) > 0
            got = lib_slots(B, rows, 1)
            assert got == (1 if sel else f32_splits(B, rows, sms)), (B, rows)
            if -(-B // F32_ROWS) < 2 * sms and rows > 4 * F32_IT:   # the streaming kernel then has > 1 item split
                assert (got == 1) == sel, (B, rows)
    # the shapes the GPU cases rely on (148 SMs)
    if sms == 148:
        assert f32_select_users(500_000, sms) == 128 and f32_select_users(600_001, sms) == 0
        assert f32_select_users(570_000, sms) == 0 and f32_select_users(30_001, sms) > 0


# ------------------------------------------------------------------------------------------------
# float64 reference and comparator
# ------------------------------------------------------------------------------------------------
TOL_C = 128.0
NEG_INF = float("-inf")


def _select(s, i, K):
    """top K by (score desc, id asc)"""
    o = torch.argsort(i, dim=1, stable=True)
    s, i = s.gather(1, o), i.gather(1, o)
    o = torch.argsort(-s, dim=1, stable=True)
    return s.gather(1, o)[:, :K], i.gather(1, o)[:, :K]


@torch.no_grad()
def fp64_reference(table, bias, row_begin, U, hist, exclude, K, query):
    """table [rows, 64] (bf16 or fp32, the shard the kernel scored), bias [rows] fp32, U [n, 64] the user states the
    kernel consumed, hist [n, L] global ids, query [n, Q] global ids (-1 = none).
    -> ref_s, ref_i [n, K] (fp64 top K), tol [n], s64 at the query ids [n, Q] (history not masked), admissible count."""
    dev = U.device
    n, rows = U.shape[0], table.shape[0]
    U = U.double()
    Ua = U.abs()
    rc = min(rows, 1 << 20)
    bc = max(1, min(n, (1 << 27) // rc))               # <= 1 GiB per [users x rows] fp64 block
    best_s = torch.full((n, K), NEG_INF, dtype=torch.float64, device=dev)
    best_i = torch.full((n, K), 1 << 62, dtype=torch.int64, device=dev)
    absmax = torch.zeros(n, dtype=torch.float64, device=dev)
    s_q = torch.full(query.shape, float("nan"), dtype=torch.float64, device=dev)
    query = query.long()
    h = torch.cat([hist.long(), torch.zeros(n, 1, dtype=torch.int64, device=dev)], 1) if exclude else None
    for r0 in range(0, rows, rc):
        r1 = min(rows, r0 + rc)
        E = table[r0:r1].double()
        Ea = E.abs()
        bb = bias[r0:r1].double()
        for b0 in range(0, n, bc):
            b1 = min(n, b0 + bc)
            A = torch.addmm(bb.abs(), Ua[b0:b1], Ea.t())
            absmax[b0:b1] = torch.maximum(absmax[b0:b1], A.amax(1))
            del A
            S = torch.addmm(bb, U[b0:b1], E.t())
            q = query[b0:b1] - row_begin - r0
            ok = (query[b0:b1] >= 0) & (q >= 0) & (q < r1 - r0)
            s_q[b0:b1] = torch.where(ok, S.gather(1, q.clamp(0, r1 - r0 - 1)), s_q[b0:b1])
            if exclude:
                loc = h[b0:b1] - row_begin - r0
                okh = (loc >= 0) & (loc < r1 - r0)
                rr = torch.arange(b1 - b0, device=dev).view(-1, 1).expand_as(loc)
                S[rr[okh], loc[okh]] = NEG_INF
            v, i = S.topk(min(K, r1 - r0), dim=1)
            del S
            best_s[b0:b1], best_i[b0:b1] = _select(torch.cat([best_s[b0:b1], v], 1),
                                                   torch.cat([best_i[b0:b1], i + row_begin + r0], 1), K)
    if exclude:
        hs = h.sort(dim=1).values
        first = torch.ones_like(hs, dtype=torch.bool)
        first[:, 1:] = hs[:, 1:] != hs[:, :-1]
        n_excl = (first & (hs >= row_begin) & (hs < row_begin + rows)).sum(1)
    else:
        n_excl = torch.zeros(n, dtype=torch.int64, device=dev)
    tol = TOL_C * 2.0 ** -24 * absmax
    return best_s, best_i, tol, s_q, rows - n_excl


def check_topk(name, got_s, got_i, ref_s, ref_i, tol, s64, n_adm, hist, exclude, row_begin, row_end):
    """The comparator of the module docstring; returns the largest |s_kernel - s64| / tol_b."""
    n, K = got_i.shape
    dev = got_i.device
    got_s, got_i = got_s.double(), got_i.long()
    n_valid = torch.clamp(n_adm, max=K)
    pos = torch.arange(K, device=dev).view(1, -1)
    valid = pos < n_valid.view(-1, 1)

    def fail(mask, what):
        bad = mask.any(1) if mask.dim() == 2 else mask
        if bool(bad.any()):
            b = int(bad.nonzero()[0])
            raise AssertionError(f"{name}: {what} for {int(bad.sum())} of {n} users; first: user {b}, "
                                 f"ids {got_i[b, :12].tolist()}, scores {got_s[b, :6].tolist()}, "
                                 f"ref ids {ref_i[b, :12].tolist()}, ref {ref_s[b, :6].tolist()}, tol {float(tol[b]):.3e}")

    fail(~valid & ((got_i != -1) | (got_s != NEG_INF)), "entries beyond the admissible count are not (-inf, -1)")
    fail(valid & ((got_i < row_begin) | (got_i >= row_end) | ~torch.isfinite(got_s)), "id out of range or score not finite")
    si = torch.where(valid, got_i, torch.full_like(got_i, -1)).sort(1).values
    fail((si[:, 1:] == si[:, :-1]) & (si[:, 1:] >= 0), "duplicate id")
    if exclude:
        in_hist = (got_i.unsqueeze(2) == hist.long().unsqueeze(1)).any(2) | (got_i == 0)
        fail(valid & in_hist, "history id or item 0 returned")
    both = valid[:, 1:]
    ordered = (got_s[:, :-1] > got_s[:, 1:]) | ((got_s[:, :-1] == got_s[:, 1:]) & (got_i[:, :-1] < got_i[:, 1:]))
    fail(both & ~ordered, "list not sorted by (score desc, id asc)")
    err = torch.where(valid, (got_s - s64).abs(), torch.zeros_like(got_s))
    fail(valid & ~(err <= tol.view(-1, 1)), "kernel score differs from the fp64 score by more than tol")
    has = n_valid > 0
    kth = ref_s.gather(1, (n_valid - 1).clamp(min=0).view(-1, 1)).view(-1)
    kth = torch.where(has, kth, torch.full_like(kth, float("inf")))
    must = (ref_s > (kth + 2 * tol).view(-1, 1)) & (pos < n_valid.view(-1, 1))
    found = (ref_i.unsqueeze(2) == got_i.unsqueeze(1)).any(2)
    fail(must & ~found, "an id clearly inside the fp64 top K is missing")
    fail(valid & (s64 < (kth - 2 * tol).view(-1, 1)), "a returned id lies clearly below the fp64 K-th score")
    fail(~torch.isfinite(ref_s) & (pos < n_valid.view(-1, 1)), "reference has fewer admissible items than counted")
    ratio = float((err / tol.view(-1, 1)).max()) if n else 0.0
    print(f"[topk] {name}: {n} users, K={K}, max |err|/tol = {ratio:.4f}")
    RATIOS[name] = ratio
    return ratio


RATIOS = {}


# ------------------------------------------------------------------------------------------------
# Inputs
# ------------------------------------------------------------------------------------------------
def _args(n):
    return SimpleNamespace(num_items=n, bert_hidden_units=64, bert_num_blocks=2, bert_dropout=0.2,
                           bert_attn_dropout=0.2, metric_ks=[1, 5, 10, 20, 50], llm_negative_sample_size=19)


def _hot_ids(rows, seg_plan, seed):
    """Ids planted as every user's best items: the scouted tail of every full-stream segment of `seg_plan` (items in
    distinct 16-item groups of all four 64-column quarters of the tail's first and last tile) and the ragged last
    tile.  Without a plan: spread over the table."""
    rng = np.random.default_rng(seed)
    n_tiles = -(-rows // BN)
    out = []
    if seg_plan is not None and seg_plan["s_full"] > 0:
        s_full, full = seg_plan["s_full"], seg_plan["full_tiles"]
        T = seg_plan["scout"] or 16
        per_tail = max(1, min(16, 160 // s_full))
        for s in range(s_full):
            n1 = (s + 1) * full // s_full
            for i in range(per_tail):
                tile = n1 - 1 if i % 2 == 0 else max(n1 - T, 0)
                col = ((i // 2) % 4) * 64 + (i // 8) * 16 + int(rng.integers(0, 16))
                out.append(tile * BN + col)
    else:
        out.extend(rng.integers(1, rows, size=150).tolist())
    last0 = (n_tiles - 1) * BN
    out.extend(last0 + rng.choice(np.arange(rows - last0), size=min(8, rows - last0), replace=False))
    hot = np.unique(np.asarray(out, dtype=np.int64))
    return hot[(hot > 0) & (hot < rows)]


def _histories(B, L, hot, rows, seed):
    """Left-padded ids [B, L]: every third user holds (up to L - 12 of) the hot items, six of them twice, and six
    random ids; the others hold 1..10 ids, some of them hot."""
    rng = np.random.default_rng(seed)
    ids = np.zeros((B, L), dtype=np.int64)
    for b in range(B):
        if b % 3 == 0:
            h = rng.permutation(hot)[: max(1, min(len(hot), L - 12))]
            seq = np.concatenate([h, h[:6], rng.integers(1, rows, size=6)])[:L]
            rng.shuffle(seq)
        else:
            n = int(rng.integers(1, 11))
            seq = rng.integers(1, rows, size=n)
            seq[: min(2, n)] = rng.choice(hot, size=min(2, n))
        ids[b, L - len(seq):] = seq
    return torch.from_numpy(ids)


def _trunc_normal_(t, g, std=0.02):
    a = (1.0 + math.erf(-2.0 / math.sqrt(2.0))) / 2.0
    b = (1.0 + math.erf(2.0 / math.sqrt(2.0))) / 2.0
    t.uniform_(2 * a - 1, 2 * b - 1, generator=g).erfinv_().mul_(std * math.sqrt(2.0))


class World:
    """A model on the device whose item table and bias follow `regime`, with hot items planted."""

    def __init__(self, rows, regime, seg_plan, seed):
        torch.manual_seed(seed)
        with torch.device("cuda"):
            m = LRURec(_args(rows - 1))
        self.rows, self.regime = rows, regime
        self.hot = _hot_ids(rows, seg_plan, seed)
        hot = torch.from_numpy(self.hot).cuda()
        g = torch.Generator(device="cuda").manual_seed(seed)
        w, bias = m.embedding.token.weight, m.model.bias
        with torch.no_grad():
            if regime == "zero":
                # positive rows, negative user states: every real score < 0 = the score of a zero-filled pad column
                w.uniform_(0.01, 0.02, generator=g)
                w[hot] = torch.rand(len(hot), 64, device="cuda", generator=g) * 0.008 + 0.001
                bias.zero_()
            else:
                _trunc_normal_(w, g)
                bias.normal_(0.0, 1.0, generator=g)
                bias[hot] = 6.0 + torch.rand(len(hot), device="cuda", generator=g)
        self.model = m.eval()

    def users(self, B, seed):
        g = torch.Generator(device="cuda").manual_seed(seed)
        u = torch.rand(B, 64, device="cuda", generator=g)
        return -(u + 0.5) if self.regime == "zero" else torch.randn(B, 64, device="cuda", generator=g)

    def run(self, x, u, K, precision, exclude=True):
        if precision == "bf16":
            return self.model.retrieve(x, k=K, exclude_history=exclude, precision="bf16", u_bf16=u.to(torch.bfloat16))
        return self.model.retrieve(x, k=K, exclude_history=exclude, precision="fp32", u=u)

    def reference(self, x, u, K, precision, query, exclude=True):
        c = self.model._prepare()
        m = self.model
        if precision == "bf16":
            table, U = c["table_bf16"], u.to(torch.bfloat16)
        else:
            table, U = c["table_f32_shard"], u
        bias = m.model.bias.detach()[m.row_begin:m.row_end]
        return fp64_reference(table, bias, m.row_begin, U, x, exclude, K, query)

    def check(self, name, x, u, res, K, precision, exclude=True, sel=None):
        got_s, got_i = res["scores"], res["ids"]
        if sel is not None:
            x, u, got_s, got_i = x[sel], u[sel], got_s[sel], got_i[sel]
        ref_s, ref_i, tol, s64, n_adm = self.reference(x, u, K, precision, got_i, exclude)
        m = self.model
        return check_topk(name, got_s, got_i, ref_s, ref_i, tol, s64, n_adm, x, exclude, m.row_begin, m.row_end)


@pytest.fixture(scope="module")
def worlds():
    """One World at a time: asking for another frees the previous table."""
    cache = {}

    def get(key, build):
        if key not in cache:
            cache.clear()
            torch.cuda.empty_cache()
            cache[key] = build()
        return cache[key]
    torch.cuda.reset_peak_memory_stats()
    yield get
    cache.clear()
    torch.cuda.empty_cache()
    print(f"[topk] peak device memory {torch.cuda.max_memory_allocated() / 2**30:.2f} GiB; max |err|/tol per case: "
          + ", ".join(f"{k}={v:.3f}" for k, v in RATIOS.items()))


def _need_148():
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if sms != 148:
        pytest.skip(f"the cases target the dispatch of a 148-SM B200; this device has {sms} SMs")
    return sms


def _assert_bf16_branch(B, rows, K, L, **want):
    """Every key of `want` must match the restated plan of the first chunk (or `chunks`: the list of all chunks)."""
    sms = _need_148()
    plan = bf16_plan(B, rows, K, sms, L)
    assert lib_slots(B, rows, 0) == max(ch["slots"] for ch in plan)
    chunks = want.pop("chunks", None)
    if chunks is not None:
        assert len(plan) == len(chunks)
        for ch, w in zip(plan, chunks):
            for k, v in w.items():
                assert ch[k] == v, (k, ch[k], v)
    for k, v in want.items():
        assert plan[0][k] == v, (k, plan[0][k], v)
    return plan


def _world_300k(worlds, regime):
    rows = 300_001
    return worlds(("300k", regime), lambda: World(rows, regime, bf16_plan(2048, rows, 50, 148)[0], seed=11))


# ------------------------------------------------------------------------------------------------
# bf16 tensor-core cases
# ------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("regime", ["zero", "bias"])
def test_cta_pairs_union_bound_scout_and_global_exclusion(worlds, regime):
    """2048 users x 300,001 rows, L = 200: CTA pairs, 9 full streams plus a shared stream, union bound with c = 3 / 2,
    scout 16, exclusion lists too long for shared memory; K = 50, 33, 21 (the K <= 50 and K <= 32 kernels); and the
    same shape without exclusion (item 0 and history items compete)."""
    B, rows, L = 2048, 300_001, 200
    for K, c, kmax in ((50, 3, 50), (33, 2, 50), (21, 2, 32)):
        plan = _assert_bf16_branch(B, rows, K, L, cg=2, s_full=9, c_share=c, scout=16, kmax=kmax, excl_in_smem=False)
        assert plan[0]["rem"] > 0 and plan[0]["y_tiles"] > 0          # a shared stream
    w = _world_300k(worlds, regime)
    x = _histories(B, L, w.hot, rows, seed=1).cuda()
    u = w.users(B, seed=2)
    for K in (50, 33, 21):
        w.check(f"pairs_{regime}_K{K}", x, u, w.run(x, u, K, "bf16"), K, "bf16")
    w.check(f"pairs_{regime}_noexcl", x, u, w.run(x, u, 50, "bf16", exclude=False), 50, "bf16", exclude=False)


@pytest.mark.gpu
def test_calculate_metrics_end_to_end_against_fp64(worlds):
    """LRURetriever.calculate_metrics with the default metric_ks (K = 50) on 2048 users x 300,001 rows with user
    states from the encoder: label ranks and Recall/MRR/NDCG against metrics_oracle on the fp64 scores."""
    B, rows, L = 2048, 300_001, 200
    _assert_bf16_branch(B, rows, 50, L, cg=2, s_full=9, c_share=3, scout=16)
    w = _world_300k(worlds, "bias")
    m = w.model
    x = _histories(B, L, w.hot, rows, seed=3).cuda()
    u, u16 = m.encode(x, want_bf16=True)
    ref_s, ref_i, tol, _, _ = w.reference(x, u, 50, "bf16", torch.full((B, 1), -1, device="cuda"))
    # half the labels inside the fp64 top 50 (at every rank), the rest random
    g = torch.Generator().manual_seed(4)
    ar = torch.arange(B, device="cuda")
    pick = ref_i[ar, ar % 50]
    labels = torch.where(ar % 2 == 0, pick,
                         torch.randint(1, rows, (B,), generator=g).cuda())
    _, _, _, s_lab, _ = w.reference(x, u, 1, "bf16", labels.view(-1, 1))
    tr = LRURetriever(_args(rows - 1), m)
    ks = tr.metric_ks
    assert ks == [1, 5, 10, 20, 50]
    got = tr.calculate_metrics((x, labels.view(-1, 1)))
    rank = m.retrieve(x, k=50, labels=labels, ks=ks)["label_rank"].long()
    # oracle on the compact fp64 rows: the top 50 plus the label (only the label's position matters)
    in_top = ref_i == labels.view(-1, 1)
    extra = torch.where(in_top.any(1, keepdim=True), torch.full_like(s_lab, NEG_INF), s_lab)
    hist_hit = (x == labels.view(-1, 1)).any(1, keepdim=True)
    extra = torch.where(hist_hit, torch.full_like(extra, NEG_INF), extra)
    scores = torch.cat([ref_s, extra], 1).cpu()
    lab_col = torch.where(in_top.any(1), in_top.float().argmax(1), torch.full((B,), 50, device="cuda")).cpu()
    want = MO.recall_mrr_ndcg(scores, lab_col, ks)
    for k, v in want.items():
        assert abs(got[k] - v) < 5e-5, (k, got[k], v)
    pos = (-scores).argsort(1).eq(lab_col.view(-1, 1)).float().argmax(1)
    want_rank = torch.where(pos < 50, pos, torch.full_like(pos, -1)).cuda()
    for b in (rank != want_rank).nonzero().view(-1).tolist():       # only swaps inside the tie band
        lo, hi = sorted(int(r) if r >= 0 else 50 for r in (rank[b], want_rank[b]))
        band = ref_s[b, lo:min(hi, 49) + 1]
        assert bool(((band - s_lab[b, 0]).abs() <= 2 * tol[b]).all()), (b, int(rank[b]), int(want_rank[b]))
    assert int((rank >= 0).sum()) >= B // 2


@pytest.mark.gpu
def test_union_bound_off_with_a_shared_stream(worlds):
    """4096 users x 1,250,001 rows, K = 50: c = ceil(50 / 8) = 7 > 6, so the union bound (and the scout) are off."""
    B, rows, K, L = 4096, 1_250_001, 50, 200
    plan = _assert_bf16_branch(B, rows, K, L, cg=2, s_full=4, c=7, c_share=0, scout=0, kmax=50)
    assert plan[0]["rem"] > 0 and plan[0]["y_tiles"] > 0
    w = worlds(("1.25M", "bias"), lambda: World(rows, "bias", plan[0], seed=21))
    x = _histories(B, L, w.hot, rows, seed=5).cuda()
    u = w.users(B, seed=6)
    w.check("no_union_bound_K50", x, u, w.run(x, u, K, "bf16"), K, "bf16")


def _world_3m(worlds):
    rows = 3_000_001
    return worlds(("3M", "zero"), lambda: World(rows, "zero", bf16_plan(300, rows, 50, 148)[0], seed=31))


@pytest.mark.gpu
@pytest.mark.parametrize("K", [32, 50])
def test_many_full_streams_ragged_last_pair_tile(worlds, K):
    """300 users x 3,000,001 rows: 37 full streams (no shared stream), c = 1, scout 16; the second pair tile holds
    256 + 44 users."""
    B, rows, L = 300, 3_000_001, 200
    plan = _assert_bf16_branch(B, rows, K, L, cg=2, m_tiles=2, s_full=37, rem=0, c_share=1, scout=16)
    assert B - 256 == 44 and plan[0]["kmax"] == (32 if K == 32 else 50)
    w = _world_3m(worlds)
    x = _histories(B, L, w.hot, rows, seed=7).cuda()
    u = w.users(B, seed=8)
    w.check(f"37_streams_K{K}", x, u, w.run(x, u, K, "bf16"), K, "bf16")


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 20, 50])
def test_single_ctas_148_streams_and_296_lists(worlds, K):
    """100 users x 3,000,001 rows: single CTAs, 148 streams per user, 296 partial lists; the merge runs from global
    memory (296 K > 1024 entries) for K = 20, 50 and from registers for K = 1."""
    B, rows, L = 100, 3_000_001, 50
    plan = _assert_bf16_branch(B, rows, K, L, cg=1, s_full=148, rem=0, slots=296, c_share=1)
    assert (296 * K > MERGE_REG_ENTRIES) == (K >= 20)
    assert plan[0]["excl_in_smem"] == (K <= 20)
    w = _world_3m(worlds)
    x = _histories(B, L, w.hot, rows, seed=9).cuda()
    u = w.users(B, seed=10)
    w.check(f"single_cta_K{K}", x, u, w.run(x, u, K, "bf16"), K, "bf16")


@pytest.mark.gpu
@pytest.mark.parametrize("K", [20, 50])
def test_one_user_on_ten_million_items(worlds, K):
    """The demo's shape: one user x 10,000,001 rows, single CTAs, 148 streams, scout 16."""
    B, rows, L = 1, 10_000_001, 50
    _assert_bf16_branch(B, rows, K, L, cg=1, s_full=148, rem=0, c_share=1, scout=16)
    w = worlds(("10M", "bias"), lambda: World(rows, "bias", bf16_plan(1, rows, 20, 148)[0], seed=41))
    for long_history in (True, False):
        x = _histories(3, L, w.hot, rows, seed=11)[0 if long_history else 1:][:1].cuda()
        u = w.users(1, seed=12)
        w.check(f"demo_K{K}_{'long' if long_history else 'short'}", x, u, w.run(x, u, K, "bf16"), K, "bf16")


def _world_200k(worlds):
    rows = 200_003
    return worlds(("200k", "zero"), lambda: World(rows, "zero", bf16_plan(18944, rows, 20, 148)[0], seed=51))


@pytest.mark.gpu
def test_cmax12_variant_one_stream_per_user(worlds):
    """18,944 users x 200,003 rows, K = 20: one launch of 74 pair tiles, one full stream per user, c = 10 (the CMAX = 12
    kernel), scout 32.  512 users sampled across all 74 pair tiles."""
    B, rows, K, L = 18944, 200_003, 20, 50
    _assert_bf16_branch(B, rows, K, L, cg=2, m_tiles=74, s_full=1, rem=0, c_share=10, cmax=12, scout=32)
    w = _world_200k(worlds)
    x = _histories(B, L, w.hot, rows, seed=13).cuda()
    u = w.users(B, seed=14)
    sel = torch.arange(0, B, 37, device="cuda")
    assert len(sel) == 512 and len(torch.unique(sel // 256)) == 74
    w.check("cmax12_K20", x, u, w.run(x, u, K, "bf16"), K, "bf16", sel=sel)


@pytest.mark.gpu
def test_two_chunk_launches(worlds):
    """19,244 users x 200,003 rows, K = 50: a launch of 18,944 users without union bound (c = 25), then one of 300 users
    with c = 1."""
    B, rows, K, L = 19244, 200_003, 50, 50
    _assert_bf16_branch(B, rows, K, L, chunks=[dict(B=18944, s_full=1, c_share=0),
                                               dict(B=300, s_full=37, c_share=1, scout=0)])
    w = _world_200k(worlds)
    x = _histories(B, L, w.hot, rows, seed=15).cuda()
    u = w.users(B, seed=16)
    sel = torch.cat([torch.arange(0, 18944, 37), torch.arange(18944, B, 3)]).cuda()
    w.check("two_chunks_K50", x, u, w.run(x, u, K, "bf16"), K, "bf16", sel=sel)


@pytest.mark.gpu
def test_fewer_admissible_items_than_k():
    """45 items, histories covering most of them, K = 50: every list ends in (-inf, -1)."""
    B, rows, K, L = 6, 46, 50, 40
    _assert_bf16_branch(B, rows, K, L, cg=1, s_full=1, c_share=0)
    w = World(rows, "bias", None, seed=61)
    rng = np.random.default_rng(17)
    ids = np.zeros((B, L), dtype=np.int64)
    for b in range(B):
        h = rng.permutation(np.arange(1, rows))[: 5 + 5 * b]
        seq = np.concatenate([h, h[:2]])
        ids[b, L - len(seq):] = seq
    x = torch.from_numpy(ids).cuda()
    u = w.users(B, seed=18)
    res = w.run(x, u, K, "bf16")
    w.check("tiny_K50", x, u, res, K, "bf16")
    assert bool((res["ids"][:, -1] == -1).all())


# ------------------------------------------------------------------------------------------------
# exact-fp32 cases
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_fp32_select_path_over_three_user_blocks(worlds):
    """300 users x 500,000 rows, K = 50, fp32: dense scores + per-user selection in blocks of 128, 128 and 44 users."""
    B, rows, K, L = 300, 500_000, 50, 200
    sms = _need_148()
    blk = f32_select_users(rows, sms)
    assert blk == 128 and lib_slots(B, rows, 1) == 1 and B - 2 * blk == 44
    w = worlds(("500k", "zero"), lambda: World(rows, "zero", None, seed=71))
    x = _histories(B, L, w.hot, rows, seed=19).cuda()
    u = w.users(B, seed=20)
    w.check("fp32_select_K50", x, u, w.run(x, u, K, "fp32"), K, "fp32")


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 300])
def test_fp32_streaming_kernel_and_row_shards(worlds, B):
    """600,001 rows, fp32: too many for the select path, so the streaming kernel runs; K = 20, 50.  Also as two row
    shards -- [0, 30001) on the select path, [30001, 600001) on the streaming kernel with row_offset 30001 -- merged
    like ranks merge them, which must equal the unsharded lists bit for bit."""
    rows, L, cut = 600_001, 200, 30_001
    sms = _need_148()
    assert f32_select_users(rows, sms) == 0 and lib_slots(B, rows, 1) == f32_splits(B, rows, sms) > 1
    assert f32_select_users(cut, sms) > 0 and f32_select_users(rows - cut, sms) == 0
    w = worlds(("600k", "bias"), lambda: World(rows, "bias", None, seed=81))
    m = w.model
    x = _histories(B, L, w.hot, rows, seed=21 + B).cuda()
    u = w.users(B, seed=22 + B)
    for K in (20, 50):
        full = w.run(x, u, K, "fp32")
        w.check(f"fp32_stream_B{B}_K{K}", x, u, full, K, "fp32")
        parts_s, parts_i = [], []
        try:
            for lo, hi in ((0, cut), (cut, rows)):
                m.set_row_shard(lo, hi)
                r = w.run(x, u, K, "fp32")
                parts_s.append(r["scores"].clone())
                parts_i.append(r["ids"].clone())
        finally:
            m.set_row_shard(0, rows)
        merged = merge_lists(torch.stack(parts_s), torch.stack(parts_i), None, k_out=K, layout="list_major")
        assert torch.equal(merged["ids"], full["ids"]) and torch.equal(merged["scores"], full["scores"])
