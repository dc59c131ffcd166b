"""CPU: the wide top-K (k in [51, 1024], DESIGN section 2.2) restated in numpy.

* The wide select (select_topk_kernel's wide variant in score.cu): drop history / out-of-shard ids, a radix select
  on the 64-bit key (score key, ~id) 8 bits per pass that stops at the pass whose bin holds exactly the entries still
  needed, collect, sort.  Checked against np.lexsort over (score desc, id asc) for K up to 1024: random scores,
  massive ties at the K-th score, -inf and NaN entries, history ids inside and outside the shard, fewer admissible
  items than K.
* The orchestration of LRURec._retrieve_wide (lattice threshold, collect, select, retry at the K-th best stored
  score, dense fallback) against a full sort, reaching paths 0, 1 and 2, on random and adversarial matrices.
* The (m, r, cap) policy, and the size queries without a device.
"""
import numpy as np
import pytest

from llamarec_b200 import _lib
from llamarec_b200.model import MAX_K_WIDE, wide_policy


def sel_key(v):
    """score.cu sel_key: order-preserving uint32 key of a float32, NaN -> 0."""
    v = np.asarray(v, np.float32)
    i = v.view(np.int32).astype(np.int64)
    k = np.where(i >= 0, i, i ^ 0x7FFFFFFF) & 0xFFFFFFFF
    k = (k ^ 0x80000000) & 0xFFFFFFFF
    return np.where(np.isnan(v), 0, k).astype(np.uint64)


def key64(scores, ids):
    return (sel_key(scores) << np.uint64(32)) | (~np.asarray(ids, np.int64) & 0xFFFFFFFF).astype(np.uint64)


def radix_select(keys, K):
    """The K_eff largest of distinct uint64 keys, found as the kernel does (histograms of 8 bits per pass)."""
    n = keys.size
    K_eff = min(K, n)
    if K_eff == 0:
        return keys[:0], 0
    prefix, need, bits = np.uint64(0), K_eff, 0
    for p in range(8):
        shift = np.uint64(56 - 8 * p)
        hi_mask = np.uint64(0) if p == 0 else np.uint64((0xFFFFFFFFFFFFFFFF << (64 - 8 * p)) & 0xFFFFFFFFFFFFFFFF)
        match = keys[(keys & hi_mask) == prefix]
        hist = np.bincount(((match >> shift) & np.uint64(255)).astype(np.int64), minlength=256)
        above = np.cumsum(hist[::-1])[::-1] - hist          # entries in higher bins
        b = int(np.nonzero((above < need) & (need <= above + hist))[0][0])
        prefix |= np.uint64(b) << shift
        need -= int(above[b])
        bits = 8 * (p + 1)
        if hist[b] == need:
            break
    sh = np.uint64(64 - bits)
    sel = keys[(keys >> sh) >= (prefix >> sh)]
    assert sel.size == K_eff
    return sel, bits


def wide_select(scores, ids, cnt, cap, K, excl, rows, row_offset):
    """-> (status, list scores, list ids, tau') of one user; status 0 ok, -1 overflow, -2 short."""
    stored = min(cnt, cap)
    s, i = scores[:stored], ids[:stored]
    local = i.astype(np.int64) - row_offset
    ok = (local >= 0) & (local < rows) & ~np.isin(i, excl)
    s, i = s[ok], i[ok]
    sel, _ = radix_select(key64(s, i), K)
    sel = np.sort(sel)[::-1]
    hi = (sel >> np.uint64(32)).astype(np.int64)
    valid = hi > int(sel_key(np.float32(-np.inf)))
    n_valid = int(valid.sum())
    out_s = ((hi[:n_valid] ^ 0x80000000)).astype(np.int64)
    out_s = np.where(out_s >= 0x80000000, out_s - (1 << 32), out_s)
    out_s = np.where(out_s >= 0, out_s, out_s ^ 0x7FFFFFFF).astype(np.int32).view(np.float32)
    out_i = (~(sel[:n_valid] & np.uint64(0xFFFFFFFF)).astype(np.int64)) & 0xFFFFFFFF
    out_i = out_i.astype(np.int64)
    if n_valid < K:
        return -2, out_s, out_i, None
    if cnt > cap:
        return -1, out_s, out_i, out_s[K - 1]
    return 0, out_s, out_i, None


def reference(scores, ids, K, excl, rows, row_offset):
    local = ids.astype(np.int64) - row_offset
    ok = (local >= 0) & (local < rows) & ~np.isin(ids, excl) & (scores > -np.inf)
    s, i = scores[ok], ids[ok]
    o = np.lexsort((i, -s.astype(np.float64)))[:K]
    return s[o], i[o]


@pytest.mark.parametrize("K", [51, 100, 257, 1024])
@pytest.mark.parametrize("kind", ["random", "ties", "inf_nan", "history", "few"])
def test_wide_select_matches_lexsort(K, kind):
    rng = np.random.default_rng(K + len(kind))
    rows, row_offset = 50_000, 1000
    n = {"few": K // 2}.get(kind, 6 * K)
    ids = rng.choice(np.arange(row_offset - 500, row_offset + rows + 500), n, replace=False).astype(np.int32)
    if kind == "ties":
        scores = rng.choice(np.float32([1.0, 0.5, 0.25]), n, p=[0.1, 0.8, 0.1]).astype(np.float32)
    else:
        scores = rng.standard_normal(n).astype(np.float32)
    if kind == "inf_nan":
        scores[rng.choice(n, n // 3, replace=False)] = -np.inf
        scores[rng.choice(n, n // 10, replace=False)] = np.nan
    excl = np.sort(rng.choice(ids, min(n // 4, 200), replace=False)) if kind in ("history", "ties") else \
        np.zeros(0, np.int32)
    st, s, i, _ = wide_select(scores, ids, n, n, K, excl, rows, row_offset)
    rs, ri = reference(scores, ids, K, excl, rows, row_offset)
    rs, ri = rs[~np.isnan(rs)], ri[~np.isnan(rs)]
    assert np.array_equal(i, ri)
    assert np.array_equal(s.view(np.int32), rs.view(np.int32))
    assert st == (0 if ri.size >= K else -2)
    if kind == "ties":
        # the tie at the K-th score is resolved by ids: the radix select needed the id passes
        _, bits = radix_select(key64(scores, ids), K)
        assert bits > 32


def orchestrate(S, hist, K, cap, m=20, rng=None):
    """LRURec._retrieve_wide on a dense score matrix S [B, rows] (ids = columns), history lists `hist`."""
    B, rows = S.shape
    r = max(1, -(-4 * K // m))
    out, paths = [], []
    for b in range(B):
        excl = np.asarray(sorted(set(hist[b]) | {0}), np.int32)
        lat = np.arange(0, rows, r)
        lat = lat[~np.isin(lat, excl)]
        ls = np.sort(S[b, lat])[::-1]
        tau = ls[m - 1] if ls.size >= m else -np.inf
        path = None
        for attempt in (0, 1):
            got = np.nonzero(S[b] >= tau)[0]
            got = rng.permutation(got).astype(np.int32)         # the collect appends in no particular order
            st, s, i, tau2 = wide_select(S[b, got], got, got.size, cap, K, excl, rows, 0)
            if st == 0:
                path = attempt
                break
            if st == -2 or attempt == 1:
                break
            tau = tau2
        if path is None:                                        # dense rows
            path = 2
            s, i = reference(S[b], np.arange(rows, dtype=np.int32), K, excl, rows, 0)
        out.append((s, i))
        paths.append(path)
    return out, paths


def test_orchestration_reaches_every_path_and_equals_full_sort():
    rng = np.random.default_rng(0)
    K, rows = 100, 20_000
    seen = set()
    cases = []
    # random
    cases.append((rng.standard_normal((6, rows)).astype(np.float32), None))
    # lattice rows planted high: tau lands above the K-th best -> short -> dense rows
    S = rng.standard_normal((4, rows)).astype(np.float32)
    r = max(1, -(-4 * K // 20))
    S[:, r * np.arange(1, 25)] = 50.0 + np.arange(24, dtype=np.float32)
    cases.append((S, None))
    # repeated rows: more than cap items tie at tau -> overflow twice -> dense rows
    S = rng.standard_normal((4, rows)).astype(np.float32)
    S[:, 3000:3000 + 1500] = 9.0
    cases.append((S, None))
    # a small cap: overflow once, then the K-th best stored score suffices (path 1)
    cases.append((rng.standard_normal((6, rows)).astype(np.float32), 300))
    for S, cap in cases:
        hist = [rng.integers(1, rows, 50) for _ in range(S.shape[0])]
        cap = cap if cap is not None else 8 * K + 52
        out, paths = orchestrate(S, hist, K, cap, rng=rng)
        seen |= set(paths)
        for b, (s, i) in enumerate(out):
            excl = np.asarray(sorted(set(hist[b]) | {0}), np.int32)
            rs, ri = reference(S[b], np.arange(rows, dtype=np.int32), K, excl, rows, 0)
            assert np.array_equal(i, ri) and np.array_equal(s.view(np.int32), rs.view(np.int32))
    assert seen == {0, 1, 2}, seen


def test_policy():
    for k in (51, 64, 100, 255, 256, 500, 1000, 1024):
        for stride in (0, 52, 204):
            m, r, cap = wide_policy(k, stride)
            assert m * r >= 4 * k and m == 20 and r == max(1, -(-4 * k // m))
            assert cap == 8 * k + stride
            for rows in (k, 10 * k, 131_073, 2_000_000, 10_000_001):
                n_lat = -(-rows // r)
                if n_lat >= m:
                    assert len(range(0, rows, r)) >= m
    assert wide_policy(100, 52, topk_cap=7)[2] == 7
    with pytest.raises(ValueError):
        wide_policy(100, 52, topk_cap=0)
    assert MAX_K_WIDE == 1024


def test_wide_size_queries_without_gpu():
    lib = _lib.load()
    a = lib.lrb_wide_sample_workspace_bytes(4096, 10_000_001, 52, 20, 20)
    assert a >= lib.lrb_score_scratch_bytes(4096) + 4096 * 52 * 4
    assert lib.lrb_wide_sample_workspace_bytes(0, 10, 0, 1, 20) == 256          # bad shape: a minimal answer
    assert lib.lrb_wide_sample_workspace_bytes(1, 10, 0, 1, 51) == 256          # m beyond the streaming limit
    ld = 10_000_004
    w = lib.lrb_wide_select_workspace_bytes(26, 10_000_001)
    assert w >= 26 * ld * 4 and w < 27 * ld * 4 + 256                          # ~1 GiB blocks of dense rows
    assert lib.lrb_wide_select_workspace_bytes(1000, 10_000_001) == w
    assert lib.lrb_wide_select_workspace_bytes(3, 1683) >= 3 * 1684 * 4
