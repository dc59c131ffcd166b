"""The stage-2 verbalizer kernels (verbalizer.cu) against a float64 reference, on the shapes the parity tests do not
reach: every instantiated hidden width, multi-word classes with masked slots, a full warp of label words, ragged user
slots, the logits path with every handler, calibration, and row offsets past 2^31 elements.

Reference (u = 2^-24):
  * Logits: float64 dot products of the exact bf16 operands the kernel read -- the hidden rows and only the C*W
    label rows of the lm_head, widened to float64 (torch DGEMM).
  * Tail: oracle.verbalizer_oracle.process_logits on float64 tensors.

Raw logit of user b and word w.  Each lane of the kernel runs an H/32-long fp32 FMA chain over its share of the row
(bf16 x bf16 products are exact in fp32, so each FMA rounds once) and the warp adds the 32 partial sums in 5
butterfly steps.  With S_bw = sum_i |h_bi w_i|:
      |logit - ref| <= tol_bw = (H/32 + 5) * u * S_bw.
With round_bf16 = 1 the logit must be bf16-representable and lie in [bf16_rn(ref - tol), bf16_rn(ref + tol)] (round
to nearest is monotonic), which holds at most two values.

The GEMV and the tail are checked apart.  The logit of word w depends only on (hidden row, label row, H), never on C,
W, the warp or the user's slot in the CTA, so a mode-0 call with the same words as C*W one-word classes and every mask
set (the "probe") returns the raw logits bit for bit (x * 1 / 1 is exact).  The probe is checked against the bound
above, and every other call against the float64 tail evaluated on the probe's fp32 logits.

Tail of one user, x_w the projected label-word logits (x - 10000 (1 - m)), m_w the word mask:
  * mode 0 (masked mean): tol = (W + 2) * u * sum_w |x_w m_w| / sum_w m_w.
  * mode 1.  D = max_w x_w - min_w x_w over the unmasked words (a masked word sits 10^4 below and its exp is 0 in
    both precisions).  d_w = x_w - max x rounds once (u D); expf is within 2 ulp (4u), so e_w carries a relative
    error <= u (D + 4); the 5-level sum of non-negative terms adds 5u; p = e / den adds u:  p_w within u (2D + 14).
    log(p + 1e-15): the add rounds (u), the input error passes through as an absolute error (d log = dp / p), and
    logf is within 1 ulp <= 2u |y| with |y| <= -log(1e-15) < 35 (70u).  So without calibration
        |dy| <= u (2D + 85).
    With calibration the calibration vector's probabilities cp carry u (2 Dc + 14), cp + 1e-15 adds u, the quotient u,
    the renormalising sum 5u on top of its terms' error, the division u; numerator and sum both carry the quotient's
    error, so p is within u (4D + 4Dc + 66) and |dy| <= u (4D + 4Dc + 137).  A subnormal or flushed exp is at most
    2^-149 / den << 1e-15 and vanishes in the + 1e-15.  The masked mean then adds (W + 2) u sum|y m| / sum m, and since
    y <= 0 that sum is |out|:
        tol = u (2D + 85)  [or u (4D + 4Dc + 137)]  + (W + 2) u |out|.
  * Logits path, handler "mean": each word logit is a sum of T masked terms and a division, within
    eps = (T + 1) u sum_t |l_t m_t| / sum_t m_t; this adds eps (mode 0), 2 eps (mode 1) or 4 (eps + eps_c) (mode 1 with
    calibration) to the bound.  "first" and "max" pick an fp32 value exactly.
A NaN where the reference is finite fails, and so does a finite value where the reference is NaN.

The fixture prints the largest err/tol ratio of each case, the file's run time and its peak device memory."""
import math
import os
import re
import time

import numpy as np
import pytest
import torch

from llamarec_b200 import ManualVerbalizer, _lib, stage2
from llamarec_b200._lib import LrbError
from oracle import verbalizer_oracle as VO

U = 2.0 ** -24
F64 = torch.float64
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LRB_ERR_UNSUPPORTED = -2
# The hidden widths lrb_verbalizer_score instantiates (NVEC = H / 256 in verbalizer.cu); every other H is refused.
WIDTHS = (256, 512, 768, 1024, 1536, 2048, 3072, 3584, 4096, 5120, 8192)
SWEEP = list(range(256, 8448 + 1, 256)) + [4000, 128]
LAYOUTS = [(1, 1), (3, 1), (7, 3), (16, 2), (1, 32), (32, 1)]
RATIOS = {}


def record(case, ratio):
    RATIOS[case] = max(RATIOS.get(case, 0.0), float(ratio))


# ------------------------------------------------------------------------------------------------
# Comparator
# ------------------------------------------------------------------------------------------------
def bf16_rn(x):
    return x.to(torch.float32).to(torch.bfloat16).to(F64)


def _same_nans(got, want, what):
    gn, wn = torch.isnan(got), torch.isnan(want)
    assert torch.equal(gn, wn), (what, "NaN where the reference is finite" if (gn & ~wn).any()
                                 else "finite where the reference is NaN")
    return ~wn


def check_logits(got, ref, absdot, H, round_bf16, what):
    """got [B, n] kernel logits, ref / absdot [B, n] float64 sum(h w) / sum|h w|.  Returns the largest err/tol; with
    round_bf16 the tolerance of that ratio also holds half a bf16 ulp of ref."""
    got = got.detach().to(F64).cpu()
    _same_nans(got, ref, what)
    tol = (H / 32 + 5) * U * absdot
    err = (got - ref).abs()
    if not round_bf16:
        ratio = (err / tol.clamp_min(1e-300)).max().item()
        assert bool((err <= tol).all()), (what, "logit outside (H/32 + 5) u sum|h w|", ratio)
        return ratio
    assert torch.equal(bf16_rn(got), got), (what, "logit is not a bf16 value")
    inside = (got >= bf16_rn(ref - tol)) & (got <= bf16_rn(ref + tol))
    half_ulp = torch.ldexp(torch.ones_like(ref), torch.frexp(ref)[1] - 9)
    ratio = (err / (tol + half_ulp)).max().item()
    assert bool(inside.all()), (what, "logit outside [bf16_rn(ref - tol), bf16_rn(ref + tol)]", ratio,
                                int((~inside).sum()))
    return ratio


def check_close(got, want, tol, what):
    """got, want, tol [B, C]; NaNs must coincide; elsewhere |got - want| <= tol.  Returns the largest err/tol."""
    got = got.detach().to(F64).cpu()
    ok = _same_nans(got, want, what)
    err = (got - want).abs()[ok]
    t = tol[ok]
    assert bool(torch.isfinite(err).all()), (what, "non-finite output")
    ratio = (err / t.clamp_min(1e-300)).max().item() if err.numel() else 0.0
    assert bool((err <= t).all()), (what, "tail outside its bound", ratio)
    return ratio


def _spread(x, on):
    xs = x.reshape(x.shape[0], -1)[:, on]
    return xs.max(1).values - xs.min(1).values


def tail_tol(x, wm, mode, want, xc=None, eps=None, eps_c=0.0):
    """Bound of the module docstring.  x [B, C, W] projected label-word logits (float64), wm [C, W], want [B, C] the
    float64 output, xc [C, W] the projected calibration logits (mode 1 with calibration), eps [B] / eps_c the handler's
    error of one word logit."""
    m = wm.to(F64)
    W = m.shape[-1]
    eps = torch.zeros(x.shape[0], dtype=F64) if eps is None else eps
    if mode == 0:
        return (W + 2) * U * (x.abs() * m).sum(-1) / m.sum(-1) + eps[:, None]
    on = m.reshape(-1) > 0
    D = _spread(x, on)
    if xc is None:
        ty = U * (2 * D + 85) + 2 * eps
    else:
        ty = U * (4 * D + 4 * _spread(xc[None], on) + 137) + 4 * (eps + eps_c)
    return ty[:, None] + (W + 2) * U * want.abs()


def tail_reference(x, wm, mode, calw=None):
    """float64 tail on fp32 label-word logits x [B, C*W] (word order of wm [C, W]); calw [C*W] the calibration
    vector's logits of the same words.  Returns (want, tol) [B, C]."""
    C, W = wm.shape
    ids = torch.arange(C * W).reshape(C, W, 1)
    tm = torch.ones(C, W, 1, dtype=torch.int64)
    wm = wm.to(torch.int64).cpu()
    x64 = x.detach().to(F64).cpu()
    calw = calw.to(F64).cpu() if (mode == 1 and calw is not None) else None
    want = VO.process_logits(x64, ids, tm, wm, bool(mode), "first", calw)
    xc = VO.project(calw[None], ids, tm, wm)[0] if calw is not None else None
    return want, tail_tol(VO.project(x64, ids, tm, wm), wm, mode, want, xc)


def handler_eps(lg64, ids, tm, handler):
    """[B] bound on the fp32 error of one word logit: only the mean handler rounds."""
    if handler != "mean":
        return torch.zeros(lg64.shape[0], dtype=F64)
    tmd = tm.to(F64)
    per = (ids.shape[-1] + 1) * U * (lg64[:, ids].abs() * tmd).sum(-1) / tmd.sum(-1).clamp_min(1)
    return per.reshape(lg64.shape[0], -1).max(1).values


def logits_reference(lg64, v, cal=None):
    """float64 process_logits of ManualVerbalizer v on logits lg64 [B, V]; returns (want, tol)."""
    ids, tm, wm, handler = v.label_words_ids, v.words_ids_mask, v.label_words_mask, v.multi_token_handler
    mode = int(v.post_log_softmax)
    cal64 = cal.to(F64) if (mode == 1 and cal is not None) else None
    want = VO.process_logits(lg64, ids, tm, wm, bool(mode), handler, cal64)
    xc = eps_c = None
    if cal64 is not None:
        xc = VO.project(cal64[None], ids, tm, wm, handler)[0]
        eps_c = handler_eps(cal64[None], ids, tm, handler)[0]
    tol = tail_tol(VO.project(lg64, ids, tm, wm, handler), wm, mode, want, xc, handler_eps(lg64, ids, tm, handler),
                   0.0 if eps_c is None else eps_c)
    return want, tol


# ------------------------------------------------------------------------------------------------
# Inputs
# ------------------------------------------------------------------------------------------------
class Tok:
    """A label word spells its own sub-token ids: '12.7.400' -> [12, 7, 400]."""

    def encode(self, word, add_special_tokens=False):
        return [int(t) for t in word.split(".")]


def verbalizer(words, post_log_softmax, handler="first", cal=None):
    """words[c][j] = sub-token ids of word j of class c."""
    v = ManualVerbalizer(Tok(), classes=list(range(len(words))),
                         label_words=[[".".join(str(t) for t in w) for w in ws] for ws in words], prefix="",
                         post_log_softmax=post_log_softmax, multi_token_handler=handler)
    if cal is not None:
        v.register_calibrate_logits(cal)
    return v


def layout_words(C, W, V, T=1, seed=0):
    """C classes: class 0 has W words, class c > 0 has 1 + (5c mod W) (unequal counts, so masked slots); word j of
    class c has 1 + (c + 2j mod T) sub-tokens (T for the first word, so the table is [C, W, T]); ids distinct in
    [1, V)."""
    g = torch.Generator().manual_seed(seed)
    counts = [W] + [1 + (5 * c) % W for c in range(1, C)]
    pool = (torch.randperm(V - 1, generator=g)[:sum(counts) * T] + 1).tolist()
    words, k = [], 0
    for c in range(C):
        ws = []
        for j in range(counts[c]):
            nt = T if c == j == 0 else 1 + (c + 2 * j) % T
            ws.append(pool[k:k + nt])
            k += nt
        words.append(ws)
    return words


def one_word_classes(ids):
    return [[[int(t)]] for t in ids]


def rand_bf16(shape, scale, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(shape, generator=g, device="cuda") * scale).to(torch.bfloat16)


def lm_head(V, H, seed):
    """Rows scaled so logits are O(4): the softmax neither saturates nor flattens."""
    return rand_bf16((V, H), 4.0 / math.sqrt(H), seed)


def calibration(V, seed, spread=8.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(V, generator=g) * 2 - 1) * spread


def ref_logits(h, lm, ids):
    """float64 (sum h w, sum |h w|) [B, n] of hidden rows h [B, H] and lm_head rows ids [n], exact bf16 operands."""
    rows = lm[ids.to(lm.device).long()].to(F64)
    hd = h.to(F64)
    return (hd @ rows.T).cpu(), (hd.abs() @ rows.abs().T).cpu()


def raw_score(h, lm, ids, mask, mode, round_bf16, cal=None, out=None):
    """lrb_verbalizer_score through ctypes; ids int32 / mask uint8 [C, W] on the device.  Returns (rc, out)."""
    B, H = h.shape
    C, W = ids.shape
    out = torch.empty(B, C, dtype=torch.float32, device="cuda") if out is None else out
    rc = _lib.load().lrb_verbalizer_score(h.data_ptr(), lm.data_ptr(), B, H, lm.shape[0], ids.data_ptr(),
                                          mask.data_ptr(), C, W, mode, int(round_bf16),
                                          cal.data_ptr() if cal is not None else None, out.data_ptr(),
                                          _lib.stream_handle())
    return rc, out


def raw_probe(h, lm, flat, round_bf16):
    n = flat.numel()
    rc, x = raw_score(h, lm, flat.reshape(n, 1).to(torch.int32).cuda(), torch.ones(n, 1, dtype=torch.uint8,
                                                                                     device="cuda"), 0, round_bf16)
    _lib.check(rc)
    return x


def check_score_layout(h, lm, words, round_bf16, cal, case):
    """Probe + mode 0 + mode 1 (calibrated when cal is given) of the class layout `words` through score_hidden."""
    H = h.shape[1]
    v0 = verbalizer(words, False)
    flat = v0.label_words_ids[:, :, 0].reshape(-1)
    wm = v0.label_words_mask
    x = verbalizer(one_word_classes(flat), False).score_hidden(h, lm, round_logits_to_bf16=round_bf16)
    ref, absdot = ref_logits(h, lm, flat)
    record(f"{case} logits", check_logits(x, ref, absdot, H, round_bf16, case))
    for mode in (0, 1):
        v = verbalizer(words, bool(mode), cal=cal if mode else None)
        got = v.score_hidden(h, lm, round_logits_to_bf16=round_bf16)
        want, tol = tail_reference(x, wm, mode, cal[flat] if (mode and cal is not None) else None)
        record(f"{case} mode {mode}", check_close(got, want, tol, (case, mode, round_bf16, h.shape[0])))


@pytest.fixture(scope="module")
def dev():
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    yield "cuda"
    torch.cuda.synchronize()
    print(f"\n[verbalizer] {time.perf_counter() - t0:.1f} s, peak device memory "
          f"{torch.cuda.max_memory_allocated() / 2**30:.2f} GiB; max err/tol per case:\n  "
          + "\n  ".join(f"{k}: {v:.3f}" for k, v in RATIOS.items()))


# ------------------------------------------------------------------------------------------------
# CPU: the dispatch list, the comparator's negative controls, the Python-boundary checks
# ------------------------------------------------------------------------------------------------
def test_instantiated_widths_match_the_dispatch():
    """WIDTHS is what the GPU sweep expects to run; it must equal the NVEC values verbalizer.cu launches."""
    with open(os.path.join(ROOT, "llamarec_b200", "csrc", "verbalizer.cu")) as f:
        src = f.read()
    nvecs = {int(n) for n in re.findall(r"LRB_VERB_LAUNCH\((\d+)\)", src)}
    assert sorted(256 * n for n in nvecs) == list(WIDTHS)


def _cpu_case(H, B=6, n=12, V=64, seed=0):
    g = torch.Generator().manual_seed(seed)
    h = torch.randn(B, H, generator=g).to(torch.bfloat16)
    lm = (torch.randn(V, H, generator=g) * 4 / math.sqrt(H)).to(torch.bfloat16)
    ids = torch.randperm(V, generator=g)[:n]
    ref, absdot = ref_logits(h, lm, ids)
    return h, lm, ids, ref, absdot


@pytest.mark.parametrize("H", [256, 8192])
def test_comparator_rejects_a_missing_chunk_and_unrounded_logits(H):
    """A label row with one 8-element chunk left out fails the raw bound; fp32 logits fail where bf16-rounded ones
    were asked for.  The reference itself, rounded to fp32 or bf16, passes."""
    h, lm, ids, ref, absdot = _cpu_case(H)
    assert check_logits(ref.float(), ref, absdot, H, False, "fp32 ref") <= 1.0
    assert check_logits(bf16_rn(ref), ref, absdot, H, True, "bf16 ref") <= 1.0
    s = 8 * 5
    chunk = (h[:, s:s + 8].to(F64) @ lm[ids][:, s:s + 8].to(F64).T)
    with pytest.raises(AssertionError):
        check_logits((ref - chunk).float(), ref, absdot, H, False, "missing chunk")
    with pytest.raises(AssertionError):
        check_logits(ref.float(), ref, absdot, H, True, "unrounded")


def _cpu_logits(B=7, V=50, seed=1):
    g = torch.Generator().manual_seed(seed)
    lg = (torch.rand(B, V, generator=g) * 2 - 1) * 90
    lg[:, 0] = 90.0                       # the padding sub-token: wins a max that ignores the mask
    return lg.to(F64)


def test_comparator_rejects_a_wrong_tail():
    """The class mean over all W words (mask ignored), calibration without the renormalisation, and a max handler
    that ignores the sub-token mask all fail the tail bound; the float64 reference passes."""
    lg = _cpu_logits()
    cal = calibration(lg.shape[1], 3, 30.0).to(F64)
    words = layout_words(5, 3, lg.shape[1], T=3, seed=2)
    v0, v1 = verbalizer(words, False, "max"), verbalizer(words, True, "max")
    ids, tm, wm = v0.label_words_ids, v0.words_ids_mask, v0.label_words_mask
    assert (wm == 0).any() and (tm[wm > 0] == 0).any()
    want0, tol0 = logits_reference(lg, v0)
    assert check_close(want0.float(), want0, tol0, "mode 0 ref") <= 1.0
    with pytest.raises(AssertionError):
        check_close(VO.project(lg, ids, tm, wm, "max").mean(-1), want0, tol0, "mean ignores the mask")
    with pytest.raises(AssertionError):
        check_close(VO.process_logits(lg, ids, torch.ones_like(tm), wm, False, "max"), want0, tol0,
                    "max ignores the sub-token mask")
    want1, tol1 = logits_reference(lg, v1, cal)
    assert check_close(want1.float(), want1, tol1, "mode 1 ref") <= 1.0
    B = lg.shape[0]
    p = torch.softmax(VO.project(lg, ids, tm, wm, "max").reshape(B, -1), -1)
    cp = torch.softmax(VO.project(cal[None], ids, tm, wm, "max").reshape(1, -1), -1)
    y = torch.log(p / (cp + 1e-15) + 1e-15).reshape(B, *wm.shape)
    with pytest.raises(AssertionError):
        check_close((y * wm).sum(-1) / wm.sum(-1), want1, tol1, "calibration without renormalisation")


def test_comparator_rejects_nan_mismatch():
    want = torch.tensor([[1.0, float("nan")]], dtype=F64)
    tol = torch.full_like(want, 1e-6)
    assert check_close(want.clone(), want, tol, "same") == 0.0
    with pytest.raises(AssertionError):
        check_close(torch.tensor([[1.0, 2.0]]), want, tol, "finite where NaN")
    with pytest.raises(AssertionError):
        check_close(torch.tensor([[float("nan"), float("nan")]]), want, tol, "NaN where finite")


def test_out_of_range_token_ids_raise_index_error():
    """Like the reference's logits[:, label_words_ids]: an id >= V (or < 0) raises IndexError at both entry points,
    before anything reaches the device."""
    v = verbalizer([[[3]], [[120]]], True)
    with pytest.raises(IndexError):
        v.score_hidden(torch.zeros(2, 256, dtype=torch.bfloat16), torch.zeros(100, 256, dtype=torch.bfloat16))
    with pytest.raises(IndexError):
        v.process_logits(torch.zeros(2, 100))
    v.label_words_ids[0, 0, 0] = -1
    with pytest.raises(IndexError):
        v.process_logits(torch.zeros(2, 200))
    with pytest.raises(IndexError):
        VO.process_logits(torch.zeros(2, 100), verbalizer([[[3]], [[120]]], True).label_words_ids,
                          v.words_ids_mask, v.label_words_mask, True)


# ------------------------------------------------------------------------------------------------
# lrb_verbalizer_score
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("H", SWEEP)
def test_width_sweep(dev, H):
    """B = 5 (a full CTA and one user), 20 one-word classes, both modes, both round_bf16: the instantiated widths match
    the float64 reference; every other width returns LRB_ERR_UNSUPPORTED and leaves `out` untouched."""
    B, V = 5, 1000
    h = rand_bf16((B, H), 1.0, seed=H)
    lm = lm_head(V, H, seed=H + 1)
    ids = torch.randperm(V - 1, generator=torch.Generator().manual_seed(H))[:20] + 1
    if H not in WIDTHS:
        out = torch.full((B, 20), -7.25, device="cuda")
        for mode in (0, 1):
            rc, _ = raw_score(h, lm, ids.reshape(20, 1).to(torch.int32).cuda(),
                              torch.ones(20, 1, dtype=torch.uint8, device="cuda"), mode, 1, out=out)
            assert rc == LRB_ERR_UNSUPPORTED, (H, rc)
        with pytest.raises(LrbError) as e:
            verbalizer(one_word_classes(ids), True).score_hidden(h, lm)
        assert e.value.code == LRB_ERR_UNSUPPORTED
        torch.cuda.synchronize()
        assert bool((out == -7.25).all())
        return
    for rnd in (False, True):
        check_score_layout(h, lm, one_word_classes(ids), rnd, None, f"width H={H} round={int(rnd)}")


@pytest.mark.gpu
@pytest.mark.parametrize("H", [4096, 768])
@pytest.mark.parametrize("C,W", LAYOUTS)
def test_class_layouts(dev, H, C, W):
    """(C, W) from one word to a full warp of 32, C*W not dividing 32, masked slots from unequal word counts; mode 0
    and calibrated mode 1; B = 1..4 (one partly empty CTA) and 4097 (a ragged last CTA)."""
    V = 5003
    lm = lm_head(V, H, seed=10 * H + C)
    cal = calibration(V, seed=W)
    words = layout_words(C, W, V, seed=C * 100 + W)
    wm = verbalizer(words, False).label_words_mask
    assert tuple(wm.shape) == (C, W) and bool((wm == 0).any()) == (C > 1 and W > 1)
    for B in (1, 2, 3, 4, 4097):
        h = rand_bf16((B, H), 1.0, seed=B)
        for rnd in (False, True):
            check_score_layout(h, lm, words, rnd, cal, f"layout H={H} C={C} W={W}")


@pytest.mark.gpu
def test_more_than_32_label_words_are_refused(dev):
    V = 500
    words = layout_words(3, 11, V)
    v = verbalizer(words, True)
    assert tuple(v.label_words_mask.shape) == (3, 11)
    for call in (lambda: v.score_hidden(rand_bf16((4, 512), 1.0, 0), lm_head(V, 512, 1)),
                 lambda: v.process_logits(torch.zeros(4, V, device="cuda"))):
        with pytest.raises(LrbError) as e:
            call()
        assert e.value.code == LRB_ERR_UNSUPPORTED


@pytest.mark.gpu
def test_user_slot_invariance(dev):
    """Permuting the hidden rows permutes the output rows bit for bit (the CTA slot never changes a result)."""
    H, V, B = 768, 5003, 4097
    lm = lm_head(V, H, 5)
    h = rand_bf16((B, H), 1.0, 6)
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(7)).cuda()
    words = layout_words(7, 3, V, seed=8)
    for mode in (0, 1):
        v = verbalizer(words, bool(mode), cal=calibration(V, 9) if mode else None)
        for rnd in (False, True):
            out = v.score_hidden(h, lm, round_logits_to_bf16=rnd)
            assert torch.equal(v.score_hidden(h[perm], lm, round_logits_to_bf16=rnd), out[perm]), (mode, rnd)


def _raw_tables(V, seed):
    """Raw-ABI layouts the class cannot express: (4, 8) with class 1 fully masked, (1, 32) with masked words."""
    g = torch.Generator().manual_seed(seed)
    m48 = torch.tensor([[1, 1, 0, 1, 0, 0, 1, 0], [0] * 8, [1] * 8, [0] * 7 + [1]], dtype=torch.uint8)
    m132 = (torch.arange(32) % 3 != 1).to(torch.uint8).reshape(1, 32)
    return [(torch.randint(1, V, tuple(m.shape), generator=g, dtype=torch.int32), m) for m in (m48, m132)]


@pytest.mark.gpu
def test_raw_masks_all_masked_class_and_mode0_calibration(dev):
    """A class with every word masked is NaN (the reference's 0/0); the other classes match.  In mode 0 a non-NULL
    calibration vector changes nothing, bit for bit."""
    H, V = 4096, 5003
    lm = lm_head(V, H, 11)
    cal = calibration(V, 12).cuda()
    for B in (3, 9):
        h = rand_bf16((B, H), 1.0, 13 + B)
        for ids, mask in _raw_tables(V, B):
            C, W = ids.shape
            flat = ids.reshape(-1)
            idsd, maskd = ids.cuda(), mask.cuda()
            for rnd in (0, 1):
                x = raw_probe(h, lm, flat, rnd)
                ref, absdot = ref_logits(h, lm, flat)
                case = f"raw masks C={C} W={W}"
                record(f"{case} logits", check_logits(x, ref, absdot, H, rnd, case))
                for mode, c in ((0, None), (1, None), (1, cal)):
                    rc, got = raw_score(h, lm, idsd, maskd, mode, rnd, c)
                    _lib.check(rc)
                    want, tol = tail_reference(x, mask, mode, cal.cpu()[flat.long()] if c is not None else None)
                    record(f"{case} mode {mode}", check_close(got, want, tol, (case, mode, rnd, c is not None)))
                    if C == 4:
                        assert bool(torch.isnan(got[:, 1]).all()) and not bool(torch.isnan(got[:, [0, 2, 3]]).any())
                rc, a = raw_score(h, lm, idsd, maskd, 0, rnd, None)
                _lib.check(rc)
                rc, b = raw_score(h, lm, idsd, maskd, 0, rnd, cal)
                _lib.check(rc)
                assert torch.equal(torch.nan_to_num(a, 1.5), torch.nan_to_num(b, 1.5))


@pytest.mark.gpu
def test_row_offset_beyond_2_pow_31_elements(dev):
    """H = 8192, V = 262,400, label ids >= 262,144: tok * H >= 2^31.  Only the label rows and row 0 are written."""
    H, V, B = 8192, 262_400, 5
    lm = torch.empty(V, H, dtype=torch.bfloat16, device="cuda")
    ids = torch.tensor([262_144 + 13 * k for k in range(19)] + [V - 1])
    assert int(ids.min()) * H >= 2 ** 31
    lm[ids.cuda()] = lm_head(20, H, 21)
    lm[0] = lm_head(1, H, 22)[0]
    h = rand_bf16((B, H), 1.0, 23)
    for rnd in (False, True):
        check_score_layout(h, lm, one_word_classes(ids), rnd, None, f"row offset >= 2^31 round={int(rnd)}")
    del lm
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------
# lrb_verbalizer_from_logits (process_logits)
# ------------------------------------------------------------------------------------------------
def _logit_inputs(lg32, variant):
    """The same logits as fp32, as a view with row pitch V + 37, or rounded to bf16 / fp16."""
    if variant == "pitch":
        wide = torch.full((lg32.shape[0], lg32.shape[1] + 37), float("nan"), device="cuda")
        wide[:, :lg32.shape[1]] = lg32
        return wide[:, :lg32.shape[1]]
    return lg32.to({"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[variant])


@pytest.mark.gpu
@pytest.mark.parametrize("T", [1, 3, 5])
@pytest.mark.parametrize("handler", ["first", "max", "mean"])
def test_from_logits_handlers(dev, handler, T):
    """Every handler x mode x calibration on / off, ragged sub-token masks, C*W = 32 and 15, B in {1, 7, 8, 9, 1000},
    fp32 / pitched fp32 / bf16 / fp16 logits spread to +-90 (the softmax underflows to the log(1e-15) floor); the
    padding token's logit is the largest, so a handler that read a masked sub-token would show."""
    V = 3001
    cal = calibration(V, 31, 30.0)
    cal[0] = 30.0
    for C, W in ((8, 4), (5, 3)):
        words = layout_words(C, W, V, T=T, seed=T * 10 + C)
        vs = [verbalizer(words, False, handler), verbalizer(words, True, handler),
              verbalizer(words, False, handler, cal), verbalizer(words, True, handler, cal)]
        tm = vs[0].words_ids_mask
        assert tuple(tm.shape) == (C, W, T) and bool((tm[vs[0].label_words_mask > 0] == 0).any()) == (T > 1)
        for B in (1, 7, 8, 9, 1000):
            g = torch.Generator(device="cuda").manual_seed(B * 7 + T)
            lg32 = (torch.rand(B, V, generator=g, device="cuda") * 2 - 1) * 90
            lg32[:, 0] = 90.0
            for variant in ("fp32", "pitch", "bf16", "fp16"):
                lg = _logit_inputs(lg32, variant)
                lg64 = lg.to(F64).cpu()
                for v in vs:
                    want, tol = logits_reference(lg64, v, v._calibrate_logits)
                    case = f"logits {handler} T={T} mode {int(v.post_log_softmax)} cal={int(v._calibrate_logits is not None)}"
                    record(case, check_close(v.process_logits(lg), want, tol, (case, C, W, B, variant)))


@pytest.mark.gpu
def test_from_logits_broadcast_rows(dev):
    """A [B, V] view of one row (stride (0, 1)) gives the same result as its dense copy, and matches float64.  For
    B = 1 the view is still stride (0, 1) after .contiguous(), so the row pitch must not be read from it."""
    V = 3001
    g = torch.Generator(device="cuda").manual_seed(41)
    row = (torch.rand(V, generator=g, device="cuda") * 2 - 1) * 20
    words = layout_words(7, 3, V, T=2, seed=42)
    for handler in ("first", "mean"):
        v = verbalizer(words, True, handler, calibration(V, 43))
        for B in (1, 9):
            lg = row.as_strided((B, V), (0, 1))
            assert lg.stride() == (0, 1)
            got = v.process_logits(lg)
            assert torch.equal(got, v.process_logits(row.repeat(B, 1)))
            want, tol = logits_reference(lg.to(F64).cpu(), v, v._calibrate_logits)
            record("logits broadcast rows", check_close(got, want, tol, ("broadcast", handler, B)))


# ------------------------------------------------------------------------------------------------
# Stage-2 metrics on the fused kernel's output
# ------------------------------------------------------------------------------------------------
def _metrics64(s, labels, ks, ties_by_lower_index=True):
    """Recall/MRR/NDCG@k in float64 with the label's rank under (score desc, index asc) -- or index desc."""
    ls = s.gather(1, labels[:, None])
    idx = torch.arange(s.shape[1])[None]
    before = idx < labels[:, None] if ties_by_lower_index else idx > labels[:, None]
    r = ((s > ls).sum(1) + ((s == ls) & before).sum(1)).to(F64)
    out = {}
    for k in ks:
        hit = (r < k).to(F64)
        out[f"Recall@{k}"] = hit.mean().item()
        out[f"MRR@{k}"] = (hit / (r + 1)).mean().item()
        out[f"NDCG@{k}"] = (hit / torch.log2(r + 2)).mean().item()
    return out


@pytest.mark.gpu
def test_rerank_metrics_on_fused_output_with_ties(dev):
    """stage2.rerank_metrics on the [4097, 20] bf16-rounded kernel output, which holds exact ties, against float64
    metrics under the merge kernel's tie rule; the opposite rule must give different metrics."""
    H, V, B = 4096, 5003, 4097
    ks = [1, 5, 10, 20, 50]
    lm = lm_head(V, H, 51)
    h = rand_bf16((B, H), 1.0, 52)
    ids = torch.randperm(V - 1, generator=torch.Generator().manual_seed(53))[:20] + 1
    scores = verbalizer(one_word_classes(ids), False).score_hidden(h, lm)
    labels = torch.randint(0, 20, (B,), generator=torch.Generator().manual_seed(54))
    s = scores.to(F64).cpu()
    label_ties = int(((s == s.gather(1, labels[:, None])).sum(1) > 1).sum())
    assert label_ties > 0
    got = stage2.rerank_metrics(scores, labels.cuda(), ks)
    want = _metrics64(s, labels, ks)
    other = _metrics64(s, labels, ks, ties_by_lower_index=False)
    # per-user values round in fp32; 8 per CTA are summed, then one atomic add per CTA
    tol = {k: ((B + 7) // 8 + 11) * U * v + 1e-12 for k, v in want.items()}
    assert set(got) == set(want)
    bad = {k: (got[k], want[k]) for k in want if abs(got[k] - want[k]) > tol[k]}
    assert not bad, bad
    record("rerank metrics", max(abs(got[k] - want[k]) / tol[k] for k in want))
    assert any(abs(other[k] - want[k]) > tol[k] for k in want)
