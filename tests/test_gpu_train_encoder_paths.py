"""The encoder (lrb_encode_fwd) and the fused train step (lrb_train_step, lrb_ce_loss_fwd) on the shapes and launch
branches the other tests do not reach, against the float64 oracle (oracle/, run with dtype=torch.float64).

The train step's launch decomposition depends on the shape: the TN GEMMs and column sums of the weight gradients
split the B*L tokens into slices of 1024 and add the slices with atomics; the item pass of the CE backward splits the
catalogue into 128-item tiles and the tokens into slices set by the SM count; the value path splits the catalogue by
splits_for.  The encoder's two token kernels loop over tiles once a batch exceeds one wave, and its scan takes a
general carry-set path on rows with holes.  Each case below names the branch it targets and asserts it, as its first
line, through a Python restatement of the host-side formulas (train.cu, ce_loss.cu, encode.cu); a CPU test pins the
value path's restatement to lrb_ce_workspace_bytes.

Comparator.  For every gradient tensor e_k = max|g_kernel - g_64| / max|g_64|, against the fp64 oracle's autograd
on the same weights and batch (dropout multipliers included), must stay <= GRAD_BAR; the fp32 oracle's own e_32 on the
same case is printed beside it for scale.  Losses: relative LOSS_BAR to fp64.  Encoder states: atol = rtol = STATE_BAR.
Measured on one NVIDIA B200 (1000 W power limit): the largest e_k of any case is 2.7e-5 (params_log at L = 200), where
the fp32 oracle's e_32 is 2.8e-5; loss errors stay below 3e-7 relative and encoder states below 1.4e-6 absolute.  The
bars leave room for fp32 summation order, and an error of one dropped token slice or item tile is 1e3 times larger.
The CPU negative controls below show that this comparator fails on the errors the cases are for.

Inputs: synth.make_state_dict weights with random LayerNorm weights and biases (it sets them to 1 and 0, under which
a swapped or dropped LayerNorm parameter cannot show) and a bias of std 0.02; left-padded rows from
synth.make_sequences with labels = the next item, the held-out item at the last position and 0 on padding, plus
empty rows and rows whose history fills every position."""
import math
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from llamarec_b200 import LRURec, _lib, synth
from llamarec_b200._lib import LrbError
from llamarec_b200.model import _draw_seed
from oracle import dropout_oracle as DO
from oracle import lru_oracle as O

F64 = torch.float64
GRAD_BAR = 1e-4
LOSS_BAR = 1e-5
STATE_BAR = 2e-5
SMS_WITHOUT_DEVICE = 148

# ------------------------------------------------------------------------------------------------
# Restatement of the host-side launch formulas
# ------------------------------------------------------------------------------------------------
M_SLICE = 1024            # train.cu:720 m_slice: gemm_tn / colsum_kernel take one z-slice per 1024 tokens (:722-724)
CR, CI = 128, 64          # train.cu:432-433: items per CTA of ce_bwd_items_kernel, staged rows
MAX_BLOCKS = 8            # train.cu:675-676: Saved sv[8], at most 8 blocks
TOK = 64                  # encode.cu: tokens per tile of embed_inproj_kernel / outproj_ffn_kernel
CE_ROWS, CE_IT = 128, 64  # ce_loss.cu: rows per CTA, items per chunk


def tn_slices(T):
    """train.cu:720-724: z-slices of the TN GEMM (and CTAs of the column sums)."""
    return -(-T // M_SLICE)


def ce_items_grid(T, rows, sms):
    """train.cu:760-766: the item pass of the CE backward, grid (item_tiles, ceil(T / m_per))."""
    item_tiles = -(-rows // CR)
    slices = (2 * sms + item_tiles - 1) // item_tiles
    max_slices = -(-T // (4 * CI))
    slices = max(1, min(slices, max_slices))
    m_per = -(-T // slices)
    return dict(item_tiles=item_tiles, slices=slices, max_slices=max_slices, m_per=m_per, y=-(-T // m_per))


def splits_for(M, rows, sms):
    """ce_loss.cu:147-156: item splits of the value path."""
    m_tiles = -(-M // CE_ROWS)
    chunks = -(-rows // CE_IT)
    want = (4 * sms + m_tiles - 1) // m_tiles
    max_splits = chunks // 8 if chunks // 8 > 0 else 1
    return max(1, min(want, max_splits, 64))


def encoder_grids(ids, sms):
    """encode.cu:562-601 for eval mode (last position only): compact tokens (positions from the first real item on;
    an empty row keeps its last position), embed_inproj tiles / CTAs, outproj_ffn last-only tiles / CTAs."""
    B, L = ids.shape
    real = ids > 0
    first = torch.where(real.any(1), real.int().argmax(1), torch.full((B,), L - 1))
    T = int((L - first).sum())
    return dict(tokens=T, inproj_tiles=-(-T // TOK), inproj_ctas=min(-(-B * L // TOK), 2 * sms),
                out_tiles=-(-B // TOK), out_ctas=min(-(-B // TOK), sms), levels=max(0, math.ceil(math.log2(L))))


def _library_sms():
    # what the library uses: the current device's SM count, 148 without a device
    return torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else SMS_WITHOUT_DEVICE


def test_splits_restatement_matches_the_library():
    """lrb_ce_workspace_bytes(M, rows) = M * (2 * splits + 1) * 4 + 256 (ce_loss.cu:163-169) on a grid of shapes,
    including the cap of 64 splits and the 512-items-per-split floor."""
    lib, sms = _lib.load(), _library_sms()
    seen = set()
    for M in (1, 90, 128, 129, 1200, 2048, 40000):
        for rows in (1, 63, 401, 4097, 8192, 12087, 40001, 1_000_001):
            s = splits_for(M, rows, sms)
            seen.add(s)
            assert lib.lrb_ce_workspace_bytes(M, rows) == M * (2 * s + 1) * 4 + 256, (M, rows, s)
    assert 1 in seen and 64 in seen and len(seen) >= 6


# ------------------------------------------------------------------------------------------------
# Inputs
# ------------------------------------------------------------------------------------------------
def make_weights(num_items, n_blocks=2, seed=5, table_scale=1.0):
    sd = synth.make_state_dict(num_items, n_blocks=n_blocks, seed=seed, bias_std=0.02, table_scale=table_scale)
    g = torch.Generator().manual_seed(seed + 1000)
    for k in sd:
        if k.endswith("layer_norm.weight"):
            sd[k] = 1.0 + 0.1 * torch.randn(64, generator=g)
        elif k.endswith("layer_norm.bias"):
            sd[k] = 0.05 * torch.randn(64, generator=g)
    return sd


def train_batch(B, L, num_items, seed, empty=(0,), full=(1,)):
    """Left-padded ids [B, L] and labels [B, L]: the next item, the held-out item last, 0 on padding.  Rows `empty`
    are all zero; rows `full` have a history in every position."""
    ids, last = synth.make_sequences(synth.Config("paths", B, num_items, L, B), seed=seed)
    rng = np.random.default_rng(seed)
    for b in full:
        ids[b] = torch.from_numpy(rng.integers(1, num_items + 1, size=L))
    for b in empty:
        ids[b] = 0
    labels = torch.zeros_like(ids)
    labels[:, :-1] = ids[:, 1:]
    labels[:, -1] = last
    labels[ids == 0] = 0
    return ids, labels


def holes_batch(B, L, num_items, seed):
    """Rows with holes (a zero after a real item): the general carry-set scan.  Row 0 is empty, row 1 full, row 2
    holds one item at position 0 only (a hole over the rest of the row), every third row from 3 loses some items
    after its first, and one row ends in a zero."""
    ids, _ = train_batch(B, L, num_items, seed, empty=(0,), full=(1,) if B > 1 else ())
    rng = np.random.default_rng(seed + 1)
    if L > 1:
        ids[2] = 0
        ids[2, 0] = int(rng.integers(1, num_items + 1))
        for b in range(3, B, 3):
            real = (ids[b] > 0).nonzero().view(-1).tolist()
            if len(real) < 2:
                continue
            drop = rng.choice(real[1:], size=max(1, len(real) // 3), replace=False)
            ids[b, torch.from_numpy(drop)] = 0
        ids[4, -1] = 0
        ids[4, 0] = 3
    return ids


def non_monotone_rows(ids):
    """Rows where a zero follows a real item."""
    m = ids > 0
    return int((m[:, :-1] & ~m[:, 1:]).any(1).sum())


# ------------------------------------------------------------------------------------------------
# Comparator
# ------------------------------------------------------------------------------------------------
def _as64(t):
    t = torch.as_tensor(t)
    return t.to(torch.complex128 if t.is_complex() else F64)


def grad_errors(got, want):
    """{name: e_k}, e_k = max|g - g_64| / max|g_64|.  A NaN anywhere in g gives e_k = NaN (torch's max propagates it);
    an all-zero reference gives 0 for an all-zero g and inf otherwise."""
    out = {}
    for k, w in want.items():
        w, g = _as64(w), _as64(got[k])
        assert g.shape == w.shape, (k, g.shape, w.shape)
        d, scale = float((g - w).abs().max()), float(w.abs().max())
        out[k] = d / scale if scale > 0 else (0.0 if d == 0 else math.inf)
    return out


def grad_failures(errors):
    """Tensors that miss the bar; NaN misses it too (no comparison with NaN is true)."""
    return {k: e for k, e in errors.items() if not e <= GRAD_BAR}


def _worst(errors):
    k = max(errors, key=lambda n: math.inf if math.isnan(errors[n]) else errors[n])
    return f"max e {errors[k]:.2e} ({k})"


def check_grads(case, loss, got, ids, labels, sd, mults=None, ignore_index=0):
    """Kernel loss / gradients against the fp64 oracle's autograd; prints e_k and the fp32 oracle's e_32."""
    loss64, want = DO.loss_and_grads(ids, labels, sd, mults, ignore_index, dtype=F64)
    loss32, ref32 = DO.loss_and_grads(ids, labels, sd, mults, ignore_index)
    e_k, e_32 = grad_errors(got, want), grad_errors(ref32, want)
    print(f"\n[{case}] loss rel err {abs(loss - loss64) / abs(loss64):.2e} (fp32 oracle "
          f"{abs(loss32 - loss64) / abs(loss64):.2e}); kernel e_k: {_worst(e_k)}; fp32 oracle e_32: {_worst(e_32)}")
    assert len(got) == len(want)
    assert abs(loss - loss64) <= LOSS_BAR * abs(loss64), (case, loss, loss64)
    bad = grad_failures(e_k)
    assert not bad, (case, bad)
    return loss64


def _args(num_items, n_blocks, p_embed=0.0, p_attn=0.0):
    return SimpleNamespace(num_items=num_items, bert_hidden_units=64, bert_num_blocks=n_blocks,
                           bert_dropout=p_embed, bert_attn_dropout=p_attn)


def _model(sd, p_embed=0.0, p_attn=0.0):
    n_blocks = O.n_blocks_of(sd)
    m = LRURec(_args(sd["model.bias"].shape[0] - 1, n_blocks, p_embed, p_attn))
    m.load_state_dict(sd)
    return m.cuda().train()


def kernel_step(m, ids, labels, **kw):
    m.zero_grad(set_to_none=True)
    loss = m.ce_loss(ids.cuda(), labels.cuda(), **kw)
    loss.backward()
    return loss.item(), {k: p.grad.detach().cpu() for k, p in m.named_parameters()}


# ------------------------------------------------------------------------------------------------
# Negative controls (CPU): the comparator fails on gradients perturbed the way each targeted bug would
# ------------------------------------------------------------------------------------------------
class _RecordingLinear:
    """Stands in for torch.nn.functional inside the oracle: records (weight, bias, output) of every F.linear."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        return getattr(torch.nn.functional, name)

    def linear(self, x, w, b=None):
        y = torch.nn.functional.linear(x, w, b)
        y.retain_grad()
        self.calls.append((w, b, y))
        return y


@pytest.fixture(scope="module")
def control_case():
    """The large-catalogue batch of test_large_catalogue_two_tn_slices (T = 1200) on a smaller catalogue."""
    sd = make_weights(3000, seed=21)
    ids, labels = train_batch(24, 50, 3000, seed=22, empty=(0, 11), full=(1, 12, 23))
    return sd, ids, labels, DO.loss_and_grads(ids, labels, sd, dtype=F64)[1]


def test_control_last_tn_slice_missing(control_case, monkeypatch):
    """(a) the last 1024-token slice's contribution dropped from in_proj / w_1 weights and biases."""
    sd, ids, labels, want = control_case
    B, L = ids.shape
    Lp = 1 << math.ceil(math.log2(L))
    rec = _RecordingLinear()
    monkeypatch.setattr(DO, "F", rec)
    leaves = {k: v.detach().to(O.complex_of(F64) if v.is_complex() else F64).requires_grad_(True)
              for k, v in sd.items()}
    DO.ce_loss_train(ids, labels, leaves).backward(retain_graph=True)
    tok = torch.arange(B * L).view(B, L) >= M_SLICE                          # kernel token b*L + l in the last slice
    last = torch.cat((torch.zeros(B, Lp - L, dtype=torch.bool), tok), 1).unsqueeze(-1)
    bad = {k: torch.from_numpy(v).clone() for k, v in want.items()}
    targets = {leaves[f"model.lru_blocks.{i}.{n}.weight"]: f"model.lru_blocks.{i}.{n}"
               for i in range(2) for n in ("lru_layer.in_proj", "feed_forward.w_1")}
    hit = 0
    for w, b, y in rec.calls:
        name = targets.get(w)
        if name is None or y.shape[1] != Lp:
            continue
        gw, gb = torch.autograd.grad(y, (w, b), grad_outputs=y.grad * last, retain_graph=True)
        bad[name + ".weight"] -= gw
        bad[name + ".bias"] -= gb
        hit += 1
    assert hit == 4
    errors = grad_errors(bad, want)
    failed = grad_failures(errors)
    assert set(failed) == {n + s for n in targets.values() for s in (".weight", ".bias")}, errors


@pytest.mark.parametrize("tile", ["first", "last"])
def test_control_one_item_tile_missing_its_ce_term(control_case, tile):
    """(b) one 128-item tile of the table / bias gradient without its CE-backward term: the hot first tile, and the
    ragged last tile of rare items, whose rows are small next to the hot ones (e_k is still about 0.08 there)."""
    sd, ids, labels, want = control_case
    sd64 = O.cast_state_dict(sd, F64)
    hid = O.hidden_states(ids, sd64).reshape(-1, 64)
    logits = hid @ sd64["embedding.token.weight"].t() + sd64["model.bias"]
    lab = labels.reshape(-1)
    counted = lab != 0
    G = torch.softmax(logits, -1)
    G[torch.arange(len(lab)), lab] -= 1.0
    G = G * counted.unsqueeze(1) / counted.sum()
    rows = logits.shape[1]
    n0 = 0 if tile == "first" else (rows - 1) // CR * CR
    sl = slice(n0, min(rows, n0 + CR))
    bad = {k: torch.from_numpy(v).clone() for k, v in want.items()}
    bad["embedding.token.weight"][sl] -= G[:, sl].t() @ hid
    bad["model.bias"][sl] -= G[:, sl].sum(0)
    failed = grad_failures(grad_errors(bad, want))
    assert set(failed) == {"embedding.token.weight", "model.bias"}, failed


def test_control_nan_and_zero_reference(control_case):
    """(d) one NaN element in a gradient (e.g. a ragged slice or tile that read unwritten workspace) fails the
    comparator, and so does a non-zero gradient where the reference is all zero; an all-zero pair passes."""
    _, _, _, want = control_case
    bad = {k: torch.from_numpy(v).clone() for k, v in want.items()}
    bad["model.lru_blocks.1.feed_forward.w_1.bias"][17] = float("nan")
    failed = grad_failures(grad_errors(bad, want))
    assert set(failed) == {"model.lru_blocks.1.feed_forward.w_1.bias"} and math.isnan(failed.popitem()[1])
    assert "nan" in _worst(grad_errors(bad, want))
    zero = {"w": np.zeros((5, 4))}
    assert grad_failures(grad_errors({"w": torch.full((5, 4), 1e-30, dtype=F64)}, zero)) == {"w": math.inf}
    assert grad_failures(grad_errors({"w": torch.zeros(5, 4, dtype=F64)}, zero)) == {}


def test_control_recurrence_gradient_without_mask(control_case, monkeypatch):
    """(c) the scan's backward without the mask: the forward value is the masked scan, the gradient that of the
    unmasked one, so gradient leaks across the masked positions (into the padding and the empty rows' neighbours)."""
    sd, ids, labels, want = control_case
    scan = O.tree_scan

    def scan_unmasked_backward(bu, lam, mask):
        free = scan(bu, lam, torch.ones_like(mask))
        return scan(bu, lam, mask).detach() + free - free.detach()

    monkeypatch.setattr(DO, "tree_scan", scan_unmasked_backward)
    _, bad = DO.loss_and_grads(ids, labels, sd, dtype=F64)
    failed = grad_failures(grad_errors(bad, want))
    assert "embedding.token.weight" in failed and "model.lru_blocks.0.lru_layer.in_proj.weight" in failed, failed


# ------------------------------------------------------------------------------------------------
# Train step (lrb_train_step / lrb_train_step_dropout through LRURec.ce_loss(...).backward())
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def large():
    """12 087 rows (95 item tiles, the last one 55 items), B = 24, L = 50: T = 1200."""
    sd = make_weights(12086, seed=31)
    ids, labels = train_batch(24, 50, 12086, seed=32, empty=(0, 11), full=(1, 12, 23))
    return sd, ids, labels


@pytest.mark.gpu
def test_large_catalogue_two_tn_slices(large):
    sd, ids, labels = large
    T, rows = ids.numel(), sd["model.bias"].shape[0]
    g = ce_items_grid(T, rows, _library_sms())
    assert tn_slices(T) == 2 and T % M_SLICE == 176 and g["item_tiles"] == 95 and rows % CR == 55 and g["slices"] > 1
    loss, got = kernel_step(_model(sd), ids, labels)
    check_grads("large catalogue, T=1200", loss, got, ids, labels, sd)


@pytest.mark.gpu
def test_large_catalogue_with_dropout(large):
    """Dropout at 0.2 (embedding, PFFN) / 0.3 (attention): the masked LayerNorm-backward copies and the GELU on two
    TN slices and 95 item tiles."""
    sd, ids, labels = large
    T = ids.numel()
    assert tn_slices(T) == 2 and ce_items_grid(T, sd["model.bias"].shape[0], _library_sms())["item_tiles"] == 95
    seed = _draw_seed(torch.Generator().manual_seed(77))
    loss, got = kernel_step(_model(sd, 0.2, 0.3), ids, labels, dropout=True, generator=torch.Generator().manual_seed(77))
    mults = DO.site_multipliers(seed, ids.shape[0], ids.shape[1], 2, 0.2, 0.3, 0.2)
    check_grads("large catalogue, dropout 0.2/0.3", loss, got, ids, labels, sd, mults)


@pytest.mark.gpu
@pytest.mark.parametrize("L,B", [(256, 8), (200, 6)])
def test_long_rows_on_golden_weights(golden_sd, L, B):
    """The scan forward / backward over 200 and 256 steps; T = 2048 (two full TN slices) and 1200 (a ragged one)."""
    ids, labels = train_batch(B, L, 400, seed=L, empty=(2,), full=(0, B - 1))
    T = B * L
    assert tn_slices(T) == 2 and L >= 200 and int((ids > 0).sum(1).max()) == L
    loss, got = kernel_step(_model(golden_sd), ids, labels)
    check_grads(f"long rows L={L}, T={T}", loss, got, ids, labels, golden_sd)


@pytest.mark.gpu
@pytest.mark.parametrize("n_blocks", [1, 3])
def test_other_block_counts(n_blocks):
    """1 and 3 blocks, B = 32, L = 40 (T = 1280: two TN slices).  The 3-block case also runs with int32 ids, which
    must give the int64 step's loss and gradients to 1e-6 (float atomics: not bitwise)."""
    sd = make_weights(2000, n_blocks=n_blocks, seed=40 + n_blocks)
    ids, labels = train_batch(32, 40, 2000, seed=41, empty=(5, 6), full=(0, 31))
    assert O.n_blocks_of(sd) == n_blocks != 2 and tn_slices(ids.numel()) == 2
    m = _model(sd)
    loss, got = kernel_step(m, ids, labels)
    check_grads(f"n_blocks={n_blocks}", loss, got, ids, labels, sd)
    if n_blocks == 3:
        loss32, got32 = kernel_step(m, ids.to(torch.int32), labels)
        assert abs(loss32 - loss) <= 1e-6 * max(1.0, abs(loss)), (loss32, loss)
        for k, g in got.items():
            scale = float(g.abs().max())
            assert torch.allclose(got32[k], g, rtol=1e-6, atol=1e-6 * scale + 1e-12), k


@pytest.mark.gpu
def test_eight_blocks_the_limit():
    sd = make_weights(400, n_blocks=MAX_BLOCKS, seed=48)
    ids, labels = train_batch(4, 20, 400, seed=48, empty=(3,), full=(0,))
    assert O.n_blocks_of(sd) == MAX_BLOCKS
    loss, got = kernel_step(_model(sd), ids, labels)
    check_grads("n_blocks=8", loss, got, ids, labels, sd)


@pytest.mark.gpu
def test_ignore_index_minus_100_counts_label_zero():
    """torch's default ignore_index: padding is labelled -100 and a label 0 (the padding item) is an ordinary class."""
    sd = make_weights(1500, seed=50)
    ids, labels = train_batch(20, 30, 1500, seed=51, empty=(4,), full=(0,))
    labels[ids == 0] = -100
    rng = np.random.default_rng(52)
    real = (ids > 0).nonzero()
    pick = real[torch.from_numpy(rng.choice(len(real), size=40, replace=False))]
    labels[pick[:, 0], pick[:, 1]] = 0
    assert int((labels == 0).sum()) == 40 and int((labels == -100).sum()) > 0
    loss, got = kernel_step(_model(sd), ids, labels, ignore_index=-100)
    loss64 = check_grads("ignore_index=-100", loss, got, ids, labels, sd, ignore_index=-100)
    assert abs(DO.ce_loss_train(ids, labels.clamp(min=0), sd, dtype=F64).item() - loss64) > 1e-3  # 0 is not ignored


@pytest.mark.gpu
@pytest.mark.parametrize("bad", ["rows", -5])
def test_out_of_range_labels_raise_in_the_train_step(bad):
    sd = make_weights(400, seed=60)
    ids, labels = train_batch(6, 20, 400, seed=60)
    labels[3, -1] = sd["model.bias"].shape[0] if bad == "rows" else bad
    with pytest.raises(LrbError) as e:
        kernel_step(_model(sd), ids, labels)
    assert e.value.code == -1 and "label" in str(e.value)


@pytest.mark.gpu
def test_out_of_range_labels_are_not_counted_by_the_value_path():
    """lrb_ce_loss_fwd does not synchronise: a label outside [0, rows) leaves the mean and gets row loss 0."""
    sd = make_weights(400, seed=61)
    ids, labels = train_batch(6, 20, 400, seed=61)
    rows = sd["model.bias"].shape[0]
    bad = labels.clone()
    bad[3, -1], bad[4, -1] = rows, -5
    with torch.no_grad():
        loss, row_loss = _model(sd).ce_loss(ids.cuda(), bad.cuda(), return_row_loss=True)
    ok = labels.clone()
    ok[3, -1] = ok[4, -1] = 0
    want = DO.ce_loss_train(ids, ok, sd, dtype=F64).item()
    assert abs(loss.item() - want) <= LOSS_BAR * abs(want), (loss.item(), want)
    assert float(row_loss[3, -1]) == 0.0 and float(row_loss[4, -1]) == 0.0


# ------------------------------------------------------------------------------------------------
# Value path (lrb_ce_loss_fwd: LRURec.ce_loss under no_grad)
# ------------------------------------------------------------------------------------------------
def check_value_path(case, sd, ids, labels):
    with torch.no_grad():
        loss, rows = _model(sd).ce_loss(ids.cuda(), labels.cuda(), return_row_loss=True)
    rows64 = DO.ce_loss_train(ids, labels, sd, dtype=F64, reduction="none").view(ids.shape)
    loss64 = float(rows64.sum() / (labels != 0).sum())
    err = float((rows.cpu().double() - rows64).abs().max())
    print(f"\n[{case}] loss rel err {abs(loss.item() - loss64) / abs(loss64):.2e}, row loss max abs err {err:.2e} "
          f"(largest row loss {float(rows64.abs().max()):.1f})")
    assert abs(loss.item() - loss64) <= LOSS_BAR * abs(loss64), (loss.item(), loss64)
    np.testing.assert_allclose(rows.cpu().double().numpy(), rows64.numpy(), rtol=LOSS_BAR,
                               atol=LOSS_BAR * float(rows64.abs().max()))
    return rows64


@pytest.mark.gpu
def test_value_path_row_losses_large_catalogue(large):
    sd, ids, labels = large
    s = splits_for(ids.numel(), sd["model.bias"].shape[0], _library_sms())
    assert 1 < s < 64
    check_value_path("value path, 12 087 rows", sd, ids, labels)


@pytest.mark.gpu
def test_value_path_logits_near_80():
    """A table scaled so the logits reach about 95 (and -50): exp() of them overflows an fp32 sum that is not
    max-shifted."""
    sd = make_weights(12086, seed=70, table_scale=72.0)
    ids, labels = train_batch(16, 30, 12086, seed=71)
    logits = O.forward_scores(ids, sd, F64)
    top = float(logits.abs().max())
    assert 60.0 <= top <= 120.0 and bool(torch.exp(logits.float()).sum(-1).isinf().any()), top
    check_value_path(f"value path, |logit| <= {top:.0f}", sd, ids, labels)


@pytest.mark.gpu
def test_value_path_many_splits():
    """M = 90 tokens on 40 001 rows: splits_for hits its cap of 64 splits, over 626 uneven item chunks."""
    sd = make_weights(40000, seed=80)
    ids, labels = train_batch(3, 30, 40000, seed=81, empty=(), full=(0,))
    M, rows = ids.numel(), sd["model.bias"].shape[0]
    assert splits_for(M, rows, _library_sms()) == 64 and -(-rows // CE_IT) % 64 != 0
    check_value_path("value path, 64 splits", sd, ids, labels)


# ------------------------------------------------------------------------------------------------
# Encoder (lrb_encode_fwd): all positions (hidden_states) and the last position (encode, with its bf16 copy)
# ------------------------------------------------------------------------------------------------
def check_encoder(case, m, sd, ids):
    ref = O.hidden_states(ids, sd, F64)
    hid = m.hidden_states(ids.cuda()).cpu()
    u, u16 = m.encode(ids.cuda(), want_bf16=True)
    u, u16 = u.cpu(), u16.cpu()
    ref32 = O.hidden_states(ids, sd)
    print(f"\n[{case}] all positions max abs err {float((hid.double() - ref).abs().max()):.2e}, last position "
          f"{float((u.double() - ref[:, -1]).abs().max()):.2e} (fp32 oracle {float((ref32.double() - ref).abs().max()):.2e})")
    np.testing.assert_allclose(hid.double().numpy(), ref.numpy(), atol=STATE_BAR, rtol=STATE_BAR)
    np.testing.assert_allclose(u.double().numpy(), ref[:, -1].numpy(), atol=STATE_BAR, rtol=STATE_BAR)
    assert torch.equal(u16, u.to(torch.bfloat16))
    # int32 ids: the same kernels read 4-byte ids; no atomics, so the states are bit for bit those of int64
    ids32 = ids.to(torch.int32).cuda()
    assert torch.equal(m.hidden_states(ids32).cpu(), hid)
    u_32, u16_32 = m.encode(ids32, want_bf16=True)
    assert torch.equal(u_32.cpu(), u) and torch.equal(u16_32.cpu(), u16)


ENCODER_CASES = [(L, 2) for L in (1, 2, 64, 65, 128, 129, 255, 256)] + [(1, 1), (65, 1), (37, 3), (256, 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("L,n_blocks", ENCODER_CASES)
def test_encoder_lengths_and_block_counts_with_holes(L, n_blocks):
    """L = 1 (no level) and 2; 2^k against 2^k + 1 (no left pad of the power-of-two frame against one of 2^k - 1) at
    6, 7 and 8 levels; 1 block (block 0 is both the gather/LN block and the last-only block) and 3 blocks."""
    ids = holes_batch(12, L, 500, seed=L + 10 * n_blocks)
    g = encoder_grids(ids, _library_sms())
    assert g["levels"] == max(0, math.ceil(math.log2(L))) and (L == 1 or non_monotone_rows(ids) >= 2)
    sd = make_weights(500, n_blocks=n_blocks, seed=90 + n_blocks)
    check_encoder(f"encoder L={L}, n_blocks={n_blocks}", _model(sd).eval(), sd, ids)


@pytest.mark.gpu
def test_encoder_eval_batch_beyond_one_wave():
    """B = 10 000 users: outproj_ffn (last-only) loops over 157 tiles on 148 CTAs and embed_inproj over the compact
    tokens on 296 CTAs.  Users are independent, so every 37th user against the fp64 oracle is an exact check."""
    sd = make_weights(3000, seed=95)
    ids, _ = train_batch(10000, 50, 3000, seed=96, empty=(0, 5000, 9999), full=(1, 7777))
    ids[::74, -1] = 0                            # every other compared user ends in a hole: the general carry-set scan
    g = encoder_grids(ids, _library_sms())
    assert g["out_tiles"] > g["out_ctas"] and g["inproj_tiles"] > g["inproj_ctas"] and g["tokens"] > 18944, g
    assert non_monotone_rows(ids[::37]) >= 50
    m = _model(sd).eval()
    u, u16 = m.encode(ids.cuda(), want_bf16=True)
    sub = ids[::37]
    ref = O.encode(sub, sd, F64)
    got = u[::37].cpu()
    print(f"\n[encoder B=10000] {g['tokens']} compact tokens, last position max abs err "
          f"{float((got.double() - ref).abs().max()):.2e} on {len(sub)} users")
    np.testing.assert_allclose(got.double().numpy(), ref.numpy(), atol=STATE_BAR, rtol=STATE_BAR)
    assert torch.equal(u16, u.to(torch.bfloat16))
