"""The training step's device kernels against float64 references on the CPU, at the shapes the benchmark trains.

Every comparison goes through ``assert_grad_close``: a relative Frobenius bound AND a relative max bound, neither with
a floor of 1, so a gradient whose entries are all far below 1 (most of XLNet's attention parameters at d = 64 / 256)
is still checked.  The helper also checks itself on every tensor it compares: the reference scaled by 1.01 and the
reference zeroed must both be rejected.

  B. the attention backward (warp form for dh = 16 / 32 / 64, item form, a head width without a warp form) and the
     dropout attention forward against float64 autograd of the attention formula itself;
  C. the whole fused step against the float64 oracle at benchmark-like widths / lengths with the default head chunk;
  D. the backward GEMMs at their real contraction lengths against a bound from the split-bf16 error model;
  E. the row / reduction kernels of the backward at their edges.

The tolerances were picked from errors measured on a B200 (1000 W power limit); each constant states the worst
error-to-tolerance ratio measured for its group.  ``T4R_TOL_REPORT=<file>`` writes the worst ratio of every test (and
the tensor it came from) to a JSON file.
"""
import json
import math
import os

import pytest
import torch
import torch.nn.functional as F

import t4r_oracle as O
from _util import make_pair, mlm_draws, synth_batch
from test_host_training_cpu import _pairs

pytestmark = [pytest.mark.gpu]


# ------------------------------------------------------------------------------------------------ A. the comparison
_WORST = {}


def _record(ratio, what):
    test = os.environ.get("PYTEST_CURRENT_TEST", "?").split(" ")[0]
    if float(ratio) >= _WORST.get(test, (0.0, ""))[0]:
        _WORST[test] = (float(ratio), what)


@pytest.fixture(scope="module", autouse=True)
def _tolerance_report():
    yield
    path = os.environ.get("T4R_TOL_REPORT")
    if path:
        old = json.load(open(path)) if os.path.exists(path) else {}
        old.update(_WORST)
        with open(path, "w") as f:
            json.dump(old, f, indent=1, sort_keys=True)


def _within(got, ref, rtol, atol_rel):
    diff = got - ref
    return bool(diff.norm() <= rtol * ref.norm()) and bool(diff.abs().max() <= atol_rel * ref.abs().max())


def assert_grad_close(name, got, ref, rtol, atol_rel):
    """``‖g − g_ref‖_F ≤ rtol ‖g_ref‖_F`` and ``max|g − g_ref| ≤ atol_rel max|g_ref|`` in float64.  A reference that is
    exactly zero needs an exactly zero product: every such case here is a sum over an empty set of terms (a parameter no
    masked row reaches), which the kernels produce as a literal 0."""
    ref = ref.detach().double().cpu()
    got = got.detach().double().cpu().reshape(ref.shape)
    assert torch.isfinite(got).all(), f"{name}: non-finite values"
    if not ref.any():
        assert not got.any(), f"{name}: reference gradient is exactly 0, product max |g| = {got.abs().max().item():.3e}"
        return
    assert not _within(1.01 * ref, ref, rtol, atol_rel), f"{name}: tolerance accepts the reference scaled by 1.01"
    assert not _within(0.0 * ref, ref, rtol, atol_rel), f"{name}: tolerance accepts a zero gradient"
    diff = got - ref
    fro = (diff.norm() / ref.norm()).item()
    mx = (diff.abs().max() / ref.abs().max()).item()
    _record(max(fro / rtol, mx / atol_rel), name)
    assert fro <= rtol and mx <= atol_rel, f"{name}: |err|_F / |ref|_F = {fro:.3e} (rtol {rtol:g}), max|err| / max|ref| = {mx:.3e} (atol_rel {atol_rel:g})"


# ------------------------------------------------------------------------------------------------ B. attention
# fp32 kernels (expf, sequential sums over dh and L) against float64.  Worst measured error-to-tolerance ratio on a
# B200 over every attention test: 0.09 (drr / drw of the relative forms at L = 50 / 64), a margin of ~10x; the bounds
# stay far below the 1 % the helper must reject.
ATTN_RTOL, ATTN_ATOL = 2e-5, 1e-4


def attn_ref64(qkv, R, rw, rr, dout, B, L, H, plm_mask=None, keep=None):
    """The attention formula in float64 with autograd: XLNet relative scores ``(q + r_w)·k_j + (q + r_r)·R[j + L − i]``
    (R, rw, rr given), GPT-2 causal scores (R None), both scaled by 1/sqrt(dh); ``plm_mask`` [B, L, L]: the two-stream
    form (rows of qkv / dout: content stream, then query stream; keys and values from the content rows; HF's
    ``score − 1e30 · mask`` where the mask is set, except on the content stream's diagonal).  ``keep`` [n_streams, B,
    H, L, L]: dropout keep scales of the probabilities.  -> (out, dqkv, dR, drw, drr)."""
    n_st = 2 if plm_mask is not None else 1
    d = qkv.shape[1] // 3
    dh = d // H
    qkv = qkv.detach().double().requires_grad_(True)
    x = qkv.view(n_st, B, L, 3, H, dh)
    q, k, v = x[:, :, :, 0], x[0, :, :, 1], x[0, :, :, 2]
    scale = 1.0 / math.sqrt(dh)
    ii, jj = torch.arange(L).view(L, 1), torch.arange(L).view(1, L)
    leaves = []
    if R is None:
        s = torch.einsum("sbihd,bjhd->sbhij", q, k) * scale
        s = s.masked_fill(jj > ii, float("-inf"))
    else:
        R, rw, rr = (t.detach().double().requires_grad_(True) for t in (R, rw, rr))
        leaves = [R, rw, rr]
        Rg = R.view(2 * L, H, dh)[jj + L - ii]                                      # [L(i), L(j), H, dh]
        s = (torch.einsum("sbihd,bjhd->sbhij", q + rw.view(H, dh), k) +
             torch.einsum("sbihd,ijhd->sbhij", q + rr.view(H, dh), Rg)) * scale
        if plm_mask is not None:
            m = plm_mask.bool().cpu().view(1, B, 1, L, L).expand(n_st, B, 1, L, L).clone()
            m[0, :, :, torch.arange(L), torch.arange(L)] = False
            s = s - 1e30 * m.double()
    p = torch.softmax(s, dim=-1)
    if keep is not None:
        p = p * keep.double().view(n_st, B, H, L, L)
    out = torch.einsum("sbhij,bjhd->sbihd", p, v).reshape(n_st * B * L, d)
    (out * dout.double()).sum().backward()
    return (out.detach(), qkv.grad) + tuple(t.grad for t in leaves)


def _keep_scales(n, p, seed, site):
    from transformers4rec_b200 import ops
    return ops.host_twin("dropout")(torch.ones(n), p, seed, site) if p > 0 else torch.ones(n)


def attn_case(form, B, L, H, dh, p, seed=0, ops_mod=None, device="cuda"):
    """Run the device attention (forward with dropped probabilities and backward) of one shape and compare it with
    ``attn_ref64``.  ``ops_mod`` / ``device`` let the same case run on the host twins (CPU rehearsal)."""
    if ops_mod is None:
        from transformers4rec_b200 import ops as ops_mod
    g = torch.Generator().manual_seed(1000 * L + 10 * dh + seed)
    d = H * dh
    n_st = 2 if form == "plm" else 1
    M = B * L
    qkv = torch.randn(n_st * M, 3 * d, generator=g)
    dout = torch.randn(n_st * M, d, generator=g)
    rel = form != "causal"
    R = torch.randn(2 * L, d, generator=g) if rel else None
    rw = 0.5 * torch.randn(d, generator=g) if rel else None
    rr = 0.5 * torch.randn(d, generator=g) if rel else None
    pm = None
    if form == "plm":
        pm = torch.rand(B, L, L, generator=g) < 0.4
        pm[0, 0, :] = True                 # a fully masked row: uniform probabilities in the query stream
    drop = (p, 977 + L, 18)
    keep = _keep_scales(n_st * B * H * L * L, p, drop[1], drop[2])
    ref_out, ref_dqkv, *ref_rel = attn_ref64(qkv, R, rw, rr, dout, B, L, H, plm_mask=pm, keep=keep)
    c = lambda t: None if t is None else t.to(device)
    tag = f"{form} B={B} L={L} H={H} dh={dh} p={p}"
    out = ops_mod.attn_drop_fwd(c(qkv), c(R), c(rw), c(rr), B, L, H, drop, plm_mask=c(pm))
    assert_grad_close(f"{tag} attn_drop_fwd", out, ref_out, ATTN_RTOL, ATTN_ATOL)
    if rel:
        dqkv, dR, drw, drr = ops_mod.xlnet_attn_bwd(c(qkv), c(R), c(rw), c(rr), c(dout), B, L, H, plm_mask=c(pm),
                                                    drop=drop if p > 0 else None)
        for name, got, want in zip(("dR", "drw", "drr"), (dR, drw, drr), ref_rel):
            assert_grad_close(f"{tag} {name}", got, want, ATTN_RTOL, ATTN_ATOL)
    else:
        dqkv = ops_mod.causal_attn_bwd(c(qkv), c(dout), B, L, H, drop=drop if p > 0 else None)
    got = dqkv.cpu().view(n_st, M, 3, d)
    want = ref_dqkv.view(n_st, M, 3, d)
    assert_grad_close(f"{tag} dq", got[:, :, 0], want[:, :, 0], ATTN_RTOL, ATTN_ATOL)
    assert_grad_close(f"{tag} dk", got[0, :, 1], want[0, :, 1], ATTN_RTOL, ATTN_ATOL)
    assert_grad_close(f"{tag} dv", got[0, :, 2], want[0, :, 2], ATTN_RTOL, ATTN_ATOL)
    if n_st == 2:   # keys / values come from the content stream only: the query stream's rows get no k / v gradient
        assert not got[1, :, 1:].any(), f"{tag}: query-stream dk / dv rows are not zero"


ATTN_LENGTHS = (1, 2, 20, 31, 32, 33, 50, 64)


@pytest.mark.parametrize("dh", (16, 32, 64))
@pytest.mark.parametrize("form", ("rel", "causal", "plm"))
def test_attention_backward_against_fp64(form, dh):
    """The warp form of the attention backward (the one the training step runs for dh = 16 / 32 / 64) over every
    sequence length class: one key slot (L <= 32), the second key slot (L = 33 .. 64), the edges 1 / 2 / 31 / 32."""
    for L in ATTN_LENGTHS:
        for p in (0.0, 0.3):
            attn_case(form, 3, L, 2, dh, p)


@pytest.mark.parametrize("form,B,L", [("rel", 2048, 20), ("causal", 2048, 20), ("rel", 512, 50), ("causal", 512, 50),
                                      ("plm", 512, 50)])
def test_attention_backward_fp64_filling_the_device(form, B, L):
    """Benchmark widths (d = 256, H = 8: dh = 32) with enough (session, head) items to fill the device."""
    attn_case(form, B, L, 8, 32, 0.3)


@pytest.mark.parametrize("form", ("rel", "causal", "plm"))
def test_attention_backward_item_form_fp64(monkeypatch, form):
    """The per-thread item form on the device (T4R_TRAIN_ATTN_ITEMS is read per call)."""
    monkeypatch.setenv("T4R_TRAIN_ATTN_ITEMS", "1")
    for L in (20, 33, 64):
        for p in (0.0, 0.3):
            attn_case(form, 5, L, 2, 32, p)


@pytest.mark.parametrize("form", ("rel", "causal", "plm"))
def test_attention_backward_fp64_head_width_without_warp_form(form):
    """d = 96, H = 4: dh = 24 has no warp instantiation, so the item form runs."""
    for L in (20, 50):
        for p in (0.0, 0.3):
            attn_case(form, 5, L, 4, 24, p)


# ------------------------------------------------------------------------------------------------ C. the whole step
# Product (split-bf16 GEMMs, fp32 everything else) against the float64 oracle.  The largest error comes from the head's
# dX_t GEMM over a full 32 768-column chunk (~1.2e-4 relative, see D), which every encoder gradient inherits.  Worst
# measured on a B200 over the six cases (label smoothing, layer 0's q): at most 1.5e-4 Frobenius and 7.6e-4 max
# relative, a ratio of 0.3 to these bounds; the loss is well inside LOSS_RTOL.
STEP_RTOL, STEP_ATOL, LOSS_RTOL = 5e-4, 3e-3, 1e-5


def _double_oracle(oracle):
    """The oracle in float64.  HF's two-stream XLNet builds its relative positions in fp32 and feeds them to the
    projection uncast (its one-stream path casts); cast them to the model's dtype, as the one-stream path does."""
    oracle.double()
    tr = oracle.transformer
    if hasattr(tr, "relative_positional_encoding"):
        pe = tr.relative_positional_encoding
        tr.relative_positional_encoding = lambda *a, **k: pe(*a, **k).to(torch.float64)
    return oracle


def _compare_step(oracle, model, ref_loss, loss, extra=()):
    assert abs(loss.item() - ref_loss.item()) <= LOSS_RTOL * abs(ref_loss.item()), (loss.item(), ref_loss.item())
    _record(abs(loss.item() - ref_loss.item()) / (LOSS_RTOL * abs(ref_loss.item())), "loss")
    checked = 0
    for name, po, pm in list(_pairs(oracle, model)) + list(extra):
        if po.grad is None and pm.grad is None:
            continue                      # parameters the path never touches (XLNet's segment embeddings)
        assert pm.grad is not None, name
        ref = po.grad if po.grad is not None else torch.zeros_like(po)
        assert_grad_close(name, pm.grad, ref.reshape(pm.grad.shape), STEP_RTOL, STEP_ATOL)
        checked += 1
    assert checked >= 15
    return checked


def _run_step(model, batch, **kw):
    from transformers4rec_b200.training import FusedTrainingStep
    step = FusedTrainingStep(model, **kw)
    assert step.head_chunk == 32768
    for prm in model.parameters():
        prm.grad = None
    loss = step.forward({k: v.cuda() for k, v in batch.items()})
    step.backward()
    return step, loss


def _clear_relu_kinks(oracle, model, batch):
    """ReLU's derivative jumps at 0, so a projection pre-activation within rounding of 0 may take different branches in
    the product and in float64 (one such entry in 10^5 moves a table row's gradient by several %).  Shift each channel's
    bias by at most 0.02 so that 0 sits in the middle of the widest gap between that channel's sorted pre-activations
    there: both branches stay exercised, and no entry is closer to the kink than half that gap."""
    tables = {n: oracle.tables[n.replace("/", "__")].weight for n in oracle.table_names}
    x = O.embed_concat(tables, {n: batch[n] for n in oracle.table_names}).reshape(-1, oracle.proj.in_features)
    pre = F.linear(x.double(), oracle.proj.weight.double(), oracle.proj.bias.double())
    v = pre.sort(0).values
    mid, gap = (v[1:] + v[:-1]) / 2, v[1:] - v[:-1]
    gap = gap.masked_fill(mid.abs() > 0.02, 0.0)
    shift = -mid.gather(0, gap.argmax(0, keepdim=True)).squeeze(0)
    lin = model.heads[0].body[0].projection_module[0][0]
    with torch.no_grad():
        oracle.proj.bias += shift.to(oracle.proj.bias.dtype)
        lin.bias.copy_(oracle.proj.bias)
    pre = F.linear(x.double(), oracle.proj.weight.double(), oracle.proj.bias.double())
    assert pre.abs().min().item() > 1e-4


def _mlm_case(cards, dims, d, H, NL, L, B, seed, arch="xlnet", masking="mlm", **kw):
    oracle, model = make_pair(cards, dims, "item_id/list", (), d, H, NL, L, arch=arch, masking=masking, weight_scale=0.08,
                              **kw)
    oracle.train(False)
    batch = synth_batch(B, L, cards, seed=seed)
    _clear_relu_kinks(oracle, model, batch)
    u, draws = mlm_draws(B, L, seed=seed + 1)
    model.heads[0].body[0].masking.set_draws(u.cuda())
    return _double_oracle(oracle), model, batch, draws


def test_step_fp64_config2_form():
    """XLNet MLM, d = 256, H = 8, L = 20, 2 layers, V = 50 001: the default head chunk (32 768) leaves a partial last
    chunk; T is not a multiple of 64."""
    oracle, model, batch, draws = _mlm_case({"item_id/list": 50_001, "category/list": 37},
                                            {"item_id/list": 256, "category/list": 64}, 256, 8, 2, 20, 40, seed=11)
    ref = oracle(batch, training=True, draws=draws)
    ref["loss"].backward()
    T = ref["labels"].numel()
    assert T % 64 != 0, T
    step, loss = _run_step(model, batch)
    assert step.T == T
    _compare_step(oracle, model, ref["loss"], loss)


def test_step_fp64_config5_form_sampled_with_accidental_hits():
    """XLNet MLM, d = 256, H = 8, L = 50, sampled softmax with 2 000 negatives; several labels are forced among the
    negatives (accidental hits: constant logits with no gradient)."""
    S = 2000
    oracle, model, batch, draws = _mlm_case({"item_id/list": 50_001}, {"item_id/list": 256}, 256, 8, 2, 50, 24, seed=21,
                                            sampled=True, max_n_samples=S)
    _, _, labels = oracle.input_block(batch, True, False, draws)
    y = labels[labels != 0]
    torch.manual_seed(4)
    raw = torch.multinomial(oracle.dist, 2 * S, replacement=True)
    raw[:8] = y.sort().values[:8]                     # small ids: they survive unique()[:S]
    neg = O.negatives_from_draws(raw, S)
    n_hits = int(torch.isin(y, neg).sum())
    assert n_hits >= 4, n_hits
    task = model.heads[0].prediction_task_dict["next-item"]
    task.set_negative_draws(raw.cuda())
    ref = oracle(batch, training=True, draws=draws, neg_samples=neg)
    ref["loss"].backward()
    _, loss = _run_step(model, batch)
    _compare_step(oracle, model, ref["loss"], loss)


def test_step_fp64_config3_form():
    """GPT-2 CLM, d = 256, H = 8, L = 20: the item id and six categorical side features (64 wide each) concatenated,
    Linear(448 -> 256) + ReLU, task_block Linear(256 -> 64) into the tied 64-wide item table."""
    cards = {"item_id/list": 50_001, "category/list": 337, "brand/list": 1000, "shop/list": 10000, "price_bin/list": 100,
             "weekday/list": 32, "hour_bin/list": 7}
    oracle, model, batch, draws = _mlm_case(cards, {n: 64 for n in cards}, 256, 8, 2, 20, 24, seed=31, arch="gpt2",
                                            masking="clm")
    assert oracle.task_block is not None
    ref = oracle(batch, training=True, draws=draws)
    ref["loss"].backward()
    _, loss = _run_step(model, batch)
    _compare_step(oracle, model, ref["loss"], loss)


def test_step_fp64_dh64_with_dropout(monkeypatch):
    """XLNet d = 256, H = 4 (dh = 64), dropout 0.1 at HF's sites: the oracle is the restated encoder carrying the
    same counter-based masks (host twin of the mask kernel)."""
    from transformers4rec_b200 import ops
    NL, H, p, seed = 2, 4, 0.1, 4242
    oracle, model, batch, draws = _mlm_case({"item_id/list": 50_001}, {"item_id/list": 256}, 256, H, NL, 20, 24, seed=41)
    enc = model.heads[0].body[1].transformer
    enc.config.dropout = p
    twin = ops.host_twin("dropout")

    def drop(site, t):
        return t * twin(torch.ones(t.numel()), p, seed, site).reshape(t.shape).to(t.dtype)

    monkeypatch.setattr(O, "hf_encoder_forward",
                        lambda hf, x: O.xlnet_forward_restated(x, dict(hf.named_parameters()), NL, H, drop=drop))
    ref = oracle(batch, training=True, draws=draws)
    ref["loss"].backward()
    from transformers4rec_b200.training import FusedTrainingStep
    step = FusedTrainingStep(model).set_dropout_seed(seed)
    enc.train()
    assert step.graph._rate() == p
    for prm in model.parameters():
        prm.grad = None
    loss = step.forward({k: v.cuda() for k, v in batch.items()})
    step.backward()
    _compare_step(oracle, model, ref["loss"], loss)


def test_step_fp64_plm():
    """PLM (two-stream XLNet) at d = 256, H = 8, L = 50."""
    cards = {"item_id/list": 50_001}
    oracle, model = make_pair(cards, {"item_id/list": 256}, "item_id/list", (), 256, 8, 2, 50, masking="plm",
                              weight_scale=0.08)
    oracle.train(False)
    enc = model.heads[0].body[1].transformer
    with torch.no_grad():
        enc.mask_emb.normal_(0.0, 0.5)
        oracle.transformer.mask_emb.copy_(enc.mask_emb.cpu())
    _double_oracle(oracle)
    B, L = 16, 50
    batch = synth_batch(B, L, cards, seed=51)
    _clear_relu_kinks(oracle, model, batch)
    g = torch.Generator().manual_seed(52)
    draws = {"u_span": torch.rand((B, L), generator=g), "u_start": torch.rand((B, L), generator=g),
             "u_force": torch.rand((B,), generator=g), "u_unmask": torch.rand((B,), generator=g),
             "perm": torch.stack([torch.randperm(L, generator=g) for _ in range(B)])}
    model.heads[0].body[0].masking.set_draws({k: v.cuda() for k, v in draws.items()})
    ref = oracle(batch, training=True, draws=draws)
    ref["loss"].backward()
    _, loss = _run_step(model, batch)
    _compare_step(oracle, model, ref["loss"], loss, extra=[("mask_emb", oracle.transformer.mask_emb, enc.mask_emb)])


def test_step_fp64_label_smoothing():
    """Label smoothing 0.1 on the full softmax (the smoothed target distribution in the head's backward, over two
    column chunks)."""
    oracle, model, batch, draws = _mlm_case({"item_id/list": 50_001}, {"item_id/list": 256}, 256, 8, 2, 20, 24, seed=61)
    model.heads[0].prediction_task_dict["next-item"].label_smoothing = 0.1
    out = oracle(batch, training=True, draws=draws)
    ref = F.cross_entropy(out["predictions"], out["labels"], label_smoothing=0.1)
    ref.backward()
    _, loss = _run_step(model, batch)
    _compare_step(oracle, model, ref, loss)


# ------------------------------------------------------------------------------------------------ D. backward GEMMs
def gemm_bound_c(K):
    """Error model of ``gemm_nt`` (three-product split-bf16, fp32 accumulation).  Each fp32 operand is a = a_hi + a_lo
    + e_a with bf16 planes (unit roundoff 2^-8), so |e_a| <= 2^-16 |a|; the kernel forms a_hi b_hi + a_hi b_lo +
    a_lo b_hi, which misses a_lo b_lo, e_a b and a e_b: at most 3 * 2^-16 |a| |b| per term (bf16 x bf16 products are
    exact in fp32).  The accumulator takes one fp32 rounding (2^-24) per K = 16 MMA step of each of the three products,
    plus the epilogue's residual add and the output rounding:
        |C_ij - (A B^T)_ij| <= c(K) (|A| |B|^T + |residual|)_ij,   c(K) = 3 * 2^-16 + (3 ceil(K / 16) + 2) * 2^-24."""
    return 3 * 2.0 ** -16 + (3 * math.ceil(K / 16) + 2) * 2.0 ** -24




def _gemm_case(M, N, K, residual, seed):
    from transformers4rec_b200.training import gemm_nt
    g = torch.Generator().manual_seed(seed)
    # gradient-like operands: signed, rows of different magnitudes (the split planes see a range of exponents)
    a = torch.randn(M, K, generator=g) * torch.exp(torch.randn(M, 1, generator=g))
    b = torch.randn(N, K, generator=g) * torch.exp(torch.randn(N, 1, generator=g))
    res = torch.randn(M, N, generator=g) * 10.0 if residual else None
    got = gemm_nt(a.cuda(), b.cuda(), residual=res.cuda() if residual else None).cpu().double()
    a64, b64 = a.double(), b.double()
    ref = a64 @ b64.t()
    env = a64.abs() @ b64.abs().t()
    if residual:
        ref += res.double()
        env += res.double().abs()
    err = (got - ref).abs()
    ratio = (err / (gemm_bound_c(K) * env)).max().item()
    _record(ratio, f"gemm ({M}, {N}, {K}) element-wise bound")
    assert ratio <= 1.0, f"({M}, {N}, {K}): error exceeds the split-bf16 bound by {ratio:.3f}x"
    # the element-wise bound alone would pass a result with a whole K block missing (|A| |B|^T grows like K, the result
    # like sqrt(K) for signed operands); the same c(K) as a Frobenius bound relative to the result is what keeps it sharp.
    # Measured on a B200: 1.4e-4 / 1.2e-4 relative at K = 40 960 / 32 768, a ratio of 0.28 to c(K).
    assert_grad_close(f"gemm ({M}, {N}, {K})", got, ref, gemm_bound_c(K), 2 * gemm_bound_c(K))


@pytest.mark.parametrize("M,N,K,residual", [
    (768, 256, 40_960, False),      # dW of Q|K|V at config 2: dy^T x over B L = 2048 * 20 rows
    (333, 256, 32_768, True),       # the head's dX_t += P W_c over a full default chunk (fused residual), T odd
    (32_768, 256, 333, False),      # the head's dW_c = P^T X_t: contraction over T
    (333, 200, 4_096, True),        # N % 32 != 0: the residual is added by a separate kernel
])
def test_backward_gemm_at_real_contraction_lengths(M, N, K, residual):
    _gemm_case(M, N, K, residual, seed=M + N + K)


# ------------------------------------------------------------------------------------------------ E. row kernels
# fp32 per-row / per-column loops against float64.  Worst measured ratio on a B200: 0.30 (LayerNorm's dgamma at
# d = 1024, a column sum over 40 967 rows); every other row kernel is below 0.05.
ROW_RTOL, ROW_ATOL = 1e-5, 1e-4


@pytest.mark.parametrize("d", (256, 1024))
def test_layer_norm_bwd_fp64(d):
    """M = 40 967 rows (not a multiple of the 256-row column-sum slab), a quarter of them nearly constant."""
    from transformers4rec_b200 import ops
    M, eps = 40_960 + 7, 0.03
    g = torch.Generator().manual_seed(d)
    x = torch.randn(M, d, generator=g)
    x[::4] = 2.0 + 1e-3 * torch.randn(x[::4].shape, generator=g)
    gamma = torch.rand(d, generator=g) + 0.5
    dy, add = torch.randn(M, d, generator=g), torch.randn(M, d, generator=g)
    dx, dg, db = ops.layer_norm_bwd(x.cuda(), gamma.cuda(), eps, dy.cuda(), add=add.cuda())
    x64 = x.double().requires_grad_(True)
    g64 = gamma.double().requires_grad_(True)
    b64 = torch.zeros(d, dtype=torch.float64, requires_grad=True)
    (F.layer_norm(x64, (d,), g64, b64, eps) * dy.double()).sum().backward()
    assert_grad_close(f"layer_norm_bwd d={d} dx", dx, x64.grad + add.double(), ROW_RTOL, ROW_ATOL)
    assert_grad_close(f"layer_norm_bwd d={d} dx (nearly constant rows)", (dx.cpu().double() - add.double())[::4],
                      x64.grad[::4], ROW_RTOL, ROW_ATOL)
    assert_grad_close(f"layer_norm_bwd d={d} dgamma", dg, g64.grad, ROW_RTOL, ROW_ATOL)
    assert_grad_close(f"layer_norm_bwd d={d} dbeta", db, b64.grad, ROW_RTOL, ROW_ATOL)


@pytest.mark.parametrize("M", (1, 255, 257))
def test_col_sum_fp64(M):
    from transformers4rec_b200 import ops
    x = torch.randn(M, 300, generator=torch.Generator().manual_seed(M))
    assert_grad_close(f"col_sum M={M}", ops.col_sum(x.cuda()), x.double().sum(0), ROW_RTOL, ROW_ATOL)


@pytest.mark.parametrize("smooth", (0.0, 0.1))
def test_softmax_ce_bwd_fp64_labels_at_chunk_edges(smooth):
    """One column chunk [v0, v0 + Vc) of a V-wide softmax; labels on its first and last column and outside it."""
    from transformers4rec_b200 import ops
    T, V, v0, Vc = 77, 5000, 1024, 2048
    g = torch.Generator().manual_seed(7)
    z = 3.0 * torch.randn(T, V, generator=g)
    lse = torch.logsumexp(z.double(), dim=1)
    labels = torch.randint(0, V, (T,), generator=g)
    labels[0::3], labels[1::3] = v0, v0 + Vc - 1
    scale = 1.0 / T
    got = ops.softmax_ce_bwd(z[:, v0:v0 + Vc].contiguous().cuda(), lse.float().cuda(), labels.cuda(), v0, scale,
                             label_smoothing=smooth, V_total=V)
    target = (1.0 - smooth) * F.one_hot(labels, V).double() + smooth / V
    ref = ((torch.softmax(z.double(), dim=1) - target) * scale)[:, v0:v0 + Vc]
    assert_grad_close(f"softmax_ce_bwd smooth={smooth}", got, ref, ROW_RTOL, ROW_ATOL)


def test_sampled_ce_bwd_fp64_with_hits():
    from transformers4rec_b200 import ops
    T, S, inv_tau = 65, 700, 1.0 / 0.7
    g = torch.Generator().manual_seed(8)
    col_ids = torch.randperm(20_000, generator=g)[:S].sort().values
    labels = torch.randint(1, 20_000, (T,), generator=g)
    labels[::4] = col_ids[torch.randint(0, S, (labels[::4].numel(),), generator=g)]     # accidental hits
    z = torch.randn(T, S, generator=g)
    bias = torch.rand(S, generator=g) * 5.0
    logits = z.double() + bias.double() * inv_tau
    hit = labels.view(T, 1) == col_ids.view(1, S)
    lse = torch.logsumexp(torch.cat([torch.randn(T, 1, generator=g).double(), logits.masked_fill(hit, -1e4)], 1), dim=1)
    scale = 1.0 / T
    got = ops.sampled_ce_bwd(z.cuda(), lse.float().cuda(), labels.cuda(), bias.cuda(), col_ids.cuda(), inv_tau, scale)
    ref = torch.exp(logits - lse.view(T, 1)).masked_fill(hit, 0.0) * scale
    assert hit.sum() >= 16
    assert not got.cpu()[hit].any()
    assert_grad_close("sampled_ce_bwd", got, ref, ROW_RTOL, ROW_ATOL)


def test_index_add_rows_fp64_duplicates_and_skip():
    from transformers4rec_b200 import ops
    n, V, width, ld, col = 5000, 300, 64, 200, 72
    g = torch.Generator().manual_seed(9)
    idx = torch.randint(0, V, (n,), generator=g)
    idx[::7] = 0                                  # the padding row: skipped
    idx[1::5] = 17                                # a heavily duplicated row
    src = torch.randn(n, ld, generator=g)
    dst = torch.randn(V, width, generator=g)
    got = ops.index_add_rows(dst.clone().cuda(), idx.cuda(), src.cuda(), col, width, skip_index=0)
    keep = idx != 0
    ref = dst.double().index_add(0, idx[keep], src[keep, col:col + width].double())
    assert torch.equal(got.cpu()[0], dst[0])
    assert_grad_close("index_add_rows", got, ref, ROW_RTOL, ROW_ATOL)
