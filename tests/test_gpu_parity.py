"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on
the same seeded inputs.  Bit-exact for integer/index work and pure copies,
1e-3 absolute (the north-star tolerance) for fp32 results -- in practice the
split-bf16 tensor-core products land near 1e-5."""
import math

import pytest
import torch

import t4r_oracle as O
from _util import make_pair, mlm_draws, synth_batch

pytestmark = pytest.mark.gpu
TOL = 1e-3


@pytest.fixture(scope="module")
def ops():
    from transformers4rec_b200 import ops as _ops
    return _ops


@pytest.mark.parametrize("M,N,K", [(128, 64, 64), (300, 64, 133), (1000, 192, 256), (257, 128, 64),
                                   (4096, 256, 256), (513, 1024, 256), (640, 256, 1024), (333, 100, 203),
                                   (130, 36, 100)])
@pytest.mark.parametrize("nprod", [3, 1])
def test_linear_matches_fp32(ops, M, N, K, nprod):
    torch.manual_seed(0)
    x = torch.randn(M, K, device="cuda")
    w = torch.randn(N, K, device="cuda") * 0.1
    b = torch.randn(N, device="cuda")
    xp, wp = ops.split_planes(x), ops.split_planes(w)
    y, yp, _ = ops.linear(xp, wp, K, bias=b, nprod=nprod)
    ref = ops.debug_sgemm_nt(x, w, b)
    ref_cpu = (x.double().cpu() @ w.double().cpu().t() + b.double().cpu()).float()
    assert (ref.cpu() - ref_cpu).abs().max() < 1e-3  # the SIMT reference itself
    tol = 2e-4 if nprod == 3 else 0.15
    err = (y.cpu() - ref_cpu).abs().max().item()
    assert err < tol, f"max err {err}"
    # planes output reproduces y: hi + lo
    rec = yp[0].float() + yp[1].float()
    assert (rec[:, :N] - y).abs().max().item() < 1e-3 * max(1.0, y.abs().max().item()) * 0.01 + 1e-4
    assert (rec[:, N:] == 0).all()  # zero padding of the planes up to a multiple of 64 columns


def test_linear_epilogues(ops):
    torch.manual_seed(1)
    M, N, K = 700, 256, 192
    x = torch.randn(M, K, device="cuda")
    w = torch.randn(N, K, device="cuda") * 0.1
    b = torch.randn(N, device="cuda")
    res = torch.randn(M, N, device="cuda")
    g, beta = torch.rand(N, device="cuda") + 0.5, torch.randn(N, device="cuda")
    mv = torch.randn(N, device="cuda")
    code = torch.randint(0, 3, (M,), device="cuda", dtype=torch.uint8)
    xp, wp = ops.split_planes(x), ops.split_planes(w)
    from transformers4rec_b200 import _lib
    # relu + mask
    y, _, _ = ops.linear(xp, wp, K, bias=b, act=_lib.ACT_RELU, row_code=code, mask_vec=mv)
    ref = torch.relu(x @ w.t() + b)
    ref = torch.where((code == 1).unsqueeze(1), mv.unsqueeze(0), ref)
    ref = torch.where((code == 2).unsqueeze(1), torch.zeros_like(ref), ref)
    assert (y - ref).abs().max().item() < 5e-4
    # gelu
    y, _, _ = ops.linear(xp, wp, K, bias=b, act=_lib.ACT_GELU)
    assert (y - torch.nn.functional.gelu(x @ w.t() + b)).abs().max().item() < 5e-4
    # residual + layernorm (+ pre-LN output)
    for eps in (0.03, 1e-5):
        y, yp, pre = ops.linear(xp, wp, K, bias=b, residual=res, ln=(g, beta), ln_eps=eps, want_pre_ln=True)
        t = x @ w.t() + b + res
        ref = torch.nn.functional.layer_norm(t, (N,), g, beta, eps)
        assert (pre - t).abs().max().item() < 5e-4
        assert (y - ref).abs().max().item() < 5e-4
        assert ((yp[0].float() + yp[1].float()) - y).abs().max().item() < 1e-4


@pytest.mark.parametrize("M,d", [(1, 64), (333, 64), (700, 128), (129, 256), (40960 // 8 + 5, 256)])
def test_fused_ffn(ops, M, d):
    """K7: LayerNorm(res + gelu(x W1^T + b1) W2^T + b2), intermediate kept in TMEM -- vs torch fp64."""
    torch.manual_seed(3)
    hidden = 4 * d
    x = torch.randn(M, d, device="cuda")
    w1 = torch.randn(hidden, d, device="cuda") * 0.08
    w2 = torch.randn(d, hidden, device="cuda") * 0.05
    b1, b2 = torch.randn(hidden, device="cuda") * 0.3, torch.randn(d, device="cuda") * 0.3
    g, beta = torch.rand(d, device="cuda") + 0.5, torch.randn(d, device="cuda")
    res = torch.randn(M, d, device="cuda")
    xp, w1p, w2p = ops.split_planes(x), ops.split_planes(w1), ops.split_planes(w2)
    xd = x.double()
    inner = torch.nn.functional.gelu(xd @ w1.double().t() + b1.double()) @ w2.double().t() + b2.double()
    for eps, residual in ((0.03, None), (1e-5, res)):
        y, yp, pre = ops.ffn(xp, w1p, b1, w2p, b2, (g, beta), eps, residual=residual, want_planes=True, want_pre_ln=True)
        t = inner + (xd if residual is None else residual.double())
        ref = torch.nn.functional.layer_norm(t, (d,), g.double(), beta.double(), eps)
        assert (pre - t.float()).abs().max().item() < 5e-4
        assert (y - ref.float()).abs().max().item() < 5e-4
        assert ((yp[0].float() + yp[1].float()) - y).abs().max().item() < 1e-4


@pytest.fixture
def kernel_variant(request, monkeypatch):
    """Select a non-default kernel through its environment switch (read per launch by the library)."""
    for k, v in request.param.items():
        monkeypatch.setenv(k, v)
    return request.param


@pytest.mark.parametrize("kernel_variant", [{"T4R_GEMM_2CTA": "0"}, {"T4R_GEMM_2CTA": "1"}], indirect=True,
                         ids=["gemm-1cta", "gemm-cta-pair"])
def test_kernel_variants_hold_parity(ops, kernel_variant):
    """Every GEMM flavour that can be selected (single-CTA, CTA pair = tcgen05 cta_group::2) against the same
    references as the defaults: plain GEMM with an odd shape, LayerNorm epilogue, fused FFN, one XLNet layer stack vs
    HF, and the head."""
    test_linear_matches_fp32(ops, 1000, 192, 256, 3)
    test_linear_matches_fp32(ops, 333, 100, 203, 3)
    test_linear_epilogues(ops)
    test_fused_ffn(ops, 700, 128)
    test_fused_ffn(ops, 40960 // 8 + 5, 256)
    test_xlnet_encoder_matches_hf(256, 8, 2, 16, 20)
    test_head_full_softmax(ops, 517, 30011, 256, 1.0)


@pytest.mark.parametrize("M,N,K", [(40960, 768, 256), (1000, 512, 256), (333, 256, 64), (257, 768, 128), (4096, 1024, 256)])
def test_planes_only_epilogue_matches_fp64(ops, M, N, K):
    """The planes-only dense epilogue (no fp32 output: the Q|K|V projection) against fp64, with and without bias + GELU
    in front, incl. partial row blocks (M % 32 != 0)."""
    from transformers4rec_b200 import _lib
    torch.manual_seed(M + N)
    x = torch.randn(M, K, device="cuda")
    w = torch.randn(N, K, device="cuda") * 0.1
    b = torch.randn(N, device="cuda")
    xp, wp = ops.split_planes(x), ops.split_planes(w)
    prod = x.double() @ w.double().t()
    for ref, kw in ((prod, {}), (torch.nn.functional.gelu(prod + b.double()), dict(bias=b, act=_lib.ACT_GELU))):
        _, planes, _ = ops.linear(xp, wp, K, want_f32=False, want_planes=True, **kw)
        got = planes[0].double() + planes[1].double()
        assert (got[:, :N] - ref).abs().max().item() < 2e-3 * max(1.0, ref.abs().max().item())


def test_forward_replayed_from_a_cuda_graph():
    """Model.graphed: the forward-only pass captured once and replayed -- same loss and label ranks as the eager call on
    the same draws, new inputs take effect through the captured buffers, a shape change is refused."""
    cards, dims = {"item_id/list": 3001, "category/list": 37}, {"item_id/list": 64, "category/list": 64}
    B, L = 48, 20
    oracle, model = make_pair(cards, dims, "item_id/list", (), 64, 4, 2, L, weight_scale=0.08)
    u, draws = mlm_draws(B, L)
    model.heads[0].body[0].masking.set_draws(u.cuda())
    b1 = {k: v.cuda() for k, v in synth_batch(B, L, cards, seed=1).items()}
    b2 = {k: v.cuda() for k, v in synth_batch(B, L, cards, seed=2).items()}
    with torch.no_grad():
        e1 = model(b1, training=True)["loss"].item()
        e2 = model(b2, training=True)["loss"].item()
        ev = model(b2, training=False, testing=True)
        ev_loss, ev_rank = ev["loss"].item(), ev.row_rank.clone()
    g = model.graphed(b1, training=True)
    assert abs(g(b1).item() - e1) < 1e-6 and abs(g(b2).item() - e2) < 1e-6 and abs(g(b1).item() - e1) < 1e-6
    assert abs(e1 - e2) > 1e-4
    ref = oracle(synth_batch(B, L, cards, seed=2), training=True, draws=draws)["loss"].item()
    assert abs(g(b2).item() - ref) < 1e-3
    ge = model.graphed(b1, training=False, testing=True)
    assert abs(ge(b2).item() - ev_loss) < 1e-6 and torch.equal(ge.row_rank, ev_rank)
    with pytest.raises(ValueError):
        g({k: v[:8] for k, v in b1.items()})


def test_unsupported_shapes_fail_loudly():
    """no silent fallback: shapes outside the kernels' envelope raise T4RError with the limit in the message"""
    import transformers4rec_b200.torch as tr
    from transformers4rec_b200 import T4RError
    hf = O.build_hf_xlnet(64, 4, 1).eval()
    blk = tr.TransformerBlock(hf).cuda()
    with pytest.raises(T4RError, match="1..64"):
        blk(torch.randn(2, 65, 64, device="cuda"))
    with pytest.raises(T4RError, match="d_model must be 64, 128 or 256"):
        tr.TransformerBlock(O.build_hf_xlnet(96, 4, 1).eval()).cuda()(torch.randn(2, 8, 96, device="cuda"))


def test_embed_concat_bit_exact(ops):
    cards = {"item": 1001, "cat": 37, "brand": 500}
    dims = {"item": 64, "cat": 13, "brand": 32}
    batch = synth_batch(64, 20, cards, continuous=("price", "age"), seed=3)
    torch.manual_seed(4)
    tables = {n: torch.randn(c, dims[n]) for n, c in cards.items()}
    ref = O.embed_concat(tables, {n: batch[n] for n in cards}, {n: batch[n] for n in ("price", "age")})
    names = sorted(list(cards) + ["price", "age"])
    col, cats, conts = 0, [], []
    for n in names:
        if n in cards:
            cats.append((tables[n].cuda(), batch[n].cuda().reshape(-1), col)); col += dims[n]
        else:
            conts.append((batch[n].cuda().reshape(-1), col)); col += 1
    of, planes, err = ops.embed_concat(cats, conts, 64 * 20, col, True, True)
    assert torch.equal(of.cpu().view(64, 20, col), ref)
    assert int(err.item()) == 0
    rec = (planes[0].float() + planes[1].float()).cpu()
    assert (rec[:, :col] - ref.view(-1, col)).abs().max().item() < 1e-4
    assert (rec[:, col:] == 0).all()


@pytest.mark.parametrize("mode", ["train", "eval_last", "eval_all", "inference"])
def test_mask_mlm_bit_exact(ops, mode):
    from transformers4rec_b200 import _lib
    B, L = 257, 20
    ids = synth_batch(B, L, {"item": 5000}, seed=5, min_len=1)["item"]
    ids[3] = 0  # an empty session
    u, draws = mlm_draws(B, L, seed=6)
    kw = dict(train=(True, False), eval_last=(False, True), eval_all=(False, True), inference=(False, False))[mode]
    rm, rl = O.mlm_compute_masked_targets(ids, kw[0], kw[1], eval_on_last_item_seq_only=(mode != "eval_all"), **draws)
    code = dict(train=_lib.MLM_TRAIN, eval_last=_lib.MLM_EVAL_LAST, eval_all=_lib.MLM_EVAL_ALL,
                inference=_lib.MLM_INFERENCE)[mode]
    m, l, rc = ops.mask_mlm(ids.cuda(), code, 0, 0.15, u.cuda())
    assert torch.equal(l.cpu(), rl) and torch.equal(m.cpu(), rm)
    assert torch.equal(rc.cpu().bool(), rm)


@pytest.mark.parametrize("mode", ["all", "last", "inference"])
def test_mask_clm_bit_exact(ops, mode):
    from transformers4rec_b200 import _lib
    B, L = 130, 20
    ids = synth_batch(B, L, {"item": 5000}, seed=7, min_len=1)["item"]
    ids[5] = 0
    if mode == "all":
        rm, rl = O.clm_compute_masked_targets(ids, True, False)
    elif mode == "last":
        rm, rl = O.clm_compute_masked_targets(ids, False, True)
    else:
        rm, rl = O.clm_compute_masked_targets(ids, False, False)
    code = dict(all=_lib.CLM_ALL, last=_lib.CLM_LAST, inference=_lib.CLM_INFERENCE)[mode]
    m, l, rc = ops.mask_clm(ids.cuda(), code, 0)
    assert torch.equal(l.cpu(), rl) and torch.equal(m.cpu(), rm)
    # row codes reproduce apply_mask_to_inputs
    x = torch.randn(B, L, 8)
    emb = torch.randn(8)
    ref = O.clm_apply_mask_to_inputs(x, rm, emb, training=(mode == "all"), testing=(mode == "last"))
    rcc = rc.cpu()
    got = torch.where((rcc == 1).unsqueeze(-1), emb, x)
    got = torch.where((rcc == 2).unsqueeze(-1), torch.zeros_like(x), got)
    assert torch.equal(got, ref)


@pytest.mark.parametrize("B,L,keep", [(300, 20, 0.2), (2048, 20, 0.13), (1, 1, 1.0), (1, 3, 0.0), (7, 5, 1.0),
                                      (33, 31, 0.5), (2048, 50, 0.1), (52, 20, 0.9)])
def test_compact_targets(ops, B, L, keep):
    """row-major order of the non-padding labels, device-side count, zero tail -- from one label to config 5's 102 400,
    none / all of them labels, sizes around the kernel's 32-label steps and 1024-label rounds"""
    torch.manual_seed(8 + B)
    labels = torch.randint(1, 10**9, (B, L))
    labels[torch.rand(B, L) >= keep] = 0
    rows, labs, count = ops.compact_targets(labels.cuda(), 0)
    T = int(count.item())
    flat = labels.flatten()
    nz = flat.nonzero().squeeze(1)
    assert T == nz.numel()
    assert torch.equal(rows[:T].cpu().long(), nz) and torch.equal(labs[:T].cpu(), flat[nz])
    assert (rows[T:] == 0).all() and (labs[T:] == 0).all()


@pytest.mark.parametrize("d,H,NL,B,L", [(64, 4, 2, 33, 20), (256, 8, 2, 16, 20), (128, 8, 1, 9, 50), (64, 1, 1, 5, 21),
                                        (64, 4, 1, 1, 2), (64, 2, 1, 3, 64), (256, 4, 1, 2, 30), (128, 4, 1, 7, 31),
                                        (256, 8, 2, 128, 20), (64, 4, 3, 256, 20), (128, 8, 1, 64, 50),
                                        (256, 8, 1, 60, 20), (64, 4, 1, 7, 20)])
def test_xlnet_encoder_matches_hf(d, H, NL, B, L):
    """incl. the edges: one session of two items, the longest supported sequence (64, FFMA attention), the last length
    of the tensor-path attention (30) and the first of the fallback (31), dh = 64; batches of several 256-row CTA-pair
    tiles, and a partial one.  Two calls on the same input must agree bit for bit."""
    import transformers4rec_b200.torch as tr
    torch.manual_seed(10)
    hf = O.build_hf_xlnet(d, H, NL).eval()
    with torch.no_grad():
        for n, p in hf.named_parameters():
            if "layer_norm" in n:
                p.add_(torch.randn_like(p) * 0.1)
            else:
                p.normal_(0.0, 0.08)
    blk = tr.TransformerBlock(hf).cuda()
    x = torch.randn(B, L, d)
    with torch.no_grad():
        ref = O.hf_encoder_forward(hf, x)
        ref2 = O.xlnet_forward_restated(x, hf.state_dict(), NL, H)
        got = blk(x.cuda()).cpu()
        again = blk(x.cuda()).cpu()
    assert torch.equal(got, again)
    assert (ref - ref2).abs().max().item() < 3e-4  # HF vs the restated math, both CPU fp32 (different op order)
    err = (got - ref).abs().max().item()
    assert err < TOL, f"max abs err {err}"


@pytest.mark.parametrize("d,H,NL,B,L", [(64, 4, 2, 33, 20), (256, 8, 2, 16, 20), (128, 2, 1, 7, 40), (64, 4, 1, 1, 2),
                                        (64, 1, 1, 2, 64), (128, 4, 1, 5, 32), (128, 4, 1, 5, 33)])
def test_gpt2_encoder_matches_hf(d, H, NL, B, L):
    import transformers4rec_b200.torch as tr
    torch.manual_seed(11)
    hf = O.build_hf_gpt2(d, H, NL, L).eval()
    with torch.no_grad():
        for n, p in hf.named_parameters():
            if "ln_" in n:
                p.add_(torch.randn_like(p) * 0.1)
            else:
                p.normal_(0.0, 0.08)
    blk = tr.TransformerBlock(hf).cuda()
    x = torch.randn(B, L, d)
    with torch.no_grad():
        ref = O.hf_encoder_forward(hf, x)
        ref2 = O.gpt2_forward_restated(x, hf.state_dict(), NL, H)
        got = blk(x.cuda()).cpu()
    assert (ref - ref2).abs().max().item() < 3e-4  # HF vs the restated math, both CPU fp32 (different op order)
    err = (got - ref).abs().max().item()
    assert err < TOL, f"max abs err {err}"


@pytest.mark.parametrize("T,V,De,tau", [(200, 10001, 64, 1.0), (517, 30011, 256, 1.0), (64, 999, 128, 0.5)])
def test_head_full_softmax(ops, T, V, De, tau):
    torch.manual_seed(12)
    xt = torch.randn(T, De)
    W = torch.randn(V, De) * 0.1
    y = torch.randint(1, V, (T,))
    ref_loss, ref_logits = O.full_softmax_head(xt, y, W, tau)
    cap = T + 37
    xt_pad = torch.zeros(cap, De); xt_pad[:T] = xt
    y_pad = torch.zeros(cap, dtype=torch.long); y_pad[:T] = y
    count = torch.tensor([T], dtype=torch.int32, device="cuda")
    xp = ops.split_planes(xt_pad.cuda())
    wp = ops.split_planes(W.cuda())
    res = ops.head_softmax_ce(xp, xt_pad.cuda(), y_pad.cuda(), wp, W.cuda(), t_dev=count, inv_temperature=1.0 / tau,
                              want_rank=True)
    assert abs(res["loss"].item() - ref_loss.item()) < 1e-4
    ref_lse = torch.logsumexp(ref_logits, dim=1)
    assert (res["row_lse"][:T].cpu() - ref_lse).abs().max().item() < 1e-4
    # ranks -> Recall@k against the reference's one-hot/topk formulation
    ks = [1, 5, 10, 20]
    ref_rec = O.recall_at_mean(ks, ref_logits, y)
    got_rec = ops.recall_from_ranks(res["row_rank"], ks, count).cpu()
    assert (got_rec - ref_rec).abs().max().item() < 1e-6
    # materialised logits
    logits = ops.head_logits(xp, wp, De, t_dev=count, inv_temperature=1.0 / tau)[:T].cpu()
    assert (logits - ref_logits).abs().max().item() < 2e-4


def test_head_sampled_softmax(ops):
    torch.manual_seed(13)
    T, V, De, S = 300, 20001, 64, 500
    xt = torch.randn(T, De)
    W = torch.randn(V, De) * 0.1
    y = torch.randint(1, V, (T,))
    dist = O.log_uniform_distr(V, 1)
    udist = O.unique_sampling_distr(dist, 2 * S)
    raw = torch.multinomial(dist, 2 * S, replacement=True)
    neg = O.negatives_from_draws(raw, S)
    neg[:5] = y[:5].sort().values  # force accidental hits
    neg = neg.unique()
    ref_loss, ref_logits = O.sampled_softmax_head(xt, y, W, neg, udist, 1.0)
    nlq = (-torch.log(udist + 1e-16)).cuda()
    xp = ops.split_planes(xt.cuda())
    negp, _ = ops.gather_rows_split(W.cuda(), neg.cuda(), None, neg.numel(), want_f32=False)
    pos = ops.label_logit(xt.cuda(), W.cuda(), y.cuda(), class_bias=nlq)
    assert (pos.cpu() - ref_logits[:, 0]).abs().max().item() < 1e-4
    res = ops.head_softmax_ce(xp, xt.cuda(), y.cuda(), negp, None, col_bias=nlq[neg.cuda()].contiguous(),
                              col_ids=neg.cuda(), hit_value=float(torch.finfo(torch.float16).min / 100.0), pos_logit=pos)
    assert abs(res["loss"].item() - ref_loss.item()) < 1e-4


def _run_pair(oracle, model, batch, training, testing, draws_u=None, draws=None):
    dev = {k: v.cuda() for k, v in batch.items()}
    inputs = model.heads[0].body[0]
    if draws_u is not None:
        inputs.masking.set_draws(draws_u.cuda())
    with torch.no_grad():
        ref = oracle(batch, training=training, testing=testing, draws=draws)
        out = model(dev, training=training, testing=testing)
    return ref, out


@pytest.mark.parametrize("arch,masking", [("xlnet", "mlm"), ("xlnet", "clm"), ("gpt2", "clm")])
def test_model_end_to_end_config1(arch, masking):
    """BASELINE configs[0]: yoochoose-like schema, 10K items, L=20, d=64, 2 layers."""
    cards = {"item_id/list": 10001, "category/list": 337}
    dims = {"item_id/list": 64, "category/list": 64}
    cont = tuple(f"cont{i}/list" for i in range(5))
    B, L = 96, 20
    oracle, model = make_pair(cards, dims, "item_id/list", cont, 64, 4, 2, L, arch=arch, masking=masking,
                              weight_scale=0.08)
    batch = synth_batch(B, L, cards, cont, seed=0)
    u, draws = mlm_draws(B, L)
    ref, out = _run_pair(oracle, model, batch, True, False, u if masking == "mlm" else None,
                         draws if masking == "mlm" else None)
    inputs = model.heads[0].body[0]
    assert torch.equal(inputs.masking.masked_targets.cpu(), ref["masked_targets"])
    assert torch.equal(inputs.masking.mask_schema.cpu(), ref["mask_schema"])
    assert torch.equal(out["labels"].cpu(), ref["labels"])
    assert abs(out["loss"].item() - ref["loss"].item()) < TOL
    assert (out["predictions"].cpu() - ref["predictions"]).abs().max().item() < TOL
    # evaluation: last item only, Recall@k
    ref_e, out_e = _run_pair(oracle, model, batch, False, True)
    assert abs(out_e["loss"].item() - ref_e["loss"].item()) < TOL
    ks = [10, 20]
    ref_rec = O.recall_at_mean(ks, ref_e["predictions"], ref_e["labels"])
    got = model.calculate_metrics(out_e)
    key = [k for k in got if k.endswith("recall_at")][0]
    assert (got[key].cpu() - ref_rec).abs().max().item() < 1e-6


def test_model_hidden_states_xlnet_base():
    """BASELINE configs[1] shape at a reduced table/batch: d=256, 8 heads, 4 layers."""
    cards = {"item_id/list": 50001}
    dims = {"item_id/list": 256}
    B, L = 48, 20
    oracle, model = make_pair(cards, dims, "item_id/list", (), 256, 8, 4, L, weight_scale=0.05)
    batch = synth_batch(B, L, cards, seed=0)
    u, draws = mlm_draws(B, L)
    ref, out = _run_pair(oracle, model, batch, True, False, u, draws)
    body = model.heads[0].body
    with torch.no_grad():
        body[0].masking.set_draws(u.cuda())
        hid = body({k: v.cuda() for k, v in batch.items()}, training=True).cpu()
    assert (hid - ref["hidden"]).abs().max().item() < TOL
    assert abs(out["loss"].item() - ref["loss"].item()) < TOL


def test_model_sampled_softmax():
    cards = {"item_id/list": 20001}
    dims = {"item_id/list": 64}
    B, L, S = 64, 20, 400
    oracle, model = make_pair(cards, dims, "item_id/list", (), 64, 4, 1, L, sampled=True, max_n_samples=S,
                              weight_scale=0.08)
    batch = synth_batch(B, L, cards, seed=1)
    u, draws = mlm_draws(B, L)
    torch.manual_seed(3)
    raw = torch.multinomial(oracle.dist, 2 * S, replacement=True)
    neg = O.negatives_from_draws(raw, S)
    task = model.heads[0].prediction_task_dict["next-item"]
    task.set_negative_draws(raw.cuda())
    model.heads[0].body[0].masking.set_draws(u.cuda())
    with torch.no_grad():
        ref = oracle(batch, training=True, draws=draws, neg_samples=neg)
        out = model({k: v.cuda() for k, v in batch.items()}, training=True)
    assert abs(out["loss"].item() - ref["loss"].item()) < TOL
    assert (out["predictions"].cpu() - ref["predictions"]).abs().max().item() < TOL


def test_inference_topk():
    cards = {"item_id/list": 3001}
    dims = {"item_id/list": 64}
    B, L = 32, 20
    oracle, model = make_pair(cards, dims, "item_id/list", (), 64, 4, 1, L, weight_scale=0.08)
    batch = synth_batch(B, L - 1, cards, seed=2)  # room for the extra [MASK] position
    batch = {k: torch.nn.functional.pad(v, (0, 1)) for k, v in batch.items()}
    with torch.no_grad():
        x, mask, labels = oracle.input_block(batch, False, False)
        h = O.hf_encoder_forward(oracle.transformer, x)
        ids = batch["item_id/list"]
        last = (ids != 0).sum(1)
        hs = h[torch.arange(B), last]
        ref_scores = hs @ oracle.item_table().t()
        scores = model({k: v.cuda() for k, v in batch.items()}, training=False, testing=False).cpu()
    assert (scores - ref_scores).abs().max().item() < TOL
    model.top_k = 10
    with torch.no_grad():
        s, i = model({k: v.cuda() for k, v in batch.items()}, training=False, testing=False)
    rs, ri = torch.topk(ref_scores, 10)
    assert (s.cpu() - rs).abs().max().item() < TOL
    assert (i.cpu() == ri).float().mean().item() > 0.98


def test_padding_known_answers_on_gpu():
    """The reference's padding known answers (tests/unit/utils/test_padding.py:34-151) through
    t4r_pad_ragged, plus a randomised comparison with the oracle."""
    from itertools import accumulate

    import transformers4rec_b200.torch as tr

    def vo(data, dtype=torch.int64):
        vals = [x for row in data for x in row]
        return torch.tensor(vals, dtype=dtype).cuda(), torch.tensor([0] + list(accumulate(len(r) for r in data))).cuda()

    v, o = vo([[1, 2], [], [3, 4, 5]])
    out = tr.pad_batch({"a__values": v, "a__offsets": o, "b": torch.tensor([[3, 6], [4, 1], [8, 4]]).cuda()}, {"a": 7, "b": 3})
    assert torch.equal(out["a"].cpu(), torch.tensor([[1, 2, 0, 0, 0, 0, 0], [0] * 7, [3, 4, 5, 0, 0, 0, 0]]))
    assert torch.equal(out["b"].cpu(), torch.tensor([[3, 6, 0], [4, 1, 0], [8, 4, 0]]))
    v, o = vo([[1, 2], [], [3, 4, 5, 4, 7]])
    out = tr.pad_batch({"a__values": v, "a__offsets": o, "b": torch.tensor([[1, 2, 3, 4], [6, 7, 8, 9]]).cuda()}, {"a": 3, "b": 2})
    assert torch.equal(out["a"].cpu(), torch.tensor([[1, 2, 0], [0, 0, 0], [3, 4, 5]]))
    assert torch.equal(out["b"].cpu(), torch.tensor([[1, 2], [6, 7]]))
    v, o = vo([[1, 2, 3, 4, 5], [6, 7, 8, 9]])
    b = torch.tensor([[3, 6], [4, 1]]).cuda()
    out = tr.pad_inputs({"a__values": v, "a__offsets": o, "b": b}, max_sequence_length=3)
    assert torch.equal(out["a"].cpu(), torch.tensor([[1, 2, 3], [6, 7, 8]])) and torch.equal(out["b"], b)
    with pytest.raises(ValueError, match="unspecified padding length"):
        tr.pad_batch({"a__values": v, "a__offsets": o}, {})
    # randomised, int64 ids and fp32 continuous values
    g = torch.Generator().manual_seed(9)
    lens = torch.randint(0, 30, (500,), generator=g)
    offs = torch.cat([torch.zeros(1, dtype=torch.long), lens.cumsum(0)])
    ids = torch.randint(1, 1000, (int(offs[-1]),), generator=g)
    fl = torch.rand(int(offs[-1]), generator=g)
    got = tr.pad_inputs({"i__values": ids.cuda(), "i__offsets": offs.cuda(), "f__values": fl.cuda(), "f__offsets": offs.cuda()}, 20)
    ref = O.pad_inputs({"i__values": ids, "i__offsets": offs, "f__values": fl, "f__offsets": offs}, 20)
    assert torch.equal(got["i"].cpu(), ref["i"]) and torch.equal(got["f"].cpu(), ref["f"])


def test_reference_fixture_body_with_standalone_mlp_and_ragged_inputs():
    """The reference's canonical model fixture (tests/unit/torch/_conftest.py:143-155):
    inputs(d_output=100, masking="causal") >> MLPBlock([64]) >> XLNet(d=64, 4 heads, 2 layers)
    >> NextItemPredictionTask(weight_tying=True); fed with ragged __values/__offsets inputs."""
    import transformers4rec_b200.torch as tr
    torch.manual_seed(21)
    cards = {"item_id/list": 5001, "category/list": 333}
    schema = tr.Schema([tr.ColumnSchema.create_categorical("item_id/list", 5000, tags=[tr.Tags.ITEM_ID]),
                        tr.ColumnSchema.create_categorical("category/list", 332),
                        tr.ColumnSchema.create_continuous("price/list")])
    inputs = tr.TabularSequenceFeatures.from_schema(schema, max_sequence_length=20, d_output=100, masking="causal")
    cfg = tr.XLNetConfig.build(d_model=64, n_head=4, n_layer=2, total_seq_length=20)
    body = tr.SequentialBlock(inputs, tr.MLPBlock([64]), tr.TransformerBlock(cfg, masking=inputs.masking))
    model = tr.NextItemPredictionTask(weight_tying=True).to_model(body, inputs, max_sequence_length=20).cuda().eval()
    with torch.no_grad():
        for n, p in body[2].transformer.named_parameters():
            if p.ndim >= 2 and "layer_norm" not in n:
                p.normal_(0.0, 0.08)
    B, L = 40, 20
    dense = synth_batch(B, L, cards, ("price/list",), seed=5)
    lens = (dense["item_id/list"] != 0).sum(1)
    offs = torch.cat([torch.zeros(1, dtype=torch.long), lens.cumsum(0)])
    valid = dense["item_id/list"] != 0
    ragged = {}
    for k, v in dense.items():
        ragged[k + "__values"] = v[valid].cuda()
        ragged[k + "__offsets"] = offs.cuda()
    with torch.no_grad():
        out_r = model(ragged, training=True)
        out_d = model({k: v[:, : int(lens.max())].cuda() for k, v in dense.items()}, training=True)
    assert abs(out_r["loss"].item() - out_d["loss"].item()) < 1e-6  # ragged ingest == dense padded input
    # oracle for the whole stack
    Lm = int(lens.max())
    d_in = {k: v[:, :Lm] for k, v in dense.items()}
    emb = inputs.categorical_module.embedding_tables
    with torch.no_grad():
        x = O.embed_concat({n: emb[n].weight.cpu() for n in cards}, {n: d_in[n] for n in cards},
                           {"price/list": d_in["price/list"]})
        lin = inputs.projection_module[0][0]
        x = O.project_relu(x, lin.weight.cpu(), lin.bias.cpu())
        mask, labels = O.clm_compute_masked_targets(d_in["item_id/list"], True, False)
        x = O.clm_apply_mask_to_inputs(x, mask, inputs.masking.masked_item_embedding.detach().cpu(), True, False)
        lin2 = body[1][0][0]
        x = O.project_relu(x, lin2.weight.cpu(), lin2.bias.cpu())
        hf = O.build_hf_xlnet(64, 4, 2).eval()
        hf.load_state_dict({k: v.cpu() for k, v in body[2].transformer.state_dict().items()}, strict=False)
        h = O.hf_encoder_forward(hf, x)
        xt, y = O.select_targets(h, labels)
        ref_loss, _ = O.full_softmax_head(xt, y, emb["item_id/list"].weight.cpu(), 1.0)
    assert abs(out_r["loss"].item() - ref_loss.item()) < TOL
    assert torch.equal(out_r["labels"].cpu(), y)


def test_no_projection_path():
    """No d_output: aggregation + masking only (embedding dim = d_model), XLNet MLM."""
    import transformers4rec_b200.torch as tr
    torch.manual_seed(22)
    schema = tr.Schema([tr.ColumnSchema.create_categorical("item_id/list", 3000, tags=[tr.Tags.ITEM_ID])])
    inputs = tr.TabularSequenceFeatures.from_schema(schema, max_sequence_length=20, masking="mlm",
                                                    embedding_dims={"item_id/list": 64})
    assert inputs.projection_module is None and tuple(inputs.output_size()) == (-1, 20, 64)
    cfg = tr.XLNetConfig.build(d_model=64, n_head=4, n_layer=1, total_seq_length=20)
    model = cfg.to_torch_model(inputs, tr.NextItemPredictionTask(weight_tying=True)).cuda().eval()
    B, L = 50, 20
    batch = synth_batch(B, L, {"item_id/list": 3001}, seed=6)
    u, draws = mlm_draws(B, L)
    inputs.masking.set_draws(u.cuda())
    with torch.no_grad():
        out = model({k: v.cuda() for k, v in batch.items()}, training=True)
        table = inputs.item_embedding_table.weight.cpu()
        x = torch.nn.functional.embedding(batch["item_id/list"], table)
        mask, labels = O.mlm_compute_masked_targets(batch["item_id/list"], True, False, **draws)
        x = O.mlm_apply_mask_to_inputs(x, mask, inputs.masking.masked_item_embedding.detach().cpu(), True, False)
        hf = O.build_hf_xlnet(64, 4, 1).eval()
        hf.load_state_dict({k: v.cpu() for k, v in model.heads[0].body[1].transformer.state_dict().items()}, strict=False)
        xt, y = O.select_targets(O.hf_encoder_forward(hf, x), labels)
        ref_loss, _ = O.full_softmax_head(xt, y, table, 1.0)
    assert abs(out["loss"].item() - ref_loss.item()) < TOL


def test_head_label_smoothing(ops):
    """nn.CrossEntropyLoss(label_smoothing=e) (transformers4rec/torch/losses.py:4-20) in the fused head."""
    torch.manual_seed(31)
    T, V, De, eps = 300, 7001, 64, 0.1
    xt = torch.randn(T, De)
    W = torch.randn(V, De) * 0.1
    y = torch.randint(1, V, (T,))
    ref_loss, _ = O.full_softmax_head(xt, y, W, 1.0, label_smoothing=eps)
    res = ops.head_softmax_ce(ops.split_planes(xt.cuda()), xt.cuda(), y.cuda(), ops.split_planes(W.cuda()), W.cuda(),
                              label_smoothing=eps)
    assert abs(res["loss"].item() - ref_loss.item()) < 1e-4


def test_context_features_are_repeated_along_the_sequence():
    """tabular/base.py:53-63: non-sequential features [B] are expanded to [B, L] before the concat."""
    import transformers4rec_b200.torch as tr
    torch.manual_seed(32)
    schema = tr.Schema([tr.ColumnSchema.create_categorical("item_id/list", 500, tags=[tr.Tags.ITEM_ID]),
                        tr.ColumnSchema.create_categorical("user_country", 60, is_list=False),
                        tr.ColumnSchema.create_continuous("user_age", is_list=False)])
    inputs = tr.TabularSequenceFeatures.from_schema(schema, max_sequence_length=12, d_output=64, masking="clm").cuda()
    B, L = 9, 12
    batch = synth_batch(B, L, {"item_id/list": 501}, seed=8)
    batch["user_country"] = torch.randint(1, 61, (B,))
    batch["user_age"] = torch.rand(B)
    with torch.no_grad():
        x = inputs({k: v.cuda() for k, v in batch.items()}, training=True).cpu()
        emb = inputs.categorical_module.embedding_tables
        ref = O.embed_concat({"item_id/list": emb["item_id/list"].weight.cpu(), "user_country": emb["user_country"].weight.cpu()},
                             {"item_id/list": batch["item_id/list"], "user_country": batch["user_country"].unsqueeze(1).expand(B, L)},
                             {"user_age": batch["user_age"].unsqueeze(1).expand(B, L)})
        lin = inputs.projection_module[0][0]
        ref = O.project_relu(ref, lin.weight.cpu(), lin.bias.cpu())
        mask, _ = O.clm_compute_masked_targets(batch["item_id/list"], True, False)
        ref = O.clm_apply_mask_to_inputs(ref, mask, inputs.masking.masked_item_embedding.detach().cpu(), True, False)
    assert (x - ref).abs().max().item() < 1e-4
