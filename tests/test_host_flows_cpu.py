"""Host logic of the package end to end on the CPU, with the kernels replaced by test doubles
(tests/_ops_double.py): module wiring, masking modes, state side channels, lazy outputs, metrics, the arithmetic
switches of the head (nprod = 3 / 2) and bench.py's accuracy leg.  The doubles compute with the oracle's arithmetic,
so the results are compared with the oracle graph itself."""
import math

import pytest
import torch

import _ops_double as D
import t4r_oracle as O
from _util import make_pair, mlm_draws, synth_batch

CARDS = {"item_id/list": 3001, "category/list": 37}
DIMS = {"item_id/list": 64, "category/list": 64}
CONT = ("cont0/list", "cont1/list")


def _pair(arch="xlnet", masking="mlm", dims=DIMS, **kw):
    return make_pair(CARDS, dims, "item_id/list", CONT, 64, 4, 1, 12, arch=arch, masking=masking, device="cpu",
                     weight_scale=0.08, **kw)


@pytest.mark.parametrize("arch,masking", [("xlnet", "mlm"), ("xlnet", "clm"), ("gpt2", "clm")])
def test_training_eval_inference_flows(monkeypatch, arch, masking):
    D.install(monkeypatch)
    oracle, model = _pair(arch, masking)
    B, L = 9, 12
    batch = synth_batch(B, L, CARDS, CONT, seed=1)
    u, draws = mlm_draws(B, L)
    inputs = model.heads[0].body[0]
    inputs.masking.set_draws(u)
    with torch.no_grad():
        ref = oracle(batch, training=True, draws=draws)
        out = model(batch, training=True)
    assert abs(out["loss"].item() - ref["loss"].item()) < 1e-4
    assert torch.equal(inputs.masking.masked_targets, ref["masked_targets"])      # state side channel
    assert torch.equal(out["labels"], ref["labels"])                             # lazy outputs
    assert (out["predictions"] - ref["predictions"]).abs().max().item() < 1e-3
    assert torch.equal(inputs.to_merge["categorical_module"].item_seq, batch["item_id/list"])
    # evaluation: ranks -> metrics through the task
    with torch.no_grad():
        ref_e = oracle(batch, training=False, testing=True)
        out_e = model(batch, training=False, testing=True)
    assert abs(out_e["loss"].item() - ref_e["loss"].item()) < 1e-4
    task = model.heads[0].prediction_task_dict["next-item"]
    got = task.calculate_metrics(out_e)
    ref_rec = O.recall_at_mean([10, 20], ref_e["predictions"], ref_e["labels"])
    name = [k for k in got if "recall" in k][0]
    assert (got[name] - ref_rec).abs().max().item() < 1e-6
    # inference: scores and top-k
    if masking == "mlm":
        short = {k: torch.nn.functional.pad(v[:, :-1], (0, 1)) for k, v in batch.items()}
    else:
        short = batch
    with torch.no_grad():
        scores = model(short, training=False, testing=False)
        model.top_k = 5
        s, i = model(short, training=False, testing=False)
        model.top_k = None
    assert scores.shape == (B, CARDS["item_id/list"])
    rs, ri = torch.sort(-scores, dim=1, stable=True)
    assert torch.equal(i, ri[:, :5]) and torch.allclose(s, -rs[:, :5])


def test_task_block_and_mixed_head_arithmetic(monkeypatch):
    """item dim != d_model -> task_block; task.nprod = 2 routes the TRAINING head through the 2-unit product (emulated
    bit-for-bit from the packed operands) and everything else through the 3-product planes."""
    D.install(monkeypatch)
    oracle, model = _pair(dims={"item_id/list": 32, "category/list": 64})
    B, L = 8, 12
    batch = synth_batch(B, L, CARDS, CONT, seed=2)
    u, draws = mlm_draws(B, L)
    model.heads[0].body[0].masking.set_draws(u)
    task = model.heads[0].prediction_task_dict["next-item"]
    assert task.task_block is not None
    from transformers4rec_b200 import ops
    calls = []
    real = ops.head_softmax_ce
    monkeypatch.setattr(ops, "head_softmax_ce", lambda *a, **k: (calls.append((k.get("nprod"), k.get("want_rank"))), real(*a, **k))[1])
    with torch.no_grad():
        ref = oracle(batch, training=True, draws=draws)["loss"].item()
        assert task.nprod == 2       # the library default since round 2 (device-side error table: profiles/)
        task.nprod = 3
        l3 = model(batch, training=True)["loss"].item()
        lse3 = task._last["row_lse"].clone()
        task.nprod = 2
        out = model(batch, training=True)
        l2 = out["loss"].item()
        lse2 = task._last["row_lse"].clone()
        assert task._last["w_planes"] is None and ("W#mixed" in task._planes._cache) and ("W" in task._planes._cache)
        preds = out["predictions"]                      # lazily, from the 3-product planes
        out_e = model(batch, training=False, testing=True)  # evaluation ignores nprod = 2
    assert abs(l3 - ref) < 1e-4 and abs(l2 - ref) < 1e-3 and abs(l2 - l3) < 2e-4
    assert (lse2 - lse3).abs().max().item() < 1e-4
    assert calls == [(3, False), (2, False), (3, True)]   # train default, train mixed, evaluation (ranks) back on 3
    assert preds.shape[1] == CARDS["item_id/list"] and math.isfinite(out_e["loss"].item())


def test_sampled_softmax_flow(monkeypatch):
    D.install(monkeypatch)
    oracle, model = _pair(sampled=True, max_n_samples=200)
    B, L, S = 8, 12, 200
    batch = synth_batch(B, L, CARDS, CONT, seed=3)
    u, draws = mlm_draws(B, L)
    model.heads[0].body[0].masking.set_draws(u)
    task = model.heads[0].prediction_task_dict["next-item"]
    torch.manual_seed(4)
    raw = torch.multinomial(oracle.dist, 2 * S, replacement=True)
    task.set_negative_draws(raw)
    with torch.no_grad():
        ref = oracle(batch, training=True, draws=draws, neg_samples=O.negatives_from_draws(raw, S))
        task.nprod = 2   # the sampled head keeps the 3-product planes
        out = model(batch, training=True)
    assert abs(out["loss"].item() - ref["loss"].item()) < 1e-4
    assert (out["predictions"] - ref["predictions"]).abs().max().item() < 1e-3


def test_bench_recall_agreement_leg(monkeypatch):
    """bench.py's accuracy leg end to end (product forward = doubles here): ranks of the two sides must agree."""
    import importlib.util
    import os
    D.install(monkeypatch)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod2", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    cfg = dict(V=2001, De=32, d=64, H=4, NL=1, L=12, B=16, arch="gpt2", masking="clm",
               side={"category/list": 37}, label="test")
    model = bench.build_product_model(cfg, torch.device("cpu"))
    batch = bench.synth_batch(cfg["B"], cfg["L"], cfg, seed=0)
    res = bench.recall_agreement(cfg, model, batch, batch, n_sample=8)
    assert res["label_rows"] == cfg["B"] and res["label_rank_max_abs_diff"] <= 1
    assert res["ours_sample"] == res["oracle_sample"]


@pytest.mark.parametrize("cfg", [
    dict(V=2001, De=16, d=32, H=2, NL=1, L=10, B=6, arch="gpt2", masking="clm", label="config3-like",
         side={"category/list": 37, "brand/list": 11, "shop/list": 53, "price_bin/list": 10, "weekday/list": 8, "hour_bin/list": 7}),
    dict(V=4001, De=32, d=32, H=2, NL=1, L=50, B=4, arch="xlnet", masking="mlm", sampled=300, label="config5-like"),
], ids=["config3-like", "config5-like"])
def test_bench_workload_builders_train_like_the_oracle(monkeypatch, cfg):
    """bench.py's model builders for BASELINE configs[2] / configs[4] (tiny sizes): the product model they build and
    the oracle carrying its weights must produce the same training loss."""
    import importlib.util
    import os
    D.install(monkeypatch)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod3", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    model = bench.build_product_model(cfg, torch.device("cpu"))
    oracle = bench.oracle_with_model_weights(cfg, model)
    batch = bench.synth_batch(cfg["B"], cfg["L"], cfg, seed=0)
    task = model.heads[0].prediction_task_dict["next-item"]
    kw = {}
    if cfg["masking"] == "mlm":
        u, draws = mlm_draws(cfg["B"], cfg["L"])
        model.heads[0].body[0].masking.set_draws(u)
        kw["draws"] = draws
    if cfg.get("sampled"):
        torch.manual_seed(4)
        raw = torch.multinomial(oracle.dist, 2 * cfg["sampled"], replacement=True)
        task.set_negative_draws(raw)
        kw["neg_samples"] = O.negatives_from_draws(raw, cfg["sampled"])
    with torch.no_grad():
        ref = oracle(batch, training=True, **kw)["loss"].item()
        got = model(batch, training=True)["loss"].item()
    assert abs(got - ref) < 1e-4, (got, ref)
    assert (task.task_block is not None) == (cfg["De"] != cfg["d"])


@pytest.mark.parametrize("sampled", [0, 300], ids=["full-softmax", "sampled-softmax"])
def test_bench_dump_outputs_are_what_the_caller_received(monkeypatch, tmp_path, sampled):
    """bench.py --dump-outputs: loss, labels and a seeded sample of prediction rows as .npy files (floats float32,
    integers float64), equal to what the forward returned; the same seed picks the same rows."""
    import importlib.util
    import os
    import numpy as np
    D.install(monkeypatch)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod6", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    cfg = dict(V=2001, De=32, d=32, H=2, NL=1, L=12, B=8, arch="xlnet", masking="mlm", sampled=sampled, label="test")
    model = bench.build_product_model(cfg, torch.device("cpu"))
    task = model.heads[0].prediction_task_dict["next-item"]
    with torch.no_grad():
        out = model(bench.synth_batch(cfg["B"], cfg["L"], cfg, seed=0), training=True)
        preds, labels = out["predictions"], out["labels"]
        T = labels.numel()
        monkeypatch.setattr(bench, "DUMP_PREDICTION_BYTES", 4 * 5 * preds.shape[1])   # room for 5 of the T rows
        for d in ("a", "b"):
            bench.dump_outputs(str(tmp_path / d), out["loss"], task)
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("loss", "labels", "predictions", "prediction_rows")}
    assert sorted(os.listdir(tmp_path / "a")) == sorted(f"{n}.npy" for n in got)
    assert [got[n].dtype for n in got] == [np.float32, np.float64, np.float32, np.float64]
    assert float(got["loss"]) == out["loss"].item() and np.array_equal(got["labels"], labels.numpy())
    rows = torch.from_numpy(got["prediction_rows"]).long()
    assert T > 5 and rows.numel() == 5 and bool((rows.diff() > 0).all()) and int(rows.max()) < T
    assert np.allclose(got["predictions"], preds[rows].numpy(), atol=1e-5)
    for n in got:
        assert np.array_equal(np.load(tmp_path / "b" / f"{n}.npy"), got[n])
    assert int(task._last["count"].item()) == T          # the task's state is left as the forward left it


def test_permutation_language_modeling_flow(monkeypatch):
    """masking="plm" end to end (kernels = doubles): labels / masks / side channels, training and evaluation loss
    against the oracle graph, whose encoder is HF XLNet's two-stream forward with perm_mask + target_mapping."""
    import transformers4rec_b200.torch as tr
    D.install(monkeypatch)
    oracle, model = make_pair({"item_id/list": 1001}, {"item_id/list": 32}, "item_id/list", (), 32, 2, 2, 12,
                              masking="plm", device="cpu", weight_scale=0.08)
    with torch.no_grad():   # the query stream starts from mask_emb: make it matter and share it with the oracle
        model.heads[0].body[1].transformer.mask_emb.normal_(0.0, 0.5)
        oracle.transformer.mask_emb.copy_(model.heads[0].body[1].transformer.mask_emb)
    B, L = 10, 12
    batch = synth_batch(B, L, {"item_id/list": 1001}, seed=5)
    g = torch.Generator().manual_seed(3)
    draws = {"u_span": torch.rand((B, L), generator=g), "u_start": torch.rand((B, L), generator=g),
             "u_force": torch.rand((B,), generator=g), "u_unmask": torch.rand((B,), generator=g),
             "perm": torch.stack([torch.randperm(L, generator=g) for _ in range(B)])}
    inputs = model.heads[0].body[0]
    assert isinstance(inputs.masking, tr.PermutationLanguageModeling)
    inputs.masking.set_draws(draws)
    with torch.no_grad():
        ref = oracle(batch, training=True, draws=draws)
        out = model(batch, training=True)
    assert torch.equal(inputs.masking.masked_targets, ref["masked_targets"])
    assert torch.equal(inputs.masking.perm_mask, oracle._plm[0].to(torch.uint8))
    assert inputs.masking.target_mapping.shape == (B, L, L)
    assert set(inputs.masking.transformer_required_arguments()) == {"target_mapping", "perm_mask"}
    assert abs(out["loss"].item() - ref["loss"].item()) < 1e-4
    with torch.no_grad():
        ref_e = oracle(batch, training=False, testing=True)
        out_e = model(batch, training=False, testing=True)
    assert abs(out_e["loss"].item() - ref_e["loss"].item()) < 1e-4
    with pytest.raises(NotImplementedError):
        tr.PermutationLanguageModeling(hidden_size=8, permute_all=True)
    # GPT-2 cannot take PLM (block/transformer.py:119-134 message)
    with pytest.raises(ValueError, match="requires the parameters"):
        tr.TransformerBlock(tr.GPT2Config.build(d_model=32, n_head=2, n_layer=1, total_seq_length=12),
                            masking=tr.PermutationLanguageModeling(hidden_size=32))


@pytest.mark.parametrize("task", ["mlm", "masked", "clm", "causal", "plm", "permutation"])
def test_body_built_with_the_shift_operator(monkeypatch, task):
    """tests/unit/torch/block/test_transformer.py:39-89 (incl. test_xlnet_with_plm): ``features >> MLPBlock([64]) >>
    TransformerBlock(config, masking=features.masking)`` on the reference's testing schema; output [B, L, 64]."""
    import transformers4rec_b200.torch as tr
    from test_abi_and_host import _testing_schema
    D.install(monkeypatch)
    schema = _testing_schema(tr)
    tab = tr.TabularSequenceFeatures.from_schema(schema, max_sequence_length=20, aggregation="concat", d_output=64,
                                                 masking=task)
    cfg = tr.XLNetConfig.build(d_model=64, n_head=4, n_layer=2, total_seq_length=20)
    block = tab >> tr.MLPBlock([64]) >> tr.TransformerBlock(transformer=cfg, masking=tab.masking)
    assert isinstance(block, tr.SequentialBlock) and len(block) == 3
    g = torch.Generator().manual_seed(0)
    batch = {}
    for col in schema:
        shape = (12, 20) if col.is_list else (12,)
        batch[col.name] = (torch.randint(1, col.int_max + 1, shape, generator=g) if col.int_max
                           else torch.rand(shape, generator=g))
    with torch.no_grad():
        out = block(batch, training=True)
    assert out.ndim == 3 and out.shape == (12, 20, 64)
    # test_transformer.py:92-120: PLM with an architecture that cannot take it
    if task in ("plm", "permutation"):
        with pytest.raises(ValueError, match="PermutationLanguageModeling requires the parameters: target_mapping, perm_mask"):
            tr.TransformerBlock(tr.GPT2Config.build(d_model=64, n_head=4, n_layer=2, total_seq_length=20), masking=tab.masking)
