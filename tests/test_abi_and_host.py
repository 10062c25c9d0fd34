"""CPU tests: the C-ABI library loads and exports every symbol include/t4r_b200.h
declares; host-side API surface (schema shim, from_schema, registries, state-dict
names, error messages) mirrors the reference.  No compute calls (no GPU here)."""
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import ctypes

    from transformers4rec_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    hdr = open(os.path.join(ROOT, "include", "t4r_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(t4r_[a-z0-9_]+)\s*\(", hdr)) - {"t4r_round_up64"}
    assert len(names) >= 20
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in sorted(names):
        assert hasattr(lib, n), f"{n} declared in include/t4r_b200.h but not exported"
    assert names == set(_lib.SIGNATURES), names ^ set(_lib.SIGNATURES)
    assert _lib.load().t4r_version() >= 100


def test_struct_layouts_match_header():
    from transformers4rec_b200 import _lib
    import ctypes as C
    assert C.sizeof(_lib.XLNetLayer) == 13 * 8 and C.sizeof(_lib.GPT2Layer) == 12 * 8
    # t4r_feature_list: 2 ints + 32 ptr + 32 ptr + 32 i64 + 32 int + 32 int + 32 ptr + 32 int
    assert C.sizeof(_lib.FeatureList) == 8 + 32 * 8 * 3 + 32 * 4 * 2 + 32 * 8 + 32 * 4


def test_no_cpu_fallback():
    from transformers4rec_b200 import T4RError, ops
    with pytest.raises(T4RError):
        ops.split_planes(torch.randn(4, 8))
    with pytest.raises(T4RError):
        ops.mask_clm(torch.zeros(2, 3, dtype=torch.long), 0)


def _schema(tr):
    return tr.Schema([tr.ColumnSchema.create_categorical("item_id/list", 51996, tags=[tr.Tags.ITEM_ID]),
                      tr.ColumnSchema.create_categorical("category/list", 332),
                      tr.ColumnSchema.create_continuous("price/list")])


def test_from_schema_surface_and_state_dict_names():
    import transformers4rec_b200.torch as tr
    s = _schema(tr)
    inp = tr.TabularSequenceFeatures.from_schema(s, max_sequence_length=20, d_output=100, masking="causal")
    assert isinstance(inp.masking, tr.CausalLanguageModeling)
    assert inp.item_id == "item_id/list"
    assert inp.item_embedding_table.num_embeddings == 51997  # int_domain.max + 1
    assert inp.aggregation == "concat"
    assert tuple(inp.output_size()) == (-1, 20, 100)
    assert inp._layout()[1] == 64 + 64 + 1
    names = [n for n, *_ in inp._layout()[0]]
    assert names == sorted(names)  # concat order = sorted feature names
    cfg = tr.XLNetConfig.build(d_model=64, n_head=4, n_layer=2, total_seq_length=20)
    assert cfg.layer_norm_eps == 0.03 and cfg.d_inner == 256 and cfg.attn_type == "bi" and cfg.vocab_size == 1
    body = tr.SequentialBlock(inp, tr.MLPBlock([64]).build(inp.output_size()), tr.TransformerBlock(cfg, masking=inp.masking))
    model = tr.NextItemPredictionTask(weight_tying=True).to_model(body, inp)
    keys = set(model.state_dict().keys())
    for k in ("heads.0.body.0.to_merge.categorical_module.embedding_tables.item_id/list.weight",
              "heads.0.body.0.projection_module.0.0.weight", "heads.0.body.0._masking.masked_item_embedding",
              "heads.0.body.2.transformer.layer.0.rel_attn.q", "heads.0.body.2.transformer.layer.1.ff.layer_2.bias"):
        assert k in keys, k
    task = model.heads[0].prediction_task_dict["next-item"]
    assert task.target_dim == 51997 and task.item_embedding_table is inp.item_embedding_table
    # HF checkpoints load unchanged
    import t4r_oracle as O
    hf = O.build_hf_xlnet(64, 4, 2)
    missing, unexpected = body[2].transformer.load_state_dict(hf.state_dict(), strict=True), None


def test_reference_error_messages():
    import transformers4rec_b200.torch as tr
    s = _schema(tr)
    with pytest.raises(ValueError, match="You cannot specify both d_output and projection"):
        tr.TabularSequenceFeatures.from_schema(s, d_output=8, projection=tr.MLPBlock([8]))
    no_item = tr.Schema([tr.ColumnSchema.create_categorical("category/list", 332)])
    with pytest.raises(ValueError, match="For masking a categorical_module is required including an item_id"):
        tr.TabularSequenceFeatures.from_schema(no_item, d_output=8, masking="mlm")
    inp = tr.TabularSequenceFeatures.from_schema(s, max_sequence_length=20, d_output=64, masking="mlm")
    gcfg = tr.GPT2Config.build(d_model=64, n_head=4, n_layer=1, total_seq_length=20)
    with pytest.raises(ValueError, match="MaskedLanguageModeling is not supported by: the GPT2Config architecture"):
        tr.TransformerBlock(gcfg, masking=inp.masking)
    inp2 = tr.TabularSequenceFeatures.from_schema(s, max_sequence_length=20, d_output=64)
    body = tr.SequentialBlock(inp2, tr.TransformerBlock(tr.XLNetConfig.build(64, 4, 1, 20)))
    with pytest.raises(ValueError, match="The input block should contain a masking schema"):
        tr.NextItemPredictionTask(weight_tying=True).to_model(body, inp2)
    assert gcfg.layer_norm_epsilon == 1e-5 and gcfg.n_positions == 20


def test_task_block_inserted_when_dims_differ():
    import transformers4rec_b200.torch as tr
    s = _schema(tr)
    inp = tr.TabularSequenceFeatures.from_schema(s, max_sequence_length=20, d_output=256, masking="clm")
    model = tr.GPT2Config.build(256, 8, 1, 20).to_torch_model(inp, tr.NextItemPredictionTask(weight_tying=True))
    task = model.heads[0].prediction_task_dict["next-item"]
    lin = task.task_block[0][0]
    assert (lin.in_features, lin.out_features) == (256, 64) and len(task.task_block[0]) == 1  # no activation


def test_schema_json_roundtrip(tmp_path):
    import json

    import transformers4rec_b200.torch as tr
    doc = {"feature": [
        {"name": "item_id/list", "type": "INT", "intDomain": {"name": "item_id/list", "min": "1", "max": "51996", "isCategorical": True},
         "valueCount": {"min": "2", "max": "185"}, "annotation": {"tag": ["item_id", "list", "categorical", "item"]}},
        {"name": "timestamp/hour/list", "type": "FLOAT", "valueCount": {"min": "2", "max": "185"},
         "annotation": {"tag": ["continuous", "time", "list"]}}]}
    p = tmp_path / "schema.json"
    p.write_text(json.dumps(doc))
    s = tr.Schema.from_json(str(p))
    assert s.select_by_tag(tr.Tags.ITEM_ID).column_names == ["item_id/list"]
    assert s.categorical_cardinalities() == {"item_id/list": 51997}
    assert s.select_by_tag("continuous").column_names == ["timestamp/hour/list"]


def test_log_uniform_sampler_host_side():
    import t4r_oracle as O
    import transformers4rec_b200.torch as tr
    smp = tr.LogUniformSampler(max_n_samples=50, max_id=1000, min_id=1)
    assert torch.equal(smp.dist, O.log_uniform_distr(1000, 1))
    assert torch.equal(smp.unique_sampling_dist, O.unique_sampling_distr(smp.dist, 100))
    assert smp.dist[0] == 0 and abs(smp.dist.sum().item() - 1.0) < 1e-5
    with pytest.raises(ValueError):
        tr.LogUniformSampler(max_n_samples=0, max_id=10)


def test_widened_input_block_surface():
    """SURVEY §8f N4 options of TabularSequenceFeatures.from_schema: layout, widths, reference errors."""
    import ctypes as C
    import transformers4rec_b200.torch as tr
    from transformers4rec_b200 import _lib
    assert C.sizeof(_lib.Feature) == 6 * 4 + 6 * 8
    schema = _schema(tr)
    soft = tr.TabularSequenceFeatures.from_schema(schema, max_sequence_length=20, continuous_soft_embeddings=True,
                                                  aggregation="concat", post="layer-norm")
    assert isinstance(soft.continuous_module, tr.SoftEmbeddingFeatures)
    assert soft.output_size()[-1] == 64 + 64 + 8  # two categorical tables + one soft embedding (dim 8 default)
    assert set(soft.categorical_module.post.feature_layer_norm.keys()) == {"item_id/list", "category/list"}
    assert "to_merge.continuous_module.embedding_tables.price/list.projection_layer.weight" in soft.state_dict()
    proj = tr.TabularSequenceFeatures.from_schema(schema, max_sequence_length=20, continuous_projection=32,
                                                  aggregation="concat")
    assert [n for n, *_ in proj._layout()[0]] == ["category/list", "continuous_projection", "item_id/list"]
    assert proj.output_size()[-1] == 64 + 32 + 64
    with pytest.raises(ValueError, match="required for element-wise aggregation"):
        tr.TabularSequenceFeatures.from_schema(schema, max_sequence_length=20, aggregation="element-wise-sum").output_size()
    ok = tr.TabularSequenceFeatures.from_schema(schema, max_sequence_length=20, aggregation="element-wise-sum-item-multi",
                                                continuous_soft_embeddings=True, soft_embedding_dim_default=64)
    assert ok.output_size()[-1] == 64
    with pytest.raises(NotImplementedError):
        tr.TabularSequenceFeatures.from_schema(schema, aggregation="stack")
    assert set(tr.ranking_metrics_registry) >= {"precision_at", "recall_at", "avg_precision_at", "map", "dcg_at",
                                                "ndcg_at", "mrr_at"}


def _testing_schema(tr):
    """The shape of the reference's testing schema (transformers4rec/data/testing/schema.json): two list
    categoricals (item max 51996, category max 332), one context categorical (max 62), ten list
    continuous features and one context continuous feature."""
    cont = ["timestamp/age_days/LogOp/Normalize/list", "timestamp/hour/list", "timestamp/weekday/list",
            "timestamp/day/list", "timestamp/month/list", "timestamp/year/list", "timestamp/hour/sin/list",
            "timestamp/hour/cos/list", "timestamp/weekday/sin/list", "timestamp/weekday/cos/list"]
    return tr.Schema([tr.ColumnSchema.create_continuous(n) for n in cont] + [
        tr.ColumnSchema.create_categorical("item_id/list", 51996, tags=[tr.Tags.ITEM_ID]),
        tr.ColumnSchema.create_categorical("category/list", 332),
        tr.ColumnSchema.create_categorical("user_country", 62, is_list=False),
        tr.ColumnSchema.create_continuous("user_age", is_list=False)])


def test_known_answers_of_the_reference_feature_tests():
    import transformers4rec_b200.torch as tr
    schema = _testing_schema(tr)
    # tests/unit/torch/features/test_sequential.py:217-223: concat width 203 = 3 x 64 + 11 scalars
    tab = tr.TabularSequenceFeatures.from_schema(schema, aggregation="concat")
    assert tab.output_size()[-1] == 203
    # tests/unit/torch/features/test_embedding.py:106-119: infer_embedding_sizes with multiplier 3 -> 46 and 13
    emb = tr.SequenceEmbeddingFeatures.from_schema(schema.select_by_tag(tr.Tags.CATEGORICAL), infer_embedding_sizes=True,
                                                   infer_embedding_sizes_multiplier=3.0)
    assert emb.embedding_tables["item_id/list"].weight.shape[1] == 46
    assert emb.embedding_tables["category/list"].weight.shape[1] == 13
    # tests/unit/torch/features/test_embedding.py:73-87: defaults and the item table size (max + 1)
    emb = tr.SequenceEmbeddingFeatures.from_schema(schema.select_by_tag(tr.Tags.CATEGORICAL))
    assert all(t.weight.shape[1] == 64 for t in emb.embedding_tables.values())
    assert emb.item_id == "item_id/list" and emb.item_embedding_table.num_embeddings == 51997


# --------------------------------------------------------------------------- #
# 2-unit product operands (nprod = 2): layout + rounding of the packing code, on the host twin of the kernel
# --------------------------------------------------------------------------- #
def _mixed_cases():
    g = torch.Generator().manual_seed(11)
    x = torch.randn(37, 200, generator=g)
    x[3] = 0.0                                   # all-zero row -> scale 1
    x[4] *= 1e-38                                # tiny row: scale clamps at 2^126
    x[5] *= 1e20                                 # huge row: negative shift
    x[6, :] = torch.exp2(torch.randint(-20, 4, (200,), generator=g).float())  # wide in-row dynamic range
    x[7, 10] = 16383.999                         # rounds up to 2^14 in fp16
    return x


def test_mixed_planes_host_twin_matches_reference_bit_exactly():
    import _mixed_ref as R
    from transformers4rec_b200 import ops
    x = _mixed_cases()
    planes, inv = ops.split_planes_mixed_host(x)
    assert planes.shape == (2, 37, 256)
    ref = R.pack(x)
    h16, hi8, lo8 = R.unpack_planes(planes)
    assert torch.equal(inv, ref["inv_scale"])
    assert torch.equal(h16.view(torch.int16), ref["h16"].view(torch.int16))
    assert torch.equal(hi8.view(torch.uint8), ref["hi8"].view(torch.uint8))
    assert torch.equal(lo8.view(torch.uint8), ref["lo8"].view(torch.uint8))
    # zero padding of K up to Kp and the scale of special rows
    assert not h16[:, 200:].any() and not hi8.view(torch.uint8)[:, 200:].any() and not lo8.view(torch.uint8)[:, 200:].any()
    assert inv[3].item() == 1.0 and inv[4].item() == 2.0 ** -126
    m = (x.abs().amax(1) / inv)[[0, 1, 2, 5, 6, 7]]
    assert ((m >= 2 ** 13) & (m < 2 ** 14)).all()
    assert h16.float().abs().max().item() <= 2.0 ** 14 and hi8.float().abs().max().item() <= 256.0
    assert lo8.float().abs().max().item() <= 256.0


def test_mixed_product_is_fp32_grade():
    """hi*hi (fp16) + lo8*hi8 + hi8*lo8 (e4m3), scaled back, against fp64: the error budget of nprod = 2."""
    import _mixed_ref as R
    g = torch.Generator().manual_seed(12)
    T, V, K = 96, 4000, 256
    x = torch.randn(T, K, generator=g)
    x = (x - x.mean(1, keepdim=True)) / x.std(1, keepdim=True)       # LayerNorm-ed hidden rows
    w = torch.randn(V, K, generator=g) * 0.05                          # features/embedding.py:461-462
    ref = x.double() @ w.double().t()
    got = R.product(R.pack(x), R.pack(w))
    err = (got - ref).abs().max().item()
    bf = lambda a: a.to(torch.bfloat16).float()
    xh, wh = bf(x), bf(w)
    x3 = xh.double() @ wh.double().t() + xh.double() @ bf(w - wh).double().t() + bf(x - xh).double() @ wh.double().t()
    err3 = (x3 - ref).abs().max().item()
    assert err < 1e-4, err                    # two orders inside the 1e-3 parity bar at |logit| ~ 1
    assert err < 4 * err3, (err, err3)        # within a small factor of the shipped 3-product bf16 split


def test_head_resident_kernel_barrier_protocol_model():
    """Discrete-event model of head_resident_kernel's producer / MMA / epilogue loops (tools/sim_head_resident.py):
    no deadlock, and every MMA reads the A slot / B stage contents of its own (unit, tile, K block)."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location(
        "sim_head_resident", os.path.join(os.path.dirname(os.path.dirname(__file__)), "tools", "sim_head_resident.py"))
    sim = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(sim)
    for tiles_m, tiles_n, nkb, npairs, chunk in [(3, 17, 4, 2, 4), (20, 40, 4, 7, 16), (1, 5, 1, 1, 16), (3, 100, 2, 2, 16)]:
        for pair in range(npairs):
            assert sim.simulate(tiles_m, tiles_n, nkb, npairs, pair, chunk=chunk, seed=pair) > 0


def test_ctypes_structs_mirror_the_compiled_layouts():
    """Every argument struct of the ABI: ctypes mirror vs sizeof() inside the compiled library, and the offset of
    the last (most recently added) field of t4r_head_args."""
    import ctypes as C
    from transformers4rec_b200 import _lib
    lib = _lib.load()
    mirrors = [_lib.HeadArgs, _lib.LinearArgs, _lib.FeatureList, _lib.Feature, _lib.XLNetLayer, _lib.GPT2Layer]
    for which, cls in enumerate(mirrors):
        assert lib.t4r_sizeof_struct(which) == C.sizeof(cls), (cls.__name__, lib.t4r_sizeof_struct(which), C.sizeof(cls))
    assert lib.t4r_sizeof_struct(99) == 0
    assert lib.t4r_head_args_last_offset() == _lib.HeadArgs.col_ids_sorted_unique.offset


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the reference's CPU torch path; needs no GPU): one JSON line with the keys the
    driver reads, on the smallest workload so that the CPU suite stays fast."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "config1",
                          "--steps", "2", "--cpu-sessions", "32"], capture_output=True, text=True, timeout=600, cwd=root)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "sessions/sec (fwd+loss)" and d["unit"] == "sessions/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sessions/step" in d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "sessions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("BASELINE.json config1")


def test_bench_recall_leg_helpers_on_cpu():
    """bench.py's Recall@20 leg: the oracle must really carry the product model's weights (built here on the CPU --
    only the forward needs a GPU), for the item-only XLNet shape and for a side-feature GPT-2 shape with task_block."""
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    for cfg in (dict(bench.CONFIGS["config1"]),
                dict(V=3001, De=32, d=64, H=4, NL=1, L=12, B=8, arch="gpt2", masking="clm",
                     side={"category/list": 37, "brand/list": 11}, label="test")):
        model = bench.build_product_model(cfg, torch.device("cpu"))
        with torch.no_grad():
            for prm in model.parameters():
                prm.add_(torch.randn_like(prm) * 0.01)   # make sure "same seed" cannot explain equal weights
        oracle = bench.oracle_with_model_weights(cfg, model)
        inputs = model.heads[0].body[0]
        for name in oracle.table_names:
            assert torch.equal(oracle.tables[name.replace("/", "__")].weight,
                               inputs.categorical_module.embedding_tables[name].weight)
        assert torch.equal(oracle.proj.weight, inputs.projection_module[0][0].weight)
        sd_o, sd_m = oracle.transformer.state_dict(), model.heads[0].body[1].transformer.state_dict()
        shared = [k for k in sd_o if k in sd_m]
        assert len(shared) >= 10 and all(torch.equal(sd_o[k], sd_m[k]) for k in shared)
        if oracle.task_block is not None:
            tl = model.heads[0].prediction_task_dict["next-item"].task_block[0][0]
            assert torch.equal(oracle.task_block.weight, tl.weight)
        batch = bench.synth_batch(6, cfg["L"], cfg, seed=0)
        ranks = bench.oracle_label_ranks(oracle, batch)
        assert ranks.shape == (6,) and int(ranks.min()) >= 0 and int(ranks.max()) < cfg["V"]


def test_bench_trained_recall_leg_on_cpu(monkeypatch):
    """bench.py's non-vacuous Recall@20 leg (train the config-1-size model with the fused step, evaluate it with the
    product's head and with the oracle carrying the trained weights), end to end on the CPU with kernel doubles: the
    two sides must agree on every label rank, and training must move the loss."""
    import importlib.util
    import os
    import _ops_double as D
    from transformers4rec_b200 import ops
    twin = ops.host_twin("adamw_step")
    D.install(monkeypatch)
    monkeypatch.setattr(ops, "adamw_step", twin)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod5", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    b = bench.skewed_stream(16, 20, 10001, 3)["item_id/list"]
    lens = (b != 0).sum(1)
    assert int(lens.min()) >= 2 and all(torch.equal(r[:n], r[0] + torch.arange(n)) for r, n in zip(b, lens.tolist()))
    rec = bench.trained_recall(torch.device("cpu"), steps=4, batch=16, n_eval=12)
    assert rec["eval_sessions"] == 12 and 0.0 <= rec["ours"] <= 1.0
    assert rec["label_rank_max_abs_diff"] <= 2 and rec["abs_diff"] <= 1.0 / 12 + 1e-9
    assert abs(rec["eval_loss_ours"] - rec["eval_loss_oracle"]) < 1e-3


def test_attention_kernels_index_algebra_emulated():
    """tools/emu_attn_mma.py: lane-level emulation (ldmatrix / mma.sync fragment layouts) of the index algebra of the
    tensor-path attention kernels, transcribed from the CUDA source.  The one-warp kernel (proven on hardware)
    validates the emulator; the two-warp kernel for 32 < L <= 64 is held to the same plain-formula reference."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location(
        "emu_attn_mma", os.path.join(os.path.dirname(os.path.dirname(__file__)), "tools", "emu_attn_mma.py"))
    emu = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(emu)
    assert emu.check(20, 16, True, two_warp=False) < 1e-9
    assert emu.check(9, 16, False, two_warp=False) < 1e-9
    for L, DH, rel in [(50, 16, True), (33, 16, True), (62, 16, True), (64, 16, False)]:
        assert emu.check(L, DH, rel, two_warp=True) < 1e-9, (L, DH, rel)


def test_bench_cpu_arm_handles_the_sampled_softmax_workload():
    """time_oracle_cpu on a config5-like (sampled softmax) shape: negatives are drawn inside the timed step."""
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod4", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    cfg = dict(V=4001, De=32, d=32, H=2, NL=1, L=50, B=4, arch="xlnet", masking="mlm", sampled=300, label="t")
    v, med, threads, b_run = bench.time_oracle_cpu(cfg, 4, 1, 0, budget_s=0.01)
    assert v > 0 and b_run % 4 == 0 and threads >= 1


# --------------------------------------------------------------------------- #
# Permutation Language Modeling masks: the kernel's per-session code (host twin) vs the upstream code's outputs
# (tests/golden/reference_vectors_plm.pt) and vs the oracle on a larger seeded batch, bit-exact
# --------------------------------------------------------------------------- #
def _plm_modes(_lib):
    return (("train", _lib.PLM_TRAIN, True, {}), ("eval", _lib.PLM_EVAL_LAST, False, {}))


@pytest.mark.parametrize("case", ["default", "p0.5_span3", "evalall"])
def test_plm_mask_host_twin_matches_upstream_vectors(case):
    import os
    from transformers4rec_b200 import _lib, ops
    gold = torch.load(os.path.join(os.path.dirname(__file__), "golden", "reference_vectors_plm.pt"), weights_only=False)
    ids, c = gold["item_ids"], gold["cases"][case]
    kw = dict(c["kwargs"])
    eval_all = kw.pop("eval_on_last_item_seq_only", True) is False
    span, prob = kw.get("max_span_length", 5), kw.get("plm_probability", 1 / 6)
    m, l, pm = ops.mask_plm_host(ids, _lib.PLM_TRAIN, 0, span, prob, c["draws"])
    ref = c["train"]
    assert torch.equal(m, ref["mask_schema"]) and torch.equal(l, ref["masked_targets"]) and torch.equal(pm, ref["perm_mask"])
    m, l, pm = ops.mask_plm_host(ids, _lib.PLM_EVAL_ALL if eval_all else _lib.PLM_EVAL_LAST)
    ref = c["eval"]
    assert torch.equal(m, ref["mask_schema"]) and torch.equal(l, ref["masked_targets"]) and torch.equal(pm, ref["perm_mask"])
    assert bool((ref["target_mapping"] == torch.eye(ids.shape[1], dtype=torch.uint8)).all())  # why it is not materialised


def test_plm_mask_host_twin_matches_oracle_large():
    import t4r_oracle as O
    from transformers4rec_b200 import _lib, ops
    g = torch.Generator().manual_seed(77)
    B, L = 700, 20
    lens = torch.randint(0, L + 1, (B,), generator=g)      # incl. empty sessions
    ids = torch.randint(1, 1000, (B, L), generator=g)
    ids = torch.where(torch.arange(L)[None] < lens[:, None], ids, torch.zeros_like(ids))
    draws = {"u_span": torch.rand((B, L), generator=g), "u_start": torch.rand((B, L), generator=g),
             "u_force": torch.rand((B,), generator=g), "u_unmask": torch.rand((B,), generator=g),
             "perm": torch.stack([torch.randperm(L, generator=g) for _ in range(B)])}
    for span, prob in ((5, 1 / 6), (2, 0.3), (7, 0.9)):
        m, l, pm = ops.mask_plm_host(ids, _lib.PLM_TRAIN, 0, span, prob, draws)
        rm, rl, _, rpm, _ = O.plm_compute_masked_targets(ids, True, draws=draws, max_span_length=span, plm_probability=prob)
        assert torch.equal(m, rm) and torch.equal(l, rl) and torch.equal(pm, rpm.to(torch.uint8)), (span, prob)
    nonempty = lens > 0   # (an empty session makes the reference index column -1; not meaningful input)
    for mode, last in ((_lib.PLM_EVAL_LAST, True), (_lib.PLM_EVAL_ALL, False)):
        m, l, pm = ops.mask_plm_host(ids, mode)
        rm, rl, _, rpm, _ = O.plm_compute_masked_targets(ids, False, eval_on_last_item_seq_only=last)
        assert torch.equal(m, rm) and torch.equal(l, rl) and torch.equal(pm, rpm.to(torch.uint8))
        assert nonempty.any()


# --------------------------------------------------------------------------- #
# N3: the training kernels' per-item code on its host twins vs torch (the doubles of tests/_ops_double.py are the
# specification the composition test uses; here the real code is held to them)
# --------------------------------------------------------------------------- #
def test_training_kernels_host_twins_match_torch():
    import _ops_double as DD
    from transformers4rec_b200 import _lib, ops
    g = torch.Generator().manual_seed(31)
    H = ops.host_twin
    x = torch.randn(37, 24, generator=g)
    dy = torch.randn(37, 24, generator=g)
    close = lambda a, b, tol=2e-6: (a - b).abs().max().item() <= tol * max(1.0, b.abs().max().item())
    assert torch.equal(H("transpose")(x), DD.transpose(x))
    for kind in (_lib.ACT_GELU, _lib.ACT_RELU):
        assert close(H("act_fwd")(kind, x), DD.act_fwd(kind, x))
        assert close(H("act_bwd")(kind, x, dy), DD.act_bwd(kind, x, dy))
    big = torch.randn(700, 24, generator=g)
    assert close(H("col_sum")(big), DD.col_sum(big), 1e-5)
    gamma, beta = torch.rand(24, generator=g) + 0.5, torch.randn(24, generator=g)
    assert close(H("layer_norm_fwd")(x, gamma, beta, 0.03), DD.layer_norm_fwd(x, gamma, beta, 0.03), 1e-5)
    add = torch.randn(37, 24, generator=g)
    for a in (None, add):
        got, ref = H("layer_norm_bwd")(x, gamma, 0.03, dy, add=a), DD.layer_norm_bwd(x, gamma, 0.03, dy, add=a)
        assert all(close(u, v, 1e-5) for u, v in zip(got, ref))
    B, L = 3, 4
    xs = torch.randn(B * L, 24, generator=g)
    wpe = torch.randn(9, 24, generator=g)
    assert close(H("add_positions")(xs, wpe, B, L), DD.add_positions(xs, wpe, B, L))
    assert close(H("sum_over_sessions")(xs, B, L), DD.sum_over_sessions(xs, B, L), 1e-5)
    code = torch.randint(0, 3, (37,), generator=g).to(torch.uint8)
    mv = torch.randn(24, generator=g)
    assert torch.equal(H("apply_row_codes")(x, code, mv), DD.apply_row_codes(x, code, mv))
    dm, dyy = H("row_codes_bwd")(dy, code)
    rm, ry = DD.row_codes_bwd(dy, code)
    assert close(dm, rm, 1e-5) and torch.equal(dyy, ry)
    idx = torch.randperm(37, generator=g)[:11].int()
    assert torch.equal(H("gather_rows")(x, idx), DD.gather_rows(x, idx))
    src = torch.randn(11, 24, generator=g)
    assert torch.equal(H("scatter_rows")(src, idx, 37), DD.scatter_rows(src, idx, 37))
    T, Vc, v0 = 9, 50, 100
    z = torch.randn(T, Vc, generator=g)
    lse = torch.logsumexp(z, 1) + 0.3
    labels = torch.randint(90, 160, (T,), generator=g)
    assert close(H("softmax_ce_bwd")(z.clone(), lse, labels, v0, 0.25), DD.softmax_ce_bwd(z.clone(), lse, labels, v0, 0.25))
    ids = torch.randint(0, 20, (37,), generator=g)
    dst1, dst2 = torch.zeros(20, 8), torch.zeros(20, 8)
    H("index_add_rows")(dst1, ids, x, 5, 8, skip_index=0)
    DD.index_add_rows(dst2, ids, x, 5, 8, skip_index=0)
    assert close(dst1, dst2, 1e-5) and not dst1[0].any()


@pytest.mark.parametrize("L,H,dh", [(5, 2, 8), (12, 3, 4), (20, 1, 16)])
def test_attention_backward_host_twin_matches_autograd(L, H, dh):
    import _ops_double as DD
    from transformers4rec_b200 import ops
    g = torch.Generator().manual_seed(32)
    B, d = 3, H * dh
    qkv = torch.randn(B * L, 3 * d, generator=g)
    R = torch.randn(2 * L, d, generator=g)
    rw, rr = torch.randn(d, generator=g), torch.randn(d, generator=g)
    dout = torch.randn(B * L, d, generator=g)
    got = ops.host_twin("xlnet_attn_bwd")(qkv, R, rw, rr, dout, B, L, H)
    ref = DD.xlnet_attn_bwd(qkv, R, rw, rr, dout, B, L, H)
    for name, a, b in zip(("dqkv", "dR", "drw", "drr"), got, ref):
        assert (a - b).abs().max().item() < 2e-4 * max(1.0, b.abs().max().item()), name
    got = ops.host_twin("causal_attn_bwd")(qkv, dout, B, L, H)
    ref = DD.causal_attn_bwd(qkv, dout, B, L, H)
    assert (got - ref).abs().max().item() < 2e-4 * max(1.0, ref.abs().max().item())


def test_descriptor_encodings_match_the_vendored_cutlass_headers(tmp_path):
    """tests/native/desc_check.cu: this repo's instruction descriptors (bf16 -- proven on hardware --, fp16 and e4m3 of
    the 2-unit product) against cute::UMMA::make_instr_desc, and the K-major SW128 shared-memory descriptor
    against cute::UMMA::SmemDescriptor's bit fields: always against CuTe's values stored in
    tests/golden/umma_descriptors.json, and against the headers themselves where an installed package vendors them."""
    import glob
    import json
    import os
    import re
    import shutil
    import subprocess
    import sys
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    incs = glob.glob(os.path.join(sys.prefix, "lib", "python*", "site-packages", "flashinfer", "data", "cutlass", "include"))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "tests", "golden", "umma_descriptors.json")) as f:
        want = json.load(f)["cute"]
    for inc in [None] + incs[:1]:
        exe = str(tmp_path / ("desc_check_cute" if inc else "desc_check"))
        cmd = [nvcc, "-std=c++17", "-w", "-gencode", "arch=compute_100a,code=sm_100a"] + (["-I" + inc] if inc else []) + [
               "-I" + os.path.join(root, "transformers4rec_b200", "csrc"), "-o", exe,
               os.path.join(root, "tests", "native", "desc_check.cu")]
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-2000:]
        run = subprocess.run([exe], capture_output=True, text=True, timeout=60)
        assert run.returncode == 0 and "MISMATCH" not in run.stdout, run.stdout
        ours = dict(re.findall(r"^(.*?)\s+ours ([0-9a-f]+)", run.stdout, flags=re.M))
        assert ours == want, run.stdout
        if inc:
            assert run.stdout.count(" ok") == len(want)


def test_every_c_abi_call_site_matches_its_ctypes_signature():
    """Static check over the package's Python sources: every ``lib.t4r_*(...)`` call passes as many arguments as the
    ctypes signature in _lib.SIGNATURES declares (``*tail`` = (stream, on_host)).  Most wrappers only run on a GPU, so
    an arity slip would otherwise surface there first."""
    import ast
    import pathlib
    from transformers4rec_b200 import _lib
    root = pathlib.Path(_lib.__file__).parent
    checked = 0
    for path in sorted(root.glob("*.py")):
        tree = ast.parse(path.read_text())
        for node in ast.walk(tree):
            if not (isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and node.func.attr.startswith("t4r_")):
                continue
            name = node.func.attr
            assert name in _lib.SIGNATURES, (path.name, node.lineno, name)
            stars = sum(isinstance(a, ast.Starred) for a in node.args)
            plain = len(node.args) - stars
            assert stars <= 1, (path.name, node.lineno, name)
            assert plain + 2 * stars == len(_lib.SIGNATURES[name][1]), (path.name, node.lineno, name)
            checked += 1
    assert checked >= 50


def test_header_prototypes_and_ctypes_signatures_agree_on_argument_counts():
    """include/t4r_b200.h vs _lib.SIGNATURES: same set of entry points, same number of arguments each (the .cu files
    include the header, so the compiler already holds the definitions to it)."""
    import pathlib
    import re
    from transformers4rec_b200 import _lib
    src = (pathlib.Path(__file__).parent.parent / "include" / "t4r_b200.h").read_text()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"//[^\n]*", "", src)
    protos = re.findall(r"\b(?:int|void|const char\s*\*|int64_t|size_t|long long)\s+(t4r_\w+)\s*\(([^;{]*?)\)\s*;", src, flags=re.S)
    assert {n for n, _ in protos} == set(_lib.SIGNATURES)
    for name, args in protos:
        args = args.strip()
        n = 0 if args in ("", "void") else args.count(",") + 1
        assert n == len(_lib.SIGNATURES[name][1]), name


class _MarshalOnlyLib:
    """Stands in for the loaded library: every entry point converts its arguments with the ctypes signature's own
    ``from_param`` (what a real call does before jumping to native code), counts the call and returns success."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        from transformers4rec_b200 import _lib
        restype, argtypes = _lib.SIGNATURES[name]

        def call(*args):
            assert len(args) == len(argtypes), (name, len(args), len(argtypes))
            for i, (t, a) in enumerate(zip(argtypes, args)):
                try:
                    t.from_param(a)
                except Exception as exc:   # noqa: BLE001
                    raise AssertionError(f"{name}: argument {i} ({a!r}) does not convert to {t}: {exc}")
            self.calls.append(name)
            return 4096 if name.endswith("workspace_bytes") else 0
        return call


def test_gpu_only_wrappers_marshal_their_arguments(monkeypatch):
    """The wrappers written after the last GPU run that have no host twin (device-only entry points) are driven on CPU
    tensors against a library stand-in that only performs ctypes' argument conversion: argument order / count / kinds of
    every call are what the signatures declare, and the Python around the call (shapes, workspace, plane handling) runs."""
    from transformers4rec_b200 import _lib, ops
    fake = _MarshalOnlyLib()
    monkeypatch.setattr(_lib, "load", lambda: fake)
    monkeypatch.setattr(ops, "_need_cuda", lambda *a, **k: None)
    monkeypatch.setattr(ops, "_stream", lambda: None)
    g = torch.Generator().manual_seed(0)
    T, V, De, B, L, H, d = 24, 200, 64, 3, 8, 2, 64
    xt, W = torch.randn(T, De, generator=g), torch.randn(V, De, generator=g)
    labels = torch.randint(1, V, (T,), generator=g)
    xp, xs = ops.split_planes_mixed(xt)
    wp, wsc = ops.split_planes_mixed(W)
    res = ops.head_softmax_ce(xp, xt, labels, wp, W, nprod=2, xt_inv_scale=xs, w_inv_scale=wsc, want_rank=True,
                              label_smoothing=0.1)
    assert res["row_lse"].shape == (T,) and res["row_rank"].dtype == torch.int32
    with pytest.raises(_lib.T4RError):
        ops.head_softmax_ce(xp, xt, labels, wp, W, nprod=2)
    assert ops.head_logits_mixed(xp, xs, wp, wsc, De).shape == (T, V)
    M = B * L
    qkv, R = torch.randn(M, 3 * d, generator=g), torch.randn(2 * L, d, generator=g)
    rw, rr = torch.randn(d, generator=g), torch.randn(d, generator=g)
    assert ops.xlnet_attn_fwd(qkv, R, rw, rr, B, L, H).shape == (M, d)
    assert ops.causal_attn_fwd(qkv, B, L, H).shape == (M, d)
    pm = torch.zeros(B, L, L, dtype=torch.bool)
    qkv2 = torch.randn(2 * M, 3 * d, generator=g)
    assert ops.xlnet_attn_plm_fwd(qkv2, R, rw, rr, B, L, H, pm).shape == (2 * M, d)
    assert ops.rel_pos_proj([torch.randn(d, d, generator=g) for _ in range(2)], L, d).shape == (2, 2 * L, d)
    layers = (_lib.XLNetLayer * 2)()
    assert ops.xlnet_encoder_plm(layers, 2, B, L, d, H, 0.03, torch.randn(2 * M, d, generator=g), pm).shape == (2 * M, d)
    u = torch.rand(B, L, generator=g)
    ids = torch.randint(1, 50, (B, L), generator=g)
    out = ops.mask_plm(ids, _lib.PLM_TRAIN, 0, 3, 1.0 / 6, {"u_span": u, "u_start": u, "u_force": u[:, 0].contiguous(),
                                                            "u_unmask": u[:, 0].contiguous(),
                                                            "perm": torch.rand(B, L, generator=g)})
    assert out is not None
    # the training primitives in device mode (same wrappers as their host twins, other tail)
    x, dy = torch.randn(M, d, generator=g), torch.randn(M, d, generator=g)
    ops.transpose(x); ops.act_fwd(_lib.ACT_GELU, x); ops.act_bwd(_lib.ACT_GELU, x, dy); ops.col_sum(x)
    ops.layer_norm_fwd(x, rw, rr, 0.03); ops.layer_norm_bwd(x, rw, 0.03, dy, add=x)
    ops.xlnet_attn_bwd(qkv, R, rw, rr, dy, B, L, H); ops.xlnet_attn_bwd(qkv2, R, rw, rr, torch.cat([dy, dy]), B, L, H, plm_mask=pm)
    ops.causal_attn_bwd(qkv, dy, B, L, H)
    ops.soft_emb_fwd(x[:, 0], rw[:10], rr[:10], W[:10]); ops.ew_add(x, dy); ops.ew_mul(x, dy)
    ops.adamw_step(x.view(-1), dy.view(-1), torch.zeros(M * d), torch.zeros(M * d), 1e-3, 0.9, 0.999, 1e-8, 0.01, 1)
    assert len(fake.calls) >= 25


def test_mixed_mma_operand_offsets_pick_matching_k_ranges():
    """The 2-unit product's MMA issue sequence (t4r_gemm.cu, ``nprod == 2`` branches), replayed on the byte layout the
    REAL packing code produces: per 64-K block and 128-byte operand row, four K = 16 fp16 MMAs at byte offsets
    ``k4 * 32`` of plane 0, then for j = 0, 1 one K = 32 e4m3 MMA of A bytes [64 + 32 j, +32) x B bytes [32 j, +32) of
    plane 1 and one of A bytes [32 j, +32) x B bytes [64 + 32 j, +32).  Summed in fp64 this must be the emulated product
    (main + lo8(A) hi8(B) + hi8(A) lo8(B)) -- i.e. the offsets pair the SAME K indices of the two operands."""
    import _mixed_ref as R
    from transformers4rec_b200 import ops
    g = torch.Generator().manual_seed(3)
    a, b = torch.randn(9, 200, generator=g), torch.randn(7, 200, generator=g) * 0.05
    (pa, ia), (pb, ib) = ops.split_planes_mixed_host(a), ops.split_planes_mixed_host(b)
    Kp = pa.shape[2]
    rows = lambda p, plane: p[plane].contiguous().view(torch.uint8).reshape(p.shape[1], Kp // 64, 128)   # [row, kb, 128 B]
    a0, a1, b0, b1 = rows(pa, 0), rows(pa, 1), rows(pb, 0), rows(pb, 1)
    f16 = lambda t: t.contiguous().view(torch.float16).double()
    f8 = lambda t: t.contiguous().view(torch.float8_e4m3fn).double()
    acc = torch.zeros((9, 7), dtype=torch.float64)
    for kb in range(Kp // 64):
        for k4 in range(4):
            acc += f16(a0[:, kb, k4 * 32:k4 * 32 + 32]) @ f16(b0[:, kb, k4 * 32:k4 * 32 + 32]).t()
        for j in range(2):
            acc += f8(a1[:, kb, 64 + j * 32:96 + j * 32]) @ f8(b1[:, kb, j * 32:32 + j * 32]).t()
            acc += f8(a1[:, kb, j * 32:32 + j * 32]) @ f8(b1[:, kb, 64 + j * 32:96 + j * 32]).t()
    got = acc * ia.double()[:, None] * ib.double()[None, :]
    want = R.product(R.pack(a), R.pack(b))
    assert torch.equal(got, want) or (got - want).abs().max().item() < 1e-12
    assert (got - a.double() @ b.double().t()).abs().max().item() < 1e-4


def test_product_path_has_no_cpu_fallback(monkeypatch, tmp_path):
    """The product fails loudly instead of computing on the CPU: module forward with CPU tensors, the training step with
    CPU tensors, every public op wrapper with CPU tensors (the host twins are reachable only through ``ops.host_twin``,
    which nothing in the package, bench.py or __graft_entry__ calls), and a missing shared library."""
    import inspect
    import pathlib
    import transformers4rec_b200.torch as tr
    from transformers4rec_b200 import T4RError, _lib, ops
    schema = tr.Schema([tr.ColumnSchema.create_categorical("item_id/list", 300, tags=[tr.Tags.ITEM_ID])])
    inputs = tr.TabularSequenceFeatures.from_schema(schema, max_sequence_length=8, d_output=64, masking="mlm")
    model = tr.XLNetConfig.build(64, 2, 1, 8).to_torch_model(inputs, tr.NextItemPredictionTask(weight_tying=True))
    batch = {"item_id/list": torch.randint(1, 301, (4, 8))}
    with pytest.raises(T4RError, match="no CPU fallback"):
        with torch.no_grad():
            model(dict(batch), training=True)
    with pytest.raises(T4RError, match="no CPU fallback"):
        tr.training_loss(model, dict(batch))
    x = torch.randn(8, 64)
    for fn, args in ((ops.split_planes, (x,)), (ops.transpose, (x,)), (ops.col_sum, (x,)), (ops.ew_add, (x, x)),
                     (ops.act_fwd, (_lib.ACT_GELU, x)), (ops.split_planes_mixed, (x,))):
        with pytest.raises(T4RError, match="no CPU fallback"):
            fn(*args)
    # nothing shipped selects a host twin
    root = pathlib.Path(_lib.__file__).parent
    shipped = list(root.glob("*.py")) + list((root / "torch").glob("*.py")) + [root.parent / "bench.py",
                                                                                   root.parent / "__graft_entry__.py"]
    for path in shipped:
        src = "\n".join(ln for ln in path.read_text().splitlines() if not ln.lstrip().startswith("#"))
        assert "_on_host=True" not in src.replace("fn(*a, _on_host=True, **k)", ""), path
        assert "host_twin(" not in src.replace("def host_twin(", ""), path
    assert "_on_host=True" in inspect.getsource(ops.host_twin)
    # missing library: a loud error, not a fallback
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(T4RError, match="no CPU/eager fallback"):
        _lib.load()
