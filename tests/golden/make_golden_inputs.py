#!/usr/bin/env python
"""Golden vectors for the widened input block and the remaining ranking metrics (SURVEY.md §8f
N2 / N4), produced -- like make_golden.py, whose stub machinery this script reuses -- by executing
the UPSTREAM source files: tabular/aggregation.py, tabular/transformations.py,
features/embedding.py (SoftEmbedding) and ranking_metric.py.  Authoring container only.

StochasticSwapNoise draws with torch.bernoulli and torch.randperm; both are patched while the
upstream code runs so that the recorded draws (``u``, ``perm``) can be replayed through the
oracle and the CUDA kernel.

Usage:  python tests/golden/make_golden_inputs.py    (writes tests/golden/reference_vectors_n4.pt)
"""
import importlib
import os
import sys
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden as G  # noqa: E402


def load_upstream():
    G.install_stubs()
    for name in ("merlin_standard_lib.utils.embedding_utils", "merlin_standard_lib.utils.misc_utils",
                 "merlin_standard_lib.utils.doc_utils", "merlin_standard_lib.registry",
                 "merlin.models.utils.schema_utils"):
        sys.modules[name] = G._Anything(name)
    fake = G._Anything("transformers4rec.torch.masking")
    sys.modules["transformers4rec.torch.masking"] = fake
    importlib.import_module("transformers4rec.torch.utils.torch_utils")
    del sys.modules["transformers4rec.torch.masking"]
    agg = importlib.import_module("transformers4rec.torch.tabular.aggregation")
    emb = importlib.import_module("transformers4rec.torch.features.embedding")
    trf = importlib.import_module("transformers4rec.torch.tabular.transformations")
    rank = importlib.import_module("transformers4rec.torch.ranking_metric")
    return agg, emb, trf, rank


class patched_ssn_draws:
    def __init__(self, u, perm):
        self.u, self.perm = u, perm

    def __enter__(self):
        self._b, self._r = torch.bernoulli, torch.randperm
        torch.bernoulli = lambda pm, *a, **k: (self.u < float(pm.flatten()[0])).to(pm.dtype)
        torch.randperm = lambda n, *a, **k: self.perm[:n].clone() if self.perm.numel() == n else (_ for _ in ()).throw(
            AssertionError(f"perm has {self.perm.numel()} entries, randperm({n}) requested"))
        return self

    def __exit__(self, *a):
        torch.bernoulli, torch.randperm = self._b, self._r


def main():
    assert os.path.isdir(G.REF), "set T4R_UPSTREAM_SRC to a source checkout of NVIDIA-Merlin/Transformers4Rec"
    agg, emb, trf, rank = load_upstream()
    g = torch.Generator().manual_seed(4321)
    out = {}

    # ------------------------------------------------------------- ranking metrics (N2)
    T, V = 48, 61
    scores = torch.rand((T, V), generator=g)
    labels = torch.randint(0, V, (T,), generator=g)
    ks = [1, 3, 5, 10, 20]
    res = {}
    for name in ("precision_at", "recall_at", "avg_precision_at", "dcg_at", "ndcg_at", "mrr_at"):
        m = rank.ranking_metrics_registry[name](top_ks=ks, labels_onehot=True)
        res[name] = m(scores, labels).clone()
    ka_scores = torch.tensor([[1, 2, 3, 4, 5, 4, 3, 2, 1]] * 3)
    ka_onehot = torch.tensor([[0, 0, 0, 0, 0, 0, 0, 1, 0], [0, 0, 0, 0, 0, 1, 0, 0, 0], [0, 0, 0, 0, 1, 0, 0, 0, 0]])
    out["metrics"] = {"scores": scores, "labels": labels, "ks": ks, "results": res,
                      "known_answer_scores": ka_scores, "known_answer_onehot": ka_onehot,
                      "known_answer_mrr": torch.tensor([0.3333, 0.3333, 0.4444, 0.4444]),  # tests/unit/torch/test_ranking_metrics.py:49-65
                      "known_answer_recall": torch.tensor([0.3333, 0.3333, 0.6667, 0.6667])}

    # ------------------------------------------------------------- aggregations (N4)
    B, L, D = 6, 7, 12
    feats = {"item": torch.randn((B, L, D), generator=g), "cat_b": torch.randn((B, L, D), generator=g),
             "aa_ctx": torch.randn((B, D), generator=g), "price": torch.randn((B, L, D), generator=g)}
    a_sum = agg.ElementwiseSum()
    a_cat = agg.ConcatFeatures()
    a_mul = agg.ElementwiseSumItemMulti()
    a_mul.schema = types.SimpleNamespace(item_id_column_name="item")
    a_mul.get_item_ids_from_inputs = lambda inputs: inputs["item"]
    out["aggregation"] = {"features": {k: v.clone() for k, v in feats.items()},
                          "concat": a_cat.forward({k: v.clone() for k, v in feats.items()}),
                          "element-wise-sum": a_sum.forward({k: v.clone() for k, v in feats.items()}),
                          "element-wise-sum-item-multi": a_mul.forward({k: v.clone() for k, v in feats.items()}),
                          "item_name": "item"}

    # ------------------------------------------------------------- per-feature LayerNorm (N4)
    ln = trf.TabularLayerNorm({"item": D, "cat_b": D})
    with torch.no_grad():
        for m in ln.feature_layer_norm.values():
            m.weight.copy_(torch.rand(D, generator=g) + 0.5)
            m.bias.copy_(torch.randn(D, generator=g))
        ln_out = ln.forward({k: feats[k] for k in ("item", "cat_b", "price")})
    out["layer_norm"] = {"inputs": {k: feats[k].clone() for k in ("item", "cat_b", "price")},
                         "params": {k: (m.weight.detach().clone(), m.bias.detach().clone())
                                    for k, m in ln.feature_layer_norm.items()},
                         "outputs": {k: v.detach().clone() for k, v in ln_out.items()}}

    # ------------------------------------------------------------- SoftEmbedding (N4)
    torch.manual_seed(11)
    se = emb.SoftEmbedding(10, 8)
    x = torch.rand((B, L), generator=g) * 4 - 2
    with torch.no_grad():
        y = se(x)
    out["soft_embedding"] = {"x": x, "table": se.embedding_table.weight.detach().clone(),
                             "proj_weight": se.projection_layer.weight.detach().clone(),
                             "proj_bias": se.projection_layer.bias.detach().clone(), "out": y.clone()}

    # ------------------------------------------------------------- StochasticSwapNoise (N4)
    ssn = trf.StochasticSwapNoise(pad_token=0, replacement_prob=0.35)
    ssn.train()
    Bs, Ls = 9, 11
    lens = torch.randint(1, Ls + 1, (Bs,), generator=g)
    ids = torch.randint(1, 300, (Bs, Ls), generator=g)
    ids = torch.where(torch.arange(Ls).unsqueeze(0) < lens.unsqueeze(1), ids, torch.zeros_like(ids))
    mask = ids != 0
    cases = {}
    for name, vals, msk in (("ids", ids, mask), ("floats", torch.rand((Bs, Ls), generator=g), mask),
                            ("context", torch.randint(1, 50, (Bs,), generator=g), mask),
                            # without a mask upstream permutes ROWS (masked.shape[0]) and only works for 1-D inputs
                            ("nomask_1d", torch.randint(1, 300, (Bs * Ls,), generator=g), None)):
        u = torch.rand(vals.shape, generator=g)
        eff = msk[:, 0] if (msk is not None and vals.dim() == msk.dim() - 1) else msk
        n_pool = int(eff.sum()) if eff is not None else vals.numel()
        perm = torch.randperm(n_pool, generator=g)
        with patched_ssn_draws(u, perm):
            res_ = ssn.augment(vals.clone(), None if msk is None else msk.clone())
        cases[name] = {"values": vals, "mask": msk, "u": u, "perm": perm, "out": res_.clone()}
    out["swap_noise"] = {"replacement_prob": 0.35, "cases": cases}

    torch.save(out, os.path.join(HERE, "reference_vectors_n4.pt"))
    print("wrote reference_vectors_n4.pt", {k: sum(v.numel() for v in G._flatten(vs)) for k, vs in out.items()})


if __name__ == "__main__":
    main()
