#!/usr/bin/env python
"""Generate golden input/output vectors by executing the UPSTREAM reference code.

Needs a source checkout of NVIDIA-Merlin/Transformers4Rec, named by the environment
variable T4R_UPSTREAM_SRC; the tests only read the stored vectors.  The reference
package cannot be imported as a whole (merlin-*,
betterproto, torchmetrics are absent and HF 5.5 dropped symbols it imports;
SURVEY.md §8c), so this script loads the individual upstream source files for the
arithmetic of the hot path -- masking.py, ranking_metric.py, the sampler / head in
model/prediction_task.py -- under stub modules for their third-party imports, runs
them on seeded inputs and stores inputs + outputs in ``tests/golden/*.pt``.

Randomness: the reference draws with torch.bernoulli / torch.multinomial.  While the
upstream code runs, both are monkey-patched to consume explicit uniforms (the rule in
oracle/t4r_oracle.py: bernoulli = u < p; multinomial over 0/1 weights = k-th set
position, k = floor(u*n)), so the very same draws can be fed to the oracle and to the
CUDA kernels.  Nothing from the reference is copied into this repository: only
tensors it produced.

Usage:  T4R_UPSTREAM_SRC=<checkout> python tests/golden/make_golden.py     (writes tests/golden/*.pt)

Every stored file stays under 1 MB; the head's vocabulary (Vh) and label rows (Th) are sized for that.
"""
import importlib
import os
import sys
import types

import numpy as np
import torch

REF = os.environ.get("T4R_UPSTREAM_SRC", "")
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(HERE)), "oracle"))
import t4r_oracle as O  # noqa: E402  (only for the uniform->draw helpers, so both sides share them)


class _DummyMeta(type):
    def __getattr__(cls, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _DummyMeta(name, (), {"__init__": lambda self, *a, **k: None, "__call__": lambda self, *a, **k: None})


class _Anything(types.ModuleType):
    """A module whose every attribute is a harmless dummy (class / decorator factory)."""

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        obj = type(name, (), {"__init__": lambda self, *a, **k: None, "__call__": lambda self, *a, **k: None})
        setattr(self, name, obj)
        return obj


class _Registry:
    def __init__(self, *a, **k):
        self._d = {}

    def register(self, name):
        def deco(x):
            self._d[name] = x
            return x
        return deco

    def register_with_multiple_names(self, *names):
        def deco(x):
            for n in names:
                self._d[n] = x
            return x
        return deco

    def parse(self, name):
        return self._d[name] if isinstance(name, str) else name

    @classmethod
    def class_registry(cls, *a, **k):
        return cls()

    def __getitem__(self, k):
        return self._d[k]


def _docstring_parameter(*a, **k):
    def deco(x):
        return x
    return deco


class _Metric(torch.nn.Module):
    """Just enough of torchmetrics.Metric for RankingMetric (add_state / __call__ / compute)."""

    def __init__(self, *a, **k):
        super().__init__()

    def add_state(self, name, default, dist_reduce_fx=None):
        setattr(self, name, list(default) if isinstance(default, list) else default)

    def forward(self, *a, **k):
        self.update(*a, **k)
        return self.compute()


def install_stubs():
    def mod(name, cls=_Anything, **attrs):
        m = cls(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m
        return m

    for name in ("merlin", "merlin.models", "merlin.models.utils", "merlin.schema", "merlin.schema.io",
                 "merlin.schema.io.proto_utils", "merlin.schema.tags", "merlin.models.utils.misc_utils",
                 "merlin_standard_lib", "merlin_standard_lib.schema", "merlin_standard_lib.schema.schema",
                 "merlin_standard_lib.utils", "merlin_standard_lib.utils.proto_utils", "merlin.dataloader",
                 "merlin.core", "merlin.io"):
        mod(name)
    mod("merlin.models.utils.doc_utils", docstring_parameter=_docstring_parameter)
    mod("merlin.models.utils.registry", Registry=_Registry)
    mod("torchmetrics", Metric=_Metric, regression=_Anything("torchmetrics.regression"),
        Precision=_DummyMeta("Precision", (), {"__init__": lambda self, *a, **k: None}),
        Recall=_DummyMeta("Recall", (), {"__init__": lambda self, *a, **k: None}),
        Accuracy=_DummyMeta("Accuracy", (), {"__init__": lambda self, *a, **k: None}))
    mod("torchmetrics.utilities")
    mod("torchmetrics.utilities.data", dim_zero_cat=lambda x: torch.cat(list(x), dim=0) if isinstance(x, (list, tuple)) else x)
    # package shells whose __path__ points at the real source tree: sub-modules are the real files
    for pkg, rel in (("transformers4rec", "transformers4rec"), ("transformers4rec.torch", "transformers4rec/torch"),
                     ("transformers4rec.torch.utils", "transformers4rec/torch/utils"),
                     ("transformers4rec.torch.model", "transformers4rec/torch/model"),
                     ("transformers4rec.torch.block", "transformers4rec/torch/block"),
                     ("transformers4rec.torch.tabular", "transformers4rec/torch/tabular"),
                     ("transformers4rec.torch.features", "transformers4rec/torch/features"),
                     ("transformers4rec.config", "transformers4rec/config")):
        m = types.ModuleType(pkg)
        m.__path__ = [os.path.join(REF, rel)]
        sys.modules[pkg] = m
    # modules that would drag in the whole framework are replaced by dummies
    mod("transformers4rec.config.schema", SchemaMixin=type("SchemaMixin", (), {}), requires_schema=lambda x: x)
    mod("transformers4rec.torch.typing")
    mod("transformers4rec.torch.block.base")
    mod("transformers4rec.torch.block.mlp")
    mod("transformers4rec.torch.model.base", PredictionTask=torch.nn.Module, BlockType=object)


class patched_draws:
    """Route torch.bernoulli / torch.multinomial through explicit uniforms."""

    def __init__(self, u_bern=None, multinomial_us=(), raw_multinomial=None):
        self.u_bern = u_bern
        self.us = list(multinomial_us)
        self.raw = raw_multinomial

    def __enter__(self):
        self._b, self._m = torch.bernoulli, torch.multinomial

        def bern(prob_matrix, *a, **k):
            p = float(prob_matrix.flatten()[0])
            return O.bernoulli_from_uniform(self.u_bern, p).to(prob_matrix.dtype)

        def multi(weights, num_samples, replacement=False, **k):
            if self.raw is not None and weights.ndim == 1:
                return self.raw
            u = self.us.pop(0)
            return O.pick_kth_set(weights > 0, u).unsqueeze(1)

        torch.bernoulli, torch.multinomial = bern, multi
        return self

    def __exit__(self, *a):
        torch.bernoulli, torch.multinomial = self._b, self._m


def main():
    assert os.path.isdir(REF), "set T4R_UPSTREAM_SRC to a source checkout of NVIDIA-Merlin/Transformers4Rec"
    install_stubs()
    # utils/torch_utils.py imports the four masking classes at class-body time (a cycle the
    # real package resolves through its __init__ order): satisfy it with placeholders first
    fake = _Anything("transformers4rec.torch.masking")
    sys.modules["transformers4rec.torch.masking"] = fake
    importlib.import_module("transformers4rec.torch.utils.torch_utils")
    del sys.modules["transformers4rec.torch.masking"]
    masking = importlib.import_module("transformers4rec.torch.masking")
    ranking = importlib.import_module("transformers4rec.torch.ranking_metric")
    ptask = importlib.import_module("transformers4rec.torch.model.prediction_task")
    out = {}

    # ---------------------------------------------------------------- masking
    g = torch.Generator().manual_seed(1234)
    B, L, d = 64, 12, 8
    lens = torch.randint(1, L + 1, (B,), generator=g)
    ids = torch.randint(1, 500, (B, L), generator=g)
    ids = torch.where(torch.arange(L).unsqueeze(0) < lens.unsqueeze(1), ids, torch.zeros_like(ids))
    x = torch.rand((B, L, d), generator=g)
    u = torch.rand((B, L + 2), generator=g)
    cases = {}
    for name, cls, kw in (("mlm", masking.MaskedLanguageModeling, {}),
                          ("mlm_all", masking.MaskedLanguageModeling, {"eval_on_last_item_seq_only": False}),
                          ("clm", masking.CausalLanguageModeling, {}),
                          ("clm_trainlast", masking.CausalLanguageModeling, {"train_on_last_item_seq_only": True}),
                          ("clm_evalall", masking.CausalLanguageModeling, {"eval_on_last_item_seq_only": False})):
        torch.manual_seed(7)
        m = cls(hidden_size=d, **kw)
        emb = m.masked_item_embedding.detach().clone()
        for training, testing in ((True, False), (False, True), (False, False)):
            with patched_draws(u_bern=u[:, :L], multinomial_us=[u[:, L], u[:, L + 1]]):
                with torch.no_grad():
                    y = m(x, item_ids=ids, training=training, testing=testing)
            cases[f"{name}/{int(training)}{int(testing)}"] = {
                "mask_schema": m.mask_schema.clone(), "masked_targets": m.masked_targets.clone(), "out": y.clone(),
                "masked_item_embedding": emb, "kwargs": kw}
    out["masking"] = {"item_ids": ids, "x": x, "u": u, "cases": cases}

    # ---------------------------------------------------------------- ranking metric
    T, V = 40, 57
    scores = torch.rand((T, V), generator=g)
    labels = torch.randint(1, V, (T,), generator=g)
    ks = [1, 2, 5, 10, 20]
    rec = ranking.RecallAt(top_ks=ks, labels_onehot=True)
    res = rec(scores, labels)
    out["recall"] = {"scores": scores, "labels": labels, "ks": ks, "recall": res.clone(),
                     "known_answer_scores": torch.tensor([[1, 2, 3, 4, 5, 4, 3, 2, 1]] * 3),
                     "known_answer_labels": torch.tensor([7, 5, 4]),
                     "known_answer_recall": torch.tensor([0.3333, 0.3333, 0.6667, 0.6667])}

    # ---------------------------------------------------------------- sampler + head
    Vh, De, Th, S = 1001, 32, 32, 200
    sampler = ptask.LogUniformSampler(max_n_samples=S, max_id=Vh, min_id=1, unique_sampling=True)
    xt = torch.randn((Th, De), generator=g)
    W = torch.randn((Vh, De), generator=g) * 0.1
    y = torch.randint(1, Vh, (Th,), generator=g)
    raw = torch.multinomial(sampler.dist, 2 * S, replacement=True, generator=g)
    raw[:4] = y[:4]  # accidental hits
    table = torch.nn.Embedding(Vh, De)
    with torch.no_grad():
        table.weight.copy_(W)
    full = ptask._NextItemPredictionTask([Th, De], Vh, weight_tying=True, item_embedding_table=table,
                                         softmax_temperature=2.0)
    with torch.no_grad():
        logits_full, _ = full(xt, targets=y, training=True)
        loss_full = torch.nn.CrossEntropyLoss()(logits_full, y)
    samp = ptask._NextItemPredictionTask([Th, De], Vh, weight_tying=True, item_embedding_table=table,
                                         softmax_temperature=1.0, sampled_softmax=True, max_n_samples=S, min_id=1)
    with patched_draws(raw_multinomial=raw):
        with torch.no_grad():
            logits_s, tgt_s = samp(xt, targets=y, training=True)
            loss_s = torch.nn.CrossEntropyLoss()(logits_s, tgt_s)
    out["head"] = {"xt": xt, "W": W, "y": y, "raw_draws": raw, "S": S, "dist": sampler.dist.clone(),
                   "unique_sampling_dist": sampler.unique_sampling_dist.clone(),
                   "logits_full_tau2": logits_full, "loss_full_tau2": loss_full,
                   "logits_sampled": logits_s, "loss_sampled": loss_s}

    # ---------------------------------------------------------------- ragged padding (N1)
    padding = importlib.import_module("transformers4rec.torch.utils.padding")
    lens = torch.randint(0, 12, (40,), generator=g)
    offs = torch.cat([torch.zeros(1, dtype=torch.long), lens.cumsum(0)])
    ids = torch.randint(1, 1000, (int(offs[-1]),), generator=g)
    fl = torch.rand(int(offs[-1]), generator=g)
    dense = torch.randint(1, 50, (40, 6), generator=g)
    inp = {"i__values": ids, "i__offsets": offs, "f__values": fl, "f__offsets": offs, "d": dense}
    out["padding"] = {"inputs": inp,
                      "pad_inputs_none": dict(padding.pad_inputs(dict(inp))),
                      "pad_inputs_8": dict(padding.pad_inputs(dict(inp), 8)),
                      "pad_batch_15_4": dict(padding.pad_batch(dict(inp), {"i": 15, "f": 15, "d": 4}))}

    torch.save(out, os.path.join(HERE, "reference_vectors.pt"))
    sizes = {k: sum(v.numel() for v in _flatten(vs)) for k, vs in out.items()}
    print("wrote reference_vectors.pt", sizes)


def _flatten(x):
    if torch.is_tensor(x):
        yield x
    elif isinstance(x, dict):
        for v in x.values():
            yield from _flatten(v)
    elif isinstance(x, (list, tuple)):
        for v in x:
            yield from _flatten(v)


if __name__ == "__main__":
    main()
